// Shared helpers for libiic_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/iic_b200.h"

namespace iic {

// ---- error plumbing: nothing throws across the C ABI ------------------------------------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define IIC_CHECK_CUDA(expr)                                                               \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::iic::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,                  \
                       cudaGetErrorString(_e));                                            \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

#define IIC_REQUIRE(cond, ...)                                                             \
  do {                                                                                     \
    if (!(cond)) {                                                                         \
      ::iic::set_error(__VA_ARGS__);                                                       \
      return 2;                                                                            \
    }                                                                                      \
  } while (0)

#define IIC_CHECK_RC(expr)                                                                 \
  do {                                                                                     \
    const int _rc = (expr);                                                                \
    if (_rc != 0) return _rc;                                                              \
  } while (0)

int sm_count_cached(int device);   // <0 on error
int current_device();

// Run-time switches of the dispatchers (runtime.cu): read from the environment once, at first use, then changed only
// through iic_b200_set_option.  All default to 0 except xchg_timeout_ms.
struct Options {
  int no_tma = 0;             // IIC_B200_NO_TMA: skip every TMA-staged kernel (generic kernels only)
  int no_tc = 0;              // IIC_B200_NO_TC: no tensor-core kernels
  int no_tc10 = 0;            // IIC_B200_NO_TC10: no tensor-core backward for K = 9, 10
  int no_fast = 0;            // IIC_B200_NO_FAST: no specialised FFMA2 kernels
  int tcp_p1 = 0;             // IIC_B200_TCP_P1: packed tensor-core joint also at padding 1 (16 <= K <= 24)
  int tcrb_p1 = 0;            // IIC_B200_TCRB_P1: row-block tensor-core backward at padding 1 whatever the map size
  int tc10_force = 0;         // IIC_B200_TC10_FORCE: K = 10 tensor-core backward whatever the map size
  int no_tcj10 = 0;           // IIC_B200_NO_TCJ10: FFMA2 joint instead of the tensor-core joint for K <= 10, padding 1
  int tc10_tf32 = 0;          // IIC_B200_TC10_TF32: the tf32 + bf16-correction K = 10 backward instead of the fp16-split one
  int no_fused_epilogue = 0;  // IIC_B200_NO_FUSED_EPILOGUE: slot reduce and epilogue as two launches
  int fin_last_cta_epilogue = 0;  // IIC_B200_FIN_LAST_CTA_EPILOGUE: small batches run their epilogues in the finish launch's last CTA
  int xchg_timeout_ms = 0;    // IIC_B200_XCHG_TIMEOUT_MS: bound of the peer wait in the joint exchange
};
const Options& options();

// Layout of the Wx / Wy buffers (iic_local_coeff_floats floats each): the coefficient tensor [patch][cin][tap][Kp] that
// iic_local_epilogue writes, then -- 1 KB aligned -- room for the operand-order "weight image" the tensor-core backward
// kernels build from it (0 bytes when (K, pad, n_patches) never selects such a kernel).  The image is per call and
// per buffer, so concurrent backwards on different streams never share scratch.  Image sizes: local_kernels.cuh.
inline size_t local_coeff_base_floats(int K, int pad, int n_patches) {
  const int T = 2 * pad + 1, Kp = (K + 3) & ~3;
  return (size_t)n_patches * K * T * T * Kp;
}
inline size_t local_coeff_image_offset(int K, int pad, int n_patches) {
  return (local_coeff_base_floats(K, pad, n_patches) + 255) & ~(size_t)255;
}

// ---- per-CTA partial-joint slots of the local joint kernels (what iic_finish / the reduce kernels read) ---------------
enum SlotLayoutKind { SLOT_STD = 0, SLOT_TC128 = 1, SLOT_PACKED = 2 };
struct SlotInfo {
  int layout;             // SLOT_STD:    slot[e], e = ((dy*T+dx)*K+i)*K+j; slots [patch][n_slots][slot_stride]
                          // SLOT_TC128:  local_joint_tc_kernel's coalesced order (K = 128), undone by tc128_out_index
                          // SLOT_PACKED: local_joint_tcp_kernel's accumulator tiles, packed_slot_index
  int n_slots;            // slots per patch
  long long slot_stride;  // floats between consecutive slots
  int nb;                 // SLOT_PACKED: accumulator columns (T * 24)
};
// slot element of (row tile mt, accumulator row m, accumulator column c): chunks of 8 columns, float4-interleaved over rows
__host__ __device__ inline size_t packed_slot_index(int mt, int m, int c, int nb) {
  return ((((size_t)mt * (nb / 8) + c / 8) * 2 + (c % 8) / 4) * 128 + m) * 4 + (c % 4);
}
// SLOT_TC128: output index ((d*128+i)*128+j) of slot element e = [d][32-column chunk][float4 of the chunk][row i][4]
__host__ __device__ inline long long tc128_out_index(long long e) {
  const long long w = e & 3, i = (e >> 2) & 127, jv = (e >> 9) & 7, ch = (e >> 12) & 3, d = e >> 14;
  return (d * 128 + i) * 128 + ch * 32 + jv * 4 + w;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize once per (device, kernel); thread-safe.  0 = ok.
int ensure_dyn_smem(const void* func, int bytes);

// ---- patch windows (contrastyou/losses/iic_loss.py:152-160) -----------------------------------------
struct PatchGrid {
  int H, W;        // full map
  int ph, pw;      // effective patch extent = min(patch, map)
  int sh, sw;      // steps
  int nh, nw;      // windows per axis
};

__host__ __device__ inline int patch_axis_count(int extent, int patch, int step) {
  // np.arange(0, extent - patch, step) has ceil((extent-patch)/step) entries when extent > patch,
  // then one more window flush with the border is appended.
  if (extent <= patch) return 1;
  return (extent - patch + step - 1) / step + 1;
}
__host__ __device__ inline int patch_axis_origin(int idx, int count, int extent, int patch, int step) {
  if (idx < count - 1) return idx * step;
  int o = extent - patch;
  return o > 0 ? o : 0;
}
__host__ inline bool make_patch_grid(int H, int W, int patch_h, int patch_w, int step_h, int step_w,
                                     PatchGrid* g) {
  if (H <= 0 || W <= 0 || patch_h <= 0 || patch_w <= 0) return false;
  if ((H > patch_h && step_h <= 0) || (W > patch_w && step_w <= 0)) return false;
  g->H = H; g->W = W;
  g->ph = patch_h < H ? patch_h : H;
  g->pw = patch_w < W ? patch_w : W;
  g->sh = step_h > 0 ? step_h : 1;
  g->sw = step_w > 0 ? step_w : 1;
  g->nh = patch_axis_count(H, patch_h, g->sh);
  g->nw = patch_axis_count(W, patch_w, g->sw);
  return true;
}

struct View4 {          // (B, K, H, W) float32 view, W-stride 1
  const float* p;
  long long sn, sc, sh;
};

// ---- warp / block reductions (fixed order -> deterministic) ------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum of doubles; `scratch` has >= 33 doubles of shared memory. All threads get the result.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double t = lane < nw ? scratch[lane] : 0.0;
    t = warp_sum(t);
    if (lane == 0) scratch[32] = t;
  }
  __syncthreads();
  return scratch[32];
}
// NaN-propagating block-wide min (fmin would drop NaNs; a NaN joint must poison the loss as in torch.min)
__device__ __forceinline__ double block_min_nan(double v, bool has_nan, double* scratch) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_min(v);
  unsigned any_nan = __ballot_sync(0xffffffffu, has_nan);
  __syncthreads();
  if (lane == 0) scratch[wid] = any_nan ? __longlong_as_double(0x7ff8000000000000LL) : v;
  __syncthreads();
  if (wid == 0) {
    double t = lane < nw ? scratch[lane] : __longlong_as_double(0x7ff0000000000000LL);
    bool n2 = (t != t);
    unsigned an = __ballot_sync(0xffffffffu, n2);
    t = warp_min(n2 ? __longlong_as_double(0x7ff0000000000000LL) : t);
    if (lane == 0) scratch[32] = an ? __longlong_as_double(0x7ff8000000000000LL) : t;
  }
  __syncthreads();
  return scratch[32];
}

}  // namespace iic
