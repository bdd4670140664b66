// TMA (cp.async.bulk.tensor) + mbarrier helpers for sm_100a, and the host-side tensor-map encoder.
// The driver entry point cuTensorMapEncodeTiled is fetched through cudaGetDriverEntryPoint so that the
// library does not link against libcuda.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace iic {

// ---- host -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// A (B, K, H, W) float32 tensor with element strides (sn, sc, sh, 1) as a rank-4 tensor map with
// box (box_w, box_h, box_c, 1), written to shared memory with swizzle `swz`; out-of-range elements are
// filled with zeros (which is exactly the zero padding of the F.conv2d at iic_loss.py:123).  Returns false
// when the tensor cannot be described (unaligned base or strides, box too large) -- the caller then uses
// another kernel.
inline bool make_map_4d(CUtensorMap* map, const float* base, int B, int K, int H, int W, long long sn,
                        long long sc, long long sh, int box_w, int box_h, int box_c,
                        CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_NONE) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return false;
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return false;
  if ((sh * 4) % 16 != 0 || (sc * 4) % 16 != 0 || (sn * 4) % 16 != 0) return false;
  if (box_w > 256 || box_h > 256 || box_c > 256 || (box_w * 4) % 16 != 0) return false;
  cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)K, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)sh * 4, (cuuint64_t)sc * 4, (cuuint64_t)sn * 4};
  cuuint32_t box[4] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_c, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// ---- device -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
#ifdef IIC_MBAR_TEST_WAIT
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#else
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#endif
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a mis-programmed copy must fault (trap), not hang the GPU.
#ifdef IIC_TMA_DEBUG
__device__ unsigned int g_tma_dbg[8];
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, unsigned code = 0) {
  uint32_t spins = 0;
  unsigned long long t_start = 0;
  (void)t_start;
  while (!mbar_try_wait(bar, parity)) {
#ifdef IIC_TMA_DEBUG
    if (++spins > (1u << 16)) {
      if (atomicCAS(&g_tma_dbg[0], 0u, code | 0x80000000u) == 0u) {
        g_tma_dbg[1] = blockIdx.x; g_tma_dbg[2] = threadIdx.x; g_tma_dbg[3] = parity; g_tma_dbg[4] = smem_u32(bar);
      }
      return;
    }
#else
    (void)code;
    // try_wait suspends the thread for a hardware-chosen time, so a spin count alone bounds nothing: 4 s by the clock
    if ((++spins & 1023u) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t_start == 0) t_start = now;
      else if (now - t_start > 4000000000ull) __trap();
    }
#endif
  }
}
__device__ __forceinline__ void tma_load_4d(void* dst_smem, const CUtensorMap* map, uint64_t* bar, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
      "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

}  // namespace iic
