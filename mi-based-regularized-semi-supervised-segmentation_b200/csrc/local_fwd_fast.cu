// Specialised local joint (contrastyou/losses/iic_loss.py:120-123) for the 3 x 3 window (padding = 1) and
// channel counts that are multiples of 10 -- the shapes of the reference's udaiic configuration
// (config/semi.yaml: 10 or 20 clusters, paddings [1, ...]).  Same output-stationary scheme as
// local_fwd_tma.cu, but every extent is a compile-time constant so that the inner loop is nothing but
// shared-memory loads at immediate offsets and packed FP32 FMAs:
//   * a 10 x 10 block of (x channel, y channel) pairs is cut into 10 jobs of 2 x 5 channels; a job keeps
//     its 2 x 5 x 9 sums as 45 float2 accumulators (pairs over the two x channels) and is owned by one warp,
//     lanes = the 32 pixel columns of the tile, walking down the 16 tile rows with a rolling 3-row window:
//     per row 6 + 5 LDS.32, 5 MOV and 45 FFMA2;
//   * 10 jobs do not spread evenly over the SM's 4 sub-partitions (3,3,2,2 warps), so jobs 0 and 1 are
//     split by rows between their own warp and a helper warp (warps 10, 11): every sub-partition then
//     issues exactly 40 row-jobs per tile;
//   * 12 warps = 3 per sub-partition leaves 168 registers per thread, so there is no dedicated producer
//     warp (a 13th warp would cap the kernel at 128 registers and spill the accumulators): lane 0 of
//     helper warp 10, which has half a job's work and therefore slack, issues the TMA loads -- rank-4
//     boxes of the x tile (with halo) and the y tile into a 4-stage full/empty mbarrier ring, out-of-range
//     elements zero-filled by the hardware (= the conv padding);
//   * K = 20, 30, ...: blockIdx.y selects the (x block, y block) pair, the tensor-map channel coordinate
//     does the slicing.
#include "common.cuh"
#include "local_kernels.cuh"
#include "tma.cuh"

namespace iic {

struct FwdFastParams {
  int B, K, H, W, tiles_h, tiles_w;
  float* partial;           // [gridDim.x][9][K][K]
  int* flags;               // non-null (and K == 10): also assert that x is a simplex over its channels
  float inv_temp;           // FROM_LOGITS: softmax(logit * inv_temp)  (SoftmaxWithT, contrastyou/trainer/_utils.py:15-23)
};

}  // namespace iic

namespace iic {

#define IIC_FWD_NS fwd3_kb10
#define IIC_FWD_KB 10
#include "local_fwd_fast3.inc"
#undef IIC_FWD_NS
#undef IIC_FWD_KB
#define IIC_FWD_NS fwd3_kb8
#define IIC_FWD_KB 8
#include "local_fwd_fast3.inc"
#undef IIC_FWD_NS
#undef IIC_FWD_KB

// Channel blocks of 10 for the udaiic cluster counts (10, 20, ..), of 8 for other multiples of 8 (.., 128).
int local_joint_fast_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, int* flags, int* checked,
                         int from_logits, float inv_temp, cudaStream_t st) {
  *checked = 0;
  if (m.K % 10 == 0 && m.K <= 40)
    return fwd3_kb10::local_joint_fast_try_kb(m, partial, max_ctas, slots, flags, checked, from_logits, inv_temp, st);
  if (m.K % 8 == 0 && m.K <= 256 && !from_logits)
    return fwd3_kb8::local_joint_fast_try_kb(m, partial, max_ctas, slots, flags, checked, 0, 1.f, st);
  return -1;
}

// ======================================================================================================
// 7 x 7 window (padding 3, the yaml default for Up_conv2: config/semi.yaml paddings [1, 3]).
// 49 displacements x 100 channel pairs do not fit one CTA's registers, so the grid's y index also selects
// ONE displacement row dy: a CTA then needs only the x rows shifted by dy (no row halo) and computes the 7
// column shifts of that row.  Inside a CTA the 10-job structure of the 3 x 3 kernel is kept (job = 2 x
// channels x 5 y channels, 35 float2 accumulators), but a lane owns 4 consecutive pixels so that the 10
// window columns of a row come from three LDS.128 per channel: lanes = 8 pixel quads x 4 row bands of the
// 32 x 32 tile.  Per row step: 11 LDS.128 and 140 FFMA2.
// ======================================================================================================
namespace fwdfast7 {
constexpr int T = 7, PAD = 3, TH = 32, TW = 32, LP = 4, XP = LP + TW + 4, RB = TH / 4;
constexpr int KB = 10, JT = 5;
constexpr int NJOBS = (KB / 2) * (KB / JT);        // 10
constexpr int NHELP = 2, NCONS = NJOBS + NHELP, NTHREADS = NCONS * 32, PRODUCER_WARP = NJOBS;
constexpr int STAGES = 2;
constexpr unsigned X_BYTES = KB * TH * XP * 4;     // one displacement row: TH rows, no row halo
constexpr unsigned Y_BYTES = KB * TH * TW * 4;
constexpr unsigned X_REGION = (X_BYTES + 127u) & ~127u;
constexpr unsigned STAGE_BYTES = X_REGION + ((Y_BYTES + 127u) & ~127u);
constexpr int XPLANE = TH * XP, YPLANE = TH * TW;
}  // namespace fwdfast7

template <int NROWS>
__device__ __forceinline__ void sweep_rows7(const float* __restrict__ xa, const float* __restrict__ xb,
                                            const float* __restrict__ y0, float2 (&acc)[fwdfast7::JT][7]) {
  using namespace fwdfast7;
#pragma unroll 1
  for (int u = 0; u < NROWS; ++u, xa += XP, xb += XP, y0 += TW) {
    // window columns -4 .. +7 around this lane's quad for both x channels (columns -3 .. +6 are used)
    float wa[12], wb[12];
#pragma unroll
    for (int v = 0; v < 3; ++v) {
      const float4 a = *reinterpret_cast<const float4*>(xa + 4 * (v - 1));
      const float4 b = *reinterpret_cast<const float4*>(xb + 4 * (v - 1));
      wa[4 * v] = a.x; wa[4 * v + 1] = a.y; wa[4 * v + 2] = a.z; wa[4 * v + 3] = a.w;
      wb[4 * v] = b.x; wb[4 * v + 1] = b.y; wb[4 * v + 2] = b.z; wb[4 * v + 3] = b.w;
    }
    float4 yv[JT];
#pragma unroll
    for (int jj = 0; jj < JT; ++jj) yv[jj] = *reinterpret_cast<const float4*>(y0 + jj * YPLANE);
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int dx = 0; dx < 7; ++dx) {
        const float2 xp = make_float2(wa[1 + p + dx], wb[1 + p + dx]);      // column 4q + p + dx - 3
#pragma unroll
        for (int jj = 0; jj < JT; ++jj) {
          const float yy = (&yv[jj].x)[p];
          acc[jj][dx] = __ffma2_rn(xp, make_float2(yy, yy), acc[jj][dx]);
        }
      }
  }
}

__global__ void __launch_bounds__(fwdfast7::NTHREADS, 1)
local_joint_fast7_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy,
                         const FwdFastParams P) {
  using namespace fwdfast7;
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  __shared__ float red[NCONS][JT * 7 * 2];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = P.B * P.tiles_h * P.tiles_w;
  const int nblk = P.K / KB;
  const int pair = (int)blockIdx.y / T, dy = (int)blockIdx.y % T;
  const int i_off = (pair / nblk) * KB, j_off = (pair % nblk) * KB;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], NCONS);
    }
    mbar_fence_init();
  }
  __syncthreads();

  auto issue = [&](int k) {          // stage the k-th work item of this CTA (if there is one)
    const int it = blockIdx.x + k * gridDim.x;
    if (it >= items) return;
    const int s = k % STAGES;
    const int n = it / (P.tiles_h * P.tiles_w);
    const int tt = it - n * (P.tiles_h * P.tiles_w);
    const int th0 = (tt / P.tiles_w) * TH, tw0 = (tt % P.tiles_w) * TW;
    unsigned char* base = smem_raw + (size_t)s * STAGE_BYTES;
    mbar_arrive_expect_tx(&full_bar[s], X_BYTES + Y_BYTES);
    tma_load_4d(base, &mapx, &full_bar[s], tw0 - LP, th0 + dy - PAD, i_off, n);   // x rows shifted by dy - pad
    tma_load_4d(base + X_REGION, &mapy, &full_bar[s], tw0, th0, j_off, n);
  };
  const bool producer = (wid == PRODUCER_WARP && lane == 0);
  if (producer) {
    tma_prefetch_desc(&mapx);
    tma_prefetch_desc(&mapy);
    for (int k = 0; k < STAGES; ++k) issue(k);
  }
  {
    const int job = wid < NJOBS ? wid : wid - NJOBS;
    const bool split = job < NHELP;                    // this job's band rows are shared with a helper warp
    const int r0 = (wid >= NJOBS) ? RB / 2 : 0;
    const int ip = job / (KB / JT), jg = job % (KB / JT);
    const int band = lane >> 3, quad = lane & 7;
    const int xoff = (2 * ip) * XPLANE + (band * RB + r0) * XP + LP + 4 * quad;
    const int yoff = (jg * JT) * YPLANE + (band * RB + r0) * TW + 4 * quad;

    float2 acc[JT][7];
#pragma unroll
    for (int jj = 0; jj < JT; ++jj)
#pragma unroll
      for (int dx = 0; dx < 7; ++dx) acc[jj][dx] = make_float2(0.f, 0.f);

    int k = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++k) {
      const int s = k % STAGES;
      const unsigned use = (unsigned)(k / STAGES);
      if (producer && k >= 1) {
        mbar_wait(&empty_bar[(k - 1) % STAGES], ((unsigned)((k - 1) / STAGES)) & 1u);
        issue(k - 1 + STAGES);
      }
      __syncwarp();
      mbar_wait(&full_bar[s], use & 1u);
      const float* xs = reinterpret_cast<const float*>(smem_raw + (size_t)s * STAGE_BYTES) + xoff;
      const float* ys = reinterpret_cast<const float*>(smem_raw + (size_t)s * STAGE_BYTES + X_REGION) + yoff;
      if (split) sweep_rows7<RB / 2>(xs, xs + XPLANE, ys, acc);
      else       sweep_rows7<RB>(xs, xs + XPLANE, ys, acc);
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);
    }

    int a = 0;
#pragma unroll
    for (int jj = 0; jj < JT; ++jj)
#pragma unroll
      for (int dx = 0; dx < 7; ++dx) {
        const float v0 = warp_sum(acc[jj][dx].x);
        const float v1 = warp_sum(acc[jj][dx].y);
        if (lane == (a & 31)) {
          red[wid][2 * a] = v0;
          red[wid][2 * a + 1] = v1;
        }
        ++a;
      }
  }
  __syncthreads();
  // this CTA's partial block: slot[dy * 7 + dx][i_off + i][j_off + j]
  float* slot = P.partial + (size_t)blockIdx.x * (T * T * P.K * P.K);
  for (int e = threadIdx.x; e < NJOBS * JT * 7 * 2; e += blockDim.x) {
    const int job = e / (JT * 7 * 2), r = e - job * (JT * 7 * 2);
    const int a = r >> 1, half = r & 1;
    const int jj = a / 7, dx = a - jj * 7;
    const int ip = job / (KB / JT), jg = job % (KB / JT);
    float v = red[job][r];
    if (job < NHELP) v += red[NJOBS + job][r];
    slot[((size_t)(dy * T + dx) * P.K + (i_off + 2 * ip + half)) * P.K + (j_off + jg * JT + jj)] = v;
  }
}

// 7 x 7 counterpart of local_joint_fast_try (probability inputs only)
int local_joint_fast7_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st) {
  using namespace fwdfast7;
  const int B = m.B, K = m.K, H = m.H, W = m.W;
  if (m.pad != PAD || K < KB || K % KB != 0 || K > 20) return -1;
  if (W % 4 != 0) return -1;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, XP, TH, KB)) return -1;
  if (!make_map_4d(&my, m.y, m, TW, TH, KB)) return -1;
  FwdFastParams P;
  P.B = B; P.K = K; P.H = H; P.W = W;
  P.flags = nullptr; P.inv_temp = 1.f;
  P.tiles_h = (H + TH - 1) / TH;
  P.tiles_w = (W + TW - 1) / TW;
  P.partial = partial;
  const int nblk = K / KB, ny = nblk * nblk * T;
  long long items = (long long)B * P.tiles_h * P.tiles_w;
  int gx = max_ctas / ny;
  if (gx < 1) gx = 1;
  if (gx > items) gx = (int)items;
  *slots = SlotInfo{SLOT_STD, gx, (long long)T * T * K * K, 0};
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_joint_fast7_kernel), (int)((int)(STAGES * STAGE_BYTES))));
  local_joint_fast7_kernel<<<dim3(gx, ny), NTHREADS, STAGES * STAGE_BYTES, st>>>(mx, my, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic
