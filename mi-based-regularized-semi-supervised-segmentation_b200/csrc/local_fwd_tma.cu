// Fast path of the local joint (contrastyou/losses/iic_loss.py:120-123) for the common case: one patch
// (patch >= map), no mask, 16-byte aligned rows.  Same output-stationary FMA scheme as local_fwd.cu, plus
//   * TMA: a dedicated producer warp streams the x tile (with halo) and the y tile of the next work item
//     into a 2-stage shared-memory ring with cp.async.bulk.tensor (rank-4 boxes; the hardware zero-fills
//     everything outside the map, which IS the conv's zero padding), signalling full/empty mbarriers;
//   * packed FP32: accumulators are float2 pairs over two x channels (i0, i0+1) and every update is one
//     fma.rn.f32x2 (FFMA2), halving the FMA issue slots so the loads and address math fit beside them.
#include "common.cuh"
#include "local_kernels.cuh"
#include "tma.cuh"

namespace iic {

struct FwdTmaParams {
  int B, K, H, W, pad;
  int TH, TWS;              // tile rows / 32-column strips
  int tiles_h, tiles_w;
  int XR, XP;               // x tile rows and pitch (floats)
  int LP;                   // left halo columns staged (multiple of 4 >= pad: TMA box starts must be 16-B aligned)
  int njobs_j, njobs, rounds;
  int nconsumers;           // consumer warps
  unsigned stage_bytes;     // bytes of one stage (x region + y region, each 128-B aligned)
  unsigned x_bytes, y_bytes, x_region;
  float* partial;           // [gridDim.x][T*T][K][K]
};

constexpr int FWD_STAGES = 2;

template <int T, int JT>
__device__ __forceinline__ void job_tile2(const FwdTmaParams& P, const float* __restrict__ xs,
                                          const float* __restrict__ ys, int i0, int j0,
                                          float2 (&acc)[JT][T][T]) {
  const int lane = threadIdx.x & 31;
  const int TW = P.TWS * 32;
  const int plane = P.XR * P.XP;
  int ca = i0, cb = i0 + 1;
  ca = ca < P.K ? ca : P.K - 1;
  cb = cb < P.K ? cb : P.K - 1;
  const float* xa = xs + (size_t)ca * plane + (P.LP - P.pad);
  const float* xb = xs + (size_t)cb * plane + (P.LP - P.pad);
  const float* yj[JT];
#pragma unroll
  for (int jj = 0; jj < JT; ++jj) {
    int c = j0 + jj; c = c < P.K ? c : P.K - 1;
    yj[jj] = ys + (size_t)c * P.TH * TW;
  }
  for (int s = 0; s < P.TWS; ++s) {
    const int c = s * 32 + lane;
    float2 xw[T][T];
#pragma unroll
    for (int r = 0; r < T - 1; ++r)
#pragma unroll
      for (int dx = 0; dx < T; ++dx) xw[r][dx] = make_float2(xa[r * P.XP + c + dx], xb[r * P.XP + c + dx]);
    for (int u0 = 0; u0 < P.TH; u0 += T) {
#pragma unroll
      for (int r = 0; r < T; ++r) {
        const int u = u0 + r;
        if (u < P.TH) {
          const int off = (u + T - 1) * P.XP + c;
#pragma unroll
          for (int dx = 0; dx < T; ++dx) xw[(r + T - 1) % T][dx] = make_float2(xa[off + dx], xb[off + dx]);
          float2 yv[JT];
#pragma unroll
          for (int jj = 0; jj < JT; ++jj) {
            const float v = yj[jj][u * TW + c];
            yv[jj] = make_float2(v, v);
          }
#pragma unroll
          for (int jj = 0; jj < JT; ++jj)
#pragma unroll
            for (int dy = 0; dy < T; ++dy)
#pragma unroll
              for (int dx = 0; dx < T; ++dx)
                acc[jj][dy][dx] = __ffma2_rn(xw[(r + dy) % T][dx], yv[jj], acc[jj][dy][dx]);
        }
      }
    }
  }
}

template <int T, int JT>
__device__ __forceinline__ void job_flush2(const FwdTmaParams& P, float* slot, int i0, int j0,
                                           float2 (&acc)[JT][T][T], bool accumulate) {
  const int lane = threadIdx.x & 31;
  int a = 0;
#pragma unroll
  for (int jj = 0; jj < JT; ++jj)
#pragma unroll
    for (int dy = 0; dy < T; ++dy)
#pragma unroll
      for (int dx = 0; dx < T; ++dx) {
        const float v0 = warp_sum(acc[jj][dy][dx].x);
        const float v1 = warp_sum(acc[jj][dy][dx].y);
        acc[jj][dy][dx] = make_float2(0.f, 0.f);
        const int j = j0 + jj;
        if (lane == (a & 31) && j < P.K) {
          float* dst = slot + ((size_t)(dy * T + dx) * P.K + i0) * P.K + j;
          if (i0 < P.K) dst[0] = accumulate ? dst[0] + v0 : v0;
          if (i0 + 1 < P.K) dst[P.K] = accumulate ? dst[P.K] + v1 : v1;
        }
        ++a;
      }
}

template <int T, int JT>
__global__ void __launch_bounds__(12 * 32, 1)
local_joint_tma_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy,
                       const FwdTmaParams P) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[FWD_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[FWD_STAGES];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = P.B * P.tiles_h * P.tiles_w;
  const int TW = P.TWS * 32;
  float* slot = P.partial + (size_t)blockIdx.x * ((size_t)T * T * P.K * P.K);

  if (threadIdx.x == 0) {
    for (int s = 0; s < FWD_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], P.nconsumers);
    }
    mbar_fence_init();
  }
  __syncthreads();

  if (wid == P.nconsumers) {
    // ===== TMA producer warp =====
    if (lane == 0) {
      tma_prefetch_desc(&mapx);
      tma_prefetch_desc(&mapy);
      int k = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x, ++k) {
        const int s = k % FWD_STAGES;
        const unsigned use = (unsigned)(k / FWD_STAGES);
        mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
        const int n = it / (P.tiles_h * P.tiles_w);
        const int tt = it - n * (P.tiles_h * P.tiles_w);
        const int th0 = (tt / P.tiles_w) * P.TH, tw0 = (tt % P.tiles_w) * TW;
        unsigned char* base = smem_raw + (size_t)s * P.stage_bytes;
        mbar_arrive_expect_tx(&full_bar[s], P.x_bytes + P.y_bytes);
        tma_load_4d(base, &mapx, &full_bar[s], tw0 - P.LP, th0 - P.pad, 0, n);
        tma_load_4d(base + P.x_region, &mapy, &full_bar[s], tw0, th0, 0, n);
      }
    }
    return;
  }

  // ===== consumer warps =====
  float2 acc[JT][T][T];
#pragma unroll
  for (int jj = 0; jj < JT; ++jj)
#pragma unroll
    for (int dy = 0; dy < T; ++dy)
#pragma unroll
      for (int dx = 0; dx < T; ++dx) acc[jj][dy][dx] = make_float2(0.f, 0.f);

  const bool single_round = (P.rounds == 1);
  bool first_flush = true;
  int k = 0;
  for (int it = blockIdx.x; it < items; it += gridDim.x, ++k) {
    const int s = k % FWD_STAGES;
    const unsigned use = (unsigned)(k / FWD_STAGES);
    mbar_wait(&full_bar[s], use & 1u);
    const float* xs = reinterpret_cast<const float*>(smem_raw + (size_t)s * P.stage_bytes);
    const float* ys = reinterpret_cast<const float*>(smem_raw + (size_t)s * P.stage_bytes + P.x_region);
    if (single_round) {
      if (wid < P.njobs) {
        const int j0 = (wid % P.njobs_j) * JT, i0 = (wid / P.njobs_j) * 2;
        job_tile2<T, JT>(P, xs, ys, i0, j0, acc);
      }
    } else {
      for (int r = 0; r < P.rounds; ++r) {
        const int job = r * P.nconsumers + wid;
        if (job < P.njobs) {
          const int j0 = (job % P.njobs_j) * JT, i0 = (job / P.njobs_j) * 2;
          job_tile2<T, JT>(P, xs, ys, i0, j0, acc);
          job_flush2<T, JT>(P, slot, i0, j0, acc, !first_flush);
        }
      }
      first_flush = false;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
  if (single_round && wid < P.njobs) {
    const int j0 = (wid % P.njobs_j) * JT, i0 = (wid / P.njobs_j) * 2;
    job_flush2<T, JT>(P, slot, i0, j0, acc, false);
  }
}

template <int T, int JT>
static int launch_fwd_tma(const CUtensorMap& mx, const CUtensorMap& my, const FwdTmaParams& P, int grid,
                          size_t smem, cudaStream_t st) {
  auto kern = local_joint_tma_kernel<T, JT>;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(kern), (int)(220 * 1024)));
  kern<<<grid, (P.nconsumers + 1) * 32, smem, st>>>(mx, my, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static int jt_for(int T) { return T == 1 ? 8 : T == 3 ? 5 : T == 5 ? 2 : 1; }

int local_joint_tma_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st) {
  const int B = m.B, K = m.K, H = m.H, W = m.W, pad = m.pad;
  const int T = 2 * pad + 1;
  if (T > 5 || K > 32 || K < 1) return -1;     // T = 7 keeps the generic kernel (register budget)
  if (W % 4 != 0) return -1;
  FwdTmaParams P;
  P.B = B; P.K = K; P.H = H; P.W = W; P.pad = pad;
  // 32-column strips per tile: 2 unless 1 wastes fewer lanes at this width (e.g. 224 = 7 x 32)
  {
    const int w1 = ((W + 31) / 32) * 32, w2 = ((W + 63) / 64) * 64;
    P.TWS = (W > 32 && w2 <= w1) ? 2 : 1;
  }
  const int TW = P.TWS * 32;
  P.LP = (pad + 3) & ~3;
  P.XP = P.LP + TW + ((pad + 3) & ~3);
  auto stage_bytes = [&](int TH, unsigned* xb, unsigned* yb, unsigned* xr) {
    *xb = (unsigned)((size_t)K * (TH + 2 * pad) * P.XP * 4);
    *yb = (unsigned)((size_t)K * TH * TW * 4);
    *xr = (*xb + 127u) & ~127u;
    return *xr + ((*yb + 127u) & ~127u);
  };
  int TH = 32;
  while (TH > 8 && TH / 2 >= H) TH >>= 1;      // small maps: do not stage rows that do not exist
  unsigned xb, yb, xr, sb;
  while (true) {
    sb = stage_bytes(TH, &xb, &yb, &xr);
    if ((size_t)sb * FWD_STAGES <= 200 * 1024 || TH <= 2) break;
    TH >>= 1;
  }
  if ((size_t)sb * FWD_STAGES > 200 * 1024) return -1;
  if (TH + 2 * pad > 256 || P.XP > 256) return -1;
  P.TH = TH; P.XR = TH + 2 * pad;
  P.tiles_h = (H + TH - 1) / TH;
  P.tiles_w = (W + TW - 1) / TW;
  P.stage_bytes = sb; P.x_bytes = xb; P.y_bytes = yb; P.x_region = xr;
  const int JT = jt_for(T);
  P.njobs_j = (K + JT - 1) / JT;
  P.njobs = ((K + 1) / 2) * P.njobs_j;
  int nw = P.njobs;
  if (nw > 11) {                       // 11 consumer warps + the producer warp = 384 threads
    int best = 11; double best_eff = 0.0;
    for (int c = 11; c >= 6; --c) {
      int r = (P.njobs + c - 1) / c;
      double eff = (double)P.njobs / ((double)r * c);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
    }
    nw = best;
  }
  P.nconsumers = nw;
  P.rounds = (P.njobs + nw - 1) / nw;
  P.partial = partial;

  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, P.XP, P.XR, K)) return -1;
  if (!make_map_4d(&my, m.y, m, TW, TH, K)) return -1;

  long long items = (long long)B * P.tiles_h * P.tiles_w;
  int grid = max_ctas;
  if (grid > items) grid = (int)items;
  *slots = SlotInfo{SLOT_STD, grid, (long long)T * T * K * K, 0};
  const size_t smem = (size_t)sb * FWD_STAGES;
  int rc;
  switch (T) {
    case 1: rc = launch_fwd_tma<1, 8>(mx, my, P, grid, smem, st); break;
    case 3: rc = launch_fwd_tma<3, 5>(mx, my, P, grid, smem, st); break;
    default: rc = launch_fwd_tma<5, 2>(mx, my, P, grid, smem, st); break;
  }
  return rc;
}

}  // namespace iic
