// Fast path of the local backward (the convolution_backward of contrastyou/losses/iic_loss.py:123) for
// one patch, no mask, 16-byte aligned rows, small windows.  Both gradients come out of ONE launch:
//   gx[i](px) = sum_{j,taps} Wx[j][tap][i] * y[j](px + tap)      gy[j](px) = sum_{i,taps} Wy[i][tap][j] * x[i](px + tap)
// (Wx/Wy are dL/dJ re-laid by the epilogue).  Per 16 x 128 output tile the CTA runs the two sweeps back to
// back; a producer warp streams the input tiles (with halo, hardware zero fill = the conv's padding) by
// input-channel chunks through a 4-stage TMA/mbarrier ring, so loads of the next chunks (and of the next
// tile) overlap the FMAs of the current one.  A consumer thread owns 2 rows x 4 pixels x all output
// channels as float2 accumulator pairs over adjacent output channels; the warp-uniform weights arrive as
// broadcast 128-bit shared-memory loads that are already (w[c], w[c+1]) pairs, so every update is one
// fma.rn.f32x2 (FFMA2).
#include "common.cuh"
#include "local_kernels.cuh"
#include "tma.cuh"

namespace iic {

constexpr int BT_WARPS = 8;          // consumer warps; each owns 2 output rows
constexpr int BT_ROWS = 2 * BT_WARPS;
constexpr int BT_TW = 128;           // 32 lanes x 4 pixels
constexpr int BT_LP = 4;             // left halo columns in the smem tile (keeps the interior 16-B aligned)
constexpr int BT_XP = BT_LP + BT_TW + 4;
constexpr int BT_STAGES = 4;

struct BwdTmaParams {
  int B, K, Kp, H, W, pad;
  int tiles_h, tiles_w;
  int CB, nchunk;            // input channels per stage, chunks per tensor
  int XR;                    // rows per staged tile
  unsigned stage_bytes, box_bytes;
  const float* Wx;           // [K][T*T][Kp]
  const float* Wy;
  const float* grad_loss;
  float* gx;
  float* gy;
  long long gx_sn, gy_sn;   // sample strides of the gradient tensors in elements
};

template <int T, int OCB>
__global__ void __launch_bounds__(BT_WARPS * 32, 1)
local_bwd_tma_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy,
                     const BwdTmaParams P) {
  constexpr int PAD = T / 2;
  constexpr int T2 = T * T;
  constexpr int OCBP = (OCB + 3) & ~3;
  constexpr int NV = OCBP / 4;
  constexpr int NP = OCB / 2;            // accumulator pairs
  constexpr int WC = 4 + 2 * PAD;        // window columns
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[BT_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[BT_STAGES];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = P.B * P.tiles_h * P.tiles_w;
  const int per_item = 2 * P.nchunk;                       // stages per work item: 2 sweeps x chunks
  const int my_items = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const unsigned total = (unsigned)my_items * per_item;    // stages this CTA runs through
  // weights for both sweeps live after the stage ring: [sweep][K][T2][OCBP]
  float* wsm = reinterpret_cast<float*>(smem_raw + (size_t)BT_STAGES * P.stage_bytes);

  // stage kk -> (work item, sweep, chunk) -> one TMA box into ring slot kk % BT_STAGES
  auto issue = [&](unsigned kk) {
    const int il = kk / per_item, rem = kk - il * per_item;
    const int sweep = rem / P.nchunk, chunk = rem - sweep * P.nchunk;
    const int it = blockIdx.x + il * gridDim.x;
    const int n = it / (P.tiles_h * P.tiles_w);
    const int tt = it - n * (P.tiles_h * P.tiles_w);
    const int th0 = (tt / P.tiles_w) * BT_ROWS, tw0 = (tt % P.tiles_w) * BT_TW;
    const int s = kk % BT_STAGES;
    mbar_arrive_expect_tx(&full_bar[s], P.box_bytes);
    tma_load_4d(smem_raw + (size_t)s * P.stage_bytes, sweep == 0 ? &mapy : &mapx, &full_bar[s], tw0 - BT_LP,
                th0 - PAD, chunk * P.CB, n);                // gx reads y, gy reads x
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < BT_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], BT_WARPS);
    }
    mbar_fence_init();
    tma_prefetch_desc(&mapx);
    tma_prefetch_desc(&mapy);
    for (unsigned kk = 0; kk < BT_STAGES - 1 && kk < total; ++kk) issue(kk);   // prologue: fill the ring
  }
  {
    const float g = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
    const int per = P.K * T2 * OCBP;
    for (int e = threadIdx.x; e < 2 * per; e += blockDim.x) {
      const int sw = e / per, r = e - sw * per;
      const int c = r % OCBP, rest = r / OCBP;          // rest = cin*T2 + tap
      const float* src = sw == 0 ? P.Wx : P.Wy;
      wsm[e] = c < P.Kp ? g * __ldg(src + (size_t)rest * P.Kp + c) : 0.f;
    }
  }
  __syncthreads();

  const int plane = P.XR * BT_XP;
  float2 acc[NP][2][4];
  for (unsigned k = 0; k < total; ++k) {
    // thread 0 keeps the ring full: stage k+STAGES-1 goes into the slot stage k-1 has just vacated
    if (threadIdx.x == 0) {
      const unsigned kk = k + BT_STAGES - 1;
      if (kk < total) {
        if (k >= 1) mbar_wait(&empty_bar[(k - 1) % BT_STAGES], ((k - 1) / BT_STAGES) & 1u);
        issue(kk);
      }
    }
    __syncwarp();
    const int il = k / per_item, rem = k - il * per_item;
    const int sweep = rem / P.nchunk, chunk = rem - sweep * P.nchunk;
    if (chunk == 0) {
#pragma unroll
      for (int c = 0; c < NP; ++c)
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[c][r][q] = make_float2(0.f, 0.f);
    }
    const int s = k % BT_STAGES;
    mbar_wait(&full_bar[s], (k / BT_STAGES) & 1u);
    const float* tile = reinterpret_cast<const float*>(smem_raw + (size_t)s * P.stage_bytes);
    const float* wbase = wsm + (size_t)sweep * P.K * T2 * OCBP;
    const int c0 = chunk * P.CB;
    for (int ch = 0; ch < P.CB; ++ch) {
      const float* tp = tile + (size_t)ch * plane + (2 * wid) * BT_XP + BT_LP + 4 * lane - PAD;
      const float4* wv = reinterpret_cast<const float4*>(wbase + (size_t)(c0 + ch) * T2 * OCBP);
      float win[T + 1][WC];
#pragma unroll
      for (int r = 0; r < T + 1; ++r) {
        const float4 cv = *reinterpret_cast<const float4*>(tp + r * BT_XP + PAD);
        win[r][PAD + 0] = cv.x; win[r][PAD + 1] = cv.y; win[r][PAD + 2] = cv.z; win[r][PAD + 3] = cv.w;
#pragma unroll
        for (int h = 0; h < PAD; ++h) {
          win[r][h] = tp[r * BT_XP + h];
          win[r][PAD + 4 + h] = tp[r * BT_XP + PAD + 4 + h];
        }
      }
#pragma unroll
      for (int ry = 0; ry < T; ++ry) {
#pragma unroll
        for (int rx = 0; rx < T; ++rx) {
          float2 w2[OCBP / 2];
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const float4 t4 = wv[(ry * T + rx) * NV + v];
            w2[2 * v] = make_float2(t4.x, t4.y);
            w2[2 * v + 1] = make_float2(t4.z, t4.w);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 a0 = make_float2(win[ry][q + rx], win[ry][q + rx]);
            const float2 a1 = make_float2(win[ry + 1][q + rx], win[ry + 1][q + rx]);
#pragma unroll
            for (int c = 0; c < NP; ++c) {
              acc[c][0][q] = __ffma2_rn(a0, w2[c], acc[c][0][q]);
              acc[c][1][q] = __ffma2_rn(a1, w2[c], acc[c][1][q]);
            }
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);

    if (chunk == P.nchunk - 1) {
      // ---- store this sweep's gradient tile ----
      const int it = blockIdx.x + il * gridDim.x;
      const int n = it / (P.tiles_h * P.tiles_w);
      const int tt = it - n * (P.tiles_h * P.tiles_w);
      const int row0 = (tt / P.tiles_w) * BT_ROWS + 2 * wid, col0 = (tt % P.tiles_w) * BT_TW + 4 * lane;
      float* out = sweep == 0 ? P.gx + (size_t)n * P.gx_sn : P.gy + (size_t)n * P.gy_sn;
      if (col0 < P.W) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const int row = row0 + r;
          if (row < P.H) {
#pragma unroll
            for (int c = 0; c < NP; ++c) {
              const int oc = 2 * c;
              float* dst = out + ((size_t)oc * P.H + row) * P.W + col0;
              if (oc < P.K)
                *reinterpret_cast<float4*>(dst) = make_float4(acc[c][r][0].x, acc[c][r][1].x, acc[c][r][2].x, acc[c][r][3].x);
              if (oc + 1 < P.K)
                *reinterpret_cast<float4*>(dst + (size_t)P.H * P.W) =
                    make_float4(acc[c][r][0].y, acc[c][r][1].y, acc[c][r][2].y, acc[c][r][3].y);
            }
          }
        }
      }
    }
  }
}

template <int T, int OCB>
static int launch_bwd_tma(const CUtensorMap& mx, const CUtensorMap& my, const BwdTmaParams& P, int grid,
                          size_t smem, cudaStream_t st) {
  auto kern = local_bwd_tma_kernel<T, OCB>;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(kern), (int)(226 * 1024)));
  kern<<<grid, BT_WARPS * 32, smem, st>>>(mx, my, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int local_bwd_tma_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, cudaStream_t st) {
  const int B = m.B, K = m.K, H = m.H, W = m.W, pad = m.pad;
  const int T = 2 * pad + 1;
  if (T > 3 || K > 12 || K < 1) return -1;
  if (W % 4 != 0) return -1;
  if ((reinterpret_cast<uintptr_t>(g.gx) & 15) || (reinterpret_cast<uintptr_t>(g.gy) & 15) || (g.gx_sn & 3) || (g.gy_sn & 3))
    return -1;
  BwdTmaParams P;
  P.B = B; P.K = K; P.Kp = (K + 3) & ~3; P.H = H; P.W = W; P.pad = pad;
  P.tiles_h = (H + BT_ROWS - 1) / BT_ROWS;
  P.tiles_w = (W + BT_TW - 1) / BT_TW;
  P.XR = BT_ROWS + 2 * pad;
  const int ocb = (K + 1) & ~1;                       // even: accumulators are channel pairs
  const int ocbp = (ocb + 3) & ~3;
  const size_t wbytes = (size_t)2 * K * T * T * ocbp * sizeof(float);
  // input channels per stage: the largest divisor of K whose 4-stage ring fits beside the weights
  int CB = 0;
  for (int d = K; d >= 1; --d) {
    if (K % d) continue;
    size_t sb = ((size_t)d * P.XR * BT_XP * 4 + 127) & ~(size_t)127;
    if (sb * BT_STAGES + wbytes <= 224 * 1024) { CB = d; break; }
  }
  if (CB == 0) return -1;
  P.CB = CB; P.nchunk = K / CB;
  P.box_bytes = (unsigned)((size_t)CB * P.XR * BT_XP * 4);
  P.stage_bytes = (P.box_bytes + 127u) & ~127u;
  P.Wx = Wx; P.Wy = Wy; P.grad_loss = g.grad_loss; P.gx = g.gx; P.gy = g.gy; P.gx_sn = g.gx_sn; P.gy_sn = g.gy_sn;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, BT_XP, P.XR, CB)) return -1;
  if (!make_map_4d(&my, m.y, m, BT_XP, P.XR, CB)) return -1;
  long long items = (long long)B * P.tiles_h * P.tiles_w;
  int grid = m.sms;
  if (grid > items) grid = (int)items;
  const size_t smem = (size_t)P.stage_bytes * BT_STAGES + wbytes;
  if (T == 1) {
    switch (ocb) {
      case 2: return launch_bwd_tma<1, 2>(mx, my, P, grid, smem, st);
      case 4: return launch_bwd_tma<1, 4>(mx, my, P, grid, smem, st);
      case 6: return launch_bwd_tma<1, 6>(mx, my, P, grid, smem, st);
      case 8: return launch_bwd_tma<1, 8>(mx, my, P, grid, smem, st);
      case 10: return launch_bwd_tma<1, 10>(mx, my, P, grid, smem, st);
      default: return launch_bwd_tma<1, 12>(mx, my, P, grid, smem, st);
    }
  }
  switch (ocb) {
    case 2: return launch_bwd_tma<3, 2>(mx, my, P, grid, smem, st);
    case 4: return launch_bwd_tma<3, 4>(mx, my, P, grid, smem, st);
    case 6: return launch_bwd_tma<3, 6>(mx, my, P, grid, smem, st);
    case 8: return launch_bwd_tma<3, 8>(mx, my, P, grid, smem, st);
    case 10: return launch_bwd_tma<3, 10>(mx, my, P, grid, smem, st);
    default: return launch_bwd_tma<3, 12>(mx, my, P, grid, smem, st);
  }
}

}  // namespace iic
