// Backward of the local IIC term: both input gradients of the shifted-window joint
//   gx[n,i,a,b] = g * sum_{d,j} GA[d,i,j] * y[n,j,a-dy+pad,b-dx+pad]
//   gy[n,j,u,v] = g * sum_{d,i} GA[d,i,j] * x[n,i,u+dy-pad,v+dx-pad]
// (what autograd's convolution_backward computes for contrastyou/losses/iic_loss.py:123), with the mask
// of :116-118 applied to the staged input and to the result.
//
// With the coefficient tensors re-laid by the epilogue (Wx flipped, Wy straight) both sweeps are the
// same K -> K channel, T x T tap stencil:  out[c](px) = sum_{cin,ry,rx} W[cin][ry*T+rx][c] * in[cin](px + (ry-pad, rx-pad)).
// Mapping: one thread owns PXT consecutive pixels of one row and OCB output channels (acc[OCB][PXT]
// in registers); the T x T taps for all output channels are warp-uniform and come from shared memory
// as broadcast 128-bit loads, so the inner loop is FMA-issue bound.  Input tiles (with halo, zero
// outside the patch) are staged in shared memory by input-channel chunks.
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"

namespace iic {

constexpr int BWD_WARPS = 8;       // tile rows (one warp per row)
constexpr int BWD_PXT = 4;         // pixels per thread along W
constexpr int BWD_TW = 32 * BWD_PXT;

struct LocalBwdParams {
  View4 in;                 // staged input of this sweep (y for gx, x for gy)
  View4 m;                  // optional mask
  float* out;               // (B,K,H,W) gradient, rows and channel planes dense
  long long out_sn;         // its sample stride in elements (K*H*W when the whole tensor is dense)
  const float* W;           // [patch][K][T*T][Kp]
  const float* grad_loss;   // device scalar or nullptr
  int B, K, Kp, H, Wd, pad;
  PatchGrid g;
  int tiles_h, tiles_w;
  int CB;                   // input channels staged per chunk
  int LP;                   // left halo padding in the smem tile (multiple of 4, >= pad)
  int XP;                   // smem pitch
  int accumulate;           // out += (more than one patch)
};

template <int T, int OCB>
__global__ void __launch_bounds__(BWD_WARPS * 32) local_bwd_kernel(const LocalBwdParams P) {
  constexpr int PXT = BWD_PXT;
  constexpr int PAD = T / 2;
  constexpr int OCBP = (OCB + 3) & ~3;     // weight row stride in shared memory
  constexpr int NV = OCBP / 4;             // weight float4s per tap
  extern __shared__ __align__(16) float smem[];
  const int T2 = T * T;
  const int XR = BWD_WARPS + 2 * PAD;
  float* tile = smem;                                    // [CB][XR][XP]
  float* wsm = smem + (size_t)P.CB * XR * P.XP;          // [CB][T2][OCBP]  (this output chunk only)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int patch = blockIdx.y;
  const int ph0 = patch_axis_origin(patch / P.g.nw, P.g.nh, P.g.H, P.g.ph, P.g.sh);
  const int pw0 = patch_axis_origin(patch % P.g.nw, P.g.nw, P.g.W, P.g.pw, P.g.sw);
  const float gscale = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
  const float* Wp = P.W + (size_t)patch * P.K * T2 * P.Kp;
  const int items = P.B * P.tiles_h * P.tiles_w;

  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int n = it / (P.tiles_h * P.tiles_w);
    const int tt = it - n * (P.tiles_h * P.tiles_w);
    const int th0 = (tt / P.tiles_w) * BWD_WARPS, tw0 = (tt % P.tiles_w) * BWD_TW;
    const int row = th0 + wid;            // output row inside the patch
    const int col = tw0 + lane * PXT;     // first output column inside the patch

    for (int oc0 = 0; oc0 < P.K; oc0 += OCB) {
      float acc[OCB][PXT];
#pragma unroll
      for (int c = 0; c < OCB; ++c)
#pragma unroll
        for (int q = 0; q < PXT; ++q) acc[c][q] = 0.f;

      for (int c0 = 0; c0 < P.K; c0 += P.CB) {
        const int cb = P.K - c0 < P.CB ? P.K - c0 : P.CB;
        __syncthreads();
        // ---- stage input chunk (zero outside the patch), masked ----
        for (int r_ = wid; r_ < cb * XR; r_ += BWD_WARPS) {
          const int ch = r_ / XR, r = r_ - ch * XR;
          const int gh = th0 + r - PAD;
          const bool row_ok = gh >= 0 && gh < P.g.ph;
          const float* src = P.in.p + n * P.in.sn + (long long)(c0 + ch) * P.in.sc + (long long)(ph0 + gh) * P.in.sh + pw0;
          const float* msrc = P.m.p ? P.m.p + n * P.m.sn + (long long)(c0 + ch) * P.m.sc + (long long)(ph0 + gh) * P.m.sh + pw0 : nullptr;
          float* dst = tile + (size_t)r_ * P.XP;
          for (int cc = lane; cc < P.XP; cc += 32) {
            const int gw = tw0 + cc - P.LP;
            float v = 0.f;
            if (row_ok && gw >= 0 && gw < P.g.pw) {
              v = __ldg(src + gw);
              if (msrc) v *= __ldg(msrc + gw);
            }
            dst[cc] = v;
          }
        }
        // ---- stage weights for (input chunk, this output chunk), pre-scaled by the upstream grad ----
        for (int e = threadIdx.x; e < cb * T2 * OCBP; e += BWD_WARPS * 32) {
          const int c = e % OCBP, rest = e / OCBP;    // rest = ch*T2 + tap
          const int oc = oc0 + c;
          wsm[e] = oc < P.Kp ? gscale * __ldg(Wp + ((size_t)c0 * T2 + rest) * P.Kp + oc) : 0.f;
        }
        __syncthreads();
        // ---- stencil ----
        for (int ch = 0; ch < cb; ++ch) {
          const float* trow = tile + ((size_t)ch * XR + wid) * P.XP + P.LP + lane * PXT - PAD;
          const float4* wv = reinterpret_cast<const float4*>(wsm + (size_t)ch * T2 * OCBP);
#pragma unroll
          for (int ry = 0; ry < T; ++ry) {
            float win[PXT + 2 * PAD];
            // centre as one 128-bit load, halo columns as scalars
            const float4 cv = *reinterpret_cast<const float4*>(trow + ry * P.XP + PAD);
            win[PAD + 0] = cv.x; win[PAD + 1] = cv.y; win[PAD + 2] = cv.z; win[PAD + 3] = cv.w;
#pragma unroll
            for (int h = 0; h < PAD; ++h) {
              win[h] = trow[ry * P.XP + h];
              win[PAD + PXT + h] = trow[ry * P.XP + PAD + PXT + h];
            }
#pragma unroll
            for (int rx = 0; rx < T; ++rx) {
              float w[OCBP];
#pragma unroll
              for (int v = 0; v < NV; ++v) {
                const float4 t4 = wv[(ry * T + rx) * NV + v];
                w[4 * v + 0] = t4.x; w[4 * v + 1] = t4.y; w[4 * v + 2] = t4.z; w[4 * v + 3] = t4.w;
              }
#pragma unroll
              for (int c = 0; c < OCB; ++c)
#pragma unroll
                for (int q = 0; q < PXT; ++q) acc[c][q] = fmaf(w[c], win[q + rx], acc[c][q]);
            }
          }
        }
      }
      // ---- write this output chunk ----
      if (row < P.g.ph && col < P.g.pw) {
        const int gh = ph0 + row, gw = pw0 + col;
        const bool full = (col + PXT <= P.g.pw);
#pragma unroll
        for (int c = 0; c < OCB; ++c) {
          const int oc = oc0 + c;
          if (oc < P.K) {
            float* dst = P.out + (size_t)n * P.out_sn + ((size_t)oc * P.H + gh) * P.Wd + gw;
            float v[PXT];
#pragma unroll
            for (int q = 0; q < PXT; ++q) v[q] = acc[c][q];
            if (P.m.p) {
              const float* mp = P.m.p + n * P.m.sn + (long long)oc * P.m.sc + (long long)gh * P.m.sh + gw;
#pragma unroll
              for (int q = 0; q < PXT; ++q)
                if (col + q < P.g.pw) v[q] *= __ldg(mp + q);
            }
            const bool vec_ok = full && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
            if (vec_ok && !P.accumulate) {
              *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
              for (int q = 0; q < PXT; ++q)
                if (col + q < P.g.pw) {
                  // overlapping patches are processed concurrently: accumulate with a reduction
                  if (P.accumulate) atomicAdd(dst + q, v[q]);
                  else dst[q] = v[q];
                }
            }
          }
        }
      }
    }
  }
}

template <int T, int OCB>
static int launch_bwd(const LocalBwdParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  auto kern = local_bwd_kernel<T, OCB>;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(kern), (int)(200 * 1024)));
  kern<<<grid, BWD_WARPS * 32, smem, st>>>(P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// wide windows (pad >= 4) are rare (the reference's configs use pad 0, 1, 3): two register blocks only
template <int T>
static int dispatch_ocb_wide(int ocb, const LocalBwdParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  if (ocb <= 8) return launch_bwd<T, 8>(P, grid, smem, st);
  return launch_bwd<T, 16>(P, grid, smem, st);
}

template <int T>
static int dispatch_ocb(int ocb, const LocalBwdParams& P, dim3 grid, size_t smem, cudaStream_t st) {
  switch (ocb) {
    case 4:  return launch_bwd<T, 4>(P, grid, smem, st);
    case 8:  return launch_bwd<T, 8>(P, grid, smem, st);
    case 10: return launch_bwd<T, 10>(P, grid, smem, st);
    case 12: return launch_bwd<T, 12>(P, grid, smem, st);
    case 16: return launch_bwd<T, 16>(P, grid, smem, st);
    default: return launch_bwd<T, 20>(P, grid, smem, st);
  }
}

}  // namespace iic

using namespace iic;

extern "C" int iic_local_backward(const float* x, long long x_sn, long long x_sc, long long x_sh,
                                  const float* y, long long y_sn, long long y_sc, long long y_sh,
                                  const float* mask, long long m_sn, long long m_sc, long long m_sh,
                                  int B, int K, int H, int W, int pad,
                                  int patch_h, int patch_w, int step_h, int step_w,
                                  float* Wx, float* Wy, const float* grad_loss,
                                  float* gx, float* gy, long long gx_sn, long long gy_sn, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (gx_sn <= 0) gx_sn = (long long)K * H * W;          // 0 = the gradient tensor is dense
  if (gy_sn <= 0) gy_sn = (long long)K * H * W;
  IIC_REQUIRE(x && y && Wx && Wy && gx && gy, "iic_local_backward: null pointer");
  IIC_REQUIRE(B > 0 && K > 0, "iic_local_backward: empty batch or channel dimension");
  IIC_REQUIRE(pad >= 0 && pad <= 7, "iic_local_backward: padding %d unsupported (0..7)", pad);
  PatchGrid g;
  IIC_REQUIRE(make_patch_grid(H, W, patch_h, patch_w, step_h, step_w, &g),
              "iic_local_backward: bad patch geometry");
  const int T = 2 * pad + 1, T2 = T * T;
  const int n_patches = g.nh * g.nw;
  const int sms = sm_count_cached(current_device());
  IIC_REQUIRE(sms > 0, "iic_local_backward: no device");

  // fast path: one patch, no mask, TMA-describable rows -> the specialised kernels (local_kernels.cuh)
  if (n_patches == 1 && mask == nullptr && !options().no_tma) {
    const LocalMaps m{{x, x_sn, x_sc, x_sh}, {y, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
    const LocalGrads gr{grad_loss, gx, gy, gx_sn, gy_sn};
    int rc = -1;
    // wide cluster heads (K = 128): tcgen05 3xTF32 sweeps (local_bwd_tc.cu)
    if (!options().no_tc) rc = local_bwd_tc_try(m, Wx, Wy, gr, st);
    // 10 clusters, padding 1 (config 2): row-block tensor-core sweeps with the leftover-slot MMA (local_bwd_tcrb10.cu);
    // fp16-split variant (6 MMAs per source row and tile) by default, tc10_tf32 selects the tf32 + bf16 one (8 MMAs)
    if (rc < 0 && !options().no_tc && !options().no_tc10)
      rc = options().tc10_tf32 ? local_bwd_tcrb10_try(m, Wx, Wy, gr, st) : local_bwd_tcrb10h_try(m, Wx, Wy, gr, 0, 1.f, st);
    // the reference's default cluster count (16 <= K <= 24), padding 1 or 3: row-block tensor-core sweeps
    // (local_bwd_tcrb.cu; at padding 1 only when the map has enough row blocks to fill the SMs, decided inside)
    if (rc < 0 && !options().no_tc) rc = local_bwd_tcrb_try(m, Wx, Wy, gr, st);
    if (rc < 0 && !options().no_fast) rc = local_bwd_fast_try(m, Wx, Wy, gr, 0, 1.f, st);
    if (rc < 0) rc = local_bwd_tma_try(m, Wx, Wy, gr, st);
    if (rc >= 0) return rc;
  }

  LocalBwdParams P;
  P.m = {mask, m_sn, m_sc, m_sh};
  P.grad_loss = grad_loss;
  P.B = B; P.K = K; P.Kp = (K + 3) & ~3; P.H = H; P.Wd = W; P.pad = pad; P.g = g;
  P.tiles_h = (g.ph + BWD_WARPS - 1) / BWD_WARPS;
  P.tiles_w = (g.pw + BWD_TW - 1) / BWD_TW;
  P.LP = (pad + 3) & ~3;
  P.XP = P.LP + BWD_TW + ((pad + 3) & ~3);
  P.accumulate = n_patches > 1 ? 1 : 0;
  // output channels per pass: the smallest supported register block that covers K (<= 20), else 16s
  static const int kOcb[] = {4, 8, 10, 12, 16, 20};
  int ocb = 16;
  if (K <= 20) for (int c : kOcb) if (c >= K) { ocb = c; break; }
  if (pad >= 4) ocb = K <= 8 ? 8 : 16;
  const int ocbp = (ocb + 3) & ~3;
  // input channels per staged chunk: fit tile + weights in ~96 KB
  const int XR = BWD_WARPS + 2 * pad;
  int CB = K;
  while (CB > 1 && (size_t)CB * ((size_t)XR * P.XP + (size_t)T2 * ocbp) * sizeof(float) > 96 * 1024) --CB;
  P.CB = CB;
  const size_t smem = (size_t)CB * ((size_t)XR * P.XP + (size_t)T2 * ocbp) * sizeof(float);
  long long items = (long long)B * P.tiles_h * P.tiles_w;
  long long per = (2LL * sms) / n_patches;
  if (per < 1) per = 1;
  if (per > items) per = items;
  dim3 grid((unsigned)per, n_patches);

  for (int sweep = 0; sweep < 2; ++sweep) {
    if (sweep == 0) { P.in = {y, y_sn, y_sc, y_sh}; P.out = gx; P.out_sn = gx_sn; P.W = Wx; }
    else            { P.in = {x, x_sn, x_sc, x_sh}; P.out = gy; P.out_sn = gy_sn; P.W = Wy; }
    int rc;
    switch (T) {
      case 1:  rc = dispatch_ocb<1>(ocb, P, grid, smem, st); break;
      case 3:  rc = dispatch_ocb<3>(ocb, P, grid, smem, st); break;
      case 5:  rc = dispatch_ocb<5>(ocb, P, grid, smem, st); break;
      case 7:  rc = dispatch_ocb<7>(ocb, P, grid, smem, st); break;
      case 9: rc = dispatch_ocb_wide<9>(ocb, P, grid, smem, st); break;
      case 11: rc = dispatch_ocb_wide<11>(ocb, P, grid, smem, st); break;
      case 13: rc = dispatch_ocb_wide<13>(ocb, P, grid, smem, st); break;
      default: rc = dispatch_ocb_wide<15>(ocb, P, grid, smem, st); break;
    }
    if (rc) return rc;
  }
  return 0;
}

// Backward of iic_local_joint_from_logits: gradients with respect to the two logit maps
extern "C" int iic_local_backward_from_logits(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                              const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                              int B, int K, int H, int W, int pad, float inv_temperature,
                                              const float* Wx, const float* Wy, const float* grad_loss,
                                              float* g_lx, float* g_ly, long long gx_sn, long long gy_sn, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (gx_sn <= 0) gx_sn = (long long)K * H * W;
  if (gy_sn <= 0) gy_sn = (long long)K * H * W;
  IIC_REQUIRE(lx && ly && Wx && Wy && g_lx && g_ly, "iic_local_backward_from_logits: null pointer");
  const int sms = sm_count_cached(current_device());
  IIC_REQUIRE(sms > 0, "iic_local_backward_from_logits: no device");
  const LocalMaps m{{lx, x_sn, x_sc, x_sh}, {ly, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
  const LocalGrads gr{grad_loss, g_lx, g_ly, gx_sn, gy_sn};
  int rc = -1;
  // the fp16-split tensor-core backward has a from-logits form (softmax in its transform warps, adjoint in its drain);
  // same shape rule as for probabilities (enough rows to fill the SMs, or tc10_force)
  if (!options().no_tc && !options().no_tc10 && !options().no_tma)
    rc = local_bwd_tcrb10h_try(m, Wx, Wy, gr, 1, inv_temperature, st);
  if (rc < 0) rc = local_bwd_fast_try(m, Wx, Wy, gr, 1, inv_temperature, st);
  if (rc < 0) {
    set_error("iic_local_backward_from_logits: shape not covered by the fused kernel (needs padding 1, K == 10, "
              "W %% 4 == 0, W <= 248, 16-byte aligned rows)");
    return IIC_UNSUPPORTED;
  }
  return rc;
}

// Backward of iic_local_joint_from_logits_stats: the stats are the ones its forward wrote.  16 <= K <= 24 where
// local_fl_tc_covered holds: row-block tensor-core sweeps on the logits; K = 128 where local_fl_tc128_covered holds: the
// tc sweeps on the logits (both lay their weight images into the tails of Wx / Wy, hence float*); the K = 10 shapes as
// iic_local_backward_from_logits.
extern "C" int iic_local_backward_from_logits_stats(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                                    const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                                    int B, int K, int H, int W, int pad, float inv_temperature,
                                                    const float* stats, float* Wx, float* Wy, const float* grad_loss,
                                                    float* g_lx, float* g_ly, long long gx_sn, long long gy_sn,
                                                    void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(lx && ly && Wx && Wy && g_lx && g_ly, "iic_local_backward_from_logits_stats: null pointer");
  const int sms = sm_count_cached(current_device());
  IIC_REQUIRE(sms > 0, "iic_local_backward_from_logits_stats: no device");
  const LocalMaps m{{lx, x_sn, x_sc, x_sh}, {ly, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
  const bool wide = local_fl_tc128_covered(m);
  if (!wide && !local_fl_tc_covered(m))
    return iic_local_backward_from_logits(lx, x_sn, x_sc, x_sh, ly, y_sn, y_sc, y_sh, B, K, H, W, pad, inv_temperature, Wx,
                                          Wy, grad_loss, g_lx, g_ly, gx_sn, gy_sn, stream);
  IIC_REQUIRE(stats, "iic_local_backward_from_logits_stats: null stats");
  if (gx_sn <= 0) gx_sn = (long long)K * H * W;
  if (gy_sn <= 0) gy_sn = (long long)K * H * W;
  const LocalGrads gr{grad_loss, g_lx, g_ly, gx_sn, gy_sn};
  const int rc = wide ? local_bwd_tc_fl_try(m, stats, inv_temperature, Wx, Wy, gr, st)
                      : local_bwd_tcrb_fl_try(m, stats, inv_temperature, Wx, Wy, gr, st);
  if (rc > 0) return rc;
  IIC_REQUIRE(rc == 0, "iic_local_backward_from_logits_stats: the tensor-core backward refused a covered shape");
  return 0;
}
