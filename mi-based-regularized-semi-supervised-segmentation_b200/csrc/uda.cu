// UDA consistency term and the simplex assertion: one-pass streaming kernels (HBM-bound).
//   MSE : torch.nn.MSELoss() as built at semi_seg/trainer.py:137,194
//   KL  : dc2:deepclustering2/loss/kl_losses.py:107-126 (KL_div.forward, reduction="mean")
//   call site: semi_seg/epocher.py:221-224 -- criterion(softmax(tf_logits), softmax(logits_tf).detach())
//   simplex: dc2:deepclustering2/utils/assertion.py:56-65
// A thread owns one pixel (o, i) and walks its C channels (stride `inner`), so a warp reads 32
// consecutive floats per channel: fully coalesced.  With from_logits the two channel softmaxes of
// epocher.py:222-223 are computed in registers and never touch HBM.
#include "common.cuh"
#include "pixel_common.cuh"

namespace iic {

// ---- simplex ---------------------------------------------------------------------------------------
__global__ void simplex_kernel(const float* __restrict__ t, long long outer, int C, long long inner,
                               long long s_outer, long long s_c, int* __restrict__ flags) {
  const long long total = outer * inner;
  bool bad = false;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    const long long o = p / inner, i = p - o * inner;
    const float* src = t + o * s_outer + i;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += __ldg(src + (long long)c * s_c);
    // torch.allclose(sum, 1, rtol=1e-4, atol=1e-4): |sum - 1| <= 1e-4 + 1e-4 * 1 ; NaN fails
    if (!(fabsf(s - 1.f) <= 1e-4f + 1e-4f * 1.f)) bad = true;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, IIC_FLAG_NOT_SIMPLEX);
}

// ---- UDA -------------------------------------------------------------------------------------------
constexpr int UDA_CMAX = 8;      // channels kept in registers; more channels re-read (L1/L2)

struct UdaWorkspace {
  unsigned int ticket;
  unsigned int pad_;
  // followed by double partial[gridDim.x]
};

template <bool FROM_LOGITS>
__device__ __forceinline__ void load_pixel(const float* __restrict__ src, long long inner, int C,
                                           float (&v)[UDA_CMAX]) {
#pragma unroll
  for (int c = 0; c < UDA_CMAX; ++c) v[c] = c < C ? __ldg(src + (long long)c * inner) : (FROM_LOGITS ? -INFINITY : 0.f);
  if (FROM_LOGITS) {
    float mx = v[0];
#pragma unroll
    for (int c = 1; c < UDA_CMAX; ++c) mx = fmaxf(mx, v[c]);
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < UDA_CMAX; ++c) { v[c] = c < C ? __expf(v[c] - mx) : 0.f; s += v[c]; }
    const float inv = 1.f / s;
#pragma unroll
    for (int c = 0; c < UDA_CMAX; ++c) v[c] *= inv;
  }
}

// kind 0: sum_c (p-t)^2 ; kind 1: sum_c -t*log((p+eps)/(t+eps))*w_c   (per pixel)
template <bool FROM_LOGITS>
__global__ void __launch_bounds__(256) uda_fwd_kernel(const float* __restrict__ prob,
                                                      const float* __restrict__ target, long long outer,
                                                      int C, long long inner, int kind, float eps,
                                                      const float* __restrict__ weight, double denom,
                                                      float* __restrict__ loss_out, int* __restrict__ flags,
                                                      int check_simplex, UdaWorkspace* ws) {
  __shared__ double scratch[40];
  __shared__ bool is_last;
  double* partial = reinterpret_cast<double*>(ws + 1);
  const long long total = outer * inner;
  float w[UDA_CMAX];
#pragma unroll
  for (int c = 0; c < UDA_CMAX; ++c) w[c] = (weight && c < C) ? __ldg(weight + c) : 1.f;
  float local = 0.f;
  bool bad = false;
  for (long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x; px < total;
       px += (long long)gridDim.x * blockDim.x) {
    const long long o = px / inner, i = px - o * inner;
    const long long base = o * C * inner + i;
    float p[UDA_CMAX], t[UDA_CMAX];
    load_pixel<FROM_LOGITS>(prob + base, inner, C, p);
    load_pixel<FROM_LOGITS>(target + base, inner, C, t);
    float sp = 0.f, st = 0.f, v = 0.f;
#pragma unroll
    for (int c = 0; c < UDA_CMAX; ++c) {
      if (c < C) {
        sp += p[c]; st += t[c];
        if (kind == 0) { const float d = p[c] - t[c]; v = fmaf(d, d, v); }
        else v += -t[c] * logf((p[c] + eps) / (t[c] + eps)) * w[c];
      }
    }
    if (check_simplex && !FROM_LOGITS) {
      if (!(fabsf(sp - 1.f) <= 2e-4f) || !(fabsf(st - 1.f) <= 2e-4f)) bad = true;
    }
    local += v;
  }
  if (check_simplex && __any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0)
    atomicOr(flags, IIC_FLAG_NOT_SIMPLEX);
  const double bsum = block_sum((double)local, scratch);
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = bsum;
    __threadfence();
    is_last = (atomicAdd(&ws->ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    const volatile double* pp = partial;
    double tot = 0.0;
    for (unsigned int b = 0; b < gridDim.x; ++b) tot += pp[b];
    tot /= denom;
    loss_out[0] = (float)tot;
    if (tot != tot) atomicOr(flags, IIC_FLAG_NAN_LOSS);
    ws->ticket = 0;
  }
}

template <bool FROM_LOGITS>
__global__ void __launch_bounds__(256) uda_bwd_kernel(const float* __restrict__ prob,
                                                      const float* __restrict__ target, long long outer,
                                                      int C, long long inner, int kind, float eps,
                                                      const float* __restrict__ weight, float inv_denom,
                                                      const float* __restrict__ grad_loss,
                                                      float* __restrict__ grad_prob) {
  const long long total = outer * inner;
  const float g = (grad_loss ? __ldg(grad_loss) : 1.f) * inv_denom;
  float w[UDA_CMAX];
#pragma unroll
  for (int c = 0; c < UDA_CMAX; ++c) w[c] = (weight && c < C) ? __ldg(weight + c) : 1.f;
  for (long long px = (long long)blockIdx.x * blockDim.x + threadIdx.x; px < total;
       px += (long long)gridDim.x * blockDim.x) {
    const long long o = px / inner, i = px - o * inner;
    const long long base = o * C * inner + i;
    float p[UDA_CMAX], t[UDA_CMAX], gp[UDA_CMAX];
    load_pixel<FROM_LOGITS>(prob + base, inner, C, p);
    load_pixel<FROM_LOGITS>(target + base, inner, C, t);
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < UDA_CMAX; ++c) {
      gp[c] = 0.f;
      if (c < C) {
        gp[c] = (kind == 0) ? 2.f * (p[c] - t[c]) * g : -t[c] / (p[c] + eps) * w[c] * g;
        dot = fmaf(gp[c], p[c], dot);
      }
    }
#pragma unroll
    for (int c = 0; c < UDA_CMAX; ++c) {
      if (c < C) {
        const float out = FROM_LOGITS ? p[c] * (gp[c] - dot) : gp[c];   // softmax adjoint
        grad_prob[base + (long long)c * inner] = out;
      }
    }
  }
}


// ---- vectorised UDA path: 4 consecutive pixels per thread, 16-byte loads/stores --------------------------
// (inner % 4 == 0, 16-byte aligned bases, outer*inner/4 < 2^31).  The maps are streamed exactly once per
// pass: forward reads 2*C floats per pixel, backward reads 2*C and writes C.
template <bool FROM_LOGITS, int C>
__device__ __forceinline__ void load_quad(const float* __restrict__ src, long long inner, float (&v)[C][4]) {
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(src + (long long)c * inner));
    v[c][0] = t.x; v[c][1] = t.y; v[c][2] = t.z; v[c][3] = t.w;
  }
  if (FROM_LOGITS) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float mx = v[0][e];
#pragma unroll
      for (int c = 1; c < C; ++c) mx = fmaxf(mx, v[c][e]);
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) { v[c][e] = __expf(v[c][e] - mx); s += v[c][e]; }
      const float inv = 1.f / s;
#pragma unroll
      for (int c = 0; c < C; ++c) v[c][e] *= inv;
    }
  }
}

template <bool FROM_LOGITS, int C>
__global__ void __launch_bounds__(256) uda_fwd_vec_kernel(const float* __restrict__ prob,
                                                          const float* __restrict__ target, unsigned nquads,
                                                          unsigned inner4, int kind, float eps,
                                                          const float* __restrict__ weight, double denom,
                                                          float* __restrict__ loss_out, int* __restrict__ flags,
                                                          int check_simplex, UdaWorkspace* ws) {
  __shared__ double scratch[40];
  __shared__ bool is_last;
  double* partial = reinterpret_cast<double*>(ws + 1);
  const long long inner = 4ll * inner4;
  float w[C];
#pragma unroll
  for (int c = 0; c < C; ++c) w[c] = weight ? __ldg(weight + c) : 1.f;
  float local = 0.f;
  bool bad = false;
  for (unsigned idx = blockIdx.x * blockDim.x + threadIdx.x; idx < nquads; idx += gridDim.x * blockDim.x) {
    const unsigned o = idx / inner4, q = idx - o * inner4;
    const long long base = (long long)o * C * inner + 4ll * q;
    float p[C][4], t[C][4];
    load_quad<FROM_LOGITS, C>(prob + base, inner, p);
    load_quad<FROM_LOGITS, C>(target + base, inner, t);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float sp = 0.f, st = 0.f, v = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        sp += p[c][e]; st += t[c][e];
        if (kind == 0) { const float d = p[c][e] - t[c][e]; v = fmaf(d, d, v); }
        else v += -t[c][e] * logf((p[c][e] + eps) / (t[c][e] + eps)) * w[c];
      }
      if (check_simplex && !FROM_LOGITS) {
        if (!(fabsf(sp - 1.f) <= 2e-4f) || !(fabsf(st - 1.f) <= 2e-4f)) bad = true;
      }
      local += v;
    }
  }
  if (check_simplex && __any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0)
    atomicOr(flags, IIC_FLAG_NOT_SIMPLEX);
  const double bsum = block_sum((double)local, scratch);
  if (threadIdx.x == 0) {
    partial[blockIdx.x] = bsum;
    __threadfence();
    is_last = (atomicAdd(&ws->ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) {
    // the last CTA adds the per-CTA sums: thread t takes partial[t], partial[t+256], ... in order, then a
    // fixed-shape block reduction -> deterministic
    __threadfence();
    const volatile double* pp = partial;
    double tsum = 0.0;
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) tsum += pp[b];
    double tot = block_sum(tsum, scratch);
    if (threadIdx.x == 0) {
      tot /= denom;
      loss_out[0] = (float)tot;
      if (tot != tot) atomicOr(flags, IIC_FLAG_NAN_LOSS);
      ws->ticket = 0;
    }
  }
}

template <bool FROM_LOGITS, int C>
__global__ void __launch_bounds__(256) uda_bwd_vec_kernel(const float* __restrict__ prob,
                                                          const float* __restrict__ target, unsigned nquads,
                                                          unsigned inner4, int kind, float eps,
                                                          const float* __restrict__ weight, float inv_denom,
                                                          const float* __restrict__ grad_loss,
                                                          float* __restrict__ grad_prob) {
  const long long inner = 4ll * inner4;
  const float g = (grad_loss ? __ldg(grad_loss) : 1.f) * inv_denom;
  float w[C];
#pragma unroll
  for (int c = 0; c < C; ++c) w[c] = weight ? __ldg(weight + c) : 1.f;
  for (unsigned idx = blockIdx.x * blockDim.x + threadIdx.x; idx < nquads; idx += gridDim.x * blockDim.x) {
    const unsigned o = idx / inner4, q = idx - o * inner4;
    const long long base = (long long)o * C * inner + 4ll * q;
    float p[C][4], t[C][4];
    load_quad<FROM_LOGITS, C>(prob + base, inner, p);
    load_quad<FROM_LOGITS, C>(target + base, inner, t);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float gp = (kind == 0) ? 2.f * (p[c][e] - t[c][e]) * g : -t[c][e] / (p[c][e] + eps) * w[c] * g;
        dot = fmaf(gp, p[c][e], dot);
        t[c][e] = gp;                      // reuse as the gradient w.r.t. the probabilities
      }
      if (FROM_LOGITS) {
#pragma unroll
        for (int c = 0; c < C; ++c) t[c][e] = p[c][e] * (t[c][e] - dot);   // softmax adjoint
      }
    }
#pragma unroll
    for (int c = 0; c < C; ++c)
      *reinterpret_cast<float4*>(grad_prob + base + (long long)c * inner) =
          make_float4(t[c][0], t[c][1], t[c][2], t[c][3]);
  }
}

// ---- wide-class UDA path (9 <= C <= 256): the channels of a pixel spread over the 8 warps of a CTA -------------------
// (pixel_common.cuh).  A tile is 32 consecutive pixel groups of the flattened outer*inner map (V = 4 needs
// inner % 4 == 0, so a group never straddles two samples); a 1-D grid of at most 8 CTAs per SM walks the tiles.  Each
// input byte is read once per pass; the softmaxes, the simplex sums and the adjoint's dot are merged in shared memory.
template <int V, int CW, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, CW >= 32 ? 1 : 2) uda_fwd_wide_kernel(const float* __restrict__ prob,
                                                           const float* __restrict__ target, long long outer, int C,
                                                           long long inner, int kind, float eps,
                                                           const float* __restrict__ weight, double denom,
                                                           float* __restrict__ loss_out, int* __restrict__ flags,
                                                           int check_simplex, UdaWorkspace* ws) {
  __shared__ float2 red_p[2][WIDE_WARPS * 32 * V], red_t[2][WIDE_WARPS * 32 * V];
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  float wt[CW];
#pragma unroll
  for (int j = 0; j < CW; ++j) wt[j] = (weight && c0 + j < C) ? __ldg(weight + c0 + j) : 1.f;
  const long long ngroups = outer * inner / V, ntiles = (ngroups + 31) / 32;
  double local = 0.0;
  bool bad = false;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane, px = q * V;
    const bool live = q < ngroups;
    const long long o = px / inner, base = o * C * inner + (px - o * inner);
    float p[CW][V], t[CW][V];
    wide_load<V, CW>(prob + base, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, p);
    wide_load<V, CW>(target + base, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, t);
    if (FROM_LOGITS) {
      int arg[V];
      wide_softmax<V, CW>(p, c0, red_p[it], nullptr, arg);
      wide_softmax<V, CW>(t, c0, red_t[it], nullptr, arg);
    }
    float sp[V], st[V];
#pragma unroll
    for (int e = 0; e < V; ++e) {
      float v = 0.f;
      sp[e] = 0.f; st[e] = 0.f;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        if (c0 + j < C) {
          sp[e] += p[j][e]; st[e] += t[j][e];
          if (kind == 0) { const float d = p[j][e] - t[j][e]; v = fmaf(d, d, v); }
          else v += -t[j][e] * logf((p[j][e] + eps) / (t[j][e] + eps)) * wt[j];
        }
      }
      if (live) local += v;
    }
    if (check_simplex && !FROM_LOGITS) {
      float2* red = red_p[it];
#pragma unroll
      for (int e = 0; e < V; ++e) red[(threadIdx.x >> 5) * 32 * V + lane * V + e] = make_float2(sp[e], st[e]);
      __syncthreads();
#pragma unroll
      for (int e = 0; e < V; ++e) {
        float2 s = red[lane * V + e];
#pragma unroll
        for (int w = 1; w < WIDE_WARPS; ++w) { s.x += red[w * 32 * V + lane * V + e].x; s.y += red[w * 32 * V + lane * V + e].y; }
        if (live && (!(fabsf(s.x - 1.f) <= 2e-4f) || !(fabsf(s.y - 1.f) <= 2e-4f))) bad = true;
      }
    }
  }
  if (check_simplex && __any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flags, IIC_FLAG_NOT_SIMPLEX);
  wide_loss_combine(local, denom, &ws->ticket, reinterpret_cast<double*>(ws + 1), loss_out, flags);
}

template <int V, int CW, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, CW >= 32 ? 1 : 2) uda_bwd_wide_kernel(const float* __restrict__ prob,
                                                           const float* __restrict__ target, long long outer, int C,
                                                           long long inner, int kind, float eps,
                                                           const float* __restrict__ weight, float inv_denom,
                                                           const float* __restrict__ grad_loss,
                                                           float* __restrict__ grad_prob) {
  __shared__ float2 red_p[2][WIDE_WARPS * 32 * V], red_t[2][WIDE_WARPS * 32 * V];
  __shared__ float red_d[2][WIDE_WARPS * 32 * V];
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  const float g = (grad_loss ? __ldg(grad_loss) : 1.f) * inv_denom;
  float wt[CW];
#pragma unroll
  for (int j = 0; j < CW; ++j) wt[j] = (weight && c0 + j < C) ? __ldg(weight + c0 + j) : 1.f;
  const long long ngroups = outer * inner / V, ntiles = (ngroups + 31) / 32;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane, px = q * V;
    const bool live = q < ngroups;
    const long long o = px / inner, base = o * C * inner + (px - o * inner);
    float p[CW][V], t[CW][V];
    wide_load<V, CW>(prob + base, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, p);
    wide_load<V, CW>(target + base, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, t);
    if (FROM_LOGITS) {
      int arg[V];
      wide_softmax<V, CW>(p, c0, red_p[it], nullptr, arg);
      wide_softmax<V, CW>(t, c0, red_t[it], nullptr, arg);
    }
#pragma unroll
    for (int e = 0; e < V; ++e) {
      float dot = 0.f;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        float gp = 0.f;
        if (c0 + j < C) {
          gp = (kind == 0) ? 2.f * (p[j][e] - t[j][e]) * g : -t[j][e] / (p[j][e] + eps) * wt[j] * g;
          dot = fmaf(gp, p[j][e], dot);
        }
        t[j][e] = gp;                      // reuse as the gradient w.r.t. the probabilities
      }
      if (FROM_LOGITS) red_d[it][(threadIdx.x >> 5) * 32 * V + lane * V + e] = dot;
    }
    if (FROM_LOGITS) {
      __syncthreads();
#pragma unroll
      for (int e = 0; e < V; ++e) {
        const float dot = wide_warp_sum<V>(red_d[it], lane * V + e);
#pragma unroll
        for (int j = 0; j < CW; ++j) t[j][e] = p[j][e] * (t[j][e] - dot);   // softmax adjoint
      }
    }
    wide_store<V, CW>(grad_prob + base, inner, c0, C, live, t);
  }
}

static bool uda_vec_ok(const void* a, const void* b, const void* c, long long outer, int C, long long inner) {
  if (C < 2 || C > 4) return false;
  if (inner % 4 != 0) return false;
  if ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) return false;
  return outer * (inner / 4) < (1ll << 31);
}

static int uda_grid(long long total) {
  int sms = sm_count_cached(current_device());
  if (sms <= 0) sms = 148;
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)sms * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

}  // namespace iic

using namespace iic;


extern "C" int iic_simplex_check(const float* t, long long outer, int C, long long inner,
                                 long long s_outer, long long s_c, int* flags, void* stream) {
  IIC_REQUIRE(t && flags, "iic_simplex_check: null pointer");
  IIC_REQUIRE(outer > 0 && C > 0 && inner > 0, "iic_simplex_check: empty tensor");
  const int grid = uda_grid(outer * inner);
  simplex_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(t, outer, C, inner, s_outer, s_c, flags);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" size_t iic_uda_workspace_bytes(int device) {
  int sms = sm_count_cached(device);
  if (sms <= 0) sms = 148;
  return sizeof(UdaWorkspace) + (size_t)sms * 8 * sizeof(double);
}

extern "C" int iic_uda_forward(const float* prob, const float* target, long long outer, int C,
                               long long inner, int kind, double eps, const float* weight,
                               int from_logits, float* loss_out, int* flags, int check_simplex,
                               void* workspace, void* stream) {
  IIC_REQUIRE(prob && target && loss_out && flags && workspace, "iic_uda_forward: null pointer");
  IIC_REQUIRE(outer > 0 && C > 0 && inner > 0, "iic_uda_forward: empty tensor");
  IIC_REQUIRE(C <= WIDE_CMAX, "iic_uda_forward: C=%d > %d channels unsupported", C, WIDE_CMAX);
  IIC_REQUIRE(kind == 0 || kind == 1, "iic_uda_forward: kind must be 0 (mse) or 1 (kl)");
  const long long total = outer * inner;
  const int grid = uda_grid(total);
  // MSELoss: mean over all elements; KL_div "mean": mean over outer*inner after the channel sum
  const double denom = kind == 0 ? (double)total * C : (double)total;
  cudaStream_t st = (cudaStream_t)stream;
  if (C > UDA_CMAX) {
    const bool vec = wide_vec_ok(prob, target, prob, inner);
    const long long ntiles = (total / (vec ? 4 : 1) + 31) / 32;
#define IIC_UDA_FWD_WIDE(VV, CW)                                                                                  \
    do {                                                                                                          \
      const auto kern = from_logits ? uda_fwd_wide_kernel<VV, CW, true> : uda_fwd_wide_kernel<VV, CW, false>;     \
      kern<<<wide_grid(kern, ntiles), 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, \
                                                                   weight, denom, loss_out, flags, check_simplex,   \
                                                                   (UdaWorkspace*)workspace);                       \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_UDA_FWD_WIDE);
#undef IIC_UDA_FWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  if (uda_vec_ok(prob, target, prob, outer, C, inner)) {
    const unsigned nquads = (unsigned)(total / 4), inner4 = (unsigned)(inner / 4);
    const int vgrid = uda_grid(total / 4);
#define IIC_UDA_FWD(FL, CC)                                                                                   \
    uda_fwd_vec_kernel<FL, CC><<<vgrid, 256, 0, st>>>(prob, target, nquads, inner4, kind, (float)eps, weight, \
                                                      denom, loss_out, flags, check_simplex, (UdaWorkspace*)workspace)
    if (from_logits) { if (C == 2) IIC_UDA_FWD(true, 2); else if (C == 3) IIC_UDA_FWD(true, 3); else IIC_UDA_FWD(true, 4); }
    else             { if (C == 2) IIC_UDA_FWD(false, 2); else if (C == 3) IIC_UDA_FWD(false, 3); else IIC_UDA_FWD(false, 4); }
#undef IIC_UDA_FWD
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  if (from_logits)
    uda_fwd_kernel<true><<<grid, 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, weight, denom,
                                               loss_out, flags, check_simplex, (UdaWorkspace*)workspace);
  else
    uda_fwd_kernel<false><<<grid, 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, weight, denom,
                                                loss_out, flags, check_simplex, (UdaWorkspace*)workspace);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int iic_uda_backward(const float* prob, const float* target, long long outer, int C,
                                long long inner, int kind, double eps, const float* weight,
                                int from_logits, const float* grad_loss, float* grad_prob, void* stream) {
  IIC_REQUIRE(prob && target && grad_prob, "iic_uda_backward: null pointer");
  IIC_REQUIRE(outer > 0 && C > 0 && inner > 0, "iic_uda_backward: empty tensor");
  IIC_REQUIRE(C <= WIDE_CMAX, "iic_uda_backward: C=%d > %d channels unsupported", C, WIDE_CMAX);
  IIC_REQUIRE(kind == 0 || kind == 1, "iic_uda_backward: kind must be 0 (mse) or 1 (kl)");
  const long long total = outer * inner;
  const int grid = uda_grid(total);
  const float inv_denom = (float)(1.0 / (kind == 0 ? (double)total * C : (double)total));
  cudaStream_t st = (cudaStream_t)stream;
  if (C > UDA_CMAX) {
    const bool vec = wide_vec_ok(prob, target, grad_prob, inner);
    const long long ntiles = (total / (vec ? 4 : 1) + 31) / 32;
#define IIC_UDA_BWD_WIDE(VV, CW)                                                                                  \
    do {                                                                                                          \
      const auto kern = from_logits ? uda_bwd_wide_kernel<VV, CW, true> : uda_bwd_wide_kernel<VV, CW, false>;     \
      kern<<<wide_grid(kern, ntiles), 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, \
                                                                   weight, inv_denom, grad_loss, grad_prob);        \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_UDA_BWD_WIDE);
#undef IIC_UDA_BWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  if (uda_vec_ok(prob, target, grad_prob, outer, C, inner)) {
    const unsigned nquads = (unsigned)(total / 4), inner4 = (unsigned)(inner / 4);
    const int vgrid = uda_grid(total / 4);
#define IIC_UDA_BWD(FL, CC)                                                                                   \
    uda_bwd_vec_kernel<FL, CC><<<vgrid, 256, 0, st>>>(prob, target, nquads, inner4, kind, (float)eps, weight, \
                                                      inv_denom, grad_loss, grad_prob)
    if (from_logits) { if (C == 2) IIC_UDA_BWD(true, 2); else if (C == 3) IIC_UDA_BWD(true, 3); else IIC_UDA_BWD(true, 4); }
    else             { if (C == 2) IIC_UDA_BWD(false, 2); else if (C == 3) IIC_UDA_BWD(false, 3); else IIC_UDA_BWD(false, 4); }
#undef IIC_UDA_BWD
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  if (from_logits)
    uda_bwd_kernel<true><<<grid, 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, weight,
                                               inv_denom, grad_loss, grad_prob);
  else
    uda_bwd_kernel<false><<<grid, 256, 0, st>>>(prob, target, outer, C, inner, kind, (float)eps, weight,
                                                inv_denom, grad_loss, grad_prob);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
