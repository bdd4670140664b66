// Per-sample flip alignment as index math (SURVEY.md section 8f row 2).
//   reference: `with FixRandomSeed(seed): torch.stack([self._affine_transformer(x) for x in batch], dim=0)` with
//   TensorRandomFlip(axis=[1, 2], threshold=0.8) -- semi_seg/epocher.py:121,148-149,160-161,264-266;
//   dc2:deepclustering2/augment/tensor_augment.py:17-41 (clone + flip per axis), dc2:decorator/decorator.py:196-212.
// The reference runs B Python-level clone/flip/flip chains and a stack (two passes over the map, ~3B launches).
//   flip_batch_kernel : the whole stack in ONE launch and one pass, per-sample flags (bit 0 = axis 1 = H, bit 1 = axis 2 = W)
//   uda_flip_*_kernel : the UDA consistency term (semi_seg/epocher.py:221-224) reading the teacher logits THROUGH the
//                       flip, so `unlabel_logits_tf` (epocher.py:160-161) is never materialised
// A W flip of a 4-pixel group is the mirrored group with its components reversed, so the 16-byte accesses survive.
#include "common.cuh"
#include "pixel_common.cuh"

namespace iic {

struct FlipWorkspace {
  unsigned int ticket;   // self-resetting arrival counter
  unsigned int pad_;
  // followed by double partial[gridDim.x * gridDim.y]
};

// grid (gx, outer); a thread moves V consecutive pixels of one (channel, row)
template <int V>
__global__ void __launch_bounds__(256) flip_batch_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                         const unsigned char* __restrict__ flips, int C, int H,
                                                         int W) {
  const long long o = blockIdx.y;
  const unsigned f = flips[o];
  const bool fh = f & IIC_FLIP_H, fw = f & IIC_FLIP_W;
  const int wg = W / V;                                  // groups per row
  const long long ngroups = (long long)C * H * wg;
  const float* src = in + o * C * H * W;
  float* dst = out + o * C * H * W;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ngroups;
       q += (long long)gridDim.x * blockDim.x) {
    const long long r = q / wg;                          // channel * H + row
    const int wq = (int)(q - r * wg);
    const long long c = r / H;
    const int h = (int)(r - c * H);
    const int hs = fh ? H - 1 - h : h;
    const int ws = fw ? wg - 1 - wq : wq;
    const float* s = src + (c * H + hs) * W + (long long)ws * V;
    float* d = dst + r * W + (long long)wq * V;
    if (V == 4) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(s));
      *reinterpret_cast<float4*>(d) = fw ? make_float4(t.w, t.z, t.y, t.x) : t;
    } else {
      d[0] = __ldg(s);
    }
  }
}

// pixel offsets (inside one channel plane) of group q of the student and of the teacher seen through the flip
template <int V>
__device__ __forceinline__ void flip_offsets(long long q, int H, int W, bool fh, bool fw, long long* off_s,
                                             long long* off_t) {
  const int wg = W / V;
  const long long h = q / wg;
  const int wq = (int)(q - h * wg);
  const long long hs = fh ? H - 1 - h : h;
  const int ws = fw ? wg - 1 - wq : wq;
  *off_s = h * W + (long long)wq * V;
  *off_t = hs * W + (long long)ws * V;
}

template <int V, int NC>
__device__ __forceinline__ void reverse_group(float (&v)[NC][V]) {
  if (V == 4) {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const float a = v[c][0], b = v[c][1 % V];
      v[c][0] = v[c][3 % V]; v[c][1 % V] = v[c][2 % V]; v[c][2 % V] = b; v[c][3 % V] = a;
    }
  }
}

// kind 0: sum_c (p-t)^2 ; kind 1: sum_c -t*log((p+eps)/(t+eps))   (per pixel; t = target seen through the flip)
template <int V, int NC, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, NC <= 4 ? 3 : 2) uda_flip_fwd_kernel(
    const float* __restrict__ prob, const float* __restrict__ target, const unsigned char* __restrict__ flips,
    int C_rt, int H, int W, int kind, float eps, double denom, float* __restrict__ loss_out,
    int* __restrict__ flags, FlipWorkspace* ws) {
  __shared__ double scratch[40];
  __shared__ bool is_last;
  double* partial = reinterpret_cast<double*>(ws + 1);
  const int C = NC < SUP_CMAX ? NC : C_rt;
  const long long o = blockIdx.y, inner = (long long)H * W;
  const unsigned f = flips[o];
  const bool fh = f & IIC_FLIP_H, fw = f & IIC_FLIP_W;
  const float* pb = prob + o * C * inner;
  const float* tb = target + o * C * inner;
  float local = 0.f;
  const long long ngroups = inner / V;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ngroups;
       q += (long long)gridDim.x * blockDim.x) {
    long long off_s, off_t;
    flip_offsets<V>(q, H, W, fh, fw, &off_s, &off_t);
    float p[NC][V], t[NC][V];
    sup_load<V, NC>(pb + off_s, inner, C, p);
    sup_load<V, NC>(tb + off_t, inner, C, t);
    if (fw) reverse_group<V, NC>(t);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      if (FROM_LOGITS) {
        sup_softmax<V, NC>(p, e);
        sup_softmax<V, NC>(t, e);
      }
      float v = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if (c < C) {
          if (kind == 0) { const float d = p[c][e] - t[c][e]; v = fmaf(d, d, v); }
          else v += -t[c][e] * logf((p[c][e] + eps) / (t[c][e] + eps));
        }
      }
      local += v;
    }
  }
  const double bsum = block_sum((double)local, scratch);
  const unsigned int ncta = gridDim.x * gridDim.y;
  if (threadIdx.x == 0) {
    partial[blockIdx.y * gridDim.x + blockIdx.x] = bsum;
    __threadfence();
    is_last = (atomicAdd(&ws->ticket, 1u) == ncta - 1);
  }
  __syncthreads();
  if (is_last) {
    // fixed-order combine of the per-CTA sums in the last CTA -> deterministic
    __threadfence();
    const volatile double* pp = partial;
    double tsum = 0.0;
    for (unsigned int b = threadIdx.x; b < ncta; b += blockDim.x) tsum += pp[b];
    double tot = block_sum(tsum, scratch);
    if (threadIdx.x == 0) {
      tot /= denom;
      loss_out[0] = (float)tot;
      if (tot != tot) atomicOr(flags, IIC_FLAG_NAN_LOSS);
      ws->ticket = 0;
    }
  }
}

// gradient w.r.t. prob (the student is not flipped, so it is written at the student's own pixel)
template <int V, int NC, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, NC <= 4 ? 3 : 2) uda_flip_bwd_kernel(
    const float* __restrict__ prob, const float* __restrict__ target, const unsigned char* __restrict__ flips,
    int C_rt, int H, int W, int kind, float eps, float inv_denom, const float* __restrict__ grad_loss,
    float* __restrict__ grad_prob) {
  const int C = NC < SUP_CMAX ? NC : C_rt;
  const long long o = blockIdx.y, inner = (long long)H * W;
  const unsigned f = flips[o];
  const bool fh = f & IIC_FLIP_H, fw = f & IIC_FLIP_W;
  const float* pb = prob + o * C * inner;
  const float* tb = target + o * C * inner;
  float* gb = grad_prob + o * C * inner;
  const float g = (grad_loss ? __ldg(grad_loss) : 1.f) * inv_denom;
  const long long ngroups = inner / V;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ngroups;
       q += (long long)gridDim.x * blockDim.x) {
    long long off_s, off_t;
    flip_offsets<V>(q, H, W, fh, fw, &off_s, &off_t);
    float p[NC][V], t[NC][V];
    sup_load<V, NC>(pb + off_s, inner, C, p);
    sup_load<V, NC>(tb + off_t, inner, C, t);
    if (fw) reverse_group<V, NC>(t);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      if (FROM_LOGITS) {
        sup_softmax<V, NC>(p, e);
        sup_softmax<V, NC>(t, e);
      }
      float dot = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        float gp = 0.f;
        if (c < C) {
          gp = (kind == 0) ? 2.f * (p[c][e] - t[c][e]) * g : -t[c][e] / (p[c][e] + eps) * g;
          dot = fmaf(gp, p[c][e], dot);
        }
        t[c][e] = gp;                          // reuse as the gradient w.r.t. the probabilities (0 on padded channels)
      }
      if (FROM_LOGITS) {
#pragma unroll
        for (int c = 0; c < NC; ++c) t[c][e] = p[c][e] * (t[c][e] - dot);   // softmax adjoint
      }
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (c < C) {
        if (V == 4)
          *reinterpret_cast<float4*>(gb + (long long)c * inner + off_s) =
              make_float4(t[c][0], t[c][1 % V], t[c][2 % V], t[c][3 % V]);
        else
          gb[(long long)c * inner + off_s] = t[c][0];
      }
    }
  }
}

// ---- wide-class path (9 <= C <= 256): the channels of a pixel spread over the 8 warps of a CTA (pixel_common.cuh) ----
// grid (gx, outer); a tile is 32 pixel groups of one sample's plane, each read through the sample's flips as above.
template <int V, int CW, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, CW >= 32 ? 1 : 2) uda_flip_fwd_wide_kernel(
    const float* __restrict__ prob, const float* __restrict__ target, const unsigned char* __restrict__ flips, int C,
    int H, int W, int kind, float eps, double denom, float* __restrict__ loss_out, int* __restrict__ flags,
    FlipWorkspace* ws) {
  __shared__ float2 red_p[2][WIDE_WARPS * 32 * V], red_t[2][WIDE_WARPS * 32 * V];
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  const long long o = blockIdx.y, inner = (long long)H * W;
  const unsigned f = flips[o];
  const bool fh = f & IIC_FLIP_H, fw = f & IIC_FLIP_W;
  const float* pb = prob + o * C * inner;
  const float* tb = target + o * C * inner;
  double local = 0.0;
  const long long ngroups = inner / V, ntiles = (ngroups + 31) / 32;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane;
    const bool live = q < ngroups;
    long long off_s, off_t;
    flip_offsets<V>(q, H, W, fh, fw, &off_s, &off_t);
    float p[CW][V], t[CW][V];
    wide_load<V, CW>(pb + off_s, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, p);
    wide_load<V, CW>(tb + off_t, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, t);
    if (fw) reverse_group<V, CW>(t);
    if (FROM_LOGITS) {
      int arg[V];
      wide_softmax<V, CW>(p, c0, red_p[it], nullptr, arg);
      wide_softmax<V, CW>(t, c0, red_t[it], nullptr, arg);
    }
#pragma unroll
    for (int e = 0; e < V; ++e) {
      float v = 0.f;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        if (c0 + j < C) {
          if (kind == 0) { const float d = p[j][e] - t[j][e]; v = fmaf(d, d, v); }
          else v += -t[j][e] * logf((p[j][e] + eps) / (t[j][e] + eps));
        }
      }
      if (live) local += v;
    }
  }
  wide_loss_combine(local, denom, &ws->ticket, reinterpret_cast<double*>(ws + 1), loss_out, flags);
}

template <int V, int CW, bool FROM_LOGITS>
__global__ void __launch_bounds__(256, CW >= 32 ? 1 : 2) uda_flip_bwd_wide_kernel(
    const float* __restrict__ prob, const float* __restrict__ target, const unsigned char* __restrict__ flips, int C,
    int H, int W, int kind, float eps, float inv_denom, const float* __restrict__ grad_loss,
    float* __restrict__ grad_prob) {
  __shared__ float2 red_p[2][WIDE_WARPS * 32 * V], red_t[2][WIDE_WARPS * 32 * V];
  __shared__ float red_d[2][WIDE_WARPS * 32 * V];
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  const long long o = blockIdx.y, inner = (long long)H * W;
  const unsigned f = flips[o];
  const bool fh = f & IIC_FLIP_H, fw = f & IIC_FLIP_W;
  const float* pb = prob + o * C * inner;
  const float* tb = target + o * C * inner;
  float* gb = grad_prob + o * C * inner;
  const float g = (grad_loss ? __ldg(grad_loss) : 1.f) * inv_denom;
  const long long ngroups = inner / V, ntiles = (ngroups + 31) / 32;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane;
    const bool live = q < ngroups;
    long long off_s, off_t;
    flip_offsets<V>(q, H, W, fh, fw, &off_s, &off_t);
    float p[CW][V], t[CW][V];
    wide_load<V, CW>(pb + off_s, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, p);
    wide_load<V, CW>(tb + off_t, inner, c0, C, live, FROM_LOGITS ? -INFINITY : 0.f, t);
    if (fw) reverse_group<V, CW>(t);
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
          gp = (kind == 0) ? 2.f * (p[j][e] - t[j][e]) * g : -t[j][e] / (p[j][e] + eps) * g;
          dot = fmaf(gp, p[j][e], dot);
        }
        t[j][e] = gp;                          // reuse as the gradient w.r.t. the probabilities
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
    wide_store<V, CW>(gb + off_s, inner, c0, C, live, t);
  }
}

static bool flip_vec_ok(const void* a, const void* b, const void* c, int W) {
  if (W % 4 != 0) return false;
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
}

}  // namespace iic

using namespace iic;

extern "C" int iic_flip_batch(const float* in, float* out, const unsigned char* flips, long long outer, int C,
                              int H, int W, void* stream) {
  IIC_REQUIRE(in && out && flips, "iic_flip_batch: null pointer");
  IIC_REQUIRE(in != out, "iic_flip_batch: in-place flips are not supported");
  IIC_REQUIRE(outer > 0 && C > 0 && H > 0 && W > 0, "iic_flip_batch: empty tensor");
  IIC_REQUIRE(outer <= 65535, "iic_flip_batch: outer=%lld > 65535 samples unsupported", outer);
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = flip_vec_ok(in, out, in, W);
  const long long groups = (long long)C * H * (vec ? W / 4 : W);
  const dim3 grid(pixel_ctas_per_sample(outer, groups, 8), (unsigned)outer);
  if (vec) flip_batch_kernel<4><<<grid, 256, 0, st>>>(in, out, flips, C, H, W);
  else     flip_batch_kernel<1><<<grid, 256, 0, st>>>(in, out, flips, C, H, W);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" size_t iic_uda_flip_workspace_bytes(int device, long long outer) {
  int sms = sm_count_cached(device);
  if (sms <= 0) sms = 148;
  long long n = (long long)sms * 8;
  if (outer > n) n = outer;
  return sizeof(FlipWorkspace) + (size_t)n * sizeof(double);
}

#define IIC_FLIP_DISPATCH(LAUNCH)                                                                        \
  do {                                                                                                   \
    if (vec) {                                                                                           \
      if (from_logits) { if (C == 2) LAUNCH(4, 2, true); else if (C == 3) LAUNCH(4, 3, true);            \
                         else if (C == 4) LAUNCH(4, 4, true); else LAUNCH(4, SUP_CMAX, true); }          \
      else             { if (C == 2) LAUNCH(4, 2, false); else if (C == 3) LAUNCH(4, 3, false);          \
                         else if (C == 4) LAUNCH(4, 4, false); else LAUNCH(4, SUP_CMAX, false); }        \
    } else {                                                                                             \
      if (from_logits) { if (C == 2) LAUNCH(1, 2, true); else if (C == 3) LAUNCH(1, 3, true);            \
                         else if (C == 4) LAUNCH(1, 4, true); else LAUNCH(1, SUP_CMAX, true); }          \
      else             { if (C == 2) LAUNCH(1, 2, false); else if (C == 3) LAUNCH(1, 3, false);          \
                         else if (C == 4) LAUNCH(1, 4, false); else LAUNCH(1, SUP_CMAX, false); }        \
    }                                                                                                    \
  } while (0)

extern "C" int iic_uda_flip_forward(const float* prob, const float* target, const unsigned char* flips,
                                    long long outer, int C, int H, int W, int kind, double eps, int from_logits,
                                    float* loss_out, int* flags, void* workspace, void* stream) {
  IIC_REQUIRE(prob && target && flips && loss_out && flags && workspace, "iic_uda_flip_forward: null pointer");
  IIC_REQUIRE(outer > 0 && C > 0 && H > 0 && W > 0, "iic_uda_flip_forward: empty tensor");
  IIC_REQUIRE(outer <= 65535, "iic_uda_flip_forward: outer=%lld > 65535 samples unsupported", outer);
  IIC_REQUIRE(C <= WIDE_CMAX, "iic_uda_flip_forward: C=%d > %d channels unsupported", C, WIDE_CMAX);
  IIC_REQUIRE(kind == 0 || kind == 1, "iic_uda_flip_forward: kind must be 0 (mse) or 1 (kl)");
  cudaStream_t st = (cudaStream_t)stream;
  const long long inner = (long long)H * W, total = outer * inner;
  const double denom = kind == 0 ? (double)total * C : (double)total;
  const bool vec = flip_vec_ok(prob, target, prob, W);
  if (C > SUP_CMAX) {
    const long long ntiles = (inner / (vec ? 4 : 1) + 31) / 32;
#define IIC_FLIP_FWD_WIDE(VV, CW)                                                                                   \
    do {                                                                                                            \
      const auto kern = from_logits ? uda_flip_fwd_wide_kernel<VV, CW, true> : uda_flip_fwd_wide_kernel<VV, CW, false>; \
      const dim3 wgrid(pixel_ctas_per_sample(outer, ntiles * 256, wide_ctas_per_sm(kern)), (unsigned)outer);         \
      kern<<<wgrid, 256, 0, st>>>(prob, target, flips, C, H, W, kind, (float)eps, denom, loss_out, flags,           \
                                  (FlipWorkspace*)workspace);                                                       \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_FLIP_FWD_WIDE);
#undef IIC_FLIP_FWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  const dim3 grid(pixel_ctas_per_sample(outer, vec ? inner / 4 : inner, C <= 4 ? 3 : 2), (unsigned)outer);
#define IIC_FLIP_FWD(VV, NN, FL)                                                                              \
  uda_flip_fwd_kernel<VV, NN, FL><<<grid, 256, 0, st>>>(prob, target, flips, C, H, W, kind, (float)eps, denom, \
                                                        loss_out, flags, (FlipWorkspace*)workspace)
  IIC_FLIP_DISPATCH(IIC_FLIP_FWD);
#undef IIC_FLIP_FWD
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int iic_uda_flip_backward(const float* prob, const float* target, const unsigned char* flips,
                                     long long outer, int C, int H, int W, int kind, double eps, int from_logits,
                                     const float* grad_loss, float* grad_prob, void* stream) {
  IIC_REQUIRE(prob && target && flips && grad_prob, "iic_uda_flip_backward: null pointer");
  IIC_REQUIRE(outer > 0 && C > 0 && H > 0 && W > 0, "iic_uda_flip_backward: empty tensor");
  IIC_REQUIRE(outer <= 65535, "iic_uda_flip_backward: outer=%lld > 65535 samples unsupported", outer);
  IIC_REQUIRE(C <= WIDE_CMAX, "iic_uda_flip_backward: C=%d > %d channels unsupported", C, WIDE_CMAX);
  IIC_REQUIRE(kind == 0 || kind == 1, "iic_uda_flip_backward: kind must be 0 (mse) or 1 (kl)");
  cudaStream_t st = (cudaStream_t)stream;
  const long long inner = (long long)H * W, total = outer * inner;
  const float inv_denom = (float)(1.0 / (kind == 0 ? (double)total * C : (double)total));
  const bool vec = flip_vec_ok(prob, target, grad_prob, W);
  if (C > SUP_CMAX) {
    const long long ntiles = (inner / (vec ? 4 : 1) + 31) / 32;
#define IIC_FLIP_BWD_WIDE(VV, CW)                                                                                   \
    do {                                                                                                            \
      const auto kern = from_logits ? uda_flip_bwd_wide_kernel<VV, CW, true> : uda_flip_bwd_wide_kernel<VV, CW, false>; \
      const dim3 wgrid(pixel_ctas_per_sample(outer, ntiles * 256, wide_ctas_per_sm(kern)), (unsigned)outer);         \
      kern<<<wgrid, 256, 0, st>>>(prob, target, flips, C, H, W, kind, (float)eps, inv_denom, grad_loss, grad_prob); \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_FLIP_BWD_WIDE);
#undef IIC_FLIP_BWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  const dim3 grid(pixel_ctas_per_sample(outer, vec ? inner / 4 : inner, C <= 4 ? 3 : 2), (unsigned)outer);
#define IIC_FLIP_BWD(VV, NN, FL)                                                                                  \
  uda_flip_bwd_kernel<VV, NN, FL><<<grid, 256, 0, st>>>(prob, target, flips, C, H, W, kind, (float)eps, inv_denom, \
                                                        grad_loss, grad_prob)
  IIC_FLIP_DISPATCH(IIC_FLIP_BWD);
#undef IIC_FLIP_BWD
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
