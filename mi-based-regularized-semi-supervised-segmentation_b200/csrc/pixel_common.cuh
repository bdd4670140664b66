// Per-pixel register helpers shared by the streaming kernels that keep all channels of V consecutive pixels in
// registers (csrc/sup.cu, csrc/flip.cu): channel-row loads (16-byte when V = 4), int64 label loads, channel softmax.
// Below them, the tile, merge and loss helpers of the wide-class kernels (csrc/uda.cu, csrc/sup.cu, csrc/flip.cu),
// which spread the channels of a pixel over the warps of a CTA.
#pragma once
#include "common.cuh"

namespace iic {

constexpr int SUP_CMAX = 8;      // channels kept in registers by the generic (run-time C) instantiations

template <int V, int NC>
__device__ __forceinline__ void sup_load(const float* __restrict__ src, long long inner, int C,
                                         float (&v)[NC][V]) {
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (c < C) {
      if (V == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(src + (long long)c * inner));
        v[c][0] = t.x; v[c][1 % V] = t.y; v[c][2 % V] = t.z; v[c][3 % V] = t.w;
      } else {
        v[c][0] = __ldg(src + (long long)c * inner);
      }
    } else {
#pragma unroll
      for (int e = 0; e < V; ++e) v[c][e] = -INFINITY;
    }
  }
}

template <int V>
__device__ __forceinline__ void sup_load_labels(const long long* __restrict__ src, long long (&l)[V]) {
  if (V == 4) {
    const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(src));
    const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(src) + 1);
    l[0] = a.x; l[1 % V] = a.y; l[2 % V] = b.x; l[3 % V] = b.y;
  } else {
    l[0] = __ldg(src);
  }
}

// softmax over the channels of pixel e, in place; returns the index of the first maximal logit
template <int V, int NC>
__device__ __forceinline__ int sup_softmax(float (&v)[NC][V], int e) {
  float mx = v[0][e];
  int arg = 0;
#pragma unroll
  for (int c = 1; c < NC; ++c) {
    if (v[c][e] > mx) { mx = v[c][e]; arg = c; }
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) { v[c][e] = __expf(v[c][e] - mx); s += v[c][e]; }   // exp(-inf) = 0 pads
  const float inv = 1.f / s;
#pragma unroll
  for (int c = 0; c < NC; ++c) v[c][e] *= inv;
  return arg;
}

// CTAs per sample (grid = (gx, outer)) for one resident wave of `ctas_per_sm` 256-thread CTAs per SM, with every
// thread walking the same number of pixel groups: k = iterations per thread, then just enough CTAs for k.
// gx * outer <= max(sms * ctas_per_sm, outer).
inline int pixel_ctas_per_sample(long long outer, long long groups, int ctas_per_sm) {
  int sms = sm_count_cached(current_device());
  if (sms <= 0) sms = 148;
  long long cap = ((long long)sms * ctas_per_sm) / outer;
  if (cap < 1) cap = 1;
  const long long k = (groups + 256 * cap - 1) / (256 * cap);
  long long gx = (groups + 256 * k - 1) / (256 * k);
  if (gx < 1) gx = 1;
  return (int)gx;
}

// ---- wide-class path (9 <= C <= 256) -------------------------------------------------------------------------------
// A 256-thread CTA owns a tile of 32*V consecutive pixels of one sample: lane l holds pixels [l*V, l*V + V) of the tile
// and warp w holds channels [w*CW, w*CW + CW) of them in registers, so one channel row of a tile is one warp access of
// at least 128 bytes.  Per-pixel quantities that need every channel (softmax max and sum, argmax, the adjoint's dot,
// the simplex sums) are merged through shared memory in warp order: the results do not depend on timing.
// Each merge buffer is used in alternate halves on alternate tiles, so one __syncthreads per merge is enough.
constexpr int WIDE_CMAX = 256;
constexpr int WIDE_WARPS = 8;

// channel slice per warp: ceil(C / 8) rounded up to a compile-time width
inline int wide_cw(int C) { return C <= 16 ? 2 : C <= 32 ? 4 : C <= 64 ? 8 : C <= 128 ? 16 : 32; }

// LAUNCH(V, CW) for the slice width of C; V = 4 (16-byte accesses) where `vec` and both maps of a pixel group fit the
// register budget (CW <= 8), else V = 1
#define IIC_WIDE_DISPATCH(vec, C, LAUNCH)                                         \
  do {                                                                            \
    switch (wide_cw(C)) {                                                         \
      case 2:  if (vec) LAUNCH(4, 2); else LAUNCH(1, 2); break;                   \
      case 4:  if (vec) LAUNCH(4, 4); else LAUNCH(1, 4); break;                   \
      case 8:  if (vec) LAUNCH(4, 8); else LAUNCH(1, 8); break;                   \
      case 16: LAUNCH(1, 16); break;                                              \
      default: LAUNCH(1, 32); break;                                              \
    }                                                                             \
  } while (0)

// channels [c0, c0 + CW) of V consecutive pixels at `src` (channel stride `inner`); channels >= C and pixels of a
// lane that is not `live` read as `pad`
template <int V, int CW>
__device__ __forceinline__ void wide_load(const float* __restrict__ src, long long inner, int c0, int C, bool live,
                                          float pad, float (&v)[CW][V]) {
#pragma unroll
  for (int j = 0; j < CW; ++j) {
    if (live && c0 + j < C) {
      if (V == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(src + (long long)(c0 + j) * inner));
        v[j][0] = t.x; v[j][1 % V] = t.y; v[j][2 % V] = t.z; v[j][3 % V] = t.w;
      } else {
        v[j][0] = __ldg(src + (long long)(c0 + j) * inner);
      }
    } else {
#pragma unroll
      for (int e = 0; e < V; ++e) v[j][e] = pad;
    }
  }
}

template <int V, int CW>
__device__ __forceinline__ void wide_store(float* __restrict__ dst, long long inner, int c0, int C, bool live,
                                           const float (&v)[CW][V]) {
  if (!live) return;
#pragma unroll
  for (int j = 0; j < CW; ++j) {
    if (c0 + j < C) {
      if (V == 4)
        *reinterpret_cast<float4*>(dst + (long long)(c0 + j) * inner) =
            make_float4(v[j][0], v[j][1 % V], v[j][2 % V], v[j][3 % V]);
      else
        dst[(long long)(c0 + j) * inner] = v[j][0];
    }
  }
}

// This warp's part of the softmax of pixel e: x (logits, -inf pads) becomes exp(x - m) for the slice maximum m; the
// returned pair is (m, sum of the exponentials); *arg is the first index of the slice maximum.  An all-pad slice gives
// (-inf, 0) and zeros.
template <int V, int CW>
__device__ __forceinline__ float2 wide_slice_exp(float (&x)[CW][V], int e, int c0, int* arg) {
  float m = x[0][e];
  int a = c0;
#pragma unroll
  for (int j = 1; j < CW; ++j) {
    if (x[j][e] > m) { m = x[j][e]; a = c0 + j; }
  }
  const float mm = m == -INFINITY ? 0.f : m;
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < CW; ++j) { x[j][e] = __expf(x[j][e] - mm); s += x[j][e]; }
  *arg = a;
  return make_float2(m, s);
}

// Combines the per-warp pairs red[w * 32V + k] of pixel slot k in warp order: m = max m_w, s = sum s_w exp(m_w - m).
// Returns the factor exp(m_own - m) / s that turns this warp's exponentials into probabilities.  With `red_arg` the
// first index of the maximal logit goes to *arg: the first warp holding the maximum wins, as in logits.max(1)[1].
template <int V>
__device__ __forceinline__ float wide_softmax_scale(const float2* red, const int* red_arg, int k, float2 own,
                                                    int* arg) {
  float m = red[k].x;
  int a = red_arg ? red_arg[k] : 0;
#pragma unroll
  for (int w = 1; w < WIDE_WARPS; ++w) {
    const float mw = red[w * 32 * V + k].x;
    if (mw > m) { m = mw; if (red_arg) a = red_arg[w * 32 * V + k]; }
  }
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < WIDE_WARPS; ++w) {
    const float2 r = red[w * 32 * V + k];
    s += r.y * __expf(r.x - m);                  // an all-pad slice has s_w = 0 and exp(-inf) = 0
  }
  if (arg) *arg = a;
  return __expf(own.x - m) / s;
}

// Sum over the warps, in warp order, of the per-warp values red[w * 32V + k] of pixel slot k
template <int V>
__device__ __forceinline__ float wide_warp_sum(const float* red, int k) {
  float s = red[k];
#pragma unroll
  for (int w = 1; w < WIDE_WARPS; ++w) s += red[w * 32 * V + k];
  return s;
}

inline bool wide_vec_ok(const void* a, const void* b, const void* c, long long inner) {
  if (inner % 4 != 0) return false;
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
}

// Softmax over the CTA's warps of the V pixels of each lane: x (this warp's logits) becomes probabilities.  `red` holds
// 32V float2 per warp (and `red_arg` 32V ints when the argmax is wanted); ends with the buffer's __syncthreads.
template <int V, int CW>
__device__ __forceinline__ void wide_softmax(float (&x)[CW][V], int c0, float2* red, int* red_arg, int (&arg)[V]) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float2 own[V];
#pragma unroll
  for (int e = 0; e < V; ++e) {
    int a;
    own[e] = wide_slice_exp<V, CW>(x, e, c0, &a);
    red[w * 32 * V + lane * V + e] = own[e];
    if (red_arg) red_arg[w * 32 * V + lane * V + e] = a;
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const float f = wide_softmax_scale<V>(red, red_arg, lane * V + e, own[e], &arg[e]);
#pragma unroll
    for (int j = 0; j < CW; ++j) x[j][e] *= f;
  }
}

// Ignore-label forms of the supervised kernels: the CTA's count of pixels that are not ignored, from the per-thread
// counts (warp sums into one shared counter; integer, so exact).  Every thread calls it and gets the count.
__device__ __forceinline__ unsigned long long cta_count(unsigned int n_local) {
  __shared__ unsigned long long s_n;
  if (threadIdx.x == 0) s_n = 0ull;
  __syncthreads();
  const unsigned int w = __reduce_add_sync(0xffffffffu, n_local);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_n, (unsigned long long)w);
  __syncthreads();
  return s_n;
}

// The mean's denominator in the ignore-label forms: the device-side count n of pixels that are not ignored, complete
// once the last CTA holds its ticket; the mean of an empty set is 0 (not NaN).
__device__ __forceinline__ double mean_over_valid(double sum, const long long* n_valid) {
  const long long n = *reinterpret_cast<const volatile long long*>(n_valid);
  return n > 0 ? sum / (double)n : 0.0;
}

// Per-CTA fp64 partial of the loss into partial[linear CTA index]; the last CTA to take a ticket adds the partials in a
// fixed order (thread t takes t, t + 256, ... then a fixed-shape block reduction) and writes sum / denom.  The ticket
// resets itself.  Deterministic for a given grid.  IGN (the ignore-label forms): each CTA adds its count of pixels that
// are not ignored (`n_local` per thread) to *n_valid before its ticket, and the last CTA divides by the final count
// instead of `denom` (mean_over_valid).
template <bool IGN = false>
__device__ __forceinline__ void wide_loss_combine(double local, double denom, unsigned int* ticket, double* partial,
                                                  float* __restrict__ loss_out, int* __restrict__ flags,
                                                  unsigned int n_local = 0u, long long* n_valid = nullptr) {
  __shared__ double scratch[40];
  __shared__ bool is_last;
  const unsigned long long cta_n = IGN ? cta_count(n_local) : 0ull;
  const double bsum = block_sum(local, scratch);
  const unsigned int ncta = gridDim.x * gridDim.y;
  if (threadIdx.x == 0) {
    partial[blockIdx.y * gridDim.x + blockIdx.x] = bsum;
    if (IGN && cta_n) atomicAdd(reinterpret_cast<unsigned long long*>(n_valid), cta_n);
    __threadfence();
    is_last = (atomicAdd(ticket, 1u) == ncta - 1);
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    const volatile double* pp = partial;
    double tsum = 0.0;
    for (unsigned int b = threadIdx.x; b < ncta; b += blockDim.x) tsum += pp[b];
    double tot = block_sum(tsum, scratch);
    if (threadIdx.x == 0) {
      tot = IGN ? mean_over_valid(tot, n_valid) : tot / denom;
      loss_out[0] = (float)tot;
      if (tot != tot) atomicOr(flags, IIC_FLAG_NAN_LOSS);
      *ticket = 0;
    }
  }
}

// CTAs of `kernel` resident per SM at 256 threads, at most 8: the loss workspaces hold 8 partials per SM
template <typename K>
inline int wide_ctas_per_sm(K kernel) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, 256, 0) != cudaSuccess || n < 1) n = 1;
  return n < 8 ? n : 8;
}

// 1-D grid over `ntiles` tiles: one resident wave of `kernel`
template <typename K>
inline unsigned wide_grid(K kernel, long long ntiles) {
  int sms = sm_count_cached(current_device());
  if (sms <= 0) sms = 148;
  const long long cap = (long long)sms * wide_ctas_per_sm(kernel);
  return (unsigned)(ntiles < cap ? ntiles : cap);
}

}  // namespace iic
