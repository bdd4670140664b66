// Supervised branch of the udaiic iteration (SURVEY.md section 8f row 4): one streaming pass each way (HBM-bound).
//   loss : sup_loss = KL_div()(label_logits.softmax(1), class2one_hot(labeled_target.squeeze(1), C))
//          semi_seg/epocher.py:165-166; dc2:deepclustering2/loss/kl_losses.py:107-126 (reduction "mean");
//          dc2:deepclustering2/utils/assertion.py:101-116 class2one_hot (a `long` one-hot; its sset assert -> BAD_LABEL flag)
//   dice : the tensors UniversalDice.add appends for (label_logits.max(1)[1], labeled_target.squeeze(1))
//          semi_seg/epocher.py:183-184; dc2:deepclustering2/meters2/individual_meters/general_dice_meter.py:41-95
//          (_intersaction = sum(pred*target), _union = sum(pred+target) over the pixels of one sample)
// With a one-hot target only the labelled class contributes: -1 * log((p_l + eps) / (1 + eps)) * w_l, the other
// classes give -0 * log(finite) = 0 (eps > 0).  The softmax, the one-hot and the argmax live in registers; the
// (B,C,H,W) int64 one-hot (8*C bytes per pixel) and the probability map are never materialised.
// A thread owns V consecutive pixels of one sample (V = 4 with 16-byte loads when the rows allow it) and keeps NC
// channels in registers: NC = C for the usual 2..4 classes (no padded work), NC = 8 with run-time guards otherwise.
#include "common.cuh"
#include "pixel_common.cuh"

namespace iic {

struct SupWorkspace {
  unsigned int ticket;   // self-resetting arrival counter
  unsigned int pad_;
  // followed by double partial[gridDim.x * gridDim.y]
};

// grid (gx, outer): blockIdx.y = sample, so the Dice counters of a CTA belong to one sample.
// IGN (the ignore-label form): a pixel labelled `ignore_index` takes the out-of-range route without the flag and is left
// out of the Dice counts; the others are counted into *n_valid (zeroed by the host), which replaces `denom`.
template <int V, int NC, bool IGN>
__global__ void __launch_bounds__(256, NC <= 4 ? 3 : 2) sup_fwd_kernel(const float* __restrict__ logits,
                                                      const long long* __restrict__ labels, int C_rt,
                                                      long long inner, float eps, const float* __restrict__ weight,
                                                      double denom, float* __restrict__ loss_out,
                                                      long long* __restrict__ dice_out, int* __restrict__ flags,
                                                      SupWorkspace* ws, long long ignore_index, long long* n_valid) {
  __shared__ double scratch[40];
  __shared__ unsigned int s_cnt[2][SUP_CMAX];
  __shared__ bool is_last;
  double* partial = reinterpret_cast<double*>(ws + 1);
  const int C = NC < SUP_CMAX ? NC : C_rt;      // the host picks NC == C for C <= 4
  const long long o = blockIdx.y, outer = gridDim.y;
  const float* lg = logits + o * C * inner;
  const long long* lb = labels + o * inner;
  if (threadIdx.x < 2 * SUP_CMAX) (&s_cnt[0][0])[threadIdx.x] = 0u;
  __syncthreads();
  float w[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) w[c] = (weight && c < C) ? __ldg(weight + c) : 1.f;
  unsigned int ci[NC], cu[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) { ci[c] = 0u; cu[c] = 0u; }
  float local = 0.f;
  bool bad = false;
  unsigned int nv = 0u;                                 // IGN: pixels not ignored
  const long long ngroups = inner / V;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ngroups;
       q += (long long)gridDim.x * blockDim.x) {
    float p[NC][V];
    long long l[V];
    sup_load<V, NC>(lg + q * V, inner, C, p);
    sup_load_labels<V>(lb + q * V, l);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      const int arg = sup_softmax<V, NC>(p, e);
      const bool ign = IGN && l[e] == ignore_index;
      const bool ok = !ign && (l[e] >= 0 && l[e] < C);
      bad |= !ok && !ign;
      nv += (unsigned)!ign;
      const int li = ok ? (int)l[e] : -1, ai = ign ? -1 : arg;
      float pl = 1.f, wl = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if (c == li) { pl = p[c][e]; wl = w[c]; }
        ci[c] += (unsigned)((c == ai) & (c == li));
        cu[c] += (unsigned)(c == ai) + (unsigned)(c == li);
      }
      // -target * log((prob + eps) / (target + eps)) * weight with target = 1 (kl_losses.py:114-118)
      local += -logf((pl + eps) / (1.f + eps)) * wl;
    }
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flags, IIC_FLAG_BAD_LABEL);
  if (dice_out != nullptr) {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (c < C) {
        const unsigned a = __reduce_add_sync(0xffffffffu, ci[c]);
        const unsigned b = __reduce_add_sync(0xffffffffu, cu[c]);
        if ((threadIdx.x & 31) == 0) {
          if (a) atomicAdd(&s_cnt[0][c], a);
          if (b) atomicAdd(&s_cnt[1][c], b);
        }
      }
    }
    __syncthreads();
    if (threadIdx.x < 2 * SUP_CMAX) {
      const int which = threadIdx.x / SUP_CMAX, c = threadIdx.x % SUP_CMAX;
      const unsigned v = s_cnt[which][c];
      // dice_out[which][sample][class]; integer atomics: the result does not depend on the order
      if (c < C && v)
        atomicAdd(reinterpret_cast<unsigned long long*>(dice_out) + ((long long)which * outer + o) * C + c,
                  (unsigned long long)v);
    }
  }
  const unsigned long long cta_n = IGN ? cta_count(nv) : 0ull;
  const double bsum = block_sum((double)local, scratch);
  const unsigned int ncta = gridDim.x * gridDim.y;
  if (threadIdx.x == 0) {
    partial[blockIdx.y * gridDim.x + blockIdx.x] = bsum;
    // the count goes in before the ticket, so the last CTA sees the final n (integer atomics: order-independent)
    if (IGN && cta_n) atomicAdd(reinterpret_cast<unsigned long long*>(n_valid), cta_n);
    __threadfence();
    is_last = (atomicAdd(&ws->ticket, 1u) == ncta - 1);
  }
  __syncthreads();
  if (is_last) {
    // the last CTA adds the per-CTA sums: thread t takes partial[t], partial[t+256], ... in order, then a
    // fixed-shape block reduction -> deterministic
    __threadfence();
    const volatile double* pp = partial;
    double tsum = 0.0;
    for (unsigned int b = threadIdx.x; b < ncta; b += blockDim.x) tsum += pp[b];
    double tot = block_sum(tsum, scratch);
    if (threadIdx.x == 0) {
      tot = IGN ? mean_over_valid(tot, n_valid) : tot / denom;
      loss_out[0] = (float)tot;
      if (tot != tot) atomicOr(flags, IIC_FLAG_NAN_LOSS);
      ws->ticket = 0;
    }
  }
}

// The loss gradient's scale g / n: the host's 1 / (outer*inner), or in the ignore-label forms 1 / n with the count the
// forward left in *n_valid (0 when every pixel is ignored)
template <bool IGN>
__device__ __forceinline__ float sup_grad_scale(const float* __restrict__ grad_loss, float inv_denom,
                                                const long long* __restrict__ n_valid) {
  const float g = grad_loss ? __ldg(grad_loss) : 1.f;
  if (!IGN) return g * inv_denom;
  const long long n = __ldg(n_valid);
  return n > 0 ? g * (float)(1.0 / (double)n) : 0.f;
}

// d loss / d logits: gp_l = -w_l / (p_l + eps) * g / (outer*inner) on the labelled class only, then the softmax
// adjoint p_c * (gp_c - sum_k gp_k p_k).  A pixel with an out-of-range or ignored label gets a zero gradient.
template <int V, int NC, bool IGN>
__global__ void __launch_bounds__(256, NC <= 4 ? 3 : 2) sup_bwd_kernel(const float* __restrict__ logits,
                                                      const long long* __restrict__ labels, int C_rt,
                                                      long long inner, float eps, const float* __restrict__ weight,
                                                      float inv_denom, const float* __restrict__ grad_loss,
                                                      float* __restrict__ grad_logits, long long ignore_index,
                                                      const long long* __restrict__ n_valid) {
  const int C = NC < SUP_CMAX ? NC : C_rt;
  const long long o = blockIdx.y;
  const float* lg = logits + o * C * inner;
  const long long* lb = labels + o * inner;
  float* gl = grad_logits + o * C * inner;
  const float g = sup_grad_scale<IGN>(grad_loss, inv_denom, n_valid);
  float w[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) w[c] = (weight && c < C) ? __ldg(weight + c) : 1.f;
  const long long ngroups = inner / V;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < ngroups;
       q += (long long)gridDim.x * blockDim.x) {
    float p[NC][V];
    long long l[V];
    sup_load<V, NC>(lg + q * V, inner, C, p);
    sup_load_labels<V>(lb + q * V, l);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      sup_softmax<V, NC>(p, e);
      const bool ign = IGN && l[e] == ignore_index;
      const int li = (!ign && l[e] >= 0 && l[e] < C) ? (int)l[e] : -1;
      float pl = 1.f, wl = 0.f;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if (c == li) { pl = p[c][e]; wl = w[c]; }
      }
      // 0 when the label is out of range (wl = 0).  IGN: such a pixel divides -1 and scales by 0 instead, since a zero
      // numerator sends the division to its slow path (at 10 % void almost every warp took it: +19 % backward time)
      const float gpl = IGN ? -(li >= 0 ? wl : 1.f) / (pl + eps) * (li >= 0 ? g : 0.f) : -wl / (pl + eps) * g;
      const float dot = gpl * pl;
#pragma unroll
      for (int c = 0; c < NC; ++c) p[c][e] = p[c][e] * ((c == li ? gpl : 0.f) - dot);
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (c < C) {
        if (V == 4)
          *reinterpret_cast<float4*>(gl + (long long)c * inner + q * V) =
              make_float4(p[c][0], p[c][1 % V], p[c][2 % V], p[c][3 % V]);
        else
          gl[(long long)c * inner + q] = p[c][0];
      }
    }
  }
}

// ---- wide-class path (9 <= C <= 256): the channels of a pixel spread over the 8 warps of a CTA (pixel_common.cuh) ----
// grid (gx, outer) as above; a CTA walks the tiles of its sample.  The warp that holds the labelled class adds the
// pixel's loss term.  Dice: the warps holding a pixel's argmax and label class count it into 2*C shared-memory
// counters, added to dice_out with integer atomics at the end (order-independent, so bit-exact).  IGN as for
// sup_fwd_kernel.
template <int V, int CW, bool IGN>
__global__ void __launch_bounds__(256, CW * V >= 32 ? 1 : 2) sup_fwd_wide_kernel(const float* __restrict__ logits,
                                                           const long long* __restrict__ labels, int C, long long inner,
                                                           float eps, const float* __restrict__ weight, double denom,
                                                           float* __restrict__ loss_out, long long* __restrict__ dice_out,
                                                           int* __restrict__ flags, SupWorkspace* ws,
                                                           long long ignore_index, long long* n_valid) {
  __shared__ float2 red[2][WIDE_WARPS * 32 * V];
  __shared__ int red_arg[2][WIDE_WARPS * 32 * V];
  __shared__ unsigned int s_cnt[2][WIDE_CMAX];                    // [intersection, union][class]
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  const long long o = blockIdx.y, outer = gridDim.y;
  const float* lg = logits + o * C * inner;
  const long long* lb = labels + o * inner;
  for (int k = threadIdx.x; k < 2 * WIDE_CMAX; k += blockDim.x) (&s_cnt[0][0])[k] = 0u;
  __syncthreads();
  double local = 0.0;
  bool bad = false;
  unsigned int nv = 0u;                                 // IGN: pixels not ignored (counted by warp 0 only)
  const long long ngroups = inner / V, ntiles = (ngroups + 31) / 32;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane;
    const bool live = q < ngroups;
    float x[CW][V];
    long long l[V];
    wide_load<V, CW>(lg + q * V, inner, c0, C, live, -INFINITY, x);
    if (live) sup_load_labels<V>(lb + q * V, l);
#pragma unroll
    for (int e = 0; e < V; ++e) if (!live) l[e] = -1;
    int arg[V];
    wide_softmax<V, CW>(x, c0, red[it], red_arg[it], arg);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      const bool ign = IGN && live && l[e] == ignore_index;
      const bool ok = !ign && (l[e] >= 0 && l[e] < C);
      bad |= live && !ok && !ign;
      if (IGN) nv += (unsigned)(live && !ign && c0 == 0);
      const int li = ok ? (int)l[e] : -1, ai = live && !ign ? arg[e] : -1;   // a lane past the end has l = -1
      float pl = 1.f;
      bool own = false;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        if (c0 + j == li) { pl = x[j][e]; own = true; }
      }
      if (dice_out != nullptr) {
        if (own) {
          atomicAdd(&s_cnt[1][li], 1u);
          if (ai == li) atomicAdd(&s_cnt[0][li], 1u);
        }
        if (ai >= c0 && ai < c0 + CW) atomicAdd(&s_cnt[1][ai], 1u);
      }
      // -target * log((prob + eps) / (target + eps)) * weight with target = 1 (kl_losses.py:114-118)
      if (own) local += -logf((pl + eps) / (1.f + eps)) * (weight ? __ldg(weight + li) : 1.f);
    }
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(flags, IIC_FLAG_BAD_LABEL);
  if (dice_out != nullptr) {
    __syncthreads();
    for (int k = threadIdx.x; k < 2 * C; k += blockDim.x) {
      const int which = k / C, c = k - which * C;
      const unsigned v = s_cnt[which][c];
      // dice_out[which][sample][class]
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(dice_out) + ((long long)which * outer + o) * C + c,
                       (unsigned long long)v);
    }
  }
  wide_loss_combine<IGN>(local, denom, &ws->ticket, reinterpret_cast<double*>(ws + 1), loss_out, flags, nv, n_valid);
}

// softmax adjoint with the dot sum_k gp_k p_k = gp_l p_l supplied by the warp that holds the label
template <int V, int CW, bool IGN>
__global__ void __launch_bounds__(256, CW * V >= 32 ? 1 : 2) sup_bwd_wide_kernel(const float* __restrict__ logits,
                                                           const long long* __restrict__ labels, int C, long long inner,
                                                           float eps, const float* __restrict__ weight, float inv_denom,
                                                           const float* __restrict__ grad_loss,
                                                           float* __restrict__ grad_logits, long long ignore_index,
                                                           const long long* __restrict__ n_valid) {
  __shared__ float2 red[2][WIDE_WARPS * 32 * V];
  __shared__ float red_d[2][WIDE_WARPS * 32 * V];
  const int lane = threadIdx.x & 31, c0 = (threadIdx.x >> 5) * CW;
  const long long o = blockIdx.y;
  const float* lg = logits + o * C * inner;
  const long long* lb = labels + o * inner;
  float* gl = grad_logits + o * C * inner;
  const float g = sup_grad_scale<IGN>(grad_loss, inv_denom, n_valid);
  const long long ngroups = inner / V, ntiles = (ngroups + 31) / 32;
  int it = 0;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, it ^= 1) {
    const long long q = tile * 32 + lane;
    const bool live = q < ngroups;
    float x[CW][V];
    long long l[V];
    wide_load<V, CW>(lg + q * V, inner, c0, C, live, -INFINITY, x);
    if (live) sup_load_labels<V>(lb + q * V, l);
#pragma unroll
    for (int e = 0; e < V; ++e) if (!live) l[e] = -1;
    int arg[V];
    wide_softmax<V, CW>(x, c0, red[it], nullptr, arg);
    int li[V];
    float gpl[V];
#pragma unroll
    for (int e = 0; e < V; ++e) {
      li[e] = (live && !(IGN && l[e] == ignore_index) && l[e] >= 0 && l[e] < C) ? (int)l[e] : -1;
      float pl = 0.f;
      bool own = false;
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        if (c0 + j == li[e]) { pl = x[j][e]; own = true; }
      }
      gpl[e] = own ? -(weight ? __ldg(weight + li[e]) : 1.f) / (pl + eps) * g : 0.f;
      red_d[it][(threadIdx.x >> 5) * 32 * V + lane * V + e] = gpl[e] * pl;
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < V; ++e) {
      const float dot = wide_warp_sum<V>(red_d[it], lane * V + e);
#pragma unroll
      for (int j = 0; j < CW; ++j) x[j][e] = x[j][e] * ((c0 + j == li[e] ? gpl[e] : 0.f) - dot);
    }
    wide_store<V, CW>(gl + q * V, inner, c0, C, live, x);
  }
}

static bool sup_vec_ok(const void* a, const void* b, const void* c, long long inner) {
  if (inner % 4 != 0) return false;
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
}

}  // namespace iic

using namespace iic;

extern "C" size_t iic_sup_workspace_bytes(int device, long long outer) {
  int sms = sm_count_cached(device);
  if (sms <= 0) sms = 148;
  long long n = (long long)sms * 8;
  if (outer > n) n = outer;
  return sizeof(SupWorkspace) + (size_t)n * sizeof(double);
}

// One host implementation for both entry-point pairs: IGN = false is iic_sup_forward / _backward (denominator
// outer*inner from the host), IGN = true the ignore-label pair (denominator counted on the device into *n_valid).
template <bool IGN>
static int sup_forward_impl(const char* fn, const float* logits, const long long* labels, long long outer, int C,
                            long long inner, double eps, const float* weight, long long ignore_index,
                            float* loss_out, long long* dice_out, long long* n_valid, int* flags, void* workspace,
                            void* stream) {
  IIC_REQUIRE(logits && labels && loss_out && flags && workspace && (!IGN || n_valid), "%s: null pointer", fn);
  IIC_REQUIRE(outer > 0 && C > 0 && inner > 0, "%s: empty tensor", fn);
  IIC_REQUIRE(outer <= 65535, "%s: outer=%lld > 65535 samples unsupported", fn, outer);
  IIC_REQUIRE(C <= WIDE_CMAX, "%s: C=%d > %d classes unsupported", fn, C, WIDE_CMAX);
  IIC_REQUIRE(eps > 0.0, "%s: eps must be > 0 (the reference's loss is NaN at eps = 0)", fn);
  cudaStream_t st = (cudaStream_t)stream;
  if (dice_out) IIC_CHECK_CUDA(cudaMemsetAsync(dice_out, 0, (size_t)2 * outer * C * sizeof(long long), st));
  if (IGN) IIC_CHECK_CUDA(cudaMemsetAsync(n_valid, 0, sizeof(long long), st));
  const double denom = (double)outer * (double)inner;
  if (C > SUP_CMAX) {
    const bool vec = wide_vec_ok(logits, labels, logits, inner);
    const long long ntiles = (inner / (vec ? 4 : 1) + 31) / 32;
#define IIC_SUP_FWD_WIDE(VV, CW)                                                                                    \
    do {                                                                                                            \
      const auto kern = sup_fwd_wide_kernel<VV, CW, IGN>;                                                           \
      const dim3 wgrid(pixel_ctas_per_sample(outer, ntiles * 256, wide_ctas_per_sm(kern)), (unsigned)outer);         \
      kern<<<wgrid, 256, 0, st>>>(logits, labels, C, inner, (float)eps, weight, denom, loss_out, dice_out, flags,    \
                                  (SupWorkspace*)workspace, ignore_index, n_valid);                                 \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_SUP_FWD_WIDE);
#undef IIC_SUP_FWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  const bool vec = sup_vec_ok(logits, labels, logits, inner);
  const dim3 grid(pixel_ctas_per_sample(outer, vec ? inner / 4 : inner, C <= 4 ? 3 : 2), (unsigned)outer);
#define IIC_SUP_FWD(VV, NN)                                                                                      \
  sup_fwd_kernel<VV, NN, IGN><<<grid, 256, 0, st>>>(logits, labels, C, inner, (float)eps, weight, denom,         \
                                                    loss_out, dice_out, flags, (SupWorkspace*)workspace,         \
                                                    ignore_index, n_valid)
  if (vec) { if (C == 2) IIC_SUP_FWD(4, 2); else if (C == 3) IIC_SUP_FWD(4, 3); else if (C == 4) IIC_SUP_FWD(4, 4); else IIC_SUP_FWD(4, SUP_CMAX); }
  else     { if (C == 2) IIC_SUP_FWD(1, 2); else if (C == 3) IIC_SUP_FWD(1, 3); else if (C == 4) IIC_SUP_FWD(1, 4); else IIC_SUP_FWD(1, SUP_CMAX); }
#undef IIC_SUP_FWD
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

template <bool IGN>
static int sup_backward_impl(const char* fn, const float* logits, const long long* labels, long long outer, int C,
                             long long inner, double eps, const float* weight, long long ignore_index,
                             const long long* n_valid, const float* grad_loss, float* grad_logits, void* stream) {
  IIC_REQUIRE(logits && labels && grad_logits && (!IGN || n_valid), "%s: null pointer", fn);
  IIC_REQUIRE(outer > 0 && C > 0 && inner > 0, "%s: empty tensor", fn);
  IIC_REQUIRE(outer <= 65535, "%s: outer=%lld > 65535 samples unsupported", fn, outer);
  IIC_REQUIRE(C <= WIDE_CMAX, "%s: C=%d > %d classes unsupported", fn, C, WIDE_CMAX);
  IIC_REQUIRE(eps > 0.0, "%s: eps must be > 0", fn);
  cudaStream_t st = (cudaStream_t)stream;
  const float inv_denom = (float)(1.0 / ((double)outer * (double)inner));   // unused by IGN: the kernel reads n_valid
  if (C > SUP_CMAX) {
    const bool vec = wide_vec_ok(logits, labels, grad_logits, inner);
    const long long ntiles = (inner / (vec ? 4 : 1) + 31) / 32;
#define IIC_SUP_BWD_WIDE(VV, CW)                                                                                    \
    do {                                                                                                            \
      const auto kern = sup_bwd_wide_kernel<VV, CW, IGN>;                                                           \
      const dim3 wgrid(pixel_ctas_per_sample(outer, ntiles * 256, wide_ctas_per_sm(kern)), (unsigned)outer);         \
      kern<<<wgrid, 256, 0, st>>>(logits, labels, C, inner, (float)eps, weight, inv_denom, grad_loss, grad_logits,   \
                                  ignore_index, n_valid);                                                           \
    } while (0)
    IIC_WIDE_DISPATCH(vec, C, IIC_SUP_BWD_WIDE);
#undef IIC_SUP_BWD_WIDE
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  const bool vec = sup_vec_ok(logits, labels, grad_logits, inner);
  const dim3 grid(pixel_ctas_per_sample(outer, vec ? inner / 4 : inner, C <= 4 ? 3 : 2), (unsigned)outer);
#define IIC_SUP_BWD(VV, NN)                                                                                      \
  sup_bwd_kernel<VV, NN, IGN><<<grid, 256, 0, st>>>(logits, labels, C, inner, (float)eps, weight, inv_denom,     \
                                                    grad_loss, grad_logits, ignore_index, n_valid)
  if (vec) { if (C == 2) IIC_SUP_BWD(4, 2); else if (C == 3) IIC_SUP_BWD(4, 3); else if (C == 4) IIC_SUP_BWD(4, 4); else IIC_SUP_BWD(4, SUP_CMAX); }
  else     { if (C == 2) IIC_SUP_BWD(1, 2); else if (C == 3) IIC_SUP_BWD(1, 3); else if (C == 4) IIC_SUP_BWD(1, 4); else IIC_SUP_BWD(1, SUP_CMAX); }
#undef IIC_SUP_BWD
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int iic_sup_forward(const float* logits, const long long* labels, long long outer, int C,
                               long long inner, double eps, const float* weight, float* loss_out,
                               long long* dice_out, int* flags, void* workspace, void* stream) {
  return sup_forward_impl<false>("iic_sup_forward", logits, labels, outer, C, inner, eps, weight, 0, loss_out,
                                 dice_out, nullptr, flags, workspace, stream);
}

extern "C" int iic_sup_backward(const float* logits, const long long* labels, long long outer, int C,
                                long long inner, double eps, const float* weight, const float* grad_loss,
                                float* grad_logits, void* stream) {
  return sup_backward_impl<false>("iic_sup_backward", logits, labels, outer, C, inner, eps, weight, 0, nullptr,
                                  grad_loss, grad_logits, stream);
}

extern "C" int iic_sup_forward_ignore(const float* logits, const long long* labels, long long outer, int C,
                                      long long inner, double eps, const float* weight, long long ignore_index,
                                      float* loss_out, long long* dice_out, long long* n_valid, int* flags,
                                      void* workspace, void* stream) {
  return sup_forward_impl<true>("iic_sup_forward_ignore", logits, labels, outer, C, inner, eps, weight, ignore_index,
                                loss_out, dice_out, n_valid, flags, workspace, stream);
}

extern "C" int iic_sup_backward_ignore(const float* logits, const long long* labels, long long outer, int C,
                                       long long inner, double eps, const float* weight, long long ignore_index,
                                       const long long* n_valid, const float* grad_loss, float* grad_logits,
                                       void* stream) {
  return sup_backward_impl<true>("iic_sup_backward_ignore", logits, labels, outer, C, inner, eps, weight,
                                 ignore_index, n_valid, grad_loss, grad_logits, stream);
}
