// Small-matrix stages of the IIC losses, all in float64:
//   * local epilogue: min-shift, per-displacement normalise, symmetrise, marginals, entropy and the
//     analytic dL/dJ                                    (contrastyou/losses/iic_loss.py:124-146,186)
//   * global joint / epilogue / backward on (N,K) rows  (contrastyou/losses/iic_loss.py:43-94)
#include "epilogue.cuh"
#include "local_kernels.cuh"

namespace iic {

// ======================================================================================================
// local epilogue: one CTA per (patch, displacement)
// ======================================================================================================
struct EpiWorkspace {       // lives at the start of the caller-provided workspace
  unsigned int ticket;      // self-resetting arrival counter
  unsigned int pad_;
};
// followed by double partial_loss[n_patches * T * T]

__global__ void __launch_bounds__(256) local_epilogue_kernel(
    const double* __restrict__ J, int K, int T, int n_patches, double lamda, float* __restrict__ loss_out,
    double* __restrict__ loss64_out, float* __restrict__ Wx, float* __restrict__ Wy,
    double* __restrict__ GA_out, int* __restrict__ flags, EpiWorkspace* ws) {
  extern __shared__ __align__(16) double sm[];
  double* partial_loss = reinterpret_cast<double*>(ws + 1);
  const int T2 = T * T;
  const int patch = blockIdx.x / T2, d = blockIdx.x % T2;
  const size_t KK = (size_t)K * K;
  const int Kp = (K + 3) & ~3;
  const int tid = threadIdx.x;
  const double scale = 1.0 / ((double)T2 * (double)n_patches);
  const double loss_d = local_epilogue_block(J + (size_t)patch * T2 * KK, K, T, d, lamda, scale,
                                             Wx + (size_t)patch * K * T2 * Kp, Wy + (size_t)patch * K * T2 * Kp,
                                             GA_out ? GA_out + ((size_t)patch * T2 + d) * KK : nullptr, sm);

  // last CTA sums the per-displacement losses in index order (deterministic)
  __shared__ bool is_last;
  if (tid == 0) {
    partial_loss[blockIdx.x] = loss_d;
    __threadfence();
    const unsigned int prev = atomicAdd(&ws->ticket, 1u);
    is_last = (prev == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last && tid == 0) {
    __threadfence();
    double total = 0.0;
    const volatile double* pl = partial_loss;
    for (unsigned int b = 0; b < gridDim.x; ++b) total += pl[b];
    total *= scale;
    loss_out[0] = (float)total;
    if (loss64_out) loss64_out[0] = total;
    if (total != total) atomicOr(flags, IIC_FLAG_NAN_LOSS);
    ws->ticket = 0;
  }
}

// ======================================================================================================
// global IIC on (N,K) rows
// ======================================================================================================
// Each thread owns output entries e = tid, tid + nt, ... (at most GLOBAL_EPT) and walks the CTA's rows,
// staged in shared memory; float64 accumulation (the contraction is tiny).
constexpr int GLOBAL_EPT = 16;
constexpr int GLOBAL_ROWS = 32;

__global__ void __launch_bounds__(1024) global_joint_kernel(const float* __restrict__ x, long long x_sn,
                                                            const float* __restrict__ y, long long y_sn,
                                                            long long N, int K, long long rows_per_cta,
                                                            double* __restrict__ partial, int* __restrict__ flags) {
  extern __shared__ __align__(16) float gsm[];
  float* xs = gsm;                       // [GLOBAL_ROWS][K]
  float* ys = gsm + GLOBAL_ROWS * K;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int KK = K * K;
  double acc[GLOBAL_EPT];
#pragma unroll
  for (int q = 0; q < GLOBAL_EPT; ++q) acc[q] = 0.0;
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta;
  if (r1 > N) r1 = N;
  for (long long rb = r0; rb < r1; rb += GLOBAL_ROWS) {
    const int nr = (int)((r1 - rb) < GLOBAL_ROWS ? (r1 - rb) : GLOBAL_ROWS);
    __syncthreads();
    for (int e = tid; e < nr * K; e += nt) {
      const int r = e / K, c = e % K;
      xs[e] = x[(rb + r) * x_sn + c];
      ys[e] = y[(rb + r) * y_sn + c];
    }
    __syncthreads();
    if (flags != nullptr && tid < 2 * nr) {
      // fused simplex assertions on both inputs (iic_loss.py:50-51,82-83): thread -> one staged row
      const float* row = (tid < nr ? xs : ys) + (tid < nr ? tid : tid - nr) * K;
      float sum = 0.f;
      for (int c = 0; c < K; ++c) sum += row[c];
      if (!(fabsf(sum - 1.f) <= 1e-4f + 1e-4f * 1.f)) atomicOr(flags, IIC_FLAG_NOT_SIMPLEX);
    }
#pragma unroll
    for (int q = 0; q < GLOBAL_EPT; ++q) {
      const int e = tid + q * nt;
      if (e < KK) {
        const int i = e / K, j = e % K;
        double a = acc[q];
        for (int r = 0; r < nr; ++r) a += (double)xs[r * K + i] * (double)ys[r * K + j];
        acc[q] = a;
      }
    }
  }
#pragma unroll
  for (int q = 0; q < GLOBAL_EPT; ++q) {
    const int e = tid + q * nt;
    if (e < KK) partial[(size_t)blockIdx.x * KK + e] = acc[q];
  }
}

__global__ void global_reduce_kernel(const double* __restrict__ partial, int ncta, int KK,
                                     double* __restrict__ J) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= KK) return;
  double s = 0.0;
  for (int c = 0; c < ncta; ++c) s += partial[(size_t)c * KK + e];
  J[e] = s;
}

// shared derivation for the global epilogue / backward: from J build S, marginals of P
struct GlobalStats { double S; };

// single CTA: P = sym(J)/S ; losses (iic_loss.py:56-69)
__global__ void __launch_bounds__(1024) global_epilogue_kernel(const double* __restrict__ J, int K,
                                                               double lamb, int symmetric,
                                                               float* __restrict__ losses_out,
                                                               float* __restrict__ P_out,
                                                               int* __restrict__ flags) {
  extern __shared__ __align__(16) double sm[];
  global_epilogue_block(J, K, lamb, symmetric, losses_out, P_out, flags, sm);
}

constexpr int GLOBAL_BWD_STAGE_FLOATS = 2048;      // rows of x (and of y) staged in shared memory by global_backward_kernel

// Every CTA rebuilds GJ = d(objective)/dJ in shared memory, then produces a slab of rows of gx = y GJ^T and gy = x GJ.
// The joint is read from global memory ONCE (symmetrised into shared memory); the kernel is a chain of small dependent
// phases, so every phase that went back to global memory for J cost a memory latency (19k cycles at (32, 10) before).
// From-logits form (FL): x and y are logit rows and J the joint of their softmax(l * inv_temp) (iic_finish's
// IIC_ITEM_GLOBAL_LOGITS).  One warp per row recomputes p of both rows with the finish launch's own functions
// (warp_row_softmax_stats, logit_p: the same bits), forms dp = GJ p and applies the softmax adjoint
// inv_temp * p * (dp - <dp, p>) to both rows.
template <bool FL>
__global__ void __launch_bounds__(256) global_backward_kernel(
    const float* __restrict__ x, long long x_sn, const float* __restrict__ y, long long y_sn, long long N,
    int K, const double* __restrict__ J, double lamb, int symmetric, const float* __restrict__ g_loss,
    const float* __restrict__ g_no_lamb, const float* __restrict__ gP, float* __restrict__ gx,
    float* __restrict__ gy, long long gx_sn, long long gy_sn,
    long long rows_per_cta, float inv_temp) {
  extern __shared__ __align__(16) double sm[];
  double* scratch = sm;            // 33
  double* pi = sm + 40;            // K
  double* pj = pi + K;             // K
  double* gi = pj + K;             // K : log(pi+eps) + pi/(pi+eps)
  double* gj = gi + K;             // K
  double* Js = gj + K;             // K*K : the (symmetrised) joint; overwritten in place by GP
  float* GJ = reinterpret_cast<float*>(Js + (size_t)K * K);    // K*K floats : dObj/dJ[i][j]
  float* rows_s = GJ + (size_t)K * K;                          // staged x and y rows of this CTA's slab (small slabs only)
  const int tid = threadIdx.x, nt = blockDim.x;
  const size_t KK = (size_t)K * K;
  const double eps = 1e-10;
  // the rows of this CTA's slab are independent of everything below: get them moving first
  const long long r0 = (long long)blockIdx.x * rows_per_cta;
  long long r1 = r0 + rows_per_cta;
  if (r1 > N) r1 = N;
  // A small slab (config 2: 32 rows of 10) is staged in shared memory now, so that its global-memory latency overlaps the
  // epilogue phases below instead of sitting in the row loop (K dependent loads per output there: ~6000 clk at K = 10).
  const long long slab = (r1 - r0) * K;
  const bool staged_rows = !FL && slab <= GLOBAL_BWD_STAGE_FLOATS;     // (FL: rows_s holds per-warp p rows)
  if (staged_rows)
    for (long long e = tid; e < slab; e += nt) {
      const long long n = r0 + e / K;
      const int c = (int)(e % K);
      rows_s[e] = x[n * x_sn + c];
      rows_s[slab + e] = y[n * y_sn + c];
    }
  const double g1 = g_loss ? (double)g_loss[0] : 0.0, g2 = g_no_lamb ? (double)g_no_lamb[0] : 0.0;
  double part = 0.0;
  for (size_t e = tid; e < KK; e += nt) {
    const int i = (int)(e / K), j = (int)(e % K);
    const double v = symmetric ? (J[(size_t)i * K + j] + J[(size_t)j * K + i]) / 2.0 : J[(size_t)i * K + j];
    Js[e] = v;
    part += v;
  }
  const double S = block_sum(part, scratch);        // (block_sum synchronises: Js is complete)
  for (int k = tid; k < K; k += nt) {
    double r = 0.0, c = 0.0;
    for (int q = 0; q < K; ++q) {
      r += Js[(size_t)k * K + q];
      c += Js[(size_t)q * K + k];
    }
    pi[k] = r / S;
    pj[k] = c / S;
    gi[k] = log(pi[k] + eps) + pi[k] / (pi[k] + eps);
    gj[k] = log(pj[k] + eps) + pj[k] / (pj[k] + eps);
  }
  __syncthreads();
  // GP = g1*GP(lamb) + g2*GP(1) + gP ;  tot = sum GP * P
  double t_part = 0.0;
  for (size_t e = tid; e < KK; e += nt) {
    const int i = (int)(e / K), j = (int)(e % K);
    const double p = Js[e] / S;
    const double base = -log(p + eps) - p / (p + eps);
    const double mterm = gj[j] + gi[i];
    double v = g1 * (base + lamb * mterm) + g2 * (base + mterm);
    if (gP) v += (double)gP[e];
    Js[e] = v;                                       // each thread overwrites only the entries it has just read
    t_part += v * p;
  }
  const double tot = block_sum(t_part, scratch);    // (GP complete)
  for (size_t e = tid; e < KK; e += nt) {
    const int i = (int)(e / K), j = (int)(e % K);
    double v;
    if (symmetric) v = ((Js[e] - tot) / S + (Js[(size_t)j * K + i] - tot) / S) / 2.0;   // adjoint of (J + J^T)/2
    else v = (Js[e] - tot) / S;
    GJ[e] = (float)v;
  }
  __syncthreads();
  if constexpr (FL) {
    const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    float* px = rows_s + (size_t)wid * 2 * K;        // this warp's p rows of x and y
    float* py = px + K;
    for (long long n = r0 + wid; n < r1; n += nw) {
      const float* xr = x + n * x_sn;
      const float* yr = y + n * y_sn;
      float mx, rx, my, ry;
      warp_row_softmax_stats(xr, K, inv_temp, &mx, &rx);
      warp_row_softmax_stats(yr, K, inv_temp, &my, &ry);
      for (int k = lane; k < K; k += 32) {
        px[k] = logit_p(xr[k], inv_temp, mx, rx);
        py[k] = logit_p(yr[k], inv_temp, my, ry);
      }
      __syncwarp();
      // dp of the row (lane c takes channels c, c + 32, ...: K <= 128), then the two dot products
      float ax[4], ay[4];
      float dx = 0.f, dy = 0.f;
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int c = lane + 32 * h;
        ax[h] = 0.f; ay[h] = 0.f;
        if (c < K) {
          for (int q = 0; q < K; ++q) {
            ax[h] = fmaf(GJ[(size_t)c * K + q], py[q], ax[h]);
            ay[h] = fmaf(GJ[(size_t)q * K + c], px[q], ay[h]);
          }
          dx = fmaf(ax[h], px[c], dx);
          dy = fmaf(ay[h], py[c], dy);
        }
      }
      dx = warp_sum(dx);
      dy = warp_sum(dy);
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int c = lane + 32 * h;
        if (c < K) {
          gx[n * gx_sn + c] = inv_temp * px[c] * (ax[h] - dx);
          gy[n * gy_sn + c] = inv_temp * py[c] * (ay[h] - dy);
        }
      }
      __syncwarp();                                  // px / py are rewritten for the next row
    }
    return;
  }
  // gx[n][i] = sum_j GJ[i][j] y[n][j] ; gy[n][j] = sum_i GJ[i][j] x[n][i]
  const long long total = (r1 - r0) * K;
  for (long long e = tid; e < total; e += nt) {
    const long long n = r0 + e / K;
    const int c = (int)(e % K);
    const float* xr = staged_rows ? rows_s + (n - r0) * K : x + n * x_sn;
    const float* yr = staged_rows ? rows_s + slab + (n - r0) * K : y + n * y_sn;
    float ax = 0.f, ay = 0.f;
    for (int q = 0; q < K; ++q) {
      ax = fmaf(GJ[(size_t)c * K + q], yr[q], ax);
      ay = fmaf(GJ[(size_t)q * K + c], xr[q], ay);
    }
    gx[n * gx_sn + c] = ax;
    gy[n * gy_sn + c] = ay;
  }
}

static int global_grid(int device, long long N, long long* rows_per_cta) {
  int sms = sm_count_cached(device);
  if (sms <= 0) sms = 148;
  long long ctas = (N + 255) / 256;          // >= 256 rows per CTA before spreading over more SMs
  if (ctas > sms) ctas = sms;
  if (ctas < 1) ctas = 1;
  *rows_per_cta = (N + ctas - 1) / ctas;
  return (int)((N + *rows_per_cta - 1) / *rows_per_cta);
}

}  // namespace iic

using namespace iic;

extern "C" size_t iic_local_coeff_floats(int K, int pad, int n_patches) {
  if (K <= 0 || pad < 0 || n_patches <= 0) return 0;
  size_t img = 0;
  if (n_patches == 1) {
    img = local_bwd_tc_image_bytes(K, pad);
    const size_t rb = local_bwd_tcrb_image_bytes(K, pad);
    if (rb > img) img = rb;
  }
  if (img == 0) return local_coeff_base_floats(K, pad, n_patches);
  return local_coeff_image_offset(K, pad, n_patches) + (img + 3) / 4;
}

extern "C" size_t iic_local_epilogue_workspace_bytes(int K, int pad, int n_patches) {
  (void)K;
  const int T = 2 * pad + 1;
  return sizeof(EpiWorkspace) + (size_t)n_patches * T * T * sizeof(double);
}

extern "C" int iic_local_epilogue(const double* J, int K, int pad, int n_patches, double lamda,
                                  float* loss_out, double* loss64_out, float* Wx, float* Wy,
                                  double* GA_out, int* flags, void* workspace, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(J && loss_out && Wx && Wy && flags && workspace, "iic_local_epilogue: null pointer");
  IIC_REQUIRE(K > 0 && pad >= 0 && n_patches > 0, "iic_local_epilogue: bad sizes K=%d pad=%d patches=%d",
              K, pad, n_patches);
  const int T = 2 * pad + 1;
  const size_t smem = (40 + 3 * (size_t)K) * sizeof(double);
  local_epilogue_kernel<<<n_patches * T * T, 256, smem, st>>>(J, K, T, n_patches, lamda, loss_out,
                                                               loss64_out, Wx, Wy, GA_out, flags,
                                                               (EpiWorkspace*)workspace);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" size_t iic_global_joint_workspace_bytes(int device, long long N, int K) {
  long long rpc;
  const int ctas = global_grid(device, N > 0 ? N : 1, &rpc);
  return (size_t)ctas * K * K * sizeof(double);
}

extern "C" int iic_global_joint(const float* x, long long x_sn, const float* y, long long y_sn,
                                long long N, int K, double* J_out, void* workspace,
                                size_t workspace_bytes, int* flags, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(x && y && J_out, "iic_global_joint: null pointer");
  IIC_REQUIRE(N > 0 && K > 0, "iic_global_joint: empty input (N=%lld K=%d)", N, K);
  IIC_REQUIRE((long long)K * K <= 1024LL * GLOBAL_EPT, "iic_global_joint: K=%d too large (max 128)", K);
  long long rpc;
  const int ctas = global_grid(current_device(), N, &rpc);
  const size_t need = (size_t)ctas * K * K * sizeof(double);
  IIC_REQUIRE(workspace && workspace_bytes >= need, "iic_global_joint: workspace too small (%zu < %zu)",
              workspace_bytes, need);
  int nt = K * K;
  nt = nt > 1024 ? 1024 : ((nt + 31) & ~31);
  const size_t smem = 2 * (size_t)GLOBAL_ROWS * K * sizeof(float);
  if (nt < 2 * GLOBAL_ROWS) nt = 2 * GLOBAL_ROWS;          // one thread per staged row for the assertion
  // a single CTA (N <= 256 rows, the udaiic case) writes J directly: no partial slots, no reduce launch
  global_joint_kernel<<<ctas, nt, smem, st>>>(x, x_sn, y, y_sn, N, K, rpc, ctas == 1 ? J_out : (double*)workspace,
                                              flags);
  IIC_CHECK_CUDA(cudaGetLastError());
  if (ctas > 1) {
    global_reduce_kernel<<<(K * K + 255) / 256, 256, 0, st>>>((const double*)workspace, ctas, K * K, J_out);
    IIC_CHECK_CUDA(cudaGetLastError());
  }
  return 0;
}

extern "C" int iic_global_epilogue(const double* J, int K, double lamb, int symmetric,
                                   float* losses_out, float* P_out, int* flags, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(J && K > 0, "iic_global_epilogue: bad arguments");
  IIC_REQUIRE(!losses_out || flags, "iic_global_epilogue: flags required with losses_out");
  const size_t smem = (40 + 2 * (size_t)K) * sizeof(double);
  int nt = K * K;
  nt = nt > 1024 ? 1024 : ((nt + 31) & ~31);
  global_epilogue_kernel<<<1, nt, smem, st>>>(J, K, lamb, symmetric, losses_out, P_out, flags);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int iic_global_backward(const float* x, long long x_sn, const float* y, long long y_sn,
                                   long long N, int K, const double* J, double lamb, int symmetric,
                                   const float* g_loss, const float* g_no_lamb, const float* gP, float* gx,
                                   float* gy, long long gx_sn, long long gy_sn, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(x && y && J && gx && gy, "iic_global_backward: null pointer");
  IIC_REQUIRE(N > 0 && K > 0 && K <= 128, "iic_global_backward: bad sizes N=%lld K=%d", N, K);
  long long rpc;
  const int ctas = global_grid(current_device(), N, &rpc);
  const size_t smem = (40 + 4 * (size_t)K + (size_t)K * K) * sizeof(double) + ((size_t)K * K + 2 * GLOBAL_BWD_STAGE_FLOATS) * sizeof(float);
  auto kern = global_backward_kernel<false>;
  // opted in once per device, for the largest K the entry point takes (128)
  if (smem > 48 * 1024) IIC_CHECK_RC(ensure_dyn_smem((const void*)kern, (int)((40 + 4 * 128 + 128 * 128) * sizeof(double) + (128 * 128 + 2 * GLOBAL_BWD_STAGE_FLOATS) * sizeof(float))));
  if (gx_sn <= 0) gx_sn = K;            // 0 = dense rows
  if (gy_sn <= 0) gy_sn = K;
  kern<<<ctas, 256, smem, st>>>(x, x_sn, y, y_sn, N, K, J, lamb, symmetric, g_loss, g_no_lamb, gP, gx, gy, gx_sn, gy_sn, rpc,
                                1.f);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int iic_global_backward_from_logits(const float* x, long long x_sn, const float* y, long long y_sn,
                                               long long N, int K, const double* J, double lamb, int symmetric,
                                               float inv_temperature, const float* g_loss, const float* g_no_lamb,
                                               const float* gP, float* gx, float* gy, long long gx_sn, long long gy_sn,
                                               void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(x && y && J && gx && gy, "iic_global_backward_from_logits: null pointer");
  IIC_REQUIRE(N > 0 && K > 0 && K <= 128, "iic_global_backward_from_logits: bad sizes N=%lld K=%d", N, K);
  long long rpc;
  const int ctas = global_grid(current_device(), N, &rpc);
  // the probability form's layout; its row stage holds the 8 warps' p rows (2 * 8 * 128 <= 2 * GLOBAL_BWD_STAGE_FLOATS)
  const size_t smem = (40 + 4 * (size_t)K + (size_t)K * K) * sizeof(double) + ((size_t)K * K + 2 * GLOBAL_BWD_STAGE_FLOATS) * sizeof(float);
  auto kern = global_backward_kernel<true>;
  if (smem > 48 * 1024) IIC_CHECK_RC(ensure_dyn_smem((const void*)kern, (int)((40 + 4 * 128 + 128 * 128) * sizeof(double) + (128 * 128 + 2 * GLOBAL_BWD_STAGE_FLOATS) * sizeof(float))));
  if (gx_sn <= 0) gx_sn = K;            // 0 = dense rows
  if (gy_sn <= 0) gy_sn = K;
  kern<<<ctas, 256, smem, st>>>(x, x_sn, y, y_sn, N, K, J, lamb, symmetric, g_loss, g_no_lamb, gP, gx, gy, gx_sn, gy_sn, rpc,
                                inv_temperature);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
