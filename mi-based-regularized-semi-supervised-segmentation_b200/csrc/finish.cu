// iic_finish: everything between the joint kernels and the backward kernels of ONE OR MANY IIC loss terms in a single
// launch --
//   phase 1 (all CTAs)   fixed-order fp64 reduction of the joint kernels' per-CTA partial slots into the joints J
//                        (what reduce_partials_kernel / reduce_packed_kernel do per term), the small global joints
//                        x^T y computed directly from the (N, K) rows (contrastyou/losses/iic_loss.py:88-89) -- or from
//                        the cluster head's logits, each row turned into softmax(l * inv_temp) on the way; under data
//                        parallelism every value is also stored into this rank's slot of every peer's exchange buffer;
//   phase 2 (last CTA)   [data parallel: publish the sequence number to every peer, wait for theirs, add the ranks'
//                        slots in rank order -- csrc/xchg.cu's protocol, ONE exchange for all terms of the iteration]
//                        then the epilogues: local terms iic_loss.py:124-146,186 (min-shift, per-displacement normalise,
//                        symmetrise, marginals, entropy, dL/dJ as the two backward weight tensors), global terms
//                        iic_loss.py:56-69,91-92 (P, the two entropy expressions).
// The "last CTA" is found with a ticket (no CTA ever waits for another CTA of the grid, so nothing depends on
// co-residency); the only wait is the last CTA's bounded wait for the peers' flags.  One warp handles one displacement
// of one term, which is why the fused epilogue is limited to K <= 32; terms with more clusters take phase 1 (+ the
// exchange) here and the multi-CTA epilogue kernels of epilogue.cu afterwards.
#include "epilogue.cuh"
#include "xchg.cuh"

namespace iic {

constexpr int FIN_MAX_ITEMS = 32;
constexpr int FIN_THREADS = 1024;
constexpr int FIN_WARPS = FIN_THREADS / 32;
constexpr int FIN_MAX_K = 32;              // fused epilogue: one warp per displacement
constexpr int FIN_MAX_UNITS = 1024;        // (term, patch, displacement) triples with a fused epilogue
constexpr int FIN_MAX_PATCHES = 256;       // (term, patch) pairs with a fused epilogue
constexpr int FIN_SMALL_UNITS = 32;        // the last CTA runs the epilogues itself only for batches this small (one round of
                                           // its warps) whose joints fit its shared-memory stage; larger batches take the
                                           // multi-CTA batched epilogue kernel as a second launch
constexpr int FIN_BIG_MAX_UNITS = 16384;   // displacement units of one batched epilogue launch (workspace: one double each)
constexpr size_t FIN_WS_TICKETS = 64;      // workspace: [0] phase-1 ticket, [1] rank-sum ticket; per-term tickets from here
constexpr size_t FIN_WS_LOSSES = 256;      // workspace: unit losses from here
constexpr int FIN_GLOBAL_LOGITS_MAX_N = 4096;    // rows of a global term from logits (ops.py: GLOBAL_ROWS_MAX)
constexpr int FIN_GL_EPT = 8;              // joint entries per thread and pass of a global term from logits
constexpr int FIN_PST_FLOATS = FIN_WARPS * 3 * FIN_MAX_K * 2;   // p rows staged by a global term from logits (wscratch)

struct FinItem {
  const float* slots;            // local terms: per-CTA partial joints
  const float* x;                // global terms: the (N, K) rows
  const float* y;
  long long x_sn, y_sn, N;
  double* J;                     // this term's joint inside the packed buffer (E doubles)
  float* loss_out;               // local [1]; global [2] = loss(lamb), loss_no_lamb
  float* Wx;                     // local: backward coefficients (iic_local_epilogue's layout)
  float* Wy;
  float* P_out;                  // global: (K, K) float32, nullable
  long long E;                   // local n_patches*T*T*K*K; global K*K
  long long slot_stride;
  int kind;                      // IIC_ITEM_LOCAL / IIC_ITEM_GLOBAL_ROWS (also for IIC_ITEM_GLOBAL_LOGITS: see inv_temp)
  int layout, n_slots, nb;
  int K, T, n_patches, symmetric, check_simplex;
  float inv_temp;                // > 0: a global term whose x / y hold logits, its joint that of softmax(l * inv_temp);
                                 // 0: probability rows.  (In the padding before lamda: the struct keeps its layout.)
  double lamda;
};

struct FinBatch {
  FinItem it[FIN_MAX_ITEMS];
  int n;
  int do_epilogue;
  long long E_total;
  double* J_all;                 // packed joints: item i's J = J_all + (sum of E of the items before it)
  int* flags;
  unsigned int* ticket;          // self-resetting arrival counter (workspace)
  int rank, world;
  int xchg_mode;                 // 1: the last CTA exchanges and sums (small batches); 2: it only publishes (xchg_sum_kernel follows)
  long long capacity;
  unsigned long long timeout_ns;
  XchgPeers peers;
};

// ---- phase 1 ------------------------------------------------------------------------------------------------------------
// One unit = 32 consecutive slot elements of one patch of one local term (1024 threads = 32 slot groups x 32 elements,
// coalesced 128-byte reads; group g adds slots g, g+32, ... in order, then the 32 group sums are added in order), or
// one whole global term.
__device__ __forceinline__ void store_joint(const FinBatch& B, const FinItem& it, long long e, double v, int par) {
  it.J[e] = v;
  // small batches publish from the last CTA (one system-scope fence on the critical path instead of one per CTA before the
  // ticket plus one after it); large batches publish from every CTA as they go
  if (B.world > 1 && B.xchg_mode == 2) {
    const long long off = (it.J - B.J_all) + e;
    for (int p = 0; p < B.world; ++p) xchg_slot(B.peers.base[p], par, B.world, B.rank, B.capacity)[off] = v;
  }
}

__device__ void reduce_unit(const FinBatch& B, const FinItem& it, long long unit, double (*sm)[33], int par) {
  const int le = threadIdx.x & 31, sg = threadIdx.x >> 5;
  const long long Eper = it.E / it.n_patches;            // T*T*K*K
  long long span = Eper;                                  // elements walked per patch, in slot order
  if (it.layout == SLOT_TC128) span = Eper;
  const long long chunks = (span + 31) / 32;
  const int patch = (int)(unit / chunks);
  const long long s = (unit - (long long)patch * chunks) * 32 + le;
  double acc[4] = {0, 0, 0, 0};
  long long dst = -1;
  if (s < span) {
    size_t off;
    if (it.layout == SLOT_PACKED) {
      const int K = it.K, T = it.T;
      const int j = (int)(s % K), i = (int)((s / K) % K), dx = (int)((s / ((long long)K * K)) % T), dy = (int)(s / ((long long)K * K * T));
      const int row = i * T + dx, col = j * T + (T - 1 - dy);
      off = packed_slot_index(row >> 7, row & 127, col, it.nb);
      dst = s;
    } else {
      off = (size_t)s;
      dst = it.layout == SLOT_TC128 ? tc128_out_index(s) : s;
    }
    const float* src = it.slots + (size_t)patch * it.n_slots * it.slot_stride + off;
    int c = sg;
    for (; c + 3 * FIN_WARPS < it.n_slots; c += 4 * FIN_WARPS) {
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[q] += (double)__ldg(src + (size_t)(c + q * FIN_WARPS) * it.slot_stride);
    }
    for (int q = 0; c < it.n_slots; c += FIN_WARPS, ++q) acc[q] += (double)__ldg(src + (size_t)c * it.slot_stride);
  }
  __syncthreads();                                       // sm is reused from the previous unit
  sm[sg][le] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
  __syncthreads();
  if (sg == 0 && s < span) {
    double t = 0;
#pragma unroll
    for (int g = 0; g < FIN_WARPS; ++g) t += sm[g][le];
    store_joint(B, it, (long long)patch * Eper + dst, t, par);
  }
}

// J = x^T y of one global term, fp64, rows walked in order by every thread (deterministic); both simplex assertions
// (iic_loss.py:50-51,82-83) ride along
__device__ void global_rows_unit(const FinBatch& B, const FinItem& it, double* scratch /* FIN_WARPS*33 doubles */, int par) {
  const int K = it.K, KK = K * K;
  // G row groups x K*K entries: group g walks rows g, g+G, ... (short dependent chains), then entry e adds the G
  // partial sums in group order -- a fixed order, so the result is deterministic
  int G = FIN_THREADS / KK;
  if (G > FIN_WARPS * 33 / KK) G = FIN_WARPS * 33 / KK;
  if (G < 1) G = 1;
  __syncthreads();
  if (G == 1) {
    for (int e = threadIdx.x; e < KK; e += FIN_THREADS) {
      const int i = e / K, j = e - i * K;
      double a = 0.0;
      for (long long n = 0; n < it.N; ++n) a += (double)__ldg(it.x + n * it.x_sn + i) * (double)__ldg(it.y + n * it.y_sn + j);
      store_joint(B, it, e, a, par);
    }
  } else {
    const int g = threadIdx.x / KK, e = threadIdx.x - g * KK;
    if (g < G) {
      const int i = e / K, j = e - i * K;
      double a = 0.0;
      for (long long n = g; n < it.N; n += G) a += (double)__ldg(it.x + n * it.x_sn + i) * (double)__ldg(it.y + n * it.y_sn + j);
      scratch[g * KK + e] = a;
    }
    __syncthreads();
    if (threadIdx.x < KK) {
      double t = 0.0;
      for (int q = 0; q < G; ++q) t += scratch[q * KK + threadIdx.x];
      store_joint(B, it, threadIdx.x, t, par);
    }
  }
  if (B.flags && it.check_simplex) {
    bool bad = false;
    for (long long r = threadIdx.x; r < 2 * it.N; r += FIN_THREADS) {
      const float* row = r < it.N ? it.x + r * it.x_sn : it.y + (r - it.N) * it.y_sn;
      float sum = 0.f;
      for (int c = 0; c < K; ++c) sum += __ldg(row + c);
      if (!(fabsf(sum - 1.f) <= 1e-4f + 1e-4f * 1.f)) bad = true;
    }
    if (bad) atomicOr(B.flags, IIC_FLAG_NOT_SIMPLEX);
  }
}

// The same joint from LOGIT rows: the rows are turned into p = softmax(l * inv_temp) chunk by chunk (one warp per row,
// warp_row_softmax_stats + logit_p: the p global_backward_kernel<true> recomputes, bit for bit) into `pst`, then
// accumulated in fp64 in a fixed order as above -- group g takes the rows n = g mod G of every chunk in increasing n.
// With one group (K > 32) a thread holds at most FIN_GL_EPT entries, so K*K > FIN_GL_EPT * 1024 (K > 90) takes more than
// one pass over the rows (finish_kernel runs at 64 registers per thread: with 8 accumulators ptxas reports 68 / 60 bytes
// of spill stores / loads, against 44 / 40 without this unit and 140 / 184 with 16).  No simplex assertion: a softmax
// row is a simplex by construction.
__device__ void global_logit_rows_unit(const FinBatch& B, const FinItem& it, double* scratch /* FIN_WARPS*33 doubles */,
                                       float* pst /* FIN_PST_FLOATS */, int par) {
  const int K = it.K, KK = K * K;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int G = FIN_THREADS / KK;
  if (G > FIN_WARPS * 33 / KK) G = FIN_WARPS * 33 / KK;
  if (G < 1) G = 1;
  const int g = threadIdx.x / KK;                         // G == 1: group 0 holds entries e = tid + q * FIN_THREADS
  const int e0 = G == 1 ? threadIdx.x : threadIdx.x - g * KK;
  const int rows_per_chunk = FIN_PST_FLOATS / (2 * K);
  const int per_pass = G == 1 ? FIN_GL_EPT * FIN_THREADS : KK;
  for (int eb = 0; eb < KK; eb += per_pass) {
    double acc[FIN_GL_EPT];
#pragma unroll
    for (int q = 0; q < FIN_GL_EPT; ++q) acc[q] = 0.0;
    __syncthreads();                                      // pst and scratch are reused from the previous unit / pass
    for (long long n0 = 0; n0 < it.N; n0 += rows_per_chunk) {
      const int nr = (int)(it.N - n0 < rows_per_chunk ? it.N - n0 : rows_per_chunk);
      for (int rr = wid; rr < 2 * nr; rr += FIN_WARPS) {  // x rows of the chunk at pst[0 .. nr*K), then its y rows
        const float* row = rr < nr ? it.x + (n0 + rr) * it.x_sn : it.y + (n0 + rr - nr) * it.y_sn;
        float m, r;
        warp_row_softmax_stats(row, K, it.inv_temp, &m, &r);
        for (int k = lane; k < K; k += 32) pst[rr * K + k] = logit_p(row[k], it.inv_temp, m, r);
      }
      __syncthreads();
      const float* px = pst;
      const float* py = pst + (size_t)nr * K;
      if (g < G) {
        const int nfirst = (int)((g - n0 % G + G) % G);
#pragma unroll
        for (int q = 0; q < FIN_GL_EPT; ++q) {
          const int e = eb + e0 + q * FIN_THREADS;
          if ((q == 0 || G == 1) && e < KK) {
            const int i = e / K, j = e - i * K;
            double a = acc[q];
            for (int n = nfirst; n < nr; n += G) a += (double)px[n * K + i] * (double)py[n * K + j];
            acc[q] = a;
          }
        }
      }
      __syncthreads();
    }
    if (G == 1) {
#pragma unroll
      for (int q = 0; q < FIN_GL_EPT; ++q) {
        const int e = eb + e0 + q * FIN_THREADS;
        if (g == 0 && e < KK) store_joint(B, it, e, acc[q], par);
      }
    } else {
      if (g < G) scratch[g * KK + e0] = acc[0];
      __syncthreads();
      if (threadIdx.x < KK) {
        double t = 0.0;
        for (int q = 0; q < G; ++q) t += scratch[q * KK + threadIdx.x];
        store_joint(B, it, threadIdx.x, t, par);
      }
    }
  }
}

__device__ __forceinline__ long long item_units(const FinItem& it) {
  if (it.kind == IIC_ITEM_GLOBAL_ROWS) return 1;
  const long long Eper = it.E / it.n_patches;
  return (long long)it.n_patches * ((Eper + 31) / 32);
}

// J was written by other CTAs of this launch (and, after an exchange, summed by this one): read it past L1 -- unless
// the last CTA has staged all joints in shared memory (small batches: config 2's 1000 doubles), where `p` points there
__device__ __forceinline__ double ldj(const double* p, bool staged) { return staged ? *p : __ldcg(p); }

// ---- phase 2: epilogues, one warp per (term, patch, displacement) -----------------------------------------------------------
// Same arithmetic as local_epilogue_kernel (epilogue.cu); sc = 3*K doubles of per-warp scratch.
__device__ double warp_local_displacement(const double* __restrict__ Jp, bool staged, int d, int K, int T, double m,
                                          double lamda, double scale, float* __restrict__ Wxp, float* __restrict__ Wyp,
                                          double* sc) {
  const int lane = threadIdx.x & 31;
  const int KK = K * K, T2 = T * T, Kp = (K + 3) & ~3;
  const double* Jd = Jp + (size_t)d * KK;
  const double eps = 1e-16;
  double* marg = sc;
  double* lm = sc + K;
  double* gm = sc + 2 * K;
  double part = 0.0;
  for (int k = lane; k < K; k += 32) {
    double rs = 0.0, cs = 0.0;
    for (int q = 0; q < K; ++q) {
      rs += ldj(Jd + k * K + q, staged) - m + 1e-16;
      cs += ldj(Jd + q * K + k, staged) - m + 1e-16;
    }
    marg[k] = rs + cs;
    part += rs;
  }
  const double s = warp_sum(part);
  const double inv_2s = 1.0 / (2.0 * s), inv_s = 2.0 * inv_2s;
  for (int k = lane; k < K; k += 32) {
    const double mk = marg[k] * inv_2s;
    marg[k] = mk;
    lm[k] = log(mk + eps);
    gm[k] = lm[k] + mk / (mk + eps);
  }
  __syncwarp();
  // pass 1 over the padded (cin, cout) grid the coefficient tensors use: loss, tot = sum GQ * Q, and GQ itself parked
  // (as float, it is read back by the same lane) in its final Wy slot -- the second log per entry is gone
  const int dy = d / T, dx = d - dy * T;
  const int dflip = (T - 1 - dy) * T + (T - 1 - dx);
  double l_part = 0.0, t_part = 0.0;
  for (int e = lane; e < K * Kp; e += 32) {
    const int i = e / Kp, j = e - i * Kp;                // i = cin, j = cout (padded)
    float gqf = 0.f;
    if (j < K) {
      const double a = ldj(Jd + i * K + j, staged) - m + 1e-16, at = ldj(Jd + j * K + i, staged) - m + 1e-16;
      const double p = (a + at) * inv_2s;
      const double lp = log(p + eps);
      l_part += -p * (lp - lamda * lm[j] - lamda * lm[i]);
      const double gq = -lp - p / (p + eps) + lamda * (gm[j] + gm[i]);
      t_part += gq * (a * inv_s);
      gqf = (float)gq;
    }
    Wyp[((size_t)i * T2 + d) * Kp + j] = gqf;
  }
  const double loss_d = warp_sum(l_part);
  const double tot = warp_sum(t_part);
  const double cs = inv_s * scale;
  // pass 2: GA = dL/dJ_d = (GQ - tot) / s, scaled by 1/(T^2 n_patches), in the two sweep layouts
  //    Wy[cin=i][dy*T+dx][j]   and   Wx[cin=j][(T-1-dy)*T+(T-1-dx)][i]  (GA is symmetric in (i, j))
  for (int e = lane; e < K * Kp; e += 32) {
    const int i = e / Kp, j = e - i * Kp;
    float* wy = Wyp + ((size_t)i * T2 + d) * Kp + j;
    const float w = j < K ? (float)(((double)*wy - tot) * cs) : 0.f;
    *wy = w;
    Wxp[((size_t)i * T2 + dflip) * Kp + j] = w;
  }
  __syncwarp();
  return loss_d;
}

// global term: P = sym(J)/S, the two entropy expressions (global_epilogue_kernel's arithmetic); sc = 2*K doubles
__device__ void warp_global_term(const FinItem& it, const double* J, bool staged, int* flags, double* sc) {
  const int lane = threadIdx.x & 31;
  const int K = it.K, KK = K * K;
  const double eps = 1e-10, lamb = it.lamda;
  const bool sym = it.symmetric != 0;
  auto Jsym = [&](int i, int j) { return sym ? (ldj(J + i * K + j, staged) + ldj(J + j * K + i, staged)) / 2.0 : ldj(J + i * K + j, staged); };
  double part = 0.0;
  for (int e = lane; e < KK; e += 32) part += Jsym(e / K, e % K);
  const double S = warp_sum(part);
  double* pi = sc;
  double* pj = sc + K;
  for (int k = lane; k < K; k += 32) {
    double r = 0.0, c = 0.0;
    for (int q = 0; q < K; ++q) {
      r += Jsym(k, q);
      c += Jsym(q, k);
    }
    // the logs of the marginals, once per cluster (they were taken per ENTRY: 3 fp64 logs for each of the K*K entries made
    // this one warp the critical path of the whole finish launch, ~10 us at K = 10)
    pi[k] = log(r / S + eps);
    pj[k] = log(c / S + eps);
  }
  __syncwarp();
  const double inv_S = 1.0 / S;
  double l1 = 0.0, l2 = 0.0;
  for (int e = lane; e < KK; e += 32) {
    const int i = e / K, j = e - i * K;
    const double p = Jsym(i, j) * inv_S;
    if (it.P_out) it.P_out[e] = (float)p;
    const double lp = log(p + eps), lj = pj[j], li = pi[i];
    l1 += -p * (lp - lamb * lj - lamb * li);
    l2 += -p * (lp - lj - li);
  }
  const double L1 = warp_sum(l1), L2 = warp_sum(l2);
  if (lane == 0 && it.loss_out) {
    it.loss_out[0] = (float)L1;
    it.loss_out[1] = (float)L2;
    if ((L1 != L1 || L2 != L2) && flags) atomicOr(flags, IIC_FLAG_NAN_LOSS);
  }
  __syncwarp();
}

#ifdef IIC_FIN_TRACE
__device__ unsigned long long g_fin_trace[16];
__device__ __forceinline__ unsigned long long fin_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define FIN_T(i) do { if (threadIdx.x == 0) g_fin_trace[i] = fin_now(); } while (0)
#else
#define FIN_T(i) do { } while (0)
#endif

__global__ void __launch_bounds__(FIN_THREADS, 1) finish_kernel(const __grid_constant__ FinBatch B) {
  __shared__ double sm[FIN_WARPS][33];
  __shared__ double unit_loss[FIN_MAX_UNITS];
  __shared__ double patch_min[FIN_MAX_PATCHES];
  __shared__ double wscratch[FIN_WARPS][3 * FIN_MAX_K];
  __shared__ double red_scratch[40];
  __shared__ unsigned long long seq_s;
  __shared__ int last_s;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
#ifdef IIC_FIN_TRACE
  if (tid == 0) atomicMin(&g_fin_trace[0], fin_now());
#endif

  XchgHeader* hdr = nullptr;
  int par = 0;
  unsigned long long seq = 0;
  if (B.world > 1) {
    hdr = reinterpret_cast<XchgHeader*>(B.peers.base[B.rank]);
    if (tid == 0) seq_s = *reinterpret_cast<volatile unsigned long long*>(&hdr->seq) + 1;   // advanced by the last CTA
    __syncthreads();
    seq = seq_s;
    par = (int)(seq & 1ull);
  }

  // ---- phase 1 ----
  {
    long long base = 0;
    for (int i = 0; i < B.n; ++i) {
      const FinItem& it = B.it[i];
      const long long nu = item_units(it);
      // units base .. base+nu-1 of this item; this CTA takes those congruent to its index
      long long first = blockIdx.x - (base % gridDim.x);
      if (first < 0) first += gridDim.x;
      for (long long u = first; u < nu; u += gridDim.x) {
        if (it.kind == IIC_ITEM_GLOBAL_ROWS) {
          if (it.inv_temp > 0.f) global_logit_rows_unit(B, it, &sm[0][0], reinterpret_cast<float*>(&wscratch[0][0]), par);
          else global_rows_unit(B, it, &sm[0][0], par);
        } else {
          reduce_unit(B, it, u, sm, par);
        }
      }
      base += nu;
    }
  }
#ifdef IIC_FIN_TRACE
  if (tid == 0) atomicMax(&g_fin_trace[1], fin_now());
  if (tid == 0 && blockIdx.x == 0) g_fin_trace[7] = fin_now();                 // a CTA with one local unit
  if (tid == 0 && blockIdx.x == gridDim.x - 1) g_fin_trace[8] = fin_now();     // (900 elements = 29 units: the global item is unit 29 -> CTA 0 again)
#endif
  if (B.world > 1 && B.xchg_mode == 2) __threadfence_system(); else __threadfence();
  __syncthreads();
  if (tid == 0) last_s = (atomicAdd(B.ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  FIN_T(2);

  // ---- phase 2, last CTA only ----
  if (B.world > 1) {
    if (B.xchg_mode == 2) {
      __threadfence_system();
    } else {
      // this rank's joints (just reduced by all CTAs, L2-resident) into its slot of every rank's buffer
      for (long long e = tid; e < B.E_total; e += FIN_THREADS) {
        const double v = __ldcg(B.J_all + e);
        for (int p = 0; p < B.world; ++p) xchg_slot(B.peers.base[p], par, B.world, B.rank, B.capacity)[e] = v;
      }
      __syncthreads();
      if (tid < B.world) __threadfence_system();      // cumulative: the CTA's stores above are ordered before the flags
    }
    if (tid < B.world) {
      XchgHeader* ph = reinterpret_cast<XchgHeader*>(B.peers.base[tid]);
      st_release_sys(&ph->flags[par][B.rank], seq);
    }
    if (B.xchg_mode == 2) {                            // large batch: xchg_sum_kernel waits and sums with all SMs
      if (tid == 0) *B.ticket = 0;
      return;
    }
    if (tid < B.world) {
      // a slow peer is waited for; the bound only keeps a dead peer from hanging the GPU and is reported as a flag
      if (!xchg_wait_flag(hdr, par, tid, seq, B.timeout_ns) && B.flags) atomicOr(B.flags, IIC_FLAG_XCHG_TIMEOUT);
    }
    __syncthreads();
    const double* src = xchg_slot(B.peers.base[B.rank], par, B.world, 0, B.capacity);
    const bool stage_now = B.do_epilogue && B.E_total <= (long long)(FIN_WARPS * 33);   // the epilogue below reads shared memory
    for (long long e = tid; e < B.E_total; e += FIN_THREADS) {
      double s = 0.0;
      for (int r = 0; r < B.world; ++r) s += __ldcg(src + (size_t)r * B.capacity + e);     // rank order: bit-identical everywhere
      B.J_all[e] = s;
      if (stage_now) (&sm[0][0])[e] = s;
    }
    __syncthreads();
    if (tid == 0) *reinterpret_cast<volatile unsigned long long*>(&hdr->seq) = seq;
  }
  if (tid == 0) *B.ticket = 0;
  if (!B.do_epilogue) return;
  __syncthreads();

  // small batches (config 2: 900 + 100 doubles): all joints into shared memory -- the phase-1 scratch is free now
  const bool staged = B.E_total <= (long long)(FIN_WARPS * 33);
  double* Js = &sm[0][0];
  if (staged && B.world == 1) {                         // (with several ranks the rank sum above has filled Js)
    for (long long e = tid; e < B.E_total; e += FIN_THREADS) Js[e] = __ldcg(B.J_all + e);
    __syncthreads();
  }
  const double* Jbase = staged ? Js : B.J_all;
  FIN_T(3);

  // per (term, patch): m = min over every displacement and both cluster axes (iic_loss.py:124), NaN-propagating
  int npatch_total = 0;
  for (int i = 0; i < B.n; ++i) {
    const FinItem& it = B.it[i];
    if (it.kind != IIC_ITEM_LOCAL) continue;
    const long long Eper = it.E / it.n_patches;
    for (int p = 0; p < it.n_patches; ++p, ++npatch_total) {
      const double* Jp = Jbase + (it.J - B.J_all) + (size_t)p * Eper;
      double mn = __longlong_as_double(0x7ff0000000000000LL);
      bool has_nan = false;
      for (long long e = tid; e < Eper; e += FIN_THREADS) {
        const double v = ldj(Jp + e, staged);
        has_nan |= (v != v);
        mn = fmin(mn, v);
      }
      const double m = block_min_nan(mn, has_nan, red_scratch);
      if (tid == 0) patch_min[npatch_total] = m;
    }
  }
  __syncthreads();
  FIN_T(4);

  // displacement units, dealt to the warps round robin
  {
    int ubase = 0, pbase = 0;
    for (int i = 0; i < B.n; ++i) {
      const FinItem& it = B.it[i];
      if (it.kind == IIC_ITEM_GLOBAL_ROWS) {
        if ((ubase % FIN_WARPS) == wid) warp_global_term(it, Jbase + (it.J - B.J_all), staged, B.flags, wscratch[wid]);
        ubase += 1;
        continue;
      }
      const int T2 = it.T * it.T, Kp = (it.K + 3) & ~3;
      const int nu = it.n_patches * T2;
      const long long Eper = it.E / it.n_patches;
      const double scale = 1.0 / ((double)T2 * (double)it.n_patches);
      int first = wid - (ubase % FIN_WARPS);
      if (first < 0) first += FIN_WARPS;
      for (int u = first; u < nu; u += FIN_WARPS) {
        const int p = u / T2, d = u - p * T2;
        const double ld = warp_local_displacement(Jbase + (it.J - B.J_all) + (size_t)p * Eper, staged, d, it.K, it.T,
                                                  patch_min[pbase + p], it.lamda, scale,
                                                  it.Wx + (size_t)p * it.K * T2 * Kp, it.Wy + (size_t)p * it.K * T2 * Kp,
                                                  wscratch[wid]);
        if (lane == 0) unit_loss[ubase + u] = ld;
      }
      ubase += nu;
      pbase += it.n_patches;
    }
  }
  __syncthreads();
  FIN_T(5);
  // per local term: the displacement losses in index order (deterministic), mean over displacements and patches
  // (one warp per term, lanes over its units, a fixed shuffle tree: deterministic, and not a serial chain of fp64 adds)
  for (int t = wid; t < B.n; t += FIN_WARPS) {
    FIN_T(10);
    int ubase = 0;
    for (int i = 0; i < t; ++i) ubase += B.it[i].kind == IIC_ITEM_GLOBAL_ROWS ? 1 : B.it[i].n_patches * B.it[i].T * B.it[i].T;
    const FinItem& it = B.it[t];
    if (it.kind == IIC_ITEM_LOCAL) {
      const int nu = it.n_patches * it.T * it.T;
      double part = 0.0;
      for (int u = lane; u < nu; u += 32) part += unit_loss[ubase + u];
      double total = warp_sum(part);
      total *= 1.0 / ((double)nu);
      FIN_T(9);
      if (lane == 0) {
        it.loss_out[0] = (float)total;
        if (total != total && B.flags) atomicOr(B.flags, IIC_FLAG_NAN_LOSS);
      }
    }
  }
  FIN_T(6);
}

#ifdef IIC_FIN_TRACE
extern "C" int iic_debug_fin_trace(unsigned long long* host16, int reset) {
  if (reset) {
    unsigned long long z[16];
    for (int i = 0; i < 16; ++i) z[i] = 0;
    z[0] = ~0ull;
    return cudaMemcpyToSymbol(g_fin_trace, z, sizeof(z)) == cudaSuccess ? 0 : 1;
  }
  return cudaMemcpyFromSymbol(host16, g_fin_trace, 16 * sizeof(unsigned long long)) == cudaSuccess ? 0 : 1;
}
#endif

// ---- large batches -----------------------------------------------------------------------------------------------------
// Second half of the exchange with all SMs: wait for every rank's flag, add the ranks' slots in rank order, last CTA
// advances the sequence counter.
__global__ void __launch_bounds__(FIN_THREADS) xchg_sum_kernel(double* __restrict__ J_all, long long E_total, XchgPeers peers,
                                                               int rank, int world, long long capacity,
                                                               unsigned long long timeout_ns, int* __restrict__ flags,
                                                               unsigned int* __restrict__ ticket) {
  XchgHeader* hdr = reinterpret_cast<XchgHeader*>(peers.base[rank]);
  __shared__ unsigned long long seq_s;
  __shared__ int last_s;
  if (threadIdx.x == 0) seq_s = *reinterpret_cast<volatile unsigned long long*>(&hdr->seq) + 1;
  __syncthreads();
  const unsigned long long seq = seq_s;
  const int par = (int)(seq & 1ull);
  if (threadIdx.x < world && !xchg_wait_flag(hdr, par, threadIdx.x, seq, timeout_ns) && flags) atomicOr(flags, IIC_FLAG_XCHG_TIMEOUT);
  __syncthreads();
  const double* src = xchg_slot(peers.base[rank], par, world, 0, capacity);
  for (long long e = (long long)blockIdx.x * FIN_THREADS + threadIdx.x; e < E_total; e += (long long)gridDim.x * FIN_THREADS) {
    double s = 0.0;
    for (int r = 0; r < world; ++r) s += __ldcg(src + (size_t)r * capacity + e);
    J_all[e] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last_s = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (last_s && threadIdx.x == 0) {
    *ticket = 0;
    *reinterpret_cast<volatile unsigned long long*>(&hdr->seq) = seq;      // every CTA has read it by now
  }
}

// All epilogues of a batch, one CTA per (term, patch, displacement) / per global term -- the arithmetic of
// local_epilogue_kernel / global_epilogue_kernel (epilogue.cuh).  Per term, the last of its CTAs adds the displacement
// losses in index order.
__global__ void __launch_bounds__(256) batched_epilogue_kernel(const __grid_constant__ FinBatch B, unsigned int* __restrict__ tickets,
                                                               double* __restrict__ unit_loss) {
  extern __shared__ __align__(16) double esm[];
  __shared__ int last_s;
  int item = 0, ubase = 0;
  for (; item < B.n; ++item) {
    const int nu = B.it[item].kind == IIC_ITEM_GLOBAL_ROWS ? 1 : B.it[item].n_patches * B.it[item].T * B.it[item].T;
    if ((int)blockIdx.x < ubase + nu) break;
    ubase += nu;
  }
  if (item >= B.n) return;
  const FinItem& it = B.it[item];
  if (it.kind == IIC_ITEM_GLOBAL_ROWS) {
    global_epilogue_block(it.J, it.K, it.lamda, it.symmetric, it.loss_out, it.P_out, B.flags, esm);
    return;
  }
  const int T2 = it.T * it.T, Kp = (it.K + 3) & ~3;
  const int u = (int)blockIdx.x - ubase, p = u / T2, d = u - p * T2, nu = it.n_patches * T2;
  const long long Eper = it.E / it.n_patches;
  const double scale = 1.0 / ((double)T2 * (double)it.n_patches);
  const double loss_d = local_epilogue_block(it.J + (size_t)p * Eper, it.K, it.T, d, it.lamda, scale,
                                             it.Wx + (size_t)p * it.K * T2 * Kp, it.Wy + (size_t)p * it.K * T2 * Kp, nullptr, esm);
  if (threadIdx.x == 0) {
    unit_loss[blockIdx.x] = loss_d;
    __threadfence();
    last_s = (atomicAdd(&tickets[item], 1u) == (unsigned)nu - 1) ? 1 : 0;
  }
  __syncthreads();
  if (last_s && threadIdx.x == 0) {
    __threadfence();
    const volatile double* pl = unit_loss + ubase;
    double total = 0.0;
    for (int q = 0; q < nu; ++q) total += pl[q];
    total *= scale;
    it.loss_out[0] = (float)total;
    if (total != total && B.flags) atomicOr(B.flags, IIC_FLAG_NAN_LOSS);
    tickets[item] = 0;
  }
}

}  // namespace iic

using namespace iic;

extern "C" size_t iic_finish_workspace_bytes(void) { return FIN_WS_LOSSES + (size_t)FIN_BIG_MAX_UNITS * sizeof(double); }

extern "C" int iic_finish(const iic_finish_item* items_host, int n_items, double* J_all, long long E_total, int* flags,
                          void* workspace, void* const* xchg_bufs_host, int rank, int world, long long xchg_capacity,
                          int want_epilogue, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(items_host && n_items > 0 && J_all && workspace, "iic_finish: null pointer or empty batch");
  IIC_REQUIRE(n_items <= FIN_MAX_ITEMS, "iic_finish: %d terms exceed the %d of one launch (split the batch)", n_items, FIN_MAX_ITEMS);
  IIC_REQUIRE(world >= 1 && world <= XCHG_MAXR && rank >= 0 && rank < world, "iic_finish: bad rank %d / world %d", rank, world);
  IIC_REQUIRE(world == 1 || (xchg_bufs_host && E_total <= xchg_capacity),
              "iic_finish: %lld joint entries exceed the exchange capacity %lld", E_total, xchg_capacity);
  FinBatch B;
  memset(&B, 0, sizeof(B));
  B.n = n_items;
  B.E_total = E_total;
  B.J_all = J_all;
  B.flags = flags;
  B.ticket = reinterpret_cast<unsigned int*>(workspace);
  B.rank = rank;
  B.world = world;
  B.capacity = xchg_capacity;
  B.timeout_ns = (unsigned long long)options().xchg_timeout_ms * 1000000ull;
  for (int r = 0; r < world && world > 1; ++r) {
    B.peers.base[r] = (unsigned char*)xchg_bufs_host[r];
    IIC_REQUIRE(B.peers.base[r], "iic_finish: exchange buffer of rank %d is not mapped", r);
  }
  long long off = 0, units = 0, epi_units = 0, epi_patches = 0;
  bool fused = want_epilogue != 0 && !options().no_fused_epilogue;
  for (int i = 0; i < n_items; ++i) {
    const iic_finish_item& s = items_host[i];
    FinItem& d = B.it[i];
    IIC_REQUIRE(s.kind == IIC_ITEM_LOCAL || s.kind == IIC_ITEM_GLOBAL_ROWS || s.kind == IIC_ITEM_GLOBAL_LOGITS,
                "iic_finish: term %d has unknown kind %d", i, s.kind);
    IIC_REQUIRE(s.K > 0, "iic_finish: term %d has K = %d", i, s.K);
    // a global term from logits is a global term whose phase-1 unit applies the softmax first
    const bool logits = s.kind == IIC_ITEM_GLOBAL_LOGITS;
    IIC_REQUIRE(!logits || (s.inv_temperature > 0.f && s.inv_temperature <= 3.0e38f),
                "iic_finish: global term %d from logits needs a positive, finite inv_temperature", i);
    d.kind = logits ? IIC_ITEM_GLOBAL_ROWS : s.kind;
    d.inv_temp = logits ? s.inv_temperature : 0.f;
    d.K = s.K;
    d.lamda = s.lamda;
    d.J = J_all + off;
    d.loss_out = s.loss_out;
    if (s.kind == IIC_ITEM_LOCAL) {
      IIC_REQUIRE(s.slots && s.n_slots > 0 && s.n_patches > 0 && s.pad >= 0 && s.pad <= 7, "iic_finish: term %d is malformed", i);
      IIC_REQUIRE(!want_epilogue || (s.loss_out && s.Wx && s.Wy), "iic_finish: term %d lacks its epilogue outputs", i);
      IIC_REQUIRE(s.layout == SLOT_STD || s.n_patches == 1, "iic_finish: term %d: only the standard slot layout has patches", i);
      d.slots = s.slots;
      d.layout = s.layout;
      d.n_slots = s.n_slots;
      d.slot_stride = s.slot_stride;
      d.nb = s.nb;
      d.T = 2 * s.pad + 1;
      d.n_patches = s.n_patches;
      d.E = (long long)s.n_patches * d.T * d.T * s.K * s.K;
      d.Wx = s.Wx;
      d.Wy = s.Wy;
      epi_units += (long long)s.n_patches * d.T * d.T;
      epi_patches += s.n_patches;
    } else {
      IIC_REQUIRE(s.x && s.y && s.N > 0, "iic_finish: global term %d is malformed", i);
      IIC_REQUIRE(s.K <= FIN_MAX_K * 4 && s.N <= (1 << 20), "iic_finish: global term %d too large for the direct joint", i);
      IIC_REQUIRE(!logits || s.N <= FIN_GLOBAL_LOGITS_MAX_N,
                  "iic_finish: global term %d from logits has %lld rows (at most %d; apply the softmax first)", i, s.N,
                  FIN_GLOBAL_LOGITS_MAX_N);
      d.x = s.x; d.y = s.y; d.x_sn = s.x_sn; d.y_sn = s.y_sn; d.N = s.N;
      d.T = 1;
      d.n_patches = 1;
      d.E = (long long)s.K * s.K;
      d.symmetric = s.symmetric;
      d.check_simplex = logits ? 0 : s.check_simplex;
      d.P_out = s.P_out;
      epi_units += 1;
    }
    units += (d.kind == IIC_ITEM_GLOBAL_ROWS) ? 1 : (long long)d.n_patches * ((d.E / d.n_patches + 31) / 32);
    off += d.E;
  }
  IIC_REQUIRE(off == E_total, "iic_finish: the terms hold %lld joint entries, E_total says %lld", off, E_total);
  // small batches (config 2: one local + one global term): the last CTA exchanges and runs the epilogues itself;
  // anything larger: phase 1 here, then the rank sum and the epilogues as multi-CTA launches
  const bool small = fused && epi_units <= FIN_SMALL_UNITS && epi_patches <= FIN_MAX_PATCHES && E_total <= (long long)FIN_WARPS * 33;
  // The epilogues of a small batch can run in the last CTA too (one launch instead of two), but they are fp64 work that one
  // SM gets through slowly: at config 2 the step is 4.7 us faster with the units spread over SMs by the batched epilogue
  // launch (0.1557 vs 0.1604 ms on the same box), so that is the default and the last-CTA form an option.
  const bool last_cta_epilogue = small && options().fin_last_cta_epilogue;
  B.do_epilogue = last_cta_epilogue ? 1 : 0;
  B.xchg_mode = small ? 1 : 2;
  int sms = sm_count_cached(current_device());
  if (sms <= 0) sms = 148;
  long long grid = units < sms ? units : sms;
  if (grid < 1) grid = 1;
  unsigned int* tickets = reinterpret_cast<unsigned int*>(workspace);
  finish_kernel<<<(unsigned)grid, FIN_THREADS, 0, st>>>(B);
  IIC_CHECK_CUDA(cudaGetLastError());
  if (last_cta_epilogue) return 0;
  if (world > 1 && !small) {                 // (a small batch was exchanged and summed by the last CTA)
    long long g2 = (E_total + FIN_THREADS - 1) / FIN_THREADS;
    if (g2 > sms) g2 = sms;
    xchg_sum_kernel<<<(unsigned)g2, FIN_THREADS, 0, st>>>(J_all, E_total, B.peers, rank, world, xchg_capacity, B.timeout_ns, flags,
                                                          tickets + 1);
    IIC_CHECK_CUDA(cudaGetLastError());
  }
  if (!want_epilogue) return 0;
  if (fused && epi_units <= FIN_BIG_MAX_UNITS) {
    int kmax = 1;
    for (int i = 0; i < n_items; ++i) kmax = items_host[i].K > kmax ? items_host[i].K : kmax;
    const size_t smem = (40 + 3 * (size_t)kmax) * sizeof(double);
    batched_epilogue_kernel<<<(unsigned)epi_units, 256, smem, st>>>(B, tickets + FIN_WS_TICKETS / sizeof(unsigned int),
                                                                    reinterpret_cast<double*>((unsigned char*)workspace + FIN_WS_LOSSES));
    IIC_CHECK_CUDA(cudaGetLastError());
    return 0;
  }
  // no_fused_epilogue / enormous batches: the single-term epilogue kernels, one launch per term
  for (int i = 0; i < n_items; ++i) {
    const iic_finish_item& s = items_host[i];
    const FinItem& d = B.it[i];
    if (s.kind == IIC_ITEM_LOCAL) {
      IIC_REQUIRE(s.epilogue_workspace, "iic_finish: term %d needs epilogue_workspace", i);
      IIC_CHECK_RC(iic_local_epilogue(d.J, s.K, s.pad, s.n_patches, s.lamda, s.loss_out, nullptr, s.Wx, s.Wy, nullptr, flags,
                                      s.epilogue_workspace, stream));
    } else {
      IIC_CHECK_RC(iic_global_epilogue(d.J, s.K, s.lamda, s.symmetric, s.loss_out, s.P_out, flags, stream));
    }
  }
  return 0;
}
