// Backward sweeps of the local IIC term on the tensor cores for the reference's default cluster count (K = 20, any
// 16 <= K <= 24) and both yaml paddings (1 and 3): "row-block" variant of local_bwd_tc.cu.  One launch computes
//   out[n,o,r,c] = g * sum_{cin,ty,tx} Wc[cin][ty*T+tx][o] * src[n,cin,r+ty-pad,c+tx-pad]          (src zero outside the map)
// = what autograd's convolution_backward yields for the F.conv2d at contrastyou/losses/iic_loss.py:123.
//
// Why a different decomposition.  Measured on B200 (local_bwd_tc.cu, everything but the MMAs ablated): an M = 128
// tcgen05.mma costs ~88 clk whatever its N (128 down to 8).  With N = 24 output channels per instruction a small-K sweep
// would be slower than the FFMA2 kernel, so N is filled with OUTPUT ROWS: a staged source row q (one A operand window
// per column tap tx) contributes to the T output rows q - ty, and the weight image holds, per (channel slice, tx), the
// T row-tap matrices stacked in descending ty -- one MMA with N = T * 24 adds a source row into the accumulators of T
// consecutive output rows at once (TMEM columns (row * 24 + channel), contiguous).  Per source row and 8-channel slice:
// T (tx) x 2 MMAs per 128-pixel tile instead of T*T x 2.
//
// A work item is a block of R output rows of one image (all accumulators = R x tiles x 24 TMEM columns <= 512).  The
// epilogue zeroes the accumulators after draining them, so every MMA accumulates.  Split product, pixel-major
// no-swizzle K-major A operand with tap column shifts as descriptor start shifts: see local_bwd_tc.cu; four issuing
// warps ((128-pixel tile 0 / 1) x (even / odd source rows)): see local_bwd_tcrb10.cu.  Per item: for each 8-channel
// slice the slice's weight image (64*T*T*24 bytes, double buffered, one bulk copy) stays resident while the
// R + T - 1 source rows stream through the operand ring.
//
// From-logits form (FL, the cluster head's SoftmaxWithT fused): the maps hold logits.  The TMA warp also stages the
// (m, r) of every staged source pixel (local_logit_stats_kernel, local_logits.cu) and the transform converts each logit
// slice to p = exp(l * inv_temp - m) * r (r = 0 in the TMA zero fill outside the map, so p stays 0 there; channels
// >= K are zeroed).  The drain holds all 24 accumulator channels g_o of its pixel and applies the softmax adjoint
//   d logit_o = inv_temp * p_o * (g_o - sum_k g_k p_k)
// with p at the OUTPUT pixel from its own logits and (m, r), read coalesced (lane = pixel) after an L2 prefetch of the
// item's rows issued while the MMAs run.  The FL form issues each tile's MMAs from ONE warp (the even / odd source-row
// split of two issuers sums into the same accumulators in a timing-dependent order), so two calls give the same bits.
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace bwdrb {
using namespace tc;

constexpr int SL = 8;                    // input channels per slice
constexpr int APX = 272;                 // pixels per row buffer; buffer pixel b holds column b - 8
constexpr int MAXW = 248;
constexpr int A_PART = 2 * APX * 16;     // fp32 part / bf16 part of one row buffer: 2 chunks x APX x 16 B = 8704
constexpr int A_ROW = 2 * A_PART;        // 17408
constexpr int NA_MAX = 6, NRAW_MAX = 8;  // ring depths are chosen per launch from the shared memory the weight slots leave
constexpr int RAW_MAX = SL * 256 * 4;    // 8192
constexpr int FL_STATS = 2 * 256 * 4;    // FL: a raw slot also holds the staged pixels' stats [2][SW] after RAW_MAX bytes
constexpr int NTHREADS = 448;            // warps: 0 TMA, 3 TMEM + weights, 1 2 12 13 MMA issuers, 4-7 transform, 8-11 epilogue
constexpr int SMEM_LIMIT = 225 * 1024;    // dynamic shared memory we may ask for (the static barriers share the 227 KB)


#ifdef IIC_TC_TRACE
__device__ long long g_trace[4][64][6];
#define TRACE(role, slot) do { if (blockIdx.x == 0 && tt >= 40 && tt < 104) g_trace[role][tt - 40][slot] = clock64(); } while (0)
#else
#define TRACE(role, slot) do { } while (0)
#endif

struct Params {
  int B, H, W, K;
  int KP, NS, R;                // channels padded to 8, channel slices, output rows per item
  int nblk, n_items;            // row blocks per image, B * nblk * npanel
  int PW, npanel;               // column panels (maps wider than one TMA box): width and count
  int wslice_bytes;             // bytes of one slice's weight image = T tiles of 64*T*KP bytes
  int na, nraw;                 // operand-ring and raw-ring depths
  const float* wimg;
  const float* grad_loss;
  float* out;
  long long out_sn;             // sample stride of `out` in elements
};

// the from-logits form's extra arguments (unused by the probability instantiations)
struct FLParams {
  CUtensorMap stats;            // the (2B, 2, H, W) stats tensor, box [2][1][PW + 8]: x stats at n, y stats at B + n
  int src_n;                    // stats sample offset of the source map (B for y, 0 for x)
  float inv_temp;
  const float* lout;            // logits of the OUTPUT map (its gradient is `out`), strides below
  long long l_sn, l_sc, l_sh;
  const float* sout;            // its (m, r) planes: sample n at sout + n * 2HW
};

// Wc[cin][ty*T+tx][Kp4] -> per (slice, tx) a tile {fp32 [2 chunks][T*KP rows][4 in], bf16 [wh, wl][T*KP rows][8 in]},
// rows ordered (T-1-ty)*KP + o
__global__ void weight_image_kernel(const float* __restrict__ Wc, float* __restrict__ img, int K, int Kp4, int KP, int NS, int T) {
  const int rows = T * KP;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= NS * T * rows) return;
  const int row = e % rows, tx = (e / rows) % T, js = e / (rows * T);
  const int ty = T - 1 - row / KP, o = row % KP;
  float v[SL];
#pragma unroll
  for (int q = 0; q < SL; ++q) {
    const int cin = js * SL + q;
    v[q] = (cin < K && o < K) ? Wc[((size_t)cin * T * T + ty * T + tx) * Kp4 + o] : 0.f;
  }
  float4* tile = reinterpret_cast<float4*>(img) + (size_t)(js * T + tx) * (4 * rows);
  tile[row] = make_float4(v[0], v[1], v[2], v[3]);
  tile[rows + row] = make_float4(v[4], v[5], v[6], v[7]);
  reinterpret_cast<uint4*>(tile)[2 * rows + row] = pack8<false>(v);     // wh (pairs with al)
  reinterpret_cast<uint4*>(tile)[3 * rows + row] = pack8<true>(v);      // wl (pairs with ah)
}

// bytes between raw-ring slots (a namespace-scope function rather than a constexpr local, which changes the probability
// instantiation's register assignment)
template <bool FL>
__device__ constexpr int raw_stride() { return FL ? RAW_MAX + FL_STATS : RAW_MAX; }

template <int T, bool FL>
__global__ void __launch_bounds__(NTHREADS, 1)
local_bwd_tcrb_kernel(const __grid_constant__ CUtensorMap maps, const Params P, const __grid_constant__ FLParams F) {
  constexpr int PAD = T / 2;
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[NRAW_MAX], raw_empty[NRAW_MAX], a_full[NA_MAX], a_empty[NA_MAX], w_full[2], w_empty[2], accum_full, tmem_ready;
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const int wslot_bytes = (P.wslice_bytes + 127) & ~127;
  unsigned char* w_ring = smem;
  unsigned char* a_ring = smem + 2 * wslot_bytes;
  unsigned char* raw_ring = a_ring + P.na * A_ROW;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int it0 = (int)((long long)blockIdx.x * P.n_items / gridDim.x);
  const int it1 = (int)((long long)(blockIdx.x + 1) * P.n_items / gridDim.x);
  const int nit = it1 - it0;
  const int SW = P.PW + 8;                                 // staged columns of a panel: col0 - 4 .. col0 + PW + 3
  const int raw_bytes = SL * SW * 4;
  const int ntile = P.PW > 128 ? 2 : 1;
  const int NQ = P.R + T - 1;                              // source rows per item
  const int KP = P.KP, NS = P.NS, R = P.R, NA = P.na, NRAW = P.nraw;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NRAW; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 4); }
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 4); mbar_init(&a_empty[s], 2); }
    for (int s = 0; s < 2; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 4); }
    mbar_init(&accum_full, 4);
    mbar_init(&tmem_ready, 4);
    mbar_fence_init();
  }
  if (wid == 3) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem_base = tmem_base_s;

  if (wid == 0) {
    // ===== TMA producer: one source row of one channel slice per stage =====
    if (lane == 0) {
      tma_prefetch_desc(&maps);
      if constexpr (FL) tma_prefetch_desc(&F.stats);
      int t = 0, s = 0;                                 // ring slot and phase as running counters: no divisions per stage
      unsigned sph = 0;
      for (int i = 0; i < nit; ++i) {
        const int item = it0 + i;
        const int panel = item % P.npanel, ib = item / P.npanel;
        const int n = ib / P.nblk, r0 = (ib - n * P.nblk) * R;
        for (int js = 0; js < NS; ++js)
          for (int q = 0; q < NQ; ++q, ++t) {
            { const int tt = t; (void)tt; TRACE(0, 0); }
            if (t >= NRAW) mbar_wait(&raw_empty[s], sph ^ 1u, 1);
            { const int tt = t; (void)tt; TRACE(0, 1); }
            mbar_arrive_expect_tx(&raw_full[s], FL ? raw_bytes + 2 * SW * 4 : raw_bytes);
            tma_load_4d(raw_ring + s * raw_stride<FL>(), &maps, &raw_full[s], panel * P.PW - 4, r0 - PAD + q, js * SL, n);
            if constexpr (FL)                              // the source pixels' (m, r), behind the logits
              tma_load_4d(raw_ring + s * raw_stride<FL>() + RAW_MAX, &F.stats, &raw_full[s], panel * P.PW - 4, r0 - PAD + q, 0,
                          F.src_n + n);
            if (++s == NRAW) { s = 0; sph ^= 1u; }
          }
      }
    }
  } else if (wid == 3) {
    // ===== weight image of a channel slice: one bulk copy, double buffered =====
    if (lane == 0) {
      const int total = nit * NS;
      for (int w = 0; w < total; ++w) {
        const int s = w & 1;
        if (w >= 2) mbar_wait(&w_empty[s], ((unsigned)(w >> 1) & 1u) ^ 1u, 2);
        mbar_arrive_expect_tx(&w_full[s], P.wslice_bytes);
        bulk_load(w_ring + s * wslot_bytes, reinterpret_cast<const unsigned char*>(P.wimg) + (size_t)(w % NS) * P.wslice_bytes,
                  P.wslice_bytes, &w_full[s]);
      }
    }
  } else if (wid == 1 || wid == 2 || wid == 12 || wid == 13) {
    // ===== MMA issuers: (pixel tile 0 / 1) x (even / odd source rows).  A lane issues an MMA only every ~88 clk and pays
    // ~300 clk per barrier poll, the pipe takes one every ~62 clk; the accumulators are zeroed and every MMA accumulates,
    // so the issue order is free (see local_bwd_tcrb10.cu) =====
    const int mt = (wid == 1 || wid == 12) ? 0 : 1;
    const int par = wid >= 12 ? 1 : 0;
    const bool mine = mt < ntile;
    const uint32_t rows = (uint32_t)(T * KP);              // rows of one weight part chunk
    int a = 0, tt = 0;
    unsigned aph = 0;
    // FL: the odd-row issuers stay out altogether (waiting on barriers they do not consume, they could fall two phases
    // behind)
    const int nit_issue = FL && par ? 0 : nit;
    for (int i = 0; i < nit_issue; ++i) {
      mbar_wait(&tmem_ready, (unsigned)i & 1u, 6);          // accumulators zeroed
      asm volatile("tcgen05.fence::after_thread_sync;");
      for (int js = 0; js < NS; ++js) {
        const int w = i * NS + js, ws = w & 1;
        mbar_wait(&w_full[ws], (unsigned)(w >> 1) & 1u, 7);
        const uint64_t w_base = make_desc_kmajor_noswz(smem_u32(w_ring + ws * wslot_bytes), rows * 16);
        for (int q = 0; q < NQ; ++q, ++tt) {
          // FL: one issuer per tile takes every source row, in order, so that the fp32 accumulation order (and the
          // gradient's bits) is the same on every call; the barrier counts hold (its last-row commits come twice)
          if (!FL && (q & 1) != par) {                   // the other issuer of this tile takes this source row
            if (++a == NA) { a = 0; aph ^= 1u; }
            continue;
          }
          if (lane == 0 && par == 0) TRACE(1 + mt, 0);
          mbar_wait(&a_full[a], aph, 5);
          asm volatile("tcgen05.fence::after_thread_sync;");
          if (lane == 0) {
            if (par == 0) TRACE(1 + mt, 1);
            if (mine) {
              // source row q feeds output rows q - ty, 0 <= q - ty < R
              const int ty_max = q < T - 1 ? q : T - 1;
              const int ty_min = q - R + 1 > 0 ? q - R + 1 : 0;
              const uint32_t nn = (uint32_t)((ty_max - ty_min + 1) * KP);
              const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((nn >> 3) << 17) | (8u << 24);
              const uint32_t idesc_bf16 = (1u << 4) | (1u << 7) | (1u << 10) | ((nn >> 3) << 17) | (8u << 24);
              const uint32_t d_tmem = tmem_base + (uint32_t)((mt * R + (q - ty_max)) * KP);
              const uint64_t a_base = make_desc_kmajor_noswz(smem_u32(a_ring + a * A_ROW), APX * 16) + (uint64_t)(mt * 128 + 8 - PAD);   // output pixel c, tap tx: column c + tx - PAD = buffer pixel c + tx + 8 - PAD
              const uint64_t b_base = w_base + (uint64_t)((T - 1 - ty_max) * KP);
#pragma unroll
              for (int tx = 0; tx < T; ++tx) {
                const uint64_t bt = b_base + (uint64_t)tx * (4 * rows);               // tile tx: 4 chunks of `rows` 16-byte rows
                umma_bf16(d_tmem, a_base + (uint64_t)(A_PART / 16 + tx), bt + 2 * rows, idesc_bf16);   // al*wh + ah*wl
                umma_tf32(d_tmem, a_base + (uint64_t)tx, bt, idesc);
              }
            }
            if (par == 0) TRACE(1 + mt, 2);
            umma_commit(&a_empty[a]);
            if (q >= NQ - 2) {                             // this issuer's last source row of the slice
              umma_commit(&w_empty[ws]);
              if (js == NS - 1) umma_commit(&accum_full);
            }
          }
          __syncwarp();
          if (++a == NA) { a = 0; aph ^= 1u; }
        }
      }
    }
  } else if (wid >= 4 && wid < 8) {
    // ===== transform: [ch][px] fp32 -> [chunk][px][16 B] operand images (fp32 and bf16 [al | ah]) =====
    const int tid = threadIdx.x - 128;
    const int total = nit * NS * NQ;
    int a = 0, s = 0;
    unsigned aph = 0, sph = 0;
    for (int t = 0; t < total; ++t) {
      const int tt = t;
      (void)tt;
      if (threadIdx.x == 128) TRACE(3, 0);
      if (t >= NA) mbar_wait(&a_empty[a], aph ^ 1u, 3);
      if (threadIdx.x == 128) TRACE(3, 1);
      mbar_wait(&raw_full[s], sph, 4);
      if (threadIdx.x == 128) TRACE(3, 2);
      unsigned char* abuf = a_ring + a * A_ROW;
      const float* raw = reinterpret_cast<const float*>(raw_ring + s * raw_stride<FL>());
      for (int px = tid; px < SW; px += 128) {
        float v[SL];
#pragma unroll
        for (int c = 0; c < SL; ++c) v[c] = raw[c * SW + px];
        if constexpr (FL) {
          const float* sm = reinterpret_cast<const float*>(raw_ring + s * raw_stride<FL>() + RAW_MAX);   // m [SW], then r [SW]
          const float mx = sm[px], rr = sm[SW + px];
          const int fjs = (t / NQ) % NS;                                // channel slice of this stage
#pragma unroll
          for (int c = 0; c < SL; ++c) v[c] = fjs * SL + c < P.K ? __expf(__fmul_rn(v[c], F.inv_temp) - mx) * rr : 0.f;
        }
        const int off = (px + 4) * 16;                                   // staged pixel px is column px - 4
        *reinterpret_cast<float4*>(abuf + off) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(abuf + off + APX * 16) = make_float4(v[4], v[5], v[6], v[7]);
        *reinterpret_cast<uint4*>(abuf + A_PART + off) = pack8<true>(v);
        *reinterpret_cast<uint4*>(abuf + A_PART + off + APX * 16) = pack8<false>(v);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&raw_empty[s]);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_full[a]);
      if (threadIdx.x == 128) TRACE(3, 3);
      if (++a == NA) { a = 0; aph ^= 1u; }
      if (++s == NRAW) { s = 0; sph ^= 1u; }
    }
  } else if (wid >= 8 && wid < 12) {
    // ===== epilogue: drain the R x tiles x KP accumulator columns, store, zero them for the next item =====
    const int q4 = wid & 3;
    const float g = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
    const size_t plane = (size_t)P.H * P.W;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
    const int ncols = ntile * R * KP;
    auto zero_accumulators = [&]() {
      for (int c = 0; c < ncols; c += 8)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(lane_base + c), "r"(0u) : "memory");
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_ready);
    };
    zero_accumulators();
    for (int i = 0; i < nit; ++i) {
      const int item = it0 + i;
      const int panel = item % P.npanel, ib = item / P.npanel;
      const int n = ib / P.nblk, r0 = (ib - n * P.nblk) * R;
      const int col0 = panel * P.PW;
      if constexpr (FL) {
        // while the MMAs run: pull the item's output logits and stats into L2 (128-byte lines, all drain lanes)
        const int rv = (P.H - r0 < R) ? P.H - r0 : R;
        const int lines = (P.PW * 4 + 127) / 128;
        const int per_plane = rv * lines;
        for (int e = threadIdx.x - 256; e < (P.K + 2) * per_plane; e += 128) {
          const int ch = e / per_plane, rem = e - ch * per_plane, row = rem / lines, ln = rem - row * lines;
          const float* src = ch < P.K ? F.lout + (size_t)n * F.l_sn + (size_t)ch * F.l_sc + (size_t)(r0 + row) * F.l_sh
                                      : F.sout + ((size_t)n * 2 + (ch - P.K)) * plane + (size_t)(r0 + row) * P.W;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(src + col0 + ln * 32));
        }
      }
      mbar_wait(&accum_full, (unsigned)i & 1u, 8);
      asm volatile("tcgen05.fence::after_thread_sync;");
      // The MMAs of the next item wait for this drain (all TMEM columns are in use), so it is kept short: the 2 x 24
      // accumulator columns of two output rows are fetched with six back-to-back tcgen05.ld and ONE wait, then stored.
      const int rv = (P.H - r0 < R) ? P.H - r0 : R;            // output rows of this item
      for (int mt = 0; mt < ntile; ++mt) {
        const int cp = mt * 128 + q4 * 32 + lane;            // column inside the panel
        const int c = col0 + cp;
        const bool live = c < P.W && cp < P.PW;
        for (int orow = 0; orow < rv; orow += 2) {
          uint32_t v[2][24];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int orh = orow + h < R ? orow + h : orow;     // the pair's second row may not exist: re-read the first
#pragma unroll
            for (int ch = 0; ch < 24; ch += 8) {
              if (ch < KP) {
                const uint32_t taddr = lane_base + (uint32_t)((mt * R + orh) * KP + ch);
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                             : "=r"(v[h][ch]), "=r"(v[h][ch + 1]), "=r"(v[h][ch + 2]), "=r"(v[h][ch + 3]), "=r"(v[h][ch + 4]),
                               "=r"(v[h][ch + 5]), "=r"(v[h][ch + 6]), "=r"(v[h][ch + 7])
                             : "r"(taddr));
              }
            }
          }
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if constexpr (FL) {
            if (live) {
  #pragma unroll
              for (int h = 0; h < 2; ++h) {
                if (orow + h < rv) {
                  const int row = r0 + orow + h;
                  float* dst = P.out + (size_t)n * P.out_sn + (size_t)row * P.W + c;
                  const float* lp = F.lout + (size_t)n * F.l_sn + (size_t)row * F.l_sh + c;
                  const float* sp = F.sout + (size_t)n * 2 * plane + (size_t)row * P.W + c;
                  const float mx = __ldg(sp), rr = __ldg(sp + plane);
                  float pr[24];
                  float dot = 0.f;
  #pragma unroll
                  for (int o = 0; o < 24; ++o) {
                    if (o < P.K) {                                          // (columns >= KP were not loaded)
                      pr[o] = __expf(__fmul_rn(__ldg(lp + (size_t)o * F.l_sc), F.inv_temp) - mx) * rr;
                      dot = fmaf(g * __uint_as_float(v[h][o]), pr[o], dot);
                    }
                  }
  #pragma unroll
                  for (int o = 0; o < 16; ++o) dst[(size_t)o * plane] = F.inv_temp * pr[o] * (g * __uint_as_float(v[h][o]) - dot);
                  if (P.K == 20) {
  #pragma unroll
                    for (int o = 16; o < 20; ++o) dst[(size_t)o * plane] = F.inv_temp * pr[o] * (g * __uint_as_float(v[h][o]) - dot);
                  } else {
  #pragma unroll
                    for (int o = 16; o < 24; ++o)
                      if (o < P.K) dst[(size_t)o * plane] = F.inv_temp * pr[o] * (g * __uint_as_float(v[h][o]) - dot);
                  }
                }
              }
            }
          } else {
            if (live) {
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                if (orow + h < rv) {
                  float* dst = P.out + (size_t)n * P.out_sn + (size_t)(r0 + orow + h) * P.W + c;
                  // straight-line stores for the channels every covered head has (K >= 16; a branch per channel costs ~10
                  // instructions and a uniform-register reload per store), the yaml default K = 20 entirely
#pragma unroll
                  for (int o = 0; o < 16; ++o) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);
                  if (P.K == 20) {
#pragma unroll
                    for (int o = 16; o < 20; ++o) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);
                  } else {
#pragma unroll
                    for (int o = 16; o < 24; ++o)
                      if (o < P.K) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);
                  }
                }
              }
            }
          }
        }
      }
      if (i + 1 < nit) zero_accumulators();
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 3) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

template <int T, bool FL>
static int launch(const CUtensorMap& m, const Params& P, const FLParams& F, int grid, size_t smem, cudaStream_t st) {
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_bwd_tcrb_kernel<T, FL>), (int)(SMEM_LIMIT)));
  local_bwd_tcrb_kernel<T, FL><<<grid, NTHREADS, smem, st>>>(m, P, F);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace bwdrb

size_t local_bwd_tcrb_image_bytes(int K, int pad) {
  if (K < 16 || K > 24 || (pad != 1 && pad != 3)) return 0;
  const int T = 2 * pad + 1, KP = (K + 7) & ~7;
  return (size_t)(KP / bwdrb::SL) * 64 * T * T * KP;
}

// Column panels, rows per item and item count of a (B, K, H, W) map; false when the family does not cover it.  Maps wider
// than one TMA box are cut into column panels: 128 columns (one pixel tile, no padding) when that divides the width, else
// equal panels of at most 248 columns.
bool local_bwd_tcrb_plan(int B, int K, int H, int W, int pad, int* PW_out, int* npanel_out, int* R_out, int* n_items_out) {
  using namespace bwdrb;
  if (K < 16 || K > 24 || (pad != 1 && pad != 3) || W % 4 != 0 || W < 8) return false;
  int npanel = 1, PW = W;
  if (W > MAXW) {
    if (W % 128 == 0) { PW = 128; npanel = W / 128; }
    else { npanel = (W + MAXW - 1) / MAXW; PW = (((W + npanel - 1) / npanel) + 3) & ~3; }
  }
  const int KP = (K + 7) & ~7;
  const int ntile = PW > 128 ? 2 : 1;
  int R = 512 / (ntile * KP);
  if (R > H) R = H;
  *PW_out = PW; *npanel_out = npanel; *R_out = R;
  *n_items_out = B * ((H + R - 1) / R) * npanel;
  return true;
}

// 3 x 3 window: the FFMA2 kernel is as fast unless there are enough row blocks to keep every SM busy (measured:
// (32,20,224,224) 0.32 ms vs 0.42 ms, (8,20,112,112) no gain)
bool local_bwd_tcrb_p1_gate(int n_items, int sms) { return n_items >= 2 * sms || options().tcrb_p1; }

// stats == nullptr: probabilities; else logits with the per-pixel (m, r) of local_logit_stats_kernel in `stats`
static int tcrb_try(const LocalMaps& m, const float* stats, float inv_temp, float* Wx, float* Wy, const LocalGrads& g,
                    cudaStream_t st) {
  using namespace bwdrb;
  const int B = m.B, K = m.K, H = m.H, W = m.W, pad = m.pad, sms = m.sms;
  int PW, npanel, R, n_items;
  if (!local_bwd_tcrb_plan(B, K, H, W, pad, &PW, &npanel, &R, &n_items)) return -1;
  const int T = 2 * pad + 1, KP = (K + 7) & ~7, NS = KP / SL, Kp4 = (K + 3) & ~3;
  const bool fl = stats != nullptr;
  const int raw_stride = fl ? RAW_MAX + FL_STATS : RAW_MAX;
  const int wslice = 64 * T * T * KP;
  // ring depths: what the two weight slots leave, shared between the operand ring (17 KB slots) and the raw ring (8 KB,
  // 10 KB from logits)
  const long long spare = (long long)SMEM_LIMIT - 1024 - 2LL * ((wslice + 127) & ~127);
  int na = 3, nraw = 2;
  if (spare < (long long)na * A_ROW + (long long)nraw * raw_stride) return -1;
  while (nraw < NRAW_MAX && spare >= (long long)na * A_ROW + (long long)(nraw + 1) * raw_stride) ++nraw;
  while (na < NA_MAX && spare >= (long long)(na + 1) * A_ROW + (long long)nraw * raw_stride) ++na;
  const size_t smem = (size_t)2 * ((wslice + 127) & ~127) + (size_t)na * A_ROW + (size_t)nraw * raw_stride + 1024;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, PW + 8, 1, SL)) return -1;
  if (!make_map_4d(&my, m.y, m, PW + 8, 1, SL)) return -1;
  const int nblk = (H + R - 1) / R;
  if (pad == 1 && !local_bwd_tcrb_p1_gate(n_items, sms)) return -1;
  const long long hw = (long long)H * W;
  FLParams Fgx{}, Fgy{};
  if (fl) {
    if (!make_map_4d(&Fgx.stats, stats, 2 * B, 2, H, W, 2 * hw, hw, W, PW + 8, 1, 2)) return -1;
    Fgy.stats = Fgx.stats;
    // dL/dx: source y (stats at B + n), output x;  dL/dy: source x, output y
    Fgx.src_n = B; Fgx.inv_temp = inv_temp; Fgx.lout = m.x.p; Fgx.l_sn = m.x.sn; Fgx.l_sc = m.x.sc; Fgx.l_sh = m.x.sh;
    Fgx.sout = stats;
    Fgy.src_n = 0; Fgy.inv_temp = inv_temp; Fgy.lout = m.y.p; Fgy.l_sn = m.y.sn; Fgy.l_sc = m.y.sc; Fgy.l_sh = m.y.sh;
    Fgy.sout = stats + 2 * B * hw;
  }
  const int grid = n_items < sms ? n_items : sms;
  // the weight image lives in the tail of the caller's coefficient buffer (common.cuh)
  float* img_x = Wx + local_coeff_image_offset(K, pad, 1);
  float* img_y = Wy + local_coeff_image_offset(K, pad, 1);
  const int wthreads = NS * T * T * KP;
  weight_image_kernel<<<(wthreads + 255) / 256, 256, 0, st>>>(Wx, img_x, K, Kp4, KP, NS, T);
  weight_image_kernel<<<(wthreads + 255) / 256, 256, 0, st>>>(Wy, img_y, K, Kp4, KP, NS, T);
  IIC_CHECK_CUDA(cudaGetLastError());
  Params Pgx{B, H, W, K, KP, NS, R, nblk, n_items, PW, npanel, wslice, na, nraw, img_x, g.grad_loss, g.gx, g.gx_sn};     // dL/dx from y
  Params Pgy{B, H, W, K, KP, NS, R, nblk, n_items, PW, npanel, wslice, na, nraw, img_y, g.grad_loss, g.gy, g.gy_sn};     // dL/dy from x
  if (fl) {
    if (T == 3) {
      if (int rc = launch<3, true>(my, Pgx, Fgx, grid, smem, st)) return rc;
      return launch<3, true>(mx, Pgy, Fgy, grid, smem, st);
    }
    if (int rc = launch<7, true>(my, Pgx, Fgx, grid, smem, st)) return rc;
    return launch<7, true>(mx, Pgy, Fgy, grid, smem, st);
  }
  if (T == 3) {
    if (int rc = launch<3, false>(my, Pgx, Fgx, grid, smem, st)) return rc;
    return launch<3, false>(mx, Pgy, Fgy, grid, smem, st);
  }
  if (int rc = launch<7, false>(my, Pgx, Fgx, grid, smem, st)) return rc;
  return launch<7, false>(mx, Pgy, Fgy, grid, smem, st);
}

int local_bwd_tcrb_try(const LocalMaps& m, float* Wx, float* Wy, const LocalGrads& g, cudaStream_t st) {
  return tcrb_try(m, nullptr, 1.f, Wx, Wy, g, st);
}

int local_bwd_tcrb_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* Wx, float* Wy, const LocalGrads& g,
                          cudaStream_t st) {
  return tcrb_try(m, stats, inv_temp, Wx, Wy, g, st);
}

}  // namespace iic
