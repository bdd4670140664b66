// Backward sweeps of the local IIC term on the tensor cores for 10 clusters, 3 x 3 window (BASELINE config 2), fp16-split
// variant of local_bwd_tcrb10.cu.  Same pipeline (TMA row loads, transform warps, four issuing warps, double-buffered
// TMEM accumulators, coalesced drain); what changes is how fp32 accuracy is obtained from the tensor pipe:
//   local_bwd_tcrb10.cu   a*w = tf32(a)*tf32(w) [kind::tf32, K = 8 per MMA] + bf16 corrections [kind::f16, K = 16]:
//                         8 MMAs per source row and 128-pixel tile, 128 bytes of operand per pixel written by the transform
//   here                  a = a1 + a2, w = w1 + w2 with a1 = fp16(a), a2 = fp16(a - a1) (22 bits together), and
//                         a*w = a1*w1 + a2*w1 + a1*w2 (+ a2*w2 ~ 2^-22, dropped).  kind::f16 takes K = 16 slots per MMA, and a
//                         reduction slot need not be "channel c of one part": the 30 (part, channel) products of a column
//                         tap fill exactly two MMAs --
//                           MMA 1: a1[0..7] | a1[8], a1[9], a2[0..5]    x   w1[0..7] | w1[8], w1[9], w1[0..5]
//                           MMA 2: a2[6..9], a1[0..3] | a1[4..9], 0, 0  x   w1[6..9], w2[0..3] | w2[4..9], 0, 0
//                         6 MMAs per source row and tile, 64 bytes of operand per pixel.  The kernel is bound by shared-memory
//                         operand traffic (MMA fetch + transform), so this is where the time goes down.
// fp16 range: the maps are probabilities (<= 1), scaled by 2^8 before the split so that the second part stays normal
// down to 2^-22 of the first; the coefficients are scaled by a power of two that brings their largest magnitude to
// [2^12, 2^13) (found by every CTA from the 2 x 900 coefficients while it builds its weight images); both scales are
// exact and are undone in the drain.
//   out[n,o,r,c] = g * sum_{cin,ty,tx} Wc[cin][ty*3+tx][o] * src[n,cin,r+ty-1,c+tx-1]     (iic_loss.py:123, backward)
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace bwdrb10h {
using namespace tc;

constexpr int T = 3, PAD = 1;
constexpr int KP = 16;                   // accumulator columns per output row (10 channels used)
constexpr int RMAX = 8;                  // output rows per item: 8 x 2 tiles x 16 = 256 TMEM columns, double buffered so that
                                         // the drain of item i overlaps the MMAs of item i+1
constexpr int TBUF = 2 * RMAX * KP;      // TMEM columns of one accumulator buffer
constexpr int APX = 272;
constexpr int MAXW = 248;
constexpr int A_CHUNK = APX * 16;        // one 16-byte chunk array: pixel b of the buffer at b * 16
constexpr int A_SLOT = 4 * A_CHUNK;      // 17408: the four chunks (c0 c1 | c2 c3) of one source row
constexpr int NA = 6;
constexpr int RAW_SLOT = 10 * 256 * 4;   // 10240
constexpr int NRAW = 6;
constexpr int WROWS = T * KP;            // 48 rows per weight chunk
constexpr int W_TILE = 2 * WROWS * 16;   // 1536: one MMA's B operand (two chunks)
constexpr int W_IMG = 6 * W_TILE;        // (tx 0, 1, 2) x (MMA 1, MMA 2)
constexpr int NTHREADS = 704;             // warps: 0 TMA, 3 TMEM (+ logit rows), 1 2 12 13 MMA issuers, 4-11 transform, 14-17 and 18-21 epilogue
constexpr int NTHREADS_FL = 704;          // (one epilogue set per pixel tile: the drain's global stores bound the kernel, see the epilogue)
constexpr int SMEM_BYTES = NA * A_SLOT + 2 * W_IMG + NRAW * RAW_SLOT + 1024;   // both sweeps' weight images stay resident
constexpr int NL = 4;                    // from-logits form: ring of output-tensor logit rows for the drain (two row pairs)
constexpr int SMEM_BYTES_FL = SMEM_BYTES + NL * RAW_SLOT;
constexpr float A_SCALE = 256.f;         // 2^8
constexpr int A_SCALE_LOG2 = 8;
constexpr int W_TARGET_LOG2 = 12;        // largest |coefficient| scaled into [2^12, 2^13)



#ifdef IIC_TC_TRACE
__device__ long long g_trace[4][64][6];
__device__ long long g_ctrace[32][8];      // per chunk i: issuer (tile 0, parity 0) [0] before / [1] after the tmem_ready wait;
                                           // drain warp 14 [2] before / [3] after the accum_full wait, [4] drained, [5] zeroed
#define TRACE(role, slot) do { if (blockIdx.x == 0 && tt >= 16 && tt < 80) g_trace[role][tt - 16][slot] = clock64(); } while (0)
#define CTRACE(slot) do { if (blockIdx.x == 0 && i < 32) g_ctrace[i][slot] = clock64(); } while (0)
#else
#define TRACE(role, slot) do { } while (0)
#define CTRACE(slot) do { } while (0)
#endif

struct Params {
  int B, H, W, K;
  const float* Wc[2];           // coefficient tensors of iic_local_epilogue: sweep 0 = Wx (dL/dx, source y), sweep 1 = Wy
  int Kp4;                      // their row length
  const float* grad_loss;
  float* out[2];
  long long out_sn[2];          // sample strides of the two gradient tensors in elements
  // from-logits form (the cluster head's SoftmaxWithT fused, contrastyou/trainer/_utils.py:15-23): the maps behind the TMA
  // descriptors hold LOGITS; the transform warps soft-max every staged pixel, the drain applies the softmax adjoint with
  // the probabilities of the OUTPUT tensor's pixel, recomputed from its logits (lout[sweep]: sweep 0 -> x, sweep 1 -> y)
  int from_logits;
  float inv_temp;
  const float* lout[2];
  long long l_sn[2], l_sc[2], l_sh[2];
};

__device__ __forceinline__ uint32_t pack_h2(float a, float b) {          // a at the lower address
  const __half2 p = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ uint4 pack_h8(const float* v) {
  return make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
}
// v -> (h, l): h = fp16(v), l = fp16(v - h)
__device__ __forceinline__ void split_h(float v, float& h, float& l) {
  h = __half2float(__float2half_rn(v));
  l = __half2float(__float2half_rn(v - h));
}

// Wc[cin][ty*3+tx][Kp4] -> per column tap tx the two B operands of the header comment, each [2 chunks][48 rows][8 fp16],
// rows ordered (2-ty)*16 + o, values scaled by 2^wexp.  Every CTA builds both sweeps' images (2 x 9 KB from 2 x 3.6 KB of
// L2-resident coefficients) straight into its own shared memory.  e = row in [0, 3 * 48).
__device__ __forceinline__ void build_weight_row(const float* __restrict__ Wc, unsigned char* img, int e, int K, int Kp4, float wscale) {
  const int row = e % WROWS, tx = e / WROWS;
  const int ty = T - 1 - row / KP, o = row % KP;
  float w1[10], w2[10];
#pragma unroll
  for (int c = 0; c < 10; ++c) {
    const float v = (c < K && o < K) ? __ldg(Wc + ((size_t)c * T * T + ty * T + tx) * Kp4 + o) * wscale : 0.f;
    split_h(v, w1[c], w2[c]);
  }
  const float c0[8] = {w1[0], w1[1], w1[2], w1[3], w1[4], w1[5], w1[6], w1[7]};
  const float c1[8] = {w1[8], w1[9], w1[0], w1[1], w1[2], w1[3], w1[4], w1[5]};
  const float c2[8] = {w1[6], w1[7], w1[8], w1[9], w2[0], w2[1], w2[2], w2[3]};
  const float c3[8] = {w2[4], w2[5], w2[6], w2[7], w2[8], w2[9], 0.f, 0.f};
  uint4* t = reinterpret_cast<uint4*>(img + (size_t)tx * 2 * W_TILE);
  t[row] = pack_h8(c0);
  t[WROWS + row] = pack_h8(c1);
  t[2 * WROWS + row] = pack_h8(c2);
  t[3 * WROWS + row] = pack_h8(c3);
}

// The chunk of image rows that starts at global row r (rows of all images, B*H) inside the CTA share [R0, R1).  Output
// rows h0 .. h0+nr-1 take source rows h0-1 .. h0+nr (local q = 0 .. nr+1).  Consecutive chunks of one image share two source
// rows (q = nr, nr+1 of one are q = 0, 1 of the next): those are staged ONCE -- the issuers add them into the next chunk's
// accumulator buffer while they finish this one (`cont_next`), and the next chunk starts at q = 2 (`q0`, `cont_prev`).
// With 7-row chunks the re-staged halo rows were 22 % of all stages.  A chunk never leaves a single row behind in its
// run (a source row may belong to two chunks, not three).
struct Chunk { int n, h0, nr, q0; bool cont_next; };
__device__ __forceinline__ Chunk next_chunk(long long r, long long R0, long long R1, int H, int rc) {
  Chunk c;
  c.n = (int)(r / H);
  c.h0 = (int)(r - (long long)c.n * H);
  int run = H - c.h0;
  if (run > R1 - r) run = (int)(R1 - r);
  c.nr = rc < run ? rc : run;
  if (run - c.nr == 1 && c.nr >= 3) c.nr -= 1;
  c.q0 = (r > R0 && c.h0 > 0) ? 2 : 0;
  c.cont_next = c.nr < run;
  return c;
}

template <bool FROM_LOGITS>
__global__ void __launch_bounds__(FROM_LOGITS ? NTHREADS_FL : NTHREADS, 1)
local_bwd_tcrb10h_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1, const Params P) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW], a_full[NA], a_empty[NA], w_full, accum_full[2], tmem_ready[2];
  __shared__ __align__(8) uint64_t l_full[NL], l_empty[NL];      // FROM_LOGITS: logit rows of the OUTPUT tensor for the drain
  __shared__ uint32_t tmem_base_s;
  __shared__ float wmax_s[4];
  __shared__ float unscale_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* a_ring = smem;
  unsigned char* w_img = smem + NA * A_SLOT;
  unsigned char* raw_ring = w_img + 2 * W_IMG;
  unsigned char* l_ring = raw_ring + NRAW * RAW_SLOT;            // FROM_LOGITS only (SMEM_BYTES_FL)
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long rows_total = (long long)P.B * P.H;
  const long long R0 = (long long)blockIdx.x * rows_total / gridDim.x;
  const long long R1 = (long long)(blockIdx.x + 1) * rows_total / gridDim.x;
  const int share = (int)(R1 - R0);
  const int nch = (share + RMAX - 1) / RMAX;
  const int rc = nch > 0 ? (share + nch - 1) / nch : RMAX;      // rows per chunk: the share cut into equal chunks <= 16
  const int SW = P.W + 8;
  const int raw_bytes = P.K * SW * 4;
  const int ntile = P.W > 128 ? 2 : 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NRAW; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 4); }
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 4); mbar_init(&a_empty[s], 2); }
    mbar_init(&w_full, 4);
    const int ndset_i = ntile == 2 ? 2 : 1;                           // epilogue warp sets (one per pixel tile)
    for (int s = 0; s < 2; ++s) { mbar_init(&accum_full[s], 4); mbar_init(&tmem_ready[s], 4 * ndset_i); }
    for (int s = 0; s < NL; ++s) { mbar_init(&l_full[s], 1); mbar_init(&l_empty[s], 4 * ndset_i); }
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
    // ===== TMA producer: one source row (all K channels) per stage =====
    if (lane == 0) {
      tma_prefetch_desc(&map0);
      tma_prefetch_desc(&map1);
      int t = 0, s = 0;
      unsigned sph = 0;
      for (int sweep = 0; sweep < 2; ++sweep)
      for (long long r = R0; r < R1;) {
        const Chunk c = next_chunk(r, R0, R1, P.H, rc);
        for (int q = c.q0; q < c.nr + T - 1; ++q, ++t) {
          { const int tt = t; (void)tt; TRACE(0, 0); }
          if (t >= NRAW) mbar_wait(&raw_empty[s], sph ^ 1u, 1);
          { const int tt = t; (void)tt; TRACE(0, 1); }
          mbar_arrive_expect_tx(&raw_full[s], raw_bytes);
          tma_load_4d(raw_ring + s * RAW_SLOT, sweep == 0 ? &map0 : &map1, &raw_full[s], -4, c.h0 - PAD + q, 0, c.n);
          if (++s == NRAW) { s = 0; sph ^= 1u; }
        }
        r += c.nr;
      }
    }
  } else if (wid == 3) {
    // ===== FROM_LOGITS: the warp that allocated TMEM is idle afterwards; it streams the logit rows of the OUTPUT tensor
    // (sweep 0 writes dL/dx: rows of x = map1; sweep 1: rows of y = map0) ahead of the drain, which needs that pixel's
    // probabilities for the softmax adjoint.  A global load inside the drain loop would put ~1 us of latency on its
    // critical path per row pair (measured: 375 us instead of ~100 us for the kernel). =====
    if (FROM_LOGITS && lane == 0) {
      int t = 0, s = 0;
      unsigned sph = 0;
      for (int sweep = 0; sweep < 2; ++sweep)
      for (long long r = R0; r < R1;) {
        const Chunk c = next_chunk(r, R0, R1, P.H, rc);
        for (int orow = 0; orow < c.nr; ++orow, ++t) {
          if (t >= NL) mbar_wait(&l_empty[s], sph ^ 1u, 9);
          mbar_arrive_expect_tx(&l_full[s], raw_bytes);
          tma_load_4d(l_ring + s * RAW_SLOT, sweep == 0 ? &map1 : &map0, &l_full[s], -4, c.h0 + orow, 0, c.n);
          if (++s == NL) { s = 0; sph ^= 1u; }
        }
        r += c.nr;
      }
    }
  } else if (wid == 1 || wid == 2 || wid == 12 || wid == 13) {
    // ===== MMA issuers.  Traced with clock64(): one lane issues an MMA every ~88 clk and every mbarrier wait costs it
    // ~300 clk even when the barrier is complete, yet the tensor pipe accepts the MMAs of two lanes side by side.  The
    // accumulators are zeroed and every MMA accumulates, so the issue order does not matter: four issuing warps --
    // (pixel tile 0 / 1) x (even / odd stages) -- each commit to the ring barriers. =====
    const int mt = (wid == 1 || wid == 12) ? 0 : 1;
    const int par = wid >= 12 ? 1 : 0;
    const bool mine = mt < ntile;
    mbar_wait(&w_full, 0u, 7);
    const uint64_t w_base0 = make_desc_kmajor_noswz(smem_u32(w_img), WROWS * 16);
    static_assert(NA % 2 == 0 && NRAW % 2 == 0, "the stage-parity split needs even ring depths");
    int a = 0, i = 0, tt = 0;                              // tt = global stage index
    unsigned aph = 0;
    for (int sweep = 0; sweep < 2; ++sweep)
    for (long long r = R0; r < R1; ++i) {
      const uint64_t w_base = w_base0 + (uint64_t)(sweep * (W_IMG / 16));
      const Chunk c = next_chunk(r, R0, R1, P.H, rc);
      const int buf = i & 1;
      if (lane == 0 && wid == 1) CTRACE(0);
      mbar_wait(&tmem_ready[buf], (unsigned)(i >> 1) & 1u, 6);   // this buffer's accumulators are zeroed
      if (lane == 0 && wid == 1) CTRACE(1);
      asm volatile("tcgen05.fence::after_thread_sync;");
      const int nq = c.nr + T - 1;
      // the chunk after this one, when it shares this chunk's last two source rows
      const int nr_next = c.cont_next ? next_chunk(r + c.nr, R0, R1, P.H, rc).nr : 0;
      for (int q = c.q0; q < nq; ++q, ++tt) {
        // Split by the GLOBAL stage parity, like the transform groups, and with even ring depths: a ring slot then always
        // belongs to the same transform group and the same issuer pair, who wait on every phase of its barriers.  (Split
        // by the row index inside the chunk, a slot changes hands after a chunk with an odd number of rows, and an issuer
        // that skipped a phase of a_full passes its parity wait two phases early: tools/barrier_sim.py.)
        if ((tt & 1) != par) {                           // the other issuer of this tile takes this source row
          if (++a == NA) { a = 0; aph ^= 1u; }
          continue;
        }
        if (lane == 0 && par == 0) TRACE(1 + mt, 0);
        mbar_wait(&a_full[a], aph, 5);
        asm volatile("tcgen05.fence::after_thread_sync;");
        if (lane == 0) {
          if (par == 0) TRACE(1 + mt, 1);
          if (mine) {
            const int ty_max = q < T - 1 ? q : T - 1;
            const int ty_min = q - c.nr + 1 > 0 ? q - c.nr + 1 : 0;
            const uint32_t nn = (uint32_t)((ty_max - ty_min + 1) * KP);
            // kind::f16, fp16 operands (a_format = b_format = 0), fp32 accumulator, M = 128, N = nn
            const uint32_t idesc_f16 = (1u << 4) | ((nn >> 3) << 17) | (8u << 24);
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * TBUF + (mt * RMAX + (q - ty_max)) * KP);
            // chunks c0 | c1 of buffer pixel mt*128 + 8 - PAD (+ tx); c2 | c3 are two chunk arrays further on
            const uint64_t a_12 = make_desc_kmajor_noswz(smem_u32(a_ring + a * A_SLOT), A_CHUNK) + (uint64_t)(mt * 128 + 8 - PAD);
            const uint64_t a_34 = a_12 + (uint64_t)(2 * A_CHUNK / 16);
            const uint64_t b_base = w_base + (uint64_t)((T - 1 - ty_max) * KP);
#pragma unroll
            for (int tx = 0; tx < T; ++tx) {
              const uint64_t bt = b_base + (uint64_t)tx * (2 * W_TILE / 16);
              umma_bf16(d_tmem, a_12 + (uint64_t)tx, bt, idesc_f16);
              umma_bf16(d_tmem, a_34 + (uint64_t)tx, bt + (uint64_t)(W_TILE / 16), idesc_f16);
            }
          }
        }
        if (c.cont_next && q >= c.nr) {
          // this source row is also row q2 = q - nr (0 or 1) of the NEXT chunk: add it into the other accumulator buffer,
          // once the drain of the chunk before this one has zeroed it
          mbar_wait(&tmem_ready[buf ^ 1], (unsigned)((i + 1) >> 1) & 1u, 6);
          asm volatile("tcgen05.fence::after_thread_sync;");
          if (lane == 0 && mine) {
            const int q2 = q - c.nr;
            const int ty_max = q2;                                     // q2 < T - 1
            const int ty_min = q2 - nr_next + 1 > 0 ? q2 - nr_next + 1 : 0;
            const uint32_t nn = (uint32_t)((ty_max - ty_min + 1) * KP);
            const uint32_t idesc_f16 = (1u << 4) | ((nn >> 3) << 17) | (8u << 24);
            const uint32_t d_tmem = tmem_base + (uint32_t)((buf ^ 1) * TBUF + (mt * RMAX + (q2 - ty_max)) * KP);
            const uint64_t a_12 = make_desc_kmajor_noswz(smem_u32(a_ring + a * A_SLOT), A_CHUNK) + (uint64_t)(mt * 128 + 8 - PAD);
            const uint64_t a_34 = a_12 + (uint64_t)(2 * A_CHUNK / 16);
            const uint64_t b_base = w_base + (uint64_t)((T - 1 - ty_max) * KP);
#pragma unroll
            for (int tx = 0; tx < T; ++tx) {
              const uint64_t bt = b_base + (uint64_t)tx * (2 * W_TILE / 16);
              umma_bf16(d_tmem, a_12 + (uint64_t)tx, bt, idesc_f16);
              umma_bf16(d_tmem, a_34 + (uint64_t)tx, bt + (uint64_t)(W_TILE / 16), idesc_f16);
            }
          }
        }
        if (lane == 0) {
          if (par == 0) TRACE(1 + mt, 2);
          umma_commit(&a_empty[a]);
        }
        __syncwarp();
        if (++a == NA) { a = 0; aph ^= 1u; }
      }
      // one arrival per issuing warp and item, after its last MMA into this buffer (a warp may have had no source row in the
      // item's tail, or none at all in a two-row item that starts at q = 2)
      if (lane == 0) umma_commit(&accum_full[buf]);
      __syncwarp();
      r += c.nr;
    }
  } else if (wid >= 4 && wid < 12) {
    // ===== transform: two groups of four warps take alternate source rows (a group's iteration is ~1300 clk, of which
    // ~550 clk are the two mbarrier polls: two groups in flight halve the period): [ch][px] fp32 -> main row buffer (channels 0-7) and leftover row buffer ((ch 8, 9) x 3 taps) =====
    const int tid = (threadIdx.x - 128) & 127;
    const int grp = wid >= 8 ? 1 : 0;
    int a = 0, s = 0, t = 0;
    unsigned aph = 0, sph = 0;
    for (int sweep = 0; sweep < 2; ++sweep)
    for (long long r = R0; r < R1;) {
      const Chunk c = next_chunk(r, R0, R1, P.H, rc);
      for (int q = c.q0; q < c.nr + T - 1; ++q, ++t) {
        if ((t & 1) != grp) {                            // the other group's source row
          if (++a == NA) { a = 0; aph ^= 1u; }
          if (++s == NRAW) { s = 0; sph ^= 1u; }
          continue;
        }
        const int tt = t;
        (void)tt;
        if (tid == 0 && wid == 4) TRACE(3, 0);
        if (t >= NA) mbar_wait(&a_empty[a], aph ^ 1u, 3);
        if (tid == 0 && wid == 4) TRACE(3, 1);
        mbar_wait(&raw_full[s], sph, 4);
        if (tid == 0 && wid == 4) TRACE(3, 2);
        unsigned char* am = a_ring + a * A_SLOT;
        const float* raw = reinterpret_cast<const float*>(raw_ring + s * RAW_SLOT);
        const int srow = c.h0 - PAD + q;                   // image row of this source row (outside the map: zero padding)
        const bool row_in = srow >= 0 && srow < P.H;
        // Two pixels per thread (tid and tid + 128), all loads first: the traced pixel loop was latency-bound (one warp of
        // the group per SM sub-partition, ~130 dependent instructions per pixel, stores and loads both in shared memory so
        // the compiler would not overlap iterations) and set the stage period.  Pairs of channels are split with
        // packed conversions -- hp = fp16x2(v), lp = fp16x2(v - float(hp)) -- and the four chunks are assembled from
        // those registers directly (every chunk boundary of the slot layout falls on an even channel).
        float v[2][10];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int px = tid + u * 128;
#pragma unroll
          for (int ch = 0; ch < 10; ++ch) v[u][ch] = (ch < P.K && px < SW) ? raw[ch * SW + px] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int px = tid + u * 128;
          if (FROM_LOGITS) {
            // softmax(logit * inv_temp) over the K channels of this pixel; pixels outside the map (TMA zero fill) must
            // stay zero PROBABILITIES (the conv padding of iic_loss.py:123), not softmax(0) = 1/K
            const int col = px - 4;
            if (row_in && col >= 0 && col < P.W) {
              float mx = v[u][0];
#pragma unroll
              for (int ch = 1; ch < 10; ++ch) if (ch < P.K) mx = fmaxf(mx, v[u][ch]);
              float sum = 0.f;
#pragma unroll
              for (int ch = 0; ch < 10; ++ch) {
                v[u][ch] = ch < P.K ? __expf((v[u][ch] - mx) * P.inv_temp) : 0.f;
                sum += v[u][ch];
              }
              const float inv = 1.f / sum;
#pragma unroll
              for (int ch = 0; ch < 10; ++ch) v[u][ch] *= inv;
            } else {
#pragma unroll
              for (int ch = 0; ch < 10; ++ch) v[u][ch] = 0.f;
            }
          }
        }
        // split of both pixels at once with packed fp32 ops: hi = the scaled value cut to 11 significant bits (a mask; exact
        // in fp16), lo = value - hi (exact in fp32, rounded to fp16 by the pack below)
        float2 hi[10], lo[10];
#pragma unroll
        for (int ch = 0; ch < 10; ++ch) {
          const float2 sv = __fmul2_rn(make_float2(v[0][ch], v[1][ch]), make_float2(A_SCALE, A_SCALE));
          hi[ch] = make_float2(__uint_as_float(__float_as_uint(sv.x) & 0xFFFFE000u), __uint_as_float(__float_as_uint(sv.y) & 0xFFFFE000u));
          lo[ch] = __ffma2_rn(hi[ch], make_float2(-1.f, -1.f), sv);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int px = tid + u * 128;
          uint32_t hp[5], lp[5];
#pragma unroll
          for (int c2 = 0; c2 < 5; ++c2) {
            const __half2 hh = u == 0 ? __floats2half2_rn(hi[2 * c2].x, hi[2 * c2 + 1].x) : __floats2half2_rn(hi[2 * c2].y, hi[2 * c2 + 1].y);
            const __half2 ll = u == 0 ? __floats2half2_rn(lo[2 * c2].x, lo[2 * c2 + 1].x) : __floats2half2_rn(lo[2 * c2].y, lo[2 * c2 + 1].y);
            hp[c2] = *reinterpret_cast<const uint32_t*>(&hh);
            lp[c2] = *reinterpret_cast<const uint32_t*>(&ll);
          }
          if (px < SW) {
            const int off = (px + 4) * 16;
            // c0 = h0..7 | c1 = h8 h9 l0..5 | c2 = l6..9 h0..3 | c3 = h4..9 0 0   (see the header comment)
            *reinterpret_cast<uint4*>(am + off) = make_uint4(hp[0], hp[1], hp[2], hp[3]);
            *reinterpret_cast<uint4*>(am + A_CHUNK + off) = make_uint4(hp[4], lp[0], lp[1], lp[2]);
            *reinterpret_cast<uint4*>(am + 2 * A_CHUNK + off) = make_uint4(lp[3], lp[4], hp[0], hp[1]);
            *reinterpret_cast<uint4*>(am + 3 * A_CHUNK + off) = make_uint4(hp[2], hp[3], hp[4], 0u);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&raw_empty[s]);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[a]);
        if (tid == 0 && wid == 4) TRACE(3, 3);
        if (++a == NA) { a = 0; aph ^= 1u; }
        if (++s == NRAW) { s = 0; sph ^= 1u; }
      }
      r += c.nr;
    }
  } else if (wid >= 14) {
    // ===== epilogue: drain, store, zero =====
    const int q4 = wid & 3;
    // from logits the drain does twice the work per pixel (softmax of the output pixel + adjoint), so a second set of
    // four warps (18-21) takes pixel tile 1; each set drains and zeroes only its tile's accumulator columns
    const int dset = wid >= 18 ? 1 : 0;
    const int ndset = ntile == 2 ? 2 : 1;
    const int mt0 = ndset == 2 ? dset : 0, mt1 = ndset == 2 ? dset + 1 : ntile;
    const int zc0 = ndset == 2 ? dset * RMAX * KP : 0, zc1 = ndset == 2 ? (dset + 1) * RMAX * KP : TBUF;
    float unscale = 1.f;
    const float g0 = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
    const size_t plane = (size_t)P.H * P.W;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
    auto zero_accumulators = [&](int buf) {
      for (int c = zc0; c < zc1; c += 8)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(lane_base + buf * TBUF + c), "r"(0u) : "memory");
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_ready[buf]);
    };
    if (dset < ndset) {
    zero_accumulators(0);
    zero_accumulators(1);
    }
    // the weight images: these four warps are idle until the first chunk is finished.  First the power-of-two scale that
    // brings the largest coefficient magnitude into [2^12, 2^13) (every CTA finds it from the 2 x K*9*Kp4 coefficients,
    // L2-resident), then the fp16 (w1, w2) images.
    if (dset == 0) {
      const int etid = threadIdx.x - 14 * 32;
      const int ncoef = P.K * T * T * P.Kp4;
      float mx = 0.f;
      for (int e = etid; e < 2 * ncoef; e += 128) mx = fmaxf(mx, fabsf(__ldg(P.Wc[e >= ncoef] + (e >= ncoef ? e - ncoef : e))));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane == 0) wmax_s[q4] = mx;
      asm volatile("bar.sync 1, 128;" ::: "memory");
      mx = fmaxf(fmaxf(wmax_s[0], wmax_s[1]), fmaxf(wmax_s[2], wmax_s[3]));
      int wexp = 0;
      if (mx > 0.f && mx < 3.0e38f) wexp = W_TARGET_LOG2 - ilogbf(mx);
      if (wexp > 100) wexp = 100;                       // denormal-sized coefficients: keep the scale finite
      const float wscale = scalbnf(1.f, wexp);
      unscale = scalbnf(1.f, -(wexp + A_SCALE_LOG2));
      for (int e = etid; e < 2 * 3 * WROWS; e += 128) {
        const int sweep = e / (3 * WROWS);
        build_weight_row(P.Wc[sweep], w_img + sweep * W_IMG, e - sweep * 3 * WROWS, P.K, P.Kp4, wscale);
      }
      if (etid == 0) unscale_s = unscale;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&w_full);
    } else {
      mbar_wait(&w_full, 0u, 7);                       // the first set has published the scale
      unscale = *reinterpret_cast<volatile float*>(&unscale_s);
    }
    const float g = g0 * unscale;
    int i = 0, ls = 0;
    unsigned lph = 0;
    for (int sweep = 0; sweep < 2 && dset < ndset; ++sweep)
    for (long long r = R0; r < R1; ++i) {
      const Chunk c = next_chunk(r, R0, R1, P.H, rc);
      const int buf = i & 1;
      if (lane == 0 && wid == 14) CTRACE(2);
      mbar_wait(&accum_full[buf], (unsigned)(i >> 1) & 1u, 8);
      if (lane == 0 && wid == 14) CTRACE(3);
      asm volatile("tcgen05.fence::after_thread_sync;");
      for (int orow = 0; orow < c.nr; orow += 2) {
        const int nrow = orow + 1 < c.nr ? 2 : 1;
        if (FROM_LOGITS) {
          // the logit rows of this row pair have landed (ring slots ls, ls + 1)
          mbar_wait(&l_full[ls], lph, 10);
          if (nrow == 2) mbar_wait(&l_full[(ls + 1) % NL], (ls + 1 == NL) ? (lph ^ 1u) : lph, 10);
        }
        for (int mt = mt0; mt < mt1; ++mt) {
          const int col = mt * 128 + q4 * 32 + lane;
          const bool live = col < P.W;
          uint32_t v[2][16];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int orh = orow + h < RMAX ? orow + h : orow;
#pragma unroll
            for (int ch = 0; ch < 16; ch += 8) {
              const uint32_t taddr = lane_base + (uint32_t)(buf * TBUF + (mt * RMAX + orh) * KP + ch);
              asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                           : "=r"(v[h][ch]), "=r"(v[h][ch + 1]), "=r"(v[h][ch + 2]), "=r"(v[h][ch + 3]), "=r"(v[h][ch + 4]),
                             "=r"(v[h][ch + 5]), "=r"(v[h][ch + 6]), "=r"(v[h][ch + 7])
                           : "r"(taddr));
            }
          }
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (live) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              if (h < nrow) {
                float* dst = P.out[sweep] + (size_t)c.n * P.out_sn[sweep] + (size_t)(c.h0 + orow + h) * P.W + col;
                if (!FROM_LOGITS) {
                  // (a branch per channel cost ~10 instructions and a uniform-register reload per store: the drain ran at
                  // one store per ~68 clk and warp; K = 10 takes the straight-line form)
                  if (P.K == 10) {
#pragma unroll
                    for (int o = 0; o < 10; ++o) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);
                  } else {
#pragma unroll
                    for (int o = 0; o < 9; ++o) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);
                  }
                } else {
                  // softmax adjoint: d logit_o = inv_temp * p_o * (g_o - sum_k g_k p_k), p = softmax of the output
                  // tensor's own logits at this pixel (staged row: column c at index c + 4, conflict-free across lanes)
                  const float* lp = reinterpret_cast<const float*>(l_ring + ((ls + h) % NL) * RAW_SLOT) + col + 4;
                  float pr[10];
                  float mx = -3.0e38f;
#pragma unroll
                  for (int o = 0; o < 10; ++o) {
                    pr[o] = o < P.K ? lp[o * SW] : -3.0e38f;
                    mx = fmaxf(mx, pr[o]);
                  }
                  float sum = 0.f;
#pragma unroll
                  for (int o = 0; o < 10; ++o) {
                    pr[o] = o < P.K ? __expf((pr[o] - mx) * P.inv_temp) : 0.f;
                    sum += pr[o];
                  }
                  const float inv = 1.f / sum;
                  float dot = 0.f;
#pragma unroll
                  for (int o = 0; o < 10; ++o) {
                    pr[o] *= inv;
                    dot = fmaf(g * __uint_as_float(v[h][o]), pr[o], dot);
                  }
                  if (P.K == 10) {
#pragma unroll
                    for (int o = 0; o < 10; ++o) dst[(size_t)o * plane] = P.inv_temp * pr[o] * (g * __uint_as_float(v[h][o]) - dot);
                  } else {
#pragma unroll
                    for (int o = 0; o < 9; ++o) dst[(size_t)o * plane] = P.inv_temp * pr[o] * (g * __uint_as_float(v[h][o]) - dot);
                  }
                }
              }
            }
          }
        }
        if (FROM_LOGITS) {
          // both tiles of the row pair are done: hand the ring slots back (one arrival per drain warp)
          __syncwarp();
          for (int h = 0; h < nrow; ++h) {
            if (lane == 0) mbar_arrive(&l_empty[ls]);
            if (++ls == NL) { ls = 0; lph ^= 1u; }
          }
        }
      }
      r += c.nr;
      if (lane == 0 && wid == 14) CTRACE(4);
      zero_accumulators(buf);
      if (lane == 0 && wid == 14) CTRACE(5);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 3) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

}  // namespace bwdrb10h

int local_bwd_tcrb10h_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, int from_logits,
                          float inv_temp, cudaStream_t st) {
  using namespace bwdrb10h;
  const int B = m.B, K = m.K, H = m.H, W = m.W, sms = m.sms;
  if ((K != 9 && K != 10) || m.pad != 1 || W % 4 != 0 || W > MAXW || W < 8) return -1;
  if ((long long)B * H < 8LL * sms && !options().tc10_force) return -1;   // too few rows to fill the SMs: FFMA2 is faster
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, W + 8, 1, K)) return -1;
  if (!make_map_4d(&my, m.y, m, W + 8, 1, K)) return -1;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_bwd_tcrb10h_kernel<false>), (int)(SMEM_BYTES)));
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_bwd_tcrb10h_kernel<true>), (int)(SMEM_BYTES_FL)));
  const int Kp4 = (K + 3) & ~3;
  Params P{B, H, W, K, {Wx, Wy}, Kp4, g.grad_loss, {g.gx, g.gy}, {g.gx_sn, g.gy_sn}, from_logits, inv_temp, {m.x.p, m.y.p},
           {m.x.sn, m.y.sn}, {m.x.sc, m.y.sc}, {m.x.sh, m.y.sh}};
  // one launch, two sweeps per CTA: dL/dx from y (sweep 0), then dL/dy from x (sweep 1)
  if (from_logits) local_bwd_tcrb10h_kernel<true><<<sms, NTHREADS_FL, SMEM_BYTES_FL, st>>>(my, mx, P);
  else local_bwd_tcrb10h_kernel<false><<<sms, NTHREADS, SMEM_BYTES, st>>>(my, mx, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic
