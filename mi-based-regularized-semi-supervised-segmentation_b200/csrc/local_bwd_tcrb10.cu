// Backward sweeps of the local IIC term on the tensor cores for 10 clusters, 3 x 3 window (BASELINE config 2: the
// udaiic default head of the benchmark): row-block scheme of local_bwd_tcrb.cu with two changes that make it pay at
// K = 10, where padding the 10 input channels to two 8-channel slices would cost as many MMAs as the FFMA2 kernel has
// FMA time:
//  * the reduction dimension of an MMA need not be "8 channels of one tap".  In the no-swizzle K-major layout the two
//    16-byte chunks of an operand row are independent arrays, so the main MMAs take channels 0-7 (one per column tap tx),
//    and ONE extra "leftover" MMA per source row takes the slots (ch 8, ch 9) x (tx 0, 1, 2): the transform warps write a
//    second row buffer whose pixel row b holds those six tap-shifted values, the weight image a matching tile.
//    8 MMAs (4 products) per source row and 128-pixel tile instead of 12.
//  * the B*H image rows are dealt to the CTAs as equal contiguous shares cut into chunks of at most 16 rows (no tail
//    wave; an item is a chunk, not a fixed block), and the whole weight image (12 KB) is loaded once per CTA.
//   out[n,o,r,c] = g * sum_{cin,ty,tx} Wc[cin][ty*3+tx][o] * src[n,cin,r+ty-1,c+tx-1]     (iic_loss.py:123, backward)
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace bwdrb10 {
using namespace tc;

constexpr int T = 3, PAD = 1;
constexpr int KP = 16;                   // accumulator columns per output row (10 channels used)
constexpr int RMAX = 8;                  // output rows per item: 8 x 2 tiles x 16 = 256 TMEM columns, double buffered so that
                                         // the drain of item i overlaps the MMAs of item i+1
constexpr int TBUF = 2 * RMAX * KP;      // TMEM columns of one accumulator buffer
constexpr int APX = 272;
constexpr int MAXW = 248;
constexpr int A_PART = 2 * APX * 16;     // 8704
constexpr int A_ROW = 2 * A_PART;        // 17408: fp32 part + bf16 part
constexpr int A_SLOT = 2 * A_ROW;        // main row buffer + leftover row buffer
constexpr int NA = 4;
constexpr int RAW_SLOT = 10 * 256 * 4;   // 10240
constexpr int NRAW = 6;
constexpr int WROWS = T * KP;            // 48 rows per weight chunk
constexpr int W_TILE = 4 * WROWS * 16;   // 3072
constexpr int W_IMG = 4 * W_TILE;        // tx 0, 1, 2 and the leftover tile
constexpr int NTHREADS = 576;             // warps: 0 TMA, 3 TMEM + weights, 1 2 12 13 MMA issuers, 4-11 transform, 14-17 epilogue
constexpr int SMEM_BYTES = NA * A_SLOT + 2 * W_IMG + NRAW * RAW_SLOT + 1024;   // both sweeps' weight images stay resident



#ifdef IIC_TC_TRACE
__device__ long long g_trace[4][64][6];
#define TRACE(role, slot) do { if (blockIdx.x == 0 && tt >= 16 && tt < 80) g_trace[role][tt - 16][slot] = clock64(); } while (0)
#else
#define TRACE(role, slot) do { } while (0)
#endif

struct Params {
  int B, H, W, K;
  const float* Wc[2];           // coefficient tensors of iic_local_epilogue: sweep 0 = Wx (dL/dx, source y), sweep 1 = Wy
  int Kp4;                      // their row length
  const float* grad_loss;
  float* out[2];
  long long out_sn[2];          // sample strides of the two gradient tensors in elements
};

// Wc[cin][ty*3+tx][Kp4] -> tiles tx = 0..2 (input channels 0-7) and the leftover tile (slots (ch 8, ch 9) x tx);
// each tile {fp32 [2 chunks][48 rows][4 slots], bf16 [wh, wl][48 rows][8 slots]}, rows ordered (2-ty)*16 + o.
// Every CTA builds both sweeps' images (2 x 12 KB from 2 x 3.6 KB of L2-resident coefficients) straight into its own
// shared memory: no extra launch, no scratch allocation.  e = row in [0, 2 * 4 * 48).
__device__ __forceinline__ void build_weight_row(const float* __restrict__ Wc, unsigned char* img, int e, int K, int Kp4) {
  const int row = e % WROWS, tile = e / WROWS;
  const int ty = T - 1 - row / KP, o = row % KP;
  float v[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    int cin, tx;
    if (tile < 3) { cin = q; tx = tile; }
    else { cin = 8 + (q & 1); tx = q >> 1; }                 // slots (8,tx0) (9,tx0) (8,tx1) (9,tx1) (8,tx2) (9,tx2) - -
    v[q] = (cin < K && o < K && tx < T) ? __ldg(Wc + ((size_t)cin * T * T + ty * T + tx) * Kp4 + o) : 0.f;
  }
  float4* t4 = reinterpret_cast<float4*>(img) + (size_t)tile * (4 * WROWS);
  t4[row] = make_float4(v[0], v[1], v[2], v[3]);
  t4[WROWS + row] = make_float4(v[4], v[5], v[6], v[7]);
  reinterpret_cast<uint4*>(t4)[2 * WROWS + row] = pack8<false>(v);
  reinterpret_cast<uint4*>(t4)[3 * WROWS + row] = pack8<true>(v);
}

// the chunk of image rows that starts at global row r (rows of all images, B*H) inside the CTA share [r, R1)
struct Chunk { int n, h0, nr; };
__device__ __forceinline__ Chunk next_chunk(long long r, long long R1, int H, int rc) {
  Chunk c;
  c.n = (int)(r / H);
  c.h0 = (int)(r - (long long)c.n * H);
  c.nr = rc;
  if (c.nr > H - c.h0) c.nr = H - c.h0;
  if (c.nr > R1 - r) c.nr = (int)(R1 - r);
  return c;
}

__global__ void __launch_bounds__(NTHREADS, 1)
local_bwd_tcrb10_kernel(const __grid_constant__ CUtensorMap map0, const __grid_constant__ CUtensorMap map1, const Params P) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW], a_full[NA], a_empty[NA], w_full, accum_full[2], tmem_ready[2];
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* a_ring = smem;
  unsigned char* w_img = smem + NA * A_SLOT;
  unsigned char* raw_ring = w_img + 2 * W_IMG;
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
    for (int s = 0; s < 2; ++s) { mbar_init(&accum_full[s], 4); mbar_init(&tmem_ready[s], 4); }
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
        const Chunk c = next_chunk(r, R1, P.H, rc);
        for (int q = 0; q < c.nr + T - 1; ++q, ++t) {
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
      const Chunk c = next_chunk(r, R1, P.H, rc);
      const int buf = i & 1;
      mbar_wait(&tmem_ready[buf], (unsigned)(i >> 1) & 1u, 6);   // this buffer's accumulators are zeroed
      asm volatile("tcgen05.fence::after_thread_sync;");
      const int nq = c.nr + T - 1;
      for (int q = 0; q < nq; ++q, ++tt) {
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
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((nn >> 3) << 17) | (8u << 24);
            const uint32_t idesc_bf16 = (1u << 4) | (1u << 7) | (1u << 10) | ((nn >> 3) << 17) | (8u << 24);
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * TBUF + (mt * RMAX + (q - ty_max)) * KP);
            const uint64_t a_main = make_desc_kmajor_noswz(smem_u32(a_ring + a * A_SLOT), APX * 16) + (uint64_t)(mt * 128 + 8 - PAD);
            const uint64_t a_left = a_main + (uint64_t)(A_ROW / 16);
            const uint64_t b_base = w_base + (uint64_t)((T - 1 - ty_max) * KP);
#pragma unroll
            for (int tx = 0; tx < T; ++tx) {
              const uint64_t bt = b_base + (uint64_t)tx * (4 * WROWS);
              umma_bf16(d_tmem, a_main + (uint64_t)(A_PART / 16 + tx), bt + 2 * WROWS, idesc_bf16);
              umma_tf32(d_tmem, a_main + (uint64_t)tx, bt, idesc);
            }
            const uint64_t bl = b_base + (uint64_t)3 * (4 * WROWS);       // leftover tile: taps are inside the row
            umma_bf16(d_tmem, a_left + (uint64_t)(A_PART / 16), bl + 2 * WROWS, idesc_bf16);
            umma_tf32(d_tmem, a_left, bl, idesc);
          }
          if (par == 0) TRACE(1 + mt, 2);
          umma_commit(&a_empty[a]);
          if (q >= nq - 2) umma_commit(&accum_full[buf]);     // this issuer's last source row of the item
        }
        __syncwarp();
        if (++a == NA) { a = 0; aph ^= 1u; }
      }
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
      const Chunk c = next_chunk(r, R1, P.H, rc);
      for (int q = 0; q < c.nr + T - 1; ++q, ++t) {
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
        unsigned char* al = am + A_ROW;
        const float* raw = reinterpret_cast<const float*>(raw_ring + s * RAW_SLOT);
        for (int px = tid; px < SW; px += 128) {
          float v[8];
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) v[ch] = raw[ch * SW + px];
          const int off = (px + 4) * 16;
          *reinterpret_cast<float4*>(am + off) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(am + off + APX * 16) = make_float4(v[4], v[5], v[6], v[7]);
          *reinterpret_cast<uint4*>(am + A_PART + off) = pack8<true>(v);
          *reinterpret_cast<uint4*>(am + A_PART + off + APX * 16) = pack8<false>(v);
          float w[8];
#pragma unroll
          for (int tx = 0; tx < 3; ++tx) {
            const bool in = px + tx < SW;
            w[2 * tx] = (in && P.K > 8) ? raw[8 * SW + px + tx] : 0.f;
            w[2 * tx + 1] = (in && P.K > 9) ? raw[9 * SW + px + tx] : 0.f;
          }
          w[6] = 0.f; w[7] = 0.f;
          *reinterpret_cast<float4*>(al + off) = make_float4(w[0], w[1], w[2], w[3]);
          *reinterpret_cast<float4*>(al + off + APX * 16) = make_float4(w[4], w[5], w[6], w[7]);
          *reinterpret_cast<uint4*>(al + A_PART + off) = pack8<true>(w);
          *reinterpret_cast<uint4*>(al + A_PART + off + APX * 16) = pack8<false>(w);
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
    const float g = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
    const size_t plane = (size_t)P.H * P.W;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q4 * 32) << 16);
    auto zero_accumulators = [&](int buf) {
      for (int c = 0; c < TBUF; c += 8)
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(lane_base + buf * TBUF + c), "r"(0u) : "memory");
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_ready[buf]);
    };
    zero_accumulators(0);
    zero_accumulators(1);
    // the weight images: these four warps are idle until the first chunk is finished
    for (int e = threadIdx.x - 14 * 32; e < 2 * 4 * WROWS; e += 128) {
      const int sweep = e / (4 * WROWS);
      build_weight_row(P.Wc[sweep], w_img + sweep * W_IMG, e - sweep * 4 * WROWS, P.K, P.Kp4);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(&w_full);
    int i = 0;
    for (int sweep = 0; sweep < 2; ++sweep)
    for (long long r = R0; r < R1; ++i) {
      const Chunk c = next_chunk(r, R1, P.H, rc);
      const int buf = i & 1;
      mbar_wait(&accum_full[buf], (unsigned)(i >> 1) & 1u, 8);
      asm volatile("tcgen05.fence::after_thread_sync;");
      for (int mt = 0; mt < ntile; ++mt) {
        const int col = mt * 128 + q4 * 32 + lane;
        const bool live = col < P.W;
        for (int orow = 0; orow < c.nr; orow += 2) {
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
              if (orow + h < c.nr) {
                float* dst = P.out[sweep] + (size_t)c.n * P.out_sn[sweep] + (size_t)(c.h0 + orow + h) * P.W + col;
#pragma unroll
                for (int o = 0; o < 9; ++o) dst[(size_t)o * plane] = g * __uint_as_float(v[h][o]);     // K is 9 or 10 here
                if (P.K == 10) dst[(size_t)9 * plane] = g * __uint_as_float(v[h][9]);
              }
            }
          }
        }
      }
      r += c.nr;
      zero_accumulators(buf);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 3) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

}  // namespace bwdrb10

int local_bwd_tcrb10_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, cudaStream_t st) {
  using namespace bwdrb10;
  const int B = m.B, K = m.K, H = m.H, W = m.W, sms = m.sms;
  if ((K != 9 && K != 10) || m.pad != 1 || W % 4 != 0 || W > MAXW || W < 8) return -1;
  if ((long long)B * H < 8LL * sms && !options().tc10_force) return -1;   // too few rows to fill the SMs: FFMA2 is faster
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, W + 8, 1, K)) return -1;
  if (!make_map_4d(&my, m.y, m, W + 8, 1, K)) return -1;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_bwd_tcrb10_kernel), (int)(SMEM_BYTES)));
  const int Kp4 = (K + 3) & ~3;
  Params P{B, H, W, K, {Wx, Wy}, Kp4, g.grad_loss, {g.gx, g.gy}, {g.gx_sn, g.gy_sn}};
  // one launch, two sweeps per CTA: dL/dx from y (sweep 0), then dL/dy from x (sweep 1)
  local_bwd_tcrb10_kernel<<<sms, NTHREADS, SMEM_BYTES, st>>>(my, mx, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic
