// Joint of the local IIC term on the tensor cores for up to 10 clusters, 3 x 3 window (BASELINE config 2):
//   J[dy][dx][i][j] = sum_{n,u,v} x[n,i,u+dy-1,v+dx-1] * y[n,j,u,v]                       (iic_loss.py:120-123)
// The FFMA2 kernel (local_fwd_fast3.inc) needs 900 FMAs per pixel and sits at 57 % of the FP32 pipe; the round-1
// tensor-core attempt lost because every x element was rewritten six times (three column shifts x fp32 + bf16 copies).
// Here every element is written ONCE:
//   * operands are fp16 hi/lo pairs (a = a1 + a2, 22 bits; all four part products are computed, fp32 accumulation),
//     staged PIXEL-major: one 128-byte group per pixel holding TWO image rows, 32 slots each
//     [a1(0..9) a2(0..9) 0 x 12 | the same for the next row], 128-byte swizzled;
//   * the MMA consumes them MN-major (reduction = pixels, 16 per instruction).  The M atoms of A are two consecutive x row
//     pairs (four rows); the N atoms of B are the SAME y row pair at three pixel shifts -- an atom stride of one pixel, i.e.
//     overlapping atoms: tools/mn_major_micro.cu shows the hardware takes them and applies the swizzle to the absolute
//     address.  One MMA (M = 128, N = 192, K = 16 pixels) adds 16 pixels of two y rows into all nine displacements:
//     D[(x row a, x slot), (shift, y row r, y slot)], dy = a - r.
// Per CTA (one per SM, its share of the B*H image rows): seven warps stage the x row pairs and seven the y row pairs
// straight from global memory (thread = two pixels of a row, 8-byte loads, the next pair's loads in flight while this one
// is split, packed and stored with swizzled 16-byte stores; the simplex assertion of iic_loss.py:113 rides along) -> two
// issuing warps, alternate pairs (these MMAs hold the issuing lane for as long as they execute) -> two TMEM accumulator
// sets taken in turn by y row pair -> four warps read each set out as soon as its pair is done (fp32 register sums: short
// tensor-core accumulation runs keep the truncation bias of the TMEM adds near 1e-6) and at the end add the
// (part x part) products and the two y rows and write this CTA's slot in the [d][i][j] layout of iic_finish.
// DESIGN.md 4.1c has the measurements behind each of these choices.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace fwdtcj10 {
using namespace tc;

constexpr int PAD = 1;
constexpr int NPXB = 248;                // pixels per row-pair buffer (15 k-steps of 16 + the two shifts, rounded to 8)
constexpr int PAIRB = NPXB * 128;        // 31744 bytes, a multiple of the 1024-byte swizzle period
constexpr int NXP = 4;                   // x pair ring; slot 0 is mirrored in slot NXP so that two consecutive slots
                                         // starting anywhere in the ring are contiguous
constexpr int NYP = 2;                   // y pair ring
constexpr int NSET = 2, NCOL = 192;      // TMEM accumulator sets (NSET == NYP: y_done of a pair is also "set full")
constexpr float SCALE = 1024.f;          // both maps are scaled by 2^10 before the split; 2^-20 in the drain
constexpr int MAXW = 224;                // two rows of W / 2 pixel pairs per staging group of 224 threads; (W + 2) <= 15 k-steps of 16
constexpr int NTHREADS = 20 * 32;        // warps: 0-6 x pairs, 7-13 y pairs, 14 and 15 MMA issue (14 allocates TMEM), 16-19 drain.
                                         // 20 warps leave 96 registers per thread; 21 would leave 80.
constexpr int GROUP = 7 * 32;            // threads of a staging group: two rows x W / 2 pixel pairs
constexpr int X_BYTES = (NXP + 1) * PAIRB;
constexpr int SMEM_BYTES = X_BYTES + NYP * PAIRB + 1024;

struct Params {
  const float* x; long long x_sn, x_sc, x_sh;
  const float* y; long long y_sn, y_sc, y_sh;
  int B, H, W, K;
  float* partial;      // [gridDim.x][9][K][K]
  int* flags;          // nullable: simplex assertion on x
  int from_logits;     // the maps hold the cluster head's LOGITS: softmax(logit * inv_temp) over the channels in the staging
  float inv_temp;      // warps (contrastyou/trainer/_utils.py:15-23 fused), before the split
#ifdef IIC_TCJ_DEBUG
  int dbg;             // harness only: 1 = no MMAs, 2 = no transform work, 8 = no global loads, 64 = drain without TMEM loads,
                       // 128 = issuers do not wait for the drain
#endif
};
#ifdef IIC_TCJ_DEBUG
#define TCJ_DBG(bit) (P.dbg & (bit))
__device__ long long g_tcj_trace[8][64];
__device__ unsigned long long g_tcj_cta[160][2];      // per CTA: %globaltimer at start and end
#define TCJ_T(role, idx) do { if (blockIdx.x == 0 && lane == 0 && (idx) < 64) g_tcj_trace[role][idx] = clock64(); } while (0)
#else
#define TCJ_T(role, idx) do { } while (0)
#define TCJ_DBG(bit) 0
#endif

// MN-major, SWIZZLE_128B: LBO = byte stride between the 64-slot atoms along M / N, SBO = stride between groups of 8 pixels
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// Walk over the chunks (rows of one image) of the CTA share [R0, R1) of the B*H image rows.  Local x row lr is image row
// h0 - 1 + lr, local y row ly is image row h0 + ly; y pair Q (rows 2Q, 2Q+1) meets x pairs Q and Q + 1 (rows 2Q .. 2Q+3).
struct Chunk {
  int n, h0, nr, npy;          // image, first row, rows, y pairs (x pairs = npy + 1)
};
__device__ __forceinline__ Chunk chunk_at(long long r, long long R1, int H) {
  Chunk c;
  c.n = (int)(r / H);
  c.h0 = (int)(r - (long long)c.n * H);
  c.nr = H - c.h0;
  if (c.nr > R1 - r) c.nr = (int)(R1 - r);
  c.npy = (c.nr + 1) >> 1;
  return c;
}

// One thread stages two consecutive pixels of one row of the pair, all channels (ten 8-byte loads).  Thread t of the 256 of
// a group: row t / npp, pixel pair t % npp (npp = W / 2 <= 128).  The staging is bound by instruction issue and latency,
// not by bytes: sixteen staging warps with little work each, and loads without predicates -- a row or column outside
// the map is read from the nearest one inside and multiplied by zero (`mul`, which otherwise carries the 2^10 scale).
struct Tile { float2 f[10]; float mul; };

template <bool IS_Y, bool FULLK>
__device__ __forceinline__ void load_tile(Tile& t, const Params& P, const Chunk& c, int pair, int pp, int rr) {
  const float* base = IS_Y ? P.y : P.x;
  const long long sn = IS_Y ? P.y_sn : P.x_sn, sc = IS_Y ? P.y_sc : P.x_sc, sh = IS_Y ? P.y_sh : P.x_sh;
  const int npp = P.W >> 1;
  const int lrow = 2 * pair + rr;
  const int row = IS_Y ? c.h0 + lrow : c.h0 - PAD + lrow;
  // y rows past the chunk belong to another CTA (or image): they must count as zero.  x rows past the rows any valid
  // y row meets only multiply those zeros, so any finite value will do (row inside the image) or zero (outside).
  const bool ok = pp < npp && row >= 0 && row < P.H && (!IS_Y || lrow < c.nr) && !TCJ_DBG(8);
  t.mul = ok ? SCALE : 0.f;
  const int rowc = min(max(row, 0), P.H - 1), ppc = min(pp, npp - 1);
  const float* ptr = base + (long long)c.n * sn + (long long)rowc * sh + 2 * ppc;
#pragma unroll
  for (int ch = 0; ch < 10; ++ch)
    t.f[ch] = __ldg(reinterpret_cast<const float2*>(ptr + (FULLK ? ch : min(ch, P.K - 1)) * sc));
}

// The cluster head's SoftmaxWithT on one thread's two pixels, in place (from-logits form).  Channels beyond K hold clamped
// duplicates of channel K - 1 and are zeroed by the store's per-channel factor, so they only must not enter max and sum.
template <bool FULLK>
__device__ __forceinline__ void softmax_tile(Tile& t, int K, float inv_temp) {
  float2 mx = t.f[0];
#pragma unroll
  for (int ch = 1; ch < 10; ++ch)
    if (FULLK || ch < K) mx = make_float2(fmaxf(mx.x, t.f[ch].x), fmaxf(mx.y, t.f[ch].y));
  float2 sum = make_float2(0.f, 0.f);
#pragma unroll
  for (int ch = 0; ch < 10; ++ch) {
    if (FULLK || ch < K) {
      t.f[ch] = make_float2(__expf((t.f[ch].x - mx.x) * inv_temp), __expf((t.f[ch].y - mx.y) * inv_temp));
      sum = __fadd2_rn(sum, t.f[ch]);
    }
  }
  const float2 inv = make_float2(1.f / sum.x, 1.f / sum.y);
#pragma unroll
  for (int ch = 0; ch < 10; ++ch)
    if (FULLK || ch < K) t.f[ch] = __fmul2_rn(t.f[ch], inv);
}

// Split, pack and store one thread's two pixels into the pair buffer(s): pixel b = column + boff, the row's three 16-byte
// chunks at ((4 * row + k) ^ (b & 7)).  Eight consecutive lanes (one phase of a 128-bit store) hold pixels 2 apart, which
// the swizzle sends to four distinct bank groups only; so the upper four lanes of a phase take their two pixels in the
// other order and the eight stores of a phase fall on eight different groups.
// Split of the value scaled by 2^10: hi = cut to 11 significant bits (a mask; exact in fp16), lo = fp16(value - hi): 21-22
// bits in all.  The scale keeps the lo parts out of the fp16 subnormals, which the tensor core reads as zero (measured:
// unscaled maps lose 1.5e-4 of the joint); what still falls below 2^-14 is at most 6e-8 of the unscaled value range.
template <bool FULLK>
__device__ __forceinline__ void store_tile(const Tile& t, unsigned char* dst, unsigned char* dst2, int boff, int pp, int rr,
                                           bool flip, int K) {
  float2 hi[10], lo[10];
#pragma unroll
  for (int ch = 0; ch < 10; ++ch) {
    const float m = (FULLK || ch < K) ? t.mul : 0.f;
    const float2 sv = __fmul2_rn(t.f[ch], make_float2(m, m));
    hi[ch] = make_float2(__uint_as_float(__float_as_uint(sv.x) & 0xFFFFE000u), __uint_as_float(__float_as_uint(sv.y) & 0xFFFFE000u));
    lo[ch] = __ffma2_rn(hi[ch], make_float2(-1.f, -1.f), sv);
  }
  const int cb = 4 * rr;
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    uint32_t hp[5], lp[5];
#pragma unroll
    for (int c2 = 0; c2 < 5; ++c2) {
      const __half2 h0 = __floats2half2_rn(hi[2 * c2].x, hi[2 * c2 + 1].x), h1 = __floats2half2_rn(hi[2 * c2].y, hi[2 * c2 + 1].y);
      const __half2 l0 = __floats2half2_rn(lo[2 * c2].x, lo[2 * c2 + 1].x), l1 = __floats2half2_rn(lo[2 * c2].y, lo[2 * c2 + 1].y);
      const uint32_t uh0 = *reinterpret_cast<const uint32_t*>(&h0), uh1 = *reinterpret_cast<const uint32_t*>(&h1);
      const uint32_t ul0 = *reinterpret_cast<const uint32_t*>(&l0), ul1 = *reinterpret_cast<const uint32_t*>(&l1);
      hp[c2] = ((s2 == 0) != flip) ? uh0 : uh1;
      lp[c2] = ((s2 == 0) != flip) ? ul0 : ul1;
    }
    const int b = 2 * pp + (s2 ^ (flip ? 1 : 0)) + boff;
    const int sw = b & 7;
    // slots [h0..h9 | l0..l9 | 0 x 12] = chunks (h0-7) (h8 h9 l0-5) (l6-9 0 0 0 0) (0)
    const uint4 c0 = make_uint4(hp[0], hp[1], hp[2], hp[3]);
    const uint4 c1 = make_uint4(hp[4], lp[0], lp[1], lp[2]);
    const uint4 c2v = make_uint4(lp[3], lp[4], 0u, 0u);
    unsigned char* px = dst + b * 128;
    *reinterpret_cast<uint4*>(px + (((cb + 0) ^ sw) << 4)) = c0;
    *reinterpret_cast<uint4*>(px + (((cb + 1) ^ sw) << 4)) = c1;
    *reinterpret_cast<uint4*>(px + (((cb + 2) ^ sw) << 4)) = c2v;
    if (dst2) {
      unsigned char* px2 = dst2 + b * 128;
      *reinterpret_cast<uint4*>(px2 + (((cb + 0) ^ sw) << 4)) = c0;
      *reinterpret_cast<uint4*>(px2 + (((cb + 1) ^ sw) << 4)) = c1;
      *reinterpret_cast<uint4*>(px2 + (((cb + 2) ^ sw) << 4)) = c2v;
    }
  }
}

// The staging loop of one group of seven warps (x: warps 0-6, y: warps 7-13).  Pair number `count` of the group (running
// over the chunks) goes to ring slot count % NRING once the slot's last occupant has been read: x slots are released by
// the issuer's x_free commits, y slots by y_done.  The next pair's loads are issued before this pair is converted; the two
// register tiles swap roles every step.
template <bool IS_Y, bool FULLK>
__device__ __forceinline__ void stage_pairs(const Params& P, long long R0, long long R1, unsigned char* ring,
                                            unsigned char* mirror, uint64_t* full, uint64_t* released) {
  constexpr int NRING = IS_Y ? NYP : NXP;
  const int tid = IS_Y ? threadIdx.x - GROUP : threadIdx.x, lane = threadIdx.x & 31;
  const int npp = P.W >> 1, rr = tid >= npp ? 1 : 0, pp = tid - rr * npp;
  const bool flip = (lane >> 2) & 1;
  long long r = R0;
  if (r >= R1) return;
  Chunk c = chunk_at(r, R1, P.H);
  int pl = 0, count = 0;
  bool bad = false;
  Tile ta, tb;
  load_tile<IS_Y, FULLK>(ta, P, c, 0, pp, rr);
  int pending = -1;       // slot written but not yet published
  auto publish = [&]() {
    if (pending < 0) return;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(&full[pending]);
    pending = -1;
  };
  // one step: issue the loads of the job after this one into `nxt`, then convert and publish `cur`; false after the last job
  auto step = [&](Tile& cur, Tile& nxt) -> bool {
    long long rn = r;
    Chunk cn = c;
    int pn = pl + 1;
    if (pn >= (IS_Y ? c.npy : c.npy + 1)) { rn = r + c.nr; pn = 0; if (rn < R1) cn = chunk_at(rn, R1, P.H); }
    const bool more = rn < R1;
    if (more) load_tile<IS_Y, FULLK>(nxt, P, cn, pn, pp, rr);
    publish();            // the previous pair: its stores have had the load issue above to drain before the fence waits for them
    if (count >= NRING) mbar_wait(&released[count % NRING], (unsigned)(count / NRING - 1) & 1u, IS_Y ? 3 : 2);
    const int slot = count % NRING;
    if (!TCJ_DBG(2)) {
      if (P.from_logits) softmax_tile<FULLK>(cur, P.K, P.inv_temp);
      if (!IS_Y && P.flags && cur.mul != 0.f) {
        // simplex(x_out) of iic_loss.py:113 on the rows of the map
        float2 sum = cur.f[0];
#pragma unroll
        for (int ch = 1; ch < 10; ++ch) sum = __fadd2_rn(sum, (FULLK || ch < P.K) ? cur.f[ch] : make_float2(0.f, 0.f));
        if (!(fabsf(sum.x - 1.f) <= 2e-4f) || !(fabsf(sum.y - 1.f) <= 2e-4f)) bad = true;
      }
      if (pp < npp)
        store_tile<FULLK>(cur, ring + slot * PAIRB, (!IS_Y && slot == 0) ? mirror : nullptr, IS_Y ? 2 : 1, pp, rr, flip, P.K);
    }
    pending = slot;
    ++count;
    r = rn; c = cn; pl = pn;
    return more;
  };
  while (true) {
    if (!step(ta, tb)) break;
    if (!step(tb, ta)) break;
  }
  publish();
  if (!IS_Y && P.flags && __any_sync(0xffffffffu, bad) && lane == 0) atomicOr(P.flags, IIC_FLAG_NOT_SIMPLEX);
}

__global__ void __launch_bounds__(NTHREADS, 1) local_joint_tcj10_kernel(const Params P) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t x_full[NXP], x_free[NXP], y_full[NYP], y_done[NYP], set_free[NSET];
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* x_ring = smem;
  unsigned char* y_ring = smem + X_BYTES;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long rows_total = (long long)P.B * P.H;
  const long long R0 = (long long)blockIdx.x * rows_total / gridDim.x;
  const long long R1 = (long long)(blockIdx.x + 1) * rows_total / gridDim.x;
  const int ksteps = (P.W + 2 + 15) / 16;
  if (wid == 0) TCJ_T(0, 0);
#ifdef IIC_TCJ_DEBUG
  if (threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_tcj_cta[blockIdx.x][0] = t; }
#endif

  if (threadIdx.x == 0) {
    for (int s = 0; s < NXP; ++s) { mbar_init(&x_full[s], 7); mbar_init(&x_free[s], 2); }
    for (int s = 0; s < NYP; ++s) { mbar_init(&y_full[s], 7); mbar_init(&y_done[s], 1); }
    for (int s = 0; s < NSET; ++s) mbar_init(&set_free[s], 4);
    mbar_fence_init();
  }
  if (wid == 14) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // the pair buffers start as zeros: the columns outside the map and the unused slots are never written again
  for (int e = threadIdx.x; e < (X_BYTES + NYP * PAIRB) / 16; e += NTHREADS) reinterpret_cast<uint4*>(smem)[e] = make_uint4(0, 0, 0, 0);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem_base = tmem_base_s;
  if (wid == 0) TCJ_T(0, 1);

  if (wid < 14) {
    if (P.K == 10) {
      if (wid < 7) stage_pairs<false, true>(P, R0, R1, x_ring, x_ring + NXP * PAIRB, x_full, x_free);
      else stage_pairs<true, true>(P, R0, R1, y_ring, nullptr, y_full, y_done);
    } else {
      if (wid < 7) stage_pairs<false, false>(P, R0, R1, x_ring, x_ring + NXP * PAIRB, x_full, x_free);
      else stage_pairs<true, false>(P, R0, R1, y_ring, nullptr, y_full, y_done);
    }
  } else {
    // ===== warps 14, 15: MMA issue (even / odd pairs); warps 16-19: drain (TMEM lane quarter = wid & 3) =====
    // Issue, per y row pair: `ksteps` MMAs (M = 128: two x pairs; N = 192: the y pair at three shifts; K = 16 pixels),
    // kind::f16, fp16 operands, fp32 accumulator, A and B MN-major (bits 15, 16).
    // Drain: every pair's accumulator set is read out as soon as its MMAs are done and added up in registers in fp32 with
    // rounding -- the tensor core adds with truncation, and runs longer than one pair (15 MMAs) would leave a bias of 1e-5
    // in the joint (measured with two sets accumulated over the CTA's whole share: 1.7e-5).  tcgen05.mma of these MN-major
    // tiles issues at the rate it executes (~130 clk each, traced: the issuing lane is held), so one warp that waits for a
    // pair's operands and then issues leaves the tensor pipe idle during the waits (~900 clk a pair): two warps take the
    // pairs in turn (one accumulator set each), the second waiting while the first issues.
    const uint32_t idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(NCOL >> 3) << 17) | (8u << 24);
    const int a = wid & 3;                      // TMEM lane quarter = x row of the A tile
    const uint32_t lane_base = tmem_base + ((uint32_t)(a * 32) << 16);
    // tot[shift][y row][j]: the hi and lo y slots added
    float tot[3][2][10];
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int yr = 0; yr < 2; ++yr)
#pragma unroll
        for (int j = 0; j < 10; ++j) tot[s][yr][j] = 0.f;

    auto issue = [&](int yq, int ql, int xpbase, bool last_of_chunk) {
      const int ys = yq % NYP;
      const int xp1 = xpbase + ql + 1;                    // the later of the two x pairs (staged in order)
      TCJ_T(2, yq);
      mbar_wait(&y_full[ys], (unsigned)(yq / NYP) & 1u, 5);
      mbar_wait(&x_full[xp1 % NXP], (unsigned)(xp1 / NXP) & 1u, 6);
      // the accumulator set of this pair has been read out by the four drain warps (pair yq - NSET)
      if (yq >= NSET && !TCJ_DBG(128)) mbar_wait(&set_free[yq % NSET], (unsigned)((yq - NSET) / NSET) & 1u, 7);
      asm volatile("tcgen05.fence::after_thread_sync;");
      TCJ_T(1, yq);
      if (lane == 0) {
        const int xs = (xpbase + ql) % NXP;
        const uint64_t a0 = make_desc_mn_sw128(smem_u32(x_ring + xs * PAIRB), PAIRB);
        const uint64_t b0 = make_desc_mn_sw128(smem_u32(y_ring + ys * PAIRB), 128);
        const uint32_t d_tmem = tmem_base + (uint32_t)((yq % NSET) * NCOL);
        for (int k = 0; k < (TCJ_DBG(1) ? 0 : ksteps); ++k)     // 16 pixels = 2048 bytes = 128 address units
          umma_bf16(d_tmem, a0 + (uint64_t)(k * 128), b0 + (uint64_t)(k * 128), idesc, k > 0 ? 1u : 0u);
        umma_commit(&y_done[ys]);
        // an x pair is read by two y pairs, issued by the two warps: each commits it once, which releases the slot when
        // both have (x_free counts 2); a chunk's first and last x pairs have one reader, which commits twice
        umma_commit(&x_free[xs]);
        if (ql == 0) umma_commit(&x_free[xs]);
        umma_commit(&x_free[(xpbase + ql + 1) % NXP]);
        if (last_of_chunk) umma_commit(&x_free[(xpbase + ql + 1) % NXP]);
      }
      __syncwarp();
      TCJ_T(3, yq);
    };
    auto drain = [&](int yq) {
      const int st = yq % NSET;
      if (wid == 16) TCJ_T(4, yq); else if (wid == 17) TCJ_T(6, yq);
      mbar_wait(&y_done[yq % NYP], (unsigned)(yq / NYP) & 1u, 9);
      asm volatile("tcgen05.fence::after_thread_sync;");
      if (wid == 16) TCJ_T(5, yq); else if (wid == 17) TCJ_T(7, yq);
      if (!TCJ_DBG(64))
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        // the 20 used slots of both y rows at this shift: 16 + 4 columns each, one wait for the four loads
        uint32_t v[2][20];
#pragma unroll
        for (int yr = 0; yr < 2; ++yr) {
          const uint32_t col = lane_base + (uint32_t)(st * NCOL + s * 64 + yr * 32);
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                       : "=r"(v[yr][0]), "=r"(v[yr][1]), "=r"(v[yr][2]), "=r"(v[yr][3]), "=r"(v[yr][4]), "=r"(v[yr][5]),
                         "=r"(v[yr][6]), "=r"(v[yr][7]), "=r"(v[yr][8]), "=r"(v[yr][9]), "=r"(v[yr][10]), "=r"(v[yr][11]),
                         "=r"(v[yr][12]), "=r"(v[yr][13]), "=r"(v[yr][14]), "=r"(v[yr][15])
                       : "r"(col));
          asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                       : "=r"(v[yr][16]), "=r"(v[yr][17]), "=r"(v[yr][18]), "=r"(v[yr][19])
                       : "r"(col + 16));
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int yr = 0; yr < 2; ++yr)
#pragma unroll
          for (int j = 0; j < 10; ++j) tot[s][yr][j] += __uint_as_float(v[yr][j]) + __uint_as_float(v[yr][10 + j]);
      }
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(&set_free[st]);
    };

    int yq = 0, xpbase = 0;
    for (long long r = R0; r < R1;) {
      const Chunk c = chunk_at(r, R1, P.H);
      for (int ql = 0; ql < c.npy; ++ql, ++yq) {
        if (wid < 16) { if ((yq & 1) == (wid & 1)) issue(yq, ql, xpbase, ql == c.npy - 1); }
        else drain(yq);
      }
      xpbase += c.npy + 1;
      r += c.nr;
    }
    if (wid >= 16) {
    if (wid == 16) TCJ_T(0, 2);
    // lane = x slot (i: hi part, 10 + i: lo part).  dy = a - (y row), dx = 2 - shift.  The two y rows land in two staging
    // arrays in shared memory (the pair buffers are free now), added when the slot is written.
    float* stage = reinterpret_cast<float*>(smem);              // [2][9][10][10]
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int yr = 0; yr < 2; ++yr) {
        const int dy = a - yr;
#pragma unroll
        for (int j = 0; j < 10; ++j) {
          const float full = tot[s][yr][j] + __shfl_down_sync(0xffffffffu, tot[s][yr][j], 10);
          if (lane < 10 && dy >= 0 && dy < 3) stage[((yr * 9 + dy * 3 + (2 - s)) * 10 + lane) * 10 + j] = full;
        }
      }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    float* slot = P.partial + (size_t)blockIdx.x * (9 * P.K * P.K);
    const int tid = threadIdx.x - 16 * 32;
    for (int e = tid; e < 9 * P.K * P.K; e += 128) {
      const int d = e / (P.K * P.K), ij = e - d * P.K * P.K;
      const int i = ij / P.K, j = ij - i * P.K;
      const int o = (d * 10 + i) * 10 + j;
      slot[e] = (stage[o] + stage[900 + o]) * (1.f / (SCALE * SCALE));
    }
    if (wid == 16) TCJ_T(0, 3);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
#ifdef IIC_TCJ_DEBUG
  if (threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); g_tcj_cta[blockIdx.x][1] = t; }
#endif
  if (wid == 14) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

}  // namespace fwdtcj10

// One slot of [9][K][K] floats per CTA.
int local_joint_tcj10_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, int* flags, int* checked,
                          int from_logits, float inv_temp, cudaStream_t st) {
  using namespace fwdtcj10;
  const int B = m.B, K = m.K, H = m.H, W = m.W;
  *checked = 0;
  if (m.pad != PAD || K < 2 || K > 10 || W < 8 || W > MAXW) return -1;
  if (from_logits && K != 10) return -1;           // the fused forward takes exactly the shapes every fused backward takes
  const long long rows = (long long)B * H;
  if (rows < 8LL * max_ctas) return -1;            // small maps: the pipeline fill dominates, the FFMA2 kernel is faster
  Params P;
  P.x = m.x.p; P.x_sn = m.x.sn; P.x_sc = m.x.sc; P.x_sh = m.x.sh;
  P.y = m.y.p; P.y_sn = m.y.sn; P.y_sc = m.y.sc; P.y_sh = m.y.sh;
  P.B = B; P.H = H; P.W = W; P.K = K;
  P.partial = partial;
  P.flags = from_logits ? nullptr : flags;      // a softmax output needs no simplex assertion
  P.from_logits = from_logits;
  P.inv_temp = inv_temp;
  auto rows16 = [&](const View4& v) {
    return (reinterpret_cast<uintptr_t>(v.p) & 15) == 0 && v.sn % 4 == 0 && v.sc % 4 == 0 && v.sh % 4 == 0;
  };
  if (W % 4 != 0 || !rows16(m.x) || !rows16(m.y)) return -1;     // 16-byte loads
#ifdef IIC_TCJ_DEBUG
  P.dbg = 0;
#endif
  *checked = P.flags != nullptr;
  *slots = SlotInfo{SLOT_STD, max_ctas, (long long)9 * K * K, 0};
  IIC_CHECK_RC(ensure_dyn_smem((const void*)local_joint_tcj10_kernel, SMEM_BYTES));
  local_joint_tcj10_kernel<<<max_ctas, NTHREADS, SMEM_BYTES, st>>>(P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic
