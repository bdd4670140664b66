// Local IIC joint on the tensor cores for the reference's default cluster count (16 <= K <= 24) and both yaml
// paddings (1 and 3): "packed" variant of local_fwd_tc.cu.  Reference arithmetic: contrastyou/losses/iic_loss.py:120-123
//   J[dy][dx][i][j] = sum_{n,u,v} x[n,i,u+dy-p,v+dx-p] * y[n,j,u,v]          (x zero outside the map)
//
// An M = 128 tcgen05.mma costs the same whatever its N (measured, local_bwd_tc.cu), so both operand dimensions are
// packed with displacements instead of padding 20 channels to 128: for a 16-pixel segment of x row q
//   A rows  = (i, dx): the x row shifted by the T column displacements         (T*K rows: one or two 128-row tiles)
//   B rows  = (j, r):  the T y rows q + p - (T-1) + r, i.e. dy = T-1-r, that pair with x row q      (N = T * 24)
// and one accumulator D[(i,dx), (j,r)] collects ALL T*T displacements: 2 MMAs per 8 pixels and 128-row tile.
// Split product (one kind::tf32 MMA + one kind::f16 correction MMA on bf16 copies), 64-byte-swizzled K-major tiles,
// TMEM accumulation runs capped and drained into the CTA's slot: see local_fwd_tc.cu.
//
//   warp 0     TMA: x as an unswizzled [24 ch x 28 px] box (columns c0-4 .. c0+23), y as a 64-byte-swizzled
//              [24 ch x T rows x 16 px] box (rows outside the map are zero-filled: no contribution)
//   warps 4-15 transform: one thread per A row (its channel's staged row shifted by dx; fp32 + bf16 [xl|xh]) and one
//              per B row (copy + bf16 [yh|yl]); the drains: warps 4-7 own row tile 0, warps 8-11 row tile 1
//   warps 1, 3 MMA issuers (one row tile each)
// The slot holds D in a coalesced permuted order; reduce_packed_kernel adds the slots in fp64 in a fixed order and
// writes J in its [dy][dx][i][j] layout.
//
// From-logits form (FL): x and y hold the cluster head's logits and local_logit_stats_kernel (local_logits.cu) has
// written each pixel's (m, r); the TMA warp also stages the stats of the staged pixels, and the transform converts
// every logit to p = exp(l * inv_temp - m) * r before the fp32 / bf16 split.  Outside the map the TMA zero fill gives
// r = 0, so p = 0 there (the conv padding), not softmax(0) = 1/K; B rows of channels K..23 are zeroed explicitly.
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace fwdtcp {
using namespace tc;

constexpr int PXB = 16;                        // pixels per k-block (64-byte operand rows)
constexpr int XRW = 28, XRU = 24;              // staged / used x columns per k-block (see local_fwd_tc.cu)
constexpr int KPC = 24;                        // channels of the TMA boxes (K <= 24; channels >= K are zero-filled)
constexpr int ATILE = 128 * PXB * 4;           // 8192: one 128-row A tile, fp32 or bf16 part
constexpr int NRAW = 4;
constexpr int NTHREADS = 512;                  // 4 control warps + 12 transform warps (A rows: threads 0..T*K-1, B rows: 192..)
constexpr int SEG_KB_DEFAULT = 64;             // k-blocks per TMEM accumulation run (1024 pixels: uniform bias <= 2e-5,
                                               // see local_fwd_tc.cu; the drain is costlier here relative to the MMAs)
constexpr int SMEM_LIMIT = 225 * 1024;
// FL: the staged stats follow the y box in a raw slot: x stats [2][XRW] at fl_sx(T), y stats [2][T][PXB] 256 bytes on
__host__ __device__ constexpr int fl_sx(int T) { return 3072 + KPC * T * 64; }
constexpr int FL_SX_BYTES = 2 * XRW * 4;       // 224
__host__ __device__ constexpr int fl_sy_bytes(int T) { return 2 * T * PXB * 4; }


#ifdef IIC_TC_TRACE
__device__ long long g_trace[3][64][6];
#define TRACE(role, slot) do { if (blockIdx.x == 0 && k >= 64 && k < 128) g_trace[role][k - 64][slot] = clock64(); } while (0)
#else
#define TRACE(role, slot) do { } while (0)
#endif

struct Params {
  int B, H, W, K, segs_w;       // segs_w = W / 16
  int nmt;                      // 128-row A tiles: ceil(T*K / 128)
  int nb;                       // B rows = T * 24
  int op_bytes, raw_bytes;      // bytes of one operand-ring / raw-ring slot
  int nop;                      // operand-ring depth
  int seg_kb;
  int dbg;                      // bring-up switches (IIC_TC_DBG): 1 no loads, 2 no MMAs, 4 no transform
  float* partial;               // [gridDim.x][slot_floats]
};

// the from-logits form's extra arguments (unused by the probability instantiations)
struct FLParams {
  CUtensorMap sx, sy;           // the (2B, 2, H, W) stats tensor: x stats at n, y stats at B + n
  float inv_temp;
};

using iic::packed_slot_index;
__host__ __device__ inline size_t slot_index(int mt, int m, int c, int nb) { return packed_slot_index(mt, m, c, nb); }

template <int T, bool FL>
__global__ void __launch_bounds__(NTHREADS, 1)
local_joint_tcp_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy, const Params P,
                       const __grid_constant__ FLParams F) {
  constexpr int PAD = T / 2;
  constexpr int NOP_MAX = 8;
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW], op_full[NOP_MAX], op_empty[NOP_MAX], accum_bar, drained_bar;
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* raw_ring = smem + (size_t)P.nop * P.op_bytes;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb_total = P.B * P.H * P.segs_w;
  const int kb0 = (int)((long long)blockIdx.x * nkb_total / gridDim.x);
  const int kb1 = (int)((long long)(blockIdx.x + 1) * nkb_total / gridDim.x);
  const int nkb = kb1 - kb0;
  const int SEG_KB = P.seg_kb;
  const int nseg = (nkb + SEG_KB - 1) / SEG_KB;
  const int NOP = P.nop, NMT = P.nmt, NB = P.nb;
  const int xraw_bytes = KPC * XRW * 4;                   // 2688
  const int b_off = NMT * 2 * ATILE;                      // B tiles follow the A tiles in an operand slot
  const int b_part = NB * 64;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NRAW; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 12); }
    for (int s = 0; s < NOP; ++s) { mbar_init(&op_full[s], 12); mbar_init(&op_empty[s], 2); }
    mbar_init(&accum_bar, 2);
    mbar_init(&drained_bar, 12);
    mbar_fence_init();
  }
  if (wid == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem_base = tmem_base_s;

  if (wid == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      tma_prefetch_desc(&mapx);
      tma_prefetch_desc(&mapy);
      if constexpr (FL) { tma_prefetch_desc(&F.sx); tma_prefetch_desc(&F.sy); }
      // (image, row, segment) of the first k-block by division, then running counters: no divisions in the loops
      const int per_img = P.H * P.segs_w;
      int n = kb0 / per_img;
      int q = (kb0 - n * per_img) / P.segs_w;
      int sg = kb0 - n * per_img - q * P.segs_w;
      for (int k = 0; k < nkb; ++k) {
        const int s = k % NRAW;
        TRACE(0, 0);
        if (k >= NRAW) mbar_wait(&raw_empty[s], ((unsigned)(k / NRAW) & 1u) ^ 1u, 1);
        TRACE(0, 1);
        const int c0 = sg * PXB;
        const int qc = q, nc = n;
        if (++sg == P.segs_w) { sg = 0; if (++q == P.H) { q = 0; ++n; } }
        unsigned char* st = raw_ring + (size_t)s * P.raw_bytes;
        if (P.dbg & 1) { mbar_arrive(&raw_full[s]); continue; }
        if constexpr (FL) {
          mbar_arrive_expect_tx(&raw_full[s], xraw_bytes + KPC * T * 64 + FL_SX_BYTES + fl_sy_bytes(T));
          tma_load_4d(st + fl_sx(T), &F.sx, &raw_full[s], c0 - 4, qc, 0, nc);
          tma_load_4d(st + fl_sx(T) + 256, &F.sy, &raw_full[s], c0, qc + PAD - (T - 1), 0, P.B + nc);
        } else {
          mbar_arrive_expect_tx(&raw_full[s], xraw_bytes + KPC * T * 64);
        }
        tma_load_4d(st, &mapx, &raw_full[s], c0 - 4, qc, 0, nc);
        tma_load_4d(st + 3072, &mapy, &raw_full[s], c0, qc + PAD - (T - 1), 0, nc);
        TRACE(0, 2);
      }
    }
  } else if (wid == 1 || wid == 3) {
    // ===== MMA issuers: warp 1 owns row tile 0, warp 3 row tile 1 (independent accumulators).  tcgen05.mma issue
    // blocks at the tensor pipe's rate, so the second warp overlaps the first one's barrier waits and loop overhead;
    // both commit to the ring barriers =====
    const int my_mt = wid == 1 ? 0 : 1;
    const uint32_t nn = (uint32_t)NB;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((nn >> 3) << 17) | (8u << 24);
    const uint32_t idesc_bf16 = (1u << 4) | (1u << 7) | (1u << 10) | ((nn >> 3) << 17) | (8u << 24);
    int o = 0, kin = 0;
    unsigned oph = 0, seg = 0;
    for (int k = 0; k < nkb; ++k) {
      if (kin == 0 && k > 0) {
        mbar_wait(&drained_bar, (seg - 1) & 1u, 6);
        asm volatile("tcgen05.fence::after_thread_sync;");
      }
      if (lane == 0) TRACE(1, 0);
      mbar_wait(&op_full[o], oph, 5);
      asm volatile("tcgen05.fence::after_thread_sync;");
      if (lane == 0) {
        TRACE(1, 1);
        const uint64_t base = make_desc_sw64(smem_u32(smem + (size_t)o * P.op_bytes));
        const uint64_t bb = base + (uint64_t)(b_off / 16);
        for (int mt = my_mt; mt < ((P.dbg & 2) ? 0 : NMT); mt += 2) {
          const uint64_t ab = base + (uint64_t)(mt * 2 * (ATILE / 16));
          const uint32_t d_tmem = tmem_base + (uint32_t)(mt * NB);
#pragma unroll
          for (int ks = 0; ks < PXB / 8; ++ks) {
            umma_bf16(d_tmem, ab + (uint64_t)(ATILE / 16 + ks * 2), bb + (uint64_t)(b_part / 16 + ks * 2), idesc_bf16,
                      (kin > 0 || ks > 0) ? 1u : 0u);                                     // xl*yh + xh*yl
            umma_tf32(d_tmem, ab + (uint64_t)(ks * 2), bb + (uint64_t)(ks * 2), idesc, 1u);
          }
        }
        if (P.dbg & 8) mbar_arrive(&op_empty[o]); else umma_commit(&op_empty[o]);      // dbg 8: plain arrive (timing experiment)
        if (kin == SEG_KB - 1 || k == nkb - 1) umma_commit(&accum_bar);
        TRACE(1, 2);
      }
      __syncwarp();
      if (++o == NOP) { o = 0; oph ^= 1u; }
      if (++kin == SEG_KB) { kin = 0; ++seg; }
    }
  } else if (wid >= 4) {
    // ===== transform warps, and the drains =====
    const int tid = threadIdx.x - 128;                         // 0 .. 383
    const int grp = (wid - 4) >> 2;                            // drains: warps 4-7 own row tile 0, warps 8-11 row tile 1
    const int q4 = wid & 3;
    const int m = q4 * 32 + lane;                              // accumulator row of this thread in the drains
    const int slot_floats = NMT * 128 * NB;
    float* slot = P.partial + (size_t)blockIdx.x * slot_floats;
    const int nrows_a = T * P.K;
    int o = 0, kin = 0, seg = 0;
    unsigned oph = 0;
    for (int k = 0; k < nkb; ++k) {
      const int s = k % NRAW;
      if (threadIdx.x == 128) TRACE(2, 0);
      mbar_wait(&raw_full[s], (unsigned)(k / NRAW) & 1u, 3);
      if (threadIdx.x == 128) TRACE(2, 1);
      if (k >= NOP) mbar_wait(&op_empty[o], oph ^ 1u, 2);
      if (threadIdx.x == 128) TRACE(2, 2);
      const unsigned char* raw = raw_ring + (size_t)s * P.raw_bytes;
      unsigned char* op = smem + (size_t)o * P.op_bytes;
      if (tid < nrows_a && !(P.dbg & 4)) {
        // A row tid = (i, dx), dx fastest (a warp's lanes read neighbouring words of a few staged rows: <= 2-way bank
        // conflicts): operand pixel p of the k-block is x column c0 + p + dx - PAD = staged column p + dx + 4 - PAD
        const int i = tid / T, dx = tid - i * T;
        const int mt = tid >> 7, r = tid & 127;
        const int sw = (r >> 1) & 3;
        const float* xs = reinterpret_cast<const float*>(raw + i * (XRW * 4)) + (dx + 4 - PAD);
        float xv[PXB];
#pragma unroll
        for (int p = 0; p < PXB; ++p) xv[p] = xs[p];
        if constexpr (FL) {
          const float* sm = reinterpret_cast<const float*>(raw + fl_sx(T)) + (dx + 4 - PAD);      // m, then r at + XRW
#pragma unroll
          for (int p = 0; p < PXB; ++p) xv[p] = __expf(__fmul_rn(xv[p], F.inv_temp) - sm[p]) * sm[XRW + p];
        }
        unsigned char* a32 = op + (mt * 2) * ATILE + r * 64;
        unsigned char* a16 = a32 + ATILE;
#pragma unroll
        for (int c = 0; c < 4; ++c)
          *reinterpret_cast<float4*>(a32 + ((c ^ sw) << 4)) = make_float4(xv[4 * c], xv[4 * c + 1], xv[4 * c + 2], xv[4 * c + 3]);
        *reinterpret_cast<uint4*>(a16 + ((0 ^ sw) << 4)) = pack8<true>(xv);
        *reinterpret_cast<uint4*>(a16 + ((1 ^ sw) << 4)) = pack8<false>(xv);
        *reinterpret_cast<uint4*>(a16 + ((2 ^ sw) << 4)) = pack8<true>(xv + 8);
        *reinterpret_cast<uint4*>(a16 + ((3 ^ sw) << 4)) = pack8<false>(xv + 8);
      }
      if (tid >= 192 && tid - 192 < NB && !(P.dbg & 4)) {
        // B row n = (channel, y row) exactly as the swizzled TMA box laid it out: copy + bf16 [yh | yl]
        const int nrow = tid - 192;
        const int sw = (nrow >> 1) & 3;
        float yv[PXB];
        unsigned char* b32 = op + b_off + nrow * 64;
        unsigned char* b16 = b32 + b_part;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int off = (c ^ sw) << 4;
          float4 t = *reinterpret_cast<const float4*>(raw + 3072 + nrow * 64 + off);
          if constexpr (FL) {
            // box row nrow = (channel, y row r); channels >= K were zero-filled logits: their p must be 0, not exp(-m) r
            const int r = nrow % T;
            const float* sm = reinterpret_cast<const float*>(raw + fl_sx(T) + 256) + r * PXB + 4 * c;   // m; r at + T*PXB
            const bool live = nrow < T * P.K;
            t.x = live ? __expf(__fmul_rn(t.x, F.inv_temp) - sm[0]) * sm[T * PXB + 0] : 0.f;
            t.y = live ? __expf(__fmul_rn(t.y, F.inv_temp) - sm[1]) * sm[T * PXB + 1] : 0.f;
            t.z = live ? __expf(__fmul_rn(t.z, F.inv_temp) - sm[2]) * sm[T * PXB + 2] : 0.f;
            t.w = live ? __expf(__fmul_rn(t.w, F.inv_temp) - sm[3]) * sm[T * PXB + 3] : 0.f;
          }
          *reinterpret_cast<float4*>(b32 + off) = t;
          yv[4 * c] = t.x; yv[4 * c + 1] = t.y; yv[4 * c + 2] = t.z; yv[4 * c + 3] = t.w;
        }
        *reinterpret_cast<uint4*>(b16 + ((0 ^ sw) << 4)) = pack8<false>(yv);
        *reinterpret_cast<uint4*>(b16 + ((1 ^ sw) << 4)) = pack8<true>(yv);
        *reinterpret_cast<uint4*>(b16 + ((2 ^ sw) << 4)) = pack8<false>(yv + 8);
        *reinterpret_cast<uint4*>(b16 + ((3 ^ sw) << 4)) = pack8<true>(yv + 8);
      }
      if (threadIdx.x == 128) TRACE(2, 3);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&op_full[o]);
        mbar_arrive(&raw_empty[s]);
      }
      if (threadIdx.x == 128) TRACE(2, 4);
      const bool run_end = kin == SEG_KB - 1 || k == nkb - 1;
      if (run_end) {
        // ---- drain this run's accumulators into the slot (first run stores, later runs add) ----
        mbar_wait(&accum_bar, (unsigned)seg & 1u, 4);
        asm volatile("tcgen05.fence::after_thread_sync;");
        if (grp < NMT) {
          const int nc8 = NB / 8;
          float4* sl4 = reinterpret_cast<float4*>(slot) + ((size_t)grp * nc8 * 2) * 128 + m;
          float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0;
          if (seg > 0) { g0 = sl4[0]; g1 = sl4[128]; }
          for (int c8 = 0; c8 < nc8; ++c8) {
            uint32_t a[8];
            const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(grp * NB + c8 * 8);
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7])
                         : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float4* dst = sl4 + (size_t)c8 * 256;
            float4 o0 = make_float4(__uint_as_float(a[0]) + g0.x, __uint_as_float(a[1]) + g0.y, __uint_as_float(a[2]) + g0.z,
                                    __uint_as_float(a[3]) + g0.w);
            float4 o1 = make_float4(__uint_as_float(a[4]) + g1.x, __uint_as_float(a[5]) + g1.y, __uint_as_float(a[6]) + g1.z,
                                    __uint_as_float(a[7]) + g1.w);
            if (seg > 0 && c8 + 1 < nc8) { g0 = dst[256]; g1 = dst[256 + 128]; }     // next chunk's slot values
            dst[0] = o0;
            dst[128] = o1;
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;");
        __syncwarp();
        if (lane == 0 && seg + 1 < nseg) mbar_arrive(&drained_bar);
      }
      if (++o == NOP) { o = 0; oph ^= 1u; }
      if (++kin == SEG_KB) { kin = 0; ++seg; }
    }
    if (nkb == 0)
      for (int e = tid; e < slot_floats; e += 384) slot[e] = 0.f;
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

// J[dy][dx][i][j] = sum over CTAs of their slot element in fp64, in a fixed order: a block is 32 slot groups x 32
// consecutive outputs; group g adds slots g, g+32, ... in order, then the 32 group sums are added in order.
__global__ void __launch_bounds__(1024)
reduce_packed_kernel(const float* __restrict__ partial, int ncta, int slot_floats, int T, int K, int nb, double* __restrict__ J) {
  __shared__ double sm[32][33];
  const int le = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int e = blockIdx.x * 32 + le;
  const int E = T * T * K * K;
  double s = 0.0;
  if (e < E) {
    const int j = e % K, i = (e / K) % K, dx = (e / (K * K)) % T, dy = e / (K * K * T);
    const int row = i * T + dx, col = j * T + (T - 1 - dy);
    const float* src = partial + slot_index(row >> 7, row & 127, col, nb);
    for (int c = g; c < ncta; c += 32) s += (double)__ldg(src + (size_t)c * slot_floats);
  }
  sm[g][le] = s;
  __syncthreads();
  if (g == 0 && e < E) {
    double t = 0.0;
#pragma unroll
    for (int q = 0; q < 32; ++q) t += sm[q][le];
    J[e] = t;
  }
}

template <int T, bool FL>
static int launch(const CUtensorMap& mx, const CUtensorMap& my, const Params& P, const FLParams& F, int grid, size_t smem,
                  cudaStream_t st) {
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_joint_tcp_kernel<T, FL>), (int)(SMEM_LIMIT)));
  local_joint_tcp_kernel<T, FL><<<grid, NTHREADS, smem, st>>>(mx, my, P, F);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace fwdtcp

size_t local_joint_tcp_slot_floats(int K, int pad) {
  if (K < 16 || K > 24 || (pad != 1 && pad != 3)) return 0;
  const int T = 2 * pad + 1;
  return (size_t)((T * K + 127) / 128) * 128 * (T * fwdtcp::KPC);
}

// stats == nullptr: probabilities; else logits with the per-pixel (m, r) of local_logit_stats_kernel in `stats`
static int tcp_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, size_t partial_floats,
                   SlotInfo* slots, cudaStream_t st) {
  using namespace fwdtcp;
  const int B = m.B, K = m.K, H = m.H, W = m.W;
  const size_t slot_floats = local_joint_tcp_slot_floats(K, m.pad);
  if (slot_floats == 0 || W % PXB != 0) return -1;
  const int T = 2 * m.pad + 1;
  const int nmt = (T * K + 127) / 128, nb = T * KPC;
  const bool fl = stats != nullptr;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, XRW, 1, KPC)) return -1;
  if (!make_map_4d(&my, m.y, m, PXB, T, KPC, CU_TENSOR_MAP_SWIZZLE_64B)) return -1;
  FLParams F{};
  F.inv_temp = inv_temp;
  if (fl) {
    const long long hw = (long long)H * W;
    if (!make_map_4d(&F.sx, stats, 2 * B, 2, H, W, 2 * hw, hw, W, XRW, 1, 2)) return -1;
    if (!make_map_4d(&F.sy, stats, 2 * B, 2, H, W, 2 * hw, hw, W, PXB, T, 2)) return -1;
  }
  const long long nkb = (long long)B * H * (W / PXB);
  long long grid = m.sms;
  if ((long long)(partial_floats / slot_floats) < grid) grid = (long long)(partial_floats / slot_floats);
  if (grid > nkb) grid = nkb;
  if (grid < 1) return -1;
  const int op_bytes = (nmt * 2 * ATILE + 2 * nb * 64 + 1023) & ~1023;
  const int raw_used = fl ? fl_sx(T) + 256 + fl_sy_bytes(T) : 3072 + KPC * T * 64;
  const int raw_bytes = (raw_used + 1023) & ~1023;
  int nop = (SMEM_LIMIT - 1024 - NRAW * raw_bytes) / op_bytes;
  if (nop > 8) nop = 8;
  if (tc::bringup_env("IIC_TC_NOP", nop) < nop) nop = tc::bringup_env("IIC_TC_NOP", nop);   // experiments (bring-up builds only)
  if (nop < 2) return -1;
  const size_t smem = (size_t)nop * op_bytes + (size_t)NRAW * raw_bytes + 1024;
  Params P{B, H, W, K, W / PXB, nmt, nb, op_bytes, raw_bytes, nop,
           tc::bringup_env("IIC_TC_SEG", SEG_KB_DEFAULT),
           tc::bringup_env("IIC_TC_DBG", 0), partial};
  int rc;
  if (fl) rc = T == 3 ? launch<3, true>(mx, my, P, F, (int)grid, smem, st) : launch<7, true>(mx, my, P, F, (int)grid, smem, st);
  else rc = T == 3 ? launch<3, false>(mx, my, P, F, (int)grid, smem, st) : launch<7, false>(mx, my, P, F, (int)grid, smem, st);
  if (rc) return rc;
  *slots = SlotInfo{SLOT_PACKED, (int)grid, (long long)slot_floats, nb};
  return 0;
}

int local_joint_tcp_try(const LocalMaps& m, float* partial, size_t partial_floats, SlotInfo* slots, cudaStream_t st) {
  return tcp_try(m, nullptr, 1.f, partial, partial_floats, slots, st);
}

int local_joint_tcp_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, size_t partial_floats,
                           SlotInfo* slots, cudaStream_t st) {
  return tcp_try(m, stats, inv_temp, partial, partial_floats, slots, st);
}

}  // namespace iic
