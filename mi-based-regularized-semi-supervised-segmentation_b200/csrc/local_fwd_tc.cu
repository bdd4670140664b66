// Local IIC joint on the 5th-generation tensor cores (tcgen05 / UMMA) for wide cluster heads: K = 128 channels,
// 3 x 3 window (padding 1) -- BASELINE config 5, "tensor cores only when K is large enough to be a real dense
// contraction" (north_star).  Reference arithmetic: contrastyou/losses/iic_loss.py:120-123
//   J[dy][dx][i][j] = sum_{n,u,v} x[n,i,u+dy-1,v+dx-1] * y[n,j,u,v]          (x zero outside the map)
// = nine 128 x 128 x Npix contractions.  fp32-level accuracy from a split product: kind::tf32 reads the top 19 bits
// of an fp32 word, so with xh = trunc19(x) and xl = x - xh (exact in fp32)  x*y = xh*yh + (xl*yh + xh*yl) + xl*yl.
// The main term is one tcgen05.mma.kind::tf32 on the raw fp32 tiles (K = 8 pixels); the two correction terms are
// 2^-11 of it and only need ~8 bits, so they share ONE tcgen05.mma.kind::f16 on bf16 copies with K = 16 =
// [xl(8 px) | xh(8 px)] x [yh(8 px) | yl(8 px)]; xl*yl (2^-22) is dropped.  Two MMAs per 8 pixels and displacement
// instead of the three of a plain 3xTF32 scheme; relative error ~2^-20 per product.
//
// One CTA = one displacement row dy (blockIdx.y) and a contiguous share of the 16-pixel row segments ("k-blocks",
// the reduction dimension of the MMA).  Per k-block:
//   warp 0     TMA producer: x rows shifted by dy as an unswizzled [128 ch x 28 px] box (columns c0-4 .. c0+23; the
//              hardware zero fill is the conv padding) and y as a 64-byte-swizzled [128 ch x 16 px] box -> raw ring.
//              (A box cannot start at a column that is not a multiple of 4 floats -- the copy faults -- so
//              the +-1 column shifts are made by the transform warps, not by TMA coordinates.)
//   warps 4-7  transform: thread = channel row; writes the eight K-major SWIZZLE_64B operand tiles of the k-block
//              (x fp32 + bf16 correction tile at the three column shifts, y fp32 + bf16) into the operand ring and
//              fences them for the async proxy.
//   warp 1     one elected lane issues 3 (dx) x 2 (8-pixel slices) x 2 MMAs, M = N = 128, into three 128-column
//              TMEM accumulators; tcgen05.commit frees the operand slot.
// Epilogue: warps 4-7 read the accumulators with tcgen05.ld (lane = x channel i, column = y channel j) and write
// the CTA's partial-joint slot in the permuted order tc_slot_index() describes (coalesced 512-byte warp accesses);
// reduce_partials_kernel (local_fwd.cu) adds the slots in fp64 in a fixed order and undoes the permutation.
// To bound the fp32 accumulation run in TMEM the k-blocks are processed in segments: after each segment the
// accumulators are drained into the slot (first segment stores, later ones add).
//
// From-logits form (FL, the cluster head's SoftmaxWithT fused): x and y hold logits and local_logit_stats_kernel
// (local_logits.cu) has written each pixel's (m, r).  The TMA warp also stages the stats of the k-block's 28 x columns
// and 16 y pixels behind the y box, and the transform converts every logit it uses to p = exp(l * inv_temp - m) * r
// (logit_p, common.cuh) before the fp32 / bf16 split.  Outside the map the TMA zero fill gives r = 0, so p = 0 there
// (the conv padding), not softmax(0) = 1/K.
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace fwdtc {
using namespace tc;

constexpr int KC = 128;                        // channels = UMMA M = UMMA N
constexpr int PXB = 16;                        // pixels per k-block (64-byte operand rows)
constexpr int XRW = 28;                        // staged x columns per k-block: c0-4 .. c0+23 (112-byte rows: conflict-free LDS.128;
                                               // columns c0-1 .. c0+16 are used)
constexpr int XRU = 24;                        // columns read by the transform
constexpr int TILE_BYTES = KC * PXB * 4;       // 8192
constexpr int XRAW_BYTES = KC * XRW * 4;       // 14336
constexpr int RAW_BYTES = XRAW_BYTES + TILE_BYTES;   // 22528
constexpr int NRAW = 4;
constexpr int OP_TILES = 8;                    // x fp32 (dx 0..2), y fp32, x bf16 [xl|xh] (dx 0..2), y bf16 [yh|yl]
constexpr int OP_BYTES = OP_TILES * TILE_BYTES;      // 65536
constexpr int NOP = 2;
constexpr int SMEM_BYTES = NRAW * RAW_BYTES + NOP * OP_BYTES + 1024;   // + alignment slack
constexpr int NTHREADS = 384;                   // 4 control warps + two transform / drain groups of 4 warps
// k-blocks per TMEM accumulation run.  The tensor core adds into the fp32 accumulator with truncation, a relative
// bias of about -1.4e-7 per 8-pixel slice that is (measured) uniform over the entries of J to 0.4 % of itself -- the
// normalisation of iic_loss.py:129 removes a uniform factor.  32 k-blocks = 512 pixels bound it at 1e-5.
constexpr int SEG_KB_DEFAULT = 32;
// FL: a raw slot also holds the staged stats after RAW_BYTES: x [2][XRW] (m, r), then y [2][PXB] 256 bytes on (a TMA
// destination must be 128-byte aligned); slots stay 1024-byte aligned (the y box is swizzled)
constexpr int FL_SX = RAW_BYTES, FL_SY = RAW_BYTES + 256;
constexpr int FL_STATS_BYTES = 2 * XRW * 4 + 2 * PXB * 4;         // 352 bytes copied
constexpr int FL_RAW_STRIDE = (FL_SY + 2 * PXB * 4 + 1023) & ~1023;
constexpr int FL_SMEM_BYTES = NRAW * FL_RAW_STRIDE + NOP * OP_BYTES + 1024;
static_assert(FL_SX % 128 == 0 && FL_SY % 128 == 0 && FL_RAW_STRIDE % 1024 == 0, "TMA destinations must stay aligned");


struct Params {
  int B, H, W, segs_w;          // segs_w = W / 16
  float* partial;               // [gridDim.x][9][128][128]
  int seg_kb;                   // k-blocks per accumulation segment
  int dbg;                      // bring-up switches (IIC_TC_DBG): 1 no loads, 4 no transform
};

// the from-logits form's extra arguments (unused by the probability instantiation)
struct FLParams {
  CUtensorMap sx, sy;           // the (2B, 2, H, W) stats tensor: x stats at n, y stats at B + n
  float inv_temp;
};

// bytes between raw-ring slots (a namespace-scope function rather than a constexpr local, which can change the
// probability instantiation's register assignment)
template <bool FL>
__device__ constexpr int raw_stride() { return FL ? FL_RAW_STRIDE : RAW_BYTES; }

template <bool FL>
__global__ void __launch_bounds__(NTHREADS, 1)
local_joint_tc_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy, const Params P,
                      const __grid_constant__ FLParams F) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[NRAW], raw_empty[NRAW], op_full[NOP], op_empty[NOP], accum_bar, drained_bar;
  __shared__ uint32_t tmem_base_s;
  // 1024-byte alignment by offset (keeps the shared address space visible to the compiler: LDS/STS, not generic LD/ST)
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* raw_ring = smem + NOP * OP_BYTES;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int dy = blockIdx.y;
  const int nkb_total = P.B * P.H * P.segs_w;
  const int kb0 = (int)((long long)blockIdx.x * nkb_total / gridDim.x);
  const int kb1 = (int)((long long)(blockIdx.x + 1) * nkb_total / gridDim.x);
  const int nkb = kb1 - kb0;
  const int SEG_KB = P.seg_kb;
  const int nseg = (nkb + SEG_KB - 1) / SEG_KB;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NRAW; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 8); }
    for (int s = 0; s < NOP; ++s) { mbar_init(&op_full[s], 8); mbar_init(&op_empty[s], 1); }
    mbar_init(&accum_bar, 1);
    mbar_init(&drained_bar, 8);
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
      // (image, row, segment) of the first k-block by division, then running counters: a division by a runtime value
      // costs this single-lane loop ~100 clk per k-block
      const int per_img = P.H * P.segs_w;
      int n = kb0 / per_img;
      int u = (kb0 - n * per_img) / P.segs_w;
      int sg = kb0 - n * per_img - u * P.segs_w;
      for (int k = 0; k < nkb; ++k) {
        const int s = k % NRAW;
        if (k >= NRAW) mbar_wait(&raw_empty[s], ((unsigned)(k / NRAW) & 1u) ^ 1u, 1);
        const int c0 = sg * PXB, uc = u, nc = n;
        if (++sg == P.segs_w) { sg = 0; if (++u == P.H) { u = 0; ++n; } }
        unsigned char* st = raw_ring + (size_t)s * raw_stride<FL>();
        if (P.dbg & 1) { mbar_arrive(&raw_full[s]); continue; }
        if constexpr (FL) {
          mbar_arrive_expect_tx(&raw_full[s], RAW_BYTES + FL_STATS_BYTES);
          tma_load_4d(st + FL_SX, &F.sx, &raw_full[s], c0 - 4, uc + dy - 1, 0, nc);
          tma_load_4d(st + FL_SY, &F.sy, &raw_full[s], c0, uc, 0, P.B + nc);
        } else {
          mbar_arrive_expect_tx(&raw_full[s], RAW_BYTES);
        }
        tma_load_4d(st, &mapx, &raw_full[s], c0 - 4, uc + dy - 1, 0, nc);
        tma_load_4d(st + XRAW_BYTES, &mapy, &raw_full[s], c0, uc, 0, nc);
      }
    }
  } else if (wid == 1) {
    // ===== MMA issuer =====
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(KC >> 3) << 17) | ((uint32_t)(KC >> 4) << 24);
    const uint32_t idesc_bf16 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(KC >> 3) << 17) | ((uint32_t)(KC >> 4) << 24);
    int kin = 0;                                // position inside the accumulation segment (running: no divisions)
    unsigned seg = 0;
    for (int k = 0; k < nkb; ++k) {
      const int o = k % NOP;
      if (kin == 0 && k > 0) {                  // the epilogue warps must have drained the previous segment
        mbar_wait(&drained_bar, (seg - 1) & 1u, 6);
        asm volatile("tcgen05.fence::after_thread_sync;");
      }
      mbar_wait(&op_full[o], (unsigned)(k / NOP) & 1u, 5);
      asm volatile("tcgen05.fence::after_thread_sync;");
      if (lane == 0) {
        // one base descriptor per operand slot; every tile / slice is a compile-time offset in 16-byte units
        const uint64_t base = make_desc_sw64(smem_u32(smem + (size_t)o * OP_BYTES));
        constexpr int TL = TILE_BYTES / 16;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const uint32_t d_tmem = tmem_base + dx * KC;
#pragma unroll
          for (int ks = 0; ks < PXB / 8; ++ks) {
            umma_bf16(d_tmem, base + (uint64_t)((4 + dx) * TL + ks * 2), base + (uint64_t)(7 * TL + ks * 2), idesc_bf16,
                      (kin > 0 || ks > 0) ? 1u : 0u);                                              // xl*yh + xh*yl
            umma_tf32(d_tmem, base + (uint64_t)(dx * TL + ks * 2), base + (uint64_t)(3 * TL + ks * 2), idesc, 1u);
          }
        }
        umma_commit(&op_empty[o]);                              // frees the operand slot when these MMAs have read it
        if (kin == SEG_KB - 1 || k == nkb - 1) umma_commit(&accum_bar);
      }
      __syncwarp();
      if (++kin == SEG_KB) { kin = 0; ++seg; }
    }
  } else if (wid >= 4) {
    // ===== transform warps, and the epilogue: two groups of four warps, a thread of each per channel row.
    // group 0 writes the x tiles of column shifts 0 and 1 and drains accumulator chunks 0-5, group 1 the x tiles of
    // shift 2, the y tiles and chunks 6-11 =====
    const int grp = wid >= 8 ? 1 : 0;
    const int r = (threadIdx.x - 128) & 127;                    // channel row
    const int sw = (r >> 1) & 3;                                // SWIZZLE_64B: 16-byte chunk index ^= address bits 7..8
    const int q4 = wid & 3;                                     // this warp reads TMEM lanes 32*q4 .. 32*q4+31
    float* slot = P.partial + (size_t)blockIdx.x * (9 * KC * KC);
    int kin = 0, seg = 0;                                       // running segment counters (no divisions in the loop)
    for (int k = 0; k < nkb; ++k) {
      const int s = k % NRAW, o = k % NOP;
      mbar_wait(&raw_full[s], (unsigned)(k / NRAW) & 1u, 3);
      if (k >= NOP) mbar_wait(&op_empty[o], ((unsigned)(k / NOP) & 1u) ^ 1u, 2);
      const unsigned char* raw = raw_ring + (size_t)s * raw_stride<FL>();
      unsigned char* op = smem + (size_t)o * OP_BYTES;
      if (!(P.dbg & 4)) {
        float v[XRU];
        const float4* xr = reinterpret_cast<const float4*>(raw + r * (XRW * 4));
#pragma unroll
        for (int q = 0; q < XRU / 4; ++q) {
          const float4 t = xr[q];
          v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
        if constexpr (FL) {
          // staged columns 3 .. 19 (group 0: shifts 0, 1) or 5 .. 20 (group 1: shift 2) are read; m [XRW], then r [XRW]
          const float* sm = reinterpret_cast<const float*>(raw + FL_SX);
#pragma unroll
          for (int q = 3; q <= 20; ++q)
            if (grp == 1 ? q >= 5 : q <= 19) v[q] = logit_p(v[q], F.inv_temp, sm[q], sm[XRW + q]);
        }
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          if ((dx == 2) != (grp == 1)) continue;
          // operand pixel p of the k-block is x column c0 + p + dx - 1 = staged column p + dx + 3
          const float* xv = v + dx + 3;
#pragma unroll
          for (int c = 0; c < 4; ++c)
            *reinterpret_cast<float4*>(op + dx * TILE_BYTES + r * 64 + ((c ^ sw) << 4)) =
                make_float4(xv[4 * c], xv[4 * c + 1], xv[4 * c + 2], xv[4 * c + 3]);
          // bf16 correction tile: per 8-pixel slice [xl | xh]
          unsigned char* cr = op + (4 + dx) * TILE_BYTES + r * 64;
          *reinterpret_cast<uint4*>(cr + ((0 ^ sw) << 4)) = pack8<true>(xv);
          *reinterpret_cast<uint4*>(cr + ((1 ^ sw) << 4)) = pack8<false>(xv);
          *reinterpret_cast<uint4*>(cr + ((2 ^ sw) << 4)) = pack8<true>(xv + 8);
          *reinterpret_cast<uint4*>(cr + ((3 ^ sw) << 4)) = pack8<false>(xv + 8);
        }
        if (grp == 1) {
        // y arrives swizzled (physical chunk c ^ sw holds pixels 4c .. 4c+3); walked in swizzle order: no bank conflicts
        float yv[PXB];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int off = r * 64 + ((c ^ sw) << 4);
          float4 t = *reinterpret_cast<const float4*>(raw + XRAW_BYTES + off);
          if constexpr (FL) {
            const float* sm = reinterpret_cast<const float*>(raw + FL_SY) + 4 * c;            // m [PXB], then r [PXB]
            t.x = logit_p(t.x, F.inv_temp, sm[0], sm[PXB + 0]);
            t.y = logit_p(t.y, F.inv_temp, sm[1], sm[PXB + 1]);
            t.z = logit_p(t.z, F.inv_temp, sm[2], sm[PXB + 2]);
            t.w = logit_p(t.w, F.inv_temp, sm[3], sm[PXB + 3]);
          }
          *reinterpret_cast<float4*>(op + 3 * TILE_BYTES + off) = t;
          yv[4 * c] = t.x; yv[4 * c + 1] = t.y; yv[4 * c + 2] = t.z; yv[4 * c + 3] = t.w;
        }
        unsigned char* cr = op + 7 * TILE_BYTES + r * 64;          // per 8-pixel slice [yh | yl]
        *reinterpret_cast<uint4*>(cr + ((0 ^ sw) << 4)) = pack8<false>(yv);
        *reinterpret_cast<uint4*>(cr + ((1 ^ sw) << 4)) = pack8<true>(yv);
        *reinterpret_cast<uint4*>(cr + ((2 ^ sw) << 4)) = pack8<false>(yv + 8);
        *reinterpret_cast<uint4*>(cr + ((3 ^ sw) << 4)) = pack8<true>(yv + 8);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&op_full[o]);
        mbar_arrive(&raw_empty[s]);
      }
      if (kin == SEG_KB - 1 || k == nkb - 1) {
        // ---- drain the accumulators of this segment into the slot ----
        mbar_wait(&accum_bar, (unsigned)seg & 1u, 4);
        asm volatile("tcgen05.fence::after_thread_sync;");
        // 12 chunks of 32 columns, 6 per group; the slot values a later segment adds to are prefetched two chunks ahead
        float4 g[2][8];
        // slot layout [dy*3+dx][32-column chunk][float4 j of the chunk][row][4]: every warp access is 512 contiguous bytes
        auto chunk_ptr = [&](int c) { return reinterpret_cast<float4*>(slot) + ((size_t)((dy * 3 + (c >> 2)) * 4 + (c & 3)) * 8) * KC + r; };
        if (seg > 0) {
#pragma unroll
          for (int p = 0; p < 2; ++p) {
            const float4* src = chunk_ptr(grp * 6 + p);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[p][j] = src[j * KC];
          }
        }
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) {
          const int c = grp * 6 + cc;
          uint32_t a[32];
          const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (c >> 2) * KC + (c & 3) * 32;
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
              "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
              "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
              : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]),
                "=r"(a[8]), "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),
                "=r"(a[16]), "=r"(a[17]), "=r"(a[18]), "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]),
                "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]), "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31])
              : "r"(taddr));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          float4* dst = chunk_ptr(c);
          float4 out[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            out[j] = make_float4(__uint_as_float(a[4 * j]), __uint_as_float(a[4 * j + 1]), __uint_as_float(a[4 * j + 2]),
                                 __uint_as_float(a[4 * j + 3]));
            if (seg > 0) {
              out[j].x += g[cc & 1][j].x; out[j].y += g[cc & 1][j].y; out[j].z += g[cc & 1][j].z; out[j].w += g[cc & 1][j].w;
            }
          }
          if (seg > 0 && cc + 2 < 6) {
            const float4* src = chunk_ptr(c + 2);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[cc & 1][j] = src[j * KC];
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) dst[j * KC] = out[j];
        }
        asm volatile("tcgen05.fence::before_thread_sync;");
        __syncwarp();
        if (lane == 0 && seg + 1 < nseg) mbar_arrive(&drained_bar);
      }
      if (++kin == SEG_KB) { kin = 0; ++seg; }
    }
    if (nkb == 0) {
      float4* dst = reinterpret_cast<float4*>(slot + (size_t)dy * 3 * KC * KC);
      for (int e = r; e < 3 * KC * KC / 4; e += 128) dst[e] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

}  // namespace fwdtc

// stats == nullptr: probabilities; else logits with the per-pixel (m, r) of local_logit_stats_kernel in `stats`
static int tc_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, int max_ctas, SlotInfo* slots,
                  cudaStream_t st) {
  using namespace fwdtc;
  const int B = m.B, H = m.H, W = m.W;
  if (m.K != KC || m.pad != 1 || W % PXB != 0 || max_ctas < 1) return -1;
  const bool fl = stats != nullptr;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, XRW, 1, KC)) return -1;
  if (!make_map_4d(&my, m.y, m, PXB, 1, KC, CU_TENSOR_MAP_SWIZZLE_64B)) return -1;
  FLParams F{};
  F.inv_temp = inv_temp;
  if (fl) {
    const long long hw = (long long)H * W;
    if (!make_map_4d(&F.sx, stats, 2 * B, 2, H, W, 2 * hw, hw, W, XRW, 1, 2)) return -1;
    if (!make_map_4d(&F.sy, stats, 2 * B, 2, H, W, 2 * hw, hw, W, PXB, 1, 2)) return -1;
  }
  const long long nkb = (long long)B * H * (W / PXB);
  int gx = m.sms / 3;                                 // three displacement rows per share of the pixels
  if (gx > max_ctas) gx = max_ctas;
  if (gx > nkb) gx = (int)nkb;
  if (gx < 1) gx = 1;
  Params P{B, H, W, W / PXB, partial, tc::bringup_env("IIC_TC_SEG", SEG_KB_DEFAULT),
           tc::bringup_env("IIC_TC_DBG", 0)};
  if (fl) {
    IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_joint_tc_kernel<true>), (int)(FL_SMEM_BYTES)));
    local_joint_tc_kernel<true><<<dim3(gx, 3), NTHREADS, FL_SMEM_BYTES, st>>>(mx, my, P, F);
  } else {
    IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_joint_tc_kernel<false>), (int)(SMEM_BYTES)));
    local_joint_tc_kernel<false><<<dim3(gx, 3), NTHREADS, SMEM_BYTES, st>>>(mx, my, P, F);
  }
  IIC_CHECK_CUDA(cudaGetLastError());
  *slots = SlotInfo{SLOT_TC128, gx, (long long)9 * KC * KC, 0};
  return 0;
}

int local_joint_tc_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st) {
  return tc_try(m, nullptr, 1.f, partial, max_ctas, slots, st);
}

int local_joint_tc_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, int max_ctas,
                          SlotInfo* slots, cudaStream_t st) {
  return tc_try(m, stats, inv_temp, partial, max_ctas, slots, st);
}

}  // namespace iic
