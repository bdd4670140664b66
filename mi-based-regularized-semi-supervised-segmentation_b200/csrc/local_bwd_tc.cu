// Backward sweeps of the local IIC term on the 5th-generation tensor cores (tcgen05 / UMMA) for wide cluster heads:
// K = 128 channels, 3 x 3 window (padding 1) -- BASELINE config 5.  One launch computes one gradient map
//   out[n,o,r,c] = g * sum_{cin,ty,tx} Wc[cin][ty*3+tx][o] * src[n,cin,r+ty-1,c+tx-1]          (src zero outside the map)
// which is what autograd's convolution_backward yields for the F.conv2d at contrastyou/losses/iic_loss.py:123 with
// Wc = the coefficient tensors iic_local_epilogue writes (Wx with src = y gives dL/dx, Wy with src = x gives dL/dy).
//
// GEMM view: M = pixels (128 per MMA, TMEM lanes), N = 128 output channels (TMEM columns), reduction = input channels
// (8 per step) x 9 taps.  fp32-level accuracy from a split product: with ah = the top 19 bits of a (what kind::tf32
// reads of an fp32 word) and al = a - ah (exact), a*w = ah*wh + (al*wh + ah*wl) + al*wl.  The main term is one
// tcgen05.mma.kind::tf32 (K = 8 channels); the two correction terms, 2^-11 of it, only need ~8 bits and share ONE
// tcgen05.mma.kind::f16 on bf16 copies with K = 16 = [al | ah] x [wh | wl]; al*wl (2^-22) is dropped.  Two MMAs per
// step instead of the three of a plain 3xTF32 scheme.
//
// The +-1 column shifts of the taps are start-address shifts of the A descriptor: the transform warps re-lay every
// staged row pixel-major, as a K-major operand WITHOUT swizzle whose rows (pixels) are 16 bytes = 4 channels and whose
// 8-row core matrices follow each other directly (stride-byte-offset 128), so pixel b of the row buffer sits at
// b * 16 bytes and a window that starts one pixel later starts 16 bytes later.  (TMA cannot make these shifts: a box may
// only start at a multiple of 4 floats.)  Row shifts pick another row buffer.
//
// One CTA per SM walks a contiguous share of the (image, row pair) work items.  Per item the accumulators are the four
// 128-column TMEM blocks [output row 0/1][pixel tile 0/1]; the 128 input channels stream through in 16 slices of 8:
//   warp 0     TMA: the slice's four source rows r-1 .. r+2 as two [8 ch x 2 rows x (W+8) px] boxes (zero fill = padding)
//   warp 3     TMEM allocation; bulk copies of the slice's nine 8 KB weight tiles (fp32 + bf16 parts, already in operand order), ring of 6
//   warps 4-7  transform: [ch][row][px] fp32 -> [row][chunk][px][16 B] operand images (fp32: 4 channels per
//              chunk; bf16: chunk 0 = al, chunk 1 = ah of the 8 channels)
//   warps 1-2  MMA issuers (one lane each, one output row each): 9 taps x 2 tiles x 2 MMAs per slice and row
//   warps 8-11 epilogue after the 16th slice: tcgen05.ld (lane = pixel, columns = channels), scale by g, coalesced stores
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tc_common.cuh"
#include "tma.cuh"

namespace iic {
namespace bwdtc {
using namespace tc;

constexpr int KC = 128;                  // channels (UMMA N = output channels, reduction = input channels)
constexpr int SL = 8;                    // input channels per slice (one UMMA K step of tf32)
constexpr int NSL = KC / SL;             // 16 slices
constexpr int APX = 272;                 // pixels per row buffer; buffer pixel b holds column b - 8, so that the window of the
                                         // centre tap starts on a 128-byte boundary (rows up to b = 264 are read)
constexpr int MAXW = 248;                // widest map: W + 8 staged columns <= 256 (TMA box limit)
constexpr int A_PART = 4 * 2 * APX * 16; // fp32 part / bf16 correction part: 4 rows x 2 chunks x APX pixels x 16 B = 34816
constexpr int A_SLOT = 2 * A_PART;       // 69632
constexpr int NA = 2;
constexpr int W_TILE = 2 * 2 * KC * 16;  // fp32 part, bf16 part x 2 chunks x 128 channels x 16 B = 8192
constexpr int NW = 6;
constexpr int RAW_HALF_MAX = SL * 2 * 256 * 4;   // 16384 (8 ch x 2 rows x up to 256 px)
constexpr int SMEM_BYTES = NA * A_SLOT + NW * W_TILE + 2 * RAW_HALF_MAX + 1024;
constexpr int NTHREADS = 384;


struct Params {
  int B, H, W;
  int n_items;                  // B * ceil(H / 2)
  const float* wimg;            // [16 slices][9 taps]{fp32 [2 chunks][128 out][4 in], bf16 [wh, wl][128 out][8 in]}
  const float* grad_loss;       // device scalar or null
  float* out;                   // (B, 128, H, W), channel planes dense
  long long out_sn;             // sample stride of `out` in elements
  int dbg;                      // bring-up switches (IIC_TC_DBG): 1 no source loads, 2 no weight loads, 4 no transform, 8 no stores
};

// Wc[cin][tap][128] (iic_local_epilogue) -> operand image: the fp32 tile and the bf16 correction tile [wh | wl]
__global__ void weight_image_kernel(const float* __restrict__ Wc, float* __restrict__ img) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;      // one (slice, tap, out) per thread: 8 input channels
  if (e >= NSL * 9 * KC) return;
  const int o = e % KC, tap = (e / KC) % 9, js = e / (KC * 9);
  float v[SL];
#pragma unroll
  for (int q = 0; q < SL; ++q) v[q] = Wc[((size_t)(js * SL + q) * 9 + tap) * KC + o];
  float4* dst = reinterpret_cast<float4*>(img) + (size_t)(js * 9 + tap) * (W_TILE / 16);
  dst[o] = make_float4(v[0], v[1], v[2], v[3]);
  dst[KC + o] = make_float4(v[4], v[5], v[6], v[7]);
  reinterpret_cast<uint4*>(dst)[2 * KC + o] = pack8<false>(v);     // wh (pairs with al)
  reinterpret_cast<uint4*>(dst)[3 * KC + o] = pack8<true>(v);      // wl (pairs with ah)
}

__global__ void __launch_bounds__(NTHREADS, 1)
local_bwd_tc_kernel(const __grid_constant__ CUtensorMap maps, const Params P) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t raw_full[2], raw_empty[2], a_full[NA], a_empty[NA], w_full[NW], w_empty[NW], accum_full, tmem_empty;
  __shared__ uint32_t tmem_base_s;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* a_ring = smem;
  unsigned char* w_ring = smem + NA * A_SLOT;
  unsigned char* raw_ring = w_ring + NW * W_TILE;
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int it0 = (int)((long long)blockIdx.x * P.n_items / gridDim.x);
  const int it1 = (int)((long long)(blockIdx.x + 1) * P.n_items / gridDim.x);
  const int nit = it1 - it0;
  const int pairs = (P.H + 1) >> 1;
  const int SW = P.W + 8;                                  // staged columns: -4 .. W+3
  const int raw_half_bytes = SL * 2 * SW * 4;
  const int ntile = P.W > 128 ? 2 : 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&raw_empty[s], 4); }
    for (int s = 0; s < NA; ++s) { mbar_init(&a_full[s], 4); mbar_init(&a_empty[s], 2); }
    for (int s = 0; s < NW; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 2); }
    mbar_init(&accum_full, 2);
    mbar_init(&tmem_empty, 4);
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
    // ===== TMA producer: source rows =====
    if (lane == 0) {
      tma_prefetch_desc(&maps);
      for (int i = 0; i < nit; ++i) {
        const int item = it0 + i;
        const int n = item / pairs, r = (item - n * pairs) * 2;
        for (int js = 0; js < NSL; ++js) {
          const int t = i * NSL + js;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (t >= 1) mbar_wait(&raw_empty[h], ((unsigned)t & 1u) ^ 1u, 1);
            if (P.dbg & 1) { mbar_arrive(&raw_full[h]); continue; }
            mbar_arrive_expect_tx(&raw_full[h], raw_half_bytes);
            tma_load_4d(raw_ring + h * RAW_HALF_MAX, &maps, &raw_full[h], -4, r - 1 + 2 * h, js * SL, n);
          }
        }
      }
    }
  } else if (wid == 3) {
    // ===== weight tiles =====
    if (lane == 0) {
      const int total = nit * NSL * 9;
      for (int w = 0; w < total; ++w) {
        const int s = w % NW;
        if (w >= NW) mbar_wait(&w_empty[s], ((unsigned)(w / NW) & 1u) ^ 1u, 2);
        if (P.dbg & 2) { mbar_arrive(&w_full[s]); continue; }
        mbar_arrive_expect_tx(&w_full[s], W_TILE);
        bulk_load(w_ring + s * W_TILE, P.wimg + (size_t)(w % (NSL * 9)) * (W_TILE / 4), W_TILE, &w_full[s]);
      }
    }
  } else if (wid == 1 || wid == 2) {
    // ===== MMA issuers: warp 1 owns the accumulators of output row 0, warp 2 those of output row 1.  With one issuing
    // lane an MMA went out every ~104 clk, with two every ~88 clk (both measured with everything else ablated, and both
    // independent of N down to N = 8: the limit is per instruction, not tensor math).  Each warp commits to the ring
    // barriers. =====
    const int orow = wid - 1;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(KC >> 3) << 17) | ((uint32_t)(KC >> 4) << 24);
    const uint32_t idesc_bf16 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(KC >> 3) << 17) | ((uint32_t)(KC >> 4) << 24);
    for (int i = 0; i < nit; ++i) {
      const int item = it0 + i;
      const int n = item / pairs, r = (item - n * pairs) * 2;
      const int nrow = (r + 1 < P.H) ? 2 : 1;
      if (i > 0) {
        mbar_wait(&tmem_empty, (unsigned)(i - 1) & 1u, 6);
        asm volatile("tcgen05.fence::after_thread_sync;");
      }
      for (int js = 0; js < NSL; ++js) {
        const int t = i * NSL + js;
        const int a = t % NA;
        mbar_wait(&a_full[a], (unsigned)(t / NA) & 1u, 5);
        // The issuing lane is latency-bound on its own instruction stream, so every descriptor is a 64-bit base plus a
        // compile-time constant (in 16-byte units): the tap / row / tile loops are fully unrolled.
        const uint64_t a_base = make_desc_kmajor_noswz(smem_u32(a_ring + (size_t)a * A_SLOT), APX * 16) + (uint64_t)(orow * 2 * APX);
        const uint32_t d_row = tmem_base + (uint32_t)(orow * 2) * KC;
        const int w0 = t * 9;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const int w = w0 + tap;
          const int s = w % NW;
          mbar_wait(&w_full[s], (unsigned)(w / NW) & 1u, 7);
          asm volatile("tcgen05.fence::after_thread_sync;");
          if (lane == 0) {
            constexpr int A_CR = A_PART / 16, B_CR = 2 * KC;          // offsets of the bf16 parts, 16-byte units
            const int ty = tap / 3, tx = tap - ty * 3;
            const uint64_t b_hi = make_desc_kmajor_noswz(smem_u32(w_ring + (size_t)s * W_TILE), KC * 16);
            const uint32_t acc0 = (tap > 0 || js > 0) ? 1u : 0u;
            // output pixel c of row r+orow reads source row r+orow+ty-1 (buffer row orow+ty), column c+tx-1 (buffer pixel c+tx+7)
            if (orow < nrow) {
              if (ntile == 2) {
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                  const int off = (ty * 2) * APX + mt * 128 + tx + 7;
                  const uint32_t d_tmem = d_row + (uint32_t)mt * KC;
                  umma_bf16(d_tmem, a_base + (uint64_t)(A_CR + off), b_hi + B_CR, idesc_bf16, acc0);   // al*wh + ah*wl
                  umma_tf32(d_tmem, a_base + (uint64_t)off, b_hi, idesc, 1u);
                }
              } else {
                const int off = (ty * 2) * APX + tx + 7;
                const uint32_t d_tmem = d_row;
                umma_bf16(d_tmem, a_base + (uint64_t)(A_CR + off), b_hi + B_CR, idesc_bf16, acc0);
                umma_tf32(d_tmem, a_base + (uint64_t)off, b_hi, idesc, 1u);
              }
            }
            umma_commit(&w_empty[s]);
            if (tap == 8) {
              umma_commit(&a_empty[a]);
              if (js == NSL - 1) umma_commit(&accum_full);
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (wid >= 4 && wid < 8) {
    // ===== transform: [ch][row][px] -> [row][chunk][px][4 ch], hi and lo =====
    const int tid = threadIdx.x - 128;
    const int total = nit * NSL;
    for (int t = 0; t < total; ++t) {
      const int a = t % NA;
      if (t >= NA) mbar_wait(&a_empty[a], ((unsigned)(t / NA) & 1u) ^ 1u, 3);
      unsigned char* ahi = a_ring + (size_t)a * A_SLOT;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        mbar_wait(&raw_full[h], (unsigned)t & 1u, 4);
        const float* raw = reinterpret_cast<const float*>(raw_ring + h * RAW_HALF_MAX);
        for (int e = tid; e < ((P.dbg & 4) ? 0 : 2 * SW); e += 128) {
          const int row = e >= SW ? 1 : 0;
          const int px = e - row * SW;
          float v[SL];
#pragma unroll
          for (int c = 0; c < SL; ++c) v[c] = raw[(c * 2 + row) * SW + px];
          const int q = 2 * h + row;
          const int off = ((q * 2) * APX + px + 4) * 16;                 // staged pixel px is column px - 4
          *reinterpret_cast<float4*>(ahi + off) = make_float4(v[0], v[1], v[2], v[3]);
          *reinterpret_cast<float4*>(ahi + off + APX * 16) = make_float4(v[4], v[5], v[6], v[7]);
          *reinterpret_cast<uint4*>(ahi + A_PART + off) = pack8<true>(v);              // al (pairs with wh)
          *reinterpret_cast<uint4*>(ahi + A_PART + off + APX * 16) = pack8<false>(v);  // ah (pairs with wl)
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&raw_empty[h]);
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> tensor-core reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_full[a]);
    }
  } else if (wid >= 8) {
    // ===== epilogue =====
    const int q4 = wid & 3;                                  // TMEM lanes 32*q4 .. 32*q4+31
    const float g = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
    const size_t plane = (size_t)P.H * P.W;
    for (int i = 0; i < nit; ++i) {
      const int item = it0 + i;
      const int n = item / pairs, r = (item - n * pairs) * 2;
      const int nrow = (r + 1 < P.H) ? 2 : 1;
      mbar_wait(&accum_full, (unsigned)i & 1u, 8);
      asm volatile("tcgen05.fence::after_thread_sync;");
      for (int orow = 0; orow < nrow; ++orow)
        for (int mt = 0; mt < ntile; ++mt) {
          const int c = mt * 128 + q4 * 32 + lane;
          float* dst = P.out + (size_t)n * P.out_sn + (size_t)(r + orow) * P.W + c;
#pragma unroll 1
          for (int ch = 0; ch < KC / 32; ++ch) {
            uint32_t v[32];
            const uint32_t taddr = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(orow * 2 + mt) * KC + ch * 32;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (c < P.W && !(P.dbg & 8)) {
#pragma unroll
              for (int o = 0; o < 32; ++o) dst[(size_t)(ch * 32 + o) * plane] = g * __uint_as_float(v[o]);
            }
          }
        }
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  if (wid == 3) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

}  // namespace bwdtc

size_t local_bwd_tc_image_bytes(int K, int pad) {
  return (K == bwdtc::KC && pad == 1) ? (size_t)bwdtc::NSL * 9 * bwdtc::W_TILE : 0;
}

int local_bwd_tc_try(const LocalMaps& m, float* Wx, float* Wy, const LocalGrads& g, cudaStream_t st) {
  using namespace bwdtc;
  const int B = m.B, K = m.K, H = m.H, W = m.W, pad = m.pad, sms = m.sms;
  if (K != KC || pad != 1 || W % 4 != 0 || W > MAXW || W < 8) return -1;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, W + 8, 2, SL)) return -1;
  if (!make_map_4d(&my, m.y, m, W + 8, 2, SL)) return -1;
  // the weight image lives in the tail of the caller's coefficient buffer (common.cuh)
  float* img_x = Wx + local_coeff_image_offset(K, pad, 1);
  float* img_y = Wy + local_coeff_image_offset(K, pad, 1);
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(local_bwd_tc_kernel), (int)(SMEM_BYTES)));
  const int n_items = B * ((H + 1) / 2);
  const int grid = n_items < sms ? n_items : sms;
  const int wthreads = NSL * 9 * KC;
  weight_image_kernel<<<(wthreads + 255) / 256, 256, 0, st>>>(Wx, img_x);
  weight_image_kernel<<<(wthreads + 255) / 256, 256, 0, st>>>(Wy, img_y);
  IIC_CHECK_CUDA(cudaGetLastError());
  const int dbg = tc::bringup_env("IIC_TC_DBG", 0);
  Params Pgx{B, H, W, n_items, img_x, g.grad_loss, g.gx, g.gx_sn, dbg};     // dL/dx from y
  local_bwd_tc_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(my, Pgx);
  Params Pgy{B, H, W, n_items, img_y, g.grad_loss, g.gy, g.gy_sn, dbg};     // dL/dy from x
  local_bwd_tc_kernel<<<grid, NTHREADS, SMEM_BYTES, st>>>(mx, Pgy);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic
