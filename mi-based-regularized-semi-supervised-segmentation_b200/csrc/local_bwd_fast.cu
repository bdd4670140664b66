// Specialised local backward (the convolution_backward of contrastyou/losses/iic_loss.py:123) for the
// reference's udaiic shapes: window 3 x 3 or 7 x 7 (padding 1 or 3, config/semi.yaml), 10 or 20 clusters (and
// any multiple of 8 up to 256, in output blocks of 8),
// one patch, no mask (maps wider than 248 pixels are cut into column panels).  Both gradients come from the same kernel:
//   gx[i](px) = sum_{j,tap} Wx[j][tap][i] * y[j](px + tap)      gy[j](px) = sum_{i,tap} Wy[i][tap][j] * x[i](px + tap)
// (Wx / Wy = dL/dJ re-laid by the epilogue kernel).
//
// Work decomposition.  The B*H image rows are dealt out in equal contiguous shares to the persistent
// CTAs (one per SM), so no SM idles in a last partial wave; a CTA walks its share in chunks of CR whole
// rows (CR * W/4 <= 512).  A thread owns one row x 4 pixels x 10 output channels = 20 float2
// accumulators (pairs over adjacent output channels); 16 consumer warps = 4 per SM sub-partition.
// Per input channel and window row a thread loads its 4 + 2*pad window values (one LDS.128, the halo
// columns come from the neighbouring lanes by shuffle).  The weights are warp-uniform, so they never touch
// a vector register or the LSU: the host copies dL/dJ (Wx, Wy) device-to-device into __constant__ memory
// in front of the launch and every update is one
//   FFMA2 acc, window.F32 (scalar), UR.F32x2 (weight pair, LDCU.64 from the constant bank), acc
// i.e. per input channel 20*T*T FFMA2 + 5*T*T uniform-datapath loads + a few shared-memory instructions.
//
// Input tiles (CR + 2*pad rows, full width + halo, 5 channels per stage) stream through a TMA ring with
// full/empty mbarriers per slot, refilled by a dedicated producer warp; the hardware zero-fills rows and
// columns outside the map, which is the conv's padding.  (The producer must be its own warp: a
// one-thread spin on an mbarrier inside the consumers' loop makes the compiler treat the loop counters
// as divergent, and the weight loads then fall off the uniform datapath -- LDC instead of LDCU.)
// With the weights in uniform registers a consumer needs ~70 registers, so 17 warps fit.
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"
#include "tma.cuh"

namespace iic {

namespace bwdfast {
constexpr int LP = 4;                  // halo columns staged left and right (keeps rows 16-byte aligned)
constexpr int WC_FLOATS = 15360;       // 60 KB of the 64 KB constant bank
}  // namespace bwdfast

// dL/dJ of this launch: [sweep][output block][cin][tap][WROW].  Launches on one stream are ordered, so the
// copy in front of launch n+1 cannot overtake launch n; when a launch needs less than half of the array
// two halves are used round-robin, which also keeps two interleaved streams apart.  More than two streams
// running this backward concurrently are not supported.
__constant__ float2 g_wc[bwdfast::WC_FLOATS / 2];

struct BwdFastParams {
  int wc_base;               // float2 index of this launch's weights in g_wc
  int sw0, nsw;              // sweeps done by this launch: [sw0, sw0 + nsw)   (0 = gx, 1 = gy)
  int ob0;                   // first output-channel block of this launch (blockIdx.y counts from it)
  int B, K, H, W;
  int PW, NPW;               // column panels: width (multiple of 4, <= 248) and count; W <= 248 is one panel
  int QW, CR, XP, XR;        // thread tiles per panel row, rows per chunk, tile pitch (floats) and rows
  int plane;                 // floats per channel plane of a stage
  long long rows_total;      // B * NPW * H: rows of all (image, panel) strips, dealt out to the CTAs
  unsigned stage_bytes, box_bytes;
  const float* grad_loss;
  float* gx;
  float* gy;
  long long gx_sn, gy_sn;    // sample strides of the gradient tensors in elements (channel planes and rows are dense)
  // FROM_LOGITS: the maps are logits; gx / gy receive the gradient with respect to the logits
  const float* lx; long long lx_sn, lx_sc, lx_sh;
  const float* ly; long long ly_sn, ly_sc, ly_sh;
  float inv_temp;
};

// v = shared[addr] where pred != 0 (a predicated LDS: no divergent branch around a one-lane load)
__device__ __forceinline__ void lds_if(float& v, uint32_t addr, int pred) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, 0;\n\t@p ld.shared.f32 %0, [%1];\n\t}" : "+f"(v) : "r"(addr), "r"(pred));
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}

// KB = output channels per CTA (10, or 8 for channel counts that are multiples of 8 but not of 10), T x T
// window; NWARPS consumer warps + one producer warp; CB input channels per stage.  P.K = all channels.
template <int KB, int T, int NWARPS, int STAGES, int CB, bool FROM_LOGITS>
__global__ void __launch_bounds__((NWARPS + 1) * 32, 1)
local_bwd_fast_kernel(const __grid_constant__ CUtensorMap mapx, const __grid_constant__ CUtensorMap mapy,
                      const BwdFastParams P) {
  using namespace bwdfast;
  constexpr int PAD = T / 2, T2 = T * T;
  constexpr int NPX = 4;
  constexpr int WROW = (KB + 3) & ~3;                       // floats per (cin, tap) weight row in the constant bank
  constexpr int K = KB;                                     // FROM_LOGITS only (P.K == KB there)
  const int nchunk = P.K / CB;                              // stages per sweep
  static_assert(PAD <= LP && PAD <= 3, "halo wider than the staged margin");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[STAGES];
  __shared__ __align__(8) uint64_t empty_bar[STAGES];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int ob_local = blockIdx.y;
  const int oc0 = (P.ob0 + ob_local) * KB;                  // this CTA's output-channel block
  const long long R0 = (long long)blockIdx.x * P.rows_total / gridDim.x;
  const long long R1 = (long long)(blockIdx.x + 1) * P.rows_total / gridDim.x;
  const int per_chunk = P.nsw * nchunk;                     // stages per row chunk

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], NWARPS);
    }
    mbar_fence_init();
  }
  __syncthreads();

  // (a warp vote makes the role test provably warp-uniform, so the consumers' loops stay on uniform
  // control flow and their weight loads on the uniform datapath)
  if (__any_sync(0xffffffffu, wid == NWARPS)) {
    // ===== producer warp: one lane walks the same (chunk, sweep, channel block) sequence as the consumers,
    // a ring slot is refilled as soon as every consumer warp has released it =====
    if (lane == 0) {
      tma_prefetch_desc(&mapx);
      tma_prefetch_desc(&mapy);
      unsigned k = 0;
      for (long long r = R0; r < R1;) {
        const int strip = (int)(r / P.H), h0 = (int)(r - (long long)strip * P.H);
        const int n = strip / P.NPW, panel = strip - n * P.NPW;
        int nr = P.CR;
        if (nr > P.H - h0) nr = P.H - h0;
        if (nr > R1 - r) nr = (int)(R1 - r);
        for (int st = 0; st < per_chunk; ++st, ++k) {
          const int sl = st / nchunk, cb = st - sl * nchunk;
          const int sweep = P.sw0 + sl;
          const int s = k % STAGES;
          if (k >= STAGES) mbar_wait(&empty_bar[s], ((k / STAGES) & 1u) ^ 1u);
          mbar_arrive_expect_tx(&full_bar[s], P.box_bytes);
          tma_load_4d(smem_raw + (size_t)s * P.stage_bytes, sweep == 0 ? &mapy : &mapx, &full_bar[s],
                      panel * P.PW - LP, h0 - PAD, cb * CB, n);       // gx reads y, gy reads x
        }
        r += nr;
      }
    }
    return;
  }

  // ===== consumer warps =====
  const float g = P.grad_loss ? __ldg(P.grad_loss) : 1.f;
  const int rr = threadIdx.x / P.QW, q = threadIdx.x - rr * P.QW;
  const bool in_tile = rr < P.CR;
  const int rr_c = in_tile ? rr : P.CR - 1;                 // idle threads read valid rows, store nothing
  const uint32_t toff = (uint32_t)(rr_c * P.XP + LP + NPX * q) * 4u;
  // the halo columns come from the neighbouring lanes, except at the warp's and the row's ends, where
  // they are read from the tile (columns < 0 and >= W hold the zero fill = the conv's padding)
  const int ld_left = (lane == 0) | (q == 0), ld_right = (lane == 31) | (q == P.QW - 1);
  const uint32_t xp4 = (uint32_t)P.XP * 4u, plane4 = (uint32_t)P.plane * 4u;
  const uint32_t smem_base = smem_u32(smem_raw);

  float2 acc[KB / 2][NPX];
  unsigned k = 0;
  for (long long r = R0; r < R1;) {
    const int strip = (int)(r / P.H), h0 = (int)(r - (long long)strip * P.H);
    const int n = strip / P.NPW, panel = strip - n * P.NPW;
    const int col0 = panel * P.PW;                          // first image column of this panel
    int nr = P.CR;
    if (nr > P.H - h0) nr = P.H - h0;
    if (nr > R1 - r) nr = (int)(R1 - r);
    const bool active = in_tile && rr < nr && col0 + NPX * q < P.W;
    const bool warp_active = __any_sync(0xffffffffu, active);
    for (int sl = 0; sl < P.nsw; ++sl) {
      const int sweep = P.sw0 + sl;
#pragma unroll
      for (int c = 0; c < KB / 2; ++c)
#pragma unroll
        for (int p = 0; p < NPX; ++p) acc[c][p] = make_float2(0.f, 0.f);
      // weight pairs of this sweep and output block: g_wc[wbase + (cin * T2 + tap) * WROW / 2 + c]
      const int wbase = P.wc_base + ((sl * (int)gridDim.y + ob_local) * P.K) * (T2 * WROW / 2);
      for (int cb = 0; cb < nchunk; ++cb, ++k) {
        const int s = k % STAGES;
        mbar_wait(&full_bar[s], (k / STAGES) & 1u);
        if constexpr (FROM_LOGITS) {
          // the staged tile holds logits: channel softmax in place (all K channels are in the stage, CB == K);
          // rows and columns outside the map must stay zero (the conv's padding)
          static_assert(!FROM_LOGITS || CB == K, "the fused softmax needs every channel of a pixel in one stage");
          float* tile = reinterpret_cast<float*>(smem_raw + (size_t)s * P.stage_bytes);
          const float k2 = P.inv_temp * 1.4426950408889634f;
          const int npos = P.XR * P.XP;
          for (int pos = threadIdx.x; pos < npos; pos += NWARPS * 32) {
            const int tr = pos / P.XP, tc = pos - tr * P.XP;
            const bool valid = (unsigned)(h0 - PAD + tr) < (unsigned)P.H && (unsigned)(col0 + tc - LP) < (unsigned)P.W;
            float v[K];
            float mx = -3.0e38f;
#pragma unroll
            for (int c = 0; c < K; ++c) { v[c] = tile[c * P.plane + pos]; mx = fmaxf(mx, v[c]); }
            float sum = 0.f;
#pragma unroll
            for (int c = 0; c < K; ++c) { v[c] = exp2f((v[c] - mx) * k2); sum += v[c]; }
            const float inv = valid ? 1.f / sum : 0.f;
#pragma unroll
            for (int c = 0; c < K; ++c) tile[c * P.plane + pos] = v[c] * inv;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(NWARPS * 32) : "memory");     // consumers only
        }
        if (warp_active) {
          uint32_t cp = smem_base + (uint32_t)s * P.stage_bytes + toff;
#pragma unroll 1
          for (int ch = 0; ch < CB; ++ch, cp += plane4) {
            const int wq = wbase + (cb * CB + ch) * (T2 * WROW / 2);
#pragma unroll
            for (int ry = 0; ry < T; ++ry) {
              // window row ry: NPX own pixels + PAD halo columns on each side
              const uint32_t rp = cp + ry * xp4;
              float win[NPX + 2 * PAD];
              const float4 v = lds128(rp);
              win[PAD + 0] = v.x; win[PAD + 1] = v.y; win[PAD + 2] = v.z; win[PAD + 3] = v.w;
#pragma unroll
              for (int h = 0; h < PAD; ++h) {
                float l = __shfl_up_sync(0xffffffffu, win[PAD + NPX - PAD + h], 1);      // left neighbour's last PAD
                float rt = __shfl_down_sync(0xffffffffu, win[PAD + h], 1);               // right neighbour's first PAD
                lds_if(l, rp - 4 * (PAD - h), ld_left);
                lds_if(rt, rp + 4 * (NPX + h), ld_right);
                win[h] = l;
                win[PAD + NPX + h] = rt;
              }
#pragma unroll
              for (int rx = 0; rx < T; ++rx) {
                float2 wp[KB / 2];
#pragma unroll
                for (int c = 0; c < KB / 2; ++c) wp[c] = g_wc[wq + (ry * T + rx) * (WROW / 2) + c];
#pragma unroll
                for (int p = 0; p < NPX; ++p) {
                  const float a = win[p + rx];
                  const float2 a2 = make_float2(a, a);
#pragma unroll
                  for (int c = 0; c < KB / 2; ++c) acc[c][p] = __ffma2_rn(a2, wp[c], acc[c][p]);
                }
              }
            }
          }
        }
        __syncwarp();
        if constexpr (FROM_LOGITS) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // our writes vs the next TMA fill
        if (lane == 0) mbar_arrive(&empty_bar[s]);
      }
      if constexpr (FROM_LOGITS) {
        // chain through the cluster head's softmax (contrastyou/trainer/_utils.py:15-23): the thread holds
        // dL/dp for all K channels of its pixels, so  dL/dlogit = p * (dL/dp - sum_k dL/dp_k p_k) / T  is a
        // per-thread epilogue; p is recomputed from the logits (one coalesced 16-byte load per channel)
        if (active) {
          const float* lg = sweep == 0 ? P.lx : P.ly;
          const long long sn = sweep == 0 ? P.lx_sn : P.ly_sn, sc = sweep == 0 ? P.lx_sc : P.ly_sc,
                          sh = sweep == 0 ? P.lx_sh : P.ly_sh;
          const float* src = lg + (long long)n * sn + (long long)(h0 + rr) * sh + col0 + NPX * q;
          const float k2 = P.inv_temp * 1.4426950408889634f;
          float4 l[K];
#pragma unroll
          for (int c = 0; c < K; ++c) l[c] = __ldg(reinterpret_cast<const float4*>(src + (long long)c * sc));
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float pv[K];
            float mx = -3.0e38f;
#pragma unroll
            for (int c = 0; c < K; ++c) { pv[c] = (&l[c].x)[e]; mx = fmaxf(mx, pv[c]); }
            float sum = 0.f;
#pragma unroll
            for (int c = 0; c < K; ++c) { pv[c] = exp2f((pv[c] - mx) * k2); sum += pv[c]; }
            const float inv = 1.f / sum;
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < K; ++c) {
              pv[c] *= inv;
              const float gc = (c & 1) ? acc[c / 2][e].y : acc[c / 2][e].x;
              dot = fmaf(gc, pv[c], dot);
            }
#pragma unroll
            for (int c = 0; c < K; ++c) {
              float& gc = (c & 1) ? acc[c / 2][e].y : acc[c / 2][e].x;
              gc = pv[c] * (gc - dot) * P.inv_temp;
            }
          }
        }
      }
      if (active) {
        float* out = (sweep == 0 ? P.gx + (size_t)n * P.gx_sn : P.gy + (size_t)n * P.gy_sn) + ((size_t)oc0 * P.H + (h0 + rr)) * P.W + col0 + NPX * q;
        const size_t cs = (size_t)P.H * P.W;
#pragma unroll
        for (int c = 0; c < KB / 2; ++c) {
          *reinterpret_cast<float4*>(out + (size_t)(2 * c) * cs) =
              make_float4(g * acc[c][0].x, g * acc[c][1].x, g * acc[c][2].x, g * acc[c][3].x);
          *reinterpret_cast<float4*>(out + (size_t)(2 * c + 1) * cs) =
              make_float4(g * acc[c][0].y, g * acc[c][1].y, g * acc[c][2].y, g * acc[c][3].y);
        }
      }
    }
    r += nr;
  }
}

template <int KB, int T, int NWARPS, int STAGES, int CB, bool FROM_LOGITS>
static int launch_bwd_fast(const CUtensorMap& mx, const CUtensorMap& my, const BwdFastParams& P, dim3 grid,
                           size_t smem, cudaStream_t st) {
  auto kern = local_bwd_fast_kernel<KB, T, NWARPS, STAGES, CB, FROM_LOGITS>;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(kern), (int)(226 * 1024)));
  kern<<<grid, (NWARPS + 1) * 32, smem, st>>>(mx, my, P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

int local_bwd_fast_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, int from_logits,
                       float inv_temp, cudaStream_t st) {
  using namespace bwdfast;
  const int B = m.B, K = m.K, H = m.H, W = m.W, pad = m.pad;
  if (pad != 1 && pad != 3) return -1;
  // output-channel block: 10 for the udaiic cluster counts (10, 20), 8 for other multiples of 8 (.., 128)
  const int KB = (K % 10 == 0 && K <= 40) ? 10 : (K % 8 == 0 ? 8 : 0);
  if (KB == 0 || K > 256) return -1;
  if (from_logits && (K != 10 || pad != 1)) return -1;
  const int WROW = (KB + 3) & ~3;
  if (W % 4 != 0 || W < 4) return -1;
  if (from_logits && W > 248) return -1;
  if ((reinterpret_cast<uintptr_t>(g.gx) & 15) || (reinterpret_cast<uintptr_t>(g.gy) & 15) || (g.gx_sn & 3) || (g.gy_sn & 3))
    return -1;
  const int T = 2 * pad + 1, T2 = T * T, Kp = (K + 3) & ~3;
  const int CB = from_logits ? 10 : (KB == 10 ? 5 : 4);   // the fused softmax needs all K channels in one stage
  const int nthreads = 512, stages = from_logits ? 2 : (pad == 1 ? 4 : 3);
  BwdFastParams P;
  P.B = B; P.K = K; P.H = H; P.W = W;
  // maps wider than one TMA box are cut into column panels of equal width (the last may be narrower)
  P.NPW = (W + 247) / 248;
  P.PW = (((W + P.NPW - 1) / P.NPW) + 3) & ~3;
  P.QW = P.PW / 4;
  P.CR = nthreads / P.QW;
  if (P.CR > 62) P.CR = 62;
  if (P.CR > H) P.CR = H;
  P.XP = P.PW + 2 * LP;
  P.XR = P.CR + 2 * pad;
  P.plane = P.XR * P.XP;
  P.rows_total = (long long)B * P.NPW * H;
  P.box_bytes = (unsigned)((size_t)CB * P.plane * 4);
  P.stage_bytes = (P.box_bytes + 127u) & ~127u;
  const size_t smem = (size_t)P.stage_bytes * stages;
  if (smem > 226 * 1024) return -1;
  P.grad_loss = g.grad_loss; P.gx = g.gx; P.gy = g.gy; P.gx_sn = g.gx_sn; P.gy_sn = g.gy_sn;
  P.lx = m.x.p; P.lx_sn = m.x.sn; P.lx_sc = m.x.sc; P.lx_sh = m.x.sh;
  P.ly = m.y.p; P.ly_sn = m.y.sn; P.ly_sc = m.y.sc; P.ly_sh = m.y.sh;
  P.inv_temp = inv_temp;
  auto rows16 = [](const View4& v) {
    return (reinterpret_cast<uintptr_t>(v.p) & 15) == 0 && v.sh % 4 == 0 && v.sc % 4 == 0 && v.sn % 4 == 0;
  };
  if (from_logits && (!rows16(m.x) || !rows16(m.y))) return -1;
  CUtensorMap mx, my;
  if (!make_map_4d(&mx, m.x, m, P.XP, P.XR, CB)) return -1;
  if (!make_map_4d(&my, m.y, m, P.XP, P.XR, CB)) return -1;
  const int nob = K / KB;

  // How many (sweep, output block) weight slabs fit in the constant bank at once decides the launches:
  // everything in one launch (3 x 3 windows; 7 x 7 with 10 clusters) or one launch per slab (7 x 7, K = 20).
  const int slab = K * T2 * WROW;                           // floats of one (sweep, output block) slab
  const bool one_launch = 2 * nob * slab <= WC_FLOATS;
  if (!one_launch && slab > WC_FLOATS) return -1;
  float2* wc_dev = nullptr;
  IIC_CHECK_CUDA(cudaGetSymbolAddress(reinterpret_cast<void**>(&wc_dev), g_wc));
  static unsigned slot_counter = 0;

  auto run = [&](int sw0, int nsw, int ob0, int nobl) -> int {
    const int need = nsw * nobl * slab;
    int base = 0;                                           // floats
    if (2 * need <= WC_FLOATS) base = (int)(slot_counter++ & 1u) * (WC_FLOATS / 2);
    // dL/dJ -> constant bank: one strided device-to-device copy per slab (stream ordered, capturable);
    // each (cin, tap) row keeps the 10 weights of the slab's output block in a 12-float row
    for (int s = 0; s < nsw; ++s)
      for (int o = 0; o < nobl; ++o) {
        const float* src = ((sw0 + s) == 0 ? Wx : Wy) + (size_t)(ob0 + o) * KB;
        float* dst = reinterpret_cast<float*>(wc_dev) + base + (size_t)(s * nobl + o) * slab;
        IIC_CHECK_CUDA(cudaMemcpy2DAsync(dst, WROW * sizeof(float), src, (size_t)Kp * sizeof(float),
                                         KB * sizeof(float), (size_t)K * T2, cudaMemcpyDeviceToDevice, st));
      }
    P.wc_base = base / 2;
    P.sw0 = sw0; P.nsw = nsw; P.ob0 = ob0;
    int gxd = m.sms / nobl;
    if (gxd < 1) gxd = 1;
    if (gxd > P.rows_total) gxd = (int)P.rows_total;
    const dim3 grid(gxd, nobl);
    if (from_logits) return launch_bwd_fast<10, 3, 16, 2, 10, true>(mx, my, P, grid, smem, st);
    if (KB == 10 && T == 3) return launch_bwd_fast<10, 3, 16, 4, 5, false>(mx, my, P, grid, smem, st);
    if (KB == 10 && T == 7) return launch_bwd_fast<10, 7, 16, 3, 5, false>(mx, my, P, grid, smem, st);
    if (KB == 8 && T == 3) return launch_bwd_fast<8, 3, 16, 4, 4, false>(mx, my, P, grid, smem, st);
    return launch_bwd_fast<8, 7, 16, 3, 4, false>(mx, my, P, grid, smem, st);
  };

  if (one_launch) return run(0, 2, 0, nob);
  for (int sw = 0; sw < 2; ++sw)
    for (int ob = 0; ob < nob; ++ob)
      if (int rc = run(sw, 1, ob, 1)) return rc;
  return 0;
}

}  // namespace iic
