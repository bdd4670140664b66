// Forward of the local IIC term: all (2*pad+1)^2 shifted-window joints
//   J[patch][dy][dx][i][j] = sum_{n,u,v} x[n,i,u+dy-pad,v+dx-pad] * y[n,j,u,v]
// i.e. the F.conv2d at contrastyou/losses/iic_loss.py:120-123 (whose "filter" is the whole map),
// with the optional mask of :116-118 folded into the tile staging.
//
// Design (DESIGN.md "local joint"): output-stationary SIMT FMA.  The contraction is a skinny GEMM
// [T*T*K x Npix] x [Npix x K]; at the segmentation sizes (K = 10..20) padding it to a tcgen05 tile
// wastes > 55 % of the MMA and the A operand must be re-read from shared memory for every one of the
// T*T shifts, so the tensor pipe is shared-memory-bound below the FP32 pipe's rate.  Instead every
// warp owns a register block acc[IT][JT][T][T] of the output (a "job"), lanes own pixel columns, and
// a warp walks down the rows of a shared-memory tile keeping a sliding T x T window of x in registers:
// per row step it loads IT*T new x values and JT y values and issues IT*JT*T*T FMAs.
// fp32 accumulation runs are short (one CTA's share of the pixels, per lane); lanes are combined
// with warp shuffles and CTAs in fp64 in a fixed order (reduce_partials_kernel), so the result is
// deterministic and its error is well below the reference's own fp32 error (DESIGN.md "numerics").
#include <stdlib.h>

#include "common.cuh"
#include "local_kernels.cuh"

namespace iic {

struct LocalFwdParams {
  View4 x, y, m;            // m.p == nullptr: no mask
  int B;
  int Ki, Kj;               // channels of x / y handled by this launch (a chunk of K)
  int i_off, j_off, K;      // position of the chunk inside the full K x K output
  int pad;
  PatchGrid g;
  int TH, TWS;              // tile rows, tile strips of 32 columns
  int tiles_h, tiles_w;     // tiles per patch
  int XR, XP;               // x tile rows (TH+2p) and pitch
  int njobs_i, njobs_j, njobs, rounds;
  float* partial;           // [patch][gridDim.x][T*T][K][K]
};

// stage one tile of x (with halo) and y into shared memory, zero outside the patch
__device__ __forceinline__ void stage_tile(const LocalFwdParams& P, float* xs, float* ys, int n,
                                           int ph0, int pw0, int th0, int tw0) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int TW = P.TWS * 32;
  const int XC = TW + 2 * P.pad;
  // x rows: (channel, r) pairs
  for (int row = wid; row < P.Ki * P.XR; row += nwarps) {
    const int ch = row / P.XR, r = row - ch * P.XR;
    const int gh = th0 + r - P.pad;                     // row inside the patch
    float* dst = xs + (size_t)row * P.XP;
    const bool row_ok = gh >= 0 && gh < P.g.ph;
    const float* src = P.x.p + n * P.x.sn + (long long)(P.i_off + ch) * P.x.sc + (long long)(ph0 + gh) * P.x.sh + pw0;
    const float* msrc = P.m.p ? P.m.p + n * P.m.sn + (long long)(P.i_off + ch) * P.m.sc + (long long)(ph0 + gh) * P.m.sh + pw0 : nullptr;
    for (int cc = lane; cc < P.XP; cc += 32) {
      const int gw = tw0 + cc - P.pad;
      float v = 0.f;
      if (row_ok && cc < XC && gw >= 0 && gw < P.g.pw) {
        v = __ldg(src + gw);
        if (msrc) v *= __ldg(msrc + gw);
      }
      dst[cc] = v;
    }
  }
  for (int row = wid; row < P.Kj * P.TH; row += nwarps) {
    const int ch = row / P.TH, r = row - ch * P.TH;
    const int gh = th0 + r;
    float* dst = ys + (size_t)row * TW;
    const bool row_ok = gh < P.g.ph;
    const float* src = P.y.p + n * P.y.sn + (long long)(P.j_off + ch) * P.y.sc + (long long)(ph0 + gh) * P.y.sh + pw0;
    const float* msrc = P.m.p ? P.m.p + n * P.m.sn + (long long)(P.j_off + ch) * P.m.sc + (long long)(ph0 + gh) * P.m.sh + pw0 : nullptr;
    for (int cc = lane; cc < TW; cc += 32) {
      const int gw = tw0 + cc;
      float v = 0.f;
      if (row_ok && gw < P.g.pw) {
        v = __ldg(src + gw);
        if (msrc) v *= __ldg(msrc + gw);
      }
      dst[cc] = v;
    }
  }
}

// One job over one staged tile.  DYB == T: full T x T window, sliding down the rows.
// DYB == 1: the job covers a single dy row of displacements (used for wide windows, T >= 9).
template <int T, int IT, int JT, int DYB>
__device__ __forceinline__ void job_tile(const LocalFwdParams& P, const float* __restrict__ xs,
                                         const float* __restrict__ ys, int i0, int j0, int dy0,
                                         float (&acc)[IT][JT][DYB][T]) {
  const int lane = threadIdx.x & 31;
  const int TW = P.TWS * 32;
  const float* xi[IT];
  const float* yj[JT];
#pragma unroll
  for (int ii = 0; ii < IT; ++ii) {
    int c = i0 + ii; c = c < P.Ki ? c : P.Ki - 1;          // clamp: padded jobs recompute a valid channel
    xi[ii] = xs + (size_t)c * P.XR * P.XP;
  }
#pragma unroll
  for (int jj = 0; jj < JT; ++jj) {
    int c = j0 + jj; c = c < P.Kj ? c : P.Kj - 1;
    yj[jj] = ys + (size_t)c * P.TH * TW;
  }
  for (int s = 0; s < P.TWS; ++s) {
    const int c = s * 32 + lane;
    if constexpr (DYB == T) {
      float xw[IT][T][T];
#pragma unroll
      for (int ii = 0; ii < IT; ++ii)
#pragma unroll
        for (int r = 0; r < T - 1; ++r)
#pragma unroll
          for (int dx = 0; dx < T; ++dx) xw[ii][r][dx] = xi[ii][r * P.XP + c + dx];
      for (int u0 = 0; u0 < P.TH; u0 += T) {
#pragma unroll
        for (int r = 0; r < T; ++r) {
          const int u = u0 + r;
          if (u < P.TH) {
#pragma unroll
            for (int ii = 0; ii < IT; ++ii)
#pragma unroll
              for (int dx = 0; dx < T; ++dx)
                xw[ii][(r + T - 1) % T][dx] = xi[ii][(u + T - 1) * P.XP + c + dx];
            float yv[JT];
#pragma unroll
            for (int jj = 0; jj < JT; ++jj) yv[jj] = yj[jj][u * TW + c];
#pragma unroll
            for (int ii = 0; ii < IT; ++ii)
#pragma unroll
              for (int jj = 0; jj < JT; ++jj)
#pragma unroll
                for (int dy = 0; dy < T; ++dy)
#pragma unroll
                  for (int dx = 0; dx < T; ++dx)
                    acc[ii][jj][dy][dx] = fmaf(xw[ii][(r + dy) % T][dx], yv[jj], acc[ii][jj][dy][dx]);
          }
        }
      }
    } else {
      for (int u = 0; u < P.TH; ++u) {
        float xr[IT][T];
#pragma unroll
        for (int ii = 0; ii < IT; ++ii)
#pragma unroll
          for (int dx = 0; dx < T; ++dx) xr[ii][dx] = xi[ii][(u + dy0) * P.XP + c + dx];
        float yv[JT];
#pragma unroll
        for (int jj = 0; jj < JT; ++jj) yv[jj] = yj[jj][u * TW + c];
#pragma unroll
        for (int ii = 0; ii < IT; ++ii)
#pragma unroll
          for (int jj = 0; jj < JT; ++jj)
#pragma unroll
            for (int dx = 0; dx < T; ++dx)
              acc[ii][jj][0][dx] = fmaf(xr[ii][dx], yv[jj], acc[ii][jj][0][dx]);
      }
    }
  }
}

// lanes -> one value per accumulator, then the owning warp adds it into this CTA's partial slot
template <int T, int IT, int JT, int DYB>
__device__ __forceinline__ void job_flush(const LocalFwdParams& P, float* slot, int i0, int j0, int dy0,
                                          float (&acc)[IT][JT][DYB][T], bool accumulate) {
  const int lane = threadIdx.x & 31;
  int a = 0;
#pragma unroll
  for (int ii = 0; ii < IT; ++ii)
#pragma unroll
    for (int jj = 0; jj < JT; ++jj)
#pragma unroll
      for (int dy = 0; dy < DYB; ++dy)
#pragma unroll
        for (int dx = 0; dx < T; ++dx) {
          const float v = warp_sum(acc[ii][jj][dy][dx]);
          acc[ii][jj][dy][dx] = 0.f;
          const int i = i0 + ii, j = j0 + jj;
          if (lane == (a & 31) && i < P.Ki && j < P.Kj) {
            float* dst = slot + ((size_t)((dy0 + dy) * T + dx) * P.K + (P.i_off + i)) * P.K + (P.j_off + j);
            *dst = accumulate ? *dst + v : v;
          }
          ++a;
        }
}

template <int T, int IT, int JT, int DYB>
__global__ void __launch_bounds__(384, 1) local_joint_kernel(const LocalFwdParams P) {
  extern __shared__ __align__(16) float smem[];
  float* xs = smem;
  float* ys = smem + (size_t)P.Ki * P.XR * P.XP;
  const int wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int patch = blockIdx.y;
  const int ph0 = patch_axis_origin(patch / P.g.nw, P.g.nh, P.g.H, P.g.ph, P.g.sh);
  const int pw0 = patch_axis_origin(patch % P.g.nw, P.g.nw, P.g.W, P.g.pw, P.g.sw);
  const int TW = P.TWS * 32;
  const int items = P.B * P.tiles_h * P.tiles_w;
  constexpr int NDY = T / DYB;
  float* slot = P.partial + ((size_t)patch * gridDim.x + blockIdx.x) * ((size_t)T * T * P.K * P.K);

  float acc[IT][JT][DYB][T];
#pragma unroll
  for (int ii = 0; ii < IT; ++ii)
#pragma unroll
    for (int jj = 0; jj < JT; ++jj)
#pragma unroll
      for (int dy = 0; dy < DYB; ++dy)
#pragma unroll
        for (int dx = 0; dx < T; ++dx) acc[ii][jj][dy][dx] = 0.f;

  // job decomposition: job = (ib, jb, dyb)
  auto decode = [&](int job, int& i0, int& j0, int& dy0) {
    const int dyb = job % NDY;
    const int t = job / NDY;
    j0 = (t % P.njobs_j) * JT;
    i0 = (t / P.njobs_j) * IT;
    dy0 = dyb * DYB;
  };

  const bool single_round = (P.rounds == 1);
  bool first_flush = true;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int n = it / (P.tiles_h * P.tiles_w);
    const int tt = it - n * (P.tiles_h * P.tiles_w);
    const int th0 = (tt / P.tiles_w) * P.TH, tw0 = (tt % P.tiles_w) * TW;
    __syncthreads();                      // previous tile fully consumed
    stage_tile(P, xs, ys, n, ph0, pw0, th0, tw0);
    __syncthreads();
    if (single_round) {
      if (wid < P.njobs) {
        int i0, j0, dy0;
        decode(wid, i0, j0, dy0);
        job_tile<T, IT, JT, DYB>(P, xs, ys, i0, j0, dy0, acc);
      }
    } else {
      for (int r = 0; r < P.rounds; ++r) {
        const int job = r * nwarps + wid;
        if (job < P.njobs) {
          int i0, j0, dy0;
          decode(job, i0, j0, dy0);
          job_tile<T, IT, JT, DYB>(P, xs, ys, i0, j0, dy0, acc);
          job_flush<T, IT, JT, DYB>(P, slot, i0, j0, dy0, acc, !first_flush);
        }
      }
      first_flush = false;
    }
  }
  if (single_round && wid < P.njobs) {
    int i0, j0, dy0;
    decode(wid, i0, j0, dy0);
    job_flush<T, IT, JT, DYB>(P, slot, i0, j0, dy0, acc, false);
  }
}

// J[p][e] = sum over CTAs of partial[p][cta][e] in float64, in a fixed order: a block is 32 slot groups x
// 32 consecutive elements (coalesced 128-byte reads); group g adds slots g, g+32, ... in order, then the 32
// group sums are added in order.
// TC_LAYOUT: the slots come from local_joint_tc_kernel (local_fwd_tc.cu) in its coalesced order
// [d][32-column chunk][float4 of the chunk][row i][4] with K = 128; J is written in the standard [d][i][j] order.
constexpr int RED_GROUPS = 32;
template <bool TC_LAYOUT>
__global__ void __launch_bounds__(RED_GROUPS * 32)
reduce_partials_kernel(const float* __restrict__ partial, int ncta, long long E, double* __restrict__ J) {
  __shared__ double sm[RED_GROUPS][33];
  const int le = threadIdx.x & 31, sg = threadIdx.x >> 5;
  const long long e = (long long)blockIdx.x * 32 + le;
  const int patch = blockIdx.y;
  double s[4] = {0, 0, 0, 0};
  if (e < E) {
    const float* src = partial + (size_t)patch * ncta * E + e;
    int c = sg;
    for (; c + 3 * RED_GROUPS < ncta; c += 4 * RED_GROUPS) {
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] += (double)__ldg(src + (size_t)(c + q * RED_GROUPS) * E);
    }
    for (int q = 0; c < ncta; c += RED_GROUPS, ++q) s[q] += (double)__ldg(src + (size_t)c * E);
  }
  sm[sg][le] = (s[0] + s[1]) + (s[2] + s[3]);
  __syncthreads();
  if (sg == 0 && e < E) {
    double t = 0;
#pragma unroll
    for (int g = 0; g < RED_GROUPS; ++g) t += sm[g][le];
    long long dst = e;
    if (TC_LAYOUT) {
      const long long w = e & 3, i = (e >> 2) & 127, jv = (e >> 9) & 7, ch = (e >> 12) & 3, d = e >> 14;
      dst = (d * 128 + i) * 128 + ch * 32 + jv * 4 + w;
    }
    J[(size_t)patch * E + dst] = t;
  }
}

// ---- host side ------------------------------------------------------------------------------------
struct FwdPlan {
  int T, IT, JT, DYB;
  int kchunk;        // channels per launch (<= 32)
  int TH, TWS, tiles_h, tiles_w, XR, XP;
  int ctas_per_patch;
  int slots_per_patch;
  int n_patches;
  size_t smem_bytes;
};

static void tile_shape_for(int T, int* IT, int* JT, int* DYB) {
  switch (T) {
    case 1: *IT = 4; *JT = 8; *DYB = 1; break;
    case 3: *IT = 2; *JT = 5; *DYB = 3; break;
    case 5: *IT = 1; *JT = 4; *DYB = 5; break;
    case 7: *IT = 1; *JT = 2; *DYB = 7; break;
    default: *IT = 1; *JT = 4; *DYB = 1; break;   // 9..15: one dy row per job
  }
}

static bool make_fwd_plan(int sms, int B, int K, const PatchGrid& g, int pad, FwdPlan* pl) {
  pl->T = 2 * pad + 1;
  if (pad < 0 || pad > 7) return false;
  tile_shape_for(pl->T, &pl->IT, &pl->JT, &pl->DYB);
  pl->kchunk = K <= 32 ? K : 32;
  pl->TWS = g.pw > 40 ? 2 : 1;
  const int TW = pl->TWS * 32;
  pl->XP = (TW + 2 * pad + 3) & ~3;
  // tile rows: as tall as a ~96 KB shared-memory budget allows, at most 32 and at most the patch
  int TH = 32;
  while (TH > 1) {
    size_t b = (size_t)pl->kchunk * ((size_t)(TH + 2 * pad) * pl->XP + (size_t)TH * TW) * sizeof(float);
    if (b <= 96 * 1024 && TH <= ((g.ph + 3) & ~3)) break;
    TH >>= 1;
  }
  pl->TH = TH;
  pl->XR = TH + 2 * pad;
  pl->tiles_h = (g.ph + TH - 1) / TH;
  pl->tiles_w = (g.pw + TW - 1) / TW;
  pl->smem_bytes = (size_t)pl->kchunk * ((size_t)pl->XR * pl->XP + (size_t)TH * TW) * sizeof(float);
  pl->n_patches = g.nh * g.nw;
  if (sms <= 0) return false;
  long long items = (long long)B * pl->tiles_h * pl->tiles_w;
  long long per = sms / pl->n_patches;
  if (per < 1) per = 1;
  pl->slots_per_patch = (int)per;          // workspace is sized for this many partial slots per patch
  if (per > items) per = items;
  pl->ctas_per_patch = (int)per;
  return true;
}

template <int T, int IT, int JT, int DYB>
static int launch_fwd(const LocalFwdParams& P, dim3 grid, int nthreads, size_t smem, cudaStream_t st) {
  auto kern = local_joint_kernel<T, IT, JT, DYB>;
  IIC_CHECK_RC(ensure_dyn_smem((const void*)(kern), (int)(200 * 1024)));
  kern<<<grid, nthreads, smem, st>>>(P);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// info == nullptr: reduce the per-CTA slots into J (fp64, fixed order) with the reduce kernel of their layout.
// info != nullptr: leave them in `partial` and describe them in *info (for iic_finish); J is unused.
static int reduce_or_describe_slots(const SlotInfo& s, const float* partial, int T, int K, int n_patches, double* J,
                                    iic_slot_info* info, cudaStream_t st) {
  if (info) {
    info->layout = s.layout;
    info->n_slots = s.n_slots;
    info->slot_stride = s.slot_stride;
    info->nb = s.nb;
    return 0;
  }
  if (s.layout == SLOT_PACKED) {
    const int E = T * T * K * K;
    fwdtcp::reduce_packed_kernel<<<(E + 31) / 32, 1024, 0, st>>>(partial, s.n_slots, (int)s.slot_stride, T, K, s.nb, J);
  } else {
    const dim3 rgrid((unsigned)((s.slot_stride + 31) / 32), n_patches);
    if (s.layout == SLOT_TC128)
      reduce_partials_kernel<true><<<rgrid, RED_GROUPS * 32, 0, st>>>(partial, s.n_slots, s.slot_stride, J);
    else
      reduce_partials_kernel<false><<<rgrid, RED_GROUPS * 32, 0, st>>>(partial, s.n_slots, s.slot_stride, J);
  }
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace iic

using namespace iic;

extern "C" int iic_local_num_patches(int H, int W, int patch_h, int patch_w, int step_h, int step_w) {
  PatchGrid g;
  if (!make_patch_grid(H, W, patch_h, patch_w, step_h, step_w, &g)) {
    set_error("iic_local_num_patches: bad patch geometry H=%d W=%d patch=(%d,%d) step=(%d,%d)", H, W,
              patch_h, patch_w, step_h, step_w);
    return -1;
  }
  return g.nh * g.nw;
}

extern "C" size_t iic_local_joint_workspace_bytes(int device, int B, int K, int H, int W, int pad,
                                                  int patch_h, int patch_w, int step_h, int step_w) {
  PatchGrid g;
  FwdPlan pl;
  if (!make_patch_grid(H, W, patch_h, patch_w, step_h, step_w, &g)) return 0;
  if (!make_fwd_plan(sm_count_cached(device), B, K, g, pad, &pl)) return 0;
  size_t bytes = (size_t)pl.n_patches * pl.slots_per_patch * pl.T * pl.T * K * K * sizeof(float);
  // the packed tensor-core joint (local_fwd_tcp.cu) keeps whole accumulator tiles per CTA slot
  const size_t tcp = local_joint_tcp_slot_floats(K, pad) * (size_t)pl.slots_per_patch * sizeof(float);
  if (pl.n_patches == 1 && tcp > bytes) bytes = tcp;
  return bytes;
}

static int local_joint_impl(const float* x, long long x_sn, long long x_sc, long long x_sh,
                            const float* y, long long y_sn, long long y_sc, long long y_sh,
                            const float* mask, long long m_sn, long long m_sc, long long m_sh,
                            int B, int K, int H, int W, int pad,
                            int patch_h, int patch_w, int step_h, int step_w,
                            double* J_out, void* workspace, size_t workspace_bytes, int* flags,
                            iic_slot_info* info, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(x && y && (J_out || info), "iic_local_joint: null pointer");
  IIC_REQUIRE(!flags || x_sh == W, "iic_local_joint: the fused simplex assertion needs dense rows (x_sh == W)");
  IIC_REQUIRE(B > 0 && K > 0, "iic_local_joint: empty batch or channel dimension (B=%d K=%d)", B, K);
  IIC_REQUIRE(pad >= 0 && pad <= 7, "iic_local_joint: padding %d unsupported (0..7)", pad);
  PatchGrid g;
  IIC_REQUIRE(make_patch_grid(H, W, patch_h, patch_w, step_h, step_w, &g),
              "iic_local_joint: bad patch geometry H=%d W=%d patch=(%d,%d) step=(%d,%d)", H, W, patch_h,
              patch_w, step_h, step_w);
  const int sms = sm_count_cached(current_device());
  FwdPlan pl;
  IIC_REQUIRE(make_fwd_plan(sms, B, K, g, pad, &pl), "iic_local_joint: cannot plan launch");
  const size_t E = (size_t)pl.T * pl.T * K * K;
  const size_t need = (size_t)pl.n_patches * pl.slots_per_patch * E * sizeof(float);
  IIC_REQUIRE(workspace && workspace_bytes >= need, "iic_local_joint: workspace too small (%zu < %zu)",
              workspace_bytes, need);
  float* partial = (float*)workspace;

  // simplex assertion on x when the joint kernel chosen below cannot fuse it: one streaming pass
  auto simplex_pass = [&]() -> int {
    if (!flags) return 0;
    return iic_simplex_check(x, B, K, (long long)H * W, x_sn, x_sc, flags, stream);
  };

  // fast path: one patch, no mask, TMA-describable rows -> the specialised kernels (local_kernels.cuh)
  if (pl.n_patches == 1 && mask == nullptr && !options().no_tma) {
    const LocalMaps m{{x, x_sn, x_sc, x_sh}, {y, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
    SlotInfo slots{};
    int rc = -1, checked = 0;
    // the reference's default cluster count (16 <= K <= 24), padding 3: packed tensor-core joint (local_fwd_tcp.cu);
    // padding 1 stays on the FFMA2 kernel unless IIC_B200_TCP_P1 is set
    if (!options().no_tc && (pad == 3 || options().tcp_p1))
      rc = local_joint_tcp_try(m, partial, workspace_bytes / sizeof(float), &slots, st);
    // wide cluster heads (K = 128): tcgen05 3xTF32 contraction (local_fwd_tc.cu)
    if (rc < 0 && !options().no_tc)
      rc = local_joint_tc_try(m, partial, pl.slots_per_patch, &slots, st);
    // 10 clusters, 3 x 3 window, large maps (BASELINE config 2): fp16-split tensor-core joint (local_fwd_tcj10.cu)
    if (rc < 0 && !options().no_tc && !options().no_tcj10 && sms <= pl.slots_per_patch)
      rc = local_joint_tcj10_try(m, partial, sms, &slots, flags, &checked, 0, 1.f, st);
    if (rc < 0 && !options().no_fast)
      rc = local_joint_fast_try(m, partial, pl.slots_per_patch, &slots, flags, &checked, 0, 1.f, st);
    if (rc < 0 && !options().no_fast)
      rc = local_joint_fast7_try(m, partial, pl.slots_per_patch, &slots, st);
    if (rc < 0)
      rc = local_joint_tma_try(m, partial, pl.slots_per_patch, &slots, st);
    if (rc > 0) return rc;
    if (rc == 0) {
      if (checked) flags = nullptr;       // done inside the joint kernel
      if (int e = simplex_pass()) return e;
      return reduce_or_describe_slots(slots, partial, pl.T, K, 1, J_out, info, st);
    }
  }

  if (int e = simplex_pass()) return e;
  LocalFwdParams P;
  P.x = {x, x_sn, x_sc, x_sh};
  P.y = {y, y_sn, y_sc, y_sh};
  P.m = {mask, m_sn, m_sc, m_sh};
  P.B = B; P.K = K; P.pad = pad; P.g = g;
  P.TH = pl.TH; P.TWS = pl.TWS; P.tiles_h = pl.tiles_h; P.tiles_w = pl.tiles_w;
  P.XR = pl.XR; P.XP = pl.XP;
  P.partial = partial;
  const int NDY = pl.T / pl.DYB;
  dim3 grid(pl.ctas_per_patch, pl.n_patches);

  for (int i_off = 0; i_off < K; i_off += pl.kchunk) {
    for (int j_off = 0; j_off < K; j_off += pl.kchunk) {
      P.i_off = i_off; P.j_off = j_off;
      P.Ki = K - i_off < pl.kchunk ? K - i_off : pl.kchunk;
      P.Kj = K - j_off < pl.kchunk ? K - j_off : pl.kchunk;
      P.njobs_i = (P.Ki + pl.IT - 1) / pl.IT;
      P.njobs_j = (P.Kj + pl.JT - 1) / pl.JT;
      P.njobs = P.njobs_i * P.njobs_j * NDY;
      // warps per CTA: one job per warp when that fits in 12 warps, else the count in [6,12] that
      // leaves the fewest idle warp-rounds
      int nw = P.njobs;
      if (nw > 12) {
        int best = 12; double best_eff = 0.0;
        for (int c = 12; c >= 6; --c) {
          int r = (P.njobs + c - 1) / c;
          double eff = (double)P.njobs / ((double)r * c);
          if (eff > best_eff + 1e-9) { best_eff = eff; best = c; }
        }
        nw = best;
      }
      P.rounds = (P.njobs + nw - 1) / nw;
      int rc = 0;
      const int nt = nw * 32;
      switch (pl.T) {
        case 1:  rc = launch_fwd<1, 4, 8, 1>(P, grid, nt, pl.smem_bytes, st); break;
        case 3:  rc = launch_fwd<3, 2, 5, 3>(P, grid, nt, pl.smem_bytes, st); break;
        case 5:  rc = launch_fwd<5, 1, 4, 5>(P, grid, nt, pl.smem_bytes, st); break;
        case 7:  rc = launch_fwd<7, 1, 2, 7>(P, grid, nt, pl.smem_bytes, st); break;
        case 9:  rc = launch_fwd<9, 1, 4, 1>(P, grid, nt, pl.smem_bytes, st); break;
        case 11: rc = launch_fwd<11, 1, 4, 1>(P, grid, nt, pl.smem_bytes, st); break;
        case 13: rc = launch_fwd<13, 1, 4, 1>(P, grid, nt, pl.smem_bytes, st); break;
        case 15: rc = launch_fwd<15, 1, 4, 1>(P, grid, nt, pl.smem_bytes, st); break;
        default: IIC_REQUIRE(false, "iic_local_joint: unsupported window %d", pl.T);
      }
      if (rc) return rc;
    }
  }
  return reduce_or_describe_slots(SlotInfo{SLOT_STD, pl.ctas_per_patch, (long long)E, 0}, partial, pl.T, K,
                                  pl.n_patches, J_out, info, st);
}

extern "C" int iic_local_joint(const float* x, long long x_sn, long long x_sc, long long x_sh,
                               const float* y, long long y_sn, long long y_sc, long long y_sh,
                               const float* mask, long long m_sn, long long m_sc, long long m_sh,
                               int B, int K, int H, int W, int pad,
                               int patch_h, int patch_w, int step_h, int step_w,
                               double* J_out, void* workspace, size_t workspace_bytes, int* flags,
                               void* stream) {
  IIC_REQUIRE(J_out, "iic_local_joint: null pointer");
  return local_joint_impl(x, x_sn, x_sc, x_sh, y, y_sn, y_sc, y_sh, mask, m_sn, m_sc, m_sh, B, K, H, W, pad, patch_h,
                          patch_w, step_h, step_w, J_out, workspace, workspace_bytes, flags, nullptr, stream);
}

extern "C" int iic_local_joint_partials(const float* x, long long x_sn, long long x_sc, long long x_sh,
                                        const float* y, long long y_sn, long long y_sc, long long y_sh,
                                        const float* mask, long long m_sn, long long m_sc, long long m_sh,
                                        int B, int K, int H, int W, int pad,
                                        int patch_h, int patch_w, int step_h, int step_w,
                                        void* workspace, size_t workspace_bytes, int* flags,
                                        iic_slot_info* info_host, void* stream) {
  IIC_REQUIRE(info_host, "iic_local_joint_partials: null pointer");
  return local_joint_impl(x, x_sn, x_sc, x_sh, y, y_sn, y_sc, y_sh, mask, m_sn, m_sc, m_sh, B, K, H, W, pad, patch_h,
                          patch_w, step_h, step_w, nullptr, workspace, workspace_bytes, flags, info_host, stream);
}

// Fused cluster-head softmax + local joint: only the shapes the fast kernel covers
extern "C" int iic_local_joint_from_logits(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                           const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                           int B, int K, int H, int W, int pad, float inv_temperature,
                                           double* J_out, void* workspace, size_t workspace_bytes,
                                           iic_slot_info* info_host, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(lx && ly && (J_out || info_host) && workspace, "iic_local_joint_from_logits: null pointer");
  IIC_REQUIRE(B > 0 && K > 0 && H > 0 && W > 0, "iic_local_joint_from_logits: empty input");
  const int sms = sm_count_cached(current_device());
  IIC_REQUIRE(sms > 0, "iic_local_joint_from_logits: no device");
  const size_t E = (size_t)9 * K * K;
  IIC_REQUIRE(workspace_bytes >= (size_t)sms * E * sizeof(float),
              "iic_local_joint_from_logits: workspace too small (%zu < %zu)", workspace_bytes,
              (size_t)sms * E * sizeof(float));
  const LocalMaps m{{lx, x_sn, x_sc, x_sh}, {ly, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
  float* partial = (float*)workspace;
  SlotInfo slots{};
  int rc = -1, checked = 0;
  // large maps: the tensor-core joint with the softmax in its staging warps (csrc/local_fwd_tcj10.cu); else the FFMA2 kernel
  if (!options().no_tc && !options().no_tcj10 && pad == 1)
    rc = local_joint_tcj10_try(m, partial, sms, &slots, nullptr, &checked, 1, inv_temperature, st);
  if (rc < 0)
    rc = local_joint_fast_try(m, partial, sms, &slots, nullptr, &checked, 1, inv_temperature, st);
  if (rc < 0) {
    set_error("iic_local_joint_from_logits: shape not covered by the fused kernel (needs padding 1, K == 10, "
              "W %% 4 == 0, 16-byte aligned rows); apply the softmax and call iic_local_joint");
    return IIC_UNSUPPORTED;
  }
  if (rc > 0) return rc;
  return reduce_or_describe_slots(slots, partial, 3, K, 1, J_out, info_host, st);
}

// Fused cluster-head softmax + local joint with caller-owned per-pixel stats: 16 <= K <= 24 where local_fl_tc_covered
// holds (stats pass, then the packed tensor-core joint on the logits), K = 128 where local_fl_tc128_covered holds (stats
// pass, then the tc joint on the logits); the K = 10 shapes of iic_local_joint_from_logits as there (stats untouched)
extern "C" int iic_local_joint_from_logits_stats(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                                 const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                                 int B, int K, int H, int W, int pad, float inv_temperature, float* stats,
                                                 double* J_out, void* workspace, size_t workspace_bytes,
                                                 iic_slot_info* info_host, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IIC_REQUIRE(lx && ly && (J_out || info_host) && workspace, "iic_local_joint_from_logits_stats: null pointer");
  IIC_REQUIRE(B > 0 && K > 0 && H > 0 && W > 0, "iic_local_joint_from_logits_stats: empty input");
  const int sms = sm_count_cached(current_device());
  IIC_REQUIRE(sms > 0, "iic_local_joint_from_logits_stats: no device");
  const LocalMaps m{{lx, x_sn, x_sc, x_sh}, {ly, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
  const bool wide = local_fl_tc128_covered(m);
  if (!wide && K == 128) {
    // (the workspace was sized for the tc joint's slots, not for the per-SM slots the K = 10 entry checks first)
    set_error("iic_local_joint_from_logits_stats: K = 128 is fused at padding 1, W %% 16 == 0, W <= 248, 16-byte aligned "
              "rows; apply the softmax and call iic_local_joint");
    return IIC_UNSUPPORTED;
  }
  if (!wide && !local_fl_tc_covered(m))
    return iic_local_joint_from_logits(lx, x_sn, x_sc, x_sh, ly, y_sn, y_sc, y_sh, B, K, H, W, pad, inv_temperature, J_out,
                                       workspace, workspace_bytes, info_host, stream);
  IIC_REQUIRE(stats && (reinterpret_cast<uintptr_t>(stats) & 15) == 0,
              "iic_local_joint_from_logits_stats: stats must be a 16-byte aligned buffer of iic_local_logit_stats_floats");
  if (wide) {
    const int max_ctas = local_fl_tc128_slots(sms);
    const size_t need = (size_t)max_ctas * 9 * K * K * sizeof(float);
    IIC_REQUIRE(workspace_bytes >= need, "iic_local_joint_from_logits_stats: workspace too small (%zu < %zu)",
                workspace_bytes, need);
    if (int e = local_logit_stats(m, inv_temperature, stats, st)) return e;
    SlotInfo slots{};
    const int rc = local_joint_tc_fl_try(m, stats, inv_temperature, (float*)workspace, max_ctas, &slots, st);
    if (rc > 0) return rc;
    IIC_REQUIRE(rc == 0, "iic_local_joint_from_logits_stats: the tensor-core joint refused a covered shape");
    return reduce_or_describe_slots(slots, (const float*)workspace, 3, K, 1, J_out, info_host, st);
  }
  const size_t need = (size_t)sms * local_joint_tcp_slot_floats(K, pad) * sizeof(float);
  IIC_REQUIRE(workspace_bytes >= need, "iic_local_joint_from_logits_stats: workspace too small (%zu < %zu)",
              workspace_bytes, need);
  if (int e = local_logit_stats(m, inv_temperature, stats, st)) return e;
  SlotInfo slots{};
  const int rc = local_joint_tcp_fl_try(m, stats, inv_temperature, (float*)workspace, workspace_bytes / sizeof(float),
                                        &slots, st);
  if (rc > 0) return rc;
  IIC_REQUIRE(rc == 0, "iic_local_joint_from_logits_stats: the packed tensor-core joint refused a covered shape");
  return reduce_or_describe_slots(slots, (const float*)workspace, 2 * pad + 1, K, 1, J_out, info_host, st);
}
