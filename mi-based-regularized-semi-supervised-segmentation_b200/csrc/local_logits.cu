// The cluster head's softmax fused into the local IIC term for the reference's default cluster count (16 <= K <= 24)
// and the wide heads (K = 128, padding 1; contrastyou/trainer/_utils.py:15-23,137-168 feeding iic_loss.py:107-149):
// per-pixel softmax statistics, the coverage rules and the size queries of the from-logits entry points.
//
// The tensor-core kernels of these K never hold all K channels of a pixel at once while they stage it (8-channel
// slices, or one channel row per thread), so they cannot normalise by themselves.  One streaming pass writes, per pixel of both maps,
//   m = max_k (l_k * inv_temp)      r = 1 / sum_k exp(l_k * inv_temp - m)
// and every consumer computes p = exp(l * inv_temp - m) * r with the same fp32 product l * inv_temp (__fmul_rn: never
// contracted into an FMA).  (m, r) rather than one log-sum-exp: with T = 0.1 the scaled logits reach a few hundred, and
// an fp32 LSE subtracted there costs ~1e-5 relative in p, the whole loss tolerance.
#include "common.cuh"
#include "local_kernels.cuh"

namespace iic {

constexpr int STATS_THREADS = 256;

// stats = [2B][2][H][W]: plane 0 = m, plane 1 = r; map 0 (x) at samples 0..B-1, map 1 (y) at B..2B-1.  4 pixels per
// thread, 16-byte loads (W % 4 == 0 and 16-byte aligned rows); blockIdx.y = map * B + sample.
__global__ void __launch_bounds__(STATS_THREADS)
local_logit_stats_kernel(const View4 x, const View4 y, int B, int K, int H, int W, float inv_temp, float* __restrict__ stats) {
  const int map = blockIdx.y >= B ? 1 : 0, n = blockIdx.y - map * B;
  const View4 v = map ? y : x;
  const int quads = H * W / 4;
  const float* base = v.p + (long long)n * v.sn;
  float* out = stats + (long long)blockIdx.y * 2 * H * W;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += gridDim.x * blockDim.x) {
    const int pix = q * 4, h = pix / W, w = pix - h * W;
    const float* src = base + (long long)h * v.sh + w;
    float4 mx = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    for (int k = 0; k < K; ++k) {
      const float4 l = __ldg(reinterpret_cast<const float4*>(src + (long long)k * v.sc));
      mx.x = fmaxf(mx.x, __fmul_rn(l.x, inv_temp));
      mx.y = fmaxf(mx.y, __fmul_rn(l.y, inv_temp));
      mx.z = fmaxf(mx.z, __fmul_rn(l.z, inv_temp));
      mx.w = fmaxf(mx.w, __fmul_rn(l.w, inv_temp));
    }
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < K; ++k) {
      const float4 l = __ldg(reinterpret_cast<const float4*>(src + (long long)k * v.sc));
      s.x += __expf(__fmul_rn(l.x, inv_temp) - mx.x);
      s.y += __expf(__fmul_rn(l.y, inv_temp) - mx.y);
      s.z += __expf(__fmul_rn(l.z, inv_temp) - mx.z);
      s.w += __expf(__fmul_rn(l.w, inv_temp) - mx.w);
    }
    *reinterpret_cast<float4*>(out + pix) = mx;
    *reinterpret_cast<float4*>(out + H * W + pix) = make_float4(1.f / s.x, 1.f / s.y, 1.f / s.z, 1.f / s.w);
  }
}

int local_logit_stats(const LocalMaps& m, float inv_temp, float* stats, cudaStream_t st) {
  const int quads = m.H * m.W / 4;
  int blocks = (quads + STATS_THREADS - 1) / STATS_THREADS;
  const int cap = (8 * m.sms + 2 * m.B - 1) / (2 * m.B);          // ~8 blocks per SM over all (map, sample) rows
  if (blocks > cap) blocks = cap > 0 ? cap : 1;
  local_logit_stats_kernel<<<dim3((unsigned)blocks, 2 * m.B), STATS_THREADS, 0, st>>>(m.x, m.y, m.B, m.K, m.H, m.W, inv_temp,
                                                                                     stats);
  IIC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static bool rows16(const View4& v) {
  return (reinterpret_cast<uintptr_t>(v.p) & 15) == 0 && (v.sn * 4) % 16 == 0 && (v.sc * 4) % 16 == 0 && (v.sh * 4) % 16 == 0;
}

// 16 <= K <= 24 from logits is fused (packed tensor-core joint + row-block tensor-core backward, both converting logits
// with the stats) when: padding 3, or padding 1 where the row-block backward's "enough row blocks to fill the SMs" gate
// holds; W % 16 == 0 (the joint's 16-pixel k-blocks); 16-byte aligned rows of both maps; the tensor-core and TMA kernels
// not switched off.  One patch and no mask are the from-logits entry points' own terms.
bool local_fl_tc_covered(const LocalMaps& m) {
  if (options().no_tc || options().no_tma) return false;
  if (m.K < 16 || m.K > 24 || (m.pad != 1 && m.pad != 3)) return false;
  if (m.B < 1 || m.H < 1 || m.W < 16 || m.W % 16 != 0 || m.sms < 1) return false;
  if (!rows16(m.x) || !rows16(m.y)) return false;
  int PW, npanel, R, n_items;
  if (!local_bwd_tcrb_plan(m.B, m.K, m.H, m.W, m.pad, &PW, &npanel, &R, &n_items)) return false;
  if (m.pad == 1 && !local_bwd_tcrb_p1_gate(n_items, m.sms)) return false;
  return true;
}

// K = 128 from logits is fused (tc joint + tc backward, both converting logits with the stats) when: padding 1;
// W % 16 == 0 (the joint's 16-pixel k-blocks); 8 <= W <= 248 (the backward stages W + 8 columns in one TMA box);
// 16-byte aligned rows of both maps; the tensor-core and TMA kernels not switched off.
bool local_fl_tc128_covered(const LocalMaps& m) {
  if (options().no_tc || options().no_tma) return false;
  if (m.K != 128 || m.pad != 1) return false;
  if (m.B < 1 || m.H < 1 || m.W < 16 || m.W % 16 != 0 || m.W > 248 || m.sms < 1) return false;
  return rows16(m.x) && rows16(m.y);
}

int local_fl_tc128_slots(int sms) { return sms / 3 > 0 ? sms / 3 : 1; }

// the K = 10 fused kernels' shapes, as include/iic_b200.h states them (local_fwd_fast3.inc, local_bwd_fast.cu)
static bool fl10_covered(const LocalMaps& m) {
  return m.K == 10 && m.pad == 1 && m.W % 4 == 0 && m.W >= 4 && m.W <= 248 && rows16(m.x) && rows16(m.y);
}

}  // namespace iic

using namespace iic;

extern "C" size_t iic_local_logit_stats_floats(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)4 * B * H * W;
}

extern "C" size_t iic_local_joint_from_logits_workspace_bytes(int device, int B, int K, int H, int W, int pad) {
  const int sms = sm_count_cached(device);
  if (sms <= 0 || B <= 0 || K <= 0 || H <= 0 || W <= 0) return 0;
  const size_t tcp = local_joint_tcp_slot_floats(K, pad);
  if (tcp) return (size_t)sms * tcp * sizeof(float);
  // K = 128: one [9][128][128] slot per share of the tc joint
  if (K == 128 && pad == 1) return (size_t)local_fl_tc128_slots(sms) * 9 * K * K * sizeof(float);
  return (size_t)sms * 9 * K * K * sizeof(float);
}

extern "C" int iic_local_from_logits_covered(int device, const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                             const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                             int B, int K, int H, int W, int pad) {
  const int sms = sm_count_cached(device);
  if (sms <= 0) {
    set_error("iic_local_from_logits_covered: no device %d", device);
    return -1;
  }
  const LocalMaps m{{lx, x_sn, x_sc, x_sh}, {ly, y_sn, y_sc, y_sh}, B, K, H, W, pad, sms};
  return (local_fl_tc_covered(m) || local_fl_tc128_covered(m) || fl10_covered(m)) ? 1 : 0;
}
