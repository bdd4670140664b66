// The specialised kernel families of the local IIC term: one declaration per family, called by the dispatchers in
// local_fwd.cu (joints) and local_bwd.cu (backwards).  The generic kernels live in the dispatchers themselves.
//
// Every *_try returns 0 when it launched its kernel(s), < 0 when the shape is not covered (the dispatcher tries the
// next family), > 0 on error (the message is in get_error()).
#pragma once
#include "common.cuh"
#include "tma.cuh"

namespace iic {

// What every family reads: the two (B, K, H, W) maps (probabilities, or logits for the from-logits forms), the window
// padding and the SM count the dispatcher queried (> 0).
struct LocalMaps {
  View4 x, y;
  int B, K, H, W, pad;
  int sms;
};

// What every backward writes: dL/dx and dL/dy (channel planes and rows dense, sample strides gx_sn / gy_sn), scaled by
// the device scalar grad_loss (nullptr: 1).
struct LocalGrads {
  const float* grad_loss;
  float* gx;
  float* gy;
  long long gx_sn, gy_sn;
};

// Tensor map of one of the maps (m.x or m.y) over the full (B, K, H, W) extent of the term.
inline bool make_map_4d(CUtensorMap* map, const View4& v, const LocalMaps& m, int box_w, int box_h, int box_c,
                        CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_NONE) {
  return make_map_4d(map, v.p, m.B, m.K, m.H, m.W, v.sn, v.sc, v.sh, box_w, box_h, box_c, swz);
}

// ---- joints: per-CTA partial slots in `partial`, described in *slots (reduced by the dispatcher or by iic_finish) ----
// flags / checked: when flags is given and the kernel ran the simplex assertion on x itself, *checked = 1.
// from_logits: x and y are logits; the kernel applies softmax(logit * inv_temp) while staging.
int local_joint_tma_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st);
int local_joint_fast_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, int* flags, int* checked,
                         int from_logits, float inv_temp, cudaStream_t st);
int local_joint_fast7_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st);
int local_joint_tc_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, cudaStream_t st);
// its from-logits form (K = 128): `stats` holds the per-pixel (m, r) of both maps (local_logit_stats, local_logits.cu)
int local_joint_tc_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, int max_ctas,
                          SlotInfo* slots, cudaStream_t st);
int local_joint_tcj10_try(const LocalMaps& m, float* partial, int max_ctas, SlotInfo* slots, int* flags, int* checked,
                          int from_logits, float inv_temp, cudaStream_t st);
int local_joint_tcp_try(const LocalMaps& m, float* partial, size_t partial_floats, SlotInfo* slots, cudaStream_t st);
// its from-logits form: `stats` holds the per-pixel (m, r) of both maps (local_logit_stats, local_logits.cu)
int local_joint_tcp_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* partial, size_t partial_floats,
                           SlotInfo* slots, cudaStream_t st);
// floats of one slot of the packed tensor-core joint (0 when it does not cover (K, pad)); the workspace is sized for it
size_t local_joint_tcp_slot_floats(int K, int pad);
namespace fwdtcp {
// SLOT_PACKED slots -> J[dy][dx][i][j] in fp64 (local_fwd_tcp.cu)
__global__ void reduce_packed_kernel(const float* __restrict__ partial, int ncta, int slot_floats, int T, int K, int nb,
                                     double* __restrict__ J);
}

// ---- backwards: Wx / Wy are the coefficient buffers of iic_local_epilogue (layout in common.cuh) ----
// The tc and tcrb families write their operand-order weight image into the buffers' tail, hence float*.
int local_bwd_tma_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, cudaStream_t st);
int local_bwd_fast_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, int from_logits,
                       float inv_temp, cudaStream_t st);
int local_bwd_tc_try(const LocalMaps& m, float* Wx, float* Wy, const LocalGrads& g, cudaStream_t st);
int local_bwd_tc_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* Wx, float* Wy, const LocalGrads& g,
                        cudaStream_t st);
int local_bwd_tcrb_try(const LocalMaps& m, float* Wx, float* Wy, const LocalGrads& g, cudaStream_t st);
int local_bwd_tcrb_fl_try(const LocalMaps& m, const float* stats, float inv_temp, float* Wx, float* Wy, const LocalGrads& g,
                          cudaStream_t st);
// the tcrb family's work split (false: not covered) and its padding-1 gate ("enough row blocks to fill the SMs")
bool local_bwd_tcrb_plan(int B, int K, int H, int W, int pad, int* PW, int* npanel, int* R, int* n_items);
bool local_bwd_tcrb_p1_gate(int n_items, int sms);
int local_bwd_tcrb10_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, cudaStream_t st);
int local_bwd_tcrb10h_try(const LocalMaps& m, const float* Wx, const float* Wy, const LocalGrads& g, int from_logits,
                          float inv_temp, cudaStream_t st);
// bytes of the weight image in the coefficient buffers' tail (0 when the family does not cover (K, pad))
size_t local_bwd_tc_image_bytes(int K, int pad);      // K = 128, padding 1
size_t local_bwd_tcrb_image_bytes(int K, int pad);    // 16 <= K <= 24, padding 1 or 3

// ---- from logits with per-pixel stats: 16 <= K <= 24 and K = 128 (local_logits.cu) ----
// THE rules that decide whether such a term runs fused, used by both entry points and by iic_local_from_logits_covered:
// 16 <= K <= 24 (tcp joint + tcrb backward on logits) and K = 128 (tc joint + tc backward on logits)
bool local_fl_tc_covered(const LocalMaps& m);
bool local_fl_tc128_covered(const LocalMaps& m);
// joints the wide heads' from-logits joint may spread over (its grid is SMs / 3 shares x 3 displacement rows)
int local_fl_tc128_slots(int sms);
// (m, r) of every pixel of both maps into stats = [2B][2][H][W] (x at n, y at B + n)
int local_logit_stats(const LocalMaps& m, float inv_temp, float* stats, cudaStream_t st);

}  // namespace iic
