/*
 * iic_b200.h -- C ABI of libiic_b200.so: the B200 (sm_100a) kernels behind the IIC
 * mutual-information losses and the UDA consistency term.
 *
 * The reference (jizongFox/MI-based-Regularized-Semi-supervised-Segmentation) is pure Python and has
 * no FFI of its own; the boundary it exposes is the loss-module API in
 * contrastyou/losses/iic_loss.py.  Each entry point below states which reference lines it replaces.
 * The Python host (package dir, ops.py) binds these with ctypes and wraps them as torch custom ops;
 * INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors are float32, innermost (W, or K for the (N,K) global case) stride 1, other strides
 *     given in ELEMENTS;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - return value 0 = ok, non-zero = error (never throws); iic_b200_last_error() gives the text of
 *     the calling thread's last error;
 *   - no entry point has a CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef IIC_B200_H_
#define IIC_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IIC_B200_ABI_VERSION 10

/* flag bits written (OR-ed) into the int* `flags` words by the kernels */
#define IIC_FLAG_NAN_LOSS 1      /* iic_loss.py:147-148,184-185 -> RuntimeError on the host  */
#define IIC_FLAG_NOT_SIMPLEX 2   /* dc2:utils/assertion.py:56-65 -> AssertionError on the host */
#define IIC_FLAG_BAD_LABEL 4     /* dc2:utils/assertion.py:101-116 class2one_hot `assert sset(seg, range(C))` -> AssertionError */
#define IIC_FLAG_XCHG_TIMEOUT 8  /* multi-GPU: a peer never published its joints within xchg_timeout_ms -> RuntimeError */

/* return code of the *_from_logits entry points for shapes their fused kernels do not cover */
#define IIC_UNSUPPORTED 3

int iic_b200_abi_version(void);
const char* iic_b200_last_error(void);
/* number of SMs of `device` (148 on B200); <0 on error */
int iic_b200_sm_count(int device);
/* Dispatch switches.  The library reads IIC_B200_* environment variables ONCE (at first use) as defaults; after that
 * only these calls change them.  Names: "no_tma", "no_tc", "no_tc10", "no_tcj10", "no_fast" (skip a kernel family),
 * "tcp_p1", "tcrb_p1", "tc10_force" (force a tensor-core kernel outside the shapes it is normally chosen for),
 * "tc10_tf32" (the tf32 + bf16-correction form of the K = 10 backward instead of the fp16-split one),
 * "no_fused_epilogue" (per-term epilogue launches), "fin_last_cta_epilogue" (a small batch's epilogues inside the finish
 * launch instead of the batched epilogue launch), "xchg_timeout_ms".  Results are the same whatever the switches; only the kernel that runs changes (the parity tests
 * use them to reach every dispatch branch).  set: 0 = ok; get: the value, -1 for an unknown name. */
int iic_b200_set_option(const char* name, int value);
int iic_b200_get_option(const char* name);

/* ------------------------------------------------------------------------------------------------
 * simplex assertion: flags |= IIC_FLAG_NOT_SIMPLEX unless |sum_c t[o,c,i] - 1| <= 2e-4 everywhere
 * (NaN fails).  t is viewed as (outer, C, inner) with element strides (s_outer, s_c, 1).
 * Replaces dc2:deepclustering2/utils/assertion.py:56-65 as called at iic_loss.py:50-51,82-83,113.
 * ---------------------------------------------------------------------------------------------- */
int iic_simplex_check(const float* t, long long outer, int C, long long inner,
                      long long s_outer, long long s_c, int* flags, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Local (shifted-window) IIC.  Replaces IIDSegmentationLoss.__call__ (iic_loss.py:107-149) and the
 * patch loop of IIDSegmentationSmallPathLoss.__call__ (iic_loss.py:171-186).
 *
 * Patches follow patch_generator (iic_loss.py:152-160): windows of (patch_h, patch_w) at steps
 * (step_h, step_w) plus a last window flush with the border; patch_h >= H and patch_w >= W means one
 * window = the whole map.  iic_local_num_patches returns how many windows that is.
 * T = 2*pad + 1.  J is laid out [patch][dy][dx][i][j] (the reference's conv output permuted as at
 * iic_loss.py:127).
 * ---------------------------------------------------------------------------------------------- */
int iic_local_num_patches(int H, int W, int patch_h, int patch_w, int step_h, int step_w);

/* bytes of scratch iic_local_joint needs (per-CTA partial joints) */
size_t iic_local_joint_workspace_bytes(int device, int B, int K, int H, int W, int pad,
                                       int patch_h, int patch_w, int step_h, int step_w);

/* J[patch][dy][dx][i][j] = sum_{n,u,v} x[n,i,u+dy-pad,v+dx-pad] * y[n,j,u,v]  over the patch, x zero
 * outside the patch (iic_loss.py:120-123, the F.conv2d).  mask (nullable; (B,1|K,H,W), m_sc = 0 for
 * one channel) multiplies both maps first (iic_loss.py:116-118).  Partial sums are fp32 inside one
 * CTA, combined across CTAs in fp64 in a fixed order (deterministic). J_out is float64.
 * flags (nullable): also run the simplex assertion of iic_loss.py:113 on x (needs x_sh == W); it is
 * fused into the joint kernel where that kernel holds all K channels of a pixel, else one extra pass. */
int iic_local_joint(const float* x, long long x_sn, long long x_sc, long long x_sh,
                    const float* y, long long y_sn, long long y_sc, long long y_sh,
                    const float* mask, long long m_sn, long long m_sc, long long m_sh,
                    int B, int K, int H, int W, int pad,
                    int patch_h, int patch_w, int step_h, int step_w,
                    double* J_out, void* workspace, size_t workspace_bytes, int* flags, void* stream);

/* iic_local_joint without the cross-CTA reduction: the joint kernel's per-CTA partial sums stay in `workspace`
 * (same size as for iic_local_joint) and *info_host says how they are laid out; iic_finish (below) reduces them -- for
 * many loss terms at once -- and runs the epilogues.  Everything else as iic_local_joint. */
typedef struct iic_slot_info {
  int layout;              /* opaque: pass through to iic_finish_item */
  int n_slots;             /* per-CTA slots per patch */
  long long slot_stride;   /* floats between slots */
  int nb;
} iic_slot_info;
int iic_local_joint_partials(const float* x, long long x_sn, long long x_sc, long long x_sh,
                             const float* y, long long y_sn, long long y_sc, long long y_sh,
                             const float* mask, long long m_sn, long long m_sc, long long m_sh,
                             int B, int K, int H, int W, int pad,
                             int patch_h, int patch_w, int step_h, int step_w,
                             void* workspace, size_t workspace_bytes, int* flags,
                             iic_slot_info* info_host, void* stream);

/* number of floats in each of the Wx / Wy buffers: the coefficient tensor [patch][cin][tap][K rounded up to 4] written
 * by iic_local_epilogue, followed (for the (K, pad) the tensor-core backward kernels cover, one patch) by scratch in
 * which iic_local_backward lays the coefficients out in MMA operand order.  The caller owns both buffers from the
 * epilogue to the end of the backward; there is no hidden allocation inside the library. */
size_t iic_local_coeff_floats(int K, int pad, int n_patches);

/* From the (all-reduced) joint: min-shift, per-displacement normalise, symmetrise, marginals, entropy
 * (iic_loss.py:124-146), mean over patches (iic_loss.py:186), and the analytic dL/dJ.
 *   loss_out[0]  float32 loss;  loss64_out[0] (nullable) the same in float64
 *   Wx, Wy       backward coefficients, dL/dJ re-laid for the two gradient sweeps
 *   GA_out       (nullable) dL/dJ in J's layout, float64
 *   flags        |= IIC_FLAG_NAN_LOSS if the loss is NaN
 *   workspace    >= iic_local_epilogue_workspace_bytes, zero-initialised once by the caller */
size_t iic_local_epilogue_workspace_bytes(int K, int pad, int n_patches);
int iic_local_epilogue(const double* J, int K, int pad, int n_patches, double lamda,
                       float* loss_out, double* loss64_out, float* Wx, float* Wy, double* GA_out,
                       int* flags, void* workspace, void* stream);

/* Both input gradients (what autograd's convolution_backward yields for iic_loss.py:123):
 *   gx[n,i,a,b] (+)= g * mask * sum_{d,j} dL/dJ[d,i,j] * (mask*y)[n,j,a-dy+pad,b-dx+pad]
 *   gy[n,j,u,v] (+)= g * mask * sum_{d,i} dL/dJ[d,i,j] * (mask*x)[n,i,u+dy-pad,v+dx-pad]
 * g = *grad_loss (device scalar; NULL means 1).  gx/gy are (B,K,H,W) with dense rows and channel planes and the sample
 * strides gx_sn / gy_sn in elements (0 = K*H*W, a fully dense tensor): a sub-head's gradient can be written straight
 * into its channel block of the gradient of the whole (B, S*K, H, W) head output (contrastyou/trainer/_utils.py:
 * 137-168), no gather pass.  With more than one patch the caller zero-fills them first and every patch accumulates.  Wx / Wy are the buffers of iic_local_epilogue
 * (iic_local_coeff_floats floats each); their scratch tail may be overwritten. */
int iic_local_backward(const float* x, long long x_sn, long long x_sc, long long x_sh,
                       const float* y, long long y_sn, long long y_sc, long long y_sh,
                       const float* mask, long long m_sn, long long m_sc, long long m_sh,
                       int B, int K, int H, int W, int pad,
                       int patch_h, int patch_w, int step_h, int step_w,
                       float* Wx, float* Wy, const float* grad_loss,
                       float* gx, float* gy, long long gx_sn, long long gy_sn, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Cluster-head softmax fused into the local term.  lx, ly are the LOGITS of LocalClusterHead
 * (contrastyou/trainer/_utils.py:137-168: 1x1 conv -> SoftmaxWithT, :15-23); the kernels apply
 * softmax(logit * inv_temperature) over the K channels on the fly, so
 *   iic_local_joint_from_logits(l1, l2)  ==  iic_local_joint(softmax(l1), softmax(l2))      (one patch, no mask)
 * and the backward returns the gradients with respect to the logits.  Between the two calls the caller
 * runs iic_local_epilogue exactly as for the probability path.  Covered shapes: padding 1, K == 10,
 * W % 4 == 0, W <= 248, 16-byte aligned rows; anything else returns IIC_UNSUPPORTED (apply the softmax
 * and use the probability entry points).  workspace: iic_b200_sm_count() * 9*K*K floats.  info_host (nullable): when
 * given, the per-CTA slots are left in `workspace` for iic_finish and described there; J_out is then unused.
 * ---------------------------------------------------------------------------------------------- */
int iic_local_joint_from_logits(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                int B, int K, int H, int W, int pad, float inv_temperature,
                                double* J_out, void* workspace, size_t workspace_bytes,
                                iic_slot_info* info_host, void* stream);
int iic_local_backward_from_logits(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                   const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                   int B, int K, int H, int W, int pad, float inv_temperature,
                                   const float* Wx, const float* Wy, const float* grad_loss,
                                   float* g_lx, float* g_ly, long long gx_sn, long long gy_sn, void* stream);

/* The same for the reference's default cluster count (16 <= K <= 24, padding 1 or 3; ABI 7) and for the wide heads
 * (K == 128, padding 1; ABI 8).  Their tensor-core kernels stage 8-channel slices or single channel rows and never hold
 * a whole pixel, so a first pass writes per pixel of both maps
 *   m = max_k(l_k * inv_temperature),  r = 1 / sum_k exp(l_k * inv_temperature - m)
 * into the caller's `stats` buffer (iic_local_logit_stats_floats floats, 16-byte aligned: [2B][2][H][W], planes m and r,
 * lx at samples 0..B-1, ly at B..2B-1), and the kernels use p = exp(l * inv_temperature - m) * r.  The caller keeps
 * stats, Wx and Wy from the forward to the backward; nothing is allocated inside the library.
 *   iic_local_from_logits_covered       1 when these entry points fuse the term on the given maps (device pointers and
 *                                       strides as for the calls), 0 when the caller must apply the softmax and use
 *                                       the probability entry points; the ONE rule both calls follow.  16 <= K <= 24:
 *                                       padding 3, or padding 1 with enough row blocks to fill the SMs; W % 16 == 0;
 *                                       16-byte aligned rows; tensor-core and TMA kernels not switched off.  K == 128:
 *                                       padding 1; W % 16 == 0 and W <= 248; 16-byte aligned rows; tensor-core and TMA
 *                                       kernels not switched off.  K == 10: the shapes of iic_local_joint_from_logits
 *                                       above.
 *   iic_local_joint_from_logits_workspace_bytes   the workspace of the joint (per-SM slots of the kernel it selects)
 *   iic_local_joint_from_logits_stats   as iic_local_joint_from_logits, also writing stats; on a K == 10 shape it is
 *                                       that call (stats untouched, may be NULL); IIC_UNSUPPORTED when not covered
 *   iic_local_backward_from_logits_stats  its backward, reading stats; Wx / Wy are writable because the K = 20 and
 *                                       K = 128 kernels lay their weight images into the buffers' tails
 *                                       (iic_local_coeff_floats) */
size_t iic_local_logit_stats_floats(int B, int H, int W);
size_t iic_local_joint_from_logits_workspace_bytes(int device, int B, int K, int H, int W, int pad);
int iic_local_from_logits_covered(int device, const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                  const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                  int B, int K, int H, int W, int pad);
int iic_local_joint_from_logits_stats(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                      const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                      int B, int K, int H, int W, int pad, float inv_temperature, float* stats,
                                      double* J_out, void* workspace, size_t workspace_bytes,
                                      iic_slot_info* info_host, void* stream);
int iic_local_backward_from_logits_stats(const float* lx, long long x_sn, long long x_sc, long long x_sh,
                                         const float* ly, long long y_sn, long long y_sc, long long y_sh,
                                         int B, int K, int H, int W, int pad, float inv_temperature,
                                         const float* stats, float* Wx, float* Wy, const float* grad_loss,
                                         float* g_lx, float* g_ly, long long gx_sn, long long gy_sn, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Global IIC on (N,K) simplex rows.  Replaces compute_joint (iic_loss.py:74-94) and IIDLoss.forward
 * (iic_loss.py:43-71).
 * ---------------------------------------------------------------------------------------------- */
size_t iic_global_joint_workspace_bytes(int device, long long N, int K);
/* J[i][j] = sum_n x[n,i]*y[n,j]  (iic_loss.py:88-89), float64 out, deterministic.
 * flags (nullable): the simplex assertions of iic_loss.py:50-51 / 82-83 on x and y, fused. */
int iic_global_joint(const float* x, long long x_sn, const float* y, long long y_sn,
                     long long N, int K, double* J_out, void* workspace, size_t workspace_bytes,
                     int* flags, void* stream);
/* P = sym(J)/sum (iic_loss.py:91-92; symmetric=0 skips the symmetrisation), and when losses_out is
 * non-NULL the two entropy expressions of iic_loss.py:63-69: losses_out[0]=loss(lamb),
 * losses_out[1]=loss_no_lamb.  P_out is float32 (K,K). */
int iic_global_epilogue(const double* J, int K, double lamb, int symmetric,
                        float* losses_out, float* P_out, int* flags, void* stream);
/* gradients of  g_loss*loss + g_no_lamb*loss_no_lamb + <gP, P>  w.r.t. x and y, from the saved J.
 * g_loss, g_no_lamb (device scalars) and gP ((K,K) float32) are the upstream gradients of the three
 * outputs of IIDLoss.forward; each is nullable and NULL means "no gradient flows into that output".
 * gx_sn / gy_sn: row strides of the (N, K) gradient tensors in elements (0 = K, dense). */
int iic_global_backward(const float* x, long long x_sn, const float* y, long long y_sn,
                        long long N, int K, const double* J, double lamb, int symmetric,
                        const float* g_loss, const float* g_no_lamb, const float* gP,
                        float* gx, float* gy, long long gx_sn, long long gy_sn, void* stream);
/* The same when x and y are the cluster head's LOGITS and J is the joint of softmax(x * inv_temperature) and
 * softmax(y * inv_temperature) (an IIC_ITEM_GLOBAL_LOGITS term of iic_finish; ABI 8): the gradients are with respect to
 * the logits, d l_k = inv_temperature * p_k * (dp_k - sum_c dp_c p_c) per row, with p computed exactly as the finish
 * launch computed it.  K <= 128. */
int iic_global_backward_from_logits(const float* x, long long x_sn, const float* y, long long y_sn,
                                    long long N, int K, const double* J, double lamb, int symmetric,
                                    float inv_temperature, const float* g_loss, const float* g_no_lamb,
                                    const float* gP, float* gx, float* gy, long long gx_sn, long long gy_sn,
                                    void* stream);

/* ------------------------------------------------------------------------------------------------
 * iic_finish: ONE launch between the joint kernels and the backward kernels of one or many IIC terms -- the (layer,
 * sub-head) calls of one iteration, semi_seg/epocher.py:249-284.  It reduces the per-CTA slots of every local term
 * (iic_local_joint_partials) into its joint in fp64 in a fixed order, computes the joints of the global terms straight
 * from their (N, K) rows (iic_loss.py:88-89, both simplex assertions fused), and -- multi-GPU -- sums ALL joints over the
 * ranks with ONE exchange over the peer buffers of iic_xchg_create (same protocol and bit-identical results as
 * iic_xchg_allreduce).  With want_epilogue it then runs every term's epilogue (iic_local_epilogue /
 * iic_global_epilogue arithmetic) in the same launch when all K <= 32, else as one extra launch per term.
 *   J_all        E_total doubles: the terms' joints back to back in batch order (term i: n_patches*T*T*K*K or K*K);
 *                kept by the caller for the global terms' backward (iic_global_backward's J)
 *   workspace    >= iic_finish_workspace_bytes(), zero-initialised once by the caller, one per stream
 *   xchg_bufs_host, rank, world, xchg_capacity   as for iic_xchg_allreduce; world == 1 means no exchange
 * At most 32 terms per call.
 * ---------------------------------------------------------------------------------------------- */
#define IIC_ITEM_LOCAL 0
#define IIC_ITEM_GLOBAL_ROWS 1
#define IIC_ITEM_GLOBAL_LOGITS 2    /* global term on logit rows: the joint of softmax(x * inv_temperature) and
                                       softmax(y * inv_temperature), each row normalised inside the launch (no simplex
                                       check: a softmax row is one); N <= 4096, K <= 128; ABI 8 */
typedef struct iic_finish_item {
  int kind;                       /* IIC_ITEM_LOCAL, IIC_ITEM_GLOBAL_ROWS or IIC_ITEM_GLOBAL_LOGITS */
  int K;
  double lamda;                   /* lamda of IIDSegmentationLoss / lamb of IIDLoss */
  /* local term: the slots left by iic_local_joint_partials and its geometry */
  const float* slots;
  int layout, n_slots, nb;
  long long slot_stride;
  int pad, n_patches;
  void* epilogue_workspace;       /* iic_local_epilogue_workspace_bytes; used when the epilogue is not fused (K > 32, very
                                     many patches, or the no_fused_epilogue switch) */
  /* global term: the rows */
  const float* x; long long x_sn;
  const float* y; long long y_sn;
  long long N;
  int symmetric, check_simplex;
  /* outputs: local loss_out[1], Wx, Wy (iic_local_coeff_floats each); global loss_out[2], P_out (K,K; nullable) */
  float* loss_out;
  float* Wx;
  float* Wy;
  float* P_out;
  float inv_temperature;          /* IIC_ITEM_GLOBAL_LOGITS: 1 / T of the head's softmax */
} iic_finish_item;
size_t iic_finish_workspace_bytes(void);
int iic_finish(const iic_finish_item* items_host, int n_items, double* J_all, long long E_total, int* flags,
               void* workspace, void* const* xchg_bufs_host, int rank, int world, long long xchg_capacity,
               int want_epilogue, void* stream);

/* ------------------------------------------------------------------------------------------------
 * UDA consistency on (outer, C, inner) contiguous maps.  kind 0 = torch.nn.MSELoss() mean over all
 * elements; kind 1 = KL_div(reduction="mean") (dc2:deepclustering2/loss/kl_losses.py:107-126):
 * sum_c -t*log((p+eps)/(t+eps)) * w_c, mean over outer*inner.  Call site semi_seg/epocher.py:221-224.
 * from_logits != 0: prob/target hold logits and the channel softmax (epocher.py:222-223) is fused in;
 * the gradient is then w.r.t. the prob logits.  The gradient flows to `prob` only.  1 <= C <= 256: up to
 * 8 channels a thread holds all channels of its pixels, from 9 the channels of a pixel are spread over the
 * warps of a CTA (DESIGN.md section 4.5).
 * ---------------------------------------------------------------------------------------------- */
size_t iic_uda_workspace_bytes(int device);
int iic_uda_forward(const float* prob, const float* target, long long outer, int C, long long inner,
                    int kind, double eps, const float* weight, int from_logits,
                    float* loss_out, int* flags, int check_simplex, void* workspace, void* stream);
int iic_uda_backward(const float* prob, const float* target, long long outer, int C, long long inner,
                     int kind, double eps, const float* weight, int from_logits,
                     const float* grad_loss, float* grad_prob, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Supervised branch of the udaiic iteration (SURVEY.md section 8f row 4), softmax and one-hot fused:
 *   loss = KL_div()(softmax(logits, 1), class2one_hot(labels, C))       semi_seg/epocher.py:165-166,
 *          = mean over outer*inner of  -log((p[label] + eps) / (1 + eps)) * w[label]
 *            (dc2:deepclustering2/loss/kl_losses.py:107-126 with a one-hot target; eps > 0)
 *   dice_out (nullable, 2*outer*C int64, overwritten): what UniversalDice.add appends for
 *          (logits.max(1)[1], labels) at semi_seg/epocher.py:183-184
 *          (dc2:deepclustering2/meters2/individual_meters/general_dice_meter.py:41-95):
 *          dice_out[0][o][c] = #pixels(argmax == c and label == c)       (_intersaction)
 *          dice_out[1][o][c] = #pixels(argmax == c) + #pixels(label == c) (_union)
 * logits (outer, C, inner) contiguous float32, 1 <= C <= 256; labels (outer, inner) contiguous int64 class
 * indices; weight (nullable) C floats, already normalised as at kl_losses.py:100.  A label outside
 * [0, C) sets IIC_FLAG_BAD_LABEL and contributes nothing.  workspace >= iic_sup_workspace_bytes,
 * zero-initialised once by the caller.  The backward writes d loss / d logits (dense, same layout).
 *
 * The _ignore pair adds an ignore label (torch's `ignore_index`; Cityscapes / VOC void = 255):
 *   - a pixel whose label equals ignore_index (any value, also one inside [0, C)) adds nothing to the
 *     loss, gets an exactly zero gradient and is left out of dice_out (neither its argmax nor its label
 *     is counted); it never sets IIC_FLAG_BAD_LABEL;
 *   - n = #pixels whose label is not ignore_index, counted on the device by the forward into *n_valid
 *     (1 int64, overwritten); the loss is the sum above over those pixels divided by n, with or without
 *     weights (KL_div's mean, not torch's division by the summed weights); n = 0 gives a loss of 0.0,
 *     a zero gradient and no IIC_FLAG_NAN_LOSS;
 *   - any other label outside [0, C) behaves as above and counts in n;
 *   - the backward reads n from the n_valid the forward wrote (stream order), so neither call
 *     synchronises the host and a graph replay may see a different n each time.
 * ---------------------------------------------------------------------------------------------- */
size_t iic_sup_workspace_bytes(int device, long long outer);
int iic_sup_forward(const float* logits, const long long* labels, long long outer, int C, long long inner,
                    double eps, const float* weight, float* loss_out, long long* dice_out, int* flags,
                    void* workspace, void* stream);
int iic_sup_backward(const float* logits, const long long* labels, long long outer, int C, long long inner,
                     double eps, const float* weight, const float* grad_loss, float* grad_logits,
                     void* stream);
int iic_sup_forward_ignore(const float* logits, const long long* labels, long long outer, int C, long long inner,
                           double eps, const float* weight, long long ignore_index, float* loss_out,
                           long long* dice_out, long long* n_valid, int* flags, void* workspace, void* stream);
int iic_sup_backward_ignore(const float* logits, const long long* labels, long long outer, int C,
                            long long inner, double eps, const float* weight, long long ignore_index,
                            const long long* n_valid, const float* grad_loss, float* grad_logits, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Per-sample flip alignment (SURVEY.md section 8f row 2).  The reference aligns the two views with
 *   with FixRandomSeed(seed): torch.stack([TensorRandomFlip(axis=[1, 2], threshold=0.8)(x) for x in batch])
 * (semi_seg/epocher.py:121,148-149,160-161,264-266; dc2:deepclustering2/augment/tensor_augment.py:17-41),
 * i.e. per sample a clone and up to two flips, then a stack.  Here the flags are drawn once on the host
 * (same generator, same order) and passed as one byte per sample: IIC_FLIP_H = axis 1 of the (C,H,W)
 * sample, IIC_FLIP_W = axis 2.
 *   iic_flip_batch        out[n,c,h,w] = in[n,c, H-1-h if H-flag else h, W-1-w if W-flag else w]; one launch,
 *                         one pass; (outer, C, H, W) contiguous float32, out != in.  Its own adjoint.
 *   iic_uda_flip_forward  iic_uda_forward(prob, flip(target)) without materialising flip(target): the UDA
 *   iic_uda_flip_backward term of semi_seg/epocher.py:221-224 on `unlabel_tf_logits` and the unflipped
 *                         `unlabel_logits` (epocher.py:160-161 fused away).  kind / eps / from_logits as for
 *                         iic_uda_forward (no class weights, no simplex pass); 1 <= C <= 256.  workspace >=
 *                         iic_uda_flip_workspace_bytes, zero-initialised once by the caller.
 * ---------------------------------------------------------------------------------------------- */
#define IIC_FLIP_H 1
#define IIC_FLIP_W 2
int iic_flip_batch(const float* in, float* out, const unsigned char* flips, long long outer, int C, int H, int W,
                   void* stream);
size_t iic_uda_flip_workspace_bytes(int device, long long outer);
int iic_uda_flip_forward(const float* prob, const float* target, const unsigned char* flips, long long outer,
                         int C, int H, int W, int kind, double eps, int from_logits, float* loss_out, int* flags,
                         void* workspace, void* stream);
int iic_uda_flip_backward(const float* prob, const float* target, const unsigned char* flips, long long outer,
                          int C, int H, int W, int kind, double eps, int from_logits, const float* grad_loss,
                          float* grad_prob, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Joint exchange over NVLink peer memory (multi-GPU, one process per GPU).  The path's only collective
 * (SURVEY.md section 8e: J is a plain sum over the batch index, iic_loss.py:89,123) without NCCL: each
 * rank stores its fp64 partial joints into its slot of every peer's buffer, publishes a sequence number,
 * waits for all peers and adds the slots in rank order (bit-identical result on every rank).  The sequence
 * counter lives in the buffer, so the call can be captured in a CUDA graph.  All ranks must issue the same
 * exchanges in the same order.
 *   iic_xchg_create      cudaMalloc + zero a buffer for `world` ranks of `capacity` doubles each
 *   iic_xchg_export      its 64-byte CUDA IPC handle (host memory), to be sent to the peers
 *   iic_xchg_import      map a peer's buffer from its handle
 *   iic_xchg_release     cudaFree (imported = 0) or cudaIpcCloseMemHandle (imported = 1)
 *   iic_xchg_allreduce   J[0..E) <- sum over ranks, in place; bufs_host[r] = this process's pointer to rank
 *                        r's buffer (host array of `world` device pointers); flags (nullable) receives
 *                        IIC_FLAG_XCHG_TIMEOUT when a peer does not arrive within the xchg_timeout_ms option
 *                        (the wait is bounded but long: a slow peer is not an error)
 * ---------------------------------------------------------------------------------------------- */
size_t iic_xchg_buffer_bytes(int world, long long capacity);
int iic_xchg_create(int world, long long capacity, void** buf_out);
int iic_xchg_export(void* buf, void* handle64_host);
int iic_xchg_import(const void* handle64_host, void** peer_out);
int iic_xchg_release(void* buf, int imported);
int iic_xchg_allreduce(double* J, long long E, long long capacity, void* const* bufs_host, int rank,
                       int world, int* flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IIC_B200_H_ */
