/*
 * spff_b200.h — C ABI of libspff_b200.so: the B200 (sm_100a) kernels behind the SPFF-UNet hot path.
 *
 * The reference (NF-91/spff-unet-spcct) is pure Python: its hot path is the sequence of ATen /
 * cuDNN / cuFFT library calls that `innovative3D/models.py` and `innovative3D/helpers.py` dispatch.
 * Each entry point below replaces one of those call sites (cited per function as file:line of the
 * reference). The host layer that binds them is `spff-unet-spcct_b200/spff_b200/_lib.py` (ctypes);
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *  - Plain C types only. Every pointer is a DEVICE pointer unless the name ends in `_host`.
 *  - Activations are bf16, position-major ("NDHWC"): element (n,d,h,w,c) of a view lives at
 *    base + (((n*D + d)*H + h)*W + w)*ld + c, `ld` = channel pitch in elements (ld >= C, ld % 8 == 0,
 *    base 16-byte aligned). A channel slice of a wider buffer (skip-concat halves) is expressed by
 *    offsetting `base` and keeping the buffer's `ld`.
 *  - The five energy bins are the D axis (reference: models.py:1551, datasets.py:228-233).
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); no call synchronises the host.
 *  - Return 0 on success, a negative SPFF_ERR_* otherwise; spff_last_error() holds the text
 *    (thread local). There is no CPU fallback: on a device that is not sm_100 every compute entry
 *    point returns SPFF_ERR_UNSUPPORTED_ARCH.
 *  - The library allocates no persistent device memory; scratch is caller-provided `workspace`.
 */
#ifndef SPFF_B200_H_
#define SPFF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPFF_OK 0
#define SPFF_ERR_BAD_ARGUMENT (-1)
#define SPFF_ERR_UNSUPPORTED_ARCH (-2)
#define SPFF_ERR_CUDA (-3)
#define SPFF_ERR_WORKSPACE (-4)

/* gate flags for the collapsed SPFF tail (spff_gate_micro_*) */
#define SPFF_GATE_EFILM 1   /* EnergyFiLM3D      models.py:1479-1512 */
#define SPFF_GATE_FOURIER 2 /* FourierGate3D     models.py:1515-1544 */
#define SPFF_GATE_SPECSE 4  /* _SpectralSE       models.py:611-614   */
#define SPFF_GATE_CHANSE 8  /* _SEChannelLite    models.py:600-609   */

typedef struct spff_shape {
  int n, d, h, w; /* samples, energy bins (depth), height, width of the position grid */
} spff_shape;

/* ---- library ------------------------------------------------------------------------------ */
int spff_version(void);
const char* spff_last_error(void);
/* 0 when the current CUDA device is sm_100 (B200); SPFF_ERR_UNSUPPORTED_ARCH otherwise. */
int spff_device_check(void);
/* Test / measurement hook (never needed in production; 0 = default everywhere). Keys:
 *   0  number of CTAs for the persistent kernels (0 = one per SM)
 *   1  non-zero disables the all-kh variant of the 32-channel weight-gradient kernel
 *   2  non-zero selects the CUDA-core fused head kernel instead of the mma.sync one
 *   3, 4  blocks per SM of the InstanceNorm statistics / backward statistics kernels
 *   4  (conv kernels) device pointer of a cycle-counter buffer; 5  timing experiments of the halo conv kernel and, in the
 *      transposed conv, no quadrant folding
 *   6  non-zero disables the aligned epilogue of the flattened-row conv kernel
 *   7  1 = always the flattened-row conv kernel, 2 = always the halo-tile kernel
 *   8  non-zero selects the fp32 FMA stem forward instead of the mma.sync one
 *   9  non-zero: the 32-channel weight gradient loads three kw-shifted x tiles instead of one halo tile */
int spff_debug_set(int key, long long value);

/* ---- 3x3x3 convolution, stride 1, zero pad 1, no bias ----------------------------------------
 * Replaces nn.Conv3d(cin, cout, (3,3,3), padding 1, bias=False) built by `_conv3x3xk`
 * (models.py:616-618) — forward, and the input / weight halves of its convolution_backward.
 * cin, cout multiples of 32 (the Cin = 1 stem has its own entry points below). */
/* Elements (bf16) of one packed weight operand: 2*27*cin*cout — the layouts of the two conv kernels back to back. */
long long spff_conv3_packed_elems(int cin, int cout);
/* nn.Conv3d weight [cout][cin][3][3][3] fp32 -> bf16 GEMM operands (either may be NULL):
 *   w_fwd   [cout/32][kh][cin/KC][2-kd][kw][32][KC]        KC = 64 if cin % 64 == 0 else 32
 *   w_dgrad [cin/32][kh][cout/KC'][2-kd][kw][32][KC']      taps flipped, in/out transposed
 * followed by the halo kernel's [cout/CO][cin/32][kh*3+kw][2-kd][CO][32] (CO = 64 if cout % 64 == 0 else 32; planes whose
 * height is a multiple of 16 and width a multiple of 8 run that kernel)
 * (opaque to callers: only spff_conv3d_k3_fwd/_fwd_stats/_dgrad consume them). */
int spff_pack_conv3_weight(const float* w, void* w_fwd, void* w_dgrad, int cout, int cin, void* stream);
/* y[n,d,h,w,0:cout] = conv3d(x)[...]  (F.conv3d at models.py:616-618 via nn.Sequential :1459-1469) */
int spff_conv3d_k3_fwd(const void* x, long long ldx, int cin, const void* w_fwd, void* y, long long ldy, int cout,
                       spff_shape s, void* stream);
/* Forward + InstanceNorm statistics of the output in the same kernel: the epilogue writes, per work
 * item, the {sum, sum of squares} of its fp32 output tile to stat_partial[n][slots][2][cout]
 * (slots = spff_conv3d_k3_stat_slots(s)); spff_in_coeffs_from_partials reduces them in a fixed
 * order. Replaces the separate spff_in_stats pass over y. */
int spff_conv3d_k3_stat_slots(spff_shape s);
int spff_conv3d_k3_fwd_stats(const void* x, long long ldx, int cin, const void* w_fwd, void* y, long long ldy, int cout,
                             spff_shape s, float* stat_partial, void* stream);
/* dx = input gradient of the same convolution (ATen convolution_backward, grad_input). */
int spff_conv3d_k3_dgrad(const void* dy, long long lddy, int cout, const void* w_dgrad, void* dx, long long lddx,
                         int cin, spff_shape s, void* stream);
/* The same, plus the per-item column statistics of dx: stat_partial[n][slots][2][cin] as in spff_conv3d_k3_fwd_stats.
 * Their sums over (n, slots) are the bias gradient of a ConvTranspose3d whose output dx is the gradient of. */
int spff_conv3d_k3_dgrad_stats(const void* dy, long long lddy, int cout, const void* w_dgrad, void* dx, long long lddx,
                               int cin, spff_shape s, float* stat_partial, void* stream);

/* dw[cout][cin][3][3][3] (fp32) = beta*dw + weight gradient (ATen convolution_backward, grad_weight).
 * Split over positions; fp32 partial tiles go to `workspace` (size from the query below, which
 * depends on the SM count of the current device) and are reduced in a fixed order. */
size_t spff_conv3d_k3_wgrad_workspace(int cin, int cout, spff_shape s);
int spff_conv3d_k3_wgrad(const void* x, long long ldx, int cin, const void* dy, long long lddy, int cout,
                         spff_shape s, float* dw, float beta, void* workspace, size_t workspace_bytes,
                         void* stream);

/* ---- the Cin = 1 stem convolution (enc1.pre.0 / enc1.b1.0: `_conv3x3xk(1, 32, 3)`, models.py:616-618 with
 * in_channels = 1 from models.py:1551) ------------------------------------------------------------
 * x is the network input as the reference holds it: fp32 [N,1,D,H,W] contiguous. w fp32 [cout][1][3][3][3]. */
int spff_conv3d_stem_fwd(const float* x, const float* w, void* y, long long ldy, int cout, spff_shape s,
                         void* stream);
/* Forward + statistics of the output in the epilogue: stat_partial[n][slots][2][cout] with
 * slots = spff_conv3d_stem_stat_slots(s), reduced by spff_in_coeffs_from_partials / spff_bn_coeffs (cout must be 32). */
int spff_conv3d_stem_stat_slots(spff_shape s);
int spff_conv3d_stem_fwd_stats(const float* x, const float* w, void* y, long long ldy, int cout, spff_shape s,
                               float* stat_partial, void* stream);
size_t spff_conv3d_stem_wgrad_workspace(int cout);
/* dw[cout][1][3][3][3] = beta*dw + gradient (per-block partials in `workspace`, fixed-order reduce). */
int spff_conv3d_stem_wgrad(const float* x, const void* dy, long long lddy, int cout, spff_shape s, float* dw,
                           float beta, void* workspace, size_t workspace_bytes, void* stream);

/* ---- ConvTranspose3d kernel = stride = (1,2,2), with bias (models.py:668-672) -------------------
 * `s` is always the COARSE grid (input of the forward); the fine tensors are [n, d, 2h, 2w, c].
 * Weight [cin][cout][1][2][2] fp32 -> bf16 operands  w_fwd [4][cin/KC][cout][KC],
 * w_dgrad [4][cout/KC'][cin][KC']  (quadrant q = 2*i + j). */
int spff_pack_convt_weight(const float* w, void* w_fwd, void* w_dgrad, int cin, int cout, void* stream);
int spff_convt_k122_fwd(const void* x, long long ldx, int cin, const void* w_fwd, const float* bias, void* y,
                        long long ldy, int cout, spff_shape s, void* stream);
int spff_convt_k122_dgrad(const void* dy, long long lddy, int cout, const void* w_dgrad, void* dx, long long lddx,
                          int cin, spff_shape s, void* stream);
size_t spff_convt_k122_wgrad_workspace(int cin, int cout, spff_shape s);
/* dw[cin][cout][1][2][2] = beta*dw + gradient. (The bias gradient is the column sum of dy: spff_in_stats.) */
int spff_convt_k122_wgrad(const void* x, long long ldx, int cin, const void* dy, long long lddy, int cout,
                          spff_shape s, float* dw, float beta, void* workspace, size_t workspace_bytes,
                          void* stream);

/* ---- InstanceNorm3d(affine, eps) + LeakyReLU + the collapsed SPFF tail ----------------------------
 * models.py:168-181 (norm, act), :1473-1478 (block), :684-685 (_post). SURVEY.md §7.3:
 *   a = lrelu(IN(x)),  out = a * P[n,d,c] + Q[n,d,c]. */
/* stats[n][c]{sum, sum of squares} += over the (d,h,w) positions of x (double; caller zeroes). */
int spff_in_stats(const void* x, long long ldx, int c, spff_shape s, double* stats, void* stream);
/* stats over `count` elements per (n,c) -> coef[n][c] = {A, B, mean, rstd}, IN(x) = x*A + B with
 * A = rstd*gamma[c], B = beta[c] - mean*A. batch_stats != 0: BatchNorm3d training statistics
 * (summed over n; models.py:170-171 / Cicek3DUNet :721). */
int spff_in_coeffs(const double* stats, const float* gamma, const float* beta, float eps, int n, int c,
                   long long count, int batch_stats, float* coef, void* stream);
/* Same coefficients from the partial statistics of spff_conv3d_k3_fwd_stats. */
int spff_in_coeffs_from_partials(const float* partial, int slots, const float* gamma, const float* beta, float eps, int n,
                                 int c, long long count, float* coef, void* stream);
/* y = lrelu(x*A + B) (bf16 -> bf16). */
int spff_norm_act_apply(const void* x, long long ldx, const float* coef, void* y, long long ldy, int c, spff_shape s,
                        float slope, void* stream);
/* S[n][d][c] = sum_{h,w} lrelu(x*A + B)  (fp32). With a workspace of spff_norm_act_reduce_workspace() bytes
 * the block partials are reduced in a fixed order and S is overwritten (bit-reproducible); with
 * workspace == NULL the blocks accumulate into S with atomics (+=; the caller zeroes S). */
size_t spff_norm_act_reduce_workspace(int c, spff_shape s);
int spff_norm_act_reduce(const void* x, long long ldx, const float* coef, float* S, int c, spff_shape s, float slope,
                         void* workspace, size_t workspace_bytes, void* stream);
/* y = lrelu(x*A+B)*P + Q; P,Q are [n][d][c] fp32 or both NULL (identity). If ypool != NULL also
 * writes the (1,2,2) max-pool of y (nn.MaxPool3d, models.py:658-665) to ypool [n,d,h/2,w/2] with pitch ldp. */
int spff_norm_act_affine_apply(const void* x, long long ldx, const float* coef, const float* P, const float* Q,
                               void* y, long long ldy, void* ypool, long long ldp, uint8_t* pool_argmax, int c, spff_shape s,
                               float slope, void* stream);
/* Parameter-only tables of the gates and their backward (EnergyFiLM3D models.py:1494-1512: g1 = 1 + tanh(gamma), bt = beta,
 * each [c][frames], from the MLP weights w0 [32][16], b0 [32], w2 [2c][32], b2 [2c] over the sinusoidal bin code;
 * FourierGate3D models.py:1537-1542: kfg [frames] = irfft(freq_mask [frames/2+1] * mag_scale [1])). A NULL w0 / freq_mask
 * skips that gate. The backward ACCUMULATES (+=) the parameter gradients from dg1 / dbt / dkfg. frames <= 16. */
int spff_gate_tables_fwd(const float* w0, const float* b0, const float* w2, const float* b2, const float* freq_mask,
                         const float* mag_scale, int c, int frames, float* g1, float* bt, float* kfg, void* stream);
int spff_gate_tables_bwd(const float* w0, const float* b0, const float* w2, const float* b2, const float* freq_mask,
                         const float* mag_scale, int c, int frames, const float* dg1, const float* dbt, const float* dkfg,
                         float* dw0, float* db0, float* dw2, float* db2, float* dfreq_mask, float* dmag_scale, void* stream);
/* Gate micro-kernel: S[n][d][c] -> P,Q[n][d][c]. Tables (fp32, device): g1[c][d] = 1 + tanh(gamma),
 * bt[c][d] = beta of EnergyFiLM (input independent, models.py:1494-1512); kfg[d]: the circular
 * kernel irfft(freq_mask*mag_scale) of FourierGate (models.py:1537-1542); se_w1[hid][c], se_b1[hid],
 * se_w2[c][hid], se_b2[c]: _SEChannelLite fc (models.py:604-607). Unused ones NULL. */
int spff_gate_micro_fwd(const float* S, const float* g1, const float* bt, const float* kfg, const float* se_w1,
                        const float* se_b1, const float* se_w2, const float* se_b2, int hid, int flags, int c,
                        spff_shape s, float* P, float* Q, void* stream);
/* Backward pass 1: R[n][d][c][6] += per-plane sums over (h,w) of
 *   {dout*a, dout, dout*m, m, dout*m*xhat, m*xhat},  m = lrelu'(z), z = x*A+B, a = lrelu(z).
 * plain != 0: only slots 2 and 4 are produced (all that spff_gate_micro_bwd(flags = 0) reads).
 * workspace as for spff_norm_act_reduce: fixed-order overwrite of the produced slots, or NULL for atomics (+=). */
size_t spff_norm_act_bwd_reduce_workspace(int c, spff_shape s, int plain);
/* S (may be NULL): the forward statistic S[n][d][c] = sum_{h,w} lrelu(x*A + B) of the same tensor
 * (spff_norm_act_reduce). With a workspace and (plain or S given) a leaner first stage runs: the two xhat sums
 * follow from the others, sum dout*m*xhat = (sum dout*a - beta*sum dout*m)/gamma and
 * sum m*xhat = (S - beta*sum m)/gamma (gamma == 0: those two read 0). */
int spff_norm_act_bwd_reduce(const void* dout, long long lddo, const void* x, long long ldx, const float* coef,
                             float* R, const float* S, int c, spff_shape s, float slope, int plain, void* workspace,
                             size_t workspace_bytes, void* stream);
/* Backward micro-kernel: consumes R (and S), recomputes the gates, produces
 *   bcoef[n][c] = {gamma*rstd, mean(dz), mean(dz*xhat), 0}, dSa[n][d][c], Pout[n][d][c]
 * and ACCUMULATES (+=) dgamma[c], dbeta[c], dg1[c][d], dbt[c][d], dkfg[d], dse_*. flags == 0 is the
 * plain InstanceNorm+LeakyReLU backward (S, dSa, Pout and the gate tables may be NULL). */
int spff_gate_micro_bwd(const float* R, const float* S, const float* coef, const float* gamma, const float* g1,
                        const float* bt, const float* kfg, const float* se_w1, const float* se_b1,
                        const float* se_w2, const float* se_b2, int hid, int flags, int c, spff_shape s,
                        float* bcoef, float* dSa, float* Pout, float* dgamma, float* dbeta, float* dg1, float* dbt,
                        float* dkfg, float* dse_w1, float* dse_b1, float* dse_w2, float* dse_b2, void* stream);
/* Backward pass 2: dx = c1*(dz - c2 - xhat*c3), dz = (dout*P + dSa)*m. P/dSa both NULL: P = 1, dSa = 0. */
int spff_norm_act_bwd_apply(const void* dout, long long lddo, const void* x, long long ldx, const float* coef,
                            const float* bcoef, const float* P, const float* dSa, void* dx, long long lddx, int c,
                            spff_shape s, float slope, void* stream);
/* Max-pool (1,2,2) backward fused with the skip add: dskip (full res) = (accumulate ? dskip : 0) +
 * scatter(dpool) at the arg-max of y in each 2x2 window (first max wins, as ATen). `s` = full-res grid. */
int spff_maxpool_bwd_add(const void* dpool, long long ldp, const void* y, long long ldy, void* dskip, long long ldd,
                         int c, spff_shape s, int accumulate, void* stream);
/* The same from the arg-max codes spff_norm_act_affine_apply wrote beside the pooled tensor (pool_argmax: uint8
 * [n,d,h/2,w/2,c], the corner 0..3 = (kh,kw) of the window's first maximum): the full-resolution activation is not read. */
int spff_maxpool_bwd_add_argmax(const void* dpool, long long ldp, const uint8_t* pool_argmax, void* dskip, long long ldd,
                                int c, spff_shape s, int accumulate, void* stream);

/* ---- head (1x1x1 conv + bias, models.py:674) and loss (helpers.py:782-803) ------------------------ */
/* logits fp32 [N,K,D,H,W] = x[pos][0..32) . w[K][32] + b[K]   (cin must be 32, K <= 16). */
int spff_head_fwd(const void* x, long long ldx, int cin, const float* w, const float* b, float* logits, int k,
                  spff_shape s, void* stream);
/* labels uint8 [N,D,H,W] = argmax_k (first max wins, torch.argmax) — inference path. */
int spff_head_argmax(const void* x, long long ldx, int cin, const float* w, const float* b, uint8_t* labels, int k,
                     spff_shape s, void* stream);
size_t spff_head_bwd_workspace(int k);
/* dx (bf16, may be NULL) = dlogits . w ; dw[K][32], db[K] = beta*old + gradient. */
int spff_head_bwd(const float* dlogits, const void* x, long long ldx, int cin, const float* w, void* dx,
                  long long lddx, float* dw, float* db, float beta, int k, spff_shape s, void* workspace,
                  size_t workspace_bytes, void* stream);
/* Cross-entropy + hard confusion tally over logits fp32 [N,K,D,H,W] (F.cross_entropy(ignore_index)
 * helpers.py:798-801; the counts of helpers.py:687-690, 716-719, 789-791):
 *   acc[0] += sum of nll over valid voxels (double), counts[0] += #valid (int64),
 *   confusion[K][K] (int64, [label][argmax]) += tallies.  label_bytes = 1 (uint8) or 8 (int64). */
int spff_ce_confusion(const float* logits, const void* labels, int label_bytes, int ignore_index, int k,
                      spff_shape s, double* acc, long long* counts, long long* confusion, void* stream);
/* dlogits = (softmax - onehot) * gscale[0] / n_valid[0] on valid voxels, 0 on ignored ones
 * (gscale may be NULL = 1). */
int spff_ce_grad(const float* logits, const void* labels, int label_bytes, int ignore_index, int k, spff_shape s,
                 const long long* n_valid, const float* gscale, float* dlogits, void* stream);

/* Fused TRAINING head: head_fwd + ce_confusion + ce_grad + head_bwd in one pass over x; the logits
 * are never materialised. acc/counts/confusion accumulate as in spff_ce_confusion; dx (bf16, may be
 * NULL), dw[K][32], db[K] (= beta*old + gradient) as in spff_head_bwd with
 * dlogits = (softmax - onehot) * gscale[0] / n_valid[0]. */
size_t spff_head_loss_workspace(int k);
int spff_head_loss_fused(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                         int label_bytes, int ignore_index, int k, spff_shape s, const long long* n_valid,
                         const float* gscale, double* acc, long long* counts, long long* confusion, void* dx,
                         long long lddx, float* dw, float* db, float beta, void* workspace, size_t workspace_bytes,
                         void* stream);
/* Fused EVALUATION head: head_fwd + ce_confusion in one pass over x, forward only; the logits are never
 * materialised. acc/counts/confusion accumulate (+=) over the batch exactly as in spff_ce_confusion (labels
 * uint8 or int64, ignore_index skipped, labels outside [0,K) counted in acc/counts but not in confusion), from
 * the logits and first-maximum arg-max of spff_head_loss_fused. sample_acc[n], sample_counts[n],
 * sample_confusion[n][K][K] receive (+=) the same tally per sample (all three NULL = off); labels_out uint8
 * [N,D,H,W] receives the arg-max the tally counts (NULL = off). Any D*H*W; N <= 65535. */
int spff_head_eval(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                   int label_bytes, int ignore_index, int k, spff_shape s, double* acc, long long* counts,
                   long long* confusion, double* sample_acc, long long* sample_counts, long long* sample_confusion,
                   uint8_t* labels_out, void* stream);
/* spff_head_eval plus the ranking statistics of the softmax: for every counted voxel (label in [0,K), not
 * ignore_index) and every class c, p_c = e_c / sum(e) (fp32, IEEE division) falls in bin min(floor(p_c * bins),
 * bins - 1); hist int64 [K][2][bins] receives (+=) the positives (label == c) in [c][0] and the negatives in [c][1],
 * sample_hist [N][K][2][bins] the same per sample. bins in [16, 1024]; hist required; sample_hist is given exactly
 * when the per-sample tallies are. Every other argument and output is that of spff_head_eval. */
int spff_head_eval_hist(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                        int label_bytes, int ignore_index, int k, spff_shape s, double* acc, long long* counts,
                        long long* confusion, double* sample_acc, long long* sample_counts, long long* sample_confusion,
                        uint8_t* labels_out, int bins, long long* hist, long long* sample_hist, void* stream);

/* ---- averaged softmax: ensembles and mirror test-time augmentation ------------------------------------------
 * Head + softmax added into a probability accumulator: for every position (n,d,h,w) of the network output,
 * p_c = e_c / sum(e) (fp32, IEEE division: the p of spff_head_eval_hist, from the same logits) and
 *   acc[n][d][h'][w'][c] = beta * acc[...][c] + p_c,   h' = H-1-h when flip & 1, w' = W-1-w when flip & 2,
 * i.e. the inverse of an input flip is folded into the store. acc: fp32 [N,D,H,W,16] (64 B per position, 16-byte
 * aligned); classes >= K are written as 0 when beta = 0 and never touched when beta = 1. Each element is written by
 * one thread per call (no atomics, deterministic); beta = 0 does not read acc. x as in spff_head_eval. k in [2,16],
 * flip in [0,3], beta 0 or 1, N <= 65535. */
int spff_head_prob_accum(const void* x, long long ldx, int cin, const float* w, const float* b, int k, spff_shape s,
                         int flip, int beta, float* acc, void* stream);
/* One pass over an accumulator of spff_head_prob_accum: p̄_c = scale * acc_c (fp32; scale = 1 / number of passes), the
 * arg-max is the first maximum of acc_c over c < K (torch.argmax; taken on acc so that the scaling cannot create ties).
 * Outputs, each optional:
 *  - labels_out uint8 [N,D,H,W]: the arg-max;
 *  - proba_out fp16 [N,K,D,H,W] (class-major, the layout of softmax(model(x), 1)): p̄_c rounded to nearest;
 *  - with labels (uint8 or int64 [N,D,H,W]; NULL = no tally, and then no tally output may be given) the tally of
 *    spff_head_eval (+=): a label equal to ignore_index is not counted; a label y in [0,K) counts in counts, adds
 *    -log(max(p̄_y, FLT_MIN)) to nll and one to confusion[y][arg]; any other label counts in counts only.
 *    sample_acc / sample_counts / sample_confusion: the same per sample (together or not at all);
 *  - hist int64 [K][2][bins] (+=, needs labels): for every voxel with a label in [0,K) and every class c, p̄_c falls in
 *    bin min(floor(p̄_c * bins), bins - 1) of [c][0] (label == c) or [c][1]; bins in [16, 1024]; sample_hist
 *    [N][K][2][bins] is given exactly when the per-sample tallies are.
 * k in [2,16], acc 16-byte aligned, N <= 65535. */
int spff_prob_finalize(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                       int ignore_index, double* nll, long long* counts, long long* confusion, double* sample_acc,
                       long long* sample_counts, long long* sample_confusion, uint8_t* labels_out, int bins,
                       long long* hist, long long* sample_hist, void* proba_out, void* stream);

/* ---- uncertainty and calibration of the averaged softmax ----------------------------------------------------
 * spff_head_prob_accum plus the expected-entropy plane: acc is written exactly as spff_head_prob_accum writes it, and
 *   ent[n][d][h'][w'] = beta * ent[...] + H(p),   H(p) = -sum_{c<K} p_c log p_c (nats, fp32),
 * at the same mirrored position. ent: fp32 [N,D,H,W], 4-byte aligned; one writer per element per call. */
int spff_head_prob_accum_ent(const void* x, long long ldx, int cin, const float* w, const float* b, int k, spff_shape s,
                             int flip, int beta, float* acc, float* ent, void* stream);

/* Outputs of spff_prob_finalize_unc; every pointer may be NULL unless a rule below needs it. A voxel is counted when its
 * label is in [0,K) and not ignore_index. Sums of real quantities (all but brier) are rounded per voxel to the fixed
 * point 2^-24 and summed in integers, so they are bit-reproducible. */
typedef struct spff_unc_out {
  const float* ent;         /* expected-entropy plane of spff_head_prob_accum_ent (sum over passes), or NULL          */
  void* entropy_out;        /* fp16 [N,D,H,W]: H[p̄] = -sum_c p̄_c log p̄_c (0 log 0 = 0), nats                         */
  void* mi_out;             /* fp16 [N,D,H,W]: max(H[p̄] - scale * ent, 0), the mutual information; needs ent           */
  long long* unc;           /* int64 [2] (+=): sum of H[p̄], sum of MI over all positions (MI: 0 without ent), 2^-24 */
  long long* sample_unc;    /* int64 [N][2] (+=): the same per sample; needs unc                                      */
  int cal_bins;             /* T in [2, 1024], when calib is given                                                    */
  long long* calib;         /* int64 [3][T] (+=), needs labels: per confidence bin min(floor(conf * T), T - 1),        */
                            /* conf = p̄_arg, the counted voxels, the correct ones (arg == label), sum conf in 2^-24   */
  long long* sample_calib;  /* int64 [N][3][T]; given exactly when the per-sample tallies are (with calib)           */
  double* brier;            /* (+=) sum over counted voxels of sum_c (p̄_c - [c == y])^2; given exactly when calib is */
  double* sample_brier;     /* [N]; given exactly when sample_calib is                                               */
} spff_unc_out;

/* spff_prob_finalize (same arguments, same outputs, bit for bit) plus the uncertainty maps, sums and calibration
 * histogram of `unc` (not NULL). */
int spff_prob_finalize_unc(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                           int ignore_index, double* nll, long long* counts, long long* confusion, double* sample_acc,
                           long long* sample_counts, long long* sample_confusion, uint8_t* labels_out, int bins,
                           long long* hist, long long* sample_hist, void* proba_out, const spff_unc_out* unc,
                           void* stream);

/* ---- temperature scaling of the averaged softmax -------------------------------------------------------------
 * spff_prob_finalize_unc with the pooled distribution tempered: with β = inv_temperature (positive, finite),
 *   p̃_c = p̄_c^β / sum_{c'<K} p̄_c'^β        (p̄_c = 0 stays 0),
 * replaces p̄ in every output: proba_out, nll, hist, H[p̃] (entropy_out and unc[0]), the confidence p̃_arg and brier
 * of `unc`. The arg-max (labels_out, confusion) is unchanged, and the mutual information (mi_out, unc[1]) stays
 * H[p̄] - mean H[p] of the untempered passes, bit for bit. unc may be NULL (the outputs of spff_prob_finalize only).
 * Every other argument is that of spff_prob_finalize_unc. */
int spff_prob_finalize_tempered(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                                int ignore_index, double* nll, long long* counts, long long* confusion,
                                double* sample_acc, long long* sample_counts, long long* sample_confusion,
                                uint8_t* labels_out, int bins, long long* hist, long long* sample_hist, void* proba_out,
                                const spff_unc_out* unc, float inv_temperature, void* stream);
/* Bytes of the workspace of spff_prob_temp_fit for k classes, shape s and g grid points (0 when they are invalid). */
size_t spff_prob_temp_fit_workspace(int k, spff_shape s, int g);
/* Statistics of the temperature fit on an accumulator of spff_head_prob_accum (p̄_c = scale * acc_c): for every voxel
 * whose label y (uint8 or int64 [N,D,H,W]) is in [0,K) and not ignore_index, and each grid value β_g (betas: fp32 [g]
 * on the device, each positive and finite; not checked, as the host does not read device memory),
 *   f(β)  = log sum_{c: p̄_c > 0} exp(β log p̄_c) - β log p̄_y   (the tempered nll; -log FLT_MIN when p̄_y = 0)
 *   f'(β) = sum_c p̃_c log p̄_c - log p̄_y                        (0 when p̄_y = 0)
 * sums fp64 [2][g] (+=) receives sum f(β_g) in [0][g] and sum f'(β_g) in [1][g], counted (+=) the voxels. f is convex
 * in β. Per-block fp64 partials in the workspace are added in a fixed order: bit-reproducible, no float atomics.
 * k in [2,16], g in [1,64], acc 16-byte aligned, N <= 65535; workspace of spff_prob_temp_fit_workspace(k, s, g) bytes
 * (SPFF_ERR_WORKSPACE otherwise). Compute-bound: g x k exponentials per voxel. */
int spff_prob_temp_fit(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                       int ignore_index, const float* betas, int g, double* sums, long long* counted, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- "3DUNet" control: Cicek3DUNet + depth adapter (models.py:718-777; config.py:283-311) ---------------
 * Its 3x3x3 convolutions, normalise + ReLU passes (slope 0), head and loss are the entry points above;
 * the ones below are what only this variant needs. */
/* ConvTranspose3d kernel = stride = (2,2,2) with bias (models.py:733-739). `s` = coarse grid; the fine
 * tensors are [n, 2d, 2h, 2w, c]. Weight [cin][cout][2][2][2] fp32, packed like the (1,2,2) one with 8 taps. */
int spff_pack_convt_weight_k222(const float* w, void* w_fwd, void* w_dgrad, int cin, int cout, void* stream);
int spff_convt_k222_fwd(const void* x, long long ldx, int cin, const void* w_fwd, const float* bias, void* y,
                        long long ldy, int cout, spff_shape s, void* stream);
int spff_convt_k222_dgrad(const void* dy, long long lddy, int cout, const void* w_dgrad, void* dx, long long lddx,
                          int cin, spff_shape s, void* stream);
size_t spff_convt_k222_wgrad_workspace(int cin, int cout, spff_shape s);
int spff_convt_k222_wgrad(const void* x, long long ldx, int cin, const void* dy, long long lddy, int cout,
                          spff_shape s, float* dw, float beta, void* workspace, size_t workspace_bytes,
                          void* stream);
/* Depth-only resampling y[n][do][e] = sum_di matrix[do][di] * x[n][di][e] over `inner` contiguous elements per
 * plane (bf16: elem_bytes 2, fp32: 4). F.interpolate(mode="trilinear", align_corners=False) with H, W unchanged
 * (`_resize_depth_like` / `_resize_logits_depth_like`, models.py:153-163) is such a matrix; its backward is the
 * same call with the transposed matrix. matrix: device fp32 [dout][din], din, dout <= 32. */
int spff_depth_resample(const void* x, void* y, int elem_bytes, int n, int din, int dout, long long inner,
                        const float* matrix, void* stream);
/* BatchNorm3d(c) coefficients (models.py:721; F.batch_norm): batch statistics over (n, d, h, w) from either the
 * conv epilogue's partials [n][slots][2][c] or spff_in_stats' stats [n][c][2] (exactly one non-NULL), summed in
 * a fixed order in double; coef[k][c] = {A, B, mean, rstd} is written for every sample k (the layout the
 * normalise kernels read). Training (eval == 0) also updates running_mean / running_var (momentum, unbiased
 * variance; may be NULL). eval != 0: coefficients from the running statistics. count = d*h*w per sample. */
size_t spff_bn_coeffs_workspace(int c);
int spff_bn_coeffs(const float* partial, int slots, const double* stats, const float* gamma, const float* beta, float eps,
                   int n, int c, long long count, float momentum, float* running_mean, float* running_var, int eval,
                   float* coef, void* workspace, size_t workspace_bytes, void* stream);
/* BatchNorm backward coefficients from R (slots 2 and 4 of spff_norm_act_bwd_reduce, plain mode):
 * bcoef[k][c] = {gamma*rstd, mean(dz), mean(dz*xhat), 0} with BATCH means, dgamma[c] += , dbeta[c] += . */
int spff_bn_bwd_coeffs(const float* R, const float* coef, const float* gamma, int c, spff_shape s, float* bcoef,
                       float* dgamma, float* dbeta, void* stream);
/* nn.MaxPool3d(2) (models.py:728-731): ypool [n, d/2, h/2, w/2, c]; backward scatters dpool to the first
 * maximum of each 2x2x2 window of y and adds it to dskip (accumulate != 0) or overwrites dskip. `s` = full grid. */
int spff_maxpool222_fwd(const void* y, long long ldy, void* ypool, long long ldp, int c, spff_shape s, void* stream);
int spff_maxpool222_bwd_add(const void* dpool, long long ldp, const void* y, long long ldy, void* dskip, long long ldd, int c,
                            spff_shape s, int accumulate, void* stream);
/* torch.optim.SGD(lr, momentum, nesterov, weight_decay), dampening 0 (models.py:844-846). first_step != 0: the
 * momentum buffer is initialised with the gradient. grad is scaled by grad_scale first (1/world under DP). */
int spff_sgd_step(float* param, const float* grad, float* momentum_buf, long long n, float lr, float momentum,
                  float weight_decay, int nesterov, int first_step, float grad_scale, void* stream);

/* ---- per-step scalars of the fused training step (no framework launches inside fit_step) ----------------------
 * Number of labels != ignore_index (the CE normaliser N_valid of F.cross_entropy, helpers.py:798); labels uint8 or int64. */
int spff_count_valid(const void* labels, int label_bytes, long long total, int ignore_index, unsigned long long* out,
                     void* stream);
/* g[i] *= factor / count (0 when count == 0): the fused step back-propagates the SUM of the per-voxel CE terms and divides
 * the finished gradients by N_valid here (F.cross_entropy's mean reduction, helpers.py:798), so that a group's backward
 * needs only its own labels on the device, not the whole batch's. */
int spff_scale_by_count(float* g, long long n, const unsigned long long* count, float factor, void* stream);
/* ce_plus_macro_dice_loss (helpers.py:782-803) from the tally spff_head_loss_fused / spff_ce_confusion accumulate:
 * out = nll / max(count, 1) + 0.5 * (1 - mean_{c=1..k-1} (2tp+s)/(2tp+fp+fn+s)), confusion [label][argmax]. */
int spff_loss_from_tally(const double* nll, const unsigned long long* count, const unsigned long long* confusion, int k,
                         double smooth, float* out, void* stream);
/* out[c] += sum_r m[r * row_stride + c] for c < cols (double accumulation, fixed order): the bias gradient of a
 * ConvTranspose3d from the column sums spff_conv3d_k3_dgrad_stats left per work item (models.py:668-672). */
size_t spff_partial_colsum_workspace(int cols);
int spff_partial_colsum(const float* m, long long rows, long long row_stride, int cols, float* out, void* workspace,
                        size_t workspace_bytes, void* stream);
/* ---- optimizer (models.py:591-594: torch.optim.Adam, lr 1e-4, betas (0.9,0.999), eps 1e-8) -------- */
int spff_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float grad_scale, void* stream);

/* ---- data path feeding the step (SURVEY.md §8f-4) -------------------------------------------------------
 * Phantom label rasterisation: labels[f][y][x] (int64, frames x height x width) = label of the LAST roi
 * (x0, y0, w0, h0, label — HOST array of nroi x 5 ints, nroi <= 64) whose inscribed ellipse contains the pixel,
 * else 0: the per-pixel loop of create_image_and_labels_for_dataset + is_pixel_in_ellipse
 * (helpers.py:125-129, 197-206), double arithmetic in the reference's order, numpy's negative-index wrap. */
int spff_roi_labels(const int* rois_host, int nroi, int frames, int height, int width, long long* labels, void* stream);
/* TrainGridAug (datasets.py:134-206) over a batch: xo[n][f][h][w] = jitter(x[n][f][A[u]][B[v]]) (+ noise, + stamp),
 * (u, v) = (h, w) or, for transposed[n] != 0 (odd rot90; needs h == w), (w, h); labels gathered the same way.
 * amap [n][h], bmap [n][w]: the composition of the flips, the rotation and the stripe shuffle
 * (_shuffle_stripes, datasets.py:56-121) drawn by the host; scale/shift [n]: x*scale + shift (1, 0 = none);
 * noise_cap [n]: noise_std of samples that get noise (amplitude min(noise_cap, 0.25*std(x)), datasets.py:180-184),
 * 0 = none; seed [n]; stamp [n]: non-zero writes x[n][0][:32][:32] = max(region) + max(max|x|, 1)*0.25
 * (datasets.py:196-201). x fp32 [n][frames][h][w]; y uint8 / int64 or NULL. Not in place. */
size_t spff_grid_aug_workspace(int n);
int spff_grid_aug(const float* x, const void* y, int label_bytes, float* xo, void* yo, int n, int frames, int h, int w,
                  const int* amap, const int* bmap, const int* transposed, const float* scale, const float* shift,
                  const float* noise_cap, const unsigned long long* seed, const int* stamp, int any_noise, int any_stamp,
                  void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPFF_B200_H_ */
