/*
 * agcn_b200.h -- C ABI of the B200-native AGCN / MMARGCN hot path (libagcn_b200.so).
 *
 * The reference (mduhme/fusion-gcn) is pure Python on top of ATen; it has no FFI of its own.
 * The boundary this library replaces is therefore the set of ATen calls made by
 *   torch_src/models/mmargcn/agcn.py:37-136  (TemporalConv, SpatialGraphConv, SpatialTemporalConv)
 *   torch_src/models/agcn/agcn.py:38-133     (unit_tcn, unit_gcn, TCN_GCN_unit)
 *   torch_src/models/mmargcn/agcn.py:183-200 (Model.forward: data_bn, pooling, fc)
 * Each entry point below cites the reference lines whose arithmetic it performs.  A maintainer
 * binds them with ctypes (see INTEGRATION.md); fusion_gcn_b200/capi.py is that binding.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer to fp32 data owned by the caller (PyTorch); the library
 *     borrows it for the duration of the stream-ordered call.  It never allocates, never
 *     synchronises the device and never changes the current device.  Scratch space is passed in as
 *     (workspace, workspace_bytes); the *_workspace_bytes functions say how much is needed.
 *   - Activations are channels-last: x[nb][t][v][c], c contiguous.  nb = N*M person-sequences.
 *     "rows" means the flattened (nb, t, v) index.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - Return value: 0 on success, otherwise an agcn_status code; agcn_last_error_string() gives a
 *     thread-local description.  Entry points are thread-safe (no global mutable state other than
 *     the thread-local error string) and CUDA-graph-capture safe (no allocation, no host sync).
 *   - `precision`: see agcn_precision.  AGCN_PREC_FP32 meets the 1e-4 parity tolerance against the reference;
 *     AGCN_PREC_TF32 has its own tolerance and is reported separately.
 */
#ifndef AGCN_B200_H
#define AGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    AGCN_OK = 0,
    AGCN_ERR_BAD_SHAPE = 1,    /* non-positive or inconsistent dimensions                       */
    AGCN_ERR_UNSUPPORTED = 2,  /* valid but outside what the kernels cover (e.g. V > 32)         */
    AGCN_ERR_MISALIGNED = 3,   /* pointer not aligned for the vector width the shape implies     */
    AGCN_ERR_WORKSPACE = 4,    /* workspace_bytes smaller than *_workspace_bytes(...)            */
    AGCN_ERR_CUDA = 5,         /* a CUDA runtime call or launch failed                           */
    AGCN_ERR_NULL = 6          /* required pointer is NULL                                       */
} agcn_status;

typedef enum {
    AGCN_PREC_FP32 = 0,       /* fp32 parity mode: 3xTF32 error-compensated tcgen05 MMAs where the shape allows, FFMA otherwise */
    AGCN_PREC_TF32 = 1,       /* single-pass tcgen05 kind::tf32 (operands truncated to TF32); own tolerance             */
    AGCN_PREC_FP32_FFMA = 2,  /* force the FFMA kernels (reference path for tests)                                       */
    AGCN_PREC_BF16X3 = 3      /* second fp32 parity mode: x = h + m (two bf16 pieces), products h.h + h.m + m.h on tcgen05
                                 kind::f16 -- half the tensor time and operand bytes of 3xTF32, ~1e-5 unit-level error (inside
                                 the 1e-4 contract); stages without a BF16x3 kernel run their 3xTF32 kernel                */
} agcn_precision;

/* joint-mix modes (agcn_joint_mix) */
typedef enum {
    AGCN_MIX_AGG_FWD = 0,   /* out[.,v,k*w+c]  = sum_u in[.,u,c]      * mat[nb,k,u,v]     (agcn.py:110 forward)  */
    AGCN_MIX_AGG_BWD = 1,   /* out[.,u,c]     (+)= sum_k sum_v in[.,v,k*w+c] * mat[nb,k,u,v] (its input gradient) */
    AGCN_MIX_SCORE_BWD = 2  /* in = [theta_0,phi_0,theta_1,...] (6 groups of w), mat = dS:
                               dtheta_k[.,u,c] = sum_v mat[k,u,v]*phi_k[.,v,c];  dphi_k[.,v,c] = sum_u mat[k,u,v]*theta_k[.,u,c]
                               (gradient of agcn.py:104-106)                                                     */
} agcn_mix_mode;

/* residual modes of agcn_bn_apply */
typedef enum { AGCN_RES_NONE = 0, AGCN_RES_TENSOR = 1, AGCN_RES_AFFINE = 2 } agcn_res_mode;

int agcn_version(void);
const char* agcn_last_error_string(void);
/* Number of CUDA kernels this library has launched in this process (monotonic; used by bench.py's gpu_launches). */
long long agcn_launch_count(void);

/* ---- dense contractions over the channel dimension ------------------------------------------------
 * Implicit GEMM with an optional temporal tap structure:
 *   y[nb][to][v][co] (+)= bias[co] + sum_{tap<taps} sum_{ci<cin} x[nb][ti(to,tap)][v][ci] * w[co][tap][ci]
 *   forward gather    (transposed=0): ti = stride*to + tap - pad
 *   transposed gather (transposed=1): ti = (to + pad - tap)/stride, used only when divisible
 * out-of-range ti contribute zero.  x: [nb][t_in][v][cin], y: [nb][t_out][v][cout], w: [cout][taps][cin].
 * Replaces nn.Conv2d forward / input-gradient at agcn.py:41-42 (9x1 temporal conv, residual 1x1 with
 * stride), :71-73 (conv_a / conv_b / conv_d 1x1), :77 (down) and nn.Linear at :178 (taps=1, v=1, t=1).
 * bias may be NULL.  accumulate!=0 adds into y instead of overwriting it.
 * workspace: agcn_conv_fwd_workspace_bytes(...) bytes of scratch (holds the TF32 hi/lo split of the weights in the
 * 3xTF32 path); may be NULL / 0, in which case AGCN_PREC_FP32 runs on the FFMA kernel.                  */
size_t agcn_conv_fwd_workspace_bytes(int cin, int cout, int taps, int precision);
int agcn_conv_fwd(const float* x, const float* w, const float* bias, float* y,
                  int nb, int t_in, int t_out, int v, int cin, int cout,
                  int taps, int stride, int pad, int transposed, int accumulate,
                  int precision, void* workspace, size_t workspace_bytes, void* stream);

/* Eval-mode convolution with its tail fused (model.eval(), torch_src/session/session.py:188-194, session/evaluation.py:36-56):
 * BatchNorm with running statistics is a per-channel affine, so Conv2d -> BatchNorm2d [-> + residual] [-> ReLU]
 * (agcn.py:49-51, 110-115, 134-136) is ONE pass:   y = act( scale[co] * (conv(x, w) + bias[co]) + shift[co] + res )
 * scale / shift: [cout] or both NULL (no affine); res: tensor of y's shape or NULL; relu != 0 applies max(., 0).
 * Forward gather only.  Same workspace as agcn_conv_fwd.                                                              */
int agcn_conv_fwd_post(const float* x, const float* w, const float* bias,
                       const float* scale, const float* shift, const float* res, int relu, float* y,
                       int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad,
                       int precision, void* workspace, size_t workspace_bytes, void* stream);

/* agcn_conv_fwd (forward gather, no accumulate) whose epilogue also leaves the per-channel sums the training-mode
 * BatchNorm that follows needs (nn.Conv2d -> nn.BatchNorm2d pairs at agcn.py:41-51,73-83): stat_part receives
 * [*stat_nparts][4][cout] floats: per partial (a fixed set of rows, deterministic) and channel the SHIFTED sums
 *   sum(y - p) | sum((y - p)^2) | p | number of rows,   p = the first value of the channel the partial saw,
 * to be combined by agcn_bn_finalize (pairwise-variance merge in fp64: E[y^2] - mean^2 on raw fp32 sums loses the variance
 * of channels with |mean| >> sigma).  *stat_nparts == 0 on return means the fused epilogue does not cover this shape:
 * y is complete, run agcn_bn_stats on it.  stat_part: agcn_conv_fwd_stats_bytes(cout) bytes, 16-byte aligned.
 * stat_nparts is a HOST pointer.                                                                          */
size_t agcn_conv_fwd_stats_bytes(int cout);
int agcn_conv_fwd_stats(const float* x, const float* w, const float* bias, float* y,
                        int nb, int t_in, int t_out, int v, int cin, int cout,
                        int taps, int stride, int pad,
                        int precision, void* workspace, size_t workspace_bytes,
                        float* stat_part, size_t stat_part_bytes, int* stat_nparts, void* stream);

/* Weight / bias gradient of the forward-gather contraction above:
 *   dw[co][tap][ci] = sum_rows dy[nb][to][v][co] * x[nb][stride*to+tap-pad][v][ci];   dbias[co] = sum_rows dy
 * Deterministic (two-phase split reduction, no atomics).  dbias may be NULL.                            */
size_t agcn_conv_wgrad_workspace_bytes(int nb, int t_in, int t_out, int v, int cin, int cout, int taps);
int agcn_conv_wgrad(const float* dy, const float* x, float* dw, float* dbias,
                    int nb, int t_in, int t_out, int v, int cin, int cout,
                    int taps, int stride, int pad,
                    void* workspace, size_t workspace_bytes, int precision, void* stream);

/* The same weight gradient (no bias gradient) from operands that ARRIVE split into the bf16 pieces the
 * parity modes multiply: dy_split [2][nb*t_out*v][cout], x_split [2][nb*t_in*v][cin] bf16, plane 0 = h = bf16(value), plane 1 =
 * m = bf16(value - h) -- written by agcn_bn_apply / agcn_bn_bwd (out_split / dy_split), the kernels that produce the activations
 * and their gradients anyway.  The in-kernel conversion of agcn_conv_wgrad is what bounds it (shared-memory bandwidth); without
 * it the kernel runs at the tensor rate of three bf16 MMAs.  Same workspace as agcn_conv_wgrad.  Returns AGCN_ERR_UNSUPPORTED
 * (no error string) unless cin and cout are multiples of 64.                                                                   */
int agcn_conv_wgrad_presplit(const void* dy_split, const void* x_split, float* dw,
                             int nb, int t_in, int t_out, int v, int cin, int cout, int taps, int stride, int pad,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- joint x joint products (the V x V attention) --------------------------------------------------
 * out[nb][chunk][g][u][v] = sum_{t in chunk} sum_{c<width} a[nb][t][u][offa+g*stridea+c] * b[nb][t][v][offb+g*strideb+c]
 * a: [nb][t][v][lda], b: [nb][t][v][ldb].  The t axis is split into nchunk contiguous chunks so that a
 * grid of nb*nchunk CTAs fills the GPU; the consumer sums the chunks in a fixed order.
 * Used for the score theta^T phi (agcn.py:104-106, a = b = [theta|phi] embedding) and for
 * dG = X^T dZ (gradient of agcn.py:110).  V <= 32 on the shared-memory-resident kernels; larger graphs: see agcn_node_mix.
 * precision: AGCN_PREC_FP32 / AGCN_PREC_TF32 run the contraction on the tensor cores (3xTF32 / single-pass TF32) when
 * groups == 3, 3*V <= 80 and width is 16 (theta|phi sharing a 32-channel row) or a multiple of 32; every other shape and
 * AGCN_PREC_FP32_FFMA use the FFMA kernel.                                                                */
int agcn_joint_gram(const float* a, const float* b, float* out,
                    int nb, int t, int v, int lda, int ldb, int groups,
                    int offa, int stridea, int offb, int strideb, int width, int nchunk, int precision, void* stream);

/* p[nb][k][:, v] = softmax_u(scale * sum_chunk s_part[nb][chunk][k][u][v]);  g = p + adj_a[k] + adj_b[k]
 * (agcn.py:98-100,106-108; softmax over dim -2, i.e. columns sum to one).                               */
int agcn_attention_fwd(const float* s_part, const float* adj_a, const float* adj_b, float* p, float* g,
                       int nb, int nchunk, int groups, int v, float scale, void* stream);

/* dG = sum_chunk dg_part;  ds = scale * p * (dG - colsum_u(p*dG));  dadj_b[k] = sum_nb dG[nb][k]
 * dg_sum: [nb][k][v][v] scratch output (the summed dG).                                                 */
int agcn_attention_bwd(const float* dg_part, const float* p, float* dg_sum, float* ds, float* dadj_b,
                       int nb, int nchunk, int groups, int v, float scale, void* stream);

/* Per-sample mixing over the joint axis, see agcn_mix_mode.  in: [nb][t][v][ldin], out: [nb][t][v][ldout],
 * mats: [nb][3][v][v], width = channels per group.  V <= 32 on the resident kernels (larger graphs: batched FFMA GEMMs).
 * precision: AGCN_PREC_FP32 / AGCN_PREC_TF32 run the mix on the tensor cores (3xTF32 / single-pass TF32) when width is a
 * multiple of 32 (AGCN_MIX_AGG_FWD / AGCN_MIX_AGG_BWD) or of 16 (AGCN_MIX_SCORE_BWD) and the workspace holds
 * agcn_joint_mix_workspace_bytes(nb) bytes (zero-padded copies of the matrices); every other case and
 * AGCN_PREC_FP32_FFMA use the FFMA kernel (workspace may then be NULL).                                                     */
size_t agcn_joint_mix_workspace_bytes(int nb);
int agcn_joint_mix(const float* in, const float* mats, float* out,
                   int nb, int t, int v, int ldin, int ldout, int width, int mode, int accumulate,
                   int precision, void* workspace, size_t workspace_bytes, void* stream);

/* AGCN_MIX_SCORE_BWD (in = e [nb][t][v][6*width], mats = dS, out = de) whose epilogue also leaves colsum[6*width] = sum over all
 * (nb, t, v) rows of out -- the bias gradient of the theta / phi convolutions (agcn.py:104-105) -- instead of a separate pass over
 * the 1.5 x Cout-wide tensor.  Tensor-core path only: returns AGCN_ERR_UNSUPPORTED (no error string) for shapes / modes it does
 * not take (V > 32, width not 16 / a multiple of 32, 6*width > 384, AGCN_PREC_FP32_FFMA); use agcn_joint_mix then.            */
size_t agcn_joint_mix_score_bwd_colsum_workspace_bytes(int nb, int width);
int agcn_joint_mix_score_bwd_colsum(const float* in, const float* mats, float* out, float* colsum,
                                    int nb, int t, int v, int width, int precision,
                                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- BatchNorm (training-mode batch statistics; nn.BatchNorm2d/1d at agcn.py:44,78,83,150) ----------
 * The tensor is addressed as x[outer][inner][c] with element offset outer*outer_stride + inner*c_total...
 * precisely: offset(o, i, ch) = o*outer_stride + i*channels + ch, rows = outer*inner.  For unit tensors
 * outer=1... (outer_stride ignored when outer==1); data_bn uses outer=N, inner=T, channels=V*C per body.
 *
 * training!=0: batch mean / biased variance over rows (eps as given; from sums shifted by the first row of x, so
 *   channels with |mean| >> sigma keep their variance), running statistics updated in
 *   place with `momentum` and the unbiased variance, *num_batches_tracked incremented (may be NULL).
 * training==0: scale/shift from the running statistics.
 * Outputs: scale[c] = gamma*invstd, shift[c] = beta - mean*scale, save_mean[c], save_invstd[c].          */
size_t agcn_bn_workspace_bytes(int channels);
int agcn_bn_stats(const float* x, int outer, int inner, long long outer_stride, int channels,
                  const float* gamma, const float* beta, float* running_mean, float* running_var,
                  long long* num_batches_tracked, float momentum, float eps, int training,
                  float* scale, float* shift, float* save_mean, float* save_invstd,
                  void* workspace, size_t workspace_bytes, void* stream);

/* The finalize half of agcn_bn_stats (training mode) on the partials produced by agcn_conv_fwd_stats:
 * part[nparts][4][channels] (shifted sum | shifted sum of squares | pivot | row count), rows = number of rows they cover. */
int agcn_bn_finalize(const float* part, int nparts, long long rows, int channels,
                     const float* gamma, const float* beta, float* running_mean, float* running_var,
                     long long* num_batches_tracked, float momentum, float eps,
                     float* scale, float* shift, float* save_mean, float* save_invstd, void* stream);

/* out = act(scale*y + shift + R),  R = 0 | res | scale2*res + shift2;  act = ReLU when relu!=0.
 * (agcn.py:113-115 and :135-136).  Same addressing as agcn_bn_stats for y / res / out.
 * Two optional outputs (NULL: not written) for the backward:
 *   mask_bits: the ReLU mask (out > 0) as ONE BIT per element, bit e & 31 of word e >> 5, e = row * channels + c, for
 *     agcn_bn_bwd (its two passes then read 1/32 of the mask bytes).  Needs agcn_bn_mask_words(outer, inner, channels) > 0.
 *   out_split: `out` once more as the bf16 pieces the parity modes multiply, [2][inner][channels] bf16, plane 0 = h = bf16(out),
 *     plane 1 = m = bf16(out - h) -- the operand format of agcn_conv_wgrad_presplit.  One more plane written by a kernel that
 *     streams the tensor anyway, instead of a conversion pass in shared memory for every tile of the weight gradient.
 *     Needs outer == 1 and a vectorisable layout.
 * An optional output the layout does not support is AGCN_ERR_UNSUPPORTED.                                                */
int agcn_bn_apply(const float* y, const float* scale, const float* shift,
                  int res_mode, const float* res, const float* scale2, const float* shift2,
                  int relu, float* out, unsigned* mask_bits, void* out_split,
                  int outer, int inner, long long outer_stride, int channels, void* stream);

/* Number of 32-bit words of the bit mask of agcn_bn_apply, or 0 when the layout is not supported (outer != 1, channels not a
 * multiple of 4, channels/4 not a divisor of 256) -- use the fp32 tensor as the mask then.                              */
size_t agcn_bn_mask_words(int outer, int inner, int channels);

/* BatchNorm backward through an optional ReLU mask:
 *   g = dout * [mask > 0]  (g = dout without a mask)
 *   dbeta = sum g;  dgamma = sum g*xhat;  dy = gamma*invstd*(g - dbeta/m - xhat*dgamma/m),  xhat = (y-mean)*invstd
 * The mask is the fp32 tensor mask_out (addressed like y) or the bits of agcn_bn_apply (mask_bits), never both; both NULL: no mask.
 * If dres != NULL the masked gradient g is also written (dres_accumulate==0) or added to dres
 * (gradient of an identity residual / of the tensor R above).  dy may be NULL (only sums wanted).
 * dy_split (NULL: not written; needs dy): dy once more as bf16 pieces, layout and restrictions of agcn_bn_apply's out_split.
 * frozen_stats != 0: mean / invstd are constants -- the backward of an eval-mode BatchNorm on its running statistics (the
 *   reference's autograd under model.eval()): dy = gamma*invstd*g, dgamma and dbeta as above.  Only with pool_rows == 0 and phase 0.
 * pool_rows > 0 (with mask_bits, outer == 1): dout is the pooled gradient of agcn_bn_apply_pool, [inner / pool_rows][channels],
 *   broadcast over its group: dout[row][c] = dpooled[row / pool_rows][c] / pool_rows.
 * phase 0: the whole backward.  Phases 1 and 2 are the two halves of a synchronised BatchNorm, either side of the caller's
 *   all-reduce: phase 1 writes only dgamma / dbeta = this rank's sums (sum g xhat | sum g); phase 2 writes dy (dy_split, dres) from
 *   global_sums [2][channels] = (sum g | sum g xhat) all-reduced over the ranks and global_rows = the rows of all ranks.
 *   global_sums / global_rows are read in phase 2 only.
 * workspace: agcn_bn_workspace_bytes(channels).                                                                              */
int agcn_bn_bwd(const float* dout, const float* mask_out, const unsigned* mask_bits, const float* y,
                const float* save_mean, const float* save_invstd, const float* gamma,
                float* dy, void* dy_split, float* dgamma, float* dbeta, float* dres, int dres_accumulate,
                int frozen_stats, int outer, int inner, long long outer_stride, int channels, int pool_rows,
                int phase, const float* global_sums, double global_rows,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- pooling (agcn.py:194-196): out[g][c] = mean over rows_per_group rows of x[g][row][c] ------------ */
int agcn_pool_fwd(const float* x, float* out, int groups, int rows_per_group, int channels, void* stream);
int agcn_pool_bwd(const float* dout, float* dx, int groups, int rows_per_group, int channels, void* stream);

/* Fused tail of the model: the last unit's out = relu(scale*y + shift + R) (agcn.py:135-136) feeds only the global mean pool
 * x.view(N, M, C, -1).mean(3).mean(1) (agcn.py:194-196), so `out` is never written: agcn_bn_apply_pool leaves the pooled means
 * pooled[groups][channels] (group g = rows [g*rows_per_group, (g+1)*rows_per_group)) and the ReLU mask bits (layout of
 * agcn_bn_apply); its backward is agcn_bn_bwd with pool_rows = rows_per_group.  channels must be a multiple of 32 with
 * agcn_bn_mask_words(1, groups*rows_per_group, channels) > 0, else AGCN_ERR_UNSUPPORTED (use the unfused calls).                  */
size_t agcn_bn_apply_pool_workspace_bytes(int groups, int channels);
int agcn_bn_apply_pool(const float* y, const float* scale, const float* shift,
                       int res_mode, const float* res, const float* scale2, const float* shift2,
                       unsigned* mask_bits, float* pooled, int groups, int rows_per_group, int channels,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Two BatchNorm backwards over the SAME masked upstream gradient in one pair of passes: the gcn half's bn and down.1 both feed the
 * ReLU of agcn.py:113-115, the temporal BatchNorm and the residual branch's both feed the one of agcn.py:135-136, so g = dout * mask
 * is read once per pass for both (8 plane passes instead of 10).  BatchNorm A may also leave dy_a as bf16 pieces (dy_a_split, see
 * agcn_bn_bwd).  workspace: 2 x agcn_bn_workspace_bytes(channels).  Returns AGCN_ERR_UNSUPPORTED (no error string) for
 * layouts without a bit mask (agcn_bn_mask_words == 0): call agcn_bn_bwd twice then.                                             */
int agcn_bn_bwd_bits_dual(const float* dout, const unsigned* mask_bits,
                          const float* y_a, const float* mean_a, const float* invstd_a, const float* gamma_a,
                          float* dy_a, void* dy_a_split, float* dgamma_a, float* dbeta_a,
                          const float* y_b, const float* mean_b, const float* invstd_b, const float* gamma_b,
                          float* dy_b, float* dgamma_b, float* dbeta_b,
                          int frozen_stats, int inner, int channels, void* workspace, size_t workspace_bytes, void* stream);

/* ---- synchronised BatchNorm halves (SURVEY 8e: optional SyncBN mode for the data-parallel path; the reference's nn.BatchNorm2d,
 * agcn.py:44,78,83,150, computes its batch statistics over the whole batch, which a batch-sharded run only reproduces when the
 * statistics are taken over all ranks).  The collectives stay with the caller; the library provides the halves either side of them.
 * agcn_bn_stats_partials: part [nparts][4][channels] = per row partition the shifted sum | shifted sum of squares | pivot | row count
 * of x -- the layout agcn_conv_fwd_stats writes and agcn_bn_finalize merges, so the partials of all ranks are concatenated
 * (all-gather) and finalised with rows = the global row count.  The backward halves are agcn_bn_bwd phases 1 and 2.             */
size_t agcn_bn_stats_partials_bytes(int channels);
int agcn_bn_stats_partials(const float* x, int outer, int inner, long long outer_stride, int channels,
                           float* part, size_t part_bytes, int* nparts, void* workspace, size_t workspace_bytes, void* stream);

/* ---- classifier head fused with its loss -------------------------------------------------------------
 * logits = x . w^T + bias (nn.Linear, agcn.py:178,198-199) and loss = mean_n( logsumexp(logits[n]) - logits[n][label[n]] )
 * (nn.CrossEntropyLoss with its defaults, torch_src/session/session.py:53 applied at procedures/step.py:41-42), one launch.
 * Also leaves dlogits[n][c] = (softmax(logits[n])[c] - [c == label[n]]) / n for the backward and the per-sample losses.
 * x: [n][cin], w: [ncls][cin], labels: int64 [n] in [0, ncls).  agcn_linear_ce_bwd: with g = *grad_loss (device scalar, may be
 * NULL = 1): dw = g * dlogits^T x, dbias = g * colsum(dlogits), dx = g * dlogits w (dbias / dx may be NULL).            */
int agcn_linear_ce_fwd(const float* x, const float* w, const float* bias, const long long* labels,
                       float* logits, float* dlogits, float* loss_per_sample, float* loss,
                       int n, int cin, int ncls, void* stream);
int agcn_linear_ce_bwd(const float* x, const float* w, const float* dlogits, const float* grad_loss,
                       float* dw, float* dbias, float* dx, int n, int cin, int ncls, void* stream);

/* ---- multi-tensor optimizer steps (torch_src/session_helper.py:48-82 builds torch.optim.{SGD, Adam, AdamW};
 * torch_src/session/procedures/step.py:48-49,67-71 steps them, under GradScaler with --mixed_precision) ------------
 * ONE launch updates every parameter tensor of a group.  `table`: device array of rows
 *     { float* param; const float* grad; float* state1; float* state2; long long numel; }      (40 bytes each)
 * `items`: device array of (row index, chunk index) int pairs, one per agcn_optim_chunk() elements of every tensor.
 * lr_dev (may be NULL) overrides `lr` with a device scalar, so a captured CUDA graph follows a learning-rate schedule.
 * grad_scale / found_inf (may be NULL) are GradScaler's device scalars: gradients are divided by *grad_scale and the
 * whole step is skipped when *found_inf != 0 -- no host synchronisation.  Hyper-parameters are doubles (Python floats): 1 - beta
 * and the Adam bias corrections are formed in double before they are rounded to fp32, as torch.optim does on the host.
 * SGD  (torch/optim/sgd.py): g += wd*p; buf = first_step ? g : momentum*buf + (1-dampening)*g (state1);
 *                            g = nesterov ? g + momentum*buf : buf; p -= lr*g.
 * Adam (torch/optim/adam.py): state1 = exp_avg, state2 = exp_avg_sq, *step_dev = steps completed before this one (the caller
 *                            increments it afterwards); decoupled != 0 is AdamW (p *= 1 - lr*wd instead of g += wd*p). */
int agcn_optim_chunk(void);
int agcn_optim_sgd(const void* table, const int* items, int nitems, double lr, const float* lr_dev,
                   double momentum, double dampening, double weight_decay, int nesterov, int first_step,
                   const float* grad_scale, const float* found_inf, void* stream);
int agcn_optim_adam(const void* table, const int* items, int nitems, double lr, const float* lr_dev,
                    double beta1, double beta2, double eps, double weight_decay, int decoupled,
                    const float* step_dev, const float* grad_scale, const float* found_inf, void* stream);

/* Node mixing with ONE fixed matrix for the whole batch -- STGCNGraphConvolution's support . adj^T
 * (torch_src/models/mmargcn/graph_convolution.py:45) and its input gradient:
 *   out[b][v][c] (+)= sum_u mat[v][u] * in[b][u][c]   (transpose_mat == 0)      sum_u mat[u][v] * in[b][u][c]   (transpose_mat != 0)
 * in / out: [batch][v][channels] channels-last, mat: [v][v].  Any V (the IMU graphs have up to 652 nodes).  The adaptive 1-D
 * graph convolution (graph_convolution.py:56-113) runs on agcn_joint_gram / agcn_attention_* / agcn_joint_mix with t = 1: for
 * V > 32 those entry points switch to batched FFMA GEMMs over the node axis (nchunk must then be 1).                            */
int agcn_node_mix(const float* in, const float* mat, float* out, int batch, int v, int channels,
                  int transpose_mat, int accumulate, void* stream);

/* Gradient buckets of the data-parallel all-reduce (the reference has no distributed code; SURVEY 8e): ONE launch packs the
 * gradients of a bucket's parameters into its flat buffer (to_flat != 0) or writes the reduced values back scaled by `scale`
 * (1 / world size).  Same table layout as the optimizer steps with param = flat slice, grad = the tensor.                     */
int agcn_bucket_copy(const void* table, const int* items, int nitems, int to_flat, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AGCN_B200_H */
