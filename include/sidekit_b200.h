/* sidekit_b200 -- C ABI of the B200-native speaker-verification inference hot path.
 *
 * The reference (deep-privacy/sidekit) is pure Python over PyTorch/numpy and has no FFI: its
 * boundary for this path is the Python API (SURVEY.md 8b).  Each entry point below names the
 * reference interface it replaces; sidekit_b200/*.py binds them with ctypes and re-creates the
 * reference's Python signatures on top (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions: plain pointers and sizes only; `*_dev` pointers are CUDA device pointers on the
 * current device, everything else is host memory; `stream` is a cudaStream_t passed as void*
 * (NULL = default stream); every function returns SKB_OK (0) or a negative error code and
 * skb_last_error() then describes the failure.  Calls on one handle must not overlap.
 */
#ifndef SIDEKIT_B200_H
#define SIDEKIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKB_OK 0
#define SKB_ERR_ARG (-1)
#define SKB_ERR_CUDA (-2)
#define SKB_ERR_WEIGHTS (-3)
#define SKB_ERR_STATE (-4)

#define SKB_ARCHI_HALFRESNET34 0 /* Xtractor(model_archi="halfresnet34"), sidekit/nnet/xvector.py:569-599 */
#define SKB_ARCHI_XVECTOR 1      /* Xtractor(model_archi="xvector") TDNN,  sidekit/nnet/xvector.py:453-498 */
#define SKB_ARCHI_RESNET34 2     /* Xtractor(model_archi="resnet34"): PreResNet34 trunk (128/256 channels, 7 layers),
                                    sidekit/nnet/res_net.py:430-498, sidekit/nnet/xvector.py:516-540 */
#define SKB_ARCHI_FASTRESNET34 3 /* Xtractor(model_archi="fastresnet34"): PreFastResNet34 trunk (7x7 stride-(1,2) stem, 16/32/64/128
                                    channels), sidekit/nnet/res_net.py:557-610, sidekit/nnet/xvector.py:539-567 */

typedef struct skb_xtractor skb_xtractor_t;

int skb_version(void);
const char* skb_last_error(void);
/* Number of CUDA kernels launched by this library since process start (bench.py reports deltas). */
int64_t skb_kernel_launches(void);

/* Device-time attribution for bench.py's roofline: while enabled, the extractor brackets each kernel group
 * with CUDA events on the launching stream.  skb_profile_read synchronises, sums the elapsed milliseconds per
 * category into ms_by_category[0..7] = {front-end, stem, tcgen05 convolutions, SE, pooling+head, -, -, -}
 * and clears the record. */
void skb_profile_enable(int on);
int skb_profile_read(float* ms_by_category, int n_categories);

/* ---- extraction: replaces sidekit.nnet.xvector.Xtractor.__init__ / load_state_dict / forward -----------
 * Weights are handed over as named fp32 host tensors using the reference's state_dict keys
 * (SURVEY.md Appendix A.6), e.g. "sequence_network.layer1.0.conv1.weight"; BatchNorm folding,
 * 16-bit conversion and UMMA packing happen inside.  compute_dtype: 0 = fp16 operands (default,
 * meets 1e-3 relative L2), 1 = bf16 operands; accumulation is always fp32. */
int skb_xtractor_create(int archi, int n_tensors, const char* const* names, const float* const* data,
                        const int64_t* const* shapes, const int* ndims, int compute_dtype, float margin_s,
                        skb_xtractor_t** out);
void skb_xtractor_destroy(skb_xtractor_t* h);
int skb_xtractor_embedding_size(const skb_xtractor_t* h);
int skb_xtractor_speaker_number(const skb_xtractor_t* h);

/* Xtractor.forward(x, is_eval=True) (sidekit/nnet/xvector.py:876-907) on a packed batch:
 * wave_dev = the n_utt utterances back to back (fp32, 16 kHz), lengths[i] samples each (host array).
 * emb_dev (n_utt, E) receives F.normalize(x); logits_dev (n_utt, n_spk) the margin-head output
 * s*cos(x, W) (may be NULL).  Utterances of different lengths are handled exactly (no padding
 * artefacts): every reduction is per utterance. */
int skb_xtractor_forward(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt,
                         int norm_embedding, float* emb_dev, float* logits_dev, void* stream);
/* The embedding BEFORE the final F.normalize of the most recent forward call (what the reference
 * returns for loss='cce' with is_eval=True, xvector.py:896-898): out_dev (n_utt, E). */
int skb_xtractor_pre_embedding(skb_xtractor_t* h, int n_utt, float* out_dev, void* stream);
/* Bulk extraction: size every work buffer and every slot of the geometry-plan cache for batches of up to `max_utts`
 * utterances and `max_total_samples` samples, so that nothing is allocated (cudaMalloc / cudaFree synchronise the device)
 * once the run has started.  Optional: without it the buffers grow on demand. */
int skb_xtractor_reserve(skb_xtractor_t* h, int max_utts, int64_t max_total_samples, void* stream);

/* fp16 range guard.  With fp16 operands (compute_dtype 0) every stored activation is converted with saturation
 * (|x| > 65504 becomes +-65504 instead of +-inf) and the storing kernels count the threads that saw a saturated value.
 * Returns the CUMULATIVE count for this handle in *count after synchronising `stream`; a caller compares it with the
 * value it saw before its forward calls: any increase means the weights / inputs do not fit fp16 and the embeddings
 * of those calls are wrong -- rebuild the handle with compute_dtype 1 (bf16).  Always 0 for bf16 handles. */
int skb_xtractor_overflow_count(skb_xtractor_t* h, void* stream, int64_t* count);
/* Makes `stream` wait until the geometry tables of the last forward call on `h` have been uploaded.  For callers that
 * stream waveforms on a second stream (Xtractor.extract_stream): the next batch's host-to-device copy must not get
 * onto the copy engine ahead of the current batch's tables. */
int skb_xtractor_wait_tables(skb_xtractor_t* h, void* stream);
/* Same call with HOST buffers: H2D of the waveforms, forward, D2H of the results, synchronous. */
int skb_xtractor_forward_host(skb_xtractor_t* h, const float* wave_host, const int64_t* lengths, int n_utt,
                              int norm_embedding, float* emb_host, float* logits_host, void* stream);

/* MelSpecFrontEnd.forward / MfccFrontEnd.forward (sidekit/nnet/preprocessor.py:267-285, :113-124):
 * feats_dev is (n_utt, n_coef, t_max) fp32, zero beyond each utterance's frame count. */
int skb_xtractor_frontend(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt, int t_max,
                          float* feats_dev, void* stream);
int skb_xtractor_num_frames(const skb_xtractor_t* h, int64_t n_samples);

/* Test hook: run the forward pass up to `stage` ("stem", "layer1.0" ... "layer4.2", "pooled") and
 * write that activation as dense fp32: trunk stages (n_utt, C, h_max, W) zero padded along h;
 * "pooled" (n_utt, 2*C*W).  Returns the number of floats written per utterance in *per_utt. */
int skb_xtractor_debug_stage(skb_xtractor_t* h, const float* wave_dev, const int64_t* lengths, int n_utt,
                             const char* stage, int h_max, float* out_dev, int64_t* per_utt, void* stream);

/* ---- stand-alone module operators (SURVEY.md 8b): the engine's kernels on DENSE fp32 tensors ------------------------
 * Conv2d (3x3 pad 1 or 1x1 pad 0, stride 1 or 2, no dilation) with the following BatchNorm folded into w / bias by the
 * caller, the activation max(v, slope * v) (0 = ReLU, 1 = identity, 0.01 = LeakyReLU), and optionally the tail of a
 * BasicBlock fused into the epilogue: y = act(conv(x) * se_scale[b][c] + residual).  Replaces conv + bn + relu of
 * sidekit/nnet/res_net.py:309-320 (BasicBlock), :238-255 (ResBlock; its pre-activation BatchNorm + LeakyReLU is the
 * optional prologue x <- lrelu(x * pre_scale[c] + pre_shift[c], pre_slope)), :549 (stem).
 * x_dev (B, Cin, H, W), residual_dev / y_dev (B, Cout, Ho, Wo) fp32 NCHW contiguous, Ho = (H - 1) / stride + 1;
 * w_host (Cout, Cin, k, k) and bias_host (Cout) are HOST arrays; pre_scale / pre_shift (Cin) and se_scale (B, Cout) device.
 * Runs on the tcgen05 convolution kernel with 16-bit operands (compute_dtype as skb_xtractor_create). */
int skb_conv2d_bn_act(const float* x_dev, int B, int Cin, int H, int W, const float* w_host, const float* bias_host, int Cout,
                      int ksize, int stride, const float* pre_scale_dev, const float* pre_shift_dev, float pre_slope,
                      float act_slope, const float* se_scale_dev, const float* residual_dev, int compute_dtype, float* y_dev,
                      void* stream);
/* fp16 range guard of the stand-alone operators: cumulative saturation count of this thread's operator context. */
int skb_ops_overflow_count(void* stream, int64_t* count);
/* AdaptiveAvgPool2d(1): x_dev (B, C, hw) -> out_dev (B, C)  (SELayer, res_net.py:264, :279). */
int skb_channel_mean(const float* x_dev, int B, int C, int64_t hw, float* out_dev, void* stream);
/* SELayer.fc: scale = sigmoid(fc2 . relu(fc1 . mean)); fc1 (R, C), fc2 (C, R) row-major, no biases (res_net.py:265-270). */
int skb_se_gate(const float* mean_dev, const float* fc1_dev, const float* fc2_dev, int B, int C, int R, float* scale_dev,
                void* stream);
/* out = act(y * scale[b][c] + res): SELayer.forward (res NULL, slope 1) and the tail of BasicBlock.forward
 * (res_net.py:316-319); scale_dev / res_dev may be NULL. */
int skb_scale_residual_act(const float* y_dev, const float* scale_dev, const float* res_dev, int B, int C, int64_t hw,
                           float slope, float* out_dev, void* stream);
/* torch.nn.functional.normalize(x, dim=1): rows of x_dev (N, D) divided by max(||row||, eps)  (loss.py:304-305). */
int skb_l2_normalize(const float* x_dev, int N, int D, float eps, float* out_dev, void* stream);
/* AttentivePooling.forward (sidekit/nnet/pooling.py:151-171) on x_dev (B, D, T) fp32, D = channels * frequencies:
 * w1 (A, 3D or D) / b1 (A), BatchNorm1d(A) as scale / shift, w2 (D, A) / b2 (D), all device fp32;
 * out_dev (B, 2D) = [weighted mean ; weighted std]. */
int skb_attentive_pool(const float* x_dev, int B, int D, int T, const float* w1_dev, const float* b1_dev,
                       const float* bn_s_dev, const float* bn_t_dev, const float* w2_dev, const float* b2_dev, int A,
                       int global_context, float* out_dev, void* stream);

/* ---- pooling ops: replace MeanStdPooling.forward (sidekit/nnet/pooling.py:55-70) ---------------------- */
/* x_dev (n_utt, D, T) fp32 contiguous -> out_dev (n_utt, 2*D) = [mean ; unbiased std]. */
int skb_meanstd_pool(const float* x_dev, int n_utt, int D, int T, float* out_dev, void* stream);

/* ---- scoring: replaces the dense algebra of sidekit/iv_scoring.py:108-109, :451-462, :192-205 ---------
 * S[i][j] = alpha * (rowterm[i] + colterm[j] + cst) + alpha * sum_k E[i][k] * T[j][k]
 * E_dev (Ne, D), T_dev (Nt, D) fp32 row-major; rowterm/colterm may be NULL (treated as 0).
 * passes: 1 = single 16-bit pass, 3 = split (hi*hi + hi*lo + lo*hi) for fp32-class accuracy,
 * 0 = choose from the operand magnitudes: 1 when an estimate of the absolute error for operands whose fp16 rounding
 * errors are uncorrelated stays below 2.5e-4 (on S, alpha included), else 3.  Coherent rounding errors (e.g. rows of one repeated value)
 * can exceed 2.5e-4 with 1 pass; passes = 3 is the bound for them.
 * out_dtype: 0 = float32, 1 = float64, 2 = float16 (halves the HBM-bound write; 11-bit mantissa: meant for cosine-range
 * scores).  out_dev is (Ne, Nt) row-major with leading dimension ld_out. */
int skb_score_gemm(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                   const float* colterm_dev, double cst, double alpha, int passes, int out_dtype, void* out_dev,
                   int64_t ld_out, void* stream);

/* The same with the test-side operand PACKED ONCE (scaled, split into fp16 hi / lo planes, tiled): scoring a test set
 * against many enrol panels -- the row-panel sharding of a 20k x 20k trial matrix over GPUs, or repeated calls --
 * then costs only the enrol panel's preparation and the GEMM.  T_dev (rows, D) fp32 row-major is read once. */
typedef struct skb_packed skb_packed_t;
int skb_packed_create(const float* T_dev, int rows, int D, skb_packed_t** out, void* stream);
void skb_packed_destroy(skb_packed_t* p);
int skb_score_gemm_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev,
                          const float* colterm_dev, double cst, double alpha, int passes, int out_dtype, void* out_dev,
                          int64_t ld_out, void* stream);

/* Trial-list mode: only the trials a mask selects are scored INTO MEMORY, compacted in row-major order -- exactly what the
 * reference extracts with `scores.scoremat[ndx.trialmask]` (sidekit/nnet/xvector.py:243-245) -- so the Ne x Nt matrix never
 * reaches HBM and the GEMM is no longer write-bound.  skb_trial_index_create turns a (Ne, Nt) byte mask (non-zero = trial,
 * leading dimension ld_mask, device) into bit words and prefix counts and returns the number of trials;
 * skb_score_gemm_trials writes out_trials_dev[k] = score of the k-th trial (float32), same formula as skb_score_gemm. */
typedef struct skb_trial_index skb_trial_index_t;
int skb_trial_index_create(const uint8_t* mask_dev, int Ne, int Nt, int64_t ld_mask, skb_trial_index_t** out, int64_t* n_trials,
                           void* stream);
void skb_trial_index_destroy(skb_trial_index_t* t);
int skb_score_gemm_trials(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                          const float* colterm_dev, double cst, double alpha, int passes, const skb_trial_index_t* trials,
                          float* out_trials_dev, void* stream);
/* The same against a test side packed once with skb_packed_create (only the enrol side is packed per call). */
int skb_score_gemm_trials_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev, const float* colterm_dev,
                                 double cst, double alpha, int passes, const skb_trial_index_t* trials, float* out_trials_dev,
                                 void* stream);

/* Pair-list mode: replaces the dense trial matrix of sidekit/iv_scoring.py:108-109, :451-462 and the N x N as-norm matrix of
 * sidekit/score_normalization.py:135-138 for lists given as (enrolment row, test row) pairs, such as VoxCeleb1-E / -H.  For
 * p < n_pairs, i = rows_dev[p], j = cols_dev[p] (int32, device):
 *   s = alpha * (rowterm[i] + colterm[j] + cst) + alpha * sum_k E[i][k] * T[j][k]    (float32 FMAs over the float32 rows)
 * and out_dev[p] = s, or, when the four statistic vectors are given (all four or none),
 *   out_dev[p] = 0.5 * (s - mean_e[i]) / std_e[i] + 0.5 * (s - mean_t[j]) / std_t[j].
 * rowterm / colterm may be NULL (0).  The bits of out_dev[p] depend on D and the two rows only (fixed reduction order), not
 * on p or n_pairs.  An index outside [0, Ne) / [0, Nt) is not dereferenced: that trial gets NaN.  Any D >= 1 (16-byte loads
 * when D % 4 == 0 and both bases are 16-byte aligned).  n_pairs == 0 is a no-op. */
int skb_score_pairs(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const int32_t* rows_dev, const int32_t* cols_dev,
                    int64_t n_pairs, const float* rowterm_dev, const float* colterm_dev, float cst, float alpha,
                    const float* mean_e_dev, const float* std_e_dev, const float* mean_t_dev, const float* std_t_dev,
                    float* out_dev, void* stream);

/* Top-k mode.  Per row i of S (same formula and arguments as skb_score_gemm_trials): the k largest S[i][j], ordered by score
 * descending, ties by lower j.  values (Ne, k) float32, indices (Ne, k) int64, device.  1 <= k <= min(Nt, 1024).  Each value
 * equals the skb_score_gemm entry of the same arguments bit for bit.  k <= 32 with D <= 256 selects inside the GEMM epilogue
 * (the Ne x Nt matrix never reaches memory); larger k or D scores row panels into a bounded scratch matrix and selects per
 * row.  The order of NaN scores is undefined (finite embeddings do not produce them). */
int skb_score_gemm_topk(const float* E_dev, const float* T_dev, int Ne, int Nt, int D, const float* rowterm_dev,
                        const float* colterm_dev, double cst, double alpha, int passes, int k, float* values_dev,
                        int64_t* indices_dev, void* stream);
int skb_score_gemm_topk_packed(const float* E_dev, int Ne, const skb_packed_t* T, const float* rowterm_dev,
                               const float* colterm_dev, double cst, double alpha, int passes, int k, float* values_dev,
                               int64_t* indices_dev, void* stream);

/* dst[i] = (double)src[i]: the float64 view of a float32 score matrix, produced chunk by chunk on its way to the host
 * (sidekit's PLDA / two-covariance scorers return float64, iv_scoring.py:205, :462). */
int skb_widen_f32_f64(const float* src_dev, double* dst_dev, int64_t n, void* stream);

/* Operand preparation for the quadratic scorers (center_stat1 statserver.py:810-817, then the
 * model_part / seg_part / Psi fold of iv_scoring.py:451-462): xc = X - mu (mu may be NULL);
 * rowterm[i] = 0.5 * xc_i^T Phi xc_i (Phi symmetric, (D, D)); Xout = xc . Psi when PsiT_dev (= Psi
 * transposed, row-major) is given, else Xout = xc.  All device fp32; split-precision GEMMs inside. */
int skb_quadratic_prepare(const float* X_dev, const float* mu_dev, const float* PsiT_dev, const float* Phi_dev, int N, int D,
                          float* Xout_dev, float* rowterm_dev, void* stream);

/* as-norm statistics (sidekit/score_normalization.py:127-133): per row of X_dev (N, D), mean and
 * unbiased std of the top_k largest scores against the (already normalised) cohort_dev (C, D). */
int skb_asnorm_stats(const float* X_dev, const float* cohort_dev, int N, int C, int D, int top_k, float* mean_dev,
                     float* std_dev, void* stream);
/* out[i][j] = 0.5*(S[i][j]-mean[i])/std[i] + 0.5*(S[i][j]-mean[j])/std[j], S = X X^T  (:135-138). */
int skb_asnorm_apply(const float* X_dev, int N, int D, const float* mean_dev, const float* std_dev, float* out_dev,
                     void* stream);

/* Multi-GPU as-norm (SURVEY.md 8e): rows [row0, row0 + n_rows) of the normalised matrix; mean_dev / std_dev hold the
 * statistics of all N embeddings (each rank computes its rows' with skb_asnorm_stats, one all_gather shares them). */
int skb_asnorm_apply_panel(const float* X_dev, int N, int D, int row0, int n_rows, const float* mean_dev,
                           const float* std_dev, float* out_dev, int64_t ld_out, void* stream);

/* ---- evaluation tail (SURVEY.md 8f rank 2): host functions, plain host pointers ------------------------------
 * Pool-adjacent-violators, sidekit/bosaris/detplot.py:289-347 (`pavx`): y[n] -> ghat[n] (including the reference's
 * wrap-around write into the last element), bin widths / heights (arrays of n, the first *n_bins entries are used). */
int skb_pavx(const double* y, int64_t n, double* ghat, int64_t* width, double* height, int64_t* n_bins);
/* ROC convex hull, detplot.py:391-441 (`rocch`): pmiss / pfa need room for n_tar + n_non + 1 vertices. */
int skb_rocch(const double* tar, int64_t n_tar, const double* non, int64_t n_non, double* pmiss, double* pfa,
              int64_t* n_points);
/* Equal error rate by bisection, sidekit/nnet/xvector.py:101-209 (`eer(negatives, positives)`). */
int skb_eer(const double* negatives, int64_t n_neg, const double* positives, int64_t n_pos, double* eer_out);

/* z-/t-norm statistics and normalisation (sidekit/score_normalization.py:44-95) on a device-resident score matrix
 * S_dev (M, N), leading dimension ld, float32 (is_f64 = 0) or float64.  axis 1: per row (mean(1), std(1)); axis 0: per
 * column.  sym = 1 (znorm(sym=True), axis 1, square matrix): the diagonal is excluded, divisor N-1, and the second output
 * is the reference's "std_per_model": row sums of (S[i][j] - mean[j])^2 without the diagonal term, over N-1.  mean_dev / std_dev: device doubles of length M (axis 1) or N (axis 0). */
int skb_scoremat_stats(const void* S_dev, int M, int N, int64_t ld, int is_f64, int axis, int sym, double* mean_dev,
                       double* std_dev, void* stream);
/* out[i][j] = (S[i][j] - sub[j]) / div[j]  (numpy broadcasting of an (N,) vector, as both znorm and tnorm do). */
int skb_scoremat_normalise(const void* S_dev, int M, int N, int64_t ld, int is_f64, const double* sub_dev,
                           const double* div_dev, void* out_dev, int64_t ld_out, void* stream);

/* ---- PLDA training (SURVEY.md 8f rank 3): FactorAnalyser.plda, sidekit/factor_analyser.py:830-932 -------------------
 * All arrays are device float64, row-major.  skb_plda_stats: mean (D), total covariance sigma_obs (D, D) and the
 * scaled per-class sums S1 (n_cls, D) of the training vectors X (n_sess, D); the classes are given as CSR lists
 * (cls_ptr (n_cls + 1), cls_rows (n_sess): the rows of class c in input order).  Synchronises the stream. */
int skb_plda_stats(const double* X_dev, int n_sess, int D, const int* cls_ptr_dev, const int* cls_rows_dev, int n_cls,
                   double scaling, double* mean_dev, double* sigma_obs_dev, double* S1_dev, void* stream);
/* skb_plda_em: nb_iter EM iterations with no host round trip (Cholesky factorisations, batched over the distinct session
 * counts, and GEMMs on the device).  cls_n (n_cls) scaled session count of each class, cls_u (n_cls) index of that count
 * in uniq_n (U), cnt_u (U) classes per count, sum_n = sum of cls_n.  F_dev (D, R): in the eigenvoice initialisation, out
 * the trained matrix; Sigma_dev (D, D): in sigma_obs, out the residual covariance.  Synchronises the stream. */
int skb_plda_em(const double* S1_dev, const double* cls_n_dev, const int* cls_u_dev, int n_cls, const double* uniq_n_dev,
                const double* cnt_u_dev, int U, const double* mean_dev, const double* sigma_obs_dev, int D, int R, int nb_iter,
                double sum_n, double* F_dev, double* Sigma_dev, void* stream);

/* ---- embedding conditioning (statserver.py:789-1054, :1279-1333): float64 scatter matrices and row transforms -------
 * X_dev (N, D) row-major with row stride ld (elements), float32 (x_is_f64 = 0, widened exactly on load) or float64;
 * 1 <= D <= 1024, N up to 2^31 - 1 rows (row offsets are 64-bit).  No call synchronises the stream.
 *
 * skb_gram_f64: G_dev (D, D) = scale * sum_i w_i (x_i - s_k(i)) (x_i - s_k(i))', float64 on mma.sync .f64 (DMMA).
 * shift_dev (K, D) float64 shift table or NULL (no shift); shift_idx_dev (N) int32 row -> table row or NULL (row 0);
 * w_dev (N) float64 row weights or NULL (1).  The shift is subtracted on load (no raw-moment shortcut); G is symmetric
 * bit for bit and bitwise reproducible: rows are split into chunks that depend on (N, D) only, and the chunk partials
 * (in a stream-ordered workspace of at most ~70 MB) are summed in a fixed order. */
int skb_gram_f64(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const double* shift_dev,
                 const int* shift_idx_dev, const double* w_dev, double scale, double* G_dev, void* stream);
/* skb_class_stats: mean_dev (D) column mean (row-chunk partials summed in a fixed order); sums_dev (n_cls, D) per-class
 * sums and counts_dev (n_cls) per-class row counts.  The classes are CSR lists: cls_ptr_dev (n_cls + 1), cls_rows_dev
 * (N, the rows of class c in input order, which is the order of summation).  Any of the three outputs may be NULL (not
 * all); the CSR lists are needed only for sums / counts. */
int skb_class_stats(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const int* cls_ptr_dev,
                    const int* cls_rows_dev, int n_cls, double* mean_dev, double* sums_dev, double* counts_dev, void* stream);
/* skb_affine_rows: y_i = ((x_i - mu) .* d) W, then, with unit_norm, y_i / max(||y_i||, 1e-8) (norm_stat1).  mu_dev (D),
 * d_dev (D) and W_dev (D, D_out) float64 may each be NULL (no centring / no scaling / identity, then D_out = D).  Y_dev
 * (N, D_out) float32 (y_is_f64 = 0) or float64, row stride ld_out, must not overlap X.  W runs on DMMA; for D_out <= 256
 * the length normalisation is fused into the same pass, above that a second row pass scales Y in place. */
int skb_affine_rows(const void* X_dev, int x_is_f64, int64_t N, int D, int64_t ld, const double* mu_dev, const double* d_dev,
                    const double* W_dev, int D_out, int unit_norm, void* Y_dev, int y_is_f64, int64_t ld_out, void* stream);

/* ---- feed path: sample-rate conversion (SURVEY.md 8f rank 1) ---------------------------------------------------
 * torchaudio.transforms.Resample(orig_freq, new_freq)(speech) as sidekit/nnet/xsets.py:435, :452 and
 * sidekit/bin/extract_xvectors.py:144 call it (Hann-windowed sinc, lowpass_filter_width 6, rolloff 0.99), on a packed
 * batch: in_dev = the waveforms back to back, out_dev receives them back to back with ceil(new_r * L / orig_r) samples
 * each.  wave_meta_dev: n_wav rows of four int64 {input offset, input length L, output offset, output length} (device);
 * max_out = the largest output length.  orig_r / new_r are the rates divided by their gcd, width the filter half-width in
 * input samples.  bank_dev / start_dev (device) are the compact polyphase filter bank: bank[k][ph] (ntap x new_r,
 * tap-major) multiplies input sample q * orig_r - width + start[ph] + k of output q * new_r + ph. */
int skb_resample(const float* in_dev, const int64_t* wave_meta_dev, int n_wav, int64_t max_out, int orig_r, int new_r,
                 int width, const float* bank_dev, const int32_t* start_dev, int ntap, float* out_dev, void* stream);

/* ---- feed path: FLAC decoding (RFC 9639, up to 24 bits per sample) -----------------------------------------------
 * Replaces torchaudio.load(path) of sidekit/nnet/xsets.py:419-464 (IdMapSet with file_extension="flac") and
 * soundfile.read of sidekit/bin/extract_xvectors.py:37-72 for .flac files: channel 0 of every file of a batch, as float32
 * int / 2^(bps - 1), back to back in out_dev.  bytes_dev: the files' frame bytes back to back (n_bytes); files_dev: n_files
 * rows of nine int64 {first frame byte, end of the file's bytes, output offset, total samples, first frame slot, frame
 * slots, sample rate, channels, bits per sample} (device), ordered by byte range and by slot; the last five come from
 * STREAMINFO, which the host parses (sidekit_b200/flac.py).  n_slots = sum of the slot counts (an upper bound on each
 * file's frame count).  work_dev: at least skb_flac_workspace_bytes(n_bytes, n_files, n_slots) bytes, 16-byte aligned.
 * status_dev (n_files, int32) receives SKB_FLAC_OK or the reason the file is corrupt; a corrupt file's output range is
 * left unwritten.  Three launches whatever n_files; no synchronisation; never reads outside bytes_dev. */
#define SKB_FLAC_OK 0
#define SKB_FLAC_BAD_FRAME 1      /* no valid frame (header CRC-8, subframes, CRC-16) where the chain needs one */
#define SKB_FLAC_BAD_NUMBER 2     /* frame / sample number or blocking strategy out of sequence */
#define SKB_FLAC_BAD_LENGTH 3     /* block sizes overrun STREAMINFO's total samples, or more frames than slots */
int64_t skb_flac_workspace_bytes(int64_t n_bytes, int n_files, int64_t n_slots);
int skb_flac_decode(const uint8_t* bytes_dev, int64_t n_bytes, const int64_t* files_dev, int n_files, int64_t n_slots,
                    void* work_dev, int64_t work_bytes, float* out_dev, int32_t* status_dev, void* stream);

/* ---- feed path: uncompressed audio (WAV and NIST SPHERE, every PCM encoding) ------------------------------------------
 * Replaces torchaudio.load(path) of sidekit/nnet/xsets.py:419-464 and soundfile.read of sidekit/bin/extract_xvectors.py:37-72
 * for .wav / .sph files: channel 0 of every file of a batch as float32, at the file's output offset in out_dev, scaled as
 * those readers do -- signed integers x / 2^(8 bytes - 1) (32-bit: rounded to float32 first), unsigned 8-bit
 * (x - 128) / 128, float32 copied, float64 rounded to float32, G.711 mu-law / A-law expanded to 16 bits (Sun g711.c) / 2^15.
 * bytes_dev: the files' sample bytes (interleaved frames); files_dev: n_files rows of eight int64 {byte offset of the
 * file's first frame in bytes_dev, frames, channels, SKB_PCM_* encoding, bytes per sample (1-4 for integers, 1 for
 * G.711, 4 or 8 for float), big-endian flag, output offset, first tile}, ordered by first tile; a file owns
 * ceil(frames / 256) tiles, numbered file after file, and n_tiles is their total.  The host parses the containers
 * (sidekit_b200/pcm.py).  Reads stay inside [offset, offset + frames * channels * bytes) of each file.  One launch
 * whatever n_files (also when n_tiles is 0, when bytes_dev and out_dev may be NULL); no synchronisation. */
#define SKB_PCM_INT 0             /* signed integer, any byte count 1-4 */
#define SKB_PCM_U8 1              /* unsigned 8-bit (WAV) */
#define SKB_PCM_FLOAT 2           /* IEEE float, 4 or 8 bytes */
#define SKB_PCM_ULAW 3            /* G.711 mu-law, 1 byte */
#define SKB_PCM_ALAW 4            /* G.711 A-law, 1 byte */
int skb_pcm_decode(const uint8_t* bytes_dev, const int64_t* files_dev, int n_files, int64_t n_tiles, float* out_dev,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SIDEKIT_B200_H */
