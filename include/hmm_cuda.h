/*
 * hmm_cuda.h -- C ABI of the B200-native continuous-HMM hot path (libhmmcu.so).
 *
 * The reference (edielsonpf/speech-recognition-hmm-continuous) has no FFI: its hot path is a set
 * of K&R C functions called from two main()s.  This header is the boundary a maintainer binds
 * INSTEAD of those functions; every entry point names the reference code it replaces.
 *   T-FS = train/source/hmm-fs/hmm_continuous_fs.c        (diagonal-covariance trainer)
 *   R-FS = test/source/recognition-fs/recognition_continuous_fs.c   (forward-score recogniser)
 *
 * Conventions
 *   - plain C: pointers and sizes only, caller-owned host buffers, `int` status (0 = ok, else a
 *     HMMCU_E* code; hmmcu_last_error() gives the text).  No CPU fallback exists: every compute
 *     entry point fails with HMMCU_ENODEV when no sm_100 device is present.
 *   - one host thread per context; a context owns one device and one stream.
 *   - model semantics are the reference's (T-FS:53-64): `inv_var` is the INVERSE variance held in
 *     `cov_matrix`, `det` the product of variances; pi = [1,0,..,0]; the last state is final.
 *   - all host arrays are row-major, double precision unless stated.
 */
#ifndef HMM_CUDA_H
#define HMM_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMMCU_OK 0
#define HMMCU_EINVAL 1   /* bad argument / call order */
#define HMMCU_ENODEV 2   /* no usable CUDA device */
#define HMMCU_ECUDA 3    /* CUDA runtime error */
#define HMMCU_ENOMEM 4
#define HMMCU_EIO 5      /* host-side file error (hmmh_* only) */

#define HMMCU_MAX_STATES 8 /* states per model the kernels are built for (reference: MAX_STATES_NUMBER 20 in the trainer, T-FS:41, 15 in the
                            * recogniser, R-FS:37); larger models are refused by both programs up front, see DESIGN.md */
#define HMMH_MAX_FILE_STATES 32 /* .hmm files with up to this many states are read and written by the host-side file code */

typedef struct hmmcu_ctx hmmcu_ctx;

/* ---------------------------------------------------------------- context ---------------- */
int hmmcu_create(int device, hmmcu_ctx **out);
void hmmcu_destroy(hmmcu_ctx *ctx);
const char *hmmcu_last_error(const hmmcu_ctx *ctx); /* ctx may be NULL: last create() error */
int hmmcu_device_count(void);
/* The context's CUDA stream as a cudaStream_t cast to void* (for callers that enqueue a
 * collective on the statistics buffer, see hmmcu_stats_device). */
void *hmmcu_stream(hmmcu_ctx *ctx);
int hmmcu_synchronize(hmmcu_ctx *ctx);
/* pinned host memory for the feature upload path */
int hmmcu_host_alloc(void **p, uint64_t bytes);
void hmmcu_host_free(void *p);

/* Tuning / A-B switches.  "tc_emis": 1 (default) = emissions on the tcgen05 tensor-core path whenever
 * its accuracy guard holds (the expanded quadratic loses ~1e-7 of sum|terms|; data whose centred
 * range is huge against the model variances, like the reference's raw-Hz fixtures, go to the
 * CUDA-core kernel, which evaluates (x-mu)^2 directly); 0 = always the CUDA-core kernel;
 * 2 = always tensor cores.  Both are device code.
 * "graphs": 1 (default) = hmmcu_estep / hmmcu_mstep replay their launch sequences as CUDA graphs from the third
 * identical call on; "ws_emis" / "ws_acc": 0 = the older single-buffered tensor-core kernels; "res_fb": 0 = the windowed
 * forward-backward kernel (k_fb) instead of the shared-memory-resident one (k_fb_res, the default whenever the utterances fit
 * and the transition matrices are banded);
 * "upload_chunks": chunks hmmcu_set_features splits the host-to-device copy into (packing overlaps the copy);
 * "mstep_fork": 1 (default) = the accuracy-guard scan and one of the two model packers of hmmcu_mstep run on side streams;
 * "dec_emis": 1 (default) = decode emissions of models with M <= 16 through k_emis_dec (frame tile resident in tensor memory, W
 * images multicast over a cluster of two CTAs, interleaved log-emission layout), 0 = k_emis_ws;
 * "dec_f16": 1 (default) = k_emis_dec with half-precision operands (per-dimension power-of-two scaling, as accurate as
 * the 3xTF32 split; used while the accuracy guard holds and the padded feature row is a multiple of 8), 0 = 3xTF32;
 * "dec_budget_kb": log-emission budget of one decode batch in KiB (0 = 6 GiB or a third of the free memory);
 * "h_acc": 1 (default) = the mixture accumulators through k_accum_h (half-precision hi / lo operands, frame tiles packed once per
 * feature set and fetched by bulk copies; taken while the padded feature row is a multiple of 8 and at most 40), 0 = k_accum_ws
 * (3xTF32, loader warps).  Any other key fails with HMMCU_EINVAL. */
int hmmcu_set_option(hmmcu_ctx *ctx, const char *key, int value);

/* ---------------------------------------------------------------- inputs ----------------- */
/* Feature vectors of U utterances, ragged: utterance u owns frames [frame_off[u], frame_off[u+1])
 * of x[F][D].  Replaces the per-frame fread loop (reading_coef, T-FS:527-548 / R-FS:518-539) that
 * the reference runs twice per utterance per EM iteration and V times per test utterance.
 * The data are copied to the device, centred and converted once. */
int hmmcu_set_features(hmmcu_ctx *ctx, const double *x, const int64_t *frame_off, int U, int D);
/* Same, but x is already a DEVICE pointer (features resident in HBM). */
int hmmcu_set_features_device(hmmcu_ctx *ctx, const double *x_dev, const int64_t *frame_off, int U, int D);

/* Streaming form of hmmcu_set_features for the ingest pipeline (hmmh_ingest below): announce the geometry, hand
 * over frame ranges [first_frame, first_frame + n_frames) of x[.][D] as they become available (each call enqueues
 * an asynchronous copy; *ticket tells hmmcu_features_wait when the source buffer may be reused; at most 16 tickets
 * are in flight), then _end forms the centre and the packed rows on the device.  The context ends up in the same
 * state as after hmmcu_set_features on the concatenated buffer.  Replaces the same fread loop as above. */
int hmmcu_features_begin(hmmcu_ctx *ctx, const int64_t *frame_off, int U, int D);
int hmmcu_features_append(hmmcu_ctx *ctx, const double *x, int64_t first_frame, int64_t n_frames, int *ticket);
int hmmcu_features_wait(hmmcu_ctx *ctx, int ticket);
int hmmcu_features_end(hmmcu_ctx *ctx);
/* Pinned staging buffer `slot` (0..3) of at least `bytes`, owned by the context and kept until hmmcu_destroy
 * (NULL on failure): what hmmh_ingest reads the files into. */
void *hmmcu_staging(hmmcu_ctx *ctx, int slot, uint64_t bytes);

/* V models of identical topology, struct-of-arrays in the semantics of `struct state` /
 * `struct mixture` (T-FS:53-64, R-FS:52-63) and transition_probab:
 *   A[V][N][N]  c[V][N][M]  mu[V][N][M][D]  inv_var[V][N][M][D]  det[V][N][M]            */
int hmmcu_set_models(hmmcu_ctx *ctx, int V, int N, int M, int D, const double *A, const double *c,
                     const double *mu, const double *inv_var, const double *det);

/* Multi-stream models (param_number > 1): the emission probability of a state is the PRODUCT over the feature streams
 * of the stream's mixture density (calc_alpha / calc_beta / calc_transition_probab, T-FS:1406-1409, 1500-1503,
 * 1606-1609; recogniser R-FS:341-364), every stream with its own coefficient count, mixture count and feature files.
 * Here every stream is a context of its own (hmmcu_set_features / hmmcu_set_models with the stream's D and M, the
 * same A, the same utterance lengths, the same device).  After hmmcu_link_streams(primary, others, n):
 *   hmmcu_estep(primary)  computes every stream's log-emissions, adds them, runs ONE forward-backward pass, and
 *     accumulates every stream's mixture statistics with the joint state posteriors; the transition statistics,
 *     den_mix, sum_logP and n_utt are copied into the linked contexts' statistics, so hmmcu_mstep (and
 *     hmmcu_stats_device / _download) on EACH context gives that stream's update (T-FS:328-346);
 *   hmmcu_forward_scores / hmmcu_viterbi_scores / hmmcu_viterbi (primary) score the product model.
 * Linked contexts run on the primary's stream; n = 0 unlinks; hmmcu_destroy unlinks. */
int hmmcu_link_streams(hmmcu_ctx *primary, hmmcu_ctx *const *others, int n);

/* creating_initial_model (T-FS:732-1317) on the device for V words at once, from the context's features:
 * utterance u belongs to word utt2model[u] (-1 = not used).  Uniform left-to-right A, uniform segmentation,
 * LBG splitting (x1.005 / x0.995) with three k-means passes per level and the empty-cell rule, per-cluster
 * variances (floored at 1e-5) and weights.  The models are left in the context as hmmcu_set_models would leave
 * them (hmmcu_get_models reads them back) and are bit-identical to hmmh_init_model()'s.  D <= 64, M <= 255. */
int hmmcu_init_models(hmmcu_ctx *ctx, const int32_t *utt2model, int V, int N, int M);

/* ---------------------------------------------------------------- emissions -------------- */
/* Parity / debug export of calc_symbol_probab + calc_gaus (T-FS:1749-1841, R-FS:860-947) for
 * utterance u against model v, as the device path computes them: logb[T][N] = log b_i(t), and
 * (post != NULL) post[T][N][M] = c_m N_m / b_i, the normalised per-mixture posterior. */
int hmmcu_emissions(hmmcu_ctx *ctx, int u, int v, double *logb, double *post);

/* ---------------------------------------------------------------- recognition ------------ */
/* logp[U][V] = log P(O_u, q_T = N-1 | model v): calc_symbol_probab + calc_alpha +
 * calc_probability for every (utterance, model) cell -- the recogniser's inner loops
 * R-FS:341-369.  Where the reference's linear-domain arithmetic underflows it yields NaN or
 * -inf (SURVEY 0.2); with emulate_underflow != 0 those cells are reported as NaN / -inf too. */
int hmmcu_forward_scores(hmmcu_ctx *ctx, double *logp, int emulate_underflow);

/* sorting_probab + the label rule (R-FS:968-995, 380-388): label[u] = index[0], second[u] =
 * index[1] of the reference's stable descending bubble sort, including its NaN behaviour.
 * weight multiplies every score first (coef_model, R-FS:366).  second may be NULL. */
int hmmcu_rank(hmmcu_ctx *ctx, const double *logp, int U, int V, double weight, int32_t *label,
               int32_t *second);

/* ---------------------------------------------------------------- Baum-Welch E-step ------ */
/* Doubles per model in the statistics vector (this is also the all-reduce payload):
 *   num_trans[N][N] den_trans[N] den_mix[N] S0[N][M] S1[N][M][D] S2c[N][M][D] sum_logp n_utt */
int64_t hmmcu_stats_size(int N, int M, int D);

/* One E-step over all utterances: utterance u is trained against model utt2model[u]
 * (-1 = leave this utterance out, used for words that have already converged).
 * Replaces the body of the EM do-loop, T-FS:272-321: calc_symbol_probab, calc_alpha, calc_beta,
 * calc_transition_probab, calc_den_mix_coef, calc_mix_param, calc_probability.
 * stats[V][hmmcu_stats_size] receives the sums (may be NULL: they stay on the device, see
 * below); logp_utt[U] the per-utterance log-probabilities (may be NULL). */
int hmmcu_estep(hmmcu_ctx *ctx, const int32_t *utt2model, double *stats, double *logp_utt);

/* The E-step of Viterbi (segmental k-means) training, as HTK's HInit re-segments: the same contract and the same
 * statistics vector as hmmcu_estep, with the forward-backward pass replaced by the best state sequence of every utterance
 * (single-precision emissions, delta in double; pi = [1,0,..], termination in the final state, lowest predecessor index
 * on a tie, as hmmcu_viterbi).  Each frame belongs to its aligned state with weight 1, so
 *   num_trans[i][j] = number of t < T-1 with (s_t, s_t+1) = (i, j)   (every pair of a full A, not only the band)
 *   den_trans[i]    = number of t < T-1 with s_t = i,   den_mix[i] = number of t < T with s_t = i
 *   S0 / S1 / S2c   the in-state mixture posteriors of the aligned state, accumulated as in hmmcu_estep
 *   sum_logp, logp_utt   the Viterbi scores; n_utt as hmmcu_estep.
 * An utterance with no path to the final state (T < N with a left-to-right A) scores -inf and adds no occupancy or
 * counts, as it does in hmmcu_estep.  path[F] (may be NULL) receives the alignment, frame-aligned with the features
 * (-1 on the frames of masked utterances): forced alignment as a by-product.  The statistics stay on the device
 * (hmmcu_stats_device), so the all-reduce and hmmcu_mstep apply unchanged.  Linked (multi-stream) contexts are refused
 * with HMMCU_EINVAL. */
int hmmcu_estep_viterbi(hmmcu_ctx *ctx, const int32_t *utt2model, double *stats, double *logp_utt, int32_t *path);

/* The E-step of maximum mutual information (MMI) training.  label[U] is the word of every utterance (-1 leaves it out),
 * kappa > 0 the acoustic scale, 1 <= max_hyp <= HMMCU_MMI_MAX_HYP.  Every (utterance, word) cell is scored as
 * hmmcu_forward_scores(ctx, ., 0) scores it (on the device, not copied back), and
 *   P(w | u) = exp(kappa S[u][w] - logsumexp_w' kappa S[u][w'])    (double)
 * The hypotheses of u are its label, always, with the label's posterior however small, then at most max_hyp - 1 other
 * words in descending posterior order (lower word index first on a tie) with P >= HMMCU_MMI_MIN_POST.  The statistics
 * (hmmcu_stats_device, and stats if not NULL) are then [2][V][hmmcu_stats_size]:
 *   block 0, numerator     hmmcu_estep(ctx, label, ..)'s statistics, bit for bit (sum_logp and n_utt included)
 *   block 1, denominator   sum over u and its hypotheses h of P(h | u) times the E-step statistics of u against model h
 *                          (raw posteriors: the pruned mass is not renormalised); its tail holds the objective:
 *                          sum_logp[v] = sum over the included utterances of word v of -log P(label | u) (a fixed order,
 *                          bit-reproducible), n_utt[v] = their number.  The MMI objective is F = -sum_v sum_logp[v].
 * An utterance whose label score is not finite (T < N with a left-to-right A) is left out of block 1.  One all-reduce of
 * the whole buffer sums both blocks and the objective over the ranks.  hmmcu_mstep and hmmcu_peer_allreduce refuse
 * this buffer (its size is not theirs); hmmcu_mstep_ebw takes it.  Linked (multi-stream) contexts are refused with
 * HMMCU_EINVAL.  hmmcu_last_kernel_ms: "mmi_score", "mmi_post", "mmi_num", "mmi_den" time the stages, "mmi_rounds" is
 * the number of denominator rounds (round 0: the labels; round r: every utterance's r-th other hypothesis). */
#define HMMCU_MMI_MIN_POST 1.0e-5 /* posterior floor of a competing hypothesis */
#define HMMCU_MMI_MAX_HYP 16      /* hypotheses per utterance, the label included */
int hmmcu_estep_mmi(hmmcu_ctx *ctx, const int32_t *label, double kappa, int max_hyp, double *stats);

/* The extended Baum-Welch update of the means and variances from hmmcu_estep_mmi's statistics, per Gaussian and
 * dimension (hmmh_mstep_ebw is the same update on the host, operation for operation):
 *   Q = S2c + 2 mu S1 - mu^2 S0 (= sum gamma x^2); with S0_num > 0 the numerator's (S0, S1, Q) are scaled by
 *   1 + tau / S0_num (I-smoothing); dg, ds, dq = numerator - denominator of S0, S1, Q;
 *   D_min = the largest real root over the dimensions of var D^2 + (dq + dg (var + mu^2) - 2 mu ds) D + (dq dg - ds^2)
 *   (0 when none is positive); D = max(2 D_min, E S0_den);
 *   mu' = (ds + D mu) / (dg + D),  var' = (dq + D (var + mu^2)) / (dg + D) - mu'^2 floored at 1e-5 (T-FS:39),
 *   inv_var and det as hmmh_mstep forms them.
 * A Gaussian with dg + D <= 0 (no occupancy in either block) is left as it is.  Mixture weights and transitions are not
 * updated, and there is no stopping rule.  With den = 0 and tau = 0 this is the textbook ML update, whose variance is
 * about the NEW mean (hmmh_mstep keeps the reference's variance about the old mean).  E > 1, tau >= 0.  The accuracy
 * guard and the model images are refreshed as after hmmcu_mstep; hmmcu_em_reset's state is not touched.  Refused with
 * HMMCU_EINVAL unless the statistics are an MMI buffer of the current model set. */
int hmmcu_mstep_ebw(hmmcu_ctx *ctx, double E, double tau);

/* Device-side statistics for multi-GPU training: after hmmcu_estep(ctx, u2m, NULL, NULL) the
 * caller all-reduces the buffer in place on hmmcu_stream() (one ncclAllReduce(sum, double) per EM
 * iteration) and then downloads it. */
double *hmmcu_stats_device(hmmcu_ctx *ctx, int64_t *n_doubles);
int hmmcu_stats_download(hmmcu_ctx *ctx, double *stats);

/* The sum of the statistics over the ranks of one NVLink / NVSwitch domain WITHOUT a library collective: every rank
 * stores its statistics straight into a receive slot of every peer (peer memory mapped through CUDA IPC), waits for the
 * peers' copies in its own area and adds them in rank order -- one short kernel on the context's stream, the same bytes
 * on every rank (the M-step that follows is bit-identical everywhere).  Set-up, once per model-set geometry:
 *   hmmcu_peer_export   (after hmmcu_set_models) allocates this rank's receive area and returns its 64-byte IPC handle
 *   [the caller exchanges the handles of all ranks, e.g. with the all-gather of its process group]
 *   hmmcu_peer_import   maps the areas of all ranks (handles[world][64]; the entry of `rank` itself is ignored)
 *   hmmcu_peer_import_pointers   the same for areas that are already addressable in this process (several contexts in
 *                       one process, tests): areas[world] device pointers from hmmcu_peer_area
 * Per EM iteration, between hmmcu_estep and hmmcu_mstep (replaces the all-reduce of hmmh_allreduce_fn):
 *   hmmcu_peer_allreduce  statistics = sum over the ranks in rank order, in ONE launch: every double travels as two 8-byte
 *                       words tagged with the iteration number (an aligned 8-byte store lands atomically), so the kernel
 *                       needs neither a system fence nor flags: a thread pushes its elements to every peer and adds the
 *                       peers' copies in rank order as they land
 * Two slot sets alternate, so a rank that runs ahead never overwrites what a slower rank still reads. */
#define HMMCU_IPC_HANDLE_BYTES 64
int hmmcu_peer_export(hmmcu_ctx *ctx, int world, void *handle_out);
int hmmcu_peer_import(hmmcu_ctx *ctx, int rank, int world, const void *handles);
void *hmmcu_peer_area(hmmcu_ctx *ctx);
int hmmcu_peer_import_pointers(hmmcu_ctx *ctx, int rank, int world, void *const *areas);
int hmmcu_peer_allreduce(hmmcu_ctx *ctx);
/* 1 when a hmmcu_peer_allreduce gave up waiting for a peer (20 s); synchronises the context's stream */
int hmmcu_peer_error(hmmcu_ctx *ctx);

/* Device-resident EM iteration.  The M-step of the trainer's main() (T-FS:326-352:
 * updating_transition_probab, updating_mix_param, changing_zero_coef, calc_det, inv_matrix) applied on
 * the device to the model set held by the context, from the statistics of the last hmmcu_estep
 * (all-reduced in place by the caller when there are several ranks), together with the per-word
 * stopping rule (T-FS:326-328, 358): model v is re-estimated iff it is still active and
 * |old_v - sum_logp_v| / |old_v| > threshold (old starts at 1.0); otherwise it becomes inactive for
 * good.  Nothing but 3V+1 doubles crosses PCIe per iteration.
 *   hmmcu_em_reset : old_v = 1.0, every model active (call after hmmcu_set_models).
 *   hmmcu_mstep    : sum_logp[V], n_utt[V], updated[V] out (each may be NULL).
 *   hmmcu_get_models: downloads the current parameters (same layout as hmmcu_set_models; NULL = skip). */
int hmmcu_em_reset(hmmcu_ctx *ctx);
int hmmcu_mstep(hmmcu_ctx *ctx, double threshold, double *sum_logp, double *n_utt, int32_t *updated);
int hmmcu_get_models(hmmcu_ctx *ctx, double *A, double *c, double *mu, double *inv_var, double *det);

/* ---------------------------------------------------------------- Viterbi ---------------- */
/* The reference has NO Viterbi decoder (SURVEY 0.1); these follow its conventions (pi=[1,0..],
 * final-state termination, lowest predecessor index on a tie).
 * hmmcu_viterbi: utterance u against model utt2model[u], double-precision emissions;
 *   score[U] and the state sequence path[F] (frame-aligned with the features).
 * hmmcu_viterbi_scores: score[U][V] for every cell (single-precision emissions). */
int hmmcu_viterbi(hmmcu_ctx *ctx, const int32_t *utt2model, double *score, int32_t *path);
int hmmcu_viterbi_scores(hmmcu_ctx *ctx, double *score);

/* ---------------------------------------------------------------- instrumentation -------- */
/* Number of kernels this library has launched on ctx since creation (bench.py's gpu_launches). */
int64_t hmmcu_launch_count(const hmmcu_ctx *ctx);
/* Device time in ms of the most recent call's kernels, by name (CUDA events on the context's
 * stream).  names: "emis", "fwdbwd", "align" (the alignment of hmmcu_estep_viterbi), "accum", "mstep", "score", "viterbi", "logb64", "pack", "init".  -1 if unknown.
 * Pseudo-names report state instead of time:
 *   "kappa"           accuracy-guard value of the current model pack
 *   "tc_active"       1 if the last emission launch ran on tensor cores
 *   "dec_f16_active"  1 if the last decode emission launch used half-precision operands
 *   "acc_h_active"    1 if the last mixture-accumulate launch was the half-precision kernel
 *   "dec_grid"        CTAs of the decode emission kernel's launch configuration (0 = not chosen yet, -1 = unusable)
 *   "res_batches"     batches of the resident forward-backward kernel for the current training map
 *                     (0 when the windowed kernel takes the E-step)
 *   "res_batch_max"   the most utterances in one of those batches (0 likewise)
 *   "res_teams"       teams that claim those batches: 4 per CTA of its launch, min(res_batches, SMs) CTAs (0 likewise) */
double hmmcu_last_kernel_ms(const hmmcu_ctx *ctx, const char *name);
void hmmcu_enable_timing(hmmcu_ctx *ctx, int on);

/* ================================================================================================
 * Host side (plain C, no device work): file formats, M-step, EM control, drop-in programs.
 * ============================================================================================== */

typedef struct hmmh_model {
  char word[64];   /* reference: MAX_WORD_SIZE 50 */
  int N, M, D;     /* states, mixtures per state, coefficients of ONE feature stream (a P-stream model is P of these sharing A and word) */
  double *A;       /* [N][N] */
  double *c;       /* [N][M] */
  double *mu;      /* [N][M][D] */
  double *inv_var; /* [N][M][D] */
  double *det;     /* [N][M] */
} hmmh_model;

int hmmh_model_alloc(hmmh_model *m, int N, int M, int D);
void hmmh_model_free(hmmh_model *m);

/* Feature file: int32 D, then T x D doubles, T implied by EOF (T-FS:527-581).  *x is malloc'd. */
int hmmh_read_features(const char *path, double **x, int *T, int *D);
int hmmh_write_features(const char *path, const double *x, int T, int D);

/* Many-files reader (SURVEY 8f-2; replaces the list walk + per-frame fread of T-FS:272-321, 527-548 and
 * R-FS:341-369, 518-539).  hmmh_read_list: the whitespace-separated names of a list file.  hmmh_scan_features:
 * frame offsets of U files from their sizes (frame_off[U+1]) and D from the first header.  hmmh_ingest: scan, then
 * a pool of `nthreads` readers (0 = $HMMCU_INGEST_THREADS or min(16, cores)) fills pinned staging buffers that are
 * streamed to the device through hmmcu_features_begin/append/end while the next ones are read; no host copy of the
 * corpus is kept.  *bad_file = index of the file that failed (HMMCU_EIO: missing, short, wrong D, or empty).
 * hmmh_ingest_to is the same pipeline into any sink (the CPU tests use a memory sink). */
typedef struct hmmh_sink {
  void *user;
  int (*begin)(void *user, const int64_t *frame_off, int U, int D);
  int (*append)(void *user, const double *x, int64_t first_frame, int64_t n_frames, int *ticket);
  int (*wait)(void *user, int ticket);
  int (*end)(void *user);
  void *(*stage_alloc)(void *user, int slot, size_t bytes); /* staging buffer `slot` (0..2), owned by the sink; NULL = malloc/free */
} hmmh_sink;
typedef struct hmmh_ingest_stats {
  double scan_s, stage_s, read_s, total_s; /* fstat pass; getting the staging buffers; read + hand-off; everything incl. the sink's end() */
  int64_t bytes;                  /* feature payload */
  int batches, threads;
} hmmh_ingest_stats;
int hmmh_read_list(const char *list_path, char ***paths, int *n);
void hmmh_free_list(char **paths, int n);
int hmmh_scan_features(const char *const *paths, int U, int nthreads, int *D, int64_t *frame_off, int *bad_file);
int hmmh_ingest_to(const hmmh_sink *sink, const char *const *paths, int U, int nthreads, int64_t stage_frames,
                   int64_t *frame_off, int *D, int *bad_file, hmmh_ingest_stats *stats);
int hmmh_ingest(hmmcu_ctx *ctx, const char *const *paths, int U, int nthreads, int64_t *frame_off, int *D,
                int *bad_file, hmmh_ingest_stats *stats);

/* .hmm model file, layout of writing_model / reading_model (T-FS:2043-2146, 604-711).
 * len_bytes: 8 = LP64 size_t header (what the reference writes here), 4 = the shipped 32-bit files,
 * 0 = auto-detect on read. */
int hmmh_read_model(const char *path, hmmh_model *m, int len_bytes);
int hmmh_write_model(const char *path, const hmmh_model *m);
/* The same file with P >= 1 feature streams (param_number, T-FS:2075-2100): stream p comes back as streams[p]
 * (its own M and D; the shared A and word in each).  HMMCU_EINVAL if the file holds more than max_streams. */
#define HMMH_MAX_STREAMS 6 /* MAX_PARAMETERS_NUMBER, T-FS:36 */
int hmmh_read_model_streams(const char *path, hmmh_model *streams, int max_streams, int *P, int len_bytes);
int hmmh_write_model_streams(const char *path, const hmmh_model *streams, int P);

/* Bulk .hmm I/O (SURVEY 8f-3): V model files of one topology <-> the struct-of-arrays layout of hmmcu_set_models.
 * Replaces the recogniser's model-list walk (R-FS:214-238) and its one-fread-per-field reading_model (R-FS:612-712):
 * one read per file, a pool of `nthreads` (0 = as hmmh_ingest), parsed straight into the arrays.  Files with the 4-byte
 * length header shipped with the reference are accepted; the writer produces the bytes of hmmh_write_model.
 * *bad_file = index of the file that failed (HMMCU_EIO: unreadable / truncated; HMMCU_EINVAL: another topology). */
typedef struct hmmh_model_set {
  int V, N, M, D;
  char (*word)[64]; /* [V], NUL-terminated */
  double *A;        /* [V][N][N] */
  double *c;        /* [V][N][M] */
  double *mu;       /* [V][N][M][D] */
  double *inv_var;  /* [V][N][M][D] */
  double *det;      /* [V][N][M] */
} hmmh_model_set;
int hmmh_model_set_alloc(hmmh_model_set *s, int V, int N, int M, int D);
void hmmh_model_set_free(hmmh_model_set *s);
int hmmh_read_model_set(const char *const *paths, int V, int nthreads, hmmh_model_set *s, int *bad_file);
int hmmh_write_model_set(const char *const *paths, const hmmh_model_set *s, int nthreads, int *bad_file);
int hmmh_upload_model_set(hmmcu_ctx *ctx, const hmmh_model_set *s);

/* creating_initial_model (T-FS:732-1317): uniform left-to-right A, uniform segmentation, LBG
 * splitting + 3 k-means passes, per-cluster variance and weights. */
int hmmh_init_model(hmmh_model *m, const double *x, const int64_t *frame_off, int U);
/* M-step from one model's statistics vector (T-FS:328-346, 1862-1955, 1338-1359). */
int hmmh_mstep(hmmh_model *m, const double *stats);
/* The extended Baum-Welch update of hmmcu_mstep_ebw on the host, from one model's numerator and denominator statistics
 * vectors (blocks 0 and 1 of hmmcu_estep_mmi's buffer); means, inverse variances and determinants in place. */
int hmmh_mstep_ebw(hmmh_model *m, const double *num, const double *den, double E, double tau);

/* hmmcu_set_models from an array of V host models of identical topology. */
int hmmh_upload_models(hmmcu_ctx *ctx, const hmmh_model *models, int V);

/* All-reduce hook for multi-process training: called once per EM iteration with the DEVICE
 * statistics buffer; must sum it in place across ranks on `stream`.  NULL = single process. */
typedef int (*hmmh_allreduce_fn)(void *user, double *dev_buf, int64_t n_doubles, void *stream);

/* The EM loop of the trainer's main() (T-FS:238-361) for V words at once: every word keeps its
 * own convergence test |old - new| / |old| > 1e-3 (old starts at 1.0) and stops on its own
 * iteration; the model returned is the one that produced the last E-step's probability.
 * utt2model maps the context's utterances to models.  mean_logp[V], iterations[V] out. */
int hmmh_train(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *utt2model, int U,
               double *mean_logp, int *iterations, int max_iter, hmmh_allreduce_fn allreduce,
               void *user);

/* The same loop with hmmcu_estep_viterbi as its E-step: Viterbi training, e.g. to refine initial models before
 * hmmh_train (a few iterations with max_iter = k, then hmmh_train from the result).  One feature stream. */
int hmmh_train_viterbi(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *utt2model, int U,
                       double *mean_logp, int *iterations, int max_iter, hmmh_allreduce_fn allreduce,
                       void *user);

/* MMI training of V words from their current models (e.g. Baum-Welch trained): upload, then per iteration
 * hmmcu_estep_mmi(label, kappa, max_hyp), the hook on the whole [2][V][stats_size] buffer, objective[k] = F / n_utt of
 * the models entering iteration k (F = -sum_v den.sum_logp[v], n_utt = sum_v den.n_utt[v], after the all-reduce), and
 * hmmcu_mstep_ebw(E, tau); the models are downloaded at the end.  A fixed number of iterations, no stopping rule.
 * objective[iterations] may be NULL.  One feature stream. */
int hmmh_train_mmi(hmmcu_ctx *ctx, hmmh_model *models, int V, const int32_t *label, int U, double kappa, int max_hyp,
                   double E, double tau, int iterations, double *objective, hmmh_allreduce_fn allreduce, void *user);

/* The same loop for models of P feature streams: ctxs[p] holds the features of stream p, models[p * V + v] is stream p
 * of word v; ctxs[1..P-1] are linked to ctxs[0] for the duration of the call (hmmcu_link_streams). */
int hmmh_train_streams(hmmcu_ctx *const *ctxs, int P, hmmh_model *models, int V, const int32_t *utt2model, int U,
                       double *mean_logp, int *iterations, int max_iter, hmmh_allreduce_fn allreduce, void *user);

/* Drop-in programs: same argv, files and exit codes as the reference's main()s
 * (T-FS:101-391 and R-FS:87-428). */
int hmmh_train_main(int argc, char **argv);
int hmmh_test_main(int argc, char **argv);

#ifdef __cplusplus
}
#endif
#endif /* HMM_CUDA_H */
