/*
 * kmerlr_b200.h -- C ABI of libkmerlr_b200.so, the B200 (sm_100a) implementation of the
 * data-parallel hot path of pbenner/kmerLr.
 *
 * The reference is a single Go `package main` with no FFI of its own; the drop-in boundary is
 * therefore the set of Go function seams listed in SURVEY.md section 8b.  Each entry point below
 * names the reference function whose BODY it replaces (the Go signature stays; INTEGRATION.md
 * shows the cgo shim).  All entry points take plain pointers and sizes, return 0 on success and
 * a non-zero code on failure (text via kmerlr_last_error()); there is no CPU fallback.
 *
 * Conventions (SURVEY 8b):
 *   - the caller owns every buffer it passes; nothing is retained after return;
 *   - matrices live in HBM behind opaque handles; rows are CSR WITHOUT the bias column:
 *     column j here is Go sparse index j+1, the implicit bias (index 0, value 1.0) is added
 *     by every kernel, so theta[0] is the bias and theta[j+1] belongs to column j;
 *   - indices strictly increasing inside a row, no explicit zeros (kmerLr_test.go:117-123);
 *   - one process drives one GPU; with kmerlr_comm_init() the rows of a matrix are this rank's
 *     SHARD and gradient / loss / select / proxgrad reduce over all ranks (NCCL).
 */
#ifndef KMERLR_B200_H
#define KMERLR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef uint64_t kmerlr_handle;

/* NewKmerCounter(M, N, complement, reverse, revcomp, maxAmbiguous, alphabet) -- kmerLr_learn.go:94,
 * kmerLr_classifier.go:96-103; binarize selects IdentifyKmers (kmerLr_data.go:257-263). */
typedef struct kmerlr_config {
  int32_t M, N;
  int32_t complement, reverse, revcomp;
  int32_t binarize;
  int32_t alphabet;       /* 0 = nucleotide; 1 = gapped nucleotide (sort-based path, N <= 11) */
  int32_t max_ambiguous;  /* -1 = nil */
} kmerlr_config;

#define KMERLR_OK             0
#define KMERLR_ERR_ARG        1   /* log.Fatal-class: bad argument / unsupported configuration */
#define KMERLR_ERR_CUDA       2   /* CUDA / NCCL runtime failure */
#define KMERLR_ERR_INTERNAL   3   /* panic("internal error")-class invariant violation */
#define KMERLR_ERR_NOGPU      4   /* no usable sm_100 device: the product path never falls back */

#define KMERLR_TIE_GO118 0        /* order of Go <= 1.18 sort.Sort (what the shipped goldens encode) */
#define KMERLR_TIE_INDEX 1        /* |g| descending, then coefficient index ascending */

#define KMERLR_FLAG_SHARDED 1     /* rows are this rank's shard; call is collective over the communicator */

/* ---- lifecycle (Go init / exit) ------------------------------------------------------------- */
int         kmerlr_init(int device);
int         kmerlr_shutdown(void);
const char *kmerlr_last_error(void);
int         kmerlr_version(void);
/* device-side time of the last call's kernels in milliseconds (CUDA events on the library stream) */
double      kmerlr_last_device_ms(void);
/* number of kernels the library has launched since kmerlr_init (bench.py reports gpu_launches) */
int64_t     kmerlr_launch_count(void);
/* per-kernel device time: CUDA events around every launch while enabled (enable clears the totals);
 * read sums the kernels whose name contains the substring; dump = "name\tms\tlaunches\n" lines */
int         kmerlr_profile(int enable);
int         kmerlr_profile_read(const char *kernel_substr, double *ms_total, int64_t *launches);
int         kmerlr_profile_dump(char *buf, int64_t buflen);

/* run-time switches (tests and experiments):
 *   "implicit" = 1 (default) lets matrices that came straight from kmerlr_extract (count or binarized, one
 *                column per class) use the matrix-free logistic pass, 0 forces the pass over the stored rows;
 *   "super_len" = length S of the super k-mer tables of that pass (S - N + 1 positions share one table
 *                entry; -1 = automatic: 10 for N <= 8, else 11; 0 = off);
 *   "hot_cols" = number of columns of that stored-row pass that accumulate in shared memory (default 6144);
 *   "fused_ticket" = rows a warp of the stored-row pass takes per ticket (default 8; 0 = static grid of blocks);
 *   "p2p"      = 1 (default) lets sharded reduced-matrix iterations exchange the gradient over NVLink peer
 *                memory, 0 forces the NCCL collectives (set it identically on every rank);
 *   "feed_growth" = growth of the chunk sizes of a pipelined host feed in per cent (default 135; measured at C2:
 *                100 .. 135 give the same 3.15 ms per extraction from host buffers);
 *   "small_long" = 1 runs the reduced-matrix solver on the sliced + column-major views of the matrix (long rows), 2 on
 *                the sliced view + a block-local column-major view (one grid barrier per iteration), 0 on the compact
 *                rows, -1 (default) chooses by the row length (8 entries per row and more: 2 when the counts fit its packed
 *                word, else 1); same bits;
 *   "persist_bps" = blocks per SM of the persistent reduced-matrix solver (0 = as many as fit, the default);
 *   "p2p_allreduce" = 1 runs the int64 all-reduce of the full-space gradient as a two-shot exchange over NVLink peer
 *                memory in one cooperative launch instead of NCCL (default 0: NCCL is faster at these sizes; same bits);
 *   "persistent" = 1 (default) runs the reduced-matrix iterations of one GPU as one cooperative launch per
 *                batch of iterations (grid barriers), 0 as one launch per iteration */
int         kmerlr_option(const char *name, int64_t value);

/* ---- sample sharding over the GPUs of one box (SURVEY 8e) ------------------------------------ */
int kmerlr_comm_unique_id(void *id128);                       /* ncclGetUniqueId, 128 bytes       */
int kmerlr_comm_init(int rank, int world, const void *id128); /* ncclCommInitRank                 */
int kmerlr_comm_destroy(void);

/* ---- stage 1: sequences -> sparse rows -------------------------------------------------------
 * Replaces the bodies of scan_sequences + NewKmerCountsList/SetKmers + convert_counts_list, i.e.
 * what compile_training_data / compile_test_data / compile_data do between import_fasta and the
 * returned KmerDataSet (kmerLr_data.go:197-357).
 *   seq, off[n+1]   concatenated sequence bytes (ASCII, any case) and their offsets
 *   frozen_*        class list of a frozen counter (sorted by (k, code)); NULL/0 = discover the
 *                   union of observed classes (unfrozen counter)
 *   features        n_features x 2 class-index pairs (convert_counts, kmerLr_data.go:210-229);
 *                   NULL/0 = one column per class (generate_features = true)
 */
int kmerlr_sequences_create(const uint8_t *seq, const int64_t *off, int64_t n, kmerlr_handle *out);
int kmerlr_extract_resident(const kmerlr_config *cfg, kmerlr_handle sequences,
                            const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                            const int32_t *features, int64_t n_features, int flags, kmerlr_handle *out);
int kmerlr_extract(const kmerlr_config *cfg, const uint8_t *seq, const int64_t *off, int64_t n,
                   const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                   const int32_t *features, int64_t n_features, int flags, kmerlr_handle *out);

/* KmerDataSet accessors (Data / Labels / Kmers, kmerLr_data.go:34-38) */
int kmerlr_matrix_info(kmerlr_handle h, int64_t *n, int64_t *m, int64_t *nnz, int64_t *n_classes);
/* len(data.Data) of the WHOLE data set: the rows of all ranks for a sharded matrix (what the reference's
 * n = len(data.Data) is, kmerLr_estimator.go:239), the same as *n otherwise */
int kmerlr_matrix_rows_global(kmerlr_handle h, int64_t *n_global);
int kmerlr_matrix_classes(kmerlr_handle h, int32_t *k_out, uint64_t *code_out);
int kmerlr_matrix_rows(kmerlr_handle h, int64_t *rowptr, int32_t *col, double *val);
int kmerlr_matrix_set_labels(kmerlr_handle h, const uint8_t *labels, int64_t n);
int kmerlr_matrix_from_csr(int64_t n, int64_t m, const int64_t *rowptr, const int32_t *col,
                           const double *val, int flags, kmerlr_handle *out);
/* per column (all ranks): sum of the values, sum of squares, largest value, number of stored entries --
 * what TransformFull.Fit computes its offsets / scales from (kmerLr_transform.go:59-252); count and
 * binarized matrices only.  The transform itself is a reparameterisation of theta on the host side. */
int kmerlr_column_moments(kmerlr_handle h, double *sum_m, double *sumsq_m, double *absmax_m, int64_t *count_m);
/* the same four moments of the pair features v_a v_b, a < b, in CoeffIndex order (position = Ind2Sub(a, b) - (m + 1)):
 * TransformFull.Fit with cooccurrence (kmerLr_transform.go:90-99,118-127); m (m - 1) / 2 entries each */
int kmerlr_pair_moments(kmerlr_handle h, double *sum_p, double *sumsq_p, double *absmax_p, int64_t *count_p);
/* Transform.Apply (kmerLr_transform.go:584-629) on the rows of a (reduced) matrix, as estimate() does before it
 * hands the data to the solver (kmerLr_estimator.go:148): offset / scale per coefficient (index 0 = bias), either
 * may be NULL.  With an offset every entry, zeros included, becomes (v - offset_j) scale_j -- dense rows, meant for
 * the reduced matrix of the selected features; scale only keeps the sparsity.  Returns a new matrix (labels copied). */
int kmerlr_matrix_transform(kmerlr_handle h, const double *offset_or_null, const double *scale_or_null, int64_t len,
                            kmerlr_handle *out);
int kmerlr_free(kmerlr_handle h);

/* ---- CoeffIndex (kmerLr_coefficients_index.go:26-54) ---------------------------------------- */
int64_t kmerlr_coeff_dim(int64_t n);
int64_t kmerlr_coeff_ind2sub(int64_t n, int64_t k1, int64_t k2);
void    kmerlr_coeff_sub2ind(int64_t n, int64_t i, int64_t *k1, int64_t *k2);

/* ---- stage 2: logisticRegression (kmerLr_logistic_regression.go:30-272) ----------------------
 * ntheta = m+1, or CoeffIndex(m).Dim() when cooccurrence != 0.  lambda NaN or 0 = no penalty. */
int kmerlr_linear_pdf(kmerlr_handle h, const double *theta, int64_t ntheta, int cooccurrence, double *out_n);
int kmerlr_logpdf    (kmerlr_handle h, const double *theta, int64_t ntheta, int cooccurrence, double *out_n);
int kmerlr_gradient  (kmerlr_handle h, const double *theta, int64_t ntheta, const double class_w[2],
                      double lambda, int cooccurrence, double *g_out);
int kmerlr_loss      (kmerlr_handle h, const double *theta, int64_t ntheta, const double class_w[2],
                      double lambda, int cooccurrence, double *loss_out);
/* compute_class_weights (kmerLr_data.go:178-193) over the (global) labels of the matrix */
int kmerlr_class_weights(kmerlr_handle h, double class_w_out[2]);

/* ---- leapfrog selection (kmerLr_feature_selection.go:78-134,179-219; kmerLr_sort.go:120-131) --
 * active_idx: full-space coefficient indices (>= 1) of the current model, active_theta their
 * values; mask_out[ntheta] receives b; *ok_out what Select returns as its third value. */
int kmerlr_select(kmerlr_handle h, const double class_w[2], int cooccurrence, int64_t N, double theta0,
                  const int64_t *active_idx, const double *active_theta, int64_t n_active, int tie,
                  double epsilon_lambda, double prev_lambda, uint8_t *mask_out, int64_t ntheta,
                  double *lambda_out, int64_t *c_out, int *ok_out, double *g_out_or_null);
/* the same selection for a gradient the caller already holds (e.g. the gradient under a data transform,
 * which is a reparameterisation on the host side): everything of Select after its gradient call */
int kmerlr_select_from_gradient(const double *g, int64_t ntheta, int64_t N, const int64_t *active_idx,
                                const double *active_theta, int64_t n_active, int tie, double epsilon_lambda,
                                double prev_lambda, uint8_t *mask_out, double *lambda_out, int64_t *c_out,
                                int *ok_out);
/* featureSelection.Data (kmerLr_feature_selection.go:309-343): sel[0] = 0 (bias) */
int kmerlr_reduce(kmerlr_handle h, const int64_t *sel, int64_t nsel, kmerlr_handle *out);

/* ---- proximal-gradient estimator (kmerLr_estimator_proximal.go:30-120; hook: _hook.go:46-99) --
 * Same shape as (*KmerLrEstimator).estimate (kmerLr_estimator.go:147): fits theta on the reduced
 * matrix.  hook_state = {loss_old, loss_new} of the Go closure, carried between calls. */
int kmerlr_step_size(kmerlr_handle h, double l2, double step_factor, double *step_out);
int kmerlr_proxgrad(kmerlr_handle h, double *theta_inout, int64_t ntheta, const double class_w[2],
                    double lambda, double l2, double step_factor, double epsilon, double epsilon_loss,
                    int64_t max_iter, double hook_state[2], int64_t *iters_out, double *delta_out);

/* ---- IRLS + coordinate-descent estimator (kmerLr_estimator_coordinate.go:31-139), reduced matrices only
 * (ntheta <= 1024: it keeps the dense Gram matrix, as the reference does), one GPU.  The reference never
 * calls it and its theta slices alias (:89-91); built with the slices de-aliased, like kmerlr_proxgrad.
 * The IRLS weights use compute_class_weights(labels) (:88), the hook's loss class_w_hook (the estimator's
 * ClassWeights, kmerLr_estimator_hook.go:36-42) and lambda = l1reg / n.  sweeps_out = coordinate sweeps done.
 * PARITY UNPINNED IN THE REFERENCE ITSELF: no test, no golden and no caller there; the numpy restatement it is
 * checked against (oracle/oracle.py:coordinate) is pinned by optimality properties only. */
int kmerlr_coordinate(kmerlr_handle h, double *theta_inout, int64_t ntheta, const double class_w_hook[2],
                      double l1reg, double l2reg, double epsilon, double epsilon_loss, int64_t max_iter,
                      double hook_state[2], int64_t *sweeps_out, double *delta_out);

/* ---- stage 3: genomicKmerLr.Predict / predict_window_genomic (kmerLr_predict_genomic.go:134-171)
 * One model = one KmerLrEnsemble; the per-window result is the sum over models of the ensemble
 * summary of log sigma(x . theta) (kmerLr_classifier_ensemble.go:64-139).
 * Accepted: every model the extraction builds -- the nucleotide alphabet with 1 <= M <= N <= 14 and any subset of
 * complement / reverse / revcomp, the gapped nucleotide alphabet with N <= 11 and any max_ambiguous, any number of
 * model classes, any window size, 1..16 ensemble members.  Refused (KMERLR_ERR_ARG): the IUPAC alphabet, more than
 * 16 members, an ensemble without a summary, classes outside [M, N] or with a code out of range, duplicate classes,
 * feature indices out of range. */
#define KMERLR_SUMMARY_NONE 0
#define KMERLR_SUMMARY_MEAN 1
#define KMERLR_SUMMARY_PRODUCT 2
#define KMERLR_SUMMARY_MIN 3
#define KMERLR_SUMMARY_MAX 4
typedef struct kmerlr_model {
  kmerlr_config   cfg;
  int64_t         n_classes;
  const int32_t  *class_k;
  const uint64_t *class_code;
  int64_t         n_features;
  const int32_t  *features;   /* n_features x 2 */
  int64_t         n_members;
  const double   *theta;      /* n_members x (n_features+1) */
  int32_t         summary;
} kmerlr_model;
int64_t kmerlr_window_slots(int64_t len, int64_t W, int64_t step);
int kmerlr_score_windows(const kmerlr_model *models, int n_models, const uint8_t *seq,
                         const int64_t *region_off, int64_t n_regions, int64_t W, int64_t step,
                         double *out);
/* predict_window of the `predict --sliding-window` command (kmerLr_predict.go:89-124): one classifier, every
 * sequence gets len - W slots (none if len <= W) and the window starting at j = 0, step, 2 step, ... < len - W
 * lands in slot j; the other slots stay 0.0.  The classifier's Transform is not applied there either. */
int kmerlr_predict_windows(const kmerlr_model *model, const uint8_t *seq, const int64_t *seq_off, int64_t n_seq,
                           int64_t W, int64_t step, double *out);
int kmerlr_score_windows_resident(const kmerlr_model *models, int n_models, kmerlr_handle sequences,
                                  int64_t W, int64_t step, double *out_host_or_null,
                                  kmerlr_handle *out_dev_or_null);

/* ---- on-disk formats either side of the path (SURVEY 8f-4) ------------------------------------
 * The bytes the reference's fmt verbs produce; filename "" = standard output where the reference allows it.
 *
 * saveWindowPredictionsWiggle (kmerLr_predict_genomic.go:37-60): "track type=wiggle_0 name=<track>", per region
 * "fixedStep chrom=<name> start=<from + W/2> step=<step> span=<step>" and one "%0.15f" of exp(prediction) per slot.
 * The records are formatted on the device: exp of a log-probability lies in [0, 1] and prints as 18 bytes, so record j
 * sits at byte 18 j (exact decimal expansion, round half to even; exp = Go's portable math.Exp, see formats.cu).
 * Predictions of region i = pred[slot_off[i], slot_off[i+1]) (kmerlr_window_slots per region); pred is a host array,
 * or NULL with `scores` = the device handle kmerlr_score_windows_resident returned. */
#define KMERLR_WIGGLE_RECORD 18
int kmerlr_wiggle_records(const double *pred, int64_t n, char *out_18n, int64_t *n_irregular_out);
int kmerlr_save_wiggle(const char *filename, const char *track_name, int64_t n_regions, const char *const *seqnames,
                       const int64_t *from, const int64_t *slot_off, const double *pred_or_null, kmerlr_handle scores,
                       int64_t window_size, int64_t window_step);
/* export_kmers (kmerLr_data.go:127-174): the class names ("aaaatt|aatttt") joined by ',', then every row dense:
 * "%d" of the counts, or "%e" when as_float != 0 (data that went through kmerlr_matrix_transform, as
 * kmerLr_export.go:45-56 does before it exports).  kmerlr_class_name: the printed name of one class. */
int kmerlr_export_kmers(kmerlr_handle data, const kmerlr_config *cfg, const char *filename, int as_float);
int kmerlr_class_name(const kmerlr_config *cfg, int32_t k, uint64_t code, char *buf, int64_t buflen);
/* KmerRegularizationPath.Export (kmerLr_estimator_path.go:41-73); estimator may be NULL (no such column);
 * theta of entry i = theta[theta_off[i], theta_off[i+1]) */
int kmerlr_export_path(const char *filename, int64_t n, const int64_t *estimator_or_null, const double *lambda,
                       const double *norm, const int64_t *theta_off, const double *theta);
/* Trace.Export (kmerLr_estimator_trace.go:28-80); durations in nanoseconds (time.Duration); lambda / loss may be NULL */
int kmerlr_export_trace(const char *filename, int64_t n, const int64_t *duration_ns, const int64_t *iteration,
                        const double *change, const int64_t *nonzero, const double *lambda_or_null,
                        const double *loss_or_null);

#ifdef __cplusplus
}
#endif
#endif
