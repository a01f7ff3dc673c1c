/*
 * trlda_b200.h — C ABI of the B200-native trlda hot path.
 *
 * This is the drop-in boundary: every entry point replaces one virtual method (or accessor) of the
 * reference's `class TRLDA::LDA` and its three subclasses, i.e. exactly what the reference's CPython
 * binding calls (`self->lda->...`).  Citations are relative to /root/reference/.
 *
 * Conventions
 *   - plain C: opaque handle, plain pointers and sizes, POD structs; no C++/torch/Python types.
 *   - every function returns an int status (TRLDA_OK == 0).  On failure the message is available from
 *     trlda_last_error(model) (or trlda_last_error(NULL) when no model exists yet).  The messages of the
 *     reference's `TRLDA::Exception`s are kept verbatim (code/trlda/include/lda.h:146-190,
 *     code/trlda/src/lda.cpp:166).
 *   - all matrices crossing the boundary are HOST pointers to float64 in COLUMN-MAJOR order, the layout of
 *     Eigen::ArrayXXd and of the arrays the reference binding returns (python/src/pyutils.cpp:25):
 *     lambda is K x V (word w's K-vector is contiguous at lambda + w*K), gamma is K x B.
 *   - a minibatch is a CSR triple on the host: doc_ptr[B+1], word_ids[N], counts[N] — the flattened form of
 *     `LDA::Documents` = vector<vector<pair<int,int>>> (code/trlda/include/lda.h:21-23).  Duplicate word ids
 *     inside a document and empty documents are legal (lda.cpp:105-109).
 *   - there is no CPU fallback: every compute entry point fails with TRLDA_ERR_CUDA if no B200 is usable.
 */
#ifndef TRLDA_B200_H
#define TRLDA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* exported from libtrlda_b200.so (everything else in the library has hidden visibility) */
#define TRLDA_API __attribute__((visibility("default")))

#define TRLDA_OK            0
#define TRLDA_ERR_ARG       1   /* reference would have thrown TRLDA::Exception -> RuntimeError */
#define TRLDA_ERR_CUDA      2   /* CUDA / NCCL failure, or no device                              */
#define TRLDA_ERR_UNSUPPORTED 3 /* e.g. inference_method == GIBBS in update_parameters / lower_bound     */
#define TRLDA_END           4   /* trlda_reader_next: no more batches                             */

/* model kinds: the three concrete subclasses of TRLDA::LDA */
#define TRLDA_KIND_ONLINE     0   /* code/trlda/include/onlinelda.h:7     */
#define TRLDA_KIND_BATCH      1   /* code/trlda/include/batchlda.h:7      */
#define TRLDA_KIND_CUMULATIVE 2   /* code/trlda/include/cumulativelda.h:7 */

/* precision of the per-document E-step working set */
#define TRLDA_PRECISION_FP64  0   /* everything in float64 (parity mode, <=1e-9 rel)                        */
#define TRLDA_PRECISION_MIXED 1   /* expElogbeta tile + inner products in float32, gamma/sstats in float64  */

#define TRLDA_INFERENCE_VI    0
#define TRLDA_INFERENCE_GIBBS 1

typedef struct trlda_model trlda_model;

/* POD mirror of `LDA::Parameters` (code/trlda/include/lda.h:32-78); same fields, same order, same defaults. */
typedef struct trlda_params {
	int32_t inference_method;     /* VI                 */
	double  threshold;            /* 0.001              */
	int32_t max_iter_inference;   /* 100 (the Online binding overrides to 20, onlineldainterface.cpp:226) */
	int32_t max_iter_tr;          /* 10                 */
	double  tau;                  /* 100.               */
	double  kappa;                /* .7                 */
	double  rho;                  /* -1. (= use schedule) */
	int32_t adaptive;             /* false              */
	int32_t num_samples;          /* 1   (Gibbs only)   */
	int32_t burn_in;              /* 2   (Gibbs only)   */
	int32_t init_gamma;           /* true               */
	int32_t update_lambda;        /* true               */
	int32_t update_alpha;         /* false              */
	int32_t update_eta;           /* false              */
	double  min_alpha;            /* 1e-6               */
	double  min_eta;              /* 1e-6               */
	int32_t max_epochs;           /* 100                */
	int32_t max_iter_alpha;       /* 10                 */
	int32_t max_iter_eta;         /* 20                 */
	double  emp_bayes_threshold;  /* 1e-8               */
	int32_t verbosity;            /* 0                  */
} trlda_params;

/* fills in the defaults of LDA::Parameters::Parameters (lda.h:56-77) */
TRLDA_API void trlda_params_default(trlda_params* p);

/* CSR view of `LDA::Documents` (host memory, not owned) */
typedef struct trlda_docs {
	int64_t        num_docs;   /* B                          */
	const int64_t* doc_ptr;    /* B+1 offsets into the pairs */
	const int32_t* word_ids;   /* N word ids, 0 <= id < V    */
	const int32_t* counts;     /* N word counts              */
} trlda_docs;

/* per-kernel device timings accumulated while profiling is on (CUDA events on the model's stream) */
#define TRLDA_NUM_KERNEL_KINDS 12
typedef struct trlda_stats {
	int64_t launches[TRLDA_NUM_KERNEL_KINDS];   /* number of launches per kernel kind */
	double  ms[TRLDA_NUM_KERNEL_KINDS];         /* summed device time per kind        */
	int64_t estep_doc_iterations;               /* sum over docs of inner iterations run by the last E-step */
	int64_t estep_docs;                         /* documents in the last E-step                             */
	int64_t total_launches;                     /* all kernels launched since the last reset                */
	int64_t h2d_bytes;                          /* host->device bytes since the last reset                  */
	int64_t d2h_bytes;                          /* device->host bytes since the last reset                  */
	int64_t estep_sweeps;                       /* sum over all E-steps since the last reset of (inner iterations + 1)
	                                               per document: how often the E-step kernels went over a tile  */
	int64_t estep_calls;                        /* E-steps (updateVariablesVI calls) since the last reset     */
} trlda_stats;
TRLDA_API const char* trlda_kernel_kind_name(int kind);

/* ---- lifetime -------------------------------------------------------------------------------------------- */

/* Replaces the constructors OnlineLDA/BatchLDA/CumulativeLDA(numWords, [numDocuments,] alpha, eta)
 * (onlinelda.cpp:18-49, batchlda.cpp:22-39, cumulativelda.cpp:22-45).  `alpha` points to K values.
 * lambda is initialised ~ Gamma(100, 1/100) (lda.cpp:71) by the device generator (Cumulative: lambda = eta,
 * cumulativelda.cpp:30).  `num_documents` is ignored for Batch/Cumulative.  `device` is a CUDA ordinal. */
TRLDA_API int trlda_create(int kind, int num_words, int num_topics, int64_t num_documents,
                 const double* alpha, double eta, int device, int precision, trlda_model** out);
TRLDA_API void trlda_destroy(trlda_model* m);   /* Distribution_dealloc, python/src/distributioninterface.cpp:30-37 */
TRLDA_API const char* trlda_last_error(const trlda_model* m);

/* process-wide generator seed; replaces `trlda.seed` -> srand (python/src/module.cpp:332-342) */
TRLDA_API void trlda_seed(uint64_t seed);

/* ---- accessors (lda.h:140-201, onlinelda.h:50-74) ---------------------------------------------------------- */
TRLDA_API int trlda_kind(const trlda_model* m);
TRLDA_API int trlda_precision(const trlda_model* m);
TRLDA_API int trlda_set_precision(trlda_model* m, int precision);
TRLDA_API int trlda_num_topics(const trlda_model* m);                        /* LDA::numTopics  lda.h:194 */
TRLDA_API int trlda_num_words(const trlda_model* m);                         /* LDA::numWords   lda.h:200 */
TRLDA_API int trlda_get_lambda(trlda_model* m, double* lambda_KxV);          /* LDA::lambda     lda.h:180 */
TRLDA_API int trlda_set_lambda(trlda_model* m, const double* lambda_KxV, int rows, int cols);  /* LDA::setLambda lda.h:186 */
TRLDA_API int trlda_get_alpha(trlda_model* m, double* alpha_K);              /* LDA::alpha      lda.h:140 */
TRLDA_API int trlda_set_alpha(trlda_model* m, const double* alpha, int n);   /* LDA::setAlpha   lda.h:146-160 (n==1: scalar form) */
TRLDA_API int trlda_get_eta(trlda_model* m, double* eta);                    /* LDA::eta        lda.h:164 */
TRLDA_API int trlda_set_eta(trlda_model* m, double eta);                     /* LDA::setEta     lda.h:170 */
TRLDA_API int trlda_get_num_documents(trlda_model* m, int64_t* n);           /* OnlineLDA::numDocuments    onlinelda.h:50 */
TRLDA_API int trlda_set_num_documents(trlda_model* m, int64_t n);            /* OnlineLDA::setNumDocuments onlinelda.h:56 */
TRLDA_API int trlda_get_update_count(trlda_model* m, int64_t* n);            /* OnlineLDA::updateCount     onlinelda.h:64 */
TRLDA_API int trlda_set_update_count(trlda_model* m, int64_t n);             /* OnlineLDA::setUpdateCount  onlinelda.h:70 */

/* ---- the hot path -------------------------------------------------------------------------------------------- */

/* LDA::updateVariables (lda.cpp:119-156) -> LDA::updateVariablesVI (lda.cpp:160-220).
 * `latents` = initial gamma, K x B column-major, or NULL to draw gamma0 ~ Gamma(100, 1/100) on the device
 * (lda.cpp:135).  latents_rows/latents_cols are validated like lda.cpp:165 ("Initial gamma has wrong
 * dimensionality.").  gamma_out (K x B) and sstats_out (K x V) may each be NULL to skip the copy-out.
 * params->inference_method == TRLDA_INFERENCE_GIBBS runs LDA::updateVariablesGibbs (lda.cpp:224-293) instead:
 * `latents` = initial theta (NULL: Dirichlet(1), lda.cpp:123-126), gamma_out receives theta ~ Dirichlet(counts),
 * sstats_out the assignment counts averaged over params->num_samples sweeps after params->burn_in; the draws come
 * from the library's counter-based generator (trlda_seed), not from rand(). */
TRLDA_API int trlda_update_variables(trlda_model* m, const trlda_docs* docs,
                           const double* latents, int latents_rows, int64_t latents_cols,
                           const trlda_params* params, double* gamma_out, double* sstats_out);

/* LDA::updateParameters: OnlineLDA (onlinelda.cpp:53-180), BatchLDA (batchlda.cpp:43-209),
 * CumulativeLDA (cumulativelda.cpp:49-153).  `*result` receives the reference's return value (the learning
 * rate rho for Online; 1.0 for Batch/Cumulative and for an empty batch). */
TRLDA_API int trlda_update_parameters(trlda_model* m, const trlda_docs* docs, const trlda_params* params, double* result);

/* Same as trlda_update_parameters but on the minibatch already resident in HBM (trlda_upload_docs): the
 * device-only leg of bench.py.  No host<->device traffic except the returned scalar. */
TRLDA_API int trlda_upload_docs(trlda_model* m, const trlda_docs* docs);
/* Several minibatches can be kept resident at once: upload into a numbered slot (0..63), then make one of them the
 * current minibatch before trlda_update_parameters_resident.  Used by bench.py so that every timed step sees a
 * minibatch the model has not been trained on, without host<->device traffic in the device-only leg. */
TRLDA_API int trlda_upload_docs_slot(trlda_model* m, const trlda_docs* docs, int slot);
TRLDA_API int trlda_select_docs(trlda_model* m, int slot);
TRLDA_API int trlda_update_parameters_resident(trlda_model* m, const trlda_params* params, double* result);

/* LDA::lowerBound (lda.cpp:297-360; OnlineLDA::lowerBound onlinelda.cpp:184-191).  Follows the INTENDED
 * bound (tests/onlineldavb.py:260-318); lda.cpp:334 mis-indexes a K x V array and is not reproduced.
 * per_doc_out (B values, may be NULL) receives the per-document terms before the num_documents factor. */
TRLDA_API int trlda_lower_bound(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows,
                      int64_t latents_cols, const trlda_params* params, int64_t num_documents,
                      double* bound_out, double* per_doc_out);

/* Document-completion predictive log-likelihood (Hoffman et al. 2013, §5); no reference counterpart.
 * Fits gamma on `observed` (the VI E-step, exactly as trlda_update_variables / trlda_lower_bound do: `latents` = initial
 * gamma or NULL for a fresh draw, params->max_iter_inference / threshold), then scores every pair of `held_out`
 * (same number of documents, document d of both belongs to the same text).  *total_out = sum over documents of
 * per_doc_out[d]; *tokens_out = sum of the held-out counts.  Multi-GPU: both CSRs are this rank's shard; total and
 * tokens are summed over ranks, per_doc_out (B values, may be NULL) is this rank's. */
TRLDA_API int trlda_predictive_log_likelihood(trlda_model* m, const trlda_docs* observed, const trlda_docs* held_out,
        const double* latents, int latents_rows, int64_t latents_cols, const trlda_params* params,
        double* total_out, int64_t* tokens_out, double* per_doc_out);

/* The n most probable topics of every (word, count) pair of `docs` under the variational distribution the E-step fits:
 * gamma as trlda_update_variables computes it (bitwise), then phi_djk = softmax_k(psi(gamma_dk) + psi(lambda_kw) - psi(sum_v lambda_kv)),
 * in fp64 from lambda in fp64 in both precision modes.  topics_out and probs_out (may be NULL) are N x n pair-major: pair j's
 * list at topics_out + j*n, ranked by descending score, equal scores by the smaller topic id.  gamma_out (K x B, may be NULL).
 * 1 <= n <= min(32, K).  Multi-GPU: docs is this rank's shard, outputs are this rank's, no exchange.  No reference counterpart. */
TRLDA_API int trlda_word_topics(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows,
                                int64_t latents_cols, const trlda_params* params, int n,
                                int32_t* topics_out, double* probs_out, double* gamma_out);

/* The n most probable words of every topic, in the order of E[beta_kw] = lambda_kw / sum_w lambda_kw: descending,
 * ties broken by the smaller word id.  ids_out is n x K column-major (topic k's list at ids_out + k*n, rank order);
 * prob_out (may be NULL) receives the matching E[beta_kw].  1 <= n <= min(32, V).  No reference counterpart. */
TRLDA_API int trlda_top_words(trlda_model* m, int n, int32_t* ids_out, double* prob_out);

/* For every topic k and ranks i, j < n of its list ids[k*n ..]: counts_out[(k*n + j)*n + i] = number of documents of
 * `docs` that contain both word ids[k*n+i] and word ids[k*n+j] (the diagonal: documents containing the word).
 * A word is contained in a document when one of its pairs there has a count > 0; duplicate ids count once.
 * *num_docs_out = number of documents (empty ones included).  Multi-GPU: `docs` is this rank's shard; counts and
 * num_docs are summed over ranks.  ids is n x K like trlda_top_words' output; 1 <= n <= 32.  No reference counterpart. */
TRLDA_API int trlda_cooccurrence(trlda_model* m, const trlda_docs* docs, const int32_t* ids, int n,
                                 int64_t* counts_out, int64_t* num_docs_out);

/* Distances between the topics of m and those of `other` (NULL: m itself), with p_i = lambda_i / sum_w lambda_iw the
 * E[beta] of topic i as in trlda_top_words (lambda in fp64 in both precision modes):
 *   TRLDA_DISTANCE_HELLINGER  D_ij = sqrt(max(0, 1 - sum_w sqrt(p_iw q_jw))), symmetric, in [0, 1];
 *   TRLDA_DISTANCE_KL         D_ij = KL(p_i || q_j) = sum_w p_iw log p_iw - sum_w p_iw log q_jw, clamped at 0.
 * out is K_m x K_other column-major: out[j*K_m + i] = D(topic i of m, topic j of other).  The result is reproducible bit
 * for bit, and a self-comparison under Hellinger is exactly symmetric.  Both models must have the same V and live on
 * the same device; a negative entry of lambda, or a zero one in `other` under KL, is an error (TRLDA_ERR_ARG).  A sharded
 * lambda gives TRLDA_ERR_UNSUPPORTED.  Multi-GPU: every rank computes the whole matrix from its own replica, no
 * exchange.  Training state is not changed.  No reference counterpart. */
#define TRLDA_DISTANCE_HELLINGER 0
#define TRLDA_DISTANCE_KL        1
TRLDA_API int trlda_topic_distances(trlda_model* m, trlda_model* other, int metric, double* out);

/* Similar documents by topic.  gamma is K x cols column-major, as trlda_update_variables returns it (Gibbs theta too);
 * a document's topic proportions are theta_d = gamma_d / sum_k gamma_dk, and the distance of two documents is the
 * Hellinger distance of theirs, D(q, d) = sqrt(max(0, 1 - C_qd)), C_qd = sum_k sqrt(theta_qk theta_dk), in fp64 in both
 * precision modes.  A negative, NaN or infinite entry, or a column whose sum is not positive, is an error
 * (TRLDA_ERR_ARG), found before any result is written.
 *
 * trlda_index_documents replaces the model's document index with the cols documents of gamma (cols == 0: no index).
 * The index stays on the device, sqrt(theta) in fp64 (8 bytes a topic and document), until it is replaced or the model is
 * destroyed; building it stages gamma through a bounded buffer.  On any failure the model is left with no index.  At most
 * INT32_MAX documents.
 *
 * trlda_similar_documents returns, for each of the Q = cols query documents, the n indexed documents nearest to it:
 * ids_out and dist_out (may be NULL) are Q x n query-major, query q's list at ids_out + q*n, ordered by C descending and
 * then by the smaller document id (distances non-decreasing; exact ties go to the smaller id).  The result is
 * reproducible bit for bit and does not depend on the other queries of the call.  1 <= n <= min(32, indexed documents);
 * Q = 0 does nothing.
 *
 * Neither call changes lambda, alpha, eta, the update count or the minibatches held on the device, and training does not
 * change the index.  Multi-GPU: every rank searches its own index, no exchange; ids are local to the rank's index.  No
 * reference counterpart. */
TRLDA_API int trlda_index_documents(trlda_model* m, const double* gamma, int rows, int64_t cols);
TRLDA_API int trlda_similar_documents(trlda_model* m, const double* gamma, int rows, int64_t cols, int n,
                                      int64_t* ids_out, double* dist_out);

/* ---- parity seams ---------------------------------------------------------------------------------------------
 * The reference draws gamma0 (lda.cpp:135) and Cumulative's lambda (cumulativelda.cpp:60) from libc rand()
 * inside updateParameters and offers no way to pass them in.  These two calls install values that the NEXT
 * trlda_update_parameters / trlda_lower_bound call uses wherever the reference would have drawn fresh ones
 * (every fresh-gamma E-step of that call uses the same gamma0).  They are consumed by that call. */
TRLDA_API int trlda_inject_initial_gamma(trlda_model* m, const double* gamma0_KxB, int rows, int64_t cols);
TRLDA_API int trlda_inject_initial_lambda(trlda_model* m, const double* lambda_KxV, int rows, int cols);

/* ---- multi-GPU: documents sharded over ranks, one exchange of the sufficient statistics per E-step ----------
 * One process per GPU.  Rank 0 obtains an id, the host plumbing broadcasts its 128 bytes, every rank calls
 * trlda_comm_init.  Afterwards `docs` passed to the hot-path calls are THIS RANK'S shard; batch-wide
 * quantities (B, word counts, sstats, alpha statistics) are summed over ranks with NCCL on the model's
 * stream.  All ranks must hold identical lambda/alpha/eta and make the same calls. */
TRLDA_API int trlda_comm_unique_id(void* id_out_128_bytes);
TRLDA_API int trlda_comm_init(trlda_model* m, const void* id_128_bytes, int rank, int nranks);
TRLDA_API int trlda_comm_size(const trlda_model* m);

/* ---- instrumentation ------------------------------------------------------------------------------------------ */
TRLDA_API void* trlda_stream(trlda_model* m);                 /* the cudaStream_t all kernels of this model run on */
TRLDA_API int trlda_synchronize(trlda_model* m);
TRLDA_API int trlda_set_profiling(trlda_model* m, int on);    /* bracket every kernel with CUDA events              */
TRLDA_API int trlda_get_stats(trlda_model* m, trlda_stats* out);
TRLDA_API int trlda_reset_stats(trlda_model* m);
TRLDA_API int trlda_get_row_sums(trlda_model* m, double* row_sums_K);   /* sum_w lambda_kw, a cheap per-step result */

/* LDA::sample (lda.cpp:88-115): num_documents documents of Poisson(length) words drawn from the model's generative
 * process (beta_k ~ Dirichlet(lambda_k), theta ~ Dirichlet(alpha)) on the device.  collapse = 0: every word is emitted
 * as (word id, 1) in the order drawn, repeated ids included, like the reference; collapse = 1: unique (word id, count)
 * pairs sorted by id, the form load_documents produces.  `out` receives a CSR view of host memory owned by the model,
 * valid until the next trlda_sample / trlda_destroy on it.  Seeded by trlda_seed. */
TRLDA_API int trlda_sample(trlda_model* m, int64_t num_documents, double length, int collapse, trlda_docs* out);

/* Test hook for the multi-GPU token list (csrc/csc.cu; no counterpart in the reference, where one process sees the whole
 * minibatch): builds, on the device, the word-sorted token list of a gathered minibatch - `ranks` segments of `max_docs`
 * documents (len, 0 for padding) and `max_pairs` token slots (ids, -1 for padding) each - restricted to the words
 * [v0, v1).  Host arrays in and out: word_ptr has num_words + 1 entries, tok_doc / tok_src ranks * max_pairs. */
TRLDA_API int trlda_debug_global_csc(trlda_model* m, const int32_t* len, const int32_t* ids, int ranks, int64_t max_docs,
                           int64_t max_pairs, int v0, int v1, int32_t* word_ptr, int32_t* tok_doc, int32_t* tok_src);

/* Native reader for the text format of python/utils/load_documents.py:6-69 (one document per line,
 * `N id:cnt id:cnt ...`, first field ignored): the file is memory-mapped and parsed by a background thread into CSR
 * minibatches of `batch_size` documents (0: the whole file) in pinned host memory, `prefetch` batches ahead of the
 * consumer.  Batches come in the reference generator's order: full batches, then the remainder — yielded even if it
 * is empty (load_documents.py:63) — then TRLDA_END.  The view handed out by trlda_reader_next stays valid until the
 * call after the next one. */
typedef struct trlda_reader trlda_reader;
TRLDA_API int trlda_reader_open(const char* path, int64_t batch_size, int prefetch, trlda_reader** out);
TRLDA_API int trlda_reader_next(trlda_reader* r, trlda_docs* out, int* pinned);
TRLDA_API void trlda_reader_close(trlda_reader* r);
TRLDA_API const char* trlda_reader_last_error(const trlda_reader* r);

/* device special functions evaluated on n host values (test hook pinning the in-kernel psi / psi' / lgamma
 * against python/tests/utils_test.py:33-51): which = 0 digamma fp64, 1 trigamma fp64, 2 lgamma fp64,
 * 3 exp(digamma) as evaluated in mixed-precision mode (beta-prep), 4 exp(digamma) as evaluated in fp64 mode,
 * 5 exp(digamma) as evaluated inside the mixed-mode E-step kernel (exp_digamma_lean). */
TRLDA_API int trlda_device_special(int device, int which, const double* x, int64_t n, double* out);

/* host special functions used by the Newton steps: polygamma(n, x) of utils.cpp:107-111 (n = 0, 1, 2) */
TRLDA_API double trlda_polygamma(int n, double x);

#ifdef __cplusplus
}
#endif
#endif
