// kernels.cuh — launch interface between the host model (model.cu) and the sm_100a kernels (kernels.cu).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace trlda {

// kernel kinds for the per-kernel timing table (trlda_stats in include/trlda_b200.h)
enum KernelKind {
	KK_ROWSUM = 0,        // row sums of lambda (K x V -> K)
	KK_BETA_PREP = 1,     // expElogbeta = exp(psi(lambda) - psi(rowsum))
	KK_ESTEP = 2,         // per-document gamma/phi fixed point
	KK_SCATTER_MSTEP = 3, // segmented scatter fused with the M-step blend and the next beta-prep
	KK_SCATTER = 4,       // segmented scatter into dense sstats
	KK_MSTEP = 5,         // dense M-step blend (+ beta-prep), used after a cross-GPU exchange
	KK_INIT_UPDATE = 6,   // phi = 1/K warm start of lambda (onlinelda.cpp:79-86) + beta-prep
	KK_REDUCE = 7,        // small deterministic reductions (partials -> K vector / scalar)
	KK_ALPHA_STATS = 8,   // sum_d psi(gamma_dk) - psi(sum_k gamma_dk)
	KK_RNG = 9,           // Gamma(100, 1/100) generator
	KK_ELBO = 10,         // lower-bound kernels
	KK_MISC = 11,         // adaptive-rate update, psi of K row sums, ...
	KK_COUNT = 12
};

// How lambda is rebuilt from the sufficient statistics.
enum MStepMode {
	MSTEP_ONLINE = 0,      // lambda = (1-rho) lambda' + rho (eta + scale * sstats)   onlinelda.cpp:99-100
	MSTEP_BATCH = 1,       // lambda = eta + sstats                                   batchlda.cpp:60
	MSTEP_CUMULATIVE = 2   // lambda = lambda' + sstats                               cumulativelda.cpp:69
};

struct MStepCoef {
	int mode;
	double rho, eta, scale;
};

// Minibatch resident in HBM: CSR by document plus the word-sorted (CSC) view used by the scatter.
struct DeviceDocs {
	int64_t B = 0, N = 0;
	int n_max = 0;                 // longest document (pairs)
	const int64_t* doc_ptr = nullptr;   // B+1
	const int32_t* word_ids = nullptr;  // N
	const int32_t* counts = nullptr;    // N
	const int32_t* word_ptr = nullptr;  // V+1 offsets into the word-sorted token list
	const int32_t* tok_doc = nullptr;   // N: document of the token
	const int32_t* tok_src = nullptr;   // N: CSR position of the token (index into the weight array)
};

struct EStepPlan {
	int cluster = 1;      // CTAs per document
	int kc = 0;           // topic rows per CTA (multiple of 32)
	int n_cap = 0;        // capacity of the per-column vectors in shared memory
	int n_fit = 0;        // columns of the tile kept in shared memory (the rest stream from L2)
	size_t smem = 0;      // dynamic shared memory per CTA
};

// plans the E-step launch for (K, longest document, element size of the expElogbeta working copy)
EStepPlan plan_estep(int K, int n_max, int elem_size, int smem_optin);

struct EStepArgs {
	int K = 0;
	const void* beta = nullptr;     // K x V expElogbeta, float or double
	const double* alpha = nullptr;  // K
	double* gamma = nullptr;        // K x B, in: initial gamma, out: final gamma
	double* etheta = nullptr;       // K x B out: exp(psi(gamma)) of the final state
	float* etheta32 = nullptr;      // optional float copy for the scatter (mixed mode)
	double* weight = nullptr;       // N out: c_j / phiNorm_j of the final state
	double* doc_stat = nullptr;     // K x B out: etheta_dk * sum_j weight_j beta_k,w_j  (row sums of sstats)
	int32_t* iterations = nullptr;  // B out
	int max_iter = 0;
	double threshold = 0;
	unsigned long long* sweeps = nullptr;  // optional counter: += inner iterations + 1 per document (tile sweeps)
	int* work = nullptr;                   // k_estep_tmem: work counter of the launch (documents handed out so far)
	unsigned long long* ticks = nullptr;   // optional phase timers (debug, TRLDA_ESTEP_TICKS=1): 16 sums of clock64 deltas
};

void launch_rowsum(const double* lambda, int K, int V, double* partials, int* num_partials, cudaStream_t s);
int rowsum_num_partials(int V);
void launch_reduce_partials(const double* partials, int num_partials, int K, double* out, cudaStream_t s);
// out[k] = digamma(in[k])
void launch_psi_vector(const double* in, int K, double* out, cudaStream_t s);
// rows_new = a * rows_prev + b + c * rows_stat ; psi_rows = digamma(rows_new)
void launch_rows_update(const double* rows_prev, const double* rows_stat, double a, double b, double c, int K,
                        double* rows_new, double* psi_rows, cudaStream_t s);

void launch_beta_prep(const double* lambda, const double* psi_rows, int K, int V, void* beta, int elem_size,
                      double* psi_partials /* V values or null */, cudaStream_t s);

// documents order[offset .. offset+count) (order == nullptr: identity) are processed by one launch
void launch_estep(const EStepPlan& plan, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order,
                  int64_t offset, int64_t count, int elem_size, cudaStream_t s);
void configure_estep(int smem_optin);

// the same kernel for documents too long for plan_estep's shared memory: the per-pair vectors live in global memory (the
// CSR arrays, args.weight and `scratch`), so the shared memory of a launch does not depend on the document length.
// scratch holds estep_long_scratch_bytes(plan, P) bytes for the P pairs of the documents order[offset .. offset+count).
EStepPlan plan_estep_long(int K, int n_max, int elem_size, int smem_optin);
size_t estep_long_scratch_bytes(const EStepPlan& plan, int64_t pairs);
void launch_estep_long(const EStepPlan& plan, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order,
                       int64_t offset, int64_t count, double* scratch, int64_t scratch_pairs, int elem_size, cudaStream_t s);

// streaming kernel (estep_stream.cu): one CTA per document, columns streamed through per-warp cp.async rings, one sweep
// per inner iteration
bool stream_estep_applicable(int K, int n_max, int elem_size, int smem_optin);
void launch_estep_stream(const EStepArgs& args, const DeviceDocs& docs, const int32_t* order, int64_t offset,
                         int64_t count, int n_max, int elem_size, cudaStream_t s);

// tensor-memory-resident kernel for the mixed mode (estep_tmem.cu): a cluster of CTAs keeps a document's float32 tile
// in tensor memory (+ registers) for all inner iterations; documents of up to tmem_estep_max_len() pairs
bool tmem_estep_applicable(int K, int elem_size);
int tmem_estep_max_len();
int launch_estep_tmem(const EStepArgs& args, const DeviceDocs& docs, const int32_t* order, int64_t offset,
                      int64_t count, int n_max, cudaStream_t s);

// collapsed Gibbs E-step (lda.cpp:224-293): theta_out K x B, sstats K x V (zeroed by the caller), topics = scratch of one
// uint16 per token occurrence, occ_ptr[d] = occurrences before document d
void launch_gibbs(const DeviceDocs& docs, int K, const void* beta, int beta_elem, const double* alpha, const double* theta0,
                  const int64_t* occ_ptr, uint16_t* topics, int num_samples, int burn_in, uint64_t seed, double* theta_out,
                  double* sstats, cudaStream_t s);

// csc.cu: word-sorted token list of the gathered (multi-GPU) minibatch restricted to the words [v0, v1), on the device
size_t global_csc_scratch_ints(int64_t B, int64_t N, int v0, int v1);
void launch_doc_lengths(const int64_t* doc_ptr, int64_t B, int64_t pad_B, int32_t* out, cudaStream_t s);
void launch_global_csc(const int32_t* len, const int32_t* ids, int R, int64_t max_B, int64_t max_N, int v0, int v1, int V,
                       int32_t* scratch, int32_t* word_ptr, int32_t* tok_doc, int32_t* tok_src, cudaStream_t s);

// LDA::sample on the device (sample.cu): row-wise CDFs of beta_k ~ Dirichlet(lambda_k), then one warp per document;
// tokens / counts / lengths are B x cap, B x cap, B device arrays
int sample_capacity(double length);
size_t sample_smem_bytes(int K, int cap);
void launch_sample_beta(const double* lambda, int K, int V, uint64_t seed, double* cdf, cudaStream_t s);
int launch_sample_docs(const double* cdf, const double* alpha, int K, int V, int64_t B, double length, int cap, bool collapse,
                       uint64_t seed, int32_t* tokens, int32_t* counts, int32_t* lengths, cudaStream_t s);

constexpr int TRLDA_MAX_RANKS = 8;    // one NVSwitch node

// segmented scatter.  If `fused`, lambda/beta are rebuilt in the same pass (single-GPU path); else the dense
// K x V statistics are written to `sstats`.
struct ScatterArgs {
	int K = 0, V = 0;
	const void* etheta = nullptr;     // K x B, float or double (etheta_elem)
	int etheta_elem = 8;
	const double* weight = nullptr;   // N
	void* beta = nullptr;             // K x V in (old) / out (new, if write_beta)
	int beta_elem = 8;
	double* sstats = nullptr;         // dense output (unfused)
	float* sstats32 = nullptr;        // dense output rounded to float32, instead of sstats
	// multi-GPU push: instead of a local dense matrix, word w's partial column is stored straight into the memory of
	// the rank that owns w (NVLink peer store), at slot [this rank][w - first word of the owner]
	int peer_ranks = 0, peer_rank = 0, peer_shard_cap = 0, peer_elem = 8;
	void* peer_out[TRLDA_MAX_RANKS] = {};
	// fused part
	bool fused = false;
	MStepCoef coef{};
	const double* lambda_prime = nullptr;
	double* lambda = nullptr;
	const double* psi_rows = nullptr; // psi of the NEW row sums
	bool write_beta = false;
	double* psi_partials = nullptr;   // V values: sum_k psi(lambda_new[k, w]) (for the eta update) or null
	int v0 = 0, v1 = -1;              // word range handled by this launch (v1 < 0: all words); the float32 vector kernel only
};
void launch_scatter(const ScatterArgs& a, const DeviceDocs& docs, cudaStream_t s);

struct MStepArgs {
	int K = 0, V = 0;
	MStepCoef coef{};
	const double* sstats = nullptr;
	const double* lambda_prime = nullptr;
	double* lambda = nullptr;
	const double* psi_rows = nullptr;
	void* beta = nullptr;
	int beta_elem = 8;
	bool write_beta = false;
	double* psi_partials = nullptr;
};
void launch_mstep(const MStepArgs& a, cudaStream_t s);

// Multi-GPU M-step over NVLink peer memory: this rank owns the words [v0, v1).  The scatter kernels of all ranks have
// PUSHED their partial columns for these words into this rank's receive buffer (peer stores, overlapped with the
// scatter itself); this kernel sums the partials in rank order, blends with lambda', and PUSHES the new expElogbeta
// column (and, on request, the new lambda column) into every rank's replica: reduce-scatter + M-step + beta-prep +
// all-gather without an intermediate K x V matrix and without NCCL on the data path.
struct ShardMStepArgs {
	int K = 0, V = 0, v0 = 0, v1 = 0, nranks = 1, rank = 0;
	MStepCoef coef{};
	const void* partials = nullptr;               // LOCAL receive buffer [nranks][shard_cap][K] filled by the peers' scatter kernels
	int shard_cap = 0;
	int sstats_elem = 8;
	void* beta[TRLDA_MAX_RANKS] = {};             // every rank's expElogbeta replica
	double* lambda[TRLDA_MAX_RANKS] = {};         // every rank's target lambda buffer
	const double* lambda_prime = nullptr;         // local
	const double* psi_rows = nullptr;
	int beta_elem = 8;
	bool write_beta = false;
	bool broadcast_lambda = false;                // write lambda to all ranks (else only to this rank's replica)
	double* psi_partials = nullptr;               // V values, this rank fills [v0, v1)
};
void launch_mstep_shard(const ShardMStepArgs& a, cudaStream_t s);

// lambda = (1-rho) lambda' + rho (eta + scale_k * wordcount_w), then beta-prep (onlinelda.cpp:79-86)
void launch_init_update(const DeviceDocs& docs, int K, int V, double rho, double eta, double scale_k,
                        const double* lambda_prime, double* lambda, const double* psi_rows, void* beta,
                        int beta_elem, const double* wordcount /* V, device */, cudaStream_t s);
// wordcount[w] = sum of counts of word w in the minibatch; also total (1 value)
void launch_wordcount(const DeviceDocs& docs, int V, double* wordcount, cudaStream_t s);

// out[k] = sum_d in[k + d*K]  (deterministic two-stage)
void launch_colsum(const double* in, int K, int64_t B, double* partials, double* out, cudaStream_t s);
int colsum_num_partials(int64_t B);

// stat[k + d*K] = psi(gamma_dk) - psi(sum_k gamma_dk)
void launch_alpha_stats(const double* gamma, int K, int64_t B, double* stat, cudaStream_t s);

void launch_gamma_rng(double* out, int64_t n, uint64_t seed, uint64_t stream_id, cudaStream_t s);
void launch_fill(double* out, int64_t n, double value, cudaStream_t s);

// sum of n doubles -> out[0] (deterministic two-stage; partials has >= 1024 slots)
void launch_sum(const double* in, int64_t n, double* partials, double* out, cudaStream_t s);

// adaptive learning rate (onlinelda.cpp:167-175): u = eta + scale*sstats - lambda'; G = (1-1/tau) G + u/tau;
// partial sums of u^2 and G^2 per block -> sq_partials[2 * nblocks]
int adaptive_num_blocks(int64_t n);
void launch_adaptive(const double* sstats, const double* lambda_prime, double* grad, int64_t n, double eta,
                     double scale, double tau, double* sq_partials, cudaStream_t s);

// ELBO: per-document terms and the global beta terms
void launch_elbo_docs(const DeviceDocs& docs, int K, const double* lambda, const double* psi_rows,
                      const double* alpha, double alpha_const, const double* gamma, double* per_doc, cudaStream_t s);
// partial[w] = sum_k (eta - lambda_kw)(psi(lambda_kw) - psi_rows_k) + lgamma(lambda_kw)
void launch_elbo_beta(const double* lambda, const double* psi_rows, int K, int V, double eta, double* partial,
                      cudaStream_t s);
// document-completion predictive log-likelihood: per_doc[d] = sum_j c_j (log sum_k s_dk lambda_{k,w_j} - log sum_k gamma_dk)
// over the pairs of `held_out` (CSR arrays only), s_dk = gamma_dk / rows_k; lambda K x V and rows K are fp64
void launch_heldout_loglik(const DeviceDocs& held_out, int K, const double* lambda, const double* rows, const double* gamma,
                           double* per_doc, cudaStream_t s);
// topics.cu: the n (<= 32) most probable words of every topic of lambda (K x V, fp64), ordered by value descending, then
// word id ascending.  The candidate pass cuts the words into top_words_chunks(K, V, n) chunks and writes every chunk's
// best n of every topic to cand_v / cand_id (chunks x K x n); the merge pass writes topic k's list to ids + k*n and
// lambda_kw / rows_k to prob + k*n.  The candidate pass serves any K x V column-major matrix: its leading dimension ld
// may exceed K, and its column ids start at id0 (id0 + V <= INT_MAX).
int top_words_chunks(int K, int V, int n);
void launch_top_words_candidates(const double* lambda, int K, int ld, int V, int id0, int n, int chunks, double* cand_v,
                                 int32_t* cand_id, cudaStream_t s);
void launch_top_words_merge(const double* cand_v, const int32_t* cand_id, const double* rows, int K, int n, int chunks,
                            int32_t* ids, double* prob, cudaStream_t s);
// the same merge into a running list: starts from init_v / init_id (K x n, may be null; may equal v / ids) and writes the
// merged values (hellinger: sqrt(max(0, 1 - value))) to v and their ids to ids
void launch_top_n_merge(const double* cand_v, const int32_t* cand_id, int K, int n, int chunks, const double* init_v,
                        const int32_t* init_id, bool hellinger, int32_t* ids, double* v, cudaStream_t s);
// counts[(k n + j) n + i] += number of documents of `docs` (CSR arrays only) holding both the words of ranks i and j of topic
// k's list (a pair counts when its count is > 0).  map_ptr (V + 1) / map_entry: for word w, the entries topic * 32 + rank
// of the lists it is on, at map_entry[map_ptr[w] .. map_ptr[w + 1])
void launch_cooccurrence(const DeviceDocs& docs, int K, int n, const int32_t* map_ptr, const int32_t* map_entry,
                         unsigned long long* counts, cudaStream_t s);
// topics.cu: distances between the topics of two lambdas (K_A x V and K_B x V, fp64) through C = f(P_A) g(P_B)^T,
// p_kw = lambda_kw / rows_k.  The words are cut into chunks of plan.chunk; per chunk the prepare pass writes f(P_A) and
// g(P_B) word-major (words x ld, topics padded with zeros) and the product pass adds the chunk to plan.splits partials of C
// (ld_x x ld_y each); the finish pass sums the partials in order and applies the metric's epilogue.
enum { DIST_OP_NONE = 0, DIST_OP_SQRT = 1, DIST_OP_IDENTITY = 2, DIST_OP_LOG = 3 };
enum { DIST_BAD_NEGATIVE = 1, DIST_BAD_ZERO = 2, DIST_BAD_EMPTY_ROW = 4 };   // bits of the prepare pass's flag
struct DistancePlan {
	int ld_x, ld_y;   // K_A and K_B rounded up to the product's tile
	int splits;       // partials of C: the words of a chunk are split into this many equal runs, one per CTA layer
	int chunk;        // words per chunk, a multiple of splits * the product's stage depth
};
// one_operand: X and Y are the same scratch (a self-comparison under Hellinger)
DistancePlan distance_plan(int KA, int KB, int V, bool one_operand);
int distance_chunk_words(const DistancePlan& plan, int remaining);   // rows of a chunk with `remaining` words left
int distance_entropy_parts(int words);                               // entropy partials the prepare pass writes per chunk
// x[r ld + k] = op_x(p_k,w0+r) for r < words (0 beyond V or K); y likewise when not null.  entropy_part (may be null):
// per part of the chunk, sum_w p log p of every topic.  flag |= DIST_BAD_* for negative entries, zeros under DIST_OP_LOG,
// and topics whose row sum is not positive
void launch_distance_prepare(const double* lambda, int K, int V, int ld, int w0, int words, const double* rows, int op_x,
                             double* x, int op_y, double* y, double* entropy_part, int* flag, cudaStream_t s);
// entropy[k] = (first ? 0 : entropy[k]) + the chunk's parts, in order
void launch_distance_entropy(const double* entropy_part, int parts, int K, int ld, bool first, double* entropy, cudaStream_t s);
// partial[s] (ld_x x ld_y, column-major) = (first ? 0 : partial[s]) + X_s^T Y_s over split s of the chunk's words
void launch_distance_product(const DistancePlan& plan, const double* x, const double* y, int words, bool first,
                             double* partial, cudaStream_t s);
// the same for the first cols_y (a multiple of 128) columns of a Y whose rows are ld_y apart; partial[s] is ld_x x cols_y
void launch_distance_product(const double* x, int ld_x, const double* y, int64_t ld_y, int cols_y, int splits, int words, bool first,
                             double* partial, cudaStream_t s);
// out[j KA + i] = sqrt(max(0, 1 - C_ij)) (metric 0) or max(0, entropy_i - C_ij) (metric 1), C = sum of the partials
void launch_distance_finish(const DistancePlan& plan, const double* partial, int KA, int KB, int metric, const double* entropy,
                            double* out, cudaStream_t s);
// topics.cu: the n (<= 32) most probable topics of every pair under phi_jk = softmax_k(psi(gamma_dk) + psi(lambda_kw) -
// psi_rows_k), fp64.  The words are taken in chunks of word_topics_chunk_words(K) ids.  The table pass writes
// table[(w - w0) K + k] = psi(lambda_kw) - psi_rows_k for the words w in [w0, w0 + count) that have pairs (word_ptr).  The
// pair pass takes the pairs of the words [w0, w1) from the word-sorted token list of `docs` (word_ptr, tok_doc, tok_src,
// word_ids); psi_gamma is K x B.  Pair j's topics go to topics + j*n (ranked by descending score, equal scores by the smaller
// topic), their phi to probs (may be null).
int word_topics_chunk_words(int K);
void launch_word_topics_table(const double* lambda, int K, int w0, int count, const int32_t* word_ptr, const double* psi_rows,
                              double* table, cudaStream_t s);
void launch_word_topics_pairs(const DeviceDocs& docs, int w0, int w1, const double* table, const double* psi_gamma, int K, int n,
                              int32_t* topics, double* probs, cudaStream_t s);
// topics.cu: similar documents.  Operands are sqrt(theta), theta = gamma / column sum, topic-major: element (k, c) at
// k * ld + c, with similar_rows(K) rows (zero beyond K) and ld = similar_ld(columns) (the product's tile; zero beyond).
int similar_rows(int K);
int64_t similar_ld(int64_t cols);
// out[k * ld + c] = sqrt(gamma_kc / sum_k gamma_kc) for k < K, c < cols (gamma K x cols column-major; the padding is left as
// it is); *flag |= 1 for a negative or non-finite entry, or a column whose sum is not positive and finite
void launch_similar_prepare(const double* gamma, int K, int cols, int64_t ld, double* out, int* flag, cudaStream_t s);
// aff[d * lda + q] = sum_{k < K} query[k * ldq + q] * index[k * ld + d] for q < nq, d < docs, as one fma chain in k order
void launch_similar_stream(const double* index, int64_t ld, int K, int docs, const double* query, int ldq, int nq, double* aff,
                           int lda, cudaStream_t s);
// out[k] = lgamma(in[k])
void launch_lgamma_vector(const double* in, int K, double* out, cudaStream_t s);

// special-function test hook
void launch_special(int which, const double* x, int64_t n, double* out, cudaStream_t s);

}  // namespace trlda
