// model.cu — host side of the C ABI (include/trlda_b200.h): model state in HBM, the three updateParameters
// drivers, minibatch upload, multi-GPU exchange and instrumentation.  Everything numerical runs in the kernels
// of kernels.cu; the host only sequences launches and does the K-vector / scalar Newton steps of the
// empirical-Bayes updates.  Reference citations are relative to /root/reference/code/trlda/.
#include "../../include/trlda_b200.h"
#include "kernels.cuh"
#include "special.cuh"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

using namespace trlda;

// ------------------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_error;
std::mutex g_seed_mutex;
uint64_t g_seed = 0x5DEECE66DULL;
uint64_t g_stream_counter = 0;

uint64_t next_stream_id() {
	std::lock_guard<std::mutex> lock(g_seed_mutex);
	return ++g_stream_counter;
}

uint64_t current_seed() {
	std::lock_guard<std::mutex> lock(g_seed_mutex);
	return g_seed;
}

// device (cudaMalloc) or page-locked host (cudaHostAlloc) memory that grows on demand and is freed by its owner;
// move-only, so that two owners of one allocation cannot exist
template <bool Pinned> struct Buf {
	void* p = nullptr;
	size_t cap = 0;

	Buf() = default;
	Buf(const Buf&) = delete;
	Buf& operator=(const Buf&) = delete;
	Buf(Buf&& o) noexcept { *this = std::move(o); }
	Buf& operator=(Buf&& o) noexcept {
		if(this != &o) {
			release();
			p = std::exchange(o.p, nullptr);
			cap = std::exchange(o.cap, 0);
		}
		return *this;
	}
	~Buf() { release(); }

	cudaError_t ensure(size_t bytes) {
		if(bytes <= cap)
			return cudaSuccess;
		release();
		// grow geometrically; device buffers from 64 MB up (the big K x V ones) are allocated exactly
		const size_t want = Pinned || bytes < (64u << 20) ? bytes + bytes / 4 + 256 : bytes;
		const cudaError_t e = Pinned ? cudaHostAlloc(&p, want, cudaHostAllocDefault) : cudaMalloc(&p, want);
		if(e == cudaSuccess)
			cap = want;
		else
			p = nullptr;
		return e;
	}
	void release() {
		if(p) {
			if(Pinned)
				cudaFreeHost(p);
			else
				cudaFree(p);
		}
		p = nullptr;
		cap = 0;
	}
	template <typename T> T* as() const { return static_cast<T*>(p); }
};
using DevBuf = Buf<false>;
using PinnedBuf = Buf<true>;

// ---- NCCL through dlopen: no link-time dependency, only needed once trlda_comm_init is called -------------------
struct NcclApi {
	void* handle = nullptr;
	ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
	ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*GroupStart)() = nullptr;
	ncclResult_t (*GroupEnd)() = nullptr;
	const char* (*GetErrorString)(ncclResult_t) = nullptr;
	bool ok = false;
};

NcclApi& nccl_api() {
	static NcclApi api;
	static std::once_flag once;
	std::call_once(once, [] {
		const char* names[] = {"libnccl.so.2", "libnccl.so"};
		for(const char* name : names) {
			api.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
			if(api.handle)
				break;
		}
		if(!api.handle)
			return;
		api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.handle, "ncclGetUniqueId"));
		api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.handle, "ncclCommInitRank"));
		api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.handle, "ncclCommDestroy"));
		api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.handle, "ncclAllReduce"));
		api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.handle, "ncclGetErrorString"));
		api.AllGather = reinterpret_cast<decltype(api.AllGather)>(dlsym(api.handle, "ncclAllGather"));
		api.Broadcast = reinterpret_cast<decltype(api.Broadcast)>(dlsym(api.handle, "ncclBroadcast"));
		api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(dlsym(api.handle, "ncclGroupStart"));
		api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(dlsym(api.handle, "ncclGroupEnd"));
		api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.AllGather && api.GetErrorString &&
		         api.Broadcast && api.GroupStart && api.GroupEnd;
	});
	return api;
}

// ---- host special functions for the Newton steps ----------------------------------------------------------------

// Hurwitz zeta(s, q) for s > 1, q > 0 by Euler–Maclaurin summation (what zeta.cpp:67-134 computes): direct
// terms up to a = q + N, then the integral, half-term and Bernoulli corrections.
double hurwitz_zeta(double s, double q) {
	if(!(s > 1.0) || !(q > 0.0))
		return NAN;
	static const double B2k[] = {1.0 / 6, -1.0 / 30, 1.0 / 42, -1.0 / 30, 5.0 / 66, -691.0 / 2730, 7.0 / 6,
	                             -3617.0 / 510, 43867.0 / 798, -174611.0 / 330};
	if(q > 1e8)
		return (1.0 / (s - 1.0) + 1.0 / (2.0 * q)) * pow(q, 1.0 - s);     // leading asymptotic terms, as zeta.cpp:98-100
	double sum = 0.0, a = q;
	for(int i = 0; i < 10 || a < 12.0; ++i) {
		sum += pow(a, -s);
		a += 1.0;
	}
	sum += pow(a, 1.0 - s) / (s - 1.0) + 0.5 * pow(a, -s);
	double fact = 1.0, poch = s, apow = pow(a, -s - 1.0);   // s (s+1) ... / (2k)! * a^(-s-2k+1)
	for(int k = 0; k < 10; ++k) {
		fact *= (2.0 * k + 1.0) * (2.0 * k + 2.0);
		const double term = B2k[k] * poch / fact * apow;
		sum += term;
		if(fabs(term) < 1e-17 * fabs(sum))
			break;
		poch *= (s + 2.0 * k + 1.0) * (s + 2.0 * k + 2.0);
		apow /= a * a;
	}
	return sum;
}

double host_polygamma(int n, double x) {
	if(n < 1)
		return digamma(x);
	if(n == 1 && x > 0.0)
		return trigamma(x);
	return pow(-1.0, n + 1) * tgamma(n + 1.0) * hurwitz_zeta(n + 1.0, x);   // utils.cpp:107-111
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------
// the model
// ------------------------------------------------------------------------------------------------------------
struct trlda_model {
	int kind = 0, K = 0, V = 0, device = 0, precision = TRLDA_PRECISION_FP64;
	int64_t num_documents = 0, update_count = 0;
	double eta = .3;
	std::vector<double> alpha;

	// adaptive learning rate (onlinelda.h:41-44)
	double ada_rho = 1. / 1000., ada_tau = 1000., ada_sq_norm = 1.;
	DevBuf ada_gradient;
	// cumulative alpha statistics (cumulativelda.h:24-25)
	std::vector<double> psi_gamma_diff;
	int64_t cum_num_documents = 0;

	cudaStream_t stream = nullptr;
	int smem_optin = 0, num_sms = 0;

	// K x V state: lambda lives in lam[cur]; the other buffer receives the next lambda (lambda' = old buffer)
	DevBuf lam[2];
	int cur = 0;
	DevBuf beta;            // expElogbeta, element size beta_elem
	int beta_elem = 8;
	bool beta_valid = false;
	DevBuf sstats;
	DevBuf rows, rows_prev, rows_stat, psi_rows, d_alpha, partials, vpartials, scalars;

	// documents sorted by length (descending) and cut into buckets; each bucket is one E-step launch whose
	// shared-memory tile is sized for the bucket's longest document
	struct Bucket { int64_t offset, count; int n_max; };
	// Multi-GPU "gather" exchange (default for the mixed mode): every rank holds the token list of the WHOLE minibatch,
	// sorted by word and restricted to the words it owns; per trust-region iteration the ranks all-gather etheta and the
	// token weights (43 MB at cfg-3), every rank scatters + blends + prepares beta for ITS word range with the single-GPU
	// kernel, and the ranks all-gather the new beta.  No K x V partial statistics cross NVLink.
	struct GlobalDocs {
		bool ready = false;
		std::vector<int64_t> shard_B, shard_N, doc_off, tok_off;      // per rank: documents, pairs, and where they start
		std::vector<int64_t> pad_B, pad_N;                             // segment sizes (padded to the largest shard)
		int64_t B = 0, N = 0;
		DevBuf len, ids, word_ptr, tok_doc, tok_src, etheta32, weight, scratch;
		DeviceDocs view;                                               // word_ptr / tok_doc / tok_src of the global batch
	};
	// one uploaded minibatch: the resident one is `mb`, parked ones (trlda_upload_docs_slot / trlda_select_docs) sit in
	// `slots` and are exchanged with it whole
	struct Minibatch {
		DeviceDocs docs;
		DevBuf b_doc_ptr, b_word_ids, b_counts, b_word_ptr, b_tok_doc, b_tok_src, b_order;
		std::vector<Bucket> buckets;
		std::vector<int> sorted_len;    // length of every document in the length-sorted order
		// documents longer than 192 / 160 / 128 / 64 pairs (prefix lengths of the length-sorted order): the cuts between
		// the tile shapes of the tensor-memory E-step kernel
		int64_t len_gt[4] = {0, 0, 0, 0};
		GlobalDocs gdocs;
		int64_t docs_total_count = 0;    // sum of all counts in the (global) minibatch
		int64_t global_B = 0;            // documents over all ranks
	};
	Minibatch mb;
	struct Slot {
		bool used = false;
		Minibatch mb;
	};
	std::vector<Slot> slots;
	int live_slot = -1;
	bool use_gather = true;                    // TRLDA_MULTI_GPU=gather (default) | peer | allreduce
	// the word-sorted token list of the resident minibatch is built lazily (ensure_csc)
	bool csc_pending = false;
	int csc_threads = 1;
	size_t stage_off[5] = {0, 0, 0, 0, 0};
	// the length buckets of one E-step run concurrently on these streams (fork/join around the main stream), so
	// that CTAs of buckets with different shared-memory footprints can share an SM and the buckets' tails overlap
	static const int kAuxStreams = 3;
	cudaStream_t aux[kAuxStreams] = {nullptr, nullptr, nullptr};
	cudaEvent_t fork_event = nullptr, join_event[kAuxStreams] = {nullptr, nullptr, nullptr};
	// documents too long for the shared-memory plan of k_estep run on their own stream, beside the other E-step kernels,
	// with their per-pair vectors in long_scratch
	cudaStream_t long_stream = nullptr;
	cudaEvent_t long_join = nullptr;
	DevBuf long_scratch;
	bool tmem_mode = true;       // TRLDA_ESTEP_TMEM=0: never use the tensor-memory-resident kernel (mixed mode)
	bool stream_ran = false;     // the streaming E-step kernel has run (its phase timers are printed by trlda_destroy)
	DevBuf sweeps;   // device counter behind trlda_stats.estep_sweeps
	// trlda_sample: row-wise CDFs of beta ~ Dirichlet(lambda), padded token buffers, and the host copy handed to the caller
	DevBuf sample_cdf, sample_tokens, sample_counts, sample_lengths;
	std::vector<int64_t> sample_ptr;
	std::vector<int32_t> sample_ids, sample_cts;
	DevBuf ticks;    // debug phase timers of the E-step kernels (TRLDA_ESTEP_TICKS=1)
	PinnedBuf staging, readback;
	bool docs_resident = false;

	// per-minibatch E-step buffers
	DevBuf gamma, etheta, etheta32, weight, doc_stat, iterations, wordcount;
	DevBuf gibbs_occ, gibbs_topics;            // Gibbs E-step scratch: occurrences before each document, one topic per occurrence
	// side CSR of the evaluation calls (the held-out part of trlda_predictive_log_likelihood, the corpus of
	// trlda_cooccurrence): it never replaces the live minibatch
	DevBuf ho_doc_ptr, ho_word_ids, ho_counts;
	// trlda_top_words: row sums of lambda, the per-chunk candidate lists and the result; trlda_cooccurrence: the inverse map
	// of the top words and the counters
	DevBuf topic_rows, top_cand_v, top_cand_id, top_ids, top_prob, co_map_ptr, co_map, co_counts;
	// trlda_topic_distances: row sums of the other model's lambda, the prepared operands of one chunk of words, the entropy
	// partials and entropies, the split partials of the product, the result and the prepare pass's flag; other_ready orders
	// this model's stream after the other model's work
	DevBuf dist_rows, dist_x, dist_y, dist_hpart, dist_h, dist_partial, dist_out, dist_flag;
	cudaEvent_t other_ready = nullptr;
	// trlda_word_topics: the call's document lengths, the scratch and the result of its word-sorted token list, the log-beta
	// table of one chunk of words, psi(gamma) and the results
	DevBuf wt_len, wt_scratch, wt_word_ptr, wt_tok_doc, wt_tok_src, wt_table, wt_psi_gamma, wt_topics, wt_probs;
	// trlda_index_documents: the document index (sqrt(theta) of sim_docs documents, similar_rows(K) x sim_ld, topic-major);
	// trlda_similar_documents: a block of queries prepared the same way, one affinity block, the candidate lists of its
	// chunks and of their first merge, the running lists of all queries and the prepare pass's flag
	DevBuf sim_index, sim_query, sim_aff, sim_cand_v, sim_cand_id, sim_merge_v, sim_merge_id, sim_res_v, sim_res_id, sim_flag;
	int64_t sim_docs = 0, sim_ld = 0;
	bool gamma_valid = false;

	// parity seams
	std::vector<double> inj_gamma;
	int64_t inj_gamma_cols = -1;
	std::vector<double> inj_lambda;

	// multi-GPU
	ncclComm_t comm = nullptr;
	int rank = 0, nranks = 1;
	// peer-mapped replicas (cudaIpc) for the fused reduce-scatter + M-step + all-gather kernel: [rank] pointers to
	// every rank's sstats, beta and the two lambda buffers; peer_ready once the handles have been exchanged
	DevBuf sstats32;                           // receive buffer of the peer exchange: partial columns pushed by all ranks
	int peer_sstats_elem = 8, peer_shard_cap = 0;
	bool lambda_sharded = false;               // debug: the last M-step left lambda complete only on the owners' shards
	bool peer_ready = false;
	bool use_peer = true;                      // TRLDA_MULTI_GPU=allreduce selects the plain NCCL all-reduce path
	void* peer_sstats[TRLDA_MAX_RANKS] = {};
	void* peer_beta[TRLDA_MAX_RANKS] = {};
	void* peer_lam[2][TRLDA_MAX_RANKS] = {};
	std::vector<void*> peer_opened;

	// instrumentation
	bool profiling = false;
	struct Span { int kind; cudaEvent_t a, b; };
	std::vector<Span> spans;
	std::vector<cudaEvent_t> event_pool;
	trlda_stats stats{};

	std::string error;
	// the reference held the GIL through every call; the binding releases it around the long ones, so calls on one
	// model from several host threads are serialised here
	std::recursive_mutex mu;

	double* lambda() { return lam[cur].as<double>(); }
	double* lambda_next() { return lam[1 - cur].as<double>(); }

	// the buffers free themselves after this body has run (trlda_destroy closes what refers to them first)
	~trlda_model() {
		for(int i = 0; i < kAuxStreams; ++i) {
			if(aux[i])
				cudaStreamDestroy(aux[i]);
			if(join_event[i])
				cudaEventDestroy(join_event[i]);
		}
		if(fork_event)
			cudaEventDestroy(fork_event);
		if(other_ready)
			cudaEventDestroy(other_ready);
		if(long_stream)
			cudaStreamDestroy(long_stream);
		if(long_join)
			cudaEventDestroy(long_join);
		if(stream)
			cudaStreamDestroy(stream);
	}
};

namespace {

int fail(trlda_model* m, int code, const std::string& msg) {
	if(m)
		m->error = msg;
	g_error = msg;
	return code;
}

#define CUDA_TRY(m, expr)                                                                              \
	do {                                                                                               \
		cudaError_t e__ = (expr);                                                                      \
		if(e__ != cudaSuccess)                                                                         \
			return fail(m, TRLDA_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #expr); \
	} while(0)

#define TRY(expr)                  \
	do {                           \
		int s__ = (expr);          \
		if(s__ != TRLDA_OK)        \
			return s__;            \
	} while(0)

#define NCCL_TRY(m, expr)                                                                                   \
	do {                                                                                                    \
		ncclResult_t r__ = (expr);                                                                          \
		if(r__ != ncclSuccess)                                                                              \
			return fail(m, TRLDA_ERR_CUDA, std::string("NCCL error: ") + nccl_api().GetErrorString(r__));  \
	} while(0)

// brackets one kernel launch for the timing table
struct Launch {
	trlda_model* m;
	int kind;
	cudaEvent_t a = nullptr, b = nullptr;
	Launch(trlda_model* m_, int kind_) : m(m_), kind(kind_) {
		nvtxRangePushA(trlda_kernel_kind_name(kind));      // NVTX range per kernel kind (beta_prep, estep, scatter_mstep, ...)
		m->stats.launches[kind]++;
		m->stats.total_launches++;
		if(m->profiling) {
			a = take();
			b = take();
			cudaEventRecord(a, m->stream);
		}
	}
	~Launch() {
		nvtxRangePop();
		if(m->profiling) {
			cudaEventRecord(b, m->stream);
			m->spans.push_back({kind, a, b});
		}
	}
	cudaEvent_t take() {
		if(!m->event_pool.empty()) {
			cudaEvent_t e = m->event_pool.back();
			m->event_pool.pop_back();
			return e;
		}
		cudaEvent_t e;
		cudaEventCreate(&e);
		return e;
	}
};

int check_launch(trlda_model* m, const char* what) {
	cudaError_t e = cudaGetLastError();
	if(e != cudaSuccess)
		return fail(m, TRLDA_ERR_CUDA, std::string("CUDA launch failed (") + what + "): " + cudaGetErrorString(e));
	return TRLDA_OK;
}

int set_device(trlda_model* m) {
	CUDA_TRY(m, cudaSetDevice(m->device));
	return TRLDA_OK;
}

size_t kv_bytes(const trlda_model* m) { return (size_t) m->K * m->V * sizeof(double); }

int ensure_beta(trlda_model* m) {
	const int elem = m->precision == TRLDA_PRECISION_MIXED ? 4 : 8;
	if(elem != m->beta_elem) {
		m->beta_elem = elem;
		m->beta_valid = false;
	}
	// the streaming E-step reads whole 16-byte-vector rounds of a column (up to K rounded up to 32 vectors): the tail of
	// the last column needs readable, finite bytes behind it
	const size_t bytes = (size_t) m->K * m->V * elem, slack = 16384;
	if(bytes + slack > m->beta.cap) {
		CUDA_TRY(m, m->beta.ensure(bytes + slack));
		CUDA_TRY(m, cudaMemsetAsync(static_cast<char*>(m->beta.p) + bytes, 0, m->beta.cap - bytes, m->stream));
		m->beta_valid = false;
	}
	return TRLDA_OK;
}

int upload_alpha(trlda_model* m) {
	CUDA_TRY(m, m->d_alpha.ensure(sizeof(double) * m->K));
	CUDA_TRY(m, cudaMemcpyAsync(m->d_alpha.p, m->alpha.data(), sizeof(double) * m->K, cudaMemcpyHostToDevice, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));   // alpha.data() may be reallocated by the caller later
	m->stats.h2d_bytes += sizeof(double) * m->K;
	return TRLDA_OK;
}

// sum over ranks, in place, on the model's stream
int allreduce(trlda_model* m, void* buf, size_t count, ncclDataType_t type) {
	if(m->nranks <= 1)
		return TRLDA_OK;
	NCCL_TRY(m, nccl_api().AllReduce(buf, buf, count, type, ncclSum, m->comm, m->stream));
	return TRLDA_OK;
}

// rows = row sums of `matrix` (K x V; K = m->K unless given, as for the other model's lambda in trlda_topic_distances)
int compute_rows(trlda_model* m, const double* matrix, double* out, int K = 0) {
	if(K <= 0)
		K = m->K;
	int P = rowsum_num_partials(m->V);
	CUDA_TRY(m, m->partials.ensure(sizeof(double) * (size_t) std::max(P, colsum_num_partials(std::max<int64_t>(m->mb.docs.B, 1))) *
	                               std::max(K, m->K)));
	{
		Launch l(m, KK_ROWSUM);
		launch_rowsum(matrix, K, m->V, m->partials.as<double>(), &P, m->stream);
	}
	{
		Launch l(m, KK_REDUCE);
		launch_reduce_partials(m->partials.as<double>(), P, K, out, m->stream);
	}
	return check_launch(m, "rowsum");
}

int ensure_small(trlda_model* m) {
	CUDA_TRY(m, m->rows.ensure(sizeof(double) * m->K));
	CUDA_TRY(m, m->rows_prev.ensure(sizeof(double) * m->K));
	CUDA_TRY(m, m->rows_stat.ensure(sizeof(double) * m->K));
	CUDA_TRY(m, m->psi_rows.ensure(sizeof(double) * m->K));
	CUDA_TRY(m, m->vpartials.ensure(sizeof(double) * std::max(m->V, 2048)));
	CUDA_TRY(m, m->scalars.ensure(sizeof(double) * 4096));
	CUDA_TRY(m, m->readback.ensure(sizeof(double) * (size_t) std::max(m->K, 4096)));
	return TRLDA_OK;
}

// beta = exp(psi(lambda) - psi(rowsum lambda)) for the CURRENT lambda (lda.cpp:172-173)
int prepare_beta(trlda_model* m, bool want_psi_partials = false) {
	TRY(ensure_beta(m));
	TRY(ensure_small(m));
	if(m->beta_valid && !want_psi_partials)
		return TRLDA_OK;
	TRY(compute_rows(m, m->lambda(), m->rows.as<double>()));
	{
		Launch l(m, KK_MISC);
		launch_psi_vector(m->rows.as<double>(), m->K, m->psi_rows.as<double>(), m->stream);
	}
	{
		Launch l(m, KK_BETA_PREP);
		launch_beta_prep(m->lambda(), m->psi_rows.as<double>(), m->K, m->V, m->beta.p, m->beta_elem,
		                 want_psi_partials ? m->vpartials.as<double>() : nullptr, m->stream);
	}
	m->beta_valid = true;
	return check_launch(m, "beta_prep");
}

int build_global_docs(trlda_model* m, int64_t B, int64_t N);

// cuts the length-sorted documents [begin, B) into length buckets, each one launch of k_estep whose shared-memory tile
// is sized for the bucket's longest document
void form_buckets(const std::vector<int>& len, int64_t begin, std::vector<trlda_model::Bucket>& buckets) {
	auto cap_of = [](int n) {
		int cap = 32;
		while(cap < n)
			cap += cap < 256 ? 32 : (cap < 512 ? 64 : cap / 4);
		return cap;
	};
	const int64_t B = (int64_t) len.size();
	const int64_t min_bucket = 128;
	buckets.clear();
	for(int64_t i = begin; i < B;) {
		const int cap = cap_of(len[i]);
		int64_t j = i;
		while(j < B && (cap_of(len[j]) == cap || j - i < min_bucket))
			++j;
		if(B - j < min_bucket)
			j = B;
		buckets.push_back({i, j - i, len[i]});
		i = j;
	}
}

// ---- minibatch upload: CSR + word-sorted token list ---------------------------------------------------------------
int upload_docs(trlda_model* m, const trlda_docs* docs) {
	TRY(set_device(m));
	// the live buffers may belong to a parked minibatch (trlda_select_docs): hand them back before overwriting
	if(m->live_slot >= 0) {
		std::swap(m->mb, m->slots[m->live_slot].mb);
		m->live_slot = -1;
	}
	trlda_model::Minibatch& mb = m->mb;
	if(!docs || docs->num_docs < 0 || (docs->num_docs > 0 && !docs->doc_ptr))
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");
	const int64_t B = docs->num_docs;
	const int64_t N = B ? docs->doc_ptr[B] : 0;
	const int V = m->V;
	if(B && docs->doc_ptr[0] != 0)
		return fail(m, TRLDA_ERR_ARG, "Document offsets must start at zero.");
	if(N < 0 || N > INT32_MAX)
		return fail(m, TRLDA_ERR_ARG, "Too many (word, count) pairs in one minibatch.");
	if(N > 0 && (!docs->word_ids || !docs->counts))
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");

	const bool host_timing = getenv("TRLDA_HOST_TIMING") != nullptr;
	auto clock_now = [] { return std::chrono::steady_clock::now(); };
	auto ms_since = [](std::chrono::steady_clock::time_point t0) {
		return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
	};
	const auto t_begin = clock_now();
	// pinned staging: [doc_ptr | word_ids | counts | word_ptr | tok_doc | tok_src]
	const size_t o_ptr = 0;
	const size_t o_ids = o_ptr + sizeof(int64_t) * (B + 1);
	const size_t o_cts = o_ids + sizeof(int32_t) * N;
	const size_t o_wptr = o_cts + sizeof(int32_t) * N;
	const size_t o_tdoc = o_wptr + sizeof(int32_t) * ((size_t) V + 1);
	const size_t o_tsrc = o_tdoc + sizeof(int32_t) * N;
	const size_t o_order = o_tsrc + sizeof(int32_t) * N;
	const size_t total = o_order + sizeof(int32_t) * std::max<int64_t>(B, 1);
	CUDA_TRY(m, m->staging.ensure(total));
	char* base = m->staging.as<char>();
	int64_t* s_ptr = reinterpret_cast<int64_t*>(base + o_ptr);
	int32_t* s_ids = reinterpret_cast<int32_t*>(base + o_ids);
	int32_t* s_cts = reinterpret_cast<int32_t*>(base + o_cts);
	int32_t* s_wptr = reinterpret_cast<int32_t*>(base + o_wptr);
	int32_t* s_tdoc = reinterpret_cast<int32_t*>(base + o_tdoc);
	int32_t* s_tsrc = reinterpret_cast<int32_t*>(base + o_tsrc);
	int32_t* s_order = reinterpret_cast<int32_t*>(base + o_order);

	// make sure the previous use of the staging buffer has been consumed
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	const double t_sync = ms_since(t_begin);

	if(B)
		memcpy(s_ptr, docs->doc_ptr, sizeof(int64_t) * (B + 1));
	else
		s_ptr[0] = 0;
	int n_max = 0;
	int64_t total_count = 0;
	int64_t len_gt[4] = {0, 0, 0, 0};
	for(int64_t d = 0; d < B; ++d) {
		const int64_t n = s_ptr[d + 1] - s_ptr[d];
		if(n < 0)
			return fail(m, TRLDA_ERR_ARG, "Document offsets must be non-decreasing.");
		n_max = std::max<int64_t>(n_max, n);
		len_gt[0] += n > 192;
		len_gt[1] += n > 160;
		len_gt[2] += n > 128;
		len_gt[3] += n > 64;
	}
	for(int i = 0; i < 4; ++i)
		mb.len_gt[i] = len_gt[i];
	// copy the id / count arrays into the pinned staging buffer (parallel slices), summing the counts and checking
	// the id range on the way.  The word-sorted token list is built later, by ensure_csc(), right before the
	// first kernel that needs it — by then the device is busy with the first E-step and the host work is hidden.
	const int T = (int) std::max(1u, std::min(8u, std::min(std::thread::hardware_concurrency(), (unsigned) (N / 65536 + 1))));
	{
		std::vector<int64_t> counts_sum(T, 0);
		std::vector<int> bad(T, 0);
		const int32_t* ids = docs->word_ids;
		const int32_t* cts = docs->counts;
		auto body = [&](int t) {
			const int64_t c0 = N * t / T, c1 = N * (t + 1) / T;
			if(c1 <= c0)
				return;
			memcpy(s_ids + c0, ids + c0, sizeof(int32_t) * (c1 - c0));
			memcpy(s_cts + c0, cts + c0, sizeof(int32_t) * (c1 - c0));
			int64_t csum = 0;
			int oob = 0;
			for(int64_t i = c0; i < c1; ++i) {
				csum += cts[i];
				oob |= (ids[i] < 0) | (ids[i] >= V) | ((cts[i] < 0) << 1);
			}
			counts_sum[t] = csum;
			bad[t] = oob;
		};
		std::vector<std::thread> pool;
		for(int t = 1; t < T; ++t)
			pool.emplace_back(body, t);
		body(0);
		for(auto& th : pool)
			th.join();
		for(int t = 0; t < T; ++t) {
			total_count += counts_sum[t];
			if(bad[t] & 2)
				return fail(m, TRLDA_ERR_ARG, "Word counts should not be negative.");
			if(bad[t])
				return fail(m, TRLDA_ERR_ARG, "Word ID out of range.");
		}
	}
	m->csc_pending = true;
	m->csc_threads = T;

	// length buckets for the E-step: counting sort by length, longest first
	mb.buckets.clear();
	mb.sorted_len.resize(B);
	if(B) {
		std::vector<int32_t> start(n_max + 2, 0);
		for(int64_t d = 0; d < B; ++d)
			start[n_max - (int) (s_ptr[d + 1] - s_ptr[d]) + 1]++;
		for(int i = 0; i <= n_max; ++i)
			start[i + 1] += start[i];
		for(int64_t d = 0; d < B; ++d)
			s_order[start[n_max - (int) (s_ptr[d + 1] - s_ptr[d])]++] = (int32_t) d;
		for(int64_t i = 0; i < B; ++i) {
			const int32_t d = s_order[i];
			mb.sorted_len[i] = (int) (s_ptr[d + 1] - s_ptr[d]);
		}
		form_buckets(mb.sorted_len, 0, mb.buckets);
	}

	const double t_host = ms_since(t_begin);
	CUDA_TRY(m, mb.b_order.ensure(sizeof(int32_t) * std::max<int64_t>(B, 1)));
	CUDA_TRY(m, mb.b_doc_ptr.ensure(sizeof(int64_t) * (B + 1)));
	CUDA_TRY(m, mb.b_word_ids.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, mb.b_counts.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, mb.b_word_ptr.ensure(sizeof(int32_t) * ((size_t) V + 1)));
	CUDA_TRY(m, mb.b_tok_doc.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, mb.b_tok_src.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, cudaMemcpyAsync(mb.b_doc_ptr.p, s_ptr, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, m->stream));
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(mb.b_word_ids.p, s_ids, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
		CUDA_TRY(m, cudaMemcpyAsync(mb.b_counts.p, s_cts, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
	}
	(void) s_wptr; (void) s_tdoc; (void) s_tsrc;
	m->stage_off[0] = o_ptr; m->stage_off[1] = o_ids; m->stage_off[2] = o_wptr; m->stage_off[3] = o_tdoc; m->stage_off[4] = o_tsrc;
	if(B)
		CUDA_TRY(m, cudaMemcpyAsync(mb.b_order.p, s_order, sizeof(int32_t) * B, cudaMemcpyHostToDevice, m->stream));
	m->stats.h2d_bytes += total;

	mb.docs.B = B;
	mb.docs.N = N;
	mb.docs.n_max = n_max;
	mb.docs.doc_ptr = mb.b_doc_ptr.as<int64_t>();
	mb.docs.word_ids = mb.b_word_ids.as<int32_t>();
	mb.docs.counts = mb.b_counts.as<int32_t>();
	mb.docs.word_ptr = mb.b_word_ptr.as<int32_t>();
	mb.docs.tok_doc = mb.b_tok_doc.as<int32_t>();
	mb.docs.tok_src = mb.b_tok_src.as<int32_t>();
	mb.docs_total_count = total_count;
	mb.global_B = B;
	m->gamma_valid = false;
	m->docs_resident = true;

	if(m->nranks > 1) {
		// batch-wide document count and token count
		TRY(ensure_small(m));
		int64_t* h = m->readback.as<int64_t>();
		h[0] = B;
		h[1] = total_count;
		CUDA_TRY(m, cudaMemcpyAsync(m->scalars.p, h, 2 * sizeof(int64_t), cudaMemcpyHostToDevice, m->stream));
		TRY(allreduce(m, m->scalars.p, 2, ncclInt64));
		CUDA_TRY(m, cudaMemcpyAsync(h, m->scalars.p, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, m->stream));
		CUDA_TRY(m, cudaStreamSynchronize(m->stream));
		mb.global_B = h[0];
		mb.docs_total_count = h[1];
	}

	// per-minibatch buffers
	const size_t kb = sizeof(double) * (size_t) m->K * std::max<int64_t>(B, 1);
	CUDA_TRY(m, m->gamma.ensure(kb));
	CUDA_TRY(m, m->etheta.ensure(kb));
	CUDA_TRY(m, m->etheta32.ensure(kb / 2));
	CUDA_TRY(m, m->doc_stat.ensure(kb));
	CUDA_TRY(m, m->weight.ensure(sizeof(double) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, m->iterations.ensure(sizeof(int32_t) * std::max<int64_t>(B, 1)));
	mb.gdocs.ready = false;
	if(m->nranks > 1 && m->use_gather && m->beta_elem == 4 && m->K % 4 == 0 && m->K <= 4096)
		TRY(build_global_docs(m, B, N));
	if(host_timing)
		fprintf(stderr, "[trlda] upload_docs: wait for stream %.2f ms, host packing (copy + counting sort + buckets) %.2f ms, total incl. H2D enqueue %.2f ms\n",
		        t_sync, t_host - t_sync, ms_since(t_begin));
	return TRLDA_OK;
}

// ---- multi-GPU gather exchange: the token list of the whole minibatch, word-sorted, for this rank's words --------
int word_begin(const trlda_model* m, int rank) { return (int) ((int64_t) m->V * rank / m->nranks); }

// `count` elements of `type` from every rank's segment of `buf` (segment r starts at element off[r], has n[r] elements)
int gather_segments(trlda_model* m, void* buf, const std::vector<int64_t>& off, const std::vector<int64_t>& n, size_t elem,
                    ncclDataType_t type) {
	// equal, contiguous segments: ONE bandwidth-optimal all-gather in place; else one broadcast per rank in a group
	bool regular = true;
	for(int r = 0; r < m->nranks; ++r)
		regular = regular && n[r] == n[0] && off[r] == (int64_t) r * n[0];
	if(regular) {
		if(n[0] > 0)
			NCCL_TRY(m, nccl_api().AllGather(static_cast<char*>(buf) + (size_t) off[m->rank] * elem, buf, (size_t) n[0], type, m->comm, m->stream));
		return TRLDA_OK;
	}
	NCCL_TRY(m, nccl_api().GroupStart());
	for(int r = 0; r < m->nranks; ++r)
		if(n[r] > 0) {
			char* seg = static_cast<char*>(buf) + (size_t) off[r] * elem;
			NCCL_TRY(m, nccl_api().Broadcast(seg, seg, (size_t) n[r], type, r, m->comm, m->stream));
		}
	NCCL_TRY(m, nccl_api().GroupEnd());
	return TRLDA_OK;
}

int build_global_docs(trlda_model* m, int64_t B, int64_t N) {
	trlda_model::GlobalDocs& g = m->mb.gdocs;
	g.ready = false;
	const int R = m->nranks;
	// sizes of all shards
	TRY(ensure_small(m));
	{
		int64_t* h = m->readback.as<int64_t>();
		for(int i = 0; i < 2 * R; ++i)
			h[i] = 0;
		h[2 * m->rank] = B;
		h[2 * m->rank + 1] = N;
		CUDA_TRY(m, cudaMemcpyAsync(m->scalars.p, h, 2 * R * sizeof(int64_t), cudaMemcpyHostToDevice, m->stream));
		TRY(allreduce(m, m->scalars.p, 2 * R, ncclInt64));
		CUDA_TRY(m, cudaMemcpyAsync(h, m->scalars.p, 2 * R * sizeof(int64_t), cudaMemcpyDeviceToHost, m->stream));
		CUDA_TRY(m, cudaStreamSynchronize(m->stream));
		g.shard_B.assign(R, 0); g.shard_N.assign(R, 0); g.doc_off.assign(R, 0); g.tok_off.assign(R, 0);
		g.pad_B.assign(R, 0); g.pad_N.assign(R, 0);
		int64_t max_B = 0, max_N = 0;
		for(int r = 0; r < R; ++r) {
			g.shard_B[r] = h[2 * r];
			g.shard_N[r] = h[2 * r + 1];
			max_B = std::max(max_B, g.shard_B[r]);
			max_N = std::max(max_N, g.shard_N[r]);
		}
		// every rank's segment of the global document / token index space is padded to the largest shard, so that the
		// per-iteration exchanges are plain all-gathers; the padding is never referenced by a token
		for(int r = 0; r < R; ++r) {
			g.doc_off[r] = r * max_B;
			g.tok_off[r] = r * max_N;
			g.pad_B[r] = max_B;
			g.pad_N[r] = max_N;
		}
		g.B = R * max_B;
		g.N = R * max_N;
	}
	if(g.N > INT32_MAX)
		return fail(m, TRLDA_ERR_ARG, "Too many (word, count) pairs in one minibatch.");
	CUDA_TRY(m, g.len.ensure(sizeof(int32_t) * std::max<int64_t>(g.B, 1)));
	CUDA_TRY(m, g.ids.ensure(sizeof(int32_t) * std::max<int64_t>(g.N, 1)));
	// everything on the device (csc.cu): no copy and no synchronisation after the sizes are known
	launch_doc_lengths(m->mb.b_doc_ptr.as<int64_t>(), B, g.pad_B[m->rank], g.len.as<int32_t>() + g.doc_off[m->rank], m->stream);
	if(g.pad_N[m->rank])
		CUDA_TRY(m, cudaMemsetAsync(g.ids.as<int32_t>() + g.tok_off[m->rank], 0xff, sizeof(int32_t) * g.pad_N[m->rank], m->stream));   // -1: no word
	if(N)
		CUDA_TRY(m, cudaMemcpyAsync(g.ids.as<int32_t>() + g.tok_off[m->rank], m->mb.b_word_ids.p, sizeof(int32_t) * N,
		                            cudaMemcpyDeviceToDevice, m->stream));
	TRY(gather_segments(m, g.len.p, g.doc_off, g.pad_B, sizeof(int32_t), ncclInt32));
	TRY(gather_segments(m, g.ids.p, g.tok_off, g.pad_N, sizeof(int32_t), ncclInt32));
	const int v0 = word_begin(m, m->rank), v1 = word_begin(m, m->rank + 1);
	CUDA_TRY(m, g.word_ptr.ensure(sizeof(int32_t) * ((size_t) m->V + 1)));
	CUDA_TRY(m, g.tok_doc.ensure(sizeof(int32_t) * std::max<int64_t>(g.N, 1)));
	CUDA_TRY(m, g.tok_src.ensure(sizeof(int32_t) * std::max<int64_t>(g.N, 1)));
	CUDA_TRY(m, g.scratch.ensure(sizeof(int32_t) * global_csc_scratch_ints(g.B, g.N, v0, v1)));
	CUDA_TRY(m, g.etheta32.ensure(sizeof(float) * (size_t) m->K * std::max<int64_t>(g.B, 1)));
	CUDA_TRY(m, g.weight.ensure(sizeof(double) * std::max<int64_t>(g.N, 1)));
	launch_global_csc(g.len.as<int32_t>(), g.ids.as<int32_t>(), R, g.pad_B[0], g.pad_N[0], v0, v1, m->V, g.scratch.as<int32_t>(),
	                  g.word_ptr.as<int32_t>(), g.tok_doc.as<int32_t>(), g.tok_src.as<int32_t>(), m->stream);
	TRY(check_launch(m, "word-sorted token list of the gathered minibatch"));
	g.view = DeviceDocs{};
	g.view.B = g.B;
	g.view.N = g.N;
	g.view.word_ptr = g.word_ptr.as<int32_t>();
	g.view.tok_doc = g.tok_doc.as<int32_t>();
	g.view.tok_src = g.tok_src.as<int32_t>();
	g.ready = true;
	return TRLDA_OK;
}

// where the E-step leaves exp(psi(gamma)) (float32) and the token weights: in the gather exchange straight into this
// rank's segment of the global arrays
float* estep_etheta32(trlda_model* m) {
	if(m->mb.gdocs.ready)
		return m->mb.gdocs.etheta32.as<float>() + (size_t) m->mb.gdocs.doc_off[m->rank] * m->K;
	return m->etheta32.as<float>();
}
double* estep_weight(trlda_model* m) {
	if(m->mb.gdocs.ready)
		return m->mb.gdocs.weight.as<double>() + m->mb.gdocs.tok_off[m->rank];
	return m->weight.as<double>();
}

// where the initial gamma of an E-step comes from
enum GammaSource { GAMMA_FRESH, GAMMA_KEEP, GAMMA_HOST };

// fresh gamma: injected values if the parity seam is armed, else Gamma(100, 1/100) from the device generator
int fresh_gamma(trlda_model* m) {
	const int64_t B = m->mb.docs.B;
	if(m->inj_gamma_cols >= 0) {
		if(m->inj_gamma_cols != B)
			return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");
		if(B) {
			CUDA_TRY(m, cudaMemcpyAsync(m->gamma.p, m->inj_gamma.data(), sizeof(double) * (size_t) m->K * B,
			                            cudaMemcpyHostToDevice, m->stream));
			m->stats.h2d_bytes += sizeof(double) * (size_t) m->K * B;
		}
		return TRLDA_OK;
	}
	Launch l(m, KK_RNG);
	launch_gamma_rng(m->gamma.as<double>(), (int64_t) m->K * B, current_seed(), next_stream_id(), m->stream);
	return check_launch(m, "gamma_rng");
}

// the shared-memory cluster kernel (kernels.cu) on the documents of `buckets` before `end`: one launch per length
// bucket, its tile sized for the bucket's longest document.  Bucket i runs on stream i % (1 + kAuxStreams) (0 = the main
// stream), so that CTAs of buckets with different shared-memory footprints can share an SM and the buckets' tails
// overlap; the main stream waits for all of them.
int launch_buckets(trlda_model* m, const EStepArgs& a, const std::vector<trlda_model::Bucket>& buckets, int64_t end) {
	size_t nb = 0;
	while(nb < buckets.size() && buckets[nb].offset < end)
		++nb;
	const bool fork = nb > 1 && m->aux[0] != nullptr;
	if(fork) {
		CUDA_TRY(m, cudaEventRecord(m->fork_event, m->stream));
		for(int i = 0; i < trlda_model::kAuxStreams; ++i)
			CUDA_TRY(m, cudaStreamWaitEvent(m->aux[i], m->fork_event, 0));
	}
	for(size_t i = 0; i < nb; ++i) {
		const trlda_model::Bucket& bucket = buckets[i];
		const int lane = fork ? (int) (i % (1 + trlda_model::kAuxStreams)) : 0;
		cudaStream_t stream = lane == 0 ? m->stream : m->aux[lane - 1];
		const EStepPlan plan = plan_estep(m->K, bucket.n_max, m->beta_elem, m->smem_optin);
		m->stats.total_launches++;
		launch_estep(plan, a, m->mb.docs, m->mb.b_order.as<int32_t>(), bucket.offset, std::min(bucket.count, end - bucket.offset),
		             m->beta_elem, stream);
	}
	if(fork)
		for(int i = 0; i < trlda_model::kAuxStreams; ++i) {
			CUDA_TRY(m, cudaEventRecord(m->join_event[i], m->aux[i]));
			CUDA_TRY(m, cudaStreamWaitEvent(m->stream, m->join_event[i], 0));
		}
	return TRLDA_OK;
}

int run_estep_buckets(trlda_model* m, const EStepArgs& a, int64_t end) {
	Launch span(m, KK_ESTEP);   // one timing span for the whole E-step (the bucket launches overlap)
	m->stats.total_launches--;  // the span itself is not a kernel; the launches are counted by launch_buckets
	return launch_buckets(m, a, m->mb.buckets, end);
}

// whether plan_estep keeps all per-pair vectors of a document of n pairs in shared memory
bool estep_fits(const trlda_model* m, int n) {
	const EStepPlan plan = plan_estep(m->K, n, m->beta_elem, m->smem_optin);
	return plan.n_cap >= n && plan.smem <= (size_t) m->smem_optin;
}

// E-step of a minibatch whose longest documents, order[0, n_over), fit neither the shared memory of k_estep nor that of
// the streaming kernel.  They go to the global-memory variant of k_estep on the long-document stream, beside the kernels
// of the other documents.  Those are routed as if the long documents were absent: [n_over, long_end) to the streaming
// kernel when it takes the longest of them, else to k_estep over buckets formed without the long documents, and
// [long_end, B) to the tensor-memory kernel.  One timing span covers the whole E-step.
int run_estep_with_long(trlda_model* m, const EStepArgs& a, int64_t n_over, int64_t long_end) {
	const int64_t B = m->mb.docs.B;
	const int32_t* order = m->mb.b_order.as<int32_t>();
	Launch span(m, KK_ESTEP);
	m->stats.total_launches--;  // the span itself is not a kernel
	int64_t pairs = 0;
	for(int64_t i = 0; i < n_over; ++i)
		pairs += m->mb.sorted_len[i];
	// no length limit is left to check: the plan's shared memory is the K-sized vectors (12 KB at K = 4096) plus as many
	// tile columns as fit beside them, and the scratch grows with the documents
	const EStepPlan plan = plan_estep_long(m->K, m->mb.sorted_len[0], m->beta_elem, m->smem_optin);
	CUDA_TRY(m, m->long_scratch.ensure(estep_long_scratch_bytes(plan, pairs)));
	CUDA_TRY(m, cudaEventRecord(m->fork_event, m->stream));
	CUDA_TRY(m, cudaStreamWaitEvent(m->long_stream, m->fork_event, 0));
	m->stats.total_launches++;
	launch_estep_long(plan, a, m->mb.docs, order, 0, n_over, m->long_scratch.as<double>(), pairs, m->beta_elem, m->long_stream);
	CUDA_TRY(m, cudaEventRecord(m->long_join, m->long_stream));
	if(n_over < long_end) {
		const int n_rest = m->mb.sorted_len[n_over];
		if(stream_estep_applicable(m->K, n_rest, m->beta_elem, m->smem_optin)) {
			m->stats.total_launches++;
			launch_estep_stream(a, m->mb.docs, order, n_over, long_end - n_over, n_rest, m->beta_elem, m->stream);
			m->stream_ran = true;
		} else {
			std::vector<trlda_model::Bucket> buckets;
			form_buckets(m->mb.sorted_len, n_over, buckets);
			TRY(launch_buckets(m, a, buckets, long_end));
		}
	}
	if(long_end < B) {
		m->stats.total_launches++;
		if(launch_estep_tmem(a, m->mb.docs, order, long_end, B - long_end, tmem_estep_max_len(), m->stream) != 0)
			return fail(m, TRLDA_ERR_CUDA, "The tensor-memory E-step kernel could not be launched.");
	}
	CUDA_TRY(m, cudaStreamWaitEvent(m->stream, m->long_join, 0));
	return TRLDA_OK;
}

// LDA::updateVariablesVI without the scatter: gamma fixed point for every document of the resident minibatch
int run_estep(trlda_model* m, GammaSource src, const double* host_gamma, int max_iter, double threshold) {
	if(src == GAMMA_FRESH)
		TRY(fresh_gamma(m));
	else if(src == GAMMA_HOST && m->mb.docs.B) {
		CUDA_TRY(m, cudaMemcpyAsync(m->gamma.p, host_gamma, sizeof(double) * (size_t) m->K * m->mb.docs.B,
		                            cudaMemcpyHostToDevice, m->stream));
		m->stats.h2d_bytes += sizeof(double) * (size_t) m->K * m->mb.docs.B;
	}
	EStepArgs a;
	a.K = m->K;
	a.beta = m->beta.p;
	a.alpha = m->d_alpha.as<double>();
	a.gamma = m->gamma.as<double>();
	a.etheta = m->etheta.as<double>();
	a.etheta32 = m->beta_elem == 4 ? estep_etheta32(m) : nullptr;
	a.weight = estep_weight(m);
	a.doc_stat = m->doc_stat.as<double>();
	a.iterations = m->iterations.as<int32_t>();
	a.max_iter = max_iter;
	a.threshold = threshold;
	a.ticks = m->ticks.as<unsigned long long>();
	a.sweeps = m->sweeps.as<unsigned long long>();
	a.work = reinterpret_cast<int*>(m->sweeps.as<unsigned long long>() + 1);
	m->stats.estep_calls++;
	// The documents are sorted by length, longest first.  In mixed mode the tensor-memory-resident kernel
	// (estep_tmem.cu) takes every document that fits its on-chip tile, [long_end, B); the longer ones, and in fp64 mode
	// all of them, go to the streaming kernel (estep_stream.cu), which re-reads the tile from L2 once per inner
	// iteration, or, for what it does not cover (unaligned K, K beyond its per-lane register tile, documents too long
	// for its shared memory), to the shared-memory cluster kernel (kernels.cu).
	const int64_t B = m->mb.docs.B;
	const int32_t* order = m->mb.b_order.as<int32_t>();
	const bool tmem = m->tmem_mode && tmem_estep_applicable(m->K, m->beta_elem);
	const int64_t long_end = tmem ? m->mb.len_gt[0] : B;
	// documents too long for both the streaming kernel and the shared memory of k_estep: order[0, n_over)
	int64_t n_over = 0;
	if(long_end > 0 && !stream_estep_applicable(m->K, m->mb.docs.n_max, m->beta_elem, m->smem_optin))
		while(n_over < long_end && !estep_fits(m, m->mb.sorted_len[n_over]))
			++n_over;
	if(n_over > 0) {
		TRY(run_estep_with_long(m, a, n_over, long_end));
	} else if(long_end > 0) {
		if(stream_estep_applicable(m->K, m->mb.docs.n_max, m->beta_elem, m->smem_optin)) {
			Launch l(m, KK_ESTEP);
			launch_estep_stream(a, m->mb.docs, order, 0, long_end, m->mb.docs.n_max, m->beta_elem, m->stream);
			m->stream_ran = true;
		} else {
			TRY(run_estep_buckets(m, a, long_end));
		}
	}
	if(long_end < B && n_over == 0) {
		Launch l(m, KK_ESTEP);
		if(launch_estep_tmem(a, m->mb.docs, order, long_end, B - long_end, tmem_estep_max_len(), m->stream) != 0)
			return fail(m, TRLDA_ERR_CUDA, "The tensor-memory E-step kernel could not be launched.");
	}
	m->gamma_valid = true;
	m->stats.estep_docs = B;
	return check_launch(m, "estep");
}

// row sums of the sufficient statistics of the last E-step (summed over ranks) -> rows_stat
int reduce_doc_stat(trlda_model* m) {
	const int P = colsum_num_partials(m->mb.docs.B);
	CUDA_TRY(m, m->partials.ensure(sizeof(double) * (size_t) std::max(P, rowsum_num_partials(m->V)) * m->K));
	{
		Launch l(m, KK_REDUCE);
		launch_colsum(m->doc_stat.as<double>(), m->K, m->mb.docs.B, m->partials.as<double>(), m->rows_stat.as<double>(), m->stream);
	}
	TRY(check_launch(m, "colsum"));
	return allreduce(m, m->rows_stat.p, m->K, ncclDouble);
}

// Builds the word-sorted token list (CSC view) of the resident minibatch from the pinned staging copy and sends it
// to the device.  Stable counting sort in O(N + T V): thread t owns a contiguous range of the token stream, counts its
// words, the per-(word, thread) offsets follow from one pass over the T histograms, and every thread places its own
// tokens — a word's tokens stay in document order whatever the number of threads.
int ensure_csc(trlda_model* m) {
	if(!m->csc_pending)
		return TRLDA_OK;
	m->csc_pending = false;
	const int64_t B = m->mb.docs.B, N = m->mb.docs.N;
	const int V = m->V;
	const int T = std::max(1, m->csc_threads);
	char* base = m->staging.as<char>();
	const int64_t* s_ptr = reinterpret_cast<const int64_t*>(base + m->stage_off[0]);
	const int32_t* ids = reinterpret_cast<const int32_t*>(base + m->stage_off[1]);
	int32_t* s_wptr = reinterpret_cast<int32_t*>(base + m->stage_off[2]);
	int32_t* s_tdoc = reinterpret_cast<int32_t*>(base + m->stage_off[3]);
	int32_t* s_tsrc = reinterpret_cast<int32_t*>(base + m->stage_off[4]);
	auto run = [&](auto&& fn) {
		std::vector<std::thread> pool;
		for(int t = 1; t < T; ++t)
			pool.emplace_back(fn, t);
		fn(0);
		for(auto& th : pool)
			th.join();
	};
	// thread t takes the documents [d0(t), d0(t+1)), cut where the token stream passes t N / T
	std::vector<int64_t> doc_cut(T + 1, B);
	doc_cut[0] = 0;
	for(int t = 1; t < T; ++t)
		doc_cut[t] = std::lower_bound(s_ptr, s_ptr + B, N * t / T) - s_ptr;
	std::vector<std::vector<int32_t>> hist(T);
	run([&](int t) {
		hist[t].assign((size_t) V, 0);
		int32_t* h = hist[t].data();
		for(int64_t i = s_ptr[doc_cut[t]]; i < s_ptr[doc_cut[t + 1]]; ++i)
			h[ids[i]]++;
	});
	// word_ptr and, in place of the counts, every thread's first slot of every word
	int32_t total = 0;
	for(int w = 0; w < V; ++w) {
		s_wptr[w] = total;
		for(int t = 0; t < T; ++t) {
			const int32_t c = hist[t][w];
			hist[t][w] = total;
			total += c;
		}
	}
	s_wptr[V] = total;
	run([&](int t) {
		int32_t* cursor = hist[t].data();
		for(int64_t d = doc_cut[t]; d < doc_cut[t + 1]; ++d)
			for(int64_t i = s_ptr[d]; i < s_ptr[d + 1]; ++i) {
				const int32_t pos = cursor[ids[i]]++;
				s_tdoc[pos] = (int32_t) d;
				s_tsrc[pos] = (int32_t) i;
			}
	});
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(m->mb.b_tok_doc.p, s_tdoc, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
		CUDA_TRY(m, cudaMemcpyAsync(m->mb.b_tok_src.p, s_tsrc, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
	}
	CUDA_TRY(m, cudaMemcpyAsync(m->mb.b_word_ptr.p, s_wptr, sizeof(int32_t) * ((size_t) V + 1), cudaMemcpyHostToDevice, m->stream));
	return TRLDA_OK;
}

// dense sufficient statistics of the last E-step (summed over ranks) -> sstats   (lda.cpp:207-217)
int run_scatter_dense(trlda_model* m, bool reduce_over_ranks = true, bool for_peers = false) {
	TRY(ensure_csc(m));
	if(!for_peers)
		CUDA_TRY(m, m->sstats.ensure(kv_bytes(m)));
	ScatterArgs a;
	a.K = m->K;
	a.V = m->V;
	a.etheta = m->beta_elem == 4 ? (void*) estep_etheta32(m) : m->etheta.p;
	a.etheta_elem = m->beta_elem == 4 ? 4 : 8;
	a.weight = estep_weight(m);
	a.beta = m->beta.p;
	a.beta_elem = m->beta_elem;
	a.sstats = m->sstats.as<double>();
	if(for_peers) {
		a.peer_ranks = m->nranks;
		a.peer_rank = m->rank;
		a.peer_shard_cap = m->peer_shard_cap;
		a.peer_elem = m->peer_sstats_elem;
		for(int r = 0; r < m->nranks; ++r)
			a.peer_out[r] = m->peer_sstats[r];
	}
	a.fused = false;
	{
		Launch l(m, KK_SCATTER);
		launch_scatter(a, m->mb.docs, m->stream);
	}
	TRY(check_launch(m, "scatter"));
	if(!reduce_over_ranks)
		return TRLDA_OK;
	return allreduce(m, m->sstats.p, (size_t) m->K * m->V, ncclDouble);
}

// all ranks have finished the work enqueued before this point (a one-element all-reduce on the model's stream)
int rank_barrier(trlda_model* m) {
	if(m->nranks <= 1)
		return TRLDA_OK;
	return allreduce(m, m->scalars.as<double>() + 4000, 1, ncclDouble);
}

// M-step: rebuild lambda from the last E-step.  lambda' is the CURRENT buffer unless `prime` is given; the new
// lambda goes to the other buffer and becomes current.  Also refreshes rows / psi_rows (by linearity of the
// blend) and, if asked, beta and the per-word psi sums for the eta update.
int run_mstep(trlda_model* m, const MStepCoef& coef, const double* prime, double* target, bool write_beta,
              bool want_psi_partials, bool force_dense, bool broadcast_lambda = true) {
	TRY(reduce_doc_stat(m));
	double a = 0, b = 0, c = 0;
	if(coef.mode == MSTEP_ONLINE) {
		a = 1. - coef.rho;
		b = coef.rho * m->V * coef.eta;
		c = coef.rho * coef.scale;
	} else if(coef.mode == MSTEP_BATCH) {
		a = 0.;
		b = m->V * coef.eta;
		c = 1.;
	} else {
		a = 1.;
		b = 0.;
		c = 1.;
	}
	{
		Launch l(m, KK_MISC);
		launch_rows_update(coef.mode == MSTEP_BATCH ? nullptr : m->rows_prev.as<double>(), m->rows_stat.as<double>(), a, b, c,
		                   m->K, m->rows.as<double>(), m->psi_rows.as<double>(), m->stream);
	}
	if(m->nranks > 1 && m->mb.gdocs.ready && !force_dense) {
		// gather exchange: (1) every rank receives all documents' etheta and token weights; (2) the single-GPU kernel
		// (scatter + blend + beta-prep) runs on this rank's words over the tokens of ALL documents; (3) the ranks
		// exchange their slices of the new beta (and, when the caller needs lambda afterwards, of lambda)
		trlda_model::GlobalDocs& g = m->mb.gdocs;
		const int v0 = word_begin(m, m->rank), v1 = word_begin(m, m->rank + 1);
		{
			std::vector<int64_t> eoff(m->nranks), en(m->nranks);
			for(int r = 0; r < m->nranks; ++r) {
				eoff[r] = g.doc_off[r] * m->K;
				en[r] = g.pad_B[r] * m->K;
			}
			nvtxRangePushA("exchange: all-gather etheta, weights");
			TRY(gather_segments(m, g.etheta32.p, eoff, en, sizeof(float), ncclFloat));
			TRY(gather_segments(m, g.weight.p, g.tok_off, g.pad_N, sizeof(double), ncclDouble));
			nvtxRangePop();
		}
		if(want_psi_partials)
			CUDA_TRY(m, cudaMemsetAsync(m->vpartials.p, 0, sizeof(double) * m->V, m->stream));
		{
			ScatterArgs sa;
			sa.K = m->K;
			sa.V = m->V;
			sa.etheta = g.etheta32.p;
			sa.etheta_elem = 4;
			sa.weight = g.weight.as<double>();
			sa.beta = m->beta.p;
			sa.beta_elem = m->beta_elem;
			sa.fused = true;
			sa.coef = coef;
			sa.lambda_prime = prime;
			sa.lambda = target;
			sa.psi_rows = m->psi_rows.as<double>();
			sa.write_beta = write_beta;
			sa.psi_partials = want_psi_partials ? m->vpartials.as<double>() : nullptr;
			sa.v0 = v0;
			sa.v1 = v1;
			// Pipeline: the word shard is cut into pieces; while the kernel works on piece c + 1 the ranks exchange piece
			// c of the new beta (and lambda) on a second stream - one broadcast per rank and piece, grouped (the pieces
			// of one exchange are not equally spaced, so it is not a single all-gather).  TRLDA_GATHER_CHUNKS=1: one
			// kernel, then one all-gather.
			// (measured at 2 GPUs: 29.9 -> 29.4 ms per step with four pieces; more ranks keep the single all-gather until
			// measured otherwise)
			static const int forced_pieces = [] { const char* e = getenv("TRLDA_GATHER_CHUNKS"); return e ? std::max(1, atoi(e)) : 0; }();
			const int pieces = forced_pieces ? forced_pieces : m->nranks == 2 ? 4 : 1;
			if(pieces > 1 && m->aux[0] && (write_beta || broadcast_lambda)) {
				auto piece_begin = [&](int r, int c) {
					const int64_t b = word_begin(m, r), e = word_begin(m, r + 1);
					return (int) (b + (e - b) * c / pieces);
				};
				nvtxRangePushA("scatter + M-step pipelined with the exchange of beta / lambda");
				for(int c = 0; c < pieces; ++c) {
					sa.v0 = piece_begin(m->rank, c);
					sa.v1 = piece_begin(m->rank, c + 1);
					{
						Launch l(m, KK_SCATTER_MSTEP);
						launch_scatter(sa, g.view, m->stream);
					}
					CUDA_TRY(m, cudaEventRecord(m->fork_event, m->stream));
					CUDA_TRY(m, cudaStreamWaitEvent(m->aux[0], m->fork_event, 0));
					NCCL_TRY(m, nccl_api().GroupStart());
					for(int r = 0; r < m->nranks; ++r) {
						const int64_t off = (int64_t) piece_begin(r, c) * m->K;
						const int64_t cnt = (int64_t) (piece_begin(r, c + 1) - piece_begin(r, c)) * m->K;
						if(cnt <= 0)
							continue;
						if(write_beta) {
							char* seg = static_cast<char*>(m->beta.p) + (size_t) off * sizeof(float);
							NCCL_TRY(m, nccl_api().Broadcast(seg, seg, (size_t) cnt, ncclFloat, r, m->comm, m->aux[0]));
						}
						if(broadcast_lambda)
							NCCL_TRY(m, nccl_api().Broadcast(target + off, target + off, (size_t) cnt, ncclDouble, r, m->comm, m->aux[0]));
					}
					NCCL_TRY(m, nccl_api().GroupEnd());
				}
				CUDA_TRY(m, cudaEventRecord(m->join_event[0], m->aux[0]));
				CUDA_TRY(m, cudaStreamWaitEvent(m->stream, m->join_event[0], 0));
				nvtxRangePop();
				TRY(check_launch(m, "mstep (word shard, pipelined)"));
				if(want_psi_partials)
					TRY(allreduce(m, m->vpartials.p, m->V, ncclDouble));
				m->beta_valid = write_beta;
				m->lambda_sharded = !broadcast_lambda;
				return TRLDA_OK;
			}
			Launch l(m, KK_SCATTER_MSTEP);
			launch_scatter(sa, g.view, m->stream);
		}
		TRY(check_launch(m, "mstep (word shard)"));
		{
			std::vector<int64_t> woff(m->nranks), wn(m->nranks);
			for(int r = 0; r < m->nranks; ++r) {
				woff[r] = (int64_t) word_begin(m, r) * m->K;
				wn[r] = (int64_t) (word_begin(m, r + 1) - word_begin(m, r)) * m->K;
			}
			nvtxRangePushA("exchange: all-gather beta / lambda");
			if(write_beta)
				TRY(gather_segments(m, m->beta.p, woff, wn, sizeof(float), ncclFloat));
			if(broadcast_lambda)
				TRY(gather_segments(m, target, woff, wn, sizeof(double), ncclDouble));
			nvtxRangePop();
		}
		if(want_psi_partials)
			TRY(allreduce(m, m->vpartials.p, m->V, ncclDouble));
		m->beta_valid = write_beta;
		m->lambda_sharded = !broadcast_lambda;
		return TRLDA_OK;
	}
	if(m->nranks > 1 && m->peer_ready && m->use_peer && !force_dense && m->K % 4 == 0) {
		// fused path over NVLink peer memory: local scatter, barrier, then one kernel per rank that pulls every
		// rank's partial statistics for its word shard, blends, and pushes beta (and lambda when the caller needs
		// the full matrix afterwards) into every replica
		TRY(run_scatter_dense(m, false, true));
		TRY(rank_barrier(m));
		const int target_index = target == m->lam[0].as<double>() ? 0 : 1;
		ShardMStepArgs sa;
		sa.K = m->K;
		sa.V = m->V;
		sa.v0 = (int) ((int64_t) m->V * m->rank / m->nranks);
		sa.v1 = (int) ((int64_t) m->V * (m->rank + 1) / m->nranks);
		sa.nranks = m->nranks;
		sa.rank = m->rank;
		sa.coef = coef;
		for(int r = 0; r < m->nranks; ++r) {
			sa.beta[r] = m->peer_beta[r];
			sa.lambda[r] = static_cast<double*>(m->peer_lam[target_index][r]);
		}
		sa.partials = m->sstats32.p;
		sa.shard_cap = m->peer_shard_cap;
		sa.sstats_elem = m->peer_sstats_elem;
		sa.lambda_prime = prime;
		sa.psi_rows = m->psi_rows.as<double>();
		sa.beta_elem = m->beta_elem;
		sa.write_beta = write_beta;
		sa.broadcast_lambda = broadcast_lambda;
		sa.psi_partials = want_psi_partials ? m->vpartials.as<double>() : nullptr;
		if(want_psi_partials)
			CUDA_TRY(m, cudaMemsetAsync(m->vpartials.p, 0, sizeof(double) * m->V, m->stream));
		{
			Launch l(m, KK_MSTEP);
			launch_mstep_shard(sa, m->stream);
		}
		TRY(check_launch(m, "mstep_shard"));
		TRY(rank_barrier(m));
		if(want_psi_partials)
			TRY(allreduce(m, m->vpartials.p, m->V, ncclDouble));
		m->beta_valid = write_beta;
		m->lambda_sharded = !broadcast_lambda;
		return TRLDA_OK;
	}
	const bool dense = force_dense || m->nranks > 1;
	if(dense) {
		TRY(run_scatter_dense(m));
		MStepArgs ma;
		ma.K = m->K;
		ma.V = m->V;
		ma.coef = coef;
		ma.sstats = m->sstats.as<double>();
		ma.lambda_prime = prime;
		ma.lambda = target;
		ma.psi_rows = m->psi_rows.as<double>();
		ma.beta = m->beta.p;
		ma.beta_elem = m->beta_elem;
		ma.write_beta = write_beta;
		ma.psi_partials = want_psi_partials ? m->vpartials.as<double>() : nullptr;
		Launch l(m, KK_MSTEP);
		launch_mstep(ma, m->stream);
	} else {
		TRY(ensure_csc(m));
		ScatterArgs sa;
		sa.K = m->K;
		sa.V = m->V;
		sa.etheta = m->beta_elem == 4 ? (void*) estep_etheta32(m) : m->etheta.p;
		sa.etheta_elem = m->beta_elem == 4 ? 4 : 8;
		sa.weight = estep_weight(m);
		sa.beta = m->beta.p;
		sa.beta_elem = m->beta_elem;
		sa.fused = true;
		sa.coef = coef;
		sa.lambda_prime = prime;
		sa.lambda = target;
		sa.psi_rows = m->psi_rows.as<double>();
		sa.write_beta = write_beta;
		sa.psi_partials = want_psi_partials ? m->vpartials.as<double>() : nullptr;
		Launch l(m, KK_SCATTER_MSTEP);
		launch_scatter(sa, m->mb.docs, m->stream);
	}
	m->beta_valid = write_beta;
	return check_launch(m, "mstep");
}

// copies n doubles device -> pinned host and waits
int read_back(trlda_model* m, const double* dev, size_t n, double* out) {
	CUDA_TRY(m, m->readback.ensure(sizeof(double) * n));
	CUDA_TRY(m, cudaMemcpyAsync(m->readback.p, dev, sizeof(double) * n, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	memcpy(out, m->readback.p, sizeof(double) * n);
	m->stats.d2h_bytes += sizeof(double) * n;
	return TRLDA_OK;
}

// psiGammaDiff_k = sum_d [psi(gamma_dk) - psi(sum_k gamma_dk)] over the whole (global) minibatch
int alpha_statistics(trlda_model* m, std::vector<double>& diff) {
	// doc_stat is free after the M-step: reuse it for the per-document terms
	{
		Launch l(m, KK_ALPHA_STATS);
		launch_alpha_stats(m->gamma.as<double>(), m->K, m->mb.docs.B, m->doc_stat.as<double>(), m->stream);
	}
	const int P = colsum_num_partials(m->mb.docs.B);
	CUDA_TRY(m, m->partials.ensure(sizeof(double) * (size_t) std::max(P, rowsum_num_partials(m->V)) * m->K));
	{
		Launch l(m, KK_REDUCE);
		launch_colsum(m->doc_stat.as<double>(), m->K, m->mb.docs.B, m->partials.as<double>(), m->rows_stat.as<double>(), m->stream);
	}
	TRY(check_launch(m, "alpha_stats"));
	TRY(allreduce(m, m->rows_stat.p, m->K, ncclDouble));
	diff.resize(m->K);
	return read_back(m, m->rows_stat.as<double>(), m->K, diff.data());
}

// Newton direction pieces (onlinelda.cpp:128-134, batchlda.cpp:90-96, cumulativelda.cpp:98-104)
double alpha_newton(const std::vector<double>& alpha, const std::vector<double>& diff, double n,
                    std::vector<double>& g, std::vector<double>& h) {
	const int K = (int) alpha.size();
	double asum = 0.0;
	for(int k = 0; k < K; ++k)
		asum += alpha[k];
	const double psi_asum = digamma(asum);
	double sgh = 0.0, sih = 0.0;
	g.resize(K);
	h.resize(K);
	for(int k = 0; k < K; ++k) {
		g[k] = diff[k] - n * (digamma(alpha[k]) - psi_asum);
		h[k] = -n * host_polygamma(1, alpha[k]);
		sgh += g[k] / h[k];
		sih += 1. / h[k];
	}
	const double z = n * host_polygamma(1, asum);
	return sgh / (1. / z + sih);
}

double alpha_objective(const std::vector<double>& a, const std::vector<double>& diff, double n) {
	double lg = 0.0, lin = 0.0, sum = 0.0;
	for(size_t k = 0; k < a.size(); ++k) {
		lg += lgamma(a[k]);
		lin += diff[k] * (a[k] - 1.);
		sum += a[k];
	}
	return n * (lgamma(sum) - lg) + lin;     // batchlda.cpp:82-83
}

// line-searched Newton ascent on alpha (batchlda.cpp:82-142, cumulativelda.cpp:91-150)
void alpha_line_search(trlda_model* m, const std::vector<double>& diff, double n, const trlda_params* p) {
	const int K = m->K;
	std::vector<double> g, h, a(K);
	double L = alpha_objective(m->alpha, diff, n);
	double Lprime = L;
	for(int i = 0; i < p->max_iter_alpha; ++i) {
		if(p->verbosity > 1)
			printf("\tCurrent function value: %g\n", L);
		const double c = alpha_newton(m->alpha, diff, n, g, h);
		double rho = .2;
		for(int j = 0; j < 20; ++j) {
			bool small = false;
			for(int k = 0; k < K; ++k) {
				a[k] = m->alpha[k] - rho * (g[k] - c) / h[k];
				if(a[k] < p->min_alpha)
					small = true;
			}
			if(small) {
				rho /= 2.;
				continue;
			}
			Lprime = alpha_objective(a, diff, n);
			if(L <= Lprime) {
				m->alpha = a;
				break;
			}
			rho /= 2.;
		}
		if(Lprime - L < p->emp_bayes_threshold)
			break;
		L = Lprime;
	}
}

// sum psi(lambda) - V sum_k psi(sum_w lambda_kw) from the per-word partials and psi_rows (onlinelda.cpp:153)
int eta_constant(trlda_model* m, double* out) {
	{
		Launch l(m, KK_REDUCE);
		launch_sum(m->vpartials.as<double>(), m->V, m->scalars.as<double>() + 16, m->scalars.as<double>(), m->stream);
	}
	{
		Launch l(m, KK_REDUCE);
		launch_sum(m->psi_rows.as<double>(), m->K, m->scalars.as<double>() + 16 + 1024, m->scalars.as<double>() + 1, m->stream);
	}
	TRY(check_launch(m, "eta_sums"));
	double h[2];
	TRY(read_back(m, m->scalars.as<double>(), 2, h));
	*out = h[0] - m->V * h[1];
	return TRLDA_OK;
}

int begin_update(trlda_model* m) {
	TRY(set_device(m));
	TRY(ensure_beta(m));
	TRY(ensure_small(m));
	CUDA_TRY(m, m->lam[1 - m->cur].ensure(kv_bytes(m)));
	return TRLDA_OK;
}

void consume_injections(trlda_model* m) {
	m->inj_gamma_cols = -1;
	m->inj_gamma.clear();
	m->inj_gamma.shrink_to_fit();
	m->inj_lambda.clear();
	m->inj_lambda.shrink_to_fit();
}

// ---- OnlineLDA::updateParameters, onlinelda.cpp:53-180 ---------------------------------------------------------------
int online_update(trlda_model* m, const trlda_params* p, double* result) {
	const int64_t B = m->mb.global_B;
	if(B == 0) {
		*result = 1.0;                                               // :54-56 (returns `true`), counter untouched
		return TRLDA_OK;
	}
	TRY(begin_update(m));

	double rho = p->rho;                                             // :59-66
	if(rho < 0.) {
		if(p->adaptive)
			rho = m->ada_rho;
		else
			rho = pow(p->tau + (double) m->update_count, -p->kappa);
	}
	const double scale = (double) m->num_documents / (double) B;
	MStepCoef coef{MSTEP_ONLINE, rho, m->eta, scale};
	const double eta_at_mstep = m->eta;
	bool have_psi_partials = false;
	bool have_dense_sstats = false;

	if(p->update_lambda) {
		const double* prime = m->lambda();                           // lambdaPrime = mLambda, :68 (no copy: buffer swap)
		double* target = m->lambda_next();
		TRY(compute_rows(m, prime, m->rows_prev.as<double>()));

		if(p->max_iter_tr > 0) {
			// phi = 1/K warm start, :79-86
			CUDA_TRY(m, m->wordcount.ensure(sizeof(double) * m->V));
			{
				Launch l(m, KK_MISC);
				launch_wordcount(m->mb.docs, m->V, m->wordcount.as<double>(), m->stream);
			}
			TRY(allreduce(m, m->wordcount.p, m->V, ncclDouble));
			const double scale_k = (double) m->num_documents / (double) B / (double) m->K;
			{
				Launch l(m, KK_MISC);
				launch_rows_update(m->rows_prev.as<double>(), nullptr, 1. - rho,
				                   rho * (m->V * m->eta + scale_k * (double) m->mb.docs_total_count), 0., m->K,
				                   m->rows.as<double>(), m->psi_rows.as<double>(), m->stream);
			}
			{
				Launch l(m, KK_INIT_UPDATE);
				launch_init_update(m->mb.docs, m->K, m->V, rho, m->eta, scale_k, prime, target, m->psi_rows.as<double>(),
				                   m->beta.p, m->beta_elem, m->wordcount.as<double>(), m->stream);
			}
			TRY(check_launch(m, "init_update"));
			m->beta_valid = true;

			for(int i = 0; i < p->max_iter_tr; ++i) {                 // :89-101
				const bool last = i == p->max_iter_tr - 1;
				TRY(run_estep(m, (i > 0 && p->init_gamma) ? GAMMA_KEEP : GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
				const bool dense = last && p->adaptive;
				TRY(run_mstep(m, coef, prime, target, !last, last && p->update_eta, dense, last));
				have_psi_partials = last && p->update_eta;
				have_dense_sstats = dense || m->nranks > 1;
			}
		} else {                                                     // :102-110
			TRY(prepare_beta(m));
			TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
			TRY(run_mstep(m, coef, prime, target, false, p->update_eta, p->adaptive));
			have_psi_partials = p->update_eta;
			have_dense_sstats = p->adaptive || m->nranks > 1;
		}
		m->cur = 1 - m->cur;                                         // the new lambda becomes current
	}

	if(p->update_alpha) {                                            // :116-142
		if(!p->update_lambda) {
			TRY(prepare_beta(m));
			TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
		}
		std::vector<double> diff, g, h;
		TRY(alpha_statistics(m, diff));
		const double c = alpha_newton(m->alpha, diff, (double) B, g, h);
		for(int k = 0; k < m->K; ++k) {
			m->alpha[k] = m->alpha[k] - rho * (g[k] - c) / h[k];
			if(m->alpha[k] < p->min_alpha)
				m->alpha[k] = p->min_alpha;
		}
		TRY(upload_alpha(m));
	}

	if(p->update_eta) {                                              // :147-162
		if(!have_psi_partials)
			TRY(prepare_beta(m, true));
		double c = 0.0;
		TRY(eta_constant(m, &c));
		const int K = m->K, N = m->V;
		const double g = c - (double) K * N * (digamma(m->eta) - digamma(N * m->eta));
		const double h = (double) K * N * (host_polygamma(1, N * m->eta) - host_polygamma(1, m->eta));
		m->eta = m->eta - rho * g / h;
		if(m->eta < p->min_eta)
			m->eta = p->min_eta;
	}

	if(p->update_lambda && p->adaptive) {                            // :167-175
		if(!have_dense_sstats)
			return fail(m, TRLDA_ERR_CUDA, "internal error: dense sufficient statistics missing for the adaptive rate");
		const size_t KV = (size_t) m->K * m->V;
		if(!m->ada_gradient.p) {
			CUDA_TRY(m, m->ada_gradient.ensure(kv_bytes(m)));
			CUDA_TRY(m, cudaMemsetAsync(m->ada_gradient.p, 0, kv_bytes(m), m->stream));
		}
		const int nb = adaptive_num_blocks((int64_t) KV);
		// after the swap the old lambda (= lambda') sits in the non-current buffer
		{
			Launch l(m, KK_MISC);
			launch_adaptive(m->sstats.as<double>(), m->lambda_next(), m->ada_gradient.as<double>(), (int64_t) KV, eta_at_mstep,
			                scale, m->ada_tau, m->scalars.as<double>(), m->stream);
		}
		TRY(check_launch(m, "adaptive"));
		std::vector<double> part(2 * nb);
		TRY(read_back(m, m->scalars.as<double>(), 2 * nb, part.data()));
		double sq = 0.0, gsq = 0.0;
		for(int i = 0; i < nb; ++i) {
			sq += part[i];
			gsq += part[nb + i];
		}
		m->ada_sq_norm = (1. - 1. / m->ada_tau) * m->ada_sq_norm + 1. / m->ada_tau * sq;
		m->ada_rho = gsq / m->ada_sq_norm;
		m->ada_tau = m->ada_tau * (1. - m->ada_rho) + 1.;
	}

	m->update_count++;                                               // :177
	*result = rho;
	return TRLDA_OK;
}



// ---- BatchLDA::updateParameters, batchlda.cpp:43-209 -------------------------------------------------------------------
int batch_update(trlda_model* m, const trlda_params* p, double* result) {
	const int64_t B = m->mb.global_B;
	*result = 1.;
	if(B == 0)
		return TRLDA_OK;
	TRY(begin_update(m));

	for(int epoch = 0; epoch < p->max_epochs; ++epoch) {
		bool have_psi_partials = false;
		if(p->update_lambda) {                                       // :54-61
			TRY(prepare_beta(m));
			TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
			MStepCoef coef{MSTEP_BATCH, 1., m->eta, 1.};
			TRY(run_mstep(m, coef, nullptr, m->lambda_next(), true, p->update_eta, false, epoch == p->max_epochs - 1));
			m->cur = 1 - m->cur;
			have_psi_partials = p->update_eta;
		}

		if(p->update_alpha) {                                        // :66-143
			if(!p->update_lambda) {
				TRY(prepare_beta(m));
				TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
			}
			std::vector<double> diff;
			TRY(alpha_statistics(m, diff));
			if(p->verbosity > 1)
				printf("Optimizing alpha...\n");
			alpha_line_search(m, diff, (double) B, p);
			TRY(upload_alpha(m));
		}

		if(p->update_eta) {                                          // :147-205
			if(!have_psi_partials)
				TRY(prepare_beta(m, true));
			double c = 0.0;
			TRY(eta_constant(m, &c));
			const double K = m->K, N = m->V;
			if(p->verbosity > 1)
				printf("Optimizing eta...\n");
			double L = (m->eta - 1) * c + K * lgamma(N * m->eta) - K * N * lgamma(m->eta);
			double Lprime = L;
			for(int i = 0; i < p->max_iter_eta; ++i) {
				if(p->verbosity > 1)
					printf("\tCurrent function value: %g\n", L);
				const double g = c - K * N * (digamma(m->eta) - digamma(N * m->eta));
				const double h = K * N * (host_polygamma(1, N * m->eta) - host_polygamma(1, m->eta));
				double rho = .5;
				for(int j = 0; j < 20; ++j) {
					const double eta = m->eta - rho * g / h;
					if(eta < p->min_eta) {
						rho /= 2.;
						continue;
					}
					Lprime = (eta - 1) * c + K * lgamma(N * eta) - K * N * lgamma(eta);
					if(L <= Lprime) {
						m->eta = eta;
						break;
					}
					rho /= 2.;
				}
				if(Lprime - L < p->emp_bayes_threshold)
					break;
				L = Lprime;
			}
		}
	}
	return TRLDA_OK;
}

// ---- CumulativeLDA::updateParameters, cumulativelda.cpp:49-153 ----------------------------------------------------------
int cumulative_update(trlda_model* m, const trlda_params* p, double* result) {
	const int64_t B = m->mb.global_B;
	*result = 1.;
	if(B == 0)
		return TRLDA_OK;
	TRY(begin_update(m));

	// lambdaPrime = mLambda (:57); mLambda = random (:60) — even when update_lambda is false
	const int prime_buf = m->cur;
	const double* prime = m->lam[prime_buf].as<double>();
	double* work = m->lam[1 - prime_buf].as<double>();
	if(!m->inj_lambda.empty()) {
		CUDA_TRY(m, cudaMemcpyAsync(work, m->inj_lambda.data(), kv_bytes(m), cudaMemcpyHostToDevice, m->stream));
		CUDA_TRY(m, cudaStreamSynchronize(m->stream));
		m->stats.h2d_bytes += kv_bytes(m);
	} else {
		Launch l(m, KK_RNG);
		launch_gamma_rng(work, (int64_t) m->K * m->V, current_seed(), next_stream_id(), m->stream);
	}
	m->cur = 1 - prime_buf;
	m->beta_valid = false;

	if(p->update_lambda && p->max_epochs > 0) {                      // :62-71
		TRY(compute_rows(m, prime, m->rows_prev.as<double>()));
		// lambda = lambda' + sstats is rebuilt in place over the random lambda: each word's column is read
		// (through beta) and rewritten by the same CTA
		for(int epoch = 0; epoch < p->max_epochs; ++epoch) {
			TRY(prepare_beta(m));
			TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
			MStepCoef coef{MSTEP_CUMULATIVE, 1., m->eta, 1.};
			TRY(run_mstep(m, coef, prime, work, true, false, false, epoch == p->max_epochs - 1));
		}
	}

	if(p->update_alpha) {                                            // :76-150
		TRY(prepare_beta(m));
		TRY(run_estep(m, GAMMA_FRESH, nullptr, p->max_iter_inference, p->threshold));
		std::vector<double> diff;
		TRY(alpha_statistics(m, diff));
		if(m->psi_gamma_diff.size() != (size_t) m->K)
			m->psi_gamma_diff.assign(m->K, 0.0);
		for(int k = 0; k < m->K; ++k)
			m->psi_gamma_diff[k] += diff[k];                         // :84
		m->cum_num_documents += B;                                   // :85
		if(p->verbosity > 1)
			printf("Optimizing alpha...\n");
		alpha_line_search(m, m->psi_gamma_diff, (double) m->cum_num_documents, p);
		TRY(upload_alpha(m));
	}
	return TRLDA_OK;
}

int update_resident(trlda_model* m, const trlda_params* p, double* result) {
	if(p->inference_method != TRLDA_INFERENCE_VI)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device.");
	double r = 1.0;
	int status;
	switch(m->kind) {
		case TRLDA_KIND_ONLINE: status = online_update(m, p, &r); break;
		case TRLDA_KIND_BATCH: status = batch_update(m, p, &r); break;
		default: status = cumulative_update(m, p, &r); break;
	}
	consume_injections(m);
	if(status != TRLDA_OK)
		return status;
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	if(result)
		*result = r;
	return TRLDA_OK;
}

void collect_spans(trlda_model* m) {
	for(auto& s : m->spans) {
		float ms = 0.f;
		if(cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess)
			m->stats.ms[s.kind] += ms;
		m->event_pool.push_back(s.a);
		m->event_pool.push_back(s.b);
	}
	m->spans.clear();
}

}  // namespace

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
extern "C" {

void trlda_params_default(trlda_params* p) {
	p->inference_method = TRLDA_INFERENCE_VI;
	p->threshold = 0.001;
	p->max_iter_inference = 100;
	p->max_iter_tr = 10;
	p->tau = 100.;
	p->kappa = .7;
	p->rho = -1.;
	p->adaptive = 0;
	p->num_samples = 1;
	p->burn_in = 2;
	p->init_gamma = 1;
	p->update_lambda = 1;
	p->update_alpha = 0;
	p->update_eta = 0;
	p->min_alpha = 1e-6;
	p->min_eta = 1e-6;
	p->max_epochs = 100;
	p->max_iter_alpha = 10;
	p->max_iter_eta = 20;
	p->emp_bayes_threshold = 1e-8;
	p->verbosity = 0;
}

const char* trlda_kernel_kind_name(int kind) {
	static const char* names[TRLDA_NUM_KERNEL_KINDS] = {
		"rowsum", "beta_prep", "estep", "scatter_mstep", "scatter", "mstep", "init_update", "reduce",
		"alpha_stats", "rng", "elbo", "misc"};
	return kind >= 0 && kind < TRLDA_NUM_KERNEL_KINDS ? names[kind] : "?";
}

const char* trlda_last_error(const trlda_model* m) { return m ? m->error.c_str() : g_error.c_str(); }

void trlda_seed(uint64_t seed) {
	std::lock_guard<std::mutex> lock(g_seed_mutex);
	g_seed = seed;
	g_stream_counter = 0;
}

int trlda_create(int kind, int num_words, int num_topics, int64_t num_documents, const double* alpha, double eta,
                 int device, int precision, trlda_model** out) {
	if(!out)
		return fail(nullptr, TRLDA_ERR_ARG, "Null output pointer.");
	*out = nullptr;
	if(kind < TRLDA_KIND_ONLINE || kind > TRLDA_KIND_CUMULATIVE)
		return fail(nullptr, TRLDA_ERR_ARG, "Unknown model kind.");
	if(num_words <= 0 || num_topics <= 0)
		return fail(nullptr, TRLDA_ERR_ARG, "The number of words and topics must be positive.");
	if(num_topics > 4096)
		return fail(nullptr, TRLDA_ERR_UNSUPPORTED, "More than 4096 topics are not supported.");
	if(num_documents < 0)
		return fail(nullptr, TRLDA_ERR_ARG, "The number of documents should not be negative.");
	if(!alpha)
		return fail(nullptr, TRLDA_ERR_ARG, "Alpha has wrong dimensionality.");
	for(int k = 0; k < num_topics; ++k)
		if(alpha[k] < 0.)
			return fail(nullptr, TRLDA_ERR_ARG, "Alpha should not be negative.");
	if(precision != TRLDA_PRECISION_FP64 && precision != TRLDA_PRECISION_MIXED)
		return fail(nullptr, TRLDA_ERR_ARG, "Unknown precision mode.");

	int count = 0;
	if(cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
		return fail(nullptr, TRLDA_ERR_CUDA, "No CUDA device available; trlda_b200 has no CPU fallback.");
	if(device < 0 || device >= count)
		return fail(nullptr, TRLDA_ERR_CUDA, "CUDA device ordinal out of range.");

	trlda_model* m = new trlda_model();
	m->kind = kind;
	m->K = num_topics;
	m->V = num_words;
	m->num_documents = num_documents;
	m->eta = eta;
	m->alpha.assign(alpha, alpha + num_topics);
	m->device = device;
	m->precision = precision;
	m->psi_gamma_diff.assign(num_topics, 0.0);
	if(const char* ft = getenv("TRLDA_ESTEP_TICKS"))
		if(atoi(ft) != 0 && m->ticks.ensure(16 * sizeof(unsigned long long)) == cudaSuccess)
			cudaMemset(m->ticks.p, 0, 16 * sizeof(unsigned long long));

	auto cleanup = [&](int code) {
		std::string msg = m->error;
		trlda_destroy(m);
		g_error = msg;
		return code;
	};
	cudaDeviceProp prop;
	if(cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
		fail(m, TRLDA_ERR_CUDA, "Cannot select the CUDA device.");
		return cleanup(TRLDA_ERR_CUDA);
	}
	if(prop.major < 10) {
		fail(m, TRLDA_ERR_CUDA, "trlda_b200 kernels are built for sm_100a (B200) only.");
		return cleanup(TRLDA_ERR_CUDA);
	}
	m->smem_optin = (int) prop.sharedMemPerBlockOptin;
	m->num_sms = prop.multiProcessorCount;
	if(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking) != cudaSuccess) {
		fail(m, TRLDA_ERR_CUDA, "Cannot create a CUDA stream.");
		return cleanup(TRLDA_ERR_CUDA);
	}
	configure_estep(m->smem_optin);
	if(const char* tm = getenv("TRLDA_ESTEP_TMEM"))
		m->tmem_mode = atoi(tm) != 0;
	cudaEventCreateWithFlags(&m->fork_event, cudaEventDisableTiming);
	cudaEventCreateWithFlags(&m->other_ready, cudaEventDisableTiming);
	for(int i = 0; i < trlda_model::kAuxStreams; ++i) {
		cudaStreamCreateWithFlags(&m->aux[i], cudaStreamNonBlocking);
		cudaEventCreateWithFlags(&m->join_event[i], cudaEventDisableTiming);
	}
	cudaStreamCreateWithFlags(&m->long_stream, cudaStreamNonBlocking);
	cudaEventCreateWithFlags(&m->long_join, cudaEventDisableTiming);

	int status = TRLDA_OK;
	auto init = [&]() -> int {
		CUDA_TRY(m, m->lam[0].ensure(kv_bytes(m)));
		CUDA_TRY(m, m->sweeps.ensure(2 * sizeof(unsigned long long)));    // [0] sweeps, [1] work counter of k_estep_tmem
		CUDA_TRY(m, cudaMemset(m->sweeps.p, 0, 2 * sizeof(unsigned long long)));
		TRY(ensure_small(m));
		TRY(upload_alpha(m));
		if(kind == TRLDA_KIND_CUMULATIVE) {
			launch_fill(m->lambda(), (int64_t) m->K * m->V, eta, m->stream);             // cumulativelda.cpp:30
		} else {
			launch_gamma_rng(m->lambda(), (int64_t) m->K * m->V, current_seed(), next_stream_id(), m->stream);   // lda.cpp:71
		}
		TRY(check_launch(m, "lambda init"));
		CUDA_TRY(m, cudaStreamSynchronize(m->stream));
		return TRLDA_OK;
	};
	status = init();
	if(status != TRLDA_OK)
		return cleanup(status);
	*out = m;
	return TRLDA_OK;
}

void trlda_destroy(trlda_model* m) {
	if(!m)
		return;
	cudaSetDevice(m->device);
	if(m->stream)
		cudaStreamSynchronize(m->stream);
	if(m->ticks.p) {
		unsigned long long t[16];
		cudaMemcpy(t, m->ticks.p, sizeof(t), cudaMemcpyDeviceToHost);
		static const char* stream_names[5] = {"document setup", "sweep (stream columns)", "fold partial sums",
		                                      "gamma/psi update + results", "convergence test"};
		static const char* resident_names[8] = {"tile -> TMEM + psi0", "pass B (acc) + butterfly", "gamma/psi update", "pass A (phi) + butterflies",
		                                        "fold in smem + barrier + send", "exchange wait", "weights", "results"};
		if(m->tmem_mode && m->beta_elem == 4 && tmem_estep_applicable(m->K, m->beta_elem)) {
			fprintf(stderr, "[trlda] TMEM E-step phase timers (one thread of rank 0, group 0 per cluster): %llu documents, %llu exchanges\n", t[15], t[14]);
			for(int i = 0; i < 8; ++i)
				fprintf(stderr, "[trlda]   %-30s %10.0f cycles/doc %8.0f cycles/exchange\n", resident_names[i],
				        t[15] ? (double) t[i] / (double) t[15] : 0.0, t[14] ? (double) t[i] / (double) t[14] : 0.0);
			if(t[10])
				fprintf(stderr, "[trlda]   busiest team %.0f cycles, mean %.0f over %llu teams (all launches): imbalance %.3f\n", (double) t[8],
				        (double) t[9] / (double) t[10], t[10], (double) t[8] * (double) t[10] / (double) t[9]);
		}
		if(m->stream_ran) {
			fprintf(stderr, "[trlda] streaming E-step phase timers: %llu documents, %llu sweeps\n", t[15], t[14]);
			for(int i = 0; i < 5; ++i)
				fprintf(stderr, "[trlda]   %-26s %10.0f cycles/doc\n", stream_names[i], t[15] ? (double) t[i] / (double) t[15] : 0.0);
		}
	}
	// the peer mappings and the communicator refer to this model's buffers: gone before the buffers are freed
	for(void* p : m->peer_opened)
		cudaIpcCloseMemHandle(p);
	if(m->comm && nccl_api().ok)
		nccl_api().CommDestroy(m->comm);
	collect_spans(m);
	for(cudaEvent_t e : m->event_pool)
		cudaEventDestroy(e);
	delete m;
}

int trlda_kind(const trlda_model* m) { return m->kind; }
int trlda_precision(const trlda_model* m) { return m->precision; }

int trlda_set_precision(trlda_model* m, int precision) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(precision != TRLDA_PRECISION_FP64 && precision != TRLDA_PRECISION_MIXED)
		return fail(m, TRLDA_ERR_ARG, "Unknown precision mode.");
	if(precision != m->precision) {
		m->precision = precision;
		m->beta_valid = false;
		m->beta.release();
		m->peer_ready = false;   // the peer-mapped beta replicas are gone: fall back to the all-reduce exchange
	}
	return TRLDA_OK;
}

int trlda_num_topics(const trlda_model* m) { return m->K; }
int trlda_num_words(const trlda_model* m) { return m->V; }

int trlda_get_lambda(trlda_model* m, double* out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	CUDA_TRY(m, cudaMemcpyAsync(out, m->lambda(), kv_bytes(m), cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += kv_bytes(m);
	return TRLDA_OK;
}

int trlda_set_lambda(trlda_model* m, const double* lambda, int rows, int cols) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(rows != m->K || cols != m->V || !lambda)
		return fail(m, TRLDA_ERR_ARG, "Lambda has wrong dimensionality.");      // lda.h:187
	TRY(set_device(m));
	CUDA_TRY(m, cudaMemcpyAsync(m->lambda(), lambda, kv_bytes(m), cudaMemcpyHostToDevice, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.h2d_bytes += kv_bytes(m);
	m->beta_valid = false;
	return TRLDA_OK;
}

int trlda_get_alpha(trlda_model* m, double* out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	memcpy(out, m->alpha.data(), sizeof(double) * m->K);
	return TRLDA_OK;
}

int trlda_set_alpha(trlda_model* m, const double* alpha, int n) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(n == 1 && m->K != 1) {                                                  // setAlpha(double), lda.h:146-150
		if(alpha[0] < 0.)
			return fail(m, TRLDA_ERR_ARG, "Alpha should not be negative.");
		std::fill(m->alpha.begin(), m->alpha.end(), alpha[0]);
	} else {                                                                   // setAlpha(ArrayXd), lda.h:154-160
		if(n != m->K)
			return fail(m, TRLDA_ERR_ARG, "Alpha has wrong dimensionality.");
		for(int k = 0; k < n; ++k)
			if(alpha[k] < 0.)
				return fail(m, TRLDA_ERR_ARG, "Alpha should not be negative.");
		m->alpha.assign(alpha, alpha + n);
	}
	TRY(set_device(m));
	return upload_alpha(m);
}

int trlda_get_eta(trlda_model* m, double* eta) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	*eta = m->eta;
	return TRLDA_OK;
}

int trlda_set_eta(trlda_model* m, double eta) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(eta < 0.)
		return fail(m, TRLDA_ERR_ARG, "Eta should not be negative.");          // lda.h:173
	m->eta = eta;
	return TRLDA_OK;
}

int trlda_get_num_documents(trlda_model* m, int64_t* n) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	*n = m->num_documents;
	return TRLDA_OK;
}

int trlda_set_num_documents(trlda_model* m, int64_t n) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(n < 0)
		return fail(m, TRLDA_ERR_ARG, "The number of documents should not be negative.");   // onlinelda.h:58
	m->num_documents = n;
	return TRLDA_OK;
}

int trlda_get_update_count(trlda_model* m, int64_t* n) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	*n = m->update_count;
	return TRLDA_OK;
}

int trlda_set_update_count(trlda_model* m, int64_t n) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(n < 0)
		return fail(m, TRLDA_ERR_ARG, "The update count should not be negative.");          // onlinelda.h:72
	m->update_count = n;
	return TRLDA_OK;
}

int trlda_upload_docs(trlda_model* m, const trlda_docs* docs) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	m->live_slot = -1;
	return upload_docs(m, docs);
}


int trlda_upload_docs_slot(trlda_model* m, const trlda_docs* docs, int slot) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(slot < 0 || slot >= 64)
		return fail(m, TRLDA_ERR_ARG, "Minibatch slot out of range.");
	if((int) m->slots.size() <= slot)
		m->slots.resize(slot + 1);
	// park the live minibatch (if it belongs to a slot), upload into fresh live buffers, finish the token list, park
	if(m->live_slot >= 0)
		std::swap(m->mb, m->slots[m->live_slot].mb);
	m->live_slot = -1;
	if(m->slots[slot].used)
		std::swap(m->mb, m->slots[slot].mb);                   // reuse the slot's buffers
	TRY(upload_docs(m, docs));
	TRY(ensure_csc(m));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));            // the pinned staging buffer is reused by the next upload
	std::swap(m->mb, m->slots[slot].mb);
	m->slots[slot].used = true;
	m->docs_resident = false;
	return TRLDA_OK;
}

int trlda_select_docs(trlda_model* m, int slot) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(slot < 0 || slot >= (int) m->slots.size() || !m->slots[slot].used)
		return fail(m, TRLDA_ERR_ARG, "No minibatch has been uploaded into this slot.");
	if(m->live_slot == slot)
		return TRLDA_OK;
	if(m->live_slot >= 0)
		std::swap(m->mb, m->slots[m->live_slot].mb);
	std::swap(m->mb, m->slots[slot].mb);
	m->live_slot = slot;
	m->docs_resident = true;
	m->csc_pending = false;
	m->gamma_valid = false;
	return TRLDA_OK;
}

// LDA::updateVariablesGibbs (lda.cpp:224-293) for the documents of `docs`: theta (K x B) and sstats (K x V, each token
// occurrence contributes 1/num_samples per collected sweep).  Only reachable through trlda_update_variables, like the
// reference's tests reach it; the parameter updates stay variational.
static int gibbs_variables(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows,
                           int64_t latents_cols, const trlda_params* params, double* theta_out, double* sstats_out) {
	if(latents && (latents_rows != m->K || latents_cols != docs->num_docs))
		return fail(m, TRLDA_ERR_ARG, "Initial theta has wrong dimensionality.");   // lda.cpp:228
	if(params->num_samples < 1 || params->burn_in < 0)
		return fail(m, TRLDA_ERR_ARG, "num_samples should be positive and burn_in non-negative.");
	if(m->nranks > 1)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "The Gibbs E-step is not sharded over GPUs.");
	TRY(upload_docs(m, docs));
	TRY(prepare_beta(m));
	const int64_t B = m->mb.docs.B;
	const size_t kb = sizeof(double) * (size_t) m->K * (size_t) B;
	std::vector<int64_t> occ((size_t) B + 1, 0);
	for(int64_t d = 0; d < B; ++d) {
		int64_t total = 0;
		for(int64_t j = docs->doc_ptr[d]; j < docs->doc_ptr[d + 1]; ++j)
			total += docs->counts[j];
		occ[(size_t) d + 1] = occ[(size_t) d] + total;
	}
	CUDA_TRY(m, m->gibbs_occ.ensure(sizeof(int64_t) * ((size_t) B + 1)));
	CUDA_TRY(m, m->gibbs_topics.ensure(sizeof(uint16_t) * (size_t) std::max<int64_t>(occ[(size_t) B], 1)));
	CUDA_TRY(m, m->sstats.ensure(kv_bytes(m)));
	CUDA_TRY(m, cudaMemcpyAsync(m->gibbs_occ.p, occ.data(), sizeof(int64_t) * ((size_t) B + 1), cudaMemcpyHostToDevice, m->stream));
	CUDA_TRY(m, cudaMemsetAsync(m->sstats.p, 0, kv_bytes(m), m->stream));
	if(latents && B) {
		CUDA_TRY(m, cudaMemcpyAsync(m->etheta.p, latents, kb, cudaMemcpyHostToDevice, m->stream));
		m->stats.h2d_bytes += kb;
	}
	{
		Launch l(m, KK_ESTEP);
		launch_gibbs(m->mb.docs, m->K, m->beta.p, m->beta_elem, m->d_alpha.as<double>(), latents ? m->etheta.as<double>() : nullptr,
		             m->gibbs_occ.as<int64_t>(), m->gibbs_topics.as<uint16_t>(), params->num_samples, params->burn_in,
		             current_seed() ^ (next_stream_id() * 0x9E3779B97F4A7C15ull), m->gamma.as<double>(), m->sstats.as<double>(),
		             m->stream);
	}
	TRY(check_launch(m, "gibbs"));
	m->gamma_valid = false;                      // the buffer holds theta, not a variational gamma
	if(theta_out && B) {
		CUDA_TRY(m, cudaMemcpyAsync(theta_out, m->gamma.p, kb, cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += kb;
	}
	if(sstats_out) {
		CUDA_TRY(m, cudaMemcpyAsync(sstats_out, m->sstats.p, kv_bytes(m), cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += kv_bytes(m);
	}
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));   // occ (host vector) must outlive its copy
	consume_injections(m);
	return TRLDA_OK;
}

int trlda_update_variables(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows,
                           int64_t latents_cols, const trlda_params* params, double* gamma_out, double* sstats_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(params->inference_method == TRLDA_INFERENCE_GIBBS)
		return gibbs_variables(m, docs, latents, latents_rows, latents_cols, params, gamma_out, sstats_out);
	if(latents && (latents_rows != m->K || latents_cols != docs->num_docs))
		return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");   // lda.cpp:166
	TRY(upload_docs(m, docs));
	TRY(prepare_beta(m));
	TRY(run_estep(m, latents ? GAMMA_HOST : GAMMA_FRESH, latents, params->max_iter_inference, params->threshold));
	if(sstats_out)
		TRY(run_scatter_dense(m));
	if(gamma_out && m->mb.docs.B) {
		CUDA_TRY(m, cudaMemcpyAsync(gamma_out, m->gamma.p, sizeof(double) * (size_t) m->K * m->mb.docs.B, cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += sizeof(double) * (size_t) m->K * m->mb.docs.B;
	}
	if(sstats_out) {
		CUDA_TRY(m, cudaMemcpyAsync(sstats_out, m->sstats.p, kv_bytes(m), cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += kv_bytes(m);
	}
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	// iteration statistics of this E-step
	if(m->mb.docs.B) {
		std::vector<int32_t> it(m->mb.docs.B);
		CUDA_TRY(m, cudaMemcpy(it.data(), m->iterations.p, sizeof(int32_t) * m->mb.docs.B, cudaMemcpyDeviceToHost));
		int64_t total = 0;
		for(int32_t v : it)
			total += v;
		m->stats.estep_doc_iterations = total;
	}
	consume_injections(m);
	return TRLDA_OK;
}

int trlda_update_parameters(trlda_model* m, const trlda_docs* docs, const trlda_params* params, double* result) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(upload_docs(m, docs));
	return update_resident(m, params, result);
}

int trlda_update_parameters_resident(trlda_model* m, const trlda_params* params, double* result) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(!m->docs_resident)
		return fail(m, TRLDA_ERR_ARG, "No minibatch resident on the device; call trlda_upload_docs first.");
	TRY(set_device(m));
	return update_resident(m, params, result);
}

int trlda_lower_bound(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows,
                      int64_t latents_cols, const trlda_params* params, int64_t num_documents, double* bound_out,
                      double* per_doc_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(params->inference_method != TRLDA_INFERENCE_VI)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device.");
	if(latents && (latents_rows != m->K || latents_cols != docs->num_docs))
		return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");
	TRY(upload_docs(m, docs));
	const int64_t B = m->mb.docs.B;
	if(m->kind == TRLDA_KIND_ONLINE && num_documents < 0)
		num_documents = m->num_documents;                                      // onlinelda.cpp:184-191
	const double factor = num_documents >= 0 ? (double) num_documents / (double) m->mb.global_B : 1.;   // lda.cpp:303-304
	TRY(prepare_beta(m));                                                      // also leaves rows / psi_rows of lambda
	TRY(run_estep(m, latents ? GAMMA_HOST : GAMMA_FRESH, latents, params->max_iter_inference, params->threshold));   // :307

	double lg_alpha = 0.0, asum = 0.0;
	for(int k = 0; k < m->K; ++k) {
		lg_alpha += lgamma(m->alpha[k]);
		asum += m->alpha[k];
	}
	const double alpha_const = lgamma(asum) - lg_alpha;                         // :355
	// per-document terms -> weight buffer is free after the E-step? keep it; use doc_stat for B values
	double* per_doc = m->doc_stat.as<double>();
	{
		Launch l(m, KK_ELBO);
		launch_elbo_docs(m->mb.docs, m->K, m->lambda(), m->psi_rows.as<double>(), m->d_alpha.as<double>(), alpha_const,
		                 m->gamma.as<double>(), per_doc, m->stream);
	}
	{
		Launch l(m, KK_ELBO);
		launch_elbo_beta(m->lambda(), m->psi_rows.as<double>(), m->K, m->V, m->eta, m->vpartials.as<double>(), m->stream);
	}
	double* sc = m->scalars.as<double>();
	{
		Launch l(m, KK_REDUCE);
		launch_sum(per_doc, B, sc + 16, sc, m->stream);
		launch_sum(m->vpartials.as<double>(), m->V, sc + 16 + 1024, sc + 1, m->stream);
		launch_lgamma_vector(m->rows.as<double>(), m->K, m->rows_stat.as<double>(), m->stream);
		launch_sum(m->rows_stat.as<double>(), m->K, sc + 16 + 2048, sc + 2, m->stream);
	}
	TRY(check_launch(m, "elbo"));
	TRY(allreduce(m, sc, 1, ncclDouble));                                      // documents are sharded; beta terms are replicated
	double h[3];
	TRY(read_back(m, sc, 3, h));
	double beta_terms = h[1];
	beta_terms -= (double) m->K * m->V * lgamma(m->eta);                        // :357
	beta_terms += m->K * lgamma(m->V * m->eta) - h[2];                          // :356
	if(bound_out)
		*bound_out = beta_terms + factor * h[0];
	if(per_doc_out && B) {
		CUDA_TRY(m, cudaMemcpy(per_doc_out, per_doc, sizeof(double) * B, cudaMemcpyDeviceToHost));
		m->stats.d2h_bytes += sizeof(double) * B;
	}
	consume_injections(m);
	return TRLDA_OK;
}

// checks a CSR like upload_docs does, sums its counts and copies it into the model's side buffers (ho_*), leaving the live
// minibatch alone
static int upload_side_docs(trlda_model* m, const trlda_docs* docs, DeviceDocs* out, int64_t* tokens) {
	if(!docs || docs->num_docs < 0 || (docs->num_docs > 0 && !docs->doc_ptr))
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");
	const int64_t B = docs->num_docs;
	const int64_t N = B ? docs->doc_ptr[B] : 0;
	if(B && docs->doc_ptr[0] != 0)
		return fail(m, TRLDA_ERR_ARG, "Document offsets must start at zero.");
	if(N < 0 || N > INT32_MAX)
		return fail(m, TRLDA_ERR_ARG, "Too many (word, count) pairs in one minibatch.");
	if(N > 0 && (!docs->word_ids || !docs->counts))
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");
	for(int64_t d = 0; d < B; ++d)
		if(docs->doc_ptr[d + 1] < docs->doc_ptr[d])
			return fail(m, TRLDA_ERR_ARG, "Document offsets must be non-decreasing.");
	int64_t total = 0;
	int bad = 0;
	for(int64_t i = 0; i < N; ++i) {
		total += docs->counts[i];
		bad |= (docs->word_ids[i] < 0) | (docs->word_ids[i] >= m->V) | ((docs->counts[i] < 0) << 1);
	}
	if(bad & 2)
		return fail(m, TRLDA_ERR_ARG, "Word counts should not be negative.");
	if(bad)
		return fail(m, TRLDA_ERR_ARG, "Word ID out of range.");
	CUDA_TRY(m, m->ho_doc_ptr.ensure(sizeof(int64_t) * (B + 1)));
	CUDA_TRY(m, m->ho_word_ids.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, m->ho_counts.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	if(B)
		CUDA_TRY(m, cudaMemcpyAsync(m->ho_doc_ptr.p, docs->doc_ptr, sizeof(int64_t) * (B + 1), cudaMemcpyHostToDevice, m->stream));
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(m->ho_word_ids.p, docs->word_ids, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
		CUDA_TRY(m, cudaMemcpyAsync(m->ho_counts.p, docs->counts, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
	}
	m->stats.h2d_bytes += (B ? sizeof(int64_t) * (B + 1) : 0) + sizeof(int32_t) * 2 * N;
	out->B = B;
	out->N = N;
	out->doc_ptr = m->ho_doc_ptr.as<int64_t>();
	out->word_ids = m->ho_word_ids.as<int32_t>();
	out->counts = m->ho_counts.as<int32_t>();
	*tokens = total;
	return TRLDA_OK;
}

int trlda_predictive_log_likelihood(trlda_model* m, const trlda_docs* observed, const trlda_docs* held_out, const double* latents,
                                    int latents_rows, int64_t latents_cols, const trlda_params* params, double* total_out,
                                    int64_t* tokens_out, double* per_doc_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(params->inference_method != TRLDA_INFERENCE_VI)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device.");
	if(m->lambda_sharded)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "predictive_log_likelihood: lambda is sharded over ranks.");
	if(!observed || !held_out)
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");
	if(latents && (latents_rows != m->K || latents_cols != observed->num_docs))
		return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");
	if(held_out->num_docs != observed->num_docs)
		return fail(m, TRLDA_ERR_ARG, "Observed and held-out documents differ in number.");
	TRY(set_device(m));
	DeviceDocs ho;
	int64_t tokens = 0;
	TRY(upload_side_docs(m, held_out, &ho, &tokens));
	// gamma of the observed part: the E-step of trlda_update_variables / trlda_lower_bound, with every route it has
	TRY(upload_docs(m, observed));
	TRY(prepare_beta(m));                                                      // also leaves rows = row sums of lambda
	TRY(run_estep(m, latents ? GAMMA_HOST : GAMMA_FRESH, latents, params->max_iter_inference, params->threshold));
	const int64_t B = m->mb.docs.B;
	double* per_doc = m->doc_stat.as<double>();                                // free after the E-step; holds >= B values
	double* sc = m->scalars.as<double>();
	{
		Launch l(m, KK_ELBO);
		launch_heldout_loglik(ho, m->K, m->lambda(), m->rows.as<double>(), m->gamma.as<double>(), per_doc, m->stream);
	}
	{
		Launch l(m, KK_REDUCE);
		launch_sum(per_doc, B, sc + 16, sc, m->stream);
	}
	TRY(check_launch(m, "heldout_loglik"));
	// the local total and token count, summed over ranks in one exchange (counts are exact in a double below 2^53)
	double* h = m->readback.as<double>();
	h[0] = (double) tokens;
	CUDA_TRY(m, cudaMemcpyAsync(sc + 1, h, sizeof(double), cudaMemcpyHostToDevice, m->stream));
	TRY(allreduce(m, sc, 2, ncclDouble));
	double r[2];
	TRY(read_back(m, sc, 2, r));
	if(total_out)
		*total_out = r[0];
	if(tokens_out)
		*tokens_out = (int64_t) r[1];
	if(per_doc_out && B) {
		CUDA_TRY(m, cudaMemcpy(per_doc_out, per_doc, sizeof(double) * B, cudaMemcpyDeviceToHost));
		m->stats.d2h_bytes += sizeof(double) * B;
	}
	consume_injections(m);
	return TRLDA_OK;
}

static const int kMaxWordTopics = 32;   // one warp lane per rank in k_word_topics_pairs

int trlda_word_topics(trlda_model* m, const trlda_docs* docs, const double* latents, int latents_rows, int64_t latents_cols,
                      const trlda_params* params, int n, int32_t* topics_out, double* probs_out, double* gamma_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(params->inference_method != TRLDA_INFERENCE_VI)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "Only variational inference ('VI') is implemented on the device.");
	if(m->lambda_sharded)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "word_topics: lambda is sharded over ranks.");
	if(n < 1 || n > kMaxWordTopics || n > m->K)
		return fail(m, TRLDA_ERR_ARG, "Number of topics per word must lie in [1, min(32, number of topics)].");
	if(!topics_out)
		return fail(m, TRLDA_ERR_ARG, "word_topics: no output buffer.");
	if(!docs)
		return fail(m, TRLDA_ERR_ARG, "Documents must be given in CSR form.");
	if(latents && (latents_rows != m->K || latents_cols != docs->num_docs))
		return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");
	// gamma exactly as trlda_update_variables fits it (upload_docs also checks the CSR)
	TRY(upload_docs(m, docs));
	TRY(prepare_beta(m));                                                      // also leaves psi_rows of lambda
	TRY(run_estep(m, latents ? GAMMA_HOST : GAMMA_FRESH, latents, params->max_iter_inference, params->threshold));
	const int K = m->K, V = m->V;
	const int64_t B = m->mb.docs.B, N = m->mb.docs.N;
	const int chunk = std::min(word_topics_chunk_words(K), V);
	CUDA_TRY(m, m->wt_len.ensure(sizeof(int32_t) * std::max<int64_t>(B, 1)));
	CUDA_TRY(m, m->wt_scratch.ensure(sizeof(int32_t) * global_csc_scratch_ints(B, N, 0, V)));
	CUDA_TRY(m, m->wt_word_ptr.ensure(sizeof(int32_t) * ((size_t) V + 1)));
	CUDA_TRY(m, m->wt_tok_doc.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, m->wt_tok_src.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, m->wt_table.ensure(sizeof(double) * (size_t) chunk * K));
	CUDA_TRY(m, m->wt_psi_gamma.ensure(sizeof(double) * (size_t) K * std::max<int64_t>(B, 1)));
	CUDA_TRY(m, m->wt_topics.ensure(sizeof(int32_t) * (size_t) std::max<int64_t>(N, 1) * n));
	if(probs_out)
		CUDA_TRY(m, m->wt_probs.ensure(sizeof(double) * (size_t) std::max<int64_t>(N, 1) * n));
	// the call's own word-sorted token list (a word's pairs in CSR order), built on the device by the builder of the
	// multi-GPU exchange with this rank's documents as the only segment.  The live minibatch's list is not used: on several
	// GPUs it covers the whole gathered minibatch.
	DeviceDocs wt = m->mb.docs;
	wt.word_ptr = m->wt_word_ptr.as<int32_t>();
	wt.tok_doc = m->wt_tok_doc.as<int32_t>();
	wt.tok_src = m->wt_tok_src.as<int32_t>();
	{
		Launch l(m, KK_MISC);
		launch_doc_lengths(wt.doc_ptr, B, B, m->wt_len.as<int32_t>(), m->stream);
		launch_global_csc(m->wt_len.as<int32_t>(), wt.word_ids, 1, B, N, 0, V, V, m->wt_scratch.as<int32_t>(),
		                  m->wt_word_ptr.as<int32_t>(), m->wt_tok_doc.as<int32_t>(), m->wt_tok_src.as<int32_t>(), m->stream);
	}
	double* psi_gamma = m->wt_psi_gamma.as<double>();
	// psi(gamma), in runs of whole documents that keep the element count in an int
	const int64_t run = std::max<int64_t>(1, INT_MAX / K);
	for(int64_t d0 = 0; d0 < B; d0 += run) {
		Launch l(m, KK_MISC);
		launch_psi_vector(m->gamma.as<double>() + d0 * K, (int) (std::min(run, B - d0) * K), psi_gamma + d0 * K, m->stream);
	}
	for(int w0 = 0; w0 < V && N > 0; w0 += chunk) {
		const int count = std::min(chunk, V - w0);
		{
			Launch l(m, KK_MISC);
			launch_word_topics_table(m->lambda(), K, w0, count, wt.word_ptr, m->psi_rows.as<double>(), m->wt_table.as<double>(),
			                         m->stream);
		}
		{
			Launch l(m, KK_MISC);
			launch_word_topics_pairs(wt, w0, w0 + count, m->wt_table.as<double>(), psi_gamma, K, n, m->wt_topics.as<int32_t>(),
			                         probs_out ? m->wt_probs.as<double>() : nullptr, m->stream);
		}
	}
	TRY(check_launch(m, "word_topics"));
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(topics_out, m->wt_topics.p, sizeof(int32_t) * (size_t) N * n, cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += sizeof(int32_t) * (size_t) N * n;
		if(probs_out) {
			CUDA_TRY(m, cudaMemcpyAsync(probs_out, m->wt_probs.p, sizeof(double) * (size_t) N * n, cudaMemcpyDeviceToHost, m->stream));
			m->stats.d2h_bytes += sizeof(double) * (size_t) N * n;
		}
	}
	if(gamma_out && B) {
		CUDA_TRY(m, cudaMemcpyAsync(gamma_out, m->gamma.p, sizeof(double) * (size_t) K * B, cudaMemcpyDeviceToHost, m->stream));
		m->stats.d2h_bytes += sizeof(double) * (size_t) K * B;
	}
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	consume_injections(m);
	return TRLDA_OK;
}

static const int kMaxTopWords = 32;   // one 32-bit mask per topic in k_cooccurrence, one warp lane per rank in the merge

int trlda_top_words(trlda_model* m, int n, int32_t* ids_out, double* prob_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(n < 1 || n > kMaxTopWords || n > m->V)
		return fail(m, TRLDA_ERR_ARG, "Number of top words must lie in [1, min(32, number of words)].");
	if(!ids_out)
		return fail(m, TRLDA_ERR_ARG, "top_words: no output buffer.");
	if(m->lambda_sharded)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "top_words: lambda is sharded over ranks.");
	TRY(set_device(m));
	const int K = m->K, V = m->V, chunks = top_words_chunks(K, V, n);
	const size_t listed = (size_t) K * n, cands = (size_t) chunks * listed;
	CUDA_TRY(m, m->topic_rows.ensure(sizeof(double) * K));
	CUDA_TRY(m, m->top_cand_v.ensure(sizeof(double) * cands));
	CUDA_TRY(m, m->top_cand_id.ensure(sizeof(int32_t) * cands));
	CUDA_TRY(m, m->top_ids.ensure(sizeof(int32_t) * listed));
	CUDA_TRY(m, m->top_prob.ensure(sizeof(double) * listed));
	TRY(compute_rows(m, m->lambda(), m->topic_rows.as<double>()));   // the row sums prepare_beta uses
	{
		Launch l(m, KK_MISC);
		launch_top_words_candidates(m->lambda(), K, K, V, 0, n, chunks, m->top_cand_v.as<double>(), m->top_cand_id.as<int32_t>(),
		                            m->stream);
	}
	{
		Launch l(m, KK_MISC);
		launch_top_words_merge(m->top_cand_v.as<double>(), m->top_cand_id.as<int32_t>(), m->topic_rows.as<double>(), K, n, chunks,
		                       m->top_ids.as<int32_t>(), m->top_prob.as<double>(), m->stream);
	}
	TRY(check_launch(m, "top_words"));
	CUDA_TRY(m, cudaMemcpyAsync(ids_out, m->top_ids.p, sizeof(int32_t) * listed, cudaMemcpyDeviceToHost, m->stream));
	if(prob_out)
		CUDA_TRY(m, cudaMemcpyAsync(prob_out, m->top_prob.p, sizeof(double) * listed, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += (sizeof(int32_t) + (prob_out ? sizeof(double) : 0)) * listed;
	return TRLDA_OK;
}

int trlda_cooccurrence(trlda_model* m, const trlda_docs* docs, const int32_t* ids, int n, int64_t* counts_out,
                       int64_t* num_docs_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(n < 1 || n > kMaxTopWords)
		return fail(m, TRLDA_ERR_ARG, "Number of top words must lie in [1, min(32, number of words)].");
	if(!ids || !counts_out)
		return fail(m, TRLDA_ERR_ARG, "cooccurrence: no top words or no output buffer.");
	const int K = m->K, V = m->V;
	// the inverse map: for every word, the (topic * 32 + rank) entries of the lists it is on
	std::vector<int32_t> map_ptr((size_t) V + 1, 0), map((size_t) K * n);
	for(int k = 0; k < K; ++k) {
		const int32_t* list = ids + (size_t) k * n;
		for(int i = 0; i < n; ++i) {
			if(list[i] < 0 || list[i] >= V)
				return fail(m, TRLDA_ERR_ARG, "Word ID out of range.");
			for(int j = 0; j < i; ++j)
				if(list[j] == list[i])
					return fail(m, TRLDA_ERR_ARG, "Top words of a topic must be distinct.");
			++map_ptr[(size_t) list[i] + 1];
		}
	}
	for(int w = 0; w < V; ++w)
		map_ptr[(size_t) w + 1] += map_ptr[w];
	{
		std::vector<int32_t> next(map_ptr.begin(), map_ptr.end() - 1);
		for(int k = 0; k < K; ++k)
			for(int i = 0; i < n; ++i)
				map[next[ids[(size_t) k * n + i]]++] = k * kMaxTopWords + i;
	}
	TRY(set_device(m));
	TRY(ensure_small(m));
	DeviceDocs d;
	int64_t tokens = 0;
	TRY(upload_side_docs(m, docs, &d, &tokens));
	const size_t cells = (size_t) K * n * n;
	CUDA_TRY(m, m->co_map_ptr.ensure(sizeof(int32_t) * map_ptr.size()));
	CUDA_TRY(m, m->co_map.ensure(sizeof(int32_t) * map.size()));
	CUDA_TRY(m, m->co_counts.ensure(sizeof(int64_t) * (cells + 1)));    // the counters, then the document count
	CUDA_TRY(m, cudaMemcpyAsync(m->co_map_ptr.p, map_ptr.data(), sizeof(int32_t) * map_ptr.size(), cudaMemcpyHostToDevice, m->stream));
	CUDA_TRY(m, cudaMemcpyAsync(m->co_map.p, map.data(), sizeof(int32_t) * map.size(), cudaMemcpyHostToDevice, m->stream));
	m->stats.h2d_bytes += sizeof(int32_t) * (map_ptr.size() + map.size());
	CUDA_TRY(m, cudaMemsetAsync(m->co_counts.p, 0, sizeof(int64_t) * cells, m->stream));
	int64_t* h = m->readback.as<int64_t>();
	h[0] = d.B;
	CUDA_TRY(m, cudaMemcpyAsync(m->co_counts.as<int64_t>() + cells, h, sizeof(int64_t), cudaMemcpyHostToDevice, m->stream));
	{
		Launch l(m, KK_MISC);
		launch_cooccurrence(d, K, n, m->co_map_ptr.as<int32_t>(), m->co_map.as<int32_t>(),
		                    reinterpret_cast<unsigned long long*>(m->co_counts.p), m->stream);
	}
	TRY(check_launch(m, "cooccurrence"));
	// counters and document count summed over ranks in one exchange; integers, so the sum is exact in any order
	TRY(allreduce(m, m->co_counts.p, cells + 1, ncclInt64));
	CUDA_TRY(m, cudaMemcpyAsync(counts_out, m->co_counts.p, sizeof(int64_t) * cells, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaMemcpyAsync(h, m->co_counts.as<int64_t>() + cells, sizeof(int64_t), cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));   // also: the host vectors of the inverse map outlive their copies
	m->stats.d2h_bytes += sizeof(int64_t) * (cells + 1);
	if(num_docs_out)
		*num_docs_out = h[0];
	return TRLDA_OK;
}

// trlda_topic_distances with both mutexes held; b is m itself or the other model
static int topic_distances(trlda_model* m, trlda_model* b, int metric, double* out) {
	if(metric != TRLDA_DISTANCE_HELLINGER && metric != TRLDA_DISTANCE_KL)
		return fail(m, TRLDA_ERR_ARG, "Unknown distance metric.");
	if(!out)
		return fail(m, TRLDA_ERR_ARG, "topic_distances: no output buffer.");
	if(b->V != m->V)
		return fail(m, TRLDA_ERR_ARG, "The two models must have the same number of words.");
	if(b->device != m->device)
		return fail(m, TRLDA_ERR_ARG, "The two models must be on the same device.");
	if(m->lambda_sharded || b->lambda_sharded)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "topic_distances: lambda is sharded over ranks.");
	TRY(set_device(m));
	TRY(ensure_small(m));
	const bool self = b == m, kl = metric == TRLDA_DISTANCE_KL;
	const int KA = m->K, KB = b->K, V = m->V;
	const DistancePlan plan = distance_plan(KA, KB, V, self && !kl);    // a self-comparison under Hellinger: X = Y
	const int max_parts = distance_entropy_parts(plan.chunk);
	CUDA_TRY(m, m->topic_rows.ensure(sizeof(double) * KA));
	CUDA_TRY(m, m->dist_rows.ensure(sizeof(double) * KB));
	CUDA_TRY(m, m->dist_x.ensure(sizeof(double) * plan.chunk * plan.ld_x));
	if(!(self && !kl))
		CUDA_TRY(m, m->dist_y.ensure(sizeof(double) * plan.chunk * plan.ld_y));
	if(kl) {
		CUDA_TRY(m, m->dist_hpart.ensure(sizeof(double) * max_parts * plan.ld_x));
		CUDA_TRY(m, m->dist_h.ensure(sizeof(double) * KA));
	}
	CUDA_TRY(m, m->dist_partial.ensure(sizeof(double) * plan.splits * plan.ld_x * plan.ld_y));
	CUDA_TRY(m, m->dist_out.ensure(sizeof(double) * KA * KB));
	CUDA_TRY(m, m->dist_flag.ensure(sizeof(int)));
	CUDA_TRY(m, cudaMemsetAsync(m->dist_flag.p, 0, sizeof(int), m->stream));
	if(!self) {
		// the other model's lambda is read on this model's stream: after whatever its own stream has queued
		CUDA_TRY(m, cudaEventRecord(m->other_ready, b->stream));
		CUDA_TRY(m, cudaStreamWaitEvent(m->stream, m->other_ready, 0));
	}
	double* rows_a = m->topic_rows.as<double>();
	double* rows_b = self ? rows_a : m->dist_rows.as<double>();
	TRY(compute_rows(m, m->lambda(), rows_a));            // the row sums of prepare_beta and trlda_top_words
	if(!self)
		TRY(compute_rows(m, b->lambda(), rows_b, KB));
	double* x = m->dist_x.as<double>();
	double* y = self && !kl ? x : m->dist_y.as<double>();
	const int op_x = kl ? DIST_OP_IDENTITY : DIST_OP_SQRT, op_y = kl ? DIST_OP_LOG : DIST_OP_SQRT;
	int* flag = m->dist_flag.as<int>();
	double* hpart = kl ? m->dist_hpart.as<double>() : nullptr;
	for(int w0 = 0; w0 < V; w0 += plan.chunk) {
		const bool first = w0 == 0;
		const int words = distance_chunk_words(plan, V - w0);
		{
			Launch l(m, KK_MISC);   // f(P_A), and g(P_A) too for a self-comparison under KL
			launch_distance_prepare(m->lambda(), KA, V, plan.ld_x, w0, words, rows_a, op_x, x, self && kl ? op_y : DIST_OP_NONE,
			                        self && kl ? y : nullptr, hpart, flag, m->stream);
		}
		if(!self) {
			Launch l(m, KK_MISC);
			launch_distance_prepare(b->lambda(), KB, V, plan.ld_y, w0, words, rows_b, op_y, y, DIST_OP_NONE, nullptr, nullptr,
			                        flag, m->stream);
		}
		if(kl) {
			Launch l(m, KK_MISC);
			launch_distance_entropy(hpart, distance_entropy_parts(words), KA, plan.ld_x, first, m->dist_h.as<double>(), m->stream);
		}
		{
			Launch l(m, KK_MISC);
			launch_distance_product(plan, x, y, words, first, m->dist_partial.as<double>(), m->stream);
		}
	}
	{
		Launch l(m, KK_MISC);
		launch_distance_finish(plan, m->dist_partial.as<double>(), KA, KB, metric, kl ? m->dist_h.as<double>() : nullptr,
		                       m->dist_out.as<double>(), m->stream);
	}
	TRY(check_launch(m, "topic_distances"));
	int* h = m->readback.as<int>();
	CUDA_TRY(m, cudaMemcpyAsync(h, flag, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	const int bad = h[0];
	if(bad & DIST_BAD_NEGATIVE)
		return fail(m, TRLDA_ERR_ARG, "topic_distances: lambda has a negative entry.");
	if(bad & DIST_BAD_EMPTY_ROW)
		return fail(m, TRLDA_ERR_ARG, "topic_distances: a topic's lambda sums to zero.");
	if(bad & DIST_BAD_ZERO)
		return fail(m, TRLDA_ERR_ARG, "topic_distances: the Kullback-Leibler distance needs a positive lambda in the second model.");
	CUDA_TRY(m, cudaMemcpyAsync(out, m->dist_out.p, sizeof(double) * KA * KB, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += sizeof(double) * KA * KB + sizeof(int);
	return TRLDA_OK;
}

int trlda_topic_distances(trlda_model* m, trlda_model* other, int metric, double* out) {
	if(!other || other == m) {
		std::scoped_lock lock__(m->mu);
		return topic_distances(m, m, metric, out);
	}
	std::scoped_lock lock__(m->mu, other->mu);   // std::lock's deadlock avoidance, whatever order other callers use
	return topic_distances(m, other, metric, out);
}

// ---- similar documents ----------------------------------------------------------------------------------------------
static const int kMaxNeighbors = 32;               // one warp lane per rank in the merge
static const size_t kSimStage = 256u << 20;        // bytes of raw gamma on the device at a time
static const size_t kSimAffinity = 256u << 20;     // bytes of one affinity block (queries x documents), at most
static const int kSimQueryBlock = 8192;            // queries per block of the product path
// at most this many queries take the streaming path: it reads the index once per group of 8 queries (1.45 ms a group at
// K = 1000, D = 2^20 on a B200), the product path costs the same (11.4 ms) for any Q up to its 128-query tile (DESIGN.md §4.2)
static const int kSimStreamMax = 56;

static const char* kSimBadGamma = "Gamma must be finite and non-negative, with a positive sum in every column.";

// sqrt(theta) of the cols columns of host gamma (K x cols) into out (element (k, c) at k * ld + c), staged through the
// device in blocks of columns; the prepare pass raises m->sim_flag for bad columns
static int prepare_columns(trlda_model* m, const double* gamma, int64_t cols, int64_t ld, double* out, DevBuf& stage) {
	const int K = m->K;
	const int64_t block = std::max<int64_t>(1, std::min<int64_t>(cols, (int64_t) (kSimStage / (sizeof(double) * K))));
	CUDA_TRY(m, stage.ensure(sizeof(double) * K * block));
	for(int64_t c0 = 0; c0 < cols; c0 += block) {
		const int64_t nc = std::min(block, cols - c0);
		CUDA_TRY(m, cudaMemcpyAsync(stage.p, gamma + c0 * K, sizeof(double) * K * nc, cudaMemcpyHostToDevice, m->stream));
		m->stats.h2d_bytes += sizeof(double) * K * nc;
		Launch l(m, KK_MISC);
		launch_similar_prepare(stage.as<double>(), K, (int) nc, ld, out + c0, m->sim_flag.as<int>(), m->stream);
	}
	return TRLDA_OK;
}

// the prepare pass's flag, read back (the stream is synchronised)
static int read_flag(trlda_model* m, int* bad) {
	int* h = m->readback.as<int>();
	CUDA_TRY(m, cudaMemcpyAsync(h, m->sim_flag.p, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += sizeof(int);
	*bad = h[0];
	return TRLDA_OK;
}

static int index_documents(trlda_model* m, const double* gamma, int rows, int64_t cols) {
	if(rows != m->K || cols < 0 || (cols > 0 && !gamma))
		return fail(m, TRLDA_ERR_ARG, "Gamma has wrong dimensionality.");
	if(cols > INT32_MAX)
		return fail(m, TRLDA_ERR_ARG, "Too many documents to index.");
	if(cols == 0)
		return TRLDA_OK;
	TRY(ensure_small(m));
	const int64_t ld = similar_ld(cols);
	const size_t bytes = sizeof(double) * (size_t) similar_rows(m->K) * ld;
	CUDA_TRY(m, m->sim_index.ensure(bytes));
	CUDA_TRY(m, m->sim_flag.ensure(sizeof(int)));
	CUDA_TRY(m, cudaMemsetAsync(m->sim_index.p, 0, bytes, m->stream));
	CUDA_TRY(m, cudaMemsetAsync(m->sim_flag.p, 0, sizeof(int), m->stream));
	DevBuf stage;   // freed on return: only the index stays
	TRY(prepare_columns(m, gamma, cols, ld, m->sim_index.as<double>(), stage));
	TRY(check_launch(m, "index_documents"));
	int bad = 0;
	TRY(read_flag(m, &bad));
	if(bad)
		return fail(m, TRLDA_ERR_ARG, kSimBadGamma);
	m->sim_docs = cols;
	m->sim_ld = ld;
	return TRLDA_OK;
}

int trlda_index_documents(trlda_model* m, const double* gamma, int rows, int64_t cols) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	// the old index goes first, so that the two never take memory together, and a failure leaves no index
	m->sim_index.release();
	m->sim_docs = m->sim_ld = 0;
	const int status = index_documents(m, gamma, rows, cols);
	if(status != TRLDA_OK || m->sim_docs == 0) {
		m->sim_index.release();
		m->sim_docs = m->sim_ld = 0;
	}
	return status;
}

int trlda_similar_documents(trlda_model* m, const double* gamma, int rows, int64_t cols, int n, int64_t* ids_out,
                            double* dist_out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(rows != m->K || cols < 0 || (cols > 0 && !gamma))
		return fail(m, TRLDA_ERR_ARG, "Gamma has wrong dimensionality.");
	if(m->sim_docs == 0)
		return fail(m, TRLDA_ERR_ARG, "similar_documents: no documents are indexed.");
	if(n < 1 || n > kMaxNeighbors || n > m->sim_docs)
		return fail(m, TRLDA_ERR_ARG, "Number of neighbors must lie in [1, min(32, number of indexed documents)].");
	if(!ids_out)
		return fail(m, TRLDA_ERR_ARG, "similar_documents: no output buffer.");
	if(cols == 0)
		return TRLDA_OK;
	TRY(set_device(m));
	TRY(ensure_small(m));
	const int K = m->K, kp = similar_rows(K), D = (int) m->sim_docs;
	const int64_t Q = cols, ld = m->sim_ld;
	const char* env = getenv("TRLDA_SIMILAR_STREAM_MAX");   // measurement knob for the crossover of the two paths
	const int stream_max = env ? std::max(0, std::min(atoi(env), kSimQueryBlock)) : kSimStreamMax;
	const bool streaming = Q <= stream_max;
	// streaming: every query in one block, affinity rows = queries; product: blocks of kSimQueryBlock, rows padded to the tile
	const int qmax = (int) std::min<int64_t>(Q, streaming ? stream_max : kSimQueryBlock);
	const int ldq_max = (int) similar_ld(qmax);
	const int lda_max = streaming ? qmax : ldq_max;
	const int64_t dblock = std::min<int64_t>(similar_ld(D), std::max<int64_t>(128, (int64_t) (kSimAffinity / (sizeof(double) * lda_max)) / 128 * 128));
	// the top n of every query over an affinity block's chunks; many chunks are merged in two levels, G groups of P chunks
	// (chunk p * G + g is chunk p of group g, so group g's lists are rows g * qb + q of a G * qb-row merge)
	auto chunking = [&](int qb, int nd, int* groups) {
		int chunks = top_words_chunks(qb, nd, n);
		*groups = 1;
		if(chunks > 32) {
			*groups = (int) std::ceil(std::sqrt((double) chunks));
			chunks = (chunks + *groups - 1) / *groups * *groups;
		}
		return chunks;
	};
	int groups = 1;
	const int nd_max = (int) std::min<int64_t>(dblock, D), q_last = (int) (Q - (Q - 1) / qmax * qmax);
	const size_t cands = std::max((size_t) chunking(qmax, nd_max, &groups) * qmax, (size_t) chunking(q_last, nd_max, &groups) * q_last) * n;
	CUDA_TRY(m, m->sim_query.ensure(sizeof(double) * (size_t) kp * ldq_max));
	CUDA_TRY(m, m->sim_aff.ensure(sizeof(double) * (size_t) lda_max * dblock));
	CUDA_TRY(m, m->sim_cand_v.ensure(sizeof(double) * cands));
	CUDA_TRY(m, m->sim_cand_id.ensure(sizeof(int32_t) * cands));
	CUDA_TRY(m, m->sim_merge_v.ensure(sizeof(double) * cands));
	CUDA_TRY(m, m->sim_merge_id.ensure(sizeof(int32_t) * cands));
	CUDA_TRY(m, m->sim_res_v.ensure(sizeof(double) * (size_t) Q * n));
	CUDA_TRY(m, m->sim_res_id.ensure(sizeof(int32_t) * (size_t) Q * n));
	CUDA_TRY(m, m->sim_flag.ensure(sizeof(int)));
	CUDA_TRY(m, cudaMemsetAsync(m->sim_flag.p, 0, sizeof(int), m->stream));
	DevBuf stage;
	double* aff = m->sim_aff.as<double>();
	for(int64_t q0 = 0; q0 < Q; q0 += qmax) {
		const int qb = (int) std::min<int64_t>(qmax, Q - q0);
		const int ldq = (int) similar_ld(qb), lda = streaming ? qb : ldq;
		double* run_v = m->sim_res_v.as<double>() + q0 * n;
		int32_t* run_id = m->sim_res_id.as<int32_t>() + q0 * n;
		CUDA_TRY(m, cudaMemsetAsync(m->sim_query.p, 0, sizeof(double) * (size_t) kp * ldq, m->stream));
		TRY(prepare_columns(m, gamma + q0 * K, qb, ldq, m->sim_query.as<double>(), stage));
		for(int64_t d0 = 0; d0 < D; d0 += dblock) {
			const int nd = (int) std::min<int64_t>(dblock, D - d0);
			const double* index = m->sim_index.as<double>() + d0;
			{
				Launch l(m, KK_MISC);
				if(streaming)
					launch_similar_stream(index, ld, K, nd, m->sim_query.as<double>(), ldq, qb, aff, lda, m->stream);
				else
					launch_distance_product(m->sim_query.as<double>(), ldq, index, ld, (int) similar_ld(nd), 1, kp, true, aff, m->stream);
			}
			int chunks = chunking(qb, nd, &groups);
			{
				Launch l(m, KK_MISC);
				launch_top_words_candidates(aff, qb, lda, nd, (int) d0, n, chunks, m->sim_cand_v.as<double>(), m->sim_cand_id.as<int32_t>(),
				                            m->stream);
			}
			const double* src_v = m->sim_cand_v.as<double>();
			const int32_t* src_id = m->sim_cand_id.as<int32_t>();
			if(groups > 1) {
				Launch l(m, KK_MISC);
				launch_top_n_merge(src_v, src_id, groups * qb, n, chunks / groups, nullptr, nullptr, false, m->sim_merge_id.as<int32_t>(),
				                   m->sim_merge_v.as<double>(), m->stream);
				src_v = m->sim_merge_v.as<double>();
				src_id = m->sim_merge_id.as<int32_t>();
				chunks = groups;
			}
			{
				Launch l(m, KK_MISC);   // into the running list; the last block turns C into the distance
				launch_top_n_merge(src_v, src_id, qb, n, chunks, d0 > 0 ? run_v : nullptr, d0 > 0 ? run_id : nullptr, d0 + nd >= D,
				                   run_id, run_v, m->stream);
			}
		}
	}
	TRY(check_launch(m, "similar_documents"));
	int bad = 0;
	TRY(read_flag(m, &bad));
	if(bad)
		return fail(m, TRLDA_ERR_ARG, kSimBadGamma);
	const size_t listed = (size_t) Q * n;
	CUDA_TRY(m, m->readback.ensure(sizeof(int32_t) * listed));
	int32_t* h = m->readback.as<int32_t>();
	CUDA_TRY(m, cudaMemcpyAsync(h, m->sim_res_id.p, sizeof(int32_t) * listed, cudaMemcpyDeviceToHost, m->stream));
	if(dist_out)
		CUDA_TRY(m, cudaMemcpyAsync(dist_out, m->sim_res_v.p, sizeof(double) * listed, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += (sizeof(int32_t) + (dist_out ? sizeof(double) : 0)) * listed;
	for(size_t i = 0; i < listed; ++i)
		ids_out[i] = h[i];
	return TRLDA_OK;
}

int trlda_debug_global_csc(trlda_model* m, const int32_t* len, const int32_t* ids, int ranks, int64_t max_docs, int64_t max_pairs,
                           int v0, int v1, int32_t* word_ptr, int32_t* tok_doc, int32_t* tok_src) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	if(!len || !ids || !word_ptr || !tok_doc || !tok_src || ranks < 1 || max_docs < 0 || max_pairs < 0 || v0 < 0 || v1 < v0 || v1 > m->V ||
	   (int64_t) ranks * max_pairs > INT32_MAX)
		return fail(m, TRLDA_ERR_ARG, "debug_global_csc: bad arguments.");
	const int64_t B = (int64_t) ranks * max_docs, N = (int64_t) ranks * max_pairs;
	DevBuf d_len, d_ids, d_wptr, d_tdoc, d_tsrc, d_scratch;
	CUDA_TRY(m, d_len.ensure(sizeof(int32_t) * std::max<int64_t>(B, 1)));
	CUDA_TRY(m, d_ids.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, d_wptr.ensure(sizeof(int32_t) * ((size_t) m->V + 1)));
	CUDA_TRY(m, d_tdoc.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, d_tsrc.ensure(sizeof(int32_t) * std::max<int64_t>(N, 1)));
	CUDA_TRY(m, d_scratch.ensure(sizeof(int32_t) * global_csc_scratch_ints(B, N, v0, v1)));
	if(B)
		CUDA_TRY(m, cudaMemcpyAsync(d_len.p, len, sizeof(int32_t) * B, cudaMemcpyHostToDevice, m->stream));
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(d_ids.p, ids, sizeof(int32_t) * N, cudaMemcpyHostToDevice, m->stream));
		CUDA_TRY(m, cudaMemsetAsync(d_tdoc.p, 0xff, sizeof(int32_t) * N, m->stream));
		CUDA_TRY(m, cudaMemsetAsync(d_tsrc.p, 0xff, sizeof(int32_t) * N, m->stream));
	}
	launch_global_csc(d_len.as<int32_t>(), d_ids.as<int32_t>(), ranks, max_docs, max_pairs, v0, v1, m->V, d_scratch.as<int32_t>(),
	                  d_wptr.as<int32_t>(), d_tdoc.as<int32_t>(), d_tsrc.as<int32_t>(), m->stream);
	TRY(check_launch(m, "debug_global_csc"));
	CUDA_TRY(m, cudaMemcpyAsync(word_ptr, d_wptr.p, sizeof(int32_t) * ((size_t) m->V + 1), cudaMemcpyDeviceToHost, m->stream));
	if(N) {
		CUDA_TRY(m, cudaMemcpyAsync(tok_doc, d_tdoc.p, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, m->stream));
		CUDA_TRY(m, cudaMemcpyAsync(tok_src, d_tsrc.p, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, m->stream));
	}
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	return TRLDA_OK;
}

int trlda_sample(trlda_model* m, int64_t num_documents, double length, int collapse, trlda_docs* out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	if(!out || num_documents < 0 || !(length >= 0.0) || length > 1e6)
		return fail(m, TRLDA_ERR_ARG, "sample: num_documents should be non-negative and length in [0, 1e6].");
	if(m->lambda_sharded)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "sample: lambda is sharded over ranks.");
	const int64_t B = num_documents;
	const int cap = sample_capacity(length);
	if(sample_smem_bytes(m->K, cap) > (size_t) m->smem_optin)
		return fail(m, TRLDA_ERR_UNSUPPORTED, "sample: too many topics / too long documents for the sampler's shared memory.");
	const uint64_t seed = current_seed() ^ (next_stream_id() * 0x9E3779B97F4A7C15ull);
	CUDA_TRY(m, m->sample_cdf.ensure(kv_bytes(m)));
	CUDA_TRY(m, m->sample_tokens.ensure(sizeof(int32_t) * (size_t) std::max<int64_t>(B, 1) * cap));
	CUDA_TRY(m, m->sample_counts.ensure(sizeof(int32_t) * (size_t) std::max<int64_t>(B, 1) * cap));
	CUDA_TRY(m, m->sample_lengths.ensure(sizeof(int32_t) * (size_t) std::max<int64_t>(B, 1)));
	TRY(upload_alpha(m));
	{
		Launch l(m, KK_RNG);
		launch_sample_beta(m->lambda(), m->K, m->V, seed, m->sample_cdf.as<double>(), m->stream);
	}
	{
		Launch l(m, KK_RNG);
		if(launch_sample_docs(m->sample_cdf.as<double>(), m->d_alpha.as<double>(), m->K, m->V, B, length, cap, collapse != 0, seed,
		                      m->sample_tokens.as<int32_t>(), m->sample_counts.as<int32_t>(), m->sample_lengths.as<int32_t>(), m->stream) != 0)
			return fail(m, TRLDA_ERR_CUDA, "sample: the kernel could not be configured.");
	}
	TRY(check_launch(m, "sample"));
	std::vector<int32_t> lengths((size_t) B), tokens((size_t) B * cap), counts(collapse ? (size_t) B * cap : 0);
	if(B) {
		CUDA_TRY(m, cudaMemcpyAsync(lengths.data(), m->sample_lengths.p, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, m->stream));
		CUDA_TRY(m, cudaMemcpyAsync(tokens.data(), m->sample_tokens.p, sizeof(int32_t) * (size_t) B * cap, cudaMemcpyDeviceToHost, m->stream));
		if(collapse)
			CUDA_TRY(m, cudaMemcpyAsync(counts.data(), m->sample_counts.p, sizeof(int32_t) * (size_t) B * cap, cudaMemcpyDeviceToHost, m->stream));
	}
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->stats.d2h_bytes += sizeof(int32_t) * (size_t) B * cap * (collapse ? 2 : 1);
	m->sample_ptr.assign((size_t) B + 1, 0);
	for(int64_t d = 0; d < B; ++d)
		m->sample_ptr[d + 1] = m->sample_ptr[d] + lengths[d];
	const int64_t N = m->sample_ptr[B];
	m->sample_ids.resize((size_t) N);
	m->sample_cts.resize((size_t) N);
	for(int64_t d = 0; d < B; ++d) {
		const int64_t o = m->sample_ptr[d];
		for(int j = 0; j < lengths[d]; ++j) {
			m->sample_ids[o + j] = tokens[(size_t) d * cap + j];
			m->sample_cts[o + j] = collapse ? counts[(size_t) d * cap + j] : 1;
		}
	}
	out->num_docs = B;
	out->doc_ptr = m->sample_ptr.data();
	out->word_ids = m->sample_ids.data();
	out->counts = m->sample_cts.data();
	return TRLDA_OK;
}

int trlda_inject_initial_gamma(trlda_model* m, const double* gamma0, int rows, int64_t cols) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(!gamma0 || rows != m->K || cols < 0)
		return fail(m, TRLDA_ERR_ARG, "Initial gamma has wrong dimensionality.");
	m->inj_gamma.assign(gamma0, gamma0 + (size_t) rows * cols);
	m->inj_gamma_cols = cols;
	return TRLDA_OK;
}

int trlda_inject_initial_lambda(trlda_model* m, const double* lambda, int rows, int cols) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(!lambda || rows != m->K || cols != m->V)
		return fail(m, TRLDA_ERR_ARG, "Lambda has wrong dimensionality.");
	m->inj_lambda.assign(lambda, lambda + (size_t) rows * cols);
	return TRLDA_OK;
}

int trlda_comm_unique_id(void* id_out) {
	if(!nccl_api().ok)
		return fail(nullptr, TRLDA_ERR_CUDA, "libnccl.so.2 could not be loaded.");
	static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
	ncclUniqueId id;
	ncclResult_t r = nccl_api().GetUniqueId(&id);
	if(r != ncclSuccess)
		return fail(nullptr, TRLDA_ERR_CUDA, std::string("NCCL error: ") + nccl_api().GetErrorString(r));
	memcpy(id_out, &id, sizeof(id));
	return TRLDA_OK;
}

int trlda_comm_init(trlda_model* m, const void* id_bytes, int rank, int nranks) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	if(nranks < 1 || rank < 0 || rank >= nranks)
		return fail(m, TRLDA_ERR_ARG, "Invalid rank / world size.");
	if(nranks == 1)
		return TRLDA_OK;
	if(!nccl_api().ok)
		return fail(m, TRLDA_ERR_CUDA, "libnccl.so.2 could not be loaded.");
	TRY(set_device(m));
	ncclUniqueId id;
	memcpy(&id, id_bytes, sizeof(id));
	NCCL_TRY(m, nccl_api().CommInitRank(&m->comm, nranks, id, rank));
	m->rank = rank;
	m->nranks = nranks;
	if(const char* mode = getenv("TRLDA_MULTI_GPU")) {
		m->use_peer = strcmp(mode, "allreduce") != 0;
		m->use_gather = strcmp(mode, "gather") == 0;
	}
	if(!m->use_peer || nranks > TRLDA_MAX_RANKS)
		return TRLDA_OK;

	// Map every rank's sstats / beta / lambda buffers into this process (cudaIpc over NVLink) for the fused
	// reduce-scatter + M-step + all-gather kernel.  The four handles travel through the communicator itself.
	TRY(ensure_beta(m));
	TRY(ensure_small(m));
	CUDA_TRY(m, m->lam[1 - m->cur].ensure(kv_bytes(m)));
	// mixed mode exchanges the per-rank partial statistics rounded to float32 (they are summed in float64)
	m->peer_sstats_elem = (m->beta_elem == 4 && m->K % 4 == 0) ? 4 : 8;
	// receive buffer for the pushed partial columns: [nranks][shard_cap][K]
	m->peer_shard_cap = (m->V + nranks - 1) / nranks + 1;
	CUDA_TRY(m, m->sstats32.ensure((size_t) nranks * m->peer_shard_cap * m->K * m->peer_sstats_elem));
	void* mine[4] = {m->sstats32.p, m->beta.p, m->lam[0].p, m->lam[1].p};
	std::vector<cudaIpcMemHandle_t> handles((size_t) 4 * nranks);
	cudaIpcMemHandle_t local[4];
	for(int i = 0; i < 4; ++i)
		CUDA_TRY(m, cudaIpcGetMemHandle(&local[i], mine[i]));
	DevBuf send, recv;
	CUDA_TRY(m, send.ensure(sizeof(local)));
	CUDA_TRY(m, recv.ensure(sizeof(local) * nranks));
	CUDA_TRY(m, cudaMemcpyAsync(send.p, local, sizeof(local), cudaMemcpyHostToDevice, m->stream));
	NCCL_TRY(m, nccl_api().AllGather(send.p, recv.p, sizeof(local), ncclUint8, m->comm, m->stream));
	CUDA_TRY(m, cudaMemcpyAsync(handles.data(), recv.p, sizeof(local) * nranks, cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	bool ok = true;
	for(int r = 0; r < nranks && ok; ++r) {
		void* ptrs[4];
		for(int i = 0; i < 4; ++i) {
			if(r == rank) {
				ptrs[i] = mine[i];
			} else if(cudaIpcOpenMemHandle(&ptrs[i], handles[(size_t) 4 * r + i], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess) {
				m->peer_opened.push_back(ptrs[i]);
			} else {
				cudaGetLastError();
				ok = false;
				break;
			}
		}
		if(ok) {
			m->peer_sstats[r] = ptrs[0];
			m->peer_beta[r] = ptrs[1];
			m->peer_lam[0][r] = ptrs[2];
			m->peer_lam[1][r] = ptrs[3];
		}
	}
	// every rank must take the same path: agree on success
	double* flag = m->scalars.as<double>() + 4001;
	const double mine_ok = ok ? 0.0 : 1.0;
	CUDA_TRY(m, cudaMemcpyAsync(flag, &mine_ok, sizeof(double), cudaMemcpyHostToDevice, m->stream));
	TRY(allreduce(m, flag, 1, ncclDouble));
	double failures = 0.0;
	CUDA_TRY(m, cudaMemcpyAsync(&failures, flag, sizeof(double), cudaMemcpyDeviceToHost, m->stream));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	m->peer_ready = failures == 0.0;
	return TRLDA_OK;
}

int trlda_comm_size(const trlda_model* m) { return m->nranks; }

void* trlda_stream(trlda_model* m) { return m->stream; }

int trlda_synchronize(trlda_model* m) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	return TRLDA_OK;
}

int trlda_set_profiling(trlda_model* m, int on) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	m->profiling = on != 0;
	return TRLDA_OK;
}

int trlda_get_stats(trlda_model* m, trlda_stats* out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	collect_spans(m);
	// inner-iteration total of the most recent E-step
	if(m->gamma_valid && m->mb.docs.B) {
		std::vector<int32_t> it(m->mb.docs.B);
		CUDA_TRY(m, cudaMemcpy(it.data(), m->iterations.p, sizeof(int32_t) * m->mb.docs.B, cudaMemcpyDeviceToHost));
		int64_t total = 0;
		for(int32_t v : it)
			total += v;
		m->stats.estep_doc_iterations = total;
		m->stats.estep_docs = m->mb.docs.B;
	}
	if(m->sweeps.p) {
		unsigned long long total = 0;
		CUDA_TRY(m, cudaMemcpy(&total, m->sweeps.p, sizeof(total), cudaMemcpyDeviceToHost));
		m->stats.estep_sweeps = (int64_t) total;
	}
	*out = m->stats;
	return TRLDA_OK;
}

int trlda_reset_stats(trlda_model* m) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	CUDA_TRY(m, cudaStreamSynchronize(m->stream));
	collect_spans(m);
	m->stats = trlda_stats{};
	if(m->sweeps.p)
		CUDA_TRY(m, cudaMemset(m->sweeps.p, 0, sizeof(unsigned long long)));
	return TRLDA_OK;
}

int trlda_get_row_sums(trlda_model* m, double* out) {
	std::lock_guard<std::recursive_mutex> lock__(m->mu);
	TRY(set_device(m));
	TRY(ensure_small(m));
	TRY(compute_rows(m, m->lambda(), m->rows_stat.as<double>()));
	return read_back(m, m->rows_stat.as<double>(), m->K, out);
}

int trlda_device_special(int device, int which, const double* x, int64_t n, double* out) {
	if(cudaSetDevice(device) != cudaSuccess)
		return fail(nullptr, TRLDA_ERR_CUDA, "No CUDA device available; trlda_b200 has no CPU fallback.");
	DevBuf dx, dy;
	if(dx.ensure(sizeof(double) * n) != cudaSuccess || dy.ensure(sizeof(double) * n) != cudaSuccess)
		return fail(nullptr, TRLDA_ERR_CUDA, "cudaMalloc failed.");
	cudaMemcpy(dx.p, x, sizeof(double) * n, cudaMemcpyHostToDevice);
	launch_special(which, dx.as<double>(), n, dy.as<double>(), 0);
	const cudaError_t e = cudaMemcpy(out, dy.p, sizeof(double) * n, cudaMemcpyDeviceToHost);
	if(e != cudaSuccess)
		return fail(nullptr, TRLDA_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
	return TRLDA_OK;
}

double trlda_polygamma(int n, double x) { return host_polygamma(n, x); }

}  // extern "C"
