// topics.cu — looking at a trained model: the most probable words of every topic (trlda_top_words), how many documents
// of a corpus contain each of those words and each pair of them (trlda_cooccurrence), the counts behind the document
// co-occurrence coherence measures (UMass, NPMI), and the Hellinger / Kullback-Leibler distances between the topics of one
// or two models (trlda_topic_distances), the most probable topics of every word of a document (trlda_word_topics), and the
// indexed documents nearest to a query document under the Hellinger distance of their topic proportions
// (trlda_index_documents, trlda_similar_documents).  None has a counterpart in the reference.
#include "kernels.cuh"
#include "special.cuh"

#include <algorithm>
#include <climits>

namespace trlda {

namespace {

// ---- top words -------------------------------------------------------------------------------------------------------
// The order is E[beta_kw] descending, then word id ascending.  E[beta_kw] = lambda_kw / rows_k is monotone in lambda_kw
// within a topic, so lambda itself is compared (in fp64, in both precision modes); the order is total, so the result does
// not depend on how the words are cut into chunks.
//
// Pass 1: CTA (slab, chunk) takes TOP_THREADS consecutive topics over one chunk of consecutive words.  lambda is K x V
// column-major, so the threads of a warp read consecutive topics of one word column (coalesced fp64 loads); each thread
// keeps its topic's best n words of the chunk, sorted, in shared memory, and rejects most entries against the n-th value
// held in a register.  Words arrive in increasing id order, so a value equal to the n-th one loses its tie and an insertion
// moves only the strictly smaller entries.
// Pass 2: one warp per topic merges the chunks' sorted lists: lane i holds rank i of the running list; a chunk's list is
// loaded in reverse, the lane-wise better of the two is bitonic and holds the best 32 of both, and five xor-shuffle
// compare-exchange steps sort it again.
constexpr int TOP_THREADS = 128;
constexpr int TOP_UNROLL = 16;       // lambda loads in flight per thread
constexpr int TOP_MIN_CHUNK = 256;   // words per chunk at least: bounds the candidate lists the merge reads
constexpr int TOP_MERGE_THREADS = 256;

__device__ __forceinline__ bool ranks_before(double a, int ia, double b, int ib) {
	return a > b || (a == b && ia < ib);
}

// row k of the K x V column-major matrix `lambda` (leading dimension ld); the ids of its columns start at id0
__global__ void __launch_bounds__(TOP_THREADS) k_top_words_candidates(const double* __restrict__ lambda, int K, int ld,
                                                                       int V, int id0, int n, int chunk,
                                                                       double* __restrict__ cand_v,
                                                                       int32_t* __restrict__ cand_id) {
	extern __shared__ double list_v[];                                          // n x TOP_THREADS, rank-major
	int32_t* list_id = reinterpret_cast<int32_t*>(list_v + n * TOP_THREADS);   // n x TOP_THREADS
	const int t = threadIdx.x;
	const int k = blockIdx.x * TOP_THREADS + t;
	if(k >= K)
		return;
	for(int r = 0; r < n; ++r) {
		list_v[r * TOP_THREADS + t] = -INFINITY;
		list_id[r * TOP_THREADS + t] = INT_MAX;
	}
	const int w0 = blockIdx.y * chunk, w1 = min(V, w0 + chunk);
	const double* col = lambda + k;
	double nth = -INFINITY;
	for(int w = w0; w < w1; w += TOP_UNROLL) {
		double v[TOP_UNROLL];
		#pragma unroll
		for(int u = 0; u < TOP_UNROLL; ++u)
			v[u] = w + u < w1 ? __ldg(col + (int64_t) (w + u) * ld) : -INFINITY;
		#pragma unroll
		for(int u = 0; u < TOP_UNROLL; ++u) {
			if(v[u] > nth) {
				int p = n - 1;
				for(; p > 0 && list_v[(p - 1) * TOP_THREADS + t] < v[u]; --p) {
					list_v[p * TOP_THREADS + t] = list_v[(p - 1) * TOP_THREADS + t];
					list_id[p * TOP_THREADS + t] = list_id[(p - 1) * TOP_THREADS + t];
				}
				list_v[p * TOP_THREADS + t] = v[u];
				list_id[p * TOP_THREADS + t] = id0 + w + u;
				nth = list_v[(n - 1) * TOP_THREADS + t];
			}
		}
	}
	const int64_t out = ((int64_t) blockIdx.y * K + k) * n;
	for(int r = 0; r < n; ++r) {
		cand_v[out + r] = list_v[r * TOP_THREADS + t];
		cand_id[out + r] = list_id[r * TOP_THREADS + t];
	}
}

// what the merge writes for a list entry of value v in row k
struct MergeDivide {          // trlda_top_words: E[beta_kw] = lambda_kw / rows_k
	const double* rows;
	__device__ double operator()(double v, int k) const { return v / rows[k]; }
};
struct MergeKeep {            // a running list that later merges continue
	__device__ double operator()(double v, int) const { return v; }
};
struct MergeHellinger {       // trlda_similar_documents: the Hellinger distance sqrt(max(0, 1 - C))
	__device__ double operator()(double v, int) const { return sqrt(fmax(0., 1. - v)); }
};

// init_v / init_id (may be null): a sorted list per row to start from, in the layout of the output (row k at k*n); lane i
// reads entry i before and writes entry i after the merge, so the output may be the initial list itself
template <class Epilogue>
__global__ void __launch_bounds__(TOP_MERGE_THREADS) k_top_words_merge(const double* __restrict__ cand_v,
                                                                        const int32_t* __restrict__ cand_id, int K, int n,
                                                                        int chunks, const double* init_v, const int32_t* init_id,
                                                                        Epilogue epilogue, int32_t* ids, double* prob) {
	const int lane = threadIdx.x & 31;
	const int k = blockIdx.x * (TOP_MERGE_THREADS / 32) + (threadIdx.x >> 5);
	if(k >= K)
		return;
	double best_v = -INFINITY;
	int best_id = INT_MAX;
	if(init_v && lane < n) {
		best_v = init_v[(int64_t) k * n + lane];
		best_id = init_id[(int64_t) k * n + lane];
	}
	const int r = 31 - lane;   // the chunk's list, reversed
	for(int c = 0; c < chunks; ++c) {
		const int64_t at = ((int64_t) c * K + k) * n + r;
		const double v = r < n ? cand_v[at] : -INFINITY;
		const int id = r < n ? cand_id[at] : INT_MAX;
		if(ranks_before(v, id, best_v, best_id)) {
			best_v = v;
			best_id = id;
		}
		#pragma unroll
		for(int j = 16; j >= 1; j >>= 1) {
			const double ov = __shfl_xor_sync(0xffffffffu, best_v, j);
			const int oid = __shfl_xor_sync(0xffffffffu, best_id, j);
			const bool take = (lane & j) ? ranks_before(best_v, best_id, ov, oid) : ranks_before(ov, oid, best_v, best_id);
			if(take) {
				best_v = ov;
				best_id = oid;
			}
		}
	}
	if(lane < n) {
		ids[(int64_t) k * n + lane] = best_id;
		prob[(int64_t) k * n + lane] = epilogue(best_v, k);
	}
}

int top_words_smem(int n) { return n * TOP_THREADS * (int) (sizeof(double) + sizeof(int32_t)); }

// ---- document co-occurrence ------------------------------------------------------------------------------------------
// One CTA per document (grid-stride).  Shared memory holds one 32-bit mask per topic (bit r: the word of rank r of the
// topic's list is in the document) and the list of topics touched by the document, K ints each: it does not depend on the
// document's length.  (1) The threads walk the document's pairs and OR each word's (topic, rank) entries of the inverse map
// into the masks; the thread that turns a mask non-zero appends the topic to the touched list.  (2) For every touched topic
// and set bit i, one thread adds 1 to the counter of (i, j) for every set bit j.  (3) Only the touched masks are cleared.
// The counters are integers, so the result does not depend on the order of the atomics.
constexpr int CO_THREADS = 256;

__global__ void __launch_bounds__(CO_THREADS) k_cooccurrence(DeviceDocs docs, int K, int n, const int32_t* __restrict__ map_ptr,
                                                             const int32_t* __restrict__ map_entry,
                                                             unsigned long long* __restrict__ counts) {
	extern __shared__ uint32_t mask[];               // K
	int32_t* touched = reinterpret_cast<int32_t*>(mask + K);   // K
	__shared__ int num_touched;
	for(int k = threadIdx.x; k < K; k += blockDim.x)
		mask[k] = 0u;
	if(threadIdx.x == 0)
		num_touched = 0;
	__syncthreads();
	for(int64_t d = blockIdx.x; d < docs.B; d += gridDim.x) {
		const int64_t end = docs.doc_ptr[d + 1];
		for(int64_t j = docs.doc_ptr[d] + threadIdx.x; j < end; j += blockDim.x) {
			if(docs.counts[j] <= 0)
				continue;
			const int w = docs.word_ids[j];
			for(int e = map_ptr[w], e1 = map_ptr[w + 1]; e < e1; ++e) {
				const int entry = map_entry[e];
				const int k = entry >> 5;
				if(atomicOr(&mask[k], 1u << (entry & 31)) == 0u)
					touched[atomicAdd(&num_touched, 1)] = k;
			}
		}
		__syncthreads();
		const int nt = num_touched;
		for(int idx = threadIdx.x; idx < nt * n; idx += blockDim.x) {
			const int t = idx / n, i = idx - t * n;
			const int k = touched[t];
			const uint32_t bits = mask[k];
			if((bits >> i) & 1u) {
				unsigned long long* column = counts + (int64_t) k * n * n + i;   // counts[(k n + j) n + i]
				for(uint32_t b = bits; b; b &= b - 1u)
					atomicAdd(column + (int64_t) (__ffs(b) - 1) * n, 1ull);
			}
		}
		__syncthreads();
		for(int t = threadIdx.x; t < nt; t += blockDim.x)
			mask[touched[t]] = 0u;
		if(threadIdx.x == 0)
			num_touched = 0;
		__syncthreads();
	}
}

// ---- distances between topics ------------------------------------------------------------------------------------------
// D = epilogue(C), C = f(P_A) g(P_B)^T: Hellinger f = g = sqrt, D = sqrt(max(0, 1 - C)); Kullback-Leibler f = identity,
// g = log, D = max(0, H_i - C) with the row entropy H_i = sum_w p_iw log p_iw.  lambda is read in fp64 in both modes.
//
// Prepare: CTAs of 32 topics x 8 rows of words; a warp reads 32 consecutive topics of one lambda column (coalesced) and
// writes them to the same place of a word-major scratch whose rows are padded to the product's tile with zeros.  The entropy
// of a topic over the CTA's 64 words is summed per thread in word order, then over the 8 threads in order.
// Product: fp64 register tiles, plain DFMA (sm_100's tensor cores have no f64 kind).  CTA (I, J, s) owns the 128 x 128 tile
// (I, J) of partial s and walks the words of split s in stages of 8: every stage is 8 coalesced runs of 128 consecutive
// topics per operand, double-buffered in shared memory through registers; each thread keeps an 8 x 8 block (rows
// tr*4 + {0..3} and 64 + tr*4 + {0..3}, columns likewise with tc) and does one fma per element and word.  Every element of
// C is thus one fma chain over its split's words in word order, started from the partial of the previous chunk; with
// f = g and X = Y, C_ij and C_ji are the same chain with the two factors swapped, so a self-comparison is exactly symmetric.
// The partials are added in split order by the finish pass: the result is reproducible bit for bit from call to call.
constexpr int DIST_TILE = 128;
constexpr int DIST_BK = 8;
constexpr int DIST_THREADS = 256;
constexpr int DIST_PREP_WORDS = 64;           // words per prepare CTA
constexpr size_t DIST_SCRATCH = 256u << 20;   // bytes of prepared operands per chunk, at most (unless one stage exceeds it)

__device__ __forceinline__ double distance_op(int op, double p) {
	return op == DIST_OP_SQRT ? sqrt(p) : op == DIST_OP_LOG ? log(p) : p;
}

__global__ void __launch_bounds__(256) k_distance_prepare(const double* __restrict__ lambda, int K, int V, int ld, int w0,
                                                          int words, const double* __restrict__ rows, int op_x,
                                                          double* __restrict__ x, int op_y, double* __restrict__ y,
                                                          double* __restrict__ entropy_part, int* __restrict__ flag) {
	__shared__ double h_s[8][32];
	const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
	const int k = blockIdx.x * 32 + tx;   // < ld
	const bool topic = k < K;
	const double r = topic ? rows[k] : 1.;
	const bool logs = op_x == DIST_OP_LOG || (y && op_y == DIST_OP_LOG);
	int bad = topic && !(r > 0.) ? DIST_BAD_EMPTY_ROW : 0;
	double h = 0.;
	#pragma unroll 4
	for(int i = 0; i < DIST_PREP_WORDS / 8; ++i) {
		const int row = blockIdx.y * DIST_PREP_WORDS + i * 8 + ty;
		if(row >= words)
			break;
		const int w = w0 + row;
		double vx = 0., vy = 0.;
		if(topic && w < V) {
			const double v = __ldg(lambda + (int64_t) w * K + k);
			bad |= v < 0. ? DIST_BAD_NEGATIVE : 0;
			bad |= logs && v == 0. ? DIST_BAD_ZERO : 0;
			const double p = v / r;
			vx = distance_op(op_x, p);
			if(y)
				vy = distance_op(op_y, p);
			if(entropy_part && p > 0.)
				h += p * log(p);
		}
		x[(int64_t) row * ld + k] = vx;
		if(y)
			y[(int64_t) row * ld + k] = vy;
	}
	if(bad)
		atomicOr(flag, bad);
	if(entropy_part) {
		h_s[ty][tx] = h;
		__syncthreads();
		if(ty == 0 && topic) {
			double sum = h_s[0][tx];
			#pragma unroll
			for(int t = 1; t < 8; ++t)
				sum += h_s[t][tx];
			entropy_part[(int64_t) blockIdx.y * ld + k] = sum;
		}
	}
}

__global__ void k_distance_entropy(const double* __restrict__ entropy_part, int parts, int K, int ld, int first,
                                   double* __restrict__ entropy) {
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k >= K)
		return;
	double acc = first ? 0. : entropy[k];
	for(int p = 0; p < parts; ++p)
		acc += entropy_part[(int64_t) p * ld + k];
	entropy[k] = acc;
}

// partial s holds ld_x x (gridDim.y tiles) elements; y's rows are ld_y apart, which may exceed the columns the grid covers
__global__ void __launch_bounds__(DIST_THREADS, 1) k_distance_product(const double* __restrict__ x, int ld_x,
                                                                      const double* __restrict__ y, int64_t ld_y,
                                                                      int split_words, int first,
                                                                      double* __restrict__ partial) {
	__shared__ __align__(16) double xs[2][DIST_BK][DIST_TILE];
	__shared__ __align__(16) double ys[2][DIST_BK][DIST_TILE];
	const int t = threadIdx.x, tr = t & 15, tc = t >> 4;
	const int i0 = blockIdx.x * DIST_TILE, j0 = blockIdx.y * DIST_TILE;
	double* out = partial + (int64_t) blockIdx.z * ld_x * gridDim.y * DIST_TILE;

	// element (a, b) of the thread's block: row i0 + orow(a), column j0 + orow(b)
	auto orow = [](int q, int a) { return (a < 4 ? 0 : 64) + q * 4 + (a & 3); };
	double acc[8][8];
	#pragma unroll
	for(int a = 0; a < 8; ++a)
		#pragma unroll
		for(int b = 0; b < 8; ++b)
			acc[a][b] = first ? 0. : out[(int64_t) (j0 + orow(tc, b)) * ld_x + i0 + orow(tr, a)];

	// stage loads: thread t moves topics (2t) % 128, +1 of words t / 64 and t / 64 + 4, in both operands
	const int lw = t >> 6, lt = (2 * t) & (DIST_TILE - 1);
	const double* xp = x + ((int64_t) blockIdx.z * split_words + lw) * ld_x + i0 + lt;
	const double* yp = y + ((int64_t) blockIdx.z * split_words + lw) * ld_y + j0 + lt;
	double2 rx0 = __ldg(reinterpret_cast<const double2*>(xp)), rx1 = __ldg(reinterpret_cast<const double2*>(xp + 4 * ld_x));
	double2 ry0 = __ldg(reinterpret_cast<const double2*>(yp)), ry1 = __ldg(reinterpret_cast<const double2*>(yp + 4 * ld_y));
	*reinterpret_cast<double2*>(&xs[0][lw][lt]) = rx0;
	*reinterpret_cast<double2*>(&xs[0][lw + 4][lt]) = rx1;
	*reinterpret_cast<double2*>(&ys[0][lw][lt]) = ry0;
	*reinterpret_cast<double2*>(&ys[0][lw + 4][lt]) = ry1;
	__syncthreads();

	const int steps = split_words / DIST_BK;
	for(int s = 0; s < steps; ++s) {
		const int cur = s & 1;
		const bool more = s + 1 < steps;
		if(more) {
			xp += (int64_t) DIST_BK * ld_x;
			yp += (int64_t) DIST_BK * ld_y;
			rx0 = __ldg(reinterpret_cast<const double2*>(xp));
			rx1 = __ldg(reinterpret_cast<const double2*>(xp + 4 * ld_x));
			ry0 = __ldg(reinterpret_cast<const double2*>(yp));
			ry1 = __ldg(reinterpret_cast<const double2*>(yp + 4 * ld_y));
		}
		#pragma unroll
		for(int k = 0; k < DIST_BK; ++k) {
			double av[8], bv[8];
			#pragma unroll
			for(int h = 0; h < 4; ++h) {
				const double2 a2 = *reinterpret_cast<const double2*>(&xs[cur][k][(h < 2 ? 0 : 64) + tr * 4 + (h & 1) * 2]);
				const double2 b2 = *reinterpret_cast<const double2*>(&ys[cur][k][(h < 2 ? 0 : 64) + tc * 4 + (h & 1) * 2]);
				av[2 * h] = a2.x;
				av[2 * h + 1] = a2.y;
				bv[2 * h] = b2.x;
				bv[2 * h + 1] = b2.y;
			}
			#pragma unroll
			for(int a = 0; a < 8; ++a)
				#pragma unroll
				for(int b = 0; b < 8; ++b)
					acc[a][b] = fma(av[a], bv[b], acc[a][b]);
		}
		if(more) {
			*reinterpret_cast<double2*>(&xs[cur ^ 1][lw][lt]) = rx0;
			*reinterpret_cast<double2*>(&xs[cur ^ 1][lw + 4][lt]) = rx1;
			*reinterpret_cast<double2*>(&ys[cur ^ 1][lw][lt]) = ry0;
			*reinterpret_cast<double2*>(&ys[cur ^ 1][lw + 4][lt]) = ry1;
		}
		__syncthreads();
	}

	#pragma unroll
	for(int b = 0; b < 8; ++b) {
		double* col = out + (int64_t) (j0 + orow(tc, b)) * ld_x + i0;
		#pragma unroll
		for(int a = 0; a < 8; a += 2)
			*reinterpret_cast<double2*>(col + orow(tr, a)) = make_double2(acc[a][b], acc[a + 1][b]);
	}
}

__global__ void k_distance_finish(const double* __restrict__ partial, int splits, int ld_x, int ld_y, int KA, int KB,
                                  int metric, const double* __restrict__ entropy, double* __restrict__ out) {
	const int64_t n = (int64_t) KA * KB, stride = (int64_t) ld_x * ld_y;
	for(int64_t idx = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t) gridDim.x * blockDim.x) {
		const int j = (int) (idx / KA), i = (int) (idx - (int64_t) j * KA);
		const double* p = partial + (int64_t) j * ld_x + i;
		double c = p[0];
		for(int s = 1; s < splits; ++s)
			c += p[s * stride];
		out[idx] = metric == 0 ? sqrt(fmax(0., 1. - c)) : fmax(0., entropy[i] - c);
	}
}

// ---- topics of the words of documents --------------------------------------------------------------------------------
// s_jk = psi(gamma_dk) + (psi(lambda_kw) - psi_rows_k) for pair j (word w, document d), phi_jk = softmax_k(s_jk), in fp64
// from lambda in fp64 in both modes.  The second term is the same for every pair of word w, so the table pass evaluates it
// once per (word of the call, topic) for one chunk of word ids, skipping the ids the call does not contain; psi(gamma) is
// filled once per call.  The pair pass walks the chunk's pairs in the call's word-sorted token list (a word's pairs are
// consecutive, so its table column is re-read from L1 / L2; a CTA takes a contiguous run of them, so that its warps share
// the columns), one warp per pair with the lanes striding over k:
//   1. s_jk for k = lane, lane + 32, ...: the lane's WT_LIST best (s, k) in registers, in the order of ranks_before
//      (s descending, then k ascending; a total order);
//   2. Sigma_k exp(s_jk - max): lane-strided in k order, then an xor butterfly, so the bits depend on K alone;
//   3. n rounds of a warp arg-max over the lanes' list heads.  Only the winning lane pops its head; a lane whose list runs
//      dry rescans its topics for the best WT_LIST ranked after the last one it gave.  Round r's result stays in lane r,
//      and lanes < n write the pair's row at its original position.
constexpr int WT_THREADS = 256;
constexpr int WT_LIST = 4;                       // per-lane candidates kept in registers when n > 1
constexpr size_t WT_TABLE = 256u << 20;          // bytes of the log-beta table per chunk, at most

__global__ void __launch_bounds__(256) k_word_topics_table(const double* __restrict__ lambda, int K, int w0, int count,
                                                           const int32_t* __restrict__ word_ptr,
                                                           const double* __restrict__ psi_rows, double* __restrict__ table) {
	for(int u = blockIdx.x; u < count; u += gridDim.x) {
		if(word_ptr[w0 + u + 1] == word_ptr[w0 + u])
			continue;
		const double* col = lambda + (int64_t) (w0 + u) * K;
		double* out = table + (int64_t) u * K;
		for(int k = threadIdx.x; k < K; k += blockDim.x)
			out[k] = digamma(__ldg(col + k)) - psi_rows[k];
	}
}

// inserts (v, id) into the sorted list (lv, lk) of M entries, dropping the last one
template <int M>
__device__ __forceinline__ void list_insert(double (&lv)[M], int (&lk)[M], double v, int id) {
	#pragma unroll
	for(int i = 0; i < M; ++i)
		if(ranks_before(v, id, lv[i], lk[i])) {
			const double tv = lv[i];
			const int tk = lk[i];
			lv[i] = v;
			lk[i] = id;
			v = tv;
			id = tk;
		}
}

// the lane's best M entries ranked after (after_v, after_k) (M entries of -inf / INT_MAX when there are fewer)
template <int M>
__device__ __forceinline__ void lane_best(const double* __restrict__ g, const double* __restrict__ t, int K, int lane,
                                          double after_v, int after_k, double (&lv)[M], int (&lk)[M]) {
	#pragma unroll
	for(int i = 0; i < M; ++i) {
		lv[i] = -INFINITY;
		lk[i] = INT_MAX;
	}
	#pragma unroll 4
	for(int k = lane; k < K; k += 32) {
		const double s = g[k] + t[k];
		if(ranks_before(after_v, after_k, s, k) && ranks_before(s, k, lv[M - 1], lk[M - 1]))
			list_insert<M>(lv, lk, s, k);
	}
}

// a / b for 1 <= b <= 2^31 (b is a sum of exp(s - max) with one term 1), without the slow path of the fp64 division: a
// float seed of 1/b, two Newton steps, and one correction of the quotient
__device__ __forceinline__ double divide_by_sum(double a, double b) {
	double r = (double) __fdividef(1.f, (float) b);
	r = fma(r, fma(-b, r, 1.), r);
	r = fma(r, fma(-b, r, 1.), r);
	const double q = a * r;
	return fma(fma(-q, b, a), r, q);
}

template <int M>
__global__ void __launch_bounds__(WT_THREADS) k_word_topics_pairs(DeviceDocs docs, int w0, int w1,
                                                                  const double* __restrict__ table,
                                                                  const double* __restrict__ psi_gamma, int K, int n,
                                                                  int32_t* __restrict__ topics, double* __restrict__ probs) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = WT_THREADS / 32;
	const int p0 = docs.word_ptr[w0], p1 = docs.word_ptr[w1];
	const int per_cta = (p1 - p0 + (int) gridDim.x - 1) / (int) gridDim.x;
	const int begin = p0 + (int) blockIdx.x * per_cta, end = min(p1, begin + per_cta);
	for(int p = begin + warp; p < end; p += nw) {
		const int64_t j = docs.tok_src[p];
		const double* g = psi_gamma + (int64_t) docs.tok_doc[p] * K;
		const double* t = table + (int64_t) (docs.word_ids[j] - w0) * K;
		double lv[M];
		int lk[M];
		lane_best<M>(g, t, K, lane, INFINITY, -1, lv, lk);
		// the maximum: a warp arg-max of the list heads
		double top = lv[0];
		#pragma unroll
		for(int o = 16; o > 0; o >>= 1)
			top = fmax(top, __shfl_xor_sync(0xffffffffu, top, o));
		double sum = 0.;
		#pragma unroll 2   // 4 spills registers around the branches of exp
		for(int k = lane; k < K; k += 32)
			sum += exp(g[k] + t[k] - top);
		sum = warp_sum(sum);
		int my_k = 0;
		double my_v = -INFINITY;
		for(int r = 0; r < n; ++r) {
			double bv = lv[0];
			int bk = lk[0];
			#pragma unroll
			for(int o = 16; o > 0; o >>= 1) {
				const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
				const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
				if(ranks_before(ov, ok, bv, bk)) {
					bv = ov;
					bk = ok;
				}
			}
			if(lane == r) {
				my_k = bk;
				my_v = bv;
			}
			if(r + 1 < n && (bk & 31) == lane) {   // the winner's head was taken
				#pragma unroll
				for(int i = 0; i + 1 < M; ++i) {
					lv[i] = lv[i + 1];
					lk[i] = lk[i + 1];
				}
				lv[M - 1] = -INFINITY;
				lk[M - 1] = INT_MAX;
				if(lk[0] == INT_MAX)
					lane_best<M>(g, t, K, lane, bv, bk, lv, lk);
			}
		}
		if(lane < n) {
			topics[j * n + lane] = my_k;
			if(probs)
				probs[j * n + lane] = divide_by_sum(exp(my_v - top), sum);   // the same exp as in the sum
		}
	}
}

// ---- similar documents ------------------------------------------------------------------------------------------------
// C_qd = sum_k sqrt(theta_qk) sqrt(theta_dk), theta = gamma / column sum, D = sqrt(max(0, 1 - C)): the Hellinger distance of
// the topic distributions of two documents.  The index holds sqrt(theta) of its D documents in the layout k_distance_product
// reads: element (k, d) at k * ld + d, ld = D rounded up to DIST_TILE, with zero rows up to K rounded up to DIST_BK.
// Prepare: one CTA per 32 columns of gamma.  Warp w sums columns w, w + 8, ... lane-strided in k order and then by an xor
// butterfly, so a column's sum depends on K and its own values alone, and an equal query column gives a bitwise equal
// operand.  The columns then go through a 32 x 32 shared-memory transpose: coalesced reads of gamma, coalesced writes of
// runs of 32 documents.
// Stream (few queries): one thread per document of the block and up to SIM_GROUP queries per CTA, the CTAs of one run of
// documents for different query groups next to each other in the grid, so that they meet the same index lines in L2.  A
// thread walks k ascending with acc_q = fma(q_qk, x_kd, acc_q) from 0: the chain of the product's element (q, d), whose
// extra zero rows add nothing, so both paths give the same C bit for bit.
constexpr int SIM_PREP_COLS = 32;
constexpr int SIM_GROUP = 8;                  // queries per CTA of the streaming pass, an accumulator each
constexpr int SIM_STREAM_THREADS = 256;
constexpr int SIM_KT = 64;                    // topics of the queries staged in shared memory at a time

__global__ void __launch_bounds__(256) k_similar_prepare(const double* __restrict__ gamma, int K, int cols, int64_t ld,
                                                         double* __restrict__ out, int* __restrict__ flag) {
	__shared__ double sum_s[SIM_PREP_COLS];
	__shared__ double tile[SIM_PREP_COLS][SIM_PREP_COLS + 1];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int c0 = blockIdx.x * SIM_PREP_COLS;
	int bad = 0;
	for(int j = warp; j < SIM_PREP_COLS; j += 8) {
		const int c = c0 + j;
		double sum = 0.;
		if(c < cols) {
			const double* col = gamma + (int64_t) c * K;
			for(int k = lane; k < K; k += 32) {
				const double v = col[k];
				bad |= !(v >= 0.) || isinf(v);
				sum += v;
			}
		}
		sum = warp_sum(sum);
		if(lane == 0) {
			bad |= c < cols && !(sum > 0. && sum < INFINITY);
			sum_s[j] = sum;
		}
	}
	if(bad)
		atomicOr(flag, 1);
	__syncthreads();
	for(int k0 = 0; k0 < K; k0 += SIM_PREP_COLS) {
		for(int j = warp; j < SIM_PREP_COLS; j += 8) {
			const int c = c0 + j, k = k0 + lane;
			if(c < cols && k < K)
				tile[j][lane] = sqrt(gamma[(int64_t) c * K + k] / sum_s[j]);
		}
		__syncthreads();
		for(int j = warp; j < SIM_PREP_COLS; j += 8) {
			const int k = k0 + j, c = c0 + lane;
			if(k < K && c < cols)
				out[(int64_t) k * ld + c] = tile[lane][j];
		}
		__syncthreads();
	}
}

// aff[d * lda + q] = C_qd for the nq queries of `query` (element (k, q) at k * ldq + q) and the documents d < docs of
// `index`; the grid is (document runs) x groups, group g taking queries g * SIM_GROUP ..
template <int G>
__global__ void __launch_bounds__(SIM_STREAM_THREADS) k_similar_stream(const double* __restrict__ index, int64_t ld, int K,
                                                                       int docs, const double* __restrict__ query, int ldq,
                                                                       int nq, int groups, double* __restrict__ aff,
                                                                       int lda) {
	__shared__ __align__(16) double qs[SIM_KT][G];
	const int g = blockIdx.x % groups, q0 = g * SIM_GROUP;
	const int d = (blockIdx.x / groups) * SIM_STREAM_THREADS + threadIdx.x;
	const int mine = min(G, nq - q0);
	double acc[G];
	#pragma unroll
	for(int i = 0; i < G; ++i)
		acc[i] = 0.;
	const double* col = index + min(d, docs - 1);
	for(int k0 = 0; k0 < K; k0 += SIM_KT) {
		const int kn = min(SIM_KT, K - k0);
		__syncthreads();
		for(int e = threadIdx.x; e < SIM_KT * G; e += SIM_STREAM_THREADS) {
			const int kk = e / G, i = e - kk * G;
			qs[kk][i] = kk < kn && i < mine ? query[(int64_t) (k0 + kk) * ldq + q0 + i] : 0.;
		}
		__syncthreads();
		#pragma unroll 8
		for(int kk = 0; kk < kn; ++kk) {
			const double x = __ldg(col + (int64_t) (k0 + kk) * ld);
			#pragma unroll
			for(int i = 0; i < G; ++i)
				acc[i] = fma(qs[kk][i], x, acc[i]);
		}
	}
	if(d < docs) {
		#pragma unroll
		for(int i = 0; i < G; ++i)
			if(i < mine)
				aff[(int64_t) d * lda + q0 + i] = acc[i];
	}
}

int sm_count() {
	static const int count = [] {
		int device = 0, c = 148;
		if(cudaGetDevice(&device) != cudaSuccess || cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || c < 1)
			c = 148;
		return c;
	}();
	return count;
}

}  // namespace

int top_words_chunks(int K, int V, int n) {
	// enough CTAs to fill every SM at the occupancy the shared-memory lists allow, in chunks of at least TOP_MIN_CHUNK words
	int per_sm = 1;
	if(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_top_words_candidates, TOP_THREADS, top_words_smem(n)) != cudaSuccess ||
	   per_sm < 1)
		per_sm = 1;
	const int slabs = (K + TOP_THREADS - 1) / TOP_THREADS;
	const int want = std::max(1, (per_sm * sm_count() + slabs - 1) / slabs);
	const int chunk = std::max(TOP_MIN_CHUNK, (V + want - 1) / want);
	return (V + chunk - 1) / chunk;
}

void launch_top_words_candidates(const double* lambda, int K, int ld, int V, int id0, int n, int chunks, double* cand_v,
                                 int32_t* cand_id, cudaStream_t s) {
	const int chunk = (V + chunks - 1) / chunks;
	const dim3 grid((unsigned) ((K + TOP_THREADS - 1) / TOP_THREADS), (unsigned) chunks);
	k_top_words_candidates<<<grid, TOP_THREADS, top_words_smem(n), s>>>(lambda, K, ld, V, id0, n, chunk, cand_v, cand_id);
}

void launch_top_words_merge(const double* cand_v, const int32_t* cand_id, const double* rows, int K, int n, int chunks,
                            int32_t* ids, double* prob, cudaStream_t s) {
	const int per_block = TOP_MERGE_THREADS / 32;
	k_top_words_merge<<<(K + per_block - 1) / per_block, TOP_MERGE_THREADS, 0, s>>>(cand_v, cand_id, K, n, chunks, nullptr,
	                                                                                nullptr, MergeDivide{rows}, ids, prob);
}

void launch_top_n_merge(const double* cand_v, const int32_t* cand_id, int K, int n, int chunks, const double* init_v,
                        const int32_t* init_id, bool hellinger, int32_t* ids, double* v, cudaStream_t s) {
	const int per_block = TOP_MERGE_THREADS / 32, blocks = (K + per_block - 1) / per_block;
	if(hellinger)
		k_top_words_merge<<<blocks, TOP_MERGE_THREADS, 0, s>>>(cand_v, cand_id, K, n, chunks, init_v, init_id, MergeHellinger{}, ids, v);
	else
		k_top_words_merge<<<blocks, TOP_MERGE_THREADS, 0, s>>>(cand_v, cand_id, K, n, chunks, init_v, init_id, MergeKeep{}, ids, v);
}

void launch_cooccurrence(const DeviceDocs& docs, int K, int n, const int32_t* map_ptr, const int32_t* map_entry,
                         unsigned long long* counts, cudaStream_t s) {
	if(docs.B == 0)
		return;
	k_cooccurrence<<<(unsigned) std::min<int64_t>(docs.B, sm_count() * 8), CO_THREADS, (size_t) K * 8, s>>>(
		docs, K, n, map_ptr, map_entry, counts);
}

DistancePlan distance_plan(int KA, int KB, int V, bool one_operand) {
	DistancePlan p;
	p.ld_x = (KA + DIST_TILE - 1) / DIST_TILE * DIST_TILE;
	p.ld_y = (KB + DIST_TILE - 1) / DIST_TILE * DIST_TILE;
	// splits: with fewer tiles than SMs, the smallest count in [lo, 4 lo] whose last wave is fullest (one CTA per SM);
	// each split keeps at least 64 words
	const int sms = sm_count(), tiles = (p.ld_x / DIST_TILE) * (p.ld_y / DIST_TILE);
	p.splits = 1;
	if(tiles < sms) {
		const int lo = (sms + tiles - 1) / tiles;
		double best = 0.;
		for(int s = lo; s <= 4 * lo; ++s) {
			const int ctas = tiles * s;
			const double fill = (double) ctas / ((double) ((ctas + sms - 1) / sms) * sms);
			if(fill > best + 1e-12) {
				best = fill;
				p.splits = s;
			}
		}
	}
	p.splits = std::max(1, std::min(p.splits, V / 64));
	const int step = p.splits * DIST_BK;
	const size_t per_word = sizeof(double) * (size_t) (p.ld_x + (one_operand ? 0 : p.ld_y));
	const int64_t fit = (int64_t) (DIST_SCRATCH / per_word) / step * step;
	const int64_t all = ((int64_t) V + step - 1) / step * step;
	p.chunk = (int) std::max<int64_t>(step, std::min(fit, all));
	return p;
}

int distance_chunk_words(const DistancePlan& plan, int remaining) {
	const int step = plan.splits * DIST_BK;
	return (std::min(plan.chunk, remaining) + step - 1) / step * step;
}

int distance_entropy_parts(int words) { return (words + DIST_PREP_WORDS - 1) / DIST_PREP_WORDS; }

void launch_distance_prepare(const double* lambda, int K, int V, int ld, int w0, int words, const double* rows, int op_x,
                             double* x, int op_y, double* y, double* entropy_part, int* flag, cudaStream_t s) {
	const dim3 grid((unsigned) (ld / 32), (unsigned) distance_entropy_parts(words));
	k_distance_prepare<<<grid, 256, 0, s>>>(lambda, K, V, ld, w0, words, rows, op_x, x, op_y, y, entropy_part, flag);
}

void launch_distance_entropy(const double* entropy_part, int parts, int K, int ld, bool first, double* entropy, cudaStream_t s) {
	k_distance_entropy<<<(K + 255) / 256, 256, 0, s>>>(entropy_part, parts, K, ld, first ? 1 : 0, entropy);
}

void launch_distance_product(const DistancePlan& plan, const double* x, const double* y, int words, bool first,
                             double* partial, cudaStream_t s) {
	launch_distance_product(x, plan.ld_x, y, plan.ld_y, plan.ld_y, plan.splits, words, first, partial, s);
}

void launch_distance_product(const double* x, int ld_x, const double* y, int64_t ld_y, int cols_y, int splits, int words, bool first,
                             double* partial, cudaStream_t s) {
	const dim3 grid((unsigned) (ld_x / DIST_TILE), (unsigned) (cols_y / DIST_TILE), (unsigned) splits);
	k_distance_product<<<grid, DIST_THREADS, 0, s>>>(x, ld_x, y, ld_y, words / splits, first ? 1 : 0, partial);
}

int word_topics_chunk_words(int K) { return (int) std::max<size_t>(1, std::min<size_t>(INT_MAX, WT_TABLE / (sizeof(double) * (size_t) K))); }

void launch_word_topics_table(const double* lambda, int K, int w0, int count, const int32_t* word_ptr, const double* psi_rows,
                              double* table, cudaStream_t s) {
	if(count > 0)
		k_word_topics_table<<<(unsigned) std::min(count, sm_count() * 16), std::min(256, (K + 31) / 32 * 32), 0, s>>>(
			lambda, K, w0, count, word_ptr, psi_rows, table);
}

void launch_word_topics_pairs(const DeviceDocs& docs, int w0, int w1, const double* table, const double* psi_gamma, int K, int n,
                              int32_t* topics, double* probs, cudaStream_t s) {
	if(docs.N == 0)
		return;
	// the chunk's pairs are counted on the device; the grid is sized for all of the call's, at least 32 per CTA
	const unsigned grid = (unsigned) std::min<int64_t>((docs.N + 31) / 32, (int64_t) sm_count() * 32);
	if(n == 1)
		k_word_topics_pairs<1><<<grid, WT_THREADS, 0, s>>>(docs, w0, w1, table, psi_gamma, K, n, topics, probs);
	else
		k_word_topics_pairs<WT_LIST><<<grid, WT_THREADS, 0, s>>>(docs, w0, w1, table, psi_gamma, K, n, topics, probs);
}

void launch_distance_finish(const DistancePlan& plan, const double* partial, int KA, int KB, int metric, const double* entropy,
                            double* out, cudaStream_t s) {
	const int64_t n = (int64_t) KA * KB;
	const unsigned blocks = (unsigned) std::min<int64_t>((n + 255) / 256, (int64_t) sm_count() * 16);
	k_distance_finish<<<blocks, 256, 0, s>>>(partial, plan.splits, plan.ld_x, plan.ld_y, KA, KB, metric, entropy, out);
}

int similar_rows(int K) { return (K + DIST_BK - 1) / DIST_BK * DIST_BK; }

int64_t similar_ld(int64_t cols) { return (cols + DIST_TILE - 1) / DIST_TILE * DIST_TILE; }

void launch_similar_prepare(const double* gamma, int K, int cols, int64_t ld, double* out, int* flag, cudaStream_t s) {
	if(cols > 0)
		k_similar_prepare<<<(unsigned) ((cols + SIM_PREP_COLS - 1) / SIM_PREP_COLS), 256, 0, s>>>(gamma, K, cols, ld, out, flag);
}

void launch_similar_stream(const double* index, int64_t ld, int K, int docs, const double* query, int ldq, int nq, double* aff,
                           int lda, cudaStream_t s) {
	if(docs <= 0 || nq <= 0)
		return;
	const int groups = (nq + SIM_GROUP - 1) / SIM_GROUP;
	const unsigned grid = (unsigned) (((int64_t) docs + SIM_STREAM_THREADS - 1) / SIM_STREAM_THREADS * groups);
	if(nq == 1)
		k_similar_stream<1><<<grid, SIM_STREAM_THREADS, 0, s>>>(index, ld, K, docs, query, ldq, nq, groups, aff, lda);
	else if(nq == 2)
		k_similar_stream<2><<<grid, SIM_STREAM_THREADS, 0, s>>>(index, ld, K, docs, query, ldq, nq, groups, aff, lda);
	else if(nq <= 4)
		k_similar_stream<4><<<grid, SIM_STREAM_THREADS, 0, s>>>(index, ld, K, docs, query, ldq, nq, groups, aff, lda);
	else
		k_similar_stream<SIM_GROUP><<<grid, SIM_STREAM_THREADS, 0, s>>>(index, ld, K, docs, query, ldq, nq, groups, aff, lda);
}

}  // namespace trlda
