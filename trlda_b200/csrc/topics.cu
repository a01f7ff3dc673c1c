// topics.cu — looking at a trained model: the most probable words of every topic (trlda_top_words) and how many documents
// of a corpus contain each of those words and each pair of them (trlda_cooccurrence), the counts behind the document
// co-occurrence coherence measures (UMass, NPMI).  Neither has a counterpart in the reference.
#include "kernels.cuh"

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

__global__ void __launch_bounds__(TOP_THREADS) k_top_words_candidates(const double* __restrict__ lambda, int K, int V, int n,
                                                                       int chunk, double* __restrict__ cand_v,
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
			v[u] = w + u < w1 ? __ldg(col + (int64_t) (w + u) * K) : -INFINITY;
		#pragma unroll
		for(int u = 0; u < TOP_UNROLL; ++u) {
			if(v[u] > nth) {
				int p = n - 1;
				for(; p > 0 && list_v[(p - 1) * TOP_THREADS + t] < v[u]; --p) {
					list_v[p * TOP_THREADS + t] = list_v[(p - 1) * TOP_THREADS + t];
					list_id[p * TOP_THREADS + t] = list_id[(p - 1) * TOP_THREADS + t];
				}
				list_v[p * TOP_THREADS + t] = v[u];
				list_id[p * TOP_THREADS + t] = w + u;
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

__global__ void __launch_bounds__(TOP_MERGE_THREADS) k_top_words_merge(const double* __restrict__ cand_v,
                                                                        const int32_t* __restrict__ cand_id,
                                                                        const double* __restrict__ rows, int K, int n,
                                                                        int chunks, int32_t* __restrict__ ids,
                                                                        double* __restrict__ prob) {
	const int lane = threadIdx.x & 31;
	const int k = blockIdx.x * (TOP_MERGE_THREADS / 32) + (threadIdx.x >> 5);
	if(k >= K)
		return;
	double best_v = -INFINITY;
	int best_id = INT_MAX;
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
		prob[(int64_t) k * n + lane] = best_v / rows[k];
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

void launch_top_words_candidates(const double* lambda, int K, int V, int n, int chunks, double* cand_v, int32_t* cand_id,
                                 cudaStream_t s) {
	const int chunk = (V + chunks - 1) / chunks;
	const dim3 grid((unsigned) ((K + TOP_THREADS - 1) / TOP_THREADS), (unsigned) chunks);
	k_top_words_candidates<<<grid, TOP_THREADS, top_words_smem(n), s>>>(lambda, K, V, n, chunk, cand_v, cand_id);
}

void launch_top_words_merge(const double* cand_v, const int32_t* cand_id, const double* rows, int K, int n, int chunks,
                            int32_t* ids, double* prob, cudaStream_t s) {
	const int per_block = TOP_MERGE_THREADS / 32;
	k_top_words_merge<<<(K + per_block - 1) / per_block, TOP_MERGE_THREADS, 0, s>>>(cand_v, cand_id, rows, K, n, chunks, ids, prob);
}

void launch_cooccurrence(const DeviceDocs& docs, int K, int n, const int32_t* map_ptr, const int32_t* map_entry,
                         unsigned long long* counts, cudaStream_t s) {
	if(docs.B == 0)
		return;
	k_cooccurrence<<<(unsigned) std::min<int64_t>(docs.B, sm_count() * 8), CO_THREADS, (size_t) K * 8, s>>>(
		docs, K, n, map_ptr, map_entry, counts);
}

}  // namespace trlda
