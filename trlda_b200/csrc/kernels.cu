// kernels.cu — hand-written sm_100a kernels of the trlda hot path.
//
// Data layout in HBM (all column-major, the reference's Eigen layout, so a word's K-vector is contiguous):
//   lambda, lambda', sstats   K x V float64
//   beta = expElogbeta        K x V float64 (fp64 mode) or float32 (mixed mode)
//   gamma, etheta, doc_stat   K x B float64 (+ a float32 copy of etheta in mixed mode)
//   minibatch                 CSR (doc_ptr, word_ids, counts) + word-sorted token list (word_ptr, tok_doc, tok_src)
//
// Reference citations are relative to /root/reference/code/trlda/src/.
#include "kernels.cuh"
#include "special.cuh"
#include "rng.cuh"

#include <cooperative_groups.h>
#include <math_constants.h>
#include <algorithm>
#include <cstdio>

namespace cg = cooperative_groups;

namespace trlda {

// SM count of the current device (one process drives one GPU): grids are sized in multiples of it
static int sm_count() {
	static const int n = [] {
		int device = 0, count = 148;
		if(cudaGetDevice(&device) != cudaSuccess || cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || count < 1)
			count = 148;
		return count;
	}();
	return n;
}

static inline int ceil_div(int64_t a, int64_t b) { return (int) ((a + b - 1) / b); }
static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

// ------------------------------------------------------------------------------------------------------------
// block-level helpers
// ------------------------------------------------------------------------------------------------------------

// deterministic block sum; every thread gets the result.  `scratch` holds >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* scratch) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
	v = warp_sum(v);
	__syncthreads();
	if(lane == 0)
		scratch[warp] = v;
	__syncthreads();
	double total = 0.0;
	for(int i = 0; i < nw; ++i)
		total += scratch[i];
	return total;
}

template <typename T> __device__ __forceinline__ T load_as(const void* p, int64_t i);
template <> __device__ __forceinline__ double load_as<double>(const void* p, int64_t i) { return static_cast<const double*>(p)[i]; }
template <> __device__ __forceinline__ float load_as<float>(const void* p, int64_t i) { return static_cast<const float*>(p)[i]; }

// ------------------------------------------------------------------------------------------------------------
// row sums of a K x V column-major matrix (lda.cpp:172 `mLambda.rowwise().sum()`), two deterministic stages
// ------------------------------------------------------------------------------------------------------------
constexpr int ROWSUM_CHUNK = 128;

__global__ void __launch_bounds__(256) k_rowsum_partial(const double* __restrict__ m, int K, int V, double* __restrict__ partials) {
	const int k = blockIdx.y * 256 + threadIdx.x;
	if(k >= K)
		return;
	const int w0 = blockIdx.x * ROWSUM_CHUNK, w1 = min(V, w0 + ROWSUM_CHUNK);
	double acc = 0.0;
	#pragma unroll 4
	for(int w = w0; w < w1; ++w)
		acc += m[(int64_t) w * K + k];
	partials[(int64_t) blockIdx.x * K + k] = acc;
}

__global__ void __launch_bounds__(256) k_reduce_partials(const double* __restrict__ partials, int P, int K, double* __restrict__ out) {
	const int k = blockIdx.x * 256 + threadIdx.x;
	if(k >= K)
		return;
	double acc = 0.0;
	for(int p = 0; p < P; ++p)
		acc += partials[(int64_t) p * K + k];
	out[k] = acc;
}

int rowsum_num_partials(int V) { return ceil_div(V, ROWSUM_CHUNK); }

void launch_rowsum(const double* lambda, int K, int V, double* partials, int* num_partials, cudaStream_t s) {
	const int P = rowsum_num_partials(V);
	k_rowsum_partial<<<dim3(P, ceil_div(K, 256)), 256, 0, s>>>(lambda, K, V, partials);
	if(num_partials)
		*num_partials = P;
}

void launch_reduce_partials(const double* partials, int P, int K, double* out, cudaStream_t s) {
	k_reduce_partials<<<ceil_div(K, 256), 256, 0, s>>>(partials, P, K, out);
}

__global__ void k_psi_vector(const double* __restrict__ in, int K, double* __restrict__ out) {
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k < K)
		out[k] = digamma(in[k]);
}

void launch_psi_vector(const double* in, int K, double* out, cudaStream_t s) {
	k_psi_vector<<<ceil_div(K, 128), 128, 0, s>>>(in, K, out);
}

__global__ void k_lgamma_vector(const double* __restrict__ in, int K, double* __restrict__ out) {
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k < K)
		out[k] = lgamma(in[k]);
}

void launch_lgamma_vector(const double* in, int K, double* out, cudaStream_t s) {
	k_lgamma_vector<<<ceil_div(K, 128), 128, 0, s>>>(in, K, out);
}

__global__ void k_rows_update(const double* __restrict__ prev, const double* __restrict__ stat, double a, double b, double c,
                              int K, double* __restrict__ rows_new, double* __restrict__ psi_rows) {
	const int k = blockIdx.x * blockDim.x + threadIdx.x;
	if(k >= K)
		return;
	const double r = a * (prev ? prev[k] : 0.0) + b + c * (stat ? stat[k] : 0.0);
	rows_new[k] = r;
	psi_rows[k] = digamma(r);
}

void launch_rows_update(const double* rows_prev, const double* rows_stat, double a, double b, double c, int K,
                        double* rows_new, double* psi_rows, cudaStream_t s) {
	k_rows_update<<<ceil_div(K, 128), 128, 0, s>>>(rows_prev, rows_stat, a, b, c, K, rows_new, psi_rows);
}

// ------------------------------------------------------------------------------------------------------------
// beta-prep: expElogbeta_kw = exp(psi(lambda_kw) - psi(sum_w lambda_kw))   (lda.cpp:172-173)
// One word (K contiguous values) per CTA iteration; streaming, read 8 B + write sizeof(T) per element.
// ------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_beta_prep(const double* __restrict__ lambda, const double* __restrict__ psi_rows,
                                                   int K, int V, T* __restrict__ beta, double* __restrict__ psi_partials) {
	__shared__ double scratch[32];
	for(int w = blockIdx.x; w < V; w += gridDim.x) {
		double psum = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x) {
			const int64_t i = (int64_t) w * K + k;
			if(psi_partials) {
				const double p = digamma(lambda[i]);
				psum += p;
				beta[i] = (T) exp(p - psi_rows[k]);
			} else {
				beta[i] = (T) exp_digamma_for<T>(lambda[i], psi_rows[k]);
			}
		}
		if(psi_partials) {
			const double total = block_sum(psum, scratch);
			if(threadIdx.x == 0)
				psi_partials[w] = total;
		}
	}
}

static inline int block_for_k(int K) { return std::min(256, std::max(32, round_up(K, 32))); }

void launch_beta_prep(const double* lambda, const double* psi_rows, int K, int V, void* beta, int elem_size,
                      double* psi_partials, cudaStream_t s) {
	const int block = block_for_k(K);
	const int grid = std::min(V, sm_count() * 16);
	if(elem_size == 8)
		k_beta_prep<double><<<grid, block, 0, s>>>(lambda, psi_rows, K, V, static_cast<double*>(beta), psi_partials);
	else
		k_beta_prep<float><<<grid, block, 0, s>>>(lambda, psi_rows, K, V, static_cast<float*>(beta), psi_partials);
}

// ------------------------------------------------------------------------------------------------------------
// per-document E-step: the gamma/phi fixed point of lda.cpp:174-204
//
// One thread-block cluster of C CTAs per document.  The K x n_d tile of expElogbeta columns is split BY TOPIC
// ROWS across the CTAs (kc rows each) and kept in shared memory for the whole fixed point, so HBM sees each
// column once.  Splitting by rows makes the gamma update, psi and exp local to a CTA; the only cross-CTA
// traffic per inner iteration is the n_d partial phi-norms (+1 scalar for the convergence test), exchanged
// through distributed shared memory: every CTA pushes its partials to the column's owner CTA, the owner sums
// them in rank order (deterministic) and pushes c_j/phiNorm_j back to all CTAs.
// ------------------------------------------------------------------------------------------------------------
constexpr int ESTEP_THREADS = 256;

struct EStepSmem {
	// byte offsets into dynamic shared memory
	size_t tile, W, W32, P, dpart, gam, eth, eth32, red, wid, cnt, total;
};

__host__ __device__ inline EStepSmem estep_smem_layout(int C, int kc, int n_cap, int n_fit, int elem) {
	EStepSmem L;
	const int nl_cap = (n_cap + C - 1) / C;
	size_t o = 0;
	auto take = [&o](size_t bytes) { size_t at = o; o += (bytes + 15) & ~size_t(15); return at; };
	L.tile = take((size_t) n_fit * kc * elem);
	L.W = take((size_t) n_cap * 8);
	L.W32 = take((size_t) n_cap * 4);
	L.P = take((size_t) C * nl_cap * 8);
	L.dpart = take((size_t) C * 8);
	L.gam = take((size_t) kc * 8);
	L.eth = take((size_t) kc * 8);
	L.eth32 = take((size_t) kc * 4);
	L.red = take((size_t) ESTEP_THREADS * 8);
	L.wid = take((size_t) n_cap * 4);
	L.cnt = take((size_t) n_cap * 4);
	L.total = o;
	return L;
}

EStepPlan plan_estep(int K, int n_max, int elem, int smem_optin) {
	EStepPlan best;
	const int n_cap = std::max(32, round_up(n_max, 32));
	const size_t budget_full = (size_t) smem_optin - 1024;          // 1 KB per CTA is reserved by the driver
	const size_t budget_half = ((size_t) smem_optin + 1024) / 2 - 2048;   // two CTAs per SM
	int candidates[4] = {1, 2, 4, 8};
	int chosen = -1;
	// pass 0: smallest cluster whose full tile fits twice per SM; pass 1: fits once per SM
	for(int pass = 0; pass < 2 && chosen < 0; ++pass)
		for(int ci = 0; ci < 4; ++ci) {
			const int C = candidates[ci];
			const int kc = round_up(ceil_div(K, C), 32);
			if((C - 1) * kc >= K && C > 1)
				continue;                                              // a CTA without rows
			if(kc > 256 && C < 8)
				continue;
			const EStepSmem L = estep_smem_layout(C, kc, n_cap, n_cap, elem);
			if(L.total <= (pass == 0 ? budget_half : budget_full)) {
				chosen = C;
				break;
			}
		}
	int C = chosen;
	if(C < 0) {
		// nothing fits entirely: largest usable cluster, keep as many columns on chip as fit
		C = 8;
		while(C > 1 && (C - 1) * round_up(ceil_div(K, C), 32) >= K)
			C /= 2;
	}
	const int kc = round_up(ceil_div(K, C), 32);
	int n_fit = n_cap;
	EStepSmem L = estep_smem_layout(C, kc, n_cap, n_fit, elem);
	if(L.total > budget_full) {
		const EStepSmem L0 = estep_smem_layout(C, kc, n_cap, 0, elem);
		n_fit = L0.total >= budget_full ? 0 : (int) ((budget_full - L0.total) / ((size_t) kc * elem));
		n_fit = n_fit / 4 * 4;
		L = estep_smem_layout(C, kc, n_cap, n_fit, elem);
	}
	best.cluster = C;
	best.kc = kc;
	best.n_cap = n_cap;
	best.n_fit = n_fit;
	best.smem = L.total;
	return best;
}

// LONG = true: the variant for documents whose per-pair vectors do not fit in shared memory (plan_estep_long).  The word
// ids and counts are read from the CSR arrays, the weights W_j are kept in their output array a.weight, and the float32
// weights and the C partial phi-norms of every pair live in `scratch`: for a launch over documents of P pairs in all,
// C * P doubles of partials followed by P floats, each document at the pairs of the documents before it in the launch.
// Those are written by one CTA of the cluster and read by others after cluster.sync(), so they are loaded through L2
// (__ldcg), never from a possibly stale L1 line.  Shared memory holds only the K-sized vectors and n_fit tile columns.
// The float32 products of the mixed mode are summed in float32 over groups of LONG_GROUP columns and the groups in
// float64, so that the rounding error does not grow with the length of the document.
constexpr int LONG_GROUP = 64;

template <typename T, bool CLUSTERED, bool LONG>
__global__ void __launch_bounds__(ESTEP_THREADS)
k_estep(EStepArgs a, DeviceDocs docs, const int32_t* __restrict__ order, int64_t doc_offset, int C, int kc, int n_cap, int n_fit,
        double* __restrict__ scratch, int64_t scratch_pairs) {
	extern __shared__ __align__(16) unsigned char smem[];
	const EStepSmem L = estep_smem_layout(C, kc, LONG ? 0 : n_cap, n_fit, (int) sizeof(T));
	T* tile = reinterpret_cast<T*>(smem + L.tile);
	double* W = reinterpret_cast<double*>(smem + L.W);
	float* W32 = reinterpret_cast<float*>(smem + L.W32);
	double* P = reinterpret_cast<double*>(smem + L.P);
	double* dpart = reinterpret_cast<double*>(smem + L.dpart);
	double* gam = reinterpret_cast<double*>(smem + L.gam);
	double* eth = reinterpret_cast<double*>(smem + L.eth);
	float* eth32 = reinterpret_cast<float*>(smem + L.eth32);
	double* red = reinterpret_cast<double*>(smem + L.red);
	const int* wid = reinterpret_cast<int*>(smem + L.wid);
	const int* cnt = reinterpret_cast<int*>(smem + L.cnt);

	cg::cluster_group cluster = cg::this_cluster();
	const int rank = CLUSTERED ? (int) cluster.block_rank() : 0;
	const int64_t slot = doc_offset + blockIdx.x / C;
	const int64_t d = order ? order[slot] : slot;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	constexpr int NW = ESTEP_THREADS / 32;
	const int K = a.K;
	const int k0 = rank * kc;
	const int kn = max(0, min(kc, K - k0));                      // rows of this CTA
	const int64_t begin = docs.doc_ptr[d];
	const int n = (int) (docs.doc_ptr[d + 1] - begin);
	const int n_in = min(n, n_fit);                              // columns resident in shared memory
	const int nl_cap = (n_cap + C - 1) / C;
	const T* __restrict__ beta = static_cast<const T*>(a.beta);
	constexpr bool F32 = sizeof(T) == 4;

	// ---- stage the document, the gamma slice and the tile ----------------------------------------------------
	if constexpr(LONG) {
		int64_t off = 0;                                         // pairs of the launch's documents before this one
		for(int64_t s = doc_offset; s < slot; ++s) {
			const int64_t e = order ? order[s] : s;
			off += docs.doc_ptr[e + 1] - docs.doc_ptr[e];
		}
		wid = docs.word_ids + begin;
		cnt = docs.counts + begin;
		W = a.weight + begin;
		P = scratch + (int64_t) C * off;
		W32 = reinterpret_cast<float*>(scratch + (int64_t) C * scratch_pairs) + off;
	} else {
		for(int j = tid; j < n; j += ESTEP_THREADS) {
			reinterpret_cast<int*>(smem + L.wid)[j] = docs.word_ids[begin + j];
			reinterpret_cast<int*>(smem + L.cnt)[j] = docs.counts[begin + j];
		}
	}
	for(int r = tid; r < kc; r += ESTEP_THREADS) {
		double g = 0.0, e = 0.0;
		if(r < kn) {
			g = a.gamma[d * K + k0 + r];
			e = exp_digamma(g);                                   // lda.cpp:174
		}
		gam[r] = g;
		eth[r] = e;
		eth32[r] = (float) e;
	}
	__syncthreads();
	for(int j = warp; j < n_in; j += NW) {
		const T* col = beta + (int64_t) wid[j] * K + k0;
		for(int r = lane; r < kc; r += 32)
			tile[(size_t) j * kc + r] = r < kn ? col[r] : T(0);
	}
	__syncthreads();

	// phiNorm partials of this CTA's rows, pushed to the owner of each column (lda.cpp:183,199)
	auto pass2_push = [&](double delta_part) {
		for(int j = warp; j < n; j += NW) {
			double part;
			if(F32) {
				float acc = 0.f;
				if(j < n_in) {
					const T* col = tile + (size_t) j * kc;
					for(int r = lane; r < kc; r += 32)
						acc = fmaf(eth32[r], (float) col[r], acc);
				} else {
					const T* col = beta + (int64_t) wid[j] * K + k0;
					for(int r = lane; r < kn; r += 32)
						acc = fmaf(eth32[r], (float) col[r], acc);
				}
				part = (double) acc;
			} else {
				double acc = 0.0;
				if(j < n_in) {
					const T* col = tile + (size_t) j * kc;
					for(int r = lane; r < kc; r += 32)
						acc = fma(eth[r], (double) col[r], acc);
				} else {
					const T* col = beta + (int64_t) wid[j] * K + k0;
					for(int r = lane; r < kn; r += 32)
						acc = fma(eth[r], (double) col[r], acc);
				}
				part = acc;
			}
			part = warp_sum(part);
			if(lane == 0) {
				if constexpr(LONG) {
					__stcg(P + (int64_t) rank * n + j, part);
				} else {
					const int owner = j % C, jl = j / C;
					double* dst = CLUSTERED ? cluster.map_shared_rank(P, owner) : P;
					dst[rank * nl_cap + jl] = part;
				}
			}
		}
		if(tid < C) {
			double* dst = CLUSTERED ? cluster.map_shared_rank(dpart, tid) : dpart;
			dst[rank] = delta_part;
		}
	};

	// owner side: sum the partials in rank order, form c_j / phiNorm_j and broadcast it to every CTA.
	// Returns the cluster-wide sum of |delta gamma| (identical bits in every CTA).
	auto exchange = [&]() -> double {
		if(CLUSTERED) cluster.sync(); else __syncthreads();
		double delta = 0.0;
		for(int src = 0; src < C; ++src)
			delta += dpart[src];
		for(int jl = tid; jl * C + rank < n; jl += ESTEP_THREADS) {
			const int j = jl * C + rank;
			double phi = 0.0;
			for(int src = 0; src < C; ++src)
				phi += LONG ? __ldcg(P + (int64_t) src * n + j) : P[src * nl_cap + jl];
			phi += 1e-100;
			const double wv = (double) cnt[j] / phi;
			if constexpr(LONG) {                                     // one copy, read by every CTA through L2
				__stcg(W + j, wv);
				__stcg(W32 + j, (float) fmin(wv, 1e30));
			} else {
				for(int dst = 0; dst < C; ++dst) {
					double* Wd = CLUSTERED ? cluster.map_shared_rank(W, dst) : W;
					float* Wf = CLUSTERED ? cluster.map_shared_rank(W32, dst) : W32;
					Wd[j] = wv;
					// float32 products: a weight that overflowed float32 (phi underflowed, lda.cpp:183's 1e-100 floor) would
					// turn 0 * inf into NaN where the fp64 reference gets 0
					Wf[j] = (float) fmin(wv, 1e30);
				}
			}
		}
		if(CLUSTERED) cluster.sync(); else __syncthreads();
		return delta;
	};

	// sum_j W_j tile[j][row] for this thread's (row, column-split); the splits are combined through `red`
	const int R = min(kc, ESTEP_THREADS);
	const int S = ESTEP_THREADS / R;
	const int r0 = tid % R, sp = tid / R;
	auto pass1_partial = [&](int row) -> double {
		if constexpr(LONG && F32) {
			double sum = 0.0;
			for(int jg = sp; jg < n_in; jg += LONG_GROUP * S) {
				float acc = 0.f;
				for(int j = jg; j < min(n_in, jg + LONG_GROUP * S); j += S)
					acc = fmaf(__ldcg(W32 + j), (float) tile[(size_t) j * kc + row], acc);
				sum += (double) acc;
			}
			if(row < kn)
				for(int jg = n_in + sp; jg < n; jg += LONG_GROUP * S) {
					float acc = 0.f;
					for(int j = jg; j < min(n, jg + LONG_GROUP * S); j += S)
						acc = fmaf(__ldcg(W32 + j), (float) beta[(int64_t) wid[j] * K + k0 + row], acc);
					sum += (double) acc;
				}
			return sum;
		} else if constexpr(LONG) {
			double acc = 0.0;
			for(int j = sp; j < n_in; j += S)
				acc = fma(__ldcg(W + j), (double) tile[(size_t) j * kc + row], acc);
			if(row < kn)
				for(int j = n_in + sp; j < n; j += S)
					acc = fma(__ldcg(W + j), (double) beta[(int64_t) wid[j] * K + k0 + row], acc);
			return acc;
		} else if(F32) {
			float acc = 0.f;
			for(int j = sp; j < n_in; j += S)
				acc = fmaf(W32[j], (float) tile[(size_t) j * kc + row], acc);
			if(row < kn)
				for(int j = n_in + sp; j < n; j += S)
					acc = fmaf(W32[j], (float) beta[(int64_t) wid[j] * K + k0 + row], acc);
			return (double) acc;
		} else {
			double acc = 0.0;
			for(int j = sp; j < n_in; j += S)
				acc = fma(W[j], (double) tile[(size_t) j * kc + row], acc);
			if(row < kn)
				for(int j = n_in + sp; j < n; j += S)
					acc = fma(W[j], (double) beta[(int64_t) wid[j] * K + k0 + row], acc);
			return acc;
		}
	};

	pass2_push(0.0);
	exchange();

	int it = 0;
	for(; it < a.max_iter; ) {
		// ---- gamma update (lda.cpp:186-197) ----------------------------------------------------------------------
		double delta_local = 0.0;
		for(int rb = 0; rb < kc; rb += R) {
			const int row = rb + r0;
			const bool active = sp < S && row < kc;
			if(active)
				red[sp * R + r0] = pass1_partial(row);
			__syncthreads();
			if(active && sp == 0 && row < kn) {
				double acc = 0.0;
				for(int q = 0; q < S; ++q)
					acc += red[q * R + r0];
				const double g_old = gam[row];
				double g_new = acc * eth[row];
				g_new += a.alpha[k0 + row];
				delta_local += fabs(g_old - g_new);
				gam[row] = g_new;
				const double e = exp_digamma(g_new);
				eth[row] = e;
				eth32[row] = (float) e;
			}
			__syncthreads();
		}
		const double delta_part = block_sum(delta_local, red);
		__syncthreads();
		// ---- phiNorm with the new exp(psi(gamma)) (lda.cpp:199), exchange, convergence test (lda.cpp:202) -----------
		pass2_push(delta_part);
		const double delta = exchange();
		++it;
		if(delta / K < a.threshold)
			break;
	}

	// ---- results: gamma, exp(psi(gamma)), token weights, the document's contribution to the row sums of sstats ---
	for(int r = tid; r < kn; r += ESTEP_THREADS) {
		a.gamma[d * K + k0 + r] = gam[r];
		a.etheta[d * K + k0 + r] = eth[r];
		if(a.etheta32)
			a.etheta32[d * K + k0 + r] = eth32[r];
	}
	if(!LONG)                                                    // LONG: the weights are already in place
		for(int j = tid * C + rank; j < n; j += ESTEP_THREADS * C)
			a.weight[begin + j] = W[j];
	if(a.doc_stat) {
		for(int rb = 0; rb < kc; rb += R) {
			const int row = rb + r0;
			const bool active = sp < S && row < kc;
			if(active)
				red[sp * R + r0] = pass1_partial(row);
			__syncthreads();
			if(active && sp == 0 && row < kn) {
				double acc = 0.0;
				for(int q = 0; q < S; ++q)
					acc += red[q * R + r0];
				a.doc_stat[d * K + k0 + row] = acc * eth[row];
			}
			__syncthreads();
		}
	}
	if(rank == 0 && tid == 0 && a.iterations)
		a.iterations[d] = it;
	if(rank == 0 && tid == 0 && a.sweeps)
		atomicAdd(a.sweeps, (unsigned long long) (it + 1));
}

static int g_estep_smem_optin = 0;

void configure_estep(int smem_optin) {
	g_estep_smem_optin = smem_optin;
	cudaFuncSetAttribute(k_estep<double, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<double, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<float, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<float, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<double, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<double, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<float, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
	cudaFuncSetAttribute(k_estep<float, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
}

template <typename T, bool CLUSTERED, bool LONG>
static void launch_estep_t(const EStepPlan& plan, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order,
                           int64_t offset, int64_t count, double* scratch, int64_t scratch_pairs, cudaStream_t s) {
	cudaLaunchConfig_t cfg = {};
	cfg.gridDim = dim3((unsigned) (count * plan.cluster));
	cfg.blockDim = dim3(ESTEP_THREADS);
	cfg.dynamicSmemBytes = plan.smem;
	cfg.stream = s;
	cudaLaunchAttribute attr[1];
	attr[0].id = cudaLaunchAttributeClusterDimension;
	attr[0].val.clusterDim.x = plan.cluster;
	attr[0].val.clusterDim.y = 1;
	attr[0].val.clusterDim.z = 1;
	cfg.attrs = attr;
	cfg.numAttrs = CLUSTERED ? 1 : 0;
	cudaLaunchKernelEx(&cfg, k_estep<T, CLUSTERED, LONG>, args, docs, order, offset, plan.cluster, plan.kc, plan.n_cap, plan.n_fit,
	                   scratch, scratch_pairs);
}

void launch_estep(const EStepPlan& plan, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order,
                  int64_t offset, int64_t count, int elem_size, cudaStream_t s) {
	if(count == 0)
		return;
	if(elem_size == 8) {
		if(plan.cluster > 1) launch_estep_t<double, true, false>(plan, args, docs, order, offset, count, nullptr, 0, s);
		else launch_estep_t<double, false, false>(plan, args, docs, order, offset, count, nullptr, 0, s);
	} else {
		if(plan.cluster > 1) launch_estep_t<float, true, false>(plan, args, docs, order, offset, count, nullptr, 0, s);
		else launch_estep_t<float, false, false>(plan, args, docs, order, offset, count, nullptr, 0, s);
	}
}

EStepPlan plan_estep_long(int K, int n_max, int elem, int smem_optin) {
	int C = 8;                                                     // the largest cluster that leaves no CTA without rows
	while(C > 1 && (C - 1) * round_up(ceil_div(K, C), 32) >= K)
		C /= 2;
	const int kc = round_up(ceil_div(K, C), 32);
	const size_t budget = (size_t) smem_optin - 1024;
	const EStepSmem L0 = estep_smem_layout(C, kc, 0, 0, elem);
	int n_fit = L0.total >= budget ? 0 : (int) ((budget - L0.total) / ((size_t) kc * elem));
	n_fit = std::min(n_fit, n_max) / 4 * 4;
	EStepPlan plan;
	plan.cluster = C;
	plan.kc = kc;
	plan.n_cap = 0;
	plan.n_fit = n_fit;
	plan.smem = estep_smem_layout(C, kc, 0, n_fit, elem).total;
	return plan;
}

size_t estep_long_scratch_bytes(const EStepPlan& plan, int64_t pairs) {
	return (size_t) pairs * ((size_t) plan.cluster * sizeof(double) + sizeof(float));
}

void launch_estep_long(const EStepPlan& plan, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order,
                       int64_t offset, int64_t count, double* scratch, int64_t scratch_pairs, int elem_size, cudaStream_t s) {
	if(count == 0)
		return;
	if(elem_size == 8) {
		if(plan.cluster > 1) launch_estep_t<double, true, true>(plan, args, docs, order, offset, count, scratch, scratch_pairs, s);
		else launch_estep_t<double, false, true>(plan, args, docs, order, offset, count, scratch, scratch_pairs, s);
	} else {
		if(plan.cluster > 1) launch_estep_t<float, true, true>(plan, args, docs, order, offset, count, scratch, scratch_pairs, s);
		else launch_estep_t<float, false, true>(plan, args, docs, order, offset, count, scratch, scratch_pairs, s);
	}
}

// ------------------------------------------------------------------------------------------------------------
// segmented scatter of the sufficient statistics (lda.cpp:207-217), optionally fused with the M-step blend
// (onlinelda.cpp:99-100 / batchlda.cpp:60 / cumulativelda.cpp:69) and the next beta-prep (lda.cpp:172-173).
//
// Tokens are sorted by word once per minibatch; one CTA owns one word's K-vector, walks the word's tokens in
// document order and accumulates weight_t * etheta[:, doc_t] in registers — no atomics, fixed summation order.
// The K x B etheta matrix (65 MB at cfg-3) is L2-resident, so HBM sees lambda', lambda and beta once each.
// ------------------------------------------------------------------------------------------------------------
constexpr int SCATTER_THREADS = 128;

__device__ __forceinline__ double mstep_value(const MStepCoef& c, double lambda_prime, double s) {
	if(c.mode == MSTEP_ONLINE) {
		const double lambda_hat = c.eta + c.scale * s;                 // onlinelda.cpp:99
		return (1. - c.rho) * lambda_prime + c.rho * lambda_hat;       // onlinelda.cpp:100
	}
	if(c.mode == MSTEP_BATCH)
		return c.eta + s;                                              // batchlda.cpp:60
	return lambda_prime + s;                                           // cumulativelda.cpp:69
}

// multi-GPU push target of word w: (owner rank, element offset of the column inside the owner's receive buffer)
__device__ __forceinline__ void* peer_column(const ScatterArgs& a, int w, int64_t* offset) {
	const int G = a.peer_ranks;
	int o = (int) ((int64_t) w * G / a.V);
	while(o > 0 && w < (int) ((int64_t) a.V * o / G))
		--o;
	while(o + 1 < G && w >= (int) ((int64_t) a.V * (o + 1) / G))
		++o;
	const int v0 = (int) ((int64_t) a.V * o / G);
	*offset = ((int64_t) a.peer_rank * a.peer_shard_cap + (w - v0)) * a.K;
	return a.peer_out[o];
}

template <typename TE, typename TB, int KPT>
__global__ void __launch_bounds__(SCATTER_THREADS, (KPT <= 8 ? 7 : 1)) k_scatter(ScatterArgs a, DeviceDocs docs) {
	__shared__ double scratch[32];
	const int K = a.K;
	const TE* __restrict__ etheta = static_cast<const TE*>(a.etheta);
	TB* beta = static_cast<TB*>(a.beta);
	const bool need_prime = a.fused && a.coef.mode != MSTEP_BATCH;
	for(int w = blockIdx.x; w < a.V; w += gridDim.x) {
		// this word's column of beta and lambda': issue the (HBM, streaming) loads first so that their latency hides
		// behind the walk over the word's tokens
		TB bcol[KPT];
		double lp[KPT];
		#pragma unroll
		for(int i = 0; i < KPT; ++i) {
			const int k = threadIdx.x + i * SCATTER_THREADS;
			const int64_t e = (int64_t) w * K + k;
			bcol[i] = k < K ? __ldcs(beta + e) : TB(0);
			lp[i] = (k < K && need_prime) ? __ldcs(a.lambda_prime + e) : 0.0;
		}

		double acc[KPT];
		#pragma unroll
		for(int i = 0; i < KPT; ++i)
			acc[i] = 0.0;
		const int t0 = docs.word_ptr[w], t1 = docs.word_ptr[w + 1];
		// software pipeline over groups of G tokens: (doc, weight) of the next group are fetched while the
		// etheta rows of the current group are in flight
		constexpr int G = KPT >= 8 ? 2 : 4;
		int dd[G];
		double ww[G];
		auto fetch = [&](int t) {
			#pragma unroll
			for(int u = 0; u < G; ++u) {
				const bool ok = t + u < t1;
				dd[u] = ok ? docs.tok_doc[t + u] : 0;
				ww[u] = ok ? a.weight[docs.tok_src[t + u]] : 0.0;
			}
		};
		if(t0 < t1)
			fetch(t0);
		for(int t = t0; t < t1; t += G) {
			TE v[G][KPT];
			#pragma unroll
			for(int u = 0; u < G; ++u) {
				const TE* col = etheta + (int64_t) dd[u] * K;
				#pragma unroll
				for(int i = 0; i < KPT; ++i) {
					const int k = threadIdx.x + i * SCATTER_THREADS;
					v[u][i] = k < K ? col[k] : TE(0);
				}
			}
			double wc[G];
			#pragma unroll
			for(int u = 0; u < G; ++u)
				wc[u] = ww[u];
			if(t + G < t1)
				fetch(t + G);
			#pragma unroll
			for(int u = 0; u < G; ++u)
				#pragma unroll
				for(int i = 0; i < KPT; ++i)
					acc[i] = fma(wc[u], (double) v[u][i], acc[i]);   // padded tokens carry weight 0 (document 0's row)
		}

		double psum = 0.0;
		#pragma unroll
		for(int i = 0; i < KPT; ++i) {
			const int k = threadIdx.x + i * SCATTER_THREADS;
			if(k >= K)
				continue;
			const int64_t e = (int64_t) w * K + k;
			const double s = acc[i] * (double) bcol[i];                  // lda.cpp:217
			if(!a.fused) {
				if(a.peer_ranks > 0) {
					int64_t off;
					void* dst = peer_column(a, w, &off);
					if(a.peer_elem == 4) static_cast<float*>(dst)[off + k] = (float) s;
					else static_cast<double*>(dst)[off + k] = s;
				} else {
					a.sstats[e] = s;
				}
				continue;
			}
			const double lam = mstep_value(a.coef, lp[i], s);
			__stcs(a.lambda + e, lam);
			if(a.psi_partials) {
				const double p = digamma(lam);
				psum += p;
				if(a.write_beta)
					__stcs(beta + e, (TB) exp(p - a.psi_rows[k]));
			} else if(a.write_beta) {
				__stcs(beta + e, (TB) exp_digamma_for<TB>(lam, a.psi_rows[k]));
			}
		}
		if(a.fused && a.psi_partials) {
			const double total = block_sum(psum, scratch);
			if(threadIdx.x == 0)
				a.psi_partials[w] = total;
		}
	}
}

// Vectorised variant for the mixed-precision path (etheta and beta in float32, K a multiple of 4): every thread
// owns NCH chunks of 4 consecutive topics, so a token costs NCH 128-bit L2 loads per thread instead of 4 NCH
// 32-bit ones, and lambda' / lambda / beta move as 128-/256-bit streaming accesses.
// L tokens' gathers are in flight at a time (L a multiple of G); the arithmetic stays in groups of G whatever L is.
template <int NT, int NCH, int G, int L = G>
__global__ void __launch_bounds__(NT, (NT == 128 && NCH <= 2 ? (L > 4 ? 4 : 5) : 1)) k_scatter_vec(ScatterArgs a, DeviceDocs docs) {
	__shared__ double scratch[32];
	const int K = a.K;
	const int chunks = K / 4;
	const float* __restrict__ etheta = static_cast<const float*>(a.etheta);
	float* beta = static_cast<float*>(a.beta);
	const bool need_prime = a.fused && a.coef.mode != MSTEP_BATCH;
	// exp(-psi(new row sum)) of this thread's topics, prepared once (the thread keeps the same topics for all words)
	float ek[NCH][4];
	#pragma unroll
	for(int i = 0; i < NCH; ++i) {
		const int c = threadIdx.x + i * NT;
		#pragma unroll
		for(int q = 0; q < 4; ++q)
			ek[i][q] = (a.fused && a.write_beta && c < chunks) ? (float) exp(-a.psi_rows[4 * c + q]) : 0.0f;
	}
	__shared__ long long s_row[2][NT];     // byte offset of the token's document row in etheta
	__shared__ float s_w[2][NT];
	const long long row_bytes = (long long) K * (long long) sizeof(float);
	// chunk of out-of-range threads (K / 4 not a multiple of NT): they load the last chunk and drop the result
	int cc[NCH];
	#pragma unroll
	for(int i = 0; i < NCH; ++i)
		cc[i] = min((int) threadIdx.x + i * NT, chunks - 1);
	auto stage_tokens = [&](int b, int begin, int end) {
		const int t = begin + (int) threadIdx.x;
		if(t < end) {
			s_row[b][threadIdx.x] = (long long) docs.tok_doc[t] * row_bytes;
			s_w[b][threadIdx.x] = (float) a.weight[docs.tok_src[t]];
		}
	};
	int buf = 0;
	const int w_begin = a.v1 < 0 ? 0 : a.v0, w_end = a.v1 < 0 ? a.V : a.v1;       // this launch's words
	// Token ranges are looked up TWO words ahead and the (document, weight) pairs of the next word's tokens travel
	// through registers while the current word is processed: none of the dependent loads word_ptr -> tok_src ->
	// weight is waited for (the first version staged the next word in one go and stalled on that chain before every
	// word's token loop: 18 % of the stall samples).
	int t0 = 0, t1 = 0, n0 = 0, n1 = 0;             // token ranges of the current and the next word
	if(w_begin + (int) blockIdx.x < w_end) {
		t0 = docs.word_ptr[w_begin + blockIdx.x];
		t1 = docs.word_ptr[w_begin + blockIdx.x + 1];
		stage_tokens(0, t0, t1);
	}
	if(w_begin + (int) (blockIdx.x + gridDim.x) < w_end) {
		n0 = docs.word_ptr[w_begin + blockIdx.x + gridDim.x];
		n1 = docs.word_ptr[w_begin + blockIdx.x + gridDim.x + 1];
	}
	__syncthreads();
	for(int w = w_begin + blockIdx.x; w < w_end; w += gridDim.x) {
		const int64_t base = (int64_t) w * K;
		float4 bcol[NCH];
		double lp[NCH][4];
		#pragma unroll
		for(int i = 0; i < NCH; ++i) {
			const int c = threadIdx.x + i * NT;
			bcol[i] = c < chunks ? __ldcs(reinterpret_cast<const float4*>(beta + base) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
			if(c < chunks && need_prime) {
				const double2 p0 = __ldcs(reinterpret_cast<const double2*>(a.lambda_prime + base) + 2 * c);
				const double2 p1 = __ldcs(reinterpret_cast<const double2*>(a.lambda_prime + base) + 2 * c + 1);
				lp[i][0] = p0.x; lp[i][1] = p0.y; lp[i][2] = p1.x; lp[i][3] = p1.y;
			} else {
				lp[i][0] = lp[i][1] = lp[i][2] = lp[i][3] = 0.0;
			}
		}
		double acc[NCH][4];
		#pragma unroll
		for(int i = 0; i < NCH; ++i)
			acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0;

		// the (document, weight) pairs of the word's tokens were staged into shared memory while the previous word was
		// processed; now the next word's (document, source index) are requested, and the range of the word after it
		const int wn = w + gridDim.x, wnn = wn + gridDim.x;
		int r_doc = 0, r_src = -1;
		if(wn < w_end && n0 + (int) threadIdx.x < n1) {
			r_doc = docs.tok_doc[n0 + threadIdx.x];
			r_src = docs.tok_src[n0 + threadIdx.x];
		}
		int nn0 = 0, nn1 = 0;
		if(wnn < w_end) {
			nn0 = docs.word_ptr[wnn];
			nn1 = docs.word_ptr[wnn + 1];
		}
		for(int ts = t0; ts < t1; ts += NT) {
			if(ts > t0) {                                              // words with more than NT tokens: restage in place
				__syncthreads();
				stage_tokens(buf, ts, t1);
				__syncthreads();
			}
			const int n = min(NT, t1 - ts);
			for(int g = 0; g < n; g += L) {
				float4 v[L][NCH];
				float wf[L];
				#pragma unroll
				for(int u = 0; u < L; ++u) {
					// the tail of a group repeats the word's last token with weight 0: unconditional loads (the repeat
					// hits in L1), no predicates, no zero-filling of the registers
					const int tt = min(g + u, n - 1);
					wf[u] = g + u < n ? s_w[buf][tt] : 0.f;
					const float4* col = reinterpret_cast<const float4*>(reinterpret_cast<const char*>(etheta) + s_row[buf][tt]);
					#pragma unroll
					for(int i = 0; i < NCH; ++i)
						v[u][i] = col[cc[i]];
				}
				// float32 products summed over the <= G tokens of the group, float64 across groups
				#pragma unroll
				for(int sg = 0; sg < L; sg += G) {
					if(sg > 0 && g + sg >= n)
						break;
					#pragma unroll
					for(int i = 0; i < NCH; ++i) {
						float g0 = 0.f, g1 = 0.f, g2 = 0.f, g3 = 0.f;
						#pragma unroll
						for(int u = sg; u < sg + G; ++u) {
							g0 = fmaf(wf[u], v[u][i].x, g0);
							g1 = fmaf(wf[u], v[u][i].y, g1);
							g2 = fmaf(wf[u], v[u][i].z, g2);
							g3 = fmaf(wf[u], v[u][i].w, g3);
						}
						acc[i][0] += (double) g0;
						acc[i][1] += (double) g1;
						acc[i][2] += (double) g2;
						acc[i][3] += (double) g3;
					}
				}
			}
		}

		const float r_w = r_src >= 0 ? (float) a.weight[r_src] : 0.f;     // arrives during the epilogue below

		double psum = 0.0;
		#pragma unroll
		for(int i = 0; i < NCH; ++i) {
			const int c = threadIdx.x + i * NT;
			if(c >= chunks)
				continue;
			const float bv[4] = {bcol[i].x, bcol[i].y, bcol[i].z, bcol[i].w};
			double lam[4];
			float bnew[4];
			#pragma unroll
			for(int q = 0; q < 4; ++q) {
				const double s = acc[i][q] * (double) bv[q];                 // lda.cpp:217
				lam[q] = a.fused ? mstep_value(a.coef, lp[i][q], s) : s;
			}
			if(!a.fused) {
				if(a.peer_ranks > 0) {
					int64_t off;
					void* dst = peer_column(a, w, &off);
					if(a.peer_elem == 4) {
						reinterpret_cast<float4*>(static_cast<float*>(dst) + off)[c] = make_float4((float) lam[0], (float) lam[1], (float) lam[2], (float) lam[3]);
					} else {
						double2* out = reinterpret_cast<double2*>(static_cast<double*>(dst) + off) + 2 * c;
						out[0] = make_double2(lam[0], lam[1]);
						out[1] = make_double2(lam[2], lam[3]);
					}
				} else if(a.sstats32) {
					reinterpret_cast<float4*>(a.sstats32 + base)[c] = make_float4((float) lam[0], (float) lam[1], (float) lam[2], (float) lam[3]);
				} else {
					double2* out = reinterpret_cast<double2*>(a.sstats + base) + 2 * c;
					out[0] = make_double2(lam[0], lam[1]);
					out[1] = make_double2(lam[2], lam[3]);
				}
				continue;
			}
			double2* out = reinterpret_cast<double2*>(a.lambda + base) + 2 * c;
			__stcs(out, make_double2(lam[0], lam[1]));
			__stcs(out + 1, make_double2(lam[2], lam[3]));
			if(a.psi_partials) {
				#pragma unroll
				for(int q = 0; q < 4; ++q) {
					const double p = digamma(lam[q]);
					psum += p;
					bnew[q] = (float) exp(p - a.psi_rows[4 * c + q]);
				}
			} else if(a.write_beta) {
				#pragma unroll
				for(int q = 0; q < 4; ++q)
					bnew[q] = exp_digamma_scaled_f32(lam[q], ek[i][q]);
			}
			if(a.write_beta)
				__stcs(reinterpret_cast<float4*>(beta + base) + c, make_float4(bnew[0], bnew[1], bnew[2], bnew[3]));
		}
		if(a.fused && a.psi_partials) {
			const double total = block_sum(psum, scratch);
			if(threadIdx.x == 0)
				a.psi_partials[w] = total;
		}
		if(r_src >= 0) {
			s_row[buf ^ 1][threadIdx.x] = (long long) r_doc * row_bytes;
			s_w[buf ^ 1][threadIdx.x] = r_w;
		}
		__syncthreads();       // the next word's tokens are staged, this word's buffer is free
		buf ^= 1;
		t0 = n0; t1 = n1;
		n0 = nn0; n1 = nn1;
	}
}

template <typename TE, typename TB>
static void launch_scatter_t(const ScatterArgs& a, const DeviceDocs& docs, cudaStream_t s) {
	const int grid = std::min(a.V, sm_count() * 64);
	const int kpt = ceil_div(a.K, SCATTER_THREADS);
	if(kpt <= 1) k_scatter<TE, TB, 1><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
	else if(kpt <= 2) k_scatter<TE, TB, 2><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
	else if(kpt <= 4) k_scatter<TE, TB, 4><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
	else if(kpt <= 8) k_scatter<TE, TB, 8><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
	else if(kpt <= 16) k_scatter<TE, TB, 16><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
	else k_scatter<TE, TB, 32><<<grid, SCATTER_THREADS, 0, s>>>(a, docs);
}

void launch_scatter(const ScatterArgs& a, const DeviceDocs& docs, cudaStream_t s) {
	if(a.etheta_elem == 4 && a.beta_elem == 4 && a.K % 4 == 0 && a.K <= 4096) {
		const int words = a.v1 < 0 ? a.V : a.v1 - a.v0;
		if(words <= 0)
			return;
		const int grid = std::min(words, sm_count() * 64);
		const int chunks = a.K / 4;
		if(chunks <= 128) k_scatter_vec<128, 1, 4><<<grid, 128, 0, s>>>(a, docs);
		else if(chunks <= 256) k_scatter_vec<128, 2, 4><<<grid, 128, 0, s>>>(a, docs);
		else if(chunks <= 512) k_scatter_vec<256, 2, 4><<<grid, 256, 0, s>>>(a, docs);
		else k_scatter_vec<256, 4, 2><<<grid, 256, 0, s>>>(a, docs);
		return;
	}
	if(a.etheta_elem == 8 && a.beta_elem == 8) launch_scatter_t<double, double>(a, docs, s);
	else if(a.etheta_elem == 4 && a.beta_elem == 4) launch_scatter_t<float, float>(a, docs, s);
	else if(a.etheta_elem == 8 && a.beta_elem == 4) launch_scatter_t<double, float>(a, docs, s);
	else launch_scatter_t<float, double>(a, docs, s);
}

// ------------------------------------------------------------------------------------------------------------
// dense M-step (after a cross-GPU exchange of sstats) + beta-prep
// ------------------------------------------------------------------------------------------------------------
template <typename TB>
__global__ void __launch_bounds__(256) k_mstep(MStepArgs a) {
	__shared__ double scratch[32];
	TB* beta = static_cast<TB*>(a.beta);
	for(int w = blockIdx.x; w < a.V; w += gridDim.x) {
		double psum = 0.0;
		for(int k = threadIdx.x; k < a.K; k += blockDim.x) {
			const int64_t e = (int64_t) w * a.K + k;
			const double lp = a.coef.mode == MSTEP_BATCH ? 0.0 : a.lambda_prime[e];
			const double lam = mstep_value(a.coef, lp, a.sstats[e]);
			a.lambda[e] = lam;
			if(a.psi_partials) {
				const double p = digamma(lam);
				psum += p;
				if(a.write_beta)
					beta[e] = (TB) exp(p - a.psi_rows[k]);
			} else if(a.write_beta) {
				beta[e] = (TB) exp_digamma_for<TB>(lam, a.psi_rows[k]);
			}
		}
		if(a.psi_partials) {
			const double total = block_sum(psum, scratch);
			if(threadIdx.x == 0)
				a.psi_partials[w] = total;
		}
	}
}

void launch_mstep(const MStepArgs& a, cudaStream_t s) {
	const int block = block_for_k(a.K);
	const int grid = std::min(a.V, sm_count() * 16);
	if(a.beta_elem == 8) k_mstep<double><<<grid, block, 0, s>>>(a);
	else k_mstep<float><<<grid, block, 0, s>>>(a);
}

// ------------------------------------------------------------------------------------------------------------
// sharded M-step over NVLink peer memory (see kernels.cuh)
// ------------------------------------------------------------------------------------------------------------
template <typename TB, typename TS>
__global__ void __launch_bounds__(256) k_mstep_shard(ShardMStepArgs a) {
	__shared__ double scratch[32];
	const int K = a.K, G = a.nranks;
	const int chunks = K / 4;
	// exp(-psi(new row sum)) of this thread's first chunk of topics (the only one when K <= 4 * blockDim)
	float ek0[4] = {0.f, 0.f, 0.f, 0.f};
	if(sizeof(TB) == 4 && a.write_beta && !a.psi_partials && (int) threadIdx.x < chunks)
		for(int q = 0; q < 4; ++q)
			ek0[q] = (float) exp(-a.psi_rows[4 * threadIdx.x + q]);
	for(int w = a.v0 + blockIdx.x; w < a.v1; w += gridDim.x) {
		const int64_t base = (int64_t) w * K;
		double psum = 0.0;
		for(int c = threadIdx.x; c < chunks; c += blockDim.x) {
			float ek[4];
			#pragma unroll
			for(int q = 0; q < 4; ++q)
				ek[q] = c == (int) threadIdx.x ? ek0[q] : ((sizeof(TB) == 4 && a.write_beta && !a.psi_partials) ? (float) exp(-a.psi_rows[4 * c + q]) : 0.f);
			// pull: all ranks' partial columns in flight at once, summed in rank order (deterministic)
			// the G partial columns of this word, pushed here by the scatter kernels of all ranks; rank order
			double s4[4] = {0.0, 0.0, 0.0, 0.0};
			const int64_t slot = (int64_t) (w - a.v0) * K;
			const int64_t stride = (int64_t) a.shard_cap * K;
			if constexpr(sizeof(TS) == 8) {
				double2 part[TRLDA_MAX_RANKS][2];
				#pragma unroll
				for(int r = 0; r < TRLDA_MAX_RANKS; ++r)
					if(r < G) {
						const double2* src = reinterpret_cast<const double2*>(static_cast<const double*>(a.partials) + r * stride + slot) + 2 * c;
						part[r][0] = __ldcs(src);
						part[r][1] = __ldcs(src + 1);
					}
				#pragma unroll
				for(int r = 0; r < TRLDA_MAX_RANKS; ++r)
					if(r < G) {
						s4[0] += part[r][0].x; s4[1] += part[r][0].y; s4[2] += part[r][1].x; s4[3] += part[r][1].y;
					}
			} else {
				float4 part[TRLDA_MAX_RANKS];
				#pragma unroll
				for(int r = 0; r < TRLDA_MAX_RANKS; ++r)
					if(r < G)
						part[r] = __ldcs(reinterpret_cast<const float4*>(static_cast<const float*>(a.partials) + r * stride + slot) + c);
				#pragma unroll
				for(int r = 0; r < TRLDA_MAX_RANKS; ++r)
					if(r < G) {
						s4[0] += (double) part[r].x; s4[1] += (double) part[r].y; s4[2] += (double) part[r].z; s4[3] += (double) part[r].w;
					}
			}
			double lp[4] = {0.0, 0.0, 0.0, 0.0};
			if(a.coef.mode != MSTEP_BATCH) {
				const double2 p0 = __ldcs(reinterpret_cast<const double2*>(a.lambda_prime + base) + 2 * c);
				const double2 p1 = __ldcs(reinterpret_cast<const double2*>(a.lambda_prime + base) + 2 * c + 1);
				lp[0] = p0.x; lp[1] = p0.y; lp[2] = p1.x; lp[3] = p1.y;
			}
			double lam[4];
			TB bnew[4];
			#pragma unroll
			for(int q = 0; q < 4; ++q) {
				lam[q] = mstep_value(a.coef, lp[q], s4[q]);
				if(a.psi_partials) {
					const double p = digamma(lam[q]);
					psum += p;
					bnew[q] = (TB) exp(p - a.psi_rows[4 * c + q]);
				} else if(a.write_beta) {
					if constexpr(sizeof(TB) == 4)
						bnew[q] = exp_digamma_scaled_f32(lam[q], ek[q]);
					else
						bnew[q] = (TB) exp_digamma_for<TB>(lam[q], a.psi_rows[4 * c + q]);
				}
			}
			// push: the new columns go to every rank's replica
			#pragma unroll
			for(int r = 0; r < TRLDA_MAX_RANKS; ++r)
				if(r < G) {
					if(r == a.rank || a.broadcast_lambda) {
						double2* out = reinterpret_cast<double2*>(a.lambda[r] + base) + 2 * c;
						out[0] = make_double2(lam[0], lam[1]);
						out[1] = make_double2(lam[2], lam[3]);
					}
					if(a.write_beta) {
						TB* out = static_cast<TB*>(a.beta[r]) + base + 4 * c;
						if constexpr(sizeof(TB) == 4) {
							*reinterpret_cast<float4*>(out) = make_float4(bnew[0], bnew[1], bnew[2], bnew[3]);
						} else {
							reinterpret_cast<double2*>(out)[0] = make_double2(bnew[0], bnew[1]);
							reinterpret_cast<double2*>(out)[1] = make_double2(bnew[2], bnew[3]);
						}
					}
				}
		}
		if(a.psi_partials) {
			const double total = block_sum(psum, scratch);
			if(threadIdx.x == 0)
				a.psi_partials[w] = total;
		}
	}
}

void launch_mstep_shard(const ShardMStepArgs& a, cudaStream_t s) {
	const int words = a.v1 - a.v0;
	if(words <= 0)
		return;
	const int block = std::min(256, std::max(32, round_up(a.K / 4, 32)));
	const int grid = std::min(words, sm_count() * 8);
	if(a.beta_elem == 8 && a.sstats_elem == 8) k_mstep_shard<double, double><<<grid, block, 0, s>>>(a);
	else if(a.beta_elem == 4 && a.sstats_elem == 4) k_mstep_shard<float, float><<<grid, block, 0, s>>>(a);
	else if(a.beta_elem == 4) k_mstep_shard<float, double><<<grid, block, 0, s>>>(a);
	else k_mstep_shard<double, float><<<grid, block, 0, s>>>(a);
}

// ------------------------------------------------------------------------------------------------------------
// phi = 1/K warm start (onlinelda.cpp:79-86) + beta-prep
// ------------------------------------------------------------------------------------------------------------
// wordcount[w] = sum of the counts of word w over the minibatch (onlinelda.cpp:79-82).  Atomic adds of integers
// held in doubles are exact, hence order-independent: the result is deterministic and needs no word-sorted list.
__global__ void __launch_bounds__(256) k_wordcount(DeviceDocs docs, double* __restrict__ wordcount) {
	const int64_t t = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if(t < docs.N)
		atomicAdd(wordcount + docs.word_ids[t], (double) docs.counts[t]);
}

void launch_wordcount(const DeviceDocs& docs, int V, double* wordcount, cudaStream_t s) {
	cudaMemsetAsync(wordcount, 0, sizeof(double) * V, s);
	if(docs.N > 0)
		k_wordcount<<<(unsigned) ((docs.N + 255) / 256), 256, 0, s>>>(docs, wordcount);
}

template <typename TB>
__global__ void __launch_bounds__(256) k_init_update(int K, int V, double rho, double eta, double scale_k,
                                                     const double* __restrict__ lambda_prime, double* __restrict__ lambda,
                                                     const double* __restrict__ psi_rows, TB* __restrict__ beta,
                                                     const double* __restrict__ wordcount, bool use_ek) {
	// float32 beta: exp(-psi(row sum)) once per topic and CTA (shared memory), then the float32 evaluation the fused
	// M-step kernel uses for every later beta of the step
	extern __shared__ float init_ek[];
	const bool fast = sizeof(TB) == 4 && use_ek;
	if(fast) {
		for(int k = threadIdx.x; k < K; k += blockDim.x)
			init_ek[k] = (float) exp(-psi_rows[k]);
		__syncthreads();
	}
	for(int w = blockIdx.x; w < V; w += gridDim.x) {
		const double target = rho * (eta + scale_k * wordcount[w]);     // onlinelda.cpp:86
		for(int k = threadIdx.x; k < K; k += blockDim.x) {
			const int64_t e = (int64_t) w * K + k;
			const double lam = (1. - rho) * lambda_prime[e] + target;   // onlinelda.cpp:85
			lambda[e] = lam;
			if(fast)
				beta[e] = (TB) exp_digamma_scaled_f32(lam, init_ek[k]);
			else
				beta[e] = (TB) exp_digamma_for<TB>(lam, psi_rows[k]);
		}
	}
}

void launch_init_update(const DeviceDocs& docs, int K, int V, double rho, double eta, double scale_k,
                        const double* lambda_prime, double* lambda, const double* psi_rows, void* beta,
                        int beta_elem, const double* wordcount, cudaStream_t s) {
	const int block = block_for_k(K);
	const int grid = std::min(V, sm_count() * 16);
	if(beta_elem == 8)
		k_init_update<double><<<grid, block, 0, s>>>(K, V, rho, eta, scale_k, lambda_prime, lambda, psi_rows,
		                                              static_cast<double*>(beta), wordcount, false);
	else
	{
		const bool use_ek = (size_t) K * sizeof(float) <= 48 * 1024;
		k_init_update<float><<<grid, block, use_ek ? (size_t) K * sizeof(float) : 0, s>>>(K, V, rho, eta, scale_k, lambda_prime, lambda,
		                                             psi_rows, static_cast<float*>(beta), wordcount, use_ek);
	}
}

// ------------------------------------------------------------------------------------------------------------
// column sums over documents of a K x B matrix: out[k] = sum_d in[k + d*K]
// ------------------------------------------------------------------------------------------------------------
constexpr int COLSUM_CHUNK = 64;

int colsum_num_partials(int64_t B) { return std::max(1, ceil_div(B, COLSUM_CHUNK)); }

__global__ void __launch_bounds__(256) k_colsum_partial(const double* __restrict__ in, int K, int64_t B, double* __restrict__ partials) {
	const int k = blockIdx.y * 256 + threadIdx.x;
	if(k >= K)
		return;
	const int64_t d0 = (int64_t) blockIdx.x * COLSUM_CHUNK, d1 = min(B, d0 + COLSUM_CHUNK);
	double acc = 0.0;
	for(int64_t d = d0; d < d1; ++d)
		acc += in[d * K + k];
	partials[(int64_t) blockIdx.x * K + k] = acc;
}

void launch_colsum(const double* in, int K, int64_t B, double* partials, double* out, cudaStream_t s) {
	const int P = colsum_num_partials(B);
	k_colsum_partial<<<dim3(P, ceil_div(K, 256)), 256, 0, s>>>(in, K, B, partials);
	k_reduce_partials<<<ceil_div(K, 256), 256, 0, s>>>(partials, P, K, out);
}

// ------------------------------------------------------------------------------------------------------------
// alpha statistics: stat_dk = psi(gamma_dk) - psi(sum_k gamma_dk)   (onlinelda.cpp:124-128)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_alpha_stats(const double* __restrict__ gamma, int K, int64_t B, double* __restrict__ stat) {
	__shared__ double scratch[32];
	for(int64_t d = blockIdx.x; d < B; d += gridDim.x) {
		double local = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x)
			local += gamma[d * K + k];
		const double psi_sum = digamma(block_sum(local, scratch));
		for(int k = threadIdx.x; k < K; k += blockDim.x)
			stat[d * K + k] = digamma(gamma[d * K + k]) - psi_sum;
	}
}

void launch_alpha_stats(const double* gamma, int K, int64_t B, double* stat, cudaStream_t s) {
	if(B == 0)
		return;
	k_alpha_stats<<<(unsigned) std::min<int64_t>(B, sm_count() * 16), block_for_k(K), 0, s>>>(gamma, K, B, stat);
}

// ------------------------------------------------------------------------------------------------------------
// Gamma(100, 1/100) generator for the initial gamma (lda.cpp:135) and lambda (lda.cpp:71).
// Counter-based (Philox4x32-10 keyed by seed, counter = element index and draw number), Marsaglia–Tsang
// rejection with Box–Muller normals: the value of element i depends only on (seed, stream, i).
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_gamma_rng(double* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream_id) {
	const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n)
		return;
	const double shape = 100.0;
	const double dd = shape - 1.0 / 3.0, cc = 1.0 / sqrt(9.0 * dd);
	double result = shape;
	for(uint32_t attempt = 0; attempt < 64; ++attempt) {
		uint32_t c[4] = {(uint32_t) i, (uint32_t) ((uint64_t) i >> 32), (uint32_t) stream_id, attempt};
		philox4x32(c, (uint32_t) seed, (uint32_t) (seed >> 32));
		// two uniforms in (0,1) with 32+21 bits, one more with 32 bits
		const double u1 = ((double) c[0] + 0.5) * (1.0 / 4294967296.0);
		const double u2 = ((double) c[1] + 0.5) * (1.0 / 4294967296.0);
		const double u3 = ((double) c[2] + 0.5) * (1.0 / 4294967296.0);
		const double x = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
		const double t = 1.0 + cc * x;
		if(t <= 0.0)
			continue;
		const double v = t * t * t;
		if(log(u3) < 0.5 * x * x + dd - dd * v + dd * log(v)) {
			result = dd * v;
			break;
		}
	}
	out[i] = result / shape;
}

void launch_gamma_rng(double* out, int64_t n, uint64_t seed, uint64_t stream_id, cudaStream_t s) {
	if(n > 0)
		k_gamma_rng<<<(unsigned) ((n + 255) / 256), 256, 0, s>>>(out, n, seed, stream_id);
}

// ------------------------------------------------------------------------------------------------------------
// Collapsed Gibbs E-step (lda.cpp:224-293).  One warp per document (documents are independent given expElogbeta,
// the sweep over a document's tokens is inherently sequential).  Per token occurrence the topic is drawn from
// p(k) ~ expElogbeta[k, w] * counts[k] (counts = alpha + the document's other assignments): lane l owns the topics
// k = l (mod 32), the 32 partial sums are scanned across the warp, the owning lane walks its topics.  Any fixed order
// of the categories gives the same distribution; the reference's order (k ascending, utils.cpp:189-199) is not kept.
// Random numbers: Philox4x32-10 keyed by the seed, counter = (document, draw) — results do not depend on the launch
// shape.  Two deliberate departures from the reference, which is only smoke-tested there:
//   * lda.cpp:254 initialises the assignments of document i from theta.col(j), j being the TOKEN index (reads past
//     the matrix once a document has more pairs than the minibatch has documents); theta.col(i) is used here;
//   * lda.cpp:284 adds into the shared sstats from all OpenMP threads without synchronisation; here atomicAdd.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double gibbs_uniform(uint64_t seed, uint32_t stream, uint64_t doc, uint32_t draw) {
	uint32_t c[4] = {(uint32_t) doc, (uint32_t) (doc >> 32), stream, draw};
	philox4x32(c, (uint32_t) seed, (uint32_t) (seed >> 32));
	return ((double) c[0] * 4294967296.0 + (double) c[1]) * (1.0 / 18446744073709551616.0);   // [0, 1)
}

// Gamma(shape, 1), shape > 0: Marsaglia–Tsang for shape >= 1, boosted by U^(1/shape) below 1
__device__ double gibbs_gamma(double shape, uint64_t seed, uint64_t doc, uint32_t element) {
	const double a = shape < 1.0 ? shape + 1.0 : shape;
	const double dd = a - 1.0 / 3.0, cc = 1.0 / sqrt(9.0 * dd);
	double result = a;
	for(uint32_t attempt = 0; attempt < 64; ++attempt) {
		uint32_t c[4] = {(uint32_t) doc, (uint32_t) (doc >> 32) ^ (element << 8), 0x9e3779b9u + element, attempt};
		philox4x32(c, (uint32_t) seed ^ 0x5bd1e995u, (uint32_t) (seed >> 32));
		const double u1 = ((double) c[0] + 0.5) * (1.0 / 4294967296.0);
		const double u2 = ((double) c[1] + 0.5) * (1.0 / 4294967296.0);
		const double u3 = ((double) c[2] + 0.5) * (1.0 / 4294967296.0);
		const double x = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
		const double t = 1.0 + cc * x;
		if(t <= 0.0)
			continue;
		const double v = t * t * t;
		if(log(u3) < 0.5 * x * x + dd - dd * v + dd * log(v)) {
			result = dd * v;
			if(shape < 1.0) {
				const double u4 = ((double) c[3] + 0.5) * (1.0 / 4294967296.0);
				result *= exp(log(u4) / shape);
			}
			break;
		}
	}
	return result;
}

// draws k with probability proportional to beta_col[k] * factor[k]; all lanes return the same k
template <typename TB>
__device__ __forceinline__ int gibbs_draw(const TB* __restrict__ beta_col, const double* factor, int K, double u, int lane) {
	double partial = 0.0;
	for(int k = lane; k < K; k += 32)
		partial += (double) beta_col[k] * factor[k];
	double scan = partial;
	#pragma unroll
	for(int o = 1; o < 32; o <<= 1) {
		const double other = __shfl_up_sync(0xffffffffu, scan, o);
		if(lane >= o)
			scan += other;
	}
	const double total = __shfl_sync(0xffffffffu, scan, 31);
	const double r = u * total;
	const unsigned above = __ballot_sync(0xffffffffu, scan > r && partial > 0.0);
	// rounding can leave no lane above r: fall back to the last lane that has mass at all
	const unsigned mass = __ballot_sync(0xffffffffu, partial > 0.0);
	int owner = above ? __ffs(above) - 1 : (mass ? 31 - __clz(mass) : 0);
	int k_found = owner < K ? owner : 0;
	if(lane == owner) {
		double left = r - (scan - partial);
		int last = lane;
		for(int k = lane; k < K; k += 32) {
			const double w = (double) beta_col[k] * factor[k];
			if(w > 0.0) {
				last = k;
				if(left < w)
					break;
				left -= w;
			}
		}
		k_found = last;
	}
	return __shfl_sync(0xffffffffu, k_found, owner);
}

template <typename TB>
__global__ void __launch_bounds__(128) k_gibbs(DeviceDocs docs, int K, const TB* __restrict__ beta, const double* __restrict__ alpha,
                                                const double* __restrict__ theta0, const int64_t* __restrict__ occ_ptr,
                                                uint16_t* __restrict__ topics, int num_samples, int burn_in, uint64_t seed,
                                                double* __restrict__ theta_out, double* __restrict__ sstats) {
	extern __shared__ __align__(16) unsigned char gibbs_smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
	double* counts = reinterpret_cast<double*>(gibbs_smem) + (size_t) warp * K;
	const double unit = 1.0 / (double) num_samples;                      // lda.cpp:232
	for(int64_t d = (int64_t) blockIdx.x * warps + warp; d < docs.B; d += (int64_t) gridDim.x * warps) {
		const int64_t begin = docs.doc_ptr[d], end = docs.doc_ptr[d + 1];
		uint16_t* z = topics + occ_ptr[d];
		uint32_t draw = 0;
		// initial theta: the caller's (lda.cpp:142-147) or Dirichlet(1) (lda.cpp:123-126): normalised Exp(1) draws
		double norm = 0.0;
		for(int k = lane; k < K; k += 32) {
			const double t = theta0 ? theta0[d * K + k] : -log(1.0 - gibbs_uniform(seed, 1u, (uint64_t) d, (uint32_t) k));
			counts[k] = t;
			norm += t;
		}
		norm = warp_sum(norm);
		__syncwarp();
		// initial assignments from p(k) ~ beta[k, w] theta[k] (blocked Gibbs, lda.cpp:247-263)
		int64_t o = 0;
		for(int64_t j = begin; j < end; ++j) {
			const TB* col = beta + (int64_t) docs.word_ids[j] * K;
			for(int c = 0; c < docs.counts[j]; ++c, ++o) {
				const int k = gibbs_draw(col, counts, K, gibbs_uniform(seed, 2u, (uint64_t) d, draw++), lane);
				if(lane == 0)
					z[o] = (uint16_t) k;
			}
		}
		__syncwarp();
		// counts = alpha + occurrences of each topic (lda.cpp:244, 261)
		for(int k = lane; k < K; k += 32)
			counts[k] = alpha[k];
		__syncwarp();
		if(lane == 0)
			for(int64_t i = 0; i < o; ++i)
				counts[z[i]] += 1.0;
		__syncwarp();
		for(int s = 0; s < num_samples + burn_in; ++s) {                   // lda.cpp:265-288
			o = 0;
			for(int64_t j = begin; j < end; ++j) {
				const int w = docs.word_ids[j];
				const TB* col = beta + (int64_t) w * K;
				for(int c = 0; c < docs.counts[j]; ++c, ++o) {
					if(lane == 0)
						counts[z[o]] -= 1.0;
					__syncwarp();
					const int k = gibbs_draw(col, counts, K, gibbs_uniform(seed, 3u, (uint64_t) d, draw++), lane);
					if(lane == 0) {
						z[o] = (uint16_t) k;
						counts[k] += 1.0;
						if(s >= burn_in)
							atomicAdd(sstats + (int64_t) w * K + k, unit);     // lda.cpp:278-286
					}
					__syncwarp();
				}
			}
		}
		// theta ~ Dirichlet(counts) (lda.cpp:291)
		double sum = 0.0;
		for(int k = lane; k < K; k += 32) {
			const double g = gibbs_gamma(counts[k], seed, (uint64_t) d, (uint32_t) k);
			counts[k] = g;
			sum += g;
		}
		sum = warp_sum(sum);
		for(int k = lane; k < K; k += 32)
			theta_out[d * K + k] = counts[k] / sum;
		__syncwarp();
	}
}

void launch_gibbs(const DeviceDocs& docs, int K, const void* beta, int beta_elem, const double* alpha, const double* theta0,
                  const int64_t* occ_ptr, uint16_t* topics, int num_samples, int burn_in, uint64_t seed, double* theta_out,
                  double* sstats, cudaStream_t s) {
	if(docs.B == 0)
		return;
	const int warps = 4;
	const size_t smem = (size_t) warps * K * sizeof(double);
	const unsigned grid = (unsigned) std::min<int64_t>((docs.B + warps - 1) / warps, sm_count() * 8);
	if(beta_elem == 4) {
		cudaFuncSetAttribute(k_gibbs<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
		k_gibbs<float><<<grid, warps * 32, smem, s>>>(docs, K, static_cast<const float*>(beta), alpha, theta0, occ_ptr, topics,
		                                              num_samples, burn_in, seed, theta_out, sstats);
	} else {
		cudaFuncSetAttribute(k_gibbs<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
		k_gibbs<double><<<grid, warps * 32, smem, s>>>(docs, K, static_cast<const double*>(beta), alpha, theta0, occ_ptr, topics,
		                                               num_samples, burn_in, seed, theta_out, sstats);
	}
}

__global__ void k_fill(double* __restrict__ out, int64_t n, double v) {
	const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if(i < n)
		out[i] = v;
}

void launch_fill(double* out, int64_t n, double value, cudaStream_t s) {
	if(n > 0)
		k_fill<<<(unsigned) ((n + 255) / 256), 256, 0, s>>>(out, n, value);
}

// ------------------------------------------------------------------------------------------------------------
// deterministic sum of n doubles
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sum_partial(const double* __restrict__ in, int64_t n, double* __restrict__ partials) {
	__shared__ double scratch[32];
	double acc = 0.0;
	for(int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x)
		acc += in[i];
	const double total = block_sum(acc, scratch);
	if(threadIdx.x == 0)
		partials[blockIdx.x] = total;
}

__global__ void k_sum_final(const double* __restrict__ partials, int P, double* __restrict__ out) {
	if(threadIdx.x == 0 && blockIdx.x == 0) {
		double acc = 0.0;
		for(int p = 0; p < P; ++p)
			acc += partials[p];
		out[0] = acc;
	}
}

void launch_sum(const double* in, int64_t n, double* partials, double* out, cudaStream_t s) {
	const int P = (int) std::max<int64_t>(1, std::min<int64_t>(1024, (n + 255) / 256));
	k_sum_partial<<<P, 256, 0, s>>>(in, n, partials);
	k_sum_final<<<1, 32, 0, s>>>(partials, P, out);
}

// ------------------------------------------------------------------------------------------------------------
// adaptive learning rate state (onlinelda.cpp:167-175)
// ------------------------------------------------------------------------------------------------------------
int adaptive_num_blocks(int64_t n) { return (int) std::max<int64_t>(1, std::min<int64_t>(1024, (n + 255) / 256)); }

__global__ void __launch_bounds__(256) k_adaptive(const double* __restrict__ sstats, const double* __restrict__ lambda_prime,
                                                  double* __restrict__ grad, int64_t n, double eta, double scale, double tau,
                                                  double* __restrict__ sq_partials) {
	__shared__ double scratch[32];
	double su = 0.0, sg = 0.0;
	for(int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
		const double u = (eta + scale * sstats[i]) - lambda_prime[i];     // lambdaHat - lambdaPrime, :168
		const double g = (1. - 1. / tau) * grad[i] + 1. / tau * u;        // :171
		grad[i] = g;
		su += u * u;
		sg += g * g;
	}
	const double tu = block_sum(su, scratch);
	const double tg = block_sum(sg, scratch);
	if(threadIdx.x == 0) {
		sq_partials[blockIdx.x] = tu;
		sq_partials[gridDim.x + blockIdx.x] = tg;
	}
}

void launch_adaptive(const double* sstats, const double* lambda_prime, double* grad, int64_t n, double eta,
                     double scale, double tau, double* sq_partials, cudaStream_t s) {
	k_adaptive<<<adaptive_num_blocks(n), 256, 0, s>>>(sstats, lambda_prime, grad, n, eta, scale, tau, sq_partials);
}

// ------------------------------------------------------------------------------------------------------------
// variational lower bound (intended formula; see include/trlda_b200.h)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_elbo_docs(DeviceDocs docs, int K, const double* __restrict__ lambda,
                                                   const double* __restrict__ psi_rows, const double* __restrict__ alpha,
                                                   double alpha_const, const double* __restrict__ gamma, double* __restrict__ per_doc) {
	extern __shared__ double elogtheta[];   // K
	__shared__ double scratch[32];
	for(int64_t d = blockIdx.x; d < docs.B; d += gridDim.x) {
		const double* g = gamma + d * K;
		double local = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x)
			local += g[k];
		const double gsum = block_sum(local, scratch);
		const double psi_gsum = digamma(gsum);
		double score = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x) {
			const double e = digamma(g[k]) - psi_gsum;                   // lda.cpp:341
			elogtheta[k] = e;
			score += (alpha[k] - g[k]) * e + lgamma(g[k]);               // lda.cpp:349-351
		}
		__syncthreads();
		for(int64_t j = docs.doc_ptr[d]; j < docs.doc_ptr[d + 1]; ++j) {
			const double* col = lambda + (int64_t) docs.word_ids[j] * K;
			// log sum_k exp(Elogtheta_k + Elogbeta_kw), max-subtracted (onlineldavb.py:289-296)
			double tmax = -CUDART_INF;
			for(int k = threadIdx.x; k < K; k += blockDim.x)
				tmax = fmax(tmax, elogtheta[k] + digamma(col[k]) - psi_rows[k]);
			#pragma unroll
			for(int o = 16; o > 0; o >>= 1)
				tmax = fmax(tmax, __shfl_xor_sync(0xffffffffu, tmax, o));
			__syncthreads();
			if((threadIdx.x & 31) == 0)
				scratch[threadIdx.x >> 5] = tmax;
			__syncthreads();
			for(int i = 0; i < (int) ((blockDim.x + 31) >> 5); ++i)
				tmax = fmax(tmax, scratch[i]);
			double sum = 0.0;
			for(int k = threadIdx.x; k < K; k += blockDim.x)
				sum += exp(elogtheta[k] + digamma(col[k]) - psi_rows[k] - tmax);
			sum = block_sum(sum, scratch);
			if(threadIdx.x == 0)
				score += docs.counts[j] * (log(sum) + tmax);
		}
		score = block_sum(score, scratch);
		if(threadIdx.x == 0)
			per_doc[d] = score - lgamma(gsum) + alpha_const;
		__syncthreads();
	}
}

void launch_elbo_docs(const DeviceDocs& docs, int K, const double* lambda, const double* psi_rows,
                      const double* alpha, double alpha_const, const double* gamma, double* per_doc, cudaStream_t s) {
	if(docs.B == 0)
		return;
	k_elbo_docs<<<(unsigned) std::min<int64_t>(docs.B, sm_count() * 8), block_for_k(K), (size_t) K * 8, s>>>(
		docs, K, lambda, psi_rows, alpha, alpha_const, gamma, per_doc);
}

__global__ void __launch_bounds__(256) k_elbo_beta(const double* __restrict__ lambda, const double* __restrict__ psi_rows,
                                                   int K, int V, double eta, double* __restrict__ partial) {
	__shared__ double scratch[32];
	for(int w = blockIdx.x; w < V; w += gridDim.x) {
		double acc = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x) {
			const double l = lambda[(int64_t) w * K + k];
			acc += (eta - l) * (digamma(l) - psi_rows[k]) + lgamma(l);   // lda.cpp:317 (beta part), :357
		}
		const double total = block_sum(acc, scratch);
		if(threadIdx.x == 0)
			partial[w] = total;
	}
}

void launch_elbo_beta(const double* lambda, const double* psi_rows, int K, int V, double eta, double* partial,
                      cudaStream_t s) {
	k_elbo_beta<<<std::min(V, sm_count() * 16), block_for_k(K), 0, s>>>(lambda, psi_rows, K, V, eta, partial);
}

// ------------------------------------------------------------------------------------------------------------
// document-completion predictive log-likelihood (Hoffman, Blei, Wang & Paisley 2013, section 5)
// ------------------------------------------------------------------------------------------------------------
// One CTA per document.  s_d = gamma_d / rows goes to shared memory; warp w then takes the groups of HELDOUT_GROUP
// consecutive held-out pairs g = w, w + nw, ... and walks their lambda columns side by side, so that every lane has
// HELDOUT_GROUP independent loads in flight per step (a lane walking one column at a time is bound by L2 latency).
// Each dot product is reduced with xor shuffles, which leave the same bits in every lane; the warp partials are added in
// warp order.  The result of a document therefore depends on K alone (through the block size), not on the launch.
constexpr int HELDOUT_GROUP = 4;

__global__ void __launch_bounds__(256) k_heldout_loglik(DeviceDocs docs, int K, const double* __restrict__ lambda,
                                                        const double* __restrict__ rows, const double* __restrict__ gamma,
                                                        double* __restrict__ per_doc) {
	extern __shared__ double s[];   // K
	__shared__ double scratch[32], partial[32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
	for(int64_t d = blockIdx.x; d < docs.B; d += gridDim.x) {
		const double* g = gamma + d * K;
		double local = 0.0;
		for(int k = threadIdx.x; k < K; k += blockDim.x) {
			const double v = g[k];
			s[k] = v / rows[k];
			local += v;
		}
		const double log_gsum = log(block_sum(local, scratch));   // the barriers of block_sum also publish s
		const int64_t end = docs.doc_ptr[d + 1];
		double acc = 0.0;
		for(int64_t j0 = docs.doc_ptr[d] + (int64_t) warp * HELDOUT_GROUP; j0 < end; j0 += (int64_t) nw * HELDOUT_GROUP) {
			const double* col[HELDOUT_GROUP];
			double dot[HELDOUT_GROUP];
			#pragma unroll
			for(int p = 0; p < HELDOUT_GROUP; ++p) {
				// a slot past the document's end re-reads the group's first column and is not counted
				col[p] = lambda + (int64_t) docs.word_ids[j0 + p < end ? j0 + p : j0] * K;
				dot[p] = 0.0;
			}
			#pragma unroll 2
			for(int k = lane; k < K; k += 32) {
				const double sk = s[k];
				#pragma unroll
				for(int p = 0; p < HELDOUT_GROUP; ++p)
					dot[p] = fma(sk, __ldg(col[p] + k), dot[p]);
			}
			#pragma unroll
			for(int p = 0; p < HELDOUT_GROUP; ++p) {
				const double total = warp_sum(dot[p]);
				if(j0 + p < end)
					acc += docs.counts[j0 + p] * (log(total) - log_gsum);
			}
		}
		if(lane == 0)
			partial[warp] = acc;
		__syncthreads();   // also: every warp is done with s before the next document overwrites it
		if(threadIdx.x == 0) {
			double total = 0.0;
			for(int i = 0; i < nw; ++i)
				total += partial[i];
			per_doc[d] = total;
		}
	}
}

void launch_heldout_loglik(const DeviceDocs& held_out, int K, const double* lambda, const double* rows, const double* gamma,
                           double* per_doc, cudaStream_t s) {
	if(held_out.B == 0)
		return;
	k_heldout_loglik<<<(unsigned) std::min<int64_t>(held_out.B, sm_count() * 8), block_for_k(K), (size_t) K * 8, s>>>(
		held_out, K, lambda, rows, gamma, per_doc);
}

// ------------------------------------------------------------------------------------------------------------
// special-function test hook
// ------------------------------------------------------------------------------------------------------------
__global__ void k_special(int which, const double* __restrict__ x, int64_t n, double* __restrict__ out) {
	const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
	if(i >= n)
		return;
	const double v = x[i];
	double r;
	switch(which) {
		case 0: r = digamma(v); break;
		case 1: r = trigamma(v); break;
		case 2: r = lgamma(v); break;
		case 3: r = exp_digamma_shifted_mixed(v, 0.0); break;
		case 5: r = exp_digamma_lean(v); break;
		default: r = exp_digamma_shifted(v, 0.0); break;
	}
	out[i] = r;
}

void launch_special(int which, const double* x, int64_t n, double* out, cudaStream_t s) {
	if(n > 0)
		k_special<<<(unsigned) ((n + 127) / 128), 128, 0, s>>>(which, x, n, out);
}

}  // namespace trlda
