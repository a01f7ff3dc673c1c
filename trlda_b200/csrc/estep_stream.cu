// estep_stream.cu — the per-document E-step (lda.cpp:174-204 of the reference), streaming design (the default path).
//
// The K x n_d tile of expElogbeta columns of a document is NOT kept on chip (150 columns x 4 KB at cfg-3: no SM holds
// it); it is streamed once per inner iteration.  Every warp pulls its own columns (K contiguous values each) through a
// private shared-memory ring — one `cp.async.bulk` per column, issued by one lane, completing on the slot's mbarrier
// (16-byte `cp.async` for columns shorter than 2 KB); there is no block-wide barrier on the data path — and, because a
// warp sees a complete column, the two passes of the reference's inner iteration fuse into ONE sweep:
//
//     phi_j = etheta . col_j  (+1e-100)      lda.cpp:183,199      warp-shuffle reduction over the K rows
//     W_j   = c_j / phi_j                    lda.cpp:192
//     acc  += W_j col_j                      lda.cpp:189-193      lane-local: every lane keeps its rows in registers
//
// After a sweep the per-warp partial sums meet in shared memory (fixed order: deterministic), gamma and
// exp(psi(gamma)) are updated (lda.cpp:194-197) and the convergence test of lda.cpp:202 is evaluated.  I inner
// iterations cost I+1 sweeps (the last one produces the token weights and the document's share of the row sums of
// the sufficient statistics); the first sweep comes from HBM, the re-sweeps from L2 (148 documents x 600 KB in flight).
//
// Launch shape: one CTA of 16 warps per document (fp32 tile; 8 warps for the fp64 tile and for short columns), handed
// out by the hardware scheduler, two ring slots per warp.  Measured at cfg-3 (fresh minibatch per step), and lost
// (DESIGN.md §4): clusters of 2 CTAs per document that split the columns and exchange their partial sums per sweep
// (102 ms/step against 74); with the bulk-copy ring, 12 warps x 3 slots (59.5 ms/step of E-step against 56.9),
// 12 x 2 (60.3) and 8 x 4 (75.1): warps, not slots; a persistent grid (7 % slower: the documents of a CTA differ in
// sweeps).
#include "kernels.cuh"
#include "special.cuh"

#include <algorithm>

namespace trlda {

constexpr int STREAM_DEPTH = 2;    // ring slots per warp

template <typename T> struct SVec;
template <> struct SVec<float> { using type = float4; static constexpr int N = 4; };
template <> struct SVec<double> { using type = double2; static constexpr int N = 2; };

__device__ __forceinline__ void svec_get(const float4& v, float (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ void svec_get(const double2& v, double (&o)[2]) { o[0] = v.x; o[1] = v.y; }


// how many per-warp partial vectors meet in shared memory at once: above 64 KB the warps fold pairwise first
__host__ __device__ constexpr int stream_reduce_width(int NW, int kp, int elem) {
	return (NW * kp * elem > 65536 && NW % 2 == 0) ? NW / 2 : NW;
}

struct StreamSmem {
	size_t ring, red, eth, gam, wsum, wid, cnt, rbar, total;
};

__host__ __device__ inline StreamSmem stream_smem_layout(int NW, int kp, int n_cap, int elem) {
	StreamSmem L;
	size_t o = 0;
	auto take = [&o](size_t bytes) { size_t at = o; o += (bytes + 15) & ~size_t(15); return at; };
	L.ring = take((size_t) NW * STREAM_DEPTH * kp * elem);
	L.red = take((size_t) stream_reduce_width(NW, kp, elem) * kp * elem);
	L.eth = take((size_t) kp * elem);
	L.gam = take((size_t) kp * 8);
	L.wsum = take((size_t) NW * 8);
	L.wid = take((size_t) n_cap * 4);
	L.cnt = take((size_t) n_cap * 4);
	L.rbar = take((size_t) NW * STREAM_DEPTH * 8);         // one mbarrier per ring slot (bulk-copy variant)
	L.total = o;
	return L;
}

static inline int stream_nvec(int K, int elem) {
	const int per_sweep = 32 * (16 / elem);
	int nvec = 1;
	while(nvec * per_sweep < K)
		nvec *= 2;
	return nvec;
}

// Columns of 2 KB and more travel by cp.async.bulk (one copy per column, written by the copy engine); 16-byte cp.async
// (LDGSTS) costs the load/store pipe 8 cycles per 512 bytes: 63.8 against 56.9 ms/step of E-step at cfg-3.  Short
// columns (K = 100 or 200: 400-1600 bytes) stay with cp.async, the per-copy cost of the bulk path does not pay: cfg-5
// (K = 200) 117 ms per batch with bulk copies and one 16-warp CTA per SM against 33 ms with two 8-warp CTAs.
static bool stream_bulk(int K, int elem) { return K * elem >= 2048; }
static int stream_warps(int K, int elem) { return elem == 4 && stream_bulk(K, elem) ? 16 : 8; }

// applicable?  (aligned columns, K small enough for the per-lane register tile, everything fits in shared memory)
bool stream_estep_applicable(int K, int n_max, int elem, int smem_optin) {
	if((K * elem) % 16 != 0)
		return false;
	const int nvec = stream_nvec(K, elem);
	if(nvec > (elem == 4 ? 8 : 16))
		return false;
	const int kp = nvec * 32 * (16 / elem);
	const int n_cap = std::max(32, (n_max + 31) / 32 * 32);
	return stream_smem_layout(stream_warps(K, elem), kp, n_cap, elem).total <= (size_t) smem_optin - 1024;
}

__device__ __forceinline__ uint32_t s_smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }

__device__ __forceinline__ void s_mbar_wait(uint32_t bar, uint32_t parity) {
	uint32_t done = 0;
	while(!done)
		asm volatile(
			"{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
			: "=r"(done) : "r"(bar), "r"(parity) : "memory");
}

template <typename T, int NW, int NVEC, bool BULK>
__global__ void __launch_bounds__(NW * 32, (NW == 8 && sizeof(T) == 4 ? 2 : 1))
k_estep_stream(EStepArgs a, DeviceDocs docs, const int32_t* __restrict__ order, int64_t doc_offset, int n_cap) {
	extern __shared__ __align__(128) unsigned char smem[];
	using V = typename SVec<T>::type;
	constexpr int VN = SVec<T>::N;
	constexpr int KP = NVEC * 32 * VN;                       // padded number of topic rows
	constexpr int NT = NW * 32;
	constexpr int RW = stream_reduce_width(NW, KP, (int) sizeof(T));
	const StreamSmem L = stream_smem_layout(NW, KP, n_cap, (int) sizeof(T));
	T* ring = reinterpret_cast<T*>(smem + L.ring);
	T* red = reinterpret_cast<T*>(smem + L.red);
	T* eth = reinterpret_cast<T*>(smem + L.eth);
	double* gam = reinterpret_cast<double*>(smem + L.gam);
	double* wsum = reinterpret_cast<double*>(smem + L.wsum);
	int* wid = reinterpret_cast<int*>(smem + L.wid);
	int* cnt = reinterpret_cast<int*>(smem + L.cnt);
	uint64_t* rbar = reinterpret_cast<uint64_t*>(smem + L.rbar);

	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int K = a.K;
	const T* __restrict__ beta = static_cast<const T*>(a.beta);

	// this lane's rows: vectors v = 0..NVEC-1 cover rows (v * 32 + lane) * VN .. + VN
	T* my_ring = ring + (size_t) warp * STREAM_DEPTH * KP;
	const uint32_t ring_addr = s_smem_u32(my_ring);
	const uint32_t rbar_addr = s_smem_u32(rbar + (size_t) warp * STREAM_DEPTH);
	// whole rounds of 32 vectors are moved, rows K..KP-1 of a column are the head of the next column (or the zeroed slack
	// behind the matrix): finite values that meet etheta = 0 in the dot product and rows nobody reads in the sums
	const uint32_t lane_bytes = (uint32_t) lane * 16u;
	const uint32_t col_bytes = (uint32_t) K * (uint32_t) sizeof(T);
	uint32_t phases = 0;                                           // bulk variant: parity of the next completion per slot
	auto issue = [&](int j, int stage) {                           // gather column j into ring slot `stage`
		if(BULK) {
			// one bulk copy of the K values per column, issued by one lane, written by the copy engine: the load/store
			// pipe only sees the LDS that read the column back (LDGSTS costs it 8 cycles per 512 bytes, LDS.128 4)
			if(lane == 0) {
				const T* src = beta + (int64_t) wid[j] * K;
				const uint32_t dst = ring_addr + (uint32_t) (stage * KP * (int) sizeof(T));
				const uint32_t mb = rbar_addr + 8u * (uint32_t) stage;
				asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(col_bytes) : "memory");
				asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
					::"r"(dst), "l"(src), "r"(col_bytes), "r"(mb) : "memory");
			}
		} else {
			const char* src = reinterpret_cast<const char*>(beta + (int64_t) wid[j] * K) + lane_bytes;
			const uint32_t dst = ring_addr + (uint32_t) (stage * KP * (int) sizeof(T)) + lane_bytes;
			#pragma unroll
			for(int v = 0; v < NVEC; ++v)
				asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + v * 512u), "l"(src + v * 512) : "memory");
		}
	};
	auto commit = [&]() {
		if(!BULK)
			asm volatile("cp.async.commit_group;" ::: "memory");
	};
	auto wait_slot = [&](int stage) {
		if(BULK) {
			s_mbar_wait(rbar_addr + 8u * (uint32_t) stage, (phases >> stage) & 1u);
			phases ^= 1u << stage;
		} else {
			asm volatile("cp.async.wait_group %0;" ::"n"(STREAM_DEPTH - 1) : "memory");
		}
	};
	if(BULK) {
		// the copies move K values, the lanes read KP: the tail of every slot is zeroed once
		for(int i = tid; i < NW * STREAM_DEPTH * (KP - K); i += NT)
			ring[(size_t) (i / (KP - K)) * KP + K + i % (KP - K)] = T(0);
		if(lane == 0) {
			for(int st = 0; st < STREAM_DEPTH; ++st)
				asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(rbar_addr + 8u * (uint32_t) st));
			asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
		}
		asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
		__syncthreads();
	}

	// debug phase timers (TRLDA_ESTEP_TICKS=1), thread 0's view: setup, stream, fold, update, test
	const bool timing = a.ticks != nullptr && tid == 0;
	long long tk[5] = {0, 0, 0, 0, 0}, t_mark = 0;
	#define TRLDA_TICK(i) if(timing) { const long long now = clock64(); tk[i] += now - t_mark; t_mark = now; }
	const int64_t slot = doc_offset + blockIdx.x;
	const int64_t d = order ? order[slot] : slot;
	const int64_t begin = docs.doc_ptr[d];
	const int n = (int) (docs.doc_ptr[d + 1] - begin);
	if(timing)
		t_mark = clock64();
	for(int j = tid; j < n; j += NT) {
		wid[j] = docs.word_ids[begin + j];
		cnt[j] = docs.counts[begin + j];
	}
	for(int r0 = tid; r0 < KP; r0 += 2 * NT) {                      // two rows per trip: their psi/exp chains overlap
		double g[2];
		T e[2];
		#pragma unroll
		for(int u = 0; u < 2; ++u) {
			const int r = r0 + u * NT;
			g[u] = r < K ? a.gamma[d * K + r] : 1.0;
		}
		#pragma unroll
		for(int u = 0; u < 2; ++u)
			e[u] = (T) exp_digamma_for<T>(g[u], 0.0);             // lda.cpp:174
		#pragma unroll
		for(int u = 0; u < 2; ++u) {
			const int r = r0 + u * NT;
			if(r < KP) {
				gam[r] = r < K ? g[u] : 0.0;
				eth[r] = r < K ? e[u] : T(0);
			}
		}
	}
	__syncthreads();

	TRLDA_TICK(0)
	int it = 0;
	bool converged = false;
	bool primed = false;   // the ring already holds the first columns of the coming sweep
	int stage = 0;
	while(true) {
		const bool final_sweep = converged || it >= a.max_iter;
		// ---- one sweep over the document's columns: this warp takes columns warp, warp + NW, ... ------------------------
		T e[NVEC][VN], acc[NVEC][VN];
		#pragma unroll
		for(int v = 0; v < NVEC; ++v) {
			svec_get(*reinterpret_cast<const V*>(eth + (v * 32 + lane) * VN), e[v]);
			#pragma unroll
			for(int q = 0; q < VN; ++q)
				acc[v][q] = T(0);
		}
		// M = number of columns of this warp.  If the ring was not primed by the previous sweep, fill it now.
		const int M = warp < n ? (n - warp + NW - 1) / NW : 0;
		if(!primed) {
			#pragma unroll
			for(int s = 0; s < STREAM_DEPTH; ++s) {
				if(s < M)
					issue(warp + s * NW, s);
				commit();
			}
			stage = 0;
		}
		// a non-final sweep is always followed by another one over the same columns: its first STREAM_DEPTH columns
		// are requested while the tail of this sweep is consumed, so the ring never drains at a sweep boundary and
		// the (L2) latency of the next sweep hides behind the reduction and the psi evaluations
		const bool prime_next = !final_sweep && M >= STREAM_DEPTH;
		for(int mcol = 0; mcol < M; ++mcol) {
			const int j = warp + mcol * NW;
			wait_slot(stage);
			__syncwarp();
			const T* col = my_ring + (size_t) stage * KP;
			T c[NVEC][VN];
			#pragma unroll
			for(int v = 0; v < NVEC; ++v)
				svec_get(*reinterpret_cast<const V*>(col + (v * 32 + lane) * VN), c[v]);
			T wt;
			if(sizeof(T) == 4) {
				// mixed mode: four independent float chains per lane, float butterfly over the warp, float division
				float part[4] = {0.f, 0.f, 0.f, 0.f};
				#pragma unroll
				for(int v = 0; v < NVEC; ++v)
					#pragma unroll
					for(int q = 0; q < VN; ++q)
						part[q & 3] = fmaf((float) e[v][q], (float) c[v][q], part[q & 3]);
				float phi = (part[0] + part[1]) + (part[2] + part[3]);
				#pragma unroll
				for(int o = 16; o > 0; o >>= 1)
					phi += __shfl_xor_sync(0xffffffffu, phi, o);
				// lda.cpp:183,192,199; the +1e-100 only matters at 0, where the weight must stay finite in float32
				wt = (T) fminf(__fdividef((float) cnt[j], fmaxf(phi, 1e-37f)), 1e30f);
			} else {
				double part = 0.0;
				#pragma unroll
				for(int v = 0; v < NVEC; ++v) {
					T chunk = e[v][0] * c[v][0];
					#pragma unroll
					for(int q = 1; q < VN; ++q)
						chunk = fma(e[v][q], c[v][q], chunk);
					part += (double) chunk;
				}
				const double phi = warp_sum(part) + 1e-100;                    // lda.cpp:183,199
				wt = (T) ((double) cnt[j] / phi);                              // lda.cpp:192
			}
			#pragma unroll
			for(int v = 0; v < NVEC; ++v)
				#pragma unroll
				for(int q = 0; q < VN; ++q)
					acc[v][q] = fma(wt, c[v][q], acc[v][q]);
			if(final_sweep && lane == 0)
				a.weight[begin + j] = (double) wt;
			__syncwarp();
			const int mn = mcol + STREAM_DEPTH;
			if(mn < M)
				issue(warp + mn * NW, stage);
			else if(prime_next)
				issue(warp + (mn - M) * NW, stage);
			commit();
			stage = stage + 1 == STREAM_DEPTH ? 0 : stage + 1;
		}
		primed = prime_next;
		if(!primed && !BULK)
			asm volatile("cp.async.wait_group 0;" ::: "memory");
		// ---- the per-warp partial sums meet in shared memory, fixed order ------------------------------------------------
		TRLDA_TICK(1)
		auto store_acc = [&](int slot) {
			#pragma unroll
			for(int v = 0; v < NVEC; ++v) {
				V out;
				T* o = reinterpret_cast<T*>(&out);
				#pragma unroll
				for(int q = 0; q < VN; ++q)
					o[q] = acc[v][q];
				*reinterpret_cast<V*>(red + (size_t) slot * KP + (v * 32 + lane) * VN) = out;
			}
		};
		if(RW < NW) {                                                  // upper half of the warps folds into the lower half
			if(warp >= RW)
				store_acc(warp - RW);
			__syncthreads();
			if(warp < RW) {
				#pragma unroll
				for(int v = 0; v < NVEC; ++v) {
					T other[VN];
					svec_get(*reinterpret_cast<const V*>(red + (size_t) warp * KP + (v * 32 + lane) * VN), other);
					#pragma unroll
					for(int q = 0; q < VN; ++q)
						acc[v][q] += other[q];
				}
			}
			__syncthreads();
			if(warp < RW)
				store_acc(warp);
		} else {
			store_acc(warp);
		}
		__syncthreads();

		TRLDA_TICK(2)
		double delta_local = 0.0;
		// two rows per thread and trip, so that their chains (sum of the partials, psi, exp) overlap
		for(int r0 = tid; r0 < K; r0 += 2 * NT) {
			double total[2], eo[2];
			int row[2];
			bool live[2];
			#pragma unroll
			for(int u = 0; u < 2; ++u) {
				live[u] = r0 + u * NT < K;
				row[u] = live[u] ? r0 + u * NT : r0;
				const int r = row[u];
				// the partials are T: they are added in T (mixed mode: one float32 rounding per partial, like the
				// accumulators themselves) and converted once — F2F.F64.F32 per partial was a cost of its own
				T part = red[r];
				#pragma unroll
				for(int q = 1; q < RW; ++q)
					part += red[(size_t) q * KP + r];
				total[u] = (double) part;
				eo[u] = (double) eth[r];
			}
			if(final_sweep) {
				#pragma unroll
				for(int u = 0; u < 2; ++u) {
					const int r = row[u];
					if(live[u]) {
						a.doc_stat[d * K + r] = total[u] * eo[u];
						a.gamma[d * K + r] = gam[r];
						a.etheta[d * K + r] = eo[u];
						if(a.etheta32)
							a.etheta32[d * K + r] = (float) eo[u];
					}
				}
			} else {                                                   // lda.cpp:186-197
				double g_new[2];
				T e_new[2];
				#pragma unroll
				for(int u = 0; u < 2; ++u) {
					g_new[u] = total[u] * eo[u];
					g_new[u] += a.alpha[row[u]];
				}
				#pragma unroll
				for(int u = 0; u < 2; ++u)
					e_new[u] = (T) exp_digamma_for<T>(g_new[u], 0.0);     // fp64 also in mixed mode: a float32 evaluation
					                                                      // (5e-7) pushed lambda past the 1e-4 bound of the mode
				#pragma unroll
				for(int u = 0; u < 2; ++u) {
					if(live[u]) {
						const int r = row[u];
						delta_local += fabs(gam[r] - g_new[u]);
						gam[r] = g_new[u];
						eth[r] = e_new[u];
					}
				}
			}
		}
		TRLDA_TICK(3)
		if(final_sweep)
			break;
		delta_local = warp_sum(delta_local);
		if(lane == 0)
			wsum[warp] = delta_local;
		__syncthreads();
		double delta = 0.0;
		for(int q = 0; q < NW; ++q)
			delta += wsum[q];
		++it;
		converged = delta / K < a.threshold;                           // lda.cpp:202
		// no second barrier: wsum and red are next written behind the barriers of the coming sweep's fold
		TRLDA_TICK(4)
	}
	if(tid == 0 && a.iterations)
		a.iterations[d] = it;
	if(tid == 0 && a.sweeps)
		atomicAdd(a.sweeps, (unsigned long long) (it + 1));
	if(timing) {
		for(int i = 0; i < 5; ++i)
			atomicAdd(a.ticks + i, (unsigned long long) tk[i]);
		atomicAdd(a.ticks + 14, (unsigned long long) (it + 1));
		atomicAdd(a.ticks + 15, 1ull);
	}
	#undef TRLDA_TICK
}

template <typename T, int NW, int NVEC, bool BULK>
static void launch_stream_k(const EStepArgs& args, const DeviceDocs& docs, const int32_t* order, int64_t offset,
                            int64_t count, int n_cap, size_t smem, cudaStream_t s) {
	auto kernel = k_estep_stream<T, NW, NVEC, BULK>;
	static size_t configured = 0;      // per instantiation: the attribute is set once (and again only if the tile grows)
	if(smem > configured) {
		cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
		configured = smem;
	}
	kernel<<<(unsigned) count, NW * 32, smem, s>>>(args, docs, order, offset, n_cap);
}

template <typename T, int NW, bool BULK>
static void launch_stream_v(int nvec, const EStepArgs& args, const DeviceDocs& docs, const int32_t* order, int64_t offset,
                            int64_t count, int n_cap, size_t smem, cudaStream_t s) {
	constexpr int MAXV = sizeof(T) == 4 ? 8 : 16;
	switch(nvec) {
		case 1: launch_stream_k<T, NW, 1, BULK>(args, docs, order, offset, count, n_cap, smem, s); break;
		case 2: launch_stream_k<T, NW, 2, BULK>(args, docs, order, offset, count, n_cap, smem, s); break;
		case 4: launch_stream_k<T, NW, 4, BULK>(args, docs, order, offset, count, n_cap, smem, s); break;
		case 8: launch_stream_k<T, NW, 8, BULK>(args, docs, order, offset, count, n_cap, smem, s); break;
		default: launch_stream_k<T, NW, MAXV, BULK>(args, docs, order, offset, count, n_cap, smem, s); break;
	}
}

// one CTA per document, handed out by the hardware scheduler as SMs free up
void launch_estep_stream(const EStepArgs& args, const DeviceDocs& docs, const int32_t* order, int64_t offset,
                         int64_t count, int n_max, int elem_size, cudaStream_t s) {
	if(count == 0)
		return;
	const int K = args.K;
	const int nvec = stream_nvec(K, elem_size);
	const int n_cap = std::max(32, (n_max + 31) / 32 * 32);
	const int kp = nvec * 32 * (16 / elem_size);
	const size_t smem = stream_smem_layout(stream_warps(K, elem_size), kp, n_cap, elem_size).total;
	if(elem_size == 4) {                                  // warps per CTA: stream_warps()
		if(stream_bulk(K, elem_size))
			launch_stream_v<float, 16, true>(nvec, args, docs, order, offset, count, n_cap, smem, s);
		else
			launch_stream_v<float, 8, false>(nvec, args, docs, order, offset, count, n_cap, smem, s);
	} else {
		if(stream_bulk(K, elem_size))
			launch_stream_v<double, 8, true>(nvec, args, docs, order, offset, count, n_cap, smem, s);
		else
			launch_stream_v<double, 8, false>(nvec, args, docs, order, offset, count, n_cap, smem, s);
	}
}

}  // namespace trlda
