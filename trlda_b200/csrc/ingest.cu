// ingest.cu — native reader for the reference's text format (python/utils/load_documents.py:6-69): one document per
// line, `N id:cnt id:cnt ...`, the first field ignored (load_documents.py:43).  The file is memory-mapped and parsed
// by a background thread into CSR minibatches in PINNED host memory, a few batches ahead of the consumer, so that the
// Python line parsing — the dominant end-to-end cost once a device step takes tens of milliseconds (1.2 M
// `int(...)` calls per cfg-3 minibatch) — leaves the training loop and the H2D copy of a batch can start from
// page-locked memory the moment the batch is asked for.  Batching follows the reference's generator with a fixed
// batch size: full batches in order, then the remainder — which is yielded even when it is empty.
#include "../../include/trlda_b200.h"

#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>

namespace {

thread_local std::string g_reader_error;

// one batch in host memory: page-locked where a CUDA device exists, plain otherwise (CPU-only tooling, tests); freed by
// its owner and move-only, so that two owners of one allocation cannot exist
struct HostArray {
	void* p = nullptr;
	size_t cap = 0;
	bool pinned = false;

	HostArray() = default;
	HostArray(const HostArray&) = delete;
	HostArray& operator=(const HostArray&) = delete;
	HostArray(HostArray&& o) noexcept { *this = std::move(o); }
	HostArray& operator=(HostArray&& o) noexcept {
		if(this != &o) {
			release();
			p = std::exchange(o.p, nullptr);
			cap = std::exchange(o.cap, 0);
			pinned = o.pinned;
		}
		return *this;
	}
	~HostArray() { release(); }

	bool ensure(size_t bytes, bool want_pinned) {
		if(bytes <= cap)
			return true;
		release();
		const size_t want = bytes + bytes / 2 + 4096;
		if(want_pinned && cudaHostAlloc(&p, want, cudaHostAllocDefault) == cudaSuccess) {
			pinned = true;
		} else {
			cudaGetLastError();
			p = malloc(want);
			pinned = false;
		}
		cap = p ? want : 0;
		return p != nullptr;
	}
	void release() {
		if(p) {
			if(pinned)
				cudaFreeHost(p);
			else
				free(p);
		}
		p = nullptr;
		cap = 0;
	}
};

struct Batch {
	HostArray ptr, ids, cts;
	int64_t B = 0, N = 0;
	bool last = false;
};

}  // namespace

struct trlda_reader {
	int fd = -1;
	const char* data = nullptr;
	size_t size = 0;
	int64_t batch_size = 0;
	bool pinned = false;
	std::vector<Batch> ring;
	// ring[produced % n] is filled by the worker once consumed + n - 1 > produced (the consumer still owns the batch
	// it was handed last)
	size_t produced = 0, consumed = 0;
	bool finished = false, stop = false;
	std::string error;
	std::mutex mu;
	std::condition_variable cv;
	std::thread worker;
};

namespace {

// parses the documents [pos, ...) into `b` until `limit` documents (0 = no limit) or the end of the file
bool parse_batch(trlda_reader* r, size_t& pos, Batch& b, std::string& error) {
	const char* p = r->data + pos;
	const char* end = r->data + r->size;
	// first pass: count lines and fields to size the arrays
	int64_t docs = 0, pairs = 0;
	{
		const char* q = p;
		while(q < end && (r->batch_size <= 0 || docs < r->batch_size)) {
			const char* nl = static_cast<const char*>(memchr(q, '\n', end - q));
			const char* stop = nl ? nl : end;
			for(const char* c = q; c < stop; ++c)
				pairs += *c == ':';
			++docs;
			q = nl ? nl + 1 : end;
		}
	}
	if(!b.ptr.ensure(sizeof(int64_t) * (docs + 1), r->pinned) || !b.ids.ensure(sizeof(int32_t) * (pairs + 1), r->pinned) ||
	   !b.cts.ensure(sizeof(int32_t) * (pairs + 1), r->pinned)) {
		error = "Out of host memory.";
		return false;
	}
	int64_t* ptr = static_cast<int64_t*>(b.ptr.p);
	int32_t* ids = static_cast<int32_t*>(b.ids.p);
	int32_t* cts = static_cast<int32_t*>(b.cts.p);
	int64_t d = 0, n = 0;
	ptr[0] = 0;
	while(p < end && d < docs) {
		// skip the first field (the number of distinct words; load_documents.py:43 ignores it)
		while(p < end && (*p == ' ' || *p == '\t' || *p == '\r'))
			++p;
		while(p < end && *p != ' ' && *p != '\t' && *p != '\r' && *p != '\n')
			++p;
		while(p < end && *p != '\n') {
			while(p < end && (*p == ' ' || *p == '\t' || *p == '\r'))
				++p;
			if(p >= end || *p == '\n')
				break;
			int64_t value[2] = {0, 0};
			for(int f = 0; f < 2; ++f) {
				bool neg = false, any = false;
				if(p < end && (*p == '-' || *p == '+')) {
					neg = *p == '-';
					++p;
				}
				while(p < end && *p >= '0' && *p <= '9') {
					value[f] = value[f] * 10 + (*p - '0');
					any = true;
					if(value[f] > INT32_MAX) {
						error = "Word IDs and counts must fit 32-bit integers.";
						return false;
					}
					++p;
				}
				if(!any || (f == 0 && (p >= end || *p != ':'))) {
					error = "Malformed document line (expected `N id:count id:count ...`).";
					return false;
				}
				if(neg)
					value[f] = -value[f];
				if(f == 0)
					++p;       // the colon
			}
			if(p < end && *p != ' ' && *p != '\t' && *p != '\r' && *p != '\n') {
				error = "Malformed document line (expected `N id:count id:count ...`).";
				return false;
			}
			ids[n] = (int32_t) value[0];
			cts[n] = (int32_t) value[1];
			++n;
		}
		if(p < end)
			++p;           // the newline
		ptr[++d] = n;
	}
	b.B = d;
	b.N = n;
	pos = p - r->data;
	b.last = pos >= r->size && (r->batch_size <= 0 || d < r->batch_size);
	return true;
}

void worker_main(trlda_reader* r) {
	size_t pos = 0;
	bool last_emitted = false;
	while(true) {
		std::unique_lock<std::mutex> lock(r->mu);
		r->cv.wait(lock, [&] { return r->stop || r->produced + 1 < r->consumed + r->ring.size(); });
		if(r->stop)
			return;
		Batch& b = r->ring[r->produced % r->ring.size()];
		lock.unlock();
		std::string error;
		bool ok = true;
		if(pos >= r->size) {
			// the reference's generator always ends with the remainder, even if it is empty (load_documents.py:63)
			ok = b.ptr.ensure(sizeof(int64_t), r->pinned);
			if(ok)
				static_cast<int64_t*>(b.ptr.p)[0] = 0;
			b.B = b.N = 0;
			b.last = true;
		} else {
			ok = parse_batch(r, pos, b, error);
		}
		last_emitted = b.last;
		lock.lock();
		if(!ok) {
			r->error = error.empty() ? "Out of host memory." : error;
			r->finished = true;
			r->cv.notify_all();
			return;
		}
		++r->produced;
		if(last_emitted)
			r->finished = true;
		r->cv.notify_all();
		if(last_emitted)
			return;
	}
}

}  // namespace

extern "C" {

const char* trlda_reader_last_error(const trlda_reader* r) { return r ? r->error.c_str() : g_reader_error.c_str(); }

int trlda_reader_open(const char* path, int64_t batch_size, int prefetch, trlda_reader** out) {
	if(!path || !out || batch_size < 0) {
		g_reader_error = "reader: path and a non-negative batch size are required.";
		return TRLDA_ERR_ARG;
	}
	trlda_reader* r = new trlda_reader;
	r->fd = open(path, O_RDONLY);
	struct stat st;
	if(r->fd < 0 || fstat(r->fd, &st) != 0) {
		g_reader_error = std::string("Cannot open ") + path + ".";
		if(r->fd >= 0)
			close(r->fd);
		delete r;
		return TRLDA_ERR_ARG;
	}
	r->size = (size_t) st.st_size;
	if(r->size) {
		void* map = mmap(nullptr, r->size, PROT_READ, MAP_PRIVATE, r->fd, 0);
		if(map == MAP_FAILED) {
			g_reader_error = std::string("Cannot map ") + path + ".";
			close(r->fd);
			delete r;
			return TRLDA_ERR_ARG;
		}
		madvise(map, r->size, MADV_SEQUENTIAL);
		r->data = static_cast<const char*>(map);
	}
	r->batch_size = batch_size;
	int devices = 0;
	r->pinned = cudaGetDeviceCount(&devices) == cudaSuccess && devices > 0;
	cudaGetLastError();
	r->ring.resize((size_t) std::max(prefetch, 1) + 2);
	r->worker = std::thread(worker_main, r);
	*out = r;
	return TRLDA_OK;
}

int trlda_reader_next(trlda_reader* r, trlda_docs* out, int* pinned) {
	if(!r || !out)
		return TRLDA_ERR_ARG;
	std::unique_lock<std::mutex> lock(r->mu);
	r->cv.wait(lock, [&] { return r->consumed < r->produced || r->finished; });
	if(r->consumed >= r->produced) {
		if(!r->error.empty())
			return TRLDA_ERR_ARG;
		return TRLDA_END;
	}
	Batch& b = r->ring[r->consumed % r->ring.size()];
	++r->consumed;
	out->num_docs = b.B;
	out->doc_ptr = static_cast<const int64_t*>(b.ptr.p);
	out->word_ids = static_cast<const int32_t*>(b.ids.p);
	out->counts = static_cast<const int32_t*>(b.cts.p);
	if(pinned)
		*pinned = b.ids.pinned ? 1 : 0;
	r->cv.notify_all();
	return TRLDA_OK;
}

void trlda_reader_close(trlda_reader* r) {
	if(!r)
		return;
	{
		std::lock_guard<std::mutex> lock(r->mu);
		r->stop = true;
	}
	r->cv.notify_all();
	if(r->worker.joinable())
		r->worker.join();
	if(r->data)
		munmap(const_cast<char*>(r->data), r->size);
	if(r->fd >= 0)
		close(r->fd);
	delete r;
}

}  // extern "C"
