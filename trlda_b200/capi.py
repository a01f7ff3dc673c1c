"""
ctypes view of the C ABI in include/trlda_b200.h — the reference-side binding a maintainer would write if the
host language were Python (the reference's own binding is the CPython extension, see trlda_b200/csrc/pymodule.cpp
and INTEGRATION.md).  Used by the parity tests and bench.py, which drive the C ABI directly with host buffers.

There is no fallback: if libtrlda_b200.so is missing this module raises, and every compute call fails with the
library's error message when no B200 is visible.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libtrlda_b200.so')

KIND = {'online': 0, 'batch': 1, 'cumulative': 2}
DISTANCE = {'hellinger': 0, 'kullback_leibler': 1}
PRECISION = {'fp64': 0, 'mixed': 1}
NUM_KERNEL_KINDS = 12

OK, ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED = 0, 1, 2, 3


class Params(C.Structure):
	"""trlda_params == LDA::Parameters (reference code/trlda/include/lda.h:32-78)"""
	_fields_ = [
		('inference_method', C.c_int32),
		('threshold', C.c_double),
		('max_iter_inference', C.c_int32),
		('max_iter_tr', C.c_int32),
		('tau', C.c_double),
		('kappa', C.c_double),
		('rho', C.c_double),
		('adaptive', C.c_int32),
		('num_samples', C.c_int32),
		('burn_in', C.c_int32),
		('init_gamma', C.c_int32),
		('update_lambda', C.c_int32),
		('update_alpha', C.c_int32),
		('update_eta', C.c_int32),
		('min_alpha', C.c_double),
		('min_eta', C.c_double),
		('max_epochs', C.c_int32),
		('max_iter_alpha', C.c_int32),
		('max_iter_eta', C.c_int32),
		('emp_bayes_threshold', C.c_double),
		('verbosity', C.c_int32)]


class Docs(C.Structure):
	"""trlda_docs: CSR view of LDA::Documents"""
	_fields_ = [
		('num_docs', C.c_int64),
		('doc_ptr', C.POINTER(C.c_int64)),
		('word_ids', C.POINTER(C.c_int32)),
		('counts', C.POINTER(C.c_int32))]


class Stats(C.Structure):
	_fields_ = [
		('launches', C.c_int64 * NUM_KERNEL_KINDS),
		('ms', C.c_double * NUM_KERNEL_KINDS),
		('estep_doc_iterations', C.c_int64),
		('estep_docs', C.c_int64),
		('total_launches', C.c_int64),
		('h2d_bytes', C.c_int64),
		('d2h_bytes', C.c_int64),
		('estep_sweeps', C.c_int64),
		('estep_calls', C.c_int64)]


_P = C.POINTER
_dbl = _P(C.c_double)

# every symbol include/trlda_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
	'trlda_params_default': (None, [_P(Params)]),
	'trlda_kernel_kind_name': (C.c_char_p, [C.c_int]),
	'trlda_create': (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, _dbl, C.c_double, C.c_int, C.c_int, _P(C.c_void_p)]),
	'trlda_destroy': (None, [C.c_void_p]),
	'trlda_last_error': (C.c_char_p, [C.c_void_p]),
	'trlda_sample': (C.c_int, [C.c_void_p, C.c_int64, C.c_double, C.c_int, _P(Docs)]),
	'trlda_debug_global_csc': (C.c_int, [C.c_void_p, _P(C.c_int32), _P(C.c_int32), C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int,
		_P(C.c_int32), _P(C.c_int32), _P(C.c_int32)]),
	'trlda_seed': (None, [C.c_uint64]),
	'trlda_kind': (C.c_int, [C.c_void_p]),
	'trlda_precision': (C.c_int, [C.c_void_p]),
	'trlda_set_precision': (C.c_int, [C.c_void_p, C.c_int]),
	'trlda_num_topics': (C.c_int, [C.c_void_p]),
	'trlda_num_words': (C.c_int, [C.c_void_p]),
	'trlda_get_lambda': (C.c_int, [C.c_void_p, _dbl]),
	'trlda_set_lambda': (C.c_int, [C.c_void_p, _dbl, C.c_int, C.c_int]),
	'trlda_get_alpha': (C.c_int, [C.c_void_p, _dbl]),
	'trlda_set_alpha': (C.c_int, [C.c_void_p, _dbl, C.c_int]),
	'trlda_get_eta': (C.c_int, [C.c_void_p, _dbl]),
	'trlda_set_eta': (C.c_int, [C.c_void_p, C.c_double]),
	'trlda_get_num_documents': (C.c_int, [C.c_void_p, _P(C.c_int64)]),
	'trlda_set_num_documents': (C.c_int, [C.c_void_p, C.c_int64]),
	'trlda_get_update_count': (C.c_int, [C.c_void_p, _P(C.c_int64)]),
	'trlda_set_update_count': (C.c_int, [C.c_void_p, C.c_int64]),
	'trlda_update_variables': (C.c_int, [C.c_void_p, _P(Docs), _dbl, C.c_int, C.c_int64, _P(Params), _dbl, _dbl]),
	'trlda_update_parameters': (C.c_int, [C.c_void_p, _P(Docs), _P(Params), _dbl]),
	'trlda_upload_docs': (C.c_int, [C.c_void_p, _P(Docs)]),
	'trlda_upload_docs_slot': (C.c_int, [C.c_void_p, _P(Docs), C.c_int]),
	'trlda_select_docs': (C.c_int, [C.c_void_p, C.c_int]),
	'trlda_update_parameters_resident': (C.c_int, [C.c_void_p, _P(Params), _dbl]),
	'trlda_lower_bound': (C.c_int, [C.c_void_p, _P(Docs), _dbl, C.c_int, C.c_int64, _P(Params), C.c_int64, _dbl, _dbl]),
	'trlda_predictive_log_likelihood': (C.c_int, [C.c_void_p, _P(Docs), _P(Docs), _dbl, C.c_int, C.c_int64, _P(Params), _dbl,
		_P(C.c_int64), _dbl]),
	'trlda_word_topics': (C.c_int, [C.c_void_p, _P(Docs), _dbl, C.c_int, C.c_int64, _P(Params), C.c_int, _P(C.c_int32), _dbl,
		_dbl]),
	'trlda_top_words': (C.c_int, [C.c_void_p, C.c_int, _P(C.c_int32), _dbl]),
	'trlda_cooccurrence': (C.c_int, [C.c_void_p, _P(Docs), _P(C.c_int32), C.c_int, _P(C.c_int64), _P(C.c_int64)]),
	'trlda_topic_distances': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, _dbl]),
	'trlda_index_documents': (C.c_int, [C.c_void_p, _dbl, C.c_int, C.c_int64]),
	'trlda_similar_documents': (C.c_int, [C.c_void_p, _dbl, C.c_int, C.c_int64, C.c_int, _P(C.c_int64), _dbl]),
	'trlda_inject_initial_gamma': (C.c_int, [C.c_void_p, _dbl, C.c_int, C.c_int64]),
	'trlda_inject_initial_lambda': (C.c_int, [C.c_void_p, _dbl, C.c_int, C.c_int]),
	'trlda_comm_unique_id': (C.c_int, [C.c_void_p]),
	'trlda_comm_init': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
	'trlda_comm_size': (C.c_int, [C.c_void_p]),
	'trlda_stream': (C.c_void_p, [C.c_void_p]),
	'trlda_synchronize': (C.c_int, [C.c_void_p]),
	'trlda_set_profiling': (C.c_int, [C.c_void_p, C.c_int]),
	'trlda_get_stats': (C.c_int, [C.c_void_p, _P(Stats)]),
	'trlda_reset_stats': (C.c_int, [C.c_void_p]),
	'trlda_get_row_sums': (C.c_int, [C.c_void_p, _dbl]),
	'trlda_device_special': (C.c_int, [C.c_int, C.c_int, _dbl, C.c_int64, _dbl]),
	'trlda_polygamma': (C.c_double, [C.c_int, C.c_double]),
	'trlda_reader_open': (C.c_int, [C.c_char_p, C.c_int64, C.c_int, _P(C.c_void_p)]),
	'trlda_reader_next': (C.c_int, [C.c_void_p, _P(Docs), _P(C.c_int)]),
	'trlda_reader_close': (None, [C.c_void_p]),
	'trlda_reader_last_error': (C.c_char_p, [C.c_void_p]),
}

_lib = None


def lib():
	"""Loads libtrlda_b200.so (built by trlda_b200/build.py); raises if it is missing — no fallback."""
	global _lib
	if _lib is None:
		if not os.path.exists(LIB_PATH):
			raise RuntimeError(
				'trlda_b200: %s is missing; build it with `python -m trlda_b200.build` '
				'(there is no CPU fallback)' % LIB_PATH)
		handle = C.CDLL(LIB_PATH)
		for name, (restype, argtypes) in PROTOTYPES.items():
			fn = getattr(handle, name)
			fn.restype = restype
			fn.argtypes = argtypes
		_lib = handle
	return _lib


def default_params(**kwargs):
	p = Params()
	lib().trlda_params_default(C.byref(p))
	for key, value in kwargs.items():
		if not hasattr(p, key):
			raise TypeError('unknown parameter ' + key)
		setattr(p, key, value)
	return p


def _dptr(a):
	return a.ctypes.data_as(_dbl) if a is not None else None


def _fortran(a):
	return np.asfortranarray(a, dtype=np.float64)


class CSR(object):
	"""Owns the three arrays of a minibatch (doc_ptr int64, word_ids int32, counts int32)."""

	def __init__(self, doc_ptr, word_ids, counts):
		self.doc_ptr = np.ascontiguousarray(doc_ptr, dtype=np.int64)
		self.word_ids = np.ascontiguousarray(word_ids, dtype=np.int32)
		self.counts = np.ascontiguousarray(counts, dtype=np.int32)
		if self.doc_ptr.ndim != 1 or self.doc_ptr.size < 1:
			raise ValueError('doc_ptr must have B+1 entries')
		if not (self.word_ids.size == self.counts.size == self.doc_ptr[-1]):
			raise ValueError('word_ids / counts do not match doc_ptr')
		self.c = Docs(
			self.doc_ptr.size - 1,
			self.doc_ptr.ctypes.data_as(_P(C.c_int64)),
			self.word_ids.ctypes.data_as(_P(C.c_int32)),
			self.counts.ctypes.data_as(_P(C.c_int32)))

	@property
	def num_docs(self):
		return self.doc_ptr.size - 1

	@property
	def num_pairs(self):
		return int(self.doc_ptr[-1])

	def nbytes(self):
		return self.doc_ptr.nbytes + self.word_ids.nbytes + self.counts.nbytes

	def slice(self, begin, end):
		lo, hi = self.doc_ptr[begin], self.doc_ptr[end]
		return CSR(self.doc_ptr[begin:end + 1] - lo, self.word_ids[lo:hi], self.counts[lo:hi])

	@classmethod
	def from_lists(cls, docs):
		doc_ptr = np.zeros(len(docs) + 1, dtype=np.int64)
		for i, doc in enumerate(docs):
			doc_ptr[i + 1] = doc_ptr[i] + len(doc)
		n = int(doc_ptr[-1])
		word_ids = np.fromiter((w for doc in docs for w, _ in doc), dtype=np.int32, count=n)
		counts = np.fromiter((c for doc in docs for _, c in doc), dtype=np.int32, count=n)
		return cls(doc_ptr, word_ids, counts)


class Model(object):
	"""Thin object wrapper over the opaque trlda_model handle."""

	def __init__(self, kind, num_words, num_topics, num_documents=0, alpha=.1, eta=.3, device=0, precision='fp64'):
		self._lib = lib()
		self.kind, self.V, self.K = kind, int(num_words), int(num_topics)
		a = np.asarray(alpha, dtype=np.float64).ravel()
		if a.size == 1:
			a = np.full(self.K, float(a[0]))
		a = np.ascontiguousarray(a)
		if a.size != self.K:
			raise RuntimeError('Alpha has wrong dimensionality.')
		handle = C.c_void_p()
		status = self._lib.trlda_create(
			KIND[kind], self.V, self.K, int(num_documents), _dptr(a), float(eta), int(device),
			PRECISION[precision], C.byref(handle))
		if status != OK:
			raise RuntimeError(self._lib.trlda_last_error(None).decode())
		self.h = handle

	def close(self):
		if getattr(self, 'h', None):
			self._lib.trlda_destroy(self.h)
			self.h = None

	def __del__(self):
		self.close()

	def _check(self, status):
		if status != OK:
			raise RuntimeError(self._lib.trlda_last_error(self.h).decode())

	# ---- accessors ------------------------------------------------------------------------------------------------
	@property
	def lambdas(self):
		out = np.empty((self.K, self.V), order='F')
		self._check(self._lib.trlda_get_lambda(self.h, _dptr(out)))
		return out

	@lambdas.setter
	def lambdas(self, value):
		value = _fortran(value)
		if value.ndim != 2:
			raise RuntimeError('Lambda has wrong dimensionality.')
		self._check(self._lib.trlda_set_lambda(self.h, _dptr(value), value.shape[0], value.shape[1]))

	@property
	def alpha(self):
		out = np.empty(self.K)
		self._check(self._lib.trlda_get_alpha(self.h, _dptr(out)))
		return out

	@alpha.setter
	def alpha(self, value):
		value = np.ascontiguousarray(np.asarray(value, dtype=np.float64).ravel())
		self._check(self._lib.trlda_set_alpha(self.h, _dptr(value), value.size))

	@property
	def eta(self):
		out = C.c_double()
		self._check(self._lib.trlda_get_eta(self.h, C.byref(out)))
		return out.value

	@eta.setter
	def eta(self, value):
		self._check(self._lib.trlda_set_eta(self.h, float(value)))

	@property
	def num_documents(self):
		out = C.c_int64()
		self._check(self._lib.trlda_get_num_documents(self.h, C.byref(out)))
		return out.value

	@num_documents.setter
	def num_documents(self, value):
		self._check(self._lib.trlda_set_num_documents(self.h, int(value)))

	@property
	def update_count(self):
		out = C.c_int64()
		self._check(self._lib.trlda_get_update_count(self.h, C.byref(out)))
		return out.value

	@update_count.setter
	def update_count(self, value):
		self._check(self._lib.trlda_set_update_count(self.h, int(value)))

	@property
	def precision(self):
		return 'mixed' if self._lib.trlda_precision(self.h) == 1 else 'fp64'

	@precision.setter
	def precision(self, value):
		self._check(self._lib.trlda_set_precision(self.h, PRECISION[value]))

	# ---- hot path -------------------------------------------------------------------------------------------------
	def update_variables(self, docs, latents=None, max_iter=100, threshold=.001, want_sstats=True, inference_method='VI',
	                     num_samples=1, burn_in=2):
		params = default_params(max_iter_inference=max_iter, threshold=threshold, num_samples=num_samples, burn_in=burn_in,
			inference_method=1 if inference_method.upper() == 'GIBBS' else 0)
		gamma = np.empty((self.K, docs.num_docs), order='F')
		sstats = np.empty((self.K, self.V), order='F') if want_sstats else None
		rows, cols = 0, 0
		if latents is not None:
			latents = _fortran(latents)
			rows, cols = latents.shape
		self._check(self._lib.trlda_update_variables(
			self.h, C.byref(docs.c), _dptr(latents), rows, cols, C.byref(params), _dptr(gamma), _dptr(sstats)))
		return gamma, sstats

	def inject(self, gamma0=None, lambda0=None):
		if gamma0 is not None:
			gamma0 = _fortran(gamma0)
			self._check(self._lib.trlda_inject_initial_gamma(self.h, _dptr(gamma0), gamma0.shape[0], gamma0.shape[1]))
		if lambda0 is not None:
			lambda0 = _fortran(lambda0)
			self._check(self._lib.trlda_inject_initial_lambda(self.h, _dptr(lambda0), lambda0.shape[0], lambda0.shape[1]))

	def update_parameters(self, docs, gamma0=None, lambda0=None, **kwargs):
		self.inject(gamma0, lambda0)
		params = default_params(**kwargs)
		result = C.c_double(0.)
		self._check(self._lib.trlda_update_parameters(self.h, C.byref(docs.c), C.byref(params), C.byref(result)))
		return result.value

	def upload_docs(self, docs):
		self._check(self._lib.trlda_upload_docs(self.h, C.byref(docs.c)))

	def upload_docs_slot(self, docs, slot):
		self._check(self._lib.trlda_upload_docs_slot(self.h, C.byref(docs.c), int(slot)))

	def select_docs(self, slot):
		self._check(self._lib.trlda_select_docs(self.h, int(slot)))

	def update_parameters_resident(self, gamma0=None, lambda0=None, **kwargs):
		self.inject(gamma0, lambda0)
		params = default_params(**kwargs)
		result = C.c_double(0.)
		self._check(self._lib.trlda_update_parameters_resident(self.h, C.byref(params), C.byref(result)))
		return result.value

	def lower_bound(self, docs, latents=None, num_documents=-1, max_iter=100, threshold=.001):
		params = default_params(max_iter_inference=max_iter, threshold=threshold)
		rows, cols = 0, 0
		if latents is not None:
			latents = _fortran(latents)
			rows, cols = latents.shape
		total = C.c_double(0.)
		per_doc = np.empty(docs.num_docs)
		self._check(self._lib.trlda_lower_bound(
			self.h, C.byref(docs.c), _dptr(latents), rows, cols, C.byref(params), int(num_documents),
			C.byref(total), _dptr(per_doc)))
		return total.value, per_doc

	def predictive_log_likelihood(self, docs, held_out, latents=None, max_iter=100, threshold=.001):
		"""document-completion predictive log-likelihood: gamma is fitted on `docs`, the pairs of `held_out` are scored;
		returns (total, tokens, per_doc)"""
		params = default_params(max_iter_inference=max_iter, threshold=threshold)
		rows, cols = 0, 0
		if latents is not None:
			latents = _fortran(latents)
			rows, cols = latents.shape
		total, tokens = C.c_double(0.), C.c_int64(0)
		per_doc = np.empty(docs.num_docs)
		self._check(self._lib.trlda_predictive_log_likelihood(
			self.h, C.byref(docs.c), C.byref(held_out.c), _dptr(latents), rows, cols, C.byref(params),
			C.byref(total), C.byref(tokens), _dptr(per_doc)))
		return total.value, tokens.value, per_doc

	def word_topics(self, docs, n=1, latents=None, max_iter=100, threshold=1e-3):
		"""the n most probable topics of every pair of `docs` under the fitted phi: (topics[N, n] int32, probs[N, n],
		gamma[K, B]), row j for the j-th pair, each row ranked by descending phi (equal phi: the smaller topic first)"""
		params = default_params(max_iter_inference=max_iter, threshold=threshold)
		rows, cols = 0, 0
		if latents is not None:
			latents = _fortran(latents)
			rows, cols = latents.shape
		pairs = int(docs.doc_ptr[-1])
		topics = np.empty((pairs, max(int(n), 0)), dtype=np.int32)
		probs = np.empty((pairs, max(int(n), 0)))
		gamma = np.empty((self.K, docs.num_docs), order='F')
		self._check(self._lib.trlda_word_topics(self.h, C.byref(docs.c), _dptr(latents), rows, cols, C.byref(params), int(n),
			topics.ctypes.data_as(_P(C.c_int32)), _dptr(probs), _dptr(gamma)))
		return topics, probs, gamma

	def top_words(self, n=10):
		"""the n most probable words of every topic: (ids[K, n] int32, probs[K, n]), each row in rank order"""
		ids = np.empty((self.K, max(int(n), 0)), dtype=np.int32)
		probs = np.empty((self.K, max(int(n), 0)))
		self._check(self._lib.trlda_top_words(self.h, int(n), ids.ctypes.data_as(_P(C.c_int32)), _dptr(probs)))
		return ids, probs

	def cooccurrence(self, docs, ids):
		"""document frequencies of the words of `ids` (K x n, e.g. top_words' ids): (counts[K, n, n] int64, num_docs) with
		counts[k, i, j] = documents of `docs` that contain both ids[k, i] and ids[k, j]"""
		ids = np.ascontiguousarray(ids, dtype=np.int32)
		if ids.ndim != 2 or ids.shape[0] != self.K:
			raise ValueError('ids must be a K x n array')
		n = ids.shape[1]
		counts = np.empty((self.K, n, n), dtype=np.int64)
		num_docs = C.c_int64(0)
		self._check(self._lib.trlda_cooccurrence(self.h, C.byref(docs.c), ids.ctypes.data_as(_P(C.c_int32)), n,
			counts.ctypes.data_as(_P(C.c_int64)), C.byref(num_docs)))
		return counts, num_docs.value

	def topic_distances(self, other=None, metric='hellinger'):
		"""distances between the topics of this model and those of `other` (None: this model): D[K, K_other] in Fortran
		order, D[i, j] = hellinger or kullback_leibler distance between E[beta] of topic i here and of topic j there"""
		k_other = self.K if other is None else other.K
		out = np.empty((self.K, k_other), order='F')
		self._check(self._lib.trlda_topic_distances(self.h, None if other is None else other.h, DISTANCE[metric], _dptr(out)))
		return out

	def index_documents(self, gamma):
		"""replaces the document index with sqrt(theta) of the columns of gamma (K x D), theta_d = gamma_d / sum_k gamma_dk;
		D = 0 frees it.  The index stays on the device until replaced; it is not pickled"""
		gamma = _fortran(gamma)
		self._check(self._lib.trlda_index_documents(self.h, _dptr(gamma), gamma.shape[0], gamma.shape[1]))

	def similar_documents(self, gamma, n=10):
		"""(ids int64 Q x n, dist float64 Q x n): the n indexed documents nearest to each column of gamma (K x Q) under
		the Hellinger distance of the topic proportions, nearest first, exact ties to the smaller id"""
		gamma = _fortran(gamma)
		q = gamma.shape[1]
		ids = np.empty((q, max(int(n), 0)), dtype=np.int64)
		dist = np.empty((q, max(int(n), 0)))
		self._check(self._lib.trlda_similar_documents(self.h, _dptr(gamma), gamma.shape[0], q, int(n),
			ids.ctypes.data_as(_P(C.c_int64)), _dptr(dist)))
		return ids, dist

	# ---- multi-GPU / instrumentation --------------------------------------------------------------------------------
	def comm_init(self, unique_id, rank, nranks):
		buf = C.create_string_buffer(bytes(unique_id), 128)
		self._check(self._lib.trlda_comm_init(self.h, buf, rank, nranks))

	@property
	def stream(self):
		return self._lib.trlda_stream(self.h)

	def synchronize(self):
		self._check(self._lib.trlda_synchronize(self.h))

	def set_profiling(self, on):
		self._check(self._lib.trlda_set_profiling(self.h, int(bool(on))))

	def reset_stats(self):
		self._check(self._lib.trlda_reset_stats(self.h))

	def stats(self):
		s = Stats()
		self._check(self._lib.trlda_get_stats(self.h, C.byref(s)))
		names = [self._lib.trlda_kernel_kind_name(i).decode() for i in range(NUM_KERNEL_KINDS)]
		return {
			'launches': {n: int(s.launches[i]) for i, n in enumerate(names)},
			'ms': {n: float(s.ms[i]) for i, n in enumerate(names)},
			'estep_doc_iterations': int(s.estep_doc_iterations),
			'estep_docs': int(s.estep_docs),
			'total_launches': int(s.total_launches),
			'h2d_bytes': int(s.h2d_bytes),
			'd2h_bytes': int(s.d2h_bytes),
			'estep_sweeps': int(s.estep_sweeps),
			'estep_calls': int(s.estep_calls)}

	def sample(self, num_documents, length, collapse=False):
		"""LDA::sample on the device; returns a CSR (collapse: unique (word, count) pairs sorted by word id)"""
		view = Docs()
		self._check(self._lib.trlda_sample(self.h, int(num_documents), float(length), int(bool(collapse)), C.byref(view)))
		B = int(view.num_docs)
		ptr = np.ctypeslib.as_array(view.doc_ptr, shape=(B + 1,)).copy()
		N = int(ptr[-1])
		ids = np.ctypeslib.as_array(view.word_ids, shape=(N,)).copy() if N else np.zeros(0, dtype=np.int32)
		cts = np.ctypeslib.as_array(view.counts, shape=(N,)).copy() if N else np.zeros(0, dtype=np.int32)
		return CSR(ptr, ids, cts)

	def debug_global_csc(self, lengths, ids, ranks, v0, v1):
		"""test hook (csrc/csc.cu): word-sorted token list of a gathered minibatch - lengths is ranks x max_docs, ids
		ranks x max_pairs with -1 padding - restricted to the words [v0, v1); returns (word_ptr, tok_doc, tok_src)"""
		lengths = np.ascontiguousarray(lengths, dtype=np.int32).reshape(ranks, -1)
		ids = np.ascontiguousarray(ids, dtype=np.int32).reshape(ranks, -1)
		i32 = lambda x: x.ctypes.data_as(_P(C.c_int32))
		word_ptr = np.empty(self.V + 1, dtype=np.int32)
		tok_doc = np.empty(max(ids.size, 1), dtype=np.int32)
		tok_src = np.empty(max(ids.size, 1), dtype=np.int32)
		self._check(self._lib.trlda_debug_global_csc(self.h, i32(lengths), i32(ids), int(ranks), lengths.shape[1], ids.shape[1],
			int(v0), int(v1), i32(word_ptr), i32(tok_doc), i32(tok_src)))
		return word_ptr, tok_doc[:int(word_ptr[-1])], tok_src[:int(word_ptr[-1])]

	def row_sums(self):
		out = np.empty(self.K)
		self._check(self._lib.trlda_get_row_sums(self.h, _dptr(out)))
		return out


class Reader(object):
	"""Native reader of the reference's text format (`N id:cnt ...` per line): a background thread parses the memory-mapped
	file into pinned CSR minibatches, `prefetch` batches ahead.  Iterating yields CSR objects in the order of the
	reference's load_documents generator (the final remainder is yielded even when empty).  With copy=False the arrays
	are views of the reader's ring buffers, valid until the batch after the next one is requested."""
	END = 4

	def __init__(self, path, batch_size=None, prefetch=2, copy=True):
		self._lib = lib()
		self.h = C.c_void_p()
		self.copy = copy
		status = self._lib.trlda_reader_open(os.fsencode(path), int(batch_size or 0), int(prefetch), C.byref(self.h))
		if status != 0:
			raise IOError(self._lib.trlda_reader_last_error(None).decode())
		self.pinned = None

	def close(self):
		if self.h:
			self._lib.trlda_reader_close(self.h)
			self.h = C.c_void_p()

	def __del__(self):
		self.close()

	def __iter__(self):
		return self

	def __next__(self):
		if not self.h:
			raise StopIteration
		view, pinned = Docs(), C.c_int(0)
		status = self._lib.trlda_reader_next(self.h, C.byref(view), C.byref(pinned))
		if status == self.END:
			self.close()
			raise StopIteration
		if status != 0:
			message = self._lib.trlda_reader_last_error(self.h).decode()
			self.close()
			raise ValueError(message)
		self.pinned = bool(pinned.value)
		B = int(view.num_docs)
		ptr = np.ctypeslib.as_array(view.doc_ptr, shape=(B + 1,))
		N = int(ptr[-1])
		ids = np.ctypeslib.as_array(view.word_ids, shape=(N,)) if N else np.zeros(0, dtype=np.int32)
		cts = np.ctypeslib.as_array(view.counts, shape=(N,)) if N else np.zeros(0, dtype=np.int32)
		if self.copy:
			ptr, ids, cts = ptr.copy(), ids.copy(), cts.copy()
		return CSR(ptr, ids, cts)


def comm_unique_id():
	buf = C.create_string_buffer(128)
	status = lib().trlda_comm_unique_id(buf)
	if status != OK:
		raise RuntimeError(lib().trlda_last_error(None).decode())
	return buf.raw


def seed(value):
	lib().trlda_seed(int(value))


def device_special(which, x, device=0):
	x = np.ascontiguousarray(x, dtype=np.float64).ravel()
	out = np.empty_like(x)
	status = lib().trlda_device_special(device, which, _dptr(x), x.size, _dptr(out))
	if status != OK:
		raise RuntimeError(lib().trlda_last_error(None).decode())
	return out


def polygamma(n, x):
	return lib().trlda_polygamma(int(n), float(x))
