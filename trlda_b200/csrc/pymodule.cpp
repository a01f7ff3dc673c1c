// pymodule.cpp — CPython 3 extension `_trlda`: the reference's Python-facing classes hosted on the C ABI.
//
// This file is the re-hosted counterpart of the reference binding (code/trlda/python/src/*.cpp, CPython 2 only):
// the same type hierarchy Distribution -> LDA -> {OnlineLDA, BatchLDA, CumulativeLDA} (module.cpp:24-330), the same
// constructor / method keyword lists and defaults, the same attribute names and array conventions (K x V and
// K x B float64, Fortran order; `lambdas` returned as a read-only copy, ldainterface.cpp:53-60; `alpha` returned
// as a K x 1 array), the same error convention (library errors -> RuntimeError, malformed documents -> TypeError)
// and the same pickle tuples (onlineldainterface.cpp:265-313).  Where the reference calls `self->lda->method()`
// on a `TRLDA::LDA*`, this binding calls the `trlda_*` entry point of include/trlda_b200.h that replaces it.
// No numerical work happens here; the only loop is the packing of the document list into CSR.
//
// Additions (all optional, defaults keep the reference behaviour):
//   constructor kwargs `device=0`, `precision='fp64'|'mixed'` (default from $TRLDA_PRECISION, else 'fp64');
//   `docs` may also be a (doc_ptr, word_ids, counts) triple of numpy arrays (CSR), skipping the list walk;
//   private kwargs `_initial_gamma` / `_initial_lambda` on update_parameters and `_latents` on lower_bound: the
//   parity seams for the values the reference draws internally from rand() (lda.cpp:135, cumulativelda.cpp:60);
//   the GIL is released while the device works.
#define PY_SSIZE_T_CLEAN
#include <Python.h>
#define NPY_NO_DEPRECATED_API NPY_1_7_API_VERSION
#include <numpy/arrayobject.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "trlda_b200.h"

namespace {

struct LDAObject {
	PyObject_HEAD
	trlda_model* m;
};

// ---- documents ---------------------------------------------------------------------------------------------------------
struct Documents {
	std::vector<int64_t> doc_ptr;
	std::vector<int32_t> word_ids, counts;
	PyObject* keep[3] = {nullptr, nullptr, nullptr};   // borrowed numpy arrays of the CSR fast path
	trlda_docs view{};
	~Documents() {
		for(PyObject* o : keep)
			Py_XDECREF(o);
	}
};

// list[list[(int, int)]] -> CSR; replaces PyList_ToDocuments (ldainterface.cpp:152-190) with a tight loop
int docs_converter(PyObject* obj, void* out_) {
	Documents& out = *static_cast<Documents*>(out_);
	if(PyTuple_Check(obj) && PyTuple_GET_SIZE(obj) == 3 && PyArray_Check(PyTuple_GET_ITEM(obj, 0))) {
		// CSR fast path
		PyObject* ptr = PyArray_FROM_OTF(PyTuple_GET_ITEM(obj, 0), NPY_INT64, NPY_ARRAY_IN_ARRAY);
		PyObject* ids = ptr ? PyArray_FROM_OTF(PyTuple_GET_ITEM(obj, 1), NPY_INT32, NPY_ARRAY_IN_ARRAY) : nullptr;
		PyObject* cts = ids ? PyArray_FROM_OTF(PyTuple_GET_ITEM(obj, 2), NPY_INT32, NPY_ARRAY_IN_ARRAY) : nullptr;
		out.keep[0] = ptr; out.keep[1] = ids; out.keep[2] = cts;
		if(!cts)
			return 0;
		const npy_intp np1 = PyArray_SIZE((PyArrayObject*) ptr), nn = PyArray_SIZE((PyArrayObject*) ids);
		const int64_t* p = static_cast<const int64_t*>(PyArray_DATA((PyArrayObject*) ptr));
		if(np1 < 1 || PyArray_SIZE((PyArrayObject*) cts) != nn || p[0] != 0 || p[np1 - 1] != nn) {
			PyErr_SetString(PyExc_TypeError, "CSR documents must be (doc_ptr[B+1], word_ids[N], counts[N]) with doc_ptr[0] == 0 and doc_ptr[B] == N.");
			return 0;
		}
		out.view.num_docs = np1 - 1;
		out.view.doc_ptr = p;
		out.view.word_ids = static_cast<const int32_t*>(PyArray_DATA((PyArrayObject*) ids));
		out.view.counts = static_cast<const int32_t*>(PyArray_DATA((PyArrayObject*) cts));
		return 1;
	}
	if(!PyList_Check(obj)) {
		PyErr_SetString(PyExc_TypeError, "Documents must be stored in a list.");              // ldainterface.cpp:156
		return 0;
	}
	const Py_ssize_t B = PyList_GET_SIZE(obj);
	out.doc_ptr.resize(B + 1);
	out.doc_ptr[0] = 0;
	size_t total = 0;
	for(Py_ssize_t d = 0; d < B; ++d) {
		PyObject* doc = PyList_GET_ITEM(obj, d);
		if(!PyList_Check(doc)) {
			PyErr_SetString(PyExc_TypeError, "Each document must be a list of tuples.");      // ldainterface.cpp:170
			return 0;
		}
		total += PyList_GET_SIZE(doc);
		out.doc_ptr[d + 1] = (int64_t) total;
	}
	out.word_ids.resize(total);
	out.counts.resize(total);
#if PY_VERSION_HEX >= 0x030C0000
	// Fast path for the common case - exact tuples of two small exact ints: a few threads walk disjoint document ranges.
	// They only READ object memory (list / tuple item slots, the int's inline digit), no reference counts, no API that
	// touches interpreter state; the calling thread holds the GIL throughout, so nothing can mutate the lists.  Anything
	// unusual (another sequence type, an int subclass, a big int, a value beyond int32) makes the whole batch take the
	// general loop below, which also produces the reference's error messages.
	if(total >= 65536) {
		const int T = (int) std::max(1u, std::min(4u, std::thread::hardware_concurrency() / 2));
		std::vector<char> unusual((size_t) T, 0);
		auto walk = [&](int th) {
			const Py_ssize_t d0 = B * th / T, d1 = B * (th + 1) / T;
			for(Py_ssize_t d = d0; d < d1; ++d) {
				PyObject* doc = PyList_GET_ITEM(obj, d);
				const Py_ssize_t n = (Py_ssize_t) (out.doc_ptr[d + 1] - out.doc_ptr[d]);
				int32_t* ids = out.word_ids.data() + out.doc_ptr[d];
				int32_t* cts = out.counts.data() + out.doc_ptr[d];
				for(Py_ssize_t j = 0; j < n; ++j) {
					PyObject* pair = PyList_GET_ITEM(doc, j);
					if(!PyTuple_CheckExact(pair) || PyTuple_GET_SIZE(pair) != 2) {
						unusual[th] = 1;
						return;
					}
					PyObject* a = PyTuple_GET_ITEM(pair, 0);
					PyObject* b = PyTuple_GET_ITEM(pair, 1);
					if(!PyLong_CheckExact(a) || !PyLong_CheckExact(b) || !PyUnstable_Long_IsCompact(reinterpret_cast<PyLongObject*>(a)) ||
					   !PyUnstable_Long_IsCompact(reinterpret_cast<PyLongObject*>(b))) {
						unusual[th] = 1;
						return;
					}
					const Py_ssize_t w = PyUnstable_Long_CompactValue(reinterpret_cast<PyLongObject*>(a));
					const Py_ssize_t c = PyUnstable_Long_CompactValue(reinterpret_cast<PyLongObject*>(b));
					if(w < INT32_MIN || w > INT32_MAX || c < INT32_MIN || c > INT32_MAX) {
						unusual[th] = 1;
						return;
					}
					ids[j] = (int32_t) w;
					cts[j] = (int32_t) c;
				}
			}
		};
		std::vector<std::thread> pool;
		int started = 1;
		try {
			for(int th = 1; th < T; ++th, ++started)
				pool.emplace_back(walk, th);
		} catch(const std::system_error&) {
			// no more threads to be had: the calling thread walks the ranges that got none
		}
		walk(0);
		for(int th = started; th < T; ++th)
			walk(th);
		for(auto& th : pool)
			th.join();
		bool clean = true;
		for(char u : unusual)
			clean = clean && !u;
		if(clean) {
			out.view.num_docs = B;
			out.view.doc_ptr = out.doc_ptr.data();
			out.view.word_ids = out.word_ids.data();
			out.view.counts = out.counts.data();
			return 1;
		}
	}
#endif
	// The loop chases two pointers per pair (list -> tuple -> int object), every one a likely cache miss at 1.2 M pairs
	// per minibatch: the tuple eight pairs ahead and the word-id object four pairs ahead are prefetched.
	auto as_long = [](PyObject* o) -> long {
#if PY_VERSION_HEX >= 0x030C0000
		if(PyLong_CheckExact(o) && PyUnstable_Long_IsCompact(reinterpret_cast<PyLongObject*>(o)))
			return (long) PyUnstable_Long_CompactValue(reinterpret_cast<PyLongObject*>(o));
#endif
		return PyLong_AsLong(o);
	};
	size_t t = 0;
	for(Py_ssize_t d = 0; d < B; ++d) {
		PyObject* doc = PyList_GET_ITEM(obj, d);
		const Py_ssize_t n = PyList_GET_SIZE(doc);
		for(Py_ssize_t j = 0; j < n; ++j, ++t) {
			if(j + 8 < n)
				__builtin_prefetch(PyList_GET_ITEM(doc, j + 8));
			if(j + 4 < n) {
				PyObject* ahead = PyList_GET_ITEM(doc, j + 4);
				if(PyTuple_Check(ahead) && PyTuple_GET_SIZE(ahead) == 2)
					__builtin_prefetch(PyTuple_GET_ITEM(ahead, 0));
			}
			PyObject* pair = PyList_GET_ITEM(doc, j);
			long w, c;
			if(PyTuple_Check(pair) && PyTuple_GET_SIZE(pair) == 2) {
				w = as_long(PyTuple_GET_ITEM(pair, 0));
				c = as_long(PyTuple_GET_ITEM(pair, 1));
				if((w == -1 || c == -1) && PyErr_Occurred())
					return 0;
			} else if(!PyArg_ParseTuple(pair, "ll", &w, &c)) {                                // ldainterface.cpp:178
				return 0;
			}
			if(w < INT32_MIN || w > INT32_MAX || c < INT32_MIN || c > INT32_MAX) {
				PyErr_SetString(PyExc_OverflowError, "Word IDs and counts must fit 32-bit integers.");
				return 0;
			}
			out.word_ids[t] = (int32_t) w;
			out.counts[t] = (int32_t) c;
		}
	}
	out.view.num_docs = B;
	out.view.doc_ptr = out.doc_ptr.data();
	out.view.word_ids = out.word_ids.data();
	out.view.counts = out.counts.data();
	return 1;
}

// ---- helpers -------------------------------------------------------------------------------------------------------------
PyObject* raise_status(trlda_model* m, int status) {
	PyErr_SetString(PyExc_RuntimeError, trlda_last_error(m));     // Exception -> RuntimeError, e.g. ldainterface.cpp:74-78
	(void) status;
	return nullptr;
}

// new float64 array in Fortran order, like PyArray_FromMatrixXd (pyutils.cpp:15-35)
PyObject* new_farray(npy_intp rows, npy_intp cols) {
	npy_intp dims[2] = {rows, cols};
	return PyArray_New(&PyArray_Type, 2, dims, NPY_DOUBLE, nullptr, nullptr, 0, NPY_ARRAY_F_CONTIGUOUS, nullptr);
}

// any array-like -> aligned float64 Fortran-order array (new reference) with its shape as (rows, cols)
PyObject* as_farray(PyObject* obj, npy_intp* rows, npy_intp* cols, const char* what) {
	PyObject* arr = PyArray_FROM_OTF(obj, NPY_DOUBLE, NPY_ARRAY_IN_FARRAY);
	if(!arr) {
		PyErr_Format(PyExc_TypeError, "%s should be of type `ndarray`.", what);               // ldainterface.cpp:67
		return nullptr;
	}
	PyArrayObject* a = (PyArrayObject*) arr;
	if(PyArray_NDIM(a) == 2) {
		*rows = PyArray_DIM(a, 0);
		*cols = PyArray_DIM(a, 1);
	} else if(PyArray_NDIM(a) == 1) {
		*rows = PyArray_DIM(a, 0);
		*cols = 1;
	} else if(PyArray_NDIM(a) == 0) {
		*rows = *cols = 1;
	} else {
		Py_DECREF(arr);
		PyErr_Format(PyExc_TypeError, "%s can have at most two dimensions.", what);
		return nullptr;
	}
	return arr;
}

int parse_inference_method(const char* s, int32_t* out) {
	if(!s)
		return 1;
	switch(s[0]) {
		case 'g': case 'G': *out = TRLDA_INFERENCE_GIBBS; return 1;
		case 'v': case 'V': *out = TRLDA_INFERENCE_VI; return 1;
		default:
			PyErr_SetString(PyExc_TypeError, "`inference_method` should be either 'GIBBS' or 'VI'.");   // ldainterface.cpp:351
			return 0;
	}
}

int default_precision() {
	const char* e = getenv("TRLDA_PRECISION");
	return e && (e[0] == 'm' || e[0] == 'M') ? TRLDA_PRECISION_MIXED : TRLDA_PRECISION_FP64;
}

int parse_precision(const char* s, int* out) {
	if(!s) {
		*out = default_precision();
		return 1;
	}
	if(!strcmp(s, "fp64") || !strcmp(s, "float64")) { *out = TRLDA_PRECISION_FP64; return 1; }
	if(!strcmp(s, "mixed") || !strcmp(s, "fp32")) { *out = TRLDA_PRECISION_MIXED; return 1; }
	PyErr_SetString(PyExc_TypeError, "`precision` should be either 'fp64' or 'mixed'.");
	return 0;
}

// alpha argument of the constructors / setter: float, int or array-like (onlineldainterface.cpp:61-83)
int alpha_vector(PyObject* alpha, int num_topics, std::vector<double>& out, bool* scalar) {
	*scalar = false;
	if(!alpha) {
		out.assign(num_topics, .1);
		*scalar = true;
		return 1;
	}
	if(PyFloat_Check(alpha) || PyLong_Check(alpha)) {
		const double v = PyFloat_AsDouble(alpha);
		if(v == -1. && PyErr_Occurred())
			return 0;
		out.assign(num_topics > 0 ? num_topics : 1, v);
		*scalar = true;
		return 1;
	}
	npy_intp rows, cols;
	PyObject* arr = as_farray(alpha, &rows, &cols, "Alpha");
	if(!arr)
		return 0;
	if(rows == 1)
		std::swap(rows, cols);
	if(cols != 1) {
		Py_DECREF(arr);
		PyErr_SetString(PyExc_TypeError, "Alpha should be one-dimensional.");                 // onlineldainterface.cpp:78
		return 0;
	}
	const double* data = static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr));
	out.assign(data, data + rows);
	Py_DECREF(arr);
	return 1;
}

int create_model(LDAObject* self, int kind, int num_words, int num_topics, long num_documents, PyObject* alpha,
                 double eta, int device, const char* precision) {
	int prec;
	if(!parse_precision(precision, &prec))
		return -1;
	std::vector<double> a;
	bool scalar;
	if(!alpha_vector(alpha, num_topics, a, &scalar))
		return -1;
	if(!scalar && (int) a.size() != num_topics) {
		PyErr_SetString(PyExc_RuntimeError, "Alpha has wrong dimensionality.");
		return -1;
	}
	if(self->m) {
		trlda_destroy(self->m);
		self->m = nullptr;
	}
	int status;
	Py_BEGIN_ALLOW_THREADS
	status = trlda_create(kind, num_words, num_topics, num_documents, a.data(), eta, device, prec, &self->m);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		PyErr_SetString(PyExc_RuntimeError, trlda_last_error(nullptr));
		return -1;
	}
	return 0;
}

// ---- Distribution / LDA base types ---------------------------------------------------------------------------------------
PyObject* Distribution_new(PyTypeObject* type, PyObject*, PyObject*) {
	LDAObject* self = (LDAObject*) type->tp_alloc(type, 0);
	if(self)
		self->m = nullptr;
	return (PyObject*) self;
}

void Distribution_dealloc(LDAObject* self) {                              // distributioninterface.cpp:30-37
	if(self->m)
		trlda_destroy(self->m);
	Py_TYPE(self)->tp_free((PyObject*) self);
}

int abstract_init(PyObject*, PyObject*, PyObject*) {
	PyErr_SetString(PyExc_NotImplementedError, "This is an abstract class.");   // ldainterface.cpp:35-38
	return -1;
}

#define REQUIRE_MODEL(self, ret)                                                        \
	if(!(self)->m) {                                                                    \
		PyErr_SetString(PyExc_RuntimeError, "The model has not been initialised.");     \
		return ret;                                                                     \
	}

PyObject* LDA_num_topics(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	return PyLong_FromLong(trlda_num_topics(self->m));
}

PyObject* LDA_num_words(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	return PyLong_FromLong(trlda_num_words(self->m));
}

PyObject* LDA_lambda(LDAObject* self, void*) {                            // ldainterface.cpp:53-60
	REQUIRE_MODEL(self, nullptr);
	PyObject* arr = new_farray(trlda_num_topics(self->m), trlda_num_words(self->m));
	if(!arr)
		return nullptr;
	int status;
	double* data = static_cast<double*>(PyArray_DATA((PyArrayObject*) arr));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_get_lambda(self->m, data);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		Py_DECREF(arr);
		return raise_status(self->m, status);
	}
	PyArray_CLEARFLAGS((PyArrayObject*) arr, NPY_ARRAY_WRITEABLE);      // "make array immutable"
	return arr;
}

int LDA_set_lambda(LDAObject* self, PyObject* value, void*) {           // ldainterface.cpp:64-87
	REQUIRE_MODEL(self, -1);
	if(!value) {
		PyErr_SetString(PyExc_TypeError, "Cannot delete lambdas.");
		return -1;
	}
	npy_intp rows, cols;
	PyObject* arr = as_farray(value, &rows, &cols, "Lambda");
	if(!arr)
		return -1;
	int status;
	const double* data = static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_set_lambda(self->m, data, (int) rows, (int) cols);
	Py_END_ALLOW_THREADS
	Py_DECREF(arr);
	if(status != TRLDA_OK) {
		raise_status(self->m, status);
		return -1;
	}
	return 0;
}

PyObject* LDA_alpha(LDAObject* self, void*) {                            // ldainterface.cpp:91-93: K x 1 array
	REQUIRE_MODEL(self, nullptr);
	PyObject* arr = new_farray(trlda_num_topics(self->m), 1);
	if(!arr)
		return nullptr;
	trlda_get_alpha(self->m, static_cast<double*>(PyArray_DATA((PyArrayObject*) arr)));
	return arr;
}

int LDA_set_alpha(LDAObject* self, PyObject* value, void*) {            // ldainterface.cpp:97-131
	REQUIRE_MODEL(self, -1);
	if(!value) {
		PyErr_SetString(PyExc_TypeError, "Cannot delete alpha.");
		return -1;
	}
	std::vector<double> a;
	bool scalar;
	if(!alpha_vector(value, 1, a, &scalar))
		return -1;
	const int status = trlda_set_alpha(self->m, a.data(), scalar ? 1 : (int) a.size());
	if(status != TRLDA_OK) {
		raise_status(self->m, status);
		return -1;
	}
	return 0;
}

PyObject* LDA_eta(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	double eta;
	trlda_get_eta(self->m, &eta);
	return PyFloat_FromDouble(eta);
}

int LDA_set_eta(LDAObject* self, PyObject* value, void*) {              // ldainterface.cpp:141-148
	REQUIRE_MODEL(self, -1);
	const double eta = value ? PyFloat_AsDouble(value) : -1.;
	if(PyErr_Occurred())
		return -1;
	const int status = trlda_set_eta(self->m, eta);
	if(status != TRLDA_OK) {
		raise_status(self->m, status);
		return -1;
	}
	return 0;
}

PyObject* LDA_precision(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	return PyUnicode_FromString(trlda_precision(self->m) == TRLDA_PRECISION_MIXED ? "mixed" : "fp64");
}

int LDA_set_precision(LDAObject* self, PyObject* value, void*) {
	REQUIRE_MODEL(self, -1);
	const char* s = value ? PyUnicode_AsUTF8(value) : nullptr;
	int prec;
	if(!s || !parse_precision(s, &prec))
		return -1;
	trlda_set_precision(self->m, prec);
	return 0;
}

// sample(num_documents, length): LDA::sample (lda.cpp:88-115) on the device (trlda_sample); returns the reference's
// list of lists of (word_id, 1) — or, with collapse=True, unique (word_id, count) pairs sorted by id
PyObject* LDA_sample(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"num_documents", "length", "collapse", nullptr};
	int num_documents;
	double length;
	int collapse = 0;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "id|p", const_cast<char**>(kwlist), &num_documents, &length, &collapse))
		return nullptr;
	trlda_docs view;
	int status;
	Py_BEGIN_ALLOW_THREADS
	status = trlda_sample(self->m, num_documents, length, collapse, &view);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		PyErr_SetString(PyExc_RuntimeError, trlda_last_error(self->m));
		return nullptr;
	}
	PyObject* docs = PyList_New(view.num_docs);
	if(!docs)
		return nullptr;
	for(int64_t d = 0; d < view.num_docs; ++d) {
		const int64_t begin = view.doc_ptr[d], end = view.doc_ptr[d + 1];
		PyObject* doc = PyList_New(end - begin);
		if(!doc) {
			Py_DECREF(docs);
			return nullptr;
		}
		for(int64_t j = begin; j < end; ++j)
			PyList_SET_ITEM(doc, j - begin, Py_BuildValue("(ii)", (int) view.word_ids[j], (int) view.counts[j]));
		PyList_SET_ITEM(docs, d, doc);
	}
	return docs;
}

// update_variables / do_e_step (ldainterface.cpp:311-390)
PyObject* LDA_update_variables(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "latents", "inference_method", "max_iter", "threshold", "num_samples", "burn_in", nullptr};
	Documents documents;
	trlda_params params;
	trlda_params_default(&params);
	PyObject* latents = nullptr;
	const char* inference_method = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|Osidii", const_cast<char**>(kwlist), &docs_converter, &documents,
			&latents, &inference_method, &params.max_iter_inference, &params.threshold, &params.num_samples, &params.burn_in))
		return nullptr;
	if(!parse_inference_method(inference_method, &params.inference_method))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* latents_arr = nullptr;
	if(latents && latents != Py_None) {
		latents_arr = as_farray(latents, &rows, &cols, "`latents`");
		if(!latents_arr)
			return nullptr;
	}
	const int K = trlda_num_topics(self->m), V = trlda_num_words(self->m);
	PyObject* gamma = new_farray(K, documents.view.num_docs);
	PyObject* sstats = gamma ? new_farray(K, V) : nullptr;
	if(!sstats) {
		Py_XDECREF(gamma);
		Py_XDECREF(latents_arr);
		return nullptr;
	}
	int status;
	const double* l = latents_arr ? static_cast<const double*>(PyArray_DATA((PyArrayObject*) latents_arr)) : nullptr;
	double* g = static_cast<double*>(PyArray_DATA((PyArrayObject*) gamma));
	double* s = static_cast<double*>(PyArray_DATA((PyArrayObject*) sstats));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_update_variables(self->m, &documents.view, l, (int) rows, (int64_t) cols, &params, g, s);
	Py_END_ALLOW_THREADS
	Py_XDECREF(latents_arr);
	if(status != TRLDA_OK) {
		Py_DECREF(gamma);
		Py_DECREF(sstats);
		return raise_status(self->m, status);
	}
	PyObject* result = Py_BuildValue("(OO)", gamma, sstats);
	Py_DECREF(gamma);
	Py_DECREF(sstats);
	return result;
}

// lower_bound (ldainterface.cpp:420-469)
PyObject* LDA_lower_bound(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "num_documents", "inference_method", "max_iter", "num_samples", "burn_in", "_latents", nullptr};
	Documents documents;
	trlda_params params;
	trlda_params_default(&params);
	int num_documents = -1;
	const char* inference_method = nullptr;
	PyObject* latents = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|isiiiO", const_cast<char**>(kwlist), &docs_converter, &documents,
			&num_documents, &inference_method, &params.max_iter_inference, &params.num_samples, &params.burn_in, &latents))
		return nullptr;
	if(!parse_inference_method(inference_method, &params.inference_method))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* latents_arr = nullptr;
	if(latents && latents != Py_None) {
		latents_arr = as_farray(latents, &rows, &cols, "`_latents`");
		if(!latents_arr)
			return nullptr;
	}
	int status;
	double bound = 0.;
	const double* l = latents_arr ? static_cast<const double*>(PyArray_DATA((PyArrayObject*) latents_arr)) : nullptr;
	Py_BEGIN_ALLOW_THREADS
	status = trlda_lower_bound(self->m, &documents.view, l, (int) rows, (int64_t) cols, &params, num_documents, &bound, nullptr);
	Py_END_ALLOW_THREADS
	Py_XDECREF(latents_arr);
	if(status != TRLDA_OK)
		return raise_status(self->m, status);
	return PyFloat_FromDouble(bound);
}

// predictive_log_likelihood (no reference counterpart): document completion, trlda_predictive_log_likelihood
PyObject* LDA_predictive_log_likelihood(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "held_out", "latents", "max_iter", nullptr};
	Documents documents, held_out;
	trlda_params params;
	trlda_params_default(&params);
	PyObject* latents = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&O&|Oi", const_cast<char**>(kwlist), &docs_converter, &documents,
			&docs_converter, &held_out, &latents, &params.max_iter_inference))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* latents_arr = nullptr;
	if(latents && latents != Py_None) {
		latents_arr = as_farray(latents, &rows, &cols, "`latents`");
		if(!latents_arr)
			return nullptr;
	}
	int status;
	double total = 0.;
	int64_t tokens = 0;
	const double* l = latents_arr ? static_cast<const double*>(PyArray_DATA((PyArrayObject*) latents_arr)) : nullptr;
	Py_BEGIN_ALLOW_THREADS
	status = trlda_predictive_log_likelihood(self->m, &documents.view, &held_out.view, l, (int) rows, (int64_t) cols, &params,
	                                         &total, &tokens, nullptr);
	Py_END_ALLOW_THREADS
	Py_XDECREF(latents_arr);
	if(status != TRLDA_OK)
		return raise_status(self->m, status);
	return Py_BuildValue("(dL)", total, (long long) tokens);
}

// word_topics (no reference counterpart): trlda_word_topics
PyObject* LDA_word_topics(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "num_topics", "latents", "max_iter", "threshold", nullptr};
	Documents documents;
	trlda_params params;
	trlda_params_default(&params);
	int n = 1;
	PyObject* latents = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|iOid", const_cast<char**>(kwlist), &docs_converter, &documents, &n, &latents,
			&params.max_iter_inference, &params.threshold))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* latents_arr = nullptr;
	if(latents && latents != Py_None) {
		latents_arr = as_farray(latents, &rows, &cols, "`latents`");
		if(!latents_arr)
			return nullptr;
	}
	const trlda_docs& view = documents.view;
	npy_intp dims[2] = {view.num_docs > 0 ? (npy_intp) view.doc_ptr[view.num_docs] : 0, std::max(n, 0)};
	PyObject* topics = PyArray_SimpleNew(2, dims, NPY_INT32);
	PyObject* probs = topics ? PyArray_SimpleNew(2, dims, NPY_DOUBLE) : nullptr;
	PyObject* gamma = probs ? new_farray(trlda_num_topics(self->m), view.num_docs) : nullptr;
	if(!gamma) {
		Py_XDECREF(topics);
		Py_XDECREF(probs);
		Py_XDECREF(latents_arr);
		return nullptr;
	}
	int status;
	const double* l = latents_arr ? static_cast<const double*>(PyArray_DATA((PyArrayObject*) latents_arr)) : nullptr;
	int32_t* t = static_cast<int32_t*>(PyArray_DATA((PyArrayObject*) topics));
	double* p = static_cast<double*>(PyArray_DATA((PyArrayObject*) probs));
	double* g = static_cast<double*>(PyArray_DATA((PyArrayObject*) gamma));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_word_topics(self->m, &view, l, (int) rows, (int64_t) cols, &params, n, t, p, g);
	Py_END_ALLOW_THREADS
	Py_XDECREF(latents_arr);
	if(status != TRLDA_OK) {
		Py_DECREF(topics);
		Py_DECREF(probs);
		Py_DECREF(gamma);
		return raise_status(self->m, status);
	}
	PyObject* result = Py_BuildValue("(OOO)", topics, probs, gamma);
	Py_DECREF(topics);
	Py_DECREF(probs);
	Py_DECREF(gamma);
	return result;
}

// top_words (no reference counterpart): trlda_top_words
PyObject* LDA_top_words(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"num_words", nullptr};
	int n = 10;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "|i", const_cast<char**>(kwlist), &n))
		return nullptr;
	npy_intp dims[2] = {trlda_num_topics(self->m), std::max(n, 0)};
	PyObject* ids = PyArray_SimpleNew(2, dims, NPY_INT32);
	PyObject* probs = ids ? PyArray_SimpleNew(2, dims, NPY_DOUBLE) : nullptr;
	if(!probs) {
		Py_XDECREF(ids);
		return nullptr;
	}
	int status;
	int32_t* i = static_cast<int32_t*>(PyArray_DATA((PyArrayObject*) ids));
	double* p = static_cast<double*>(PyArray_DATA((PyArrayObject*) probs));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_top_words(self->m, n, i, p);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		Py_DECREF(ids);
		Py_DECREF(probs);
		return raise_status(self->m, status);
	}
	PyObject* result = Py_BuildValue("(OO)", ids, probs);
	Py_DECREF(ids);
	Py_DECREF(probs);
	return result;
}

// cooccurrence (no reference counterpart): trlda_cooccurrence
PyObject* LDA_cooccurrence(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "top_words", nullptr};
	Documents documents;
	PyObject* top_words = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&O", const_cast<char**>(kwlist), &docs_converter, &documents, &top_words))
		return nullptr;
	const int K = trlda_num_topics(self->m);
	// any integer array: ids beyond int32 become -1, which the library rejects as out of range
	PyObject* arr = PyArray_FROM_OTF(top_words, NPY_INT64, NPY_ARRAY_IN_ARRAY);
	if(!arr)
		return nullptr;
	PyArrayObject* a = (PyArrayObject*) arr;
	if(PyArray_NDIM(a) != 2 || PyArray_DIM(a, 0) != K) {
		Py_DECREF(arr);
		PyErr_SetString(PyExc_ValueError, "`top_words` should be a num_topics x n array of word IDs.");
		return nullptr;
	}
	const npy_intp n = PyArray_DIM(a, 1);
	const int64_t* src = static_cast<const int64_t*>(PyArray_DATA(a));
	std::vector<int32_t> ids((size_t) K * n);
	for(size_t j = 0; j < ids.size(); ++j)
		ids[j] = src[j] < INT32_MIN || src[j] > INT32_MAX ? -1 : (int32_t) src[j];
	Py_DECREF(arr);
	npy_intp dims[3] = {K, n, n};
	PyObject* counts = PyArray_SimpleNew(3, dims, NPY_INT64);
	if(!counts)
		return nullptr;
	int status;
	int64_t num_docs = 0;
	int64_t* c = static_cast<int64_t*>(PyArray_DATA((PyArrayObject*) counts));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_cooccurrence(self->m, &documents.view, ids.data(), (int) std::min<npy_intp>(n, INT32_MAX), c, &num_docs);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		Py_DECREF(counts);
		return raise_status(self->m, status);
	}
	PyObject* result = Py_BuildValue("(OL)", counts, (long long) num_docs);
	Py_DECREF(counts);
	return result;
}

extern PyTypeObject LDA_type;

// topic_distances (no reference counterpart): trlda_topic_distances
PyObject* LDA_topic_distances(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"other", "metric", nullptr};
	PyObject* other = Py_None;
	const char* metric = "hellinger";
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "|Os", const_cast<char**>(kwlist), &other, &metric))
		return nullptr;
	LDAObject* o = self;
	if(other != Py_None) {
		if(!PyObject_TypeCheck(other, &LDA_type)) {
			PyErr_SetString(PyExc_TypeError, "`other` should be a model (OnlineLDA, BatchLDA or CumulativeLDA).");
			return nullptr;
		}
		o = (LDAObject*) other;
		REQUIRE_MODEL(o, nullptr);
	}
	int code;
	if(!strcmp(metric, "hellinger"))
		code = TRLDA_DISTANCE_HELLINGER;
	else if(!strcmp(metric, "kullback_leibler"))
		code = TRLDA_DISTANCE_KL;
	else {
		PyErr_SetString(PyExc_ValueError, "`metric` should be either 'hellinger' or 'kullback_leibler'.");
		return nullptr;
	}
	PyObject* out = new_farray(trlda_num_topics(self->m), trlda_num_topics(o->m));
	if(!out)
		return nullptr;
	int status;
	double* d = static_cast<double*>(PyArray_DATA((PyArrayObject*) out));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_topic_distances(self->m, o->m, code, d);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK) {
		Py_DECREF(out);
		return raise_status(self->m, status);
	}
	return out;
}

// index_documents (no reference counterpart): trlda_index_documents
PyObject* LDA_index_documents(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"gamma", nullptr};
	PyObject* gamma = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O", const_cast<char**>(kwlist), &gamma))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* arr = as_farray(gamma, &rows, &cols, "Gamma");
	if(!arr)
		return nullptr;
	int status;
	const double* g = static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_index_documents(self->m, g, (int) rows, (int64_t) cols);
	Py_END_ALLOW_THREADS
	Py_DECREF(arr);
	if(status != TRLDA_OK)
		return raise_status(self->m, status);
	Py_RETURN_NONE;
}

// similar_documents (no reference counterpart): trlda_similar_documents
PyObject* LDA_similar_documents(LDAObject* self, PyObject* args, PyObject* kwds) {
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"gamma", "num_neighbors", nullptr};
	PyObject* gamma = nullptr;
	int n = 10;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O|i", const_cast<char**>(kwlist), &gamma, &n))
		return nullptr;
	npy_intp rows = 0, cols = 0;
	PyObject* arr = as_farray(gamma, &rows, &cols, "Gamma");
	if(!arr)
		return nullptr;
	npy_intp dims[2] = {cols, std::max(n, 0)};
	PyObject* ids = PyArray_SimpleNew(2, dims, NPY_INT64);
	PyObject* dist = ids ? PyArray_SimpleNew(2, dims, NPY_DOUBLE) : nullptr;
	if(!dist) {
		Py_XDECREF(ids);
		Py_DECREF(arr);
		return nullptr;
	}
	int status;
	const double* g = static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr));
	int64_t* i = static_cast<int64_t*>(PyArray_DATA((PyArrayObject*) ids));
	double* d = static_cast<double*>(PyArray_DATA((PyArrayObject*) dist));
	Py_BEGIN_ALLOW_THREADS
	status = trlda_similar_documents(self->m, g, (int) rows, (int64_t) cols, n, i, d);
	Py_END_ALLOW_THREADS
	Py_DECREF(arr);
	if(status != TRLDA_OK) {
		Py_DECREF(ids);
		Py_DECREF(dist);
		return raise_status(self->m, status);
	}
	PyObject* result = Py_BuildValue("(OO)", ids, dist);
	Py_DECREF(ids);
	Py_DECREF(dist);
	return result;
}

PyObject* LDA_str(PyObject* self_) {                                      // ldainterface.cpp:473-490
	LDAObject* self = (LDAObject*) self_;
	REQUIRE_MODEL(self, nullptr);
	const int K = trlda_num_topics(self->m);
	std::vector<double> alpha(K);
	double eta;
	trlda_get_alpha(self->m, alpha.data());
	trlda_get_eta(self->m, &eta);
	double lo = alpha[0], hi = alpha[0];
	for(double a : alpha) {
		lo = a < lo ? a : lo;
		hi = a > hi ? a : hi;
	}
	char buffer[256];
	snprintf(buffer, sizeof(buffer), "Number of topics: %d\nEta: %.4g\nAlpha: %.4g, %.4g (min, max)\n", K, eta, lo, hi);
	return PyUnicode_FromString(buffer);
}

// installs the private parity seams before an update_parameters call
int install_injections(LDAObject* self, PyObject* gamma0, PyObject* lambda0) {
	if(gamma0 && gamma0 != Py_None) {
		npy_intp rows, cols;
		PyObject* arr = as_farray(gamma0, &rows, &cols, "`_initial_gamma`");
		if(!arr)
			return 0;
		const int status = trlda_inject_initial_gamma(self->m, static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr)), (int) rows, (int64_t) cols);
		Py_DECREF(arr);
		if(status != TRLDA_OK) {
			raise_status(self->m, status);
			return 0;
		}
	}
	if(lambda0 && lambda0 != Py_None) {
		npy_intp rows, cols;
		PyObject* arr = as_farray(lambda0, &rows, &cols, "`_initial_lambda`");
		if(!arr)
			return 0;
		const int status = trlda_inject_initial_lambda(self->m, static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr)), (int) rows, (int) cols);
		Py_DECREF(arr);
		if(status != TRLDA_OK) {
			raise_status(self->m, status);
			return 0;
		}
	}
	return 1;
}

PyObject* run_update(LDAObject* self, Documents& documents, const trlda_params& params) {
	int status;
	double result = 0.;
	Py_BEGIN_ALLOW_THREADS
	status = trlda_update_parameters(self->m, &documents.view, &params, &result);
	Py_END_ALLOW_THREADS
	if(status != TRLDA_OK)
		return raise_status(self->m, status);
	return PyFloat_FromDouble(result);
}

// pickle support shared by the three classes: (type, ctor args, state)
PyObject* reduce_common(LDAObject* self, bool online) {
	REQUIRE_MODEL(self, nullptr);
	PyObject* alpha = LDA_alpha(self, nullptr);
	PyObject* lambda = alpha ? LDA_lambda(self, nullptr) : nullptr;
	if(!lambda) {
		Py_XDECREF(alpha);
		return nullptr;
	}
	double eta;
	trlda_get_eta(self->m, &eta);
	PyObject *ctor, *state;
	if(online) {                                                          // onlineldainterface.cpp:265-290
		int64_t D, count;
		trlda_get_num_documents(self->m, &D);
		trlda_get_update_count(self->m, &count);
		ctor = Py_BuildValue("(iilOd)", trlda_num_words(self->m), trlda_num_topics(self->m), (long) D, alpha, eta);
		state = Py_BuildValue("(Ol)", lambda, (long) count);
	} else {                                                              // batchldainterface.cpp:181-203
		ctor = Py_BuildValue("(iiOd)", trlda_num_words(self->m), trlda_num_topics(self->m), alpha, eta);
		state = Py_BuildValue("(O)", lambda);
	}
	PyObject* result = (ctor && state) ? Py_BuildValue("(OOO)", Py_TYPE(self), ctor, state) : nullptr;
	Py_DECREF(alpha);
	Py_DECREF(lambda);
	Py_XDECREF(ctor);
	Py_XDECREF(state);
	return result;
}

// ---- OnlineLDA -----------------------------------------------------------------------------------------------------------
int OnlineLDA_init(LDAObject* self, PyObject* args, PyObject* kwds) {    // onlineldainterface.cpp:35-90
	const char* kwlist[] = {"num_words", "num_topics", "num_documents", "alpha", "eta", "kappa_", "tau_", "device", "precision", nullptr};
	int num_words, num_topics, device = 0;
	long num_documents;
	PyObject* alpha = nullptr;
	double eta = .3, kappa_ = 0., tau_ = 0.;   // kappa_/tau_: accepted for old pickles and ignored, as in the reference
	const char* precision = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "iil|Odddiz", const_cast<char**>(kwlist), &num_words, &num_topics,
			&num_documents, &alpha, &eta, &kappa_, &tau_, &device, &precision))
		return -1;
	return create_model(self, TRLDA_KIND_ONLINE, num_words, num_topics, num_documents, alpha, eta, device, precision);
}

PyObject* OnlineLDA_num_documents(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	int64_t n;
	trlda_get_num_documents(self->m, &n);
	return PyLong_FromLongLong(n);
}

int OnlineLDA_set_num_documents(LDAObject* self, PyObject* value, void*) {
	REQUIRE_MODEL(self, -1);
	const long long n = value ? PyLong_AsLongLong(value) : -1;
	if(PyErr_Occurred())
		return -1;
	if(trlda_set_num_documents(self->m, n) != TRLDA_OK) {
		raise_status(self->m, 1);
		return -1;
	}
	return 0;
}

PyObject* OnlineLDA_update_count(LDAObject* self, void*) {
	REQUIRE_MODEL(self, nullptr);
	int64_t n;
	trlda_get_update_count(self->m, &n);
	return PyLong_FromLongLong(n);
}

int OnlineLDA_set_update_count(LDAObject* self, PyObject* value, void*) {
	REQUIRE_MODEL(self, -1);
	const long long n = value ? PyLong_AsLongLong(value) : -1;
	if(PyErr_Occurred())
		return -1;
	if(trlda_set_update_count(self->m, n) != TRLDA_OK) {
		raise_status(self->m, 1);
		return -1;
	}
	return 0;
}

PyObject* OnlineLDA_update_parameters(LDAObject* self, PyObject* args, PyObject* kwds) {   // onlineldainterface.cpp:204-256
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "max_iter_tr", "max_iter_inference", "kappa", "tau", "rho", "adaptive", "init_gamma",
		"update_lambda", "update_alpha", "update_eta", "min_alpha", "min_eta", "verbosity", "_initial_gamma", nullptr};
	Documents documents;
	trlda_params p;
	trlda_params_default(&p);
	p.max_iter_inference = 20;                                            // onlineldainterface.cpp:226-227
	PyObject* gamma0 = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|iidddpppppddiO", const_cast<char**>(kwlist), &docs_converter, &documents,
			&p.max_iter_tr, &p.max_iter_inference, &p.kappa, &p.tau, &p.rho, &p.adaptive, &p.init_gamma, &p.update_lambda,
			&p.update_alpha, &p.update_eta, &p.min_alpha, &p.min_eta, &p.verbosity, &gamma0))
		return nullptr;
	if(!install_injections(self, gamma0, nullptr))
		return nullptr;
	return run_update(self, documents, p);                                // returns the learning rate used
}

PyObject* OnlineLDA_reduce(LDAObject* self, PyObject*) { return reduce_common(self, true); }

PyObject* OnlineLDA_setstate(LDAObject* self, PyObject* state) {         // onlineldainterface.cpp:292-313
	PyObject* lambda;
	long update_count;
	if(!PyArg_ParseTuple(state, "Ol", &lambda, &update_count))
		return nullptr;
	if(LDA_set_lambda(self, lambda, nullptr) < 0)
		return nullptr;
	if(trlda_set_update_count(self->m, update_count) != TRLDA_OK)
		return raise_status(self->m, 1);
	Py_RETURN_NONE;
}

// ---- BatchLDA ------------------------------------------------------------------------------------------------------------
int BatchLDA_init(LDAObject* self, PyObject* args, PyObject* kwds) {     // batchldainterface.cpp:33-80
	const char* kwlist[] = {"num_words", "num_topics", "alpha", "eta", "device", "precision", nullptr};
	int num_words, num_topics, device = 0;
	PyObject* alpha = nullptr;
	double eta = .3;
	const char* precision = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "ii|Odiz", const_cast<char**>(kwlist), &num_words, &num_topics, &alpha, &eta, &device, &precision))
		return -1;
	return create_model(self, TRLDA_KIND_BATCH, num_words, num_topics, 0, alpha, eta, device, precision);
}

PyObject* BatchLDA_update_parameters(LDAObject* self, PyObject* args, PyObject* kwds) {    // batchldainterface.cpp:126-172
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "max_epochs", "max_iter_inference", "max_iter_alpha", "max_iter_eta", "update_lambda",
		"update_alpha", "update_eta", "min_alpha", "min_eta", "emp_bayes_threshold", "verbosity", "_initial_gamma", nullptr};
	Documents documents;
	trlda_params p;
	trlda_params_default(&p);
	PyObject* gamma0 = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|iiiipppdddiO", const_cast<char**>(kwlist), &docs_converter, &documents,
			&p.max_epochs, &p.max_iter_inference, &p.max_iter_alpha, &p.max_iter_eta, &p.update_lambda, &p.update_alpha,
			&p.update_eta, &p.min_alpha, &p.min_eta, &p.emp_bayes_threshold, &p.verbosity, &gamma0))
		return nullptr;
	if(!install_injections(self, gamma0, nullptr))
		return nullptr;
	return run_update(self, documents, p);
}

PyObject* Simple_reduce(LDAObject* self, PyObject*) { return reduce_common(self, false); }

PyObject* Simple_setstate(LDAObject* self, PyObject* state) {            // batchldainterface.cpp:205-227
	PyObject* lambda;
	if(!PyArg_ParseTuple(state, "O", &lambda))
		return nullptr;
	if(LDA_set_lambda(self, lambda, nullptr) < 0)
		return nullptr;
	Py_RETURN_NONE;
}

// ---- CumulativeLDA -------------------------------------------------------------------------------------------------------
int CumulativeLDA_init(LDAObject* self, PyObject* args, PyObject* kwds) {   // cumulativeldainterface.cpp:30-77
	const char* kwlist[] = {"num_words", "num_topics", "alpha", "eta", "device", "precision", nullptr};
	int num_words, num_topics, device = 0;
	PyObject* alpha = nullptr;
	double eta = .3;
	const char* precision = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "ii|Odiz", const_cast<char**>(kwlist), &num_words, &num_topics, &alpha, &eta, &device, &precision))
		return -1;
	return create_model(self, TRLDA_KIND_CUMULATIVE, num_words, num_topics, 0, alpha, eta, device, precision);
}

PyObject* CumulativeLDA_update_parameters(LDAObject* self, PyObject* args, PyObject* kwds) {   // cumulativeldainterface.cpp:119-162
	REQUIRE_MODEL(self, nullptr);
	const char* kwlist[] = {"docs", "max_epochs", "max_iter_inference", "max_iter_alpha", "update_lambda", "update_alpha",
		"min_alpha", "emp_bayes_threshold", "inference_threshold", "verbosity", "_initial_gamma", "_initial_lambda", nullptr};
	Documents documents;
	trlda_params p;
	trlda_params_default(&p);
	PyObject *gamma0 = nullptr, *lambda0 = nullptr;
	if(!PyArg_ParseTupleAndKeywords(args, kwds, "O&|iiippdddiOO", const_cast<char**>(kwlist), &docs_converter, &documents,
			&p.max_epochs, &p.max_iter_inference, &p.max_iter_alpha, &p.update_lambda, &p.update_alpha, &p.min_alpha,
			&p.emp_bayes_threshold, &p.threshold, &p.verbosity, &gamma0, &lambda0))
		return nullptr;
	if(!install_injections(self, gamma0, lambda0))
		return nullptr;
	return run_update(self, documents, p);
}

// ---- module functions ------------------------------------------------------------------------------------------------------
PyObject* module_seed(PyObject*, PyObject* args) {                       // module.cpp:332-342
	long long seed;
	if(!PyArg_ParseTuple(args, "L", &seed))
		return nullptr;
	trlda_seed((uint64_t) seed);
	srand((unsigned) seed);
	Py_RETURN_NONE;
}

PyObject* module_polygamma(PyObject*, PyObject* args) {                  // utilsinterface.cpp: polygamma(n, x)
	int n;
	PyObject* x;
	if(!PyArg_ParseTuple(args, "iO", &n, &x))
		return nullptr;
	if(PyFloat_Check(x) || PyLong_Check(x))
		return PyFloat_FromDouble(trlda_polygamma(n, PyFloat_AsDouble(x)));
	PyObject* arr = PyArray_FROM_OTF(x, NPY_DOUBLE, NPY_ARRAY_IN_ARRAY);
	if(!arr)
		return nullptr;
	PyObject* out = PyArray_NewLikeArray((PyArrayObject*) arr, NPY_CORDER, nullptr, 0);
	if(out) {
		const double* src = static_cast<const double*>(PyArray_DATA((PyArrayObject*) arr));
		double* dst = static_cast<double*>(PyArray_DATA((PyArrayObject*) out));
		const npy_intp size = PyArray_SIZE((PyArrayObject*) arr);
		for(npy_intp i = 0; i < size; ++i)
			dst[i] = trlda_polygamma(n, src[i]);
	}
	Py_DECREF(arr);
	return out;
}

// ---- type tables -----------------------------------------------------------------------------------------------------------
const char* update_variables_doc =
	"update_variables(docs, latents=None, inference_method='VI', max_iter=100, threshold=0.001, num_samples=1, burn_in=2)\n\n"
	"Computes beliefs over topic assignments for the given documents (E-step) on the GPU.  Returns a tuple of the\n"
	"K x N Dirichlet parameters gamma and the K x W sufficient statistics (float64, Fortran order).";

const char* predictive_log_likelihood_doc =
	"predictive_log_likelihood(docs, held_out, latents=None, max_iter=100)\n\n"
	"Document-completion predictive log-likelihood (Hoffman, Blei, Wang & Paisley 2013, section 5) on the GPU.  gamma is\n"
	"fitted on `docs` (the observed part of each document, the E-step of update_variables; `latents` is the initial\n"
	"gamma, a fresh draw if None), then every held-out token w of document d is scored with\n"
	"log sum_k E[theta_dk] E[beta_kw].  `held_out` has one document for each of `docs`, and both take the list or the\n"
	"(doc_ptr, word_ids, counts) form; trlda.utils.split_documents makes such a pair.  Returns the tuple\n"
	"(log_likelihood, num_tokens): the summed log-likelihood and the number of held-out tokens.  The per-word figure is\n"
	"log_likelihood / num_tokens and the perplexity exp(-log_likelihood / num_tokens); returning the pair lets batches\n"
	"of held-out documents be added up.  The model's parameters are not changed.";

const char* word_topics_doc =
	"word_topics(docs, num_topics=1, latents=None, max_iter=100, threshold=0.001)\n\n"
	"The num_topics (1 to 32, at most the model's num_topics) most probable topics of every (word, count) pair of `docs`\n"
	"(the list or the (doc_ptr, word_ids, counts) form), computed on the GPU.  gamma is fitted exactly as update_variables\n"
	"fits it (`latents` is the initial gamma, a fresh draw if None), then pair j with word w in document d gets\n"
	"phi_jk = exp(s_jk) / sum_k' exp(s_jk'),  s_jk = psi(gamma_dk) + psi(lambda_kw) - psi(sum_v lambda_kv),\n"
	"the responsibility of topic k for the word that the E-step uses, evaluated in float64 in both precision modes.\n"
	"Returns the tuple (topics, probs, gamma): int32 and float64 arrays of shape (num_pairs, num_topics), row j for the j-th\n"
	"pair in the given order, its topics by descending phi (equal phi: the smaller topic id first) and their phi; and\n"
	"gamma (num_topics x num_documents, float64, Fortran order), the same as update_variables returns.  Pairs with count 0\n"
	"and repeated words get rows like any other pair.  A token's topic is topics[j, 0]; the tokens of topic k in the batch\n"
	"are counts[topics[:, 0] == k].sum().  Like update_variables, the call replaces the minibatch held on the GPU; the\n"
	"model's parameters are not changed.";

const char* top_words_doc =
	"top_words(num_words=10)\n\n"
	"The num_words (1 to 32, at most num_words of the model) most probable words of every topic, on the GPU: words ordered\n"
	"by E[beta_kw] = lambda_kw / sum_w lambda_kw, descending, ties broken by the smaller word id.  Returns the tuple\n"
	"(ids, probs) of two num_topics x num_words arrays, int32 word ids and their float64 E[beta_kw], each row in rank\n"
	"order.  Only the lists leave the device, not lambda.";

const char* cooccurrence_doc =
	"cooccurrence(docs, top_words)\n\n"
	"Document frequencies of each topic's top words in `docs` (the list or the (doc_ptr, word_ids, counts) form), counted\n"
	"on the GPU.  `top_words` is a num_topics x n integer array of word IDs (1 <= n <= 32, distinct within a row), e.g.\n"
	"the ids of top_words().  Returns the tuple (counts, num_docs): counts[k, i, j] is the number of documents that\n"
	"contain both top_words[k, i] and top_words[k, j] (the diagonal: documents that contain the word), num_docs the\n"
	"number of documents.  A word is in a document when one of its pairs there has a positive count.  Both are integers,\n"
	"so the results of several batches of documents can be added up; trlda.utils.topic_coherence does that and turns\n"
	"them into UMass or NPMI coherence.  The model's parameters are not changed.";

const char* topic_distances_doc =
	"topic_distances(other=None, metric='hellinger')\n\n"
	"Distances between the topics of this model and those of `other` (another model with the same num_words on the same\n"
	"GPU; None: this model), computed on the GPU from E[beta_k] = lambda_k / sum_w lambda_kw.  Returns a float64 array\n"
	"of shape (num_topics, other.num_topics) in Fortran order, D[i, j] between topic i here and topic j there.\n\n"
	"metric='hellinger': D_ij = sqrt(max(0, 1 - sum_w sqrt(p_iw q_jw))), symmetric and in [0, 1].\n"
	"metric='kullback_leibler': D_ij = KL(p_i || q_j) = sum_w p_iw log(p_iw / q_jw), clamped at 0; other's lambda\n"
	"must be positive.\n\n"
	"The inner sum is accumulated in float64 over the vocabulary, so its rounding error is about num_words * 1e-16:\n"
	"distances below about 1e-5 (Hellinger, the square root of that error) and 1e-9 (Kullback-Leibler) are not\n"
	"resolved, and a topic's distance to itself comes out at that floor rather than 0.  The result is reproducible\n"
	"bit for bit, the same in both precision modes, and exactly symmetric for model.topic_distances().\n\n"
	"To match the topics of two runs (the order of topics is arbitrary), e.g. with scipy:\n\n"
	"    from scipy.optimize import linear_sum_assignment\n"
	"    d = model.topic_distances(other)\n"
	"    rows, cols = linear_sum_assignment(d)   # topic rows[i] here is topic cols[i] there\n"
	"    print(d[rows, cols].mean())\n\n"
	"The model's parameters are not changed.";

const char* index_documents_doc =
	"index_documents(gamma)\n\n"
	"Replaces the model's document index with the documents of `gamma` (num_topics x D, as update_variables returns it;\n"
	"Gibbs theta works too), for similar_documents.  A document's topic proportions are theta_d = gamma_d / sum_k gamma_dk.\n"
	"The index stays on the GPU, 8 bytes per topic and document (8.4 GB for 1000 topics and 2^20 documents), until it is\n"
	"replaced, emptied with a gamma of 0 columns, or the model is deleted.  It is not pickled with the model, and training\n"
	"does not change it.  Gamma must be finite and non-negative, with a positive sum in every column; on any error the\n"
	"model is left with no index.  The model's parameters are not changed.";

const char* similar_documents_doc =
	"similar_documents(gamma, num_neighbors=10)\n\n"
	"The num_neighbors indexed documents nearest to each of the Q query documents of `gamma` (num_topics x Q), under the\n"
	"Hellinger distance of their topic proportions: D(q, d) = sqrt(max(0, 1 - sum_k sqrt(theta_qk theta_dk))), in float64\n"
	"on the GPU.  Returns (ids, distances), int64 and float64 arrays of shape (Q, num_neighbors): row q lists the column\n"
	"numbers of the indexed gamma, nearest first; exact ties go to the smaller id.  The result is reproducible bit for bit\n"
	"and does not depend on the other queries.  1 <= num_neighbors <= min(32, indexed documents).  On several GPUs every\n"
	"rank searches its own index.\n\n"
	"    model.index_documents(model.update_variables(corpus)[0])\n"
	"    ids, dist = model.similar_documents(model.update_variables(queries)[0], 10)\n\n"
	"The model's parameters are not changed.";

PyGetSetDef LDA_getset[] = {
	{"num_topics", (getter) LDA_num_topics, nullptr, "Number of topics.", nullptr},
	{"num_words", (getter) LDA_num_words, nullptr, "Number of words.", nullptr},
	{"lambdas", (getter) LDA_lambda, (setter) LDA_set_lambda, "Parameters of the Dirichlet beliefs over topics (K x W).", nullptr},
	{"_lambda", (getter) LDA_lambda, (setter) LDA_set_lambda, "Alias for lambdas.", nullptr},
	{"alpha", (getter) LDA_alpha, (setter) LDA_set_alpha, "Parameters of the Dirichlet prior over topic proportions.", nullptr},
	{"eta", (getter) LDA_eta, (setter) LDA_set_eta, "Parameter of the Dirichlet prior over topics.", nullptr},
	{"precision", (getter) LDA_precision, (setter) LDA_set_precision, "'fp64' or 'mixed' (float32 tile, float64 accumulation).", nullptr},
	{nullptr, nullptr, nullptr, nullptr, nullptr}};

PyMethodDef LDA_methods[] = {
	{"sample", (PyCFunction) LDA_sample, METH_VARARGS | METH_KEYWORDS, "sample(num_documents, length, collapse=False)"},
	{"update_variables", (PyCFunction) LDA_update_variables, METH_VARARGS | METH_KEYWORDS, update_variables_doc},
	{"do_e_step", (PyCFunction) LDA_update_variables, METH_VARARGS | METH_KEYWORDS, update_variables_doc},   // module.cpp:99-106
	{"lower_bound", (PyCFunction) LDA_lower_bound, METH_VARARGS | METH_KEYWORDS,
		"lower_bound(docs, num_documents=-1, inference_method='VI', max_iter=100, num_samples=1, burn_in=2)"},
	{"predictive_log_likelihood", (PyCFunction) LDA_predictive_log_likelihood, METH_VARARGS | METH_KEYWORDS,
		predictive_log_likelihood_doc},
	{"word_topics", (PyCFunction) LDA_word_topics, METH_VARARGS | METH_KEYWORDS, word_topics_doc},
	{"top_words", (PyCFunction) LDA_top_words, METH_VARARGS | METH_KEYWORDS, top_words_doc},
	{"cooccurrence", (PyCFunction) LDA_cooccurrence, METH_VARARGS | METH_KEYWORDS, cooccurrence_doc},
	{"topic_distances", (PyCFunction) LDA_topic_distances, METH_VARARGS | METH_KEYWORDS, topic_distances_doc},
	{"index_documents", (PyCFunction) LDA_index_documents, METH_VARARGS | METH_KEYWORDS, index_documents_doc},
	{"similar_documents", (PyCFunction) LDA_similar_documents, METH_VARARGS | METH_KEYWORDS, similar_documents_doc},
	{nullptr, nullptr, 0, nullptr}};

PyGetSetDef OnlineLDA_getset[] = {
	{"num_documents", (getter) OnlineLDA_num_documents, (setter) OnlineLDA_set_num_documents, "Number of documents of the full corpus.", nullptr},
	{"update_count", (getter) OnlineLDA_update_count, (setter) OnlineLDA_set_update_count, "Number of calls to update_parameters so far.", nullptr},
	{nullptr, nullptr, nullptr, nullptr, nullptr}};

PyMethodDef OnlineLDA_methods[] = {
	{"update_parameters", (PyCFunction) OnlineLDA_update_parameters, METH_VARARGS | METH_KEYWORDS,
		"update_parameters(docs, max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100, rho=-1, adaptive=False, init_gamma=True, "
		"update_lambda=True, update_alpha=False, update_eta=False, min_alpha=1e-6, min_eta=1e-6, verbosity=0)\n\n"
		"Trust-region update of the beliefs over topics; returns the learning rate used."},
	{"__reduce__", (PyCFunction) OnlineLDA_reduce, METH_NOARGS, "Method used by Pickle."},
	{"__setstate__", (PyCFunction) OnlineLDA_setstate, METH_O, "Method used by Pickle."},
	{nullptr, nullptr, 0, nullptr}};

PyMethodDef BatchLDA_methods[] = {
	{"update_parameters", (PyCFunction) BatchLDA_update_parameters, METH_VARARGS | METH_KEYWORDS,
		"update_parameters(docs, max_epochs=100, max_iter_inference=100, max_iter_alpha=10, max_iter_eta=20, update_lambda=True, "
		"update_alpha=False, update_eta=False, min_alpha=1e-6, min_eta=1e-6, emp_bayes_threshold=1e-8, verbosity=0)"},
	{"__reduce__", (PyCFunction) Simple_reduce, METH_NOARGS, "Method used by Pickle."},
	{"__setstate__", (PyCFunction) Simple_setstate, METH_O, "Method used by Pickle."},
	{nullptr, nullptr, 0, nullptr}};

PyMethodDef CumulativeLDA_methods[] = {
	{"update_parameters", (PyCFunction) CumulativeLDA_update_parameters, METH_VARARGS | METH_KEYWORDS,
		"update_parameters(docs, max_epochs=100, max_iter_inference=100, max_iter_alpha=10, update_lambda=True, update_alpha=False, "
		"min_alpha=1e-6, emp_bayes_threshold=1e-8, inference_threshold=0.001, verbosity=0)"},
	{"__reduce__", (PyCFunction) Simple_reduce, METH_NOARGS, "Method used by Pickle."},
	{"__setstate__", (PyCFunction) Simple_setstate, METH_O, "Method used by Pickle."},
	{nullptr, nullptr, 0, nullptr}};

PyTypeObject Distribution_type = {PyVarObject_HEAD_INIT(nullptr, 0)};
PyTypeObject LDA_type = {PyVarObject_HEAD_INIT(nullptr, 0)};
PyTypeObject OnlineLDA_type = {PyVarObject_HEAD_INIT(nullptr, 0)};
PyTypeObject BatchLDA_type = {PyVarObject_HEAD_INIT(nullptr, 0)};
PyTypeObject CumulativeLDA_type = {PyVarObject_HEAD_INIT(nullptr, 0)};

void fill_type(PyTypeObject& t, const char* name, const char* doc, PyTypeObject* base, initproc init,
               PyMethodDef* methods, PyGetSetDef* getset) {
	t.tp_name = name;
	t.tp_basicsize = sizeof(LDAObject);
	t.tp_flags = Py_TPFLAGS_DEFAULT | Py_TPFLAGS_BASETYPE;
	t.tp_doc = doc;
	t.tp_base = base;
	t.tp_init = init;
	t.tp_methods = methods;
	t.tp_getset = getset;
	if(!base) {
		t.tp_new = Distribution_new;
		t.tp_dealloc = (destructor) Distribution_dealloc;
	}
}

// _pack_documents(docs) -> (doc_ptr, word_ids, counts): the binding's list walk on its own, as numpy CSR arrays - what
// every method does with its `docs` argument before it calls the C ABI (no device needed; used by tests and to time it)
PyObject* module_pack_documents(PyObject*, PyObject* args) {
	Documents documents;
	if(!PyArg_ParseTuple(args, "O&", &docs_converter, &documents))
		return nullptr;
	const npy_intp B1 = (npy_intp) documents.view.num_docs + 1;
	const npy_intp N = (npy_intp) documents.view.doc_ptr[documents.view.num_docs];
	PyObject* ptr = PyArray_SimpleNew(1, &B1, NPY_INT64);
	PyObject* ids = PyArray_SimpleNew(1, &N, NPY_INT32);
	PyObject* cts = PyArray_SimpleNew(1, &N, NPY_INT32);
	if(!ptr || !ids || !cts) {
		Py_XDECREF(ptr); Py_XDECREF(ids); Py_XDECREF(cts);
		return nullptr;
	}
	memcpy(PyArray_DATA((PyArrayObject*) ptr), documents.view.doc_ptr, sizeof(int64_t) * B1);
	if(N) {
		memcpy(PyArray_DATA((PyArrayObject*) ids), documents.view.word_ids, sizeof(int32_t) * N);
		memcpy(PyArray_DATA((PyArrayObject*) cts), documents.view.counts, sizeof(int32_t) * N);
	}
	PyObject* result = Py_BuildValue("(OOO)", ptr, ids, cts);
	Py_DECREF(ptr); Py_DECREF(ids); Py_DECREF(cts);
	return result;
}

PyMethodDef module_methods[] = {
	{"_pack_documents", module_pack_documents, METH_VARARGS, "_pack_documents(docs)\n\nThe binding's list -> CSR conversion on its own."},
	{"seed", module_seed, METH_VARARGS, "seed(value)\n\nSeeds the generators used for the initial gamma / lambda."},
	{"polygamma", module_polygamma, METH_VARARGS, "polygamma(n, x)\n\nThe n-th derivative of the digamma function."},
	{nullptr, nullptr, 0, nullptr}};

PyModuleDef module_def = {
	PyModuleDef_HEAD_INIT, "_trlda", "B200-native implementation of trust-region latent Dirichlet allocation.", -1, module_methods,
	nullptr, nullptr, nullptr, nullptr};

}  // namespace

PyMODINIT_FUNC PyInit__trlda(void) {
	import_array();
	fill_type(Distribution_type, "trlda_b200.models.Distribution", "Abstract base class.", nullptr, (initproc) abstract_init, nullptr, nullptr);
	fill_type(LDA_type, "trlda_b200.models.LDA", "Abstract base class.", &Distribution_type, (initproc) abstract_init, LDA_methods, LDA_getset);
	LDA_type.tp_str = LDA_str;
	fill_type(OnlineLDA_type, "trlda_b200.models.OnlineLDA",
		"An implementation of an online trust region method for latent Dirichlet allocation.\n\n"
		"    model = OnlineLDA(num_words=7000, num_topics=100, num_documents=10000, alpha=.1, eta=.3)\n\n"
		"alpha can be a scalar or an array with one entry for each topic.",
		&LDA_type, (initproc) OnlineLDA_init, OnlineLDA_methods, OnlineLDA_getset);
	fill_type(BatchLDA_type, "trlda_b200.models.BatchLDA", "Batch variational Bayes for latent Dirichlet allocation.",
		&LDA_type, (initproc) BatchLDA_init, BatchLDA_methods, nullptr);
	fill_type(CumulativeLDA_type, "trlda_b200.models.CumulativeLDA", "Streaming (SDA-Bayes style) latent Dirichlet allocation.",
		&LDA_type, (initproc) CumulativeLDA_init, CumulativeLDA_methods, nullptr);

	PyTypeObject* types[] = {&Distribution_type, &LDA_type, &OnlineLDA_type, &BatchLDA_type, &CumulativeLDA_type};
	for(PyTypeObject* t : types)
		if(PyType_Ready(t) < 0)
			return nullptr;
	PyObject* module = PyModule_Create(&module_def);
	if(!module)
		return nullptr;
	const char* names[] = {"Distribution", "LDA", "OnlineLDA", "BatchLDA", "CumulativeLDA"};   // module.cpp:386-390
	for(int i = 0; i < 5; ++i) {
		Py_INCREF(types[i]);
		PyModule_AddObject(module, names[i], (PyObject*) types[i]);
	}
	return module;
}
