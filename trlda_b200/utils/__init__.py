"""trlda.utils of the reference (code/trlda/python/utils/__init__.py): the helpers on the hot path's boundary.

`load_users` / `load_users_as_dict` (collaborative-filtering loaders) are outside the scope of this build."""
from .load_documents import load_documents, load_documents_csr
from .._sample import random_select, sample_dirichlet, split_documents
from .._coherence import coherence_from_counts, topic_coherence


def polygamma(n, x):
	"""n-th derivative of the digamma function (reference: utils.cpp:107-111 through utilsinterface.cpp)."""
	from .. import _trlda
	return _trlda.polygamma(n, x)


__all__ = ['load_documents', 'load_documents_csr', 'random_select', 'sample_dirichlet', 'split_documents', 'coherence_from_counts',
	'topic_coherence', 'polygamma']
