from trlda_b200.utils import load_documents, load_documents_csr, random_select, sample_dirichlet, split_documents, \
	coherence_from_counts, topic_coherence, polygamma

__all__ = ['load_documents', 'load_documents_csr', 'random_select', 'sample_dirichlet', 'split_documents', 'coherence_from_counts',
	'topic_coherence', 'polygamma']
