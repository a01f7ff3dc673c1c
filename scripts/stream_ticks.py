"""Phase timers of the streaming E-step kernel inside real update_parameters steps on the cfg-3 shape (fresh minibatch
per step).  PREC=fp64 runs every document on it; in mixed mode it takes the documents of more than 192 pairs."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ['TRLDA_ESTEP_TICKS'] = '1'
import numpy as np
from trlda_b200 import capi
from trlda_b200.synth import make_corpus
K, V, B = 1000, 100000, int(os.environ.get('B', 8192))
steps = int(os.environ.get('STEPS', 2))
m = capi.Model('online', V, K, 1000000, .1, .2, precision=os.environ.get('PREC', 'mixed'))
for s in range(steps):
    docs = capi.CSR(*make_corpus(B, V, K, .1, .2, seed=1003 + s))
    m.update_parameters(docs, max_iter_tr=10, max_iter_inference=20, kappa=.7, tau=100.)
m.synchronize()
print('steps', steps, flush=True)
m.close()
