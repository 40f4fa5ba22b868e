"""Fine-grained phase stamps of the cluster GRU phases (step_mode 3); needs libg4r.so built with -DG4R_CF_FINE.
Rows s < 500 hold the normal stamps of step s, rows s + 500 the cluster-phase stamps of the same step."""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import bench
from gru4rec_b200 import _lib
import gru4rec as g4
wl = bench.WORKLOADS['cfg2']                  # the headline workload of bench.py
mk = dict(wl['model'])
K = 1000
cfg = _lib.make_config(wl['n_items'], mk, sample_store=bench.SAMPLE_STORE, max_resident_steps=K + 8, step_mode=3)
eng = _lib.Engine(cfg)
gru = g4.GRU4Rec(**mk); gru.n_items = wl['n_items']
for name, w in gru._init_host_weights().items():
    eng.set(name, w)
items, offset, order, supports = bench.build_workload(wl, 3 * K)
P = supports.astype(np.float64) ** mk['sample_alpha']; P = P.cumsum() / P.sum(); P[-1] = 1
eng.set_sampling_cdf(P.astype(np.float32)); eng.generate_samples()
sched = _lib.Schedule(items, offset, order, mk['batch_size'], mk['n_sample'], mode=0)
eng.upload_steps(sched, 0, K); eng.run_uploaded(K, False)
eng.persistent_stamps(True)
eng.upload_steps(sched, K, K); c, ms = eng.run_uploaded(K, True)
st = eng.persistent_stamps(True, K).astype(np.int64)
print('fast windows', eng.fast_windows(), 'ms/step', ms / K)
n = st[10:490]; f = st[510:990]
seg = [('b1 end(15) -> bwd entry', n[:, 15], f[:, 0]), ('wait b1_done', f[:, 0], f[:, 1]), ('dy + elementwise', f[:, 1], f[:, 2]), ('partials + push', f[:, 2], f[:, 3]),
       ('cluster barrier 1', f[:, 3], f[:, 4]), ('da_r + release', f[:, 4], f[:, 5]), ('dense main', f[:, 5], f[:, 6]), ('bias + arrive', f[:, 6], f[:, 7]),
       ('f1: stage H', f[:, 7], f[:, 8]), ('f1: dot', f[:, 8], f[:, 9]), ('f1: wait in_done', f[:, 9], f[:, 10]), ('f1: epilogue', f[:, 10], f[:, 11]),
       ('f1: cluster wait 2', f[:, 11], f[:, 12]), ('f1: pushes', f[:, 12], f[:, 13]), ('f1: cluster barrier 3', f[:, 13], f[:, 14]), ('f2', f[:, 14], f[:, 15]),
       ('f2 end -> release(8)', f[:, 15], n[:, 8])]
for name, a, b in seg:
    d = (b - a) / 1000.0
    print('%-28s mean %6.2f us  p50 %6.2f' % (name, d.mean(), np.median(d)))
