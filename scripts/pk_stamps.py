"""Phase breakdown of the persistent kernel from %globaltimer stamps (headline workload)."""
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
cfg = _lib.make_config(wl['n_items'], mk, sample_store=bench.SAMPLE_STORE, max_resident_steps=K + 8, step_mode=int(sys.argv[1]) if len(sys.argv) > 1 else 1)
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
if cfg.step_mode >= 2:
    print('fast windows', eng.fast_windows())
    names = [('wait h + stage', 0, 1), (' targets+scores', 1, 9), (' partial stats', 9, 10), (' B2 + parallel combine', 10, 2), (' RS load + cost', 2, 11), (' g + dby', 11, 12), (' dSy + part', 12, 13), (' sparse update', 13, 14), (' B3', 14, 3),
             ('b1 (+release)', 3, 15), ('rows wait + prefetch issue', 15, 4), ('b2 + grp', 4, 5), ('dense + grp', 5, 6), ('f1 + grp', 6, 7), ('f2', 7, 8)]
    if cfg.step_mode == 3:   # GRU phases on one thread-block cluster
        names[-4:] = [('backward -> dvec', 4, 5), ('dense (resident)', 5, 6), ('f1 (+in_done, barriers)', 6, 7), ('f2', 7, 8)]
    else:                    # step_mode 2: the GRU role reuses the column role's fine slots 1, 4, 9, 10, 11, 12
        names = [('wait h .. B2 + combine', 0, 2), (' RS, g, dby, dSy, part', 2, 13),
                 (' row update (in B3)', 13, 14), (' B3 wait', 14, 3), ('b1 (+release)', 3, 15),
                 ('dense stage, lanes, b1_done wait, b2', 15, 5), ('rows wait', 5, 4),
                 ('prefetch issue', 4, 10), ('dense ph0 + stage H', 10, 1),
                 ('B2 grp wait', 1, 9), ('da_r + Wr update', 9, 6),
                 ('f1 product', 6, 11), ('f1 in_done wait', 11, 12), ('f1 epilogue + grp', 12, 7), ('f2', 7, 8)]
    st = st[:-1]
else:
  names = [('gru_rz(f1)', 0, 6), ('gru_h(f2)', 6, 1), ('score', 1, 2), ('stats', 2, 3), ('lossgrad', 3, 4), ('b1', 4, 7), ('b2', 7, 8), ('dense+sparse_in', 8, 5)]
print('ms/step', ms / K)
for n, a, b in names:
    d = (st[:, b] - st[:, a]) / 1000.0
    print('%-38s mean %.2f us  p50 %.2f' % (n, d[10:].mean(), np.median(d[10:])))
print('step total', ((st[1:, 0] - st[:-1, 0]) / 1000.0)[10:].mean())
