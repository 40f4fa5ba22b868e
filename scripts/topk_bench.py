"""Per-call cost of serving top-k recommendations at the RSC15 and Rees46 shapes (random weights):
  (a) GRU4Rec.recommend_next_batch                      -- device scoring + top-k, only [batch x k] comes back
  (b) GRU4Rec.predict_next_batch + np.argpartition/sort -- the full items x batch DataFrame, selection on the host
  (c) Engine.predict + the same host selection           -- the full score matrix without the DataFrame
Call times are host wall-clock around calls that end in a device synchronise.  Kernel times are the CUDA durations of the
scoring kernels (k_topk_score + k_topk_merge against k_eval_score<true> + k_predict_act) taken with torch.profiler over the same
calls; the device span of a whole call (staging, GRU forward, scoring, copy back) is timed with CUDA events on the library's
stream.  Usage: python scripts/topk_bench.py [--iters N] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import numpy as np
import pandas as pd
import torch
import gru4rec as g4

WORKLOADS = [
    dict(name='rsc15_b100_k20', n_items=37483, mk=dict(layers=[100]), batch=100, k=20),
    dict(name='rsc15_b512_k20', n_items=37483, mk=dict(layers=[100]), batch=512, k=20),
    dict(name='rees46_b240_k20', n_items=172000, mk=dict(layers=[512], constrained_embedding=True), batch=240, k=20),
    dict(name='rees46_b240_k100', n_items=172000, mk=dict(layers=[512], constrained_embedding=True), batch=240, k=100),
]
TOPK_KERNELS = ('k_topk_score', 'k_topk_merge')
PREDICT_KERNELS = ('k_eval_score', 'k_predict_act')


def host_topk(S, k, axis):
    """top-k indices of every row (axis=1) / column (axis=0) of S, sorted by score descending"""
    part = np.argpartition(-S, k - 1, axis=axis).take(np.arange(k), axis=axis)
    vals = np.take_along_axis(S, part, axis=axis)
    order = np.argsort(-vals, axis=axis, kind='stable')
    return np.take_along_axis(part, order, axis=axis)


def model(w):
    mk = dict(loss='bpr-max', final_act='elu-0.5', batch_size=32, n_sample=2048, **w['mk'])
    gru = g4.GRU4Rec(**mk)
    gru.n_items = w['n_items']
    gru.itemidmap = pd.Series(data=np.arange(gru.n_items), index=np.arange(gru.n_items) * 7 + 1000, name='ItemIdx')
    gru._host = gru._init_host_weights()
    gru.error_during_train = False
    gru.predict = None
    return gru


def timed(fn, iters):
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter(); fn(); ts.append((time.perf_counter() - t0) * 1e3)
    return dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), mean_ms=float(np.mean(ts)))


def kernel_ms(fn, iters, names):
    """mean CUDA time per call of the kernels whose names contain one of `names`"""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for n in names:
            if n in ev.name:
                per[n] = per.get(n, 0.0) + getattr(ev, 'device_time', getattr(ev, 'cuda_time', 0.0)) / 1e3
    per = {k: v / iters for k, v in per.items()}
    return sum(per.values()), per


def event_ms(eng, fn, iters):
    st = torch.cuda.ExternalStream(eng.stream())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(iters):
        a.record(st); fn(); b.record(st); b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=30)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True).stdout.strip()
    res = dict(gpu=gpu, iters=args.iters, workloads=[])
    rs = np.random.RandomState(0)
    for w in WORKLOADS:
        gru = model(w)
        B, k = w['batch'], w['k']
        ids = gru.itemidmap.index.values
        sess = np.arange(B)
        inp = lambda: ids[rs.randint(0, len(ids), B)]
        arm_a = lambda: gru.recommend_next_batch(sess, inp(), k=k, batch=B)
        arm_b = lambda: host_topk(gru.predict_next_batch(sess, inp(), batch=B).values, k, axis=0)
        arm_a(); arm_b()
        eng = gru._engine
        arm_c = lambda: host_topk(eng.predict(gru.itemidmap[inp()].values), k, axis=1)
        arm_c()
        r = dict(name=w['name'], n_items=w['n_items'], layers=w['mk']['layers'], batch=B, k=k,
                 constrained_embedding=bool(w['mk'].get('constrained_embedding')))
        r['a_recommend_next_batch'] = timed(arm_a, args.iters)
        r['b_predict_next_batch_host_select'] = timed(arm_b, args.iters)
        r['c_engine_predict_host_select'] = timed(arm_c, args.iters)
        X = gru.itemidmap[inp()].values
        r['kernel_ms_topk'], r['kernels_topk'] = kernel_ms(lambda: eng.predict_topk(X, k), args.iters, TOPK_KERNELS)
        r['kernel_ms_predict'], r['kernels_predict'] = kernel_ms(lambda: eng.predict(X), args.iters, PREDICT_KERNELS)
        r['kernel_ratio_topk_over_predict'] = r['kernel_ms_topk'] / r['kernel_ms_predict']
        r['device_call_ms_topk'] = event_ms(eng, lambda: eng.predict_topk(X, k), args.iters)
        r['device_call_ms_predict'] = event_ms(eng, lambda: eng.predict(X), args.iters)
        res['workloads'].append(r)
        print(json.dumps(r), flush=True)
        eng.close()
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=gpu)))


if __name__ == '__main__':
    main()
