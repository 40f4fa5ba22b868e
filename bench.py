#!/usr/bin/env python
"""bench.py -- mini-batches/sec of the GRU4Rec session-parallel training step on synthetic sessions of the BASELINE.json shapes.

Contract: python bench.py --gpus N --steps K --warmup W   (torchrun for N>1) prints ONE JSON line.
  value   : whole-job mini-batches/s, device-timed (CUDA events on the library's stream, max over ranks), with the schedule
            window, the column plans, the sample store and the parameters resident in HBM when the timed region starts
  e2e     : the same metric through the reference-facing call g4r_train_steps (host schedule arrays -> H2D -> column plans ->
            steps -> D2H costs), wall clock between barriers
  roofline: the kernel that ran in the timed region: whole-step algorithmic bytes (SURVEY 8d) / measured step time vs the
            measured HBM peak; the per-phase `k_lossgrad` figure is kept as a sub-field
  cpu_baseline: the NumPy oracle (port of the reference; Theano is not installable) on the host cores, bounded sample
--impl reference : times that CPU port alone (rank 0 only), same metric / config.
--workload cfg1|cfg2|cfg2x|cfg3|cfg4 : the other BASELINE.json configurations (default cfg2 = the headline)
--dump-outputs DIR : after the timed steps, DIR/<name>.npy holds what they computed (see dump_outputs); the inputs are seeded,
            so two builds run with the same arguments can be compared output for output
"""
import argparse
import json
import os
import sys
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

# BASELINE.json configs; shapes from SURVEY.md section 8(d).  cfg2 = configs[1] is the headline (param_samples/rsc15_bpr-max.py).
WORKLOADS = {
    'cfg1': dict(name='synthetic_xe_gru100_b32_1k_items', n_items=1000, params='run.py -ps loss=cross-entropy,final_act=softmax,layers=100,batch_size=32',
                 model=dict(layers=[100], loss='cross-entropy', final_act='softmax', batch_size=32, n_sample=2048), published=1380.0,
                 published_src='XE, B=32, L=100 without dropout/momentum, A30 (img/training_time_xe_batch_size.png)'),
    'cfg2': dict(name='rsc15_bprmax_gru100_b32_ns2048', n_items=37483, params='param_samples/rsc15_bpr-max.py',
                 model=dict(layers=[100], loss='bpr-max', final_act='elu-0.5', hidden_act='tanh', batch_size=32, dropout_p_embed=0.0,
                            dropout_p_hidden=0.0, learning_rate=0.2, momentum=0.3, sample_alpha=0.0, n_sample=2048, bpreg=1.0,
                            constrained_embedding=False), published=1235.0,
                 published_src='BPR-max, B=32, GRU(100), n_sample=2048, with momentum, A30 (img/training_time_bprmax_batch_size.png, README.md:302)'),
    'cfg2x': dict(name='rsc15_xe_shared_gru100_b32_ns2048', n_items=37483, params='paramfiles/rsc15_xe_shared_100_best.py',
                  model=dict(layers=[100], loss='cross-entropy', final_act='softmax', constrained_embedding=True, batch_size=32,
                             dropout_p_hidden=0.4, learning_rate=0.2, momentum=0.2, n_sample=2048, sample_alpha=0.5, bpreg=0.0, logq=1.0), published=1120.0,
                  published_src='XE, B=32, L=100 with dropout/momentum, A30 (img/training_time_xe_batch_size.png)'),
    'cfg3': dict(name='rees46_xe_shared_gru512_b240_ns2048', n_items=172000, params='paramfiles/rees46_xe_shared_best.py',
                 model=dict(layers=[512], loss='cross-entropy', final_act='softmax', constrained_embedding=True, batch_size=240,
                            dropout_p_embed=0.45, learning_rate=0.065, momentum=0.0, n_sample=2048, sample_alpha=0.5, bpreg=0.0, logq=1.0), published=545.0,
                 published_src='XE, B=256, L=500 with dropout, A30 (img/training_time_xe_batch_size.png; nearest published shape)'),
    'cfg4': dict(name='retailrocket_bprmax_shared_3xgru100_b80_ns2048', n_items=37000, params='paramfiles/retailrocket_bprmax_shared_best.py with layers=100/100/100',
                 model=dict(layers=[100, 100, 100], loss='bpr-max', final_act='elu-0.5', constrained_embedding=True, batch_size=80,
                            dropout_p_embed=0.5, dropout_p_hidden=0.05, learning_rate=0.05, momentum=0.4, n_sample=2048, sample_alpha=0.4, bpreg=1.95), published=1026.0,
                 published_src='RetailRocket BPR-max shared, 1xGRU(224), B=80, A30 (README.md:153-169; nearest published shape)'),
}
SAMPLE_STORE = 10000000
DUMP_ROWS = 16384                   # item-table rows kept by --dump-outputs: under 64 MB in all at every workload


def dump_outputs(eng, names, costs, n_items, out_dir):
    """What the timed steps computed, as float32 DIR/<name>.npy: `cost` (one per timed mini-batch, the last is the last step's)
    and, as they stand after the last step, every parameter and the GRU hidden state H<i>.  Tables with one row per item and more
    than DUMP_ROWS items are cut to a fixed seeded sample of rows, whose item ids `item_rows` holds."""
    rows = np.sort(np.random.RandomState(0).choice(n_items, DUMP_ROWS, replace=False)) if n_items > DUMP_ROWS else None
    out = {'cost': np.asarray(costs, dtype=np.float32)}
    for name in names:
        a = eng.get(name)
        out[name] = a[rows] if rows is not None and a.shape[0] == n_items else a
    if rows is not None:
        out['item_rows'] = rows.astype(np.float32)
    assert sum(a.nbytes for a in out.values()) <= 64 << 20, 'dump larger than 64 MB'
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def algo_bytes_step(mk):
    """SURVEY.md section 8(d): algorithmic HBM bytes of one mini-batch (fp32)."""
    B, S, layers = mk['batch_size'], mk['n_sample'], mk['layers']
    L, L0, N = layers[-1], layers[0], mk['batch_size'] + mk['n_sample']
    T = 4 + (2 if mk.get('momentum', 0.0) > 0 else 0)
    shared, emb = bool(mk.get('constrained_embedding')), int(mk.get('embedding', 0) or 0)
    if shared:
        rows_in, rows_out = 0, B + N
    elif emb:
        rows_in, rows_out = B * emb, N
    else:
        rows_in, rows_out = B * 3 * L0, N
    dense = 0
    for i, Li in enumerate(layers):
        in_l = (L if shared else emb) if i == 0 else layers[i - 1]
        has_wx = i > 0 or shared or emb
        dense += 4 * ((in_l * 3 * Li if has_wx else 0) + Li * Li + 2 * Li * Li + 3 * Li)
    idx = 8 * B + 8 * S + B + (4 * N if mk.get('logq', 0) else 0)
    return T * 4 * (rows_in + rows_out * L + N) + T * dense + 8 * sum(B * Li for Li in layers) + idx


def algo_bytes_lossgrad(N, L, mom=True):
    """sparse Adagrad(+momentum) of the N gathered Wy rows + By: (param, acc[, vel]) read + write."""
    T = 6 if mom else 4
    return T * 4 * (N * L + N)


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled through NVML every ~2 ms for the whole measurement (a 20-step timed region lasts
    under a millisecond, so the record covers warm-up + timed region + e2e arm; `samples_timed` counts those inside the
    marked timed regions)."""

    def __init__(self, gpu_index=0):
        threading.Thread.__init__(self, daemon=True)
        self.rows, self.stop_flag, self.gpu_index, self.timed = [], False, gpu_index, False
        self.err, self.source = None, 'NVML, 2 ms period, whole measurement'

    def run(self):
        names = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu_index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception as e:            # no usable NVML binding: poll nvidia-smi instead (slower period, same fields)
            self.err = repr(e)
            self.source = 'nvidia-smi, ~30 ms period, whole measurement'
            q = ['nvidia-smi', '-i', str(self.gpu_index), '--query-gpu=clocks.sm,clocks.max.sm,clocks_throttle_reasons.active',
                 '--format=csv,noheader,nounits']
            while not self.stop_flag:
                try:
                    f = subprocess.run(q, capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                    rs = int(f[2].strip(), 16)
                    self.rows.append((float(f[0]), float(f[1]), [k for k, v in names.items() if rs & v], self.timed))
                except Exception as e2:
                    self.err = repr(e2)
                time.sleep(0.02)
            return
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((sm, mx, [k for k, v in names.items() if rs & v], self.timed))
            except Exception as e:
                self.err = repr(e)
            time.sleep(0.002)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0, 'error': self.err}
        sm = [r[0] for r in self.rows]
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(self.rows[0][1]), 'reasons': reasons, 'samples': len(sm),
                'samples_timed': int(sum(1 for r in self.rows if r[3])), 'source': self.source}


def peak_tensor():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['bf16_tflops_sustained']), 'measured sustained bf16 (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 2250.0, 'nominal dense bf16 (B200_PROFILING.md)'


def peak_hbm():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(wl):
    """DRAM bytes per mini-batch of the dominant kernel from the committed ncu --set full capture (profiles/ncu_traffic.json)."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        d = json.load(open(p))
        e = d.get(wl)
        if e:
            return e['dram_bytes_per_step'], e['source'], e.get('kernel')
    except Exception:
        pass
    return None, None, None


def build_workload(wl, n_steps_needed, seed=0):
    from gru4rec_b200.synth import make_session_arrays
    B = wl['model']['batch_size']
    n_events = max(int((n_steps_needed + 64) * B * 1.6) + 20000, 4 * wl['n_items'])
    return make_session_arrays(wl['n_items'], n_events, seed=seed)


def bench_config(wl, world, extra=None):
    """`config` of the JSON line: identical keys (and values, except the run-specific ones) in both arms."""
    mk = wl['model']
    c = {'workload': wl['name'], 'n_items': wl['n_items'], 'global_batch': mk['batch_size'] * world, 'n_sample': mk['n_sample'],
         'layers': mk['layers'], 'params': wl['params'], 'loss': mk['loss'], 'constrained_embedding': bool(mk.get('constrained_embedding', False))}
    if extra:
        c.update(extra)
    return c


def oracle_steps_per_sec(wl, items, offset, order, supports, n_warm, n_steps, budget_s):
    """The NumPy restatement of the reference step (oracle/) on the host cores."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import gru4rec_oracle as orc
    mk = dict(wl['model'])
    m = orc.OracleGRU4Rec(**mk)
    m.init(wl['n_items'])
    P = orc.sampling_cdf(supports, mk.get('sample_alpha', 0.75)).astype(np.float32)
    if mk.get('logq', 0):
        m.P0 = np.maximum(supports, 1).astype(np.float32)
    B = mk['batch_size']
    # literal schedule restatement on a prefix of the data (the schedule itself is outside the timed step)
    n_sess = int(np.searchsorted(offset, (n_warm + n_steps + 8) * B * 3))
    n_sess = max(min(n_sess, len(offset) - 1), B + 1)
    steps = orc.build_train_schedule(items, offset[:n_sess + 1], order[:n_sess], B, mk['n_sample'])
    steps = steps[:n_warm + n_steps]
    # the negative samples of every step are drawn before the clock starts (in the reference they come from the device store)
    rs = np.random.RandomState(1)
    smps = [orc.searchsorted_k2(P, rs.rand(mk['n_sample']).astype(np.float32)) for _ in steps]
    t_start = time.time()
    done = 0
    t0 = None
    for k, st in enumerate(steps):
        if k == n_warm:
            t0 = time.time()
        m.train_step(st['X'], st['Y'], st['R'], samples=smps[k], slots=st['slots'])
        if k >= n_warm:
            done += 1
            if time.time() - t_start > budget_s:
                break
    dt = time.time() - t0
    try:
        from threadpoolctl import threadpool_info
        cores = max([p.get('num_threads', 1) for p in threadpool_info()] + [1])
    except Exception:
        cores = os.cpu_count()
    return done / dt, done, cores


def run_reference(args, rank, world):
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    n = args.steps
    items, offset, order, supports = build_workload(wl, min(n, 4000) + args.warmup)
    v, done, cores = oracle_steps_per_sec(wl, items, offset, order, supports, args.warmup, n, budget_s=150.0)
    out = {
        'metric': 'mini-batches/sec', 'value': v, 'unit': 'mb/s', 'n_gpus': args.gpus, 'steps': done, 'warmup': args.warmup,
        'ms_per_step': 1000.0 / v, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': v / wl['published'], 'dtype': 'f32', 'data': 'synthetic',
        'impl': 'reference',
        'config': bench_config(wl, world, {'note': 'reference CPU path = NumPy restatement of gru4rec.py (oracle/); Theano is not installable offline; '
                                                     'one process on the host cores whatever --gpus says'}),
        'cpu_baseline': {'value': v, 'unit': 'mb/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d timed mini-batches of the same workload after %d warm-up (time-bounded)' % (done, args.warmup)},
        'e2e': {'value': v, 'unit': 'mb/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=4000)
    ap.add_argument('--warmup', type=int, default=200)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--replicated', action='store_true', help='N>1: replicated tables + NCCL exchange (round-1 path) instead of row sharding')
    ap.add_argument('--step-mode', type=int, default=2, help='0 per-phase kernels (CUDA graph), 1 persistent kernel, 2 role-specialised persistent kernel (default), 3 = 2 with the GRU phases on one thread-block cluster')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the costs of the timed steps and the parameters after the last one to DIR/<name>.npy (one GPU)')
    args = ap.parse_args()
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (world > 1 or args.impl != 'b200'):
        ap.error('--dump-outputs needs the b200 path on one GPU')
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    import torch
    from gru4rec_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    wl = WORKLOADS[args.workload]
    K, W = args.steps, max(args.warmup, 3)
    mk = dict(wl['model'])
    B = mk['batch_size']
    N = B + mk['n_sample']
    gen_rows = SAMPLE_STORE // mk['n_sample']
    cfg = _lib.make_config(wl['n_items'], mk, sample_store=SAMPLE_STORE, eval_lanes=0,
                           max_resident_steps=min(max(K, W), gen_rows) + 8, step_mode=args.step_mode, world_size=world, rank=rank,
                           replicated=args.replicated)
    eng = _lib.Engine(cfg, device=local_rank)
    if world > 1:
        try:
            eng.init_multi_gpu(dist)
        except NotImplementedError as e:
            # e.g. BASELINE configs[4] (Rees46 x 8 GPUs): constrained-embedding models have no multi-GPU training path (DESIGN.md section 6)
            if rank == 0:
                print(json.dumps({'metric': 'mini-batches/sec', 'n_gpus': world, 'config': bench_config(wl, world), 'unavailable': str(e)}))
            eng.close()
            dist.barrier()
            dist.destroy_process_group()
            return
    sharded = world > 1 and eng.sharded()
    # parameters: the reference's initialisation (gru4rec.py:254-294); data: synthetic sessions of the workload's shape, disjoint per rank
    import gru4rec as g4
    gru = g4.GRU4Rec(**mk)
    gru.n_items = wl['n_items']
    host = gru._init_host_weights()
    for name, w in host.items():
        eng.set(name, w)
    need_steps = 2 * K + W + min(K, 512) + 64         # warm-up, timed region, e2e arm, the per-kernel profiling / stamp passes
    grow = 1.0
    while True:                                       # synthetic sessions until the schedule covers every arm
        items, offset, order, supports = build_workload(wl, int(need_steps * grow), seed=rank)
        sched = _lib.Schedule(items, offset, order, B, mk['n_sample'], mode=0)
        if sched.n_steps >= need_steps or grow > 8:
            break
        grow *= 1.5
    assert sched.n_steps >= need_steps, 'synthetic workload too small'
    P = supports.astype(np.float64) ** mk.get('sample_alpha', 0.75)
    P = P.cumsum() / P.sum(); P[-1] = 1
    eng.set_sampling_cdf(P.astype(np.float32))
    if mk.get('logq', 0):
        eng.set_logq_support(np.maximum(supports, 1).astype(np.float32))
    eng.generate_samples()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    clocks = ClockSampler(local_rank); clocks.start()
    h2d = B * (4 + 4 + 4 + 1) + 12
    first = W + K
    cap = int(cfg.max_resident_steps)
    if sharded:
        cap = min(cap, 256)                       # MG_CAP: lock steps per window of the sharded kernel
    device_timed = world == 1 or sharded
    if device_timed:
        # ---- device-resident arm: warm-up, then K timed steps from uploaded windows.  A window never crosses a refill of the
        # negative-sample store (4882 mini-batches at n_sample = 2048): uploads, column plans (and, sharded, the plan exchange)
        # and refills happen between the timed windows; `value` sums the CUDA-event times of the windows, max over ranks (the
        # e2e arm below times everything, refills included).
        eng.reset_hidden()
        done = 0
        while done < W:
            n = min(W - done, cap)
            eng.upload_steps(sched, done, n); eng.run_uploaded(n, want_cost=False); done += n
        gen_len = eng.sample_store_rows()
        launches0 = eng.kernel_launches()
        barrier()
        clocks.timed = True
        t0 = time.time()
        dev_ms, done, cost_parts, plan_s, n_win = 0.0, 0, [], 0.0, 0
        while done < K:
            if eng.get_sample_pointer() >= gen_len:
                eng.generate_samples()
            n = min(K - done, gen_len - eng.get_sample_pointer(), cap)
            torch.cuda.synchronize(); tp = time.time()
            eng.upload_steps(sched, W + done, n)
            torch.cuda.synchronize(); plan_s += time.time() - tp; n_win += 1
            if dist is not None:
                barrier()                        # ranks enter every timed window together (the lock step is what is measured)
            c, ms = eng.run_uploaded(n, want_cost=True)
            dev_ms += ms; done += n; cost_parts.append(c)
        barrier()
        clocks.timed = False
        wall = time.time() - t0
        costs = np.concatenate(cost_parts)
        launches = eng.kernel_launches() - launches0
        if args.dump_outputs:                    # before the e2e arm trains on
            dump_outputs(eng, sorted(host) + ['H%d' % i for i in range(len(mk['layers']))], costs, wl['n_items'], args.dump_outputs)
        if dist is not None:
            t = torch.tensor([dev_ms], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); dev_ms = float(t.item())
        value = world * K / (dev_ms / 1000.0)
        # ---- end-to-end arm: host schedule arrays in, costs out, every window (H2D + plans + steps + D2H inside the timing)
        if dist is not None:
            eng.train_steps(sched, first + K, 4)     # first use of this entry point (its step-count agreement is a fresh NCCL collective)
        barrier()
        clocks.timed = True
        t0 = time.time()
        c2 = eng.train_steps(sched, first, K)
        barrier()
        clocks.timed = False
        e2e_s = time.time() - t0
        assert np.isfinite(c2).all()
        if dist is not None:
            t = torch.tensor([e2e_s], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
    else:
        # ---- replicated NCCL path (shapes the row-sharded kernel does not cover): one merged update per mini-batch inside
        # g4r_train_steps.  The call takes HOST schedule arrays, so this IS the end-to-end path; barrier + synchronize on both
        # sides, max over ranks.
        eng.reset_hidden()
        eng.train_steps(sched, 0, W)
        launches0 = eng.kernel_launches()
        barrier()
        clocks.timed = True
        t0 = time.time()
        costs = eng.train_steps(sched, W, K)
        barrier()
        clocks.timed = False
        wall = time.time() - t0
        launches = eng.kernel_launches() - launches0
        t = torch.tensor([wall], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); wall = float(t.item())
        dev_ms = wall * 1000.0
        value = world * K / wall
        e2e_s = wall
    assert np.isfinite(costs).all(), 'non-finite cost in the timed region'
    e2e_value = world * K / e2e_s
    fastw = list(eng.fast_windows())
    # ---- per-kernel view from CUDA events around every launch of one more pass over a short window (single GPU)
    prof_n = min(K, 512)
    prof = None
    if world == 1:
        if eng.get_sample_pointer() + prof_n > eng.sample_store_rows():
            eng.generate_samples()
        eng.upload_steps(sched, first + K, prof_n)
        prof = eng.profile_uploaded()
    peak, peak_src = peak_hbm()
    step_bytes = algo_bytes_step(mk)
    lg_bytes = algo_bytes_lossgrad(N, mk['layers'][-1], mk.get('momentum', 0.0) > 0)
    fast_phase = None
    if world == 1 and int(cfg.step_mode) in (2, 3) and fastw[0] > 0:
        # the update phase INSIDE the production kernel k_fast, from %globaltimer stamps of CTA 0 (slot 2 = row statistics
        # ready, slot 14 = chunk's rows updated): loss gradient + dSy + partial dL/dh + sparse update of the chunk's rows
        eng.persistent_stamps(True)
        if eng.get_sample_pointer() + prof_n > eng.sample_store_rows():
            eng.generate_samples()
        eng.upload_steps(sched, first + K, prof_n)
        eng.run_uploaded(prof_n, want_cost=False)
        st = eng.persistent_stamps(False, prof_n).astype(np.int64)
        lo = min(8, prof_n - 1)
        seg_us = float(np.mean((st[lo:, 14] - st[lo:, 2]) / 1000.0))
        fast_phase = {'us': seg_us, 'achieved_GBs': lg_bytes / (seg_us * 1e-6) / 1e9, 'frac': lg_bytes / (seg_us * 1e-6) / 1e9 / peak,
                      'algorithmic_bytes': lg_bytes,
                      'note': 'k_fast: statistics-ready -> rows-updated segment of a chunk CTA (globaltimer), sparse Adagrad/momentum update of the Wy/By rows'}
    clocks.stop_flag = True
    clocks.join(2.0)
    per_phase = None
    if prof is not None:
        lg_ms, lg_n = prof['lossgrad_update']
        per_phase = {'kernel': 'k_lossgrad in per-phase mode (step_mode 0; NOT the kernel of the timed region)',
                     'achieved': lg_bytes / (lg_ms / lg_n * 1e-3) / 1e9, 'frac': lg_bytes / (lg_ms / lg_n * 1e-3) / 1e9 / peak,
                     'algorithmic_bytes_per_launch': lg_bytes, 'us_per_launch': lg_ms / lg_n * 1000.0,
                     'phase_us': {k: round(v[0] / v[1] * 1000.0, 3) for k, v in prof.items()}}
    if sharded:
        kernel = 'k_fast_mg (row-sharded role-specialised persistent kernel: peer TMA row fetch, in-kernel NVLink exchange, owner-side update)'
    elif world > 1:
        kernel = 'per-phase kernels + NCCL (replicated path)'
    elif fastw[0] > 0 and fastw[1] == 0:
        kernel = 'k_fast_t (role-specialised persistent kernel, one launch per window: the whole step)'
    else:
        kernel = 'k_persistent (generic persistent kernel, one launch per window: the whole step)' if int(cfg.step_mode) >= 1 else 'per-phase kernels (CUDA graph)'
    step_s = dev_ms / 1000.0 / K                      # lock-step time (every rank moves step_bytes per lock step)
    achieved = step_bytes / step_s / 1e9
    tensor = None
    if world == 1 and eng.uses_tensor_cores():
        # the step ran on the tcgen05 path (g4r_tcstep.cuh): the contractions bound it, not the row traffic.  fp32-equivalent
        # FLOPs of the eight products: gates, candidate, scores, dSy, dL/dh, d(H*r), dL/d(input), dense gradients
        L = mk['layers'][-1]
        macs = 16.0 * B * L * L + 3.0 * B * N * L
        tf_peak, tf_src = peak_tensor()
        tensor = {'flops_per_step': 2.0 * macs, 'achieved': 2.0 * macs / step_s / 1e12, 'peak': tf_peak / 6.0, 'unit': 'TFLOP/s',
                  'peak_source': tf_src + '; bf16 dense / 2 (TF32 rate) / 3 (3xTF32: three tensor-core products per fp32 product)'}
        tensor['frac'] = tensor['achieved'] / tensor['peak']
        kernel = ('k_ts_gemm (tcgen05 kind::tf32, 3xTF32, 128x256 tiles, K split over thread-block clusters; 8 products per mini-batch on 3 streams '
                  '+ operand-preparation / loss / sparse-update kernels; one CUDA graph per 16 mini-batches)')
    traffic, traffic_src, traffic_kernel = ncu_traffic(args.workload) if world == 1 else (None, None, None)
    if world == 1:
        par = 'dp1'
    elif sharded:
        par = ('dp%d: item tables row-sharded (row i on rank i %% %d), parameter rows fetched from their owners by TMA over NVLink, gradient rows stored '
               'into the owners\' inboxes, owner-side merged update, dense GRU gradients pushed to all peers and summed in rank order -- all inside the '
               'persistent kernel; NCCL only for the per-window all-gather of the sorted column lists' % (world, world))
    else:
        par = 'dp%d: replicated parameters, NCCL all-gather of row gradients + all-reduce of dense gradients per mini-batch, identical merged update on every rank' % world
    out = {
        'metric': 'mini-batches/sec', 'value': value, 'unit': 'mb/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': dev_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': value / wl['published'],
        'dtype': 'f32', 'data': 'synthetic',
        'config': bench_config(wl, world, {
            'parallelism': par,
            'l2': 'inputs larger than L2 at the headline shape: item tables + Adagrad/momentum state = 180 MB, rows touched change every step (no flush '
                  'between steps; ncu shows the sampled rows staying L2-resident in steady state, see roofline.traffic)',
            'step_mode': int(cfg.step_mode), 'fast_windows': fastw, 'upload_and_plan_ms_per_window': (plan_s / max(n_win, 1) * 1000.0) if device_timed else None, 'events_per_sec': value * B, 'timing': 'cuda events, max over ranks' if device_timed else 'wall clock between barriers, max over ranks',
            'vs_baseline_source': 'BASELINE.md: ~%g mb/s published by the reference: %s' % (wl['published'], wl['published_src'])}),
        'e2e': {'value': e2e_value, 'unit': 'mb/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4},
        'gpu_launches': int(launches),
        'clocks': clocks.summary(),
        'roofline': {'bound': 'tensor' if tensor else 'hbm', 'kernel': kernel,
                     'achieved': tensor['achieved'] if tensor else achieved, 'peak': tensor['peak'] if tensor else peak,
                     'unit': 'TFLOP/s' if tensor else 'GB/s', 'frac': tensor['frac'] if tensor else achieved / peak,
                     'tensor': tensor, 'hbm': {'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak},
                     # DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum) on the same footing as algorithmic_bytes_per_launch:
                     # the committed capture's bytes per mini-batch x the K mini-batches of the timed region
                     'traffic': (traffic * K) if traffic is not None else None, 'traffic_per_step': traffic,
                     'traffic_source': traffic_src, 'traffic_kernel': traffic_kernel,
                     'peak_source': peak_src, 'algorithmic_bytes_per_launch': step_bytes * K, 'algorithmic_bytes_per_step': step_bytes,
                     'us_per_step': step_s * 1e6,
                     'note': ('tensor-core path: a chain of 7 dependent split-K products per mini-batch (each ~4 us of tcgen05 issue + ~12 us of launch, '
                              'operand fetch, L2 exchange and epilogue latency); the fraction is against the 3xTF32-equivalent tensor peak') if tensor else
                             ('latency-bound: ~15 dependent phases per mini-batch over an L2-resident working set (SURVEY fact 5); the HBM roofline is the '
                              'contract\'s denominator, not the binding limit'),
                     'k_fast_update_phase': fast_phase, 'per_phase_mode': per_phase},
        'wall_s_timed_region': wall,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, done, cores = oracle_steps_per_sec(wl, items, offset, order, supports, 5, 2000, budget_s=20.0)
        out['cpu_baseline'] = {'value': v, 'unit': 'mb/s', 'cores': cores, 'kind': 'port',
                               'sample': '%d mini-batches of the same workload through the NumPy oracle (~20 s)' % done}
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
