"""-m gpu: 2-GPU synchronous data-parallel step vs the oracle on the merged mini-batch (needs >= 2 devices)."""
import os
import subprocess
import sys
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(world, port):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world), '--master-addr', '127.0.0.1', '--master-port', str(port),
           os.path.join(ROOT, 'tests', 'mg_worker.py')]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    return out.stdout


def test_two_gpu_parity():
    """row-sharded in-kernel exchange (3 cases) + replicated NCCL path (2 cases) vs the oracle on the merged mini-batch"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    out = _run(2, 29533)
    assert out.count('multi-gpu parity ok') == 5, out[-2000:]
    assert out.count('sharded') >= 3


def test_all_gpu_parity():
    """the same on every GPU of the box (8 on an HGX node)"""
    import torch
    n = torch.cuda.device_count()
    if n < 4:
        pytest.skip('needs >= 4 GPUs')
    out = _run(n, 29534)
    assert out.count('multi-gpu parity ok') >= 4, out[-2000:]


def _metric_lines(text):
    return [ln.strip() for ln in text.splitlines() if ln.startswith('Recall@')]


@pytest.mark.parametrize('case, ps', [
    # no-embedding, one layer: the row-sharded in-kernel path
    ('sharded', 'loss=bpr-max,final_act=elu-0.5,layers=48,batch_size=16,n_sample=64,n_epochs=2,momentum=0.2,learning_rate=0.1,sample_alpha=0.5'),
    # separate embedding, two layers: the replicated NCCL path behind the same calls
    ('replicated', 'loss=cross-entropy,final_act=softmax,layers=24/16,embedding=20,batch_size=12,n_sample=48,n_epochs=2,learning_rate=0.1,dropout_p_hidden=0.1'),
])
def test_run_py_under_torchrun(tmp_path, case, ps):
    """The reference's command line, launched with torchrun on 2 GPUs: fit() trains data-parallel, evaluate_gpu() scores a shard
    of the test sessions per rank, only rank 0 prints / saves.  The metrics of the job must equal those of ONE process
    loading the saved model and scoring the whole test set (sessions are independent, the sums are exact in double)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    sys.path.insert(0, ROOT)
    from gru4rec_b200.synth import make_sessions, train_test_split
    df = make_sessions(n_items=300, n_events=9000, seed=11)
    tr, te = train_test_split(df, 0.25)
    trp, tep, mp_ = str(tmp_path / 'train.tsv'), str(tmp_path / 'test.tsv'), str(tmp_path / 'model.pickle')
    tr.to_csv(trp, sep='\t', index=False); te.to_csv(tep, sep='\t', index=False)
    port = 29541 if case == 'sharded' else 29543
    tor = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1', '--master-port', str(port)]
    run = os.path.join(ROOT, 'run.py')
    out = subprocess.run(tor + [run, trp, '-ps', ps, '-t', tep, '-m', '1', '5', '20', '-s', mp_, '-ss', '4096'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    epochs = [ln for ln in out.stdout.splitlines() if ln.startswith('Epoch')]
    assert len(epochs) == 2, out.stdout[-2000:]                   # one line per epoch for the whole job (rank 0 only)
    losses = [float(ln.split('loss:')[1].split()[0]) for ln in epochs]
    assert all(l == l and abs(l) < 1e6 for l in losses) and losses[1] < losses[0], epochs
    multi = _metric_lines(out.stdout)
    assert len(multi) == 3 and os.path.exists(mp_), out.stdout[-2000:]
    env1 = dict(os.environ, CUDA_VISIBLE_DEVICES='0')
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env1.pop(k, None)
    one = subprocess.run([sys.executable, run, mp_, '-l', '-t', tep, '-m', '1', '5', '20'], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env1)
    assert one.returncode == 0, (one.stdout[-3000:], one.stderr[-3000:])
    single = _metric_lines(one.stdout)
    assert single == multi, (single, multi)
    # a saved model scored by the 2-process job (every rank loads the pickle, rank r scores every second session)
    two = subprocess.run(tor[:-1] + [str(port + 1)] + [run, mp_, '-l', '-t', tep, '-m', '1', '5', '20'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert two.returncode == 0, (two.stdout[-3000:], two.stderr[-3000:])
    assert _metric_lines(two.stdout) == single
    print('run.py under torchrun ok:', case, epochs[-1].strip(), '|', multi[-1])
