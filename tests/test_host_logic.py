"""CPU-side tests (-m "not gpu"): the C-ABI library loads and exports every symbol include/g4r.h declares,
the C++ schedule builder equals the oracle's literal restatement, and the host class keeps the reference surface."""
import os
import re
import numpy as np
import pytest
import gru4rec_oracle as orc
from gru4rec_b200 import _lib
from gru4rec_b200.synth import make_sessions

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, 'include', 'g4r.h')).read()
    declared = set(re.findall(r'^(?:int|int64_t|void\*|const char\*)\s+(g4r_[a-z0-9_]+)\s*\(', hdr, flags=re.M))
    assert declared, 'no declarations parsed'
    for name in sorted(declared):
        assert hasattr(lib, name), 'libg4r.so does not export %s' % name
    assert set(_lib.EXPORTS) == declared
    assert lib.g4r_version() >= 100


@pytest.mark.parametrize('B,n_sample,seed', [(4, 8, 0), (8, 0, 1), (16, 4, 2), (3, 0, 3)])
def test_train_schedule_equals_oracle(B, n_sample, seed):
    df = make_sessions(n_items=50, n_events=600, seed=seed)
    d = orc.prepare_fit_data(df)
    steps = orc.build_train_schedule(d['data_items'], d['offset_sessions'], d['base_order'], B, n_sample)
    s = _lib.Schedule(d['data_items'], d['offset_sessions'], d['base_order'], B, n_sample, mode=0)
    e = s.export()
    assert s.n_steps == len(steps)
    assert s.n_events == sum(st['M'] for st in steps)
    np.testing.assert_array_equal(s.batch_sizes(), e['M'])      # the M-only export fit() uses for the epoch loss weights
    for k, st in enumerate(steps):
        M = st['M']
        assert e['M'][k] == M
        np.testing.assert_array_equal(e['X'][k, :M], st['X'])
        np.testing.assert_array_equal(e['Y'][k, :M], st['Y'])
        np.testing.assert_array_equal(e['F'][k, :M] & 1, st['R'].astype(np.uint8))
        np.testing.assert_array_equal(e['slots'][k, :M], st['slots'])


@pytest.mark.parametrize('B,seed', [(5, 0), (11, 1), (32, 2)])
def test_eval_schedule_equals_oracle(B, seed):
    df = make_sessions(n_items=50, n_events=700, seed=seed)
    d = orc.prepare_fit_data(df)
    steps = orc.build_eval_schedule(d['data_items'], d['offset_sessions'], B)
    s = _lib.Schedule(d['data_items'], d['offset_sessions'], None, B, 0, mode=1)
    e = s.export()
    assert s.n_steps == len(steps)
    for k, st in enumerate(steps):
        M = st['M']
        assert e['M'][k] == M
        np.testing.assert_array_equal(e['X'][k, :M], st['X'])
        np.testing.assert_array_equal(e['Y'][k, :M], st['Y'])
        np.testing.assert_array_equal((e['F'][k, :M] >> 1) & 1, st['Z'].astype(np.uint8))
        np.testing.assert_array_equal(e['slots'][k, :M], st['slots'])


def test_schedule_too_few_sessions_is_index_error():
    df = make_sessions(n_items=20, n_events=30, seed=0)
    d = orc.prepare_fit_data(df)
    with pytest.raises(IndexError):
        _lib.Schedule(d['data_items'], d['offset_sessions'], d['base_order'], 64, 8, mode=0)


def test_engine_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    from gpu_utils import make_cfg
    with pytest.raises(RuntimeError):
        _lib.Engine(make_cfg(10, dict(layers=[4], batch_size=2, n_sample=0)))
    with pytest.raises(RuntimeError):
        _lib.Engine(make_cfg(10, dict(layers=[4], batch_size=2, n_sample=0)), use_torch_allocator=False)


def test_set_params_surface(capsys):
    import gru4rec
    g = gru4rec.GRU4Rec()
    g.set_params(layers='100/50', loss='cross-entropy', final_act='softmax', constrained_embedding='True', momentum='0.2', batch_size='64')
    assert g.layers == [100, 50] and g.constrained_embedding is True and g.momentum == 0.2 and g.batch_size == 64
    out = capsys.readouterr().out
    assert 'SET   layers' in out and "(type: <class 'list'>)" in out
    with pytest.raises(NotImplementedError):
        g.set_params(no_such_param=1)
    with pytest.raises(NotImplementedError):
        g.set_params(constrained_embedding='maybe')
    with pytest.raises(NotImplementedError):
        gru4rec.GRU4Rec(loss='nope')


def test_mrg_constants_self_consistency():
    """A1p72 / A1p134 are powers of the one-step MRG31k3p transition matrices (checks the recalled constants)."""
    A1 = np.array([[0, 4194304, 129], [1, 0, 0], [0, 1, 0]], dtype=object)
    A2 = np.array([[32768, 0, 32769], [1, 0, 0], [0, 1, 0]], dtype=object)

    def mpow(A, e, m):
        R = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=object)
        while e:
            if e & 1:
                R = R.dot(A) % m
            A = A.dot(A) % m
            e >>= 1
        return R
    assert (mpow(A1, 2 ** 72, orc.M1) == orc.A1p72.astype(object)).all()
    assert (mpow(A2, 2 ** 72, orc.M2) == orc.A2p72.astype(object)).all()
    assert (mpow(A1, 2 ** 134, orc.M1) == orc.A1p134.astype(object)).all()
    assert (mpow(A2, 2 ** 134, orc.M2) == orc.A2p134.astype(object)).all()


def test_loadmodel_reads_reference_written_pickle():
    """A pickle written by the REFERENCE class (tests/golden/bprmax_none.refmodel.pickle, made by oracle/make_golden.py
    under the Theano shim: class path gru4rec.GRU4Rec, bound graph-builder methods, NumPy weights) loads into this class."""
    import gru4rec
    from golden_utils import load_golden, GOLDEN_DIR
    g = load_golden('bprmax_none')
    m = gru4rec.GRU4Rec.loadmodel(os.path.join(GOLDEN_DIR, 'bprmax_none.refmodel.pickle'))
    from gru4rec_b200.gru4rec import GRU4Rec as B200Class
    assert type(m) is B200Class
    assert m.layers == [12] and m.loss == 'bpr-max' and m.final_act == 'elu-0.5' and m.n_items == int(g['n_items'])
    np.testing.assert_array_equal(m._host['Wy'], g['final_Wy'])
    np.testing.assert_array_equal(m._host['Wx0'], g['final_Wx0'])
    assert list(m.itemidmap.index.values) == list(g['itemidmap_index'])
    assert m._engine is None          # no device work until predict / evaluate is called


def test_pickle_written_here_loads_into_the_reference_class(tmp_path):
    """savemodel() of this class writes what tests/golden/bprmax_none.b200model.pickle holds -- same classes, state keys, types
    and values.  The REFERENCE's GRU4Rec.loadmodel + evaluate_gpu (run on the Theano shim by oracle/make_standalone_golden.py)
    loaded that pickle and reproduced the oracle's Recall/MRR, recorded in bprmax_none.b200model.json."""
    import json
    from golden_utils import load_golden, b200_model_from_golden, pickle_structure, GOLDEN_DIR
    g = load_golden('bprmax_none')
    fn = str(tmp_path / 'b200_model.pickle')
    b200_model_from_golden(g).savemodel(fn)
    assert pickle_structure(fn) == pickle_structure(os.path.join(GOLDEN_DIR, 'bprmax_none.b200model.pickle'))
    ref = json.load(open(os.path.join(GOLDEN_DIR, 'bprmax_none.b200model.json')))
    np.testing.assert_allclose(ref['recall'], g['eval_standard_recall'], rtol=1e-6)
    np.testing.assert_allclose(ref['mrr'], g['eval_standard_mrr'], rtol=1e-6)


def test_datatools_behaves_like_the_reference_module():
    """gru4rec_b200/datatools.py is an independent implementation; the reference's datatools.py was run on the same random
    frames by oracle/make_standalone_golden.py (tests/golden/datatools_cases.json): same printed decision, same in-place
    result, same int32 offsets."""
    import json
    from golden_utils import datatools_cases, datatools_outcome, GOLDEN_DIR
    from gru4rec_b200 import datatools as mine
    ref = json.load(open(os.path.join(GOLDEN_DIR, 'datatools_cases.json')))
    n_cases = 0
    for k, case in enumerate(datatools_cases()):
        assert datatools_outcome(mine.sort_if_needed, mine.compute_offset, *case) == ref[k], (k, case[1:])
        n_cases += 1
    assert n_cases == len(ref) == 192


def test_set_params_matches_the_reference_class():
    """set_params (gru4rec.py:162-187) of the reference, run through the shim by oracle/make_set_params_golden.py: same printed
    lines, same attribute values and types, same exception -- including string coercions, `layers=100/50`, `embedding=layersize`,
    bool strings, unknown keys and invalid values."""
    import io, json, contextlib
    import gru4rec
    cases = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'set_params_cases.json')))
    assert len(cases) >= 12
    for case in cases:
        g = gru4rec.GRU4Rec()
        buf = io.StringIO()
        exc = None
        with contextlib.redirect_stdout(buf):
            try:
                g.set_params(**case['kwargs'])
            except BaseException as e:       # noqa: BLE001
                exc = type(e).__name__
        assert exc == case['exception'], (case['kwargs'], exc)
        assert buf.getvalue() == case['stdout'], (case['kwargs'], buf.getvalue(), case['stdout'])
        for a, v in case['attrs'].items():
            mine = getattr(g, a)
            assert type(mine).__name__ == case['attr_types'][a], (case['kwargs'], a, type(mine).__name__, case['attr_types'][a])
            assert (list(mine) if isinstance(mine, (list, tuple)) else mine) == v, (case['kwargs'], a, mine, v)


@pytest.mark.parametrize('seed', range(12))
def test_schedules_equal_oracle_on_random_session_structures(seed):
    """Randomised sweep of the C++ schedule builder against the oracle's literal restatement of the reference loops
    (gru4rec.py:585-651, evaluation.py:84-147): single-event sessions (they occupy a lane for zero steps), very long sessions,
    batch sizes from 2 up to almost the number of sessions, arbitrary session orders, with and without samples."""
    rs = np.random.RandomState(100 + seed)
    n_sess = int(rs.randint(12, 80))
    kind = seed % 4
    if kind == 0:
        lens = rs.randint(1, 4, n_sess)                       # many single-event sessions
    elif kind == 1:
        lens = np.minimum(1 + rs.geometric(0.4, n_sess), 30)
    elif kind == 2:
        lens = rs.randint(2, 6, n_sess); lens[rs.randint(0, n_sess, 3)] = rs.randint(40, 90, 3)   # a few very long ones
    else:
        lens = rs.randint(1, 12, n_sess)
    offset = np.zeros(n_sess + 1, dtype=np.int32); offset[1:] = np.cumsum(lens)
    items = rs.randint(0, 37, int(offset[-1])).astype(np.int64)
    order = rs.permutation(n_sess) if seed % 2 else np.arange(n_sess)
    usable = int((lens > 1).sum())
    for B in sorted(set([2, 3, max(2, usable // 3), max(2, min(usable - 1, n_sess - 1))])):
        for n_sample in (0, 5):
            try:
                steps = orc.build_train_schedule(items, offset, order, B, n_sample)
            except IndexError:
                with pytest.raises(IndexError):
                    _lib.Schedule(items, offset, order, B, n_sample, mode=0)
                continue
            s = _lib.Schedule(items, offset, order, B, n_sample, mode=0)
            e = s.export()
            assert s.n_steps == len(steps), (seed, B, n_sample)
            for k, st in enumerate(steps):
                M = st['M']
                assert e['M'][k] == M
                np.testing.assert_array_equal(e['X'][k, :M], st['X'])
                np.testing.assert_array_equal(e['Y'][k, :M], st['Y'])
                np.testing.assert_array_equal(e['F'][k, :M] & 1, st['R'].astype(np.uint8))
                np.testing.assert_array_equal(e['slots'][k, :M], st['slots'])
        try:
            steps = orc.build_eval_schedule(items, offset, B)
        except IndexError:
            with pytest.raises(IndexError):
                _lib.Schedule(items, offset, None, B, 0, mode=1)
            continue
        s = _lib.Schedule(items, offset, None, B, 0, mode=1)
        e = s.export()
        assert s.n_steps == len(steps), (seed, B, 'eval')
        for k, st in enumerate(steps):
            M = st['M']
            assert e['M'][k] == M
            np.testing.assert_array_equal(e['X'][k, :M], st['X'])
            np.testing.assert_array_equal(e['Y'][k, :M], st['Y'])
            np.testing.assert_array_equal((e['F'][k, :M] >> 1) & 1, st['Z'].astype(np.uint8))
            np.testing.assert_array_equal(e['slots'][k, :M], st['slots'])


def test_run_py_outside_a_launcher_is_a_single_process(monkeypatch):
    """run.py joins a torch.distributed job only when a launcher describes one (WORLD_SIZE > 1)."""
    import importlib
    for k in ('WORLD_SIZE', 'RANK', 'LOCAL_RANK'):
        monkeypatch.delenv(k, raising=False)
    run = importlib.import_module('run')
    assert run._join_distributed_job() == (1, 0)
    monkeypatch.setenv('WORLD_SIZE', '1')
    assert run._join_distributed_job() == (1, 0)
    from gru4rec_b200 import parallel
    assert parallel.env_world() == (1, 0, 0) and parallel.init_from_env() == (1, 0)
    monkeypatch.setenv('WORLD_SIZE', '4'); monkeypatch.setenv('RANK', '2'); monkeypatch.setenv('LOCAL_RANK', '2')
    assert parallel.env_world() == (4, 2, 2)
    np.testing.assert_array_equal(parallel.shard_eval_sessions(10, 2, 4), [2, 6])
    assert len(parallel.shard_eval_sessions(2, 3, 4)) == 0               # a rank without sessions contributes zeros


def test_c_caller_links_against_the_abi(tmp_path):
    """include/g4r.h is plain C99 and a C program can drive the host-side entry points of libg4r.so (INTEGRATION.md section 3)."""
    import shutil
    import subprocess
    gcc = shutil.which('gcc')
    if gcc is None:
        pytest.skip('no gcc')
    inc, libdir = os.path.join(ROOT, 'include'), os.path.join(ROOT, 'gru4rec_b200')
    r = subprocess.run([gcc, '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-fsyntax-only', '-x', 'c', os.path.join(inc, 'g4r.h')], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    exe = str(tmp_path / 'c_abi_caller')
    cuda_lib = '/usr/local/cuda/lib64'
    r = subprocess.run([gcc, '-std=c99', '-Wall', '-Wextra', '-pedantic', '-I' + inc, os.path.join(ROOT, 'tests', 'c_abi_caller.c'), '-L' + libdir, '-lg4r',
                        '-Wl,-rpath,' + libdir, '-L' + cuda_lib, '-Wl,-rpath,' + cuda_lib, '-o', exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert 'c caller ok' in r.stdout and 'step 0: M=2 X=[5,1] Y=[6,2] reset=[0,1]' in r.stdout
