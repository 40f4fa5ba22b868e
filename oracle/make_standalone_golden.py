"""TEST INFRASTRUCTURE ONLY.  Records what two modules of a checkout of the reference (hidasib/GRU4Rec) do, so that the tests
comparing with them run without that checkout:
  tests/golden/datatools_cases.json          its datatools.sort_if_needed / compute_offset on the cases of
                                             golden_utils.datatools_cases() (printed lines, digests of frame and offsets)
  tests/golden/bprmax_none.b200model.pickle  a pickle written by this project's savemodel() that the reference's
  tests/golden/bprmax_none.b200model.json    GRU4Rec.loadmodel + evaluate_gpu (on the Theano shim) loaded and scored: the
                                             Recall/MRR it printed, checked here against the oracle's golden numbers
Usage:  python oracle/make_standalone_golden.py PATH_TO_REFERENCE_CHECKOUT"""
import importlib.util
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
sys.path.insert(0, os.path.join(ROOT, 'tests')); sys.path.insert(0, ROOT)
from golden_utils import datatools_cases, datatools_outcome, b200_model_from_golden, load_golden, frames  # noqa: E402


def datatools(ref_dir):
    spec = importlib.util.spec_from_file_location('ref_datatools', os.path.join(ref_dir, 'datatools.py'))
    ref = importlib.util.module_from_spec(spec); spec.loader.exec_module(ref)
    out = [datatools_outcome(ref.sort_if_needed, ref.compute_offset, *case) for case in datatools_cases()]
    with open(os.path.join(GOLDEN, 'datatools_cases.json'), 'w') as f:
        json.dump(out, f, indent=0)
    print('datatools: %d cases' % len(out))


def pickle_compat(ref_dir):
    g = load_golden('bprmax_none')
    fn = os.path.join(GOLDEN, 'bprmax_none.b200model.pickle')
    b200_model_from_golden(g).savemodel(fn)
    _, te = frames(g)
    with tempfile.TemporaryDirectory() as tmp:
        te_fn = os.path.join(tmp, 'test.pickle'); te.to_pickle(te_fn)
        code = (
            "import sys, os, io, json, contextlib\n"
            "sys.path.insert(0, %r); import theano_shim; theano_shim.install()\n"
            "sys.path.insert(0, %r); cwd = os.getcwd()\n"
            "import gru4rec as ref, evaluation as ev, pandas as pd; os.chdir(cwd)\n"
            "g = ref.GRU4Rec.loadmodel(%r)\n"
            "assert type(g).__module__ == 'gru4rec' and hasattr(g.Wy, 'get_value')\n"
            "te = pd.read_pickle(%r)\n"
            "buf = io.StringIO()\n"
            "with contextlib.redirect_stdout(buf): rec, mrr = ev.evaluate_gpu(g, te, cut_off=[1, 5, 20], batch_size=7)\n"
            "print(json.dumps([[float(x) for x in rec], [float(x) for x in mrr]]))\n"
        ) % (HERE, os.path.abspath(ref_dir), fn, te_fn)
        out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300, cwd=tmp)
    assert out.returncode == 0, out.stderr[-2000:]
    rec, mrr = json.loads(out.stdout.strip().splitlines()[-1])
    np.testing.assert_allclose(rec, g['eval_standard_recall'], rtol=1e-6)
    np.testing.assert_allclose(mrr, g['eval_standard_mrr'], rtol=1e-6)
    with open(os.path.join(GOLDEN, 'bprmax_none.b200model.json'), 'w') as f:
        json.dump({'cut_off': [1, 5, 20], 'batch_size': 7, 'recall': rec, 'mrr': mrr}, f, indent=1)
    print('pickle: reference Recall', rec, 'MRR', mrr)


if __name__ == '__main__':
    if len(sys.argv) != 2 or not os.path.exists(os.path.join(sys.argv[1], 'gru4rec.py')):
        raise SystemExit(__doc__)
    datatools(sys.argv[1])
    pickle_compat(sys.argv[1])
