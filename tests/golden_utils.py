"""Helpers to replay tests/golden/*.npz (made by oracle/make_golden.py from the reference's own code)."""
import glob
import os
import numpy as np
import pandas as pd

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, '*.npz')))


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + '.npz'), allow_pickle=True))
    from collections import OrderedDict  # noqa: F401  (repr of kwargs may reference it)
    g['model_kwargs'] = eval(str(g['model_kwargs']))
    g['fit_kwargs'] = eval(str(g['fit_kwargs']))
    return g


def frames(g):
    tr = pd.DataFrame({'SessionId': g['train_SessionId'], 'ItemId': g['train_ItemId'], 'Time': g['train_Time']})
    te = pd.DataFrame({'SessionId': g['test_SessionId'], 'ItemId': g['test_ItemId'], 'Time': g['test_Time']})
    return tr, te


def init_weights(g, prefix='init_'):
    nl = len(g['model_kwargs']['layers'])
    w = dict(Wx=[g['%sWx%d' % (prefix, i)] for i in range(nl)], Wh=[g['%sWh%d' % (prefix, i)] for i in range(nl)],
             Wrz=[g['%sWrz%d' % (prefix, i)] for i in range(nl)], Bh=[g['%sBh%d' % (prefix, i)] for i in range(nl)],
             Wy=g[prefix + 'Wy'], By=g[prefix + 'By'])
    if (prefix + 'E') in g:
        w['E'] = g[prefix + 'E']
    return w


def dropout_sites(mk):
    """creation order of the reference's dropout sites: embed first (gru4rec.py:443/451), then hidden layers."""
    sites = []
    if mk.get('dropout_p_embed', 0) > 0 and (mk.get('constrained_embedding') or mk.get('embedding')):
        sites.append('e')
    if mk.get('dropout_p_hidden', 0) > 0:
        for i in range(len(mk['layers'])):
            sites.append(('h', i))
    return sites


def step_masks(g, s, M):
    mk = g['model_kwargs']
    out = {}
    for j, site in enumerate(dropout_sites(mk)):
        p = mk['dropout_p_embed'] if site == 'e' else mk['dropout_p_hidden']
        b = g['dropmask_site%d' % j][s, :M]
        out[site] = (b / np.float32(1.0 - p)).astype(np.float32)
    return out


def step_samples(g, s):
    """negative samples the reference used at train step s (row STI of the current store)."""
    if 'sample_stores' not in g:
        return None
    fs = g['store_first_step']
    k = int(np.searchsorted(fs, s, side='right') - 1)
    return g['sample_stores'][k][s - fs[k]]


def fit_data(orc, g, tr):
    """prepare_fit_data with the model's time_sort option (gru4rec.py:585)."""
    return orc.prepare_fit_data(tr, time_sort=g['model_kwargs'].get('time_sort', True))


def epoch_order(g, d, e):
    """session order of epoch e: recorded np.random.permutation for train_random_order (gru4rec.py:593), else base_order"""
    return g['epoch_orders'][e] if 'epoch_orders' in g else d['base_order']


# ---- datatools cases (tests/golden/datatools_cases.json, made by oracle/make_standalone_golden.py) ----
def datatools_cases():
    """(frame, sort columns, any_order_first_dim) of the 192 datatools comparisons, in a fixed seeded order: sorted, partly
    sorted, grouped-but-unordered and random frames of 1 to 300 rows."""
    rs = np.random.RandomState(0)
    for n in (1, 2, 50, 300):
        for trial in range(8):
            df = pd.DataFrame({'SessionId': rs.randint(0, max(2, n // 4), n), 'Time': rs.randint(0, 40, n), 'ItemId': rs.randint(0, 9, n)})
            if trial % 4 == 1: df = df.sort_values(['SessionId', 'Time']).reset_index(drop=True)
            if trial % 4 == 2: df = df.sort_values(['SessionId', 'Time', 'ItemId']).reset_index(drop=True)
            if trial % 4 == 3:      # sessions grouped but in arbitrary order
                df = df.sort_values(['SessionId', 'Time']).reset_index(drop=True)
                df = pd.concat([df[df.SessionId == s] for s in rs.permutation(df['SessionId'].unique())]).reset_index(drop=True)
            for cols in (['SessionId', 'Time'], ['SessionId', 'Time', 'ItemId'], ['SessionId']):
                for any_order in (False, True):
                    yield df.copy(), cols, any_order


def datatools_outcome(sort_if_needed, compute_offset, df, cols, any_order):
    """What sort_if_needed (printed decision, frame left in place) and compute_offset do to one case: the printed lines without
    the timing line, and SHA-256 digests of the frame (index, column names, dtypes, values) and of the offsets (dtype, values)."""
    import contextlib, hashlib, io
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        sort_if_needed(df, cols, any_order)
    h = hashlib.sha256(np.asarray(df.index.values, dtype=np.int64).tobytes())
    for c in df.columns:
        h.update(('%s:%s' % (c, df[c].dtype)).encode()); h.update(np.ascontiguousarray(df[c].values).tobytes())
    off = compute_offset(df, 'SessionId')
    return {'stdout': [l for l in buf.getvalue().splitlines() if not l.startswith('Data is sorted in')], 'frame_sha256': h.hexdigest(),
            'offset_sha256': hashlib.sha256(str(off.dtype).encode() + np.ascontiguousarray(off).tobytes()).hexdigest()}


# ---- pickle compatibility (tests/golden/bprmax_none.b200model.pickle, made by oracle/make_standalone_golden.py) ----
def b200_model_from_golden(g):
    """This project's class holding the reference's final weights of golden run `g`, ready for savemodel()."""
    import gru4rec
    m = gru4rec.GRU4Rec(**g['model_kwargs'])
    m.n_items = int(g['n_items'])
    m.itemidmap = pd.Series(data=np.arange(m.n_items), index=g['itemidmap_index'], name='ItemIdx')
    fw = init_weights(g, 'final_')
    m._host = {'Wx0': fw['Wx'][0], 'Wh0': fw['Wh'][0], 'Wrz0': fw['Wrz'][0], 'Bh0': fw['Bh'][0], 'Wy': fw['Wy'], 'By': fw['By']}
    m.error_during_train = False
    return m


def pickle_structure(path):
    """The content of a model pickle as plain comparable values, without importing any class it names from `gru4rec`: objects
    of those classes become (class name, state), bound methods taken from them become (class name, method name), arrays
    become (dtype, shape, bytes), pandas objects (type, name, index, values)."""
    import pickle

    class Stand(object):
        def __setstate__(self, st):
            self.__dict__['_state'] = st

        def __getattr__(self, name):
            if name.startswith('__'):
                raise AttributeError(name)
            return ('bound method', type(self).__name__, name)

    stand_ins = {}

    class Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            if module == 'gru4rec':
                return stand_ins.setdefault(name, type(name, (Stand,), {}))
            return pickle.Unpickler.find_class(self, module, name)

    def plain(v):
        if isinstance(v, Stand):
            return ('object', type(v).__name__, plain(v.__dict__.get('_state')))
        if isinstance(v, dict):
            return ('dict', sorted((k, plain(x)) for k, x in v.items()))
        if isinstance(v, (list, tuple)):
            return (type(v).__name__, [plain(x) for x in v])
        if isinstance(v, np.ndarray):
            return ('ndarray', v.dtype.str, v.shape, v.tobytes())
        if isinstance(v, (pd.Series, pd.Index)):
            return (type(v).__name__, v.name, plain(np.asarray(v.index if isinstance(v, pd.Series) else [])), plain(np.asarray(v.values)))
        return (type(v).__name__, v)

    with open(path, 'rb') as f:
        return plain(Unpickler(f).load())
