"""-m gpu: on-device top-k (g4r_predict_topk / Engine.predict_topk / GRU4Rec.recommend_next_batch) against the predict path.
Elementwise final activations: exactly the first k of a stable sort of predict()'s rows, scores bit-equal.  Softmax family:
a valid top-k of predict()'s rows at 1e-5 relative.  Recorded outputs of the original: a valid top-k at the fixtures' 2e-4."""
import os

import numpy as np
import pandas as pd
import pytest

from gru4rec_b200 import _lib
from golden_utils import GOLDEN_DIR, golden_names, load_golden, init_weights
from gpu_utils import make_pair, make_cfg, push_weights

pytestmark = pytest.mark.gpu

ELEMENTWISE = ['linear', 'relu', 'tanh', 'leaky-0.1', 'elu-0.5', 'selu-1.05-1.7']


def ref_topk(P, k, cols=None):
    """first k of each row by (score desc, column index asc); cols: the item index of every column"""
    cols = np.arange(P.shape[1]) if cols is None else np.asarray(cols)
    kth = -np.partition(-P, k - 1, axis=1)[:, k - 1]
    items = np.empty((P.shape[0], k), dtype=np.int64); scores = np.empty((P.shape[0], k), dtype=np.float32)
    for b in range(P.shape[0]):
        c = np.nonzero(P[b] >= kth[b])[0]
        o = c[np.lexsort((cols[c], -P[b, c]))][:k]
        items[b], scores[b] = cols[o], P[b, o]
    return items, scores


def engines(n_items, mk, lanes, seed, edit=None):
    """two engines with identical random weights (edit(m) may change the oracle's weights before they are pushed)"""
    e1, m, _, rs = make_pair(n_items, mk, seed=seed, eval_lanes=lanes)
    if edit is not None:
        edit(m, rs)
        push_weights(e1, m)
    e2 = _lib.Engine(make_cfg(n_items, mk, eval_lanes=lanes))
    push_weights(e2, m)
    return e1, e2, rs


def lockstep_exact(n_items, mk, batch, k, seed=0, steps=2, edit=None):
    e1, e2, rs = engines(n_items, mk, batch, seed, edit)
    try:
        for s in range(steps):
            X = rs.randint(0, n_items, batch)
            R = (rs.rand(batch) < 0.3).astype(np.uint8) if s else np.ones(batch, np.uint8)
            P = e1.predict(X, R)
            items, scores = e2.predict_topk(X, k, R)
            ri, rsc = ref_topk(P, k)
            assert items.shape == (batch, k) and scores.dtype == np.float32
            np.testing.assert_array_equal(items, ri, err_msg='%s step %d' % (mk, s))
            np.testing.assert_array_equal(scores.view(np.uint32), rsc.view(np.uint32), err_msg='%s step %d' % (mk, s))
    finally:
        e1.close(); e2.close()


def _mk(layers, emb, act):
    loss = {'softmax': 'cross-entropy', 'softmax_logit': 'xe_logit'}.get(act, 'bpr-max')
    mk = dict(layers=layers, batch_size=8, n_sample=16, loss=loss, final_act=act)
    if emb == 'embed':
        mk['embedding'] = 24
    elif emb == 'constrained':
        mk['constrained_embedding'] = True
    return mk


# (n_items, layers, embedding mode, batch, k): every item count, width, batch, k and embedding mode of the grid appears
CASES = [
    (70, [16], 'none', 6, 20),
    (70, [100], 'embed', 1, 70),
    (70, [130, 16], 'none', 512, 1),
    (1000, [100], 'none', 100, 256),
    (1000, [130], 'embed', 6, 100),
    (1000, [512], 'constrained', 1, 1),
    (1000, [16, 100], 'none', 100, 20),
    (37483, [100], 'none', 512, 20),
    (37483, [130], 'constrained', 100, 100),
    (37483, [512], 'embed', 6, 256),
    (37483, [16], 'constrained', 1, 256),
]


@pytest.mark.parametrize('case', CASES, ids=lambda c: '%d-%s-%s-b%d-k%d' % (c[0], 'x'.join(map(str, c[1])), c[2], c[3], c[4]))
def test_topk_exact_against_predict(case):
    n_items, layers, emb, batch, k = case
    for i, act in enumerate(ELEMENTWISE):
        lockstep_exact(n_items, _mk(layers, emb, act), batch, k, seed=i)


@pytest.mark.parametrize('act', ['linear', 'relu', 'elu-0.5'])
def test_topk_exact_ties(act):
    """Duplicated Wy / By rows (exact score ties) and, for relu, a large negative bias that flattens most scores to 0: lower item
    indices come first among ties."""
    def dup(m, rs):
        src = rs.randint(0, 300, 900)
        m.Wy[100:1000] = m.Wy[src]; m.By[100:1000] = m.By[src]
        if act == 'relu':
            m.By[:] -= 1.0
    lockstep_exact(1000, _mk([100], 'none', act), 100, 256, seed=5, steps=3, edit=dup)
    lockstep_exact(1000, _mk([130], 'none', act), 6, 20, seed=6, steps=3, edit=dup)


def check_valid_topk(items, scores, P, cols, k, rtol, atol=0.0):
    """items/scores a top-k of P (columns = item indices `cols`): rows non-increasing, scores match P at the items, and nothing
    left out scores above the smallest returned one (within the tolerance)."""
    cols = np.asarray(cols)
    pos = {c: j for j, c in enumerate(cols)}
    for b in range(P.shape[0]):
        assert len(set(items[b])) == k
        assert np.all(np.diff(scores[b]) <= 0), scores[b]
        j = np.array([pos[i] for i in items[b]])
        np.testing.assert_allclose(scores[b], P[b, j], rtol=rtol, atol=atol)
        rest = np.delete(P[b], j)
        if rest.size:
            lo = P[b, j].min()
            assert rest.max() <= lo + rtol * abs(lo) + atol, (rest.max(), lo)


@pytest.mark.parametrize('act', ['softmax', 'softmax_logit'])
@pytest.mark.parametrize('n_items,layers,batch,k', [(1000, [100], 100, 20), (37483, [130], 6, 256), (37483, [512], 512, 100)])
def test_topk_softmax_family(act, n_items, layers, batch, k):
    mk = _mk(layers, 'none', act)
    e1, e2, rs = engines(n_items, mk, batch, seed=11)
    try:
        for s in range(2):
            X = rs.randint(0, n_items, batch)
            R = np.ones(batch, np.uint8) if s == 0 else np.zeros(batch, np.uint8)
            if s == 0:          # whole catalogue
                P = e1.predict(X, R)
                items, scores = e2.predict_topk(X, k, R)
                check_valid_topk(items, scores, P, np.arange(n_items), k, rtol=1e-5)
            else:               # candidate subset: predict_next_batch's renormalised values
                cand = rs.choice(n_items, max(k, n_items // 3), replace=False)
                P = e1.predict(X, R)[:, cand]
                P = P / P.sum(axis=1, keepdims=True)
                items, scores = e2.predict_topk(X, k, R, cand=cand)
                check_valid_topk(items, scores, P, cand, k, rtol=1e-5)
    finally:
        e1.close(); e2.close()


def test_topk_subset_exact_elementwise():
    """candidate subset, elementwise activation: exact against predict() restricted to the candidates (ties by item index)"""
    mk = _mk([100], 'none', 'relu')
    e1, e2, rs = engines(5000, mk, 100, seed=12)
    try:
        for s in range(2):
            X = rs.randint(0, 5000, 100)
            cand = rs.choice(5000, 1700, replace=False)
            P = e1.predict(X)
            items, scores = e2.predict_topk(X, 50, cand=cand)
            ri, rsc = ref_topk(P[:, cand], 50, cols=cand)
            np.testing.assert_array_equal(items, ri)
            np.testing.assert_array_equal(scores.view(np.uint32), rsc.view(np.uint32))
    finally:
        e1.close(); e2.close()


def _golden_model(g):
    import gru4rec
    mk = g['model_kwargs']
    gru = gru4rec.GRU4Rec(**mk)
    gru.n_items = int(g['n_items'])
    gru.itemidmap = pd.Series(data=np.arange(gru.n_items), index=g['itemidmap_index'], name='ItemIdx')
    fw = init_weights(g, 'final_')
    host = {'Wy': fw['Wy'], 'By': fw['By']}
    for i in range(len(mk['layers'])):
        host.update({'Wx%d' % i: fw['Wx'][i], 'Wh%d' % i: fw['Wh'][i], 'Wrz%d' % i: fw['Wrz'][i], 'Bh%d' % i: fw['Bh'][i]})
    if 'E' in fw:
        host['E'] = fw['E']
    gru._host = host
    gru.error_during_train = False
    gru.predict = None
    return gru


def _check_recorded(gru, g, k_max=20):
    """the probe of the fixtures through recommend_next_batch: a valid top-k of the original's recorded predict outputs"""
    probe = g['predict_probe_items']
    ids = np.asarray(gru.itemidmap.index.values)
    k = min(k_max, gru.n_items)
    for sess, inp, key in ((np.arange(5), probe, 'predict_out1'), (np.arange(5), probe[::-1].copy(), 'predict_out2')):
        rec, sc = gru.recommend_next_batch(sess, inp, k=k, batch=5)
        check_valid_topk(gru.itemidmap[rec.reshape(-1)].values.reshape(rec.shape), sc, np.asarray(g[key]).T, np.arange(gru.n_items), k,
                         rtol=2e-4, atol=1e-6)
    sub = np.asarray(g['predict_sub_items'])
    ks = min(k_max, len(sub))
    for sess, inp, key in ((np.arange(5) + 200, probe, 'predict_sub_out1'), (np.arange(5) + 200, probe[::-1].copy(), 'predict_sub_out2')):
        rec, sc = gru.recommend_next_batch(sess, inp, k=ks, predict_for_item_ids=sub, batch=5)
        assert set(rec.reshape(-1)) <= set(sub)
        check_valid_topk(rec, sc, np.asarray(g[key]).T, sub, ks, rtol=2e-4, atol=1e-6)
    return ids


@pytest.mark.parametrize('name', golden_names())
def test_topk_against_recorded_outputs(name):
    g = load_golden(name)
    _check_recorded(_golden_model(g), g)


def test_topk_reference_pickle():
    import gru4rec
    g = load_golden('bprmax_none')
    m = gru4rec.GRU4Rec.loadmodel(os.path.join(GOLDEN_DIR, 'bprmax_none.refmodel.pickle'))
    _check_recorded(m, g)


def test_recommend_interleaved_with_predict_next_batch():
    """Two models from one pickle: A calls only predict_next_batch, B alternates both methods while session ids change per lane;
    B's top-k equals the top-k of A's DataFrame at every step (exact: same scores, elementwise activation)."""
    import gru4rec
    fn = os.path.join(GOLDEN_DIR, 'bprmax_none.refmodel.pickle')
    a, b = gru4rec.GRU4Rec.loadmodel(fn), gru4rec.GRU4Rec.loadmodel(fn)
    ids = a.itemidmap.index.values
    rs = np.random.RandomState(7)
    sess = np.arange(6)
    for step in range(12):
        sess = np.where(rs.rand(6) < 0.3, sess + 100, sess)
        inp = ids[rs.randint(0, len(ids), 6)]
        cand = None if step % 3 else ids[rs.choice(len(ids), 25, replace=False)]
        df = a.predict_next_batch(sess, inp, cand, batch=6)
        if step % 2:
            b.predict_next_batch(sess, inp, cand, batch=6)
            continue
        rec, sc = b.recommend_next_batch(sess, inp, k=10, predict_for_item_ids=cand, batch=6)
        ri, rsc = ref_topk(df.values.T.copy(), 10)
        np.testing.assert_array_equal(rec, df.index.values[ri])
        np.testing.assert_array_equal(sc.view(np.uint32), rsc.view(np.uint32))


def test_topk_large_shape():
    """Rees46 shape once: 172k items, GRU(512), constrained embedding, batch 240, k = 100."""
    mk = dict(layers=[512], batch_size=8, n_sample=16, loss='bpr-max', final_act='elu-0.5', constrained_embedding=True)
    lockstep_exact(172000, mk, 240, 100, seed=3, steps=2)


def test_topk_errors():
    import gru4rec
    m = gru4rec.GRU4Rec.loadmodel(os.path.join(GOLDEN_DIR, 'bprmax_none.refmodel.pickle'))
    ids = m.itemidmap.index.values
    for k in (0, 257, m.n_items + 1):
        with pytest.raises(ValueError):
            m.recommend_next_batch(np.arange(2), ids[:2], k=k, batch=2)
    with pytest.raises(ValueError):
        m.recommend_next_batch(np.arange(2), ids[:2], k=3, predict_for_item_ids=ids[:2], batch=2)
    with pytest.raises(ValueError):
        m.recommend_next_batch(np.arange(2), ids[:2], k=2, predict_for_item_ids=[ids[0], ids[1], ids[1]], batch=2)
    with pytest.raises(KeyError):
        m.recommend_next_batch(np.arange(2), [ids[0], 'no-such-item' if isinstance(ids[0], str) else max(ids) + 1], k=2, batch=2)
    rec, sc = m.recommend_next_batch(np.arange(2), ids[:2], k=2, batch=2)
    assert rec.shape == (2, 2) and sc.shape == (2, 2)
    eng = m._engine
    n = m.n_items
    with pytest.raises(IndexError):
        eng.predict_topk(np.array([0, n]), 2)
    with pytest.raises(IndexError):
        eng.predict_topk(np.array([0, 1]), 2, cand=np.array([0, n]))
    with pytest.raises(NotImplementedError):        # G4R_ERR_INVALID at engine level: bad k, duplicates, batch above the lanes
        eng.predict_topk(np.array([0, 1]), 0)
    with pytest.raises(NotImplementedError):
        eng.predict_topk(np.array([0, 1]), 2, cand=np.array([3, 3]))
    with pytest.raises(NotImplementedError):
        eng.predict_topk(np.zeros(eng.cfg.eval_batch_size + 1, np.int32), 2)
