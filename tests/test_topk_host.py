"""CPU tests of the host side of GRU4Rec.recommend_next_batch(): argument checks, id mapping and the session bookkeeping it shares
with predict_next_batch, driven through an engine double whose predict_topk selects from the oracle's predict() output."""
import os

import numpy as np
import pytest

import oracle_engine
from golden_utils import GOLDEN_DIR


class TopkOracleEngine(oracle_engine.OracleEngine):
    """OracleEngine plus predict_topk: stable selection (score desc, index asc) from predict(); the softmax family renormalised
    over the candidates."""
    calls = 0

    def predict_topk(self, X, k, reset_mask=None, cand=None):
        TopkOracleEngine.calls += 1
        P = self.predict(X, reset_mask)
        idx = np.arange(P.shape[1]) if cand is None else np.asarray(cand)
        P = P[:, idx]
        if self.mk['final_act'] in ('softmax', 'softmax_logit') and cand is not None:
            P = P / P.sum(axis=1, keepdims=True)
        items = np.empty((len(X), k), dtype=np.int32); scores = np.empty((len(X), k), dtype=np.float32)
        for b in range(len(X)):
            o = np.lexsort((idx, -P[b]))[:k]
            items[b], scores[b] = idx[o], P[b, o]
        return items, scores


def _install(monkeypatch, gru):
    from gru4rec_b200 import _lib
    made = []

    def make(cfg, device=0):
        eng = TopkOracleEngine(cfg, oracle_engine.model_kwargs_of(gru), device)
        made.append(eng)
        return eng
    monkeypatch.setattr(_lib, 'Engine', make)
    return made


def _load():
    import gru4rec
    return gru4rec.GRU4Rec.loadmodel(os.path.join(GOLDEN_DIR, 'bprmax_none.refmodel.pickle'))


def test_recommend_matches_predict_dataframe_and_interleaves(monkeypatch):
    """Model A only calls predict_next_batch; model B alternates predict_next_batch and recommend_next_batch while session ids
    change per lane.  B's recommendations are the top-k of A's DataFrame at every step, as original item ids."""
    a, b = _load(), _load()
    _install(monkeypatch, a); _install(monkeypatch, b)
    ids = a.itemidmap.index.values
    rs = np.random.RandomState(3)
    sess = np.arange(4)
    for step in range(8):
        sess = np.where(rs.rand(4) < 0.4, sess + 10, sess)
        inp = ids[rs.randint(0, len(ids), 4)]
        cand = None if step % 3 else ids[rs.choice(len(ids), 15, replace=False)]
        df = a.predict_next_batch(sess, inp, cand, batch=4)
        if step % 2:
            b.predict_next_batch(sess, inp, cand, batch=4)
            continue
        rec, sc = b.recommend_next_batch(sess, inp, k=5, predict_for_item_ids=cand, batch=4)
        assert rec.shape == (4, 5) and sc.shape == (4, 5) and sc.dtype == np.float32
        for lane in range(4):
            col = df.iloc[:, lane]
            order = np.lexsort((np.arange(len(col)), -col.values))[:5]
            assert list(rec[lane]) == list(col.index.values[order])
            np.testing.assert_array_equal(sc[lane], col.values[order])


def test_recommend_rejects_bad_arguments_before_touching_the_engine(monkeypatch):
    gru = _load()
    made = _install(monkeypatch, gru)
    ids = gru.itemidmap.index.values
    for k in (0, 257, gru.n_items + 1, 2.0, True):
        with pytest.raises(ValueError):
            gru.recommend_next_batch(np.arange(2), ids[:2], k=k, batch=2)
    with pytest.raises(ValueError):
        gru.recommend_next_batch(np.arange(2), ids[:2], k=3, predict_for_item_ids=ids[:2], batch=2)      # k > candidates
    with pytest.raises(ValueError):
        gru.recommend_next_batch(np.arange(2), ids[:2], k=2, predict_for_item_ids=[ids[0], ids[1], ids[0]], batch=2)
    unknown = max(ids) + 1 if np.issubdtype(np.asarray(ids).dtype, np.number) else 'no-such-item'
    with pytest.raises(KeyError):
        gru.recommend_next_batch(np.arange(2), [ids[0], unknown], k=2, batch=2)
    with pytest.raises(KeyError):
        gru.recommend_next_batch(np.arange(2), ids[:2], k=2, predict_for_item_ids=[ids[0], unknown], batch=2)
    assert made == [] and gru.predict is None
    rec, _ = gru.recommend_next_batch(np.arange(2), ids[:2], k=np.int64(3), batch=2)
    assert rec.shape == (2, 3) and len(made) == 1
