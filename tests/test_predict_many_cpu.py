"""Host logic of prediction that needs no GPU: the argument errors BSR.predict_many and the single-estimator methods raise before
any library call, the concatenated packed table they upload, the group tables they hand to capi.predict_groups, and the malformed
dense models bsr_predict_many and bsr_predict_trees refuse before they look for a device."""
import ctypes

import numpy as np
import pytest

from mcmc_symreg_b200 import BSR, capi
from mcmc_symreg_b200 import experiments
from mcmc_symreg_b200.trees import OP_ADD, OP_LT


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(capi, "load", refuse)
    monkeypatch.setattr(capi, "predict_groups", refuse)


def _fake_fit(MM, K, rng, **params):
    """an estimator holding a fit of MM random restarts of K trees (what _set_results receives from a run)"""
    nn = rng.integers(1, 12, (MM, K)).astype(np.int32)
    n = int(nn.sum())
    ptok = rng.integers(0, 11, n).astype(np.uint32) | (rng.integers(0, 3, n).astype(np.uint32) << 16)
    n_lt = int(np.count_nonzero((ptok & 0xFF) == 2))
    est = BSR(K, MM, **params)
    est._set_results(dict(nn=nn, ptok=ptok, pab=rng.normal(size=(n_lt, 2)), beta=rng.normal(size=(MM, K + 1)), sse=rng.random(MM),
                          counters=rng.integers(0, 99, (MM, capi.N_COUNTERS)), done=np.ones(MM, np.int32),
                          nerr=rng.integers(1, 5, MM).astype(np.int32), err=rng.random((MM, 6)), sweeps=10))
    return est


def test_argument_errors_before_any_library_call(no_library):
    rng = np.random.default_rng(0)
    a, b = _fake_fit(4, 3, rng), _fake_fit(5, 3, rng)
    X = np.zeros((7, 2))
    with pytest.raises(ValueError, match="2 fits and 1 test sets"):
        BSR.predict_many([a, b], [X])
    with pytest.raises(ValueError, match="method must be"):
        BSR.predict_many([a, b], [X, X], method="median")
    with pytest.raises(ValueError, match="treeNum = 2, fit 0 has 3"):
        BSR.predict_many([a, _fake_fit(4, 2, rng)], [X, X])
    with pytest.raises(ValueError, match="on device 1, fit 0 on device 0"):
        BSR.predict_many([a, _fake_fit(4, 3, rng, device=1)], [X, X])
    with pytest.raises(ValueError, match="last_ind = 5 is outside 1 .. 4"):
        BSR.predict_many([a, b], [X, X], last_ind=5)
    with pytest.raises(ValueError, match="last_ind = 0"):
        BSR.predict_many([a, b], [X, X], last_ind=0)
    with pytest.raises(ValueError, match="2 fits and 1 data sets"):
        experiments.summarize_many([a, b], [dict(X=X)])
    assert BSR.predict_many([], []) == []
    assert experiments.summarize_many([], []) == []


def test_unfitted_estimator_fails_like_predict(no_library):
    fitted, unfitted = _fake_fit(4, 3, np.random.default_rng(1)), BSR(3, 4)
    X = np.zeros((3, 2))
    with pytest.raises(AttributeError) as single:
        unfitted.predict(X)
    with pytest.raises(AttributeError) as many:
        BSR.predict_many([fitted, unfitted], [X, X])
    assert str(many.value) == str(single.value)


def test_concatenated_table_decodes_to_each_fits_trees():
    """PackedTrees.concat: model m of fit i is model first[i] + m of the concatenated table, tree for tree"""
    rng = np.random.default_rng(2)
    fits = [_fake_fit(MM, 4, rng) for MM in (3, 1, 6, 2)]
    cat = capi.PackedTrees.concat([f._packed_ for f in fits])
    first = np.cumsum([0] + [f._packed_.nn.shape[0] for f in fits])
    assert cat.nn.shape == (first[-1], 4)
    for i, f in enumerate(fits):
        for m in range(f._packed_.nn.shape[0]):
            for k in range(4):
                for x, y in zip(cat.tree(int(first[i] + m), k), f._packed_.tree(m, k)):
                    np.testing.assert_array_equal(x, y)
    dense = cat.dense()
    for i, f in enumerate(fits):
        for x, y in zip(dense, f._packed_.dense()):
            np.testing.assert_array_equal(x[first[i]:first[i + 1]], y)


def test_selected_models_decode_to_their_trees():
    """PackedTrees.select: model j of the selection is model idx[j] of the table, in any order and with repeats"""
    pk = _fake_fit(9, 4, np.random.default_rng(5))._packed_
    for idx in ([3], [8, 0, 5], [2, 2, 7], list(range(9))):
        for x, y in zip(pk.select(idx).dense(), pk.dense()):
            np.testing.assert_array_equal(x, y[idx])


def test_single_fit_predictions_upload_only_the_selected_models(monkeypatch):
    """predict, predict_best and predict_mean hand capi.predict_groups one group over the selected restarts' own table"""
    est = _fake_fit(6, 3, np.random.default_rng(6))
    X = np.zeros((4, 2))
    calls = []

    def fake(device, nn, tok, ab, beta, sets, grp_set, grp_models, grp_reduce):
        calls.append(dict(pk=capi.PackedTrees(nn, tok, ab), beta=beta, grp_models=[list(m) for m in grp_models], grp_reduce=grp_reduce))
        n = sets[0].shape[0]
        return [np.full((2, n), 7.0) if grp_reduce[0] else np.full((len(grp_models[0]), n), 5.0)], np.array([4], np.int32)

    monkeypatch.setattr(capi, "predict_groups", fake)
    assert est.predict(X, last_ind=2).shape == (4, 1)
    m, s = est.predict_mean(X, chains=[4, 1], return_std=True)
    assert m.shape == s.shape == (4, 1) and est.n_used_ == 4
    for c, idx in zip(calls, ([4], [4, 1])):
        assert c["grp_models"] == [list(range(len(idx)))]
        np.testing.assert_array_equal(c["beta"], np.stack(est.betas_)[idx, :, 0])
        for x, y in zip(c["pk"].dense(), est._packed_.dense()):
            np.testing.assert_array_equal(x, y[idx])
    assert [c["grp_reduce"] for c in calls] == [[False], [True]]


def test_group_tables(monkeypatch):
    """what predict_many and summarize_many hand to capi.predict_groups: the concatenated models and betas, one group per fit (per
    fit and set for summarize_many) with global model indices, and the per-group results back in the methods' shapes"""
    rng = np.random.default_rng(3)
    fits = [_fake_fit(MM, 3, rng) for MM in (4, 2, 5)]
    Xs = [rng.normal(size=(n, 2)) for n in (3, 1, 8)]
    calls = []

    def fake(device, nn, tok, ab, beta, sets, grp_set, grp_models, grp_reduce):
        calls.append(dict(nn=nn, tok=tok, ab=ab, beta=beta, sets=sets, grp_set=list(grp_set), grp_models=[list(m) for m in grp_models],
                          grp_reduce=list(grp_reduce)))
        blocks = [np.full((2, sets[s].shape[0]), 10.0 * g) if r else np.full((len(m), sets[s].shape[0]), float(g))
                  for g, (s, m, r) in enumerate(zip(grp_set, grp_models, grp_reduce))]
        return blocks, np.arange(len(grp_set), dtype=np.int32) + 100

    monkeypatch.setattr(capi, "predict_groups", fake)
    out = BSR.predict_many(fits, Xs, last_ind=2)
    c = calls[-1]
    assert c["grp_set"] == [0, 1, 2] and c["grp_models"] == [[2], [4], [9]] and c["grp_reduce"] == [False] * 3
    np.testing.assert_array_equal(c["nn"], np.concatenate([f._packed_.nn for f in fits]))
    np.testing.assert_array_equal(c["beta"], np.concatenate([np.stack(f.betas_)[:, :, 0] for f in fits]))
    assert [o.shape for o in out] == [(3, 1), (1, 1), (8, 1)] and [float(o[0, 0]) for o in out] == [0.0, 1.0, 2.0]
    BSR.predict_many(fits, Xs, method="best")
    assert calls[-1]["grp_models"] == [[f.best_chain() + o] for f, o in zip(fits, (0, 4, 6))]
    out = BSR.predict_many(fits, Xs, method="mean", return_std=True)
    assert calls[-1]["grp_models"] == [[0, 1, 2, 3], [4, 5], [6, 7, 8, 9, 10]] and calls[-1]["grp_reduce"] == [True] * 3
    assert [f.n_used_ for f in fits] == [100, 101, 102]
    assert all(m.shape == s.shape == (X.shape[0], 1) for (m, s), X in zip(out, Xs))
    data = [dict(X=X, X_test=X[:1], X_extra=2 * X) for X in Xs]
    monkeypatch.setattr(experiments, "_summary", lambda est, dat, preds: preds)
    rows = experiments.summarize_many(fits, data)
    c = calls[-1]
    assert len(c["sets"]) == 9 and c["grp_set"] == [s for s in range(9) for _ in range(3)]
    assert c["grp_reduce"] == [False, False, True] * 9
    assert [f.n_used_ for f in fits] == [108, 117, 126]
    assert [float(rows[1]["test"][j][0]) for j in range(3)] == [12.0, 13.0, 140.0]


def test_restart_index_out_of_range_before_any_library_call(no_library):
    est = _fake_fit(4, 3, np.random.default_rng(4))
    X = np.zeros((3, 2))
    for call in (lambda: est.predict(X, last_ind=0), lambda: est.predict(X, last_ind=5),
                 lambda: est.predict_mean(X, chains=[-1]), lambda: est.predict_mean(X, chains=[0, 4])):
        with pytest.raises(IndexError, match="outside 0 .. 3"):
            call()


def _dense(M, K):
    """M models of K trees (+ (lt x1) x0) in dense [M][K][64] slots"""
    tok = np.zeros((M, K, capi.MAX_NODES), np.uint32)
    tok[:, :, :4] = [OP_ADD, OP_LT, 1 << 16, 0]
    pa, pb = np.full(tok.shape, 2.0), np.full(tok.shape, 0.5)
    return dict(tok=tok, pa=pa, pb=pb, nn=np.full((M, K), 4, np.int32), beta=np.ones((M, K + 1)))


def _predict_dense(entry, a, X):
    lib = capi.load()
    M, K = a["nn"].shape
    p = {k: None if v is None else capi._ptr(v) for k, v in a.items()}
    out = np.zeros((M, X.shape[0]))
    if entry == "bsr_predict_trees":
        rc = lib.bsr_predict_trees(0, K, p["tok"], p["pa"], p["pb"], p["nn"], p["beta"], capi._ptr(X), X.shape[0], X.shape[1],
                                   capi._ptr(out))
    else:
        rc = lib.bsr_predict_many(0, M, K, p["tok"], p["pa"], p["pb"], p["nn"], p["beta"], capi._ptr(X), X.shape[0], X.shape[1], 0,
                                  capi._ptr(out), ctypes.byref(ctypes.c_int32()))
    capi._ck(rc)


@pytest.mark.parametrize("entry", ["bsr_predict_many", "bsr_predict_trees"])
def test_dense_entry_points_refuse_malformed_models(entry):
    """each malformed model is refused on the host under the entry point's own name, before the library looks for a device"""
    M = 3 if entry == "bsr_predict_many" else 1
    X = np.zeros((5, 2))

    def changed(name, index, value):
        a = _dense(M, 2)
        if value is None:
            a[name] = None
        else:
            a[name][index] = value
        return a

    cases = [("unknown opcode", changed("tok", (M - 1, 1, 2), 11)),
             ("not a pre-order tree", changed("tok", (M - 1, 1, 3), OP_ADD)),                    # a leaf turned into +
             ("reads a feature the data does not have", changed("tok", (0, 0, 2), 2 << 16)),
             ("tree size out of range", changed("nn", (M - 1, 0), 0)),
             ("tree size out of range", changed("nn", (0, 1), 65)),
             ("null argument", changed("pa", None, None))]
    for match, a in cases:
        with pytest.raises(capi.BsrError, match=entry + ": .*" + match):
            _predict_dense(entry, a, X)


@pytest.mark.parametrize("entry", ["bsr_predict_many", "bsr_predict_trees"])
def test_dense_entry_points_have_no_cpu_fallback(entry):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    M = 3 if entry == "bsr_predict_many" else 1
    with pytest.raises(capi.BsrError, match=entry + r": no CUDA device \(no CPU fallback\)"):
        _predict_dense(entry, _dense(M, 2), np.zeros((5, 2)))
