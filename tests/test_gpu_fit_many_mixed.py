"""GPU tests of data sets of different feature counts in one handle (bsr_set_datasets_mixed_host) and of
BSR.fit_many(mixed_features=True): the chains of data set b end bit for bit where the chains of a handle that holds only data set b
(with its own d_b features) end, keyed the same way, whenever data set b's rows lie in the batch's first row split."""
import numpy as np
import pytest

import parity_helpers as H
from test_gpu_fit_many import _assert_same_chains, _fits_equal, _state

pytestmark = pytest.mark.gpu

FEATURES = (1, 2, 3, 5, 8)
ROWS = (3, 97, 1025, 3001)


def _target(X):
    g = (lambda v: v, lambda v: v * v, np.sin, np.cos)
    y = sum(g[j % 4](X[:, j]) / (j + 1) for j in range(X.shape[1]))
    return y + (X[:, 0] * X[:, -1] if X.shape[1] > 1 else 0.0)


def _datasets(shapes, lo=-3.0, hi=3.0, seed=41):
    rng = np.random.default_rng(seed)
    Xs = [rng.uniform(lo, hi, (n, d)) for n, d in shapes]
    return Xs, [_target(X) for X in Xs]


def _layout(D, C, layout):
    if layout == "contiguous":
        return np.repeat(np.arange(D), C), np.tile(np.arange(C), D)
    return np.arange(D * C) % D, np.arange(D * C) // D


def _mixed_and_singles(Xs, ys, seeds, K, C, precision="fp32", mode="fixed", layout="contiguous"):
    D = len(Xs)
    stop = dict(val=100, plateau=True) if mode == "until" else dict(val=0, plateau=False)
    chain_ds, ids = _layout(D, C, layout)
    batch = H.default_engine(K, D * C, max(X.shape[1] for X in Xs), precision=precision, **stop)
    batch.set_datasets_mixed(Xs, ys, chain_ds)
    batch.init_chains_keyed(np.asarray(seeds)[chain_ds], ids)
    singles = []
    for b in range(D):
        e = H.default_engine(K, C, Xs[b].shape[1], precision=precision, **stop)
        e.set_data(Xs[b], ys[b])
        e.init_chains(seeds[b])
        singles.append(e)
    return batch, singles, chain_ds


def _run(engines, mode, run):
    for e in engines:
        if mode == "fixed":
            e.run(run)
        else:
            e.run_until_done(3000, check_every=32)


def _close(*engines):
    for e in engines:
        e.close()


def _leaf_features(trees):
    """largest leaf feature of every chain's trees (tok [C][K][64], nn [C][K]); -1 for a chain without leaves"""
    tok, _, _, nn = trees
    tok = tok.astype(np.int64)
    used = np.arange(tok.shape[2])[None, None, :] < nn[:, :, None]
    leaf = used & ((tok & 0xFF) == 0)
    return np.where(leaf, tok >> 16, -1).reshape(tok.shape[0], -1).max(axis=1)


@pytest.mark.parametrize("layout", ["contiguous", "interleaved"])
@pytest.mark.parametrize("mode", ["fixed", "until"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_mixed_match_single_handles(precision, mode, layout):
    """1 ... 8 features crossed with 3 ... 3001 rows, 24 chains each: every chain equals its single-data-set run, bit for bit"""
    shapes = [(n, d) for d in FEATURES for n in ROWS]
    Xs, ys = _datasets(shapes)
    batch, singles, chain_ds = _mixed_and_singles(Xs, ys, [7 * (b + 1) for b in range(len(shapes))], 3, 24, precision, mode, layout)
    g = batch.window_geometry()
    assert g["splits"] == 1 and g["rows_per_split"] >= max(ROWS)
    _run([batch] + singles, mode, 30)
    got = _state(batch)
    for b, e in enumerate(singles):
        assert e.window_geometry()["splits"] == 1
        _assert_same_chains(got, np.nonzero(chain_ds == b)[0], _state(e))
    assert got["stats"]["counters"][:, 1].sum() > 0          # the chains moved
    _close(batch, *singles)


def test_mixed_double_range_k10():
    """K = 10 (live-column cache, checked first pass): feature counts 1, 3, 8 on row counts on both sides of the K = 10 tile; data set
    1 drives exp out of the fp32 range, so its proposals take the double-range path on its own rows"""
    from mcmc_symreg_b200 import capi
    probe = H.default_engine(10, 16, 2)
    probe.set_data(np.random.default_rng(0).uniform(-3, 3, (4000, 2)), np.zeros(4000))
    tile = probe.window_geometry()["tile_rows"]
    probe.close()
    assert 900 <= tile <= 1024
    shapes = [(tile - 13, 1), (tile + 11, 3), (2 * tile + 5, 8)]
    Xs, ys = _datasets(shapes, seed=43)
    Xs[1] = np.random.default_rng(44).uniform(-100.0, 100.0, Xs[1].shape)
    ys[1] = np.sin(Xs[1][:, 0] / 20.0) + 0.01 * Xs[1][:, 2]
    batch, singles, chain_ds = _mixed_and_singles(Xs, ys, [51, 52, 53], 10, 16)
    assert batch.window_geometry()["tile_rows"] == tile
    _run([batch] + singles, "fixed", 20)
    got = _state(batch)
    for b, e in enumerate(singles):
        _assert_same_chains(got, np.nonzero(chain_ds == b)[0], _state(e))
    assert got["stats"]["counters"][chain_ds == 1, capi.CNT["fp64_sweeps"]].sum() > 0
    _close(batch, *singles)


def test_mixed_leaf_features_stay_in_range():
    """after a long run, no live or reported tree of a chain holds a leaf feature >= its data set's feature count, and the chains
    of the wide data sets use their wide columns"""
    shapes = [(200, d) for d in FEATURES]
    Xs, ys = _datasets(shapes, seed=45)
    chain_ds = np.arange(len(shapes) * 32) % len(shapes)
    eng = H.default_engine(3, chain_ds.size, 8)
    eng.set_datasets_mixed(Xs, ys, chain_ds)
    eng.init_chains(3)
    eng.run(400)
    d_of = np.asarray(FEATURES)[chain_ds]
    for current in (True, False):
        top = _leaf_features(eng.get_trees(current=current))
        assert np.all(top < d_of), (top, d_of)
    top = _leaf_features(eng.get_trees(current=True))
    assert top[d_of == 8].max() >= 5                           # columns 5 .. 7 exist for the 8-feature chains only
    assert eng.get_stats()["counters"][:, 1].sum() > 0
    eng.close()


def test_mixed_one_feature_count_is_ragged():
    """bsr_set_datasets_mixed_host with one feature count gives the chains bsr_set_datasets_ragged_host gives"""
    Xs, ys = _datasets([(n, 3) for n in (40, 100, 257, 31)], seed=46)
    cd = np.arange(4 * 16) % 4
    a = H.default_engine(3, 64, 3)
    a.set_datasets_mixed(Xs, ys, cd)
    b = H.default_engine(3, 64, 3)
    b.set_datasets_ragged(Xs, ys, cd)
    for e in (a, b):
        e.init_chains(9)
        e.run(30)
    assert a.window_geometry() == b.window_geometry()
    _assert_same_chains(_state(a), np.arange(64), _state(b))
    _close(a, b)


def test_fit_many_mixed_equals_loop_of_fits():
    """BSR.fit_many(mixed_features=True) equals a loop of cloned fits; predict_many / summarize_many over the mixed fits equal the
    per-fit methods; a test set narrower than its fit's data is refused"""
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR
    from mcmc_symreg_b200.experiments import summarize, summarize_many
    shapes = [(30, 1), (100, 5), (300, 2), (57, 8), (80, 3)]
    Xs, ys = _datasets(shapes, seed=47)
    est = BSR(3, 16, val=60)
    np.random.seed(6)
    fits = est.fit_many(list(zip(Xs, ys)), mixed_features=True)
    np.random.seed(6)
    loop = []
    for X, y in zip(Xs, ys):
        e = clone(est)
        e.fit(X, y)
        loop.append(e)
    rng = np.random.default_rng(48)
    Xt = [rng.uniform(-3, 3, (50 + 7 * b, d)) for b, (_, d) in enumerate(shapes)]
    for a, b, X in zip(fits, loop, Xt):
        _fits_equal(a, b, X)
    for method, single in (("last", lambda e, X: e.predict(X)), ("best", lambda e, X: e.predict_best(X)),
                           ("mean", lambda e, X: e.predict_mean(X))):
        got = BSR.predict_many(fits, Xt, method=method)
        for f, X, p in zip(fits, Xt, got):
            np.testing.assert_array_equal(p, single(f, X))
    mean_std = BSR.predict_many(fits, Xt, method="mean", return_std=True)
    for f, X, (m, s) in zip(fits, Xt, mean_std):
        m1, s1 = f.predict_mean(X, return_std=True)
        np.testing.assert_array_equal(m, m1)
        np.testing.assert_array_equal(s, s1)
    data = [dict(func="mixed", formula="", X=X, y=y, X_test=T, y_test=_target(T), X_extra=2 * T, y_extra=_target(2 * T))
            for X, y, T in zip(Xs, ys, Xt)]
    import json
    dump = lambda rows: [json.dumps(o, sort_keys=True, default=str) for o in rows]
    assert dump(summarize_many(fits, data)) == dump([summarize(f, d) for f, d in zip(fits, data)])
    # the 8-feature fit on a 2-column test set: its models read columns the set does not have
    wide = int(np.argmax([d for _, d in shapes]))
    narrow = list(Xt)
    narrow[wide] = Xt[wide][:, :2]
    tok = fits[wide]._packed_.tok
    assert ((tok & 0xFF) == 0).any() and ((tok >> 16)[(tok & 0xFF) == 0] >= 2).any()
    with pytest.raises(ValueError, match="reads feature"):
        BSR.predict_many(fits, narrow, method="mean")
    # one feature count: mixed_features=True is ragged=True
    Xe, ye = _datasets([(30, 2), (90, 2), (45, 2)], seed=49)
    rag = est.fit_many(list(zip(Xe, ye)), seeds=[1, 2, 3], ragged=True)
    mix = est.fit_many(list(zip(Xe, ye)), seeds=[1, 2, 3], mixed_features=True)
    for a, b in zip(rag, mix):
        _fits_equal(a, b, Xt[2])


def test_mixed_refusals():
    """what bsr_set_datasets_mixed_host refuses, what a handle of different feature counts refuses besides, and that it still works"""
    from mcmc_symreg_b200 import capi
    lib = capi.load()
    Xs, ys = _datasets([(40, 2), (60, 5)], seed=50)
    X = np.concatenate([x.ravel() for x in Xs])
    y = np.concatenate(ys)
    cd = (np.arange(8) % 2).astype(np.int32)
    eng = H.default_engine(3, 8, 5)

    def call(n_rows=(40, 60), n_features=(2, 5), chains=cd, x=X, D=2):
        nr = None if n_rows is None else np.asarray(n_rows, dtype=np.int64)
        nf = None if n_features is None else np.asarray(n_features, dtype=np.int32)
        capi._ck(lib.bsr_set_datasets_mixed_host(eng._h, D, capi._ptr(x), capi._ptr(y), capi._ptr(nr), capi._ptr(nf), capi._ptr(chains)))

    with pytest.raises(capi.BsrError, match="bsr_set_datasets_mixed_host: null argument"):
        call(n_features=None)
    with pytest.raises(capi.BsrError, match="bsr_set_datasets_mixed_host: null argument"):
        call(n_rows=None)
    with pytest.raises(capi.BsrError, match=r"n_rows\[1\] = 0: every data set needs at least one row"):
        call(n_rows=(40, 0))
    with pytest.raises(capi.BsrError, match=r"n_features\[0\] = 0 is outside 1 \.\. 65535"):
        call(n_features=(0, 5))
    with pytest.raises(capi.BsrError, match=r"n_features\[1\] = 65536 is outside 1 \.\. 65535"):
        call(n_features=(2, 65536))
    with pytest.raises(capi.BsrError, match=r"chain_dataset\[1\] = 2 is outside \[0, 2\)"):
        call(chains=np.array([0, 2, 0, 0, 0, 0, 0, 0], dtype=np.int32))
    with pytest.raises(capi.BsrError, match="n_datasets must be in"):
        call(D=0)
    with pytest.raises(capi.BsrError, match="below 2\\^32"):       # checked before any data is read: X holds 380 values
        call(n_rows=(1 << 20, 5), n_features=(2, 4096))
    eng.set_datasets_mixed(Xs, ys, cd)
    eng.init_chains(1)
    eng.run(5)
    # replacing the data under live chains: fewer features for a chain is refused, the handle keeps its data and runs on
    Xn, yn = _datasets([(40, 2), (60, 3)], seed=51)
    with pytest.raises(capi.BsrError, match="chain 1 has trees over 5 features and would get a data set of 3 features"):
        eng.set_datasets_mixed(Xn, yn, cd)
    with pytest.raises(capi.BsrError, match="would get a data set of 2 features"):
        eng.set_datasets_ragged([Xn[0], Xn[0]], [yn[0], yn[0]], cd)
    eng.run(5)
    # bsr_set_state: a leaf feature >= the chain's own feature count
    tok, pa, pb, nn = eng.get_trees(current=True)
    st = eng.get_stats()
    bad = tok.copy()
    c0 = 0                                                          # a chain of the 2-feature data set
    j = int(np.nonzero((bad[c0, 0, :nn[c0, 0]] & 0xFF) == 0)[0][0])
    bad[c0, 0, j] = (bad[c0, 0, j] & 0xFFFF) | (3 << 16)
    with pytest.raises(capi.BsrError, match="bsr_set_state: tree 0 of chain 0 reads feature 3; the chain's data set has 2 features"):
        eng.set_state(bad, pa, pb, nn, st["sigma"], st["sa"], st["sb"], seed=1)
    eng.set_state(tok, pa, pb, nn, st["sigma"], st["sa"], st["sb"], seed=1)
    # bsr_predict against the chain's own feature count
    Xt = np.random.default_rng(52).uniform(-3, 3, (20, 5))
    with pytest.raises(capi.BsrError, match="bsr_predict: feature count differs"):
        eng.predict(0, Xt)
    with pytest.raises(capi.BsrError, match="bsr_predict: feature count differs"):
        eng.predict(1, Xt[:, :2])
    tok, pa, pb, nn = eng.get_trees(current=False)
    beta = eng.get_stats()["beta"]
    for c, Xc in ((0, Xt[:, :2]), (1, Xt)):
        np.testing.assert_array_equal(eng.predict(c, Xc), capi.predict_many(0, tok[c:c + 1], pa[c:c + 1], pb[c:c + 1], nn[c:c + 1],
                                                                            beta[c:c + 1], Xc)[0])
    # the refusals of several data sets stay
    with pytest.raises(capi.BsrError, match="bsr_eval_trees: not available on a handle with several data sets"):
        eng.eval_trees(tok[0], pa[0], pb[0], nn[0])
    for fn in (eng.sweep_propose, eng.sweep_eval, eng.sweep_resolve):
        with pytest.raises(capi.BsrError, match="not available on a handle with several data sets"):
            fn()
    eng.run(5)                                                      # bsr_run itself works
    assert np.all(_leaf_features(eng.get_trees(current=True)) < np.array([2, 5])[cd])
    # more features for every chain is accepted: the chains are refitted on the new data
    Xw, yw = _datasets([(40, 3), (60, 6)], seed=53)
    eng.set_datasets_mixed(Xw, yw, cd)
    eng.run(5)
    eng.close()
    rs = capi.Engine(3, 8, list(range(1, 11)), [0.1] * 10, row_sharded=True)
    with pytest.raises(capi.BsrError, match="bsr_set_datasets_mixed_host: not available on row-sharded handles"):
        rs.set_datasets_mixed(Xs, ys, cd)
    rs.close()
    seq = H.default_engine(3, 8, 2)
    seq.set_pipeline(True)
    with pytest.raises(capi.BsrError, match="proposal-by-proposal pipeline"):
        seq.set_datasets_mixed(Xs, ys, cd)
    seq.close()
