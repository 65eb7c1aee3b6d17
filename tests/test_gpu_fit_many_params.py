"""GPU tests of per-chain priors (bsr_set_chain_priors) and of BSR.fit_many(params=...): every chain of a batch of several operator
sets, split exponents and stop rules ends bit for bit where the chain of a handle created with its own prior (and holding only its
own data set) ends, keyed the same way."""
import numpy as np
import pytest

from test_gpu_fit_many import _assert_same_chains, _fits_equal, _state
from test_gpu_fit_many_mixed import _datasets

pytestmark = pytest.mark.gpu

DEFAULT = dict(ops=list(range(1, 11)), op_weights=[0.1] * 10)
OPS7 = dict(ops=[9, 10, 4, 5, 6, 7, 2], op_weights=[0.3, 0.2, 0.1, 0.1, 0.1, 0.1, 0.1])    # +, *, sin, cos, exp, square, lt
OPS3 = dict(ops=[9, 10, 5], op_weights=[0.4, 0.4, 0.2])                                  # +, *, cos
PRIORS = [dict(DEFAULT, beta=-1.0, val=100, plateau_rule=True), dict(DEFAULT, beta=-0.5, val=50, plateau_rule=False),
          dict(DEFAULT, beta=-2.0, val=0, plateau_rule=True), dict(OPS7, beta=-1.0, val=100, plateau_rule=False),
          dict(OPS3, beta=-0.5, val=0, plateau_rule=False), dict(OPS7, beta=-2.0, val=50, plateau_rule=True)]
SHAPES = dict(ragged=[(40, 2), (97, 2), (300, 2)], mixed=[(40, 1), (97, 3), (300, 5)])


def _engine(K, C, prior, precision="fp32"):
    from mcmc_symreg_b200 import capi
    return capi.Engine(K, C, prior["ops"], prior["op_weights"], beta=prior["beta"], val=prior["val"], plateau_rule=prior["plateau_rule"],
                       precision=precision)


def _upload(eng, kind, Xs, ys, chain_ds):
    if kind == "ragged":
        eng.set_datasets_ragged(Xs, ys, chain_ds)
    else:
        eng.set_datasets_mixed(Xs, ys, chain_ds)


def _run(engines, mode):
    for e in engines:
        if mode == "fixed":
            e.run(30)
        else:
            e.run_until_done(400, check_every=32)


def _grid_and_singles(kind, Xs, ys, priors, K, C, precision, layout):
    """a batch of every (data set, prior) entry, C chains each, and one handle per entry"""
    entries = [(b, q) for b in range(len(Xs)) for q in range(len(priors))]
    E = len(entries)
    if layout == "contiguous":
        entry, ids = np.repeat(np.arange(E), C), np.tile(np.arange(C), E)
    else:
        entry, ids = np.arange(E * C) % E, np.arange(E * C) // E
    ent = np.asarray(entries)
    seeds = 11 * np.arange(1, E + 1)
    batch = _engine(K, E * C, priors[0], precision)
    batch.set_chain_priors(priors, ent[entry, 1])
    _upload(batch, kind, Xs, ys, ent[entry, 0])
    batch.init_chains_keyed(seeds[entry], ids)
    singles = []
    for e, (b, q) in enumerate(entries):
        s = _engine(K, C, priors[q], precision)
        s.set_data(Xs[b], ys[b])
        s.init_chains(int(seeds[e]))
        singles.append(s)
    return batch, singles, entry


def _close(*engines):
    for e in engines:
        e.close()


@pytest.mark.parametrize("kind", ["ragged", "mixed"])
@pytest.mark.parametrize("layout", ["contiguous", "interleaved"])
@pytest.mark.parametrize("mode", ["fixed", "until"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_priors_match_single_handles(precision, mode, layout, kind):
    """3 data sets x 6 priors (beta -1 / -0.5 / -2, 10 / 7 / 3 operators, val 0 / 50 / 100, plateau on / off), 16 chains each: every
    chain equals its own single handle, bit for bit -- trees, betas, sigmas, counters, done and RMSE traces"""
    from mcmc_symreg_b200 import capi
    Xs, ys = _datasets(SHAPES[kind], seed=61)
    batch, singles, entry = _grid_and_singles(kind, Xs, ys, PRIORS, 3, 16, precision, layout)
    _run([batch] + singles, mode)
    got = _state(batch)
    exec_col = capi.CNT["node_evals_exec"]
    for e, s in enumerate(singles):
        rows, want = np.nonzero(entry == e)[0], _state(s)
        if s.window_geometry()["ring"] != batch.window_geometry()["ring"]:
            # the ring depth sizes the record cache (2 when every chain has val > 0): it changes how many trees are interpreted,
            # nothing else
            want["stats"]["counters"][:, exec_col] = got["stats"]["counters"][rows, exec_col]
        _assert_same_chains(got, rows, want)
    assert batch.window_geometry()["ring"] == 8 and singles[0].window_geometry()["ring"] == 2
    done = got["stats"]["done"]
    assert got["stats"]["counters"][:, 1].sum() > 0
    if mode == "until":     # the stop rules differ: val = 0 without plateau never stops, val = 50 stops
        q = entry % len(PRIORS)
        assert not done[q == 4].any() and done[q == 1].any()
    _close(batch, *singles)


def test_one_prior_explicit_is_no_call():
    """one prior passed explicitly (once, or twice under two indices) gives the bits of a handle without the call"""
    Xs, ys = _datasets([(60, 2), (150, 2)], seed=62)
    cd = np.arange(64) % 2
    p = dict(DEFAULT, beta=-1.0, val=100, plateau_rule=True)
    engines = [_engine(3, 64, p) for _ in range(3)]
    engines[1].set_chain_priors([p], np.zeros(64))
    engines[2].set_chain_priors([p, dict(p)], np.arange(64) % 2)
    for e in engines:
        e.set_datasets_ragged(Xs, ys, cd)
        e.init_chains(5)
        e.run_until_done(400, check_every=32)
    ref = _state(engines[0])
    for e in engines[1:]:
        _assert_same_chains(_state(e), np.arange(64), ref)
    _close(*engines)


def _operators_in_set(trees, entry, priors):
    """every operator token of every chain's trees is in its prior's operator set and its op_ind below the set's size"""
    tok, _, _, nn = trees
    tok = tok.astype(np.int64)
    used = np.arange(tok.shape[2])[None, None, :] < nn[:, :, None]
    op, oi = tok & 0xFF, (tok >> 8) & 0xFF
    for c in range(tok.shape[0]):
        p = priors[entry[c]]
        sel = used[c] & (op[c] != 0)
        assert np.isin(op[c][sel], p["ops"]).all(), (c, np.unique(op[c][sel]), p["ops"])
        assert (oi[c][sel] < len(p["ops"])).all()
    return op, used


def test_long_run_keeps_every_chain_in_its_operator_set():
    Xs, ys = _datasets([(200, 2)], seed=63)
    priors = [dict(p, val=0, plateau_rule=False) for p in PRIORS]
    entry = np.arange(6 * 32) % 6
    eng = _engine(3, entry.size, priors[0])
    eng.set_chain_priors(priors, entry)
    eng.set_data(Xs[0], ys[0])
    eng.init_chains(3)
    eng.run(400)
    for current in (True, False):
        op, used = _operators_in_set(eng.get_trees(current=current), entry, priors)
    assert (op[entry == 4][used[entry == 4]] == 5).any()          # cos, the only unary operator of the 3-operator set, is used
    assert eng.get_stats()["counters"][:, 1].sum() > 0
    eng.close()


def test_fit_many_params_equals_loop_of_fits(monkeypatch):
    """fit_many(params=...) equals the clone-and-fit loop entry by entry; entries of the same (X, y) objects share one data set;
    predict_many / summarize_many on the grid's fits equal the per-fit methods"""
    import json
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR, capi
    from mcmc_symreg_b200.experiments import summarize, summarize_many
    uploads = []
    real = capi.Engine.set_datasets

    def spy(self, X, y, chain_dataset):
        uploads.append(np.asarray(X).shape[0])
        return real(self, X, y, chain_dataset)
    monkeypatch.setattr(capi.Engine, "set_datasets", spy)
    Xs, ys = _datasets([(80, 2), (80, 2)], seed=64)
    grid = [dict(beta=-1.0), dict(beta=-0.5, val=40, ops=["+", "*", "cos"], op_weights=[0.4, 0.4, 0.2]),
            dict(beta=-2.0, plateau_rule=False, ops=["+", "*", "sin", "cos", "exp", "square", "ln"],
                 op_weights=[0.3, 0.2, 0.1, 0.1, 0.1, 0.1, 0.1])]
    pairs = [(Xs[f], ys[f]) for f in range(2) for _ in grid]
    params = [p for _ in range(2) for p in grid]
    est = BSR(3, 16, val=60)
    np.random.seed(8)
    fits = est.fit_many(pairs, params=params)
    np.random.seed(8)
    loop = []
    for (X, y), p in zip(pairs, params):
        e = clone(est).set_params(**p)
        e.fit(X, y)
        loop.append(e)
    assert uploads == [2]                                            # two folds, not six entries
    rng = np.random.default_rng(65)
    Xt = [rng.uniform(-3, 3, (40 + 3 * b, 2)) for b in range(len(pairs))]
    for a, b, X, p in zip(fits, loop, Xt, params):
        _fits_equal(a, b, X)
        assert a.get_params() == b.get_params()
    for method, single in (("last", lambda e, X: e.predict(X)), ("best", lambda e, X: e.predict_best(X)),
                           ("mean", lambda e, X: e.predict_mean(X))):
        for f, X, got in zip(fits, Xt, BSR.predict_many(fits, Xt, method=method)):
            np.testing.assert_array_equal(got, single(f, X))
    data = [dict(func="grid", formula="", X=X, y=y, X_test=T, y_test=T[:, 0], X_extra=2 * T, y_extra=2 * T[:, 0])
            for (X, y), T in zip(pairs, Xt)]
    dump = lambda rows: [json.dumps(o, sort_keys=True, default=str) for o in rows]
    assert dump(summarize_many(fits, data)) == dump([summarize(f, d) for f, d in zip(fits, data)])
    # one fold under three settings: the handle holds one data set
    uploads.clear()
    fits = est.fit_many(pairs[:3], seeds=[1, 2, 3], params=grid)
    assert uploads == [1] and len(fits) == 3


def test_chain_prior_refusals():
    """what bsr_set_chain_priors refuses (the previous priors stay), what a handle of several priors refuses, and that it works on"""
    import ctypes
    from mcmc_symreg_b200 import capi
    lib = capi.load()
    Xs, ys = _datasets([(60, 2)], seed=66)
    C = 8
    cp = (np.arange(C) % 2).astype(np.int32)
    two = [PRIORS[0], PRIORS[4]]
    eng = _engine(3, C, PRIORS[0])
    eng.set_chain_priors(two, cp)

    def call(priors=two, chains=cp, n=None):
        arr = (capi.BsrPrior * max(1, len(priors)))()
        for p, d in zip(arr, priors):
            p.n_ops = d.get("n_ops", len(d["ops"]))
            for i, (o, w) in enumerate(zip(d["ops"], d["op_weights"])):
                p.ops[i], p.op_weights[i] = o, w
            p.beta, p.val, p.plateau_rule = d["beta"], d["val"], int(d["plateau_rule"])
        capi._ck(lib.bsr_set_chain_priors(eng._h, len(priors) if n is None else n, ctypes.cast(arr, capi._P), capi._ptr(chains)))

    with pytest.raises(capi.BsrError, match="bsr_set_chain_priors: null argument"):
        capi._ck(lib.bsr_set_chain_priors(eng._h, 1, None, capi._ptr(cp)))
    with pytest.raises(capi.BsrError, match="bsr_set_chain_priors: null argument"):
        call(chains=None)
    with pytest.raises(capi.BsrError, match="n_priors must be >= 1"):
        call(n=0)
    bad = dict(PRIORS[0])
    for change, msg in ((dict(n_ops=0), r"priors\[1\]: n_ops must be in \[1, 16\]"), (dict(n_ops=17), r"priors\[1\]: n_ops must be in"),
                        (dict(ops=[11, 10], op_weights=[0.5, 0.5]), r"priors\[1\]: unknown opcode"),
                        (dict(ops=[9, 10], op_weights=[1.5, -0.5]), r"priors\[1\]: operator weights must be positive"),
                        (dict(ops=[9, 10], op_weights=[0.5, 0.6]), r"priors\[1\]: operator weights must sum to 1")):
        with pytest.raises(capi.BsrError, match=msg):
            call(priors=[PRIORS[1], dict(bad, **change)])
    with pytest.raises(capi.BsrError, match=r"chain_prior\[3\] = 2 is outside \[0, 2\)"):
        call(chains=np.array([0, 1, 0, 2, 0, 0, 0, 0], dtype=np.int32))
    with pytest.raises(capi.BsrError, match=r"chain_prior\[0\] = -1 is outside"):
        call(chains=np.array([-1, 1, 0, 0, 0, 0, 0, 0], dtype=np.int32))
    # the refused calls left `two` in place: the handle runs as a fresh handle of `two`
    ref = _engine(3, C, PRIORS[0])
    ref.set_chain_priors(two, cp)
    for e in (eng, ref):
        e.set_data(Xs[0], ys[0])
        e.init_chains(4)
        e.run(20)
    _assert_same_chains(_state(eng), np.arange(C), _state(ref))
    ref.close()
    with pytest.raises(capi.BsrError, match="the chains are initialised"):
        call()
    # several priors: the refusals of several data sets
    tok, pa, pb, nn = eng.get_trees(current=True)
    with pytest.raises(capi.BsrError, match="bsr_eval_trees: not available on a handle with several priors"):
        eng.eval_trees(tok[0], pa[0], pb[0], nn[0])
    for fn in (eng.sweep_propose, eng.sweep_eval, eng.sweep_resolve):
        with pytest.raises(capi.BsrError, match="not available on a handle with several priors"):
            fn()
    with pytest.raises(capi.BsrError, match="bsr_peer_export: not available on a handle with several priors"):
        eng.peer_export(1)
    with pytest.raises(capi.BsrError, match="bsr_set_pipeline: not available on a handle with several priors"):
        eng.set_pipeline(True)
    # bsr_set_state: an operator outside its chain's set, an op_ind past its chain's operators (chain 1 has 3 operators)
    st = eng.get_stats()
    op = tok.astype(np.int64) & 0xFF
    j = int(np.nonzero(op[1, 0, :nn[1, 0]] != 0)[0][0])
    bad_tok = tok.copy()
    bad_tok[1, 0, j] = (tok[1, 0, j] & ~np.uint32(0xFF)) | np.uint32(3)           # neg: not in {+, *, cos}
    with pytest.raises(capi.BsrError, match="bsr_set_state: tree 0 of chain 1 holds opcode 3, which is not in the chain's operator set"):
        eng.set_state(bad_tok, pa, pb, nn, st["sigma"], st["sa"], st["sb"], seed=1)
    bad_tok = tok.copy()
    bad_tok[1, 0, j] = (tok[1, 0, j] & ~np.uint32(0xFF00)) | np.uint32(5 << 8)
    with pytest.raises(capi.BsrError, match="bsr_set_state: tree 0 of chain 1 has op_ind 5; the chain's prior has 3 operators"):
        eng.set_state(bad_tok, pa, pb, nn, st["sigma"], st["sa"], st["sb"], seed=1)
    eng.set_state(tok, pa, pb, nn, st["sigma"], st["sa"], st["sb"], seed=1)
    eng.run(10)
    _operators_in_set(eng.get_trees(current=True), cp, two)
    eng.close()
    rs = capi.Engine(3, C, list(range(1, 11)), [0.1] * 10, row_sharded=True)
    with pytest.raises(capi.BsrError, match="bsr_set_chain_priors: not available on row-sharded handles"):
        rs.set_chain_priors(two, cp)
    rs.close()
    seq = _engine(3, C, PRIORS[0])
    seq.set_pipeline(True)
    with pytest.raises(capi.BsrError, match="several priors need the window path of bsr_run"):
        seq.set_chain_priors(two, cp)
    seq.set_chain_priors([PRIORS[1]], np.zeros(C))                  # one prior: the pipeline reads it
    seq.set_data(Xs[0], ys[0])
    seq.init_chains(2)
    seq.run(5)
    seq.close()
