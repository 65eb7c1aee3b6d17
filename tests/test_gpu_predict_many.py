"""GPU tests of grouped prediction (bsr_predict_groups, capi.predict_groups, BSR.predict_many, experiments.summarize_many): every
value of the multi-fit route is bit for bit what the single-fit route returns (the single-estimator methods, and bsr_predict_many
on dense models), across grouping, set offsets, row chunks, packing, non-finite models and more models than one launch dimension
holds; malformed tables are refused before the device reads them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FUNCS = ("f1", "f2", "f3", "f4", "f5", "f6")
MM = 16                                   # restarts per fit


def _datasets(sizes, seed):
    from mcmc_symreg_b200.experiments import TARGETS
    rng = np.random.default_rng(seed)
    Xs = [rng.uniform(-3, 3, (n, 2)) for n in sizes]
    return [(X, TARGETS[FUNCS[b % len(FUNCS)]][0](X)) for b, X in enumerate(Xs)]


@pytest.fixture(scope="module")
def fits():
    from mcmc_symreg_b200 import BSR
    return BSR(3, MM, val=60).fit_many(_datasets((30, 100, 57, 80, 41), seed=51), seeds=[1, 2, 3, 4, 5], ragged=True)


def _chunk_rows(models_reduced):
    """rows per chunk of bsr_predict_groups when `models_reduced` models are reduced in one call (bsr_capi.cu)"""
    return max(256, (32 << 20) // models_reduced) // 2 * 2


def _test_sets(n_fits, seed, big):
    """1 row, an odd count, more than 256 rows, more than one chunk of rows, then more of the small sizes"""
    rng = np.random.default_rng(seed)
    sizes = [1, 77, 301, big] + [5, 130, 2, 999][:n_fits - 4]
    return [rng.uniform(-4, 4, (n, 2)) for n in sizes]


def test_methods_bit_identical(fits):
    from mcmc_symreg_b200 import BSR
    big = _chunk_rows(MM * len(fits)) + 1001
    Xs = _test_sets(len(fits), 52, big)
    for last_ind in (1, 3):
        got = BSR.predict_many(fits, Xs, last_ind=last_ind)
        for f, X, g in zip(fits, Xs, got):
            assert g.shape == (X.shape[0], 1)
            np.testing.assert_array_equal(g, f.predict(X, last_ind=last_ind))
    for f, X, g in zip(fits, Xs, BSR.predict_many(fits, Xs, method="best")):
        np.testing.assert_array_equal(g, f.predict_best(X))
    want = []
    for f, X in zip(fits, Xs):
        want.append(f.predict_mean(X, return_std=True) + (f.n_used_,))
        f.n_used_ = None
    got = BSR.predict_many(fits, Xs, method="mean", return_std=True)
    for f, (m, s), (wm, ws, wu) in zip(fits, got, want):
        np.testing.assert_array_equal(m, wm)
        np.testing.assert_array_equal(s, ws)
        assert f.n_used_ == wu
    for f, m, (wm, _, _) in zip(fits, BSR.predict_many(fits, Xs, method="mean"), want):
        np.testing.assert_array_equal(m, wm)


def test_non_finite_models(fits):
    """test sets with entries near 1e120 (and beyond 1e154, where a square overflows): some models are not finite on some rows, the
    mean and std leave them out exactly as predict_mean does, and n_used_ drops"""
    from mcmc_symreg_b200 import BSR, capi
    rng = np.random.default_rng(53)
    Xs = []
    for f in fits:
        X = rng.uniform(-3, 3, (40, 2))
        X[::3, 0] = 1e120 * rng.choice([-1.0, 1.0], X[::3].shape[0])
        X[1::5, 1] = 3e154
        Xs.append(X)
    per_model = [capi.predict_many(0, *f._enc_, np.stack(f.betas_)[:, :, 0], X) for f, X in zip(fits, Xs)]
    assert any(not np.all(np.isfinite(p)) for p in per_model)                 # the case is really exercised
    want = []
    for f, X in zip(fits, Xs):
        want.append(f.predict_mean(X, return_std=True) + (f.n_used_,))
    assert min(w[2] for w in want) < MM
    got = BSR.predict_many(fits, Xs, method="mean", return_std=True)
    for f, (m, s), (wm, ws, wu) in zip(fits, got, want):
        np.testing.assert_array_equal(m, wm)
        np.testing.assert_array_equal(s, ws)
        assert f.n_used_ == wu
    for f, X, g in zip(fits, Xs, BSR.predict_many(fits, Xs, last_ind=2)):
        np.testing.assert_array_equal(g, f.predict(X, last_ind=2))


def test_summarize_many_equals_summarize(fits):
    import json
    from mcmc_symreg_b200.experiments import make_dataset, summarize, summarize_many
    data = [make_dataset(FUNCS[b], 50, 30, seed=60 + b) for b in range(len(fits))]
    loop = [summarize(f, d) for f, d in zip(fits, data)]
    used = [f.n_used_ for f in fits]
    for f in fits:
        f.n_used_ = None
    many = summarize_many(fits, data)
    assert [json.dumps(o, sort_keys=True, default=str) for o in loop] == [json.dumps(o, sort_keys=True, default=str) for o in many]
    assert [f.n_used_ for f in fits] == used


def _tiled(fits, M, seed):
    """M models cycling through the restarts of the fits, each with its own betas"""
    from mcmc_symreg_b200 import capi
    pk = capi.PackedTrees.concat([f._packed_ for f in fits])
    n = pk.nn.shape[0]
    reps = -(-M // n)
    nn = np.tile(pk.nn, (reps, 1))[:M]
    n_tok = int(nn.sum())
    tok = np.tile(pk.tok, reps)[:n_tok]
    n_lt = int(np.count_nonzero((tok & 0xFF) == 2))
    ab = np.tile(pk.ab, (reps, 1))[:n_lt]
    beta = np.concatenate([np.stack(f.betas_)[:, :, 0] for f in fits])
    beta = np.tile(beta, (reps, 1))[:M] * (1 + 0.01 * np.random.default_rng(seed).normal(size=(M, nn.shape[1] + 1)))
    return nn, tok, ab, beta


def test_more_models_than_one_launch_dimension(fits):
    """70000 models in one plain and one reducing group, on enough rows that the reduction runs in several chunks: the plain block
    equals capi.predict_many over all the models and over slices of at most 65535 models bit for bit, the reduction a float64 numpy
    mean / std to 1e-12"""
    from mcmc_symreg_b200 import capi
    M = 70000
    nn, tok, ab, beta = _tiled(fits, M, 54)
    rows = _chunk_rows(M) + 97
    assert _chunk_rows(M) < rows
    rng = np.random.default_rng(55)
    X, X2 = rng.uniform(-3, 3, (rows, 2)), rng.uniform(-3, 3, (3, 2))
    small = np.arange(5, M, 9000)
    blocks, used = capi.predict_groups(0, nn, tok, ab, beta, [X2, X], [1, 1, 0], [np.arange(M), np.arange(M), small], [False, True, False])
    assert [b.shape for b in blocks] == [(M, rows), (2, rows), (small.size, 3)]
    assert list(used) == [M, M, small.size]
    dense = capi.PackedTrees(nn, tok, ab).dense()
    np.testing.assert_array_equal(blocks[0], capi.predict_many(0, *dense, beta, X))
    for lo in range(0, M, 65535):
        hi = min(M, lo + 65535)
        want = capi.predict_many(0, dense[0][lo:hi], dense[1][lo:hi], dense[2][lo:hi], dense[3][lo:hi], beta[lo:hi], X)
        np.testing.assert_array_equal(blocks[0][lo:hi], want)
    np.testing.assert_array_equal(blocks[2], capi.predict_many(0, dense[0][small], dense[1][small], dense[2][small], dense[3][small],
                                                               beta[small], X2))
    assert np.all(np.isfinite(blocks[0]))
    scale = 1e-12 * float(np.abs(blocks[0]).max())          # rows where the models' predictions cancel
    np.testing.assert_allclose(blocks[1][0], blocks[0].mean(axis=0), rtol=1e-12, atol=scale)
    np.testing.assert_allclose(blocks[1][1], blocks[0].std(axis=0, ddof=1), rtol=1e-12, atol=scale)


def test_refusals(fits):
    """each malformed table is refused with BsrError before the device reads it, and the library stays usable"""
    from mcmc_symreg_b200 import capi
    lib = capi.load()
    pk = capi.PackedTrees.concat([f._packed_ for f in fits[:2]])
    M, K = pk.nn.shape
    beta = np.concatenate([np.stack(f.betas_)[:, :, 0] for f in fits[:2]])
    Xs = [np.random.default_rng(56).uniform(-3, 3, (n, 2)) for n in (9, 4)]
    X = np.ascontiguousarray(np.concatenate(Xs))
    base = dict(M=M, K=K, nn=pk.nn.astype(np.int32), tok=pk.tok.astype(np.uint32), n_tok=pk.tok.size, ab=np.ascontiguousarray(pk.ab),
                n_lt=pk.ab.shape[0], beta=beta, S=2, d=2, X=X, set_off=np.array([0, 9, 13], np.int64), G=2,
                grp_set=np.array([0, 1], np.int32), grp_off=np.array([0, 3, 3 + M], np.int64),
                grp_models=np.concatenate([[0, 5, 7], np.arange(M)]).astype(np.int32), grp_reduce=np.array([0, 1], np.int32))

    def call(**over):
        a = dict(base, **over)
        out = np.zeros(3 * 9 + 2 * 4)
        used = np.zeros(2, np.int32)
        p = lambda v: None if v is None else capi._ptr(np.ascontiguousarray(v))
        capi._ck(lib.bsr_predict_groups(0, a["M"], a["K"], p(a["nn"]), p(a["tok"]), a["n_tok"], p(a["ab"]), a["n_lt"], p(a["beta"]), a["S"],
                                        a["d"], p(a["X"]), p(a["set_off"]), a["G"], p(a["grp_set"]), p(a["grp_off"]), p(a["grp_models"]),
                                        p(a["grp_reduce"]), capi._ptr(out), capi._ptr(used)))
        return out, used

    ok = call()
    blocks, used = capi.predict_groups(0, pk.nn, pk.tok, pk.ab, beta, Xs, [0, 1], [[0, 5, 7], np.arange(M)], [False, True])
    np.testing.assert_array_equal(ok[0], np.concatenate([b.ravel() for b in blocks]))
    leaf = int(np.nonzero((pk.tok & 0xFF) == 0)[0][0])
    lt = int(np.nonzero((pk.tok & 0xFF) == 2)[0][0])
    cases = [
        ("null argument", dict(nn=None)),
        ("bad shape", dict(K=0)),
        ("bad shape", dict(K=17)),
        ("tree size out of range", dict(nn=_set(base["nn"], (0, 0), 0))),
        ("tree size out of range", dict(nn=_set(base["nn"], (1, 2), 65))),
        ("more tokens than tok holds", dict(n_tok=base["n_tok"] - 1)),
        ("fewer tokens than tok holds", dict(n_tok=base["n_tok"] + 1, tok=np.append(base["tok"], 0).astype(np.uint32))),
        ("differ in number", dict(n_lt=base["n_lt"] - 1)),
        ("differ in number", dict(tok=_set(base["tok"], lt, 3))),                      # an lt node turned into neg: one pair too many
        ("reads a feature the data does not have", dict(tok=_set(base["tok"], leaf, 5 << 16))),
        ("unknown opcode", dict(tok=_set(base["tok"], leaf, 11))),
        ("not a pre-order tree", dict(tok=_set(base["tok"], leaf, 9))),                # a leaf turned into +
        ("set_off decreases", dict(set_off=np.array([0, 9, 8], np.int64))),
        ("test set 1 has no rows", dict(set_off=np.array([0, 9, 9], np.int64))),
        (r"set_off\[0\] must be 0", dict(set_off=np.array([1, 9, 13], np.int64))),
        ("grp_off decreases", dict(grp_off=np.array([0, 3, 2], np.int64))),
        ("group 0 has no models", dict(grp_off=np.array([0, 0, M], np.int64))),
        (r"grp_models\[1\] is outside \[0, M\)", dict(grp_models=_set(base["grp_models"], 1, M))),
        (r"grp_models\[0\] is outside \[0, M\)", dict(grp_models=_set(base["grp_models"], 0, -1))),
        (r"grp_set\[1\] is outside \[0, S\)", dict(grp_set=np.array([0, 2], np.int32))),
        (r"grp_set\[0\] is outside \[0, S\)", dict(grp_set=np.array([-1, 0], np.int32))),
    ]
    for match, over in cases:
        with pytest.raises(capi.BsrError, match="bsr_predict_groups: .*" + match):
            call(**over)
    again = call()
    np.testing.assert_array_equal(again[0], ok[0])
    np.testing.assert_array_equal(again[1], ok[1])


def _set(a, i, v):
    a = a.copy()
    a[i] = v
    return a
