"""Host logic of a grid of prior settings in one run that needs no GPU: BSR.fit_many(params=...)'s checks before any library call,
the priors and chain -> prior map it hands capi.Engine.set_chain_priors, the uploads shared by entries of the same (X, y) objects,
the overrides every returned estimator carries, and experiments.run_suite / --beta over such a grid."""
import numpy as np
import pytest

from mcmc_symreg_b200 import BSR, capi
from mcmc_symreg_b200.trees import DEFAULT_OPS, NAME_OP


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(capi, "load", refuse)
    monkeypatch.setattr(capi, "Engine", refuse)


def _data(n_sets, n=20, d=2, seed=0):
    rng = np.random.default_rng(seed)
    return [(rng.normal(size=(n, d)), rng.normal(size=n)) for _ in range(n_sets)]


@pytest.mark.parametrize("params, match", [
    ([dict(beta=-1.0)], r"^fit_many: 1 params for 2 data sets$"),
    ([dict(beta=-1.0), dict(treeNum=4)], r"params\[1\] sets 'treeNum', which every entry of one run shares"),
    ([dict(itrNum=3), dict()], r"params\[0\] sets 'itrNum'"),
    ([dict(), dict(precision="fp64")], r"params\[1\] sets 'precision'"),
    ([dict(), dict(fixed_sweeps=10)], r"params\[1\] sets 'fixed_sweeps'"),
    ([dict(), dict(max_sweeps=10)], r"params\[1\] sets 'max_sweeps'"),
    ([dict(), dict(err_cap=10)], r"params\[1\] sets 'err_cap'"),
    ([dict(), dict(device=1)], r"params\[1\] sets 'device'"),
    ([dict(), dict(distributed=True)], r"params\[1\] sets 'distributed'"),
    ([dict(), dict(seed=3)], r"params\[1\] sets 'seed'"),
    ([dict(gamma=1.0), dict()], r"params\[0\] sets 'gamma', which is not a parameter of BSR"),
    ([dict(ops=["+", "*", "tan"]), dict()], r"params\[0\]: unknown operator 'tan'"),
    ([dict(), dict(ops=["+", "*"], op_weights=[1.0])], r"params\[1\]: 2 operators and 1 op_weights"),
    ([dict(), dict(ops=["+", "*", "sin"])], r"params\[1\]: 3 operators and 2 op_weights"),
])
def test_params_errors_before_any_library_call(no_library, params, match):
    est = BSR(3, 4, seed=1, ops=["+", "*"], op_weights=[0.5, 0.5])
    with pytest.raises(ValueError, match=match):
        est.fit_many(_data(2), params=params)


def test_old_messages_unchanged(no_library):
    with pytest.raises(ValueError, match=r"^fit_many: no data sets$"):
        BSR(3, 4, seed=1).fit_many([], params=[])
    with pytest.raises(ValueError, match=r"^fit_many: data set 1 is 10 x 3, data set 0 is 10 x 2: all data sets must have the same shape$"):
        BSR(3, 4, seed=1).fit_many([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 3)), np.zeros(10))], params=[{}, {}])
    with pytest.raises(ValueError, match=r"^fit_many: 3 seeds for 2 data sets$"):
        BSR(3, 4).fit_many(_data(2), seeds=[1, 2, 3], params=[{}, {}])


class _FakeEngine:
    """records what fit_many hands the engine and returns a result of single-leaf trees"""
    calls = []

    def __init__(self, K, C, ops, w, **kw):
        self.K, self.C = K, C
        self.log = dict(init=dict(K=K, C=C, ops=list(ops), w=list(w), **kw))
        _FakeEngine.calls.append(self.log)

    def set_chain_priors(self, priors, chain_prior):
        self.log["priors"] = [dict(p) for p in priors]
        self.log["chain_prior"] = np.asarray(chain_prior).copy()

    def set_datasets(self, X, y, chain_dataset):
        self.log["upload"] = ("same_shape", [x for x in X], np.asarray(chain_dataset).copy())

    def set_datasets_ragged(self, Xs, ys, chain_dataset):
        self.log["upload"] = ("ragged", list(Xs), np.asarray(chain_dataset).copy())

    def set_datasets_mixed(self, Xs, ys, chain_dataset):
        self.log["upload"] = ("mixed", list(Xs), np.asarray(chain_dataset).copy())

    def init_chains_keyed(self, seeds, ids):
        self.log["keys"] = (np.asarray(seeds).copy(), np.asarray(ids).copy())

    def run(self, n):
        self.log["run"] = n

    def run_until_done(self, max_sweeps, check_every=16):
        self.log["run_until_done"] = max_sweeps
        return 32

    def get_trees_packed(self, current=False):
        return capi.PackedTrees(np.ones((self.C, self.K), dtype=np.int32), np.zeros(self.C * self.K, dtype=np.uint32), np.zeros((0, 2)))

    def get_stats(self):
        C, K = self.C, self.K
        return dict(beta=np.zeros((C, K + 1)), sigma=np.ones(C), sa=np.ones((C, K)), sb=np.ones((C, K)), sse=np.ones(C),
                    counters=np.zeros((C, capi.N_COUNTERS), dtype=np.int64), done=np.ones(C, dtype=np.int32), nerr=np.zeros(C, dtype=np.int32))

    def get_err_trace(self):
        return np.zeros((self.C, 4))

    def close(self):
        pass


@pytest.fixture
def fake_engine(monkeypatch):
    _FakeEngine.calls = []
    monkeypatch.setattr(capi, "Engine", _FakeEngine)
    return _FakeEngine.calls


OPS7 = dict(ops=["+", "*", "sin", "cos", "exp", "square", "ln"], op_weights=[0.3, 0.2, 0.1, 0.1, 0.1, 0.1, 0.1])


def test_priors_and_chain_map_handed_to_the_engine(fake_engine):
    data = _data(2)
    grid = [dict(beta=-1.0), dict(beta=-0.5, val=50), dict(beta=-2.0, plateau_rule=False, **OPS7)]
    pairs = [data[f] for f in range(2) for _ in grid]               # the same (X, y) objects for every setting of a fold
    params = [p for _ in range(2) for p in grid]
    MM = 4
    fits = BSR(3, MM, val=100).fit_many(pairs, seeds=list(range(6)), params=params)
    log = fake_engine[0]
    default = dict(ops=[NAME_OP[o] for o in DEFAULT_OPS], op_weights=[0.1] * 10)
    want = [dict(default, beta=-1.0, val=100, plateau_rule=True), dict(default, beta=-0.5, val=50, plateau_rule=True),
            dict(ops=[NAME_OP[o] for o in OPS7["ops"]], op_weights=OPS7["op_weights"], beta=-2.0, val=100, plateau_rule=False)] * 2
    assert log["priors"] == want
    np.testing.assert_array_equal(log["chain_prior"], np.repeat(np.arange(6), MM))
    kind, Xs, chain_ds = log["upload"]
    assert kind == "same_shape" and len(Xs) == 2                     # two folds uploaded, not six entries
    np.testing.assert_array_equal(Xs[0], data[0][0])
    np.testing.assert_array_equal(Xs[1], data[1][0])
    np.testing.assert_array_equal(chain_ds, np.repeat([0, 0, 0, 1, 1, 1], MM))
    np.testing.assert_array_equal(log["keys"][0], np.repeat(np.arange(6), MM))
    np.testing.assert_array_equal(log["keys"][1], np.tile(np.arange(MM), 6))
    assert len(fits) == 6
    for e, p in zip(fits, params):
        got = e.get_params()
        for k, v in p.items():
            assert got[k] == v, (k, got[k], v)
        assert got["treeNum"] == 3 and got["itrNum"] == MM
        assert len(e.betas_) == MM


def test_shared_uploads_compare_identity_not_value(fake_engine):
    X, y = _data(1)[0]
    pairs = [(X, y), (X.copy(), y), (X, y), (X, y.copy()), (X, y)]  # equal values, different objects: uploaded again
    BSR(3, 2, seed=1).fit_many(pairs, ragged=True)
    kind, Xs, chain_ds = fake_engine[0]["upload"]
    assert kind == "ragged" and len(Xs) == 3
    np.testing.assert_array_equal(chain_ds, np.repeat([0, 1, 0, 2, 0], 2))
    assert "priors" not in fake_engine[0]                           # params=None: no per-chain priors


def test_fixed_sweeps_turn_every_stop_rule_off(fake_engine):
    data = _data(2)
    fits = BSR(3, 2, seed=1, fixed_sweeps=5).fit_many(data, params=[dict(val=30, plateau_rule=True), dict(beta=-2.0)])
    assert [(p["val"], p["plateau_rule"]) for p in fake_engine[0]["priors"]] == [(0, False), (0, False)]
    assert fake_engine[0]["run"] == 5
    assert fits[0].get_params()["val"] == 30 and fits[1].get_params()["beta"] == -2.0


def test_inert_alpha_and_mixed_features(fake_engine):
    rng = np.random.default_rng(1)
    data = [(rng.normal(size=(10, 1)), rng.normal(size=10)), (rng.normal(size=(12, 3)), rng.normal(size=12))]
    fits = BSR(3, 2, seed=1).fit_many(data, mixed_features=True, params=[dict(alpha1=0.1, alpha2=0.2), dict(ops=["+", "cos"])])
    pri = fake_engine[0]["priors"]
    assert pri[0]["ops"] == [NAME_OP[o] for o in DEFAULT_OPS]
    assert pri[1]["ops"] == [NAME_OP["+"], NAME_OP["cos"]] and pri[1]["op_weights"] == [0.5, 0.5]
    assert fake_engine[0]["upload"][0] == "mixed"
    assert fits[0].get_params()["alpha1"] == 0.1 and fits[1].get_params()["ops"] == ["+", "cos"]


def test_engine_set_chain_priors_packs_the_struct(monkeypatch):
    seen = {}

    class _Lib:
        def bsr_set_chain_priors(self, h, n, priors, chain_prior):
            import ctypes
            arr = ctypes.cast(priors, ctypes.POINTER(capi.BsrPrior))
            seen["priors"] = [(arr[i].n_ops, list(arr[i].ops[:arr[i].n_ops]), list(arr[i].op_weights[:arr[i].n_ops]), arr[i].beta,
                               arr[i].val, arr[i].plateau_rule) for i in range(n)]
            seen["chain_prior"] = np.ctypeslib.as_array(ctypes.cast(chain_prior, ctypes.POINTER(ctypes.c_int32)), shape=(4,)).copy()
            return 0

    eng = capi.Engine.__new__(capi.Engine)
    eng._lib, eng._h, eng.C = _Lib(), None, 4
    eng.set_chain_priors([dict(ops=[9, 10], op_weights=[0.25, 0.75], beta=-0.5, val=0, plateau_rule=False),
                          dict(ops=[5], op_weights=[1.0], beta=-2.0, val=40, plateau_rule=True)], [1, 0, 1, 1])
    assert seen["priors"] == [(2, [9, 10], [0.25, 0.75], -0.5, 0, 0), (1, [5], [1.0], -2.0, 40, 1)]
    np.testing.assert_array_equal(seen["chain_prior"], [1, 0, 1, 1])
    with pytest.raises(ValueError, match="one prior index per chain"):
        eng.set_chain_priors([dict(ops=[9], op_weights=[1.0], beta=-1, val=0, plateau_rule=0)], [0, 0])
    eng._h = None


def test_run_suite_crosses_jobs_with_params(monkeypatch, fake_engine):
    from mcmc_symreg_b200 import experiments as E
    seen = []
    monkeypatch.setattr(E, "summarize_many", lambda fits, data: [dict(func=d["func"]) for d in data])
    monkeypatch.setattr(E, "run_experiment", lambda f, **kw: (seen.append((f, kw)) or dict(func=f), None, None))
    grid = [dict(beta=-1.0), dict(beta=-0.5)]
    loop = E.run_suite(("f1", "f2"), repeats=2, params=grid, K=3, MM=2, val=40)
    assert [(o["func"], o["repeat"], o["params"]) for o in loop] == [(f, r, p) for f in ("f1", "f2") for r in range(2) for p in grid]
    assert [(f, kw["seed"], kw["beta"], kw["val"]) for f, kw in seen] == [(f, r, p["beta"], 40) for f in ("f1", "f2") for r in range(2)
                                                                         for p in grid]
    rows = E.run_suite(("f1", "f2"), repeats=2, batched=True, params=grid, K=3, MM=2, val=40)
    assert [(o["func"], o["repeat"], o["params"]) for o in rows] == [(o["func"], o["repeat"], o["params"]) for o in loop]
    log = fake_engine[0]
    assert [p["beta"] for p in log["priors"]] == [-1.0, -0.5] * 4
    np.testing.assert_array_equal(log["keys"][0], np.repeat([0, 0, 1, 1, 0, 0, 1, 1], 2))   # the loop's seeds: seed + repeat
    assert len(log["upload"][1]) == 4                                 # one upload per (function, repeat)
    assert all("params" not in o for o in E.run_suite(("f1",), params=None, K=3, MM=2))


def test_cli_beta_list(monkeypatch):
    from mcmc_symreg_b200 import experiments as E
    seen = {}
    monkeypatch.setattr(E, "run_suite", lambda funcs, repeats, **kw: seen.update(kw) or [])
    E.main(["--func", "f1", "--beta", "-1,-0.5,-2", "--MM", "8"])
    assert seen["params"] == [dict(beta=-1.0), dict(beta=-0.5), dict(beta=-2.0)] and seen["MM"] == 8
    E.main(["--beta=-1.5"])
    assert seen["params"] == [dict(beta=-1.5)]
    E.main(["--func", "f2"])
    assert seen["params"] is None
