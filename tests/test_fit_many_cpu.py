"""Host logic of BSR.fit_many that needs no GPU: shape checks before any library call, the per-data-set split of gathered
results, and the seeds it derives."""
import numpy as np
import pytest

from mcmc_symreg_b200 import BSR, capi, parallel
from mcmc_symreg_b200.bsr_class import check_datasets, dataset_seeds


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(capi, "load", refuse)
    monkeypatch.setattr(capi, "Engine", refuse)


@pytest.mark.parametrize("datasets, match", [
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((11, 2)), np.zeros(11))], "same shape"),
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 3)), np.zeros(10))], "same shape"),
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 2)), np.zeros(9))], "disagree on the number of rows"),
    ([], "no data sets"),
])
def test_shape_errors_before_any_library_call(no_library, datasets, match):
    with pytest.raises(ValueError, match=match):
        BSR(3, 4, seed=1).fit_many(datasets)


def test_seed_count_error_before_any_library_call(no_library):
    with pytest.raises(ValueError, match="2 seeds for 3 data sets"):
        BSR(3, 4).fit_many([(np.zeros((5, 2)), np.zeros(5))] * 3, seeds=[1, 2])


def test_check_datasets_accepts_equal_shapes():
    check_datasets([(np.zeros((7, 3)), np.zeros(7))] * 4)


def test_seeds_consume_numpy_state_like_a_loop_of_fits():
    np.random.seed(123)
    loop = [int(np.random.randint(0, 2 ** 31 - 1)) for _ in range(5)]       # what five fit() calls with seed=None draw
    after_loop = np.random.rand()
    np.random.seed(123)
    assert dataset_seeds(None, 5) == loop
    assert np.random.rand() == after_loop
    state = np.random.get_state()[1].copy()
    assert dataset_seeds(9, 3) == [9, 9, 9]
    assert dataset_seeds(None, 2, seeds=[4, 5]) == [4, 5]
    np.testing.assert_array_equal(np.random.get_state()[1], state)       # given seeds draw nothing


def _fake_result(B, MM, K, rng):
    C = B * MM
    nn = rng.integers(1, 9, (C, K)).astype(np.int32)
    ptok = rng.integers(0, 11, int(nn.sum())).astype(np.uint32) | (rng.integers(0, 3, int(nn.sum())).astype(np.uint32) << 16)
    n_lt = int(np.count_nonzero((ptok & 0xFF) == 2))
    return dict(nn=nn, ptok=ptok, pab=rng.normal(size=(n_lt, 2)), beta=rng.normal(size=(C, K + 1)), sigma=rng.normal(size=C),
                sa=rng.normal(size=(C, K)), sb=rng.normal(size=(C, K)), sse=rng.normal(size=C),
                counters=rng.integers(0, 99, (C, capi.N_COUNTERS)), done=rng.integers(0, 2, C).astype(np.int32),
                nerr=rng.integers(0, 5, C).astype(np.int32), err=rng.normal(size=(C, 6)), sweeps=77)


def test_split_results_per_dataset():
    """each part is what one fit of MM chains would hold: its rows, its packed trees, the batch's sweep count"""
    B, MM, K = 3, 5, 4
    res = _fake_result(B, MM, K, np.random.default_rng(0))
    parts = parallel.split_results(res, B, MM)
    full = capi.PackedTrees(res["nn"], res["ptok"], res["pab"])
    assert len(parts) == B
    for b, p in enumerate(parts):
        rows = slice(b * MM, (b + 1) * MM)
        for key in ("nn", "beta", "sigma", "sa", "sb", "sse", "counters", "done", "nerr", "err"):
            np.testing.assert_array_equal(p[key], res[key][rows])
        assert p["sweeps"] == 77
        pk = capi.PackedTrees(p["nn"], p["ptok"], p["pab"])
        for m in range(MM):
            for k in range(K):
                for x, y in zip(pk.tree(m, k), full.tree(b * MM + m, k)):
                    np.testing.assert_array_equal(x, y)
    assert sum(p["ptok"].size for p in parts) == res["ptok"].size
    assert sum(p["pab"].shape[0] for p in parts) == res["pab"].shape[0]
