"""Host logic of data sets of different row counts that needs no GPU: BSR.fit_many(ragged=True)'s checks before any library call,
and the jobs and seeds of the learning-curve grid of run_suite."""
import numpy as np
import pytest

from mcmc_symreg_b200 import BSR, capi
from mcmc_symreg_b200.bsr_class import check_datasets
from mcmc_symreg_b200.experiments import _sizes, suite_jobs


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(capi, "load", refuse)
    monkeypatch.setattr(capi, "Engine", refuse)


def test_ragged_accepts_different_row_counts():
    check_datasets([(np.zeros((n, 3)), np.zeros(n)) for n in (3, 30, 1025)], ragged=True)


@pytest.mark.parametrize("datasets, match", [
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((11, 3)), np.zeros(11))], "data set 1 has 3 features, data set 0 has 2: .*same number of features"),
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((12, 2)), np.zeros(9))], "disagree on the number of rows"),
    ([], "no data sets"),
])
def test_ragged_errors_before_any_library_call(no_library, datasets, match):
    with pytest.raises(ValueError, match=match):
        BSR(3, 4, seed=1).fit_many(datasets, ragged=True)


def test_strict_default_names_ragged_for_row_counts_only(no_library):
    rows = [(np.zeros((10, 2)), np.zeros(10)), (np.zeros((11, 2)), np.zeros(11))]
    with pytest.raises(ValueError, match=r"same shape \(ragged=True accepts different row counts\)"):
        BSR(3, 4, seed=1).fit_many(rows)
    feats = [(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 3)), np.zeros(10))]
    with pytest.raises(ValueError, match=r"same shape$"):
        BSR(3, 4, seed=1).fit_many(feats)


def test_suite_jobs_grid():
    """function x size x repeat, in that order; repeat r is seeded seed + r at every size"""
    jobs = suite_jobs(("f1", "f4"), 2, (30, 100, 300), seed=7)
    assert jobs == [(f, n, r, 7 + r) for f in ("f1", "f4") for n in (30, 100, 300) for r in range(2)]
    assert len(jobs) == 12


def test_suite_jobs_one_size_is_the_plain_suite():
    assert suite_jobs(("f1", "f2", "f3"), 3, 100) == [(f, 100, r, r) for f in ("f1", "f2", "f3") for r in range(3)]
    assert suite_jobs(("f6",), 2, np.int64(50), seed=4) == [("f6", 50, 0, 4), ("f6", 50, 1, 5)]


def test_n_train_option():
    assert _sizes("100") == 100
    assert _sizes("30,100,300") == (30, 100, 300)
    assert _sizes("1000,") == (1000,)
