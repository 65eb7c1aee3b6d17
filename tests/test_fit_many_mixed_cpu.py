"""Host logic of data sets of different feature counts that needs no GPU: BSR.fit_many(mixed_features=True)'s checks before any
library call, and capi.predict_groups over test sets of different widths (zero-padded to the widest after a per-group feature
check)."""
import ctypes

import numpy as np
import pytest

from mcmc_symreg_b200 import BSR, capi
from mcmc_symreg_b200.bsr_class import check_datasets


@pytest.fixture
def no_library(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the library was called")
    monkeypatch.setattr(capi, "load", refuse)
    monkeypatch.setattr(capi, "Engine", refuse)


def test_mixed_accepts_different_rows_and_features():
    check_datasets([(np.zeros((n, d)), np.zeros(n)) for n, d in ((3, 1), (30, 8), (1025, 2))], mixed_features=True)
    check_datasets([(np.zeros((n, d)), np.zeros(n)) for n, d in ((3, 1), (30, 8))], ragged=True, mixed_features=True)


@pytest.mark.parametrize("datasets, match", [
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((12, 3)), np.zeros(9))], "data set 1: train_data and train_y disagree on the number of rows"),
    ([(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 0)), np.zeros(10))], "data set 1 has no features"),
    ([], "no data sets"),
])
def test_mixed_errors_before_any_library_call(no_library, datasets, match):
    with pytest.raises(ValueError, match=match):
        BSR(3, 4, seed=1).fit_many(datasets, mixed_features=True)


def test_old_messages_unchanged(no_library):
    feats = [(np.zeros((10, 2)), np.zeros(10)), (np.zeros((11, 3)), np.zeros(11))]
    with pytest.raises(ValueError, match=r"^fit_many: data set 1 has 3 features, data set 0 has 2: all data sets must have the same number "
                                         r"of features \(mixed_features=True accepts different feature counts\)$"):
        BSR(3, 4, seed=1).fit_many(feats, ragged=True)
    same_rows = [(np.zeros((10, 2)), np.zeros(10)), (np.zeros((10, 3)), np.zeros(10))]
    with pytest.raises(ValueError, match=r"^fit_many: data set 1 is 10 x 3, data set 0 is 10 x 2: all data sets must have the same shape$"):
        BSR(3, 4, seed=1).fit_many(same_rows)


class _FakeLib:
    """captures what capi.predict_groups hands bsr_predict_groups (the arrays read while the call lasts)"""

    def __init__(self):
        self.calls = []

    def bsr_predict_groups(self, device, M, K, nn, tok, n_tok, ab, n_lt, beta, S, d, X, set_off, G, grp_set, grp_off, models, reduce,
                           out, used):
        def arr(p, ctype, n):
            return np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ctype)), shape=(n,)).copy()
        offs = arr(set_off, ctypes.c_int64, S + 1)
        self.calls.append(dict(S=S, d=d, set_off=offs, X=arr(X, ctypes.c_double, int(offs[-1]) * d).reshape(-1, d),
                               grp_set=arr(grp_set, ctypes.c_int32, G)))
        return 0


def _models(features):
    """one single-leaf tree per model (K = 1), model m reading feature features[m]"""
    M = len(features)
    nn = np.ones((M, 1), dtype=np.int32)
    tok = (np.asarray(features, dtype=np.uint32) << 16)
    beta = np.tile([0.0, 1.0], (M, 1))
    return nn, tok, np.zeros((0, 2)), beta


def test_predict_groups_pads_to_the_widest(monkeypatch):
    fake = _FakeLib()
    monkeypatch.setattr(capi, "load", lambda: fake)
    nn, tok, ab, beta = _models([0, 1, 4, 2])
    rng = np.random.default_rng(3)
    sets = [rng.normal(size=(3, 1)), rng.normal(size=(5, 5)), rng.normal(size=(2, 3))]
    blocks, _ = capi.predict_groups(0, nn, tok, ab, beta, sets, [0, 1, 2, 1], [[0], [1, 2], [3, 0], [0]], [False, True, False, False])
    call = fake.calls[0]
    assert call["S"] == 3 and call["d"] == 5
    np.testing.assert_array_equal(call["set_off"], [0, 3, 8, 10])
    np.testing.assert_array_equal(call["grp_set"], [0, 1, 2, 1])
    X = call["X"]
    for s, lo in zip(sets, call["set_off"][:-1]):
        np.testing.assert_array_equal(X[lo:lo + s.shape[0], :s.shape[1]], s)
        assert np.all(X[lo:lo + s.shape[0], s.shape[1]:] == 0.0)
    assert [b.shape for b in blocks] == [(1, 3), (2, 5), (2, 2), (1, 5)]


def test_predict_groups_equal_widths_unchanged(monkeypatch):
    fake = _FakeLib()
    monkeypatch.setattr(capi, "load", lambda: fake)
    nn, tok, ab, beta = _models([0, 1])
    sets = [np.ones((3, 2)), 2 * np.ones((4, 2))]
    capi.predict_groups(0, nn, tok, ab, beta, sets, [0, 1], [[0], [1]], [False, False])
    assert fake.calls[0]["d"] == 2
    np.testing.assert_array_equal(fake.calls[0]["X"], np.concatenate(sets))


@pytest.mark.parametrize("groups, sets_of, match", [
    ([[2]], [1], "group 0: model 2 reads feature 4, its test set 1 has 3 features"),
    ([[0], [1, 3]], [0, 0], "group 1: model 1 reads feature 1, its test set 0 has 1 features"),
    ([[0, 1, 3]], [2], "group 0: model 3 reads feature 5, its test set 2 has 5 features"),
])
def test_predict_groups_refuses_a_narrow_test_set(no_library, groups, sets_of, match):
    nn, tok, ab, beta = _models([0, 1, 4, 5])
    sets = [np.zeros((3, 1)), np.zeros((4, 3)), np.zeros((2, 5))]
    with pytest.raises(ValueError, match=match):
        capi.predict_groups(0, nn, tok, ab, beta, sets, sets_of, groups, [False] * len(groups))


def test_predict_groups_leaves_malformed_tables_to_the_library(monkeypatch):
    """node counts that do not cover tok, or a model index out of range: no host error, the library's refusals decide"""
    fake = _FakeLib()
    monkeypatch.setattr(capi, "load", lambda: fake)
    nn, tok, ab, beta = _models([0, 1])
    sets = [np.zeros((3, 1)), np.zeros((4, 3))]
    capi.predict_groups(0, nn, tok[:1], ab, beta, sets, [0, 1], [[0], [1]], [False, False])
    capi.predict_groups(0, nn, tok, ab, beta, sets, [0, 1], [[0], [7]], [False, False])
    assert len(fake.calls) == 2 and all(c["d"] == 3 for c in fake.calls)
