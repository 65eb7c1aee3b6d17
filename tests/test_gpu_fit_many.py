"""GPU tests of several data sets in one handle (bsr_set_datasets_host, bsr_init_chains_keyed) and of BSR.fit_many: the chains of
data set b end bit for bit where the chains of a handle that holds only data set b end, keyed the same way."""
import ctypes
import json
import os
import socket
import sys

import numpy as np
import pytest

import parity_helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

FUNCS = ("f1", "f2", "f3", "f4", "f5")


def _datasets(D, n=300, lo=-3.0, hi=3.0, seed=11):
    from mcmc_symreg_b200.experiments import TARGETS
    rng = np.random.default_rng(seed)
    Xs, ys = [], []
    for b in range(D):
        X = rng.uniform(lo, hi, (n, 2))
        Xs.append(X)
        ys.append(TARGETS[FUNCS[b % len(FUNCS)]][0](X))
    return Xs, ys


def _state(eng):
    st = eng.get_stats()
    err = eng.get_err_trace()
    return dict(live=eng.get_trees(current=True), roots=eng.get_trees(current=False), stats=st,
                err=[err[c, :st["nerr"][c]] for c in range(eng.C)])


def _assert_same_chains(batch, rows, single):
    """chains `rows` of the batch state equal every chain of the single-data-set state, bit for bit"""
    for key in ("live", "roots"):
        for a, b in zip(batch[key], single[key]):
            np.testing.assert_array_equal(a[rows], b)
    for k, v in single["stats"].items():
        np.testing.assert_array_equal(batch["stats"][k][rows], v, err_msg=k)
    for c, r in enumerate(rows):
        np.testing.assert_array_equal(batch["err"][r], single["err"][c])


def _compare(Xs, ys, seeds, K=3, C=64, precision="fp32", mode="fixed", layout="contiguous", run=30):
    D = len(Xs)
    stop = dict(val=100, plateau=True) if mode == "until" else dict(val=0, plateau=False)
    if layout == "contiguous":
        chain_ds, ids = np.repeat(np.arange(D), C), np.tile(np.arange(C), D)
    else:
        chain_ds, ids = np.arange(D * C) % D, np.arange(D * C) // D
    batch = H.default_engine(K, D * C, Xs[0].shape[1], precision=precision, **stop)
    batch.set_datasets(np.stack(Xs), np.stack(ys), chain_ds)
    batch.init_chains_keyed(np.asarray(seeds)[chain_ds], ids)
    singles = []
    for b in range(D):
        e = H.default_engine(K, C, Xs[b].shape[1], precision=precision, **stop)
        e.set_data(Xs[b], ys[b])
        e.init_chains(seeds[b])
        assert e.window_geometry() == batch.window_geometry()
        singles.append(e)
    for e in [batch] + singles:
        if mode == "fixed":
            e.run(run)
        else:
            e.run_until_done(3000, check_every=32)
    got = _state(batch)
    for b, e in enumerate(singles):
        _assert_same_chains(got, np.nonzero(chain_ds == b)[0], _state(e))
        e.close()
    batch.close()
    return got, chain_ds


@pytest.mark.parametrize("mode", ["fixed", "until"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_datasets_match_single_handles(precision, mode):
    """five data sets (f1 ... f5, different X), 64 chains each, contiguous: every chain equals its single-data-set run"""
    Xs, ys = _datasets(5)
    got, _ = _compare(Xs, ys, [101, 202, 303, 404, 505], precision=precision, mode=mode)
    assert got["stats"]["counters"][:, 1].sum() > 0          # the chains moved


@pytest.mark.parametrize("mode", ["fixed", "until"])
def test_datasets_interleaved(mode):
    """chain c on data set c mod D: the chains of a data set need not be contiguous"""
    Xs, ys = _datasets(5, seed=12)
    _compare(Xs, ys, [7, 8, 9, 10, 11], mode=mode, layout="interleaved")


def test_datasets_double_range_k10():
    """K = 10 (live-column cache, checked first pass): data set 1 drives exp out of the fp32 range, so its proposals take the
    double-range path, which must read the data set's own X"""
    Xs, ys = _datasets(2, seed=13)
    Xs[1] = np.random.default_rng(14).uniform(-100.0, 100.0, Xs[1].shape)
    ys[1] = np.sin(Xs[1][:, 0] / 20.0) + 0.01 * Xs[1][:, 1]
    got, chain_ds = _compare(Xs, ys, [21, 22], K=10, C=32, run=20)
    from mcmc_symreg_b200 import capi
    assert got["stats"]["counters"][chain_ds == 1, capi.CNT["fp64_sweeps"]].sum() > 0


def test_one_dataset_equals_set_data():
    """bsr_set_datasets_host with D = 1 is bsr_set_data_host"""
    Xs, ys = _datasets(1)
    a = H.default_engine(3, 64, 2)
    a.set_datasets(Xs[0][None], ys[0][None], np.zeros(64, dtype=np.int32))
    a.init_chains(5)
    b = H.default_engine(3, 64, 2)
    b.set_data(Xs[0], ys[0])
    b.init_chains(5)
    a.run(30); b.run(30)
    _assert_same_chains(_state(a), np.arange(64), _state(b))


def _fits_equal(a, b, X):
    from mcmc_symreg_b200.trees import Express
    assert a.model() == b.model()
    for m in range(len(a.betas_)):
        assert [Express(t) for t in a.roots_[m]] == [Express(t) for t in b.roots_[m]]
        np.testing.assert_array_equal(a.betas_[m], b.betas_[m])
    for x, y in zip(a._enc_, b._enc_):
        np.testing.assert_array_equal(x, y)
    assert a.train_err_ == b.train_err_ and a.train_err_truncated_ == b.train_err_truncated_
    np.testing.assert_array_equal(a.counters_, b.counters_)
    np.testing.assert_array_equal(a.done_, b.done_)
    np.testing.assert_array_equal(a.final_rmse_, b.final_rmse_)
    np.testing.assert_array_equal(a.predict(X), b.predict(X))
    np.testing.assert_array_equal(a.predict_best(X), b.predict_best(X))
    np.testing.assert_array_equal(a.predict_mean(X), b.predict_mean(X))


def test_fit_many_equals_loop_of_fits():
    """BSR.fit_many equals a loop of cloned fits; seeds=None draws one seed per data set from numpy's global state"""
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR
    Xs, ys = _datasets(4, n=100, seed=15)
    est = BSR(3, 16, val=60)
    np.random.seed(3)
    fits = est.fit_many(list(zip(Xs, ys)))
    after = np.random.randint(0, 1000)
    np.random.seed(3)
    loop = []
    for X, y in zip(Xs, ys):
        e = clone(est)
        e.fit(X, y)
        loop.append(e)
    assert np.random.randint(0, 1000) == after
    Xt = np.random.default_rng(16).uniform(-3, 3, (50, 2))
    for a, b in zip(fits, loop):
        assert a.get_params() == est.get_params()
        _fits_equal(a, b, Xt)


def test_run_suite_batched_rows():
    """run_suite(batched=True) gives the unbatched rows outside the timing fields"""
    from mcmc_symreg_b200.experiments import run_suite
    kw = dict(K=3, MM=8, n_train=100, n_test=20, val=60, seed=4)
    loop = run_suite(("f1", "f4"), 2, **kw)
    batch = run_suite(("f1", "f4"), 2, batched=True, **kw)
    assert len(loop) == len(batch) == 4
    for a, b in zip(loop, batch):
        assert b["batch_seconds"] > 0 and b["fit_seconds"] == b["batch_seconds"] / 4
        strip = lambda o: json.dumps({k: v for k, v in o.items() if k not in ("fit_seconds", "batch_seconds")}, sort_keys=True, default=str)
        assert strip(a) == strip(b)


def test_refusals():
    """what a handle of several data sets does not do, it refuses with a message"""
    from mcmc_symreg_b200 import capi
    Xs, ys = _datasets(2, n=100)
    X, y, cd = np.stack(Xs), np.stack(ys), np.arange(8) % 2
    eng = H.default_engine(3, 8, 2)
    with pytest.raises(capi.BsrError, match=r"chain_dataset\[1\] = 2 is outside \[0, 2\)"):
        eng.set_datasets(X, y, np.array([0, 2, 0, 0, 0, 0, 0, 0]))
    lib = capi.load()
    with pytest.raises(capi.BsrError, match="below 2\\^32"):      # the size guard is checked before any data is read
        capi._ck(lib.bsr_set_datasets_host(eng._h, 2, capi._ptr(X), capi._ptr(y), 1 << 30, 4, capi._ptr(cd.astype(np.int32))))
    eng.set_datasets(X, y, cd)
    eng.init_chains(1)
    with pytest.raises(capi.BsrError, match="bsr_set_pipeline: not available on a handle with several data sets"):
        eng.set_pipeline(True)
    for call in (eng.sweep_propose, eng.sweep_eval, eng.sweep_resolve):
        with pytest.raises(capi.BsrError, match="not available on a handle with several data sets"):
            call()
    tok, pa, pb, nn = eng.get_trees(current=True)
    with pytest.raises(capi.BsrError, match="bsr_eval_trees: not available on a handle with several data sets"):
        eng.eval_trees(tok[0], pa[0], pb[0], nn[0])
    with pytest.raises(capi.BsrError, match="bsr_peer_export: not available on a handle with several data sets"):
        eng.peer_export(2)
    with pytest.raises(capi.BsrError, match="bsr_peer_import: not available on a handle with several data sets"):
        capi._ck(lib.bsr_peer_import(eng._h, 0, 2, ctypes.create_string_buffer(128)))
    eng.run(2)                                                     # bsr_run itself works
    eng.close()
    rs = capi.Engine(3, 8, list(range(1, 11)), [0.1] * 10, row_sharded=True)
    for Xr, yr, cr in ((X, y, cd), (X[:1], y[:1], np.zeros(8))):     # one data set too: set_data carries the global row count
        with pytest.raises(capi.BsrError, match="not available on row-sharded handles"):
            rs.set_datasets(Xr, yr, cr)
    rs.close()
    seq = H.default_engine(3, 8, 2)
    seq.set_pipeline(True)
    with pytest.raises(capi.BsrError, match="proposal-by-proposal pipeline"):
        seq.set_datasets(X, y, cd)
    seq.close()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from mcmc_symreg_b200 import BSR
    Xs, ys = _datasets(3, n=100, seed=17)
    fits = BSR(3, 13, seed=5, val=60).fit_many(list(zip(Xs, ys)), seeds=[5, 6, 7])
    q.put((rank, [f.model() for f in fits], [[len(e) for e in f.train_err_] for f in fits], [f.betas_[4].ravel().tolist() for f in fits]))
    dist.destroy_process_group()


def test_fit_many_two_ranks():
    """fit_many under a 2-rank NCCL group (3 x 13 chains sharded over the ranks) equals the one-rank result"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
    assert res[0][1:] == res[1][1:]
    from mcmc_symreg_b200 import BSR
    Xs, ys = _datasets(3, n=100, seed=17)
    fits = BSR(3, 13, seed=5, val=60, distributed=False).fit_many(list(zip(Xs, ys)), seeds=[5, 6, 7])
    assert [f.model() for f in fits] == res[0][1]
    assert [[len(e) for e in f.train_err_] for f in fits] == res[0][2]
    assert [f.betas_[4].ravel().tolist() for f in fits] == res[0][3]
