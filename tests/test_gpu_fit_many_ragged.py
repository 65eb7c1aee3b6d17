"""GPU tests of data sets of different row counts in one handle (bsr_set_datasets_ragged_host) and of BSR.fit_many(ragged=True):
the chains of data set b end bit for bit where the chains of a handle that holds only data set b end, keyed the same way, whenever
data set b's rows lie in the batch's first row split (and its own handle runs one split); else up to the fp64 summation order of the
splits."""
import ctypes
import json
import os
import socket
import sys

import numpy as np
import pytest

import parity_helpers as H
from test_gpu_fit_many import _assert_same_chains, _fits_equal, _state

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

FUNCS = ("f1", "f2", "f3", "f4", "f5", "f6")
ROWS = (3, 7, 30, 97, 100, 513, 1024, 1025, 3001)     # below K + 1, not a multiple of 4, at and across one 1024-row tile, several tiles


def _datasets(sizes, lo=-3.0, hi=3.0, seed=21):
    from mcmc_symreg_b200.experiments import TARGETS
    rng = np.random.default_rng(seed)
    Xs = [rng.uniform(lo, hi, (n, 2)) for n in sizes]
    return Xs, [TARGETS[FUNCS[b % len(FUNCS)]][0](X) for b, X in enumerate(Xs)]


def _layout(D, C, layout):
    if layout == "contiguous":
        return np.repeat(np.arange(D), C), np.tile(np.arange(C), D)
    return np.arange(D * C) % D, np.arange(D * C) // D


def _ragged_and_singles(Xs, ys, seeds, K, C, precision="fp32", mode="fixed", layout="contiguous"):
    D = len(Xs)
    stop = dict(val=100, plateau=True) if mode == "until" else dict(val=0, plateau=False)
    chain_ds, ids = _layout(D, C, layout)
    batch = H.default_engine(K, D * C, Xs[0].shape[1], precision=precision, **stop)
    batch.set_datasets_ragged(Xs, ys, chain_ds)
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


@pytest.mark.parametrize("layout", ["contiguous", "interleaved"])
@pytest.mark.parametrize("mode", ["fixed", "until"])
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_ragged_match_single_handles(precision, mode, layout):
    """nine data sets of 3 ... 3001 rows, 24 chains each: every chain equals its single-data-set run, bit for bit"""
    Xs, ys = _datasets(ROWS)
    batch, singles, chain_ds = _ragged_and_singles(Xs, ys, [11 * (b + 1) for b in range(len(ROWS))], 3, 24, precision, mode, layout)
    g = batch.window_geometry()
    assert g["splits"] == 1 and g["rows_per_split"] >= max(ROWS)
    _run([batch] + singles, mode, 30)
    got = _state(batch)
    for b, e in enumerate(singles):
        assert e.window_geometry()["splits"] == 1
        _assert_same_chains(got, np.nonzero(chain_ds == b)[0], _state(e))
    assert got["stats"]["counters"][:, 1].sum() > 0          # the chains moved
    _close(batch, *singles)


def test_ragged_double_range_k10():
    """K = 10 (live-column cache, checked first pass): row counts on both sides of the K = 10 tile; data set 1 drives exp out of
    the fp32 range, so its proposals take the double-range path on its own rows"""
    from mcmc_symreg_b200 import capi
    probe = H.default_engine(10, 16, 2)
    probe.set_data(np.random.default_rng(0).uniform(-3, 3, (4000, 2)), np.zeros(4000))
    tile = probe.window_geometry()["tile_rows"]
    probe.close()
    assert 900 <= tile <= 1024
    sizes = (tile - 13, tile + 11, 2 * tile + 5)
    Xs, ys = _datasets(sizes, seed=23)
    Xs[1] = np.random.default_rng(24).uniform(-100.0, 100.0, Xs[1].shape)
    ys[1] = np.sin(Xs[1][:, 0] / 20.0) + 0.01 * Xs[1][:, 1]
    batch, singles, chain_ds = _ragged_and_singles(Xs, ys, [31, 32, 33], 10, 16)
    assert batch.window_geometry()["tile_rows"] == tile
    _run([batch] + singles, "fixed", 20)
    got = _state(batch)
    for b, e in enumerate(singles):
        _assert_same_chains(got, np.nonzero(chain_ds == b)[0], _state(e))
    assert got["stats"]["counters"][chain_ds == 1, capi.CNT["fp64_sweeps"]].sum() > 0
    _close(batch, *singles)


def _floats_close(batch, rows, single, rtol=1e-10):
    """trees and counters exactly, the fp64 sums behind the floats up to a relative rtol of each array's scale"""
    for key in ("live", "roots"):
        for a, b in zip(batch[key], single[key]):
            np.testing.assert_array_equal(a[rows], b)
    for k, v in single["stats"].items():
        if v.dtype.kind == "f":
            np.testing.assert_allclose(batch["stats"][k][rows], v, rtol=rtol, atol=rtol * float(np.max(np.abs(v), initial=0.0)), err_msg=k)
        else:
            np.testing.assert_array_equal(batch["stats"][k][rows], v, err_msg=k)
    for c, r in enumerate(rows):
        np.testing.assert_allclose(batch["err"][r], single["err"][c], rtol=rtol, atol=0)


def test_ragged_row_splits():
    """largest data set of 40000 rows, 4 chains per data set: several row splits.  Data sets whose rows lie in the first split equal
    their single handles bit for bit; the largest equals its own in trees and counters, and in floats to 1e-10"""
    sizes = (300, 9000, 40000)
    Xs, ys = _datasets(sizes, seed=25)
    batch, singles, chain_ds = _ragged_and_singles(Xs, ys, [41, 42, 43], 3, 4)
    g = batch.window_geometry()
    assert g["splits"] > 1 and sizes[1] <= g["rows_per_split"] < sizes[2]
    for step in ("init", "run"):
        if step == "run":
            _run([batch] + singles, "fixed", 15)
        got = _state(batch)
        for b, e in enumerate(singles):
            rows = np.nonzero(chain_ds == b)[0]
            if sizes[b] <= g["rows_per_split"]:
                assert e.window_geometry()["splits"] == 1
                _assert_same_chains(got, rows, _state(e))
            else:
                _floats_close(got, rows, _state(e))
    _close(batch, *singles)


def test_ragged_equal_rows_is_set_datasets():
    """bsr_set_datasets_ragged_host with equal row counts gives the chains bsr_set_datasets_host gives"""
    Xs, ys = _datasets((100,) * 4, seed=26)
    cd = np.arange(4 * 16) % 4
    a = H.default_engine(3, 64, 2)
    a.set_datasets_ragged(Xs, ys, cd)
    b = H.default_engine(3, 64, 2)
    b.set_datasets(np.stack(Xs), np.stack(ys), cd)
    for e in (a, b):
        e.init_chains(9)
        e.run(30)
    assert a.window_geometry() == b.window_geometry()
    _assert_same_chains(_state(a), np.arange(64), _state(b))
    _close(a, b)


def test_fit_many_ragged_equals_loop_of_fits():
    """BSR.fit_many(ragged=True) equals a loop of cloned fits on data sets of different sizes, predictions included"""
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR
    Xs, ys = _datasets((30, 100, 300, 57), seed=27)
    est = BSR(3, 16, val=60)
    np.random.seed(5)
    fits = est.fit_many(list(zip(Xs, ys)), ragged=True)
    np.random.seed(5)
    loop = []
    for X, y in zip(Xs, ys):
        e = clone(est)
        e.fit(X, y)
        loop.append(e)
    Xt = np.random.default_rng(28).uniform(-3, 3, (50, 2))
    for a, b in zip(fits, loop):
        _fits_equal(a, b, Xt)
    # equal row counts: ragged=True is ragged=False
    Xe, ye = _datasets((80,) * 3, seed=29)
    strict = est.fit_many(list(zip(Xe, ye)), seeds=[1, 2, 3])
    rag = est.fit_many(list(zip(Xe, ye)), seeds=[1, 2, 3], ragged=True)
    for a, b in zip(strict, rag):
        _fits_equal(a, b, Xt)


def test_run_suite_learning_curve_rows():
    """run_suite(n_train=(30, 100), batched=True) gives the loop's rows outside the timing fields, each with its n_train"""
    from mcmc_symreg_b200.experiments import run_suite
    kw = dict(K=3, MM=8, n_train=(30, 100), n_test=20, val=60, seed=4)
    loop = run_suite(("f1", "f4"), 2, **kw)
    batch = run_suite(("f1", "f4"), 2, batched=True, **kw)
    assert len(loop) == len(batch) == 8
    assert [o["n_train"] for o in batch] == [30, 30, 100, 100] * 2
    strip = lambda o: json.dumps({k: v for k, v in o.items() if k not in ("fit_seconds", "batch_seconds")}, sort_keys=True, default=str)
    for a, b in zip(loop, batch):
        assert strip(a) == strip(b)


def test_ragged_refusals():
    """what bsr_set_datasets_ragged_host refuses, and what a handle of several data sets of different sizes does not do"""
    from mcmc_symreg_b200 import capi
    lib = capi.load()
    Xs, ys = _datasets((40, 60), seed=30)
    X, y = np.concatenate(Xs), np.concatenate(ys)
    cd = (np.arange(8) % 2).astype(np.int32)
    eng = H.default_engine(3, 8, 2)

    def call(n_rows, d=2, x=X, yy=y, chains=cd):
        nr = None if n_rows is None else np.asarray(n_rows, dtype=np.int64)
        capi._ck(lib.bsr_set_datasets_ragged_host(eng._h, 2, capi._ptr(x), capi._ptr(yy), capi._ptr(nr), d, capi._ptr(chains)))

    with pytest.raises(capi.BsrError, match=r"n_rows\[1\] = 0: every data set needs at least one row"):
        call([40, 0])
    with pytest.raises(capi.BsrError, match="bsr_set_datasets_ragged_host: null argument"):
        call(None)
    with pytest.raises(capi.BsrError, match=r"chain_dataset\[1\] = 2 is outside \[0, 2\)"):
        call([40, 60], chains=np.array([0, 2, 0, 0, 0, 0, 0, 0], dtype=np.int32))
    with pytest.raises(capi.BsrError, match="below 2\\^32"):       # checked before any data is read: X holds 100 rows, not 2^30
        call([1 << 30, 5], d=4)
    eng.set_datasets_ragged(Xs, ys, cd)
    eng.init_chains(1)
    with pytest.raises(capi.BsrError, match="bsr_set_pipeline: not available on a handle with several data sets"):
        eng.set_pipeline(True)
    for fn in (eng.sweep_propose, eng.sweep_eval, eng.sweep_resolve):
        with pytest.raises(capi.BsrError, match="not available on a handle with several data sets"):
            fn()
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
    with pytest.raises(capi.BsrError, match="bsr_set_datasets_ragged_host: not available on row-sharded handles"):
        rs.set_datasets_ragged(Xs, ys, cd)
    rs.close()
    seq = H.default_engine(3, 8, 2)
    seq.set_pipeline(True)
    with pytest.raises(capi.BsrError, match="proposal-by-proposal pipeline"):
        seq.set_datasets_ragged(Xs, ys, cd)
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
    Xs, ys = _datasets((40, 130, 75), seed=31)
    fits = BSR(3, 13, seed=5, val=60).fit_many(list(zip(Xs, ys)), seeds=[5, 6, 7], ragged=True)
    q.put((rank, [f.model() for f in fits], [[len(e) for e in f.train_err_] for f in fits], [f.betas_[4].ravel().tolist() for f in fits]))
    dist.destroy_process_group()


def test_fit_many_ragged_two_ranks():
    """fit_many(ragged=True) under a 2-rank NCCL group (3 x 13 chains sharded over the ranks) equals the one-rank result"""
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
    Xs, ys = _datasets((40, 130, 75), seed=31)
    fits = BSR(3, 13, seed=5, val=60, distributed=False).fit_many(list(zip(Xs, ys)), seeds=[5, 6, 7], ragged=True)
    assert [f.model() for f in fits] == res[0][1]
    assert [[len(e) for e in f.train_err_] for f in fits] == res[0][2]
    assert [f.betas_[4].ravel().tolist() for f in fits] == res[0][3]
