"""Measures what fitting many small data sets in one GPU run (BSR.fit_many) saves; prints one JSON line.

1. The suite of the paper's Table 1 at the reference's own size: f1 ... f6 x R repeats, BSR(3, 50, val=100) on n = 100 rows.
   Wall clock of the loop of BSR.fit calls against one BSR.fit_many over the same data sets and seeds, alternated, each timing
   ending in a device synchronise; the two must give equal results (checked in the same run).
   With several sizes (--rows 30,100,300,1000) the suite is f1 ... f6 x those sizes x R repeats, and fit_many runs with ragged=True.
2. The summaries of those fits (experiments.summarize: RMSE of the last, best and mean prediction on the training, test and
   extrapolation sets, 9 predictions per fit): the summarize loop against summarize_many (one grouped prediction call), alternated,
   each timing ending in a device synchronise, rows compared; and per method the 3 x (data sets) single-estimator prediction calls
   against one BSR.predict_many per set.
3. Engine throughput: D data sets x 50 chains on n = 100 rows (the first of --rows), fixed sweeps, device-timed (CUDA events)
   proposals per second.  With several sizes, one more line: the largest D with the data sets cycling through the sizes (a ragged
   batch, every chain on its own rows) against the same chains on data sets of the largest size.
4. A suite of different feature counts (``mixed``): d in {1, 2, 3, 5, 8} x R repeats on n = 100 rows (the first of --rows), the
   synthetic targets of ``mixed_target``, BSR(3, 50, val=100).  The loop of BSR.fit calls against one
   BSR.fit_many(mixed_features=True), alternated, each timing ending in a device synchronise, results compared.

    python scripts/bench_fit_many.py [--repeats 50] [--rounds 3] [--sweeps 300] [--datasets 1,16,128,1024] [--rows 100 | 30,100,300,1000]
                                     [--sections suite,summaries,engine,mixed]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=60).stdout.strip()
    except Exception as e:  # the name still identifies the card
        power = "unknown (%s)" % type(e).__name__
    return name, power


def suite_data(repeats, sizes):
    from mcmc_symreg_b200.experiments import make_dataset, suite_jobs
    jobs = suite_jobs(("f1", "f2", "f3", "f4", "f5", "f6"), repeats, sizes[0] if len(sizes) == 1 else sizes)
    return jobs, [make_dataset(f, n, 30, seed=s) for f, n, _, s in jobs]


def fingerprint(est):
    return (est.model(), [b.ravel().tolist() for b in est.betas_], est.train_err_, est.counters_.tolist(), est.done_.tolist())


def bench_suite(repeats, rounds, sizes):
    import torch
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR
    jobs, data = suite_data(repeats, sizes)
    ragged = len(sizes) > 1
    est = BSR(3, 50, val=100)
    seeds = [s for _, _, _, s in jobs]
    pairs = [(d["X"], d["y"]) for d in data]

    def loop():
        out = []
        for (X, y), s in zip(pairs, seeds):
            e = clone(est).set_params(seed=s)
            e.fit(X, y)
            out.append(e)
        torch.cuda.synchronize()
        return out

    def batch():
        out = est.fit_many(pairs, seeds=seeds, ragged=ragged)
        torch.cuda.synchronize()
        return out

    loop(); batch()                               # module loads, allocations
    t_loop, t_batch, equal = [], [], True
    for _ in range(rounds):
        t0 = time.perf_counter(); a = loop(); t_loop.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); b = batch(); t_batch.append(time.perf_counter() - t0)
        equal = equal and all(fingerprint(x) == fingerprint(y) for x, y in zip(a, b))
    assert equal, "fit_many and the loop of fits disagree"
    return dict(datasets=len(jobs), chains_per_fit=50, rows=sizes[0] if len(sizes) == 1 else list(sizes), ragged=ragged, loop_seconds=t_loop, fit_many_seconds=t_batch,
                loop_ms_per_fit=1e3 * float(np.median(t_loop)) / len(jobs), fit_many_ms_per_fit=1e3 * float(np.median(t_batch)) / len(jobs),
                speedup_median=float(np.median(t_loop) / np.median(t_batch)), results_equal=equal)


def bench_summaries(repeats, rounds, sizes):
    """The summaries of the suite's fits: the per-estimator summarize loop (9 prediction calls per fit) against summarize_many (one
    grouped call), alternated, each timing ending in a device synchronise, rows compared as JSON.  Then the predictions alone: per
    method, one call per (fit, set) against one BSR.predict_many per set."""
    import torch
    from mcmc_symreg_b200 import BSR
    from mcmc_symreg_b200.experiments import SETS, summarize, summarize_many
    jobs, data = suite_data(repeats, sizes)
    fits = BSR(3, 50, val=100).fit_many([(d["X"], d["y"]) for d in data], seeds=[s for _, _, _, s in jobs], ragged=len(sizes) > 1)
    dump = lambda rows: [json.dumps(o, sort_keys=True, default=str) for o in rows]

    def timed(fn):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, out

    loop = lambda: [summarize(e, d) for e, d in zip(fits, data)]
    many = lambda: summarize_many(fits, data)
    loop(); many()                                # module loads, allocations
    t_loop, t_many, equal = [], [], True
    for _ in range(rounds):
        ta, a = timed(loop)
        tb, b = timed(many)
        t_loop.append(ta); t_many.append(tb)
        equal = equal and dump(a) == dump(b)
    assert equal, "summarize_many and the summarize loop disagree"
    single = dict(last=lambda e, X: e.predict(X), best=lambda e, X: e.predict_best(X), mean=lambda e, X: e.predict_mean(X))
    per_method = {}
    for method, call in single.items():
        singles = lambda: [call(e, d[Xk]) for _, Xk, _ in SETS for e, d in zip(fits, data)]
        grouped = lambda: [BSR.predict_many(fits, [d[Xk] for d in data], method=method) for _, Xk, _ in SETS]
        singles(); grouped()
        ts, tg, same = [], [], True
        for _ in range(rounds):
            t, a = timed(singles)
            ts.append(t)
            t, b = timed(grouped)
            tg.append(t)
            same = same and all(np.array_equal(x, y) for x, y in zip(a, [p for per_set in b for p in per_set]))
        assert same, "predict_many(method=%r) and the single calls disagree" % method
        per_method[method] = dict(single_calls=len(fits) * len(SETS), single_seconds=ts, predict_many_calls=len(SETS),
                                  predict_many_seconds=tg, speedup_median=float(np.median(ts) / np.median(tg)))
    return dict(fits=len(fits), loop_seconds=t_loop, summarize_many_seconds=t_many,
                loop_ms_per_fit=1e3 * float(np.median(t_loop)) / len(fits), summarize_many_ms_per_fit=1e3 * float(np.median(t_many)) / len(fits),
                speedup_median=float(np.median(t_loop) / np.median(t_many)), results_equal=equal, predictions=per_method)


def bench_engine(D, sweeps, n, C=50, K=3):
    """n: the rows of every data set, or a sequence the data sets cycle through (a ragged batch)"""
    import torch
    from mcmc_symreg_b200 import capi
    from mcmc_symreg_b200.experiments import TARGETS
    rng = np.random.default_rng(D)
    sizes = [n] * D if np.isscalar(n) else [n[b % len(n)] for b in range(D)]
    X = [rng.uniform(-3, 3, (sizes[b], 2)) for b in range(D)]
    y = [TARGETS["f%d" % (1 + b % 6)][0](X[b]) for b in range(D)]
    eng = capi.Engine(K, D * C, list(range(1, 11)), [0.1] * 10, val=0, plateau_rule=False)
    try:
        if np.isscalar(n):
            eng.set_datasets(np.stack(X), np.stack(y), np.repeat(np.arange(D), C))
        else:
            eng.set_datasets_ragged(X, y, np.repeat(np.arange(D), C))
        eng.init_chains_keyed(np.repeat(np.arange(D) + 1000, C), np.tile(np.arange(C), D))
        stream = torch.cuda.current_stream()
        eng.run(20, stream.cuda_stream)                      # warm-up: allocations, module loads
        p0 = int(eng.get_stats()["counters"][:, capi.CNT["proposals"]].sum())
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        eng.run(sweeps, stream.cuda_stream)
        b.record(stream)
        b.synchronize()
        ms = a.elapsed_time(b)
        p1 = int(eng.get_stats()["counters"][:, capi.CNT["proposals"]].sum())
    finally:
        eng.close()
    return dict(datasets=D, chains=D * C, rows=n if np.isscalar(n) else list(n), sweeps=sweeps, device_ms=ms, proposals=p1 - p0, proposals_per_s=(p1 - p0) / (ms * 1e-3))


MIXED_FEATURES = (1, 2, 3, 5, 8)


def mixed_target(X):
    """y of the mixed suite on an (n, d) X: sum_j g_j(x_j) / (j + 1) with g_j cycling through x, x^2, sin x, cos x, plus the
    interaction x_0 x_{d-1} when d > 1"""
    g = (lambda v: v, lambda v: v * v, np.sin, np.cos)
    y = sum(g[j % 4](X[:, j]) / (j + 1) for j in range(X.shape[1]))
    return y + (X[:, 0] * X[:, -1] if X.shape[1] > 1 else 0.0)


def bench_mixed(repeats, rounds, n):
    """fit loop against fit_many(mixed_features=True) on data sets of 1 ... 8 features"""
    import torch
    from sklearn.base import clone
    from mcmc_symreg_b200 import BSR
    rng = np.random.default_rng(12345)
    feats = [d for d in MIXED_FEATURES for _ in range(repeats)]
    pairs = []
    for d in feats:
        X = rng.uniform(-3, 3, (n, d))
        pairs.append((X, mixed_target(X)))
    seeds = list(range(len(pairs)))
    est = BSR(3, 50, val=100)

    def loop():
        out = [clone(est).set_params(seed=s) for s in seeds]
        for e, (X, y) in zip(out, pairs):
            e.fit(X, y)
        torch.cuda.synchronize()
        return out

    def batch():
        out = est.fit_many(pairs, seeds=seeds, mixed_features=True)
        torch.cuda.synchronize()
        return out

    loop(); batch()                               # module loads, allocations
    t_loop, t_batch, equal = [], [], True
    for _ in range(rounds):
        t0 = time.perf_counter(); a = loop(); t_loop.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); b = batch(); t_batch.append(time.perf_counter() - t0)
        equal = equal and all(fingerprint(x) == fingerprint(y) for x, y in zip(a, b))
    assert equal, "fit_many(mixed_features=True) and the loop of fits disagree"
    return dict(datasets=len(pairs), features=list(MIXED_FEATURES), repeats=repeats, chains_per_fit=50, rows=n, loop_seconds=t_loop,
                fit_many_seconds=t_batch, loop_ms_per_fit=1e3 * float(np.median(t_loop)) / len(pairs),
                fit_many_ms_per_fit=1e3 * float(np.median(t_batch)) / len(pairs), speedup_median=float(np.median(t_loop) / np.median(t_batch)),
                results_equal=equal)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--repeats", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rows", default="100", help="rows per data set, or a comma list of sizes (30,100,300,1000)")
    ap.add_argument("--sweeps", type=int, default=300)
    ap.add_argument("--datasets", default="1,16,128,1024")
    ap.add_argument("--sections", default="suite,summaries,engine,mixed", help="comma list of the sections to run")
    a = ap.parse_args(argv)
    sections = set(a.sections.split(","))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_fit_many: needs a CUDA device")
    import __graft_entry__ as g
    g.build()
    name, power = gpu_info()
    out = dict(gpu=name, power_limit=power)
    sizes = [int(v) for v in a.rows.split(",")]
    Ds = [int(D) for D in a.datasets.split(",")]
    if "suite" in sections:
        out["suite"] = bench_suite(a.repeats, a.rounds, sizes)
    if "summaries" in sections:
        out["summaries"] = bench_summaries(a.repeats, a.rounds, sizes)
    if "engine" in sections:
        out["engine"] = [bench_engine(D, a.sweeps, sizes[0]) for D in Ds]
    if "mixed" in sections:
        out["mixed"] = bench_mixed(a.repeats, a.rounds, sizes[0])
    if "engine" in sections and len(sizes) > 1:
        # the same chains on the ragged batch and on data sets of the largest size: what rows a chain does not hold cost nothing
        r, p = bench_engine(max(Ds), a.sweeps, sizes), bench_engine(max(Ds), a.sweeps, max(sizes))
        out["engine_ragged"] = dict(ragged=r, padded=p, throughput_ratio=r["proposals_per_s"] / p["proposals_per_s"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
