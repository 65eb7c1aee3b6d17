"""Experiment drivers: what the reference's scripts do around ``BSR`` (SURVEY.md 8f 4).

``codes/simulations.py:60-107`` draws a training set and two test sets (the training range and twice that range) for one
benchmark function, fits ``BSR(K, MM)``, predicts and shows the trees; ``codes/BSR.py`` is the same recipe as a usage
template; ``archive/data_generate_funcs.py`` holds the generators of the paper's benchmark functions.  Here the same
recipe is one call -- ``run_experiment`` -- and a command line (``python -m mcmc_symreg_b200.experiments --func f6``),
with the restarts running as chains on the GPU and the summaries the scripts produce by hand (RMSE on the training
range and under extrapolation, model size, expressions, best restart, across-restart diagnostics) returned as a dict.

The genetic-programming comparison of the script (gplearn, ``codes/simulations.py:150-175``) is not rebuilt.
"""
import argparse
import json
import sys
import time

import numpy as np

# The benchmark suite: the paper's f1 ... f6 (bsr_paper.pdf p.5, Eqs. 3-8); "sim" is the function the script itself uses
# (codes/simulations.py:71, = f6).  All take an (n, 2) matrix.
TARGETS = {
    "f1": (lambda X: 2.5 * X[:, 0] ** 4 - 1.3 * X[:, 0] ** 3 + 0.5 * X[:, 1] ** 2 - 1.7 * X[:, 1], "2.5 x0^4 - 1.3 x0^3 + 0.5 x1^2 - 1.7 x1"),
    "f2": (lambda X: 8 * X[:, 0] ** 2 + 8 * X[:, 1] ** 3 - 15, "8 x0^2 + 8 x1^3 - 15"),
    "f3": (lambda X: 0.2 * X[:, 0] ** 3 + 0.5 * X[:, 1] ** 3 - 1.2 * X[:, 1] - 0.5 * X[:, 0], "0.2 x0^3 + 0.5 x1^3 - 1.2 x1 - 0.5 x0"),
    "f4": (lambda X: 1.5 * np.exp(X[:, 0]) + 5 * np.cos(X[:, 1]), "1.5 exp(x0) + 5 cos(x1)"),
    "f5": (lambda X: 6.0 * np.sin(X[:, 0]) * np.cos(X[:, 1]), "6 sin(x0) cos(x1)"),
    "f6": (lambda X: 1.35 * X[:, 0] * X[:, 1] + 5.5 * np.sin((X[:, 0] - 1) * (X[:, 1] - 1)), "1.35 x0 x1 + 5.5 sin((x0 - 1)(x1 - 1))"),
}
TARGETS["sim"] = TARGETS["f6"]


def make_dataset(func, n_train=100, n_test=30, lo=-3.0, hi=3.0, extrapolate=2.0, seed=None):
    """Training set on U(lo, hi)^2, a test set on the same range and one on the range stretched by ``extrapolate``
    (codes/simulations.py:64-85: n = 100 on (-3, 3), 30 + 30 test points on (-3, 3) and (-6, 6)).  ``seed=None`` draws from
    numpy's global state like the script does."""
    f = TARGETS[func][0]
    rng = np.random.default_rng(seed) if seed is not None else np.random
    X = rng.uniform(lo, hi, (n_train, 2))
    Xt = rng.uniform(lo, hi, (n_test, 2))
    Xe = rng.uniform(lo * extrapolate, hi * extrapolate, (n_test, 2))
    return dict(func=func, formula=TARGETS[func][1], X=X, y=f(X), X_test=Xt, y_test=f(Xt), X_extra=Xe, y_extra=f(Xe))


def rmse(pred, y):
    with np.errstate(all="ignore"):
        return float(np.sqrt(np.mean((np.asarray(pred).ravel() - np.asarray(y).ravel()) ** 2)))


SETS = (("train", "X", "y"), ("test", "X_test", "y_test"), ("extrapolation", "X_extra", "y_extra"))


def summarize(est, data):
    """What the script reads off a fitted estimator (codes/simulations.py:98-107, 127-128 and the commented diagnostics)."""
    preds = {}
    for tag, Xk, _ in SETS:
        # the reference's own answer (the last restart), the best restart, the posterior-predictive mean over restarts
        preds[tag] = (est.predict(data[Xk]), est.predict_best(data[Xk]), est.predict_mean(data[Xk]))
    return _summary(est, data, preds)


def summarize_many(fits, data):
    """``[summarize(e, d) for e, d in zip(fits, data)]`` with the 3 x 3 predictions of every fit (last, best, mean on the training,
    test and extrapolation sets) made by one grouped GPU call (``bsr_predict_groups``) instead of 9 calls per fit.  Sets each fit's
    ``n_used_`` as ``summarize`` does."""
    from .bsr_class import _as_matrix, predict_fit_groups
    fits, data = list(fits), list(data)
    if len(fits) != len(data):
        raise ValueError("summarize_many: %d fits and %d data sets" % (len(fits), len(data)))
    if not fits:
        return []
    sets, groups = [], []
    for b, (est, dat) in enumerate(zip(fits, data)):
        M, best = len(est.betas_), est.best_chain()
        for _, Xk, _ in SETS:
            s = len(sets)
            sets.append(_as_matrix(dat[Xk]))
            groups += [(b, s, [M - 1], False), (b, s, [best], False), (b, s, np.arange(M), True)]
    blocks, used = predict_fit_groups(fits, sets, groups)
    rows = []
    for b, (est, dat) in enumerate(zip(fits, data)):
        g = 3 * len(SETS) * b
        preds = {tag: tuple(blocks[g + 3 * i + j][0] for j in range(3)) for i, (tag, _, _) in enumerate(SETS)}
        est.n_used_ = int(used[g + 3 * len(SETS) - 1])              # predict_mean on the last set, as in summarize
        rows.append(_summary(est, dat, preds))
    return rows


def _summary(est, data, preds):
    """summarize's row from its predictions: preds[tag] = (last, best, mean) on the set of that tag."""
    best = est.best_chain()
    out = dict(func=data["func"], formula=data["formula"], restarts=len(est.betas_), K=est.treeNum)
    for tag, _, yk in SETS:
        for kind, p in zip(("last", "best", "mean"), preds[tag]):
            out["rmse_%s_%s" % (tag, kind)] = rmse(p, data[yk])
    out["model_last"] = est.model()
    out["complexity_last"] = est.complexity()
    out["model_best"] = est.model(last_ind=len(est.betas_) - best)
    out["beta_best"] = [float(v) for v in np.asarray(est.betas_[best]).ravel()]
    nn = est._packed_.nn
    out["complexity_best"] = int(nn[best].sum())
    out["complexity_mean"] = float(nn.sum(axis=1).mean())
    c = est.counters_
    out["proposals"] = int(c[:, 0].sum())
    out["accept_rate"] = float(c[:, 1].sum() / max(1, c[:, 0].sum()))
    out["accepts_per_restart"] = float(np.mean([len(e) for e in est.train_err_]))
    out["diagnostics"] = est.chain_diagnostics()
    return out


def run_experiment(func="sim", K=3, MM=50, n_train=100, n_test=30, val=100, seed=0, data_seed=None, **bsr_kwargs):
    """One benchmark function end to end: data, ``BSR(K, MM).fit``, predictions on both test sets, summaries."""
    from .bsr_class import BSR
    data = make_dataset(func, n_train, n_test, seed=seed if data_seed is None else data_seed)
    est = BSR(K, MM, val=val, seed=seed, **bsr_kwargs)
    t0 = time.perf_counter()
    est.fit(data["X"], data["y"])
    out = summarize(est, data)
    out["fit_seconds"] = time.perf_counter() - t0
    return out, est, data


def suite_jobs(funcs, repeats, n_train=100, seed=0):
    """The data sets of ``run_suite`` as (function, n_train, repeat, seed), function by function, then training size (``n_train``: one
    size or a sequence of sizes), then repeat.  Repeat r draws its data and its chains from seed + r at every size, so the training
    sets of a learning curve share their draws."""
    sizes = [int(n_train)] if np.isscalar(n_train) else [int(n) for n in n_train]
    return [(f, n, r, seed + r) for f in funcs for n in sizes for r in range(repeats)]


def run_suite(funcs=("f1", "f2", "f3", "f4", "f5", "f6"), repeats=1, batched=False, params=None, **kw):
    """The whole benchmark suite (the paper's Table 1 recipe: every function, ``repeats`` independent data sets).

    ``n_train`` may be a sequence of training sizes: the suite then runs every function at every size (a learning curve), and every
    row carries its ``n_train``.  ``params``: None, or a list of dicts of estimator settings (``beta``, ``ops``, ``op_weights``, ``val``,
    ``plateau_rule``): every (function, size, repeat) job then runs once per dict, job by job, and every row carries its ``params``.
    batched=True fits all data sets in one GPU run (``BSR.fit_many``, ``ragged=True`` for several sizes, one upload per job and
    ``params`` for the settings) with the seeds the loop uses and summarizes the fits with one grouped prediction call
    (``summarize_many``); the rows are the loop's rows, except that ``fit_seconds`` is the batch's wall clock (fit and summaries)
    divided by the number of fits, and ``batch_seconds`` is that wall clock."""
    rows = []
    seed0 = kw.pop("seed", 0)
    n_train = kw.pop("n_train", 100)
    grid = not np.isscalar(n_train)
    jobs = suite_jobs(funcs, repeats, n_train, seed0)
    settings = [None] if params is None else [dict(p) for p in params]
    runs = [(job, p) for job in jobs for p in settings]
    if not batched:
        for (f, n, r, s), p in runs:
            out, _, _ = run_experiment(f, n_train=n, seed=s, **dict(kw, **(p or {})))
            if grid:
                out["n_train"] = n
            out["repeat"] = r
            if p is not None:
                out["params"] = p
            rows.append(out)
        return rows
    from .bsr_class import BSR
    K, MM, n_test, val = kw.pop("K", 3), kw.pop("MM", 50), kw.pop("n_test", 30), kw.pop("val", 100)
    data_seed = kw.pop("data_seed", None)
    data = [make_dataset(f, n, n_test, seed=s if data_seed is None else data_seed) for f, n, _, s in jobs]
    run_data = [d for d in data for _ in settings]
    t0 = time.perf_counter()
    fits = BSR(K, MM, val=val, **kw).fit_many([(d["X"], d["y"]) for d in run_data], seeds=[s for (_, _, _, s), _ in runs], ragged=grid,
                                              params=None if params is None else [p for _, p in runs])
    rows = summarize_many(fits, run_data)
    batch = time.perf_counter() - t0
    for o, ((_, n, r, _), p) in zip(rows, runs):
        o["fit_seconds"] = batch / len(runs)
        o["batch_seconds"] = batch
        if grid:
            o["n_train"] = n
        o["repeat"] = r
        if p is not None:
            o["params"] = p
    return rows


def format_row(o):
    return ("%-4s restarts %5d | RMSE train / test / extrapolation: last %.3g / %.3g / %.3g  best %.3g / %.3g / %.3g  mean %.3g / %.3g / %.3g | "
            "nodes last %d best %d mean %.1f | accept %.2f %% | %.2f s" %
            (o["func"], o["restarts"], o["rmse_train_last"], o["rmse_test_last"], o["rmse_extrapolation_last"], o["rmse_train_best"],
             o["rmse_test_best"], o["rmse_extrapolation_best"], o["rmse_train_mean"], o["rmse_test_mean"], o["rmse_extrapolation_mean"],
             o["complexity_last"], o["complexity_best"], o["complexity_mean"], 100 * o["accept_rate"], o["fit_seconds"]))


def _sizes(text):
    """--n-train: one size (an int), or a comma list of sizes (a tuple)"""
    parts = [int(v) for v in text.split(",") if v.strip()]
    return tuple(parts) if "," in text else parts[0]


def _floats(text):
    """--beta: a comma list of numbers"""
    return [float(v) for v in text.split(",") if v.strip()]


def main(argv=None):
    ap = argparse.ArgumentParser(description="BSR benchmark-function experiments on the GPU (codes/simulations.py recipe)")
    ap.add_argument("--func", default="sim", help="one of %s, or 'all'" % ", ".join(sorted(TARGETS)))
    ap.add_argument("--K", type=int, default=3)
    ap.add_argument("--MM", type=int, default=50, help="restarts (chains on the GPU)")
    ap.add_argument("--n-train", type=_sizes, default=100, help="training rows, or a comma list of sizes (a learning curve: 30,100,300)")
    ap.add_argument("--n-test", type=int, default=30)
    ap.add_argument("--val", type=int, default=100)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--repeats", type=int, default=1)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--json", action="store_true", help="one JSON object per experiment instead of the table")
    ap.add_argument("--batched", action="store_true", help="fit all (function, size, repeat) data sets in one GPU run (BSR.fit_many)")
    ap.add_argument("--beta", type=_floats, default=None, help="split exponents to run every data set with, a comma list (-1,-0.5,-2)")
    argv = list(sys.argv[1:] if argv is None else argv)
    # "--beta -1,-0.5": argparse takes a value that starts with "-" and is not a single number for an option
    argv = [a + "=" + argv[i + 1] if a == "--beta" and i + 1 < len(argv) else a for i, a in enumerate(argv)
            if not (i > 0 and argv[i - 1] == "--beta")]
    a = ap.parse_args(argv)
    funcs = ("f1", "f2", "f3", "f4", "f5", "f6") if a.func == "all" else (a.func,)
    params = None if a.beta is None else [dict(beta=b) for b in a.beta]
    rows = run_suite(funcs, a.repeats, batched=a.batched, params=params, K=a.K, MM=a.MM, n_train=a.n_train, n_test=a.n_test, val=a.val,
                     seed=a.seed, precision=a.precision)
    for o in rows:
        if a.json:
            print(json.dumps(o))
        else:
            if "params" in o:
                print("     params %s" % json.dumps(o["params"], sort_keys=True))
            print(format_row(o))
            print("     target     y = %s" % o["formula"])
            print("     best model y = %.4g + %s" % (o["beta_best"][0], " + ".join("%.4g * [%s]" % (b, e) for b, e in zip(o["beta_best"][1:], o["model_best"]))))
    return rows


if __name__ == "__main__":
    main()
