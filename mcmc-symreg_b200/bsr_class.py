"""``BSR`` estimator: the reference's public API (codes/bsr_class.py:26-278) over the B200 engine.

Same constructor arguments, ``fit / predict / model / complexity`` and fitted attributes
(``roots_``, ``betas_``, ``train_err_``) as the reference.  The reference runs its ``itrNum`` independent
restarts one after another (codes/bsr_class.py:99); here they are ``itrNum`` chains stepping in lock-step on
the GPU.  Extra keyword-only arguments expose what the reference hard-codes (operator set / weights,
codes/bsr_class.py:110-112) and what a batched sampler needs (seed, sweep budget, precision, device).
"""
import numpy as np

try:  # sklearn is what the reference derives from (codes/bsr_class.py:19,26); keep get_params/set_params/score
    from sklearn.base import BaseEstimator, RegressorMixin
except Exception:  # pragma: no cover
    class BaseEstimator(object):
        pass

    class RegressorMixin(object):
        pass

from . import capi, parallel
from .trees import DEFAULT_OPS, NAME_OP, Express, decode_tree, getNum


class BSR(BaseEstimator, RegressorMixin):
    def __init__(self, treeNum=3, itrNum=5000, alpha1=0.4, alpha2=0.4, beta=-1, disp=False, val=100, *,
                 seed=None, max_sweeps=100000, fixed_sweeps=None, ops=None, op_weights=None, precision="fp32",
                 device=None, err_cap=512, plateau_rule=True, distributed=None):
        self.treeNum = treeNum
        self.itrNum = itrNum
        self.alpha1 = alpha1      # stored and never used, as in the reference (bsr_class.py:94-95)
        self.alpha2 = alpha2
        self.beta = beta
        self.disp = disp
        self.val = val
        self.seed = seed
        self.max_sweeps = max_sweeps
        self.fixed_sweeps = fixed_sweeps
        self.ops = ops
        self.op_weights = op_weights
        self.precision = precision
        self.device = device
        self.err_cap = err_cap
        self.plateau_rule = plateau_rule
        self.distributed = distributed

    # ---- reference API ------------------------------------------------------------------------------
    def model(self, last_ind=1):
        """codes/bsr_class.py:37-41"""
        return [Express(self.roots_[-last_ind][i]) for i in range(self.treeNum)]

    def complexity(self):
        """codes/bsr_class.py:43-51 (total node count of the last restart)"""
        return int(sum(getNum(self.roots_[-1][i]) for i in range(self.treeNum)))

    def predict(self, test_data, method="last", last_ind=1):
        """codes/bsr_class.py:53-68: (n_test, 1) predictions of restart ``-last_ind`` (evaluated on the GPU)."""
        X = _as_matrix(test_data)
        if method != "last":
            # the reference only implements 'last' and dies on anything else (bsr_class.py:59,68)
            raise UnboundLocalError("predict: only method='last' is implemented (as in the reference)")
        m = len(self.betas_) - last_ind
        return self._predict_chains([m], X)[0].reshape(-1, 1)

    def fit(self, train_data, train_y):
        """codes/bsr_class.py:77-278.  ``itrNum`` chains; each stops after ``val`` consecutive rejections or on
        the RMSE plateau rule, exactly as one reference restart does."""
        X = _as_matrix(train_data)
        y = np.asarray(train_y, dtype=np.float64).ravel()
        if X.shape[0] != y.shape[0]:
            raise ValueError("train_data and train_y disagree on the number of rows")
        MM, K = int(self.itrNum), int(self.treeNum)
        opcodes, w = self._op_tables()
        seed = self.seed
        if seed is None:          # the reference draws from the global numpy state; so does the default seed
            seed = int(np.random.randint(0, 2 ** 31 - 1))
        dist = parallel.context(self.distributed)
        seed = dist.broadcast_int(seed)
        lo, hi = parallel.shard_range(MM, dist.rank, dist.world)
        fixed = self.fixed_sweeps is not None
        res = None
        if hi > lo:
            eng = capi.Engine(K, hi - lo, opcodes, w, beta=float(self.beta), val=(0 if fixed else int(self.val)),
                              plateau_rule=(self.plateau_rule and not fixed), precision=self.precision,
                              err_cap=int(self.err_cap), device=self._device_index(), chain_offset=lo)
            try:
                eng.set_data(X, y)
                eng.init_chains(seed)
                if self.disp:
                    print("starting training...")
                if fixed:
                    eng.run(int(self.fixed_sweeps))
                    sweeps = int(self.fixed_sweeps)
                else:
                    # 32 sweeps per stop-rule check; the RMSE-at-accept trace grows between checks (never truncated)
                    sweeps = eng.run_until_done(int(self.max_sweeps), check_every=32)
                res = parallel.collect(eng)
                res["sweeps"] = sweeps
            finally:
                eng.close()
        res = dist.gather_results(res, MM, K)
        self._set_results(res)
        n_open = int(MM - np.count_nonzero(self.done_))
        if n_open and not fixed:
            # the reference loops until its stop rule fires (bsr_class.py:174); a sweep budget that ends earlier is said out loud
            import warnings
            warnings.warn("BSR.fit: %d of %d restarts had not met their stop rule after max_sweeps = %d sweeps; roots_ / betas_ hold "
                          "their current states (see done_)" % (n_open, MM, int(self.max_sweeps)), RuntimeWarning)
        if self.disp:
            c = res["counters"]
            print("chains: %d  proposals: %d  accepts: %d  rank-rejects: %d" % (MM, c[:, 0].sum(), c[:, 1].sum(), c[:, 2].sum()))
        return

    def fit_many(self, datasets, seeds=None, *, ragged=False, mixed_features=False, params=None):
        """Fit this estimator to each of several data sets in one GPU run; returns one fitted ``BSR`` per data set.

        ``datasets``: a sequence of (X, y) pairs of the same shape (n rows, d features); with ``ragged=True`` the row counts may
        differ (a learning curve, cross-validation folds, groups of different sizes), the number of features may not.  The
        ``itrNum`` restarts of every data set run as chains of one handle (chains never interact), so the B fits share one upload,
        one sequence of launches and one result read.  Estimator b is identical -- ``roots_`` / ``model()``, ``betas_``,
        ``train_err_``, ``train_err_truncated_``, ``counters_``, ``done_``, ``final_rmse_`` and every ``predict*`` -- to
        ``clone(self).set_params(seed=seeds[b]).fit(*datasets[b])``: its chains draw from Philox under the keys
        (seeds[b], 0 ... itrNum - 1) that fit gives them.  This holds whenever the window geometry of the batch equals that of
        a single fit, which it always does below 16384 rows; above, with few chains, the row-split count depends on the chain
        count and the results agree up to the fp64 summation order of the splits.  With ``ragged=True`` the batch takes the
        geometry of its largest data set, and data set b is identical to its fit when its n_b rows fit in the batch's first row
        split and its own fit runs one split (always below 16384 rows), else equal up to the fp64 summation order of the splits.
        With equal row counts ``ragged=True`` gives the estimators ``ragged=False`` gives.  With ``mixed_features=True`` the row counts
        and the numbers of features may both differ (a benchmark suite of problems with 1 to 9 inputs): every data set's chains draw
        their leaf features from its own d_b features and charge its own tree prior, so data set b is identical to its fit under the
        condition ``ragged=True`` states (n_b in the batch's first row split, its own fit one split: always below 16384 rows), else
        equal up to the fp64 summation order of the splits.  The device holds every data set with the columns of the widest (zeros
        no chain reads), B * d_max * n_max values per precision.  With one feature count ``mixed_features=True`` gives the
        estimators ``ragged=True`` gives.  ``n_sweeps_`` reports the sweeps of the
        whole batch (the stop rules are checked for all chains together), not the count a single fit would have needed.

        ``seeds``: one seed per data set; None gives every data set ``self.seed``, or, when that is None, draws one seed per
        data set from numpy's global state, in order, exactly as a loop of ``fit`` calls would.  The returned estimators
        carry the parameters of ``self``.

        ``params``: None, or one dict per entry of ``datasets`` overriding the settings ``GRID_PARAMS`` names (``beta``, ``ops``,
        ``op_weights``, ``val``, ``plateau_rule`` and the inert ``alpha1``, ``alpha2``) for that entry: a grid of prior settings
        over cross-validation folds in one run.  Estimator b then equals ``clone(self).set_params(seed=seeds[b], **params[b])
        .fit(*datasets[b])`` under the same row-split conditions, and its ``get_params()`` carries the overrides.  Every other key
        raises ValueError before any library call (``treeNum``, ``itrNum``, ``precision``, the sweep budgets, ``err_cap``, ``device``
        and ``distributed`` shape the whole run).  Under ``fixed_sweeps`` the stop rule is off for every entry, as in ``fit``.
        Entries whose X and y are the same objects as an earlier entry's share its upload (a grid of G settings over F folds
        uploads F data sets)."""
        datasets = list(datasets)
        entries = grid_estimators(self, params, len(datasets))
        data = [(_as_matrix(X), np.asarray(y, dtype=np.float64).ravel()) for X, y in datasets]
        check_datasets(data, ragged, mixed_features)
        B = len(data)
        uploads, entry_ds = shared_uploads(datasets)
        data = [data[b] for b in uploads]
        seeds = dataset_seeds(self.seed, B, seeds)
        MM, K = int(self.itrNum), int(self.treeNum)
        opcodes, w = self._op_tables()
        dist = parallel.context(self.distributed)
        seeds = [dist.broadcast_int(s) for s in seeds]
        lo, hi = parallel.shard_range(B * MM, dist.rank, dist.world)
        fixed = self.fixed_sweeps is not None
        res = None
        if hi > lo:
            eng = capi.Engine(K, hi - lo, opcodes, w, beta=float(self.beta), val=(0 if fixed else int(self.val)),
                              plateau_rule=(self.plateau_rule and not fixed), precision=self.precision,
                              err_cap=int(self.err_cap), device=self._device_index(), chain_offset=lo)
            try:
                g = np.arange(lo, hi)
                entry, ids = g // MM, g % MM
                ds = entry_ds[entry]
                if entries is not None:
                    eng.set_chain_priors([e._prior(fixed) for e in entries], entry)
                if mixed_features:
                    eng.set_datasets_mixed([X for X, _ in data], [y for _, y in data], ds)
                elif ragged:
                    eng.set_datasets_ragged([X for X, _ in data], [y for _, y in data], ds)
                else:
                    eng.set_datasets(np.stack([X for X, _ in data]), np.stack([y for _, y in data]), ds)
                eng.init_chains_keyed(np.asarray(seeds, dtype=object)[entry], ids)
                if fixed:
                    eng.run(int(self.fixed_sweeps))
                    sweeps = int(self.fixed_sweeps)
                else:
                    sweeps = eng.run_until_done(int(self.max_sweeps), check_every=32)
                res = parallel.collect(eng)
                res["sweeps"] = sweeps
            finally:
                eng.close()
        res = dist.gather_results(res, B * MM, K)
        fits = []
        for b, part in enumerate(parallel.split_results(res, B, MM)):
            est = type(self)(**(self if entries is None else entries[b]).get_params())
            est._set_results(part)
            fits.append(est)
        open_sets = [b for b, est in enumerate(fits) if not np.all(est.done_)]
        if open_sets and not fixed:
            import warnings
            warnings.warn("BSR.fit_many: data sets %s have restarts that had not met their stop rule after max_sweeps = %d sweeps; "
                          "their roots_ / betas_ hold the current states (see done_)" % (open_sets, int(self.max_sweeps)), RuntimeWarning)
        return fits

    @staticmethod
    def predict_many(fits, test_data, method="last", last_ind=1, return_std=False):
        """Predict many fitted estimators, each on its own test set, in one GPU call; returns one result per fit.

        ``fits``: fitted estimators of one ``treeNum`` and device (``fit_many``'s result, cross-validation folds, ...);
        ``test_data``: one X per fit, row counts may differ.  ``method="last"`` gives ``fit.predict(X, last_ind=last_ind)``,
        ``"best"`` ``fit.predict_best(X)``, ``"mean"`` ``fit.predict_mean(X, return_std=return_std)`` (and sets each fit's
        ``n_used_`` as that does): (n_b, 1) arrays, or (mean, std) pairs, bit for bit what those methods return.  All models go up
        in one upload and are evaluated in one launch (``bsr_predict_groups``)."""
        fits, test_data = list(fits), list(test_data)
        if len(fits) != len(test_data):
            raise ValueError("predict_many: %d fits and %d test sets" % (len(fits), len(test_data)))
        if method not in ("last", "best", "mean"):
            raise ValueError("predict_many: method must be 'last', 'best' or 'mean', not %r" % (method,))
        if not fits:
            return []
        check_same_engine(fits)
        Xs = [_as_matrix(X) for X in test_data]
        if method == "last":
            sel = []
            for b, f in enumerate(fits):
                m = len(f.betas_) - last_ind
                if not 0 <= m < len(f.betas_):
                    raise ValueError("predict_many: last_ind = %r is outside 1 .. %d for fit %d" % (last_ind, len(f.betas_), b))
                sel.append([m])
        elif method == "best":
            sel = [[f.best_chain()] for f in fits]
        else:
            sel = [np.arange(len(f.betas_)) for f in fits]
        blocks, used = predict_fit_groups(fits, Xs, [(b, b, idx, method == "mean") for b, idx in enumerate(sel)])
        if method != "mean":
            return [blk[0].reshape(-1, 1) for blk in blocks]
        out = []
        for f, blk, u in zip(fits, blocks, used):
            f.n_used_ = int(u)
            out.append((blk[0].reshape(-1, 1), blk[1].reshape(-1, 1)) if return_std else blk[0].reshape(-1, 1))
        return out

    # ---- beyond the reference: what a batch of restarts allows (SURVEY.md 8f 1, 3) ----------------------
    def best_chain(self):
        """Index of the restart with the lowest training RMSE at its last accept (codes/simulations.py:127-128 picks restarts
        by their training error by hand).  Restarts that never accepted rank by the RMSE of their initial fit."""
        return int(np.nanargmin(self.final_rmse_))

    def predict_best(self, test_data):
        """predict() of the best restart instead of the last one (the reference reads the last: quirk Q17)."""
        return self._predict_chains([self.best_chain()], _as_matrix(test_data))[0].reshape(-1, 1)

    def predict_mean(self, test_data, chains=None, return_std=False):
        """Posterior-predictive mean over restarts: every restart's model is evaluated on the GPU (float64) and the predictions
        are averaged on the device; restarts whose prediction is not finite are left out.  ``chains``: indices to use
        (default: all).  Returns (n_test, 1) [and the per-row standard deviation across restarts]."""
        X = _as_matrix(test_data)
        idx = np.arange(len(self.betas_)) if chains is None else np.asarray(chains, dtype=np.int64)
        mean, std, used = self._predict_chains(idx, X, reduce=True)
        self.n_used_ = int(used)
        return (mean.reshape(-1, 1), std.reshape(-1, 1)) if return_std else mean.reshape(-1, 1)

    def chain_diagnostics(self, tail=0.5):
        """Across-restart convergence summary: the best restart, the spread of the final training RMSE, and the Gelman-Rubin
        statistic R-hat of log RMSE-at-accept over the last ``tail`` share of the accepts, on the restarts that have at least
        the median number of accepts (traces cut to that common length)."""
        lens = np.array([len(e) for e in self.train_err_])
        out = dict(best=self.best_chain(), final_rmse_median=float(np.nanmedian(self.final_rmse_)),
                   final_rmse_best=float(np.nanmin(self.final_rmse_)), accepts_median=float(np.median(lens)))
        L = int(np.median(lens))
        sel = [np.log(np.asarray(e[:L])) for e in self.train_err_ if len(e) >= L and L >= 4]
        if len(sel) >= 2:
            A = np.stack(sel)[:, int(L * (1 - tail)):]
            A = A[np.all(np.isfinite(A), axis=1)]
        if len(sel) >= 2 and A.shape[0] >= 2 and A.shape[1] >= 2:
            n = A.shape[1]
            W = float(np.mean(np.var(A, axis=1, ddof=1)))
            B = float(n * np.var(np.mean(A, axis=1), ddof=1))
            out["rhat"] = float(np.sqrt(((n - 1) / n * W + B / n) / W)) if W > 0 else float("inf")
            out["rhat_chains"], out["rhat_length"] = int(A.shape[0]), int(n)
        else:
            out["rhat"] = float("nan")
        return out

    # ---- helpers ------------------------------------------------------------------------------------
    def _op_tables(self):
        ops = list(self.ops) if self.ops is not None else list(DEFAULT_OPS)
        opcodes = [NAME_OP[o] if isinstance(o, str) else int(o) for o in ops]
        w = list(self.op_weights) if self.op_weights is not None else [1.0 / len(ops)] * len(ops)
        return opcodes, w

    def _prior(self, fixed):
        """this estimator's settings as ``capi.Engine.set_chain_priors`` takes them (the stop rule off under ``fixed_sweeps``)"""
        opcodes, w = self._op_tables()
        return dict(ops=opcodes, op_weights=w, beta=float(self.beta), val=(0 if fixed else int(self.val)),
                    plateau_rule=(bool(self.plateau_rule) and not fixed))

    def _device_index(self):
        if self.device is not None:
            return int(self.device)
        return parallel.default_device()

    def _predict_chains(self, idx, X, reduce=False):
        """The restarts ``idx`` on X as one group of one ``capi.predict_groups`` call: their (len(idx), n) predictions, or, with
        ``reduce``, (mean, std, n_used) over them.  Only their rows of the packed table go to the device (a large fit's whole table
        would cost predict() of one restart more than the prediction).  An index outside [0, len(betas_)) raises IndexError."""
        idx = np.asarray(idx, dtype=np.int64).ravel()
        bad = idx[(idx < 0) | (idx >= len(self.betas_))]
        if bad.size:
            raise IndexError("restart index %d is outside 0 .. %d" % (int(bad[0]), len(self.betas_) - 1))
        pk = self._packed_.select(idx)
        beta = np.stack([np.asarray(self.betas_[m], dtype=np.float64).ravel() for m in idx])
        blocks, used = capi.predict_groups(self._device_index(), pk.nn, pk.tok, pk.ab, beta, [X], [0], [np.arange(idx.size)], [reduce])
        if reduce:
            return blocks[0][0], blocks[0][1], int(used[0])
        return blocks[0]

    def _set_results(self, res):
        self._packed_ = capi.PackedTrees(res["nn"], res["ptok"], res["pab"])
        MM, K = res["nn"].shape
        self.roots_ = _LazyRoots(self._packed_)
        self.betas_ = [res["beta"][m].reshape(K + 1, 1).copy() for m in range(MM)]
        ne = res["nerr"]
        cap = res["err"].shape[1]
        # the newest min(nerr, capacity) entries; run_until_done grows the capacity, so nothing is lost under fit()
        self.train_err_ = [[float(v) for v in res["err"][m, :min(int(ne[m]), cap)]] for m in range(MM)]
        self.train_err_truncated_ = bool(np.any(ne > cap))
        self.counters_ = res["counters"]
        self.done_ = res["done"].astype(bool)
        self.n_sweeps_ = res.get("sweeps")
        # RMSE of every restart's final state: its last accept, or the initial fit (K-column SSE is not it: use the trace / nan)
        self.final_rmse_ = np.array([e[-1] if e else np.nan for e in self.train_err_])
        if np.all(np.isnan(self.final_rmse_)):
            self.final_rmse_ = np.sqrt(np.maximum(res["sse"], 0) / max(1, res.get("n_rows", 1)))

    @property
    def _enc_(self):
        """dense [MM][K][64] encodings (tok, pa, pb, nn) of roots_"""
        return self._packed_.dense()

    def __getstate__(self):
        return dict(self.__dict__)


class _LazyRoots:
    """``roots_``: a list (over restarts) of lists of K ``Node`` trees, decoded from the packed device result on first access
    (a fit of thousands of restarts does not pay for Python tree objects nobody looks at)."""

    def __init__(self, packed):
        self._pk, self._cache = packed, {}

    def __len__(self):
        return self._pk.nn.shape[0]

    def _get(self, m):
        if m not in self._cache:
            K = self._pk.nn.shape[1]
            self._cache[m] = [decode_tree(*self._pk.tree(m, k)) for k in range(K)]
        return self._cache[m]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._get(m) for m in range(*i.indices(len(self)))]
        n = len(self)
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError("list index out of range")
        return self._get(i)

    def __iter__(self):
        return (self._get(m) for m in range(len(self)))

    def __getstate__(self):
        return dict(_pk=self._pk, _cache={})


def check_datasets(data, ragged=False, mixed_features=False):
    """``fit_many``'s data sets, as (X (n, d), y) pairs, must share n (unless ``ragged`` or ``mixed_features``) and d (unless
    ``mixed_features``), and each X must agree with its y: else ValueError."""
    if len(data) == 0:
        raise ValueError("fit_many: no data sets")
    n, d = data[0][0].shape
    for b, (X, y) in enumerate(data):
        if X.shape[0] != y.shape[0]:
            raise ValueError("fit_many: data set %d: train_data and train_y disagree on the number of rows" % b)
        if mixed_features:
            if X.shape[1] < 1:
                raise ValueError("fit_many: data set %d has no features" % b)
            continue
        if ragged and X.shape[1] != d:
            raise ValueError("fit_many: data set %d has %d features, data set 0 has %d: all data sets must have the same number of features"
                             " (mixed_features=True accepts different feature counts)" % (b, X.shape[1], d))
        if not ragged and X.shape != (n, d):
            raise ValueError("fit_many: data set %d is %d x %d, data set 0 is %d x %d: all data sets must have the same shape%s"
                             % (b, X.shape[0], X.shape[1], n, d, " (ragged=True accepts different row counts)" if X.shape[1] == d else ""))


GRID_PARAMS = ("beta", "ops", "op_weights", "val", "plateau_rule", "alpha1", "alpha2")


def grid_estimators(est, params, n_entries):
    """``fit_many``'s ``params``: None (returns None), or one dict per entry of keys in ``GRID_PARAMS``; returns the estimator of
    every entry, ``est`` with the entry's overrides.  ValueError for a wrong length, any other key, an unknown operator name, or
    operators and weights of different lengths -- all before any library call."""
    if params is None:
        return None
    params = list(params)
    if len(params) != n_entries:
        raise ValueError("fit_many: %d params for %d data sets" % (len(params), n_entries))
    known = est.get_params()
    out = []
    for b, p in enumerate(params):
        for k in p:
            if k in GRID_PARAMS:
                continue
            if k in known:
                raise ValueError("fit_many: params[%d] sets %r, which every entry of one run shares; only %s may differ"
                                 % (b, k, ", ".join(GRID_PARAMS)))
            raise ValueError("fit_many: params[%d] sets %r, which is not a parameter of %s" % (b, k, type(est).__name__))
        e = type(est)(**dict(known, **p))
        ops = list(e.ops) if e.ops is not None else list(DEFAULT_OPS)
        bad = [o for o in ops if isinstance(o, str) and o not in NAME_OP]
        if bad:
            raise ValueError("fit_many: params[%d]: unknown operator %r (known: %s)" % (b, bad[0], ", ".join(sorted(NAME_OP))))
        opcodes, w = e._op_tables()
        if len(w) != len(opcodes):
            raise ValueError("fit_many: params[%d]: %d operators and %d op_weights" % (b, len(opcodes), len(w)))
        out.append(e)
    return out


def shared_uploads(datasets):
    """Entries of ``datasets`` whose X and y are the same objects as an earlier entry's share its upload: returns the entries
    uploaded (first of each such group, in order) and every entry's index among them.  Compared by identity, not by value."""
    first, uploads, entry_ds = {}, [], []
    for b, (X, y) in enumerate(datasets):
        key = (id(X), id(y))
        if key not in first:
            first[key] = len(uploads)
            uploads.append(b)
        entry_ds.append(first[key])
    return uploads, np.asarray(entry_ds, dtype=np.int64)


def check_same_engine(fits):
    """The fits one grouped prediction serves must share ``treeNum`` and device (else ValueError) and be fitted (else the
    AttributeError ``predict`` raises on an unfitted estimator)."""
    K, dev = int(fits[0].treeNum), fits[0]._device_index()
    for b, f in enumerate(fits):
        if int(f.treeNum) != K:
            raise ValueError("predict_many: fit %d has treeNum = %d, fit 0 has %d" % (b, int(f.treeNum), K))
        if f._device_index() != dev:
            raise ValueError("predict_many: fit %d is on device %d, fit 0 on device %d" % (b, f._device_index(), dev))
    for f in fits:
        len(f.betas_)                 # an unfitted estimator: AttributeError, as from predict


def predict_fit_groups(fits, test_sets, groups):
    """The models of several fits on several test sets in one ``capi.predict_groups`` call.  ``groups``: (fit b, test set s, model
    indices within fit b, reduce) tuples.  The fits' packed trees are concatenated as they are (no per-tree work on the host).
    Returns (blocks, n_used) of ``capi.predict_groups``."""
    check_same_engine(fits)
    K = int(fits[0].treeNum)
    pk = capi.PackedTrees.concat([f._packed_ for f in fits])
    first = np.zeros(len(fits) + 1, dtype=np.int64)
    np.cumsum([f._packed_.nn.shape[0] for f in fits], out=first[1:])
    beta = np.concatenate([np.asarray(f.betas_, dtype=np.float64).reshape(-1, K + 1) for f in fits])
    return capi.predict_groups(fits[0]._device_index(), pk.nn, pk.tok, pk.ab, beta, test_sets, [s for _, s, _, _ in groups],
                               [first[b] + np.asarray(idx, dtype=np.int64) for b, _, idx, _ in groups], [r for _, _, _, r in groups])


def dataset_seeds(seed, n_datasets, seeds=None):
    """One seed per data set of ``fit_many``: ``seeds`` as given, else ``seed`` for all, else (seed None) one draw per data set from
    numpy's global state -- the draws a loop of ``fit`` calls would make, in the same order."""
    if seeds is not None:
        seeds = [int(s) for s in seeds]
        if len(seeds) != n_datasets:
            raise ValueError("fit_many: %d seeds for %d data sets" % (len(seeds), n_datasets))
        return seeds
    if seed is not None:
        return [int(seed)] * n_datasets
    return [int(np.random.randint(0, 2 ** 31 - 1)) for _ in range(n_datasets)]


def _as_matrix(data):
    if hasattr(data, "values"):
        data = data.values
    X = np.asarray(data, dtype=np.float64)
    if X.ndim == 1:
        X = X.reshape(-1, 1)
    return np.ascontiguousarray(X)
