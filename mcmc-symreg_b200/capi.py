"""ctypes binding of libbsr_b200.so (include/bsr_b200.h).  Fails loudly when the library is missing."""
import ctypes as C
import os

import numpy as np

MAX_NODES = 64
MAX_OPS = 16
N_COUNTERS = 8
TRACE_DOUBLES = 24
CNT = dict(proposals=0, accepts=1, rank_rejects=2, capacity_rejects=3, fp64_sweeps=4, node_evals_ref=5,
           node_evals_exec=6, sweeps=7)
TR = dict(move=0, change=1, Q=2, Qinv=3, hratio=4, detjacob=5, new_sigma=6, new_sa2=7, new_sb2=8, rank_reject=9,
          logR=10, accepted=11, sse_new=12, sse_old=13, ndraws=14, flags=15, u=16, fs_new=17, fs_old=18, m_new=19,
          pivot_min=20, sv_ratio=21, rank_path=22, wide=23)

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libbsr_b200.so")


class BsrConfig(C.Structure):
    _fields_ = [("K", C.c_int32), ("n_chains", C.c_int32), ("chain_offset", C.c_int64), ("n_ops", C.c_int32),
                ("ops", C.c_int32 * MAX_OPS), ("op_weights", C.c_double * MAX_OPS), ("beta", C.c_double),
                ("val", C.c_int32), ("plateau_rule", C.c_int32), ("precision", C.c_int32), ("err_cap", C.c_int32),
                ("device", C.c_int32), ("row_sharded", C.c_int32), ("reserved", C.c_int32 * 7)]


_P = C.c_void_p
_SIGS = {
    "bsr_last_error": (C.c_char_p, []),
    "bsr_version": (C.c_int, []),
    "bsr_max_nodes": (C.c_int, []),
    "bsr_create": (C.c_int, [C.POINTER(BsrConfig), C.POINTER(_P)]),
    "bsr_destroy": (C.c_int, [_P]),
    "bsr_set_data_host": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int64]),
    "bsr_set_data_device": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int64, C.c_int64]),
    "bsr_set_datasets_host": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64, C.c_int32, _P]),
    "bsr_set_datasets_ragged_host": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int32, _P]),
    "bsr_set_datasets_mixed_host": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P]),
    "bsr_init_chains": (C.c_int, [_P, C.c_uint64]),
    "bsr_init_chains_keyed": (C.c_int, [_P, _P, _P]),
    "bsr_set_state": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_uint64]),
    "bsr_run": (C.c_int, [_P, C.c_int32, _P]),
    "bsr_get_launch_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "bsr_set_launch_geometry": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "bsr_run_until_done": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.POINTER(C.c_int32)]),
    "bsr_sweep_propose": (C.c_int, [_P, _P]),
    "bsr_sweep_eval": (C.c_int, [_P, _P]),
    "bsr_sweep_resolve": (C.c_int, [_P, _P]),
    "bsr_gram_buffer": (C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bsr_get_y_stats": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "bsr_set_y_stats": (C.c_int, [_P, C.c_double, C.c_double]),
    "bsr_finish_init": (C.c_int, [_P]),
    "bsr_set_tape": (C.c_int, [_P, _P, _P, C.c_int32]),
    "bsr_get_trace": (C.c_int, [_P, _P]),
    "bsr_get_proposals": (C.c_int, [_P, _P, _P, _P, _P]),
    "bsr_trace_trees": (C.c_int, [_P]),
    "bsr_get_trace_trees": (C.c_int, [_P, _P, _P, _P, _P]),
    "bsr_set_peer_timeout": (C.c_int, [_P, C.c_double]),
    "bsr_get_exchange_profile": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "bsr_record_draws": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "bsr_get_recorded_draws": (C.c_int, [_P, _P, _P]),
    "bsr_get_trees": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P]),
    "bsr_pack_trees": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "bsr_read_packed": (C.c_int, [_P, _P, _P, _P]),
    "bsr_alloc_host": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "bsr_free_host": (C.c_int, [_P]),
    "bsr_get_stats": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "bsr_get_err_trace": (C.c_int, [_P, _P]),
    "bsr_reserve_err": (C.c_int, [_P, C.c_int32]),
    "bsr_get_err_cap": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "bsr_count_done": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "bsr_eval_trees": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, C.c_int32, _P]),
    "bsr_predict": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int64, C.c_int32, _P]),
    "bsr_predict_trees": (C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, _P]),
    "bsr_predict_many": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P,
                                   C.POINTER(C.c_int32)]),
    "bsr_predict_groups": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_int64, _P, C.c_int64, _P, C.c_int32, C.c_int32, _P, _P,
                                     C.c_int32, _P, _P, _P, _P, _P, _P]),
    "bsr_peer_export": (C.c_int, [_P, C.c_int32, _P]),
    "bsr_peer_import": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "bsr_set_window": (C.c_int, [_P, C.c_int32]),
    "bsr_get_window_geometry": (C.c_int, [_P, _P]),
    "bsr_set_pipeline": (C.c_int, [_P, C.c_int32]),
    "bsr_set_profiling": (C.c_int, [_P, C.c_int32]),
    "bsr_get_profile": (C.c_int, [_P, _P, _P]),
}
EXPORTED = sorted(_SIGS)
_lib = None


def load():
    """Load libbsr_b200.so (built in-tree by ``__graft_entry__.build()``); raises if it is missing."""
    global _lib
    if _lib is None:
        path = os.environ.get("BSR_LIB", LIB_PATH)     # A/B builds of the same library (scripts/build_variant.sh)
        if not os.path.exists(path):
            raise RuntimeError("libbsr_b200.so not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'`; "
                               "there is no CPU fallback" % path)
        lib = C.CDLL(path)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class BsrError(RuntimeError):
    pass


def _ck(rc):
    if rc != 0:
        raise BsrError(load().bsr_last_error().decode())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def predict_many(device, tok, pa, pb, nn, beta, X, reduce=False):
    """BSR.predict for M models at once (codes/bsr_class.py:53-68 per model).  tok / pa / pb: [M][K][MAX_NODES], nn [M][K],
    beta [M][K+1].  reduce=False: (M, n_test) predictions.  reduce=True: (mean, std, n_used) over the models, reduced on the
    device (a model is left out of the rows where its prediction is not finite)."""
    lib = load()
    tok = np.ascontiguousarray(tok, dtype=np.uint32)
    M, K = tok.shape[0], tok.shape[1]
    pa = np.ascontiguousarray(pa, dtype=np.float64).reshape(M, K, MAX_NODES)
    pb = np.ascontiguousarray(pb, dtype=np.float64).reshape(M, K, MAX_NODES)
    nn = np.ascontiguousarray(nn, dtype=np.int32).reshape(M, K)
    beta = np.ascontiguousarray(beta, dtype=np.float64).reshape(M, K + 1)
    X = np.ascontiguousarray(X, dtype=np.float64)
    used = C.c_int32(0)
    out = np.zeros((2 if reduce else M, X.shape[0]))
    _ck(lib.bsr_predict_many(int(device), M, K, _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn), _ptr(beta), _ptr(X), X.shape[0], X.shape[1],
                             int(bool(reduce)), _ptr(out), C.byref(used)))
    if reduce:
        return out[0], out[1], used.value
    return out


def predict_groups(device, nn, tok, ab, beta, test_sets, grp_set, grp_models, grp_reduce):
    """Many models on many test sets in one call (``bsr_predict_groups``).  Models packed as ``PackedTrees`` holds them: nn [M][K],
    tok the tokens of tree after tree, ab [n_lt][2]; beta [M][K+1].  ``test_sets``: S arrays (n_s, d_s).  Group g evaluates the
    model indices ``grp_models[g]`` on ``test_sets[grp_set[g]]``.  Returns (blocks, n_used): blocks[g] is (n_models_g, n_s), or, for
    ``grp_reduce[g]``, (2, n_s) with the mean over the models and their standard deviation (what ``predict_many`` returns for
    reduce=False / True); n_used [G] the smallest number of models any row of a group used.

    Test sets of different widths (the fits of ``fit_many(mixed_features=True)``) go to the library padded with zero columns to the
    widest; first, every model of a group must read only features below the width of its own test set (else ValueError), the check
    the library makes against the one width it is given."""
    nn = np.ascontiguousarray(nn, dtype=np.int32)
    M, K = nn.shape
    tok = np.ascontiguousarray(tok, dtype=np.uint32).ravel()
    ab = np.ascontiguousarray(ab, dtype=np.float64).reshape(-1, 2)
    beta = np.ascontiguousarray(beta, dtype=np.float64).reshape(M, K + 1)
    Xs = [np.asarray(X, dtype=np.float64) for X in test_sets]
    if not Xs or any(X.ndim != 2 for X in Xs):
        raise ValueError("predict_groups: test_sets must be one or more (n_s, d_s) arrays")
    models = [np.asarray(m, dtype=np.int32).ravel() for m in grp_models]
    G = len(models)
    grp_set = np.ascontiguousarray(grp_set, dtype=np.int32).ravel()
    grp_reduce = np.ascontiguousarray([int(bool(r)) for r in grp_reduce], dtype=np.int32)
    if grp_set.size != G or grp_reduce.size != G or G == 0:
        raise ValueError("predict_groups: grp_set, grp_models and grp_reduce must describe the same one or more groups")
    widths = np.array([X.shape[1] for X in Xs], dtype=np.int64)
    if np.any(widths != widths[0]):
        _check_group_features(nn, tok, widths, grp_set, models)
        d = int(widths.max())
        Xs = [X if X.shape[1] == d else np.pad(X, ((0, 0), (0, d - X.shape[1]))) for X in Xs]
    set_off = np.zeros(len(Xs) + 1, dtype=np.int64)
    np.cumsum([X.shape[0] for X in Xs], out=set_off[1:])
    X = np.ascontiguousarray(np.concatenate(Xs, axis=0))
    grp_off = np.zeros(G + 1, dtype=np.int64)
    np.cumsum([m.size for m in models], out=grp_off[1:])
    flat = np.ascontiguousarray(np.concatenate(models))
    rows = np.array([Xs[s].shape[0] if 0 <= s < len(Xs) else 0 for s in grp_set], dtype=np.int64)
    sizes = np.where(grp_reduce != 0, 2, grp_off[1:] - grp_off[:-1]) * rows
    out = np.zeros(int(sizes.sum()))
    used = np.zeros(G, dtype=np.int32)
    lib = load()
    _ck(lib.bsr_predict_groups(int(device), M, K, _ptr(nn), _ptr(tok), tok.size, _ptr(ab), ab.shape[0], _ptr(beta), len(Xs), X.shape[1],
                               _ptr(X), _ptr(set_off), G, _ptr(grp_set), _ptr(grp_off), _ptr(flat), _ptr(grp_reduce), _ptr(out), _ptr(used)))
    ends = np.cumsum(sizes)
    blocks = [out[e - z:e].reshape(-1, int(r)) for e, z, r in zip(ends, sizes, rows)]
    return blocks, used


def _check_group_features(nn, tok, widths, grp_set, models):
    """Every model of group g reads only features below widths[grp_set[g]]: else ValueError.  Vectorised over the packed tokens; a
    table whose node counts do not cover tok, or a group naming a model or test set that does not exist, is left to the library's
    own refusals."""
    M, K = nn.shape
    if np.any(nn < 0) or int(nn.sum()) != tok.size:
        return
    model_of = np.repeat(np.arange(M * K) // K, nn.ravel())
    leaf = (tok & 0xFF) == 0
    widest = np.full(M, -1, dtype=np.int64)             # largest leaf feature of every model
    np.maximum.at(widest, model_of[leaf], (tok[leaf] >> 16).astype(np.int64))
    for g, (s, m) in enumerate(zip(grp_set, models)):
        if not 0 <= s < widths.size:
            continue
        m = m[(m >= 0) & (m < M)]
        over = m[widest[m] >= widths[s]]
        if over.size:
            raise ValueError("predict_groups: group %d: model %d reads feature %d, its test set %d has %d features"
                             % (g, int(over[0]), int(widest[over[0]]), int(s), int(widths[s])))


class PackedTrees:
    """Trees without the padding of their device slots (``bsr_pack_trees``): ``nn`` [C][K] node counts, ``tok`` the tokens of
    tree after tree, ``ab`` the (a, b) pairs of the lt nodes in node order.  ``tree(c, k)`` / ``dense()`` give the fixed-capacity
    arrays the rest of the host code works with."""

    def __init__(self, nn, tok, ab):
        self.nn, self.tok, self.ab = nn, tok, ab
        self._off = None

    @staticmethod
    def concat(packs):
        """The models of several PackedTrees of the same K, one table after another: model m of packs[i] becomes model
        sum(models of packs[:i]) + m (its nodes and lt pairs follow those of the packs before it)."""
        return PackedTrees(np.concatenate([p.nn for p in packs]), np.concatenate([p.tok for p in packs]),
                           np.concatenate([np.asarray(p.ab, dtype=np.float64).reshape(-1, 2) for p in packs]))

    def select(self, models):
        """The models ``models`` (indices, in that order) as a table of their own: model j of the result is model models[j]."""
        off, lt_before, is_lt = self._offsets()
        models = np.asarray(models, dtype=np.int64).ravel()
        trees = (models[:, None] * self.nn.shape[1] + np.arange(self.nn.shape[1])).ravel()
        lens = off[trees + 1] - off[trees]
        node = np.repeat(off[trees] - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
        ab = np.asarray(self.ab, dtype=np.float64).reshape(-1, 2)
        return PackedTrees(self.nn[models], self.tok[node], ab[lt_before[node][is_lt[node]]])

    @property
    def nbytes(self):
        return self.nn.nbytes + self.tok.nbytes + self.ab.nbytes

    def _offsets(self):
        if self._off is None:
            flat = self.nn.reshape(-1).astype(np.int64)
            off = np.zeros(flat.size + 1, dtype=np.int64)
            np.cumsum(flat, out=off[1:])
            is_lt = (self.tok & 0xFF) == 2
            lt_before = np.zeros(self.tok.size + 1, dtype=np.int64)
            np.cumsum(is_lt, out=lt_before[1:])
            self._off = (off, lt_before, is_lt)
        return self._off

    def tree(self, c, k):
        """(tok, pa, pb, n) of one tree as MAX_NODES-long arrays"""
        off, lt_before, is_lt = self._offsets()
        g = c * self.nn.shape[1] + k
        lo, hi = off[g], off[g + 1]
        n = int(hi - lo)
        tok = np.zeros(MAX_NODES, dtype=np.uint32); pa = np.zeros(MAX_NODES); pb = np.zeros(MAX_NODES)
        tok[:n] = self.tok[lo:hi]
        sel = np.nonzero(is_lt[lo:hi])[0]
        if sel.size:
            prm = self.ab[lt_before[lo]:lt_before[hi]]
            pa[sel], pb[sel] = prm[:, 0], prm[:, 1]
        return tok, pa, pb, n

    def dense(self):
        """the [C][K][MAX_NODES] arrays of ``Engine.get_trees``"""
        off, lt_before, is_lt = self._offsets()
        Cn, K = self.nn.shape
        tok = np.zeros((Cn * K, MAX_NODES), dtype=np.uint32); pa = np.zeros((Cn * K, MAX_NODES)); pb = np.zeros((Cn * K, MAX_NODES))
        flat = self.nn.reshape(-1).astype(np.int64)
        tree_of = np.repeat(np.arange(flat.size), flat)
        pos = np.arange(self.tok.size) - np.repeat(off[:-1], flat)
        tok[tree_of, pos] = self.tok
        if self.ab.shape[0]:
            pa[tree_of[is_lt], pos[is_lt]] = self.ab[:, 0]
            pb[tree_of[is_lt], pos[is_lt]] = self.ab[:, 1]
        s = (Cn, K, MAX_NODES)
        return tok.reshape(s), pa.reshape(s), pb.reshape(s), self.nn


class Engine:
    """Thin object wrapper over one ``bsr_handle`` (one device, a contiguous range of global chain ids)."""

    def __init__(self, K, n_chains, ops, weights, beta=-1.0, val=100, plateau_rule=True, precision="fp32", err_cap=512,
                 device=0, chain_offset=0, row_sharded=False):
        lib = load()
        cfg = BsrConfig()
        cfg.K, cfg.n_chains, cfg.chain_offset = int(K), int(n_chains), int(chain_offset)
        cfg.n_ops = len(ops)
        for i, (o, w) in enumerate(zip(ops, weights)):
            cfg.ops[i] = int(o)
            cfg.op_weights[i] = float(w)
        cfg.beta = float(beta)
        cfg.val = int(val)
        cfg.plateau_rule = int(bool(plateau_rule))
        cfg.precision = {"fp32": 0, "fp64": 1}[precision]
        cfg.err_cap = int(err_cap)
        cfg.device = int(device)
        cfg.row_sharded = int(bool(row_sharded))
        self.K, self.C, self.err_cap = int(K), int(n_chains), int(err_cap)
        self.n = self.d = 0
        self._h = _P()
        _ck(lib.bsr_create(C.byref(cfg), C.byref(self._h)))
        self._lib = lib

    def _free_pinned(self):
        self._tree_pinned = None
        self._packed_pinned = None
        lib = getattr(self, "_lib", None)
        for p in getattr(self, "_pinned_ptrs", []):
            if lib is not None:
                lib.bsr_free_host(p)
        self._pinned_ptrs = []

    def close(self):
        self._free_pinned()
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.bsr_destroy(self._h)
            self._h = None

    __del__ = close

    # ---- data -------------------------------------------------------------------------------------
    def set_data(self, X, y, n_total=0):
        X = np.ascontiguousarray(X, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64).ravel()
        if X.ndim != 2 or X.shape[0] != y.shape[0]:
            raise ValueError("X must be (n, d) and y (n,)")
        self.n, self.d = X.shape
        _ck(self._lib.bsr_set_data_host(self._h, _ptr(X), _ptr(y), self.n, self.d, int(n_total)))

    def set_datasets(self, X, y, chain_dataset):
        """D data sets of the same shape: X (D, n, d), y (D, n); chain c fits data set ``chain_dataset[c]``."""
        X = np.ascontiguousarray(X, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if X.ndim != 3 or y.ndim != 2 or X.shape[:2] != y.shape:
            raise ValueError("X must be (D, n, d) and y (D, n)")
        cd = np.ascontiguousarray(chain_dataset, dtype=np.int32).ravel()
        if cd.size != self.C:
            raise ValueError("chain_dataset must hold one data set index per chain")
        _ck(self._lib.bsr_set_datasets_host(self._h, X.shape[0], _ptr(X), _ptr(y), X.shape[1], X.shape[2], _ptr(cd)))
        self.n, self.d = X.shape[1], X.shape[2]

    def set_datasets_ragged(self, Xs, ys, chain_dataset):
        """D data sets of the same number of features and any row counts: Xs a sequence of (n_b, d) arrays, ys of (n_b,) arrays; chain
        c fits data set ``chain_dataset[c]``.  ``n`` becomes the largest row count."""
        Xs = [np.asarray(X, dtype=np.float64) for X in Xs]
        ys = [np.asarray(y, dtype=np.float64).ravel() for y in ys]
        if len(Xs) == 0 or len(Xs) != len(ys):
            raise ValueError("set_datasets_ragged: one y per X, and at least one data set")
        if any(X.ndim != 2 or X.shape[0] != y.shape[0] for X, y in zip(Xs, ys)):
            raise ValueError("set_datasets_ragged: every X must be (n_b, d) and its y (n_b,)")
        d = Xs[0].shape[1]
        if any(X.shape[1] != d for X in Xs):
            raise ValueError("set_datasets_ragged: all data sets must have the same number of features")
        cd = np.ascontiguousarray(chain_dataset, dtype=np.int32).ravel()
        if cd.size != self.C:
            raise ValueError("chain_dataset must hold one data set index per chain")
        n_rows = np.array([X.shape[0] for X in Xs], dtype=np.int64)
        X = np.ascontiguousarray(np.concatenate(Xs, axis=0))
        y = np.ascontiguousarray(np.concatenate(ys))
        _ck(self._lib.bsr_set_datasets_ragged_host(self._h, len(Xs), _ptr(X), _ptr(y), _ptr(n_rows), d, _ptr(cd)))
        self.n, self.d = int(n_rows.max()), d

    def set_datasets_mixed(self, Xs, ys, chain_dataset):
        """D data sets of any row and feature counts: Xs a sequence of (n_b, d_b) arrays, ys of (n_b,) arrays; chain c fits data set
        ``chain_dataset[c]`` with its own d_b features.  ``n`` becomes the largest row count, ``d`` the largest feature count."""
        Xs = [np.asarray(X, dtype=np.float64) for X in Xs]
        ys = [np.asarray(y, dtype=np.float64).ravel() for y in ys]
        if len(Xs) == 0 or len(Xs) != len(ys):
            raise ValueError("set_datasets_mixed: one y per X, and at least one data set")
        if any(X.ndim != 2 or X.shape[0] != y.shape[0] for X, y in zip(Xs, ys)):
            raise ValueError("set_datasets_mixed: every X must be (n_b, d_b) and its y (n_b,)")
        cd = np.ascontiguousarray(chain_dataset, dtype=np.int32).ravel()
        if cd.size != self.C:
            raise ValueError("chain_dataset must hold one data set index per chain")
        n_rows = np.array([X.shape[0] for X in Xs], dtype=np.int64)
        n_features = np.array([X.shape[1] for X in Xs], dtype=np.int32)
        X = np.ascontiguousarray(np.concatenate([X.ravel() for X in Xs]))
        y = np.ascontiguousarray(np.concatenate(ys))
        _ck(self._lib.bsr_set_datasets_mixed_host(self._h, len(Xs), _ptr(X), _ptr(y), _ptr(n_rows), _ptr(n_features), _ptr(cd)))
        self.n, self.d = int(n_rows.max()), int(n_features.max())

    def set_data_device(self, x_ptr, y_ptr, n, d, ld, n_total=0):
        self.n, self.d = int(n), int(d)
        _ck(self._lib.bsr_set_data_device(self._h, C.c_void_p(x_ptr), C.c_void_p(y_ptr), int(n), int(d), int(ld), int(n_total)))

    # ---- state ------------------------------------------------------------------------------------
    def init_chains(self, seed):
        _ck(self._lib.bsr_init_chains(self._h, C.c_uint64(int(seed) & (2 ** 64 - 1))))

    def init_chains_keyed(self, seeds, ids):
        """Prior initialisation with chain c drawing from Philox under the key (seeds[c], ids[c])."""
        seeds = np.array([int(v) & (2 ** 64 - 1) for v in np.ravel(seeds)], dtype=np.uint64)
        ids = np.ascontiguousarray(ids, dtype=np.int64).ravel()
        if seeds.size != self.C or ids.size != self.C:
            raise ValueError("seeds and ids must hold one entry per chain")
        _ck(self._lib.bsr_init_chains_keyed(self._h, _ptr(seeds), _ptr(ids)))

    def set_state(self, tok, pa, pb, nn, sigma, sa, sb, seed=0):
        CK = self.C * self.K
        tok = np.ascontiguousarray(tok, dtype=np.uint32).reshape(CK, MAX_NODES)
        pa = np.ascontiguousarray(pa, dtype=np.float64).reshape(CK, MAX_NODES)
        pb = np.ascontiguousarray(pb, dtype=np.float64).reshape(CK, MAX_NODES)
        nn = np.ascontiguousarray(nn, dtype=np.int32).reshape(CK)
        sigma = np.ascontiguousarray(sigma, dtype=np.float64).reshape(self.C)
        sa = np.ascontiguousarray(sa, dtype=np.float64).reshape(CK)
        sb = np.ascontiguousarray(sb, dtype=np.float64).reshape(CK)
        _ck(self._lib.bsr_set_state(self._h, _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn), _ptr(sigma), _ptr(sa), _ptr(sb),
                                    C.c_uint64(int(seed))))

    # ---- running ----------------------------------------------------------------------------------
    def run(self, n_sweeps, stream=None):
        _ck(self._lib.bsr_run(self._h, int(n_sweeps), C.c_void_p(stream or 0)))

    def launch_count(self):
        n = C.c_int64(0)
        _ck(self._lib.bsr_get_launch_count(self._h, C.byref(n)))
        return n.value

    def peer_export(self, world):
        """row-sharded handles: allocate the window exchange buffer, return its 64-byte CUDA IPC handle"""
        buf = C.create_string_buffer(64)
        _ck(self._lib.bsr_peer_export(self._h, int(world), C.cast(buf, _P)))
        return bytes(buf.raw)

    def peer_import(self, rank, world, handles):
        """handles: the concatenated 64-byte IPC handles of all ranks, in rank order"""
        assert len(handles) == 64 * world
        buf = C.create_string_buffer(handles, len(handles))
        _ck(self._lib.bsr_peer_import(self._h, int(rank), int(world), C.cast(buf, _P)))

    def set_window(self, window):
        """proposals per speculative window of ``run`` (1..64); the chains do not depend on it"""
        _ck(self._lib.bsr_set_window(self._h, int(window)))

    def window_geometry(self):
        """dict(splits, rows_per_split, tile_rows, ring, window) of the window kernels for the current data (diagnostics)"""
        g = np.zeros(5, dtype=np.int64)
        _ck(self._lib.bsr_get_window_geometry(self._h, g.ctypes.data_as(_P)))
        return dict(splits=int(g[0]), rows_per_split=int(g[1]), tile_rows=int(g[2]), ring=int(g[3]), window=int(g[4]))

    def set_pipeline(self, sequential):
        """sequential=True: ``run`` uses the proposal-by-proposal pipeline (call before set_data)"""
        _ck(self._lib.bsr_set_pipeline(self._h, int(bool(sequential))))

    def set_launch_geometry(self, threads_eval=0, n_groups=0):
        _ck(self._lib.bsr_set_launch_geometry(self._h, int(threads_eval), int(n_groups)))

    def run_until_done(self, max_sweeps, check_every=16, stream=None):
        done = C.c_int32(0)
        _ck(self._lib.bsr_run_until_done(self._h, int(max_sweeps), int(check_every), C.c_void_p(stream or 0), C.byref(done)))
        return done.value

    def sweep_propose(self, stream=None):
        _ck(self._lib.bsr_sweep_propose(self._h, C.c_void_p(stream or 0)))

    def sweep_eval(self, stream=None):
        _ck(self._lib.bsr_sweep_eval(self._h, C.c_void_p(stream or 0)))

    def sweep_resolve(self, stream=None):
        _ck(self._lib.bsr_sweep_resolve(self._h, C.c_void_p(stream or 0)))

    def gram_buffer(self):
        p, ns, nm = _P(), C.c_int64(), C.c_int64()
        _ck(self._lib.bsr_gram_buffer(self._h, C.byref(p), C.byref(ns), C.byref(nm)))
        return p.value, ns.value, nm.value

    def get_y_stats(self):
        a, b = C.c_double(), C.c_double()
        _ck(self._lib.bsr_get_y_stats(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_y_stats(self, sum_y, yy):
        _ck(self._lib.bsr_set_y_stats(self._h, float(sum_y), float(yy)))

    def finish_init(self):
        _ck(self._lib.bsr_finish_init(self._h))

    def count_done(self):
        n = C.c_int32(0)
        _ck(self._lib.bsr_count_done(self._h, C.byref(n)))
        return n.value

    # ---- tape / trace -----------------------------------------------------------------------------
    def set_tape(self, tapes, steps):
        """tapes: per chain, a list of ``steps`` per-proposal draw lists (or None: Philox + trace only)."""
        if tapes is None:
            _ck(self._lib.bsr_set_tape(self._h, None, None, int(steps)))
            return
        flat, off = [], [0]
        for c in range(self.C):
            assert len(tapes[c]) == steps
            for s in range(steps):
                flat.extend(tapes[c][s])
                off.append(len(flat))
        flat = np.asarray(flat if flat else [0.0], dtype=np.float64)
        off = np.asarray(off, dtype=np.int64)
        _ck(self._lib.bsr_set_tape(self._h, _ptr(flat), _ptr(off), int(steps)))
        self._tape_steps = steps

    def clear_tape(self):
        _ck(self._lib.bsr_set_tape(self._h, None, None, 0))

    def get_trace(self, steps):
        out = np.zeros((self.C, steps, TRACE_DOUBLES))
        _ck(self._lib.bsr_get_trace(self._h, _ptr(out)))
        return out

    def trace_trees(self):
        """keep the proposed tree of every traced proposal (call after set_tape)"""
        _ck(self._lib.bsr_trace_trees(self._h))

    def get_trace_trees(self, steps):
        tok = np.zeros((self.C, steps, MAX_NODES), dtype=np.uint32)
        pa = np.zeros((self.C, steps, MAX_NODES))
        pb = np.zeros((self.C, steps, MAX_NODES))
        nn = np.zeros((self.C, steps), dtype=np.int32)
        _ck(self._lib.bsr_get_trace_trees(self._h, _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn)))
        return tok, pa, pb, nn

    def set_peer_timeout(self, seconds):
        _ck(self._lib.bsr_set_peer_timeout(self._h, float(seconds)))

    def exchange_profile(self):
        ms, n = C.c_double(0), C.c_int64(0)
        _ck(self._lib.bsr_get_exchange_profile(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def record_draws(self, steps, capacity=256):
        _ck(self._lib.bsr_record_draws(self._h, int(steps), int(capacity)))
        self._rec = (steps, capacity)

    def get_recorded_draws(self):
        steps, cap = self._rec
        tape = np.zeros((self.C, steps, cap))
        cnt = np.zeros((self.C, steps), dtype=np.int32)
        _ck(self._lib.bsr_get_recorded_draws(self._h, _ptr(tape), _ptr(cnt)))
        return tape, cnt

    # ---- results ----------------------------------------------------------------------------------
    def _tree_buffers(self):
        CK = self.C * self.K
        return (np.zeros((CK, MAX_NODES), dtype=np.uint32), np.zeros((CK, MAX_NODES)), np.zeros((CK, MAX_NODES)),
                np.zeros(CK, dtype=np.int32))

    def _pinned(self, shape, dtype):
        """numpy array over page-locked memory owned by this engine (freed by close)"""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = _P()
        _ck(self._lib.bsr_alloc_host(n, C.byref(p)))
        self._pinned_ptrs = getattr(self, "_pinned_ptrs", []) + [p]
        buf = (C.c_char * n).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def get_trees_packed(self, current=False):
        """roots_ (or the live trees) as a PackedTrees: only node-count-long prefixes cross the bus, into page-locked buffers of
        the engine that are reused (and overwritten) by the next call."""
        n_nodes, n_lt = C.c_int64(0), C.c_int64(0)
        _ck(self._lib.bsr_pack_trees(self._h, int(bool(current)), C.byref(n_nodes), C.byref(n_lt)))
        n_nodes, n_lt = n_nodes.value, n_lt.value
        pk = getattr(self, "_packed_pinned", None)
        if pk is None or pk[1].size < n_nodes or pk[2].shape[0] < n_lt:
            cap_n, cap_l = max(1024, int(n_nodes * 1.25)), max(256, int(n_lt * 1.25))
            pk = (self._pinned((self.C, self.K), np.int32), self._pinned((cap_n,), np.uint32), self._pinned((cap_l, 2), np.float64))
            self._packed_pinned = pk
        _ck(self._lib.bsr_read_packed(self._h, _ptr(pk[0]), _ptr(pk[1]), _ptr(pk[2])))
        self.last_tree_bytes = pk[0].nbytes + 4 * n_nodes + 16 * n_lt
        return PackedTrees(pk[0], pk[1][:n_nodes], pk[2][:n_lt])

    def get_trees(self, current=False, reuse=False):
        """roots_ (or the live trees with current=True) as (tok, pa, pb, nn).  reuse=True: the packed transfer of
        ``get_trees_packed`` (node-count-long prefixes into page-locked buffers), expanded on the host."""
        if reuse:
            return self.get_trees_packed(current).dense()
        if False:
            if getattr(self, "_tree_pinned", None) is None:
                CK = self.C * self.K
                self._tree_pinned = (self._pinned((CK, MAX_NODES), np.uint32), self._pinned((CK, MAX_NODES), np.float64),
                                     self._pinned((CK, MAX_NODES), np.float64), self._pinned((CK,), np.int32))
            tok, pa, pb, nn = self._tree_pinned
        else:
            tok, pa, pb, nn = self._tree_buffers()
        _ck(self._lib.bsr_get_trees(self._h, int(bool(current)), _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn)))
        s = (self.C, self.K)
        return tok.reshape(s + (MAX_NODES,)), pa.reshape(s + (MAX_NODES,)), pb.reshape(s + (MAX_NODES,)), nn.reshape(s)

    def get_proposals(self):
        tok, pa, pb, nn = self._tree_buffers()
        _ck(self._lib.bsr_get_proposals(self._h, _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn)))
        s = (self.C, self.K)
        return tok.reshape(s + (MAX_NODES,)), pa.reshape(s + (MAX_NODES,)), pb.reshape(s + (MAX_NODES,)), nn.reshape(s)

    def get_stats(self):
        Cn, K = self.C, self.K
        out = dict(sigma=np.zeros(Cn), sa=np.zeros((Cn, K)), sb=np.zeros((Cn, K)), beta=np.zeros((Cn, K + 1)),
                   sse=np.zeros(Cn), counters=np.zeros((Cn, N_COUNTERS), dtype=np.int64), done=np.zeros(Cn, dtype=np.int32),
                   nerr=np.zeros(Cn, dtype=np.int32))
        _ck(self._lib.bsr_get_stats(self._h, _ptr(out["sigma"]), _ptr(out["sa"]), _ptr(out["sb"]), _ptr(out["beta"]),
                                    _ptr(out["sse"]), _ptr(out["counters"]), _ptr(out["done"]), _ptr(out["nerr"])))
        return out

    def reserve_err(self, err_cap):
        _ck(self._lib.bsr_reserve_err(self._h, int(err_cap)))

    def get_err_trace(self):
        cap = C.c_int32(0)
        _ck(self._lib.bsr_get_err_cap(self._h, C.byref(cap)))
        self.err_cap = cap.value            # run_until_done grows the trace so that it never truncates
        err = np.zeros((self.C, self.err_cap))
        _ck(self._lib.bsr_get_err_trace(self._h, _ptr(err)))
        return err

    def eval_trees(self, tok, pa, pb, nn, precision="fp32"):
        tok = np.ascontiguousarray(tok, dtype=np.uint32).reshape(-1, MAX_NODES)
        T = tok.shape[0]
        pa = np.ascontiguousarray(pa, dtype=np.float64).reshape(T, MAX_NODES)
        pb = np.ascontiguousarray(pb, dtype=np.float64).reshape(T, MAX_NODES)
        nn = np.ascontiguousarray(nn, dtype=np.int32).reshape(T)
        out = np.zeros((T, self.n))
        _ck(self._lib.bsr_eval_trees(self._h, T, _ptr(tok), _ptr(pa), _ptr(pb), _ptr(nn), {"fp32": 0, "fp64": 1}[precision], _ptr(out)))
        return out

    def predict(self, chain, X, reported=True):
        X = np.ascontiguousarray(X, dtype=np.float64)
        out = np.zeros(X.shape[0])
        _ck(self._lib.bsr_predict(self._h, int(chain), int(bool(reported)), _ptr(X), X.shape[0], X.shape[1], _ptr(out)))
        return out

    def set_profiling(self, enabled=True):
        _ck(self._lib.bsr_set_profiling(self._h, int(bool(enabled))))

    def get_profile(self):
        ms = np.zeros(5)
        ln = np.zeros(5, dtype=np.int64)
        _ck(self._lib.bsr_get_profile(self._h, _ptr(ms), _ptr(ln)))
        # window path: one "launch" = one window iteration (classify + propose, k_weval [+ k_weval_fix], k_wresolve) of the
        # main batch of a run (the short rounds that finish chains delayed by an accept are not timed);
        # sequential pipeline: one sweep (k_propose, k_trees + Gram kernel, k_resolve)
        return dict(ms=dict(propose=ms[0], eval=ms[1], resolve=ms[2]), kernels_ms=dict(eval_main=ms[3], eval_second=ms[4]),
                    iterations=int(ln[0]))
