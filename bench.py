#!/usr/bin/env python
"""bench.py -- BSR sampling hot path on B200: MH proposals scored/s (+ tree-node evals/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5|c1] [--dump-outputs DIR]

A *step* is `sweeps_per_step` sweeps (each sweep = K newProp calls per chain, codes/bsr_class.py:179) of every chain over
the synthetic data set.  Default workload = BASELINE.json configs[1] (SURVEY.md C2): K=3, 4096 chains, n=1000 rows, d=2, and
the default --steps 10 x 500 sweeps = the 5000 iterations the config names.  For N>1 (torchrun, one rank per GPU) every rank
runs its own 4096 chains (global chain ids offset by rank, no data-path collective): weak scaling.

Prints ONE JSON line (rank 0):
  value          device-timed, inputs resident in HBM, CUDA events around every step on the stream bsr_run is given
  e2e            through the C-ABI with host buffers: H2D of X, y and D2H of the results inside the timed region
  roofline       the dominant kernel (k_weval) against the bound it actually meets -- instruction issue (SURVEY 8d: the data of
                 C1-C4 is L1/L2 resident) -- with the HBM figures of the contract kept beside it
  cpu_baseline   the unmodified reference (oracle/_ref: newProp sweeps as codes/bsr_class.py:174-255 runs them) on the host
                 cores, bounded sample; the numpy oracle port is timed beside it
  from_init      the first 5000 sweeps from bsr_init_chains, no warm-up (acceptance ~1 %, where BSR.fit lives)
  fit_e2e        BSR(3, 4096).fit wall clock with the reference's stop rule (val = 100)
  workloads      short runs of the other BASELINE configs on the same ranks: c4 (65536 chains sharded over the ranks: strong
                 scaling), c5 (rows sharded over the ranks, 12.5 M rows per GPU, peer-memory windows; exchange time per
                 window), c3 (K = 10, 31-node initial trees, transcendental operator set)
`--impl reference` times the unmodified reference on the host cores for the same metric / config (rank 0 only).
"""
import argparse
import hashlib
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_OPS = list(range(1, 11))          # inv, ln(lt), neg, sin, cos, exp, square, cubic, +, *   (codes/bsr_class.py:110)
C3_OPS = [6, 2, 4, 5, 1, 9, 10]           # exp, lt, sin, cos, inv, +, *                        (SURVEY.md 8d, C3)

WORKLOADS = {
    # name: (K, chains_per_gpu, n, d, sweeps_per_step, target)
    "c1": dict(K=3, chains=50, n=100, d=2, sweeps=100, target="f1", seed=1001),
    "c2": dict(K=3, chains=4096, n=1000, d=2, sweeps=500, target="sim", seed=2001),
    # BASELINE configs[2]: K = 10 deep trees, transcendental-heavy operator set, 8 features, 16384 chains, n = 10k; every chain
    # starts from 31-node trees of height >= 6 made by a seeded generator, y = sum of three such trees + N(0, 0.1)
    "c3": dict(K=10, chains=16384, n=10000, d=8, sweeps=8, target="deep3", seed=3001, ops=C3_OPS, deep_init=True),
    # BASELINE configs[3]: 65536 chains in total, sharded over the ranks (strong scaling); `chains` = the whole job
    "c4": dict(K=5, chains=65536, n=5000, d=8, sweeps=32, target="mix8", seed=4001, strong=True),
    # large-data fit (BASELINE configs[4]): rows sharded over the ranks, 12.5 M rows per GPU (1e8 at 8 GPUs), the same 256
    # chains on every rank; data generated on the device; k_wresolve reads the ranks' partial sums over NVLink peer memory
    "c5": dict(K=5, chains=256, n=12500000, d=8, sweeps=13, target="mix8", seed=5001, row_sharded=True),
}


def deep_tree(rng, d, ops, n_nodes=31, min_height=6):
    """Seeded generator of the C3 initial trees (SURVEY.md 8d): exactly n_nodes nodes, height >= min_height, operators from
    `ops` (device opcodes), as pre-order arrays (op, oi, ft, a, b).  A spine of min_height operators first, then random
    leaves are expanded (unary: +1 node, binary: +2) until the node count is reached."""
    unary = [o for o in ops if o < 9]
    binary = [o for o in ops if o >= 9]
    # nodes as [op, children]; leaves are [0, feature]
    root = None

    def leaf():
        return [0, int(rng.integers(0, d))]

    def count(nd):
        return 1 if nd[0] == 0 else 1 + sum(count(c) for c in nd[1])

    def leaves(nd, out):
        if nd[0] == 0:
            out.append(nd)
        else:
            for c in nd[1]:
                leaves(c, out)
        return out

    root = leaf()
    cur = root
    for _ in range(min_height):          # the spine
        op = int(rng.choice(ops))
        kids = [leaf()] if op < 9 else [leaf(), leaf()]
        cur[0], cur[1] = op, kids
        cur = kids[0]
    while count(root) < n_nodes:
        ls = leaves(root, [])
        nd = ls[int(rng.integers(0, len(ls)))]
        room = n_nodes - count(root)
        op = int(rng.choice(ops if room >= 2 else unary))
        nd[0], nd[1] = op, ([leaf()] if op < 9 else [leaf(), leaf()])
    op_l, oi_l, ft_l, a_l, b_l = [], [], [], [], []

    def emit(nd):
        if nd[0] == 0:
            op_l.append(0); oi_l.append(0); ft_l.append(nd[1]); a_l.append(0.0); b_l.append(0.0)
            return
        op_l.append(nd[0]); oi_l.append(ops.index(nd[0])); ft_l.append(0)
        if nd[0] == 2:                   # lt: a ~ N(1, 1), b ~ N(0, 1) like the prior's draws (codes/funcs.py:104-107)
            a_l.append(float(rng.normal(1.0, 1.0))); b_l.append(float(rng.normal(0.0, 1.0)))
        else:
            a_l.append(0.0); b_l.append(0.0)
        for c in nd[1]:
            emit(c)

    emit(root)
    assert len(op_l) == n_nodes
    return op_l, oi_l, ft_l, a_l, b_l


def eval_enc(enc, X):
    """allcal (codes/funcs.py:175-220) of a pre-order encoded tree in numpy float64 (bench data generation only)."""
    op, oi, ft, a, b = enc
    st = []
    with np.errstate(all="ignore"):
        for i in range(len(op) - 1, -1, -1):
            o = op[i]
            if o == 0:
                st.append(X[:, ft[i]].astype(np.float64))
            elif o == 9:
                l = st.pop(); r = st.pop(); st.append(l + r)
            elif o == 10:
                l = st.pop(); r = st.pop(); st.append(l * r)
            else:
                v = st.pop()
                if o == 2: v = a[i] * v + b[i]
                elif o == 6: v = np.where(v <= 200, np.exp(np.minimum(v, 200)), 1e10)
                elif o == 1: v = np.where(v == 0, 0.0, 1.0 / np.where(v == 0, 1.0, v))
                elif o == 3: v = -v
                elif o == 4: v = np.sin(v)
                elif o == 5: v = np.cos(v)
                elif o == 7: v = v * v
                elif o == 8: v = v * v * v
                st.append(v)
    return st[0]


def make_data(w):
    rng = np.random.default_rng(w["seed"])
    X = rng.uniform(-3, 3, (w["n"], w["d"]))           # codes/simulations.py:66-67
    if w["target"] == "f1":
        y = 2.5 * X[:, 0] ** 4 - 1.3 * X[:, 0] ** 3 + 0.5 * X[:, 1] ** 2 - 1.7 * X[:, 1]
    elif w["target"] == "sim":                         # codes/simulations.py:71
        y = 1.35 * X[:, 0] * X[:, 1] + 5.5 * np.sin((X[:, 0] - 1) * (X[:, 1] - 1))
    elif w["target"] == "deep3":
        y = rng.normal(0, 0.1, w["n"])
        got = 0
        while got < 3:                                 # three random deep trees whose values stay tame
            col = eval_enc(deep_tree(rng, w["d"], w.get("ops", DEFAULT_OPS)), X)
            if np.all(np.isfinite(col)) and np.max(np.abs(col)) < 1e3 and np.std(col) > 1e-3:
                y = y + col
                got += 1
    else:
        y = np.exp(0.5 * X[:, 0]) + 2.0 * np.cos(X[:, 1]) + 0.3 * X[:, 7] * X[:, 2] + np.sin(X[:, 3] * X[:, 4]) + rng.normal(0, 0.1, w["n"])
    return X, y


def deep_state(w, C, chain_offset):
    """Initial state of the C3 workload: K deep trees per chain (seeded by global chain id), sigma = sigma_a = sigma_b = 1."""
    K, d, ops = w["K"], w["d"], w.get("ops", DEFAULT_OPS)
    tok = np.zeros((C, K, 64), dtype=np.uint32)
    pa = np.zeros((C, K, 64)); pb = np.zeros((C, K, 64))
    nn = np.zeros((C, K), dtype=np.int32)
    # 64 distinct trees per tree slot are enough to keep chains different; each chain draws its K trees from the pool by id
    pool_rng = np.random.default_rng(w["seed"] + 17)
    pool = [deep_tree(pool_rng, d, ops) for _ in range(256)]
    enc = []
    for t in pool:
        op, oi, ft, a, b = t
        tk = np.zeros(64, dtype=np.uint32); ta = np.zeros(64); tb = np.zeros(64)
        for i in range(len(op)):
            tk[i] = op[i] | (oi[i] << 8) | (ft[i] << 16); ta[i] = a[i]; tb[i] = b[i]
        enc.append((tk, ta, tb, len(op)))
    for c in range(C):
        g = np.random.default_rng((w["seed"] << 20) + chain_offset + c)
        for k, j in enumerate(g.integers(0, len(pool), K)):
            tok[c, k], pa[c, k], pb[c, k], nn[c, k] = enc[j]
    return tok, pa, pb, nn, np.ones(C), np.ones((C, K)), np.ones((C, K))


def workload_config(args, name, w, world):
    """The `config` object of the JSON line: what defines the workload.  The reference arm reports the same object (the
    bounded sample it actually times is described in its cpu_baseline.sample)."""
    K, n, d = w["K"], args.rows or w["n"], w["d"]
    S = args.sweeps_per_step or w["sweeps"]
    row_sharded = bool(w.get("row_sharded"))
    strong = bool(w.get("strong"))
    C_total = args.chains or w["chains"]
    if strong or row_sharded:
        per_gpu = C_total if row_sharded else -(-C_total // world)
        total = C_total
    else:
        per_gpu, total = C_total, C_total * world
    return dict(workload=name, K=K, chains_per_gpu=per_gpu, chains_total=total, n_rows=n * (world if row_sharded else 1), d=d, sweeps_per_step=S,
                proposals_per_step=total * K * S, l2_flush_between_steps=True, target=w["target"], precision=args.precision,
                window=max(1, min(64, int(os.environ.get("BSR_WINDOW", "64")))), rng="philox4x32-10",
                ops=("exp,lt,sin,cos,inv,+,*" if w.get("ops") else "default10"), initial_trees=("31-node seeded" if w.get("deep_init") else "prior"),
                parallelism=("rows x%d (peer-memory windows)" % world if row_sharded else ("chains x%d%s" % (world, " (strong)" if strong else ""))))


# ------------------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (oracle/_ref) and the numpy oracle port, one chain per host core
# ------------------------------------------------------------------------------------------------------
_REF_STATE = {}


def _ref_worker_init(X, y, K, seed):
    """Per-process state of one reference chain: exactly what BSR.fit sets up before its loop (codes/bsr_class.py:105-142)."""
    import copy
    import pandas as pd
    from oracle import ref_loader
    bsr = ref_loader.load()
    from scipy.stats import invgamma
    np.random.seed(seed)
    st = _REF_STATE
    st["bsr"], st["copy"] = bsr, copy
    st["X"], st["y"] = pd.DataFrame(X), pd.Series(y)           # README.md:27-29: DataFrame rows, Series with default index
    st["K"], st["n_feature"] = K, X.shape[1]
    st["Ops"] = ['inv', 'ln', 'neg', 'sin', 'cos', 'exp', 'square', 'cubic', '+', '*']      # codes/bsr_class.py:110-112
    st["Op_weights"] = [1.0 / len(st["Ops"])] * len(st["Ops"])
    st["Op_type"] = [1, 1, 1, 1, 1, 1, 1, 1, 2, 2]
    st["beta"] = -1
    st["sigma"] = invgamma.rvs(1)
    st["Roots"], st["Siga"], st["Sigb"] = [], [], []
    for _ in range(K):
        Root = bsr.Node(0)
        sa, sb = invgamma.rvs(1), invgamma.rvs(1)
        bsr.grow(Root, st["n_feature"], st["Ops"], st["Op_weights"], st["Op_type"], st["beta"], sa, sb)
        st["Roots"].append(Root); st["Siga"].append(sa); st["Sigb"].append(sb)
    return True


def _ref_worker_step(sweeps):
    """`sweeps` sweeps of the reference's own loop body (codes/bsr_class.py:179-233): newProp per tree, the bookkeeping of an
    accept (deepcopy, node counts, intercept refit, RMSE with its per-row Python loop).  Stop rules are not applied."""
    st = _REF_STATE
    bsr, copy = st["bsr"], st["copy"]
    K, X, y = st["K"], st["X"], st["y"]
    n_train = X.shape[0]
    props = evals = accepts = 0
    t0 = time.perf_counter()
    for _ in range(sweeps):
        for count in range(K):
            Roots = list(st["Roots"])
            m_all = sum(bsr.getNum(r) for r in Roots)
            try:
                res, sigma, Root, sa, sb = bsr.newProp(Roots, count, st["sigma"], y, X, st["n_feature"], st["Ops"], st["Op_weights"],
                                                       st["Op_type"], st["beta"], st["Siga"][count], st["Sigb"][count])
            except np.linalg.LinAlgError:                  # NaN columns abort the reference (quirk Q15): count the call, keep the state
                props += 1
                continue
            props += 1
            evals += n_train * (bsr.getNum(Root) + m_all) if res else n_train * (m_all + m_all // K)
            st["sigma"], st["Siga"][count], st["Sigb"][count] = sigma, sa, sb
            if res is True:
                accepts += 1
                st["Roots"][count] = copy.deepcopy(Root)
                XX = np.zeros((n_train, K))
                for i in range(K):
                    temp = bsr.allcal(st["Roots"][i], X)
                    temp.shape = (temp.shape[0])
                    XX[:, i] = temp
                XX = np.concatenate((np.ones((n_train, 1)), XX), axis=1)
                scale = np.max(np.abs(XX))
                XX = XX / scale
                eps = np.eye(XX.shape[1]) * 1e-6
                yy = np.array(y); yy.shape = (yy.shape[0], 1)
                Beta = np.matmul(np.linalg.inv(np.matmul(XX.transpose(), XX) + eps), np.matmul(XX.transpose(), yy))
                output = np.matmul(XX, Beta)
                error = 0
                for i in range(n_train):
                    error += (output[i, 0] - y[i]) * (output[i, 0] - y[i])
    return props, evals, accepts, time.perf_counter() - t0


def _oracle_worker_init(X, y, K, seed):
    _REF_STATE.update(X=X, y=y, K=K, seed=seed, state=None, round=0)
    return True


def _oracle_worker_step(sweeps):
    """Continue one oracle chain for `sweeps` sweeps (fixed-sweep mode, like the GPU bench)."""
    from oracle import bsr_oracle as O
    st = _REF_STATE
    cfg = O.Config(n_feature=st["X"].shape[1])
    dr = O.GeneratorDraws(st["seed"] + 100003 * st["round"])
    st["round"] += 1
    t0 = time.perf_counter()
    r = O.run_chain(st["X"], st["y"], st["K"], cfg, dr, val=0, max_sweeps=sweeps, fixed_sweeps=True, init=st["state"])
    dt = time.perf_counter() - t0
    st["state"] = dict(sigma=r.sigma, trees=r.final_state, sigma_a=r.sigma_a, sigma_b=r.sigma_b)
    return r.n_proposals, r.node_evals_ref, r.n_accepts, dt


class CpuChains:
    """`procs` persistent worker processes, one reference (or oracle-port) chain each, all on the same (X, y)."""

    def __init__(self, w, procs, kind):
        import multiprocessing as mp
        self.w, self.procs, self.kind = w, procs, kind
        self.X, self.y = make_data(w)
        ctx = mp.get_context("fork")
        self.pools = [ctx.Pool(1) for _ in range(procs)]
        init = _ref_worker_init if kind == "reference" else _oracle_worker_init
        self.step_fn = _ref_worker_step if kind == "reference" else _oracle_worker_step
        for r in [p.apply_async(init, (self.X, self.y, w["K"], 7919 * (i + 1))) for i, p in enumerate(self.pools)]:
            r.get()

    def step(self, sweeps):
        t0 = time.perf_counter()
        res = [r.get() for r in [p.apply_async(self.step_fn, (sweeps,)) for p in self.pools]]
        wall = time.perf_counter() - t0
        return sum(r[0] for r in res), sum(r[1] for r in res), sum(r[2] for r in res), wall

    def close(self):
        for p in self.pools:
            p.terminate()


def reference_available():
    try:
        from oracle import ref_loader
        return ref_loader.available()
    except Exception:
        return False


def cpu_sample_rows(w):
    # the CPU samplers cannot hold 1e7..1e8 rows per chain in reasonable time: they are timed at n = 1e5 rows (their cost per
    # proposal is linear in n) and the full-size figure is labelled extrapolated (SURVEY.md 8d)
    return 100000 if w.get("row_sharded") else w["n"]


def time_cpu_chains(w, kind, budget_s, procs=None):
    """Proposals/s of `kind` ("reference" | "port") on all host cores for about budget_s seconds of wall clock."""
    procs = procs or (os.cpu_count() or 1)
    n_full = w["n"]
    w = dict(w, n=cpu_sample_rows(w))
    pool = CpuChains(w, procs, kind)
    try:
        p, e, a, dt = pool.step(1)                         # warm-up (imports, first touch) and a first cost estimate
        per_sweep = max(dt, 1e-3)
        sweeps = max(1, int(min(budget_s / 3.0, 4.0) / per_sweep))
        props = evals = acc = 0
        wall = 0.0
        while wall < budget_s:
            p, e, a, dt = pool.step(sweeps)
            props += p; evals += e; acc += a; wall += dt
        out = dict(value=props / wall, unit="proposals/s", cores=procs, kind=kind, node_evals_ref_per_s=evals / wall,
                   accept_rate=acc / max(props, 1),
                   sample="%d %s chains (1 per core) x %d sweeps x %d proposals on the same X, y (n=%d, d=%d, K=%d), %.1f s wall"
                          % (procs, "unmodified-reference" if kind == "reference" else "oracle-port", int(round(props / procs / w["K"])), w["K"],
                             w["n"], w["d"], w["K"], wall))
        if w["n"] != n_full:
            out.update(extrapolated_to_rows=n_full, extrapolated_value=props / wall * w["n"] / n_full,
                       note="timed at n=%d rows, scaled linearly in n to %d rows per GPU" % (w["n"], n_full))
        return out
    finally:
        pool.close()


def cpu_baseline(w, budget_s=12.0):
    """The reported CPU baseline of the JSON line: the unmodified reference when oracle/_ref travelled with the snapshot
    (kind "reference"), with the oracle port's figure beside it; the port alone otherwise."""
    if w.get("ops") or w.get("deep_init"):
        return None                                        # the reference hard-codes its operator set and prior initialisation
    if reference_available():
        out = time_cpu_chains(w, "reference", budget_s)
        port = time_cpu_chains(w, "port", max(4.0, budget_s / 3))
        out["port_value"] = port["value"]
        out["port_sample"] = port["sample"]
        return out
    return time_cpu_chains(w, "port", budget_s)


def run_reference(args, name, w):
    """--impl reference: the unmodified reference's newProp sweeps on every host core (oracle/_ref; the oracle port if the copy
    did not travel).  Each step is a bounded sample of the workload: one chain per core, `sweeps` sweeps."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    kind = "reference" if reference_available() else "port"
    ws = dict(w, n=cpu_sample_rows(w))
    pool = CpuChains(ws, procs, kind)
    p, e, a, dt = pool.step(1)
    sweeps = max(1, int(2.0 / max(dt, 1e-3)))            # about 2 s of wall clock per step
    for _ in range(args.warmup):
        pool.step(sweeps)
    props = evals = 0
    wall = 0.0
    for _ in range(args.steps):
        p, e, a, dt = pool.step(sweeps)
        props += p; evals += e; wall += dt
    pool.close()
    v = props / wall
    sample = "%d chains (1 per host core) x %d sweeps per step, %d steps; n=%d rows" % (procs, sweeps, args.steps, ws["n"])
    line = dict(metric="mh_proposals_per_sec", value=v, unit="proposals/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * wall / args.steps, higher_is_better=True, scaling="strong" if w.get("strong") else "weak", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference", config=workload_config(args, name, w, world),
                node_evals_ref_per_sec=evals / wall,
                cpu_baseline=dict(value=v, unit="proposals/s", cores=procs, kind=kind, sample=sample,
                                  what=("unmodified reference (oracle/_ref): newProp sweeps as codes/bsr_class.py:179-233 runs them"
                                        if kind == "reference" else "numpy oracle port (oracle/_ref did not travel)")),
                e2e=dict(value=v, unit="proposals/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    if ws["n"] != w["n"]:
        line["cpu_baseline"]["note"] = "timed at n=%d rows; per-proposal cost is linear in n (the workload has %d rows per GPU)" % (ws["n"], w["n"])
    emit(line)


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return dict(sm_mhz=None, sm_max_mhz=self.max_mhz, reasons=[])
        return dict(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons))


def csrc_hash():
    """sha256 over the kernel sources: ties the ncu figures kept in profiles/traffic.json to the build that produced them."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "mcmc-symreg_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(d, f), "rb") as fh:
                h.update(f.encode()); h.update(fh.read())
    return h.hexdigest()[:16]


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def vmax(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def vsum(self, vals):
        t = self.torch.tensor([float(v) for v in vals], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t)
        return [float(v) for v in t.tolist()]

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def setup_engine(D, args, name, w):
    """Engine + data + initial chains of workload `w` on this rank.  Returns (eng, run, X, y, C, n, chain-sharding factor)."""
    import torch
    from mcmc_symreg_b200 import capi
    K, d = w["K"], w["d"]
    n = args.rows or w["n"]
    ops = w.get("ops", DEFAULT_OPS)
    weights = [1.0 / len(ops)] * len(ops)
    row_sharded = bool(w.get("row_sharded"))
    C_cfg = args.chains or w["chains"]
    run = None
    keep = []
    if row_sharded:
        # rows [rank * n, (rank + 1) * n) of a global data set of world * n rows, generated on the device (fp32, column-major)
        from mcmc_symreg_b200 import parallel
        C = C_cfg
        ld = (n + 3) // 4 * 4
        gen = torch.Generator(device="cuda").manual_seed(w["seed"] + D.rank)
        Xd = torch.rand((d, ld), generator=gen, device="cuda", dtype=torch.float32) * 6 - 3
        yd = (torch.exp(0.5 * Xd[0]) + 2.0 * torch.cos(Xd[1]) + 0.3 * Xd[7] * Xd[2] + torch.sin(Xd[3] * Xd[4])
              + 0.1 * torch.randn(ld, generator=gen, device="cuda", dtype=torch.float32)).contiguous()
        keep += [Xd, yd]
        X, y = None, None
        eng = capi.Engine(K, C, ops, weights, beta=-1.0, val=0, plateau_rule=False, precision=args.precision, device=D.local,
                          chain_offset=0, row_sharded=D.world > 1)
        eng.set_data_device(Xd.data_ptr(), yd.data_ptr(), n, d, ld, n_total=n * D.world)
        if D.world > 1:
            rs = parallel.RowShardedEngine(eng, n * D.world)
            rs.init_chains(w["seed"])
            assert rs.enable_peer_windows()
            keep.append(rs)
            run = lambda sweeps, stream=None: rs.run(sweeps)
        else:
            eng.init_chains(w["seed"])
        lo = 0
    else:
        X, y = make_data(dict(w, n=n))
        if w.get("strong"):
            lo, hi = (C_cfg * D.rank) // D.world, (C_cfg * (D.rank + 1)) // D.world
        else:
            lo, hi = D.rank * C_cfg, (D.rank + 1) * C_cfg
        C = hi - lo
        eng = capi.Engine(K, C, ops, weights, beta=-1.0, val=0, plateau_rule=False, precision=args.precision, device=D.local,
                          chain_offset=lo)
        eng.set_data(X, y)
        if w.get("deep_init"):
            eng.set_state(*deep_state(w, C, lo), seed=w["seed"])
        else:
            eng.init_chains(w["seed"])
    if run is None:
        run = eng.run
    eng._keep = keep
    return eng, run, X, y, C, n, lo


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, eng, stats, chain_offset):
    """--dump-outputs: what the timed bsr_run calls leave for their caller -- bsr_get_stats and the live and the reported
    trees (bsr_get_trees) of this rank's chains -- as float64 DIR/<name>.npy, first axis = chain.  Tree tokens are
    op | op_ind << 8 | feature << 16 (include/bsr_b200.h); slots past a tree's node count are written as 0.  When the chains
    need more than DUMP_BYTES, a fixed seeded sample of them is written; chain_id.npy holds the global ids written."""
    arrays = dict(stats)
    for prefix, current in (("tree", True), ("roots", False)):
        tok, pa, pb, nn = eng.get_trees(current=current)
        used = np.arange(tok.shape[-1]) < nn[..., None]
        arrays.update({prefix + "_tok": tok * used, prefix + "_a": pa * used, prefix + "_b": pb * used, prefix + "_nodes": nn})
    arrays["chain_id"] = chain_offset + np.arange(eng.C)
    per_chain = sum(8 * (a.size // eng.C) for a in arrays.values())
    budget = DUMP_BYTES - 256 * len(arrays)                       # (npy headers)
    idx = np.arange(eng.C)
    if eng.C * per_chain > budget:
        idx = np.sort(np.random.default_rng(0).choice(eng.C, budget // per_chain, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a)[idx].astype(np.float64))


def measure(D, args, name, w, steps, warmup, full, dump_dir=None):
    """Device-timed steps + per-stage profile + e2e of one workload on the ranks of D.  `full`: also the roofline object and
    the slower extras of the headline line.  `dump_dir`: see dump_outputs."""
    import torch
    K, d = w["K"], w["d"]
    S = args.sweeps_per_step or w["sweeps"]
    row_sharded = bool(w.get("row_sharded"))
    world = D.world
    eng, run, X, y, C, n, lo = setup_engine(D, args, name, w)
    eng.set_launch_geometry(0, args.groups)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    for _ in range(warmup):
        run(S, stream)
    D.barrier()
    c0 = eng.get_stats()["counters"].sum(axis=0)
    sampler = ClockSampler(D.local)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    D.barrier()
    l0 = eng.launch_count()
    t_wall0 = time.perf_counter()
    for i in range(steps):
        flush.fill_(i & 0xFF)                      # L2 flush between timed iterations (outside the event pair)
        evs[i][0].record()
        run(S, stream)
        evs[i][1].record()
    D.barrier()
    t_wall = time.perf_counter() - t_wall0
    n_launches = eng.launch_count() - l0
    clocks = sampler.result()
    ms_total = float(sum(a.elapsed_time(b) for a, b in evs))
    stats = eng.get_stats()
    c1 = stats["counters"].sum(axis=0)
    if dump_dir and D.rank == 0:
        dump_outputs(dump_dir, eng, stats, lo)
    dc = c1 - c0
    ms_max = D.vmax(ms_total)
    props, ev_ref, ev_exec, accepts, rank_rej, fp64_sw, cap_rej = D.vsum([dc[0], dc[5], dc[6], dc[1], dc[2], dc[4], dc[3]])
    if row_sharded:      # every rank runs the same chains on its own rows: proposals are not additive, node evaluations are
        props, accepts, rank_rej, fp64_sw, cap_rej = [v / world for v in (props, accepts, rank_rej, fp64_sw, cap_rej)]
    value = props / (ms_max * 1e-3)

    # ---- per-stage / per-kernel device time (CUDA events on the run's stream, separate short run) ----
    eng.set_profiling(True)
    prof_sweeps = min(S, 128)          # 128 K proposals per chain = 2 K full 64-slot windows
    run(prof_sweeps, stream)
    torch.cuda.synchronize()
    prof = eng.get_profile()
    x_ms, x_n = eng.exchange_profile()
    eng.set_profiling(False)
    tok, pa, pb, nn = eng.get_trees(current=True)
    mean_nodes = float(nn.mean())
    iters = max(1, prof["iterations"])
    stage_ms = dict((k, v / iters) for k, v in prof["ms"].items())          # per window iteration
    k_ms = prof["kernels_ms"]["eval_main"] / iters                           # k_weval alone
    total_ms = sum(stage_ms.values())
    W = max(1, min(64, int(os.environ.get("BSR_WINDOW", "64"))))      # bsr_run's window (library default 64)

    out = dict(value=value, ms_per_step=ms_max / steps, steps=steps, warmup=warmup, proposals=props,
               node_evals_ref_per_sec=ev_ref / (ms_max * 1e-3), node_evals_exec_per_sec=ev_exec / (ms_max * 1e-3),
               accept_rate=accepts / max(props, 1), rank_reject_rate=rank_rej / max(props, 1), fp64_sweeps=fp64_sw, capacity_rejects=cap_rej,
               mean_nodes_per_tree=mean_nodes, gpu_launches=int(n_launches), wall_s=t_wall, clocks=clocks,
               stage_ms_per_window=stage_ms, kernel_ms=dict(k_weval=k_ms),
               share_of_window=dict((k, v / total_ms) for k, v in stage_ms.items()), windows_profiled=iters)
    if row_sharded and world > 1:
        out["exchange_ms_per_window"] = x_ms / max(1, x_n)      # k_wsignal + k_wwait between a rank's evaluation and its resolve
        out["exchange_bytes_per_window_per_peer"] = C * W * (K + 4) * 8 * eng.window_geometry()["splits"]
        # every rank must hold the same chains: compare a digest of the live trees across ranks
        dig = int(hashlib.sha256(tok.tobytes() + nn.tobytes()).hexdigest()[:12], 16)
        lo_, hi_ = D.vmax(dig), -D.vmax(-dig)
        out["ranks_identical"] = bool(lo_ == hi_)

    # ---- end to end through the C-ABI with host buffers ----
    e2e_steps = max(2, min(steps, 10))

    def e2e_step():
        if X is not None:                          # (the row-sharded workload generates its shard on the device)
            eng.set_data(X, y)                     # H2D of this step's inputs (host float64 row-major, as BSR.fit receives them)
        run(S, stream)
        st = eng.get_stats()                       # D2H of the step's results
        tr = eng.get_trees_packed(current=False)    # node-count-long prefixes into the engine's page-locked result buffers
        return sum(v.nbytes for v in st.values()) + eng.last_tree_bytes

    for _ in range(2 if full else 1):              # untimed: first-use allocations (page-locked result buffers, staging)
        d2h = e2e_step()
    D.barrier()
    t0 = time.perf_counter()
    e2e_step_ms = []
    for _ in range(e2e_steps):
        t1 = time.perf_counter()
        d2h = e2e_step()
        e2e_step_ms.append(1e3 * (time.perf_counter() - t1))
    D.barrier()
    e2e_wall = D.vmax(time.perf_counter() - t0)
    chains_all = C if row_sharded else D.vsum([C])[0]
    out["e2e"] = dict(value=chains_all * K * S * e2e_steps / e2e_wall, unit="proposals/s",
                      h2d_bytes_per_step=int(X.nbytes + y.nbytes) if X is not None else 0, d2h_bytes_per_step=int(d2h), steps=e2e_steps,
                      ms_per_step=1e3 * e2e_wall / e2e_steps, ms_per_step_median=float(np.median(e2e_step_ms)),
                      note="bsr_set_data_host (pageable host X, y) + bsr_run + bsr_get_stats + bsr_get_trees (node-count-long prefixes into page-locked result arrays) per step, wall clock")

    if full:
        # Dominant kernel: k_weval.  One launch interprets, for every chain, its K live trees and the W proposals of the
        # window on all n rows and reduces K + 4 fp64 sums per proposal (DESIGN.md section 5).  The data (X, y) is shared by
        # every chain and L1/L2 resident, so the kernel meets the instruction-issue roof, not HBM (SURVEY.md 8d).
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        alg_bytes = 4.0 * d * n + 8.0 * n + C * ((K + W) * mean_nodes * 20.0 + W * (K + 4) * 8.0)
        ncu = {}
        try:   # per-launch figures of the same kernel from the committed ncu --set full capture
            ncu = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(name) or {}
        except Exception:
            pass
        src = csrc_hash()
        stale = ncu.get("csrc_sha16") != src
        sm_mhz = clocks.get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        inst = ncu.get("warp_instructions_per_launch")
        # issue roof: 4 warp-instructions per cycle per SM (one per scheduler).  achieved = warp-instructions of one launch (ncu,
        # same build when not stale) / (launch time measured in THIS run x SM clock sampled in this run x 148 SMs)
        ipc_live = (inst / (k_ms * 1e-3 * sm_mhz * 1e6 * 148)) if inst else None
        per_rank_exec = ev_exec / world
        per_rank_props = props if row_sharded else props / world
        node_row_evals = per_rank_exec / max(per_rank_props, 1.0) * C * W
        interpreted_share = min(1.0, node_row_evals / (C * n * (K + W) * mean_nodes))
        fp64_fma = C * n * W * (K + 3) * interpreted_share
        out["roofline"] = dict(
            bound="issue", achieved=ipc_live, peak=4.0, unit="warp-inst/cycle/SM", frac=(ipc_live / 4.0) if ipc_live else None,
            traffic=ncu.get("dram_bytes_per_launch"),
            kernel="k_weval<float,%d> (K live + %d proposed trees per chain: interpreter + fused Gram sums)" % (K, W),
            ms_per_launch=k_ms, sm_mhz=sm_mhz,
            how="warp-instructions per launch from the committed ncu capture (profiles/traffic.json, smsp__inst_executed.sum) / "
                "(launch time by CUDA events in this run x sampled SM clock x 148 SMs x 4 schedulers)",
            ncu=dict(csrc_sha16=ncu.get("csrc_sha16"), csrc_sha16_now=src, stale=bool(stale), inst_per_cycle_per_sm=ncu.get("inst_per_cycle_per_sm"),
                     issue_active_pct=ncu.get("issue_active_pct"), warp_instructions_per_launch=inst, pipes_pct=ncu.get("pipes_pct"),
                     l1_data_pipe_pct=ncu.get("l1_data_pipe_pct"), source=ncu.get("source")),
            hbm=dict(bound="hbm", achieved=alg_bytes / (k_ms * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s",
                     frac=alg_bytes / (k_ms * 1e-3) / 1e9 / hbm_peak, algorithmic_bytes_per_launch=alg_bytes,
                     peak_source="measured" if peaks else "fallback",
                     note="the data (%.0f KB) is shared by every chain and L1/L2-resident: frac against HBM is small by construction" % ((4 * d + 8) * n / 1e3)),
            compute=dict(node_row_evals_per_s_in_k_weval=node_row_evals / (k_ms * 1e-3), fp64_fma_per_s_in_k_weval=fp64_fma / (k_ms * 1e-3),
                         interpreted_share=interpreted_share, source="BSR_CNT_NODE_EVALS_EXEC of the timed region / k_weval time per window"))
    eng.close()
    del flush
    torch.cuda.empty_cache()
    return out


def from_init_run(D, args, name, w):
    """The regime BSR.fit lives in: the first 5000 sweeps from bsr_init_chains, no warm-up (acceptance ~1 %)."""
    import torch
    eng, run, X, y, C, n, lo = setup_engine(D, args, name, w)
    K = w["K"]
    stream = torch.cuda.current_stream().cuda_stream
    total, chunk = 5000, 250
    run(1, stream)                                     # first launch: module load, window buffers (1 of the 5000 sweeps, untimed)
    D.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range((total - 1) // chunk):
        run(chunk, stream)
    run((total - 1) % chunk or chunk, stream) if (total - 1) % chunk else None
    b.record()
    D.barrier()
    ms = D.vmax(a.elapsed_time(b))
    cnt = eng.get_stats()["counters"].sum(axis=0)
    props, acc = D.vsum([cnt[0], cnt[1]])
    eng.close()
    return dict(value=(props - C * K * D.world) / (ms * 1e-3), unit="proposals/s", sweeps=total, ms=ms, accept_rate=acc / max(props, 1),
                note="first %d sweeps after bsr_init_chains (prior-sized trees, nothing warmed up), device-timed" % total)


def fit_e2e_run(args, w):
    """BSR(K, chains).fit wall clock with the reference's stop rule (val consecutive rejections / plateau), rank 0."""
    from mcmc_symreg_b200 import BSR
    X, y = make_data(w)
    # (distributed=False: this is one rank's own fit, not a collective of the process group the bench may be running under)
    est = BSR(w["K"], args.chains or w["chains"], val=100, seed=w["seed"], precision=args.precision, distributed=False)
    walls = []
    for _ in range(3):            # a 30-ms job on a freshly used device: single shots vary by a factor of two (allocations); all are reported
        t0 = time.perf_counter()
        est.fit(X, y)
        walls.append(time.perf_counter() - t0)
    wall = float(np.median(walls))
    props = float(est.counters_[:, 0].sum())
    t1 = time.perf_counter()
    model = est.model()
    t_model = time.perf_counter() - t1
    return dict(value=props / wall, unit="proposals/s", wall_s=wall, wall_s_runs=walls, proposals=props, proposals_per_chain=props / est.counters_.shape[0],
                accept_rate=float(est.counters_[:, 1].sum()) / max(props, 1.0), sweeps=est.n_sweeps_, model_ms=1e3 * t_model,
                note="BSR(%d, %d, val=100).fit(X, y): set_data + init + run_until_done + result gather, wall clock (median of three fits); roots_ decode lazily"
                     % (w["K"], args.chains or w["chains"]))


def run_ours(args, name, w):
    import __graft_entry__ as g
    g.build()
    D = Dist()
    main = measure(D, args, name, w, args.steps, args.warmup, True, dump_dir=args.dump_outputs)
    row_sharded = bool(w.get("row_sharded"))
    line = dict(metric="mh_proposals_per_sec", value=main["value"], unit="proposals/s", n_gpus=D.world, steps=args.steps, warmup=args.warmup,
                ms_per_step=main["ms_per_step"], higher_is_better=True, scaling="strong" if w.get("strong") else "weak", vs_baseline=None,
                dtype="f32" if args.precision == "fp32" else "f64", data="synthetic", config=workload_config(args, name, w, D.world))
    for k in ("node_evals_ref_per_sec", "node_evals_exec_per_sec", "accept_rate", "rank_reject_rate", "fp64_sweeps", "capacity_rejects",
              "mean_nodes_per_tree", "gpu_launches", "wall_s", "clocks", "e2e", "roofline"):
        line[k] = main[k]
    for k in ("stage_ms_per_window", "kernel_ms", "share_of_window", "windows_profiled"):
        line["roofline"][k] = main[k]
    if "exchange_ms_per_window" in main:
        line["exchange_ms_per_window"] = main["exchange_ms_per_window"]
        line["ranks_identical"] = main["ranks_identical"]
    if not args.no_extras and not row_sharded and not w.get("strong") and not w.get("deep_init"):
        line["from_init"] = from_init_run(D, args, name, w)
    # (before the other workloads: a 30-ms fit measured after they moved tens of GB through cudaMalloc / cudaFree took 110 - 180 ms)
    if D.rank == 0 and not args.no_extras and not row_sharded and not w.get("deep_init"):
        try:
            line["fit_e2e"] = fit_e2e_run(args, w)
        except Exception as ex:
            line["fit_e2e"] = dict(error="%s: %s" % (type(ex).__name__, ex))
    D.barrier()
    if not args.no_extras:
        extras = {}
        for other in [x for x in args.extra_workloads.split(",") if x and x != name]:
            wo = WORKLOADS[other]
            a2 = argparse.Namespace(**vars(args))
            a2.chains = a2.rows = a2.sweeps_per_step = 0
            try:
                r = measure(D, a2, other, wo, 2, 1, False)
                r["config"] = workload_config(a2, other, wo, D.world)
                r["scaling"] = "strong" if wo.get("strong") else "weak"
                extras[other] = r
            except Exception as ex:          # an extra workload must not cost the headline line
                extras[other] = dict(error="%s: %s" % (type(ex).__name__, ex))
                D.barrier()
        line["workloads"] = extras
    if D.rank == 0:
        if not args.no_cpu_baseline and D.world == 1:
            cb = cpu_baseline(w)
            if cb is not None:
                line["cpu_baseline"] = cb
    D.barrier()
    if D.rank == 0:
        emit(line)
    D.close()


_JSON_FD = None


def emit(line):
    """The one JSON line of the contract, on the process's real stdout."""
    out = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(out.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, out)


def main():
    # stdout carries exactly one JSON line: whatever libraries print to fd 1 meanwhile (NCCL's version banner when
    # NCCL_DEBUG is set on the box, worker processes) goes to stderr
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (the whole job for the strong-scaling workload c4)")
    ap.add_argument("--rows", type=int, default=0, help="rows (per GPU for the row-sharded workload)")
    ap.add_argument("--sweeps-per-step", type=int, default=0)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip from_init, fit_e2e and the short runs of the other workloads")
    ap.add_argument("--extra-workloads", default="c4,c5,c3", help="other BASELINE configs measured briefly after the headline workload")
    ap.add_argument("--groups", type=int, default=0, help="chain groups pipelined on separate streams (0 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step left for the caller (stats, trees of rank 0's chains) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, args.workload, w)
    else:
        run_ours(args, args.workload, w)


if __name__ == "__main__":
    main()
