"""Host-side sharding of independent chains over GPUs (one process per GPU, ``torch.distributed``).

Chains are independent (codes/bsr_class.py:99: restarts share nothing but the data), so rank r owns the global
chain ids [lo, hi); the Philox streams are keyed by global id, hence the fitted model does not depend on the
number of GPUs.  The only communication is the final gather of results.  ``torch`` is plumbing here
(process group, gather); nothing on this path computes.
"""
import os

import numpy as np


def shard_range(n_items, rank, world):
    """Contiguous balanced partition: the first (n_items % world) ranks get one extra item."""
    base, extra = divmod(int(n_items), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def row_range(n_rows, rank, world):
    return shard_range(n_rows, rank, world)


def default_device():
    return int(os.environ.get("LOCAL_RANK", "0")) if _dist_initialised() else 0


def _dist_initialised():
    try:
        import torch.distributed as dist
        return dist.is_available() and dist.is_initialized()
    except Exception:
        return False


def collect(eng):
    """Everything BSR.fit reports, as host arrays for the chains of one engine."""
    pk = eng.get_trees_packed(current=False)      # node-count-long prefixes only (views of the engine's page-locked buffers: copy)
    st = eng.get_stats()
    return dict(nn=pk.nn.copy(), ptok=pk.tok.copy(), pab=pk.ab.copy(), beta=st["beta"], sigma=st["sigma"], sa=st["sa"], sb=st["sb"],
                sse=st["sse"], counters=st["counters"], done=st["done"], nerr=st["nerr"], err=eng.get_err_trace())


def split_results(res, n_datasets, MM):
    """The gathered results of ``BSR.fit_many`` (chains b * MM ... (b + 1) * MM - 1 fit data set b) as one result dict per data
    set, each shaped as ``collect`` / ``gather_results`` shape the results of one fit of MM chains."""
    nn = np.asarray(res["nn"])
    assert nn.shape[0] == n_datasets * MM
    node_off = np.zeros(nn.shape[0] + 1, dtype=np.int64)
    np.cumsum(nn.sum(axis=1), out=node_off[1:])
    lt_off = np.zeros(res["ptok"].size + 1, dtype=np.int64)         # lt nodes before every node of the packed token stream
    np.cumsum((res["ptok"] & 0xFF) == 2, out=lt_off[1:])
    out = []
    for b in range(n_datasets):
        c0, c1 = b * MM, (b + 1) * MM
        n0, n1 = node_off[c0], node_off[c1]
        part = {}
        for key, v in res.items():
            if key == "ptok":
                part[key] = v[n0:n1].copy()
            elif key == "pab":
                part[key] = v[lt_off[n0]:lt_off[n1]].copy()
            elif key == "sweeps":
                part[key] = v
            else:
                part[key] = v[c0:c1].copy()
        out.append(part)
    return out


class _Local:
    rank, world = 0, 1

    def broadcast_int(self, v):
        return int(v)

    def gather_results(self, res, MM, K):
        return res


class _Dist:
    """torch.distributed backed context (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.rank, self.world = dist.get_rank(), dist.get_world_size()

    def broadcast_int(self, v):
        obj = [int(v)]
        self.dist.broadcast_object_list(obj, src=0)
        return int(obj[0])

    def gather_results(self, res, MM, K):
        parts = [None] * self.world
        self.dist.all_gather_object(parts, res)
        parts = [p for p in parts if p is not None]
        out = {}
        for key in parts[0]:
            if key == "sweeps":
                out[key] = max(p[key] for p in parts)
            elif key == "err":             # the ranks may have grown their RMSE traces to different capacities
                cap = max(p[key].shape[1] for p in parts)
                out[key] = np.concatenate([np.pad(p[key], ((0, 0), (0, cap - p[key].shape[1]))) for p in parts], axis=0)
            else:
                out[key] = np.concatenate([p[key] for p in parts], axis=0)
        assert out["nn"].shape[0] == MM
        return out


def context(distributed=None):
    """distributed=None: use torch.distributed iff a process group is initialised."""
    if distributed is False:
        return _Local()
    if _dist_initialised():
        return _Dist()
    if distributed:
        raise RuntimeError("distributed=True but torch.distributed is not initialised")
    return _Local()


# ------------------------------------------------------------------------------------------------------------
# Row sharding (large-n fits, SURVEY.md 8e): every rank holds a slice of the rows and ALL chains.
# ------------------------------------------------------------------------------------------------------------
class _DevView:
    """Exposes a raw device pointer through __cuda_array_interface__ so torch can alias it (no copy)."""

    def __init__(self, ptr, n, typestr="<f8"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class RowShardedEngine:
    """Drives a `row_sharded` handle phase by phase.  Every rank proposes identically (same Philox key => same trees,
    no broadcast), evaluates its own rows, then the per-chain Gram partials are all-reduced over NCCL (SUM for
    G / C'y / column sums, MAX for max|column|) and every rank resolves identically from the identical buffers.
    The only data-path exchange per sweep is C*(P(P+1)/2+3P) doubles (53 KB for C=256, K=5)."""

    def __init__(self, engine, n_total):
        import torch
        import torch.distributed as dist
        self.eng, self.torch, self.dist = engine, torch, dist
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        ptr, n_sum, n_max = engine.gram_buffer()
        C = engine.C
        self.sums = torch.as_tensor(_DevView(ptr, C * n_sum), device="cuda")
        self.maxs = torch.as_tensor(_DevView(ptr + 8 * C * n_sum, C * n_max), device="cuda")
        self.n_total = int(n_total)

    def _allreduce(self):
        if self.world > 1:
            self.dist.all_reduce(self.sums, op=self.dist.ReduceOp.SUM)
            self.dist.all_reduce(self.maxs, op=self.dist.ReduceOp.MAX)

    def sync_y_stats(self):
        s, q = self.eng.get_y_stats()
        t = self.torch.tensor([s, q], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t)
        self.eng.set_y_stats(float(t[0]), float(t[1]))

    def init_chains(self, seed):
        self.sync_y_stats()
        self.eng.init_chains(seed)          # leaves the initial Gram partials in the buffer
        self.torch.cuda.synchronize()
        self._allreduce()
        self.eng.finish_init()

    def set_state(self, *a, **k):
        self.sync_y_stats()
        self.eng.set_state(*a, **k)
        self.torch.cuda.synchronize()
        self._allreduce()
        self.eng.finish_init()

    def enable_peer_windows(self):
        """Switch ``run`` to speculative windows with the cross-rank reduction fused into the resolve kernel: every
        rank maps the other ranks' window records (CUDA IPC, NVLink peer access) and k_wresolve sums them in rank
        order -- no collective call on the data path.  Call once after the data is set (one node, world <= 8)."""
        if self.world < 2:
            return False
        rank = self.dist.get_rank()
        mine = self.eng.peer_export(self.world)
        handles = [None] * self.world
        self.dist.all_gather_object(handles, mine)
        self.eng.peer_import(rank, self.world, b"".join(handles))
        self.dist.barrier()
        self.peer_windows = True
        return True

    def run(self, n_sweeps):
        stream = self.torch.cuda.current_stream().cuda_stream
        if getattr(self, "peer_windows", False):
            self.eng.run(int(n_sweeps), stream)
            return
        for _ in range(int(n_sweeps)):
            self.eng.sweep_propose(stream)
            self.eng.sweep_eval(stream)
            self._allreduce()
            self.eng.sweep_resolve(stream)
