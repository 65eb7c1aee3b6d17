"""bench.py's reference arm runs on host cores only, so its side of the output contract is checked here on CPU:
exactly one JSON line on stdout (library banners go to stderr), the keys the driver reads, and rank != 0 printing nothing."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "0"]
    return subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)


def test_reference_arm_prints_one_json_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mh_proposals_per_sec" and d["unit"] == "proposals/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    # the unmodified reference when oracle/_ref is present (built by __graft_entry__.build() where /root/reference exists), else the port
    from oracle import ref_loader
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_loader.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == dict(value=d["value"], unit=d["unit"], h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert d["config"]["workload"] == "c1" and d["config"]["K"] == 3 and d["config"]["chains_per_gpu"] == 50


def test_reference_arm_other_ranks_print_nothing():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_reference_copy_is_the_reference(tmp_path):
    """oracle/_ref holds byte-for-byte copies (sha256 manifest) and the loader imports the reference's own package from there.
    The reference is not part of this repository, so the copy is made from a stand-in of its codes/ directory; a copy already
    under oracle/_ref must match its manifest."""
    sys.path.insert(0, ROOT)
    import pytest
    from oracle import build_ref, ref_loader
    if ref_loader.available():
        assert build_ref.build(verbose=False, ref_root=str(tmp_path / "absent")) is not None
    ref_root, ref_dir = tmp_path / "reference", str(tmp_path / "_ref")
    assert build_ref.build(verbose=False, ref_root=str(ref_root), ref_dir=ref_dir) is None and not ref_loader.available(ref_dir)
    codes = ref_root / "codes"
    codes.mkdir(parents=True)
    (codes / "__init__.py").write_text("from .funcs import *\nfrom .bsr_class import *\n")
    (codes / "funcs.py").write_text("def newProp(*args):\n    return args\n")
    (codes / "bsr_class.py").write_text("class BSR:\n    pass\n")
    man = build_ref.build(verbose=False, ref_root=str(ref_root), ref_dir=ref_dir)
    assert sorted(man["files"]) == sorted(build_ref.FILES)
    for f, digest in man["files"].items():
        copied = os.path.join(ref_dir, "bsr", f)
        assert open(copied, "rb").read() == (codes / f).read_bytes() and build_ref.sha256(copied) == digest
    # without the source, the earlier copy is what build() returns, checked against its manifest
    assert build_ref.build(verbose=False, ref_root=str(tmp_path / "absent"), ref_dir=ref_dir) == man
    copied = os.path.join(ref_dir, "bsr", "funcs.py")
    with open(copied, "a") as fh:
        fh.write("# edited\n")
    with pytest.raises(RuntimeError, match="does not match its manifest"):
        build_ref.build(verbose=False, ref_root=str(tmp_path / "absent"), ref_dir=ref_dir)
    build_ref.build(verbose=False, ref_root=str(ref_root), ref_dir=ref_dir)
    saved = {m: sys.modules.pop(m) for m in list(sys.modules) if m == "bsr" or m.startswith("bsr.")}
    path = list(sys.path)
    try:
        bsr = ref_loader.load(ref_dir)
        assert os.path.abspath(bsr.__file__).startswith(ref_dir)
        assert callable(bsr.newProp) and callable(bsr.BSR)
    finally:
        sys.path[:] = path
        for m in [m for m in sys.modules if m == "bsr" or m.startswith("bsr.")]:
            del sys.modules[m]
        sys.modules.update(saved)


def test_c3_deep_initial_trees():
    """The seeded generator of the C3 workload (SURVEY.md 8d): 31 nodes, height >= 6, operators from the transcendental set."""
    sys.path.insert(0, ROOT)
    import bench
    from oracle import bsr_oracle as O
    rng = np.random.default_rng(5)
    for _ in range(50):
        op, oi, ft, a, b = bench.deep_tree(rng, 8, bench.C3_OPS)
        t = O.Tree(op, oi, ft, a, b)
        assert len(t) == 31 and O.subtree_sizes(t.op)[0] == 31 and O.get_height(t) >= 6
        assert set(o for o in op if o != 0) <= set(bench.C3_OPS) and all(bench.C3_OPS[i] == o for o, i in zip(op, oi) if o != 0)
        assert max(ft) < 8
    w = dict(bench.WORKLOADS["c3"], n=200)
    X, y = bench.make_data(w)
    assert np.all(np.isfinite(y)) and np.std(y) > 0
    tok, pa, pb, nn, sig, sa, sb = bench.deep_state(w, 5, 100)
    assert (nn == 31).all() and tok.shape == (5, 10, 64)
    tok2 = bench.deep_state(w, 3, 102)[0]
    assert np.array_equal(tok[2:], tok2)            # keyed by global chain id: independent of the sharding
    col = bench.eval_enc((op, oi, ft, a, b), X)
    ref = O.eval_tree(t, X)
    assert np.allclose(col, ref, equal_nan=True)


class _StandInEngine:
    """What bench.dump_outputs reads from a capi.Engine: C, K and get_trees."""

    def __init__(self, C, K):
        self.C, self.K = C, K
        rng = np.random.default_rng(C)
        self.trees = [(rng.integers(0, 1 << 20, (C, K, 64)).astype(np.uint32), rng.normal(size=(C, K, 64)), rng.normal(size=(C, K, 64)),
                       rng.integers(1, 65, (C, K)).astype(np.int32)) for _ in range(2)]

    def get_trees(self, current=False):
        return self.trees[int(current)]


def test_dump_outputs_bound_and_sample(tmp_path):
    """--dump-outputs writes float64 arrays with the chain on the first axis, at most 64 MB in all: every chain when they fit,
    else the same seeded sample of chains on every call."""
    sys.path.insert(0, ROOT)
    import bench
    for C, K in ((4096, 3), (16384, 10)):
        eng = _StandInEngine(C, K)
        stats = dict(sigma=np.ones(C), beta=np.ones((C, K + 1)), counters=np.ones((C, 8), dtype=np.int64))
        dirs = [tmp_path / ("%d_%d" % (C, i)) for i in range(2)]
        for d in dirs:
            bench.dump_outputs(str(d), eng, stats, 7)
        files = sorted(os.listdir(dirs[0]))
        assert files == sorted(["sigma.npy", "beta.npy", "counters.npy", "chain_id.npy"]
                               + [p + s for p in ("tree", "roots") for s in ("_tok.npy", "_a.npy", "_b.npy", "_nodes.npy")])
        assert sum(os.path.getsize(dirs[0] / f) for f in files) <= 64e6
        ids = np.load(dirs[0] / "chain_id.npy")
        assert (len(ids) == C) == (C == 4096) and np.all(np.diff(ids) > 0) and ids[0] >= 7 and ids[-1] < 7 + C
        for f in files:
            a, b = np.load(dirs[0] / f), np.load(dirs[1] / f)
            assert a.dtype == np.float64 and a.shape[0] == len(ids) and np.array_equal(a, b)
        sel = (ids - 7).astype(int)
        tok, _, pb, nn = eng.get_trees(current=True)
        got, got_b = np.load(dirs[0] / "tree_tok.npy"), np.load(dirs[0] / "tree_b.npy")
        used = np.arange(64) < nn[sel][..., None]
        assert np.array_equal(got[used], tok[sel][used]) and not got[~used].any()
        assert np.array_equal(got_b[used], pb[sel][used]) and not got_b[~used].any()
