#!/usr/bin/env python
"""Generate the committed golden fixtures from the UNMODIFIED reference (run in the build container).

    python tests/golden/gen_golden.py          # writes tests/golden/*.json.gz

What is recorded (SURVEY.md §4.3):
  steps_*.json.gz   seeded chains of reference ``newProp`` calls: value-level RNG tape per call, the
                    pre-order encoding of every tree before/after, and the reference's own
                    Prop / auxProp / logR intermediates (captured by wrapping module globals -- the
                    reference's code is not edited)
  fits_*.json.gz    whole ``BSR(K, MM).fit`` runs: tape, roots_, betas_, train_err_, model(),
                    complexity(), predict()
The reference arithmetic is untouched; only np.random.* / scipy rvs are wrapped to *record*.
"""
import builtins
import gzip
import json
import lzma
import os
import sys

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from ref_shim import TapeRecorder, load_reference  # noqa: E402

NAME_TO_OP = {"inv": 1, "ln": 2, "neg": 3, "sin": 4, "cos": 5, "exp": 6, "square": 7, "cubic": 8, "+": 9, "*": 10}
OPS = ['inv', 'ln', 'neg', 'sin', 'cos', 'exp', 'square', 'cubic', '+', '*']      # bsr_class.py:110
OP_TYPE = [1, 1, 1, 1, 1, 1, 1, 1, 2, 2]                                           # bsr_class.py:112


def encode(node):
    """Reference Node tree -> pre-order arrays (op, oi, ft, a, b)."""
    op, oi, ft, a, b = [], [], [], [], []

    def rec(nd):
        if nd.type == 0:
            op.append(0); oi.append(0); ft.append(int(np.asarray(nd.feature).ravel()[0])); a.append(0.0); b.append(0.0)
            return
        op.append(NAME_TO_OP[nd.operator]); oi.append(int(nd.op_ind)); ft.append(0)
        if nd.operator == 'ln':
            a.append(float(nd.a)); b.append(float(nd.b))
        else:
            a.append(0.0); b.append(0.0)
        rec(nd.left)
        if nd.type == 2:
            rec(nd.right)

    rec(node)
    return dict(op=op, oi=oi, ft=ft, a=a, b=b)


def make_data(kind, n, d, seed):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-3, 3, (n, d))
    if kind == "f1":
        y = 2.5 * X[:, 0] ** 4 - 1.3 * X[:, 0] ** 3 + 0.5 * X[:, 1] ** 2 - 1.7 * X[:, 1]
    elif kind == "f6":
        y = 1.35 * X[:, 0] * X[:, 1] + 5.5 * np.sin((X[:, 0] - 1) * (X[:, 1] - 1))
    else:
        y = np.exp(0.5 * X[:, 0]) + 2.0 * np.cos(X[:, 1]) + 0.3 * X[:, d - 1] * X[:, 0] + rng.normal(0, 0.1, n)
    return X, y


def gen_steps(name, kind, n, d, K, beta, n_chains, n_steps, seed, weights=None, store_cols=8):
    funcs, cls = load_reference()
    X, y = make_data(kind, n, d, seed)
    Xdf, ys = pd.DataFrame(X), pd.Series(y)
    w = [1.0 / len(OPS)] * len(OPS) if weights is None else list(weights)
    cap = {}
    o_prop, o_aux = funcs.Prop, funcs.auxProp

    def w_prop(*a, **k):
        r = o_prop(*a, **k)
        cap["change"], cap["Q"], cap["Qinv"] = r[3], float(r[4]), float(r[5])
        return r

    def w_aux(*a, **k):
        r = o_aux(*a, **k)
        cap["aux"] = [float(v) for v in r]
        cap["proposed"] = encode(a[2])           # Root after the lt parameters were assigned
        cap["pcol"] = funcs.allcal(a[2], Xdf).ravel()[:store_cols].tolist()
        return r

    def w_min(a, b):
        if isinstance(b, int) and b == 0:        # the min(logR, 0) call at funcs.py:1298, not min(1, 4/(Nt+2))
            cap["logR"] = float(a)
        return builtins.min(a, b)

    funcs.Prop, funcs.auxProp, funcs.min = w_prop, w_aux, w_min
    chains = []
    try:
        for c in range(n_chains):
            np.random.seed(seed * 1000 + c)
            with TapeRecorder() as rec:
                sigma = float(funcs.invgamma.rvs(1))
                roots, sa, sb = [], [], []
                for k in range(K):
                    root = funcs.Node(0)
                    s_a = float(funcs.invgamma.rvs(1)); s_b = float(funcs.invgamma.rvs(1))
                    funcs.grow(root, d, OPS, w, OP_TYPE, beta, s_a, s_b)
                    roots.append(root); sa.append(s_a); sb.append(s_b)
                init_len = rec.mark()
                chain = dict(init=dict(sigma=sigma, sa=list(sa), sb=list(sb), trees=[encode(r) for r in roots]),
                             init_tape=list(rec.tape[:init_len]), steps=[])
                for s in range(n_steps):
                    count = s % K
                    cap.clear()
                    m0 = rec.mark()
                    try:
                        res, sigma_o, root_o, sa_o, sb_o = funcs.newProp(roots, count, sigma, ys, Xdf, d, OPS, w, OP_TYPE,
                                                                         beta, sa[count], sb[count])
                    except np.linalg.LinAlgError:
                        break                       # NaN columns abort the reference (quirk Q15)
                    st = dict(count=count, tape=list(rec.tape[m0:rec.mark()]), accepted=bool(res),
                              change={'': 0, 'expansion': 1, 'shrinkage': 2}[cap["change"]], Q=cap["Q"], Qinv=cap["Qinv"],
                              aux=cap["aux"], logR=cap.get("logR"), rank_reject=("logR" not in cap),
                              proposed=cap["proposed"], pcol=cap["pcol"])
                    if res:
                        st["tree"] = encode(root_o)
                        st["height"] = int(funcs.getHeight(root_o)); st["numlt"] = int(funcs.numLT(root_o))
                        st["num"] = int(funcs.getNum(root_o)); st["expr"] = funcs.Express(root_o)
                        roots = list(roots); roots[count] = root_o
                    sigma = float(sigma_o); sa[count] = float(sa_o); sb[count] = float(sb_o)
                    st["sigma"], st["sa"], st["sb"] = sigma, sa[count], sb[count]
                    chain["steps"].append(st)
                chain["final"] = [encode(r) for r in roots]
                chain["final_cols"] = [funcs.allcal(r, Xdf).ravel().tolist() for r in roots]
            chains.append(chain)
    finally:
        funcs.Prop, funcs.auxProp = o_prop, o_aux
        del funcs.min
    out = dict(name=name, kind=kind, n=n, d=d, K=K, beta=beta, seed=seed, weights=w, X=X.tolist(), y=y.tolist(), chains=chains)
    dump(out, "steps_%s.json.gz" % name)
    nst = sum(len(c["steps"]) for c in chains)
    nacc = sum(s["accepted"] for c in chains for s in c["steps"])
    nrk = sum(s["rank_reject"] for c in chains for s in c["steps"])
    print("steps_%s: %d chains, %d steps, %d accepted, %d rank-rejects" % (name, len(chains), nst, nacc, nrk))


def gen_fit(name, kind, n, d, K, MM, val, seed, beta=-1):
    funcs, cls = load_reference()
    X, y = make_data(kind, n, d, seed)
    Xt, _ = make_data(kind, 17, d, seed + 7)
    np.random.seed(seed)
    with TapeRecorder() as rec:
        est = cls.BSR(K, MM, beta=beta, val=val)
        est.fit(pd.DataFrame(X), pd.Series(y))
    out = dict(name=name, kind=kind, n=n, d=d, K=K, MM=MM, val=val, beta=beta, seed=seed, X=X.tolist(), y=y.tolist(),
               Xtest=Xt.tolist(), tape=rec.tape,
               roots=[[encode(r) for r in rs] for rs in est.roots_],
               betas=[np.asarray(b).ravel().tolist() for b in est.betas_],
               train_err=[[float(e) for e in el] for el in est.train_err_],
               model=est.model(), model_first=est.model(last_ind=MM), complexity=int(est.complexity()),
               predict=est.predict(Xt).ravel().tolist(), predict_train=est.predict(X).ravel().tolist())
    dump(out, "fits_%s.json.gz" % name)
    print("fits_%s: tape %d draws, accepts per restart %s, model %s" % (name, len(rec.tape), [len(e) for e in est.train_err_], est.model()))


def dump(obj, fname):
    with gzip.open(os.path.join(HERE, fname), "wt", compresslevel=9) as f:
        json.dump(obj, f, separators=(",", ":"))


def dump_tape(tape, fname):
    with lzma.open(os.path.join(HERE, fname), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(np.asarray(tape, dtype="<f8").tobytes())


if __name__ == "__main__":
    gen_steps("f1_d2_k3", "f1", n=64, d=2, K=3, beta=-1, n_chains=24, n_steps=60, seed=11)
    gen_steps("mix_d8_k5", "mix", n=48, d=8, K=5, beta=-1, n_chains=12, n_steps=60, seed=12)
    gen_steps("deep_d3_k2", "f6", n=40, d=3, K=2, beta=-0.45, n_chains=16, n_steps=60, seed=13)
    # non-uniform Op_weights: where the stale op_ind of reassignOperator (quirk Q7, funcs.py:812,829,879,900) enters Q / Qinv / fStruc
    gen_steps("w_d3_k3", "f6", n=50, d=3, K=3, beta=-1, n_chains=16, n_steps=90, seed=14,
              weights=[0.05, 0.2, 0.05, 0.1, 0.1, 0.05, 0.1, 0.05, 0.2, 0.1])
    gen_fit("f1_k3", "f1", n=100, d=2, K=3, MM=4, val=60, seed=21)
    gen_fit("f6_k2", "f6", n=80, d=2, K=2, MM=3, val=100, seed=22)
    # BASELINE.json configs[0] / README.md:26 usage: BSR(K=3, MM=50) on the paper's f1, n = 100, default val = 100
    gen_fit("c1_readme", "f1", n=100, d=2, K=3, MM=50, val=100, seed=1001)


def gen_plateau():
    """A restart long enough (>100 accepts) for the RMSE plateau stop of bsr_class.py:248-252 to fire, which also
    exercises quirk Q16 (ROOTS keeps the pre-accept snapshot while BETAS is post-accept).  Tiny noisy data keeps the
    likelihood weak, so the reference accepts often enough to get there."""
    for seed in range(31, 80):
        funcs, cls = load_reference()
        rng = np.random.default_rng(seed)
        X = rng.uniform(-3, 3, (6, 2))
        y = rng.normal(0, 3, 6)
        np.random.seed(seed)
        with TapeRecorder() as rec:
            est = cls.BSR(2, 1, val=2500)
            est.fit(pd.DataFrame(X), pd.Series(y))
        e = est.train_err_[0]
        fired = len(e) > 100 and 1 - np.min(e[-10:]) / np.mean(e[-10:]) < 0.05
        print("plateau probe seed", seed, "accepts", len(e), "draws", len(rec.tape), "fired", fired, flush=True)
        if fired and len(rec.tape) < 600000:
            Xt = rng.uniform(-3, 3, (9, 2))
            # the 138 k-draw tape goes beside the fixture in binary (tests/conftest.py:load_golden): as JSON text it passes 1 MB
            dump_tape(rec.tape, "fits_plateau.tape.f64.xz")
            out = dict(name="plateau", kind="noise", n=6, d=2, K=2, MM=1, val=2500, beta=-1, seed=seed, X=X.tolist(), y=y.tolist(),
                       Xtest=Xt.tolist(), tape_file="fits_plateau.tape.f64.xz", roots=[[encode(r) for r in rs] for rs in est.roots_],
                       betas=[np.asarray(b).ravel().tolist() for b in est.betas_],
                       train_err=[[float(v) for v in el] for el in est.train_err_], model=est.model(), model_first=est.model(last_ind=1),
                       complexity=int(est.complexity()), predict=est.predict(Xt).ravel().tolist(), predict_train=est.predict(X).ravel().tolist())
            dump(out, "fits_plateau.json.gz")
            return
    raise SystemExit("no seed produced a plateau stop")
