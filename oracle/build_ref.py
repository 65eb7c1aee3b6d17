#!/usr/bin/env python
"""Recipe for oracle/_ref: the UNMODIFIED reference sampler, placed where it can travel to the GPU box.

TEST / MEASUREMENT INFRASTRUCTURE ONLY (like everything under oracle/): the product (mcmc-symreg_b200/) never imports
it.  Users: bench.py's ``--impl reference`` arm and ``cpu_baseline`` leg, and tests that validate the oracle port.

The reference (ying531/MCMC-SymReg) is pure Python: codes/funcs.py (the sampler: grow, Prop, auxProp, allcal, ylogLike,
newProp) and codes/bsr_class.py (the estimator and its fit loop), re-exported by codes/__init__.py.  There is nothing to
compile; "building" it means copying those three files, byte for byte, from /root/reference/codes into
oracle/_ref/bsr/ (the package name its absolute imports expect, codes/bsr_class.py:10-12).  oracle/_ref/ is listed in
.gitignore (no reference source enters the history) and not in .gpurunignore (it ships to the GPU box with the
snapshot, where /root/reference does not exist).  A manifest with the sha256 of every copied file is written next to
them so that a run can state which reference it timed.

    python oracle/build_ref.py            # copies when /root/reference is present, else keeps what is there
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("BSR_REFERENCE_ROOT", "/root/reference")
FILES = ("__init__.py", "funcs.py", "bsr_class.py")


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def build(verbose=True, ref_root=REF_ROOT, ref_dir=os.path.join(HERE, "_ref")):
    """Copies <ref_root>/codes into <ref_dir>/bsr.  Returns the manifest dict, or None when neither the reference nor an
    earlier copy is available."""
    src = os.path.join(ref_root, "codes")
    dest = os.path.join(ref_dir, "bsr")
    manifest_path = os.path.join(ref_dir, "MANIFEST.json")
    if os.path.isdir(src):
        os.makedirs(dest, exist_ok=True)
        man = dict(source=src, files={})
        for f in FILES:
            shutil.copyfile(os.path.join(src, f), os.path.join(dest, f))
            man["files"][f] = sha256(os.path.join(dest, f))
        with open(manifest_path, "w") as fh:
            json.dump(man, fh, indent=1)
        if verbose:
            print("[oracle/_ref] copied %s from %s" % (", ".join(FILES), src))
        return man
    if os.path.exists(manifest_path):
        with open(manifest_path) as fh:
            man = json.load(fh)
        for f, digest in man["files"].items():
            if sha256(os.path.join(dest, f)) != digest:
                raise RuntimeError("%s does not match its manifest" % os.path.join(dest, f))
        return man
    return None


if __name__ == "__main__":
    m = build()
    if m is None:
        print("reference not present at %s and no earlier copy under oracle/_ref" % REF_ROOT)
        sys.exit(1)
