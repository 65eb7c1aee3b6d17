"""Import the unmodified reference from oracle/_ref (see oracle/build_ref.py) -- TEST / MEASUREMENT INFRASTRUCTURE ONLY.

The files under oracle/_ref/bsr are byte-for-byte copies of /root/reference/codes/{__init__,funcs,bsr_class}.py.  The one
thing the reference needs that this image lacks is matplotlib (codes/bsr_class.py:22 imports pyplot and never uses it):
an empty stub module is registered when the real one cannot be imported.  Nothing of the reference is patched.
"""
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")


def available(ref_dir=REF_DIR):
    return os.path.exists(os.path.join(ref_dir, "bsr", "funcs.py"))


def load(ref_dir=REF_DIR):
    """Returns the reference package (``bsr``: BSR, newProp, grow, allcal, ... as codes/__init__.py exports them)."""
    if not available(ref_dir):
        raise RuntimeError("oracle/_ref is empty: run `python oracle/build_ref.py` where /root/reference exists")
    try:
        import matplotlib.pyplot  # noqa: F401
    except Exception:
        mpl = types.ModuleType("matplotlib")
        plt = types.ModuleType("matplotlib.pyplot")
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import bsr
    if not os.path.abspath(bsr.__file__).startswith(ref_dir):
        raise RuntimeError("another package named `bsr` shadows oracle/_ref: %s" % bsr.__file__)
    return bsr
