"""Build (if needed) and load oracle/_build/liboracle.so.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle.so")
_SRCS = ["pool_oracle.c", "assign_oracle.c", "lcm_oracle.c"]
_lib = None


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, s) for s in _SRCS]
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc, "-O3", "-Wall", "-fPIC", "-shared", "-o", _SO] + srcs)
    return _SO


def build_ref(force: bool = False, ref_dir: str | None = None):
    """Compile the reference's own pool_n.c (where it lies) into oracle/_ref/pool_n_big.

    ref_dir defaults to $TD_REFERENCE_DIR, a checkout of boguszjelinski/taxidispatcher.
    Returns the binary path, or None when neither the binary nor the reference tree exists.
    """
    ref_dir = ref_dir or os.environ.get("TD_REFERENCE_DIR", "")
    out = os.path.join(_HERE, "_ref", "pool_n_big")
    if os.path.exists(out) and os.path.exists(out + "64") and os.path.exists(out + "512") and not force:
        return out
    if not ref_dir or not os.path.exists(os.path.join(ref_dir, "pool_n.c")):
        return out if os.path.exists(out) else None
    subprocess.check_call(["make", "-C", _HERE, "ref", "REF=" + ref_dir])
    return out


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib
