"""Edit-operation alignment restated in C (oracle/align_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/ and tools/bench_align.py's "port" arm import this module; the product package never
does.  The shared library is compiled with gcc on first use into a per-user cache directory keyed
by the source's hash, so a read-only checkout works too.
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from . import pack_strings

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "align_oracle.c")
_LIB = None


def build() -> str:
    with open(_SRC, "rb") as f:
        tag = hashlib.sha256(f.read()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"pllb_align_oracle_{os.getuid()}")
    so = os.path.join(out_dir, f"libalign_oracle_{tag}.so")
    if not os.path.exists(so):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11",
                               "-shared", "-o", tmp, _SRC])
        os.replace(tmp, so)                      # atomic: concurrent builders never load a partial file
    return so


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        i32p = ctypes.POINTER(ctypes.c_int32)
        i64p = ctypes.POINTER(ctypes.c_int64)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        L.oracle_align_batch.restype = None
        L.oracle_align_batch.argtypes = [i32p, i64p, i32p, i64p, i32p, ctypes.c_int32, i64p, u8p, i32p, i32p]
        _LIB = L
    return _LIB


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


def align_batch(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref):
    """Edit-operation alignment of (ref[pair_ref[i]], hyp i) pairs (DESIGN.md §3.10).
    Returns (ops list[str] of 'U'/'S'/'I'/'D' strings, counts int32 [n, 4] = U, S, I, D)."""
    ref_cp = np.ascontiguousarray(ref_cp, np.int32)
    hyp_cp = np.ascontiguousarray(hyp_cp, np.int32)
    ref_off = np.ascontiguousarray(ref_off, np.int64)
    hyp_off = np.ascontiguousarray(hyp_off, np.int64)
    pair_ref = np.ascontiguousarray(pair_ref, np.int32)
    n = len(pair_ref)
    slot = np.diff(ref_off)[pair_ref] + np.diff(hyp_off)[:n]
    ops_off = np.zeros(n + 1, np.int64)
    np.cumsum(slot, out=ops_off[1:])
    ops = np.zeros(max(int(ops_off[-1]), 1), np.uint8)
    n_ops = np.zeros(n, np.int32)
    counts = np.zeros((n, 4), np.int32)
    lib().oracle_align_batch(_p(ref_cp, ctypes.c_int32), _p(ref_off, ctypes.c_int64), _p(hyp_cp, ctypes.c_int32),
                             _p(hyp_off, ctypes.c_int64), _p(pair_ref, ctypes.c_int32), n, _p(ops_off, ctypes.c_int64),
                             _p(ops, ctypes.c_uint8), _p(n_ops, ctypes.c_int32), _p(counts, ctypes.c_int32))
    raw = ops.tobytes()
    return [raw[o:o + k].decode("ascii") for o, k in zip(ops_off[:-1].tolist(), n_ops.tolist())], counts


def align_strings(refs, hyps):
    """align_batch over list[str] pairs (no stripping: the caller passes what is aligned)."""
    rc, ro = pack_strings(refs)
    hc, ho = pack_strings(hyps)
    return align_batch(rc, ro, hc, ho, np.arange(len(hyps), dtype=np.int32))
