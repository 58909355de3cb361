"""ctypes binding of the proposal-pair parse in C (oracle/proposal_parse.c).  TEST INFRASTRUCTURE ONLY.

Compiles libproposal_parse.so with gcc on first use, next to the source when that directory is writable, otherwise
in a temporary directory.  See proposal_parse.py for the numpy specification this C code must equal.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .c_oracle import CGeometry, _Geom, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "proposal_parse.c")
_DEPS = (_SRC, os.path.join(_HERE, "ppn_oracle.c"))
CFLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra"]


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libproposal_parse.so")
    if not os.access(_HERE, os.W_OK):
        so = os.path.join(tempfile.gettempdir(), f"libproposal_parse_{os.getuid()}.so")
    if force or not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in _DEPS):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run([os.environ.get("CC", "gcc"), *CFLAGS, _SRC, "-o", tmp, "-shared", "-lpthread", "-lm"],
                       check=True, capture_output=True)
        os.replace(tmp, so)
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        i32p, f32p = C.POINTER(C.c_int32), C.POINTER(C.c_float)
        _lib.ppn_oracle_proposal_parse_batch.argtypes = [f32p, C.c_int, C.POINTER(_Geom), C.c_int, i32p, i32p, i32p, f32p,
                                                         f32p, i32p]
    return _lib


def proposal_parse_batch(head: np.ndarray, g, n_threads: int = 1, stats: bool = False):
    """The proposal-pair parse (C twin of oracle/proposal_parse.py) of head [B,C,H,W] fp32 -> dict(count [B],
    root_cell [B, HW], part_cell [B, HW, K], part_score, part_box; slots past count: -1 / 0), plus, with ``stats``,
    n_prop [B, K] proposals per part and n_pairs [B, E] candidate pairs per limb.  Raises ValueError when the track
    orders are not a tree."""
    head = np.ascontiguousarray(head, np.float32)
    B = head.shape[0]
    assert head.shape[1:] == (g.C, g.H, g.W), head.shape
    HW, K = g.H * g.W, g.K
    cg = CGeometry(g)
    r = dict(count=np.zeros(B, np.int32), root_cell=np.full((B, HW), -1, np.int32),
             part_cell=np.full((B, HW, K), -1, np.int32), part_score=np.zeros((B, HW, K), np.float32),
             part_box=np.zeros((B, HW, K, 4), np.float32))
    st = np.zeros((B, K + g.E), np.int32) if stats else None
    rc = lib().ppn_oracle_proposal_parse_batch(_p(head, C.c_float), B, C.byref(cg.c), n_threads,
                                               _p(r["count"], C.c_int32), _p(r["root_cell"], C.c_int32),
                                               _p(r["part_cell"], C.c_int32), _p(r["part_score"], C.c_float),
                                               _p(r["part_box"], C.c_float), None if st is None else _p(st, C.c_int32))
    if rc == -2:
        raise ValueError("track orders do not form a tree rooted at part 0")
    assert rc == 0, rc
    if stats:
        r["n_prop"], r["n_pairs"] = st[:, :K], st[:, K:]
    return r
