"""Move-tree perft by the CPU oracle's own generator (tests/perft_ref.c), the independent count that
shogidrl_b200.perft is checked against.  The C file includes oracle/keisei_oracle.c unchanged and is compiled with the
oracle's flags into a temporary directory, once per process."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from typing import Optional

import numpy as np

from oracle import oracle as orc  # checker only

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="perft_ref_"), "libperft_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-shared", "-o",
                               out, os.path.join(_HERE, "perft_ref.c"), "-lpthread"])
        L = C.CDLL(out)
        L.ref_perft.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.ref_perft.restype = C.c_int64
        _lib = L
    return _lib


def perft(sfen: Optional[str], depth: int, divide: bool = False):
    """perft of ``sfen`` (None: the start position) to ``depth`` plies; with ``divide`` a dict {root action: count}."""
    if sfen is None:
        b, h, m = orc.OracleGame().export()
        side = int(m[0])
    else:
        b, h, side, _ = orc.parse_sfen(sfen)
    b = np.ascontiguousarray(b, np.int8)
    h = np.ascontiguousarray(h, np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    if not divide:
        return int(lib().ref_perft(p(b), p(h), int(side), int(depth), None))
    out = np.full(orc.NACT, -1, np.int64)
    lib().ref_perft(p(b), p(h), int(side), int(depth), p(out))
    return {int(a): int(out[a]) for a in np.flatnonzero(out >= 0)}
