"""Checking moves and mates in one by the CPU oracle's own rules (tests/checks_ref.c), the independent answer that
kz_check_bitmap and VecShogiEnv.mate_in_one are checked against.  The C file includes oracle/keisei_oracle.c unchanged and
is compiled with the oracle's flags into a temporary directory, once per process."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor
from typing import Optional

import numpy as np

from oracle import oracle as orc  # checker only

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib: Optional[C.CDLL] = None
WORDS = 423
CLASSES = ("direct", "discovered", "double", "drop", "no_king", "promotion_only")


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="checks_ref_"), "libchecks_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-shared", "-o",
                               out, os.path.join(_HERE, "checks_ref.c"), "-lpthread"])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.ref_checks.argtypes = [vp, vp, C.c_int, vp, vp, vp]
        L.ref_checks.restype = C.c_int
        L.ref_checks_batch.argtypes = [C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp]
        L.ref_checks_batch.restype = None
        _lib = L
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def checks(sfen: str) -> dict:
    """One position: {"legal", "checks", "mates", "king_capture_mates": sorted action lists, "classes": {action: class
    name(s)}, "enemy_in_check": bool}."""
    b, h, side, _ = orc.parse_sfen(sfen)
    b = np.ascontiguousarray(b, np.int8)
    h = np.ascontiguousarray(h, np.uint8)
    cls = np.zeros(orc.NACT, np.uint8)
    mate = np.zeros(orc.NACT, np.uint8)
    eic = C.c_int(0)
    lib().ref_checks(_p(b), _p(h), int(side), _p(cls), _p(mate), C.byref(eic))
    legal = np.flatnonzero(cls != 0xFF)
    chk = legal[cls[legal] != 0]
    names = {}
    for a in chk.tolist():
        c = int(cls[a])
        names[a] = CLASSES[(c & 7) - 1] + ("+promotion_only" if c & 8 else "")
    return {"legal": legal.tolist(), "checks": chk.tolist(), "mates": np.flatnonzero(mate == 1).tolist(),
            "king_capture_mates": np.flatnonzero(mate == 2).tolist(), "classes": names, "enemy_in_check": bool(eic.value)}


def checks_batch(boards, hands, sides, threads: Optional[int] = None) -> dict:
    """Many positions (boards int8 [n, 81], hands uint8 [n, 14], sides uint8 [n]): legal / check uint32 [n, 423] bitmaps,
    mate_count / mate_lowest int32 [n] (mates that do not capture the king), class_counts int32 [n, 6] (CLASSES order) and
    enemy_in_check uint8 [n].  Split over threads (the ctypes calls release the GIL)."""
    b = np.ascontiguousarray(boards, np.int8)
    h = np.ascontiguousarray(hands, np.uint8)
    s = np.ascontiguousarray(sides, np.uint8)
    n = len(s)
    out = {"legal": np.zeros((n, WORDS), np.uint32), "check": np.zeros((n, WORDS), np.uint32),
           "mate_count": np.zeros(n, np.int32), "mate_lowest": np.zeros(n, np.int32),
           "class_counts": np.zeros((n, 6), np.int32), "enemy_in_check": np.zeros(n, np.uint8)}
    L = lib()
    step = 256

    def run(first):
        L.ref_checks_batch(first, min(step, n - first), _p(b), _p(h), _p(s), _p(out["legal"]), _p(out["check"]),
                           _p(out["mate_count"]), _p(out["mate_lowest"]), _p(out["class_counts"]), _p(out["enemy_in_check"]))

    with ThreadPoolExecutor(max_workers=threads or os.cpu_count() or 4) as ex:
        list(ex.map(run, range(0, n, step)))
    return out
