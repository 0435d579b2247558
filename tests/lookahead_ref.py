"""The one-ply look-ahead opponent by the CPU oracle's own rules (tests/lookahead_ref.c), the independent answer that
kz_capture_gain, kz_lookahead_select and VecShogiEnv.lookahead_actions are checked against.  The C file includes
oracle/keisei_oracle.c unchanged and is compiled with the oracle's flags into a temporary directory, once per process;
the pick among the tied moves is added here with the engine's random stream (heuristic_ref.rand32)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from concurrent.futures import ThreadPoolExecutor
from typing import Optional

import numpy as np

from oracle import oracle as orc  # checker only
from tests.heuristic_ref import rand32

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib: Optional[C.CDLL] = None
MATE = 1_000_000
MAX_MOVES = 1024
SALT = 0x4C6F6F6B416864  # VecShogiEnv.LOOKAHEAD_SALT
VALUE = (1, 3, 4, 5, 6, 8, 10, 0, 6, 6, 6, 6, 10, 12)  # by type P L N S G B R K +P +L +N +S +B +R


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="lookahead_ref_"), "liblookahead_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-std=gnu11", "-shared", "-o",
                               out, os.path.join(_HERE, "lookahead_ref.c"), "-lpthread"])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.ref_lookahead.argtypes = [vp, vp, C.c_int, vp, vp, vp]
        L.ref_lookahead.restype = C.c_int
        L.ref_lookahead_batch.argtypes = [C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]
        L.ref_lookahead_batch.restype = None
        L.ref_capture_gain_batch.argtypes = [C.c_int, C.c_int, vp, vp, vp, vp, vp]
        L.ref_capture_gain_batch.restype = None
        _lib = L
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def lookahead(sfen: str) -> dict:
    """One position: {"scores": {action: score} over the legal actions, "best": int, "ties": sorted tied actions}."""
    b, h, side, _ = orc.parse_sfen(sfen)
    b = np.ascontiguousarray(b, np.int8)
    h = np.ascontiguousarray(h, np.uint8)
    score = np.zeros(orc.NACT, np.int32)
    best, ties = C.c_int32(0), C.c_int32(0)
    lib().ref_lookahead(_p(b), _p(h), int(side), _p(score), C.byref(best), C.byref(ties))
    legal = np.flatnonzero(score != np.iinfo(np.int32).min)
    scores = {int(a): int(score[a]) for a in legal}
    return {"scores": scores, "best": best.value, "ties": [a for a in scores if scores[a] == best.value]}


def _batches(n: int, step: int, run, threads: Optional[int]) -> None:
    with ThreadPoolExecutor(max_workers=threads or os.cpu_count() or 4) as ex:
        list(ex.map(run, range(0, n, step)))


def capture_gain_batch(boards, hands, sides, threads: Optional[int] = None) -> dict:
    """R of many positions: gain / count int32 [n], the largest gain over the side to move's legal moves and how many
    moves reach it (0 and 0 without a legal move)."""
    b = np.ascontiguousarray(boards, np.int8)
    h = np.ascontiguousarray(hands, np.uint8)
    s = np.ascontiguousarray(sides, np.uint8)
    n = len(s)
    out = {"gain": np.zeros(n, np.int32), "count": np.zeros(n, np.int32)}
    L = lib()

    def run(first):
        L.ref_capture_gain_batch(first, min(1024, n - first), _p(b), _p(h), _p(s), _p(out["gain"]), _p(out["count"]))

    _batches(n, 1024, run, threads)
    return out


def lookahead_batch(boards, hands, sides, threads: Optional[int] = None) -> dict:
    """Many positions (boards int8 [n, 81], hands uint8 [n, 14], sides uint8 [n]): best / ties int32 [n] and tied uint16
    [n, MAX_MOVES] (the first ties[p] entries of row p, ascending).  Split over threads (the ctypes calls release the
    GIL)."""
    b = np.ascontiguousarray(boards, np.int8)
    h = np.ascontiguousarray(hands, np.uint8)
    s = np.ascontiguousarray(sides, np.uint8)
    n = len(s)
    out = {"best": np.zeros(n, np.int32), "ties": np.zeros(n, np.int32), "tied": np.zeros((n, MAX_MOVES), np.uint16)}
    L = lib()
    step = 64

    def run(first):
        L.ref_lookahead_batch(first, min(step, n - first), _p(b), _p(h), _p(s), _p(out["best"]), _p(out["ties"]),
                              _p(out["tied"]))

    _batches(n, step, run, threads)
    return out


def picks(ref: dict, seed: int, step: int, env_offset: int = 0) -> np.ndarray:
    """The look-ahead pick of every position of a lookahead_batch result: the k-th tied action, k = mulhi(rand32(seed ^
    SALT, env_offset + p, step), ties); -1 without a legal move."""
    out = np.full(len(ref["ties"]), -1, np.int64)
    for p, t in enumerate(ref["ties"].tolist()):
        if t > 0:
            out[p] = int(ref["tied"][p, (rand32(seed ^ SALT, env_offset + p, step) * t) >> 32])
    return out
