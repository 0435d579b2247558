"""The ctypes binding against include/keisei_b200.h, without a GPU: every exported function's argtypes list is as long as
its declaration's parameter list.  A short or extra list shifts raw pointers into the wrong parameters, and that only
shows once something runs on the device."""
import os
import re

from shogidrl_b200 import _native as nv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _parameter_counts():
    src = open(os.path.join(ROOT, "include", "keisei_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    counts = {}
    for name, params in re.findall(r"\b(kz_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        params = params.strip()
        counts[name] = 0 if params in ("", "void") else params.count(",") + 1
    return counts


def test_argtypes_match_header_declarations():
    L = nv.lib()
    counts = _parameter_counts()
    assert sorted(counts) == sorted(nv.EXPORTS)
    for name in nv.EXPORTS:
        got = len(getattr(L, name).argtypes or ())
        assert got == counts[name], f"{name}: {got} ctypes argtypes, {counts[name]} parameters in the header"
