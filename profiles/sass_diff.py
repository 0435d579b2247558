"""Compare the compiled kz_step_kernel instantiations of two versions of the engine, instruction for instruction.

    python profiles/sass_diff.py <git revision>

builds csrc/kz_engine.cu of the revision and of the working tree for sm_100a (in a temporary directory), prints each
build's ptxas register / spill line for every kz_step_kernel instantiation and diffs the SASS of the instantiations
both builds have.  Kernel names differ between builds (the anonymous namespace's hash, template arguments), so each
body is compared under its template arguments only, with the name tokens masked out.  Needs nvcc and cuobjdump, no
GPU.  Every local-memory instruction (STL / LDL: spills) of each step instantiation (modes 1, 2) is listed with its position in the
body.  Exit status 1 when a common instantiation differs."""
from __future__ import annotations

import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC", "-cubin",
         "-Xptxas", "-v"]
FILES = ["shogidrl_b200/csrc/kz_engine.cu", "shogidrl_b200/csrc/kz_common.cuh", "include/keisei_b200.h"]


def tree_of(rev: str | None, dst: str) -> str:
    for f in FILES:
        os.makedirs(os.path.join(dst, os.path.dirname(f)), exist_ok=True)
        if rev is None:
            data = open(os.path.join(ROOT, f), "rb").read()
        else:
            data = subprocess.run(["git", "-C", ROOT, "show", f"{rev}:{f}"], check=True, capture_output=True).stdout
        open(os.path.join(dst, f), "wb").write(data)
    return os.path.join(dst, FILES[0])


def targs(mangled: str) -> str:
    """'<1>' / '<1,false>' -> the template arguments with the default POOL = false made explicit."""
    m = re.search(r"kz_step_kernelILi(\d)E(?:Lb([01])E)?E", mangled)
    return f"<{m.group(1)},{'true' if m.group(2) == '1' else 'false'}>"


def build(src: str, out: str):
    r = subprocess.run([f"{CUDA}/bin/nvcc"] + FLAGS + [src, "-o", out], capture_output=True, text=True)
    if r.returncode:
        sys.exit(r.stderr)
    usage, cur = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S*kz_step_kernel\S*)'", line)
        if m:
            cur = targs(m.group(1))
        elif cur and ("spill" in line or "Used" in line):
            usage[cur] = usage.get(cur, "") + " " + line.split(":", 1)[-1].strip()
            if "Used" in line:
                cur = None
    sass = subprocess.run([f"{CUDA}/bin/cuobjdump", "-sass", out], check=True, capture_output=True, text=True).stdout
    bodies, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = targs(m.group(1)) if "kz_step_kernel" in m.group(1) else None
            if cur:
                bodies[cur] = []
            continue
        if cur and re.match(r"\s*/\*[0-9a-f]{4,}\*/", line):
            bodies[cur].append(re.sub(r"_Z\w+", "<sym>", line.split(";")[0]).strip())
    return usage, bodies


def main() -> int:
    rev = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
    with tempfile.TemporaryDirectory() as tmp:
        old = build(tree_of(rev, os.path.join(tmp, "old")), os.path.join(tmp, "old.cubin"))
        new = build(tree_of(None, os.path.join(tmp, "new")), os.path.join(tmp, "new.cubin"))
    bad = 0
    for name, (usage, bodies) in ((rev, old), ("working tree", new)):
        print(f"{name}:")
        for k in sorted(bodies):
            print(f"  kz_step_kernel{k}: {len(bodies[k])} instructions;{usage.get(k, '')}")
    for name, (_, bodies) in ((rev, old), ("working tree", new)):
        for k in sorted(bodies):
            local = [(i, ins) for i, ins in enumerate(bodies[k]) if re.search(r"\b(STL|LDL)\b", ins)]
            if local and not k.startswith("<0"):  # the refresh kernel's many spills are off the step path
                print(f"{name} kz_step_kernel{k} local memory (instruction index / {len(bodies[k])}):")
                for i, ins in local:
                    print(f"    {i:5d}  {ins}")
    for k in sorted(set(old[1]) & set(new[1])):
        same = old[1][k] == new[1][k]
        bad += not same
        print(f"kz_step_kernel{k}: SASS {'identical' if same else 'DIFFERS'}")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
