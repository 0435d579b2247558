"""Throughput of move expansion and device perft.

    python profiles/perft_probe.py [--out profiles/perft_probe_r2.json]

On one GPU:
  * perft(5) and perft(6) from the start position (shogidrl_b200.perft): wall time from the call to a device sync
    (torch.cuda.synchronize() inside the timed window), and nodes/s = count / time; each after one untimed warm-up run of
    the same depth, and each count checked against the published value;
  * kz_expand time per 1 M items on a frontier of 65,536 self-play games (bench.py's 640-ply random pre-roll, max_moves
    500): every legal action of every game is an item (in kz_legal_list order, items of one game adjacent), timed with
    CUDA events over 20 launches after 3 warm-ups, in two forms -- counts only (legal_count, no rows, no children: perft's
    last level) and with the legal-bitmap and compact-observation rows (what a search that evaluates children reads);
  * kz_step_rollout at the same 65,536 games (bitmap + compact observation rows, fused random actions), the same way, for
    scale.
The card name and power limit are read in the same run (nvidia-smi)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shogidrl_b200 import VecShogiEnv  # noqa: E402
from shogidrl_b200 import _native as nv  # noqa: E402
from shogidrl_b200.perft import perft  # noqa: E402

PUBLISHED = {5: 19861490, 6: 547581517}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, reps=20, warm=3) -> float:
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def perft_rows() -> dict:
    out = {}
    for d in (5, 6):
        assert perft(depth=d) == [PUBLISHED[d]]  # warm-up (and the check)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = perft(depth=d)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        assert got == [PUBLISHED[d]], (d, got)
        out[f"perft{d}"] = {"nodes": got[0], "seconds": round(s, 4), "nodes_per_s": round(got[0] / s)}
    return out


def expand_rows(n: int) -> dict:
    env = VecShogiEnv(n, max_moves_per_game=500, seed=1234)
    env.refresh(random_actions=True)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    for i in range(640):  # bench.py's pre-roll
        env.step(acts[i % 2], next_out=acts[(i + 1) % 2], random_actions=True)
    _, parent, actions = env.legal_actions()
    m = int(parent.numel())
    L, sp, d = nv.lib(), nv.stream_ptr(env.device), env.device
    count = torch.empty(m, dtype=torch.int32, device=d)
    bitmap = torch.empty((m, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
    cobs = torch.empty((m, nv.COBS_WORDS), dtype=torch.int32, device=d)

    def expand(rows: bool):
        nv.check(L.kz_expand(env.state.data_ptr(), n, env.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1, m, None, 0,
                             bitmap.data_ptr() if rows else None, nv.BITMAP_WORDS, cobs.data_ptr() if rows else None,
                             None, None, None, None, None, count.data_ptr(), None, None, 0, sp), "kz_expand")

    ms_counts = timed(lambda: expand(False))
    ms_rows = timed(lambda: expand(True))
    rb = torch.empty((n, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
    rc = torch.empty((n, nv.COBS_WORDS), dtype=torch.int32, device=d)
    nxt = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    k = [0]

    def step():
        env.step_rollout(nxt[k[0] % 2], None, rb, next_out=nxt[(k[0] + 1) % 2], cobs=rc, random_actions=True)
        k[0] += 1

    ms_step = timed(step)
    return {"games": n, "items": m, "items_per_game": round(m / n, 2),
            "kz_expand_counts_ms": round(ms_counts, 4), "kz_expand_counts_ms_per_1M_items": round(ms_counts * 1e6 / m, 4),
            "kz_expand_rows_ms": round(ms_rows, 4), "kz_expand_rows_ms_per_1M_items": round(ms_rows * 1e6 / m, 4),
            "kz_step_rollout_ms": round(ms_step, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "perft_probe_r2.json"))
    ap.add_argument("--envs", type=int, default=65536)
    args = ap.parse_args()
    res = {"card": card(), "nvcc_sm": "sm_100a"}
    res.update(perft_rows())
    res["expand"] = expand_rows(args.envs)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
