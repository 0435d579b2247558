"""Checking moves and mate in one on the device.

    python profiles/mate_probe.py [--out profiles/mate_probe_r2.json]

On one GPU, from 65,536 self-play games after bench.py's 640-ply random pre-roll (max_moves 500):
  * kz_check_bitmap time per launch over the 65,536 legal-bitmap rows, CUDA events over 20 launches after 3 warm-ups;
  * the mean number of legal moves and of checking moves per game, and the games with a mate in one;
  * VecShogiEnv.mate_in_one() from the call to a device sync (torch.cuda.synchronize() inside the timed window), against
    the route it replaces -- list every legal move (legal_actions), expand all of them and keep Tsumi -- timed the same
    way; each the median of 5 runs after one warm-up, alternating, and both results asserted equal.
The card name and power limit are read in the same run (nvidia-smi)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shogidrl_b200 import VecShogiEnv  # noqa: E402
from shogidrl_b200 import _native as nv  # noqa: E402


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


def all_moves_route(env):
    """Mates in one by expanding every legal move (what mate_in_one replaces)."""
    _, parent, actions = env.legal_actions()
    out = env.expand(parent, actions)
    mate = (out["reason"] == nv.TSUMI) & ((out["err"] & nv.ERR_KING_CAPTURE) == 0)
    p = parent.long()
    count = torch.zeros(env.n, dtype=torch.int32, device=env.device).index_add_(0, p, mate.to(torch.int32))
    first = torch.full((env.n,), nv.NUM_ACTIONS, dtype=torch.int64, device=env.device)
    first.scatter_reduce_(0, p, torch.where(mate, actions, nv.NUM_ACTIONS), "amin")
    return {"action": torch.where(count > 0, first, -1), "count": count}


def wall(fn) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mate_probe_r2.json"))
    ap.add_argument("--games", type=int, default=65536)
    args = ap.parse_args()
    n = args.games
    env = VecShogiEnv(n, max_moves_per_game=500, seed=1234)
    env.refresh(random_actions=True)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    for i in range(640):  # bench.py's pre-roll
        env.step(acts[i % 2], next_out=acts[(i + 1) % 2], random_actions=True)
    bitmap = torch.empty((n, nv.BITMAP_WORDS), dtype=torch.int32, device=env.device)
    env.legal_bitmap(bitmap)
    legal = env.legal_count.clone()
    out = torch.empty_like(bitmap)
    count = torch.empty(n, dtype=torch.int32, device=env.device)
    L, sp = nv.lib(), nv.stream_ptr(env.device)

    def launch():
        nv.check(L.kz_check_bitmap(env.state.data_ptr(), n, env.hist_cap, bitmap.data_ptr(), nv.BITMAP_WORDS, out.data_ptr(),
                                   nv.BITMAP_WORDS, count.data_ptr(), sp), "kz_check_bitmap")

    ms = timed(launch)
    a, b = env.mate_in_one(), all_moves_route(env)
    assert torch.equal(a["count"], b["count"]) and torch.equal(a["action"], b["action"])
    t_new, t_old = [], []
    for _ in range(5):
        t_new.append(wall(env.mate_in_one))
        t_old.append(wall(lambda: all_moves_route(env)))
    res = {
        "card": card(), "games": n, "preroll_plies": 640,
        "check_bitmap_ms_per_launch": round(ms, 4),
        "mean_legal_moves": round(float(legal.double().mean()), 3),
        "mean_checking_moves": round(float(count.double().mean()), 3),
        "games_with_mate_in_one": int((a["count"] > 0).sum()),
        "mating_moves": int(a["count"].sum()),
        "mate_in_one_ms": round(1e3 * statistics.median(t_new), 3),
        "expand_all_legal_ms": round(1e3 * statistics.median(t_old), 3),
        "items_expanded": {"checking": int(count.sum()), "all_legal": int(legal.sum())},
        "results_equal": True,
    }
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
