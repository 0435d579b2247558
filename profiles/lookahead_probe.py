"""The one-ply look-ahead opponent on the device.

    python profiles/lookahead_probe.py [--out profiles/lookahead_probe_r2.json]

On one GPU, from self-play games after bench.py's 640-ply random pre-roll (max_moves 500), at 16,384 and 65,536 games:
  * items per decision: the children (legal moves) and the checking replies that the mate-in-one route expands, per game;
  * VecShogiEnv.lookahead_actions() from the call to a device sync, the median of 5 runs after one warm-up, and the
    peak device memory it allocates at the default max_items;
  * kz_capture_gain over the children of the first chunk and kz_lookahead_select over every game, CUDA events over 20
    launches after 3 warm-ups.
Then evaluation at 16,384 envs with 500-move games (one game per env): games/s and wins / draws / losses of the
look-ahead player against "random" and against "heuristic".  The card name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
from mate_probe import card, timed, wall  # noqa: E402
from shogidrl_b200 import VecShogiEnv  # noqa: E402
from shogidrl_b200 import _native as nv  # noqa: E402
from shogidrl_b200._batch import chunks  # noqa: E402
from shogidrl_b200.evaluation import evaluate_vs_opponent  # noqa: E402


def preroll(n: int) -> VecShogiEnv:
    env = VecShogiEnv(n, max_moves_per_game=500, seed=1234)
    env.refresh(random_actions=True)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    for i in range(640):  # bench.py's pre-roll
        env.step(acts[i % 2], next_out=acts[(i + 1) % 2], random_actions=True)
    return env


def at_size(n: int) -> dict:
    env = preroll(n)
    L, d, sp = nv.lib(), env.device, nv.stream_ptr(env.device)
    env.lookahead_actions()  # warm-up
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ref = env.lookahead_actions().clone()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    t = [wall(env.lookahead_actions) for _ in range(5)]
    assert torch.equal(env.lookahead_actions(), ref)

    # the pipeline's intermediate arrays, as lookahead_actions builds them, for the kernel timings
    offsets, parent, actions = env.legal_actions()
    m = int(parent.numel())
    done, reason, err = (torch.empty(m, dtype=torch.uint8, device=d) for _ in range(3))
    gain, mates = (torch.empty(m, dtype=torch.int32, device=d) for _ in range(2))
    off_h = offsets.cpu().numpy()
    chunk = 1 << 20
    for a, b in chunks(off_h, chunk):
        env._lookahead_chunk(int(off_h[a]), int(off_h[b]), parent, actions, done, reason, err, gain, mates)
    # the first chunk's children again, for kz_capture_gain and their checking replies
    m0 = min(m, chunk)
    total = C.c_int64()
    nv.check(L.kz_state_layout(m0, 1, None, C.byref(total)), "kz_state_layout")
    child = torch.empty(total.value, dtype=torch.uint8, device=d)
    rows = torch.empty((m0, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
    nv.check(L.kz_expand(env.state.data_ptr(), n, env.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1, m0, None, 0,
                         rows.data_ptr(), nv.BITMAP_WORDS, None, None, None, None, None, None, None, None,
                         child.data_ptr(), 1, sp), "kz_expand")
    g0 = torch.empty(m0, dtype=torch.int32, device=d)
    checks = torch.empty(m0, dtype=torch.int32, device=d)
    crow = torch.empty_like(rows)
    nv.check(L.kz_check_bitmap(child.data_ptr(), m0, 1, rows.data_ptr(), nv.BITMAP_WORDS, crow.data_ptr(), nv.BITMAP_WORDS,
                               checks.data_ptr(), sp), "kz_check_bitmap")
    del crow

    def capture_gain():
        nv.check(L.kz_capture_gain(child.data_ptr(), m0, 1, rows.data_ptr(), nv.BITMAP_WORDS, g0.data_ptr(), None, sp),
                 "kz_capture_gain")

    pick = torch.empty(n, dtype=torch.int64, device=d)
    seed = (env.seed ^ env.LOOKAHEAD_SALT) & 0xFFFFFFFFFFFFFFFF

    def select():
        nv.check(L.kz_lookahead_select(env.state.data_ptr(), n, env.hist_cap, offsets.data_ptr(), m, actions.data_ptr(), 1,
                                       done.data_ptr(), reason.data_ptr(), err.data_ptr(), gain.data_ptr(), mates.data_ptr(),
                                       seed, env.step_index, env.env_offset, pick.data_ptr(), 1, None, None, sp),
                 "kz_lookahead_select")

    cg_ms, sel_ms = timed(capture_gain), timed(select)
    assert torch.equal(pick, ref) and torch.equal(g0, gain[:m0])
    checks_per_child = float(checks.double().mean())
    return {
        "games": n,
        "children_per_decision": round(m / n, 3),
        "checking_replies_per_child": round(checks_per_child, 3),
        "checking_replies_per_decision": round(checks_per_child * m / n, 3),
        "lookahead_actions_ms": round(1e3 * statistics.median(t), 3),
        "lookahead_actions_ms_runs": [round(1e3 * x, 3) for x in t],
        "peak_memory_gb_default_max_items": round(peak / 1e9, 3),
        "capture_gain_ms": {"items": m0, "ms_per_launch": round(cg_ms, 4)},
        "lookahead_select_ms": {"games": n, "items": m, "ms_per_launch": round(sel_ms, 4)},
    }


def evaluation(n: int) -> dict:
    out = {}
    for opp in ("random", "heuristic"):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = evaluate_vs_opponent("lookahead", n, opponent=opp, num_envs=n, max_moves_per_game=500, seed=7)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out[f"lookahead_vs_{opp}"] = {"games": r.games, "wins": r.agent_wins, "draws": r.draws, "losses": r.opponent_wins,
                                      "mean_length": round(r.mean_length, 1), "seconds": round(dt, 2),
                                      "games_per_s": round(r.games / dt, 1)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "lookahead_probe_r2.json"))
    ap.add_argument("--sizes", default="16384,65536")
    ap.add_argument("--eval-envs", type=int, default=16384)
    args = ap.parse_args()
    res = {"card": card(), "preroll_plies": 640, "max_moves": 500,
           "sizes": [at_size(int(s)) for s in args.sizes.split(",")],
           "evaluation": {"envs": args.eval_envs, **evaluation(args.eval_envs)}}
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
