"""Probe: the scripted heuristic opponent on the device.  Prints one JSON line with
  - kernel time of kz_heuristic_actions in mask form and in bitmap form (CUDA events over many launches) next to
    kz_step of the same run, on 65,536 games after a 640-ply random pre-roll (the position mix of bench.py's `value`);
  - the bytes each form reads per game and the rate that makes;
  - evaluation throughput (games/s) of evaluate_vs_opponent at 16,384 envs: "heuristic" vs "random" and an untrained
    agent vs "heuristic", and the heuristic's score against random play at 500 moves per game;
  - the card's name and power limit, read in the same run.
Usage: python profiles/opponent_probe.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from shogidrl_b200 import VecShogiEnv  # noqa: E402
from shogidrl_b200 import _native as nv  # noqa: E402
from shogidrl_b200.evaluation import evaluate_vs_opponent  # noqa: E402

N, PREROLL, REPS = 65536, 640, 200
EVAL_ENVS = 16384


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power = torch.cuda.get_device_name(), None
    return {"name": name, "power_limit": power}


def timed_ms(fn, reps=REPS):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def games_per_s(player, opponent, games, agent_seed=0):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = evaluate_vs_opponent(player, games, opponent=opponent, num_envs=EVAL_ENVS, max_moves_per_game=500, seed=agent_seed)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return r, {"games": r.games, "seconds": round(dt, 3), "games_per_s": round(r.games / dt, 1),
               "mean_length": round(r.mean_length, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("opponent_probe.py needs a CUDA device")
    dev = torch.device("cuda:0")
    env = VecShogiEnv(N, max_moves_per_game=500, device=dev, seed=1234)
    env.refresh(random_actions=True)
    acts = [env.next_actions, torch.empty(N, dtype=torch.int64, device=dev)]
    for i in range(PREROLL):  # untimed: spread the games over all phases of play
        env.step(acts[i % 2], random_actions=True, next_out=acts[(i + 1) % 2])
    bitmap = torch.zeros((N, nv.BITMAP_WORDS), dtype=torch.int32, device=dev)
    env.legal_bitmap(bitmap)
    env.refresh()
    out = torch.empty(N, dtype=torch.int64, device=dev)
    tier = torch.empty(N, dtype=torch.uint8, device=dev)
    cnt = torch.empty(N, dtype=torch.int32, device=dev)
    ms_mask = timed_ms(lambda: env.heuristic_actions(out=out, tier=tier))
    top_mask = out.clone()
    ms_bitmap = timed_ms(lambda: env.heuristic_actions(out=out, bitmap=bitmap, tier=tier, tier_count=cnt))
    same = bool(torch.equal(top_mask, out))
    tiers = torch.bincount(tier.long(), minlength=256)
    state = {"i": PREROLL}

    def step():
        i = state["i"]
        env.step(acts[i % 2], random_actions=True, next_out=acts[(i + 1) % 2])
        state["i"] = i + 1

    ms_step = timed_ms(step)
    # bytes a game's pick reads: the legal set (846 16-byte windows of the mask row / words 0..422 of the bitmap row), the
    # 81 board bytes and the side byte; the action written is 8 bytes
    board_b = 81 + 1 + 8
    mask_b, bitmap_b = 846 * 16 + board_b, 423 * 4 + board_b
    res = {
        "probe": "opponent_probe", "games": N, "preroll_plies": PREROLL, "launches_timed": REPS,
        "kz_heuristic_actions_mask_ms": round(ms_mask, 4), "kz_heuristic_actions_bitmap_ms": round(ms_bitmap, 4),
        "kz_step_ms": round(ms_step, 4), "mask_and_bitmap_agree": same,
        "bytes_per_game": {"mask": mask_b, "bitmap": bitmap_b},
        "read_gbs": {"mask": round(N * mask_b / ms_mask / 1e6, 1), "bitmap": round(N * bitmap_b / ms_bitmap / 1e6, 1)},
        "working_set_mb": {"mask": round(N * mask_b / 1e6, 1), "bitmap": round(N * bitmap_b / 1e6, 1)},
        "top_tier_share": {k: round(float(tiers[t]) / N, 4) for k, t in (("capture", 0), ("pawn", 1), ("other", 2),
                                                                           ("none", 255))},
    }
    from shogidrl_b200.core import ActorCritic, PPOAgent
    from tests.helpers import make_config
    torch.manual_seed(0)
    agent = PPOAgent(ActorCritic(46, 13527), make_config(), dev, use_mixed_precision=True)
    evaluate_vs_opponent("heuristic", 64, opponent="random", num_envs=64, max_moves_per_game=20)  # warm-up
    evaluate_vs_opponent(agent, 64, opponent="heuristic", num_envs=64, max_moves_per_game=20)
    r_hr, res["eval_heuristic_vs_random"] = games_per_s("heuristic", "random", EVAL_ENVS)
    _, res["eval_random_vs_random"] = games_per_s("random", "random", EVAL_ENVS)
    _, res["eval_agent_vs_heuristic"] = games_per_s(agent, "heuristic", EVAL_ENVS)
    res["heuristic_vs_random_500_moves"] = {"games": r_hr.games, "heuristic_wins": r_hr.agent_wins,
                                            "random_wins": r_hr.opponent_wins, "draws": r_hr.draws,
                                            "heuristic_win_rate": round(r_hr.win_rate, 4)}
    res["card"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
