"""Cost of restarting finished games from a start-position pool (kz_step_pool) next to the start-position reset.

    python profiles/start_pool_probe.py [--out profiles/start_pool_probe_r2.json]

On one GPU, 65,536 games (bench.py's default) after bench.py's 640-ply random pre-roll, max_moves 500, and a pool of the
128 drop-heavy endgame SFENs of tests/golden/traces_endgame.npz plus hirate:
  * ms per launch of kz_step (mask form) vs kz_step_pool (mask form), and of kz_step_rollout vs kz_step_pool (rollout
    form: legal bitmap + compact observation, no observation rows), each with fused random actions; the two variants of a
    pair are alternated in blocks of 50 launches, 10 blocks each, timed with CUDA events around the step launches alone.
    Both envs start the timing from the SAME games (the pool env's state is a copy of the pre-rolled hirate env's) and
    draw the same actions, so they differ only in where finished games restart; the ratio pool / hirate compares the
    reset paths plus the positions the restarted games then play (endgames from the pool against opening positions);
  * resets per step (finished games) of each variant, counted in separate untimed launches after the timed ones;
  * BASELINE config 3 self-play (16,384 games, horizon 128, the CNN policy-value net under bf16 autocast, rollout replayed
    from a CUDA graph): rollout samples/s of SelfPlayTrainer.collect with and without the pool, alternated.
The card name and power limit are read in the same run (nvidia-smi)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shogidrl_b200 import VecShogiEnv  # noqa: E402

HIRATE = "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def pool_sfens() -> list:
    with np.load(os.path.join(ROOT, "tests", "golden", "traces_endgame.npz")) as z:
        return [str(s) for s in z["sfens"]] + [HIRATE]


def engine(args) -> dict:
    n, out = args.envs, {}
    envs = {"hirate": VecShogiEnv(n, max_moves_per_game=500, seed=1234),
            "pool": VecShogiEnv(n, max_moves_per_game=500, seed=1234, start_positions=pool_sfens())}
    h, p = envs["hirate"], envs["pool"]
    h.refresh(random_actions=True)
    acts = [h.next_actions.clone(), torch.empty_like(h.next_actions)]
    for i in range(640):  # bench.py's pre-roll
        h.step(acts[i % 2], next_out=acts[(i + 1) % 2], random_actions=True)
    p.state.copy_(h.state)  # the same games in both envs (the finished-episode counters included)
    p.step_index = h.step_index
    bufs = {}
    for k, e in envs.items():
        bm = torch.zeros((n, 448), dtype=torch.int32, device=e.device)
        cobs = torch.zeros((n, 40), dtype=torch.int32, device=e.device)
        e.legal_bitmap(bm, cobs=cobs)
        bufs[k] = ([acts[0].clone(), torch.empty_like(acts[0])], bm, cobs, torch.zeros(n, device=e.device),
                   torch.zeros(n, dtype=torch.uint8, device=e.device))
    torch.cuda.synchronize()

    def launch(k, form, i):
        e, (a2, bm, cobs, rew, done) = envs[k], bufs[k]
        a, nx = a2[i % 2], a2[(i + 1) % 2]
        if form == "mask":
            e.step(a, next_out=nx, random_actions=True)
            return e.done
        e.step_rollout(a, None, bm, reward=rew, done=done, next_out=nx, random_actions=True, cobs=cobs)
        return done

    def block(k, form, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            launch(k, form, i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def resets(k, form, reps=100):
        total = torch.zeros((), dtype=torch.int64, device=envs[k].device)
        for i in range(reps):
            total += launch(k, form, i).sum()
        return int(total) / reps

    for form, names in (("mask", ("kz_step", "kz_step_pool (mask)")), ("rollout", ("kz_step_rollout", "kz_step_pool (rollout)"))):
        for k in envs:
            block(k, form, 20)  # warm-up
        ms = {k: [] for k in envs}
        for _ in range(args.blocks):
            for k in envs:
                ms[k].append(block(k, form, args.reps))
        for k, name in zip(envs, names):
            out[name] = {"ms_per_launch_median": float(np.median(ms[k])), "ms_per_launch_blocks": ms[k],
                         "resets_per_step": resets(k, form)}
        a, b = np.median(ms["hirate"]), np.median(ms["pool"])
        out[f"{form}: pool / hirate"] = float(b / a)
    return out


def selfplay(args) -> dict:
    from tests.helpers import make_config
    from shogidrl_b200.core import ActorCritic
    from shogidrl_b200.training.selfplay import SelfPlayTrainer
    N, T = args.ppo_envs, 128
    trs = {}
    for k, sf in (("hirate", None), ("pool", pool_sfens())):
        cfg = make_config(ppo_epochs=10, minibatch_size=16384, steps_per_epoch=N * T)
        cfg.env.seed = 1234
        torch.manual_seed(1234)
        trs[k] = SelfPlayTrainer(ActorCritic(46, 13527), cfg, N, T, "cuda", start_positions=sf)
        for _ in range(3):  # eager rollout, capture + replay, replay
            trs[k].collect()
            trs[k].buffer.clear()
    torch.cuda.synchronize()
    rates = {k: [] for k in trs}
    episodes = {k: 0 for k in trs}
    for _ in range(args.ppo_rounds):
        for k, tr in trs.items():
            t0 = time.perf_counter()
            st = tr.collect()
            torch.cuda.synchronize()
            rates[k].append(N * T / (time.perf_counter() - t0))
            episodes[k] += st["episodes"]
            tr.buffer.clear()
    return {k: {"rollout_samples_per_s_median": float(np.median(v)), "rollout_samples_per_s": v,
                "resets_per_step": episodes[k] / (args.ppo_rounds * T)} for k, v in rates.items()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--blocks", type=int, default=10)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--ppo-envs", type=int, default=16384)
    ap.add_argument("--ppo-rounds", type=int, default=6)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = {"card": card(), "envs": args.envs, "pool": "128 endgame SFENs (tests/golden/traces_endgame.npz) + hirate",
           "engine": engine(args), "config3_selfplay": selfplay(args)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
