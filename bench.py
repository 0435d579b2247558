#!/usr/bin/env python
"""bench.py -- legal-masked Shogi env steps/sec on B200 (BASELINE.json metric, config 2).

    python bench.py --gpus N --steps K --warmup W            # product arm (CUDA kernels, C ABI)
    python bench.py --impl reference --steps K --warmup W    # reference arm: CPU oracle port, all host threads
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs as DIR/<name>.npy

A "step" is one pass of the hot path over one batch: kz_step over 65,536 device-resident games per GPU
(apply the action, generate the successor's legal moves, termination, auto-reset, write the 13,527-byte
legal mask + 46x9x9 fp32 observation + reward/done/reason/winner), actions = uniform-random legal via the
counter-based RNG keyed (seed, env, step).  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "legal-masked Shogi env steps/sec"
UNIT = "env_steps/s"
ENVS_PER_GPU = 65536
MAX_MOVES = 500
SEED = 1234
PREROLL = 640  # untimed plies that spread the games over all phases (synthetic input preparation)

# SURVEY.md section 8(d): algorithmic bytes per env step
OBS_B, MASK_B, SCALARS_B, ACTION_B, STATE_B, HIST_APPEND_B = 14904, 13527, 7, 8, 238, 16


def algorithmic_bytes_per_step(mean_ply: float) -> float:
    """SURVEY.md section 8(d): 28,438 written + 8 action + 238 state + 16 history append + 8*ply history scan."""
    return OBS_B + MASK_B + SCALARS_B + ACTION_B + STATE_B + HIST_APPEND_B + 8.0 * mean_ply


def implementation_bytes_per_step() -> float:
    """What this implementation must move per env step: the same outputs and action, 96+32 B of state read and
    written, and one 512 B probe + 16 B update of the repetition table (no per-ply scan)."""
    return OBS_B + MASK_B + SCALARS_B + ACTION_B + 2 * 128 + 512 + 16


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline_sample(threads: int, seconds_budget: float = 20.0):
    """The oracle port timed on the host cores on a bounded sample of the same workload."""
    from oracle import oracle as orc
    n = GAMES_PER_THREAD * threads
    batch = orc.OracleBatch(n, MAX_MOVES, SEED, threads)
    batch.run(8)  # warm caches / threads
    t0 = time.perf_counter()
    steps, T = 0, 0
    while True:
        steps += batch.run(40)
        T += 40
        dt = time.perf_counter() - t0
        if dt > seconds_budget or T >= 640:
            break
    return {"value": steps / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n} games x {T} plies from the start position with auto-reset (max_moves {MAX_MOVES}), "
                      f"legal moves + mask + make_move + observation per ply, {dt:.1f} s, C oracle (oracle/keisei_oracle.c)"}


def real_reference_ppo_sample(threads: int, timesteps: int = 256, epochs: int = 10, minibatch: int = 64):
    """BASELINE.md section 3.2 on this box: the unmodified reference's sequential PPO loop (baseline/ref_ppo_loop.py over
    baseline/_ref), one process with `threads` torch threads, one epoch of `timesteps` steps.  None without the install."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "keisei")):
        return None
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", WANDB_DISABLED="true", WANDB_MODE="disabled")
    try:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "ref_ppo_loop.py"), ref_dir, str(timesteps),
                              str(epochs), str(minibatch), str(threads)], capture_output=True, text=True, env=env, timeout=600)
        r = json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as ex:
        return {"unavailable": "baseline/_ref is present but the reference PPO loop did not run here: "
                               + (str(ex) + " " + (locals().get("out").stderr[-300:] if locals().get("out") else "")).replace("\n", " | ")}
    return {"value": r["samples_per_s"], "unit": "samples/s", "cores": threads, "kind": "reference",
            "rollout_samples_per_s": timesteps / r["collect_s"], "update_samples_per_s": timesteps / r["update_s"],
            "sample": f"1 epoch of {timesteps} timesteps (reference default 2048), minibatch {minibatch}, ppo_epochs {epochs}: keisei "
                      f"ShogiGame + PolicyOutputMapper + PPOAgent.select_action / learn + ExperienceBuffer + ActorCritic(46, 13527) "
                      f"from baseline/_ref on the CPU, one process, {threads} torch threads (collect {r['collect_s']:.1f} s, "
                      f"update {r['update_s']:.1f} s)"}


GAMES_PER_THREAD = 256  # both CPU legs (cpu_baseline of the product line, --impl reference) step this many games per host thread


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself is pure Python and
    cannot travel to the GPU box) on all host threads.  One step = one env step of every game of the batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as orc
    threads = os.cpu_count() or 1
    n = GAMES_PER_THREAD * threads
    batch = orc.OracleBatch(n, MAX_MOVES, SEED, threads)
    batch.run(256)  # untimed pre-roll: spread the games over the phases of play
    for _ in range(args.warmup):
        batch.run(1)
    t0 = time.perf_counter()
    plies = 0.0
    for _ in range(args.steps):
        batch.run(1)
        plies += batch.mean_ply
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "threads": threads,
        "config": {"workload": f"random-legal self-play, {n} games per step = {GAMES_PER_THREAD} per host thread x {threads} "
                               f"threads (bounded sample of BASELINE config 2: 65,536 games/GPU; the CPU rate does not depend "
                               f"on the batch size), max_moves {MAX_MOVES}, auto-reset, 256-ply pre-roll",
                   "mean_ply": plies / max(1, args.steps)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{n} games x {args.steps} timed plies, C oracle port of keisei.shogi (the pure-Python "
                                   "reference is timed separately: cpu_baseline_reference)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    ref = real_reference_sample(threads)
    if ref is not None:
        line["cpu_baseline_reference"] = ref
    if not args.no_ppo:
        # the second half of BASELINE.json's metric on the host: same minibatch size as the product arm states
        line["ppo"] = measure_reference_ppo(args.ppo_minibatch, args.ppo_minibatch, args.ppo_epochs, 1, 0, threads)
        line["ppo_reference_defaults"] = measure_reference_ppo(args.ref_ppo_steps, 64, args.ppo_epochs, 1, 0, threads)
        rp = real_reference_ppo_sample(threads, epochs=args.ppo_epochs)
        if rp is not None:
            line["ppo_cpu_baseline_reference"] = rp
    emit(line)
    return 0


def real_reference_sample(threads: int, seconds: float = 30.0):
    """The UNMODIFIED Python reference (keisei.shogi.ShogiGame + PolicyOutputMapper from baseline/_ref, installed with
    `pip install --no-deps --target baseline/_ref`), BASELINE.md section 3.1 loop -- get_legal_moves, get_legal_mask,
    make_move with the config-1 action rule -- in `threads` processes for `seconds` of wall time.  None when the install
    is not on this box (it is git-ignored and only travels with an untracked copy of the tree)."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "keisei")):
        return None
    code = (
        "import sys, time, random\n"
        f"sys.path.insert(0, {ref_dir!r})\n"
        "import torch; torch.set_num_threads(1)\n"
        "from keisei.shogi import ShogiGame\n"
        "from keisei.utils import PolicyOutputMapper\n"
        "seed, budget = int(sys.argv[1]), float(sys.argv[2])\n"
        "rng = random.Random(seed); mapper = PolicyOutputMapper(); g = ShogiGame(max_moves_per_game=500)\n"
        "dev = torch.device('cpu'); n = 0; t0 = time.perf_counter()\n"
        "while time.perf_counter() - t0 < budget:\n"
        "    lm = g.get_legal_moves()\n"
        "    if not lm or g.game_over:\n"
        "        g.reset(); continue\n"
        "    mapper.get_legal_mask(lm, dev)\n"
        "    idx = sorted(mapper.shogi_move_to_policy_index(m) for m in lm)\n"
        "    g.make_move(mapper.policy_index_to_shogi_move(idx[rng.randrange(len(idx))]))\n"
        "    n += 1\n"
        "print(n, time.perf_counter() - t0)\n")
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", WANDB_DISABLED="true", WANDB_MODE="disabled")
    t0 = time.perf_counter()
    procs = [subprocess.Popen([sys.executable, "-c", code, str(100 + i), str(seconds)], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True, env=env) for i in range(threads)]
    steps, ok, err = 0, 0, ""
    for p in procs:
        try:
            out, e = p.communicate(timeout=seconds + 240)
            a, _ = out.split()
            steps += int(a); ok += 1
        except Exception as ex:  # import failure on this box, timeout, ...
            p.kill()
            err = (locals().get("e") or str(ex))[-300:]
    wall = time.perf_counter() - t0
    if ok == 0:
        return {"unavailable": "baseline/_ref is present but the reference did not run here: " + err.strip().replace("\n", " | ")}
    return {"value": steps / seconds, "unit": UNIT, "cores": ok, "kind": "reference", "per_core": steps / seconds / ok,
            "sample": f"{ok} processes x {seconds:.0f} s of keisei.shogi.ShogiGame from baseline/_ref (get_legal_moves + "
                      f"get_legal_mask + make_move, uniform-random legal play from the start position, max_moves 500), "
                      f"{steps} plies, {wall:.0f} s wall incl. imports"}


def measure_reference_ppo(S, MB, EPOCHS, steps, warm, threads):
    """The reference's sequential CPU trainer restated -- one game, batch-1 select_action (masked softmax + Categorical
    sample, ppo_agent.py:134-223), ExperienceBuffer GAE (experience_buffer.py:99-145), then PPOAgent.learn
    (ppo_agent.py:243-460: ppo_epochs x minibatches of MB, clipped surrogate + value MSE + entropy, clip_grad_norm_ 0.5,
    Adam) -- on the oracle engine and the default CNN (neural_network.py:10-29) in plain fp32 PyTorch on all host threads.
    One step = one epoch of S timesteps; value = timesteps per second."""
    import numpy as np
    import torch
    import torch.nn as nn
    from oracle import oracle as orc
    torch.set_num_threads(threads)
    torch.manual_seed(SEED)
    gamma, lam, clip_eps, cv, ce = 0.99, 0.95, 0.2, 0.5, 0.01

    class Net(nn.Module):  # keisei/core/neural_network.py:10-29
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(46, 16, 3, padding=1)
            self.policy_head = nn.Linear(16 * 81, 13527)
            self.value_head = nn.Linear(16 * 81, 1)

        def forward(self, x):
            h = torch.relu(self.conv(x)).flatten(1)
            return self.policy_head(h), self.value_head(h).squeeze(-1)

    def dist_of(logits, mask):
        probs = torch.softmax(torch.where(mask, logits, torch.full((), float("-inf"))), dim=-1)
        return torch.distributions.Categorical(probs=probs)

    model = Net()
    opt = torch.optim.Adam(model.parameters(), lr=3e-4)
    game = orc.OracleGame(MAX_MOVES)
    shuffle_rng = np.random.default_rng(SEED)

    def epoch():
        obs = np.zeros((S, 46, 9, 9), np.float32); masks = np.zeros((S, 13527), np.uint8)
        act = np.zeros(S, np.int64); lp = np.zeros(S, np.float32); val = np.zeros(S, np.float32)
        rew = np.zeros(S, np.float32); done = np.zeros(S, np.uint8)
        t_roll = time.perf_counter()
        for t in range(S):
            obs[t] = game.observation(); masks[t] = game.legal_mask()
            with torch.no_grad():
                logits, v = model(torch.from_numpy(obs[t:t + 1]))
                d = dist_of(logits, torch.from_numpy(masks[t:t + 1]).bool())
                a = d.sample()
                lp[t] = float(d.log_prob(a)); val[t] = float(v); act[t] = int(a)
            r, dn, _, _ = game.make_move(int(a))
            rew[t], done[t] = r, dn
            if dn:
                game.reset()
        with torch.no_grad():
            last_v = float(model(torch.from_numpy(game.observation()[None]))[1])
        adv, ret = orc.gae(rew[:, None], val[:, None], done[:, None], np.float32(last_v), gamma, lam)
        t_roll = time.perf_counter() - t_roll
        to = torch.from_numpy
        obs_t, mask_t, act_t = to(obs), to(masks).bool(), to(act)
        lp_t, adv_t, ret_t = to(lp), to(adv[:, 0].copy()), to(ret[:, 0].copy())
        adv_t = (adv_t - adv_t.mean()) / (adv_t.std() + 1e-8)
        for _ in range(EPOCHS):
            idx = shuffle_rng.permutation(S)  # ppo_agent.py:298
            for s0 in range(0, S, MB):
                mb = torch.from_numpy(idx[s0:s0 + MB])
                logits, v = model(obs_t[mb])
                d = dist_of(logits, mask_t[mb])
                new_lp, ent = d.log_prob(act_t[mb]), d.entropy()
                ratio = torch.exp(new_lp - lp_t[mb])
                pol = -torch.min(ratio * adv_t[mb], torch.clamp(ratio, 1 - clip_eps, 1 + clip_eps) * adv_t[mb]).mean()
                loss = pol + cv * torch.nn.functional.mse_loss(v, ret_t[mb]) - ce * ent.mean()
                opt.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(model.parameters(), 0.5)
                opt.step()
        return t_roll

    for _ in range(warm):
        epoch()
    t0 = time.perf_counter()
    roll = sum(epoch() for _ in range(steps))
    dt = time.perf_counter() - t0
    value = S * steps / dt
    sample = (f"{steps} epoch(s) x {S} timesteps of one game (reference default: 2048), minibatch {MB}, ppo_epochs {EPOCHS}, "
              f"C oracle engine + fp32 PyTorch CPU model on {threads} threads (the pure-Python reference cannot run on the GPU box)")
    return {"metric": "PPO self-play samples/sec", "value": value, "unit": "samples/s", "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * dt / steps, "dtype": "f32", "threads": threads, "minibatch": MB, "timesteps_per_epoch": S,
            "ppo_epochs": EPOCHS, "rollout_samples_per_s": S * steps / roll,
            "update_samples_per_s": S * steps / max(1e-9, dt - roll), "kind": "port", "sample": sample}


def run_reference_ppo(args):
    """--impl reference --workload ppo: the PPO arm on the host as its own line."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    S = args.ref_ppo_steps
    MB = min(args.ppo_minibatch, S) if args.ref_same_minibatch else 64
    r = measure_reference_ppo(S, MB, args.ppo_epochs, max(1, min(args.steps, 8)), min(args.warmup, 1), threads)
    emit({"impl": "reference", "metric": r["metric"], "value": r["value"], "unit": r["unit"], "n_gpus": args.gpus,
          "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "threads": threads,
          "config": {"workload": "BASELINE config 3 on the host: PPO self-play, cnn policy-value net, sequential trainer; " + r["sample"],
                     "rollout_samples_per_s": r["rollout_samples_per_s"], "update_samples_per_s": r["update_samples_per_s"]},
          "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": threads, "kind": "port", "sample": r["sample"]},
          "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0})
    return 0


def run_product(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from shogidrl_b200 import VecShogiEnv, MASK_PAD_STRIDE

    n = args.envs
    env = VecShogiEnv(n, MAX_MOVES, dev, seed=SEED, env_offset=rank * n, auto_reset=True, step_streams=args.step_streams)
    # rollout storage the kernel writes straight into: 2 slots of [n] obs / masks (1.86 GB per slot >> 126 MB L2)
    SLOTS = 2
    obs_buf = torch.zeros((SLOTS, n, 46, 9, 9), dtype=torch.float32, device=dev)
    mask_buf = torch.zeros((SLOTS, n, MASK_PAD_STRIDE), dtype=torch.uint8, device=dev)
    act = [torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    it = [0]

    def step():
        # actions were chosen by the fused uniform-random legal policy of the previous launch (ping-pong buffers)
        i = it[0]
        it[0] += 1
        env.step(act[i & 1], obs=obs_buf[i % SLOTS], mask=mask_buf[i % SLOTS][:, :13527], random_actions=True,
                 next_out=act[(i + 1) & 1])

    env.refresh(random_actions=True, next_out=act[0])
    for i in range(args.preroll):
        step()
    for i in range(args.warmup):
        step()
    barrier()

    # mean ply of the positions the timed steps start from (for the algorithmic-bytes figure)
    ply0 = float(env.export()[2][:, 1].float().mean())
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev0.record()
    for i in range(args.steps):
        kev[i][0].record()
        step()
        kev[i][1].record()
    ev1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev0.elapsed_time(ev1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    ply1 = float(env.export()[2][:, 1].float().mean())
    errs = int((env.errors() != 0).sum())
    if args.dump_outputs and rank == 0:
        last = it[0] - 1  # the last timed step wrote these slots and the next actions it chose
        dump_step_outputs(args.dump_outputs, env, obs_buf[last % SLOTS], mask_buf[last % SLOTS][:, :13527], act[it[0] & 1])

    # ---- end-to-end through the public API with HOST buffers: per step the actions come from pinned host
    # memory (H2D) and the step's results + the next legal actions are read back to pinned host memory (D2H).
    # (a) serial: one batch, copy -> kernel -> copy -> synchronise, latencies add up;
    # (b) HostPipelinedEnv: the same games in two groups on two streams, the host serves one group while the other
    #     group's kernel runs.  (b) is the e2e figure; (a) is reported next to it.
    h_act = torch.zeros(n, dtype=torch.int64).pin_memory()
    h_res = torch.zeros(n * 15, dtype=torch.uint8).pin_memory()
    h_act.copy_(act[it[0] & 1])
    torch.cuda.synchronize(dev)
    e2e_steps = max(4, min(args.steps, 64))

    def e2e_step(i):
        a = act[i & 1]
        a.copy_(h_act, non_blocking=True)                                  # H2D 8 B/env
        env.step(a, obs=obs_buf[i % SLOTS], mask=mask_buf[i % SLOTS][:, :13527], random_actions=True,
                 next_out=env.next_actions)
        h_res.copy_(env.results, non_blocking=True)                        # D2H 15 B/env: next action, reward, done, reason, winner
        torch.cuda.current_stream(dev).synchronize()
        h_act.copy_(h_res[: 8 * n].view(torch.int64))                      # host-side hand-over of the chosen actions

    for i in range(3):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    barrier()
    serial_ms = 1e3 * (time.perf_counter() - t0)

    # (c) every output on the host: as (a), plus the step's 46x9x9 observations and 13,527-byte legal masks copied to
    #     pinned host memory -- what a caller that keeps the policy tower off the GPU would pay (PCIe-bound).
    h_obs = torch.empty((n, 46, 9, 9), dtype=torch.float32).pin_memory()
    h_mask = torch.empty((n, MASK_PAD_STRIDE), dtype=torch.uint8).pin_memory()
    full_steps = 4

    def full_step(i):
        a = act[i & 1]
        a.copy_(h_act, non_blocking=True)
        env.step(a, obs=obs_buf[i % SLOTS], mask=mask_buf[i % SLOTS][:, :13527], random_actions=True,
                 next_out=env.next_actions)
        h_res.copy_(env.results, non_blocking=True)
        h_obs.copy_(obs_buf[i % SLOTS], non_blocking=True)
        h_mask.copy_(mask_buf[i % SLOTS], non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        h_act.copy_(h_res[: 8 * n].view(torch.int64))

    full_step(0)
    barrier()
    t0 = time.perf_counter()
    for i in range(full_steps):
        full_step(i)
    barrier()
    full_ms = 1e3 * (time.perf_counter() - t0)
    full_d2h = 15 * n + h_obs.numel() * 4 + h_mask.numel()
    del h_obs, h_mask

    from shogidrl_b200.host_env import HostPipelinedEnv
    G = 2
    del env
    pipe = HostPipelinedEnv(n, groups=G, max_moves_per_game=MAX_MOVES, device=dev, seed=SEED, env_offset=rank * n)
    ng = n // G

    def views(i, g):
        return obs_buf[i % SLOTS][g * ng:(g + 1) * ng], mask_buf[i % SLOTS][g * ng:(g + 1) * ng, :13527]

    pipe.prime(random_actions=True)
    for i in range(args.preroll + args.warmup):                            # the same pre-roll as the device-timed leg: steady-state mix
        for g in range(G):
            pipe.h_actions[g].copy_(pipe.wait(g)[0])
            pipe.submit(g, *views(i, g), random_actions=True)
    pipe.synchronize()
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        for g in range(G):
            pipe.h_actions[g].copy_(pipe.wait(g)[0])                       # host hand-over of the chosen actions
            pipe.submit(g, *views(i, g), random_actions=True)              # H2D 8 B/env, kernel, D2H 15 B/env
    for g in range(G):
        pipe.wait(g)
    pipe.synchronize()
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    errs += sum(int((e.errors() != 0).sum()) for e in pipe.envs)
    e2e_mean_ply = float(torch.cat([e.export()[2][:, 1].float() for e in pipe.envs]).mean())
    del pipe, obs_buf, mask_buf
    torch.cuda.empty_cache()
    ppo = None
    if not args.no_ppo:
        ppo = measure_ppo(args, dev, world, rank, barrier)

    if world > 1:
        t = torch.tensor([ms_total, e2e_ms, kernel_ms, serial_ms, full_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_ms, kernel_ms, serial_ms, full_ms = [float(x) for x in t]
        e = torch.tensor([errs], device=dev)
        dist.all_reduce(e)
        errs = int(e)

    if rank == 0:
        mean_ply = 0.5 * (ply0 + ply1)
        bytes_per_launch = algorithmic_bytes_per_step(mean_ply) * n
        achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
        peak, peak_src = measured_peak_gbs()
        traffic, traffic_src = None, None
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel (profiles/)
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
                if int(tj.get("envs", 0)) == n:
                    traffic = tj["dram_bytes_per_launch"]
                    traffic_src = f"profiles/traffic.json: {tj.get('source', 'ncu --set full')} (kernel sources {tj.get('src_sha', '?')})"
        except Exception:
            pass
        from shogidrl_b200 import _native as nv
        build = nv.build_info()
        line = {
            "metric": METRIC, "value": world * n * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"BASELINE config 2: batched random-legal self-play, {n} games per GPU, legal mask + obs + "
                                   f"step, no network; max_moves {MAX_MOVES}, auto-reset, actions = fused uniform-random legal "
                                   f"(counter RNG seed {SEED})",
                       "envs_per_gpu": n, "parallelism": f"env-shard x{world} (no data-path collective)",
                       "preroll_steps": args.preroll, "mean_ply": mean_ply,
                       "l2": "each step writes 1.86 GB of fresh obs+mask rows per GPU (2-slot ring), far above the 126 MB L2",
                       "algorithmic_bytes_per_env_step": algorithmic_bytes_per_step(mean_ply), "env_error_flags": errs},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "kz_step_kernel", "kernel_ms": kernel_ms,
                         "peak_source": peak_src,
                         "achieved_implementation_bytes": implementation_bytes_per_step() * n / (kernel_ms * 1e-3) / 1e9,
                         "frac_implementation_bytes": implementation_bytes_per_step() * n / (kernel_ms * 1e-3) / 1e9 / peak},
            "e2e": {"value": world * n * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * n,
                    "d2h_bytes_per_step": 15 * n, "steps": e2e_steps, "preroll_steps": args.preroll, "mean_ply": e2e_mean_ply,
                    "serial_value": world * n * e2e_steps / (serial_ms * 1e-3),
                    "note": "HostPipelinedEnv (2 groups, 2 streams), same pre-roll and position mix as `value`: actions from "
                            "pinned host memory, reward/done/reason/winner/next-action read back to pinned host memory every "
                            "step, host waits for each group's results before submitting its next actions; obs/mask stay in "
                            "HBM for the policy tower; it can exceed `value` because the two groups run ahead of each other "
                            "(one group's CTAs fill the SMs the other's draining grid leaves idle); serial_value = the same "
                            "through one VecShogiEnv with copy -> kernel -> copy -> synchronise in sequence"},
            # what a caller of the reference's scalar API (observation + mask as host arrays) would see: PCIe-bound
            "e2e_host_outputs": {"value": world * n * full_steps / (full_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 8 * n,
                                 "d2h_bytes_per_step": full_d2h, "steps": full_steps,
                                 "note": "the serial path when the 46x9x9 observations and 13,527-byte legal masks are ALSO "
                                         "copied to pinned host memory every step (1.86 GB per 65,536 games); only a caller "
                                         "that keeps its policy network off the GPU needs that"},
            "build": build,
            "gpu_launches": args.steps,
            "clocks": clocks,
        }
        if ppo is not None:
            line["ppo"] = ppo
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            line["cpu_baseline"] = cpu_baseline_sample(threads)
            ref = real_reference_sample(threads)  # the unmodified Python reference, when baseline/_ref travelled here
            if ref is not None:
                line["cpu_baseline_reference"] = ref
            if ppo is not None:
                rp = real_reference_ppo_sample(threads, epochs=args.ppo_epochs)
                if rp is not None:
                    ppo["cpu_baseline_reference"] = rp
        emit(line)
    finish_process_group(world)
    return 0


DUMP_OBS_ROWS = 512  # games whose observation + legal-mask rows --dump-outputs writes: 512 x 69 KB = 35 MB as float32
DUMP_GAME_ROWS = 1 << 19  # games whose per-game results it writes: at most 7 x 2 MB


def _dump_rows(n: int, k: int):
    """All n games, or a fixed seeded sample of k of them in ascending order."""
    import numpy as np
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(SEED).choice(n, k, replace=False))


def dump_step_outputs(out_dir: str, env, obs, mask, next_actions):
    """--dump-outputs: what one VecShogiEnv.step returned to its caller, as float32 .npy files under out_dir (every
    value is a small integer or an fp32 number, so float32 holds it exactly).  obs / legal_mask hold the rows of
    obs_rows (a seeded sample when there are more than DUMP_OBS_ROWS games); the per-game results those of game_rows."""
    import numpy as np
    import torch
    n = env.n
    obs_rows, game_rows = _dump_rows(n, DUMP_OBS_ROWS), _dump_rows(n, DUMP_GAME_ROWS)
    oi, gi = torch.from_numpy(obs_rows).to(obs.device), torch.from_numpy(game_rows).to(obs.device)
    arrays = {"obs": obs.index_select(0, oi), "legal_mask": mask.index_select(0, oi),
              "next_action": next_actions[:n], "reward": env.reward, "done": env.done, "reason": env.reason,
              "winner": env.winner, "ep_len": env.ep_len, "legal_count": env.legal_count}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if name not in ("obs", "legal_mask"):
            t = t.index_select(0, gi)
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    np.save(os.path.join(out_dir, "obs_rows.npy"), obs_rows.astype(np.float64))
    np.save(os.path.join(out_dir, "game_rows.npy"), game_rows.astype(np.float64))


def cfg5_positions(n: int):
    """BASELINE config 5's start mix for n games: [hirate | drops-heavy endgames | 4-ply-cycle scripts], a third each.  The
    endgames are the fixed list of 128 reference-validated SFENs in tests/golden/traces_endgame.npz (two kings, a few
    pieces, full hands), tiled; the cycle script is the reference test-suite's sennichite position
    (tests/shogi/test_shogi_game_core_logic.py:1126-1179).  -> boards, hands, sides, move_counts, (n_hirate, n_endgame, n_cycle)"""
    import numpy as np
    from shogidrl_b200.shogi.sfen import pack_sfen
    n_e = n_c = n // 3
    n_h = n - n_e - n_c
    with np.load(os.path.join(ROOT, "tests", "golden", "traces_endgame.npz")) as z:
        eg = [pack_sfen(str(x)) for x in z["sfens"]]
    hirate = pack_sfen("lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1")
    cyc = pack_sfen("4k4/9/9/9/9/R8/9/9/4K4 b - 1")
    idx = np.arange(n_e) % len(eg)
    boards = np.concatenate([np.tile(hirate[0], (n_h, 1)), np.stack([p[0] for p in eg])[idx], np.tile(cyc[0], (n_c, 1))])
    hands = np.concatenate([np.tile(hirate[1], (n_h, 1)), np.stack([p[1] for p in eg])[idx], np.tile(cyc[1], (n_c, 1))])
    sides = np.concatenate([np.zeros(n_h, np.uint8), np.asarray([p[2] for p in eg], np.uint8)[idx], np.zeros(n_c, np.uint8)])
    return boards.astype(np.int8), hands.astype(np.uint8), sides, np.zeros(n, np.int32), (n_h, n_e, n_c)


CYCLE_MOVES = [(5, 0, 5, 1, False), (0, 4, 0, 3, False), (5, 1, 5, 0, False), (0, 3, 0, 4, False)]


def run_cfg5(args):
    """--workload cfg5: BASELINE config 5, the long-game stress -- `--envs` games per GPU (262,144), max_moves 500 with
    500-ply repetition tables, start mix of cfg5_positions; the scripted third plays the 4-ply rook / king cycle and must
    end by sennichite on ply 13; every finished game restarts from hirate.  One step = kz_step over the whole batch (legal
    mask + obs + step, as config 2).  Reports steps/s over K timed steps after the pre-roll, the termination-reason
    histogram of every game finished since the start, and the history memory.  (The histogram is checked against the
    oracle on 4,096 sampled games of the same full-size batch by tests/test_gpu_engine.py::test_config5_full_size.)"""
    import numpy as np
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from shogidrl_b200 import VecShogiEnv, MASK_PAD_STRIDE
    from shogidrl_b200.utils import move_to_index

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    n = args.envs
    boards, hands, sides, mcs, (n_h, n_e, n_c) = cfg5_positions(n)
    env = VecShogiEnv(n, MAX_MOVES, dev, seed=SEED, env_offset=rank * n, auto_reset=True)
    env.load_positions(boards, hands, sides, mcs, eval_termination=False)
    env.step_index = 0
    SLOTS = 2
    obs_buf = torch.zeros((SLOTS, n, 46, 9, 9), dtype=torch.float32, device=dev)
    mask_buf = torch.zeros((SLOTS, n, MASK_PAD_STRIDE), dtype=torch.uint8, device=dev)
    act = [torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)]
    env.refresh(random_actions=True, next_out=act[0])
    cycle = [move_to_index(m) for m in CYCLE_MOVES]
    hist = torch.zeros(5, dtype=torch.int64, device=dev)
    senn13 = torch.zeros((), dtype=torch.int64, device=dev)
    it = [0]

    def step():
        i = it[0]
        it[0] += 1
        a = act[i & 1]
        if i < 13:
            a[n_h + n_e:] = cycle[i % 4]  # the scripted third
        out = env.step(a, obs=obs_buf[i % SLOTS], mask=mask_buf[i % SLOTS][:, :13527], random_actions=True,
                       next_out=act[(i + 1) & 1])
        return out

    for i in range(args.preroll + args.warmup):
        out = step()
        hist += torch.bincount(out["reason"].long(), minlength=5)
        if i == 12:
            senn13 += (out["reason"][n_h + n_e:] == 4).sum()
    barrier()
    ply0 = float(env.export()[2][:, 1].float().mean())
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        step()
    ev1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev0.elapsed_time(ev1)
    ply1 = float(env.export()[2][:, 1].float().mean())
    errs = int((env.errors() != 0).sum())
    stats = torch.cat([hist, senn13.reshape(1), torch.tensor([errs], device=dev)])
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t)
        dist.all_reduce(stats)
    if rank == 0:
        import ctypes as C
        from shogidrl_b200 import _native as nv
        offs, total = (C.c_int64 * 3)(), C.c_int64()
        nv.lib().kz_state_layout(n, MAX_MOVES, offs, C.byref(total))
        mean_ply = 0.5 * (ply0 + ply1)
        peak, peak_src = measured_peak_gbs()
        achieved = algorithmic_bytes_per_step(mean_ply) * n / (ms_total / args.steps * 1e-3) / 1e9
        h = stats.tolist()
        emit({"metric": METRIC, "value": world * n * args.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world,
              "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
              "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
              "config": {"workload": f"BASELINE config 5: long-game stress, {n} games per GPU x {world}, max_moves {MAX_MOVES}, "
                                     f"start mix {n_h} hirate / {n_e} drops-heavy endgames (128 fixed SFENs) / {n_c} 4-ply-cycle "
                                     f"scripts per GPU, auto-reset to hirate, legal mask + obs + step, random-legal play",
                         "envs_per_gpu": n, "preroll_steps": args.preroll + args.warmup, "mean_ply": mean_ply,
                         "state_bytes_per_gpu": int(total.value), "history_bytes_per_gpu": int(total.value - offs[2]),
                         "output_ring_bytes_per_gpu": int(obs_buf.numel() * 4 + mask_buf.numel()),
                         "finished_games_by_reason": {"Tsumi": h[1], "stalemate": h[2], "Max moves reached": h[3], "Sennichite": h[4]},
                         "scripted_cycles_ended_by_sennichite_on_ply_13": f"{h[5]} of {n_c * world}",
                         "env_error_flags": h[6]},
              "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                           "traffic": None, "kernel": "kz_step_kernel", "kernel_ms": ms_total / args.steps, "peak_source": peak_src},
              "gpu_launches": args.steps, "clocks": clocks})
    finish_process_group(world)
    return 0


_JSON_OUT = None


def isolate_stdout():
    """Libraries write to fd 1 (NCCL prints its version line there): keep the real stdout for the one JSON line
    and send everything else to stderr."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# SURVEY.md section 8(d): algorithmic bytes per rollout sample (configs 3/4) = B_env + the tower's re-read of the observation
# + logits written and read once (bf16) + the sampler's read of the mask row + action / log-prob / value writes
def rollout_bytes_per_sample(mean_ply: float) -> float:
    return algorithmic_bytes_per_step(mean_ply) + OBS_B + 2 * 13527 * 2 + MASK_B + 16


def tower_mfu(model_kind: str, samples_per_gpu_epoch: int, ppo_epochs: int, epoch_ms: float):
    """Dense-contraction throughput of the policy/value tower (the only tensor-core work on the path): forward FLOPs per
    sample measured by SURVEY section 8(d) (ActorCritic 36.1 MFLOP, ResTower 9x256 SE 1.74 GFLOP); a PPO sample costs one
    rollout forward + ppo_epochs x (forward + backward = 3 forwards).  Against the measured sustained bf16 rate."""
    fwd = 1.74e9 if model_kind == "resnet" else 36.1e6
    flop = samples_per_gpu_epoch * fwd * (1 + 3 * ppo_epochs)
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["bf16_tflops_sustained"])
        src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        peak, src = 1400.0, "fallback"
    tf = flop / (epoch_ms * 1e-3) / 1e12
    return {"fwd_flop_per_sample": fwd, "fwd_equivalents_per_sample": 1 + 3 * ppo_epochs, "achieved_tflops_per_gpu": tf,
            "peak_tflops": peak, "mfu": tf / peak, "peak_source": src}


def measure_ppo(args, dev, world, rank, barrier):
    """BASELINE config 3 (or 4 with --ppo-model resnet): PPO self-play with the policy-value net under bf16 autocast,
    `--ppo-envs` games per GPU, rollout T = `--ppo-horizon` (tower forward, fused masked sampling on the engine's legal
    bitmaps, engine step writing observations / bitmaps / rewards straight into the rollout buffer, device GAE), then the
    PPO update (ppo_epochs x minibatches, fused masked evaluation, loss, clip + Adam, replayed from a CUDA graph).  One
    step = one epoch (collect + update).  Returns the `ppo` record (rank 0) or None."""
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace
    from shogidrl_b200 import rl
    from shogidrl_b200.core import ActorCritic, ActorCriticResTower
    from shogidrl_b200.training.selfplay import SelfPlayTrainer

    N, T, mb = args.ppo_envs, args.ppo_horizon, args.ppo_minibatch
    cfg = SimpleNamespace(
        env=SimpleNamespace(device=str(dev), seed=SEED, input_channels=46, num_actions_total=13527, max_moves_per_game=MAX_MOVES),
        training=SimpleNamespace(learning_rate=3e-4, gamma=0.99, lambda_gae=0.95, clip_epsilon=0.2, value_loss_coeff=0.5,
                                 entropy_coef=0.01, ppo_epochs=args.ppo_epochs, minibatch_size=mb, steps_per_epoch=N * T,
                                 total_timesteps=N * T * 8, gradient_clip_max_norm=0.5, normalize_advantages=True,
                                 enable_value_clipping=False, weight_decay=0.0, lr_schedule_type=None,
                                 lr_schedule_step_on="epoch", lr_schedule_kwargs=None,
                                 cuda_graph_rollout=not args.no_graph_rollout),
        display=SimpleNamespace(display_moves=False, turn_tick=0.0))
    torch.manual_seed(SEED + rank)
    if args.ppo_model == "resnet":
        model = ActorCriticResTower(46, 13527, tower_depth=9, tower_width=256, se_ratio=0.25)
    else:
        model = ActorCritic(46, 13527)
    tr = SelfPlayTrainer(model, cfg, N, T, dev, use_mixed_precision=True)
    warm = max(1 if args.no_graph_rollout else 2, args.ppo_warmup)  # epoch 1 captures the update graph, epoch 2 the rollout graph
    for _ in range(warm):
        tr.run_epoch()
    barrier()
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    steps = args.ppo_steps
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    roll_ms = upd_ms = 0.0
    m = {}
    t0 = time.perf_counter()
    for _ in range(steps):
        ev[0].record(); tr.collect(); ev[1].record(); m = tr.update(); ev[2].record()
        torch.cuda.synchronize(dev)
        roll_ms += ev[0].elapsed_time(ev[1]); upd_ms += ev[1].elapsed_time(ev[2])
    barrier()
    total_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    mean_ply = float(tr.env.export()[2][:, 1].float().mean())

    # ---- the hand-written kernels of the path, timed live on this run's data (CUDA events, current stream)
    b = tr.buffer
    kern = {}

    def timed(fn, reps=20):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps

    peak, peak_src = measured_peak_gbs()
    rows = min(mb, N)
    logits = torch.randn((rows, 13536), device=dev).bfloat16()[:, :13527]
    legal = float(tr.env.legal_count.float().mean())  # legal actions per position (~50 under a near-uniform policy)
    bm = b.bitmaps[1][:rows]
    acts = b.actions[1][:rows].contiguous()
    sectors = legal * 32.0  # one 32-byte sector per legal logit
    ms = timed(lambda: rl.sample_masked(logits, bm, seed=1, offset=0))
    kern["kz_sample_bitmap"] = {"ms": ms, "rows": rows, "survey_bytes_per_row": 13527 * 2 + 13527,
                                "implementation_bytes_per_row": 1792 + sectors + 12}
    lg = logits.detach().clone().requires_grad_(True)
    lp, en = rl.evaluate_masked(lg, bm, acts)
    ms = timed(lambda: rl.evaluate_masked(lg, bm, acts))
    kern["kz_eval_bitmap_fwd"] = {"ms": ms, "rows": rows, "survey_bytes_per_row": 13527 * 2 + 13527,
                                  "implementation_bytes_per_row": 1792 + 2 * sectors + 24}
    g1, g2 = torch.ones_like(lp), torch.ones_like(en)
    ms_fb = timed(lambda: torch.autograd.grad((lp, en), lg, (g1, g2), retain_graph=True))
    kern["kz_eval_bitmap_bwd"] = {"ms": ms_fb, "rows": rows, "survey_bytes_per_row": 13527 * 2 + 13527 + 13527 * 2,
                                  "implementation_bytes_per_row": 1792 + sectors + 13536 * 2 + 16,
                                  "note": "includes the dense dlogits row (27 KB) the two gradient GEMMs read"}
    for k in kern.values():
        t = k["ms"] * 1e-3
        k["achieved_gbs"] = k["survey_bytes_per_row"] * k["rows"] / t / 1e9
        k["achieved_implementation_gbs"] = k["implementation_bytes_per_row"] * k["rows"] / t / 1e9
        k["frac_implementation_bytes"] = k["achieved_implementation_gbs"] / peak
    del lg, lp, en, logits

    if world > 1:
        t = torch.tensor([total_ms, roll_ms, upd_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, roll_ms, upd_ms = [float(x) for x in t]
    rec = None
    if rank == 0:
        samples = world * N * T * steps
        n_upd = -(-N * T // mb) * args.ppo_epochs
        cnn = args.ppo_model == "cnn"
        rb = rollout_bytes_per_sample(mean_ply)
        rec = {"metric": "PPO self-play samples/sec", "value": samples / (total_ms * 1e-3), "unit": "samples/s",
               "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": total_ms / steps,
               "higher_is_better": True, "scaling": "weak", "dtype": "bf16", "data": "synthetic",
               "config": {"workload": f"BASELINE config {3 if cnn else 4}: PPO self-play, {args.ppo_model} policy-value net "
                                      f"(bf16 autocast), {N} envs/GPU, T={T}, fused masked sampling on legal bitmaps + device "
                                      f"GAE, ppo_epochs={args.ppo_epochs}, minibatch={mb} ({n_upd} updates per epoch)"
                                      + (", eager rollout loop" if args.no_graph_rollout else ", rollout replayed from a CUDA graph"),
                          "envs_per_gpu": N, "horizon": T, "minibatch": mb, "ppo_epochs": args.ppo_epochs,
                          "parallelism": f"env-shard x{world}, gradient all-reduce over NCCL in the update" if world > 1 else "1 GPU",
                          "rollout_storage_gb": (b.obs.numel() * 4 + b.bitmaps.numel() * 4) / 1e9},
               "rollout_samples_per_s": samples / (roll_ms * 1e-3), "update_samples_per_s": samples / (upd_ms * 1e-3),
               "rollout_ms": roll_ms / steps, "update_ms": upd_ms / steps,
               "rollout_step_ms": roll_ms / steps / T, "update_minibatch_ms": upd_ms / steps / n_upd,
               "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak, "peak_source": peak_src,
                            "rollout": {"bytes_per_sample": rb, "achieved": rb * N * T / (roll_ms / steps * 1e-3) / 1e9,
                                        "frac": rb * N * T / (roll_ms / steps * 1e-3) / 1e9 / peak,
                                        "note": "SURVEY section 8(d) bytes per rollout sample over the whole rollout step "
                                                "(tower GEMM included, which is tensor-bound, not HBM-bound)"},
                            "kernels": kern},
               "tower": tower_mfu(args.ppo_model, N * T, args.ppo_epochs, total_ms / steps),
               "last_metrics": {k: float(v) for k, v in m.items()},
               "clocks": clocks,
               # own kernels per epoch: rollout steps (kz_step, kz_sample_bitmap, + kz_obs_conv_fwd for the CNN), kz_gae, and per
               # minibatch update kz_eval_bitmap_fwd/bwd, kz_ppo_loss, 3 x kz_adam_clip (+ kz_obs_conv_fwd and 2 wgrad kernels)
               "gpu_launches": steps * (T * (3 if cnn else 2) + 1 + n_upd * (9 if cnn else 6))}
    if world > 1:
        # the captured update graph holds NCCL work: release it before the process group goes away
        import gc
        barrier()
        tr.agent._drop_graph()
        gc.collect()
        torch.cuda.synchronize(dev)
    del tr
    return rec


def run_ppo(args):
    """--workload ppo: the PPO record as its own JSON line (the default env workload carries it as line["ppo"])."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    args.ppo_steps = args.steps if args.steps <= 16 else 2
    rec = measure_ppo(args, dev, world, rank, barrier)
    if rank == 0:
        rec["vs_baseline"] = None
        emit(rec)
    finish_process_group(world)
    return 0


def finish_process_group(world):
    """Never let a stuck communicator teardown outlive the measurement."""
    if world > 1:
        import threading
        import torch.distributed as dist
        killer = threading.Timer(30.0, lambda: os._exit(0))
        killer.daemon = True
        killer.start()
        dist.destroy_process_group()
        killer.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--warmup", type=int, default=16)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="games per GPU (BASELINE config 2: 65,536)")
    ap.add_argument("--preroll", type=int, default=PREROLL)
    ap.add_argument("--step-streams", type=int, default=None,
                    help="ranges of games a step is launched as, on as many streams (kz_step_range; default 1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="env", choices=["env", "ppo", "cfg5"],
                    help="env: BASELINE config 2 (default, the headline; carries the config-3 PPO record); ppo: config 3 (or 4 with "
                         "--ppo-model resnet --ppo-envs 32768) as its own line; cfg5: the long-game stress (--envs 262144)")
    ap.add_argument("--ppo-envs", type=int, default=16384)
    ap.add_argument("--ppo-horizon", type=int, default=128)
    ap.add_argument("--ppo-epochs", type=int, default=10)
    ap.add_argument("--ppo-minibatch", type=int, default=16384)
    ap.add_argument("--ppo-model", default="cnn", choices=["cnn", "resnet"])
    ap.add_argument("--ref-ppo-steps", type=int, default=512, help="timesteps per epoch of the CPU PPO reference arm")
    ap.add_argument("--ref-same-minibatch", action="store_true", help="--impl reference --workload ppo: minibatch = min(--ppo-minibatch, steps) instead of the reference's 64")
    ap.add_argument("--no-ppo", action="store_true", help="skip the PPO (config 3) record of the default workload")
    ap.add_argument("--no-graph-rollout", action="store_true", help="run the rollout loop eagerly (one warm-up epoch suffices then)")
    ap.add_argument("--ppo-steps", type=int, default=2, help="timed PPO epochs of the `ppo` record")
    ap.add_argument("--ppo-warmup", type=int, default=2, help="untimed PPO epochs (the first captures the update graph, the second the rollout graph)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (observations, legal masks, rewards, done "
                         "flags, next actions, ...) as float32 DIR/<name>.npy, at most 64 MB (default env workload only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "product" or args.workload != "env"):
        ap.error("--dump-outputs applies to the default workload (--impl product --workload env)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference_ppo(args) if args.workload == "ppo" else run_reference(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    isolate_stdout()
    if args.workload == "ppo":
        return run_ppo(args)
    if args.workload == "cfg5":
        if args.envs == ENVS_PER_GPU:
            args.envs = 262144
        return run_cfg5(args)
    return run_product(args)


if __name__ == "__main__":
    sys.exit(main())
