"""GPU parity tests of the engine kernels (kz_step / kz_refresh) through the C ABI.

Checked against (a) golden traces produced by the Python reference itself (tests/golden/) and
(b) the C oracle (oracle/) on the same seeded inputs.  Bit-exact: legal sets, masks, successor
boards / hands / side / move_count, rewards, dones, reasons, winners, observation tensors."""
import hashlib
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests.helpers import random_endgames as _random_endgames  # noqa: E402


def _digest(obs_row: np.ndarray) -> int:
    return int.from_bytes(hashlib.blake2b(np.ascontiguousarray(obs_row, np.float32).tobytes(), digest_size=8).digest(), "little")


def _fmt_pos(board, hands, side):
    sym = "PLNSGBRK"
    rows = []
    for r in range(9):
        row = []
        for c in range(9):
            code = int(board[r * 9 + c])
            if code == 0:
                row.append(" . ")
            else:
                t, col = (code - 1) % 14, (code - 1) // 14
                s = ("+" + sym[{8: 0, 9: 1, 10: 2, 11: 3, 12: 5, 13: 6}[t]]) if t >= 8 else (" " + sym[t])
                row.append((s.lower() if col else s) + " ")
        rows.append("".join(row))
    return "\n".join(rows) + f"\nhands B={list(hands[:7])} W={list(hands[7:])} side={side}"


def _explain(board, hands, side, got_idx, want_idx):
    got, want = set(int(x) for x in got_idx), set(int(x) for x in want_idx)
    return (f"\n{_fmt_pos(board, hands, side)}\nGPU-only: {[orc.index_to_move(i) for i in sorted(got - want)]}"
            f"\nreference-only: {[orc.index_to_move(i) for i in sorted(want - got)]}")


@pytest.fixture(scope="module")
def traces(golden_dir):
    with np.load(os.path.join(golden_dir, "traces_random.npz")) as z:
        return {k: z[k] for k in z.files}


def _replay_group(z, games, dev):
    """Replay the golden games `games` (same T and max_moves) in one device batch, auto_reset off."""
    from shogidrl_b200 import VecShogiEnv

    n = len(games)
    T, mm = int(z["T"][games[0]]), int(z["max_moves"][games[0]])
    starts = np.concatenate([[0], np.cumsum(z["T"])])[:-1]
    env = VecShogiEnv(n, max_moves_per_game=mm, device=dev, auto_reset=False)
    for t in range(T):
        ix = [int(starts[g]) + t for g in games]
        mask = env.mask.cpu().numpy()
        b, h, m = [x.cpu().numpy() for x in env.export()]
        for e, i in enumerate(ix):
            want = z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]].astype(np.int64)
            got = np.nonzero(mask[e])[0]
            assert np.array_equal(got, want), (games[e], t, _explain(b[e], h[e], m[e, 0], got, want))
            assert int(env.legal_count[e]) == len(want)
        acts = torch.as_tensor(z["actions"][ix].astype(np.int64), device=dev)
        out = env.step(acts)
        torch.cuda.synchronize()
        assert int(env.errors().abs().sum()) == 0
        b, h, m = [x.cpu().numpy() for x in env.export()]
        obs = out["obs"].cpu().numpy()
        assert np.array_equal(b, z["boards"][ix]), (t,)
        assert np.array_equal(h, z["hands"][ix]), (t,)
        assert np.array_equal(m[:, 0], z["sides"][ix]) and np.array_equal(m[:, 1], z["move_counts"][ix]), (t,)
        assert np.array_equal(out["reward"].cpu().numpy(), z["rewards"][ix]), (t,)
        assert np.array_equal(out["done"].cpu().numpy(), z["dones"][ix]), (t, out["reason"].cpu().numpy(), z["reasons"][ix])
        assert np.array_equal(out["reason"].cpu().numpy(), z["reasons"][ix]), (t,)
        assert np.array_equal(out["winner"].cpu().numpy(), z["winners"][ix]), (t,)
        for e, i in enumerate(ix):
            assert _digest(obs[e]) == int(z["digests"][i]), (games[e], t)
        d = out["done"].bool()
        if bool(d.any()):
            env.reset(env_mask=d)  # what StepManager.handle_episode_end does (step_manager.py:437-440)
    return n * T


def test_golden_traces_replay(traces):
    """Every ply of the Python reference's own random-play games, replayed on the GPU."""
    dev = torch.device("cuda:0")
    z = traces
    total = 0
    groups = {}
    for g in range(len(z["env"])):
        groups.setdefault((int(z["T"][g]), int(z["max_moves"][g])), []).append(g)
    for games in groups.values():
        total += _replay_group(z, games, dev)
    assert total == len(z["actions"])


def test_golden_endgame_traces_replay(golden_dir):
    """Drop-heavy endgames played by the Python reference (oracle/gen_golden_endgame.py), replayed on the GPU in one
    batch loaded from the fixture's SFENs: legal masks before every ply, successor boards / hands / side / move count,
    reward, done, reason, winner and the observation digest after it.  Games that ended early idle on a finished
    position (make_move then returns the terminal tuple again) and are no longer compared."""
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    plies = _replay_sfen_traces(z)
    assert plies == len(z["actions"]) and int((z["actions"] >= 12960).sum()) > 1000


def test_golden_stalemate(golden_dir):
    """Stalemate (no legal move, not in check) is a DRAW in the reference (shogi_game.py:431-435): reason 2, no winner,
    reward 0.  Fixture from the imported reference (oracle/gen_golden_stalemate.py): the reference test-suite's
    stalemate-at-load and stalemate-by-move positions, and 12 bare-king endgames whose random play ends in stalemate."""
    from shogidrl_b200 import VecShogiEnv

    with np.load(os.path.join(golden_dir, "traces_stalemate.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    dev = torch.device("cuda:0")
    env = VecShogiEnv(2, max_moves_per_game=500, device=dev, auto_reset=False)
    env.load_sfens([str(z["kat_load_sfen"]), str(z["kat_move_sfen"])])
    _, _, m = [x.cpu().numpy() for x in env.export()]
    assert (m[0, 3], m[0, 4]) == (2, -1) == (int(z["kat_load_reason"]), int(z["kat_load_winner"]))  # over at load: stalemate
    assert int(env.legal_count[0]) == 0 and int(env.mask[0].sum()) == 0
    assert np.array_equal(env.obs[0].cpu().numpy(), z["kat_load_obs"])
    assert m[1, 3] == 0 and np.array_equal(np.nonzero(env.mask[1].cpu().numpy())[0], z["kat_move_legal"].astype(np.int64))
    out = env.step(torch.as_tensor([0, int(z["kat_move_action"])], dtype=torch.int64, device=dev))
    assert (float(out["reward"][1]), int(out["done"][1]), int(out["reason"][1]), int(out["winner"][1])) == (0.0, 1, 2, -1)
    assert np.array_equal(out["obs"][1].cpu().numpy(), z["kat_move_obs"]) and int(out["legal_count"][1]) == 0
    # make_move on the game that was already over returns its terminal tuple again (shogi_game.py:589-593)
    assert (float(out["reward"][0]), int(out["done"][0]), int(out["reason"][0]), int(out["winner"][0])) == (0.0, 1, 2, -1)
    plies = _replay_sfen_traces(z)
    assert plies == len(z["actions"])
    ends = np.cumsum(z["T"]) - 1
    assert np.all(z["reasons"][ends] == 2) and np.all(z["winners"][ends] == -1) and np.all(z["rewards"][ends] == 0)
    # the same through auto-reset: the finished games restart from the initial position in the same launch
    n = len(z["sfens"])
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, auto_reset=True)
    env.load_sfens([str(s) for s in z["sfens"]])
    starts = np.concatenate([[0], np.cumsum(z["T"])])[:-1]
    env.refresh(random_actions=True)  # games whose trace has ended play on from the start position with random legal moves
    for t in range(int(z["T"].max())):
        live = np.nonzero(z["T"] > t)[0]
        acts = env.next_actions.clone()
        acts[torch.as_tensor(live, device=dev)] = torch.as_tensor(z["actions"][starts[live] + t].astype(np.int64), device=dev)
        out = env.step(acts, random_actions=True)
        last = live[z["T"][live] == t + 1]
        if len(last):
            li = torch.as_tensor(last, device=dev)
            assert bool((out["done"][li] == 1).all()) and bool((out["reason"][li] == 2).all())
            assert bool((out["winner"][li] == -1).all()) and bool((out["reward"][li] == 0).all())
            assert bool((out["legal_count"][li] == 30).all())  # reset to the start position


def _replay_sfen_traces(z):
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    n = len(z["sfens"])
    starts = np.concatenate([[0], np.cumsum(z["T"])])[:-1]
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, auto_reset=False)
    env.load_sfens([str(s) for s in z["sfens"]])
    b, h, _ = [x.cpu().numpy() for x in env.export()]
    assert np.array_equal(b, z["start_boards"]) and np.array_equal(h, z["start_hands"])
    plies = 0
    for t in range(int(z["T"].max())):
        live = np.nonzero(z["T"] > t)[0]
        ix = starts[live] + t
        mask = env.mask.cpu().numpy()
        b, h, m = [x.cpu().numpy() for x in env.export()]
        for e, i in zip(live, ix):
            want = z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]].astype(np.int64)
            got = np.nonzero(mask[e])[0]
            assert np.array_equal(got, want), (e, t, _explain(b[e], h[e], m[e, 0], got, want))
        acts = np.zeros(n, np.int64)
        acts[live] = z["actions"][ix]
        out = env.step(torch.as_tensor(acts, device=dev))
        b, h, m = [x.cpu().numpy() for x in env.export()]
        obs = out["obs"].cpu().numpy()
        assert np.array_equal(b[live], z["boards"][ix]) and np.array_equal(h[live], z["hands"][ix]), t
        assert np.array_equal(m[live, 0], z["sides"][ix]) and np.array_equal(m[live, 1], z["move_counts"][ix]), t
        assert np.array_equal(out["reward"].cpu().numpy()[live], z["rewards"][ix]), t
        assert np.array_equal(out["done"].cpu().numpy()[live], z["dones"][ix]), t
        assert np.array_equal(out["reason"].cpu().numpy()[live], z["reasons"][ix]), t
        assert np.array_equal(out["winner"].cpu().numpy()[live], z["winners"][ix]), t
        for e, i in zip(live, ix):
            assert _digest(obs[e]) == int(z["digests"][i]), (e, t)
        assert int(env.errors()[torch.as_tensor(live, device=dev)].abs().sum()) == 0
        plies += len(live)
    return plies


def test_golden_full_observations(traces):
    """Raw observation tensors (not only digests) at the sampled plies."""
    from shogidrl_b200 import VecShogiEnv

    z = traces
    dev = torch.device("cuda:0")
    idx = z["full_obs_idx"]
    starts = np.concatenate([[0], np.cumsum(z["T"])])
    game_of = np.searchsorted(starts, idx, side="right") - 1
    n = len(idx)
    mm = z["max_moves"][game_of]
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, auto_reset=False)
    env.load_positions(z["boards"][idx], z["hands"][idx], z["sides"][idx], z["move_counts"][idx], mm,
                       eval_termination=False)
    torch.cuda.synchronize()
    assert np.array_equal(env.obs.cpu().numpy(), z["full_obs"])


def test_kat_positions(golden_dir):
    """Known-answer SFEN positions of the reference's test-suite (+ pins, uchifuzume, oddities)."""
    from shogidrl_b200 import VecShogiEnv

    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    dev = torch.device("cuda:0")
    n = len(z["sfens"])
    parsed = [orc.parse_sfen(str(s)) for s in z["sfens"]]
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, auto_reset=False)
    env.load_positions(np.stack([p[0] for p in parsed]), np.stack([p[1] for p in parsed]),
                       np.asarray([p[2] for p in parsed]), np.asarray([p[3] for p in parsed]))
    torch.cuda.synchronize()
    b, h, m = [x.cpu().numpy() for x in env.export()]
    mask = env.mask.cpu().numpy()
    obs = env.obs.cpu().numpy()
    for i, sfen in enumerate(z["sfens"]):
        want = z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]].astype(np.int64)
        got = np.nonzero(mask[i])[0]
        assert np.array_equal(got, want), (str(sfen), _explain(b[i], h[i], m[i, 0], got, want))
        assert (m[i, 3] != 0) == bool(z["game_over"][i]), sfen
        assert m[i, 3] == z["reason"][i] and m[i, 4] == z["winner"][i], sfen
        assert np.array_equal(obs[i], z["obs"][i]), sfen


def test_scripted_sennichite(golden_dir):
    from shogidrl_b200 import VecShogiEnv

    with np.load(os.path.join(golden_dir, "scripted.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    dev = torch.device("cuda:0")
    env = VecShogiEnv(2, max_moves_per_game=500, device=dev, auto_reset=False)
    p = orc.parse_sfen(str(z["senn_sfen"]))
    start = orc.OracleGame().export()
    env.load_positions(np.stack([p[0], start[0]]), np.stack([p[1], start[1]]), np.asarray([p[2], 0]),
                       np.asarray([p[3], 0]))
    a0, a1 = z["senn_actions"], z["senn2_actions"]
    for t in range(max(len(a0), len(a1))):
        acts = torch.tensor([int(a0[min(t, len(a0) - 1)]), int(a1[min(t, len(a1) - 1)])], device=dev)
        out = env.step(acts)
        if t < len(a0):
            assert int(out["done"][0]) == int(z["senn_dones"][t]) and int(out["reason"][0]) == int(z["senn_reasons"][t]), t
        if t < len(a1):
            assert int(out["done"][1]) == int(z["senn2_dones"][t]) and int(out["reason"][1]) == int(z["senn2_reasons"][t]), t
    assert int(z["senn_reasons"][-1]) == 4 and len(a0) == 13


@pytest.mark.parametrize("n,T,max_moves", [(1024, 160, 500), (512, 120, 40), (1001, 48, 30), (3, 64, 20)])  # last two: ragged batches (not a multiple of the 8 games a CTA runs in lockstep)
def test_selfplay_vs_oracle(n, T, max_moves):
    """Device self-play with the fused uniform-random legal action and auto-reset, against the C oracle
    playing the same counter-based RNG: actions, rewards, dones, reasons, legal counts every step, and
    the final boards / hands / masks / observations."""
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    seed = 4321
    env = VecShogiEnv(n, max_moves_per_game=max_moves, device=dev, seed=seed, auto_reset=True)
    env.refresh(random_actions=True)
    acts, rews, dones, reasons, counts = [], [], [], [], []
    for t in range(T):
        a = env.next_actions.clone()
        counts.append(env.legal_count.clone())
        out = env.step(a, random_actions=True)
        acts.append(a); rews.append(out["reward"].clone()); dones.append(out["done"].clone())
        reasons.append(out["reason"].clone())
    torch.cuda.synchronize()
    assert int(env.errors().abs().sum()) == 0
    ref = orc.selfplay(n, T, max_moves=max_moves, seed=seed, threads=os.cpu_count() or 1)
    got_a = torch.stack(acts).cpu().numpy()
    bad = np.argwhere(got_a != ref["actions"])
    assert len(bad) == 0, ("first action mismatch (t, env):", bad[:5], got_a[tuple(bad[0])], ref["actions"][tuple(bad[0])])
    assert np.array_equal(torch.stack(counts).cpu().numpy(), ref["legal_counts"])
    assert np.array_equal(torch.stack(rews).cpu().numpy(), ref["rewards"])
    assert np.array_equal(torch.stack(dones).cpu().numpy(), ref["dones"])
    assert np.array_equal(torch.stack(reasons).cpu().numpy(), ref["reasons"])
    b, h, m = [x.cpu().numpy() for x in env.export()]
    assert np.array_equal(b, ref["boards"]) and np.array_equal(h, ref["hands"])
    assert np.array_equal(m[:, :2], ref["meta"][:, :2])
    assert np.array_equal(env.mask.cpu().numpy(), ref["mask"])
    assert np.array_equal(env.obs.cpu().numpy(), ref["obs"])
    assert ref["dones"].sum() > 0  # the run crossed episode boundaries


def test_mask_layouts_agree():
    """Vectorised (16-byte rows) and byte-granular (contiguous 13,527-byte rows) mask writers agree, as do
    observation rows at both 16-byte phases."""
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    env = VecShogiEnv(64, device=dev, seed=7)
    env.refresh(random_actions=True)
    for _ in range(40):
        env.step(env.next_actions.clone(), random_actions=True)
    contiguous = torch.zeros((64, 13527), dtype=torch.uint8, device=dev)
    obs2 = torch.zeros((64, 46, 9, 9), dtype=torch.float32, device=dev)
    env.refresh(obs=obs2, mask=contiguous)
    padded, obs1 = env.mask.clone(), env.obs.clone()
    env.refresh()
    assert torch.equal(contiguous, env.mask) and torch.equal(padded, env.mask)
    assert torch.equal(obs2, env.obs) and torch.equal(obs1, env.obs)
    assert torch.equal(env.mask.sum(1).int(), env.legal_count)


def test_illegal_actions_set_error_bits():
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    env = VecShogiEnv(4, device=dev, auto_reset=False)
    b0, h0, m0 = [x.clone() for x in env.export()]
    # out of range / empty source square / illegal pattern (pawn two squares) / drop without a piece in hand
    a = torch.tensor([20000, ((40 * 80 + 30) * 2), ((54 * 80 + 36) * 2), 12960 + 40 * 7], device=dev)
    out = env.step(a)
    err = env.errors().cpu().numpy()
    assert list(err) == [1, 1, 2, 1]
    b1, h1, m1 = env.export()
    assert torch.equal(b0, b1) and torch.equal(h0, h1) and torch.equal(m0[:, :5], m1[:, :5])
    assert int(out["done"].sum()) == 0 and float(out["reward"].abs().sum()) == 0.0


def test_selfplay_from_drop_heavy_endgames():
    """Step-mode parity from drop-heavy endgames: exercises the specialised uchifuzume test, drops that answer
    checks, promoted sliders, and auto-reset back to the start position."""
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    n, T, max_moves, seed = 2048, 70, 60, 97
    start = _random_endgames(n, 5)
    env = VecShogiEnv(n, max_moves_per_game=max_moves, device=dev, seed=seed, auto_reset=True)
    env.load_positions(*start, eval_termination=False)
    env.step_index = 0
    env.refresh(random_actions=True)
    acts, rews, reasons, counts = [], [], [], []
    for t in range(T):
        a = env.next_actions.clone()
        counts.append(env.legal_count.clone())
        out = env.step(a, random_actions=True)
        acts.append(a); rews.append(out["reward"].clone()); reasons.append(out["reason"].clone())
    torch.cuda.synchronize()
    assert int(env.errors().abs().sum()) == 0
    ref = orc.selfplay(n, T, max_moves=max_moves, seed=seed, threads=os.cpu_count() or 1, start=start)
    got_c = torch.stack(counts).cpu().numpy()
    bad = np.argwhere(got_c != ref["legal_counts"])
    assert len(bad) == 0, ("first legal-count mismatch (t, env):", bad[:5])
    assert np.array_equal(torch.stack(acts).cpu().numpy(), ref["actions"])
    assert np.array_equal(torch.stack(rews).cpu().numpy(), ref["rewards"])
    assert np.array_equal(torch.stack(reasons).cpu().numpy(), ref["reasons"])
    b, h, m = [x.cpu().numpy() for x in env.export()]
    assert np.array_equal(b, ref["boards"]) and np.array_equal(h, ref["hands"])
    assert np.array_equal(env.mask.cpu().numpy(), ref["mask"]) and np.array_equal(env.obs.cpu().numpy(), ref["obs"])
    assert (ref["reasons"] == 1).sum() > 0  # checkmates happened


def test_uchifuzume_fast_path_agrees_with_nested_generation():
    """The same positions through refresh mode (nested generation, UFZ_GENERIC) and, one ply later, through
    step mode (UFZ_FAST) must give the oracle's legal sets; pawn-drop mates must actually occur in the sample."""
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    n = 4096
    start = _random_endgames(n, 11)
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, seed=3, auto_reset=False)
    env.load_positions(*start, eval_termination=False)
    env.step_index = 0
    env.refresh(random_actions=True)
    for t in range(3):
        env.step(env.next_actions.clone(), random_actions=True)
    torch.cuda.synchronize()
    b, h, m = [x.cpu().numpy() for x in env.export()]
    mask = env.mask.cpu().numpy()
    ufz_seen = 0
    for e in range(n):
        if m[e, 3] != 0:
            continue
        g = orc.OracleGame.from_arrays(b[e], h[e], int(m[e, 0]), int(m[e, 1]), 500, evaluate_termination=False)
        want = g.legal_indices()
        got = np.nonzero(mask[e])[0]
        assert np.array_equal(got, want), (e, _explain(b[e], h[e], m[e, 0], got, want))
        # count positions where a pawn drop in front of the enemy king is excluded although the square is free
        side = int(m[e, 0])
        if h[e][side * 7] > 0:
            ke = np.nonzero(b[e] == (22 if side == 0 else 8))[0]
            if len(ke):
                D = int(ke[0]) + (9 if side == 0 else -9)
                if 0 <= D < 81 and b[e][D] == 0 and mask[e][12960 + D * 7] == 0:
                    col = D % 9
                    nifu = any(b[e][r * 9 + col] == 1 + 14 * side for r in range(9))
                    if not nifu and D // 9 != (0 if side == 0 else 8) and not g.in_check(side):
                        ufz_seen += 1
    assert ufz_seen > 0


def test_long_game_stress_mix():
    """BASELINE config 5 in miniature: one batch mixing start positions, drop-heavy endgames and 4-ply-cycle
    scripts that must end by sennichite on ply 13, with max-move truncation, at 262,144-env layout sizes checked
    for memory only (state bytes) and 6,144 envs stepped against the oracle's termination histogram."""
    import ctypes as C
    from shogidrl_b200 import VecShogiEnv, _native as nv

    offs, total = (C.c_int64 * 3)(), C.c_int64()
    assert nv.lib().kz_state_layout(262144, 500, offs, C.byref(total)) == 0
    assert total.value < 5 * 2**30  # 4.3 GB of state per GPU for 262,144 games with 500-ply repetition tables

    dev = torch.device("cuda:0")
    n_each, T, max_moves, seed = 2048, 90, 80, 21
    n = 3 * n_each
    start = orc.OracleGame().export()
    eg = _random_endgames(n_each, 77)
    cyc = orc.parse_sfen("4k4/9/9/9/9/R8/9/9/4K4 b - 1")
    boards = np.concatenate([np.tile(start[0], (n_each, 1)), eg[0], np.tile(cyc[0], (n_each, 1))])
    hands = np.concatenate([np.tile(start[1], (n_each, 1)), eg[1], np.tile(cyc[1], (n_each, 1))])
    sides = np.concatenate([np.zeros(n_each, np.uint8), eg[2], np.zeros(n_each, np.uint8)])
    mcs = np.zeros(n, np.int32)
    env = VecShogiEnv(n, max_moves_per_game=max_moves, device=dev, seed=seed, auto_reset=True)
    env.load_positions(boards, hands, sides, mcs, eval_termination=False)
    env.step_index = 0
    env.refresh(random_actions=True)
    # scripted third: the 4-ply rook/king cycle; others: random legal
    from shogidrl_b200.utils import move_to_index
    cycle = [move_to_index(m) for m in [(5, 0, 5, 1, False), (0, 4, 0, 3, False), (5, 1, 5, 0, False), (0, 3, 0, 4, False)]]
    reasons = []
    senn_at = np.full(n_each, -1)
    for t in range(T):
        a = env.next_actions.clone()
        if t < 13:
            a[2 * n_each:] = cycle[t % 4]
        out = env.step(a, random_actions=True)
        r = out["reason"].cpu().numpy()
        reasons.append(r.copy())
        if t < 13:
            assert (r[2 * n_each:] == (4 if t == 12 else 0)).all(), t  # sennichite exactly on the 13th ply
    torch.cuda.synchronize()
    assert int(env.errors().abs().sum()) == 0
    reasons = np.stack(reasons)
    # the random two thirds against the oracle (same RNG, same starts)
    ref = orc.selfplay(2 * n_each, T, max_moves=max_moves, seed=seed, threads=os.cpu_count() or 1,
                       start=(boards[:2 * n_each], hands[:2 * n_each], sides[:2 * n_each], mcs[:2 * n_each]))
    assert np.array_equal(reasons[:, :2 * n_each], ref["reasons"])
    hist = np.bincount(reasons[:, :2 * n_each].ravel(), minlength=5)
    assert hist[1] > 0 and hist[3] > 0  # checkmates and max-move truncations both occur


def test_full_size_stress_properties():
    """BASELINE config 5 at its full per-GPU size (262,144 games, 500-ply repetition tables): a mix of start
    positions, drop-heavy endgames and sennichite cycles stepped with random legal play under max-move truncation.
    The oracle cannot follow at this size, so the check is through size-independent properties every step:
    no error bits; piece conservation (board + hands) per game between resets; the mask row's popcount equals the
    kernel's legal count and the pre-selected next action is legal; move counters never pass max_moves; a reset
    game is exactly the start position; and at the end kz_refresh reproduces the obs / mask that kz_step wrote."""
    from shogidrl_b200 import VecShogiEnv
    dev = torch.device("cuda:0")
    n, max_moves, T = 262144, 96, 40
    n_each = 2048
    start = orc.OracleGame().export()
    eg = _random_endgames(n_each, 123)
    cyc = orc.parse_sfen("4k4/9/9/9/9/R8/9/9/4K4 b - 1")
    reps = n // (4 * n_each)
    boards = np.concatenate([np.tile(start[0], (2 * n_each, 1)), eg[0], np.tile(cyc[0], (n_each, 1))] * reps)
    hands = np.concatenate([np.tile(start[1], (2 * n_each, 1)), eg[1], np.tile(cyc[1], (n_each, 1))] * reps)
    sides = np.concatenate([np.zeros(2 * n_each, np.uint8), eg[2], np.zeros(n_each, np.uint8)] * reps)
    rng = np.random.default_rng(5)
    mcs = rng.integers(0, max_moves - 8, n).astype(np.int32)      # staggered move counters: truncations at every step
    assert boards.shape[0] == n
    env = VecShogiEnv(n, max_moves_per_game=max_moves, device=dev, seed=99, auto_reset=True)
    env.load_positions(boards, hands, sides, mcs, eval_termination=False)
    env.refresh(random_actions=True)
    start_b = torch.as_tensor(start[0], device=dev)
    b0, h0, _ = env.export()
    pieces = (b0 != 0).sum(1) + h0.sum(1, dtype=torch.int64)
    reasons = torch.zeros(5, dtype=torch.int64, device=dev)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    for t in range(T):
        a = acts[t & 1]
        assert bool(env.mask.gather(1, a[:, None]).all())                      # pre-selected action is legal
        out = env.step(a, random_actions=True, next_out=acts[(t + 1) & 1])
        done = out["done"].bool()
        reasons += torch.bincount(out["reason"].long(), minlength=5)
        b, h, m = env.export()
        now = (b != 0).sum(1) + h.sum(1, dtype=torch.int64)
        assert bool((now[~done] == pieces[~done]).all())                       # conservation while a game runs
        assert bool((b[done] == start_b).all()) and bool((h[done] == 0).all()) and bool((m[done, 1] == 0).all())
        assert bool((m[done, 0] == 0).all())                                   # reset games: start position, Black to move
        pieces = torch.where(done, torch.full_like(pieces, 40), pieces)
        assert int(m[:, 1].max()) < max_moves and int(env.errors().abs().sum()) == 0
        if t % 8 == 0 or t == T - 1:
            assert torch.equal(env.mask.sum(1, dtype=torch.int32), out["legal_count"].int())
            assert int(out["legal_count"].min()) > 0                           # live games always have a legal move
    obs_k, mask_k = env.obs.clone(), env.mask.clone()
    env.refresh()
    assert torch.equal(env.obs, obs_k) and torch.equal(env.mask, mask_k)       # refresh == what the step kernel wrote
    r = reasons.tolist()
    assert r[1] > 0 and r[3] > 0 and r[4] > 0, r                               # checkmates, truncations and sennichite all occur


def test_config5_full_size():
    """BASELINE config 5 at its stated per-GPU shape -- 262,144 games, max_moves 500, the 1/3 hirate / 1/3 drops-heavy
    endgames / 1/3 4-ply-cycle start mix that ``bench.py --workload cfg5`` runs -- stepped for 520 plies with random legal
    play, so that every kind of ending occurs: checkmates, 500-ply truncations, sennichite (all scripted games exactly on
    ply 13).  A sample of 4,096 games of THIS batch (2,048 hirate + 2,048 endgame starts, each keyed by its own position
    in the batch) is replayed by the oracle: per-step termination reasons, hence the histogram, must be identical."""
    import bench
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200.utils import move_to_index

    dev = torch.device("cuda:0")
    n, T, seed, k = 262144, 520, 1234, 2048
    boards, hands, sides, mcs, (n_h, n_e, n_c) = bench.cfg5_positions(n)
    assert n_h + n_e + n_c == n and min(n_h, n_e, n_c) >= n // 3
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, seed=seed, auto_reset=True)
    assert env.state_bytes < 5 * 2 ** 30  # 4.3 GB of state: 500-ply repetition tables for 262,144 games
    env.load_positions(boards, hands, sides, mcs, eval_termination=False)
    env.step_index = 0
    acts = [torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)]
    env.refresh(random_actions=True, next_out=acts[0])
    cycle = [move_to_index(m) for m in bench.CYCLE_MOVES]
    blocks = [(0, k), (n_h, n_h + k)]  # the sampled games: first 2,048 hirate starts, first 2,048 endgame starts
    sample = torch.cat([torch.arange(a, b, device=dev) for a, b in blocks])
    reasons = torch.zeros((T, sample.numel()), dtype=torch.uint8, device=dev)
    hist = torch.zeros(5, dtype=torch.int64, device=dev)
    for t in range(T):
        a = acts[t & 1]
        if t < 13:
            a[n_h + n_e:] = cycle[t % 4]
        out = env.step(a, random_actions=True, next_out=acts[(t + 1) & 1])
        reasons[t] = out["reason"][sample]
        hist += torch.bincount(out["reason"].long(), minlength=5)
        if t < 13:
            want = 4 if t == 12 else 0
            assert bool((out["reason"][n_h + n_e:] == want).all()), t  # sennichite exactly on the 13th ply, all 87,381 games
    assert int(env.errors().abs().sum()) == 0
    h = hist.tolist()
    assert h[1] > 0 and h[3] > 0 and h[4] >= n_c, h  # Tsumi, max-moves and sennichite all occur
    got = reasons.cpu().numpy()
    for j, (a, b) in enumerate(blocks):
        ref = orc.selfplay(b - a, T, env0=a, max_moves=500, seed=seed, threads=os.cpu_count() or 1, want_final=False,
                           start=(boards[a:b], hands[a:b], sides[a:b], mcs[a:b]))
        assert np.array_equal(got[:, j * k:(j + 1) * k], ref["reasons"]), j
        assert np.bincount(ref["reasons"].ravel(), minlength=5)[1:].sum() > 0


def test_storage_and_action_validation_on_a_live_env():
    """The Python layer refuses storage the kernel would overrun or mis-stride (the C ABI only sees pointers)."""
    from shogidrl_b200 import VecShogiEnv

    dev = torch.device("cuda:0")
    env = VecShogiEnv(8, device=dev)
    good = torch.zeros(8, dtype=torch.int64, device=dev)
    for bad in (torch.zeros(7, dtype=torch.int64, device=dev), torch.zeros(8, dtype=torch.float32, device=dev),
                torch.zeros(16, dtype=torch.int64, device=dev)[::2], torch.zeros(8, dtype=torch.int64)):
        with pytest.raises(ValueError):
            env.step(bad)
    with pytest.raises(ValueError):
        env.step(good, obs=torch.zeros((7, 46, 9, 9), device=dev))
    with pytest.raises(ValueError):
        env.step(good, mask=torch.zeros((8, 13000), dtype=torch.uint8, device=dev))
    with pytest.raises(ValueError):
        env.refresh(obs=torch.zeros((8, 46, 9, 9), dtype=torch.float64, device=dev))
    with pytest.raises(ValueError):
        env.step(good, random_actions=True, next_out=good)
    assert int(env.errors().abs().sum()) == 0 and env.step_index == 0  # nothing was launched
    out = env.step(torch.full((8,), 13526 + 1, dtype=torch.int64, device=dev))  # out-of-range index: per-env error bit
    assert int(out["done"].sum()) == 0 and bool((env.errors() & 1).all())


@pytest.mark.parametrize("n,T", [(4096, 90), (8, 70)])
def test_row_writer_variants_agree(n, T):
    """kz_step composes 32-byte aligned, padded mask rows once from the legal bitmap, and writes exactly-13,527-byte rows
    byte by byte; the rollout form (kz_step_rollout) leaves the bitmap itself; a batch may be stepped as concurrent
    ranges of games (kz_step_range, ``step_streams``).  Triplet batches must produce identical masks, observations,
    scalars and next actions every step, across auto-resets."""
    from shogidrl_b200 import VecShogiEnv, rl

    dev = torch.device("cuda:0")
    envs = [VecShogiEnv(n, max_moves_per_game=60, device=dev, seed=11, step_streams=k) for k in (1, 2 if n >= 64 else 1, 2 if n >= 64 else 1)]
    assert envs[2].step_streams == (2 if n >= 64 else 1)
    acts = [[torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)] for _ in range(3)]
    for e, a in zip(envs, acts):
        e.refresh(random_actions=True, next_out=a[0])
    contiguous = torch.zeros((n, 13527), dtype=torch.uint8, device=dev)
    bitmap = torch.zeros((n, 448), dtype=torch.int32, device=dev)
    obs_r = torch.zeros((n, 46, 9, 9), dtype=torch.float32, device=dev)
    finished = 0
    for t in range(T):
        for e in envs[:1]:
            e.obs.fill_(-3.0); e._mask_store.fill_(5)
        contiguous.fill_(9); envs[1].obs.fill_(7.0); obs_r.fill_(-1.0); bitmap.fill_(-1)
        o0 = envs[0].step(acts[0][t & 1], random_actions=True, next_out=acts[0][(t + 1) & 1])            # composed once
        o1 = envs[1].step(acts[1][t & 1], mask=contiguous, random_actions=True, next_out=acts[1][(t + 1) & 1])  # byte rows
        o2 = envs[2].step_rollout(acts[2][t & 1], obs_r, bitmap, random_actions=True, next_out=acts[2][(t + 1) & 1])
        assert torch.equal(envs[0].mask, contiguous), t
        assert torch.equal(envs[0].obs, envs[1].obs) and torch.equal(envs[0].obs, obs_r), t
        assert torch.equal(rl.bitmap_to_mask(bitmap).view(torch.uint8), contiguous), t
        assert bool((envs[0]._mask_store[:, 13527:] == 0).all())
        for k in ("reward", "done", "reason", "winner", "ep_len", "legal_count"):
            assert torch.equal(o0[k], o1[k]) and torch.equal(o0[k], o2[k]), (t, k)
        assert torch.equal(acts[0][(t + 1) & 1], acts[1][(t + 1) & 1]) and torch.equal(acts[0][(t + 1) & 1], acts[2][(t + 1) & 1])
        finished += int(o0["done"].sum())
    assert finished > 0
    for e in envs:
        assert int(e.errors().abs().sum()) == 0
    assert all(torch.equal(x, y) for x, y in zip(envs[0].export(), envs[2].export()))
    b2 = torch.zeros_like(bitmap)
    envs[0].legal_bitmap(b2)
    assert torch.equal(b2, bitmap)
