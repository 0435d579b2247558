"""Checking moves (kz_check_bitmap), mate in one (VecShogiEnv.mate_in_one) and the mate-in-one evaluation, against the
CPU oracle's own rules (tests/checks_ref.c: every legal move applied to a copy, check = king_in_check of the opponent,
mate = check and no legal reply) and against the all-moves device route (legal_actions + expand)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests import checks_ref  # noqa: E402  (checker only)

DEV = torch.device("cuda:0")
WORDS = 423
CHUNK = 8192


def _env(n, max_moves=500, hist_cap=4, **kw):
    from shogidrl_b200 import VecShogiEnv
    return VecShogiEnv(n, max_moves_per_game=max_moves, device=DEV, hist_cap=hist_cap, auto_reset=False, **kw)


def _blob(env):
    """The state blob without its trailing scheduling block (the work counter kz_expand may write)."""
    return env.state[: env.state_bytes - 256].clone()


def _popcount(words: np.ndarray) -> np.ndarray:
    return np.unpackbits(words.view(np.uint8), axis=1).sum(1)


def _all_moves_mates(env):
    """The route mate_in_one replaces: expand every legal move, keep Tsumi that does not capture a king."""
    _, parent, actions = env.legal_actions()
    count = torch.zeros(env.n, dtype=torch.int64, device=DEV)
    first = torch.full((env.n,), 1 << 20, dtype=torch.int64, device=DEV)
    if parent.numel():
        out = env.expand(parent, actions)
        mate = (out["reason"] == 1) & ((out["err"] & 4) == 0)
        count.index_add_(0, parent.long(), mate.long())
        first.scatter_reduce_(0, parent.long(), torch.where(mate, actions, 1 << 20), "amin")
    return count.cpu().numpy(), np.where(count.cpu().numpy() > 0, first.cpu().numpy(), -1)


def _compare(env, label, totals):
    """Check rows and mates of every env's current position against the oracle; adds the classes of the compared
    in-contract checking moves to totals."""
    bitmap = torch.zeros((env.n, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    before = _blob(env)
    rows, count = env.check_bitmap(bitmap)
    mates = env.mate_in_one()
    torch.cuda.synchronize()
    assert torch.equal(_blob(env), before), (label, "state blob written")
    b, h, m = [x.cpu().numpy() for x in env.export()]
    ref = checks_ref.checks_batch(b, h, m[:, 0])
    finished = m[:, 3] != 0
    full = ref["enemy_in_check"] != 0  # out of contract (or no enemy king): the row is every legal move
    want = np.where(full[:, None], ref["legal"], ref["check"])
    want[finished] = 0
    got = rows.cpu().numpy().view(np.uint32)
    dev_legal = bitmap.cpu().numpy().view(np.uint32)
    assert np.array_equal(dev_legal[:, :WORDS], ref["legal"]), (label, "legal rows")
    bad = np.flatnonzero((got[:, :WORDS] != want).any(1))
    assert bad.size == 0, (label, "check rows differ", bad[:8].tolist(), [env.to_sfen([int(i)])[0] for i in bad[:3]])
    assert not got[:, WORDS:].any(), (label, "words 423..")
    assert not (got[:, WORDS - 1] >> 23).any(), (label, "pad bits")
    assert not (got[:, :WORDS] & ~dev_legal[:, :WORDS]).any(), (label, "not a subset of the legal row")
    assert np.array_equal(count.cpu().numpy(), _popcount(got)), (label, "count")
    want_count = np.where(finished, 0, ref["mate_count"])
    want_first = np.where(finished, -1, ref["mate_lowest"])
    assert np.array_equal(mates["count"].cpu().numpy(), want_count), (label, "mate count")
    assert np.array_equal(mates["action"].cpu().numpy(), want_first), (label, "lowest mate")
    c2, f2 = _all_moves_mates(env)
    assert np.array_equal(c2, want_count) and np.array_equal(f2, want_first), (label, "all-moves route")
    torch.cuda.synchronize()
    assert torch.equal(_blob(env), before), (label, "state blob written")
    keep = ~full & ~finished
    totals["positions"] += int(keep.sum())
    totals["classes"] += ref["class_counts"][keep].sum(0)
    totals["mates"] += int((want_count > 0).sum())


def _compare_positions(boards, hands, sides, label, totals):
    """Load positions (no history, max_moves high enough that none ends at load by the move limit) in chunks."""
    for c0 in range(0, len(sides), CHUNK):
        sl = slice(c0, c0 + CHUNK)
        n = len(sides[sl])
        env = _env(n, max_moves=65535)
        env.load_positions(boards[sl], hands[sl], sides[sl], np.zeros(n, np.int32))
        _compare(env, f"{label}[{c0}:]", totals)


def test_check_rows_and_mates_match_oracle(golden_dir):
    """Every ply of the random and endgame golden traces, the known-answer positions and 114,688 device self-play
    positions: rows bit for bit, counts, mates (count and lowest action) against the oracle and the all-moves route."""
    totals = {"positions": 0, "classes": np.zeros(6, np.int64), "mates": 0}
    for name in ("traces_random", "traces_endgame"):
        with np.load(os.path.join(golden_dir, f"{name}.npz")) as z:
            _compare_positions(z["boards"], z["hands"], z["sides"], name, totals)
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as z:
        kat = [str(s) for s in z["sfens"]]
    env = _env(len(kat), max_moves=65535)
    env.load_sfens(kat)
    _compare(env, "kat", totals)
    # self-play: 16,384 games with auto-reset, 7 snapshots
    from shogidrl_b200 import VecShogiEnv
    env = VecShogiEnv(16384, max_moves_per_game=500, device=DEV, seed=77, auto_reset=True)
    env.refresh(random_actions=True)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    snaps = {20, 60, 100, 150, 220, 320, 450}
    for ply in range(max(snaps) + 1):
        if ply in snaps:
            _compare(env, f"selfplay ply {ply}", totals)
        env.step(acts[ply % 2], next_out=acts[(ply + 1) % 2], random_actions=True)
    assert totals["positions"] >= 25200 + 5920 + 100000
    direct, discovered, double, drop, _, promo_only = totals["classes"].tolist()
    assert min(discovered, double, drop, promo_only) >= 300, totals
    assert direct > 0 and totals["mates"] > 0, totals


def test_strides_and_pad_bits():
    """Row strides 423 and 448 give the same rows; pad bits and words 423.. of the input change nothing."""
    from shogidrl_b200 import _native as nv
    from shogidrl_b200 import VecShogiEnv
    env = VecShogiEnv(1000, max_moves_per_game=500, device=DEV, seed=5, auto_reset=True)
    env.refresh(random_actions=True)
    for _ in range(80):
        env.step(env.next_actions.clone(), random_actions=True)
    bitmap = torch.zeros((env.n, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    rows, count = env.check_bitmap(bitmap)
    assert int(count.sum()) > 0
    dirty = bitmap.clone()
    dirty[:, WORDS - 1] |= torch.tensor(-(1 << 23), dtype=torch.int32)  # bits 13,527..13,535
    dirty[:, WORDS:] = -1
    out = torch.full((env.n, 448), -1, dtype=torch.int32, device=DEV)
    rows2, count2 = env.check_bitmap(dirty, out=out)
    assert rows2 is out and torch.equal(rows2, rows) and torch.equal(count2, count)
    src = bitmap[:, :WORDS].contiguous()
    dst = torch.full((env.n, WORDS), -1, dtype=torch.int32, device=DEV)
    cnt = torch.full((env.n,), -1, dtype=torch.int32, device=DEV)
    nv.check(nv.lib().kz_check_bitmap(env.state.data_ptr(), env.n, env.hist_cap, src.data_ptr(), WORDS, dst.data_ptr(),
                                      WORDS, cnt.data_ptr(), nv.stream_ptr(env.device)), "kz_check_bitmap")
    assert torch.equal(dst, rows[:, :WORDS]) and torch.equal(cnt, count)
    # count may be NULL
    dst.fill_(-1)
    nv.check(nv.lib().kz_check_bitmap(env.state.data_ptr(), env.n, env.hist_cap, src.data_ptr(), WORDS, dst.data_ptr(),
                                      WORDS, None, nv.stream_ptr(env.device)), "kz_check_bitmap")
    assert torch.equal(dst, rows[:, :WORDS])
    with pytest.raises(ValueError, match="bitmap"):
        env.check_bitmap(bitmap[:, :WORDS])


TABLE = [  # sfen, legal, row (checking moves on the device), mates (count, lowest)
    ("lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1", 30, 0, 0, -1),
    ("4k4/9/4P4/9/9/9/9/9/4K4 b G 1", 85, 7, 1, 13055),
    ("7nk/9/8G/9/9/9/9/9/4K4 b P 1", 78, 2, 0, -1),
    ("3gkg3/9/3PSP3/9/4R4/9/9/9/4K4 b - 1", 31, 12, 4, 3544),
    ("9/9/9/9/9/9/9/9/4K4 b G 1", 85, 85, 85, 12292),  # enemy king missing
    ("4k4/9/9/9/4R4/9/9/9/4K4 b - 1", 23, 23, 0, -1),  # enemy already in check: row = every legal move (superset)
]


def test_fixture_positions_on_the_device():
    sfens = [t[0] for t in TABLE]
    env = _env(len(sfens))
    env.load_sfens(sfens)
    bitmap = torch.zeros((env.n, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    rows, count = env.check_bitmap(bitmap)
    mates = env.mate_in_one()
    assert env.legal_count.tolist() == [t[1] for t in TABLE]
    assert count.tolist() == [t[2] for t in TABLE]
    assert mates["count"].tolist() == [t[3] for t in TABLE]
    assert mates["action"].tolist() == [t[4] for t in TABLE]
    offsets, parent, actions = env.checking_actions()
    assert offsets.tolist() == [0] + np.cumsum([t[2] for t in TABLE]).tolist()
    for g, s in enumerate(sfens[:4]):
        assert actions[offsets[g]:offsets[g + 1]].tolist() == checks_ref.checks(s)["checks"], s
        assert (parent[offsets[g]:offsets[g + 1]] == g).all()


def test_finished_games_get_empty_rows():
    """A game finished by Tsumi (auto_reset off) and one finished at load by the move limit while it still has a mate."""
    from shogidrl_b200.shogi.sfen import pack_sfen
    p = pack_sfen("4k4/9/4P4/9/9/9/9/9/4K4 b G 7")  # move count 6
    env = _env(2)
    env.load_positions(np.stack([p[0]] * 2), np.stack([p[1]] * 2), np.zeros(2, np.uint8), np.array([p[3]] * 2, np.int32),
                       max_moves=np.array([500, p[3]], np.int32))
    assert env.export()[2][:, 3].tolist() == [0, 3]  # game 1 ended at load: Max moves reached
    out = env.step(torch.tensor([13055, 0], dtype=torch.int64, device=DEV))  # G*5b mates in game 0
    assert out["reason"].tolist() == [1, 3]
    bitmap = torch.zeros((2, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    rows, count = env.check_bitmap(bitmap)
    assert count.tolist() == [0, 0] and int(rows.abs().sum()) == 0
    assert int(env.legal_count[1]) == 85  # the finished game still lists its moves, the mate among them
    m = env.mate_in_one()
    assert m["count"].tolist() == [0, 0] and m["action"].tolist() == [-1, -1]
    offsets, parent, actions = env.checking_actions()
    assert offsets.tolist() == [0, 0, 0] and parent.numel() == 0 and actions.numel() == 0


def test_harvest_is_deterministic_and_every_position_has_a_mate():
    from shogidrl_b200.evaluation import harvest_mate_in_one
    a = harvest_mate_in_one(64, seed=3, num_envs=512, max_moves_per_game=200, device=DEV)
    b = harvest_mate_in_one(64, seed=3, num_envs=512, max_moves_per_game=200, device=DEV)
    assert len(a) == 64 and a == b
    for s in a:
        assert checks_ref.checks(s)["mates"], s


class _Scripted:
    """A stub agent that plays a precomputed move per position, in the order evaluate_mate_in_one loads them."""

    def __init__(self, moves):
        self.moves, self.i = list(moves), 0

    def select_actions(self, obs, mask, is_training=False):
        n = obs.shape[0]
        a = (self.moves[self.i:self.i + n] + [0] * n)[:n]
        self.i += n
        return torch.tensor(a, dtype=torch.int64, device=obs.device), None


def test_evaluate_mate_in_one_players():
    from shogidrl_b200.evaluation import evaluate_mate_in_one, harvest_mate_in_one
    mated = harvest_mate_in_one(150, seed=11, num_envs=1024, max_moves_per_game=300, device=DEV)
    none = ["lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1", "7nk/9/8G/9/9/9/9/9/4K4 b P 1"]
    positions = mated[:70] + none + mated[70:]
    refs = [checks_ref.checks(s) for s in positions]
    seed = 21
    r = evaluate_mate_in_one("random", positions, num_envs=64, device=DEV, seed=seed)  # 3 batches, the last padded
    want = [orc.OracleGame.from_sfen(s, max_moves=65535).pick_action(seed, i, 0) in ref["mates"]
            for i, (s, ref) in enumerate(zip(positions, refs))]
    assert r.positions == len(positions) and r.with_mate == len(mated)
    assert r.mate_flags == [bool(ref["mates"]) for ref in refs]
    assert r.solved_flags == want and r.solved == sum(want)
    best = evaluate_mate_in_one(_Scripted([ref["mates"][0] if ref["mates"] else ref["legal"][0] for ref in refs]),
                                positions, num_envs=64, device=DEV)
    assert best.solve_rate == 1.0 and best.solved == len(mated)
    quiet = [[a for a in ref["legal"] if a not in ref["mates"]] for ref in refs]
    assert all(quiet)
    worst = evaluate_mate_in_one(_Scripted([q[0] for q in quiet]), positions, num_envs=64, device=DEV)
    assert worst.solve_rate == 0.0 and worst.with_mate == len(mated) and not any(worst.solved_flags)
    h = evaluate_mate_in_one("heuristic", positions, num_envs=64, device=DEV, seed=seed)
    assert h.with_mate == len(mated) and 0 <= h.solved <= len(mated)
