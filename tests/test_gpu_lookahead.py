"""The one-ply look-ahead opponent on the device (kz_capture_gain, kz_lookahead_select, VecShogiEnv.lookahead_actions and
the "lookahead" player of evaluation) against the CPU oracle's own rules (tests/lookahead_ref.c) and, for games with
history, against a composition of existing public calls."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests import checks_ref, lookahead_ref  # noqa: E402  (checker only)
from tests.heuristic_ref import fixture_positions, rand32  # noqa: E402

DEV = torch.device("cuda:0")
WORDS = 423
CHUNK = 8192
MATE = lookahead_ref.MATE
VALUE = torch.tensor(lookahead_ref.VALUE, dtype=torch.int32)
BASE = torch.tensor([0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3, 5, 6])
PROMOTED = torch.tensor([8, 9, 10, 11, 4, 12, 13, 7, 8, 9, 10, 11, 12, 13])
KNOWN = ["8k/9/9/9/4r4/9/9/4R4/K8 b - 1", "4k4/4g4/9/9/9/9/9/4R4/K8 b - 1", "8k/9/9/4S4/9/9/9/9/K8 b - 1",
         "4k4/9/4P4/9/8s/9/9/9/4K3L b G 1",
         "1pR4+Nb/l1P1Pp2P/2p1knp2/1ss4pl/p2s1gPG1/n1b1G2P1/lP1g2S2/+n2P+pR2L/+p1K6 b 3P 2",
         "2l2G+LGp/+P+P2+PS3/2p2+N2+S/1P1P2pk1/plGppp1p1/Ppgs5/4S1P+n1/+p3R1+bB1/+n+p+n+r4K b L 2",
         "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"]


def _env(n, max_moves=65535, hist_cap=4, **kw):
    from shogidrl_b200 import VecShogiEnv
    return VecShogiEnv(n, max_moves_per_game=max_moves, device=DEV, hist_cap=hist_cap, auto_reset=False, **kw)


def _blob(env):
    """The state blob without its trailing scheduling block (the work counter kz_expand may write)."""
    return env.state[: env.state_bytes - 256].clone()


def _capture_gain(env, rows, stride):
    from shogidrl_b200 import _native as nv
    gain = torch.full((env.n,), -7, dtype=torch.int32, device=DEV)
    count = torch.full((env.n,), -7, dtype=torch.int32, device=DEV)
    nv.check(nv.lib().kz_capture_gain(env.state.data_ptr(), env.n, env.hist_cap, rows.data_ptr(), stride, gain.data_ptr(),
                                      count.data_ptr(), nv.stream_ptr(DEV)), "kz_capture_gain")
    return gain, count


def _compare(env, label, seeds=(0, 91), steps=(0, 37)):
    """R (gain and count) at strides 448 and 423 with set pad bits, and lookahead_actions for two seeds and two step
    indices (and at max_items 1,024), against the oracle; the state blob stays unchanged."""
    b, h, m = [x.cpu().numpy() for x in env.export()]
    finished = m[:, 3] != 0
    ref_r = lookahead_ref.capture_gain_batch(b, h, m[:, 0])
    ref = lookahead_ref.lookahead_batch(b, h, m[:, 0])
    bitmap = torch.zeros((env.n, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    before = _blob(env)
    want_gain = np.where(finished, 0, ref_r["gain"])
    want_count = np.where(finished, 0, ref_r["count"])
    dirty = bitmap.clone()
    dirty[:, WORDS - 1] |= torch.tensor(-(1 << 23), dtype=torch.int32)  # pad bits 13,527..13,535
    dirty[:, WORDS:] = -1
    narrow = bitmap[:, :WORDS].contiguous()
    for rows, stride, what in ((bitmap, 448, "448"), (dirty, 448, "pad bits"), (narrow, WORDS, "423")):
        gain, count = _capture_gain(env, rows, stride)
        assert np.array_equal(gain.cpu().numpy(), want_gain), (label, what, "R")
        assert np.array_equal(count.cpu().numpy(), want_count), (label, what, "R count")
    best = np.where(finished, 0, ref["best"])
    ties = np.where(finished, 0, ref["ties"])
    seed0, step0 = env.seed, env.step_index
    for seed in seeds:
        for step in steps:
            env.seed, env.step_index = seed, step
            want = np.where(finished, -1, lookahead_ref.picks(ref, seed, step, env.env_offset))
            score = torch.empty(env.n, dtype=torch.int32, device=DEV)
            tie = torch.empty(env.n, dtype=torch.int32, device=DEV)
            got = env.lookahead_actions(score=score, ties=tie)
            assert np.array_equal(score.cpu().numpy(), best), (label, seed, step, "score")
            assert np.array_equal(tie.cpu().numpy(), ties), (label, seed, step, "ties")
            bad = np.flatnonzero(got.cpu().numpy() != want)
            assert bad.size == 0, (label, seed, step, "action", bad[:8].tolist(), env.to_sfen([int(bad[0])]))
            assert env.step_index == step
    small = env.lookahead_actions(max_items=1024)
    assert torch.equal(small, got), (label, "max_items 1024")
    env.seed, env.step_index = seed0, step0
    torch.cuda.synchronize()
    assert torch.equal(_blob(env), before), (label, "state blob written")


def _in_contract(sfens):
    """Positions in which the side not to move is not in check and both kings stand (the engine's contract)."""
    keep = []
    for s in sfens:
        b = orc.parse_sfen(s)[0]
        if (b == 8).any() and (b == 22).any() and not checks_ref.checks(s)["enemy_in_check"]:
            keep.append(s)
    return keep


def test_capture_gain_and_picks_match_oracle(golden_dir):
    """Every ply of both golden traces, the known-answer positions, the reference's fixture positions and 12,288 device
    self-play positions loaded through load_positions."""
    fx = fixture_positions(golden_dir)
    n = len(fx["sides"])
    for c0 in range(0, n, CHUNK):
        sl = slice(c0, c0 + CHUNK)
        k = len(fx["sides"][sl])
        env = _env(k)
        env.load_positions(fx["boards"][sl], fx["hands"][sl], fx["sides"][sl], np.zeros(k, np.int32))
        _compare(env, f"traces[{c0}:]")
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as z:
        kat = _in_contract([str(s) for s in z["sfens"]]) + KNOWN
    env = _env(len(kat))
    env.load_sfens(kat)
    _compare(env, "kat + known")
    from shogidrl_b200 import VecShogiEnv
    play = VecShogiEnv(4096, max_moves_per_game=500, device=DEV, seed=123, auto_reset=True)
    play.refresh(random_actions=True)
    boards, hands, sides = [], [], []
    for ply in range(301):
        if ply in (40, 140, 300):
            b, h, m = [x.cpu().numpy() for x in play.export()]
            boards.append(b); hands.append(h); sides.append(m[:, 0].astype(np.uint8))
        play.step(play.next_actions.clone(), random_actions=True)
    boards, hands, sides = np.concatenate(boards), np.concatenate(hands), np.concatenate(sides)
    for c0 in range(0, len(sides), CHUNK):
        sl = slice(c0, c0 + CHUNK)
        k = len(sides[sl])
        env = _env(k, env_offset=5)
        env.load_positions(boards[sl], hands[sl], sides[sl], np.zeros(k, np.int32))
        _compare(env, f"selfplay[{c0}:]", seeds=(4,), steps=(9,))


def test_finished_games_and_inactive_envs_get_minus_one_and_add_no_items():
    from shogidrl_b200.shogi.sfen import pack_sfen
    p = pack_sfen("4k4/9/4P4/9/9/9/9/9/4K4 b G 7")  # move count 6
    env = _env(4, max_moves=500)
    env.load_positions(np.stack([p[0]] * 4), np.stack([p[1]] * 4), np.zeros(4, np.uint8), np.array([p[3]] * 4, np.int32),
                       max_moves=np.array([500, p[3], 500, 500], np.int32))
    env.step(torch.tensor([13055, 0, 0, 0], dtype=torch.int64, device=DEV))  # game 0 mated, game 1 ended at load
    assert env.export()[2][:, 3].tolist()[:2] == [1, 3]
    chunks = []
    real = env._lookahead_chunk
    env._lookahead_chunk = lambda i0, i1, *a: (chunks.append((i0, i1)), real(i0, i1, *a))
    score = torch.full((4,), 5, dtype=torch.int32, device=DEV)
    ties = torch.full((4,), 5, dtype=torch.int32, device=DEV)
    active = torch.tensor([True, True, False, True], device=DEV)
    out = env.lookahead_actions(active=active, score=score, ties=ties)
    assert out.tolist()[:3] == [-1, -1, -1] and score.tolist()[:3] == [0, 0, 0] and ties.tolist()[:3] == [0, 0, 0]
    # only game 3 (the position after 0-index action 0 was rejected: the same as the loaded one) lists its moves
    assert int(env.legal_count[3]) > 0 and chunks == [(0, int(env.legal_count[3]))]
    assert int(score[3]) == MATE and int(ties[3]) == 1 and int(out[3]) == 13055
    chunks.clear()
    out32 = torch.empty(4, dtype=torch.int32, device=DEV)
    env.lookahead_actions(out=out32, active=torch.zeros(4, dtype=torch.uint8, device=DEV))
    assert out32.tolist() == [-1] * 4 and chunks == []


def _composed(env):
    """Per-env (best score, ties, tied actions) of the look-ahead from public calls: legal_actions, expand, a gain
    computation on export() boards, and mate_in_one / legal_actions on an env holding the children."""
    from shogidrl_b200 import _native as nv
    offsets, parent, actions = env.legal_actions()
    m = int(parent.numel())
    child = _env(m, hist_cap=1)
    out = {k: torch.empty(m, dtype=dt, device=DEV) for k, dt in (("done", torch.uint8), ("reason", torch.uint8),
                                                                   ("err", torch.uint8))}
    nv.check(nv.lib().kz_expand(env.state.data_ptr(), env.n, env.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1, m,
                                None, 0, None, 0, None, None, out["done"].data_ptr(), out["reason"].data_ptr(), None,
                                None, None, out["err"].data_ptr(), child.state.data_ptr(), 1, nv.stream_ptr(DEV)),
             "kz_expand")
    ref = env.expand(parent, actions)
    for k in out:
        assert torch.equal(out[k], ref[k])

    def gains(e, par, act):
        b, _, meta = e.export()
        b, side = b.long().cpu(), meta[:, 0].long().cpu()
        par, act = par.long().cpu(), act.cpu()
        board = act < 12960
        pair = torch.where(board, act, 0) >> 1
        frm, t = pair // 80, pair % 80
        to = t + (t >= frm).long()
        dst, src = b[par, to], b[par, frm]
        enemy = (dst != 0) & ((dst >= 15).long() != side[par])
        dt, st = (dst - 1) % 14, (src - 1) % 14
        g = torch.where(enemy, VALUE[dt] + VALUE[BASE[dt]], 0)
        g = g + torch.where((act & 1).bool() & (src != 0), VALUE[PROMOTED[st]] - VALUE[st], 0)
        return torch.where(board, g, 0)

    g = gains(env, parent, actions)
    c_off, c_par, c_act = child.legal_actions()
    cg = gains(child, c_par, c_act)
    r = torch.zeros(m, dtype=torch.int64).scatter_reduce_(0, c_par.long().cpu(), cg.long(), "amax")
    r = torch.where(child.export()[2][:, 3].cpu() != 0, 0, r)
    mates = child.mate_in_one()["count"].cpu() > 0
    done, reason, err = out["done"].cpu() != 0, out["reason"].cpu(), out["err"].cpu()
    s = torch.where(mates, -MATE, g - r)
    s = torch.where(done, torch.where((reason == 1) & ((err & 4) == 0), MATE, g), s)
    per = []
    off = offsets.cpu().tolist()
    act_h = actions.cpu()
    for e in range(env.n):
        row = s[off[e]:off[e + 1]]
        if row.numel() == 0:
            per.append((0, 0, []))
            continue
        bst = int(row.max())
        per.append((bst, int((row == bst).sum()), act_h[off[e]:off[e + 1]][row == bst].tolist()))
    return per, (parent, actions, out, g, r, mates, offsets)


def _check_composed(env, label):
    per, _ = _composed(env)
    score = torch.empty(env.n, dtype=torch.int32, device=DEV)
    ties = torch.empty(env.n, dtype=torch.int32, device=DEV)
    got = env.lookahead_actions(score=score, ties=ties).cpu().tolist()
    finished = (env.export()[2][:, 3] != 0).cpu().tolist()
    salt = env.seed ^ lookahead_ref.SALT
    for e, (bst, t, tied) in enumerate(per):
        if finished[e] or t == 0:
            assert (got[e], int(score[e]), int(ties[e])) == (-1, 0, 0), (label, e)
            continue
        assert (int(score[e]), int(ties[e])) == (bst, t), (label, e)
        assert got[e] == tied[(rand32(salt, env.env_offset + e, env.step_index) * t) >> 32], (label, e)


def test_sennichite_move_scores_rule_2(golden_dir):
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200 import _native as nv
    with np.load(os.path.join(golden_dir, "scripted.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    env = VecShogiEnv(1, max_moves_per_game=500, device=DEV, auto_reset=False)
    env.load_sfens([str(z["senn_sfen"])])
    acts = z["senn_actions"]
    for t in range(len(acts) - 1):  # one ply before the 4th repetition
        env.step(torch.tensor([int(acts[t])], device=DEV))
    _check_composed(env, "sennichite")
    per, (parent, actions, out, g, r, mates, offsets) = _composed(env)
    rep = (actions == int(acts[-1])).nonzero().flatten().tolist()
    assert len(rep) == 1 and int(out["reason"][rep[0]]) == 4
    i = rep[0]
    # the repeating move alone through kz_lookahead_select: a draw scores its gain (rule 2), whatever the replies
    one = torch.tensor([0, 1], dtype=torch.int64, device=DEV)
    items = [actions[i:i + 1].contiguous(), out["done"][i:i + 1].contiguous(), out["reason"][i:i + 1].contiguous(),
             out["err"][i:i + 1].contiguous(), torch.tensor([99], dtype=torch.int32, device=DEV),
             torch.tensor([1], dtype=torch.int32, device=DEV)]
    pick = torch.empty(1, dtype=torch.int64, device=DEV)
    score = torch.empty(1, dtype=torch.int32, device=DEV)
    tie = torch.empty(1, dtype=torch.int32, device=DEV)
    nv.check(nv.lib().kz_lookahead_select(env.state.data_ptr(), 1, env.hist_cap, one.data_ptr(), 1, items[0].data_ptr(), 1,
                                          *[t.data_ptr() for t in items[1:]], 0, 0, 0, pick.data_ptr(), 1, score.data_ptr(),
                                          tie.data_ptr(), nv.stream_ptr(DEV)), "kz_lookahead_select")
    assert int(pick[0]) == int(acts[-1]) and int(score[0]) == int(g[i]) and int(tie[0]) == 1


def test_selfplay_with_history_matches_public_composition():
    """4,096 self-play games with their repetition history at plies 50, 150 and 300."""
    from shogidrl_b200 import VecShogiEnv
    env = VecShogiEnv(4096, max_moves_per_game=500, device=DEV, seed=17, auto_reset=True)
    env.refresh(random_actions=True)
    for ply in range(301):
        if ply in (50, 150, 300):
            _check_composed(env, f"ply {ply}")
        env.step(env.next_actions.clone(), random_actions=True)


def test_offsets_are_clamped():
    """Out-of-range and non-monotone offsets read nothing outside the m items."""
    from shogidrl_b200 import _native as nv
    env = _env(4)
    env.load_sfens([KNOWN[0]] * 4)
    offsets, parent, actions = env.legal_actions()
    m = int(parent.numel())
    out = env.expand(parent, actions)
    rg = torch.zeros(m, dtype=torch.int32, device=DEV)
    rm = torch.zeros(m, dtype=torch.int32, device=DEV)
    for offs, want_empty in (([-5, 15, 10, 60, 10 ** 12], [False, True, False, True]), ([0, m, m, m, m], [False, True, True, True])):
        o = torch.tensor(offs, dtype=torch.int64, device=DEV)
        pick = torch.empty(4, dtype=torch.int64, device=DEV)
        ties = torch.empty(4, dtype=torch.int32, device=DEV)
        nv.check(nv.lib().kz_lookahead_select(env.state.data_ptr(), 4, env.hist_cap, o.data_ptr(), m, actions.data_ptr(), 1,
                                              out["done"].data_ptr(), out["reason"].data_ptr(), out["err"].data_ptr(),
                                              rg.data_ptr(), rm.data_ptr(), 0, 0, 0, pick.data_ptr(), 1, None,
                                              ties.data_ptr(), nv.stream_ptr(DEV)), "kz_lookahead_select")
        assert [p == -1 for p in pick.tolist()] == want_empty
        assert all(p == -1 or 0 <= p < 13527 for p in pick.tolist())


def test_ties_on_hirate_are_uniform():
    from scipy.stats import chisquare
    env = _env(4096, max_moves=500)
    counts = np.zeros(13527, np.int64)
    for step in range(8):
        env.step_index = step
        a = env.lookahead_actions().cpu().numpy()
        np.add.at(counts, a, 1)
    legal = np.flatnonzero(env.mask[0].cpu().numpy())
    assert len(legal) == 30 and counts[legal].sum() == 8 * 4096
    assert chisquare(counts[legal]).pvalue > 1e-4


def test_mate_suite_is_solved():
    from shogidrl_b200.evaluation import evaluate_mate_in_one, harvest_mate_in_one
    positions = harvest_mate_in_one(200, seed=5, num_envs=1024, max_moves_per_game=300, device=DEV)
    r = evaluate_mate_in_one("lookahead", positions, num_envs=128, device=DEV, seed=3)
    assert r.with_mate == len(positions) and r.solved == r.with_mate


class _FirstLegal:
    """A stub agent: the lowest legal action."""

    def select_actions(self, obs, mask, is_training=False):
        return mask.to(torch.uint8).argmax(1), None


def test_evaluation_against_random_and_heuristic():
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200.evaluation import evaluate_vs_opponent
    kw = dict(num_envs=16, max_moves_per_game=200, device=DEV, seed=8)
    runs = {}
    for agent, opp in (("lookahead", "random"), ("random", "lookahead"), ("lookahead", "heuristic"),
                       ("heuristic", "lookahead"), (_FirstLegal(), "lookahead")):
        r = evaluate_vs_opponent(agent, 24, opponent=opp, **kw)
        assert r.games == 24 and len(r.outcomes) == 24
        runs[(str(agent), opp)] = r
    again = evaluate_vs_opponent("lookahead", 24, opponent="heuristic", **kw)
    assert again.outcomes == runs[("lookahead", "heuristic")].outcomes
    assert runs[("lookahead", "random")].agent_wins > runs[("lookahead", "random")].opponent_wins
    # with `active` (only the envs where the look-ahead player moves) and without it (every env computed): same games
    real = VecShogiEnv.lookahead_actions
    try:
        VecShogiEnv.lookahead_actions = lambda self, out=None, *, active=None, **k: real(self, out, **k)
        full = evaluate_vs_opponent("lookahead", 24, opponent="heuristic", **kw)
        full2 = evaluate_vs_opponent("random", 24, opponent="lookahead", **kw)
    finally:
        VecShogiEnv.lookahead_actions = real
    assert full.outcomes == runs[("lookahead", "heuristic")].outcomes
    assert full2.outcomes == runs[("random", "lookahead")].outcomes
    assert full.mean_length == runs[("lookahead", "heuristic")].mean_length
