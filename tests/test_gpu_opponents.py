"""The scripted heuristic opponent on the device (kz_heuristic_actions / VecShogiEnv.heuristic_actions) against the
test-side restatement of the reference's rule (tests/heuristic_ref.py) and the CPU oracle, and the scripted players
through the batched evaluation layer."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests import heuristic_ref as H  # noqa: E402
from tests.helpers import make_config, random_endgames  # noqa: E402


def _all_positions(golden_dir):
    """The 31,120 trace positions and the 38 known-answer positions: boards, hands, sides, move counts, legal sets."""
    P = H.fixture_positions(golden_dir)
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    parsed = [orc.parse_sfen(str(s)) for s in z["sfens"]]
    legal = P["legal"] + [z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]] for i in range(len(parsed))]
    return (np.concatenate([P["boards"], np.stack([p[0] for p in parsed])]),
            np.concatenate([P["hands"], np.stack([p[1] for p in parsed])]),
            np.concatenate([P["sides"], np.asarray([p[2] for p in parsed], np.uint8)]),
            np.concatenate([P["move_counts"], np.asarray([p[3] for p in parsed], np.int32)]), legal)


def test_heuristic_actions_match_the_reference_rule(golden_dir):
    """Mask form (padded and unaligned rows) and bitmap form, int64 and int32 outputs: action, tier and tier size of
    every fixture position equal the restated rule, bit for bit, for several seeds and steps."""
    from shogidrl_b200 import VecShogiEnv
    boards, hands, sides, mcs, legal = _all_positions(golden_dir)
    n = len(legal)
    assert n == 31120 + 38
    dev = torch.device("cuda:0")
    env = VecShogiEnv(n, max_moves_per_game=500, device=dev, auto_reset=False)
    env.load_positions(boards, hands, sides, mcs, eval_termination=False)
    assert np.array_equal(env.legal_count.cpu().numpy(), [len(x) for x in legal])
    top = [H.top_tier(boards[i], int(sides[i]), legal[i]) for i in range(n)]
    want_tier = np.asarray([t for t, _ in top], np.uint8)
    want_cnt = np.asarray([len(m) for _, m in top], np.int32)
    assert (want_tier == 255).any() and all((want_tier == t).any() for t in range(3))
    bitmap = torch.zeros((n, 448), dtype=torch.int32, device=dev)
    env.legal_bitmap(bitmap)
    unaligned = torch.zeros((n, 13527), dtype=torch.uint8, device=dev)  # rows at every 16-byte phase
    env.refresh(mask=unaligned)
    tier = torch.empty(n, dtype=torch.uint8, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev)
    for seed, step in [(0, 0), (1234, 1), (2**40 + 17, 77), (99, 2**31)]:
        env.seed, env.step_index = seed, step
        key = seed ^ env.HEURISTIC_SALT
        want = np.asarray([H.pick(m, key, i, step) for i, (_, m) in enumerate(top)], np.int64)
        for form in ("mask", "unaligned", "bitmap", "int32"):
            tier.fill_(7); cnt.fill_(-7)
            if form == "mask":
                got = env.heuristic_actions(tier=tier, tier_count=cnt)
            elif form == "unaligned":
                got = env.heuristic_actions(mask=unaligned, tier=tier, tier_count=cnt)
            elif form == "bitmap":
                got = env.heuristic_actions(bitmap=bitmap, tier=tier, tier_count=cnt)
            else:
                got = env.heuristic_actions(out=torch.empty(n, dtype=torch.int32, device=dev), tier=tier, tier_count=cnt)
            got = got.cpu().numpy().astype(np.int64)
            bad = np.nonzero(got != want)[0]
            assert len(bad) == 0, (form, seed, step, bad[:5], got[bad[:5]], want[bad[:5]])
            assert np.array_equal(tier.cpu().numpy(), want_tier), (form, seed, step)
            assert np.array_equal(cnt.cpu().numpy(), want_cnt), (form, seed, step)


def test_heuristic_actions_reject_bad_arguments():
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200 import _native as nv
    dev = torch.device("cuda:0")
    n = 16
    env = VecShogiEnv(n, device=dev)
    bitmap = torch.zeros((n, 448), dtype=torch.int32, device=dev)
    env.legal_bitmap(bitmap)
    with pytest.raises(ValueError):
        env.heuristic_actions(mask=env.mask, bitmap=bitmap)  # both
    with pytest.raises(ValueError):
        env.heuristic_actions(mask=env.mask[: n - 1])  # too few rows
    with pytest.raises(ValueError):
        env.heuristic_actions(mask=torch.zeros((n, 13000), dtype=torch.uint8, device=dev))  # short rows
    with pytest.raises(ValueError):
        env.heuristic_actions(mask=env.mask.cpu())  # host tensor
    with pytest.raises(ValueError):
        env.heuristic_actions(bitmap=bitmap[:, :440])
    with pytest.raises(ValueError):
        env.heuristic_actions(out=torch.empty(n, dtype=torch.float32, device=dev))
    with pytest.raises(ValueError):
        env.heuristic_actions(out=torch.empty(n - 1, dtype=torch.int64, device=dev))
    with pytest.raises(ValueError):
        env.heuristic_actions(tier=torch.empty(n, dtype=torch.int32, device=dev))
    L = nv.lib()
    out = torch.empty(n, dtype=torch.int64, device=dev)
    st, mp, bp = env.state.data_ptr(), env.mask.data_ptr(), bitmap.data_ptr()
    sp = nv.stream_ptr(env.device)
    args = lambda **kw: [kw.get("state", st), kw.get("n", n), env.hist_cap, kw.get("mask", mp), kw.get("ms", 13536),
                         kw.get("bitmap", None), kw.get("bs", 448), kw.get("out", out.data_ptr()), 1, None, None, 0, 0, 0, sp]
    assert L.kz_heuristic_actions(*args()) == 0
    assert L.kz_heuristic_actions(*args(mask=None, bitmap=bp)) == 0
    for bad in (dict(mask=None), dict(bitmap=bp), dict(state=None), dict(n=0), dict(ms=13526), dict(out=None),
                dict(mask=None, bitmap=bp, bs=422), dict(mask=None, bitmap=bp + 2), dict(out=out.data_ptr() + 4)):
        assert L.kz_heuristic_actions(*args(**bad)) == -1, bad
    torch.cuda.synchronize()


def test_heuristic_vs_random_selfplay_replays_in_the_oracle():
    """1,024 games x 600 plies with auto-reset, half of them from drop-heavy endgames: the heuristic moves for Black in
    even envs and for White in odd ones, the engine's fused uniform-random action for the other side.  Every game is
    replayed ply by ply in the CPU oracle with the restated rule; actions, rewards, dones, reasons and winners agree."""
    from shogidrl_b200 import VecShogiEnv
    dev = torch.device("cuda:0")
    n, T, mm, seed = 1024, 600, 500, 2024
    sb, sh, _ = orc.OracleGame().export()
    eb, eh, es, emc = random_endgames(n // 2, 31)
    boards = np.concatenate([np.repeat(sb[None], n // 2, 0), eb])
    hands = np.concatenate([np.repeat(sh[None], n // 2, 0), eh])
    sides = np.concatenate([np.zeros(n // 2, np.uint8), es])
    env = VecShogiEnv(n, max_moves_per_game=mm, device=dev, seed=seed, auto_reset=True)
    env.load_positions(boards, hands, sides, np.zeros(n, np.int32), eval_termination=False)
    env.step_index = 0
    env.refresh(random_actions=True)
    heur_is_black = (torch.arange(n, device=dev) % 2) == 0
    heur = torch.empty(n, dtype=torch.int64, device=dev)
    rec = {k: [] for k in ("actions", "reward", "done", "reason", "winner")}
    for t in range(T):
        env.heuristic_actions(out=heur)
        a = torch.where((env.obs[:, 42, 0, 0] > 0.5) == heur_is_black, heur, env.next_actions).contiguous()
        out = env.step(a, random_actions=True)
        rec["actions"].append(a)
        for k in ("reward", "done", "reason", "winner"):
            rec[k].append(out[k].clone())
    torch.cuda.synchronize()
    assert int(env.errors().abs().sum()) == 0
    got = {k: torch.stack(v).cpu().numpy() for k, v in rec.items()}
    key = seed ^ env.HEURISTIC_SALT
    games = 0
    for e in range(n):
        g = orc.OracleGame.from_arrays(boards[e], hands[e], sides[e], 0, mm, evaluate_termination=False)
        for t in range(T):
            b, _, m = g.export()
            side = int(m[0])
            if side == e % 2:
                want = H.pick(H.top_tier(b, side, g.legal_indices())[1], key, e, t)
            else:
                want = g.pick_action(seed, e, t)
            assert got["actions"][t, e] == want, (e, t)
            reward, done, reason, winner = g.make_move(want)
            assert (got["reward"][t, e], got["done"][t, e], got["reason"][t, e], got["winner"][t, e]) == \
                (reward, done, reason, winner), (e, t)
            if done:
                games += 1
                g.reset()
    assert games > n  # crossed episode boundaries
    finished = got["done"] != 0
    heur_won = finished & (got["winner"] == (np.arange(n) % 2)[None, :])
    print(f"heuristic vs random, {int(finished.sum())} finished games: heuristic won {int(heur_won.sum())}, "
          f"random won {int((finished & (got['winner'] >= 0)).sum() - heur_won.sum())}")


def test_uniform_within_the_tier():
    """On a position whose capture tier has several members, the draws over (env, step) are uniform over it (chi^2)."""
    from scipy.stats import chisquare
    from shogidrl_b200 import VecShogiEnv
    # Black's rook can take three pawns, one of them with or without promotion: four capture actions
    sfen = "k8/4p4/9/1p5p1/p1p1R1p1p/9/9/9/4K4 b - 1"
    b, h, side, mc = orc.parse_sfen(sfen)
    dev = torch.device("cuda:0")
    n, steps = 4096, 16
    env = VecShogiEnv(n, device=dev, seed=3, auto_reset=False)
    env.load_positions(np.repeat(b[None], n, 0), np.repeat(h[None], n, 0), np.full(n, side, np.uint8),
                       np.full(n, mc, np.int32), eval_termination=False)
    tier, members = H.top_tier(b, side, orc.OracleGame.from_arrays(b, h, side, mc).legal_indices())
    assert tier == 0 and len(members) == 4
    counts = dict.fromkeys(members, 0)
    for s in range(steps):
        env.step_index = s
        for a in env.heuristic_actions().cpu().numpy().tolist():
            counts[a] += 1
    obs = np.asarray(list(counts.values()))
    assert obs.sum() == n * steps
    assert chisquare(obs).pvalue > 1e-4, counts


def test_evaluation_with_scripted_players():
    from shogidrl_b200.core import ActorCritic, PPOAgent
    from shogidrl_b200.evaluation import evaluate_benchmark, evaluate_tournament, evaluate_vs_opponent
    from shogidrl_b200.utils import SimpleHeuristicOpponent, SimpleRandomOpponent
    torch.manual_seed(11)
    agent = PPOAgent(ActorCritic(46, 13527), make_config(), torch.device("cuda"), use_mixed_precision=True)
    kw = dict(num_envs=48, max_moves_per_game=60, seed=5, deterministic=False)

    def check(res, n):
        assert res.games == n and len(res.outcomes) == n
        assert res.agent_wins + res.opponent_wins + res.draws == n
        assert res.outcomes.count("agent_win") == res.agent_wins and res.outcomes.count("draw") == res.draws

    check(evaluate_vs_opponent(agent, 100, opponent="heuristic", **kw), 100)
    check(evaluate_vs_opponent("heuristic", 100, opponent="random", **kw), 100)
    check(evaluate_vs_opponent(SimpleHeuristicOpponent(), 64, opponent=SimpleRandomOpponent(), **kw), 64)
    check(evaluate_vs_opponent("random", 64, opponent="heuristic", **kw), 64)
    check(evaluate_vs_opponent("heuristic", 64, opponent="heuristic", **kw), 64)
    with pytest.raises(ValueError):
        evaluate_vs_opponent(agent, 8, opponent="minimax", **kw)
    standings, results = evaluate_tournament(agent, {"random": None, "heuristic": "heuristic",
                                                     "heuristic_obj": SimpleHeuristicOpponent()}, 32, **kw)
    assert standings["overall_tournament_stats"]["total_games"] == 96
    for r in results.values():
        check(r, 32)
    perf, cases = evaluate_benchmark(agent, {"benchmark_random": None, "benchmark_heuristic": "heuristic"}, 16, **kw)
    assert set(perf["per_benchmark_case_results"]) == {"benchmark_random", "benchmark_heuristic"}
    assert perf["overall_benchmark_pass_rate"] == sum(r.agent_wins for r in cases.values()) / 32


def test_facade_heuristic_opponent_on_a_device_game():
    """The reference-API class on the device-backed ShogiGame facade picks from the top tier of the game's position."""
    import random
    from shogidrl_b200.shogi import ShogiGame
    from shogidrl_b200.utils import PolicyOutputMapper, SimpleHeuristicOpponent
    mapper = PolicyOutputMapper()
    opp = SimpleHeuristicOpponent()
    random.seed(8)
    g = ShogiGame(max_moves_per_game=200)
    for _ in range(60):
        if g.game_over:
            break
        legal = [mapper.shogi_move_to_policy_index(m) for m in g.get_legal_moves()]
        board = np.zeros(81, np.int8)
        for r in range(9):
            for c in range(9):
                p = g.get_piece(r, c)
                board[r * 9 + c] = 0 if p is None else 1 + p.type.value + 14 * p.color.value
        _, members = H.top_tier(board, g.current_player.value, legal)
        move = opp.select_move(g)
        assert mapper.shogi_move_to_policy_index(move) in members
        g.make_move(random.choice(g.get_legal_moves()))
