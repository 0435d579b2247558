"""Start-position pools on the device: the records against the load path, a bit-for-bit replay of pooled self-play on the
CPU oracle (mask form, rollout form, two step ranges), the selection rules, validation, CUDA-graph rollouts and paired
evaluation."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests.helpers import make_config  # noqa: E402

HIRATE = "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"
MASK64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def pool_sfens(golden_dir):
    """128 drop-heavy endgames + 12 stalemate-trace starts + hirate."""
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as z:
        eg = [str(s) for s in z["sfens"]]
    with np.load(os.path.join(golden_dir, "traces_stalemate.npz")) as z:
        st = [str(s) for s in z["sfens"]]
    return eg + st + [HIRATE]


def _mulhi(r: int, n: int) -> int:
    return (r * n) >> 32


def _state_rows(env):
    """(boards [n, 96], meta [n, 32]) bytes of the env's state blob."""
    n = env.n
    return env.state[: 96 * n].view(n, 96), env.state[96 * n: 128 * n].view(n, 32)


def test_pool_records_equal_the_load_path(pool_sfens):
    from shogidrl_b200 import VecShogiEnv
    P = len(pool_sfens)
    env = VecShogiEnv(8, max_moves_per_game=500, seed=3, start_positions=pool_sfens)
    rec = env.pool.cpu().numpy().view(np.uint32)
    assert rec.shape == (P, 512)
    ref = VecShogiEnv(P, max_moves_per_game=500, seed=3)
    ref.load_sfens(pool_sfens)
    in_check = torch.zeros(P, dtype=torch.uint8, device=ref.device)
    ref.refresh(in_check=in_check)
    count = ref.legal_count.clone()
    bitmap = torch.zeros((P, 448), dtype=torch.int32, device=ref.device)
    ref.legal_bitmap(bitmap)
    b, h, m = [x.cpu().numpy() for x in ref.export()]
    boards, meta = [x.cpu().numpy() for x in _state_rows(ref)]
    rb = rec[:, :24].copy().view(np.uint8)
    rm = rec[:, 24:32].copy().view(np.uint8)
    assert np.array_equal(rb[:, :81].view(np.int8), b)
    assert np.array_equal(rb[:, 84:96], boards[:, 84:96])  # key words x, y, z
    assert np.array_equal(rm[:, 28:32], meta[:, 28:32])  # key word w
    assert np.array_equal(rm[:, :14], h)
    assert np.array_equal(rm[:, 14], m[:, 0])
    assert np.array_equal(rm[:, 18].astype(np.int32) | (rm[:, 19].astype(np.int32) << 8), m[:, 1])
    assert (rm[:, 15] == 0).all() and (rm[:, 16] == 0xFF).all() and (rm[:, 17] == 0).all()
    assert np.array_equal(rec[:, 64:], bitmap.cpu().numpy().view(np.uint32))
    assert np.array_equal(rec[:, 32].astype(np.int32), count.cpu().numpy())
    assert np.array_equal(rec[:, 33], in_check.cpu().numpy().astype(np.uint32))
    assert (rec[:, 34:64] == 0).all()


def _replay_on_oracle(pool_sfens, seed, n, T, max_moves, rec, salt, reset_salt):
    """Per-env CPU replay of pooled random self-play: returns the per-step traces and the final oracle games."""
    packed = [orc.parse_sfen(s) for s in pool_sfens]
    P = len(packed)
    games, sid, eps = [], np.zeros(n, np.int64), np.zeros(n, np.int64)
    load = lambda k: orc.OracleGame.from_arrays(*packed[k][:2], packed[k][2], packed[k][3], max_moves)  # noqa: E731
    for g in range(n):
        k = _mulhi(orc.rand32((seed ^ reset_salt) & MASK64, g, 0), P)
        sid[g] = k
        games.append(load(k))
    assert np.array_equal(sid, rec["start0"]), "initial pool draws differ"
    assert np.array_equal(np.array([gm.pick_action(seed, g, 0) for g, gm in enumerate(games)]), rec["next0"])
    for t in range(T):
        s = t + 1
        for g in range(n):
            gm = games[g]
            a = int(rec["actions"][t, g])
            r, done, reason, winner = gm.make_move(a)
            ep_len = int(gm.meta[1]) if done else 0
            if done:
                eps[g] += 1
                k = _mulhi(orc.rand32((seed ^ salt) & MASK64, g, int(eps[g])), P)
                sid[g] = k
                gm = games[g] = load(k)
            got = (rec["reward"][t, g], rec["done"][t, g], rec["reason"][t, g], rec["winner"][t, g], rec["ep_len"][t, g],
                   rec["legal"][t, g], rec["next"][t, g], rec["sid"][t, g])
            want = (r, int(done), reason, winner, ep_len, len(gm.legal_indices()), gm.pick_action(seed, g, s), sid[g])
            assert tuple(float(x) for x in got) == tuple(float(x) for x in want), (t, g, got, want)
    return games


def test_pooled_selfplay_replays_on_the_oracle(pool_sfens):
    """~1,000 envs x 400 plies with max_moves 80 (every env restarts several times) from a 141-entry pool, fused random
    actions: the mask form is replayed step by step on the CPU oracle; the rollout form (bitmap + compact observation)
    and a two-range launch (step_streams = 2) give exactly the mask form's results at every step."""
    from shogidrl_b200 import VecShogiEnv, rl
    n, T, mm, seed = 1024, 400, 80, 77
    A = VecShogiEnv(n, max_moves_per_game=mm, seed=seed, start_positions=pool_sfens)
    B = VecShogiEnv(n, max_moves_per_game=mm, seed=seed, start_positions=pool_sfens)
    Cs = VecShogiEnv(n, max_moves_per_game=mm, seed=seed, start_positions=pool_sfens, step_streams=2)
    assert Cs.step_streams == 2
    dev = A.device
    for e in (A, B, Cs):
        e.refresh(random_actions=True)
    rec = {"start0": A.start_ids.cpu().numpy().copy(), "next0": A.next_actions.cpu().numpy().copy()}
    assert torch.equal(B.start_ids, A.start_ids) and torch.equal(Cs.start_ids, A.start_ids)
    bm = torch.zeros((n, 448), dtype=torch.int32, device=dev)
    cobs = torch.zeros((n, 40), dtype=torch.int32, device=dev)
    obs_b = torch.zeros((n, 46, 9, 9), device=dev)
    ref_bm = torch.zeros_like(bm)
    ref_cobs = torch.zeros_like(cobs)
    nb = B.next_actions.clone()
    keys = ["actions", "reward", "done", "reason", "winner", "ep_len", "legal", "next", "sid"]
    trace = {k: [] for k in keys}
    resets = 0
    for t in range(T):
        a = A.next_actions.clone()
        oa = A.step(a, random_actions=True)
        row = [a, oa["reward"], oa["done"], oa["reason"], oa["winner"], oa["ep_len"], oa["legal_count"], A.next_actions,
               A.start_ids]
        for k, v in zip(keys, row):
            trace[k].append(v.clone())
        resets += int(oa["done"].sum())
        ob = B.step_rollout(a, obs_b, bm, random_actions=True, next_out=nb, cobs=cobs)
        oc = Cs.step(a, random_actions=True)
        for o in (ob, oc):
            for k in ("reward", "done", "reason", "winner", "ep_len", "legal_count"):
                assert torch.equal(o[k], oa[k]), (t, k)
        assert torch.equal(nb, A.next_actions) and torch.equal(Cs.next_actions, A.next_actions), t
        assert torch.equal(B.start_ids, A.start_ids) and torch.equal(Cs.start_ids, A.start_ids), t
        assert torch.equal(obs_b, A.obs) and torch.equal(Cs.obs, A.obs) and torch.equal(Cs.mask, A.mask), t
        assert torch.equal(rl.bitmap_to_mask(bm).view(torch.uint8), A.mask), t
        A.legal_bitmap(ref_bm, cobs=ref_cobs)  # the refresh path's rows of the same positions
        assert torch.equal(bm, ref_bm) and torch.equal(cobs, ref_cobs), t
    assert resets > 2 * n, resets  # several restarts per env
    rec.update({k: torch.stack(v).cpu().numpy() for k, v in trace.items()})
    games = _replay_on_oracle(pool_sfens, seed, n, T, mm, rec, A.POOL_SALT, A.POOL_RESET_SALT)
    b, h, m = [x.cpu().numpy() for x in A.export()]
    obs, mask = A.obs.cpu().numpy(), A.mask.cpu().numpy()
    for g, gm in enumerate(games):
        ob_, oh, om = gm.export()
        assert np.array_equal(b[g], ob_) and np.array_equal(h[g], oh) and m[g, 0] == om[0] and m[g, 1] == om[1], g
        assert np.array_equal(obs[g], gm.observation()) and np.array_equal(mask[g], gm.legal_mask()), g
    assert (A.errors() == 0).all()


def test_explicit_start_pick_is_honoured(pool_sfens):
    from shogidrl_b200 import VecShogiEnv
    n, P = 256, len(pool_sfens)
    env = VecShogiEnv(n, max_moves_per_game=60, seed=5, start_positions=pool_sfens)
    pick = ((torch.arange(n, device=env.device) * 7 + 3) % P).to(torch.int32)
    env.reset(start_pick=pick)
    assert torch.equal(env.start_ids, pick)
    want = [pool_sfens[int(k)] for k in pick.tolist()]
    ref = VecShogiEnv(n, max_moves_per_game=60, seed=5)
    ref.load_sfens(want)
    (b, h, m), (rb, rh, rm) = env.export(), ref.export()
    assert torch.equal(b, rb) and torch.equal(h, rh) and torch.equal(m[:, :7], rm[:, :7])
    assert torch.equal(env.obs, ref.obs) and torch.equal(env.mask, ref.mask)
    # auto-reset inside the step: games that finish restart from pick2
    pick2 = ((torch.arange(n, device=env.device) * 11 + 1) % P).to(torch.int32)
    env.refresh(random_actions=True)
    restarted = torch.zeros(n, dtype=torch.bool, device=env.device)
    for _ in range(70):
        before = env.start_ids.clone()
        out = env.step(env.next_actions.clone(), random_actions=True, start_pick=pick2)
        d = out["done"] != 0
        assert torch.equal(env.start_ids[d], pick2[d]) and torch.equal(env.start_ids[~d], before[~d])
        restarted |= d
    assert bool(restarted.all())  # max_moves 60: every game has finished by ply 70
    with pytest.raises(ValueError, match="start_pick"):
        env.step(env.next_actions.clone(), random_actions=True, start_pick=pick2.long())


def test_pool_draws_are_uniform(golden_dir):
    from scipy.stats import chisquare
    from shogidrl_b200 import VecShogiEnv
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as z:
        sfens = [" ".join(str(s).split()[:3] + ["1"]) for s in z["sfens"][:16]]
    n = 8192
    env = VecShogiEnv(n, max_moves_per_game=2, seed=11, start_positions=sfens)  # every game ends after two plies
    env.refresh(random_actions=True)
    counts = torch.zeros(16, dtype=torch.int64, device=env.device)
    for _ in range(8):
        out = env.step(env.next_actions.clone(), random_actions=True)
        d = out["done"] != 0
        counts += torch.bincount(env.start_ids[d].long(), minlength=16)
    c = counts.cpu().numpy()
    assert c.sum() >= 20000, c.sum()
    assert chisquare(c).pvalue > 1e-3, c


def test_validation_rejects_terminal_and_king_capture_entries(golden_dir):
    from shogidrl_b200 import VecShogiEnv
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as z:
        mated = [str(s) for s, g, r in zip(z["sfens"], z["game_over"], z["reason"]) if g and r == 1]
    assert mated
    env = VecShogiEnv(8, max_moves_per_game=500, seed=1)
    for s in mated:
        with pytest.raises(ValueError, match="start position 1 is terminal"):
            env.set_start_positions([HIRATE, s])
    with pytest.raises(ValueError, match="start position 2 lets the side to move capture"):
        env.set_start_positions([HIRATE, HIRATE, "4k4/9/9/9/9/9/9/4R4/4K4 b - 1"])
    assert env.pool is None  # a rejected pool leaves the env as it was
    with pytest.raises(ValueError, match="start position 0 .*does not parse"):
        env.set_start_positions(["4k4/9/9/9/9/9/9/4R4/4K4 q - 1"])
    env.set_start_positions([HIRATE], reset=True)
    assert (env.start_ids == 0).all()
    env.set_start_positions(None)
    assert (env.start_ids == 0).all()  # the games in progress started from entry 0 of the pool that was set
    env.reset()
    assert (env.start_ids == -1).all()


def test_start_ids_across_pool_changes_and_start_pick_needs_auto_reset():
    from shogidrl_b200 import VecShogiEnv
    n = 64
    env = VecShogiEnv(n, max_moves_per_game=30, seed=9, start_positions=[HIRATE, HIRATE])
    env.refresh(random_actions=True)
    ids = env.start_ids.clone()
    assert ((ids == 0) | (ids == 1)).all()
    env.set_start_positions(None)
    restarted = torch.zeros(n, dtype=torch.bool, device=env.device)
    for _ in range(40):  # max_moves 30: every game finishes once and restarts from the start position
        d = env.step(env.next_actions.clone(), random_actions=True)["done"] != 0
        restarted |= d
        assert torch.equal(env.start_ids[~restarted], ids[~restarted]) and (env.start_ids[restarted] == -1).all()
    assert bool(restarted.all())
    fixed = VecShogiEnv(8, max_moves_per_game=30, seed=9, auto_reset=False, start_positions=[HIRATE])
    with pytest.raises(ValueError, match="auto_reset=False"):
        fixed.step(fixed.next_actions.clone(), start_pick=torch.zeros(8, dtype=torch.int32, device=fixed.device))
    fixed.reset(start_pick=torch.zeros(8, dtype=torch.int32, device=fixed.device))
    assert (fixed.start_ids == 0).all()


def _trainer(sfens, graph: bool, seed: int = 42):
    from shogidrl_b200.core import ActorCritic
    from shogidrl_b200.training.selfplay import SelfPlayTrainer
    cfg = make_config(cuda_graph_rollout=graph)
    cfg.env.max_moves_per_game = 24  # above every pool entry's move number (at most 18): short games, many restarts
    torch.manual_seed(seed)
    return SelfPlayTrainer(ActorCritic(46, 13527), cfg, 256, 16, "cuda", start_positions=sfens)


def test_graphed_rollout_draws_fresh_starts_and_equals_eager(pool_sfens):
    G, E = _trainer(pool_sfens, True), _trainer(pool_sfens, False)
    E.agent.model.load_state_dict(G.agent.model.state_dict())
    T = G.buffer.T
    seen = []
    for i in range(3):
        if i == 2:
            E.env.step_index = T  # the replayed graph repeats the rng_step values it was captured with
        for tr in (G, E):
            tr.collect()
            tr.buffer.clear()
        assert (G.driver._graph is not None) == (i >= 1)
        for k in ("actions", "rewards", "dones"):
            assert torch.equal(getattr(G.buffer, k), getattr(E.buffer, k)), (i, k)
        assert torch.equal(G.env.start_ids, E.env.start_ids), i
        assert torch.equal(G.env.state[:-256], E.env.state[:-256]), i  # all but the launch scheduling words
        seen.append(G.env.start_ids.clone())
    assert not torch.equal(seen[1], seen[2])  # two replays of one graph, different starts
    # a new pool: the graph (which names the old one) is dropped and recaptured
    G.set_start_positions(pool_sfens[:16])
    assert G.driver._graph is None
    G.collect()
    G.buffer.clear()
    assert G.driver._graph is not None and G.driver._graph_pool == (G.env.pool.data_ptr(), 16)


class _Lowest:
    """Deterministic agent: the legal move with the lowest (or highest) policy index; records the first observations."""

    def __init__(self, highest=False):
        self.highest, self.first_obs, self.paired = highest, None, []

    def select_actions(self, obs, mask, is_training=False):
        if self.first_obs is None:
            self.first_obs = obs.clone()
        self.paired.append(bool(torch.equal(obs[0::2], obs[0:1].expand_as(obs[0::2])) and
                                torch.equal(obs[1::2], obs[1:2].expand_as(obs[1::2]))))
        m = mask.bool()
        idx = torch.arange(m.shape[1], device=m.device)
        score = torch.where(m, idx if self.highest else -idx, torch.iinfo(torch.int64).min)
        return (score.argmax(1),)


def test_evaluation_without_a_pool_repeats_two_games():
    from shogidrl_b200.evaluation import evaluate_vs_opponent
    a, b = _Lowest(), _Lowest(highest=True)
    r = evaluate_vs_opponent(a, 32, opponent=b, num_envs=16, max_moves_per_game=40)
    assert r.games == 32 and r.start_ids == []
    assert all(a.paired)  # every even env plays env 0's game, every odd env env 1's: two distinct games in all


def test_paired_evaluation_plays_every_opening_from_both_sides(pool_sfens):
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200.evaluation import evaluate_vs_opponent
    openings = pool_sfens[:64]
    runs = []
    for _ in range(2):
        a, b = _Lowest(), _Lowest(highest=True)
        r = evaluate_vs_opponent(a, 128, opponent=b, num_envs=1024, max_moves_per_game=60, start_positions=openings)
        runs.append((r, a))
    r, a = runs[0]
    assert r.games == 128 and len(r.start_ids) == len(r.outcomes) == 128
    assert sorted(r.start_ids) == sorted(list(range(64)) * 2)
    ref = VecShogiEnv(128, max_moves_per_game=60, seed=0)
    ref.load_sfens([openings[e // 2] for e in range(128)])  # env 2i (agent Black) and 2i+1 (agent White): opening i
    assert torch.equal(a.first_obs, ref.obs)
    r2 = runs[1][0]
    assert (r2.outcomes, r2.start_ids, r2.agent_wins, r2.draws) == (r.outcomes, r.start_ids, r.agent_wins, r.draws)
    assert not all(a.paired)
