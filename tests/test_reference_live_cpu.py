"""Live differential checks against the Python reference (tachyon-beep/shogidrl), where a checkout of it is at hand:
SHOGIDRL_REFERENCE names its root.  Skipped without it -- the committed golden fixtures, written by the reference,
stand in.  Fresh seeds every round trip through the same comparisons as the golden tests: oracle vs reference
self-play, the mapper's whole table, SFEN text, ExperienceBuffer host semantics."""
import os
import random
import sys

import numpy as np
import pytest
import torch

REF = os.environ.get("SHOGIDRL_REFERENCE", "")
pytestmark = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "keisei")),
                                reason="reference checkout not present (set SHOGIDRL_REFERENCE)")


@pytest.fixture(scope="module")
def ref():
    sys.dont_write_bytecode = True  # the reference tree is read-only
    if REF not in sys.path:
        sys.path.append(REF)  # appended: must not shadow this repo's `tests` package
    import keisei.shogi as rshogi
    from keisei.core.experience_buffer import ExperienceBuffer as RBuffer
    from keisei.utils import PolicyOutputMapper as RMapper
    return {"shogi": rshogi, "Buffer": RBuffer, "Mapper": RMapper}


def test_mapper_table_identical(ref):
    from shogidrl_b200.utils import PolicyOutputMapper
    ours, theirs = PolicyOutputMapper(), ref["Mapper"]()
    assert ours.get_total_actions() == theirs.get_total_actions() == 13527
    for i in range(13527):
        a, b = ours.policy_index_to_shogi_move(i), theirs.policy_index_to_shogi_move(i)
        assert tuple(getattr(x, "value", x) for x in a) == tuple(getattr(x, "value", x) for x in b), i
    for i in (0, 1, 12959, 12960, 13526):
        assert ours.action_idx_to_usi_move(i) == theirs.action_idx_to_usi_move(i)


def test_oracle_tracks_reference_on_fresh_games(ref):
    """Two short random games with seeds that are not in the fixtures: legal sets, outcomes and observations."""
    from oracle import oracle as orc
    mapper = ref["Mapper"]()
    seed0 = int.from_bytes(os.urandom(2), "little")
    for gi in range(2):
        rng = random.Random(seed0 + gi)
        g = ref["shogi"].ShogiGame(max_moves_per_game=60)
        o = orc.OracleGame(60)
        for ply in range(45):
            want = sorted(mapper.shogi_move_to_policy_index(m) for m in g.get_legal_moves())
            assert o.legal_indices().tolist() == want, (seed0, gi, ply)
            a = want[rng.randrange(len(want))]
            obs, reward, done, info = g.make_move(mapper.policy_index_to_shogi_move(a))
            r2, d2, reason, winner = o.make_move(a)
            assert (reward, done) == (r2, d2) and np.array_equal(obs, o.observation()), (seed0, gi, ply)
            assert orc.parse_sfen(g.to_sfen_string())[0].tolist() == o.export()[0].tolist(), (seed0, gi, ply)
            if done:
                break


def test_sfen_text_identical(ref):
    from shogidrl_b200.shogi.sfen import HostPosition, pack_sfen
    for sfen in ("lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1",
                 "4k4/9/9/9/9/R8/9/9/4K4 b - 1", "9/9/9/9/4K4/9/9/9/4k4 w 2P3p 7",
                 "l2+R2s1l/4gk3/p1n1pp1pp/2pp2p2/9/2P1P4/PP1P1PPPP/1B5R1/LNSGKGSNL w BGSNP 20"):
        b, h, side, mc = pack_sfen(sfen)
        theirs = ref["shogi"].ShogiGame.from_sfen(sfen)
        assert HostPosition(b, h, side, mc).to_sfen_string() == theirs.to_sfen_string()


def test_experience_buffer_host_semantics(ref):
    from shogidrl_b200.core import ExperienceBuffer
    rng = np.random.default_rng(5)
    ours, theirs = ExperienceBuffer(6, 0.99, 0.95, "cpu"), ref["Buffer"](6, 0.99, 0.95, "cpu")
    for i in range(8):  # two more than the capacity: both drop the overflow
        obs = torch.from_numpy(rng.random((46, 9, 9), dtype=np.float32))
        mask = torch.from_numpy(rng.random(13527) < 0.01)
        args = (obs, int(rng.integers(0, 13527)), float(rng.random()), float(-rng.random()), float(rng.random()), bool(i == 3), mask)
        ours.add(*args)
        theirs.add(*args)
    assert len(ours) == len(theirs) == 6 and ours.capacity() == theirs.capacity()
    for name in ("obs", "actions", "rewards", "log_probs", "values", "dones", "legal_masks"):
        assert torch.equal(getattr(ours, name), getattr(theirs, name)), name
    with pytest.raises(RuntimeError) as e1:
        ours.get_batch()
    with pytest.raises(RuntimeError) as e2:
        theirs.get_batch()
    assert str(e1.value) == str(e2.value)
    fmt_o, fmt_t = ours.get_worker_batch_format(), theirs.get_worker_batch_format()
    assert set(fmt_o) == set(fmt_t) and all(torch.equal(fmt_o[k], fmt_t[k]) for k in fmt_t)
    big_o, big_t = ExperienceBuffer(9, 0.99, 0.95, "cpu"), ref["Buffer"](9, 0.99, 0.95, "cpu")
    big_o.add_from_worker_batch(fmt_o)
    big_t.add_from_worker_batch(fmt_t)
    big_o.merge_from_parallel_buffers([ours])
    big_t.merge_from_parallel_buffers([theirs])
    assert big_o.size() == big_t.size() == 9
    for name in ("obs", "actions", "rewards", "log_probs", "values", "dones", "legal_masks"):
        assert torch.equal(getattr(big_o, name), getattr(big_t, name)), name
    ours.clear()
    theirs.clear()
    assert len(ours) == len(theirs) == 0


def test_checkpoint_written_here_resumes_in_the_reference_on_cpu(ref, tmp_path):
    """PPOAgent.save_model writes the reference's checkpoint dictionary (ppo_agent.py:462-487) with the optimizer state
    the reference's own Adam writes -- capturable False, `step` a CPU fp32 tensor -- so the reference's
    PPOAgent.load_model + learn() resumes from it on a CPU-only host (torch's Adam asserts that capturable state lives
    on CUDA).  Built here on CPU with the state laid out the way the fused CUDA tail keeps it."""
    import copy
    from types import SimpleNamespace

    from keisei.core.experience_buffer import ExperienceBuffer as RBuffer
    from keisei.core.neural_network import ActorCritic as RActorCritic
    from keisei.core.ppo_agent import PPOAgent as RAgent

    from shogidrl_b200.core import ActorCritic, PPOAgent
    from tests.helpers import make_config

    cfg = make_config(device="cpu", ppo_epochs=1, minibatch_size=8, steps_per_epoch=8)
    torch.manual_seed(0)
    agent = PPOAgent(ActorCritic(46, 13527), cfg, torch.device("cpu"))
    for p in agent.model.parameters():  # optimizer state as kz_adam_clip_step keeps it: tensors, step as fp32 scalar tensor
        agent.optimizer.state[p] = {"step": torch.tensor(3.0), "exp_avg": torch.full_like(p, 1e-3),
                                    "exp_avg_sq": torch.full_like(p, 1e-6)}
    agent.optimizer.param_groups[0]["capturable"] = True  # what the CUDA agent's optimizer carries
    path = str(tmp_path / "ck.pth")
    agent.save_model(path, 123, 4, {"black_wins": 2, "white_wins": 1, "draws": 1})

    class Cfg(SimpleNamespace):
        def model_copy(self, deep=True):
            return copy.deepcopy(self)

    rcfg = Cfg(env=Cfg(**vars(cfg.env)), training=Cfg(**vars(cfg.training)))
    ragent = RAgent(RActorCritic(46, 13527), rcfg, torch.device("cpu"))
    out = ragent.load_model(path)
    assert out.get("global_timestep") == 123 and out.get("black_wins") == 2 and "error" not in out
    for (k, a), (_, b) in zip(agent.model.state_dict().items(), ragent.model.state_dict().items()):
        assert torch.equal(a, b), k
    assert ragent.optimizer.param_groups[0]["capturable"] is False
    # and the reference trains on from it
    buf = RBuffer(8, 0.99, 0.95, "cpu")
    mask = torch.zeros(13527, dtype=torch.bool)
    mask[:30] = True
    for t in range(8):
        buf.add(torch.rand(46, 9, 9), t, 0.1 * t, -3.0, 0.0, t == 7, mask)
    buf.compute_advantages_and_returns(0.0)
    m = ragent.learn(buf)
    assert all(np.isfinite(v) for v in m.values())
    st = next(iter(ragent.optimizer.state.values()))
    assert float(st["step"]) == 4.0  # continued from the saved step count


def test_oracle_rule_queries_match_the_reference(ref):
    """The oracle's restatements of generate_piece_potential_moves, is_uchi_fu_zume, can_drop_piece and
    get_king_legal_moves -- the checker of tests/test_gpu_api.py::test_rule_queries_match_oracle_on_random_endgames --
    against the reference's own methods on drop-heavy endgames and on the uchifuzume known-answer positions."""
    from oracle import oracle as orc
    from tests.helpers import random_endgames
    rshogi = ref["shogi"]
    Color, PieceType, Piece = rshogi.Color, rshogi.PieceType, rshogi.Piece
    boards, hands, sides, _ = random_endgames(24, 31)
    sfens = ["7gk/9/7GP/9/9/9/9/9/K8 b P 1", "8k/9/8P/9/9/9/9/9/K8 b P 1", "6R1k/9/7G1/9/9/9/9/9/K8 b P 1",
             "k8/9/1G7/9/9/9/9/9/K7R b P 1"]
    cases = [orc.OracleGame.from_arrays(boards[i], hands[i], int(sides[i]), 0, 500, evaluate_termination=False) for i in range(24)]
    cases += [orc.OracleGame.from_sfen(s, evaluate_termination=False) for s in sfens]
    rng = random.Random(3)
    ufz = 0
    for o in cases:
        b, h, m = o.export()
        g = rshogi.ShogiGame()
        g.board = [[None] * 9 for _ in range(9)]
        for sq in range(81):
            if b[sq]:
                g.board[sq // 9][sq % 9] = Piece(PieceType((int(b[sq]) - 1) % 14), Color((int(b[sq]) - 1) // 14))
        for color in (0, 1):
            for t in range(7):
                g.hands[color][PieceType(t)] = int(h[color * 7 + t])
        g.current_player = Color(int(m[0]))
        for sq in range(81):
            p = g.board[sq // 9][sq % 9]
            if p is not None:
                want = np.zeros(81, np.uint8)
                for (r, c) in g.get_individual_piece_moves(p, sq // 9, sq % 9):
                    want[r * 9 + c] = 1
                assert np.array_equal(o.piece_targets(sq), want), sq
        for color in (Color.BLACK, Color.WHITE):
            assert o.king_legal_moves(color.value) == g.get_king_legal_moves(color)
            squares = [rng.randrange(81) for _ in range(4)]
            ek = g.find_king(color.opponent())
            if ek is not None and 0 <= ek[0] + (1 if color == Color.BLACK else -1) < 9:
                squares.append((ek[0] + (1 if color == Color.BLACK else -1)) * 9 + ek[1])
            for sq in squares:
                want = bool(g.is_uchi_fu_zume(sq // 9, sq % 9, color))
                assert o.is_uchi_fu_zume(sq, color.value) == want, (sq, color)
                ufz += int(want)
                for t in range(7):
                    assert o.can_drop(t, sq, color.value) == bool(g.can_drop_piece(PieceType(t), sq // 9, sq % 9, color)), (t, sq)
    assert ufz >= 1  # the known-answer uchifuzume position is among the cases


def test_move_descriptions_identical(ref):
    """shogidrl_b200.utils.move_formatting writes the reference's demo-log strings (keisei/utils/move_formatting.py):
    every board move and drop of the 13,527-entry table, with and without the piece, promotions and odd inputs."""
    import keisei.utils.move_formatting as rmf
    from keisei.shogi.shogi_core_definitions import Color as RColor, Piece as RPiece, PieceType as RPT
    from keisei.utils import PolicyOutputMapper as RefMapper
    import shogidrl_b200.utils.move_formatting as mf
    from shogidrl_b200.shogi.definitions import Color, Piece, PieceType
    from shogidrl_b200.utils import PolicyOutputMapper

    rmap, omap = RefMapper(), PolicyOutputMapper()
    rng = random.Random(5)
    for idx in rng.sample(range(13527), 1500):
        rmove, omove = rmap.policy_index_to_shogi_move(idx), omap.policy_index_to_shogi_move(idx)
        assert rmf.format_move_with_description(rmove, rmap) == mf.format_move_with_description(omove, omap)
        assert rmf.format_move_with_description_enhanced(rmove, rmap, None) == \
            mf.format_move_with_description_enhanced(omove, omap, None)
        v = rng.randrange(14)
        assert rmf.format_move_with_description_enhanced(rmove, rmap, RPiece(RPT(v), RColor.BLACK)) == \
            mf.format_move_with_description_enhanced(omove, omap, Piece(PieceType(v), Color.BLACK))
    for v in range(14):
        for promo in (False, True):
            assert rmf._get_piece_name(RPT(v), promo) == mf._get_piece_name(PieceType(v), promo)
    assert rmf.format_move_with_description(None, rmap) == mf.format_move_with_description(None, omap) == "None"
    assert rmf.format_move_with_description_enhanced(None, rmap) == mf.format_move_with_description_enhanced(None, omap)
    assert [rmf._coords_to_square_name(r, c) for r in range(9) for c in range(9)] == \
        [mf._coords_to_square_name(r, c) for r in range(9) for c in range(9)]
