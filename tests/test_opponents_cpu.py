"""The reference's scripted opponents (keisei/utils/opponents.py) without a GPU: the tier rule restated over policy
indices (tests/heuristic_ref.py) on every position of the golden traces, with the legal sets the reference itself
wrote, and the scalar reference-API classes (shogidrl_b200.utils.opponents) on duck-typed games built from the CPU
oracle.  A live comparison with the reference's own classes runs where its checkout is at hand (SHOGIDRL_REFERENCE)."""
import os
import random
import sys
from unittest import mock

import numpy as np
import pytest

from oracle import oracle as orc  # checker only
from shogidrl_b200.shogi.definitions import Color, Piece
from shogidrl_b200.utils import BaseOpponent, SimpleHeuristicOpponent, SimpleRandomOpponent
from tests import heuristic_ref as H


@pytest.fixture(scope="module")
def positions(golden_dir):
    return H.fixture_positions(golden_dir)


class OracleDuckGame:
    """The three members the scripted opponents read, over an oracle game: legal moves as MoveTuples in ascending
    index order (index_to_move), pieces decoded from the exported board."""

    def __init__(self, g):
        b, _, m = g.export()
        self._board = b
        self.current_player = Color(int(m[0]))
        self.legal = [int(a) for a in g.legal_indices()]

    def get_legal_moves(self):
        return [orc.index_to_move(a) for a in self.legal]

    def get_piece(self, r, c):
        return Piece.from_code(int(self._board[r * 9 + c]))


def _game(P, i):
    return orc.OracleGame.from_arrays(P["boards"][i], P["hands"][i], P["sides"][i], P["move_counts"][i], 500,
                                      evaluate_termination=False)


def test_rand32_restatement_matches_oracle():
    for seed, env, step in [(0, 0, 0), (1234, 7, 3), (2**63 + 5, 65535, 2**31 + 1), (H.MASK64, 2**32 - 1, 2**32 - 1)]:
        assert H.rand32(seed, env, step) == orc.rand32(seed, env, step)


def test_fixture_positions_reproduce_the_reference_legal_sets(positions):
    """The positions rebuilt from the traces are the ones the reference played from: the oracle generates exactly the
    legal set the reference recorded for each of them."""
    P = positions
    assert len(P["legal"]) == 25200 + 5920
    for i in range(len(P["legal"])):
        assert np.array_equal(_game(P, i).legal_indices(), P["legal"][i].astype(np.int32)), i


def test_tiers_on_the_reference_legal_sets(positions):
    """Every ply of both traces classified; all three tiers occur as the top tier (the frequencies are printed)."""
    P = positions
    top = np.zeros((2, 4), np.int64)  # [source][capture, pawn, other, none]
    for i, legal in enumerate(P["legal"]):
        t = H.tiers(P["boards"][i], int(P["sides"][i]), legal)
        assert sum(len(x) for x in t) == len(legal)
        for a in t[0] + t[1]:  # board moves only, and never onto an own piece
            frm, r = divmod(a >> 1, 80)
            to = r + (r >= frm)
            dest = int(P["boards"][i][to])
            assert a < 12960 and (dest == 0 or (dest >= 15) != bool(P["sides"][i])), (i, a)
        tier, members = H.top_tier(P["boards"][i], int(P["sides"][i]), legal)
        top[P["source"][i], min(tier, 3)] += 1
    print("top tier (capture, pawn, other, none): random traces", top[0].tolist(), "endgames", top[1].tolist())
    assert (top.sum(0)[:3] > 0).all() and top.sum() == len(P["legal"])


def test_scalar_heuristic_picks_random_choice_of_the_top_tier(positions):
    """SimpleHeuristicOpponent.select_move hands random.choice exactly the top tier, in the game's list order, and
    returns what random.choice returns under the same random state."""
    P = positions
    opp = SimpleHeuristicOpponent()
    assert isinstance(opp, BaseOpponent) and opp.name == "SimpleHeuristicOpponent"
    for i in range(0, len(P["legal"]), 5):
        g = OracleDuckGame(_game(P, i))
        _, members = H.top_tier(P["boards"][i], int(P["sides"][i]), g.legal)
        want_list = [orc.index_to_move(a) for a in members]
        seen = []
        real_choice = random.choice
        with mock.patch("random.choice", side_effect=lambda seq: (seen.append(list(seq)), real_choice(seq))[1]):
            random.seed(i)
            got = opp.select_move(g)
        assert seen == [want_list], i
        random.seed(i)
        assert got == random.choice(want_list), i


def test_scalar_random_opponent_returns_a_legal_move(positions):
    P = positions
    opp = SimpleRandomOpponent()
    random.seed(5)
    for i in range(0, len(P["legal"]), 97):
        g = OracleDuckGame(_game(P, i))
        assert opp.select_move(g) in g.get_legal_moves()


def test_no_legal_moves_raise_value_error():
    class NoMoves:
        current_player = Color.BLACK

        def get_legal_moves(self):
            return []

        def get_piece(self, r, c):
            return None

    for cls in (SimpleRandomOpponent, SimpleHeuristicOpponent):
        with pytest.raises(ValueError, match="No legal moves available"):
            cls().select_move(NoMoves())


REF = os.environ.get("SHOGIDRL_REFERENCE", "")


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "keisei")),
                    reason="reference checkout not present (set SHOGIDRL_REFERENCE)")
def test_live_against_the_reference_opponents():
    """On fresh random reference games: the reference's SimpleHeuristicOpponent and ours hand random.choice the same
    candidates (as sets) and return the same move under the same random state; the error strings agree."""
    sys.dont_write_bytecode = True  # the reference tree is read-only
    if REF not in sys.path:
        sys.path.append(REF)  # appended: must not shadow this repository's `tests` package
    from keisei.shogi import ShogiGame as RGame
    from keisei.utils import opponents as ropp

    rng = random.Random(int.from_bytes(os.urandom(2), "little"))
    ours = {"h": SimpleHeuristicOpponent(), "r": SimpleRandomOpponent()}
    theirs = {"h": ropp.SimpleHeuristicOpponent(), "r": ropp.SimpleRandomOpponent()}
    real_choice = random.choice
    for _ in range(3):
        g = RGame(max_moves_per_game=200)
        while not g.game_over and g.move_count < 200:
            for k in ("h", "r"):
                cands = []
                with mock.patch("random.choice", side_effect=lambda seq: (cands.append(list(seq)), real_choice(seq))[1]):
                    state = rng.getrandbits(32)
                    random.seed(state)
                    m_ref = theirs[k].select_move(g)
                    random.seed(state)
                    m_ours = ours[k].select_move(g)
                assert len(cands) == 2 and set(cands[0]) == set(cands[1]) and cands[0] == cands[1]
                assert m_ref == m_ours
            g.make_move(real_choice(g.get_legal_moves()))

    class NoMoves:
        def get_legal_moves(self):
            return []

    for k in ("h", "r"):
        with pytest.raises(ValueError) as e_ref:
            theirs[k].select_move(NoMoves())
        with pytest.raises(ValueError) as e_ours:
            ours[k].select_move(NoMoves())
        assert str(e_ref.value) == str(e_ours.value)
