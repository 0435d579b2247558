"""The one-ply look-ahead opponent without a GPU: the oracle reference (tests/lookahead_ref.c) on positions with known
answers, the argument checks of kz_capture_gain and kz_lookahead_select (which return before any device work) and the
evaluation's player kind."""
import pytest

from shogidrl_b200 import _native as nv
from tests import lookahead_ref

MATE = lookahead_ref.MATE


def test_free_rook_capture():
    # the white rook on 5e attacks the black rook on 5h and nothing defends it: R x 5e gains 10 + 10 and leaves White
    # nothing to take; every move that leaves the rook on the file loses it (-20)
    r = lookahead_ref.lookahead("8k/9/9/9/4r4/9/9/4R4/K8 b - 1")
    assert len(r["scores"]) == 15
    assert r["scores"][10800] == 20 and r["best"] == 20 and r["ties"] == [10800]


def test_defended_capture_scores_below_a_quiet_move():
    # R x 5b takes the gold (6 + 6, promoting +2 more) but the king retakes the rook (10 + 10) or the dragon (12 + 10):
    # -8 either way; quiet moves that keep the rook safe score 0
    r = lookahead_ref.lookahead("4k4/4g4/9/9/9/9/9/4R4/K8 b - 1")
    assert r["scores"][10746] == -8 and r["scores"][10747] == -8
    assert r["best"] == 0 and 10746 not in r["ties"] and 10747 not in r["ties"]
    assert set(r["scores"].values()) == {-20, -8, 0}


def test_promotion_bonus():
    # the silver on 5d promotes on each of its three forward moves into the zone: +1 (6 - 5); the rest gain 0
    r = lookahead_ref.lookahead("8k/9/9/4S4/9/9/9/9/K8 b - 1")
    assert len(r["scores"]) == 11
    assert r["best"] == 1 and r["ties"] == [5003, 5005, 5007]
    assert all(a & 1 for a in r["ties"])


def test_mate_in_one_is_chosen_over_a_capture():
    # G*5b mates; L x 1e would take an undefended silver (5 + 5)
    r = lookahead_ref.lookahead("4k4/9/4P4/9/8s/9/9/9/4K3L b G 1")
    assert r["best"] == MATE and r["ties"] == [13055]
    assert max(s for a, s in r["scores"].items() if a != 13055) == 10


def test_the_one_move_that_does_not_allow_a_mate_in_one():
    # a position from the random golden traces: 47 of Black's 48 legal moves let White mate in one
    r = lookahead_ref.lookahead("1pR4+Nb/l1P1Pp2P/2p1knp2/1ss4pl/p2s1gPG1/n1b1G2P1/lP1g2S2/+n2P+pR2L/+p1K6 b 3P 2")
    assert len(r["scores"]) == 48
    assert sorted(r["scores"].values()).count(-MATE) == 47
    assert r["ties"] == [11014] and r["best"] == -13


def test_every_move_allows_a_mate_in_one():
    # from the endgame golden traces: all six of Black's legal moves tie at -1,000,000
    r = lookahead_ref.lookahead("2l2G+LGp/+P+P2+PS3/2p2+N2+S/1P1P2pk1/plGppp1p1/Ppgs5/4S1P+n1/+p3R1+bB1/+n+p+n+r4K b L 2")
    assert len(r["scores"]) == 6
    assert r["best"] == -MATE and len(r["ties"]) == 6


def test_hirate_every_move_scores_zero():
    r = lookahead_ref.lookahead("lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1")
    assert len(r["scores"]) == 30 and set(r["scores"].values()) == {0}
    assert r["best"] == 0 and len(r["ties"]) == 30


def test_picks_follow_the_random_stream():
    ref = {"ties": lookahead_ref.np.array([0, 1, 3], lookahead_ref.np.int32),
           "tied": lookahead_ref.np.array([[0] * 4, [7, 0, 0, 0], [5, 6, 9, 0]], lookahead_ref.np.uint16)}
    from tests.heuristic_ref import rand32
    got = lookahead_ref.picks(ref, seed=3, step=5, env_offset=10)
    assert got[0] == -1 and got[1] == 7
    assert got[2] == [5, 6, 9][(rand32(3 ^ lookahead_ref.SALT, 12, 5) * 3) >> 32]


def test_capture_gain_rejects_bad_arguments_before_device_work():
    L = nv.lib()
    z, p = None, 1 << 20  # p: an aligned address that is never dereferenced
    b, g = p + (1 << 16), p + (1 << 17)
    assert L.kz_capture_gain(z, 4, 1, b, 448, g, z, z) == -1
    assert L.kz_capture_gain(p, 4, 1, z, 448, g, z, z) == -1
    assert L.kz_capture_gain(p, 4, 1, b, 448, z, z, z) == -1
    for n in (0, -1):
        assert L.kz_capture_gain(p, n, 1, b, 448, g, z, z) == -1
    assert L.kz_capture_gain(p, 4, -1, b, 448, g, z, z) == -1
    assert L.kz_capture_gain(p, 4, 70000, b, 448, g, z, z) == -1
    assert L.kz_capture_gain(p, 4, 1, b, 422, g, z, z) == -1  # short stride
    assert L.kz_capture_gain(p + 16, 4, 1, b, 448, g, z, z) == -1  # misaligned state
    assert L.kz_capture_gain(p, 4, 1, b + 2, 448, g, z, z) == -1  # misaligned rows
    assert L.kz_capture_gain(p, 4, 1, b, 448, g + 2, z, z) == -1  # misaligned gain
    assert L.kz_capture_gain(p, 4, 1, b, 448, g, g + 66, z) == -1  # misaligned count


def test_lookahead_select_rejects_bad_arguments_before_device_work():
    L = nv.lib()
    z, p = None, 1 << 20
    o, it, out = p + (1 << 16), p + (1 << 17), p + (1 << 18)

    def call(state=p, n=4, hist_cap=1, offsets=o, m=8, actions=it, ai64=1, done=it, reason=it, err=it, rg=it, rm=it,
             aout=out, oi64=1, score=z, ties=z):
        return L.kz_lookahead_select(state, n, hist_cap, offsets, m, actions, ai64, done, reason, err, rg, rm, 0, 0, 0,
                                     aout, oi64, score, ties, z)
    assert call(state=z) == -1
    assert call(offsets=z) == -1
    assert call(aout=z) == -1
    assert call(n=0) == -1 and call(n=-1) == -1
    assert call(m=-1) == -1
    assert call(hist_cap=-1) == -1
    assert call(state=p + 16) == -1  # misaligned state
    assert call(offsets=o + 4) == -1  # misaligned offsets
    assert call(aout=out + 4) == -1  # int64 out at a 4-byte address
    assert call(score=out + 2) == -1 and call(ties=out + 2) == -1
    for name in ("actions", "done", "reason", "err", "rg", "rm"):  # per-item arrays are required when m > 0
        assert call(**{name: z}) == -1
    assert call(actions=it + 4) == -1  # int64 actions at a 4-byte address
    assert call(rg=it + 2) == -1 and call(rm=it + 2) == -1


def test_player_kind_accepts_lookahead():
    from shogidrl_b200.evaluation import _player_kind
    assert _player_kind("lookahead") == "lookahead"
    assert _player_kind("heuristic") == "heuristic" and _player_kind(None) == "random"
    with pytest.raises(ValueError, match="lookahead"):
        _player_kind("minimax")


def test_lookahead_actions_refuses_small_chunks():
    from shogidrl_b200 import VecShogiEnv
    env = VecShogiEnv.__new__(VecShogiEnv)  # the check comes before anything touches the device
    with pytest.raises(ValueError, match="max_items"):
        env.lookahead_actions(max_items=1023)
