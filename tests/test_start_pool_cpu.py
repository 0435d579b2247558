"""Start-position pools without a GPU: SFEN validation before any device call, the even-num_games rule of paired
evaluation, and the paired opening schedule against a plain restatement."""
import pytest
import torch

from shogidrl_b200.evaluation import _num_envs, evaluate_vs_opponent, paired_openings
from shogidrl_b200.vec_env import parse_start_positions

HIRATE = "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"


def test_parse_accepts_and_packs():
    b, h, s, mc = parse_start_positions([HIRATE, "4k4/9/9/9/9/9/9/9/4K4 w 2P 31"], 500)
    assert b.shape == (2, 81) and h.shape == (2, 14)
    assert s.tolist() == [0, 1] and mc.tolist() == [0, 30]
    assert int(h[1, 0]) == 2 and int(b[1, 76]) == 8 and int(b[1, 4]) == 22


@pytest.mark.parametrize("sfens, index, what", [
    (["not a sfen"], 0, "does not parse"),
    ([HIRATE, HIRATE, "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL x - 1"], 2, "does not parse"),
    ([HIRATE, "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 0"], 1, "does not parse"),
    ([HIRATE, "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 81"], 1, "terminal at load"),
])
def test_parse_errors_name_the_index(sfens, index, what):
    with pytest.raises(ValueError, match=rf"start position {index} .*{what}"):
        parse_start_positions(sfens, 80)


def test_parse_rejects_a_bare_string_and_an_empty_pool():
    with pytest.raises(ValueError, match="one string"):
        parse_start_positions(HIRATE, 500)
    with pytest.raises(ValueError, match="empty"):
        parse_start_positions([], 500)


def test_paired_evaluation_needs_an_even_number_of_games():
    # rejected before any environment (or device) exists
    with pytest.raises(ValueError, match="must be even"):
        evaluate_vs_opponent("random", 7, start_positions=[HIRATE], device="cpu")


@pytest.mark.parametrize("num_games, num_envs, paired, want", [
    (128, 1024, True, 128), (128, 1, True, 2), (128, 3, True, 2), (128, 7, True, 6), (2, 1, True, 2), (0, 16, True, 2),
    (128, 1, False, 1), (7, 1024, False, 7), (7, 3, False, 3), (1, 16, False, 2),
])
def test_evaluation_env_count(num_games, num_envs, paired, want):
    assert _num_envs(num_games, num_envs, paired) == want


@pytest.mark.parametrize("n, pool_size", [(2, 1), (8, 3), (128, 64), (16, 5), (1024, 129)])
def test_paired_schedule_matches_restatement(n, pool_size):
    g = torch.Generator().manual_seed(n * 1000 + pool_size)
    begun = torch.randint(0, 9, (n,), generator=g)
    got = paired_openings(begun, pool_size)
    assert got.dtype == torch.int32
    for e in range(n):
        i, j = e // 2, int(begun[e])
        assert int(got[e]) == (i + (n // 2) * j) % pool_size


def test_paired_schedule_plays_every_opening_from_both_sides():
    # 64 openings, 128 games on 128 envs (one game each): every (opening, colour) exactly once
    n, pool = 128, 64
    first = paired_openings(torch.zeros(n, dtype=torch.int64), pool).tolist()
    black = sorted(first[0::2])  # envs 2i: the agent plays Black
    white = sorted(first[1::2])
    assert black == list(range(pool)) and white == list(range(pool))
    assert first[0::2] == first[1::2]
    # four games per env on 32 envs (16 pairs): the pairs walk through the pool side by side
    n = 32
    seen = [paired_openings(torch.full((n,), j, dtype=torch.int64), pool).tolist() for j in range(4)]
    assert sorted(sum((s[0::2] for s in seen), [])) == list(range(pool))
    assert all(s[0::2] == s[1::2] for s in seen)
