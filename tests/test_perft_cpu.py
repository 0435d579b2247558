"""perft without a GPU: the oracle generator's move-tree counts (tests/perft_ref.c) against the published hirate values and
against a Python recursion over OracleGame, and perft()'s argument checks (which run before any device is touched)."""
import os

import numpy as np
import pytest

from oracle import oracle as orc  # checker only
from tests import perft_ref

HIRATE = [1, 30, 900, 25470, 719731]  # published perft counts of the start position, depths 0..4


@pytest.mark.parametrize("depth", [0, 1, 2, 3, 4])
def test_oracle_perft_hirate(depth):
    assert perft_ref.perft(None, depth) == HIRATE[depth]


def _perft_py(g: orc.OracleGame, depth: int) -> int:
    """Move-tree perft by recursion over make_move on fresh games (export / from_arrays: no history, no termination)."""
    if depth == 0:
        return 1
    total = 0
    b, h, m = g.export()
    for a in g.legal_indices():
        c = orc.OracleGame.from_arrays(b, h, int(m[0]), int(m[1]), 65535, evaluate_termination=False)
        c.make_move(int(a))
        nb, nh, nm = c.export()
        total += _perft_py(orc.OracleGame.from_arrays(nb, nh, int(nm[0]), int(nm[1]), 65535, evaluate_termination=False),
                           depth - 1)
    return total


def test_oracle_perft_divide_matches_python_recursion(golden_dir):
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as zf:
        sfens = [str(s) for s in zf["sfens"]]
    assert len(sfens) == 38
    for s in sfens:
        g = orc.OracleGame.from_sfen(s, max_moves=65535, evaluate_termination=False)
        div = perft_ref.perft(s, 2, divide=True)
        assert sorted(div) == g.legal_indices().tolist(), s
        b, h, m = g.export()
        for a, k in div.items():
            c = orc.OracleGame.from_arrays(b, h, int(m[0]), int(m[1]), 65535, evaluate_termination=False)
            c.make_move(a)
            nb, nh, nm = c.export()
            child = orc.OracleGame.from_arrays(nb, nh, int(nm[0]), int(nm[1]), 65535, evaluate_termination=False)
            assert k == len(child.legal_indices()), (s, a)
        assert sum(div.values()) == _perft_py(g, 2) == perft_ref.perft(s, 2), s


def test_perft_argument_checks():
    from shogidrl_b200.perft import perft
    with pytest.raises(ValueError, match="depth"):
        perft(depth=-1)
    with pytest.raises(ValueError, match="depth"):
        perft()
    with pytest.raises(ValueError, match="does not parse"):
        perft(["lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNX b - 1"], 2)
    with pytest.raises(ValueError, match="does not parse"):
        perft("not a position", 1)
    assert perft(depth=0) == [1]
    assert perft(["4k4/9/9/9/9/9/9/9/4K4 b - 1"] * 2, 0, divide=True) == [{}, {}]


def test_chunks_of_whole_games():
    """The chunking perft and the look-ahead opponent share: consecutive games of at most max_items items, a game above
    the limit alone, and no chunk without items."""
    from shogidrl_b200._batch import chunks

    def off(counts):
        return np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    assert chunks(off([]), 4) == []
    assert chunks(off([0, 0, 0]), 4) == []  # empty games only
    assert chunks(off([0, 2, 0, 2, 0]), 4) == [(0, 5)]  # an exact fit, with the empty games around it
    assert chunks(off([2, 2, 2, 2, 0]), 4) == [(0, 2), (2, 5)]
    assert chunks(off([2, 3, 4]), 4) == [(0, 1), (1, 2), (2, 3)]
    assert chunks(off([1, 9, 1]), 4) == [(0, 1), (1, 2), (2, 3)]  # a game above the limit is a chunk of its own
    assert chunks(off([0, 9]), 4) == [(1, 2)]  # an empty game before a large one is a chunk without items
