"""Checking moves and mates in one without a GPU: the oracle reference (tests/checks_ref.c) on known positions,
kz_check_bitmap's argument checks (which return before any device work) and the host batching of evaluate_mate_in_one."""
import pytest

from shogidrl_b200 import _native as nv
from tests import checks_ref

# sfen, legal moves, checking moves, mates (that do not capture a king), "mates" that capture the king, enemy in check
TABLE = [
    ("lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1", 30, 0, [], [], False),
    ("4k4/9/4P4/9/9/9/9/9/4K4 b G 1", 85, 7, [13055], [], False),  # head gold: G*5b
    ("7nk/9/8G/9/9/9/9/9/4K4 b P 1", 78, 2, [], [], False),  # P*1b would mate but is uchifuzume, so not legal
    ("3gkg3/9/3PSP3/9/4R4/9/9/9/4K4 b - 1", 31, 12, [3544, 3545, 3548, 3549], [], False),  # discovered / double checks
    ("9/9/9/9/9/9/9/9/4K4 b G 1", 85, 85, None, [], True),  # enemy king missing: every move "checks" and "mates"
    ("4k4/9/9/9/4R4/9/9/9/4K4 b - 1", 23, 15, [], [6408, 6409], True),  # enemy already in check (out of contract)
]


@pytest.mark.parametrize("sfen,legal,checks,mates,kc,eic", TABLE)
def test_reference_fixture_positions(sfen, legal, checks, mates, kc, eic):
    r = checks_ref.checks(sfen)
    assert len(r["legal"]) == legal
    assert len(r["checks"]) == checks
    assert r["mates"] == (r["legal"] if mates is None else mates)
    assert r["king_capture_mates"] == kc
    assert r["enemy_in_check"] == eic
    assert set(r["checks"]) <= set(r["legal"])


def test_reference_classes():
    r = checks_ref.checks("3gkg3/9/3PSP3/9/4R4/9/9/9/4K4 b - 1")
    kinds = set(r["classes"].values())
    assert {"direct", "discovered", "double"} <= kinds
    assert any(k.endswith("+promotion_only") for k in kinds)
    assert set(checks_ref.checks("4k4/9/4P4/9/9/9/9/9/4K4 b G 1")["classes"].values()) == {"direct", "drop"}


def test_check_bitmap_rejects_bad_arguments_before_device_work():
    L = nv.lib()
    z, p = None, 1 << 20  # p: an aligned address that is never dereferenced
    assert L.kz_check_bitmap(z, 4, 500, p, 448, p + (1 << 16), 448, z, z) == -1
    assert L.kz_check_bitmap(p, 4, 500, z, 448, p + (1 << 16), 448, z, z) == -1
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 448, z, 448, z, z) == -1
    for n in (0, -1):
        assert L.kz_check_bitmap(p, n, 500, p + (1 << 16), 448, p + (1 << 17), 448, z, z) == -1
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 422, p + (1 << 17), 448, z, z) == -1  # short strides
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 448, p + (1 << 17), 100, z, z) == -1
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16) + 4, 448, p + (1 << 17), 448, z, z) == -1  # misaligned rows
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 448, p + (1 << 17) + 8, 448, z, z) == -1
    assert L.kz_check_bitmap(p + 16, 4, 500, p + (1 << 16), 448, p + (1 << 17), 448, z, z) == -1  # misaligned state
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 448, p + (1 << 17), 448, p + 2, z) == -1  # misaligned count
    assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 448, p + (1 << 16) + 448 * 4, 448, z, z) == -1  # overlap
    assert L.kz_check_bitmap(p, 4, -1, p + (1 << 16), 448, p + (1 << 17), 448, z, z) == -1
    # well-formed arguments (stride 423 included) pass the checks and reach the tables test: without a GPU, and so
    # without tables, that is KZ_E_NOT_INIT (with a GPU the call would launch on these fake pointers, so it is skipped)
    import torch
    if not torch.cuda.is_available():
        assert L.kz_check_bitmap(p, 4, 500, p + (1 << 16), 423, p + (1 << 17), 423, z, z) == -3


def test_mate_batches_pad_the_last_batch():
    from shogidrl_b200.evaluation import mate_batches
    assert mate_batches(10, 4) == [(0, 4, 4), (4, 4, 4), (8, 2, 4)]
    assert mate_batches(3, 8) == [(0, 3, 3)]
    assert mate_batches(8, 8) == [(0, 8, 8)]
    assert mate_batches(0, 8) == []
    for total, envs in ((1, 1), (7, 3), (1000, 64), (65, 64)):
        b = mate_batches(total, envs)
        assert sum(c for _, c, _ in b) == total
        assert all(n == min(total, envs) and 0 < c <= n for _, c, n in b)
        assert [f for f, _, _ in b] == list(range(0, total, min(total, envs)))
    with pytest.raises(ValueError):
        mate_batches(4, 0)


def test_evaluate_mate_in_one_without_positions_or_with_unknown_player():
    from shogidrl_b200.evaluation import evaluate_mate_in_one
    r = evaluate_mate_in_one("random", [])
    assert (r.positions, r.with_mate, r.solved, r.solve_rate) == (0, 0, 0, 0.0)
    with pytest.raises(ValueError, match="unknown scripted player"):
        evaluate_mate_in_one("minimax", ["4k4/9/4P4/9/9/9/9/9/4K4 b G 1"])
