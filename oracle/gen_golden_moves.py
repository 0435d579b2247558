"""Golden strings of the demo-log move descriptions (shogidrl_b200.utils.move_formatting), for machines without a checkout
of the reference:

    python oracle/gen_golden_moves.py

Unlike the other gen_golden_* scripts this one records this repository's module, not the reference's.  The module is
unchanged since the commit that checked it string for string against keisei/utils/move_formatting.py
(tests/test_reference_live_cpu.py::test_move_descriptions_identical, which samples the same moves); the fixture pins
those strings.  Writes tests/golden/move_descriptions.json."""
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import shogidrl_b200.utils.move_formatting as mf  # noqa: E402
from shogidrl_b200.shogi.definitions import Color, Piece, PieceType  # noqa: E402
from shogidrl_b200.utils import PolicyOutputMapper  # noqa: E402


def main():
    mapper = PolicyOutputMapper()
    rng = random.Random(5)
    moves = []
    for idx in rng.sample(range(13527), 1500):
        move = mapper.policy_index_to_shogi_move(idx)
        v = rng.randrange(14)
        moves.append([idx, v, mf.format_move_with_description(move, mapper),
                      mf.format_move_with_description_enhanced(move, mapper, None),
                      mf.format_move_with_description_enhanced(move, mapper, Piece(PieceType(v), Color.BLACK))])
    out = {"moves": moves,
           "piece_names": [[mf._get_piece_name(PieceType(v), promo) for promo in (False, True)] for v in range(14)],
           "square_names": [mf._coords_to_square_name(r, c) for r in range(9) for c in range(9)],
           "none": [mf.format_move_with_description(None, mapper), mf.format_move_with_description_enhanced(None, mapper)]}
    dst = os.path.join(ROOT, "tests", "golden", "move_descriptions.json")
    with open(dst, "w", encoding="utf-8") as f:
        json.dump(out, f, ensure_ascii=False, separators=(",", ":"))
    print("wrote", dst, len(moves), "moves")


if __name__ == "__main__":
    main()
