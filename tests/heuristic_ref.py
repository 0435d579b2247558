"""Test-side restatement of the scripted heuristic opponent (keisei/utils/opponents.py SimpleHeuristicOpponent) over
policy indices, independent of the CUDA kernel's window arithmetic, and the positions of the golden traces the
reference wrote, rebuilt as they stood BEFORE each recorded ply (the fixtures store the successor states)."""
import os

import numpy as np

MASK64 = (1 << 64) - 1


def rand32(seed: int, env: int, step: int) -> int:
    """The engine's counter-based random stream (kz_common.cuh rand32 / the oracle's orc_rand32)."""
    x = (seed ^ ((env * 0x9E3779B97F4A7C15) & MASK64) ^ ((step * 0xBF58476D1CE4E5B9) & MASK64)) & MASK64
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & MASK64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & MASK64
    x ^= x >> 31
    return x >> 32


def tiers(board, side: int, legal):
    """(captures, non-promoting pawn moves, others) of the legal action indices, each ascending.  A capture lands on a
    piece of the other colour; a pawn move starts on the mover's unpromoted pawn (code 1 + 14*side) and does not
    promote; drops (index >= 12960) are never either."""
    out = ([], [], [])
    for a in sorted(int(x) for x in legal):
        t = 2
        if a < 12960:
            pair, promote = a >> 1, a & 1
            frm, r = divmod(pair, 80)
            to = r + (r >= frm)
            dest = int(board[to])
            if dest != 0 and (dest >= 15) != bool(side):
                t = 0
            elif int(board[frm]) == 1 + 14 * side and not promote:
                t = 1
        out[t].append(a)
    return out


def top_tier(board, side: int, legal):
    """(tier index 0/1/2 or 255, its members ascending)."""
    for t, members in enumerate(tiers(board, side, legal)):
        if members:
            return t, members
    return 255, []


def pick(tier_members, seed: int, env: int, step: int) -> int:
    """k-th member in ascending order, k = mulhi(rand32, size); -1 for an empty tier."""
    if not tier_members:
        return -1
    return tier_members[(rand32(seed, env, step) * len(tier_members)) >> 32]


def fixture_positions(golden_dir):
    """Every ply of traces_random.npz and traces_endgame.npz as the position it was played from: dict of boards int8
    [P, 81], hands uint8 [P, 14], sides uint8 [P], move_counts int32 [P] and legal (list of the reference's legal index
    arrays), plus source (0 random traces, 1 endgames)."""
    from oracle import oracle as orc
    start_b, start_h, _ = orc.OracleGame().export()
    boards, hands, sides, mcs, legal, source = [], [], [], [], [], []
    with np.load(os.path.join(golden_dir, "traces_random.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    i = 0
    for T in z["T"]:
        for t in range(int(T)):
            if t == 0 or z["dones"][i - 1]:
                b, h, s, mc = start_b, start_h, 0, 0
            else:
                b, h, s, mc = z["boards"][i - 1], z["hands"][i - 1], int(z["sides"][i - 1]), int(z["move_counts"][i - 1])
            boards.append(b); hands.append(h); sides.append(s); mcs.append(mc)
            legal.append(z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]])
            source.append(0)
            i += 1
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    i = 0
    for g, T in enumerate(z["T"]):
        _, _, s0, mc0 = orc.parse_sfen(str(z["sfens"][g]))
        for t in range(int(T)):
            if t == 0:
                b, h, s, mc = z["start_boards"][g], z["start_hands"][g], s0, mc0
            else:
                b, h, s, mc = z["boards"][i - 1], z["hands"][i - 1], int(z["sides"][i - 1]), int(z["move_counts"][i - 1])
            boards.append(b); hands.append(h); sides.append(s); mcs.append(mc)
            legal.append(z["legal"][z["legal_off"][i]:z["legal_off"][i + 1]])
            source.append(1)
            i += 1
    return dict(boards=np.stack(boards).astype(np.int8), hands=np.stack(hands).astype(np.uint8),
                sides=np.asarray(sides, np.uint8), move_counts=np.asarray(mcs, np.int32), legal=legal,
                source=np.asarray(source, np.uint8))
