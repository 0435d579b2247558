"""perft: the number of legal move sequences of a given length from a position, counted on the device.

Perft is the standard exhaustive test of a move generator (every legal line to a fixed depth, compared with published
counts) and the throughput figure shogi engines report (nodes/s).  Here a tree level is two launches: list_moves turns
the frontier's legal bitmaps into a list of (node, action) items, and GameBatch.expand applies every item to a copy of
its node.
Levels 1 .. depth-2 are materialised as child state blobs plus legal bitmaps; the last level is only counted: perft(d) is
the sum of the legal counts of the level-(d-1) items, so that launch writes no rows and no children.

Children carry no history (GameBatch.expand), so perft counts the move tree: a mated or stalemated node has no children and
repetition never ends a line.  Roots are loaded with max_moves 65535, so the move-count limit never prunes the tree."""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch

from . import _native as nv
from ._batch import GameBatch, chunks, list_moves
from .vec_env import parse_start_positions

HIRATE = "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"
MAX_MOVES = 65535
CHILD_HIST_CAP = 1  # the smallest repetition table (64 slots, 1 KB per child): children have no history to hold


class _Level:
    """Frontier nodes of one tree level: a GameBatch, its legal rows and counts, and the tag of each node (its root, and
    with divide its root move, as root * NUM_ACTIONS + action)."""

    def __init__(self, batch: GameBatch, rows: torch.Tensor, count: torch.Tensor, tags: torch.Tensor):
        self.batch, self.rows, self.count, self.tags = batch, rows, count, tags


def perft(positions: Optional[Union[str, Sequence[str]]] = None, depth: Optional[int] = None, *, divide: bool = False,
          device="cuda", max_items: int = 1 << 24) -> Union[List[int], List[Dict[int, int]]]:
    """Perft of each root position to ``depth`` plies: -> one count per root, or with ``divide=True`` one dict per root
    from each legal root action (policy index) to the count below it.

    ``positions``: SFEN strings (one string is one root; None: the start position).  ``max_items`` bounds the items of
    one expansion launch: a level that would pass it is split by frontier nodes and each chunk is expanded and recursed
    into depth-first, so memory stays bounded whatever the depth (about 3 KB per materialised item, 16 B per counted
    one).  Raises ValueError for a negative depth or a position that does not parse."""
    if depth is None or int(depth) != depth or depth < 0:
        raise ValueError(f"perft: depth must be an integer >= 0, got {depth!r}")
    depth = int(depth)
    if max_items < 1024:
        raise ValueError(f"perft: max_items must be at least 1024, got {max_items}")
    sfens = [HIRATE] if positions is None else ([positions] if isinstance(positions, str) else list(positions))
    parsed = parse_start_positions(sfens, MAX_MOVES)
    R = len(parsed[2])
    if depth == 0:
        return [{} for _ in range(R)] if divide else [1] * R
    device = nv.require_cuda(device)
    nv.init_tables(device)
    with torch.cuda.device(device):
        batch = GameBatch(R, CHILD_HIST_CAP, device).load(*parsed, MAX_MOVES)
        roots = _Level(batch, *batch.legal_rows(), torch.arange(R, dtype=torch.int64, device=device))
        bins = R * nv.NUM_ACTIONS if divide else R
        acc = torch.zeros(bins, dtype=torch.int64, device=device)
        _count(roots, depth, acc, divide, True, max_items)
        if not divide:
            return [int(x) for x in acc.cpu()]
        # every legal root move gets an entry, also those with no line below them (a mate at depth >= 2)
        _, parent, acts = list_moves(roots.rows, roots.count)
        acc_h, par_h, act_h = acc.cpu().numpy(), parent.cpu().numpy(), acts.cpu().numpy()
        out: List[Dict[int, int]] = [{} for _ in range(R)]
        for r, a in zip(par_h.tolist(), act_h.tolist()):
            out[r][a] = int(acc_h[r * nv.NUM_ACTIONS + a])
        return out


def _count(lv: _Level, depth: int, acc: torch.Tensor, divide: bool, is_root: bool, max_items: int) -> None:
    """acc[tag] += perft(node, depth) for every node of the level (depth >= 1)."""
    if depth == 1:
        if divide and is_root:  # each root move is one line
            _, parent, actions = list_moves(lv.rows, lv.count)
            acc.index_add_(0, lv.tags[parent.long()] * nv.NUM_ACTIONS + actions, torch.ones_like(actions))
        else:
            acc.index_add_(0, lv.tags, lv.count.long())
        return
    offsets_h = np.concatenate([[0], np.cumsum(lv.count.cpu().numpy().astype(np.int64))])
    for a, b in chunks(offsets_h, max_items):  # one node's moves always fit
        _, parent, actions = list_moves(lv.rows[a:b], lv.count[a:b])
        parent += a  # parent indexes the whole level
        tags = (lv.tags[parent.long()] * nv.NUM_ACTIONS + actions) if (divide and is_root) else lv.tags[parent.long()]
        _expand(lv, parent, actions, tags, depth, acc, divide, max_items)


def _expand(lv: _Level, parent: torch.Tensor, actions: torch.Tensor, tags: torch.Tensor, depth: int, acc: torch.Tensor,
            divide: bool, max_items: int) -> None:
    """Expand the items (depth >= 2 below the level): counted when depth == 2, materialised and recursed into otherwise."""
    m = int(parent.numel())
    count = torch.empty(m, dtype=torch.int32, device=parent.device)
    if depth == 2:
        lv.batch.expand(parent, actions, legal_count=count)
        acc.index_add_(0, tags, count.long())
        return
    rows = torch.empty((m, nv.BITMAP_WORDS), dtype=torch.int32, device=parent.device)
    child = lv.batch.expand(parent, actions, rows=rows, legal_count=count, child_hist_cap=CHILD_HIST_CAP)
    del parent, actions
    _count(_Level(child, rows, count, tags), depth - 1, acc, divide, False, max_items)
