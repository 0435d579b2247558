"""perft: the number of legal move sequences of a given length from a position, counted on the device.

Perft is the standard exhaustive test of a move generator (every legal line to a fixed depth, compared with published
counts) and the throughput figure shogi engines report (nodes/s).  Here a tree level is two launches: kz_legal_list turns
the frontier's legal bitmaps into a list of (node, action) items, and kz_expand applies every item to a copy of its node.
Levels 1 .. depth-2 are materialised as child state blobs plus legal bitmaps; the last level is only counted: perft(d) is
the sum of the legal counts of the level-(d-1) items, so that launch writes no rows and no children.

Children carry no history (kz_expand), so perft counts the move tree: a mated or stalemated node has no children and
repetition never ends a line.  Roots are loaded with max_moves 65535, so the move-count limit never prunes the tree."""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch

from . import _native as nv
from .vec_env import parse_start_positions

HIRATE = "lnsgkgsnl/1r5b1/ppppppppp/9/9/9/PPPPPPPPP/1B5R1/LNSGKGSNL b - 1"
MAX_MOVES = 65535
CHILD_HIST_CAP = 1  # the smallest repetition table (64 slots, 1 KB per child): children have no history to hold


class _Level:
    """Frontier nodes of one tree level: a state blob of n games, their legal bitmaps and counts, and the tag of each
    node (its root, and with divide its root move, as root * NUM_ACTIONS + action)."""

    def __init__(self, blob: torch.Tensor, n: int, hist_cap: int, bitmap: torch.Tensor, count: torch.Tensor,
                 tags: torch.Tensor):
        self.blob, self.n, self.hist_cap, self.bitmap, self.count, self.tags = blob, n, hist_cap, bitmap, count, tags


def _blob(L, n: int, hist_cap: int, device) -> torch.Tensor:
    total = C.c_int64()
    nv.check(L.kz_state_layout(n, hist_cap, None, C.byref(total)), "kz_state_layout")
    return torch.empty(total.value, dtype=torch.uint8, device=device)


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
    boards, hands, sides, mcs = parse_start_positions(sfens, MAX_MOVES)
    R = len(sides)
    if depth == 0:
        return [{} for _ in range(R)] if divide else [1] * R
    device = nv.require_cuda(device)
    L = nv.lib()
    nv.init_tables(device)
    with torch.cuda.device(device):
        sp = nv.stream_ptr(device)
        dev = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(device)  # noqa: E731
        b, h, s, mc = dev(boards, torch.int8), dev(hands, torch.uint8), dev(sides, torch.uint8), dev(mcs, torch.int32)
        mm = torch.full((R,), MAX_MOVES, dtype=torch.int32, device=device)
        blob = _blob(L, R, CHILD_HIST_CAP, device)
        nv.check(L.kz_load_positions(blob.data_ptr(), R, CHILD_HIST_CAP, b.data_ptr(), h.data_ptr(), s.data_ptr(),
                                     mc.data_ptr(), mm.data_ptr(), sp), "kz_load_positions")
        bitmap = torch.empty((R, nv.BITMAP_WORDS), dtype=torch.int32, device=device)
        count = torch.empty(R, dtype=torch.int32, device=device)
        nv.check(L.kz_legal_bitmap(blob.data_ptr(), R, CHILD_HIST_CAP, None, 0, bitmap.data_ptr(), nv.BITMAP_WORDS, None,
                                   count.data_ptr(), sp), "kz_legal_bitmap")
        roots = _Level(blob, R, CHILD_HIST_CAP, bitmap, count, torch.arange(R, dtype=torch.int64, device=device))
        bins = R * nv.NUM_ACTIONS if divide else R
        acc = torch.zeros(bins, dtype=torch.int64, device=device)
        _count(L, roots, depth, acc, divide, True, max_items, sp)
        if not divide:
            return [int(x) for x in acc.cpu()]
        # every legal root move gets an entry, also those with no line below them (a mate at depth >= 2)
        parent, acts = _list(L, roots, 0, R, sp)
        acc_h, par_h, act_h = acc.cpu().numpy(), parent.cpu().numpy(), acts.cpu().numpy()
        out: List[Dict[int, int]] = [{} for _ in range(R)]
        for r, a in zip(par_h.tolist(), act_h.tolist()):
            out[r][a] = int(acc_h[r * nv.NUM_ACTIONS + a])
        return out


def _count(L, lv: _Level, depth: int, acc: torch.Tensor, divide: bool, is_root: bool, max_items: int, sp) -> None:
    """acc[tag] += perft(node, depth) for every node of the level (depth >= 1)."""
    if depth == 1:
        if divide and is_root:  # each root move is one line
            parent, actions = _list(L, lv, 0, lv.n, sp)
            acc.index_add_(0, lv.tags[parent.long()] * nv.NUM_ACTIONS + actions, torch.ones_like(actions))
        else:
            acc.index_add_(0, lv.tags, lv.count.long())
        return
    offsets_h = np.concatenate([[0], np.cumsum(lv.count.cpu().numpy().astype(np.int64))])
    a = 0
    while a < lv.n:  # chunks of consecutive nodes with at most max_items items (one node's moves always fit)
        b = int(np.searchsorted(offsets_h, offsets_h[a] + max_items, side="right")) - 1
        b = max(b, a + 1)
        m = int(offsets_h[b] - offsets_h[a])
        if m > 0:
            parent, actions = _list(L, lv, a, b, sp)
            tags = (lv.tags[parent.long()] * nv.NUM_ACTIONS + actions) if (divide and is_root) else lv.tags[parent.long()]
            _expand(L, lv, parent, actions, tags, depth, acc, divide, max_items, sp)
        a = b


def _list(L, lv: _Level, a: int, b: int, sp):
    """(parent int32, action int64) of every legal move of nodes [a, b) of the level; parent indexes the whole level."""
    count = lv.count[a:b]
    offsets = torch.zeros(b - a + 1, dtype=torch.int64, device=count.device)
    offsets[1:] = torch.cumsum(count, 0, dtype=torch.int64)
    m = int(offsets[-1])
    parent = torch.empty(m, dtype=torch.int32, device=count.device)
    actions = torch.empty(m, dtype=torch.int64, device=count.device)
    if m:
        nv.check(L.kz_legal_list(lv.bitmap[a].data_ptr(), nv.BITMAP_WORDS, b - a, offsets.data_ptr(), parent.data_ptr(),
                                 actions.data_ptr(), 1, sp), "kz_legal_list")
        parent += a
    return parent, actions


def _expand(L, lv: _Level, parent: torch.Tensor, actions: torch.Tensor, tags: torch.Tensor, depth: int, acc: torch.Tensor,
            divide: bool, max_items: int, sp) -> None:
    """Expand the items (depth >= 2 below the level): counted when depth == 2, materialised and recursed into otherwise."""
    m = int(parent.numel())
    d = parent.device
    count = torch.empty(m, dtype=torch.int32, device=d)
    if depth == 2:
        nv.check(L.kz_expand(lv.blob.data_ptr(), lv.n, lv.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1, m, None, 0,
                             None, 0, None, None, None, None, None, None, count.data_ptr(), None, None, 0, sp), "kz_expand")
        acc.index_add_(0, tags, count.long())
        return
    child = _blob(L, m, CHILD_HIST_CAP, d)
    bitmap = torch.empty((m, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
    nv.check(L.kz_expand(lv.blob.data_ptr(), lv.n, lv.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1, m, None, 0,
                         bitmap.data_ptr(), nv.BITMAP_WORDS, None, None, None, None, None, None, count.data_ptr(), None,
                         child.data_ptr(), CHILD_HIST_CAP, sp), "kz_expand")
    del parent, actions
    _count(L, _Level(child, m, CHILD_HIST_CAP, bitmap, count, tags), depth - 1, acc, divide, False, max_items, sp)
