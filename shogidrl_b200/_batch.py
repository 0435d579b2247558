"""GameBatch: n games in one state blob (kz_state_layout), and the launches that read a batch without moving its games --
legal rows, checking rows, move expansion, mates in one and capture gains -- with the CSR move listing (list_moves) and
its chunking by whole games (chunks) that VecShogiEnv, the look-ahead opponent and perft share."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _native as nv


def _dev(a, dtype, device) -> torch.Tensor:
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device).contiguous()


def _rows(t: Optional[torch.Tensor], width: int):
    """(data pointer, row stride in elements) of optional row storage."""
    return (None, 0) if t is None else (t.data_ptr(), t.stride(0) if t.dim() > 1 else width)


class GameBatch:
    """n games with repetition tables for ``hist_cap`` plies on ``device``.  The blob is allocated uninitialised: load
    positions, reset or expand into it before reading it.  ``blob_args`` are the (state, n, hist_cap) arguments of the
    entry points that take the batch."""

    def __init__(self, n: int, hist_cap: int, device: torch.device):
        self.n, self.hist_cap, self.device = int(n), int(hist_cap), device
        total = C.c_int64()
        nv.check(nv.lib().kz_state_layout(self.n, self.hist_cap, None, C.byref(total)), "kz_state_layout")
        self.state = torch.empty(total.value, dtype=torch.uint8, device=device)
        self.blob_args = (self.state.data_ptr(), self.n, self.hist_cap)

    def load(self, boards, hands, side, move_count, max_moves) -> "GameBatch":
        """kz_load_positions of parsed positions (host arrays: boards [n, 81], hands [n, 14], side [n], move_count [n];
        ``max_moves`` one int for every game or [n]) -> self."""
        d = self.device
        b, h = _dev(boards, torch.int8, d), _dev(hands, torch.uint8, d)
        s, mc = _dev(side, torch.uint8, d), _dev(move_count, torch.int32, d)
        mm = (torch.full((self.n,), max_moves, dtype=torch.int32, device=d) if isinstance(max_moves, int)
              else _dev(max_moves, torch.int32, d))
        nv.require(b.shape == (self.n, 81) and h.shape == (self.n, 14), f"load: boards [{self.n}, 81], hands [{self.n}, 14]")
        nv.check(nv.lib().kz_load_positions(*self.blob_args, b.data_ptr(), h.data_ptr(), s.data_ptr(), mc.data_ptr(),
                                            mm.data_ptr(), nv.stream_ptr(d)), "kz_load_positions")
        return self

    def legal_rows(self):
        """kz_legal_bitmap into new rows: -> (legal rows int32 [n, 448], legal counts int32 [n])."""
        rows = torch.empty((self.n, nv.BITMAP_WORDS), dtype=torch.int32, device=self.device)
        count = torch.empty(self.n, dtype=torch.int32, device=self.device)
        nv.check(nv.lib().kz_legal_bitmap(*self.blob_args, None, 0, rows.data_ptr(), nv.BITMAP_WORDS, None, count.data_ptr(),
                                          nv.stream_ptr(self.device)), "kz_legal_bitmap")
        return rows, count

    def check_rows(self, rows: torch.Tensor, out: Optional[torch.Tensor] = None):
        """kz_check_bitmap of legal rows -> (the rows of their checking moves, ``out`` or new int32 [n, 448]; their
        counts int32 [n])."""
        if out is None:
            out = torch.empty((self.n, nv.BITMAP_WORDS), dtype=torch.int32, device=self.device)
        count = torch.empty(self.n, dtype=torch.int32, device=self.device)
        nv.check(nv.lib().kz_check_bitmap(*self.blob_args, rows.data_ptr(), rows.stride(0), out.data_ptr(), out.stride(0),
                                          count.data_ptr(), nv.stream_ptr(self.device)), "kz_check_bitmap")
        return out, count

    def expand(self, parent: torch.Tensor, actions: torch.Tensor, *, obs=None, rows=None, cobs=None, reward=None, done=None,
               reason=None, winner=None, ep_len=None, legal_count=None, err=None,
               child_hist_cap: Optional[int] = None) -> Optional["GameBatch"]:
        """kz_expand of the M >= 1 items parent int32 [M], actions int64 / int32 [M] into the outputs given by name (each
        holding at least M items; ``rows`` receives the legal rows).  With ``child_hist_cap`` the successors go to a new
        batch of M games, which is returned."""
        m = int(parent.numel())
        items = (reward, done, reason, winner, ep_len, legal_count, err)
        for t, width in ((obs, nv.OBS_FLOATS), (rows, nv.BITMAP_WORDS), (cobs, nv.COBS_WORDS), *((t, 1) for t in items)):
            nv.require(t is None or t.numel() >= m * width, f"expand: every output must hold {m} items")
        child = None if child_hist_cap is None else GameBatch(m, child_hist_cap, self.device)
        nv.check(nv.lib().kz_expand(*self.blob_args, 0, parent.data_ptr(), actions.data_ptr(),
                                    int(actions.dtype == torch.int64), m, *_rows(obs, nv.OBS_FLOATS),
                                    *_rows(rows, nv.BITMAP_WORDS), nv.ptr(cobs), *map(nv.ptr, items),
                                    *((None, 0) if child is None else child.blob_args[::2]), nv.stream_ptr(self.device)),
                 "kz_expand")
        return child

    def mates_in_one(self, rows: torch.Tensor):
        """Mates in one of the games from their legal rows (int32 [n, 448]): -> (the lowest mating action int64 [n], -1 for
        none; the number of mating moves int32 [n]).  A mate must give check, so kz_check_bitmap keeps the checking moves,
        list_moves lists them and kz_expand decides them: Tsumi without capturing a king.  One host read (of the number
        of checking moves)."""
        d = self.device
        _, parent, actions = list_moves(*self.check_rows(rows))
        m = int(parent.numel())
        mates = torch.zeros(self.n, dtype=torch.int32, device=d)
        action = torch.full((self.n,), -1, dtype=torch.int64, device=d)
        if m == 0:
            return action, mates
        reason = torch.empty(m, dtype=torch.uint8, device=d)
        err = torch.empty(m, dtype=torch.uint8, device=d)
        self.expand(parent, actions, reason=reason, err=err)
        mate = (reason == nv.TSUMI) & ((err & nv.ERR_KING_CAPTURE) == 0)
        p = parent.long()
        mates.index_add_(0, p, mate.to(torch.int32))
        first = torch.full((self.n,), nv.NUM_ACTIONS, dtype=torch.int64, device=d)
        first.scatter_reduce_(0, p, torch.where(mate, actions, nv.NUM_ACTIONS), "amin")
        return torch.where(mates > 0, first, action), mates

    def capture_gain(self, rows: torch.Tensor, gain: torch.Tensor) -> None:
        """kz_capture_gain: the largest gain over the moves of each game's legal row into ``gain`` (int32 [n])."""
        nv.check(nv.lib().kz_capture_gain(*self.blob_args, rows.data_ptr(), rows.stride(0), gain.data_ptr(), None,
                                          nv.stream_ptr(self.device)), "kz_capture_gain")


def list_moves(rows: torch.Tensor, count: torch.Tensor, host_offsets: bool = False):
    """The moves of legal or checking rows (int32 [n, >= 423]) whose per-row counts are ``count`` (int32 [n]) as a list
    grouped by row (CSR): -> (offsets int64 [n+1], parent int32 [M], actions int64 [M]); row g's actions are
    actions[offsets[g]:offsets[g+1]] in ascending order and parent[i] is the row of move i.  One host read: M, or with
    ``host_offsets`` all the offsets, returned as a fourth element (int64 numpy [n+1]).  No launch when M is 0."""
    n, d = int(count.numel()), count.device
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=d)
    offsets[1:] = torch.cumsum(count, 0, dtype=torch.int64)
    offsets_h = offsets.cpu().numpy() if host_offsets else None
    m = int(offsets_h[-1]) if host_offsets else int(offsets[-1])
    parent = torch.empty(m, dtype=torch.int32, device=d)
    actions = torch.empty(m, dtype=torch.int64, device=d)
    if m > 0:  # an empty tensor has no storage to hand to kz_legal_list
        nv.check(nv.lib().kz_legal_list(rows.data_ptr(), rows.stride(0), n, offsets.data_ptr(), parent.data_ptr(),
                                        actions.data_ptr(), 1, nv.stream_ptr(d)), "kz_legal_list")
    return (offsets, parent, actions, offsets_h) if host_offsets else (offsets, parent, actions)


def chunks(offsets_host, max_items: int):
    """Ranges [a, b) of consecutive games, in order, of the CSR offsets ``offsets_host`` (int64 [n+1]) that hold at most
    ``max_items`` items each -- a single game above the limit is a range of its own -- leaving out ranges without items."""
    out, a = [], 0
    while a < len(offsets_host) - 1:
        b = max(int(np.searchsorted(offsets_host, offsets_host[a] + max_items, side="right")) - 1, a + 1)
        if offsets_host[b] > offsets_host[a]:
            out.append((a, b))
        a = b
    return out
