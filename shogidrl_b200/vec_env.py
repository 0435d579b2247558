"""VecShogiEnv -- N device-resident Shogi games stepped by one kernel launch.

Batched counterpart of ``keisei.shogi.ShogiGame`` + the reset-on-done handling of
``keisei.training.step_manager.StepManager`` (step_manager.py:98-348, 437-440).  All arrays live on the
GPU; observations and masks are written by the kernel straight into caller-provided rollout storage."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import numpy as np
import torch

from . import _native as nv


def parse_start_positions(sfens: Sequence[str], max_moves: int):
    """Parse a start-position pool on the host: -> (boards int8 [P, 81], hands uint8 [P, 14], sides uint8 [P],
    move_counts int32 [P]).  Raises ValueError naming the index of the first entry that does not parse or whose move
    number already reaches ``max_moves``."""
    from .shogi.sfen import pack_sfen
    if isinstance(sfens, str):
        raise ValueError("start positions: expected a sequence of SFEN strings, got one string")
    packed = []
    for i, s in enumerate(sfens):
        try:
            p = pack_sfen(str(s))
        except Exception as e:  # the SFEN parser raises ValueError, KeyError or IndexError on malformed text
            raise ValueError(f"start position {i} ({s!r}) does not parse: {e}") from e
        if p[3] >= max_moves:
            raise ValueError(f"start position {i} ({s!r}) is terminal at load: move count {p[3]} >= max_moves {max_moves}")
        packed.append(p)
    if not packed:
        raise ValueError("start positions: the pool is empty (pass None to restart from the start position)")
    return (np.stack([p[0] for p in packed]), np.stack([p[1] for p in packed]),
            np.asarray([p[2] for p in packed], np.uint8), np.asarray([p[3] for p in packed], np.int32))


class VecShogiEnv:
    # Pool draws are keyed by seed ^ POOL_SALT (auto-reset inside kz_step_pool) and seed ^ POOL_RESET_SALT (explicit
    # reset), so that they are independent of the fused random actions and of each other: a reset() right after an
    # auto-reset (same finished-episode counter) does not redraw the same entry.
    POOL_SALT = 0x506F6F6C5374  # "PoolSt"
    POOL_RESET_SALT = 0x506F6F6C5273  # "PoolRs"

    def __init__(self, num_envs: int, max_moves_per_game: int = 500, device="cuda", seed: int = 1234,
                 env_offset: int = 0, auto_reset: bool = True, hist_cap: Optional[int] = None,
                 step_streams: Optional[int] = None, start_positions: Optional[Sequence[str]] = None):
        self.device = nv.require_cuda(device)
        self.n = int(num_envs)
        self.max_moves = int(max_moves_per_game)
        self.hist_cap = int(hist_cap if hist_cap is not None else max_moves_per_game)
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        self.auto_reset = bool(auto_reset)
        self._L = nv.lib()
        nv.init_tables(self.device)
        offs = (C.c_int64 * 3)()
        total = C.c_int64()
        nv.check(self._L.kz_state_layout(self.n, self.hist_cap, offs, C.byref(total)), "kz_state_layout")
        self.state = torch.zeros(total.value, dtype=torch.uint8, device=self.device)
        self.state_bytes = total.value
        # persistent per-step outputs
        d = self.device
        self.obs = torch.zeros((self.n, 46, 9, 9), dtype=torch.float32, device=d)
        self._mask_store = torch.zeros((self.n, nv.MASK_PAD_STRIDE), dtype=torch.uint8, device=d)
        self.mask = self._mask_store[:, : nv.NUM_ACTIONS]  # uint8 view, row stride 13536
        # per-step scalar results live in ONE contiguous buffer (15 bytes per env: next_actions i64, reward f32,
        # done u8, reason u8, winner i8) so that a host consumer fetches them with a single device-to-host copy
        n = self.n
        self.results = torch.zeros(15 * n, dtype=torch.uint8, device=d)
        self.next_actions = self.results[: 8 * n].view(torch.int64)
        self.reward = self.results[8 * n: 12 * n].view(torch.float32)
        self.done = self.results[12 * n: 13 * n]
        self.reason = self.results[13 * n: 14 * n]
        self.winner = self.results[14 * n:].view(torch.int8)
        self.ep_len = torch.zeros(self.n, dtype=torch.int32, device=d)
        self.legal_count = torch.zeros(self.n, dtype=torch.int32, device=d)
        self.step_index = 0
        # A step can be launched as `step_streams` ranges of games on as many streams (kz_step_range; results identical to
        # one launch).  Off by default: joined back into the caller's stream after every step, the ranges only share the
        # SMs within one step and the step gets no shorter (measured on B200, 65,536 games: 0.344 ms as one launch, 0.356
        # as two ranges, 0.364 as four).  What does pay is letting ranges run AHEAD of each other across steps, which
        # needs a caller that consumes each range's results separately: HostPipelinedEnv.
        if step_streams is None:
            step_streams = 1
        self.step_streams = max(1, int(step_streams))
        if self.n % (8 * self.step_streams) != 0:
            self.step_streams = 1
        self._side_streams = [torch.cuda.Stream(device=d) for _ in range(self.step_streams)] if self.step_streams > 1 else []
        # start-position pool (set_start_positions): records on the device, and the pool index of each env's current game
        # (-1: begun from the start position).  _ids_in_use: some entry may still name a pool entry while no pool is set,
        # so resets from the start position must write -1 over it.
        self.pool: Optional[torch.Tensor] = None
        self.start_ids = torch.full((self.n,), -1, dtype=torch.int32, device=d)
        self._ids_in_use = False
        if start_positions is not None:
            self.set_start_positions(start_positions, reset=False)
        self.reset()

    # ------------------------------------------------------------------ helpers
    def _sp(self):
        return nv.stream_ptr(self.device)

    def _rows_arg(self, t: Optional[torch.Tensor], what: str, dtypes, row_elems: int, n: Optional[int] = None):
        """(data pointer, row stride in elements) of caller storage the kernel writes ``n`` rows into (default: one per
        env); rejects anything the kernel would write out of bounds (the C ABI sees raw pointers only)."""
        n = self.n if n is None else n
        if t is None:
            return None, 0
        if t.device != self.device or t.dtype not in dtypes:
            raise ValueError(f"{what}: expected a {dtypes[0]} tensor on {self.device}, got {t.dtype} on {t.device}")
        if t.dim() > 1:
            rows, stride = t.shape[0], t.stride(0)
            inner = t[0]
        else:
            rows, stride, inner = 1, row_elems, t
        if rows < n or inner.numel() < row_elems or not inner.is_contiguous():
            raise ValueError(f"{what}: need at least {n} rows of {row_elems} contiguous elements, got shape "
                             f"{tuple(t.shape)} with strides {tuple(t.stride())}")
        return t.data_ptr(), stride

    def _obs_args(self, obs: Optional[torch.Tensor], n: Optional[int] = None):
        return self._rows_arg(obs, "obs", (torch.float32,), nv.OBS_FLOATS, n)

    def _mask_args(self, mask: Optional[torch.Tensor]):
        return self._rows_arg(mask, "mask", (torch.uint8, torch.bool), nv.NUM_ACTIONS)

    def _vec_arg(self, t: Optional[torch.Tensor], what: str, dtypes, n: Optional[int] = None):
        """Data pointer of a contiguous [n] vector on the env's device (default n: one element per env; None stays
        None)."""
        n = self.n if n is None else n
        if t is None:
            return None
        if t.device != self.device or t.dtype not in dtypes or not t.is_contiguous() or t.numel() < n:
            raise ValueError(f"{what}: expected a contiguous {'/'.join(str(d)[6:] for d in dtypes)} [{n}] tensor on "
                             f"{self.device}, got {tuple(t.shape)} {t.dtype} on {t.device}")
        return t.data_ptr()

    def _pick_arg(self, start_pick: Optional[torch.Tensor], in_step: bool = True):
        if start_pick is None:
            return None
        if self.pool is None:
            raise ValueError("start_pick needs a start-position pool (set_start_positions)")
        if in_step and not self.auto_reset:
            raise ValueError("start_pick: this env does not reset finished games (auto_reset=False), so no game would "
                             "start from it; use reset(start_pick=...)")
        return self._vec_arg(start_pick, "start_pick", (torch.int32,))

    # ------------------------------------------------------------------ API
    def set_start_positions(self, sfens: Optional[Sequence[str]], reset: bool = False) -> None:
        """Restart finished games from a pool of SFEN positions instead of the start position (None: back to the start
        position).  Every game that finishes from now on -- in ``step`` / ``step_rollout`` or through ``reset()`` --
        starts from a uniformly drawn entry, or from the entry a step's ``start_pick`` names.  ``start_ids`` (int32 [n])
        holds, for each env's current game, its entry in the pool that was set when that game started, or -1 if it
        started from the start position; games in progress continue and keep their ids when the pool changes, and
        ``reset=True`` restarts every env from the new pool (or the start position) at once.  Each entry is parsed on the host and its record (board, hands, side to move, move number, position key,
        legal bitmap, legal count, in-check flag) is computed once on the device by the engine's refresh path
        (kz_pool_records).  Raises ValueError naming the index of an entry that does not parse, is terminal at load
        (checkmate, stalemate, move number >= max_moves) or lets the side to move capture the opponent's king."""
        if sfens is None:
            self.pool = None
        else:
            self.pool = self._build_pool(parse_start_positions(sfens, self.max_moves))
            self._ids_in_use = True
        if reset:
            self.reset()

    def _build_pool(self, parsed) -> torch.Tensor:
        """Pool records (int32 [P, POOL_RECORD_WORDS]) of parsed positions: kz_load_positions + kz_refresh
        (termination, in-check) + kz_legal_bitmap on a scratch batch of the P positions, then kz_pool_records."""
        boards, hands, sides, mcs = parsed
        P, d, sp = len(sides), self.device, self._sp()
        offs, total = (C.c_int64 * 3)(), C.c_int64()
        nv.check(self._L.kz_state_layout(P, 0, offs, C.byref(total)), "kz_state_layout")
        state = torch.zeros(total.value, dtype=torch.uint8, device=d)
        dev = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(d).contiguous()  # noqa: E731
        b, h, s, mc = dev(boards, torch.int8), dev(hands, torch.uint8), dev(sides, torch.uint8), dev(mcs, torch.int32)
        mm = torch.full((P,), self.max_moves, dtype=torch.int32, device=d)
        nv.check(self._L.kz_load_positions(state.data_ptr(), P, 0, b.data_ptr(), h.data_ptr(), s.data_ptr(), mc.data_ptr(),
                                           mm.data_ptr(), sp), "kz_load_positions")
        count = torch.zeros(P, dtype=torch.int32, device=d)
        check = torch.zeros(P, dtype=torch.uint8, device=d)
        nv.check(self._L.kz_refresh(state.data_ptr(), P, 0, None, 0, None, 0, count.data_ptr(), None, 1, 0, 0, 0, 1,
                                    check.data_ptr(), sp), "kz_refresh")
        bitmap = torch.zeros((P, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
        nv.check(self._L.kz_legal_bitmap(state.data_ptr(), P, 0, None, 0, bitmap.data_ptr(), nv.BITMAP_WORDS, None,
                                         count.data_ptr(), sp), "kz_legal_bitmap")
        meta = torch.empty((P, 8), dtype=torch.int32, device=d)
        nv.check(self._L.kz_export_positions(state.data_ptr(), P, 0, None, None, meta.data_ptr(), sp), "kz_export_positions")
        # a legal board move onto the square of the opponent's king (kz_step flags that as KZ_ERR_KING_CAPTURE)
        side = s.long()
        ksq = torch.where(b == (8 + 14 * (1 - side))[:, None], torch.arange(81, device=d), 81).amin(1)  # 81: no king
        frm = torch.arange(81, device=d)[None, :]
        to = ksq[:, None].clamp(max=80)
        idx = ((frm * 80 + to - (to > frm).long()) * 2)[:, :, None] + torch.arange(2, device=d)
        bits = (bitmap.long().gather(1, (idx >> 5).view(P, -1)) >> (idx & 31).view(P, -1)) & 1
        ok_from = ((frm != to) & (ksq[:, None] < 81))[:, :, None].expand(P, 81, 2).reshape(P, -1)
        king_capture = ((bits != 0) & ok_from).any(1)
        status, count_h, kc = meta[:, 3].cpu(), count.cpu(), king_capture.cpu()
        for i in range(P):
            if int(status[i]) != 0 or int(count_h[i]) == 0:
                raise ValueError(f"start position {i} is terminal at load ({nv.REASONS.get(int(status[i])) or 'no legal move'})")
            if bool(kc[i]):
                raise ValueError(f"start position {i} lets the side to move capture the opponent's king")
        records = torch.empty((P, nv.POOL_RECORD_WORDS), dtype=torch.int32, device=d)
        nv.check(self._L.kz_pool_records(state.data_ptr(), P, 0, bitmap.data_ptr(), nv.BITMAP_WORDS, count.data_ptr(),
                                         check.data_ptr(), records.data_ptr(), sp), "kz_pool_records")
        return records

    def reset(self, env_mask: Optional[torch.Tensor] = None, refresh: bool = True, random_actions: bool = False,
              start_pick: Optional[torch.Tensor] = None):
        """ShogiGame.reset for all (or the masked) envs; returns (obs, mask) of the new positions.  With a start-position
        pool the envs restart from pool entries (``start_pick``: int32 [n] entry per env, default a uniform draw)."""
        mp = None
        if env_mask is not None:
            env_mask = env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mp = env_mask.data_ptr()
        pk = self._pick_arg(start_pick, in_step=False)
        if self.pool is not None:
            nv.check(self._L.kz_reset_pool(self.state.data_ptr(), self.n, self.hist_cap, mp, self.max_moves,
                                           self.pool.data_ptr(), self.pool.shape[0], pk,
                                           (self.seed ^ self.POOL_RESET_SALT) & 0xFFFFFFFFFFFFFFFF, self.env_offset,
                                           self.start_ids.data_ptr(), self._sp()), "kz_reset_pool")
        else:
            nv.check(self._L.kz_reset(self.state.data_ptr(), self.n, self.hist_cap, mp, self.max_moves, self._sp()),
                     "kz_reset")
            if self._ids_in_use:
                if env_mask is None:
                    self.start_ids.fill_(-1)
                    self._ids_in_use = False
                else:
                    self.start_ids.masked_fill_(env_mask != 0, -1)
        if env_mask is None:
            self.step_index = 0
        if refresh:
            self.refresh(random_actions=random_actions)
        return self.obs, self.mask

    def refresh(self, obs: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
                eval_termination: bool = False, random_actions: bool = False,
                next_out: Optional[torch.Tensor] = None, in_check: Optional[torch.Tensor] = None):
        """Recompute obs / mask / legal_count (and optionally uniform-random legal actions) in place."""
        obs = self.obs if obs is None else obs
        mask = self.mask if mask is None else mask
        op, os_ = self._obs_args(obs)
        mp, ms = self._mask_args(mask)
        nv.check(self._L.kz_refresh(self.state.data_ptr(), self.n, self.hist_cap, op, os_, mp, ms,
                                    self.legal_count.data_ptr(),
                                    (self.next_actions if next_out is None else next_out).data_ptr() if random_actions else None,
                                    1, self.seed, self.step_index, self.env_offset, int(eval_termination),
                                    nv.ptr(in_check), self._sp()),
                 "kz_refresh")
        return obs, mask

    def step(self, actions: torch.Tensor, obs: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
             random_actions: bool = False, write_obs: bool = True, write_mask: bool = True,
             next_out: Optional[torch.Tensor] = None, start_pick: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """make_move for every env.  ``obs`` / ``mask`` may point into a rollout buffer (e.g. obs_buf[t+1]).
        With ``random_actions`` the kernel also writes a uniform-random legal action for the returned state
        into ``next_out`` (default ``self.next_actions``; must not alias ``actions``).  With a start-position pool,
        ``start_pick`` (int32 [n]) names the entry each env restarts from if its game finishes in this step."""
        obs = (self.obs if obs is None else obs) if write_obs else None
        mask = (self.mask if mask is None else mask) if write_mask else None
        self._launch(actions, self._obs_args(obs), self._mask_args(mask), (None, 0), None, self.reward, self.done,
                     random_actions, next_out, start_pick)
        return {"obs": obs, "mask": mask, "reward": self.reward, "done": self.done, "reason": self.reason,
                "winner": self.winner, "ep_len": self.ep_len, "legal_count": self.legal_count}

    def step_rollout(self, actions: torch.Tensor, obs: Optional[torch.Tensor], bitmap: torch.Tensor,
                     reward: Optional[torch.Tensor] = None, done: Optional[torch.Tensor] = None,
                     random_actions: bool = False, next_out: Optional[torch.Tensor] = None,
                     cobs: Optional[torch.Tensor] = None, start_pick: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """``step`` in its rollout form (kz_step_rollout): the successor's legal set is written as the 13,527-bit legal
        bitmap (int32 [n, 448] rows, e.g. ``RolloutBuffer.bitmaps[t + 1]``) instead of the byte mask -- 1.8 KB instead
        of 13.5 KB per game here and in every later pass of the sampler / PPO update over it.  ``obs`` as in ``step``
        (None: no observation rows); ``reward`` / ``done`` may point into rollout storage (fp32 / uint8 [n]); ``cobs``
        (int32 [n, 40]) receives the compact observations the policy network's input layer reads (kz_cobs_conv_*);
        ``start_pick`` as in ``step``."""
        reward = self.reward if reward is None else reward
        done = self.done if done is None else done
        self._vec_arg(reward, "reward", (torch.float32,))
        self._vec_arg(done, "done", (torch.uint8,))
        self._launch(actions, self._obs_args(obs), (None, 0), self._bitmap_args(bitmap), self._cobs_arg(cobs), reward, done,
                     random_actions, next_out, start_pick)
        return {"obs": obs, "bitmap": bitmap, "reward": reward, "done": done, "reason": self.reason,
                "winner": self.winner, "ep_len": self.ep_len, "legal_count": self.legal_count}

    def _launch(self, actions: torch.Tensor, obs, mask, bitmap, cobs, reward: torch.Tensor, done: torch.Tensor,
                random_actions: bool, next_out: Optional[torch.Tensor], start_pick: Optional[torch.Tensor]) -> None:
        """One step of every env in the mask form (``mask`` rows) or the rollout form (``bitmap`` rows); ``obs`` / ``mask``
        / ``bitmap`` are validated (pointer, row stride) pairs and ``cobs`` a validated pointer.  Validates the arguments
        both forms share, then launches kz_step_pool when finished games restart from a pool, kz_step_range otherwise:
        once on the current stream, or as ``step_streams`` ranges of games (each with its own work counter) forked from
        and joined back into it."""
        ap = self._vec_arg(actions, "actions", (torch.int64, torch.int32))
        nxt = None
        if random_actions:
            nxt = self.next_actions if next_out is None else next_out
            if actions.dtype == torch.int32 and nxt.dtype == torch.int64:
                nxt = nxt.view(torch.int32)[: self.n]
            if nxt.data_ptr() == ap:
                raise ValueError("next_out must not alias actions (the kernel reads one while writing the other)")
            nxt = nxt.data_ptr()
        pick = self._pick_arg(start_pick)
        self.step_index += 1  # after validation: a rejected call leaves the RNG counter where it was
        args = (ap, int(actions.dtype == torch.int64), *obs, *mask, *bitmap, cobs, reward.data_ptr(), done.data_ptr(),
                self.reason.data_ptr(), self.winner.data_ptr(), self.ep_len.data_ptr(), self.legal_count.data_ptr(), nxt,
                self.seed, self.step_index, self.env_offset)
        if self.pool is not None and self.auto_reset:
            fn, name = self._L.kz_step_pool, "kz_step_pool"
            args += (self.pool.data_ptr(), self.pool.shape[0], pick, (self.seed ^ self.POOL_SALT) & 0xFFFFFFFFFFFFFFFF,
                     self.start_ids.data_ptr())
        else:
            fn, name = self._L.kz_step_range, "kz_step_range"
            args += (int(self.auto_reset),)
        state = self.state.data_ptr()
        if self.step_streams == 1:  # no events: rollout steps are captured into a CUDA graph
            nv.check(fn(state, self.n, self.hist_cap, 0, self.n, 0, *args, self._sp()), name)
        else:
            cur = torch.cuda.current_stream(self.device)
            per = self.n // self.step_streams
            fork = torch.cuda.Event()
            fork.record(cur)
            for i, st in enumerate(self._side_streams):
                st.wait_event(fork)
                nv.check(fn(state, self.n, self.hist_cap, i * per, per, i, *args, st.cuda_stream), name)
                join = torch.cuda.Event()
                join.record(st)
                cur.wait_event(join)
        self._restarted_from_start(done)

    def _restarted_from_start(self, done: torch.Tensor) -> None:
        """After a launch without a pool: games that finished restarted from the start position (start_ids -1)."""
        if self._ids_in_use and self.pool is None and self.auto_reset:
            self.start_ids.masked_fill_(done[: self.n] != 0, -1)

    def legal_bitmap(self, bitmap: torch.Tensor, obs: Optional[torch.Tensor] = None, cobs: Optional[torch.Tensor] = None):
        """Legal bitmap (and optionally the observation rows / compact observations) of the CURRENT positions
        (kz_legal_bitmap)."""
        bp, bs = self._bitmap_args(bitmap)
        op, os_ = self._obs_args(obs)
        nv.check(self._L.kz_legal_bitmap(self.state.data_ptr(), self.n, self.hist_cap, op, os_, bp, bs, self._cobs_arg(cobs),
                                         self.legal_count.data_ptr(), self._sp()), "kz_legal_bitmap")
        return obs, bitmap

    def legal_actions(self):
        """Every legal move of every env's CURRENT position as a list grouped by env (CSR): -> (offsets int64 [n+1],
        parent int32 [M], actions int64 [M]); env g's legal actions are actions[offsets[g]:offsets[g+1]] in ascending
        order, and parent[i] is the env of move i.  kz_legal_bitmap into scratch rows, then kz_legal_list; one host read
        (of M, to size the list)."""
        d, sp = self.device, self._sp()
        bitmap = torch.empty((self.n, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
        count = torch.empty(self.n, dtype=torch.int32, device=d)
        nv.check(self._L.kz_legal_bitmap(self.state.data_ptr(), self.n, self.hist_cap, None, 0, bitmap.data_ptr(),
                                         nv.BITMAP_WORDS, None, count.data_ptr(), sp), "kz_legal_bitmap")
        offsets = torch.zeros(self.n + 1, dtype=torch.int64, device=d)
        offsets[1:] = torch.cumsum(count, 0, dtype=torch.int64)
        m = int(offsets[-1])
        parent = torch.empty(m, dtype=torch.int32, device=d)
        actions = torch.empty(m, dtype=torch.int64, device=d)
        nv.check(self._L.kz_legal_list(bitmap.data_ptr(), nv.BITMAP_WORDS, self.n, offsets.data_ptr(), parent.data_ptr(),
                                       actions.data_ptr(), 1, sp), "kz_legal_list")
        return offsets, parent, actions

    def expand(self, parent: torch.Tensor, actions: torch.Tensor, *, obs: Optional[torch.Tensor] = None,
               bitmap: Optional[torch.Tensor] = None, cobs: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """What would happen if env ``parent[i]`` played ``actions[i]``, for M items at once, without moving any env
        (kz_expand): -> dict of per-item tensors reward, done, reason, winner, ep_len, legal_count and err (error bits),
        each exactly what ``step`` (without auto-reset) would report for that one move on a copy of the env, its
        repetition history included.  ``parent`` int32 [M] (each in [0, n)), ``actions`` int64 / int32 [M]; ``obs``
        (fp32 [M, 46, 9, 9]), ``bitmap`` (int32 [M, 448]) and ``cobs`` (int32 [M, 40]) optionally receive the successors'
        rows as ``step_rollout`` writes them.  Items of one env should be adjacent (as ``legal_actions`` lists them)."""
        m = int(parent.numel())
        pp = self._vec_arg(parent, "parent", (torch.int32,), m)
        ap = self._vec_arg(actions, "actions", (torch.int64, torch.int32), m)
        nv.require(int(actions.numel()) == m, "parent and actions must have the same length")
        d = self.device
        out = {"reward": torch.zeros(m, dtype=torch.float32, device=d), "done": torch.zeros(m, dtype=torch.uint8, device=d),
               "reason": torch.zeros(m, dtype=torch.uint8, device=d), "winner": torch.zeros(m, dtype=torch.int8, device=d),
               "ep_len": torch.zeros(m, dtype=torch.int32, device=d),
               "legal_count": torch.zeros(m, dtype=torch.int32, device=d), "err": torch.zeros(m, dtype=torch.uint8, device=d)}
        if m == 0:
            return out
        if bool(((parent < 0) | (parent >= self.n)).any()):
            raise ValueError(f"parent: every entry must name an env in [0, {self.n})")
        op, os_ = self._obs_args(obs, m)
        bp, bs = (None, 0) if bitmap is None else self._bitmap_args(bitmap, m)
        nv.check(self._L.kz_expand(self.state.data_ptr(), self.n, self.hist_cap, 0, pp, ap, int(actions.dtype == torch.int64),
                                   m, op, os_, bp, bs, self._cobs_arg(cobs, m), out["reward"].data_ptr(),
                                   out["done"].data_ptr(), out["reason"].data_ptr(), out["winner"].data_ptr(),
                                   out["ep_len"].data_ptr(), out["legal_count"].data_ptr(), out["err"].data_ptr(), None, 0,
                                   self._sp()), "kz_expand")
        return out

    def check_bitmap(self, bitmap: torch.Tensor, out: Optional[torch.Tensor] = None):
        """The legal moves of every env's CURRENT position that give check (kz_check_bitmap): ``bitmap`` holds the legal
        rows (int32 [n, 448], as ``legal_bitmap`` writes them) -> (out rows of the checking moves, count int32 [n]).
        ``out`` (default: new rows) must not overlap ``bitmap``.  Exact for positions in which the side not to move is
        not in check (every position reached by play); a loaded position in which it is gets all its legal moves.
        Finished games get an empty row."""
        bp, bs = self._bitmap_args(bitmap)
        if out is None:
            out = torch.empty((self.n, nv.BITMAP_WORDS), dtype=torch.int32, device=self.device)
        op, os_ = self._bitmap_args(out)
        count = torch.empty(self.n, dtype=torch.int32, device=self.device)
        nv.check(self._L.kz_check_bitmap(self.state.data_ptr(), self.n, self.hist_cap, bp, bs, op, os_, count.data_ptr(),
                                         self._sp()), "kz_check_bitmap")
        return out, count

    def checking_actions(self):
        """Every legal move that gives check, of every env's CURRENT position, in ``legal_actions``' CSR form: ->
        (offsets int64 [n+1], parent int32 [M], actions int64 [M]).  kz_legal_bitmap, kz_check_bitmap, then kz_legal_list
        on the check rows; one host read (of M)."""
        d, sp = self.device, self._sp()
        bitmap = torch.empty((self.n, nv.BITMAP_WORDS), dtype=torch.int32, device=d)
        count = torch.empty(self.n, dtype=torch.int32, device=d)
        nv.check(self._L.kz_legal_bitmap(self.state.data_ptr(), self.n, self.hist_cap, None, 0, bitmap.data_ptr(),
                                         nv.BITMAP_WORDS, None, count.data_ptr(), sp), "kz_legal_bitmap")
        rows, count = self.check_bitmap(bitmap)
        offsets = torch.zeros(self.n + 1, dtype=torch.int64, device=d)
        offsets[1:] = torch.cumsum(count, 0, dtype=torch.int64)
        m = int(offsets[-1])
        parent = torch.empty(m, dtype=torch.int32, device=d)
        actions = torch.empty(m, dtype=torch.int64, device=d)
        if m > 0:  # empty tensors have no storage to hand to kz_legal_list
            nv.check(self._L.kz_legal_list(rows.data_ptr(), nv.BITMAP_WORDS, self.n, offsets.data_ptr(), parent.data_ptr(),
                                           actions.data_ptr(), 1, sp), "kz_legal_list")
        return offsets, parent, actions

    def mate_in_one(self) -> Dict[str, torch.Tensor]:
        """Mates in one of every env's CURRENT position: -> {"action": int64 [n] the lowest-index mating move (-1: none),
        "count": int32 [n] the number of mating moves}.  A mate must give check, so only ``checking_actions`` are
        expanded (``expand``); a move mates when its expansion ends the game by Tsumi without capturing a king (capturing
        a king is outside the engine's contract, as in ``step``).  No env moves."""
        _, parent, actions = self.checking_actions()
        d = self.device
        count = torch.zeros(self.n, dtype=torch.int32, device=d)
        action = torch.full((self.n,), -1, dtype=torch.int64, device=d)
        if parent.numel() == 0:
            return {"action": action, "count": count}
        m = int(parent.numel())
        reason = torch.empty(m, dtype=torch.uint8, device=d)
        err = torch.empty(m, dtype=torch.uint8, device=d)
        # kz_expand directly rather than expand(): the parents come from kz_legal_list and need no host-side check
        nv.check(self._L.kz_expand(self.state.data_ptr(), self.n, self.hist_cap, 0, parent.data_ptr(), actions.data_ptr(), 1,
                                   m, None, 0, None, 0, None, None, None, reason.data_ptr(), None, None, None,
                                   err.data_ptr(), None, 0, self._sp()), "kz_expand")
        mate = (reason == nv.TSUMI) & ((err & nv.ERR_KING_CAPTURE) == 0)
        p = parent.long()
        count.index_add_(0, p, mate.to(torch.int32))
        first = torch.full((self.n,), nv.NUM_ACTIONS, dtype=torch.int64, device=d)
        first.scatter_reduce_(0, p, torch.where(mate, actions, nv.NUM_ACTIONS), "amin")
        action = torch.where(count > 0, first, action)
        return {"action": action, "count": count}

    # The heuristic opponent draws from the env's random stream keyed by seed ^ HEURISTIC_SALT, so its pick is independent
    # of the fused uniform-random action (next_actions, keyed by the seed itself) drawn for the same step and env.
    HEURISTIC_SALT = 0x48657572697374  # "Heurist"

    def heuristic_actions(self, out: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
                          bitmap: Optional[torch.Tensor] = None, tier: Optional[torch.Tensor] = None,
                          tier_count: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The scripted SimpleHeuristicOpponent's move (keisei/utils/opponents.py) for every env's CURRENT position
        (kz_heuristic_actions): a uniform pick among the captures if there are any, else among the non-promoting moves of
        an unpromoted pawn, else among all other legal moves; -1 where there is no legal move.  The legal set is read from
        ``mask`` (default ``self.mask``) or from ``bitmap`` rows (int32 [n, 448], as ``step_rollout`` writes them), not
        both.  ``out`` int64 / int32 [n] (default: a new int64 tensor); ``tier`` (uint8 [n]: 0 capture, 1 pawn, 2 other,
        255 none) and ``tier_count`` (int32 [n]: size of the chosen tier) are optional.  Draws with ``step_index``."""
        if mask is not None and bitmap is not None:
            raise ValueError("heuristic_actions: give the legal set as mask or as bitmap, not both")
        mp, ms, bp, bs = None, 0, None, 0
        if bitmap is not None:
            bp, bs = self._bitmap_args(bitmap)
        else:
            mp, ms = self._mask_args(self.mask if mask is None else mask)
        if out is None:
            out = torch.empty(self.n, dtype=torch.int64, device=self.device)
        op = self._vec_arg(out, "out", (torch.int64, torch.int32))
        tp, cp = self._vec_arg(tier, "tier", (torch.uint8,)), self._vec_arg(tier_count, "tier_count", (torch.int32,))
        nv.check(self._L.kz_heuristic_actions(self.state.data_ptr(), self.n, self.hist_cap, mp, ms, bp, bs, op,
                                              int(out.dtype == torch.int64), tp, cp,
                                              (self.seed ^ self.HEURISTIC_SALT) & 0xFFFFFFFFFFFFFFFF, self.step_index,
                                              self.env_offset, self._sp()), "kz_heuristic_actions")
        return out

    def _cobs_arg(self, cobs: Optional[torch.Tensor], n: Optional[int] = None):
        n = self.n if n is None else n
        if cobs is None:
            return None
        if (cobs.device != self.device or cobs.dtype != torch.int32 or cobs.dim() != 2 or cobs.shape[0] < n
                or cobs.shape[1] != nv.COBS_WORDS or not cobs.is_contiguous()):
            raise ValueError(f"cobs: expected a contiguous int32 [{n}, {nv.COBS_WORDS}] tensor on {self.device}")
        return cobs.data_ptr()

    def _bitmap_args(self, bitmap: torch.Tensor, n: Optional[int] = None):
        n = self.n if n is None else n
        if (bitmap.device != self.device or bitmap.dtype != torch.int32 or bitmap.dim() != 2 or bitmap.shape[0] < n
                or bitmap.shape[1] != nv.BITMAP_WORDS or bitmap.stride(1) != 1 or bitmap.stride(0) % 4
                or bitmap.data_ptr() % 16):
            raise ValueError(f"bitmap: expected int32 [{n}, {nv.BITMAP_WORDS}] rows (16-byte aligned) on {self.device}")
        return bitmap.data_ptr(), bitmap.stride(0)

    def load_positions(self, boards, hands, side, move_count, max_moves=None, eval_termination: bool = True):
        """ShogiGame.from_sfen for every env from already-parsed arrays (numpy or torch)."""
        d = self.device
        b = torch.as_tensor(np.ascontiguousarray(boards), dtype=torch.int8).to(d).contiguous()
        h = torch.as_tensor(np.ascontiguousarray(hands), dtype=torch.uint8).to(d).contiguous()
        s = torch.as_tensor(np.ascontiguousarray(side), dtype=torch.uint8).to(d).contiguous()
        mc = torch.as_tensor(np.ascontiguousarray(move_count), dtype=torch.int32).to(d).contiguous()
        if max_moves is None:
            max_moves = np.full(self.n, self.max_moves, np.int32)
        mm = torch.as_tensor(np.ascontiguousarray(max_moves), dtype=torch.int32).to(d).contiguous()
        nv.require(b.shape == (self.n, 81) and h.shape == (self.n, 14), "b.shape == (self.n, 81) and h.shape == (self.n, 14)")
        nv.check(self._L.kz_load_positions(self.state.data_ptr(), self.n, self.hist_cap, b.data_ptr(), h.data_ptr(),
                                           s.data_ptr(), mc.data_ptr(), mm.data_ptr(), self._sp()), "kz_load_positions")
        self.refresh(eval_termination=eval_termination)
        return self.obs, self.mask

    def export(self):
        """-> boards int8 [n,81], hands uint8 [n,14], meta int32 [n,8] (side, move_count, max_moves, status,
        winner, error bits, plies since reset, finished episodes) as torch tensors on the device."""
        d = self.device
        b = torch.empty((self.n, 81), dtype=torch.int8, device=d)
        h = torch.empty((self.n, 14), dtype=torch.uint8, device=d)
        m = torch.empty((self.n, 8), dtype=torch.int32, device=d)
        nv.check(self._L.kz_export_positions(self.state.data_ptr(), self.n, self.hist_cap, b.data_ptr(), h.data_ptr(),
                                             m.data_ptr(), self._sp()), "kz_export_positions")
        return b, h, m

    def to_games(self, env_ids=None):
        """Host snapshots (``shogi.sfen.HostPosition``) of the selected device games: SFEN / board text / KIF
        headers for debugging, parity dumps and displays (SURVEY.md section 8 f-3).  One export launch + one D2H."""
        from .shogi.sfen import HostPosition
        b, h, m = [x.cpu().numpy() for x in self.export()]
        ids = range(self.n) if env_ids is None else [int(i) for i in env_ids]
        return [HostPosition(b[i], h[i], m[i, 0], m[i, 1], status=m[i, 3], winner=m[i, 4]) for i in ids]

    def to_sfen(self, env_ids=None):
        """SFEN strings of the selected device games (shogi_game_io.py:312-379 format)."""
        return [g.to_sfen_string() for g in self.to_games(env_ids)]

    def load_sfens(self, sfens, eval_termination: bool = True):
        """ShogiGame.from_sfen (shogi_game.py:283-345) for a whole batch: one SFEN per env."""
        from .shogi.sfen import pack_sfen
        nv.require(len(sfens) == self.n, "len(sfens) == self.n")
        packed = [pack_sfen(s) for s in sfens]
        return self.load_positions(np.stack([p[0] for p in packed]), np.stack([p[1] for p in packed]),
                                   np.asarray([p[2] for p in packed], np.uint8), np.asarray([p[3] for p in packed], np.int32),
                                   eval_termination=eval_termination)

    def errors(self, clear: bool = False) -> torch.Tensor:
        out = torch.empty(self.n, dtype=torch.int32, device=self.device)
        nv.check(self._L.kz_errors(self.state.data_ptr(), self.n, self.hist_cap, out.data_ptr(), int(clear), self._sp()),
                 "kz_errors")
        return out

    def piece_targets(self, squares) -> torch.Tensor:
        """Pseudo-legal target sets (81-bit, 3 x uint32 per env) of the pieces on ``squares`` [n]."""
        sq = torch.as_tensor(np.ascontiguousarray(squares), dtype=torch.int32).to(self.device).contiguous()
        out = torch.zeros((self.n, 3), dtype=torch.int32, device=self.device)
        nv.check(self._L.kz_piece_targets(self.state.data_ptr(), self.n, self.hist_cap, sq.data_ptr(), out.data_ptr(),
                                          self._sp()), "kz_piece_targets")
        return out
