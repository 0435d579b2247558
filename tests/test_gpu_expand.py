"""Move expansion (kz_expand), legal-move lists (kz_legal_list) and device perft.

Expansion is checked bit for bit against kz_step_rollout(auto_reset=0) on CLONES: every item's parent is copied into a
fresh blob (board row, meta row and repetition table sliced out of the kz_state_layout sections) and stepped with the
item's action.  Perft is checked against the published hirate counts and against the C oracle's own move generator."""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)
from tests import perft_ref  # noqa: E402  (checker only)

DEV = torch.device("cuda:0")
NA = 13527
CHUNK = 1 << 16


def _layout(L, n, hist_cap):
    offs, total = (C.c_int64 * 3)(), C.c_int64()
    assert L.kz_state_layout(n, hist_cap, offs, C.byref(total)) == 0
    return [int(o) for o in offs], int(total.value)


def _sections(state, n, hist_cap, L):
    (ob, om, oh), total = _layout(L, n, hist_cap)
    boards = state[ob:ob + 96 * n].view(n, 96)
    meta = state[om:om + 32 * n].view(n, 32)
    hist = state[oh:total - 256].view(n, -1)
    return boards, meta, hist


def _rows(m):
    return (torch.full((m, 46 * 81), -1.0, device=DEV), torch.full((m, 448), -1, dtype=torch.int32, device=DEV),
            torch.full((m, 40), -1, dtype=torch.int32, device=DEV))


def _scalars(m):
    return {"reward": torch.full((m,), 9.0, device=DEV), "done": torch.full((m,), 7, dtype=torch.uint8, device=DEV),
            "reason": torch.full((m,), 7, dtype=torch.uint8, device=DEV),
            "winner": torch.full((m,), 7, dtype=torch.int8, device=DEV),
            "ep_len": torch.full((m,), -7, dtype=torch.int32, device=DEV),
            "legal_count": torch.full((m,), -7, dtype=torch.int32, device=DEV)}


def _expand_raw(env, parent, actions, child_hist_cap=1, counter_slot=0):
    """kz_expand with every output: scalars, err, obs / bitmap / cobs rows and a child blob."""
    from shogidrl_b200 import _native as nv
    L = nv.lib()
    m = int(parent.numel())
    obs, bm, cobs = _rows(m)
    s = _scalars(m)
    err = torch.full((m,), 0xEE, dtype=torch.uint8, device=DEV)
    child = torch.full((_layout(L, m, child_hist_cap)[1],), 0xAB, dtype=torch.uint8, device=DEV)
    nv.check(L.kz_expand(env.state.data_ptr(), env.n, env.hist_cap, counter_slot, parent.data_ptr(), actions.data_ptr(), 1, m,
                         obs.data_ptr(), 46 * 81, bm.data_ptr(), 448, cobs.data_ptr(), s["reward"].data_ptr(),
                         s["done"].data_ptr(), s["reason"].data_ptr(), s["winner"].data_ptr(), s["ep_len"].data_ptr(),
                         s["legal_count"].data_ptr(), err.data_ptr(), child.data_ptr(), child_hist_cap,
                         torch.cuda.current_stream().cuda_stream), "kz_expand")
    s["err"] = err
    return s, obs, bm, cobs, child


def _step_clones(env, parent, actions):
    """The reference side: clone each item's parent into a fresh blob and call kz_step_rollout(auto_reset=0)."""
    from shogidrl_b200 import _native as nv
    L = nv.lib()
    m = int(parent.numel())
    _, total = _layout(L, m, env.hist_cap)
    clone = torch.zeros(total, dtype=torch.uint8, device=DEV)
    sb, sm, sh = _sections(env.state, env.n, env.hist_cap, L)
    cb, cm, ch = _sections(clone, m, env.hist_cap, L)
    p = parent.long()
    cb.copy_(sb[p]); cm.copy_(sm[p]); ch.copy_(sh[p])
    obs, bm, cobs = _rows(m)
    s = _scalars(m)
    nv.check(L.kz_step_rollout(clone.data_ptr(), m, env.hist_cap, actions.data_ptr(), 1, obs.data_ptr(), 46 * 81,
                               bm.data_ptr(), 448, cobs.data_ptr(), s["reward"].data_ptr(), s["done"].data_ptr(),
                               s["reason"].data_ptr(), s["winner"].data_ptr(), s["ep_len"].data_ptr(),
                               s["legal_count"].data_ptr(), None, 0, 0, 0, 0, torch.cuda.current_stream().cuda_stream),
             "kz_step_rollout")
    err = torch.empty(m, dtype=torch.int32, device=DEV)
    nv.check(L.kz_errors(clone.data_ptr(), m, env.hist_cap, err.data_ptr(), 0, torch.cuda.current_stream().cuda_stream),
             "kz_errors")
    s["err"] = err.to(torch.uint8)
    return s, obs, bm, cobs, clone


def _export(state, n, hist_cap):
    from shogidrl_b200 import _native as nv
    b = torch.empty((n, 81), dtype=torch.int8, device=DEV)
    h = torch.empty((n, 14), dtype=torch.uint8, device=DEV)
    m = torch.empty((n, 8), dtype=torch.int32, device=DEV)
    nv.check(nv.lib().kz_export_positions(state.data_ptr(), n, hist_cap, b.data_ptr(), h.data_ptr(), m.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream), "kz_export_positions")
    return b, h, m


def _items(env, rng, extra=True):
    """Every legal action of every game, plus (extra) per game one random index, -1 and 13527 (pattern-invalid and
    out-of-range actions; finished games reject nothing and return their terminal tuple)."""
    offsets, parent, actions = env.legal_actions()
    if extra:
        n = env.n
        g = torch.arange(n, dtype=torch.int32, device=DEV)
        rnd = torch.as_tensor(rng.integers(0, NA, n), device=DEV)
        parent = torch.cat([parent, g, g, g])
        actions = torch.cat([actions, rnd, torch.full((n,), -1, device=DEV), torch.full((n,), NA, device=DEV)])
        order = torch.argsort(parent, stable=True)  # items of one parent adjacent
        parent, actions = parent[order].contiguous(), actions[order].contiguous()
    return parent, actions


def _check_expansion(env, parent, actions, label):
    from shogidrl_b200 import _native as nv
    L = nv.lib()
    (_, _, _), total = _layout(L, env.n, env.hist_cap)
    before = env.state[: total - 256].clone()
    for c0 in range(0, int(parent.numel()), CHUNK):
        p, a = parent[c0:c0 + CHUNK].contiguous(), actions[c0:c0 + CHUNK].contiguous()
        m = int(p.numel())
        got, g_obs, g_bm, g_cobs, child = _expand_raw(env, p, a)
        want, w_obs, w_bm, w_cobs, clone = _step_clones(env, p, a)
        for k in want:
            assert torch.equal(got[k], want[k]), (label, k, int((got[k] != want[k]).sum()))
        assert torch.equal(g_bm, w_bm), (label, "bitmap")
        assert torch.equal(g_cobs, w_cobs), (label, "cobs")
        assert torch.equal(g_obs, w_obs), (label, "obs")
        # the child is the clone's successor with no history: same board row (with the key), same meta row apart from the
        # error bits, plies since reset and episodes (0), and an empty repetition table
        cb, cm, ch = _sections(child, m, 1, L)
        kb, km, _ = _sections(clone, m, env.hist_cap, L)
        assert torch.equal(cb, kb), (label, "child board rows")
        keep = [i for i in range(32) if i not in (17, 20, 21, 24, 25, 26, 27)]
        assert torch.equal(cm[:, keep], km[:, keep]), (label, "child meta rows")
        assert int(cm[:, [17, 20, 21, 24, 25, 26, 27]].abs().sum()) == 0, label
        assert int(ch.abs().sum()) == 0, label
        eb, eh, em = _export(child, m, 1)
        xb, xh, xm = _export(clone, m, env.hist_cap)
        assert torch.equal(eb, xb) and torch.equal(eh, xh) and torch.equal(em[:, :5], xm[:, :5]), label
        # the env's own entry point reports the same scalars
        if bool(((p >= 0) & (p < env.n)).all()):
            out = env.expand(p, a)
            for k in want:
                assert torch.equal(out[k], want[k]), (label, "env.expand", k)
    torch.cuda.synchronize()
    assert torch.equal(env.state[: total - 256], before), (label, "source blob written")


def _golden_random():
    with np.load(os.path.join(os.path.dirname(__file__), "golden", "traces_random.npz")) as z:
        return {k: z[k] for k in z.files}


def test_expand_matches_step_on_clones_golden_traces():
    """The reference's random traces replayed with kz_step to plies 0 / 50 / 150 / 300 (populated repetition tables,
    some games finished, some with error bits from steps past their trace)."""
    from shogidrl_b200 import VecShogiEnv
    z = _golden_random()
    n = len(z["T"])
    starts = np.concatenate([[0], np.cumsum(z["T"])])[:-1]
    env = VecShogiEnv(n, max_moves_per_game=500, device=DEV, auto_reset=False)
    start = orc.OracleGame().export()
    env.load_positions(np.repeat(start[0][None], n, 0), np.repeat(start[1][None], n, 0), np.zeros(n), np.zeros(n),
                       max_moves=z["max_moves"].astype(np.int32))
    rng = np.random.default_rng(5)
    ply = 0
    for target in (0, 50, 150, 300):
        while ply < target:
            acts = [int(z["actions"][starts[g] + ply]) if ply < z["T"][g] else 0 for g in range(n)]
            env.step(torch.tensor(acts, dtype=torch.int64, device=DEV))
            ply += 1
        parent, actions = _items(env, rng)
        _check_expansion(env, parent, actions, f"golden ply {target}")
    assert int((env.export()[2][:, 3] != 0).sum()) > 0  # finished games took part


def test_expand_endgames_and_bad_parents(golden_dir):
    """The 128 drop-heavy endgames; items whose parent lies outside the batch."""
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200 import _native as nv
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        sfens = [str(s) for s in zf["sfens"]]
    env = VecShogiEnv(len(sfens), max_moves_per_game=500, device=DEV, auto_reset=False)
    env.load_sfens(sfens)
    parent, actions = _items(env, np.random.default_rng(7))
    _check_expansion(env, parent, actions, "endgames")
    # parents outside [0, n): KZ_ERR_BAD_ACTION and the outputs of a rejected action on an empty board
    p = torch.tensor([-1, env.n, 1 << 30, -(1 << 30)], dtype=torch.int32, device=DEV)
    a = torch.tensor([0, 100, 12960, 5], dtype=torch.int64, device=DEV)
    (_, _, _), total = _layout(nv.lib(), env.n, env.hist_cap)
    before = env.state[: total - 256].clone()
    got, _, bm, _, child = _expand_raw(env, p, a)
    assert got["err"].tolist() == [1] * 4
    assert got["reward"].tolist() == [0.0] * 4 and got["done"].tolist() == [0] * 4 and got["reason"].tolist() == [0] * 4
    assert got["winner"].tolist() == [-1] * 4 and got["ep_len"].tolist() == [0] * 4 and got["legal_count"].tolist() == [0] * 4
    assert int(bm.abs().sum()) == 0
    eb, _, em = _export(child, 4, 1)
    assert int(eb.abs().sum()) == 0 and em[:, 3].tolist() == [0] * 4 and em[:, 4].tolist() == [-1] * 4
    assert torch.equal(env.state[: total - 256], before)
    with pytest.raises(ValueError, match="parent"):
        env.expand(p[:1].contiguous(), a[:1].contiguous())


def test_expand_sennichite_on_exactly_the_repeating_move(golden_dir):
    from shogidrl_b200 import VecShogiEnv
    with np.load(os.path.join(golden_dir, "scripted.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    env = VecShogiEnv(1, max_moves_per_game=500, device=DEV, auto_reset=False)
    env.load_sfens([str(z["senn_sfen"])])
    acts = z["senn_actions"]
    for t in range(len(acts) - 1):  # one ply before the 4th repetition
        out = env.step(torch.tensor([int(acts[t])], device=DEV))
        assert int(out["done"][0]) == 0
    parent, actions = _items(env, np.random.default_rng(3), extra=False)
    out = env.expand(parent, actions)
    rep = actions == int(acts[-1])
    assert int(rep.sum()) == 1
    assert out["reason"][rep].tolist() == [4] and out["done"][rep].tolist() == [1]
    assert int((out["reason"][~rep] == 4).sum()) == 0
    _check_expansion(env, parent, actions, "sennichite")
    # the same move through kz_step ends the game by sennichite
    assert int(env.step(torch.tensor([int(acts[-1])], device=DEV))["reason"][0]) == 4


def test_expand_selfplay_snapshots():
    """4,096 random self-play games, sampled every 50 plies up to 400: every legal action plus rejected ones."""
    from shogidrl_b200 import VecShogiEnv
    env = VecShogiEnv(4096, max_moves_per_game=500, device=DEV, seed=11, auto_reset=True)
    env.refresh(random_actions=True)
    rng = np.random.default_rng(9)
    for ply in range(401):
        if ply % 50 == 0:
            parent, actions = _items(env, rng)
            assert int(parent.numel()) > 4096 * 30, ply  # 30 at the start position, more later, + 3 rejected per game
            _check_expansion(env, parent, actions, f"selfplay ply {ply}")
        env.step(env.next_actions.clone(), random_actions=True)


def test_legal_actions_and_short_offsets(golden_dir):
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200 import _native as nv
    from shogidrl_b200 import rl
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        sfens = [str(s) for s in zf["sfens"]]
    env = VecShogiEnv(len(sfens), max_moves_per_game=500, device=DEV, auto_reset=False)
    env.load_sfens(sfens)
    offsets, parent, actions = env.legal_actions()
    bitmap = torch.zeros((env.n, 448), dtype=torch.int32, device=DEV)
    env.legal_bitmap(bitmap)
    mask = rl.bitmap_to_mask(bitmap).view(torch.uint8).cpu().numpy()
    off, par, act = offsets.cpu().numpy(), parent.cpu().numpy(), actions.cpu().numpy()
    assert off[0] == 0 and off[-1] == len(act) == int(env.legal_count.sum())
    for g in range(env.n):
        assert np.array_equal(act[off[g]:off[g + 1]], np.nonzero(mask[g])[0]), g
        assert (par[off[g]:off[g + 1]] == g).all()
    # offsets that disagree with the bitmap: every row writes only inside its own range
    cnt = np.diff(off)
    short = np.concatenate([[0], np.cumsum(np.where(np.arange(env.n) % 2 == 0, cnt // 2, cnt + 3))]).astype(np.int64)
    so = torch.as_tensor(short, device=DEV)
    out_a = torch.full((int(short[-1]),), -7, dtype=torch.int32, device=DEV)
    out_p = torch.full((int(short[-1]),), -7, dtype=torch.int32, device=DEV)
    nv.check(nv.lib().kz_legal_list(bitmap.data_ptr(), 448, env.n, so.data_ptr(), out_p.data_ptr(), out_a.data_ptr(), 0,
                                    torch.cuda.current_stream().cuda_stream), "kz_legal_list")
    oa, op = out_a.cpu().numpy(), out_p.cpu().numpy()
    for g in range(env.n):
        seg, segp = oa[short[g]:short[g + 1]], op[short[g]:short[g + 1]]
        k = min(cnt[g], short[g + 1] - short[g])
        assert np.array_equal(seg[:k], act[off[g]:off[g] + k]) and (segp[:k] == g).all(), g
        assert (seg[k:] == -7).all() and (segp[k:] == -7).all(), g


HIRATE = [30, 900, 25470, 719731, 19861490]


def test_perft_hirate():
    from shogidrl_b200.perft import perft
    g = orc.OracleGame(max_moves=65535)
    for d, want in enumerate(HIRATE, start=1):
        got = perft(depth=d)
        assert got == [want], (d, got)
        if d <= 4:
            assert perft_ref.perft(None, d) == want
    div = perft(depth=3, divide=True)[0]
    assert div == perft_ref.perft(None, 3, divide=True)
    assert perft(depth=1, divide=True)[0] == {a: 1 for a in g.legal_indices().tolist()}


def _oracle_divide(sfen, depth):
    return perft_ref.perft(sfen, depth, divide=True)


def test_perft_divide_vs_oracle(golden_dir):
    from shogidrl_b200.perft import perft
    with np.load(os.path.join(golden_dir, "kat_positions.npz")) as zf:
        kat = [str(s) for s in zf["sfens"]]
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        end = [str(s) for s in zf["sfens"]]
    sfens = kat + end
    got = perft(sfens, 3, divide=True)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:  # the oracle's ctypes calls release the GIL
        want = list(ex.map(lambda s: _oracle_divide(s, 3), sfens))
    for s, a, b in zip(sfens, got, want):
        assert a == b, s
    assert perft(sfens, 2) == [sum(d.values()) for d in (_oracle_divide(s, 2) for s in sfens)]


def test_perft_chunked_equals_unchunked(golden_dir):
    from shogidrl_b200.perft import perft
    with np.load(os.path.join(golden_dir, "traces_endgame.npz")) as zf:
        end = [str(s) for s in zf["sfens"]][:16]
    roots = [None, end]
    for r in roots:
        assert perft(r, 4, max_items=4096) == perft(r, 4)
        assert perft(r, 3, divide=True, max_items=4096) == perft(r, 3, divide=True)
