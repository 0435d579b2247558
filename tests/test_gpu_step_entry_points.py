"""kz_step and kz_step_rollout, the whole-batch step entry points that INTEGRATION.md tells outside hosts to bind.
VecShogiEnv launches kz_step_range / kz_step_pool, so nothing in the package calls these two: they are pinned here by
raw ctypes calls against VecShogiEnv on twin batches."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n", [1000, 4096])
def test_whole_batch_entry_points_match_vec_env(n):
    """Twin batches, max_moves 60 and 72 plies, so that every game auto-resets; 1,000 games take the static-stride launch,
    4,096 the tile-claiming one.  Batch a steps through VecShogiEnv.step, b through kz_step; c through
    VecShogiEnv.step_rollout, d through kz_step_rollout (every third step without observation rows).  Rows, scalars,
    next actions and the exported state agree at every step."""
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200 import _native as nv

    dev = torch.device("cuda:0")
    T, seed = 72, 23
    a, b, c, d = (VecShogiEnv(n, max_moves_per_game=60, device=dev, seed=seed) for _ in range(4))
    L, sp = nv.lib(), nv.stream_ptr(dev)
    acts = [[torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)] for _ in range(4)]
    for e, x in zip((a, b, c, d), acts):
        e.refresh(random_actions=True, next_out=x[0])
    bm_c, bm_d = (torch.zeros((n, 448), dtype=torch.int32, device=dev) for _ in range(2))
    cobs_c, cobs_d = (torch.zeros((n, 40), dtype=torch.int32, device=dev) for _ in range(2))
    for t in range(T):
        cur, nxt = t & 1, (t + 1) & 1
        a.obs.fill_(-1.0); b.obs.fill_(-2.0); c.obs.fill_(-3.0); d.obs.fill_(-4.0)
        a._mask_store.fill_(5); b._mask_store.fill_(7); bm_c.fill_(-1); bm_d.fill_(-2)
        oa = a.step(acts[0][cur], random_actions=True, next_out=acts[0][nxt])
        nv.check(L.kz_step(b.state.data_ptr(), n, b.hist_cap, acts[1][cur].data_ptr(), 1, b.obs.data_ptr(), nv.OBS_FLOATS,
                           b._mask_store.data_ptr(), nv.MASK_PAD_STRIDE, b.reward.data_ptr(), b.done.data_ptr(),
                           b.reason.data_ptr(), b.winner.data_ptr(), b.ep_len.data_ptr(), b.legal_count.data_ptr(),
                           acts[1][nxt].data_ptr(), seed, t + 1, 0, 1, sp), "kz_step")
        with_obs = t % 3 != 2
        oc = c.step_rollout(acts[2][cur], c.obs if with_obs else None, bm_c, random_actions=True, next_out=acts[2][nxt],
                            cobs=cobs_c)
        nv.check(L.kz_step_rollout(d.state.data_ptr(), n, d.hist_cap, acts[3][cur].data_ptr(), 1,
                                   d.obs.data_ptr() if with_obs else None, nv.OBS_FLOATS, bm_d.data_ptr(), 448,
                                   cobs_d.data_ptr(), d.reward.data_ptr(), d.done.data_ptr(), d.reason.data_ptr(),
                                   d.winner.data_ptr(), d.ep_len.data_ptr(), d.legal_count.data_ptr(),
                                   acts[3][nxt].data_ptr(), seed, t + 1, 0, 1, sp), "kz_step_rollout")
        assert torch.equal(a.obs, b.obs) and torch.equal(a.mask, b.mask), t
        assert torch.equal(bm_c, bm_d) and torch.equal(cobs_c, cobs_d), t
        if with_obs:
            assert torch.equal(c.obs, d.obs) and torch.equal(c.obs, a.obs), t
        for k in ("reward", "done", "reason", "winner", "ep_len", "legal_count"):
            assert torch.equal(oa[k], getattr(b, k)) and torch.equal(oc[k], getattr(d, k)), (t, k)
            assert torch.equal(oa[k], oc[k]), (t, k)
        for x in acts[1:]:
            assert torch.equal(x[nxt], acts[0][nxt]), t
        ea, ec = a.export(), c.export()
        assert all(torch.equal(x, y) for x, y in zip(ea, b.export())), t
        assert all(torch.equal(x, y) for x, y in zip(ec, d.export())), t
        assert all(torch.equal(x, y) for x, y in zip(ea, ec)), t
    assert bool((a.export()[2][:, 7] >= 1).all())  # every game has finished and restarted at least once
    for e in (a, b, c, d):
        assert int(e.errors().abs().sum()) == 0
