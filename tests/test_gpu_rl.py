"""GPU tests of kz_sample_masked and kz_gae through the C ABI (shogidrl_b200.rl)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as orc  # noqa: E402  (checker only)

A = 13527


def _torch_reference(logits, mask):
    """base_actor_critic.py:64-116 in plain fp32 torch."""
    masked = torch.where(mask.bool(), logits.float(), torch.tensor(float("-inf"), device=logits.device))
    probs = torch.softmax(masked, dim=-1)
    nan_rows = torch.isnan(probs).any(dim=1, keepdim=True)
    probs = torch.where(nan_rows, torch.full_like(probs, 1.0 / A), probs)  # out of place: keeps autograd usable
    return probs, torch.distributions.Categorical(probs=probs)


def _random_case(n, dev, seed=0, legal_p=0.004):
    g = torch.Generator(device="cpu").manual_seed(seed)
    logits = (torch.randn(n, A, generator=g) * 3).to(dev)
    mask = (torch.rand(n, A, generator=g) < legal_p).to(dev)
    mask[:, 17] |= ~mask.any(dim=1)
    return logits, mask


def test_sample_support_and_logprob():
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    logits, mask = _random_case(512, dev)
    act, logp, ent = rl.sample_masked(logits, mask, seed=3, offset=11, want_entropy=True)
    assert bool(mask.gather(1, act[:, None]).all())
    probs, dist = _torch_reference(logits, mask)
    ref_lp = dist.log_prob(act)
    # fp32 softmax; tolerance 1e-5 relative (+1e-6 absolute) on log-probabilities and entropy
    assert torch.allclose(logp, ref_lp, rtol=1e-5, atol=1e-6), float((logp - ref_lp).abs().max())
    assert torch.allclose(ent, dist.entropy(), rtol=1e-5, atol=1e-5), float((ent - dist.entropy()).abs().max())


def test_sample_deterministic_is_argmax():
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    logits, mask = _random_case(256, dev, seed=1)
    act, logp, _ = rl.sample_masked(logits, mask, deterministic=True)
    probs, dist = _torch_reference(logits, mask)
    assert torch.equal(act, torch.argmax(probs, dim=-1))
    assert torch.allclose(logp, dist.log_prob(act), rtol=1e-5, atol=1e-6)


def test_sample_single_legal_and_all_illegal():
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    logits = torch.randn(4, A, device=dev)
    mask = torch.zeros(4, A, dtype=torch.bool, device=dev)
    mask[0, 5] = True
    mask[1, A - 1] = True
    act, logp, _ = rl.sample_masked(logits, mask, seed=9)
    assert int(act[0]) == 5 and int(act[1]) == A - 1
    eps = torch.finfo(torch.float32).eps
    assert abs(float(logp[0]) - float(np.log(np.float32(1.0) - np.float32(eps)))) < 1e-9
    # all-illegal rows: uniform over all actions (base_actor_critic.py:93-101)
    assert 0 <= int(act[2]) < A and abs(float(logp[2]) - float(np.log(1.0 / A))) < 1e-5


def test_sample_bf16_and_strided_mask():
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    logits, mask = _random_case(128, dev, seed=2)
    lb = logits.to(torch.bfloat16)
    store = torch.zeros(128, 13536, dtype=torch.uint8, device=dev)
    store[:, :A] = mask
    act, logp, _ = rl.sample_masked(lb, store[:, :A], seed=5)
    assert bool(mask.gather(1, act[:, None]).all())
    _, dist = _torch_reference(lb.float(), mask)
    assert torch.allclose(logp, dist.log_prob(act), rtol=1e-5, atol=1e-6)


def test_sample_frequencies_chi2():
    """Statistical parity with the masked softmax: chi-square on 160k draws over 12 legal actions."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    legal = torch.tensor([3, 40, 41, 999, 5000, 5001, 8191, 8192, 12959, 12960, 13000, 13526], device=dev)
    row = torch.randn(A, device=dev)
    row[legal] = torch.linspace(-1.5, 2.0, len(legal), device=dev)
    n = 16000
    logits = row[None].expand(n, A).contiguous()
    mask = torch.zeros(n, A, dtype=torch.bool, device=dev)
    mask[:, legal] = True
    counts = torch.zeros(A, device=dev)
    for rep in range(10):
        act, _, _ = rl.sample_masked(logits, mask, seed=77, offset=rep * n)
        counts += torch.bincount(act, minlength=A).float()
    assert float(counts.sum()) == 10 * n and float(counts[legal].sum()) == 10 * n
    p = torch.softmax(row[legal], 0)
    expected = p * 10 * n
    chi2 = float((((counts[legal] - expected) ** 2) / expected).sum())
    assert chi2 < 40.0, chi2  # 11 dof: P(chi2 > 40) ~ 4e-5


def test_gae_golden_and_oracle(golden_dir):
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    with np.load(os.path.join(golden_dir, "gae_golden.npz")) as zf:
        z = {k: zf[k] for k in zf.files}
    for i in range(int(z["n_cases"])):
        r = torch.as_tensor(z[f"c{i}_r"][:, None]).to(dev)
        v = torch.as_tensor(z[f"c{i}_v"][:, None]).to(dev)
        d = torch.as_tensor(z[f"c{i}_d"][:, None]).to(dev)
        lv = torch.tensor([float(z[f"c{i}_last"])], device=dev)
        gamma, lam = float(z[f"c{i}_gamma"]), float(z[f"c{i}_lam"])
        adv, ret = rl.gae(r, v, d, lv, gamma, lam, exact=True)  # column kernel: bit-exact with the reference
        assert np.array_equal(adv[:, 0].cpu().numpy(), z[f"c{i}_adv"]), i
        assert np.array_equal(ret[:, 0].cpu().numpy(), z[f"c{i}_ret"]), i
        adv2, ret2 = rl.gae(r, v, d, lv, gamma, lam)             # narrow -> warp-scan kernel: 1e-5 relative
        scale = max(1.0, float(np.abs(z[f"c{i}_adv"]).max()))
        assert float((adv2[:, 0].cpu() - torch.as_tensor(z[f"c{i}_adv"])).abs().max()) <= 1e-5 * scale, i
        assert float((ret2[:, 0].cpu() - torch.as_tensor(z[f"c{i}_ret"])).abs().max()) <= 1e-5 * scale, i
    # wide rollout: [T=128, N=4096] against the oracle, bit-exact
    g = torch.Generator(device="cpu").manual_seed(5)
    T, N = 128, 4096
    r = torch.randn(T, N, generator=g); v = torch.randn(T, N, generator=g)
    d = torch.rand(T, N, generator=g) < 0.03
    lv = torch.randn(N, generator=g)
    adv, ret = rl.gae(r.to(dev), v.to(dev), d.to(dev), lv.to(dev), 0.99, 0.95)
    a_ref, r_ref = orc.gae(r.numpy(), v.numpy(), d.numpy(), lv.numpy(), 0.99, 0.95)
    assert np.array_equal(adv.cpu().numpy(), a_ref) and np.array_equal(ret.cpu().numpy(), r_ref)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fused_evaluate_matches_torch_forward_and_backward(dtype):
    """rl.evaluate_masked (kz_eval_masked_fwd/bwd) against the PyTorch formulation of evaluate_actions
    (base_actor_critic.py:118-184): log-probs, entropy and the gradient w.r.t. the logits."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    n = 192
    logits, mask = _random_case(n, dev, seed=4, legal_p=0.003)
    mask[5] = False            # a row without legal actions: uniform fallback, zero gradient
    mask[6] = False; mask[6, 77] = True   # single legal action: p = 1 -> clamp saturates, zero log-prob gradient
    logits = logits.to(dtype).float()
    actions = torch.stack([torch.nonzero(mask[i])[0, 0] if mask[i].any() else torch.tensor(3, device=dev) for i in range(n)])
    w_lp = torch.randn(n, device=dev); w_ent = torch.randn(n, device=dev)

    ref_in = logits.clone().requires_grad_()
    probs, dist = _torch_reference(ref_in, mask)
    ref_lp, ref_ent = dist.log_prob(actions), dist.entropy()
    ((ref_lp * w_lp).sum() + (ref_ent * w_ent).sum()).backward()

    # padded storage + row indirection, as PPOAgent.learn uses it
    store = torch.zeros(2 * n, 13536, dtype=torch.uint8, device=dev)
    rows = torch.randperm(2 * n, device=dev)[:n]
    store[rows, :A] = mask.to(torch.uint8)
    x = logits.to(dtype).clone().requires_grad_()
    lp, ent = rl.evaluate_masked(x, store[:, :A], actions, mask_rows=rows)
    ((lp * w_lp).sum() + (ent * w_ent).sum()).backward()
    assert torch.allclose(lp, ref_lp, rtol=1e-5, atol=2e-6), float((lp - ref_lp).abs().max())
    assert torch.allclose(ent, ref_ent, rtol=1e-5, atol=1e-5), float((ent - ref_ent).abs().max())
    g, g_ref = x.grad.float(), ref_in.grad
    tol = 1e-5 if dtype == torch.float32 else 1e-2  # bf16 gradients are rounded to 8 bits of mantissa
    assert torch.allclose(g, g_ref, rtol=tol, atol=tol * 0.1), float((g - g_ref).abs().max())
    assert float(g[5].abs().max()) == 0.0 and bool((g[~mask.bool()] == 0).all())


@pytest.mark.parametrize("legal_p", [0.25, 1.0])
def test_dense_masks_take_the_multi_piece_path(legal_p):
    """Masks far denser than any Shogi position overflow the per-row compaction list and are consumed in
    pieces; unaligned rows (row stride 13527) exercise the byte-assembled edge windows.  Same law, same numbers."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    n = 96
    logits, mask = _random_case(n, dev, seed=9, legal_p=legal_p)
    assert mask.stride(0) == A  # rows start at every alignment mod 16
    act, logp, ent = rl.sample_masked(logits, mask, seed=5, offset=0, want_entropy=True)
    assert bool(mask.gather(1, act[:, None]).all())
    probs, dist = _torch_reference(logits, mask)
    assert torch.allclose(logp, dist.log_prob(act), rtol=1e-5, atol=2e-6)
    assert torch.allclose(ent, dist.entropy(), rtol=1e-5, atol=1e-5)
    det, _, _ = rl.sample_masked(logits, mask, deterministic=True)
    assert torch.equal(det, torch.argmax(probs, dim=-1))
    # fused evaluation, forward and backward
    w_lp = torch.randn(n, device=dev); w_ent = torch.randn(n, device=dev)
    ref_in = logits.clone().requires_grad_()
    _, rdist = _torch_reference(ref_in, mask)
    ((rdist.log_prob(act) * w_lp).sum() + (rdist.entropy() * w_ent).sum()).backward()
    x = logits.clone().requires_grad_()
    lp, e2 = rl.evaluate_masked(x, mask, act)
    ((lp * w_lp).sum() + (e2 * w_ent).sum()).backward()
    assert torch.allclose(lp, rdist.log_prob(act).detach(), rtol=1e-5, atol=2e-6)
    assert torch.allclose(e2, rdist.entropy().detach(), rtol=1e-5, atol=1e-5)
    assert torch.allclose(x.grad, ref_in.grad, rtol=1e-4, atol=1e-6), float((x.grad - ref_in.grad).abs().max())


def test_dense_mask_sampling_law():
    """Inverse-CDF over a 2,000-entry support (several list pieces per lane): empirical frequencies of the 20
    heaviest actions match the softmax within 5 sigma."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(21)
    row_logits = (torch.randn(A, generator=g) * 2).to(dev)
    row_mask = torch.zeros(A, dtype=torch.bool, device=dev)
    row_mask[torch.randperm(A, generator=g)[:6000].to(dev)] = True
    n = 65536
    logits = row_logits.expand(n, A).contiguous()
    mask = row_mask.expand(n, A).contiguous()
    act, _, _ = rl.sample_masked(logits, mask, seed=123, offset=0)
    probs, _ = _torch_reference(logits[:1], mask[:1])
    top = torch.topk(probs[0], 20).indices
    freq = torch.bincount(act, minlength=A).float() / n
    sigma = torch.sqrt(probs[0, top] * (1 - probs[0, top]) / n)
    assert bool(((freq[top] - probs[0, top]).abs() < 5 * sigma + 1e-6).all())


def _conv_case(n, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    obs = torch.rand(n, 46, 9, 9, generator=g)
    obs[:, :28] = (obs[:, :28] < 0.05).float()          # piece planes are 0/1, like real observations
    w = torch.randn(16, 46, 3, 3, generator=g) * 0.05
    b = torch.randn(16, generator=g) * 0.1
    return obs.cuda(), w.cuda(), b.cuda()


@pytest.mark.parametrize("n", [1, 37, 1500])
@pytest.mark.parametrize("relu", [True, False])
def test_obs_conv_forward_and_weight_gradient(n, relu):
    """kz_obs_conv_fwd / kz_obs_conv_wgrad against an fp64 convolution of the bf16-rounded operands (what bf16
    autocast feeds cuDNN): outputs within one bf16 rounding, weight / bias gradients within 1e-4 of their scale."""
    from shogidrl_b200 import nn_ops
    import torch.nn.functional as F
    obs, w, b = _conv_case(n, seed=n)
    wp, bp = w.clone().requires_grad_(), b.clone().requires_grad_()
    y = nn_ops.obs_conv(obs, wp, bp, relu=relu)
    assert y.dtype == torch.bfloat16 and y.shape == (n, 16, 9, 9)
    xd, wd, bd = obs.bfloat16().double(), w.bfloat16().double().requires_grad_(), b.bfloat16().double().requires_grad_()
    pre = F.conv2d(xd, wd, bd, padding=1)
    ref = pre.relu() if relu else pre
    err = (y.double() - ref).abs()
    assert bool((err <= ref.abs() * 2.0 ** -8 + 1e-3).all()), float(err.max())
    g = torch.Generator(device="cpu").manual_seed(5)
    dy = torch.randn(n, 16, 9, 9, generator=g).cuda()
    for dyk in (dy.bfloat16(), dy):
        wp.grad = bp.grad = None
        y2 = nn_ops.obs_conv(obs, wp, bp, relu=relu)
        y2.backward(dyk.to(y2.dtype) if dyk.dtype == torch.bfloat16 else dyk)
        # reference: the ReLU gate of the kernel's own (bf16) output, dy rounded to bf16
        gate = (y2.double() > 0) if relu else torch.ones_like(pre, dtype=torch.bool)
        dyd = torch.where(gate, dyk.bfloat16().double(), torch.zeros((), dtype=torch.float64, device="cuda"))
        gw, gb = torch.autograd.grad(pre, (wd, bd), dyd, retain_graph=True)
        assert float((wp.grad.double() - gw).abs().max()) <= 1e-4 * float(gw.abs().max()) + 1e-6
        assert float((bp.grad.double() - gb).abs().max()) <= 1e-4 * float(gb.abs().max()) + 1e-6


def test_actor_critic_uses_fused_input_layer_under_autocast():
    """Default CNN under bf16 autocast: fused input layer vs the cuDNN path -- same logits/values within bf16
    noise, same parameter gradients within 2 %."""
    from shogidrl_b200.core import ActorCritic
    from shogidrl_b200 import nn_ops
    torch.manual_seed(0)
    model = ActorCritic(46, A).cuda()
    obs, _, _ = _conv_case(64, seed=3)
    outs = []
    for fused in (True, False):
        model.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            assert nn_ops.obs_conv_applicable(model.conv, obs)
            if fused:
                logits, value = model(obs)
            else:
                x = model.flatten(model.relu(model.conv(obs)))
                logits, value = model.policy_head(x), model.value_head(x)
        (logits.float().square().mean() + value.float().square().mean()).backward()
        outs.append((logits.float().detach().clone(), value.float().detach().clone(), model.conv.weight.grad.clone(),
                     model.conv.bias.grad.clone()))
    (l1, v1, gw1, gb1), (l2, v2, gw2, gb2) = outs
    assert torch.allclose(l1, l2, rtol=2e-2, atol=2e-2) and torch.allclose(v1, v2, rtol=2e-2, atol=2e-2)
    assert float((gw1 - gw2).abs().max()) <= 2e-2 * float(gw2.abs().max())
    assert float((gb1 - gb2).abs().max()) <= 2e-2 * float(gb2.abs().max())


def test_fused_minibatch_forward_matches_unfused_path():
    """ActorCritic.forward(obs_store, rows=, actions=, legal_mask=, mask_rows=) -- the PPO update's in-place
    minibatch evaluation -- against gather + forward + evaluate_from_logits: same log-probs / entropy / value and
    the same gradients for every parameter (bf16 tolerances)."""
    from shogidrl_b200.core import ActorCritic
    torch.manual_seed(1)
    dev = torch.device("cuda:0")
    model = ActorCritic(46, A).to(dev)
    store_n, n = 300, 128
    obs, _, _ = _conv_case(store_n, seed=8)
    _, mask = _random_case(store_n, dev, seed=12)
    mask_store = torch.zeros(store_n, 13536, dtype=torch.uint8, device=dev)
    mask_store[:, :A] = mask
    rows = torch.randperm(store_n, device=dev)[:n]
    actions = torch.stack([torch.nonzero(mask[i])[0, 0] for i in rows.tolist()])
    w_lp, w_ent, w_v = torch.randn(n, device=dev), torch.randn(n, device=dev) * 0.1, torch.randn(n, device=dev)
    results = []
    for fused in (True, False):
        model.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if fused:
                lp, ent, v = model(obs, rows=rows, actions=actions, legal_mask=mask_store[:, :A], mask_rows=rows)
            else:
                x = model.flatten(model.relu(model.conv(obs[rows])))
                logits, value = model.policy_head(x), model.value_head(x)
                lp, ent, v = ActorCritic.evaluate_from_logits(logits, value, actions, mask[rows])
        ((lp * w_lp).sum() + (ent * w_ent).sum() + (v.float() * w_v).sum()).backward()
        results.append((lp.detach().clone(), ent.detach().clone(), v.float().detach().clone(),
                        {k: p.grad.clone() for k, p in model.named_parameters()}))
    (lp1, e1, v1, g1), (lp2, e2, v2, g2) = results
    assert torch.allclose(lp1, lp2, rtol=2e-2, atol=2e-2), float((lp1 - lp2).abs().max())
    assert torch.allclose(e1, e2, rtol=2e-2, atol=2e-2) and torch.allclose(v1, v2, rtol=2e-2, atol=2e-2)
    for k in g1:
        scale = float(g2[k].abs().max())
        assert float((g1[k] - g2[k]).abs().max()) <= 3e-2 * scale + 1e-6, (k, float((g1[k] - g2[k]).abs().max()), scale)


@pytest.mark.parametrize("n", [7, 1024, 16384])
def test_fused_ppo_loss_matches_torch(n):
    """kz_ppo_loss against the reference formulas (ppo_agent.py:332-372) written in torch: loss, the five
    metrics and the gradients w.r.t. new log-probs / entropy / values, with ratios on both sides of the clip range."""
    from shogidrl_b200 import rl
    g = torch.Generator(device="cpu").manual_seed(n)
    old_lp = (-torch.rand(n, generator=g) * 5).cuda()
    new_lp = (old_lp.cpu() + torch.randn(n, generator=g) * 0.3).cuda().requires_grad_()
    ent = (torch.rand(n, generator=g) * 4).cuda().requires_grad_()
    new_v = torch.randn(n, generator=g).cuda().requires_grad_()
    adv, ret = torch.randn(n, generator=g).cuda(), torch.randn(n, generator=g).cuda()
    adv[::5] = 0.0
    eps, cv, ce, scale = 0.2, 0.5, 0.01, 0.5
    loss, stats = rl.ppo_loss(new_lp, ent, new_v, old_lp, adv, ret, eps, cv, ce, scale)
    loss.backward()
    got = [t.grad.clone() for t in (new_lp, ent, new_v)]
    for t in (new_lp, ent, new_v):
        t.grad = None
    ratio = torch.exp(new_lp - old_lp)
    pol = -torch.min(ratio * adv, torch.clamp(ratio, 1 - eps, 1 + eps) * adv).mean()
    val = torch.nn.functional.mse_loss(new_v, ret)
    el = -ent.mean()
    ref = pol + cv * val + ce * el
    (ref * scale).backward()
    assert torch.allclose(loss, ref, rtol=1e-5, atol=1e-6)
    want = torch.stack([ref, pol, val, el, (old_lp - new_lp).mean(), ((ratio - 1).abs() > eps).float().mean()]).detach()
    assert torch.allclose(stats, want, rtol=1e-5, atol=1e-6), (stats, want)
    for a, t in zip(got, (new_lp, ent, new_v)):
        assert torch.allclose(a, t.grad, rtol=1e-5, atol=1e-9), float((a - t.grad).abs().max())


_ADAM_SHAPES = [(1353, 129), (16, 46, 3, 3), (4096,), (7,), (1,), (3, 4099), (32, 24, 3, 3)]
# 40 non-empty tensors = three launch groups of 16 / 16 / 8 (numel around the 4,096-element per-CTA chunk), plus a
# zero-element tensor (left out of the groups) and, last, a parameter that gets no gradient
_ADAM_GROUPS = [(4095,), (4096,), (4097,), (0,)] + [(37 * k + 1,) for k in range(30)] + \
    [(64, 65), (4095,), (4097,), (3, 4096), (5, 7), (1,), (4096, 2)]


@pytest.mark.parametrize("weight_decay,max_norm,shapes,no_grad", [
    pytest.param(0.0, 0.5, _ADAM_SHAPES, False, id="0.0-0.5"),
    pytest.param(0.01, 0.5, _ADAM_SHAPES, False, id="0.01-0.5"),
    pytest.param(0.0, 1e9, _ADAM_SHAPES, False, id="0.0-1000000000.0"),
    pytest.param(0.01, 0.5, _ADAM_GROUPS, True, id="three_groups"),
])
def test_fused_clip_adam_matches_torch(weight_decay, max_norm, shapes, no_grad):
    """kz_adam_clip_step against torch.nn.utils.clip_grad_norm_ + torch.optim.Adam(capturable) (ppo_agent.py:405-413)
    over several steps on tensors of ragged sizes (vector body, scalar tails, a 1-element tensor; or several launch
    groups with an empty tensor and one without a gradient): parameters, both moments, the step counters and the
    reported gradient norm.  fp32 tolerance 1e-5 relative."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(5)
    shapes = shapes + [(300,)] if no_grad else shapes
    base = [torch.randn(s, generator=g) for s in shapes]
    pa = [torch.nn.Parameter(b.clone().to(dev)) for b in base]
    pb = [torch.nn.Parameter(b.clone().to(dev)) for b in base]
    # the last tensor lives in channels_last memory (the ResNet tower's convolution weights) and gets default-layout
    # gradients: the fused tail pairs elements by their logical index, not by their position in the storage
    if len(shapes[-1]) == 4:
        pa[-1].data = pa[-1].data.contiguous(memory_format=torch.channels_last)
        assert not pa[-1].is_contiguous()
    kw = dict(lr=3e-4, weight_decay=weight_decay, capturable=True)
    oa, ob = torch.optim.Adam(pa, **kw), torch.optim.Adam(pb, **kw)
    assert rl.adam_clip_applicable(oa)
    for it in range(6):
        grads = [torch.randn(s, generator=g) * (10.0 if it % 2 else 0.01) for s in shapes]  # clipped and unclipped steps
        for p, q, gr in zip(pa[:len(pa) - no_grad], pb, grads):
            p.grad = gr.clone().to(dev)
            q.grad = gr.clone().to(dev)
        gn_a = rl.adam_clip_step(oa, max_norm)
        gn_b = torch.nn.utils.clip_grad_norm_(pb, max_norm=max_norm)
        ob.step()
        assert torch.allclose(gn_a, gn_b, rtol=1e-5), (float(gn_a), float(gn_b))
        for p, q in zip(pa, pb):
            assert torch.allclose(p, q, rtol=1e-5, atol=1e-7), (it, tuple(p.shape), float((p - q).abs().max()))
            if p.grad is None:
                assert len(oa.state[p]) == len(ob.state[q]) == 0 and torch.equal(p, q)
                continue
            sa, sb = oa.state[p], ob.state[q]
            assert float(sa["step"]) == float(sb["step"]) == it + 1
            assert torch.allclose(sa["exp_avg"], sb["exp_avg"], rtol=1e-5, atol=1e-9)
            assert torch.allclose(sa["exp_avg_sq"], sb["exp_avg_sq"], rtol=1e-5, atol=1e-12)
    # the state is torch's own: the stock optimizer continues from it, and a state_dict round trip keeps it
    sd = oa.state_dict()
    oc = torch.optim.Adam(pa, **kw)
    oc.load_state_dict(sd)
    assert float(oc.state[pa[0]]["step"]) == 6 and torch.equal(oc.state[pa[0]]["exp_avg"], oa.state[pa[0]]["exp_avg"])


def test_fused_clip_adam_rejects_what_it_cannot_mirror():
    from shogidrl_b200 import rl
    p = [torch.nn.Parameter(torch.zeros(8, device="cuda"))]
    assert rl.adam_clip_applicable(torch.optim.Adam(p, lr=1e-3))
    assert not rl.adam_clip_applicable(torch.optim.Adam(p, lr=1e-3, amsgrad=True))
    assert not rl.adam_clip_applicable(torch.optim.AdamW(p, lr=1e-3))
    assert not rl.adam_clip_applicable(torch.optim.SGD(p, lr=1e-3))
    assert not rl.adam_clip_applicable(torch.optim.Adam([{"params": p}, {"params": [torch.nn.Parameter(torch.zeros(2, device="cuda"))]}], lr=1e-3))


# ------------------------------------------------------------------------------------------------
# legal sets as the engine's 13,527-bit bitmap rows (kz_sample_bitmap, kz_eval_bitmap_*, kz_bitmap_expand)
def _pack_bitmap(mask):
    """bool [n, 13527] -> int32 [n, 448] (bit i of a row = action i), on the mask's device."""
    n = mask.shape[0]
    padded = torch.zeros((n, 448 * 32), dtype=torch.int64, device=mask.device)
    padded[:, :A] = mask.long()
    words = (padded.view(n, 448, 32) << torch.arange(32, device=mask.device)).sum(-1)
    return (words & 0xFFFFFFFF).to(torch.int64).where(words < 2 ** 31, words - 2 ** 32).to(torch.int32).contiguous()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("legal_p", [0.004, 0.3])
def test_bitmap_rows_equal_byte_mask_rows(dtype, legal_p):
    """The bitmap entry points return, bit for bit, what the byte-mask entry points return for 16-byte aligned rows of
    the same legal sets: sampled actions, arg-max actions, log-probs, entropies, dlogits and the bias gradient; and
    both stay within 1e-5 of the fp32 torch formulation."""
    from shogidrl_b200 import rl, nn_ops
    dev = torch.device("cuda:0")
    n = 777
    logits, mask = _random_case(n, dev, seed=5, legal_p=legal_p)
    mask[3] = False  # an all-illegal row (uniform fallback) in both encodings
    mask[5] = False; mask[5, A - 1] = True  # the last action only
    logits = logits.to(dtype)
    store = torch.zeros((n, 13536), dtype=torch.uint8, device=dev)  # aligned rows, as the engine writes them
    store[:, :A] = mask
    bytes_ = store[:, :A]
    bm = _pack_bitmap(mask)
    assert torch.equal(rl.bitmap_to_mask(bm), mask)
    rows = torch.randperm(n, device=dev)[:100]
    assert torch.equal(rl.bitmap_to_mask(bm, rows), mask[rows])
    odd = torch.zeros((n, A + 3), dtype=torch.bool, device=dev)[:, 1:A + 1]  # unaligned destination rows
    assert torch.equal(rl.bitmap_to_mask(bm, out=odd), mask)
    for det in (False, True):
        a1, l1, e1 = rl.sample_masked(logits, bytes_, seed=9, offset=4, deterministic=det, want_entropy=True)
        a2, l2, e2 = rl.sample_masked(logits, bm, seed=9, offset=4, deterministic=det, want_entropy=True)
        assert torch.equal(a1, a2) and torch.equal(l1, l2) and torch.equal(e1, e2)
    ok = mask.any(1)
    assert bool(mask[ok].gather(1, a2[ok, None]).all())
    # evaluation forward / backward
    lg1 = logits.clone().requires_grad_(True)
    lg2 = logits.clone().requires_grad_(True)
    act = a2.clone()
    lp1, en1 = rl.evaluate_masked(lg1, bytes_, act)
    lp2, en2 = rl.evaluate_masked(lg2, bm, act)
    assert torch.equal(lp1, lp2) and torch.equal(en1, en2)
    w = torch.randn(n, device=dev)
    (lp1 * w).sum().backward(retain_graph=True); (en1 * w * 0.3).sum().backward()
    (lp2 * w).sum().backward(retain_graph=True); (en2 * w * 0.3).sum().backward()
    assert torch.equal(lg1.grad, lg2.grad)
    if dtype == torch.float32:
        ref = logits.clone().requires_grad_(True)
        probs, dist = _torch_reference(ref, mask)
        assert torch.allclose(lp2, dist.log_prob(act), rtol=1e-5, atol=1e-6)
        assert torch.allclose(en2, dist.entropy(), rtol=1e-5, atol=1e-5)
    # through row indices into a larger storage, as the PPO update reads the rollout buffer
    perm = torch.randperm(n, device=dev)
    lp3, en3 = rl.evaluate_masked(logits[perm].contiguous(), bm, act[perm], mask_rows=perm)
    assert torch.equal(lp3, lp2[perm]) and torch.equal(en3, en2[perm])


def test_policy_head_bias_gradient_is_deterministic_and_matches_column_sums():
    """kz_eval_*_bwd accumulates the policy head's bias gradient in Q20.44 fixed point: identical bits run to run
    (an fp32 atomicAdd is not), equal for the byte-mask and bitmap forms, and equal to the column sums of dlogits."""
    from shogidrl_b200 import nn_ops
    dev = torch.device("cuda:0")
    n, k = 4096, 64
    g = torch.Generator(device="cpu").manual_seed(2)
    h = torch.randn(n, k, generator=g).to(dev).bfloat16()
    lin = torch.nn.Linear(k, A).to(dev)
    _, mask = _random_case(n, dev, seed=8, legal_p=0.01)
    store = torch.zeros((n, 13536), dtype=torch.uint8, device=dev)
    store[:, :A] = mask
    bm = _pack_bitmap(mask)
    act = torch.multinomial(mask.float(), 1).squeeze(1)
    wl = torch.randn(n, device=dev)
    grads = []
    for legal in (store[:, :A], bm, store[:, :A], bm):
        lin.zero_grad()
        lp, en = nn_ops.policy_head_evaluate(h, lin, legal, act)
        ((lp * wl).sum() + 0.01 * en.sum()).backward()
        grads.append((lin.bias.grad.clone(), lin.weight.grad.clone()))
    for b, w in grads[1:]:
        assert torch.equal(b, grads[0][0]) and torch.equal(w, grads[0][1])
    # against the dense formulation in fp32
    lin32 = torch.nn.Linear(k, A).to(dev)
    lin32.load_state_dict(lin.state_dict())
    logits = torch.nn.functional.linear(h.float(), lin32.weight.bfloat16().float(), lin32.bias.bfloat16().float())
    logits = logits.detach().bfloat16().float().requires_grad_(True)
    probs, dist = _torch_reference(logits, mask)
    ((dist.log_prob(act) * wl).sum() + 0.01 * dist.entropy().sum()).backward()
    ref_db = logits.grad.sum(0)
    assert torch.allclose(grads[0][0], ref_db, rtol=2e-3, atol=2e-3 * float(ref_db.abs().max()))


# ------------------------------------------------------------------------------------------------
# compact observations (kz_step_rollout's cobs output) and the input layer that reads them (kz_cobs_conv_*)
def test_compact_observation_is_the_observation():
    """The 160-byte compact observation the engine writes beside every observation row decodes to exactly that row
    (piece-plane index per square, rotated for White to move, + the 18 constant-plane values), across resets."""
    from tests.helpers import obs_from_cobs, rollout_positions
    obs, cobs = rollout_positions()
    assert torch.equal(obs_from_cobs(cobs), obs)
    assert bool((cobs.view(torch.uint8).reshape(-1, 160)[:, 81:84] == 0xFF).all())  # pad bytes of the square table
    side_black = obs[:, 42, 0, 0] == 1.0
    assert bool(side_black.any()) and bool((~side_black).any())  # both perspectives occur


@pytest.mark.parametrize("relu", [True, False])
def test_input_layer_from_compact_observations(relu):
    """kz_cobs_conv_fwd (sparse: nine weight look-ups per output + constant planes, no dense product) and
    kz_cobs_conv_wgrad (tensor-core tile patched from the compact observation) against the dense kernels reading the
    fp32 rows of the same positions and against torch's conv2d on bf16-rounded operands; rows gathered in place."""
    from shogidrl_b200 import nn_ops
    dev = torch.device("cuda:0")
    from tests.helpers import rollout_positions
    obs, cobs = rollout_positions(1024, 30)
    g = torch.Generator(device="cpu").manual_seed(4)
    w = (torch.randn(16, 46, 3, 3, generator=g) * 0.05).to(dev).requires_grad_(True)
    b = (torch.randn(16, generator=g) * 0.1).to(dev).requires_grad_(True)
    rows = torch.randperm(obs.shape[0], device=dev)[:5000]
    y_c = nn_ops.obs_conv(obs, w, b, relu=relu, rows=rows, cobs=cobs)
    y_d = nn_ops.obs_conv(obs, w, b, relu=relu, rows=rows)
    ref = torch.nn.functional.conv2d(obs[rows].bfloat16().float(), w.detach().bfloat16().float(), b.detach().bfloat16().float(), padding=1)
    ref = torch.relu(ref) if relu else ref
    scale = float(ref.abs().max())
    assert float((y_c.detach().float() - ref).abs().max()) <= 2.0 ** -7 * scale + 1e-3   # bf16 output rounding
    assert float((y_c.float() - y_d.float()).abs().max()) <= 2.0 ** -7 * scale + 1e-3
    assert float((y_c.float() - y_d.float()).abs().mean()) <= 1e-4 * scale           # almost always the same bf16 value
    dy = torch.randn(y_c.shape, generator=torch.Generator(device="cpu").manual_seed(5)).to(dev).bfloat16()
    gw_c, gb_c = torch.autograd.grad(y_c, (w, b), dy, retain_graph=True)
    gw_d, gb_d = torch.autograd.grad(y_d, (w, b), dy, retain_graph=True)
    # the two weight-gradient kernels multiply the same bf16 tiles: equal up to the order of the per-CTA partial sums
    assert torch.allclose(gw_c, gw_d, rtol=1e-4, atol=1e-4 * float(gw_d.abs().max()))
    assert torch.allclose(gb_c, gb_d, rtol=1e-4, atol=1e-4 * float(gb_d.abs().max()))
    # without row indices, and a batch smaller than one CTA wave
    y1 = nn_ops.obs_conv(obs[:37], w, b, relu=relu, cobs=cobs[:37].contiguous())
    assert float((y1.float() - nn_ops.obs_conv(obs[:37], w, b, relu=relu).float()).abs().max()) <= 2.0 ** -7 * scale + 1e-3


def test_ppo_update_reads_compact_observations():
    """PPOAgent.learn over a RolloutBuffer feeds the input layer from the compact observations; the same update from the
    fp32 observation rows (compact form withheld) gives the same metrics and parameters within bf16 tolerance."""
    from shogidrl_b200 import VecShogiEnv
    from shogidrl_b200.core import ActorCritic, PPOAgent, RolloutBuffer
    from shogidrl_b200.training import VecStepManager
    from tests.helpers import make_config
    dev = torch.device("cuda")
    N, T = 512, 8

    def run(withhold):
        cfg = make_config(minibatch_size=1024, ppo_epochs=2)
        torch.manual_seed(1)
        env = VecShogiEnv(N, max_moves_per_game=40, device=dev, seed=5)
        agent = PPOAgent(ActorCritic(46, 13527), cfg, dev, use_mixed_precision=True)
        agent.model.sample_seed = 99
        buf = RolloutBuffer(T, N, 0.99, 0.95, dev)
        drv = VecStepManager(env, agent, buf)
        drv.collect(); drv.finish()
        if withhold:
            full = buf.get_batch
            buf.get_batch = lambda: {k: v for k, v in full().items() if k != "compact_obs"}
        m = agent.learn(buf)
        return m, [p.detach().clone() for p in agent.model.parameters()], buf.actions.clone()

    import shogidrl_b200.core.base_actor_critic as bac
    import itertools
    bac._sample_counter = itertools.count()
    m1, p1, a1 = run(False)
    bac._sample_counter = itertools.count()
    m2, p2, a2 = run(True)
    assert torch.equal(a1, a2)  # the rollouts agree action for action (same sampler stream, logits equal up to bf16 ties)
    for k in m1:
        assert abs(m1[k] - m2[k]) <= 2e-3 * max(1.0, abs(m2[k])), (k, m1[k], m2[k])
    for x, y in zip(p1, p2):
        assert torch.allclose(x, y, rtol=1e-3, atol=2e-4), float((x - y).abs().max())
