"""The rest of a PPO minibatch update against fp64 references at their edges: the input layer (kz_obs_conv_fwd / _wgrad,
kz_cobs_conv_fwd / _wgrad through nn_ops.obs_conv), the loss (kz_ppo_loss through rl.ppo_loss) and the clip + Adam tail
(kz_adam_clip_step through rl.adam_clip_step).  Each reference restates in fp64 what the fused kernel replaces: conv2d
[+ ReLU] of bf16-rounded operands, PPOAgent._minibatch_update's unfused loss branch, and clip_grad_norm_ +
torch.optim.Adam(capturable=True).  Tolerances are per element and come from the summation each kernel performs, so a
dropped or doubled term fails; NaN goes where torch sends it."""
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24        # fp32 unit roundoff
U_MMA = 2.0 ** -23    # per term of a tensor-core fp32 accumulation, which may truncate instead of rounding
B16 = 2.0 ** -8       # bf16 unit roundoff
NAN = float("nan")
INF = float("inf")


def _nan_close(got, ref, tol, what):
    """NaN exactly where the reference has NaN; elsewhere |got - ref| <= tol, element by element."""
    got, ref = got.double(), ref.double()
    nan = torch.isnan(ref)
    assert torch.equal(torch.isnan(got), nan), (what, int(torch.isnan(got).sum()), int(nan.sum()))
    bad = ~((got - ref).abs() <= tol) & ~nan
    if bool(bad.any()):
        i = torch.nonzero(bad)[0].tolist()
        raise AssertionError((what, int(bad.sum()), i, float(got[tuple(i)]), float(ref[tuple(i)]), float(tol[tuple(i)])))


# ------------------------------------------------------------------------------------------------
# input layer
def _wgrad_ctas(n, compact):
    from shogidrl_b200 import _native as nv
    L = nv.lib()
    return int((L.kz_cobs_conv_wgrad_ctas if compact else L.kz_obs_conv_wgrad_ctas)(n))


def _size(spec, compact):
    """A batch size, or one relative to R, the weight gradient's resident grid."""
    if isinstance(spec, int):
        return spec
    R = _wgrad_ctas(1 << 30, compact)
    return {"R-1": R - 1, "R": R, "R+1": R + 1, "2R+3": 2 * R + 3}[spec]


def _synthetic_cobs(n, ctas, seed):
    """n compact observations within the format (one plane index 0-27 or 0xFF per square, bytes 81-83 0xFF, 18 fp32
    constant-plane values in words 21-38), built so that:
      - every plane (and empty) comes to every square: board b holds plane (7 b + s) % 29 at square s (28: empty);
      - a CTA of the weight gradient, which takes boards b, b + ctas, b + 2 ctas, ..., sees full and empty boards in
        turn, so its patched tile has to clear every square that became empty; every 11th board is empty as well;
      - the constant planes are all zero, all non-zero, non-zero one at a time, or values bf16 cannot hold (1/3, 0.3)."""
    rng = np.random.default_rng(seed)
    b = np.arange(n)[:, None]
    planes = ((7 * b + np.arange(81)[None, :]) % 29).astype(np.uint8)
    planes[planes == 28] = 0xFF
    empty = ((np.arange(n) // ctas) % 2 == 1) | (np.arange(n) % 11 == 5)
    planes[empty] = 0xFF
    vals = np.zeros((n, 18), np.float32)
    mode = np.arange(n) % 4
    full = mode == 1
    vals[full] = rng.uniform(-2.0, 2.0, (int(full.sum()), 18)).astype(np.float32)
    one = np.nonzero(mode == 2)[0]
    vals[one, one % 18] = rng.uniform(0.5, 2.0, one.size).astype(np.float32)
    odd = mode == 3
    vals[odd] = np.resize(np.array([1 / 3, 0.3, -1 / 3, 1.0, 0.0, 2.0], np.float32), 18)
    by = np.full((n, 160), 0xFF, np.uint8)
    by[:, :81] = planes
    by[:, 84:] = 0
    by[:, 84:156] = vals.view(np.uint8).reshape(n, 72)
    return torch.from_numpy(by.view(np.int32).copy()).cuda()


def _layer_weights(seed=4):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(16, 46, 3, 3, generator=g) * 0.05).cuda(), (torch.randn(16, generator=g) * 0.1).cuda()


def _check_layer(obs, cobs, rows, w, b, relu, dy_dtype, seed=5):
    """Forward and weight / bias gradient of nn_ops.obs_conv (compact when cobs is given) against fp64."""
    from shogidrl_b200 import nn_ops
    compact = cobs is not None
    y = nn_ops.obs_conv(obs, w, b, relu=relu, rows=rows, cobs=cobs)
    n = y.shape[0]
    x = (obs if rows is None else obs[rows]).bfloat16().double()
    w16 = w.bfloat16().double()
    b16 = b.bfloat16().double() if b is not None else None
    pre = F.conv2d(x, w16, b16, padding=1)
    ref = torch.relu(pre) if relu else pre
    # one fp32 accumulator per output: 46 x 9 products and the bias; then one bf16 rounding
    mag = F.conv2d(x.abs(), w16.abs(), b16.abs() if b16 is not None else None, padding=1)
    e = (46 * 9 + 1) * U_MMA * mag
    _nan_close(y, ref, B16 * (ref.abs() + e) + e, ("forward", compact, relu, b is not None))
    # backward: the gate is the saved (bf16) output, as torch's threshold_backward(dy, y, 0); dy rounded to bf16.  The
    # layer's backward is called directly: autograd would cast an fp32 dy to the output's bf16 before it gets there.
    dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(seed)).cuda().to(dy_dtype)
    ctx = SimpleNamespace(saved_tensors=(obs, y.detach(), rows, cobs), needs_input_grad=(False, True, True),
                          relu=relu, has_bias=b is not None, wdtype=torch.float32)
    _, dw, db = nn_ops._ObsConv.backward(ctx, dy)[:3]
    d = dy.bfloat16().double()
    if relu:
        d = torch.where(y.detach().double() <= 0, torch.zeros((), dtype=torch.float64, device=d.device), d)
    gw = torch.nn.grad.conv2d_weight(x, tuple(w.shape), d, padding=1)
    mw = torch.nn.grad.conv2d_weight(x.abs(), tuple(w.shape), d.abs(), padding=1)
    # per weight: each CTA sums its boards (96 products per board, squares padded to 96) in one fp32 accumulator, then
    # the partials of the ctas CTAs are added in turn
    ctas = _wgrad_ctas(n, compact)
    k = -(-n // ctas) * 96 + ctas
    _nan_close(dw, gw, k * U_MMA * mw, ("dweight", compact, relu, b is not None, n))
    if b is not None:
        _nan_close(db, d.sum((0, 2, 3)), k * U_MMA * d.abs().sum((0, 2, 3)), ("dbias", compact, relu, n))
    return y


@pytest.mark.parametrize("compact", [False, True], ids=["dense", "compact"])
@pytest.mark.parametrize("size", [1, 2, 3, 4, 5, 37, "R-1", "R", "R+1", "2R+3", 16384])
def test_input_layer_synthetic_boards(size, compact):
    """Every plane at every square, empty boards, full and empty boards in turn within a CTA's stride, constant planes
    zero / non-zero / one at a time / not bf16-exact; with and without bias and ReLU, dy in fp32 and bf16."""
    n = _size(size, compact)
    cobs = _synthetic_cobs(n, _wgrad_ctas(n, compact), seed=n)
    from tests.helpers import obs_from_cobs
    obs = obs_from_cobs(cobs)
    w, b = _layer_weights()
    for relu, bias, dt in ((True, True, torch.float32), (False, True, torch.bfloat16), (True, False, torch.bfloat16),
                           (False, False, torch.float32)):
        y = _check_layer(obs, cobs if compact else None, None, w, b if bias else None, relu, dt)
        if relu and n >= 37:
            assert bool((y == 0).any())  # outputs exactly 0 at the ReLU gate


@pytest.mark.parametrize("compact", [False, True], ids=["dense", "compact"])
@pytest.mark.parametrize("rows_kind", ["none", "permutation", "duplicates", "one_row"])
def test_input_layer_real_positions(rows_kind, compact):
    """Self-play positions from kz_step_rollout, read in place through minibatch rows: none, a permutation, rows with
    duplicates, and one row n times (the compact weight gradient's patch then changes nothing from board to board)."""
    from tests.helpers import rollout_positions
    obs, cobs = rollout_positions(512, 9)
    N = obs.shape[0]
    g = torch.Generator().manual_seed(11)
    rows = {"none": None, "permutation": torch.randperm(N, generator=g),
            "duplicates": torch.randint(0, N // 8, (N // 2,), generator=g),
            "one_row": torch.full((3000,), 1234, dtype=torch.int64)}[rows_kind]
    rows = rows.cuda() if rows is not None else None
    w, b = _layer_weights(7)
    for relu, dt in ((True, torch.float32), (False, torch.bfloat16)):
        _check_layer(obs, cobs if compact else None, rows, w, b, relu, dt)


@pytest.mark.parametrize("compact", [False, True], ids=["dense", "compact"])
@pytest.mark.parametrize("where", ["weight", "bias"])
def test_input_layer_nan(where, compact):
    """A NaN weight (centre tap of a constant plane that is non-zero on every board, so that the compact forward meets
    it at every square) or a NaN bias: that output channel is NaN, with ReLU too, and its weight and bias gradients
    are what torch gives (threshold_backward passes dy where the output is NaN)."""
    n = 600
    cobs = _synthetic_cobs(n, _wgrad_ctas(n, compact), seed=3)
    cobs[:, 21] = torch.tensor([1.0]).view(torch.int32).item()  # constant plane 28 is 1 on every board
    from tests.helpers import obs_from_cobs
    obs = obs_from_cobs(cobs)
    w, b = _layer_weights()
    if where == "weight":
        w[3, 28, 1, 1] = NAN
    else:
        b[5] = NAN
    for relu in (True, False):
        y = _check_layer(obs, cobs if compact else None, None, w, b, relu, torch.float32)
        o = 3 if where == "weight" else 5
        assert bool(torch.isnan(y[:, o]).all()) and not bool(torch.isnan(y[:, [c for c in range(16) if c != o]]).any())


# ------------------------------------------------------------------------------------------------
# PPO loss
def _loss_ref(new_lp, ent, new_v, old_lp, adv, ret, eps, cv, ce, scale):
    """PPOAgent._minibatch_update's unfused branch in fp64 (value clipping off): loss, the five metrics and
    d(loss * scale) / d(new_lp, entropy, new_v)."""
    lp, en, v = (t.double().requires_grad_(True) for t in (new_lp, ent, new_v))
    olp, a, r = old_lp.double(), adv.double(), ret.double()
    ratio = torch.exp(lp - olp)
    pol = -torch.min(ratio * a, torch.clamp(ratio, 1 - eps, 1 + eps) * a).mean()
    val = F.mse_loss(v, r)
    el = -en.mean()
    loss = pol + cv * val + ce * el
    (loss * scale).backward()
    stats = torch.stack([loss, pol, val, el, (olp - lp).mean(), ((ratio - 1.0).abs() > eps).double().mean()]).detach()
    return stats, (lp.grad, en.grad, v.grad)


def _loss_tols(new_lp, ent, new_v, old_lp, adv, ret, eps, cv, ce, stats, grads):
    """Per-output bounds of the one-CTA kernel: each of its 1,024 threads sums ceil(n / 1024) terms, then two five-level
    shuffle trees; every term carries its own roundings (the ratio: the fp32 difference and expf's 2 ulp)."""
    n = new_lp.numel()
    k = -(-n // 1024) + 12
    z = lambda t: t.double().nan_to_num(0.0, 0.0, 0.0)  # a NaN row's bound does not matter: its output must be NaN
    d = z(new_lp - old_lp).abs()
    pol = torch.exp(d) * z(adv).abs()                  # >= |min(ratio A, clamp(ratio) A)|
    dv2 = z(new_v - ret) ** 2

    def mean_tol(terms, per_term):
        return float((per_term.sum() + k * U * terms.sum()) / n)

    t_pol, t_val = mean_tol(pol, pol * (d + 6) * U), mean_tol(dv2, dv2 * 4 * U)
    t_ent, t_kl = mean_tol(z(ent).abs(), torch.zeros(())), mean_tol(d, d * U)
    st = stats.nan_to_num(0.0).abs()
    tol = torch.tensor([t_pol + abs(cv) * t_val + abs(ce) * t_ent, t_pol, t_val, t_ent, t_kl, 0.0], dtype=torch.float64)
    tol = tol + 3 * U * st
    tol[0] += 3 * U * float(st[1] + abs(cv) * st[2] + abs(ce) * st[3])
    gt = (z(grads[0]).abs() * (d + 10) * U, z(grads[1]).abs() * 6 * U, z(grads[2]).abs() * 8 * U)
    return tol, gt


def _loss_case(n, eps, seed):
    g = torch.Generator().manual_seed(seed)
    old_lp = -torch.rand(n, generator=g) * 5
    new_lp = old_lp + torch.randn(n, generator=g) * 0.3
    tie = torch.rand(n, generator=g) < 0.15
    new_lp[tie] = old_lp[tie]                         # ratio exactly 1: a tie of min's arguments
    if eps > 0:
        # no assertion about a branch within a few ulp of a bound (expf and exp may differ by an ulp there)
        for _ in range(3):
            r = torch.exp(new_lp.double() - old_lp.double())
            near = ((r - (1 - eps)).abs() < 1e-5) | ((r - (1 + eps)).abs() < 1e-5)
            new_lp[near] += 1e-3
    adv = torch.randn(n, generator=g)
    adv[torch.rand(n, generator=g) < 0.2] = 0.0
    ent = torch.rand(n, generator=g) * 4
    new_v, ret = torch.randn(n, generator=g), torch.randn(n, generator=g)
    return new_lp, ent, new_v, old_lp, adv, ret


def _check_loss(inputs, eps, cv, ce, scale):
    from shogidrl_b200 import rl
    new_lp, ent, new_v, old_lp, adv, ret = inputs
    dev = [t.cuda() for t in inputs]
    lp_g, en_g, v_g = (t.clone().requires_grad_(True) for t in dev[:3])
    loss, stats = rl.ppo_loss(lp_g, en_g, v_g, dev[3], dev[4], dev[5], eps, cv, ce, scale)
    loss.backward()
    ref_stats, ref_grads = _loss_ref(*inputs, eps, cv, ce, scale)
    tol, gtol = _loss_tols(*inputs, eps, cv, ce, ref_stats, ref_grads)
    _nan_close(stats.cpu(), ref_stats, tol, "stats")
    assert float(loss) == float(stats[0]) or (math.isnan(float(loss)) and math.isnan(float(stats[0])))
    for name, got, ref, t in zip(("d new_lp", "d entropy", "d new_v"), (lp_g.grad, en_g.grad, v_g.grad), ref_grads, gtol):
        _nan_close(got.cpu(), ref, t, name)


@pytest.mark.parametrize("eps,cv,ce,scale", [(0.2, 0.5, 0.01, 1.0), (0.0, 0.5, 0.01, 0.5), (0.2, 0.0, 0.0, 0.25)],
                         ids=["eps0.2", "eps0", "coef0"])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 1023, 1024, 1025, 16384, 262144])
def test_ppo_loss_edges(n, eps, cv, ce, scale):
    """Ratios on both sides of both clip bounds with positive, negative and zero advantages; exact ties (ratio 1, on
    both bounds at once when clip_eps = 0: the tie gradient and the strict '>' of the clip fraction); coefficients 0 and
    grad_scale != 1; n around the 1,024 threads of the single CTA."""
    inputs = _loss_case(n, eps, seed=n)
    if n >= 1023:
        r = torch.exp(inputs[0].double() - inputs[3].double())
        lo, hi = r < 1 - eps, r > 1 + eps
        for side in (lo, hi):
            for sgn in (inputs[4] > 0, inputs[4] < 0, inputs[4] == 0):
                assert bool((side & sgn).any())
    _check_loss(inputs, eps, cv, ce, scale)


@pytest.mark.parametrize("name", ["new_lp", "entropy", "new_v", "old_lp", "adv", "ret"])
def test_ppo_loss_nan(name):
    """One NaN in one input: the loss, the five metrics and the three gradients follow torch (clamp and min propagate
    NaN; minimum's backward sends the gradient to both sides when neither is smaller)."""
    inputs = list(_loss_case(1025, 0.2, seed=7))
    idx = ["new_lp", "entropy", "new_v", "old_lp", "adv", "ret"].index(name)
    inputs[idx][517] = NAN
    inputs[idx][3] = NAN
    _check_loss(inputs, 0.2, 0.5, 0.01, 1.0)
    _check_loss(inputs, 0.2, 0.5, 0.0, 1.0)


# ------------------------------------------------------------------------------------------------
# clip + Adam
LR, B1, B2, AEPS = 3e-4, 0.9, 0.999, 1e-8


def _adam_ref(ps, gs, ms, vs, step, coef, wd):
    """Adam(capturable=True).step() in fp64 after the gradients were scaled by coef, with the hyper-parameters as
    torch's fp32 arithmetic sees them: betas rounded to fp32 in pow / mul, 1 - beta formed in double; and per-element
    bounds of the kernel's roundings."""
    f = lambda x: float(np.float32(x))
    b1, b2, omb1, omb2 = f(B1), f(B2), f(1.0 - B1), f(1.0 - B2)
    bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
    ss = f(LR) / bc1
    out = []
    for p, g, m, v in zip(ps, gs, ms, vs):
        p, g, m, v = p.double(), g.double(), m.double(), v.double()
        gc = g * coef + wd * p
        egc = 2 * U * ((g * coef).abs() + abs(wd) * p.abs())
        m2 = m + (gc - m) * omb1
        em = 4 * U * (m.abs() + gc.abs() * omb1) + egc * omb1
        v2 = b2 * v + omb2 * gc * gc
        ev = 4 * U * (b2 * v + omb2 * gc * gc) + omb2 * 2 * gc.abs() * egc
        den = v2.sqrt() / math.sqrt(bc2) + f(AEPS)
        rden = torch.where(v2 > 0, ev / (2 * v2.clamp(min=1e-300)), torch.zeros_like(v2)) + 8 * U
        s = ss * m2 / den
        p2 = p - s
        ep = 2 * U * p2.abs() + ss * (em + m2.abs() * rden) / den + 8 * U * s.abs()
        out.append((p2, m2, v2, ep, em, ev))
    return out


def _norm_ref(gs):
    """Total L2 norm as the fp32 sum of squares gives it (inf once that sum overflows fp32), and its bound: one thread
    sums 16 squares, then 8 warps, the partials of 1,024 threads, 32 warps."""
    sq = sum(float((g.double() ** 2).sum()) for g in gs)
    if math.isnan(sq):
        return NAN, 0.0
    if sq > float(np.finfo(np.float32).max):
        return INF, 0.0
    parts = sum(-(-g.numel() // 4096) for g in gs)
    return math.sqrt(sq), (16 + 5 + 8 + -(-parts // 1024) + 10 + 2) * U * math.sqrt(sq)


def _adam_case(shapes, grads_fn, max_norm, step0=0, wd=0.0, seed=3):
    """One rl.adam_clip_step on fresh parameters whose state (moments and the step counter step0) was loaded, against
    the fp64 reference: the norm, the clip coefficient, and every parameter and moment."""
    from shogidrl_b200 import rl
    g = torch.Generator().manual_seed(seed)
    base = [torch.randn(s, generator=g) for s in shapes]
    grads = grads_fn([torch.randn(s, generator=g) for s in shapes])
    ms = [torch.randn(s, generator=g) * 0.01 for s in shapes] if step0 else [torch.zeros(s) for s in shapes]
    vs = [torch.rand(s, generator=g) * 1e-4 for s in shapes] if step0 else [torch.zeros(s) for s in shapes]
    ps = [torch.nn.Parameter(b.cuda()) for b in base]
    opt = torch.optim.Adam(ps, lr=LR, betas=(B1, B2), eps=AEPS, weight_decay=wd, capturable=True)
    for p, gr, m, v in zip(ps, grads, ms, vs):
        p.grad = gr.cuda()
        opt.state[p] = {"step": torch.tensor(float(step0), device="cuda"), "exp_avg": m.cuda(), "exp_avg_sq": v.cuda()}
    out2 = torch.empty(2, device="cuda")
    rl.adam_clip_step(opt, max_norm, out2)
    norm, coef = (float(x) for x in out2.cpu())
    rnorm, enorm = _norm_ref(grads)
    if math.isnan(rnorm):
        assert math.isnan(norm) and math.isnan(coef), (norm, coef)
    else:
        assert norm == rnorm or abs(norm - rnorm) <= enorm, (norm, rnorm)
        rcoef = min(1.0, max_norm / (rnorm + 1e-6)) if rnorm < INF else 0.0
        assert abs(coef - rcoef) <= 4 * U * rcoef + enorm / max(rnorm, 1e-30) * rcoef, (coef, rcoef)
    ref = _adam_ref(base, grads, ms, vs, step0 + 1, coef, wd)
    for p, (p2, m2, v2, ep, em, ev) in zip(ps, ref):
        st = opt.state[p]
        assert float(st["step"]) == step0 + 1
        _nan_close(p.detach().cpu(), p2, ep, ("param", tuple(p.shape)))
        _nan_close(st["exp_avg"].cpu(), m2, em, ("exp_avg", tuple(p.shape)))
        _nan_close(st["exp_avg_sq"].cpu(), v2, ev, ("exp_avg_sq", tuple(p.shape)))
    return norm, coef, ps, opt


_SHAPES = [(1353, 129), (16, 46, 3, 3), (4096,), (7,), (1,), (3, 4099)]


def _poke(i, value):
    def fn(grads):
        grads[i].view(-1)[i * 37 % grads[i].numel()] = value
        return grads
    return fn


def test_adam_clip_nan_gradient_poisons_every_parameter():
    """One NaN gradient element: the norm and the clip coefficient are NaN (torch.clamp keeps NaN), so every parameter
    and moment comes out NaN, as clip_grad_norm_ + Adam.step() leave them."""
    norm, coef, ps, opt = _adam_case(_SHAPES, _poke(2, NAN), 0.5)
    for p in ps:
        assert bool(torch.isnan(p).all()) and bool(torch.isnan(opt.state[p]["exp_avg"]).all())


@pytest.mark.parametrize("value", [INF, -INF])
def test_adam_clip_inf_gradient(value):
    """One +-inf element: norm inf, coefficient 0, every finite gradient zeroed, the inf element NaN (inf x 0)."""
    norm, coef, ps, opt = _adam_case(_SHAPES, _poke(1, value), 0.5)
    assert norm == INF and coef == 0.0
    assert int(sum(int(torch.isnan(p).sum()) for p in ps)) == 1


def test_adam_clip_norm_overflows_fp32():
    """|g| ~ 1e20: the fp32 sum of squares overflows, as torch's does: norm inf, coefficient 0, a zero-gradient step."""
    def fn(grads):
        grads[0] *= 1e20
        return grads
    norm, coef, _, _ = _adam_case(_SHAPES, fn, 0.5)
    assert norm == INF and coef == 0.0


@pytest.mark.parametrize("max_norm", [0.0, 0.5, 1e9])
@pytest.mark.parametrize("step0", [0, 10 ** 4, 10 ** 6])
def test_adam_clip_steps_and_max_norm(step0, max_norm):
    """Step counters loaded at 0, 10^4 and 10^6 (the bias corrections' powf against pow at large exponents), with
    max_norm 0 (every gradient zeroed), a clipping 0.5 and an unclipped 1e9; weight decay on the last."""
    wd = 0.01 if max_norm > 1 else 0.0
    norm, coef, _, _ = _adam_case(_SHAPES, lambda gr: [x * 10 for x in gr], max_norm, step0=step0, wd=wd)
    assert (coef == 0.0) if max_norm == 0 else (coef < 1.0 if max_norm == 0.5 else coef == 1.0)


def test_adam_clip_many_tensors():
    """1,100 small parameter tensors: 69 launch groups of 16, beyond the 64 a fixed array held."""
    shapes = [(1 + (7 * i) % 23,) for i in range(1100)]
    norm, coef, _, _ = _adam_case(shapes, lambda gr: gr, 0.5)
    assert 0.0 < coef < 1.0
