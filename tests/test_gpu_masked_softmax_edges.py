"""The masked-softmax kernels (kz_sample_masked / kz_sample_bitmap, kz_eval_masked_fwd / kz_eval_masked_bwd_bias,
kz_eval_bitmap_fwd / _bwd) against an fp64 restatement of BaseActorCriticModel.evaluate_from_logits' non-CUDA branch, at
the inputs where they branch: -inf / NaN / +inf logits, ties, finite extremes, the eps clamp, list-piece boundaries, mask
bytes other than 0/1 and bitmap pad bits; and rl.gae against an fp64 recurrence on both sides of its dispatch."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

A = 13527
LD = 13536          # logits / dlogits row stride and bias length: the pad columns 13,527-13,535 exist in every buffer
EPS = float(np.finfo(np.float32).eps)
SENTINEL = 768.0    # dlogits prefill, exact in fp32 and bf16: columns >= 13,527 must keep it
INF = float("inf")


# ------------------------------------------------------------------------------------------------
# fp64 reference
def _reference(x, legal, actions, w_lp, w_ent):
    """evaluate_from_logits' non-CUDA branch in fp64 on the logits as stored: (probs, log-prob of ``actions``, entropy,
    d(sum(w_lp * logp + w_ent * entropy)) / d logits, fallback rows).  A fallback row (NaN softmax -> uniform) is a
    constant of the logits: its gradient is zero by contract (autograd would give NaN through the NaN softmax)."""
    x = x.double().requires_grad_(True)
    masked = torch.where(legal, x, torch.tensor(-INF, dtype=torch.float64))
    p = torch.softmax(masked, dim=-1)
    fb = torch.isnan(p).any(dim=1)
    p = torch.where(fb[:, None], torch.full_like(p, 1.0 / A), p)
    logc = torch.log(p.clamp(min=EPS, max=1.0 - EPS))
    lp = logc.gather(1, actions[:, None]).squeeze(1)
    ent = -(p * logc).sum(1)
    (lp * w_lp.double() + ent * w_ent.double()).sum().backward()
    grad = torch.where(fb[:, None], torch.zeros((), dtype=torch.float64), x.grad)
    return p.detach(), lp.detach(), ent.detach(), grad, fb


def _close(got, ref, what, names, rel=1e-5, abs_=2e-6):
    got = got.detach().cpu().double()
    err = (got - ref).abs()
    bad = torch.nonzero(~(err <= rel * ref.abs() + abs_)).flatten().tolist()
    assert not bad, (what, [(names[i], float(got[i]), float(ref[i])) for i in bad])


def _pack_bitmap(legal):
    """bool [n, 13527] -> int32 [n, 448] legal-bitmap rows (bit i of a row = action i), on the CPU."""
    bits = np.zeros((legal.shape[0], 448 * 32), dtype=np.uint8)
    bits[:, :A] = legal.numpy()
    return torch.from_numpy(np.packbits(bits, axis=1, bitorder="little").view("<i4").copy())


# ------------------------------------------------------------------------------------------------
# the cases: one row each, n = 8k + 3 rows (rows share CTAs of 8 warps, the last CTA is partial)
def _cases(dtype):
    g = torch.Generator().manual_seed(20261020)
    big = 3e38 if dtype == torch.float32 else float(torch.finfo(torch.bfloat16).max)
    rows = []  # (name, logits fp32 [LD], legal bool [A], mask byte, action or None)

    def pick(k, lo=0, hi=A):
        return (torch.randperm(hi - lo, generator=g)[:k] + lo).sort().values

    def add(name, idx, vals=None, byte=1, action=None):
        x = torch.randn(LD, generator=g) * 3
        legal = torch.zeros(A, dtype=torch.bool)
        legal[idx] = True
        if vals is not None:
            x[idx] = vals if torch.is_tensor(vals) else torch.full((len(idx),), float(vals))
        rows.append((name, x, legal, byte, action))
        return x

    # -inf at legal entries mixed with finite ones: 40 legal actions below 2,000 (the first list entry of every lane)
    # at -inf, 60 finite legal actions above 2,100
    lo, hi = pick(40, 0, 2000), pick(60, 2100, A)
    add("ninf_first", torch.cat([lo, hi]), torch.cat([torch.full((40,), -INF), torch.randn(60, generator=g)]),
        action=int(hi[7]))
    add("ninf_first_taken", torch.cat([lo, hi]), torch.cat([torch.full((40,), -INF), torch.randn(60, generator=g)]),
        action=int(lo[3]))                                               # the taken action has probability 0
    x = add("ninf_dense", torch.arange(A), action=9000)                  # legal_mask=None with -inf on [0, 8192)
    x[:8192] = -INF
    for k, frac in ((300, 0.3), (1500, 0.5), (6000, 0.7)):
        idx = pick(k)
        x = add(f"ninf_random_{k}", idx)
        x[idx[torch.rand(k, generator=g) < frac]] = -INF
    add("all_ninf", pick(50), -INF)
    add("all_ninf_dense", torch.arange(A), -INF)
    # non-finite legal logits: the reference's softmax row is NaN -> uniform fallback
    for name, v in (("nan_legal", float("nan")), ("pinf_legal", INF)):
        idx = pick(100)
        x = add(name, idx)
        x[idx[37]] = v
    idx = pick(3000)
    x = add("pinf_dense_late", idx)                                      # the +inf entry is in a later list piece
    x[idx[2900]] = INF
    idx = pick(100)
    x = add("ninf_and_pinf", idx)
    x[idx[:20]] = -INF
    x[idx[50]] = INF
    # finite extremes
    idx = pick(64)
    add("extremes", idx, torch.tensor([big, -big, 0.0, 1.0] * 16), action=int(idx[0]))
    add("all_minus_big", pick(40), -big)                                 # ties at the most negative finite logit
    idx = pick(40)
    add("minus_flt_max_and_ninf", idx, torch.tensor([-3.4028234663852886e38, -INF] * 20), action=int(idx[0]))
    idx = pick(50)
    v = torch.rand(50, generator=g)
    v[11] = 1e4                                                          # p_max rounds to 1: the clamp saturates
    add("spread_taken_max", idx, v, action=int(idx[11]))
    add("spread_taken_min", idx, v, action=int(idx[12]))
    # probabilities near the clamp: 0.5 eps and 2 eps next to one dominant action, a factor 2 from eps on both sides
    idx = pick(41)
    v = torch.cat([torch.zeros(1), torch.full((20,), math.log(0.5 * EPS)), torch.full((20,), math.log(2 * EPS))])
    add("near_eps_taken_2eps", idx, v, action=int(idx[30]))
    add("near_eps_taken_half_eps", idx, v, action=int(idx[5]))
    # ties: all legal logits equal; the lowest index (16, window 1) is not lane 0's first list entry
    tie_idx = torch.tensor([16] + [512 * k for k in range(1, 26)] + [13526])
    add("tie_all", tie_idx, 0.5)
    idx = pick(40)
    add("tie_bf16", idx, 1.0 + 1e-4 * torch.randperm(40, generator=g).float())  # distinct in fp32, equal in bf16
    x = add("tie_across_pieces", torch.arange(A))
    x[:A] = torch.randn(A, generator=g)
    x[[100, 9000]] = 10.0
    # legal counts around the warp width and the 2,048-entry list piece, and the first / last action
    for k in (1, 31, 32, 33, 2047, 2048, 2049, A):
        add(f"count_{k}", pick(k))
    add("only_0", torch.tensor([0]))
    add("only_13526", torch.tensor([A - 1]))
    add("first_and_last", torch.tensor([0, A - 1]))
    # mask bytes other than 1 (byte forms only; bitmap rows carry the bit)
    for b in (2, 0x80, 0xFF):
        add(f"byte_{b}", torch.cat([torch.tensor([0, A - 1]), pick(200, 1, A - 1)]).unique(), byte=b)
    idx = pick(30)
    illegal = int(torch.nonzero(~torch.isin(torch.arange(A), idx))[500])
    add("taken_illegal", idx, action=illegal)
    # ordinary rows up to n = 8k + 3
    while len(rows) % 8 != 3:
        add(f"random_{len(rows)}", pick(int(torch.randint(20, 600, (1,), generator=g))))

    n = len(rows)
    logits = torch.stack([r[1] for r in rows])
    legal = torch.stack([r[2] for r in rows])
    byte = torch.tensor([r[3] for r in rows], dtype=torch.uint8)
    actions = torch.empty(n, dtype=torch.int64)
    for i, (_, x, lg, _, a) in enumerate(rows):
        if a is None:
            fin = torch.nonzero(lg & torch.isfinite(x[:A])).flatten()
            a = int(fin[torch.randint(len(fin), (1,), generator=g)]) if len(fin) else int(torch.nonzero(lg)[0])
        actions[i] = a
    w_lp, w_ent = torch.randn(n, generator=g), torch.randn(n, generator=g)
    return [r[0] for r in rows], logits.to(dtype), legal, byte, actions, w_lp, w_ent


# ------------------------------------------------------------------------------------------------
# one run of every entry point over a batch
def _run(logits, form, legal, byte, actions, w_lp, w_ent, seed=7):
    """-> dict of outputs of the sampler (stochastic and deterministic, with entropy), the evaluation forward and the
    evaluation backward with the bias gradient, for the legal sets given as ``form``."""
    from shogidrl_b200 import _native as nv, rl
    dev = logits.device
    n = logits.shape[0]
    if form == "bytes_13527":            # rows at every 16-byte phase
        mask = (legal.to(torch.uint8) * byte[:, None]).to(dev)
        mptr, ldm, bitmap = mask, A, False
    elif form == "bytes_13536":          # 16-byte aligned rows, as the engine writes them
        store = torch.zeros((n, LD), dtype=torch.uint8)
        store[:, :A] = legal.to(torch.uint8) * byte[:, None]
        mask = store.to(dev)[:, :A]
        mptr, ldm, bitmap = mask, LD, False
    else:
        bm = _pack_bitmap(legal)
        if form == "bitmap_pad":         # pad bits 13,527-13,535 of word 422 and words 423-447 set
            bm[:, 422] |= torch.tensor(np.array([0xFF800000], dtype=np.uint32).view(np.int32))
            bm[:, 423:] = -1
        mask = bm.to(dev)
        mptr, ldm, bitmap = mask, 448, True
    L, st = nv.lib(), nv.stream_ptr(dev)
    lv = logits[:, :A]
    out = {}
    for det in (False, True):
        a, lp, ent = rl.sample_masked(lv, mask, seed=seed, offset=1000, deterministic=det, want_entropy=True)
        out[f"act{int(det)}"], out[f"slp{int(det)}"], out[f"sent{int(det)}"] = a, lp, ent
    bf = int(logits.dtype == torch.bfloat16)
    act, wl, we = actions.to(dev), w_lp.to(dev), w_ent.to(dev)
    lp = torch.empty(n, device=dev); ent = torch.empty(n, device=dev); saved = torch.empty((n, 4), device=dev)
    fwd = L.kz_eval_bitmap_fwd if bitmap else L.kz_eval_masked_fwd
    nv.check(fwd(logits.data_ptr(), bf, LD, mptr.data_ptr(), ldm, None, act.data_ptr(), n, lp.data_ptr(), ent.data_ptr(),
                 saved.data_ptr(), st), "eval fwd")
    dl = torch.full((n, LD), SENTINEL, dtype=logits.dtype, device=dev)
    db = torch.zeros(LD, dtype=torch.int64, device=dev)
    bwd = L.kz_eval_bitmap_bwd if bitmap else L.kz_eval_masked_bwd_bias
    nv.check(bwd(logits.data_ptr(), bf, LD, mptr.data_ptr(), ldm, None, act.data_ptr(), n, wl.data_ptr(), we.data_ptr(), saved.data_ptr(), dl.data_ptr(), LD, db.data_ptr(), st), "eval bwd")
    out.update(elp=lp, eent=ent, dlogits=dl, dbias=db)
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in out.items()}


def _check_against_reference(names, logits, legal, actions, w_lp, w_ent, out, form):
    x = logits[:, :A].double()
    p, lp_ref, ent_ref, g_ref, fb = _reference(x, legal, actions, w_lp, w_ent)
    where = lambda key: f"{form}: {key}"
    # evaluation forward
    _close(out["elp"], lp_ref, where("eval log-prob"), names)
    _close(out["eent"], ent_ref, where("eval entropy"), names)
    # sampler: deterministic = torch.argmax (lowest index on ties); every draw has p > 0; log-prob of the draw, entropy
    ref_arg = torch.argmax(p, dim=1)
    bad = torch.nonzero(out["act1"] != ref_arg).flatten().tolist()
    assert not bad, (form, "argmax", [(names[i], int(out["act1"][i]), int(ref_arg[i])) for i in bad])
    for d in (0, 1):
        a = out[f"act{d}"]
        assert bool(((a >= 0) & (a < A)).all()), (form, "action range")
        pa = p.gather(1, a[:, None]).squeeze(1)
        zero = torch.nonzero(pa == 0).flatten().tolist()
        assert not zero, (form, "sampled p = 0", [(names[i], int(a[i])) for i in zero])
        _close(out[f"slp{d}"], torch.log(pa.clamp(EPS, 1.0 - EPS)), where(f"sample log-prob det={d}"), names)
        _close(out[f"sent{d}"], ent_ref, where(f"sample entropy det={d}"), names)
    # fallback rows: uniform, arg-max 0, log(1 / 13527), entropy log 13527, zero gradient
    assert bool((out["act1"][fb] == 0).all())
    assert torch.allclose(out["elp"][fb].double(), torch.full((int(fb.sum()),), -math.log(A), dtype=torch.float64),
                          rtol=1e-6, atol=0)
    # gradients: exact zeros off the legal set and on fallback rows; the pad columns keep the prefill
    g = out["dlogits"][:, :A].double()
    assert bool((out["dlogits"][:, A:] == SENTINEL).all()), (form, "dlogits pad columns written")
    assert bool((g[~legal] == 0).all()) and bool((g[fb] == 0).all()), (form, "dlogits off the legal set")
    rowmax = g_ref.abs().amax(1, keepdim=True)
    if logits.dtype == torch.float32:
        tol = 1e-5 * rowmax + 1e-7
    else:                                # one bf16 rounding of the fp32 gradient
        tol = 2.0 ** -8 * g_ref.abs() + 1e-6 * rowmax
    err = (g - g_ref).abs()
    bad = torch.nonzero((~(err <= tol)).any(1)).flatten().tolist()
    assert not bad, (form, "dlogits", [(names[i], float(err[i].max()), float(rowmax[i])) for i in bad])
    # bias gradient: Q20.44 column sums of the fp32 gradients, against the fp64 column sums
    db = out["dbias"].double() * 2.0 ** -44
    assert bool((out["dbias"][A:] == 0).all()), (form, "dbias pad columns")
    col = g_ref.sum(0)
    ctol = 1e-5 * g_ref.abs().sum(0) + 1e-7 * legal.sum(0).double()
    bad = torch.nonzero(~((db[:A] - col).abs() <= ctol)).flatten().tolist()
    assert not bad, (form, "dbias", bad[:8], float((db[:A] - col).abs().max()))


def _bits(t):
    return t.view({torch.float32: torch.int32, torch.bfloat16: torch.int16}.get(t.dtype, t.dtype))


def _same(o1, o2, what):
    for k in o1:
        assert torch.equal(_bits(o1[k]), _bits(o2[k])), (what, k)


DTYPES = [torch.float32, torch.bfloat16]


@pytest.mark.parametrize("dtype", DTYPES)
def test_masked_softmax_edge_rows_match_fp64_reference(dtype):
    """Every edge row in one batch, through every entry point, with byte-mask rows at every 16-byte phase, aligned
    byte-mask rows and bitmap rows, against the fp64 reference; aligned byte rows and bitmap rows bit-identical."""
    names, logits, legal, byte, actions, w_lp, w_ent = _cases(dtype)
    assert logits.shape[0] % 8 == 3
    ldev = logits.to("cuda:0")
    outs = {form: _run(ldev, form, legal, byte, actions, w_lp, w_ent) for form in ("bytes_13527", "bytes_13536", "bitmap")}
    for form, out in outs.items():
        _check_against_reference(names, logits, legal, actions, w_lp, w_ent, out, form)
    _same(outs["bytes_13536"], outs["bitmap"], "aligned byte rows vs bitmap rows")


@pytest.mark.parametrize("dtype", DTYPES)
def test_bitmap_pad_bits_are_ignored(dtype):
    """Bits 13,527-13,535 of word 422 and words 423-447 set in every bitmap row: the same bits out as with them clear,
    the dlogits pad columns keep their prefill and the bias gradient's pad entries stay zero (the buffers are 13,536
    wide, so a stray access stays inside them)."""
    names, logits, legal, byte, actions, w_lp, w_ent = _cases(dtype)
    ldev = logits.to("cuda:0")
    clear, pad = (_run(ldev, form, legal, byte, actions, w_lp, w_ent) for form in ("bitmap", "bitmap_pad"))
    assert bool((pad["dlogits"][:, A:] == SENTINEL).all()), "dlogits pad columns written"
    assert bool((pad["dbias"][A:] == 0).all()), "bias gradient pad entries written"
    assert bool((pad["act0"] < A).all()) and bool((pad["act1"] < A).all()), "sampled a pad bit"
    _same(clear, pad, "bitmap pad bits set vs clear")


@pytest.mark.parametrize("dtype", DTYPES)
def test_nonfinite_illegal_logits_change_nothing(dtype):
    """NaN, +inf and -inf at every illegal entry give the same bits as the finite values there."""
    names, logits, legal, byte, actions, w_lp, w_ent = _cases(dtype)
    poisoned = logits.clone()
    ill = torch.nonzero(~legal)
    poisoned[ill[:, 0], ill[:, 1]] = torch.tensor([float("nan"), INF, -INF]).to(dtype)[torch.arange(len(ill)) % 3]
    for form in ("bytes_13527", "bitmap"):
        _same(_run(logits.to("cuda:0"), form, legal, byte, actions, w_lp, w_ent),
              _run(poisoned.to("cuda:0"), form, legal, byte, actions, w_lp, w_ent), f"{form}: non-finite illegal logits")


def _sample_many(row_logits, legal_row, n, seed):
    """n copies of one row, stochastic draws through the bitmap and the aligned byte-mask sampler (identical)."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    logits = row_logits[:A].to(dev).expand(n, A)
    store = torch.zeros((n, LD), dtype=torch.uint8, device=dev)
    store[:, :A] = legal_row.to(dev)
    bm = _pack_bitmap(legal_row[None]).to(dev).expand(n, 448)
    a1, lp1, _ = rl.sample_masked(logits.contiguous(), store[:, :A], seed=seed, offset=0)
    a2, lp2, _ = rl.sample_masked(logits.contiguous(), bm.contiguous(), seed=seed, offset=0)
    assert torch.equal(a1, a2) and torch.equal(lp1, lp2)
    return a1.cpu(), lp1.cpu()


@pytest.mark.parametrize("dense", [False, True])
def test_ninf_mixed_row_sampling_law(dense):
    """The law of a row whose legal set mixes -inf and finite logits (every lane meets -inf first, or the dense
    legal_mask=None pattern) is the softmax over the finite ones: chi-square over 65,536 draws."""
    g = torch.Generator().manual_seed(3)
    x = torch.full((LD,), -INF)
    legal = torch.zeros(A, dtype=torch.bool)
    if dense:
        legal[:] = True
        fin = torch.arange(8192, 8192 + 60)   # -inf on [0, 8192) as a model masking its own logits; 60 finite
        x[8192:A] = -30.0                     # the rest finite but far below (mass ~1e-11 in all)
    else:
        legal[(torch.randperm(2000, generator=g)[:40])] = True
        fin = torch.randperm(A - 2100, generator=g)[:60] + 2100
        legal[fin] = True
    x[fin] = torch.randn(60, generator=g) * 0.5
    n = 65536
    act, lp = _sample_many(x, legal, n, seed=41)
    p = torch.softmax(x[:A].double(), 0)
    assert bool((p[act] > 0).all()), "drew an action of probability 0"
    assert torch.allclose(lp.double(), torch.log(p[act]), rtol=1e-5, atol=2e-6)
    counts = torch.bincount(act, minlength=A).double()
    assert float(counts[fin].sum()) >= n - 2   # the -30 logits carry ~1e-11 of the mass
    expected = p[fin] / p[fin].sum() * float(counts[fin].sum())
    chi2 = float(((counts[fin] - expected) ** 2 / expected).sum())
    assert chi2 < 105.0, chi2  # 59 dof: P(chi2 > 105) ~ 2e-4


def test_fallback_rows_draw_uniformly():
    """Rows with a legal NaN, a legal +inf, or only -inf legal logits: uniform over all 13,527 actions (chi-square
    over 64 bins of [0, 13527) on 49,152 draws), log-prob log(1/13527), entropy log(13527), arg-max 0."""
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(4)
    n = 3 * 16384
    x = torch.randn(n, A, generator=g)
    legal = torch.rand(n, A, generator=g) < 0.01
    legal[:, 5] = True
    kind = torch.arange(n) % 3
    x[kind == 0, 5] = float("nan")
    x[kind == 1, 5] = INF
    x[kind == 2] = torch.where(legal[kind == 2], torch.tensor(-INF), x[kind == 2])
    bm = _pack_bitmap(legal).to(dev)
    xd = x.to(dev)
    act, lp, ent = rl.sample_masked(xd, bm, seed=5, offset=0, want_entropy=True)
    det, dlp, _ = rl.sample_masked(xd, bm, deterministic=True)
    assert bool((det == 0).all())
    for v in (lp, dlp):
        assert torch.allclose(v.cpu().double(), torch.full((n,), -math.log(A), dtype=torch.float64), rtol=1e-6, atol=0)
    assert torch.allclose(ent.cpu().double(), torch.full((n,), math.log(A), dtype=torch.float64), rtol=1e-6, atol=0)
    act = act.cpu()
    assert bool(((act >= 0) & (act < A)).all())
    bins = act * 64 // A
    counts = torch.bincount(bins, minlength=64).double()
    width = torch.bincount(torch.arange(A) * 64 // A, minlength=64).double()
    expected = width / A * n
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert chi2 < 125.0, chi2  # 63 dof: P(chi2 > 125) ~ 6e-6
    for k in range(3):  # each kind on its own spreads over the whole range, not a few actions
        assert int(torch.bincount(bins[kind == k], minlength=64).min()) > 150  # expected 256 per bin


# ------------------------------------------------------------------------------------------------
# GAE on both sides of kz_gae's dispatch (warp scan below 2,048 envs, one thread per column from 2,048)
def _gae_reference(r, v, d, lv, gamma, gl):
    """fp64 recurrence with the kernel's fp32 coefficients; also the first-order rounding scale C_t =
    sum over the non-terminal stretch from t of prod(gamma * lambda) * (|r| + gamma |nv| + |v|)."""
    T, N = r.shape
    adv = np.zeros((T, N)); C = np.zeros((T, N))
    gae = np.zeros(N); c = np.zeros(N); nv = lv.astype(np.float64)
    for t in range(T - 1, -1, -1):
        m = 1.0 - d[t].astype(np.float64)
        delta = r[t] + gamma * nv * m - v[t]
        gae = delta + gl * m * gae
        c = np.abs(r[t]) + gamma * np.abs(nv) * m + np.abs(v[t]) + gl * m * c
        adv[t], C[t] = gae, c
        nv = v[t].astype(np.float64)
    return adv, adv + v, C


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.0, 0.95)])
@pytest.mark.parametrize("T", [1, 31, 32, 33, 200])
def test_gae_matches_fp64_recurrence(T, gamma, lam):
    from shogidrl_b200 import rl
    dev = torch.device("cuda:0")
    g = np.random.default_rng(T * 1000 + int(gamma * 100) + int(lam * 10))
    g32, gl32 = float(np.float32(gamma)), float(np.float32(gamma * lam))
    for N in (2, 37, 2047, 2048):
        r = g.standard_normal((T, N)).astype(np.float32)
        v = g.standard_normal((T, N)).astype(np.float32)
        d = g.random((T, N)) < 0.05
        d[0, 0::3] = True                      # done at t = 0
        d[T - 1, 1::3] = True                  # done at t = T - 1
        d[T // 3:T // 3 + 5, 2::5] = True      # runs of dones
        scalar = N % 2 == 1
        lv = np.full(N, np.float32(0.37), dtype=np.float32) if scalar else g.standard_normal(N).astype(np.float32)
        lv_t = torch.tensor([0.37]) if scalar else torch.from_numpy(lv)
        a_ref, r_ref, C = _gae_reference(r, v, d, lv, g32, gl32)
        bound = (2 * T + 64) * 2.0 ** -24 * C
        args = (torch.from_numpy(r).to(dev), torch.from_numpy(v).to(dev), torch.from_numpy(d).to(dev), lv_t.to(dev))
        for exact in (False, True):
            adv, ret = rl.gae(*args, gamma, lam, exact=exact)
            ea = np.abs(adv.cpu().numpy() - a_ref)
            er = np.abs(ret.cpu().numpy() - r_ref)
            assert (ea <= bound).all(), (N, exact, "adv", float((ea / bound).max()))
            assert (er <= bound).all(), (N, exact, "ret", float((er / bound).max()))
