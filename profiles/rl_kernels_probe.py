"""Probe: device time of the agent/buffer kernels through the C ABI with preallocated buffers
(kz_sample_masked / kz_sample_bitmap, kz_eval_masked_fwd/bwd, kz_eval_bitmap_fwd/bwd, kz_gae), against the measured HBM
peak.  KZ_LIB_PATH selects the library, so two builds can be timed alternately in one session."""
import json, os, subprocess, sys, torch
sys.path.insert(0, ".")
from shogidrl_b200 import _native as nv
dev = torch.device("cuda")
peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"] if os.path.exists("MEASURED_PEAKS.json") else 6650.0
L = nv.lib(); st = nv.stream_ptr(dev)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                      capture_output=True, text=True).stdout.strip()
print(f"library {nv.LIB_PATH} ({L.kz_build_info().decode()}); card {card}")
def timed(fn, reps=200):
    for _ in range(5): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps
n, A, LD = 16384, 13527, 13536
g = torch.Generator(device="cuda").manual_seed(0)
mask = (torch.rand(n, LD, device=dev, generator=g) < 0.004).to(torch.uint8)
mask[:, 0] = 1
mask[:, A:] = 0
legal = float(mask[:, :A].sum()) / n
words = (torch.nn.functional.pad(mask[:, :A], (0, 448 * 32 - A)).view(n, 448, 32).long() << torch.arange(32, device=dev)).sum(-1)
bitmap = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32).contiguous()  # the same legal sets
acts = torch.zeros(n, dtype=torch.int64, device=dev)
logp = torch.empty(n, device=dev); ent = torch.empty(n, device=dev); saved = torch.empty(n, 4, device=dev)
ones = torch.ones(n, device=dev)
for dtype, nb in ((torch.bfloat16, 2), (torch.float32, 4)):
    logits = torch.randn(n, LD, device=dev, generator=g).to(dtype)
    grad = torch.empty_like(logits)
    bf = int(dtype == torch.bfloat16)
    for form, mp, ldm, mbytes in (("masked", mask, LD, LD), ("bitmap", bitmap, 448, 448 * 4)):
        need = n * (mbytes + legal * 32)   # mask row + one 32-byte sector per legal logit
        sample = getattr(L, f"kz_sample_{form}")
        ms = timed(lambda: sample(logits.data_ptr(), bf, LD, mp.data_ptr(), ldm, n, 1, 0, None, acts.data_ptr(), 1,
                                  logp.data_ptr(), None, 0, st))
        print(f"kz_sample_{form} {dtype} ({legal:.0f} legal/row): {ms*1e3:.1f} us / {n} rows; bytes needed "
              f"{need/ms/1e6:.0f} GB/s = {need/ms/1e6/peak:.2f} of HBM peak")
        fwd = getattr(L, f"kz_eval_{form}_fwd")
        ms = timed(lambda: fwd(logits.data_ptr(), bf, LD, mp.data_ptr(), ldm, None, acts.data_ptr(), n,
                               logp.data_ptr(), ent.data_ptr(), saved.data_ptr(), st))
        print(f"kz_eval_{form}_fwd {dtype}: {ms*1e3:.1f} us; bytes needed {need/ms/1e6:.0f} GB/s = {need/ms/1e6/peak:.2f}")
        bwd = getattr(L, f"kz_eval_{form}_bwd")
        extra = (None,) if form == "bitmap" else ()   # the bitmap backward takes an optional bias-gradient buffer
        ms = timed(lambda: bwd(logits.data_ptr(), bf, LD, mp.data_ptr(), ldm, None, acts.data_ptr(), n,
                               ones.data_ptr(), ones.data_ptr(), saved.data_ptr(), grad.data_ptr(), LD, *extra, st))
        needb = need + n * A * nb
        print(f"kz_eval_{form}_bwd {dtype}: {ms*1e3:.1f} us; bytes needed (dense dlogits write) {needb/ms/1e6:.0f} GB/s = "
              f"{needb/ms/1e6/peak:.2f}")
for T, N in ((128, 16384), (128, 65536), (2048, 1)):
    r, v = torch.randn(T, N, device=dev), torch.randn(T, N, device=dev)
    d = (torch.rand(T, N, device=dev) < 0.01).to(torch.uint8); lv = torch.randn(N, device=dev)
    adv, ret = torch.empty_like(r), torch.empty_like(r)
    for name in ("kz_gae", "kz_gae_exact"):
        ms = timed(lambda: getattr(L, name)(r.data_ptr(), v.data_ptr(), d.data_ptr(), lv.data_ptr(), T, N, 0.99, 0.99 * 0.95,
                                            adv.data_ptr(), ret.data_ptr(), st))
        print(f"{name} [T={T}, N={N}]: {ms*1e3:.1f} us, {T*N*17/ms/1e6:.0f} GB/s = {T*N*17/ms/1e6/peak:.2f}")
