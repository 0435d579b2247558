"""Outputs of the masked-softmax kernels on one seeded all-finite batch, for comparing two builds bit for bit.

    KZ_LIB_PATH=<lib> python profiles/masked_softmax_ab.py dump OUT.npz
    python profiles/masked_softmax_ab.py compare A.npz B.npz

65,536 rows (legal sets ~0.5 % dense, every 16th row 30 % dense so that rows take several list pieces), fp32 and bf16
logits, 16-byte aligned byte masks and bitmap rows: sampled and arg-max actions, log-probs, entropies, the evaluation
forward's outputs, and the backward's dlogits (as a sha256 of their bytes) and bias sums."""
import hashlib, sys
import numpy as np
import torch
sys.path.insert(0, ".")
A, LD, n = 13527, 13536, 65536


def dump(path):
    from shogidrl_b200 import _native as nv, rl
    dev = torch.device("cuda")
    L, st = nv.lib(), nv.stream_ptr(dev)
    g = torch.Generator(device="cuda").manual_seed(1234)
    dense = (torch.arange(n, device=dev) % 16 == 0)[:, None]
    u = torch.rand(n, A, device=dev, generator=g)
    legal = torch.where(dense, u < 0.3, u < 0.005)
    store = torch.zeros((n, LD), dtype=torch.uint8, device=dev)
    store[:, :A] = legal
    words = (torch.nn.functional.pad(legal.long(), (0, 448 * 32 - A)).view(n, 448, 32) << torch.arange(32, device=dev)).sum(-1)
    bitmap = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32).contiguous()
    del u, words
    acts = torch.multinomial(legal.float() + 1e-9, 1, generator=g).squeeze(1)
    w_lp, w_ent = torch.randn(n, device=dev, generator=g), torch.randn(n, device=dev, generator=g)
    out = {"build": np.frombuffer(L.kz_build_info(), dtype=np.uint8)}
    for dtype in (torch.float32, torch.bfloat16):
        logits = (torch.randn(n, LD, device=dev, generator=g) * 3).to(dtype)
        bf = int(dtype == torch.bfloat16)
        for form, m, ldm in (("bytes", store, LD), ("bitmap", bitmap, 448)):
            key = f"{str(dtype)[6:]}_{form}"
            mv = m[:, :A] if form == "bytes" else m
            for det in (0, 1):
                a, lp, ent = rl.sample_masked(logits[:, :A], mv, seed=77, offset=5, deterministic=bool(det), want_entropy=True)
                out[f"{key}_act{det}"], out[f"{key}_lp{det}"], out[f"{key}_ent{det}"] = a, lp, ent
            fam = "masked" if form == "bytes" else "bitmap"
            lp = torch.empty(n, device=dev); ent = torch.empty(n, device=dev); saved = torch.empty((n, 4), device=dev)
            nv.check(getattr(L, f"kz_eval_{fam}_fwd")(logits.data_ptr(), bf, LD, m.data_ptr(), ldm, None, acts.data_ptr(),
                                                      n, lp.data_ptr(), ent.data_ptr(), saved.data_ptr(), st), "fwd")
            dl = torch.zeros((n, LD), dtype=dtype, device=dev)
            db = torch.zeros(LD, dtype=torch.int64, device=dev)
            bwd = L.kz_eval_masked_bwd_bias if form == "bytes" else L.kz_eval_bitmap_bwd
            nv.check(bwd(logits.data_ptr(), bf, LD, m.data_ptr(), ldm, None, acts.data_ptr(), n, w_lp.data_ptr(),
                         w_ent.data_ptr(), saved.data_ptr(), dl.data_ptr(), LD, db.data_ptr(), st), "bwd")
            torch.cuda.synchronize()
            out[f"{key}_elp"], out[f"{key}_eent"], out[f"{key}_saved"], out[f"{key}_dbias"] = lp, ent, saved, db
            out[f"{key}_dlogits_sha256"] = np.frombuffer(
                hashlib.sha256(dl.view(torch.uint8).cpu().numpy().tobytes()).digest(), dtype=np.uint8)
            del dl
    np.savez(path, **{k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in out.items()})
    print(f"dumped {len(out)} arrays to {path}")


def compare(pa, pb):
    a, b = np.load(pa), np.load(pb)
    print("A:", bytes(a["build"]).decode(), "\nB:", bytes(b["build"]).decode())
    keys = [k for k in a.files if k != "build"]
    diff = [k for k in keys if a[k].tobytes() != b[k].tobytes()]
    for k in keys:
        print(f"{k:28s} {'IDENTICAL' if k not in diff else 'DIFFERENT'}")
    print(f"{len(keys) - len(diff)} of {len(keys)} outputs bit-identical")
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(dump(sys.argv[2]) if sys.argv[1] == "dump" else compare(sys.argv[2], sys.argv[3]))
