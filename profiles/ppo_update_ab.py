"""Outputs of the PPO update's input layer, loss and clip + Adam kernels on one seeded all-finite batch of production
size, for comparing two builds bit for bit.

    KZ_LIB_PATH=<lib> python profiles/ppo_update_ab.py dump OUT.npz
    python profiles/ppo_update_ab.py compare A.npz B.npz

16,384 boards (random compact observations and the fp32 rows they decode to): kz_obs_conv_fwd / _wgrad and
kz_cobs_conv_fwd / _wgrad with ReLU and bias, dy in bf16; kz_ppo_loss at n = 16,384 (its metrics and three gradients);
six kz_adam_clip_step calls over the default CNN's parameters, clipped and unclipped (norms, parameters, moments)."""
import sys
import numpy as np
import torch
sys.path.insert(0, ".")
n = 16384


def dump(path):
    from shogidrl_b200 import _native as nv, nn_ops, rl
    from shogidrl_b200.core import ActorCritic
    from tests.helpers import obs_from_cobs
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(4321)
    out = {"build": np.frombuffer(nv.lib().kz_build_info(), dtype=np.uint8)}
    # input layer
    planes = torch.randint(0, 28, (n, 81), device=dev, generator=g)
    planes = torch.where(torch.rand(n, 81, device=dev, generator=g) < 0.3, planes, 0xFF).to(torch.uint8)
    by = torch.full((n, 160), 0xFF, dtype=torch.uint8, device=dev)
    by[:, :81] = planes
    vals = torch.where(torch.rand(n, 18, device=dev, generator=g) < 0.5, torch.rand(n, 18, device=dev, generator=g), 0.0)
    by[:, 84:156] = vals.contiguous().view(torch.uint8)
    by[:, 156:] = 0
    cobs = by.view(torch.int32).contiguous()
    obs = obs_from_cobs(cobs)
    w = (torch.randn(16, 46, 3, 3, device=dev, generator=g) * 0.05).requires_grad_(True)
    b = (torch.randn(16, device=dev, generator=g) * 0.1).requires_grad_(True)
    dy = torch.randn(n, 16, 9, 9, device=dev, generator=g).bfloat16()
    for form, c in (("dense", None), ("compact", cobs)):
        y = nn_ops.obs_conv(obs, w, b, relu=True, cobs=c)
        dw, db = torch.autograd.grad(y, (w, b), dy)
        out[f"conv_{form}_y"], out[f"conv_{form}_dw"], out[f"conv_{form}_db"] = y.view(torch.int16), dw, db
    # loss
    old_lp = -torch.rand(n, device=dev, generator=g) * 5
    new_lp = (old_lp + torch.randn(n, device=dev, generator=g) * 0.3).requires_grad_(True)
    ent = (torch.rand(n, device=dev, generator=g) * 4).requires_grad_(True)
    new_v = torch.randn(n, device=dev, generator=g).requires_grad_(True)
    adv, ret = torch.randn(n, device=dev, generator=g), torch.randn(n, device=dev, generator=g)
    loss, stats = rl.ppo_loss(new_lp, ent, new_v, old_lp, adv, ret, 0.2, 0.5, 0.01, 1.0)
    loss.backward()
    out["loss_stats"], out["loss_dlp"], out["loss_dent"], out["loss_dv"] = stats, new_lp.grad, ent.grad, new_v.grad
    # clip + Adam
    torch.manual_seed(5)
    model = ActorCritic(46, 13527).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=3e-4, capturable=True)
    norms = []
    for it in range(6):
        for p in model.parameters():
            p.grad = torch.randn(p.shape, device=dev, generator=g) * (10.0 if it % 2 else 0.01)
        norm2 = torch.empty(2, device=dev)
        rl.adam_clip_step(opt, 0.5, norm2)
        norms.append(norm2)
    out["adam_norms"] = torch.stack(norms)
    for i, p in enumerate(model.parameters()):
        st = opt.state[p]
        out[f"adam_p{i}"], out[f"adam_m{i}"], out[f"adam_v{i}"] = p.detach(), st["exp_avg"], st["exp_avg_sq"]
    torch.cuda.synchronize()
    np.savez(path, **{k: (v.detach().cpu().numpy() if torch.is_tensor(v) else v) for k, v in out.items()})
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
