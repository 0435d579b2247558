"""Shared test helpers: a duck-typed stand-in for the reference's pydantic AppConfig (config_schema.py)."""
from types import SimpleNamespace


def make_config(device="cuda", **training):
    tr = dict(learning_rate=3e-4, gamma=0.99, lambda_gae=0.95, clip_epsilon=0.2, value_loss_coeff=0.5,
              entropy_coef=0.01, ppo_epochs=2, minibatch_size=64, steps_per_epoch=128, total_timesteps=1024,
              gradient_clip_max_norm=0.5, normalize_advantages=True, enable_value_clipping=False, weight_decay=0.0,
              lr_schedule_type=None, lr_schedule_step_on="epoch", lr_schedule_kwargs=None)
    tr.update(training)
    return SimpleNamespace(
        env=SimpleNamespace(device=device, seed=42, input_channels=46, num_actions_total=13527, max_moves_per_game=500),
        training=SimpleNamespace(**tr),
        display=SimpleNamespace(display_moves=False, turn_tick=0.0))


def random_endgames(n, seed):
    """Drop-heavy endgame positions: two kings, a few random pieces, pieces in both hands (BASELINE config 5's
    'drops-heavy endgames').  Filtered with the oracle so that the side not to move is not in check and the
    side to move has a legal move."""
    import numpy as np
    from oracle import oracle as orc  # checker only
    rng = np.random.default_rng(seed)
    boards, hands, sides = [], [], []
    types = [0, 0, 0, 1, 2, 3, 4, 4, 5, 6, 8, 9, 10, 11, 12, 13]
    while len(boards) < n:
        b = np.zeros(81, np.int8)
        k0, k1 = rng.choice(81, 2, replace=False)
        if max(abs(k0 // 9 - k1 // 9), abs(k0 % 9 - k1 % 9)) < 2:
            continue
        b[k0], b[k1] = 8, 22
        for color in (0, 1):
            for _ in range(int(rng.integers(0, 6))):
                sq = int(rng.integers(0, 81))
                t = int(rng.choice(types))
                r = sq // 9
                if b[sq] != 0:
                    continue
                last, second = (0, 1) if color == 0 else (8, 7)
                if t in (0, 1) and r == last:
                    continue
                if t == 2 and r in (last, second):
                    continue
                if t == 0 and any(b[rr * 9 + sq % 9] == 1 + 14 * color for rr in range(9)):
                    continue
                b[sq] = 1 + t + 14 * color
        h = np.zeros(14, np.uint8)
        for color in (0, 1):
            h[color * 7 + 0] = rng.integers(0, 5)
            for t in range(1, 7):
                h[color * 7 + t] = rng.integers(0, 3) if rng.random() < 0.5 else 0
        side = int(rng.integers(0, 2))
        g = orc.OracleGame.from_arrays(b, h, side, 0, 500, evaluate_termination=False)
        if g.in_check(1 - side) or len(g.legal_indices()) == 0:
            continue
        boards.append(b); hands.append(h); sides.append(side)
    return np.stack(boards), np.stack(hands), np.asarray(sides, np.uint8), np.zeros(n, np.int32)


def obs_from_cobs(cobs):
    """int32 [n, 40] compact observations -> fp32 [n, 46, 9, 9] (what they summarise), in plain torch."""
    import torch
    n = cobs.shape[0]
    by = cobs.view(torch.uint8).reshape(n, 160)
    planes = by[:, :81].long()
    obs = torch.zeros((n, 46, 81), dtype=torch.float32, device=cobs.device)
    has = planes < 28
    idx = torch.nonzero(has)
    obs[idx[:, 0], planes[has], idx[:, 1]] = 1.0
    pv = cobs[:, 21:39].contiguous().view(torch.float32)
    obs[:, 28:46, :] = pv[:, :, None]
    return obs.reshape(n, 46, 9, 9)


def rollout_positions(n=2048, T=40):
    """(obs fp32 [(T + 1) n, 46, 9, 9], cobs int32 [(T + 1) n, 40]) of n random self-play games over T + 1 plies on cuda:0,
    written by kz_step_rollout (games restart as they finish)."""
    import torch
    from shogidrl_b200 import VecShogiEnv
    dev = torch.device("cuda:0")
    env = VecShogiEnv(n, max_moves_per_game=60, device=dev, seed=17)
    obs = torch.zeros((T + 1, n, 46, 9, 9), dtype=torch.float32, device=dev)
    bm = torch.zeros((T + 1, n, 448), dtype=torch.int32, device=dev)
    cobs = torch.full((T + 1, n, 40), -7, dtype=torch.int32, device=dev)
    acts = [torch.zeros(n, dtype=torch.int64, device=dev) for _ in range(2)]
    env.refresh(random_actions=True, next_out=acts[0])
    env.legal_bitmap(bm[0], obs=obs[0], cobs=cobs[0])
    for t in range(T):
        env.step_rollout(acts[t & 1], obs[t + 1], bm[t + 1], random_actions=True, next_out=acts[(t + 1) & 1], cobs=cobs[t + 1])
    return obs.reshape(-1, 46, 9, 9), cobs.reshape(-1, 40)
