"""SelfPlayTrainer -- the batched counterpart of one TrainingLoopManager epoch + Trainer.perform_ppo_update
(keisei/training/training_loop_manager.py:325-454, trainer.py:214-269): T steps of N device-resident games
(tower forward in bf16, fused masked sampling, engine step writing straight into the rollout buffer), bootstrap
values, GAE on the device, PPO update, buffer hand-over.  One process per GPU; under torch.distributed each rank
owns its own games and only gradients (DDP) and three normalisation scalars cross NVLink."""
from __future__ import annotations

import time
from typing import Callable, Dict, Iterable, Optional, Sequence

import torch

from ..core.experience_buffer import RolloutBuffer
from ..core.ppo_agent import PPOAgent
from ..vec_env import VecShogiEnv
from . import distributed as kd
from .step_manager import VecStepManager


class SelfPlayTrainer:
    def __init__(self, model, config, num_envs: int, horizon: int, device="cuda", use_mixed_precision: bool = True,
                 total_envs: Optional[int] = None, start_positions: Optional[Sequence[str]] = None):
        rank, world = kd.world()
        self.device = torch.device(device)
        offset = kd.shard_envs(total_envs, rank, world)[0] if total_envs else rank * num_envs
        seed = getattr(config.env, "seed", 0) or 0
        self.env = VecShogiEnv(num_envs, max_moves_per_game=config.env.max_moves_per_game, device=self.device,
                               seed=int(seed), env_offset=offset, auto_reset=True, start_positions=start_positions)
        self.agent = PPOAgent(model, config, self.device, use_mixed_precision=use_mixed_precision)
        self.agent.model.sample_seed = int(seed) * 7919 + rank
        self.agent.enable_ddp()
        self.buffer = RolloutBuffer(horizon, num_envs, config.training.gamma, config.training.lambda_gae, self.device)
        self.driver = VecStepManager(self.env, self.agent, self.buffer)
        self.global_timestep = 0
        self.current_epoch = 0
        self.rank, self.world = rank, world

    def set_start_positions(self, sfens: Optional[Sequence[str]]) -> None:
        """Start the games that finish from now on from this pool of SFEN positions (None: the start position again),
        e.g. a curriculum that changes between epochs; games in progress continue.  See
        ``VecShogiEnv.set_start_positions``.  The captured rollout graph names the old pool and is recaptured on the next
        ``collect``."""
        self.env.set_start_positions(sfens)
        self.driver.drop_graph()

    def collect(self) -> Dict[str, int]:
        self.driver.collect()
        stats = self.driver.finish()
        self.global_timestep += self.buffer.T * self.buffer.N
        return stats

    def update(self) -> Dict[str, float]:
        metrics = self.agent.learn(self.buffer)
        self.buffer.clear()
        return metrics

    def run_epoch(self) -> Dict[str, float]:
        stats = self.collect()
        metrics = self.update()
        metrics.update({f"episodes/{k}": float(v) for k, v in stats.items()})
        return metrics

    def run(self, total_timesteps: Optional[int] = None, log: Optional[Callable[[str], None]] = None,
            callbacks: Iterable[Callable[["SelfPlayTrainer", Dict[str, float]], None]] = (),
            checkpoint_path: Optional[str] = None, checkpoint_interval_timesteps: Optional[int] = None
            ) -> Dict[str, float]:
        """The batched TrainingLoopManager.run (training_loop_manager.py:80-166): epochs of T x N timesteps until
        ``total_timesteps`` (default ``config.training.total_timesteps``; counted per rank like the reference's
        ``global_timestep``), a PPO update after every epoch except one that reaches the target (``:125-133``), then
        the step callbacks (``callback(trainer, metrics)``; the reference's checkpoint / evaluation callbacks hang
        here) and, on rank 0, a checkpoint every ``checkpoint_interval_timesteps`` in the reference's format
        (``PPOAgent.save_model`` with the cumulative win / draw counters, trainer.py:288-339).  ``metrics`` carries the
        PPO metrics, the epoch's episode statistics and ``speed/sps`` (timesteps per second over the epoch)."""
        target = int(total_timesteps if total_timesteps is not None else self.agent.config.training.total_timesteps)
        log = log or (lambda msg: None)
        callbacks = list(callbacks)
        metrics: Dict[str, float] = {}
        next_ckpt = self.global_timestep + checkpoint_interval_timesteps if checkpoint_interval_timesteps else None
        while self.global_timestep < target:
            self.current_epoch += 1
            t0 = time.perf_counter()
            stats = self.collect()
            if self.global_timestep >= target:
                log(f"Target timesteps ({target}) reached during epoch {self.current_epoch}.")
                metrics = {f"episodes/{k}": float(v) for k, v in stats.items()}
                self.buffer.clear()
            else:
                metrics = self.update()
                metrics.update({f"episodes/{k}": float(v) for k, v in stats.items()})
            torch.cuda.synchronize(self.device)
            metrics["speed/sps"] = self.buffer.T * self.buffer.N / max(1e-9, time.perf_counter() - t0)
            metrics["epoch"] = float(self.current_epoch)
            metrics["global_timestep"] = float(self.global_timestep)
            for cb in callbacks:
                cb(self, metrics)
            if next_ckpt is not None and checkpoint_path and self.global_timestep >= next_ckpt:
                self.save_checkpoint(checkpoint_path)
                next_ckpt += checkpoint_interval_timesteps
        if checkpoint_path:
            self.save_checkpoint(checkpoint_path)
        return metrics

    def save_checkpoint(self, path: str) -> None:
        """Rank 0 writes the reference's checkpoint dictionary (ppo_agent.py:462-487: unwrapped model state, optimizer
        state, global_timestep, total_episodes_completed, black_wins / white_wins / draws)."""
        if self.rank != 0:
            return
        d = self.driver
        self.agent.save_model(path, self.global_timestep, d.episodes,
                              {"black_wins": d.black_wins, "white_wins": d.white_wins, "draws": d.draws})

    def load_checkpoint(self, path: str) -> Dict[str, float]:
        """Resume: model + optimizer state and the counters a reference checkpoint carries (trainer.py:120-152)."""
        out = self.agent.load_model(path)
        if "error" not in out:
            self.global_timestep = int(out.get("global_timestep", 0))
            d = self.driver
            d.episodes = int(out.get("total_episodes_completed", 0))
            d.black_wins, d.white_wins, d.draws = int(out.get("black_wins", 0)), int(out.get("white_wins", 0)), int(out.get("draws", 0))
        return out
