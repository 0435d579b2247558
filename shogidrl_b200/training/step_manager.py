"""StepManager -- per-timestep composition of the reference (keisei/training/step_manager.py:98-348 execute_step,
:350-481 handle_episode_end, :483-534 reset / update) over injected game / agent / mapper / buffer objects, plus
``VecStepManager``: the same composition for N device-resident games per kernel launch, where observations and
masks are written by the engine straight into the [T, N] rollout buffer."""
from __future__ import annotations

import time
from dataclasses import dataclass
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from ..shogi.definitions import Color
from ..utils.move_formatting import format_move_with_description_enhanced

_CAPTURE_VALUE = {"PAWN": 1, "LANCE": 3, "KNIGHT": 3, "SILVER": 5, "GOLD": 6, "BISHOP": 8, "ROOK": 10}


@dataclass
class EpisodeState:
    current_obs: np.ndarray
    current_obs_tensor: torch.Tensor
    episode_reward: float
    episode_length: int


@dataclass
class StepResult:
    next_obs: np.ndarray
    next_obs_tensor: torch.Tensor
    reward: float
    done: bool
    info: Dict[str, Any]
    selected_move: Optional[Tuple]
    policy_index: int
    log_prob: float
    value_pred: float
    success: bool = True
    error_message: Optional[str] = None


class StepManager:
    def __init__(self, config, game, agent, policy_mapper, experience_buffer):
        self.config = config
        self.game = game
        self.agent = agent
        self.policy_mapper = policy_mapper
        self.experience_buffer = experience_buffer
        self.device = torch.device(config.env.device)
        self.move_history: List[Tuple] = []
        self.move_log: List[str] = []
        self._reset_counters()

    def _reset_counters(self) -> None:
        self.sente_best_capture: Optional[str] = None
        self.sente_best_capture_value = 0
        self.gote_best_capture: Optional[str] = None
        self.gote_best_capture_value = 0
        self.sente_capture_count = self.gote_capture_count = 0
        self.sente_drop_count = self.gote_drop_count = 0
        self.sente_promo_count = self.gote_promo_count = 0

    def _obs_tensor(self, obs: np.ndarray) -> torch.Tensor:
        return torch.tensor(obs, dtype=torch.float32, device=self.device).unsqueeze(0)

    def _failure(self, obs, done: bool, info: Dict[str, Any], message: str) -> StepResult:
        return StepResult(next_obs=obs, next_obs_tensor=self._obs_tensor(obs), reward=0.0, done=done, info=info,
                          selected_move=None, policy_index=0, log_prob=0.0, value_pred=0.0, success=False,
                          error_message=message)

    def execute_step(self, episode_state: EpisodeState, global_timestep: int, logger_func: Callable) -> StepResult:
        try:
            legal = self.game.get_legal_moves()
            if not legal:
                msg = (f"No legal moves available at timestep {global_timestep}. "
                       f"Game should be in terminal state (checkmate/stalemate).")
                logger_func(f"TERMINAL: {msg} Resetting episode.", True, None, "info")
                return self._failure(self.game.reset(), True, {"terminal_reason": "no_legal_moves"}, msg)
            mask = self.policy_mapper.get_legal_mask(legal, device=self.device)
            move, policy_index, log_prob, value_pred = self.agent.select_action(episode_state.current_obs, mask,
                                                                                is_training=True)
            if move is None:
                msg = f"Agent failed to select a move at timestep {global_timestep}"
                logger_func(f"CRITICAL: {msg}. Resetting episode.", True, None, "error")
                return self._failure(self.game.reset(), False, {}, msg)

            if self.config.display.display_moves:
                piece = None
                try:
                    if move[0] is not None and move[1] is not None:
                        piece = self.game.get_piece(move[0], move[1])
                except (AttributeError, IndexError, ValueError):
                    pass
                self._handle_demo_mode(move, episode_state.episode_length, piece)

            mover = self.game.current_player
            is_drop = move[0] is None and move[1] is None
            is_promotion = isinstance(move[4], bool) and move[4]
            result = self.game.make_move(move)
            if not (isinstance(result, tuple) and len(result) == 4):
                raise ValueError(f"Invalid move result: {type(result)}")
            next_obs, reward, done, info = result
            self._count(mover, info.get("captured_piece_type"), is_drop, is_promotion)
            self.experience_buffer.add(episode_state.current_obs_tensor.squeeze(0), policy_index, reward, log_prob,
                                       value_pred, done, mask)
            return StepResult(next_obs=next_obs, next_obs_tensor=self._obs_tensor(next_obs), reward=reward, done=done,
                              info=info, selected_move=move, policy_index=policy_index, log_prob=log_prob,
                              value_pred=value_pred, success=True)
        except ValueError as e:
            msg = f"Error during training step: {e}"
            logger_func(f"CRITICAL: {msg}. Resetting episode.", True, None, "error")
            try:
                return self._failure(self.game.reset(), False, {}, msg)
            except Exception as reset_error:
                return StepResult(next_obs=episode_state.current_obs, next_obs_tensor=episode_state.current_obs_tensor,
                                  reward=0.0, done=True, info={}, selected_move=None, policy_index=0, log_prob=0.0,
                                  value_pred=0.0, success=False,
                                  error_message=f"{msg}; Reset also failed: {reset_error}")

    def _count(self, mover, captured_name, is_drop: bool, is_promotion: bool) -> None:
        black = mover == Color.BLACK or getattr(mover, "value", mover) == 0
        if captured_name:
            base = captured_name.replace("PROMOTED_", "")
            value = _CAPTURE_VALUE.get(base, 0)
            if black:
                self.sente_capture_count += 1
                if value > self.sente_best_capture_value:
                    self.sente_best_capture, self.sente_best_capture_value = base.title(), value
            else:
                self.gote_capture_count += 1
                if value > self.gote_best_capture_value:
                    self.gote_best_capture, self.gote_best_capture_value = base.title(), value
        if is_drop:
            if black:
                self.sente_drop_count += 1
            else:
                self.gote_drop_count += 1
        if is_promotion:
            if black:
                self.sente_promo_count += 1
            else:
                self.gote_promo_count += 1

    def _prepare_demo_info(self, legal_shogi_moves) -> Optional[Any]:
        """The piece the FIRST legal move would move (None for drops / bad input): step_manager.py:536-560."""
        if not legal_shogi_moves or legal_shogi_moves[0] is None:
            return None
        try:
            mv = legal_shogi_moves[0]
            if len(mv) == 5 and mv[0] is not None and mv[1] is not None:
                return self.game.get_piece(mv[0], mv[1])
        except (AttributeError, IndexError, ValueError):
            pass
        return None

    def _handle_demo_mode(self, selected_move: Tuple, episode_length: int, piece_info_for_demo: Optional[Any]) -> None:
        """Move-log line "Move N (Sente|Gote): <usi> - <description>." + the optional per-move delay (:562-608)."""
        if hasattr(self.game, "current_player"):
            player = getattr(self.game.current_player, "name", str(self.game.current_player))
        else:
            player = "Unknown"
        text = format_move_with_description_enhanced(selected_move, self.policy_mapper, piece_info_for_demo)
        shown = {"BLACK": "Sente", "WHITE": "Gote"}.get(player.upper(), player)
        self.move_log.append(f"Move {episode_length + 1} ({shown}): {text}")
        self.move_history.append(selected_move)
        delay = self.config.display.turn_tick
        if delay > 0:
            time.sleep(delay)

    def handle_episode_end(self, episode_state: EpisodeState, step_result: StepResult, game_stats: Dict[str, int],
                           total_episodes_completed: int, logger_func: Callable[..., None]
                           ) -> Tuple[EpisodeState, Optional[str]]:
        winner, reason = self._determine_winner_and_reason(step_result.info)
        stats = dict(game_stats)
        key = {"black": "black_wins", "white": "white_wins", None: "draws"}.get(winner)
        if key is not None:
            stats[key] = stats.get(key, 0) + 1
        total = stats["black_wins"] + stats["white_wins"] + stats["draws"]
        rate = (lambda k: stats[k] / total if total > 0 else 0.0)
        logger_func(
            f"Episode {total_episodes_completed + 1} finished. Length: {episode_state.episode_length}, "
            f"Reward: {episode_state.episode_reward:.2f}. {self._format_game_outcome_message(winner, reason)}",
            also_to_wandb=True,
            wandb_data={"episode_reward": episode_state.episode_reward, "episode_length": episode_state.episode_length,
                        "game_outcome": winner, "game_reason": reason, "black_wins_total": stats["black_wins"],
                        "white_wins_total": stats["white_wins"], "draws_total": stats["draws"],
                        "black_win_rate": rate("black_wins"), "white_win_rate": rate("white_wins"),
                        "draw_rate": rate("draws")},
            log_level="info")
        try:
            obs = self.game.reset()
            if not isinstance(obs, np.ndarray):
                raise RuntimeError("Game reset failed after episode end")
            self.move_history.clear()
            self.move_log.clear()
            self._reset_counters()
            return EpisodeState(obs, self._obs_tensor(obs), 0.0, 0), winner
        except (RuntimeError, ValueError, OSError) as e:
            logger_func(f"CRITICAL: Game reset failed after episode end: {e}", True, None, "error")
            return episode_state, winner

    def _determine_winner_and_reason(self, step_info: Optional[Dict[str, Any]]) -> Tuple[Optional[str], str]:
        """(winner in lower case | None, reason) from the step's info; a "Tsumi" without a winner entry takes the game's
        own winner (step_manager.py:610-634)."""
        winner, reason = None, "Unknown"
        if step_info:
            winner = step_info.get("winner")
            reason = step_info.get("reason", "Unknown")
        final = winner.lower() if winner and isinstance(winner, str) else winner
        if reason == "Tsumi" and winner is None and getattr(self.game, "winner", None) is not None:
            if self.game.winner == Color.BLACK:
                final = "black"
            elif self.game.winner == Color.WHITE:
                final = "white"
        return final, reason

    @staticmethod
    def _format_game_outcome_message(winner: Optional[str], reason: str) -> str:
        if winner == "black":
            return f"Sente wins by {reason}."
        if winner == "white":
            return f"Gote wins by {reason}."
        if winner is None:
            return f"Draw by {reason}."
        return f"Game ended: {winner} by {reason}."

    def reset_episode(self) -> EpisodeState:
        obs = self.game.reset()
        self.move_history.clear()
        self.move_log.clear()
        self._reset_counters()
        return EpisodeState(obs, self._obs_tensor(obs), 0.0, 0)

    def update_episode_state(self, episode_state: EpisodeState, step_result: StepResult) -> EpisodeState:
        return EpisodeState(step_result.next_obs, step_result.next_obs_tensor,
                            episode_state.episode_reward + step_result.reward, episode_state.episode_length + 1)


class VecStepManager:
    """Batched rollout driver: for t in [0, T): obs[t], bitmaps[t] -> agent.select_actions -> kz_step_rollout, which
    writes reward/done and the next observation / legal bitmap straight into obs[t+1] / bitmaps[t+1] of the RolloutBuffer.  The
    stored transition is the reference's (obs before the move, action, reward to the mover, log-prob, value,
    done, mask before the move; step_manager.py:272-301); finished games are reset inside the same launch and
    both colours' plies share one sequence per env, with no sign flips (SURVEY appendix A)."""

    def __init__(self, env, agent, buffer):
        self.env, self.agent, self.buffer = env, agent, buffer
        if buffer.N != env.n:
            raise ValueError(f"the rollout buffer holds {buffer.N} games per step but the environment has {env.n}")
        self.episodes = 0
        self.black_wins = self.white_wins = self.draws = 0
        self._started = False
        self._stat = torch.zeros(4, dtype=torch.int64, device=env.device)
        self._draws = torch.zeros(1, dtype=torch.int64, device=env.device)  # sampling counter, advanced on the device
        tr = getattr(getattr(agent, "config", None), "training", None)
        self.graph_rollout = bool(getattr(tr, "cuda_graph_rollout", True))
        self._graph = None
        self._graph_pool = None  # the start-position pool (address, size) the captured rollout launches with
        self._eager_runs = 0
        self.model_eval_mode = False  # True: sample from the network in eval() (the reference's worker processes)

    def start(self) -> None:
        self.env.reset(refresh=False)
        self.env.legal_bitmap(self.buffer.bitmaps[0], obs=self.buffer.obs[0], cobs=self.buffer.cobs[0])
        self._started = True

    def collect(self) -> None:
        """Fill the buffer with T steps of N games.  No host synchronisation inside the loop; the sampler writes the
        action / log-prob rows and the engine writes reward / done / next observation / next legal bitmap straight
        into the rollout storage.

        The loop is launch-bound on the host side (about 25 small launches per step against ~0.8 ms of device work, and
        worse when several ranks share the host's cores), so from the second call on the whole T-step rollout is ONE
        CUDA graph: every address it touches is fixed (rollout storage, engine state, model parameters), the sampler's
        draw counter lives on the device, and nothing in the loop reads device results on the host."""
        if not self._started:
            self.start()
        model = getattr(self.agent, "model", None)
        cached = hasattr(model, "cache_inference_weights") and getattr(self.agent, "use_mixed_precision", False)
        if cached:
            model.cache_inference_weights()  # once per rollout, outside the captured loop (fixed addresses)
        try:
            if self.graph_rollout and self.env.device.type == "cuda":
                pool = self._pool_key()
                if self._graph is not None and pool != self._graph_pool:
                    self.drop_graph()  # its step launches name the replaced (or removed) start-position pool
                if self._graph is None and self._eager_runs >= 1:
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        self._collect_steps()
                    self._graph, self._graph_pool = graph, pool
                if self._graph is not None:
                    self._graph.replay()
                    return
            self._collect_steps()
            self._eager_runs += 1
        finally:
            if cached:
                model.cache_inference_weights(live=False)  # the parameters are about to change (PPO update)

    def _pool_key(self):
        pool = getattr(self.env, "pool", None)
        return None if pool is None else (pool.data_ptr(), pool.shape[0])

    def drop_graph(self) -> None:
        """Forget the captured rollout; the next ``collect`` captures a new one."""
        self._graph, self._graph_pool = None, None

    def _collect_steps(self) -> None:
        b, env = self.buffer, self.env
        for t in range(b.T):
            _, _, value = self.agent.select_actions(b.obs[t], b.bitmaps[t], is_training=True,
                                                    out=(b.actions[t], b.log_probs[t]), cobs=b.cobs[t],
                                                    draw_counter=self._draws, eval_mode=self.model_eval_mode)
            b.values[t].copy_(value)
            out = env.step_rollout(b.actions[t], b.obs[t + 1], b.bitmaps[t + 1], reward=b.rewards[t], done=b.dones[t],
                                   cobs=b.cobs[t + 1])
            w = out["winner"]
            d = b.dones[t] != 0
            self._stat += torch.stack([d.sum(), (d & (w == 0)).sum(), (d & (w == 1)).sum(), (d & (w < 0)).sum()])

    def finish(self) -> Dict[str, int]:
        """Bootstrap values for the last observations, GAE; returns episode statistics (one host sync)."""
        b = self.buffer
        last_values = self.agent.get_values(b.obs[b.T], cobs=b.cobs[b.T])
        b.compute_advantages_and_returns(last_values)
        s = self._stat.tolist()
        self._stat.zero_()
        self.episodes += s[0]; self.black_wins += s[1]; self.white_wins += s[2]; self.draws += s[3]
        return {"episodes": s[0], "black_wins": s[1], "white_wins": s[2], "draws": s[3]}
