"""Batched evaluation games on the device engine (SURVEY 8f-2).

The reference's evaluation strategies each run a scalar ``get_legal_moves -> get_legal_mask -> select_action ->
make_move`` loop per game (keisei/evaluation/strategies/single_opponent.py:162-221).  Here N games are played at
once on a VecShogiEnv: one player moves for one colour, the other for the other; games that finish are reset and keep
counting until ``num_games`` have been completed.  A player is an agent-like object (``select_actions(obs, mask)``) or
one of the reference's scripted opponents (keisei/utils/opponents.py), played on the device: ``"random"`` /
``SimpleRandomOpponent`` (the engine's fused uniform-random legal action) or ``"heuristic"`` /
``SimpleHeuristicOpponent`` (``VecShogiEnv.heuristic_actions``, one launch per step) -- and the one-ply look-ahead
player ``"lookahead"`` (``VecShogiEnv.lookahead_actions``: mates, material and the opponent's best reply for every
legal move), which has no scalar counterpart in the reference."""
from __future__ import annotations

import json
from dataclasses import dataclass, field
from pathlib import Path
from typing import Any, Dict, List, Mapping, Optional, Sequence, Tuple

import torch

from . import _native as nv
from .utils.opponents import BaseOpponent, SimpleHeuristicOpponent, SimpleRandomOpponent
from .vec_env import VecShogiEnv

OUTCOMES = ("draw", "agent_win", "opponent_win")  # the reference's result strings (elo_registry.py:86)


@dataclass
class EvaluationResult:
    games: int
    agent_wins: int
    opponent_wins: int
    draws: int
    mean_length: float
    outcomes: List[str] = field(default_factory=list)  # one of OUTCOMES per finished game, in completion order
    start_ids: List[int] = field(default_factory=list)  # with start_positions: the opening of each game of outcomes

    @property
    def win_rate(self) -> float:
        return self.agent_wins / max(1, self.games)


def _player_kind(player) -> str:
    """"random", "heuristic", "lookahead" or "agent" for a player of evaluate_vs_opponent (None = the uniform-random
    player)."""
    if player is None or isinstance(player, SimpleRandomOpponent) or (isinstance(player, str) and player == "random"):
        return "random"
    if isinstance(player, SimpleHeuristicOpponent) or (isinstance(player, str) and player == "heuristic"):
        return "heuristic"
    if isinstance(player, str) and player == "lookahead":
        return "lookahead"
    if isinstance(player, (str, BaseOpponent)):
        raise ValueError(f"unknown scripted player {player!r}: expected 'random', 'heuristic', 'lookahead', "
                         "SimpleRandomOpponent, SimpleHeuristicOpponent or an agent with select_actions(obs, mask)")
    return "agent"


def paired_openings(games_begun: torch.Tensor, pool_size: int) -> torch.Tensor:
    """Opening of the next game of every env in a paired evaluation: envs 2i and 2i+1 form pair i, and the j-th game
    (j = ``games_begun``, counted from 0) of both envs of pair i starts from opening (i + (n/2) * j) mod pool_size, so
    the pairs walk through the pool side by side and each opening is played once from each side before any repeats.
    -> int32 [n] on the device of ``games_begun``."""
    n = games_begun.shape[0]
    pair = torch.arange(n, device=games_begun.device) // 2
    return ((pair + (n // 2) * games_begun) % pool_size).to(torch.int32)


def _num_envs(num_games: int, num_envs: int, paired: bool) -> int:
    """Envs of an evaluation batch: at most one per game and at least two; with paired openings an even number (pairs
    of envs share an opening and a quota), two even when ``num_envs`` is 1."""
    if num_games < 0 or num_envs < 1:
        raise ValueError(f"num_games = {num_games}, num_envs = {num_envs}: need num_games >= 0 and num_envs >= 1")
    n = min(num_envs, max(2, num_games))
    if paired:
        if num_games % 2:
            raise ValueError(f"num_games = {num_games}: with start_positions every opening is played from both sides, so "
                             "num_games must be even")
        n = max(2, n - n % 2)
    return n


def evaluate_vs_opponent(agent, num_games: int, *, opponent=None, num_envs: int = 1024, max_moves_per_game: int = 500,
                         device="cuda", seed: int = 0, deterministic: bool = True,
                         max_steps: Optional[int] = None, start_positions: Optional[Sequence[str]] = None
                         ) -> EvaluationResult:
    """Play ``num_games`` games of ``agent`` against ``opponent`` (None = uniform-random legal moves).  Either side may
    be an agent-like object, ``"random"``, ``"heuristic"``, ``"lookahead"`` or an instance of the two scripted opponent
    classes; results are counted from ``agent``'s side.  A ``"lookahead"`` player is computed each step only for the envs
    where it is to move (``lookahead_actions(active=...)``).  The agent plays Black in even-numbered envs and White in odd-numbered ones.
    Every env has a fixed QUOTA of games (``num_games`` spread evenly over the envs): the first ``quota`` games an env finishes are counted and later ones
    are ignored, so the sample is ``num_games`` independent games exactly as the reference's sequential loop plays them
    -- counting "the first num_games completions of the batch" would over-sample short (decisive) games, because a
    fast env restarts and finishes again while the long draws are still running.  Every tensor stays on the device;
    the host reads four counters per step.

    ``start_positions`` (a sequence of SFEN strings): games start from these openings instead of the start position,
    paired -- both games of a pair of envs start from the same opening, the agent playing Black in one and White in the
    other (``paired_openings``) -- so that two deterministic players do not repeat the same two games.  ``num_games`` must
    then be even (and at least two envs run); ``EvaluationResult.start_ids`` gives each counted game's opening.  A game's
    length (``mean_length``) is its move count at the end, which continues from the opening's move number as the
    reference's ``ShogiGame.from_sfen`` does: subtract ``move number - 1`` of the opening for the plies played."""
    kinds = (_player_kind(agent), _player_kind(opponent))
    random_actions = "random" in kinds
    n = _num_envs(num_games, num_envs, start_positions is not None)
    env = VecShogiEnv(n, max_moves_per_game=max_moves_per_game, device=device, seed=seed, auto_reset=True,
                      start_positions=start_positions)
    dev = env.device
    agent_is_black = (torch.arange(n, device=dev) % 2) == 0
    quota = torch.full((n,), num_games // n, dtype=torch.int64, device=dev)
    quota[: num_games % n] += 1
    completed = torch.zeros(n, dtype=torch.int64, device=dev)
    pooled = env.pool is not None
    if pooled:
        pool_size = env.pool.shape[0]
        finished = torch.zeros(n, dtype=torch.int64, device=dev)  # games each env has finished, quota or not
        env.reset(refresh=False, start_pick=paired_openings(finished, pool_size))
    env.refresh(random_actions=True)
    heuristic = env.heuristic_actions() if "heuristic" in kinds else None
    lookahead = torch.full((n,), -1, dtype=torch.int64, device=dev) if "lookahead" in kinds else None

    def actions_of(player, kind):
        if kind == "random":
            return env.next_actions
        if kind == "heuristic":
            return heuristic
        if kind == "lookahead":
            return lookahead
        return player.select_actions(env.obs, env.mask, is_training=not deterministic)[0]

    # side to move per env: read from plane 42 of the observation (1.0 = Black to move)
    done_games = agent_w = opp_w = draws = 0
    length_sum = 0
    outcomes: List[str] = []
    start_ids: List[int] = []
    steps = 0
    limit = max_steps if max_steps is not None else (max_moves_per_game + 1) * (1 + num_games // n) + 8
    while done_games < num_games and steps < limit:
        black_to_move = env.obs[:, 42, 0, 0] > 0.5
        agent_turn = black_to_move == agent_is_black
        if lookahead is not None:  # for the envs where a look-ahead player is to move
            env.lookahead_actions(out=lookahead, active=None if kinds[0] == kinds[1] else
                                  (agent_turn if kinds[0] == "lookahead" else ~agent_turn))
        a_agent = actions_of(agent, kinds[0])
        a_opp = actions_of(opponent, kinds[1])
        actions = torch.where(agent_turn, a_agent, a_opp).contiguous()
        if pooled:
            playing = env.start_ids.clone()  # the openings of the games this step may finish
            out = env.step(actions, random_actions=random_actions, start_pick=paired_openings(finished + 1, pool_size))
            finished += out["done"] != 0
        else:
            out = env.step(actions, random_actions=random_actions)
        if heuristic is not None:
            env.heuristic_actions(out=heuristic)  # for the returned state (auto-reset applied)
        steps += 1
        d = (out["done"] != 0) & (completed < quota)  # finished games that still count towards their env's quota
        completed += d
        if bool(d.any()):
            w = out["winner"]
            agent_won = d & (((w == 0) & agent_is_black) | ((w == 1) & ~agent_is_black))
            opp_won = d & (w >= 0) & ~agent_won
            codes = (agent_won.long() + 2 * opp_won.long())[d]  # index into OUTCOMES, env order
            parts = [torch.stack([d.sum(), agent_won.sum(), opp_won.sum(), (out["ep_len"] * d).sum()]), codes]
            if pooled:
                parts.append(playing.long()[d])
            stats = torch.cat(parts).tolist()  # one device-to-host read per step that finished a game
            done_games += stats[0]; agent_w += stats[1]; opp_w += stats[2]; length_sum += stats[3]
            draws += stats[0] - stats[1] - stats[2]
            outcomes.extend(OUTCOMES[c] for c in stats[4: 4 + stats[0]])
            start_ids.extend(stats[4 + stats[0]:])
    return EvaluationResult(done_games, agent_w, opp_w, draws, length_sum / max(1, done_games), outcomes, start_ids)


# ---------------------------------------------------------------------------------------------------------------
# Mate in one: can a player see a mate that is there?  Positions with a mate in one are harvested from random play on the
# device (no external tsume collection needed); a player's move solves a position when its expansion ends the game by
# Tsumi.

@dataclass
class MateInOneResult:
    positions: int  # positions evaluated
    with_mate: int  # positions that have a mate in one (only these count toward the rate)
    solved: int  # positions whose move by the player mates
    solved_flags: List[bool] = field(default_factory=list)  # per position: the player's move mates
    mate_flags: List[bool] = field(default_factory=list)  # per position: a mate in one exists

    @property
    def solve_rate(self) -> float:
        return self.solved / max(1, self.with_mate)


def harvest_mate_in_one(num_positions: int, *, seed: int = 0, num_envs: int = 1024, max_moves_per_game: int = 500,
                        device="cuda", max_steps: Optional[int] = None) -> List[str]:
    """SFENs of ``num_positions`` positions that have a mate in one, collected from uniform-random self-play on the
    device: after every step, the positions of the envs whose ``mate_in_one().count >= 1`` are kept, in env order, until
    there are enough.  Deterministic for a seed.  Stops after ``max_steps`` steps (default 100 x max_moves_per_game) with
    what it has."""
    if num_positions < 0 or num_envs < 1:
        raise ValueError(f"num_positions = {num_positions}, num_envs = {num_envs}: need num_positions >= 0 and num_envs >= 1")
    env = VecShogiEnv(num_envs, max_moves_per_game=max_moves_per_game, device=device, seed=seed, auto_reset=True)
    env.refresh(random_actions=True)
    acts = [env.next_actions.clone(), torch.empty_like(env.next_actions)]
    out: List[str] = []
    limit = max_steps if max_steps is not None else 100 * max_moves_per_game
    for i in range(limit):
        if len(out) >= num_positions:
            break
        env.step(acts[i % 2], next_out=acts[(i + 1) % 2], random_actions=True)
        ids = torch.nonzero(env.mate_in_one()["count"] > 0).flatten().tolist()
        if ids:
            out.extend(env.to_sfen(ids[: num_positions - len(out)]))
    return out


def mate_batches(num_positions: int, num_envs: int) -> List[Tuple[int, int, int]]:
    """Host batching of evaluate_mate_in_one: -> [(first, count, n)] with n = min(num_envs, num_positions) envs per batch;
    batch b evaluates positions [first, first + count) and pads its last n - count envs (the last batch only) with
    copies of its first position, whose results are dropped."""
    if num_envs < 1:
        raise ValueError(f"num_envs = {num_envs}: need num_envs >= 1")
    n = min(num_envs, num_positions)
    return [(f, min(n, num_positions - f), n) for f in range(0, num_positions, n)] if n > 0 else []


def evaluate_mate_in_one(player, positions: Sequence[str], *, num_envs: int = 1024, device="cuda", seed: int = 0,
                         deterministic: bool = True) -> MateInOneResult:
    """Mate-in-one score of ``player`` on ``positions`` (SFEN strings, e.g. from harvest_mate_in_one): the player is an
    agent (``select_actions(obs, mask)``), ``"random"``, ``"heuristic"`` or ``"lookahead"``, as in evaluate_vs_opponent.
    The positions are loaded in batches of ``num_envs`` (``load_sfens``, the last batch padded), the player picks one
    move per position, and the move solves the position when ``expand`` ends the game by Tsumi without capturing a king.  Positions without a
    mate in one (``mate_in_one``) do not count toward the rate.  The random player's move on position i is the engine's
    fused uniform-random legal action keyed (seed, i, step 0); the heuristic player's draw is keyed the same way
    (with its own salt, as ``heuristic_actions``), and so is the look-ahead player's (``lookahead_actions``)."""
    kind = _player_kind(player)
    positions = [str(s) for s in positions]
    batches = mate_batches(len(positions), num_envs)
    solved_flags: List[bool] = []
    mate_flags: List[bool] = []
    if not batches:
        return MateInOneResult(0, 0, 0)
    n = batches[0][2]
    # max_moves 65535: a harvested position keeps its move number, which must not end the game at load; history is not
    # needed (a mate does not depend on it), so one repetition slot per game suffices
    env = VecShogiEnv(n, max_moves_per_game=65535, device=device, seed=seed, auto_reset=False, hist_cap=1)
    ids = torch.arange(n, dtype=torch.int32, device=env.device)
    for first, count, _ in batches:
        batch = positions[first:first + count]
        env.env_offset = first  # position i draws from the random stream of index i
        env.load_sfens(batch + [batch[0]] * (n - count))
        if kind == "random":
            env.refresh(random_actions=True)
            actions = env.next_actions.clone()
        elif kind == "heuristic":
            actions = env.heuristic_actions()
        elif kind == "lookahead":
            actions = env.lookahead_actions()
        else:
            actions = player.select_actions(env.obs, env.mask, is_training=not deterministic)[0]
            actions = actions.to(device=env.device, dtype=torch.int64).contiguous()
        out = env.expand(ids, actions)
        solved = (out["reason"] == nv.TSUMI) & ((out["err"] & nv.ERR_KING_CAPTURE) == 0)
        has = env.mate_in_one()["count"] > 0
        flags = torch.stack([solved, has]).cpu().tolist()
        solved_flags.extend(bool(x) for x in flags[0][:count])
        mate_flags.extend(bool(x) for x in flags[1][:count])
    return MateInOneResult(len(positions), sum(mate_flags), sum(solved_flags), solved_flags, mate_flags)


# ---------------------------------------------------------------------------------------------------------------
# Tournament and ladder evaluation on top of evaluate_vs_opponent (keisei/evaluation/strategies/tournament.py,
# ladder.py): the scheduling and the rating arithmetic are host-side and follow the reference; the games run batched.

class EloRegistry:
    """keisei/evaluation/opponents/elo_registry.py:15-135: match-level Elo update, ratings persisted as JSON in the
    reference's layout ({"ratings": {...}, "metadata": {"initial_rating", "k_factor"}})."""

    def __init__(self, file_path: Optional[Path] = None, initial_rating: float = 1500.0, k_factor: float = 32.0):
        self.file_path = Path(file_path) if file_path is not None else None
        self.initial_rating = initial_rating
        self.k_factor = k_factor
        self.ratings: Dict[str, float] = {}
        self.load()

    def load(self) -> None:
        if self.file_path is not None and self.file_path.exists():
            try:
                with open(self.file_path, "r", encoding="utf-8") as f:
                    self.ratings = {k: float(v) for k, v in json.load(f).get("ratings", {}).items()}
            except (OSError, ValueError):
                self.ratings = {}

    def save(self) -> None:
        if self.file_path is None:
            return
        self.file_path.parent.mkdir(parents=True, exist_ok=True)
        with open(self.file_path, "w", encoding="utf-8") as f:
            json.dump({"ratings": self.ratings,
                       "metadata": {"initial_rating": self.initial_rating, "k_factor": self.k_factor}}, f, indent=2)

    def get_rating(self, player_id: str) -> float:
        return self.ratings.setdefault(player_id, self.initial_rating)

    def set_rating(self, player_id: str, rating: float) -> None:
        self.ratings[player_id] = rating

    def update_ratings(self, player1_id: str, player2_id: str, results: List[str]) -> None:
        """One update per match from the mean score of player 1 (elo_registry.py:77-121)."""
        if not results:
            return
        r1, r2 = self.get_rating(player1_id), self.get_rating(player2_id)
        score1 = 0.0
        for res in results:
            if res == "agent_win":
                score1 += 1.0
            elif res == "draw":
                score1 += 0.5
        score2 = len(results) - score1
        expected1 = 1.0 / (1.0 + 10.0 ** ((r2 - r1) / 400.0))
        expected2 = 1.0 - expected1
        self.set_rating(player1_id, r1 + self.k_factor * (score1 / len(results) - expected1))
        self.set_rating(player2_id, r2 + self.k_factor * (score2 / len(results) - expected2))

    def get_all_ratings(self) -> Dict[str, float]:
        return self.ratings.copy()

    def get_top_players(self, limit: int = 10) -> List[Tuple[str, float]]:
        return sorted(self.ratings.items(), key=lambda kv: kv[1], reverse=True)[:limit]


class EloTracker:
    """keisei/evaluation/strategies/ladder.py:54-97: game-by-game Elo update inside one match (the expectation is
    recomputed after every game, so the order of the results matters)."""

    def __init__(self, default_rating: float = 1500.0, k_factor: float = 32):
        self.ratings: Dict[str, float] = {}
        self.default_rating = default_rating
        self.k_factor = k_factor

    def get_agent_rating(self, agent_id: str) -> float:
        return self.ratings.get(agent_id, self.default_rating)

    def update_ratings(self, agent_id: str, opponent_id: str, results: List[str]) -> None:
        a, o = self.get_agent_rating(agent_id), self.get_agent_rating(opponent_id)
        for res in results:
            expected = 1 / (1 + 10 ** ((o - a) / 400))
            actual = 1.0 if res == "agent_win" else 0.5 if res == "draw" else 0.0
            da = self.k_factor * (actual - expected)
            do = self.k_factor * ((1 - actual) - (1 - expected))
            a += da
            o += do
        self.ratings[agent_id] = a
        self.ratings[opponent_id] = o

    def get_elo_snapshot(self) -> Dict[str, float]:
        return self.ratings.copy()


def tournament_standings(results: Mapping[str, EvaluationResult]) -> Dict[str, Any]:
    """The reference's tournament analytics (tournament.py:631-696) from per-opponent match results."""
    overall = {"total_games": 0, "agent_total_wins": 0, "agent_total_losses": 0, "agent_total_draws": 0,
               "agent_overall_win_rate": 0.0}
    per: Dict[str, Dict[str, Any]] = {}
    for name, r in results.items():
        per[name] = {"played": r.games, "wins": r.agent_wins, "losses": r.opponent_wins, "draws": r.draws,
                     "win_rate": r.agent_wins / r.games if r.games > 0 else 0.0}
        overall["total_games"] += r.games
        overall["agent_total_wins"] += r.agent_wins
        overall["agent_total_losses"] += r.opponent_wins
        overall["agent_total_draws"] += r.draws
    if overall["total_games"] > 0:
        overall["agent_overall_win_rate"] = overall["agent_total_wins"] / overall["total_games"]
    return {"overall_tournament_stats": overall, "per_opponent_results": per}


def evaluate_tournament(agent, opponents: Mapping[str, Any], num_games_per_opponent: int,
                        **kwargs) -> Tuple[Dict[str, Any], Dict[str, EvaluationResult]]:
    """Round of matches against every opponent of the pool (name -> a player of evaluate_vs_opponent: an agent-like
    object, "random" / None, "heuristic", "lookahead" or a scripted opponent instance), colours balanced inside each match; returns
    (standings, per-opponent results)."""
    results = {name: evaluate_vs_opponent(agent, num_games_per_opponent, opponent=opp, **kwargs)
               for name, opp in opponents.items()}
    return tournament_standings(results), results


def benchmark_performance(results: Mapping[str, EvaluationResult]) -> Dict[str, Any]:
    """The reference's benchmark analytics (keisei/evaluation/strategies/benchmark.py:639-686) from per-case match results:
    a case is "passed" by a game the agent wins; cases without games report the reference's empty record."""
    per: Dict[str, Dict[str, Any]] = {}
    for name, r in results.items():
        if r.games == 0:
            per[name] = {"played": 0, "wins_or_passes": 0, "pass_rate": 0, "details": "No games played"}
        else:
            per[name] = {"played": r.games, "wins_or_passes": r.agent_wins, "pass_rate": r.agent_wins / r.games}
    played = sum(p["played"] for p in per.values())
    overall = sum(p["wins_or_passes"] for p in per.values()) / played if played else 0
    return {"per_benchmark_case_results": per, "overall_benchmark_pass_rate": overall}


def evaluate_benchmark(agent, suite: Mapping[str, Any], num_games_per_case: int,
                       **kwargs) -> Tuple[Dict[str, Any], Dict[str, EvaluationResult]]:
    """The benchmark strategy (benchmark.py:330-426, 556-637) on the vectorised engine: ``num_games_per_case`` games against
    every case of the suite (name -> a player of evaluate_vs_opponent; the reference's default suite is
    {"benchmark_random": None, "benchmark_heuristic": "heuristic"}), colours balanced; returns (the reference's performance
    dictionary, per-case results)."""
    results = {name: evaluate_vs_opponent(agent, num_games_per_case, opponent=opp, **kwargs) for name, opp in suite.items()}
    return benchmark_performance(results), results


def select_ladder_opponents(agent_rating: float, pool_ratings: Mapping[str, float], num_opponents_to_select: int = 5,
                            window: float = 400.0) -> List[str]:
    """ladder.py:700-732: opponents rated within +-400 of the agent, ascending by rating, the first N."""
    near = [(r, i, name) for i, (name, r) in enumerate(pool_ratings.items())
            if agent_rating - window <= r <= agent_rating + window]
    near.sort(key=lambda t: (t[0], t[1]))  # stable: pool order breaks rating ties, as list.sort does in the reference
    return [name for _, _, name in near[:num_opponents_to_select]]


def evaluate_ladder(agent, agent_id: str, pool: Mapping[str, Any], tracker: Optional[EloTracker] = None,
                    num_games_per_match: int = 2, num_opponents_to_select: int = 5,
                    **kwargs) -> Tuple[Dict[str, float], Dict[str, EvaluationResult]]:
    """One ladder pass (ladder.py:490-558): select opponents near the agent's rating, play a colour-balanced match
    against each (pool: name -> a player of evaluate_vs_opponent), update the ratings game by game; returns (rating
    snapshot, per-opponent results)."""
    tracker = tracker if tracker is not None else EloTracker()
    ratings = {name: tracker.get_agent_rating(name) for name in pool}
    chosen = select_ladder_opponents(tracker.get_agent_rating(agent_id), ratings, num_opponents_to_select)
    results: Dict[str, EvaluationResult] = {}
    for name in chosen:
        r = evaluate_vs_opponent(agent, num_games_per_match, opponent=pool[name], **kwargs)
        tracker.update_ratings(agent_id, name, r.outcomes)
        results[name] = r
    return tracker.get_elo_snapshot(), results
