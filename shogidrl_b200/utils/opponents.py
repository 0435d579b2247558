"""Scripted opponents of the reference (keisei/utils/opponents.py:13-90, BaseOpponent from keisei/utils/utils.py).

These are the scalar, reference-API players: ``select_move(game) -> MoveTuple`` on one game, with Python's
``random.choice`` as the reference draws.  They read only ``get_legal_moves()``, ``get_piece(r, c)`` and
``current_player``, so they play on the device-backed ``ShogiGame`` facade and on any duck-typed game.  Batched
evaluation (``shogidrl_b200.evaluation``) accepts instances of the two players and plays them on the device instead:
``SimpleRandomOpponent`` as the engine's fused uniform-random action, ``SimpleHeuristicOpponent`` as
``VecShogiEnv.heuristic_actions`` (the same tiers, drawn from the engine's counter-based random stream)."""
from __future__ import annotations

import random
from abc import ABC, abstractmethod
from typing import Any, List

from ..shogi.definitions import PieceType


class BaseOpponent(ABC):
    """An opponent that picks one move of a game (keisei/utils/utils.py BaseOpponent)."""

    def __init__(self, name: str = "BaseOpponent"):
        self.name = name

    @abstractmethod
    def select_move(self, game_instance: Any) -> Any:
        """The move (a MoveTuple) to play in ``game_instance``."""


class SimpleRandomOpponent(BaseOpponent):
    """A uniformly random legal move."""

    def __init__(self, name: str = "SimpleRandomOpponent"):
        super().__init__(name)

    def select_move(self, game_instance: Any) -> Any:
        legal_moves = game_instance.get_legal_moves()
        if not legal_moves:
            raise ValueError("No legal moves available for SimpleRandomOpponent, game should be over.")
        return random.choice(legal_moves)


class SimpleHeuristicOpponent(BaseOpponent):
    """Prefers captures, then non-promoting pawn moves, then anything else; uniform within the tier."""

    def __init__(self, name: str = "SimpleHeuristicOpponent"):
        super().__init__(name)

    def select_move(self, game_instance: Any) -> Any:
        legal_moves = game_instance.get_legal_moves()
        if not legal_moves:
            raise ValueError("No legal moves available for SimpleHeuristicOpponent, game should be over.")
        capturing_moves: List[Any] = []
        non_promoting_pawn_moves: List[Any] = []
        other_moves: List[Any] = []
        for move_tuple in legal_moves:
            is_capture = False
            is_pawn_move_no_promo = False
            if move_tuple[0] is not None:  # board move (drops have None as their source row)
                from_r, from_c, to_r, to_c, promote = move_tuple
                destination_piece = game_instance.get_piece(to_r, to_c)
                if destination_piece is not None and destination_piece.color != game_instance.current_player:
                    is_capture = True
                if not is_capture:
                    source_piece = game_instance.get_piece(from_r, from_c)
                    # compared by value: a duck-typed game may carry its own PieceType enum
                    if (source_piece is not None and getattr(source_piece.type, "value", None) == PieceType.PAWN.value
                            and not promote):
                        is_pawn_move_no_promo = True
            if is_capture:
                capturing_moves.append(move_tuple)
            elif is_pawn_move_no_promo:
                non_promoting_pawn_moves.append(move_tuple)
            else:
                other_moves.append(move_tuple)
        if capturing_moves:
            return random.choice(capturing_moves)
        if non_promoting_pawn_moves:
            return random.choice(non_promoting_pawn_moves)
        return random.choice(other_moves)
