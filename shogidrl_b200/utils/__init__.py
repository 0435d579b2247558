from .move_formatting import (_coords_to_square_name, _get_piece_name, format_move_with_description,  # noqa: F401
                              format_move_with_description_enhanced)
from .opponents import BaseOpponent, SimpleHeuristicOpponent, SimpleRandomOpponent  # noqa: F401
from .policy_mapper import PolicyOutputMapper, index_to_move, move_to_index  # noqa: F401

__all__ = ["PolicyOutputMapper", "index_to_move", "move_to_index", "format_move_with_description",
           "format_move_with_description_enhanced"]
