"""splendor-rl-gym_b200 -- B200-native (sm_100a) frontier expansion for the Splendor
fastest-win solver of IamJasonBian/Splendor-RL-Gym.

Scope: ONE hot path -- per-turn successor generation, visited-set dedup, heuristic scoring
and beam top-k (reference: src/solver.py BFS/beam loop + src/gems.py + src/buys.py) --
behind the reference's own State / HEURISTICS / solve() surface.  Everything is computed
by hand-written CUDA kernels in libsplendor_b200.so (C ABI: include/splendor_b200.h).
"""
from ._lib import EXPORTS, LIB_PATH, SplendorB200Error, lib  # noqa: F401  (raises if the .so is missing)
from .buys import get_buys, load_buys, possible_buys  # noqa: F401
from .cardparser import Card, get_deck, sort_cards  # noqa: F401
from .color import COLOR_NUM, Color  # noqa: F401
from .engine import Engine, LevelSolver  # noqa: F401
from .formula import Formula  # noqa: F401
from .gems import MAX_GEMS, get_takes, increase_bonus, subtract_with_bonus, take_gems  # noqa: F401
from .realistic import CardMarket, GameConfig, GemPool, MultiPlayerState, PlayerState, solve_many  # noqa: F401
from .solver import HEURISTICS, State  # noqa: F401

__all__ = ['State', 'HEURISTICS', 'Formula', 'GameConfig', 'GemPool', 'CardMarket', 'PlayerState', 'MultiPlayerState', 'solve_many', 'Engine', 'LevelSolver', 'Card', 'Color', 'COLOR_NUM', 'MAX_GEMS', 'get_deck',
           'get_takes', 'get_buys', 'possible_buys', 'load_buys', 'take_gems', 'subtract_with_bonus',
           'increase_bonus', 'sort_cards', 'SplendorB200Error']
