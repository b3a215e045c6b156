"""Mirror of torchreid.metrics (reference torchreid/metrics/__init__.py:3-5) for the hot path, plus ranked lists and
alpha query expansion."""
from .rank import evaluate_rank
from .distance import compute_distance_matrix
from .lists import rank_lists, retrieve
from .qe import query_expansion

__all__ = ['evaluate_rank', 'compute_distance_matrix', 'rank_lists', 'retrieve', 'query_expansion']
