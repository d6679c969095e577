"""marl_sat_b200 -- B200-native (sm_100a) batched SATEnv hot path of kongqg/marl-sat.

Host-side mirror of the reference's interface for this path (``SATEnv``, ``SATDataWrapper``, the
rollout auto-reset / RNG chain and the MAPPO GAE scan) over the C ABI of ``libmarlsat_b200.so``
(``include/marl_sat_b200.h``).  PyTorch is used for device memory, streams and
``torch.distributed`` only.  Importing the package loads the CUDA library and raises if it has not
been built: there is no CPU fallback.
"""
from . import _lib

_lib.load()   # fail loudly when the CUDA library is missing

from .env import FormulaBank, SATEnv, SATState, create_agent_groups   # noqa: E402
from .gae import (advantage_stats, allreduce_stats, calculate_gae, mean_std_from_stats,  # noqa: E402
                  normalize_advantages)
from .rollout import (RolloutBuffer, RolloutKeys, VecSATEnv, derive_env_keys, merge_state_dicts,  # noqa: E402
                      prng_key, shard_range)
from .wrapper import GNNWrapperState, SATDataWrapper  # noqa: E402
from .features import (GNNInput, StaticGraph, dynamic_features, flip_gains, gnn_input_from_state,  # noqa: E402
                       static_graph)
from .metrics import metrics_from_sums, rollout_metric_sums, rollout_metrics  # noqa: E402
from .evaluate import evaluate_policy  # noqa: E402
from .local_search import WalkSATResult, walksat  # noqa: E402
from .curriculum import problem_stats, problem_weights, unsolved_weights  # noqa: E402
from .sampling import sample_actions  # noqa: E402
from . import dimacs  # noqa: E402

__all__ = ["SATEnv", "SATState", "FormulaBank", "create_agent_groups", "SATDataWrapper", "GNNWrapperState",
           "VecSATEnv", "RolloutBuffer", "RolloutKeys", "derive_env_keys", "merge_state_dicts", "shard_range",
           "prng_key", "calculate_gae",
           "advantage_stats", "normalize_advantages", "allreduce_stats", "mean_std_from_stats", "metrics_from_sums", "GNNInput", "StaticGraph", "static_graph", "dynamic_features",
           "gnn_input_from_state", "flip_gains", "rollout_metrics", "rollout_metric_sums", "evaluate_policy", "walksat", "WalkSATResult", "problem_stats",
           "problem_weights", "unsolved_weights", "sample_actions", "dimacs"]
__version__ = "0.1.0"
