"""B200-native batched Scotland Yard environment (drop-in for the reference's
src/environment hot path).  See DESIGN.md / INTEGRATION.md at the repo root."""
from ._cabi import LIB_PATH, SyError, load_library  # noqa: F401
from .graphs import GraphSpec, generate_connected_graph, generate_graph_pool, pack_csr  # noqa: F401
from .env import (  # noqa: F401
    DEFAULT_REWARD_WEIGHTS,
    REWARD_WEIGHT_NAMES,
    BatchedScotlandYardEnv,
    dense_action_mask,
    numpy_reward_tables,
)

from .sharding import allreduce_stats, shard_range  # noqa: F401,E402
from .compat import CustomEnvironment  # noqa: F401,E402
from .torchrl_env import make_torchrl_env  # noqa: F401,E402
from .rollout import RolloutCollector, batched_graph_data, masked_sample  # noqa: F401,E402
from .policy import GNNPolicy, HeuristicPolicy, MappoPolicy, gcn_in_edges  # noqa: F401,E402

__all__ = [
    "allreduce_stats", "shard_range", "CustomEnvironment", "make_torchrl_env", "RolloutCollector", "batched_graph_data",
    "masked_sample", "GNNPolicy", "HeuristicPolicy", "MappoPolicy", "gcn_in_edges",
    "BatchedScotlandYardEnv", "GraphSpec", "generate_connected_graph", "generate_graph_pool", "pack_csr",
    "dense_action_mask", "numpy_reward_tables", "DEFAULT_REWARD_WEIGHTS", "REWARD_WEIGHT_NAMES", "SyError",
    "load_library", "LIB_PATH",
]
