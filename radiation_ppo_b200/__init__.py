"""radiation_ppo_b200 -- B200-native (sm_100a) RadSearch environment step + PPO rollout/GAE path.

Drop-in for the per-env Python loop of bentotten/radiation_ppo: `RadSearch` keeps the gym reset/step/observation API of
gym_rad_search.envs.RadSearch, `PPOBuffer` the interface of algos.multiagent.ppo.PPOBuffer; the work runs in hand-written
CUDA kernels behind the C ABI declared in include/radsearch_b200.h.  There is no CPU fallback.
"""
from . import _lib
from ._lib import RadSearchLibraryError
from .envs.rad_search_env import HostStepBuffers, RadSearch, StepResult
from .ppo_buffer import (BatchedPPOBuffer, PPOBuffer, advantage_statistics, combined_shape, gae_advantages,
                         normalize_advantages_)
from .dist import shard_range
from .maps_buffer import BatchedMapsBuffer, MapsBuffer, episode_ranges
from .evaluate import (MonteCarloEvaluator, MonteCarloResults, TeamEvalPolicy, TeamMonteCarloResults,
                       uniform_policy)
from .rollout_stats import EpisodeStats
from .rollout import RolloutCollector, TeamRolloutCollector, TeamRolloutPolicy
from .policy import FusedGruPolicy

__all__ = ["RadSearch", "StepResult", "HostStepBuffers", "PPOBuffer", "BatchedPPOBuffer", "gae_advantages", "advantage_statistics",
           "normalize_advantages_", "combined_shape", "shard_range", "BatchedMapsBuffer", "MapsBuffer", "MonteCarloEvaluator", "MonteCarloResults", "TeamMonteCarloResults",
           "TeamEvalPolicy", "uniform_policy", "EpisodeStats", "RolloutCollector",
           "TeamRolloutCollector", "TeamRolloutPolicy", "FusedGruPolicy", "episode_ranges", "RadSearchLibraryError", "_lib"]
