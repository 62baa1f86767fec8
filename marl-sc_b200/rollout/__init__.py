from .baselines import AdaptiveBaseStock, base_stock_levels, baseline_rollout, constant_actions, random_actions
from .collector import Rollout, RolloutCollector, shard_envs
from .evaluate import EpisodeMetrics, evaluate
from .graph import GraphedEpisode
from .gae import compute_gae, standardize_, standardize_columns_
from .obs_filter import MeanStdFilter
from .obs_stats import compute_obs_statistics
from .policy import ActorCritic, CentralizedActorCritic, StackedLinear, env_meta_from_algorithm_config, mlp, stacked_mlp
from .ppo import GradBuckets, PPOLearner, lr_schedule
from .trainer import Trainer

__all__ = ["Trainer", "lr_schedule","AdaptiveBaseStock", "constant_actions", "random_actions", "base_stock_levels", "baseline_rollout", "Rollout", "RolloutCollector", "shard_envs", "compute_gae", "compute_obs_statistics", "standardize_", "ActorCritic", "CentralizedActorCritic", "mlp", "PPOLearner", "GraphedEpisode", "GradBuckets", "MeanStdFilter", "StackedLinear", "stacked_mlp", "standardize_columns_", "env_meta_from_algorithm_config", "EpisodeMetrics", "evaluate"]
