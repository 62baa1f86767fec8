"""Episode metrics without a device: the C entry point is exported, the ctypes struct follows the header, the fill-rate
rule and EpisodeMetrics.summary(), and the argument checks of BatchedInventoryEnv / evaluate()."""
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import marlsc_b200  # noqa: F401
from marlsc_b200 import _capi
from marlsc_b200.envs.batched_env import METRICS_PER_ENV, METRICS_PER_ROW, fill_rate
from marlsc_b200.rollout import EpisodeMetrics, evaluate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_set_metrics_is_exported_and_struct_matches_header():
    assert hasattr(_capi.lib(), "marlsc_env_set_metrics")
    with open(os.path.join(ROOT, "include", "marlsc_b200.h")) as f:
        header = f.read()
    body = re.search(r"typedef struct marlsc_episode_metrics \{(.*?)\} marlsc_episode_metrics_t;", header, re.S).group(1)
    fields = re.findall(r"^\s*double\* (\w+);", body, re.M)
    assert fields == [name for name, _ in _capi.EpisodeMetricsC._fields_]
    assert fields == list(METRICS_PER_ROW + METRICS_PER_ENV)
    assert all(t is __import__("ctypes").c_void_p for _, t in _capi.EpisodeMetricsC._fields_)
    assert re.search(r"int marlsc_env_set_metrics\(marlsc_env_t\* env, const marlsc_episode_metrics_t\* m\);", header)


def test_fill_rate_is_one_where_nothing_was_demanded():
    demand = torch.tensor([10.0, 0.0, 4.0, 0.0], dtype=torch.float64)
    lost = torch.tensor([2.0, 0.0, 4.0, 0.0], dtype=torch.float64)
    assert fill_rate(demand, lost).tolist() == [0.8, 1.0, 0.0, 1.0]


def _accumulators(N=2, E=3, W=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    v = {k: torch.rand((N, E, W), generator=g, dtype=torch.float64) * 10 for k in METRICS_PER_ROW}
    v["demand_units"] = torch.tensor([[10.0, 0.0, 5.0], [8.0, 4.0, 0.0]], dtype=torch.float64)
    v["lost_units"] = torch.tensor([[1.0, 0.0, 5.0], [2.0, 1.0, 0.0]], dtype=torch.float64)
    return v


def test_episode_metrics_summary():
    acc = _accumulators()
    m = EpisodeMetrics.from_accumulators(acc)
    assert torch.equal(m["total_cost"], acc["holding_cost"] + acc["penalty_cost"] + acc["outbound_cost"] + acc["inbound_cost"])
    assert m["fill_rate"].tolist() == [[0.9, 1.0, 0.0], [0.75, 0.75, 1.0]]
    s = m.summary()
    assert set(s) == set(METRICS_PER_ROW + METRICS_PER_ENV) | {"total_cost", "fill_rate"}
    fr = np.array([0.9, 1.0, 0.0, 0.75, 0.75, 1.0])
    assert s["fill_rate"]["mean"] == pytest.approx(fr.mean()) and s["fill_rate"]["std"] == pytest.approx(fr.std())
    ret = acc["episode_return"].sum(-1).reshape(-1).numpy()          # per (episode, environment): summed over warehouses
    assert s["episode_return"]["mean"] == pytest.approx(ret.mean()) and s["episode_return"]["std"] == pytest.approx(ret.std())
    assert s["demand_units"]["mean"] == pytest.approx(27.0 / 6)
    assert m.per_env("shipped_units").shape == (2, 3)


def _fake_env(metrics=True, layout="wide"):
    return SimpleNamespace(num_envs=4, n_warehouses=3, n_skus=2, obs_dim=5, has_episode_metrics=metrics, layout=layout,
                           device=torch.device("cpu"), env_config=SimpleNamespace(action_space=SimpleNamespace(type="direct")))


def test_argument_checks():
    from golden.scenarios import large_network
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    from marlsc_b200.rollout import ActorCritic
    cfg = environment_config_from_dict(dict(large_network(), allow_region_mismatch=True))
    with pytest.raises(ValueError, match="fused"):
        BatchedInventoryEnv(cfg, 8, layout="compact", fused_kernel=True, episode_metrics=True)
    level = np.zeros((3, 2))
    with pytest.raises(ValueError, match="num_episodes"):
        evaluate(_fake_env(), level, 0)
    with pytest.raises(ValueError, match="episode_metrics=True"):
        evaluate(_fake_env(metrics=False), level, 1)
    with pytest.raises(ValueError, match="shape"):
        evaluate(_fake_env(), np.zeros((2, 3)), 1)
    with pytest.raises(ValueError, match="shape"):
        evaluate(_fake_env(), torch.zeros((5, 3, 2)), 1)
    with pytest.raises(ValueError, match="actor must be"):
        evaluate(_fake_env(), "base-stock", 1)
    with pytest.raises(ValueError, match="ActorCritic"):
        evaluate(_fake_env(), ActorCritic(7, 3, 2), 1)
