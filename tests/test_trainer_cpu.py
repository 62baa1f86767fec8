"""CPU: the learning-rate schedule and the per-update rule of the trainer, the algorithm fields the trainer refuses (before
any CUDA work), and the config round trip its checkpoints rely on."""
import copy

import pytest
import torch

from golden.scenarios import small_default
from marlsc_b200.config import algorithm_config_from_dict, environment_config_from_dict
from marlsc_b200.rollout import Trainer, lr_schedule
from test_host_logic import IPPO


def test_lr_schedule_points_midpoints_and_hold():
    f = lr_schedule([[0, 1e-3], [1000, 5e-4], [3000, 1e-4]])
    assert f(0) == pytest.approx(1e-3, rel=0, abs=0)
    assert f(1000) == pytest.approx(5e-4, rel=1e-12)
    assert f(3000) == pytest.approx(1e-4, rel=1e-12)
    assert f(500) == pytest.approx(7.5e-4, rel=1e-12)
    assert f(2000) == pytest.approx(3e-4, rel=1e-12)
    assert f(2500) == pytest.approx(2e-4, rel=1e-12)
    for t in (3001, 10 ** 6, 10 ** 12):
        assert f(t) == pytest.approx(1e-4, rel=1e-12)


def test_lr_schedule_scalar_is_constant():
    f = lr_schedule(3e-4)
    assert all(f(t) == 3e-4 for t in (0, 1, 10 ** 9))
    assert lr_schedule(1)(5) == 1.0


def test_update_i_uses_the_schedule_at_i_times_the_batch():
    sched = [[0, 1e-3], [100_000, 1e-4], [250_000, 0.0]]
    f = lr_schedule(sched)
    tr = Trainer.__new__(Trainer)        # lr_at needs only the schedule and the batch size
    tr.schedule, tr.steps_per_iteration = f, 4096 * 25
    for i in range(6):
        assert tr.lr_at(i) == f(i * 4096 * 25)
    assert tr.lr_at(0) == 1e-3                        # update 0: the first point, as from_algorithm_config sets it
    assert tr.lr_at(3) == 0.0


def _algo(**specific):
    d = copy.deepcopy(IPPO)
    for k, v in specific.items():
        node, path = d["algorithm"]["algorithm_specific"], k.split(".")
        for p in path[:-1]:
            node = node[p]
        node[path[-1]] = v
    return algorithm_config_from_dict(d)


@pytest.fixture
def no_cuda(monkeypatch):
    """Any CUDA call fails the test: the refusals come first."""
    def boom(*a, **k):
        raise AssertionError("CUDA was touched before the configuration was refused")
    for name in ("current_device", "synchronize", "is_available", "device_count", "get_device_name"):
        monkeypatch.setattr(torch.cuda, name, boom)


MLP = dict(type="mlp", config=dict(hidden_sizes=[32], activation="relu"))
REFUSED = [
    ("networks.shared_layers", dict(**{"networks.shared_layers": MLP})),
    ("networks.use_mu_sigma_head", {"networks.use_mu_sigma_head": True}),
    ("networks.actor.config.output_activation", {"networks.actor.config.output_activation": "tanh"}),
    ("networks.critic.config.output_activation", {"networks.critic.config.output_activation": "tanh"}),
    ("networks.actor.config.output_activation_mu", {"networks.use_mu_sigma_head": True,
                                                    "networks.actor.config.output_activation_mu": "tanh"}),
    ("networks.critic.config.activation", {"networks.critic.config.activation": "tanh"}),
    ("actor_obs_type", {"actor_obs_type": "global"}),
    ("warmstart_weights_path", {"warmstart_weights_path": "/nowhere/checkpoint"}),
    ("use_gae", {"use_gae": False}),
]


@pytest.mark.parametrize("field,over", REFUSED, ids=[r[0] for r in REFUSED])
def test_trainer_refuses_fields_it_cannot_honour(field, over, no_cuda, tmp_path):
    env = environment_config_from_dict(small_default())
    with pytest.raises(ValueError, match=field.replace(".", r"\.")):
        Trainer(env, _algo(**over), 80, str(tmp_path / "run"))
    assert not (tmp_path / "run").exists()


def test_trainer_needs_a_horizon_when_num_envs_does_not_divide_batch_size(no_cuda, tmp_path):
    env = environment_config_from_dict(small_default())
    algo = _algo()                                    # batch_size 8000
    with pytest.raises(ValueError, match="batch_size.*num_envs.*horizon"):
        Trainer(env, algo, 4096, str(tmp_path))
    with pytest.raises(ValueError, match="horizon"):
        Trainer(env, algo, 80, str(tmp_path), horizon=0)


def test_configs_survive_the_checkpoint_round_trip():
    """A checkpoint stores model_dump() of both configs; the loaders rebuild equal objects from it."""
    env = environment_config_from_dict(small_default())
    algo = _algo()
    assert environment_config_from_dict(env.model_dump()) == env
    assert algorithm_config_from_dict(algo.model_dump()) == algo
    d = copy.deepcopy(IPPO)
    d["algorithm"]["shared"]["learning_rate"] = [[0, 1e-3], [5000, 1e-4]]
    sched = algorithm_config_from_dict(d)
    assert algorithm_config_from_dict(sched.model_dump()) == sched
