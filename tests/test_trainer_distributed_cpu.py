"""CPU: the rank-order merge of observation-filter buffers, and the data-parallel trainer's world-size refusals (before any CUDA
work), under a two-rank process group whose collectives do nothing."""
import pytest
import torch
import torch.distributed as dist

from golden.scenarios import small_default
from marlsc_b200.config import environment_config_from_dict
from marlsc_b200.rollout import MeanStdFilter, Trainer
from marlsc_b200.rollout.obs_filter import merge_buffers
from marlsc_b200.rollout.trainer import CHECKPOINT_VERSION, shard_path
from test_trainer_cpu import _algo, no_cuda  # noqa: F401  (no_cuda is a fixture)


def _fed(obs_dim, *batches):
    f = MeanStdFilter(obs_dim, "cpu")
    for b in batches:
        f(b.clone())
    return f


def _moments(f):
    return f.count, f.mean, f.m2


@pytest.mark.parametrize("k", [1, 2, 5])
def test_rank_order_merge_equals_a_filter_fed_the_concatenation(k):
    g = torch.Generator().manual_seed(k)
    D = 7
    prev = [torch.randn(40, D, generator=g, dtype=torch.float64).float() * 3 + 1 for _ in range(2)]
    # every rank's buffer: the moments of what it added since the last sync, itself several filter calls
    ranks = [[torch.randn(int(torch.randint(1, 60, (1,), generator=g)), D, generator=g) * (r + 1) - r for _ in range(3)]
             for r in range(k)]
    base = _fed(D, *prev)
    merged = merge_buffers(_moments(base), [_moments(_fed(D, *batches)) for batches in ranks])
    want = _fed(D, torch.cat(prev + [b for batches in ranks for b in batches]))
    for got, ref in zip(merged, _moments(want)):
        torch.testing.assert_close(got, ref, rtol=1e-12, atol=0)


def test_buffer_holds_what_was_added_since_the_last_sync():
    g = torch.Generator().manual_seed(0)
    D = 5
    a, b, c = (torch.randn(30, D, generator=g) for _ in range(3))
    f = _fed(D, a)
    f.track_buffer()
    f(b.clone())
    f(c.clone())
    for got, ref in zip(f.buffer, _moments(_fed(D, torch.cat([b, c])))):
        torch.testing.assert_close(got, ref, rtol=1e-12, atol=0)
    for got, ref in zip(f.synced, _moments(_fed(D, a))):
        assert torch.equal(got, ref)


@pytest.fixture
def two_ranks():
    """The default process group of a rank 1 of 2 whose collectives do nothing."""
    from torch.testing._internal.distributed.fake_pg import FakeStore
    dist.init_process_group("fake", store=FakeStore(), rank=1, world_size=2)
    yield
    dist.destroy_process_group()


def test_trainer_refuses_num_envs_the_world_does_not_divide(two_ranks, no_cuda, tmp_path):  # noqa: F811
    env = environment_config_from_dict(small_default())
    with pytest.raises(ValueError, match=r"num_envs \(81\).*world size \(2\)"):
        Trainer(env, _algo(), 81, str(tmp_path / "run"), horizon=4)
    assert not (tmp_path / "run").exists()


def test_trainer_refuses_fewer_eval_envs_than_ranks(two_ranks, no_cuda, tmp_path):  # noqa: F811
    env = environment_config_from_dict(small_default())
    with pytest.raises(ValueError, match=r"num_eval_envs \(1\).*world size \(2\)"):
        Trainer(env, _algo(), 80, str(tmp_path / "run"), num_eval_envs=1)
    assert not (tmp_path / "run").exists()


def _checkpoint(path, **extra):
    torch.save(dict(version=CHECKPOINT_VERSION, iteration=2, **extra), path)
    return str(path)


def test_resume_refuses_another_world_size(two_ranks, no_cuda, tmp_path):  # noqa: F811
    single = _checkpoint(tmp_path / "checkpoint_2.pt")              # world 1 writes no world_size
    with pytest.raises(ValueError, match="world size 1.*world size 2"):
        Trainer.resume(single)
    four = _checkpoint(tmp_path / "checkpoint_4.pt", world_size=4)
    with pytest.raises(ValueError, match="world size 4.*world size 2"):
        Trainer.resume(four)


def test_resume_of_a_sharded_checkpoint_needs_a_group_of_its_size(no_cuda, tmp_path):  # noqa: F811
    two = _checkpoint(tmp_path / "checkpoint_2.pt", world_size=2)
    with pytest.raises(ValueError, match="world size 2.*world size 1"):
        Trainer.resume(two)


def test_resume_refuses_a_missing_shard_by_name(two_ranks, no_cuda, tmp_path):  # noqa: F811
    main = _checkpoint(tmp_path / "checkpoint_2.pt", world_size=2)
    torch.save(dict(rank=0, iteration=2), shard_path(main, 0))      # rank 0's shard is there, rank 1's is not
    assert shard_path(main, 1).endswith("checkpoint_2.rank1.pt")
    with pytest.raises(ValueError, match=r"checkpoint_2\.rank1\.pt"):
        Trainer.resume(main)
