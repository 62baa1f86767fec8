"""The compact layout's in-transit ring (ring_qty uint8 [E,L,W,S], indexed by placement time): where a step's new orders
land, which snapshots may be loaded into it, and the base-stock heuristic's view of what is in transit - both the policy
evaluated inside the step (K1a') and the policy kernel (K5) - before and after the ring wraps."""
import numpy as np
import pytest
import torch

from parity_common import _lean_env_dict

pytestmark = pytest.mark.gpu


def _compact_env(W, S, R, L, E, leads=None, seed=0):
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    rng = np.random.default_rng(seed)
    d = _lean_env_dict(rng, W, S, R, "shipment", True, L)
    if leads is not None:
        d["components"]["lead_time_sampler"]["params"]["expected_lead_times"] = leads.tolist()
    d["episode_length"] = 2 * L + 8
    cfg = environment_config_from_dict(dict(d, allow_region_mismatch=True))
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, layout="compact")
    assert env.layout == "compact" and env.ring_qty.shape == (E, L, W, S)
    lead = np.asarray(d["components"]["lead_time_sampler"]["params"]["expected_lead_times"])
    maxq = np.asarray(d["action_space"]["params"]["max_order_quantities"])
    return env, lead, maxq, rng


def _orders(rng, E, S, R):
    from marlsc_b200.demand import pack_orders
    per_env = [[(int(rng.integers(0, R)), np.where(rng.random(S) < 0.3, rng.integers(1, 9, S), 0).astype(float))
                for _ in range(int(rng.integers(0, 12)))] for _ in range(E)]
    return pack_orders(per_env, S)


@pytest.mark.parametrize("L", [1, 5, 16])
def test_step_writes_new_orders_into_plane_t_mod_L(L):
    """After step t every cell's clipped order quantity, 0 included, is in plane t % L; the other planes keep the orders
    of the L - 1 steps before."""
    W, S, R, E = 4, 36, 6, 9
    env, _, maxq, rng = _compact_env(W, S, R, L, E, seed=L)
    env.ring_qty.fill_(7)
    env.reset()
    placed = []
    for t in range(2 * L + 3):
        qa = rng.integers(0, 40, (E, W, S)).astype(np.uint8)          # some above the SKU's maximum: clipped
        qa[rng.random((E, W, S)) < 0.3] = 0
        env.step(torch.from_numpy(qa).cuda(), orders=_orders(rng, E, S, R))
        placed.append(np.minimum(qa, maxq).astype(np.uint8))
        ring = env.ring_qty.cpu().numpy()
        for a in range(min(t + 1, L)):                                 # plane (t - a) % L: the orders of step t - a
            assert np.array_equal(ring[:, (t - a) % L], placed[t - a]), (t, a)
        if t < L - 1:
            assert not ring[:, t + 1:].any(), t                        # planes no step has written yet: cleared by reset
    env.close()


def test_snapshot_of_the_arrival_indexed_ring_is_refused():
    """A snapshot taken before the ring was indexed by placement time has no ring entry in its fingerprint; with W = L
    its ring tensor even has the same shape. Loading it must fail and name the ring, as must a ring of another shape."""
    W = L = 6
    S, R, E = 36, 5, 4
    env, _, _, rng = _compact_env(W, S, R, L, E)
    env.reset()
    for _ in range(3):
        env.step(torch.from_numpy(rng.integers(0, 9, (E, W, S)).astype(np.uint8)).cuda(), orders=_orders(rng, E, S, R))
    sd = env.state_dict()
    old = dict(sd, fingerprint={k: v for k, v in sd["fingerprint"].items() if k != "ring_qty"})
    with pytest.raises(ValueError, match="ring_qty"):
        env.load_state_dict(old)
    env.load_state_dict(sd)                                            # the snapshot as taken still loads

    env2, _, _, _ = _compact_env(5, S, R, 3, E)                        # W != L: the old [E,W,L,S] ring has another shape
    env2.reset()
    sd2 = env2.state_dict()
    sd2["tensors"]["ring_qty"] = sd2["tensors"]["ring_qty"].permute(0, 2, 1, 3).contiguous()
    with pytest.raises(ValueError, match="ring_qty"):
        env2.load_state_dict(sd2)
    env.close()
    env2.close()


def test_base_stock_in_transit_before_and_after_wrap():
    """The base-stock heuristic orders clip(level - stock - in transit, 0, max) on the state before the step, where in
    transit counts the orders of age 1 .. lead (this step's arrivals included). Leads 1 and L side by side in every row;
    steps 0 .. 2L + 2. The quantities the step placed with the in-step policy are read back from the ring, the policy
    kernel's actions are compared as floats."""
    W, S, R, E, L = 5, 36, 6, 13, 7
    leads = np.random.default_rng(3).integers(1, L + 1, (W, S))
    leads[:, 0::3] = 1
    leads[:, 1::3] = L
    env, lead, maxq, rng = _compact_env(W, S, R, L, E, leads=leads)
    level_np = rng.integers(0, 70, (W, S)).astype(np.float32)          # integers: the quantities are exact
    level = torch.from_numpy(level_np).cuda()
    env.reset()
    for t in range(2 * L + 3):
        inv = env.inventory.cpu().numpy().astype(np.int64)
        ring = env.ring_qty.cpu().numpy().astype(np.int64)
        pend = np.zeros((E, W, S), np.int64)
        for a in range(1, L + 1):                                      # the orders placed a steps ago, still on their way
            if t - a >= 0:
                pend += ring[:, (t - a) % L] * (lead >= a)[None]
        want = np.clip(level_np.astype(np.float64)[None] - inv - pend, 0.0, maxq)
        k5 = env.base_stock_actions(level).cpu().numpy()
        np.testing.assert_allclose(k5, (2.0 * want / maxq - 1.0).astype(np.float32), rtol=0, atol=1e-6, err_msg=f"K5 t={t}")
        assert np.array_equal(env.pending_matrix().cpu().numpy(), pend.astype(np.float32)), t
        env.step(None, orders=_orders(rng, E, S, R), base_stock_level=level)
        assert np.array_equal(env.ring_qty[:, t % L].cpu().numpy(), want.astype(np.uint8)), t
    env.close()
