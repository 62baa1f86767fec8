"""The device samplers K4 (marlsc_demand_sample, marlsc_demand_sample_lines) and K4b (marlsc_lead_sample) against the
NumPy reference in sampler_reference.py: draw for draw (the Philox counters are reproduced on the host), then their law
against scipy with 2^20 or more draws, then the environment plumbing that feeds them.

Replayed inversions may differ from the float64 reference only where u lies within the stated margin of a CDF step
(sampler_reference.Inverter): 2^-22 for a float32 table entry, (k + 2) 2^-22 for a float32 running sum that reached k.
Such draws are counted, printed and must stay below 1e-4 of all draws."""
import ctypes as C

import numpy as np
import pytest

from sampler_reference import (Inverter, device_streams, inclusion_split, philox4x32_10, poisson_cdf, ref_demand_dense,
                               ref_demand_lines, ref_lead)

P_CRIT = 1e-6


# ------------------------------------------------------------------------------------------------------------ CPU
def test_philox_known_answers():
    """Random123's known-answer vectors for Philox4x32-10."""
    vec = [([0, 0, 0, 0], 0, [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 4, 0xffffffffffffffff, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], 0x299f31d0a4093822,
            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, out in vec:
        assert philox4x32_10(np.array(ctr, dtype=np.uint64), key).tolist() == out
    batch = philox4x32_10(np.array([v[0] for v in vec], dtype=np.uint64)[:1].repeat(3, 0), 0)   # vectorised = scalar
    assert (batch == np.array(vec[0][2], dtype=np.uint32)).all()


def test_inclusion_split_has_probability_p():
    for p in (0.0, 1e-4, 1e-3, 0.2, 0.667, 1.0 / 3.0, 0.5, 1.0 - 1e-12, 1.0):
        t, f = (int(x[0]) for x in inclusion_split(np.array([p])))
        assert 0 <= f < 2 ** 20 and 0 <= t <= 4096
        assert abs(t / 4096 + f / 2 ** 32 - p) <= 2.0 ** -33, p


def _scalar_words(e, row, step, s, seed):
    w = philox4x32_10(np.array([e, row | 0x80000000, step & 0xffffffff, (s & ~127) + (s & 31)], dtype=np.uint64), seed)
    return int(w[(s >> 5) & 3])


def _scalar_draws(lam_o, prob, lam_q, e, seed, step):
    """One environment's orders, written as the thread kernel's loops: [(region, [(sku, q)...])...]."""
    R, S = lam_q.shape
    t, f = inclusion_split(prob)
    out = []
    row = 0
    for r in range(R):
        w = philox4x32_10(np.array([e, (e >> 32) ^ 0x5bd1e995, step & 0xffffffff, r], dtype=np.uint64), seed)
        u = (int(w[0]) >> 8) * 2.0 ** -24
        n = int(np.searchsorted(poisson_cdf(float(np.float32(lam_o[r]))), u, side="left"))
        for _ in range(n):
            cells = []
            for s in range(S):
                x = _scalar_words(e, row, step, s, seed)
                b12, b20 = x & 0xfff, x >> 12
                if b12 < t[r] or (b12 == t[r] and b20 < f[r]):
                    uq = float(np.float32(b20) * (np.float32(1.0 / f[r]) if b12 == t[r] else np.float32(2.0 ** -20)))
                    k = int(np.searchsorted(poisson_cdf(float(np.float32(lam_q[r, s]))), uq, side="left"))
                    cells.append((s, min(max(k, 1), 255)))
            out.append((r, cells))
            row += 1
    return out


def test_reference_layouts_match_a_scalar_transcription():
    """The vectorised reference builders against the kernels' loops transcribed one draw at a time: dense rows with a cut
    at omax, lane streams (pairs of orders, SKU map, padding, cut at stride) and lead times."""
    rng = np.random.default_rng(4)
    R, S, E, seed, step = 4, 70, 9, (3 << 32) + 17, (1 << 32) + 5
    lam_o = np.array([1.5, 0.0, 2.5, 0.7])
    prob = np.array([0.3, 0.5, 1.0 / 3.0, 0.05])
    lam_q = rng.uniform(0.5, 20.0, (R, S))
    draws = [_scalar_draws(lam_o, prob, lam_q, e, seed, step) for e in range(E)]
    omax = 5
    dense = ref_demand_dense(lam_o, prob, lam_q, E, seed, step, omax)
    assert dense["overflow"] == any(len(d) > omax for d in draws)
    for e, d in enumerate(draws):
        assert dense["counts"][e] == min(len(d), omax)
        for i, (r, cells) in enumerate(d[:omax]):
            q = np.zeros(S, np.uint8)
            for s, v in cells:
                q[s] = v
            assert dense["region"][e, i] == r and np.array_equal(dense["qty"][e, i], q), (e, i)
    rmap = np.array([3, 0, 2, 1])
    for stride in (64, 6):
        lines = ref_demand_lines(lam_o, prob, lam_q, E, seed, step, stride, rmap)
        over = False
        for e, d in enumerate(draws):
            streams = [[] for _ in range(32)]
            row_of_region = {}
            for r, cells in d:
                row_of_region.setdefault(r, []).append(cells)
            for r in sorted(row_of_region):
                orders = row_of_region[r]
                for i in range(0, len(orders), 2):
                    for lane in range(32):
                        for cells in orders[i:i + 2]:
                            for s, v in cells:
                                if s % 32 == lane:
                                    streams[lane].append(v | int(rmap[r]) << 8 | (s // 32) << 14)
            cnt = [min(2 + len(x), stride) for x in streams]
            over = over or any(2 + len(x) > stride for x in streams)
            rounds = 0 if max(cnt) <= 2 else (max(cnt) + 1) & ~1
            assert lines["counts"][e] == rounds, (stride, e)
            for lane in range(32 if rounds else 0):
                m = sum((lane + 32 * k if lane + 32 * k < S else 255) << (8 * k) for k in range(4))
                want = [m & 0xffff, m >> 16] + streams[lane][:stride - 2]
                want += [0] * (rounds - len(want))
                assert lines["streams"][e, lane, :rounds].tolist() == want[:rounds], (stride, e, lane)
        assert lines["overflow"] == over
    exp = rng.integers(1, 250, (3, 7))
    md = np.array([0, 1, 3, 9, 2, 0, 12])
    lead = ref_lead(exp, md, 5, seed, step)
    for i in range(5 * 21):
        w = philox4x32_10(np.array([i // 4, 0x1ead71e5, step & 0xffffffff, step >> 32], dtype=np.uint64), seed)[i % 4]
        cell = i % 21
        d = int(md[cell % 7])
        v = int(exp.reshape(-1)[cell]) + ((int(w) * (2 * d + 1)) >> 32) - d
        assert lead.reshape(-1)[i] == min(max(v, 1), 255)


# ------------------------------------------------------------------------------------------------------------ GPU
class _Sampler:
    """A marlsc_demand handle and the calls of the C ABI, results on the host."""

    def __init__(self, lam_o, prob, lam_q):
        from marlsc_b200 import _capi
        self.L = _capi.lib()
        self.check = _capi.check
        self.params = [np.ascontiguousarray(v, np.float64) for v in (lam_o, prob, lam_q)]
        self.R, self.S = self.params[2].shape
        dbl = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
        self.h = C.c_void_p()
        self.check(self.L.marlsc_demand_create(self.R, self.S, *(dbl(v) for v in self.params), 0, C.byref(self.h)))

    def _stream(self):
        import torch
        return torch.cuda.current_stream().cuda_stream

    def dense(self, E, seed, step, omax):
        import torch
        counts = torch.full((E,), -1, dtype=torch.int32, device="cuda")
        region = torch.full((E * omax,), -1, dtype=torch.int16, device="cuda")
        qty = torch.zeros(E * omax * self.S + 16, dtype=torch.uint8, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        self.check(self.L.marlsc_demand_sample(self.h, E, seed, step, omax, counts.data_ptr(), region.data_ptr(), qty.data_ptr(),
                                               flag.data_ptr(), self._stream()))
        return dict(counts=counts.cpu().numpy(), region=region.cpu().numpy().reshape(E, omax),
                    qty=qty.cpu().numpy()[:E * omax * self.S].reshape(E, omax, self.S), overflow=bool(flag.item()))

    def lines(self, E, seed, step, stride, region_map=None):
        import torch
        lines = torch.full((E * stride, 32), -1, dtype=torch.int16, device="cuda")
        counts = torch.full((E,), -1, dtype=torch.int32, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        rm = None if region_map is None else torch.from_numpy(np.asarray(region_map, np.int32)).cuda()
        self.check(self.L.marlsc_demand_sample_lines(self.h, E, seed, step, stride, None if rm is None else rm.data_ptr(),
                                                     lines.data_ptr(), counts.data_ptr(), flag.data_ptr(), self._stream()))
        return dict(counts=counts.cpu().numpy(), streams=device_streams(lines.cpu().numpy(), E, stride), overflow=bool(flag.item()))

    def close(self):
        self.L.marlsc_demand_destroy(self.h)


def _check_dense(smp, E, seed, step, omax, inv):
    """Replay of one dense draw; returns the reference (its per-region counts are checked)."""
    dev = smp.dense(E, seed, step, omax)
    ref = ref_demand_dense(*smp.params, E, seed, step, omax, device=dev, inv=inv)
    assert inv.rejected == 0, inv.summary()
    assert np.array_equal(dev["counts"], ref["counts"])
    assert dev["overflow"] == ref["overflow"]
    for e in range(E):
        n = ref["counts"][e]
        assert np.array_equal(dev["region"][e, :n], ref["region"][e, :n]), e
        assert np.array_equal(dev["qty"][e, :n], ref["qty"][e, :n]), e
    return ref


def _check_lines(smp, E, seed, step, stride, inv, region_map=None, per_region=None):
    dev = smp.lines(E, seed, step, stride, region_map)
    ref = ref_demand_lines(*smp.params, E, seed, step, stride, region_map, device=dev, inv=inv, per_region=per_region)
    assert inv.rejected == 0, inv.summary()
    assert np.array_equal(dev["counts"], ref["counts"])
    assert dev["overflow"] == ref["overflow"]
    for e in range(E):
        n = ref["counts"][e]
        assert np.array_equal(dev["streams"][e, :, :n], ref["streams"][e, :, :n]), e
    return ref


def _rates(rng, R, S, kind, per_cell):
    """Order rates, inclusion probabilities and quantity rates for a replay case. ``kind``: 'grid' keeps 4096 p an
    integer and every rate below 30; 'any' draws p freely; 'high' adds rates of 30 and more."""
    lam_o = rng.uniform(0.05, 1.2, R)
    lam_o[rng.random(R) < 0.15] = 0.0
    if kind == "grid":
        prob = rng.integers(0, 4097, R) / 4096.0
    else:
        prob = rng.uniform(0.0, 1.0, R)
        special = rng.random(R) < 0.3
        prob[special] = rng.choice([1e-4, 1e-3, 0.2, 0.667], int(special.sum()))
    prob[rng.random(R) < 0.15] = 0.0
    prob[rng.random(R) < 0.15] = 1.0
    top = 60.0 if kind == "high" else 25.0
    lam_q = rng.choice([0.0, 0.3, 1.0, 5.0, 12.5, 18.0, 24.0, top, 2 * top], (R, S if per_cell else 1))
    lam_q = np.where(lam_q > 25.0, lam_q if kind == "high" else 20.0, lam_q)
    if kind == "high":
        lam_o[:2] = 31.5
        lam_q[rng.random(lam_q.shape) < 0.1] = 100.0
    return lam_o, prob, np.broadcast_to(lam_q, (R, S)).copy()


DENSE_CASES = [(1, 1), (2, 3), (16, 32), (17, 33), (32, 64), (33, 3), (100, 50), (128, 32), (129, 5), (300, 100), (2, 100)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "any", "high"])
@pytest.mark.parametrize("per_cell", [False, True])
@pytest.mark.parametrize("S,R", DENSE_CASES)
def test_dense_sampler_replays_reference(S, R, per_cell, kind):
    """marlsc_demand_sample draw for draw: the thread kernel (S <= 16) and the warp kernel (both SKU blocks past 128),
    per-region and per-cell rates, rates in the CDF table's tail, rate 0, p in {0, 1}, E not a multiple of 4 or 128,
    seeds and steps past 2^32, and an omax that cuts the orders."""
    rng = np.random.default_rng(S * 1000 + R + 7 * per_cell + len(kind))
    smp = _Sampler(*_rates(rng, R, S, kind, per_cell))
    E = 203 if S * R < 3000 else 37
    inv = Inverter()
    try:
        for seed, step in ((5, 0), ((7 << 32) + 3, 9), (11, (1 << 32) + 2)):
            total = smp.params[0].sum()
            omax = int(total + 6 * np.sqrt(total + 1) + 8)
            ref = _check_dense(smp, E, seed, step, omax, inv)
            assert not ref["overflow"]
        # an omax that cuts most environments: the flag is set, every row before the cut is exact
        cut = max(1, int(0.5 * smp.params[0].sum()))
        ref = _check_dense(smp, E, 3, 4, cut, inv)
        assert ref["overflow"] == bool((ref["per_region"].sum(1) > cut).any())
    finally:
        smp.close()
    print(f"dense S={S} R={R} per_cell={per_cell} {kind}: {inv.summary()}")
    assert inv.accepted <= 1e-4 * inv.draws, inv.summary()


LINE_CASES = [(1, 1), (2, 3), (16, 32), (17, 33), (32, 64), (33, 3), (100, 50), (128, 32), (128, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "any", "high"])
@pytest.mark.parametrize("S,R", LINE_CASES)
def test_lines_sampler_replays_reference(S, R, kind):
    """marlsc_demand_sample_lines draw for draw: the lane streams (SKU map, pairs of orders, padding, the environment's
    even entry count, 0 for an environment without demand), with and without a region map, per-cell rates, and a
    stride that cuts the streams (flag set, every entry before the cut exact). The order counts are the dense
    kernel's at the same seed and step, checked against the reference first."""
    rng = np.random.default_rng(S * 100 + R + len(kind))
    smp = _Sampler(*_rates(rng, R, S, kind, per_cell=S % 2 == 1))
    E = 133
    inv = Inverter()
    rmap = rng.integers(0, 64, R)
    try:
        omax = int(smp.params[0].sum() * 3 + 40)
        wide = 2 + 4 * omax                                          # room for every cell of omax orders in one lane
        for seed, step, stride, region_map in ((5, 0, wide, None), ((9 << 32) + 1, (1 << 32) + 7, wide, rmap), (13, 2, 6, None)):
            pr = _check_dense(smp, E, seed, step, omax, inv)["per_region"]
            ref = _check_lines(smp, E, seed, step, stride, inv, region_map, pr)
            if stride == 6:
                assert ref["overflow"] or (ref["counts"] <= 6).all()
            else:
                assert not ref["overflow"]
    finally:
        smp.close()
    print(f"lines S={S} R={R} {kind}: {inv.summary()}")
    assert inv.accepted <= 1e-4 * inv.draws, inv.summary()


@pytest.mark.gpu
@pytest.mark.parametrize("W,S,E", [(3, 5, 1001), (2, 7, 3), (10, 100, 333), (1, 1, 5)])
def test_lead_sampler_replays_reference(W, S, E):
    """marlsc_lead_sample bit for bit: cell counts not a multiple of 4, deviations larger than the expected lead
    (clipped at 1), expected + deviation above 255 (clipped at 255), seeds and steps past 2^32, and an output pointer
    one byte off alignment (the scalar store path)."""
    import torch
    from marlsc_b200 import _capi
    rng = np.random.default_rng(W * S + E)
    exp = rng.integers(1, 256, (W, S)).astype(np.int32)
    exp.reshape(-1)[::3] = rng.integers(1, 4, exp.size)[::3]
    exp.reshape(-1)[1::5] = 250
    md = rng.integers(0, 12, S).astype(np.int32)
    md[0] = 9
    ed, mdd = torch.from_numpy(exp).cuda(), torch.from_numpy(md).cuda()
    n = E * W * S
    for seed, step, off in ((3, 0, 0), ((5 << 32) + 1, 7, 1), (2, (3 << 32) + 11, 0), (1 << 40, (1 << 33), 1)):
        buf = torch.zeros(n + 8, dtype=torch.uint8, device="cuda")
        _capi.check(_capi.lib().marlsc_lead_sample(E, W, S, ed.data_ptr(), mdd.data_ptr(), seed, step, buf.data_ptr() + off,
                                                   torch.cuda.current_stream().cuda_stream))
        got = buf.cpu().numpy()
        assert np.array_equal(got[off:off + n].reshape(E, W, S), ref_lead(exp, md, E, seed, step)), (seed, step, off)
        assert not got[:off].any() and not got[off + n:].any()               # nothing written outside the cells
    if n >= 1000:
        want = ref_lead(exp, md, E, 3, 0)
        assert want.min() == 1 and want.max() == 255                          # both clips were exercised


# ------------------------------------------------------------------------------------------------ law against scipy
def _chi2_poisson(x, lam, floor=0):
    """Chi-square of draws ``x`` against max(floor, Poisson(lam)), bins with expectation below 5 pooled into the tails."""
    from scipy import stats
    n = x.size
    kmax = int(lam + 12 * np.sqrt(lam) + 30)
    pmf = stats.poisson.pmf(np.arange(kmax + 1), lam)
    if floor:
        pmf[floor] += pmf[:floor].sum()
        pmf[:floor] = 0.0
    lo = max(floor, int(np.argmax(np.cumsum(pmf) * n >= 5)))
    hi = int(kmax - np.argmax(np.cumsum(pmf[::-1]) * n >= 5))
    edges_p = np.concatenate([[pmf[:lo + 1].sum()], pmf[lo + 1:hi], [1.0 - pmf[:hi].sum()]])
    obs = np.concatenate([[(x <= lo).sum()], [(x == k).sum() for k in range(lo + 1, hi)], [(x >= hi).sum()]])
    chi2 = float(((obs - n * edges_p) ** 2 / (n * edges_p)).sum())
    return chi2, float(stats.chi2.ppf(1 - P_CRIT, edges_p.size - 1))


LAWS = [0.3, 5.0, 29.5, 30.0, 45.5, 100.0, 150.0]


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAWS)
def test_order_counts_follow_poisson(lam):
    """2^20 order counts of one region at rate lam against Poisson(lam)."""
    E = 1 << 20
    smp = _Sampler([lam], [0.0], [[1.0]])
    try:
        dev = smp.dense(E, 21, 3, int(lam + 8 * np.sqrt(lam) + 12))
    finally:
        smp.close()
    assert not dev["overflow"]
    chi2, crit = _chi2_poisson(dev["counts"].astype(np.int64), lam)
    print(f"order counts lambda={lam}: chi2 {chi2:.1f} (critical {crit:.1f} at p=1e-6)")
    assert chi2 < crit, (lam, chi2, crit)


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAWS)
def test_quantities_follow_poisson(lam):
    """2^21 quantities at rate lam (every SKU included) against max(1, Poisson(lam)); the thread kernel and the lines
    kernel draw them too (they share the inversion), so one of each is checked on a smaller batch."""
    E, S = 1 << 14, 128
    smp = _Sampler([1.0], [1.0], np.full((1, S), lam))
    try:
        dev = smp.dense(E, 8, 1, 16)
        n = dev["counts"]
        q = np.concatenate([dev["qty"][e, :n[e]].reshape(-1) for e in range(E)]).astype(np.int64)
        ln = smp.lines(E, 8, 1, 64)
    finally:
        smp.close()
    assert not dev["overflow"] and not ln["overflow"] and q.size >= 1 << 20
    assert q.min() >= 1
    chi2, crit = _chi2_poisson(q, lam, floor=1)
    print(f"quantities lambda={lam}: chi2 {chi2:.1f} (critical {crit:.1f} at p=1e-6), {q.size} draws")
    assert chi2 < crit, (lam, chi2, crit)
    qs = np.concatenate([ln["streams"][e, :, 2:ln["counts"][e]].reshape(-1) for e in range(E)]).astype(np.int64)
    qs = qs[qs != 0] & 0xFF
    chi2, crit = _chi2_poisson(qs, lam, floor=1)
    assert chi2 < crit, ("lines", lam, chi2, crit)


@pytest.mark.gpu
@pytest.mark.parametrize("p", [1e-4, 1e-3, 0.2, 0.667])
def test_sku_inclusion_rate_is_p(p):
    """The share of included cells over 2^23 cells against p, 5-sigma binomial band (the warp and the lines kernel)."""
    E, S = 1 << 14, 128
    smp = _Sampler([4.0], [p], np.full((1, S), 5.0))
    try:
        dev = smp.dense(E, 31, 2, 40)
        ln = smp.lines(E, 31, 2, 128)
    finally:
        smp.close()
    assert not dev["overflow"] and not ln["overflow"]
    n = dev["counts"]
    rows = int(n.sum())
    hits = sum(int((dev["qty"][e, :n[e]] > 0).sum()) for e in range(E))
    cells = rows * S
    band = 5 * np.sqrt(p * (1 - p) / cells)
    rate = hits / cells
    print(f"inclusion p={p}: {rate:.6g} over {cells} cells (band +-{band:.2g})")
    assert abs(rate - p) < band, (p, rate, band)
    line_hits = int(sum(((ln["streams"][e, :, 2:ln["counts"][e]]) != 0).sum() for e in range(E)))
    assert line_hits == hits                                    # the lines kernel includes the very same cells


@pytest.mark.gpu
def test_per_cell_rates_through_the_warp_kernel_follow_poisson():
    """Per-cell quantity rates (sku_stride 1) at S = 100, R = 50: every cell of a given rate follows its own law."""
    R, S, E = 50, 100, 4096
    vals = np.array([0.5, 3.0, 12.0, 29.5, 45.5])
    idx = (np.arange(R)[:, None] * 7 + np.arange(S)[None, :]) % vals.size
    smp = _Sampler(np.full(R, 0.1), np.full(R, 1.0), vals[idx])
    try:
        dev = smp.dense(E, 4, 6, 40)
    finally:
        smp.close()
    assert not dev["overflow"]
    n = dev["counts"]
    for i, lam in enumerate(vals):
        q = np.concatenate([dev["qty"][e, :n[e]][idx[dev["region"][e, :n[e]]] == i] for e in range(E)]).astype(np.int64)
        chi2, crit = _chi2_poisson(q, lam, floor=1)
        assert q.size > 100_000 and chi2 < crit, (lam, chi2, crit)


# ------------------------------------------------------------------------------------------------ environment plumbing
def _dense_params(env):
    lam_o, prob, lam_q = env.spec.components["demand_sampler"].dense_params()
    R, S = env.n_regions, env.n_skus
    return (np.broadcast_to(np.asarray(lam_o, np.float64), (R,)), np.broadcast_to(np.asarray(prob, np.float64), (R,)),
            np.broadcast_to(np.asarray(lam_q, np.float64).reshape(R, -1), (R, S)))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["wide", "compact"])
def test_env_device_demand_draws_reference_at_each_step(layout):
    """BatchedInventoryEnv(device_demand=True, demand_seed=s) stepped across a reset draws ref(seed=s, step=t) at its
    t-th step, in the wide layout's dense rows and in the compact layout's lines."""
    import torch
    from golden.scenarios import large_network, small_default
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    d = large_network(episode_length=6) if layout == "compact" else dict(small_default(), episode_length=6)
    cfg = environment_config_from_dict(dict(d, allow_region_mismatch=True))
    E, seed = 77, (1 << 32) + 12
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=seed, layout=layout)
    assert env.layout == layout
    W, S = env.n_warehouses, env.n_skus
    params = _dense_params(env)
    smp = _Sampler(*params)
    inv = Inverter()
    gen = torch.Generator(device="cuda:0").manual_seed(2)
    try:
        env.reset()
        for t in range(9):
            if t == 5:
                env.reset()
            env.step(torch.rand((E, W, S), device="cuda:0", generator=gen) * 2 - 1)
            dd = env._dd
            if layout == "compact":
                b = t & 1
                dev = dict(counts=dd["counts"][b].cpu().numpy(),
                           streams=device_streams(dd["lines"][b].cpu().numpy(), E, dd["stride"]))
                pr = _check_dense(smp, E, seed, t, 256, inv)["per_region"]
                ref = ref_demand_lines(*params, E, seed, t, dd["stride"], env.spec.tables["region_map"], device=dev,
                                       inv=inv, per_region=pr)
                assert np.array_equal(dev["counts"], ref["counts"]), t
                for e in range(E):
                    assert np.array_equal(dev["streams"][e, :, :ref["counts"][e]], ref["streams"][e, :, :ref["counts"][e]]), (t, e)
            else:
                omax = dd["omax"]
                dev = dict(counts=dd["counts"].cpu().numpy(), region=dd["region"].cpu().numpy().reshape(E, omax),
                           qty=dd["qty"].cpu().numpy()[:E * omax * S].reshape(E, omax, S))
                ref = ref_demand_dense(*params, E, seed, t, omax, device=dev, inv=inv)
                assert np.array_equal(dev["counts"], ref["counts"]), t
                for e in range(E):
                    n = ref["counts"][e]
                    assert np.array_equal(dev["region"][e, :n], ref["region"][e, :n]) and np.array_equal(dev["qty"][e, :n], ref["qty"][e, :n]), (t, e)
            assert inv.rejected == 0, inv.summary()
        assert not env.demand_overflowed()
    finally:
        smp.close()
        env.close()
    print(f"env {layout}: {inv.summary()}")
    assert inv.accepted <= 1e-4 * inv.draws


@pytest.mark.gpu
def test_env_device_leads_draw_reference_at_each_step():
    """enable_device_leads(seed) draws ref_lead(seed, t) at the environment's t-th step, across a reset."""
    import torch
    from golden.scenarios import allfeat_ratio_stochastic
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg = environment_config_from_dict(allfeat_ratio_stochastic())
    E, seed = 301, (2 << 32) + 5
    env = BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=1)
    env.enable_device_leads(seed=seed)
    md = np.array([0, 1, 2, 1, 0])
    exp = np.asarray(env.expected_lead_times, dtype=np.int64)
    gen = torch.Generator(device="cuda:0").manual_seed(3)
    env.reset()
    for t in range(7):
        if t == 4:
            env.reset()
        env.step(torch.rand((E, 3, 5), device="cuda:0", generator=gen) * 2 - 1)
        assert np.array_equal(env._dl["actual"].cpu().numpy(), ref_lead(exp, md, E, seed, t)), t
    env.close()


@pytest.mark.gpu
def test_compact_side_stream_prefetch_matches_in_order_draws():
    """The compact layout drawing step t+1's lines on a side stream while step t runs (``_dd["overlap"] = True``) gives
    the same lines, state, observations and rewards as drawing each step's lines in order."""
    import torch
    from golden.scenarios import large_network
    from marlsc_b200.config import environment_config_from_dict
    from marlsc_b200.envs import BatchedInventoryEnv
    cfg = environment_config_from_dict(dict(large_network(episode_length=8), allow_region_mismatch=True))
    E = 517
    envs = [BatchedInventoryEnv(cfg, E, device="cuda:0", host_samplers=False, device_demand=True, demand_seed=3, layout="compact")
            for _ in range(2)]
    envs[1]._dd["overlap"] = True
    gen = torch.Generator(device="cuda:0").manual_seed(4)
    for env in envs:
        env.reset()
    for t in range(12):
        if t == 8:
            for env in envs:
                env.reset()
        act = torch.rand((E, 10, 100), device="cuda:0", generator=gen) * 2 - 1
        out = [env.step(act) for env in envs]
        b = t & 1
        a, c = envs[0]._dd, envs[1]._dd
        assert torch.equal(a["counts"][b], c["counts"][b]), t
        assert torch.equal(a["lines"][b], c["lines"][b]), t
        assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1]), t
        assert torch.equal(envs[0].inventory, envs[1].inventory) and torch.equal(envs[0].ring_qty, envs[1].ring_qty), t
    assert envs[1]._dd["drawn"] == 12                                   # the side stream drew ahead
    for env in envs:
        env.close()
