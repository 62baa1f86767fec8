"""NumPy reference of the device samplers in csrc/samplers.cu: K4 (marlsc_demand_sample, marlsc_demand_sample_lines)
and K4b (marlsc_lead_sample).

The kernels draw from Philox4x32-10 keyed by the seed, with counters that name the draw (environment, tag, step,
region or SKU), so every draw can be recomputed here and compared draw for draw:

- order counts of environment e, region r at step t: counter {e, (e >> 32) ^ 0x5bd1e995, t, r}, uniform from the top
  24 bits of word 0;
- SKU cells of order row i (the i-th order of the environment, regions ascending): counter
  {e, i | 0x80000000, t, s0 + lane}, word j holding SKU s0 + lane + 32 j (s0 = 0, 128, 256, ...). Of each word the low
  12 bits decide inclusion and the high 20 bits are the quantity uniform;
- lead times: counter {q, (q >> 32) ^ 0x1ead71e5, t, t >> 32} for the four cells 4q .. 4q + 3.

The step enters the demand counters with its low 32 bits only, like the kernels. Counts and quantities are Poisson
inversions: the smallest k with u <= F(k). The kernels evaluate F in float32 (order counts, the tail of the quantity
table) or read a float32 table built in double, so near a CDF step their k may differ from the float64 inversion done
here. ``invert`` accepts the device's k where u lies within a stated margin of the steps that bracket it, counts
those draws and then carries on from the device's value; every other draw must be identical.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
from scipy.special import gammaln

M32 = np.uint64(0xFFFFFFFF)
COUNT_TAG = 0x5bd1e995
LEAD_TAG = 0x1ead71e5
KCDF = 16                     # tabulated quantity CDF entries per cell (kCdf in samplers.cu)
MARGIN_TABLE = 2.0 ** -22     # a float32 table entry rounded from double: half an ulp below 1 is 2^-25


def margin_sum(k):
    """Margin of a float32 running CDF sum that reached term k: a few ulp of F per term."""
    return (np.asarray(k, dtype=np.float64) + 2.0) * 2.0 ** -22


# ------------------------------------------------------------------------------------------------------------ Philox
def philox4x32_10(ctr, seed: int) -> np.ndarray:
    """Philox4x32-10 (Salmon et al., SC'11; Random123) of counters ``ctr`` [..., 4] (any integer dtype, taken mod 2^32)
    under the 64-bit key ``seed`` (low word first). Returns uint32 [..., 4]."""
    c = np.asarray(ctr).astype(np.uint64) & M32
    c0, c1, c2, c3 = (c[..., i].copy() for i in range(4))
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    w0, w1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2            # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = ((p1 >> s32) ^ c1 ^ k0), p1 & M32, ((p0 >> s32) ^ c3 ^ k1), p0 & M32
        k0, k1 = (k0 + w0) & M32, (k1 + w1) & M32
    return np.stack([c0, c1, c2, c3], axis=-1).astype(np.uint32)


def u24(w: np.ndarray) -> np.ndarray:
    """The kernels' u01: the top 24 bits of a word over 2^24 (exact in float32 and float64)."""
    return (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


# --------------------------------------------------------------------------------------------------- inversion
def poisson_cdf(lam: float, kmax: Optional[int] = None) -> np.ndarray:
    """P(X <= k) for X ~ Poisson(lam), k = 0 .. kmax, in float64 (pmf in log space, then a cumulative sum)."""
    if kmax is None:
        kmax = int(lam + 12.0 * np.sqrt(lam) + 60.0)
    k = np.arange(kmax + 1, dtype=np.float64)
    if lam <= 0.0:
        return np.ones(kmax + 1)
    return np.cumsum(np.exp(k * np.log(lam) - lam - gammaln(k + 1.0)))


class Inverter:
    """Poisson inversion in float64 with the device's value accepted inside a margin.

    ``invert(lam, u, margin, dev, floor)`` returns max(floor, k) for the k to use. Where the device's value differs from
    max(floor, k) of the float64 inversion, it is accepted (and counted in ``accepted``) if u lies within
    ``margin(k_dev)`` of the CDF steps that bracket it, F(k_dev - 1) - m < u <= F(k_dev) + m (no lower bound when
    k_dev == floor): the device's k is the exact inversion of a CDF off by at most m. Any other difference is counted
    in ``rejected`` and the float64 value is kept, so the comparison that follows fails. A negative device value means
    "not known" (a draw the device dropped) and takes the float64 value."""

    def __init__(self):
        self._cdf: Dict[float, np.ndarray] = {}
        self.draws = 0
        self.accepted = 0
        self.rejected = 0

    def cdf(self, lam: float) -> np.ndarray:
        if lam not in self._cdf:
            self._cdf[lam] = poisson_cdf(lam)
        return self._cdf[lam]

    def invert(self, lam, u, margin, dev=None, floor: int = 0) -> np.ndarray:
        lam = np.asarray(lam, dtype=np.float64)
        u = np.asarray(u, dtype=np.float64)
        lam, u = np.broadcast_arrays(lam, u)
        k = np.zeros(u.shape, dtype=np.int64)
        lo = np.zeros(u.shape)
        hi = np.zeros(u.shape)
        dk = None if dev is None else np.broadcast_to(np.asarray(dev, dtype=np.int64), u.shape)
        for v in np.unique(lam):
            sel = lam == v
            F = self.cdf(float(v))
            k[sel] = np.minimum(np.searchsorted(F, u[sel], side="left"), F.size - 1)
            if dk is not None:
                kd = np.clip(dk[sel], 0, F.size - 1)
                hi[sel] = F[kd]
                lo[sel] = np.where(kd > floor, F[np.maximum(kd - 1, 0)], -np.inf)
        self.draws += u.size
        k = np.maximum(k, floor)
        if dk is None:
            return k
        diff = (dk >= 0) & (dk != k)
        if diff.any():
            m = margin(dk)
            ok = diff & (u <= hi + m) & (u > lo - m)
            self.accepted += int(ok.sum())
            self.rejected += int((diff & ~ok).sum())
            k = np.where(ok, dk, k)
        return k

    def summary(self) -> str:
        return f"{self.accepted} of {self.draws} inversions accepted within the margin, {self.rejected} rejected"


def rates32(x) -> np.ndarray:
    """The rates as the kernels see them: float32, widened back to float64."""
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def inclusion_split(prob) -> tuple:
    """Per region: include a cell when b12 < t or (b12 == t and b20 < f), with t = floor(4096 p) and f =
    round(frac(4096 p) 2^20) - probability p to within 2^-33. A cell included with b12 == t takes b20 * float(1 / f) as
    its quantity uniform, any other b20 / 2^20."""
    x = np.asarray(prob, dtype=np.float64) * 4096.0
    t = np.floor(x)
    f = np.rint((x - t) * 2.0 ** 20)
    carry = f >= 2.0 ** 20
    return np.where(carry, t + 1, t).astype(np.int64), np.where(carry, 0, f).astype(np.int64)


def _cells(words: np.ndarray, t: np.ndarray, f: np.ndarray):
    """Inclusion mask and quantity uniform (float32 arithmetic, like the kernels) of cell words."""
    w = words.astype(np.int64)
    b12, b20 = w & 0xFFF, w >> 12
    inc = (b12 < t) | ((b12 == t) & (b20 < f))
    uq = (b20.astype(np.float32) * np.float32(2.0 ** -20)).astype(np.float64)
    edge = inc & (b12 == t)                                   # included on the boundary bucket: b20 is uniform below f
    if edge.any():
        inv_f = (1.0 / np.broadcast_to(f, w.shape)[edge].astype(np.float64)).astype(np.float32)
        uq[edge] = (b20[edge].astype(np.float32) * inv_f).astype(np.float64)
    return inc, uq


def _qty_margin(k):
    k = np.asarray(k)
    return np.where(k < KCDF - 1, MARGIN_TABLE, margin_sum(k))


def _sku_words(E: int, rows: np.ndarray, env: np.ndarray, S: int, seed: int, step: int) -> np.ndarray:
    """Cell words [n, S] of order rows (row index ``rows`` of environment ``env``)."""
    nblk = (S + 127) // 128
    lanes = np.arange(32)
    out = np.zeros((rows.size, nblk * 128), dtype=np.uint32)
    for b in range(nblk):
        ctr = np.zeros((rows.size, 32, 4), dtype=np.uint64)
        ctr[..., 0] = env[:, None]
        ctr[..., 1] = (rows[:, None].astype(np.uint64) | np.uint64(0x80000000))
        ctr[..., 2] = np.uint64(step) & M32
        ctr[..., 3] = b * 128 + lanes[None, :]
        w = philox4x32_10(ctr, seed)                                # [n, 32 lanes, 4 words]: SKU b*128 + lane + 32 j
        out[:, b * 128:(b + 1) * 128] = w.transpose(0, 2, 1).reshape(rows.size, 128)
    return out[:, :S]


def _order_counts(lam_o32, E: int, seed: int, step: int, inv: Inverter, dev_counts=None) -> np.ndarray:
    R = lam_o32.size
    e = np.arange(E, dtype=np.uint64)
    ctr = np.zeros((E, R, 4), dtype=np.uint64)
    ctr[..., 0] = e[:, None]
    ctr[..., 1] = ((e >> np.uint64(32)) ^ np.uint64(COUNT_TAG))[:, None]
    ctr[..., 2] = np.uint64(step) & M32
    ctr[..., 3] = np.arange(R)[None, :]
    u = u24(philox4x32_10(ctr, seed)[..., 0])
    return inv.invert(np.broadcast_to(lam_o32, (E, R)), u, margin_sum, dev_counts)


def _orders(per_region: np.ndarray):
    """Row-major order list of every environment: (env, row, region) for each order, regions ascending."""
    E, R = per_region.shape
    n = per_region.sum(1)
    env = np.repeat(np.arange(E), n)
    reg = np.concatenate([np.repeat(np.arange(R), per_region[e]) for e in range(E)]) if n.sum() else np.zeros(0, np.int64)
    start = np.concatenate([[0], np.cumsum(n)[:-1]])
    row = np.arange(n.sum()) - np.repeat(start, n)
    return env, row, reg


def _quantities(words, reg, lam_q32, t, f, inv: Inverter, dev_q=None):
    """Quantities [n, S] of order rows with cell words ``words`` [n, S]: 0 if excluded, else clip(max(1, Poisson), 255)."""
    inc, uq = _cells(words, t[reg][:, None], f[reg][:, None])
    lam = lam_q32[reg]                                       # [n, S]
    q = np.zeros(words.shape, dtype=np.int64)
    if inc.any():
        dev = None if dev_q is None else dev_q.astype(np.int64)[inc]
        q[inc] = np.minimum(inv.invert(lam[inc], uq[inc], _qty_margin, dev, floor=1), 255)
    return q


def _device_per_region(region: np.ndarray, counts: np.ndarray, R: int, omax: int) -> np.ndarray:
    """Per-region order counts [E, R] read off the device's rows; -1 where a cut at omax hides them."""
    E = counts.size
    out = np.zeros((E, R), dtype=np.int64)
    for e in range(E):
        out[e] = np.bincount(region[e, :counts[e]].astype(np.int64), minlength=R)[:R]
        if counts[e] >= omax:                                # the last region present and all after it may be cut
            last = int(region[e, counts[e] - 1]) if counts[e] else 0
            out[e, last:] = -1
    return out


def ref_demand_dense(lam_o, prob, lam_q, E: int, seed: int, step: int, omax: int,
                     device: Optional[dict] = None, inv: Optional[Inverter] = None) -> dict:
    """What ``marlsc_demand_sample`` writes, for rates ``lam_o`` [R], inclusion probabilities ``prob`` [R] and quantity
    rates ``lam_q`` [R, S]: ``counts`` [E], ``region`` [E, omax], ``qty`` [E, omax, S] (uint8) and ``overflow``. Rows
    at and past ``counts[e]`` are zero here; the kernel leaves them untouched. ``device`` (dict with ``counts`` [E],
    ``region`` [E, omax], ``qty`` [E, omax, S]) lets the inversions accept the device's k near a CDF step (see
    Inverter); pass ``inv`` to collect the statistics. ``per_region`` [E, R] of the result holds the order counts."""
    inv = inv or Inverter()
    lam_o32 = rates32(lam_o).reshape(-1)
    R = lam_o32.size
    lam_q32 = rates32(lam_q)
    S = lam_q32.shape[1]
    t, f = inclusion_split(np.asarray(prob, np.float64).reshape(R))
    dev_pr = None
    if device is not None:
        dev_pr = _device_per_region(np.asarray(device["region"]).reshape(E, omax), np.asarray(device["counts"]), R, omax)
    per_region = _order_counts(lam_o32, E, seed, step, inv, dev_pr)
    total = per_region.sum(1)
    counts = np.minimum(total, omax)
    # truncate each environment's region-major order list at omax
    keep = np.minimum(per_region, np.maximum(0, omax - np.concatenate([np.zeros((E, 1), np.int64),
                                                                       np.cumsum(per_region, 1)[:, :-1]], 1)))
    env, row, reg = _orders(keep)
    words = _sku_words(E, row.astype(np.uint64), env.astype(np.uint64), S, seed, step)
    dev_q = None
    if device is not None:
        dev_counts = np.asarray(device["counts"]).astype(np.int64)
        if np.array_equal(dev_counts, counts):
            dev_q = np.asarray(device["qty"]).reshape(E, omax, S)[env, row]
    q = _quantities(words, reg, lam_q32, t, f, inv, dev_q)
    region = np.zeros((E, omax), dtype=np.int16)
    region[env, row] = reg
    qty = np.zeros((E, omax, S), dtype=np.uint8)
    qty[env, row] = q
    return dict(counts=counts.astype(np.int32), region=region, qty=qty, overflow=bool((total > omax).any()),
                per_region=per_region)


def ref_demand_lines(lam_o, prob, lam_q, E: int, seed: int, step: int, stride: int, region_map=None,
                     device: Optional[dict] = None, inv: Optional[Inverter] = None,
                     per_region: Optional[np.ndarray] = None) -> dict:
    """What ``marlsc_demand_sample_lines`` writes: ``counts`` [E] (entries of every lane's stream, 0 for an environment
    without demand) and ``streams`` [E, 32, stride] uint16 - entry p of lane l. Entries 0 and 1 hold the lane's SKU map
    (SKU lane + 32 k in byte k, 255 past S), then every included cell of the lane's SKUs as q | rm << 8 | j << 14 (SKU
    lane + 32 j, rm the mapped region); orders go in pairs, the first order's cells of a lane before the second's; each
    stream is zero-padded to the environment's even entry count; entries past ``stride`` are dropped and set
    ``overflow``. ``device`` (dict with ``streams`` as ``device_streams`` returns them) accepts the device's quantities
    near a CDF step. The lines carry no per-order record, so order counts near a CDF step cannot be read back from
    them: pass ``per_region`` (e.g. the result of ``ref_demand_dense`` checked against the dense kernel at the same seed
    and step) to use counts already checked."""
    inv = inv or Inverter()
    lam_o32 = rates32(lam_o).reshape(-1)
    R = lam_o32.size
    lam_q32 = rates32(lam_q)
    S = lam_q32.shape[1]
    t, f = inclusion_split(np.asarray(prob, np.float64).reshape(R))
    rm = np.arange(R) if region_map is None else np.asarray(region_map, dtype=np.int64)
    if per_region is None:
        per_region = _order_counts(lam_o32, E, seed, step, inv)
    env, row, reg = _orders(per_region)
    words = _sku_words(E, row.astype(np.uint64), env.astype(np.uint64), S, seed, step)
    inc, _ = _cells(words, t[reg][:, None], f[reg][:, None])
    # position of each included cell in its lane's stream: orders in pairs (rows 2i, 2i+1 of a region's run share a
    # pair), within a pair and lane the first order's slots j = 0..3, then the second's
    start = np.concatenate([[0], np.cumsum(per_region.reshape(-1))[:-1]]).reshape(E, R)
    first_row = start - np.concatenate([[0], np.cumsum(per_region.sum(1))[:-1]])[:, None]     # row of a region's first order
    within = row - first_row[env, reg]                         # index of the order inside its region's run
    s_idx = np.nonzero(inc)
    o_idx, sk = s_idx
    lane, j = sk % 32, sk // 32
    pair_key = row[o_idx] - (within[o_idx] & 1)                # row of the pair's first order
    second = within[o_idx] & 1
    order = np.lexsort((j, second, pair_key, lane, env[o_idx]))
    o_idx, sk, lane, j = o_idx[order], sk[order], lane[order], j[order]
    e_of = env[o_idx]
    # quantities of the included cells
    q = np.zeros(o_idx.size, dtype=np.int64)
    dev_q = None
    streams = np.zeros((E, 32, stride), dtype=np.uint16)
    key = e_of * 32 + lane
    n_key = np.bincount(key, minlength=E * 32) if key.size else np.zeros(E * 32, np.int64)
    first = np.concatenate([[0], np.cumsum(n_key)[:-1]])
    pos = 2 + np.arange(o_idx.size) - first[key] if key.size else np.zeros(0, np.int64)
    if device is not None and o_idx.size:
        ds = np.asarray(device["streams"]).astype(np.int64)
        inside = pos < stride
        dev_q = np.full(o_idx.size, -1, dtype=np.int64)
        dev_q[inside] = ds[e_of[inside], lane[inside], pos[inside]] & 0xFF
    if o_idx.size:
        uq = _cells(words[o_idx, sk], t[reg[o_idx]], f[reg[o_idx]])[1]
        q = np.minimum(inv.invert(lam_q32[reg[o_idx], sk], uq, _qty_margin, dev_q, floor=1), 255)
    entry = (q | (rm[reg[o_idx]] << 8) | (j << 14)).astype(np.uint16)
    inside = pos < stride
    streams[e_of[inside], lane[inside], pos[inside]] = entry[inside]
    cnt = np.minimum(2 + n_key.reshape(E, 32), stride)
    longest = cnt.max(1)
    rounds = np.where(longest > 2, (longest + 1) & ~1, 0)
    smap = np.zeros(32, dtype=np.int64)
    lanes = np.arange(32)
    for k4 in range(4):
        s = lanes + 32 * k4
        smap |= np.where(s < S, s, 255) << (8 * k4)
    has = rounds > 0
    streams[has, :, 0] = (smap & 0xFFFF).astype(np.uint16)[None, :]
    streams[has, :, 1] = (smap >> 16).astype(np.uint16)[None, :]
    return dict(counts=rounds.astype(np.int32), streams=streams, overflow=bool((2 + n_key > stride).any()),
                per_region=per_region)


def device_streams(lines: np.ndarray, E: int, stride: int) -> np.ndarray:
    """The device's line buffer ([E * stride, 32] 16-bit words; entry p of lane l at row 2 (p >> 1) + l // 16, column
    2 (l % 16) + (p & 1)) as [E, 32, stride] streams."""
    a = np.asarray(lines).view(np.uint16).reshape(E, stride // 2, 32, 2)     # [env, entry pair, lane, entry & 1]
    return a.transpose(0, 2, 1, 3).reshape(E, 32, stride)


def ref_lead(expected, max_dev, E: int, seed: int, step: int) -> np.ndarray:
    """What ``marlsc_lead_sample`` writes: [E, W, S] uint8, clip(expected[w, s] + umulhi(word, 2d + 1) - d, 1, 255) with
    d = max_dev[s], four consecutive cells per Philox call."""
    expected = np.asarray(expected, dtype=np.int64)
    W, S = expected.shape
    n = E * W * S
    nq = (n + 3) // 4
    q = np.arange(nq, dtype=np.uint64)
    ctr = np.zeros((nq, 4), dtype=np.uint64)
    ctr[:, 0] = q & M32
    ctr[:, 1] = (q >> np.uint64(32)) ^ np.uint64(LEAD_TAG)
    ctr[:, 2] = np.uint64(step & 0xFFFFFFFF)
    ctr[:, 3] = np.uint64((step >> 32) & 0xFFFFFFFF)
    w = philox4x32_10(ctr, seed).reshape(-1)[:n].astype(np.uint64)
    cell = np.arange(n) % (W * S)
    d = np.asarray(max_dev, dtype=np.int64).reshape(-1)[cell % S]
    dev = ((w * (2 * d + 1).astype(np.uint64)) >> np.uint64(32)).astype(np.int64) - d
    return np.clip(expected.reshape(-1)[cell] + dev, 1, 255).astype(np.uint8).reshape(E, W, S)
