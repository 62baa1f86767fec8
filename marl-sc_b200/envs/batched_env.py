"""BatchedInventoryEnv - E independent inventory environments advanced by one fused CUDA kernel per
timestep (csrc/env_step.cu). Tensor-in / tensor-out counterpart of the reference's
``InventoryEnvironment`` (src/environment/envs/multi_env.py:38-366); the dict-based single-env API of
the reference is provided on top of it by ``marlsc_b200.envs.InventoryEnvironment``.

State is struct-of-arrays on the device, env-major (include/marlsc_b200.h ``marlsc_env_state``):
``inventory [E,W,S]``, ``ring_qty [E,D,W,S]`` (+ ``ring_lead`` for stochastic lead times),
``demand_hist [E,5,W,S]``, ``forecast [E,W,S]``. Observations are written once per warehouse as
``obs [E,W,obs_dim]``; flattened over W this *is* the centralised-critic global state, so the
reference's per-agent ``[local_i | global]`` vector is only materialised on request
(``agent_observations``).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .. import _capi
from ..config.schema import (EnvironmentConfig, InitialInventoryCustom, InitialInventoryUniform,
                             InitialInventoryZero)
from ..demand import LineBatch, OrderBatch, pack_lines, pack_orders
from ..seeds import ENVIRONMENT_SEEDS, SeedManager
from ..spec import EnvSpec, build_env_spec


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# marlsc_episode_metrics (include/marlsc_b200.h), in field order: [E,W] accumulators, then the [E] ones
METRICS_PER_ROW = ("holding_cost", "penalty_cost", "outbound_cost", "inbound_cost", "ordered_units", "shipped_units",
                   "episode_return")
METRICS_PER_ENV = ("demand_units", "lost_units")
COST_METRICS = ("holding_cost", "penalty_cost", "outbound_cost", "inbound_cost")


def fill_rate(demand_units: torch.Tensor, lost_units: torch.Tensor) -> torch.Tensor:
    """Unit fill rate 1 - lost / demand, and 1 where nothing was demanded."""
    return torch.where(demand_units > 0, 1.0 - lost_units / demand_units.clamp(min=1.0), torch.ones_like(demand_units))


class DeviceOrders:
    """One step of demand resident on the device (CSR, see marlsc_b200.demand)."""

    def __init__(self, offsets: torch.Tensor, region: torch.Tensor, qty: torch.Tensor, n_orders: int):
        self.offsets, self.region, self.qty, self.n_orders = offsets, region, qty, n_orders

    @property
    def qty_bytes(self) -> int:
        return self.qty.element_size()

    @staticmethod
    def from_host(batch: OrderBatch, device) -> "DeviceOrders":
        region = batch.region if batch.region.size else np.zeros(1, np.int16)
        qty = torch.from_numpy(batch.qty.view(np.uint8)).to(device)
        if batch.qty_bytes == 2:
            qty = qty.view(torch.int16)   # 2-byte rows; only the element size matters to the kernel
        return DeviceOrders(torch.from_numpy(batch.offsets).to(device), torch.from_numpy(region).to(device),
                            qty, batch.n_orders)


class DeviceLines:
    """One step of demand as sparse lines on the device (CSR over environments, see marlsc_b200.demand.pack_lines and
    ``marlsc_step_io.lines`` in include/marlsc_b200.h): the native input of the compact layout."""

    def __init__(self, offsets: torch.Tensor, lines: torch.Tensor, n_lines: int, n_rounds: int):
        self.offsets, self.lines, self.n_lines, self.n_rounds = offsets, lines, int(n_lines), int(n_rounds)

    @staticmethod
    def from_host(batch: LineBatch, device) -> "DeviceLines":
        # uint16 entries travel as int16 storage (same bytes)
        return DeviceLines(torch.from_numpy(batch.offsets).to(device), torch.from_numpy(batch.lines.view(np.int16)).to(device),
                           batch.n_lines, batch.n_rounds)


class BatchedInventoryEnv:
    metadata = {"render_modes": ["human"], "name": "multi_env"}

    def __init__(self, env_config: EnvironmentConfig, num_envs: int, device: Union[str, torch.device, None] = None,
                 seed: Optional[int] = None, env_meta: Optional[Dict[str, Any]] = None,
                 region_map: Optional[Sequence[int]] = None, env_seeds: Optional[Sequence[int]] = None,
                 host_samplers: bool = True, diagnostics: bool = False, team_size: int = 0,
                 generic_kernel: bool = False, fused_kernel: bool = False, device_demand: bool = False, demand_seed: int = 0,
                 max_orders_per_env: Optional[int] = None, layout: Optional[str] = None, episode_metrics: bool = False):
        if num_envs < 1:
            raise ValueError("num_envs must be positive")
        if episode_metrics and fused_kernel and layout == "compact":
            raise ValueError("episode_metrics needs the compact layout's split step: the fused kernel does not accumulate them")
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedInventoryEnv needs a CUDA device: this path has no CPU implementation")
        meta = env_meta or {}
        self.env_config = env_config
        self.num_envs = int(num_envs)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.n_warehouses, self.n_skus, self.n_regions = env_config.n_warehouses, env_config.n_skus, env_config.n_regions
        self.episode_length = env_config.episode_length
        self.feature_config = env_config.features
        self.rolling_window = 5
        self.obs_normalization = meta.get("obs_normalization", "off")
        self.obs_stats = meta.get("obs_stats", None)
        self.include_warehouse_id = bool(meta.get("include_warehouse_id", False))
        self._num_eval_episodes = meta.get("num_eval_episodes", None)
        self.agents = [f"warehouse_{i}" for i in range(self.n_warehouses)]
        self.possible_agents = list(self.agents)
        self.diagnostics = diagnostics

        self.spec: EnvSpec = build_env_spec(env_config, self.obs_normalization, self.obs_stats, self.include_warehouse_id,
                                            region_map=region_map, data_mode=meta.get("data_mode", "train"),
                                            preprocessed_data=meta.get("preprocessed_data"))
        s = self.spec.scalars
        self.max_expected_lead_time = s["max_expected_lead"]
        self.ring_depth = s["ring_depth"]
        self.stochastic_lead = s["lead_mode"] == 1
        self.expected_lead_times = self.spec.tables["expected_lead"].copy()
        self.home_regions = self.spec.tables["home_region"].copy()

        L = _capi.lib()
        self._spec_c = self.spec.to_c()
        handle = C.c_void_p()
        with torch.cuda.device(self.device):
            _capi.check(L.marlsc_env_create(C.byref(self._spec_c), self.device.index, C.byref(handle)))
        self._h = handle
        # State layout (include/marlsc_b200.h): "compact" (narrow state, one fused kernel, sparse demand lines) when the
        # configuration qualifies and nothing asks for the general kernels; "wide" otherwise.
        if layout not in (None, "wide", "compact"):
            raise ValueError("layout must be None, 'wide' or 'compact'")
        compact = L.marlsc_env_layout(self._h) == _capi.LAYOUT_COMPACT
        wants_wide = (bool(diagnostics or team_size or generic_kernel or (fused_kernel and layout != "compact"))
                      or self._stock_bound() >= 32768)
        if layout == "compact":
            if wants_wide:
                raise ValueError("layout='compact' excludes diagnostics / team_size / generic_kernel and needs "
                                 "initial stock + episode_length * max order quantity < 32768")
            _capi.check(L.marlsc_env_set_layout(self._h, _capi.LAYOUT_COMPACT))
        elif compact and (layout == "wide" or wants_wide):
            _capi.check(L.marlsc_env_set_layout(self._h, _capi.LAYOUT_WIDE))
        self.layout = "compact" if L.marlsc_env_layout(self._h) == _capi.LAYOUT_COMPACT else "wide"
        if team_size:
            _capi.check(L.marlsc_env_set_team_size(self._h, team_size))
        if generic_kernel:      # tests: bypass the lean instantiation of the step kernel
            _capi.check(L.marlsc_env_set_generic(self._h, 1))
        if fused_kernel:        # comparisons: keep lean launches in the single fused kernel instead of the split step
            _capi.check(L.marlsc_env_set_fused(self._h, 1))
        self.obs_dim = int(L.marlsc_env_obs_dim(self._h))            # local_obs_dim of the reference
        self.global_obs_dim = self.n_warehouses * self.obs_dim

        E, W, S, D, dev = self.num_envs, self.n_warehouses, self.n_skus, self.ring_depth, self.device
        if self.layout == "compact":
            # uint16 stock / history (int16 storage: values stay below 32768, see _stock_bound), uint8 ring indexed by
            # arrival time: ring_qty[e, w, a % L, s] holds the order arriving at step a
            Lm = self.max_expected_lead_time
            self.inventory = torch.zeros((E, W, S), dtype=torch.int16, device=dev)
            self.ring_qty = torch.zeros((E, W, Lm, S), dtype=torch.uint8, device=dev)
            self.ring_lead = None
            self.demand_hist = (torch.zeros((E, 5, W, S), dtype=torch.int16, device=dev)
                                if L.marlsc_env_needs_history(self._h) else None)
            self.forecast = None
        else:
            self.inventory = torch.zeros((E, W, S), dtype=torch.int32, device=dev)
            self.ring_qty = torch.zeros((E, D, W, S), dtype=torch.int32, device=dev)
            self.ring_lead = torch.zeros((E, D, W, S), dtype=torch.uint8, device=dev) if self.stochastic_lead else None
            self.demand_hist = (torch.zeros((E, 5, W, S), dtype=torch.int32, device=dev)
                                if L.marlsc_env_needs_history(self._h) else None)
            self.forecast = torch.zeros((E, W, S), dtype=torch.float32, device=dev) if L.marlsc_env_needs_forecast(self._h) else None
        self._state = _capi.EnvStateC(E, _ptr(self.inventory), _ptr(self.ring_qty), _ptr(self.ring_lead),
                                      _ptr(self.demand_hist), _ptr(self.forecast),
                                      _capi.LAYOUT_COMPACT if self.layout == "compact" else _capi.LAYOUT_WIDE)
        self.obs = torch.zeros((E, W, self.obs_dim), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((E, W), dtype=torch.float32, device=dev)
        self.truncated = torch.zeros((E,), dtype=torch.uint8, device=dev)
        self._empty_orders = DeviceOrders(torch.zeros(E + 1, dtype=torch.int32, device=dev),
                                          torch.zeros(1, dtype=torch.int16, device=dev),
                                          torch.zeros(16, dtype=torch.uint8, device=dev), 0)
        self.diag: Dict[str, torch.Tensor] = {}
        if diagnostics or (episode_metrics and self.layout == "wide"):    # a wide handle folds its metrics from these
            R = self.n_regions
            self.diag = dict(
                cost_breakdown=torch.zeros((E, W, 4), dtype=torch.float32, device=dev),
                ordered=torch.zeros((E, W, S), dtype=torch.int32, device=dev),
                ship_by_sku=torch.zeros((E, W, R, S), dtype=torch.int32, device=dev),
                ship_counts=torch.zeros((E, W, R), dtype=torch.int32, device=dev),
                unfulfilled=torch.zeros((E, R, S), dtype=torch.int32, device=dev),
                lost_orders=torch.zeros((E, R), dtype=torch.int32, device=dev),
                lost_sales=torch.zeros((E, W, S), dtype=torch.float32, device=dev))
        # per-episode accumulators (marlsc_env_set_metrics): zeroed by reset, added to by every step
        self._metrics: Dict[str, torch.Tensor] = {}
        if episode_metrics:
            self._metrics = {k: torch.zeros((E, W), dtype=torch.float64, device=dev) for k in METRICS_PER_ROW}
            self._metrics.update({k: torch.zeros(E, dtype=torch.float64, device=dev) for k in METRICS_PER_ENV})
            self._metrics_c = _capi.EpisodeMetricsC(*[self._metrics[k].data_ptr() for k in METRICS_PER_ROW + METRICS_PER_ENV])
            _capi.check(L.marlsc_env_set_metrics(self._h, C.byref(self._metrics_c)))
        self.timestep = 0
        self._seed, self._episode = seed, 0  # reproducible device-side initial stock (see _initial_inventory)
        self._frame = None                   # empirical demand: the packed frame on the device (marlsc_b200.data)
        self._frame_start = None             # ... and every environment's window start for the running episode
        self._empirical = env_config.components.demand_sampler.type == "empirical"
        self._dd = None                      # device demand sampler state (enable_device_demand)
        self._dl = None                      # device lead-time sampler state (enable_device_leads)
        self._demand_step = 0
        if device_demand:
            self.enable_device_demand(demand_seed, max_orders_per_env)

        # host-side seeding / sampling that replays the reference's NumPy streams (optional)
        self.seed_managers: List[SeedManager] = []
        self.demand_samplers: List[Any] = []
        self.lead_time_samplers: List[Any] = []
        self._host_samplers = host_samplers
        if host_samplers:
            from ..registry import get_demand_sampler, get_lead_time_sampler
            if env_seeds is None:
                env_seeds = [None if seed is None else SeedManager.derive_env_seed(seed, 0, i) for i in range(E)]
            if len(env_seeds) != E:
                raise ValueError("env_seeds must have one entry per environment")
            self._seeded_at_construction = all(sd is not None for sd in env_seeds)
            for sd in env_seeds:
                self.seed_managers.append(SeedManager(root_seed=sd, seed_registry=ENVIRONMENT_SEEDS))
                self.demand_samplers.append(get_demand_sampler(env_config, context=self.spec.context))
                self.lead_time_samplers.append(get_lead_time_sampler(env_config, context=self.spec.context))

    # ------------------------------------------------------------------ on-device demand (K4)
    def enable_device_demand(self, seed: int = 0, max_orders_per_env: Optional[int] = None) -> None:
        """Draw demand on the device with the distribution of the reference's PoissonDemandSampler
        (components/demand_sampler.py:105-163): Poisson order counts and quantities by exact inversion at every rate,
        SKU inclusion with probability p (to within 2^-33). The stream is Philox keyed by (seed, env, step):
        reproducible, but not the reference's NumPy stream - use host samplers or replay when trajectories must match."""
        smp = self.spec.components["demand_sampler"]
        if not hasattr(smp, "dense_params"):
            raise ValueError("device demand needs the 'poisson' demand sampler")
        lam_o, prob, lam_q = smp.dense_params()
        total = float(lam_o.sum())
        omax = max_orders_per_env or int(np.ceil(total + 6.0 * np.sqrt(max(total, 1.0)) + 8.0))
        omax = (omax + 3) & ~3
        L = _capi.lib()
        h = C.c_void_p()
        dbl = lambda a: np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
        keep = (np.ascontiguousarray(lam_o, np.float64), np.ascontiguousarray(prob, np.float64), np.ascontiguousarray(lam_q, np.float64))
        with torch.cuda.device(self.device):
            _capi.check(L.marlsc_demand_create(self.n_regions, self.n_skus, dbl(keep[0]), dbl(keep[1]), dbl(keep[2]),
                                               self.device.index, C.byref(h)))
        E, S, dev = self.num_envs, self.n_skus, self.device
        self._dd = dict(handle=h, seed=int(seed), omax=omax, overflow=torch.zeros(1, dtype=torch.int32, device=dev))
        if self.layout == "compact":
            # the sampler writes sparse lines, the compact kernels' native demand format: a stream holds the cells of four
            # SKUs of every order, mean lam_orders * p * 4 per step, whole round pairs
            # (compound Poisson: Poisson(lam_orders) orders, Binomial(4, p) cells each); ten sigma and some slack on top
            per_stream = float((lam_o * prob).sum()) * 4.0
            var = float((lam_o * (4.0 * prob * (1.0 - prob) + 16.0 * prob * prob)).sum())
            stride = (int(np.ceil(per_stream + 10.0 * np.sqrt(max(var, 1.0)) + 10.0)) + 1) & ~1   # + 2 entries: the lane's SKU map
            rm = self.spec.tables["region_map"]
            # two buffers so that the sampler can draw step t+1 on a side stream while the kernels of step t run
            # (``_dd["overlap"] = True``). Measured at the large config: 3.63 ms per step against 3.67 ms in sequence - both
            # launches fill the machine and both are bound by instruction issue - so it is off by default.
            self._dd.update(lines=[torch.zeros((E * stride, 32), dtype=torch.int16, device=dev) for _ in range(2)], stride=stride,
                            counts=[torch.zeros(E, dtype=torch.int32, device=dev) for _ in range(2)],
                            region_map=None if rm is None else torch.from_numpy(np.ascontiguousarray(rm, np.int32)).to(dev),
                            side=torch.cuda.Stream(device=dev), ready=[torch.cuda.Event(), torch.cuda.Event()],
                            free=[torch.cuda.Event(), torch.cuda.Event()], drawn=-1, overlap=False)
        else:
            self._dd.update(counts=torch.zeros(E, dtype=torch.int32, device=dev),
                            region=torch.zeros(E * omax, dtype=torch.int16, device=dev),
                            qty=torch.zeros(E * omax * S + 16, dtype=torch.uint8, device=dev))

    def _draw_lines(self, step_index: int, stream: int) -> None:
        d = self._dd
        b = step_index & 1
        _capi.check(_capi.lib().marlsc_demand_sample_lines(d["handle"], self.num_envs, d["seed"], step_index, d["stride"],
                                                           _ptr(d["region_map"]), d["lines"][b].data_ptr(), d["counts"][b].data_ptr(),
                                                           d["overflow"].data_ptr(), stream))
        d["drawn"] = step_index

    def sample_device_demand(self) -> None:
        """Fill the device order buffers for the next step (called by step() when no orders are passed). Compact layout: the
        draw for step t normally already ran on the side stream, overlapped with the kernels of step t-1."""
        d = self._dd
        if "lines" in d:
            b = self._demand_step & 1
            cur = torch.cuda.current_stream(self.device)
            if d["drawn"] == self._demand_step:
                cur.wait_event(d["ready"][b])
            else:
                self._draw_lines(self._demand_step, cur.cuda_stream)
        else:
            _capi.check(_capi.lib().marlsc_demand_sample(d["handle"], self.num_envs, d["seed"], self._demand_step, d["omax"],
                                                         d["counts"].data_ptr(), d["region"].data_ptr(), d["qty"].data_ptr(),
                                                         d["overflow"].data_ptr(), self._stream()))
        self._demand_step += 1

    def _prefetch_device_demand(self) -> None:
        """After the step that consumed buffer b was queued: draw the next step's lines into the other buffer on the side
        stream (it was freed by the step before this one)."""
        d = self._dd
        if "lines" not in d or not d["overlap"]:
            return
        cur = torch.cuda.current_stream(self.device)
        used = (self._demand_step - 1) & 1
        d["free"][used].record(cur)
        nxt = self._demand_step & 1
        d["side"].wait_event(d["free"][nxt])
        self._draw_lines(self._demand_step, d["side"].cuda_stream)
        d["ready"][nxt].record(d["side"])

    def enable_device_leads(self, seed: int = 0) -> None:
        """Draw the actual lead times of every step on the device with the distribution of the reference's
        StochasticLeadTimeSampler (components/lead_time_sampler.py:169-197): expected + U{-d..+d} per cell,
        clipped to >= 1. Philox stream keyed by (seed, cell, step), not the reference's NumPy stream."""
        if not self.stochastic_lead:
            raise ValueError("device lead times need the 'stochastic' lead-time sampler")
        smp = self.spec.components["lead_time_sampler"]
        md = np.broadcast_to(np.asarray(smp.max_deviation, dtype=np.int32), (self.n_skus,))
        dev = self.device
        self._dl = dict(seed=int(seed), step=0,
                        expected=torch.from_numpy(np.ascontiguousarray(self.expected_lead_times, dtype=np.int32)).to(dev),
                        max_dev=torch.from_numpy(np.array(md, dtype=np.int32)).to(dev),
                        actual=torch.zeros((self.num_envs, self.n_warehouses, self.n_skus), dtype=torch.uint8, device=dev))

    def sample_device_leads(self) -> torch.Tensor:
        """Actual lead times [E,W,S] (uint8) of the next step (called by step() when none are passed)."""
        d = self._dl
        _capi.check(_capi.lib().marlsc_lead_sample(self.num_envs, self.n_warehouses, self.n_skus, d["expected"].data_ptr(),
                                                   d["max_dev"].data_ptr(), d["seed"], d["step"], d["actual"].data_ptr(),
                                                   self._stream()))
        d["step"] += 1
        return d["actual"]

    def lines_from_orders(self, orders: DeviceOrders, stride: int = 128) -> DeviceLines:
        """Dense device orders -> sparse lines on the device (``marlsc_lines_from_orders``), compacted to the CSR form.
        For pre-converting replayed demand once; ``step`` also accepts dense orders and converts them per call."""
        if self.layout != "compact":
            raise ValueError("demand lines need the compact layout")
        E, dev = self.num_envs, self.device
        padded = torch.empty((E, stride, 32), dtype=torch.int16, device=dev)
        counts = torch.empty(E, dtype=torch.int32, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        io = _capi.StepIOC()
        io.order_offsets, io.order_region, io.order_qty = orders.offsets.data_ptr(), orders.region.data_ptr(), orders.qty.data_ptr()
        io.order_qty_bytes = orders.qty_bytes
        _capi.check(_capi.lib().marlsc_lines_from_orders(self._h, E, C.byref(io), stride, padded.data_ptr(), counts.data_ptr(),
                                                         flag.data_ptr(), self._stream()))
        if int(flag.item()):
            raise ValueError(f"a line stream needs more than {stride} rounds; raise stride")
        offsets = torch.zeros(E + 1, dtype=torch.int32, device=dev)
        offsets[1:] = counts.cumsum(0)
        keep = torch.arange(stride, device=dev)[None, :] < counts[:, None]
        lines = padded[keep]                                           # [n_rounds, 32]
        n_rounds = int(offsets[-1].item())
        if n_rounds == 0:
            lines = torch.zeros((1, 32), dtype=torch.int16, device=dev)
        n_lines = int((lines != 0).sum().item()) - 64 * int((counts > 0).sum().item())     # minus the SKU-map entries
        return DeviceLines(offsets, lines.contiguous(), n_lines, n_rounds)

    def demand_overflowed(self) -> bool:
        """True when some environment drew more orders than max_orders_per_env (the surplus was dropped)."""
        return bool(self._dd is not None and int(self._dd["overflow"].item()) != 0)

    # ------------------------------------------------------------------ per-episode metrics
    @property
    def has_episode_metrics(self) -> bool:
        return bool(self._metrics)

    def episode_metrics(self) -> Dict[str, torch.Tensor]:
        """What the steps since the last reset added up to (reference: collect_step_info, multi_env.py:330-362, summed over
        the episode), float64 on the device: ``holding_cost``, ``penalty_cost``, ``outbound_cost``, ``inbound_cost``
        (unscaled), ``ordered_units``, ``shipped_units``, ``episode_return`` and ``total_cost`` per warehouse [E,W];
        ``demand_units``, ``lost_units`` and the unit ``fill_rate`` (1 where nothing was demanded) per environment [E].
        The accumulators themselves, not copies: the next step or reset changes them. Needs ``episode_metrics=True``."""
        if not self._metrics:
            raise ValueError("construct the environment with episode_metrics=True")
        m = dict(self._metrics)
        m["total_cost"] = sum(m[k] for k in COST_METRICS)
        m["fill_rate"] = fill_rate(m["demand_units"], m["lost_units"])
        return m

    # ------------------------------------------------------------------ heuristic policies (K5)
    def base_stock_actions(self, level: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Actions of the reference's base-stock heuristic (run_baselines.py:133-207) for every environment:
        order up to ``level[w,s]`` given on-hand stock and units in transit, clipped to the order maximum."""
        E, W, S = self.num_envs, self.n_warehouses, self.n_skus
        lvl = level.to(device=self.device, dtype=torch.float32).contiguous()
        if lvl.shape not in ((W, S), (E, W, S)):
            raise ValueError(f"level must have shape {(W, S)} (shared) or {(E, W, S)} (one per environment)")
        act = torch.empty((E, W, S), device=self.device) if out is None else out
        fn = _capi.lib().marlsc_policy_base_stock if lvl.dim() == 2 else _capi.lib().marlsc_policy_base_stock_per_env
        _capi.check(fn(self._h, C.byref(self._state), lvl.data_ptr(), self.timestep, act.data_ptr(), self._stream()))
        self._keep_level = lvl
        return act

    # ------------------------------------------------------------------ helpers
    def _stock_bound(self) -> int:
        """Upper bound of on-hand stock over an episode: initial stock + one maximal order per step (nothing else adds
        stock, multi_env.py:903-919); the compact layout keeps stock in 16 bits."""
        ic = self.env_config.initial_inventory
        if isinstance(ic, InitialInventoryUniform):
            init = int(ic.params["max"])
        elif isinstance(ic, InitialInventoryCustom):
            init = int(np.max(np.asarray(ic.params["values"])))
        else:
            init = 0
        a = self.env_config.action_space
        if a.type != "direct":
            return 1 << 30
        return init + self.episode_length * int(np.max(np.asarray(a.params.max_order_quantities)))

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def close(self):
        if getattr(self, "_dd", None):
            _capi.lib().marlsc_demand_destroy(self._dd["handle"])
            self._dd = None
        if getattr(self, "_h", None):
            _capi.lib().marlsc_env_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def team_size(self) -> int:
        return int(_capi.lib().marlsc_env_team_size(self._h))

    def set_timing(self, on: bool) -> None:
        """Measurement aid: record CUDA events around every kernel a step launches (marlsc_env_set_timing)."""
        _capi.check(_capi.lib().marlsc_env_set_timing(self._h, int(on)))

    def last_step_timing(self) -> list:
        """Per-launch milliseconds of the last timed step: [place, allocate, features, rewards] for the split
        step, one entry for the fused kernel. Waits for that step."""
        buf = (C.c_float * 8)()
        n = _capi.lib().marlsc_env_last_timing(self._h, buf, 8)
        if n < 0:
            _capi.check(n)
        return [float(buf[i]) for i in range(n)]

    def _compute_local_obs_dim(self) -> int:
        return self.obs_dim

    def agent_observations(self, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[E,W,(1+W)*obs_dim]: the reference's per-agent vector ``[local_i | local_0..local_{W-1}]``
        (multi_env.py:560-573). Materialises W copies of the global state - use only for compatibility."""
        o = self.obs if obs is None else obs
        E, W, D = o.shape
        return torch.cat([o, o.reshape(E, 1, W * D).expand(E, W, W * D)], dim=2)

    def global_state(self, obs: Optional[torch.Tensor] = None) -> torch.Tensor:
        o = self.obs if obs is None else obs
        return o.reshape(o.shape[0], -1)

    def pending_matrix(self) -> torch.Tensor:
        """Units in transit per (env, warehouse, SKU) (reference ``_compute_pending_matrix``)."""
        if self.layout == "compact":      # every plane of the arrival-indexed ring is an order still on its way
            return self.ring_qty.sum(dim=2, dtype=torch.int32).to(torch.float32)
        t = self.timestep
        D = self.ring_depth
        tau = torch.tensor([t - 1 - ((t - 1 - d) % D) for d in range(D)], device=self.device).view(1, D, 1, 1)
        if self.stochastic_lead:
            lead = self.ring_lead.to(torch.int64)
        else:
            lead = torch.from_numpy(self.expected_lead_times).to(self.device).view(1, 1, *self.expected_lead_times.shape).to(torch.int64)
        live = (tau >= 0) & (self.ring_qty > 0) & (tau + lead >= t)
        return (self.ring_qty * live).sum(dim=1).to(torch.float32)

    # ------------------------------------------------------------------ reset
    def _initial_inventory(self) -> Tuple[torch.Tensor, int]:
        """(int32 device tensor, per_env flag) following multi_env.py:504-539."""
        W, S = self.n_warehouses, self.n_skus
        ic = self.env_config.initial_inventory
        if isinstance(ic, InitialInventoryUniform):
            lo, hi = ic.params["min"], ic.params["max"]
            if self._host_samplers:
                vals = np.stack([sm.get_rng("inventory").integers(lo, hi + 1, size=(W, S)) for sm in self.seed_managers])
                return torch.from_numpy(vals.astype(np.int32)).to(self.device), 1
            # no host samplers: a device generator keyed by (env seed, episode) so that resets are reproducible
            # (the reference draws from the seeded "inventory" stream on every reset, multi_env.py:504-520)
            g = torch.Generator(device=self.device)
            g.manual_seed((int(self._seed or 0) * 1000003 + self._episode) & 0x7fffffffffffffff)
            return torch.randint(lo, hi + 1, (self.num_envs, W, S), dtype=torch.int32, device=self.device, generator=g), 1
        if isinstance(ic, InitialInventoryCustom):
            v = ic.params["values"]
            arr = np.full((W, S), v, dtype=np.int32) if isinstance(v, int) else np.array(v, dtype=np.int32)
            return torch.from_numpy(arr).to(self.device), 0
        assert isinstance(ic, InitialInventoryZero)
        return torch.zeros((W, S), dtype=torch.int32, device=self.device), 0

    def reset(self, seed: Optional[int] = None, init_inventory: Optional[torch.Tensor] = None,
              obs_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if self._host_samplers:
            for i, sm in enumerate(self.seed_managers):   # multi_env.py:218-231
                if self._seeded_at_construction:
                    if self._num_eval_episodes is not None and (seed is not None or sm._episode_counter >= self._num_eval_episodes):
                        sm._episode_counter = 0
                    sm.advance_episode()
                elif seed is not None:
                    sm.update_root_seed(SeedManager.derive_env_seed(seed, 0, i))
                else:
                    sm.advance_episode()
                for name, comp in (("demand_sampler", self.demand_samplers[i]), ("lead_time_sampler", self.lead_time_samplers[i])):
                    comp.reset(rng=sm.get_rng(name))
        self._episode += 1
        self._frame_start = None
        if init_inventory is None:
            init, per_env = self._initial_inventory()
        else:
            init = init_inventory.to(device=self.device, dtype=torch.int32).contiguous()
            if init.shape == (self.num_envs, self.n_warehouses, self.n_skus):
                per_env = 1
            elif init.shape == (self.n_warehouses, self.n_skus):
                per_env = 0
            else:
                raise ValueError(f"init_inventory must be [E,W,S] or [W,S], got {tuple(init.shape)}")
            if self.layout == "compact" and int(init.max()) + self._stock_bound() >= 32768:
                raise ValueError("init_inventory too large for the compact layout (16-bit stock); construct with layout='wide'")
        out = self._check_obs_out(obs_out)
        _capi.check(_capi.lib().marlsc_env_reset(self._h, C.byref(self._state), init.data_ptr(), per_env, out.data_ptr(), self._stream()))
        self._keep = init
        self.timestep = 0
        return out

    def _check_obs_out(self, obs_out: Optional[torch.Tensor]) -> torch.Tensor:
        if obs_out is None:
            return self.obs
        if (obs_out.shape != self.obs.shape or obs_out.dtype != torch.float32 or obs_out.device != self.device
                or not obs_out.is_contiguous()):
            raise ValueError(f"obs_out must be a contiguous float32 tensor of shape {tuple(self.obs.shape)} on {self.device}")
        return obs_out

    # ------------------------------------------------------------------ step
    def frame_orders(self) -> DeviceOrders:
        """This step's orders of every environment from the empirical demand frame (reference
        components/demand_sampler.py:214-261), sliced on the device. With host samplers the window starts are the ones
        their reference-identical NumPy streams draw; without, one device draw per episode."""
        from ..data import DeviceDemandFrame
        if self._frame is None:
            from ..registry import get_demand_sampler
            smp = self.demand_samplers[0] if self.demand_samplers else get_demand_sampler(self.env_config, context=self.spec.context)
            self._frame = DeviceDemandFrame(smp.frame, self.episode_length, self.device)
        if self._frame_start is None:
            if self._host_samplers:
                starts = torch.tensor([smp.start_index() for smp in self.demand_samplers], dtype=torch.int64)
            else:
                g = torch.Generator()
                g.manual_seed((int(self._seed or 0) * 1000003 + 7919 * self._episode) & 0x7fffffffffffffff)
                starts = torch.randint(0, self._frame.max_start() + 1, (self.num_envs,), generator=g)
            self._frame_start = starts.to(self.device)
        offsets, region, qty, n = self._frame.step_orders(self._frame_start, self.timestep)
        if self._frame.qty_bytes == 2:
            qty = qty.view(torch.int16)
        return DeviceOrders(offsets, region, qty, n)

    def sample_host_demand(self) -> Tuple[OrderBatch, Optional[np.ndarray]]:
        """Draw this step's orders (and lead times) from the per-environment host samplers, in the
        reference's call order: lead times first (multi_env.py:866), then demand (:295)."""
        if not self._host_samplers:
            raise RuntimeError("host samplers are disabled for this environment")
        leads = None
        if self.stochastic_lead:
            leads = np.stack([lt.sample() for lt in self.lead_time_samplers]).astype(np.uint8)
        per_env = [ds.sample(self.timestep) for ds in self.demand_samplers]
        return pack_orders(per_env, self.n_skus), leads

    def step(self, actions: Optional[torch.Tensor], orders: Union[DeviceOrders, OrderBatch, DeviceLines, LineBatch, None] = None,
             actual_lead: Union[torch.Tensor, np.ndarray, None] = None, obs_out: Optional[torch.Tensor] = None,
             rewards_out: Optional[torch.Tensor] = None, base_stock_level: Optional[torch.Tensor] = None
             ) -> Tuple[torch.Tensor, torch.Tensor, bool]:
        """Advance every environment by one timestep.

        actions: float32 [E,W,S] in [-1,1] on the device. orders: this step's demand; ``None`` draws
        from the host samplers (reference-identical NumPy streams; slow, meant for parity and the
        single-env adapter). Returns ``(obs [E,W,obs_dim], rewards [E,W], truncated)``; all
        environments truncate together at ``episode_length`` and never terminate (multi_env.py:325-327).
        The returned tensors are reused by the next call unless ``obs_out`` / ``rewards_out`` are given.
        """
        E, W, S = self.num_envs, self.n_warehouses, self.n_skus
        level = None
        if actions is None:
            # the base-stock heuristic evaluated inside the step kernel (compact layout): ``base_stock_level`` [W,S] or [E,W,S]
            if base_stock_level is None:
                raise ValueError("actions is None: pass base_stock_level to let the step evaluate the base-stock heuristic")
            if self.layout != "compact":
                raise ValueError("the in-step base-stock policy needs the compact layout; use base_stock_actions() + step(actions)")
            level = base_stock_level.to(device=self.device, dtype=torch.float32).contiguous()
            if level.shape not in ((W, S), (E, W, S)):
                raise ValueError(f"base_stock_level must have shape {(W, S)} or {(E, W, S)}")
        qty_actions = actions is not None and actions.dtype == torch.uint8
        if actions is not None:
            if qty_actions and self.layout != "compact":
                raise ValueError("uint8 quantity actions need the compact layout")
            if actions.shape != (E, W, S) or (actions.dtype != torch.float32 and not qty_actions) or actions.device != self.device:
                raise ValueError(f"actions must be a float32 (or, compact layout, uint8 quantity) tensor of shape {(E, W, S)} on {self.device}")
            actions = actions.contiguous()
        use_dd = orders is None and self._dd is not None
        if use_dd:
            self.sample_device_demand()
            orders = self._empty_orders
        if self.stochastic_lead and actual_lead is None and self._dl is not None:
            actual_lead = self.sample_device_leads()
        if orders is None and self._empirical:
            orders = self.frame_orders()
            if self.stochastic_lead and actual_lead is None:
                actual_lead = np.stack([lt.sample() for lt in self.lead_time_samplers]).astype(np.uint8)
        if orders is None:
            host_orders, host_leads = self.sample_host_demand()
            orders = host_orders
            if actual_lead is None:
                actual_lead = host_leads
        if isinstance(orders, OrderBatch):
            if self.layout == "compact" and orders.qty_bytes == 1:
                orders = pack_lines(orders, self.spec.tables["region_map"])
            else:
                orders = DeviceOrders.from_host(orders, self.device)
        if isinstance(orders, LineBatch):
            orders = DeviceLines.from_host(orders, self.device)
        lines = orders if isinstance(orders, DeviceLines) else None
        if lines is not None:
            if self.layout != "compact":
                raise ValueError("demand lines need the compact layout")
            if lines.offsets.shape != (E + 1,) or lines.offsets.dtype != torch.int32 or lines.offsets.device != self.device:
                raise ValueError(f"lines.offsets must be int32 [E+1] on {self.device}")
            if lines.lines.device != self.device or lines.lines.numel() < 32 * max(1, lines.n_rounds):
                raise ValueError("lines.lines is smaller than offsets[E] rounds of 32 entries")
            orders = self._empty_orders
        lead_t = None
        if self.stochastic_lead:
            if actual_lead is None:
                raise ValueError("actual_lead [E,W,S] is required with a stochastic lead-time sampler")
            lead_t = (torch.from_numpy(np.ascontiguousarray(actual_lead, dtype=np.uint8)).to(self.device)
                      if isinstance(actual_lead, np.ndarray) else actual_lead.to(device=self.device, dtype=torch.uint8).contiguous())
            if lead_t.shape != (E, W, S):
                raise ValueError(f"actual_lead must have shape {(E, W, S)}")
        if orders.offsets.shape != (E + 1,) or orders.offsets.dtype != torch.int32 or orders.offsets.device != self.device:
            raise ValueError(f"orders.offsets must be int32 [E+1] on {self.device}")
        if lines is None and not use_dd:
            # cheap host-side consistency checks of user-supplied device orders (n_orders is host knowledge)
            if orders.region.device != self.device or orders.qty.device != self.device:
                raise ValueError(f"orders must live on {self.device}")
            need = (orders.n_orders * S * orders.qty_bytes + 3) & ~3      # the kernels read the rows as aligned 32-bit words
            if orders.region.numel() < max(1, orders.n_orders) or orders.qty.numel() * orders.qty.element_size() < need:
                raise ValueError("orders.region / orders.qty are smaller than offsets[E] rows (qty padded to whole 32-bit words)")
        out = self._check_obs_out(obs_out)
        rew = self.rewards if rewards_out is None else rewards_out
        if rew.shape != (E, W) or rew.dtype != torch.float32 or not rew.is_contiguous() or rew.device != self.device:
            raise ValueError(f"rewards_out must be a contiguous float32 [E,W] tensor on {self.device}")
        d = self.diag
        if d:
            for k in ("ship_by_sku", "ship_counts", "unfulfilled", "lost_orders"):
                d[k].zero_()
        io = _capi.StepIOC(
            None if (qty_actions or actions is None) else actions.data_ptr(), orders.offsets.data_ptr(), orders.region.data_ptr(), orders.qty.data_ptr(),
            orders.qty_bytes, _ptr(lead_t), rew.data_ptr(), out.data_ptr(), self.truncated.data_ptr(),
            _ptr(d.get("cost_breakdown")), _ptr(d.get("ordered")), _ptr(d.get("ship_by_sku")), _ptr(d.get("ship_counts")),
            _ptr(d.get("unfulfilled")), _ptr(d.get("lost_orders")), _ptr(d.get("lost_sales")))
        if qty_actions:
            io.action_qty = actions.data_ptr()
        if level is not None:
            io.actions = None
            io.base_stock_level, io.base_stock_per_env = level.data_ptr(), int(level.dim() == 3)
        if lines is not None:
            io.lines, io.line_offsets = lines.lines.data_ptr(), lines.offsets.data_ptr()
        if use_dd:
            dd = self._dd
            if "lines" in dd:
                b = (self._demand_step - 1) & 1
                io.lines, io.line_offsets, io.line_counts, io.line_stride = dd["lines"][b].data_ptr(), None, dd["counts"][b].data_ptr(), dd["stride"]
            else:
                io.order_offsets, io.order_region, io.order_qty, io.order_qty_bytes = None, dd["region"].data_ptr(), dd["qty"].data_ptr(), 1
                io.order_counts, io.order_stride = dd["counts"].data_ptr(), dd["omax"]
        _capi.check(_capi.lib().marlsc_env_step(self._h, C.byref(self._state), C.byref(io), self.timestep, self._stream()))
        if use_dd:
            self._prefetch_device_demand()
        self._keep = (actions, orders, lines, lead_t, level)   # keep inputs alive until the stream has consumed them
        self.timestep += 1
        return out, rew, self.timestep >= self.episode_length


class HostRollout:
    """Rollout segments driven from HOST buffers through ``marlsc_env_rollout_host``: the reference-facing
    way to call the path (NumPy/pinned tensors in, rewards out) with the copies of step i+1 overlapped with
    the kernel of step i. Holds the two device staging sets the C call needs.

    Dense orders + float actions (``run``) work with every layout; the compact layout also takes sparse demand
    lines and integer order quantities (``run_lines``), which is 2.3x fewer bytes over PCIe at the large shape."""

    def __init__(self, env: BatchedInventoryEnv, max_orders_per_step: int = 0, qty_bytes: int = 1, max_rounds_per_step: int = 0):
        self.env = env
        E, W, S, dev = env.num_envs, env.n_warehouses, env.n_skus, env.device
        self.qty_bytes = qty_bytes
        self.max_orders = int(max_orders_per_step)
        self.max_rounds = int(max_rounds_per_step)
        if self.max_rounds and env.layout != "compact":
            raise ValueError("demand lines need the compact layout")
        self.sets = []
        for _ in range(2):
            self.sets.append(dict(
                actions=torch.empty((E, W, S), device=dev), offsets=torch.empty(E + 1, dtype=torch.int32, device=dev),
                region=torch.empty(max(1, self.max_orders), dtype=torch.int16, device=dev),
                qty=torch.empty(max(16, self.max_orders * S * qty_bytes + 16), dtype=torch.uint8, device=dev),
                lead=torch.empty((E, W, S), dtype=torch.uint8, device=dev) if env.stochastic_lead else None,
                obs=torch.empty_like(env.obs),
                lines=torch.empty((max(1, self.max_rounds), 32), dtype=torch.int16, device=dev) if self.max_rounds else None,
                line_offsets=torch.empty(E + 1, dtype=torch.int32, device=dev) if self.max_rounds else None,
                action_qty=torch.empty((E, W, S), dtype=torch.uint8, device=dev) if self.max_rounds else None))
        self._staging = (_capi.StepIOC * 2)()
        for i, st in enumerate(self.sets):
            io = _capi.StepIOC(st["actions"].data_ptr(), st["offsets"].data_ptr(), st["region"].data_ptr(),
                               st["qty"].data_ptr(), qty_bytes, _ptr(st["lead"]), None, st["obs"].data_ptr(),
                               env.truncated.data_ptr(), None, None, None, None, None, None, None)
            io.lines, io.line_offsets, io.action_qty = _ptr(st["lines"]), _ptr(st["line_offsets"]), _ptr(st["action_qty"])
            self._staging[i] = io

    def _call(self, hs, T, rewards_dev) -> torch.Tensor:
        env = self.env
        if env.timestep + T > env.episode_length:
            raise ValueError("segment crosses the end of the episode; reset first")
        _capi.check(_capi.lib().marlsc_env_rollout_host(env._h, C.byref(env._state), self._staging, hs, T, env.timestep,
                                                        rewards_dev.data_ptr(), env._stream()))
        env.timestep += T
        return self.sets[(T - 1) & 1]["obs"]

    def run(self, actions, offsets, regions, qtys, n_orders, rewards_host, rewards_dev, leads=None, obs_host=None) -> torch.Tensor:
        """Each argument is a per-step list of (pinned) host tensors; ``rewards_host`` / ``rewards_dev`` are
        [T,E,W] float32 (pinned host / device); ``obs_host`` an optional per-step list of pinned [E,W,obs_dim] tensors the
        observations are copied back into. Steps the env T times starting at its current timestep and
        returns the observation buffer that holds the last step's observations."""
        T = len(actions)
        if max(n_orders) > self.max_orders:
            raise ValueError("a step has more orders than the staging buffers hold")
        hs = (_capi.HostStepC * T)()
        for i in range(T):
            hs[i] = _capi.HostStepC(actions[i].data_ptr(), offsets[i].data_ptr(), regions[i].data_ptr(), qtys[i].data_ptr(),
                                    int(n_orders[i]), None if leads is None else leads[i].data_ptr(),
                                    rewards_host[i].data_ptr(), None if obs_host is None else obs_host[i].data_ptr())
        return self._call(hs, T, rewards_dev)

    def run_lines(self, actions, line_offsets, lines, n_rounds, rewards_host, rewards_dev, obs_host=None) -> torch.Tensor:
        """Compact layout: ``actions`` is a per-step list of pinned host tensors, float32 [E,W,S] actions or uint8 [E,W,S]
        order quantities; ``line_offsets`` / ``lines`` / ``n_rounds`` the step's demand as packed by
        ``marlsc_b200.demand.pack_lines`` (pinned int32 [E+1], int16/uint16 [n_rounds,32])."""
        T = len(actions)
        if max(n_rounds) > self.max_rounds:
            raise ValueError("a step has more line rounds than the staging buffers hold")
        hs = (_capi.HostStepC * T)()
        for i in range(T):
            h = _capi.HostStepC()
            if actions[i].dtype == torch.uint8:
                h.action_qty = actions[i].data_ptr()
            else:
                h.actions = actions[i].data_ptr()
            h.lines, h.line_offsets, h.n_rounds = lines[i].data_ptr(), line_offsets[i].data_ptr(), int(n_rounds[i])
            h.rewards = rewards_host[i].data_ptr()
            h.obs = None if obs_host is None else obs_host[i].data_ptr()
            hs[i] = h
        return self._call(hs, T, rewards_dev)
