"""Sharding of cells over GPUs and the one collective of the path: basin aggregates.

Cells (catchments / raster pixels) never read each other -- the only cross-cell operations in the
reference are the ``np.sum`` sites of the diagnostic integrals (reference ``bmi_topoflow_glacier.py:567-568``,
``:613-614``, ``:623-624``, ``:1486-1494``) and the driver-side ``* da_m2`` (``examples/run_topoflow_glacier.py:115``).
So every rank owns a contiguous block of cells with no halo, runs the fused kernel on it, and the per-basin,
area-weighted sums ``[T_chunk, n_basin, 3]`` are combined with ONE ``all_reduce(SUM, float64)`` per chunk.
``torch.distributed`` (NCCL over NVLink on GPUs, gloo in the CPU tests) carries it.
"""

from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

__all__ = ["shard_bounds", "shard_sizes", "BasinAggregates", "agg_contributions", "agg_scaling", "basin_sums_host", "dist_info",
           "ShardedMeltEngine"]

AGG_NAMES = ("runoff_m3s", "swe_m3", "iwe_m3")  # sum(M_total*da_m2), sum(h_swe*da_m2), sum(h_iwe*da_m2)


def shard_sizes(n_cells: int, world: int, align: int = 128) -> list[int]:
    """Cells per rank: contiguous blocks, every block but the last a multiple of ``align`` cells.

    The ``align``-cell groups are dealt out as evenly as possible (sizes differ by at most one group), so no rank is
    left without cells while another holds several groups; fewer groups than ranks is an error -- a rank with zero
    cells would sit out the collectives of the others."""
    if world < 1 or n_cells < 0 or align < 1:
        raise ValueError("bad world size / cell count / alignment")
    groups = -(-n_cells // align)
    if n_cells > 0 and groups < world:
        raise ValueError(f"{n_cells} cells are {groups} groups of {align}: too few to give each of {world} ranks a share")
    base, extra = divmod(groups, world)
    sizes = [(base + (1 if r < extra else 0)) * align for r in range(world)]
    over = sum(sizes) - n_cells          # the last group may be partial; with extra < world it may sit mid-list
    for r in range(world - 1, -1, -1):
        if over <= 0:
            break
        cut = min(over, sizes[r])
        sizes[r] -= cut
        over -= cut
    if n_cells > 0 and min(sizes) <= 0:
        raise ValueError(f"sharding {n_cells} cells over {world} ranks leaves a rank without cells")
    return sizes


def shard_bounds(n_cells: int, world: int, rank: int, align: int = 128) -> Tuple[int, int]:
    """Half-open cell range ``[lo, hi)`` owned by ``rank``."""
    sizes = shard_sizes(n_cells, world, align)
    lo = int(np.sum(sizes[:rank]))
    return lo, lo + sizes[rank]


def dist_info() -> Tuple[int, int]:
    """(rank, world) of the default process group, (0, 1) when not initialised."""
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except Exception:  # noqa: BLE001
        pass
    return 0, 1


def agg_contributions(basin_id, n_basin: int):
    """Contributions of one timestep to each basin's exact aggregate: ``(cells, warps)``, int64 ``[n_basin]`` tensors.

    The kernel adds one partial sum per warp of 32 consecutive cells that lie in one basin (``warps``) and one value
    per cell of a warp that straddles basins (``cells``); lanes past the last cell carry the last cell's basin.  Counts
    are exact, so they add over 128-cell aligned shards.  ``basin_id`` is a torch tensor (any device) or None."""
    import torch

    if basin_id is None or basin_id.numel() == 0:
        z = torch.zeros(max(int(n_basin), 0), dtype=torch.int64)
        return z, z.clone()
    b = basin_id.reshape(-1).to(torch.int64)
    n = b.numel()
    if int(b.min()) < 0 or int(b.max()) >= n_basin:
        raise ValueError(f"basin ids must lie in [0, n_basin = {n_basin})")
    w = torch.cat([b, b[-1:].expand((-n) % 32)]).view(-1, 32)
    uniform = (w == w[:, :1]).all(dim=1)
    warps = torch.bincount(w[uniform, 0], minlength=n_basin)
    real = (torch.arange(w.numel(), device=b.device) < n).view(-1, 32)
    cells = torch.bincount(w[~uniform][real[~uniform]], minlength=n_basin)
    return cells, warps


def agg_scaling(da_max: float, cells, warps):
    """``(E0, E1, E2, L)`` of exact aggregates over cells of at most ``da_max`` m2 and the per-basin contribution counts
    ``cells``, ``warps`` of ``agg_contributions`` (summed over all ranks whose words are added).

    E_q bounds a 32-cell partial sum: |partial| < 2^E_q for M_total < 2^-8 m/s and depths < 2^17 m.  A contribution
    adds less than 2^L to the low word, so with C = max over basins of (cells + warps) contributions the low word stays
    below C * 2^L <= 2^62 for L = min(42, 62 - ceil(log2 C)).  The high word gains less than 2^35 per cell (one cell is
    at most 1/32 of the bound of a partial) and less than 2^40 per warp partial; a layout that could take it to 2^63
    has no safe scaling and raises ValueError, as the words would otherwise wrap without notice."""
    e_da = int(np.ceil(np.log2(max(float(da_max), 1e-30) * 32.0)))
    per_basin = [int(c) + int(w) for c, w in zip(cells, warps)]
    n_max = max(per_basin, default=1) or 1
    lo_bits = min(42, 62 - (n_max - 1).bit_length())
    hi_max = max((int(c) * 2**35 + int(w) * 2**40 for c, w in zip(cells, warps)), default=0)
    if lo_bits < 1 or hi_max >= 2**63:
        raise ValueError(f"exact aggregates: {n_max} contributions to one basin and step could overflow the int64 "
                         "words; split the basin or use the floating-point aggregates")
    return e_da - 8, e_da + 17, e_da + 17, lo_bits


def basin_sums_host(values: np.ndarray, da_m2: np.ndarray, basin_id: np.ndarray, n_basin: int) -> np.ndarray:
    """Host statement of one aggregate: ``out[b] = sum(values[i] * da_m2[i] for basin_id[i] == b)``."""
    return np.bincount(basin_id, weights=np.asarray(values, dtype=np.float64) * da_m2, minlength=n_basin)


class BasinAggregates:
    """Per-rank partial sums -> global sums.

    Default: ``buffer`` is the ``[T_chunk, n_basin, 3]`` float64 tensor the kernel accumulates into with
    floating-point atomics; ``reduce`` makes it global (in place) with one ``all_reduce(SUM)``.  Reproducible to
    rounding (~1e-15), not bit for bit: the order of the atomics is not fixed.

    ``exponents=(E0, E1, E2, L)`` (``MeltEngine.agg_exponents()``, which agrees them across ranks with all-reduces --
    every rank must scale with the same exponents; a 3-tuple means L = 42) selects ORDER-INDEPENDENT sums instead: the
    kernel splits every contribution into two fixed-point int64 words and adds them with integer atomics
    (``TFG_OPT_EXACT_AGG``); ``accumulator`` is that int64 tensor (pass it to ``MeltEngine.run(basin_agg=...)`` of an
    engine that scales with the same exponents), ``reduce`` all-reduces the integers -- exactly -- and decodes them into
    ``buffer``.  The result is bit-identical for any GPU count (shards are 128-cell aligned), launch split or
    scheduling order, and lies within C * 2^(E-40-L) of the exact sum of the contributions (C of them, each truncated
    once) plus the rounding of the decode.  Works on CUDA tensors with NCCL and on CPU tensors with gloo.
    """

    def __init__(self, chunk_steps: int, n_basin: int, device=None, group=None, exponents=None):
        import torch

        self.torch = torch
        self.group = group
        self.n_basin = int(n_basin)
        self.chunk_steps = int(chunk_steps)
        self.buffer = torch.zeros(self.chunk_steps, self.n_basin, 3, dtype=torch.float64, device=device)
        self.exponents = None if exponents is None else tuple(int(e) for e in exponents)
        self.accumulator = None
        if self.exponents is not None:
            if len(self.exponents) == 3:
                self.exponents += (42,)
            if len(self.exponents) != 4:
                raise ValueError(f"exponents must be (E0, E1, E2) or (E0, E1, E2, L), got {exponents!r}")
            self.accumulator = torch.zeros(self.chunk_steps * self.n_basin * 3 * 2 + 1, dtype=torch.int64, device=device)
            e = torch.tensor(self.exponents[:3], dtype=torch.float64, device=device)
            self._scale_hi, self._scale_lo = torch.exp2(e - 40.0), torch.exp2(e - 40.0 - self.exponents[3])

    @property
    def target(self):
        """What ``MeltEngine.run(basin_agg=...)`` should accumulate into."""
        return self.buffer if self.accumulator is None else self.accumulator

    @property
    def n_left_out(self) -> int:
        """Exact mode: contributions the kernel left out (non-finite, or beyond 2^E_q); 0 for sane inputs."""
        return 0 if self.accumulator is None else int(self.accumulator[-1].item())

    def zero(self):
        self.buffer.zero_()
        if self.accumulator is not None:
            self.accumulator.zero_()
        return self.target

    def decode(self):
        """int64 {hi, lo} words -> float64 ``buffer`` (value = hi * 2^(E-40) + lo * 2^(E-40-L)); a pure function of
        the integer sums, hence as reproducible as they are."""
        w = self.accumulator[:-1].view(self.chunk_steps, self.n_basin, 3, 2).to(self.torch.float64)
        self.torch.add(w[..., 0] * self._scale_hi, w[..., 1] * self._scale_lo, out=self.buffer)
        return self.buffer

    def reduce(self, async_op: bool = False):
        import torch.distributed as dist

        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1
        if self.accumulator is not None:
            if multi:
                dist.all_reduce(self.accumulator, op=dist.ReduceOp.SUM, group=self.group)
            self.decode()
            return None
        if multi:
            return dist.all_reduce(self.buffer, op=dist.ReduceOp.SUM, group=self.group, async_op=async_op)
        return None

    def basin_area(self, da_m2, basin_id) -> "object":
        """Static per-basin area (all ranks): ``sum(da_m2)`` by basin."""
        import torch.distributed as dist

        torch = self.torch
        area = torch.zeros(self.n_basin, dtype=torch.float64, device=da_m2.device)
        area.index_add_(0, basin_id.to(torch.int64), da_m2.to(torch.float64))
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            dist.all_reduce(area, op=dist.ReduceOp.SUM, group=self.group)
        return area


class ShardedMeltEngine:
    """The ensemble of ALL cells advanced by all ranks of a ``torch.distributed`` group, one shard per GPU.

    The multi-GPU counterpart of ``MeltEngine`` for users of the product API (``bench.py`` uses it too): every rank
    constructs it with the same arguments, keeps the 128-aligned contiguous block ``bounds = shard_bounds(n_total,
    world, rank)`` of the cells on its own GPU, and ``run`` returns the GLOBAL per-basin aggregates -- the only
    quantity that crosses GPUs on this path (reference ``np.sum`` sites ``bmi_topoflow_glacier.py:567-568,
    :1486-1494`` and the driver's ``* da_m2``, ``examples/run_topoflow_glacier.py:115``).  With ``exact=True``
    (default) the sums are order-independent fixed-point accumulators: 1, 2, 4 or 8 GPUs return the same bits.

    ``cells`` is either the mapping of GLOBAL float64 ``[n_total]`` arrays ``MeltEngine`` takes (sliced here), or a
    callable ``(lo, hi) -> mapping`` that produces the shard's arrays (host arrays keyed like ``cells``, or device
    tables keyed like ``tfg_statics`` + ``h0_*``) for grids too large to materialise on every rank; then pass
    ``n_total``.  ``basin_id`` / ``tz_idx`` / ``forcing_index`` are global arrays (or callables ``(lo, hi)``); so is
    ``cell_params``: a mapping of global per-cell parameter arrays (``MeltEngine(cell_params=...)``), sliced here, or a
    callable ``(lo, hi) -> mapping`` of the shard's arrays; ``forcing_adjust`` likewise (``MeltEngine(forcing_adjust=...)``).
    ``forcing_noise`` (``MeltEngine(forcing_noise=...)``) takes a global per-cell ``stream``, sliced here; without one
    every cell is its own stream with its GLOBAL cell index as id, so that the ranks together equal one engine.
    Attribute access falls through to the local ``MeltEngine`` (``state``, ``row``, ``step_index`` ...).
    """

    def __init__(self, cells, consts, start_time, *, n_total: Optional[int] = None, basin_id=None, n_basin: int = 0,
                 tz_idx=None, forcing_index=None, cell_params=None, forcing_adjust=None, forcing_noise=None, group=None,
                 exact: bool = True,
                 device: Optional[int] = None, **kw):
        import os

        import torch

        from .engine import MeltEngine

        self.group = group
        try:
            import torch.distributed as dist

            on = dist.is_available() and dist.is_initialized()
            self.rank, self.world = (dist.get_rank(group), dist.get_world_size(group)) if on else (0, 1)
        except ImportError:
            self.rank, self.world = 0, 1
        if callable(cells):
            if n_total is None:
                raise ValueError("n_total is required when cells is a factory")
        else:
            n_total = int(np.size(cells["lat"]))
        self.n_total = int(n_total)
        lo, hi = shard_bounds(self.n_total, self.world, self.rank)
        self.bounds = (lo, hi)
        part = (lambda a: None if a is None else (a(lo, hi) if callable(a) else a[lo:hi]))
        local = cells(lo, hi) if callable(cells) else {k: np.asarray(v)[lo:hi] for k, v in cells.items()}
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", self.rank)) % max(torch.cuda.device_count(), 1)
        if cell_params is not None:
            cell_params = cell_params(lo, hi) if callable(cell_params) else {k: v[lo:hi] for k, v in cell_params.items()}
        if forcing_adjust is not None:
            forcing_adjust = (forcing_adjust(lo, hi) if callable(forcing_adjust)
                              else {k: v[lo:hi] for k, v in forcing_adjust.items()})
        if forcing_noise is not None:
            forcing_noise = dict(forcing_noise)
            st = forcing_noise.get("stream")
            forcing_noise["stream"] = np.arange(lo, hi, dtype=np.int64) if st is None else st[lo:hi]
        dev_tables = "a_elev" in local
        self.exact = bool(exact)
        self.engine = MeltEngine(None if dev_tables else local, consts, start_time, basin_id=part(basin_id),
                                 n_basin=n_basin, tz_idx=part(tz_idx), forcing_index=part(forcing_index), device=device,
                                 device_statics=local if dev_tables else None, cell_params=cell_params,
                                 forcing_adjust=forcing_adjust, forcing_noise=forcing_noise, **kw)
        self._aggs: dict = {}

    def __getattr__(self, name):
        if name == "engine":
            raise AttributeError(name)
        return getattr(self.engine, name)

    def local(self, global_block):
        """This rank's columns ``[..., lo:hi]`` of a per-cell array or forcing block laid out over ALL cells."""
        lo, hi = self.bounds
        return global_block[..., lo:hi]

    def aggregates(self, n_steps: int) -> BasinAggregates:
        """The (cached) aggregate buffers for launches of ``n_steps`` timesteps."""
        a = self._aggs.get(n_steps)
        if a is None:
            exps = self.engine.agg_exponents() if self.exact else None   # collective: all ranks get here together
            a = self._aggs[n_steps] = BasinAggregates(n_steps, self.engine.n_basin, device=self.engine.device,
                                                      group=self.group, exponents=exps)
        return a

    def run(self, forcing, n_steps: Optional[int] = None, record=None, aggregate: bool = True):
        """Advance the local shard and combine the basin aggregates over all ranks.

        ``forcing`` is this rank's block ``[T, 5, n_local]`` (``[T, 5, n_forcing_cols]`` with a forcing map).
        Returns ``(records, agg)``: the local recorded series and the GLOBAL ``[T, n_basin, 3]`` float64 sums
        (``None`` when the engine has no basins or ``aggregate=False``); the buffer is reused by the next call."""
        T = int(n_steps if n_steps is not None else forcing.shape[0])
        if not aggregate or self.engine.n_basin <= 0 or self.engine.basin_id is None:
            return self.engine.run(forcing, T, record=record), None
        agg = self.aggregates(T)
        rec = self.engine.run(forcing, T, record=record, basin_agg=agg.zero())
        agg.reduce()
        return rec, agg.buffer

    def set_objective(self, quantity, obs=None, obs_step0: int = 0, obs_index=None):
        """``MeltEngine.set_objective`` on every rank.  ``obs`` is the whole ``[T_obs, n_obs_cols]`` block (every rank
        holds it); ``obs_index`` is a GLOBAL per-cell array, sliced here like ``cell_params``.  Without it each cell reads
        its forcing column when a forcing map is bound, else its own global column (``n_obs_cols == n_total``)."""
        lo, hi = self.bounds
        if quantity is not None and obs_index is None and self.engine.forcing_index is None:
            obs_index = np.arange(self.n_total, dtype=np.int32)
        if obs_index is not None:
            obs_index = obs_index[lo:hi]
        self.engine.set_objective(quantity, obs, obs_step0=obs_step0, obs_index=obs_index)

    def scores(self, gather: bool = True) -> dict:
        """The local shard's ``MeltEngine.scores()``; with ``gather`` (a collective: call on all ranks) the scores of all
        ``n_total`` cells on every rank, so that each rank can pick the best candidate per catchment."""
        import torch

        local = self.engine.scores()
        if not gather or self.world == 1:
            return local
        import torch.distributed as dist

        names = list(local)
        block = torch.stack([local[k] for k in names])                      # [K, n_local]
        if dist.get_backend(self.group) == "gloo":
            block = block.cpu()
        sizes = [b - a for a, b in (shard_bounds(self.n_total, self.world, r) for r in range(self.world))]
        pad = torch.full((len(names), max(sizes)), float("nan"), dtype=torch.float64, device=block.device)
        pad[:, :block.shape[1]] = block
        parts = [torch.empty_like(pad) for _ in range(self.world)]
        dist.all_gather(parts, pad, group=self.group)
        full = torch.cat([p[:, :n] for p, n in zip(parts, sizes)], dim=1).to(local[names[0]].device)
        return {k: full[i] for i, k in enumerate(names)}

    def basin_area(self):
        """Global per-basin area ``sum(da_m2)`` (all ranks)."""
        return self.aggregates(1).basin_area(self.engine.static["da_m2"], self.engine.basin_id)

    def close(self):
        self.engine.close()
