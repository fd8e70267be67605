"""Exact basin aggregates (TFG_OPT_EXACT_AGG) word for word against a host replica of the kernel's accumulator, and the
auxiliary kernels -- FIR routing and the forcing conversions -- at shapes that wrap their grid-stride loops.

The replica follows run_kernel (tfg_run.cuh): a contribution is ``(double)value * da``, rounded once; lanes past the
last cell replicate it with area 0; a warp whose 32 lanes share a basin adds one butterfly partial (lanes l and l+16,
then +8, +4, +2, +1), any other warp one contribution per real cell; each contribution is split into
``a = trunc(v * 2^(40-E))`` and ``b = trunc(frac * 2^L)``, or counted as left out when ``!(|s| < 2^40)``.  The words are
accumulated in Python ints, so the replica also shows whether they stay inside int64.  The SASS of every aggregating
instantiation forms the products with DMUL and the butterfly with DADD (no contraction), which the replica models.
"""
from fractions import Fraction

import numpy as np
import pytest

MODES = ("f64", "f64_fast", "f32")
AGG_KEYS = ("M_total", "h_swe", "h_iwe")
U = 2.0 ** -53


# ---- host replica -------------------------------------------------------------------------------------------------
def warp_partial(v):
    """The kernel's butterfly over the last axis (32 lanes): lane l + lane l^16, then ^8, ^4, ^2, ^1.  IEEE addition is
    commutative, so these pairwise sums are the bits lane 0 (8, 16) ends with."""
    x = v[..., :16] + v[..., 16:]
    x = x[..., :8] + x[..., 8:16]
    x = x[..., :4] + x[..., 4:8]
    x = x[..., :2] + x[..., 2:4]
    return x[..., 0] + x[..., 1]


def _int_sums(vals, basins, n_basin):
    """Per-basin sums of int64 values as Python ints (chunks of 2^20: |a| < 2^40, |b| < 2^42 cannot wrap inside one)."""
    out = np.zeros(n_basin, dtype=object)
    for i in range(0, vals.size, 1 << 20):
        part = np.zeros(n_basin, np.int64)
        np.add.at(part, basins[i:i + (1 << 20)], vals[i:i + (1 << 20)])
        out += part.astype(object)
    return out


def warp_layout(basin_id):
    """(lane -> cell, real-lane mask [W, 32], basin per lane [W, 32], uniform-warp mask [W]) as run_kernel sees them."""
    N = basin_id.size
    lanes = np.minimum(np.arange(-(-N // 32) * 32), N - 1)
    real = (np.arange(lanes.size) < N).reshape(-1, 32)
    bw = np.asarray(basin_id)[lanes].reshape(-1, 32)
    return lanes, real, bw, (bw == bw[:, :1]).all(axis=1)


def agg_replica(series, da_m2, basin_id, n_basin, exps):
    """Words ``[T, n_basin, 3, {hi, lo}]`` (Python ints), the left-out count, and per (step, quantity) the basins and
    float64 values of the contributions that were added."""
    E, L = exps[:3], (exps[3] if len(exps) > 3 else 42)
    T = series[0].shape[0]
    lanes, real, bw, uni = warp_layout(basin_id)
    da = np.where(real, np.asarray(da_m2, np.float64)[lanes].reshape(-1, 32), 0.0)   # replica lanes carry area 0
    words = np.zeros((T, n_basin, 3, 2), dtype=object)
    n_left, added = 0, {}
    for t in range(T):
        for q in range(3):
            with np.errstate(invalid="ignore", over="ignore"):
                v = np.asarray(series[q][t], np.float64)[lanes].reshape(-1, 32) * da
                c = np.concatenate([warp_partial(v[uni]), v[~uni][real[~uni]]])
                s = c * 2.0 ** (40 - E[q])
                ok = np.abs(s) < 2.0 ** 40          # NaN compares false: left out, as in agg_add_exact
            b = np.concatenate([bw[uni, 0], bw[~uni][real[~uni]]])
            n_left += int((~ok).sum())
            s, b = s[ok], b[ok]
            a = np.trunc(s)
            lo = np.trunc((s - a) * 2.0 ** L)
            words[t, :, q, 0] += _int_sums(a.astype(np.int64), b, n_basin)
            words[t, :, q, 1] += _int_sums(lo.astype(np.int64), b, n_basin)
            added[t, q] = (b, c[ok])
    return words, n_left, added


def exact_sum(x) -> Fraction:
    """The exact rational sum of float64 values (mantissas summed per binary exponent in Python ints)."""
    x = np.asarray(x, np.float64).ravel()
    m, e = np.frexp(x)
    mi, e = (m * 2.0 ** 53).astype(np.int64), e.astype(np.int64) - 53
    total = Fraction(0)
    for ee in np.unique(e):
        sel = mi[e == ee]
        total += Fraction(sum(int(sel[i:i + 512].sum()) for i in range(0, sel.size, 512))) * Fraction(2) ** int(ee)
    return total


def gamma(n):
    return n * U / (1 - n * U)


def fits_int64(words):
    return all(-2 ** 63 <= int(w) < 2 ** 63 for w in words.ravel())


def check_decoded(decoded, words, added, exps, quantities=(0, 1, 2)):
    """decoded == exact sum of the added contributions within the derived bound: one truncation of at most
    2^(E-40-L) per contribution, plus the decode's roundings (two conversions and one addition)."""
    E, L = exps[:3], (exps[3] if len(exps) > 3 else 42)
    for (t, q), (b, c) in added.items():
        if q not in quantities:
            continue
        for k in range(words.shape[1]):
            sel = b == k
            exact = exact_sum(c[sel])
            H = abs(Fraction(int(words[t, k, q, 0]))) * Fraction(2) ** (E[q] - 40)
            Lo = abs(Fraction(int(words[t, k, q, 1]))) * Fraction(2) ** (E[q] - 40 - L)
            bound = int(sel.sum()) * Fraction(2) ** (E[q] - 40 - L) + Fraction(2.0000001) * Fraction(U) * (H + Lo)
            err = abs(Fraction(float(decoded[t, k, q])) - exact)
            assert err <= bound, (t, k, AGG_KEYS[q], float(err), float(bound), float(err / max(abs(exact), 1)))


# ---- CPU self-checks of the replica --------------------------------------------------------------------------------
def test_exact_sum_is_exact():
    rng = np.random.default_rng(0)
    x = rng.normal(size=3000) * 10.0 ** rng.integers(-300, 300, 3000)
    x[:5] = [5e-324, -5e-324, 0.0, -0.0, 1.7976931348623157e308]
    assert exact_sum(x) == sum(map(Fraction, x))
    assert exact_sum([1e16, 1.0, -1e16]) == 1                      # where float64 summation loses the 1


def test_butterfly_replica_matches_the_kernels_shuffle_code():
    """warp_partial against a lane-by-lane statement of run_kernel's three-quantity butterfly (xor shuffles)."""
    rng = np.random.default_rng(1)
    for _ in range(200):
        v = [rng.normal(size=32) * 10.0 ** rng.integers(-8, 9, 32) for _ in range(3)]
        lane = np.arange(32)
        hi = (lane & 16) != 0
        k0 = np.where(hi, v[2], v[0]).copy()
        k1 = np.where(hi, 0.0, v[1]).copy()
        send0, send1 = np.where(hi, v[0], v[2]), np.where(hi, v[1], 0.0)
        k0 = k0 + send0[lane ^ 16]
        k1 = k1 + send1[lane ^ 16]
        hi2 = (lane & 8) != 0
        k = np.where(hi2, k1, k0)
        k = k + np.where(hi2, k0, k1)[lane ^ 8]
        for m in (4, 2, 1):
            k = k + k[lane ^ m]
        for q, l in enumerate((0, 8, 16)):
            assert k[l].tobytes() == warp_partial(v[q]).tobytes()


def test_fraction_fma_rounds_once():
    a, b, c = 1.0 + 2.0 ** -30, 1.0 - 2.0 ** -30, -1.0
    assert a * b + c == 0.0                                       # two roundings lose it
    assert fma_exact(a, b, c) == -(2.0 ** -60)                    # one rounding keeps it
    assert fma_exact(0.1, 10.0, -1.0) == float(Fraction(0.1) * 10 - 1)


def test_contribution_counts_and_scaling():
    """sharding.agg_contributions == the replica's count; agg_scaling keeps L = 42 for 4096-cell basins (the bench
    raster) and lowers it where one basin collects more than 2^20 contributions."""
    import torch

    from topoflow_glacier_b200.sharding import agg_contributions, agg_scaling

    rng = np.random.default_rng(2)
    for N in (1, 31, 33, 4017, 6000):
        for bid in layouts(N, 9, rng).values():
            _, real, bw, uni = warp_layout(bid)
            want = np.bincount(bw[uni, 0], minlength=9), np.bincount(bw[~uni][real[~uni]], minlength=9)
            cells, warps = agg_contributions(torch.as_tensor(bid), 9)
            assert np.array_equal(warps.numpy(), want[0]) and np.array_equal(cells.numpy(), want[1])
    assert agg_scaling(1e6, np.zeros(4096), np.full(4096, 128))[3] == 42
    assert agg_scaling(1e6, np.array([2 ** 20]), np.array([0]))[3] == 42
    assert agg_scaling(1e6, np.array([2 ** 20 + 1]), np.array([0]))[3] == 41
    assert agg_scaling(1e6, np.array([4_718_743]), np.array([0])) == (17, 42, 42, 39)
    with pytest.raises(ValueError):
        agg_scaling(1e6, np.array([2 ** 28]), np.array([0]))       # high word: 2^28 cells x 2^35 reach 2^63


def test_low_word_overflow_on_the_host():
    """The overflow the scaling prevents, shown with the replica: 4.7 M snow-covered cells of one basin in warps that
    straddle basins push the low word past 2^63 with L = 42, and stay inside int64 with the L agg_scaling picks."""
    import torch

    from topoflow_glacier_b200.sharding import agg_contributions, agg_scaling

    N = 2 ** 23 + 2 ** 20 + 301
    rng = np.random.default_rng(7)
    swe = rng.uniform(0.05, 2.0, N)
    bid = (np.arange(N) % 2).astype(np.int32)
    cells, warps = agg_contributions(torch.as_tensor(bid), 2)
    exps = agg_scaling(1e6, cells.numpy(), warps.numpy())
    zero = np.zeros((1, N))
    for L, ok in ((42, False), (exps[3], True)):
        words, n_left, _ = agg_replica([zero, swe[None], zero], np.full(N, 1e6), bid, 2, exps[:3] + (L,))
        assert n_left == 0 and fits_int64(words) == ok, (L, [int(w) / 2 ** 63 for w in words[0, :, 1, 1]])


def test_decode_scales_the_low_word_by_its_fraction_bits():
    """BasinAggregates decodes hi * 2^(E-40) + lo * 2^(E-40-L); three exponents mean L = 42 (the words of old callers)."""
    import torch

    from topoflow_glacier_b200.sharding import BasinAggregates

    hi, lo = 123456789, -(2 ** 62) + 3 * 2 ** 20
    for exps, L in (((3, 20, -7), 42), ((3, 20, -7, 39), 39)):
        agg = BasinAggregates(1, 1, exponents=exps)
        assert agg.exponents[3] == L
        agg.accumulator[:6] = torch.tensor([hi, lo] * 3)
        got = agg.decode()[0, 0].tolist()
        for q, e in enumerate(exps[:3]):
            exact = Fraction(hi) * Fraction(2) ** (e - 40) + Fraction(lo) * Fraction(2) ** (e - 40 - L)
            assert got[q] == float(exact)      # both words exact in float64 here: one rounding, in the addition
    with pytest.raises(ValueError):
        BasinAggregates(1, 1, exponents=(1, 2))


# ---- layouts --------------------------------------------------------------------------------------------------------
def layouts(N, NB, rng):
    mixed = rng.integers(0, NB, N)
    mixed[N // 4:3 * N // 4] = np.sort(mixed[N // 4:3 * N // 4])
    return {
        "sorted": np.minimum(np.arange(N) // 256, NB - 1),                   # every warp inside one basin
        "random": rng.integers(0, NB, N),                                     # (almost) no warp inside one basin
        "mixed": mixed,
        "alternating": np.arange(N) % 2,
        "tail": (np.arange(N) // 32) % NB,   # uniform warps; the partial tail warp's basin differs from the warp before
    }


N_CELLS, N_BASIN, T_STEPS = 4017, 23, 6          # 4017 cells: not a multiple of 32 or 128


def _cells(N, rng, da_km2):
    swe = rng.uniform(0, 1.5, N)
    iwe = rng.uniform(0, 60, N) * (rng.uniform(size=N) < 0.4)
    return {"da": da_km2, "slope": rng.uniform(0, 120, N), "aspect": rng.uniform(0, 360, N),
            "lon": rng.uniform(-122.1, -121.4, N), "lat": rng.uniform(46.5, 47.1, N), "elev": rng.uniform(1200, 4300, N),
            "h0_snow": swe * 20.0, "h0_ice": iwe * (1000.0 / 917.0), "h0_swe": swe, "h0_iwe": iwe,
            "T_rain_snow": np.zeros(N)}


def _engine(statics, mode, basin_id, n_basin, T):
    from helpers import default_constants
    from topoflow_glacier_b200.engine import MeltEngine

    return MeltEngine(statics, default_constants(), "2013040100", zones=[-8.0], mode=mode,
                      basin_id=np.asarray(basin_id, np.int32), n_basin=n_basin, horizon_steps=T + 1)


def _run_exact(statics, forcing, mode, basin_id, n_basin, exps=None, record=True):
    """One launch with exact aggregates: (accumulator words [T, NB, 3, 2] int64, left-out count, decoded sums,
    recorded series, engine's da_m2, exponents used)."""
    import torch

    from topoflow_glacier_b200.sharding import BasinAggregates

    T = forcing.shape[0]
    eng = _engine(statics, mode, basin_id, n_basin, T)
    if exps is not None:
        eng.set_agg_exponents(exps)
    agg = BasinAggregates(T, n_basin, device=eng.device, exponents=eng.agg_exponents())
    rec = eng.run(torch.as_tensor(forcing).to(eng.device, eng.dtype).contiguous(), record=AGG_KEYS if record else None,
                  basin_agg=agg.zero())
    agg.reduce()
    out = (agg.accumulator[:-1].view(T, n_basin, 3, 2).cpu().numpy(), agg.n_left_out, agg.buffer.cpu().numpy(),
           [rec[k].cpu().numpy() for k in AGG_KEYS] if record else None, eng.static["da_m2"].cpu().numpy(),
           eng.agg_exponents())
    eng.close()
    return out


# ---- GPU: words against the replica ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["sorted", "random", "mixed", "alternating", "tail"])
@pytest.mark.parametrize("mode", MODES)
def test_exact_words_equal_host_replica(mode, layout, cuda_device):
    """The int64 words and the left-out count equal the replica's bit for bit; the decoded sums lie within the derived
    bound of the exact sum of the contributions; the float-atomic path lies within gamma_(n-1) * sum|v| of it."""
    import torch

    import bench

    rng = np.random.default_rng(10 * MODES.index(mode) + len(layout))
    basin_id = layouts(N_CELLS, N_BASIN, rng)[layout].astype(np.int32)
    statics = _cells(N_CELLS, rng, rng.uniform(5e-4, 2e-3, N_CELLS))
    _, forcing = bench.synthetic_host_sample(N_CELLS, T_STEPS, seed=17)
    words, n_left, decoded, series, da_m2, exps = _run_exact(statics, forcing, mode, basin_id, N_BASIN)
    want, want_left, added = agg_replica(series, da_m2, basin_id, N_BASIN, exps)
    assert fits_int64(want)
    assert np.array_equal(words, want.astype(np.int64)) and n_left == want_left == 0
    check_decoded(decoded, want, added, exps)
    if layout == "sorted":
        assert all(len(b) == -(-N_CELLS // 32) for b, _ in added.values())      # one partial per warp
    if layout == "random":
        assert all(len(b) > 0.99 * N_CELLS for b, _ in added.values())

    # float64 atomics: same contributions, added in some order
    eng = _engine(statics, mode, basin_id, N_BASIN, T_STEPS)
    buf = torch.zeros(T_STEPS, N_BASIN, 3, dtype=torch.float64, device=eng.device)
    rec = eng.run(torch.as_tensor(forcing).to(eng.device, eng.dtype).contiguous(), record=AGG_KEYS, basin_agg=buf)
    for q, k in enumerate(AGG_KEYS):
        assert rec[k].cpu().numpy().tobytes() == series[q].tobytes()
    got = buf.cpu().numpy()
    eng.close()
    for (t, q), (b, c) in added.items():
        for k in range(N_BASIN):
            sel = b == k
            n = int(sel.sum())
            exact = exact_sum(c[sel])
            bound = Fraction(gamma(max(n - 1, 0))) * exact_sum(np.abs(c[sel]))
            assert abs(Fraction(float(got[t, k, q])) - exact) <= bound, (t, k, q)


def _cold_dry(T, N):
    f = np.empty((T, 5, N))
    f[:, 0], f[:, 1], f[:, 2], f[:, 3], f[:, 4] = 0.0, -15.0, 80000.0, 1e-3, 2.0
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_exact_left_out_contributions(mode, cuda_device):
    """NaN forcing in one cell of a uniform warp and one of a straddling warp: exactly the replica's contributions are
    left out (one per affected warp partial or cell) and the words of every basin without a cell in those two warps
    equal those of a clean run.
    Contributions at 2^E are counted, those just below are added."""
    import bench

    rng = np.random.default_rng(5)
    basin_id = layouts(N_CELLS, N_BASIN, rng)["mixed"].astype(np.int32)
    statics = _cells(N_CELLS, rng, rng.uniform(5e-4, 2e-3, N_CELLS))
    _, forcing = bench.synthetic_host_sample(N_CELLS, T_STEPS, seed=19)
    _, _, bw, uni = warp_layout(basin_id)
    c_uni = int(np.nonzero(uni)[0][len(np.nonzero(uni)[0]) // 2]) * 32 + 5
    sorted_part = (np.arange(uni.size) > N_CELLS // 4 // 32) & (np.arange(uni.size) < 3 * N_CELLS // 4 // 32)
    c_mix = int(np.nonzero(~uni & sorted_part)[0][0]) * 32 + 3     # a warp across a basin boundary of the sorted part
    bad = forcing.copy()
    bad[2:, 0:2, [c_uni, c_mix]] = np.nan                     # precipitation and temperature missing from step 2 on
    words, n_left, _, series, da_m2, exps = _run_exact(statics, bad, mode, basin_id, N_BASIN)
    want, want_left, _ = agg_replica(series, da_m2, basin_id, N_BASIN, exps)
    assert want_left > 0 and n_left == want_left
    assert np.array_equal(words, want.astype(np.int64))
    clean, n0, _, _, _, _ = _run_exact(statics, forcing, mode, basin_id, N_BASIN)
    assert n0 == 0
    # basins without a cell in the two warps (the fast mode runs a warp with a non-finite input in its strict arithmetic,
    # so the poisoned cells' warp-mates change by rounding there)
    others = np.setdiff1d(np.arange(N_BASIN), bw[[c_uni // 32, c_mix // 32]])
    assert others.size > N_BASIN // 2
    assert np.array_equal(words[:, others], clean[:, others])

    # the boundary of agg_add_exact, both ways: cells of 1 m2 (E1 = 22) holding h_swe = 2^22 (|s| = 2^40: counted),
    # the float below it (added) and 3 * 2^22 (counted), in warps that straddle two basins; cold, dry steps keep them
    N = 256
    cells = _cells(N, rng, np.full(N, 1e-6))
    below = np.nextafter(np.float32(2.0 ** 22), np.float32(0)) if mode == "f32" else np.nextafter(2.0 ** 22, 0)
    cells["h0_swe"][[3, 5, 7]] = [2.0 ** 22, float(below), 3 * 2.0 ** 22]
    bid = (np.arange(N) % 2).astype(np.int32)
    words, n_left, _, series, da_m2, exps = _run_exact(cells, _cold_dry(2, N), mode, bid, 2)
    assert exps[1] == 22 and np.all(da_m2 == 1.0)
    assert np.array_equal(series[1][:, [3, 5, 7]], np.array([[2.0 ** 22, below, 3 * 2.0 ** 22]] * 2, series[1].dtype))
    want, want_left, _ = agg_replica(series, da_m2, bid, 2, exps)
    assert n_left == want_left == 2 * 2                        # two cells at or above 2^E1, two steps
    assert np.array_equal(words, want.astype(np.int64))


@pytest.mark.gpu
def test_exact_aggregates_of_a_large_basin(cuda_device):
    """9.4 M cells alternating between 2 basins (no warp inside one basin): 4.7 M contributions per basin and step.
    With the low word's 42 fraction bits their sum passes 2^63 and the int64 atomics wrap; the decoded h_swe sums
    must nevertheless equal the exact sum within the truncation bound, with words that fit int64."""
    N = 2 ** 23 + 2 ** 20 + 301
    rng = np.random.default_rng(11)
    cells = _cells(N, rng, np.full(N, 1.0))
    cells["h0_swe"] = rng.uniform(0.05, 2.0, N)
    cells["h0_snow"] = cells["h0_swe"] * 20.0
    cells["h0_ice"][:] = 0.0
    cells["h0_iwe"][:] = 0.0
    bid = (np.arange(N) % 2).astype(np.int32)
    words, n_left, decoded, series, da_m2, exps = _run_exact(cells, _cold_dry(2, N), "f64_fast", bid, 2)
    want, want_left, added = agg_replica(series, da_m2, bid, 2, exps)
    check_decoded(decoded, want, added, exps, quantities=(1,))
    assert fits_int64(want), [int(w) / 2 ** 63 for w in want[:, :, 1, 1].ravel()]
    assert n_left == want_left == 0 and np.array_equal(words, want.astype(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_exact_aggregates_of_shards_in_different_binades(mode, cuda_device):
    """Two single-process engines over 128-aligned shards whose largest cell areas straddle 2^20 m2 (own exponents
    differ), pinned to the exponents of one engine over all cells: their words add up to that engine's, bit for bit."""
    import bench

    N, NB, T = 2048, 7, 5
    rng = np.random.default_rng(13)
    da = np.concatenate([rng.uniform(0.5, 0.9, 1024), rng.uniform(0.5, 1.1, 1024)]) * 2.0 ** 20 / 1e6
    da[[100, 1500]] = 0.9 * 2.0 ** 20 / 1e6, 1.1 * 2.0 ** 20 / 1e6
    statics = _cells(N, rng, da)
    basin_id = layouts(N, NB, rng)["mixed"].astype(np.int32)
    _, forcing = bench.synthetic_host_sample(N, T, seed=23)
    whole, n_left, _, _, _, exps = _run_exact(statics, forcing, mode, basin_id, NB, record=False)
    assert n_left == 0
    own = []
    for s in (slice(0, 1024), slice(1024, N)):
        e = _engine({k: v[s] for k, v in statics.items()}, mode, basin_id[s], NB, T)
        own.append(e.agg_exponents())
        e.close()
    assert own[0][1] != own[1][1]                               # the shards' own scalings differ
    total = np.zeros_like(whole)
    for s in (slice(0, 1024), slice(1024, N)):
        part, n_left, _, _, _, _ = _run_exact({k: v[s] for k, v in statics.items()}, forcing[:, :, s], mode,
                                              basin_id[s], NB, exps=exps, record=False)
        assert n_left == 0
        total += part
    assert np.array_equal(total, whole)


@pytest.mark.gpu
def test_pinned_exponents_are_checked(cuda_device):
    rng = np.random.default_rng(3)
    eng = _engine(_cells(256, rng, np.full(256, 1.0)), "f64_fast", np.arange(256) % 2, 2, 2)
    e = eng.agg_exponents()
    assert len(e) == 4
    with pytest.raises(ValueError):
        eng.set_agg_exponents((e[0] - 1,) + e[1:])
    with pytest.raises(ValueError):
        eng.set_agg_exponents(e[:3] + (e[3] + 1,))
    eng.set_agg_exponents((e[0] + 2, e[1], e[2]))                  # larger exponents are fine; 3 values mean L = 42
    assert eng.agg_exponents() == (e[0] + 2, e[1], e[2], 42)
    eng.close()


# ---- FIR routing ---------------------------------------------------------------------------------------------------
def fma_exact(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))      # exact, then rounded once to nearest-even


def fir_replica(x, w):
    """fir_kernel for one series: acc = fma(w[k], x[t-k], acc) for k = 0 .. min(taps - 1, t)."""
    out = np.empty(x.size)
    for t in range(x.size):
        acc = 0.0
        for k in range(min(w.size, t + 1)):
            acc = fma_exact(float(w[k]), float(x[t - k]), acc)
        out[t] = acc
    return out


@pytest.fixture(scope="module")
def small_engine():
    from helpers import load_case, make_engine

    def make(mode):
        return make_engine(load_case("cats288"), mode=mode)

    return make


@pytest.mark.gpu
@pytest.mark.parametrize("taps", ["1", "7", "20", "T", "T+5"])
def test_fir_wraps_grid_stride_loop(taps, small_engine, cuda_device):
    """64 steps x 9001 series = 576 064 outputs (> 303 104 threads, not a multiple of 256), non-uniform weights of
    both signs: bit-exact against the replica on sampled series, and within the derived bound of a float64
    convolution everywhere (both lie within gamma_n * sum|w x| of the exact convolution)."""
    import torch

    T, M = 64, 9001
    n_taps = {"T": T, "T+5": T + 5}.get(taps) or int(taps)
    rng = np.random.default_rng(n_taps)
    x = rng.normal(size=(T, M)) * 10.0 ** rng.integers(-3, 4, (T, M))
    w = rng.normal(size=n_taps)
    eng = small_engine("f64")
    got = eng.route_fir(torch.as_tensor(x), w).cpu().numpy()
    eng.close()
    for j in (0, 1, 4500, 8999, M - 1):
        assert got[:, j].tobytes() == fir_replica(x[:, j], w).tobytes(), j
    ref, mag = np.zeros((T, M)), np.zeros((T, M))
    for k in range(min(n_taps, T)):
        ref[k:] += w[k] * x[:T - k]
        mag[k:] += abs(w[k] * x[:T - k])
    n = np.minimum(np.arange(T) + 1, n_taps)[:, None]
    bound = 2 * gamma(n) / (1 - gamma(n)) * mag + 2 * 5e-324
    assert np.all(np.abs(got - ref) <= bound)


@pytest.mark.gpu
def test_fir_single_step(small_engine, cuda_device):
    import torch

    rng = np.random.default_rng(4)
    x = rng.normal(size=(1, 1000))
    eng = small_engine("f64")
    for taps in (1, 7):
        w = rng.normal(size=taps)
        got = eng.route_fir(torch.as_tensor(x), w).cpu().numpy()
        assert got.tobytes() == (w[0] * x).tobytes()
    eng.close()


# ---- forcing conversion ----------------------------------------------------------------------------------------------
def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes()


T_CONV, N_CONV = 3, 500_003                       # 1 500 009 elements: more than the 1 212 416 threads of the launch


def _raw_block(rng):
    raw = np.stack([rng.exponential(0.4, (T_CONV, N_CONV)), 273.15 + rng.normal(0, 6, (T_CONV, N_CONV)),
                    88900 + rng.normal(0, 300, (T_CONV, N_CONV)), rng.uniform(1e-3, 6e-3, (T_CONV, N_CONV)),
                    rng.normal(0, 3, (T_CONV, N_CONV)), rng.normal(0, 3, (T_CONV, N_CONV))], axis=1)
    edge = [np.nan, np.inf, -np.inf, -0.0, 0.0, 5e-324, 1e-310, 1e-40, 1e39, -1e39, 3.5e38, 1e200, -1e200, 1e300]
    for i, v in enumerate(edge):                      # every edge value in every variable, also at the block's end
        raw[:, :, i] = v
        raw[:, :, N_CONV - 1 - i] = v
    raw[:, 4:6, 20] = 0.0                             # U = V = 0
    raw[:, 4, 21], raw[:, 5, 21] = 1e160, -1e160      # u*u overflows: uz = inf on both sides
    raw[-1, :, N_CONV // 2] = np.nan
    return raw


def _convert(eng, src, packing=None):
    import torch

    from topoflow_glacier_b200 import _lib

    d_src = torch.as_tensor(src).to(eng.device)
    out = torch.empty(T_CONV, 5, N_CONV, dtype=eng.dtype, device=eng.device)
    if packing is None:
        _lib.check(eng.lib.tfg_convert_forcing(eng.ctx, d_src.data_ptr(), d_src.element_size(), out.data_ptr(), T_CONV,
                                               N_CONV, eng.stream_ptr), "tfg_convert_forcing")
    else:
        sc, of = (np.ascontiguousarray(a, dtype=np.float64) for a in packing)
        _lib.check(eng.lib.tfg_convert_forcing_packed(eng.ctx, d_src.data_ptr(), sc.ctypes.data, of.ctypes.data,
                                                      out.data_ptr(), T_CONV, N_CONV, eng.stream_ptr),
                   "tfg_convert_forcing_packed")
    return out.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f32"])
def test_convert_forcing_edges_and_grid_stride(mode, small_engine, cuda_device):
    """tfg_convert_forcing from float64 and float32 sources == convert_on_host bit for bit (cast to the context's
    type), with NaN, +-inf, -0.0, subnormals, U = V = 0, u*u overflowing and float32 outputs that round to inf."""
    from topoflow_glacier_b200.forcing import convert_on_host

    raw = _raw_block(np.random.default_rng(6))
    eng = small_engine(mode)
    dt = np.float32 if mode == "f32" else np.float64
    with np.errstate(over="ignore", invalid="ignore"):
        raw32 = raw.astype(np.float32)
        for src, host in ((raw, raw), (raw32, raw32.astype(np.float64))):
            want = convert_on_host(host).astype(dt)
            assert same_bits(_convert(eng, src), want), src.dtype
    assert np.isinf(want[:, 4, 21]).all()
    if mode == "f32":
        assert np.isinf(want[:, 2, 10]).all()          # 3.5e38 Pa rounds to inf in float32
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["f64", "f32"])
def test_convert_forcing_packed_edges_and_grid_stride(mode, small_engine, cuda_device):
    """tfg_convert_forcing_packed == convert_on_host(unpack_forcing(...)) bit for bit, with -32768, -1, 0 and 32767 in
    every variable, with the default packing and with one whose extremes overflow float32."""
    from topoflow_glacier_b200.forcing import DEFAULT_PACKING, convert_on_host, unpack_forcing

    rng = np.random.default_rng(8)
    packed = rng.integers(-32768, 32768, (T_CONV, 6, N_CONV)).astype(np.int16)
    for i, v in enumerate((-32768, -1, 0, 32767)):
        packed[:, :, i] = v
        packed[:, :, N_CONV - 1 - i] = v
    eng = small_engine(mode)
    dt = np.float32 if mode == "f32" else np.float64
    wide = (np.array([0.005, 0.005, 2e35, 1e-6, 1e150, 0.005]), np.array([163.84, 273.15, 0.0, 0.0325, 0.0, -1e3]))
    for packing in (DEFAULT_PACKING, wide):
        with np.errstate(over="ignore", invalid="ignore"):
            want = convert_on_host(unpack_forcing(packed, packing)).astype(dt)
        assert same_bits(_convert(eng, packed, packing), want)
    eng.close()
