"""The threshold path and the float64 recombinations at the ends of the float32 range and on inf / NaN, against the oracle.

tile_scores_kernel (qa_tile_scores_f32) drives mixed-tile-threshold and the threshold sweep.  Its bf16 kernel rounds groups
with maxima E >= 24 by magic numbers in group units and the others bit by bit, and it takes the bf16 slot of a bf16 tile
from the tile itself.  The float64 recombinations of the tile-stat table (qa_assignment_sums*, qa_random_samples) take the
maximum |x - y| over tiles.  These cases sit on both sides of those paths:
  * denormal-only groups beside a group of normals in the same tile, and whole denormal tile rows;
  * group maxima at the biased exponents E = 1, 23, 24, 25, 76, 190, 191, 253, 254, with one element at the largest bf16
    value (it rounds up to the format's clamp) in every E = 254 group;
  * tiles of values near 2^-100, whose (a - mean)^2 underflows to 0 while |a - y| > 0 (the zero-denominator branch);
  * single elements and whole groups at 2^64, at the largest bf16 value and (float32) at FLT_MAX, so that squares and dot
    products overflow, and tiles of finite values near 2^127 whose sum overflows while |a - y| stays finite;
  * single +inf, -inf and NaN elements and whole groups of them, and -inf among large negative values.
Each pattern is built as bf16-exact data and with 24-bit significands (float32), at 64 x 1024, 45 x 77 and as a 1-D vector
with a ragged last row.  Scores are compared bit for bit and NaN positions must match.
"""
import math

import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc

pytestmark = pytest.mark.gpu

MIXED = list(orc.MIXED_FORMATS)
METRICS = ("pcc", "mae", "atol")
SHAPES = {"vec": (64, 1024), "ragged": (45, 77), "1d": (3000,)}
BOUND_E = (1, 23, 24, 25, 76, 190, 191, 253, 254)
NONFINITE = ["posinf", "neginf", "nan"]
BF16_PATTERNS = ["denorm", "bound", "under", "over_2p64", "over_bf16max", "bigtile"] + NONFINITE
F32_PATTERNS = BF16_PATTERNS + ["over_f32max"]
CASES = [(p, s, False) for p in BF16_PATTERNS for s in SHAPES] + [(p, s, True) for p in F32_PATTERNS for s in SHAPES]
IDS = [f"{p}-{s}-{'f32' if f else 'bf16'}" for p, s, f in CASES]
case_params = pytest.mark.parametrize("pattern,shape,f32", CASES, ids=IDS)


# --------------------------------------------------------------------------------------------------------------------------
# inputs (seeded NumPy)
# --------------------------------------------------------------------------------------------------------------------------
def _f32(bits):
    return np.ascontiguousarray(bits, dtype=np.uint32).view(np.float32)


def _values(rng, shape, e_lo, e_hi, sign=True):
    """bf16-exact values with biased exponents in [e_lo, e_hi] (0 = denormal), random 7-bit significands and signs."""
    e = rng.integers(e_lo, e_hi + 1, shape).astype(np.uint32)
    s = rng.integers(0, 2, shape).astype(np.uint32) << 31 if sign else np.zeros(shape, np.uint32)
    m = rng.integers(0, 128, shape).astype(np.uint32) << 16
    m[(e == 0) & (m == 0)] |= 1 << 16      # a denormal draw is never a zero
    return _f32(s | (e << 23) | m)


def _perturb(x, rng):
    """24-bit significands: low bits below bf16's rounding half-way point on every finite non-zero element (each bf16
    image is unchanged, so the groups keep their exponents)."""
    b = x.view(np.uint32).copy()
    ok = ((b & 0x7FFFFFFF) != 0) & ((b & 0x7F800000) != 0x7F800000)
    b[ok] |= rng.integers(1, 1 << 12, b.shape).astype(np.uint32)[ok]
    return _f32(b)


def _per_tile(x, v, R, C):
    """Per tile, by (tile row + tile column) % 3: one element, a whole 16-element group, or nothing at the value v."""
    for tr in range(-(-R // 32)):
        for tc in range(-(-C // 32)):
            k = (tr + tc) % 3
            if k == 0 and tr * 32 + 3 < R and tc * 32 + 5 < C:
                x[tr * 32 + 3, tc * 32 + 5] = v
            elif k == 1 and tr * 32 + 7 < R:
                x[tr * 32 + 7, tc * 32:tc * 32 + 16] = v


def _pattern(name, R, C, f32, seed):
    rng = np.random.default_rng(seed)
    g = np.arange(C)[None, :] // 16 + np.zeros((R, 1), np.int64)
    r = np.arange(R)[:, None] + np.zeros((1, C), np.int64)
    special = None
    if name == "denorm":                      # denormal-only groups beside normal groups near 2^-124; tile row 0 all denormal
        x = np.where(g % 2 == 0, _values(rng, (R, C), 0, 0), _values(rng, (R, C), 1, 3))
        x = np.where(r < 32, _values(rng, (R, C), 0, 0), x)
    elif name == "bound":                     # per tile one group-maximum exponent E; every group's maximum exactly at E
        tw = -(-C // 32)
        E = np.asarray(BOUND_E)[((r // 32) * tw + np.arange(C)[None, :] // 32) % len(BOUND_E)]
        x = _values(rng, (R, C), 0, 0)
        for e in BOUND_E:
            x = np.where(E == e, _values(rng, (R, C), max(e - 3, 0), e - 1 if e > 1 else e), x)
        lead = np.arange(C)[None, :] % 16 == (g * 7) % 16                 # the element that sets the group's E
        top = _f32((E.astype(np.uint32) << 23) | (rng.integers(0, 128, (R, C)).astype(np.uint32) << 16)
                   | (rng.integers(0, 2, (R, C)).astype(np.uint32) << 31))
        x = np.where(lead, top, x)
        clamp = np.arange(C)[None, :] % 16 == (g * 7 + 3) % 16          # rounds up to the clamp in every format
        special = np.where((E == 254) & clamp, _f32(np.uint32(0x7F7F0000)), np.float32(np.nan))
    elif name == "under":                     # |a - mean| ~ 2^-100: every square underflows, |a - y| > 0 for the BFP formats
        x = _values(rng, (R, C), 25, 28)
    elif name.startswith("over_"):
        v = {"2p64": _f32(np.uint32(0x5F800000)), "bf16max": _f32(np.uint32(0x7F7F0000)),
             "f32max": _f32(np.uint32(0x7F7FFFFF))}[name[5:]][0]
        ev = (int(v.view(np.uint32)) >> 23) & 0xFF
        x = _values(rng, (R, C), ev - 10, ev - 8)
        special = np.full((R, C), np.float32(np.nan))
        _per_tile(special, v, R, C)
    elif name == "bigtile":                   # positive values in [2^126, 2^127.99): every tile's float32 sum overflows
        x = _values(rng, (R, C), 253, 253, sign=False)
    elif name in NONFINITE:
        v = {"posinf": np.float32(np.inf), "neginf": np.float32(-np.inf), "nan": np.float32(np.nan)}[name]
        x = _values(rng, (R, C), 120, 130)
        if name == "neginf":                  # a background of large negative values in every other tile column
            x = np.where((np.arange(C)[None, :] // 32) % 2 == 0, -np.abs(_values(rng, (R, C), 220, 227)), x)
        mark = np.zeros((R, C), np.float32)
        _per_tile(mark, np.float32(1), R, C)
        special = np.where(mark == 1, v, np.float32(np.nan))
        if name == "nan":
            x = np.where(mark == 1, v, x)
            special = None
    else:
        raise KeyError(name)
    x = np.ascontiguousarray(x, dtype=np.float32)
    if f32:
        x = _perturb(x, rng)
    if special is not None:                   # set after the perturbation: these values stay exactly as given
        sel = ~np.isnan(special)
        x = np.where(sel, special, x).astype(np.float32)
    return np.ascontiguousarray(x, dtype=np.float32)


_CACHE = {}


def _case(pattern, shape, f32):
    key = (pattern, shape, f32)
    if key not in _CACHE:
        dims = SHAPES[shape]
        seed = 3000 + 41 * F32_PATTERNS.index(pattern) + 7 * list(SHAPES).index(shape) + int(f32)
        if len(dims) == 1:
            n = dims[0]
            x = _pattern(pattern, -(-n // 32), 32, f32, seed).reshape(-1)[:n].copy()
        else:
            x = _pattern(pattern, dims[0], dims[1], f32, seed)
        with np.errstate(all="ignore"):
            scores = {m: orc.padded_tile_scores(x, MIXED, m) for m in METRICS}
        _CACHE[key] = (x, scores)
    return _CACHE[key]


# --------------------------------------------------------------------------------------------------------------------------
# comparison rules
# --------------------------------------------------------------------------------------------------------------------------
def _same_f32(got, want, tag):
    """Bit-equal float32 values, NaN positions equal (NaN payloads are not compared)."""
    got = np.asarray(got, dtype=np.float32).reshape(-1)
    want = np.asarray(want, dtype=np.float32).reshape(-1)
    assert got.shape == want.shape, tag
    gn, wn = np.isnan(got), np.isnan(want)
    bad = np.nonzero((gn != wn) | (~gn & ~wn & (got.view(np.uint32) != want.view(np.uint32))))[0]
    assert bad.size == 0, (tag, bad[:8].tolist(), got[bad[:8]].tolist(), want[bad[:8]].tolist())


def _close_f64(got, want, tag, rel=1e-9):
    """Same NaN positions, same infinities, relative 1e-9 where finite."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (tag, got, want)
    fin = np.isfinite(want)
    assert np.array_equal(got[~fin & ~np.isnan(want)], want[~fin & ~np.isnan(want)]), (tag, got, want)
    assert np.allclose(got[fin], want[fin], rtol=rel, atol=0), (tag, got, want)


def _exact_f64(got, want, tag):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert np.array_equal(got, want, equal_nan=True), (tag, got, want)


@pytest.fixture(scope="module")
def qa():
    from quantization_analysis_b200 import engine, sweep
    from quantization_analysis_b200 import compression_algorithms as ca
    from quantization_analysis_b200.compression_algorithms import tile_utils
    return {"eng": engine, "sweep": sweep, "ca": ca, "tu": tile_utils}


def test_patterns_are_what_they_claim():
    """The inputs hold what the module docstring lists (checked on the host)."""
    for pattern, shape, f32 in CASES:
        x, _ = _case(pattern, shape, f32)
        low = (x.view(np.uint32) & 0xFFFF) != 0
        assert low.any() == f32, (pattern, shape, f32)
        if pattern in NONFINITE:
            assert (~np.isfinite(x)).any(), pattern
        else:
            assert np.isfinite(x).all(), pattern
    x, _ = _case("bound", "vec", False)
    e = (x.view(np.uint32).reshape(64, 64, 16) >> 23) & 0xFF
    assert set(np.unique(e.max(axis=-1)).tolist()) == set(BOUND_E)
    x, _ = _case("bigtile", "vec", False)
    assert np.isinf(orc.np_pairwise_sum(x[:32, :32].reshape(1, -1))).all()


# --------------------------------------------------------------------------------------------------------------------------
# per-tile scores
# --------------------------------------------------------------------------------------------------------------------------
@case_params
def test_tile_scores(qa, pattern, shape, f32):
    """qa_tile_scores_f32: all 4 formats x 3 metrics against orc.padded_tile_scores."""
    eng = qa["eng"]
    x, want = _case(pattern, shape, f32)
    p = eng.prepare_tiles(x)
    assert p.dtype_code == (1 if f32 else 0), (pattern, shape, f32)
    got = eng.tile_scores(p, MIXED).cpu().numpy()
    for mi, m in enumerate(METRICS):
        for fi, f in enumerate(MIXED):
            _same_f32(got[mi, fi], want[m][f], (pattern, shape, f32, m, f))


@case_params
def test_tile_metrics_pair(qa, pattern, shape, f32):
    """tile_utils.tile_metrics (qa_tile_scores_pair_f32) on the padded tiles and each format's reconstruction, against
    orc.tile_scores_f32."""
    tu = qa["tu"]
    x, _ = _case(pattern, shape, f32)
    pad, _info, _pi = orc.to_padded_2d(x)
    tx = orc.tiles_from_padded(pad)
    for f in MIXED:
        with np.errstate(all="ignore"):
            tq = orc.tiles_from_padded(orc.to_padded_2d(orc.quantize(x, f))[0])
        for m in METRICS:
            with np.errstate(all="ignore"):
                want = orc.tile_scores_f32(tx, tq, m)
            _same_f32(tu.tile_metrics(tx, tq, m), want, (pattern, shape, f32, f, m))


def _thresholds(scores):
    """Per metric a threshold between the formats' per-tile scores (a fixed value where they are all NaN)."""
    out = {"pcc": 0.999}
    for m in ("mae", "atol"):
        v = scores[m]["bfp4"]
        v = v[np.isfinite(v)]
        out[m] = float(np.median(v)) if v.size else 1.0
    return out


@case_params
def test_threshold_algorithm(qa, pattern, shape, f32):
    """mixed-tile-threshold for pcc, mae and atol: map and counts against orc.threshold_assign."""
    ca = qa["ca"]
    x, scores = _case(pattern, shape, f32)
    pad_info = orc.to_padded_2d(x)[2]
    th, tw = pad_info[2] // 32, pad_info[3] // 32
    for m, thr in _thresholds(scores).items():
        res = ca.create_algorithm("mixed-tile-threshold", {"metric": m, "threshold": thr}).run(x, MIXED, None, None)[0]
        a, counts = orc.threshold_assign(scores[m], MIXED, m, thr, th, tw)
        tag = (pattern, shape, f32, m, thr)
        assert np.array_equal(np.asarray(res.meta["assignment"]).reshape(a.shape), a), tag
        assert res.tile_counts == counts, tag


# --------------------------------------------------------------------------------------------------------------------------
# threshold sweep
# --------------------------------------------------------------------------------------------------------------------------
def _lowest(scores, m):
    """A lowest-metric-val on the right side of the sweep's start (the bf16 slot's max / min), so that the sweep runs."""
    if m == "pcc":
        start = float(np.max(scores[m]["bf16"]))
        return start - 0.5 if np.isfinite(start) else 0.5
    start = float(np.min(scores[m]["bf16"]))
    v = scores[m]["bfp2"]
    v = v[np.isfinite(v)]
    top = float(v.max()) if v.size else 0.0
    return max(top, start if np.isfinite(start) else 0.0) + 1.0


@case_params
def test_sweep(qa, pattern, shape, f32):
    """sweep_tensor with default thresholds: the start value (np.max / np.min of the bf16 slot, NaN included), the maps
    against orc.sweep_assign, the rows against orc.wq_scores_restated of the reconstruction and, with scoring="exact",
    atol and mae against orc.exact_metrics_f64.  The exact pcc is deliberately held to the float64 recombination of the
    oracle's table (_metrics_of_map) rather than to orc.exact_metrics_f64: the table sums float32 products, as the
    reference's greedy forms them, so its x*x and x*y overflow and underflow where exact_metrics_f64's float64 products
    do not, and on the overflow and underflow patterns the two pcc values differ by design."""
    sw = qa["sweep"]
    x, scores = _case(pattern, shape, f32)
    steps = 6
    for m in METRICS:
        lowest = _lowest(scores, m)
        tag = (pattern, shape, f32, m)
        rows, maps = sw.sweep_tensor(x, MIXED, m, steps=steps, lowest=lowest)
        start = np.max(scores[m]["bf16"]) if m == "pcc" else np.min(scores[m]["bf16"])
        thr = np.asarray([r["threshold"] for r in rows])
        assert np.array_equal(thr, np.linspace(float(start), lowest, steps), equal_nan=True), (tag, thr, start)
        want_maps = orc.sweep_assign(scores[m], MIXED, m, [float(t) for t in thr])
        maps = maps.cpu().numpy()
        assert np.array_equal(maps, want_maps), tag
        ref, exact = {}, {}
        with np.errstate(all="ignore"):
            tab = _table_arrays(orc.tile_stat_table(x))
        for i in range(steps):
            key = maps[i].tobytes()
            if key not in ref:
                with np.errstate(all="ignore"):
                    y = orc.apply_assignment(x, maps[i])
                    ref[key] = orc.wq_scores_restated(x, y)
                    exact[key] = orc.exact_metrics_f64(x, y)
            for k in METRICS:
                _same_f32(rows[i][k], ref[key][k], (tag, i, k))
        rows_x, _ = sw.sweep_tensor(x, MIXED, m, steps=steps, lowest=lowest, scoring="exact")
        for i in range(steps):
            w = exact[maps[i].tobytes()]
            _exact_f64(rows_x[i]["atol"], w["atol"], (tag, i, "exact atol"))
            _close_f64(rows_x[i]["mae"], w["mae"], (tag, i, "exact mae"))
            # pcc from the table's sums of float32 products (which overflow and underflow like the reference's)
            _close_f64(rows_x[i]["pcc"], _metrics_of_map(tab, maps[i].astype(np.int64), float(x.size))[0], (tag, i, "exact pcc"))


# --------------------------------------------------------------------------------------------------------------------------
# whole-tensor float32 scorer
# --------------------------------------------------------------------------------------------------------------------------
@case_params
def test_tensor_scores(qa, pattern, shape, f32):
    """engine.tensor_scores_f32 of each format's reconstruction against orc.wq_scores_restated: 64 x 1024 takes the
    pipelined path (n >= 16384), the other shapes the short one."""
    eng = qa["eng"]
    x, _ = _case(pattern, shape, f32)
    xd = torch.from_numpy(x.reshape(-1).copy()).cuda()
    if not f32:
        xd = xd.to(torch.bfloat16)
    for f in MIXED:
        with np.errstate(all="ignore"):
            y = orc.quantize(x, f)
            want = orc.wq_scores_restated(x, y)
        got = eng.tensor_scores_f32(xd, torch.from_numpy(y.reshape(-1).copy()).cuda())[0]
        for k, i in (("pcc", 0), ("mae", 1), ("atol", 2)):
            _same_f32(got[i], want[k], (pattern, shape, f32, f, k))


# --------------------------------------------------------------------------------------------------------------------------
# float64 recombinations of the tile-stat table
# --------------------------------------------------------------------------------------------------------------------------
def _table_arrays(want):
    """orc.tile_stat_table -> float64 [22, T] in the library's layout (sx, sx2, then sy, sy2, sxy, sabs, amax per format)."""
    rows = [want["sx"], want["sx2"]]
    for f in MIXED:
        rows += [want[f][k] for k in ("sy", "sy2", "sxy", "sabs", "amax")]
    return np.ascontiguousarray(np.stack(rows, axis=0), dtype=np.float64)


def _metrics_of_map(tab, a, n):
    """pcc / mae / atol of map `a` from the table, as orc.random_samples_exact forms them (fsum, np.max)."""
    ar = np.arange(tab.shape[1])
    col = lambda k: tab[2 + 5 * a + k, ar]            # noqa: E731
    sx, sx2 = math.fsum(tab[0]), math.fsum(tab[1])
    sy, sy2, sxy, sabs = (math.fsum(col(k)) for k in range(4))
    amax = float(col(4).max())
    am2, bm2 = max(sx2 - sx * sx / n, 0.0), max(sy2 - sy * sy / n, 0.0)
    den = math.sqrt(am2 * bm2)
    pcc = (1.0 if amax == 0.0 else 0.0) if den == 0.0 else (sxy - sx * sy / n) / den
    return (pcc, sabs / n, amax)


def _check_metrics(got, want, tag):
    _exact_f64(got[2], want[2], (tag, "atol"))
    _close_f64(got[0], want[0], (tag, "pcc"))
    _close_f64(got[1], want[1], (tag, "mae"))


@case_params
def test_recombinations(qa, pattern, shape, f32):
    """engine.assignment_sums (per format and per map), assignment_sums_batch and random_samples (k = 2 and 4) on the
    oracle's table: atol exactly (NaN included), pcc and mae with the same NaN positions and to 1e-9 where finite.  The
    reference is the table-driven recombination (_metrics_of_map, orc.random_samples_exact), deliberately not
    orc.exact_metrics_f64, for the reason test_sweep gives; feeding the oracle's table isolates these kernels from the
    tile-stat kernels.  The kernels' own table is then held to orc.exact_metrics_f64 per format for atol and mae, which
    involve no products: that is what metrics_exact reports."""
    eng = qa["eng"]
    x, _ = _case(pattern, shape, f32)
    with np.errstate(all="ignore"):
        want = orc.tile_stat_table(x)
        tab = _table_arrays(want)
        n = float(x.size)
        td = torch.from_numpy(tab).cuda()
        nt = tab.shape[1]
        rng = np.random.default_rng(len(pattern) + nt)
        maps = [np.full(nt, fi, np.int8) for fi in range(4)] + [rng.integers(0, 4, nt).astype(np.int8) for _ in range(3)]
        wants = [_metrics_of_map(tab, a.astype(np.int64), n) for a in maps]
        tag = (pattern, shape, f32)
        for fi in range(4):
            s = eng.assignment_sums(td, fmt=fi).cpu().numpy()
            m = eng.metrics_from_sums(s, x.size)
            _check_metrics((m["pcc"], m["mae"], m["atol"]), wants[fi], (tag, "fmt", fi))
        for j, a in enumerate(maps):
            s = eng.assignment_sums(td, torch.from_numpy(a).cuda()).cpu().numpy()
            m = eng.metrics_from_sums(s, x.size)
            _check_metrics((m["pcc"], m["mae"], m["atol"]), wants[j], (tag, "map", j))
        sb = eng.assignment_sums_batch(td, torch.from_numpy(np.stack(maps)).cuda()).cpu().numpy()
        for j in range(len(maps)):
            m = eng.metrics_from_sums(sb[j], x.size)
            _check_metrics((m["pcc"], m["mae"], m["atol"]), wants[j], (tag, "batch", j))
        for fmts in (["bfp8", "bfp2"], MIXED):
            ch, met, _counts = eng.random_samples(td, x.size, fmts, 6, eng.make_rng(23))
            wch, wmet = orc.random_samples_exact(want, fmts, 6, 23)
            assert np.array_equal(ch.cpu().numpy(), wch), (tag, fmts)
            met = met.cpu().numpy()
            for s in range(6):
                _check_metrics(met[s], wmet[s], (tag, "random", len(fmts), s))
        own = eng.tile_stats(eng.prepare_tiles(x), MIXED)
        for fi, f in enumerate(MIXED):
            m = eng.metrics_from_sums(eng.assignment_sums(own, fmt=fi).cpu().numpy(), x.size)
            w = orc.exact_metrics_f64(x, orc.quantize(x, f))
            _exact_f64(m["atol"], w["atol"], (tag, "own table", f, "atol"))
            _close_f64(m["mae"], w["mae"], (tag, "own table", f, "mae"))


# --------------------------------------------------------------------------------------------------------------------------
# tile-stat kernels and the greedy on inf / NaN (the E = 255 groups test_gpu_tile_stat_extremes.py leaves out)
# --------------------------------------------------------------------------------------------------------------------------
NONFINITE_CASES = [(p, s, f) for p, s, f in CASES if p in NONFINITE]
NONFINITE_IDS = [f"{p}-{s}-{'f32' if f else 'bf16'}" for p, s, f in NONFINITE_CASES]
nonfinite_params = pytest.mark.parametrize("pattern,shape,f32", NONFINITE_CASES, ids=NONFINITE_IDS)
KEYS = ("sy", "sy2", "sxy", "sabs", "amax")


def _columns(tab):
    """(name, column) of a float64 [22, T] table in the library's layout."""
    yield "sx", tab[0]
    yield "sx2", tab[1]
    for i, f in enumerate(MIXED):
        for j, k in enumerate(KEYS):
            yield f"{f}.{k}", tab[2 + 5 * i + j]


def _check_table(got, want, tag, rel):
    """Every column bit-equal with equal NaN positions and equal infinities, except the columns in `rel` (name ->
    relative bound): the rules of test_gpu_tile_stat_extremes.py for the sums whose order differs."""
    for (name, g), (_n, w) in zip(_columns(got), _columns(want)):
        assert np.array_equal(np.isnan(g), np.isnan(w)), (tag, name, np.nonzero(np.isnan(g) != np.isnan(w))[0][:8])
        if name in rel:
            assert np.allclose(g, w, rtol=rel[name], atol=0, equal_nan=True), (tag, name)
        else:
            assert np.array_equal(g, w, equal_nan=True), (tag, name, g[~np.isclose(g, w, equal_nan=True)][:4])


@nonfinite_params
def test_tile_stats_nonfinite(qa, pattern, shape, f32):
    """Every tile-stat kernel on the inf / NaN patterns against orc.tile_stat_table: bf16 fast in both |x-y| modes, the
    descriptor batch, float32 in both modes, and strict.  The BFP slots' max |x-y| and the bf16 slot's sum and max |x-y|
    are NaN wherever an element is."""
    eng = qa["eng"]
    L = eng._lib.lib()
    x, _ = _case(pattern, shape, f32)
    with np.errstate(all="ignore"):
        want = _table_arrays(orc.tile_stat_table(x))
    tag = (pattern, shape, f32)
    p = eng.prepare_tiles(x)
    assert p.dtype_code == (1 if f32 else 0), tag
    if f32:
        rel = {"sx": 1e-13, "sx2": 1e-13, "bf16.sy2": 1e-13, **{f"{f}.sxy": 1e-13 for f in MIXED}}
    else:
        rel = {"sx2": 1e-13, "bf16.sy2": 1e-13, "bf16.sxy": 1e-13}
    approx = {**rel, **{f"{f}.sabs": 1e-6 for f in MIXED}}
    _check_table(eng.tile_stats(p, MIXED).cpu().numpy(), want, (tag, "fast"), rel)
    _check_table(eng.tile_stats(p, MIXED, exact_abs=False).cpu().numpy(), want, (tag, "approx_abs"), approx)
    _check_table(eng.tile_stats(p, MIXED, strict=True).cpu().numpy(), want, (tag, "strict"), {})
    if not f32:
        t = torch.zeros((22, p.ntiles), dtype=torch.float64, device="cuda")
        descs, n, items, _b = eng.batch_descriptors([(p.data.data_ptr(), t.data_ptr(), 0, p.rows, p.cols)], torch.device("cuda"))
        assert items == L.qa_tile_stats_items(p.rows, p.cols), tag
        for exact in (True, False):
            t.zero_()
            eng.tile_stats_batch(descs, n, items, MIXED, exact_abs=exact)
            _check_table(t.cpu().numpy(), want, (tag, "batch", exact), rel if exact else approx)


@nonfinite_params
def test_greedy_nonfinite(qa, pattern, shape, f32):
    """mixed-tile-greedy on the inf / NaN patterns for pcc, mae and atol, with the cluster chain (and its certificate) and
    with the one-thread chain: the map and counts of orc.greedy_assign.  NaN sums fail every pcc / mae test, and a NaN
    maximum every atol test, as in the reference."""
    ca = qa["ca"]
    x, scores = _case(pattern, shape, f32)
    with np.errstate(all="ignore"):
        table = orc.tile_stat_table(x)
    v = scores["atol"]["bfp4"]
    v = v[np.isfinite(v)]
    thr = {"pcc": 0.999, "mae": 1.0, "atol": float(np.median(v)) if v.size else 1.0}
    for m, th in thr.items():
        with np.errstate(all="ignore"):
            a, counts = orc.greedy_assign(table, MIXED, m, th, 17)
        for seq in (False, True):
            algo = ca.create_algorithm("mixed-tile-greedy", {"metric": m, "threshold": th, "seed": 17, "sequential_chain": seq})
            res = algo.run(x, MIXED, None, None)[0]
            tag = (pattern, shape, f32, m, seq)
            assert np.array_equal(np.asarray(res.meta["assignment"]).reshape(a.shape), a), tag
            assert res.tile_counts == counts, tag
