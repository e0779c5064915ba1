"""The tile-stat kernels at the ends of the float32 range, against the oracle's float32-product semantics.

The reference forms x*x, y*y and x*y as float32 arrays and sums them in float64 (mixed_tile_greedy.py:147-174), so its
table underflows where a square falls below float32's normal range, overflows to inf where a product passes FLT_MAX, and
still counts groups that hold only denormals.  The fast kernels keep most of their arithmetic in exact group units and
route the groups where those effects can matter to a generic per-element path; these cases sit on both sides of every
routing bound:
  * denormal-only groups: a whole tile of them, beside groups of tiny normals, and one inside a normal tile (a control);
  * the underflow band: each group's first element 2^(E-127), the other fifteen 135 * 2^-77 (135^2 = 17 mod 32 maximises
    the float32 rounding of its square) for group maxima E = 72, 74, 75, 76, 78;
  * overflow: single elements and whole groups at 2^64, 1.5 * 2^64, -2^100 and the largest bf16 value; for float32 also
    0x5F7FFFFF, which rounds to bf16 2^64;
  * group maxima at the biased exponents E = 1, 71, 72, 75, 76, 190, 191 and 254.
Each pattern is built at 64 x 1024 (the 256-bit loads), 45 x 77 (the scalar loads) and as a 1-D vector with a ragged last
row, as bf16-exact data (the bf16 kernels) and with 24-bit significands (the float32 kernel).  The background of every
pattern spans few enough octaves that every tile sum the rules hold bit-equal is exactly representable.  No input is inf
or NaN.
"""
import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc

pytestmark = pytest.mark.gpu

MIXED = list(orc.MIXED_FORMATS)
KEYS = ("sy", "sy2", "sxy", "sabs", "amax")
SHAPES = {"vec": (64, 1024), "ragged": (45, 77), "1d": (3000,)}
OVER = {"2p64": 0x5F80, "1p5x2p64": 0x5FC0, "m2p100": 0xF180, "bf16max": 0x7F7F}
UNDER_E = (72, 74, 75, 76, 78)
BOUND_FINITE = (1, 71, 72, 75, 76, 190)
BOUND_OVER = (190, 191, 254)
# patterns whose oracle table is finite everywhere (the end-to-end greedy runs on these)
FINITE = ["denorm_tile", "denorm_tiny", "denorm_control"] + [f"under{e}" for e in UNDER_E] + ["bound_finite"]
BF16_PATTERNS = FINITE + [f"over_{k}" for k in OVER] + ["bound_over"]
F32_PATTERNS = BF16_PATTERNS + ["over_5f7fffff"]
BF16_CASES = [(p, s) for p in BF16_PATTERNS for s in SHAPES]
F32_CASES = [(p, s) for p in F32_PATTERNS for s in SHAPES]


# --------------------------------------------------------------------------------------------------------------------------
# inputs (seeded NumPy)
# --------------------------------------------------------------------------------------------------------------------------
def _f32(bits):
    return np.ascontiguousarray(bits, dtype=np.uint32).view(np.float32)


def _values(rng, shape, e_lo, e_hi, f32, cap=(254,)):
    """Random-signed values with biased exponents in [e_lo, e_hi] (0 = denormal) and random significands: 7 bits (bf16)
    or 23 bits (float32).  In the binades `cap`, float32 significands stay below the bf16 rounding that carries into the
    next binade (254: inf; 190: 2^64, whose bf16 square overflows)."""
    e = rng.integers(e_lo, e_hi + 1, shape).astype(np.uint32)
    s = rng.integers(0, 2, shape).astype(np.uint32) << 31
    m = rng.integers(0, 1 << 23, shape).astype(np.uint32) if f32 else rng.integers(0, 128, shape).astype(np.uint32) << 16
    if f32:
        m[np.isin(e, cap)] &= 0x7EFFFF
    m[(e == 0) & (m == 0)] |= 1 << 16      # a denormal draw is never a zero
    return _f32(s | (e << 23) | m)


def _perturb(x, rng):
    """24-bit significands: set low bits below bf16's rounding half-way point (so every bf16 image is unchanged)."""
    b = x.view(np.uint32).copy()
    nz = (b & 0x7FFFFFFF) != 0
    b[nz] |= rng.integers(1, 1 << 12, b.shape).astype(np.uint32)[nz]
    return _f32(b)


def _pattern(name, R, C, f32, seed):
    """Pattern `name` on an R x C grid (groups of 16 along the columns, 32 x 32 tiles)."""
    rng = np.random.default_rng(seed)
    g = np.arange(C)[None, :] // 16 + np.zeros((R, 1), np.int64)
    r = np.arange(R)[:, None] + np.zeros((1, C), np.int64)
    if name == "denorm_tile":                      # mixed-sign denormals only
        x = _values(rng, (R, C), 0, 0, f32)
    elif name == "denorm_tiny":                    # denormal-only groups (positive) beside groups of normals near 2^-120
        x = _values(rng, (R, C), 7, 7, f32)
        d = np.abs(_values(rng, (R, C), 0, 0, f32))
        x = np.where((r + g) % 2 == 0, d, x)
    elif name == "denorm_control":                 # one denormal-only group inside every tile of normal values
        x = _values(rng, (R, C), 120, 124, f32)
        d = np.abs(_values(rng, (R, C), 0, 0, f32))
        x = np.where((r % 32 == 5) & (g % 2 == 0), d, x)
    elif name.startswith("under"):                 # group max 2^(E-127), fifteen elements 135 * 2^-77
        E = int(name[5:])
        x = np.full((R, C), np.float32(135.0 * 2.0 ** -77))
        if f32:
            x = _perturb(x, rng)
        x[:, ::16] = np.float32(2.0 ** (E - 127))
    elif name.startswith("over_"):                 # per tile: one element / a whole group / nothing at v
        key = name[5:]
        v = (_f32(np.uint32(0x5F7FFFFF)) if key == "5f7fffff" else _f32(np.uint32(OVER[key] << 16)))[0]
        ev = (int(v.view(np.uint32)) >> 23) & 0xFF
        x = _values(rng, (R, C), ev - 10, ev - 8, f32)       # close enough that a finite tile sum y^2 stays exact
        for tr in range(-(-R // 32)):
            for tc in range(-(-C // 32)):
                k = (tr + tc) % 3
                if k == 0 and tr * 32 + 3 < R and tc * 32 + 5 < C:
                    x[tr * 32 + 3, tc * 32 + 5] = v
                elif k == 1 and tr * 32 + 7 < R:
                    x[tr * 32 + 7, tc * 32:tc * 32 + 16] = v
    elif name.startswith("bound_"):                # per tile one maximum exponent E; every group's max exactly at E
        es = BOUND_FINITE if name == "bound_finite" else BOUND_OVER
        cap = (190, 254) if name == "bound_finite" else (254,)
        tw = -(-C // 32)
        E = np.asarray(es)[((r // 32) * tw + np.arange(C)[None, :] // 32) % len(es)]
        x = _values(rng, (R, C), 0, 0, f32)
        for e in es:
            x = np.where(E == e, _values(rng, (R, C), max(e - 3, 0), e, f32, cap), x)
        pos = rng.integers(0, 16, (R, (C + 15) // 16))
        for gi in range((C + 15) // 16):
            c = np.minimum(gi * 16 + pos[:, gi], C - 1)
            e_tile = E[np.arange(R), c]
            m = rng.integers(0, 1 << 23, R).astype(np.uint32) if f32 else rng.integers(0, 128, R).astype(np.uint32) << 16
            if f32:
                m[np.isin(e_tile, cap)] &= 0x7EFFFF
            sgn = rng.integers(0, 2, R).astype(np.uint32) << 31
            x[np.arange(R), c] = _f32(sgn | (e_tile.astype(np.uint32) << 23) | m)
    else:
        raise KeyError(name)
    return np.ascontiguousarray(x, dtype=np.float32)


_CASES = {}


def _case(pattern, shape, f32):
    """(input, oracle table), cached for the module."""
    key = (pattern, shape, f32)
    if key not in _CASES:
        dims = SHAPES[shape]
        seed = 1000 + 37 * F32_PATTERNS.index(pattern) + 7 * list(SHAPES).index(shape) + int(f32)
        if len(dims) == 1:
            n = dims[0]
            x = _pattern(pattern, -(-n // 32), 32, f32, seed).reshape(-1)[:n].copy()
        else:
            x = _pattern(pattern, dims[0], dims[1], f32, seed)
        with np.errstate(all="ignore"):
            want = orc.tile_stat_table(x)
        _CASES[key] = (x, want)
    return _CASES[key]


def _finite(want):
    cols = [want["sx"], want["sx2"]] + [want[f][k] for f in MIXED for k in KEYS]
    return all(np.isfinite(c).all() for c in cols)


# --------------------------------------------------------------------------------------------------------------------------
# comparison rules
# --------------------------------------------------------------------------------------------------------------------------
def _table(t):
    tb = t.cpu().numpy()
    out = {"sx": tb[0], "sx2": tb[1]}
    for i, f in enumerate(MIXED):
        out[f] = {k: tb[2 + 5 * i + j] for j, k in enumerate(KEYS)}
    return out


def _columns(tab):
    yield "sx", tab["sx"]
    yield "sx2", tab["sx2"]
    for f in MIXED:
        for k in KEYS:
            yield f"{f}.{k}", tab[f][k]


def _check_inf(got, want, tag):
    """Every inf of the oracle is the same inf in the kernel's table, and the kernel has no other non-finite value."""
    for (name, g), (_n, w) in zip(_columns(got), _columns(want)):
        assert np.array_equal(np.isposinf(g), np.isposinf(w)) and np.array_equal(np.isneginf(g), np.isneginf(w)), (tag, name)
        assert not np.isnan(g).any(), (tag, name)


def _check_strict(got, want, tag):
    for (name, g), (_n, w) in zip(_columns(got), _columns(want)):
        assert np.array_equal(g, w), (tag, name)


def _check_bf16_fast(got, want, tag):
    """The rule of test_gpu_parity.test_tile_stats_fast_matches_oracle: bit-equal except sum x^2 (and the bf16 slot's
    sum y^2 and sum x*y, which are sum x^2) within 1e-13 relative."""
    _check_inf(got, want, tag)
    assert np.array_equal(got["sx"], want["sx"]), tag
    assert np.allclose(got["sx2"], want["sx2"], rtol=1e-13, atol=0), tag
    for f in MIXED:
        for k in KEYS:
            if f == "bf16" and k in ("sy2", "sxy"):
                assert np.allclose(got[f][k], want[f][k], rtol=1e-13, atol=0), (tag, f, k)
            else:
                assert np.array_equal(got[f][k], want[f][k]), (tag, f, k)


def _check_f32_fast_table(got, want, tag, exact=True):
    """As test_gpu_parity._check_f32_fast_table: sums of exactly representable terms are bit-equal; sum x, sum x^2 and
    sum x*y of 24-bit data round differently in another order (held to 1e-13 relative, a few ulp).  The bf16 slot's sum y^2
    squares the bf16 images exactly where the reference rounds y*y below 2^-67 in float32's denormal range: held to 1e-13
    as the bf16 kernel's sum x^2 is (the underflow-band cases reach that)."""
    _check_inf(got, want, tag)
    for k in ("sx", "sx2"):
        assert np.allclose(got[k], want[k], rtol=1e-13, atol=0, equal_nan=True), (tag, k)
    assert np.allclose(got["bf16"]["sy2"], want["bf16"]["sy2"], rtol=1e-13, atol=0, equal_nan=True), (tag, "bf16", "sy2")
    for f in MIXED:
        for k in ("sy", "sy2", "sabs", "amax"):
            if f == "bf16" and k == "sy2":
                continue
            if exact or k == "amax":
                assert np.array_equal(got[f][k], want[f][k], equal_nan=True), (tag, f, k)
            else:
                assert np.allclose(got[f][k], want[f][k], rtol=1e-13, atol=1e-300, equal_nan=True), (tag, f, k)
        assert np.allclose(got[f]["sxy"], want[f]["sxy"], rtol=1e-13, atol=0, equal_nan=True), (tag, f)


def _approx_abs(got, want, tag):
    """exact_abs=False keeps sum |x-y| in float32 group partials: 1e-6 relative; the other columns follow the exact rule."""
    for f in MIXED:
        assert np.allclose(got[f]["sabs"], want[f]["sabs"], rtol=1e-6, atol=0), (tag, f)
        got[f]["sabs"] = want[f]["sabs"]
    return got


@pytest.fixture(scope="module")
def qa():
    from quantization_analysis_b200 import _lib, engine
    from quantization_analysis_b200 import compression_algorithms as ca
    return {"L": _lib.lib(), "lib": _lib, "eng": engine, "ca": ca}


def _stream():
    return torch.cuda.current_stream().cuda_stream


# --------------------------------------------------------------------------------------------------------------------------
# bf16 kernels
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern,shape", BF16_CASES)
def test_bf16_kernels(qa, pattern, shape):
    """stats_fast_kernel (both load paths, both |x-y| modes), stats_strict_kernel and qa_tile_stats_rows in two pieces."""
    eng, L, lib = qa["eng"], qa["L"], qa["lib"]
    x, want = _case(pattern, shape, False)
    tag = (pattern, shape)
    p = eng.prepare_tiles(x)
    assert p.dtype_code == 0, tag
    fast = eng.tile_stats(p, MIXED, strict=False)
    _check_bf16_fast(_table(fast), want, tag)
    approx = _table(eng.tile_stats(p, MIXED, strict=False, exact_abs=False))
    _check_bf16_fast(_approx_abs(approx, want, tag), want, (tag, "approx_abs"))
    strict = _table(eng.tile_stats(p, MIXED, strict=True))
    _check_strict(strict, want, (tag, "strict"))
    th = p.tiles_h
    t = torch.zeros_like(fast)
    for lo, hi in ((0, 1), (1, th)) if th > 1 else ((0, 1),):
        lib.check(L.qa_tile_stats_rows(p.data.data_ptr(), 0, p.rows, p.cols, p.cols, 0xF, 0, t.data_ptr(), lo, hi, _stream()),
                  "qa_tile_stats_rows")
    assert torch.equal(t.nan_to_num(nan=-1.0), fast.nan_to_num(nan=-1.0)), tag


def test_bf16_batch_kernel(qa):
    """qa_tile_stats_batch: one launch over every bf16 case (vector and scalar loads in one grid), each table checked
    against the oracle."""
    eng, L, lib = qa["eng"], qa["L"], qa["lib"]
    preps, tables, wants = [], [], []
    for pattern, shape in BF16_CASES:
        x, want = _case(pattern, shape, False)
        p = eng.prepare_tiles(x)
        preps.append(p)
        tables.append(torch.zeros((22, p.ntiles), dtype=torch.float64, device="cuda"))
        wants.append(want)
    descs, n, items, _blocks = eng.batch_descriptors([(p.data.data_ptr(), t.data_ptr(), 0, p.rows, p.cols)
                                                      for p, t in zip(preps, tables)], torch.device("cuda"))
    assert items == sum(L.qa_tile_stats_items(p.rows, p.cols) for p in preps)
    eng.tile_stats_batch(descs, n, items, MIXED, exact_abs=True)
    for (pattern, shape), t, want in zip(BF16_CASES, tables, wants):
        _check_bf16_fast(_table(t), want, (pattern, shape, "batch"))


# --------------------------------------------------------------------------------------------------------------------------
# float32 kernel
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pattern,shape", F32_CASES)
def test_f32_kernels(qa, pattern, shape):
    """stats_f32_kernel<0, .> (both |x-y| modes), stats_strict_kernel<F32> and qa_tile_stats_f32 over tile-row ranges."""
    eng, L, lib = qa["eng"], qa["L"], qa["lib"]
    x, want = _case(pattern, shape, True)
    tag = (pattern, shape, "f32")
    p = eng.prepare_tiles(x)
    assert p.dtype_code == 1, tag
    fast = eng.tile_stats(p, MIXED)
    _check_f32_fast_table(_table(fast), want, tag)
    approx = _table(eng.tile_stats(p, MIXED, exact_abs=False))
    _check_f32_fast_table(_approx_abs(approx, want, tag), want, (tag, "approx_abs"))
    _check_strict(_table(eng.tile_stats(p, MIXED, strict=True)), want, (tag, "strict"))
    th = p.tiles_h
    t = torch.zeros_like(fast)
    for lo, hi in ((0, 1), (1, th)) if th > 1 else ((0, 1),):
        lib.check(L.qa_tile_stats_f32(p.data.data_ptr(), p.rows, p.cols, p.cols, 0xF, 0, t.data_ptr(), lo, hi, _stream()),
                  "qa_tile_stats_f32")
    assert torch.equal(t.nan_to_num(nan=-1.0), fast.nan_to_num(nan=-1.0)), tag


# --------------------------------------------------------------------------------------------------------------------------
# fp8 e4m3fn with block scales
# --------------------------------------------------------------------------------------------------------------------------
def test_fp8_blocks_at_both_ends(qa):
    """qa_tile_stats_fp8 on 128 x 128 scale blocks, one with scale_inv 2^-140 (every element denormal or zero), one with
    2^58 (448 * scale past 2^64), the others normal: bit-equal to the float32 kernel on the dequantized tensor and held to
    the oracle by the float32 rule, in both |x-y| modes."""
    from quantization_analysis_b200 import synthetic
    eng = qa["eng"]
    wt, sct = synthetic.fp8_checkpoint_cpu((256, 384), 31)
    w, sc = wt.numpy(), sct.numpy().copy()
    sc[0, 1] = np.float32(2.0 ** -140)
    sc[1, 2] = np.float32(2.0 ** 58)
    xo = orc.fp8_block_dequant(w, sc)
    xd, _, _ = eng.fp8_block_dequant(torch.from_numpy(w), torch.from_numpy(sc), want_bf16=False)
    xd = xd.cpu().numpy()
    assert np.array_equal(xd.view(np.uint32), xo.view(np.uint32))
    blk = xo[:128, 128:256]
    assert (np.abs(blk) < np.float32(2.0 ** -126)).all() and (blk != 0).any()
    assert np.abs(xo[128:, 256:]).max() > 2.0 ** 64
    p = eng.prepare_tiles(xd)
    assert p.dtype_code == 1
    with np.errstate(all="ignore"):
        want = orc.tile_stat_table(xo)
    assert np.isinf(want["sx2"]).any() and np.isfinite(want["sx2"]).any()
    for exact in (True, False):
        table, _ = eng.tile_stats_fp8(torch.from_numpy(w), torch.from_numpy(sc), exact_abs=exact)
        assert torch.equal(table.nan_to_num(nan=-1.0), eng.tile_stats(p, MIXED, exact_abs=exact).nan_to_num(nan=-1.0)), exact
        got = _table(table)
        if not exact:
            got = _approx_abs(got, want, "fp8")
        _check_f32_fast_table(got, want, ("fp8", exact))


# --------------------------------------------------------------------------------------------------------------------------
# end to end: the certified greedy on every case with a finite oracle table
# --------------------------------------------------------------------------------------------------------------------------
def _thresholds(want, numel):
    """A threshold per metric that falls between the formats' whole-tensor values, so the greedy has choices to make."""
    mae = [float(np.sum(want[f]["sabs"])) / numel for f in ("bfp8", "bfp4")]
    amax = want["bfp4"]["amax"]
    return {"pcc": 0.999, "mae": 0.5 * (mae[0] + mae[1]), "atol": float(np.median(amax))}


@pytest.mark.parametrize("f32", [False, True], ids=["bf16", "f32"])
@pytest.mark.parametrize("pattern,shape", [(p, s) for p in FINITE for s in SHAPES])
def test_certified_greedy(qa, pattern, shape, f32):
    """mixed-tile-greedy with certify on, for pcc, mae and atol: the map and counts of orc.greedy_assign on the oracle's
    table."""
    ca = qa["ca"]
    x, want = _case(pattern, shape, f32)
    assert _finite(want), (pattern, shape, f32)
    for metric, thr in _thresholds(want, x.size).items():
        algo = ca.create_algorithm("mixed-tile-greedy", {"metric": metric, "threshold": thr, "seed": 17, "certify": True})
        res = algo.run(x, MIXED, None, None)[0]
        a, counts = orc.greedy_assign(want, MIXED, metric, thr, 17)
        tag = (pattern, shape, f32, metric, thr)
        assert np.array_equal(np.asarray(res.meta["assignment"]).reshape(a.shape), a), tag
        assert res.tile_counts == counts, tag
