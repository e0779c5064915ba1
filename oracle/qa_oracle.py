"""CPU oracle for the quantize-and-score hot path (TEST INFRASTRUCTURE ONLY).

This module is a NumPy restatement of the reference algorithm
(johanna-rock/quantization_analysis).  It is the *checker* for the CUDA path:
only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  Nothing under
``quantization_analysis_b200/`` imports it, and the product path raises when
the CUDA library is missing instead of falling back to this file.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4),
so this oracle is pinned against the *reference itself*, imported from
``/root/reference`` in the build container by ``tests/golden/make_golden.py``;
the resulting fixtures are committed under ``tests/golden/`` and re-checked by
``tests/test_oracle_golden.py`` on every run (CPU).  Command-line goldens (``tests/golden/cli``) are the files the
reference's own ``wq`` and sweep programs wrote (``tests/golden/make_golden_cli.py``).  ``oracle/make_ref.sh`` additionally
copies the unmodified reference into the git-ignored ``oracle/_ref/`` (it travels to the GPU box): the CPU arm of ``bench.py``
times it, and ``tests/test_gpu_cli.py`` runs its programs over this repository's drop-in modules.

Third-party arithmetic the reference's results depend on (not vendored in the
reference; ``requirements.txt`` is unpinned; this image has numpy 2.3.5 with
OpenBLAS 0.3.30, SkylakeX kernels):
  * ``np.add.reduce`` pairwise summation          -> :func:`np_pairwise_sum`
  * ``np.dot`` on float32 vectors (``cblas_sdot``) -> :func:`np_sdot_f32`
  * ``np.random.Generator(PCG64)``                -> :class:`Pcg64`
Each restatement below cites the reference line it follows.
"""
from __future__ import annotations

import math

import numpy as np

TILE = 32
GROUP = 16
MIXED_FORMATS = ("bf16", "bfp8", "bfp4", "bfp2")          # tile_utils.py:8
BYTES_PER_ELEM = {"bf16": 2.0, "bfp8": 1.088, "bfp4": 0.50097, "bfp2": 0.25097}  # tile_utils.py:9-14
MANT_BITS = {"bfp8": 7, "bfp4": 3, "bfp2": 1}             # quantization_formats.py:186-191
WQ_BYTES_PER_ELEM = {"mxfp4": 0.5, "nvfp4": 0.5, "bf16": 2.0, "bfp8": 1.088,
                     "bfp4": 0.50097, "bfp2": 0.25097, "fp0": 0.0}  # wq:132-140


# --------------------------------------------------------------------------- #
# Format emulation (quantization_formats.py)
# --------------------------------------------------------------------------- #
def bf16_round(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 (RNE on the bit pattern, no NaN special case) -> fp32.

    Follows quantization_formats.py:29-45.
    """
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    keep = (u + (np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1)))) >> np.uint32(16)
    return (keep << np.uint32(16)).view(np.float32).reshape(np.shape(x))


def _rows_view(x: np.ndarray) -> tuple[np.ndarray, tuple]:
    """Collapse to [rows, width]; BFP groups never cross a row.

    quantization_formats.py:89-99 keeps (batch, H, W); because a shared
    exponent only spans 16 contiguous elements of the last axis the batch/H
    split cannot change a value, so rows = prod(shape[:-1]).
    """
    x = np.asarray(x, dtype=np.float32)
    shp = x.shape
    if x.ndim == 0:
        return x.reshape(1, 1), shp
    if x.ndim == 1:
        return x.reshape(1, -1), shp
    return x.reshape(-1, shp[-1]), shp


def bfp_quantize(x: np.ndarray, mant_bits: int) -> np.ndarray:
    """TTNN-style BFP quantize->dequantize, one shared exponent per 16-wide row group.

    Restates quantization_formats.py:84-164 group-wise:
      E   = max biased exponent of the group                        (:118-119)
      m24 = (1<<23 | frac) >> (E - e)   (anything shifted >= 24 is 0) (:125-131)
      q   = RNE(m24 / 2^(24-mb)), clamped to 2^mb - 1               (:133-141)
      q   = 0 for exp == 0 inputs; sign dropped when q == 0          (:143-145)
      out = sign | (E - (mb-1-msb(q))) << 23 | normalised mantissa   (:147-158)
    """
    x2, shp = _rows_view(x)
    if x2.size == 0:
        return np.asarray(x, dtype=np.float32).copy()
    rows, width = x2.shape
    wpad = -(-width // GROUP) * GROUP
    buf = np.zeros((rows, wpad), dtype=np.uint32)
    buf[:, :width] = np.ascontiguousarray(x2).view(np.uint32)
    g = buf.reshape(rows, wpad // GROUP, GROUP)
    e = (g >> np.uint32(23)) & np.uint32(0xFF)
    big_e = e.max(axis=-1, keepdims=True)
    sign = g >> np.uint32(31)
    m24 = (g & np.uint32(0x7FFFFF)) | np.uint32(1 << 23)
    d = (big_e - e).astype(np.uint32)
    m = np.where(d >= 24, np.uint32(0), m24 >> np.minimum(d, np.uint32(31)))
    drop = np.uint32(24 - mant_bits)
    low = m & np.uint32((1 << (24 - mant_bits)) - 1)
    half = np.uint32(1 << (24 - mant_bits - 1))
    q = m >> drop
    up = (low > half) | ((low == half) & ((q & np.uint32(1)) == 1))
    q = np.minimum(q + up.astype(np.uint32), np.uint32((1 << mant_bits) - 1))
    q = np.where(e == 0, np.uint32(0), q)
    nz = q != 0
    qs = np.where(nz, q, np.uint32(1))
    msb = np.floor(np.log2(qs.astype(np.float64))).astype(np.uint32)
    lshift = np.uint32(mant_bits - 1) - msb
    frac = (qs << (lshift + np.uint32(1))) & np.uint32((1 << mant_bits) - 1)
    e_out = (big_e.astype(np.uint32) - lshift).astype(np.uint32)      # uint32 wrap as in :154
    bits = (sign << np.uint32(31)) | (e_out << np.uint32(23)) | (frac << np.uint32(23 - mant_bits))
    bits = np.where(nz, bits, np.uint32(0)).astype(np.uint32)
    out = bits.reshape(rows, wpad)[:, :width]
    return np.ascontiguousarray(out).view(np.float32).reshape(shp)


def quantize(x: np.ndarray, fmt: str) -> np.ndarray:
    """Dispatch of quantization_formats.py:171-194 for the in-scope formats."""
    f = fmt.lower()
    x = np.asarray(x, dtype=np.float32)
    if f == "bf16":
        return bf16_round(x)
    if f in MANT_BITS:
        return bfp_quantize(x, MANT_BITS[f])
    if f == "fp0":
        return np.zeros_like(x, dtype=np.float32)
    if f == "mxfp4":
        return scalar_proxy(x, "mxfp4")
    if f == "nvfp4":
        return scalar_proxy(x, "nvfp4")
    raise ValueError(f"Unsupported weight format: {f}")


# --------------------------------------------------------------------------- #
# mxfp4 / nvfp4 scalar proxies (quantization_formats.py:171-183, 197-278)
# --------------------------------------------------------------------------- #
_FP4_LEVELS = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0], dtype=np.float32)


def _fp4_nearest(a: np.ndarray) -> np.ndarray:
    """quantize_fp4_e2m1 on non-negative float32 (:197-202): first argmin of the float32 |a - level|."""
    d = np.abs(a[..., None] - _FP4_LEVELS[None, :])
    return _FP4_LEVELS[np.argmin(d, axis=-1)]


def _exponent_f32(a: np.ndarray) -> np.ndarray:
    """floor(log2(a)) for positive finite float32, exactly (the reference takes np.log2 in float32, whose rounding can
    differ for an argument within ~|k| * 4e-8 of a power of two 2^k; never the case for the quotients of bf16 values)."""
    m, e = np.frexp(a.astype(np.float64))
    return (e - 1).astype(np.int32)


def _fp8_e4m3(ax: np.ndarray) -> np.ndarray:
    """quantize_fp8_e4m3 on non-negative float32 (:205-251)."""
    out = np.zeros_like(ax, dtype=np.float32)
    nz = ax > 0
    if not nz.any():
        return out
    a = ax[nz]
    e = _exponent_f32(a)
    res = np.zeros_like(a, dtype=np.float32)
    normal, sub, big = (e >= -6) & (e <= 7), e < -6, e > 7          # e_min = 1 - bias = -6, e_max = 14 - bias = 7
    if normal.any():
        en = e[normal].astype(np.int64)
        m = a[normal].astype(np.float64) / (2.0 ** en)
        fq = np.round((m - 1.0) * 8.0) / 8.0
        bumped = fq >= 1.0
        fq = np.where(bumped, 0.0, fq)
        en = np.where(bumped, np.minimum(en + 1, 7), en)
        res[normal] = ((1.0 + fq) * (2.0 ** en)).astype(np.float32)
    if sub.any():
        step = np.float32(2.0 ** -9)
        res[sub] = np.round(a[sub] / step) * step
    if big.any():
        res[big] = np.float32(240.0)                                        # (1 + 7/8) * 2^7
    out[nz] = res
    return out


def scalar_proxy(x: np.ndarray, fmt: str) -> np.ndarray:
    """Elementwise mxfp4 / nvfp4 proxy: every magnitude is treated as the amax of a block of identical values."""
    x = np.asarray(x, dtype=np.float32)
    ax = np.abs(x).reshape(-1)
    q = np.zeros_like(ax)
    fin = np.isfinite(ax) & (ax > 0)
    a = ax[fin]
    with np.errstate(all="ignore"):
        if fmt == "mxfp4":
            s = (a.astype(np.float64) / 6.0).astype(np.float32)            # python-float division, then float32 (:256-257)
            ok = s > 0
            m, e = np.frexp(s.astype(np.float64))
            k = np.where(m == 0.5, e - 1, e).astype(np.float64)           # ceil(log2(s))
            sq = np.where(ok, np.exp2(k), 0.0).astype(np.float32)
        else:
            s = a / np.float32(6.0)                                        # float32 division (:266)
            sq = _fp8_e4m3(s)
            ok = sq > 0
        r = np.zeros_like(a)
        r[ok] = _fp4_nearest(a[ok] / sq[ok]) * sq[ok]
    q[fin] = r
    q[~np.isfinite(ax)] = np.nan                                            # inf / nan propagate as nan
    return (np.sign(x).reshape(-1) * q).reshape(x.shape).astype(np.float32)


# --------------------------------------------------------------------------- #
# NumPy / OpenBLAS arithmetic orders (SURVEY.md Appendix B)
# --------------------------------------------------------------------------- #
def np_pairwise_sum(a: np.ndarray) -> np.ndarray:
    """numpy ``add.reduce`` over the last axis of a contiguous array, same dtype.

    Order: blocks of <=128 use 8 strided accumulators, combined as
    ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and then the n%8 tail one by one;
    longer inputs split at n/2 rounded down to a multiple of 8.  Vectorised
    over all leading axes.
    """
    n = a.shape[-1]
    if n < 8:
        r = np.zeros(a.shape[:-1], dtype=a.dtype)
        for i in range(n):
            r = r + a[..., i]
        return r
    if n <= 128:
        r = [a[..., k] for k in range(8)]
        i = 8
        while i < n - (n % 8):
            for k in range(8):
                r[k] = r[k] + a[..., i + k]
            i += 8
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
        while i < n:
            res = res + a[..., i]
            i += 1
        return res
    n2 = n // 2
    n2 -= n2 % 8
    return np_pairwise_sum(a[..., :n2]) + np_pairwise_sum(a[..., n2:])


def _fma_f32(a: np.ndarray, b: np.ndarray, c: np.ndarray) -> np.ndarray:
    """Correctly rounded float32 fma(a, b, c), vectorised (round-to-odd in f64).

    The product of two float32 values is exact in float64 and cannot overflow it, so a non-finite float64 sum s means an
    inf or NaN operand: s is then the IEEE result (inf * 0 and inf - inf are NaN) and is returned as it is."""
    p = a.astype(np.float64) * b.astype(np.float64)          # exact (48 bits)
    cc = c.astype(np.float64)
    s = p + cc
    bb = s - p
    err = (p - (s - bb)) + (cc - bb)                          # TwoSum error term
    bits = s.view(np.uint64) if s.ndim else np.array(s).view(np.uint64)
    inexact = (err != 0.0) & np.isfinite(s)
    even = (bits & np.uint64(1)) == 0
    # round-to-odd: if inexact and the f64 result is even, step one ulp towards the true value
    toward_up = (err > 0.0) == (s > 0.0)
    fix = inexact & even
    bits = np.where(fix & toward_up, bits + np.uint64(1), bits)
    bits = np.where(fix & ~toward_up, bits - np.uint64(1), bits)
    # (an even mantissa minus one is odd; crossing zero cannot happen for |err| < ulp)
    return bits.view(np.float64).astype(np.float32)


def np_sdot_f32(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """``np.dot`` of float32 vectors as OpenBLAS 0.3.30's SkylakeX ``sdot`` evaluates it (pinned against np.dot in
    tests/test_oracle_golden.py for many n, same image).

    n1 = n & -32 elements go through the vector kernel: blocks of 64 feed 64 FMA accumulators (4 vectors x 16 lanes;
    element i -> accumulator (i%64)//16, lane i%16, increasing i); lanes l and l+8 of each accumulator are added
    (-> 4 x 8 lanes); a remaining block of 32 is one more FMA into those 4 x 8 lanes; then ((A0+A1)+A2)+A3, lanes l and
    l+4, (v0+v1)+(v2+v3).  The last n%32 elements are summed separately: float32 products accumulated in a DOUBLE that
    starts at 0; the result is float32(double_tail + kernel).  Vectorised over leading axes.
    """
    n = x.shape[-1]
    lead = x.shape[:-1]
    n1 = n & -32
    n64 = n1 & ~63
    acc = np.zeros(lead + (4, 16), dtype=np.float32)
    if n64:
        xs = x[..., :n64].reshape(lead + (n64 // 64, 4, 16))
        ys = y[..., :n64].reshape(lead + (n64 // 64, 4, 16))
        for it in range(n64 // 64):
            acc = _fma_f32(xs[..., it, :, :], ys[..., it, :, :], acc)
    h = acc[..., :, :8] + acc[..., :, 8:]
    if n1 - n64 == 32:
        h = _fma_f32(x[..., n64:n1].reshape(lead + (4, 8)), y[..., n64:n1].reshape(lead + (4, 8)), h)
    s = ((h[..., 0, :] + h[..., 1, :]) + h[..., 2, :]) + h[..., 3, :]
    q = s[..., :4] + s[..., 4:]
    kern = ((q[..., 0] + q[..., 1]) + (q[..., 2] + q[..., 3])).astype(np.float32)
    if n1 == n:
        return kern
    tail = np.zeros(lead, dtype=np.float64)
    for i in range(n1, n):
        tail = tail + (y[..., i] * x[..., i]).astype(np.float32).astype(np.float64)
    return (tail + kern.astype(np.float64)).astype(np.float32)


def pearson_f32_restated(a: np.ndarray, b: np.ndarray) -> float:
    """metrics.py:6-16 on whole (flattened) tensors with the NumPy / OpenBLAS summation orders restated explicitly:
    the value the reference prints, reproduced without calling np.mean / np.dot (what the CUDA scorer is checked against)."""
    a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
    b = np.ascontiguousarray(b, dtype=np.float32).reshape(-1)
    if a.size == 0:
        return 1.0
    n = np.float32(a.size)
    am = a - np.float32(np_pairwise_sum(a) / n)
    bm = b - np.float32(np_pairwise_sum(b) / n)
    na = np.sqrt(np.float32(np_sdot_f32(am, am)))
    nb = np.sqrt(np.float32(np_sdot_f32(bm, bm)))
    denom = float(np.float32(na * nb))
    if denom == 0.0:
        return 1.0 if np.max(np.abs(a - b)) == 0.0 else 0.0
    return float(np.float32(np_sdot_f32(am, bm)) / np.float32(denom))


def wq_scores_restated(x: np.ndarray, y: np.ndarray) -> dict:
    """wq:684-687 (mae, atol, pcc of a result against the input), restated orders."""
    x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1)
    y = np.ascontiguousarray(y, dtype=np.float32).reshape(-1)
    d = np.abs(x - y)
    mae = float(np.float32(np_pairwise_sum(d) / np.float32(d.size))) if d.size else float("nan")
    return {"pcc": pearson_f32_restated(x, y), "mae": mae, "atol": float(d.max()) if d.size else float("nan")}


# --------------------------------------------------------------------------- #
# Metrics (compression_algorithms/metrics.py, tile_utils.py:46-57)
# --------------------------------------------------------------------------- #
def pearson_f32(a: np.ndarray, b: np.ndarray) -> float:
    """metrics.py:6-16 evaluated with NumPy itself (float32 end to end)."""
    a = np.asarray(a, dtype=np.float32).reshape(-1)
    b = np.asarray(b, dtype=np.float32).reshape(-1)
    if a.size == 0:
        return 1.0
    am = a - np.mean(a)
    bm = b - np.mean(b)
    denom = float(np.linalg.norm(am) * np.linalg.norm(bm))
    if denom == 0.0:
        return 1.0 if np.max(np.abs(a - b)) == 0.0 else 0.0
    return float(np.dot(am, bm) / denom)


def pearson_f32_rows(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Row-wise metrics.py:6-16 for [N, 1024] inputs, with the NumPy/OpenBLAS
    summation orders restated explicitly (bit-faithful, CPU-model independent)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    n = np.float32(a.shape[-1])
    am = a - (np_pairwise_sum(a) / n)[..., None]
    bm = b - (np_pairwise_sum(b) / n)[..., None]
    na = np.sqrt(np_sdot_f32(am, am))
    nb = np.sqrt(np_sdot_f32(bm, bm))
    denom = (na * nb).astype(np.float32)
    dots = np_sdot_f32(am, bm)
    exact = np.max(np.abs(a - b), axis=-1) == 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        r = (dots / denom).astype(np.float32)
    return np.where(denom == 0.0, np.where(exact, np.float32(1.0), np.float32(0.0)), r).astype(np.float32)


def metric_f32(a: np.ndarray, b: np.ndarray, metric: str) -> float:
    """metrics.py:19-27."""
    if metric == "pcc":
        return pearson_f32(a, b)
    diff = np.abs(np.asarray(a, dtype=np.float32) - np.asarray(b, dtype=np.float32))
    if metric == "mae":
        return float(np.mean(diff))
    if metric == "atol":
        return float(np.max(diff))
    raise ValueError(f"Unsupported metric: {metric}")


def is_good(value, metric: str, threshold: float) -> bool:
    """metrics.py:30-33 (NumPy-2 scalar promotion applies when value is np.float32)."""
    return bool(value >= threshold) if metric == "pcc" else bool(value <= threshold)


def is_better(a, b, metric: str) -> bool:
    """metrics.py:36-39."""
    return bool(a > b) if metric == "pcc" else bool(a < b)


def tile_scores_f32(ref_tiles: np.ndarray, q_tiles: np.ndarray, metric: str) -> np.ndarray:
    """tile_utils.py:46-57 on padded [N,32,32] tiles -> float32[N] (restated orders)."""
    n = ref_tiles.shape[0]
    a = np.ascontiguousarray(ref_tiles, dtype=np.float32).reshape(n, -1)
    b = np.ascontiguousarray(q_tiles, dtype=np.float32).reshape(n, -1)
    if metric == "pcc":
        return pearson_f32_rows(a, b)
    diff = np.abs(a - b)
    if metric == "mae":
        return (np_pairwise_sum(diff) / np.float32(diff.shape[1])).astype(np.float32)
    if metric == "atol":
        return diff.max(axis=1)
    raise ValueError(f"Unsupported metric: {metric}")


def exact_metrics_f64(x: np.ndarray, y: np.ndarray) -> dict:
    """fp64 evaluation of the same formulas (what the fast GPU path must match to 1e-6)."""
    a = np.asarray(x, dtype=np.float64).reshape(-1)
    b = np.asarray(y, dtype=np.float64).reshape(-1)
    n = float(a.size)
    if a.size == 0:
        return {"pcc": 1.0, "mae": 0.0, "atol": 0.0}
    d = np.abs(a - b)
    sx, sy = math.fsum(a), math.fsum(b)
    sxx, syy, sxy = math.fsum(a * a), math.fsum(b * b), math.fsum(a * b)
    am2 = max(sxx - sx * sx / n, 0.0)
    bm2 = max(syy - sy * sy / n, 0.0)
    den = math.sqrt(am2 * bm2)
    if den == 0.0:
        pcc = 1.0 if float(d.max()) == 0.0 else 0.0
    else:
        pcc = (sxy - sx * sy / n) / den
    return {"pcc": pcc, "mae": math.fsum(d) / n, "atol": float(d.max())}


# --------------------------------------------------------------------------- #
# Tiling (tile_utils.py:91-132)
# --------------------------------------------------------------------------- #
def to_padded_2d(x: np.ndarray):
    """tile_utils.py:91-115: nd -> [prod(shape[:-1]), W]; 1-D -> rows of 32; pad to x32."""
    x = np.asarray(x, dtype=np.float32)
    if x.ndim == 0:
        d2, info = x.reshape(1, 1), ("scalar", x.shape)
    elif x.ndim == 1:
        n = x.shape[0]
        d2 = np.zeros((-(-n // TILE), TILE), dtype=np.float32)
        d2.reshape(-1)[:n] = x
        info = ("vector", n)
    else:
        d2, info = x.reshape(-1, x.shape[-1]), ("nd", x.shape)
    h, w = d2.shape
    hp, wp = -(-h // TILE) * TILE, -(-w // TILE) * TILE
    pad = np.zeros((hp, wp), dtype=np.float32)
    pad[:h, :w] = d2
    return pad, info, (h, w, hp, wp)


def tiles_from_padded(p: np.ndarray) -> np.ndarray:
    hp, wp = p.shape
    return p.reshape(hp // TILE, TILE, wp // TILE, TILE).transpose(0, 2, 1, 3).reshape(-1, TILE, TILE)


def from_tiles(tiles: np.ndarray, info, pad_info) -> np.ndarray:
    """tile_utils.py:118-132."""
    h, w, hp, wp = pad_info
    p = tiles.reshape(hp // TILE, wp // TILE, TILE, TILE).transpose(0, 2, 1, 3).reshape(hp, wp)
    d2 = p[:h, :w]
    if info[0] == "scalar":
        return np.array(d2[0, 0], dtype=np.float32)
    if info[0] == "vector":
        return d2.reshape(-1)[: info[1]].astype(np.float32)
    return d2.reshape(info[1]).astype(np.float32)


def total_bytes(counts: dict) -> float:
    """tile_utils.py:32-37 (dict insertion order matters for the float sum)."""
    t = 0.0
    for fmt, c in counts.items():
        t += float(c) * 1024.0 * BYTES_PER_ELEM.get(fmt, 0.0)
    return t


# --------------------------------------------------------------------------- #
# Per-tile statistic table (the quantities mixed_tile_greedy.py:135-220,245-254 sums)
# --------------------------------------------------------------------------- #
def _valid_views(pad_info, info, th, tw):
    """Yield per tile the list of (row_slice, col_slice) the greedy sums over
    (mixed_tile_greedy.py:103-131): the un-padded region, with the ragged last
    row of a 1-D input as its own view."""
    h, w, _hp, _wp = pad_info
    vec_partial_tr, vec_cols = -1, TILE
    if info[0] == "vector":
        last = int(info[1]) % TILE or TILE
        if last != TILE:
            vec_partial_tr, vec_cols = (h - 1) // TILE, last
    for tr in range(th):
        r_end = int(np.clip(h - tr * TILE, 0, TILE))
        for tc in range(tw):
            c_end = int(np.clip(w - tc * TILE, 0, TILE))
            if tr == vec_partial_tr:
                views = []
                if r_end - 1 > 0:
                    views.append((slice(0, r_end - 1), slice(0, c_end)))
                views.append((slice(r_end - 1, r_end), slice(0, vec_cols)))
                yield views
            else:
                yield [(slice(0, r_end), slice(0, c_end))]


def tile_stat_table(x: np.ndarray, formats=MIXED_FORMATS) -> dict:
    """float64 per-tile sums exactly as the greedy forms them: float32 products,
    ``np.sum(..., dtype=float64)`` over the valid view(s) of each 32x32 tile
    (NumPy pairwise order over the flattened view).

    Returns {"sx","sx2": [T]; fmt: {"sy","sy2","sxy","sabs","amax": [T]}; geometry}.
    """
    pad, info, pad_info = to_padded_2d(x)
    th, tw = pad_info[2] // TILE, pad_info[3] // TILE
    tx = tiles_from_padded(pad)
    nt = tx.shape[0]
    full = (pad_info[0] == pad_info[2]) and (pad_info[1] == pad_info[3]) and not (
        info[0] == "vector" and int(info[1]) % TILE)
    out = {"th": th, "tw": tw, "numel": int(np.asarray(x).size), "info": info, "pad_info": pad_info}
    views = None if full else list(_valid_views(pad_info, info, th, tw))

    def reduce_tiles(arr3: np.ndarray) -> np.ndarray:
        if full:
            return np_pairwise_sum(arr3.reshape(nt, -1).astype(np.float64))
        res = np.zeros(nt, dtype=np.float64)
        for t in range(nt):
            acc = 0.0
            for rs, cs in views[t]:
                acc += float(np.sum(arr3[t][rs, cs], dtype=np.float64))
            res[t] = acc
        return res

    def max_tiles(arr3: np.ndarray) -> np.ndarray:
        if full:
            return arr3.reshape(nt, -1).max(axis=1).astype(np.float64)
        res = np.zeros(nt, dtype=np.float64)
        for t in range(nt):
            m = 0.0
            for rs, cs in views[t]:
                v = arr3[t][rs, cs]
                lm = float(np.max(v)) if v.size else 0.0
                if lm > m or lm != lm:          # np.max over the views: a nan wins (Python's max(0.0, nan) is 0.0)
                    m = lm
            res[t] = m
        return res

    out["sx"] = reduce_tiles(tx)
    out["sx2"] = reduce_tiles(tx * tx)
    for fmt in formats:
        ty = quantize(tx, fmt)
        diff = np.abs(tx - ty)
        out[fmt] = {
            "sy": reduce_tiles(ty),
            "sy2": reduce_tiles(ty * ty),
            "sxy": reduce_tiles(tx * ty),
            "sabs": reduce_tiles(diff),
            "amax": max_tiles(diff),
        }
    return out


# --------------------------------------------------------------------------- #
# NumPy Generator(PCG64) stream (SURVEY.md Appendix B3) — pure Python, small n only
# --------------------------------------------------------------------------- #
_PCG_MULT = 0x2360ED051FC65DA44385DF649FCCF645
_M128 = (1 << 128) - 1
_M64 = (1 << 64) - 1


class Pcg64:
    """Continues a ``np.random.default_rng(seed)`` stream from its exported state."""

    def __init__(self, seed: int):
        st = np.random.default_rng(seed).bit_generator.state
        self.state = int(st["state"]["state"])
        self.inc = int(st["state"]["inc"])
        self.has32 = bool(st["has_uint32"])
        self.buf32 = int(st["uinteger"])

    def next64(self) -> int:
        self.state = (self.state * _PCG_MULT + self.inc) & _M128
        hi, lo = self.state >> 64, self.state & _M64
        x, rot = hi ^ lo, self.state >> 122
        return ((x >> rot) | (x << ((64 - rot) & 63))) & _M64

    def next32(self) -> int:
        if self.has32:
            self.has32 = False
            return self.buf32
        v = self.next64()
        self.has32, self.buf32 = True, v >> 32
        return v & 0xFFFFFFFF

    def interval(self, mx: int) -> int:
        if mx == 0:
            return 0
        mask = (1 << mx.bit_length()) - 1
        while True:
            v = self.next32() & mask
            if v <= mx:
                return v

    def permutation(self, n: int) -> np.ndarray:
        a = list(range(n))
        for i in range(n - 1, 0, -1):
            j = self.interval(i)
            a[i], a[j] = a[j], a[i]
        return np.asarray(a, dtype=np.int64)

    def integers(self, k: int, size: int) -> np.ndarray:
        """``integers(0, k, size, dtype=int64)``: Lemire's 32-bit method."""
        out = np.zeros(size, dtype=np.int64)
        if k <= 1:
            return out
        thr = ((1 << 32) - k) % k
        for i in range(size):
            m = self.next32() * k
            while (m & 0xFFFFFFFF) < thr:
                m = self.next32() * k
            out[i] = m >> 32
        return out


# --------------------------------------------------------------------------- #
# Assignment algorithms, table-driven
# --------------------------------------------------------------------------- #
def _pcc_from_sums(n, sx, sx2, sy, sy2, sxy, sabs) -> float:
    """mixed_tile_greedy.py:176-190, Python-float (f64) evaluation order."""
    if n == 0.0:
        return 1.0
    mx = sx / n
    my = sy / n
    am2 = sx2 - n * mx * mx
    bm2 = sy2 - n * my * my
    if am2 < 0.0:
        am2 = 0.0
    if bm2 < 0.0:
        bm2 = 0.0
    den = math.sqrt(am2 * bm2)
    if den == 0.0:
        return 1.0 if sabs == 0.0 else 0.0
    return (sxy - n * mx * my) / den


def greedy_assign(table: dict, tile_formats, metric: str, threshold: float, seed: int):
    """mixed_tile_greedy.py:72-352 driven by the per-tile table.

    Visits, per candidate format, the not-yet-fixed tiles in
    ``default_rng(seed).permutation`` order and accepts a tile's switch iff the
    global metric recomputed from running float64 sums still passes.
    Returns (assignment int8 [th,tw], counts dict).
    """
    nt = table["th"] * table["tw"]
    n = float(table["numel"])
    idx = {f: i for i, f in enumerate(MIXED_FORMATS)}
    base = tile_formats[0]
    assign = np.full(nt, idx[base], dtype=np.int8)
    fixed = np.zeros(nt, dtype=bool)
    counts = {f: 0 for f in MIXED_FORMATS}
    counts[base] = nt
    b = table[base]
    cur = {k: b[k].copy() for k in ("sy", "sy2", "sxy", "sabs", "amax")}
    sx = sx2 = sy = sy2 = sxy = sabs = 0.0
    for t in range(nt):                         # sequential f64 accumulation, tile order (:165-170)
        sx += float(table["sx"][t]); sx2 += float(table["sx2"][t])
        sy += float(cur["sy"][t]); sy2 += float(cur["sy2"][t])
        sxy += float(cur["sxy"][t]); sabs += float(cur["sabs"][t])
    if metric == "atol":
        max_abs = float(np.max(cur["amax"]))
        max_cnt = int(np.sum(cur["amax"] == max_abs))
    rng = np.random.default_rng(seed)
    for fmt in tile_formats:
        cand = np.where(~fixed)[0]
        if cand.size == 0:
            break
        order = rng.permutation(cand)
        f = table[fmt]
        fi = idx[fmt]
        for t in order:
            prev = int(assign[t])
            if metric == "pcc":
                if prev == fi:
                    if not is_good(_pcc_from_sums(n, sx, sx2, sy, sy2, sxy, sabs), metric, threshold):
                        fixed[t] = True
                    continue
                c_sy = sy + (float(f["sy"][t]) - float(cur["sy"][t]))
                c_sy2 = sy2 + (float(f["sy2"][t]) - float(cur["sy2"][t]))
                c_sxy = sxy + (float(f["sxy"][t]) - float(cur["sxy"][t]))
                c_sabs = sabs + (float(f["sabs"][t]) - float(cur["sabs"][t]))
                if is_good(_pcc_from_sums(n, sx, sx2, c_sy, c_sy2, c_sxy, c_sabs), metric, threshold):
                    sy, sy2, sxy, sabs = c_sy, c_sy2, c_sxy, c_sabs
                    for k in ("sy", "sy2", "sxy", "sabs"):
                        cur[k][t] = f[k][t]
                    counts[MIXED_FORMATS[prev]] -= 1
                    counts[fmt] += 1
                    assign[t] = fi
                else:
                    fixed[t] = True
            elif metric == "mae":
                if prev == fi:
                    if not is_good(sabs / n if n else 0.0, metric, threshold):
                        fixed[t] = True
                    continue
                c_sabs = sabs + (float(f["sabs"][t]) - float(cur["sabs"][t]))
                if is_good(c_sabs / n if n else 0.0, metric, threshold):
                    sabs = c_sabs
                    cur["sabs"][t] = f["sabs"][t]
                    counts[MIXED_FORMATS[prev]] -= 1
                    counts[fmt] += 1
                    assign[t] = fi
                else:
                    fixed[t] = True
            else:  # atol (:304-346): running max with multiplicity
                if prev == fi:
                    if not is_good(max_abs, metric, threshold):
                        fixed[t] = True
                    continue
                new_max, old_max = float(f["amax"][t]), float(cur["amax"][t])
                c_max, c_cnt = max_abs, max_cnt
                if new_max > max_abs:
                    c_max, c_cnt = new_max, 1
                elif new_max == max_abs:
                    if old_max != max_abs:
                        c_cnt = max_cnt + 1
                elif old_max == max_abs:
                    if max_cnt > 1:
                        c_cnt = max_cnt - 1
                    else:
                        upd = cur["amax"].copy()
                        upd[t] = new_max
                        c_max = float(np.max(upd))
                        c_cnt = int(np.sum(upd == c_max))
                if is_good(c_max, metric, threshold):
                    cur["amax"][t] = new_max
                    max_abs, max_cnt = c_max, c_cnt
                    counts[MIXED_FORMATS[prev]] -= 1
                    counts[fmt] += 1
                    assign[t] = fi
                else:
                    fixed[t] = True
    return assign.reshape(table["th"], table["tw"]), counts


def padded_tile_scores(x: np.ndarray, tile_formats, metric: str) -> dict:
    """Per-format float32 tile scores on zero-padded tiles (mixed_tile_threshold.py:97-109)."""
    pad, _info, _pi = to_padded_2d(x)
    tx = tiles_from_padded(pad)
    scores = {}
    for fmt in tile_formats:
        yq = quantize(np.asarray(x, dtype=np.float32), fmt)
        pq, _i2, _p2 = to_padded_2d(yq)
        scores[fmt] = tile_scores_f32(tx, tiles_from_padded(pq), metric)
    return scores


def threshold_assign(scores: dict, tile_formats, metric: str, threshold: float, th: int, tw: int):
    """mixed_tile_threshold.py:111-123: cheapest (ascending bytes, stable) passing format,
    else the max-bytes format.  float32 score vs Python-float threshold compares in float32."""
    idx = {f: i for i, f in enumerate(MIXED_FORMATS)}
    by_prec = sorted(tile_formats, key=lambda f: BYTES_PER_ELEM.get(f, 0.0))
    best = max(by_prec, key=lambda f: BYTES_PER_ELEM.get(f, 0.0))
    nt = th * tw
    assign = np.full(nt, idx[best], dtype=np.int8)
    done = np.zeros(nt, dtype=bool)
    thr32 = np.float32(threshold)
    for fmt in by_prec:
        s = scores[fmt].astype(np.float32)
        good = (s >= thr32) if metric == "pcc" else (s <= thr32)
        pick = good & ~done
        assign[pick] = idx[fmt]
        done |= pick
    counts = {f: 0 for f in MIXED_FORMATS}
    for fmt in tile_formats:
        counts[fmt] = int(np.sum(assign == idx[fmt]))
    return assign.reshape(th, tw), counts


def sweep_assign(scores: dict, tile_formats, metric: str, thresholds) -> np.ndarray:
    """scripts/sweep_mixed_tile_threshold.py:145-155: index into the ascending-bytes order,
    first passing format, last one forced.  Returns int8 [len(thr), T] of MIXED_FORMATS indices."""
    idx = {f: i for i, f in enumerate(MIXED_FORMATS)}
    by_prec = sorted(tile_formats, key=lambda f: BYTES_PER_ELEM.get(f, 0.0))
    stack = np.stack([scores[f].astype(np.float32) for f in by_prec], axis=0)
    out = []
    for thr in thresholds:
        good = (stack >= thr) if metric == "pcc" else (stack <= thr)
        good[-1, :] = True
        first = np.argmax(good, axis=0)
        out.append(np.asarray([idx[by_prec[i]] for i in first], dtype=np.int8))
    return np.stack(out, axis=0)


def apply_assignment(x: np.ndarray, assignment: np.ndarray) -> np.ndarray:
    """Gather per-tile reconstructions by assignment (mixed_tile_threshold.py:125-130)."""
    pad, info, pad_info = to_padded_2d(x)
    tx = tiles_from_padded(pad)
    out = tx.copy()
    flat = np.asarray(assignment).reshape(-1)
    for i, fmt in enumerate(MIXED_FORMATS):
        ids = np.where(flat == i)[0]
        if ids.size:
            out[ids] = quantize(tx[ids], fmt)
    return from_tiles(out, info, pad_info)


def random_assign(x: np.ndarray, tile_formats, metric: str, threshold: float, iters: int, seed: int):
    """mixed_tile_random.py:88-183 with float32 whole-tensor metrics per sample.

    Returns (best assignment [th,tw] int8, counts, samples list)."""
    x = np.asarray(x, dtype=np.float32)
    pad, info, pad_info = to_padded_2d(x)
    th, tw = pad_info[2] // TILE, pad_info[3] // TILE
    tx = tiles_from_padded(pad)
    nt = tx.shape[0]
    fidx = np.asarray([MIXED_FORMATS.index(f) for f in tile_formats], dtype=np.int8)
    per_fmt = {i: quantize(tx, MIXED_FORMATS[i]) for i in set(int(v) for v in fidx)}
    bpe32 = np.asarray([BYTES_PER_ELEM[f] for f in MIXED_FORMATS], dtype=np.float32)
    rng = np.random.default_rng(seed)
    best_bytes = best_metric = best_assign = None
    samples = []
    for sid in range(max(1, iters)):
        choice = rng.integers(0, len(fidx), size=nt, dtype=np.int64)
        a = fidx[choice].astype(np.int8)
        tq = tx.copy()
        for i, arr in per_fmt.items():
            ids = np.where(a == i)[0]
            if ids.size:
                tq[ids] = arr[ids]
        y = from_tiles(tq, info, pad_info)
        score = metric_f32(x, y, metric)
        diff = np.abs(x - y)
        mae, atol, pcc = float(np.mean(diff)), float(np.max(diff)), pearson_f32(x, y)
        carr = np.bincount(a.astype(np.int64), minlength=len(MIXED_FORMATS))
        counts = {f: int(carr[i]) for i, f in enumerate(MIXED_FORMATS)}
        samples.append({"id": sid, "counts": counts, "total_bytes": total_bytes(counts),
                        "pcc": pcc, "mae": mae, "atol": atol})
        if is_good(score, metric, threshold):
            tb = float(np.sum(carr * bpe32) * (TILE * TILE))
            if best_bytes is None or tb < best_bytes:
                best_bytes, best_metric, best_assign = tb, score, a.copy()
        elif best_bytes is None:
            if best_metric is None or is_better(score, best_metric, metric):
                best_metric, best_assign = score, a.copy()
    counts = {f: int(np.sum(best_assign == i)) for i, f in enumerate(MIXED_FORMATS)}
    return best_assign.reshape(th, tw), counts, samples


def random_samples_exact(table: dict, tile_formats, iters: int, seed: int):
    """Table-driven fp64 evaluation of every random sample's whole-tensor
    pcc/mae/atol (what the GPU's exact path reports).  Returns (choices [iters,T] int8,
    metrics [iters,3] f64)."""
    nt = table["th"] * table["tw"]
    n = float(table["numel"])
    fidx = np.asarray([MIXED_FORMATS.index(f) for f in tile_formats], dtype=np.int8)
    rng = np.random.default_rng(seed)
    sx, sx2 = math.fsum(table["sx"]), math.fsum(table["sx2"])
    stack = {k: np.stack([table[f][k] for f in MIXED_FORMATS], axis=0) for k in ("sy", "sy2", "sxy", "sabs", "amax")}
    ar = np.arange(nt)
    ch, met = [], []
    for _ in range(iters):
        a = fidx[rng.integers(0, len(fidx), size=nt, dtype=np.int64)].astype(np.int8)
        sy, sy2 = math.fsum(stack["sy"][a, ar]), math.fsum(stack["sy2"][a, ar])
        sxy, sabs = math.fsum(stack["sxy"][a, ar]), math.fsum(stack["sabs"][a, ar])
        amax = float(stack["amax"][a, ar].max())
        am2, bm2 = max(sx2 - sx * sx / n, 0.0), max(sy2 - sy * sy / n, 0.0)
        den = math.sqrt(am2 * bm2)
        pcc = (1.0 if amax == 0.0 else 0.0) if den == 0.0 else (sxy - sx * sy / n) / den
        ch.append(a)
        met.append((pcc, sabs / n, amax))
    return np.stack(ch, axis=0), np.asarray(met, dtype=np.float64)


def wq_scores(x: np.ndarray, y: np.ndarray) -> dict:
    """wq:684-687 — float32 whole-tensor mae / atol / pcc exactly as NumPy evaluates them."""
    x = np.asarray(x, dtype=np.float32)
    y = np.asarray(y, dtype=np.float32)
    diff = np.abs(x - y)
    return {"mae": float(np.mean(diff)), "atol": float(np.max(diff)), "pcc": pearson_f32(x, y)}


# --------------------------------------------------------------------------- #
# fp8 e4m3fn block dequantization (hf_model_utils.py:199-215, used at :266-281): the step in front of the path
# --------------------------------------------------------------------------- #
def fp8_e4m3fn_table() -> np.ndarray:
    """float32 value of each of the 256 e4m3fn bit patterns (bias 7, no inf, 0x7f / 0xff = nan)."""
    out = np.zeros(256, dtype=np.float32)
    for b in range(256):
        sgn = -1.0 if b & 0x80 else 1.0
        e, m = (b >> 3) & 0xF, b & 7
        if e == 15 and m == 7:
            v = np.nan
        elif e == 0:
            v = sgn * m * 2.0 ** -9
        else:
            v = sgn * (1.0 + m / 8.0) * 2.0 ** (e - 7)
        out[b] = v
    out[0x80] = -0.0
    return out


def fp8_block_dequant(w_bits: np.ndarray, scale_inv: np.ndarray) -> np.ndarray:
    """tensor.float() * inv_scale.repeat_interleave(block)[:rows, :cols] with block = ceil(shape / scale shape), float32."""
    w = np.asarray(w_bits, dtype=np.uint8)
    sc = np.asarray(scale_inv, dtype=np.float32)
    assert w.ndim == 2 and sc.ndim == 2
    br = max(1, -(-w.shape[0] // sc.shape[0])) if sc.shape[0] > 0 else 1
    bc = max(1, -(-w.shape[1] // sc.shape[1])) if sc.shape[1] > 0 else 1
    full = np.repeat(np.repeat(sc, br, axis=0), bc, axis=1)[: w.shape[0], : w.shape[1]]
    with np.errstate(all="ignore"):
        return (fp8_e4m3fn_table()[w] * full).astype(np.float32)
