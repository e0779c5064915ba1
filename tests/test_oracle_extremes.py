"""CPU: the oracle's float32 arithmetic restatements at the ends of the float32 range and on inf / NaN.

_fma_f32 is held to an exact reference (fractions.Fraction, rounded to float32 by hand; the IEEE rules for inf and NaN
operands).  np_pairwise_sum, np_sdot_f32 and pearson_f32_rows are held to NumPy itself on vectors that contain +-inf,
NaN, denormals and values near FLT_MAX: NaN positions must match, every other value bit for bit.
"""
import itertools
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import qa_oracle as orc

FLT_MAX = float(np.finfo(np.float32).max)
DENORM_MIN = 2.0 ** -149


def _openblas_is_skylakex():
    from threadpoolctl import threadpool_info
    arch = {d.get("architecture") for d in threadpool_info() if d.get("internal_api") == "openblas"}
    return not arch or arch == {"SkylakeX"}


def _round_f32(q: Fraction) -> float:
    """q rounded to the nearest float32 (ties to even), as a Python float; overflow gives +-inf."""
    if q == 0:
        return 0.0
    neg, v = q < 0, abs(q)
    e = v.numerator.bit_length() - v.denominator.bit_length()
    if Fraction(2) ** e > v:
        e -= 1                                            # now 2^e <= v < 2^(e+1)
    ulp = Fraction(2) ** (max(e, -126) - 23)
    m = v / ulp
    n = m.numerator // m.denominator
    rem = m - n
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and n % 2 == 1):
        n += 1
    r = n * ulp
    out = math.inf if r >= Fraction(2) ** 128 else float(r)
    return -out if neg else out


def _fma_ref(a: float, b: float, c: float) -> float:
    """IEEE 754 fusedMultiplyAdd on float32 operands, rounded to nearest even."""
    if math.isnan(a) or math.isnan(b) or math.isnan(c):
        return math.nan
    if math.isinf(a) or math.isinf(b):
        if a == 0.0 or b == 0.0:
            return math.nan                               # inf * 0
        p = math.copysign(math.inf, a) * math.copysign(1.0, b)
        if math.isinf(c) and c != p:
            return math.nan                               # inf - inf
        return p
    if math.isinf(c):
        return c
    p, q = Fraction(a) * Fraction(b), Fraction(a) * Fraction(b) + Fraction(c)
    if q == 0:
        # an exact zero: -0 only when both addends are zeros of negative sign (round to nearest)
        p_neg = p == 0 and (math.copysign(1.0, a) * math.copysign(1.0, b)) < 0
        return -0.0 if p == 0 and c == 0 and p_neg and math.copysign(1.0, c) < 0 else 0.0
    return _round_f32(q)


# operands: signed zeros, denormals, the normal boundary, near-ties around 1, large values, FLT_MAX, +-inf, NaN
_GRID = [0.0, -0.0, DENORM_MIN, -3 * DENORM_MIN, 2.0 ** -127, 2.0 ** -126, -(2.0 ** -100), 2.0 ** -30, 2.0 ** -24,
         1.0, -1.0, 1.0 + 2.0 ** -12, 1.0 - 2.0 ** -12, 1.0 + 2.0 ** -23, 3.0, -5.0, 2.0 ** 64, -(2.0 ** 100),
         FLT_MAX, -FLT_MAX, math.inf, -math.inf, math.nan]


def test_fma_f32_matches_exact_reference():
    """Every triple of the grid: products that overflow to inf, sums that cancel FLT_MAX, denormal results, results
    exactly half-way between two float32 values ((1 + 2^-12)^2 = 1 + 2^-11 + 2^-24), and every inf / NaN rule."""
    trip = np.asarray(list(itertools.product(_GRID, repeat=3)), dtype=np.float32)
    with np.errstate(all="ignore"):
        got = orc._fma_f32(trip[:, 0], trip[:, 1], trip[:, 2])
    want = np.asarray([_fma_ref(float(a), float(b), float(c)) for a, b, c in trip], dtype=np.float32)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    bad = np.nonzero(got[~nan].view(np.uint32) != want[~nan].view(np.uint32))[0]
    assert bad.size == 0, [tuple(trip[~nan][i]) for i in bad[:5]]


def test_fma_f32_infinite_cases():
    """The cases a round-to-odd fix-up on a non-finite float64 sum turned into NaN."""
    f = np.float32
    with np.errstate(all="ignore"):
        assert orc._fma_f32(np.array(f(1)), np.array(f(1)), np.array(f(-np.inf))) == -np.inf
        assert orc._fma_f32(np.array(f(-np.inf)), np.array(f(1)), np.array(f(0))) == -np.inf
        assert orc._fma_f32(np.array(f(np.inf)), np.array(f(-1)), np.array(f(5))) == -np.inf
        assert orc._fma_f32(np.array(f(FLT_MAX)), np.array(f(2)), np.array(f(0))) == np.inf
        assert orc._fma_f32(np.array(f(FLT_MAX)), np.array(f(2)), np.array(f(-FLT_MAX))) == f(FLT_MAX)


def _extreme_rows(n, seed):
    """Rows of length n: a normal-range background with, per row, one kind of extreme value placed at seeded positions."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((12, n)).astype(np.float32)
    rows = base.copy()
    pos = rng.integers(0, n, (12, 3))
    rows[0, pos[0, 0]] = np.inf
    rows[1, pos[1, 0]] = -np.inf
    rows[2, pos[2, 0]] = np.nan
    rows[3, pos[3, :2]] = (np.inf, -np.inf)
    rows[4] = (rng.standard_normal(n) * 2.0 ** -135).astype(np.float32)                      # denormals only
    rows[5] = (rng.standard_normal(n) * 2.0 ** -135).astype(np.float32)
    rows[5, pos[5, 0]] = 1.0                                                                # denormals and a normal
    rows[6] = np.float32(FLT_MAX) * np.where(rng.random(n) < 0.5, 1, -1).astype(np.float32)  # sums overflow, squares too
    rows[7] = np.float32(2.0 ** 120) * rng.random(n).astype(np.float32)
    rows[8, pos[8, 0]] = np.float32(FLT_MAX)
    rows[9] = -np.abs(rows[9]) * np.float32(2.0 ** 100)
    rows[9, pos[9, 0]] = -np.inf                                                            # -inf among large negatives
    rows[10] = (rng.standard_normal(n) * 2.0 ** -70).astype(np.float32)                     # squares underflow
    rows[11, pos[11, 0]] = np.float32(DENORM_MIN)
    return rows


@pytest.mark.parametrize("n", [5, 100, 1024, 1000, 3001])
def test_pairwise_sum_on_extremes(n):
    x = _extreme_rows(n, 11 + n)
    with np.errstate(all="ignore"):
        got, want = orc.np_pairwise_sum(x), np.add.reduce(x, axis=1)
    assert np.array_equal(got, want, equal_nan=True)
    assert np.array_equal(got[~np.isnan(got)].view(np.uint32), want[~np.isnan(want)].view(np.uint32))


@pytest.mark.parametrize("n", [31, 64, 100, 1024, 3001])
def test_sdot_and_pearson_on_extremes(n):
    """np_sdot_f32 against np.dot (x.x and x.y, y another extreme row set), pearson_f32_rows against pearson_f32 (np.mean,
    np.linalg.norm, np.dot) for [N, 1024] rows.  Only where np.dot runs OpenBLAS's SkylakeX sdot, whose order is restated."""
    if not _openblas_is_skylakex():
        pytest.skip("np.dot uses a different OpenBLAS kernel here")
    x = _extreme_rows(n, 101 + n)
    y = np.roll(_extreme_rows(n, 202 + n), 3, axis=0)
    with np.errstate(all="ignore"):
        for a, b in ((x, x), (x, y)):
            got = orc.np_sdot_f32(a, b)
            want = np.array([np.dot(a[i], b[i]) for i in range(a.shape[0])], dtype=np.float32)
            assert np.array_equal(got, want, equal_nan=True), (got, want)
        if n == 1024:
            for b in (x, y, orc.bf16_round(x)):
                got = orc.pearson_f32_rows(x, b)
                want = np.array([orc.pearson_f32(x[i], b[i]) for i in range(x.shape[0])], dtype=np.float32)
                assert np.array_equal(got, want, equal_nan=True), (got, want)
