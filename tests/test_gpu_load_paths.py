"""Every load path of the whole-tensor scorer (qa_tensor_scores_f32) and of the row kernels, against the oracle.

The scorer picks its kernels from n, from the alignment of both base pointers and of the row stride, and from the batch size:
the TMA ring of sdot_pipe_kernel (n >= 16384, 32-byte aligned operands; 8 / 6 stages, 3 from 74 items, 2 from 296), the
vector leaves + sdot_kernel (aligned, shorter), and the scalar leaves + sdot_kernel (anything unaligned).  Each path is run
at the n that reach its tails (leftover chain steps after the last full stage, the odd 32-block, the double-accumulated
n % 32 tail), with padded and poisoned row strides, and compared bit for bit with the oracle's restated NumPy / OpenBLAS
orders, column 3 (mean of y) included.  Batches over 65535 items (CUDA's gridDim.y limit) go through the scorer, the
threshold assignment, the random search and the sweep.

The row kernels take a leading dimension and choose a vector or a scalar path from cols % 16, ld % 16 and the base
address: each is called through the C ABI on a matrix placed at row strides ld > cols and at offset base pointers, with
every byte outside the matrix poisoned, and must give the oracle's bits (or, where the contiguous table is already pinned
to the oracle by test_gpu_parity.py, the contiguous call's bits)."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc

pytestmark = pytest.mark.gpu

MIXED = list(orc.MIXED_FORMATS)
BIG = 65536                    # one past CUDA's gridDim.y limit of 65535
DT = {"bf16": torch.bfloat16, "f32": torch.float32}


@pytest.fixture(scope="module")
def qa():
    from quantization_analysis_b200 import _lib, engine, sweep
    from quantization_analysis_b200 import compression_algorithms as ca
    return SimpleNamespace(L=_lib.lib(), lib=_lib, eng=engine, ca=ca, sweep=sweep)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _code(t):
    return 0 if t.dtype == torch.bfloat16 else 1


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


# --------------------------------------------------------------------------------------------------------------------------
# whole-tensor scorer
# --------------------------------------------------------------------------------------------------------------------------
POISON = (np.nan, 3e38, -3e38)


def _poisoned(n_alloc, dtype):
    """Device buffer of n_alloc elements cycling through NaN, +3e38, -3e38."""
    v = np.resize(np.asarray(POISON, np.float32), n_alloc)
    return torch.from_numpy(v).cuda().to(dtype)


def _vals(rng, n, dtype):
    """float32 values of n elements, exactly representable in `dtype`."""
    x = (rng.standard_normal(n) * 0.02).astype(np.float32)
    if dtype == "bf16":
        x = torch.from_numpy(x).to(torch.bfloat16).float().numpy()
    return x


def _candidate(x32, k, dtype, rng):
    """The k-th distinct candidate reconstruction of x, exactly representable in `dtype`."""
    if dtype == "bf16":
        return orc.quantize(x32.reshape(1, -1), MIXED[k % 4]).reshape(-1)
    return (x32 + rng.standard_normal(x32.size).astype(np.float32) * np.float32(1e-3 * (k + 1))).astype(np.float32)


def _score(qa, x, y, n, stride=0, nb=1):
    """qa_tensor_scores_f32 on raw views: x, y are device tensors whose data_ptr() is the first element (y None: fp0);
    y holds nb rows `stride` elements apart."""
    host, plan = qa.eng._plan(n, x.device)
    out = torch.empty((nb, 4), dtype=torch.float32, device=x.device)
    work = torch.empty(qa.L.qa_tensor_scores_work_bytes(int(host[2]), nb), dtype=torch.uint8, device=x.device)
    qa.lib.check(qa.L.qa_tensor_scores_f32(x.data_ptr(), _code(x), None if y is None else y.data_ptr(),
                                           1 if y is None else _code(y), stride, nb, n, plan.data_ptr(), host.ctypes.data,
                                           out.data_ptr(), work.data_ptr(), _stream()), "qa_tensor_scores_f32")
    return out.cpu().numpy()


def _want(x32, y32):
    """{pcc, mae, atol, mean(y)} in the reference's float32 orders; y32 None = fp0."""
    n = x32.size
    with np.errstate(all="ignore"):
        w = orc.wq_scores_restated(x32, np.zeros_like(x32) if y32 is None else y32)
        mean = np.float32(0.0) if y32 is None else np.float32(orc.np_pairwise_sum(y32) / np.float32(n))
    return np.array([w["pcc"], w["mae"], w["atol"], mean], dtype=np.float32)


def _same(got, want, tag):
    """Bit equality of the float32 patterns; a NaN matches any NaN (the device and NumPy may carry different payloads)."""
    g, w = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert g.shape == w.shape, tag
    nan = np.isnan(w)
    assert np.array_equal(np.isnan(g), nan), (tag, g, w)
    assert np.array_equal(_bits(g)[~nan], _bits(w)[~nan]), (tag, g, w)


def _layout(x32, ys32, xdt, ydt, x_shift=0, y_shift=0, m=None):
    """Device operands with poison around them: x at element x_shift of a buffer, the rows of ys32 at y_shift + i * m.
    -> (x view, y view or None, stride m)."""
    n = x32.size
    xb = _poisoned(x_shift + n + 64, DT[xdt])
    xb[x_shift:x_shift + n] = torch.from_numpy(x32).cuda().to(DT[xdt])
    if ys32 is None:
        return xb[x_shift:], None, 0
    nb = ys32.shape[0]
    m = m or -(-(n + 1) // 16) * 16             # padded and 32-byte aligned for both dtypes
    yb = _poisoned(y_shift + nb * m + 64, DT[ydt])
    rows = yb[y_shift:y_shift + nb * m].view(nb, m)
    rows[:, :n] = torch.from_numpy(ys32).cuda().to(DT[ydt])
    return xb[x_shift:], yb[y_shift:], m


DTYPES = [(a, b) for a in ("bf16", "f32") for b in ("bf16", "f32", None)]
PIPE_N = [
    16384,                          # exactly 4 stages
    16384 + 64,                     # one leftover chain step
    16384 + 64 * 63 + 32 + 31,      # 63 leftover steps, the 32-block and a 31-element tail
    16384 + 32,                     # the 32-block alone
    16384 + 17,                     # a tail alone
    4096 * 19 + 64 * 7 + 32 + 5,    # 19 stages: an 8- (6-) stage ring wraps twice
    16383,                          # just below the pipeline
]


@pytest.mark.parametrize("xdt,ydt", DTYPES)
def test_scorer_pipelined_tails(qa, xdt, ydt):
    """Aligned operands, y rows at a padded stride (m * sizeof(y) % 32 == 0): the TMA ring for n >= 16384 whatever n % 32,
    the vector path just below; every padding element is NaN or +-3e38."""
    for n in PIPE_N:
        rng = np.random.default_rng(n)
        x32 = _vals(rng, n, xdt)
        y32 = None if ydt is None else _candidate(x32, 2, ydt, rng)
        x, y, m = _layout(x32, None if y32 is None else y32[None], xdt, ydt)
        _same(_score(qa, x, y, n, m)[0], _want(x32, y32), (xdt, ydt, n))


_ORACLE_CACHE: dict = {}


@pytest.mark.parametrize("nb", [74, 296])
@pytest.mark.parametrize("xdt,ydt", [("bf16", "bf16"), ("f32", "f32"), ("bf16", "f32")])
def test_scorer_ring_depths(qa, xdt, ydt, nb):
    """Batches that shrink the ring to 3 (74 items) and 2 (296 items) stages, at a wrapping n with every tail; the rows
    cycle through three distinct candidates and every row is checked."""
    n = 4096 * 19 + 64 * 7 + 32 + 5
    rng = np.random.default_rng(3)
    x32 = _vals(rng, n, xdt)
    cands = np.stack([_candidate(x32, k, ydt, rng) for k in range(3)])
    key = (xdt, ydt)
    if key not in _ORACLE_CACHE:
        _ORACLE_CACHE[key] = [_want(x32, c) for c in cands]
    want = _ORACLE_CACHE[key]
    idx = np.arange(nb) % 3
    x, y, m = _layout(x32, cands[idx], xdt, ydt)
    got = _score(qa, x, y, n, m, nb)
    for b in range(nb):
        _same(got[b], want[idx[b]], (xdt, ydt, nb, b))


@pytest.mark.parametrize("n", [1000, 16384 + 64 * 63 + 32 + 31])
@pytest.mark.parametrize("xdt,ydt", DTYPES)
def test_scorer_unaligned(qa, xdt, ydt, n):
    """The scalar path: x one element off an aligned base, y rows one element off, a row stride that is not a multiple of
    32 bytes, and at a pipelined-size n the same tails as the ring."""
    rng = np.random.default_rng(n + 7)
    x32 = _vals(rng, n, xdt)
    ys32 = None if ydt is None else np.stack([_candidate(x32, k, ydt, rng) for k in range(2)])
    want = [_want(x32, None if ys32 is None else ys32[k]) for k in range(1 if ys32 is None else 2)]
    variants = [(1, 0, None)] + ([] if ydt is None else [(0, 1, None), (1, 1, None), (0, 0, n + 1)])
    for xs, ys, m in variants:
        x, y, stride = _layout(x32, ys32, xdt, ydt, xs, ys, m)
        got = _score(qa, x, y, n, stride, len(want))
        for k, w in enumerate(want):
            _same(got[k], w, (xdt, ydt, n, xs, ys, m, k))


@pytest.mark.parametrize("aligned", [True, False])
def test_scorer_nan_inside_propagates(qa, aligned):
    """Poison beyond n changes nothing (the other tests); a NaN inside the first n elements propagates as NumPy does."""
    n = 16384 + 64 * 63 + 32 + 31
    rng = np.random.default_rng(19)
    for where in ("x", "y"):
        for xdt, ydt in (("bf16", "bf16"), ("f32", "f32")):
            x32 = _vals(rng, n, xdt)
            y32 = _candidate(x32, 1, ydt, rng)
            (x32 if where == "x" else y32)[n // 3] = np.nan
            sh = 0 if aligned else 1
            x, y, m = _layout(x32, y32[None], xdt, ydt, sh, sh)
            _same(_score(qa, x, y, n, m)[0], _want(x32, y32), (where, xdt, aligned))


@pytest.mark.parametrize("path", ["short", "unaligned", "pipelined"])
def test_scorer_batch_over_65535(qa, path):
    """65543 candidate rows in one call: the leaf and chain kernels are launched over batch ranges of at most 65535."""
    n = 16401 if path == "pipelined" else 100
    nb = BIG + 7
    rng = np.random.default_rng(nb)
    x32 = _vals(rng, n, "bf16")
    cands = np.stack([_candidate(x32, k, "bf16", rng) for k in range(4)])
    want = [_want(x32, c) for c in cands]
    m = -(-(n + 1) // 16) * 16
    sh = 1 if path == "unaligned" else 0
    x = torch.from_numpy(x32).cuda().to(torch.bfloat16)
    cd = torch.full((4, m), float("nan"), device="cuda", dtype=torch.bfloat16)
    cd[:, :n] = torch.from_numpy(cands).cuda().to(torch.bfloat16)
    idx = (np.arange(nb) * 7 // 3) % 4
    yb = torch.empty(nb * m + sh, dtype=torch.bfloat16, device="cuda")
    yb[sh:].view(nb, m).copy_(cd[torch.from_numpy(idx).cuda()])
    got = _score(qa, x, yb[sh:], n, m, nb)
    for b in (0, BIG - 2, BIG - 1, BIG, nb - 1):
        _same(got[b], want[idx[b]], (path, b))
    wb = np.stack(want)[idx]
    assert np.array_equal(_bits(got), _bits(wb)), path


def test_threshold_sweep_over_65535_steps(qa):
    """sweep_tensor with 65573 thresholds: one qa_threshold_assign call; every row's map and counts are the oracle's."""
    rng = np.random.default_rng(8)
    x = (rng.standard_normal((96, 160)) * 0.02).astype(np.float32)
    steps = BIG + 37
    rows, maps = qa.sweep.sweep_tensor(x, MIXED, "pcc", steps=steps, lowest=0.9)
    sc = orc.padded_tile_scores(x, MIXED, "pcc")
    thr = np.linspace(float(np.max(sc["bf16"])), 0.9, steps)
    assert [r["threshold"] for r in rows] == [float(t) for t in thr]
    maps = maps.cpu().numpy()
    assert maps.shape == (steps, 15)
    prev = None
    for i in range(steps):
        a, counts = orc.threshold_assign(sc, MIXED, "pcc", float(thr[i]), 3, 5)
        assert np.array_equal(maps[i], a.reshape(-1)), i
        assert rows[i]["counts"] == counts, i
        if prev is None or not np.array_equal(a, prev):
            w = orc.wq_scores_restated(x, orc.apply_assignment(x, a))
            assert all(rows[i][k] == w[k] for k in ("pcc", "mae", "atol")), i
        prev = a


def test_random_search_over_65535_samples(qa):
    """mixed-tile-random with 65636 samples on 4 tiles: the draws are NumPy's, every sample's float32 scores are the oracle's
    for its map (all of them scored in one qa_tensor_scores_f32 call), and the selection is the reference's."""
    eng = qa.eng
    rng = np.random.default_rng(2)
    x = torch.from_numpy((rng.standard_normal((64, 64)) * 0.02).astype(np.float32)).to(torch.bfloat16).float().numpy()
    iters, seed, thr = BIG + 100, 11, 0.999
    want_draws = np.random.default_rng(seed)
    draws = np.stack([want_draws.integers(0, 4, size=4, dtype=np.int64) for _ in range(iters)]).astype(np.int8)
    p = eng.prepare_tiles(x)
    choices, _, _ = eng.random_samples(eng.tile_stats(p, MIXED), p.numel, MIXED, iters, eng.make_rng(seed, p.data.device))
    assert np.array_equal(choices.cpu().numpy(), draws)
    algo = qa.ca.create_algorithm("mixed-tile-random", {"metric": "pcc", "threshold": thr, "iters": iters, "seed": seed})
    dr = algo.run_prepared(p, MIXED)
    samples = dr.meta["samples"]
    assert len(samples) == iters
    keys = draws.astype(np.int64) @ np.array([64, 16, 4, 1])
    scores = {}
    for k in np.unique(keys):
        a = draws[np.argmax(keys == k)].reshape(2, 2)
        w = orc.wq_scores_restated(x, orc.apply_assignment(x, a))
        scores[int(k)] = np.array([w["pcc"], w["mae"], w["atol"]], dtype=np.float32)
    got = np.array([[s["pcc"], s["mae"], s["atol"]] for s in samples], dtype=np.float32)
    want = np.stack([scores[int(k)] for k in keys])
    assert np.array_equal(_bits(got), _bits(want))
    # mixed_tile_random.py:149-160: smallest bytes among passing samples (first wins ties), else strictly best pcc
    bpe32 = np.asarray([orc.BYTES_PER_ELEM[f] for f in MIXED], dtype=np.float32)
    best_id = best_bytes = best_metric = None
    npass = 0
    for sid in range(iters):
        carr = np.bincount(draws[sid].astype(np.int64), minlength=4)
        assert samples[sid]["counts"] == {f: int(carr[i]) for i, f in enumerate(MIXED)}, sid
        score = float(want[sid, 0])
        if orc.is_good(score, "pcc", thr):
            npass += 1
            tb = float(np.sum(carr * bpe32) * 1024)
            if best_bytes is None or tb < best_bytes:
                best_bytes, best_metric, best_id = tb, score, sid
        elif best_bytes is None and (best_metric is None or orc.is_better(score, best_metric, "pcc")):
            best_metric, best_id = score, sid
    assert 0 < npass < iters
    assert dr.meta["best_id"] == best_id
    assert np.array_equal(dr.assignment_numpy().reshape(-1), draws[best_id])


# --------------------------------------------------------------------------------------------------------------------------
# row kernels: leading dimension and base offset
# --------------------------------------------------------------------------------------------------------------------------
SHAPES = [(64, 512), (70, 530), (33, 1040), (1, 16)]
LD_EXTRA = [0, 1, 16, 37]
ITEM = {torch.bfloat16: 2, torch.float32: 4, torch.uint8: 1}


def _place(m, dtype, ld, off, poison):
    """The logical matrix m ([rows, cols] float32, or uint8 bytes) at element off + r * ld + c of a device buffer whose every
    other element is `poison`.  -> (buffer, pointer to the first element)."""
    rows, cols = m.shape
    total = off + (rows - 1) * ld + cols + 64
    if dtype == torch.uint8:
        buf = torch.full((total,), poison, dtype=torch.uint8, device="cuda")
        src = torch.from_numpy(np.ascontiguousarray(m)).cuda()
    else:
        buf = torch.full((total,), poison, dtype=torch.float32, device="cuda").to(dtype)
        src = torch.from_numpy(np.ascontiguousarray(m, dtype=np.float32)).cuda().to(dtype)
    torch.as_strided(buf, (rows, cols), (ld, 1), off).copy_(src)
    return buf, buf.data_ptr() + off * ITEM[dtype]


def _layouts(cols, dtype):
    """(ld, offset, poison) for every leading dimension x {0, 1 element, 32 bytes}; poison alternates between a NaN and a
    large finite value (for e4m3 bytes: 0x7F = NaN, 0x7E = 448)."""
    poisons = (0x7F, 0x7E) if dtype == torch.uint8 else (float("nan"), 3e38)
    out = []
    for i, extra in enumerate(LD_EXTRA):
        for j, off in enumerate((0, 1, 32 // ITEM[dtype])):
            out.append((cols + extra, off, poisons[(i + j) % 2]))
    return out


def _matrix(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * 0.02 * np.exp2(rng.integers(-6, 6, (shape[0], 1)))).astype(np.float32)
    if dtype == "bf16":
        x = torch.from_numpy(x).to(torch.bfloat16).float().numpy()
    return x


def _out_bufs(n, shift):
    """Four bf16 outputs of n elements; `shift` = 1 offsets the bfp4 one by 2 bytes (forces the scalar path)."""
    bufs = [torch.empty(n + 1, dtype=torch.bfloat16, device="cuda") for _ in range(4)]
    views = [b[shift:shift + n] if f == 2 else b[:n] for f, b in enumerate(bufs)]
    return bufs, views


def _ptr_array(views):
    import ctypes as C
    arr = (C.c_void_p * 4)()
    for i, v in enumerate(views):
        arr[i] = v.data_ptr()
    return arr


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("xdt", ["bf16", "f32"])
def test_quant_recon_strided(qa, shape, xdt):
    """qa_quant_recon and qa_quant_recon_cols: bits of orc.quantize of the logical matrix (for the column form, of its
    transpose, transposed back), at every layout, with every output aligned and with one output 2 bytes off."""
    rows, cols = shape
    x = _matrix(shape, xdt, rows * cols)
    want = {f: orc.quantize(x, f) for f in MIXED}
    want_c = {f: orc.quantize(np.ascontiguousarray(x.T), f).T for f in MIXED}
    for ld, off, poison in _layouts(cols, DT[xdt]):
        _buf, ptr = _place(x, DT[xdt], ld, off, poison)
        for shift in (0, 1):
            for fn, w in (("qa_quant_recon", want), ("qa_quant_recon_cols", want_c)):
                _bufs, views = _out_bufs(rows * cols, shift)
                qa.lib.check(getattr(qa.L, fn)(ptr, _code(_buf), rows, cols, ld, 0xF, _ptr_array(views), _stream()), fn)
                for f, v in zip(MIXED, views):
                    got = v.float().cpu().numpy().reshape(rows, cols)
                    assert np.array_equal(_bits(got), _bits(w[f])), (fn, xdt, shape, ld, off, shift, f)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("xdt", ["bf16", "f32"])
def test_apply_assignment_strided(qa, shape, xdt):
    """qa_apply_assignment: bits of orc.apply_assignment at every layout, output aligned and 2 bytes off."""
    rows, cols = shape
    x = _matrix(shape, xdt, rows + cols)
    th, tw = -(-rows // 32), -(-cols // 32)
    a = np.random.default_rng(rows * 7 + cols).integers(0, 4, th * tw).astype(np.int8)
    want = orc.apply_assignment(x, a.reshape(th, tw))
    ad = torch.from_numpy(a).cuda()
    for ld, off, poison in _layouts(cols, DT[xdt]):
        _buf, ptr = _place(x, DT[xdt], ld, off, poison)
        for shift in (0, 1):
            ob = torch.empty(rows * cols + 1, dtype=torch.bfloat16, device="cuda")
            out = ob[shift:shift + rows * cols]
            qa.lib.check(qa.L.qa_apply_assignment(ptr, _code(_buf), rows, cols, ld, ad.data_ptr(), out.data_ptr(), _stream()),
                         "qa_apply_assignment")
            got = out.float().cpu().numpy().reshape(rows, cols)
            assert np.array_equal(_bits(got), _bits(want)), (xdt, shape, ld, off, shift)


def _table_dict(t):
    tb = t.cpu().numpy()
    out = {"sx": tb[0], "sx2": tb[1]}
    for i, f in enumerate(MIXED):
        out[f] = {k: tb[2 + 5 * i + j] for j, k in enumerate(("sy", "sy2", "sxy", "sabs", "amax"))}
    return out


def _ntiles(rows, cols):
    return -(-rows // 32) * -(-cols // 32)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("xdt", ["bf16", "f32"])
def test_tile_stats_strict_strided(qa, shape, xdt):
    """qa_tile_stats (strict): bit-equal to the oracle's NumPy-order table at every layout."""
    rows, cols = shape
    x = _matrix(shape, xdt, 3 * rows + cols)
    want = orc.tile_stat_table(x)
    for ld, off, poison in _layouts(cols, DT[xdt]):
        _buf, ptr = _place(x, DT[xdt], ld, off, poison)
        t = torch.zeros((22, _ntiles(rows, cols)), dtype=torch.float64, device="cuda")
        qa.lib.check(qa.L.qa_tile_stats(ptr, _code(_buf), rows, cols, ld, 0, 0xF, 1, t.data_ptr(), _stream()), "qa_tile_stats")
        got = _table_dict(t)
        tag = (xdt, shape, ld, off)
        assert np.array_equal(got["sx"], want["sx"]) and np.array_equal(got["sx2"], want["sx2"]), tag
        for f in MIXED:
            for k in ("sy", "sy2", "sxy", "sabs", "amax"):
                assert np.array_equal(got[f][k], want[f][k]), (tag, f, k)


@pytest.mark.parametrize("shape", SHAPES)
def test_tile_stats_fast_strided(qa, shape):
    """qa_tile_stats (fast, both |x-y| modes), qa_tile_stats_rows in two pieces and qa_tile_stats_batch over descriptors
    with ld > cols and offset bases: the same bits as qa_tile_stats on the contiguous matrix."""
    rows, cols = shape
    nt, th = _ntiles(rows, cols), -(-rows // 32)
    x = _matrix(shape, "bf16", 5 * rows + cols)
    xc = torch.from_numpy(x).cuda().to(torch.bfloat16)
    ref = {}
    for mode in (0, 2):
        ref[mode] = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
        qa.lib.check(qa.L.qa_tile_stats(xc.data_ptr(), 0, rows, cols, cols, 0, 0xF, mode, ref[mode].data_ptr(), _stream()),
                     "qa_tile_stats")
    layouts = _layouts(cols, torch.bfloat16)
    keep, entries = [], []
    for ld, off, poison in layouts:
        buf, ptr = _place(x, torch.bfloat16, ld, off, poison)
        keep.append(buf)
        tag = (shape, ld, off)
        for mode in (0, 2):
            t = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
            qa.lib.check(qa.L.qa_tile_stats(ptr, 0, rows, cols, ld, 0, 0xF, mode, t.data_ptr(), _stream()), "qa_tile_stats")
            assert torch.equal(t, ref[mode]), (tag, mode)
        t = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
        for lo, hi in ((0, 1), (1, th)) if th > 1 else ((0, 1),):
            qa.lib.check(qa.L.qa_tile_stats_rows(ptr, 0, rows, cols, ld, 0xF, 0, t.data_ptr(), lo, hi, _stream()),
                         "qa_tile_stats_rows")
        assert torch.equal(t, ref[0]), (tag, "rows")
        table = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
        keep.append(table)
        entries.append((ptr, table, ld))
    arr = (qa.lib.BatchDesc * len(entries))()
    items = 0
    for d, (ptr, table, ld) in zip(arr, entries):
        d.x, d.table, d.init, d.rows, d.cols, d.ld = ptr, table.data_ptr(), None, rows, cols, ld
        d.item_begin, d.block_begin = items, 0
        items += qa.L.qa_tile_stats_items(rows, cols)
    descs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).cuda()
    qa.lib.check(qa.L.qa_tile_stats_batch(descs.data_ptr(), len(entries), items, 0xF, 0, _stream()), "qa_tile_stats_batch")
    for (ld, off, _p), (_ptr, table, _ld) in zip(layouts, entries):
        assert torch.equal(table, ref[0]), (shape, ld, off, "batch")


@pytest.mark.parametrize("shape", SHAPES)
def test_tile_stats_f32_strided(qa, shape):
    """qa_tile_stats_f32 (a per-row alignment check picks the 256-bit loads): the contiguous call's bits at every layout,
    whole and in two tile-row pieces."""
    rows, cols = shape
    nt, th = _ntiles(rows, cols), -(-rows // 32)
    x = _matrix(shape, "f32", 11 * rows + cols)
    xc = torch.from_numpy(x).cuda()
    ref = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
    qa.lib.check(qa.L.qa_tile_stats_f32(xc.data_ptr(), rows, cols, cols, 0xF, 0, ref.data_ptr(), 0, -1, _stream()),
                 "qa_tile_stats_f32")
    for ld, off, poison in _layouts(cols, torch.float32):
        _buf, ptr = _place(x, torch.float32, ld, off, poison)
        for pieces in (((0, -1),), ((0, 1), (1, th)) if th > 1 else ((0, -1),)):
            t = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
            for lo, hi in pieces:
                qa.lib.check(qa.L.qa_tile_stats_f32(ptr, rows, cols, ld, 0xF, 0, t.data_ptr(), lo, hi, _stream()),
                             "qa_tile_stats_f32")
            assert torch.equal(t, ref), (shape, ld, off, pieces)


@pytest.mark.parametrize("shape", SHAPES)
def test_tile_stats_fp8_strided(qa, shape):
    """qa_tile_stats_fp8 (a per-group alignment check picks the 128-bit loads): the contiguous call's table and inexact count
    at every layout, with the bytes around the matrix 0x7F (NaN) or 0x7E (448)."""
    rows, cols = shape
    nt = _ntiles(rows, cols)
    rng = np.random.default_rng(rows * cols + 1)
    w = rng.integers(0, 256, shape, dtype=np.uint8)
    w[(w & 0x7F) == 0x7F] = 0x3C
    sr, sc_ = min(rows, 3), min(cols, 4)
    sc = torch.from_numpy(np.exp(rng.uniform(np.log(1e-4), np.log(3e-3), (sr, sc_))).astype(np.float32)).cuda()

    def run(ptr, ld):
        t = torch.zeros((22, nt), dtype=torch.float64, device="cuda")
        cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
        qa.lib.check(qa.L.qa_tile_stats_fp8(ptr, sc.data_ptr(), rows, cols, ld, sr, sc_, 0xF, 0, t.data_ptr(), 0, -1,
                                            cnt.data_ptr(), _stream()), "qa_tile_stats_fp8")
        return t, int(cnt.item())

    wc = torch.from_numpy(w).cuda()
    ref, ref_cnt = run(wc.data_ptr(), cols)
    assert ref_cnt > 0
    for ld, off, poison in _layouts(cols, torch.uint8):
        _buf, ptr = _place(w, torch.uint8, ld, off, poison)
        t, cnt = run(ptr, ld)
        assert torch.equal(t, ref) and cnt == ref_cnt, (shape, ld, off, poison)


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("xdt", ["bf16", "f32"])
def test_tile_scores_strided(qa, shape, xdt):
    """qa_tile_scores_f32: bit-equal to orc.padded_tile_scores for all three metrics at every layout."""
    rows, cols = shape
    nt = _ntiles(rows, cols)
    x = _matrix(shape, xdt, 13 * rows + cols)
    with np.errstate(all="ignore"):
        want = {m: orc.padded_tile_scores(x, MIXED, m) for m in ("pcc", "mae", "atol")}
    for ld, off, poison in _layouts(cols, DT[xdt]):
        _buf, ptr = _place(x, DT[xdt], ld, off, poison)
        s = torch.zeros((3, 4, nt), dtype=torch.float32, device="cuda")
        qa.lib.check(qa.L.qa_tile_scores_f32(ptr, _code(_buf), rows, cols, ld, 0xF, s.data_ptr(), _stream()), "qa_tile_scores_f32")
        got = s.cpu().numpy()
        for mi, m in enumerate(("pcc", "mae", "atol")):
            for fi, f in enumerate(MIXED):
                w = np.asarray(want[m][f], np.float32).reshape(-1)
                assert np.array_equal(_bits(got[mi, fi]), _bits(w)), (xdt, shape, ld, off, m, f)
