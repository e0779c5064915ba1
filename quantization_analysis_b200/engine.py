"""Device engine: marshals tensors to the C ABI (include/qa_b200.h).  PyTorch is plumbing only
(device memory, streams); all arithmetic on the path happens in libqa_b200.so kernels.

Geometry.  The quantizers treat an n-d tensor as rows of its last axis (groups of 16 never
cross a row; quantization_formats.py:89-119).  The mixed-tile algorithms tile
``[prod(shape[:-1]), W]`` (1-D: rows of 32, zero-padded; tile_utils.py:91-115).  ``Prepared``
holds a device copy in the tile geometry; for >= 2-D inputs the two geometries coincide.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, tensor_source
from ._lib import (METRIC_CODE, NFMT, NSTAT, QA_DT_BF16, QA_DT_F32, STATS_FAST, STATS_FAST_APPROX_ABS, STATS_STRICT,
                   check)

MIXED_FORMATS = ("bf16", "bfp8", "bfp4", "bfp2")
FMT_INDEX = {f: i for i, f in enumerate(MIXED_FORMATS)}
TILE = 32


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.QaError("CUDA device required: the quantize-and-score path has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: torch.Tensor | None) -> int:
    return 0 if t is None else t.data_ptr()


def fmt_mask(formats) -> int:
    m = 0
    for f in formats:
        m |= 1 << FMT_INDEX[f]
    return m


@dataclass
class Prepared:
    """A tensor resident on the device in [rows, cols] row-major layout."""
    data: torch.Tensor          # bfloat16 or float32, contiguous, rows*cols elements
    dtype_code: int             # QA_DT_BF16 / QA_DT_F32
    rows: int
    cols: int
    numel: int                  # elements of the original tensor
    shape: tuple                # original shape
    kind: str                   # "nd" | "vector" | "scalar"
    vec_tail: int = 0           # valid elements in the ragged last row of a 1-D input (0: none)

    @property
    def tiles_h(self) -> int:
        return -(-self.rows // TILE)

    @property
    def tiles_w(self) -> int:
        return -(-self.cols // TILE)

    @property
    def ntiles(self) -> int:
        return self.tiles_h * self.tiles_w


class Fp8Prepared(Prepared):
    """A 2-D fp8 e4m3fn checkpoint tensor with per-block inverse scales (hf_model_utils.py:199-215).  The tile-stat pass reads
    the bytes directly (tile_stats_fp8); `data`, the float32 image the reference would have built, is only materialised
    (qa_fp8_block_dequant) by a consumer that needs it: the reconstruction writer, the strict fallback, the float32 scorer."""

    def __init__(self, w_fp8: torch.Tensor, scale_inv: torch.Tensor):
        dev = _require_cuda()
        w = w_fp8.to(dev).contiguous()
        self.w8 = w.view(torch.uint8) if w.dtype != torch.uint8 else w
        self.scale_inv = scale_inv.to(dev, torch.float32).contiguous()
        if self.w8.dim() != 2 or self.scale_inv.dim() != 2:
            raise ValueError("Fp8Prepared expects 2-D weight and scale tensors")
        rows, cols = (int(v) for v in self.w8.shape)
        super().__init__(None, QA_DT_F32, rows, cols, rows * cols, (rows, cols), "nd")

    @property
    def data(self):
        if self._data is None:
            self._data = fp8_block_dequant(self.w8, self.scale_inv, want_bf16=False)[0].reshape(-1)
        return self._data

    @data.setter
    def data(self, v):
        self._data = v


def to_device(x, want_bf16: bool = True) -> tuple[torch.Tensor, int]:
    """Host fp32 ndarray / torch tensor -> contiguous device tensor (bf16 when exactly representable)."""
    dev = _require_cuda()
    if isinstance(x, torch.Tensor):
        t = x.detach()
        if t.dtype == torch.bfloat16:
            return t.to(dev).contiguous(), QA_DT_BF16
        t = t.to(device=dev, dtype=torch.float32).contiguous()
    else:
        a = np.ascontiguousarray(np.asarray(x, dtype=np.float32))
        t = torch.from_numpy(a).to(dev, non_blocking=False)
    if not want_bf16 or t.numel() == 0:
        return t, QA_DT_F32
    out = torch.empty(t.shape, dtype=torch.bfloat16, device=dev)
    bad = torch.zeros(1, dtype=torch.int64, device=dev)
    check(_lib.lib().qa_f32_to_bf16_checked(_ptr(t), t.numel(), _ptr(out), _ptr(bad), _stream()), "qa_f32_to_bf16_checked")
    if int(bad.item()) == 0:
        return out, QA_DT_BF16
    return t, QA_DT_F32


def prepare_loaded(x) -> Prepared:
    """What tensor_source's loaders return -> Prepared in the mixed-tile geometry: Fp8Prepared for a block-scaled fp8 weight
    (its bytes go to the device as they are), prepare_tiles for a host array or torch tensor; a Prepared is returned as is."""
    if isinstance(x, Prepared):
        return x
    if isinstance(x, tensor_source.Fp8Blocks):
        return Fp8Prepared(x.weight, x.scale_inv)
    return prepare_tiles(x)


_ELEM_BYTES = {torch.uint8: 1, torch.bfloat16: 2, torch.float32: 4}


def transpose_2d(t: torch.Tensor) -> torch.Tensor:
    """Contiguous device copy of t.T for a 2-D device tensor of 1-, 2- or 4-byte elements (qa_transpose_2d)."""
    if t.dim() != 2 or t.dtype not in _ELEM_BYTES:
        raise ValueError(f"transpose_2d expects a 2-D uint8 / bfloat16 / float32 tensor, got {t.dtype} {tuple(t.shape)}")
    if t.stride(1) != 1:
        t = t.contiguous()
    rows, cols = int(t.shape[0]), int(t.shape[1])
    out = torch.empty((cols, rows), dtype=t.dtype, device=t.device)
    check(_lib.lib().qa_transpose_2d(_ptr(t), _ELEM_BYTES[t.dtype], rows, cols, max(int(t.stride(0)), cols), _ptr(out), _stream()),
          "qa_transpose_2d")
    return out


def prepare_transposed(x) -> Prepared:
    """The device layout: a linear weight W [out, in] is held on the device as W^T [in, out], and the BFP groups and the
    32x32 tiles are taken there.  -> prepare_loaded(x.T) for a 2-D x (the tile grid is [ceil(cols/32), ceil(rows/32)]):
    one H2D copy (bf16 when the values are bf16-exact, as prepare_tiles), then qa_transpose_2d on the device.  An fp8
    weight (tensor_source.Fp8Blocks or Fp8Prepared) stays fp8: its bytes and its scale grid are transposed, and
    dequant(w^T, s^T) == dequant(w, s)^T element for element.  A Prepared already on the device is transposed there.
    0-D and 1-D inputs: x.T is x, so this is prepare_loaded(x).  3 or more dimensions: ValueError."""
    shape = tuple(x.shape)
    if len(shape) > 2:
        raise ValueError(f"the transposed (device) layout needs a 0-, 1- or 2-D tensor, got shape {shape}")
    if len(shape) < 2:
        return prepare_loaded(x)
    if isinstance(x, tensor_source.Fp8Blocks):
        x = Fp8Prepared(x.weight, x.scale_inv)
    if isinstance(x, Fp8Prepared):
        return Fp8Prepared(transpose_2d(x.w8), transpose_2d(x.scale_inv))
    p = x if isinstance(x, Prepared) else prepare_tiles(x)
    data = p.data.reshape(p.rows, p.cols)
    return Prepared(transpose_2d(data).reshape(-1), p.dtype_code, p.cols, p.rows, p.numel, (p.cols, p.rows), "nd")


def prepare_rows(x) -> Prepared:
    """Quantizer geometry: rows of the last axis (1-D: one row)."""
    shape = tuple(x.shape)
    t, code = to_device(x)
    if len(shape) == 0:
        rows, cols, kind = 1, 1, "scalar"
    elif len(shape) == 1:
        rows, cols, kind = 1, shape[0], "vector"
    else:
        rows, cols, kind = int(np.prod(shape[:-1])), shape[-1], "nd"
    return Prepared(t.reshape(-1), code, rows, cols, int(np.prod(shape)) if shape else 1, shape, kind)


def prepare_tiles(x) -> Prepared:
    """Mixed-tile geometry (tile_utils.py:91-115)."""
    shape = tuple(x.shape)
    t, code = to_device(x)
    numel = int(np.prod(shape)) if shape else 1
    if len(shape) == 0:
        return Prepared(t.reshape(-1), code, 1, 1, 1, shape, "scalar")
    if len(shape) == 1:
        n = shape[0]
        rows = -(-n // TILE)
        if rows * TILE != n:
            pad = torch.zeros(rows * TILE, dtype=t.dtype, device=t.device)
            pad[:n] = t
            t = pad
        tail = n % TILE
        return Prepared(t.reshape(-1), code, rows, TILE, numel, shape, "vector", vec_tail=tail)
    return Prepared(t.reshape(-1), code, int(np.prod(shape[:-1])), shape[-1], numel, shape, "nd")


# --------------------------------------------------------------------------------------------
# kernels
# --------------------------------------------------------------------------------------------
def quant_recon(p: Prepared, formats) -> dict[str, torch.Tensor]:
    """bf16 reconstructions for `formats` (subset of MIXED_FORMATS) in one pass."""
    formats = [f for f in formats if f in FMT_INDEX]
    outs: dict[str, torch.Tensor] = {}
    arr = (C.c_void_p * NFMT)()
    for f in formats:
        o = torch.empty(p.rows * p.cols, dtype=torch.bfloat16, device=p.data.device)
        outs[f] = o
        arr[FMT_INDEX[f]] = o.data_ptr()
    if p.rows * p.cols and formats:
        check(_lib.lib().qa_quant_recon(_ptr(p.data), p.dtype_code, p.rows, p.cols, p.cols, fmt_mask(formats), arr, _stream()),
              "qa_quant_recon")
    return outs


def quant_recon_cols(x, formats) -> tuple[dict[str, torch.Tensor], tuple]:
    """bf16 reconstructions with the shared exponent along axis 0 (16 consecutive rows of a column; transpose.py:13-33:
    quantize x.T, transpose back - computed in place by qa_quant_recon_cols, no transposed copy).  x: >= 2-D."""
    shape = tuple(x.shape)
    t, code = to_device(x)
    rows, cols = int(shape[0]), int(np.prod(shape[1:]))
    formats = [f for f in formats if f in FMT_INDEX]
    outs: dict[str, torch.Tensor] = {}
    arr = (C.c_void_p * NFMT)()
    for f in formats:
        o = torch.empty(rows * cols, dtype=torch.bfloat16, device=t.device)
        outs[f] = o
        arr[FMT_INDEX[f]] = o.data_ptr()
    if rows * cols and formats:
        check(_lib.lib().qa_quant_recon_cols(_ptr(t), code, rows, cols, cols, fmt_mask(formats), arr, _stream()), "qa_quant_recon_cols")
    return outs, shape


def tile_stats(p: Prepared, formats=MIXED_FORMATS, strict: bool | None = None, exact_abs: bool = True) -> torch.Tensor:
    """float64 [NSTAT, ntiles] tile-stat table.  strict=None / False: the fast kernels (qa_tile_stats for bf16 input,
    qa_tile_stats_f32 for float32 input that is not bf16-exact); strict=True: NumPy-order sums (validation, certificate
    fallback).  exact_abs=False lets the fast kernels keep sum|x-y| in fp32 group partials (~1e-9 relative): fine when
    that column only feeds a reported mae or an is-zero test (pcc / atol assignment).  An Fp8Prepared takes the fused pass
    over its bytes (tile_stats_fp8; the same table as qa_tile_stats_f32 on its float32 image, which stays unmaterialised)
    unless strict."""
    if isinstance(p, Fp8Prepared) and not strict:
        return tile_stats_fp8(p.w8, p.scale_inv, formats, exact_abs=exact_abs)[0]
    table = torch.zeros((NSTAT, p.ntiles), dtype=torch.float64, device=p.data.device)
    mode = STATS_STRICT if strict else (STATS_FAST if exact_abs else STATS_FAST_APPROX_ABS)
    if p.dtype_code == QA_DT_F32 and not strict:
        check(_lib.lib().qa_tile_stats_f32(_ptr(p.data), p.rows, p.cols, p.cols, fmt_mask(formats), mode, _ptr(table), 0, -1,
                                           _stream()), "qa_tile_stats_f32")
        return table
    check(_lib.lib().qa_tile_stats(_ptr(p.data), p.dtype_code, p.rows, p.cols, p.cols, p.vec_tail, fmt_mask(formats), mode,
                                   _ptr(table), _stream()), "qa_tile_stats")
    return table


def tile_stats_fp8(w_fp8: torch.Tensor, scale_inv: torch.Tensor, formats=MIXED_FORMATS, exact_abs: bool = True):
    """Tile-stat table straight from fp8 e4m3fn weights + per-block inverse scales (qa_tile_stats_fp8: the dequantization of
    hf_model_utils.py:199-215 fused into the read; the float32 tensor is never materialised).
    -> (table float64 [NSTAT, ntiles], number of products that are not bf16-exact as a device int64[1])."""
    dev = _require_cuda()
    w = w_fp8.to(dev).contiguous()
    w8 = w.view(torch.uint8) if w.dtype != torch.uint8 else w
    sc = scale_inv.to(dev, torch.float32).contiguous()
    if w8.dim() != 2 or sc.dim() != 2:
        raise ValueError("tile_stats_fp8 expects 2-D weight and scale tensors")
    rows, cols = w8.shape
    ntiles = (-(-rows // TILE)) * (-(-cols // TILE))
    table = torch.zeros((NSTAT, ntiles), dtype=torch.float64, device=dev)
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    mode = STATS_FAST if exact_abs else STATS_FAST_APPROX_ABS
    check(_lib.lib().qa_tile_stats_fp8(_ptr(w8), _ptr(sc), rows, cols, cols, sc.shape[0], sc.shape[1], fmt_mask(formats), mode,
                                       _ptr(table), 0, -1, _ptr(cnt), _stream()), "qa_tile_stats_fp8")
    return table, cnt


def batch_descriptors(entries, device):
    """Device-resident qa_batch_desc array for a list of resident bf16 tensors.
    entries: (x data_ptr, table data_ptr, init data_ptr or 0, rows, cols) per tensor.
    -> (uint8 device tensor holding the array, n, total tile-stat items, total 256-tile delta blocks)."""
    L = _lib.lib()
    arr = (_lib.BatchDesc * len(entries))()
    items = blocks = 0
    for d, (xp, tp, ip, rows, cols) in zip(arr, entries):
        d.x, d.table, d.init, d.rows, d.cols, d.ld = xp, tp, ip or None, rows, cols, cols
        d.item_begin, d.block_begin = items, blocks
        items += L.qa_tile_stats_items(rows, cols)
        blocks += -(-((-(-rows // TILE)) * (-(-cols // TILE))) // 256)
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    return host.to(device), len(entries), int(items), int(blocks)


def tile_stats_batch(descs: torch.Tensor, n: int, total_items: int, formats=MIXED_FORMATS, exact_abs: bool = True) -> None:
    """qa_tile_stats (fast) for a whole descriptor array in one launch; the tables named by the descriptors are filled."""
    mode = STATS_FAST if exact_abs else STATS_FAST_APPROX_ABS
    check(_lib.lib().qa_tile_stats_batch(_ptr(descs), n, total_items, fmt_mask(formats), mode, _stream()), "qa_tile_stats_batch")


def fp8_block_dequant(w_fp8: torch.Tensor, scale_inv: torch.Tensor, want_bf16: bool = True):
    """fp8 e4m3fn [rows, cols] (uint8 or float8_e4m3fn storage) * scale_inv blocks -> (float32 tensor, bf16 tensor or None,
    number of products that are not bf16-exact).  hf_model_utils.py:199-215 on the device."""
    dev = _require_cuda()
    w = w_fp8.to(dev).contiguous()
    w8 = w.view(torch.uint8) if w.dtype != torch.uint8 else w
    sc = scale_inv.to(dev, torch.float32).contiguous()
    if w8.dim() != 2 or sc.dim() != 2:
        raise ValueError("fp8_block_dequant expects 2-D weight and scale tensors")
    rows, cols = w8.shape
    out = torch.empty((rows, cols), dtype=torch.float32, device=dev)
    ob = torch.empty((rows, cols), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    check(_lib.lib().qa_fp8_block_dequant(_ptr(w8), _ptr(sc), rows, cols, sc.shape[0], sc.shape[1], _ptr(out), _ptr(ob), _ptr(cnt),
                                          _stream()), "qa_fp8_block_dequant")
    return out, ob, int(cnt.item())


def scalar_proxy(x: torch.Tensor, which: int, out: torch.Tensor) -> torch.Tensor:
    """mxfp4 (0) / nvfp4 (1) scalar proxy of a contiguous bf16 / float32 device tensor into a float32 tensor."""
    code = _lib.QA_DT_BF16 if x.dtype == torch.bfloat16 else _lib.QA_DT_F32
    check(_lib.lib().qa_scalar_proxy(_ptr(x), code, x.numel(), int(which), _ptr(out), _stream()), "qa_scalar_proxy")
    return out


def tile_scores(p: Prepared, formats=MIXED_FORMATS) -> torch.Tensor:
    """float32 [3 metrics, NFMT, ntiles] NumPy-faithful padded-tile scores."""
    s = torch.zeros((3, NFMT, p.ntiles), dtype=torch.float32, device=p.data.device)
    check(_lib.lib().qa_tile_scores_f32(_ptr(p.data), p.dtype_code, p.rows, p.cols, p.cols, fmt_mask(formats), _ptr(s), _stream()),
          "qa_tile_scores_f32")
    return s


def tile_scores_pair(ref_tiles: np.ndarray, q_tiles: np.ndarray) -> np.ndarray:
    """float32 [3, N] NumPy-faithful (pcc, mae, atol) of two arbitrary [N,32,32] float32 tile stacks."""
    dev = _require_cuda()
    r = torch.from_numpy(np.ascontiguousarray(ref_tiles, dtype=np.float32).reshape(-1)).to(dev)
    q = torch.from_numpy(np.ascontiguousarray(q_tiles, dtype=np.float32).reshape(-1)).to(dev)
    n = r.numel() // 1024
    s = torch.empty((3, n), dtype=torch.float32, device=dev)
    check(_lib.lib().qa_tile_scores_pair_f32(_ptr(r), _ptr(q), n, _ptr(s), _stream()), "qa_tile_scores_pair_f32")
    return s.cpu().numpy()


def make_rng(seed: int, device=None) -> torch.Tensor:
    """Device-resident qa_pcg64 seeded like np.random.default_rng(seed) (SeedSequence on host)."""
    device = device or _require_cuda()
    st = np.random.default_rng(seed).bit_generator.state
    s, inc = int(st["state"]["state"]), int(st["state"]["inc"])
    m64 = (1 << 64) - 1
    words = np.array([s >> 64, s & m64, inc >> 64, inc & m64,
                      (int(st["has_uint32"]) & 0xFFFFFFFF) | ((int(st["uinteger"]) & 0xFFFFFFFF) << 32)], dtype=np.uint64)
    return torch.from_numpy(words.view(np.int64).copy()).to(device)


def numpy_permutation(rng: torch.Tensor, n: int, parallel: bool = True) -> torch.Tensor:
    """np.random.Generator.permutation(n) continued from `rng` on the device (int32)."""
    out = torch.empty(n, dtype=torch.int32, device=rng.device)
    L = _lib.lib()
    if parallel:
        work = torch.empty(L.qa_greedy_par_work_bytes(max(n, 1)), dtype=torch.uint8, device=rng.device)
        check(L.qa_numpy_permutation_par(_ptr(rng), n, _ptr(out), _ptr(work), _stream()), "qa_numpy_permutation_par")
    else:
        work = torch.empty(2 * max(n, 1), dtype=torch.int32, device=rng.device)
        check(L.qa_numpy_permutation(_ptr(rng), n, _ptr(out), _ptr(work), _stream()), "qa_numpy_permutation")
    return out


def numpy_integers(rng: torch.Tensor, k: int, n: int) -> torch.Tensor:
    out = torch.empty(n, dtype=torch.int8, device=rng.device)
    check(_lib.lib().qa_numpy_integers(_ptr(rng), k, n, _ptr(out), _stream()), "qa_numpy_integers")
    return out


def enqueue_perm_prefetch(rng0: torch.Tensor, nt: int, three: bool, bufs, side, side2, events) -> None:
    """Enqueue the data-independent permutations of a greedy run over nt tiles, drawn from the stream state `rng0` (not
    modified): resolves #1 (stream position only) and #2 in one cluster launch on `side`, then #2's apply on `side2`
    next to resolve #3 and #3's apply on `side`.  Without `three` (fewer than three formats) only #2 is applied, on `side`.
    bufs = (jarr int32[3, nt], pre_order int32[2, nt], rngs [3, 5], awork uint8[2, qa_perm_apply_work_bytes(nt)]): the
    chain reads pre_order (visiting orders of passes 2 and 3) and rngs[1:] (stream states after permutations #2 and #3).
    events = (resolved, applied2, applied3), recorded once #1 and #2 are resolved, once pre_order[0] is written and once
    pre_order[1] is (three only)."""
    L = _lib.lib()
    jarr, pre_order, rngs, awork = bufs
    resolved, applied2, applied3 = events
    check(L.qa_perm_resolve_chain(_ptr(rng0), nt, 2, 0b10, _ptr(jarr), _ptr(rngs), side.cuda_stream), "qa_perm_resolve_chain")
    resolved.record(side)
    s2 = side
    if three:
        side2.wait_event(resolved)
        s2 = side2
    check(L.qa_perm_apply(_ptr(jarr[1]), nt, None, _ptr(pre_order[0]), _ptr(awork[0]), s2.cuda_stream), "qa_perm_apply")
    applied2.record(s2)
    if three:
        check(L.qa_perm_resolve(_ptr(rngs[1]), nt, _ptr(jarr[2]), _ptr(rngs[2]), side.cuda_stream), "qa_perm_resolve")
        check(L.qa_perm_apply(_ptr(jarr[2]), nt, None, _ptr(pre_order[1]), _ptr(awork[1]), side.cuda_stream), "qa_perm_apply")
        applied3.record(side)


def greedy_prefetch(rng: torch.Tensor, ntiles: int, nfmt: int = NFMT):
    """enqueue_perm_prefetch on the current stream, for greedy_assign(prefetched=...).
    -> (pre_order int32[1 or 2][ntiles], pre_rng[1 or 2]).  `rng` is not modified."""
    L = _lib.lib()
    dev = rng.device
    three = nfmt >= 3
    bufs = (torch.empty((3, ntiles), dtype=torch.int32, device=dev), torch.empty((2, ntiles), dtype=torch.int32, device=dev),
            torch.stack([rng, rng, rng]).contiguous(), torch.empty((2, L.qa_perm_apply_work_bytes(ntiles)), dtype=torch.uint8, device=dev))
    cur = torch.cuda.current_stream(dev)
    enqueue_perm_prefetch(rng, ntiles, three, bufs, cur, cur, [torch.cuda.Event() for _ in range(3)])
    k = 2 if three else 1
    return bufs[1][:k], bufs[2][1:1 + k]


def numpy_permutation_staged(rng: torch.Tensor, n: int) -> torch.Tensor:
    """numpy permutation(n) as qa_perm_resolve (one cluster) + qa_perm_apply (grid kernels); advances `rng`."""
    L = _lib.lib()
    dev = rng.device
    jarr = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    out = torch.empty(n, dtype=torch.int32, device=dev)
    if n == 0:
        return out
    work = torch.empty(L.qa_perm_apply_work_bytes(n), dtype=torch.uint8, device=dev)
    check(L.qa_perm_resolve(_ptr(rng), n, _ptr(jarr), _ptr(rng), _stream()), "qa_perm_resolve")
    check(L.qa_perm_apply(_ptr(jarr), n, None, _ptr(out), _ptr(work), _stream()), "qa_perm_apply")
    return out


def greedy_init(table: torch.Tensor, metric: str, fmt_order) -> torch.Tensor:
    """Initial sums + per-transition delta records of a greedy run (qa_greedy_init_deltas, qa_greedy_init_sums_range);
    consumed by greedy_assign(init=...)."""
    L = _lib.lib()
    nt = table.shape[1]
    init = torch.empty(L.qa_greedy_init_bytes(nt), dtype=torch.uint8, device=table.device)
    iargs = (_ptr(table), nt, METRIC_CODE[metric], _lib.int32_array([FMT_INDEX[f] for f in fmt_order]), len(fmt_order), _ptr(init))
    check(L.qa_greedy_init_deltas(*iargs, _stream()), "qa_greedy_init_deltas")
    check(L.qa_greedy_init_sums_range(*iargs, 0, nt, _stream()), "qa_greedy_init_sums_range")
    return init


def greedy_assign(table: torch.Tensor, numel: int, metric: str, threshold: float, fmt_order, rng: torch.Tensor,
                  parallel: bool | None = None, prefetched=None, init: torch.Tensor | None = None, split_at: int | None = None):
    """-> (assignment int8[ntiles], counts int64[4], state float64[24]) on device.
    parallel=None: the cluster-parallel kernel for pcc / mae, the one-thread chain for atol.
    prefetched = greedy_prefetch(...) and init = greedy_init(...) are optional stages computed ahead of time; without init the
    first launch computes it into its work buffer."""
    nt = table.shape[1]
    dev = table.device
    L = _lib.lib()
    if parallel is None:
        parallel = metric in ("pcc", "mae")
    assignment = torch.empty(nt, dtype=torch.int8, device=dev)
    counts = torch.zeros(NFMT, dtype=torch.int64, device=dev)
    state = torch.zeros(24, dtype=torch.float64, device=dev)
    order = _lib.int32_array([FMT_INDEX[f] for f in fmt_order])
    if parallel:
        work = torch.empty(L.qa_greedy_par_work_bytes(nt), dtype=torch.uint8, device=dev)
        pre_order, pre_rng = prefetched if prefetched is not None else (None, None)
        if pre_order is not None and len(fmt_order) >= 3 and pre_order.shape[0] < 2:
            raise ValueError("prefetched permutations were drawn for fewer formats than fmt_order has")
        ranges = [(0, len(fmt_order))] if not split_at else [(0, split_at), (split_at, len(fmt_order))]
        for b, e in ranges:          # split_at: the same run as two launches (qa_greedy_assign_passes)
            check(L.qa_greedy_assign_passes(_ptr(table), nt, float(numel), METRIC_CODE[metric], float(threshold), order,
                                            len(fmt_order), _ptr(rng), _ptr(assignment), _ptr(counts), _ptr(state), _ptr(work),
                                            _ptr(pre_order), _ptr(pre_rng), _ptr(init), b, e, 0, _stream()), "qa_greedy_assign_par")
    else:
        work = torch.empty(L.qa_greedy_work_bytes(nt), dtype=torch.uint8, device=dev)
        check(L.qa_greedy_assign(_ptr(table), nt, float(numel), METRIC_CODE[metric], float(threshold), order, len(fmt_order),
                                 _ptr(rng), _ptr(assignment), _ptr(counts), _ptr(state), _ptr(work), _stream()),
              "qa_greedy_assign")
    return assignment, counts, state


def greedy_sweep(table: torch.Tensor, numel: int, metric: str, thresholds, fmt_order, rng: torch.Tensor, prefetched=None,
                 init: torch.Tensor | None = None):
    """The greedy chains of every threshold over one table in one launch (qa_greedy_assign_sweep): row k is what
    greedy_assign gives for thresholds[k] from the stream state `rng` (not modified).  prefetched = greedy_prefetch(...) or
    the permutation cache, init = greedy_init(...): shared by every chain (pcc / mae; atol runs the one-thread chain and
    needs neither).  -> (maps int8 [K, ntiles], counts int64 [K, 4], states float64 [K, 24]) on the device."""
    nt = table.shape[1]
    dev = table.device
    L = _lib.lib()
    thr = torch.tensor(np.asarray(list(thresholds), dtype=np.float64).reshape(-1), device=dev)
    k = thr.numel()
    maps = torch.empty((k, nt), dtype=torch.int8, device=dev)
    counts = torch.zeros((k, NFMT), dtype=torch.int64, device=dev)
    states = torch.zeros((k, 24), dtype=torch.float64, device=dev)
    per = L.qa_greedy_sweep_work_bytes(nt, METRIC_CODE[metric])
    work = torch.empty(max(k, 1) * max(per, 0), dtype=torch.uint8, device=dev)
    pre_order, pre_rng = prefetched if prefetched is not None else (None, None)
    if pre_order is not None and len(fmt_order) >= 3 and pre_order.shape[0] < 2:
        raise ValueError("prefetched permutations were drawn for fewer formats than fmt_order has")
    order = _lib.int32_array([FMT_INDEX[f] for f in fmt_order])
    check(L.qa_greedy_assign_sweep(_ptr(table), nt, float(numel), METRIC_CODE[metric], _ptr(thr), k, order, len(fmt_order), _ptr(rng),
                                   _ptr(maps), _ptr(counts), _ptr(states), _ptr(work), _ptr(pre_order), _ptr(pre_rng), _ptr(init), 0,
                                   _stream()), "qa_greedy_assign_sweep")
    return maps, counts, states


_STAGE_STREAMS: dict = {}


def greedy_assign_staged(table: torch.Tensor, numel: int, metric: str, threshold: float, fmt_order, rng: torch.Tensor):
    """greedy_assign for one tensor with the stages overlapped on side streams: the data-independent permutations
    (enqueue_perm_prefetch) next to the initial sums and delta records (qa_greedy_init_sums_range / qa_greedy_init_deltas),
    then the chain by pass range (qa_greedy_assign_passes).
    Same outputs, bit for bit, as greedy_assign; about half its latency on a large tensor.  `rng` is advanced."""
    if metric not in ("pcc", "mae") or len(fmt_order) < 2:
        return greedy_assign(table, numel, metric, threshold, fmt_order, rng)
    L = _lib.lib()
    dev = table.device
    nt, nf = table.shape[1], len(fmt_order)
    three = nf >= 3
    key = (dev.index, "stage")
    if key not in _STAGE_STREAMS:
        _STAGE_STREAMS[key] = (torch.cuda.Stream(device=dev, priority=-1), torch.cuda.Stream(device=dev, priority=-1))
    side, side2 = _STAGE_STREAMS[key]
    cur = torch.cuda.current_stream(dev)
    order = _lib.int32_array([FMT_INDEX[f] for f in fmt_order])
    assignment = torch.empty(nt, dtype=torch.int8, device=dev)
    counts = torch.zeros(NFMT, dtype=torch.int64, device=dev)
    state = torch.zeros(24, dtype=torch.float64, device=dev)
    work = torch.empty(L.qa_greedy_par_work_bytes(nt), dtype=torch.uint8, device=dev)
    init = torch.empty(L.qa_greedy_init_bytes(nt), dtype=torch.uint8, device=dev)
    jarr = torch.empty((3, nt), dtype=torch.int32, device=dev)
    pre_order = torch.empty((2, nt), dtype=torch.int32, device=dev)
    rngs = torch.stack([rng, rng, rng]).contiguous()
    awork = torch.empty((2, L.qa_perm_apply_work_bytes(nt)), dtype=torch.uint8, device=dev)
    ev_a2, ev_a3 = torch.cuda.Event(), torch.cuda.Event()
    side.wait_stream(cur)
    side2.wait_stream(cur)
    enqueue_perm_prefetch(rng, nt, three, (jarr, pre_order, rngs, awork), side, side2, (torch.cuda.Event(), ev_a2, ev_a3))
    iargs = (_ptr(table), nt, METRIC_CODE[metric], order, nf, _ptr(init))
    check(L.qa_greedy_init_deltas(*iargs, _stream()), "qa_greedy_init_deltas")
    check(L.qa_greedy_init_sums_range(*iargs, 0, nt, _stream()), "qa_greedy_init_sums_range")
    pargs = (_ptr(table), nt, float(numel), METRIC_CODE[metric], float(threshold), order, nf, _ptr(rng), _ptr(assignment),
             _ptr(counts), _ptr(state), _ptr(work), _ptr(pre_order), _ptr(rngs[1]), _ptr(init))
    cur.wait_event(ev_a2)
    if three:
        check(L.qa_greedy_assign_passes(*pargs, 0, 2, 0, _stream()), "qa_greedy_assign_passes")
        cur.wait_event(ev_a3)
        check(L.qa_greedy_assign_passes(*pargs, 2, nf, 0, _stream()), "qa_greedy_assign_passes")
    else:
        check(L.qa_greedy_assign_passes(*pargs, 0, nf, 0, _stream()), "qa_greedy_assign_passes")
    for t in (work, init, jarr, pre_order, rngs, awork):       # buffers used on side streams: keep them until `cur` is past
        t.record_stream(side)
        t.record_stream(side2)
    return assignment, counts, state


def threshold_assign(scores_metric: torch.Tensor, order_fmts, is_pcc: bool, thresholds) -> tuple[torch.Tensor, torch.Tensor]:
    """scores_metric float32 [NFMT, ntiles]; thresholds: iterable of floats (cast to float32 like NumPy 2).
    -> (assignment int8 [nthr, ntiles], counts int64 [nthr, 4])."""
    nt = scores_metric.shape[1]
    dev = scores_metric.device
    thr = torch.tensor(np.asarray(list(thresholds), dtype=np.float32), device=dev)
    nthr = thr.numel()
    assignment = torch.empty((nthr, nt), dtype=torch.int8, device=dev)
    counts = torch.zeros((nthr, NFMT), dtype=torch.int64, device=dev)
    order = _lib.int32_array([FMT_INDEX[f] for f in order_fmts])
    check(_lib.lib().qa_threshold_assign(_ptr(scores_metric), nt, order, len(order_fmts), 1 if is_pcc else 0, _ptr(thr), nthr,
                                         _ptr(assignment), _ptr(counts), _stream()), "qa_threshold_assign")
    return assignment, counts


def random_samples(table: torch.Tensor, numel: int, fmt_list, iters: int, rng: torch.Tensor):
    """-> (choices int8 [iters, ntiles], metrics f64 [iters, 3], counts int64 [iters, 4])."""
    nt = table.shape[1]
    dev = table.device
    k = len(fmt_list)
    choices = torch.empty((iters, nt), dtype=torch.int8, device=dev)
    ready = 0
    if k & (k - 1):  # rejection sampling possible: draw sequentially on device, then map to format indices
        raw = numpy_integers(rng, k, iters * nt)
        lut = torch.tensor([FMT_INDEX[f] for f in fmt_list], dtype=torch.int8, device=dev)
        choices = lut[raw.long()].reshape(iters, nt).contiguous()
        ready = 1
    metrics = torch.zeros((iters, 3), dtype=torch.float64, device=dev)
    counts = torch.zeros((iters, NFMT), dtype=torch.int64, device=dev)
    idx = _lib.int32_array([FMT_INDEX[f] for f in fmt_list])
    check(_lib.lib().qa_random_samples(_ptr(table), nt, float(numel), idx, k, iters, _ptr(rng), _ptr(choices), ready,
                                       _ptr(metrics), _ptr(counts), _stream()), "qa_random_samples")
    return choices, metrics, counts


def apply_assignment(p: Prepared, assignment: torch.Tensor) -> torch.Tensor:
    out = torch.empty(p.rows * p.cols, dtype=torch.bfloat16, device=p.data.device)
    a = assignment.to(torch.int8).contiguous().reshape(-1)
    check(_lib.lib().qa_apply_assignment(_ptr(p.data), p.dtype_code, p.rows, p.cols, p.cols, _ptr(a), _ptr(out), _stream()),
          "qa_apply_assignment")
    return out


def assignment_sums(table: torch.Tensor, assignment: torch.Tensor | None = None, fmt: int = -1) -> torch.Tensor:
    out = torch.zeros(8, dtype=torch.float64, device=table.device)
    a = None if assignment is None else assignment.to(torch.int8).contiguous().reshape(-1)
    check(_lib.lib().qa_assignment_sums(_ptr(table), table.shape[1], _ptr(a), int(fmt), _ptr(out), _stream()),
          "qa_assignment_sums")
    return out


def assignment_sums_batch(table: torch.Tensor, maps: torch.Tensor) -> torch.Tensor:
    """Whole-tensor sums of every row of `maps` (int8 [nmaps, ntiles]) in one launch -> float64 [nmaps, 8]."""
    m = maps.to(torch.int8).contiguous()
    out = torch.zeros((m.shape[0], 8), dtype=torch.float64, device=table.device)
    check(_lib.lib().qa_assignment_sums_batch(_ptr(table), table.shape[1], _ptr(m), m.shape[0], _ptr(out), _stream()),
          "qa_assignment_sums_batch")
    return out


def pair_sums(a, b=None) -> tuple[np.ndarray, int]:
    """{sum a, sum a^2, sum b, sum b^2, sum ab, sum|a-b|, max|a-b|} over two arrays (b=None: zeros), float64."""
    dev = _require_cuda()

    def as_f32(t):
        if isinstance(t, torch.Tensor):
            return t.detach().to(device=dev, dtype=torch.float32).contiguous().reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(np.asarray(t, dtype=np.float32))).to(dev).reshape(-1)

    ta = as_f32(a)
    tb = None if b is None else as_f32(b)
    if tb is not None and tb.numel() != ta.numel():
        raise ValueError("pair_sums: size mismatch")
    L = _lib.lib()
    out = torch.zeros(8, dtype=torch.float64, device=dev)
    work = torch.empty(L.qa_pair_sums_work_bytes(), dtype=torch.uint8, device=dev)
    if ta.numel():
        check(L.qa_pair_sums(_ptr(ta), _ptr(tb), ta.numel(), _ptr(out), _ptr(work), _stream()), "qa_pair_sums")
    return out.cpu().numpy(), int(ta.numel())


def metrics_from_sums(s, numel: int) -> dict:
    """pcc / mae / atol from {sx, sx2, sy, sy2, sxy, sabs, max}: float64 recombination of the
    formulas in metrics.py:6-27 (the mathematically exact value the reference's float32 approximates)."""
    sx, sx2, sy, sy2, sxy, sabs, amax = [float(v) for v in s[:7]]
    n = float(numel)
    if n == 0:
        return {"pcc": 1.0, "mae": 0.0, "atol": 0.0}
    am2 = max(sx2 - sx * sx / n, 0.0)
    bm2 = max(sy2 - sy * sy / n, 0.0)
    den = math.sqrt(am2 * bm2)
    if den == 0.0:
        pcc = 1.0 if amax == 0.0 else 0.0
    else:
        pcc = (sxy - sx * sy / n) / den
    return {"pcc": pcc, "mae": sabs / n, "atol": amax}


def result_to_numpy(p: Prepared, y_bf16: torch.Tensor) -> np.ndarray:
    """Device bf16 reconstruction in p's geometry -> float32 ndarray of the original shape."""
    y = y_bf16.reshape(-1)
    if p.kind == "vector" and y.numel() != p.numel:
        y = y[: p.numel]
    return y.to(torch.float32).cpu().numpy().reshape(p.shape)


# --------------------------------------------------------------------------------------------
# whole-tensor NumPy-float32-faithful scores (metrics.py:6-27 as wq:684-687 evaluates them)
# --------------------------------------------------------------------------------------------
_PLANS: dict = {}


def candidate_chunk(per: int, wanted: int, device) -> int:
    """How many bf16 reconstructions of `per` elements to materialise and score per qa_tensor_scores_f32 call: each call costs
    one chain latency (n / 64 dependent FMAs) whatever the batch, so the batch takes up to half of the free HBM (<= 48 GiB)
    rather than a fixed few GiB - 180 GB of HBM3e is what makes a 1000-sample run a handful of calls."""
    free, _total = torch.cuda.mem_get_info(device)
    budget = min(48 << 30, free // 2)
    return int(max(1, min(wanted, budget // max(2 * per, 1))))


def pairwise_plan_host(n: int) -> np.ndarray:
    """Shape of np.add.reduce's pairwise-summation tree over n contiguous elements (qa_pairwise_plan_build; host only)."""
    L = _lib.lib()
    words = L.qa_pairwise_plan_words(int(n))
    plan = np.zeros(max(words, 4), dtype=np.int32)
    check(L.qa_pairwise_plan_build(int(n), plan.ctypes.data), "qa_pairwise_plan_build")
    return plan


def _plan(n: int, dev: torch.device):
    key = (int(n), dev.index)
    if key not in _PLANS:
        if len(_PLANS) > 32:
            _PLANS.clear()
        host = pairwise_plan_host(n)
        _PLANS[key] = (host, torch.from_numpy(host).to(dev))
    return _PLANS[key]


def tensor_scores_f32(x: torch.Tensor, y: torch.Tensor | None, n: int | None = None) -> np.ndarray:
    """float32 {pcc, mae, atol, mean(y)} of `y` against `x`, bit-faithful to the reference's NumPy evaluation on the
    flattened tensors.  x: device tensor (bf16 / float32), its first n elements are scored; y: None (all zeros = fp0), a
    tensor of >= n elements, or a [nbatch, m >= n] tensor of candidates scored in one call.  -> float32 [nbatch, 4]."""
    dev = x.device
    L = _lib.lib()
    xf = x.reshape(-1)
    n = int(xf.numel() if n is None else n)
    if n <= 0:
        raise ValueError("tensor_scores_f32: empty input")
    code = lambda t: QA_DT_BF16 if t.dtype == torch.bfloat16 else QA_DT_F32      # noqa: E731
    if xf.dtype not in (torch.bfloat16, torch.float32):
        xf = xf.float()
    if y is None:
        nb, stride, yp, ydt = 1, 0, None, QA_DT_F32
    else:
        if y.dtype not in (torch.bfloat16, torch.float32):
            y = y.float()
        y2 = y.reshape(1, -1) if y.dim() <= 1 or y.numel() == xf.numel() else y.reshape(y.shape[0], -1)
        y2 = y2.contiguous()
        nb, stride, yp, ydt = y2.shape[0], y2.shape[1], y2, code(y2)
        if stride < n:
            raise ValueError("tensor_scores_f32: y is shorter than x")
    host, plan = _plan(n, dev)
    out = torch.empty((nb, 4), dtype=torch.float32, device=dev)
    work = torch.empty(L.qa_tensor_scores_work_bytes(int(host[2]), nb), dtype=torch.uint8, device=dev)
    check(L.qa_tensor_scores_f32(_ptr(xf), code(xf), _ptr(yp), ydt, stride, nb, n, _ptr(plan), host.ctypes.data, _ptr(out), _ptr(work),
                                 _stream()), "qa_tensor_scores_f32")
    return out.cpu().numpy()
