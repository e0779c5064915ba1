"""qa_transpose_2d (the copy behind the device layout): out [cols, rows] == x.t() for 1-, 2- and 4-byte elements, on tiny,
ragged and padded shapes, with `ld > cols` and odd base offsets, and with every byte around the output poisoned and
checked afterwards."""
import numpy as np
import pytest
import torch

from quantization_analysis_b200 import _lib, engine

NP = {1: np.uint8, 2: np.uint16, 4: np.uint32}
GUARD = 0xA5
SHAPES = [(1, 1), (1, 77), (77, 1), (33, 70), (70, 45), (64, 64), (65, 129), (200, 3), (4, 260), (130, 96)]


def _run(a: np.ndarray, ld: int, off: int, out_off: int) -> tuple[np.ndarray, np.ndarray]:
    """x = a placed at element `off` of a poisoned buffer with row stride `ld`; out at element `out_off` of a GUARD-filled
    buffer.  -> (out [cols, rows] as read back, the whole output buffer's bytes)."""
    rows, cols = a.shape
    e = a.dtype.itemsize
    rng = np.random.default_rng(rows * 1000 + cols)
    xb = rng.integers(0, 256, size=(off + rows * ld + 16) * e, dtype=np.uint8)      # whatever lies between the rows
    view = xb[off * e: (off + rows * ld) * e].view(a.dtype).reshape(rows, ld)
    view[:, :cols] = a
    xd = torch.from_numpy(xb).cuda()
    ob = torch.full(((out_off + rows * cols + 16) * e,), GUARD, dtype=torch.uint8, device="cuda")
    L = _lib.lib()
    _lib.check(L.qa_transpose_2d(xd.data_ptr() + off * e, e, rows, cols, ld, ob.data_ptr() + out_off * e,
                                 torch.cuda.current_stream().cuda_stream), "qa_transpose_2d")
    host = ob.cpu().numpy()
    out = host[out_off * e: (out_off + rows * cols) * e].view(a.dtype).reshape(cols, rows)
    return out, host


@pytest.mark.gpu
@pytest.mark.parametrize("elem", [1, 2, 4])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_transpose_equals_torch_t(elem, shape):
    rows, cols = shape
    rng = np.random.default_rng(elem * 7 + rows + cols)
    a = rng.integers(0, 2 ** (8 * elem), size=shape, dtype=np.uint64).astype(NP[elem])
    want = torch.from_numpy(a.astype(np.int64)).t().contiguous().numpy().astype(NP[elem])
    # (ld, x offset, out offset): packed and aligned (the vector path), padded rows, odd offsets (the element path)
    for ld, off, out_off in ((cols, 0, 0), (cols + 4, 4, 8), (cols + 1, 1, 3), (cols + 33, 3, 1)):
        out, host = _run(a, ld, off, out_off)
        assert np.array_equal(out, want), (ld, off, out_off)
        e = a.dtype.itemsize
        assert (host[: out_off * e] == GUARD).all() and (host[(out_off + rows * cols) * e:] == GUARD).all(), (ld, off, out_off)


@pytest.mark.gpu
def test_transpose_of_device_tensors_and_bad_arguments():
    """engine.transpose_2d on bf16 / float32 / uint8 device tensors (strided views included) == .t().contiguous(); an
    elem_bytes other than 1, 2, 4 and an ld below cols are rejected with a message, and nothing is written."""
    g = torch.Generator(device="cpu").manual_seed(3)
    base = torch.randn((150, 300), generator=g)
    for t in (base.to(torch.bfloat16), base, (base * 50).to(torch.int16).to(torch.uint8)):
        d = t.cuda()
        assert torch.equal(engine.transpose_2d(d), d.t().contiguous())
        v = d[5:100, 7:250]                                              # ld = 300 > cols, offset base
        assert torch.equal(engine.transpose_2d(v), v.t().contiguous())
    L = _lib.lib()
    x = torch.zeros(64, dtype=torch.uint8, device="cuda")
    out = torch.full((64,), GUARD, dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    for eb in (0, 3, 8, -1):
        assert L.qa_transpose_2d(x.data_ptr(), eb, 4, 4, 4, out.data_ptr(), s) != 0
        assert b"elem_bytes" in L.qa_last_error()
    assert L.qa_transpose_2d(x.data_ptr(), 1, 4, 8, 4, out.data_ptr(), s) != 0
    assert L.qa_transpose_2d(x.data_ptr(), 2, 0, 5, 5, out.data_ptr(), s) == 0     # empty: nothing to do
    torch.cuda.synchronize()
    assert (out.cpu().numpy() == GUARD).all()
