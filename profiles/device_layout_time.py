"""What the device layout (``"transpose": true``) costs on o_proj (DeepSeek-R1 layer 0, 7168 x 16384): the copy itself and
the mixed-tile runs with and without the flag.

1. qa_transpose_2d on the bf16 weight (2 B / element) and on the fp8 e4m3fn bytes (1 B / element) plus their 128 x 128 scale
   grid: CUDA-event time per call (median of 20, after warm-up) and the bytes moved (read + write) over that time, next to
   the device-to-device copy rate of the same buffer (torch copy_, i.e. cudaMemcpyAsync) measured the same way.  The
   buffers (235 MB / 117 MB) are larger than the 126 MB L2 once read and written.
2. MixedTileGreedyCompression.run_prepared (pcc >= 0.999, seed 123, bf16 > bfp8 > bfp4 > bfp2) and
   MixedTileThresholdCompression.run_prepared (pcc >= 0.999) on the device-resident tensor, unflagged against flagged.
   The flagged time is split into the transposition of x (engine.prepare_transposed of the resident Prepared), the run
   on x.T, and the reconstruction in x's layout (DeviceResult.y_device: apply on x.T, then the transposition back, timed
   apart).  Host clock around
   work that ends in a device synchronise, median of 5 after one warm-up; the two variants alternate.
3. The same for the fp8 form (Fp8Prepared: the greedy's table comes from the bytes; the threshold scores read the
   float32 image, which the run materialises).

    python profiles/device_layout_time.py
"""
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from quantization_analysis_b200 import engine, synthetic  # noqa: E402
from quantization_analysis_b200.compression_algorithms import create_algorithm  # noqa: E402

NAME = "model.layers.0.self_attn.o_proj.weight"
FMTS = ["bf16", "bfp8", "bfp4", "bfp2"]


def gpu_power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def event_ms(fn, reps: int = 20) -> float:
    for _ in range(3):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def wall_ms(fn) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def copy_rows(label: str, t: torch.Tensor) -> None:
    nbytes = t.numel() * t.element_size()
    dst = torch.empty_like(t)
    tt = event_ms(lambda: engine.transpose_2d(t))
    tc = event_ms(lambda: dst.copy_(t))
    gt, gc = 2 * nbytes / tt / 1e6, 2 * nbytes / tc / 1e6
    print(f"{label:<34} {nbytes / 1e6:>9.1f} {tt:>10.3f} {gt:>9.0f} {tc:>10.3f} {gc:>9.0f} {gt / gc:>8.2f}")


def times_only(out: dict) -> dict:
    """Drop a run's tensors, so that every repetition reuses the allocator's cached blocks (a retained 235 MB result makes
    the next one a fresh cudaMalloc, which would be timed with the kernel)."""
    return {k: v for k, v in out.items() if isinstance(v, float)}


def run_pair(label: str, p: engine.Prepared, algo: str, params: dict, reps: int = 5) -> None:
    plain = create_algorithm(algo, dict(params))
    flagged = create_algorithm(algo, {**params, "transpose": True})

    def once_plain():
        if isinstance(p, engine.Fp8Prepared):
            p._data = None            # both variants materialise their float32 image, as a fresh tensor would
        out = {}
        out["run"] = wall_ms(lambda: out.__setitem__("dr", plain.run_prepared(p, FMTS)))
        out["apply"] = wall_ms(lambda: out.__setitem__("y", engine.apply_assignment(p, out["dr"].assignment)))
        out["yT"] = 0.0
        return times_only(out)

    def once_flagged():
        out = {}
        out["xt"] = wall_ms(lambda: out.__setitem__("pt", engine.prepare_transposed(p)))
        out["run"] = wall_ms(lambda: out.__setitem__("dr", flagged.run_prepared(out["pt"], FMTS)))
        pt = out["pt"]          # DeviceResult.y_device in its two steps: apply on x.T, then the transposition back
        out["apply"] = wall_ms(lambda: out.__setitem__("y", engine.apply_assignment(pt, out["dr"].assignment)))
        out["yT"] = wall_ms(lambda: engine.transpose_2d(out["y"].reshape(pt.rows, pt.cols)))
        return times_only(out)

    once_plain(), once_flagged()
    rp, rf = [], []
    for k in range(reps):
        for which in ((0, 1) if k % 2 == 0 else (1, 0)):
            if which == 0:
                rp.append(once_plain())
            else:
                rf.append(once_flagged())
    med = lambda rows, k: statistics.median(r[k] for r in rows)      # noqa: E731
    tp = med(rp, "run") + med(rp, "apply")
    tf = med(rf, "xt") + med(rf, "run") + med(rf, "apply") + med(rf, "yT")
    print(f"{label:<30} {'-':>8} {med(rp, 'run'):>9.2f} {med(rp, 'apply'):>8.2f} {'-':>8} {tp:>9.2f}   unflagged")
    print(f"{'':<30} {med(rf, 'xt'):>8.2f} {med(rf, 'run'):>9.2f} {med(rf, 'apply'):>8.2f} {med(rf, 'yT'):>8.2f} {tf:>9.2f}   "
          f"transposed ({tf / tp:.2f}x)")
    torch.cuda.empty_cache()


def main() -> int:
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.cuda.set_device(0)
    shape = synthetic.DEEPSEEK_R1_SHAPES[NAME]
    print(f"GPU: {torch.cuda.get_device_name()}, power limit {gpu_power_limit()}")
    print(f"tensor: {NAME} {shape[0]}x{shape[1]} ({np.prod(shape) / 1e6:.1f} M elements)")
    xb = synthetic.randn_bf16_cpu(shape, 100)
    w, s = synthetic.fp8_checkpoint_cpu(shape, 101)
    p_bf16 = engine.prepare_loaded(xb)
    p_fp8 = engine.Fp8Prepared(w.view(torch.float8_e4m3fn), s)
    torch.cuda.synchronize()

    print("\n1. qa_transpose_2d (CUDA events, median of 20; GB/s = (read + write) bytes / time)")
    print(f"{'operand':<34} {'MB':>9} {'T ms':>10} {'T GB/s':>9} {'copy ms':>10} {'copy GB/s':>9} {'T/copy':>8}")
    copy_rows("bf16 weight [7168, 16384]", p_bf16.data.reshape(shape))
    copy_rows("fp8 bytes [7168, 16384]", p_fp8.w8)
    copy_rows("fp8 scale grid [56, 128] float32", p_fp8.scale_inv)

    print("\n2./3. mixed-tile runs on the resident tensor (ms; host clock + synchronise, median of 5, variants alternating)")
    print(f"{'run':<30} {'x.T':>8} {'run':>9} {'apply':>8} {'y.T':>8} {'total':>9}")
    run_pair("greedy pcc 0.999, bf16", p_bf16, "mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 123})
    run_pair("threshold pcc 0.999, bf16", p_bf16, "mixed-tile-threshold", {"metric": "pcc", "threshold": 0.999})
    run_pair("greedy pcc 0.999, fp8", p_fp8, "mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 123})
    run_pair("threshold pcc 0.999, fp8", p_fp8, "mixed-tile-threshold", {"metric": "pcc", "threshold": 0.999})
    print("\nx.T: engine.prepare_transposed of the resident tensor (bf16: one qa_transpose_2d; fp8: the bytes and the scale "
          "grid); run: run_prepared; apply: qa_apply_assignment of the map (fp8: on the float32 image, materialised here by the "
          "greedy); y.T: the transposition of y back to x's layout")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
