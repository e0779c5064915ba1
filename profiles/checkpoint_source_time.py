"""wq over a local fp8 checkpoint (--checkpoint-dir) against wq over the same tensors as the reference's float32 cache.

Writes, into a temporary directory removed afterwards, the five layer-0 attention weights of DeepSeek-R1 as an fp8 checkpoint
(synthetic.fp8_checkpoint_cpu: e4m3fn bytes + 128 x 128 F32 block scales, one shard per weight + model.safetensors.index.json)
and the same tensors as the reference's float32 cache (dequantized on the CPU with torch, as the reference's loader does).
Then times `wq` with compression_configs/greedy.json (mixed-tile-greedy, pcc >= 0.999, seed 123) over both routes in one
process, alternating them, and reports wall time per route and per tensor (load + evaluation, device synchronised), the
bytes each route reads from its files, and whether the two result trees are identical.  The processed-array cache of the
`none` baseline is not written (--no-save-processed): that write is the same for both routes.

    python profiles/checkpoint_source_time.py [--reps 3]
"""
import argparse
import contextlib
import io
import json
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from safetensors.torch import save_file  # noqa: E402

from quantization_analysis_b200 import synthetic, tensor_source, wq  # noqa: E402
from tests.cli_util import compare_trees  # noqa: E402

REPO = "local/DeepSeek-R1-attention"
CONFIG = ROOT / "compression_configs" / "greedy.json"


def write_sources(tmp: Path) -> tuple[Path, Path, dict]:
    """-> (checkpoint dir, float32 cache dir, {name: (checkpoint bytes, cache bytes)})."""
    ckpt, cache = tmp / "ckpt", tmp / "hf-cache"
    ckpt.mkdir()
    d = cache / "tensor-fp32" / tensor_source.safe_repo_revision_key(REPO, "main")
    d.mkdir(parents=True)
    weight_map, sizes = {}, {}
    for i, name in enumerate(synthetic.ATTN_NAMES):
        w, s = synthetic.fp8_checkpoint_cpu(synthetic.DEEPSEEK_R1_SHAPES[name], 100 + i)
        w = w.view(torch.float8_e4m3fn)
        shard = f"model-{i + 1:05d}-of-{len(synthetic.ATTN_NAMES):05d}.safetensors"
        save_file({name: w, f"{name}_scale_inv": s}, str(ckpt / shard), metadata={"format": "pt"})
        weight_map[name] = weight_map[f"{name}_scale_inv"] = shard
        npy = d / f"{tensor_source.safe_tensor_key(name)}.npy"
        np.save(npy, tensor_source.Fp8Blocks(w, s).dequantize_cpu())
        sizes[name] = ((ckpt / shard).stat().st_size, npy.stat().st_size)
    (ckpt / tensor_source.CHECKPOINT_INDEX).write_text(json.dumps({"metadata": {}, "weight_map": weight_map}, indent=2))
    return ckpt, cache, sizes


class PerTensorClock:
    """Wall time of TensorIndex.load + wq.evaluate_tensor per tensor, each ending in a device synchronise."""

    def __init__(self):
        self.t: dict[str, float] = {}
        self._load, self._eval = tensor_source.TensorIndex.load, wq.evaluate_tensor
        clock = self

        def load(index, name):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            x = clock._load(index, name)
            clock.t[name] = clock.t.get(name, 0.0) + time.perf_counter() - t0
            return x

        def evaluate(name, *a, **k):
            t0 = time.perf_counter()
            out = clock._eval(name, *a, **k)
            torch.cuda.synchronize()
            clock.t[name] = clock.t.get(name, 0.0) + time.perf_counter() - t0
            return out
        tensor_source.TensorIndex.load, wq.evaluate_tensor = load, evaluate

    def restore(self):
        tensor_source.TensorIndex.load, wq.evaluate_tensor = self._load, self._eval


def run_wq(tmp: Path, route: str, k: int, ckpt: Path, cache: Path) -> tuple[float, dict, Path]:
    root = tmp / "results" / route / str(k)
    argv = [REPO, "model.layers.0", "--compression-config", str(CONFIG), "--recompute", "--summary", "--no-save-processed",
            "--results-root", str(root), "--processed-root", str(tmp / "processed" / route), "--cache-dir", str(cache)]
    if route == "checkpoint":
        argv += ["--checkpoint-dir", str(ckpt)]
    clock = PerTensorClock()
    try:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            assert wq.run(argv) == 0
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    finally:
        clock.restore()
    base = root / REPO.replace("/", "__") / "mixed-tile-greedy"
    return wall, clock.t, sorted(base.iterdir())[-1]


def gpu_power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print(f"GPU: {torch.cuda.get_device_name()}, power limit {gpu_power_limit()}")
    tmp = Path(tempfile.mkdtemp(prefix="ckpt_source_"))
    try:
        ckpt, cache, sizes = write_sources(tmp)
        routes = ("checkpoint", "fp32-cache")
        for route in routes:                                         # warm-up: library load, plans, allocator
            run_wq(tmp, route, -1, ckpt, cache)
        walls = {r: [] for r in routes}
        per = {r: {n: [] for n in synthetic.ATTN_NAMES} for r in routes}
        trees = {}
        for k in range(args.reps):
            for route in (routes if k % 2 == 0 else routes[::-1]):
                wall, t, tree = run_wq(tmp, route, k, ckpt, cache)
                walls[route].append(wall)
                for n in synthetic.ATTN_NAMES:
                    per[route][n].append(t[n])
                trees[route, k] = tree
        identical = all(compare_trees(trees["checkpoint", k], trees["fp32-cache", k]) == []
                        and compare_trees(trees["fp32-cache", k], trees["checkpoint", k]) == [] for k in range(args.reps))
        print(f"wq {CONFIG.name} over {len(synthetic.ATTN_NAMES)} tensors ({sum(int(np.prod(synthetic.DEEPSEEK_R1_SHAPES[n])) for n in synthetic.ATTN_NAMES) / 1e6:.1f} M elements), "
              f"{args.reps} timed runs per route, alternating")
        print(f"result trees identical (every run): {identical}")
        print()
        print(f"{'route':<12} {'wall s (each run)':<30} {'median s':>9} {'bytes read from files':>22}")
        for i, route in enumerate(routes):
            nbytes = sum(v[i] for v in sizes.values())
            print(f"{route:<12} {', '.join(f'{w:.3f}' for w in walls[route]):<30} {statistics.median(walls[route]):>9.3f} {nbytes:>22,}")
        print()
        print(f"{'tensor':<52} {'shape':>14} {'ckpt s':>8} {'cache s':>8} {'ckpt B':>13} {'cache B':>13}")
        for n in synthetic.ATTN_NAMES:
            shp = "x".join(str(v) for v in synthetic.DEEPSEEK_R1_SHAPES[n])
            print(f"{n:<52} {shp:>14} {statistics.median(per['checkpoint'][n]):>8.3f} {statistics.median(per['fp32-cache'][n]):>8.3f} "
                  f"{sizes[n][0]:>13,} {sizes[n][1]:>13,}")
        print("\nper tensor: median over the timed runs of TensorIndex.load + wq.evaluate_tensor (device synchronised); bytes are "
              "the sizes of the files each route reads (shard, or .npy), served from the page cache after the first run")
        return 0 if identical else 1
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    raise SystemExit(main())
