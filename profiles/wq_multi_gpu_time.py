"""wq over a DeepSeek-R1-layout fp8 checkpoint: in one process against `--gpus N` (N = 1, 2, 4, 8, capped at the visible
devices).

Writes, into a temporary directory removed afterwards, 64 routed experts of one MoE layer (gate / up / down, 192 matrices,
2.82 G elements) as DeepSeek-R1 stores them (synthetic.fp8_checkpoint_cpu: e4m3fn bytes + 128 x 128 F32 weight_scale_inv,
one shard per expert + model.safetensors.index.json).  Runs `wq --checkpoint-dir` with compression_configs/greedy.json
(mixed-tile-greedy, pcc >= 0.999) once untimed, so the shards are in the page cache and this process has loaded the library,
then every arm twice, alternating.  The in-process arm runs in this already warm process; a `--gpus N` arm starts N
fresh worker processes, each importing torch and initialising CUDA.  Per run it reports the wall time, split at the first
tensor result the parent receives (start-up: for --gpus N the spawn, torch import and CUDA init of the workers plus one
tensor), and whether the run's result tree equals the first in-process run's up to TIME(s).  The processed-array cache of
the `none` baseline is not written (--no-save-processed): it would be 2.82 G float32 elements per format.

    python profiles/wq_multi_gpu_time.py [--experts 64] [--reps 2]
"""
import argparse
import contextlib
import io
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402
from safetensors.torch import save_file  # noqa: E402

from quantization_analysis_b200 import multi_gpu, synthetic, wq  # noqa: E402
from quantization_analysis_b200.tensor_source import CHECKPOINT_INDEX  # noqa: E402
from tests.cli_util import compare_trees  # noqa: E402

REPO = "local/DeepSeek-R1-experts"
CONFIG = ROOT / "compression_configs" / "greedy.json"
LAYER = 3


def write_checkpoint(d: Path, experts: int) -> int:
    """-> elements written."""
    d.mkdir(parents=True)
    weight_map, numel = {}, 0
    per_expert = len(synthetic.EXPERT_SHAPES)
    tensors = synthetic.expert_tensor_list(experts, LAYER)
    for e in range(experts):
        shard = f"model-{e + 1:05d}-of-{experts:05d}.safetensors"
        contents = {}
        for i, (name, shape) in enumerate(tensors[e * per_expert:(e + 1) * per_expert]):
            w, s = synthetic.fp8_checkpoint_cpu(shape, 7000 + e * per_expert + i)
            contents[name], contents[f"{name}_scale_inv"] = w.view(torch.float8_e4m3fn), s
            numel += shape[0] * shape[1]
        save_file(contents, str(d / shard), metadata={"format": "pt"})
        weight_map.update(dict.fromkeys(contents, shard))
    (d / CHECKPOINT_INDEX).write_text(json.dumps({"metadata": {}, "weight_map": weight_map}, indent=2))
    return numel


class FirstResult:
    """Time of the first tensor result the parent receives: wq.run_tensor returning in process, the first message of any
    worker under --gpus."""

    def __init__(self, gpus):
        self.t = None
        self.gpus = gpus

    def __enter__(self):
        clock = self
        if self.gpus is None:
            self._saved = ("run_tensor", wq.run_tensor)
            orig = wq.run_tensor

            def run_tensor(job, name):
                out = orig(job, name)
                if clock.t is None:
                    torch.cuda.synchronize()
                    clock.t = time.perf_counter()
                return out
            wq.run_tensor = run_tensor
        else:
            self._saved = ("_receive", multi_gpu._receive)
            orig = multi_gpu._receive

            def receive(*a):
                for msg in orig(*a):
                    if clock.t is None:
                        clock.t = time.perf_counter()
                    yield msg
            multi_gpu._receive = receive
        return self

    def __exit__(self, *exc):
        mod = wq if self._saved[0] == "run_tensor" else multi_gpu
        setattr(mod, *self._saved)


def run_wq(tmp: Path, ckpt: Path, arm: str, k: int):
    gpus = None if arm == "in-process" else int(arm.split()[-1])
    root = tmp / "results" / arm.replace(" ", "") / str(k)
    argv = [REPO, f"model.layers.{LAYER}", "--compression-config", str(CONFIG), "--recompute", "--no-save-processed",
            "--summary", "--checkpoint-dir", str(ckpt), "--results-root", str(root), "--processed-root", str(tmp / "processed")]
    if gpus is not None:
        argv += ["--gpus", str(gpus)]
    with FirstResult(gpus) as first:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            rc = wq.run(argv)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    assert rc == 0, arm
    tree = sorted((root / REPO.replace("/", "__") / "mixed-tile-greedy").iterdir())[-1]
    return wall, first.t - t0, tree


def gpu_info() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True,
                             timeout=30)
        return out.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--experts", type=int, default=64)
    ap.add_argument("--reps", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    visible = torch.cuda.device_count()
    print(f"visible CUDA devices: {visible}")
    print(gpu_info())
    arms = ["in-process"] + [f"--gpus {n}" for n in (1, 2, 4, 8) if n <= visible]
    tmp = Path(tempfile.mkdtemp(prefix="wq_multi_gpu_"))
    try:
        t0 = time.perf_counter()
        numel = write_checkpoint(tmp / "ckpt", args.experts)
        print(f"checkpoint: {3 * args.experts} fp8 matrices, {numel / 1e9:.2f} G elements, "
              f"{sum(f.stat().st_size for f in (tmp / 'ckpt').iterdir()) / 1e9:.2f} GB, written in {time.perf_counter() - t0:.0f} s")
        print(f"wq {CONFIG.name} --checkpoint-dir --no-save-processed; one untimed in-process run, then {args.reps} runs per arm, "
              f"alternating")
        run_wq(tmp, tmp / "ckpt", "in-process", -1)
        runs = {a: [] for a in arms}
        for k in range(args.reps):
            for arm in (arms if k % 2 == 0 else arms[::-1]):
                runs[arm].append(run_wq(tmp, tmp / "ckpt", arm, k))
        ref = runs["in-process"][0][2]
        print()
        print(f"{'arm':<12} {'run':>3} {'wall s':>8} {'start-up s':>11} {'rest s':>8} {'tree == in-process':>19}")
        equal_all = True
        for arm in arms:
            for k, (wall, first, tree) in enumerate(runs[arm]):
                equal = compare_trees(tree, ref) == [] and compare_trees(ref, tree) == []
                equal_all &= equal
                print(f"{arm:<12} {k:>3} {wall:>8.2f} {first:>11.2f} {wall - first:>8.2f} {str(equal):>19}")
        print(f"\nevery result tree equal to the in-process run's up to TIME(s): {equal_all}")
        print("start-up: from the call of wq.run to the first tensor result in the parent (--gpus N: worker spawn, torch import, "
              "CUDA init, library load and one tensor; in-process: one tensor in an already warm process)")
        return 0 if equal_all else 1
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    raise SystemExit(main())
