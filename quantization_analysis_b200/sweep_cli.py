"""Threshold-sweep CLI (scripts/sweep_mixed_tile_threshold.py:36-102, 581-841 of the reference): same arguments, same
``details/<tensor>/sweep_config.json`` + ``sweep_results.csv``; the plots (matplotlib) are out of scope.

    python -m quantization_analysis_b200.sweep_cli <repo_or_url> <tensor_name> [--no-regex] [--metric pcc|mae|atol]
           [--lowest-metric-val V] [--steps N] [--formats bf16,bfp8,bfp4,bfp2] [--out-dir DIR] [--checkpoint-dir DIR] [--gpus N]

Tensors come from ``tensor_source`` like wq's: the shards of ``--checkpoint-dir`` when given, else the float32 cache.  With
``--gpus N`` the matched tensors are split over N GPUs of the node like wq's (``multi_gpu``); the files are the same.
"""
from __future__ import annotations

import argparse
import contextlib
import fnmatch
import math
import re
import sys
import time
from dataclasses import dataclass
from pathlib import Path

from . import multi_gpu, sweep, tensor_source
from .compression_algorithms.tile_utils import MIXED_TILE_FORMATS


def _parse_formats(value: str) -> list[str]:
    out = []
    for part in (p.strip().lower() for p in value.split(",")):
        if not part:
            continue
        if part not in MIXED_TILE_FORMATS:
            raise ValueError(f"Unsupported mixed-tile format: {part}")
        if part not in out:
            out.append(part)
    if not out:
        raise ValueError("No valid mixed-tile formats selected.")
    return out


def select_tensors(index, query: str, use_regex: bool) -> list[str]:
    """sweep:313-345: regex search (default), exact name, fnmatch pattern, then the wq filter."""
    names = list(index.tensor_to_file)
    weight_like = [n for n in names if "weight" in n.lower() and not n.lower().endswith("_scale_inv")]
    cand = weight_like if weight_like else names
    if use_regex:
        try:
            pat = re.compile(query)
        except re.error as exc:
            raise RuntimeError(f"Invalid regex '{query}': {exc}") from exc
        hits = [n for n in cand if pat.search(n)]
        if hits:
            return sorted(hits)
        raise RuntimeError("No tensors matched the regex query.")
    if query in cand:
        return [query]
    if any(ch in query for ch in "*?[]"):
        hits = [n for n in cand if fnmatch.fnmatch(n, query)]
        if hits:
            return sorted(hits)
    return tensor_source.filter_tensor_names(cand, query)


@dataclass
class SweepJob:
    """Everything the per-tensor sweep needs besides the tensor's name; under --gpus, pickled to every worker."""
    index: tensor_source.TensorIndex
    detail: Path
    repo_or_url: str
    revision: str
    backend: str
    formats: list[str]
    metric: str
    lowest: float
    steps: int


def sweep_one(job: SweepJob, name: str) -> str | None:
    """Sweep one tensor and write its ``details/<tensor>/`` files.  -> None, or the message of its SweepRangeError (nothing
    is written for that tensor)."""
    x = job.index.load(name)
    try:
        rows, _maps = sweep.sweep_tensor(x, job.formats, job.metric, job.steps, job.lowest)
    except sweep.SweepRangeError as exc:
        return str(exc)
    out = job.detail / name.replace("/", "_").replace(".", "_")
    sweep.write_sweep_config(out, job.repo_or_url, name, job.revision, job.backend, job.formats, job.metric, job.lowest, job.steps)
    sweep.write_sweep_csv(out, rows, job.formats)
    return None


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(description="Sweep mixed-tile-threshold over a range of metric thresholds.")
    ap.add_argument("repo_or_url")
    ap.add_argument("tensor_name")
    ap.add_argument("--regex", action="store_true", default=True)
    ap.add_argument("--no-regex", dest="regex", action="store_false")
    ap.add_argument("--list-matches", action="store_true")
    ap.add_argument("--revision", default="main")
    ap.add_argument("--cache-dir", default="data/hf-cache")
    ap.add_argument("--backend", choices=["emulation", "ttnn"], default="emulation")
    ap.add_argument("--formats", default="bf16,bfp8,bfp4,bfp2")
    ap.add_argument("--metric", choices=["pcc", "mae", "atol"], default="pcc")
    ap.add_argument("--lowest-metric-val", type=float, default=0.9)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out-dir", default=None)
    ap.add_argument("--checkpoint-dir", default=None,
                    help="Directory of *.safetensors shards to read the tensors from (the float32 cache is then not used).")
    ap.add_argument("--gpus", type=int, default=None,
                    help="Split the matched tensors over N GPUs of this node (one worker process per GPU, tensors balanced by "
                         "element count); the files equal a one-GPU run's.  When --lowest-metric-val is out of range for a tensor, "
                         "the error of the first such tensor in name order is printed and the exit code is 1, as without the "
                         "flag, but other GPUs may already have written tensors that come after it in name order.")
    return ap


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    if args.gpus is not None:
        err = multi_gpu.gpu_count_error(args.gpus)
        if err is not None:
            print(f"error: {err}", file=sys.stderr)
            return 1
    formats = _parse_formats(args.formats)
    if args.backend == "ttnn":
        raise RuntimeError("TTNN backend requires `ttnn` in the active Python environment.")
    index = tensor_source.build_tensor_index(args.repo_or_url, args.revision, args.cache_dir, checkpoint_dir=args.checkpoint_dir)
    selected = select_tensors(index, args.tensor_name, args.regex)
    if not selected:
        print("error: no tensors matched the filter query")
        return 1
    if args.list_matches:
        print(f"Matched {len(selected)} tensor(s):")
        for n in selected:
            print(f"  {n}")
        return 0
    base = Path(args.out_dir) if args.out_dir else (Path("results") / index.repo_id.replace("/", "__") / "mixed_tile_threshold_sweep"
                                                    / time.strftime("%Y%m%d-%H%M%S"))
    detail = base / "details"
    detail.mkdir(parents=True, exist_ok=True)
    job = SweepJob(index, detail, args.repo_or_url, args.revision, args.backend, formats, args.metric, args.lowest_metric_val,
                   args.steps)
    if args.gpus is None:
        results = ((name, sweep_one(job, name)) for name in selected)
    else:
        sizes = [math.prod(index.shape(name)) for name in selected]
        results = multi_gpu.run_sharded(sweep_one, job, selected, sizes, args.gpus)
    with contextlib.closing(results):
        try:
            for _name, error in results:
                if error is not None:
                    print(f"error: {error}")
                    return 1
        except multi_gpu.ShardError as exc:
            print(f"error: {exc}", file=sys.stderr)
            return 1
    print(f"Wrote sweep results to {base}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
