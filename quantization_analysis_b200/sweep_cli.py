"""Threshold-sweep CLI (scripts/sweep_mixed_tile_threshold.py:36-102, 581-841 of the reference): same arguments, same
``details/<tensor>/sweep_config.json`` + ``sweep_results.csv``; the plots (matplotlib) are out of scope.

    python -m quantization_analysis_b200.sweep_cli <repo_or_url> <tensor_name> [--no-regex] [--metric pcc|mae|atol]
           [--lowest-metric-val V] [--steps N] [--formats bf16,bfp8,bfp4,bfp2] [--out-dir DIR] [--checkpoint-dir DIR] [--gpus N]
           [--algorithm mixed-tile-threshold|mixed-tile-greedy] [--seed S] [--highest-metric-val V]

``--algorithm mixed-tile-greedy`` sweeps the greedy instead (sweep.greedy_sweep_tensor: one table and one launch for all
thresholds per tensor), from ``--highest-metric-val`` (default: the first format's whole-tensor score) down to
``--lowest-metric-val``; the first of ``--formats`` is its base format.  ``--seed`` is the greedy's (0, the default, draws
one), drawn once for the run and recorded in every ``sweep_config.json``.  Files go under ``mixed_tile_greedy_sweep/``.

Tensors come from ``tensor_source`` like wq's: the shards of ``--checkpoint-dir`` when given, else the float32 cache.  With
``--gpus N`` the matched tensors are split over N GPUs of the node like wq's (``multi_gpu``); the files are the same.
"""
from __future__ import annotations

import argparse
import contextlib
import fnmatch
import math
import re
import secrets
import sys
import time
from dataclasses import dataclass
from pathlib import Path

from . import multi_gpu, sweep, tensor_source
from .compression_algorithms.tile_utils import MIXED_TILE_FORMATS

ALGORITHMS = ("mixed-tile-threshold", "mixed-tile-greedy")


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
    algorithm: str = "mixed-tile-threshold"
    seed: int = 0                         # greedy: the resolved seed (never 0 here)
    highest: float | None = None          # greedy: --highest-metric-val


def sweep_one(job: SweepJob, name: str) -> str | None:
    """Sweep one tensor and write its ``details/<tensor>/`` files.  -> None, or the message of its SweepRangeError (nothing
    is written for that tensor)."""
    x = job.index.load(name)
    greedy = job.algorithm == "mixed-tile-greedy"
    try:
        if greedy:
            rows, _maps = sweep.greedy_sweep_tensor(x, job.formats, job.metric, job.steps, job.lowest, highest=job.highest, seed=job.seed)
        else:
            rows, _maps = sweep.sweep_tensor(x, job.formats, job.metric, job.steps, job.lowest)
    except sweep.SweepRangeError as exc:
        return str(exc)
    out = job.detail / name.replace("/", "_").replace(".", "_")
    # highest_metric_val: the first threshold swept (the base format's score unless --highest-metric-val gave it)
    extra = {"algorithm": job.algorithm, "seed": job.seed, "highest_metric_val": rows[0]["threshold"]} if greedy else None
    sweep.write_sweep_config(out, job.repo_or_url, name, job.revision, job.backend, job.formats, job.metric, job.lowest, job.steps,
                             greedy=extra)
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
    ap.add_argument("--algorithm", default="mixed-tile-threshold",
                    help=f"Algorithm to sweep: {' or '.join(ALGORITHMS)} (default mixed-tile-threshold).")
    ap.add_argument("--seed", type=int, default=None,
                    help="mixed-tile-greedy only: the greedy's seed; 0 (the default) draws one, recorded in sweep_config.json.")
    ap.add_argument("--highest-metric-val", type=float, default=None,
                    help="mixed-tile-greedy only: first (tightest) threshold; default: the first format's whole-tensor score.")
    return ap


def greedy_args_error(args) -> str | None:
    """The message for an --algorithm / --seed / --highest-metric-val combination that cannot run, else None."""
    if args.algorithm not in ALGORITHMS:
        return f"--algorithm must be one of {', '.join(ALGORITHMS)}, not {args.algorithm!r}"
    if args.algorithm != "mixed-tile-greedy":
        for flag, v in (("--seed", args.seed), ("--highest-metric-val", args.highest_metric_val)):
            if v is not None:
                return f"{flag} applies to --algorithm mixed-tile-greedy only"
        return None
    if args.seed is not None and not 0 <= args.seed < 2 ** 63:
        return "--seed must be 0 (random) or a positive integer"
    if args.highest_metric_val is not None and not math.isfinite(args.highest_metric_val):
        return "--highest-metric-val must be a finite number"
    return None


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    err = greedy_args_error(args)
    if err is not None:
        print(f"error: {err}", file=sys.stderr)
        return 1
    greedy = args.algorithm == "mixed-tile-greedy"
    seed = 0
    if greedy:      # resolved once here, so that every tensor on every GPU uses the recorded seed
        seed = args.seed if args.seed else secrets.randbits(31)
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
    kind = "mixed_tile_greedy_sweep" if greedy else "mixed_tile_threshold_sweep"
    base = Path(args.out_dir) if args.out_dir else (Path("results") / index.repo_id.replace("/", "__") / kind
                                                    / time.strftime("%Y%m%d-%H%M%S"))
    detail = base / "details"
    detail.mkdir(parents=True, exist_ok=True)
    job = SweepJob(index, detail, args.repo_or_url, args.revision, args.backend, formats, args.metric, args.lowest_metric_val,
                   args.steps, args.algorithm, seed, args.highest_metric_val)
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
