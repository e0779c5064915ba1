"""`wq` for the B200 build: the reference CLI (wq:37-79, 549-884) - same arguments, same per-tensor loop, same tables,
same ``results/<model>/<algorithm>/<timestamp>/`` tree - with the hot region (wq:679-709: ``algo.run`` + whole-tensor
scoring) on the device path.  Scores are the reference's float32 numbers (qa_tensor_scores_f32), so ``table.txt`` matches
the reference's column for column except TIME(s).

Tensors come from ``tensor_source``: the ``*.safetensors`` shards of ``--checkpoint-dir`` when it is given (read as stored;
block-scaled fp8 weights are scored from their bytes), else the reference's on-disk float32 tensor cache when it is
populated for the repo, or the synthetic DeepSeek-R1 shapes for the pseudo-repo ``synthetic`` (no Hugging Face access in
this build).

With ``--gpus N`` the matched tensors are split over N GPUs of the node (``multi_gpu``: one worker process per GPU, tensors
bin-packed by element count); the output is the same as one GPU's except TIME(s).

    python -m quantization_analysis_b200.wq <repo_or_url> [filter ...] --compression-config cfg.json [--checkpoint-dir DIR]
           [--limit N] [--recompute] [--summary] [--gpus N]
"""
from __future__ import annotations

import argparse
import contextlib
import csv
import json
import math
import re
import secrets
import sys
import time
from dataclasses import dataclass
from datetime import datetime
from pathlib import Path

import numpy as np
import torch

from . import engine, multi_gpu, tensor_source
from .compression_algorithms import create_algorithm, load_compression_config
from .compression_algorithms.cache import CacheContext
from .compression_algorithms.tile_utils import MIXED_TILE_FORMATS
from .quantization_formats import SUPPORTED_FORMATS
from .tensor_source import filter_tensor_names, resolve_format_list          # noqa: F401  (re-exported)

FORMAT_BYTES_PER_ELEM = {"mxfp4": 0.5, "nvfp4": 0.5, "bf16": 2.0, "bfp8": 1.088, "bfp4": 0.50097, "bfp2": 0.25097,
                         "fp0": 0.0}                                           # wq:132-140
MIXED_ALGOS = ("mixed-tile-greedy", "mixed-tile-random", "mixed-tile-threshold")


def _slug(s: str) -> str:
    return re.sub(r"[^a-zA-Z0-9._-]+", "_", s).strip("_") or "tensor"


def resolve_seed(config, algo_params: dict):
    """Seed precedence of wq:553-586."""
    used, source = None, None
    if config.seed is not None:
        used, source = (secrets.randbits(31), "random") if int(config.seed) == 0 else (int(config.seed), "config")
    elif config.random_seed:
        used, source = secrets.randbits(31), "random"
    if used is not None:
        algo_params["seed"] = used
    elif "seed" in algo_params:
        try:
            v = int(algo_params["seed"])
        except (TypeError, ValueError):
            return algo_params["seed"], "params"
        used, source = (secrets.randbits(31), "random") if v == 0 else (v, "params")
        algo_params["seed"] = used
    return used, source


def _mapping(assignment: np.ndarray, transposed: bool = False) -> dict:
    """The mapping JSON; a map over the tiles of x.T (the device layout) says so with "layout": "transposed"."""
    m = {"tile_hw": 32, "format_to_int": {f: i for i, f in enumerate(MIXED_TILE_FORMATS)},
         "int_to_format": MIXED_TILE_FORMATS, "assignment_shape": list(assignment.shape)}
    if transposed:
        m["layout"] = "transposed"
    return m


def write_assignment(out_dir: Path, algo_dir: str, tensor_name: str, assignment: np.ndarray, transposed: bool = False) -> None:
    """assignment.npy + assignment_mapping.json (wq:295-316)."""
    d = out_dir / algo_dir / _slug(tensor_name)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "assignment.npy", assignment.astype(np.int8))
    (d / "assignment_mapping.json").write_text(json.dumps(_mapping(assignment, transposed), indent=2))


def write_random_outputs(out_dir: Path, tensor_name: str, samples, tile_formats, assignment, transposed: bool = False) -> None:
    """<slug>.csv + <slug>_assignment.npy + mapping (wq:151-194)."""
    if not samples:
        return
    d = out_dir / "mixed_tile_random"
    d.mkdir(parents=True, exist_ok=True)
    slug = _slug(tensor_name)
    with (d / f"{slug}.csv").open("w", newline="", encoding="utf-8") as f:
        wr = csv.writer(f)
        wr.writerow(["sample_id", *[f"{fmt}_tiles" for fmt in tile_formats], "total_gb", "pcc", "mae", "atol"])
        for s in samples:
            wr.writerow([s["id"], *[s["counts"].get(fmt, 0) for fmt in tile_formats], float(s["total_bytes"]) / 1e9,
                         s["pcc"], s["mae"], s["atol"]])
    if assignment is not None:
        np.save(d / f"{slug}_assignment.npy", assignment.astype(np.int8))
        (d / f"{slug}_assignment_mapping.json").write_text(json.dumps(_mapping(assignment, transposed), indent=2))


@dataclass
class Row:
    """wq:487-497."""
    fmt: str
    compression: str
    pcc: float
    mae: float
    atol: float
    time_s: float
    gb: float
    tile_counts: dict | None = None
    tile_bytes: float | None = None


def tensor_meta_str(x_dev: torch.Tensor, shape) -> str:
    """``shape=... min=... mean=... max=...`` (wq:82-84); the mean is NumPy's float32 pairwise mean (scorer output 3)."""
    flat = x_dev.reshape(-1)
    mean = float(engine.tensor_scores_f32(flat, flat)[0, 3])
    return f"shape={tuple(shape)} min={float(flat.min().float()):.3e} mean={mean:.3e} max={float(flat.max().float()):.3e}"


def evaluate_tensor(name: str, x, algorithms, formats, out_dir: Path | None, cache_ctx: CacheContext | None,
                    save_processed: bool = True):
    """The hot region of wq:679-742 for one tensor -> ({compression: [Row]}, meta line).  x: what TensorIndex.load returns (a
    float32 host array, a host torch tensor as stored, tensor_source.Fp8Blocks) or an engine.Prepared."""
    rows: dict[str, list[Row]] = {}
    p = engine.prepare_loaded(x)                                  # one H2D; bf16 on the device when the values allow it
    shape = p.shape
    meta = tensor_meta_str(p.data if p.kind != "vector" else p.data[: p.numel], shape)
    x_flat = p.data
    table = None
    for algo in algorithms:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if algo.name in ("none", "transpose"):
            from .compression_algorithms.none import quantize_all
            from .compression_algorithms.transpose import quantize_all_transposed
            xd = (p.data[: p.numel] if p.kind == "vector" else p.data).reshape(shape)
            have = {}
            if cache_ctx is not None:
                for f in formats:
                    y = cache_ctx.load_array(algo.name, f)
                    if y is not None and tuple(y.shape) == tuple(shape):
                        have[f] = torch.from_numpy(np.ascontiguousarray(y, dtype=np.float32)).to(xd.device)
            missing = [f for f in formats if f not in have]
            fresh = (quantize_all if algo.name == "none" else quantize_all_transposed)(xd, missing) if missing else {}
            if cache_ctx is not None and save_processed:
                for f in missing:
                    cache_ctx.save_array(algo.name, f, fresh[f].float().cpu().numpy().reshape(shape))
            torch.cuda.synchronize()
            elapsed = time.perf_counter() - t0
            for f in formats:
                y = have.get(f, fresh.get(f))
                s = engine.tensor_scores_f32(x_flat, None if f == "fp0" else y.reshape(-1), n=p.numel)[0]
                rows.setdefault(algo.name, []).append(Row(f.upper(), algo.name, float(s[0]), float(s[1]), float(s[2]), elapsed,
                                                          float(p.numel) * float(FORMAT_BYTES_PER_ELEM.get(f, 0.0)) / 1e9
                                                          if f in FORMAT_BYTES_PER_ELEM else 0.0))
            continue
        tile_formats = getattr(algo, "tile_formats", None) or getattr(algo, "formats", None) or algo._filter_from_formats(formats)
        # "transpose": true - the mixed algorithm runs over x.T (the device layout) with its own copy and table
        pm = engine.prepare_transposed(p) if getattr(algo, "transpose", False) else p
        if table is None and getattr(algo, "strict", False) is False and algo.name != "mixed-tile-threshold":
            table = engine.tile_stats(pm, engine.MIXED_FORMATS)
        dr = algo.run_prepared(pm, tile_formats, table=table)
        dr.y_device()                                            # the reference's run() returns y: part of TIME(s)
        torch.cuda.synchronize()
        elapsed = time.perf_counter() - t0
        m = dr.metrics
        rows.setdefault(algo.name, []).append(Row("MIXED", algo.name, m["pcc"], m["mae"], m["atol"], elapsed, float(dr.tile_bytes) / 1e9,
                                                  dr.counts, dr.tile_bytes))
        if out_dir is not None:
            a = dr.assignment_numpy()
            if algo.name == "mixed-tile-random":
                write_random_outputs(out_dir, name, dr.meta["samples"], dr.tile_formats, a, dr.transposed)
            else:
                write_assignment(out_dir, algo.name.replace("-", "_"), name, a, dr.transposed)
    return rows, meta


def format_block(rows: list[Row], comp: str, comp_w: int) -> list[str]:
    """The table of one (tensor, algorithm) in the reference's layout (wq:753-848)."""
    fmt_w = max(len(r.fmt) for r in rows)
    mixed = comp in MIXED_ALGOS
    w = {"time": len("TIME(s)"), "gb": len("GB"), "pcc": len("PCC"), "mae": len("MAE"), "atol": len("ATOL"), "bytes": len("BYTES")}
    cw = {k: len(k.upper()) for k in MIXED_TILE_FORMATS}
    for r in rows:
        w["time"] = max(w["time"], len(f"{r.time_s:.3f}"))
        w["gb"] = max(w["gb"], len(f"{r.gb:.3f}"))
        w["pcc"] = max(w["pcc"], len(f"{r.pcc: .5f}"))
        w["mae"] = max(w["mae"], len(f"{r.mae:.3e}"))
        w["atol"] = max(w["atol"], len(f"{r.atol:.3e}"))
        if mixed:
            for k in MIXED_TILE_FORMATS:
                cw[k] = max(cw[k], len(str((r.tile_counts or {}).get(k, 0))))
            if r.tile_bytes is not None:
                w["bytes"] = max(w["bytes"], len(f"{r.tile_bytes:,.0f}"))
    head = (f"  {'COMP'.ljust(comp_w)}  {'FORMAT'.ljust(fmt_w)}  {'PCC'.rjust(w['pcc'])}  {'MAE'.rjust(w['mae'])}  "
            f"{'ATOL'.rjust(w['atol'])}  {'TIME(s)'.rjust(w['time'])}  {'GB'.rjust(w['gb'])}")
    if mixed:
        head += "  " + "  ".join(k.upper().rjust(cw[k]) for k in MIXED_TILE_FORMATS) + "  " + "BYTES".rjust(w["bytes"])
    lines = [head]
    for r in rows:
        line = (f"  {r.compression.ljust(comp_w)}  {r.fmt.ljust(fmt_w)}  {f'{r.pcc: .5f}'.rjust(w['pcc'])}  "
                f"{f'{r.mae:.3e}'.rjust(w['mae'])}  {f'{r.atol:.3e}'.rjust(w['atol'])}  {f'{r.time_s:.3f}'.rjust(w['time'])}  "
                f"{f'{r.gb:.3f}'.rjust(w['gb'])}")
        if mixed:
            counts = r.tile_counts or {}
            line += ("  " + "  ".join(str(counts.get(k, 0)).rjust(cw[k]) for k in MIXED_TILE_FORMATS) + "  "
                     + f"{(r.tile_bytes or 0.0):,.0f}".rjust(w["bytes"]))
        lines.append(line)
    return lines


@dataclass
class TensorJob:
    """Everything wq's per-tensor step needs besides the tensor's name; built once by `run` (after the seed is resolved) and,
    under --gpus, pickled to every worker."""
    index: tensor_source.TensorIndex
    algorithms: list
    comp_names: list[str]
    comp_w: int
    formats: list[str]
    results_dir: Path
    processed_root: Path
    backend: str
    recompute: bool
    run_tag: str
    save_processed: bool


def run_tensor(job: TensorJob, name: str) -> tuple[str, list[str], list[Row]]:
    """wq's per-tensor step, the same with and without --gpus: load and evaluate one tensor, write its maps and processed arrays.
    -> (the screen line naming where it was read from, its block of screen / table.txt lines, its rows in block order)."""
    describe = job.index.describe(name)
    x = job.index.load(name)
    ctx = CacheContext(root=job.processed_root, tensor_name=name, backend=job.backend, recompute=job.recompute, run_tag=job.run_tag)
    rows_by_comp, meta = evaluate_tensor(name, x, job.algorithms, job.formats, job.results_dir, ctx, save_processed=job.save_processed)
    block, rows = [name, f"  {meta}"], []
    for comp in job.comp_names:
        comp_rows = rows_by_comp.get(comp, [])
        if not comp_rows:
            continue
        rows += comp_rows
        block += format_block(comp_rows, comp, job.comp_w) + [""]
    return describe, block, rows


def _hierarchy_lines(names) -> list[str]:
    """Tree of the dotted tensor names with leaf counts (wq:460-546; screen only, not part of table.txt)."""
    root: dict = {}
    for n in sorted(names):
        node = root
        for part in n.split("."):
            node = node.setdefault(part, {})

    def leaves(node):
        return 1 if not node else sum(leaves(c) for c in node.values())

    def render(node, prefix=""):
        out = []
        items = sorted(node.items())
        for i, (k, child) in enumerate(items):
            last = i == len(items) - 1
            c = leaves(child)
            out.append(f"{prefix}{'└── ' if last else '├── '}{k}{f' ({c})' if c > 1 else ''}")
            if child:
                out += render(child, prefix + ("    " if last else "│   "))
        return out
    return render(root)


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="wq", description="Weight quantization analyzer (B200 device path).")
    ap.add_argument("repo_or_url", help="Model repo/URL (names the results tree; its float32 tensor cache is the source "
                                        "without --checkpoint-dir), or 'synthetic'.")
    ap.add_argument("filter_query", nargs="*", help="Optional filter: substring, or dotted torch-style prefix path.")
    ap.add_argument("--revision", default="main", help="Revision (default: main).")
    ap.add_argument("--cache-dir", default="data/hf-cache", help="Shared local cache for float32 tensors (default: data/hf-cache).")
    ap.add_argument("--limit", type=int, default=None, help="Optional max matched tensors.")
    ap.add_argument("--backend", choices=["emulation", "ttnn"], default="emulation")
    ap.add_argument("--compression-config", type=str, default=None, help="Path to a JSON compression config file (default: none).")
    ap.add_argument("--recompute", action="store_true", help="Recompute and overwrite cached quantized tensors.")
    ap.add_argument("--summary", action="store_true", help="Print the aggregate summary (default: off).")
    # extensions of this build
    ap.add_argument("--results-root", default="results", help="Root of the results tree (default: results, like the reference).")
    ap.add_argument("--processed-root", default="data/processed", help="Root of the quantized-array cache (default: data/processed).")
    ap.add_argument("--no-save-processed", action="store_true", help="Do not write quantized arrays of none/transpose to disk.")
    ap.add_argument("--synthetic-seed", type=int, default=1000, help="Base seed of the synthetic tensors.")
    ap.add_argument("--checkpoint-dir", default=None,
                    help="Directory of *.safetensors shards (a local export or a hub snapshot) to read the tensors from; "
                         "the float32 cache is then neither read nor written.")
    ap.add_argument("--gpus", type=int, default=None,
                    help="Split the matched tensors over N GPUs of this node (one worker process per GPU, tensors balanced by "
                         "element count); output equals a one-GPU run's except TIME(s).  Default: this process, on the current GPU.")
    return ap


def run(argv=None) -> int:
    args = build_parser().parse_args(argv)
    if args.gpus is not None:
        err = multi_gpu.gpu_count_error(args.gpus)
        if err is not None:
            print(f"error: {err}", file=sys.stderr)
            return 1
    run_tag = datetime.now().strftime("%Y%m%d-%H%M%S")
    config = load_compression_config(args.compression_config)
    algo_params = dict(config.params)
    used_seed, seed_source = resolve_seed(config, algo_params)
    selected = create_algorithm(config.algorithm, algo_params)
    baseline = create_algorithm("none", {})
    algorithms = [baseline] if selected.name == "none" else [baseline, selected]
    filter_query = " ".join(args.filter_query).strip() or None
    formats = resolve_format_list(config.quantization_formats, SUPPORTED_FORMATS)
    index = tensor_source.build_tensor_index(args.repo_or_url, args.revision, args.cache_dir, args.synthetic_seed,
                                             checkpoint_dir=args.checkpoint_dir)
    names = tensor_source.resolve_selected_tensors(index, filter_query)
    if args.limit is not None:
        names = names[: max(0, args.limit)]
    if not names:
        print("No tensors matched.", file=sys.stderr)
        return 1
    if args.backend == "ttnn":
        print("error: TTNN backend requires `ttnn` in the active Python environment.", file=sys.stderr)
        return 1
    comp_names = [a.name for a in algorithms]
    comp_w = max(len("COMP"), max(len(n) for n in comp_names))
    print(f"{index.repo_id} @{index.revision} - {len(names)} tensors")
    print(f"formats: {', '.join(formats)}")
    print(f"compression: {', '.join(comp_names)}")
    print(f"backend: {args.backend}")
    if args.compression_config:
        print(f"config: {args.compression_config}")
    print()
    print("Hierarchy")
    for line in _hierarchy_lines(names):
        print(f"  {line}")
    print()
    results_dir = Path(args.results_root) / index.repo_id.replace("/", "__") / selected.name / run_tag
    results_dir.mkdir(parents=True, exist_ok=True)
    used_params = dict(algo_params)
    if used_seed is not None:
        used_params.pop("seed", None)
    used = {"algorithm": config.algorithm, "quantization_formats": formats, "params": used_params}
    if used_seed is not None:
        used["seed"] = used_seed
        if seed_source:
            used["seed_source"] = seed_source
    (results_dir / "compression_config.used.json").write_text(json.dumps(used, indent=2), encoding="utf-8")
    processed_root = Path(args.processed_root) / tensor_source.safe_repo_revision_key(index.repo_id, index.revision)
    job = TensorJob(index, algorithms, comp_names, comp_w, formats, results_dir, processed_root, args.backend, args.recompute,
                    run_tag, not args.no_save_processed)
    if args.gpus is None:
        results = ((name, run_tensor(job, name)) for name in names)
    else:
        sizes = [math.prod(index.shape(name)) for name in names]
        results = multi_gpu.run_sharded(run_tensor, job, names, sizes, args.gpus)
    aggregate: dict[tuple[str, str], list[Row]] = {}
    table_lines: list[str] = []
    with contextlib.closing(results):
        try:
            for _name, (describe, block, rows) in results:
                print(describe)
                print("\n".join(block))
                for r in rows:
                    aggregate.setdefault((r.compression, r.fmt), []).append(r)
                table_lines += block
        except multi_gpu.ShardError as exc:
            print(f"error: {exc}", file=sys.stderr)
            return 1
    if args.summary:
        print("Summary (mean across matched tensors)")
        table_lines.append("Summary (mean across matched tensors)")
        for comp in comp_names:
            for fmt in (["MIXED"] if comp in MIXED_ALGOS else [f.upper() for f in formats]):
                rows = aggregate.get((comp, fmt), [])
                if not rows:
                    continue
                pcc = float(np.mean([r.pcc for r in rows]))
                mae = float(np.mean([r.mae for r in rows]))
                atol = float(np.mean([r.atol for r in rows]))
                bv = [r.tile_bytes for r in rows if r.tile_bytes is not None]
                line = f"  {comp.ljust(comp_w)} {fmt:>5}  pcc={pcc: .5f}  mae={mae:.3e}  atol={atol:.3e}" + (
                    f"  bytes={float(np.mean(bv)):,.0f}" if bv else "")
                print(line)
                table_lines.append(line)
    (results_dir / "table.txt").write_text("\n".join(table_lines) + "\n", encoding="utf-8")
    return 0


if __name__ == "__main__":
    sys.exit(run())
