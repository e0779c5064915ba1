"""Threshold sweep on the device (core of scripts/sweep_mixed_tile_threshold.py:623-797).

Per tensor: one pass for the NumPy-faithful per-tile scores (qa_tile_scores_f32); the thresholds are
``np.linspace(start, lowest, steps)`` in float64 with start = max (pcc) or min (mae / atol) of the highest-precision format's
scores (:659-670); all thresholds are assigned in ONE launch (qa_threshold_assign: index into the ascending-bytes order, last
format forced, float32 comparison like NumPy 2, :145-155); every distinct assignment is materialised
(qa_apply_assignment) and scored with the reference's float32 whole-tensor arithmetic (qa_tensor_scores_f32, :746-749) -
consecutive equal assignments reuse the previous row like the reference (:736-742).
"""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import torch

from . import engine
from .compression_algorithms.mixed_tile_threshold import formats_by_precision
from .compression_algorithms.tile_utils import MIXED_TILE_BYTES_PER_ELEM, MIXED_TILE_FORMATS, mixed_tile_total_bytes

_ROW = {"pcc": 0, "mae": 1, "atol": 2}


class SweepRangeError(ValueError):
    """--lowest-metric-val lies on the wrong side of the start metric (the reference prints an error and returns 1)."""


def sweep_thresholds(scores_metric: torch.Tensor, tile_formats, metric: str, steps: int, lowest: float) -> np.ndarray:
    """float64 ``np.linspace(start, lowest, max(1, steps))`` (sweep:659-670): start = max of the highest-precision format's
    per-tile scores for pcc, min for mae / atol; a `lowest` on the wrong side of it is an error."""
    order = formats_by_precision(tile_formats)
    highest = max(order, key=lambda f: MIXED_TILE_BYTES_PER_ELEM.get(f, 0.0))
    row = scores_metric[engine.FMT_INDEX[highest]]
    if metric == "pcc":
        start = float(row.max().item())
        if lowest > start:
            raise SweepRangeError("lowest-metric-val must be <= start metric for pcc")
    else:
        start = float(row.min().item())
        if lowest < start:
            raise SweepRangeError("lowest-metric-val must be >= start metric for mae/atol")
    return np.linspace(start, lowest, max(1, steps))


def _score_maps(p: engine.Prepared, maps: torch.Tensor, rows_idx) -> dict[int, np.ndarray]:
    """float32 (pcc, mae, atol) of the reconstructions of the given rows of `maps`, batched."""
    L = engine._lib.lib()
    per = p.rows * p.cols
    chunk = engine.candidate_chunk(per, len(rows_idx), p.data.device)
    ys = torch.empty((chunk, per), dtype=torch.bfloat16, device=p.data.device)
    out = {}
    for s0 in range(0, len(rows_idx), chunk):
        part = rows_idx[s0:s0 + chunk]
        for j, i in enumerate(part):
            engine.check(L.qa_apply_assignment(p.data.data_ptr(), p.dtype_code, p.rows, p.cols, p.cols, maps[i].data_ptr(),
                                               ys[j].data_ptr(), engine._stream()), "qa_apply_assignment")
        sc = engine.tensor_scores_f32(p.data, ys[:len(part)], n=p.numel)
        for j, i in enumerate(part):
            out[i] = sc[j, :3]
    return out


def sweep_tensor(x, tile_formats=MIXED_TILE_FORMATS, metric: str = "pcc", steps: int = 32, lowest: float = 0.9,
                 thresholds=None, scoring: str = "reference"):
    """x: a host array or tensor, what tensor_source's loaders return (tensor_source.Fp8Blocks included), or an
    engine.Prepared.  -> (rows, maps): rows = list of dicts {threshold (float64), counts, total_bytes, pcc, mae, atol} and the int8 maps
    [steps, ntiles] in MIXED_TILE_FORMATS numbering.  scoring="reference": the reference's float32 whole-tensor values
    (every distinct map is materialised and scored); "exact": float64 recombination of the tile-stat table, all maps in one
    launch, no reconstruction (the mathematically exact value of the same formulas)."""
    tile_formats = list(tile_formats)
    p = engine.prepare_loaded(x)
    scores = engine.tile_scores(p, tile_formats)[_ROW[metric]].contiguous()
    if thresholds is None:
        thresholds = sweep_thresholds(scores, tile_formats, metric, steps, lowest)
    thresholds = np.asarray(thresholds, dtype=np.float64)
    order = formats_by_precision(tile_formats)
    maps, counts = engine.threshold_assign(scores, order, metric == "pcc", thresholds)       # compared as float32 (NumPy 2)
    counts = counts.cpu().numpy()
    # the reference recomputes a row only when the assignment differs from the previous step's (sweep:736-742)
    same_as_prev = [False] + [bool(torch.equal(maps[i], maps[i - 1])) for i in range(1, maps.shape[0])]
    distinct = [i for i, s in enumerate(same_as_prev) if not s]
    if scoring == "exact":
        table = engine.tile_stats(p, MIXED_TILE_FORMATS)
        sums = engine.assignment_sums_batch(table, maps).cpu().numpy()
        sc = {}
        for i in distinct:
            m = engine.metrics_from_sums(sums[i], p.numel)
            sc[i] = (m["pcc"], m["mae"], m["atol"])
    else:
        sc = _score_maps(p, maps, distinct)
    rows, last = [], None
    for i, thr in enumerate(thresholds):
        if not same_as_prev[i]:
            c = {f: int(counts[i, j]) for j, f in enumerate(MIXED_TILE_FORMATS)}
            s = sc[i]
            last = {"counts": c, "total_bytes": mixed_tile_total_bytes(c), "pcc": float(s[0]), "mae": float(s[1]), "atol": float(s[2])}
        rows.append({"threshold": float(thr), **last})
    return rows, maps


def baseline_points(x, tile_formats, metric: str, lowest: float) -> list[dict]:
    """Whole-tensor baseline of every candidate format (sweep:688-717), kept if it lies inside the swept range."""
    p = engine.prepare_loaded(x)
    recon = engine.quant_recon(p, list(tile_formats))
    sc = engine.tensor_scores_f32(p.data, torch.stack([recon[f] for f in tile_formats]), n=p.numel)
    pts = []
    for i, f in enumerate(tile_formats):
        pcc, mae, atol = float(sc[i, 0]), float(sc[i, 1]), float(sc[i, 2])
        value = {"pcc": pcc, "mae": mae, "atol": atol}[metric]
        if (metric == "pcc" and value < lowest) or (metric != "pcc" and value > lowest):
            continue
        pts.append({"label": f.upper(), "size": float(p.numel) * float(MIXED_TILE_BYTES_PER_ELEM.get(f, 0.0)), "metric": value,
                    "kind": "baseline", "pcc": pcc, "mae": mae, "atol": atol, f"{f}_tiles": int(p.ntiles)})
    return pts


def write_sweep_csv(out_dir, rows, formats=MIXED_TILE_FORMATS):
    """``sweep_results.csv`` in the reference's layout (scripts/sweep_mixed_tile_threshold.py:792-797):
    step,threshold,size_bytes,pcc,mae,atol,<fmt>_tiles... with ``str()`` of Python floats."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    headers = ["step", "threshold", "size_bytes", "pcc", "mae", "atol", *[f"{fmt}_tiles" for fmt in formats]]
    with (out / "sweep_results.csv").open("w", encoding="utf-8") as f:
        f.write(",".join(headers) + "\n")
        for i, r in enumerate(rows):
            vals = {"step": i, "threshold": float(r["threshold"]), "size_bytes": r["total_bytes"], "pcc": r["pcc"], "mae": r["mae"],
                    "atol": r["atol"], **{f"{fmt}_tiles": r["counts"].get(fmt, 0) for fmt in formats}}
            f.write(",".join(str(vals.get(h, "")) for h in headers) + "\n")
    return out / "sweep_results.csv"


def write_sweep_config(out_dir, repo_or_url, tensor_name, revision, backend, formats, metric, lowest, steps):
    """``sweep_config.json`` (sweep:675-686)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    payload = {"repo_or_url": repo_or_url, "tensor_name": tensor_name, "revision": revision, "backend": backend,
               "formats": list(formats), "metric": metric, "lowest_metric_val": lowest, "steps": steps}
    (out / "sweep_config.json").write_text(json.dumps(payload, indent=2), encoding="utf-8")
