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
import secrets
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


def base_format_score(p: engine.Prepared, fmt: str, metric: str) -> float:
    """Whole-tensor float32 score of one format, as wq's `none` row prints it (the quantizers' geometry)."""
    from .compression_algorithms.none import quantize_all
    xd = (p.data[: p.numel] if p.kind == "vector" else p.data).reshape(p.shape)
    y = quantize_all(xd, [fmt])[fmt]
    return float(engine.tensor_scores_f32(p.data, y.reshape(-1), n=p.numel)[0, _ROW[metric]])


def greedy_thresholds(highest: float, metric: str, steps: int, lowest: float) -> np.ndarray:
    """float64 ``np.linspace(highest, lowest, max(1, steps))``; a `lowest` on the wrong side of `highest` is an error."""
    if metric == "pcc" and lowest > highest:
        raise SweepRangeError("lowest-metric-val must be <= highest metric for pcc")
    if metric != "pcc" and lowest < highest:
        raise SweepRangeError("lowest-metric-val must be >= highest metric for mae/atol")
    return np.linspace(highest, lowest, max(1, steps))


def greedy_sweep_tensor(x, tile_formats=MIXED_TILE_FORMATS, metric: str = "pcc", steps: int = 32, lowest: float = 0.9,
                        highest: float | None = None, seed: int = 0, thresholds=None, scoring: str = "reference",
                        certify: bool = True, margin_bound: float = 2e-13):
    """mixed-tile-greedy over a range of thresholds: one tile-stat table, one init, one set of permutations and one launch
    for all the chains (engine.greedy_sweep).  Row k equals MixedTileGreedyCompression({"threshold": thresholds[k],
    "seed": seed, ...}).run_prepared on the same tensor: map, counts, state, certificate and metrics.

    x: as sweep_tensor.  tile_formats: the greedy's order, the first is the base format.  Thresholds: float64
    ``np.linspace(highest, lowest, steps)`` unless given; `highest` defaults to the base format's whole-tensor float32 score
    (wq's `none` row).  seed 0 draws one at random (as the greedy does); every row records the seed used.  Certificate: a
    pcc / mae chain whose decision margin (state[20]) is below `margin_bound` is redone alone from NumPy-order tile sums with
    the one-thread chain (the strict table is built once); its row has fallback=True.
    -> (rows, maps): rows = dicts {threshold, counts, total_bytes, pcc, mae, atol, min_margin, fallback, seed, state (the
    chain's float64 [24], as run_prepared's meta["state"])} and the int8
    maps [steps, ntiles] in MIXED_TILE_FORMATS numbering.  scoring as in sweep_tensor; "exact" recombines from the table the
    row's chain used (the strict one after a fallback)."""
    from .batch import cached_permutations
    tile_formats = list(tile_formats)
    if not tile_formats or any(f not in engine.FMT_INDEX for f in tile_formats):
        raise ValueError(f"tile_formats must be a non-empty list of {', '.join(MIXED_TILE_FORMATS)}")
    if metric not in _ROW:
        raise ValueError(f"Unsupported metric: {metric}")
    if seed == 0:
        seed = secrets.randbits(31)           # mixed_tile_greedy.py:222-224
    p = engine.prepare_loaded(x)
    if thresholds is None:
        if highest is None:
            highest = base_format_score(p, tile_formats[0], metric)
        thresholds = greedy_thresholds(float(highest), metric, steps, lowest)
    thresholds = np.asarray(thresholds, dtype=np.float64).reshape(-1)
    table = engine.tile_stats(p, MIXED_TILE_FORMATS, exact_abs=(metric == "mae"))      # as run_prepared builds it
    dev = table.device
    nt, nf = table.shape[1], len(tile_formats)
    rng = engine.make_rng(seed, dev)
    fast = metric != "atol"                   # pcc / mae: the cluster chain; atol: the one-thread chain (no certificate)
    init = prefetched = None
    if fast:
        init = engine.greedy_init(table, metric, tile_formats)
        if nf >= 2:
            hit = cached_permutations(dev, seed, nt, nf)
            k = 2 if nf >= 3 else 1
            prefetched = (hit["pre_order"][:k], hit["rngs"][1:1 + k])
    maps, counts, states = engine.greedy_sweep(table, p.numel, metric, thresholds, tile_formats, rng, prefetched, init)
    st = states.cpu().numpy()
    margins = [float(st[i, 20]) if fast else None for i in range(len(thresholds))]
    redo = [i for i in range(len(thresholds)) if fast and certify and not (margins[i] >= margin_bound)]
    strict = engine.tile_stats(p, MIXED_TILE_FORMATS, strict=True) if redo else None
    for i in redo:
        a, c, s_ = engine.greedy_assign(strict, p.numel, metric, float(thresholds[i]), tile_formats, engine.make_rng(seed, dev),
                                        parallel=False)
        maps[i], counts[i], states[i] = a, c, s_
    fallback = [i in redo for i in range(len(thresholds))]
    counts, st = counts.cpu().numpy(), states.cpu().numpy()
    # a row is scored again only when its map (or, for exact scores, the table behind it) differs from the previous row's
    same_as_prev = [False] + [fallback[i] == fallback[i - 1] and bool(torch.equal(maps[i], maps[i - 1]))
                              for i in range(1, maps.shape[0])]
    distinct = [i for i, s_ in enumerate(same_as_prev) if not s_]
    if scoring == "exact":
        sums = engine.assignment_sums_batch(table, maps).cpu().numpy()
        if redo:
            sums[redo] = engine.assignment_sums_batch(strict, maps[redo]).cpu().numpy()
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
            s_ = sc[i]
            last = {"counts": c, "total_bytes": mixed_tile_total_bytes(c), "pcc": float(s_[0]), "mae": float(s_[1]), "atol": float(s_[2])}
        rows.append({"threshold": float(thr), **last, "min_margin": margins[i], "fallback": fallback[i], "seed": seed, "state": st[i]})
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


def write_sweep_config(out_dir, repo_or_url, tensor_name, revision, backend, formats, metric, lowest, steps, greedy=None):
    """``sweep_config.json`` (sweep:675-686).  greedy: {"algorithm", "seed", "highest_metric_val"} of a greedy sweep, appended."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    payload = {"repo_or_url": repo_or_url, "tensor_name": tensor_name, "revision": revision, "backend": backend,
               "formats": list(formats), "metric": metric, "lowest_metric_val": lowest, "steps": steps, **(greedy or {})}
    (out / "sweep_config.json").write_text(json.dumps(payload, indent=2), encoding="utf-8")
