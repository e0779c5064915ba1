"""mixed-tile-random on the device (reference: compression_algorithms/mixed_tile_random.py:18-209).

All `iters` uniform assignments are drawn from the NumPy PCG64 stream on the device and scored
from the tile-stat table in one launch (qa_random_samples); selection over the per-sample
scalars follows the reference's rules (smallest bytes among passing samples, first wins ties;
otherwise strictly best metric).  The per-sample pcc / mae / atol are the reference's float32 whole-tensor values
(mixed_tile_random.py:137-141): every sample's reconstruction is materialised by qa_apply_assignment and scored by
qa_tensor_scores_f32 in batches, so the selection - ties and near-ties included - is the reference's.
``params["sample_scoring"] = "exact"`` (extension) keeps the float64 table recombinations instead (no reconstruction).
"""
from __future__ import annotations

import numpy as np

from .. import engine
from .base import CompressionAlgorithm, CompressionResult
from . import _mixed_common as mc
from .metrics import metric_better, metric_is_good
from .tile_utils import MIXED_TILE_BYTES_PER_ELEM, MIXED_TILE_FORMATS


class MixedTileRandomCompression(CompressionAlgorithm):
    name = "mixed-tile-random"

    def __init__(self, params: dict | None = None) -> None:
        super().__init__(params=params)
        self.metric = self.params.get("metric", "pcc")
        self.threshold = float(self.params.get("threshold", 0.999))
        self.iters = int(self.params.get("iters", 50))
        self.seed = int(self.params.get("seed", 0))
        self.formats = mc.parse_formats(self.params.get("formats"))
        self.sample_scoring = str(self.params.get("sample_scoring", "reference"))
        self.transpose = mc.parse_transpose(self.params)          # extension: the device layout (tiles of x.T)
        if self.metric not in mc.VALID_METRICS:
            raise ValueError(f"Unsupported metric: {self.metric}")
        if self.iters < 1:
            raise ValueError("iters must be >= 1")

    @classmethod
    def from_params(cls, params: dict | None = None) -> "MixedTileRandomCompression":
        return cls(params=params or {})

    def expected_evals(self, formats) -> int:
        return 1

    _parse_formats = staticmethod(mc.parse_formats)

    @staticmethod
    def _filter_from_formats(formats):
        return mc.filter_formats(formats, "mixed-tile-random")

    def run_prepared(self, p: engine.Prepared, tile_formats, table=None) -> mc.DeviceResult:
        if table is None:
            table = engine.tile_stats(p, MIXED_TILE_FORMATS)
        fmt_list = list(tile_formats) or list(MIXED_TILE_FORMATS)
        rng = engine.make_rng(self.seed, p.data.device)     # seed 0 is NOT randomised here (:116)
        iters = max(1, self.iters)
        choices, metrics_dev, counts_dev = engine.random_samples(table, p.numel, fmt_list, iters, rng)
        met = metrics_dev.cpu().numpy()
        if self.sample_scoring != "exact":
            met = self._reference_scores(p, choices)
        cnt = counts_dev.cpu().numpy().astype(np.int64)
        bpe32 = np.asarray([MIXED_TILE_BYTES_PER_ELEM[f] for f in MIXED_TILE_FORMATS], dtype=np.float32)
        col = {"pcc": 0, "mae": 1, "atol": 2}[self.metric]
        samples, best_id, best_bytes, best_metric = [], None, None, None
        for sid in range(iters):
            counts = {f: int(cnt[sid, i]) for i, f in enumerate(MIXED_TILE_FORMATS)}
            samples.append({"id": sid, "counts": counts, "total_bytes": mc.total_bytes(counts),
                            "pcc": float(met[sid, 0]), "mae": float(met[sid, 1]), "atol": float(met[sid, 2])})
            score = float(met[sid, col])
            if metric_is_good(score, self.metric, self.threshold):
                tb = float(np.sum(cnt[sid] * bpe32) * (32 * 32))            # :158
                if best_bytes is None or tb < best_bytes:
                    best_bytes, best_metric, best_id = tb, score, sid
            elif best_bytes is None:
                if best_metric is None or metric_better(score, best_metric, self.metric):
                    best_metric, best_id = score, sid
        assignment = choices[best_id].contiguous()
        counts = {f: int(cnt[best_id, i]) for i, f in enumerate(MIXED_TILE_FORMATS)}
        metrics = {"pcc": float(met[best_id, 0]), "mae": float(met[best_id, 1]), "atol": float(met[best_id, 2])}
        transposed = mc.is_transposed(p, self.transpose)
        dr = mc.DeviceResult(self.name, p, assignment, counts, mc.total_bytes(counts), metrics, fmt_list,
                             meta={"samples": samples, "best_id": best_id}, transposed=transposed)
        if self.sample_scoring != "exact" and not transposed:
            dr._metrics = dict(metrics)            # already the reference's float32 values of the chosen sample
        # transposed: the samples are scored over x.T's flatten order; dr.metrics scores the chosen one in x's layout
        return dr

    @staticmethod
    def _reference_scores(p: engine.Prepared, choices) -> np.ndarray:
        """float32 (pcc, mae, atol) of every sample, [iters, 3] as float64 values of the float32 results."""
        import torch
        iters = choices.shape[0]
        per = p.rows * p.cols
        chunk = engine.candidate_chunk(per, iters, p.data.device)
        out = np.zeros((iters, 3), dtype=np.float64)
        ys = torch.empty((chunk, per), dtype=torch.bfloat16, device=p.data.device)
        L = engine._lib.lib()
        for s0 in range(0, iters, chunk):
            k = min(chunk, iters - s0)
            for j in range(k):
                engine.check(L.qa_apply_assignment(p.data.data_ptr(), p.dtype_code, p.rows, p.cols, p.cols,
                                                   choices[s0 + j].data_ptr(), ys[j].data_ptr(), engine._stream()), "qa_apply_assignment")
            out[s0:s0 + k] = engine.tensor_scores_f32(p.data, ys[:k], n=p.numel)[:, :3].astype(np.float64)
        return out

    def _compress(self, xf, quantizer, tile_formats):
        if mc.numel_of(xf) == 0:
            y, counts, assignment = mc.empty_result(xf)
            return y, counts, assignment, []
        dr = self.run_prepared(mc.prepare(xf, self.transpose), tile_formats)
        y, counts, assignment = mc.finish(dr, xf)
        return y, counts, assignment, dr.meta["samples"]

    def run(self, xf, formats, quantizer=None, cache=None):
        tile_formats = self.formats or self._filter_from_formats(formats)
        y, counts, assignment, samples = self._compress(xf=xf, quantizer=quantizer, tile_formats=tile_formats)
        return [CompressionResult(fmt="MIXED", compression=self.name, y=y, tile_counts=counts,
                                  tile_bytes=mc.total_bytes(counts),
                                  meta={"samples": samples, "tile_formats": tile_formats, "assignment": assignment})]
