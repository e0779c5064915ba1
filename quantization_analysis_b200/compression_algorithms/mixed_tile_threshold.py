"""mixed-tile-threshold on the device (reference: compression_algorithms/mixed_tile_threshold.py:19-162).

Per-tile scores are the reference's float32 values, reproduced bit-for-bit on the GPU
(qa_tile_scores_f32); every tile then takes the cheapest format whose float32 score passes the
float32 threshold (qa_threshold_assign), else the highest-precision candidate.
"""
from __future__ import annotations

from .. import engine
from .base import CompressionAlgorithm, CompressionResult
from . import _mixed_common as mc
from .tile_utils import MIXED_TILE_BYTES_PER_ELEM, MIXED_TILE_FORMATS

_METRIC_ROW = {"pcc": 0, "mae": 1, "atol": 2}


def formats_by_precision(tile_formats) -> list[str]:
    """Ascending bytes/elem, stable (mixed_tile_threshold.py:112-114)."""
    return sorted(tile_formats, key=lambda f: MIXED_TILE_BYTES_PER_ELEM.get(f, 0.0))


class MixedTileThresholdCompression(CompressionAlgorithm):
    name = "mixed-tile-threshold"

    def __init__(self, params: dict | None = None) -> None:
        super().__init__(params=params)
        self.metric = self.params.get("metric", "pcc")
        self.threshold = float(self.params.get("threshold", 0.999))
        raw = self.params.get("formats", self.params.get("tile_formats"))
        self.tile_formats = mc.parse_formats(raw) if raw is not None else None
        self.transpose = mc.parse_transpose(self.params)          # extension: the device layout (tiles of x.T)
        if self.metric not in mc.VALID_METRICS:
            raise ValueError(f"Unsupported metric: {self.metric}")

    @classmethod
    def from_params(cls, params: dict | None = None) -> "MixedTileThresholdCompression":
        return cls(params=params or {})

    def expected_evals(self, formats) -> int:
        return 1

    _parse_formats = staticmethod(mc.parse_formats)

    @staticmethod
    def _filter_from_formats(formats):
        return mc.filter_formats(formats, "mixed-tile-threshold")

    def run_prepared(self, p: engine.Prepared, tile_formats, scores=None, table=None) -> mc.DeviceResult:
        if scores is None:
            scores = engine.tile_scores(p, tile_formats)
        order = formats_by_precision(tile_formats)
        # best_precision = max by bytes; with the ascending stable sort that is the last entry,
        # which qa_threshold_assign uses as the fallback.
        assignment, counts_dev = engine.threshold_assign(scores[_METRIC_ROW[self.metric]].contiguous(), order,
                                                         self.metric == "pcc", [self.threshold])
        counts = mc.counts_dict(counts_dev[0])
        metrics = None                       # float64 recombination only when the caller already has the table
        if table is not None:
            metrics = engine.metrics_from_sums(engine.assignment_sums(table, assignment[0]).cpu().numpy(), p.numel)
        return mc.DeviceResult(self.name, p, assignment[0], counts, mc.total_bytes(counts), metrics, list(tile_formats),
                               meta={"scores": scores}, transposed=mc.is_transposed(p, self.transpose))

    def _compress(self, xf, quantizer, tile_formats):
        if mc.numel_of(xf) == 0:
            return mc.empty_result(xf)
        dr = self.run_prepared(mc.prepare(xf, self.transpose), tile_formats)
        return mc.finish(dr, xf)

    def run(self, xf, formats, quantizer=None, cache=None):
        tile_formats = self.tile_formats or self._filter_from_formats(formats)
        y, counts, assignment = self._compress(xf=xf, quantizer=quantizer, tile_formats=tile_formats)
        return [CompressionResult(fmt="MIXED", compression=self.name, y=y, tile_counts=counts,
                                  tile_bytes=mc.total_bytes(counts),
                                  meta={"assignment": assignment, "tile_formats": tile_formats})]
