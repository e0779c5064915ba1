"""mixed-tile-greedy on the device (reference: compression_algorithms/mixed_tile_greedy.py:20-378).

One fused pass builds the per-tile statistic table (qa_tile_stats); the greedy decision chain -
NumPy-stream permutation per candidate format, accept a tile's switch iff the global metric
recomputed from running float64 sums still passes - runs on the device over that table
(qa_greedy_assign); the final reconstruction is a per-tile apply (qa_apply_assignment).
"""
from __future__ import annotations

import secrets

from .. import engine
from .base import CompressionAlgorithm, CompressionResult
from . import _mixed_common as mc
from .tile_utils import MIXED_TILE_FORMATS


class MixedTileGreedyCompression(CompressionAlgorithm):
    name = "mixed-tile-greedy"

    def __init__(self, params: dict | None = None) -> None:
        super().__init__(params=params)
        raw = self.params.get("formats", self.params.get("tile_formats"))
        self.metric = self.params.get("metric", "pcc")
        self.threshold = float(self.params.get("threshold", 0.999))
        self.seed = int(self.params.get("seed", 0))
        self.strict = bool(self.params.get("strict_sums", False))   # extension: NumPy-order float64 tile sums
        self.sequential = bool(self.params.get("sequential_chain", False))  # extension: one-thread decision chain
        # extension: certify the map.  The cluster kernel reports a lower bound of min |value - thr| / thr over all its decisions
        # (state[20]); the fast path's sums can differ from the reference's by at most `margin_bound` in relative terms (the
        # fast tile-stat kernel's sum x^2 is 1e-13-close per tile, the initial sums of zero-mean tensors are tree sums), so a
        # run whose margin stays above the bound made the reference's decisions.  Below it the tensor is redone with
        # NumPy-order tile sums and the one-thread reference-order chain.
        self.certify = bool(self.params.get("certify", True))
        self.margin_bound = float(self.params.get("margin_bound", 2e-13))
        self.tile_formats = mc.parse_formats(raw) if raw is not None else None
        if self.metric not in mc.VALID_METRICS:
            raise ValueError(f"Unsupported metric: {self.metric}")

    @classmethod
    def from_params(cls, params: dict | None = None) -> "MixedTileGreedyCompression":
        return cls(params=params or {})

    def expected_evals(self, formats) -> int:
        return 1

    _parse_formats = staticmethod(mc.parse_formats)

    @staticmethod
    def _filter_from_formats(formats):
        return mc.filter_formats(formats, "mixed-tile-greedy")

    def run_prepared(self, p: engine.Prepared, tile_formats, table=None, seed: int | None = None) -> mc.DeviceResult:
        """Device-resident run; `table` may be shared between algorithms on the same tensor."""
        if table is None:
            table = engine.tile_stats(p, MIXED_TILE_FORMATS, strict=True if self.strict else None,
                                      exact_abs=(self.metric == "mae"))
        seed = self.seed if seed is None else seed
        if seed == 0:
            seed = secrets.randbits(31)           # mixed_tile_greedy.py:222-224
        dev = table.device
        rng = engine.make_rng(seed, dev)
        if self.sequential or self.metric == "atol":
            assignment, counts_dev, state = engine.greedy_assign(table, p.numel, self.metric, self.threshold, tile_formats, rng,
                                                                 parallel=False if self.sequential else None)
        else:   # stages overlapped on side streams: same bits, about half the latency
            assignment, counts_dev, state = engine.greedy_assign_staged(table, p.numel, self.metric, self.threshold, tile_formats, rng)
        cert = {"min_margin": None, "fallback": False}
        fast = not (self.sequential or self.metric == "atol")
        if fast:
            st = state.cpu().numpy()
            cert["min_margin"], cert["flags"] = float(st[20]), int(st[6]) & 7
            if self.certify and not self.strict and not (cert["min_margin"] >= self.margin_bound):
                # a decision closer to the threshold than the sums are to the reference's: reference-order everything
                cert["fallback"] = True
                table = engine.tile_stats(p, MIXED_TILE_FORMATS, strict=True)
                rng = engine.make_rng(seed, dev)
                assignment, counts_dev, state = engine.greedy_assign(table, p.numel, self.metric, self.threshold, tile_formats, rng,
                                                                     parallel=False)
        counts = mc.counts_dict(counts_dev)
        sums = engine.assignment_sums(table, assignment)
        metrics = engine.metrics_from_sums(sums.cpu().numpy(), p.numel)
        return mc.DeviceResult(self.name, p, assignment, counts, mc.total_bytes(counts), metrics, list(tile_formats),
                               meta={"seed": seed, "state": state, "table": table, "certificate": cert})

    def run_fp8_blocks(self, w_fp8, scale_inv, formats=None, seed: int | None = None) -> mc.DeviceResult:
        """Extension for real checkpoints: an fp8 e4m3fn tensor + per-block inverse scales as stored on disk
        (hf_model_utils.py:199-215,271-281).  The table comes from one pass over the bytes (engine.tile_stats on an Fp8Prepared);
        the result is what `run` gives on the reference's dequantized float32 tensor."""
        tile_formats = self.tile_formats or self._filter_from_formats(formats or MIXED_TILE_FORMATS)
        return self.run_prepared(engine.Fp8Prepared(w_fp8, scale_inv), tile_formats, seed=seed)

    def _compress(self, xf, quantizer, tile_formats):
        if mc.numel_of(xf) == 0:
            return mc.empty_result(xf)
        dr = self.run_prepared(engine.prepare_tiles(xf), tile_formats)
        return mc.finish(dr, xf)

    def run(self, xf, formats, quantizer=None, cache=None):
        tile_formats = self.tile_formats or self._filter_from_formats(formats)
        y, counts, assignment = self._compress(xf=xf, quantizer=quantizer, tile_formats=tile_formats)
        return [CompressionResult(fmt="MIXED", compression=self.name, y=y, tile_counts=counts,
                                  tile_bytes=mc.total_bytes(counts),
                                  meta={"assignment": assignment, "tile_formats": tile_formats})]
