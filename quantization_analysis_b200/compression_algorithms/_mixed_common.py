"""Shared host logic of the three mixed-tile algorithms: parameter parsing, device results."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from .. import engine
from .tile_utils import MIXED_TILE_FORMATS, mixed_tile_total_bytes

VALID_METRICS = {"pcc", "mae", "atol"}


def parse_formats(value) -> list[str]:
    """'bfp8,bfp4' or ['bfp8', ...] -> de-duplicated list of mixed-tile formats, order kept."""
    if value is None or value == "":
        return []
    if isinstance(value, str):
        items = value.split(",")
    elif isinstance(value, list):
        items = [str(v) for v in value]
    else:
        raise ValueError("formats must be a comma-separated string or a list of strings")
    out: list[str] = []
    for raw in items:
        name = raw.strip().lower()
        if not name:
            continue
        if name not in MIXED_TILE_FORMATS:
            raise ValueError(f"Unsupported mixed-tile format: {name}")
        if name not in out:
            out.append(name)
    return out


def filter_formats(formats, algo_name: str) -> list[str]:
    allowed = [f for f in formats if f in MIXED_TILE_FORMATS]
    if not allowed:
        raise ValueError(
            f"{algo_name} requires at least one of {', '.join(MIXED_TILE_FORMATS)} in quantization_formats")
    return allowed


@dataclass
class DeviceResult:
    """What one algorithm run leaves on the device (nothing is copied to the host unless asked).  transposed: the run was
    in the device layout - `prepared` holds x.T (engine.prepare_transposed) and the map is over its tiles - while y_device()
    and `metrics` are in x's layout."""
    compression: str
    prepared: engine.Prepared
    assignment: torch.Tensor | None        # int8 [ntiles] (device) for mixed results
    counts: dict
    tile_bytes: float
    metrics_exact: dict                    # float64 recombination of pcc / mae / atol from the tile-stat table
    tile_formats: list[str]
    meta: dict = field(default_factory=dict)
    transposed: bool = False
    _y: torch.Tensor | None = None
    _metrics: dict | None = None

    @property
    def shape(self) -> tuple:
        """Shape of x (and of y)."""
        p = self.prepared
        return tuple(reversed(p.shape)) if self.transposed else p.shape

    @property
    def metrics(self) -> dict:
        """pcc / mae / atol of the result as the reference reports them (wq:684-687): float32, NumPy's summation orders
        (qa_tensor_scores_f32 over x and the materialised reconstruction, both in x's layout)."""
        if self._metrics is None:
            p = self.prepared
            s = engine.tensor_scores_f32(self.x_device(), self.y_device(), n=p.numel)[0]
            self._metrics = {"pcc": float(s[0]), "mae": float(s[1]), "atol": float(s[2])}
        return self._metrics

    def x_device(self) -> torch.Tensor:
        """x on the device in its own layout (flat; a transposed run transposes its copy back)."""
        p = self.prepared
        if not self.transposed:
            return p.data
        return engine.transpose_2d(p.data.reshape(p.rows, p.cols)).reshape(-1)

    def y_device(self) -> torch.Tensor:
        """bf16 reconstruction on the device (materialised on first use), flat, in x's layout."""
        if self._y is None:
            y = engine.apply_assignment(self.prepared, self.assignment)
            if self.transposed:
                p = self.prepared
                y = engine.transpose_2d(y.reshape(p.rows, p.cols)).reshape(-1)
            self._y = y
        return self._y

    def assignment_numpy(self) -> np.ndarray:
        """The map [tiles_h, tiles_w] over the tiles of the layout the run used (x.T's when transposed)."""
        p = self.prepared
        return self.assignment.cpu().numpy().astype(np.int8).reshape(p.tiles_h, p.tiles_w)


def counts_dict(counts_dev) -> dict:
    c = counts_dev.cpu().numpy().astype(np.int64).reshape(-1)
    return {f: int(c[i]) for i, f in enumerate(MIXED_TILE_FORMATS)}


def empty_result(xf):
    """Empty input (mixed_tile_greedy.py:78-83)."""
    return np.asarray(xf, dtype=np.float32), {f: 0 for f in MIXED_TILE_FORMATS}, np.zeros((1, 1), dtype=np.int8)


def is_torch(x) -> bool:
    return isinstance(x, torch.Tensor)


def numel_of(x) -> int:
    return int(x.numel()) if is_torch(x) else int(np.asarray(x).size)


def finish(dr: DeviceResult, xf, extra_meta: dict | None = None):
    """DeviceResult -> the reference's (y, counts, assignment) triple in the caller's array type; y has x's shape."""
    y_dev = dr.y_device()
    if dr.transposed:
        y = y_dev.reshape(dr.shape)
        if not is_torch(xf):
            y = y.to(torch.float32).cpu().numpy()
    elif is_torch(xf):
        p = dr.prepared
        y = y_dev[: p.numel].reshape(p.shape) if p.kind == "vector" else y_dev.reshape(p.shape)
    else:
        y = engine.result_to_numpy(dr.prepared, y_dev)
    return y, dr.counts, dr.assignment_numpy()


def parse_transpose(params: dict) -> bool:
    """params["transpose"] (default False): run in the device layout, over the tiles of x.T.  Only a bool is accepted."""
    v = params.get("transpose", False)
    if not isinstance(v, bool):
        raise ValueError(f"transpose must be true or false, not {v!r}")
    return v


def prepare(xf, transpose: bool) -> engine.Prepared:
    """x in the layout an algorithm runs in: x.T's tiles when `transpose` (engine.prepare_transposed), else x's."""
    return engine.prepare_transposed(xf) if transpose else engine.prepare_tiles(xf)


def is_transposed(p: engine.Prepared, transpose: bool) -> bool:
    """Whether a run with the flag over `p` is in a layout other than x's (0-D and 1-D inputs: x.T is x)."""
    return bool(transpose) and p.kind == "nd"


def total_bytes(counts: dict) -> float:
    return mixed_tile_total_bytes(counts)
