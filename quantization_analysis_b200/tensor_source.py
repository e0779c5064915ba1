"""Where `wq`, the sweep and `reconstruct` get their tensors (replaces the network half of hf_model_utils.py:80-287).

The reference resolves a Hugging Face repo, downloads safetensors shards, dequantizes fp8 blocks and keeps every tensor as
float32 ``.npy`` under ``<cache-dir>/tensor-fp32/<repo--rev--sha1[:12]>/<tensor--sha1[:12]>.npy`` (hf_model_utils.py:114-132,
245-287).  This build has no network.  Three sources, in this order of precedence:

* a local checkpoint directory (``checkpoint_dir``: ``*.safetensors`` shards, a plain export or a hub snapshot): tensors are
  read as stored - bf16 stays bf16, block-scaled fp8 stays fp8 bytes + scale grid (`Fp8Blocks`) - and the float32 cache is
  neither read nor written;
* the reference's float32 cache when it is populated for the repo (a cache filled by the reference - or by a test - is a
  drop-in source);
* the pseudo-repo ``synthetic``, mapped to the synthetic DeepSeek-R1 shapes of ``synthetic.py``.
"""
from __future__ import annotations

import hashlib
import json
import re
from dataclasses import dataclass, field
from pathlib import Path
from urllib.parse import urlparse

import numpy as np
import torch

from . import synthetic

CHECKPOINT_INDEX = "model.safetensors.index.json"
# stored dtypes handed to the device as they are: engine.to_device keeps bf16, widens the others to float32 on the device
# (exact, or for F64 the same rounding as the reference's .to(torch.float32))
FLOAT_DTYPES = ("BF16", "F16", "F32", "F64", "F8_E4M3", "F8_E5M2")

SYNTHETIC_REPO = "synthetic/DeepSeek-R1-shapes"


def normalize_repo_id(raw: str) -> str:
    """`org/name`, or a huggingface.co URL of a model repo (hf_model_utils.py:25-57)."""
    value = raw.strip()
    if not value:
        raise ValueError("Empty repo value.")
    if "://" not in value:
        return value.strip("/")
    u = urlparse(value)
    host = u.netloc.lower()
    host = host[4:] if host.startswith("www.") else host
    if host not in ("huggingface.co", "hf.co"):
        raise ValueError(f"Unsupported host: {u.netloc}")
    parts = [p for p in u.path.split("/") if p]
    if not parts:
        raise ValueError("URL path does not contain a repo id.")
    if parts[0] in ("models", "model"):
        parts = parts[1:]
    elif parts[0] in ("datasets", "spaces"):
        raise ValueError("Only model repos are supported.")
    for i, p in enumerate(parts):
        if p in ("tree", "blob", "resolve", "commit", "discussions"):
            parts = parts[:i]
            break
    return "/".join(parts[:2]) if len(parts) >= 2 else parts[0]


def safe_repo_revision_key(repo_id: str, revision: str) -> str:
    """hf_model_utils.py:114-118."""
    digest = hashlib.sha1(f"{repo_id}@{revision}".encode("utf-8")).hexdigest()[:12]
    return f"{repo_id.replace('/', '__')}--{re.sub(r'[^A-Za-z0-9._-]+', '_', revision)}--{digest}"


def safe_tensor_key(tensor_name: str) -> str:
    """hf_model_utils.py:121-126."""
    digest = hashlib.sha1(tensor_name.encode("utf-8")).hexdigest()[:12]
    safe = re.sub(r"[^A-Za-z0-9._-]+", "_", tensor_name).strip("_") or "tensor"
    return f"{safe}--{digest}"


def filter_tensor_names(names, query):
    """Substring, or dotted prefix path (hf_model_utils.py:60-77)."""
    if not query or not query.strip():
        return sorted(names)
    q = query.strip()
    if "." in q:
        qp = [p.lower() for p in q.split(".") if p]
        return sorted(n for n in names if n.lower().split(".")[: len(qp)] == qp)
    return sorted(n for n in names if q.lower() in n.lower())


def resolve_format_list(values, supported):
    """hf_model_utils.py:317-335."""
    if not values:
        return list(supported)
    out = []
    for raw in values:
        v = raw.strip().lower()
        if v == "all":
            out += [s for s in supported if s not in out]
            continue
        if v not in supported:
            raise ValueError(f"Unsupported format '{raw}'. Supported: {', '.join(supported)}, all")
        if v not in out:
            out.append(v)
    return out


@dataclass
class Fp8Blocks:
    """A block-scaled fp8 weight as DeepSeek-V3/R1 checkpoints store it: e4m3fn bytes and a float32 grid of per-block inverse
    scales, block = ceil(shape / grid shape) (hf_model_utils.py:199-215).  engine.prepare_loaded makes an Fp8Prepared of it."""
    weight: torch.Tensor            # float8_e4m3fn [rows, cols], host
    scale_inv: torch.Tensor         # float32 [grid rows, grid cols], host

    @property
    def shape(self) -> tuple:
        return tuple(self.weight.shape)

    def dequantize_cpu(self) -> np.ndarray:
        """The reference's float32 image on the host: every byte widened to float32 times its block's scale (one rounding)."""
        rows, cols = self.shape
        br, bc = -(-rows // self.scale_inv.shape[0]), -(-cols // self.scale_inv.shape[1])
        s = self.scale_inv.repeat_interleave(br, 0).repeat_interleave(bc, 1)[:rows, :cols]
        return (self.weight.to(torch.float32) * s).numpy()


def check_scale_grid(name: str, shape, grid) -> None:
    """A 2-D grid of blocks ceil(shape / grid): every grid row and column must hold at least one element of the weight."""
    for n, g in zip(shape, grid):
        if g < 1 or n < 1 or -(-n // -(-n // g)) != g:
            raise ValueError(f"{name}: scale grid {tuple(grid)} does not tile the weight {tuple(shape)} in blocks of "
                             f"ceil(shape / grid); only 2-D F32 block grids are supported")


def _header(path: Path) -> dict[str, tuple[str, tuple]]:
    """name -> (safetensors dtype string, shape), from the shard's header only."""
    from safetensors import safe_open
    out = {}
    with safe_open(str(path), framework="pt") as f:
        for k in f.keys():
            sl = f.get_slice(k)
            out[k] = (sl.get_dtype(), tuple(sl.get_shape()))
    return out


def _read_tensor(path: str, name: str) -> torch.Tensor:
    from safetensors import safe_open
    with safe_open(path, framework="pt") as f:
        return f.get_tensor(name)


def scan_checkpoint(checkpoint_dir) -> tuple[dict[str, str], dict[str, str], dict[str, tuple]]:
    """Index of a directory of ``*.safetensors`` shards (hf_model_utils.py:80-111): ``model.safetensors.index.json``'s
    weight_map when present, else every shard's header.  -> ({name: shard path}, {name: stored dtype}, {name: shape})."""
    d = Path(checkpoint_dir)
    if not d.is_dir():
        raise FileNotFoundError(f"Checkpoint directory {d} does not exist")
    files: dict[str, str] = {}
    dtypes: dict[str, str] = {}
    shapes: dict[str, tuple] = {}
    index_file = d / CHECKPOINT_INDEX
    if index_file.is_file():
        weight_map = json.loads(index_file.read_text(encoding="utf-8")).get("weight_map")
        if not isinstance(weight_map, dict):
            raise ValueError(f"{index_file} has no weight_map")
        by_shard: dict[str, list[str]] = {}
        for name, shard in weight_map.items():
            by_shard.setdefault(str(shard), []).append(name)
        for shard, names in sorted(by_shard.items()):
            path = d / shard
            if not path.is_file():
                raise FileNotFoundError(f"{index_file.name} maps {names[0]} to {shard}, which is not in {d}")
            header = _header(path)
            for name in names:
                if name not in header:
                    raise ValueError(f"{index_file.name} maps {name} to {shard}, which does not hold it")
                files[name], (dtypes[name], shapes[name]) = str(path), header[name]
    else:
        shards = sorted(d.glob("*.safetensors"))
        if not shards:
            raise FileNotFoundError(f"No *.safetensors shards and no {CHECKPOINT_INDEX} in {d}")
        for path in shards:
            for name, (dt, shape) in _header(path).items():
                if name in files:
                    raise ValueError(f"Tensor {name} is in two shards: {Path(files[name]).name} and {path.name}")
                files[name], dtypes[name], shapes[name] = str(path), dt, shape
    order = sorted(files)
    return {n: files[n] for n in order}, {n: dtypes[n] for n in order}, {n: shapes[n] for n in order}


@dataclass
class TensorIndex:
    """The part of hf_model_utils.ModelIndex (:103-111) the analysis loop uses."""
    repo_id: str
    revision: str
    cache_dir: Path
    tensor_to_file: dict = field(default_factory=dict)      # name -> .npy path, shard path, or "synthetic"
    synthetic_seed: int = 1000
    checkpoint_dir: Path | None = None
    dtypes: dict = field(default_factory=dict)              # name -> stored safetensors dtype (checkpoint source only)
    shapes: dict = field(default_factory=dict)              # name -> stored shape (checkpoint source only)

    def fp32_cache_dir(self) -> Path:
        return Path(self.cache_dir) / "tensor-fp32" / safe_repo_revision_key(self.repo_id, self.revision)

    def cache_file(self, name: str) -> Path:
        return self.fp32_cache_dir() / f"{safe_tensor_key(name)}.npy"

    def scale_name(self, name: str) -> str | None:
        """The ``<name>_scale_inv`` sibling of a block-scaled fp8 weight, or None."""
        s = f"{name}_scale_inv"
        return s if self.dtypes.get(name) == "F8_E4M3" and s in self.tensor_to_file else None

    def describe(self, name: str) -> str:
        """Where `name` is read from (the per-tensor screen line of wq)."""
        if self.checkpoint_dir is not None:
            s = self.scale_name(name)
            blocks = f" + {self.dtypes[s]} {s.rsplit('.', 1)[-1]}" if s else ""
            return f"checkpoint: {Path(self.tensor_to_file[name]).name} {self.dtypes[name]}{blocks}"
        cf = self.cache_file(name)
        return f"cache: fp32 hit ({cf})" if cf.exists() else "cache: synthetic tensor"

    def shape(self, name: str) -> tuple:
        """The shape `load(name)` returns, from headers only (safetensors header, ``.npy`` header, synthetic table): sizes a
        tensor list without reading its data."""
        if self.checkpoint_dir is not None:
            return self.shapes[name]
        src = self.tensor_to_file[name]
        if src == "synthetic":
            return tuple(synthetic.DEEPSEEK_R1_SHAPES[name])
        return tuple(np.load(src, mmap_mode="r").shape)

    def load(self, name: str):
        """What the analysis reads for `name`: from a checkpoint the host torch tensor as stored, or `Fp8Blocks` for a
        block-scaled fp8 weight; otherwise the float32 ndarray of the cache or the synthetic provider."""
        if self.checkpoint_dir is None:
            return np.asarray(self.load_fp32(name), dtype=np.float32)
        dt = self.dtypes[name]
        if dt not in FLOAT_DTYPES:
            raise ValueError(f"{name}: stored as {dt}; only floating-point tensors can be analysed")
        w = _read_tensor(self.tensor_to_file[name], name)
        s = self.scale_name(name)
        if s is None:
            return w
        if w.dim() != 2:
            raise ValueError(f"{name}: a block-scaled fp8 weight must be 2-D, got shape {tuple(w.shape)}")
        if self.dtypes[s] != "F32":
            raise ValueError(f"{name}: scale grid {s} is {self.dtypes[s]}; only 2-D F32 block grids are supported")
        sc = _read_tensor(self.tensor_to_file[s], s)
        if sc.dim() != 2:
            raise ValueError(f"{name}: scale grid {s} has shape {tuple(sc.shape)}; only 2-D F32 block grids are supported")
        check_scale_grid(name, w.shape, sc.shape)
        return Fp8Blocks(w, sc)

    def load_fp32(self, name: str) -> np.ndarray:
        """The float32 values the reference's loader hands to the algorithms (hf_model_utils.py:241-287)."""
        if self.checkpoint_dir is not None:
            x = self.load(name)
            return x.dequantize_cpu() if isinstance(x, Fp8Blocks) else x.to(torch.float32).numpy()
        src = self.tensor_to_file[name]
        if src == "synthetic":
            i = list(self.tensor_to_file).index(name)
            return synthetic.randn_f32_np(synthetic.DEEPSEEK_R1_SHAPES[name], self.synthetic_seed + i)
        return np.load(src)


def build_tensor_index(repo_or_url: str, revision: str = "main", cache_dir="data/hf-cache", synthetic_seed: int = 1000,
                       checkpoint_dir=None) -> TensorIndex:
    """checkpoint_dir given: the shards there, and nothing else.  Otherwise the float32 cache, then ``synthetic``."""
    repo_id = normalize_repo_id(repo_or_url)
    idx = TensorIndex(repo_id=repo_id, revision=revision, cache_dir=Path(cache_dir), synthetic_seed=synthetic_seed)
    if checkpoint_dir is not None:
        idx.checkpoint_dir = Path(checkpoint_dir)
        idx.tensor_to_file, idx.dtypes, idx.shapes = scan_checkpoint(checkpoint_dir)
        return idx
    d = idx.fp32_cache_dir()
    names = {}
    if d.is_dir():
        for f in sorted(d.glob("*.npy")):
            stem = f.name[:-4]
            if "--" not in stem:
                continue
            name, digest = stem.rsplit("--", 1)
            # the cache key keeps tensor names made of [A-Za-z0-9._-] verbatim; the digest tells whether it did
            if hashlib.sha1(name.encode("utf-8")).hexdigest()[:12] == digest:
                names[name] = str(f)
    if names:
        idx.tensor_to_file = names
        return idx
    if repo_id.split("/")[0].lower() == "synthetic" or repo_id.lower() == "synthetic":
        idx.tensor_to_file = {n: "synthetic" for n in synthetic.DEEPSEEK_R1_SHAPES}
        return idx
    raise RuntimeError(
        f"No cached float32 tensors for {repo_id}@{revision} under {d} and no network access in this build: "
        f"populate that directory (the reference's own cache layout), name a local checkpoint with --checkpoint-dir, or use the "
        f"repo name 'synthetic'.")


def resolve_selected_tensors(index: TensorIndex, filter_query) -> list[str]:
    """hf_model_utils.py:290-301."""
    names = list(index.tensor_to_file)
    weight_like = [n for n in names if "weight" in n.lower() and not n.lower().endswith("_scale_inv")]
    sel = filter_tensor_names(weight_like if weight_like else names, filter_query)
    if not sel:
        sel = filter_tensor_names(names, filter_query)
    if not sel:
        raise RuntimeError("No tensors matched the filter query.")
    return sel
