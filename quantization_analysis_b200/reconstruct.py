"""Reconstruct a tensor from a saved mixed-tile assignment on the device.

Mirrors scripts/reconstruct_mixed_tile_assignment.py:40-137 of the reference: read ``assignment.npy`` (int8
``[tiles_h, tiles_w]``) and its mapping JSON (``int_to_format``), quantize every 32x32 tile of the tensor in the format the
map names (qa_apply_assignment: one pass, 4 B/element) and return / save the float32 reconstruction.  The reference loads
the tensor from the model; this module takes the tensor itself, a tensor name resolved through the ``*.safetensors`` shards
of ``--checkpoint-dir`` (as wq reads them), a ``.npy`` file, or a DeepSeek-R1 weight name resolved through ``synthetic.py``.
"""
from __future__ import annotations

import argparse
import json
from pathlib import Path

import numpy as np
import torch

from . import engine, synthetic, tensor_source

_DEVICE_FORMATS = ("bf16", "bfp8", "bfp4", "bfp2")


def load_mapping(path) -> list[str]:
    """``int_to_format`` of an assignment mapping JSON (reconstruct_mixed_tile_assignment.py:62-79)."""
    data = json.loads(Path(path).read_text())
    formats = data.get("int_to_format")
    if not isinstance(formats, list) or not formats:
        raise ValueError("assignment mapping must contain int_to_format list")
    return [str(x).strip().lower() for x in formats]


def reconstruct_from_assignment(x, assignment: np.ndarray, int_to_format=None) -> np.ndarray:
    """-> float32 array of x's shape: tile (i, j) quantized in format ``int_to_format[assignment[i, j]]``.  x: a host array or
    tensor, or what tensor_source's loaders return (tensor_source.Fp8Blocks included)."""
    int_to_format = list(int_to_format) if int_to_format is not None else list(_DEVICE_FORMATS)
    p = engine.prepare_loaded(x)
    a = np.asarray(assignment, dtype=np.int8)
    expected = (p.tiles_h, p.tiles_w)
    if a.shape != expected:
        raise ValueError(f"Assignment shape {a.shape} does not match expected {expected}")   # :100-101
    if a.size and (a.min() < 0 or a.max() >= len(int_to_format)):
        raise ValueError("assignment value outside the mapping")
    remap = np.empty(len(int_to_format), dtype=np.int8)
    for i, f in enumerate(int_to_format):
        if f not in _DEVICE_FORMATS:
            raise ValueError(f"format '{f}' cannot be reconstructed per tile on the device")
        remap[i] = engine.FMT_INDEX[f]
    dev_map = torch.from_numpy(remap[a.reshape(-1)]).to(p.data.device)
    return engine.result_to_numpy(p, engine.apply_assignment(p, dev_map))


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description="Reconstruct a tensor from a mixed-tile assignment")
    ap.add_argument("tensor_name", help="tensor name in --checkpoint-dir, a .npy file with the tensor, or (without "
                                        "--checkpoint-dir) a weight name of synthetic.DEEPSEEK_R1_SHAPES")
    ap.add_argument("--assignment", required=True)
    ap.add_argument("--assignment-mapping", required=True)
    ap.add_argument("--seed", type=int, default=0, help="seed of the synthetic tensor")
    ap.add_argument("--out", default=None)
    ap.add_argument("--checkpoint-dir", default=None, help="directory of *.safetensors shards holding tensor_name")
    args = ap.parse_args(argv)
    if args.checkpoint_dir is not None:
        index = tensor_source.build_tensor_index(str(args.checkpoint_dir), checkpoint_dir=args.checkpoint_dir)
        if args.tensor_name not in index.tensor_to_file:
            ap.error(f"{args.tensor_name} is not in the checkpoint {args.checkpoint_dir}")
        x = index.load(args.tensor_name)
    elif args.tensor_name.endswith(".npy"):
        x = np.load(args.tensor_name)
    else:
        x = synthetic.randn_bf16_cpu(synthetic.DEEPSEEK_R1_SHAPES[args.tensor_name], args.seed).float().numpy()
    y = reconstruct_from_assignment(x, np.load(args.assignment), load_mapping(args.assignment_mapping))
    out = args.out or str(Path(args.assignment).with_suffix("")) + "_recon.npy"
    np.save(out, y)
    print(f"Wrote reconstructed tensor to {out}")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
