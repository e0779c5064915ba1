"""Local safetensors checkpoints as a tensor source (tensor_source.build_tensor_index(checkpoint_dir=...)) for wq, the sweep
and reconstruct.

The fixture checkpoint is written under a temporary directory from values already in the tree: layer 0 is the tiny CLI
'repository' of tests/cli_util.py (q_a_proj stored as F32, the bf16-exact rest as BF16), layer 1 is the ragged fp8 golden
of tests/golden/fp8_dequant.npz (300 x 520 e4m3fn bytes, a 3 x 5 F32 scale grid) whose reference dequantization is
``rag__out``.  Host tests check the index and the loader; device tests check the programs against the reference's goldens
and the fp8 route against the float32-cache route.
"""
import json
import os
import re
from pathlib import Path

import numpy as np
import pytest
import torch
from safetensors.torch import load_file, save_file

from quantization_analysis_b200 import tensor_source
from quantization_analysis_b200.tensor_source import CHECKPOINT_INDEX, Fp8Blocks
from tests import cli_util as U
from tests import golden_util as G

L1 = "model.layers.1.self_attn.q_b_proj.weight"
SHARDS = ("model-00001-of-00002.safetensors", "model-00002-of-00002.safetensors")


def fp8_golden():
    """-> (e4m3fn bytes uint8 [300, 520], scale grid float32 [3, 5], the reference's float32 dequantization)."""
    z = G.npz("fp8_dequant.npz")
    w = z["rag__w"]
    return w, z["rag__s"], z["rag__out"].view(np.float32).reshape(w.shape)


def shard_contents() -> dict[str, dict[str, torch.Tensor]]:
    layer0 = {}
    for name, x in U.tensors().items():
        t = torch.from_numpy(x)
        if name != U.SWEEP_TENSOR:                     # q_a_proj is not bf16-exact: stored as F32
            assert torch.equal(t.to(torch.bfloat16).float(), t), name
            t = t.to(torch.bfloat16)
        layer0[name] = t
    w, s, _ = fp8_golden()
    layer1 = {L1: torch.from_numpy(w).view(torch.float8_e4m3fn), f"{L1}_scale_inv": torch.from_numpy(s)}
    return {SHARDS[0]: layer0, SHARDS[1]: layer1}


def write_checkpoint(d: Path, with_index: bool = True) -> Path:
    d.mkdir(parents=True, exist_ok=True)
    contents = shard_contents()
    for shard, tensors in contents.items():
        save_file(tensors, str(d / shard), metadata={"format": "pt"})
    if with_index:
        weight_map = {n: shard for shard, tensors in contents.items() for n in tensors}
        (d / CHECKPOINT_INDEX).write_text(json.dumps({"metadata": {}, "weight_map": weight_map}, indent=2))
    return d


def one_shard(d: Path, tensors: dict) -> tensor_source.TensorIndex:
    d.mkdir(parents=True, exist_ok=True)
    save_file(tensors, str(d / "model.safetensors"), metadata={"format": "pt"})
    return tensor_source.build_tensor_index(U.REPO, checkpoint_dir=d)


def raw(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.uint8)


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    return write_checkpoint(tmp_path_factory.mktemp("ckpt") / "tiny-r1")


# ------------------------------------------------------------------------------------------------------------------------
# host
# ------------------------------------------------------------------------------------------------------------------------
def test_index_json_equals_header_scan(ckpt, tmp_path):
    """weight_map of model.safetensors.index.json == the headers of every shard; a hub snapshot (shards are symlinks into
    a blob store) is read the same way."""
    by_json = tensor_source.scan_checkpoint(ckpt)
    snap = tmp_path / "snapshots" / "abc123"
    blobs = tmp_path / "blobs"
    snap.mkdir(parents=True)
    blobs.mkdir()
    for i, shard in enumerate(SHARDS):
        (blobs / f"blob{i}").write_bytes((ckpt / shard).read_bytes())
        os.symlink(blobs / f"blob{i}", snap / shard)
    by_scan = tensor_source.scan_checkpoint(snap)
    rel = lambda files: {n: Path(f).name for n, f in files.items()}          # noqa: E731
    assert rel(by_json[0]) == rel(by_scan[0]) and by_json[1] == by_scan[1]
    assert sorted(by_json[0]) == sorted(n for ts in shard_contents().values() for n in ts)
    assert by_json[1][L1] == "F8_E4M3" and by_json[1][f"{L1}_scale_inv"] == "F32"
    assert by_json[1][U.SWEEP_TENSOR] == "F32" and by_json[1]["model.layers.0.input_layernorm.weight"] == "BF16"


def test_loaded_tensors_are_the_stored_bytes(ckpt):
    """TensorIndex.load gives each tensor bit-equal to safetensors.torch.load_file of its shard: the torch tensor as stored,
    or Fp8Blocks (bytes + scale grid) for the block-scaled fp8 weight.  load_fp32 gives the reference's float32 values."""
    index = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=ckpt)
    stored = {n: t for shard in SHARDS for n, t in load_file(str(ckpt / shard)).items()}
    for name in U.tensors():
        got = index.load(name)
        assert isinstance(got, torch.Tensor) and got.dtype == stored[name].dtype and got.shape == stored[name].shape
        assert torch.equal(raw(got), raw(stored[name])), name
        assert np.array_equal(G.bits(index.load_fp32(name)), G.bits(U.tensors()[name])), name
    got = index.load(L1)
    assert isinstance(got, Fp8Blocks) and got.weight.dtype == torch.float8_e4m3fn and got.shape == (300, 520)
    assert torch.equal(raw(got.weight), raw(stored[L1])) and torch.equal(got.scale_inv, stored[f"{L1}_scale_inv"])
    _, _, ref = fp8_golden()
    assert np.array_equal(G.bits(index.load_fp32(L1)), G.bits(ref))        # the reference's _dequantize_tensor_with_scale_inv
    assert index.describe(L1) == f"checkpoint: {SHARDS[1]} F8_E4M3 + F32 weight_scale_inv"
    assert index.describe(U.SWEEP_TENSOR) == f"checkpoint: {SHARDS[0]} F32"


def test_scale_inv_names_are_never_selected(ckpt):
    from quantization_analysis_b200 import sweep_cli
    index = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=ckpt)
    assert f"{L1}_scale_inv" in index.tensor_to_file
    for q in (None, "model.layers.1", "q_b_proj", "model.layers.1.self_attn", "weight"):
        sel = tensor_source.resolve_selected_tensors(index, q)
        assert sel and not any(n.endswith("_scale_inv") for n in sel), q
    assert tensor_source.resolve_selected_tensors(index, "model.layers.1") == [L1]
    assert sweep_cli.select_tensors(index, "layers\\.1\\.", True) == [L1]
    with pytest.raises(RuntimeError):
        sweep_cli.select_tensors(index, "scale_inv", True)


def test_checkpoint_wins_over_the_float32_cache(ckpt, tmp_path):
    """--checkpoint-dir is explicit: a populated float32 cache for the same repo is not read."""
    cache = tmp_path / "hf-cache"
    U.seed_fp32_cache(cache)
    index = tensor_source.build_tensor_index(U.REPO, cache_dir=cache, checkpoint_dir=ckpt)
    assert index.checkpoint_dir == ckpt and L1 in index.tensor_to_file
    assert all(Path(f).parent == ckpt for f in index.tensor_to_file.values())
    assert isinstance(index.load("model.layers.0.mlp.down_proj.weight"), torch.Tensor)
    plain = tensor_source.build_tensor_index(U.REPO, cache_dir=cache)            # without the flag: today's cache route
    assert plain.checkpoint_dir is None and sorted(plain.tensor_to_file) == sorted(U.tensors())


def test_missing_shard_is_rejected(tmp_path):
    d = write_checkpoint(tmp_path / "c")
    (d / SHARDS[1]).unlink()
    with pytest.raises(FileNotFoundError, match=re.escape(SHARDS[1])):
        tensor_source.scan_checkpoint(d)


def test_index_naming_a_shard_without_the_tensor_is_rejected(tmp_path):
    d = write_checkpoint(tmp_path / "c")
    meta = json.loads((d / CHECKPOINT_INDEX).read_text())
    meta["weight_map"][L1] = SHARDS[0]
    (d / CHECKPOINT_INDEX).write_text(json.dumps(meta))
    with pytest.raises(ValueError, match=re.escape(L1)):
        tensor_source.scan_checkpoint(d)


def test_duplicate_name_without_index_is_rejected(tmp_path):
    d = write_checkpoint(tmp_path / "c", with_index=False)
    save_file({U.SWEEP_TENSOR: torch.zeros(2, 2)}, str(d / "extra.safetensors"))
    with pytest.raises(ValueError, match=re.escape(U.SWEEP_TENSOR)):
        tensor_source.scan_checkpoint(d)


@pytest.mark.parametrize("dtype", [torch.int32, torch.int8, torch.bool])
def test_integer_and_bool_tensors_are_rejected(tmp_path, dtype):
    index = one_shard(tmp_path / "c", {"model.layers.0.mlp.gate.weight": torch.zeros((4, 4), dtype=dtype)})
    stored = index.dtypes["model.layers.0.mlp.gate.weight"]
    with pytest.raises(ValueError, match=re.escape("model.layers.0.mlp.gate.weight") + ".*" + stored):
        index.load("model.layers.0.mlp.gate.weight")


FP8_BAD = {
    "weight_1d": ((64,), torch.ones((1, 1))),
    "grid_empty": ((300, 520), torch.ones((0, 5))),
    "grid_too_large": ((300, 520), torch.ones((301, 5))),
    "grid_1d": ((300, 520), torch.ones(5)),
    "grid_bf16": ((300, 520), torch.ones((3, 5), dtype=torch.bfloat16)),
}


@pytest.mark.parametrize("case", sorted(FP8_BAD))
def test_unsupported_fp8_layouts_are_rejected(tmp_path, case):
    shape, scale = FP8_BAD[case]
    name = "model.layers.5.mlp.up_proj.weight"
    index = one_shard(tmp_path / "c", {name: torch.zeros(shape).to(torch.float8_e4m3fn), f"{name}_scale_inv": scale})
    with pytest.raises(ValueError, match=re.escape(name)):
        index.load(name)


# ------------------------------------------------------------------------------------------------------------------------
# device
# ------------------------------------------------------------------------------------------------------------------------
def _wq(root: Path, case: str, filt: str, source: list[str]) -> tuple[int, Path]:
    from quantization_analysis_b200 import wq
    cfg = root / f"{case}.json"
    root.mkdir(parents=True, exist_ok=True)
    cfg.write_text(json.dumps(U.WQ_CASES[case]))
    rc = wq.run([U.REPO, filt, "--compression-config", str(cfg), "--recompute", "--summary", "--results-root", str(root / "results"),
                 "--processed-root", str(root / "processed")] + source)
    return rc, U.latest_results_dir(root / "results", U.WQ_CASES[case]["algorithm"])


def _seed_layer1_cache(cache: Path) -> None:
    _, _, ref = fp8_golden()
    d = cache / "tensor-fp32" / tensor_source.safe_repo_revision_key(U.REPO, U.REVISION)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{tensor_source.safe_tensor_key(L1)}.npy", ref)


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(U.WQ_CASES))
def test_wq_checkpoint_matches_reference_output_tree(ckpt, tmp_path, case):
    """wq --checkpoint-dir over the layer-0 shards == the tree the unmodified reference wrote from its float32 cache; the
    (empty) float32 cache stays empty."""
    cache = tmp_path / "hf-cache"
    cache.mkdir()
    rc, got = _wq(tmp_path, case, U.FILTER, ["--checkpoint-dir", str(ckpt), "--cache-dir", str(cache)])
    assert rc == 0
    assert U.compare_trees(got, U.CLI_GOLDEN / "wq" / case) == []
    assert list(cache.iterdir()) == []


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(U.SWEEP_CASES))
def test_sweep_checkpoint_matches_reference_csv(ckpt, tmp_path, case):
    from quantization_analysis_b200 import sweep_cli
    cache = tmp_path / "hf-cache"
    cache.mkdir()
    rc = sweep_cli.main([U.REPO, U.SWEEP_TENSOR, "--no-regex", "--checkpoint-dir", str(ckpt), "--cache-dir", str(cache),
                         "--out-dir", str(tmp_path / "out")] + U.SWEEP_CASES[case])
    assert rc == 0
    assert U.compare_trees(tmp_path / "out", U.CLI_GOLDEN / "sweep" / case) == []
    assert list(cache.iterdir()) == []


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(U.WQ_CASES))
def test_wq_fp8_checkpoint_equals_float32_cache(ckpt, tmp_path, case):
    """The block-scaled fp8 weight scored from its bytes == the same tensor as the reference's dequantized float32 cache."""
    cache = tmp_path / "hf-cache"
    _seed_layer1_cache(cache)
    rc_a, via_ckpt = _wq(tmp_path / "ckpt", case, "model.layers.1", ["--checkpoint-dir", str(ckpt)])
    rc_b, via_cache = _wq(tmp_path / "cache", case, "model.layers.1", ["--cache-dir", str(cache)])
    assert rc_a == rc_b == 0
    assert U.compare_trees(via_ckpt, via_cache) == [] and U.compare_trees(via_cache, via_ckpt) == []


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(U.SWEEP_CASES))
def test_sweep_fp8_checkpoint_equals_float32_cache(ckpt, tmp_path, case):
    from quantization_analysis_b200 import sweep_cli
    cache = tmp_path / "hf-cache"
    _seed_layer1_cache(cache)
    base = [U.REPO, L1, "--no-regex"] + U.SWEEP_CASES[case]
    rc_a = sweep_cli.main(base + ["--checkpoint-dir", str(ckpt), "--out-dir", str(tmp_path / "a")])
    rc_b = sweep_cli.main(base + ["--cache-dir", str(cache), "--out-dir", str(tmp_path / "b")])
    assert rc_a == rc_b
    if rc_a == 0:
        a, b = tmp_path / "a", tmp_path / "b"
        assert U.compare_trees(a, b) == [] and U.compare_trees(b, a) == []


@pytest.mark.gpu
def test_reconstruct_through_checkpoint(ckpt, tmp_path):
    """reconstruct --checkpoint-dir of the fp8 weight from the greedy run's map == reconstructing the reference's float32
    dequantization with the same map."""
    from quantization_analysis_b200 import reconstruct
    rc, got = _wq(tmp_path, "greedy", "model.layers.1", ["--checkpoint-dir", str(ckpt)])
    assert rc == 0
    d = got / "mixed_tile_greedy" / L1
    out = tmp_path / "recon.npy"
    assert reconstruct.main([L1, "--checkpoint-dir", str(ckpt), "--assignment", str(d / "assignment.npy"),
                             "--assignment-mapping", str(d / "assignment_mapping.json"), "--out", str(out)]) == 0
    _, _, ref = fp8_golden()
    a = np.load(d / "assignment.npy")
    want = reconstruct.reconstruct_from_assignment(ref, a, reconstruct.load_mapping(d / "assignment_mapping.json"))
    y = np.load(out)
    assert y.dtype == np.float32 and y.shape == ref.shape
    assert np.array_equal(G.bits(y), G.bits(want))


@pytest.mark.gpu
def test_fp8_prepared_tile_stats_take_the_fused_pass():
    """engine.tile_stats on an Fp8Prepared == engine.tile_stats_fp8 on its bytes, bit for bit, without materialising the
    float32 image."""
    from quantization_analysis_b200 import engine
    w, s, _ = fp8_golden()
    p = engine.prepare_loaded(Fp8Blocks(torch.from_numpy(w).view(torch.float8_e4m3fn), torch.from_numpy(s)))
    assert isinstance(p, engine.Fp8Prepared)
    for exact_abs in (True, False):
        got = engine.tile_stats(p, exact_abs=exact_abs)
        want, _ = engine.tile_stats_fp8(torch.from_numpy(w), torch.from_numpy(s), exact_abs=exact_abs)
        assert torch.equal(got.nan_to_num(nan=-1.0), want.nan_to_num(nan=-1.0)), exact_abs
    assert p._data is None
