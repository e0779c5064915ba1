"""The device layout through the programs: wq with ``"transpose": true``, ``sweep_cli --transpose`` and reconstruct of a
transposed map, over a small safetensors checkpoint (bf16, float32 and block-scaled fp8 tensors, a 1-D vector).

The expected files come from the same programs without the flag over a second checkpoint that stores every 2-D tensor
transposed (an fp8 weight with its scale grid transposed too): the maps, the sweep CSVs and the sweep configs must agree;
wq's MIXED rows score x against y in the stored layout, so they are checked against the oracle instead."""
import json
import re
from pathlib import Path

import numpy as np
import pytest
import torch
from safetensors.torch import save_file

from oracle import qa_oracle as orc
from quantization_analysis_b200 import reconstruct, sweep_cli, tensor_source, wq
from tests import cli_util as U
from tests import golden_util as G
from tests.test_checkpoint_source import L1, shard_contents

CONFIG = {"algorithm": "mixed-tile-greedy", "quantization_formats": U.FORMATS5,
          "params": {"metric": "pcc", "threshold": 0.999, "transpose": True}, "seed": 123}
MATRICES = ["model.layers.0.self_attn.kv_a_proj_with_mqa.weight", "model.layers.0.mlp.down_proj.weight", U.SWEEP_TENSOR, L1]
VECTOR = "model.layers.0.input_layernorm.weight"


def _write(d: Path, transposed: bool) -> Path:
    d.mkdir(parents=True, exist_ok=True)
    for i, (_shard, tensors) in enumerate(shard_contents().items()):
        out = {}
        for n, t in tensors.items():
            if transposed and t.dim() == 2:
                t = t.view(torch.uint8).t().contiguous().view(t.dtype) if t.dtype == torch.float8_e4m3fn else t.t().contiguous()
            out[n] = t
        save_file(out, str(d / f"model-{i:05d}.safetensors"), metadata={"format": "pt"})
    return d


@pytest.fixture(scope="module")
def ckpts(tmp_path_factory):
    root = tmp_path_factory.mktemp("layout")
    return _write(root / "stored", False), _write(root / "transposed", True)


def _wq(root: Path, ckpt: Path, cfg: dict, extra=()) -> Path:
    root.mkdir(parents=True, exist_ok=True)
    (root / "cfg.json").write_text(json.dumps(cfg))
    rc = wq.run([U.REPO, "model.layers", "--compression-config", str(root / "cfg.json"), "--checkpoint-dir", str(ckpt),
                 "--results-root", str(root / "results"), "--processed-root", str(root / "processed"), "--no-save-processed",
                 *extra])
    assert rc == 0
    return U.latest_results_dir(root / "results", cfg["algorithm"])


def _x(ckpt: Path, name: str) -> np.ndarray:
    x = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=ckpt).load(name)
    if isinstance(x, tensor_source.Fp8Blocks):
        return orc.fp8_block_dequant(x.weight.view(torch.uint8).numpy(), x.scale_inv.numpy())
    return x.float().numpy() if isinstance(x, torch.Tensor) else np.asarray(x, dtype=np.float32)


def _mixed_row(table: str, name: str) -> list[str]:
    block = table.split(name + "\n", 1)[1]
    line = next(ln for ln in block.splitlines() if "mixed-tile-greedy" in ln and "MIXED" in ln)
    return line.split()


@pytest.mark.gpu
def test_wq_transposed_maps_rows_and_reconstruct(ckpts, tmp_path):
    stored, transposed = ckpts
    got = _wq(tmp_path / "a", stored, CONFIG)
    unflagged = {**CONFIG, "params": {k: v for k, v in CONFIG["params"].items() if k != "transpose"}}
    ref = _wq(tmp_path / "b", transposed, unflagged)
    used = json.loads((got / "compression_config.used.json").read_text())
    assert used["params"]["transpose"] is True
    table = (got / "table.txt").read_text()
    for name in MATRICES:
        d, dr = got / "mixed_tile_greedy" / name, ref / "mixed_tile_greedy" / name
        a = np.load(d / "assignment.npy")
        x = _x(stored, name)
        assert a.shape == (-(-x.shape[1] // 32), -(-x.shape[0] // 32))
        assert np.array_equal(a, np.load(dr / "assignment.npy")), name
        mapping = json.loads((d / "assignment_mapping.json").read_text())
        assert mapping.pop("layout") == "transposed" and mapping == json.loads((dr / "assignment_mapping.json").read_text())
        # the MIXED row: float32 scores of x against y in the stored layout
        xt = np.ascontiguousarray(x.T)
        y = orc.apply_assignment(xt, a).T
        s = orc.wq_scores(x, y)
        row = _mixed_row(table, name)
        assert row[2:5] == [f"{s['pcc']: .5f}".strip(), f"{s['mae']:.3e}", f"{s['atol']:.3e}"], (name, row, s)
        # reconstruct reads the layout from the mapping and writes y in x's shape
        out = tmp_path / f"{name}.npy"
        assert reconstruct.main([name, "--checkpoint-dir", str(stored), "--assignment", str(d / "assignment.npy"),
                                 "--assignment-mapping", str(d / "assignment_mapping.json"), "--out", str(out)]) == 0
        r = np.load(out)
        assert r.shape == x.shape and np.array_equal(G.bits(r), G.bits(y)), name
        # --no-transpose overrides the mapping: the map no longer fits x's own tile grid (unless that is square)
        if a.shape != (-(-x.shape[0] // 32), -(-x.shape[1] // 32)):
            with pytest.raises(ValueError, match="does not match"):
                reconstruct.main([name, "--checkpoint-dir", str(stored), "--assignment", str(d / "assignment.npy"),
                                  "--assignment-mapping", str(d / "assignment_mapping.json"), "--out", str(out), "--no-transpose"])
    # the 1-D tensor is its own transpose: an ordinary map without the layout key
    mv = json.loads((got / "mixed_tile_greedy" / VECTOR / "assignment_mapping.json").read_text())
    assert "layout" not in mv
    assert np.array_equal(np.load(got / "mixed_tile_greedy" / VECTOR / "assignment.npy"),
                          np.load(ref / "mixed_tile_greedy" / VECTOR / "assignment.npy"))


@pytest.mark.gpu
def test_wq_transposed_rows_equal_oracle_exactly(ckpts):
    """evaluate_tensor's MIXED row, unrounded: the oracle's float32 wq scores of x against yt.T."""
    stored, _ = ckpts
    alg = wq.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 77, "transpose": True})
    index = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=stored)
    for name in MATRICES:
        rows, _meta = wq.evaluate_tensor(name, index.load(name), [wq.create_algorithm("none", {}), alg], U.FORMATS5, None, None)
        r = rows["mixed-tile-greedy"][0]
        x = _x(stored, name)
        xt = np.ascontiguousarray(x.T)
        a, counts = orc.greedy_assign(orc.tile_stat_table(xt), G.MIXED, "pcc", 0.999, 77)
        s = orc.wq_scores(x, orc.apply_assignment(xt, a).T)
        assert (np.float32(r.pcc), np.float32(r.mae), np.float32(r.atol)) == (np.float32(s["pcc"]), np.float32(s["mae"]),
                                                                               np.float32(s["atol"])), name
        assert r.tile_counts == counts and r.tile_bytes == orc.total_bytes(counts)


@pytest.mark.gpu
def test_wq_transposed_two_gpus_same_tree(ckpts, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    stored, _ = ckpts
    one = _wq(tmp_path / "one", stored, CONFIG)
    two = _wq(tmp_path / "two", stored, CONFIG, ["--gpus", "2"])
    assert U.compare_trees(two, one) == [] and U.compare_trees(one, two) == []


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["mixed-tile-threshold", "mixed-tile-greedy"])
@pytest.mark.parametrize("name", [U.SWEEP_TENSOR, L1])
def test_sweep_cli_transpose_equals_unflagged_sweep_of_the_transposed_checkpoint(ckpts, tmp_path, algo, name):
    stored, transposed = ckpts
    args = [U.REPO, name, "--no-regex", "--algorithm", algo, "--metric", "pcc", "--lowest-metric-val", "0.95", "--steps", "6",
            "--formats", "bfp8,bfp4,bfp2"] + (["--seed", "31"] if algo == "mixed-tile-greedy" else [])
    assert sweep_cli.main(args + ["--checkpoint-dir", str(stored), "--out-dir", str(tmp_path / "a"), "--transpose"]) == 0
    assert sweep_cli.main(args + ["--checkpoint-dir", str(transposed), "--out-dir", str(tmp_path / "b")]) == 0
    sub = Path("details") / re.sub(r"[/.]", "_", name)
    a, b = tmp_path / "a" / sub, tmp_path / "b" / sub
    assert (a / "sweep_results.csv").read_text() == (b / "sweep_results.csv").read_text()
    ca, cb = json.loads((a / "sweep_config.json").read_text()), json.loads((b / "sweep_config.json").read_text())
    assert ca.pop("transpose") is True and "transpose" not in cb and ca == cb
