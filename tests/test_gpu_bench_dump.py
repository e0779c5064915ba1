"""GPU: bench.py --dump-outputs writes what the timed path computed in its last step.  For the default workload the maps and
counts are the reference's (tests/golden/cfg2_bench_workload.*) and pcc / mae / atol are the fp64 evaluation of the
reference formulas; for the other configs the files are complete, float32 / float64, within 64 MB and self-consistent."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import qa_oracle as orc
from tests import golden_util as G

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def _bench(out_dir: Path, *args) -> dict:
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
                         + list(args), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    files = list(out_dir.iterdir())
    assert files and sum(f.stat().st_size for f in files) <= 64 << 20
    assert all(f.suffix == ".npy" and np.load(f).dtype in (np.float32, np.float64) for f in files)
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs_are_reference_maps(tmp_path):
    from quantization_analysis_b200 import synthetic
    d = tmp_path / "dump"
    line = _bench(d, "--steps", "2", "--warmup", "1")
    assert line["steps"] == 2 and line["result_check"]["maps_equal_reference"] is True
    meta, maps = G.js("cfg2_bench_workload.json"), G.npz("cfg2_bench_workload.npz")
    assert sorted(p.name for p in d.iterdir()) == sorted(f"{n}.{a}.npy" for n in synthetic.ATTN_NAMES for a in ("assignment", "counts", "metrics"))
    for name in synthetic.ATTN_NAMES:
        key = name.split(".")[-2]
        a = np.load(d / f"{name}.assignment.npy")
        assert a.dtype == np.float32 and np.array_equal(a, maps[key].astype(np.float32)), key
        c = np.load(d / f"{name}.counts.npy")
        assert c.dtype == np.float64 and c.tolist() == [meta[key]["counts"][f] for f in G.MIXED], key
        m = np.load(d / f"{name}.metrics.npy")
        assert m.dtype == np.float64 and m.shape == (3,) and m[0] >= 0.999, key
        if key in ("kv_a_proj_with_mqa", "q_a_proj"):          # the two smallest tensors: fp64 metrics of the oracle's y
            x = synthetic.randn_bf16_cpu(tuple(meta[key]["shape"]), meta[key]["seed"]).float().numpy()
            want = orc.exact_metrics_f64(x, orc.apply_assignment(x, maps[key]))
            assert m.tolist() == pytest.approx([want["pcc"], want["mae"], want["atol"]], rel=1e-6, abs=0), key


def _bincount(a: np.ndarray) -> list:
    return np.bincount(a.astype(np.int64).reshape(-1), minlength=4).astype(np.float64).tolist()


@pytest.mark.parametrize("config", ["cfg1", "cfg3", "cfg4", "cfg5", "cfg2-fp8"])
def test_bench_dump_outputs_other_configs(tmp_path, config):
    d = tmp_path / "dump"
    line = _bench(d, "--config", config, "--steps", "1", "--warmup", "1")
    arrays = {p.name[:-4]: np.load(p) for p in d.iterdir()}
    stems = {k.rsplit(".", 1)[0] for k in arrays}
    if config == "cfg1":                          # steps come in rounds of 8 buffers: the last step is buffer 7's
        import torch
        from quantization_analysis_b200 import synthetic
        j = (line["steps"] - 1) % 8
        assert sorted(arrays) == [f"buffer{j}.{f}.sample" for f in ("bfp2", "bfp4", "bfp8")]
        x = synthetic.device_randn_bf16((1536, 7168), 100 + j, "cuda").float().cpu().numpy()
        idx = np.sort(np.random.default_rng(0).choice(x.size, 1 << 21, replace=False))      # the documented fixed sample
        for fmt in ("bfp8", "bfp4", "bfp2"):
            want = torch.from_numpy(orc.quantize(x, fmt).reshape(-1)[idx]).to(torch.bfloat16).float().numpy()
            assert np.array_equal(arrays[f"buffer{j}.{fmt}.sample"], want), fmt
        return
    assert line["steps"] == 1
    if config == "cfg2-fp8":
        assert line["result_check"]["maps_equal_reference_order_run_on_dequantized_float32"] is True
    if config == "cfg4":                          # the selected map is one of the 1000 maps of NumPy's stream for seed 42
        s = "model.layers.0.self_attn.kv_a_proj_with_mqa.weight"
        a = arrays[f"{s}.assignment"]
        choices = np.random.default_rng(42).integers(0, 4, size=(1000, a.size), dtype=np.int64)
        hit = np.where((choices == a.astype(np.int64)).all(axis=1))[0]
        assert hit.size and (arrays[f"{s}.samples"][hit] == arrays[f"{s}.metrics"]).all(axis=1).any()
    for s in stems:
        if config == "cfg3":
            rows, maps = arrays[f"{s}.rows"], arrays[f"{s}.maps_sample"]
            assert rows.shape == (32, 9) and maps.shape[0] == 32 and set(np.unique(maps)) <= {0.0, 1.0, 2.0, 3.0}
            assert len(set(rows[:, 1:5].sum(axis=1))) == 1                    # every threshold assigns every tile
            assert (np.diff(rows[:, 5]) <= 0).all()                          # a lower threshold never costs more bytes
            continue
        a, c, m = arrays[f"{s}.assignment"], arrays[f"{s}.counts"], arrays[f"{s}.metrics"]
        assert c.tolist() == _bincount(a) and m.shape == (3,)
        if config == "cfg4":
            assert arrays[f"{s}.samples"].shape == (1000, 3) and (arrays[f"{s}.samples"] == m).all(axis=1).any()
        else:
            assert m[0] >= 0.999
    if config == "cfg5":
        assert len(stems) == 768
