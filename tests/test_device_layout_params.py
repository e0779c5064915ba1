"""CPU: the ``transpose`` parameter of the mixed-tile algorithms, the CLI flags that carry it, and the files that record it
(the mapping JSON's ``layout`` key, sweep_config.json)."""
import json

import numpy as np
import pytest

from quantization_analysis_b200 import engine, reconstruct, sweep, sweep_cli, wq
from quantization_analysis_b200.compression_algorithms import create_algorithm, load_compression_config

ALGOS = ["mixed-tile-greedy", "mixed-tile-threshold", "mixed-tile-random"]


@pytest.mark.parametrize("algo", ALGOS)
def test_transpose_param_defaults_false_and_takes_bools_only(algo):
    assert create_algorithm(algo, {}).transpose is False
    assert create_algorithm(algo, {"transpose": True}).transpose is True
    assert create_algorithm(algo, {"transpose": False}).transpose is False
    for bad in (1, 0, "true", "false", None, [True]):
        with pytest.raises(ValueError, match="transpose"):
            create_algorithm(algo, {"transpose": bad})


def test_config_file_carries_the_param(tmp_path):
    cfg = tmp_path / "c.json"
    cfg.write_text(json.dumps({"algorithm": "mixed-tile-greedy", "params": {"metric": "pcc", "transpose": True}}))
    c = load_compression_config(str(cfg))
    assert create_algorithm(c.algorithm, dict(c.params)).transpose is True


def test_three_dimensional_input_is_rejected_before_any_device_work():
    with pytest.raises(ValueError, match=r"\(2, 3, 4\)"):
        engine.prepare_transposed(np.zeros((2, 3, 4), np.float32))


def test_mapping_json_layout_key_only_when_transposed(tmp_path):
    a = np.zeros((3, 2), np.int8)
    wq.write_assignment(tmp_path, "algo", "t.weight", a)
    wq.write_assignment(tmp_path, "algo_t", "t.weight", a, transposed=True)
    plain = json.loads((tmp_path / "algo" / "t.weight" / "assignment_mapping.json").read_text())
    moved = json.loads((tmp_path / "algo_t" / "t.weight" / "assignment_mapping.json").read_text())
    assert "layout" not in plain and moved.pop("layout") == "transposed" and moved == plain
    # byte-identical to the file written before the layout existed
    assert (tmp_path / "algo" / "t.weight" / "assignment_mapping.json").read_text() == json.dumps(
        {"tile_hw": 32, "format_to_int": {"bf16": 0, "bfp8": 1, "bfp4": 2, "bfp2": 3},
         "int_to_format": ["bf16", "bfp8", "bfp4", "bfp2"], "assignment_shape": [3, 2]}, indent=2)
    assert reconstruct.load_layout(tmp_path / "algo" / "t.weight" / "assignment_mapping.json") is False
    assert reconstruct.load_layout(tmp_path / "algo_t" / "t.weight" / "assignment_mapping.json") is True
    bad = tmp_path / "bad.json"
    bad.write_text(json.dumps({**plain, "layout": "columns"}))
    with pytest.raises(ValueError, match="columns"):
        reconstruct.load_layout(bad)
    wq.write_random_outputs(tmp_path, "r.weight", [{"id": 0, "counts": {}, "total_bytes": 0.0, "pcc": 1.0, "mae": 0.0, "atol": 0.0}],
                            ["bfp8"], a, transposed=True)
    assert json.loads((tmp_path / "mixed_tile_random" / "r.weight_assignment_mapping.json").read_text())["layout"] == "transposed"


def test_sweep_config_records_transpose_only_when_set(tmp_path):
    args = ("repo", "t", "main", "emulation", ["bfp8", "bfp4"], "pcc", 0.9, 8)
    sweep.write_sweep_config(tmp_path / "a", *args)
    sweep.write_sweep_config(tmp_path / "b", *args, transpose=True)
    sweep.write_sweep_config(tmp_path / "c", *args, greedy={"algorithm": "mixed-tile-greedy", "seed": 3, "highest_metric_val": 0.99},
                             transpose=True)
    a = json.loads((tmp_path / "a" / "sweep_config.json").read_text())
    b = json.loads((tmp_path / "b" / "sweep_config.json").read_text())
    c = json.loads((tmp_path / "c" / "sweep_config.json").read_text())
    assert "transpose" not in a and b.pop("transpose") is True and a == b
    assert list(c)[-1] == "transpose" and c["seed"] == 3


def test_sweep_cli_flag_reaches_the_job():
    ap = sweep_cli.build_parser()
    assert ap.parse_args(["r", "t"]).transpose is False
    assert ap.parse_args(["r", "t", "--transpose"]).transpose is True
    assert sweep_cli.SweepJob(None, None, "r", "main", "emulation", ["bfp8"], "pcc", 0.9, 4).transpose is False
