"""`wq --gpus N` and `sweep_cli --gpus N`: the matched tensors split over the GPUs of a node (multi_gpu.run_sharded).

Results do not depend on which GPU scores which tensor, so a sharded run must write the tree a one-process run writes, up
to TIME(s).  Host tests cover the header-only tensor sizes the split uses, the order-restoring merge and the flag checks;
device tests compare sharded runs with the committed goldens and with in-process runs, over the tiny float32-cache
'repository' of tests/cli_util.py and the two-shard checkpoint of tests/test_checkpoint_source.py.  The two-GPU cases run
when two devices are visible and are skipped otherwise.
"""
import json
import multiprocessing
import random
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from safetensors.torch import save_file

from quantization_analysis_b200 import multi_gpu, sweep_cli, tensor_source, wq
from tests import cli_util as U
from tests.test_checkpoint_source import L1, write_checkpoint


def _gpus(n: int) -> int:
    if n > torch.cuda.device_count():
        pytest.skip(f"needs {n} visible GPUs")
    return n


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    return write_checkpoint(tmp_path_factory.mktemp("ckpt") / "tiny-r1")


@pytest.fixture(scope="module")
def cache(tmp_path_factory):
    c = tmp_path_factory.mktemp("hf") / "hf-cache"
    U.seed_fp32_cache(c)
    return c


# ------------------------------------------------------------------------------------------------------------------------
# host
# ------------------------------------------------------------------------------------------------------------------------
def test_shape_from_checkpoint_headers(ckpt):
    """Every tensor of the two-shard checkpoint, the fp8 weight (loaded as Fp8Blocks) and its scale grid included."""
    index = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=ckpt)
    assert L1 in index.tensor_to_file and f"{L1}_scale_inv" in index.tensor_to_file
    for name in index.tensor_to_file:
        assert index.shape(name) == tuple(index.load(name).shape), name
    assert index.shape(L1) == (300, 520) and index.shape(f"{L1}_scale_inv") == (3, 5)


def test_shape_from_float32_cache_headers(cache):
    index = tensor_source.build_tensor_index(U.REPO, cache_dir=cache)
    assert sorted(index.tensor_to_file) == sorted(U.tensors())
    for name in index.tensor_to_file:
        assert index.shape(name) == tuple(index.load(name).shape) == U.tensors()[name].shape, name


def test_shape_of_synthetic_tensors():
    index = tensor_source.build_tensor_index("synthetic")
    for name in index.tensor_to_file:
        assert index.shape(name) == tuple(index.load(name).shape), name


NAMES = [f"model.layers.{i}.mlp.down_proj.weight" for i in range(7)]


def _when_complete(arrival: list[str]) -> list[int]:
    """For each name in NAMES order: how many messages had arrived when it and every earlier name had."""
    seen, out = set(), []
    for k, name in enumerate(arrival, 1):
        seen.add(name)
        while len(out) < len(NAMES) and NAMES[len(out)] in seen:
            out.append(k)
    return out


def test_merge_restores_name_order_as_prefixes_complete():
    rng = random.Random(3)
    orders = [NAMES, NAMES[::-1]] + [rng.sample(NAMES, len(NAMES)) for _ in range(30)]
    for arrival in orders:
        consumed = []

        def messages():
            for name in arrival:
                consumed.append(name)
                yield name, None, ("result of", name)
        got, when = [], []
        for name, result in multi_gpu.merge_in_order(NAMES, messages()):
            got.append((name, result))
            when.append(len(consumed))
        assert got == [(n, ("result of", n)) for n in NAMES], arrival
        assert when == _when_complete(arrival), arrival          # yielded as soon as the prefix is complete, not later


def test_merge_reports_a_failure_in_any_position_with_its_name():
    rng = random.Random(4)
    for failing in NAMES:
        for _ in range(4):
            arrival = rng.sample(NAMES, len(NAMES))
            msgs = [(n, "ValueError on cuda:1: stored as I32" if n == failing else None, n) for n in arrival]
            with pytest.raises(multi_gpu.ShardError, match=re.escape(failing) + ": ValueError on cuda:1: stored as I32"):
                list(multi_gpu.merge_in_order(NAMES, msgs))


def test_wq_rejects_zero_gpus(capsys):
    assert wq.run([U.REPO, U.FILTER, "--gpus", "0"]) == 1
    err = capsys.readouterr().err
    assert "--gpus 0" in err and f"which is {torch.cuda.device_count()}" in err
    assert multiprocessing.active_children() == []


@pytest.mark.parametrize("cli", ["wq", "sweep_cli"])
def test_more_gpus_than_visible_are_rejected(capsys, tmp_path, cli):
    """Without CUDA (0 visible devices) --gpus 2 fails before any worker starts; on a GPU node, one more than visible."""
    visible = torch.cuda.device_count()
    n = max(2, visible + 1)
    if cli == "wq":
        rc = wq.run([U.REPO, U.FILTER, "--results-root", str(tmp_path / "results"), "--gpus", str(n)])
    else:
        rc = sweep_cli.main([U.REPO, U.SWEEP_TENSOR, "--out-dir", str(tmp_path / "out"), "--gpus", str(n)])
    assert rc == 1
    err = capsys.readouterr().err
    assert len(err.strip().splitlines()) == 1 and f"--gpus {n}" in err and f"which is {visible}" in err
    assert multiprocessing.active_children() == []
    assert list(tmp_path.iterdir()) == []


# ------------------------------------------------------------------------------------------------------------------------
# device
# ------------------------------------------------------------------------------------------------------------------------
def _run_wq(root: Path, cfg: dict, filt: str, source: list[str], gpus: int | None, capsys) -> tuple[int, str, str, Path | None]:
    root.mkdir(parents=True, exist_ok=True)
    p = root.parent / "config.json"                   # one path for the runs a test compares: stdout prints it
    p.write_text(json.dumps(cfg))
    argv = [U.REPO, filt, "--compression-config", str(p), "--recompute", "--summary", "--results-root", str(root / "results"),
            "--processed-root", str(root / "processed")] + source
    capsys.readouterr()
    rc = wq.run(argv + ([] if gpus is None else ["--gpus", str(gpus)]))
    out = capsys.readouterr()
    base = root / "results" / U.REPO.replace("/", "__") / cfg["algorithm"]
    tree = sorted(base.iterdir())[-1] if base.is_dir() else None
    return rc, out.out, out.err, tree


def _same_trees(a: Path, b: Path) -> bool:
    return U.compare_trees(a, b) == [] and U.compare_trees(b, a) == []


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [1, 2])
@pytest.mark.parametrize("case", sorted(U.WQ_CASES))
def test_wq_sharded_matches_reference_output_tree(cache, tmp_path, capsys, case, gpus):
    """The golden tree of every WQ_CASES case; stdout equals the in-process run's (tensor blocks in the same order) but for
    TIME(s)."""
    gpus = _gpus(gpus)
    source = ["--cache-dir", str(cache)]
    rc_a, out_a, _, _ = _run_wq(tmp_path / "a", U.WQ_CASES[case], U.FILTER, source, None, capsys)
    rc_b, out_b, err_b, sharded = _run_wq(tmp_path / "b", U.WQ_CASES[case], U.FILTER, source, gpus, capsys)
    assert rc_a == 0 and rc_b == 0, err_b
    assert U.compare_trees(sharded, U.CLI_GOLDEN / "wq" / case) == []
    assert U.strip_times(out_b) == U.strip_times(out_a)
    assert [ln for ln in out_b.splitlines() if ln in U.tensors()] == sorted(U.tensors())
    assert multiprocessing.active_children() == []


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(U.WQ_CASES))
def test_wq_sharded_checkpoint_equals_in_process(ckpt, tmp_path, capsys, case):
    """--checkpoint-dir over model.layers (BF16, F32 and the block-scaled fp8 weight) on two GPUs (one on a one-GPU node)."""
    gpus = min(2, torch.cuda.device_count())
    source = ["--checkpoint-dir", str(ckpt)]
    rc_a, out_a, _, inproc = _run_wq(tmp_path / "a", U.WQ_CASES[case], "model.layers", source, None, capsys)
    rc_b, out_b, err_b, sharded = _run_wq(tmp_path / "b", U.WQ_CASES[case], "model.layers", source, gpus, capsys)
    assert rc_a == 0 and rc_b == 0, err_b
    assert L1 in out_b and "model.layers.0.self_attn.q_a_proj.weight" in out_b
    assert _same_trees(sharded, inproc)
    assert U.strip_times(out_b) == U.strip_times(out_a)


@pytest.mark.gpu
@pytest.mark.parametrize("algorithm", ["mixed-tile-greedy", "mixed-tile-random"])
def test_seed_is_resolved_once_for_every_gpu(ckpt, tmp_path, capsys, algorithm):
    """"seed": 0 draws one seed in the parent: every tensor on every GPU uses the one recorded in
    compression_config.used.json, so the maps equal an in-process run given that seed."""
    gpus = min(2, torch.cuda.device_count())
    params = {"metric": "pcc", "threshold": 0.999} if algorithm == "mixed-tile-greedy" else {"metric": "pcc", "threshold": 0.99, "iters": 4}
    cfg = {"algorithm": algorithm, "quantization_formats": U.FORMATS5, "params": params, "seed": 0}
    source = ["--checkpoint-dir", str(ckpt)]
    rc, _, err, sharded = _run_wq(tmp_path / "sharded", cfg, "model.layers", source, gpus, capsys)
    assert rc == 0, err
    used = json.loads((sharded / "compression_config.used.json").read_text())
    assert used["seed_source"] == "random" and used["seed"] > 0
    rc, _, _, inproc = _run_wq(tmp_path / "inproc", dict(cfg, seed=used["seed"]), "model.layers", source, None, capsys)
    assert rc == 0
    sub = algorithm.replace("-", "_")
    assert len(list((sharded / sub).rglob("*.npy"))) == 5
    assert _same_trees(sharded / sub, inproc / sub)
    assert U.strip_times((sharded / "table.txt").read_text()) == U.strip_times((inproc / "table.txt").read_text())


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [1, 2])
def test_sweep_sharded_equals_in_process(ckpt, tmp_path, gpus):
    """The regex matches the four 2-D weights of the checkpoint: BF16, F32 and the block-scaled fp8 one."""
    gpus = _gpus(gpus)
    base = [U.REPO, "proj", "--checkpoint-dir", str(ckpt)] + U.SWEEP_CASES["pcc"]
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "a")]) == 0
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "b"), "--gpus", str(gpus)]) == 0
    details = sorted(p.name for p in (tmp_path / "b" / "details").iterdir())
    assert len(details) == 4 and L1.replace(".", "_") in details
    assert _same_trees(tmp_path / "b", tmp_path / "a")
    assert multiprocessing.active_children() == []


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [1, 2])
@pytest.mark.parametrize("case", sorted(U.SWEEP_CASES))
def test_sweep_sharded_matches_reference_csv(cache, tmp_path, case, gpus):
    gpus = _gpus(gpus)
    out = tmp_path / "out"
    rc = sweep_cli.main([U.REPO, U.SWEEP_TENSOR, "--no-regex", "--cache-dir", str(cache), "--out-dir", str(out), "--gpus", str(gpus)]
                        + U.SWEEP_CASES[case])
    assert rc == 0
    assert U.compare_trees(out, U.CLI_GOLDEN / "sweep" / case) == []


@pytest.mark.gpu
def test_sweep_sharded_range_error_like_in_process(ckpt, tmp_path, capsys):
    """A lowest pcc above every tensor's start metric: the sharded run prints the in-process run's one error line and
    returns 1."""
    gpus = min(2, torch.cuda.device_count())
    base = [U.REPO, "proj", "--checkpoint-dir", str(ckpt), "--metric", "pcc", "--lowest-metric-val", "1.5"]
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "a")]) == 1
    want = capsys.readouterr().out
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "b"), "--gpus", str(gpus)]) == 1
    assert capsys.readouterr().out == want == "error: lowest-metric-val must be <= start metric for pcc\n"
    assert multiprocessing.active_children() == []


@pytest.mark.gpu
def test_worker_exception_names_the_tensor_and_leaves_no_process(tmp_path, capsys):
    """An integer tensor among the matched ones: TensorIndex.load raises ValueError in a worker before any device work."""
    d = write_checkpoint(tmp_path / "c", with_index=False)
    bad = "model.layers.0.mlp.gate.weight"
    save_file({bad: torch.zeros((64, 64), dtype=torch.int32)}, str(d / "extra.safetensors"), metadata={"format": "pt"})
    gpus = min(2, torch.cuda.device_count())
    rc, out, err, _ = _run_wq(tmp_path / "run", U.WQ_CASES["greedy"], "model.layers.0", ["--checkpoint-dir", str(d)], gpus, capsys)
    assert rc == 1
    assert f"error: {bad}: ValueError on cuda:" in err and "stored as I32" in err
    assert multiprocessing.active_children() == []


_PARENT_NO_CUDA = r'''
import sys
sys.path.insert(0, sys.argv[1])
import torch
from quantization_analysis_b200 import wq
rc = wq.run(sys.argv[2:])
print("parent_cuda_initialized", torch.cuda.is_initialized())
sys.exit(rc)
'''


@pytest.mark.gpu
def test_parent_does_no_cuda_work(cache, tmp_path):
    """The parent of a sharded run never initialises CUDA, so it holds no memory on GPU 0."""
    cfg = tmp_path / "greedy.json"
    cfg.write_text(json.dumps(U.WQ_CASES["greedy"]))
    argv = [U.REPO, U.FILTER, "--compression-config", str(cfg), "--recompute", "--summary", "--cache-dir", str(cache),
            "--results-root", str(tmp_path / "r"), "--processed-root", str(tmp_path / "p"), "--gpus", "1"]
    out = subprocess.run([sys.executable, "-c", _PARENT_NO_CUDA, str(U.ROOT)] + argv, capture_output=True, text=True, timeout=600,
                         cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "parent_cuda_initialized False" in out.stdout
    got = U.latest_results_dir(tmp_path / "r", "mixed-tile-greedy")
    assert U.compare_trees(got, U.CLI_GOLDEN / "wq" / "greedy") == []
    assert np.load(got / "mixed_tile_greedy" / "model.layers.0.mlp.down_proj.weight" / "assignment.npy").dtype == np.int8
