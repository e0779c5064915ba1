"""The greedy sweep: every threshold's mixed-tile-greedy chain over one tile-stat table, one init and one set of permutations,
all chains in one launch (qa_greedy_assign_sweep, engine.greedy_sweep, sweep.greedy_sweep_tensor, sweep_cli --algorithm
mixed-tile-greedy).

Each row must be what a single-threshold run gives: the CPU oracle's map and counts, and MixedTileGreedyCompression's map,
counts, state, certificate and metrics.  Host tests cover the C entry point's argument checks and the CLI flag checks.
"""
import json

import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc
from quantization_analysis_b200 import _lib, engine, sweep, sweep_cli, synthetic, tensor_source
from quantization_analysis_b200.compression_algorithms.mixed_tile_greedy import MixedTileGreedyCompression
from tests import cli_util as U
from tests import golden_util as G
from tests.test_checkpoint_source import L1, fp8_golden, write_checkpoint

FORMAT_LISTS = [list(G.MIXED), ["bfp8", "bfp4", "bfp2"], ["bfp4", "bfp2"], ["bfp8"]]
# per metric: the first threshold accepts nothing (not even the base format passes), the last accepts every candidate
THRESHOLDS = {"pcc": [1.5, 0.99999, 0.9995, 0.995, 0.95, -2.0],
              "mae": [-1.0, 1e-5, 1e-4, 1e-3, 1e-2, 1e9],
              "atol": [-1.0, 1e-4, 1e-3, 1e-2, 0.1, 1e9]}
# state entries that do not count SM cycles: sums, flags + speculation rounds, value, max |x - y|, cluster size, chunks, margin
STATE_DET = [0, 1, 2, 3, 4, 5, 6, 7, 11, 12, 19, 20]


def _f32_not_bf16_exact(shape, seed):
    x = (np.random.default_rng(seed).standard_normal(shape) * 0.02).astype(np.float32)
    assert not np.array_equal(x, orc.bf16_round(x))
    return x


def _case(name):
    """-> (what greedy_sweep_tensor is given, the float32 array the reference would see)."""
    if name == "fp8":
        w, s, deq = fp8_golden()
        return tensor_source.Fp8Blocks(torch.from_numpy(w).view(torch.float8_e4m3fn), torch.from_numpy(s)), deq
    kind, src = name.split(":")
    if src.startswith("f32_"):
        shape = {"f32_1d": (1000,), "f32_3d": (2, 40, 64), "f32_96x160": (96, 160)}[src]
        x = _f32_not_bf16_exact(shape, 5)
    else:
        x = G.algo_input(src)
    return (torch.from_numpy(x).to(torch.bfloat16) if kind == "bf16" else x), x


CASES = ["bf16:het_256x512", "np:het_70x45", "np:zero_and_const_tiles", "bf16:het_1d_1000", "bf16:het_3d_2x40x64",
         "np:f32_1d", "np:f32_3d", "np:f32_96x160", "fp8"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_sweep_rows_equal_oracle(case):
    """Golden inputs, a ragged 1-D and a 3-D tensor, as bf16, float32 that is not bf16-exact and fp8 + block scales; every
    metric and format lists of 4, 3, 2 and 1 formats: each row is orc.greedy_assign at its threshold."""
    x, xf = _case(case)
    table = orc.tile_stat_table(xf)
    for metric, thr in THRESHOLDS.items():
        for fmts in FORMAT_LISTS:
            rows, maps = sweep.greedy_sweep_tensor(x, fmts, metric, thresholds=thr, seed=11)
            assert [r["threshold"] for r in rows] == thr
            for r, m, t in zip(rows, maps.cpu().numpy(), thr):
                want, counts = orc.greedy_assign(table, fmts, metric, t, 11)
                assert np.array_equal(m, want.reshape(-1)), (case, metric, fmts, t)
                assert r["counts"] == counts, (case, metric, fmts, t)
            # nothing accepted: every tile keeps the base format; everything accepted: every tile takes the last one
            assert rows[0]["counts"][fmts[0]] == maps.shape[1] and rows[-1]["counts"][fmts[-1]] == maps.shape[1]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["np:het_256x512", "np:f32_1d", "fp8"])
def test_sweep_rows_equal_single_runs(case):
    """Row k == MixedTileGreedyCompression(threshold k).run_prepared: map, counts, state, certificate, the reference's float32
    metrics, and with scoring="exact" the float64 recombination (metrics_exact)."""
    x, _ = _case(case)
    p = engine.prepare_loaded(x)
    for metric in ("pcc", "mae", "atol"):
        thr = THRESHOLDS[metric][1:-1]
        for fmts in (list(G.MIXED), ["bfp8", "bfp4"]):
            rows, maps = sweep.greedy_sweep_tensor(p, fmts, metric, thresholds=thr, seed=21)
            rows_x, maps_x = sweep.greedy_sweep_tensor(p, fmts, metric, thresholds=thr, seed=21, scoring="exact")
            assert torch.equal(maps, maps_x)
            for r, rx, m, t in zip(rows, rows_x, maps, thr):
                dr = MixedTileGreedyCompression({"metric": metric, "threshold": t, "seed": 21}).run_prepared(p, fmts)
                tag = (case, metric, fmts, t)
                assert torch.equal(m, dr.assignment) and r["counts"] == dr.counts and r["total_bytes"] == dr.tile_bytes, tag
                cert = dr.meta["certificate"]
                assert r["min_margin"] == cert["min_margin"] and r["fallback"] == cert["fallback"], tag
                want = dr.meta["state"].cpu().numpy()
                idx = STATE_DET if metric != "atol" and not cert["fallback"] else list(range(24))
                assert np.array_equal(r["state"][idx], want[idx]), tag
                assert {k: r[k] for k in ("pcc", "mae", "atol")} == dr.metrics, tag
                assert {k: rx[k] for k in ("pcc", "mae", "atol")} == dr.metrics_exact, tag


@pytest.mark.gpu
def test_shared_inputs_are_read_only():
    """The table, init, prefetched permutations and starting stream state are byte-equal before and after a sweep of 64
    thresholds; computing init inside the call (init=None) gives the same rows."""
    x = G.algo_input("het_256x512")
    p = engine.prepare_tiles(x)
    fmts = list(G.MIXED)
    table = engine.tile_stats(p, engine.MIXED_FORMATS, exact_abs=False)
    init = engine.greedy_init(table, "pcc", fmts)
    rng = engine.make_rng(9)
    pre = engine.greedy_prefetch(rng, table.shape[1], len(fmts))
    before = [t.clone() for t in (table, init, pre[0], pre[1], rng)]
    thr = np.linspace(0.99999, 0.9, 64)
    maps, counts, states = engine.greedy_sweep(table, p.numel, "pcc", thr, fmts, rng, pre, init)
    torch.cuda.synchronize()
    for a, b in zip(before, (table, init, pre[0], pre[1], rng)):
        assert torch.equal(a.view(torch.uint8) if a.dtype != torch.uint8 else a, b.view(torch.uint8) if b.dtype != torch.uint8 else b)
    maps2, counts2, states2 = engine.greedy_sweep(table, p.numel, "pcc", thr, fmts, rng, pre, None)
    assert torch.equal(maps, maps2) and torch.equal(counts, counts2) and torch.equal(states[:, :8], states2[:, :8])
    assert len({bytes(m.cpu().numpy()) for m in maps}) > 4         # the thresholds span several distinct maps


@pytest.mark.gpu
def test_cluster_caps_residency_and_permutation_cache():
    """A 65 536-tile tensor (the automatic cluster size is 16): caps 1, 2, 4, 8 and 16 give the same rows; a sweep of 300
    thresholds at cap 16 (more clusters than fit on the GPU at once) equals single runs; with and without prefetched
    permutations the rows are the same."""
    L = _lib.lib()
    x = synthetic.randn_bf16_cpu((2048, 32768), 17).cuda()
    p = engine.prepare_tiles(x)
    fmts = list(G.MIXED)
    table = engine.tile_stats(p, engine.MIXED_FORMATS, exact_abs=False)
    assert table.shape[1] == 65536
    init = engine.greedy_init(table, "pcc", fmts)
    rng = engine.make_rng(123)
    pre = engine.greedy_prefetch(rng, table.shape[1], len(fmts))
    thr = np.linspace(0.99999, 0.999, 8)
    cols = [0, 1, 2, 3, 4, 5, 7, 11]           # the speculation rounds and margins depend on the cluster size, the results do not
    ref = None
    for cap in (16, 1, 2, 4, 8):
        prev = L.qa_greedy_cluster_cap(cap)
        try:
            maps, counts, states = engine.greedy_sweep(table, p.numel, "pcc", thr, fmts, rng, pre, init)
        finally:
            L.qa_greedy_cluster_cap(prev)
        assert (states[:, 12] == cap).all(), cap
        if ref is None:
            ref = (maps, counts, states)
            assert len({bytes(m.cpu().numpy()) for m in maps}) > 2
        else:
            assert torch.equal(maps, ref[0]) and torch.equal(counts, ref[1]), cap
            assert torch.equal(states[:, cols], ref[2][:, cols]), cap
    maps, counts, states = engine.greedy_sweep(table, p.numel, "pcc", thr, fmts, rng, None, init)
    assert torch.equal(maps, ref[0]) and torch.equal(counts, ref[1]) and torch.equal(states[:, :8], ref[2][:, :8])
    prev = L.qa_greedy_cluster_cap(16)
    try:
        thr300 = np.linspace(0.999999, 0.99, 300)
        maps, counts, states = engine.greedy_sweep(table, p.numel, "pcc", thr300, fmts, rng, pre, init)
        for i in range(0, 300, 23):
            a, c, s = engine.greedy_assign(table, p.numel, "pcc", float(thr300[i]), fmts, engine.make_rng(123), prefetched=pre, init=init)
            assert torch.equal(maps[i], a) and torch.equal(counts[i], c) and torch.equal(states[i, :8], s[:8]), i
    finally:
        L.qa_greedy_cluster_cap(prev)


@pytest.mark.gpu
def test_certificate_falls_back_per_threshold():
    """A threshold equal to a value the chain reached: that row alone is redone in reference order (and equals the oracle);
    the other rows of the sweep keep their fast results.  The default first point on bf16-exact data with bf16 as the base
    format (pcc exactly 1.0) takes the same path."""
    x = G.algo_input("het_256x512")
    fmts = list(G.MIXED)
    dr = MixedTileGreedyCompression({"metric": "pcc", "threshold": 0.995, "seed": 3}).run_prepared(engine.prepare_tiles(x), fmts)
    tie = float(dr.meta["state"].cpu().numpy()[7])
    thr = [0.999, 0.995, tie, 0.99]
    rows, maps = sweep.greedy_sweep_tensor(x, fmts, "pcc", thresholds=thr, seed=3)
    assert [r["fallback"] for r in rows] == [False, False, True, False]
    assert rows[2]["min_margin"] < 2e-13
    table = orc.tile_stat_table(x)
    for r, m, t in zip(rows, maps.cpu().numpy(), thr):
        want, counts = orc.greedy_assign(table, fmts, "pcc", t, 3)
        assert np.array_equal(m, want.reshape(-1)) and r["counts"] == counts, t
    xb = engine.prepare_loaded(torch.from_numpy(x).to(torch.bfloat16))
    rows, maps = sweep.greedy_sweep_tensor(xb, fmts, "pcc", steps=3, lowest=0.99, seed=3)
    highest = sweep.base_format_score(xb, "bf16", "pcc")
    assert highest == 1.0 and [r["threshold"] for r in rows] == list(np.linspace(highest, 0.99, 3))
    assert rows[0]["fallback"] is True
    for r, m in zip(rows, maps.cpu().numpy()):
        want, counts = orc.greedy_assign(table, fmts, "pcc", r["threshold"], 3)
        assert np.array_equal(m, want.reshape(-1)) and r["counts"] == counts
    with pytest.raises(sweep.SweepRangeError):
        sweep.greedy_sweep_tensor(x, fmts, "pcc", steps=3, lowest=1.5)
    with pytest.raises(sweep.SweepRangeError):
        sweep.greedy_sweep_tensor(x, fmts, "mae", steps=3, lowest=0.0, highest=1e-3)


@pytest.mark.gpu
def test_full_size_sweep_reproduces_reference_map():
    """bench.py's q_a_proj (1536 x 7168, cfg2) swept with the golden's seed over thresholds around 0.999: the 0.999 row is the
    reference's committed map (tests/golden/cfg2_bench_workload.*)."""
    gold = G.GOLDEN
    meta = json.loads((gold / "cfg2_bench_workload.json").read_text())["q_a_proj"]
    want = dict(np.load(gold / "cfg2_bench_workload.npz"))["q_a_proj"].reshape(-1)
    x = synthetic.randn_bf16_cpu(tuple(meta["shape"]), meta["seed"]).cuda()
    thr = [0.9999, 0.9995, 0.999, 0.995, 0.99]
    rows, maps = sweep.greedy_sweep_tensor(x, list(G.MIXED), "pcc", thresholds=thr, seed=123)
    assert np.array_equal(maps[2].cpu().numpy(), want)
    assert rows[2]["counts"] == {k: int(v) for k, v in meta["counts"].items()}


# ------------------------------------------------------------------------------------------------------------------------
# CLI
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cache(tmp_path_factory):
    c = tmp_path_factory.mktemp("hf") / "hf-cache"
    U.seed_fp32_cache(c)
    return c


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    return write_checkpoint(tmp_path_factory.mktemp("ckpt") / "tiny-r1")


def _read_csv(path):
    lines = path.read_text().strip().splitlines()
    head = lines[0].split(",")
    return [dict(zip(head, ln.split(","))) for ln in lines[1:]]


def _check_cli_tree(out, index, names, metric, formats, seed):
    for name in names:
        d = out / "details" / name.replace("/", "_").replace(".", "_")
        cfg = json.loads((d / "sweep_config.json").read_text())
        rows = _read_csv(d / "sweep_results.csv")
        assert cfg["algorithm"] == "mixed-tile-greedy" and cfg["seed"] == seed and cfg["formats"] == formats
        assert cfg["highest_metric_val"] == float(rows[0]["threshold"])
        p = engine.prepare_loaded(index.load(name))
        for r in rows:
            dr = MixedTileGreedyCompression({"metric": metric, "threshold": float(r["threshold"]), "seed": seed}).run_prepared(p, formats)
            got = {k: r[k] for k in ("size_bytes", "pcc", "mae", "atol")}
            assert got == {"size_bytes": str(dr.tile_bytes), **{k: str(float(v)) for k, v in dr.metrics.items()}}, (name, r)
            assert {f: int(r[f"{f}_tiles"]) for f in formats} == {f: dr.counts[f] for f in formats}, (name, r)


@pytest.mark.gpu
@pytest.mark.parametrize("metric,lowest", [("pcc", "0.99"), ("mae", "0.005")])
def test_cli_greedy_sweep_rows_equal_single_runs(cache, tmp_path, metric, lowest):
    """The float32-cache repository (2-D, ragged and 1-D tensors): every CSV row is the single-threshold run's."""
    out = tmp_path / "out"
    argv = [U.REPO, U.FILTER, "--cache-dir", str(cache), "--out-dir", str(out), "--algorithm", "mixed-tile-greedy",
            "--metric", metric, "--lowest-metric-val", lowest, "--steps", "4", "--seed", "7", "--formats", "bfp8,bfp4,bfp2"]
    assert sweep_cli.main(argv) == 0
    index = tensor_source.build_tensor_index(U.REPO, U.REVISION, str(cache))
    names = sweep_cli.select_tensors(index, U.FILTER, True)
    assert len(names) == 4
    _check_cli_tree(out, index, names, metric, ["bfp8", "bfp4", "bfp2"], 7)


@pytest.mark.gpu
def test_cli_greedy_sweep_checkpoint_and_random_seed(ckpt, tmp_path):
    """The safetensors checkpoint (bf16, float32 and block-scaled fp8 weights), seed drawn once: every tensor records the
    same seed and every CSV row is the single-threshold run with it."""
    out = tmp_path / "out"
    argv = [U.REPO, "proj", "--checkpoint-dir", str(ckpt), "--out-dir", str(out), "--algorithm", "mixed-tile-greedy",
            "--metric", "pcc", "--lowest-metric-val", "0.99", "--steps", "3"]
    assert sweep_cli.main(argv) == 0
    index = tensor_source.build_tensor_index(U.REPO, checkpoint_dir=ckpt)
    names = sweep_cli.select_tensors(index, "proj", True)
    assert L1 in names and len(names) == 4
    seeds = {json.loads((d / "sweep_config.json").read_text())["seed"] for d in (out / "details").iterdir()}
    assert len(seeds) == 1 and seeds.pop() > 0
    seed = json.loads(next((out / "details").iterdir()).joinpath("sweep_config.json").read_text())["seed"]
    _check_cli_tree(out, index, names, "pcc", list(G.MIXED), seed)


@pytest.mark.gpu
def test_cli_greedy_sweep_two_gpus_write_the_same_files(ckpt, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 visible GPUs")
    base = [U.REPO, "proj", "--checkpoint-dir", str(ckpt), "--algorithm", "mixed-tile-greedy", "--metric", "pcc",
            "--lowest-metric-val", "0.99", "--steps", "3", "--seed", "5"]
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "a")]) == 0
    assert sweep_cli.main(base + ["--out-dir", str(tmp_path / "b"), "--gpus", "2"]) == 0
    fa = sorted(p.relative_to(tmp_path / "a") for p in (tmp_path / "a").rglob("*") if p.is_file())
    fb = sorted(p.relative_to(tmp_path / "b") for p in (tmp_path / "b").rglob("*") if p.is_file())
    assert fa == fb and len(fa) == 8
    for f in fa:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f


@pytest.mark.gpu
def test_cli_greedy_highest_below_lowest_is_a_range_error(cache, tmp_path, capsys):
    argv = [U.REPO, U.SWEEP_TENSOR, "--no-regex", "--cache-dir", str(cache), "--out-dir", str(tmp_path / "o"),
            "--algorithm", "mixed-tile-greedy", "--highest-metric-val", "0.9", "--lowest-metric-val", "0.99"]
    assert sweep_cli.main(argv) == 1
    assert capsys.readouterr().out == "error: lowest-metric-val must be <= highest metric for pcc\n"


@pytest.mark.parametrize("extra,needle", [
    (["--algorithm", "mixed-tile-random"], "--algorithm must be one of"),
    (["--seed", "5"], "--seed applies to --algorithm mixed-tile-greedy only"),
    (["--highest-metric-val", "0.99"], "--highest-metric-val applies to --algorithm mixed-tile-greedy only"),
    (["--algorithm", "mixed-tile-greedy", "--seed", "-3"], "--seed must be"),
    (["--algorithm", "mixed-tile-greedy", "--highest-metric-val", "nan"], "--highest-metric-val must be a finite number"),
])
def test_cli_rejects_bad_greedy_flags(tmp_path, capsys, extra, needle):
    """Host only: a bad --algorithm / --seed / --highest-metric-val combination prints one error line and returns 1 before
    any tensor is read."""
    assert sweep_cli.main([U.REPO, U.SWEEP_TENSOR, "--out-dir", str(tmp_path / "o")] + extra) == 1
    err = capsys.readouterr().err
    assert len(err.strip().splitlines()) == 1 and err.startswith("error: ") and needle in err
    assert not (tmp_path / "o").exists()


def test_cli_greedy_flags_parse():
    args = sweep_cli.build_parser().parse_args(["r", "t", "--algorithm", "mixed-tile-greedy", "--seed", "0",
                                                "--highest-metric-val", "0.9999"])
    assert sweep_cli.greedy_args_error(args) is None
    assert (args.algorithm, args.seed, args.highest_metric_val) == ("mixed-tile-greedy", 0, 0.9999)
    args = sweep_cli.build_parser().parse_args(["r", "t"])
    assert args.algorithm == "mixed-tile-threshold" and sweep_cli.greedy_args_error(args) is None


# ------------------------------------------------------------------------------------------------------------------------
# C entry point: argument checks (host only: every case fails before anything is enqueued)
# ------------------------------------------------------------------------------------------------------------------------
def _sweep_call(**kw):
    L = _lib.lib()
    fake = 256                                   # never dereferenced: every call below fails its checks first
    a = dict(table=fake, ntiles=64, numel=65536.0, metric=0, thresholds=fake, nthr=4, order=[0, 1, 2, 3], rng=fake,
             assignment=fake, counts=fake, state=fake, work=fake)
    a.update(kw)
    order = _lib.int32_array(a["order"]) if a["order"] is not None else None
    rc = L.qa_greedy_assign_sweep(a["table"], a["ntiles"], a["numel"], a["metric"], a["thresholds"], a["nthr"], order,
                                  len(a["order"] or []), a["rng"], a["assignment"], a["counts"], a["state"], a["work"],
                                  None, None, None, 0, None)
    return rc, L.qa_last_error().decode()


@pytest.mark.parametrize("kw,needle", [
    ({"table": None}, "bad args"), ({"thresholds": None}, "bad args"), ({"rng": None}, "bad args"),
    ({"assignment": None}, "bad args"), ({"counts": None}, "bad args"), ({"state": None}, "bad args"),
    ({"work": None}, "bad args"), ({"nthr": 0}, "bad args"), ({"nthr": -5}, "bad args"), ({"ntiles": 0}, "bad args"),
    ({"ntiles": 0x40000000}, "bad args"), ({"metric": 3}, "bad metric"), ({"metric": -1}, "bad metric"),
    ({"order": None}, "bad format order"), ({"order": [0, 1, 2, 3, 0]}, "bad format order"),
    ({"order": [0, 7]}, "bad format index"), ({"nthr": 1 << 28}, "too many thresholds"),
])
def test_sweep_entry_point_rejects_bad_arguments(kw, needle):
    rc, msg = _sweep_call(**kw)
    assert rc != 0 and msg.startswith("qa_greedy_assign_sweep: ") and needle in msg, (kw, msg)


def test_sweep_work_bytes():
    L = _lib.lib()
    for nt in (1, 1000, 65536):
        assert L.qa_greedy_sweep_work_bytes(nt, 0) == L.qa_greedy_sweep_work_bytes(nt, 1) >= L.qa_greedy_par_work_bytes(nt) + 40
        assert L.qa_greedy_sweep_work_bytes(nt, 2) >= L.qa_greedy_work_bytes(nt) + 40
        assert L.qa_greedy_sweep_work_bytes(nt, 0) % 256 == 0
    assert L.qa_greedy_sweep_work_bytes(0, 0) == -1 and L.qa_greedy_sweep_work_bytes(10, 3) == -1
    assert L.qa_greedy_sweep_work_bytes(0x40000000, 0) == -1
