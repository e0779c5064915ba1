"""Command-line parity against goldens written by the UNMODIFIED reference programs (tests/golden/make_golden_cli.py):
`table.txt` (every column but TIME(s)), `compression_config.used.json`, assignment maps + mapping JSON, random-sample
CSVs and `sweep_results.csv` must come out identical

* from this package's own CLIs (`quantization_analysis_b200.wq`, `.sweep_cli`), and
* from the reference's own `wq` / sweep script running over this package's drop-in modules (install_drop_in()).
"""
import json

import pytest

from tests import cli_util as U

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    w = tmp_path_factory.mktemp("cli")
    U.seed_fp32_cache(w / "data" / "hf-cache")
    return w


@pytest.mark.parametrize("case", sorted(U.WQ_CASES))
def test_wq_cli_matches_reference_output_tree(workdir, case):
    from quantization_analysis_b200 import wq
    cfg = workdir / f"{case}.json"
    cfg.write_text(json.dumps(U.WQ_CASES[case]))
    root = workdir / "own" / case
    rc = wq.run([U.REPO, U.FILTER, "--compression-config", str(cfg), "--recompute", "--summary", "--cache-dir",
                 str(workdir / "data" / "hf-cache"), "--results-root", str(root), "--processed-root", str(workdir / "own-processed")])
    assert rc == 0
    got = U.latest_results_dir(root, U.WQ_CASES[case]["algorithm"])
    assert U.compare_trees(got, U.CLI_GOLDEN / "wq" / case) == []


@pytest.mark.parametrize("case", sorted(U.SWEEP_CASES))
def test_sweep_cli_matches_reference_csv(workdir, case):
    from quantization_analysis_b200 import sweep_cli
    out = workdir / "own-sweep" / case
    rc = sweep_cli.main([U.REPO, U.SWEEP_TENSOR, "--no-regex", "--cache-dir", str(workdir / "data" / "hf-cache"), "--out-dir", str(out)]
                        + U.SWEEP_CASES[case])
    assert rc == 0
    assert U.compare_trees(out, U.CLI_GOLDEN / "sweep" / case) == []


def test_sweep_range_errors_like_reference(workdir):
    """lowest-metric-val on the wrong side of the start metric: error message + return code 1 (sweep:659-670)."""
    from quantization_analysis_b200 import sweep_cli
    base = [U.REPO, U.SWEEP_TENSOR, "--no-regex", "--cache-dir", str(workdir / "data" / "hf-cache"), "--out-dir", str(workdir / "err")]
    assert sweep_cli.main(base + ["--metric", "pcc", "--lowest-metric-val", "1.5"]) == 1
    assert sweep_cli.main(base + ["--metric", "mae", "--lowest-metric-val", "0.0"]) == 1


_DROPIN_GOLDENS = r'''
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import quantization_analysis_b200 as q
q.install_drop_in()
from compression_algorithms import create_algorithm          # the names the reference's programs import
from compression_algorithms.metrics import pearson_corr
from compression_algorithms.quantizer import Quantizer
import quantization_formats
from tests import golden_util as G
assert "quantization_analysis_b200" in quantization_formats.__file__
quantizer = Quantizer(backend="emulation")
for name in G.algo_case_names():
    x = G.algo_input(name)
    for key, m, want_a, want_y in G.algo_runs(name):
        res = create_algorithm(m["algo"], dict(m["params"])).run(xf=x, formats=G.FORMATS, quantizer=quantizer, cache=None)[0]
        d = np.abs(x - res.y)
        assert np.array_equal(np.asarray(res.meta["assignment"], dtype=np.int8), want_a), key
        assert np.array_equal(G.bits(res.y), want_y.reshape(-1)), key
        assert res.tile_counts == m["counts"] and res.tile_bytes == m["tile_bytes"], key
        assert pearson_corr(x, res.y) == m["pcc_f32"] and float(np.mean(d)) == m["mae_f32"] and float(np.max(d)) == m["atol_f32"], key
print("drop_in_ok")
'''


def test_drop_in_modules_reproduce_reference_goldens():
    """install_drop_in() in a fresh interpreter: the reference's module names (compression_algorithms.*, quantization_formats)
    resolve to this package, and every recorded reference run (tests/golden/algo_small.*), called the way the reference's
    programs call it, gives the reference's maps, reconstructions, counts, bytes and float32 scores."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, "-c", _DROPIN_GOLDENS, str(U.ROOT)], capture_output=True, text=True, timeout=600, cwd=str(U.ROOT))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "drop_in_ok" in out.stdout


def test_unmodified_reference_programs_over_drop_in(workdir):
    """The reference's own `wq` and sweep script, unmodified, import this package through install_drop_in() and must
    write the same trees as when they ran on the reference's NumPy modules."""
    if not (U.REF_COPY / "wq").exists():
        pytest.skip("oracle/_ref not populated (run oracle/make_ref.sh in the build container)")
    w = workdir / "dropin"
    (w / "data").mkdir(parents=True)
    U.seed_fp32_cache(w / "data" / "hf-cache")
    jobs = []
    for case, cfg in U.WQ_CASES.items():
        p = w / f"{case}.json"
        p.write_text(json.dumps(cfg))
        jobs.append((U.REF_COPY / "wq", [U.REPO, U.FILTER, "--compression-config", str(p), "--recompute", "--summary"]))
    for case, args in U.SWEEP_CASES.items():
        jobs.append((U.REF_COPY / "scripts" / "sweep_mixed_tile_threshold.py",
                     [U.REPO, U.SWEEP_TENSOR, "--no-regex", "--out-dir", str(w / "sweep" / case)] + args))
    U.run_reference_programs_over_dropin(jobs, w)
    problems = []
    seen_algos = {}
    for case, cfg in U.WQ_CASES.items():
        base = w / "results" / U.REPO.replace("/", "__") / cfg["algorithm"]
        runs = sorted(p for p in base.iterdir() if p.is_dir())
        k = seen_algos.get(cfg["algorithm"], 0)            # two greedy configs share one algorithm directory (one run each, in order)
        seen_algos[cfg["algorithm"]] = k + 1
        problems += [f"wq/{case}: {d}" for d in U.compare_trees(runs[k], U.CLI_GOLDEN / "wq" / case)]
    for case in U.SWEEP_CASES:
        problems += [f"sweep/{case}: {d}" for d in U.compare_trees(w / "sweep" / case, U.CLI_GOLDEN / "sweep" / case)]
    assert problems == []
