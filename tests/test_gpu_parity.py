"""GPU parity: the CUDA path (through the C ABI, via the drop-in Python API) against the golden
fixtures made from the reference and against the CPU oracle on the same seeded inputs."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc
from tests import golden_util as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def qa():
    from quantization_analysis_b200 import _lib, engine, quantization_formats as qf
    from quantization_analysis_b200 import compression_algorithms as ca
    _lib.lib()
    return {"engine": engine, "qf": qf, "ca": ca}


@pytest.mark.parametrize("name", G.kat_cases())
def test_formats_bit_exact_vs_reference(qa, name):
    x, outs = G.kat(name)
    for fmt in G.FORMATS:
        y = qa["qf"].quantize_weight_values(x, fmt)
        assert y.shape == x.shape and y.dtype == np.float32
        assert np.array_equal(G.bits(y), outs[fmt]), f"{name}/{fmt}"


def test_formats_torch_bf16_path(qa):
    x, outs = G.kat("rand_bf16_spread12")
    xt = torch.from_numpy(x).cuda().to(torch.bfloat16)
    for fmt in ("bf16", "bfp8", "bfp4", "bfp2"):
        y = qa["qf"].quantize_weight_values(xt, fmt)
        assert y.dtype == torch.bfloat16 and y.is_cuda
        assert np.array_equal(G.bits(y.float().cpu().numpy()), outs[fmt])


def test_unsupported_format_raises(qa):
    with pytest.raises(ValueError):
        qa["qf"].quantize_weight_values(np.zeros(4, np.float32), "int3")


def test_cfg1_reconstructions_sha(qa):
    from quantization_analysis_b200 import synthetic
    meta = G.js("cfg1_q_a_proj.json")
    x = synthetic.randn_f32_np((1536, 7168), 0)
    assert hashlib.sha256(x.tobytes()).hexdigest() == meta["input_sha256"]
    res = qa["ca"].create_algorithm("none").run(x, G.FORMATS, qa["ca"].quantizer.Quantizer("emulation"), None)
    for r in res:
        assert hashlib.sha256(np.ascontiguousarray(r.y).tobytes()).hexdigest() == meta["none"][r.fmt.lower()]["y_sha256"]


def _table_from_device(t, table):
    tb = t.cpu().numpy()
    out = {"sx": tb[0], "sx2": tb[1]}
    for i, f in enumerate(G.MIXED):
        out[f] = {k: tb[2 + 5 * i + j] for j, k in enumerate(("sy", "sy2", "sxy", "sabs", "amax"))}
    return out


@pytest.mark.parametrize("name", G.algo_case_names())
def test_tile_stats_strict_bit_exact(qa, name):
    eng = qa["engine"]
    x = G.algo_input(name)
    want = orc.tile_stat_table(x)
    p = eng.prepare_tiles(x)
    got = _table_from_device(eng.tile_stats(p, G.MIXED, strict=True), None)
    assert np.array_equal(got["sx"], want["sx"]) and np.array_equal(got["sx2"], want["sx2"])
    for f in G.MIXED:
        for k in ("sy", "sy2", "sxy", "sabs", "amax"):
            assert np.array_equal(got[f][k], want[f][k]), (name, f, k)


@pytest.mark.parametrize("name", G.algo_case_names())
def test_tile_stats_fast_matches_oracle(qa, name):
    """Fast table vs the NumPy-order oracle: every sum whose float64 value is exactly representable
    must be bit-identical; sum x^2 over tiles with a very wide exponent spread is order-dependent
    in float64 even in NumPy, so it is held to 1e-13 relative (a few ulp)."""
    eng = qa["engine"]
    x = G.algo_input(name)
    want = orc.tile_stat_table(x)
    p = eng.prepare_tiles(x)
    assert p.dtype_code == 0
    got = _table_from_device(eng.tile_stats(p, G.MIXED, strict=False), None)
    assert np.array_equal(got["sx"], want["sx"]), name
    assert np.allclose(got["sx2"], want["sx2"], rtol=1e-13, atol=0), name
    for f in G.MIXED:
        for k in ("sy", "sy2", "sxy", "sabs", "amax"):
            if f == "bf16" and k in ("sy2", "sxy"):
                assert np.allclose(got[f][k], want[f][k], rtol=1e-13, atol=0), (name, f, k)
            else:
                assert np.array_equal(got[f][k], want[f][k]), (name, f, k)


@pytest.mark.parametrize("name", G.algo_case_names())
def test_tile_scores_bit_exact_vs_reference(qa, name):
    eng = qa["engine"]
    x = G.algo_input(name)
    z = G.npz("algo_small.npz")
    s = eng.tile_scores(eng.prepare_tiles(x), G.MIXED).cpu().numpy()
    for mi, metric in enumerate(("pcc", "mae", "atol")):
        for fi, fmt in enumerate(G.MIXED):
            want = z[f"{name}__tilescore__{fmt}__{metric}"]
            assert np.array_equal(s[mi, fi].view(np.uint32), want.view(np.uint32)), (name, fmt, metric)


@pytest.mark.parametrize("parallel", [False, True])
def test_numpy_rng_streams(qa, parallel):
    eng = qa["engine"]
    z = G.npz("numpy_rng.npz")
    for seed in (1, 123, 2**31 - 1):
        rng = eng.make_rng(seed)
        perm = lambda n: eng.numpy_permutation(rng, n, parallel=parallel).cpu().numpy()   # noqa: E731
        assert np.array_equal(perm(10752), z[f"s{seed}__perm_10752"])
        assert np.array_equal(perm(777), z[f"s{seed}__perm_777"])
        assert np.array_equal(eng.numpy_integers(rng, 4, 1000).cpu().numpy(), z[f"s{seed}__int4_1000"])
        assert np.array_equal(eng.numpy_integers(rng, 3, 1000).cpu().numpy(), z[f"s{seed}__int3_1000"])
        assert np.array_equal(perm(4096), z[f"s{seed}__perm_4096"])
        assert np.array_equal(eng.numpy_integers(rng, 2, 777).cpu().numpy(), z[f"s{seed}__int2_777"])
        assert np.array_equal(perm(2), z[f"s{seed}__perm_2"])
        assert np.array_equal(perm(1), z[f"s{seed}__perm_1"])
        assert np.array_equal(perm(65537), z[f"s{seed}__perm_65537"])


def test_parallel_greedy_equals_sequential_chain(qa):
    """The block-parallel greedy must reproduce the one-thread chain exactly: assignment, counts,
    final float64 state and the RNG stream position, on a tensor large enough for many chunks."""
    from quantization_analysis_b200 import synthetic
    eng = qa["engine"]
    for shape, seed, maker in [((2048, 1536), 5, synthetic.randn_f32_np), ((1024, 2048), 6, synthetic.heterogeneous_f32_np)]:
        p = eng.prepare_tiles(maker(shape, seed))
        for metric, thr in (("pcc", 0.999), ("pcc", 0.99), ("mae", 3e-4)):
            table = eng.tile_stats(p, G.MIXED, exact_abs=True)
            r1, r2 = eng.make_rng(77), eng.make_rng(77)
            a1, c1, s1 = eng.greedy_assign(table, p.numel, metric, thr, list(G.MIXED), r1, parallel=False)
            a2, c2, s2 = eng.greedy_assign(table, p.numel, metric, thr, list(G.MIXED), r2, parallel=True)
            assert torch.equal(a1, a2), (shape, metric, thr)
            assert torch.equal(c1, c2)
            assert torch.equal(r1, r2)
            s1, s2 = s1.cpu().numpy(), s2.cpu().numpy()
            flags = int(s2[6]) & 0xFFFF
            # sequentially rounded sums that drive the decisions are bit-identical; in pcc mode sum|x-y| is a
            # plain sum (only its zero test is ever used) and sum x / sum y may be flagged as tree / fixed-grid sums
            sel = [1, 3, 4, 7] if metric == "pcc" else [5, 7]
            assert np.array_equal(s1[sel], s2[sel]), (metric, s1, s2)
            if metric == "pcc":
                assert s2[5] == pytest.approx(s1[5], rel=1e-12)
                if not (flags & 7):
                    assert np.array_equal(s1[[0, 2]], s2[[0, 2]])
                else:
                    assert np.allclose(s1[[0, 2]], s2[[0, 2]], rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("name", G.algo_case_names())
def test_algorithms_match_reference(qa, name, strict):
    ca = qa["ca"]
    x = G.algo_input(name)
    for key, m, want_assign, want_y in G.algo_runs(name):
        params = dict(m["params"])
        if m["algo"] == "mixed-tile-greedy":
            params["strict_sums"] = strict
            params["sequential_chain"] = strict      # strict run = NumPy-order sums + one-thread chain
        elif strict:
            continue
        res = ca.create_algorithm(m["algo"], params).run(x, G.FORMATS, ca.quantizer.Quantizer("emulation"), None)[0]
        if m["algo"] == "mixed-tile-random":
            # every sample: the reference's float32 whole-tensor values, bit for bit (mixed_tile_random.py:137-155)
            assert res.meta["samples"] == m["samples"], key
        assert np.array_equal(res.meta["assignment"], want_assign), key
        assert res.tile_counts == m["counts"], key
        assert res.tile_bytes == m["tile_bytes"], key
        assert np.array_equal(G.bits(res.y), want_y.reshape(-1)), key


def test_cfg1_greedy_and_threshold_goldens(qa):
    from quantization_analysis_b200 import synthetic
    ca = qa["ca"]
    meta, z = G.js("cfg1_q_a_proj.json"), G.npz("cfg1_q_a_proj.npz")
    x = synthetic.randn_f32_np((1536, 7168), 0)
    g = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 123})
    r = g.run(x, G.FORMATS, None, None)[0]
    assert np.array_equal(r.meta["assignment"], z["greedy_pcc0999_seed123"])
    assert r.tile_counts == meta["greedy_pcc0999_seed123"]["counts"]
    assert r.tile_bytes == meta["greedy_pcc0999_seed123"]["tile_bytes"]
    assert hashlib.sha256(np.ascontiguousarray(r.y).tobytes()).hexdigest() == meta["greedy_pcc0999_seed123"]["y_sha256"]
    t = ca.create_algorithm("mixed-tile-threshold", {"metric": "pcc", "threshold": 0.9937})
    r = t.run(x, G.FORMATS, None, None)[0]
    assert np.array_equal(r.meta["assignment"], z["threshold_pcc09937"])
    assert r.tile_counts == meta["threshold_pcc09937"]["counts"]


def test_cfg1_exact_metrics_vs_fp64_oracle(qa):
    """pcc / mae / atol within 1e-6 relative of the fp64 evaluation of the reference formulas."""
    from quantization_analysis_b200 import synthetic
    eng = qa["engine"]
    meta = G.js("cfg1_q_a_proj.json")
    x = synthetic.randn_f32_np((1536, 7168), 0)
    p = eng.prepare_tiles(x)
    table = eng.tile_stats(p, G.MIXED)
    for fi, fmt in enumerate(G.MIXED):
        m = eng.metrics_from_sums(eng.assignment_sums(table, None, fi).cpu().numpy(), p.numel)
        ex = orc.exact_metrics_f64(x, orc.quantize(x, fmt))
        for k in ("pcc", "mae", "atol"):
            assert m[k] == pytest.approx(ex[k], rel=1e-6, abs=1e-300), (fmt, k)
        ref = meta["none"][fmt]
        assert m["atol"] == ref["atol_f32"]
        assert m["mae"] == pytest.approx(ref["mae_f32"], rel=2e-6, abs=1e-300)
        assert abs(m["pcc"] - ref["pcc_f32"]) < 5e-5        # float32 noise of the reference (SURVEY fact 7)


def test_random_samples_match_exact_oracle(qa):
    eng = qa["engine"]
    x = G.algo_input("het_256x512")
    table_o = orc.tile_stat_table(x)
    p = eng.prepare_tiles(x)
    table = eng.tile_stats(p, G.MIXED)
    for fmts in (list(G.MIXED), ["bfp8", "bfp4"], ["bfp8", "bfp4", "bfp2"], ["bfp4"]):
        ch_o, met_o = orc.random_samples_exact(table_o, fmts, 7, 99)
        ch, met, cnt = eng.random_samples(table, p.numel, fmts, 7, eng.make_rng(99))
        assert np.array_equal(ch.cpu().numpy(), ch_o), fmts
        assert np.allclose(met.cpu().numpy(), met_o, rtol=1e-9, atol=0), fmts


def test_empty_and_scalar_inputs(qa):
    ca, qf = qa["ca"], qa["qf"]
    e = np.zeros((0, 8), dtype=np.float32)
    assert qf.quantize_weight_values(e, "bfp8").shape == (0, 8)
    r = ca.create_algorithm("mixed-tile-greedy", {"seed": 1}).run(e, G.FORMATS, None, None)[0]
    assert r.meta["assignment"].shape == (1, 1) and r.tile_counts == {f: 0 for f in G.MIXED}
    s = np.array(0.3, dtype=np.float32)
    assert qf.quantize_weight_values(s, "bfp4").shape == ()


def test_sweep_matches_oracle(qa):
    """Threshold sweep (scripts/sweep_mixed_tile_threshold.py:145-155, 659-670): float64 thresholds from the max (pcc) or
    the min (mae / atol) of the highest-precision format's scores, maps bit-equal for all thresholds, whole-tensor
    metrics equal to the reference's float32 values (restated orders)."""
    from quantization_analysis_b200 import sweep
    rng = np.random.default_rng(4)
    for x in (G.algo_input("het_256x512"), (rng.standard_normal((96, 128)) * 0.02).astype(np.float32)):   # 2nd: not bf16-exact
        for metric, lowest in (("pcc", 0.9), ("mae", 5e-3), ("atol", 0.05)):
            sc = orc.padded_tile_scores(x, G.MIXED, metric)
            top = float(np.max(sc["bf16"])) if metric == "pcc" else float(np.min(sc["bf16"]))
            thr = np.linspace(top, lowest, 16)
            want = orc.sweep_assign(sc, G.MIXED, metric, thr.astype(np.float32))
            rows, maps = sweep.sweep_tensor(x, G.MIXED, metric, steps=16, lowest=lowest)
            assert [r["threshold"] for r in rows] == [float(t) for t in thr]
            assert np.array_equal(maps.cpu().numpy(), want), metric
            for i in (0, 7, 15):
                w = orc.wq_scores_restated(x, orc.apply_assignment(x, want[i]))
                for k in ("pcc", "mae", "atol"):
                    assert rows[i][k] == w[k], (metric, i, k)
    with pytest.raises(sweep.SweepRangeError):
        sweep.sweep_tensor(x, G.MIXED, "mae", steps=4, lowest=-1.0)


def test_wq_cli_writes_reference_artifacts(qa, tmp_path):
    """The synthetic provider through the reference's argv (wq:37-79) and output tree (wq:630-647, 295-316)."""
    import json
    from quantization_analysis_b200 import wq
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps({"algorithm": "mixed-tile-greedy", "quantization_formats": ["bf16", "bfp8", "bfp4", "bfp2", "fp0"],
                               "params": {"metric": "pcc", "threshold": 0.999}, "seed": 123}))
    rc = wq.run(["synthetic", "kv_a_proj", "--compression-config", str(cfg), "--results-root", str(tmp_path / "res"),
                 "--cache-dir", str(tmp_path / "hf"), "--no-save-processed"])
    assert rc == 0
    run_dir = next((tmp_path / "res" / "synthetic" / "mixed-tile-greedy").iterdir())
    used = json.loads((run_dir / "compression_config.used.json").read_text())
    assert used["seed"] == 123 and used["seed_source"] == "config" and "seed" not in used["params"]
    assert (run_dir / "table.txt").read_text().startswith("model.layers.0.self_attn.kv_a_proj_with_mqa.weight\n  shape=(576, 7168)")
    maps = list(run_dir.rglob("assignment.npy"))
    assert len(maps) == 1
    a = np.load(maps[0])
    assert a.dtype == np.int8 and a.shape == (18, 224)
    mapping = json.loads((maps[0].parent / "assignment_mapping.json").read_text())
    assert mapping["int_to_format"] == G.MIXED and mapping["assignment_shape"] == [18, 224]


def test_striped_tables_concatenate_in_tile_order(qa):
    """Row stripes (sharding.row_stripes) produce table slices that concatenate to the full table."""
    from quantization_analysis_b200 import sharding
    eng = qa["engine"]
    x = G.algo_input("het_256x512")
    full = eng.tile_stats(eng.prepare_tiles(x), G.MIXED)
    parts = []
    for a, b in sharding.row_stripes(x.shape[0], 3):
        parts.append(eng.tile_stats(eng.prepare_tiles(x[a:b]), G.MIXED))
    assert torch.equal(torch.cat(parts, dim=1), full)


@pytest.mark.parametrize("kind", ["constant", "zeros", "one_tile", "mean_heavy", "tiny_values", "alternating_scale", "ragged"])
def test_parallel_greedy_degenerate_inputs(qa, kind):
    """Edge cases of the greedy: den == 0 branches, empty deltas, a non-zero mean (sum y is then a monotone sum
    carried with the reference's rounding sequence), binade changes, ragged tiles.  Parallel == one-thread chain,
    and both == the CPU oracle."""
    eng = qa["engine"]
    rng = np.random.default_rng(3)
    if kind == "constant":
        x = np.full((96, 128), 0.25, dtype=np.float32)
    elif kind == "zeros":
        x = np.zeros((64, 96), dtype=np.float32)
    elif kind == "one_tile":
        x = (rng.standard_normal((32, 32)) * 0.02).astype(np.float32)
    elif kind == "mean_heavy":
        x = (1.0 + rng.standard_normal((256, 384)) * 0.01).astype(np.float32)
    elif kind == "tiny_values":
        x = (rng.standard_normal((128, 256)) * 1e-30).astype(np.float32)
    elif kind == "alternating_scale":
        x = (rng.standard_normal((256, 256)) * 0.02).astype(np.float32)
        x[::2] *= 1000.0
    else:
        x = (rng.standard_normal((130, 75)) * 0.02).astype(np.float32)
    x = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    p = eng.prepare_tiles(x)
    table_o = orc.tile_stat_table(x)
    for metric, thr in (("pcc", 0.999), ("pcc", 0.9), ("mae", 1e-4)):
        table = eng.tile_stats(p, G.MIXED, exact_abs=True)
        a1, c1, s1 = eng.greedy_assign(table, p.numel, metric, thr, list(G.MIXED), eng.make_rng(5), parallel=False)
        a2, c2, s2 = eng.greedy_assign(table, p.numel, metric, thr, list(G.MIXED), eng.make_rng(5), parallel=True)
        assert torch.equal(a1, a2), (kind, metric, thr)
        assert torch.equal(c1, c2)
        want, counts = orc.greedy_assign(table_o, list(G.MIXED), metric, thr, 5)
        assert np.array_equal(a2.cpu().numpy().reshape(want.shape), want), (kind, metric, thr)
        assert {f: int(c2[i]) for i, f in enumerate(G.MIXED)} == counts
        if kind == "mean_heavy" and metric == "pcc":
            flags = int(s2.cpu().numpy()[6]) & 0xFFFF
            assert flags == 0, flags                      # nothing degraded: all sums carried faithfully
            assert np.array_equal(s1.cpu().numpy()[:5], s2.cpu().numpy()[:5])


def test_staged_permutation_matches_numpy(qa):
    """qa_perm_resolve (cluster) + qa_perm_apply (grid kernels) == numpy Generator.permutation, stream position included."""
    eng = qa["engine"]
    for seed, n in ((3, 0), (3, 1), (3, 2), (4, 97), (5, 98), (6, 5000), (7, 40000), (123, 114688)):
        r1, r2 = eng.make_rng(seed), eng.make_rng(seed)
        got = eng.numpy_permutation_staged(r1, n).cpu().numpy()
        gen = np.random.default_rng(seed)
        want = gen.permutation(n)
        assert np.array_equal(got, want), (seed, n)
        # same stream position afterwards: the next draws agree
        nxt = eng.numpy_permutation(r1, 50, parallel=False).cpu().numpy()
        assert np.array_equal(nxt, gen.permutation(50)), (seed, n)
        eng.numpy_permutation(r2, n, parallel=False)


def test_table_and_init_in_pieces(qa):
    """qa_tile_stats_rows + qa_greedy_init_sums_range over consecutive pieces == the one-shot calls (table and init header)."""
    import torch
    from quantization_analysis_b200 import _lib
    from quantization_analysis_b200._lib import METRIC_CODE, check
    eng = qa["engine"]
    L = _lib.lib()
    x = G.algo_input("het_256x512")
    p = eng.prepare_tiles(x)
    fmts = list(G.MIXED)
    order = _lib.int32_array([eng.FMT_INDEX[f] for f in fmts])
    for exact_abs, mode in ((True, _lib.STATS_FAST), (False, _lib.STATS_FAST_APPROX_ABS)):
        whole = eng.tile_stats(p, fmts, exact_abs=exact_abs)
        nt = whole.shape[1]
        pieces = torch.zeros_like(whole)
        th = p.tiles_h
        cuts = [0, 1, 3, th]
        for metric in ("pcc", "mae"):
            init_whole = eng.greedy_init(whole, metric, fmts)
            init_pieces = torch.zeros_like(init_whole)
            for a, b in zip(cuts[:-1], cuts[1:]):
                check(L.qa_tile_stats_rows(p.data.data_ptr(), _lib.QA_DT_BF16, p.rows, p.cols, p.cols, 0xF, mode, pieces.data_ptr(), a, b,
                                           torch.cuda.current_stream().cuda_stream), "qa_tile_stats_rows")
                check(L.qa_greedy_init_sums_range(pieces.data_ptr(), nt, METRIC_CODE[metric], order, len(fmts), init_pieces.data_ptr(),
                                                  a * p.tiles_w, b * p.tiles_w, torch.cuda.current_stream().cuda_stream),
                      "qa_greedy_init_sums_range")
            assert torch.equal(whole, pieces)
            hw = init_whole.view(torch.float64)[:7].cpu().numpy()
            hp = init_pieces.view(torch.float64)[:7].cpu().numpy()
            assert np.array_equal(hw, hp), (metric, hw, hp)


def test_greedy_staged_equals_inline(qa):
    """Prefetched permutations (engine.greedy_prefetch: the product's enqueue_perm_prefetch) and a precomputed init buffer
    (qa_greedy_init_deltas + qa_greedy_init_sums_range) given to qa_greedy_assign_passes give the same map, counts, state
    and stream position as the call that computes init into its work buffer and draws every permutation itself, in every
    combination of stages - including a base state that already fails, a pass 2 that accepts every tile (speculative
    third permutation used) and one that does not."""
    eng = qa["engine"]
    x = G.algo_input("het_256x512")
    p = eng.prepare_tiles(x)
    table = eng.tile_stats(p, G.MIXED, exact_abs=True)
    seen_spec, seen_nospec = False, False
    for metric, thr, fmts in (("pcc", 0.995, list(G.MIXED)), ("mae", 3e-4, list(G.MIXED)), ("pcc", 0.9999, ["bfp4", "bfp2"]),
                              ("pcc", 0.99, ["bfp8", "bfp4", "bfp2"]), ("pcc", 0.99999, list(G.MIXED)),
                              ("mae", 1e-5, list(G.MIXED)), ("pcc", 0.9, ["bfp2", "bfp4", "bfp8"])):
        r1 = eng.make_rng(31)
        a1, c1, s1 = eng.greedy_assign(table, p.numel, metric, thr, fmts, r1, parallel=True)
        if len(fmts) >= 3:
            if int(c1[eng.FMT_INDEX[fmts[0]]]) == 0:
                seen_spec = True
            elif int(c1[eng.FMT_INDEX[fmts[0]]]) < p.ntiles:
                seen_nospec = True
        for use_pre in (False, True):
            for use_init in (False, True):
                if not (use_pre or use_init):
                    continue
                r2 = eng.make_rng(31)
                pre = eng.greedy_prefetch(r2, p.ntiles, nfmt=len(fmts)) if use_pre else None
                init = eng.greedy_init(table, metric, fmts) if use_init else None
                a2, c2, s2 = eng.greedy_assign(table, p.numel, metric, thr, fmts, r2, parallel=True, prefetched=pre, init=init)
                assert torch.equal(a1, a2) and torch.equal(c1, c2), (metric, thr, fmts, use_pre, use_init)
                assert torch.equal(r1, r2), (metric, thr, fmts, use_pre, use_init)
                assert torch.equal(s1[:8], s2[:8])
                if len(fmts) >= 3:          # the same run as two launches (passes [0,2) and [2,n)) and as three
                    for cut in (1, 2):
                        r3 = eng.make_rng(31)
                        a3, c3, s3 = eng.greedy_assign(table, p.numel, metric, thr, fmts, r3, parallel=True, prefetched=pre, init=init,
                                                       split_at=cut)
                        assert torch.equal(a1, a3) and torch.equal(c1, c3) and torch.equal(r1, r3), (metric, thr, fmts, cut)
                        assert torch.equal(s1[:8], s3[:8])
    assert seen_spec and seen_nospec


def test_metrics_api_matches_fp64_formulas(qa):
    """metrics.pearson_corr / metric_value return the reference's own float32 numbers (qa_tensor_scores_f32);
    pearson_corr_exact is the float64 recombination (qa_pair_sums) of the same formula."""
    from quantization_analysis_b200.compression_algorithms import metrics
    x = G.algo_input("het_256x512")
    for fmt in ("bfp8", "bfp4", "bfp2", "fp0"):
        y = orc.quantize(x, fmt)
        ex = orc.exact_metrics_f64(x, y)
        ref = orc.wq_scores_restated(x, y)       # == NumPy's own values (tests/test_oracle_golden.py pins that on the CPU)
        assert metrics.pearson_corr_exact(x, y) == pytest.approx(ex["pcc"], rel=1e-9, abs=1e-12)
        assert metrics.pearson_corr(x, y) == ref["pcc"]
        assert metrics.metric_value(x, y, "mae") == ref["mae"]
        assert metrics.metric_value(x, y, "atol") == ref["atol"] == ex["atol"]
    assert metrics.pearson_corr(x, x) == 1.0 or metrics.pearson_corr(x, x) == pytest.approx(1.0, abs=1e-12)
    assert metrics.pearson_corr(np.zeros(0, np.float32), np.zeros(0, np.float32)) == 1.0
    c = np.full(64, 0.5, np.float32)
    assert metrics.pearson_corr(c, c) == 1.0 and metrics.pearson_corr(c, c + 1) == 0.0      # denom == 0 branch
    with pytest.raises(ValueError):
        metrics.metric_value(x, x, "rmse")
    assert metrics.metric_is_good(0.95, "pcc", 0.94) and not metrics.metric_is_good(0.5, "mae", 0.1)
    assert metrics.metric_better(0.9, 0.8, "pcc") and metrics.metric_better(0.1, 0.2, "atol")


def test_fp32_inputs_take_the_general_path(qa):
    """Non-bf16-exact float32 tensors (what a dequantised fp8 checkpoint looks like, hf_model_utils.py:209-215):
    never truncated - strict NumPy-order stats, faithful tile scores, greedy / threshold maps all match the oracle (the greedy
    runs on the fast float32 table, qa_tile_stats_f32, under the decision-margin certificate)."""
    eng, ca = qa["engine"], qa["ca"]
    rng = np.random.default_rng(17)
    x = (rng.standard_normal((96, 200)) * 0.02).astype(np.float32)
    x[5, 7] = 0.0
    p = eng.prepare_tiles(x)
    assert p.dtype_code == 1                                   # stayed float32
    want = orc.tile_stat_table(x)
    got = _table_from_device(eng.tile_stats(p, G.MIXED, strict=True), None)
    assert np.array_equal(got["sx"], want["sx"]) and np.array_equal(got["sx2"], want["sx2"])
    for f in G.MIXED:
        for k in ("sy", "sy2", "sxy", "sabs", "amax"):
            assert np.array_equal(got[f][k], want[f][k]), (f, k)
    s = eng.tile_scores(p, G.MIXED).cpu().numpy()
    for mi, metric in enumerate(("pcc", "mae", "atol")):
        sc = orc.padded_tile_scores(x, G.MIXED, metric)
        for fi, f in enumerate(G.MIXED):
            assert np.array_equal(s[mi, fi].view(np.uint32), sc[f].view(np.uint32)), (metric, f)
    r = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.995, "seed": 4}).run(x, G.FORMATS, None, None)[0]
    a, counts = orc.greedy_assign(want, list(G.MIXED), "pcc", 0.995, 4)
    assert np.array_equal(r.meta["assignment"], a) and r.tile_counts == counts
    assert np.array_equal(G.bits(r.y), G.bits(orc.apply_assignment(x, a)))
    t = ca.create_algorithm("mixed-tile-threshold", {"metric": "mae", "threshold": 3e-4}).run(x, G.FORMATS, None, None)[0]
    sc = orc.padded_tile_scores(x, G.MIXED, "mae")
    a2, c2 = orc.threshold_assign(sc, list(G.MIXED), "mae", 3e-4, want["th"], want["tw"])
    assert np.array_equal(t.meta["assignment"], a2) and t.tile_counts == c2


def test_random_bit_patterns_property(qa):
    """Property test: random shapes (incl. ragged) filled with random bf16 / fp32 bit patterns (subnormals, inf, nan,
    wide exponent spreads) - the device quantizers equal the oracle bit for bit."""
    qf = qa["qf"]
    rng = np.random.default_rng(2026)
    for trial in range(40):
        nd = int(rng.integers(1, 4))
        shape = tuple(int(v) for v in rng.integers(1, 70, size=nd))
        bits = rng.integers(0, 2**32, size=shape, dtype=np.uint64).astype(np.uint32)
        mode = trial % 4
        if mode == 0:
            bits &= np.uint32(0xFFFF0000)                                   # arbitrary bf16 patterns
        elif mode == 1:                                                     # narrow exponent band, bf16
            e = rng.integers(100, 140, size=shape).astype(np.uint32)
            bits = (bits & np.uint32(0x807F0000)) | (e << np.uint32(23))
        elif mode == 2:                                                     # full fp32 mantissas, narrow band
            e = rng.integers(110, 130, size=shape).astype(np.uint32)
            bits = (bits & np.uint32(0x807FFFFF)) | (e << np.uint32(23))
        x = bits.view(np.float32)
        with np.errstate(all="ignore"):
            for fmt in ("bf16", "bfp8", "bfp4", "bfp2"):
                assert np.array_equal(G.bits(qf.quantize_weight_values(x, fmt)), G.bits(orc.quantize(x, fmt))), (trial, shape, fmt)


def test_batch_graph_replay_equals_eager(qa):
    """GreedyBatch.run_graph (one captured CUDA graph per pass) gives the same maps / counts / states as eager enqueueing,
    and replays pick up newly loaded inputs."""
    import torch
    from quantization_analysis_b200.batch import GreedyBatch
    from quantization_analysis_b200 import synthetic
    shapes = [(256, 512), (96, 320), (512, 256)]
    xs = [synthetic.randn_bf16_cpu(s, 40 + i) for i, s in enumerate(shapes)]
    xs2 = [synthetic.randn_bf16_cpu(s, 50 + i) for i, s in enumerate(shapes)]
    eng = qa["engine"]
    for metric, thr, fmts in (("pcc", 0.999, list(G.MIXED)), ("mae", 3e-4, list(G.MIXED)), ("pcc", 0.9995, ["bfp8", "bfp4"]),
                              ("atol", 2e-3, list(G.MIXED))):
        b = GreedyBatch(shapes + [shapes[0]], metric=metric, threshold=thr, seed=9, tile_formats=fmts)   # two tensors share a tile count
        for data in (xs, xs2):
            b.load_device(data + [data[0]])
            b.run()
            eager = b.collect()
            for s in b.slots:
                s["assignment"].fill_(-1)
                s["counts"].zero_()
            b.run_graph()
            graph = b.collect()
            for e, g in zip(eager, graph):
                assert np.array_equal(e["assignment"], g["assignment"]), (metric, fmts)
                assert e["counts"] == g["counts"]
                assert np.array_equal(e["state"][:8], g["state"][:8])
            assert np.array_equal(graph[0]["assignment"], graph[3]["assignment"])        # the follower of a shared prefetch
            # and against the single-call engine path on the first tensor
            p = eng.prepare_tiles(data[0].cuda())
            table = eng.tile_stats(p, G.MIXED, exact_abs=(metric == "mae"))
            a1, c1, _ = eng.greedy_assign(table, p.numel, metric, thr, fmts, eng.make_rng(9))
            assert np.array_equal(a1.cpu().numpy().reshape(graph[0]["assignment"].shape), graph[0]["assignment"]), (metric, fmts)


def test_batch_from_host_async_equals_sync(qa):
    """enqueue_from_host / finish on two alternating batches == run_from_host == device-resident run."""
    from quantization_analysis_b200.batch import GreedyBatch
    from quantization_analysis_b200 import synthetic
    shapes = [(256, 512), (96, 320)]
    xs = [synthetic.randn_bf16_cpu(s, 60 + i).pin_memory() for i, s in enumerate(shapes)]
    b0 = GreedyBatch(shapes, metric="pcc", threshold=0.999, seed=9)
    b1 = GreedyBatch(shapes, metric="pcc", threshold=0.999, seed=9)
    want = b0.run_from_host(xs)
    b0.enqueue_from_host(xs)
    b1.enqueue_from_host(xs)
    for got in (b0.finish(), b1.finish()):
        for w, g in zip(want, got):
            assert np.array_equal(w["assignment"], g["assignment"]) and w["counts"] == g["counts"]
            assert np.array_equal(w["state"][:8], g["state"][:8])
    b0.load_device(xs)
    b0.run()
    for w, g in zip(want, b0.collect()):
        assert np.array_equal(w["assignment"], g["assignment"]) and w["counts"] == g["counts"]


def test_reconstruct_from_saved_assignment_and_sweep_csv(qa, tmp_path):
    """reconstruct.py (scripts/reconstruct_mixed_tile_assignment.py) and the sweep CSV writer on a golden case."""
    import json
    from quantization_analysis_b200 import reconstruct, sweep, wq
    x = G.algo_input("het_256x512")
    rng = np.random.default_rng(3)
    p_th, p_tw = x.shape[0] // 32, x.shape[1] // 32
    a = rng.integers(0, 4, size=(p_th, p_tw)).astype(np.int8)
    wq.write_assignment(tmp_path, "mixed_tile_greedy", "t.weight", a)
    d = tmp_path / "mixed_tile_greedy" / wq._slug("t.weight")
    fm = reconstruct.load_mapping(d / "assignment_mapping.json")
    y = reconstruct.reconstruct_from_assignment(x, np.load(d / "assignment.npy"), fm)
    want = orc.apply_assignment(x, a)
    assert np.array_equal(y.view(np.uint32), want.view(np.uint32))
    # a permuted mapping names the same formats through different integers
    perm = ["bfp2", "bf16", "bfp4", "bfp8"]
    a2 = np.vectorize(lambda v: perm.index(list(G.MIXED)[v]))(a).astype(np.int8)
    y2 = reconstruct.reconstruct_from_assignment(x, a2, perm)
    assert np.array_equal(y2.view(np.uint32), want.view(np.uint32))
    with pytest.raises(ValueError):
        reconstruct.reconstruct_from_assignment(x, a[:-1], fm)
    rows, _maps = sweep.sweep_tensor(x, metric="pcc", steps=5, lowest=0.9)
    path = sweep.write_sweep_csv(tmp_path / "sweep", rows)
    lines = path.read_text().strip().splitlines()
    assert lines[0] == "step,threshold,size_bytes,pcc,mae,atol,bf16_tiles,bfp8_tiles,bfp4_tiles,bfp2_tiles"
    assert len(lines) == 6 and lines[1].split(",")[0] == "0"
    assert sum(int(v) for v in lines[3].split(",")[6:]) == p_th * p_tw


def test_scalar_proxies_match_reference_goldens_on_device(qa):
    """qa_scalar_proxy (mxfp4 / nvfp4) vs the reference on every bf16 pattern (bf16 and float32 inputs) and on 20 000
    random float32 values."""
    import torch
    from quantization_analysis_b200 import quantization_formats as qf
    z = G.npz("scalar_proxies.npz")
    u16 = np.arange(65536, dtype=np.uint32)
    x16 = (u16 << 16).view(np.float32)
    xb = torch.from_numpy(u16.astype(np.int32).astype(np.int16)).view(torch.bfloat16).cuda()
    xr = z["rand__in"].view(np.float32)
    for fmt in ("mxfp4", "nvfp4"):
        w16 = z[f"bf16__{fmt}"]
        nan = np.isnan(w16.view(np.float32))
        for got in (qf.quantize_weight_values(x16, fmt), qf.quantize_weight_values(xb, fmt).cpu().numpy()):
            assert got.dtype == np.float32
            assert np.array_equal(np.isnan(got), nan), fmt
            assert np.array_equal(got.view(np.uint32)[~nan], w16[~nan]), fmt
        gr = qf.quantize_weight_values(xr.reshape(100, 200), fmt)
        assert gr.shape == (100, 200)
        assert np.array_equal(gr.reshape(-1).view(np.uint32), z[f"rand__{fmt}"]), fmt
    assert qf.quantize_weight_values(np.zeros((0, 4), np.float32), "mxfp4").shape == (0, 4)


def test_none_compression_with_wq_default_formats(qa):
    """NoneCompression over wq's default format list (mxfp4, nvfp4 first: hf_model_utils.py:317-319) vs the oracle."""
    from quantization_analysis_b200 import compression_algorithms as ca
    x = G.algo_input("het_256x512")
    fmts = ["mxfp4", "nvfp4", "bf16", "bfp8", "bfp4", "bfp2", "fp0"]
    res = ca.create_algorithm("none", {}).run(x, fmts, None, None)
    assert [r.fmt for r in res] == [f.upper() for f in fmts]
    for r, f in zip(res, fmts):
        with np.errstate(all="ignore"):
            want = orc.quantize(x, f)
        assert np.array_equal(np.asarray(r.y, dtype=np.float32).view(np.uint32), want.view(np.uint32)), f


def test_fp8_block_dequant_matches_reference_goldens_on_device(qa):
    """qa_fp8_block_dequant vs hf_model_utils._dequantize_tensor_with_scale_inv (goldens through torch's float8_e4m3fn):
    float32 products bit-equal, bf16 patterns = RNE of them, inexact count = products with non-zero low bits."""
    import torch
    eng = qa["engine"]
    z = G.npz("fp8_dequant.npz")
    for tag in ("all", "rag"):
        w, s = z[f"{tag}__w"], z[f"{tag}__s"]
        out, ob, cnt = eng.fp8_block_dequant(torch.from_numpy(w), torch.from_numpy(s))
        got = out.cpu().numpy()
        want = z[f"{tag}__out"].view(np.float32).reshape(got.shape)
        nan = np.isnan(want)
        assert np.array_equal(np.isnan(got), nan)
        assert np.array_equal(got.view(np.uint32)[~nan], want.view(np.uint32)[~nan]), tag
        fin = want[~nan]
        assert cnt == int(((want.view(np.uint32) & 0xFFFF) != 0).sum())
        assert np.array_equal(ob.float().cpu().numpy()[~nan].view(np.uint32), orc.bf16_round(fin).view(np.uint32))
    # a power-of-two scale keeps every product bf16-exact: the bf16 kernels apply
    w = z["rag__w"]
    out, ob, cnt = eng.fp8_block_dequant(torch.from_numpy(w).view(torch.float8_e4m3fn), torch.full((3, 5), 2.0 ** -7))
    assert cnt == 0 and torch.equal(ob.float(), out)


def test_batch_degenerate_inputs_match_oracle(qa):
    """The staged batch schedule (graph replay) on the degenerate tensors - den == 0 branches, all-zero tables, one tile,
    a non-zero mean, tiny values, ragged tiles - against the CPU oracle, for pcc and mae."""
    import torch
    from quantization_analysis_b200.batch import GreedyBatch
    rng = np.random.default_rng(3)
    xs = [np.full((96, 128), 0.25, dtype=np.float32), np.zeros((64, 96), dtype=np.float32),
          (rng.standard_normal((32, 32)) * 0.02).astype(np.float32),
          (1.0 + rng.standard_normal((256, 384)) * 0.01).astype(np.float32),
          (rng.standard_normal((128, 256)) * 1e-30).astype(np.float32),
          (rng.standard_normal((130, 75)) * 0.02).astype(np.float32)]
    xs = [torch.from_numpy(x).to(torch.bfloat16) for x in xs]
    shapes = [tuple(x.shape) for x in xs]
    for metric, thr in (("pcc", 0.999), ("pcc", 0.9), ("mae", 1e-4)):
        b = GreedyBatch(shapes, metric=metric, threshold=thr, seed=5)
        b.load_device(xs)
        b.run_graph()
        for x, r in zip(xs, b.collect()):
            xf = x.float().numpy()
            want, counts = orc.greedy_assign(orc.tile_stat_table(xf), list(G.MIXED), metric, thr, 5)
            assert np.array_equal(r["assignment"], want), (metric, thr, xf.shape)
            assert r["counts"] == counts


def test_greedy_assign_staged_single_tensor_equals_inline(qa):
    """engine.greedy_assign_staged (side-stream prefetch + init + chain by pass range for ONE tensor - what
    MixedTileGreedyCompression.run uses) == engine.greedy_assign, including the stream position."""
    import torch
    eng = qa["engine"]
    x = G.algo_input("het_256x512")
    p = eng.prepare_tiles(x)
    for metric, thr, fmts in (("pcc", 0.995, list(G.MIXED)), ("mae", 3e-4, list(G.MIXED)), ("pcc", 0.9999, ["bfp4", "bfp2"]),
                              ("pcc", 0.99999, list(G.MIXED)), ("atol", 2e-3, list(G.MIXED))):
        table = eng.tile_stats(p, G.MIXED, exact_abs=True)
        r1, r2 = eng.make_rng(31), eng.make_rng(31)
        a1, c1, s1 = eng.greedy_assign(table, p.numel, metric, thr, fmts, r1)
        for _ in range(2):                                   # twice: the side streams are reused
            r2 = eng.make_rng(31)
            a2, c2, s2 = eng.greedy_assign_staged(table, p.numel, metric, thr, fmts, r2)
            torch.cuda.synchronize()
            assert torch.equal(a1, a2) and torch.equal(c1, c2) and torch.equal(r1, r2), (metric, thr, fmts)
            assert torch.equal(s1[:8], s2[:8])


def test_greedy_batch_perm_cache_gives_the_same_maps(qa):
    """GreedyBatch(perm_cache=True): permutations drawn once per (seed, tile count) for the process and shared by every
    step / list == the per-step prefetch == the oracle; eager, graph replay and end-to-end forms."""
    from quantization_analysis_b200 import synthetic
    from quantization_analysis_b200.batch import GreedyBatch
    shapes = [(256, 512), (96, 320), (256, 512), (64, 64)]
    xs = [synthetic.randn_bf16_cpu(s, 30 + i) for i, s in enumerate(shapes)]
    want = []
    for xb in xs:
        xf = xb.float().numpy()
        want.append(orc.greedy_assign(orc.tile_stat_table(xf), list(G.MIXED), "pcc", 0.999, 77))
    for cache in (False, True, True):          # the second cached batch starts from a warm process-wide cache
        b = GreedyBatch(shapes, metric="pcc", threshold=0.999, seed=77, perm_cache=cache)
        b.load_device(xs)
        b.run()
        eager = b.collect()
        b.run_graph()
        b.run_graph()
        graph = b.collect()
        e2e = b.run_from_host([x.pin_memory() for x in xs])
        for res in (eager, graph, e2e):
            for r, (a, c) in zip(res, want):
                assert np.array_equal(r["assignment"], a) and r["counts"] == c, cache
    two = GreedyBatch(shapes[:2], metric="mae", threshold=3e-4, seed=5, tile_formats=["bfp8", "bfp4"], perm_cache=True)
    two.load_device(xs[:2])
    two.run_graph()
    for r, xb in zip(two.collect(), xs[:2]):
        a, c = orc.greedy_assign(orc.tile_stat_table(xb.float().numpy()), ["bfp8", "bfp4"], "mae", 3e-4, 5)
        assert np.array_equal(r["assignment"], a) and r["counts"] == c


def test_greedy_certificate_margin_and_forced_fallback(qa):
    """state[20]: lower bound of the smallest relative distance between a decision and the threshold.  A threshold that
    equals the value reached at some accepted step makes that distance exactly 0: the certified plug-in must notice, redo
    the tensor in reference order (NumPy-order tile sums + one-thread chain), and still return the reference's map."""
    ca, eng = qa["ca"], qa["engine"]
    x = G.algo_input("het_256x512")
    table_o = orc.tile_stat_table(x)
    a0 = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.995, "seed": 3})
    dr = a0.run_prepared(eng.prepare_tiles(x), list(G.MIXED))
    cert = dr.meta["certificate"]
    assert cert["fallback"] is False and cert["min_margin"] > 2e-13 and cert["min_margin"] < 1e-2
    want, wc = orc.greedy_assign(table_o, list(G.MIXED), "pcc", 0.995, 3)
    assert np.array_equal(dr.assignment_numpy(), want)
    # the final state's value is one the chain accepted: use it as the threshold itself
    tie = float(dr.meta["state"].cpu().numpy()[7])
    a1 = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": tie, "seed": 3})
    dr1 = a1.run_prepared(eng.prepare_tiles(x), list(G.MIXED))
    assert dr1.meta["certificate"]["min_margin"] < 2e-13 and dr1.meta["certificate"]["fallback"] is True
    want1, wc1 = orc.greedy_assign(table_o, list(G.MIXED), "pcc", tie, 3)
    assert np.array_equal(dr1.assignment_numpy(), want1) and dr1.counts == wc1
    # certify=False keeps the fast result (and still reports the margin)
    a2 = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": tie, "seed": 3, "certify": False})
    dr2 = a2.run_prepared(eng.prepare_tiles(x), list(G.MIXED))
    assert dr2.meta["certificate"]["fallback"] is False and dr2.meta["certificate"]["min_margin"] < 2e-13
    # the batch reports the same certificate inputs per tensor
    from quantization_analysis_b200.batch import GreedyBatch
    xb = torch.from_numpy(x).to(torch.bfloat16)
    b = GreedyBatch([x.shape], metric="pcc", threshold=0.995, seed=3)
    b.load_device([xb])
    b.run()
    r = b.collect()[0]
    assert np.array_equal(r["assignment"], want) and r["min_margin"] == cert["min_margin"] and r["flags"] == cert["flags"]


def _check_f32_fast_table(got, want, tag, exact=True):
    """qa_tile_stats_f32 / qa_tile_stats_fp8 against the NumPy-order oracle: sums of exactly representable terms are bit-equal;
    sum x, sum x^2 and sum x*y of 24-bit data round differently in another order (held to 1e-13 relative, a few ulp).
    exact=False: a tensor whose tiles span ~40 octaves - no float64 tile sum is exactly representable, all are order-dependent."""
    for k in ("sx", "sx2"):
        assert np.allclose(got[k], want[k], rtol=1e-13, atol=0, equal_nan=True), (tag, k)
    for f in G.MIXED:
        for k in ("sy", "sy2", "sabs", "amax"):
            if exact or k == "amax":
                assert np.array_equal(got[f][k], want[f][k], equal_nan=True), (tag, f, k)
            else:
                assert np.allclose(got[f][k], want[f][k], rtol=1e-13, atol=1e-300, equal_nan=True), (tag, f, k)
        assert np.allclose(got[f]["sxy"], want[f]["sxy"], rtol=1e-13, atol=0, equal_nan=True), (tag, f)


def test_fast_tile_stats_for_float32_inputs(qa):
    """The fast tile-stat kernel for inputs that are not bf16-exact (24-bit significands: the alignment shift truncates before the
    round, products are float32 arrays) on normal, heavy-tailed, tiny, denormal-bearing, ragged and 1-D tensors."""
    eng = qa["engine"]
    rng = np.random.default_rng(23)
    cases = {
        "normal": (rng.standard_normal((96, 200)) * 0.02).astype(np.float32),
        "heavy": (rng.standard_t(2, (64, 544)) * 0.05).astype(np.float32),
        "ragged": rng.standard_normal((45, 77)).astype(np.float32),
        "vector": rng.standard_normal(1000).astype(np.float32),
        "tiny": (rng.standard_normal((32, 64)) * 1e-22).astype(np.float32),
        "wide": (rng.standard_normal((64, 64)) * np.exp2(rng.integers(-30, 10, (64, 64)))).astype(np.float32),
    }
    cases["normal"][5, 7] = 0.0
    cases["wide"][3, :16] = 0.0
    cases["wide"][4, 16:32] = np.float32(1e-41)          # a denormal-only group
    cases["wide"][9, 40] = np.float32(3e-39)
    for tag, x in cases.items():
        p = eng.prepare_tiles(x)
        assert p.dtype_code == 1, tag
        want = orc.tile_stat_table(x)
        for exact_abs in (True, False):
            got = _table_from_device(eng.tile_stats(p, G.MIXED, exact_abs=exact_abs), None)
            if not exact_abs:            # fp32 group partials of sum |x-y|: close, not exact
                for f in G.MIXED:
                    assert np.allclose(got[f]["sabs"], want[f]["sabs"], rtol=1e-6, atol=0), (tag, f)
                    got[f]["sabs"] = want[f]["sabs"]
            _check_f32_fast_table(got, want, tag, exact=(tag != "wide"))
        # piecewise production of the same table
        if p.tiles_h >= 2:
            whole = eng.tile_stats(p, G.MIXED)
            from quantization_analysis_b200 import _lib
            t2 = torch.zeros_like(whole)
            for lo, hi in ((0, 1), (1, p.tiles_h)):
                _lib.check(_lib.lib().qa_tile_stats_f32(p.data.data_ptr(), p.rows, p.cols, p.cols, 0xF, 0, t2.data_ptr(), lo, hi,
                                                        torch.cuda.current_stream().cuda_stream), "qa_tile_stats_f32")
            assert torch.equal(whole, t2), tag


def test_fp8_fused_tile_stats_and_greedy(qa):
    """qa_tile_stats_fp8 (e4m3fn bytes + block scales in, table out) == the float32 kernel on the dequantized tensor, bit for
    bit, and == the oracle on the reference's dequantization goldens; the greedy map from the fused table is the oracle's."""
    eng, ca = qa["engine"], qa["ca"]
    z = G.npz("fp8_dequant.npz")
    w, s = z["rag__w"], z["rag__s"]                       # 300 x 520 with 100 x 104 blocks: groups straddle scale blocks
    xf = z["rag__out"].view(np.float32).reshape(w.shape)
    table, cnt = eng.tile_stats_fp8(torch.from_numpy(w), torch.from_numpy(s))
    assert int(cnt.item()) == int(((xf.view(np.uint32) & 0xFFFF) != 0).sum())
    p = eng.prepare_tiles(xf)
    if p.dtype_code == 1:
        assert torch.equal(table.nan_to_num(nan=-1.0), eng.tile_stats(p, G.MIXED).nan_to_num(nan=-1.0))
    with np.errstate(all="ignore"):
        want = orc.tile_stat_table(xf)
    # uniformly random bytes span all 17 octaves of e4m3 inside a tile: no float64 tile sum is exactly representable
    _check_f32_fast_table(_table_from_device(table, None), want, "rag", exact=False)
    # a checkpoint-like tensor: randn * 0.02 quantized per 128 x 128 block to e4m3fn (amax / 448 inverse scales)
    from quantization_analysis_b200 import synthetic
    rng = np.random.default_rng(5)
    wt, sct = synthetic.fp8_checkpoint_cpu((512, 1024), 5)
    w, sc = wt.numpy(), sct.numpy()
    out, _, bad = eng.fp8_block_dequant(torch.from_numpy(w), torch.from_numpy(sc), want_bf16=False)
    assert bad > 0
    x = out.cpu().numpy()
    table, _ = eng.tile_stats_fp8(torch.from_numpy(w), torch.from_numpy(sc), exact_abs=False)
    want = orc.tile_stat_table(x)
    got = _table_from_device(table, None)
    for f in G.MIXED:
        assert np.allclose(got[f]["sabs"], want[f]["sabs"], rtol=1e-6, atol=0)
        got[f]["sabs"] = want[f]["sabs"]
    _check_f32_fast_table(got, want, "ckpt")
    algo = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 9})
    dr = algo.run_fp8_blocks(torch.from_numpy(w), torch.from_numpy(sc), list(G.MIXED))
    a, counts = orc.greedy_assign(want, list(G.MIXED), "pcc", 0.999, 9)
    assert np.array_equal(dr.assignment_numpy(), a) and dr.counts == counts
    assert dr.meta["certificate"]["fallback"] is False
    assert np.array_equal(G.bits(eng.result_to_numpy(dr.prepared, dr.y_device())), G.bits(orc.apply_assignment(x, a)))
    # the batched schedule on fp8 sources (graph replay and the host -> device form): same maps
    from quantization_analysis_b200.batch import GreedyBatch
    w2 = rng.integers(0, 256, (1100, 2048), dtype=np.uint8)        # 35 x 64 tiles: the pipelined three-range table
    w2[(w2 & 0x7F) == 0x7F] = 0x3C
    sc2 = np.exp(rng.uniform(np.log(1e-4), np.log(3e-3), (9, 16))).astype(np.float32)
    srcs = [(torch.from_numpy(w), torch.from_numpy(sc)), (torch.from_numpy(w2), torch.from_numpy(sc2))]
    b = GreedyBatch([(512, 1024), (1100, 2048)], metric="pcc", threshold=0.999, seed=9, source="fp8", perm_cache=True)
    b.PIPELINE_MIN_TILES = 2048
    b.load_device(srcs)
    b.run_graph()
    res = b.collect()
    x2 = eng.fp8_block_dequant(*srcs[1], want_bf16=False)[0].cpu().numpy()
    a2, c2 = orc.greedy_assign(orc.tile_stat_table(x2), list(G.MIXED), "pcc", 0.999, 9)
    assert np.array_equal(res[0]["assignment"], a) and res[0]["counts"] == counts
    assert np.array_equal(res[1]["assignment"], a2) and res[1]["counts"] == c2
    assert b.input_bytes() == 512 * 1024 + 1100 * 2048 + 4 * (4 * 8 + 9 * 16)
    pinned = [(t.pin_memory(), s_.pin_memory()) for t, s_ in srcs]
    res = b.run_from_host(pinned)
    assert np.array_equal(res[1]["assignment"], a2) and res[0]["counts"] == counts


def test_descriptor_array_batch_equals_per_tensor_calls(qa):
    """qa_tile_stats_batch / qa_greedy_init_deltas_batch (one launch for a list of tensors, SURVEY 8(b)(8)) fill the same bits as
    one call per tensor - incl. a ragged tensor that takes the scalar-load path - and GreedyBatch with grouped launches gives
    the maps of the per-tensor schedule."""
    from quantization_analysis_b200 import _lib, synthetic
    from quantization_analysis_b200.batch import GreedyBatch
    eng = qa["engine"]
    L = _lib.lib()
    shapes = [(256, 1024), (96, 320), (45, 77), (512, 512), (64, 2048)]
    xs = [synthetic.randn_bf16_cpu(s, 40 + i).cuda() for i, s in enumerate(shapes)]
    preps = [eng.prepare_tiles(x) for x in xs]
    want = [eng.tile_stats(p, G.MIXED, exact_abs=False) for p in preps]
    tables = [torch.zeros_like(t) for t in want]
    inits = [torch.zeros(L.qa_greedy_init_bytes(p.ntiles), dtype=torch.uint8, device="cuda") for p in preps]
    descs, n, items, blocks = eng.batch_descriptors(
        [(p.data.data_ptr(), t.data_ptr(), i_.data_ptr(), p.rows, p.cols) for p, t, i_ in zip(preps, tables, inits)], torch.device("cuda"))
    assert items == sum(L.qa_tile_stats_items(p.rows, p.cols) for p in preps)
    eng.tile_stats_batch(descs, n, items, G.MIXED, exact_abs=False)
    for t, w in zip(tables, want):
        assert torch.equal(t, w)
    order = _lib.int32_array([0, 1, 2, 3])
    sp = torch.cuda.current_stream().cuda_stream
    _lib.check(L.qa_greedy_init_deltas_batch(descs.data_ptr(), n, blocks, order, 4, sp), "qa_greedy_init_deltas_batch")
    for p, t, i_ in zip(preps, want, inits):
        ref = torch.zeros_like(i_)
        _lib.check(L.qa_greedy_init_deltas(t.data_ptr(), p.ntiles, 0, order, 4, ref.data_ptr(), sp), "qa_greedy_init_deltas")
        assert torch.equal(i_[256:], ref[256:])            # the delta records (behind the 256-byte header the sums kernel writes)
    vshapes = [s for s in shapes if s != (45, 77)]
    vx = [x for x, s in zip(xs, shapes) if s != (45, 77)]
    for metric, thr in (("pcc", 0.999), ("mae", 3e-4), ("atol", 2e-3)):
        a = GreedyBatch(vshapes, metric=metric, threshold=thr, seed=7, stats_group=0)
        b = GreedyBatch(vshapes, metric=metric, threshold=thr, seed=7, stats_group=3)
        for bb in (a, b):
            bb.load_device(vx)
            bb.run_graph()
        for ra, rb in zip(a.collect(), b.collect()):
            assert np.array_equal(ra["assignment"], rb["assignment"]) and ra["counts"] == rb["counts"], metric
            assert ra["metrics"] == rb["metrics"], metric
