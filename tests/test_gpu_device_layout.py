"""The mixed-tile algorithms in the device layout (``"transpose": true``): a run on x equals the reference algorithm on
xt = x.T - map over xt's tiles, counts, tile_bytes, per-tile scores, random samples and selection - with y = yt.T in x's
shape, and float32 whole-tensor scores of x against y in x's layout.  Expected values come from the NumPy oracle on
np.ascontiguousarray(x.T); the greedy's chain state and certificate margin, which the oracle does not have, from this
package's unflagged run on x.T.  Inputs: bf16-exact, float32 that is not bf16-exact, and fp8 e4m3fn bytes with block scales
(ragged blocks included)."""
import numpy as np
import pytest
import torch

from oracle import qa_oracle as orc
from quantization_analysis_b200 import engine, sweep
from quantization_analysis_b200 import compression_algorithms as ca
from quantization_analysis_b200 import synthetic
from quantization_analysis_b200.tensor_source import Fp8Blocks
from tests import golden_util as G

# the chain state's deterministic entries (the others of the cluster chain are cycle counters)
STATE_DET = [0, 1, 2, 3, 4, 5, 6, 7, 11, 12, 19, 20]
ORDERS = [["bf16", "bfp8", "bfp4", "bfp2"], ["bfp8", "bfp4", "bfp2"], ["bfp8", "bfp2"], ["bfp4"]]


def _bf16_exact(shape, seed):
    return synthetic.heterogeneous_f32_np(shape, seed)


def _f32(shape, seed):
    x = (np.random.default_rng(seed).standard_normal(shape) * 0.02).astype(np.float32)
    assert not np.array_equal(torch.from_numpy(x).to(torch.bfloat16).float().numpy(), x)
    return x


def _fp8(shape, seed, block=(128, 128)):
    """-> (Fp8Blocks, its float32 dequantization as the reference computes it)."""
    w, inv = synthetic.fp8_checkpoint_cpu(shape, seed, block=block)
    src = Fp8Blocks(w.view(torch.float8_e4m3fn), inv)
    return src, orc.fp8_block_dequant(w.numpy(), inv.numpy())


def _inputs():
    return {"bf16_70x45": lambda: (_bf16_exact((70, 45), 22),) * 2,
            "bf16_96x160": lambda: (_bf16_exact((96, 160), 21),) * 2,
            "f32_70x45": lambda: (_f32((70, 45), 5),) * 2,
            "f32_96x160": lambda: (_f32((96, 160), 6),) * 2,
            "fp8_300x520": lambda: _fp8((300, 520), 7)}


def _xt(x):
    return np.ascontiguousarray(np.asarray(x, dtype=np.float32).T)


def _metric_threshold(xt, metric):
    if metric == "pcc":
        return 0.999
    d4 = np.abs(xt - orc.quantize(xt, "bfp4"))
    return float(np.mean(d4)) * 0.6 if metric == "mae" else float(np.max(d4)) * 0.5


def _check_scores(dr, x, y):
    want = orc.wq_scores(x, y)
    got = dr.metrics
    for k in ("pcc", "mae", "atol"):
        assert np.float32(got[k]) == np.float32(want[k]), (k, got[k], want[k])


def _unflagged(params):
    return {k: v for k, v in params.items() if k != "transpose"}


# ------------------------------------------------------------------------------------------------------------------------
# greedy
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_inputs()))
@pytest.mark.parametrize("metric", ["pcc", "mae", "atol"])
def test_greedy_transposed_equals_oracle_on_xt(case, metric):
    src, x = _inputs()[case]()
    xt = _xt(x)
    table = orc.tile_stat_table(xt)
    thr = _metric_threshold(xt, metric)
    for fmts in ORDERS:
        params = {"metric": metric, "threshold": thr, "seed": 11, "formats": fmts, "transpose": True}
        alg = ca.create_algorithm("mixed-tile-greedy", params)
        dr = alg.run_prepared(engine.prepare_transposed(src), fmts)
        want, wc = orc.greedy_assign(table, fmts, metric, thr, 11)
        assert dr.transposed and dr.assignment_numpy().shape == (-(-x.shape[1] // 32), -(-x.shape[0] // 32))
        assert np.array_equal(dr.assignment_numpy(), want), fmts
        assert dr.counts == wc and dr.tile_bytes == orc.total_bytes(wc)
        y = orc.apply_assignment(xt, want).T
        got_y = dr.y_device().to(torch.float32).cpu().numpy().reshape(x.shape)
        assert np.array_equal(G.bits(got_y), G.bits(y))
        _check_scores(dr, x, y)
        # chain state and certificate: the unflagged device run on x.T
        ref = ca.create_algorithm("mixed-tile-greedy", _unflagged(params)).run_prepared(engine.prepare_loaded(
            Fp8Blocks(torch.from_numpy(np.ascontiguousarray(src.weight.view(torch.uint8).numpy().T)).view(torch.float8_e4m3fn),
                      torch.from_numpy(np.ascontiguousarray(src.scale_inv.numpy().T)))
            if isinstance(src, Fp8Blocks) else xt), fmts)
        idx = STATE_DET if metric != "atol" and not ref.meta["certificate"]["fallback"] else list(range(24))
        assert np.array_equal(np.nan_to_num(dr.meta["state"].cpu().numpy()[idx], nan=-7.0),
                              np.nan_to_num(ref.meta["state"].cpu().numpy()[idx], nan=-7.0))
        assert dr.meta["certificate"] == ref.meta["certificate"]
        assert dr.metrics_exact == ref.metrics_exact


@pytest.mark.gpu
def test_greedy_run_and_fp8_blocks_entry_points():
    """`run` (host array in, y in x's shape) and `run_fp8_blocks` prepare x.T themselves."""
    x = _bf16_exact((96, 160), 21)
    xt = _xt(x)
    fmts = ORDERS[0]
    res = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.995, "seed": 4, "transpose": True}).run(
        x, fmts, None, None)[0]
    want, wc = orc.greedy_assign(orc.tile_stat_table(xt), fmts, "pcc", 0.995, 4)
    assert np.array_equal(res.meta["assignment"], want) and res.tile_counts == wc
    assert res.y.shape == x.shape and np.array_equal(G.bits(res.y), G.bits(orc.apply_assignment(xt, want).T))
    # torch input: y comes back as a device tensor of x's shape
    rt = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.995, "seed": 4, "transpose": True}).run(
        torch.from_numpy(x), fmts, None, None)[0]
    assert tuple(rt.y.shape) == x.shape and np.array_equal(G.bits(rt.y.float().cpu().numpy()), G.bits(res.y))
    src, xf = _fp8((300, 520), 7)
    alg = ca.create_algorithm("mixed-tile-greedy", {"metric": "mae", "threshold": 3e-4, "seed": 9, "transpose": True})
    dr = alg.run_fp8_blocks(src.weight, src.scale_inv, fmts)
    want, wc = orc.greedy_assign(orc.tile_stat_table(_xt(xf)), fmts, "mae", 3e-4, 9)
    assert np.array_equal(dr.assignment_numpy(), want) and dr.counts == wc
    assert np.array_equal(G.bits(dr.y_device().float().cpu().numpy().reshape(xf.shape)),
                          G.bits(orc.apply_assignment(_xt(xf), want).T))


@pytest.mark.gpu
def test_greedy_transposed_full_size_and_forced_fallback():
    """[1536, 7168] (the shape of q_a_proj) with pcc; then a threshold equal to a value the chain reached forces the
    certificate's fallback, which must still give the oracle's map on x.T."""
    x = synthetic.randn_bf16_cpu((1536, 7168), 13).float().numpy()
    xt = _xt(x)
    table = orc.tile_stat_table(xt)
    fmts = ORDERS[0]
    alg = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": 0.999, "seed": 3, "transpose": True})
    p = engine.prepare_transposed(x)
    dr = alg.run_prepared(p, fmts)
    want, wc = orc.greedy_assign(table, fmts, "pcc", 0.999, 3)
    assert dr.assignment_numpy().shape == (224, 48)
    assert np.array_equal(dr.assignment_numpy(), want) and dr.counts == wc
    y = orc.apply_assignment(xt, want).T
    assert np.array_equal(G.bits(dr.y_device().float().cpu().numpy().reshape(x.shape)), G.bits(y))
    _check_scores(dr, x, y)
    tie = float(dr.meta["state"].cpu().numpy()[7])
    dr1 = ca.create_algorithm("mixed-tile-greedy", {"metric": "pcc", "threshold": tie, "seed": 3, "transpose": True}).run_prepared(p, fmts)
    assert dr1.meta["certificate"]["fallback"] is True and dr1.meta["certificate"]["min_margin"] < 2e-13
    want1, wc1 = orc.greedy_assign(table, fmts, "pcc", tie, 3)
    assert np.array_equal(dr1.assignment_numpy(), want1) and dr1.counts == wc1


# ------------------------------------------------------------------------------------------------------------------------
# threshold and random
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_inputs()))
@pytest.mark.parametrize("metric", ["pcc", "mae", "atol"])
def test_threshold_transposed_equals_oracle_on_xt(case, metric):
    src, x = _inputs()[case]()
    xt = _xt(x)
    th, tw = -(-xt.shape[0] // 32), -(-xt.shape[1] // 32)
    thr = {"pcc": 0.99, "mae": _metric_threshold(xt, "mae"), "atol": _metric_threshold(xt, "atol")}[metric]
    for fmts in ORDERS:
        alg = ca.create_algorithm("mixed-tile-threshold", {"metric": metric, "threshold": thr, "formats": fmts, "transpose": True})
        dr = alg.run_prepared(engine.prepare_transposed(src), fmts)
        sc = orc.padded_tile_scores(xt, fmts, metric)
        row = {"pcc": 0, "mae": 1, "atol": 2}[metric]
        got_sc = dr.meta["scores"].cpu().numpy()
        for f in fmts:
            assert np.array_equal(got_sc[row, engine.FMT_INDEX[f]].view(np.uint32), sc[f].astype(np.float32).view(np.uint32)), f
        want, wc = orc.threshold_assign(sc, fmts, metric, thr, th, tw)
        assert np.array_equal(dr.assignment_numpy(), want) and dr.counts == wc and dr.tile_bytes == orc.total_bytes(wc)
        y = orc.apply_assignment(xt, want).T
        assert np.array_equal(G.bits(dr.y_device().float().cpu().numpy().reshape(x.shape)), G.bits(y))
        _check_scores(dr, x, y)


@pytest.mark.gpu
def test_threshold_transposed_full_size():
    x = synthetic.randn_bf16_cpu((1536, 7168), 14).float().numpy()
    xt = _xt(x)
    res = ca.create_algorithm("mixed-tile-threshold", {"metric": "pcc", "threshold": 0.999, "transpose": True}).run(
        x, ORDERS[0], None, None)[0]
    sc = orc.padded_tile_scores(xt, ORDERS[0], "pcc")
    want, wc = orc.threshold_assign(sc, ORDERS[0], "pcc", 0.999, 224, 48)
    assert np.array_equal(res.meta["assignment"], want) and res.tile_counts == wc
    assert np.array_equal(G.bits(res.y), G.bits(orc.apply_assignment(xt, want).T))


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(_inputs()))
def test_random_transposed_equals_oracle_on_xt(case):
    src, x = _inputs()[case]()
    xt = _xt(x)
    for fmts, metric in ((ORDERS[0], "pcc"), (ORDERS[1], "mae"), (ORDERS[2], "atol"), (ORDERS[3], "pcc")):
        thr = _metric_threshold(xt, metric) if metric != "pcc" else 0.99
        alg = ca.create_algorithm("mixed-tile-random", {"metric": metric, "threshold": thr, "iters": 5, "seed": 42, "formats": fmts,
                                                        "transpose": True})
        dr = alg.run_prepared(engine.prepare_transposed(src), fmts)
        want, wc, samples = orc.random_assign(xt, fmts, metric, thr, 5, 42)
        assert np.array_equal(dr.assignment_numpy(), want) and dr.counts == wc
        for got, exp in zip(dr.meta["samples"], samples, strict=True):
            assert got["counts"] == exp["counts"] and got["total_bytes"] == exp["total_bytes"]
            for k in ("pcc", "mae", "atol"):
                assert np.float32(got[k]) == np.float32(exp[k]), (k, got, exp)
        y = orc.apply_assignment(xt, want).T
        assert np.array_equal(G.bits(dr.y_device().float().cpu().numpy().reshape(x.shape)), G.bits(y))
        _check_scores(dr, x, y)


# ------------------------------------------------------------------------------------------------------------------------
# 0-D / 1-D / n-D, and the sweeps
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["mixed-tile-greedy", "mixed-tile-threshold", "mixed-tile-random"])
def test_vector_input_ignores_the_flag_and_3d_raises(algo):
    v = synthetic.heterogeneous_f32_np((1000,), 23)
    params = {"metric": "pcc", "threshold": 0.99, "seed": 5, "iters": 3}
    a = ca.create_algorithm(algo, {**params, "transpose": True}).run(v, G.MIXED, None, None)[0]
    b = ca.create_algorithm(algo, params).run(v, G.MIXED, None, None)[0]
    assert np.array_equal(a.meta["assignment"], b.meta["assignment"]) and a.tile_counts == b.tile_counts
    assert np.array_equal(G.bits(a.y), G.bits(b.y))
    with pytest.raises(ValueError, match=r"\(4, 40, 48\)"):
        ca.create_algorithm(algo, {**params, "transpose": True}).run(np.ones((4, 40, 48), np.float32), G.MIXED, None, None)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["bf16_96x160", "f32_70x45", "fp8_300x520"])
def test_sweeps_transposed_equal_unflagged_sweeps_of_xt(case):
    src, x = _inputs()[case]()
    xt_src = engine.prepare_transposed(src)           # the unflagged sweeps below run on this x.T as their input
    for metric, lowest in (("pcc", 0.9), ("mae", 0.01)):
        a, ma = sweep.sweep_tensor(src, G.MIXED, metric, 6, lowest, transpose=True)
        b, mb = sweep.sweep_tensor(xt_src, G.MIXED, metric, 6, lowest)
        assert a == b and torch.equal(ma, mb)
        fmts = ["bfp8", "bfp4", "bfp2"]
        a, ma = sweep.greedy_sweep_tensor(src, fmts, metric, 5, lowest if metric == "pcc" else 0.02, seed=8, transpose=True)
        b, mb = sweep.greedy_sweep_tensor(xt_src, fmts, metric, 5, lowest if metric == "pcc" else 0.02, seed=8)
        assert torch.equal(ma, mb)
        for ra, rb in zip(a, b, strict=True):
            sa, sb = ra.pop("state"), rb.pop("state")
            idx = STATE_DET if not ra["fallback"] else list(range(24))
            assert ra == rb and np.array_equal(np.nan_to_num(sa[idx], nan=-7.0), np.nan_to_num(sb[idx], nan=-7.0))
