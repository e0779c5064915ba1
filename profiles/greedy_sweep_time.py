"""Greedy sweep timing: one launch for every threshold's chain (qa_greedy_assign_sweep) against one qa_greedy_assign_passes call
per threshold on one stream, and the other parts of sweep.greedy_sweep_tensor.

Inputs: the o_proj tensor of bench.py's cfg2 workload (7168 x 16384 bf16, synthetic.randn_bf16_cpu seed 1004: 114 688 tiles)
and, separately, its fp8 e4m3fn + 128 x 128 block-scale form (synthetic.fp8_checkpoint_cpu, same seed).  K = 50 pcc thresholds
np.linspace(0.9999, 0.99, 50), formats bf16, bfp8, bfp4, bfp2, seed 123.  Every part is timed with CUDA events after a
warm-up, `--reps` times (min and median reported).  The 50 one-call-per-threshold chains reuse preallocated buffers and the
same shared init / prefetched permutations as the sweep, so the comparison is the chains alone.

    python profiles/greedy_sweep_time.py [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from quantization_analysis_b200 import _lib, engine, sweep, synthetic, tensor_source  # noqa: E402
from quantization_analysis_b200.batch import cached_permutations  # noqa: E402

FMTS = ["bf16", "bfp8", "bfp4", "bfp2"]
SEED = 123
SHAPE = (7168, 16384)


def timed(fn, reps):
    """-> (min ms, median ms, last result) of fn() between two events on the current stream."""
    out, ms = None, []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return min(ms), statistics.median(ms), out


def one_input(tag, x, thr, reps, say):
    L = _lib.lib()
    p = engine.prepare_loaded(x)
    k = len(thr)
    say(f"\n== {tag}: {p.rows} x {p.cols}, {p.ntiles} tiles, K = {k} pcc thresholds {thr[0]} .. {thr[-1]}")
    res = {}

    def row(name, fn):
        fn()                                                # warm-up
        lo, med, out = timed(fn, reps)
        say(f"  {name:<44s} min {lo:9.3f} ms   median {med:9.3f} ms")
        res[name] = out
        return out

    table = row("table pass (tile_stats, fast)", lambda: engine.tile_stats(p, engine.MIXED_FORMATS, exact_abs=False))
    init = row("init (delta records + initial sums)", lambda: engine.greedy_init(table, "pcc", FMTS))
    nt = table.shape[1]
    hit = cached_permutations(table.device, SEED, nt, len(FMTS))
    pre = (hit["pre_order"][:2], hit["rngs"][1:3])
    rng = engine.make_rng(SEED)
    maps_by_cap = {}
    for cap in (4, 8, 16):
        prev = L.qa_greedy_cluster_cap(cap)
        try:
            maps_by_cap[cap] = row(f"sweep launch, cluster cap {cap:2d} (one launch, K chains)",
                                   lambda: engine.greedy_sweep(table, p.numel, "pcc", thr, FMTS, rng, pre, init))[0]
        finally:
            L.qa_greedy_cluster_cap(prev)
    # today's route through the ABI: one qa_greedy_assign_passes call per threshold on one stream (automatic cluster size)
    dev = table.device
    maps = torch.empty((k, nt), dtype=torch.int8, device=dev)
    counts = torch.zeros((k, 4), dtype=torch.int64, device=dev)
    states = torch.zeros((k, 24), dtype=torch.float64, device=dev)
    rngs = torch.stack([rng] * k).contiguous()
    work = torch.empty(L.qa_greedy_par_work_bytes(nt), dtype=torch.uint8, device=dev)
    order = _lib.int32_array([engine.FMT_INDEX[f] for f in FMTS])

    def calls():
        rngs.copy_(rng.expand(k, -1))
        for i in range(k):
            _lib.check(L.qa_greedy_assign_passes(table.data_ptr(), nt, float(p.numel), 0, float(thr[i]), order, len(FMTS),
                                                 rngs[i].data_ptr(), maps[i].data_ptr(), counts[i].data_ptr(), states[i].data_ptr(),
                                                 work.data_ptr(), pre[0].data_ptr(), pre[1].data_ptr(), init.data_ptr(), 0,
                                                 len(FMTS), 0, engine._stream()), "qa_greedy_assign_passes")
        return maps
    row(f"{k} x qa_greedy_assign_passes, one stream", calls)
    for cap, m in maps_by_cap.items():
        assert torch.equal(m, maps), f"sweep at cap {cap} differs from the per-threshold calls"
    same = [False] + [bool(torch.equal(maps[i], maps[i - 1])) for i in range(1, k)]
    distinct = [i for i, s in enumerate(same) if not s]
    row(f"scoring of the {len(distinct)} distinct maps (_score_maps)", lambda: sweep._score_maps(p, maps, distinct))
    rows = row("greedy_sweep_tensor, highest = 0.9999",
               lambda: sweep.greedy_sweep_tensor(p, FMTS, "pcc", k, float(thr[-1]), highest=float(thr[0]), seed=SEED))[0]
    say(f"    fallbacks: {sum(r['fallback'] for r in rows)} of {len(rows)}; bytes {rows[0]['total_bytes']:.0f} .. "
        f"{rows[-1]['total_bytes']:.0f}")
    rows = row("greedy_sweep_tensor, default highest",
               lambda: sweep.greedy_sweep_tensor(p, FMTS, "pcc", k, float(thr[-1]), seed=SEED))[0]
    say(f"    default highest = {rows[0]['threshold']!r}; fallbacks: {sum(r['fallback'] for r in rows)} of {len(rows)} "
        f"(rows {[i for i, r in enumerate(rows) if r['fallback']]})")


def main(argv=None) -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    say(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {smi[0] if smi else 'n/a'}")
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}; CUDA events, {args.reps} timed repetitions after one warm-up")
    thr = np.linspace(0.9999, 0.99, 50)
    one_input("bf16", synthetic.randn_bf16_cpu(SHAPE, 1004).cuda(), thr, args.reps, say)
    w8, inv = synthetic.fp8_checkpoint_cpu(SHAPE, 1004)
    one_input("fp8 + 128x128 block scales", tensor_source.Fp8Blocks(w8.view(torch.float8_e4m3fn), inv), thr, args.reps, say)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
