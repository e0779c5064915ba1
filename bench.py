#!/usr/bin/env python3
"""Headline benchmark: bf16 weight GB/s quantized + scored (+ assigned) - BASELINE.json's metric.

Default workload (N = 1, BASELINE.json configs[1]): mixed-tile-greedy, metric pcc >= 0.999, seed 123, candidate formats
bf16/bfp8/bfp4/bfp2, over the five DeepSeek-R1 layer-0 self_attn weight shapes (187.1 M elements, 374 MB of bf16 - larger
than the 126 MB L2, so no flush is needed).  A step = one pass of the hot path over that tensor list: fused quantize +
tile statistics, greedy assignment and whole-tensor scoring, per tensor.  With N GPUs every rank runs the same shapes for
its own layer of the tensor list (weak scaling, no data-path collective; result rows are gathered to rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg1|cfg2|cfg3|cfg4|cfg5|cfg2-fp8]
                    [--dump-outputs DIR]

--config selects another of BASELINE.json's configs (same JSON contract; `config.workload` names it):
  cfg1  `none`, formats bf16/bfp8/bfp4/bfp2/fp0 on [1536,7168] (8 rotating buffers > L2), reconstructions + reference scores
  cfg3  threshold sweep, 32 thresholds, layer-0 attention + dense MLP shapes
  cfg4  mixed-tile-random, 1000 samples per tensor (reference float32 score of every sample), same 8 shapes
  cfg5  one MoE layer, 768 expert matrices (22.5 GB) bin-packed over the ranks: STRONG scaling
`--impl reference` times the UNMODIFIED reference (oracle/_ref, see oracle/make_ref.sh) on the host cores, on a bounded
sample of the same config.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

UNIT = "GB/s"
GREEDY = {"metric": "pcc", "threshold": 0.999, "seed": 123}
FORMATS5 = ["bf16", "bfp8", "bfp4", "bfp2", "fp0"]
INFLIGHT = int(os.environ.get("QA_BENCH_INFLIGHT", "12"))          # tensor lists in flight for the device-resident throughput
CFG5_INFLIGHT = int(os.environ.get("QA_BENCH_CFG5_INFLIGHT", "3"))      # cfg5: copies of the rank's shard in flight (22.5 GB / world each)
# cfg2: CTAs per chain cluster (0: automatic, up to 16).  Smaller clusters hold fewer SMs per tensor: the throughput schedule
# (profiles/r2_step_sweep3.txt: 12 lists x 4-CTA clusters 0.250 ms per step at 1.19 ms for a step alone; automatic clusters 0.265 ms
# at 0.52 ms).  The line reports the latter as `latency_schedule`.
CLUSTER_CAP = int(os.environ.get("QA_BENCH_CLUSTER_CAP", "4"))
TABLE_BYTES_PER_TILE = 22 * 8
METRICS = {
    "cfg1": "bf16 weight GB/s quantized+scored (none: bf16/bfp8/bfp4/bfp2/fp0 on q_a_proj [1536,7168])",
    "cfg2": "bf16 weight GB/s quantized+scored (mixed-tile-greedy pcc>=0.999, DeepSeek-R1 layer-0 self_attn shapes)",
    "cfg3": "bf16 weight GB/s quantized+scored (mixed-tile-threshold sweep, 32 thresholds, layer-0 attention + dense MLP shapes)",
    "cfg4": "bf16 weight GB/s quantized+scored (mixed-tile-random, 1000 samples per tensor, layer-0 attention + dense MLP shapes)",
    "cfg5": "bf16 weight GB/s quantized+scored (mixed-tile-greedy pcc>=0.999, one MoE layer: 256 experts x gate/up/down)",
    "cfg2-fp8": "bf16-equivalent weight GB/s quantized+scored (cfg2's tensor list stored as fp8 e4m3fn + 128x128 block scales, "
                "dequantization fused into the tile-stat read)",
}


def workload(rank: int):
    from quantization_analysis_b200 import synthetic
    return [(n.replace("layers.0", f"layers.{rank}"), synthetic.DEEPSEEK_R1_SHAPES[n], 1000 * (rank + 1) + i)
            for i, n in enumerate(synthetic.ATTN_NAMES)]


# --------------------------------------------------------------------------------------------
# clocks sampler (NVML)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int, enabled: bool = True):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        self.nv = None
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.004)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)

    def summary(self) -> dict:
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# --------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the UNMODIFIED reference (oracle/_ref) on host cores; the oracle port only if that is absent
# --------------------------------------------------------------------------------------------
REF_DIR = ROOT / "oracle" / "_ref"
CPU_SAMPLES = {      # (shape, synthetic seed) per config: a bounded part of the workload
    "cfg1": [((1536, 7168), 0)],
    "cfg2": [((576, 7168), 1002), ((1536, 7168), 1000)],       # kv_a_proj + q_a_proj of the tensor list
    "cfg3": [((576, 7168), 1002)],
    "cfg4": [((576, 7168), 1002)],
    "cfg5": [((2048, 7168), 50)],                                # one expert's gate_proj
}
CFG4_CPU_ITERS = 8


def _cpu_one(args):
    """One sample tensor through the reference's own code path for the config.  -> (seconds, elements, kind)."""
    cfg, shape, seed = args
    import numpy as np
    from quantization_analysis_b200 import synthetic
    x = synthetic.randn_f32_np(shape, seed)
    kind = "reference"
    if (REF_DIR / "compression_algorithms").is_dir():
        sys.path.insert(0, str(REF_DIR))
        sys.path.insert(0, str(REF_DIR / "scripts"))
        from compression_algorithms import create_algorithm          # the reference's modules (unmodified copies)
        from compression_algorithms.metrics import pearson_corr
        from compression_algorithms.quantizer import Quantizer
        q = Quantizer(backend="emulation")

        def score(y):                                                 # wq:684-687
            d = np.abs(x - y)
            return float(np.mean(d)), float(np.max(d)), pearson_corr(x, y)

        class _NoCache:
            def load_array(self, *a):
                return None

            def save_array(self, *a):
                return None

        t0 = time.perf_counter()
        if cfg == "cfg1":
            for r in create_algorithm("none", {}).run(xf=x, formats=FORMATS5, quantizer=q, cache=_NoCache()):
                score(r.y)
        elif cfg in ("cfg2", "cfg5"):
            r = create_algorithm("mixed-tile-greedy", dict(GREEDY)).run(xf=x, formats=FORMATS5, quantizer=q, cache=None)[0]
            score(r.y)
        elif cfg == "cfg3":
            import sweep_mixed_tile_threshold as sw                   # the reference's script: its sweep core, inline
            from compression_algorithms.tile_utils import (MIXED_TILE_BYTES_PER_ELEM, reconstruct_from_tiles,
                                                           reshape_to_2d_with_padding, tile_metrics)
            fm = ["bf16", "bfp8", "bfp4", "bfp2"]
            padded, si, pi = reshape_to_2d_with_padding(x)
            th, tw = pi[2] // 32, pi[3] // 32
            tiles = lambda a: a.reshape(th, 32, tw, 32).transpose(0, 2, 1, 3).reshape(-1, 32, 32)     # noqa: E731
            tr = tiles(padded)
            tq = {f: tiles(reshape_to_2d_with_padding(q.quantize(x, f))[0]) for f in fm}
            sc = {f: tile_metrics(tr, tq[f], "pcc") for f in fm}
            order = sorted(fm, key=lambda f: MIXED_TILE_BYTES_PER_ELEM[f])
            ss, ts = np.stack([sc[f] for f in order]), np.stack([tq[f] for f in order])
            last = None
            for thr in np.linspace(float(np.max(sc["bf16"])), 0.9, 32):
                a = sw._compute_assignment(ss, "pcc", float(thr))
                if last is None or not np.array_equal(a, last):
                    score(reconstruct_from_tiles(ts[a, np.arange(a.size)], si, pi))
                    last = a
        elif cfg == "cfg4":
            p = dict(metric="pcc", threshold=0.99, iters=CFG4_CPU_ITERS, seed=42)
            r = create_algorithm("mixed-tile-random", p).run(xf=x, formats=FORMATS5, quantizer=q, cache=None)[0]
            score(r.y)
        dt = time.perf_counter() - t0
    else:
        kind = "port"
        from oracle import qa_oracle as orc
        t0 = time.perf_counter()
        table = orc.tile_stat_table(x)
        a, _c = orc.greedy_assign(table, list(orc.MIXED_FORMATS), GREEDY["metric"], GREEDY["threshold"], GREEDY["seed"])
        orc.wq_scores(x, orc.apply_assignment(x, a))
        dt = time.perf_counter() - t0
    return dt, int(np.prod(shape)), kind


def cpu_sample_run(cfg: str, procs: int):
    """Time the bounded CPU sample on `procs` host processes (the reference is single-threaded NumPy: one tensor per
    process, the sample shapes alternating with different seeds until every core has one).  -> (aggregate GB/s of bf16
    weights, processes, wall seconds, kind)."""
    import multiprocessing as mp
    samples = CPU_SAMPLES[cfg]
    tasks = [(cfg, samples[i % len(samples)][0], samples[i % len(samples)][1] + 7 * (i // len(samples)))
             for i in range(max(procs, 1) if procs > 1 else len(samples))]
    t0 = time.perf_counter()
    if procs > 1:
        os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")      # one core per process: no oversubscription by np.dot
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        with mp.get_context("spawn").Pool(procs) as pool:        # spawn: a parent that ran torch has live OpenMP threads
            res = pool.map(_cpu_one, tasks, chunksize=1)
    else:
        res = [_cpu_one(a) for a in tasks]
    wall = time.perf_counter() - t0
    elems = sum(r[1] for r in res)
    compute = max(r[0] for r in res) if procs > 1 else sum(r[0] for r in res)
    scale = 1000.0 / CFG4_CPU_ITERS if cfg == "cfg4" else 1.0   # cfg4: 8 of the 1000 iterations timed, linear in iterations
    return 2.0 * elems / (compute * scale) / 1e9, (procs if procs > 1 else 1), wall, res[0][2]


def cpu_sample_desc(cfg: str, kind: str) -> str:
    what = {"cfg1": "NoneCompression.run (5 formats) + wq:684-687 scoring on q_a_proj [1536,7168]",
            "cfg2": "MixedTileGreedyCompression.run (pcc>=0.999, seed 123) + wq:684-687 scoring on kv_a_proj [576,7168] and q_a_proj "
                    "[1536,7168] of the tensor list",
            "cfg3": "sweep core (scripts/sweep_mixed_tile_threshold.py:623-790, 32 thresholds, pcc) on kv_a_proj [576,7168]",
            "cfg4": f"MixedTileRandomCompression.run with {CFG4_CPU_ITERS} of the 1000 iterations on kv_a_proj [576,7168], scaled linearly to 1000",
            "cfg5": "MixedTileGreedyCompression.run + wq:684-687 scoring on one expert gate_proj [2048,7168]"}[cfg]
    src = "the unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port (oracle/_ref absent)"
    return (f"{src}: {what}; one tensor per host process on every core (the reference is single-threaded NumPy); aggregate "
            "elements / slowest process; input generation excluded")


def run_reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = max(1, os.cpu_count() or 1)
    metric_key = args.config
    if args.config == "cfg2-fp8":      # the reference dequantizes on load and then runs cfg2's path on the float32 tensors
        args.config = "cfg2"
    for _ in range(min(args.warmup, 1)):                         # warm-up is page-cache / import warm only
        cpu_sample_run(args.config, procs)
    vals, t0 = [], time.perf_counter()
    kind, cores = "reference", procs
    steps = max(1, args.steps if args.config == "cfg2" else min(args.steps, 3))
    for _ in range(steps):
        v, cores, _w, kind = cpu_sample_run(args.config, procs)
        vals.append(v)
    wall = time.perf_counter() - t0
    value = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": METRICS[metric_key], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * wall / steps, "higher_is_better": True,
            "scaling": "strong" if args.config == "cfg5" else "weak", "vs_baseline": None,
            "dtype": "f32 values, f64 sums (NumPy)", "data": "synthetic", "config": config_dict(args.config, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": cpu_sample_desc(args.config, kind)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def config_dict(cfg: str, n_gpus: int) -> dict:
    if cfg == "cfg2":
        return {"workload": "configs[1]: mixed-tile-greedy pcc>=0.999 seed 123 over q_a/q_b/kv_a/kv_b/o_proj (synthetic randn*0.02 "
                            "bf16), one such tensor list per GPU",
                "tensors_per_gpu": 5, "elements_per_gpu": 187105280, "formats": "bf16,bfp8,bfp4,bfp2",
                "l2": "inputs_larger_than_l2 (374 MB per step vs 126 MB L2)", "parallelism": f"tensor-list x{n_gpus}",
                "launch": "one CUDA graph per step for the device-resident value (kernels of all tensors on ~20 captured streams); "
                          "eager stream launches for e2e",
                "inflight": f"up to {INFLIGHT} tensor lists in flight (lists_in_flight: the count used, the largest that divides the timed steps), each with its own buffers (the tile-stat passes of later steps overlap the greedy chains of earlier ones); "
                            "step_latency_ms is one step alone",
                "clusters": (f"chain clusters capped at {CLUSTER_CAP} CTAs per tensor (throughput schedule: a tensor's chain holds fewer SMs for longer); "
                             "latency_schedule = one step alone with automatic cluster sizes") if CLUSTER_CAP else "automatic cluster sizes (up to 16 CTAs per tensor)",
                "perm_cache": "value: the NumPy permutations of each (seed, tile count) are drawn once per process and reused by every "
                              "step - what a multi-layer model run does, every layer repeating the same shapes under one seed; "
                              "value_uncached redraws them on the device in every step"}
    w = {"cfg1": "configs[0]: none, bf16/bfp8/bfp4/bfp2/fp0 on q_a_proj [1536,7168]; 8 distinct input buffers rotate (176 MB > L2)",
         "cfg3": "configs[2]: threshold sweep, 32 thresholds (pcc, lowest 0.9), q_a/q_b/kv_a/kv_b/o_proj + gate/up/down dense MLP shapes",
         "cfg4": "configs[3]: mixed-tile-random, 1000 samples per tensor (pcc>=0.99), same 8 shapes, every sample scored in the reference's float32",
         "cfg5": "configs[4]: mixed-tile-greedy pcc>=0.999 seed 123 over one MoE layer (256 experts x gate/up [2048,7168] + down "
                 "[7168,2048] = 768 tensors, 22.5 GB), bin-packed over the ranks by partition_tensors"}[cfg]
    out = {"workload": w, "parallelism": f"tensor-list over {n_gpus} rank(s)", "l2": "inputs_larger_than_l2"}
    if cfg == "cfg5":
        out["inflight"] = (f"{CFG5_INFLIGHT} copies of the rank's shard in flight (each with its own buffers): the chains of a step's last tensors "
                           "run under the next step's tile-stat passes; step_latency_ms is one step alone")
    return out


def maps_vs_reference_goldens(items, *result_sets):
    """Rank 0's tensors are the ones tests/golden/cfg2_bench_workload.* holds the UNMODIFIED reference's greedy maps for
    (made by tests/golden/make_golden.py cfg2): compare the maps this run produced - device-resident and end-to-end - with
    them.  True / False, or None when the fixtures are not there."""
    import numpy as np
    gold = ROOT / "tests" / "golden" / "cfg2_bench_workload.npz"
    if not gold.exists():
        return None
    maps = dict(np.load(gold))
    ok = True
    for results in result_sets:
        for (name, _shape, _seed), r in zip(items, results):
            key = name.split(".")[-2]
            ok = ok and key in maps and bool(np.array_equal(r["assignment"], maps[key]))
    return ok


DUMP_SAMPLE = 1 << 21        # cfg1: reconstruction elements kept per format (3 x 8 MB)
DUMP_MAP_COLUMNS = 8192      # cfg3: tiles kept of each tensor's 32 threshold maps (8 x 1 MB)


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write DIR/<name>.npy for every array (float32 or float64; at most 44 MB in all, cfg5's maps)."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(d / f"{name}.npy", a)


def fixed_sample(n: int, k: int):
    """Sorted indices of a seeded sample of k of n positions (all of them when n <= k): the same for every run."""
    import numpy as np
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def other_outputs(cfg: str, names, K: int, out) -> dict:
    """What the last timed step of cfg1 / cfg3 / cfg4 computed.
    cfg1: the bfp8 / bfp4 / bfp2 reconstructions of the step's buffer (bf16 is the input itself, fp0 is zero), a fixed sample
          of DUMP_SAMPLE elements each (float32).
    cfg3: per tensor, one row per threshold [threshold, counts bf16/bfp8/bfp4/bfp2, total bytes, pcc, mae, atol] (float64)
          and the threshold maps at a fixed sample of at most DUMP_MAP_COLUMNS tiles (float32 [32, columns]).
    cfg4: per tensor, the selected map (float32), its counts and [pcc, mae, atol], and [pcc, mae, atol] of every sample
          (float64 [1000, 3])."""
    import numpy as np
    from quantization_analysis_b200.batch import MIXED
    res = {}
    if cfg == "cfg1":
        j = (K - 1) % 8
        for fmt, y in zip(("bfp8", "bfp4", "bfp2"), out):
            y = y.float().cpu().numpy()
            res[f"buffer{j}.{fmt}.sample"] = y[fixed_sample(y.size, DUMP_SAMPLE)]
        return res
    for name, r in zip(names, out):
        if cfg == "cfg3":
            rows, maps = r
            res[f"{name}.rows"] = np.array([[row["threshold"]] + [row["counts"][f] for f in MIXED]
                                            + [row["total_bytes"], row["pcc"], row["mae"], row["atol"]] for row in rows], dtype=np.float64)
            maps = maps.cpu().numpy()
            res[f"{name}.maps_sample"] = maps[:, fixed_sample(maps.shape[1], DUMP_MAP_COLUMNS)].astype(np.float32)
        else:
            res[f"{name}.assignment"] = r.assignment.cpu().numpy().astype(np.float32)
            res[f"{name}.counts"] = np.array([r.counts[f] for f in MIXED], dtype=np.float64)
            res[f"{name}.metrics"] = np.array([r.metrics_exact[k] for k in ("pcc", "mae", "atol")], dtype=np.float64)
            res[f"{name}.samples"] = np.array([[s_["pcc"], s_["mae"], s_["atol"]] for s_ in r.meta["samples"]], dtype=np.float64)
    return res


def greedy_outputs(items, results) -> dict:
    """What a GreedyBatch caller receives for each tensor: the tile map (float32), the tile counts in bf16/bfp8/bfp4/bfp2
    order and [pcc, mae, atol] (float64)."""
    import numpy as np
    from quantization_analysis_b200.batch import MIXED
    out = {}
    for (name, _shape, _seed), r in zip(items, results):
        out[f"{name}.assignment"] = r["assignment"].astype(np.float32)
        out[f"{name}.counts"] = np.array([r["counts"][f] for f in MIXED], dtype=np.float64)
        out[f"{name}.metrics"] = np.array([r["metrics"][k] for k in ("pcc", "mae", "atol")], dtype=np.float64)
    return out


def pin_rank_to_cores(local: int, world: int) -> list[int] | None:
    """Give every rank of the node its own slice of the host cores before any pinned buffer is allocated: the launch
    threads and the pinned pages of one rank then do not migrate under the others (round 1: e2e fell to 0.42 efficiency
    at 8 ranks with every rank floating over cores 0-31)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world <= 1 or len(cpus) < 2 * world:
            return None
        per = len(cpus) // world
        mine = cpus[local * per:(local + 1) * per]
        os.sched_setaffinity(0, mine)
        return mine
    except Exception:
        return None


class Env:
    pass


def setup():
    e = Env()
    e.world = int(os.environ.get("WORLD_SIZE", "1"))
    e.rank = int(os.environ.get("RANK", "0"))
    e.local = int(os.environ.get("LOCAL_RANK", "0"))
    e.cores = pin_rank_to_cores(e.local, e.world)          # before torch starts its threads and pins any memory
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(e.local)
    e.dev = torch.device("cuda", e.local)
    if e.world > 1:
        dist.init_process_group("nccl", device_id=e.dev)
    from quantization_analysis_b200 import _lib
    _lib.lib()
    e.torch, e.dist = torch, dist

    def barrier():
        if e.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(v: float) -> float:
        if e.world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=e.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(v: float) -> list[float]:
        if e.world == 1:
            return [v]
        t = torch.tensor([v], dtype=torch.float64, device=e.dev)
        buf = [torch.zeros_like(t) for _ in range(e.world)]
        dist.all_gather(buf, t)
        return [float(b.item()) for b in buf]

    e.barrier, e.reduce_max, e.gather_floats = barrier, reduce_max, gather_floats
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    e.peak = float(peaks.get("hbm_gbs", 6650.0))
    e.peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return e


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` summary of
    this round (profiles/r2_traffic.json, written by profiles/make_summary.py), or None."""
    f = ROOT / "profiles" / "r2_traffic.json"
    if not f.exists():
        return None
    try:
        return json.loads(f.read_text()).get(kernel)
    except Exception:
        return None


def attach_cpu_baseline(line: dict, cfg: str, enabled: bool) -> None:
    if not enabled:
        return
    import subprocess
    try:      # fresh interpreter (no CUDA context, no inherited thread pools), bounded by a timeout
        out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                              "--config", cfg], capture_output=True, text=True, timeout=300, check=True)
        ref = json.loads(out.stdout.strip().splitlines()[-1])
        line["cpu_baseline"] = dict(ref["cpu_baseline"], host_cpus=os.cpu_count())
    except Exception as exc:  # report, never hang the GPU line
        line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                                "sample": f"failed: {type(exc).__name__}: {exc}"[:300]}


# --------------------------------------------------------------------------------------------
# cfg2 (default) and cfg5: mixed-tile-greedy over a tensor list through GreedyBatch
# --------------------------------------------------------------------------------------------
def bench_greedy(args, e) -> None:
    torch, dist = e.torch, e.dist
    from quantization_analysis_b200 import sharding, synthetic
    from quantization_analysis_b200.batch import GreedyBatch
    cfg5 = args.config == "cfg5"
    W, K = max(3, args.warmup), max(1, args.steps)
    dev, world, rank = e.dev, e.world, e.rank
    if cfg5:
        all_items = synthetic.expert_tensor_list(256)
        mine = sharding.partition_tensors([s[0] * s[1] for _n, s in all_items], world)[rank]
        items = [(all_items[i][0], all_items[i][1], 5000 + i) for i in mine]
        uniq = [synthetic.randn_bf16_cpu(s, 50 + j).pin_memory() for j, s in enumerate(synthetic.EXPERT_SHAPES.values())]
        host = [uniq[list(synthetic.EXPERT_SHAPES.values()).index(tuple(s))] for (_n, s, _sd) in items]   # 3 distinct host tensors
        inflight = CFG5_INFLIGHT
    else:
        items = workload(rank)
        host = [synthetic.randn_bf16_cpu(shape, seed).pin_memory() for (_n, shape, seed) in items]
        # lists in flight: every list runs its steps one after the other, so the K timed steps are spread evenly - the largest
        # count up to INFLIGHT that divides K (20 steps: 10 lists x 2; 24: 12 x 2), unless QA_BENCH_INFLIGHT fixes it
        inflight = min(INFLIGHT, K)
        if "QA_BENCH_INFLIGHT" not in os.environ:
            even = [n for n in range(inflight, 5, -1) if K % n == 0]
            inflight = even[0] if even else inflight
    shapes = [s for (_n, s, _sd) in items]

    def make_batches(perm_cache: bool, n: int, cap: int = CLUSTER_CAP):
        sg = int(os.environ["QA_BENCH_STATS_GROUP"]) if "QA_BENCH_STATS_GROUP" in os.environ else None      # None: the batch's own choice
        bs = [GreedyBatch(shapes, **GREEDY, device=dev, perm_cache=perm_cache, stats_group=sg) for _ in range(n)]
        if not cfg5:                                   # cfg5 keeps the batch's own choice for long lists (2-CTA clusters)
            for b in bs:
                b.cluster_cap = cap
        for b in bs:
            b.load_device(host)
        torch.cuda.synchronize()
        for b in bs:
            b.capture()
        return bs

    batches = make_batches(True, inflight)
    batch = batches[0]
    nbytes = batch.total_bytes()
    total_bytes = nbytes * world if not cfg5 else int(sum(2 * s[0] * s[1] for _n, s in synthetic.expert_tensor_list(256)))
    lanes = [torch.cuda.Stream(device=dev) for _ in range(inflight)]

    def run_steps(bs, n_steps: int, lanes_used: int) -> None:
        cur = torch.cuda.current_stream(dev)
        for ln in lanes[:lanes_used]:
            ln.wait_stream(cur)
        for k in range(n_steps):
            with torch.cuda.stream(lanes[k % lanes_used]):
                bs[k % lanes_used].run_graph()
        for ln in lanes[:lanes_used]:
            cur.wait_stream(ln)

    def timed(bs, n_steps: int, lanes_used: int) -> float:
        run_steps(bs, W, lanes_used)
        e.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e.barrier()
        a.record()
        run_steps(bs, n_steps, lanes_used)
        b.record()
        e.barrier()
        return a.elapsed_time(b)

    # SM clocks / throttle reasons are sampled over both timed regions, on rank 0 only (NVML queries from every rank of a
    # node serialise in the driver and steal host time from the launch threads)
    clk = ClockSampler(e.local, enabled=(rank == 0))
    clk.__enter__()
    ms_local = timed(batches, K, inflight)
    if args.dump_outputs:                                        # step k of the timed loop ran on list k % inflight
        dump_outputs(args.dump_outputs, greedy_outputs(items, batches[(K - 1) % inflight].collect()))
    ms = e.reduce_max(ms_local)
    per_rank_ms = e.gather_floats(ms_local / K)
    value = total_bytes * K / (ms * 1e-3) / 1e9
    ms_single = e.reduce_max(timed(batches, K, 1)) / K          # latency of one step with nothing else in flight
    results = batch.collect()
    latency_schedule = None
    if not cfg5 and CLUSTER_CAP != 0:                            # the same step alone with automatic cluster sizes
        lb = make_batches(True, 1, cap=0)
        ms_lat = e.reduce_max(timed(lb, K, 1)) / K
        for r0, r1 in zip(results, lb[0].collect()):
            assert (r0["assignment"] == r1["assignment"]).all() and r0["counts"] == r1["counts"]
        latency_schedule = {"cluster_cap": "automatic (up to 16 CTAs per tensor)", "step_latency_ms": ms_lat,
                            "note": "one step alone; with 12 lists in flight this schedule runs at 0.265 ms per step (profiles/r2_step_sweep3.txt)"}
        del lb
    for b in batches[1:]:                                        # every in-flight list produced the same maps
        for r0, r1 in zip(results, b.collect()):
            assert (r0["assignment"] == r1["assignment"]).all() and r0["counts"] == r1["counts"]

    # the same steps with the permutations redrawn on the device in every step (round 1's schedule)
    value_unc = ms_unc = launches_unc = None
    if not cfg5:
        unc = make_batches(False, inflight)
        ms_unc = e.reduce_max(timed(unc, K, inflight))
        value_unc = total_bytes * K / (ms_unc * 1e-3) / 1e9
        for r0, r1 in zip(results, unc[0].collect()):
            assert (r0["assignment"] == r1["assignment"]).all() and r0["counts"] == r1["counts"]
        launches_unc = unc[0].launches_per_step * K
        ms_unc = ms_unc / K
        del unc

    # ---- end to end: pinned host bf16 -> H2D -> path -> D2H of maps and metric rows ------------
    # Two batches alternate (enqueue_from_host / finish): the next list's H2D copies keep the PCIe link busy while the
    # previous list's chain finishes and its results travel back.  Every step's results are read on the host.
    eb = batches if (len(batches) > 1 or cfg5) else batches + make_batches(True, 1)

    def e2e_steps(n_steps: int):
        res = None
        for k in range(n_steps):
            b = eb[k % len(eb)]
            if k >= len(eb):
                res = b.finish()
            b.enqueue_from_host(host)
        for k in range(min(n_steps, len(eb))):
            res = eb[(n_steps - min(n_steps, len(eb)) + k) % len(eb)].finish()
        return res

    Ke = K if not cfg5 else max(1, min(K, 3))
    e2e_steps(2)
    e.barrier()
    t0 = time.perf_counter()
    res_e2e = e2e_steps(Ke)
    torch.cuda.synchronize()
    e2e_s = e.reduce_max(time.perf_counter() - t0)
    e2e_value = total_bytes * Ke / e2e_s / 1e9
    clk.__exit__()
    # the ceiling of that number: a plain pinned-host -> device copy of the same bytes, alone and with every rank copying
    big = max(range(len(host)), key=lambda i: host[i].numel())
    dst = torch.empty_like(host[big], device=dev)

    def copy_rate(concurrent: bool) -> float:
        for _ in range(2):
            dst.copy_(host[big], non_blocking=True)
        torch.cuda.synchronize()
        if concurrent:
            e.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            dst.copy_(host[big], non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        return 5 * host[big].numel() * 2 / (c0.elapsed_time(c1) * 1e-3) / 1e9

    h2d_concurrent = e.gather_floats(copy_rate(True))
    if world > 1:                      # one rank at a time
        alone = 0.0
        for r in range(world):
            if r == rank:
                alone = copy_rate(False)
            e.barrier()
        h2d_alone = e.gather_floats(alone)
    else:
        h2d_alone = h2d_concurrent
    del dst

    # ---- the plug-in call a drop-in user makes: numpy float32 in, y float32 numpy out + wq:684-687 scoring ----------
    e2e_plugin = None
    if not cfg5:
        from quantization_analysis_b200 import compression_algorithms as ca
        from quantization_analysis_b200.compression_algorithms import metrics as M
        xs32 = [h.float().numpy() for h in host]
        algo = ca.create_algorithm("mixed-tile-greedy", dict(GREEDY))

        import numpy as np

        def plugin_step():
            out = []
            for x in xs32:
                r = algo.run(x, FORMATS5, ca.quantizer.Quantizer("emulation"), None)[0]
                d = np.abs(x - r.y)                                   # wq:684-687, as the reference's wq does on top of run()
                out.append((r.meta["assignment"], M.pearson_corr(x, r.y), float(np.mean(d)), float(np.max(d))))
            return out

        plugin_step()
        e.barrier()
        t0 = time.perf_counter()
        reps = max(1, min(K, 3))
        for _ in range(reps):
            pres = plugin_step()
        torch.cuda.synchronize()
        ps = e.reduce_max(time.perf_counter() - t0)
        e2e_plugin = {"value": total_bytes * reps / ps / 1e9, "unit": UNIT, "steps": reps,
                      "api": "create_algorithm('mixed-tile-greedy', params).run(x float32 numpy, formats, Quantizer('emulation'), None) -> y float32 "
                             "numpy, then wq:684-687 on top of it (np.abs / np.mean / np.max on the host, pearson_corr through the drop-in); pageable host arrays",
                      "h2d_bytes_per_step": 2 * nbytes * 3, "d2h_bytes_per_step": 2 * nbytes,
                      "maps_equal_device_resident": all(bool((a[0].reshape(-1) == r["assignment"].reshape(-1)).all()) for a, r in zip(pres, results))}

    # ---- the one real exchange of the partition: a row-striped tensor, tables all-gathered, one global greedy -------
    striped = None
    if world > 1 and not cfg5:
        name, shape, seed = items[-1] if items[-1][1] == (7168, 16384) else max(items, key=lambda t: t[1][0] * t[1][1])
        x_full = synthetic.randn_bf16_cpu(shape, 1004)            # the same tensor on every rank; each keeps its stripe
        a, b = sharding.row_stripes(shape[0], world)[rank]
        stripe = x_full[a:b].to(dev)
        torch.cuda.synchronize()
        e.barrier()
        g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        from quantization_analysis_b200 import engine
        g0.record()
        p = engine.prepare_tiles(stripe.reshape(-1, shape[1]))
        local_t = engine.tile_stats(p, engine.MIXED_FORMATS, exact_abs=False)
        g1.record()
        full = sharding.gather_tables(local_t)
        g2.record()
        amap, counts, _st = engine.greedy_assign(full, x_full.numel(), "pcc", 0.999, list(engine.MIXED_FORMATS), engine.make_rng(123, dev))
        torch.cuda.synchronize()
        ok = None
        if rank == 0:
            pf = engine.prepare_tiles(x_full.to(dev))
            tf = engine.tile_stats(pf, engine.MIXED_FORMATS, exact_abs=False)
            a1, c1, _s = engine.greedy_assign(tf, pf.numel, "pcc", 0.999, list(engine.MIXED_FORMATS), engine.make_rng(123, dev))
            ok = bool(torch.equal(full, tf) and torch.equal(a1, amap) and torch.equal(c1, counts))
        striped = {"tensor": f"{shape[0]}x{shape[1]}", "stripes": world, "striped_equals_single": ok,
                   "stats_ms_max": e.reduce_max(g0.elapsed_time(g1)), "allgather_ms_max": e.reduce_max(g1.elapsed_time(g2)),
                   "table_bytes": int(full.numel() * 8)}
    if world > 1:                                   # per-tensor result rows to rank 0 (tiny)
        rows = [[r["metrics"]["pcc"], r["metrics"]["mae"], r["metrics"]["atol"]] for r in res_e2e]
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(rows, gathered, dst=0)

    # ---- per-kernel timing for the roofline (events on the launching stream, all tensors of the list) ----
    def time_phase(stats: bool, assign: bool, reps: int = 5) -> float:
        for _ in range(2):
            batch.run_graph(stats=stats, assign=assign)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            batch.run_graph(stats=stats, assign=assign)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    if batch.stats_group > 0:        # descriptor-array launches: one tile-stat kernel per group of tensors
        n_stats_launches = len(batch._groups)
    else:
        n_stats_launches = sum(3 if (s["ntiles"] >= batch.PIPELINE_MIN_TILES and -(-s["rows"] // 32) >= 8) else 1 for s in batch.slots)
    ms_stats = time_phase(True, False)
    ms_assign = time_phase(False, True, reps=2)
    ntiles = sum(s["ntiles"] for s in batch.slots)
    alg_stats = nbytes + ntiles * TABLE_BYTES_PER_TILE            # read x once + write the tile-stat table
    alg_assign = ntiles * (TABLE_BYTES_PER_TILE + 1)              # read the table once + write the int8 map
    step_ms = ms / K
    hbm = {"kernel": "stats_fast_kernel", "ms_per_step": ms_stats, "launches_per_step": n_stats_launches,
           "alg_bytes_per_step": alg_stats, "achieved_gbs": alg_stats / (ms_stats * 1e-3) / 1e9}
    chain = {"kernel": "greedy chain group (greedy_init_kernel, greedy_delta_kernel, greedy_par_kernel)", "ms_per_step": ms_assign,
             "launches_per_step": batch.launches_per_step - n_stats_launches, "alg_bytes_per_step": alg_assign,
             "achieved_gbs": alg_assign / (ms_assign * 1e-3) / 1e9,
             "note": "latency-bound cluster kernels over the 20 MB table; they overlap the next list's tile-stat pass"}
    for k in (hbm, chain):
        k["frac"] = k["achieved_gbs"] / e.peak
    step_gbs = alg_stats / (step_ms * 1e-3) / 1e9                 # this rank's weights + table bytes of one step
    big = max(batch.slots, key=lambda s_: s_["ntiles"])           # its last row range is the largest tile-stat launch
    th_, tw_ = -(-big["rows"] // 32), -(-big["cols"] // 32)
    if big["ntiles"] >= batch.PIPELINE_MIN_TILES and th_ >= 8:
        sp1 = max(1, min(th_ - 2, -(-max(batch.PIPELINE_FIRST_TILES, big["ntiles"] // 8) // tw_)))
        rows_largest = th_ - max(sp1 + 1, th_ // 2)
    else:
        rows_largest = th_
    alg_largest = rows_largest * tw_ * (2 * 1024 + TABLE_BYTES_PER_TILE)
    roofline = {"bound": "hbm", "kernel": "stats_fast_kernel", "achieved": hbm["achieved_gbs"], "peak": e.peak, "unit": "GB/s",
                "frac": hbm["frac"], "traffic": ncu_traffic("stats_fast_kernel"), "traffic_launch_alg_bytes": alg_largest,
                "traffic_note": "dram__bytes_read + dram__bytes_write of the largest launch (the last row range of the largest tensor) from this "
                                "round's `ncu --set full` capture (profiles/r2_traffic.json); traffic_launch_alg_bytes = algorithmic bytes of that launch",
                "peak_source": e.peak_src, "alg_bytes_per_launch": alg_stats / n_stats_launches,
                "avg_launch_ms": ms_stats / n_stats_launches,
                "step_frac": step_gbs / e.peak, "step_achieved_gbs": step_gbs,
                "note": "the HBM-bearing kernel of the step (reads every weight once, writes the tile-stat table), timed alone over "
                        "the tensor list; step_frac = (weights + table bytes of one step) / ms_per_step / peak, per GPU"}
    if rank == 0:
        line = {"metric": METRICS[args.config], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong" if cfg5 else "weak", "vs_baseline": None,
                "dtype": "bf16 in; f32 group-scaled + f64 sums", "data": "synthetic", "config": dict(config_dict(args.config, world), **({} if cfg5 else {"lists_in_flight": inflight})),
                "clocks": clk.summary(),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": batch.d2h_bytes(),
                        "steps": Ke, "h2d_copy_gbs": h2d_alone[0], "h2d_copy_gbs_per_rank_alone": h2d_alone,
                        "h2d_copy_gbs_per_rank_concurrent": h2d_concurrent, "cores_of_rank0": e.cores,
                        "api": "GreedyBatch.enqueue_from_host(pinned bf16 host tensors) / finish() -> assignment maps + pcc/mae/atol on host, two batches alternating"},
                "e2e_plugin": e2e_plugin,
                "gpu_launches": batch.launches_per_step * K,
                "value_uncached": value_unc, "ms_per_step_uncached": ms_unc, "gpu_launches_uncached": launches_unc,
                "step_latency_ms": ms_single, "latency_schedule": latency_schedule,
                "per_rank_ms_per_step": per_rank_ms,
                "roofline": roofline, "roofline_by_kernel": [hbm, chain],
                "pct_of_8TBs": 100.0 * value / world / 8000.0,
                "result_check": {"counts_first_tensor": results[0]["counts"], "pcc_first_tensor": results[0]["metrics"]["pcc"],
                                 "maps_equal_reference": None if cfg5 else maps_vs_reference_goldens(items, results, res_e2e),
                                 "striped": striped}}
        attach_cpu_baseline(line, args.config, world == 1 and not args.no_cpu_baseline)
        print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# cfg2-fp8: the same tensor list as a real checkpoint stores it (SURVEY section 8 row f1) - e4m3fn bytes + block scales in,
# dequantization (hf_model_utils.py:199-215) fused into the tile-stat read.  Not a BASELINE config: one extra line.
# --------------------------------------------------------------------------------------------
def bench_fp8(args, e) -> None:
    torch = e.torch
    import numpy as np
    from quantization_analysis_b200 import compression_algorithms as ca, engine, synthetic
    from quantization_analysis_b200.batch import GreedyBatch
    W, K = max(3, args.warmup), max(1, args.steps)
    dev, world, rank = e.dev, e.world, e.rank
    items = workload(rank)
    shapes = [s for (_n, s, _sd) in items]
    host = [tuple(t.pin_memory() for t in synthetic.fp8_checkpoint_cpu(shape, seed)) for (_n, shape, seed) in items]
    inflight = max(2, INFLIGHT)
    batches = [GreedyBatch(shapes, **GREEDY, device=dev, perm_cache=True, source="fp8") for _ in range(inflight)]
    for b in batches:
        b.load_device(host)
    torch.cuda.synchronize()
    for b in batches:
        b.capture()
    batch = batches[0]
    lanes = [torch.cuda.Stream(device=dev) for _ in range(inflight)]

    def run_steps(n_steps: int, lanes_used: int) -> None:
        cur = torch.cuda.current_stream(dev)
        for ln in lanes[:lanes_used]:
            ln.wait_stream(cur)
        for k in range(n_steps):
            with torch.cuda.stream(lanes[k % lanes_used]):
                batches[k % lanes_used].run_graph()
        for ln in lanes[:lanes_used]:
            cur.wait_stream(ln)

    def timed(n_steps: int, lanes_used: int) -> float:
        run_steps(W, lanes_used)
        e.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e.barrier()
        a.record()
        run_steps(n_steps, lanes_used)
        b.record()
        e.barrier()
        return a.elapsed_time(b)

    clk = ClockSampler(e.local, enabled=(rank == 0))
    clk.__enter__()
    ms = e.reduce_max(timed(K, inflight))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, greedy_outputs(items, batches[(K - 1) % inflight].collect()))
    ms_single = e.reduce_max(timed(K, 1)) / K
    eq_bytes, in_bytes = batch.total_bytes(), batch.input_bytes()
    value = eq_bytes * world * K / (ms * 1e-3) / 1e9
    results = batch.collect()

    def e2e_steps(n_steps: int):
        res = None
        for k in range(n_steps):
            b = batches[k % 2]
            if k >= 2:
                res = b.finish()
            b.enqueue_from_host(host)
        for k in range(min(n_steps, 2)):
            res = batches[(n_steps - min(n_steps, 2) + k) % 2].finish()
        return res

    e2e_steps(2)
    e.barrier()
    t0 = time.perf_counter()
    res_e2e = e2e_steps(K)
    torch.cuda.synchronize()
    e2e_s = e.reduce_max(time.perf_counter() - t0)
    clk.__exit__()

    # the tile-stat pass alone (events on the launching stream)
    for _ in range(2):
        batch.run_graph(stats=True, assign=False)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        batch.run_graph(stats=True, assign=False)
    b.record()
    torch.cuda.synchronize()
    ms_stats = a.elapsed_time(b) / 5
    ntiles = sum(s_["ntiles"] for s_ in batch.slots)
    n_launches = sum(3 if (s_["ntiles"] >= batch.PIPELINE_MIN_TILES and -(-s_["rows"] // 32) >= 8) else 1 for s_ in batch.slots)
    alg = in_bytes + ntiles * TABLE_BYTES_PER_TILE

    # result check: the two smallest tensors through the plug-in on the reference's dequantized float32 image (strict sums,
    # one-thread chain: reference order everywhere) give the same maps as the fused fp8 batch
    algo = ca.create_algorithm("mixed-tile-greedy", dict(GREEDY, strict_sums=True, sequential_chain=True))
    small = sorted(range(len(items)), key=lambda i: shapes[i][0] * shapes[i][1])[:2]
    same = True
    for i in small:
        x32 = engine.fp8_block_dequant(host[i][0], host[i][1], want_bf16=False)[0].cpu().numpy()
        r = algo.run(x32, FORMATS5, None, None)[0]
        same = same and bool(np.array_equal(r.meta["assignment"], results[i]["assignment"])) \
            and bool(np.array_equal(r.meta["assignment"], res_e2e[i]["assignment"]))
    if rank == 0:
        elems = sum(s_["numel"] for s_ in batch.slots)
        line = {"metric": METRICS["cfg2-fp8"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp8 e4m3fn x f32 block scale in; f32 products + f64 sums", "data": "synthetic",
                "config": {"workload": "cfg2's tensor list (q_a/q_b/kv_a/kv_b/o_proj) quantized to fp8 e4m3fn with 128x128 block inverse scales "
                                       "(synthetic randn*0.02); mixed-tile-greedy pcc>=0.999 seed 123; value counts 2 bytes per element (the bf16 "
                                       "metric's unit) - the pass reads 1 byte per element",
                           "elements_per_gpu": elems, "input_bytes_per_step": in_bytes, "l2": "inputs_larger_than_l2 (187 MB per step vs 126 MB L2)",
                           "inflight": f"{inflight} tensor lists in flight", "perm_cache": "on", "parallelism": f"tensor-list x{world}"},
                "clocks": clk.summary(),
                "elements_per_s": elems * world * K / (ms * 1e-3),
                "e2e": {"value": eq_bytes * world * K / e2e_s / 1e9, "unit": UNIT, "h2d_bytes_per_step": in_bytes,
                        "d2h_bytes_per_step": batch.d2h_bytes(), "steps": K, "input_gbs": in_bytes * world * K / e2e_s / 1e9,
                        "api": "GreedyBatch(source='fp8').enqueue_from_host(pinned e4m3fn bytes + scale grids) / finish() -> maps + pcc/mae/atol on host"},
                "gpu_launches": batch.launches_per_step * K, "step_latency_ms": ms_single,
                "roofline": {"bound": "hbm", "kernel": "stats_f32_kernel<fp8>", "achieved": alg / (ms_stats * 1e-3) / 1e9, "peak": e.peak,
                             "unit": "GB/s", "frac": alg / (ms_stats * 1e-3) / 1e9 / e.peak, "traffic": None, "peak_source": e.peak_src,
                             "alg_bytes_per_launch": alg / n_launches, "avg_launch_ms": ms_stats / n_launches,
                             "note": "1 B/elem + scale grid read, 176 B per tile written; the kernel is bound by float32 -> float64 conversions "
                                     "(seven per element: the reference's float32 product arrays summed in float64), not by HBM"},
                "cpu_baseline": None,
                "result_check": {"maps_equal_reference_order_run_on_dequantized_float32": same,
                                 "counts_first_tensor": results[0]["counts"], "pcc_first_tensor": results[0]["metrics"]["pcc"]}}
        print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# cfg1 / cfg3 / cfg4 through the product API (device tensors in, device results)
# --------------------------------------------------------------------------------------------
def bench_other(args, e) -> None:
    torch = e.torch
    from quantization_analysis_b200 import engine, sweep, synthetic
    from quantization_analysis_b200 import compression_algorithms as ca
    cfg, dev = args.config, e.dev
    W = max(3, args.warmup) if cfg == "cfg1" else 1
    K = max(1, args.steps) if cfg == "cfg1" else max(1, min(args.steps, 2))
    names = synthetic.ATTN_NAMES + synthetic.MLP_NAMES
    if cfg == "cfg1":
        import ctypes as C
        from quantization_analysis_b200 import _lib
        xs = [synthetic.device_randn_bf16((1536, 7168), 100 + i, dev) for i in range(8)]      # 8 x 22 MB > L2
        preps = [engine.prepare_rows(x) for x in xs]
        # one step = qa_quant_recon of one buffer into resident outputs (bf16 aliases the input, fp0 is not materialised); the
        # 8 buffers' steps are captured into one CUDA graph so that the ~20 us host launch path does not bound a 19 us kernel
        outs = [[torch.empty(p.rows * p.cols, dtype=torch.bfloat16, device=dev) for _ in range(3)] for p in preps]
        arrs = []
        for o3 in outs:
            arr = (C.c_void_p * 4)()
            arr[1], arr[2], arr[3] = (o.data_ptr() for o in o3)
            arrs.append(arr)

        def launch8():
            sp = torch.cuda.current_stream().cuda_stream
            for p, arr in zip(preps, arrs):
                _lib.check(_lib.lib().qa_quant_recon(p.data.data_ptr(), p.dtype_code, p.rows, p.cols, p.cols, 0b1110, arr, sp), "qa_quant_recon")
        launch8()
        torch.cuda.synchronize()
        graph8 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph8):
            launch8()
        K = 8 * max(1, (max(K, 64) + 7) // 8)            # steps come in rounds of the 8 rotating buffers
        W = 8

        def step(k):
            if k % 8 == 0:
                graph8.replay()
            return outs[k % 8]
        per_step_elems = xs[0].numel()
        alg_bytes = 8 * per_step_elems
        kernel = "recon_fast_kernel"
    else:
        xs = [synthetic.device_randn_bf16(synthetic.DEEPSEEK_R1_SHAPES[n], 300 + i, dev) for i, n in enumerate(names)]
        per_step_elems = sum(x.numel() for x in xs)
        alg_bytes = int(2.17 * per_step_elems)
        kernel = "tile_scores_kernel" if cfg == "cfg3" else "stats_fast_kernel"
        scoring = os.environ.get("QA_BENCH_SCORING", "reference")      # "exact": float64 table recombination instead of the
        if cfg == "cfg3":                                               # reference's float32 whole-tensor arithmetic
            def step(k):
                return [sweep.sweep_tensor(x, engine.MIXED_FORMATS, "pcc", steps=32, lowest=0.9, scoring=scoring) for x in xs]
        else:
            algo = ca.create_algorithm("mixed-tile-random", {"metric": "pcc", "threshold": 0.99, "iters": 1000, "seed": 42,
                                                              "sample_scoring": scoring})

            def step(k):
                return [algo.run_prepared(engine.prepare_tiles(x), list(engine.MIXED_FORMATS)) for x in xs]
    for k in range(W):
        step(k)
    e.barrier()
    clk = ClockSampler(e.local, enabled=(e.rank == 0))
    clk.__enter__()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(K):
        out = step(k)
    b.record()
    e.barrier()
    clk.__exit__()
    ms = e.reduce_max(a.elapsed_time(b))
    value = e.world * 2.0 * per_step_elems * K / (ms * 1e-3) / 1e9
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, other_outputs(cfg, names, K, out))
    if cfg != "cfg1":
        out = [r[0][-1]["counts"] for r in out] if cfg == "cfg3" else [r.counts for r in out]
    # cfg1 end to end through the plug-in: numpy float32 in, five float32 reconstructions out + reference scores
    e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if cfg == "cfg1":
        from quantization_analysis_b200.compression_algorithms import metrics as M
        x32 = xs[0].float().cpu().numpy()
        algo = ca.create_algorithm("none", {})

        def plug():
            rs = algo.run(x32, FORMATS5, ca.quantizer.Quantizer("emulation"), None)
            return [(r.fmt, M.pearson_corr(x32, r.y), M.metric_value(x32, r.y, "mae"), M.metric_value(x32, r.y, "atol")) for r in rs]
        plug()
        t0 = time.perf_counter()
        for _ in range(3):
            rows = plug()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
        e2e = {"value": 2.0 * x32.size / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": 4 * x32.size * 11, "d2h_bytes_per_step": 4 * x32.size * 5,
               "api": "NoneCompression.run(x float32 numpy, 5 formats) -> 5 float32 arrays + pearson_corr / metric_value per format",
               "pcc_rows": {r[0]: r[1] for r in rows}}
    achieved = alg_bytes * K / (ms * 1e-3) / 1e9
    if e.rank == 0:
        line = {"metric": METRICS[cfg], "value": value, "unit": UNIT, "n_gpus": e.world, "steps": K, "warmup": W, "ms_per_step": ms / K,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 in; f32 / f64 sums", "data": "synthetic",
                "config": dict(config_dict(cfg, e.world), scoring=os.environ.get("QA_BENCH_SCORING", "reference") if cfg in ("cfg3", "cfg4") else "reference"),
                "clocks": clk.summary(), "e2e": e2e, "gpu_launches": None,
                "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": e.peak, "unit": "GB/s", "frac": achieved / e.peak,
                             "traffic": ncu_traffic(kernel), "peak_source": e.peak_src,
                             "note": "whole step over algorithmic bytes (cfg1: 8 B/elem; cfg3/4: 2.17 B/elem - the step also materialises and "
                                     "scores every distinct map / sample in the reference's float32 order, which dominates its time)"},
                "result_check": {"last": str(out)[:200]}}
        attach_cpu_baseline(line, cfg, e.world == 1 and not args.no_cpu_baseline)
        print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(METRICS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<tensor>.<array>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl b200")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    e = setup()
    if args.config == "cfg2-fp8":
        bench_fp8(args, e)
    elif args.config in ("cfg2", "cfg5"):
        bench_greedy(args, e)
    else:
        bench_other(args, e)
    if e.world > 1:
        e.dist.barrier()
        e.dist.destroy_process_group()


if __name__ == "__main__":
    main()
