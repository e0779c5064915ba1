r"""Multi-tensor batching of the quantize-and-score path (the per-tensor loop of wq:655-709).

``GreedyBatch`` owns every device buffer for a list of same-run tensors and enqueues, per
tensor, the stages of the path on a small pool of CUDA streams, with no host synchronisation
until ``collect()`` / ``finish()``.  Tensors are independent (the reference processes them one
after another), so a rank's shard is just a sub-list.

Schedule of one tensor (every stage is a C-ABI call; see DESIGN.md section 3.5):

    side stream   resolve permutations #1,#2 ........ resolve #3 .. apply #3 ..............\
    side2 stream                       apply #2 ......\                                    \
    stats stream  tile stats [rows A | B | C] . deltas \                                    \
    main stream        init sums A ... B ........ C ... chain passes 0-1 ... chain passes 2+ ... (D2H)

* the permutations depend on (seed, tile count) only: tensors of equal tile count share them;
* the table of a large tensor is produced in row ranges, its sequential init sums run underneath;
* tile-stat passes of all tensors are serialized largest first, cluster kernels get priority;
* with ``perm_cache`` the permutations are drawn once per (device, seed, tile count, format count) for the whole process
  (every layer of a model repeats the same shapes under one seed) and the per-step prefetch launches disappear;
* ``capture()`` / ``run_graph()`` replay the whole list as one CUDA graph;
* ``enqueue_from_host()`` / ``finish()`` is the asynchronous end-to-end form (pinned host in, pinned host out).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, engine
from ._lib import METRIC_CODE, NFMT, NSTAT, STATS_FAST, STATS_FAST_APPROX_ABS, check

MIXED = engine.MIXED_FORMATS

# (device index, seed, ntiles, nfmt) -> {"pre_order": int32 [2, ntiles], "rngs": stream states after permutations #1..#3}.
# NumPy's permutation of n items from a freshly seeded generator depends on nothing else, and the reference re-seeds per
# tensor (mixed_tile_greedy.py:222-225): every tensor with the same tile count - the experts of a MoE layer, the same
# projection in each of a model's 61 layers - visits its tiles in the same order.
_PERM_CACHE: dict = {}


def cached_permutations(device, seed: int, ntiles: int, nfmt: int):
    """Visiting orders of greedy passes 2 and 3 and the generator states after permutations #1..#3, drawn once (synchronous,
    outside any timed region or graph capture) and kept for the life of the process."""
    key = (torch.device(device).index, int(seed), int(ntiles), int(nfmt))
    hit = _PERM_CACHE.get(key)
    if hit is not None:
        return hit
    L = _lib.lib()
    dev = torch.device(device)
    rng0 = engine.make_rng(seed, dev)
    jarr = torch.empty((3, ntiles), dtype=torch.int32, device=dev)
    pre_order = torch.empty((2, ntiles), dtype=torch.int32, device=dev)
    rngs = torch.stack([rng0, rng0, rng0]).contiguous()
    awork = torch.empty((2, L.qa_perm_apply_work_bytes(ntiles)), dtype=torch.uint8, device=dev)
    cur = torch.cuda.current_stream(dev)
    engine.enqueue_perm_prefetch(rng0, ntiles, nfmt >= 3, (jarr, pre_order, rngs, awork), cur, cur,
                                 [torch.cuda.Event() for _ in range(3)])
    cur.synchronize()
    _PERM_CACHE[key] = {"pre_order": pre_order, "rngs": rngs}
    return _PERM_CACHE[key]


class GreedyBatch:
    PIPELINE_MIN_TILES = 32768      # tensors at least this large produce their table in three row ranges (see _enqueue)
    PIPELINE_FIRST_TILES = 4096    # ... the first of at least this many tiles (or an eighth of the tensor)

    def __init__(self, shapes, metric: str = "pcc", threshold: float = 0.999, seed: int = 123,
                 tile_formats=MIXED, n_streams: int | None = None, device=None, perm_cache: bool = False,
                 source: str = "bf16", scale_block=(128, 128), stats_group: int | None = None):
        """source="bf16": resident bf16 tensors (the default).  source="fp8": e4m3fn bytes + a float32 inverse-scale grid per
        tensor, one scale per `scale_block` elements as checkpoints store them (hf_model_utils.py:199-215); the tile-stat pass
        dequantizes on the fly (qa_tile_stats_fp8) and everything behind the table is unchanged."""
        if source not in ("bf16", "fp8"):
            raise ValueError("source must be 'bf16' or 'fp8'")
        # stats_group = G > 0: the device-resident pass (run / run_graph) issues the tile-stat pass and the delta records of G
        # tensors at a time as ONE descriptor-array launch each (qa_tile_stats_batch, qa_greedy_init_deltas_batch) instead of
        # one launch per tensor.  Off by default: on cfg5 (768 expert tensors in one CUDA graph) one launch per tensor lets
        # every tensor's chain start behind its own 17 us tile-stat kernel, a group's chains wait for the whole group
        # (15.6 ms per step ungrouped, 17.2 / 20.8 / 21.9 ms with G = 8 / 32 / 96; profiles/r2_cfg5_group_sweep.txt).  The
        # entry points are for callers without a graph, where 3 000 launches per step cost host time.
        if stats_group is None:
            stats_group = 0
        self.stats_group = int(stats_group) if source == "bf16" else 0
        self.source, self.scale_block = source, (int(scale_block[0]), int(scale_block[1]))
        self.device = device or engine._require_cuda()
        self.perm_cache = bool(perm_cache)
        self.metric, self.threshold, self.seed = metric, float(threshold), int(seed)
        self.tile_formats = list(tile_formats)
        self.shapes = [tuple(int(v) for v in s) for s in shapes]
        # one stream per tensor; a long list (one MoE layer = hundreds of equal tensors) is throughput-bound on SM time, not
        # on one tensor's latency: more tensors in flight on smaller clusters (cluster_cap, applied while enqueueing)
        self.cluster_cap = 2 if len(self.shapes) > 32 else 0
        n_streams = min(32 if self.cluster_cap else 16, len(self.shapes)) if n_streams is None else n_streams
        # Cluster kernels (resolve / init / chain) can only start when a whole GPC's worth of SMs is free at once, which a
        # streaming kernel that keeps refilling every SM rarely allows: they go on high-priority streams, the tile-stat
        # kernels on normal-priority ones, so the block scheduler drains SMs for a pending cluster first.
        self.streams = [torch.cuda.Stream(device=self.device, priority=-1) for _ in range(max(1, n_streams))]
        self.side_streams = [torch.cuda.Stream(device=self.device, priority=-1) for _ in range(max(1, n_streams))]
        self.side2_streams = [torch.cuda.Stream(device=self.device, priority=-1) for _ in range(max(1, n_streams))]
        # The tile-stat kernels are bandwidth-bound and each fills the GPU: run concurrently they only slow each other
        # down, and the largest tensor - whose init/chain is the critical path - would get its table last.  A short
        # list of large tensors therefore streams its tile-stat passes one after the other, largest first; a long list
        # of small ones (one MoE layer = 768 tensors) keeps a few streams to hide launch gaps.
        self.stats_streams = [torch.cuda.Stream(device=self.device) for _ in range(1 if len(self.shapes) <= 16 else 4)]
        self._stats_rr = 0
        self.prefetch = metric != "atol" and len(self.tile_formats) >= 2
        self.perm_cache = self.perm_cache and self.prefetch
        L = _lib.lib()
        self.slots = []
        rng0 = engine.make_rng(self.seed, self.device)
        # Permutations #1..#3 depend only on (seed, ntiles): tensors with the same tile count share them (every expert of a
        # MoE layer, every layer of a model).  The first such tensor in run order (largest first) draws them.
        nts = [(-(-r // 32)) * (-(-c // 32)) for (r, c) in self.shapes]
        leader_of = {}
        for i in sorted(range(len(nts)), key=lambda i: -nts[i]):
            leader_of.setdefault(nts[i], i)
        for idx, (r, c) in enumerate(self.shapes):
            nt = nts[idx]
            lead = leader_of[nt] == idx
            self.slots.append({
                "leader": leader_of[nt],
                "rows": r, "cols": c, "ntiles": nt, "numel": r * c,
                "x": torch.empty(r * c, dtype=torch.bfloat16 if source == "bf16" else torch.uint8, device=self.device),
                "scale": None if source == "bf16" else torch.ones((-(-r // self.scale_block[0]), -(-c // self.scale_block[1])),
                                                                   dtype=torch.float32, device=self.device),
                "table": torch.zeros((NSTAT, nt), dtype=torch.float64, device=self.device),
                "assignment": torch.empty(nt, dtype=torch.int8, device=self.device),
                "counts": torch.zeros(NFMT, dtype=torch.int64, device=self.device),
                "state": torch.zeros(24, dtype=torch.float64, device=self.device),
                "sums": torch.zeros(8, dtype=torch.float64, device=self.device),
                "work": torch.empty(max(L.qa_greedy_work_bytes(nt), L.qa_greedy_par_work_bytes(nt)), dtype=torch.uint8,
                                    device=self.device),
                "rng": rng0.clone(),
                "pre_order": torch.empty((2, nt), dtype=torch.int32, device=self.device) if lead else None,
                "rngs": torch.stack([rng0, rng0, rng0]).contiguous() if lead else None,   # stream states after permutations #1, #2, #3
                "init": torch.empty(L.qa_greedy_init_bytes(nt), dtype=torch.uint8, device=self.device),
                "jarr": torch.empty((3, nt), dtype=torch.int32, device=self.device) if lead else None,
                "apply_work": torch.empty((2, L.qa_perm_apply_work_bytes(nt)), dtype=torch.uint8, device=self.device) if lead else None,
                "ev": torch.cuda.Event(),
                "ev_a2": torch.cuda.Event(),
                "ev_a3": torch.cuda.Event(),
                "ev2": torch.cuda.Event(),
                "ev3": torch.cuda.Event(),
            })
        for s_ in self.slots:                 # followers read the leader's permutations
            ld = self.slots[s_["leader"]]
            s_["pre_order"], s_["rngs"] = ld["pre_order"], ld["rngs"]
        if self.perm_cache:                   # ... or everybody reads the process-wide cache
            for s_ in self.slots:
                hit = cached_permutations(self.device, self.seed, s_["ntiles"], len(self.tile_formats))
                s_["pre_order"], s_["rngs"] = hit["pre_order"], hit["rngs"]
        self._groups = []
        if self.stats_group > 0:
            run_order = sorted(range(len(self.slots)), key=lambda i: -self.slots[i]["ntiles"])
            for g0 in range(0, len(run_order), self.stats_group):
                members = run_order[g0:g0 + self.stats_group]
                descs, n, items, blocks = engine.batch_descriptors(
                    [(self.slots[i]["x"].data_ptr(), self.slots[i]["table"].data_ptr(), self.slots[i]["init"].data_ptr(),
                      self.slots[i]["rows"], self.slots[i]["cols"]) for i in members], self.device)
                grp = {"members": members, "descs": descs, "n": n, "items": items, "blocks": blocks, "ev": torch.cuda.Event()}
                self._groups.append(grp)
                for i in members:
                    self.slots[i]["group"] = grp
        self._rng0 = rng0
        self._graphs = {}
        self.trace = None            # set to {} to record per-tensor stage events during eager run() (see timeline())
        self._order = _lib.int32_array([engine.FMT_INDEX[f] for f in self.tile_formats])
        # kernels of ours per tensor and step.  atol: tile_stats + greedy + assignment_sums.  pcc / mae: tile_stats,
        # init sums, init deltas, the chain (two launches with three or more formats) and the prefetched permutations (one
        # chained resolve kernel, 7 grid kernels per apply); a pipelined large tensor adds two tile_stats and two init launches
        self.launches_per_step = 0
        for s in self.slots:
            if metric == "atol":
                n = 3
            elif not self.prefetch:
                n = 4
            else:
                lead = self.slots[s["leader"]] is s
                n = 5 if len(self.tile_formats) >= 3 else 4
                if self.perm_cache and len(self.tile_formats) >= 3:
                    n -= 1                       # resident permutations: the chain is one launch
                if lead and not self.perm_cache:
                    n += (2 + 2 * 7) if len(self.tile_formats) >= 3 else (1 + 7)
            if self.stats_group > 0:
                n -= 1 if metric == "atol" else 2            # tile-stat pass and delta records come from the group launches
            elif metric != "atol" and s["ntiles"] >= self.PIPELINE_MIN_TILES and -(-s["rows"] // 32) >= 8:
                n += 4
            self.launches_per_step += n
        self.launches_per_step += len(self._groups) * (1 if metric == "atol" else 2)

    # ---- data movement -------------------------------------------------------------------
    def load_device(self, tensors) -> None:
        """Copy the inputs (host or device) into the resident buffers: bf16 tensors, or (uint8 e4m3fn bytes, float32 inverse
        scale grid) pairs for source="fp8"."""
        for slot, t in zip(self.slots, tensors):
            self._copy_in(slot, t)

    def _copy_in(self, slot, t) -> None:
        if self.source == "fp8":
            w, sc = t
            w = w.view(torch.uint8) if w.dtype != torch.uint8 else w
            slot["x"].copy_(w.reshape(-1), non_blocking=True)
            slot["scale"].copy_(sc.reshape(slot["scale"].shape), non_blocking=True)
        else:
            slot["x"].copy_(t.reshape(-1), non_blocking=True)

    def total_bytes(self) -> int:
        """bf16-equivalent bytes of the weights (2 per element: the unit of BASELINE's metric, whatever the storage format)."""
        return sum(2 * s["numel"] for s in self.slots)

    def input_bytes(self) -> int:
        """Bytes the tile-stat pass actually reads per step (and an end-to-end step copies to the device)."""
        if self.source == "fp8":
            return sum(s["numel"] + 4 * s["scale"].numel() for s in self.slots)
        return self.total_bytes()

    def _stats(self, slot, mode, lo, hi, sp) -> None:
        """One tile-stat launch over tile rows [lo, hi) of the slot's table."""
        L = _lib.lib()
        if self.source == "fp8":
            sc = slot["scale"]
            check(L.qa_tile_stats_fp8(slot["x"].data_ptr(), sc.data_ptr(), slot["rows"], slot["cols"], slot["cols"], sc.shape[0],
                                      sc.shape[1], 0xF, mode, slot["table"].data_ptr(), lo, hi, None, sp), "qa_tile_stats_fp8")
        else:
            check(L.qa_tile_stats_rows(slot["x"].data_ptr(), _lib.QA_DT_BF16, slot["rows"], slot["cols"], slot["cols"], 0xF, mode,
                                       slot["table"].data_ptr(), lo, hi, sp), "qa_tile_stats_rows")

    # ---- compute -------------------------------------------------------------------------
    def _enqueue(self, slot, stream, stats: bool = True, assign: bool = True, side=None, pre_event=None) -> None:
        """pre_event: the tensor's table (and delta records) come from a group launch that signals this event; only the
        per-tensor cluster kernels are enqueued here."""
        L = _lib.lib()
        sp = stream.cuda_stream
        pre = assign and self.prefetch and side is not None

        def mark(tag, on=None):
            if self.trace is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(on or stream)
                self.trace.setdefault(id(slot), {})[tag] = ev

        mark("start")
        lead = self.slots[slot["leader"]] is slot
        cached = pre and self.perm_cache           # permutations already resident: nothing to draw, nothing to wait for
        if cached:
            side, side2 = side
            side2.wait_stream(stream)
            with torch.cuda.stream(side2):
                slot["rng"].copy_(self._rng0, non_blocking=True)
            lead = False
        elif pre and not lead:
            side, side2 = side
            side2.wait_stream(stream)
            with torch.cuda.stream(side2):
                slot["rng"].copy_(self._rng0, non_blocking=True)      # off the stats -> init -> chain path
        if pre and lead and not cached:
            # the first permutations depend only on (seed, ntiles): draw them on side streams while the tile-stat pass
            # streams the tensor.  Resolves chain through the RNG state (#1 -> #2 -> #3, one cluster each); each apply
            # only needs its own swap targets and runs as grid kernels, #2's on a second side stream next to resolve #3.
            side, side2 = side
            three = len(self.tile_formats) >= 3
            side.wait_stream(stream)
            if three:
                # every tensor restarts the seeded stream: a 40-byte copy node, kept off the stats -> init -> chain path
                # (side2 is idle until the second resolve is done; the chain joins it before its first launch)
                side2.wait_stream(stream)
                with torch.cuda.stream(side2):
                    slot["rng"].copy_(self._rng0, non_blocking=True)
            # resolves #1 (stream position only) and #2 in one launch: the cluster keeps its SMs while the tile-stat
            # kernels flood the rest of the GPU.  #3 is a second launch so that #2's apply - all the first chain launch
            # needs - can start as soon as #2 is resolved; #3 has until the later passes start.
            resolved = slot["ev"] if self.trace is None else torch.cuda.Event(enable_timing=True)
            engine.enqueue_perm_prefetch(self._rng0, slot["ntiles"], three,
                                         (slot["jarr"], slot["pre_order"], slot["rngs"], slot["apply_work"]), side, side2,
                                         (resolved, slot["ev_a2"], slot["ev_a3"]))
            if self.trace is not None:
                self.trace.setdefault(id(slot), {})["resolve"] = resolved
            mark("prefetch", side)
        mode = STATS_FAST if self.metric == "mae" else STATS_FAST_APPROX_ABS
        iargs = (slot["table"].data_ptr(), slot["ntiles"], METRIC_CODE[self.metric], self._order, len(self.tile_formats),
                 slot["init"].data_ptr())
        split = 0            # tile rows in the first piece of a pipelined table (0: one piece)
        if stats:
            ss = self.stats_streams[self._stats_rr % len(self.stats_streams)]
            self._stats_rr += 1
            ss.wait_stream(stream)                       # the tensor's input is in place (H2D copy / previous pass)
            tiles_h, tiles_w = -(-slot["rows"] // 32), -(-slot["cols"] // 32)
            if assign and self.metric != "atol" and slot["ntiles"] >= self.PIPELINE_MIN_TILES and tiles_h >= 8:
                # Large tensor: the sequential initial sums spend most of their rounds on the first few thousand tiles
                # (the running sums double often while they are small).  Produce the table in two pieces and let the
                # sums over the first piece run while the tile-stat pass streams the rest of the tensor.
                first = max(self.PIPELINE_FIRST_TILES, slot["ntiles"] // 8)       # first cut: about an eighth of the tiles
                split = max(1, min(tiles_h - 2, -(-first // tiles_w)))
                split2 = max(split + 1, tiles_h // 2)                      # second cut: half of the tensor
                self._stats(slot, mode, 0, split, ss.cuda_stream)
                slot["ev2"].record(ss)
                self._stats(slot, mode, split, split2, ss.cuda_stream)
                slot["ev3"].record(ss)
                self._stats(slot, mode, split2, tiles_h, ss.cuda_stream)
                stream.wait_event(slot["ev2"])
                check(L.qa_greedy_init_sums_range(*iargs, 0, split * tiles_w, sp), "qa_greedy_init_sums_range")
                stream.wait_event(slot["ev3"])
                check(L.qa_greedy_init_sums_range(*iargs, split * tiles_w, split2 * tiles_w, sp), "qa_greedy_init_sums_range")
                split = split2
            else:
                self._stats(slot, mode, 0, tiles_h, ss.cuda_stream)
            stream.wait_stream(ss)
            mark("stats")
        elif pre_event is not None:
            stream.wait_event(pre_event)
            mark("stats")
        if assign:
            if not pre or (lead and len(self.tile_formats) < 3):
                slot["rng"].copy_(self._rng0, non_blocking=True)      # every tensor restarts the seeded stream
            args = (slot["table"].data_ptr(), slot["ntiles"], float(slot["numel"]),
                    METRIC_CODE[self.metric], self.threshold, self._order, len(self.tile_formats),
                    slot["rng"].data_ptr(), slot["assignment"].data_ptr(), slot["counts"].data_ptr(),
                    slot["state"].data_ptr(), slot["work"].data_ptr())
            if self.metric == "atol":
                check(L.qa_greedy_assign(*args, sp), "qa_greedy_assign")
            else:
                # initial sums + delta records on the main stream (overlaps the prefetch), then the chain
                if stats:
                    # the delta records are a plain grid kernel: on the tile-stat stream right behind this tensor's pass,
                    # next to the (latency-bound, one-cluster) sums rather than in front of them
                    check(L.qa_greedy_init_deltas(*iargs, ss.cuda_stream), "qa_greedy_init_deltas")
                    tiles_w = -(-slot["cols"] // 32)
                    check(L.qa_greedy_init_sums_range(*iargs, split * tiles_w, slot["ntiles"], sp), "qa_greedy_init_sums_range")
                    stream.wait_stream(ss)
                else:
                    if pre_event is None:
                        check(L.qa_greedy_init_deltas(*iargs, sp), "qa_greedy_init_deltas")
                    check(L.qa_greedy_init_sums_range(*iargs, 0, slot["ntiles"], sp), "qa_greedy_init_sums_range")
                mark("init")
                pargs = args + (slot["pre_order"].data_ptr() if pre else None, slot["rngs"][1].data_ptr() if pre else None,
                                slot["init"].data_ptr())
                nf = len(self.tile_formats)
                SKIP = 1          # QA_GREEDY_SKIP_FINAL_STREAM: nobody reads slot['rng'] after the run (the reference drops its generator too)
                ld = self.slots[slot["leader"]]
                if pre and nf >= 3:
                    # passes 0-1 only need permutation #2 (applied on side2 while #3 is still being drawn); the later
                    # passes wait for the speculative #3 (applied last on the leader's side stream)
                    stream.wait_stream(side2)                 # own seed copy (and, for a leader, apply #2)
                    if cached:                                # both permutations are resident: one launch for all passes
                        check(L.qa_greedy_assign_passes(*pargs, 0, nf, SKIP, sp), "qa_greedy_assign_passes")
                    else:
                        stream.wait_event(ld["ev_a2"])
                        check(L.qa_greedy_assign_passes(*pargs, 0, 2, 0, sp), "qa_greedy_assign_passes")
                        stream.wait_event(ld["ev_a3"])
                        check(L.qa_greedy_assign_passes(*pargs, 2, nf, SKIP, sp), "qa_greedy_assign_passes")
                else:
                    if pre:
                        stream.wait_stream(side2 if not lead else side)
                        if not cached:
                            stream.wait_event(ld["ev_a2"])
                    check(L.qa_greedy_assign_passes(*pargs, 0, nf, SKIP, sp), "qa_greedy_assign_passes")
            mark("chain")
            if self.metric == "atol":      # the cluster kernel leaves the final sums (and max) in `state`
                check(L.qa_assignment_sums(slot["table"].data_ptr(), slot["ntiles"], slot["assignment"].data_ptr(), -1,
                                           slot["sums"].data_ptr(), sp), "qa_assignment_sums")

    def run(self, stats: bool = True, assign: bool = True) -> None:
        """Enqueue one pass over every tensor; returns immediately (no host sync)."""
        cur = torch.cuda.current_stream(self.device)
        order = sorted(range(len(self.slots)), key=lambda i: -self.slots[i]["ntiles"])   # longest chain first
        prev_cap = _lib.lib().qa_greedy_cluster_cap(self.cluster_cap)
        try:
            self._run_ordered(cur, order, stats, assign)
        finally:
            _lib.lib().qa_greedy_cluster_cap(prev_cap)

    def _run_ordered(self, cur, order, stats, assign) -> None:
        grouped = stats and self.stats_group > 0
        if grouped:
            L = _lib.lib()
            mode = STATS_FAST if self.metric == "mae" else STATS_FAST_APPROX_ABS
            for gi, grp in enumerate(self._groups):
                ss = self.stats_streams[gi % len(self.stats_streams)]
                ss.wait_stream(cur)
                check(L.qa_tile_stats_batch(grp["descs"].data_ptr(), grp["n"], grp["items"], 0xF, mode, ss.cuda_stream), "qa_tile_stats_batch")
                if assign and self.metric != "atol":
                    check(L.qa_greedy_init_deltas_batch(grp["descs"].data_ptr(), grp["n"], grp["blocks"], self._order, len(self.tile_formats),
                                                        ss.cuda_stream), "qa_greedy_init_deltas_batch")
                grp["ev"].record(ss)
        for k, i in enumerate(order):
            st = self.streams[k % len(self.streams)]
            st.wait_stream(cur)
            with torch.cuda.stream(st):
                self._enqueue(self.slots[i], st, stats and not grouped, assign,
                              side=(self.side_streams[k % len(self.side_streams)], self.side2_streams[k % len(self.side2_streams)]),
                              pre_event=self.slots[i]["group"]["ev"] if grouped else None)
        for st in self.streams:
            cur.wait_stream(st)

    def capture(self, stats: bool = True, assign: bool = True) -> None:
        """Record one pass (all tensors, all streams) into a CUDA graph; ``run_graph`` replays it with one launch.
        The pass is ~25 small launches per tensor, so eager enqueueing costs about as much host time as the GPU
        needs to run it; the inputs are the resident ``slot['x']`` buffers, so replays see whatever was loaded last."""
        self.run(stats, assign)                       # eager once: module load, kernel attributes, allocator warm-up
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.run(stats, assign)
        self._graphs[(stats, assign)] = g

    def run_graph(self, stats: bool = True, assign: bool = True) -> None:
        if (stats, assign) not in self._graphs:
            self.capture(stats, assign)
        self._graphs[(stats, assign)].replay()

    def timeline(self) -> list[dict]:
        """After an eager run() with ``self.trace = {}``: per tensor, ms from its stream's start mark to each stage's end."""
        torch.cuda.synchronize(self.device)
        out = []
        t0 = min((tr["start"] for tr in self.trace.values()), key=lambda e: 0)     # any start (all follow the same fork)
        for s in self.slots:
            tr = self.trace.get(id(s), {})
            row = {"shape": (s["rows"], s["cols"])}
            for tag, ev in tr.items():
                if tag != "start":
                    row[tag] = t0.elapsed_time(ev)
            out.append(row)
        return out

    def enqueue_from_host(self, host_tensors) -> None:
        """End-to-end pass, asynchronous half: pinned host bf16 (or fp8 bytes + scale grids) -> device, quantize+score+assign, results into pinned host
        buffers.  Returns immediately; ``finish()`` waits for this pass only, so a caller with two batches can keep the
        PCIe link busy with the next list's inputs while this one computes."""
        cur = torch.cuda.current_stream(self.device)
        order = sorted(range(len(self.slots)), key=lambda i: -self.slots[i]["ntiles"])
        if getattr(self, "_pending", None) is not None:
            cur.wait_event(self._pending)             # a pass still in flight on these buffers goes first
        prev_cap = _lib.lib().qa_greedy_cluster_cap(self.cluster_cap)      # thread-local in the library
        try:
            for k, i in enumerate(order):
                st = self.streams[k % len(self.streams)]
                st.wait_stream(cur)
                with torch.cuda.stream(st):
                    self._copy_in(self.slots[i], host_tensors[i])
                    self._enqueue(self.slots[i], st, side=(self.side_streams[k % len(self.side_streams)], self.side2_streams[k % len(self.side2_streams)]))
                    self._d2h(self.slots[i])                     # behind this tensor's chain, on its own stream
        finally:
            _lib.lib().qa_greedy_cluster_cap(prev_cap)
        self._pending = torch.cuda.Event()
        if not hasattr(self, "_join_stream"):
            self._join_stream = torch.cuda.Stream(device=self.device)
        join = self._join_stream
        for st in self.streams:
            join.wait_stream(st)
        self._pending.record(join)

    def _d2h(self, s) -> None:
        if "h_assignment" not in s:
            s["h_assignment"] = torch.empty(s["ntiles"], dtype=torch.int8).pin_memory()
            s["h_counts"] = torch.empty(NFMT, dtype=torch.int64).pin_memory()
            s["h_state"] = torch.empty(24, dtype=torch.float64).pin_memory()
        s["h_assignment"].copy_(s["assignment"], non_blocking=True)
        s["h_counts"].copy_(s["counts"], non_blocking=True)
        src = s["sums"] if self.metric == "atol" else s["state"]
        s["h_state"][: src.numel()].copy_(src, non_blocking=True)

    def finish(self) -> list[dict]:
        """Wait for the pass started by ``enqueue_from_host`` and return its results."""
        self._pending.synchronize()
        return [self._result(s, s["h_assignment"], s["h_counts"], s["h_state"][: (8 if self.metric == "atol" else 24)]) for s in self.slots]

    def run_from_host(self, host_tensors) -> list[dict]:
        """End-to-end pass: pinned host bf16 -> device, quantize+score+assign, results back to host."""
        self.enqueue_from_host(host_tensors)
        return self.finish()

    def _result(self, s, a, c, sums) -> dict:
        counts = {f: int(c[i]) for i, f in enumerate(MIXED)}
        v = sums.numpy()
        if self.metric != "atol":      # state = {sx, sx2, sy, sy2, sxy, sabs, flags, value, cycles x3, max|x-y|, ...}
            v = np.array([v[0], v[1], v[2], v[3], v[4], v[5], v[11]])
        out = {"assignment": a.numpy().reshape(-(-s["rows"] // 32), -(-s["cols"] // 32)).copy(), "counts": counts,
               "metrics": engine.metrics_from_sums(v, s["numel"]), "state": sums.numpy().copy()}
        if self.metric != "atol":
            # certificate inputs (see MixedTileGreedyCompression): flag bits of the initial sums / relaxed grid, and a lower bound
            # of min |value - thr| / thr over every decision the chain evaluated
            full = sums.numpy()
            out["flags"], out["min_margin"] = int(full[6]) & 7, float(full[20])
        return out

    def collect(self) -> list[dict]:
        """Device -> host: assignment maps, counts and exact pcc/mae/atol per tensor (synchronises)."""
        packs = []
        for s in self.slots:
            packs.append((s["assignment"].to("cpu", non_blocking=True), s["counts"].to("cpu", non_blocking=True),
                          (s["sums"] if self.metric == "atol" else s["state"]).to("cpu", non_blocking=True)))
        torch.cuda.current_stream(self.device).synchronize()
        return [self._result(s, a, c, sums) for s, (a, c, sums) in zip(self.slots, packs)]

    def d2h_bytes(self) -> int:
        return sum(s["ntiles"] + 8 * NFMT + 8 * 8 for s in self.slots)
