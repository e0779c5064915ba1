"""Graph-replayed times of the parts of one o_proj step (stats, init, prefetch, chain) alone and combined."""
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

from quantization_analysis_b200 import _lib, synthetic
from quantization_analysis_b200._lib import METRIC_CODE, STATS_FAST_APPROX_ABS, check
from quantization_analysis_b200.batch import GreedyBatch

dev = torch.device("cuda:0")
name = [n for n in synthetic.ATTN_NAMES if "o_proj" in n][0]
shape = synthetic.DEEPSEEK_R1_SHAPES[name]
b = GreedyBatch([shape], metric="pcc", threshold=0.999, seed=123)
b.load_device([synthetic.device_randn_bf16(shape, 7, dev)])
b.run(); torch.cuda.synchronize()
L = _lib.lib()
s = b.slots[0]
n = s["ntiles"]


def stats(st):
    check(L.qa_tile_stats(s["x"].data_ptr(), _lib.QA_DT_BF16, s["rows"], s["cols"], s["cols"], 0, 0xF, STATS_FAST_APPROX_ABS,
                          s["table"].data_ptr(), st.cuda_stream), "stats")


def init(st):
    iargs = (s["table"].data_ptr(), n, METRIC_CODE["pcc"], b._order, 4, s["init"].data_ptr())
    check(L.qa_greedy_init_deltas(*iargs, st.cuda_stream), "init deltas")
    check(L.qa_greedy_init_sums_range(*iargs, 0, n, st.cuda_stream), "init sums")


def resolves(st, k):
    check(L.qa_perm_resolve_chain(b._rng0.data_ptr(), n, k, 0b110 & ((1 << k) - 1), s["jarr"].data_ptr(), s["rngs"].data_ptr(),
                                  st.cuda_stream), "resolve chain")


def apply(st, i):
    check(L.qa_perm_apply(s["jarr"][i + 1].data_ptr(), n, None, s["pre_order"][i].data_ptr(), s["apply_work"][i].data_ptr(), st.cuda_stream), "apply")


def chain(st):
    chain_passes(st, 0, 4)


def chain_passes(st, b0, e0):
    if b0 == 0:
        s["rng"].copy_(b._rng0, non_blocking=True)
    check(L.qa_greedy_assign_passes(s["table"].data_ptr(), n, float(s["numel"]), METRIC_CODE["pcc"], 0.999, b._order, 4,
                                    s["rng"].data_ptr(), s["assignment"].data_ptr(), s["counts"].data_ptr(), s["state"].data_ptr(),
                                    s["work"].data_ptr(), s["pre_order"].data_ptr(), s["rngs"][1].data_ptr(), s["init"].data_ptr(),
                                    b0, e0, 0, st.cuda_stream), "chain passes")


def timed(fn, reps=20):
    g = torch.cuda.CUDAGraph()
    fn(torch.cuda.current_stream()); torch.cuda.synchronize()
    with torch.cuda.graph(g):
        fn(torch.cuda.current_stream())
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


side = torch.cuda.Stream()


def full(st, with_stats=True, with_pre=True):
    if with_pre:
        side.wait_stream(st)
        with torch.cuda.stream(side):
            resolves(side, 3); apply(side, 0); apply(side, 1)
    if with_stats:
        stats(st)
    init(st)
    if with_pre:
        st.wait_stream(side)
    chain(st)


print(f"stats                {timed(stats):7.1f} us")
print(f"init                 {timed(init):7.1f} us")
print(f"stats -> init        {timed(lambda st: (stats(st), init(st))):7.1f} us")
print(f"resolve x1           {timed(lambda st: resolves(st, 1)):7.1f} us")
print(f"resolve x3           {timed(lambda st: resolves(st, 3)):7.1f} us")
print(f"apply x1             {timed(lambda st: apply(st, 0)):7.1f} us")
print(f"chain                {timed(chain):7.1f} us")
print(f"chain passes 0-1     {timed(lambda st: chain_passes(st, 0, 2)):7.1f} us")
print(f"chain passes 0-1, 2-3 {timed(lambda st: (chain_passes(st, 0, 2), chain_passes(st, 2, 4))):7.1f} us")
print(f"init -> chain        {timed(lambda st: (init(st), chain(st))):7.1f} us")
print(f"stats->init->chain   {timed(lambda st: (stats(st), init(st), chain(st))):7.1f} us")
print(f"prefetch | init -> chain   {timed(lambda st: full(st, with_stats=False)):7.1f} us")
print(f"prefetch | stats -> init -> chain   {timed(full):7.1f} us")
side = torch.cuda.Stream(priority=-1)
print(f"same, prefetch stream at high priority   {timed(full):7.1f} us")
lo, hi = torch.cuda.Stream(priority=0), torch.cuda.Stream(priority=-1)


def full2(st):
    side.wait_stream(st); lo.wait_stream(st); hi.wait_stream(st)
    with torch.cuda.stream(side):
        resolves(side, 3); apply(side, 0); apply(side, 1)
    with torch.cuda.stream(lo):
        stats(lo)
    hi.wait_stream(lo)
    with torch.cuda.stream(hi):
        init(hi)
        hi.wait_stream(side)
        chain(hi)
    st.wait_stream(hi)


print(f"stats on a normal-priority stream, cluster kernels on high-priority streams   {timed(full2):7.1f} us")
