"""Phase breakdown of the greedy cluster kernel on the cfg2 tensors (CUDA events + in-kernel clock64 diagnostics).
Usage (GPU box): python profiles/greedy_phases.py [tensor-name-substring]"""
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

from quantization_analysis_b200 import engine, synthetic


def timed(fn, reps=5):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    for _ in range(reps):
        e0.record(); out = fn(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best, out


def main():
    sel = sys.argv[1] if len(sys.argv) > 1 else ""
    dev = torch.device("cuda:0")
    for name in synthetic.ATTN_NAMES:
        shape = synthetic.DEEPSEEK_R1_SHAPES[name]
        if sel not in name:
            continue
        x = synthetic.device_randn_bf16(shape, 7, dev)
        p = engine.prepare_tiles(x)
        table = engine.tile_stats(p, engine.MIXED_FORMATS, exact_abs=False)
        nt = table.shape[1]
        fm = list(engine.MIXED_FORMATS)
        t_pre, pre = timed(lambda: engine.greedy_prefetch(engine.make_rng(123), nt))
        t_init, init = timed(lambda: engine.greedy_init(table, "pcc", fm))
        t_g, (a, c, st) = timed(lambda: engine.greedy_assign(table, p.numel, "pcc", 0.999, fm, engine.make_rng(123), prefetched=pre, init=init))
        t_i, (a2, c2, st2) = timed(lambda: engine.greedy_assign(table, p.numel, "pcc", 0.999, fm, engine.make_rng(123)))
        assert torch.equal(a, a2)
        s = st.cpu().numpy(); s2 = st2.cpu().numpy()
        mhz = 1e-3
        print(f"{name} {shape} ntiles={nt} cluster={int(s[12])} counts={c.tolist()}")
        print(f"  prefetch {t_pre*1e3:.0f} us | init kernel {t_init*1e3:.0f} us | chain (staged) {t_g*1e3:.0f} us | single call {t_i*1e3:.0f} us (incl. rng/alloc launches)")
        for tag, v in (("staged", s), ("single", s2)):
            print(f"  [{tag}] kcycles: init {v[8]*mhz:.0f} (pos-sums {v[13]*mhz:.0f}, signed {v[14]*mhz:.0f}, rounds {int(v[15])}) "
                  f"perm {v[9]*mhz:.0f} (resolve {v[21]*mhz:.0f}, apply {v[22]*mhz:.0f}, sweeps {int(v[23]) % 65536}, rounds {int(v[23]) // 65536}) "
                  f"chain {v[10]*mhz:.0f} (gather {v[18]*mhz:.0f}, commit {v[17]*mhz:.0f}, kernel total {v[16]*mhz:.0f}, chunks {int(v[19])}, min margin {v[20]:.2e}, "
                  f"chain rounds {int(v[6]) // 65536}) flags {int(v[6]) % 65536}")


if __name__ == "__main__":
    main()
