#!/usr/bin/env python3
"""Per-kernel SASS opcode summary of libqa_b200.so (cuobjdump, no GPU needed): registers / spills from the cubin's resource
usage and the static instruction mix of every kernel.  Writes profiles/r2_sass_summary.md."""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
lib = ROOT / "quantization_analysis_b200" / "libqa_b200.so"
sass = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
res = subprocess.run(["cuobjdump", "-res-usage", str(lib)], capture_output=True, text=True, check=True).stdout
usage = {}
cur = None
for line in res.splitlines():
    m = re.search(r"Function (\S+):", line)
    if m:
        cur = m.group(1)
        continue
    m = re.search(r"REG:(\d+).*?SHARED:(\d+).*?LOCAL:(\d+)", line)
    if m and cur:
        usage[cur] = (int(m.group(1)), int(m.group(2)), int(m.group(3)))
        cur = None
kern = collections.OrderedDict()
fn = None
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        fn = m.group(1)
        kern[fn] = collections.Counter()
        continue
    m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", line)
    if m and fn:
        kern[fn][m.group(1)] += 1
demangle = subprocess.run(["c++filt"], input="\n".join(kern), capture_output=True, text=True).stdout.splitlines()
INTEREST = ["FFMA2", "FADD2", "FMUL2", "FFMA", "FADD", "FMUL", "FMNMX", "FMNMX3", "HFMA2", "DFMA", "DADD", "DMUL", "F2F", "LOP3", "SHF",
            "PRMT", "IADD3", "IMAD", "LDG", "STG", "LDS", "STS", "LDL", "STL", "SHFL", "BAR", "SYNCS", "UBLKCP", "F2FP", "ATOMS", "MUFU", "UCGABAR_ARV", "UCGABAR_WAIT"]
out = ["# SASS summary of libqa_b200.so (sm_100a), round 2", "",
       "`python profiles/sass_summary.py` (cuobjdump -sass / -res-usage on the in-tree library; static counts, whole kernel).", "",
       "| kernel | regs | smem B | local B | instrs | " + " | ".join(INTEREST) + " |", "|---|---:|---:|---:|---:|" + "---:|" * len(INTEREST)]
for (mangled, c), name in zip(kern.items(), demangle):
    base = collections.Counter()
    for op, n in c.items():
        base[op.split(".")[0]] += n
    wide = sum(n for op, n in c.items() if op.startswith("LDG") and ".256" in op)
    short = re.sub(r"\(.*", "", name).replace("void ", "").replace("qa::", "")
    u = usage.get(mangled, ("?", "?", "?"))
    out.append(f"| `{short}` | {u[0]} | {u[1]} | {u[2]} | {sum(c.values())} | " + " | ".join(str(base.get(k, 0)) for k in INTEREST) + " |"
               + (f" <!-- {wide} x LDG.256 -->" if wide else ""))
out += ["", "Markers: packed fp32 (`FFMA2` / `FADD2` / `FMUL2`), `FMNMX3`, `FMNMX.XORSIGN` and 256-bit `LDG.E...256` loads in the streaming kernels;",
        "`SYNCS` (mbarrier) + distributed-shared-memory stores and `UCGABAR_*` in the cluster kernels; TMA bulk copies (`UBLKCP.S.G`, completing on",
        "`SYNCS.ARRIVE.TRANS64` mbarriers) in `sdot_pipe_kernel`; `F2FP` = the hardware e4m3x2 -> f16x2 and f32 -> bf16x2",
        "conversions of `stats_f32_kernel`; no tensor-core instructions (the path is not a contraction)."]
(ROOT / "profiles" / "r2_sass_summary.md").write_text("\n".join(out) + "\n")
print("\n".join(out[:12]))
