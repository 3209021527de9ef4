#!/usr/bin/env python
"""SASS listing of the headline kernels -> profiles/<round>_sass_headline_kernels.txt
(evidence of UBLKCP = cp.async.bulk, SYNCS = mbarrier, LDG.E.*.CONSTANT = ld.global.nc)."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
rnd = sys.argv[1] if len(sys.argv) > 1 else "r1"
WANT = [r"csr_stream_kernelILi512ELi4ELi2ELi4096ELi1ELb1ELb0ELi0EiE",   # C2 / C5 headline: row-wise staged tiles, plain epilogue
        r"csr_stream_kernelILi512ELi4ELi2ELi4096ELi1ELb1ELb0ELi1ExE",   # ... push epilogue, 64-bit offsets (C5 boundary rows)
        r"hll_warp_kernelILi0EE",                                        # HLL headline (C2)
        r"hll_pipe_kernelILi2ELi0EE", r"csr_pipe_kernelILi2ELi176EiE",   # short rows (C1): per-warp bulk-copy rings
        r"sell_kernelILi0ELb0EE", r"sell_kernelILi2ELb0EE",              # C3 column panels: first / later panels
        r"sell_kernelILi0ELb1EE",                                        # C4 virtual rows
        r"sell_mm_kernelILi2ELi0ELb1EE"]                                 # SpMM, 2 right-hand sides, virtual rows
txt = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, "spmv_scpa_b200/lib/libspmv_b200.so")],
                     capture_output=True, text=True).stdout
parts = re.split(r"(?=\t\tFunction : )", txt)
out = []
for p in parts:
    m = re.match(r"\t\tFunction : (\S+)", p)
    if m and any(re.search(w, m.group(1)) for w in WANT):
        code = [l for l in p.splitlines() if re.search(r"/\*[0-9a-f]{4}\*/", l) or "Function" in l]
        ops = re.findall(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", "\n".join(code))
        hist = {}
        for o in ops:
            k = o.split(".")[0]
            hist[k] = hist.get(k, 0) + 1
        out.append(f"==== {m.group(1)}\n# opcode histogram: " +
                   ", ".join(f"{k}:{v}" for k, v in sorted(hist.items(), key=lambda kv: -kv[1])) + "\n" +
                   "\n".join(re.sub(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", "", l) for l in code
                             if not re.match(r"\s*/\* 0x", l)))
open(os.path.join(ROOT, "profiles", f"{rnd}_sass_headline_kernels.txt"), "w").write("\n\n".join(out) + "\n")
print(len(out), "kernels dumped")
