#!/bin/bash
# SASS evidence for profiles/: opcode histogram of every kernel in libljmd.so and the hot loop of each
# (Blackwell-specific mnemonics: FFMA2/FMUL2/FADD2 packed FP32, UBLKCP + SYNCS = cp.async.bulk + mbarrier,
# UCGABAR = hardware cluster barrier, LDGSTS = cp.async).   scripts/sass_evidence.sh OUTDIR
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd); OUT=${1:-$ROOT/profiles/r2}; mkdir -p "$OUT"
LIB=$ROOT/jax_tpus_benchmark_physics_simulation_b200/libljmd.so
cuobjdump -sass "$LIB" > /tmp/ljmd_all.sass
python - "$OUT" <<'PY'
import re, sys, collections
out = sys.argv[1]
txt = open('/tmp/ljmd_all.sass').read()
blocks = re.split(r"\n\s*Function : ", txt)[1:]
keys = ["FFMA2", "FMUL2", "FADD2", "FFMA", "MUFU.RCP", "UBLKCP", "SYNCS", "UCGABAR", "LDGSTS", "LDS", "STS", "SHFL",
        "ATOMG", "RED", "MEMBAR", "FENCE", "BAR.SYNC", "HMMA", "UTMALDG", "UTCHMMA"]
with open(f"{out}/sass_opcode_histogram.txt", "w") as f:
    f.write("opcode counts per kernel of libljmd.so (cuobjdump -sass, sm_100a)\n")
    for b in blocks:
        name = b.split("\n", 1)[0].strip()
        ops = re.findall(r"/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_.]*)", b)
        c = collections.Counter()
        for o in ops:
            for k in keys:
                if o == k or o.startswith(k + ".") or o.startswith(k + "_"):
                    c[k] += 1
        short = re.sub(r"_GLOBAL__N__[0-9a-f]+_\d+_", "", name)
        f.write(f"\n{short}\n  {len(ops)} instructions: " + ", ".join(f"{k} {c[k]}" for k in keys if c[k]) + "\n")
# hot loops: the instructions around the first UBLKCP / densest FFMA2 window of the main kernels (the force-only
# instantiations, VIR = false; the <..., true> ones add the virial on energy steps)
def excerpt(kern, anchor, before, after, fname, title):
    b = next(x for x in blocks if kern in x.split("\n", 1)[0])
    lines = [l for l in b.split("\n") if re.match(r"\s+/\*[0-9a-f]{4,6}\*/", l)]
    idx = [i for i, l in enumerate(lines) if anchor in l]
    if not idx:
        return
    i = idx[len(idx) // 2]
    with open(f"{out}/{fname}", "w") as f:
        f.write(title + "\n")
        for l in lines[max(0, i - before): i + after]:
            f.write(re.sub(r"\s*/\* 0x[0-9a-f]+ \*/", "", l).rstrip() + "\n")
excerpt("cells_persistent_kernelILb0E", "UBLKCP", 60, 12, "sass_cells_bulk_copy_issue.txt",
        "cells_persistent_kernel: arming the mbarrier (SYNCS.ARRIVE.TRANS64) and the bulk copies (UBLKCP) of a unit")
excerpt("cells_persistent_kernelILb0E", "SYNCS.PHASECHK", 6, 130, "sass_cells_pair_loop.txt",
        "cells_persistent_kernel: mbarrier wait (SYNCS.PHASECHK.TRYWAIT) and the packed-FP32 pair loop over one-byte list entries")
excerpt("ap_persistent_kernelILi3ELb1ELb0E", "SHFL", 40, 60, "sass_allpairs_tile_loop.txt",
        "ap_persistent_kernel<3,true>: Newton's-third-law tile step (packed pair evaluation + shuffle rotation)")
excerpt("ap_cluster_kernelILb1ELb0E", "UCGABAR", 80, 10, "sass_cluster_step.txt",
        "ap_cluster_kernel<true>: end of a step: st.shared::cluster pushes and the hardware cluster barrier (UCGABAR)")
PY
ls -la "$OUT"/sass_*
