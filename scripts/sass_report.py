#!/usr/bin/env python
"""profiles/<tag>_ptxas_resources.txt and profiles/<tag>_sass_histogram.txt from the in-tree build (no GPU needed):
registers / stack / spill bytes of every kernel (`-Xptxas -v`), and per kernel the SASS instruction histogram, the TMA /
mbarrier mnemonics that prove the bulk-tensor paths, and -- for the rollout kernels -- the FP64 instructions of the stage
loop by the number of distinct vector-register operands not served by the reuse cache (the operand-delivery cost model of
DESIGN.md section 7: cycles = sum of max(2, operands)).  profiles/<tag>_stage_loop.txt lists every FP64 instruction of those
stage loops with its uncached-operand count and the source line it comes from (nvdisasm line table of the -lineinfo build).
    python scripts/sass_report.py <tag>"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from openkite_b200 import build as kb  # noqa: E402

FP64 = ("DFMA", "DMUL", "DADD", "DSETP")


def parse(sass):
    rows = []
    for ln in sass.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(@!?U?P[0-9T]+ )?([A-Z0-9_]+)([.\w]*)\s*(.*?);", ln)
        if m:
            rows.append((int(m.group(1), 16), m.group(3), m.group(3) + m.group(4), [o.strip() for o in m.group(5).split(",")]))
    return rows


def source_lines(obj, fn):
    """{address: 'file:line'} of kernel `fn` in `obj`, from nvdisasm's line table."""
    out, src, inside = {}, "?", False
    with tempfile.TemporaryDirectory() as d:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(obj)], cwd=d, capture_output=True)
        for cub in sorted(f for f in os.listdir(d) if f.endswith(".cubin")):
            txt = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(d, cub)], capture_output=True, text=True).stdout
            for ln in txt.splitlines():
                if ln.startswith("//----"):
                    inside = fn in ln
                    continue
                if not inside:
                    continue
                m = re.match(r'\s*//## File "([^"]+)", line (\d+)', ln)
                if m:
                    src = "%s:%s" % (os.path.basename(m.group(1)), m.group(2))
                    continue
                m = re.match(r"\s+/\*([0-9a-f]{4,})\*/", ln)
                if m:
                    out[int(m.group(1), 16)] = src
    return out


def operand_model(rows, lo, hi, listing=None):
    prev, stats, cyc = {}, collections.Counter(), 0
    for a, op, full, ops in rows:
        if not (lo <= a <= hi):
            continue
        srcs = ops[1:] if op != "DSETP" else ops[2:]
        cur = {}
        if op in FP64:
            nv, seen = 0, set()
            for i, o in enumerate(srcs):
                mm = re.match(r"[-|~]*(R\d+)(\.reuse)?", o)
                if mm and mm.group(1) != "RZ":
                    reg = mm.group(1)
                    if not (prev.get(i) == reg or reg in seen):
                        nv += 1
                    seen.add(reg)
                    if mm.group(2):
                        cur[i] = reg
            stats[nv] += 1
            cyc += max(2, nv)
            if listing is not None:
                listing.append((a, nv, full, ", ".join(ops)))
        else:
            for i, o in enumerate(srcs):
                mm = re.match(r"[-|~]*(R\d+)\.reuse", o)
                if mm:
                    cur[i] = mm.group(1)
        prev = cur
    return stats, cyc


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "r2"
    kb.build()
    out = os.path.join(ROOT, "profiles")
    with open(os.path.join(out, "%s_ptxas_resources.txt" % tag), "w") as fh:
        fh.write("nvcc %s  (per kernel: registers, stack frame, spill stores, spill loads in bytes)\n" % " ".join(kb.NVCC_FLAGS))
        for name, regs, stack, sst, sld in kb.resource_report():
            dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
            fh.write("%-88s regs=%3d stack=%4d spill_st=%4d spill_ld=%4d\n" % (dem[:88], regs, stack, sst, sld))
    loop_fh = open(os.path.join(out, "%s_stage_loop.txt" % tag), "w")
    loop_fh.write("FP64 instructions of the rollout stage loops: address, vector-register operands not served by the reuse cache, "
                  "instruction, source line\n")
    with open(os.path.join(out, "%s_sass_histogram.txt" % tag), "w") as fh:
        fh.write("cuobjdump -sass of openkite_b200/_obj/*.o (sm_100a): instruction histograms of the product kernels\n")
        for unit, pat in (("launch_rollout_a", "k_rk4_rolloutILi1ELb0ELb0"), ("launch_rollout_b", "k_rk4_rolloutILi2ELb0ELb1"),
                          ("launch_sens", "k_sens_fusedILb0ELb0ELb1"), ("launch_ekf", "k_ekf_predict_tmaILb0ELb0"),
                          ("launch_ekf", "k_ekf_update"), ("launch_colloc", "k_colloc_evalILb0ELi4ELi0"),
                          ("launch_colloc", "k_colloc_evalILb0ELi4ELi1")):
            obj = os.path.join(kb.OBJ, unit + ".o")
            syms = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
            fn = [ln.split()[-1] for ln in syms.splitlines() if ln.strip().startswith("Function :") and pat in ln]
            if not fn:
                continue
            sass = subprocess.run(["cuobjdump", "-sass", "-fun", fn[0], obj], capture_output=True, text=True).stdout
            rows = parse(sass)
            hist = collections.Counter(op for _, op, _, _ in rows)
            dem = subprocess.run(["c++filt", fn[0]], capture_output=True, text=True).stdout.strip()
            fh.write("\n== %s\n" % dem)
            fh.write("instructions %d: %s\n" % (len(rows), ", ".join("%s %d" % kv for kv in hist.most_common(24))))
            tma = collections.Counter(full for _, op, full, _ in rows if op in ("UTMALDG", "UTMASTG", "SYNCS", "UTMACMDFLUSH", "UBLKCP") or full.startswith("LDGSTS"))
            if tma:
                fh.write("TMA / mbarrier: %s\n" % ", ".join("%s %d" % kv for kv in sorted(tma.items())))
            local = sum(hist[k] for k in ("STL", "LDL"))
            fh.write("local-memory instructions (spills): %d\n" % local)
            loops = []
            for a, op, _, ops in rows:
                if op == "BRA":
                    t = re.search(r"0x([0-9a-f]+)", " ".join(ops))
                    if t and int(t.group(1), 16) < a:
                        loops.append((int(t.group(1), 16), a))
            if "rollout" in pat and loops:
                lo, hi = loops[0]
                body = collections.Counter(op for a, op, _, _ in rows if lo <= a <= hi)
                listing = []
                stats, cyc = operand_model(rows, lo, hi, listing)
                n = sum(stats.values())
                src = source_lines(obj, fn[0])
                loop_fh.write("\n== %s  stage loop 0x%x-0x%x\n" % (dem, lo, hi))
                by_line = collections.Counter(src.get(a, "?") for a, nv, _, _ in listing if nv >= 3)
                loop_fh.write("three-operand instructions by source line: %s\n" % ", ".join("%s %d" % kv for kv in sorted(by_line.items())))
                for a, nv, full, ops in listing:
                    loop_fh.write("%04x %s %-7s %-44s %s\n" % (a, "*3" if nv >= 3 else " %d" % nv, full, ops, src.get(a, "?")))
                fh.write("stage loop 0x%x-0x%x: %d instructions, %d on the FP64 pipe (%s)\n" %
                         (lo, hi, sum(body.values()), n, ", ".join("%s %d" % (k, body[k]) for k in FP64)))
                fh.write("  FP64 instructions by uncached vector-register operands: %s -> %d cycles per stage at max(2, operands) (%.2f per instruction)\n" %
                         (dict(sorted(stats.items())), cyc, cyc / max(n, 1)))
    loop_fh.close()
    print(open(os.path.join(out, "%s_sass_histogram.txt" % tag)).read())


if __name__ == "__main__":
    main()
