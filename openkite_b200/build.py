"""In-tree build of libkite_b200.so for sm_100a with nvcc (cross-compiles without a GPU).

    python -m openkite_b200.build [--force] [--verbose]

Each kernel family is its own translation unit so the eight host cores build them in parallel.
The .so stays in-tree (git-ignored, shipped to the GPU box by gpurun).
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
LIB = os.path.join(HERE, "libkite_b200.so")
LIB_CASADI = os.path.join(HERE, "libkite_casadi.so")     # CasADi external-function shim (host C++, links LIB)
UNITS = ["kite_capi", "launch_point", "launch_rollout_a", "launch_rollout_b", "launch_sens", "launch_ekf", "launch_colloc"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xptxas", "-v"]


def _newest_header():
    t = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            if f.endswith((".h", ".cuh")):
                t = max(t, os.path.getmtime(os.path.join(root, f)))
    return t


def _compile(unit, verbose):
    src = os.path.join(CSRC, unit + ".cu")
    obj = os.path.join(OBJ, unit + ".o")
    log = os.path.join(OBJ, unit + ".ptxas.log")
    cmd = ["nvcc", *NVCC_FLAGS, "-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(log, "w") as fh:
        fh.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s" % (unit, r.stdout + r.stderr))
    if verbose:
        print(r.stderr)
    return obj


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = _newest_header()
    todo = []
    for u in UNITS:
        src = os.path.join(CSRC, u + ".cu")
        obj = os.path.join(OBJ, u + ".o")
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            todo.append(u)
    if todo:
        with ThreadPoolExecutor(max_workers=min(8, len(todo))) as ex:
            list(ex.map(lambda u: _compile(u, verbose), todo))
    objs = [os.path.join(OBJ, u + ".o") for u in UNITS]
    if todo or not os.path.exists(LIB):
        cmd = ["nvcc", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    build_casadi_shim(force or bool(todo))
    return LIB


def build_casadi_shim(force=False):
    """libkite_casadi.so: `dynamics`, `dyn_jacobian`, `Aero`, `RK4` in CasADi's external-function C convention
    (csrc/kite_casadi.cpp, plain g++), on top of the B = 1 entry points of libkite_b200.so."""
    src = os.path.join(CSRC, "kite_casadi.cpp")
    inc = os.path.join(os.path.dirname(HERE), "include")
    newest = max([os.path.getmtime(src), os.path.getmtime(os.path.join(CSRC, "kite_sparsity.h"))] +
                 [os.path.getmtime(os.path.join(inc, "openkite", f)) for f in os.listdir(os.path.join(inc, "openkite"))])
    if not force and os.path.exists(LIB_CASADI) and os.path.getmtime(LIB_CASADI) >= newest:
        return LIB_CASADI
    cmd = ["g++", "-O2", "-std=c++14", "-fPIC", "-shared", "-Wall", "-o", LIB_CASADI, src, "-L" + HERE, "-lkite_b200",
           "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("libkite_casadi.so failed:\n" + r.stdout + r.stderr)
    return LIB_CASADI


def resource_report():
    """(kernel, registers, spill bytes) parsed from the saved ptxas logs."""
    import re

    rows = []
    for u in UNITS:
        log = os.path.join(OBJ, u + ".ptxas.log")
        if not os.path.exists(log):
            continue
        txt = open(log).read()
        for m in re.finditer(r"Compiling entry function '(\w+)'[^\n]*\n[^\n]*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n[^\n]*Used (\d+) registers", txt):
            rows.append((m.group(1), int(m.group(5)), int(m.group(2)), int(m.group(3)), int(m.group(4))))
    return rows


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(lib)
    for name, regs, stack, sst, sld in resource_report():
        print("%-70s regs=%3d stack=%4d spill_st=%4d spill_ld=%4d" % (name[:70], regs, stack, sst, sld))
