#!/usr/bin/env python
"""GPU experiment (not part of the product): time the RK4 + sensitivity step (Phi, Gamma) for one or more batch sizes.
Usage (on the GPU box): python scripts/gpu_bench_sens.py [B ...]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctypes as C
import torch
import openkite_b200 as okb
FLOPS = 27800.0
eng = okb.Engine(okb.load_properties(os.path.join(ROOT, "data", "umx_radian.yaml")), okb.KITE, device=0)
peak = eng.fp64_peak(20000)
reps = int(os.environ.get("REPS", "10"))
for B in [int(a) for a in sys.argv[1:]] or [262144, 1048576]:
    x0, u = eng.synth_inputs(B, 1)
    us = u[0].contiguous()
    outs = (eng.empty(13, B), eng.empty(169, B), eng.empty(39, B))
    w = eng.workspace(eng.L.kite_rk4_sens_work_bytes(B))
    pp = lambda t: C.c_void_p(t.data_ptr())
    def sens():
        eng._use_torch_stream()
        eng._ck(eng.L.kite_rk4_sens_step(eng.ctx, B, B, 0.02, pp(x0), pp(us), pp(outs[0]), pp(outs[1]), pp(outs[2]), pp(w)))
    for _ in range(3): sens()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): sens()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    tf = FLOPS * B / (ms * 1e-3) / 1e12
    print("sens B=%d: %.3f ms  %.3e units/s  %.2f TF  frac %.4f (peak %.2f)  out %.0f GB/s" % (
        B, ms, B / ms * 1e3, tf, tf / peak, peak, 1768.0 * B / ms / 1e6))
