#!/usr/bin/env python
"""GPU experiment (not part of the product): rollout roofline fraction vs batch size / horizon / control mode.
Usage (on the GPU box): python scripts/gpu_sweep_rollout.py [B,N,mode ...]"""
import os, sys, json, subprocess, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import openkite_b200 as okb

FLOPS = 1888.0
props = okb.load_properties(os.path.join(ROOT, "data", "umx_radian.yaml"))
eng = okb.Engine(props, okb.KITE, device=0)
eng_id = okb.Engine(props, okb.KITE_ID, device=0)
peak = eng.fp64_peak(20000)
print("fp64 peak %.2f TF" % peak)
cases = sys.argv[1:] or ["262144,100,1", "262144,1000,1", "1048576,100,1", "1048576,1000,1", "1048576,1000,3", "1048576,1000,0",
                         "1048576,1000,2"]
def smi():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw,temperature.gpu", "--format=csv,noheader,nounits"],
                              capture_output=True, text=True).stdout.strip()
    except Exception:
        return "?"
for c in cases:
    B, N, mode = [int(t) for t in c.split(",")]
    if mode == 5:          # config-5 shape: id-variant RHS, per-sample coefficients, shared control log, fused cost
        import numpy as np
        p = eng_id.synth_id_params(B)
        kk = np.arange(N)
        ul = torch.from_numpy(np.stack([0.1 * np.ones(N), 0.1 * np.sign(np.sin(0.037 * kk)), 0.1 * np.sign(np.sin(0.023 * kk + 1))], 1)).cuda()
        x1, _ = eng.synth_inputs(1, 1)
        y = eng_id.rollout(x1, ul, N, 1e-3, okb.U_SHARED, p=p[:, :1].contiguous(), save_every=1)["traj"].reshape(N, 13).contiguous()
        xi = x1.expand(13, B).contiguous(); xf = eng.empty(13, B); co = eng.empty(B); st = torch.empty(B, dtype=torch.int32, device="cuda")
        go = lambda: eng_id.rollout(xi, ul, N, 1e-3, okb.U_SHARED, p=p, y=y, out=xf, cost_out=co, status_out=st)
        go(); torch.cuda.synchronize()
        ts = []
        for r in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); go(); b.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = min(ts); tf = (FLOPS + 39) * B * N / (ms * 1e-3) / 1e12
        print("B=%d N=%d mode=5(id sweep)  best %.3f ms  %.3e steps/s  %.2f TF  frac %.4f" % (B, N, ms, B * N / ms * 1e3, tf, tf / peak))
        del p, xi, xf, co, st
        torch.cuda.empty_cache()
        continue
    x0, u = eng.synth_inputs(B, N if mode == 1 else 1)
    if mode == 0: uu = u[0].contiguous()
    elif mode == 1: uu = u
    elif mode == 2: uu = u[:, :, 0].contiguous().expand(1, 3).repeat(N, 1).contiguous()
    else: uu = None
    xf = eng.empty(13, B)
    def go():
        if mode == 3: eng.rollout(None, None, N, 1e-3, okb.U_SYNTH, out=xf, want_status=False, B=B)
        else: eng.rollout(x0, uu, N, 1e-3, mode, out=xf, want_status=False)
    go(); torch.cuda.synchronize()
    ts = []
    for r in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); go(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ms = min(ts)
    tf = FLOPS * B * N / (ms * 1e-3) / 1e12
    print("B=%d N=%d mode=%d  ms=%s  best %.3f ms  %.3e steps/s  %.2f TF  frac %.4f   smi[%s]" % (B, N, mode, ["%.2f" % t for t in ts], ms, B * N / ms * 1e3, tf, tf / peak, smi()))
    del x0, u, uu, xf
    torch.cuda.empty_cache()
