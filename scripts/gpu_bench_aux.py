#!/usr/bin/env python
"""GPU experiment / secondary figures: EKF predict (config 5), NMPC collocation G + dG (config 4) and the identification
sweep rollout (config 5: per-sample coefficients, shared control log, fused cost).  Not the headline bench."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import openkite_b200 as okb

which = sys.argv[1:] or ["ekf", "colloc", "id"]
prm = okb.load_properties(os.path.join(ROOT, "data", "umx_radian.yaml"))
eng = okb.Engine(prm, okb.KITE, device=0)
peak = eng.fp64_peak(20000)
golden = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))["cases"]

def timeit(fn, reps=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps

def report(name, B, ms, flops, bytes_):
    tf = flops * B / (ms * 1e-3) / 1e12
    print("%-28s B=%d  %.3f ms  %.3e units/s  %.2f TF (%.1f%% of %.1f)  %.0f GB/s algorithmic" % (
        name, B, ms, B / ms * 1e3, tf, 100 * tf / peak, peak, bytes_ * B / ms / 1e6))

if "ekf" in which:
    B = 1 << 20
    x, u = eng.synth_inputs(B, 1)
    u0 = u[0].contiguous()
    W = np.diag(np.array([.5, .5, .5, .5, .5, .5, .5, .1, .1, .01, .05, .05, .05]) ** 2)
    P = torch.from_numpy((10 * W).reshape(169, 1)).cuda().expand(169, B).contiguous()
    out = (eng.empty(13, B), eng.empty(169, B))
    ms = timeit(lambda: eng.ekf_predict(x, u0, 0.0084, P, W, out=out))
    report("ekf_predict", B, ms, 13400.0, 8.0 * (13 + 3 + 169 + 13 + 169))
    z = x[6:13].contiguous()
    V = np.eye(7) * 1e-4
    xs, Ps = out[0].clone(), out[1].clone()
    ms = timeit(lambda: eng.ekf_update(z, V, xs, Ps))
    report("ekf_update", B, ms, 6000.0, 8.0 * (7 + 13 + 169) * 2)

if "colloc" in which:
    B, M = 65536, 11
    c = golden["colloc_nmpc_P5_S2_scaled"]
    rng = np.random.default_rng(0)
    z = torch.from_numpy(np.ascontiguousarray((np.array(c["z"])[None, :] * (1 + 0.01 * rng.standard_normal((B, 209)))).T)).cuda()
    from openkite_b200.collocation import comp_diff_matrix
    compD = comp_diff_matrix(5, 2)
    out = (eng.empty(M * 15, B), eng.empty(M * 225, B), eng.empty(M * 60, B), eng.empty(B))
    ms = timeit(lambda: eng.colloc_eval(z, M, compD, 0.25, c["sx"], c["su"], out=out))
    report("colloc_eval G+JX+JU", B, ms, 31600.0, 8.0 * (209 + 165 + 11 * 285))
    outs = (out[0], eng.empty(M * eng.colloc_nnz_per_node(), B), out[3])
    ms = timeit(lambda: eng.colloc_eval_sparse(z, M, compD, 0.25, c["sx"], c["su"], out=outs))
    report("colloc_eval_sparse G+JV", B, ms, 31600.0, 8.0 * (209 + 165 + 11 * eng.colloc_nnz_per_node()))
    out2 = (out[0], None, None, out[3])
    ms = timeit(lambda: eng.colloc_eval(z, M, compD, 0.25, c["sx"], c["su"], out=out2))
    report("colloc_eval G only", B, ms, 11 * 420.0 + 2000, 8.0 * (209 + 165))

if "id" in which:
    e = okb.Engine(prm, okb.KITE_ID, device=0)
    B, N = 1 << 20, 200
    pnom = np.array(golden["rhs_id"]["nominal"]["p"])
    rng = np.random.default_rng(1)
    p = torch.from_numpy(np.ascontiguousarray((pnom[None] * (1 + 0.1 * (2 * rng.random((B, 21)) - 1))).T)).cuda()
    x0 = torch.from_numpy(np.array(golden["rollout_config1"]["x0"]).reshape(13, 1)).cuda().expand(13, B).contiguous()
    k = np.arange(N)
    u = torch.from_numpy(np.stack([0.1 * np.ones(N), 0.1 * np.sign(np.sin(0.37 * k)), 0.1 * np.sign(np.sin(0.23 * k + 1))], 1)).cuda().contiguous()
    y = torch.zeros(N, 13, dtype=torch.float64, device="cuda")
    xf = e.empty(13, B)
    ms = timeit(lambda: e.rollout(x0, u, N, 1e-3, okb.U_SHARED, p=p, y=y, out=xf, want_status=False), reps=3)
    report("id sweep rollout (x%d steps)" % N, B * N, ms, 1888.0, 0.0)
