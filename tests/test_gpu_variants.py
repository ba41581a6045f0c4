"""Every compiled kernel instantiation against the oracle.

The kernels are templates instantiated per model (kite / identification / rigid body), per control mode, per output format
and per store path (TMA or direct stores), and the C ABI picks one from the arguments of the call.  The parity suite
(test_gpu_parity.py, test_gpu_fullsize.py) covers the headline paths; this file launches the others: the rigid-body and
per-trajectory-coefficient rollouts in every control mode with trajectory and fitting-cost output, the multi-chunk host
pipeline, rigid and tether-arm sensitivities, the rigid and identification EKF predict, the EKF update at ragged shapes and
in a predict -> update loop, and the collocation kernels across node counts on both of their code paths (compact rows of
compD from the constant bank for M <= 16 nodes and <= 8 non-zeros per row, the dense walk otherwise).  Most calls go
through the C ABI with a leading dimension ld > B and check that the padding columns keep their sentinel.

KERNEL_TESTS at the bottom maps every built kernel to the tests that launch it; test_every_kernel_has_a_test (CPU) fails
when the library gains an instantiation that no test names.
Tolerance as everywhere: |gpu - ref| <= 1e-9 max(|ref|, 1).
"""
import ast
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import assert_close
from test_gpu_parity import aos, okb, params, soa  # noqa: F401  (fixtures)

RTOL = 1e-9
SENT = -7.0                              # sentinel of output buffers: columns >= B (and unused slots) must keep it
ERR_ARG, ERR_STATE = -1, -4              # kite_status
KITE, KITE_ID, RIGID_BODY = 0, 1, 2
U_CONST, U_PER_STEP, U_SHARED, U_SYNTH = 0, 1, 2, 3
# weights of the identification cost, kite_identification_test.cpp:193 (restated, not read from the kernel source)
ID_COST_Q = np.array([1e3, 1e2, 1e2, 1e2, 1e2, 1e2, 1e1, 1e1, 1e2, 1e2, 1e2, 1e2, 1e2])
# the 21 identification coefficients inside the oracle's 39-vector (order of kite.cpp:571-572)
IDX21 = [9, 10, 12, 13, 14, 15, 17, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29, 30, 31, 32]
ARM = (0.012, -0.004, 0.021)


# ---------------------------------------------------------------- fixtures and helpers ------------------
@pytest.fixture(scope="module")
def engines(okb, params):
    es = {k: okb.Engine(params, k) for k in (KITE, KITE_ID, RIGID_BODY)}
    yield es
    for e in es.values():
        e.close()


@pytest.fixture(scope="module")
def arm_setup(okb, params, yaml_path):
    """Engine and oracle with the same non-zero tether arm."""
    from oracle.oracle_py import Oracle, PARAM_FIELDS, params_from_yaml
    p2 = okb.KiteParams.from_buffer_copy(params)
    p2.rx, p2.ry, p2.rz = ARM
    prm = params_from_yaml(yaml_path)
    for key, v in zip(("rx", "ry", "rz"), ARM):
        prm[PARAM_FIELDS.index(("tether", key))] = v
    e = okb.Engine(p2, KITE)
    yield e, Oracle(prm)
    e.close()


@pytest.fixture(scope="module")
def pnom(golden):
    return np.array(golden["rhs_id"]["nominal"]["p"])


def ptr(t, off=0):
    return None if t is None else C.c_void_p(t.data_ptr() + 8 * off)


def padded(a, ld, off=0):
    """numpy AoS [B, n...] -> CUDA [n][ld] with the units in columns off .. off + B - 1, zeros elsewhere"""
    a = np.asarray(a, dtype=np.float64).reshape(len(a), -1)
    t = torch.zeros(a.shape[1], ld, dtype=torch.float64, device="cuda")
    t[:, off:off + a.shape[0]] = torch.from_numpy(np.ascontiguousarray(a.T)).cuda()
    return t


def sentinel(*shape, dtype=torch.float64):
    return torch.full(shape, SENT, dtype=dtype, device="cuda")


def assert_untouched(t, lo, hi, what):
    """Columns outside [lo, hi) of the last axis still hold the sentinel."""
    t = t.detach().cpu().double()
    rest = torch.cat([t[..., :lo].reshape(-1), t[..., hi:].reshape(-1)])
    assert rest.numel() == 0 or float((rest - SENT).abs().max()) == 0.0, "%s: padding written" % what


def same_bits(a, b):
    """Bitwise equality of two tensors, NaN included (torch.equal treats NaN as unequal to itself)."""
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.nan_to_num(a), torch.nan_to_num(b))


def p_batch(pnom, B, seed):
    rng = np.random.default_rng(seed)
    return pnom[None] * (1 + 0.1 * (2 * rng.random((B, 21)) - 1))


def kite_p21(params):
    """The context's own 21 identification coefficients (kite_synth_id_params order)."""
    return np.array([params.CL0, params.CLa_total, params.CD0_total, params.CYb, params.Cm0, params.Cma, params.Cnb,
                     params.Clb, params.CLq, params.Cmq, params.CYr, params.Cnr, params.Clr, params.CYp, params.Clp,
                     params.Cnp, params.CLde, params.CYdr, params.Cmde, params.Cndr, params.Cldr])


# ---------------------------------------------------------------- 0. pointwise --------------------------
@pytest.mark.gpu
def test_point_eval_rigid_and_coefficient_batches(engines, oracle, pnom):
    """k_point_eval for the rigid body and with per-unit coefficients, on ragged batches (not only B = 1 goldens)."""
    for B in (31, 257):
        x = oracle.synth_x0(40, B); u = oracle.synth_controls(40, B, 1)[:, 0, :]
        rb = engines[RIGID_BODY]
        assert_close(aos(rb.rhs(soa(x), soa(u))), oracle.rhs(x, u, kind=RIGID_BODY), RTOL, what="rigid f B=%d" % B)
        Jx, Ju = rb.jac(soa(x), None)
        rJx, _ = oracle.jac(x, u, kind=RIGID_BODY)
        assert_close(aos(Jx, 13, 13), rJx, RTOL, what="rigid Jx B=%d" % B)
        assert float(Ju.abs().max()) == 0.0
        e = engines[KITE_ID]
        p = p_batch(pnom, B, B)
        assert_close(aos(e.rhs(soa(x), soa(u), soa(p))), oracle.rhs(x, u, p=p, kind=KITE_ID), RTOL, what="id f B=%d" % B)
        Jx, Ju = e.jac(soa(x), soa(u), soa(p))
        rJx, rJu = oracle.jac(x, u, p=p, kind=KITE_ID)
        assert_close(aos(Jx, 13, 13), rJx, RTOL, what="id Jx B=%d" % B)
        assert_close(aos(Ju, 13, 3), rJu, RTOL, what="id Ju B=%d" % B)
        assert_close(aos(e.aero(soa(x), soa(u), soa(p))), oracle.aero(x, u, p=p, kind=KITE_ID), RTOL, what="id aero B=%d" % B)


# ---------------------------------------------------------------- 1. rollout matrix ---------------------
# (B, ld, save_every) -- ragged sizes around the 128-thread block; ld > B for half of them; save_every 1, 7 (N = 23 is not a
# multiple of 7) and N.  The fitting cost is on for every other size, so both branches of the kernel run.
ROLL_N, ROLL_H = 23, 1e-3
ROLL_SHAPES = [(1, 1, 1), (31, 40, 7), (33, 33, ROLL_N), (77, 128, 1), (255, 255, 7), (257, 263, ROLL_N)]
ROLL_CASES = [   # (model kind, control mode, per-trajectory coefficients, controls given)
    (KITE, U_CONST, False, True), (KITE, U_PER_STEP, False, True), (KITE, U_SHARED, False, True), (KITE, U_SYNTH, False, True),
    (KITE_ID, U_CONST, True, True), (KITE_ID, U_PER_STEP, True, True), (KITE_ID, U_SHARED, True, True),
    (KITE_ID, U_SYNTH, True, True),
    (RIGID_BODY, U_CONST, False, True), (RIGID_BODY, U_CONST, False, False), (RIGID_BODY, U_PER_STEP, False, True),
    (RIGID_BODY, U_SHARED, False, True),
]


def run_rollout(e, B, ld, N, h, mode, x0=None, u=None, p=None, y=None, save_every=0, index0=0):
    """kite_rk4_rollout through the C ABI on [rows][ld] buffers.  Inputs are numpy (x0 [B,13]; u [B,3] | [B,N,3] | [N,3];
    p [B,21]; y [N,13]).  The trajectory buffer has one extra slot and every output starts as the sentinel; the padding
    columns and the extra slot are checked here.  Returns (rc, dict of numpy AoS results)."""
    xd = padded(x0, ld) if x0 is not None else None
    if u is None or mode == U_SYNTH:
        ud = None
    elif mode == U_CONST:
        ud = padded(u, ld)
    elif mode == U_PER_STEP:
        ud = torch.zeros(max(N, 1), 3, ld, dtype=torch.float64, device="cuda")
        ud[:N, :, :B] = torch.from_numpy(np.ascontiguousarray(u.transpose(1, 2, 0))).cuda()
    else:
        ud = torch.from_numpy(np.ascontiguousarray(u)).cuda()
    pd = padded(p, ld) if p is not None else None
    yd = torch.from_numpy(np.ascontiguousarray(y)).cuda() if y is not None else None
    nsave = N // save_every if save_every else 0
    xf, cost, st = sentinel(13, ld), (sentinel(ld) if y is not None else None), sentinel(ld, dtype=torch.int32)
    traj = sentinel(nsave + 1, 13, ld) if save_every else None
    e._use_torch_stream()
    rc = e.L.kite_rk4_rollout(e.ctx, B, ld, N, h, ptr(xd), ptr(ud), mode, ptr(pd), ptr(xf), ptr(traj), save_every, ptr(yd),
                              ptr(cost), ptr(st), index0)
    torch.cuda.synchronize()
    if rc != 0:
        for t in (xf, traj, cost, st):
            if t is not None:
                assert_untouched(t, 0, 0, "failed call")
        return rc, None
    assert_untouched(xf, 0, B, "xf")
    assert_untouched(st, 0, B, "status")
    out = dict(xf=aos(xf[:, :B]), status=st[:B].cpu().numpy())
    if traj is not None:
        assert_untouched(traj[:nsave], 0, B, "traj")
        assert_untouched(traj[nsave], 0, 0, "traj sentinel slot")
        out["traj"] = traj[:nsave, :, :B].cpu().numpy().transpose(0, 2, 1)        # [slot][B][13]
    if cost is not None:
        assert_untouched(cost, 0, B, "cost")
        out["cost"] = cost[:B].cpu().numpy()
    return rc, out


def id_cost_ref(traj, y):
    """(1/N) sum_k sum_c Q_c (y[k][c] - x_c(k+1))^2 from the oracle trajectory [B][N+1][13]."""
    N = y.shape[0]
    d = y[None, :, :] - traj[:, 1:, :]
    return (ID_COST_Q[None, None, :] * d * d).sum((1, 2)) / N


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode,percoef,with_u", ROLL_CASES,
                         ids=["%s-%s%s%s" % ("kite id rigid".split()[k], "const per_step shared synth".split()[m],
                                              "-p" if pc else "", "" if wu else "-no_u") for k, m, pc, wu in ROLL_CASES])
def test_rollout_matrix(engines, oracle, pnom, kind, mode, percoef, with_u):
    """k_rk4_rollout<mode, rigid, per-trajectory coefficients>: final state, trajectory slots, fitting cost and status of
    every unit against the oracle, padding and the sentinel trajectory slot untouched."""
    e = engines[kind]
    N, h = ROLL_N, ROLL_H
    for j, (B, ld, se) in enumerate(ROLL_SHAPES):
        i0 = 1000 + 977 * j
        x0 = oracle.synth_x0(i0, B)
        uall = oracle.synth_controls(i0, B, N)                              # [B][N][3]
        p = p_batch(pnom, B, j) if percoef else None
        u_ref = {U_CONST: uall[:, 0, :].copy(), U_PER_STEP: uall, U_SHARED: uall[0].copy(), U_SYNTH: None}[mode]
        if mode == U_CONST and not with_u:
            u_ref = np.zeros((B, 3))
        if mode == U_SYNTH:
            rxf, rtraj = oracle.rollout(None, None, N, h, u_mode=3, p=p, kind=kind, want_traj=True, traj0=i0, n=B)
        else:
            rxf, rtraj = oracle.rollout(x0, u_ref, N, h, u_mode=mode, p=p, kind=kind, want_traj=True)
        y = None
        if j % 2 == 0:                                                      # measurement log: a perturbed trajectory
            y = rtraj[0, 1:, :] * (1 + 0.01 * np.sin(np.arange(N * 13).reshape(N, 13)))
        rc, out = run_rollout(e, B, ld, N, h, mode, x0=None if mode == U_SYNTH else x0,
                              u=u_ref if with_u else None, p=p, y=y, save_every=se, index0=i0)
        assert rc == 0
        what = "B=%d ld=%d" % (B, ld)
        assert not out["status"].any(), what
        assert_close(out["xf"], rxf, RTOL, what="xf " + what)
        assert_close(out["traj"], rtraj[:, se::se, :].transpose(1, 0, 2), RTOL, what="traj (save_every %d) %s" % (se, what))
        if y is not None:
            assert_close(out["cost"], id_cost_ref(rtraj, y), RTOL, scale=1e-9, what="cost " + what)


@pytest.mark.gpu
def test_rollout_rejected_arguments(engines, okb, oracle, pnom):
    """Rigid body with synthetic inputs or coefficients is KITE_ERR_STATE; a fitting cost over N = 0 steps (0 / 0) is
    KITE_ERR_ARG on the device and the host entry points; nothing is written."""
    B, ld, N = 33, 40, 5
    x0 = oracle.synth_x0(0, B); u = oracle.synth_controls(0, B, 1)[:, 0, :]
    rb = engines[RIGID_BODY]
    assert run_rollout(rb, B, ld, N, 1e-3, U_SYNTH, save_every=1)[0] == ERR_STATE
    assert run_rollout(rb, B, ld, N, 1e-3, U_CONST, x0=x0, u=u, p=p_batch(pnom, B, 0))[0] == ERR_STATE
    y = np.ones((1, 13))
    for kind in (KITE, KITE_ID, RIGID_BODY):
        e = engines[kind]
        p = p_batch(pnom, B, 1) if kind == KITE_ID else None
        for mode, uu in ((U_CONST, u), (U_SHARED, u[:1]), (U_SYNTH, None)):
            if kind == RIGID_BODY and mode == U_SYNTH:
                continue
            assert run_rollout(e, B, ld, 0, 1e-3, mode, x0=x0, u=uu, p=p, y=y)[0] == ERR_ARG, (kind, mode)
        # without the cost, N = 0 stays legal: the initial states come back
        rc, out = run_rollout(e, B, ld, 0, 1e-3, U_CONST, x0=x0, u=u, p=p)
        assert rc == 0 and np.array_equal(out["xf"], x0)
    e = engines[KITE]
    x0_h = torch.from_numpy(np.ascontiguousarray(x0.T)); u_h = torch.from_numpy(np.ascontiguousarray(u.T))
    xf_h = torch.full((13, B), SENT, dtype=torch.float64); cost_h = torch.full((B,), SENT, dtype=torch.float64)
    y_h = torch.ones(1, 13, dtype=torch.float64)
    hp = lambda t: C.c_void_p(t.data_ptr())
    e.L.kite_reset_stream(e.ctx)
    assert e.L.kite_rk4_rollout_host(e.ctx, B, 0, 1e-3, hp(x0_h), hp(u_h), U_CONST, None, hp(xf_h), hp(y_h), hp(cost_h), None) == ERR_ARG
    assert float((xf_h - SENT).abs().max()) == 0.0 and float((cost_h - SENT).abs().max()) == 0.0
    with pytest.raises(okb.KiteError):
        e.rollout(soa(x0), soa(u), 0, 1e-3, U_CONST, y=torch.ones(1, 13, dtype=torch.float64, device="cuda"))


# ---------------------------------------------------------------- 2. host pipeline, several chunks -----------
def host_chunk(N, u_mode, with_u, with_p):
    """Trajectories per chunk of kite_rk4_rollout_host (restated from rollout_host_pipeline in kite_capi.cu: ~512 MiB of
    per-trajectory input per buffer, a multiple of 1024 trajectories)."""
    u_rows = 0 if not with_u else (3 * N if u_mode == U_PER_STEP else (3 if u_mode == U_CONST else 0))
    bytes_per_traj = 8.0 * (13 + u_rows + (21 if with_p else 0) + 13 + 1) + 4.0
    bc = int(512.0 * 1024 * 1024 / bytes_per_traj)
    return max(1024, (bc // 1024) * 1024)


@pytest.mark.gpu
def test_rollout_host_pipeline_chunks(engines, okb):
    """kite_rk4_rollout_host with three chunks and a ragged last one (both double buffers reused): bitwise the device-pointer
    rollout on the same inputs.  U_PER_STEP with status; U_SHARED with per-trajectory coefficients and the fitting cost."""
    hp = lambda t: C.c_void_p(t.data_ptr())
    # U_PER_STEP, status
    e = engines[KITE]
    N, h = 10, 1e-3
    Bc = host_chunk(N, U_PER_STEP, True, False)
    B = 2 * Bc + 333
    x0, u = e.synth_inputs(B, N, index0=77)
    ref = e.rollout(x0, u, N, h, U_PER_STEP)
    x0_h, u_h = x0.cpu().pin_memory(), u.cpu().pin_memory()
    xf_h = torch.full((13, B), SENT, dtype=torch.float64).pin_memory()
    st_h = torch.full((B,), -1, dtype=torch.int32).pin_memory()
    e.L.kite_reset_stream(e.ctx)
    e._ck(e.L.kite_rk4_rollout_host(e.ctx, B, N, h, hp(x0_h), hp(u_h), U_PER_STEP, None, hp(xf_h), None, None, hp(st_h)))
    assert same_bits(xf_h, ref["xf"].cpu()), "host pipeline (per step) differs from the device rollout"
    assert torch.equal(st_h, ref["status"].cpu())
    del x0, u, x0_h, u_h, xf_h, st_h, ref
    # U_SHARED, per-trajectory coefficients, fitting cost
    e = engines[KITE_ID]
    N = 30
    Bc = host_chunk(N, U_SHARED, True, True)
    B = 2 * Bc + 777
    x0, _ = e.synth_inputs(B, 0, index0=5, want_u=False)
    p = e.synth_id_params(B, index0=11)
    rng = np.random.default_rng(6)
    us = torch.from_numpy(0.1 * rng.standard_normal((N, 3))).cuda()
    y = x0[:, :1].T.repeat(N, 1).contiguous() + 0.01                             # [N][13]
    ref = e.rollout(x0, us, N, h, U_SHARED, p=p, y=y)
    x0_h, p_h, us_h, y_h = x0.cpu().pin_memory(), p.cpu().pin_memory(), us.cpu(), y.cpu()
    xf_h = torch.full((13, B), SENT, dtype=torch.float64).pin_memory()
    cost_h = torch.full((B,), SENT, dtype=torch.float64).pin_memory()
    e.L.kite_reset_stream(e.ctx)
    e._ck(e.L.kite_rk4_rollout_host(e.ctx, B, N, h, hp(x0_h), hp(us_h), U_SHARED, hp(p_h), hp(xf_h), hp(y_h), hp(cost_h), None))
    assert same_bits(xf_h, ref["xf"].cpu()), "host pipeline (shared, p) differs from the device rollout"
    assert same_bits(cost_h, ref["cost"].cpu()), "host pipeline fitting cost differs from the device rollout"
    assert float((cost_h - SENT).abs().min()) > 0.0, "a chunk's fitting cost was never written"


# ---------------------------------------------------------------- 3. sensitivities ---------------------------
def sens_rollout_c(e, B, ld, N, h, x0, uall):
    """kite_rk4_sens_rollout on [N][rows][ld] buffers initialised to the sentinel; padding checked in every slab."""
    xd = padded(x0, ld)
    ud = torch.zeros(N, 3, ld, dtype=torch.float64, device="cuda")
    ud[:, :, :B] = torch.from_numpy(np.ascontiguousarray(uall.transpose(1, 2, 0))).cuda()
    xs, Phi, Gam = sentinel(N, 13, ld), sentinel(N, 169, ld), sentinel(N, 39, ld)
    w = e.workspace(e.L.kite_rk4_sens_work_bytes(B))
    e._use_torch_stream()
    e._ck(e.L.kite_rk4_sens_rollout(e.ctx, B, ld, N, h, ptr(xd), ptr(ud), ptr(xs), ptr(Phi), ptr(Gam), ptr(w)))
    torch.cuda.synchronize()
    for t, name in ((xs, "xs"), (Phi, "Phi"), (Gam, "Gamma")):
        assert_untouched(t, 0, B, "sens rollout %s B=%d ld=%d" % (name, B, ld))
    f = lambda t, *s: t[:, :, :B].cpu().numpy().transpose(2, 0, 1).reshape(B, N, *s)
    return f(xs, 13), f(Phi, 13, 13), f(Gam, 13, 3)


def chained_sens_ref(orc, x0, uall, h, p=None, kind=KITE):
    """Per-step oracle sensitivities, chained (the oracle's sens rollout takes no coefficients)."""
    B, N = uall.shape[0], uall.shape[1]
    xs, Ps, Gs = np.empty((B, N, 13)), np.empty((B, N, 13, 13)), np.empty((B, N, 13, 3))
    x = x0
    for k in range(N):
        x, Ps[:, k], Gs[:, k] = orc.rk4_sens(x, uall[:, k, :].copy(), h, p=p, kind=kind)
        xs[:, k] = x
    return xs, Ps, Gs


def check_sens(got, ref, what):
    for a, b, name in zip(got, ref, ("x", "Phi", "Gamma")):
        assert_close(a, b, RTOL, what="%s %s" % (name, what))


@pytest.mark.gpu
def test_sens_rigid_batches(engines, oracle):
    """k_sens_fused<rigid>: single steps and rollouts of ragged batches against oracle.rk4_sens*(kind=RIGID_BODY)."""
    rb = engines[RIGID_BODY]
    h = 0.02
    for B in (1, 31, 33, 77, 255, 257):
        x = oracle.synth_x0(300 + B, B); u = oracle.synth_controls(300 + B, B, 1)[:, 0, :]
        got = rb.sens_step(soa(x), soa(u), h)
        ref = oracle.rk4_sens(x, u, h, kind=RIGID_BODY)
        check_sens((aos(got[0]), aos(got[1], 13, 13), aos(got[2], 13, 3)), ref, "rigid step B=%d" % B)
        assert float(got[2].abs().max()) == 0.0
    for B, ld, N in ((77, 77, 6), (256, 262, 5), (257, 260, 5)):
        x0 = oracle.synth_x0(17, B); uall = oracle.synth_controls(17, B, N)
        got = sens_rollout_c(rb, B, ld, N, h, x0, uall)
        check_sens(got, oracle.rk4_sens_rollout(x0, uall, h, kind=RIGID_BODY), "rigid rollout B=%d ld=%d" % (B, ld))


@pytest.mark.gpu
def test_sens_tether_arm_rollout(arm_setup):
    """k_sens_fused<arm> over a horizon (N = 6) at even B (TMA output) and odd B (direct stores), ld = B and ld > B."""
    e, orc = arm_setup
    h = 0.02
    for B, ld in ((258, 258), (77, 77), (130, 136), (33, 35)):
        N = 6
        x0 = orc.synth_x0(23, B); uall = orc.synth_controls(23, B, N)
        got = sens_rollout_c(e, B, ld, N, h, x0, uall)
        check_sens(got, orc.rk4_sens_rollout(x0, uall, h), "arm rollout B=%d ld=%d" % (B, ld))


@pytest.mark.gpu
def test_sens_rollout_padded(engines, oracle):
    """kite_rk4_sens_rollout with ld > B: even pitch and B (TMA tensor stores over the N slabs), odd pitch (direct stores).
    The padding of every one of the N slabs keeps its sentinel; both paths agree bitwise."""
    e = engines[KITE]
    h, N = 0.02, 5
    for B in (254, 1, 31, 256):
        x0 = oracle.synth_x0(600, B); uall = oracle.synth_controls(600, B, N)
        ref = oracle.rk4_sens_rollout(x0, uall, h)
        res = []
        for ld in (B + (B & 1) + 8, B + 1 - (B & 1) + 8):                   # even pitch, odd pitch
            got = sens_rollout_c(e, B, ld, N, h, x0, uall)
            check_sens(got, ref, "rollout B=%d ld=%d" % (B, ld))
            res.append(got)
        for a, b in zip(*res):
            assert np.array_equal(a, b), "TMA and direct stores differ (B=%d)" % B


@pytest.mark.gpu
def test_sens_identification_engine(engines, oracle, params):
    """A KITE_ID context without coefficients integrates the model without regularisers with its own coefficients:
    oracle kind=KITE_ID with those coefficients, single steps and a rollout."""
    e = engines[KITE_ID]
    p21 = kite_p21(params)
    h = 0.02
    for B in (33, 256):
        x = oracle.synth_x0(71, B); uall = oracle.synth_controls(71, B, 4)
        p = np.tile(p21, (B, 1))
        got = e.sens_step(soa(x), soa(uall[:, 0, :]), h)
        ref = oracle.rk4_sens(x, uall[:, 0, :].copy(), h, p=p, kind=KITE_ID)
        check_sens((aos(got[0]), aos(got[1], 13, 13), aos(got[2], 13, 3)), ref, "id step B=%d" % B)
        got = sens_rollout_c(e, B, B, 4, h, x, uall)
        check_sens(got, chained_sens_ref(oracle, x, uall, h, p=p, kind=KITE_ID), "id rollout B=%d" % B)


# ---------------------------------------------------------------- 4. EKF -------------------------------------
def random_cov(W, B, seed, scale=0.1):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((B, 13, 13)) * scale
    return 10 * W[None] + A @ A.transpose(0, 2, 1)


def ekf_predict_c(e, B, ld, dt, x, u, P, W):
    """kite_ekf_predict_batch on [rows][ld] buffers (outputs start as the sentinel, padding checked).  u may be None."""
    xd, Pd = padded(x, ld), padded(P.reshape(B, 169), ld)
    ud = padded(u, ld) if u is not None else None
    xn, Pn = sentinel(13, ld), sentinel(169, ld)
    Wh = np.ascontiguousarray(W)
    e._use_torch_stream()
    e._ck(e.L.kite_ekf_predict_batch(e.ctx, B, ld, dt, ptr(xd), ptr(ud), ptr(Pd), Wh.ctypes.data_as(C.c_void_p), ptr(xn),
                                     ptr(Pn), None))
    torch.cuda.synchronize()
    assert_untouched(xn, 0, B, "ekf xn B=%d ld=%d" % (B, ld)); assert_untouched(Pn, 0, B, "ekf Pn B=%d ld=%d" % (B, ld))
    return aos(xn[:, :B]), aos(Pn[:, :B], 13, 13)


@pytest.mark.gpu
def test_ekf_predict_rigid(engines, oracle):
    """Rigid-body EKF predict on both kernels (even B and pitch: TMA boxes; odd: direct loads), with and without u.
    A kite-model predict runs first on the same shapes, so the shared-memory Jacobian tiles hold the kite's entries of rows
    0..5, which the rigid model never writes: the rigid kernels must not read them."""
    W, _ = oracle.ekf_defaults()
    dt = 0.0084
    ek, rb = engines[KITE], engines[RIGID_BODY]
    for B, ld in ((258, 264), (2, 2), (40000, 40000), (77, 77), (257, 260), (40001, 40003)):
        x = oracle.synth_x0(B, B); u = oracle.synth_controls(B, B, 1)[:, 0, :]
        P = random_cov(W, B, B)
        ekf_predict_c(ek, B, ld, dt, x, u, P, W)                                 # leaves kite Jacobian entries behind
        rxn, rPn = oracle.ekf_predict(x, np.zeros((B, 3)), dt, P, W, kind=RIGID_BODY)
        for uu in (u, None):
            xn, Pn = ekf_predict_c(rb, B, ld, dt, x, uu, P, W)
            what = "rigid EKF B=%d ld=%d u=%s" % (B, ld, uu is not None)
            assert_close(xn, rxn, RTOL, what="xn " + what)
            assert_close(Pn, rPn, RTOL, what="Pn " + what)


@pytest.mark.gpu
def test_ekf_predict_identification(engines, oracle, params):
    """KITE_ID context (no regularisers, its own coefficients): x+ from the oracle's RK4 step, Pn = A P A^T + W with
    A = I + dt Jx(x, u) from the oracle's Jacobian (the oracle's ekf_predict takes no coefficients).  TMA and direct."""
    e = engines[KITE_ID]
    W, _ = oracle.ekf_defaults()
    dt = 0.0084
    p21 = kite_p21(params)
    for B, ld in ((130, 130), (77, 80)):
        x = oracle.synth_x0(55, B); u = oracle.synth_controls(55, B, 1)[:, 0, :]
        P = random_cov(W, B, 8)
        p = np.tile(p21, (B, 1))
        rxn = oracle.rollout(x, u, 1, dt, u_mode=0, p=p, kind=KITE_ID)
        Jx, _ = oracle.jac(x, u, p=p, kind=KITE_ID)
        A = np.eye(13)[None] + dt * Jx
        rPn = np.einsum("bij,bjk,blk->bil", A, P, A) + W[None]
        xn, Pn = ekf_predict_c(e, B, ld, dt, x, u, P, W)
        assert_close(xn, rxn, RTOL, what="id EKF xn B=%d" % B)
        assert_close(Pn, rPn, RTOL, what="id EKF Pn B=%d" % B)


def check_update(oracle, xu, Pu, z, V, x, P, what):
    """The update against the oracle, measured against the 80-bit extended-precision update: an entry may exceed 1e-9 only
    by 16 x the double-precision oracle's own error for that filter (test_ekf_predict_vs_oracle_batch)."""
    rxu, rPu = oracle.ekf_update(z, V, x, P)
    lxu, lPu = oracle.ekf_update_ld(z, V, x, P)
    own_x = np.abs(rxu - lxu) / np.maximum(np.abs(lxu), 1.0)
    own_P = np.abs(rPu - lPu) / np.maximum(np.abs(lPu), 1e-3)
    err_x = np.abs(xu - lxu) / np.maximum(np.abs(lxu), 1.0)
    err_P = np.abs(Pu - lPu) / np.maximum(np.abs(lPu), 1e-3)
    assert bool((err_x <= np.maximum(RTOL, 16 * own_x.max(1, keepdims=True))).all()), "ekf update x " + what
    assert bool((err_P <= np.maximum(RTOL, 16 * own_P.max((1, 2), keepdims=True))).all()), "ekf update P " + what


def ekf_update_c(e, B, ld, z, V, x, P):
    """kite_ekf_update_batch in place on [rows][ld] buffers whose padding holds the sentinel."""
    zd = padded(z, ld)
    xd, Pd = sentinel(13, ld), sentinel(169, ld)
    xd[:, :B] = soa(x); Pd[:, :B] = soa(P.reshape(B, 169))
    Vh = np.ascontiguousarray(V)
    e._use_torch_stream()
    e._ck(e.L.kite_ekf_update_batch(e.ctx, B, ld, ptr(zd), Vh.ctypes.data_as(C.c_void_p), ptr(xd), ptr(Pd)))
    torch.cuda.synchronize()
    assert_untouched(xd, 0, B, "update x B=%d ld=%d" % (B, ld)); assert_untouched(Pd, 0, B, "update P B=%d ld=%d" % (B, ld))
    return aos(xd[:, :B]), aos(Pd[:, :B], 13, 13)


@pytest.mark.gpu
def test_ekf_update_shapes(engines, oracle):
    """k_ekf_update at B = 1, around the 128-thread block and across many blocks, with ld = B and ld > B."""
    e = engines[KITE]
    W, V = oracle.ekf_defaults()
    rng = np.random.default_rng(21)
    for B, ld in ((1, 1), (127, 127), (128, 128), (129, 129), (4097, 4097), (1, 8), (129, 200), (4097, 4100)):
        x = oracle.synth_x0(B + ld, B)
        P = random_cov(W, B, ld)
        z = x[:, 6:13] + 0.01 * rng.standard_normal((B, 7))
        xu, Pu = ekf_update_c(e, B, ld, z, V, x, P)
        check_update(oracle, xu, Pu, z, V, x, P, "B=%d ld=%d" % (B, ld))


@pytest.mark.gpu
def test_ekf_predict_update_cycles(engines, oracle):
    """20 predict -> update cycles on the same device buffers (predict ping-pongs between two pairs, the update works in
    place).  Every cycle is checked against the oracle started from the GPU's previous state, so errors cannot pile up."""
    e = engines[KITE]
    W, V = oracle.ekf_defaults()
    dt = 0.0084
    rng = np.random.default_rng(5)
    for B in (130, 77):                                                     # TMA predict, direct predict
        x = oracle.synth_x0(900, B); u = oracle.synth_controls(900, B, 20)
        truth = x.copy()
        xa, Pa = soa(x), soa(random_cov(W, B, 9).reshape(B, 169))
        xb, Pb = e.empty(13, B), e.empty(169, B)
        for k in range(20):
            xprev, Pprev = aos(xa), aos(Pa, 13, 13)
            uk = u[:, k, :].copy()
            e.ekf_predict(xa, soa(uk), dt, Pa, W, out=(xb, Pb))
            rxn, rPn = oracle.ekf_predict(xprev, uk, dt, Pprev, W)
            assert_close(aos(xb), rxn, RTOL, what="cycle %d predict xn B=%d" % (k, B))
            assert_close(aos(Pb, 13, 13), rPn, RTOL, what="cycle %d predict Pn B=%d" % (k, B))
            truth = oracle.rollout(truth, uk, 1, dt)
            z = truth[:, 6:13] + 0.001 * rng.standard_normal((B, 7))
            xpred, Ppred = aos(xb), aos(Pb, 13, 13)
            e.ekf_update(soa(z), V, xb, Pb)
            check_update(oracle, aos(xb), aos(Pb, 13, 13), z, V, xpred, Ppred, "cycle %d B=%d" % (k, B))
            xa, xb, Pa, Pb = xb, xa, Pb, Pa
        assert bool(torch.isfinite(Pa).all())


# ---------------------------------------------------------------- 5. collocation across node counts -----------
# M = 2, 3, 4, 15, 16 (compact constant-bank rows), 17, 17, 101 (dense walk)
COLLOC_PS = [(1, 1), (2, 1), (3, 1), (7, 2), (5, 3), (8, 2), (4, 4), (10, 10)]
COLLOC_TAU = 0.25


def colloc_z(golden, M, B, seed):
    """Decision vectors of M nodes made from the nodes of the golden NMPC case, perturbed per scenario."""
    c = golden["colloc_nmpc_P5_S2_scaled"]
    z0 = np.array(c["z"])
    X0, U0 = z0[:11 * 15].reshape(11, 15), z0[11 * 15:].reshape(11, 4)
    idx = np.arange(M) % 11
    zm = np.concatenate([X0[idx].ravel(), U0[idx].ravel()])
    rng = np.random.default_rng(seed)
    return zm[None, :] * (1 + 0.03 * rng.standard_normal((B, M * 19))), np.array(c["sx"]), np.array(c["su"])


def colloc_prm(yaml_path, pnom, B, seed, arm=None):
    from oracle.oracle_py import PARAM_FIELDS, params_from_yaml
    prm = params_from_yaml(yaml_path)
    if arm:
        for key, v in zip(("rx", "ry", "rz"), arm):
            prm[PARAM_FIELDS.index(("tether", key))] = v
    p = p_batch(pnom, B, seed)
    prm_b = np.tile(prm, (B, 1))
    prm_b[:, IDX21] = p
    return p, prm_b


def check_colloc(e, orc, z, P, S, sx, su, p=None, prm_b=None, what=""):
    """Dense, sparse and values-only evaluations against oracle.colloc_eval."""
    from openkite_b200.collocation import comp_diff_matrix
    M, B = S * P + 1, z.shape[0]
    compD = comp_diff_matrix(P, S)
    rG, rJX, rJU = orc.colloc_eval(z, P, S, 0.0, 2 * S * COLLOC_TAU, sx, su, prm_batch=prm_b)
    pd = soa(p) if p is not None else None
    G, JX, JU, gn = e.colloc_eval(soa(z), M, compD, COLLOC_TAU, sx, su, p=pd)
    assert_close(aos(G), rG, RTOL, what="G " + what)
    assert_close(aos(JX, M, 15, 15), rJX, RTOL, what="JX " + what)
    assert_close(aos(JU, M, 15, 4), rJU, RTOL, what="JU " + what)
    assert_close(gn.cpu().numpy(), (rG ** 2).sum(1), RTOL, what="|G|^2 " + what)
    G2, JV, gn2 = e.colloc_eval_sparse(soa(z), M, compD, COLLOC_TAU, sx, su, p=pd)
    rows, cols = e.colloc_sparsity()
    dense = np.concatenate([rJX, rJU], axis=3)                              # [B][M][15][19]
    assert_close(aos(G2), rG, RTOL, what="sparse G " + what)
    assert_close(aos(JV, M, len(rows)), dense[:, :, rows, cols], RTOL, what="JV " + what)
    G3, nx, nu, gn3 = e.colloc_eval(soa(z), M, compD, COLLOC_TAU, sx, su, p=pd, want_jac=False)
    assert nx is None and nu is None
    assert_close(aos(G3), rG, RTOL, what="values-only G " + what)
    assert_close(gn3.cpu().numpy(), (rG ** 2).sum(1), RTOL, what="values-only |G|^2 " + what)


@pytest.mark.gpu
@pytest.mark.parametrize("P,S", COLLOC_PS, ids=["P%d_S%d" % ps for ps in COLLOC_PS])
def test_colloc_node_counts(engines, okb, oracle, golden, yaml_path, pnom, P, S):
    """k_colloc_eval (dense / sparse / values only, nominal and per-scenario coefficients) and k_colloc_cost at node
    counts below, at and across the 4 node rows of a CTA and the compact-row limit (16 nodes, 8 non-zeros)."""
    from openkite_b200.collocation import quad_weights
    e = engines[KITE]
    M, B = S * P + 1, 77
    z, sx, su = colloc_z(golden, M, B, 10 * P + S)
    check_colloc(e, oracle, z, P, S, sx, su, what="M=%d" % M)
    p, prm_b = colloc_prm(yaml_path, pnom, B, M)
    check_colloc(e, oracle, z, P, S, sx, su, p=p, prm_b=prm_b, what="M=%d per-scenario" % M)
    for q, alt in (((np.cos(np.pi / 8), 0.0, np.sin(np.pi / 8), 0.0), 0.0), ((1.0, 0.0, 0.0, 0.0), 1.5)):
        rcost, rgrad = oracle.colloc_cost(z, P, S, 0.0, 2 * S * COLLOC_TAU, sx, oracle.nmpc_cost_params(sx, q_rot=q, altitude=alt))
        cost, grad = e.colloc_cost(soa(z), P, S, quad_weights(P), COLLOC_TAU, sx, okb.NmpcCost.defaults(sx, q_rot=q, altitude=alt))
        assert_close(cost.cpu().numpy(), rcost, RTOL, what="cost M=%d" % M)
        assert_close(aos(grad), rgrad, RTOL, what="cost gradient M=%d" % M)


@pytest.mark.gpu
@pytest.mark.parametrize("P,S", [(7, 2), (8, 2)], ids=["P7_S2", "P8_S2"])
def test_colloc_tether_arm_node_counts(arm_setup, golden, yaml_path, pnom, P, S):
    """The tether-arm context (its own sparse format) against an oracle with the same arm, on a compact (M = 15) and a
    dense-walk (M = 17) shape."""
    e, orc = arm_setup
    M, B = S * P + 1, 66
    z, sx, su = colloc_z(golden, M, B, 3)
    check_colloc(e, orc, z, P, S, sx, su, what="arm M=%d" % M)
    p, prm_b = colloc_prm(yaml_path, pnom, B, 4, arm=ARM)
    check_colloc(e, orc, z, P, S, sx, su, p=p, prm_b=prm_b, what="arm M=%d per-scenario" % M)


@pytest.mark.gpu
@pytest.mark.parametrize("P,S", [(2, 1), (5, 3), (8, 2), (10, 10)], ids=["P2_S1", "P5_S3", "P8_S2", "P10_S10"])
def test_colloc_sub_batch_offset(engines, okb, oracle, golden, P, S):
    """ld > B: a sub-batch at a column offset of wider [rows][ld] buffers (dense, sparse, values only, cost); the
    neighbouring columns on both sides keep their sentinel."""
    from openkite_b200.collocation import comp_diff_matrix, quad_weights
    e = engines[KITE]
    M, ld, off, B = S * P + 1, 128, 40, 37
    z, sx, su = colloc_z(golden, M, ld, 8)
    rG, rJX, rJU = oracle.colloc_eval(z[off:off + B], P, S, 0.0, 2 * S * COLLOC_TAU, sx, su)
    cp = okb.NmpcCost.defaults(sx)
    rcost, rgrad = oracle.colloc_cost(z[off:off + B], P, S, 0.0, 2 * S * COLLOC_TAU, sx, oracle.nmpc_cost_params(sx))
    zd = soa(z)
    h = lambda a: np.ascontiguousarray(a, dtype=np.float64)
    cd, sxa, sua, qwa = h(comp_diff_matrix(P, S)), h(sx), h(su), h(quad_weights(P))
    hp = lambda a: a.ctypes.data_as(C.c_void_p)
    nnz = e.colloc_nnz_per_node()
    rows, cols = e.colloc_sparsity()
    e._use_torch_stream()
    for jac in ("dense", "sparse", "none"):
        G, gn = sentinel(M * 15, ld), sentinel(ld)
        JX = sentinel(M * 225, ld) if jac == "dense" else (sentinel(M * nnz, ld) if jac == "sparse" else None)
        JU = sentinel(M * 60, ld) if jac == "dense" else None
        if jac == "sparse":
            rc = e.L.kite_colloc_eval_sparse(e.ctx, B, ld, M, hp(cd), COLLOC_TAU, hp(sxa), hp(sua), ptr(zd, off), None,
                                             ptr(G, off), ptr(JX, off), ptr(gn, off))
        else:
            rc = e.L.kite_colloc_eval(e.ctx, B, ld, M, hp(cd), COLLOC_TAU, hp(sxa), hp(sua), ptr(zd, off), None, ptr(G, off),
                                      ptr(JX, off) if JX is not None else None, ptr(JU, off) if JU is not None else None,
                                      ptr(gn, off))
        e._ck(rc)
        torch.cuda.synchronize()
        what = "%s M=%d" % (jac, M)
        for t in (G, gn, JX, JU):
            if t is not None:
                assert_untouched(t, off, off + B, what)
        assert_close(aos(G[:, off:off + B]), rG, RTOL, what="G " + what)
        assert_close(gn[off:off + B].cpu().numpy(), (rG ** 2).sum(1), RTOL, what="|G|^2 " + what)
        if jac == "dense":
            assert_close(aos(JX[:, off:off + B], M, 15, 15), rJX, RTOL, what="JX " + what)
            assert_close(aos(JU[:, off:off + B], M, 15, 4), rJU, RTOL, what="JU " + what)
        elif jac == "sparse":
            dense = np.concatenate([rJX, rJU], axis=3)
            assert_close(aos(JX[:, off:off + B], M, nnz), dense[:, :, rows, cols], RTOL, what="JV " + what)
    cost, grad = sentinel(ld), sentinel(M * 19, ld)
    e._ck(e.L.kite_colloc_cost(e.ctx, B, ld, P, S, hp(qwa), COLLOC_TAU, hp(sxa), C.byref(cp), ptr(zd, off), ptr(cost, off),
                               ptr(grad, off)))
    torch.cuda.synchronize()
    assert_untouched(cost, off, off + B, "cost M=%d" % M); assert_untouched(grad, off, off + B, "grad M=%d" % M)
    assert_close(cost[off:off + B].cpu().numpy(), rcost, RTOL, what="cost sub-batch M=%d" % M)
    assert_close(aos(grad[:, off:off + B]), rgrad, RTOL, what="grad sub-batch M=%d" % M)


@pytest.mark.parametrize("P,S", COLLOC_PS, ids=["P%d_S%d" % ps for ps in COLLOC_PS])
def test_comp_diff_matrix_matches_oracle(oracle, P, S):
    """collocation.comp_diff_matrix (what Python callers hand to kite_colloc_eval) against the oracle's operator."""
    from openkite_b200.collocation import comp_diff_matrix, quad_weights
    assert_close(comp_diff_matrix(P, S), oracle.cheb_compdiff(P, S), 1e-12, what="compD P=%d S=%d" % (P, S))
    assert_close(quad_weights(P), oracle.cheb_weights(P), 1e-12, what="weights P=%d" % P)


# ---------------------------------------------------------------- 6. the table that keeps this complete --------
# Every kernel of libkite_b200.so (substring of its mangled name, template arguments included) -> the tests that launch it.
_P = "test_gpu_parity.py::"
_V = "test_gpu_variants.py::"
_F = "test_gpu_fullsize.py::"
KERNEL_TESTS = {
    "k_math_selftestILi0E": [_P + "test_lean_math_accuracy"],
    "k_synth_inputsILi0E": [_P + "test_synth_inputs_bit_identical"],
    "k_synth_id_paramsILi0E": [_F + "test_config5_full_size_id_sweep_and_ekf", _V + "test_rollout_host_pipeline_chunks"],
    # k_point_eval<rigid, per-unit coefficients, Jacobian>
    "k_point_evalILb0ELb0ELb0E": [_P + "test_rhs_jac_vs_oracle_batch"],
    "k_point_evalILb0ELb0ELb1E": [_P + "test_rhs_jac_vs_oracle_batch"],
    "k_point_evalILb0ELb1ELb0E": [_V + "test_point_eval_rigid_and_coefficient_batches"],
    "k_point_evalILb0ELb1ELb1E": [_V + "test_point_eval_rigid_and_coefficient_batches"],
    "k_point_evalILb1ELb0ELb0E": [_V + "test_point_eval_rigid_and_coefficient_batches"],
    "k_point_evalILb1ELb0ELb1E": [_V + "test_point_eval_rigid_and_coefficient_batches"],
    # k_rk4_rollout<control mode, rigid, per-trajectory coefficients>
    "k_rk4_rolloutILi0ELb0ELb0E": [_V + "test_rollout_matrix", _P + "test_rollout_vs_oracle"],
    "k_rk4_rolloutILi0ELb0ELb1E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi0ELb1ELb0E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi1ELb0ELb0E": [_V + "test_rollout_matrix", _V + "test_rollout_host_pipeline_chunks"],
    "k_rk4_rolloutILi1ELb0ELb1E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi1ELb1ELb0E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi2ELb0ELb0E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi2ELb0ELb1E": [_V + "test_rollout_matrix", _V + "test_rollout_host_pipeline_chunks"],
    "k_rk4_rolloutILi2ELb1ELb0E": [_V + "test_rollout_matrix"],
    "k_rk4_rolloutILi3ELb0ELb0E": [_V + "test_rollout_matrix", _P + "test_rollout_vs_oracle"],
    "k_rk4_rolloutILi3ELb0ELb1E": [_V + "test_rollout_matrix"],
    # k_sens_fused<tether arm, rigid, TMA output>
    "k_sens_fusedILb0ELb0ELb0E": [_V + "test_sens_rollout_padded", _V + "test_sens_identification_engine"],
    "k_sens_fusedILb0ELb0ELb1E": [_V + "test_sens_rollout_padded", _V + "test_sens_identification_engine"],
    "k_sens_fusedILb1ELb0ELb0E": [_V + "test_sens_tether_arm_rollout"],
    "k_sens_fusedILb1ELb0ELb1E": [_V + "test_sens_tether_arm_rollout"],
    "k_sens_fusedILb0ELb1ELb0E": [_V + "test_sens_rigid_batches"],
    # EKF predict <tether arm, rigid>: direct loads (odd B or pitch) and TMA boxes (even)
    "k_ekf_predictILb0ELb0E": [_P + "test_ekf_predict_vs_oracle_batch", _V + "test_ekf_predict_update_cycles"],
    "k_ekf_predictILb1ELb0E": [_P + "test_tether_arm_batch_vs_oracle"],
    "k_ekf_predictILb0ELb1E": [_V + "test_ekf_predict_rigid"],
    "k_ekf_predict_tmaILb0ELb0E": [_V + "test_ekf_predict_update_cycles", _V + "test_ekf_predict_identification"],
    "k_ekf_predict_tmaILb1ELb0E": [_P + "test_tether_arm_batch_vs_oracle"],
    "k_ekf_predict_tmaILb0ELb1E": [_V + "test_ekf_predict_rigid"],
    "k_ekf_updateILi0E": [_V + "test_ekf_update_shapes", _V + "test_ekf_predict_update_cycles"],
    # collocation <per-scenario coefficients, node rows per CTA, format: 0 dense, 1 sparse, 2 sparse with arm, 3 values>
    "k_colloc_costILi4E": [_V + "test_colloc_node_counts", _V + "test_colloc_sub_batch_offset"],
    "k_colloc_evalILb0ELi4ELi0E": [_V + "test_colloc_node_counts", _V + "test_colloc_sub_batch_offset"],
    "k_colloc_evalILb0ELi4ELi1E": [_V + "test_colloc_node_counts", _V + "test_colloc_sub_batch_offset"],
    "k_colloc_evalILb0ELi4ELi2E": [_V + "test_colloc_tether_arm_node_counts"],
    "k_colloc_evalILb0ELi4ELi3E": [_V + "test_colloc_node_counts", _V + "test_colloc_sub_batch_offset"],
    "k_colloc_evalILb1ELi4ELi0E": [_V + "test_colloc_node_counts"],
    "k_colloc_evalILb1ELi4ELi1E": [_V + "test_colloc_node_counts"],
    "k_colloc_evalILb1ELi4ELi2E": [_V + "test_colloc_tether_arm_node_counts"],
    "k_colloc_evalILb1ELi4ELi3E": [_V + "test_colloc_node_counts"],
}
BENCH_ONLY = ["k_fp64_peakILi0E", "k_fp64_peak3ILi0E"]      # roofline microbenchmarks of bench.py, no numerical output


def test_every_kernel_has_a_test():
    """The set of kernels in the build equals the keys of KERNEL_TESTS (plus the benchmark-only ones), each kernel matches
    exactly one key, and every test named there exists."""
    from openkite_b200 import build as b
    b.build()
    names = [r[0] for r in b.resource_report()]
    assert len(names) >= 40, "ptxas logs missing: run python -m openkite_b200.build --force"
    keys = list(KERNEL_TESTS) + BENCH_ONLY
    for n in names:
        hits = [k for k in keys if k in n]
        assert len(hits) == 1, "kernel %s matches %s in KERNEL_TESTS: every instantiation needs a test" % (n, hits)
    for k in keys:
        assert any(k in n for n in names), "KERNEL_TESTS lists %s, which the build does not contain" % k
    here = os.path.dirname(os.path.abspath(__file__))
    defined = {}
    for ref in sorted({t for ts in KERNEL_TESTS.values() for t in ts}):
        mod, fn = ref.split("::")
        if mod not in defined:
            tree = ast.parse(open(os.path.join(here, mod)).read())
            defined[mod] = {n.name for n in tree.body if isinstance(n, ast.FunctionDef)}
        assert fn in defined[mod], "KERNEL_TESTS names %s, which does not exist" % ref
