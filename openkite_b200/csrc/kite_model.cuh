// =====================================================================================
// kite_model.cuh -- device-side rigid-wing kite model for sm_100a (hand-written, FP64).
//
// Computes the same function as the reference's CasADi graph (kite.cpp:197-322, :448-573,
// :622-661) but is NOT a transcription of it: the four quaternion sandwich products are
// replaced by one attitude matrix M(q) = (s^2-a.a) I + 2 a a^T + 2 s [a]x  (exact also for
// |q| != 1), the wind->body rotation uses cos/sin(aoa) = (x,z)/hypot and cos(ss) =
// sqrt(1-sin^2) instead of four half-angle trig calls, constant coefficient products are
// folded on the host, and the state/control Jacobians are derived analytically block by
// block (no AD tape).  Everything is straight-line code on register-resident scalars.
//
// Parity against the oracle (which follows the reference literally) is <= 1e-9 (tests/).
// =====================================================================================
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <type_traits>

#include "kite_math.cuh"

namespace kite {

// Derived aerodynamic coefficients (from the 21 raw coefficients, kite.cpp:571-572 order).
struct AeroCoef {
    double CL0, CLa, CD0, CYb;
    double cCm0, cCma;       // c*{Cm0,Cma}: the pitch moment is (c Cm) q S (kite.cpp:278), so the chord is folded in here
    double bCnb, bClb;       // b*{Cnb,Clb}: likewise the span for the yaw / roll moments (kite.cpp:274,282)
    double kLq;              // 0.25*CLq*c*S*ro          (kite.cpp:210)
    double kmq;              // Cmq*0.25*S*c^2*ro        (kite.cpp:279)
    double kYr, kYp;         // 0.25*b*ro*S*{CYr,CYp}    (kite.cpp:213)
    double knr, klr, klp, knp;  // 0.25*ro*b^2*S*{Cnr,Clr,Clp,Cnp}  (kite.cpp:275,283)
    double CLde, CYdr;
    double cCmde, bCndr, bCldr;  // c*Cmde, b*Cndr, b*Cldr
};

// Which coefficient types select the table-driven exponential (kite_eval_c): volatile AeroCoef (identification sweeps, per-
// trajectory records in shared memory) does; AeroCoefPlain is the same record read from shared memory WITHOUT changing the
// arithmetic -- for kernels whose results must stay bitwise equal to the constant-bank instantiations (collocation, FMT 2).
struct AeroCoefPlain : AeroCoef {};
template <class AC> struct exp_table_for : std::is_volatile<AC> {};
template <> struct exp_table_for<volatile AeroCoefPlain> : std::false_type {};

struct KiteConsts {
    AeroCoef A;              // nominal coefficients (from kite_params)
    double eps;              // 1e-4 standard model (kite.cpp:200-201), 0 identification model (:451-452)
    double cqS;              // 0.5*ro*S  -> qS = cqS*V^2 (dynamic pressure times wing area)
    double b, c;
    double inv_piAR;         // 1/(pi*e_o*AR)
    double bCn0, bCl0;       // b*Cn0, b*Cl0
    double inv_mass, g;
    double Lt, Ks, Kd;
    double arm0, arm1, arm2; // tether attachment arm (rx,ry,rz)
    double Ixx, Iyy, Izz, Ixz, Ji00, Ji02, Ji11, Ji22;
    double IzmIy, IymIx, IzmIx;  // Izz-Iyy, Iyy-Ixx, Izz-Ixx: w x (J w) in factored form
    double lambda;           // quaternion-norm stabiliser gain: -5 kite, -10 rigid body
    double sLq, smq, sY, sb2;  // factors that turn raw CLq, Cmq, CY*, C{l,n}* into AeroCoef entries
    int has_arm;
    int model_kind;
};

__host__ __device__ inline void derive_coef(const KiteConsts& K, const double p[21], AeroCoef& A) {
    A.CL0 = p[0]; A.CLa = p[1]; A.CD0 = p[2]; A.CYb = p[3];
    A.cCm0 = K.c * p[4]; A.cCma = K.c * p[5]; A.bCnb = K.b * p[6]; A.bClb = K.b * p[7];
    A.kLq = K.sLq * p[8];
    A.kmq = K.smq * p[9];
    A.kYr = K.sY * p[10];
    A.knr = K.sb2 * p[11];
    A.klr = K.sb2 * p[12];
    A.kYp = K.sY * p[13];
    A.klp = K.sb2 * p[14];
    A.knp = K.sb2 * p[15];
    A.CLde = p[16]; A.CYdr = p[17]; A.cCmde = K.c * p[18]; A.bCndr = K.b * p[19]; A.bCldr = K.b * p[20];
}

// ---- small helpers ---------------------------------------------------------------------
// d(M y)/dq (3x4) for M(q) y = (s^2-a.a) y + 2 (a.y) a + 2 s (a x y); SGN=-1 gives d(M^T y)/dq.
template <int SGN>
__device__ __forceinline__ void dM_dq_apply(double s, const double (&a)[3], const double (&y)[3], double (&D)[3][4]) {
    const double sg = (SGN > 0) ? 2.0 : -2.0;
    const double axy0 = a[1] * y[2] - a[2] * y[1];
    const double axy1 = a[2] * y[0] - a[0] * y[2];
    const double axy2 = a[0] * y[1] - a[1] * y[0];
    const double ts = 2.0 * s;
    D[0][0] = fma(ts, y[0], sg * axy0);
    D[1][0] = fma(ts, y[1], sg * axy1);
    D[2][0] = fma(ts, y[2], sg * axy2);
    const double ady2 = 2.0 * (a[0] * y[0] + a[1] * y[1] + a[2] * y[2]);
    const double ss_ = sg * s;   // +-2 s
    // column a_j: -2 a_j y + 2 y_j a + 2 (a.y) e_j +- 2 s (e_j x y)
    // e_1 x y = (0,-y2,y1); e_2 x y = (y2,0,-y0); e_3 x y = (-y1,y0,0)
    const double c[3][3] = {{0.0, -y[2], y[1]}, {y[2], 0.0, -y[0]}, {-y[1], y[0], 0.0}};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            double t = 2.0 * (y[j] * a[i] - a[j] * y[i]);
            if (i == j) t += ady2;
            D[i][j + 1] = fma(ss_, c[j][i], t);
        }
    }
}

// Attitude matrix M(q) = (s^2 - a.a) I + 2 a a^T + 2 s [a]x and the squared norm nq = |q|^2 in 21 FP64 operations:
// doubled vector part t = 2a, off-diagonals as one FMA each, M11 and M22 from M00 by two-term corrections.
__device__ __forceinline__ void attitude_matrix(double s, const double (&a)[3], double (&M)[3][3], double& nq) {
    const double t0 = a[0] + a[0], t1 = a[1] + a[1], t2 = a[2] + a[2];
    const double st0 = s * t0, st1 = s * t1, st2 = s * t2;
    M[0][1] = fma(t0, a[1], -st2); M[1][0] = fma(t0, a[1], st2);
    M[0][2] = fma(t0, a[2], st1);  M[2][0] = fma(t0, a[2], -st1);
    M[1][2] = fma(t1, a[2], -st0); M[2][1] = fma(t1, a[2], st0);
    const double p = fma(s, s, a[0] * a[0]);
    const double r = fma(a[1], a[1], a[2] * a[2]);
    M[0][0] = p - r;
    nq = p + r;
    const double q0 = fma(-t0, a[0], M[0][0]);
    M[1][1] = fma(t1, a[1], q0);
    M[2][2] = fma(t2, a[2], q0);
}

struct NoSink {
    __device__ __forceinline__ void jx(int, int, double) const {}
    __device__ __forceinline__ void ju(int, int, double) const {}
    __device__ __forceinline__ void aero(double, double, double) const {}
};

// =====================================================================================
// f(x,u) and (optionally) the analytic Jacobians d f/d x, d f/d u.
// Jacobian entries are emitted through `sink.jx(row, col, value)` / `sink.ju(row, col, value)`
// with compile-time-constant row/col after unrolling, exactly once per structural non-zero
// (104 + 7 entries when the tether arm is zero, +21 otherwise).
// =====================================================================================
// Everything the right-hand side needs from the control u = [T dE dR]: the five coefficient sums that are affine in dE / dR.
// RK4 holds u for all four stages (kitemath.cpp:36-51), so the integrators evaluate these once per step, not per stage.
struct CtrlTerms {
    double Tm;       // thrust / mass
    double cydr;     // CYdr dR                 (side force,  kite.cpp:212)
    double cl0;      // b (Cl0 + Cldr dR)       (roll moment, kite.cpp:274)
    double cm0;      // c (Cm0 + Cmde dE)       (pitch moment, kite.cpp:278)
    double cn0;      // b (Cn0 + Cndr dR)       (yaw moment,  kite.cpp:282)
    double nzde;     // -CLde dE                (elevator force / (q S), kite.cpp:228)
};
template <class AC>
__device__ __forceinline__ CtrlTerms ctrl_terms(const KiteConsts& K, const AC& A, const double (&u)[3]) {
    CtrlTerms c;
    c.Tm = u[0] * K.inv_mass;
    c.cydr = A.CYdr * u[2];
    c.cl0 = fma(A.bCldr, u[2], K.bCl0);
    c.cm0 = fma(A.cCmde, u[1], A.cCm0);
    c.cn0 = fma(A.bCndr, u[2], K.bCn0);
    c.nzde = -A.CLde * u[1];
    return c;
}

// AC: AeroCoef, or volatile AeroCoef when the coefficients live in shared memory and must be re-read at every use instead of
// being hoisted into (and spilled from) registers (identification sweeps, k_rk4_rollout<.., PERCOEF>).
template <bool JAC, class Sink, class AC>
__device__ __forceinline__ void kite_eval_c(const KiteConsts& K, const AC& A, const double (&x)[13],
                                            const CtrlTerms& uc, double (&f)[13], Sink& sink) {
    const double v[3] = {x[0], x[1], x[2]};
    const double w[3] = {x[3], x[4], x[5]};
    const double r[3] = {x[6], x[7], x[8]};
    const double s = x[9];
    const double a[3] = {x[10], x[11], x[12]};

    // ---- airspeed, angles (lean special functions, kite_math.cuh) ------------------------------
    const double V2 = fma(v[0], v[0], fma(v[1], v[1], v[2] * v[2]));
    const double rV = fast_rsqrt(V2);                         // 1/V (also d V/d v = v rV in the Jacobian)
    const double V = is_pos(V2) ? V2 * rV : 0.0;              // v = 0 is a legal state of the standard model
    const double iVe = fast_rcp(V + K.eps);
    const double sb = v[1] * iVe;                             // sin(sideslip)
    const double c2 = fma(-sb, sb, 1.0);
    const double rcb = fast_rsqrt(c2);                        // 1/cos(sideslip)
    const double cb = is_pos(c2) ? c2 * rcb : 0.0;            // cos(sideslip) >= 0
    const double xe = v[0] + K.eps;
    const double irho = fast_rsqrt(fma(xe, xe, v[2] * v[2]));
    const double ca = xe * irho, sa = v[2] * irho;            // cos/sin(angle of attack)
    // both angles from their (sin, cos) pairs, branch free for any sideslip and any angle of attack (all four
    // quadrants): two interleaved polynomial chains, no division, no libm, no warp divergence (kite_math.cuh)
    // Angles: table + short series in every kernel (asin_sc<true>, kite_math.cuh: config 2 +1.6 %).  Exponential of the
    // tether logistic: the 2^(j/32) table form only where the coefficients come from shared memory (identification sweeps:
    // +1.6 % on top of the angle table there, -0.5 % on the config-2 kernel: profiles/r2e_sweep_tables.log, r2r_sweep.log)
    constexpr bool TAB = exp_table_for<AC>::value;
    const double ss = asin_sc<true>(sb, cb);
    const double aoa = atan2_sc<true>(sa, ca);
    const double qS = K.cqS * V2;
    // rate damping terms are linear in V w: the airspeed scales the rates once, not each coefficient sum
    const double Vw0 = V * w[0], Vw1 = V * w[1], Vw2 = V * w[2];

    // ---- aerodynamic force in the wind frame, rotated to body ---------------------------
    const double CL = fma(A.CLa, aoa, A.CL0);
    const double CD = fma(CL * CL, K.inv_piAR, A.CD0);
    const double LIFT = fma(CL, qS, A.kLq * Vw1);
    const double DRAG = CD * qS;
    const double cy = fma(A.CYb, ss, uc.cydr);
    const double SF = fma(cy, qS, fma(A.kYr, Vw2, A.kYp * Vw0));
    const double Zde = uc.nzde * qS;
    const double X1 = fma(sa, LIFT, -ca * DRAG);
    const double Z1 = -fma(sa, DRAG, ca * LIFT);
    const double Fx = fma(cb, X1, -sa * Zde);
    const double Fy = fma(sb, X1, SF);
    const double Fz = fma(ca, Zde, Z1);
    sink.aero(Fx, Fy, Fz);                                    // body-frame aerodynamic force: Function "Aero" (kite.cpp:330)

    // ---- attitude matrix M(q):  q (x) [0,y] (x) conj(q) = M y,   conj(q) (x) [0,y] (x) q = M^T y ----
    double M[3][3], nq;
    attitude_matrix(s, a, M, nq);

    // Matrix-vector products are written as COLUMN sweeps: the three FMAs of a sweep share v[j] in the same operand slot, so two of
    // them find it in the register-reuse cache and issue in 2 cycles instead of 3 (three distinct vector-register operands cost
    // an extra cycle on the FP64 pipe: profiles/r2j_dfma_operands.log).  Same for M^T n and the quaternion rate below.
    double vi[3];   // inertial velocity = r_dot
#pragma unroll
    for (int i = 0; i < 3; ++i) vi[i] = M[i][2] * v[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) vi[i] = fma(M[i][1], v[1], vi[i]);
#pragma unroll
    for (int i = 0; i < 3; ++i) vi[i] = fma(M[i][0], v[0], vi[i]);

    // ---- tether: R = -tau n, tau = (Ks (d-Lt) + Kd n.vi) * logistic(4 (d-Lt)) -------------
    const double d2 = fma(r[0], r[0], fma(r[1], r[1], r[2] * r[2]));
    const double id = fast_rsqrt(d2);
    const double d = d2 * id;
    const double n[3] = {r[0] * id, r[1] * id, r[2] * id};
    const double e = d - K.Lt;
    const double H = fast_logistic4<TAB>(e);                        // K/(1+exp(-4x)), kitemath.cpp:31-34
    const double nv = fma(n[0], vi[0], fma(n[1], vi[1], n[2] * vi[2]));
    const double tens = fma(K.Ks, e, K.Kd * nv);
    const double tau = tens * H;
    double m[3];    // M^T n
#pragma unroll
    for (int i = 0; i < 3; ++i) m[i] = M[2][i] * n[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) m[i] = fma(M[1][i], n[1], m[i]);
#pragma unroll
    for (int i = 0; i < 3; ++i) m[i] = fma(M[0][i], n[0], m[i]);

    // ---- v_dot = (Faero + T e1 + R_b)/m + g M^T e3 - w x v,  R_b = -tau m ------------------
    const double tm = -tau * K.inv_mass;                              // R_b / mass = tm * m
    f[0] = fma(tm, m[0], fma(Fx, K.inv_mass, fma(K.g, M[2][0], fma(w[2], v[1], fma(-w[1], v[2], uc.Tm)))));
    f[1] = fma(tm, m[1], fma(Fy, K.inv_mass, fma(K.g, M[2][1], fma(w[0], v[2], -w[2] * v[0]))));
    f[2] = fma(tm, m[2], fma(Fz, K.inv_mass, fma(K.g, M[2][2], fma(w[1], v[0], -w[0] * v[1]))));

    // ---- moments (b and c are folded into the coefficient sums: cl = b Cl, cm = c Cm, cn = b Cn) ----
    const double cl = fma(A.bClb, ss, uc.cl0);
    const double cm = fma(A.cCma, aoa, uc.cm0);
    const double cn = fma(A.bCnb, ss, uc.cn0);
    const double Lm = fma(cl, qS, fma(A.klr, Vw2, A.klp * Vw0));
    const double Mm = fma(cm, qS, A.kmq * Vw1);
    const double Nm = fma(cn, qS, fma(A.knp, Vw0, A.knr * Vw2));
    const double Max = fma(ca, Lm, -sa * Nm);
    const double Maz = fma(sa, Lm, ca * Nm);
    // rh = M_aero - w x (J w) with J = [Ixx 0 Ixz; 0 Iyy 0; Ixz 0 Izz], factored:
    //   (w x J w)_0 = w1 (Ixz w0 + (Izz-Iyy) w2),  (w x J w)_2 = w1 ((Iyy-Ixx) w0 - Ixz w2),
    //   (w x J w)_1 = (Ixx-Izz) w0 w2 + Ixz (w2^2 - w0^2)
    const double G0 = fma(K.Ixz, w[0], K.IzmIy * w[2]);
    const double G2 = fma(K.IymIx, w[0], -K.Ixz * w[2]);
    double rh0 = fma(-w[1], G0, Max);
    double rh1 = fma(K.IzmIx, w[0] * w[2], fma(K.Ixz, fma(w[0], w[0], -w[2] * w[2]), Mm));
    double rh2 = fma(-w[1], G2, Maz);
    if (K.has_arm) {
        const double Rb[3] = {-tau * m[0], -tau * m[1], -tau * m[2]};
        rh0 += K.arm1 * Rb[2] - K.arm2 * Rb[1];
        rh1 += K.arm2 * Rb[0] - K.arm0 * Rb[2];
        rh2 += K.arm0 * Rb[1] - K.arm1 * Rb[0];
    }
    f[3] = fma(K.Ji00, rh0, K.Ji02 * rh2);
    f[4] = K.Ji11 * rh1;
    f[5] = fma(K.Ji02, rh0, K.Ji22 * rh2);

    // ---- kinematics --------------------------------------------------------------------------
    f[6] = vi[0]; f[7] = vi[1]; f[8] = vi[2];
    const double hl = 0.5 * K.lambda;
    const double mu = fma(nq, hl, -hl);                                // (lambda / 2) (|q|^2 - 1)
    const double hw[3] = {0.5 * w[0], 0.5 * w[1], 0.5 * w[2]};         // q_dot = q (x) [0, w/2] + mu q
    // (sweeps over hw[2], hw[1], hw[0], mu: each shares its second operand across the four rows)
    f[9] = -a[2] * hw[2];                 f[10] = a[1] * hw[2];                 f[11] = -a[0] * hw[2];                f[12] = s * hw[2];
    f[9] = fma(-a[1], hw[1], f[9]);       f[10] = fma(-a[2], hw[1], f[10]);     f[11] = fma(s, hw[1], f[11]);         f[12] = fma(a[0], hw[1], f[12]);
    f[9] = fma(-a[0], hw[0], f[9]);       f[10] = fma(s, hw[0], f[10]);         f[11] = fma(a[2], hw[0], f[11]);      f[12] = fma(-a[1], hw[0], f[12]);
    f[9] = fma(s, mu, f[9]);              f[10] = fma(a[0], mu, f[10]);         f[11] = fma(a[1], mu, f[11]);         f[12] = fma(a[2], mu, f[12]);

    if constexpr (JAC) {
        const double Rb[3] = {-tau * m[0], -tau * m[1], -tau * m[2]};
        const double kYw = fma(A.kYr, w[2], A.kYp * w[0]);
        const double klw = fma(A.klr, w[2], A.klp * w[0]);
        const double knw = fma(A.knp, w[0], A.knr * w[2]);
        const double Jw0 = fma(K.Ixx, w[0], K.Ixz * w[2]);
        const double Jw1 = K.Iyy * w[1];
        const double Jw2 = fma(K.Ixz, w[0], K.Izz * w[2]);
        // =========================== gradients w.r.t. v of the aero scalars =======================
        const double dV[3] = {v[0] * rV, v[1] * rV, v[2] * rV};
        const double icb = rcb;
        // d sb = iVe (e1 - sb dV);  d ss = d sb / cb
        double dss[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) dss[j] = iVe * icb * ((j == 1 ? 1.0 : 0.0) - sb * dV[j]);
        const double daoa[3] = {-sa * irho, 0.0, ca * irho};
        const double tq = 2.0 * K.cqS;
        const double dqS[3] = {tq * v[0], tq * v[1], tq * v[2]};
        double dFx[3], dFy[3], dFz[3], dMax[3], dMy[3], dMaz[3];
        const double dCDfac = 2.0 * CL * K.inv_piAR * A.CLa;   // dCD = dCDfac * daoa
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double dCL = A.CLa * daoa[j];
            const double dL = fma(dCL, qS, fma(CL, dqS[j], A.kLq * w[1] * dV[j]));
            const double dD = fma(dCDfac * daoa[j], qS, CD * dqS[j]);
            const double dSF = fma(A.CYb * qS, dss[j], fma(cy, dqS[j], kYw * dV[j]));
            const double dZde = uc.nzde * dqS[j];
            const double dX1 = fma(-Z1, daoa[j], fma(sa, dL, -ca * dD));
            const double dZ1 = fma(X1, daoa[j], -fma(sa, dD, ca * dL));
            const double dsb = cb * dss[j], dcb = -sb * dss[j];
            const double dsa = ca * daoa[j], dca = -sa * daoa[j];
            dFx[j] = fma(dcb, X1, fma(cb, dX1, -fma(dsa, Zde, sa * dZde)));
            dFy[j] = fma(dsb, X1, fma(sb, dX1, dSF));
            dFz[j] = dZ1 + fma(dca, Zde, ca * dZde);
            const double dLm = fma(A.bClb * qS, dss[j], fma(cl, dqS[j], klw * dV[j]));
            const double dMm = fma(A.cCma * qS, daoa[j], fma(cm, dqS[j], A.kmq * w[1] * dV[j]));
            const double dNm = fma(A.bCnb * qS, dss[j], fma(cn, dqS[j], knw * dV[j]));
            dMax[j] = fma(-Maz, daoa[j], fma(ca, dLm, -sa * dNm));
            dMy[j] = dMm;
            dMaz[j] = fma(Max, daoa[j], fma(sa, dLm, ca * dNm));
        }

        // =========================== tether derivatives ==========================================
        // d R_b / d v = -(Kd H) m m^T
        const double kdH = K.Kd * H;
        double dRb_v[3][3];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) dRb_v[i][j] = -kdH * m[i] * m[j];
        // d tau / d r = H (Ks n + Kd pv) + 4 tau (1-H) n,  pv = (vi - nv n)/d
        double dtau_r[3], dRb_r[3][3];
        const double t4 = 4.0 * tau * (1.0 - H);
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const double pv = (vi[j] - nv * n[j]) * id;
            dtau_r[j] = fma(H, fma(K.Ks, n[j], K.Kd * pv), t4 * n[j]);
        }
        const double tid = tau * id;
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) dRb_r[i][j] = -fma(m[i], dtau_r[j], tid * (M[j][i] - m[i] * n[j]));
        // d vi / d q, d m / d q, d R_b / d q
        double dvi_q[3][4], dm_q[3][4], dRb_q[3][4];
        dM_dq_apply<+1>(s, a, v, dvi_q);
        dM_dq_apply<-1>(s, a, n, dm_q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double dtau = kdH * fma(n[0], dvi_q[0][j], fma(n[1], dvi_q[1][j], n[2] * dvi_q[2][j]));
#pragma unroll
            for (int i = 0; i < 3; ++i) dRb_q[i][j] = -fma(dtau, m[i], tau * dm_q[i][j]);
        }

        // =========================== rows v_dot (0..2) ============================================
        const double im = K.inv_mass;
        const double dF[3][3] = {{dFx[0], dFx[1], dFx[2]}, {dFy[0], dFy[1], dFy[2]}, {dFz[0], dFz[1], dFz[2]}};
        // -d(w x v)/dv = -[w]x ;  -d(w x v)/dw = +[v]x
        const double Wx[3][3] = {{0.0, -w[2], w[1]}, {w[2], 0.0, -w[0]}, {-w[1], w[0], 0.0}};
        const double Vx[3][3] = {{0.0, -v[2], v[1]}, {v[2], 0.0, -v[0]}, {-v[1], v[0], 0.0}};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(i, j, fma(dF[i][j] + dRb_v[i][j], im, -Wx[i][j]));
        // d/dw: aero damping terms
        const double X1w1 = sa * A.kLq * V, Z1w1 = -ca * A.kLq * V;
        const double dFw[3][3] = {{0.0, cb * X1w1, 0.0}, {A.kYp * V, sb * X1w1, A.kYr * V}, {0.0, Z1w1, 0.0}};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                if (i == 0 && j == 0) continue;      // structurally zero (SURVEY.md Appendix A)
                if (i == 2 && j == 2) continue;
                sink.jx(i, 3 + j, fma(dFw[i][j], im, Vx[i][j]));
            }
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(i, 6 + j, dRb_r[i][j] * im);
        // d/dq: tether + gravity  (d(g M^T e3)/dq = g * [dM20, dM21, dM22]/dq)
        const double gq[3][4] = {{-2.0 * a[1], 2.0 * a[2], -2.0 * s, 2.0 * a[0]},
                                 {2.0 * a[0], 2.0 * s, 2.0 * a[2], 2.0 * a[1]},
                                 {2.0 * s, -2.0 * a[0], -2.0 * a[1], 2.0 * a[2]}};
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) sink.jx(i, 9 + j, fma(dRb_q[i][j], im, K.g * gq[i][j]));
        // d/du
        const double ZdE = -A.CLde * qS;
        sink.ju(0, 0, im);
        sink.ju(0, 1, -sa * ZdE * im);
        sink.ju(2, 1, ca * ZdE * im);
        sink.ju(1, 2, A.CYdr * qS * im);

        // =========================== rows w_dot (3..5) ============================================
        // d rhs / d v
        double drh[3][3];
#pragma unroll
        for (int j = 0; j < 3; ++j) { drh[0][j] = dMax[j]; drh[1][j] = dMy[j]; drh[2][j] = dMaz[j]; }
        if (K.has_arm) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                drh[0][j] += K.arm1 * dRb_v[2][j] - K.arm2 * dRb_v[1][j];
                drh[1][j] += K.arm2 * dRb_v[0][j] - K.arm0 * dRb_v[2][j];
                drh[2][j] += K.arm0 * dRb_v[1][j] - K.arm1 * dRb_v[0][j];
            }
        }
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            sink.jx(3, j, fma(K.Ji00, drh[0][j], K.Ji02 * drh[2][j]));
            sink.jx(4, j, K.Ji11 * drh[1][j]);
            sink.jx(5, j, fma(K.Ji02, drh[0][j], K.Ji22 * drh[2][j]));
        }
        // d rhs / d w = d Maero/dw - d(w x Jw)/dw
        {
            const double Lw0 = A.klp * V, Lw2 = A.klr * V, Nw0 = A.knp * V, Nw2 = A.knr * V;
            double g_[3][3];
            g_[0][0] = fma(ca, Lw0, -sa * Nw0) - (w[1] * K.Ixz);
            g_[0][1] = -(Jw2 - w[2] * K.Iyy);
            g_[0][2] = fma(ca, Lw2, -sa * Nw2) - (w[1] * K.Izz - Jw1);
            g_[1][0] = -(w[2] * K.Ixx - Jw2 - w[0] * K.Ixz);
            g_[1][1] = A.kmq * V;
            g_[1][2] = -(Jw0 + w[2] * K.Ixz - w[0] * K.Izz);
            g_[2][0] = fma(sa, Lw0, ca * Nw0) - (Jw1 - w[1] * K.Ixx);
            g_[2][1] = -(w[0] * K.Iyy - Jw0);
            g_[2][2] = fma(sa, Lw2, ca * Nw2) + (w[1] * K.Ixz);
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                sink.jx(3, 3 + j, fma(K.Ji00, g_[0][j], K.Ji02 * g_[2][j]));
                sink.jx(4, 3 + j, K.Ji11 * g_[1][j]);
                sink.jx(5, 3 + j, fma(K.Ji02, g_[0][j], K.Ji22 * g_[2][j]));
            }
        }
        if (K.has_arm) {
            // d(arm x R_b)/d r and /d q
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const double c0 = K.arm1 * dRb_r[2][j] - K.arm2 * dRb_r[1][j];
                const double c1 = K.arm2 * dRb_r[0][j] - K.arm0 * dRb_r[2][j];
                const double c2 = K.arm0 * dRb_r[1][j] - K.arm1 * dRb_r[0][j];
                sink.jx(3, 6 + j, fma(K.Ji00, c0, K.Ji02 * c2));
                sink.jx(4, 6 + j, K.Ji11 * c1);
                sink.jx(5, 6 + j, fma(K.Ji02, c0, K.Ji22 * c2));
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double c0 = K.arm1 * dRb_q[2][j] - K.arm2 * dRb_q[1][j];
                const double c1 = K.arm2 * dRb_q[0][j] - K.arm0 * dRb_q[2][j];
                const double c2 = K.arm0 * dRb_q[1][j] - K.arm1 * dRb_q[0][j];
                sink.jx(3, 9 + j, fma(K.Ji00, c0, K.Ji02 * c2));
                sink.jx(4, 9 + j, K.Ji11 * c1);
                sink.jx(5, 9 + j, fma(K.Ji02, c0, K.Ji22 * c2));
            }
        }
        // d/du
        {
            const double MdE = A.cCmde * qS;
            const double LdR = A.bCldr * qS, NdR = A.bCndr * qS;
            const double r0 = fma(ca, LdR, -sa * NdR), r2 = fma(sa, LdR, ca * NdR);
            sink.ju(4, 1, K.Ji11 * MdE);
            sink.ju(3, 2, fma(K.Ji00, r0, K.Ji02 * r2));
            sink.ju(5, 2, fma(K.Ji02, r0, K.Ji22 * r2));
        }

        // =========================== rows r_dot (6..8) ============================================
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(6 + i, j, M[i][j]);
#pragma unroll
            for (int j = 0; j < 4; ++j) sink.jx(6 + i, 9 + j, dvi_q[i][j]);
        }

        // =========================== rows q_dot (9..12) ===========================================
        // d/dw: row0 = -a/2 ; rows 1..3 = (s I + [a]x)/2
        const double hs = 0.5 * s, h0 = 0.5 * a[0], h1 = 0.5 * a[1], h2 = 0.5 * a[2];
        const double Qw[4][3] = {{-h0, -h1, -h2}, {hs, -h2, h1}, {h2, hs, -h0}, {-h1, h0, hs}};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(9 + i, 3 + j, Qw[i][j]);
        // d/dq: Omega(w)/2 + mu I + lambda q q^T
        const double g0 = 0.5 * w[0], g1 = 0.5 * w[1], g2 = 0.5 * w[2];
        const double Om[4][4] = {{0.0, -g0, -g1, -g2}, {g0, 0.0, g2, -g1}, {g1, -g2, 0.0, g0}, {g2, g1, -g0, 0.0}};
        const double qv[4] = {s, a[0], a[1], a[2]};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                sink.jx(9 + i, 9 + j, fma(K.lambda * qv[i], qv[j], Om[i][j] + (i == j ? mu : 0.0)));
    }
}

template <bool JAC, class Sink, class AC>
__device__ __forceinline__ void kite_eval(const KiteConsts& K, const AC& A, const double (&x)[13],
                                          const double (&u)[3], double (&f)[13], Sink& sink) {
    kite_eval_c<JAC>(K, A, x, ctrl_terms(K, A, u), f, sink);
}

// Rigid-body kinematics (kite.cpp:622-661): v_dot = w_dot = 0.
template <bool JAC, class Sink>
__device__ __forceinline__ void rigid_eval(const KiteConsts& K, const double (&x)[13], double (&f)[13], Sink& sink) {
    const double v[3] = {x[0], x[1], x[2]};
    const double w[3] = {x[3], x[4], x[5]};
    const double s = x[9];
    const double a[3] = {x[10], x[11], x[12]};
    double M[3][3], nq;
    attitude_matrix(s, a, M, nq);
#pragma unroll
    for (int i = 0; i < 6; ++i) f[i] = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) f[6 + i] = fma(M[i][0], v[0], fma(M[i][1], v[1], M[i][2] * v[2]));
    const double hl = 0.5 * K.lambda;
    const double mu = fma(nq, hl, -hl);                                // (lambda / 2) (|q|^2 - 1)
    const double hw[3] = {0.5 * w[0], 0.5 * w[1], 0.5 * w[2]};         // q_dot = q (x) [0, w/2] + mu q
    f[9] = fma(mu, s, -fma(a[0], hw[0], fma(a[1], hw[1], a[2] * hw[2])));
    f[10] = fma(mu, a[0], fma(s, hw[0], fma(a[1], hw[2], -a[2] * hw[1])));
    f[11] = fma(mu, a[1], fma(s, hw[1], fma(a[2], hw[0], -a[0] * hw[2])));
    f[12] = fma(mu, a[2], fma(s, hw[2], fma(a[0], hw[1], -a[1] * hw[0])));
    if constexpr (JAC) {
        double dvi_q[3][4];
        dM_dq_apply<+1>(s, a, v, dvi_q);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(6 + i, j, M[i][j]);
#pragma unroll
            for (int j = 0; j < 4; ++j) sink.jx(6 + i, 9 + j, dvi_q[i][j]);
        }
        const double hs = 0.5 * s, h0 = 0.5 * a[0], h1 = 0.5 * a[1], h2 = 0.5 * a[2];
        const double Qw[4][3] = {{-h0, -h1, -h2}, {hs, -h2, h1}, {h2, hs, -h0}, {-h1, h0, hs}};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) sink.jx(9 + i, 3 + j, Qw[i][j]);
        const double g0 = 0.5 * w[0], g1 = 0.5 * w[1], g2 = 0.5 * w[2];
        const double Om[4][4] = {{0.0, -g0, -g1, -g2}, {g0, 0.0, g2, -g1}, {g1, -g2, 0.0, g0}, {g2, g1, -g0, 0.0}};
        const double qv[4] = {s, a[0], a[1], a[2]};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                sink.jx(9 + i, 9 + j, fma(K.lambda * qv[i], qv[j], Om[i][j] + (i == j ? mu : 0.0)));
    }
}

// Model dispatch (RIGID is a compile-time flag so the kite kernels carry no dead code).
template <bool RIGID, bool JAC, class Sink, class AC>
__device__ __forceinline__ void model_eval(const KiteConsts& K, const AC& A, const double (&x)[13],
                                           const double (&u)[3], double (&f)[13], Sink& sink) {
    if constexpr (RIGID) rigid_eval<JAC>(K, x, f, sink);
    else kite_eval<JAC>(K, A, x, u, f, sink);
}

template <bool RIGID, bool JAC, class Sink, class AC>
__device__ __forceinline__ void model_eval_c(const KiteConsts& K, const AC& A, const double (&x)[13],
                                             const CtrlTerms& uc, double (&f)[13], Sink& sink) {
    if constexpr (RIGID) rigid_eval<JAC>(K, x, f, sink);
    else kite_eval_c<JAC>(K, A, x, uc, f, sink);
}

// One classical RK4 step in registers (kitemath.cpp:36-51): x <- x + h/6 (k1 + 2 k2 + 2 k3 + k4).
// Tableau of the classical RK4 step for one step size, filled on the host and read from the kernel's constant bank:
//   an[st] = offset of the NEXT stage (h/2, h/2, h, -), w[st] = weight (1, 2, 2, 1), h6 = h / 6.
// Indexed by the (uniform) stage counter they arrive as uniform-register operands: `fma(an, k, x)` then reads two vector
// registers instead of three (an FP64 instruction with three distinct vector-register operands issues every 3 cycles, not 2:
// profiles/r2j_dfma_operands.log), and h / 6 is not an FP64 division (MUFU seed + Newton chain + slow-path CALL) per step.
struct RkTab {
    double an[4], w[4], h6;
};
__host__ __device__ inline RkTab make_rk_tab(double h) {
    RkTab t;
    t.an[0] = 0.5 * h; t.an[1] = 0.5 * h; t.an[2] = h; t.an[3] = 0.0;
    t.w[0] = 1.0; t.w[1] = 2.0; t.w[2] = 2.0; t.w[3] = 1.0;
    t.h6 = h / 6.0;
    return t;
}
struct NoHook {
    __device__ __forceinline__ void operator()(int, const double (&)[13]) const {}
};
// JAC: stage 1 also emits d f/d x and d f/d u at the pre-step state through `sink`.  `hook(st, xs)` runs before stage st
// (0..3) with that stage's input state xs.
template <bool RIGID, bool JAC = false, class AC, class Sink = NoSink, class Hook = NoHook>
__device__ __forceinline__ void rk4_step(const KiteConsts& K, const AC& A, double (&x)[13], const double (&u)[3],
                                         const RkTab& rk, const Sink& sink = Sink{}, const Hook& hook = Hook{}) {
    NoSink ns;
    double k[13], acc[13], xt[13];
    const CtrlTerms uc = ctrl_terms(K, A, u);                    // the control is held for all four stages
    // Stage 1 is peeled off the loop: it reads the base state directly and its slope IS the accumulator (b_1 = 1), so the step
    // needs neither the 26 register moves xt = x, nor the 13 zeroings, nor the 13 FMAs acc = 0 + 1 * k (bitwise the same
    // result).  Stages 2..4 run as a real loop (one more copy of the RHS in the instruction stream: the fully unrolled body was
    // ~100 KB of SASS and stalled on instruction fetch, profiles/r1a_rollout_ncu_summary.txt; two copies do not).
    // Config 2: 77.8 -> 75.6 ms.
    hook(0, x);
    model_eval_c<RIGID, JAC>(K, A, x, uc, k, sink);
#pragma unroll
    for (int i = 0; i < 13; ++i) { acc[i] = k[i]; xt[i] = fma(rk.an[0], k[i], x[i]); }
#pragma unroll 1
    for (int st = 1; st < 4; ++st) {
        hook(st, xt);
        model_eval_c<RIGID, false>(K, A, xt, uc, k, ns);
        const double wgt = rk.w[st];                             // tableau weights b = (1,2,2,1)/6
        const double an = rk.an[st];                             // next stage offset a = (1/2, 1/2, 1, 0)
        // (one loop, accumulator and next stage input side by side: the two FMAs of a component share k[i] in the same operand
        // slot.  Split into two loops, or with the last stage's unused input skipped by a uniform branch, the step is 1 % slower:
        // 76.2 - 76.5 ms against 75.6, profiles/r2y_sweep_skiplast.log, r2y_sweep_fused.log)
#pragma unroll
        for (int i = 0; i < 13; ++i) { acc[i] = fma(wgt, k[i], acc[i]); xt[i] = fma(an, k[i], x[i]); }
    }
#pragma unroll
    for (int i = 0; i < 13; ++i) x[i] = fma(rk.h6, acc[i], x[i]);
}

// ---- counter-based synthetic inputs (workload definition; identical to oracle::counter_uniform) ----
__host__ __device__ inline uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__host__ __device__ inline double counter_uniform(uint64_t seed, uint64_t traj, uint64_t step, uint64_t channel) {
    uint64_t k = splitmix64(seed ^ splitmix64(traj ^ splitmix64((step << 8) | channel)));
    return double(k >> 11) * (1.0 / 9007199254740992.0);
}
#define KITE_SYNTH_SEED 0x6b697465ULL

__device__ __forceinline__ void synth_control(uint64_t traj, uint64_t step, double (&u)[3]) {
    const double amax = 8.0 * (3.14159265358979323846 / 180.0);
    u[0] = __dmul_rn(0.3, counter_uniform(KITE_SYNTH_SEED, traj, step, 0));
    u[1] = __dmul_rn(amax, __dadd_rn(__dmul_rn(2.0, counter_uniform(KITE_SYNTH_SEED, traj, step, 1)), -1.0));
    u[2] = __dmul_rn(amax, __dadd_rn(__dmul_rn(2.0, counter_uniform(KITE_SYNTH_SEED, traj, step, 2)), -1.0));
}
__device__ __forceinline__ void synth_x0(uint64_t traj, double (&x0)[13]) {
    const double base[13] = {6.1977743e+00, -2.8407148e-02, 9.1815942e-01, 2.9763089e-01, -2.2052198e+00,
                             -1.4827499e-01, -4.1624807e-01, -2.2601052e+00, 1.2903439e+00, 3.5646195e-02,
                             -6.9986094e-02, 8.2660637e-01, 5.5727089e-01};   // kite_model_test.cpp:58-60
    const double amp[13] = {0.5, 0.5, 0.5, 0.2, 0.2, 0.2, 0.2, 0.2, 0.2, 0.05, 0.05, 0.05, 0.05};
    // explicit _rn intrinsics: no FMA contraction, same operation order as the oracle, so the
    // generated inputs are bit-identical to the CPU generator under any sharding.
#pragma unroll
    for (int c = 0; c < 13; ++c) {
        const double t = __dadd_rn(__dmul_rn(2.0, counter_uniform(KITE_SYNTH_SEED, traj, 0xFFFFFFULL, c)), -1.0);
        x0[c] = __dadd_rn(base[c], __dmul_rn(amp[c], t));
    }
    const double nrm = sqrt(__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(x0[9], x0[9]), __dmul_rn(x0[10], x0[10])),
                                                __dmul_rn(x0[11], x0[11])), __dmul_rn(x0[12], x0[12])));
#pragma unroll
    for (int c = 9; c < 13; ++c) x0[c] = x0[c] / nrm;
}

// Identification sweep (SURVEY.md 8d config 5): parameter sample `traj` = reference coefficients perturbed uniformly inside
// the bounds of kite_identification_test.cpp:127-148 (fractions of |ref|), keyed on the GLOBAL sample index.
#define KITE_ID_BOUNDS_LO {-0.1, -0.05, -0.1, -0.5, -0.5, -0.1, -0.5, -0.5, -0.2, -0.3, -0.3, -0.5, -0.5, -0.5, -0.5, -0.3, -0.5, -0.5, -0.5, -0.5, -0.5}
#define KITE_ID_BOUNDS_HI {0.1, 0.1, 0.25, 0.5, 0.5, 0.30, 0.5, 0.5, 0.2, 0.3, 0.3, 0.5, 0.5, 0.5, 0.5, 1.0, 0.5, 0.5, 0.5, 0.5, 0.5}
__host__ __device__ inline double synth_id_param(uint64_t traj, int c, double ref) {
    const double lo[21] = KITE_ID_BOUNDS_LO, hi[21] = KITE_ID_BOUNDS_HI;
    const double t = counter_uniform(KITE_SYNTH_SEED, traj, 0xFFFFFEULL, (uint64_t)c);
#ifdef __CUDA_ARCH__
    const double frac = __dadd_rn(lo[c], __dmul_rn(__dadd_rn(hi[c], -lo[c]), t));
    return __dadd_rn(ref, __dmul_rn(fabs(ref), frac));
#else
    const double w = hi[c] - lo[c];
    const double frac = lo[c] + w * t;
    return ref + fabs(ref) * frac;
#endif
}

}  // namespace kite
