// kite_consts.h -- host-side folding of kite_params (the KiteProperties subset, include/kite_b200.h)
// into the constants the device model consumes.  Environmental constants g, ro: kite.cpp:93-94.
#pragma once
#include "../../include/kite_b200.h"
#include "kite_model.cuh"

namespace kite {

inline KiteConsts make_consts(const kite_params& P, int model_kind) {
    const double g = 9.80665, ro = 1.2985, pi = 3.14159265358979323846;
    KiteConsts K{};
    K.model_kind = model_kind;
    K.eps = (model_kind == KITE_MODEL_KITE) ? 1e-4 : 0.0;
    K.cqS = 0.5 * ro * P.S;
    K.b = P.b; K.c = P.c;
    K.inv_piAR = 1.0 / (pi * P.e_oswald * P.AR);
    K.bCn0 = P.b * P.Cn0; K.bCl0 = P.b * P.Cl0;
    K.inv_mass = 1.0 / P.mass; K.g = g;
    K.Lt = P.tether_length; K.Ks = P.Ks; K.Kd = P.Kd;
    K.arm0 = P.rx; K.arm1 = P.ry; K.arm2 = P.rz;
    K.has_arm = (P.rx != 0.0 || P.ry != 0.0 || P.rz != 0.0) ? 1 : 0;
    K.Ixx = P.Ixx; K.Iyy = P.Iyy; K.Izz = P.Izz; K.Ixz = P.Ixz;
    K.IzmIy = P.Izz - P.Iyy; K.IymIx = P.Iyy - P.Ixx; K.IzmIx = P.Izz - P.Ixx;
    const double det = P.Ixx * P.Izz - P.Ixz * P.Ixz;     // closed-form inverse of J (SURVEY.md Q7)
    K.Ji00 = P.Izz / det; K.Ji02 = -P.Ixz / det; K.Ji11 = 1.0 / P.Iyy; K.Ji22 = P.Ixx / det;
    K.lambda = (model_kind == KITE_MODEL_RIGID_BODY) ? -10.0 : -5.0;    // kite.cpp:316 / :639
    K.sLq = 0.25 * P.c * P.S * ro;
    K.smq = 0.25 * P.S * P.c * P.c * ro;
    K.sY = 0.25 * P.b * ro * P.S;
    K.sb2 = 0.25 * ro * P.b * P.b * P.S;
    const double p[21] = {P.CL0, P.CLa_total, P.CD0_total, P.CYb, P.Cm0, P.Cma, P.Cnb, P.Clb, P.CLq, P.Cmq, P.CYr,
                          P.Cnr, P.Clr, P.CYp, P.Clp, P.Cnp, P.CLde, P.CYdr, P.Cmde, P.Cndr, P.Cldr};
    derive_coef(K, p, K.A);
    return K;
}

}  // namespace kite
