// =====================================================================================
// kite_math.cuh -- lean FP64 special functions for the kite kernels (sm_100a).
//
// More than half of the FP64 instructions of one RHS evaluation were CUDA libm special functions
// (profiles/r1a_*: 1210 FP64 instr per RK4 step, ~160 per RHS in sqrt/div/asin/atan2/exp incl. their
// special-case paths).  These replacements keep ~1 ulp accuracy on the value ranges the model can
// produce, drop the denormal/NaN slow paths (non-finite trajectories are flagged by the kernels
// instead) and share work between related quantities:
//   rcp / rsqrt : MUFU seed (rcp.approx / rsqrt.approx .ftz.f64) + ONE cubically convergent step
//   asin        : odd minimax polynomial on |x| <= 0.7072 (scripts/fit_math_polys.py), complement identity
//                 asin(s) = sign(s) (pi/2 - asin(cos)) beyond, so the whole range is branch free
//   logistic    : exp by Cody-Waite reduction + degree-11 polynomial, then rcp
// Host builds (tests/cpu_shim) emulate the MUFU seeds with float precision so the same source is
// checked on the CPU.
// =====================================================================================
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

namespace kite {

__device__ __forceinline__ double rcp_seed(double a) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    return y;
#else
    return (double)(1.0f / (float)a);
#endif
}
__device__ __forceinline__ double rsqrt_seed(double a) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    return y;
#else
    return (double)(1.0f / sqrtf((float)a));
#endif
}

// High word of a double as a signed integer.  Sign and magnitude tests on it run on the integer pipe (ISETP) and leave the
// FP64 pipe to the arithmetic: for finite a, hi(a) > 0 <=> a >= 2^-1022 (a positive normal), hi(a) < 0 <=> sign bit set.
__device__ __forceinline__ int hi_word(double a) {
#ifdef __CUDA_ARCH__
    return __double2hiint(a);
#else
    int64_t b; memcpy(&b, &a, sizeof b); return (int)(b >> 32);
#endif
}
// Measured against FP64 compares (profiles/r2b_sweep.log): 82.51 -> 81.91 ms per config-2 pass, 7 DSETP per RHS off the FP64 pipe.
__device__ __forceinline__ bool is_pos(double a) {            // a > 0 (denormals count as 0 in the integer form)
    return hi_word(a) > 0;
}
__device__ __forceinline__ bool is_neg(double a) {            // a < 0
    return hi_word(a) < 0;
}

// 1/a: seed error e0 <= 2^-19  ->  y0 (1 + e + e^2), e = 1 - a y0, error e0^3 <= 2^-57.   MUFU + 3 DFMA.
__device__ __forceinline__ double fast_rcp(double a) {
    const double y0 = rcp_seed(a);
    const double e = fma(-a, y0, 1.0);
    const double e2 = fma(e, e, e);
    return fma(y0, e2, y0);
}
// 1/sqrt(a): y0 (1 + e/2 + 3 e^2/8), e = 1 - a y0^2, error ~ (5/16) e0^3.   MUFU + 5 FP64.
__device__ __forceinline__ double fast_rsqrt(double a) {
    const double y0 = rsqrt_seed(a);
    const double t = a * y0;
    const double e = fma(-t, y0, 1.0);
    const double p = fma(0.375, e, 0.5) * e;
    return fma(y0, p, y0);
}

// NOTE: the coefficients are written as literals on purpose.  FP64 instructions on sm_100a take constants only through
// uniform registers; a coefficient TABLE (__constant__ or constexpr array) is hoisted out of the stage loop into
// ~40 uniform registers, which overflow into vector registers and from there into local memory (228 B of spills
// in k_rk4_rollout).  Literals are re-materialised next to their use (2 UMOV each) and cost no registers.

// asin(x) = x + x u P(u), u = x^2, |x| <= 0.7072; degree 16, max relative error 4.4e-16 (scripts/fit_math_polys.py)
#define KITE_ASIN_POLY_MAX 0.7072
__device__ __forceinline__ double asin_poly(double x) {
    const double u = x * x;
    double p = 5.27314318387392955e-01;
    p = fma(p, u, -1.67855479930664897e+00);
    p = fma(p, u, 2.55375757459231778e+00);
    p = fma(p, u, -2.35809246022577668e+00);
    p = fma(p, u, 1.48923001382088138e+00);
    p = fma(p, u, -6.56023493249017098e-01);
    p = fma(p, u, 2.23097241478172448e-01);
    p = fma(p, u, -4.34132617562938208e-02);
    p = fma(p, u, 1.89243203271123074e-02);
    p = fma(p, u, 1.03696475274575421e-02);
    p = fma(p, u, 1.40738595019858897e-02);
    p = fma(p, u, 1.73458138976341353e-02);
    p = fma(p, u, 2.23724499523806075e-02);
    p = fma(p, u, 3.03819370896512217e-02);
    p = fma(p, u, 4.46428572403844703e-02);
    p = fma(p, u, 7.49999999994898220e-02);
    p = fma(p, u, 1.66666666666667102e-01);
    return fma(x * u, p, x);
}
// {cos(theta_k), theta_k} for theta_k = asin(k / 64), k = 0..47 (scripts: mpmath, correctly rounded)
#define KITE_ANGLE_TAB_VALUES { 1.00000000000000000e+00, 0.00000000000000000e+00, 9.99877922236009797e-01, 1.56256358527369493e-02, 9.99511599482467261e-01, 3.12550884994951539e-02, 9.98900763026538074e-01, 4.68921831332818687e-02, 9.98044963916956962e-01, 6.25407617964913870e-02, 9.96943571309329424e-01, 7.82046919347542807e-02, 9.95595770129624413e-01, 9.38878751075164775e-02, 9.94000558035557646e-01, 1.09594255910533803e-01, 9.92156741649221519e-01, 1.25327831168065396e-01, 9.90062932027555465e-01, 1.41092659455893887e-01, 9.87717539329944216e-01, 1.56892871020461205e-01, 9.85118766634257126e-01, 1.72732678164473352e-01, 9.82264602843856971e-01, 1.88616386175404105e-01, 9.79152814618331147e-01, 2.04548404880551649e-01, 9.75780937249749680e-01, 2.20533260920833335e-01, 9.72146264393892512e-01, 2.36575610845542905e-01, 9.68245836551854255e-01, 2.52680255142078647e-01, 9.64076428181396827e-01, 2.68852153328471066e-01, 9.59634533299005499e-01, 2.85096440252746219e-01, 9.54916349412345156e-01, 3.01418443762183463e-01, 9.49917759598166489e-01, 3.17823703927880730e-01, 9.44634312511990037e-01, 3.34317994036368416e-01, 9.39061200082294989e-01, 3.50907343591081111e-01, 9.33193232602444467e-01, 3.67598063603275793e-01, 9.27024810886957873e-01, 3.84396774495639082e-01, 9.20549895103464744e-01, 4.01310436993840502e-01, 9.13761969825840348e-01, 4.18346386443468110e-01, 9.06654004775250488e-01, 4.35512371064433745e-01, 8.99218410621134945e-01, 4.52816594744925582e-01, 8.91446989099744513e-01, 4.70267765085970069e-01, 8.83330876568910628e-01, 4.87875147540292931e-01, 8.74860479948088687e-01, 5.05648626651396538e-01, 8.66025403784438597e-01, 5.23598775598298927e-01, 8.56814366928449700e-01, 5.41736935498202010e-01, 8.47215106982872390e-01, 5.60075306226581970e-01, 8.37214270288675899e-01, 5.78627050899099715e-01, 8.26797284707684543e-01, 5.97406416645350213e-01, 8.15948211821681757e-01, 6.16428874921707171e-01, 8.04649574348983321e-01, 6.35711285401302173e-01, 7.92882153522829647e-01, 6.55272088500942207e-01, 7.80624749799799789e-01, 6.75131532937031653e-01, 7.67853898456600903e-01, 6.95311946456768082e-01, 7.54543529228102305e-01, 7.15838060225111206e-01, 7.40664555905708233e-01, 7.36737400489643868e-01, 7.26184377413890636e-01, 7.58040765426235996e-01, 7.11066265811422071e-01, 7.79782810980313545e-01, 6.95268608165218405e-01, 8.02002777803618505e-01, 6.78743957155421018e-01, 8.24745403185475734e-01 }
#ifdef __CUDA_ARCH__
static __device__ const double ANGLE_TAB[96] = KITE_ANGLE_TAB_VALUES;
#else
static const double ANGLE_TAB[96] = KITE_ANGLE_TAB_VALUES;
#endif
// Angle phi in [-pi/4 - , pi/4 + ] from x = sin(phi), y = cos(phi) by table + short series instead of the degree-16 polynomial:
//   k = rint(64 x), theta_k = asin(k / 64) from the table, d = sin(phi - theta_k) = x cos(theta_k) - y (k / 64), |d| <= 0.0112,
//   phi = theta_k + d (1 + d^2 (1/6 + 3/40 d^2 + 15/336 d^4))     (next term 35/1152 d^9: 7e-18 relative)
// 9 FP64 instructions and a 9-deep dependency chain against 19 / 19; absolute error <= 3e-16 (test_lean_math_accuracy).
// k / 64 comes straight out of the rounding constant (t / 64 - magic / 64 is exact), and the series ends in one FMA onto
// theta_k, so no instruction reads three fresh vector registers.
// The product kernels use this form everywhere: config 2 81.38 -> 80.10 ms against the polynomial (profiles/r2r_sweep.log).
__device__ __forceinline__ double asin_red(double x, double y) {
    const double magic = 6755399441055744.0;              // 1.5 * 2^52: the low word of x * 64 + magic is rint(64 x)
    const double t = fma(x, 64.0, magic);
    const double kf = fma(t, 0.015625, -magic * 0.015625);  // k / 64, exact
#ifdef __CUDA_ARCH__
    int k = __double2loint(t);
    k = k < 0 ? -k : k;
    const double2 e = __ldg(reinterpret_cast<const double2*>(ANGLE_TAB) + k);      // one 16-byte gather, L1 resident
    const double ck = e.x, thk = e.y;
#else
    int64_t bits; memcpy(&bits, &t, sizeof bits);
    int k = (int)(int32_t)(bits & 0xFFFFFFFF);
    k = k < 0 ? -k : k;
    const double ck = ANGLE_TAB[2 * k], thk = ANGLE_TAB[2 * k + 1];
#endif
    const double d = fma(-y, kf, x * ck);
    const double u = d * d;
    double p = fma(4.46428571428571425e-02, u, 7.49999999999999972e-02);
    p = fma(p, u, 1.66666666666666657e-01);
    p = fma(p, u, 1.0);
    return fma(d, p, copysign(thk, kf));
}
// Angle in [-pi/2, pi/2] from its sine s and cosine c >= 0 (s^2 + c^2 = 1), branch free over the whole range:
//   |s| <= 1/sqrt2 : asin(s)            |s| > 1/sqrt2 : sign(s) (pi/2 - asin(c)),  c < 1/sqrt2
// so the polynomial argument never leaves |x| <= 0.7072 and a warp never diverges into libm (random-control
// rollouts sit at |sideslip| > 37 deg for ~40% of the horizon: profiles/r1f sweep).
template <bool TAB>
__device__ __forceinline__ double asin_sc(double s, double c) {
    // |s| > 0.70710678 on the high words (0x3FE6A09E = hi(1/sqrt 2); the polynomial is valid up to 0.7072 on either side)
    const bool big = (hi_word(s) & 0x7fffffff) > 0x3FE6A09E;
    const double r = TAB ? asin_red(big ? c : s, big ? fabs(s) : c) : asin_poly(big ? c : s);
    const double t = (1.5707963267948966 - r) + 6.123233995736766e-17;
    return big ? copysign(t, s) : r;
}
// atan2(y, x) from the normalised pair s = y/hypot, c = x/hypot, any quadrant, branch free:
//   c >= 0 : asin_sc(s, c)              c < 0 : sign(s) pi - asin_sc(s, -c)
template <bool TAB>
__device__ __forceinline__ double atan2_sc(double s, double c) {
    const double r = asin_sc<TAB>(s, fabs(c));
    const double t = (copysign(3.141592653589793, s) - r) + copysign(1.2246467991473532e-16, s);
    return is_neg(c) ? t : r;
}

// 2^(j/32), j = 0..31 (mpmath, correctly rounded)
#define KITE_EXP2_TAB_VALUES { 1.00000000000000000e+00, 1.02189714865411663e+00, 1.04427378242741375e+00, 1.06714040067682370e+00, 1.09050773266525769e+00, 1.11438674259589243e+00, 1.13878863475669156e+00, 1.16372485877757748e+00, 1.18920711500272103e+00, 1.21524735998046896e+00, 1.24185781207348400e+00, 1.26905095719173322e+00, 1.29683955465100964e+00, 1.32523664315974132e+00, 1.35425554693689265e+00, 1.38390988196383202e+00, 1.41421356237309515e+00, 1.44518080697704665e+00, 1.47682614593949935e+00, 1.50916442759342284e+00, 1.54221082540794074e+00, 1.57598084510788650e+00, 1.61049033194925428e+00, 1.64575547815396495e+00, 1.68179283050742900e+00, 1.71861929812247793e+00, 1.75625216037329945e+00, 1.79470907500310717e+00, 1.83400808640934243e+00, 1.87416763411029996e+00, 1.91520656139714740e+00, 1.95714412417540018e+00 }
#ifdef __CUDA_ARCH__
static __device__ const double EXP2_TAB[32] = KITE_EXP2_TAB_VALUES;
#else
static const double EXP2_TAB[32] = KITE_EXP2_TAB_VALUES;
#endif

// logistic(4 e) = 1 / (1 + exp(-4 e)), the tether's smoothed step; argument clamped to |4 e| <= 700 (result 0 / 1 to within
// 1e-304 beyond).  exp(a) at a = -4 e is evaluated on the reduced argument r' = r / (-4): every literal below is the one of
// the plain exp(a) form times a power of two ((-4)^k for the k-th polynomial coefficient, -1/4 for the reduction constants,
// -4 for the rounding product), so each rounding lands on the same scaled value and the result is bitwise that of exp(a)
// with a = -4 e, without the FP64 instruction that forms a.
template <bool TAB>
__device__ __forceinline__ double fast_logistic4(double e) {
    e = fmax(fmin(e, 175.0), -175.0);
    if constexpr (TAB)
    // exp(a) = 2^m * 2^(j/32) * exp(r): n = rint(a * 32 / ln2) = 32 m + j, r = a - n ln2/32 (Cody-Waite), |r| <= ln2/64 = 0.0108,
    // exp(r) by a degree-6 Taylor polynomial (r^7/5040 = 3.5e-18): 12 FP64 instructions against 17 with the degree-11 one.
    {
        const double magic = 6755399441055744.0;
        const double tn = fma(e, -4.0 * 4.61662413084468283e+01, magic);
        const double nf = tn - magic;
        double r = fma(nf, 0.25 * 2.16608493865351193e-02, e);
        r = fma(nf, 0.25 * 5.96317165397058656e-12, r);
        double p = 4096.0 * 1.38888888888888894e-03;
        p = fma(p, r, -1024.0 * 8.33333333333333322e-03);
        p = fma(p, r, 256.0 * 4.16666666666666644e-02);
        p = fma(p, r, -64.0 * 1.66666666666666657e-01);
        p = fma(p, r, 16.0 * 5.00000000000000000e-01);
        p = fma(p, r, -4.0 * 1.00000000000000000e+00);
        p = fma(p, r, 1.00000000000000000e+00);
        int64_t bits;
        memcpy(&bits, &tn, sizeof bits);
        const int n = (int32_t)(bits & 0xFFFFFFFF);
#ifdef __CUDA_ARCH__
        const double tj = __ldg(EXP2_TAB + (n & 31));
#else
        const double tj = EXP2_TAB[n & 31];
#endif
        const int64_t sb = (int64_t)((n >> 5) + 1023) << 52;             // 2^m, |m| <= 32: normal
        double scale;
        memcpy(&scale, &sb, sizeof scale);
        const double ex = (p * tj) * scale;
        return fast_rcp(1.0 + ex);
    }
    // n = rint(a * log2(e)) by the 1.5 * 2^52 trick; r = a - n ln2 (Cody-Waite, hi part has 32 trailing zero bits)
    const double magic = 6755399441055744.0;
    const double tn = fma(e, -4.0 * 1.44269504088896339e+00, magic);
    const double nf = tn - magic;
    double r = fma(nf, 0.25 * 6.93146705627441406e-01, e);
    r = fma(nf, 0.25 * 4.74932503903167256e-07, r);
    // exp(r), |r| <= ln2/2, degree 11 (scripts/fit_math_polys.py)
    double p = -4194304.0 * 2.51100492048186583e-08;
    p = fma(p, r, 1048576.0 * 2.76326547225277896e-07);
    p = fma(p, r, -262144.0 * 2.75572408872298695e-06);
    p = fma(p, r, 65536.0 * 2.48014854415613131e-05);
    p = fma(p, r, -16384.0 * 1.98412698900764028e-04);
    p = fma(p, r, 4096.0 * 1.38888889523528631e-03);
    p = fma(p, r, -1024.0 * 8.33333333331958900e-03);
    p = fma(p, r, 256.0 * 4.16666666664879531e-02);
    p = fma(p, r, -64.0 * 1.66666666666666796e-01);
    p = fma(p, r, 16.0 * 5.00000000000001887e-01);
    p = fma(p, r, -4.0 * 1.00000000000000000e+00);
    p = fma(p, r, 1.00000000000000000e+00);
    // scale by 2^n: n is in the low word of tn (|n| <= 1010, so the biased exponent stays normal)
    int64_t bits;
    memcpy(&bits, &tn, sizeof bits);
    const int64_t n = (int64_t)(int32_t)(bits & 0xFFFFFFFF);
    const int64_t sb = (n + 1023) << 52;
    double scale;
    memcpy(&scale, &sb, sizeof scale);
    const double ex = p * scale;                  // exp(-4 e)
    return fast_rcp(1.0 + ex);
}
// logistic(x) = 1 / (1 + exp(-x)): x / 4 is exact, so this is bitwise the logistic of x.
template <bool TAB>
__device__ __forceinline__ double fast_logistic(double x) {
    return fast_logistic4<TAB>(0.25 * x);
}

}  // namespace kite
