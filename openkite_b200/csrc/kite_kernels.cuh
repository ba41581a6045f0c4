// =====================================================================================
// kite_kernels.cuh -- sm_100a kernels of the batched kite engine.
//
// Data layout: structure-of-arrays, component c of unit i at ptr[c*ld + i]; a warp touches 32
// consecutive units of one component = one 256 B coalesced request.  All kernels are FP64
// FMA-pipe bound (no tensor cores: the work is scalar per-trajectory arithmetic, SURVEY.md 8d);
// model constants travel as a __grid_constant__ kernel parameter so they are read straight from
// the constant bank as DFMA operands and cost no registers.
// =====================================================================================
#pragma once
#include <cuda.h>
#include <cuda_pipeline.h>

#include "kite_model.cuh"
#include "kite_sparsity.h"

namespace kite {

// ---- compact Jacobian storage -----------------------------------------------------------------
// Structural non-zeros of [Jx | Ju] (SURVEY.md Appendix A), row-major slot numbering.  The 21 entries
// that only exist with a tether arm (rows w_dot, cols r,q) get slots too but are only touched when
// has_arm.  The slot tables of the kernels (SENS_TAB) are built from these predicates.
constexpr int JX_SLOTS = 125;
constexpr int JAC_SLOTS = JX_SLOTS + 7;   // 132
constexpr int JAC_SLOTS_NOARM = 111;      // 104 + 7 structural non-zeros of a zero-arm model (+ 21 with a tether arm)

// Sink: dense 13x13 / 13x3 row-major, SoA over units (buffers pre-zeroed by the caller).
struct DenseSink {
    double* jxp; double* jup; long ld;
    __device__ __forceinline__ void jx(int i, int j, double v) const { if (jxp) jxp[(long)(i * 13 + j) * ld] = v; }
    __device__ __forceinline__ void ju(int i, int j, double v) const { if (jup) jup[(long)(i * 3 + j) * ld] = v; }
    __device__ __forceinline__ void aero(double, double, double) const {}
};

__device__ __forceinline__ void load_coef(const KiteConsts& K, const double* __restrict__ p, long ld, long i, AeroCoef& A) {
    double raw[21];
#pragma unroll
    for (int c = 0; c < 21; ++c) raw[c] = __ldg(p + (long)c * ld + i);
    derive_coef(K, raw, A);
}

__device__ __forceinline__ bool all_finite13(const double (&x)[13]) {
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < 13; ++c) s += x[c] * 0.0;     // NaN/Inf poison the sum
    return s == 0.0;
}

// Per-unit status flags (include/kite_b200.h, kite_status_flag) of a state the kite model is evaluated at: the airspeed
// and tether-length singularities of the RHS (SURVEY.md section 5).  Callers OR in KITE_FLAG_NONFINITE for their results.
constexpr int FLAG_NONFINITE = 1, FLAG_LOW_AIRSPEED = 2, FLAG_ZERO_TETHER = 4;
template <bool RIGID>
__device__ __forceinline__ int singularity_flags(const double (&x)[13]) {
    if constexpr (RIGID) return 0;                  // the rigid-body kinematics have neither term
    const double V2 = fma(x[0], x[0], fma(x[1], x[1], x[2] * x[2]));
    const double d2 = fma(x[6], x[6], fma(x[7], x[7], x[8] * x[8]));
    return (V2 < 1e-12 ? FLAG_LOW_AIRSPEED : 0) | (d2 < 1e-18 ? FLAG_ZERO_TETHER : 0);
}

// ================================================================================================
// rhs_batch / jac_batch : pointwise evaluators (kite.cpp:324, :327-328)
// ================================================================================================
struct PointArgs {
    KiteConsts K;
    long B, ld;
    const double* x; const double* u; const double* p;
    double* f; double* Jx; double* Ju;
    double* fa;              // [3][ld] body-frame aerodynamic force (Function "Aero", kite.cpp:330) or null
};
struct AeroSink {           // RHS-only evaluation that also captures the aerodynamic force
    double* fap; long ld;
    __device__ __forceinline__ void jx(int, int, double) const {}
    __device__ __forceinline__ void ju(int, int, double) const {}
    __device__ __forceinline__ void aero(double fx, double fy, double fz) const { if (fap) { fap[0] = fx; fap[ld] = fy; fap[2 * ld] = fz; } }
};

template <bool RIGID, bool PERCOEF, bool JAC>
__global__ void __launch_bounds__(128) k_point_eval(const __grid_constant__ PointArgs a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.B) return;
    double x[13], u[3], f[13];
#pragma unroll
    for (int c = 0; c < 13; ++c) x[c] = __ldg(a.x + (long)c * a.ld + i);
#pragma unroll
    for (int c = 0; c < 3; ++c) u[c] = a.u ? __ldg(a.u + (long)c * a.ld + i) : 0.0;
    AeroCoef A = a.K.A;
    if constexpr (PERCOEF) load_coef(a.K, a.p, a.ld, i, A);
    if constexpr (JAC) {
        DenseSink s{a.Jx ? a.Jx + i : nullptr, a.Ju ? a.Ju + i : nullptr, a.ld};
        model_eval<RIGID, true>(a.K, A, x, u, f, s);
    } else {
        AeroSink s{a.fa ? a.fa + i : nullptr, a.ld};
        model_eval<RIGID, false>(a.K, A, x, u, f, s);
    }
    if (a.f) {
#pragma unroll
        for (int c = 0; c < 13; ++c) a.f[(long)c * a.ld + i] = f[c];
    }
}

// ================================================================================================
// rk4_rollout : B trajectories x N steps, thread per trajectory, state in registers.
//   HBM traffic per state-step: 24 B of controls (KITE_U_PER_STEP), nothing else -> FP64-pipe bound.
// ================================================================================================
struct RolloutArgs {
    KiteConsts K;
    long B, ld, N;
    double h;
    RkTab rk;                // RK4 tableau for h (host-computed)
    const double* x0; const double* u; const double* p;
    double* xf; double* traj; long save_every;
    const double* y; double* cost;
    int32_t* status;
    long index0;
};

constexpr int ROLLOUT_BLOCK = 128;
// dynamic shared memory of a rollout CTA: the per-trajectory coefficients (PERCOEF)
constexpr size_t rollout_smem_bytes(bool percoef) {
    return percoef ? sizeof(AeroCoef) * ROLLOUT_BLOCK : 0;
}

// Per-warp scratch lines that are written and re-read within microseconds (stage states of the sensitivity kernel, Jacobian
// tiles of the EKF predict): L2 only, lowest eviction priority class "evict_last", so that the streaming output (which passes
// through the same L2) does not push the dirty lines out to HBM between the write and the read.
__device__ __forceinline__ unsigned long long scratch_policy() {
    unsigned long long pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));     // pure: the compiler may re-materialise it
    return pol;
}
__device__ __forceinline__ void st_scratch(double* p, double v) {
    asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" :: "l"(p), "d"(v), "l"(scratch_policy()) : "memory");
}
__device__ __forceinline__ double ld_scratch(const double* p) {
    double v;
    asm volatile("ld.global.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(scratch_policy()) : "memory");
    return v;
}

// Global thread index from the special registers, opaque to the optimiser: the rollout recomputes it after the time loop
// instead of keeping 2 registers alive (or spilled) across the whole horizon.
__device__ __forceinline__ long fresh_thread_index() {
    unsigned t, b, n;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
    asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(b));
    asm volatile("mov.u32 %0, %%ntid.x;" : "=r"(n));
    return (long)b * n + t;
}

template <int UMODE, bool RIGID, class AC>
__device__ __forceinline__ void rollout_body(const RolloutArgs& a, double (&x)[13], double (&u)[3], const AC& A);

template <int UMODE, bool RIGID, bool PERCOEF>
__global__ void __launch_bounds__(ROLLOUT_BLOCK, 3) k_rk4_rollout(const __grid_constant__ RolloutArgs a) {
    // per-trajectory aero coefficients (identification sweeps) live in shared memory, one 21-double record per thread
    // (odd stride: conflict free): 42 registers the RHS cannot spare (they spilled: 96 B / 80 B per thread in round 1)
    extern __shared__ __align__(16) unsigned char rollout_smem[];
    if (fresh_thread_index() >= a.B) return;
    double x[13], u[3];
    {
        const long i = fresh_thread_index();
        if constexpr (UMODE == 3) {
            synth_x0((uint64_t)(a.index0 + i), x);
        } else {
#pragma unroll
            for (int c = 0; c < 13; ++c) x[c] = __ldg(a.x0 + (long)c * a.ld + i);
        }
        if constexpr (PERCOEF) {
            AeroCoef At;
            load_coef(a.K, a.p, a.ld, i, At);
            reinterpret_cast<AeroCoef*>(rollout_smem)[threadIdx.x] = At;
        }
    }
    if constexpr (PERCOEF) rollout_body<UMODE, RIGID>(a, x, u, reinterpret_cast<const volatile AeroCoef*>(rollout_smem)[threadIdx.x]);
    else rollout_body<UMODE, RIGID>(a, x, u, a.K.A);
}

template <int UMODE, bool RIGID, class AC>
__device__ __forceinline__ void rollout_body(const RolloutArgs& a, double (&x)[13], double (&u)[3], const AC& A) {
    const long i = fresh_thread_index();

    // Controls.  KITE_U_PER_STEP streams 24 B per state-step from HBM; the loads of step k + 1 are issued at the top of step k
    // (below) and have a whole step (~4 us) to land, so nothing else is needed: the L2 prefetch two steps ahead that round 1
    // used cost 1.4 % once the loads were a step ahead (78.88 -> 77.78 ms, profiles/r2w_sweep_nopf.log).
    // Loop state is kept small on purpose (the RHS leaves few spare registers): a 32-bit step counter and ONE running pointer
    // per stream instead of 64-bit index arithmetic per step.
    const int N = (int)a.N;                         // < 2^31 (checked by the host)
    const long ustep = 3 * a.ld;
    const double* up = (UMODE == 1) ? a.u + i : a.u;            // per-trajectory stream / shared log / held control
    auto load_u = [&](int k, double (&uu)[3]) {
        if constexpr (UMODE == 0) {
#pragma unroll
            for (int c = 0; c < 3; ++c) uu[c] = __ldg(a.u + (long)c * a.ld + i);
        } else if constexpr (UMODE == 1) {
#pragma unroll
            for (int c = 0; c < 3; ++c) uu[c] = __ldg(up + (long)c * a.ld);
        } else if constexpr (UMODE == 2) {
#pragma unroll
            for (int c = 0; c < 3; ++c) uu[c] = __ldg(up + c);
        } else {
            synth_control((uint64_t)(a.index0 + i), (uint64_t)k, uu);
        }
    };
    if constexpr (UMODE == 0) load_u(0, u);         // one control per trajectory, held for all steps
    double cost = 0.0;
    const double Qc[13] = {1e3, 1e2, 1e2, 1e2, 1e2, 1e2, 1e1, 1e1, 1e2, 1e2, 1e2, 1e2, 1e2};  // kite_identification_test.cpp:193
    const double* yp = a.y;
    int next_save = (int)a.save_every;
    // Controls of step k + 1 are loaded at the TOP of step k and fly behind its arithmetic (three register pairs).
    // Round 1 rejected this (61.5 % against 65.0 %) because the kernel spilled;
    // spill free (and still spill free at a 152-register cap) it is worth 1.5 %: 80.05 -> 78.85 ms (profiles/r2w_sweep_ureg.log).
    double un[3] = {0.0, 0.0, 0.0};
    if constexpr (UMODE == 1) { if (N > 0) load_u(0, un); up += ustep; }      // (N = 0 is legal: the control buffer may be empty)
    for (int k = 0; k < N; ++k) {
        if constexpr (UMODE == 1) {
#pragma unroll
            for (int c = 0; c < 3; ++c) u[c] = un[c];
            if (k + 1 < N) {
                load_u(k + 1, un);
                up += ustep;
            }
        } else if constexpr (UMODE == 2) {           // shared log: every thread reads the same three words (L1 broadcast hits)
            load_u(k, u);
            up += 3;
        } else if constexpr (UMODE == 3) {
            load_u(k, u);
        }
        rk4_step<RIGID>(a.K, A, x, u, a.rk);
        if (yp) {                                   // uniform branch: identification cost fused into the rollout
            double e = 0.0;
#pragma unroll
            for (int c = 0; c < 13; ++c) {
                const double dlt = __ldg(yp + c) - x[c];
                e = fma(Qc[c] * dlt, dlt, e);
            }
            cost += e;
            yp += 13;
        }
        if (a.traj && k + 1 == next_save) {         // rare: the slot and the thread index are recomputed, not kept alive
            double* const tp = a.traj + (long)(next_save / (int)a.save_every - 1) * 13 * a.ld + fresh_thread_index();
#pragma unroll
            for (int c = 0; c < 13; ++c) tp[(long)c * a.ld] = x[c];
            next_save += (int)a.save_every;
        }
    }
    const long io = fresh_thread_index();
#pragma unroll
    for (int c = 0; c < 13; ++c) a.xf[(long)c * a.ld + io] = x[c];
    if (a.y) a.cost[io] = cost * (1.0 / (double)a.N);
    if (a.status) a.status[io] = all_finite13(x) ? 0 : 1;
}

// Fill the synthetic workload buffers (x0 [13][ld], u [N][3][ld]).
struct SynthArgs { long B, ld, N, index0; double* x0; double* u; };
template <int DUMMY = 0>
__global__ void __launch_bounds__(256) k_synth_inputs(const __grid_constant__ SynthArgs a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.B) return;
    if (blockIdx.y == 0 && a.x0) {
        double x0[13];
        synth_x0((uint64_t)(a.index0 + i), x0);
#pragma unroll
        for (int c = 0; c < 13; ++c) a.x0[(long)c * a.ld + i] = x0[c];
    }
    if (a.u) {
        for (long k = blockIdx.y; k < a.N; k += gridDim.y) {
            double u[3];
            synth_control((uint64_t)(a.index0 + i), (uint64_t)k, u);
#pragma unroll
            for (int c = 0; c < 3; ++c) a.u[((long)k * 3 + c) * a.ld + i] = u[c];
        }
    }
}

// Parameter samples of the identification sweep (p [21][ld]) for global indices [index0, index0 + B).
struct SynthParamArgs { long B, ld, index0; double ref[21]; double* p; };
template <int DUMMY = 0>
__global__ void __launch_bounds__(256) k_synth_id_params(const __grid_constant__ SynthParamArgs a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.B) return;
#pragma unroll
    for (int c = 0; c < 21; ++c) a.p[(long)c * a.ld + i] = synth_id_param((uint64_t)(a.index0 + i), c, a.ref[c]);
}

// ================================================================================================
// RK4 step sensitivities: one persistent kernel, every warp independent (no CTA barrier anywhere), the stage Jacobians
// never leave the SM.  A warp owns groups of 32 units, claimed from a global counter.  Per group:
//   step 1 (lane = unit, 32 units): the primal RK4 step (RHS only, few registers).  xn leaves; the four stage states and
//                           the control are parked in the warp's private 16 KB line of global scratch (L2 resident).
//   then four rounds of 8 units each:
//   step 2 (lane = (unit, STAGE): 8 units x 4 stages): the four stage Jacobians of a unit are independent once the stage
//                           states are known, so ONE pass of the analytic Jacobian code evaluates all four stages of
//                           8 units.  That is what shrinks the Jacobians in flight from 32 units x 4 stages = 114 KB per
//                           warp (an L2 / HBM round trip in the earlier version: 3.7 GB of write-back per 1 M units) to
//                           8 units x 4 stages = 27 KB: they stay in the warp's SHARED-memory tile
//                           [stage][pass][slot][4 units], written conflict free straight from the Jacobian code.
//   phase B (8 consecutive lanes = unit, 4 units per pass, 2 passes): lane l of a unit owns tangent columns {l, l + 8} of
//                           [Phi | Gamma] and runs the recursion D_i = E + a_i h S_{i-1}, S_i = [Jx_i | Ju_i] D_i in
//                           registers (E = seed [I | 0; 0 | I]); stage 1 is a pure gather of two Jacobian columns through
//                           a shared offset table.  Jacobian entries are one-wavefront broadcast LDS.64 with immediate
//                           offsets.
//   output:                 [Phi | Gamma] of a round is staged as ONE [169][8 units] and ONE [39][8 units] box in pass 0's
//                           dead tiles (TMA 64-byte swizzle, per-lane offset table: conflict-free stores) and leaves by
//                           two TMA tensor stores of 64-byte rows; the tensor map clips the ragged tail.  A direct-store
//                           instantiation (TMA_OUT = false) serves layouts the TMA cannot address.
//   No TMA loads, no mbarriers, no ring: producer and consumer are the same warp, ordered by __syncwarp.
//   Multiple-shooting rollouts (N steps, the state of step k feeding step k + 1) run in the SAME launch: the work items
//   are (step, group) pairs claimed in step-major order, a warp that claims step k of a group waits (normally not at
//   all: the item was issued a whole wave earlier) until the group's step k - 1 has published its state.  One launch and
//   one tail for the whole horizon instead of one per step.
// ================================================================================================
struct SensArgs {
    alignas(64) CUtensorMap tmPhi;    // [N][169][B] rows of ld doubles, box [1][169][8 units]  (only read by the TMA-output kernels)
    alignas(64) CUtensorMap tmGam;    // [N][39][B], box [1][39][8 units]
    KiteConsts K;
    long B, ld;
    long N;                           // steps of the multiple-shooting rollout (1: a single step)
    RkTab rk;                         // RK4 tableau for h (host-computed)
    const double* x; const double* u; // x [13][ld] (state before step 0), u [N][3][ld]
    double* xn; double* Phi; double* Gamma;   // xn [N][13][ld] (state after each step), Phi [N][169][ld], Gamma [N][39][ld]
    double* Sw;     // scratch: [resident warp][4 stages][16 = x(13) | u(3)][32 units]
    unsigned long long* next_group;   // device counter (zeroed before the launch): work items are handed out dynamically
    int* done;      // [groups] steps finished per group (zeroed before the launch; only used when N > 1)
    int32_t* status;  // [ld] per-unit flags, OR over the steps (zeroed before the launch), or null
};


// ---- compact slots of the sensitivity tile ------------------------------------------------------------------
// Row-major over the structural non-zeros: Jx first, then Ju, then the tether-arm extras.  The 12 entries
// d q_dot / d w = {+-q/2} (kite_model.cuh, Qw) that repeat a value WITH ITS SIGN share a slot (12 -> 7): 106 slots
// without a tether arm (127 with), so that eight warps' tiles fit one SM's shared memory.
struct SensTab { int jx[13][13]; int ju[13][3]; int col[13][16]; };
constexpr int SENS_SLOTS_NOARM = JAC_SLOTS_NOARM - 5, SENS_SLOTS = JAC_SLOTS - 5;
// slots the state Jacobian spans (the EKF needs no Ju): the 99 zero-arm Jx slots come first; the tether-arm extras follow Ju
template <bool ARM> constexpr int JX_SENS_SLOTS = ARM ? SENS_SLOTS : SENS_SLOTS_NOARM - 7;
constexpr SensTab make_sens_tab() {
    SensTab t{};
    // value id of Qw[i][j]: +-1 = +-a0/2, +-2 = +-a1/2, +-3 = +-a2/2, 4 = s/2
    const int qw[4][3] = {{-1, -2, -3}, {4, -3, 2}, {3, 4, -1}, {-2, 1, 4}};
    int s = 0;
    for (int i = 0; i < 13; ++i)
        for (int j = 0; j < 13; ++j) {
            t.jx[i][j] = -1;
            if (!jx_nz(i, j, false)) continue;
            if (i >= 9 && j >= 3 && j < 6) {
                int found = -1;
                for (int i2 = 9; i2 <= i && found < 0; ++i2)
                    for (int j2 = 3; j2 < 6 && found < 0; ++j2)
                        if ((i2 < i || j2 < j) && qw[i2 - 9][j2 - 3] == qw[i - 9][j - 3]) found = t.jx[i2][j2];
                if (found >= 0) { t.jx[i][j] = found; continue; }
            }
            t.jx[i][j] = s++;
        }
    for (int i = 0; i < 13; ++i)
        for (int j = 0; j < 3; ++j) t.ju[i][j] = ju_nz(i, j) ? s++ : -1;
    for (int i = 0; i < 13; ++i)
        for (int j = 0; j < 13; ++j)
            if (jx_nz(i, j, true) && !jx_nz(i, j, false)) t.jx[i][j] = s++;
    for (int i = 0; i < 13; ++i)
        for (int c = 0; c < 16; ++c) t.col[i][c] = (c < 13) ? t.jx[i][c] : t.ju[i][c - 13];
    return t;
}
__device__ constexpr SensTab SENS_TAB = make_sens_tab();
static_assert(make_sens_tab().ju[5][2] == SENS_SLOTS_NOARM - 1, "sens slot numbering");
static_assert(make_sens_tab().jx[5][12] == SENS_SLOTS - 1, "sens slot numbering");
static_assert(make_sens_tab().jx[10][3] == make_sens_tab().jx[12][5] && make_sens_tab().jx[9][3] == make_sens_tab().jx[11][5],
              "shared quaternion-rate slots");

// upper bound of warps per CTA (one CTA per SM): 8 warps x 255 registers = the whole register file, 2 warps per scheduler
constexpr int SF_WARPS = 8;
constexpr size_t SF_SMEM_MAX = 227 * 1024;
constexpr long SF_SCRATCH_PER_WARP = 4L * 16 * 32;      // doubles: [stage][x(13) | u(3)][32 units]
template <bool ARM> struct SfCfg {
    static constexpr int NS = ARM ? SENS_SLOTS : SENS_SLOTS_NOARM;    // slots a stage Jacobian occupies
    // A stage tile holds the compact Jacobians of 4 units as two HALF tiles [slot][2 units] (units 0,1 | units 2,3), each
    // with one extra "zero" slot (the target of the gather's structural zeros; step 2 never writes there).  Bank layout
    // (16-byte groups, 8 per 128-byte wavefront): the half, stage and pass strides are == h, s, p (mod 8) groups with all
    // eight subset sums of {h, s, p} distinct, so that
    //   * the 16 lanes of a half-warp store of step 2 (2 stages x 2 passes x 2 halves x 2 units) fill one wavefront,
    //   * a phase-B broadcast load (4 units = 2 groups) is one wavefront, and
    //   * the stage-1 gather, where the 8 lanes of a unit read 8 (mostly consecutive) slots, sees 8 x 16 contiguous bytes per
    //     half-warp instead of 16 of every 32 bytes (the [slot][4 units] layout made that load 2-way conflicted by
    //     construction: 17.5 M excess wavefronts per 1 M units, profiles/r2a).
    static constexpr int HALF_S = (NS + 1) * 2 + (((NS + 1) * 2) % 4 == 2 ? 0 : 2);     // doubles; HALF_S / 2 odd
    static constexpr int TILE = 2 * HALF_S;                           // doubles per stage tile
    static constexpr int TILE_S = TILE + ((TILE % 16 == 4 || TILE % 16 == 12) ? 0 : ((4 - TILE % 16) + 16) % 16);   // == 4 or 12 (mod 16)
    static constexpr int PASS_S = 4 * TILE_S + ((8 - (4 * TILE_S) % 16) + 16) % 16;                                 // == 8 (mod 16)
    // per-warp stride: a multiple of 512 bytes, so that the TMA's 64-byte swizzle (a function of address bits 7..8) is
    // the same for every warp's output boxes
    static constexpr size_t SMEM_PER_WARP = (sizeof(double) * 2 * PASS_S + 511) / 512 * 512;
    static constexpr int FIT = (int)((SF_SMEM_MAX - 4096) / SMEM_PER_WARP);
    static constexpr int WARPS = SF_WARPS < FIT ? SF_WARPS : FIT;
    static constexpr size_t SMEM_TILES = SMEM_PER_WARP * WARPS;
    static constexpr size_t SMEM = SMEM_TILES + sizeof(unsigned) * 13 * 32;       // + gather table
    // TMA output: the [169][8] and [39][8] boxes of a ROUND (both passes) are staged in pass 0's tiles, all four dead once
    // pass 0 has consumed them (bytes from the warp's base, 128-byte aligned).  The [169] box runs over the zero slots of
    // pass 0's stage-1 tile, which are restored after the TMA has read the box.
    __host__ __device__ static constexpr size_t up128(size_t v) { return (v + 127) / 128 * 128; }
    static constexpr size_t BOX_PHI = 0;
    static constexpr size_t BOX_GAM = (sizeof(double) * 169 * 8 + 127) / 128 * 128;
    // element (slot s, unit w of the pass) of a stage tile, in doubles from the tile's base
    __host__ __device__ static constexpr int at(int s, int w) { return (w >> 1) * HALF_S + s * 2 + (w & 1); }
};
constexpr bool sf_banks_ok(int half, int tile, int pass) {     // all 8 subset sums of the three strides distinct mod 8 (16-byte groups)
    const int h = (half / 2) % 8, t = (tile / 2) % 8, q = (pass / 2) % 8;
    bool seen[8] = {};
    for (int m = 0; m < 8; ++m) {
        const int v = ((m & 1 ? h : 0) + (m & 2 ? t : 0) + (m & 4 ? q : 0)) % 8;
        if (seen[v]) return false;
        seen[v] = true;
    }
    return true;
}
static_assert(SfCfg<false>::SMEM_PER_WARP % 128 == 0 && SfCfg<true>::SMEM_PER_WARP % 128 == 0, "TMA staging alignment");
static_assert(SfCfg<false>::BOX_GAM + 39 * 64 <= sizeof(double) * (SfCfg<false>::PASS_S - 8) &&
              SfCfg<true>::BOX_GAM + 39 * 64 <= sizeof(double) * (SfCfg<true>::PASS_S - 8), "staging boxes fit pass 0's tiles");
static_assert(sf_banks_ok(SfCfg<false>::HALF_S, SfCfg<false>::TILE_S, SfCfg<false>::PASS_S) &&
              sf_banks_ok(SfCfg<true>::HALF_S, SfCfg<true>::TILE_S, SfCfg<true>::PASS_S), "conflict-free tile strides");
static_assert(SfCfg<false>::HALF_S % 2 == 0 && SfCfg<false>::TILE_S % 2 == 0 && SfCfg<false>::WARPS == 8, "tile geometry (no arm): 8 warps per SM");

struct StageSink {      // the warp's tile: slot s of this lane's (unit, stage) at base[2 s], base = &tile[pass][stage][half][0][unit & 1]
    double* base;
    __device__ __forceinline__ void jx(int i, int j, double v) const { base[SENS_TAB.jx[i][j] * 2] = v; }
    __device__ __forceinline__ void ju(int i, int j, double v) const { base[SENS_TAB.ju[i][j] * 2] = v; }
    __device__ __forceinline__ void aero(double, double, double) const {}
};

// y = J v for two vectors at once: J = [Jx | Ju] (NC = 16 input columns) or Jx (NC = 13) in compact slots, read from the
// shared tile column of one unit (tile rows [slot][STRIDE units]).
// The control columns 13..15 update y1 only.  The one caller with NC = 16 (phase B of k_sens_fused) passes the control
// part of its seed there, which is 0 in v0 (the lane's first tangent column c0 < 8 is a column of Phi) and e_(c1 - 13) in
// v1.  The zero products must be skipped, not just saved: fma(jv, 0, y) is not bitwise y (-0 + 0 gives +0, and an
// infinite or NaN entry gives NaN).
// Column-major traversal: the (up to 13) entries J[i][j] of input row j update 26 independent chains, so consecutive DFMAs
// never depend on each other.  Operand order matters: a DFMA with three distinct vector-register operands issues every 3
// cycles, with two every 2 (profiles/r2j_dfma_operands.log).  The two FMAs of an entry share jv; alternating which vector
// goes first makes the first FMA of the NEXT entry share v[.][j] with the one before it, so that every FMA finds one
// operand in the reuse cache: ... (v0, jv1) (v1, jv1) (v1, jv2) (v0, jv2) (v0, jv3) ...
template <bool ARM, bool RIGID, int STRIDE, int NC>
__device__ __forceinline__ void jac_times2(const double* __restrict__ T, const double (&v0)[NC], const double (&v1)[NC],
                                           double (&y0)[13], double (&y1)[13]) {
    static_assert(NC == 13 || NC == 16, "Jx or [Jx | Ju]");
#pragma unroll
    for (int i = 0; i < 13; ++i) { y0[i] = 0.0; y1[i] = 0.0; }
    int flip = 0;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
#pragma unroll
        for (int i = (RIGID ? 6 : 0); i < 13; ++i) {
            if ((j < 13) ? jx_nz(i, j, ARM) : (!RIGID && ju_nz(i, j - 13))) {
                const double jv = T[SENS_TAB.col[i][j] * STRIDE];     // broadcast LDS.64, immediate offset
                if (j >= 13) {
                    y1[i] = fma(jv, v1[j], y1[i]);
                } else if (flip) {
                    y1[i] = fma(jv, v1[j], y1[i]);
                    y0[i] = fma(jv, v0[j], y0[i]);
                } else {
                    y0[i] = fma(jv, v0[j], y0[i]);
                    y1[i] = fma(jv, v1[j], y1[i]);
                }
                flip ^= 1;
            }
        }
    }
}

template <bool ARM, bool RIGID, bool TMA_OUT>
__global__ void __launch_bounds__(SfCfg<ARM>::WARPS * 32, 1) k_sens_fused(const __grid_constant__ SensArgs a) {
    using C = SfCfg<ARM>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* const tile = reinterpret_cast<double*>(smem_raw + (size_t)warp * C::SMEM_PER_WARP);
    double* const Sw = a.Sw + ((long)blockIdx.x * C::WARPS + warp) * SF_SCRATCH_PER_WARP;
    const long ngroups = (a.B + 31) / 32;
    // phase B: 8 consecutive lanes = one unit, so that the 4 addresses of a Jacobian-entry load are each shared by a
    // contiguous lane octet: ONE shared-memory wavefront per LDS.64 (with the unit in the low lane bits it takes two)
    const int lu = lane >> 3, l = lane & 7;
    const int c0 = l, c1 = l + 8;                  // tangent columns of this lane in phase B

    // zero rows of the stage-1 tiles (targets of the gather's structural zeros); step 2 never writes there
    if (lane < 8) tile[(lane >> 2) * C::PASS_S + C::at(C::NS, lane & 3)] = 0.0;
    // gather table: byte offsets (within a tile, lane's unit included) of the entries of Jacobian columns c0 (low half)
    // and c1 (high half) of this lane, one word per row; structural zeros point at the zero row.  [13][32 lanes].
    unsigned* const goff = reinterpret_cast<unsigned*>(smem_raw + C::SMEM_TILES) + lane;
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < 13; ++i) {
            int s0 = C::NS, s1 = C::NS;
#pragma unroll
            for (int c = 0; c < 16; ++c) {
                const int sl = SENS_TAB.col[i][c];
                const bool ok = sl >= 0 && sl < C::NS && !(RIGID && (i < 6 || c >= 13));
                if (ok && c == c0) s0 = sl;
                if (ok && c == c1) s1 = sl;
            }
            goff[i * 32] = (unsigned)(C::at(s0, lu) * 8) | ((unsigned)(C::at(s1, lu) * 8) << 16);
        }
    }
    // staging (TMA output): row i of this lane's two output columns goes to the [169][8] / [39][8] boxes of the round, which
    // use the TMA's 64-byte swizzle (16-byte chunk index ^= address bits 7..8), so the eight rows of a half-warp store land in
    // eight different 16-byte bank groups: conflict free instead of 4-way at the dense 64-byte row pitch.  The swizzled
    // offset is COMPUTED (box row R = i * stride + column: chunk bits = (8 R + 16 (box address >> 7)) & 0x30, three integer
    // instructions on the idle ALU pipe); round 2 looked it up in a per-lane table in shared memory, and the stores waited
    // on those lookups for 10 % of the kernel's time (profiles/r2t ncu source page: short_scoreboard on the LOP3 after the LDS).
    const unsigned wb_abs = (unsigned)__cvta_generic_to_shared(smem_raw) + (unsigned)(warp * C::SMEM_PER_WARP);
    const bool gam1 = c1 >= 13;                     // lanes 5..7: the second column is a column of Gamma
    const unsigned col1 = gam1 ? c1 - 13 : c1;
    const unsigned box1 = gam1 ? (unsigned)C::BOX_GAM : (unsigned)C::BOX_PHI;
    const unsigned sA0 = (unsigned)C::BOX_PHI + (unsigned)c0 * 64u, sA1 = box1 + col1 * 64u;             // offset of row 0 of the column
    const unsigned sE0 = 8u * c0 + (((wb_abs + (unsigned)C::BOX_PHI) >> 7) << 4), sE1 = 8u * col1 + (((wb_abs + box1) >> 7) << 4);
    const unsigned sR1 = gam1 ? 3u : 13u;           // box rows per matrix row
    __syncthreads();
    const double h6 = a.rk.h6, hh = a.rk.an[0], h = a.rk.an[2];
    // Groups are claimed from a global counter instead of a fixed stride: warps that share a scheduler run at different
    // speeds, and a static split would leave the fast ones idle at the end.  The next group's input lines are pulled
    // into L2 while this one is computed (register free).
    // work item t = step * ngroups + group, claimed from a global counter in step-major order
    const long nitems = ngroups * a.N;
    auto claim_item = [&]() -> long {
        unsigned long long t = 0;
        if (lane == 0) t = atomicAdd(a.next_group, 1ULL);
        t = __shfl_sync(0xffffffffu, t, 0);
        if ((long)t < nitems) {
            const long kk = (long)t / ngroups, first = ((long)t - kk * ngroups) * 32;
            const int row = lane >> 1;                                  // 13 rows of x, 3 of u, 2 x 128 B each
            // step 0 reads x, later steps read the state their predecessor has just written (in L2 anyway)
            const double* p = (row < 13 ? (kk == 0 ? a.x + (long)row * a.ld : nullptr)
                                        : a.u + (kk * 3 + (row - 13)) * a.ld);
            if (p && first + (lane & 1) * 16 < a.B) asm volatile("prefetch.global.L2 [%0];" :: "l"(p + first + (lane & 1) * 16));
        }
        return (long)t;
    };
    long item = claim_item();
    __syncwarp();

    while (item < nitems) {
        const long item_next = claim_item();
        const long ks = item / ngroups, g = item - ks * ngroups;        // step, group
        const double* const xin = (ks == 0) ? a.x : a.xn + (ks - 1) * 13 * a.ld;
        const double* const uin = a.u + ks * 3 * a.ld;
        double* const xout = a.xn + ks * 13 * a.ld;
        if (ks > 0) {                                                   // the group's previous step has published its state
            if (lane == 0) {
                int v;
                do { asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(a.done + g) : "memory"); } while (v < (int)ks);
            }
            __syncwarp();
        }
        // ---------------- step 1: lane = unit, primal RK4 step -------------------------------------------------
        {
            const long unit = g * 32 + lane;
            const long ui = unit < a.B ? unit : a.B - 1;         // ragged tail: recompute the last unit, store nothing
            double x[13], u[3], k[13], xt[13], acc[13];
#pragma unroll
            for (int c = 0; c < 13; ++c) { x[c] = __ldcg(xin + (long)c * a.ld + ui); xt[c] = x[c]; }
#pragma unroll
            for (int c = 0; c < 3; ++c) u[c] = RIGID ? 0.0 : __ldcs(uin + (long)c * a.ld + ui);
#pragma unroll
            for (int c = 0; c < 3; ++c) st_scratch(Sw + (13 + c) * 32 + lane, u[c]);     // (after ALL loads: may-alias stores serialise them)
            // (not rk4_step: its peeled first stage puts a second copy of the RHS into this kernel's instruction stream,
            // which made the kernel 1-4 % slower at 1 M units on a B200, 1000 W)
            NoSink ns;
#pragma unroll 1
            for (int st = 0; st < 4; ++st) {
#pragma unroll
                for (int c = 0; c < 13; ++c) st_scratch(Sw + (st * 16 + c) * 32 + lane, xt[c]);
                model_eval<RIGID, false>(a.K, a.K.A, xt, u, k, ns);
                const double wgt = (st == 0 || st == 3) ? 1.0 : 2.0;
                const double an = (st == 2) ? h : hh;
#pragma unroll
                for (int c = 0; c < 13; ++c) {
                    acc[c] = (st == 0) ? k[c] : fma(wgt, k[c], acc[c]);
                    xt[c] = fma(an, k[c], x[c]);
                }
            }
            if (unit < a.B) {
#pragma unroll
                for (int c = 0; c < 13; ++c) { acc[c] = fma(h6, acc[c], x[c]); __stcg(xout + (long)c * a.ld + unit, acc[c]); }
                if (a.status) {                         // (warp-uniform) flags of this step, OR-ed into the unit's word
                    const int fl = singularity_flags<RIGID>(x) | (all_finite13(acc) ? 0 : FLAG_NONFINITE);
                    if (fl) atomicOr(a.status + unit, fl);
                }
            }
            if (a.N > 1) {                              // publish: step ks of this group is done (release after every lane's stores)
                __threadfence();
                __syncwarp();
                if (lane == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" :: "l"(a.done + g), "r"((int)ks + 1) : "memory");
            }
        }
        __syncwarp();                                   // the stage states of all 32 units are visible to the warp

#pragma unroll 1
        for (int r = 0; r < 4; ++r) {
            // ---------------- step 2: lane = (unit, stage), four stage Jacobians of 8 units -> shared tile ----------
            {
                const int u8 = lane & 7, s = lane >> 3;
                double xt[13], u[3], k[13];
#pragma unroll
                for (int c = 0; c < 13; ++c) xt[c] = ld_scratch(Sw + (s * 16 + c) * 32 + r * 8 + u8);
#pragma unroll
                for (int c = 0; c < 3; ++c) u[c] = ld_scratch(Sw + (13 + c) * 32 + r * 8 + u8);
                StageSink sink{tile + (u8 >> 2) * C::PASS_S + s * C::TILE_S + C::at(0, u8 & 3)};
                if (TMA_OUT) {                          // the previous round's output boxes have left the tiles
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    __syncwarp();
                    if (lane < 4) tile[C::at(C::NS, lane)] = 0.0;      // pass 0's zero slots lay under the [169][8] box
                }
                model_eval<RIGID, true>(a.K, a.K.A, xt, u, k, sink);
            }
            __syncwarp();                               // the tile is complete and visible to all lanes
            // ---------------- phase B: 8 lanes = unit, 4 units per pass ---------------------------------------------
            double D[2][16], N0[13], N1[13], A0[13], A1[13];   // D[.][13..15]: the control part of the seed (constant)
#pragma unroll
            for (int m = 13; m < 16; ++m) { D[0][m] = (m == c0) ? 1.0 : 0.0; D[1][m] = (m == c1) ? 1.0 : 0.0; }
#pragma unroll 1
            for (int p = 0; p < 2; ++p) {
                const long unit = g * 32 + r * 8 + p * 4 + lu;
                // ---- stage 1: D = E, so S_1 = [Jx | Ju] E is a gather of two Jacobian columns (no FMAs)
                {
                    const char* const T = reinterpret_cast<const char*>(tile + p * C::PASS_S);
#pragma unroll
                    for (int i = 0; i < 13; ++i) {
                        const unsigned o = goff[i * 32];
                        N0[i] = *reinterpret_cast<const double*>(T + (o & 0xffffu));
                        N1[i] = *reinterpret_cast<const double*>(T + (o >> 16));
                    }
#pragma unroll
                    for (int i = 0; i < 13; ++i) {
                        A0[i] = N0[i]; A1[i] = N1[i];
                        D[0][i] = fma(hh, N0[i], (i == c0) ? 1.0 : 0.0);
                        D[1][i] = fma(hh, N1[i], (i == c1) ? 1.0 : 0.0);
                    }
                }
                // ---- stages 2..4: S_i = [Jx_i | Ju_i] D_i, one copy of the code (rolled: instruction-cache footprint)
#pragma unroll 1
                for (int st = 1; st < 4; ++st) {
                    jac_times2<ARM, RIGID, 2>(tile + p * C::PASS_S + st * C::TILE_S + C::at(0, lu), D[0], D[1], N0, N1);
                    const double wgt = (st == 3) ? 1.0 : 2.0;
                    const double an = (st == 2) ? h : hh;
#pragma unroll
                    for (int i = 0; i < 13; ++i) {
                        A0[i] = fma(wgt, N0[i], A0[i]);
                        A1[i] = fma(wgt, N1[i], A1[i]);
                    }
                    if (st < 3) {                                   // (warp-uniform) the last stage feeds no further one
#pragma unroll
                        for (int i = 0; i < 13; ++i) {
                            D[0][i] = fma(an, N0[i], (i == c0) ? 1.0 : 0.0);
                            D[1][i] = fma(an, N1[i], (i == c1) ? 1.0 : 0.0);
                        }
                    }
                }
                if (TMA_OUT) {
                    // [Phi | Gamma] = E + h/6 A staged in the [169][8] / [39][8] boxes of the round (units 4 p .. 4 p + 3 of
                    // every row; swizzled offsets from the staging table) and, after the second pass, written by two
                    // TMA tensor stores of 64-byte rows: the LSU sees 26 conflict-free shared stores per pass instead of
                    // 26 eight-sector global stores with 64-bit address arithmetic; units >= B are clipped by the
                    // tensor map
                    unsigned char* const wb = smem_raw + (size_t)warp * C::SMEM_PER_WARP;
                    unsigned char* const bphi = wb + C::BOX_PHI;
                    unsigned char* const bgam = wb + C::BOX_GAM;
                    if (p == 0) __syncwarp();           // every lane is done with pass 0's tiles (the box lies over them)
                    const unsigned fo = (unsigned)lu * 8u + (p ? 32u : 0u);     // this lane's unit within the 64-byte row
#pragma unroll
                    for (int i = 0; i < 13; ++i) {
                        const unsigned o0 = sA0 + (unsigned)i * 832u + (((sE0 + (unsigned)i * 104u) & 0x30u) ^ fo);
                        const unsigned o1 = sA1 + (unsigned)i * (sR1 * 64u) + (((sE1 + (unsigned)i * (sR1 * 8u)) & 0x30u) ^ fo);
                        *reinterpret_cast<double*>(wb + o0) = fma(h6, A0[i], (i == c0) ? 1.0 : 0.0);
                        *reinterpret_cast<double*>(wb + o1) = fma(h6, A1[i], (i == c1) ? 1.0 : 0.0);
                    }
                    if (p == 1) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            const int ux = (int)(g * 32 + r * 8);
                            asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                                         :: "l"(reinterpret_cast<unsigned long long>(&a.tmPhi)), "r"(ux), "r"(0), "r"((int)ks),
                                            "r"((unsigned)__cvta_generic_to_shared(bphi)) : "memory");
                            asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                                         :: "l"(reinterpret_cast<unsigned long long>(&a.tmGam)), "r"(ux), "r"(0), "r"((int)ks),
                                            "r"((unsigned)__cvta_generic_to_shared(bgam)) : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                    }
                } else if (unit < a.B) {
                    // [Phi | Gamma] = E + h/6 A: row i of this lane's two columns; a warp store covers 8 rows x 4 units (32 B)
                    double* const o0 = (c0 < 13) ? a.Phi + (ks * 169 + c0) * a.ld + unit : a.Gamma + (ks * 39 + c0 - 13) * a.ld + unit;
                    double* const o1 = (c1 < 13) ? a.Phi + (ks * 169 + c1) * a.ld + unit : a.Gamma + (ks * 39 + c1 - 13) * a.ld + unit;
                    const long r0 = (c0 < 13 ? 13 : 3) * a.ld, r1 = (c1 < 13 ? 13 : 3) * a.ld;
#pragma unroll
                    for (int i = 0; i < 13; ++i) {
                        __stcs(o0 + i * r0, fma(h6, A0[i], (i == c0) ? 1.0 : 0.0));
                        __stcs(o1 + i * r1, fma(h6, A1[i], (i == c1) ? 1.0 : 0.0));
                    }
                }
            }
            __syncwarp();                               // every lane is done reading the tile before the next round
        }
        item = item_next;
    }
    if (TMA_OUT && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ================================================================================================
// EKF predict (kiteEKF.cpp:75-98): xn = RK4(x,u,dt); A = I + dt Jx(x,u) at the PRE-step state; Pn = A P A^T + W.
// One persistent kernel, every warp independent; the Jacobian never leaves the SM.
//   phase A (ekf_filter_step, lane = filter, 32 filters per group): the RK4 step -> xn; the Jacobian at the pre-step state
//            -> the warp's shared tile Jt[pass = lane / 4][slot][lane % 4].
//   phase B (8 lanes = filter, 4 filters per pass): lane l owns rows {2l, 2l+1} of P (lanes 0..6; 13 rows):
//            Q = P A^T  (row r: q = p + dt J p), transposed through a small shared buffer, then Pn = A Q + W
//            (column c: q + dt J q + W[:, c]).  Jacobian entries are conflict-free broadcast LDS with immediate offsets.
// ================================================================================================
struct EkfArgs {
    KiteConsts K;
    long B, ld;
    double dt;
    RkTab rk;                // RK4 tableau for dt (host-computed)
    const double* x; const double* u; const double* P;
    double* xn; double* Pn;
    const double* W;         // device [169]
    unsigned long long* next_group;   // device counter (zeroed before the launch): groups are handed out dynamically
    int32_t* status;         // [ld] per-filter flags or null
};
template <bool ARM> struct EfCfg {
    // state-Jacobian slots, numbered as in the sensitivity kernel (repeated +-q/2 entries share a slot): 99 without a
    // tether arm, so that SEVEN warps' tiles and transpose buffers fit one SM
    static constexpr int NS = JX_SENS_SLOTS<ARM>;
    // pass stride == 4 (mod 16) doubles: the 8 four-lane groups of a phase-A store land in distinct bank octets
    static constexpr int PS = NS * 4 + ((NS * 4) % 16 == 12 ? 8 : ((NS * 4) % 16 == 0 ? 4 : (20 - (NS * 4) % 16) % 16));
    static constexpr int QR = 15;                                     // transpose buffer row stride (odd: conflict-free rows)
    static constexpr int QS = 4 * 13 * QR;                            // transpose buffer [4 filters][13][QR]
    static constexpr int PER_WARP = 8 * PS + QS;                      // doubles
    static constexpr int WARPS = (int)((SF_SMEM_MAX - 176 * sizeof(double)) / (sizeof(double) * PER_WARP)) < 8
                                     ? (int)((SF_SMEM_MAX - 176 * sizeof(double)) / (sizeof(double) * PER_WARP)) : 8;
    static constexpr size_t SMEM = sizeof(double) * (WARPS * PER_WARP + 176);      // + W (13 x 13, one copy per CTA)
};
static_assert(make_sens_tab().jx[12][12] == SENS_SLOTS_NOARM - 8, "state-Jacobian slots come first");
static_assert(EfCfg<false>::PS % 16 == 4 && EfCfg<true>::PS % 16 == 4, "bank-conflict-free pass stride");

struct SmemSink {       // compact slots of this lane's filter in the warp's shared tile
    double* base;       // &Jt[lane / 4][0][lane % 4]
    __device__ __forceinline__ void jx(int i, int j, double v) const { base[SENS_TAB.jx[i][j] * 4] = v; }
    __device__ __forceinline__ void ju(int, int, double) const {}     // the EKF uses the state Jacobian only
    __device__ __forceinline__ void aero(double, double, double) const {}
};

// W (13 x 13 row-major) -> shared memory, one copy per CTA (the caller synchronises the block).  The kernel passes
// threadIdx.x: read there, its range comes from the kernel's launch bounds, and with at most 169 threads the compiler
// drops the loop's entry test.
__device__ __forceinline__ void ekf_stage_W(double* Ws, const double* W, int tid) {
    for (int t = tid; t < 169; t += blockDim.x) Ws[t] = __ldg(W + t);
}

// groups are claimed from a global counter: the warps of a CTA share 4 schedulers and do not all run at the same speed
__device__ __forceinline__ long ekf_claim_group(unsigned long long* next_group, int lane) {
    unsigned long long g = 0;
    if (lane == 0) g = atomicAdd(next_group, 1ULL);
    return (long)__shfl_sync(0xffffffffu, g, 0);
}

// The filter step of both predict kernels, one filter `unit` per lane: the RK4 step's first stage evaluates f and d f/d x
// at the pre-step state in ONE pass, giving the Jacobian (into `sink`) AND k1 (the reference evaluates both at the same
// point, kiteEKF.cpp:80,93); `after_k1()` runs next, then three more RHS evaluations finish the step -> xn and the status word.
// Ragged tail: lanes past B recompute the last filter and store nothing.
template <bool RIGID, class Sink, class AfterK1>
__device__ __forceinline__ void ekf_filter_step(const EkfArgs& a, long unit, Sink sink, AfterK1&& after_k1) {
    const long ui = unit < a.B ? unit : a.B - 1;
    double x[13], u[3];
#pragma unroll
    for (int c = 0; c < 13; ++c) x[c] = __ldcs(a.x + (long)c * a.ld + ui);
#pragma unroll
    for (int c = 0; c < 3; ++c) u[c] = a.u ? __ldcs(a.u + (long)c * a.ld + ui) : 0.0;
    const int pre = a.status ? singularity_flags<RIGID>(x) : 0;
    rk4_step<RIGID, true>(a.K, a.K.A, x, u, a.rk, sink, [&](int st, const double (&)[13]) { if (st == 1) after_k1(); });
    if (unit < a.B) {
#pragma unroll
        for (int c = 0; c < 13; ++c) __stcs(a.xn + (long)c * a.ld + unit, x[c]);
        if (a.status) a.status[unit] = pre | (all_finite13(x) ? 0 : FLAG_NONFINITE);
    }
}

template <bool ARM, bool RIGID>
__global__ void __launch_bounds__(EfCfg<ARM>::WARPS * 32, 1) k_ekf_predict(const __grid_constant__ EkfArgs a) {
    using C = EfCfg<ARM>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* const Jt = reinterpret_cast<double*>(smem_raw) + (size_t)warp * C::PER_WARP;
    double* const Qt = Jt + 8 * C::PS;
    double* const Ws = reinterpret_cast<double*>(smem_raw) + (size_t)C::WARPS * C::PER_WARP;   // W (13 x 13 row-major), one copy per CTA
    const long ngroups = (a.B + 31) / 32;
    const int lu = lane >> 3, l = lane & 7;
    const int r0 = 2 * l, r1 = 2 * l + 1;          // rows of P (phase B, first product) = columns of Pn (second product)
    const bool v0 = r0 < 13, v1 = r1 < 13;
    ekf_stage_W(Ws, a.W, threadIdx.x);
    __syncthreads();
    // rows r0, r1 of P for the 4 filters of a pass (registers; issued one pass ahead so the loads fly behind the FMAs)
    auto load_rows = [&](long g, int p, double (&q0)[13], double (&q1)[13]) {
        const long unit = g * 32 + p * 4 + lu;
        const long ui = unit < a.B ? unit : a.B - 1;
#pragma unroll
        for (int k = 0; k < 13; ++k) {
            q0[k] = v0 ? __ldcs(a.P + (long)(r0 * 13 + k) * a.ld + ui) : 0.0;
            q1[k] = v1 ? __ldcs(a.P + (long)(r1 * 13 + k) * a.ld + ui) : 0.0;
        }
    };

    for (long g = ekf_claim_group(a.next_group, lane); g < ngroups; g = ekf_claim_group(a.next_group, lane)) {
        double pn0[13], pn1[13];
        // ---------------- phase A: lane = filter ------------------------------------------------------------
        ekf_filter_step<RIGID>(a, g * 32 + lane, SmemSink{Jt + (lane >> 2) * C::PS + (lane & 3)}, [] {});
        __syncwarp();
        // (the first pass's rows are fetched here, not behind phase A: 52 more live registers across the Jacobian code spilled)
        load_rows(g, 0, pn0, pn1);
        // ---------------- phase B: 8 lanes = filter, 4 filters per pass -------------------------------------
#pragma unroll 1
        for (int p = 0; p < 8; ++p) {
            const long unit = g * 32 + p * 4 + lu;
            const double* __restrict__ T = Jt + p * C::PS + lu;
            double* const Q = Qt + lu * (13 * C::QR);
            double p0[13], p1[13], n0[13], n1[13];
#pragma unroll
            for (int k = 0; k < 13; ++k) { p0[k] = pn0[k]; p1[k] = pn1[k]; }
            if (p < 7) load_rows(g, p + 1, pn0, pn1);
            jac_times2<ARM, RIGID, 4>(T, p0, p1, n0, n1);
            __syncwarp();                               // the previous pass is done reading the transpose buffer
#pragma unroll
            for (int k = 0; k < 13; ++k) {              // rows r0, r1 of Q = P A^T
                if (v0) Q[r0 * C::QR + k] = fma(a.dt, n0[k], p0[k]);
                if (v1) Q[r1 * C::QR + k] = fma(a.dt, n1[k], p1[k]);
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 13; ++k) {              // columns r0, r1 of Q
                p0[k] = v0 ? Q[k * C::QR + r0] : 0.0;
                p1[k] = v1 ? Q[k * C::QR + r1] : 0.0;
            }
            jac_times2<ARM, RIGID, 4>(T, p0, p1, n0, n1);
            if (unit < a.B) {
#pragma unroll
                for (int i = 0; i < 13; ++i) {          // columns r0, r1 of Pn = A Q + W
                    if (v0) __stcs(a.Pn + (long)(i * 13 + r0) * a.ld + unit, fma(a.dt, n0[i], p0[i]) + Ws[i * 13 + r0]);
                    if (v1) __stcs(a.Pn + (long)(i * 13 + r1) * a.ld + unit, fma(a.dt, n1[i], p1[i]) + Ws[i * 13 + r1]);
                }
            }
        }
        __syncwarp();                                   // phase B is done with the Jacobian tile before the next group
    }
}

// ================================================================================================
// EKF predict, round-based with TMA boxes (the product path when the covariance layout is TMA-addressable: 16-byte
// aligned base and pitch, even B).  Same arithmetic as k_ekf_predict; what changes is how P moves and where the Jacobian
// waits.  A warp owns groups of 32 filters:
//   step 1 (ekf_filter_step, lane = filter, 32 filters): the RK4 step -> xn.  The 99 Jacobian entries of a filter go to the
//       warp's line of an L2-resident scratch laid out [round][slot][8 filters]; the filters of round 0 also write them
//       straight into the shared tile.  Once k1 is known, the bulk copy of round 1's tile is issued.  (Round 1 evaluated
//       the Jacobian once per round with 4 replica lanes per filter: 30 % of the kernel's time for 3 redundant evaluations,
//       profiles/r2a ncu source page; a 32-filter tile in shared memory would leave room for 4 warps per SM.)
//   four rounds of 8 filters:
//     the round's [99][8] Jacobian tile arrives by ONE 1-D bulk copy (cp.async.bulk, mbarrier) issued a round ahead into the
//       other of two tile buffers; the [169][8 filters] box of P (64-byte rows, 64-byte swizzle) arrives by ONE TMA tensor
//       load issued half a round ahead; phase B (8 lanes = filter, 2 passes of 4 filters) reads the rows of P from the box,
//       writes Q = P A^T back IN PLACE (a lane only overwrites what it read), reads the columns of Q from the same box (the
//       box is the transpose buffer), writes the columns of Pn = A Q + W in place, and the box leaves by ONE TMA tensor store.
//   The LSU sees conflict-free shared accesses through per-lane offset tables instead of 52 eight-sector global accesses
//   with 64-bit address arithmetic per pass (profiles/r1zb_ekf_before_ncu_summary.txt: LSU data pipe 63 % busy).
// ================================================================================================
struct EkfTmaArgs {
    alignas(64) CUtensorMap tmP;      // [1][169][B] rows of ld doubles, box [1][169][8 filters], 64-byte swizzle
    alignas(64) CUtensorMap tmPn;
    EkfArgs e;
    double* Jw;                       // scratch: [resident warp][4 rounds][NS slots][8 filters]
};
template <bool ARM> struct EtCfg {
    static constexpr int NS = JX_SENS_SLOTS<ARM>;
    static constexpr int TILE_D = NS * 8;                                         // doubles per round tile [slot][8 filters]
    static constexpr unsigned TILE_BYTES = TILE_D * 8;
    static constexpr size_t BOX = (169 * 64 + 511) / 512 * 512;                   // 10816 -> 11264: both boxes see the same swizzle
    static constexpr unsigned BOX_BYTES = 169 * 64;
    static constexpr size_t PER_WARP = (2 * BOX + 2 * TILE_BYTES + 511) / 512 * 512;
    static constexpr int FIT = (int)((SF_SMEM_MAX - 8192) / PER_WARP);
    static constexpr int WARPS = FIT < 8 ? FIT : 8;
    static constexpr size_t SMEM_WARPS = PER_WARP * WARPS;
    static constexpr size_t OFF_W = SMEM_WARPS;                                   // W (13 x 13), one copy per CTA
    static constexpr size_t OFF_BAR = OFF_W + sizeof(double) * 176;               // four mbarriers per warp (2 boxes, 2 tiles)
    static constexpr size_t SMEM = OFF_BAR + sizeof(unsigned long long) * 4 * WARPS;
    static constexpr long SCRATCH_PER_WARP = 4L * TILE_D;                         // doubles of L2 scratch per resident warp
    static constexpr long SCRATCH_PER_CTA = WARPS * SCRATCH_PER_WARP;
};
static_assert(EtCfg<false>::SMEM <= SF_SMEM_MAX && EtCfg<true>::SMEM <= SF_SMEM_MAX, "shared memory");
static_assert(EtCfg<false>::TILE_BYTES % 16 == 0 && EtCfg<true>::TILE_BYTES % 16 == 0, "bulk-copy granularity");
// doubles of Jacobian scratch per SM that ekf_predict_scratch_bytes() allocates: one CTA of either configuration
constexpr long ET_SCRATCH_PER_CTA_MAX = EtCfg<true>::SCRATCH_PER_CTA > EtCfg<false>::SCRATCH_PER_CTA ? EtCfg<true>::SCRATCH_PER_CTA : EtCfg<false>::SCRATCH_PER_CTA;

struct EkfTileSink {    // state-Jacobian slot s of this lane's filter: scratch line [round][s][8] (+ the shared tile for round 0)
    double* g;          // &Jw[lane / 8][0][lane % 8]
    double* sh;         // &tile0[0][lane] for lanes 0..7, null otherwise
    __device__ __forceinline__ void jx(int i, int j, double v) const {
        st_scratch(g + SENS_TAB.jx[i][j] * 8, v);
        if (sh) sh[SENS_TAB.jx[i][j] * 8] = v;
    }
    __device__ __forceinline__ void ju(int, int, double) const {}
    __device__ __forceinline__ void aero(double, double, double) const {}
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra WAIT_%=;\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

template <bool ARM, bool RIGID>
__global__ void __launch_bounds__(EtCfg<ARM>::WARPS * 32, 1) k_ekf_predict_tma(const __grid_constant__ EkfTmaArgs ta) {
    using C = EtCfg<ARM>;
    const EkfArgs& a = ta.e;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* const wb = smem_raw + (size_t)warp * C::PER_WARP;              // [box 0][box 1][tile 0][tile 1]
    double* const Jt = reinterpret_cast<double*>(wb + 2 * C::BOX);
    double* const Ws = reinterpret_cast<double*>(smem_raw + C::OFF_W);
    unsigned long long* const bars = reinterpret_cast<unsigned long long*>(smem_raw + C::OFF_BAR) + warp * 4;   // [box 0, box 1, tile 0, tile 1]
    static_assert(C::WARPS * C::SCRATCH_PER_WARP <= ET_SCRATCH_PER_CTA_MAX, "the warps' scratch lines fit the host's allocation");
    double* const Jw = ta.Jw + ((long)blockIdx.x * C::WARPS + warp) * C::SCRATCH_PER_WARP;
    const long ngroups = (a.B + 31) / 32;
    const int lu = lane >> 3, l = lane & 7;
    const int r0 = l, r1 = l + 8;                  // rows of P (first product) = columns of Pn (second product)
    const bool v1 = r1 < 13;

    ekf_stage_W(Ws, a.W, threadIdx.x);
    if (lane < 4) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_u32(bars + lane)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // box of the warp's round `t` (filters first .. first + 7) -> buffer t & 1, one TMA tensor load issued by lane 0
    auto issue_load = [&](unsigned t, long first) {
        if (lane == 0) {
            const unsigned bar = smem_u32(bars + (t & 1));
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(C::BOX_BYTES) : "memory");
            asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                         :: "r"(smem_u32(wb + (t & 1) * C::BOX)), "l"(reinterpret_cast<unsigned long long>(&ta.tmP)),
                            "r"((int)first), "r"(0), "r"(0), "r"(bar) : "memory");
        }
    };
    // Jacobian tile of round r of the current group: scratch line [r] -> tile buffer t & 1, one 1-D bulk copy issued by lane 0
    auto issue_tile = [&](unsigned t, int r) {
        if (lane == 0) {
            const unsigned bar = smem_u32(bars + 2 + (t & 1));
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(C::TILE_BYTES) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(smem_u32(Jt + (t & 1) * C::TILE_D)), "l"(Jw + (long)r * C::TILE_D), "r"(C::TILE_BYTES), "r"(bar) : "memory");
        }
    };
    unsigned t = 0;                                 // rounds done by this warp (buffer and mbarrier phase bookkeeping)
    unsigned tile_ph0 = 0, tile_ph1 = 0;            // phases of the two tile barriers (only bulk-copied rounds flip them)
    long g = ekf_claim_group(a.next_group, lane);
    if (g < ngroups) issue_load(0, g * 32);
    while (g < ngroups) {
        const long g_next = ekf_claim_group(a.next_group, lane);
        // ---------------- step 1: lane = filter ----------------------------------------------------------------
        // (t is even here: a group has four rounds, so round 0 always uses tile buffer 0)
        ekf_filter_step<RIGID>(a, g * 32 + lane, EkfTileSink{Jw + (lane >> 3) * C::TILE_D + (lane & 7), lane < 8 ? Jt + lane : nullptr}, [&] {
            // the scratch lines of rounds 1..3 are read by the async proxy (bulk copies issued by lane 0)
            // (each lane orders its own generic-proxy stores before later async-proxy reads; __syncwarp makes them
            // visible to lane 0, which issues the copy.  A full __threadfence here cost 5 % of the kernel: ERRBAR + CCTL.IVALL)
            asm volatile("fence.proxy.async;" ::: "memory");
            __syncwarp();
            issue_tile(t + 1, 1);                  // buffer 1: last read by the previous group's round 3
        });
        __syncwarp();                               // round 0's tile (written by lanes 0..7) is visible to the warp
#pragma unroll 1
        for (int r = 0; r < 4; ++r, ++t) {
            const double* const Tt = Jt + (t & 1) * C::TILE_D;
            if (r > 0) {                            // the round's Jacobian tile has landed
                if (t & 1) { mbar_wait(bars + 3, tile_ph1); tile_ph1 ^= 1; }
                else { mbar_wait(bars + 2, tile_ph0); tile_ph0 ^= 1; }
            }
            unsigned char* const box = wb + (t & 1) * C::BOX;
            mbar_wait(bars + (t & 1), (t >> 1) & 1);
            // ---------------- phase B: 8 lanes = filter, 2 passes of 4 filters ---------------------------------
            // Box entry (row, col) of this lane's filter sits at box + (row * 13 + col) * 64 + filter * 8 with the TMA's 64-byte
            // swizzle (16-byte chunk index ^= address bits 7..8).  The swizzled address is computed from the absolute shared
            // address (3 integer instructions on the idle ALU pipe) instead of being looked up in a per-lane offset table in
            // shared memory: 104 of the 406 shared-memory instructions of a pass, and one LDS latency in front of every
            // product, were table lookups (profiles/r2o ncu source page).
            // (boxes are 512-byte aligned, so address bits 7..8 are those of the offset)
            auto sw = [](unsigned o) -> unsigned { return o ^ ((o >> 3) & 0x30u); };
            auto BX = [&](unsigned o) -> double& { return *reinterpret_cast<double*>(box + sw(o)); };
            auto next_box = [&](int r) {
                // half a round after the previous round's store was issued: its buffer has been read out, the next
                // round's box may land in it (next round of this group, or round 0 of the next group)
                const long nfirst = (r < 3) ? g * 32 + (r + 1) * 8 : g_next * 32;
                if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                if (r < 3 || g_next < ngroups) issue_load(t + 1, nfirst);
            };
#pragma unroll 1
            for (int p = 0; p < 2; ++p) {
                const double* __restrict__ T = Tt + p * 4 + lu;
                const unsigned fo = (unsigned)(p * 4 + lu) * 8u;                           // this lane's filter column of the box
                const unsigned row0 = fo + (unsigned)(r0 * 13) * 64u, row1 = fo + (unsigned)((v1 ? r1 : r0) * 13) * 64u;   // entry (r, 0)
                const unsigned col0 = fo + (unsigned)r0 * 64u, col1 = fo + (unsigned)(v1 ? r1 : r0) * 64u;                 // entry (0, c)
                double p0[13], p1[13], n0[13], n1[13];
#pragma unroll
                for (int k = 0; k < 13; ++k) {          // rows r0, r1 of P
                    p0[k] = BX(row0 + k * 64u);
                    p1[k] = v1 ? BX(row1 + k * 64u) : 0.0;
                }
                jac_times2<ARM, RIGID, 8>(T, p0, p1, n0, n1);
#pragma unroll
                for (int k = 0; k < 13; ++k) {          // rows r0, r1 of Q = P A^T, in place
                    BX(row0 + k * 64u) = fma(a.dt, n0[k], p0[k]);
                    if (v1) BX(row1 + k * 64u) = fma(a.dt, n1[k], p1[k]);
                }
                __syncwarp();
                if (p == 0) next_box(r);
#pragma unroll
                for (int k = 0; k < 13; ++k) {          // columns r0, r1 of Q
                    p0[k] = BX(col0 + k * (13 * 64u));
                    p1[k] = v1 ? BX(col1 + k * (13 * 64u)) : 0.0;
                }
                jac_times2<ARM, RIGID, 8>(T, p0, p1, n0, n1);
#pragma unroll
                for (int i = 0; i < 13; ++i) {          // columns r0, r1 of Pn = A Q + W, in place
                    BX(col0 + i * (13 * 64u)) = fma(a.dt, n0[i], p0[i]) + Ws[i * 13 + r0];
                    if (v1) BX(col1 + i * (13 * 64u)) = fma(a.dt, n1[i], p1[i]) + Ws[i * 13 + r1];
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();                           // every lane is done with the tile and the box of this round
            if (r < 2) issue_tile(t + 2, r + 2);    // this round's tile buffer is free: the tile of round r + 2 lands a round ahead
            if (lane == 0) {                            // filters >= B are clipped by the tensor map
                asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                             :: "l"(reinterpret_cast<unsigned long long>(&ta.tmPn)), "r"((int)(g * 32 + r * 8)), "r"(0), "r"(0),
                                "r"(smem_u32(box)) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
        }
        g = g_next;
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// EKF measurement update with H = [0_{7x6} I_7] (kiteEKF.cpp:115-125), thread per filter, IN PLACE:
//   S = H P H^T + V (7x7), K = P H^T S^-1 (13x7), x += K (z - H x), P <- P - K H P.
// S is inverted in place (Gauss-Jordan sweep on 49 registers; S is SPD so no pivoting), the gain K is parked in shared
// memory ([91 + 13][block] columns, conflict free) because K (182 registers) and S^-1 (98) do not fit together, and the
// covariance update then walks P column by column with the 7 entries of H P for that column in registers.
// In place without a staging copy: every entry of P is read before it is written (column c is only written after all
// reads of column c, and K only needs columns 6..12 BEFORE any write).  What made the first in-place version slow
// (1.65 ms per 1 M filters against 1.27 ms for out-of-place + copy back) was not the missing read-only path but ordering:
// with loads and stores on the same buffer the compiler may not hoist a load above an earlier store, so
// "load, 7 FMAs, store" per entry became 169 dependent memory round trips.  Here the loads of a column PAIR (26, which
// contain (H P) of the pair: rows 6..12 of the columns themselves) are issued in one batch, one pair AHEAD of the stores of
// the previous pair, the pair after that is pulled into L2 by register-free prefetches, every gain entry read from shared
// memory serves two columns, four rows of K are in flight at once, and the state update is one batch at the end.  The
// kernel is latency bound at 8 warps per SM (the gain's 832 B of shared memory per filter cap the occupancy, and the
// alternative -- M = S^-1 (H P) in registers next to S^-1 -- needs the same 196+ registers): round 2, 0.88 -> 0.75 ms per
// 1 M filters (profiles/r2v_ekf_update_*.log).
struct EkfUpdArgs {
    long B, ld;
    const double* z; double* P; double* x;
    const double* V;         // device [49]
    int32_t* status;         // [ld] per-filter flag (non-finite updated state: singular innovation covariance) or null
};
constexpr int EKFU_BLOCK = 128;
constexpr int EKFU_COLS = 2;         // covariance columns per pass of the update
constexpr int EKFU_KUNROLL = 4;      // rows of K in flight: 28 loads instead of 7 between dependent DRAM round trips (0.88 -> 0.81 ms)
template <int DUMMY = 0>
__global__ void __launch_bounds__(EKFU_BLOCK, 2) k_ekf_update(const __grid_constant__ EkfUpdArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* const Ks = reinterpret_cast<double*>(smem_raw) + threadIdx.x;        // K[r][c] at Ks[(r*7+c)*EKFU_BLOCK], dx[r] at Ks[(91+r)*EKFU_BLOCK]
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.B) return;
    double* const P = a.P + i;
    const long ld = a.ld;
    double S[7][7];
#pragma unroll
    for (int r = 0; r < 7; ++r)
#pragma unroll
        for (int c = 0; c < 7; ++c) S[r][c] = P[(long)((6 + r) * 13 + 6 + c) * ld] + __ldg(a.V + r * 7 + c);
#pragma unroll
    for (int c = 0; c < 7; ++c) {                  // in-place inverse
        const double d = 1.0 / S[c][c];
#pragma unroll
        for (int j = 0; j < 7; ++j) if (j != c) S[c][j] *= d;
#pragma unroll
        for (int r = 0; r < 7; ++r) {
            if (r == c) continue;
            const double f = S[r][c];
#pragma unroll
            for (int j = 0; j < 7; ++j) if (j != c) S[r][j] = fma(-f, S[c][j], S[r][j]);
            S[r][c] = -f * d;
        }
        S[c][c] = d;
    }
    double y[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) y[k] = __ldg(a.z + (long)k * ld + i) - a.x[(long)(6 + k) * ld + i];
#pragma unroll EKFU_KUNROLL
    for (int r = 0; r < 13; ++r) {                 // K row r = P[r][6:13] S^-1; state increment (no global store in this loop)
        double pk[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) pk[k] = P[(long)(r * 13 + 6 + k) * ld];
        double dx = 0.0;
#pragma unroll
        for (int c = 0; c < 7; ++c) {
            double kv = 0.0;
#pragma unroll
            for (int k = 0; k < 7; ++k) kv = fma(pk[k], S[k][c], kv);
            Ks[(r * 7 + c) * EKFU_BLOCK] = kv;
            dx = fma(kv, y[c], dx);
        }
        Ks[(91 + r) * EKFU_BLOCK] = dx;
    }
    {                                              // x += K y: 13 loads, then 13 stores
        double xv[13];
#pragma unroll
        for (int r = 0; r < 13; ++r) xv[r] = a.x[(long)r * ld + i];
#pragma unroll
        for (int r = 0; r < 13; ++r) { xv[r] += Ks[(91 + r) * EKFU_BLOCK]; a.x[(long)r * ld + i] = xv[r]; }
        if (a.status) a.status[i] = all_finite13(xv) ? 0 : FLAG_NONFINITE;
    }
    // P[:, c] <- P[:, c] - K (H P)[:, c], TWO columns per pass: every gain entry read from shared memory serves both, the next
    // pair's 26 loads fly behind this pair's FMAs, and the pair after that is pulled into L2 (register free).  (H P)[:, c] is
    // rows 6..12 of column c itself: no separate loads.  Column 13 does not exist: the last pass handles column 12 alone.
    constexpr int NC = EKFU_COLS;
    double pv[NC][13], pq[NC][13];
#pragma unroll
    for (int j = 0; j < NC; ++j)
#pragma unroll
        for (int r = 0; r < 13; ++r) pv[j][r] = P[(long)(r * 13 + j) * ld];
#pragma unroll 1
    for (int c = 0; c < 13; c += NC) {
        if ((threadIdx.x & 15) == 0) {
#pragma unroll
            for (int j = 0; j < NC; ++j)
                if (c + 2 * NC + j < 13) {
#pragma unroll
                    for (int r = 0; r < 13; ++r) asm volatile("prefetch.global.L2 [%0];" :: "l"(P + (long)(r * 13 + c + 2 * NC + j) * ld));
                }
        }
#pragma unroll
        for (int j = 0; j < NC; ++j)
#pragma unroll
            for (int r = 0; r < 13; ++r) pq[j][r] = (c + NC + j < 13) ? P[(long)(r * 13 + c + NC + j) * ld] : 0.0;
#pragma unroll
        for (int r = 0; r < 13; ++r) {
            double v[NC];
#pragma unroll
            for (int j = 0; j < NC; ++j) v[j] = pv[j][r];
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const double kk = Ks[(r * 7 + k) * EKFU_BLOCK];
#pragma unroll
                for (int j = 0; j < NC; ++j) v[j] = fma(-kk, pv[j][6 + k], v[j]);
            }
#pragma unroll
            for (int j = 0; j < NC; ++j)
                if (c + j < 13) P[(long)(r * 13 + c + j) * ld] = v[j];
        }
#pragma unroll
        for (int j = 0; j < NC; ++j)
#pragma unroll
            for (int r = 0; r < 13; ++r) pv[j][r] = pq[j][r];
    }
}

// ================================================================================================
// NMPC collocation constraint + Jacobian blocks (chebyshev.hpp:241-271, kiteNMPF.cpp:58-111,169-171).
//   block = 32 scenarios x M nodes (warp k <-> node k); thread (s,k) evaluates the scaled augmented RHS and
//   its Jacobian at node k of scenario s and the row block k of (compD (x) I) X.
// ================================================================================================
struct CollocArgs {
    KiteConsts K;
    long B, ld;
    int M;
    double tau;
    double sx[15], isx[15], su[4], isu[4];
    const double* compD;     // device [M][M]
    // compact rows of compD in the constant bank (M <= 16 nodes, <= 8 non-zeros per row: every NMPC / test configuration of the
    // reference): column indices and values of row k, read with the warp-uniform k -- no dependent global load per column
    int cd_compact;          // 1: use cd_nz / cd_col / cd_val, 0: walk the dense row in global memory
    int cd_nz[16];
    signed char cd_col[16][8];
    double cd_val[16][8];
    const double* z; const double* p;
    double* G; double* JX; double* JU; double* gnorm;
    int32_t* status;         // [ld] per-scenario flags, OR over the nodes, or null
};

struct CollocSink {
    double* jxp; double* jup; long ld;
    const double* sx; const double* isx; const double* isu;
    __device__ __forceinline__ void jx(int i, int j, double v) const { if (jxp) jxp[(long)(i * 15 + j) * ld] = sx[i] * v * isx[j]; }
    __device__ __forceinline__ void ju(int i, int j, double v) const { if (jup) jup[(long)(i * 4 + j) * ld] = sx[i] * v * isu[j]; }
    __device__ __forceinline__ void aero(double, double, double) const {}
};

// ---- compact node blocks: structural non-zeros only, in CCS (column-major) order ------------------------------------
// The reference's AugJacobian is a SPARSE CasADi matrix (kiteNMPF.cpp:169-171): per node it carries the 104 (+ 21 with a
// tether arm) non-zeros of d f / d x, the 7 of d f / d u and the two constant entries of the augmented rows
// (theta_dot = V1: (13, 14); V1_dot = u_v: (14, 15 + 3)).  Slot numbering = position in a column-major walk over the
// 15 x 19 node block [d f_s / d x_s | d f_s / d u_s]; the same table answers kite_colloc_sparsity().
__host__ __device__ constexpr bool colloc_nz(int i, int j, bool arm) {       // i in 0..14, j in 0..18
    if (j < 15) {
        if (i < 13 && j < 13) return jx_nz(i, j, arm);
        return i == 13 && j == 14;
    }
    if (i < 13 && j - 15 < 3) return ju_nz(i, j - 15);
    return i == 14 && j == 18;
}
struct CollocTab { int slot[15][19]; int nnz; };
constexpr CollocTab make_colloc_tab(bool arm) {
    CollocTab t{};
    int s = 0;
    for (int j = 0; j < 19; ++j)
        for (int i = 0; i < 15; ++i) t.slot[i][j] = colloc_nz(i, j, arm) ? s++ : -1;
    t.nnz = s;
    return t;
}
__device__ constexpr CollocTab COLLOC_TAB_NOARM = make_colloc_tab(false);
__device__ constexpr CollocTab COLLOC_TAB_ARM = make_colloc_tab(true);
constexpr int COLLOC_NNZ_NOARM = make_colloc_tab(false).nnz, COLLOC_NNZ_ARM = make_colloc_tab(true).nnz;
static_assert(COLLOC_NNZ_NOARM == 104 + 7 + 2 && COLLOC_NNZ_ARM == 125 + 7 + 2, "node-block non-zeros");

template <bool ARM>
struct CollocSparseSink {       // value of entry (i, j) of the node block goes to row slot(i, j) of the node's [nnz][ld] slab
    double* jv; long ld;
    const double* sx; const double* isx; const double* isu;
    __device__ __forceinline__ void jx(int i, int j, double v) const {
        const int sl = (ARM ? COLLOC_TAB_ARM : COLLOC_TAB_NOARM).slot[i][j];
        if (sl >= 0) jv[(long)sl * ld] = sx[i] * v * isx[j];
    }
    __device__ __forceinline__ void ju(int i, int j, double v) const {
        const int sl = (ARM ? COLLOC_TAB_ARM : COLLOC_TAB_NOARM).slot[i][15 + j];
        if (sl >= 0) jv[(long)sl * ld] = sx[i] * v * isu[j];
    }
    __device__ __forceinline__ void aero(double, double, double) const {}
};

// FMT 0: dense 15 x 15 / 15 x 4 node blocks (JX, JU);  1 / 2: structural non-zeros only (JV), without / with tether arm;  3: G only.
template <bool PERCOEF, int NPB, int FMT>
__global__ void __launch_bounds__(32 * NPB) k_colloc_eval(const __grid_constant__ CollocArgs a) {
    __shared__ double red[NPB][32];                // partial ||G||^2 per node row of the block
    __shared__ int redf[NPB][32];                  // flags per node row of the block
    int flags = 0;
    // per-scenario aero coefficients live in shared memory (one 21-double record per thread, re-read at every use): held in
    // registers they pushed the Jacobian code over the 255-register limit (136 B / 184 B of spills in round 1)
    __shared__ AeroCoef coef_sh[PERCOEF ? 32 * NPB : 1];
    const int lane = threadIdx.x;
    const int ky = threadIdx.y;
    const long s = (long)blockIdx.x * 32 + lane;
    const int M = a.M;
    double g2 = 0.0;
    {
        // Pull the CTA's whole block of decision variables (19 M rows x 32 scenarios, 2 lines per row) towards the SM before
        // anything depends on it: a thread otherwise meets a first-touch DRAM miss at its own node AND in every column of its
        // (compD (x) I) X row block (the neighbour nodes' rows: dependent misses, 36 % of the sparse kernel's time,
        // profiles/r2v ncu source page).  128 threads, <= 4 prefetches each, no registers held.
        const int nlines = 2 * 19 * M;
        const long s0 = (long)blockIdx.x * 32;
        for (int t = ky * 32 + lane; t < nlines; t += 32 * NPB) {
            const long col = s0 + (t & 1) * 16;
            if (col < a.B) asm volatile("prefetch.global.L2 [%0];" :: "l"(a.z + (long)(t >> 1) * a.ld + col));
        }
    }
    // shared coefficients with the tether-arm entries (FMT 2): read from shared memory as well -- as uniform operands from the
    // constant bank that instantiation alone spilled (88 B); one record per CTA, broadcast loads
    constexpr bool COEF_SH = !PERCOEF && FMT == 2;
    if constexpr (COEF_SH) {
        if (lane == 0 && ky == 0) coef_sh[0] = a.K.A;
        __syncthreads();
    }
    if (s < a.B) {
        if constexpr (PERCOEF) {
            AeroCoef At;
            load_coef(a.K, a.p, a.ld, s, At);
            coef_sh[ky * 32 + lane] = At;
        }
        const volatile AeroCoef& Av = coef_sh[PERCOEF ? ky * 32 + lane : 0];
        for (int k = ky; k < M; k += NPB) {
            double x[13], u[3], f[13];
            const double* zx = a.z + (long)(k * 15) * a.ld + s;
            const double* zu = a.z + (long)(M * 15 + k * 4) * a.ld + s;
#pragma unroll
            for (int c = 0; c < 13; ++c) x[c] = a.isx[c] * __ldg(zx + (long)c * a.ld);
            const double x14 = a.isx[14] * __ldg(zx + 14L * a.ld);
#pragma unroll
            for (int c = 0; c < 3; ++c) u[c] = a.isu[c] * __ldg(zu + (long)c * a.ld);
            const double u3 = a.isu[3] * __ldg(zu + 3L * a.ld);
            flags |= singularity_flags<false>(x);
            if constexpr (FMT == 3) {              // constraint values only (what a line search asks for): no Jacobian code at all
                NoSink sink;
                if constexpr (PERCOEF) kite_eval<false>(a.K, Av, x, u, f, sink);
                else kite_eval<false>(a.K, a.K.A, x, u, f, sink);
            } else if constexpr (FMT == 0) {
                CollocSink sink{a.JX ? a.JX + (long)(k * 225) * a.ld + s : nullptr,
                                a.JU ? a.JU + (long)(k * 60) * a.ld + s : nullptr, a.ld, a.sx, a.isx, a.isu};
                if constexpr (PERCOEF) kite_eval<true>(a.K, Av, x, u, f, sink);
                else kite_eval<true>(a.K, a.K.A, x, u, f, sink);
                // augmented rows: theta_dot = V1 (x[14]), V1_dot = u_v (u[3])   (kiteNMPF.cpp:62-73)
                if (a.JX) sink.jxp[(long)(13 * 15 + 14) * a.ld] = a.sx[13] * a.isx[14];
                if (a.JU) sink.jup[(long)(14 * 4 + 3) * a.ld] = a.sx[14] * a.isu[3];
                // structural zeros of the dense node blocks are written here, once, instead of a memset pass over the
                // 25 KB/scenario output beforehand (the kernel is HBM-write bound: every byte is stored exactly once)
                if (a.JX) {
                    const bool arm = a.K.has_arm != 0;
#pragma unroll
                    for (int i = 0; i < 15; ++i)
#pragma unroll
                        for (int j = 0; j < 15; ++j) {
                            const bool kite_blk = (i < 13 && j < 13);
                            const bool nz_noarm = kite_blk ? jx_nz(i, j, false) : (i == 13 && j == 14);
                            const bool nz_arm = kite_blk ? jx_nz(i, j, true) : (i == 13 && j == 14);
                            if (!nz_arm || (!nz_noarm && !arm)) sink.jxp[(long)(i * 15 + j) * a.ld] = 0.0;
                        }
                }
                if (a.JU) {
#pragma unroll
                    for (int i = 0; i < 15; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (!((i < 13 && j < 3) ? ju_nz(i, j) : (i == 14 && j == 3))) sink.jup[(long)(i * 4 + j) * a.ld] = 0.0;
                }
            } else {
                constexpr bool ARM = (FMT == 2);
                constexpr int NNZ = ARM ? COLLOC_NNZ_ARM : COLLOC_NNZ_NOARM;
                CollocSparseSink<ARM> sink{a.JX + (long)(k * NNZ) * a.ld + s, a.ld, a.sx, a.isx, a.isu};
                if constexpr (PERCOEF) kite_eval<true>(a.K, Av, x, u, f, sink);
                else if constexpr (COEF_SH) kite_eval<true>(a.K, reinterpret_cast<const volatile AeroCoefPlain&>(coef_sh[0]), x, u, f, sink);
                else kite_eval<true>(a.K, a.K.A, x, u, f, sink);
                sink.jv[(long)(ARM ? COLLOC_TAB_ARM : COLLOC_TAB_NOARM).slot[13][14] * a.ld] = a.sx[13] * a.isx[14];
                sink.jv[(long)(ARM ? COLLOC_TAB_ARM : COLLOC_TAB_NOARM).slot[14][18] * a.ld] = a.sx[14] * a.isu[3];
            }
            double fa[15];
#pragma unroll
            for (int c = 0; c < 13; ++c) fa[c] = a.sx[c] * f[c];
            fa[13] = a.sx[13] * x14;
            fa[14] = a.sx[14] * u3;
            // G_k = sum_l compD[k][l] X_l - tau f_s
            double acc[15];
#pragma unroll
            for (int c = 0; c < 15; ++c) acc[c] = 0.0;
            if (a.cd_compact) {                    // (uniform) the row's non-zeros come from the constant bank: the 15 loads of
                const int nz = a.cd_nz[k];         // every column are independent of everything but the column index
                auto column = [&](int t) {
                    const double dkl = a.cd_val[k][t];
                    const double* zl = a.z + (long)(a.cd_col[k][t] * 15) * a.ld + s;
#pragma unroll
                    for (int c = 0; c < 15; ++c) acc[c] = fma(dkl, __ldg(zl + (long)c * a.ld), acc[c]);
                };
                if constexpr (FMT == 0 || FMT == 2) {   // dense blocks are HBM-write bound; there and with the tether-arm entries the unrolled loop spills
                    for (int t = 0; t < nz; ++t) column(t);
                } else {                           // two columns' loads in flight (the rows sit in L2 by now): 0.183 -> 0.170 ms sparse
#pragma unroll 2
                    for (int t = 0; t < nz; ++t) column(t);
                }
            } else {
                for (int l = 0; l < M; ++l) {
                    const double dkl = __ldg(a.compD + k * M + l);
                    if (dkl != 0.0) {              // warp-uniform: k is the same for the whole warp
                        const double* zl = a.z + (long)(l * 15) * a.ld + s;
#pragma unroll
                        for (int c = 0; c < 15; ++c) acc[c] = fma(dkl, __ldg(zl + (long)c * a.ld), acc[c]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 15; ++c) {
                const double gv = fma(-a.tau, fa[c], acc[c]);
                a.G[(long)(k * 15 + c) * a.ld + s] = gv;
                g2 = fma(gv, gv, g2);
            }
        }
    }
    if (a.gnorm || a.status) {
        red[ky][lane] = g2;
        redf[ky][lane] = flags;
        __syncthreads();
        if (ky == 0 && s < a.B) {
            double t = 0.0;
            int fl = 0;
#pragma unroll
            for (int l = 0; l < NPB; ++l) { t += red[l][lane]; fl |= redf[l][lane]; }
            if (a.gnorm) a.gnorm[s] = t;
            if (a.status) a.status[s] = fl | ((t * 0.0 == 0.0) ? 0 : FLAG_NONFINITE);     // a non-finite G poisons ||G||^2
        }
    }
}

// ================================================================================================
// NMPC performance index and gradient (Chebyshev::CollocateCost chebyshev.hpp:280-333 on the Lagrange / Mayer terms of
// kiteNMPF.cpp:116-143).  Thread (scenario, node): reads the 9 components of z the cost depends on, writes the 19
// gradient entries of its node (structural zeros included, so every output byte is stored exactly once) and adds its
// weighted Lagrange value to the scenario's cost through shared memory.  HBM bound: 72 B in, 152 B out per node.
// ================================================================================================
struct CostArgs {
    long B, ld;
    int M;
    double sx6[3], isx13, sx13;         // Scale_X entries used by the cost
    double Q[3], R[4], W, vref;         // weights, scaled reference velocity
    double rc[3], rs[3], ra[3];         // path(theta) = rc cos(theta) + rs sin(theta) + ra  (radius, altitude, rotation folded)
    const double* wnode;                // device [M]: tau * (sum of the quadrature weights of the segments a node belongs to)
    const double* z; double* cost; double* grad;
};
template <int NPB>
__global__ void __launch_bounds__(32 * NPB) k_colloc_cost(const __grid_constant__ CostArgs a) {
    __shared__ double red[NPB][32];
    const int lane = threadIdx.x, ky = threadIdx.y;
    const long s = (long)blockIdx.x * 32 + lane;
    const int M = a.M;
    double acc = 0.0;
    if (s < a.B) {
        for (int k = ky; k < M; k += NPB) {
            const double* zx = a.z + (long)(k * 15) * a.ld + s;
            const double* zu = a.z + (long)(M * 15 + k * 4) * a.ld + s;
            double xr[3], us[4];
#pragma unroll
            for (int c = 0; c < 3; ++c) xr[c] = __ldg(zx + (long)(6 + c) * a.ld);
            const double x13 = __ldg(zx + 13L * a.ld), x14 = __ldg(zx + 14L * a.ld);
#pragma unroll
            for (int c = 0; c < 4; ++c) us[c] = __ldg(zu + (long)c * a.ld);
            double sn, cs;
            sincos(a.isx13 * x13, &sn, &cs);
            double pc = 0.0, dth = 0.0, gr[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const double pp = fma(a.rc[c], cs, fma(a.rs[c], sn, a.ra[c]));
                const double dpp = fma(a.rs[c], cs, -a.rc[c] * sn);
                const double r = fma(a.sx6[c], pp, -xr[c]);
                const double qr = a.Q[c] * r;
                pc = fma(qr, r, pc);
                gr[c] = -2.0 * qr;
                dth = fma(2.0 * qr * a.sx6[c], dpp, dth);
            }
            dth *= a.isx13;
            const double dv = a.vref - x14;
            double L = fma(a.W * dv, dv, pc);
#pragma unroll
            for (int c = 0; c < 4; ++c) L = fma(a.R[c] * us[c], us[c], L);
            const double w = __ldg(a.wnode + k);
            const double wm = (k == 0) ? w + 1.0 : w;          // Mayer term sits on node 0 (the final time) with weight 1
            acc = fma(w, L, acc);
            if (k == 0) acc += pc;
            if (a.grad) {
                double* gx = a.grad + (long)(k * 15) * a.ld + s;
                double* gu = a.grad + (long)(M * 15 + k * 4) * a.ld + s;
#pragma unroll
                for (int c = 0; c < 15; ++c) {
                    double v = 0.0;
                    if (c >= 6 && c < 9) v = wm * gr[c - 6];
                    else if (c == 13) v = wm * dth;
                    else if (c == 14) v = -2.0 * w * a.W * dv;
                    gx[(long)c * a.ld] = v;
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) gu[(long)c * a.ld] = 2.0 * w * a.R[c] * us[c];
            }
        }
    }
    red[ky][lane] = acc;
    __syncthreads();
    if (ky == 0 && s < a.B) {
        double t = 0.0;
#pragma unroll
        for (int l = 0; l < NPB; ++l) t += red[l][lane];
        a.cost[s] = t;
    }
}

// ================================================================================================
// FP64 FMA peak microbenchmark: 8 independent register-resident DFMA chains per thread.
// ================================================================================================
template <int DUMMY = 0>
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double seed) {
    double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    const double m = 0.9999999, b = 1e-7;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
            a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
        }
    }
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}
constexpr long FP64_PEAK_FMAS_PER_ITER = 64;
// The same with THREE distinct vector-register operands per DFMA (a_i = a_i b_i + c_i, b_i and c_i per-thread values): the FP64
// pipe then issues one warp instruction every 3 cycles instead of every 2 (operand delivery, not the multiplier, is the limit):
// the practical ceiling of register-operand code such as the kite RHS (profiles/r2j_dfma_operands.log).
template <int DUMMY = 0>
__global__ void __launch_bounds__(256) k_fp64_peak3(double* out, int iters, double seed) {
    double a[8], b[8], c[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = seed + i + threadIdx.x; b[i] = 0.9999999 + 1e-9 * (i + threadIdx.x * seed); c[i] = 1e-7 * (i + 1) * seed + 1e-13 * threadIdx.x; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = fma(a[i], b[i], c[i]);
        }
    }
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += a[i];
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = t;
}

// Accuracy self-test of kite_math.cuh on the real MUFU seeds: which = 0 rcp, 1 rsqrt, 2 asin_poly, 3 logistic, 4 asin_sc(x, sqrt(1-x^2)),
// 5 / 6: the table forms of 4 / 3 (asin_red, 2^(j/32) table) that the identification-sweep kernels use.
template <int DUMMY = 0>
__global__ void __launch_bounds__(256) k_math_selftest(const double* __restrict__ x, double* __restrict__ out, long n, int which) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double a = x[i];
    double r;
    switch (which) {
        case 0: r = fast_rcp(a); break;
        case 1: r = fast_rsqrt(a); break;
        case 2: r = asin_poly(a); break;
        case 3: r = fast_logistic<false>(a); break;
        case 5: { const double c2 = fma(-a, a, 1.0); r = asin_sc<true>(a, c2 > 0.0 ? c2 * fast_rsqrt(c2) : 0.0); } break;
        case 6: r = fast_logistic<true>(a); break;
        default: { const double c2 = fma(-a, a, 1.0); r = asin_sc<false>(a, c2 > 0.0 ? c2 * fast_rsqrt(c2) : 0.0); } break;
    }
    out[i] = r;
}

}  // namespace kite
