/* =====================================================================================
 * kite_b200.h -- C ABI of the B200-native batched kite-dynamics engine (libkite_b200.so).
 *
 * This is the drop-in boundary for openKITE's kite_model hot path.  Every entry point
 * names the reference interface it replaces (paths under /root/reference/src).  In the
 * reference those interfaces are casadi::Function objects evaluated one point at a time
 * on one CPU thread; here each call evaluates B independent points/trajectories on the
 * GPU.  B = 1 reproduces the single-point semantics of the reference API.
 *
 * Conventions
 *   - plain C: opaque context pointer, POD parameter struct, raw pointers + sizes.
 *   - all numerical data is FP64.
 *   - "_d" pointers are DEVICE pointers, structure-of-arrays: component c of unit i is at
 *     ptr[c * ld + i] (ld >= B, the leading dimension in elements).  Consecutive units are
 *     adjacent in memory, so a warp's loads/stores are coalesced.
 *   - "_host" entry points take HOST pointers in the same SoA layout and perform the
 *     host<->device copies themselves on the context's stream (chunked and overlapped with
 *     compute for the long rollouts).
 *   - state   x = [v(3) w(3) r(3) q(4)]  (kite.cpp:320), control u = [T dE dR] (kite.cpp:321)
 *   - matrices are row-major flattened into the component index: Jx component = i*13 + j.
 *   - every function returns 0 on success, a negative kite_status otherwise; never throws.
 *     kite_last_error() gives a message.  Calls are stream-ordered on the context's stream;
 *     a context is not thread-safe (the reference is single-threaded); many contexts may exist.
 *   - there is NO CPU fallback: without a CUDA device kite_create fails with KITE_ERR_CUDA.
 * ===================================================================================== */
#ifndef KITE_B200_H
#define KITE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KITE_NX 13
#define KITE_NU 3
#define KITE_NP 21      /* identification parameters, order of kite.cpp:571-572 */
#define KITE_NX_AUG 15  /* NMPC augmented state  (kiteNMPF.cpp:58-73) */
#define KITE_NU_AUG 4

typedef enum kite_status {
    KITE_OK = 0,
    KITE_ERR_ARG = -1,     /* null pointer, bad size, bad enum */
    KITE_ERR_CUDA = -2,    /* CUDA runtime error (message in kite_last_error) */
    KITE_ERR_NCCL = -3,    /* NCCL error / NCCL library not found */
    KITE_ERR_STATE = -4    /* call not valid for this context (e.g. model kind) */
} kite_status;

/* Per-unit status flags (int32, OR-ed): what the rollout's status_d and the buffer of kite_set_status_buffer carry. */
typedef enum kite_status_flag {
    KITE_FLAG_NONFINITE = 1,     /* a result of this unit is NaN / Inf */
    KITE_FLAG_LOW_AIRSPEED = 2,  /* evaluated at |v|^2 < 1e-12: the aerodynamic angles are regulariser-dominated (kite.cpp:200-201) */
    KITE_FLAG_ZERO_TETHER = 4    /* evaluated at |r|^2 < 1e-18: the tether direction r/|r| is undefined (kite.cpp:247-258) */
} kite_status_flag;

/* Which right-hand side the context evaluates. */
typedef enum kite_model_kind {
    KITE_MODEL_KITE = 0,       /* KiteDynamics(props, algo)        kite.cpp:90-363  (1e-4 regularisers) */
    KITE_MODEL_KITE_ID = 1,    /* KiteDynamics(props, algo, id)    kite.cpp:365-616 (no regularisers, p[21]) */
    KITE_MODEL_RIGID_BODY = 2  /* RigidBodyKinematics              kite.cpp:622-661 */
} kite_model_kind;

/* The subset of KiteProperties (kite.h:9-87) the dynamics consume (kite.cpp:99-175). */
typedef struct kite_params {
    double b, c, AR, S;                         /* geometry.b, c, AR, S */
    double mass, Ixx, Iyy, Izz, Ixz;            /* inertia.* */
    double CL0, CLa_total, e_oswald, CD0_total, CYb, Cm0, Cma, Cn0, Cnb, Cl0, Clb;
    double CLq, Cmq, CYr, Cnr, Clr, CYp, Clp, Cnp;
    double CLde, CYdr, Cmde, Cndr, Cldr;
    double Ks, Kd, tether_length, rx, ry, rz;   /* tether.* (rx/ry/rz default 0 when absent) */
} kite_params;

typedef struct kite_ctx kite_ctx;

/* How the control argument of a rollout is laid out. */
typedef enum kite_u_mode {
    KITE_U_CONST = 0,      /* u[3][ld]: one control per trajectory, held for all steps (ODESolver semantics) */
    KITE_U_PER_STEP = 1,   /* u[N][3][ld]: control of trajectory i at step k is u[(k*3 + c)*ld + i] */
    KITE_U_SHARED = 2,     /* u[N][3]: one control log shared by all trajectories (identification sweeps) */
    KITE_U_SYNTH = 3       /* x0 AND u generated on device by the counter RNG keyed on the global index */
} kite_u_mode;

/* ---------------------------------------------------------------- lifecycle ------------- */
/* Replaces: KiteDynamics constructors (kite.cpp:90, :365), RigidBodyKinematics (kite.cpp:622). */
int kite_create(kite_ctx** out, const kite_params* params, int model_kind, int device);
int kite_destroy(kite_ctx* ctx);
/* Launch on an existing cudaStream_t (e.g. torch's current stream); NULL = the CUDA default stream.
 * A new context launches on its own non-blocking stream; kite_reset_stream returns to it. */
int kite_set_stream(kite_ctx* ctx, void* cuda_stream);
int kite_reset_stream(kite_ctx* ctx);
/* Per-unit status flags next to the results (SURVEY.md section 5).  While a buffer is set (status_d: DEVICE int32 [ld]; NULL
 * switches it off), kite_rk4_sens_step / _rollout, kite_ekf_predict_batch / _update_batch and kite_colloc_eval[_sparse]
 * write one kite_status_flag word per unit: non-finite results and the V -> 0 / |r| -> 0 singularities of the state(s) the
 * model was evaluated at (pre-step state for the integrators, OR over the steps of a rollout and over the nodes of a
 * scenario).  The reference has no such channel: CasADi returns NaN silently.  kite_rk4_rollout has its own status_d. */
int kite_set_status_buffer(kite_ctx* ctx, int32_t* status_d);
int kite_synchronize(kite_ctx* ctx);
const char* kite_last_error(const kite_ctx* ctx);
const char* kite_version(void);
/* Number of kernel launches issued by this context since creation (bench.py's gpu_launches). */
long long kite_launch_count(const kite_ctx* ctx);

/* Device-memory helpers so that an FFI host (C++, cgo, JNI, ctypes) needs no CUDA runtime binding of its own.
 * Copies are issued on the context's stream and complete before returning. */
int kite_device_malloc(void** ptr_out, size_t bytes);   /* on the CURRENT device of the calling thread */
int kite_device_free(void* ptr);
/* Same, on the context's device (use these when a process owns contexts on several GPUs). */
int kite_ctx_malloc(kite_ctx* ctx, void** ptr_out, size_t bytes);
int kite_ctx_free(kite_ctx* ctx, void* ptr);
int kite_copy_h2d(kite_ctx* ctx, void* dst_d, const void* src_h, size_t bytes);
int kite_copy_d2h(kite_ctx* ctx, void* dst_h, const void* src_d, size_t bytes);

/* ---------------------------------------------------------------- pointwise ------------- */
/* Replaces: Function "dynamics"(x,u[,p]) -> xdot   kite.cpp:324 / :575.   p_d may be NULL. */
int kite_rhs_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d,
                   double* f_d);
/* Replaces: Function "Aero"(x,u) -> body-frame aerodynamic force Faero_b (3)   kite.cpp:224-234, :330
 * (KiteDynamics::getAeroDynamicForces, kite.h:126).  F_d [3][ld]. */
int kite_aero_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d,
                    double* F_d);
/* Replaces: Function "dyn_jacobian"(x,u[,p]) -> d f/d x (13x13)   kite.cpp:327-328 / :578-579.
 * Also returns d f/d u (13x3), which the reference only exposes inside AugJacobian (kiteNMPF.cpp:169-171).
 * Jx_d: [169][ld], Ju_d: [39][ld] (either may be NULL). */
int kite_jac_batch(kite_ctx* ctx, long B, long ld, const double* x_d, const double* u_d, const double* p_d,
                   double* Jx_d, double* Ju_d);

/* Structural non-zeros of d f/d x (wrt_u = 0; 104, or 125 with a tether arm; 49 for the rigid body) or d f/d u (wrt_u = 1;
 * 7) in compressed-column order: row_out[nnz], col_out[nnz] (either may be NULL to only count); returns nnz.  This is the
 * sparsity the reference's SX::jacobian yields (kite.cpp:327-328, SURVEY.md Appendix A).  Needs no context and no GPU. */
int kite_jac_sparsity(int model_kind, int has_arm, int wrt_u, int* row_out, int* col_out);

/* ---------------------------------------------------------------- RK4 ------------------- */
/* Replaces: Function "RK4"(X,U,dT) kite.cpp:332-338 == ODESolver::rk4_solve integrator.cpp:86-98, looped by
 * the caller (simulator.cpp:43-51).  Advances B trajectories by N classical RK4 steps of size h.
 *   x0_d [13][ld]          (ignored for KITE_U_SYNTH)
 *   u_d                    per kite_u_mode
 *   p_d  [21][ld] or NULL  per-trajectory aero coefficients (mandatory for KITE_MODEL_KITE_ID sweeps)
 *   xf_d [13][ld]          final states
 *   traj_d NULL or [N/save_every][13][ld]: state after every save_every-th step
 *   y_d NULL or [N][13]: shared measurement log; if given, cost_d[ld] receives the identification cost
 *        (1/N) sum_k sum_c Q_c (y[k][c] - x_c(k+1))^2   (kite_identification_test.cpp:193-205)
 *        which has no value for N = 0: y_d with N = 0 is rejected with KITE_ERR_ARG (also by kite_rk4_rollout_host)
 *   status_d NULL or int32[ld]: 0 = ok, 1 = non-finite state reached
 *   index0: global index of trajectory 0 of this call (only used by KITE_U_SYNTH; sharding-invariant inputs) */
int kite_rk4_rollout(kite_ctx* ctx, long B, long ld, long N, double h, const double* x0_d, const double* u_d, int u_mode,
                     const double* p_d, double* xf_d, double* traj_d, long save_every, const double* y_d, double* cost_d,
                     int32_t* status_d, long index0);

/* Same, HOST pointers (SoA, ld = B).  Copies are chunked over trajectories and overlapped with compute. */
int kite_rk4_rollout_host(kite_ctx* ctx, long B, long N, double h, const double* x0_h, const double* u_h, int u_mode,
                          const double* p_h, double* xf_h, const double* y_h, double* cost_h, int32_t* status_h);

/* Fill x0_d [13][ld] and u_d [N][3][ld] with the synthetic config-2 workload for global indices
 * [index0, index0+B) (SURVEY.md 8d).  Workload definition, not reference behaviour. */
int kite_synth_inputs(kite_ctx* ctx, long B, long ld, long N, long index0, double* x0_d, double* u_d);

/* Fill p_d [21][ld] with the parameter samples of the identification sweep for global indices [index0, index0+B)
 * (SURVEY.md 8d config 5): the reference coefficients (pref_h[21] HOST, order of kite.cpp:571-572; NULL = the context's
 * own) perturbed uniformly inside the bounds of kite_identification_test.cpp:127-148, keyed on the global index so that
 * the samples are identical under any sharding.  Workload definition, not reference behaviour. */
int kite_synth_id_params(kite_ctx* ctx, long B, long ld, long index0, const double* pref_h, double* p_d);

/* ---------------------------------------------------------------- sensitivities ---------- */
/* One RK4 step with forward-mode sensitivities for B independent shooting intervals:
 *   xn = RK4(x,u,h), Phi = d xn/d x (13x13), Gamma = d xn/d u (13x3).
 * Replaces: SX::jacobian chained through rk4_symbolic (kite.cpp:327,337; MATLAB RK4_JACOBIAN kite_sim.m:300-301).
 *   x_d [13][ld], u_d [3][ld], xn_d [13][ld], Phi_d [169][ld], Gamma_d [39][ld]
 *   work_d: device scratch of AT LEAST kite_rk4_sens_work_bytes(B) bytes (stage states of the resident warps of the
 *           persistent kernel, 16 KB per warp; independent of B beyond one wave: ~19 MB on a B200.  The stage Jacobians
 *           themselves never leave shared memory).
 *   Phi_d / Gamma_d are written by TMA tensor stores when their base and pitch are 16-byte aligned (even ld) and B is
 *   even, by ordinary stores otherwise: same values either way. */
size_t kite_rk4_sens_work_bytes(long B);
int kite_rk4_sens_step(kite_ctx* ctx, long B, long ld, double h, const double* x_d, const double* u_d, double* xn_d,
                       double* Phi_d, double* Gamma_d, void* work_d);
/* Multiple-shooting rollout: B trajectories x N steps, chained primal, per-step sensitivities, ONE kernel launch for the
 * whole horizon (the (step, group-of-32) work items are walked in step-major order; results are bitwise those of N
 * chained kite_rk4_sens_step calls).
 *   x0_d [13][ld], u_d [N][3][ld]; xs_d [N][13][ld] (state after each step), Phi_d [N][169][ld], Gamma_d [N][39][ld]
 *   work_d: kite_rk4_sens_work_bytes(B) bytes, as for the single step (it includes the per-group step counters). */
int kite_rk4_sens_rollout(kite_ctx* ctx, long B, long ld, long N, double h, const double* x0_d, const double* u_d,
                          double* xs_d, double* Phi_d, double* Gamma_d, void* work_d);

/* ---------------------------------------------------------------- collocation ------------ */
/* NMPC Chebyshev-collocation constraint and Jacobian for B scenarios.
 * Replaces: Chebyshev<SX,P,S,15,4,0>::CollocateDynamics (chebyshev.hpp:241-271) on the scaled augmented
 * dynamics (kiteNMPF.cpp:58-111) and AugJacobian (kiteNMPF.cpp:169-171).
 *   M = S*P+1 nodes (node 0 = final time).  compD [M][M] row-major HOST pointer (from Chebyshev::CompD before
 *   the kron with I; copied to the device once per call), tau = (tf-t0)/(2S), sx[15], su[4] HOST diagonal scalings.
 *   z_d  [M*15 + M*4][ld]     decision vector [X ; U] (scaled)
 *   p_d  [21][ld] or NULL     per-scenario aero coefficients (parameter perturbations)
 *   G_d  [M*15][ld]           G = (compD (x) I15) X - tau F
 *   JX_d [M*225][ld] or NULL  node blocks d f_s/d x_s (15x15 row-major per node); AugJacobian's varying part is -tau*JX
 *   JU_d [M*60][ld]  or NULL  node blocks d f_s/d u_s (15x4)
 *   gnorm_d [ld] or NULL      per-scenario ||G||_2^2 (warp-shuffle reduction over the nodes)
 * With JX_d = JU_d = NULL a values-only kernel runs (no Jacobian code: what a line search asks for). */
int kite_colloc_eval(kite_ctx* ctx, long B, long ld, int M, const double* compD_h, double tau, const double* sx_h,
                     const double* su_h, const double* z_d, const double* p_d, double* G_d, double* JX_d, double* JU_d,
                     double* gnorm_d);

/* The same evaluation with the node blocks in SPARSE form: only the structural non-zeros of [d f_s/d x_s | d f_s/d u_s]
 * (15 x 19 per node) are written, which is how the reference holds AugJacobian (a sparse CasADi matrix in CCS,
 * kiteNMPF.cpp:169-171) and 2.5x fewer bytes on an HBM-write-bound kernel.
 *   kite_colloc_nnz_per_node: 113 = 104 (d f/d x) + 7 (d f/d u) + 2 (augmented rows); 134 with a tether arm.
 *   kite_colloc_sparsity:     row_out[nnz], col_out[nnz] (row 0..14, column 0..18 of the node block) in CCS order
 *                             (column-major, rows ascending inside a column); returns nnz.  Entry (i, j) of node k is entry
 *                             (15 k + i, 15 k + j) of d G/d X for j < 15 and (15 k + i, 15 M + 4 k + j - 15) of d G/d U
 *                             otherwise, each scaled by -tau (the constant part of d G/d z is compD (x) I15).
 *   JV_d [M * nnz][ld]        value of non-zero s of node k at JV_d[(k * nnz + s) * ld + i]; the other arguments as above. */
int kite_colloc_nnz_per_node(const kite_ctx* ctx);
int kite_colloc_sparsity(const kite_ctx* ctx, int* row_out, int* col_out);
int kite_colloc_eval_sparse(kite_ctx* ctx, long B, long ld, int M, const double* compD_h, double tau, const double* sx_h,
                            const double* su_h, const double* z_d, const double* p_d, double* G_d, double* JV_d,
                            double* gnorm_d);

/* NMPC performance index and its gradient for B scenarios.
 * Replaces: Chebyshev<SX,P,S,15,4,0>::CollocateCost (chebyshev.hpp:280-333) applied to the Lagrange and Mayer terms
 * of KiteNMPF::createNLP (kiteNMPF.cpp:116-143) -- the NLP objective "f" IPOPT evaluates every iteration:
 *   residual = Sx[6:9] path(x[13] / Sx[13]) - x[6:9],  L = sum Q residual^2 + W (vref - x[14])^2 + sum R u^2,
 *   cost = Mayer(X_0) + sum_segments tau sum_m w_m L(X_{seg P + m}, U_{seg P + m}),  Mayer = sum Q residual^2.
 * The path is a circle of path_radius / path_altitude rotated by the unit quaternion path_q, which is how both callers
 * of the reference build it (nmpf_node.cpp:31-39, kite_control_test.cpp:242-247).
 *   qw_h [P+1] HOST Clenshaw-Curtis weights (Chebyshev::QWeights), tau = (tf-t0)/(2S), sx_h[15] HOST state scaling
 *   z_d [M*15 + M*4][ld] (M = S*P+1, same layout as kite_colloc_eval), cost_d [ld], grad_d [M*19][ld] or NULL. */
typedef struct kite_nmpc_cost {
    double Q[3], R[4], W;                 /* kiteNMPF.cpp:32-34: Q = 1e2 diag(10,10,100), R = diag(1e-4,1e-1,1e-1,1e-3), W = 1e-3 */
    double vref_scaled;                   /* Scale_X(14,14) * vel_ref (kiteNMPF.h:34) */
    double path_radius, path_altitude, path_q[4];
} kite_nmpc_cost;
int kite_colloc_cost(kite_ctx* ctx, long B, long ld, int P, int S, const double* qw_h, double tau, const double* sx_h,
                     const kite_nmpc_cost* cost, const double* z_d, double* cost_d, double* grad_d);

/* ---------------------------------------------------------------- EKF -------------------- */
/* Replaces: KiteEKF::propagate (kiteEKF.cpp:75-98): xn = RK4(x,u,dt); A = I + Jx(x,u) dt; Pn = A P A^T + W.
 *   x_d [13][ld], u_d [3][ld], P_d [169][ld], W_h HOST 13x13 row-major; xn_d, Pn_d like x_d, P_d.
 *   work_d: device scratch of kite_ekf_work_bytes(B) bytes (currently 0: the Jacobian stays in shared memory; may be NULL).
 *   P_d and Pn_d must not alias.  The covariance moves as TMA boxes when P_d / Pn_d have a 16-byte aligned base and
 *   pitch (even ld) and B is even, through ordinary loads / stores otherwise: same arithmetic either way. */
size_t kite_ekf_work_bytes(long B);
int kite_ekf_predict_batch(kite_ctx* ctx, long B, long ld, double dt, const double* x_d, const double* u_d,
                           const double* P_d, const double* W_h, double* xn_d, double* Pn_d, void* work_d);
/* Replaces: the update half of KiteEKF::_estimate (kiteEKF.cpp:115-125) with H = [0 I7]:
 *   z_d [7][ld] measurements, V_h HOST 7x7; x_d, P_d updated in place (one kernel, no staging copy of P). */
int kite_ekf_update_batch(kite_ctx* ctx, long B, long ld, const double* z_d, const double* V_h, double* x_d, double* P_d);

/* ---------------------------------------------------------------- multi-GPU -------------- */
/* One process per GPU.  Trajectories are independent, so the only exchange is the final gather of
 * per-rollout costs and final states (NCCL over NVLink).  libnccl is resolved at run time (dlopen). */
int kite_comm_unique_id(char id_out[128]);
int kite_comm_init(kite_ctx* ctx, int nranks, int rank, const char id[128]);
/* recv_d[nranks*count] <- concatenation over ranks of send_d[count] (ncclAllGather, FP64). */
int kite_allgather(kite_ctx* ctx, const double* send_d, double* recv_d, long count);
int kite_comm_destroy(kite_ctx* ctx);

/* ---------------------------------------------------------------- diagnostics ------------ */
/* Register-resident dependent-DFMA microbenchmark: returns measured FP64 FMA throughput in TFLOP/s
 * (FMA = 2 flops) over `iters` iterations; the roofline denominator reported by bench.py. */
int kite_fp64_peak(kite_ctx* ctx, int iters, double* tflops_out);
/* The same chains with THREE distinct vector-register operands per DFMA (a = a b + c, all per-thread registers) instead of one
 * register and two constants: on B200 the FP64 pipe then issues every 3 cycles instead of every 2 (measured 24.2 against
 * 36.3 TFLOP/s), the practical ceiling of register-operand code.  Reported by bench.py next to the roofline peak. */
int kite_fp64_peak_reg3(kite_ctx* ctx, int iters, double* tflops_out);
/* Accuracy self-test of the engine's lean special functions on the device (MUFU seed + refinement):
 * out[i] = f(x[i]) with which = 0: 1/x, 1: 1/sqrt(x), 2: asin(x) for |x| <= 0.7072 (polynomial core),
 * 3: 1/(1+exp(-x)), 4: asin(x) for |x| <= 1 through the (sin, cos) pair form the model uses,
 * 5 / 6: the table-driven forms of 4 / 3 used by the kernels with per-trajectory coefficients (identification sweeps). */
int kite_math_selftest(kite_ctx* ctx, long n, const double* x_d, double* out_d, int which);

#ifdef __cplusplus
}
#endif
#endif /* KITE_B200_H */
