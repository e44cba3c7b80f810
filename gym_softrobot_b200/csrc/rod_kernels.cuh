// rod_kernels.cuh — the fused K-substep Cosserat-rod kernel for sm_100a.
//
// Mapping: one warp owns one rod (one env).  Lane l holds EPL consecutive
// elements k = l*EPL + j (and node k, Voronoi point k) entirely in registers for
// the whole launch; the difference / quadrature stencils (Delta_h, A_h) and the
// Q_{k+1} access of the curvature are warp shuffles at lane boundaries.  State is
// read from HBM once at launch entry and written once at exit (coalesced,
// vectorised EPL-wide), so a launch of K substeps moves 16(18n+6)/(nK) bytes per
// rod-element-substep (0.725 B at n=50, K=400): the kernel is FP64-pipe bound.
//
// What one substep computes (SURVEY.md Appendix A.2/A.3; reference boundary
// /root/reference/gym_softrobot/envs/soft_pendulum/soft_pendulum.py:183-184):
//   x += dt/2 v ; Q <- exp(dt/2 w) Q ; constrain values ;
//   l, t, e, eps ; sigma = e Q t - z ; n = S sigma ; f = Delta_h(Q^T n / e) ;
//   kappa = log(Q_{k+1} Q_k^T)/D ; tau = B kappa ;
//   T = Delta_h(tau/eps^3) + A_h(kappa x tau D/eps^3) + (Qt x n) l0 + (Jw/e) x w + (Jw/e) de/dt / e ;
//   gravity + actuation ; v += dt (f+F)/m ; w += dt J^-1 (T) e ; constrain rates ; damping ;
//   x += dt/2 v ; Q <- exp(dt/2 w) Q ; constrain values.
#pragma once
#include <stdint.h>
#include "rod_math.cuh"

namespace sr {

// field indices inside one env's [n_fields][stride] block
enum : int {
  F_POS = 0, F_VEL = 3, F_DIR = 6, F_OMEGA = 15, F_TAN = 18, F_KAPPA = 21, F_SIGMA = 24,
  F_DIL = 27,
  F_EDGE = 28,   // FP32 handles only: element edge vectors x_{k+1} - x_k kept as state (strain resolution)
  F_GAMMA = 31,  // (L/n) / rest_length_k: the reference derives every rest length from the rounded linspace
                 // positions, so they differ from L/n by ~1e-14 relative; the stretch strain must see that
  N_FIELDS = 32
};
constexpr int BC_DIM = 12;   // per-env anchors: fixed_position(3), fixed_directors(9)
constexpr int HEAD_DIM = 20;  // rigid head: x(3) v(3) Q(9) w(3) pinned z(1) pad(1)
constexpr int AUX_DIM = 8;   // per-env model scratch (3D pendulum: base position(3), velocity(3))
constexpr int WARPS_PER_CTA = 4;

enum : int { BC_FREE = 0, BC_ONE_END_FIXED = 1, BC_PENDULUM_SLIDER = 2, BC_MOVING_BASE = 3 };
enum : int { MODEL_ROD = 0, MODEL_SOFT_PENDULUM = 1, MODEL_SOFT_PENDULUM_3D = 2 };
enum : int { MATH_FAST = 0, MATH_FAITHFUL = 1 };

// Uniform-rod constants (all rods built by the reference are uniform:
// CosseratRod.straight_rod with scalar radius, soft_pendulum/build.py:54-61).
// Passed as a __grid_constant__ kernel parameter: operands come straight from
// the constant bank, costing neither registers nor load instructions.
template <typename T> struct RodArgs {
  T *state;            // [n_env][N_FIELDS][stride]
  const T *bc;         // [n_env][BC_DIM]
  T *aux;              // [n_env][AUX_DIM]
  const float *action; // [n_env][action_dim]
  float *obs;          // [n_env][obs_dim]
  double *reward;      // [n_env]
  uint8_t *terminated; // [n_env]
  int n_env, n_elem, stride, n_substeps;
  int bc_kind, model, point_force, damp_first, damping_on, laplace_order, action_dim, obs_dim;
  T dt, half_dt;
  T rest_len, inv_rest_len, rest_vor, inv_rest_vor;
  T S[3], B[3], J[3], Jinv[3];
  T mass, inv_mass, dt_inv_mass;  // interior node (end nodes carry half the mass)
  T g[3], gdt[3];
  T S_over_l[3], gdt_cv[3];   // S / rest_len ; dt g c_v  (packed kernel)
  T c_v, c_w[3], logc_w[3];
  T base_limit, inv_move_period; float base_step_f32;   // SoftPendulum3D base controller
  // RodPlaneContactWithAnisotropicFriction (SURVEY A.5) + per-env rest curvature (flat_env.py:310-311)
  const T *rest_kappa;  // [n_env][3][stride] or nullptr
  int contact_on, contact_before_forcing;
  T plane_origin[3], plane_normal[3], contact_k, contact_nu, slip_tol, inv_slip_tol, surface_tol;
  T kin_mu[3], stat_mu[3], vol_over_pi;
  // the contact models' internal frame: z = plane normal.  lab2int rotates lab vectors into it (identity / unused when
  // the normal is +z: rot_on = 0); plane_z0 = height of the plane in that frame; gm = interior nodal mass x gravity there
  T lab2int[9], plane_z0, gm[3]; int rot_on;
  // optional per-rod inputs (nullptr = off): ControllableFixConstraint ratios [n_rods] acting on index sucker_index;
  // external nodal forces (lab frame) / element couples (material frame) [n_rods][3][stride]; tapered-rod table
  const T *sucker; int sucker_index;
  const int *sucker_idx;              // [n_rods] per-rod index (python indexing: -1 = last node / last element) or nullptr = sucker_index
  const T *ext_force, *ext_couple;
  // COOMM TransverseMuscle under ApplyMuscles (tapered rods): per-rod scalar activation [n_rods] or nullptr = off; the
  // per-element factor -max_stress * rest_muscle_area is row ET_TM of elem_tab
  const T *tm_act;
  const T *elem_tab;                  // [ET_FIELDS][stride] element constants (VARY instantiations)
  // multi-rod environments (octopus: n_rod arms + one rigid Cylinder head joined by FixedJoint2Rigid,
  // envs/octopus/build.py:52-217, utils/custom_elastica/joint.py, constraint.py)
  int n_rod, has_head;
  T *head;                       // [n_env][HEAD_DIM]
  T joint_k, joint_nu, joint_kt, joint_radius, joint_cs[16][2];   // cos/sin of each arm's mounting angle
  T head_dt_inv_mass, head_J[3], head_Jinv[3];
  int isotropic;       // J1 == J2 (circular cross-section): c_w[0] == c_w[1]
  // fast-only / fallback pair of the packed kernel: envs that leave the fast-math domain are flagged in
  // redo[] by the fast-only kernel (which leaves their state untouched) and re-run by the safe kernel
  int *redo; int redo_filter;   // redo_filter: this (safe) launch steps flagged envs only and clears the flag
  unsigned long long *redo_count;   // running number of env-steps handed to the fallback (adaptive switch)
  // MuscleTorques travelling wave (continuum_snake.py:186-198): [n_env][muscle_dim] = time, wave number, beta[n]
  double *muscle; int muscle_on, muscle_dim;
  double mus_omega, mus_ramp, mus_phase; T mus_dir[3];
  // MuscleTorquesWithVaryingBetaSplines (muscle_torques_with_bspline.py): [n_env][spline_dim] state, basis table
  double *spline; const double *spline_tab; int spline_mask, spline_p, spline_dim;
  double spline_scale, spline_rate, spline_inv_dx;
  PolyCoef<T> poly;
  // ---- lean kernel (rod_kernel_lean.cuh) ---------------------------------------------------------------------
  // circular cross-section shortcuts and host-made tables
  T BDH;                              // (B3 - B1) D / 2
  T half_inv_rest_vor;                // 1 / (2 D)
  T dt_Jinv0;                         // dt / J1
  T bendw[10];                        // -theta'/(2 D sin theta') as a polynomial in |axial(R - R^T)|^2 (SR_COEF_BENDW)
  T bendw_mid[14]; int lim_bendm_hi;  // the same on the wider range of the plane models (SR_COEF_BENDW_MID)
  T cwp[2][3];                        // c_w^e as a quadratic in (e - 1), components 0 (= 1) and 2
  // the lean kernel's plane models: c_w^e to degree 6 (|z| <= kLeanExpZc), D / 2, the travelling wave's rotation
  // per substep (cos / sin of mus_omega dt) and 1 / ramp-up time
  T cwc[2][7], half_rest_vor; int lim_em1c_hi;
  double mus_cd, mus_sd, mus_inv_ramp;
  double sincg[3], cosch[3];          // sin(t)/t = 1 + q g(q), (1 - cos t)/t^2 = 1/2 + q h(q)  (the rotation update is FP64 in both modes)
  // double copies of what the FP64 part of the mixed (FP32-storage) mode reads
  double k_dt, k_half_dt, k_c_v, k_gdt_cv[3], k_dt_inv_mass, k_inv_rest_len;
  float limf_bend, limf_em1;          // range limits of the mixed mode's FP32 quantities
  int lim_rot_hi, lim_bend_hi, lim_em1_hi;   // range limits as high words (integer-pipe compares)
  // stream-K schedule: items of sk_rods_per_cta envs; sk_split = slots own equal substep ranges and hand partial
  // items over through sk_scratch[slot][18][NT] / sk_flag[slot]
  // sk_rodsync: per-rod named barriers inside the substep loop where the layout allows them; always 1 (fill_args), but
  // kept a run-time operand: folding it into the barrier choice changes ptxas's register allocation and spills
  int sk_rods_per_cta, sk_items, sk_split, sk_rodsync;
  double *sk_scratch; int *sk_flag;
  // ---- COOMM muscle layers with per-element activations (LMUS instantiation of the packed kernel; OctoReach-v0 /
  // OctoArmTwo-v0: reach_env.py:214-227, arm_two_env.py:222-247, create_es_muscle_layers build.py:292-338) ----
  const T *mus_act;                   // [n_rods][3][n_elem]: longitudinal 1, longitudinal 2, transverse; nullptr = off
  T lm_px[2], lm_py[2];               // material-frame offset of the longitudinal muscles, in units of the element radius
  T lm_gain;                          // max_stress(LM) / -max_stress(TM): scales row ET_TM (= -max_stress(TM) x rest area)
  int head_fixed;                     // OneEndFixedBC on the rigid head (reach_env.py:128-132): all its rates are zeroed
  // several ControllableFixConstraints per rod at fixed indices (arm_two_env.py:133-145): ratios [n_rods][3], nullptr = off
  const T *msucker; int msucker_n, msucker_loc[3];
};

// per-thread copy of the element / node / Voronoi constants of a tapered rod, and the rows of the HBM table they come from
template <typename T> struct ElemConst {
  T rest_len, inv_rest_len, rest_vor, inv_rest_vor, S[3], S_over_l[3], B[3], J[3], Jinv[3], c_w[3], logc_w[3], vol_over_pi;
  int isotropic;
};
enum : int { ET_REST_LEN = 0, ET_REST_VOR, ET_S0, ET_S2, ET_B0, ET_B2, ET_J0, ET_J2, ET_LOGCW0, ET_LOGCW2, ET_VOL_PI, ET_MASS, ET_TM, ET_FIELDS };

template <typename T, int EPL> struct Vec;
template <> struct Vec<double, 1> { using type = double; };
template <> struct Vec<double, 2> { using type = double2; };
template <> struct Vec<double, 4> { using type = double4; };
template <> struct Vec<float, 1> { using type = float; };
template <> struct Vec<float, 2> { using type = float2; };
template <> struct Vec<float, 4> { using type = float4; };

// EPL consecutive slots of one field row, as a single vector access (coalesced
// across the warp: 32 * EPL * sizeof(T) contiguous bytes).
template <typename T, int EPL>
__device__ __forceinline__ void load_row(const T *row, int lane, T (&out)[EPL]) {
  using VT = typename Vec<T, EPL>::type;
  VT v = reinterpret_cast<const VT *>(row)[lane];
  const T *p = reinterpret_cast<const T *>(&v);
#pragma unroll
  for (int j = 0; j < EPL; j++) out[j] = p[j];
}
template <typename T, int EPL>
__device__ __forceinline__ void store_row(T *row, int lane, const T (&in)[EPL]) {
  using VT = typename Vec<T, EPL>::type;
  VT v;
  T *p = reinterpret_cast<T *>(&v);
#pragma unroll
  for (int j = 0; j < EPL; j++) p[j] = in[j];
  reinterpret_cast<VT *>(row)[lane] = v;
}

// value of the same quantity at slot k+1 / k-1 (neighbour lane at the edges)
template <typename T, int EPL>
__device__ __forceinline__ void shift_next(const T (&a)[EPL], T (&out)[EPL]) {
  T edge = __shfl_down_sync(FULL, a[0], 1);
#pragma unroll
  for (int j = 0; j < EPL; j++) out[j] = (j < EPL - 1) ? a[(j + 1) % EPL] : edge;
}
template <typename T, int EPL>
__device__ __forceinline__ void shift_prev(const T (&a)[EPL], int lane, T (&out)[EPL]) {
  T edge = __shfl_up_sync(FULL, a[EPL - 1], 1);
  if (lane == 0) edge = T(0);  // slot -1 does not exist: stencils see 0 there
#pragma unroll
  for (int j = 0; j < EPL; j++) out[j] = (j > 0) ? a[(j + EPL - 1) % EPL] : edge;
}

// ---- Rodrigues update Q <- R(h w) Q  (SURVEY A.2.1) -------------------------
// reference operation order (elastica/_rotations.py:_get_rotation_matrix); also the
// large-rotation fallback of the fast path, kept out of line to keep the hot loop small.
template <typename T> struct Mat9 { T m[9]; };

template <typename T>
__device__ __noinline__ Mat9<T> rotate_directors_ref_val(T a0, T a1, T a2, Mat9<T> Qin) {
  const T *Q = Qin.m;
  Mat9<T> out;
  T *n = out.m;
  T q = a0 * a0 + a1 * a1 + a2 * a2;
  T theta = sqrt_(q);
  T d = theta + T(1e-14);
  T v0 = a0 / d, v1 = a1 / d, v2 = a2 / d;
  T up, cs;
  sincos_(theta, &up, &cs);
  T us = T(1.0) - cs;
  T R00 = T(1.0) - us * (v1 * v1 + v2 * v2);
  T R11 = T(1.0) - us * (v0 * v0 + v2 * v2);
  T R22 = T(1.0) - us * (v0 * v0 + v1 * v1);
  T R01 = up * v2 + us * v0 * v1, R10 = -up * v2 + us * v0 * v1;
  T R02 = -up * v1 + us * v0 * v2, R20 = up * v1 + us * v0 * v2;
  T R12 = up * v0 + us * v1 * v2, R21 = -up * v0 + us * v1 * v2;
#pragma unroll
  for (int m = 0; m < 3; m++) {
    n[0 + m] = R00 * Q[0 + m] + R01 * Q[3 + m] + R02 * Q[6 + m];
    n[3 + m] = R10 * Q[0 + m] + R11 * Q[3 + m] + R12 * Q[6 + m];
    n[6 + m] = R20 * Q[0 + m] + R21 * Q[3 + m] + R22 * Q[6 + m];
  }
  return out;
}
// registers in, registers out: the directors never have their address taken in the hot loop
template <typename T> __device__ __forceinline__ void rotate_directors_ref(T a0, T a1, T a2, T (&Q)[9]) {
  Mat9<T> in;
#pragma unroll
  for (int i = 0; i < 9; i++) in.m[i] = Q[i];
  Mat9<T> out = rotate_directors_ref_val<T>(a0, a1, a2, in);
#pragma unroll
  for (int i = 0; i < 9; i++) Q[i] = out.m[i];
}

// fast path: R = I + A K + B K^2 with A = sin(t)/t, B = (1-cos t)/t^2, applied as Q += D Q.
// `eps` carries the reference's guard: axis = a/(|a| + 1e-14) shortens each half-step
// rotation by 1e-14 rad (2e-14 for a merged full step):  A *= rho, B *= rho^2 with
// rho = |a| / (|a| + eps)  (-> 0 as |a| -> 0, like the reference).  Measured: dropping this
// guard moves the velocity error after 2400 substeps from 2e-11 to 5e-10 (it is a systematic 2e-10
// relative slow-down of every rotation), for a 1 % speed-up — it stays.
template <typename T, bool NARROW = false>
__device__ __forceinline__ void rotate_directors_fast(const PolyCoef<T> &C, T a0, T a1, T a2, T q, T eps,
                                                      T (&Q)[9]) {
  T A, B;
  if (NARROW) sinc_cosc_narrow(C, q, A, B);
  else sinc_cosc(C, q, A, B);
  if (sizeof(T) == 8) {   // a 1e-14 rad shortening is far below FP32 resolution
    // rho = |a| / (|a| + eps) exactly (see rotate_directors_lean: the expansion 1 - eps / sqrt(q + eps^2) is off by tens
    // of per cent of a 1e-14 rad rotation while a rod that starts from rest passes through |a| ~ eps)
    T rho = fma(-eps, rcp_approx(fma(q, rsqrt_approx(q + T(1e-300)), eps)), T(1.0));
    A *= rho;
    B *= rho * rho;
  }
  T Aa0 = A * a0, Aa1 = A * a1, Aa2 = A * a2;
  T Ba0 = B * a0, Ba1 = B * a1, Ba2 = B * a2;
  T D[9];
  D[0] = -fma(Ba1, a1, Ba2 * a2); D[4] = -fma(Ba0, a0, Ba2 * a2); D[8] = -fma(Ba0, a0, Ba1 * a1);
  D[1] = fma(Ba0, a1, Aa2); D[3] = fma(Ba0, a1, -Aa2);
  D[2] = fma(Ba0, a2, -Aa1); D[6] = fma(Ba0, a2, Aa1);
  D[5] = fma(Ba1, a2, Aa0); D[7] = fma(Ba1, a2, -Aa0);
  // Q += D Q in three sweeps over k; inside a sweep the three FMAs of a row share D[i][k] (operand-reuse
  // cache: a DFMA with three fresh register operands issues at 2/3 rate on B200, see DESIGN.md §4)
  T n[9];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) n[3 * i + m] = fma(D[3 * i], Q[m], Q[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) n[3 * i + m] = fma(D[3 * i + 1], Q[3 + m], n[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) n[3 * i + m] = fma(D[3 * i + 2], Q[6 + m], n[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 9; i++) Q[i] = n[i];
}

// -theta / (2 sin(theta + 1e-14)), theta = acos(1 - 2u): the reference's log-map factor
// (elastica/_rotations.py:_inv_rotate), used verbatim by the faithful path and as the
// large-bend fallback of the fast path.
template <typename T> __device__ __noinline__ T bend_factor_ref(T u) {
  T theta = acos_(T(1.0) - T(2.0) * u);
  if (sizeof(T) == 4 && !(theta > T(1e-3))) return T(-0.5) * (T(1.0) + theta * theta * T(1.0 / 6.0));
  return T(-0.5) * theta / sin_(theta + T(1e-14));
}
template <typename T> __device__ __noinline__ T exp_ref(T x) { return exp_(x); }

// numpy's pairwise float64 row sum (np.mean over the contiguous axis): 8 running sums for
// blocks of <= 128 values, recursive halving above (numpy/core/src/umath/loops_utils.h.src).  The halving is unrolled
// into DEPTH levels of distinct functions instead of recursion, so that the stack a kernel needs is known at compile
// time (a recursive call chain runs in the default 1 KB stack, which a 2048-element rod's five levels overflow).
// DEPTH = 6 covers n <= 128 * 2^6 = 8192 (every level halves).
template <int DEPTH = 6, typename T> __device__ __noinline__ double np_pairwise_sum(const T *a, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; i++) r += (double)a[i];
    return r;
  }
  if constexpr (DEPTH > 0) {
    if (n > 128) {
      int n2 = n / 2;
      n2 -= n2 % 8;
      return np_pairwise_sum<DEPTH - 1>(a, n2) + np_pairwise_sum<DEPTH - 1>(a + n2, n - n2);
    }
  }
  double r[8];
  for (int j = 0; j < 8; j++) r[j] = (double)a[j];
  int i;
  for (i = 8; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; j++) r[j] += (double)a[i + j];
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; i++) res += (double)a[i];
  return res;
}

__device__ inline double np_mod(double a, double b) {
  double m = fmod(a, b);
  if (m != 0.0) { if ((b < 0) != (m < 0)) m += b; }
  else m = copysign(0.0, b);
  return m;
}

// SoftPendulum-v0 observation / reward from the (stale) tangents in shared memory
// (reference soft_pendulum.py:149-161, 196-214)
template <typename T>
__device__ inline void soft_pendulum_outputs(const T *tan_smem, int stride, int n, double x0,
                                             double vx0, float prev_action, bool invalid,
                                             float *obs, double *reward, uint8_t *terminated) {
  const double PI = 3.141592653589793;
  double mx = np_pairwise_sum(tan_smem + 0 * stride, n) / (double)n;
  double my = np_pairwise_sum(tan_smem + 1 * stride, n) / (double)n;
  double theta = atan(mx / my);
  theta = np_mod(theta + PI, 2 * PI) - PI;
  obs[0] = (float)x0;
  obs[1] = (float)vx0;
  obs[2] = prev_action;
  obs[3] = (float)theta;
  if (reward) {
    double forward = 0.0, survive = 0.0;
    if (invalid) survive = -50.0;
    else forward = fabs(x0) * 10 + theta * theta;
    *reward = forward - 0.0 + survive;
    *terminated = invalid ? 1 : 0;
  }
}

// SoftPendulum3D-v0 observation / reward (reference soft_pendulum_3d.py:94-104,122-158)
template <typename T>
__device__ inline void soft_pendulum_3d_outputs(const T *tan_smem, int stride, int n, const double x0[3],
                                                const double v0[3], float a0, float a1, double base_x,
                                                double base_y, bool invalid, float *obs, double *reward,
                                                uint8_t *terminated, T *tilt_out) {
  double t[3];
  for (int c = 0; c < 3; c++) t[c] = np_pairwise_sum(tan_smem + c * stride, n) / (double)n;
  double nrm = sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
  double tz = t[2] / nrm;
  tz = fmin(fmax(tz, -1.0), 1.0);
  double tilt = acos(tz);
  for (int c = 0; c < 3; c++) { obs[c] = (float)x0[c]; obs[3 + c] = (float)v0[c]; }
  obs[6] = a0; obs[7] = a1; obs[8] = (float)tilt;
  if (tilt_out) *tilt_out = (T)tilt;
  if (reward) {
    double base_distance = sqrt(base_x * base_x + base_y * base_y);
    float aa = __fadd_rn(__fmul_rn(a0, a0), __fmul_rn(a1, a1));       // np.dot on float32
    float pen = __fmul_rn(0.001f, aa);                                  // 1e-3 * float32 -> float32 (NEP 50)
    double r = -(tilt * tilt + 0.1 * (base_distance * base_distance) + (double)pen);
    *reward = invalid ? -50.0 : r;
    *terminated = invalid ? 1 : 0;
  }
}

template <typename T, int EPL, int MATH, int MINB>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, MINB)
rod_substeps_kernel(const __grid_constant__ RodArgs<T> A) {
  __shared__ T tan_smem[WARPS_PER_CTA][3 * 32 * EPL];
  const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  const int env = blockIdx.x * WARPS_PER_CTA + wic;
  if (env >= A.n_env) return;
  const int n = A.n_elem, stride = A.stride;
  T *st = A.state + (size_t)env * N_FIELDS * stride;

  T x[3][EPL], v[3][EPL], Q[9][EPL], w[3][EPL];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    load_row<T, EPL>(st + (F_POS + c) * stride, lane, x[c]);
    load_row<T, EPL>(st + (F_VEL + c) * stride, lane, v[c]);
    load_row<T, EPL>(st + (F_OMEGA + c) * stride, lane, w[c]);
  }
#pragma unroll
  for (int c = 0; c < 9; c++) load_row<T, EPL>(st + (F_DIR + c) * stride, lane, Q[c]);

  // Slots past the rod end hold a benign state (x = v = w = 0, Q = I) that never changes:
  // their time-step multipliers are zero, so no per-update selects are needed.
  bool elem_ok[EPL], node_ok[EPL], vor_ok[EPL];
  T dtim[EPL], gmask[EPL], dte[EPL], gam[EPL];
  load_row<T, EPL>(st + F_GAMMA * stride, lane, gam);
#pragma unroll
  for (int j = 0; j < EPL; j++) {
    int k = lane * EPL + j;
    elem_ok[j] = k < n;
    node_ok[j] = k <= n;
    vor_ok[j] = k < n - 1;
    dtim[j] = node_ok[j] ? A.dt_inv_mass * ((k == 0 || k == n) ? T(2) : T(1)) : T(0);
    gmask[j] = node_ok[j] ? T(1) : T(0);
    dte[j] = elem_ok[j] ? A.dt : T(0);
  }
  // per-env anchors and actuation (only lane 0 / node 0 uses them)
  const T *bc = A.bc + (size_t)env * BC_DIM;
  T act0 = T(0), base_px = T(0), base_py = T(0), base_vx = T(0), base_vy = T(0);
  if (A.action_dim > 0) act0 = (T)A.action[(size_t)env * A.action_dim];
  if (A.bc_kind == BC_MOVING_BASE) {
    const T *aux = A.aux + (size_t)env * AUX_DIM;
    base_px = aux[0]; base_py = aux[1]; base_vx = aux[3]; base_vy = aux[4];
  }

  auto constrain_values = [&]() {
    if (lane == 0) {
      if (A.bc_kind == BC_PENDULUM_SLIDER) {
        x[1][0] = bc[1]; x[2][0] = bc[2];
#pragma unroll
        for (int m = 0; m < 3; m++) { Q[0 + m][0] = bc[3 + m]; Q[6 + m][0] = bc[9 + m]; }
      } else if (A.bc_kind == BC_ONE_END_FIXED) {
#pragma unroll
        for (int c = 0; c < 3; c++) x[c][0] = bc[c];
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c][0] = bc[3 + c];
      } else if (A.bc_kind == BC_MOVING_BASE) {
        x[0][0] = base_px; x[1][0] = base_py; x[2][0] = bc[2];
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c][0] = bc[3 + c];
      }
    }
  };
  auto constrain_rates = [&]() {
    if (lane == 0) {
      if (A.bc_kind == BC_PENDULUM_SLIDER) {
        v[1][0] = T(0); v[2][0] = T(0); w[0][0] = T(0); w[2][0] = T(0);
      } else if (A.bc_kind == BC_ONE_END_FIXED) {
#pragma unroll
        for (int c = 0; c < 3; c++) { v[c][0] = T(0); w[c][0] = T(0); }
      } else if (A.bc_kind == BC_MOVING_BASE) {
        v[0][0] = base_vx; v[1][0] = base_vy; v[2][0] = T(0);
#pragma unroll
        for (int c = 0; c < 3; c++) w[c][0] = T(0);
      }
    }
  };
  // x += hh v ; Q <- R(hh w) Q.  In the fast path hh is dt/2 (first/last update of the
  // launch) or dt: the half step that ends substep s and the one that starts s+1 use the
  // same v, w and compose exactly (same rotation axis; every BC of this build overwrites
  // its constrained components), so they are merged into one update.
  auto kinematic = [&](T hh, T eps) {
    T a[3][EPL], q[EPL];
    bool fast = (MATH == MATH_FAST);
#pragma unroll
    for (int j = 0; j < EPL; j++) {
#pragma unroll
      for (int c = 0; c < 3; c++) {
        x[c][j] = fma(hh, v[c][j], x[c][j]);
        a[c][j] = hh * w[c][j];
      }
      q[j] = fma(a[2][j], a[2][j], fma(a[1][j], a[1][j], a[0][j] * a[0][j]));
      // The base element is excluded from the vote when a BC owns its directors: every BC of
      // this build overwrites the rows that R changes (ONE_END_FIXED / MOVING_BASE: all of Q;
      // PENDULUM_SLIDER: rows d1,d3, and its rate constraint keeps w = (0,w1,0) so row d2 is
      // exactly invariant: D10 = D11 = D12 = 0).  The reference env lets w1 of that element
      // grow without bound (nothing restores it), which must not push the warp off the fast path.
      const bool owned_by_bc = (j == 0) && (lane == 0) && (A.bc_kind != BC_FREE);
      if (!(q[j] <= T(kSmallRotQ)) && !owned_by_bc) fast = false;
    }
    if (MATH == MATH_FAST) fast = !__any_sync(FULL, !fast);
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      T Qj[9];
#pragma unroll
      for (int c = 0; c < 9; c++) Qj[c] = Q[c][j];
      if (fast) rotate_directors_fast<T>(A.poly, a[0][j], a[1][j], a[2][j], q[j], eps, Qj);
      else rotate_directors_ref<T>(a[0][j], a[1][j], a[2][j], Qj);
#pragma unroll
      for (int c = 0; c < 9; c++) Q[c][j] = Qj[c];
    }
  };

  const T h = A.half_dt, dt = A.dt;
  if (MATH == MATH_FAST && A.n_substeps > 0) { kinematic(h, T(1e-14)); constrain_values(); }

#pragma unroll 1
  for (int s = 0; s < A.n_substeps; s++) {
    const bool last = (s == A.n_substeps - 1);
    if (MATH != MATH_FAST) { kinematic(h, T(1e-14)); constrain_values(); }

    // ---------------- geometry, shear/stretch strain, internal force ----------
    T xn[3][EPL], vn[3][EPL];
#pragma unroll
    for (int c = 0; c < 3; c++) { shift_next<T, EPL>(x[c], xn[c]); shift_next<T, EPL>(v[c], vn[c]); }
    T lg[EPL], e[EPL], inv_e[EPL], edot[EPL];
    T tng[3][EPL], sig[3][EPL], nst[3][EPL], Qt[3][EPL], sfl[3][EPL];
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      T dx[3], dv[3];
#pragma unroll
      for (int c = 0; c < 3; c++) { dx[c] = xn[c][j] - x[c][j]; dv[c] = vn[c][j] - v[c][j]; }
      if (!elem_ok[j]) dx[2] = A.rest_len;  // keeps every quantity of a padding slot finite
      T t[3];
      if (MATH == MATH_FAST) {
        T l2 = dot3(dx, dx);
        T il = rsqrt_nr(l2);
        T l = l2 * il;
        lg[j] = l + T(1e-14);                     // reference guard on the length
        T ilg = fma(T(-1e-14) * il, il, il);      // 1/(l + 1e-14) to first order in 1e-14/l
#pragma unroll
        for (int c = 0; c < 3; c++) t[c] = dx[c] * ilg;
        e[j] = lg[j] * A.inv_rest_len * gam[j];
        inv_e[j] = A.rest_len * ilg;
        edot[j] = dot3(dx, dv) * (ilg * A.inv_rest_len);   // = t . dv / l0
      } else {
        lg[j] = sqrt_(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]) + T(1e-14);
#pragma unroll
        for (int c = 0; c < 3; c++) t[c] = dx[c] / lg[j];
        e[j] = lg[j] / A.rest_len * gam[j];
        inv_e[j] = T(1.0) / e[j];
        // r.v terms exactly as elastica/rod/cosserat_rod.py:_compute_dilatation_rate
        T xk[3] = {x[0][j], x[1][j], x[2][j]}, vk[3] = {v[0][j], v[1][j], v[2][j]};
        T xk1[3] = {xn[0][j], xn[1][j], xn[2][j]}, vk1[3] = {vn[0][j], vn[1][j], vn[2][j]};
        T rv0 = xk[0] * vk[0] + xk[1] * vk[1] + xk[2] * vk[2];
        T rv1 = xk1[0] * vk1[0] + xk1[1] * vk1[1] + xk1[2] * vk1[2];
        T rp1v = xk1[0] * vk[0] + xk1[1] * vk[1] + xk1[2] * vk[2];
        T rvp1 = xk[0] * vk1[0] + xk[1] * vk1[1] + xk[2] * vk1[2];
        edot[j] = (rv0 + rv1 - rvp1 - rp1v) / lg[j] / A.rest_len;
      }
#pragma unroll
      for (int i = 0; i < 3; i++) {
        tng[i][j] = t[i];
        T qt = (MATH == MATH_FAST)
                   ? fma(Q[3 * i + 2][j], t[2], fma(Q[3 * i + 1][j], t[1], Q[3 * i][j] * t[0]))
                   : (Q[3 * i][j] * t[0] + Q[3 * i + 1][j] * t[1] + Q[3 * i + 2][j] * t[2]);
        Qt[i][j] = qt;
        sig[i][j] = e[j] * qt - (i == 2 ? T(1) : T(0));
        nst[i][j] = A.S[i] * sig[i][j];
      }
#pragma unroll
      for (int i = 0; i < 3; i++) {
        T sv = (MATH == MATH_FAST)
                   ? fma(Q[6 + i][j], nst[2][j], fma(Q[3 + i][j], nst[1][j], Q[i][j] * nst[0][j])) * inv_e[j]
                   : (Q[i][j] * nst[0][j] + Q[3 + i][j] * nst[1][j] + Q[6 + i][j] * nst[2][j]) / e[j];
        sfl[i][j] = elem_ok[j] ? sv : T(0);
      }
    }
    T f[3][EPL];
#pragma unroll
    for (int i = 0; i < 3; i++) {
      T sp[EPL];
      shift_prev<T, EPL>(sfl[i], lane, sp);
#pragma unroll
      for (int j = 0; j < EPL; j++) f[i][j] = sfl[i][j] - sp[j];
    }

    // ---------------- curvature, bending couple, internal torque --------------
    T Qn[9][EPL], lgn[EPL];
#pragma unroll
    for (int c = 0; c < 9; c++) shift_next<T, EPL>(Q[c], Qn[c]);
    shift_next<T, EPL>(lg, lgn);
    T kap[3][EPL], mcp[3][EPL], ccp[3][EPL];  // kappa ; tau/eps^3 ; (kappa x tau) D / eps^3
    bool bend_fast = (MATH == MATH_FAST);
    T uu[EPL], vec[3][EPL];
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      // Rm = Q_{k+1} Q_k^T ; vec = axial(Rm - Rm^T) ; trace
      auto rm = [&](int a, int b) {
        return (MATH == MATH_FAST)
                   ? fma(Qn[3 * a + 2][j], Q[3 * b + 2][j], fma(Qn[3 * a + 1][j], Q[3 * b + 1][j], Qn[3 * a][j] * Q[3 * b][j]))
                   : (Qn[3 * a][j] * Q[3 * b][j] + Qn[3 * a + 1][j] * Q[3 * b + 1][j] + Qn[3 * a + 2][j] * Q[3 * b + 2][j]);
      };
      vec[0][j] = rm(2, 1) - rm(1, 2);
      vec[1][j] = rm(0, 2) - rm(2, 0);
      vec[2][j] = rm(1, 0) - rm(0, 1);
      T tr = rm(0, 0) + rm(1, 1) + rm(2, 2);
      // 1 - cos(theta_ref) with the reference's 1e-10 guard, halved: u = sin^2(theta_ref/2)
      T u = T(0.5) * ((T(1.5) - T(0.5) * tr) + T(1e-10));
      uu[j] = vor_ok[j] ? u : T(5e-11);
      if (!(uu[j] <= T(kSmallBendU))) bend_fast = false;
    }
    if (MATH == MATH_FAST) bend_fast = !__any_sync(FULL, !bend_fast);
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      T fac;
      if (bend_fast) {
        // -theta/(2 sin(theta + 1e-14)) = -g(u)/2 * (1 - 1e-14 cot(theta)),
        // cot(theta) = (1 - 2u) / sqrt(4u(1-u)); u >= 5e-11 by the 1e-10 guard, so no singularity
        T u = uu[j];
        T cot = fma(T(-2.0), u, T(1.0)) * rsqrt_approx(T(4.0) * u * (T(1.0) - u));
        fac = T(-0.5) * theta_over_sin(A.poly, u) * fma(T(-1e-14), cot, T(1.0));
      } else {
        fac = bend_factor_ref<T>(uu[j]);
      }
      T tau[3], kxt[3], kp[3];
#pragma unroll
      for (int i = 0; i < 3; i++) {
        kp[i] = (MATH == MATH_FAST) ? vec[i][j] * (fac * A.inv_rest_vor) : (vec[i][j] * fac) / A.rest_vor;
        kap[i][j] = kp[i];
        tau[i] = A.B[i] * kp[i];
      }
      cross3(kp, tau, kxt);
      T eps = (MATH == MATH_FAST) ? (T(0.5) * (lgn[j] + lg[j])) * A.inv_rest_vor
                                  : (T(0.5) * (lgn[j] + lg[j])) / A.rest_vor;
      T ie3 = (MATH == MATH_FAST) ? rcp_nr(eps * eps * eps) : T(1.0) / (eps * eps * eps);
      if (!vor_ok[j]) ie3 = T(0);
#pragma unroll
      for (int i = 0; i < 3; i++) {
        mcp[i][j] = tau[i] * ie3;
        ccp[i][j] = kxt[i] * (A.rest_vor * ie3);
      }
    }
    T tq[3][EPL];
#pragma unroll
    for (int i = 0; i < 3; i++) {
      if (MATH == MATH_FAST) {
        // T_k = (m_k - m_{k-1}) + (c_k + c_{k-1})/2 = P_k + N_{k-1}; one shuffle instead of two
        T P[EPL], N[EPL], Np[EPL];
#pragma unroll
        for (int j = 0; j < EPL; j++) {
          P[j] = fma(T(0.5), ccp[i][j], mcp[i][j]);
          N[j] = fma(T(0.5), ccp[i][j], -mcp[i][j]);
        }
        shift_prev<T, EPL>(N, lane, Np);
#pragma unroll
        for (int j = 0; j < EPL; j++) tq[i][j] = P[j] + Np[j];
      } else {
        T mp[EPL], cp[EPL];
        shift_prev<T, EPL>(mcp[i], lane, mp);
        shift_prev<T, EPL>(ccp[i], lane, cp);
#pragma unroll
        for (int j = 0; j < EPL; j++) tq[i][j] = (mcp[i][j] - mp[j]) + T(0.5) * (ccp[i][j] + cp[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      T qt[3] = {Qt[0][j], Qt[1][j], Qt[2][j]}, ns[3] = {nst[0][j], nst[1][j], nst[2][j]};
      T wj[3] = {w[0][j], w[1][j], w[2][j]};
      T ssc[3], jw[3], lt[3];
      cross3(qt, ns, ssc);
#pragma unroll
      for (int i = 0; i < 3; i++) jw[i] = (MATH == MATH_FAST) ? (A.J[i] * wj[i]) * inv_e[j] : (A.J[i] * wj[i]) / e[j];
      cross3(jw, wj, lt);
      T ede = edot[j] * inv_e[j];
#pragma unroll
      for (int i = 0; i < 3; i++) {
        if (MATH == MATH_FAST) tq[i][j] = fma(jw[i], ede, fma(ssc[i], A.rest_len, tq[i][j]) + lt[i]);
        else tq[i][j] = tq[i][j] + ssc[i] * A.rest_len + lt[i] + jw[i] * edot[j] / e[j];
      }
    }

    // stale observables of the reference (tangents/kappa/sigma/dilatation are only
    // refreshed here, half a kinematic step before the final state: SURVEY A.6)
    if (last) {
#pragma unroll
      for (int i = 0; i < 3; i++) {
        store_row<T, EPL>(st + (F_TAN + i) * stride, lane, tng[i]);
        store_row<T, EPL>(st + (F_KAPPA + i) * stride, lane, kap[i]);
        store_row<T, EPL>(st + (F_SIGMA + i) * stride, lane, sig[i]);
        store_row<T, EPL>(&tan_smem[wic][i * 32 * EPL], lane, tng[i]);
      }
      store_row<T, EPL>(st + F_DIL * stride, lane, e);
    }

    // ---------------- external loads + dynamic step ---------------------------
#pragma unroll
    for (int j = 0; j < EPL; j++) {
      const bool base_node = (lane == 0 && j == 0);
      if (MATH == MATH_FAST) {
#pragma unroll
        for (int i = 0; i < 3; i++) {
          T fi = f[i][j], gd = A.gdt[i];
          if (i == 0 && A.point_force && base_node) { fi += act0; gd = T(0); }
          v[i][j] = fma(gmask[j], gd, fma(fi, dtim[j], v[i][j]));
          w[i][j] = fma(dte[j] * e[j], A.Jinv[i] * tq[i][j], w[i][j]);
        }
      } else {
        T m = ((lane * EPL + j) == 0 || (lane * EPL + j) == n) ? A.mass * T(0.5) : A.mass;
#pragma unroll
        for (int i = 0; i < 3; i++) {
          T fe = A.g[i] * m;
          if (i == 0 && A.point_force && base_node) fe = act0;
          T acc = (f[i][j] + fe) / m;
          v[i][j] = node_ok[j] ? v[i][j] + dt * acc : v[i][j];
          T alpha = (A.Jinv[i] * tq[i][j]) * e[j];
          w[i][j] = elem_ok[j] ? w[i][j] + dt * alpha : w[i][j];
        }
      }
    }

    // ---------------- rate constraints and dissipation -------------------------
    auto dampen = [&]() {
      if (A.damping_on) {
        bool ef = (MATH == MATH_FAST);
        T z[3][EPL];
        if (MATH == MATH_FAST) {
#pragma unroll
          for (int j = 0; j < EPL; j++)
#pragma unroll
            for (int i = 0; i < 3; i++) {
              z[i][j] = (e[j] - T(1)) * A.logc_w[i];
              if (!(fabs_(z[i][j]) <= T(kSmallExpZ))) ef = false;
            }
          ef = !__any_sync(FULL, !ef);
        }
#pragma unroll
        for (int j = 0; j < EPL; j++)
#pragma unroll
          for (int i = 0; i < 3; i++) {
            v[i][j] = v[i][j] * A.c_v;
            T cw;
            if (ef) cw = A.c_w[i] * exp_small(A.poly, z[i][j]);
            else if (MATH == MATH_FAST) cw = exp_ref<T>(e[j] * A.logc_w[i]);
            else cw = pow_(A.c_w[i], e[j]);
            w[i][j] = w[i][j] * cw;
          }
      }
    };
    if (A.damp_first) { dampen(); constrain_rates(); }
    else { constrain_rates(); dampen(); }

    if (MATH == MATH_FAST) kinematic(last ? h : dt, last ? T(1e-14) : T(2e-14));
    else kinematic(h, T(1e-14));
    constrain_values();
  }

  // ---------------- write back + NaN guard + model outputs ---------------------
#pragma unroll
  for (int c = 0; c < 3; c++) {
    store_row<T, EPL>(st + (F_POS + c) * stride, lane, x[c]);
    store_row<T, EPL>(st + (F_VEL + c) * stride, lane, v[c]);
    store_row<T, EPL>(st + (F_OMEGA + c) * stride, lane, w[c]);
  }
#pragma unroll
  for (int c = 0; c < 9; c++) store_row<T, EPL>(st + (F_DIR + c) * stride, lane, Q[c]);
  bool invalid_any = false;
#pragma unroll
  for (int j = 0; j < EPL; j++)
#pragma unroll
    for (int c = 0; c < 3; c++)
      if (node_ok[j] && (x[c][j] != x[c][j] || v[c][j] != v[c][j])) invalid_any = true;
  invalid_any = __any_sync(FULL, invalid_any);
  __syncwarp();
  if (lane == 0) {
    if (A.model == MODEL_SOFT_PENDULUM) {
      soft_pendulum_outputs<T>(tan_smem[wic], 32 * EPL, n, (double)x[0][0], (double)v[0][0],
                               (float)act0, invalid_any, A.obs + (size_t)env * A.obs_dim,
                               A.reward + env, A.terminated + env);
    } else {
      A.reward[env] = 0.0;
      A.terminated[env] = invalid_any ? 1 : 0;
    }
  }
  if (A.model == MODEL_ROD) {
    // plain rod: obs = tip position (3) + tip velocity (3); node n lives at lane n/EPL slot n%EPL
#pragma unroll
    for (int j = 0; j < EPL; j++)
      if (lane * EPL + j == n) {
        float *o = A.obs + (size_t)env * A.obs_dim;
        for (int c = 0; c < 3; c++) { o[c] = (float)x[c][j]; o[3 + c] = (float)v[c][j]; }
      }
  }
}

// ---- reset: CosseratRod.straight_rod + finalize-time anchors (SURVEY A.1, B-7) ----
template <typename T>
__global__ void rod_reset_kernel(T *state, T *bc, T *aux, const int32_t *env_idx, int n_reset,
                                 const double *init, int n, int stride, double base_length, int n_rod,
                                 int init_dim, double *muscle, int muscle_dim, double *spline, int spline_dim) {
  // one block per rod to rebuild: block r -> env slot r / n_rod, rod r % n_rod
  int r = blockIdx.x;
  if (r >= n_reset * n_rod) return;
  int e = r / n_rod, arm = r - e * n_rod;
  int env = (env_idx ? env_idx[e] : e) * n_rod + arm;   // global rod slot
  const double *ip = init + (size_t)e * init_dim + (size_t)arm * 9;
  double start[3] = {ip[0], ip[1], ip[2]}, dir[3] = {ip[3], ip[4], ip[5]}, nor[3] = {ip[6], ip[7], ip[8]};
  double nn = sqrt(nor[0] * nor[0] + nor[1] * nor[1] + nor[2] * nor[2]);
  for (int c = 0; c < 3; c++) nor[c] = nor[c] / nn;
  T *st = state + (size_t)env * N_FIELDS * stride;
  // np.linspace(start, end, n+1): k*step + start, last point = end exactly
  double step[3], end[3];
  for (int c = 0; c < 3; c++) {
    end[c] = __dadd_rn(start[c], __dmul_rn(dir[c], base_length));
    step[c] = (end[c] - start[c]) / (double)n;
  }
  auto pos = [&](int c, int k) { return k == n ? end[c] : __dadd_rn(__dmul_rn((double)k, step[c]), start[c]); };
  for (int k = threadIdx.x; k < stride; k += blockDim.x) {
    double xk[3] = {0, 0, 0}, t[3] = {0, 0, 1}, Qk[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    double tang[3] = {0, 0, 0}, sg[3] = {0, 0, 0}, dil = 1.0, gam = 1.0;
    if (k <= n) for (int c = 0; c < 3; c++) xk[c] = pos(c, k);
    if (k < n) {
      double d[3];
      for (int c = 0; c < 3; c++) d[c] = pos(c, k + 1) - xk[c];
      double rl = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(d[0], d[0]), __dmul_rn(d[1], d[1])), __dmul_rn(d[2], d[2])));
      for (int c = 0; c < 3; c++) t[c] = d[c] / rl;
      gam = (base_length / (double)n) / rl;
      for (int c = 0; c < 3; c++) { Qk[c] = nor[c]; Qk[6 + c] = t[c]; }
      Qk[3] = __dadd_rn(__dmul_rn(t[1], nor[2]), -__dmul_rn(t[2], nor[1]));
      Qk[4] = __dadd_rn(__dmul_rn(t[2], nor[0]), -__dmul_rn(t[0], nor[2]));
      Qk[5] = __dadd_rn(__dmul_rn(t[0], nor[1]), -__dmul_rn(t[1], nor[0]));
      double lg = rl + 1e-14;
      for (int c = 0; c < 3; c++) tang[c] = d[c] / lg;
      dil = lg / rl;
      for (int i = 0; i < 3; i++) {
        double qt = __dadd_rn(__dadd_rn(__dmul_rn(Qk[3 * i], tang[0]), __dmul_rn(Qk[3 * i + 1], tang[1])),
                              __dmul_rn(Qk[3 * i + 2], tang[2]));
        sg[i] = __dmul_rn(dil, qt) - (i == 2 ? 1.0 : 0.0);
      }
    }
    for (int c = 0; c < 3; c++) {
      st[(F_POS + c) * stride + k] = (T)xk[c];
      st[(F_VEL + c) * stride + k] = T(0);
      st[(F_OMEGA + c) * stride + k] = T(0);
      st[(F_TAN + c) * stride + k] = (T)tang[c];
      st[(F_KAPPA + c) * stride + k] = T(0);
      st[(F_SIGMA + c) * stride + k] = (T)sg[c];
    }
    for (int c = 0; c < 9; c++) st[(F_DIR + c) * stride + k] = (T)Qk[c];
    st[F_DIL * stride + k] = (T)dil;
    st[F_GAMMA * stride + k] = (T)gam;
    for (int c = 0; c < 3; c++) st[(F_EDGE + c) * stride + k] = (T)((k < n) ? pos(c, k + 1) - xk[c] : 0.0);
    if (k == 0) {
      T *b = bc + (size_t)env * BC_DIM;
      for (int c = 0; c < 3; c++) b[c] = (T)xk[c];
      for (int c = 0; c < 9; c++) b[3 + c] = (T)Qk[c];
      if (arm == 0) {   // aux is per environment, not per rod
        T *a = aux + (size_t)(env / n_rod) * AUX_DIM;
        for (int c = 0; c < AUX_DIM; c++) a[c] = T(0);
        if (muscle) muscle[(size_t)(env / n_rod) * muscle_dim] = 0.0;   // simulation time restarts
        if (spline) {   // a fresh forcing instance: zero targets / cached points / flags / magnitudes
          double *sp = spline + (size_t)(env / n_rod) * spline_dim;
          for (int c = 0; c < spline_dim; c++) sp[c] = 0.0;
        }
      }
    }
  }
}

// Cylinder(start, direction, normal, length, ...) of the octopus head (SURVEY D.1): centre of mass at
// start + direction L/2, rows of Q = normal, direction x normal, direction; BodyBoundaryCondition pins z.
template <typename T>
__global__ void head_reset_kernel(T *head, const int32_t *env_idx, int n_reset, const double *init,
                                  int init_dim, int n_rod, double head_length) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_reset) return;
  int env = env_idx ? env_idx[e] : e;
  const double *ip = init + (size_t)e * init_dim + (size_t)n_rod * 9;
  T *h = head + (size_t)env * HEAD_DIM;
  double d[3] = {ip[3], ip[4], ip[5]}, nr[3] = {ip[6], ip[7], ip[8]};
  for (int c = 0; c < 3; c++) { h[c] = (T)(ip[c] + d[c] * head_length / 2); h[3 + c] = T(0); h[15 + c] = T(0); }
  double b[3] = {d[1] * nr[2] - d[2] * nr[1], d[2] * nr[0] - d[0] * nr[2], d[0] * nr[1] - d[1] * nr[0]};
  for (int c = 0; c < 3; c++) { h[6 + c] = (T)nr[c]; h[9 + c] = (T)b[c]; h[12 + c] = (T)d[c]; }
  h[18] = h[2];
  h[19] = T(0);
}

// observation of the current state without stepping (reset obs; soft_pendulum.py:149-161)
template <typename T>
__global__ void rod_observe_kernel(const T *state, const float *prev_action, float *obs, int n_env,
                                   int n, int stride, int model, int action_dim, int obs_dim) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_env) return;
  const T *st = state + (size_t)env * N_FIELDS * stride;
  float pa = (prev_action && action_dim > 0) ? prev_action[(size_t)env * action_dim] : 0.0f;
  if (model == MODEL_SOFT_PENDULUM) {
    soft_pendulum_outputs<T>(st + F_TAN * stride, stride, n, (double)st[F_POS * stride],
                             (double)st[F_VEL * stride], pa, false, obs + (size_t)env * obs_dim,
                             nullptr, nullptr);
  } else if (model == MODEL_SOFT_PENDULUM_3D) {
    double x0[3], v0[3];
    for (int c = 0; c < 3; c++) { x0[c] = (double)st[(F_POS + c) * stride]; v0[c] = (double)st[(F_VEL + c) * stride]; }
    float a0 = prev_action ? prev_action[(size_t)env * action_dim] : 0.0f;
    float a1 = prev_action ? prev_action[(size_t)env * action_dim + 1] : 0.0f;
    soft_pendulum_3d_outputs<T>(st + F_TAN * stride, stride, n, x0, v0, a0, a1, 0.0, 0.0, false,
                                obs + (size_t)env * obs_dim, nullptr, nullptr, (T *)nullptr);
  } else {
    float *o = obs + (size_t)env * obs_dim;
    for (int c = 0; c < 3; c++) {
      o[c] = (float)st[(F_POS + c) * stride + n];
      o[3 + c] = (float)st[(F_VEL + c) * stride + n];
    }
  }
}

}  // namespace sr
