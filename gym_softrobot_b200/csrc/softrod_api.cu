// softrod_api.cu — C-ABI (include/softrod.h) over the fused rod kernels.
//
// Host side of the boundary that replaces
//   `time = PositionVerlet().step(simulator, time, dt)` x step_skip
//   (/root/reference/gym_softrobot/envs/soft_pendulum/soft_pendulum.py:183-184)
// and `CosseratRod.straight_rod(...)` + plugin registration
//   (/root/reference/gym_softrobot/envs/soft_pendulum/build.py:54-113).
// Rod constants follow SURVEY.md Appendix A.1 / A.4 in FP64 on the host.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/softrod.h"
#include "copy_kernels.cuh"
#include "launch.cuh"
#include "util_kernels.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}

#define SR_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return fail(SR_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

}  // namespace

struct sr_handle {
  sr_config cfg;
  int epl = 0, stride = 0, obs_dim = 0, action_dim = 0;
  size_t elem_size = 8;
  void *state = nullptr, *bc = nullptr, *aux = nullptr, *rest_kappa = nullptr, *head = nullptr;
  double *muscle = nullptr; int muscle_dim = 0;
  double *spline = nullptr, *spline_tab = nullptr; int spline_dim = 0;
  void *sucker = nullptr, *ext_force = nullptr, *ext_couple = nullptr, *elem_tab = nullptr;
  int32_t *sucker_idx = nullptr;   // per-rod ControllableFixConstraint index (python indexing)
  void *tm_act = nullptr;          // per-rod TransverseMuscle activation
  double *mus_act = nullptr;       // per-element activations of the three muscle layers [n_rods][3][n_elem]
  double *msucker = nullptr;       // ratios of the fixed-index ControllableFixConstraints [n_rods][3]
  int *redo = nullptr;   // per-env flags of the fast-only / fallback kernel pair
  unsigned long long *redo_count = nullptr, *h_redo_count = nullptr, pair_last_count = 0;   // counts: see count_redo (lean kernel)
  cudaEvent_t pair_event = nullptr; bool pair_copy_pending = false;
  long long pair_steps = 0, pair_off_until = 0, pair_steps_at_copy = 0, pair_steps_at_prev_copy = 0;
  unsigned long long planar_last_count = 0; long long planar_off_until = 0;   // the planar model's own window
  int n_rod = 1, init_dim = 9;
  sr::RodArgs<double> a64;
  sr::RodArgs<float> a32;
  // staging for the host-buffer entry points
  float *d_action = nullptr, *d_obs = nullptr, *h_action = nullptr, *h_obs = nullptr;
  double *d_reward = nullptr, *h_reward = nullptr, *d_init = nullptr, *h_init = nullptr;
  uint8_t *d_term = nullptr, *h_term = nullptr;
  int32_t *d_idx = nullptr;
  cudaStream_t own_stream = nullptr;
  int64_t launches = 0;
  // stream-K schedule of the lean kernel: SM count, slots the hand-over scratch and flags are allocated for
  int sk_sms = 0, sk_slots = 0; void *sk_scratch = nullptr; int *sk_flag = nullptr;
  long long sk_slot_threads = 0;   // slots x CTA threads sk_scratch holds (LEAN_SCR_FOLD rows each)
  void *copy_stage = nullptr; size_t copy_stage_bytes = 0;   // sr_copy_envs within one handle: the source rows, gathered
};

namespace {

// SURVEY A.1 / A.4: constants of a uniform straight rod, FP64 on the host.
template <typename T> void fill_args(const sr_config &c, int stride, sr::RodArgs<T> &A) {
  const double PI = 3.141592653589793;
  const int n = c.n_elem;
  const double rl = c.base_length / n;
  const double r = c.base_radius;
  const double A0 = PI * r * r;
  const double I1 = A0 * A0 / (4.0 * PI), I2 = I1, I3 = 2.0 * I2;
  const double E = c.youngs_modulus;
  const double G = c.shear_modulus > 0.0 ? c.shear_modulus : E / (2.0 * (1.0 + 0.5));
  const double ac = 27.0 / 28.0;
  const double rho_l = c.density * rl;
  const double J[3] = {I1 * rho_l, I2 * rho_l, I3 * rho_l};
  const double S[3] = {ac * G * A0, ac * G * A0, E * A0};
  const double Bv[3] = {E * I1, E * I2, G * I3};  // uniform rod: Voronoi average = element value
  const double volume = PI * (r * r) * rl;
  const double mass = c.density * volume;  // interior node; end nodes carry mass/2
  memset(&A, 0, sizeof(A));
  A.n_env = c.n_env; A.n_elem = n; A.stride = stride;
  A.bc_kind = c.bc_kind; A.model = c.model; A.point_force = c.point_force_on_base;
  A.damp_first = c.damping_before_constraints; A.damping_on = c.damping_constant >= 0.0;
  A.laplace_order = c.laplace_filter_order;
  A.dt = (T)c.dt; A.half_dt = (T)(0.5 * c.dt);
  A.rest_len = (T)rl; A.inv_rest_len = (T)(1.0 / rl);
  A.rest_vor = (T)rl; A.inv_rest_vor = (T)(1.0 / rl);
  for (int i = 0; i < 3; i++) {
    A.S[i] = (T)S[i]; A.B[i] = (T)Bv[i]; A.J[i] = (T)J[i]; A.Jinv[i] = (T)(1.0 / J[i]);
    A.g[i] = (T)c.gravity[i]; A.gdt[i] = (T)(c.gravity[i] * c.dt);
  }
  A.mass = (T)mass; A.inv_mass = (T)(1.0 / mass); A.dt_inv_mass = (T)(c.dt / mass);
  for (int i = 0; i < 3; i++) {
    A.S_over_l[i] = (T)(S[i] / rl);
    A.gdt_cv[i] = (T)(c.gravity[i] * c.dt * (c.damping_constant >= 0.0 ? exp(-c.damping_constant * c.dt) : 1.0));
  }
  A.base_limit = (T)c.base_limit;
  A.inv_move_period = (T)(c.base_move_period > 0.0 ? 1.0 / c.base_move_period : 0.0);
  A.base_step_f32 = (float)c.base_step;
  A.rest_kappa = nullptr;
  A.n_rod = c.n_rod_per_env > 1 ? c.n_rod_per_env : 1; A.has_head = c.has_head; A.head = nullptr;
  A.sk_rodsync = 1;
  A.joint_k = (T)c.joint_k; A.joint_nu = (T)c.joint_nu; A.joint_kt = (T)c.joint_kt; A.joint_radius = (T)c.joint_radius;
  for (int a = 0; a < 16; a++) {   // z_rotation(): theta = angle / 180 * pi
    double th = c.joint_angle_deg[a] / 180.0 * PI;
    A.joint_cs[a][0] = (T)cos(th); A.joint_cs[a][1] = (T)sin(th);
  }
  if (c.has_head) {   // Cylinder (SURVEY D.1): m = rho pi r^2 L ; J = diag(I0) rho L, I0 = (A^2/4pi, A^2/4pi, A^2/2pi)
    const double Ah = PI * c.head_radius * c.head_radius, Ih = Ah * Ah / (4.0 * PI);
    const double mh = PI * c.head_radius * c.head_radius * c.head_length * c.head_density;
    const double Jh[3] = {Ih * c.head_density * c.head_length, Ih * c.head_density * c.head_length,
                          2.0 * Ih * c.head_density * c.head_length};
    A.head_dt_inv_mass = (T)(c.dt / mh);
    for (int i = 0; i < 3; i++) { A.head_J[i] = (T)Jh[i]; A.head_Jinv[i] = (T)(1.0 / Jh[i]); }
  }
  A.contact_on = c.contact_on; A.contact_before_forcing = c.contact_before_forcing;
  {
    double nn = sqrt(c.plane_normal[0] * c.plane_normal[0] + c.plane_normal[1] * c.plane_normal[1] + c.plane_normal[2] * c.plane_normal[2]);
    double N[3] = {0.0, 0.0, 1.0};
    for (int i = 0; i < 3; i++) {
      if (nn > 0) N[i] = c.plane_normal[i] / nn;
      A.plane_origin[i] = (T)c.plane_origin[i];
      A.plane_normal[i] = (T)N[i];
      A.kin_mu[i] = (T)c.kinetic_mu[i]; A.stat_mu[i] = (T)c.static_mu[i];
    }
    // internal frame of the contact models: z = plane normal.  Rotation taking N to z about N x z (Rodrigues); its
    // entries are exactly 0 / +-1 for an axis-aligned normal, so the frame change is then a signed permutation.
    double R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    A.rot_on = 0;
    if (c.contact_on && !(N[0] == 0.0 && N[1] == 0.0 && N[2] == 1.0)) {
      A.rot_on = 1;
      const double vx = N[1], vy = -N[0], s2 = vx * vx + vy * vy, cz = N[2];   // v = N x z = (N_y, -N_x, 0)
      if (s2 == 0.0) { R[4] = -1; R[8] = -1; }                                 // N = -z: half turn about x
      else {
        const double k = (1.0 - cz) / s2;
        // I + [v]x + k [v]x^2 with v = (vx, vy, 0)
        R[0] = 1 - k * vy * vy; R[1] = k * vx * vy;     R[2] = vy;
        R[3] = k * vx * vy;     R[4] = 1 - k * vx * vx; R[5] = -vx;
        R[6] = -vy;             R[7] = vx;              R[8] = 1 - k * s2;
      }
    }
    double gl[3], z0 = 0.0;
    for (int i = 0; i < 3; i++) {
      gl[i] = R[3 * i] * c.gravity[0] + R[3 * i + 1] * c.gravity[1] + R[3 * i + 2] * c.gravity[2];
      z0 += N[i] * c.plane_origin[i];
    }
    const double cv = c.damping_constant >= 0.0 ? exp(-c.damping_constant * c.dt) : 1.0;
    for (int i = 0; i < 9; i++) A.lab2int[i] = (T)R[i];
    A.plane_z0 = (T)z0;
    for (int i = 0; i < 3; i++) {
      A.gm[i] = (T)(gl[i] * mass);
      if (A.rot_on) { A.gdt_cv[i] = (T)(gl[i] * c.dt * cv); A.gdt[i] = (T)(gl[i] * c.dt); A.g[i] = (T)gl[i]; }
    }
    // lab-frame direction of the travelling-wave muscle torque (MuscleTorques(direction=...)): same frame change
    for (int i = 0; i < 3; i++)
      A.mus_dir[i] = (T)(R[3 * i] * c.muscle_direction[0] + R[3 * i + 1] * c.muscle_direction[1] + R[3 * i + 2] * c.muscle_direction[2]);
  }
  A.contact_k = (T)c.contact_k; A.contact_nu = (T)c.contact_nu; A.slip_tol = (T)c.slip_velocity_tol;
  A.inv_slip_tol = (T)(c.slip_velocity_tol > 0 ? 1.0 / c.slip_velocity_tol : 0.0);
  A.surface_tol = (T)c.surface_tol; A.vol_over_pi = (T)((r * r) * rl);
  A.muscle = nullptr; A.muscle_on = c.muscle_on; A.muscle_dim = n + 2;
  A.mus_omega = c.muscle_period > 0.0 ? 2.0 * PI / c.muscle_period : 0.0;
  A.mus_ramp = c.muscle_ramp_up_time; A.mus_phase = c.muscle_phase_shift;
  A.spline = nullptr; A.spline_tab = nullptr; A.spline_mask = c.spline_dir_mask & 7; A.spline_p = c.spline_n_ctrl;
  A.spline_dim = 3 * (2 * c.spline_n_ctrl + 2) + 3 * n;
  A.spline_scale = c.spline_scale; A.spline_rate = c.spline_max_rate;
  A.spline_inv_dx = c.spline_n_ctrl > 0 ? (c.spline_n_ctrl + 1) / c.base_length : 0.0;
  A.isotropic = 1;  // straight_rod builds circular cross-sections: I1 == I2
  {
    const double cs[] = SR_COEF_SINC, cc[] = SR_COEF_COSC, cb[] = SR_COEF_BEND, ce[] = SR_COEF_EXP;
    for (int i = 0; i < 6; i++) { A.poly.sinc[i] = (T)cs[i]; A.poly.cosc[i] = (T)cc[i]; A.poly.expz[i] = (T)ce[i]; }
    for (int i = 0; i < 14; i++) A.poly.bend[i] = (T)cb[i];
    const double ns[] = SR_COEF_SINC3, nc[] = SR_COEF_COSC3, nb[] = SR_COEF_BEND7, ne[] = SR_COEF_EXP3;
    for (int i = 0; i < 4; i++) { A.poly.sinc3[i] = (T)ns[i]; A.poly.cosc3[i] = (T)nc[i]; A.poly.exp3[i] = (T)ne[i]; }
    for (int i = 0; i < 8; i++) A.poly.bend7[i] = (T)nb[i];
    const double nm[] = SR_COEF_BEND9;
    for (int i = 0; i < 10; i++) A.poly.bend9[i] = (T)nm[i];
  }
  double lcw[3] = {0.0, 0.0, 0.0};
  if (c.damping_constant >= 0.0) {
    // element mass incl. the end-element correction equals `mass` for a uniform rod
    A.c_v = (T)exp(-c.damping_constant * c.dt);
    for (int i = 0; i < 3; i++) {
      double lc = -c.damping_constant * c.dt * mass * (1.0 / J[i]);
      lcw[i] = lc;
      A.logc_w[i] = (T)lc;
      A.c_w[i] = (T)exp(lc);
    }
  } else {
    A.c_v = (T)1.0;
    for (int i = 0; i < 3; i++) { A.logc_w[i] = (T)0.0; A.c_w[i] = (T)1.0; }
  }
  // ---- lean kernel tables (rod_kernel_lean.cuh) ----------------------------------------------------------------
  auto hi_word = [](double x) { long long b; memcpy(&b, &x, 8); return (int)((b >> 32) & 0x7fffffff); };
  A.BDH = (T)((Bv[2] - Bv[0]) * 0.5 * rl);
  A.half_inv_rest_vor = (T)(0.5 / rl);
  A.dt_Jinv0 = (T)(c.dt / J[0]);
  {
    const double cw2[] = SR_COEF_BENDW, sg[] = SR_COEF_SINCG, ch[] = SR_COEF_COSCH;
    for (int i = 0; i < 10; i++) A.bendw[i] = (T)(cw2[i] * (-0.5 / rl));
    { const double cm[] = SR_COEF_BENDW_MID; for (int i = 0; i < 14; i++) A.bendw_mid[i] = (T)(cm[i] * (-0.5 / rl)); }
    for (int i = 0; i < 3; i++) { A.sincg[i] = sg[i]; A.cosch[i] = ch[i]; }
    // c_w^e = c_w exp(z), z = (e - 1) ln c_w, |z| <= kLeanExpZ: 1 + z + z^2/2 with the powers of ln c_w folded in
    double lmax = 0.0;
    for (int k = 0; k < 2; k++) {
      const double lc = lcw[2 * k], cw = exp(lc);
      lmax = fmax(lmax, fabs(lc));
      A.cwp[k][0] = (T)cw; A.cwp[k][1] = (T)(cw * lc); A.cwp[k][2] = (T)(cw * 0.5 * lc * lc);
      double term = cw;
      for (int i = 0; i < 7; i++) { A.cwc[k][i] = (T)term; term *= lc / (double)(i + 1); }
    }
    A.k_dt = c.dt; A.k_half_dt = 0.5 * c.dt; A.k_dt_inv_mass = c.dt / mass; A.k_inv_rest_len = 1.0 / rl;
    A.k_c_v = c.damping_constant >= 0.0 ? exp(-c.damping_constant * c.dt) : 1.0;
    for (int i = 0; i < 3; i++) A.k_gdt_cv[i] = c.gravity[i] * c.dt * A.k_c_v;
    A.limf_bend = (float)sr::kNarrowBendW2;
    A.limf_em1 = lmax > 0.0 ? (float)fmin(sr::kLeanExpZ / lmax, 1e30) : 3.0e38f;
    A.lim_rot_hi = hi_word(sr::kNarrowRotQ);
    A.lim_bend_hi = hi_word(sr::kNarrowBendW2);
    A.lim_bendm_hi = hi_word(sr::kMidBendW2);
    A.lim_em1_hi = lmax > 0.0 ? hi_word(fmin(sr::kLeanExpZ / lmax, 1e300)) : 0x7fefffff;   // no damper: any finite stretch
    A.lim_em1c_hi = lmax > 0.0 ? hi_word(fmin(sr::kLeanExpZc / lmax, 1e300)) : 0x7fefffff;
    A.half_rest_vor = (T)(0.5 * rl);
    A.mus_cd = cos(A.mus_omega * c.dt); A.mus_sd = sin(A.mus_omega * c.dt);
    A.mus_inv_ramp = 1.0 / A.mus_ramp;   // (ramp 0: inf, and fmin(1, t * inf) = 1 like the reference's t / 0)
  }
}

int cuda_fail(const char *what, cudaError_t e) {
  return fail(SR_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

// The run-time switches, read once per process.  Each picks between kernels that give every env the same bits (FOLD:
// outside the padding slots); the default is the measured winner, the other serves as the reference in tests and A/B runs.
struct Switches {
  bool fastpath;   // SOFTROD_FASTPATH=0: the single safe kernel with per-thread fallbacks instead of the pair
  bool planar;     // SOFTROD_LEAN_PLANAR=0: rods in the x-y plane take the 3D kernels too
  bool cluster;    // SOFTROD_LEAN_CLUSTER=1: rods of 512-1023 elements take the cluster layout too
  bool fold;       // SOFTROD_LEAN_FOLD=0: a rod of 512 elements takes a 544-thread CTA instead of the fold layout
};
const Switches &switches() {
  static const Switches s = [] {
    auto on = [](const char *name, bool dflt) { const char *e = getenv(name); return e ? atoi(e) != 0 : dflt; };
    return Switches{on("SOFTROD_FASTPATH", true), on("SOFTROD_LEAN_PLANAR", true), on("SOFTROD_LEAN_CLUSTER", false),
                    on("SOFTROD_LEAN_FOLD", true)};
  }();
  return s;
}

// Whether this step runs the fast-only kernel + fallback pair.  Both ways give every env the same bits (the safe
// kernel falls back per thread, and inside the range evaluates exactly what the fast-only kernel evaluates), so
// this is a pure scheduling choice: one flagged env re-runs its whole CTA (4-5 envs) in the fallback, and the pair
// only pays while about 1 % of the envs or fewer leave the fast-math range (a pair gains 5-10 %).  The fast-only
// kernel counts the env-steps it hands over (redo_count); every 8 steps the count is fetched asynchronously, and
// when more than 1 % of a window's env-steps fell back (violently actuated arms do) the handle uses the single
// safe kernel for the next 512 steps, then probes again.
template <typename T> bool use_fast_pair(sr_handle *h, sr::RodArgs<T> &A, cudaStream_t s) {
  if (!switches().fastpath || !A.redo) return false;
  h->pair_steps++;
  if (h->pair_off_until > h->pair_steps) return false;
  cudaError_t q = h->pair_copy_pending ? cudaEventQuery(h->pair_event) : cudaErrorNotReady;
  if (h->pair_copy_pending && q == cudaErrorNotReady) (void)cudaGetLastError();   // "not ready" is an answer, not an error to report later
  if (h->pair_copy_pending && q == cudaSuccess) {
    h->pair_copy_pending = false;
    const unsigned long long seen = h->h_redo_count[0], delta = seen - h->pair_last_count;
    const unsigned long long seen_np = h->h_redo_count[4], delta_np = seen_np - h->planar_last_count;
    const long long window = (h->pair_steps_at_copy - h->pair_steps_at_prev_copy) * (long long)A.n_env;
    h->pair_last_count = seen;
    h->planar_last_count = seen_np;
    h->pair_steps_at_prev_copy = h->pair_steps_at_copy;
    // the same rule for envs that are not planar: the handle steps with the 3D pair for a while (see launch_lean)
    if (window > 0 && (double)delta_np > 0.01 * (double)window) h->planar_off_until = h->pair_steps + 512;
    if (window > 0 && (double)delta > 0.01 * (double)window) { h->pair_off_until = h->pair_steps + 512; return false; }
  }
  if (!h->pair_copy_pending && h->pair_steps % 8 == 0) {
    cudaMemcpyAsync(h->h_redo_count, h->redo_count, 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s);
    cudaEventRecord(h->pair_event, s);
    h->pair_copy_pending = true;
    h->pair_steps_at_copy = h->pair_steps;
  }
  A.redo_count = h->redo_count;
  return true;
}

// The one pair runner: the fast-only kernel, then the safe one over the envs it flagged (an empty launch in the normal
// case), or the safe kernel alone.  use_fast_pair is asked only for a kernel that pairs, since asking advances the
// pair's step count, its polling of the fallback counts and its windows.  launch(std::true_type()) launches the
// fast-only kernel, launch(std::false_type()) the safe one.
template <typename T, typename L> int run_pair(sr_handle *h, sr::RodArgs<T> &A, bool pair, cudaStream_t s, L &&launch) {
  if (pair && use_fast_pair(h, A, s)) {
    const int rc = launch(std::true_type());
    if (rc != SR_OK) return rc;
    A.redo_filter = 1;
  }
  return launch(std::false_type());
}

// The one CTA-size dispatcher: a run-time CTA size to the <NT, MINB> template arguments of the sizes build.py compiles
// (PACKED_SIZES; MINB = the resident CTAs per SM the kernels are compiled for).
template <int NT_, int MINB_> struct Cta { static constexpr int NT = NT_, MINB = MINB_; };
template <typename F> int with_cta(int nt, F &&launch) {
  switch (nt) {
    case 256: return launch(Cta<256, 2>());
    case 384: return launch(Cta<384, 1>());
    case 512: return launch(Cta<512, 1>());
    case 544: return launch(Cta<544, 1>());
    case 768: return launch(Cta<768, 1>());
    case 1024: return launch(Cta<1024, 1>());
  }
  return fail(SR_E_INVALID, "no kernel is built for CTAs of " + std::to_string(nt) + " threads");
}

using sr::LeanLayout;
using sr::LeanModel;

// Of those sizes, the ones build.py's LEAN_UNITS compile a one-CTA lean model and layout at: the fold layout at 512
// threads only, the planar model up to 512 and at 768 (planar_threads_setting) and the filter model up to 768 (its
// 1024-thread CTA would need 243 KB of shared memory).
constexpr bool lean_built(LeanModel model, LeanLayout layout, int nt) {
  return layout == LeanLayout::FOLD ? nt == 512
         : model == LeanModel::PLANAR ? nt <= 512 || nt == 768
         : model == LeanModel::FILTER ? nt <= 768
                                      : true;
}

// CTA size of the generic kernel and of the assembly model.  Registers cap the SM at 512 resident threads (128 regs),
// so the choice is 2 x 256 or 1 x 512; take whichever wastes fewer lanes for this rod length
// (n = 50: 5 x 51 = 255/256; n = 100: 2 x 101 = 202/256 but 5 x 101 = 505/512).
int packed_threads_setting(int n_elem, int n_rod = 1, int has_head = 0) {
  const int tpr = (n_rod > 1 ? n_rod : 1) * (n_elem + 1) + has_head;   // threads per env group
  auto util = [&](int nt) { return (double)((nt / tpr) * tpr) / nt; };
  // 2 x 256 (128 regs) is the default; 1 x 384 (168 regs) / 1 x 512 (128 regs) only when they waste
  // clearly fewer lanes for this group size
  int best = 256;
  if (util(384) > util(best) + 0.02) best = 384;
  if (util(512) > util(best) + 0.02) best = 512;
  // long rods: one rod per CTA, as few warps as hold it so that each thread keeps as many registers as
  // possible (544 threads: 120 registers, 768: 80, 1024: 64)
  if (tpr > 512) best = tpr <= 544 ? 544 : (tpr <= 768 ? 768 : 1024);
  return best;
}

// CTA size of the one-CTA lean kernels of a single rod.  With per-rod barriers one 512-thread CTA per SM (16 warps,
// 10 rods of n = 50) beats two of 256 (measured: 1.51 vs 1.64 ms per 4096-env step): take 512 whenever it wastes no
// more lanes.
int lean_threads_setting(int n_elem) {
  const int tpr = n_elem + 1;
  if (tpr > 512) return packed_threads_setting(n_elem);
  auto util = [&](int nt) { return (double)((nt / tpr) * tpr) / nt; };
  int best = 512;
  if (util(384) > util(best) + 0.02) best = 384;
  if (util(256) > util(best) + 0.02) best = 256;
  return best;
}

// CTA size of the planar model's fast-only kernel.  Its nine state doubles per thread fit the 80 registers of one
// 768-thread CTA per SM: 24 warps, six per scheduler instead of four, to hide the substep's dependent chains.  Taken
// wherever those 768 threads hold 2-15 rods of >= 32 threads (the per-rod barriers), even where they leave more lanes
// idle than lean_threads_setting's CTA: measured (B200, 1000 W, 1965 MHz), n = 50 (15 x 51 = 765 / 768 lanes against
// 10 x 51 = 510 / 512) steps 7 % faster than in 512 threads, n = 100 (7 x 101 = 707 / 768 against 505 / 512) 9 %.
// Also measured faster at n = 95, 160 (the most idle lanes relative to 512), 255 and 256; the other lengths of 48-383
// elements are not measured and follow these six (DESIGN.md §4.1).
// Otherwise that CTA, which the 3D pair and the safe fallback use in any case.
int planar_threads_setting(int n_elem) {
  const int tpr = n_elem + 1, rods = 768 / tpr;
  return tpr >= 32 && rods >= 2 && rods <= 15 ? 768 : lean_threads_setting(n_elem);
}

// CTAs of the cluster that holds one rod of n elements in the cluster layout: n + 1 threads of 512 per CTA
int lean_cluster_size(int n_elem) { return (n_elem + sr::LEAN_CLUSTER_NT) / sr::LEAN_CLUSTER_NT; }

// The model a rod steps with in the cluster layout: the plain model, SoftPendulum3D-v0's (the Laplace filter and the
// moving base), the rod on the frictional plane with rest-curvature actuation (`loads`) and the travelling-wave
// muscle, or SoftArmTracking-v0's spline torques.  sr_create checks its cluster shape for rods of 1024-4095 elements,
// the only models it admits there.
LeanModel lean_cluster_model(int laplace_order, int bc_kind, bool loads, bool muscle_on, bool spline) {
  if (spline) return LeanModel::SPLINE;
  if (loads) return muscle_on ? LeanModel::MUSCLE : LeanModel::PLANE;
  return laplace_order > 0 || bc_kind == sr::BC_MOVING_BASE ? LeanModel::FILTER : LeanModel::PLAIN;
}

// The one cluster dispatcher: a run-time cluster model to the template argument of the cluster kernels build.py
// compiles; launch(std::integral_constant<LeanModel, M>()).
template <typename F> auto with_cluster_model(LeanModel model, F &&launch) {
  using M = LeanModel;
  switch (model) {
    case M::FILTER: return launch(std::integral_constant<M, M::FILTER>());
    case M::PLANE: return launch(std::integral_constant<M, M::PLANE>());
    case M::MUSCLE: return launch(std::integral_constant<M, M::MUSCLE>());
    case M::SPLINE: return launch(std::integral_constant<M, M::SPLINE>());
    default: return launch(std::integral_constant<M, M::PLAIN>());   // (lean_cluster_model returns no other model)
  }
}

// What steps a handle (classify): the launcher of one kernel, and the launch's shape.
template <typename T> struct StepKernel {
  int (*launch)(sr_handle *, sr::RodArgs<T> &, const StepKernel &, cudaStream_t);
  int nt;        // CTA size of the one-CTA lean kernels and the generic kernel
  bool pair;     // fast-only kernel + fallback (run_pair)
  bool planar;   // plain model, CTA layout: the fast-only kernel is the planar model's while the handle's planar window allows
  int planar_nt;  // CTA size of that planar kernel (planar_threads_setting)
};

template <typename T, int NT, int MINB, bool LAPLACE, bool MOVING, bool CONTACT, bool MULTI, bool TORQUE = false,
          bool FASTONLY = false>
int launch_packed_impl(sr_handle *h, sr::RodArgs<T> &A, cudaStream_t s) {
  const int group = (MULTI ? A.n_rod : 1) * (A.n_elem + 1) + (MULTI ? A.has_head : 0);   // threads per env
  const int rods_per_cta = NT / group;
  if (rods_per_cta < 1) return fail(SR_E_INVALID, "environment does not fit one CTA of the packed kernel");
  const int grid = (A.n_env + rods_per_cta - 1) / rods_per_cta;
  cudaError_t e = sr::launch_packed_kernel<T, NT, MINB, LAPLACE, MOVING, CONTACT, MULTI, TORQUE, FASTONLY>(A, rods_per_cta, grid, s);
  h->launches++;
  if (e != cudaSuccess) return cuda_fail("rod_packed_kernel launch", e);
  return SR_OK;
}

// Lean FP64 path: grid and stream-K schedule.  With more items than resident CTA slots the grid is the slot
// count and every slot gets the same number of item-substeps (rod_kernel_lean.cuh); partial items travel through
// sk_scratch.  The fallback launch (redo_filter) visits flagged envs only and keeps one CTA per item.
template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT>
int launch_lean_impl(sr_handle *h, sr::RodArgs<T> &A, cudaStream_t s) {
  const bool multi = MODEL == LeanModel::ASSEMBLY, fold = LAYOUT == LeanLayout::FOLD;   // (fold: the tip node lives in the last element's thread)
  const int group = fold ? A.n_elem : (multi ? A.n_rod : 1) * (A.n_elem + 1) + (multi ? A.has_head : 0);
  const int rods_per_cta = NT / group;   // env groups per CTA
  if (rods_per_cta < 1) return fail(SR_E_INVALID, "environment does not fit one CTA of the lean kernel");
  const int items = (A.n_env + rods_per_cta - 1) / rods_per_cta;
  // resident CTAs per SM of this kernel (a property of the kernel and the device model: asked once); the slot count
  // differs between the kernels of a handle, the scratch is sized for the largest
  static int ctas_per_sm = 0;
  if (ctas_per_sm == 0) ctas_per_sm = sr::lean_ctas_per_sm<T, NT, MINB, FASTONLY, MODEL, LAYOUT>();
  if (ctas_per_sm < 1) return fail(SR_E_CUDA, "lean kernel: occupancy query failed");
  if (h->sk_sms == 0) {
    cudaDeviceProp prop;
    SR_CUDA(cudaGetDeviceProperties(&prop, h->cfg.device));
    h->sk_sms = prop.multiProcessorCount;
  }
  const int slots = h->sk_sms * ctas_per_sm;
  // (the kernels of a handle may differ in CTA size too: the planar one's 768 threads against the 3D pair's 512)
  if (slots > h->sk_slots || (long long)slots * NT > h->sk_slot_threads) {
    const int n_slots = std::max(slots, h->sk_slots);
    const long long n_threads = std::max((long long)slots * NT, h->sk_slot_threads);
    cudaFree(h->sk_scratch); cudaFree(h->sk_flag);
    h->sk_scratch = nullptr; h->sk_flag = nullptr; h->sk_slots = 0; h->sk_slot_threads = 0;
    SR_CUDA(cudaMalloc(&h->sk_scratch, (size_t)n_threads * sr::LEAN_SCR_FOLD * sizeof(double)));
    SR_CUDA(cudaMalloc(&h->sk_flag, (size_t)n_slots * sizeof(int)));
    SR_CUDA(cudaMemset(h->sk_flag, 0, (size_t)n_slots * sizeof(int)));
    h->sk_slots = n_slots; h->sk_slot_threads = n_threads;
  }
  A.sk_rods_per_cta = rods_per_cta; A.sk_items = items;
  A.sk_split = (!A.redo_filter && items > slots && A.n_substeps > 0) ? 1 : 0;
  A.sk_scratch = (double *)h->sk_scratch; A.sk_flag = h->sk_flag;
  const int grid = A.sk_split ? slots : items;
  cudaError_t e = sr::launch_lean_kernel<T, NT, MINB, FASTONLY, MODEL, LAYOUT>(A, grid, s);
  h->launches++;
  if (e != cudaSuccess) return cuda_fail("rod_lean_kernel launch", e);
  return SR_OK;
}

// the planar model's fast-only kernel (FP64) in CTAs of nt threads
template <typename T> int launch_planar(sr_handle *h, sr::RodArgs<T> &A, int nt, cudaStream_t s) {
  return with_cta(nt, [&](auto cta) {
    using C = decltype(cta);
    if constexpr (!std::is_same<T, double>::value || !lean_built(LeanModel::PLANAR, LeanLayout::CTA, C::NT))
      return fail(SR_E_INVALID, "rod_lean_kernel: the planar model is not built for this type or " + std::to_string(C::NT) + " threads");
    else return launch_lean_impl<T, C::NT, C::MINB, true, LeanModel::PLANAR, LeanLayout::CTA>(h, A, s);
  });
}

// the lean kernel (rod_kernel_lean.cuh) of one model in the CTA or fold layout, in CTAs of k.nt threads (the planar
// fast-only kernel in CTAs of k.planar_nt)
template <typename T, LeanModel MODEL, LeanLayout LAYOUT> int launch_lean(sr_handle *h, sr::RodArgs<T> &A, const StepKernel<T> &k, cudaStream_t s) {
  return with_cta(k.nt, [&](auto cta) {
    using C = decltype(cta);
    if constexpr (!lean_built(MODEL, LAYOUT, C::NT)) {
      static const char *const model[] = {"plain", "plane", "muscle", "assembly", "filter", "spline", "planar"};   // LeanModel's order
      static const char *const layout[] = {"CTA", "fold", "cluster"};                                            // LeanLayout's order
      return fail(SR_E_INVALID, std::string("rod_lean_kernel: the ") + model[(int)MODEL] + " model in the " + layout[(int)LAYOUT] +
                                    " layout is not built for " + std::to_string(C::NT) + " threads");
    } else {
      return run_pair(h, A, k.pair, s, [&](auto fast) {
        constexpr bool FAST = decltype(fast)::value;
        if constexpr (FAST && MODEL == LeanModel::PLAIN && LAYOUT == LeanLayout::CTA && std::is_same<T, double>::value) {
          // when more than 1 % of a window's env-steps were handed over for not being planar, the handle steps with
          // the 3D pair for the next 512 steps (use_fast_pair)
          if (k.planar && h->pair_steps >= h->planar_off_until) return launch_planar(h, A, k.planar_nt, s);
        }
        return launch_lean_impl<T, C::NT, C::MINB, FAST, MODEL, LAYOUT>(h, A, s);
      });
    }
  });
}

// the lean kernel of one model in the cluster layout: one rod per thread-block cluster, no stream-K split
template <LeanModel MODEL> int launch_cluster(sr_handle *h, sr::RodArgs<double> &A, const StepKernel<double> &k, cudaStream_t s) {
  const int C = lean_cluster_size(A.n_elem);
  A.sk_rods_per_cta = 1; A.sk_items = A.n_env; A.sk_split = 0;
  A.sk_scratch = nullptr; A.sk_flag = nullptr;
  return run_pair(h, A, k.pair, s, [&](auto fast) {
    constexpr bool FAST = decltype(fast)::value;
    if constexpr (FAST && MODEL == LeanModel::SPLINE) {
      return fail(SR_E_INVALID, "rod_lean_kernel: the spline model on clusters is built as the safe kernel only");
    } else {
      cudaError_t e = sr::launch_lean_cluster_kernel<FAST, MODEL>(A, C, s);
      h->launches++;
      if (e != cudaSuccess) return cuda_fail("rod_lean_kernel (cluster) launch", e);
      return SR_OK;
    }
  });
}

// the generic kernel (rod_kernel_packed.cuh) with the features of one group
enum { G_FILTER, G_CONTACT, G_TORQUE, G_MULTI };   // Laplace filter + moving base / plane contact / + forcing torques / assemblies
template <typename T, int G> int launch_generic(sr_handle *h, sr::RodArgs<T> &A, const StepKernel<T> &k, cudaStream_t s) {
  return with_cta(k.nt, [&](auto cta) {
    using C = decltype(cta);
    return run_pair(h, A, k.pair, s, [&](auto fast) {
      constexpr bool FAST = decltype(fast)::value;
      if constexpr (FAST && !std::is_same<T, double>::value) {
        return fail(SR_E_INVALID, "rod_packed_kernel: the fast-only kernel is built for FP64 only");
      } else {
        return launch_packed_impl<T, C::NT, C::MINB, G == G_FILTER, G == G_FILTER, G != G_FILTER, G == G_MULTI, G == G_TORQUE, FAST>(h, A, s);
      }
    });
  });
}

// tapered rods: safe kernel with per-element constants in registers (CTA sizes 384 / 1024 only)
template <int NT> int launch_tapered(sr_handle *h, sr::RodArgs<double> &A, const StepKernel<double> &, cudaStream_t s) {
  const bool multi = A.n_rod > 1 || A.has_head;
  const int group = (multi ? A.n_rod : 1) * (A.n_elem + 1) + (multi ? A.has_head : 0);
  const int rods_per_cta = NT / group;
  if (rods_per_cta < 1) return fail(SR_E_INVALID, "environment does not fit one CTA of the packed kernel");
  const int grid = (A.n_env + rods_per_cta - 1) / rods_per_cta;
  if (A.mus_act) {
    if (NT != 384 || !multi) return fail(SR_E_INVALID, "muscle layers: multi-rod assemblies of at most 384 threads only");
    cudaError_t el = sr::launch_packed_lmus_kernel<384>(A, rods_per_cta, grid, s);
    h->launches++;
    if (el != cudaSuccess) return cuda_fail("rod_packed_kernel (muscle layers) launch", el);
    return SR_OK;
  }
  cudaError_t e = multi ? sr::launch_packed_kernel<double, NT, 1, false, false, true, true, false, false, true>(A, rods_per_cta, grid, s)
                        : sr::launch_packed_kernel<double, NT, 1, false, false, true, false, false, false, true>(A, rods_per_cta, grid, s);
  h->launches++;
  if (e != cudaSuccess) return cuda_fail("rod_packed_kernel (tapered) launch", e);
  return SR_OK;
}

// faithful math (libm calls in the reference's operation order): warp-per-rod kernel, the parity build
int launch_faithful(sr_handle *h, sr::RodArgs<double> &A, const StepKernel<double> &, cudaStream_t s) {
  const int grid = (A.n_env + sr::WARPS_PER_CTA - 1) / sr::WARPS_PER_CTA;
  cudaError_t e = h->epl == 1 ? sr::launch_warp_faithful<double, 1>(A, grid, s)
                  : h->epl == 2 ? sr::launch_warp_faithful<double, 2>(A, grid, s)
                                : sr::launch_warp_faithful<double, 4>(A, grid, s);
  h->launches++;
  if (e != cudaSuccess) return cuda_fail("rod_substeps_kernel launch", e);
  return SR_OK;
}

// The one classification: the kernel that steps this handle.  One row per kernel in precedence order; a config takes
// the first row whose model it is.  The lean kernel's models share their exclusions: none of them steps suckers,
// external loads or per-element constants, and all but the plain one need FP64 and no base point force.
template <typename T> StepKernel<T> classify(const sr_handle *h, const sr::RodArgs<T> &A) {
  constexpr bool F64 = std::is_same<T, double>::value;
  const Switches &sw = switches();
  const int n = A.n_elem, bc = A.bc_kind;
  const int lean_nt = lean_threads_setting(n), packed_nt = packed_threads_setting(n, A.n_rod, A.has_head);
  const bool assembly = A.n_rod > 1 || A.has_head;
  const bool free_or_clamped = bc == sr::BC_FREE || bc == sr::BC_ONE_END_FIXED;
  const bool lean_plain = !(A.sucker || A.ext_force || A.ext_couple || A.elem_tab);
  const bool lean = F64 && lean_plain && !A.point_force;
  const bool loads = A.contact_on || A.rest_kappa || A.muscle_on;   // the plane models' plane and actuations
  // the plain model: one rod under gravity, damping and the base point force, with a free, clamped or slider end
  const bool plain = lean_plain && !assembly && !loads && !A.spline_mask && A.laplace_order == 0 && bc != sr::BC_MOVING_BASE;
  // the filter model, SoftPendulum3D-v0's: the order-7 LaplaceDissipationFilter, or none with the moving base; a moving,
  // clamped or free base (n >= 8: the filter's ghost records assume one reflection per end)
  const bool filter = lean && !assembly && !loads && !A.spline_mask && n >= 8 &&
                      (A.laplace_order == 7 || (A.laplace_order == 0 && bc == sr::BC_MOVING_BASE)) &&
                      (free_or_clamped || bc == sr::BC_MOVING_BASE);
  // the plane / muscle models: one rod on the frictional plane / with rest-curvature actuation / with the
  // travelling-wave muscle
  const bool contact = lean && !assembly && loads && !A.spline_mask && A.laplace_order == 0 && free_or_clamped;
  // the spline model, SoftArmTracking-v0's spline muscle torques; the safe kernel alone, as it updates the forcing's
  // cached control values and magnitudes inside the launch
  const bool spline = lean && A.spline_mask && !assembly && !loads && A.laplace_order == 0 && free_or_clamped;
  if constexpr (F64) {
    if (h->cfg.math != SR_MATH_FAST) return {launch_faithful};
    if (A.elem_tab) return {h->n_rod * (n + 1) + (A.has_head ? 1 : 0) <= 384 ? launch_tapered<384> : launch_tapered<1024>};
    // rods of 1024-4095 elements, and filter rods of 768-1023, whose CTA layout would not fit its shared memory
    if (n >= 1024 || (n >= 768 && filter) || (sw.cluster && n >= 512 && (plain || filter || contact || spline)))
      return with_cluster_model(lean_cluster_model(A.laplace_order, bc, loads, A.muscle_on, A.spline_mask != 0), [](auto m) {
        return StepKernel<T>{launch_cluster<decltype(m)::value>, 0, decltype(m)::value != LeanModel::SPLINE};
      });
    // the assembly model (OctoFlat: arms + rigid head + FixedJoint2Rigid joints on the plane)
    if (lean && assembly && !A.spline_mask && !A.muscle_on && A.laplace_order == 0 && bc == sr::BC_FREE && A.rot_on == 0)
      return {launch_lean<T, LeanModel::ASSEMBLY, LeanLayout::CTA>, packed_nt, true};
    if (spline) return {launch_lean<T, LeanModel::SPLINE, LeanLayout::CTA>, lean_nt, false};
    if (filter) return {launch_lean<T, LeanModel::FILTER, LeanLayout::CTA>, lean_nt, true};
    // the plain / plane model in the fold layout: a rod of exactly 512 elements in 512 threads, the tip node folded
    // into the last one (128 registers), instead of 513 threads in a 544-thread CTA (96 registers)
    if (sw.fold && n == 512 && A.model == sr::MODEL_ROD && !A.muscle_on && (contact || plain))
      return {contact ? launch_lean<T, LeanModel::PLANE, LeanLayout::FOLD> : launch_lean<T, LeanModel::PLAIN, LeanLayout::FOLD>,
              512, true};
    if (contact)
      return {A.muscle_on ? launch_lean<T, LeanModel::MUSCLE, LeanLayout::CTA> : launch_lean<T, LeanModel::PLANE, LeanLayout::CTA>,
              lean_nt, true};
  }
  if (plain) {
    // Its fast-only kernel may be the planar model's when the model keeps the out-of-plane components exact zeros
    // once the state has them: FP64, gravity in the x-y plane, the base point force along x (the only direction the
    // kernel applies it in), and a BC that pins in-plane rows (slider, clamp) or none.  The kernel checks the state
    // itself, per rod, and hands the rods that are not planar over to the safe kernel.
    const bool planar = F64 && sw.planar && lean_nt <= 512 && (double)A.gdt_cv[2] == 0.0 &&
                        (free_or_clamped || bc == sr::BC_PENDULUM_SLIDER);
    return {launch_lean<T, LeanModel::PLAIN, LeanLayout::CTA>, lean_nt, true, planar, planar_threads_setting(n)};
  }
  // The generic kernel: FP32 storage of the other models, suckers, external loads, the base point force with other
  // forcings, filter orders other than 7.  The single rod on the plane (OctoArmSingle's model) takes the lean CTA-size
  // rule: one 512-thread CTA per SM measured 4 % ahead of two of 256 (3.85 vs 4.04 ms per 4096-env step).
  const int nt = A.contact_on && !A.muscle_on && !A.spline_mask && !assembly ? lean_nt : packed_nt;
  const bool pair = F64 && !A.spline_mask;   // (the spline forcing updates its cache inside the launch: safe kernel only)
  if (assembly) return {launch_generic<T, G_MULTI>, nt, pair};
  if (A.muscle_on || A.spline_mask) return {launch_generic<T, G_TORQUE>, nt, pair};
  if (A.contact_on || A.rest_kappa || A.sucker || A.ext_force || A.ext_couple) return {launch_generic<T, G_CONTACT>, nt, pair};
  return {launch_generic<T, G_FILTER>, nt, pair};
}

template <typename T> int launch_step(sr_handle *h, sr::RodArgs<T> &A, cudaStream_t s) {
  const StepKernel<T> k = classify(h, A);
  return k.launch(h, A, k, s);
}

// The per-env buffers of a handle: everything that evolves or parametrises an env, which sr_copy_from clones and
// sr_copy_envs copies row by row.  Env e's row of a buffer is the `bytes` bytes at base + e * bytes (rod-level buffers
// hold an env's n_rod rows back to back); base is null for a buffer the handle has not allocated.  `lazy`: allocated
// on first use by its getter, zero until then (alloc_lazy_like).
struct EnvBuf { void *base; size_t bytes; bool lazy; };
enum { EB_STATE, EB_BC, EB_AUX, EB_HEAD, EB_REST_KAPPA, EB_EXT_FORCE, EB_EXT_COUPLE, EB_SUCKER, EB_SUCKER_IDX, EB_TM_ACT,
       EB_MUS_ACT, EB_MSUCKER, EB_MUSCLE, EB_SPLINE, EB_COUNT };
static_assert(EB_COUNT <= sr::COPY_MAX_BUFS, "sr::CopyTable holds every per-env buffer");
void env_buffers(const sr_handle *h, EnvBuf (&b)[EB_COUNT]) {
  const size_t nr = (size_t)h->n_rod, es = h->elem_size, rows3 = nr * 3 * h->stride * es;
  b[EB_STATE] = {h->state, nr * sr::N_FIELDS * h->stride * es, false};
  b[EB_BC] = {h->bc, nr * sr::BC_DIM * es, false};
  b[EB_AUX] = {h->aux, sr::AUX_DIM * es, false};
  b[EB_HEAD] = {h->head, sr::HEAD_DIM * es, false};
  b[EB_REST_KAPPA] = {h->rest_kappa, rows3, true};
  b[EB_EXT_FORCE] = {h->ext_force, rows3, true};
  b[EB_EXT_COUPLE] = {h->ext_couple, rows3, true};
  b[EB_SUCKER] = {h->sucker, nr * es, false};
  b[EB_SUCKER_IDX] = {h->sucker_idx, nr * sizeof(int32_t), false};
  b[EB_TM_ACT] = {h->tm_act, nr * es, false};
  b[EB_MUS_ACT] = {h->mus_act, nr * 3 * (size_t)h->cfg.n_elem * sizeof(double), false};
  b[EB_MSUCKER] = {h->msucker, nr * 3 * sizeof(double), false};
  b[EB_MUSCLE] = {h->muscle, (size_t)h->muscle_dim * sizeof(double), false};
  b[EB_SPLINE] = {h->spline, (size_t)h->spline_dim * sizeof(double), false};
}

// The lazily allocated buffers `src` has and `dst` has not, allocated in dst through their getters.
int alloc_lazy_like(sr_handle *dst, const sr_handle *src) {
  void *p = nullptr, *q = nullptr;
  if (src->rest_kappa) {
    const int rc = sr_get_rest_kappa(dst, &p);
    if (rc != SR_OK) return rc;
  }
  if (src->ext_force) {
    const int rc = sr_get_ext_loads(dst, &p, &q);
    if (rc != SR_OK) return rc;
  }
  return SR_OK;
}

// The shapes sr_copy_from and sr_copy_envs need to agree, apart from the env count.
bool same_env_shape(const sr_handle *a, const sr_handle *b) {
  return a->cfg.n_elem == b->cfg.n_elem && a->n_rod == b->n_rod && a->cfg.dtype == b->cfg.dtype && a->cfg.model == b->cfg.model &&
         a->cfg.has_head == b->cfg.has_head && a->stride == b->stride && a->muscle_dim == b->muscle_dim &&
         a->spline_dim == b->spline_dim;
}

// The widest unit (16, 8 or 4 bytes) that divides the row size and both bases.
int copy_vec(const void *src, const void *dst, size_t bytes) {
  const uintptr_t m = (uintptr_t)src | (uintptr_t)dst | (uintptr_t)bytes;
  return m % 16 == 0 ? 16 : m % 8 == 0 ? 8 : 4;
}

// One launch of copy_envs_kernel over the n pairs of the index arrays (h: the handle whose launches it counts).
int launch_copy(sr_handle *h, sr::CopyTable &t, const int32_t *dst_idx, const int32_t *src_idx, int n, cudaStream_t s) {
  unsigned long long units = 0;   // the largest row in units of its vector width
  for (int k = 0; k < t.n_buf; k++) units = std::max(units, t.buf[k].bytes / t.buf[k].vec);
  // about four units per thread of a row; pairs on grid.y (at most 65535, the kernel strides over the rest)
  const unsigned gx = (unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>((units + 4 * sr::COPY_NT - 1) / (4 * sr::COPY_NT), 1024));
  const dim3 grid(gx, (unsigned)std::min(n, 65535));
  sr::copy_envs_kernel<<<grid, sr::COPY_NT, 0, s>>>(t, dst_idx, src_idx, n);
  h->launches++;
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SR_OK : cuda_fail("copy_envs_kernel launch", e);
}

}  // namespace

extern "C" {

int sr_abi_version(void) { return SR_ABI_VERSION; }
const char *sr_last_error(void) { return g_err.c_str(); }

int sr_create(const sr_config *cfg, sr_handle **out) {
  if (!cfg || !out) return fail(SR_E_INVALID, "sr_create: null argument");
  *out = nullptr;
  if (cfg->struct_size != (int32_t)sizeof(sr_config))
    return fail(SR_E_INVALID, "sr_create: sr_config.struct_size mismatch (ABI skew)");
  if (cfg->n_env <= 0 || cfg->n_elem < 3) return fail(SR_E_INVALID, "sr_create: n_env > 0 and n_elem >= 3 required");
  if (cfg->n_elem > 4095)
    return fail(SR_E_INVALID, "sr_create: n_elem <= 4095 (rods of 1024-4095 elements span a thread-block cluster of up to 8 CTAs)");
  // rods of 1024-4095 elements, on clusters: the plain model, SoftPendulum3D-v0's (filter), the rod on the frictional
  // plane with rest-curvature actuation and / or the travelling-wave muscle (plane / muscle), or SoftArmTracking-v0's
  // spline torques (spline)
  const bool loads = cfg->contact_on || cfg->muscle_on;
  const bool rod_free_or_clamped = cfg->model == SR_MODEL_ROD && (cfg->bc_kind == SR_BC_FREE || cfg->bc_kind == SR_BC_ONE_END_FIXED) &&
                                   cfg->laplace_filter_order == 0 && !cfg->point_force_on_base;
  const bool long_rod_model =
      cfg->spline_dir_mask ? rod_free_or_clamped && !loads
                           : ((cfg->model == SR_MODEL_ROD || cfg->model == SR_MODEL_SOFT_PENDULUM) &&
                              (cfg->bc_kind == SR_BC_FREE || cfg->bc_kind == SR_BC_ONE_END_FIXED || cfg->bc_kind == SR_BC_PENDULUM_SLIDER) &&
                              cfg->laplace_filter_order == 0 && !loads) ||
                                 (cfg->model == SR_MODEL_SOFT_PENDULUM_3D && cfg->bc_kind == SR_BC_MOVING_BASE &&
                                  cfg->laplace_filter_order == 7 && !cfg->point_force_on_base && !loads) ||
                                 (rod_free_or_clamped && loads);
  if (cfg->n_elem > 1023 &&
      (cfg->dtype != SR_DTYPE_F64 || cfg->math != SR_MATH_FAST || !long_rod_model ||
       cfg->n_rod_per_env > 1 || cfg->has_head || cfg->tip_radius > 0.0 || cfg->sucker_on ||
       cfg->tm_muscle_on || cfg->muscle_layers_on))
    return fail(SR_E_INVALID, "sr_create: n_elem of 1024-4095 is built for SR_DTYPE_F64, SR_MATH_FAST, SR_MODEL_ROD or "
                              "SR_MODEL_SOFT_PENDULUM, one untapered rod per env with a free, clamped or slider end, gravity, "
                              "damping and the base point force; for SR_MODEL_ROD with a free or clamped end on the frictional "
                              "plane (contact_on) and / or with the travelling-wave muscle (muscle_on), rest curvature, "
                              "gravity and damping, without the base point force; for SR_MODEL_ROD with a free or clamped end "
                              "and spline torques (spline_dir_mask), gravity and damping, without the base point force, "
                              "contact, the muscle wave or rest curvature; no suckers, transverse muscle, muscle layers or "
                              "Laplace filter, and spline torques with no other model; "
                              "and for SR_MODEL_SOFT_PENDULUM_3D with SR_BC_MOVING_BASE and laplace_filter_order = 7, "
                              "without the base point force");
  if (cfg->n_elem > 127 && cfg->math != SR_MATH_FAST) return fail(SR_E_INVALID, "sr_create: faithful math supports n_elem <= 127");
  if (cfg->dtype != SR_DTYPE_F64 && cfg->dtype != SR_DTYPE_F32) return fail(SR_E_INVALID, "sr_create: bad dtype");
  if (cfg->dtype == SR_DTYPE_F32 && cfg->math != SR_MATH_FAST)
    return fail(SR_E_INVALID, "sr_create: SR_DTYPE_F32 is built for SR_MATH_FAST (packed kernel) only");
  if (cfg->model != SR_MODEL_ROD && cfg->model != SR_MODEL_SOFT_PENDULUM && cfg->model != SR_MODEL_SOFT_PENDULUM_3D)
    return fail(SR_E_INVALID, "sr_create: unsupported model");
  if (cfg->bc_kind < SR_BC_FREE || cfg->bc_kind > SR_BC_MOVING_BASE)
    return fail(SR_E_INVALID, "sr_create: unsupported bc_kind");
  if (cfg->laplace_filter_order < 0 || cfg->laplace_filter_order > 64)
    return fail(SR_E_INVALID, "sr_create: laplace_filter_order out of range");
  if (cfg->math != SR_MATH_FAST && (cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE ||
                                    cfg->model == SR_MODEL_SOFT_PENDULUM_3D))
    return fail(SR_E_INVALID, "sr_create: Laplace filter / moving base are built for SR_MATH_FAST only");
  if (cfg->n_rod_per_env > 1 || cfg->has_head) {
    const int nr = cfg->n_rod_per_env > 1 ? cfg->n_rod_per_env : 1;
    if (cfg->math != SR_MATH_FAST || cfg->model != SR_MODEL_ROD || cfg->bc_kind != SR_BC_FREE || cfg->laplace_filter_order != 0)
      return fail(SR_E_INVALID, "sr_create: multi-rod assemblies need SR_MATH_FAST, SR_MODEL_ROD, SR_BC_FREE, no Laplace filter");
    if (nr > 16) return fail(SR_E_INVALID, "sr_create: at most 16 rods per environment");
    if (nr * (cfg->n_elem + 1) + (cfg->has_head ? 1 : 0) > 1024)
      return fail(SR_E_INVALID, "sr_create: one environment must fit a 1024-thread CTA");
    if (cfg->has_head && (!(cfg->head_length > 0.0) || !(cfg->head_radius > 0.0) || !(cfg->head_density > 0.0)))
      return fail(SR_E_INVALID, "sr_create: head_length, head_radius, head_density must be > 0");
  }
  if (cfg->contact_on) {
    if (cfg->math != SR_MATH_FAST) return fail(SR_E_INVALID, "sr_create: contact is built for SR_MATH_FAST only");
    if (cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE)
      return fail(SR_E_INVALID, "sr_create: contact cannot be combined with the Laplace filter / moving base yet");
    if (!(cfg->slip_velocity_tol > 0.0) || !(cfg->contact_k >= 0.0) || !(cfg->contact_nu >= 0.0))
      return fail(SR_E_INVALID, "sr_create: contact needs slip_velocity_tol > 0, k >= 0, nu >= 0");
    double nn = cfg->plane_normal[0] * cfg->plane_normal[0] + cfg->plane_normal[1] * cfg->plane_normal[1] + cfg->plane_normal[2] * cfg->plane_normal[2];
    if (!(nn > 0.0)) return fail(SR_E_INVALID, "sr_create: plane_normal must be non-zero");
    const bool z_up = cfg->plane_normal[0] == 0.0 && cfg->plane_normal[1] == 0.0 && cfg->plane_normal[2] > 0.0;
    if (!z_up && (cfg->n_rod_per_env > 1 || cfg->has_head))
      return fail(SR_E_INVALID, "sr_create: multi-rod assemblies stand on a plane with normal +z (FixedJoint2Rigid / BodyBoundaryCondition are written for z up)");
    if (!z_up && cfg->bc_kind != SR_BC_FREE && cfg->bc_kind != SR_BC_ONE_END_FIXED)
      return fail(SR_E_INVALID, "sr_create: a contact plane whose normal is not +z needs SR_BC_FREE or SR_BC_ONE_END_FIXED");
  }
  if (cfg->muscle_on) {
    if (cfg->math != SR_MATH_FAST) return fail(SR_E_INVALID, "sr_create: muscle torques are built for SR_MATH_FAST only");
    if (cfg->n_rod_per_env > 1 || cfg->has_head || cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE)
      return fail(SR_E_INVALID, "sr_create: muscle torques cannot be combined with assemblies / Laplace filter / moving base yet");
    if (!(cfg->muscle_period > 0.0) || !(cfg->muscle_ramp_up_time > 0.0))
      return fail(SR_E_INVALID, "sr_create: muscle_period and muscle_ramp_up_time must be > 0");
  }
  if (cfg->spline_dir_mask) {
    if (cfg->math != SR_MATH_FAST) return fail(SR_E_INVALID, "sr_create: spline torques are built for SR_MATH_FAST only");
    if (cfg->n_rod_per_env > 1 || cfg->has_head || cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE)
      return fail(SR_E_INVALID, "sr_create: spline torques cannot be combined with assemblies / Laplace filter / moving base yet");
    if (cfg->spline_dir_mask & ~7) return fail(SR_E_INVALID, "sr_create: spline_dir_mask has bits 0..2 only");
    if (cfg->spline_n_ctrl < 2 || cfg->spline_n_ctrl > 14) return fail(SR_E_INVALID, "sr_create: spline_n_ctrl must be in [2, 14]");
    if (!(cfg->spline_max_rate > 0.0)) return fail(SR_E_INVALID, "sr_create: spline_max_rate must be > 0 (inf = unlimited)");
  }
  if (cfg->tip_radius > 0.0) {
    if (cfg->dtype != SR_DTYPE_F64 || cfg->math != SR_MATH_FAST)
      return fail(SR_E_INVALID, "sr_create: tapered rods (tip_radius) are built for SR_DTYPE_F64 / SR_MATH_FAST");
    if (cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE || cfg->bc_kind == SR_BC_PENDULUM_SLIDER ||
        cfg->model != SR_MODEL_ROD || cfg->muscle_on || cfg->spline_dir_mask)
      return fail(SR_E_INVALID, "sr_create: tapered rods are built for SR_MODEL_ROD with the plane-contact / multi-rod model family");
  }
  if (cfg->sucker_on) {
    if (cfg->math != SR_MATH_FAST || cfg->model != SR_MODEL_ROD || cfg->laplace_filter_order != 0 || cfg->bc_kind == SR_BC_MOVING_BASE)
      return fail(SR_E_INVALID, "sr_create: ControllableFixConstraint is built for SR_MATH_FAST / SR_MODEL_ROD");
    if (cfg->sucker_index < 0 || cfg->sucker_index >= cfg->n_elem)
      return fail(SR_E_INVALID, "sr_create: sucker_index must address an element (0 .. n_elem - 1)");
  }
  if (cfg->taper_node_mean && !(cfg->tip_radius > 0.0))
    return fail(SR_E_INVALID, "sr_create: taper_node_mean needs tip_radius > 0");
  if (cfg->tm_muscle_on) {
    if (!(cfg->tip_radius > 0.0) || !(cfg->tm_radius_ref > 0.0))
      return fail(SR_E_INVALID, "sr_create: the transverse muscle is built for tapered rods (tip_radius > 0) and needs tm_radius_ref > 0");
  }
  if (cfg->muscle_layers_on) {
    if (!cfg->tm_muscle_on || !(cfg->tm_max_stress != 0.0) || !cfg->has_head || cfg->dtype != SR_DTYPE_F64 || cfg->n_elem < 3)
      return fail(SR_E_INVALID, "sr_create: muscle_layers_on needs tm_muscle_on (non-zero tm_max_stress), FP64, n_elem >= 3 and a multi-rod assembly with a head");
    if ((cfg->n_rod_per_env > 1 ? cfg->n_rod_per_env : 1) * (cfg->n_elem + 1) + 1 > 384)
      return fail(SR_E_INVALID, "sr_create: muscle_layers_on: the assembly must fit one 384-thread CTA (n_rod * (n_elem + 1) + 1 <= 384)");
    if (cfg->contact_on) return fail(SR_E_INVALID, "sr_create: muscle_layers_on is built without plane contact");
    if (cfg->n_fixed_sucker < 0 || cfg->n_fixed_sucker > 3) return fail(SR_E_INVALID, "sr_create: n_fixed_sucker must be 0 .. 3");
    for (int a = 0; a < cfg->n_fixed_sucker; a++) {
      if (cfg->fixed_sucker_index[a] < 0 || cfg->fixed_sucker_index[a] >= cfg->n_elem)
        return fail(SR_E_INVALID, "sr_create: fixed_sucker_index must address an element (0 .. n_elem - 1)");
      for (int b = 0; b < a; b++)
        if (cfg->fixed_sucker_index[a] == cfg->fixed_sucker_index[b])
          return fail(SR_E_INVALID, "sr_create: fixed_sucker_index entries must be distinct");
    }
  } else if (cfg->head_fixed || cfg->n_fixed_sucker) {
    return fail(SR_E_INVALID, "sr_create: head_fixed / n_fixed_sucker are honoured by the muscle-layer kernel only (muscle_layers_on)");
  }
  if (cfg->model == SR_MODEL_SOFT_PENDULUM_3D && (cfg->bc_kind != SR_BC_MOVING_BASE || !(cfg->base_move_period > 0.0)))
    return fail(SR_E_INVALID, "sr_create: SoftPendulum3D needs SR_BC_MOVING_BASE and base_move_period > 0");
  if (!(cfg->dt > 0.0) || !(cfg->base_length > 0.0) || !(cfg->base_radius > 0.0) || !(cfg->density > 0.0) ||
      !(cfg->youngs_modulus > 0.0))
    return fail(SR_E_INVALID, "sr_create: dt, base_length, base_radius, density, youngs_modulus must be > 0");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SR_E_NO_DEVICE, "sr_create: no CUDA device (this library has no CPU fallback)");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(SR_E_INVALID, "sr_create: bad device ordinal");
  SR_CUDA(cudaSetDevice(cfg->device));
  if (cfg->n_elem > 1023) {
    const int C = lean_cluster_size(cfg->n_elem);
    const int n_active = with_cluster_model(lean_cluster_model(cfg->laplace_filter_order, cfg->bc_kind, loads, cfg->muscle_on,
                                                               cfg->spline_dir_mask != 0),
                                            [&](auto m) { return sr::lean_cluster_max_active<decltype(m)::value>(C); });
    if (n_active < 1)
      return fail(SR_E_CUDA, "sr_create: n_elem = " + std::to_string(cfg->n_elem) + " needs a cluster of " + std::to_string(C) +
                                 " CTAs of 512 threads, and this device cannot launch one");
  }

  sr_handle *h = new (std::nothrow) sr_handle();
  if (!h) return fail(SR_E_ALLOC, "sr_create: out of host memory");
  h->cfg = *cfg;
  h->n_rod = cfg->n_rod_per_env > 1 ? cfg->n_rod_per_env : 1;
  h->init_dim = 9 * (h->n_rod + (cfg->has_head ? 1 : 0));
  // nodes 0..n need n+1 slots in 32*EPL
  h->epl = (cfg->n_elem + 1 <= 32) ? 1 : (cfg->n_elem + 1 <= 64) ? 2 : 4;
  // the warp-per-rod kernel reads 32*EPL slots per row; longer rods (packed kernel only) round up to 32
  h->stride = (cfg->n_elem + 1 <= 128) ? 32 * h->epl : 32 * ((cfg->n_elem + 1 + 31) / 32);
  h->elem_size = cfg->dtype == SR_DTYPE_F32 ? 4 : 8;
  if (cfg->model == SR_MODEL_SOFT_PENDULUM) { h->obs_dim = 4; h->action_dim = 1; }
  else if (cfg->model == SR_MODEL_SOFT_PENDULUM_3D) { h->obs_dim = 9; h->action_dim = 2; }
  else { h->obs_dim = 6; h->action_dim = 0; }
  const size_t n_env = (size_t)cfg->n_env, n_rods = n_env * h->n_rod;
  const size_t state_bytes = n_rods * sr::N_FIELDS * h->stride * h->elem_size;
  cudaError_t e;
  if ((e = cudaMalloc(&h->state, state_bytes)) != cudaSuccess ||
      (e = cudaMalloc(&h->bc, n_rods * sr::BC_DIM * h->elem_size)) != cudaSuccess ||
      (e = cudaMalloc(&h->head, n_env * sr::HEAD_DIM * h->elem_size)) != cudaSuccess ||
      (e = cudaMalloc(&h->aux, n_env * sr::AUX_DIM * h->elem_size)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_action, n_env * (h->action_dim ? h->action_dim : 1) * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_obs, n_env * h->obs_dim * sizeof(float))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_reward, n_env * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_term, n_env)) != cudaSuccess ||
      (e = cudaMalloc(&h->d_init, n_env * h->init_dim * sizeof(double))) != cudaSuccess ||
      (e = cudaMalloc(&h->d_idx, n_env * sizeof(int32_t))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_action, n_env * (h->action_dim ? h->action_dim : 1) * sizeof(float))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_obs, n_env * h->obs_dim * sizeof(float))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_reward, n_env * sizeof(double))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_term, n_env)) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_init, n_env * h->init_dim * sizeof(double))) != cudaSuccess ||
      (e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMalloc(&h->redo, n_env * sizeof(int))) != cudaSuccess ||
      (e = cudaMemset(h->redo, 0, n_env * sizeof(int))) != cudaSuccess ||
      (e = cudaMalloc(&h->redo_count, 5 * sizeof(unsigned long long))) != cudaSuccess ||     // [0] total, [1..3] by cause, [4] not planar (lean kernel)
      (e = cudaMemset(h->redo_count, 0, 5 * sizeof(unsigned long long))) != cudaSuccess ||
      (e = cudaMallocHost(&h->h_redo_count, 5 * sizeof(unsigned long long))) != cudaSuccess ||
      (e = cudaEventCreateWithFlags(&h->pair_event, cudaEventDisableTiming)) != cudaSuccess ||
      (e = cudaMemset(h->state, 0, state_bytes)) != cudaSuccess) {
    std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
    sr_destroy(h);
    return fail(SR_E_ALLOC, m);
  }
  if (cfg->muscle_on) {
    h->muscle_dim = cfg->n_elem + 2;
    const size_t mb = n_env * h->muscle_dim * sizeof(double);
    if ((e = cudaMalloc(&h->muscle, mb)) != cudaSuccess || (e = cudaMemset(h->muscle, 0, mb)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->spline_dir_mask) {
    const int P = cfg->spline_n_ctrl;
    h->spline_dim = 3 * (2 * P + 2) + 3 * cfg->n_elem;
    const size_t sb = n_env * h->spline_dim * sizeof(double), tb = (size_t)(P + 1) * P * 4 * sizeof(double);
    std::vector<double> tab((size_t)(P + 1) * P * 4);
    sr_spline_basis(P, cfg->base_length, tab.data());
    if ((e = cudaMalloc(&h->spline, sb)) != cudaSuccess || (e = cudaMemset(h->spline, 0, sb)) != cudaSuccess ||
        (e = cudaMalloc(&h->spline_tab, tb)) != cudaSuccess ||
        (e = cudaMemcpy(h->spline_tab, tab.data(), tb, cudaMemcpyHostToDevice)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->sucker_on) {
    const size_t sb = n_rods * h->elem_size;
    std::vector<int32_t> idx(n_rods, cfg->sucker_index);
    if ((e = cudaMalloc(&h->sucker, sb)) != cudaSuccess || (e = cudaMemset(h->sucker, 0, sb)) != cudaSuccess ||
        (e = cudaMalloc(&h->sucker_idx, n_rods * sizeof(int32_t))) != cudaSuccess ||
        (e = cudaMemcpy(h->sucker_idx, idx.data(), n_rods * sizeof(int32_t), cudaMemcpyHostToDevice)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->tm_muscle_on) {
    const size_t sb = n_rods * h->elem_size;
    if ((e = cudaMalloc(&h->tm_act, sb)) != cudaSuccess || (e = cudaMemset(h->tm_act, 0, sb)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->muscle_layers_on) {
    const size_t sb = n_rods * 3 * (size_t)cfg->n_elem * sizeof(double);
    if ((e = cudaMalloc(&h->mus_act, sb)) != cudaSuccess || (e = cudaMemset(h->mus_act, 0, sb)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->n_fixed_sucker > 0) {
    const size_t sb = n_rods * 3 * sizeof(double);
    if ((e = cudaMalloc(&h->msucker, sb)) != cudaSuccess || (e = cudaMemset(h->msucker, 0, sb)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  if (cfg->tip_radius > 0.0) {
    // SURVEY A.1 / A.4 per element: radius_k = linspace(base, tip, n)[k]; uniform rest lengths L/n (the per-element
    // deviation of the reference's linspace positions is carried by F_GAMMA as for uniform rods)
    const int n = cfg->n_elem, st = h->stride;
    const double PI = 3.141592653589793, rl = cfg->base_length / n, E = cfg->youngs_modulus;
    const double G = cfg->shear_modulus > 0.0 ? cfg->shear_modulus : E / (2.0 * (1.0 + 0.5)), ac = 27.0 / 28.0;
    std::vector<double> tab((size_t)sr::ET_FIELDS * st, 1.0), rad(n), Bel0(n), Bel2(n), mel(n), J0(n), J2(n);
    const double stepr = n > 1 ? (cfg->tip_radius - cfg->base_radius) / (n - 1) : 0.0;
    const double stepn = (cfg->tip_radius - cfg->base_radius) / n;
    for (int k = 0; k < n; k++) {
      rad[k] = (k == n - 1 && n > 1) ? cfg->tip_radius : k * stepr + cfg->base_radius;
      if (cfg->taper_node_mean) {
        // radius = np.linspace(base, tip, n + 1); element radius = mean of its two nodes (arm_push_env.py:161-175)
        const double r0 = k * stepn + cfg->base_radius, r1 = (k + 1 == n) ? cfg->tip_radius : (k + 1) * stepn + cfg->base_radius;
        rad[k] = (r0 + r1) / 2.0;
      }
      // TransverseMuscle(rest_muscle_area=(radius / radius_base)**2, max_muscle_stress) handing -max_stress to its base
      // class (envs/octopus/build.py:329-333): the per-element factor of the muscle force
      tab[sr::ET_TM * st + k] = cfg->tm_muscle_on ? -cfg->tm_max_stress * ((rad[k] / cfg->tm_radius_ref) * (rad[k] / cfg->tm_radius_ref)) : 0.0;
      const double A0 = PI * rad[k] * rad[k], I1 = A0 * A0 / (4.0 * PI), I3 = 2.0 * I1;
      J0[k] = I1 * cfg->density * rl; J2[k] = I3 * cfg->density * rl;
      Bel0[k] = E * I1; Bel2[k] = G * I3;
      mel[k] = cfg->density * PI * (rad[k] * rad[k]) * rl;
      tab[sr::ET_REST_LEN * st + k] = rl;
      tab[sr::ET_S0 * st + k] = ac * G * A0; tab[sr::ET_S2 * st + k] = E * A0;
      tab[sr::ET_J0 * st + k] = J0[k]; tab[sr::ET_J2 * st + k] = J2[k];
      tab[sr::ET_VOL_PI * st + k] = (rad[k] * rad[k]) * rl;
    }
    for (int k = 0; k < n - 1; k++) {
      tab[sr::ET_REST_VOR * st + k] = rl;
      tab[sr::ET_B0 * st + k] = (Bel0[k + 1] * rl + Bel0[k] * rl) / (rl + rl);
      tab[sr::ET_B2 * st + k] = (Bel2[k + 1] * rl + Bel2[k] * rl) / (rl + rl);
    }
    std::vector<double> mnode(n + 1, 0.0);
    for (int k = 0; k < n; k++) { mnode[k] += 0.5 * mel[k]; mnode[k + 1] += 0.5 * mel[k]; }
    for (int k = 0; k <= n; k++) tab[sr::ET_MASS * st + k] = mnode[k];
    for (int k = 0; k < n; k++) {
      double em = 0.5 * (mnode[k + 1] + mnode[k]);
      if (k == 0) em += 0.5 * mnode[0];
      if (k == n - 1) em += 0.5 * mnode[n];
      const double c = cfg->damping_constant >= 0.0 ? cfg->damping_constant : 0.0;
      tab[sr::ET_LOGCW0 * st + k] = -c * cfg->dt * em / J0[k];
      tab[sr::ET_LOGCW2 * st + k] = -c * cfg->dt * em / J2[k];
    }
    const size_t tb = tab.size() * sizeof(double);
    if ((e = cudaMalloc(&h->elem_tab, tb)) != cudaSuccess ||
        (e = cudaMemcpy(h->elem_tab, tab.data(), tb, cudaMemcpyHostToDevice)) != cudaSuccess) {
      std::string m = std::string("sr_create: allocation failed: ") + cudaGetErrorString(e);
      sr_destroy(h);
      return fail(SR_E_ALLOC, m);
    }
  }
  for (int i = 0; i < 5; i++) h->h_redo_count[i] = 0;
  fill_args<double>(*cfg, h->stride, h->a64);
  h->a64.spline = h->spline; h->a64.spline_tab = h->spline_tab;
  h->a64.redo = h->redo;
  h->a64.sucker = (const double *)h->sucker; h->a64.sucker_index = cfg->sucker_index; h->a64.elem_tab = (const double *)h->elem_tab;
  h->a64.sucker_idx = h->sucker_idx; h->a64.tm_act = (const double *)h->tm_act;
  h->a64.muscle = h->muscle;
  h->a64.mus_act = h->mus_act; h->a64.head_fixed = cfg->head_fixed;
  h->a64.lm_gain = cfg->muscle_layers_on ? cfg->lm_max_stress / -cfg->tm_max_stress : 0.0;
  for (int m = 0; m < 2; m++) { h->a64.lm_px[m] = cfg->lm_px[m]; h->a64.lm_py[m] = cfg->lm_py[m]; h->a32.lm_px[m] = h->a32.lm_py[m] = 0.0f; }
  h->a32.mus_act = nullptr; h->a32.head_fixed = 0; h->a32.lm_gain = 0.0f;
  h->a64.msucker = h->msucker; h->a64.msucker_n = cfg->n_fixed_sucker; h->a32.msucker = nullptr; h->a32.msucker_n = 0;
  for (int a = 0; a < 3; a++) h->a64.msucker_loc[a] = h->a32.msucker_loc[a] = (a < cfg->n_fixed_sucker) ? cfg->fixed_sucker_index[a] : -1;
  h->a64.state = (double *)h->state; h->a64.bc = (const double *)h->bc; h->a64.aux = (double *)h->aux;
  h->a64.action_dim = h->action_dim; h->a64.obs_dim = h->obs_dim; h->a64.head = (double *)h->head;
  fill_args<float>(*cfg, h->stride, h->a32);
  h->a32.spline = h->spline; h->a32.spline_tab = h->spline_tab;
  h->a32.redo = h->redo;
  h->a32.sucker = (const float *)h->sucker; h->a32.sucker_index = cfg->sucker_index;
  h->a32.sucker_idx = h->sucker_idx; h->a32.tm_act = nullptr;
  h->a32.muscle = h->muscle;
  h->a32.state = (float *)h->state; h->a32.bc = (const float *)h->bc; h->a32.aux = (float *)h->aux;
  h->a32.action_dim = h->action_dim; h->a32.obs_dim = h->obs_dim; h->a32.head = (float *)h->head;
  *out = h;
  return SR_OK;
}

void sr_destroy(sr_handle *h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  cudaFree(h->mus_act); cudaFree(h->msucker);
  cudaFree(h->state); cudaFree(h->bc); cudaFree(h->aux); cudaFree(h->rest_kappa); cudaFree(h->head); cudaFree(h->muscle); cudaFree(h->spline); cudaFree(h->spline_tab); cudaFree(h->redo); cudaFree(h->redo_count); cudaFree(h->sucker); cudaFree(h->sucker_idx); cudaFree(h->tm_act); cudaFree(h->ext_force); cudaFree(h->ext_couple); cudaFree(h->elem_tab); cudaFree(h->sk_scratch); cudaFree(h->sk_flag); cudaFree(h->copy_stage); cudaFreeHost(h->h_redo_count); if (h->pair_event) cudaEventDestroy(h->pair_event); cudaFree(h->d_action); cudaFree(h->d_obs);
  cudaFree(h->d_reward); cudaFree(h->d_term); cudaFree(h->d_init); cudaFree(h->d_idx);
  cudaFreeHost(h->h_action); cudaFreeHost(h->h_obs); cudaFreeHost(h->h_reward); cudaFreeHost(h->h_term);
  cudaFreeHost(h->h_init);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

int sr_obs_dim(const sr_handle *h) { return h ? h->obs_dim : 0; }
int sr_action_dim(const sr_handle *h) { return h ? h->action_dim : 0; }
int sr_init_dim(const sr_handle *h) { return h ? h->init_dim : 0; }
int64_t sr_launch_count(const sr_handle *h) { return h ? h->launches : 0; }
static void read_fallback_counters(const sr_handle *h, unsigned long long (&v)[5]) {
  for (int i = 0; i < 5; i++) v[i] = 0;
  if (!h || !h->redo_count) return;
  int prev = 0;
  cudaGetDevice(&prev); cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  cudaMemcpy(v, h->redo_count, sizeof(v), cudaMemcpyDeviceToHost);
  cudaSetDevice(prev);
}
int64_t sr_fallback_count(const sr_handle *h) {
  unsigned long long v[5];
  read_fallback_counters(h, v);
  return (int64_t)v[0];
}
int sr_fallback_causes(const sr_handle *h, int64_t out[3]) {
  if (!h || !out) return fail(SR_E_INVALID, "sr_fallback_causes: null argument");
  unsigned long long v[5];
  read_fallback_counters(h, v);
  for (int i = 0; i < 3; i++) out[i] = (int64_t)v[1 + i];
  return SR_OK;
}
int64_t sr_nonplanar_count(const sr_handle *h) {
  unsigned long long v[5];
  read_fallback_counters(h, v);
  return (int64_t)v[4];
}

int sr_reset(sr_handle *h, const int32_t *env_idx_dev, int n, const double *init_dev, void *stream) {
  if (!h || !init_dev) return fail(SR_E_INVALID, "sr_reset: null argument");
  if (n < 0 || n > h->cfg.n_env) return fail(SR_E_INVALID, "sr_reset: n out of range");
  if (n == 0) return SR_OK;
  SR_CUDA(cudaSetDevice(h->cfg.device));
  const int nblk = n * h->n_rod;
  if (h->cfg.dtype == SR_DTYPE_F32) {
    sr::rod_reset_kernel<float><<<nblk, 64, 0, (cudaStream_t)stream>>>(
        (float *)h->state, (float *)h->bc, (float *)h->aux, env_idx_dev, n, init_dev, h->cfg.n_elem,
        h->stride, h->cfg.base_length, h->n_rod, h->init_dim, h->muscle, h->muscle_dim, h->spline, h->spline_dim);
    if (h->cfg.has_head)
      sr::head_reset_kernel<float><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
          (float *)h->head, env_idx_dev, n, init_dev, h->init_dim, h->n_rod, h->cfg.head_length);
  } else {
    sr::rod_reset_kernel<double><<<nblk, 64, 0, (cudaStream_t)stream>>>(
        (double *)h->state, (double *)h->bc, (double *)h->aux, env_idx_dev, n, init_dev, h->cfg.n_elem,
        h->stride, h->cfg.base_length, h->n_rod, h->init_dim, h->muscle, h->muscle_dim, h->spline, h->spline_dim);
    if (h->cfg.has_head)
      sr::head_reset_kernel<double><<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
          (double *)h->head, env_idx_dev, n, init_dev, h->init_dim, h->n_rod, h->cfg.head_length);
  }
  h->launches++;
  SR_CUDA(cudaGetLastError());
  return SR_OK;
}

int sr_step(sr_handle *h, const float *action_dev, int n_substeps, float *obs_dev, double *reward_dev,
            uint8_t *terminated_dev, void *stream) {
  if (!h || !obs_dev || !reward_dev || !terminated_dev) return fail(SR_E_INVALID, "sr_step: null output pointer");
  if (h->action_dim > 0 && !action_dev) return fail(SR_E_INVALID, "sr_step: action required for this model");
  if (n_substeps < 0) return fail(SR_E_INVALID, "sr_step: n_substeps < 0");
  SR_CUDA(cudaSetDevice(h->cfg.device));
  if (h->cfg.dtype == SR_DTYPE_F32) {
    sr::RodArgs<float> A = h->a32;
    A.action = action_dev; A.obs = obs_dev; A.reward = reward_dev; A.terminated = terminated_dev;
    A.n_substeps = n_substeps;
    return launch_step<float>(h, A, (cudaStream_t)stream);
  }
  sr::RodArgs<double> A = h->a64;
  A.action = action_dev; A.obs = obs_dev; A.reward = reward_dev; A.terminated = terminated_dev;
  A.n_substeps = n_substeps;
  return launch_step<double>(h, A, (cudaStream_t)stream);
}

int sr_observe(sr_handle *h, const float *prev_action_dev, float *obs_dev, void *stream) {
  if (!h || !obs_dev) return fail(SR_E_INVALID, "sr_observe: null argument");
  SR_CUDA(cudaSetDevice(h->cfg.device));
  int bs = 128, grid = (h->cfg.n_env + bs - 1) / bs;
  if (h->cfg.dtype == SR_DTYPE_F32)
    sr::rod_observe_kernel<float><<<grid, bs, 0, (cudaStream_t)stream>>>(
        (const float *)h->state, prev_action_dev, obs_dev, h->cfg.n_env, h->cfg.n_elem, h->stride,
        h->cfg.model, h->action_dim, h->obs_dim);
  else
    sr::rod_observe_kernel<double><<<grid, bs, 0, (cudaStream_t)stream>>>(
        (const double *)h->state, prev_action_dev, obs_dev, h->cfg.n_env, h->cfg.n_elem, h->stride,
        h->cfg.model, h->action_dim, h->obs_dim);
  h->launches++;
  SR_CUDA(cudaGetLastError());
  return SR_OK;
}

int sr_reset_host(sr_handle *h, const int32_t *env_idx_host, int n, const double *init_host) {
  if (!h || !init_host) return fail(SR_E_INVALID, "sr_reset_host: null argument");
  if (n < 0 || n > h->cfg.n_env) return fail(SR_E_INVALID, "sr_reset_host: n out of range");
  if (n == 0) return SR_OK;
  SR_CUDA(cudaSetDevice(h->cfg.device));
  cudaStream_t s = h->own_stream;
  memcpy(h->h_init, init_host, (size_t)n * h->init_dim * sizeof(double));
  SR_CUDA(cudaMemcpyAsync(h->d_init, h->h_init, (size_t)n * h->init_dim * sizeof(double), cudaMemcpyHostToDevice, s));
  if (env_idx_host)
    SR_CUDA(cudaMemcpyAsync(h->d_idx, env_idx_host, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  int rc = sr_reset(h, env_idx_host ? h->d_idx : nullptr, n, h->d_init, s);
  if (rc != SR_OK) return rc;
  SR_CUDA(cudaStreamSynchronize(s));
  return SR_OK;
}

int sr_step_host(sr_handle *h, const float *action_host, int n_substeps, float *obs_host,
                 double *reward_host, uint8_t *terminated_host) {
  if (!h || !obs_host || !reward_host || !terminated_host) return fail(SR_E_INVALID, "sr_step_host: null output pointer");
  if (h->action_dim > 0 && !action_host) return fail(SR_E_INVALID, "sr_step_host: action required for this model");
  SR_CUDA(cudaSetDevice(h->cfg.device));
  cudaStream_t s = h->own_stream;
  const size_t n_env = (size_t)h->cfg.n_env;
  if (h->action_dim > 0) {
    memcpy(h->h_action, action_host, n_env * h->action_dim * sizeof(float));
    SR_CUDA(cudaMemcpyAsync(h->d_action, h->h_action, n_env * h->action_dim * sizeof(float),
                            cudaMemcpyHostToDevice, s));
  }
  int rc = sr_step(h, h->action_dim > 0 ? h->d_action : nullptr, n_substeps, h->d_obs, h->d_reward, h->d_term, s);
  if (rc != SR_OK) return rc;
  SR_CUDA(cudaMemcpyAsync(h->h_obs, h->d_obs, n_env * h->obs_dim * sizeof(float), cudaMemcpyDeviceToHost, s));
  SR_CUDA(cudaMemcpyAsync(h->h_reward, h->d_reward, n_env * sizeof(double), cudaMemcpyDeviceToHost, s));
  SR_CUDA(cudaMemcpyAsync(h->h_term, h->d_term, n_env, cudaMemcpyDeviceToHost, s));
  SR_CUDA(cudaStreamSynchronize(s));
  memcpy(obs_host, h->h_obs, n_env * h->obs_dim * sizeof(float));
  memcpy(reward_host, h->h_reward, n_env * sizeof(double));
  memcpy(terminated_host, h->h_term, n_env);
  return SR_OK;
}

int sr_get_state(sr_handle *h, sr_state_view *out) {
  if (!h || !out) return fail(SR_E_INVALID, "sr_get_state: null argument");
  out->base = h->state;
  out->n_env = h->cfg.n_env * h->n_rod;   /* rod rows: env-major, rod-minor */
  out->n_fields = sr::N_FIELDS; out->stride = h->stride;
  out->elem_size = (int32_t)h->elem_size;
  out->f_position = sr::F_POS; out->f_velocity = sr::F_VEL; out->f_director = sr::F_DIR;
  out->f_omega = sr::F_OMEGA; out->f_tangents = sr::F_TAN; out->f_kappa = sr::F_KAPPA;
  out->f_sigma = sr::F_SIGMA; out->f_dilatation = sr::F_DIL;
  return SR_OK;
}

int sr_get_muscle(sr_handle *h, double **muscle_dev, int32_t *dim) {
  if (!h || !muscle_dev || !dim) return fail(SR_E_INVALID, "sr_get_muscle: null argument");
  if (!h->muscle) return fail(SR_E_INVALID, "sr_get_muscle: handle was created without muscle_on");
  *muscle_dev = h->muscle; *dim = h->muscle_dim;
  return SR_OK;
}

int sr_get_spline(sr_handle *h, double **spline_dev, int32_t *dim) {
  if (!h || !spline_dev || !dim) return fail(SR_E_INVALID, "sr_get_spline: null argument");
  if (!h->spline) return fail(SR_E_INVALID, "sr_get_spline: handle was created without spline_dir_mask");
  *spline_dev = h->spline; *dim = h->spline_dim;
  return SR_OK;
}

int sr_spline_basis(int32_t P, double base_length, double *out) {
  if (!out || P < 2 || P > 14 || !(base_length > 0.0)) return fail(SR_E_INVALID, "sr_spline_basis: bad argument");
  // not-a-knot cubic through x_m = m dx, m = 0..N (N = P + 1 intervals), one unit control value at a time:
  // second derivatives M from  M_{m-1} + 4 M_m + M_{m+1} = 6 (y_{m-1} - 2 y_m + y_{m+1}) / dx^2  (m = 1..N-1)
  // and third-derivative continuity at x_1 and x_{N-1}; solved densely (N + 1 <= 16 unknowns).
  const int N = P + 1, K = N + 1;
  const double dx = base_length / N;
  for (int i = 0; i < P; i++) {
    double y[16] = {0}, Am[16][17] = {{0}};
    y[i + 1] = 1.0;
    Am[0][0] = 1.0; Am[0][1] = -2.0; Am[0][2] = 1.0;
    Am[N][N] = 1.0; Am[N][N - 1] = -2.0; Am[N][N - 2] = 1.0;
    for (int m = 1; m < N; m++) {
      Am[m][m - 1] = 1.0; Am[m][m] = 4.0; Am[m][m + 1] = 1.0;
      Am[m][K] = 6.0 * (y[m - 1] - 2.0 * y[m] + y[m + 1]) / (dx * dx);
    }
    for (int c = 0; c < K; c++) {   // Gaussian elimination with partial pivoting
      int piv = c;
      for (int r2 = c + 1; r2 < K; r2++) if (fabs(Am[r2][c]) > fabs(Am[piv][c])) piv = r2;
      for (int k = 0; k <= K; k++) std::swap(Am[c][k], Am[piv][k]);
      for (int r2 = 0; r2 < K; r2++) {
        if (r2 == c) continue;
        const double f = Am[r2][c] / Am[c][c];
        for (int k = c; k <= K; k++) Am[r2][k] -= f * Am[c][k];
      }
    }
    double M[16];
    for (int m = 0; m < K; m++) M[m] = Am[m][K] / Am[m][m];
    for (int m = 0; m < N; m++) {
      double *o = out + ((size_t)m * P + i) * 4;
      o[0] = y[m];
      o[1] = (y[m + 1] - y[m]) / dx - dx * (2.0 * M[m] + M[m + 1]) / 6.0;
      o[2] = 0.5 * M[m];
      o[3] = (M[m + 1] - M[m]) / (6.0 * dx);
    }
  }
  return SR_OK;
}

int sr_get_rest_kappa(sr_handle *h, void **rest_kappa_dev) {
  if (!h || !rest_kappa_dev) return fail(SR_E_INVALID, "sr_get_rest_kappa: null argument");
  if (h->cfg.math != SR_MATH_FAST) return fail(SR_E_INVALID, "sr_get_rest_kappa: rest curvature is built for SR_MATH_FAST only");
  // (above 1023 elements only the rods on the plane / with the muscle wave step on a kernel that reads it: the plane
  // and muscle models on clusters)
  if (h->cfg.n_elem > 1023 && !h->cfg.contact_on && !h->cfg.muscle_on)
    return fail(SR_E_INVALID, "sr_get_rest_kappa: rest curvature is built for n_elem <= 1023, and above for rods with "
                              "contact_on or muscle_on");
  if (!h->rest_kappa) {
    SR_CUDA(cudaSetDevice(h->cfg.device));
    size_t bytes = (size_t)h->cfg.n_env * h->n_rod * 3 * h->stride * h->elem_size;
    SR_CUDA(cudaMalloc(&h->rest_kappa, bytes));
    SR_CUDA(cudaMemset(h->rest_kappa, 0, bytes));
    h->a64.rest_kappa = (const double *)h->rest_kappa;
    h->a32.rest_kappa = (const float *)h->rest_kappa;
  }
  *rest_kappa_dev = h->rest_kappa;
  return SR_OK;
}

int sr_get_sucker(sr_handle *h, void **ratio_dev) {
  if (!h || !ratio_dev) return fail(SR_E_INVALID, "sr_get_sucker: null argument");
  if (!h->sucker) return fail(SR_E_INVALID, "sr_get_sucker: handle was created without sucker_on");
  *ratio_dev = h->sucker;
  return SR_OK;
}

int sr_get_sucker_index(sr_handle *h, int32_t **index_dev) {
  if (!h || !index_dev) return fail(SR_E_INVALID, "sr_get_sucker_index: null argument");
  if (!h->sucker_idx) return fail(SR_E_INVALID, "sr_get_sucker_index: handle was created without sucker_on");
  *index_dev = h->sucker_idx;
  return SR_OK;
}

int sr_get_fixed_suckers(sr_handle *h, void **ratio_dev) {
  if (!h || !ratio_dev) return fail(SR_E_INVALID, "sr_get_fixed_suckers: null argument");
  if (!h->msucker) return fail(SR_E_INVALID, "sr_get_fixed_suckers: handle was created without n_fixed_sucker");
  *ratio_dev = h->msucker;
  return SR_OK;
}

int sr_get_muscle_activation(sr_handle *h, void **activation_dev) {
  if (!h || !activation_dev) return fail(SR_E_INVALID, "sr_get_muscle_activation: null argument");
  if (!h->mus_act) return fail(SR_E_INVALID, "sr_get_muscle_activation: handle was created without muscle_layers_on");
  *activation_dev = h->mus_act;
  return SR_OK;
}

int sr_get_tm_activation(sr_handle *h, void **activation_dev) {
  if (!h || !activation_dev) return fail(SR_E_INVALID, "sr_get_tm_activation: null argument");
  if (!h->tm_act) return fail(SR_E_INVALID, "sr_get_tm_activation: handle was created without tm_muscle_on");
  *activation_dev = h->tm_act;
  return SR_OK;
}

int sr_get_ext_loads(sr_handle *h, void **force_dev, void **couple_dev) {
  if (!h || !force_dev || !couple_dev) return fail(SR_E_INVALID, "sr_get_ext_loads: null argument");
  if (h->cfg.math != SR_MATH_FAST || h->cfg.model != SR_MODEL_ROD || h->cfg.laplace_filter_order != 0 ||
      h->cfg.bc_kind == SR_BC_MOVING_BASE)
    return fail(SR_E_INVALID, "sr_get_ext_loads: external loads are built for SR_MATH_FAST / SR_MODEL_ROD without filter / moving base");
  if (h->cfg.n_elem > 1023) return fail(SR_E_INVALID, "sr_get_ext_loads: external loads are built for n_elem <= 1023");
  if (!h->ext_force) {
    SR_CUDA(cudaSetDevice(h->cfg.device));
    const size_t bytes = (size_t)h->cfg.n_env * h->n_rod * 3 * h->stride * h->elem_size;
    SR_CUDA(cudaMalloc(&h->ext_force, bytes));
    SR_CUDA(cudaMalloc(&h->ext_couple, bytes));
    SR_CUDA(cudaMemset(h->ext_force, 0, bytes));
    SR_CUDA(cudaMemset(h->ext_couple, 0, bytes));
    h->a64.ext_force = (const double *)h->ext_force; h->a64.ext_couple = (const double *)h->ext_couple;
    h->a32.ext_force = (const float *)h->ext_force; h->a32.ext_couple = (const float *)h->ext_couple;
  }
  *force_dev = h->ext_force; *couple_dev = h->ext_couple;
  return SR_OK;
}

int sr_get_head(sr_handle *h, void **head_dev, int32_t *dim) {
  if (!h || !head_dev || !dim) return fail(SR_E_INVALID, "sr_get_head: null argument");
  if (!h->cfg.has_head) return fail(SR_E_INVALID, "sr_get_head: this handle has no rigid head");
  *head_dev = h->head;
  *dim = sr::HEAD_DIM;
  return SR_OK;
}

int sr_get_aux(sr_handle *h, void **aux_dev, int32_t *dim) {
  if (!h || !aux_dev || !dim) return fail(SR_E_INVALID, "sr_get_aux: null argument");
  *aux_dev = h->aux;   /* element type follows sr_config.dtype */
  *dim = sr::AUX_DIM;
  return SR_OK;
}

int sr_set_state(sr_handle *h, const sr_state_view *src, void *stream) {
  if (!h || !src || !src->base) return fail(SR_E_INVALID, "sr_set_state: null argument");
  if (src->n_env != h->cfg.n_env * h->n_rod || src->n_fields != sr::N_FIELDS || src->stride != h->stride ||
      src->elem_size != (int32_t)h->elem_size)
    return fail(SR_E_INVALID, "sr_set_state: layout mismatch");
  SR_CUDA(cudaSetDevice(h->cfg.device));
  size_t bytes = (size_t)h->cfg.n_env * h->n_rod * sr::N_FIELDS * h->stride * h->elem_size;
  SR_CUDA(cudaMemcpyAsync(h->state, src->base, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SR_OK;
}

int sr_copy_from(sr_handle *dst, sr_handle *src, void *stream) {
  if (!dst || !src) return fail(SR_E_INVALID, "sr_copy_from: null argument");
  const sr_config &a = dst->cfg, &b = src->cfg;
  if (a.n_env != b.n_env || !same_env_shape(dst, src))
    return fail(SR_E_INVALID, "sr_copy_from: the two handles were created with different shapes");
  SR_CUDA(cudaSetDevice(a.device));
  cudaStream_t s = (cudaStream_t)stream;
  const int rc = alloc_lazy_like(dst, src);
  if (rc != SR_OK) return rc;
  EnvBuf d[EB_COUNT], sb[EB_COUNT];
  env_buffers(dst, d);
  env_buffers(src, sb);
  for (int k = 0; k < EB_COUNT; k++) {
    if (!d[k].base || !sb[k].base) continue;
    const size_t bytes = (size_t)a.n_env * d[k].bytes;
    SR_CUDA(a.device == b.device ? cudaMemcpyAsync(d[k].base, sb[k].base, bytes, cudaMemcpyDeviceToDevice, s)
                                 : cudaMemcpyPeerAsync(d[k].base, a.device, sb[k].base, b.device, bytes, s));
  }
  return SR_OK;
}

int sr_copy_envs(sr_handle *dst, const int32_t *dst_idx_dev, const sr_handle *src, const int32_t *src_idx_dev, int n,
                 void *stream) {
  if (!dst || !src) return fail(SR_E_INVALID, "sr_copy_envs: null handle");
  if (n < 0 || n > dst->cfg.n_env) return fail(SR_E_INVALID, "sr_copy_envs: n out of range (0 <= n <= n_env of dst)");
  if (n == 0) return SR_OK;
  if (!dst_idx_dev || !src_idx_dev) return fail(SR_E_INVALID, "sr_copy_envs: null index array");
  if (dst->cfg.device != src->cfg.device)
    return fail(SR_E_INVALID, "sr_copy_envs: the two handles are on different devices (sr_copy_from copies across devices)");
  if (!same_env_shape(dst, src))
    return fail(SR_E_INVALID, "sr_copy_envs: the two handles were created with different shapes (n_elem, n_rod, dtype, model, "
                              "head, muscle or spline forcing)");
  SR_CUDA(cudaSetDevice(dst->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  const int rc = alloc_lazy_like(dst, src);
  if (rc != SR_OK) return rc;
  EnvBuf d[EB_COUNT], sb[EB_COUNT];
  env_buffers(dst, d);
  env_buffers(src, sb);
  // a buffer dst has and src has not: zeros for the lazy ones (their value before first use), untouched otherwise
  // (as sr_copy_from leaves it)
  sr::CopyTable t{};
  for (int k = 0; k < EB_COUNT; k++) {
    if (!d[k].base || (!sb[k].base && !d[k].lazy)) continue;
    t.buf[t.n_buf++] = {(const char *)sb[k].base, (char *)d[k].base, d[k].bytes, copy_vec(sb[k].base, d[k].base, d[k].bytes)};
  }
  t.n_src = src->cfg.n_env;
  t.n_dst = dst->cfg.n_env;
  if (src != dst) return launch_copy(dst, t, dst_idx_dev, src_idx_dev, n, s);
  // within one handle every source row is read before any destination row is written: gather the n source rows into
  // the staging buffer (one region of n rows per buffer), then scatter them
  size_t stage = 0;
  for (int k = 0; k < t.n_buf; k++) stage += ((size_t)n * t.buf[k].bytes + 15) / 16 * 16;
  if (stage > dst->copy_stage_bytes) {
    cudaFree(dst->copy_stage);
    dst->copy_stage = nullptr; dst->copy_stage_bytes = 0;
    SR_CUDA(cudaMalloc(&dst->copy_stage, stage));
    dst->copy_stage_bytes = stage;
  }
  sr::CopyTable gather = t, scatter = t;
  gather.mode = sr::COPY_GATHER;
  scatter.mode = sr::COPY_SCATTER;
  char *region = (char *)dst->copy_stage;
  for (int k = 0; k < t.n_buf; k++) {
    gather.buf[k].dst = region;
    scatter.buf[k].src = region;
    // (the region's base is 16-byte aligned, so the vector width of the row size holds on both sides)
    region += ((size_t)n * t.buf[k].bytes + 15) / 16 * 16;
  }
  const int rg = launch_copy(dst, gather, dst_idx_dev, src_idx_dev, n, s);
  return rg != SR_OK ? rg : launch_copy(dst, scatter, dst_idx_dev, src_idx_dev, n, s);
}

static int measure_fp64_peak_impl(int device, double *tflops_out, bool three_regs) {
  if (!tflops_out) return fail(SR_E_INVALID, "sr_measure_fp64_peak: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SR_E_NO_DEVICE, "sr_measure_fp64_peak: no CUDA device");
  }
  SR_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SR_CUDA(cudaGetDeviceProperties(&prop, device));
  const int threads = 256, blocks = prop.multiProcessorCount * 8, iters = 1 << 15;
  double *d = nullptr;
  SR_CUDA(cudaMalloc(&d, (size_t)threads * blocks * sizeof(double)));
  cudaEvent_t e0, e1;
  SR_CUDA(cudaEventCreate(&e0));
  SR_CUDA(cudaEventCreate(&e1));
  double *din = nullptr;
  SR_CUDA(cudaMalloc(&din, 64 * sizeof(double)));
  double hin[64];
  for (int i = 0; i < 64; i++) hin[i] = 1.0 + 1e-9 * i;
  SR_CUDA(cudaMemcpy(din, hin, sizeof(hin), cudaMemcpyHostToDevice));
  const double per_iter = three_regs ? 16.0 : 8.0;
  double best = 0.0;
  for (int rep = 0; rep < 6; rep++) {
    SR_CUDA(cudaEventRecord(e0));
    if (three_regs) sr::dfma_peak_regs_kernel<<<blocks, threads>>>(d, din, iters);
    else sr::dfma_peak_kernel<<<blocks, threads>>>(d, iters);
    SR_CUDA(cudaEventRecord(e1));
    SR_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    SR_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    double flops = 2.0 * per_iter * (double)iters * threads * blocks;
    double tf = flops / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d); cudaFree(din);
  *tflops_out = best;
  return SR_OK;
}

int sr_measure_fp64_peak(int device, double *tflops_out) { return measure_fp64_peak_impl(device, tflops_out, false); }
int sr_measure_fp64_peak_regs(int device, double *tflops_out) { return measure_fp64_peak_impl(device, tflops_out, true); }

int sr_probe_latency(int device, double *out) {
  if (!out) return fail(SR_E_INVALID, "sr_probe_latency: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(SR_E_NO_DEVICE, "no CUDA device"); }
  SR_CUDA(cudaSetDevice(device));
  double *d = nullptr;
  SR_CUDA(cudaMalloc(&d, 8 * sizeof(double)));
  SR_CUDA(cudaMemset(d, 0, 8 * sizeof(double)));
  for (int rep = 0; rep < 2; rep++) sr::latency_probe_kernel<<<1, 32>>>(d, 1.0);
  SR_CUDA(cudaGetLastError());
  cudaError_t e = cudaMemcpy(out, d, 8 * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(SR_E_CUDA, cudaGetErrorString(e));
  return SR_OK;
}

int sr_selftest_reciprocals(int device, int32_t n, double lo, double hi, double *out) {
  if (!out || n < 2 || !(lo > 0.0) || !(hi > lo)) return fail(SR_E_INVALID, "sr_selftest_reciprocals: bad argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(SR_E_NO_DEVICE, "no CUDA device"); }
  SR_CUDA(cudaSetDevice(device));
  double *d = nullptr;
  SR_CUDA(cudaMalloc(&d, 2 * sizeof(double)));
  SR_CUDA(cudaMemset(d, 0, 2 * sizeof(double)));
  sr::reciprocal_selftest_kernel<<<(n + 255) / 256, 256>>>(n, lo, hi, d);
  SR_CUDA(cudaGetLastError());
  cudaError_t e = cudaMemcpy(out, d, 2 * sizeof(double), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(SR_E_CUDA, cudaGetErrorString(e));
  return SR_OK;
}

}  // extern "C"
