/* softrod.h — C-ABI of the B200-native batched Cosserat-rod stepper.
 *
 * The reference (skim0119/gym-softrobot) has no FFI: its physics-step boundary
 * is PyElastica's Python plugin API,
 *     time = PositionVerlet().step(simulator, time, dt)
 *   (/root/reference/gym_softrobot/envs/soft_pendulum/soft_pendulum.py:137-139,184;
 *    keyword form at /root/reference/gym_softrobot/envs/snake/continuum_snake.py:377)
 * plus live NumPy views of the rod arrays (position/velocity/director/omega
 * _collection, tangents, kappa, sigma: soft_pendulum.py:152-154,
 * envs/octopus/flat_env.py:233-247).  This header is what a ctypes binding on
 * the reference side would bind instead (stub in INTEGRATION.md).
 *
 * Conventions: plain C, plain pointers and sizes, no torch/CUDA types in the
 * signatures (`stream` is a cudaStream_t passed as void*; NULL = default stream).
 * Every call returns 0 on success or a negative SR_E_* code; the message is
 * available from sr_last_error() (thread-local).  A handle belongs to one CUDA
 * device and is not thread-safe; calls are stream-ordered.  Device pointers
 * passed in are borrowed for the duration of the call only.
 */
#ifndef SOFTROD_H
#define SOFTROD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SR_ABI_VERSION 1

/* status codes */
#define SR_OK 0
#define SR_E_INVALID (-1)  /* bad argument / unsupported configuration */
#define SR_E_CUDA (-2)     /* CUDA runtime error (message has the detail) */
#define SR_E_NO_DEVICE (-3)
#define SR_E_ALLOC (-4)

/* environment models (which plugins are fused around the rod substep) */
#define SR_MODEL_ROD 0            /* plain rod: BC + gravity + damping (BASELINE config 3) */
#define SR_MODEL_SOFT_PENDULUM 1  /* replaces build_soft_pendulum + SoftPendulumEnv.step
                                     (envs/soft_pendulum/build.py:29-115, soft_pendulum.py:176-251) */
#define SR_MODEL_SOFT_PENDULUM_3D 2 /* envs/soft_pendulum_3d/build.py:23-86, soft_pendulum_3d.py:122-158 */

/* boundary conditions on node 0 / element 0 */
#define SR_BC_FREE 0
#define SR_BC_ONE_END_FIXED 1    /* PyElastica OneEndFixedBC */
#define SR_BC_PENDULUM_SLIDER 2  /* PendulumBoundaryConditions, soft_pendulum/build.py:65-85 */
#define SR_BC_MOVING_BASE 3      /* MovingBaseConstraint, soft_pendulum_3d/build.py:23-40 */

/* arithmetic type of the state and of the kernel */
#define SR_DTYPE_F64 0
#define SR_DTYPE_F32 1

/* kernel math variant */
#define SR_MATH_FAST 0     /* strength-reduced (polynomial exp/log maps, shared reciprocals) */
#define SR_MATH_FAITHFUL 1 /* libm calls in the reference's operation order */

/* Replaces CosseratRod.straight_rod(...) + the plugin registrations of the
 * reference build functions (soft_pendulum/build.py:54-113).  All rods of a
 * handle share these parameters; per-env data (initial direction/normal, BC
 * anchors, actions) is given to sr_reset / sr_step. */
typedef struct sr_config {
  int32_t struct_size;  /* = sizeof(sr_config), checked */
  int32_t device;       /* CUDA device ordinal */
  int32_t model;        /* SR_MODEL_* */
  int32_t dtype;        /* SR_DTYPE_* */
  int32_t math;         /* SR_MATH_* */
  int32_t n_env;        /* independent environments (one rod each) */
  int32_t n_elem;       /* elements per rod: 3-1023; 1024-4095 (one rod per thread-block cluster of up to 8 CTAs) for
                         * SR_DTYPE_F64, SR_MATH_FAST, one untapered rod per env without suckers or muscle layers, and
                         * either SR_MODEL_ROD / SR_MODEL_SOFT_PENDULUM with a free, clamped or slider end, no contact,
                         * muscle, spline torques or filter; or SR_MODEL_ROD with a free or clamped end on the
                         * frictional plane (contact_on) and / or with the travelling-wave muscle (muscle_on), with
                         * rest curvature (sr_get_rest_kappa) and no base point force, spline torques or filter; or
                         * SR_MODEL_ROD with a free or clamped end and spline torques (spline_dir_mask), without
                         * contact, muscle, rest curvature, base point force or filter; or
                         * SR_MODEL_SOFT_PENDULUM_3D with SR_BC_MOVING_BASE, laplace_filter_order = 7 and no base point
                         * force */
  int32_t bc_kind;      /* SR_BC_* */
  int32_t point_force_on_base; /* F_ext[0,0] = action[env,0] each substep (build.py:94-105) */
  int32_t damping_before_constraints; /* 1: [dampen_rates, constrain_rates]; 0 (the envs): [constrain_rates, dampers] = build-code call order */
  int32_t laplace_filter_order;       /* LaplaceDissipationFilter order, 0 = off */
  int32_t n_rod_per_env; /* rods per environment; 0 or 1 = single rod.  > 1: multi-rod assembly (octopus) */
  double dt;            /* substep */
  double base_length, base_radius, density, youngs_modulus;
  double shear_modulus; /* <= 0: PyElastica default E/(2(1+0.5)) */
  double gravity[3];
  double damping_constant; /* AnalyticalLinearDamper; < 0 = off */
  /* SR_MODEL_SOFT_PENDULUM_3D only (soft_pendulum_3d.py:55-56,106-120): the action moves the base by
   * base_step * action per env-step, clipped to +-base_limit; its velocity is displacement / base_move_period
   * with base_move_period = step_skip * time_step as computed by the host in double. */
  double base_step, base_limit, base_move_period;
  /* RodPlaneContactWithAnisotropicFriction on Plane(origin, normal) (envs/octopus/build.py:173-200,258-283);
   * contact_on = 0 disables.  contact_before_forcing = 1 runs the contact operator before gravity / joints /
   * muscle torques inside `synchronize`; 0 (what the envs use: the reference's build code registers the
   * contact last, DESIGN.md 4.1) lets it see those loads; mu arrays are [forward, backward, sideways]. */
  int32_t contact_on, contact_before_forcing;
  double plane_origin[3], plane_normal[3];
  double contact_k, contact_nu, slip_velocity_tol, surface_tol;
  double static_mu[3], kinetic_mu[3];
  /* Multi-rod assembly (envs/octopus/build.py:52-217): n_rod_per_env arms + (has_head) one rigid Cylinder
   * head held upright by BodyBoundaryCondition and tied to node 0 / element 0 of every arm by a
   * FixedJoint2Rigid(k, nu, kt, angle, radius) (utils/custom_elastica/joint.py, constraint.py).
   * joint_angle_deg[a] is arm a's mounting angle.  sr_reset then expects 9*(n_rod+1) doubles per env:
   * start/direction/normal of every arm followed by those of the head cylinder. */
  int32_t has_head, reserved1;
  double head_length, head_radius, head_density;
  double joint_k, joint_nu, joint_kt, joint_radius;
  double joint_angle_deg[16];

  /* Travelling-wave muscle torque (PyElastica `MuscleTorques`; envs/snake/continuum_snake.py:186-198,325-337):
   * element couples of magnitude min(1, t/ramp) * beta(s) * sin(2 pi t/period - wave_number s + phase)
   * about `muscle_direction` (material frame), iterated tail-to-head.  beta(s) and wave_number are
   * per-env device data the caller fills before sr_step (sr_get_muscle); the handle keeps each
   * env's simulation time (advanced by dt/2 twice per substep, zeroed by sr_reset). */
  int32_t muscle_on, reserved2;
  double muscle_period, muscle_ramp_up_time, muscle_phase_shift;
  double muscle_direction[3];

  /* Spline muscle torques (`MuscleTorquesWithVaryingBetaSplines`, utils/custom_elastica/muscle_torque/
   * muscle_torques_with_bspline.py:8-228; envs/soft_arm/soft_arm_tracking.py:366-400): bit d of
   * spline_dir_mask enables one forcing instance adding  scale * spline(cumsum(lengths))_k  to
   * external_torques[d, k] (material frame).  The spline is the not-a-knot cubic through spline_n_ctrl
   * equidistant control values (zero at both ends); whenever the rate-limited cached values differ from
   * the caller's targets it is re-fitted and re-evaluated at the CURRENT element lengths, inside the
   * substep where the reference does it.  Targets / cached values / cached magnitudes: sr_get_spline. */
  int32_t spline_dir_mask, spline_n_ctrl;
  double spline_scale, spline_max_rate;

  /* Tapered rod: `base_radius` an array np.linspace(base_radius, tip_radius, n_elem)
   * (envs/octopus/build_muscle_octopus.py:61-63); <= 0: uniform radius.  FP64, SR_MATH_FAST, plane-contact / multi-rod
   * model family only (the element constants then travel in an HBM table instead of the constant bank). */
  double tip_radius;
  /* ControllableFixConstraint (envs/octopus/controllable_constraint.py:24-69, the octopus arms' "sucker"): after the
   * dampers, velocity and angular velocity of node / element `sucker_index` of every rod are scaled by
   * 1 - reduction_ratio; the per-rod ratios (0 = released) are device data the caller writes (sr_get_sucker). */
  int32_t sucker_on, sucker_index;
  /* 1: the taper is given on the NODES, np.linspace(base_radius, tip_radius, n_elem + 1), each element taking the mean of
   * its two nodes (envs/octopus/arm_push_env.py:161-175,524-538); 0: np.linspace(base, tip, n_elem) on the elements. */
  int32_t taper_node_mean;
  /* COOMM `ApplyMuscles` with the `TransverseMuscle(rest_muscle_area=(radius / tm_radius_ref)**2,
   * max_muscle_stress=tm_max_stress)` of create_es_muscle_layers (envs/octopus/build.py:292-338; registered at
   * build_muscle_octopus.py:165-177, arm_push_env.py:198-209,601-606) evaluated every substep; tapered rods only.  The
   * two longitudinal muscles of that layer set never receive a non-zero activation in OctoCrawl / OctoArmPush /
   * OctoArmPullWeight and are not evaluated.  Per-rod scalar activations: sr_get_tm_activation.  coomm is not part of
   * the reference tree: the published model is restated (DESIGN.md section 2). */
  int32_t tm_muscle_on;
  double tm_max_stress, tm_radius_ref;
  /* The whole layer set of create_es_muscle_layers with PER-ELEMENT activations (OctoReach-v0, OctoArmTwo-v0:
   * envs/octopus/reach_env.py:214-227, arm_two_env.py:222-247): two `LongitudinalMuscle(max_muscle_stress=
   * lm_max_stress)` at material-frame offsets (lm_px[m], lm_py[m]) x element radius (ratio_muscle_position rotated by
   * muscle_init_angle) plus the transverse muscle above.  Needs tm_muscle_on and a multi-rod assembly of tapered rods;
   * activations: sr_get_muscle_activation (the per-rod scalars of sr_get_tm_activation are then ignored). */
  int32_t muscle_layers_on;
  /* OneEndFixedBC(constrained_position_idx=(0,), constrained_director_idx=(0,)) on the rigid head, on top of its
   * BodyBoundaryCondition (envs/octopus/reach_env.py:128-132): the head stays at its reset pose, all rates zero.
   * Honoured by the muscle-layer kernel only (muscle_layers_on). */
  int32_t head_fixed;
  double lm_max_stress, lm_px[2], lm_py[2];
  /* Up to three ControllableFixConstraints per rod at FIXED, distinct node / element indices (OctoArmTwo-v0:
   * envs/octopus/arm_two_env.py:78-82,133-145) next to the muscle layers (muscle_layers_on); the reduction ratios are
   * device data [n_env * n_rod_per_env][3] the caller writes every step (sr_get_fixed_suckers).  0 = none. */
  int32_t n_fixed_sucker, fixed_sucker_index[3];
} sr_config;

/* Device views of the structure-of-arrays state (replaces the NumPy views the
 * reference env code reads).  Field f of env e, slot k is at
 *   base + ((e * n_fields + f) * stride + k) * elem_size.
 * Nodes use slots 0..n_elem, elements 0..n_elem-1, Voronoi points 0..n_elem-2. */
typedef struct sr_state_view {
  void *base;
  int32_t n_env, n_fields, stride, elem_size;
  /* first field index of each quantity (component-major, reference order) */
  int32_t f_position;  /* 3 fields: x,y,z              (position_collection) */
  int32_t f_velocity;  /* 3                            (velocity_collection) */
  int32_t f_director;  /* 9: Q[i][j] at f_director+3i+j (director_collection) */
  int32_t f_omega;     /* 3                            (omega_collection)    */
  int32_t f_tangents;  /* 3  stale, last force evaluation (SURVEY A.6)       */
  int32_t f_kappa;     /* 3  stale                                           */
  int32_t f_sigma;     /* 3  stale                                           */
  int32_t f_dilatation;/* 1  stale                                           */
} sr_state_view;

typedef struct sr_handle sr_handle;

int sr_abi_version(void);
const char *sr_last_error(void);

/* Allocate device state for cfg->n_env rods and precompute rod constants. */
int sr_create(const sr_config *cfg, sr_handle **out);
void sr_destroy(sr_handle *h);

/* per-env sizes for the chosen model */
int sr_obs_dim(const sr_handle *h);
int sr_action_dim(const sr_handle *h);
int sr_init_dim(const sr_handle *h); /* doubles per env expected by sr_reset: 9 = start, direction, normal */

/* (Re)build rods: replaces Env.reset -> build_* -> simulator.finalize().
 * env_idx: int32 device array of n env indices, or NULL for envs 0..n-1.
 * init: double device array [n][9] = start(3), direction(3), normal(3). */
int sr_reset(sr_handle *h, const int32_t *env_idx_dev, int n, const double *init_dev, void *stream);

/* Advance every env by n_substeps PositionVerlet substeps in ONE kernel launch
 * and evaluate the model's observation / reward / NaN guard
 * (replaces the loop at soft_pendulum.py:183-184 and lines 196-214,149-161).
 *   action_dev      float  [n_env][action_dim]   (may be NULL if action_dim == 0)
 *   obs_dev         float  [n_env][obs_dim]
 *   reward_dev      double [n_env]
 *   terminated_dev  uint8  [n_env]   1 = NaN in position/velocity */
int sr_step(sr_handle *h, const float *action_dev, int n_substeps, float *obs_dev,
            double *reward_dev, uint8_t *terminated_dev, void *stream);

/* Same with HOST buffers: H2D of actions, launch, D2H of results, synchronised. */
int sr_reset_host(sr_handle *h, const int32_t *env_idx_host, int n, const double *init_host);
int sr_step_host(sr_handle *h, const float *action_host, int n_substeps, float *obs_host,
                 double *reward_host, uint8_t *terminated_host);
/* current observation without stepping (reset obs) */
int sr_observe(sr_handle *h, const float *prev_action_dev, float *obs_dev, void *stream);

int sr_get_state(sr_handle *h, sr_state_view *out);
/* Copy the structure-of-arrays ROD block (the fields of sr_state_view, same layout, device memory) into the handle.
 * Rod arrays only: BC anchors, the rigid head, rest curvatures, the 3D pendulum's base controller and the
 * forcings' state are not part of the view — use sr_copy_from to clone a whole handle. */
int sr_set_state(sr_handle *h, const sr_state_view *src, void *stream);
/* ControllableFixConstraint ratios, [n_env * n_rod_per_env] of the handle's element type (needs sucker_on). */
int sr_get_sucker(sr_handle *h, void **ratio_dev);
/* Per-rod index the ControllableFixConstraint acts on, int32 [n_env * n_rod_per_env], initialised to cfg.sucker_index;
 * what `controller.index = ...` sets every env-step (crawl_env.py:239-241, arm_push_env.py:255-270).  Python indexing of
 * the reference's arrays: i >= 0 scales node i and element i; i < 0 scales node n_elem + 1 + i and element n_elem + i. */
int sr_get_sucker_index(sr_handle *h, int32_t **index_dev);
/* Per-rod activation of the transverse muscle, [n_env * n_rod_per_env] of the handle's element type (needs tm_muscle_on);
 * what `muscle_layers[2].apply_activation(a)` sets (crawl_env.py:242, arm_push_env.py:259,271). */
int sr_get_tm_activation(sr_handle *h, void **activation_dev);
/* Per-element activations of the three muscle layers, [n_env * n_rod_per_env][3][n_elem] doubles: longitudinal 1,
 * longitudinal 2, transverse (needs muscle_layers_on); replaces `muscle.apply_activation(array)` of
 * envs/octopus/reach_env.py:221-225 / arm_two_env.py:243-245.  Constant during a launch; zeroed by sr_create only. */
int sr_get_muscle_activation(sr_handle *h, void **activation_dev);
/* Reduction ratios of the fixed-index ControllableFixConstraints, [n_env * n_rod_per_env][3] doubles (slot s acts on
 * index fixed_sucker_index[s]; needs n_fixed_sucker > 0); replaces `controller.reduction_ratio = ...` of
 * envs/octopus/arm_two_env.py:233-234.  Zeroed (released) by sr_create only. */
int sr_get_fixed_suckers(sr_handle *h, void **ratio_dev);
/* Generic per-element external loads evaluated every substep as a forcing (what COOMM's ApplyMuscles would feed,
 * envs/octopus/build_muscle_octopus.py:171-176): nodal forces in the lab frame, [n_rods][3][stride] slots 0..n_elem,
 * and element couples in the material frame, [n_rods][3][stride] slots 0..n_elem-1, of the handle's element type;
 * allocated (zeroed) by the first call.  Plane-contact / multi-rod / forcing model family (the lean path stays lean). */
int sr_get_ext_loads(sr_handle *h, void **force_dev, void **couple_dev);

/* Clone everything that evolves or parametrises the envs of `src` into `dst` (created with the same shapes): rod
 * arrays, BC anchors, model scratch, rigid heads, rest curvatures, muscle / spline forcing state.  Checkpoint /
 * restore; works across devices (peer copy).  Stream-ordered on `stream` of dst's device. */
int sr_copy_from(sr_handle *dst, sr_handle *src, void *stream);
/* Fork envs: for i < n, env dst_idx[i] of `dst` takes everything that evolves or parametrises env src_idx[i] of `src`
 * (the per-env rows of what sr_copy_from clones: rod arrays, BC anchors, model scratch, rigid head, rest curvatures,
 * external loads, sucker ratios and indices, muscle activations, muscle / spline forcing state).  `src` may be `dst`.
 * Index arrays are int32 device arrays.  Stream-ordered on `stream` (dst's device).  A copy within one handle goes
 * through a staging buffer the handle owns: issue the copies of one handle on one stream (or order their streams), as
 * for the handle's other calls.
 *   - Every source row is read before any destination row is written, so permutations and swaps within one handle
 *     work; destinations must be distinct; a pair with src_idx[i] == dst_idx[i] within one handle leaves the env as is.
 *   - 0 <= n <= dst's n_env (n = 0: nothing to do).  Both handles on the same device, created with the same shapes
 *     apart from n_env (as for sr_copy_from).  A pair with an index outside [0, n_env) of its handle is skipped.
 *   - A rest-curvature or external-load buffer the source never allocated zeroes the destination rows (its initial
 *     value); one the destination lacks is allocated first.
 *   - Handle-level state is not copied (fallback counters and windows, launch count): it does not change an env's bits. */
int sr_copy_envs(sr_handle *dst, const int32_t *dst_idx_dev, const sr_handle *src, const int32_t *src_idx_dev,
                 int n, void *stream);

/* Per-env model scratch, [n_env][*dim] of the handle's dtype: SoftPendulum3D keeps the base controller there
 * (0-2 position, 3-5 velocity, 6 last tilt angle, `info["tilt"]` of soft_pendulum_3d.py:157). */
int sr_get_aux(sr_handle *h, void **aux_dev, int32_t *dim);

/* Rigid head of a multi-rod assembly, [n_env][*dim] of the handle's dtype:
 * 0-2 position, 3-5 velocity, 6-14 directors (rows), 15-17 omega, 18 pinned height. */
int sr_get_head(sr_handle *h, void **head_dev, int32_t *dim);

/* Per-env rest curvature (the actuation of the octopus-arm envs: `rod.rest_kappa[0, :] = ...`,
 * envs/octopus/arm_single_env.py:226-235, flat_env.py:288-311), [n_env][3][stride] of the handle's
 * dtype (n_env * n_rod_per_env rows for assemblies), Voronoi points in slots 0..n_elem-2; allocated on
 * first use, zero-initialised.  Above 1023 elements, for handles with contact_on or muscle_on only. */
int sr_get_rest_kappa(sr_handle *h, void **rest_kappa_dev);

/* Per-env muscle-torque data (muscle_on handles), [n_env][*dim] float64 whatever the handle's dtype:
 * 0 simulation time, 1 wave_number, 2..2+n_elem-1 beta(s_k) at s_k = cumsum(rest_lengths)_k / L
 * (`MuscleTorques.__init__`, re-run by `set_action` of continuum_snake.py:186-198). */
int sr_get_muscle(sr_handle *h, double **muscle_dev, int32_t *dim);

/* Per-env spline-torque data (spline_dir_mask handles), [n_env][*dim] float64; with P = spline_n_ctrl,
 * channel d = 0..2 occupies [d*(2P+2), (d+1)*(2P+2)): P targets (what `points_func_array` returns),
 * P cached values, the initial-call flag, one pad; then 3 x n_elem cached torque magnitudes. */
int sr_get_spline(sr_handle *h, double **spline_dev, int32_t *dim);
/* Cardinal polynomials of the not-a-knot cubic spline through n_ctrl + 2 equidistant points on
 * [0, base_length] with zero end values (what scipy's make_interp_spline(x, y) returns, as used at
 * muscle_torques_with_bspline.py:146-148): out[(m * n_ctrl + i) * 4 + p] is the coefficient of t^p,
 * t = s - x_m, of control value i's contribution on interval m (n_ctrl + 1 intervals).  Host-only. */
int sr_spline_basis(int32_t n_ctrl, double base_length, double *out);

/* number of kernels this library launched on behalf of the handle so far */
int64_t sr_launch_count(const sr_handle *h);
/* Env-steps the fast-only kernels handed to the safe kernel since sr_create (arguments outside the polynomial maps'
 * ranges; csrc/rod_kernel_lean.cuh).  Synchronises the handle's device: a diagnostic, not for the step loop. */
int64_t sr_fallback_count(const sr_handle *h);
/* The same count by cause, for the kernels of csrc/rod_kernel_lean.cuh (an env-step can count under several):
 * out[0] rotation per kinematic update > 0.1 rad, out[1] bend between neighbouring elements beyond the log map's
 * polynomial range, out[2] stretch beyond the rotational damper's polynomial range. */
int sr_fallback_causes(const sr_handle *h, int64_t out[3]);
/* Env-steps the planar model of the lean kernel (a rod in the x-y plane, FP64) handed to the 3D safe kernel because
 * the rod's state was not planar (out-of-plane components not exactly zero).  Not range failures: sr_fallback_count
 * does not include them.  Synchronises the handle's device. */
int64_t sr_nonplanar_count(const sr_handle *h);

/* Measure the device's FP64 FMA issue peak with a register-resident DFMA chain
 * (roofline denominator; not in MEASURED_PEAKS.json).  Returns TFLOP/s. */
int sr_measure_fp64_peak(int device, double *tflops_out);
/* Same probe with three distinct 64-bit register operands per DFMA (the common case in real code):
 * on B200 the register file delivers two 64-bit operands per 2-cycle issue slot, so this rate is 2/3 of
 * the figure above (24.7 vs 36.4 TFLOP/s measured).  Context for the roofline fraction, not its denominator. */
int sr_measure_fp64_peak_regs(int device, double *tflops_out);
/* Diagnostic: dependent-issue latencies (cycles per operation, one warp) of the instruction kinds the substep's
 * critical path is made of.  out[0] DFMA, [1] DADD, [2] MUFU.RSQ64H + DFMA, [3] shared store -> barrier -> load
 * round trip (two barriers), [4] DFMA with an immediate multiplicand; out must hold 8 doubles. */
int sr_probe_latency(int device, double *out);

/* Self-test of the kernels' Newton-refined reciprocals (csrc/rod_math.cuh: rsqrt_nr, rcp_nr — MUFU seed + one
 * third-order step) against the correctly rounded IEEE results over n log-spaced arguments in [lo, hi]:
 * out[0] = max relative error of rsqrt_nr, out[1] = of rcp_nr (both should be <= ~1 ulp = 2.2e-16). */
int sr_selftest_reciprocals(int device, int32_t n, double lo, double hi, double *out);

#ifdef __cplusplus
}
#endif
#endif /* SOFTROD_H */
