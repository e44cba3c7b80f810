// rod_kernel_lean.cuh — the product kernel, sm_100a.  An instantiation is one model (which substep runs) in one layout
// (where a rod's nodes live), the template parameters MODEL and LAYOUT (LeanModel, LeanLayout in launch.cuh).  The
// headline is the plain model in the CTA layout: FP64 or FP32 storage, single rod per env, no contact / filter / joints /
// forcing (SoftPendulum-v0 and plain rods: BASELINE configs 2 and 3).  The other models put the plane contact + rest
// curvature, + the travelling-wave muscle, assemblies (arms + rigid head + joints), the Laplace filter + moving base,
// spline muscle torques and rods that stay in the lab x-y plane (out-of-plane terms left out, same bits) on the same
// skeleton; the fold layout puts the tip node into the last thread, and the cluster layout spreads a rod of 512-4095
// elements over a thread-block cluster of 2-8 CTAs (same substep, same bits).  See the comment at the kernel.
//
// Same mapping as rod_kernel_packed.cuh (one thread per node/element, rods packed back to back across a
// 256-thread CTA, state in registers for the whole launch, neighbour data through array-of-structures
// records in shared memory, two CTA barriers per substep), with two things the generic kernel does not have:
//
// 1. Work is dealt to the SMs by substep count, not by CTA (stream-K style).  A launch is n_items x K
//    "item-substeps" (item = the rods one CTA holds).  When there are more items than resident CTA slots the
//    grid is exactly the resident slot count and slot p owns the contiguous range [p W/P, (p+1) W/P) of the
//    item-major linear index: a few whole items plus at most one item shared with slot p-1 and one shared with
//    slot p+1.  A slot runs the part it shares with its successor FIRST (substeps 0..a of that item, no
//    dependency), hands the 18 integrated values per thread over through global scratch + a flag, runs its
//    whole items, and finishes with the part it shares with its predecessor (substeps b..K-1), whose input has
//    long been published by then.  Every slot therefore executes the same number of substeps (+-1) and the
//    2.77-wave tail of 4096 envs on 296 slots disappears.  Arithmetic is unchanged by the split: the registers
//    that would have stayed live are stored and re-loaded bit for bit.
//
// 2. The arithmetic is trimmed to what a uniform rod with a circular cross-section needs (every rod the
//    reference builds: CosseratRod.straight_rod, /root/reference/gym_softrobot/envs/soft_pendulum/build.py:54-61):
//    J1 = J2, B1 = B2, S1 = S2 make (J w) x w, kappa x (B kappa) and (Q t) x n two-term expressions; the
//    log-map factor theta/sin(theta) is a polynomial in |axial(R - R^T)|^2 (no trace needed); the rotational
//    damper c_w^e is a cubic in (e - 1) with host-made coefficients; range checks run on the integer pipe.
//
// Range handling (both kernels compute bit-identical results for every thread whose arguments are in range):
//   FASTONLY = true : no fallback code; a thread that leaves the range flags its env, whose state is then not
//                     written back and which the safe kernel re-runs (redo[]).
//   FASTONLY = false: per-thread fallback to the libm-class reference maps (never a warp vote: an env's bits
//                     must not depend on which other envs share its warps).
//
// Algorithm: SURVEY.md Appendix A.2/A.3; reference boundary
// /root/reference/gym_softrobot/envs/soft_pendulum/soft_pendulum.py:183-184.
#pragma once
#include <cooperative_groups.h>
#include <type_traits>
#include "launch.cuh"
#include "rod_kernels.cuh"

namespace sr {

// high word of a double as an ordered integer (x >= 0): range tests on the integer pipe instead of DSETP.
// NaN compares as "large" (0x7ff8....), i.e. out of range, which is what the callers want.
__device__ __forceinline__ int hi_abs(double x) { return __double2hiint(x) & 0x7fffffff; }

// Q <- R Q with R = I + A K + B K^2, A = sin(t)/t = 1 + q g(q), B = (1 - cos t)/t^2 = 1/2 + q h(q), q = t^2 <= 0.01
// (g, h: SR_COEF_SINCG / SR_COEF_COSCH, leading constants exact so that they are instruction immediates).  The
// reference's guard (axis = a / (|a| + eps)) multiplies A by rho and B by rho^2, rho = |a| / (|a| + eps) = 1 - d with
// d = eps / (|a| + eps) EXACTLY — two MUFU approximations are enough, d only needs 1e-6 relative.  (Round 1 used the
// expansion d ~ eps / |a|: fine at 1e-10, but a rod that starts from exact rest passes through |a| ~ 1e-14 in its first
// ten substeps, where the expansion is off by tens of per cent of a 1e-14 rad rotation; the 1e-14 rad of director
// error it left next to a clamp then rang through the rod as 2e-10 rad/s of omega — 2e-9 of |omega| when the test
// looked, scripts/diag_omega.py.)  A rho = A - A d is one FMA.  B rho^2 multiplies K^2 = O(|a|^2): its guard changes the
// rotation by |a|^2 d <= eps |a| <= 1e-15 rad per update and is left out.
__device__ __forceinline__ void rotate_directors_lean(const double (&cg)[3], const double (&ch)[3], double a0, double a1,
                                                      double a2, double q, double eps, double (&Q)[9]) {
  const double d = eps * rcp_approx(fma(q, rsqrt_approx(q), eps));   // |a| = q / sqrt(q); the caller's q carries +1e-300
  double pa = fma(cg[2], q, cg[1]), pb = fma(ch[2], q, ch[1]);
  pa = fma(pa, q, cg[0]); pb = fma(pb, q, ch[0]);
  const double A1 = fma(pa, q, 1.0), B = fma(pb, q, 0.5);
  const double A = fma(-A1, d, A1);
  const double Aa0 = A * a0, Aa1 = A * a1, Aa2 = A * a2;
  const double Ba0 = B * a0, Ba1 = B * a1, Ba2 = B * a2;
  double D[9];
  D[0] = -fma(Ba1, a1, Ba2 * a2); D[4] = -fma(Ba0, a0, Ba2 * a2); D[8] = -fma(Ba0, a0, Ba1 * a1);
  D[1] = fma(Ba0, a1, Aa2); D[3] = fma(Ba0, a1, -Aa2);
  D[2] = fma(Ba0, a2, -Aa1); D[6] = fma(Ba0, a2, Aa1);
  D[5] = fma(Ba1, a2, Aa0); D[7] = fma(Ba1, a2, -Aa0);
  double nq[9];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) nq[3 * i + m] = fma(D[3 * i], Q[m], Q[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) nq[3 * i + m] = fma(D[3 * i + 1], Q[3 + m], nq[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int m = 0; m < 3; m++) nq[3 * i + m] = fma(D[3 * i + 2], Q[6 + m], nq[3 * i + m]);
#pragma unroll
  for (int i = 0; i < 9; i++) Q[i] = nq[i];
}

// rotate_directors_lean for a rod in the lab x-y plane (planar model): the rotation vector is (0, a1, 0) about d2 = +-z, and
// only d1 = (Q0, Q1, 0) and d3 = (Q6, Q7, 0) move.  The same terms as above in the same order, with the ones that carry
// an exact zero factor left out (D = [[-B a1^2, 0, -A a1], [0, 0, 0], [A a1, 0, -B a1^2]]): the same roundings.
__device__ __forceinline__ void rotate_directors_planar(const double (&cg)[3], const double (&ch)[3], double a1, double q,
                                                        double eps, double (&Q)[9]) {
  const double d = eps * rcp_approx(fma(q, rsqrt_approx(q), eps));
  double pa = fma(cg[2], q, cg[1]), pb = fma(ch[2], q, ch[1]);
  pa = fma(pa, q, cg[0]); pb = fma(pb, q, ch[0]);
  const double A1 = fma(pa, q, 1.0), B = fma(pb, q, 0.5);
  const double A = fma(-A1, d, A1);
  const double Aa1 = A * a1, Ba11 = (B * a1) * a1;
  const double q0 = fma(-Aa1, Q[6], fma(-Ba11, Q[0], Q[0])), q1 = fma(-Aa1, Q[7], fma(-Ba11, Q[1], Q[1]));
  const double q6 = fma(-Ba11, Q[6], fma(Aa1, Q[0], Q[6])), q7 = fma(-Ba11, Q[7], fma(Aa1, Q[1], Q[7]));
  Q[0] = q0; Q[1] = q1; Q[6] = q6; Q[7] = q7;
}

constexpr int LEAN_REC = 18;        // exchange record per thread (doubles), 144-byte stride: conflict-free LDS.128
constexpr int LEAN_JREC = 10;      // assemblies: joint record of an arm's first thread {reaction force, couple on the head, couple on element 0, -}
// filter model: records of 6 doubles with 6 ghost records on either side of every rod (rods of >= 9 threads)
// (8 ghost records per side, 6 used: a rod's records then start a multiple of 8 records = 96 words after where the
// previous rod's would continue, so a quarter-warp that straddles two rods still hits eight distinct 4-bank groups).
// A CTA of more than 512 threads holds one rod of >= 512 elements and at most the head of an idle second group, whose
// records and taps end within 30 records past NT: sized as rods of >= 9 threads, its ghost array alone would take
// 73 KB at 544 threads and push the 768- and 1024-thread CTAs past the 227 KB a CTA can have.
constexpr int lean_ghost_records(int nt) { return nt <= 512 ? nt + 16 * (nt / 9) + 16 : nt + 48; }
// records of each exchange array beyond the NT threads' own: the cluster layout has a halo record before thread 0, two
// after thread NT - 1 and a zero record; the others a zero record and a spare one
__host__ __device__ constexpr int lean_extra_records(LeanLayout layout) { return layout == LeanLayout::CLUSTER ? 4 : 2; }
// filter model on clusters: each rank's ghost-padded filter records hold the rod indices [NT c - 8, NT c + NT + 8) (6 of
// the 8 halo records per side used, as the CTA layout pads them)
constexpr int lean_smem_words(int nt, LeanModel model, LeanLayout layout) {
  return (LEAN_REC + 6 + (model == LeanModel::ASSEMBLY ? LEAN_JREC : 0)) * (nt + lean_extra_records(layout)) +
         (model != LeanModel::FILTER ? 0 : layout == LeanLayout::CLUSTER ? 6 * (nt + 16) : 6 * lean_ghost_records(nt));
}

// cluster layout: the address of `p` in the shared memory of CTA `rank` of this cluster (DSMEM)
template <typename T> __device__ __forceinline__ T *cluster_smem(T *p, int rank) {
  return cooperative_groups::this_cluster().map_shared_rank(p, (unsigned)rank);
}
__device__ __forceinline__ void cluster_sync() { cooperative_groups::this_cluster().sync(); }

// float overloads of the reciprocal helpers for the FP32 force evaluation of the mixed mode
__device__ __forceinline__ bool out_of_range(double x, int lim_hi, float) { return hi_abs(x) > lim_hi; }
__device__ __forceinline__ bool out_of_range(float x, int, float limf) { return !(fabsf(x) <= limf); }

// ST = storage type of the state in HBM.
//   ST = double: everything in FP64 (the default; parity 1e-9).
//   ST = float : the optional FP32 mode (SR_DTYPE_F32), mixed precision.  What limits a plain FP32 rod step is not
//     the accumulation but the force evaluation's input: the stretch / shear strains are differences of O(1)
//     quantities, Q dx / l0 - z, and every 6e-8 of rounding in Q or dx becomes S * 6e-8 = 5e-4 N of force noise per
//     element and substep (measured with the all-FP32 kernel of round 1: velocities 4e-4, omega 2e-3 after 1200
//     substeps).  So the state registers (x, v, Q, w), the kinematic update, the edge vectors, Q dx and the
//     relative rotation Q+ Q^T stay in FP64 inside a launch (about 130 of the 226 FP64 instructions of a substep);
//     stresses, couples, damper and all the scalar algebra run in FP32.  Between launches the state is stored in
//     FP32, with the element edge vectors as fields of their own (F_EDGE) so that the strain survives the
//     rounding of absolute positions: the launch rebuilds FP64 node positions from node 0 + the running sum of edges.
//     Measured (4096 x SoftPendulum, B200): 1.644 ms per env step against 1.524 ms in FP64 — this mode halves the
//     state in HBM, it is not the fast mode.  Pushing more into FP32 (FP32 rates, FP32 rotation increments accumulated
//     into FP64 frames: 56 FP64 instructions + 35 conversions per element-substep) was tried and was slower still,
//     1.728 ms: F2F conversions issue at the FP64 rate, and velocity error rose to 3.6e-5 (scripts/gpu_r2n.sh).
//
// Models (MODEL: which substep runs; every model but PLAIN is FP64 only):
//   PLAIN    one rod under gravity, damping and the base point force, with a free, clamped or slider end.
//   PLANE    (CONTACT, FP64 only) the same skeleton for a single rod on the frictional plane — per-env rest curvature
//            (flat_env.py:310-311 style actuation), RodPlaneContactWithAnisotropicFriction (SURVEY A.5; two more
//            exchanges and per-rod barriers per substep), and the internal frame whose z axis is the plane normal (see
//            rod_kernel_packed.cuh).  OctoArmSingle-v0 and BASELINE config 5.
//   MUSCLE   PLANE + the MuscleTorques travelling wave of ContinuumSnake-v0.
//   ASSEMBLY PLANE for assemblies: several rods + one rigid head thread per env, FixedJoint2Rigid joints,
//            BodyBoundaryCondition on the head (OctoFlat-v0).
//   FILTER   SoftPendulum3D-v0: LaplaceDissipationFilter + host-commanded moving base (no contact).
//   SPLINE   clamped / free rod + MuscleTorquesWithVaryingBetaSplines (SoftArmTracking-v0); safe kernel only, see below.
//   PLANAR   PLAIN for a rod that stays in the lab x-y plane (SoftPendulum-v0, planar clamped / free rods; the host
//            checks gravity and the base force).  x_z, v_z, d1_z, d3_z, d2_x, d2_y, w_0, w_2, kappa_0, kappa_2 and
//            sigma_1 are exact zeros at every substep, and every product that carries one of them is left out: the same
//            terms in the same order, so the same roundings as PLAIN (up to the sign of zeros).  Nine state registers per
//            thread instead of 18.  Each segment checks those zeros in its input (and the padding of slot n: Q = I,
//            w = 0, which the stale observables of the last element and the tip assume); a rod that fails is flagged
//            like a range failure (cause bit 8) and re-run by PLAIN's safe kernel.
//
// Layouts (LAYOUT: where a rod's nodes live):
//   CTA      rods of n elements packed back to back into one CTA, n + 1 threads each (every model).
//   FOLD     (PLAIN, PLANE) the tip node folded into the last element's thread: a rod of n elements then takes n
//            threads, not n + 1 — what lets the 512-element rod (BASELINE config 5) run in a 512-thread CTA with 128
//            registers instead of a 544-thread one capped at 96 (17 warps put five on one scheduler).  One rod per CTA.
//   CLUSTER  (PLAIN, FILTER, PLANE, MUSCLE, SPLINE) a rod of 512-4095 elements spread over a thread-block cluster of
//            C = ceil((n + 1) / NT) CTAs (one rod per cluster, launched with the cluster dimension set at run time):
//            CTA rank c holds nodes / elements j = NT c + tid.  The substep is the model's, instruction for instruction.
//            Only where the records come from changes: each exchange array has a halo record before thread 0 (the
//            stress record of element j - 1, stored there by the previous rank's last thread) and two after thread
//            NT - 1 (the x, v, Q records of nodes j + 1, j + 2, stored there by the next rank's threads 0 and 1), so
//            every read of the substep stays a local shared-memory load at the same offset.  The substep's two barriers
//            become cluster barriers; they order the DSMEM halo stores as the CTA barriers order the local ones (a halo
//            slot is rewritten only after the barrier that follows its last read).  Env-level decisions (range flags,
//            NaN flag) are reduced into rank 0's shared memory through DSMEM atomics and read back by every CTA.
//            FILTER: the filter's pass 0 reads the rate records of j - 1 and j + 1: rec gets a halo at -1 too, and the
//            filter's own record is pushed into the neighbours' halos -1 / NT.  Each rank's ghost-padded array gb holds
//            the rod indices [NT c - 8, NT c + NT + 8), and a g record of index k is stored into every rank whose taps
//            read it (put_g below); the reflected ghosts follow the same rule.  The filter's two barriers become
//            cluster barriers as well: four per substep.
//            PLANE, MUSCLE: the plane's two extra exchanges read across the rank boundary too, so the last thread
//            pushes its stage-1 load into the next rank's rec halo -1 (words 16-17) and its final plane load into the
//            next rank's sn halo -1; thread 0 pushes its stress record into the previous rank's sn halo NT and its
//            stage-1 load into the previous rank's rec halo NT (words 16-17).  The contact's two barriers become
//            cluster barriers: four per substep.  DESIGN.md §4.1 gives the slot-by-slot order.
//            SPLINE (safe kernel only): rank 0's lead keeps the forcing's bookkeeping and stores `need` into every rank's
//            sh_need[0] before the second barrier; the arc-length prefix sum continues a per-rank carry, the earlier
//            ranks' length words summed in order through DSMEM by warp 0, behind one CTA barrier in substeps that re-fit.
template <typename ST, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT>
__global__ void __launch_bounds__(NT, MINB)
rod_lean_kernel(const __grid_constant__ RodArgs<ST> A) {
  using D = double;
  constexpr bool MIXED = sizeof(ST) == 4;
  constexpr bool CONTACT = MODEL == LeanModel::PLANE || MODEL == LeanModel::MUSCLE || MODEL == LeanModel::ASSEMBLY;
  constexpr bool MUS = MODEL == LeanModel::MUSCLE, MULTI = MODEL == LeanModel::ASSEMBLY;
  constexpr bool LAPL = MODEL == LeanModel::FILTER;
  constexpr bool SPL = MODEL == LeanModel::SPLINE;
  constexpr bool PLANAR = MODEL == LeanModel::PLANAR;
  constexpr bool FOLD = LAYOUT == LeanLayout::FOLD;
  constexpr bool CLUSTER = LAYOUT == LeanLayout::CLUSTER;
  static_assert(!PLANAR || FASTONLY, "the planar model is fast-only: its fallback is the 3D safe kernel");
  static_assert((MODEL == LeanModel::PLAIN && LAYOUT == LeanLayout::CTA) || !MIXED, "FP64 only");
  static_assert(!FOLD || LEAN_SCR_FOLD >= 27, "hand-over rows of the folded tip");
  constexpr int SCR = FOLD ? LEAN_SCR_FOLD : CONTACT ? LEAN_SCR_CONTACT : LEAN_REC;   // rows of a slot's hand-over scratch
  using F = typename std::conditional<MIXED, float, double>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int SNR = MIXED ? 8 : 6;
  constexpr int RX = lean_extra_records(LAYOUT);
  constexpr int ZR = CLUSTER ? NT + 2 : NT;   // record ZR = zeros (left of element 0); cluster layout: -1, NT, NT + 1 are halos
  D *rec = reinterpret_cast<D *>(smem_raw) + (CLUSTER ? LEAN_REC : 0);   // {x0 x1 | x2 v0 | v1 v2 | Q0 Q1 | ... | Q6 Q7 | Q8 - | - -}
  // {s0 s1 | s2 N0 | N1 m2} (FP64: 48-byte records; mixed: 8 floats, 32-byte records)
  F *sn = reinterpret_cast<F *>(reinterpret_cast<D *>(smem_raw) + LEAN_REC * (NT + RX)) + (CLUSTER ? SNR : 0);
  __shared__ int sh_flag[256], sh_dom[256];   // one per rod of the CTA (<= NT / 4)
  __shared__ int sh_need[SPL ? 128 : 1];      // spline model: which directions re-fit their magnitudes this substep, per rod
  // filter model: the moving base's command, per rod (rods of >= 9 threads; cluster layout: rank 0's one rod in row 0)
  __shared__ double sh_base[LAPL && !CLUSTER ? 128 : 1][4];

  const int tid = threadIdx.x;
  const int n = A.n_elem, stride = A.stride, tpr = FOLD ? n : n + 1;
  // env group = the threads of one env: a rod, or (assemblies) n_rod rods of tpr threads + one head thread
  const int n_rod = MULTI ? A.n_rod : 1, has_head = MULTI ? A.has_head : 0;
  const int G = n_rod * tpr + has_head;
  const int rods_per_cta = A.sk_rods_per_cta;       // env groups per CTA
  const int c_rank = CLUSTER ? (int)cooperative_groups::this_cluster().block_rank() : 0;
  const int c_size = CLUSTER ? (int)cooperative_groups::this_cluster().num_blocks() : 1;
  const int r = CLUSTER ? 0 : tid / G, u_grp = CLUSTER ? NT * c_rank + tid : tid - r * G;
  const bool is_head = MULTI && has_head && (u_grp == G - 1);
  const int arm = (MULTI && !is_head) ? u_grp / tpr : 0;
  const int j = is_head ? 0 : u_grp - arm * tpr;
  const bool in_cta = r < rods_per_cta && (!CLUSTER || j <= n);   // (cluster layout: the last rank's threads past the tip idle)
  const bool first = (j == 0) && !is_head;          // first thread of a rod
  const bool lead = first && arm == 0;              // one thread per env: env-level flags and outputs
  const int t_head = r * G + G - 1;                 // where this env's head publishes its state
  // past the stress records: assemblies: joint records (LEAN_JREC doubles per thread slot)
  D *sj = reinterpret_cast<D *>(sn - (CLUSTER ? SNR : 0) + 6 * (NT + RX));
  D *gb = sj;                                       // filter model: ghost-padded records of the filtered rates
  if (tid < SNR) sn[SNR * ZR + tid] = F(0);
  if (CLUSTER && tid < 256) { sh_dom[tid] = 0; sh_flag[tid] = 0; }   // (rank 0's are the cluster's env-level flags)
  if (CONTACT && tid < 2) rec[LEAN_REC * ZR + 16 + tid] = D(0);   // stage-1 contact load "left of element 0"
  if (FOLD && tid < LEAN_REC) rec[LEAN_REC * NT + tid] = D(0);     // the folded tip's record: x, v published by the last thread, the rest finite
  __syncthreads();   // (the per-rod barriers below do not order this store against the other rods' reads)
  if constexpr (CLUSTER) cluster_sync();   // every CTA of the cluster runs, with its flags zeroed, before DSMEM is touched

  // Barriers: data only crosses threads of the same rod, so a substep's two synchronisations can be per rod
  // (named barriers over the warps that hold the rod's threads; a warp holding the end of one rod and the start of
  // the next takes part in both, in rod order) instead of CTA-wide: rods then drift apart and fill each other's
  // pipeline bubbles.  Needs tpr >= 32 (a warp touches at most two rods) and <= 15 rods per CTA (barrier ids 1..15).
  // Planar model: warps past the last rod join the last rod's barrier, so that every warp has a first barrier.
  int bar_id0 = 0, bar_cnt0 = 0, bar_id1 = 0, bar_cnt1 = 0;
  const bool rod_barriers = A.sk_rodsync && G >= 32 && rods_per_cta >= 2 && rods_per_cta <= 15;
  if (rod_barriers) {
    const int wp = tid >> 5;
    for (int rr = 0; rr < rods_per_cta; rr++) {
      const int wa = (rr * G) >> 5, wb = (PLANAR && rr == rods_per_cta - 1) ? NT / 32 - 1 : (rr * G + G - 1) >> 5;
      if (wp >= wa && wp <= wb) {
        if (bar_cnt0 == 0) { bar_id0 = rr + 1; bar_cnt0 = 32 * (wb - wa + 1); }
        else { bar_id1 = rr + 1; bar_cnt1 = 32 * (wb - wa + 1); }
      }
    }
  }
  // planar model: whether this warp holds the start of a second rod, voted once so that the compiler knows it is the same
  // for the whole warp: the predicated second barrier then needs no WARPSYNC, and the substep loop branches uniformly
  const bool bar_two = PLANAR && __any_sync(0xffffffffu, bar_cnt1 != 0);
  auto rod_sync = [&]() {
    if (CLUSTER) { cluster_sync(); return; }
    if (!rod_barriers) { __syncthreads(); return; }
    if (bar_cnt0) asm volatile("bar.sync %0, %1;" ::"r"(bar_id0), "r"(bar_cnt0) : "memory");
    if (bar_cnt1) asm volatile("bar.sync %0, %1;" ::"r"(bar_id1), "r"(bar_cnt1) : "memory");
  };

  // plane models: lab <-> internal frame (z = plane normal), a signed permutation for axis-aligned normals
  const bool rot_frame = CONTACT && A.rot_on;
  auto to_int = [&](D (&u)[3]) {
    if (!rot_frame) return;
    const D a = u[0], b = u[1], c = u[2];
#pragma unroll
    for (int i = 0; i < 3; i++) u[i] = fma((D)A.lab2int[3 * i + 2], c, fma((D)A.lab2int[3 * i + 1], b, (D)A.lab2int[3 * i] * a));
  };
  auto to_lab = [&](D (&u)[3]) {      // transpose
    if (!rot_frame) return;
    const D a = u[0], b = u[1], c = u[2];
#pragma unroll
    for (int i = 0; i < 3; i++) u[i] = fma((D)A.lab2int[6 + i], c, fma((D)A.lab2int[3 + i], b, (D)A.lab2int[i] * a));
  };
  auto rows_to_int = [&](D (&M)[9]) {
#pragma unroll
    for (int i = 0; i < 3; i++) { D u[3] = {M[3 * i], M[3 * i + 1], M[3 * i + 2]}; to_int(u); M[3 * i] = u[0]; M[3 * i + 1] = u[1]; M[3 * i + 2] = u[2]; }
  };
  auto rows_to_lab = [&](D (&M)[9]) {
#pragma unroll
    for (int i = 0; i < 3; i++) { D u[3] = {M[3 * i], M[3 * i + 1], M[3 * i + 2]}; to_lab(u); M[3 * i] = u[0]; M[3 * i + 1] = u[1]; M[3 * i + 2] = u[2]; }
  };

  // constants of the FP64 part (the mixed mode reads double copies: a float dt would be off by 1e-8)
  const D c_dt = MIXED ? A.k_dt : (D)A.dt, c_half_dt = MIXED ? A.k_half_dt : (D)A.half_dt;
  const D c_cv = MIXED ? A.k_c_v : (D)A.c_v;

  // redo_count: [0] env-steps handed over for leaving the fast-math range, [1..3] by cause (an env can count under
  // several); [4] env-steps the planar model handed over for not being planar (no range failure)
  auto count_redo = [&](int dom) {
    if (PLANAR && (dom & 8)) { atomicAdd(A.redo_count + 4, 1ULL); return; }
    atomicAdd(A.redo_count, 1ULL);
    for (int b = 0; b < 3; b++) if (dom >> b & 1) atomicAdd(A.redo_count + 1 + b, 1ULL);
  };

  // ---- the segments this CTA runs ------------------------------------------------------------------------------
  const int K = A.n_substeps;
  const int P = gridDim.x, p = CLUSTER ? blockIdx.x / c_size : blockIdx.x;   // (cluster layout: one item per cluster)
  int i0, i1, off0, end1;
  if (A.sk_split) {
    const long long W = (long long)A.sk_items * K, b0 = W * p / P, b1 = W * (p + 1) / P;
    if (b1 <= b0) return;
    i0 = (int)(b0 / K); off0 = (int)(b0 - (long long)i0 * K);
    i1 = (int)((b1 - 1) / K); end1 = (int)(b1 - (long long)i1 * K);
  } else {
    i0 = i1 = p; off0 = 0; end1 = K;
  }
  // order: shared-with-successor part first, whole items next, shared-with-predecessor part last
  const bool tail_first = (i1 > i0) && (end1 < K);
  const bool head_last = (off0 > 0) && (i1 > i0);
  const int n_seg = i1 - i0 + 1;
  const int mid_lo = i0 + (head_last ? 1 : 0), n_mid = (i1 - (tail_first ? 1 : 0)) - mid_lo + 1;

  for (int q = 0; q < n_seg; q++) {
    int item;
    if (tail_first && q == 0) item = i1;
    else {
      const int k = q - (tail_first ? 1 : 0);
      item = (k < n_mid) ? mid_lo + k : i0;
    }
    const int s_begin = (item == i0) ? off0 : 0, s_end = (item == i1) ? end1 : K;
    const int env = item * rods_per_cta + r;
    const bool in_grid = in_cta && (env < A.n_env);
    bool selected = true;
    if (!FASTONLY && A.redo_filter) {   // fallback launch: flagged envs only; most CTAs have none and leave
      selected = in_grid && A.redo[env] != 0;
      if (!__syncthreads_or(selected)) continue;
    }
    const bool live = in_grid && selected;             // a thread of an env that is being stepped
    const bool active = live && !is_head;              // ... that owns a node / element of a rod
    const int rod = env * n_rod + arm;                 // global rod slot in the state arrays
    int dom_bad = 0;                                   // which range a fast-only thread left: 1 rotation, 2 bend, 4 stretch (damper map)
    const bool elem_ok = active && j < n, vor_ok = active && j < n - 1;
    // (fold layout: the tip node's record is record NT, published by the last element's thread)
    const int t_next = elem_ok ? ((FOLD && j == n - 1) ? NT : tid + 1) : tid;
    const int t_next2 = vor_ok ? ((FOLD && j == n - 2) ? NT : tid + 2) : t_next;
    const int t_prev = (active && j > 0) ? tid - 1 : ZR;

    D x[3] = {D(0), D(0), D(0)}, v[3] = {D(0), D(0), D(0)}, w[3] = {D(0), D(0), D(0)};
    D Q[9] = {D(1), D(0), D(0), D(0), D(1), D(0), D(0), D(0), D(1)};
    D xt[3] = {D(0), D(0), D(0)}, vt[3] = {D(0), D(0), D(0)};   // fold layout: the tip node, integrated by the last element's thread
    const bool is_last = FOLD && active && j == n - 1;
    ST *st = A.state + (size_t)(active ? rod : 0) * N_FIELDS * stride;
    const ST *bc = A.bc + (size_t)(active ? rod : 0) * BC_DIM;
    ST *hd = (MULTI && is_head && live) ? A.head + (size_t)env * HEAD_DIM : nullptr;   // the rigid head's state
    // travelling-wave muscle torque (muscle model): time, (sin, cos) of the wave's common phase w t + phi, and this
    // element's two amplitude combinations (below)
    const bool mus = MUS && A.muscle_on;
    D mus_t = D(0), mus_S = D(0), mus_C = D(1);
    if (s_begin > 0) {
      // continue an item the previous slot started: wait for its hand-over, then take the registers back
      if (tid == 0) {
        volatile int *f = A.sk_flag + (p - 1);
        while (*f == 0) __nanosleep(200);
        __threadfence();
      }
      __syncthreads();
      const D *sc = A.sk_scratch + (size_t)(p - 1) * SCR * NT;
      if constexpr (PLANAR) {   // rows: x0 x1 v0 v1 w1 Q0 Q1 Q6 Q7
        x[0] = sc[tid]; x[1] = sc[NT + tid]; v[0] = sc[2 * NT + tid]; v[1] = sc[3 * NT + tid]; w[1] = sc[4 * NT + tid];
        Q[0] = sc[5 * NT + tid]; Q[1] = sc[6 * NT + tid]; Q[6] = sc[7 * NT + tid]; Q[7] = sc[8 * NT + tid];
      } else {
#pragma unroll
        for (int c = 0; c < 3; c++) { x[c] = sc[c * NT + tid]; v[c] = sc[(3 + c) * NT + tid]; w[c] = sc[(15 + c) * NT + tid]; }
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c] = sc[(6 + c) * NT + tid];
      }
      if (CONTACT) { mus_S = sc[18 * NT + tid]; mus_C = sc[19 * NT + tid]; mus_t = sc[20 * NT + tid]; }
      if (FOLD) {
#pragma unroll
        for (int c = 0; c < 3; c++) { xt[c] = sc[(21 + c) * NT + tid]; vt[c] = sc[(24 + c) * NT + tid]; }
      }
      __syncthreads();
      if (tid == 0) A.sk_flag[p - 1] = 0;   // (graph-safe: the flag is back to 0 before the launch ends)
    } else {
      if (PLANAR && active) {
        x[0] = (D)st[F_POS * stride + j]; x[1] = (D)st[(F_POS + 1) * stride + j];
        v[0] = (D)st[F_VEL * stride + j]; v[1] = (D)st[(F_VEL + 1) * stride + j];
        w[1] = (D)st[(F_OMEGA + 1) * stride + j];
        Q[0] = (D)st[F_DIR * stride + j]; Q[1] = (D)st[(F_DIR + 1) * stride + j];
        Q[6] = (D)st[(F_DIR + 6) * stride + j]; Q[7] = (D)st[(F_DIR + 7) * stride + j];
      } else if (active) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
          x[c] = (D)st[(F_POS + c) * stride + j];
          v[c] = (D)st[(F_VEL + c) * stride + j];
          w[c] = (D)st[(F_OMEGA + c) * stride + j];   // slot n holds 0 (never written by anyone)
        }
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c] = (D)st[(F_DIR + c) * stride + j];  // slot n holds I
        if (CONTACT) { to_int(x); to_int(v); rows_to_int(Q); }
        if (is_last) {
#pragma unroll
          for (int c = 0; c < 3; c++) { xt[c] = (D)st[(F_POS + c) * stride + n]; vt[c] = (D)st[(F_VEL + c) * stride + n]; }
          if (CONTACT) { to_int(xt); to_int(vt); }
        }
      }
      if (MULTI && hd) {     // (assemblies stand on a z-normal plane: sr_create checks, no rotation here)
#pragma unroll
        for (int c = 0; c < 3; c++) { x[c] = (D)hd[c]; v[c] = (D)hd[3 + c]; w[c] = (D)hd[15 + c]; }
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c] = (D)hd[6 + c];
      }
      if (MIXED) {
        // FP64 node positions whose differences are the stored FP32 edge vectors exactly: node 0 (after the BC's
        // overwrite) + the running sum of the rod's edges, accumulated in element order
        D *eb = rec;   // 3 rows of NT + 2
#pragma unroll
        for (int c = 0; c < 3; c++) eb[c * (NT + 2) + tid] = elem_ok ? (D)st[(F_EDGE + c) * stride + j] : D(0);
        __syncthreads();
        if (active) {
          D xb[3];
#pragma unroll
          for (int c = 0; c < 3; c++) xb[c] = (D)st[(F_POS + c) * stride];
          if (A.bc_kind == BC_PENDULUM_SLIDER) { xb[1] = (D)bc[1]; xb[2] = (D)bc[2]; }
          else if (A.bc_kind != BC_FREE) { xb[0] = (D)bc[0]; xb[1] = (D)bc[1]; xb[2] = (D)bc[2]; }
          for (int i = 0; i < j; i++) {
#pragma unroll
            for (int c = 0; c < 3; c++) xb[c] += eb[c * (NT + 2) + tid - j + i];
          }
#pragma unroll
          for (int c = 0; c < 3; c++) x[c] = xb[c];
        }
        __syncthreads();
      }
    }
    // per-thread constants: zero where there is nothing to integrate (tip thread's pseudo-element, idle threads).
    // Only three 64-bit values stay live across the substep loop (dtim_cv, irg, base0): the kernel sits at the
    // 128-register cap of 2 x 256 threads per SM, and every further invariant becomes a local-memory reload per substep.
    const D dtim_cv = active ? (MIXED ? A.k_dt_inv_mass : (D)A.dt_inv_mass) * c_cv * ((j == 0 || j == n) ? D(2) : D(1)) : D(0);
    // 1 / rest_length_j (F_GAMMA = (L/n) / l0_j); the mixed mode's uniform 1/l0 is the double copy
    const D irg = (MIXED ? A.k_inv_rest_len : (D)A.inv_rest_len) * (elem_ok ? (D)st[F_GAMMA * stride + j] : D(1));
    const bool bc_thread = active && first && A.bc_kind != BC_FREE;
    // BCs pin node 0 / element 0 by overwriting after every kinematic update; applying the overwrite once and
    // never moving the pinned quantities is the same thing (see rod_kernel_packed.cuh): the BC thread integrates its
    // frame with a zero rotation vector
    if constexpr (PLANAR) {
      // the zeros this model relies on, in the pre-launch state (the same for every segment of an item)
      if (active) {
        auto f = [&](int field) { return (D)st[field * stride + j]; };
        bool flat = f(F_POS + 2) == D(0) && f(F_VEL + 2) == D(0);
        if (j < n)
          flat = flat && f(F_DIR + 2) == D(0) && f(F_DIR + 3) == D(0) && f(F_DIR + 4) == D(0) && f(F_DIR + 8) == D(0) &&
                 f(F_OMEGA) == D(0) && f(F_OMEGA + 2) == D(0);
        else      // slot n: the padding
          flat = flat && f(F_DIR) == D(1) && f(F_DIR + 1) == D(0) && f(F_DIR + 2) == D(0) && f(F_DIR + 3) == D(0) &&
                 f(F_DIR + 4) == D(1) && f(F_DIR + 5) == D(0) && f(F_DIR + 6) == D(0) && f(F_DIR + 7) == D(0) &&
                 f(F_DIR + 8) == D(1) && f(F_OMEGA) == D(0) && f(F_OMEGA + 1) == D(0) && f(F_OMEGA + 2) == D(0);
        if (bc_thread)
          flat = flat && (D)bc[2] == D(0) && (D)bc[5] == D(0) && (D)bc[11] == D(0) &&
                 (A.bc_kind == BC_PENDULUM_SLIDER || ((D)bc[6] == D(0) && (D)bc[7] == D(0)));
        if (!flat) dom_bad |= 8;
      }
      if (bc_thread) {
        if (A.bc_kind != BC_PENDULUM_SLIDER) x[0] = (D)bc[0];
        x[1] = (D)bc[1];
        Q[0] = (D)bc[3]; Q[1] = (D)bc[4]; Q[6] = (D)bc[9]; Q[7] = (D)bc[10];
      }
    } else if (bc_thread) {
      if (A.bc_kind == BC_PENDULUM_SLIDER) {
        x[1] = (D)bc[1]; x[2] = (D)bc[2];
#pragma unroll
        for (int m = 0; m < 3; m++) { Q[0 + m] = (D)bc[3 + m]; Q[6 + m] = (D)bc[9 + m]; }
      } else {
#pragma unroll
        for (int c = 0; c < 9; c++) Q[c] = (D)bc[3 + c];
        // (a moving base is positioned by its controller below — and, when this CTA continues an item another one
        // started, by the hand-over: the anchor stored at finalize time is not where the base is)
        if (!(LAPL && A.bc_kind == BC_MOVING_BASE)) {
#pragma unroll
          for (int c = 0; c < 3; c++) x[c] = (D)bc[c];
        }
        if (CONTACT) { rows_to_int(Q); to_int(x); }
      }
    }
    // plane models: rest curvature at Voronoi point j (actuation), constant during a launch; the muscle wave
    D rk[3] = {D(0), D(0), D(0)};
    D mus_P = D(0), mus_R = D(0);
    if constexpr (CONTACT) {
      if (A.rest_kappa && vor_ok) {
#pragma unroll
        for (int c = 0; c < 3; c++) rk[c] = (D)A.rest_kappa[((size_t)rod * 3 + c) * stride + j];
      }
      if (mus && active) {
        // (the cluster layout: every rank reads the clock mu[0] here, ahead of its first cluster barrier of the item;
        // rank 0's lead alone writes it back, after the last one)
        // MuscleTorques (continuum_snake.py:186-198): element k gets Q_k d (m_k [k >= 1] - m_{k+1} [k <= n-2]),
        // m_k = min(1, t/ramp) beta_{n-1-k} sin(w t - kw s_{n-1-k} + phi).  sin(p - s) = sin p cos s - cos p sin s, so
        // m_k - m_{k+1} = ramp (sin p * P - cos p * R) with per-element constants P = b0 cos s0 - b1 cos s1,
        // R = b0 sin s0 - b1 sin s1; (sin p, cos p) advance by the fixed angle w dt per substep (a rotation, seeded
        // from sincos at the start of the launch) instead of two libm sines per element and substep.
        const double *mu = A.muscle + (size_t)env * A.muscle_dim;
        if (s_begin == 0) {
          mus_t = mu[0];
          sincos(A.mus_omega * (mus_t + (double)c_half_dt) + A.mus_phase, &mus_S, &mus_C);
        }
        if (elem_ok) {
          const double kw = mu[1], inv_n = 1.0 / (double)n;
          const int k0 = n - 1 - j, k1 = n - 2 - j;
          double b0 = 0.0, s0 = 0.0, b1 = 0.0, s1 = 0.0;
          if (j >= 1) { b0 = mu[2 + k0]; s0 = kw * ((double)(k0 + 1) * inv_n); }
          if (j <= n - 2) { b1 = mu[2 + k1]; s1 = kw * ((double)(k1 + 1) * inv_n); }
          double sn0, cs0, sn1, cs1;
          sincos(s0, &sn0, &cs0); sincos(s1, &sn1, &cs1);
          mus_P = b0 * cs0 - b1 * cs1; mus_R = b0 * sn0 - b1 * sn1;
        }
      }
    }
    // MuscleTorquesWithVaryingBetaSplines (muscle_torques_with_bspline.py:126-160,181-228): per enabled material
    // direction d, external_torques[d, k] += mag_d[k]; mag is re-evaluated (not-a-knot cubic through the rate-limited
    // control values, at s = cumsum(current lengths)) in every substep that finds the cached values different from the
    // caller's targets, and kept otherwise — across launches too (the cache lives in HBM, A.spline).  The forcing
    // mutates that cache inside the launch, so this model only exists as the safe kernel (a fast-only run that is
    // re-done would apply the rate limit twice).
    const bool spl = SPL && A.spline_mask != 0;
    double *sp = (spl && active) ? A.spline + (size_t)env * A.spline_dim : nullptr;
    const int sP = A.spline_p, sCH = 2 * sP + 2;
    D smag[3] = {D(0), D(0), D(0)};
    if constexpr (SPL) {
      if (spl && elem_ok) {
#pragma unroll
        for (int d = 0; d < 3; d++)
          if (A.spline_mask >> d & 1) smag[d] = sp[3 * sCH + d * n + j];
      }
    }
    // SoftPendulum3D-v0: the base is commanded by the host (set_action, soft_pendulum_3d.py:106-120): float32
    // displacement, float64 clipped position, velocity = actual displacement / (step_skip * time_step); the base jumps
    // at once and is re-pinned after every kinematic update.  The controller's state (aux) is only written back by the
    // epilogue of the item's last segment, so a fallback re-run or a split item recomputes the same command from the
    // pre-launch aux.
    // (Only the rod's first thread uses the command, so it lives in shared memory, sh_base[r] = {x, y, v_x, v_y}, not
    // in four 64-bit registers of every thread: the filter's taps need the registers, see below.)
    const bool moving = LAPL && bc_thread && A.bc_kind == BC_MOVING_BASE;
    if constexpr (LAPL) {
      if (moving) {
        const ST *aux = A.aux + (size_t)env * AUX_DIM;
        D pin_x = (D)aux[0], pin_y = (D)aux[1], base_vx = (D)aux[3], base_vy = (D)aux[4];
        if (A.model == MODEL_SOFT_PENDULUM_3D && K > 0) {
          const float act_f0 = A.action_dim > 0 ? A.action[(size_t)env * A.action_dim] : 0.0f;
          const float act_f1 = A.action_dim > 1 ? A.action[(size_t)env * A.action_dim + 1] : 0.0f;
          const D px = pin_x, py = pin_y;
          D nx = px + (D)__fmul_rn(A.base_step_f32, act_f0), ny = py + (D)__fmul_rn(A.base_step_f32, act_f1);
          nx = fmin(fmax(nx, -(D)A.base_limit), (D)A.base_limit);
          ny = fmin(fmax(ny, -(D)A.base_limit), (D)A.base_limit);
          base_vx = (nx - px) * A.inv_move_period; base_vy = (ny - py) * A.inv_move_period;
          pin_x = nx; pin_y = ny;
        }
        if (s_begin == 0) { x[0] = pin_x; x[1] = pin_y; x[2] = (D)bc[2]; }
        sh_base[r][0] = pin_x; sh_base[r][1] = pin_y; sh_base[r][2] = base_vx; sh_base[r][3] = base_vy;   // (own thread only: no barrier)
      }
    }
    const bool pin_slider = bc_thread && A.bc_kind == BC_PENDULUM_SLIDER;
    const bool pin_fixed = bc_thread && A.bc_kind != BC_PENDULUM_SLIDER && !moving;
    const bool z12 = pin_slider || pin_fixed;   // v_y, v_z, w_x, w_z are pinned by both; v_x, w_y by the clamp only
    // x component of the velocity update's constant term: dt c_v g_x, or, on the node that carries the base point
    // force, dt c_v F / m (soft_pendulum/build.py:94-105: the force REPLACES gravity's x component there)
    D base0 = MIXED ? A.k_gdt_cv[0] : (D)A.gdt_cv[0];
    if (!LAPL && active && first && A.point_force) base0 = (A.action_dim > 0 ? (D)A.action[(size_t)env * A.action_dim] : D(0)) * dtim_cv;

    // x += hh v ; Q <- R(hh w) Q (merged half steps)
    auto kinematic = [&](D hh, D eps) {
      const D hw = bc_thread ? D(0) : hh;
      if constexpr (PLANAR) {
        const D a1 = hw * w[1];
        x[0] = fma(hh, v[0], x[0]); x[1] = fma(hh, v[1], x[1]);
        const D q = fma(a1, a1, D(1e-300));
        if (hi_abs(q) > A.lim_rot_hi) dom_bad |= 1;
        rotate_directors_planar(A.sincg, A.cosch, a1, q, eps, Q);
        return;
      }
      D a0 = hw * w[0], a1 = hw * w[1], a2 = hw * w[2];
#pragma unroll
      for (int c = 0; c < 3; c++) x[c] = fma(hh, v[c], x[c]);
      if (FOLD && is_last) {
#pragma unroll
        for (int c = 0; c < 3; c++) xt[c] = fma(hh, vt[c], xt[c]);
      }
      if (LAPL && moving) { x[0] = sh_base[r][0]; x[1] = sh_base[r][1]; }
      D q = fma(a2, a2, fma(a1, a1, fma(a0, a0, D(1e-300))));   // (+1e-300: rsqrt(q) below stays finite at rest)
      const bool out = hi_abs(q) > A.lim_rot_hi;
      if (FASTONLY) {
        if (out) dom_bad |= 1;
        rotate_directors_lean(A.sincg, A.cosch, a0, a1, a2, q, eps, Q);
      } else if (!out) rotate_directors_lean(A.sincg, A.cosch, a0, a1, a2, q, eps, Q);
      else rotate_directors_ref<D>(a0, a1, a2, Q);
    };

    // BodyBoundaryCondition on the head (utils/custom_elastica/constraint.py:43-58): z pinned, d3 = z, d1 / d2 renormalised in-plane
    auto head_constrain_values = [&]() {
      if (MULTI && hd) {
        x[2] = (D)hd[18];
        Q[6] = D(0); Q[7] = D(0); Q[8] = D(1);
#pragma unroll
        for (int i = 0; i < 2; i++) {
          const D il = rsqrt_nr(Q[3 * i] * Q[3 * i] + Q[3 * i + 1] * Q[3 * i + 1]);   // rows stay ~unit: never 0
          Q[3 * i] *= il; Q[3 * i + 1] *= il; Q[3 * i + 2] = D(0);
        }
      }
    };
    if (s_begin == 0 && K > 0) { kinematic(c_half_dt, D(1e-14)); head_constrain_values(); }

    bool spl_settled = false;   // spline model: the cached control values have reached their targets
    // first substep of the segment: rule out a state that starts beyond 90 degrees of bend (the planar model runs that
    // substep as a copy of its own instead)
    bool check_trace = true;
    auto substep = [&](auto last_tag, int s_now) {
      constexpr bool last = decltype(last_tag)::value;
      D mtq[3] = {D(0), D(0), D(0)};
      // zero, but not provably so (a launch never has 2^30 substeps): see the bend polynomial below
      const int oz = (CONTACT || LAPL || SPL) ? (s_now >> 30) : 0;
      const RodArgs<ST> &Z = (&A)[oz];   // the kernel parameters through that index: constant-bank loads that stay inside the loop
      if constexpr (CONTACT) {
        if (mus) {
          mus_t += (double)c_half_dt;   // time of the force evaluation: after the first half step
          const D cf = fmin(1.0, mus_t * A.mus_inv_ramp) * fma(mus_S, mus_P, -(mus_C * mus_R));
#pragma unroll
          for (int i = 0; i < 3; i++)
            mtq[i] = fma(Q[3 * i + 2], (D)A.mus_dir[2], fma(Q[3 * i + 1], (D)A.mus_dir[1], Q[3 * i] * (D)A.mus_dir[0])) * cf;
          mus_t += (double)c_half_dt;
          const D nS = fma(mus_C, A.mus_sd, mus_S * A.mus_cd);   // phase += w dt
          mus_C = fma(-mus_S, A.mus_sd, mus_C * A.mus_cd);
          mus_S = nS;
        }
      }
      // ---- publish what the neighbours need ----------------------------------------------------------------
      {
        double2 *o = reinterpret_cast<double2 *>(rec + LEAN_REC * tid);
        o[0] = make_double2(x[0], x[1]); o[1] = make_double2(x[2], v[0]); o[2] = make_double2(v[1], v[2]);
        o[3] = make_double2(Q[0], Q[1]); o[4] = make_double2(Q[2], Q[3]); o[5] = make_double2(Q[4], Q[5]);
        o[6] = make_double2(Q[6], Q[7]); rec[LEAN_REC * tid + 14] = Q[8];
        if (CLUSTER && tid < 2 && c_rank > 0) {   // nodes j + 1, j + 2 of the previous rank's last two threads
          double2 *h = cluster_smem(reinterpret_cast<double2 *>(rec + LEAN_REC * (NT + tid)), c_rank - 1);
#pragma unroll
          for (int k = 0; k < 7; k++) h[k] = o[k];
          reinterpret_cast<D *>(h)[14] = Q[8];
        }
        if (FOLD && is_last) {
          double2 *ot = reinterpret_cast<double2 *>(rec + LEAN_REC * NT);
          ot[0] = make_double2(xt[0], xt[1]); ot[1] = make_double2(xt[2], vt[0]); ot[2] = make_double2(vt[1], vt[2]);
        }
      }
      rod_sync();

      // ---- geometry, shear/stretch strain, internal force ---------------------------------------------------
      D dx[3], dv[3], dx2[3], Qn[9];
      {
        const double2 *qq = reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next);
        const double2 a0 = qq[0], a1 = qq[1], a2 = qq[2], a3 = qq[3], a4 = qq[4], a5 = qq[5], a6 = qq[6];
        Qn[0] = a3.x; Qn[1] = a3.y; Qn[2] = a4.x; Qn[3] = a4.y; Qn[4] = a5.x; Qn[5] = a5.y;
        Qn[6] = a6.x; Qn[7] = a6.y; Qn[8] = rec[LEAN_REC * t_next + 14];
        const double2 b0 = *reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next2);
        const D b2 = rec[LEAN_REC * t_next2 + 2];
        dx[0] = a0.x - x[0]; dx[1] = a0.y - x[1]; dx[2] = a1.x - x[2];
        dv[0] = a1.y - v[0]; dv[1] = a2.x - v[1]; dv[2] = a2.y - v[2];
        dx2[0] = b0.x - a0.x; dx2[1] = b0.y - a0.y; dx2[2] = b2 - a1.x;
      }
      if (!elem_ok) dx[2] = (D)A.rest_len;   // keeps the pseudo-element's quantities finite
      if (!vor_ok) dx2[2] = (D)A.rest_len;
      // lengths: squared in FP64 (they are sums of squares of the FP64 edge), roots and everything after in F
      const F l2 = (F)dot3(dx, dx), l2n = (F)dot3(dx2, dx2);
      const F il = rsqrt_nr(l2), iln = rsqrt_nr(l2n);
      const F lg = fma(l2, il, F(1e-14));                 // |dx| + 1e-14 (reference guard)
      const F ilg = MIXED ? il : fma(F(-1e-14) * il, il, il);   // 1/(l + 1e-14) to first order in 1e-14/l
      const F lgn = fma(l2n, iln, F(1e-14));              // length of element j+1, recomputed locally
      if constexpr (SPL) {
        if (spl) {
          rec[LEAN_REC * tid + 15] = lg;     // element length, for the arc-length prefix sums below (spare word of the record)
          // the forcing's own bookkeeping, once per env.  The targets cannot change during a launch and the cached
          // values only change here, so once a substep finds them equal nothing happens until the launch ends: the
          // first thread then stops re-reading the cache from HBM (a chain of dependent global loads ahead of the
          // barrier the whole rod waits at).
          if (active && first && !spl_settled) {
            int need = 0;
            for (int d = 0; d < 3; d++) {
              if (!(A.spline_mask >> d & 1)) continue;
              double *ch = sp + d * sCH;
              bool differ = ch[2 * sP] == 0.0;                      // initial_call_flag
              for (int i = 0; i < sP; i++) differ = differ || !(ch[sP + i] == ch[i]);   // not np.array_equal
              if (differ) {
                ch[2 * sP] = 1.0;
                for (int i = 0; i < sP; i++) {                      // filter_activation
                  const double dd = ch[i] - ch[sP + i];
                  const double sg = (double)((dd > 0.0) - (dd < 0.0));
                  ch[sP + i] += sg * fmin(A.spline_rate, fabs(dd));
                }
                need |= 1 << d;
              }
            }
            if constexpr (CLUSTER) {   // every rank reads it, also when 0: rank 0's lead stores it into each rank's sh_need[0]
              for (int c = 0; c < c_size; c++) *cluster_smem(&sh_need[0], c) = need;
            } else {
              sh_need[r] = need;
            }
            spl_settled = (need == 0);
          }
        }
      }
      const F e = lg * (F)irg;
      const F em1 = fma(lg, (F)irg, F(-1.0));
      const F inv_e = A.rest_len * ilg;
      const F inv_e_s = elem_ok ? inv_e : F(0);           // the tip thread's pseudo-element carries no stress
      const F ede = (F)dot3(dx, dv) * (ilg * ilg);        // (de/dt) / e = (dx . dv) / l^2
      // sigma = e Q t - z = Q dx / l0 - z exactly (e t = dx / l0): no tangent needed here.  FP64 in both modes: this
      // is the difference of O(1) quantities everything else hangs on.
      D Qdx[3];
#pragma unroll
      for (int i = 0; i < 3; i++) Qdx[i] = Q[3 * i] * dx[0];
#pragma unroll
      for (int i = 0; i < 3; i++) Qdx[i] = fma(Q[3 * i + 1], dx[1], Qdx[i]);
#pragma unroll
      for (int i = 0; i < 3; i++) Qdx[i] = fma(Q[3 * i + 2], dx[2], Qdx[i]);
      const D s3 = fma(Qdx[2], irg, D(-1.0));             // stretch strain, against the element's own rest length
      // n = S (sigma - 0): shear components are O(strain); the stretch component is a difference of near-equal numbers
      const F qd0 = (F)Qdx[0], qd1 = (F)Qdx[1], qd2 = (F)Qdx[2];
      F nst[3];
      nst[0] = A.S_over_l[0] * qd0;
      nst[1] = A.S_over_l[0] * qd1;
      nst[2] = MIXED ? A.S[2] * (F)s3 : (F)fma((D)A.S[2], Qdx[2] * irg, -(D)A.S[2]);
      F sfl[3];
      {
        D sd[3];
        const D n0 = (D)nst[0], n1 = (D)nst[1], n2 = (D)nst[2];
#pragma unroll
        for (int i = 0; i < 3; i++) sd[i] = Q[i] * n0;
#pragma unroll
        for (int i = 0; i < 3; i++) sd[i] = fma(Q[3 + i], n1, sd[i]);
#pragma unroll
        for (int i = 0; i < 3; i++) sd[i] = fma(Q[6 + i], n2, sd[i]);
#pragma unroll
        for (int i = 0; i < 3; i++) sfl[i] = (F)sd[i] * inv_e_s;
      }

      if constexpr (MULTI) {
        // FixedJoint2Rigid(head, -1, arm, 0) (utils/custom_elastica/joint.py:48-123 forces, :125-219 torques): spring
        // + normal damping between the head's rim point and node 0, restoring force on node 1 towards the mounting
        // direction.  Joint a of an env is computed by the env's a-th thread (not by arm a's own first thread): the
        // joints of an env then share one warp's instructions instead of costing every warp that holds the start of an
        // arm the whole block.  Inputs come from the published records; the result {reaction on the head, couple on
        // the head, couple on element 0} goes to the joint record of arm a's first thread, which re-reads its share
        // after the barrier, as the head does.
        if (live && u_grp < n_rod && has_head) {
          const int ta = r * G + u_grp * tpr;                    // arm u_grp's first thread
          D hx[3], hv[3], d2[3], Qh[9], ax_[3], av[3], aQ[9], adx[3];
          {
            const double2 *qh = reinterpret_cast<const double2 *>(rec + LEAN_REC * t_head);
            const double2 h0 = qh[0], h1 = qh[1], h2 = qh[2], h3 = qh[3], h4 = qh[4], h5 = qh[5], h6 = qh[6];
            hx[0] = h0.x; hx[1] = h0.y; hx[2] = h1.x; hv[0] = h1.y; hv[1] = h2.x; hv[2] = h2.y;
            Qh[0] = h3.x; Qh[1] = h3.y; Qh[2] = h4.x; Qh[3] = h4.y; Qh[4] = h5.x; Qh[5] = h5.y; Qh[6] = h6.x; Qh[7] = h6.y;
            Qh[8] = rec[LEAN_REC * t_head + 14];
            d2[0] = Qh[3]; d2[1] = Qh[4]; d2[2] = Qh[5];
            const double2 *qa = reinterpret_cast<const double2 *>(rec + LEAN_REC * ta);
            const double2 a0 = qa[0], a1 = qa[1], a2 = qa[2], a3 = qa[3], a4 = qa[4], a5 = qa[5], a6 = qa[6];
            ax_[0] = a0.x; ax_[1] = a0.y; ax_[2] = a1.x; av[0] = a1.y; av[1] = a2.x; av[2] = a2.y;
            aQ[0] = a3.x; aQ[1] = a3.y; aQ[2] = a4.x; aQ[3] = a4.y; aQ[4] = a5.x; aQ[5] = a5.y; aQ[6] = a6.x; aQ[7] = a6.y;
            aQ[8] = rec[LEAN_REC * ta + 14];
            const double2 b0 = *reinterpret_cast<const double2 *>(rec + LEAN_REC * (ta + 1));
            adx[0] = b0.x - ax_[0]; adx[1] = b0.y - ax_[1]; adx[2] = rec[LEAN_REC * (ta + 1) + 2] - ax_[2];
          }
          const D cs = (D)A.joint_cs[u_grp][0], sn_ = (D)A.joint_cs[u_grp][1];
          const D dir[3] = {-(cs * d2[0] - sn_ * d2[1]), -(sn_ * d2[0] + cs * d2[1]), -d2[2]};   // -Rz(angle) d2
          const D anchor[3] = {hx[0] + A.joint_radius * dir[0], hx[1] + A.joint_radius * dir[1], D(0) + A.joint_radius * dir[2]};
          const D dd[3] = {ax_[0] - anchor[0], ax_[1] - anchor[1], ax_[2] - anchor[2]};
          const D dist2 = dot3(dd, dd);
          const D inv = (dist2 <= D(4.930380657631324e-24)) ? D(0) : rsqrt_nr(dist2);   // 1 / dist; the reference's guard dist <= 1e4 eps (discards rsqrt(0))
          const D nh[3] = {dd[0] * inv, dd[1] * inv, dd[2] * inv};
          const D rvn = (av[0] - hv[0]) * nh[0] + (av[1] - hv[1]) * nh[1] + (av[2] - hv[2]) * nh[2];
          D cf[3], fd[3], tauj[3];
#pragma unroll
          for (int c = 0; c < 3; c++) {
            cf[c] = A.joint_k * dd[c] - A.joint_nu * (rvn * nh[c]);
            const D tgt = anchor[c] + A.rest_len * dir[c];
            fd[c] = -A.joint_kt * ((ax_[c] + adx[c]) - tgt);    // node 1 of the arm
          }
          cross3(adx, fd, tauj);                                 // link_direction x force
          D *o = sj + LEAN_JREC * ta;
#pragma unroll
          for (int i = 0; i < 3; i++) {
            o[i] = cf[i];
            o[3 + i] = -(Qh[3 * i] * tauj[0] + Qh[3 * i + 1] * tauj[1] + Qh[3 * i + 2] * tauj[2]);
            o[6 + i] = aQ[3 * i] * tauj[0] + aQ[3 * i + 1] * tauj[1] + aQ[3 * i + 2] * tauj[2];
          }
        }
      }
      // ---- curvature, bending couple --------------------------------------------------------------------------
      F vec[3];
      {
        // axial part of Rm - Rm^T (Rm = Q_{j+1} Q_j^T), each component one 6-term FMA chain (FP64: differences of products)
        auto rm_diff = [&](int a, int b) {
          D t = Qn[3 * a] * Q[3 * b];
          t = fma(Qn[3 * a + 1], Q[3 * b + 1], t);
          t = fma(Qn[3 * a + 2], Q[3 * b + 2], t);
          t = fma(-Qn[3 * b], Q[3 * a], t);
          t = fma(-Qn[3 * b + 1], Q[3 * a + 1], t);
          return fma(-Qn[3 * b + 2], Q[3 * a + 2], t);
        };
        vec[0] = (F)rm_diff(2, 1); vec[1] = (F)rm_diff(0, 2); vec[2] = (F)rm_diff(1, 0);
      }
      // |vec|^2 = 4 sin^2(theta): below 90 degrees the log-map factor -theta'/(2 sin theta') / D (theta' the
      // reference's guarded angle acos(cos(theta) - 1e-10)) is a smooth function of it alone.  A bend cannot pass
      // the polynomial's range unseen: every element rotates by <= 0.1 rad per update (the rotation range check),
      // so the angle between neighbours grows by <= 0.2 rad per substep and lands in (range, 90 degrees) first;
      // the first substep of a segment checks the trace once to rule out a state that starts beyond.
      F w2 = dot3(vec, vec);
      if (!vor_ok) w2 = F(0);
      constexpr bool MIDBEND = MODEL == LeanModel::PLANE || MODEL == LeanModel::MUSCLE;   // actuated arms on the plane: the 37-degree map
      bool bend_out = out_of_range(w2, MIDBEND ? A.lim_bendm_hi : A.lim_bend_hi, A.limf_bend);
      F u_ref = F(0);
      if constexpr (MULTI) {
        // the 10-element arms of the octopus assemblies bend up to ~45 degrees per element: full-range map in
        // u = sin^2(theta'/2) from the trace (u <= 1/4, 60 degrees), as in rod_kernel_packed.cuh
        const D tr = fma(Qn[8], Q[8], fma(Qn[7], Q[7], fma(Qn[6], Q[6], fma(Qn[5], Q[5], fma(Qn[4], Q[4], fma(Qn[3], Q[3],
                     fma(Qn[2], Q[2], fma(Qn[1], Q[1], Qn[0] * Q[0]))))))));
        u_ref = fma(D(-0.25), tr, D(0.75 + 0.5e-10));
        if (!vor_ok) u_ref = D(5e-11);
        bend_out = !(u_ref <= D(kSmallBendU));
      } else if (check_trace || !FASTONLY) {
        check_trace = false;
        const D tr = fma(Qn[8], Q[8], fma(Qn[7], Q[7], fma(Qn[6], Q[6], fma(Qn[5], Q[5], fma(Qn[4], Q[4], fma(Qn[3], Q[3],
                     fma(Qn[2], Q[2], fma(Qn[1], Q[1], Qn[0] * Q[0]))))))));
        bend_out = bend_out || (vor_ok && !(tr > D(2.0)));   // cos(theta) <= 1/2
        u_ref = (F)fma(D(-0.25), tr, D(0.75 + 0.5e-10));     // sin^2(theta'/2), for the reference map
      }
      if (FASTONLY && bend_out) dom_bad |= 2;
      F fs;
      if constexpr (MULTI) {
        const D g = theta_over_sin(Z.poly, u_ref);
        const D cot = fma(D(-2.0), u_ref, D(1.0)) * rsqrt_approx(D(4.0) * u_ref * (D(1.0) - u_ref));   // scales the 1e-14 guard term only
        fs = g * fma(D(0.5e-14), cot, D(-0.5)) * A.inv_rest_vor;
      } else {
        // ascending powers of w2 (degree 9), pre-multiplied by -1/(2 D); even / odd halves interleaved.  (Plane
        // models: indexed through a register the compiler cannot see through, so that the ten coefficients are
        // constant-bank loads inside the loop instead of hoisted, spilled and reloaded registers.)
        const F *c = MIDBEND ? Z.bendw_mid : Z.bendw;
        const F z = w2 * w2;
        F pe, po;
        if constexpr (MIDBEND) {      // degree 13
          pe = fma(c[12], z, c[10]); po = fma(c[13], z, c[11]);
          pe = fma(pe, z, c[8]); po = fma(po, z, c[9]);
          pe = fma(pe, z, c[6]); po = fma(po, z, c[7]);
        } else {                      // degree 9
          pe = fma(c[8], z, c[6]); po = fma(c[9], z, c[7]);
        }
        pe = fma(pe, z, c[4]); po = fma(po, z, c[5]);
        pe = fma(pe, z, c[2]); po = fma(po, z, c[3]);
        pe = fma(pe, z, c[0]); po = fma(po, z, c[1]);
        fs = fma(po, w2, pe);
      }
      // reference map (elastica/_rotations.py:_inv_rotate) for this thread only
      if (!FASTONLY && bend_out) fs = bend_factor_ref<F>(u_ref) * A.inv_rest_vor;
      F kp[3], tau[3];
#pragma unroll
      for (int i = 0; i < 3; i++) kp[i] = vec[i] * fs;
      F kx0, kx1, kx2 = F(0);
      if constexpr (CONTACT) {
        // with a rest curvature the cross product keeps all its terms: kappa x (B (kappa - kappa0)), times D / 2
        tau[0] = A.B[0] * (kp[0] - rk[0]); tau[1] = A.B[0] * (kp[1] - rk[1]); tau[2] = A.B[2] * (kp[2] - rk[2]);
        kx0 = fma(kp[1], tau[2], -(kp[2] * tau[1])) * A.half_rest_vor;
        kx1 = fma(kp[2], tau[0], -(kp[0] * tau[2])) * A.half_rest_vor;
        kx2 = fma(kp[0], tau[1], -(kp[1] * tau[0])) * A.half_rest_vor;
      } else {
        tau[0] = A.B[0] * kp[0]; tau[1] = A.B[0] * kp[1]; tau[2] = A.B[2] * kp[2];
        // kappa x (B kappa) with B1 = B2:  ((B3 - B1) k2 k3, (B1 - B3) k1 k3, 0)
        const F k2b = kp[2] * A.BDH;                        // (B3 - B1) D / 2: the quadrature weight of A_h folded in
        kx0 = kp[1] * k2b; kx1 = -(kp[0] * k2b);
      }
      const F eps_v = (lgn + lg) * A.half_inv_rest_vor;
      F ie3 = rcp_nr(eps_v * eps_v * eps_v);
      if (!vor_ok) ie3 = F(0);
      const F m0 = tau[0] * ie3, m1 = tau[1] * ie3, m2 = tau[2] * ie3;
      // local couples share one 1/e factor:  (Qt x n) l0 + (Jw/e) x w + (Jw/e) (de/dt)/e
      //   = [ (Q dx) x n + (Jw) x w + (Jw) (de/dt)/e ] / e ; with S1 = S2 and J1 = J2 the cross products collapse:
      //   (Q dx) x n = (Qdx1 c, -Qdx0 c, 0), c = n3 - S1' Qdx3 ;  (Jw) x w = (w1 t, -w0 t, 0), t = (J1 - J3) w3
      const F wf0 = (F)w[0], wf1 = (F)w[1], wf2 = (F)w[2];
      const F cc = fma(-A.S_over_l[0], qd2, nst[2]);
      const F tg = -(wf2 * A.J[0]);                       // (J1 - J3) w3 = -J1 w3 for a circular section (J3 = 2 J1)
      const F je = ede * A.J[0], je2 = je + je;
      const F h0 = fma(qd1, cc, fma(wf1, tg, je * wf0));
      const F h1 = fma(-qd0, cc, fma(-wf0, tg, je * wf1));
      const F h2 = je2 * wf2;
      F tql[3];
      tql[0] = fma(h0, inv_e, fma(kx0, ie3, m0));          // + m_j + c_j/2  (own element)
      tql[1] = fma(h1, inv_e, fma(kx1, ie3, m1));
      tql[2] = CONTACT ? fma(h2, inv_e, fma(kx2, ie3, m2)) : fma(h2, inv_e, m2);
      // {s0 s1 | s2 N0 | N1 m2}: N = c_j/2 - m_j goes to element j+1 (third component: -m2, negated by the reader)
      if (MIXED) {
        float4 *o = reinterpret_cast<float4 *>(sn + SNR * tid);
        o[0] = make_float4((float)sfl[0], (float)sfl[1], (float)sfl[2], (float)fma(kx0, ie3, -m0));
        o[1] = make_float4((float)fma(kx1, ie3, -m1), (float)m2, 0.0f, 0.0f);
      } else {
        double2 *o = reinterpret_cast<double2 *>(sn + SNR * tid);
        o[0] = make_double2((double)sfl[0], (double)sfl[1]);
        o[1] = make_double2((double)sfl[2], (double)fma(kx0, ie3, -m0));
        o[2] = make_double2((double)fma(kx1, ie3, -m1), CONTACT ? (double)fma(-kx2, ie3, m2) : (double)m2);   // (the reader subtracts)
        if (CLUSTER && tid == NT - 1 && c_rank + 1 < c_size) {   // element j - 1 of the next rank's thread 0
          double2 *h = cluster_smem(reinterpret_cast<double2 *>(sn - SNR), c_rank + 1);
          h[0] = o[0]; h[1] = o[1]; h[2] = o[2];
        }
        if (CLUSTER && CONTACT && tid == 0 && c_rank > 0) {   // element j + 1 of the previous rank's last thread (the plane's stage 1)
          double2 *h = cluster_smem(reinterpret_cast<double2 *>(sn + SNR * NT), c_rank - 1);
          h[0] = o[0]; h[1] = o[1];
        }
      }
      // rotational damper c_w^e = c_w exp((e-1) ln c_w) as a quadratic in (e-1) (coefficients made on the host; the
      // range limit keeps the dropped cubic term below 1.4e-15); c_w1 = c_w2 for a circular cross-section
      F cw0, cw2;
      {
        const bool out = out_of_range(em1, (CONTACT || LAPL || SPL) ? A.lim_em1c_hi : A.lim_em1_hi, A.limf_em1);
        if (FASTONLY && out && elem_ok) dom_bad |= 4;
        if (FASTONLY || !out) {
          if constexpr (CONTACT || LAPL || SPL) {   // harder dampers, larger stretches: degree 6, |z| <= kLeanExpZc
            F p0 = fma(Z.cwc[0][6], em1, Z.cwc[0][5]), p2 = fma(Z.cwc[1][6], em1, Z.cwc[1][5]);
#pragma unroll
            for (int k = 4; k >= 0; k--) { p0 = fma(p0, em1, Z.cwc[0][k]); p2 = fma(p2, em1, Z.cwc[1][k]); }
            cw0 = p0; cw2 = p2;
          } else {
            cw0 = fma(fma(A.cwp[0][2], em1, A.cwp[0][1]), em1, A.cwp[0][0]);
            cw2 = fma(fma(A.cwp[1][2], em1, A.cwp[1][1]), em1, A.cwp[1][0]);
          }
        } else {
          cw0 = exp_ref<F>(e * A.logc_w[0]);
          cw2 = exp_ref<F>(e * A.logc_w[2]);
        }
      }
      if (last && active) {
        // stale observables of the reference (SURVEY A.6): last force evaluation
        D tg_out[3] = {dx[0] * (D)ilg, dx[1] * (D)ilg, dx[2] * (D)ilg};
        if (CONTACT) to_lab(tg_out);
#pragma unroll
        for (int i = 0; i < 3; i++) {
          st[(F_TAN + i) * stride + j] = (ST)tg_out[i];
          st[(F_KAPPA + i) * stride + j] = (ST)kp[i];
        }
        st[(F_SIGMA + 0) * stride + j] = (ST)(Qdx[0] * irg);
        st[(F_SIGMA + 1) * stride + j] = (ST)(Qdx[1] * irg);
        st[(F_SIGMA + 2) * stride + j] = (ST)s3;
        st[F_DIL * stride + j] = (ST)e;
      }
      rod_sync();

      // ---- add the left neighbour's share, dynamic step ---------------------------------------------------------
      F fint[3], tq[3];
      if (MIXED) {
        const float4 *qq = reinterpret_cast<const float4 *>(sn + SNR * t_prev);
        const float4 a0 = qq[0], a1 = qq[1];
        fint[0] = sfl[0] - (F)a0.x; fint[1] = sfl[1] - (F)a0.y; fint[2] = sfl[2] - (F)a0.z;
        tq[0] = tql[0] + (F)a0.w; tq[1] = tql[1] + (F)a1.x; tq[2] = tql[2] - (F)a1.y;
      } else {
        const double2 *qq = reinterpret_cast<const double2 *>(sn + SNR * t_prev);
        const double2 a0 = qq[0], a1 = qq[1], a2 = qq[2];
        fint[0] = sfl[0] - (F)a0.x; fint[1] = sfl[1] - (F)a0.y; fint[2] = sfl[2] - (F)a1.x;
        tq[0] = tql[0] + (F)a1.y; tq[1] = tql[1] + (F)a2.x; tq[2] = tql[2] - (F)a2.y;
      }
      if constexpr (SPL) {
        if (spl) {
          // (cluster layout: every thread reads it, the last rank's idle ones too, as all of them join the carry's barrier)
          const int need = (CLUSTER || active) ? sh_need[r] : 0;
          double s_k = 0.0;                                          // np.cumsum(system.lengths)[j]
          if constexpr (CLUSTER) {
            // l_0 + ... + l_{NT c - 1}, added left to right, is an exact intermediate of the sequential sum: warp 0 adds
            // the earlier ranks' length words (DSMEM, written before the last barrier and rewritten only after the next
            // substep's first) into that carry, and every thread of the rank continues it over its own rank's words.
            // Each lane loads one word of 32 and every lane adds the 32 in order, so the chain is the reference's.
            __shared__ double sh_carry;
            if (need && c_rank > 0) {
              if (tid < 32) {
                double cs = 0.0;
                for (int c = 0; c < c_rank; c++) {
                  const D *w = cluster_smem(rec, c) + 15;
                  for (int b = 0; b < NT; b += 32) {
                    const double l = w[LEAN_REC * (b + tid)];
#pragma unroll
                    for (int k = 0; k < 32; k++) cs += __shfl_sync(0xffffffffu, l, k);
                  }
                }
                if (tid == 0) sh_carry = cs;
              }
              __syncthreads();
              s_k = sh_carry;
            }
          }
          const int jl = CLUSTER ? tid : j;   // this element's index among the words this CTA holds
          if (need && elem_ok) {
            for (int i = 0; i <= jl; i++) s_k += rec[LEAN_REC * (tid - jl + i) + 15];
            const int m = min(max((int)floor(s_k * A.spline_inv_dx), 0), sP);
            const double t = s_k - (double)m / A.spline_inv_dx;
            for (int d = 0; d < 3; d++) {
              if (!(need >> d & 1)) continue;
              const double *ch = sp + d * sCH, *tb = A.spline_tab + (size_t)m * sP * 4;
              double val = 0.0;
              for (int i = 0; i < sP; i++)
                val += ch[sP + i] * (tb[4 * i] + t * (tb[4 * i + 1] + t * (tb[4 * i + 2] + t * tb[4 * i + 3])));
              val *= A.spline_scale;
              sp[3 * sCH + d * n + j] = val;
              smag[d] = val;
            }
          }
#pragma unroll
          for (int i = 0; i < 3; i++) tq[i] += smag[i];
        }
      }
      D fj[3] = {D(0), D(0), D(0)}, tj[3] = {D(0), D(0), D(0)};   // assemblies: joint force on node 0 / couple on element 0
      if constexpr (MULTI) {
        if (active && first && has_head) {
          const D *o = sj + LEAN_JREC * tid;
#pragma unroll
          for (int i = 0; i < 3; i++) { fj[i] = -o[i]; tj[i] = o[6 + i]; }
        }
        if (!A.contact_before_forcing) {   // the joint is registered before the contact: the friction balance sees its loads
#pragma unroll
          for (int i = 0; i < 3; i++) { fint[i] += fj[i]; tq[i] += tj[i]; }
        }
      }
      D ct[3] = {D(0), D(0), D(0)};      // fold layout: the tip node's half of the plane's load on the last element
      if constexpr (CONTACT) {
        // forcing registered before the contact: the static-friction torque balance sees the muscle couple
        if (mus && !A.contact_before_forcing) {
#pragma unroll
          for (int i = 0; i < 3; i++) tq[i] += mtq[i];
        }
        if (A.contact_on) {
          // RodPlaneContactWithAnisotropicFriction (elastica/_contact_functions.py, SURVEY A.5), per element j between
          // nodes j and j+1, in the frame whose z axis is the plane normal.  Stage 1: normal response + kinetic friction
          // from the nodal forces accumulated so far; stage 2: static friction from the forces INCLUDING stage 1 of both
          // neighbours (nodal forces mix adjacent elements), hence two more exchanges: stage-1 in-plane loads through the
          // spare words 16..17 of the state records, the final loads through the (by then fully read) stress records.
          const bool end0 = (j == 0), end1 = (j + 1 == n);
          // element load = a0 f_j + a1 f_{j+1} (half of each node's force, an end node's in full); the mass weights of
          // the element velocity: end nodes carry half a mass
          const D a0 = end0 ? D(1.0) : D(0.5), a1 = end1 ? D(1.0) : D(0.5);
          const D w0 = (end0 == end1) ? D(0.5) : end0 ? D(1.0 / 3.0) : D(2.0 / 3.0), w1 = D(1.0) - w0;
          D etf[3], evel[3], t[3];
          {
            const double2 *qs = reinterpret_cast<const double2 *>(sn + SNR * t_next);
            const double2 s01 = qs[0];
            const D s2n = sn[SNR * t_next + 2];
            const double2 *qr = reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next);
            const double2 r1 = qr[1], r2 = qr[2];
            const D sN[3] = {s01.x, s01.y, s2n}, vN[3] = {r1.y, r2.x, r2.y};
#pragma unroll
            for (int i = 0; i < 3; i++) {
              const D f1 = sN[i] - sfl[i];                       // internal force on node j+1 (node j's is fint)
              // external loads so far: gravity (a0 hm0 + a1 hm1 = 1 for every element: one whole nodal weight)
              const D gi = A.contact_before_forcing ? D(0) : (D)Z.gm[i];
              etf[i] = fma(a1, f1, fma(a0, fint[i], gi));
              evel[i] = fma(w1, vN[i], w0 * v[i]);
              t[i] = dx[i] * ilg;
            }
          }
          const D rad2 = Z.vol_over_pi * ilg, inv_rad = rsqrt_nr(rad2), rad = rad2 * inv_rad;   // sqrt(V / (pi l))
          const D fn = etf[2], vn = evel[2];
          // sign tests and clamps of non-negative quantities run on the integer pipe (high words / bit patterns), not DSETP
          const D gap = (fma(D(0.5), dx[2], x[2]) - Z.plane_z0) - rad, pen = (__double2hiint(gap) < 0) ? gap : D(0);   // min(gap, 0)
          const bool nocontact = !elem_ok || (gap > Z.surface_tol);
          const D fn_neg = (__double2hiint(fn) < 0) ? -fn : D(0);        // max(-fn, 0): the plane only pushes
          // no contact: zero response, and every friction term below is bounded by or proportional to it
          const D resp_mag = nocontact ? D(0) : fn_neg;
          D c1[3];
          c1[2] = nocontact ? D(0) : fma(-Z.contact_nu, vn, fma(-Z.contact_k, pen, fn_neg));
          // axial direction = the tangent's projection on the plane, normalised with the reference's guard
          // 1 / (|tp| + 1e-14) (to first order in 1e-14 / |tp|); rolling direction = axial x normal
          const D tp2 = fma(t[1], t[1], t[0] * t[0]);
          const D rtp = rsqrt_nr(tp2 + D(1e-300));   // (a rod standing on end: tp = 0, axial direction 0)
          const D inv_tp = fma(D(-1e-14) * rtp, rtp, rtp);
          const D ax0 = t[0] * inv_tp, ax1 = t[1] * inv_tp, rl0 = ax1, rl1 = -ax0;
          // find_slipping_elements on a = |v| (|axial| = |rolling| = 1 - 1e-14 / |tp|: taken as 1):
          // a <= tol: 1;  a > tol: |1 - min(1, a / tol - 1)|  =  clamp(2 - a / tol, 0, 1) in both cases
          auto slip_fn = [&](D a) {
            const D u = fma(-a, Z.inv_slip_tol, D(2.0));
            const int hu = __double2hiint(u);
            return (hu < 0) ? D(0) : (hu >= 0x3ff00000) ? D(1) : u;
          };
          // min(a, b) for a, b >= 0: doubles of one sign order like their bit patterns
          auto min_pos = [](D a, D b) { return (__double_as_longlong(a) < __double_as_longlong(b)) ? a : b; };
          // sign(a) with sign(0) = +1: every use below multiplies a factor that vanishes with a
          auto sgn1 = [](D a) { return __hiloint2double((__double2hiint(a) & 0x80000000) | 0x3ff00000, 0); };
          const D vax = fma(evel[1], ax1, evel[0] * ax0);
          const D kmu = (__double2hiint(vax) < 0) ? (D)Z.kin_mu[1] : (D)Z.kin_mu[0];
          const D slipa = slip_fn(fabs(vax));
          // velocity of the contact point relative to the axis: Q^T (w x Q arm) = (Q^T w) x arm, arm = -rad z, i.e.
          // (-rad W_y, rad W_x, 0) with W = Q^T w the angular velocity in the plane's frame
          const D W0 = fma(Q[6], w[2], fma(Q[3], w[1], Q[0] * w[0])), W1 = fma(Q[7], w[2], fma(Q[4], w[1], Q[1] * w[0]));
          const D rv0 = -(rad * W1), rv1 = rad * W0;
          const D smag = fma(evel[1] + rv1, rl1, (evel[0] + rv0) * rl0);
          const D slipr = slip_fn(fabs(smag));
          const D ut0 = fma(smag, rl0, vax * ax0), ut1 = fma(smag, rl1, vax * ax1);
          const D ug0 = ut0 + D(1e-14), ug1 = ut1 + D(1e-14);
          const D iun = rsqrt_nr(fma(ug1, ug1, fma(ug0, ug0, D(1e-28))));
          // u . axial = vax |axial|^2, u . rolling = smag |rolling|^2, and |axial|^2 = |rolling|^2 = 1 - 2e-14 / |tp|: taken as 1
          const D uax = vax * iun, url = smag * iun;
          const D ka = -((D(1) - slipa) * kmu * resp_mag * uax);
          const D kr = -((D(1) - slipr) * Z.kin_mu[2] * resp_mag * url);
          D fr0 = kr * rl0, fr1 = kr * rl1;
          c1[0] = fma(ka, ax0, fr0); c1[1] = fma(ka, ax1, fr1);
          // couple of the rolling friction: Q (arm x F) = Q (rad F_y, -rad F_x, 0); kept in the plane's frame until the end
          D cr0 = rad * fr1, cr1 = -(rad * fr0);
          *reinterpret_cast<double2 *>(rec + LEAN_REC * tid + 16) = make_double2(c1[0], c1[1]);
          if constexpr (CLUSTER) {   // the stage-1 neighbours across the rank boundary: rec halos NT and -1, words 16-17
            double2 *h = nullptr;
            if (tid == 0 && c_rank > 0) h = cluster_smem(reinterpret_cast<double2 *>(rec + LEAN_REC * NT + 16), c_rank - 1);
            if (tid == NT - 1 && c_rank + 1 < c_size) h = cluster_smem(reinterpret_cast<double2 *>(rec - LEAN_REC + 16), c_rank + 1);
            if (h) *h = make_double2(c1[0], c1[1]);
          }
          rod_sync();
          // stage 2: static friction (in-plane components only)
          D e2[2];
          {
            // stage-1 response on nodes j, j+1: (left + own) / 2, (own + right) / 2, weighted a0, a1 like the loads above
            // (the tip thread's own stage-1 load is zero: no select for the last element's right neighbour)
            const double2 cl = *reinterpret_cast<const double2 *>(rec + LEAN_REC * t_prev + 16);
            const double2 cr = *reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next + 16);
            const D b0 = D(0.5) * a0, b1 = D(0.5) * a1, bm = b0 + b1;
            e2[0] = fma(b1, cr.x, fma(b0, cl.x, fma(bm, c1[0], etf[0])));
            e2[1] = fma(b1, cr.y, fma(b0, cl.y, fma(bm, c1[1], etf[1])));
          }
          const D fax = fma(e2[1], ax1, e2[0] * ax0);
          const D smu = (__double2hiint(fax) < 0) ? (D)Z.stat_mu[1] : (D)Z.stat_mu[0];
          const D sa = -(min_pos(fabs(fax), slipa * smu * resp_mag) * sgn1(fax));
          // in-plane components of the couples so far, Q^T (tq + Q cr) = Q^T tq + cr
          const D tt0 = fma(Q[6], tq[2], fma(Q[3], tq[1], fma(Q[0], tq[0], cr0))), tt1 = fma(Q[7], tq[2], fma(Q[4], tq[1], fma(Q[1], tq[0], cr1)));
          const D noslip = -((rad * fma(e2[1], rl1, e2[0] * rl0) - D(2) * fma(tt1, ax1, tt0 * ax0)) * (D(1.0 / 3.0) * inv_rad));
          const D sr_ = min_pos(fabs(noslip), slipr * Z.stat_mu[2] * resp_mag) * sgn1(noslip);
          fr0 = sr_ * rl0; fr1 = sr_ * rl1;
          const D p0 = c1[0] + fma(sa, ax0, fr0), p1 = c1[1] + fma(sa, ax1, fr1);
          *reinterpret_cast<double2 *>(sn + SNR * tid) = make_double2(p0, p1);
          sn[SNR * tid + 2] = c1[2];
          if (CLUSTER && tid == NT - 1 && c_rank + 1 < c_size) {   // element j - 1 of the next rank's thread 0: sn halo -1
            D *h = cluster_smem(reinterpret_cast<D *>(sn - SNR), c_rank + 1);
            *reinterpret_cast<double2 *>(h) = make_double2(p0, p1);
            h[2] = c1[2];
          }
          cr0 = fma(rad, fr1, cr0); cr1 = fma(-rad, fr0, cr1);   // both stages' rolling couples
#pragma unroll
          for (int i = 0; i < 3; i++) tq[i] = fma(Q[3 * i + 1], cr1, fma(Q[3 * i], cr0, tq[i]));
          rod_sync();
          {   // node j collects half of the plane's load on elements j-1 and j
            const double2 l01 = *reinterpret_cast<const double2 *>(sn + SNR * t_prev);
            const D l2v = sn[SNR * t_prev + 2];
            fint[0] += D(0.5) * (p0 + l01.x); fint[1] += D(0.5) * (p1 + l01.y); fint[2] += D(0.5) * (c1[2] + l2v);
            if (FOLD) { ct[0] = D(0.5) * p0; ct[1] = D(0.5) * p1; ct[2] = D(0.5) * c1[2]; }
          }
        }
        if (mus && A.contact_before_forcing) {
#pragma unroll
          for (int i = 0; i < 3; i++) tq[i] += mtq[i];
        }
      }
      if constexpr (MULTI) {
        if (A.contact_before_forcing) {
#pragma unroll
          for (int i = 0; i < 3; i++) { fint[i] += fj[i]; tq[i] += tj[i]; }
        }
      }
      if (MULTI && is_head) {
        // rigid head: a = F/m, alpha = J^-1 ((J w) x w + T)  (SURVEY D.1); loads = the joints' reactions, summed in
        // connection order; no gravity, no damper (octopus/build.py:141-152); then the rate part of
        // BodyBoundaryCondition: v_z = 0, w_x = w_y = 0
        if (hd) {
          D Fh[3] = {D(0), D(0), D(0)}, Th[3] = {D(0), D(0), D(0)};
          for (int a = 0; a < n_rod; a++) {
            const D *o = sj + LEAN_JREC * (r * G + a * tpr);
#pragma unroll
            for (int i = 0; i < 3; i++) { Fh[i] += o[i]; Th[i] += o[3 + i]; }
          }
          const D Jw[3] = {A.head_J[0] * w[0], A.head_J[1] * w[1], A.head_J[2] * w[2]};
          D lt[3];
          cross3(Jw, w, lt);
#pragma unroll
          for (int i = 0; i < 3; i++) {
            v[i] = fma(Fh[i], (D)A.head_dt_inv_mass, v[i]);
            w[i] = fma(c_dt, A.head_Jinv[i] * (lt[i] + Th[i]), w[i]);
          }
          v[2] = D(0); w[0] = D(0); w[1] = D(0);
        }
      } else {
        if (FOLD && is_last) {   // tip node (half a nodal mass): internal force -s_{n-1}, its share of the plane's load, gravity, damper
          const D dtim_tip = (D)A.dt_inv_mass * c_cv * D(2);
#pragma unroll
          for (int i = 0; i < 3; i++) vt[i] = fma(ct[i] - (D)sfl[i], dtim_tip, fma(vt[i], c_cv, (D)A.gdt_cv[i]));
        }
        // v <- c_v (v + dt f/m + dt g): the translational damper folded into the update (FP64 accumulation)
        v[0] = fma((D)fint[0], dtim_cv, fma(v[0], c_cv, base0));
        v[1] = fma((D)fint[1], dtim_cv, fma(v[1], c_cv, MIXED ? A.k_gdt_cv[1] : (D)A.gdt_cv[1]));
        v[2] = fma((D)fint[2], dtim_cv, fma(v[2], c_cv, MIXED ? A.k_gdt_cv[2] : (D)A.gdt_cv[2]));
        {
          const F g = elem_ok ? e * A.dt_Jinv0 : F(0), g2 = g * F(0.5);   // dt e / J ; J3 = 2 J1 for a circular section
          w[0] = fma((D)g, (D)tq[0], w[0]) * (D)cw0;
          w[1] = fma((D)g, (D)tq[1], w[1]) * (D)cw0;
          w[2] = fma((D)g2, (D)tq[2], w[2]) * (D)cw2;
        }
        // rate constraints (zeroing BCs commute with the multiplicative damper)
        auto constrain_rates = [&]() {
          v[0] = pin_fixed ? D(0) : v[0]; v[1] = z12 ? D(0) : v[1]; v[2] = z12 ? D(0) : v[2];
          w[0] = z12 ? D(0) : w[0]; w[1] = pin_fixed ? D(0) : w[1]; w[2] = z12 ? D(0) : w[2];
          if (LAPL && moving) {
            // [constrain, dampen] order: the analytical damper (already applied above) rescales the commanded velocity too
            const D sc = A.damp_first ? D(1) : c_cv;
            v[0] = sh_base[r][2] * sc; v[1] = sh_base[r][3] * sc; v[2] = D(0);
            w[0] = D(0); w[1] = D(0); w[2] = D(0);
          }
        };
        if constexpr (LAPL) {
          // LaplaceDissipationFilter of order 7 (elastica/dissipation.py:nb_filter_rate, SURVEY A.4): seven passes of
          // f <- (-f[k+1] - f[k-1] + 2 f[k]) / 4 on interior nodes / elements with the ends held at 0 (pass 0 sees the
          // unfiltered ends), then rate -= f.  After pass 0 the field g vanishes at both ends, and six more passes of a
          // symmetric stencil with zero ends are ONE 13-tap convolution of g's odd extension about the ends,
          //   f7[k] = sum_m c_m g[k+m],  c_m = (-1)^m C(12, 6+m) / 4096,  g[-k] = -g[k], g[last+k] = -g[last-k]:
          // two exchanges and barriers instead of seven.  The odd extension is materialised by the threads next to
          // the ends, which also write their (negated) g into ghost records beyond the rod; every thread then reads
          // its twelve neighbours at fixed offsets.  Nodes reflect about node n, elements about element n-1, so the
          // two halves of a right-hand ghost record come from different threads.
          auto laplace = [&]() {
            if (A.laplace_order != 7) return;    // (the host only selects this model for order 7 or none)
            const bool node_in = active && j > 0 && j < n, elem_in = active && j > 0 && j < n - 1;
            double2 *own = reinterpret_cast<double2 *>(rec + LEAN_REC * tid);
            own[0] = make_double2(v[0], v[1]); own[1] = make_double2(v[2], w[0]); own[2] = make_double2(w[1], w[2]);
            if constexpr (CLUSTER) {   // the neighbours of pass 0 across the rank boundary: halos NT and -1
              double2 *h = nullptr;
              if (tid == 0 && c_rank > 0) h = cluster_smem(reinterpret_cast<double2 *>(rec + LEAN_REC * NT), c_rank - 1);
              if (tid == NT - 1 && c_rank + 1 < c_size) h = cluster_smem(reinterpret_cast<double2 *>(rec - LEAN_REC), c_rank + 1);
              if (h) { h[0] = make_double2(v[0], v[1]); h[1] = make_double2(v[2], w[0]); h[2] = make_double2(w[1], w[2]); }
            }
            rod_sync();
            D g[6];
            {
              // end nodes / elements (and idle threads) take themselves as both neighbours: (-f - f + 2 f) / 4 = 0 exactly
              const double2 *ql = reinterpret_cast<const double2 *>(rec + LEAN_REC * (node_in ? tid - 1 : tid));
              const double2 *qr = reinterpret_cast<const double2 *>(rec + LEAN_REC * (node_in ? tid + 1 : tid));
              const double2 l0 = ql[0], l1 = ql[1], l2 = ql[2], r0 = qr[0], r1 = qr[1], r2 = qr[2];
              const D lv[6] = {l0.x, l0.y, l1.x, elem_in ? l1.y : w[0], elem_in ? l2.x : w[1], elem_in ? l2.y : w[2]};
              const D rv[6] = {r0.x, r0.y, r1.x, elem_in ? r1.y : w[0], elem_in ? r2.x : w[1], elem_in ? r2.y : w[2]};
              const D mv[6] = {v[0], v[1], v[2], w[0], w[1], w[2]};
#pragma unroll
              for (int c = 0; c < 6; c++) g[c] = ((-rv[c] - lv[c]) + D(2) * mv[c]) * D(0.25);
            }
            D *slot = gb + 6 * (CLUSTER ? 8 + tid : r * (tpr + 16) + 8 + j);
            // put_g(k, store): `store` writes into the record of rod index k.  Cluster layout: into that of every rank whose
            // taps read index k, i.e. whose window [NT c - 6, NT c + NT + 6) holds it — its owner, the previous rank for
            // the first six indices of a rank, the next one for the last six; the ghosts beyond both ends alike.  A
            // thread stores its own index and ghosts at most 13 indices away, so only its own rank and the two next to
            // it can hold them.
            auto put_g = [&](int k, auto &&store) {
              if constexpr (!CLUSTER) {
                store(slot + 6 * (k - j));
              } else {
                static_assert(NT > 13 + 6, "a rank's window reaches into its neighbours only");
#pragma unroll
                for (int d = -1; d <= 1; d++) {
                  const int t = c_rank + d, loc = k - NT * t + 8;
                  if (t < 0 || t >= c_size || loc < 2 || loc >= NT + 14) continue;
                  if (d == 0) store(gb + 6 * loc);
                  else store(cluster_smem(gb + 6 * loc, t));
                }
              }
            };
            if (!CLUSTER || in_cta) {   // (cluster layout: the last rank's idle threads hold indices past the ghosts)
              put_g(j, [&](D *p) {
                double2 *o = reinterpret_cast<double2 *>(p);
                if (j < n) { o[0] = make_double2(g[0], g[1]); o[1] = make_double2(g[2], g[3]); o[2] = make_double2(g[4], g[5]); }
                else { o[0] = make_double2(g[0], g[1]); p[2] = g[2]; }   // tip node: its record's element half is element n-2's ghost
              });
              if (j >= 1 && j <= 6) {              // left ghosts: both fields reflect about index 0
                put_g(-j, [&](D *p) {
                  double2 *gl = reinterpret_cast<double2 *>(p);
                  gl[0] = make_double2(-g[0], -g[1]); gl[1] = make_double2(-g[2], -g[3]); gl[2] = make_double2(-g[4], -g[5]);
                });
              }
              if (j >= n - 6 && j <= n - 1) {      // right ghosts of the node field: about node n
                put_g(2 * n - j, [&](D *gr) { gr[0] = -g[0]; gr[1] = -g[1]; gr[2] = -g[2]; });
              }
              if (j >= n - 7 && j <= n - 2) {      // right ghosts of the element field: about element n - 1
                put_g(2 * (n - 1) - j, [&](D *gr) { gr[3] = -g[3]; gr[4] = -g[4]; gr[5] = -g[5]; });
              }
            }
            rod_sync();
            D acc[6] = {v[0], v[1], v[2], w[0], w[1], w[2]};
            constexpr double cm[7] = {924.0 / 4096.0, -792.0 / 4096.0, 495.0 / 4096.0, -220.0 / 4096.0, 66.0 / 4096.0, -12.0 / 4096.0, 1.0 / 4096.0};
#pragma unroll
            for (int c = 0; c < 6; c++) acc[c] = fma(D(-cm[0]), g[c], acc[c]);
            // one third of a record at a time (two components, twelve independent 128-bit loads in flight, four
            // accumulator registers) rather than tap by tap: at the 128-register cap the compiler otherwise issues
            // the loads two at a time, each pair followed at once by its consumers
#pragma unroll
            for (int part = 0; part < 3; part++) {
              double2 lv[6], rv[6];
#pragma unroll
              for (int m = 1; m <= 6; m++) {
                lv[m - 1] = reinterpret_cast<const double2 *>(slot - 6 * m)[part];
                rv[m - 1] = reinterpret_cast<const double2 *>(slot + 6 * m)[part];
              }
#pragma unroll
              for (int m = 1; m <= 6; m++) {
                acc[2 * part] = fma(D(-cm[m]), lv[m - 1].x + rv[m - 1].x, acc[2 * part]);
                acc[2 * part + 1] = fma(D(-cm[m]), lv[m - 1].y + rv[m - 1].y, acc[2 * part + 1]);
              }
            }
            // ends: g and its odd extension give exactly 0 there; the selects only keep idle lanes and the tip's pseudo-element clean
            if (node_in) { v[0] = acc[0]; v[1] = acc[1]; v[2] = acc[2]; }
            if (elem_in) { w[0] = acc[3]; w[1] = acc[4]; w[2] = acc[5]; }
          };
          if (!A.damp_first) constrain_rates();     // (one copy of the filter, two of the small constraint)
          laplace();
          if (A.damp_first) constrain_rates();
        } else {
          constrain_rates();
        }
      }

      kinematic(last ? c_half_dt : c_dt, last ? D(1e-14) : D(2e-14));
      head_constrain_values();
    };
    // planar model: the substep above with the out-of-plane terms left out (see PLANAR).  Records {x0 x1 | v0 v1 | Q0 Q1 |
    // Q6 Q7} and {s0 s1 | N1}.  The pseudo-element of the tip / idle threads lies along x here instead of z (same
    // length; its stress is discarded either way), so the tip's stale observables are rebuilt in the last substep.
    // NAMED: the per-rod barriers (rod_barriers), chosen once outside the loop; every warp takes part in its first
    // rod's barrier, and a warp that holds the end of one rod and the start of the next in the next rod's as well.
    // FIRST: the segment's first substep, the only one that runs the trace check.  It is a copy of its own so that the
    // check's reads of the pre-launch state (st, bc, stride, j) are not live across the loop: at the 80-register cap
    // they made ptxas re-derive the thread's indices and addresses in every substep.
    auto substep_planar = [&](auto last_tag, auto named_tag, auto first_tag) {
      constexpr bool last = decltype(last_tag)::value, NAMED = decltype(named_tag)::value;
      constexpr bool FIRST = decltype(first_tag)::value;
      auto sync = [&]() {
        if constexpr (NAMED) {
          asm volatile("bar.sync %0, %1;" ::"r"(bar_id0), "r"(bar_cnt0) : "memory");
          asm volatile("{ .reg .pred p; setp.ne.s32 p, %2, 0; @p bar.sync %0, %1; }" ::"r"(bar_id1), "r"(bar_cnt1),
                       "r"((int)bar_two) : "memory");
        } else {
          __syncthreads();
        }
      };
      {
        double2 *o = reinterpret_cast<double2 *>(rec + LEAN_REC * tid);
        o[0] = make_double2(x[0], x[1]); o[1] = make_double2(v[0], v[1]);
        o[2] = make_double2(Q[0], Q[1]); o[3] = make_double2(Q[6], Q[7]);
      }
      sync();
      D dx0, dx1, dv0, dv1, dn0, dn1, Qn0, Qn1, Qn6, Qn7;
      {
        const double2 *qq = reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next);
        const double2 a0 = qq[0], a1 = qq[1], a2 = qq[2], a3 = qq[3];
        const double2 b0 = *reinterpret_cast<const double2 *>(rec + LEAN_REC * t_next2);
        Qn0 = a2.x; Qn1 = a2.y; Qn6 = a3.x; Qn7 = a3.y;
        dx0 = a0.x - x[0]; dx1 = a0.y - x[1]; dv0 = a1.x - v[0]; dv1 = a1.y - v[1];
        dn0 = b0.x - a0.x; dn1 = b0.y - a0.y;
      }
      if (!elem_ok) dx0 = (D)A.rest_len;
      if (!vor_ok) dn0 = (D)A.rest_len;
      const D l2 = fma(dx1, dx1, dx0 * dx0), l2n = fma(dn1, dn1, dn0 * dn0);
      const D il = rsqrt_nr(l2), iln = rsqrt_nr(l2n);
      const D lg = fma(l2, il, D(1e-14));
      const D ilg = fma(D(-1e-14) * il, il, il);
      const D lgn = fma(l2n, iln, D(1e-14));
      const D e = lg * irg;
      const D em1 = fma(lg, irg, D(-1.0));
      const D inv_e = A.rest_len * ilg;
      const D inv_e_s = elem_ok ? inv_e : D(0);
      const D ede = fma(dx1, dv1, dx0 * dv0) * (ilg * ilg);
      const D Qdx0 = fma(Q[1], dx1, Q[0] * dx0), Qdx2 = fma(Q[7], dx1, Q[6] * dx0);   // Q dx = (Qdx0, 0, Qdx2)
      const D s3 = fma(Qdx2, irg, D(-1.0));
      const D n0 = A.S_over_l[0] * Qdx0;
      const D n2 = fma((D)A.S[2], Qdx2 * irg, -(D)A.S[2]);
      const D sf0 = fma(Q[6], n2, Q[0] * n0) * inv_e_s, sf1 = fma(Q[7], n2, Q[1] * n0) * inv_e_s;
      // curvature: axial(Qn Q^T - Q Qn^T) = (0, vec1, 0)
      const D vec1 = fma(-Qn7, Q[1], fma(-Qn6, Q[0], fma(Qn1, Q[7], Qn0 * Q[6])));
      D w2 = vec1 * vec1;
      if (!vor_ok) w2 = D(0);
      bool bend_out = out_of_range(w2, A.lim_bend_hi, A.limf_bend);
      if constexpr (FIRST) {
        if (vor_ok) {
          // d2 = (0, 0, d2z) of this element and the next: invariant under in-plane rotations, read from the
          // pre-launch state (the clamp's from its anchor)
          const D z_own = pin_fixed ? (D)bc[8] : (D)st[(F_DIR + 5) * stride + j], z_next = (D)st[(F_DIR + 5) * stride + j + 1];
          const D tr = fma(Qn7, Q[7], fma(Qn6, Q[6], fma(z_next, z_own, fma(Qn1, Q[1], Qn0 * Q[0]))));
          bend_out = bend_out || !(tr > D(2.0));
        }
      }
      if (bend_out) dom_bad |= 2;
      D fs;
      {
        D c[10];
#pragma unroll
        for (int k = 0; k < 10; k++) c[k] = (D)A.bendw[k];   // (F = D here)
        const D z = w2 * w2;
        D pe = fma(c[8], z, c[6]), po = fma(c[9], z, c[7]);
        pe = fma(pe, z, c[4]); po = fma(po, z, c[5]);
        pe = fma(pe, z, c[2]); po = fma(po, z, c[3]);
        pe = fma(pe, z, c[0]); po = fma(po, z, c[1]);
        fs = fma(po, w2, pe);
      }
      const D kp1 = vec1 * fs;
      const D tau1 = A.B[0] * kp1;
      const D eps_v = (lgn + lg) * A.half_inv_rest_vor;
      D ie3 = rcp_nr(eps_v * eps_v * eps_v);
      if (!vor_ok) ie3 = D(0);
      const D m1 = tau1 * ie3;
      const D cc = fma(-(D)A.S_over_l[0], Qdx2, n2);
      const D je = ede * A.J[0];
      const D h1 = fma(-Qdx0, cc, je * w[1]);
      const D tql1 = fma(h1, inv_e, m1);
      {
        double2 *o = reinterpret_cast<double2 *>(sn + SNR * tid);
        o[0] = make_double2(sf0, sf1);
        sn[SNR * tid + 2] = -m1;
      }
      D cw0;
      {
        if (out_of_range(em1, A.lim_em1_hi, A.limf_em1) && elem_ok) dom_bad |= 4;
        cw0 = fma(fma((D)A.cwp[0][2], em1, (D)A.cwp[0][1]), em1, (D)A.cwp[0][0]);
      }
      if (last && active) {
        // stale observables, as the plain model computes them.  Its tip thread holds Q = I and the edge (0, 0, l0); its
        // last element forms the curvature against that I: axial(I Q^T - Q) = (d2z - Q7, Q6, Q1).
        D tg[3] = {dx0 * ilg, dx1 * ilg, D(0)}, kp[3] = {D(0), kp1, D(0)};
        D sg0 = Qdx0 * irg, sg2 = s3;
        if (j == n) {
          tg[0] = D(0); tg[2] = dx0 * ilg; kp[1] = D(0); sg0 = D(0); sg2 = fma(Qdx0, irg, D(-1.0));
        } else if (j == n - 1) {
          const D z_own = pin_fixed ? (D)bc[8] : (D)st[(F_DIR + 5) * stride + j];
          kp[0] = (z_own - Q[7]) * fs; kp[2] = Q[1] * fs;
        }
#pragma unroll
        for (int i = 0; i < 3; i++) {
          st[(F_TAN + i) * stride + j] = (ST)tg[i];
          st[(F_KAPPA + i) * stride + j] = (ST)kp[i];
        }
        st[F_SIGMA * stride + j] = (ST)sg0;
        st[(F_SIGMA + 1) * stride + j] = ST(0);
        st[(F_SIGMA + 2) * stride + j] = (ST)sg2;
        st[F_DIL * stride + j] = (ST)e;
      }
      sync();
      D f0, f1, tq1;
      {
        const double2 l = *reinterpret_cast<const double2 *>(sn + SNR * t_prev);
        f0 = sf0 - l.x; f1 = sf1 - l.y; tq1 = tql1 + sn[SNR * t_prev + 2];
      }
      v[0] = fma(f0, dtim_cv, fma(v[0], c_cv, base0));
      v[1] = fma(f1, dtim_cv, fma(v[1], c_cv, (D)A.gdt_cv[1]));
      {
        const D g = elem_ok ? e * A.dt_Jinv0 : D(0);
        w[1] = fma(g, tq1, w[1]) * cw0;
      }
      v[0] = pin_fixed ? D(0) : v[0]; v[1] = z12 ? D(0) : v[1]; w[1] = pin_fixed ? D(0) : w[1];
      kinematic(last ? c_half_dt : c_dt, last ? D(1e-14) : D(2e-14));
    };
    // the item's last substep ends with a half kinematic step and exports the stale observables: its own copy of the
    // body, so that the loop carries neither the selects nor the branch
    const int s_loop_end = (s_end == K) ? K - 1 : s_end;
    if constexpr (PLANAR) {
      using yes = std::true_type;
      using no = std::false_type;
      auto run = [&](auto named_tag) {
        if (s_begin < s_loop_end) {
          substep_planar(no{}, named_tag, yes{});
#pragma unroll 1
          for (int s = s_begin + 1; s < s_loop_end; s++) substep_planar(no{}, named_tag, no{});
          if (s_end == K) substep_planar(yes{}, named_tag, no{});
        } else if (s_end == K && s_begin < K) {   // a segment of the item's last substep alone
          substep_planar(yes{}, named_tag, yes{});
        }
      };
      if (rod_barriers) run(std::true_type{});
      else run(std::false_type{});
    } else {
#pragma unroll 1
      for (int s = s_begin; s < s_loop_end; s++) substep(std::false_type{}, s);
      if (s_end == K && s_begin < K) substep(std::true_type{}, K - 1);
    }

    __syncthreads();   // all reads of the exchange buffers are done
    if (s_end < K) {
      // ---- hand the item over to the next slot -------------------------------------------------------------------
      if (FASTONLY) {
        if (tid < 256) sh_dom[tid] = 0;
        __syncthreads();
        if (live && dom_bad) atomicOr(&sh_dom[r], dom_bad);
        __syncthreads();
        if (active && lead && sh_dom[r] != 0 && atomicExch(&A.redo[env], 1) == 0 && A.redo_count) count_redo(sh_dom[r]);
      }
      D *sc = A.sk_scratch + (size_t)p * SCR * NT;
      if constexpr (PLANAR) {
        sc[tid] = x[0]; sc[NT + tid] = x[1]; sc[2 * NT + tid] = v[0]; sc[3 * NT + tid] = v[1]; sc[4 * NT + tid] = w[1];
        sc[5 * NT + tid] = Q[0]; sc[6 * NT + tid] = Q[1]; sc[7 * NT + tid] = Q[6]; sc[8 * NT + tid] = Q[7];
      } else {
#pragma unroll
        for (int c = 0; c < 3; c++) { sc[c * NT + tid] = x[c]; sc[(3 + c) * NT + tid] = v[c]; sc[(15 + c) * NT + tid] = w[c]; }
#pragma unroll
        for (int c = 0; c < 9; c++) sc[(6 + c) * NT + tid] = Q[c];
      }
      if (CONTACT) { sc[18 * NT + tid] = mus_S; sc[19 * NT + tid] = mus_C; sc[20 * NT + tid] = mus_t; }
      if (FOLD) {
#pragma unroll
        for (int c = 0; c < 3; c++) { sc[(21 + c) * NT + tid] = xt[c]; sc[(24 + c) * NT + tid] = vt[c]; }
      }
      __threadfence();
      __syncthreads();
      if (tid == 0) { *(volatile int *)(A.sk_flag + p) = 1; }
      continue;
    }

    // ---- write back, NaN guard, model outputs --------------------------------------------------------------------
    bool redo = false;
    if (FASTONLY && CLUSTER) {
      // the cluster's OR in rank 0's sh_dom[0], which every CTA reads back: a flagged env leaves no part of its rod
      // written back.  (redo[env] is read ahead of the barrier after which the lead may set it.)
      const bool flagged = live && A.redo[env] != 0;
      if (live && dom_bad) atomicOr(cluster_smem(&sh_dom[0], 0), dom_bad);
      cluster_sync();
      const int dom = *cluster_smem(&sh_dom[0], 0);
      redo = live && (dom != 0 || flagged);
      if (redo && lead && atomicExch(&A.redo[env], 1) == 0 && A.redo_count) count_redo(dom);
    } else if (FASTONLY) {    // env-level OR of the range flags; a flagged env keeps its pre-launch state in global memory
      if (tid < 256) sh_dom[tid] = 0;
      __syncthreads();
      if (live && dom_bad) atomicOr(&sh_dom[r], dom_bad);
      __syncthreads();
      // (a part of this item run by the previous slot may have flagged the env already)
      redo = live && (sh_dom[r] != 0 || A.redo[env] != 0);
      if (redo && lead && atomicExch(&A.redo[env], 1) == 0 && A.redo_count) count_redo(sh_dom[r]);
    }
    constexpr int RS = NT + 2;
    if (MIXED) {       // edge vectors of the final FP64 positions: the strain state the next launch starts from
#pragma unroll
      for (int c = 0; c < 3; c++) rec[c * RS + tid] = x[c];
      __syncthreads();
      if (active && !redo) {
#pragma unroll
        for (int c = 0; c < 3; c++) st[(F_EDGE + c) * stride + j] = elem_ok ? (ST)(rec[c * RS + tid + 1] - x[c]) : ST(0);
      }
      __syncthreads();
    }
    bool bad = false;
    if (MULTI && hd && !redo) {
#pragma unroll
      for (int c = 0; c < 3; c++) { hd[c] = (ST)x[c]; hd[3 + c] = (ST)v[c]; hd[15 + c] = (ST)w[c]; }
#pragma unroll
      for (int c = 0; c < 9; c++) hd[6 + c] = (ST)Q[c];
      float *o = A.obs + (size_t)env * A.obs_dim;
      for (int c = 0; c < 3; c++) { o[c] = (float)x[c]; o[3 + c] = (float)v[c]; }
    }
    if (PLANAR && active && !redo) {   // the out-of-plane fields keep their zeros (the clamp's d2z is its anchor's)
      for (int c = 0; c < 2; c++) {
        st[(F_POS + c) * stride + j] = (ST)x[c];
        st[(F_VEL + c) * stride + j] = (ST)v[c];
        bad = bad || (x[c] != x[c]) || (v[c] != v[c]);
      }
      if (j < n) {
        st[(F_OMEGA + 1) * stride + j] = (ST)w[1];
        st[F_DIR * stride + j] = (ST)Q[0]; st[(F_DIR + 1) * stride + j] = (ST)Q[1];
        st[(F_DIR + 6) * stride + j] = (ST)Q[6]; st[(F_DIR + 7) * stride + j] = (ST)Q[7];
        if (pin_fixed) st[(F_DIR + 5) * stride + j] = bc[8];
      }
    } else if (active && !redo) {
      if (CONTACT) { to_lab(x); to_lab(v); rows_to_lab(Q); }   // (final: nothing below reads them in the internal frame)
#pragma unroll
      for (int c = 0; c < 3; c++) {
        st[(F_POS + c) * stride + j] = (ST)x[c];
        st[(F_VEL + c) * stride + j] = (ST)v[c];
        bad = bad || (x[c] != x[c]) || (v[c] != v[c]);
      }
      if (j < n) {
#pragma unroll
        for (int c = 0; c < 3; c++) st[(F_OMEGA + c) * stride + j] = (ST)w[c];
#pragma unroll
        for (int c = 0; c < 9; c++) st[(F_DIR + c) * stride + j] = (ST)Q[c];
      }
      if (FOLD && is_last) {
        if (CONTACT) { to_lab(xt); to_lab(vt); }
#pragma unroll
        for (int c = 0; c < 3; c++) {
          st[(F_POS + c) * stride + n] = (ST)xt[c];
          st[(F_VEL + c) * stride + n] = (ST)vt[c];
          bad = bad || (xt[c] != xt[c]) || (vt[c] != vt[c]);
        }
        if (A.model == MODEL_ROD) {
          float *o = A.obs + (size_t)env * A.obs_dim;
          for (int c = 0; c < 3; c++) { o[c] = (float)xt[c]; o[3 + c] = (float)vt[c]; }
        }
      }
    }
    // per-rod NaN flag and tangents for the observation (rod r occupies tids r*tpr .. r*tpr+n)
    D *sh_t = rec;   // 3 rows of NT + 2
    if constexpr (CLUSTER) {
      // the cluster's OR in rank 0's sh_flag[0]; the barrier also orders every rank's tangents (written to the state
      // block in the last substep) before the lead's reads of them
      if (active && bad) atomicOr(cluster_smem(&sh_flag[0], 0), 1);
      cluster_sync();
    } else {
      if (tid < 256) sh_flag[tid] = 0;
      if (active && (A.model == MODEL_SOFT_PENDULUM || (LAPL && A.model == MODEL_SOFT_PENDULUM_3D))) {
#pragma unroll
        for (int i = 0; i < 3; i++) sh_t[i * RS + tid] = (j < n) ? (D)st[(F_TAN + i) * stride + j] : D(0);
      }
      __syncthreads();
      if (active && bad) atomicOr(&sh_flag[r], 1);
      __syncthreads();
    }
    if (!FASTONLY && A.redo_filter && active && lead) A.redo[env] = 0;
    if (active && lead && !redo) {
      const bool invalid = sh_flag[r] != 0;
      if (mus) A.muscle[(size_t)env * A.muscle_dim] = mus_t;
      const D *tan = sh_t + tid;
      int tan_stride = RS;
      if constexpr (CLUSTER) { tan = st + F_TAN * stride; tan_stride = stride; }   // (the state block: every rank's)
      if (A.model == MODEL_SOFT_PENDULUM) {
        soft_pendulum_outputs<D>(tan, tan_stride, n, x[0], v[0],
                                 A.action_dim > 0 ? A.action[(size_t)env * A.action_dim] : 0.0f, invalid,
                                 A.obs + (size_t)env * A.obs_dim, A.reward + env, A.terminated + env);
      } else if (LAPL && A.model == MODEL_SOFT_PENDULUM_3D) {
        const double x0[3] = {x[0], x[1], x[2]}, v0[3] = {v[0], v[1], v[2]};
        ST *aux = A.aux + (size_t)env * AUX_DIM;
        if (moving && K > 0) {   // the base controller's state, deferred from the prologue
          aux[0] = (ST)sh_base[r][0]; aux[1] = (ST)sh_base[r][1]; aux[3] = (ST)sh_base[r][2]; aux[4] = (ST)sh_base[r][3]; aux[5] = ST(0);
        }
        const float act_f0 = A.action_dim > 0 ? A.action[(size_t)env * A.action_dim] : 0.0f;
        const float act_f1 = A.action_dim > 1 ? A.action[(size_t)env * A.action_dim + 1] : 0.0f;
        soft_pendulum_3d_outputs<D>(tan, tan_stride, n, x0, v0, act_f0, act_f1, (double)aux[0], (double)aux[1],
                                    invalid, A.obs + (size_t)env * A.obs_dim, A.reward + env, A.terminated + env,
                                    reinterpret_cast<D *>(aux + 6));
      } else {
        A.reward[env] = 0.0;
        A.terminated[env] = invalid ? 1 : 0;
      }
    }
    if (active && A.model == MODEL_ROD && j == n && !MULTI && !redo) {
      float *o = A.obs + (size_t)env * A.obs_dim;
      for (int c = 0; c < 3; c++) { o[c] = (float)x[c]; o[3 + c] = (float)v[c]; }
    }
    __syncthreads();   // the staging rows are free again before the next item publishes
  }
  if constexpr (CLUSTER) cluster_sync();   // no CTA leaves while another may still access its shared memory
}

}  // namespace sr
