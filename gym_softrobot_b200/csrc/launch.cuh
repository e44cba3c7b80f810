// launch.cuh — host-callable launchers of the kernel instantiations.  Every (type, CTA size, feature set) is
// compiled in its own translation unit (inst_*.cu, selected by -D macros from build.py) so that the library
// builds in parallel; softrod_api.cu sees declarations only.
#pragma once
#include <cuda_runtime.h>
#include "rod_kernels.cuh"

namespace sr {

// generic CTA-packed kernel (rod_kernel_packed.cuh); opts the dynamic shared memory in on the current device
template <typename T, int NT, int MINB, bool LAPLACE, bool MOVING, bool CONTACT, bool MULTI, bool TORQUE, bool FASTONLY, bool VARY = false>
cudaError_t launch_packed_kernel(const RodArgs<T> &A, int rods_per_cta, int grid, cudaStream_t s);

// tapered multi-rod assembly with the COOMM muscle layers (two longitudinal + transverse, per-element activations)
template <int NT> cudaError_t launch_packed_lmus_kernel(const RodArgs<double> &A, int rods_per_cta, int grid, cudaStream_t s);

// An instantiation of the lean kernel (rod_kernel_lean.cuh) is one model in one layout.  The model is which substep runs:
enum class LeanModel {
  PLAIN,      // one rod under gravity, damping and the base point force (SoftPendulum-v0, plain rods)
  PLANE,      // one rod on the frictional plane with per-env rest curvature (OctoArmSingle-v0)
  MUSCLE,     // PLANE + the travelling-wave muscle torque (ContinuumSnake-v0)
  ASSEMBLY,   // arms + rigid head + joints on the plane (OctoFlat-v0)
  FILTER,     // the Laplace dissipation filter + moving base (SoftPendulum3D-v0)
  SPLINE,     // spline muscle torques (SoftArmTracking-v0); safe kernel only, in the CTA and cluster layouts
  PLANAR,     // PLAIN for a rod that stays in the lab x-y plane; fast-only kernel only
};
// The layout is where a rod's nodes live:
enum class LeanLayout {
  CTA,        // rods of n elements packed back to back into a CTA, n + 1 threads each
  FOLD,       // one rod of n elements per CTA of n threads, the tip node folded into the last one
  CLUSTER,    // one rod per thread-block cluster of LEAN_CLUSTER_NT-thread CTAs
};

constexpr int LEAN_SCR_CONTACT = 21;   // rows of a stream-K slot's hand-over scratch (plane models: 18 + the travelling wave's sin, cos, time)
constexpr int LEAN_SCR_FOLD = 27;      // fold layout: + position and velocity of the tip node
// lean kernel (T = storage type: double = FP64, float = mixed precision) in the CTA and fold layouts; grid / split
// schedule in A.sk_*
template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT>
cudaError_t launch_lean_kernel(const RodArgs<T> &A, int grid, cudaStream_t s);
// resident CTAs per SM of that instantiation on the current device (sizes the stream-K grid)
template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT> int lean_ctas_per_sm();
// cluster layout (FP64, 512 threads): one rod per thread-block cluster of `cluster` CTAs, grid = n_env x cluster CTAs
constexpr int LEAN_CLUSTER_NT = 512;
template <bool FASTONLY, LeanModel MODEL> cudaError_t launch_lean_cluster_kernel(const RodArgs<double> &A, int cluster, cudaStream_t s);
// clusters of that shape that both kernels of MODEL's pair (the spline model: its safe kernel) can keep resident at once
// on the current device (0: none)
template <LeanModel MODEL> int lean_cluster_max_active(int cluster);

// warp-per-rod kernel, faithful (libm, reference operation order) math: the parity build
template <typename T, int EPL> cudaError_t launch_warp_faithful(const RodArgs<T> &A, int grid, cudaStream_t s);

}  // namespace sr
