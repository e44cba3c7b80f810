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

constexpr int LEAN_SCR_CONTACT = 21;   // rows of a stream-K slot's hand-over scratch (contact variant: 18 + the travelling wave's sin, cos, time)
constexpr int LEAN_SCR_FOLD = 27;      // folded-tip variants: + position and velocity of the tip node
// lean kernel (rod_kernel_lean.cuh; T = storage type: double = FP64, float = mixed precision); grid / split schedule in A.sk_*
template <typename T, int NT, int MINB, bool FASTONLY, int CONTACT = 0> cudaError_t launch_lean_kernel(const RodArgs<T> &A, int grid, cudaStream_t s);
// resident CTAs per SM of that instantiation on the current device (sizes the stream-K grid)
template <typename T, int NT, int MINB, bool FASTONLY, int CONTACT = 0> int lean_ctas_per_sm();
// cluster variants 9-12 (FP64, 512 threads): one rod per thread-block cluster of `cluster` CTAs, grid = n_env x cluster CTAs
constexpr int LEAN_CLUSTER_NT = 512;
template <bool FASTONLY, int CVAR> cudaError_t launch_lean_cluster_kernel(const RodArgs<double> &A, int cluster, cudaStream_t s);
// clusters of that shape that both kernels of variant CVAR's pair can keep resident at once on the current device (0: none)
template <int CVAR> int lean_cluster_max_active(int cluster);

// warp-per-rod kernel, faithful (libm, reference operation order) math: the parity build
template <typename T, int EPL> cudaError_t launch_warp_faithful(const RodArgs<T> &A, int grid, cudaStream_t s);

}  // namespace sr
