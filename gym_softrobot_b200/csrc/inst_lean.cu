// inst_lean.cu — the lean kernel (rod_kernel_lean.cuh) for one storage type and CTA size:
//   -DSR_TU_T=double|float -DSR_TU_NT=<threads> -DSR_TU_MINB=<n> [-DSR_TU_CONTACT=1|2|3|4: contact variant without / with the muscle wave / for assemblies; 4: filter + moving base; 5: spline torques; 6 / 7: variants 0 / 1 with the tip node folded into the last thread; 8: variant 0 in the x-y plane, fast-only kernel only; 9 / 10 / 11 / 12: variant 0 / 4 / 1 / 2 on thread-block clusters, 512 threads only; FP64 only]
#include <atomic>
#include "launch.cuh"
#include "rod_kernel_lean.cuh"

namespace sr {

template <typename T, int NT, int MINB, bool FASTONLY, int CONTACT> static cudaError_t lean_opt_in() {
  // the opt-in above 48 KB is a per-device attribute of the function: one bit per device ordinal
  static std::atomic<unsigned long long> opted{0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ULL << (dev & 63);
  if (!(opted.load(std::memory_order_relaxed) & bit)) {
    e = cudaFuncSetAttribute(rod_lean_kernel<T, NT, MINB, FASTONLY, CONTACT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(lean_smem_words(NT, CONTACT) * sizeof(double)));
    if (e != cudaSuccess) return e;
    opted.fetch_or(bit, std::memory_order_relaxed);
  }
  return cudaSuccess;
}

template <typename T, int NT, int MINB, bool FASTONLY, int CONTACT> cudaError_t launch_lean_kernel(const RodArgs<T> &A, int grid, cudaStream_t s) {
  cudaError_t e = lean_opt_in<T, NT, MINB, FASTONLY, CONTACT>();
  if (e != cudaSuccess) return e;
  rod_lean_kernel<T, NT, MINB, FASTONLY, CONTACT><<<grid, NT, lean_smem_words(NT, CONTACT) * sizeof(double), s>>>(A);
  return cudaGetLastError();
}

template <typename T, int NT, int MINB, bool FASTONLY, int CONTACT> int lean_ctas_per_sm() {
  if (lean_opt_in<T, NT, MINB, FASTONLY, CONTACT>() != cudaSuccess) return 0;
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rod_lean_kernel<T, NT, MINB, FASTONLY, CONTACT>, NT,
                                                    lean_smem_words(NT, CONTACT) * sizeof(double)) != cudaSuccess) return 0;
  return nb;
}

#ifndef SR_TU_CONTACT
#define SR_TU_CONTACT 0
#endif
#if SR_TU_CONTACT >= 9 && SR_TU_CONTACT <= 12
static_assert(SR_TU_NT == LEAN_CLUSTER_NT, "the cluster variants are built for 512-thread CTAs");
constexpr int CV = SR_TU_CONTACT;

static cudaLaunchConfig_t cluster_config(int grid, int cluster, cudaStream_t s, cudaLaunchAttribute *attr) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(LEAN_CLUSTER_NT);
  cfg.dynamicSmemBytes = lean_smem_words(LEAN_CLUSTER_NT, CV) * sizeof(double);
  cfg.stream = s;
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = (unsigned)cluster; attr->val.clusterDim.y = 1; attr->val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cfg;
}

template <bool FASTONLY, int CVAR> cudaError_t launch_lean_cluster_kernel(const RodArgs<double> &A, int cluster, cudaStream_t s) {
  static_assert(CVAR == CV, "one cluster variant per translation unit");
  cudaError_t e = lean_opt_in<double, LEAN_CLUSTER_NT, 1, FASTONLY, CV>();
  if (e != cudaSuccess) return e;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = cluster_config(A.n_env * cluster, cluster, s, &attr);
  return cudaLaunchKernelEx(&cfg, rod_lean_kernel<double, LEAN_CLUSTER_NT, 1, FASTONLY, CV>, A);
}

template <bool FASTONLY> static int cluster_max_active(int cluster) {
  if (lean_opt_in<double, LEAN_CLUSTER_NT, 1, FASTONLY, CV>() != cudaSuccess) return 0;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = cluster_config(cluster, cluster, nullptr, &attr);
  int nc = 0;
  if (cudaOccupancyMaxActiveClusters(&nc, rod_lean_kernel<double, LEAN_CLUSTER_NT, 1, FASTONLY, CV>, &cfg) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return nc;
}

template <int CVAR> int lean_cluster_max_active(int cluster) {
  static_assert(CVAR == CV, "one cluster variant per translation unit");
  const int a = cluster_max_active<true>(cluster), b = cluster_max_active<false>(cluster);
  return a < b ? a : b;
}

template int lean_cluster_max_active<CV>(int);
template cudaError_t launch_lean_cluster_kernel<true, CV>(const RodArgs<double> &, int, cudaStream_t);
template cudaError_t launch_lean_cluster_kernel<false, CV>(const RodArgs<double> &, int, cudaStream_t);
#else
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, SR_TU_CONTACT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, SR_TU_CONTACT>();
#if SR_TU_CONTACT != 8   // (the planar variant's fallback is variant 0's safe kernel)
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, SR_TU_CONTACT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, SR_TU_CONTACT>();
#endif
#endif

}  // namespace sr
