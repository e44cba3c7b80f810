// inst_lean.cu — the lean kernel (rod_kernel_lean.cuh) for one storage type, CTA size, model and layout:
//   -DSR_TU_T=double|float -DSR_TU_NT=<threads> -DSR_TU_MINB=<n> -DSR_TU_MODEL=<LeanModel> -DSR_TU_LAYOUT=<LeanLayout>
// (the models and layouts by their enumerator names in launch.cuh; every model but PLAIN in the CTA layout is FP64 only,
// the cluster layout is built for LEAN_CLUSTER_NT threads only)
#include <atomic>
#include "launch.cuh"
#include "rod_kernel_lean.cuh"

namespace sr {

template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT> static cudaError_t lean_opt_in() {
  // the opt-in above 48 KB is a per-device attribute of the function: one bit per device ordinal
  static std::atomic<unsigned long long> opted{0};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ULL << (dev & 63);
  if (!(opted.load(std::memory_order_relaxed) & bit)) {
    e = cudaFuncSetAttribute(rod_lean_kernel<T, NT, MINB, FASTONLY, MODEL, LAYOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(lean_smem_words(NT, MODEL, LAYOUT) * sizeof(double)));
    if (e != cudaSuccess) return e;
    opted.fetch_or(bit, std::memory_order_relaxed);
  }
  return cudaSuccess;
}

template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT>
cudaError_t launch_lean_kernel(const RodArgs<T> &A, int grid, cudaStream_t s) {
  cudaError_t e = lean_opt_in<T, NT, MINB, FASTONLY, MODEL, LAYOUT>();
  if (e != cudaSuccess) return e;
  rod_lean_kernel<T, NT, MINB, FASTONLY, MODEL, LAYOUT><<<grid, NT, lean_smem_words(NT, MODEL, LAYOUT) * sizeof(double), s>>>(A);
  return cudaGetLastError();
}

template <typename T, int NT, int MINB, bool FASTONLY, LeanModel MODEL, LeanLayout LAYOUT> int lean_ctas_per_sm() {
  if (lean_opt_in<T, NT, MINB, FASTONLY, MODEL, LAYOUT>() != cudaSuccess) return 0;
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, rod_lean_kernel<T, NT, MINB, FASTONLY, MODEL, LAYOUT>, NT,
                                                    lean_smem_words(NT, MODEL, LAYOUT) * sizeof(double)) != cudaSuccess) return 0;
  return nb;
}

constexpr LeanModel TU_MODEL = LeanModel::SR_TU_MODEL;
constexpr LeanLayout TU_LAYOUT = LeanLayout::SR_TU_LAYOUT;

// The preprocessor cannot compare the names SR_TU_MODEL and SR_TU_LAYOUT stand for, so its tests paste a name onto
// SR_IS_: SR_IS_CLUSTER and SR_IS_PLANAR are 1, and any other SR_IS_<name> is undefined, which #if reads as 0.
// SR_SAFE_ONLY(<model>) is 1 for the models whose cluster layout is built as the safe kernel alone (SPLINE).
#define SR_IS_PASTE(name) SR_IS_##name
#define SR_IS(name) SR_IS_PASTE(name)
#define SR_IS_CLUSTER 1
#define SR_IS_PLANAR 1
#define SR_SAFE_ONLY_PASTE(name) SR_SAFE_ONLY_##name
#define SR_SAFE_ONLY(name) SR_SAFE_ONLY_PASTE(name)
#define SR_SAFE_ONLY_SPLINE 1

#if SR_IS(SR_TU_LAYOUT)   // the cluster layout
static_assert(TU_LAYOUT == LeanLayout::CLUSTER && SR_TU_NT == LEAN_CLUSTER_NT, "the cluster layout is built for 512-thread CTAs");

static cudaLaunchConfig_t cluster_config(int grid, int cluster, cudaStream_t s, cudaLaunchAttribute *attr) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(LEAN_CLUSTER_NT);
  cfg.dynamicSmemBytes = lean_smem_words(LEAN_CLUSTER_NT, TU_MODEL, TU_LAYOUT) * sizeof(double);
  cfg.stream = s;
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = (unsigned)cluster; attr->val.clusterDim.y = 1; attr->val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cfg;
}

template <bool FASTONLY, LeanModel MODEL> cudaError_t launch_lean_cluster_kernel(const RodArgs<double> &A, int cluster, cudaStream_t s) {
  static_assert(MODEL == TU_MODEL, "one cluster model per translation unit");
  cudaError_t e = lean_opt_in<double, LEAN_CLUSTER_NT, 1, FASTONLY, MODEL, TU_LAYOUT>();
  if (e != cudaSuccess) return e;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = cluster_config(A.n_env * cluster, cluster, s, &attr);
  return cudaLaunchKernelEx(&cfg, rod_lean_kernel<double, LEAN_CLUSTER_NT, 1, FASTONLY, MODEL, TU_LAYOUT>, A);
}

template <bool FASTONLY> static int cluster_max_active(int cluster) {
  if (lean_opt_in<double, LEAN_CLUSTER_NT, 1, FASTONLY, TU_MODEL, TU_LAYOUT>() != cudaSuccess) return 0;
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = cluster_config(cluster, cluster, nullptr, &attr);
  int nc = 0;
  if (cudaOccupancyMaxActiveClusters(&nc, rod_lean_kernel<double, LEAN_CLUSTER_NT, 1, FASTONLY, TU_MODEL, TU_LAYOUT>, &cfg) != cudaSuccess) {
    (void)cudaGetLastError();
    return 0;
  }
  return nc;
}

template <LeanModel MODEL> int lean_cluster_max_active(int cluster) {
  static_assert(MODEL == TU_MODEL, "one cluster model per translation unit");
#if SR_SAFE_ONLY(SR_TU_MODEL)
  return cluster_max_active<false>(cluster);
#else
  const int a = cluster_max_active<true>(cluster), b = cluster_max_active<false>(cluster);
  return a < b ? a : b;
#endif
}

template int lean_cluster_max_active<TU_MODEL>(int);
#if !SR_SAFE_ONLY(SR_TU_MODEL)   // (the spline model updates its forcing's cache inside the launch: no fast-only kernel)
template cudaError_t launch_lean_cluster_kernel<true, TU_MODEL>(const RodArgs<double> &, int, cudaStream_t);
#endif
template cudaError_t launch_lean_cluster_kernel<false, TU_MODEL>(const RodArgs<double> &, int, cudaStream_t);
#else
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, TU_MODEL, TU_LAYOUT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, TU_MODEL, TU_LAYOUT>();
#if !SR_IS(SR_TU_MODEL)   // (the planar model's fallback is the plain model's safe kernel)
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, TU_MODEL, TU_LAYOUT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, TU_MODEL, TU_LAYOUT>();
#endif
#endif

}  // namespace sr
