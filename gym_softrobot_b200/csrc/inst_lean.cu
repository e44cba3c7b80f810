// inst_lean.cu — the lean kernel (rod_kernel_lean.cuh) for one storage type and CTA size:
//   -DSR_TU_T=double|float -DSR_TU_NT=<threads> -DSR_TU_MINB=<n> [-DSR_TU_CONTACT=1|2|3|4: contact variant without / with the muscle wave / for assemblies; 4: filter + moving base; 5: spline torques; 6 / 7: variants 0 / 1 with the tip node folded into the last thread; 8: variant 0 in the x-y plane, fast-only kernel only; FP64 only]
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
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, SR_TU_CONTACT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, true, SR_TU_CONTACT>();
#if SR_TU_CONTACT != 8   // (the planar variant's fallback is variant 0's safe kernel)
template cudaError_t launch_lean_kernel<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, SR_TU_CONTACT>(const RodArgs<SR_TU_T> &, int, cudaStream_t);
template int lean_ctas_per_sm<SR_TU_T, SR_TU_NT, SR_TU_MINB, false, SR_TU_CONTACT>();
#endif

}  // namespace sr
