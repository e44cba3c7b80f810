// copy_kernels.cuh — the env copy of sr_copy_envs (not on the hot path); included by softrod_api.cu only.
#pragma once
#include <stdint.h>

namespace sr {

constexpr int COPY_MAX_BUFS = 16;   // per-env buffers of a handle (softrod_api.cu: env_buffers) fit with room to spare
constexpr int COPY_NT = 256;

// One per-env buffer of a copy: row e of a buffer is the `bytes` bytes at base + e * bytes, moved in units of `vec`
// bytes (4, 8 or 16; base and bytes are multiples of it).  src == nullptr writes zeros.
struct CopyBuf {
  const char *src;
  char *dst;
  unsigned long long bytes;
  int vec;
};

// How pair i moves its rows: straight from row src_idx[i] to row dst_idx[i], or through row i of a staging buffer
// (GATHER: src_idx[i] -> i, then SCATTER: i -> dst_idx[i]).
enum CopyMode : int { COPY_DIRECT = 0, COPY_GATHER = 1, COPY_SCATTER = 2 };

struct CopyTable {
  CopyBuf buf[COPY_MAX_BUFS];
  int n_buf;
  int n_src, n_dst;   // env counts of the source / destination handle: a pair with an index outside them is skipped
  int mode;           // CopyMode
};

template <typename V> __device__ __forceinline__ void copy_row(const CopyBuf &b, long long s, long long d, long long u0, long long du) {
  const long long units = (long long)(b.bytes / sizeof(V));
  V *dst = reinterpret_cast<V *>(b.dst + d * b.bytes);
  if (b.src) {
    const V *src = reinterpret_cast<const V *>(b.src + s * b.bytes);
    for (long long u = u0; u < units; u += du) dst[u] = src[u];
  } else {
    const V z{};
    for (long long u = u0; u < units; u += du) dst[u] = z;
  }
}

// Pair i (blockIdx.y, striding by gridDim.y) copies every buffer's row; the blocks of blockIdx.x stride over each row.
// Both launches of a staged copy skip the same pairs: the check reads both index arrays whatever the mode.
__global__ void __launch_bounds__(COPY_NT) copy_envs_kernel(const __grid_constant__ CopyTable t, const int32_t *dst_idx,
                                                           const int32_t *src_idx, int n) {
  const long long u0 = (long long)blockIdx.x * COPY_NT + threadIdx.x, du = (long long)gridDim.x * COPY_NT;
  for (int i = blockIdx.y; i < n; i += gridDim.y) {
    const int s = src_idx[i], d = dst_idx[i];
    if (s < 0 || s >= t.n_src || d < 0 || d >= t.n_dst) continue;
    const long long rs = t.mode == COPY_SCATTER ? i : s, rd = t.mode == COPY_GATHER ? i : d;
    for (int k = 0; k < t.n_buf; k++) {
      const CopyBuf &b = t.buf[k];
      if (b.vec == 16) copy_row<int4>(b, rs, rd, u0, du);
      else if (b.vec == 8) copy_row<int2>(b, rs, rd, u0, du);
      else copy_row<int>(b, rs, rd, u0, du);
    }
  }
}

}  // namespace sr
