// Shared device/host helpers of the phifem_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/phifem_b200.h"

namespace phifem {

void set_error(const char* fmt, ...);

#define PHIFEM_CHECK_ARG(cond, msg)                         \
  do {                                                      \
    if (!(cond)) {                                          \
      ::phifem::set_error("%s: %s", __func__, msg);         \
      return PHIFEM_ERR_ARGUMENT;                           \
    }                                                       \
  } while (0)

#define PHIFEM_CHECK_LAUNCH()                                                         \
  do {                                                                                \
    cudaError_t err__ = cudaGetLastError();                                           \
    if (err__ != cudaSuccess) {                                                       \
      ::phifem::set_error("%s: CUDA error: %s", __func__, cudaGetErrorString(err__)); \
      return PHIFEM_ERR_CUDA;                                                         \
    }                                                                                 \
  } while (0)

// Reference-cell traits (dolfinx conventions, SURVEY.md Appendix C): simplex local facet i is opposite
// local vertex i, its vertices listed in ascending local order; quadrilateral and hexahedron facets in tensor order.
template <int CT> struct CellTraits;
template <> struct CellTraits<PHIFEM_TRIANGLE> {
  static constexpr int nv = 3, nf = 3, nvf = 2, gdim = 2;
  __host__ __device__ static constexpr int fv(int f, int k) {
    constexpr int t[3][2] = {{1, 2}, {0, 2}, {0, 1}};
    return t[f][k];
  }
};
template <> struct CellTraits<PHIFEM_QUADRILATERAL> {
  static constexpr int nv = 4, nf = 4, nvf = 2, gdim = 2;
  __host__ __device__ static constexpr int fv(int f, int k) {
    constexpr int t[4][2] = {{0, 1}, {0, 2}, {1, 3}, {2, 3}};
    return t[f][k];
  }
};
template <> struct CellTraits<PHIFEM_TETRAHEDRON> {
  static constexpr int nv = 4, nf = 4, nvf = 3, gdim = 3;
  __host__ __device__ static constexpr int fv(int f, int k) {
    constexpr int t[4][3] = {{1, 2, 3}, {0, 2, 3}, {0, 1, 3}, {0, 1, 2}};
    return t[f][k];
  }
};
// vertices in tensor order (v = i + 2 j + 4 k at (i, j, k)), faces (a, b, c, d) in tensor order: a face point (s, t)
// sits at v_a + s (v_b - v_a) + t (v_c - v_a)
template <> struct CellTraits<PHIFEM_HEXAHEDRON> {
  static constexpr int nv = 8, nf = 6, nvf = 4, gdim = 3;
  __host__ __device__ static constexpr int fv(int f, int k) {
    constexpr int t[6][4] = {{0, 1, 2, 3}, {0, 1, 4, 5}, {0, 2, 4, 6}, {1, 3, 5, 7}, {2, 3, 6, 7}, {4, 5, 6, 7}};
    return t[f][k];
  }
};

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// ---- TMA 1-D bulk copies global -> shared with mbarrier completion (sm_90+; SASS UBLKCP / SYNCS) -------------------
// The streaming kernels stage their contiguous index arrays (cells, f2c) through shared memory with these: one elected
// thread posts whole tiles several stages ahead, so the bytes in flight per SM no longer depend on how many warps
// are resident or on which phase of their loop they are in.
namespace tma {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// makes the freshly initialised barriers visible to the async proxy (the TMA unit)
__device__ __forceinline__ void fence_init() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// dst, src and bytes multiples of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t ok = 0;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
  } while (!ok);
}
}  // namespace tma

// Persistent grid-stride kernels: exactly one resident wave (SMs x occupancy), never more CTAs than tiles.
template <typename K>
inline int persistent_grid(K kernel, int block, int64_t n_tiles) {
  int per_sm = 0, dev = 0, sms = kNumSMs;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, 0) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  int64_t cap = (int64_t)sms * per_sm;
  if (n_tiles < 1) n_tiles = 1;
  return (int)(n_tiles < cap ? n_tiles : cap);
}

inline int grid_for(int64_t n, int block, int ctas_per_sm) {
  int64_t need = (n + block - 1) / block;
  int64_t cap = (int64_t)kNumSMs * ctas_per_sm;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

}  // namespace phifem
