// K1: level-set cut-cell classification on sm_100a.
//
// Replaces reference src/phifem/mesh_scripts.py `_compute_detection_vector` (:95-134),
// `_tag_cells` (:284-390), `_tag_facets` (:393-558) and the candidate search of
// `_compute_integration_entities` (:137-192).
//
// Bit-exactness: the detection ratio is compared with ==1.0 / ==-1.0 in the reference
// (:343-347), so this file restates the FFCx arithmetic literally -- sequential sums of
// fl(phi_q * |detJ|), no FMA contraction (the file is compiled with -fmad=false), IEEE
// division and sqrt.  Everything here is HBM/L2-bound integer + fp64 streaming work: one
// thread per cell / facet, coalesced index loads, gathers that hit L2, warp-ballot counters.
#include <type_traits>

#include <stdlib.h>

#include "common.cuh"

namespace phifem {
namespace {

constexpr int kMaxDofs = 20;  // P3 tetrahedron
constexpr int kBlock = 256;

// Bounds of the cell-local arrays (vertices, facets, level-set dofs) per cell type.  Simplices and quadrilaterals keep
// the sizes their kernels were tuned with; only hexahedra (8 vertices, 6 facets, 27 dofs of Q2) get larger ones.
template <int CT> struct LocalBounds {
  static constexpr int nv = CellTraits<CT>::nv > 4 ? CellTraits<CT>::nv : 4;
  static constexpr int nf = CellTraits<CT>::nf > 4 ? CellTraits<CT>::nf : 4;
  static constexpr int nd = CT == PHIFEM_HEXAHEDRON ? 27 : kMaxDofs;
};

__device__ __forceinline__ double seq_dot(const double* __restrict__ w, int wstride,
                                          const double* v, int vstride, int n) {
  // sum_k w[k] v[k], left to right, exact-zero weights skipped, unit weights not multiplied
  double acc = 0.0;
  bool first = true;
  for (int k = 0; k < n; ++k) {
    const double wk = __ldg(w + k * wstride);
    if (wk == 0.0) continue;
    const double term = (wk == 1.0) ? v[k * vstride] : wk * v[k * vstride];
    acc = first ? term : acc + term;
    first = false;
  }
  return acc;
}

__device__ __forceinline__ int classify(double num, double den) {
  // mesh_scripts.py:124-128 then :343-347
  const double d = (den > 0.0) ? num / den : 0.5;
  if (d > -1.0 && d < 1.0) return 2;
  if (d == 1.0) return 3;
  if (d == -1.0) return 1;
  return 0;
}

__device__ __forceinline__ bool is_close_to_zero(double den) { return fabs(den) <= 1e-8; }

// sm_100 256-bit read-only load (LDG.E.256)
__device__ __forceinline__ void ldg256(const double* p, double& a, double& b, double& c, double& d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}

template <int CT>
__device__ __forceinline__ void load_cell(const phifem_mesh& m, int64_t c, int (&v)[LocalBounds<CT>::nv],
                                          double (&xc)[LocalBounds<CT>::nv][3]) {
  using T = CellTraits<CT>;
#pragma unroll
  for (int k = 0; k < T::nv; ++k) v[k] = __ldg(m.cells + c * T::nv + k);
#pragma unroll
  for (int k = 0; k < T::nv; ++k)
#pragma unroll
    for (int d = 0; d < T::gdim; ++d) xc[k][d] = __ldg(m.x + (int64_t)v[k] * T::gdim + d);
}

// |det J| of a simplex, same operation order as oracle/tags.py cell_scale
template <int CT>
__device__ __forceinline__ double simplex_detj(const double (&xc)[4][3]) {
  if (CT == PHIFEM_TRIANGLE) {
    const double j00 = xc[1][0] - xc[0][0], j01 = xc[2][0] - xc[0][0];
    const double j10 = xc[1][1] - xc[0][1], j11 = xc[2][1] - xc[0][1];
    return fabs(j00 * j11 - j01 * j10);
  } else {
    double a[3], b[3], c[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      a[d] = xc[1][d] - xc[0][d];
      b[d] = xc[2][d] - xc[0][d];
      c[d] = xc[3][d] - xc[0][d];
    }
    const double det = (a[0] * (b[1] * c[2] - c[1] * b[2]) - b[0] * (a[1] * c[2] - c[1] * a[2])) +
                       c[0] * (a[1] * b[2] - b[1] * a[2]);
    return fabs(det);
  }
}

// facet integral scale: edge length (2D) or |e1 x e2| (3D); oracle/tags.py facet_scale
template <int CT>
__device__ __forceinline__ double facet_scale(const double (&xc)[4][3], int lf) {
  using T = CellTraits<CT>;
  int a = 0, b = 0, c = 0;
#pragma unroll
  for (int f = 0; f < T::nf; ++f)
    if (f == lf) {
      a = T::fv(f, 0);
      b = T::fv(f, 1);
      c = T::nvf == 3 ? T::fv(f, T::nvf - 1) : 0;
    }
  if constexpr (T::nvf == 2) {
    const double d0 = xc[b][0] - xc[a][0], d1 = xc[b][1] - xc[a][1];
    return sqrt(d0 * d0 + d1 * d1);
  } else {
    double e1[3], e2[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      e1[d] = xc[b][d] - xc[a][d];
      e2[d] = xc[c][d] - xc[a][d];
    }
    const double cx = e1[1] * e2[2] - e1[2] * e2[1];
    const double cy = e1[2] * e2[0] - e1[0] * e2[2];
    const double cz = e1[0] * e2[1] - e1[1] * e2[0];
    return sqrt((cx * cx + cy * cy) + cz * cz);
  }
}

// ---- hexahedra: the trilinear map evaluated per point from the reference gradients g[8][3] of ls.coord_grad ----------
// Jacobian column d x / d X_ax, summed like oracle/tags_hex.py
__device__ __forceinline__ void hex_jcol(const double* g, const double (&xc)[8][3], int ax, double (&col)[3]) {
#pragma unroll
  for (int d = 0; d < 3; ++d) col[d] = seq_dot(g + ax, 3, &xc[0][d], 3, 8);
}

// |det J| at a point, the cofactor expansion of simplex_detj on the columns of J
__device__ __forceinline__ double hex_detj(const double* g, const double (&xc)[8][3]) {
  double a[3], b[3], c[3];
  hex_jcol(g, xc, 0, a);
  hex_jcol(g, xc, 1, b);
  hex_jcol(g, xc, 2, c);
  const double det = (a[0] * (b[1] * c[2] - c[1] * b[2]) - b[0] * (a[1] * c[2] - c[1] * a[2])) +
                     c[0] * (a[1] * b[2] - b[1] * a[2]);
  return fabs(det);
}

// |dx/ds x dx/dt| at a point of local face lf = (a, b, c, d): v_b - v_a and v_c - v_a are reference axes, so the two
// tangents are columns of J
__device__ __forceinline__ double hex_facet_scale(const double* g, const double (&xc)[8][3], int lf) {
  using T = CellTraits<PHIFEM_HEXAHEDRON>;
  int sa = 0, ta = 0;
#pragma unroll
  for (int f = 0; f < T::nf; ++f)
    if (f == lf) {
      const int db = T::fv(f, 1) - T::fv(f, 0), dc = T::fv(f, 2) - T::fv(f, 0);
      sa = db == 1 ? 0 : (db == 2 ? 1 : 2);
      ta = dc == 1 ? 0 : (dc == 2 ? 1 : 2);
    }
  double e1[3], e2[3];
  hex_jcol(g, xc, sa, e1);
  hex_jcol(g, xc, ta, e2);
  const double cx = e1[1] * e2[2] - e1[2] * e2[1];
  const double cy = e1[2] * e2[0] - e1[0] * e2[2];
  const double cz = e1[0] * e2[1] - e1[1] * e2[0];
  return sqrt((cx * cx + cy * cy) + cz * cz);
}

template <int NV>
__device__ __forceinline__ void load_coeffs(const phifem_mesh& m, const phifem_levelset& ls, int nvpc,
                                            int64_t c, const int (&v)[NV], double* cd) {
  const int nd = ls.n_dofs_per_cell;
  if (ls.dofmap == nullptr) {
    for (int i = 0; i < nvpc; ++i) cd[i] = __ldg(ls.coeffs + v[i]);
  } else {
    for (int i = 0; i < nd; ++i) cd[i] = __ldg(ls.coeffs + __ldg(ls.dofmap + c * nd + i));
  }
}

// ---- tag counters: per-thread registers -> warp redux -> shared -> one global atomic per block --------
struct BlockCounters {
  unsigned int* s;
  __device__ BlockCounters(unsigned int* smem, int n) : s(smem) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) s[i] = 0u;
    __syncthreads();
  }
  __device__ __forceinline__ void vote(bool pred, int slot) {
    const unsigned int b = __ballot_sync(0xffffffffu, pred);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(&s[slot], __popc(b));
  }
  __device__ __forceinline__ void add(unsigned int local, int slot) {  // all 32 lanes must call
    const unsigned int w = __reduce_add_sync(0xffffffffu, local);
    if ((threadIdx.x & 31) == 0 && w) atomicAdd(&s[slot], w);
  }
  __device__ void flush(int64_t* counters, int base, int n) {
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x)
      if (s[i]) atomicAdd(reinterpret_cast<unsigned long long*>(counters + base + i),
                          (unsigned long long)s[i]);
  }
};

// ---- K1a: P1 level set, detection degree 1, simplices: the headline kernel ------------------
// Per cell: 4 (3) vertex ids (coalesced 16 B / 12 B), 4 (3) fp64 gathers of phi (8 B x Nv, mostly
// L1/L2 hits), and -- only where the sign test cannot decide -- the vertex coordinates for |det J|.
// Uncut cells whose products phi*|detJ| can neither vanish, overflow nor land near the
// RuntimeWarning threshold are decided from the signs alone, which is bit-identical to the
// sequential sum (all terms share a sign => num == +-den exactly).
// HBM-latency bound: every thread keeps kUnroll independent cells in flight (index loads first, then
// all gathers), counters stay in registers until the end of the grid-stride loop.
constexpr int kTagCellsMinBlocks = 3;
constexpr int kUnroll = 4;

// exact path for cells the sign test cannot decide; scalars in / packed (tag | zden << 8) out so
// that the call does not force the caller's arrays into local memory
template <int CT>
__device__ __noinline__ int tag_cell_exact(const double* __restrict__ x, int v0, int v1, int v2, int v3,
                                           double p0, double p1, double p2, double p3) {
  using T = CellTraits<CT>;
  const int v[4] = {v0, v1, v2, v3};
  const double p[4] = {p0, p1, p2, p3};
  double xc[4][3];
#pragma unroll
  for (int k = 0; k < T::nv; ++k)
#pragma unroll
    for (int d = 0; d < T::gdim; ++d) xc[k][d] = __ldg(x + (int64_t)v[k] * T::gdim + d);
  const double s = simplex_detj<CT>(xc);
  double num = 0.0, den = 0.0;
#pragma unroll
  for (int k = 0; k < T::nv; ++k) {
    const double t = p[k] * s;
    num = num + t;
    den = den + fabs(t);
  }
  return classify(num, den) | ((int)is_close_to_zero(den) << 8);
}

// Level-set evaluation over the vertices (= P1 dofs), one coalesced pass: a class byte per vertex
//   bit 0: phi > 0   bit 1: phi < 0   bit 2: 1e-150 <= |phi| <= 1e150 (products cannot over/underflow)
//   bit 3: |phi| * detj_min > 2e-8 (one such vertex puts the cell's denominator clear of the
//          RuntimeWarning threshold of mesh_scripts.py:129, whatever the other vertices hold)
//   bit 4: 4 |phi| * detj_max < 0.5e-8 (all vertices such: the denominator is below the threshold)
// The cell kernel then gathers 1 byte per vertex instead of 8 (the byte array of 8.6 M vertices stays in
// L1/L2), and reads phi itself only for the few cells the bytes cannot decide.
__global__ void __launch_bounds__(kBlock) k_vertex_class(const double* __restrict__ phi, int64_t n,
                                                         double detj_min, double detj_max,
                                                         uint8_t* __restrict__ vclass) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
  for (int64_t base = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; base < n; base += stride) {
    unsigned int packed = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t i = base + k;
      const double p = i < n ? __ldg(phi + i) : 0.0;
      const double ap = fabs(p);
      unsigned int c = (p > 0.0 ? 1u : 0u) | (p < 0.0 ? 2u : 0u);
      c |= (ap >= 1e-150 && ap <= 1e150) ? 4u : 0u;
      c |= (ap * detj_min > 2e-8) ? 8u : 0u;
      c |= (4.0 * ap * detj_max < 0.5e-8) ? 16u : 0u;
      packed |= c << (8 * k);
    }
    if (base + 3 < n) {
      *reinterpret_cast<unsigned int*>(vclass + base) = packed;  // base is a multiple of 4
    } else {
      for (int k = 0; k < 4 && base + k < n; ++k) vclass[base + k] = (uint8_t)(packed >> (8 * k));
    }
  }
}

template <int CT>
__global__ void __launch_bounds__(kBlock, kTagCellsMinBlocks) k_tag_cells_p1(phifem_mesh m, const double* __restrict__ phi,
                                                            const uint8_t* __restrict__ vclass,
                                                            bool exact_zero_den,
                                                            int32_t* __restrict__ tags,
                                                            int8_t* __restrict__ tags8,
                                                            int64_t* counters) {
  using T = CellTraits<CT>;
  __shared__ unsigned int scnt[6];
  // Cells the class bytes cannot decide (the cut cells and a few more: ~1.5 % of config E) are not evaluated where
  // they are found -- one such lane makes its whole warp walk the exact path (coordinate gathers, |det J|, the
  // sequential sums), which was ~40 % of the kernel's instructions -- but parked in shared memory and evaluated
  // densely, one per thread, after the tile's barrier.  Two lists alternate between tiles; their fill counts only grow
  // (`done` = the count every thread saw at the previous use), so one barrier per tile suffices.
  __shared__ int s_pend[2][kBlock * kUnroll];
  __shared__ unsigned int s_np[2];
  if (threadIdx.x < 2) s_np[threadIdx.x] = 0u;
  BlockCounters cnt(scnt, 6);  // (its constructor synchronises the block)
  unsigned int local[6] = {0u, 0u, 0u, 0u, 0u, 0u};
  unsigned int done[2] = {0u, 0u};
  int par = 0;
  // kUnroll cells per thread, strided by the block size: every index load is one coalesced line per
  // warp (the consecutive-cells mapping with vector stores measured slower here: 0.32 vs 0.27 ms)
  const int64_t tile = (int64_t)blockDim.x * kUnroll;
  for (int64_t base = (int64_t)blockIdx.x * tile; base < m.n_cells; base += (int64_t)gridDim.x * tile) {
    int v[kUnroll][4];
    bool valid[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t c = base + (int64_t)u * blockDim.x + threadIdx.x;
      valid[u] = c < m.n_cells;
      const int64_t cc = valid[u] ? c : 0;
      if (T::nv == 4) {
        const int4 q = __ldg(reinterpret_cast<const int4*>(m.cells) + cc);
        v[u][0] = q.x; v[u][1] = q.y; v[u][2] = q.z; v[u][3] = q.w;
      } else {
#pragma unroll
        for (int k = 0; k < T::nv; ++k) v[u][k] = __ldg(m.cells + cc * T::nv + k);
      }
    }
    unsigned int all[kUnroll], any[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      all[u] = 0xffu;
      any[u] = 0u;
#pragma unroll
      for (int k = 0; k < T::nv; ++k) {
        const unsigned int c = __ldg(vclass + v[u][k]);
        all[u] &= c;
        any[u] |= c;
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      // same sign everywhere and no product can vanish or overflow: num == +-den bit-exactly, the tag
      // follows from the sign.  The isclose(den, 0) flag behind the RuntimeWarning (mesh_scripts.py:129)
      // is decided from the magnitude bits where they are conclusive; the rest is counted as ambiguous
      // (the host re-runs with exact_zero_den only if no cell settled the warning) or evaluated exactly.
      bool fast = (all[u] & 3u) != 0u && (all[u] & 4u) != 0u;
      int tag = (all[u] & 1u) ? 3 : 1;
      bool zden = false, ambiguous = false;
      if (fast && !(any[u] & 8u)) {
        if (all[u] & 16u) zden = true;
        else if (exact_zero_den) fast = false;
        else ambiguous = true;
      }
      if (!fast && valid[u]) {  // parked: position inside the tile
        const unsigned int i = atomicAdd(&s_np[par], 1u) - done[par];
        s_pend[par][i] = u * (int)blockDim.x + (int)threadIdx.x;
      } else if (valid[u]) {
        const int64_t c = base + (int64_t)u * blockDim.x + threadIdx.x;
        if (tags) tags[c] = tag;
        tags8[c] = (int8_t)tag;
        local[0] += tag == 1;
        local[1] += tag == 2;
        local[2] += tag == 3;
        local[3] += tag == 0;
        local[4] += zden;
        local[5] += ambiguous;
      }
    }
    __syncthreads();
    const unsigned int end = s_np[par];
    for (unsigned int i = done[par] + threadIdx.x; i < end; i += blockDim.x) {
      const int64_t c = base + s_pend[par][i - done[par]];
      int w[4] = {0, 0, 0, 0};
      double p[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int k = 0; k < T::nv; ++k) {
        w[k] = __ldg(m.cells + c * T::nv + k);
        p[k] = __ldg(phi + w[k]);
      }
      const int r = tag_cell_exact<CT>(m.x, w[0], w[1], w[2], w[3], p[0], p[1], p[2], p[3]);
      const int tag = r & 0xff;
      if (tags) tags[c] = tag;
      tags8[c] = (int8_t)tag;
      local[0] += tag == 1;
      local[1] += tag == 2;
      local[2] += tag == 3;
      local[3] += tag == 0;
      local[4] += (r >> 8) != 0;
    }
    done[par] = end;
    par ^= 1;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) cnt.add(local[i], i);
  cnt.flush(counters, PHIFEM_CNT_INTERIOR, 6);
}

// The same classifier with `cells` staged through shared memory by TMA bulk copies (the default).  A tile is
// kBlock * kUnroll cells (16 KB of tetrahedra, 12 KB of triangles); thread 0 keeps kCellStages tiles in flight per CTA, so
// the 0.8 GB index stream -- the only HBM traffic of the kernel that matters -- is requested as whole tiles several tiles
// ahead instead of by per-thread LDG.128s whose number in flight follows the resident warps' loop phase, and a warp no
// longer waits out a DRAM round trip before it can issue its class-byte gathers.  The cell -> thread mapping stays the
// strided one (slot u of thread t = cell t + 256 u of the tile: a gather instruction of a warp covers 32 consecutive
// cells, i.e. a handful of sectors of the class array); the tag bytes of a tile are collected in shared memory and leave
// as one coalesced 32-bit word per thread AFTER the next tile's barrier, when the exact path has filled in the parked
// cells (three 1 KB output buffers rotate so that one barrier per tile suffices).
constexpr int kCellStages = 2;
constexpr int kTagCellsStagedMinBlocks = 4;
constexpr int kCellTile = kBlock * kUnroll;
template <int CT> constexpr size_t staged_cells_smem() {
  return (size_t)kCellStages * kCellTile * CellTraits<CT>::nv * sizeof(int32_t);
}

template <int CT>
__global__ void __launch_bounds__(kBlock, kTagCellsStagedMinBlocks) k_tag_cells_p1_staged(
    phifem_mesh m, const double* __restrict__ phi, const uint8_t* __restrict__ vclass, bool exact_zero_den,
    int32_t* __restrict__ tags, int8_t* __restrict__ tags8, int64_t* counters) {
  using T = CellTraits<CT>;
  constexpr int NV = T::nv;
  extern __shared__ __align__(128) int32_t s_cells[];  // [kCellStages][kCellTile * NV]
  __shared__ alignas(8) uint64_t s_bar[kCellStages];
  __shared__ unsigned int scnt[6];
  __shared__ int s_pend[2][kCellTile];
  __shared__ unsigned int s_np[2];
  __shared__ alignas(16) unsigned int s_out[3][kCellTile / 4];
  if (threadIdx.x < 2) s_np[threadIdx.x] = 0u;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kCellStages; ++s) tma::mbar_init(&s_bar[s], 1);
    tma::fence_init();
  }
  BlockCounters cnt(scnt, 6);  // (its constructor synchronises the block)
  unsigned int local[6] = {0u, 0u, 0u, 0u, 0u, 0u};
  unsigned int done[2] = {0u, 0u};
  int par = 0, ob = 0;
  constexpr uint32_t kTileBytes = kCellTile * NV * 4;
  const int64_t n_full = m.n_cells / kCellTile;
  auto post = [&](int64_t t, int s) {
    tma::mbar_expect_tx(&s_bar[s], kTileBytes);
    tma::bulk_g2s(s_cells + (size_t)s * kCellTile * NV, m.cells + t * kCellTile * NV, kTileBytes, &s_bar[s]);
  };
  if (threadIdx.x == 0)
    for (int s = 0; s < kCellStages; ++s) {
      const int64_t t = blockIdx.x + (int64_t)s * gridDim.x;
      if (t < n_full) post(t, s);
    }
  auto decide = [&](const int (&v)[kUnroll][4], const bool (&valid)[kUnroll], int64_t base) {
    unsigned int all[kUnroll], any[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      all[u] = 0xffu;
      any[u] = 0u;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const unsigned int c = __ldg(vclass + v[u][k]);
        all[u] &= c;
        any[u] |= c;
      }
    }
    uint8_t* out = reinterpret_cast<uint8_t*>(s_out[ob]);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int pos = u * kBlock + (int)threadIdx.x;
      bool fast = (all[u] & 3u) != 0u && (all[u] & 4u) != 0u;
      const int tag = (all[u] & 1u) ? 3 : 1;
      bool zden = false, ambiguous = false;
      if (fast && !(any[u] & 8u)) {
        if (all[u] & 16u) zden = true;
        else if (exact_zero_den) fast = false;
        else ambiguous = true;
      }
      if (!valid[u]) continue;
      if (!fast) {  // parked: position inside the tile
        const unsigned int i = atomicAdd(&s_np[par], 1u) - done[par];
        s_pend[par][i] = pos;
        continue;
      }
      out[pos] = (uint8_t)tag;
      if (tags) tags[base + pos] = tag;
      local[0] += tag == 1;
      local[2] += tag == 3;
      local[4] += zden;
      local[5] += ambiguous;
    }
  };
  auto exact_pass = [&](int64_t base) {  // after the tile's barrier: the parked cells, one per thread
    uint8_t* out = reinterpret_cast<uint8_t*>(s_out[ob]);
    const unsigned int end = s_np[par];
    for (unsigned int i = done[par] + threadIdx.x; i < end; i += blockDim.x) {
      const int pos = s_pend[par][i - done[par]];
      const int64_t c = base + pos;
      int w[4] = {0, 0, 0, 0};
      double p[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        w[k] = __ldg(m.cells + c * NV + k);
        p[k] = __ldg(phi + w[k]);
      }
      const int r = tag_cell_exact<CT>(m.x, w[0], w[1], w[2], w[3], p[0], p[1], p[2], p[3]);
      const int tag = r & 0xff;
      if (tags) tags[c] = tag;
      out[pos] = (uint8_t)tag;
      local[0] += tag == 1;
      local[1] += tag == 2;
      local[2] += tag == 3;
      local[3] += tag == 0;
      local[4] += (r >> 8) != 0;
    }
    done[par] = end;
    par ^= 1;
  };
  auto flush = [&](int buf, int64_t base) {  // the tags of a finished tile: one word per thread
    const int64_t c0 = base + (int64_t)threadIdx.x * 4;
    const unsigned int w = s_out[buf][threadIdx.x];
    if (c0 + 3 < m.n_cells) {
      *reinterpret_cast<unsigned int*>(tags8 + c0) = w;
    } else {
      for (int q = 0; q < 4; ++q)
        if (c0 + q < m.n_cells) tags8[c0 + q] = (int8_t)(w >> (8 * q));
    }
  };
  int64_t prev_base = -1;
  auto finish_tile = [&](int64_t base) {  // called by every thread right after the tile's barrier
    if (prev_base >= 0) flush(ob == 0 ? 2 : ob - 1, prev_base);
    exact_pass(base);
    prev_base = base;
    ob = ob == 2 ? 0 : ob + 1;
  };
  int k = 0;
  for (int64_t t = blockIdx.x; t < n_full; t += gridDim.x, ++k) {
    const int s = k % kCellStages;
    tma::mbar_wait(&s_bar[s], (uint32_t)(k / kCellStages) & 1u);
    const int32_t* tile = s_cells + (size_t)s * kCellTile * NV;
    int v[kUnroll][4];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int pos = u * kBlock + (int)threadIdx.x;
      if constexpr (NV == 4) {
        const int4 q = reinterpret_cast<const int4*>(tile)[pos];
        v[u][0] = q.x; v[u][1] = q.y; v[u][2] = q.z; v[u][3] = q.w;
      } else {
#pragma unroll
        for (int q = 0; q < NV; ++q) v[u][q] = tile[pos * NV + q];
        v[u][3] = 0;
      }
    }
    const bool valid[kUnroll] = {true, true, true, true};
    decide(v, valid, t * kCellTile);
    __syncthreads();  // parked list and output bytes complete, every thread done with the stage
    if (threadIdx.x == 0) {
      const int64_t tn = t + (int64_t)kCellStages * gridDim.x;
      if (tn < n_full) post(tn, s);
    }
    finish_tile(t * kCellTile);
  }
  if (blockIdx.x == (unsigned)(n_full % gridDim.x) && n_full * kCellTile < m.n_cells) {  // the ragged end
    const int64_t base = n_full * kCellTile;
    int v[kUnroll][4];
    bool valid[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int64_t c = base + u * kBlock + (int64_t)threadIdx.x;
      valid[u] = c < m.n_cells;
#pragma unroll
      for (int q = 0; q < 4; ++q) v[u][q] = (valid[u] && q < NV) ? __ldg(m.cells + c * NV + q) : 0;
    }
    decide(v, valid, base);
    __syncthreads();
    finish_tile(base);
  }
  __syncthreads();  // the last tile's exact path has written its bytes
  if (prev_base >= 0) flush(ob == 0 ? 2 : ob - 1, prev_base);
#pragma unroll
  for (int i = 0; i < 6; ++i) cnt.add(local[i], i);
  cnt.flush(counters, PHIFEM_CNT_INTERIOR, 6);
}

// ---- K1b: generic table-driven cell classification (P1..P3 / Q1..Q3, any detection degree) ----
template <int CT>
__global__ void __launch_bounds__(kBlock) k_tag_cells_generic(phifem_mesh m, phifem_levelset ls,
                                                              int32_t* __restrict__ tags,
                                                              int8_t* __restrict__ tags8,
                                                              int64_t* counters) {
  using T = CellTraits<CT>;
  __shared__ unsigned int scnt[5];
  BlockCounters cnt(scnt, 5);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int npts = ls.n_cell_points, nd = ls.n_dofs_per_cell;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < m.n_cells; base += stride) {
    const int64_t c = base + threadIdx.x;
    int tag = -1;
    bool zden = false;
    if (c < m.n_cells) {
      int v[LocalBounds<CT>::nv];
      double xc[LocalBounds<CT>::nv][3];
      load_cell<CT>(m, c, v, xc);
      double cd[LocalBounds<CT>::nd];
      if (ls.mode == 0) load_coeffs(m, ls, T::nv, c, v, cd);
      double s = 0.0;
      if constexpr (CT == PHIFEM_TRIANGLE || CT == PHIFEM_TETRAHEDRON) s = simplex_detj<CT>(xc);
      double num = 0.0, den = 0.0;
      for (int q = 0; q < npts; ++q) {
        if constexpr (CT == PHIFEM_HEXAHEDRON) {
          s = hex_detj(ls.coord_grad + q * 24, xc);  // [8 vertices][3]
        } else if (CT == PHIFEM_QUADRILATERAL) {
          const double* g = ls.coord_grad + q * 8;  // [4 vertices][2]
          const double j00 = seq_dot(g + 0, 2, &xc[0][0], 3, 4);
          const double j01 = seq_dot(g + 1, 2, &xc[0][0], 3, 4);
          const double j10 = seq_dot(g + 0, 2, &xc[0][1], 3, 4);
          const double j11 = seq_dot(g + 1, 2, &xc[0][1], 3, 4);
          s = fabs(j00 * j11 - j01 * j10);
        }
        const double ph = ls.mode == 0 ? seq_dot(ls.cell_table + q * nd, 1, cd, 1, nd)
                                       : __ldg(ls.cell_values + c * npts + q);
        const double t = ph * s;
        num = num + t;
        den = den + fabs(t);
      }
      tag = classify(num, den);
      zden = is_close_to_zero(den);
      if (tags) tags[c] = tag;
      tags8[c] = (int8_t)tag;
    }
    cnt.vote(tag == 1, 0);
    cnt.vote(tag == 2, 1);
    cnt.vote(tag == 3, 2);
    cnt.vote(tag == 0, 3);
    cnt.vote(zden, 4);
  }
  cnt.flush(counters, PHIFEM_CNT_INTERIOR, 5);
}

// ---- single_layer_cut (mesh_scripts.py:349-358) --------------------------------------------------
__global__ void k_single_layer_mark(const int32_t* __restrict__ cells, int nv, int64_t n_cells,
                                    const int8_t* __restrict__ tags8, uint8_t* vflag) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells || tags8[c] != 1) return;
  for (int k = 0; k < nv; ++k) vflag[cells[c * nv + k]] = 1;  // benign race: everybody stores 1
}

__global__ void k_single_layer_apply(const int32_t* __restrict__ cells, int nv, int64_t n_cells,
                                     int32_t* tags, int8_t* tags8, const uint8_t* __restrict__ vflag,
                                     int64_t* counters) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_cells || tags8[c] != 2) return;
  bool touches = false;
  for (int k = 0; k < nv; ++k) touches |= vflag[cells[c * nv + k]] != 0;
  if (!touches) {  // isolated cut cell -> exterior
    if (tags) tags[c] = 3;
    tags8[c] = 3;
    atomicAdd(reinterpret_cast<unsigned long long*>(counters + PHIFEM_CNT_EXTERIOR), 1ull);
    atomicAdd(reinterpret_cast<unsigned long long*>(counters + PHIFEM_CNT_CUT), ~0ull);  // -1
  }
}

// ---- K1c: facet tags ------------------------------------------------------------------------------
// ds-detection of the owner cell of a mesh-boundary facet (mesh_scripts.py:434-452): per exterior
// facet sum_q phi_q*s_f, added into the cell entry in ascending facet index.
template <int CT>
__device__ __noinline__ bool owner_is_ds_cut(const phifem_mesh& m, const phifem_levelset& ls, int64_t c,
                                int32_t this_facet, bool* first_of_cell, bool* zden) {
  using T = CellTraits<CT>;
  int v[LocalBounds<CT>::nv];
  double xc[LocalBounds<CT>::nv][3];
  load_cell<CT>(m, c, v, xc);
  double cd[LocalBounds<CT>::nd];
  if (ls.mode == 0) load_coeffs(m, ls, T::nv, c, v, cd);
  int32_t fid[LocalBounds<CT>::nf];
  bool isb[LocalBounds<CT>::nf];
  int32_t smallest = INT32_MAX;
#pragma unroll
  for (int i = 0; i < T::nf; ++i) {
    fid[i] = __ldg(m.c2f + c * T::nf + i);
    isb[i] = __ldg(m.f2c + 2 * (int64_t)fid[i] + 1) < 0;
    if (isb[i] && fid[i] < smallest) smallest = fid[i];
  }
  *first_of_cell = (smallest == this_facet);
  const int nq = ls.n_facet_points, nd = ls.n_dofs_per_cell;
  double num = 0.0, den = 0.0;
  int32_t last = -1;
  for (int round = 0; round < T::nf; ++round) {
    int lf = -1;
    int32_t best = INT32_MAX;
#pragma unroll
    for (int i = 0; i < T::nf; ++i)
      if (isb[i] && fid[i] > last && fid[i] < best) {
        best = fid[i];
        lf = i;
      }
    if (lf < 0) break;
    last = best;
    double sc = 0.0;  // hexahedra: per point (faces need not be planar)
    if constexpr (CT != PHIFEM_HEXAHEDRON) sc = facet_scale<CT>(xc, lf);
    double fn = 0.0, fd = 0.0;
    for (int q = 0; q < nq; ++q) {
      const double ph = ls.mode == 0
                            ? seq_dot(ls.facet_table + ((int64_t)lf * nq + q) * nd, 1, cd, 1, nd)
                            : __ldg(ls.facet_values + (c * T::nf + lf) * nq + q);
      if constexpr (CT == PHIFEM_HEXAHEDRON)
        sc = hex_facet_scale(ls.coord_grad + ((int64_t)ls.n_cell_points + lf * nq + q) * 24, xc, lf);
      const double t = ph * sc;
      fn = fn + t;
      fd = fd + fabs(t);
    }
    num = num + fn;
    den = den + fd;
  }
  *zden = is_close_to_zero(den);
  const double d = (den > 0.0) ? num / den : 0.5;
  return d > -1.0 && d < 1.0;
}

// The facet algebra of mesh_scripts.py:454-497 for ONE facet: membership flags in, tag out (bit 8 = the
// reference would emit the facet twice).  Evaluated at compile time into a lookup table for interior
// facets and at run time for the (rare) mesh-boundary facets.
__host__ __device__ constexpr int facet_algebra(int t0, int t1, bool bnd, bool k, bool anyE) {
  const bool inI = (t0 == 1) | (t1 == 1), inC = (t0 == 2) | (t1 == 2), inE = (t0 == 3) | (t1 == 3);
  const bool cut_bnd = bnd && k;                                  // :454-456
  const bool uncut_bnd = bnd && !k && !inE && !inI;               // :457-461
  const bool int_bnd = inI && inC;                                // :464-466
  bool boundary = anyE ? ((inE && inC) || uncut_bnd) : bnd;       // :469-474
  const bool direct = inE && inI;                                 // :476-478
  const bool cutf = (inC && !(boundary || int_bnd || direct || uncut_bnd)) || cut_bnd;  // :480-485
  const bool rem = int_bnd || boundary || direct;
  const bool interior = inI && !rem;                              // :488-490
  const bool exterior = inE && !rem;                              // :493-495
  boundary = boundary && !cutf;                                   // :497
  // stacking order [5,1,3,2,4,6] of :524-552; the last writer wins when the algebra is inconsistent
  int tag = 0;
  if (exterior) tag = 5;
  if (interior) tag = 1;
  if (int_bnd) tag = 3;
  if (cutf) tag = 2;
  if (boundary) tag = 4;
  if (direct) tag = 6;
  const int n = (int)exterior + (int)interior + (int)int_bnd + (int)cutf + (int)boundary + (int)direct;
  return tag | (n > 1 ? 0x100 : 0);
}

// interior facets: 4 bits per (t0, t1) pair, t in 0..3 (for them `anyE` cannot change the outcome: it
// only matters when a tag-3 cell exists, and then anyE is true)
__host__ __device__ constexpr unsigned long long interior_facet_lut(bool conflicts) {
  unsigned long long lut = 0;
  for (int t0 = 0; t0 < 4; ++t0)
    for (int t1 = 0; t1 < 4; ++t1) {
      const int r = facet_algebra(t0, t1, false, false, true);
      const unsigned long long v = conflicts ? (unsigned long long)(r >> 8) : (unsigned long long)(r & 0xf);
      lut |= v << (4 * (t0 * 4 + t1));
    }
  return lut;
}

// mesh-boundary facet: needs the ds detection of its owner cell; returns the tag, updates counters
template <int CT>
__device__ __forceinline__ int tag_boundary_facet(const phifem_mesh& m, const phifem_levelset& ls,
                                                  int owner, int t0, int32_t f, bool anyE,
                                                  unsigned int& n_zden, unsigned int& n_conflict,
                                                  unsigned int& n_owner) {
  bool zden = false, owner_first = false;
  const bool k = owner_is_ds_cut<CT>(m, ls, owner, f, &owner_first, &zden);
  const int r = facet_algebra(t0, 0, true, k, anyE);
  n_conflict += r >> 8;
  n_zden += owner_first && zden;
  n_owner += owner_first;
  return r & 0xf;
}

// second pass over the (precomputed, mesh-level) list of mesh-boundary facets: keeps the heavy
// table-driven ds detection out of the streaming kernel
template <int CT>
__global__ void __launch_bounds__(kBlock) k_tag_boundary_facets(phifem_mesh m, phifem_levelset ls,
                                                                const int8_t* __restrict__ ctags,
                                                                int32_t* __restrict__ ftags,
                                                                int8_t* __restrict__ ftags8,
                                                                int64_t* counters) {
  __shared__ unsigned int scnt[4];
  BlockCounters cnt(scnt, 3);
  unsigned int n_zden = 0, n_conflict = 0, n_owner = 0;
  const bool anyE = *reinterpret_cast<volatile int64_t*>(counters + PHIFEM_CNT_EXTERIOR) > 0;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m.n_boundary_facets) {
    const int32_t f = __ldg(m.boundary_facets + i);
    const int owner = __ldg(m.f2c + 2 * (int64_t)f);
    const int tag = tag_boundary_facet<CT>(m, ls, owner, __ldg(ctags + owner) & 3, f, anyE, n_zden,
                                           n_conflict, n_owner);
    if (ftags) ftags[f] = tag;
    ftags8[f] = (int8_t)tag;
  }
  cnt.add(n_zden, 0);
  cnt.add(n_conflict, 1);
  cnt.add(n_owner, 2);
  cnt.flush(counters, PHIFEM_CNT_FACET_ZERO_DEN, 3);
}

template <int CT, bool kInlineBoundary>
__global__ void __launch_bounds__(kBlock, 4) k_tag_facets(phifem_mesh m, phifem_levelset ls,
                                                          const int8_t* __restrict__ ctags,
                                                          int32_t* __restrict__ ftags,
                                                          int8_t* __restrict__ ftags8, int64_t* counters) {
  constexpr unsigned long long kTagLut = interior_facet_lut(false);
  constexpr unsigned long long kConflictLut = interior_facet_lut(true);
  __shared__ unsigned int scnt[4];
  BlockCounters cnt(scnt, 3);
  unsigned int n_zden = 0, n_conflict = 0, n_owner = 0;
  // "no exterior cell at all" switches the meaning of mesh-boundary facets (:469-474)
  const bool anyE = *reinterpret_cast<volatile int64_t*>(counters + PHIFEM_CNT_EXTERIOR) > 0;
  // each thread owns kUnroll CONSECUTIVE facets: 32 bytes of f2c in, 16 + 4 bytes of tags out
  const int64_t tile = (int64_t)blockDim.x * kUnroll;
  for (int64_t base = (int64_t)blockIdx.x * tile; base < m.n_facets; base += (int64_t)gridDim.x * tile) {
    const int64_t f0 = base + (int64_t)threadIdx.x * kUnroll;
    int2 cc[kUnroll];
    bool valid[kUnroll];
    static_assert(kUnroll == 4, "vector loads / stores below assume 4 facets per thread");
    if (f0 + kUnroll <= m.n_facets) {
      const int4 a = __ldg(reinterpret_cast<const int4*>(m.f2c) + f0 / 2);
      const int4 b = __ldg(reinterpret_cast<const int4*>(m.f2c) + f0 / 2 + 1);
      cc[0] = make_int2(a.x, a.y); cc[1] = make_int2(a.z, a.w);
      cc[2] = make_int2(b.x, b.y); cc[3] = make_int2(b.z, b.w);
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) valid[u] = true;
    } else {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        valid[u] = f0 + u < m.n_facets;
        cc[u] = valid[u] ? __ldg(reinterpret_cast<const int2*>(m.f2c) + f0 + u) : make_int2(0, -1);
      }
    }
    int t0[kUnroll], t1[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      t0[u] = __ldg(ctags + cc[u].x) & 3;
      t1[u] = cc[u].y < 0 ? 0 : (__ldg(ctags + cc[u].y) & 3);
    }
    int out[kUnroll];
    bool all_interior = valid[kUnroll - 1];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      out[u] = -1;
      if (!valid[u]) continue;
      const int sh = 4 * (t0[u] * 4 + t1[u]);
      int tag = (int)((kTagLut >> sh) & 0xfull);
      if (cc[u].y < 0) {
        if (!kInlineBoundary) {  // tagged by k_tag_boundary_facets
          all_interior = false;
          continue;
        }
        tag = tag_boundary_facet<CT>(m, ls, cc[u].x, t0[u], (int32_t)(f0 + u), anyE, n_zden, n_conflict,
                                     n_owner);
      } else {
        n_conflict += (unsigned int)((kConflictLut >> sh) & 1ull);
      }
      out[u] = tag;
    }
    if (all_interior) {
      if (ftags) *reinterpret_cast<int4*>(ftags + f0) = make_int4(out[0], out[1], out[2], out[3]);
      *reinterpret_cast<unsigned int*>(ftags8 + f0) =
          (unsigned)out[0] | ((unsigned)out[1] << 8) | ((unsigned)out[2] << 16) | ((unsigned)out[3] << 24);
    } else {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u)
        if (out[u] >= 0) {
          if (ftags) ftags[f0 + u] = out[u];
          ftags8[f0 + u] = (int8_t)out[u];
        }
    }
  }
  cnt.add(n_zden, 0);
  cnt.add(n_conflict, 1);
  cnt.add(n_owner, 2);
  cnt.flush(counters, PHIFEM_CNT_FACET_ZERO_DEN, 3);
}

// ---- mesh-boundary facets from per-mesh records ----------------------------------------------------------------------
// k_tag_boundary_facets walks c2f -> f2c -> coordinates for every mesh-boundary facet on every step: five levels of
// dependent gathers over 0.25 M threads, 66 us at config E that do not overlap with the streaming kernel (the facet phase
// measured 0.236 ms = 0.174 + 0.068).  Which facets of the owner lie on the mesh boundary, in which order they are
// summed, whether this facet is the owner's first, and the integration scales are properties of the MESH: tabulated once
// (k_boundary_records), they leave the per-step pass with one level of gathers (the owner's level-set values).
template <int CT>
__global__ void __launch_bounds__(kBlock) k_boundary_records(phifem_mesh m, uint32_t* __restrict__ owner_meta,
                                                             double* __restrict__ scale) {
  using T = CellTraits<CT>;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m.n_boundary_facets) return;
  const int32_t f = __ldg(m.boundary_facets + i);
  const int c = __ldg(m.f2c + 2 * (int64_t)f);
  int v[4];
  double xc[4][3];
  load_cell<CT>(m, c, v, xc);
  int32_t fid[4];
  bool isb[4];
  int32_t smallest = INT32_MAX;
#pragma unroll
  for (int j = 0; j < T::nf; ++j) {
    fid[j] = __ldg(m.c2f + (int64_t)c * T::nf + j);
    isb[j] = __ldg(m.f2c + 2 * (int64_t)fid[j] + 1) < 0;
    if (isb[j] && fid[j] < smallest) smallest = fid[j];
  }
  uint32_t meta = smallest == f ? (1u << 12) : 0u;
  double sc[4] = {0.0, 0.0, 0.0, 0.0};
  int n = 0;
  int32_t last = -1;
  for (int round = 0; round < T::nf; ++round) {  // ascending facet index, as owner_is_ds_cut sums them
    int lf = -1;
    int32_t best = INT32_MAX;
#pragma unroll
    for (int j = 0; j < T::nf; ++j)
      if (isb[j] && fid[j] > last && fid[j] < best) {
        best = fid[j];
        lf = j;
      }
    if (lf < 0) break;
    last = best;
    if constexpr (CT != PHIFEM_QUADRILATERAL) sc[n] = facet_scale<CT>(xc, lf);
    meta |= (uint32_t)lf << (4 + 2 * n);
    ++n;
  }
  meta |= (uint32_t)n;
  owner_meta[2 * i] = (uint32_t)c;
  owner_meta[2 * i + 1] = meta;
#pragma unroll
  for (int q = 0; q < 4; ++q) scale[4 * i + q] = sc[q];
}

template <int CT>
__global__ void __launch_bounds__(kBlock) k_tag_boundary_facets_rec(phifem_mesh m, phifem_levelset ls,
                                                                    const int8_t* __restrict__ ctags,
                                                                    int32_t* __restrict__ ftags,
                                                                    int8_t* __restrict__ ftags8,
                                                                    int64_t* counters) {
  using T = CellTraits<CT>;
  __shared__ unsigned int scnt[4];
  BlockCounters cnt(scnt, 3);
  unsigned int n_zden = 0, n_conflict = 0, n_owner = 0;
  const bool anyE = *reinterpret_cast<volatile int64_t*>(counters + PHIFEM_CNT_EXTERIOR) > 0;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m.n_boundary_facets) {
    const int32_t f = __ldg(m.boundary_facets + i);
    const uint2 om = __ldg(reinterpret_cast<const uint2*>(m.boundary_owner) + i);
    double sc[4];
    ldg256(m.boundary_scale + 4 * i, sc[0], sc[1], sc[2], sc[3]);
    const int64_t c = (int64_t)om.x;
    const uint32_t meta = om.y;
    const int t0 = __ldg(ctags + c) & 3;
    const int nq = ls.n_facet_points, nd = ls.n_dofs_per_cell;
    double cd[kMaxDofs];
    if (ls.mode == 0) {
      int v[4] = {0, 0, 0, 0};
      if (ls.dofmap == nullptr) {
#pragma unroll
        for (int k = 0; k < T::nv; ++k) v[k] = __ldg(m.cells + c * T::nv + k);
      }
      load_coeffs(m, ls, T::nv, c, v, cd);
    }
    double num = 0.0, den = 0.0;
    const int n = (int)(meta & 0xfu);
    for (int r = 0; r < n; ++r) {
      const int lf = (int)((meta >> (4 + 2 * r)) & 3u);
      double s = sc[0];
#pragma unroll
      for (int q = 1; q < 4; ++q)
        if (r == q) s = sc[q];
      double fn = 0.0, fd = 0.0;
      for (int q = 0; q < nq; ++q) {
        const double ph = ls.mode == 0
                              ? seq_dot(ls.facet_table + ((int64_t)lf * nq + q) * nd, 1, cd, 1, nd)
                              : __ldg(ls.facet_values + (c * T::nf + lf) * nq + q);
        const double t = ph * s;
        fn = fn + t;
        fd = fd + fabs(t);
      }
      num = num + fn;
      den = den + fd;
    }
    const double d = (den > 0.0) ? num / den : 0.5;
    const bool k = d > -1.0 && d < 1.0;
    const bool first = (meta >> 12) & 1u;
    const int rr = facet_algebra(t0, 0, true, k, anyE);
    n_conflict += rr >> 8;
    n_zden += first && is_close_to_zero(den);
    n_owner += first;
    const int tag = rr & 0xf;
    if (ftags) ftags[f] = tag;
    ftags8[f] = (int8_t)tag;
  }
  cnt.add(n_zden, 0);
  cnt.add(n_conflict, 1);
  cnt.add(n_owner, 2);
  cnt.flush(counters, PHIFEM_CNT_FACET_ZERO_DEN, 3);
}

// The interior-facet pass with f2c staged through shared memory by TMA bulk copies (the default when the mesh carries
// its list of mesh-boundary facets, which k_tag_boundary_facets finishes).  A tile is kBlock * kUnroll facets = 8 KB of
// f2c; thread 0 keeps kFacetStages tiles in flight per CTA (mbarrier expect_tx / complete_tx), every thread takes 4
// CONSECUTIVE facets out of the landed tile (two 16-byte shared-memory reads), gathers the 8 cell tags and writes its 4
// facet tags as one 32-bit word.  Against the per-thread LDG.128 loop of k_tag_facets (each warp instruction touching 32
// half-used sectors, bytes in flight tied to the resident warps' loop phase) the requests for f2c leave the SM as whole
// 8 KB copies issued three tiles ahead.
constexpr int kFacetStages = 4;
constexpr int kTagFacetsMinBlocks = 5;
constexpr int kFacetTile = kBlock * kUnroll;

template <int CT>
__global__ void __launch_bounds__(kBlock, kTagFacetsMinBlocks) k_tag_facets_staged(
    phifem_mesh m, const int8_t* __restrict__ ctags, int32_t* __restrict__ ftags, int8_t* __restrict__ ftags8,
    int64_t* counters) {
  constexpr unsigned long long kTagLut = interior_facet_lut(false);
  constexpr unsigned long long kConflictLut = interior_facet_lut(true);
  __shared__ alignas(128) int4 s_f2c[kFacetStages][kFacetTile / 2];
  __shared__ alignas(8) uint64_t s_bar[kFacetStages];
  __shared__ unsigned int scnt[4];
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kFacetStages; ++s) tma::mbar_init(&s_bar[s], 1);
    tma::fence_init();
  }
  BlockCounters cnt(scnt, 1);  // (its constructor synchronises the block)
  unsigned int n_conflict = 0;
  constexpr uint32_t kTileBytes = kFacetTile * 8;
  const int64_t n_full = m.n_facets / kFacetTile;  // whole tiles go through TMA, the ragged end through plain loads
  const int2* __restrict__ f2c2 = reinterpret_cast<const int2*>(m.f2c);
  auto post = [&](int64_t t, int s) {
    tma::mbar_expect_tx(&s_bar[s], kTileBytes);
    tma::bulk_g2s(&s_f2c[s][0], f2c2 + t * kFacetTile, kTileBytes, &s_bar[s]);
  };
  if (threadIdx.x == 0)
    for (int s = 0; s < kFacetStages; ++s) {
      const int64_t t = blockIdx.x + (int64_t)s * gridDim.x;
      if (t < n_full) post(t, s);
    }
  // gather: the 8 cell tags of 4 facets; finish: decision table and stores
  auto gather = [&](const int2 (&cc)[kUnroll], int (&t0)[kUnroll], int (&t1)[kUnroll]) {
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      t0[u] = __ldg(ctags + cc[u].x);
      t1[u] = cc[u].y < 0 ? 0 : __ldg(ctags + cc[u].y);
    }
  };
  auto finish = [&](const int2 (&cc)[kUnroll], const int (&t0)[kUnroll], const int (&t1)[kUnroll],
                    const bool (&valid)[kUnroll], int64_t f0) {
    int out[kUnroll];
    bool all_interior = valid[kUnroll - 1];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      out[u] = -1;
      if (!valid[u]) continue;
      if (cc[u].y < 0) {  // tagged by k_tag_boundary_facets
        all_interior = false;
        continue;
      }
      const int sh = 4 * ((t0[u] & 3) * 4 + (t1[u] & 3));
      n_conflict += (unsigned int)((kConflictLut >> sh) & 1ull);
      out[u] = (int)((kTagLut >> sh) & 0xfull);
    }
    if (all_interior) {
      if (ftags) *reinterpret_cast<int4*>(ftags + f0) = make_int4(out[0], out[1], out[2], out[3]);
      *reinterpret_cast<unsigned int*>(ftags8 + f0) =
          (unsigned)out[0] | ((unsigned)out[1] << 8) | ((unsigned)out[2] << 16) | ((unsigned)out[3] << 24);
    } else {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u)
        if (out[u] >= 0) {
          if (ftags) ftags[f0 + u] = out[u];
          ftags8[f0 + u] = (int8_t)out[u];
        }
    }
  };
  static_assert(kUnroll == 4, "4 facets = two int4 per thread");
  int k = 0;
  for (int64_t t = blockIdx.x; t < n_full; t += gridDim.x, ++k) {
    const int s = k % kFacetStages;
    tma::mbar_wait(&s_bar[s], (uint32_t)(k / kFacetStages) & 1u);
    const int4 a = s_f2c[s][2 * threadIdx.x], b = s_f2c[s][2 * threadIdx.x + 1];
    const int2 cc[kUnroll] = {make_int2(a.x, a.y), make_int2(a.z, a.w), make_int2(b.x, b.y), make_int2(b.z, b.w)};
    int t0[kUnroll], t1[kUnroll];
    // The gathers are issued BEFORE the barrier: their addresses need the facet's cells, so every thread's shared-memory
    // reads have returned when it arrives -- the bulk copy that refills the stage runs in the async proxy and is not
    // ordered behind reads still queued in the load/store unit (a barrier alone let 2 360 of 102 M facets at config E
    // see the next tile's f2c).
    gather(cc, t0, t1);
    __syncthreads();
    if (threadIdx.x == 0) {
      const int64_t tn = t + (int64_t)kFacetStages * gridDim.x;
      if (tn < n_full) post(tn, s);
    }
    const bool valid[kUnroll] = {true, true, true, true};
    finish(cc, t0, t1, valid, t * kFacetTile + (int64_t)threadIdx.x * kUnroll);
  }
  if (blockIdx.x == (unsigned)(n_full % gridDim.x) && n_full * kFacetTile < m.n_facets) {  // the ragged end
    const int64_t f0 = n_full * kFacetTile + (int64_t)threadIdx.x * kUnroll;
    int2 cc[kUnroll];
    bool valid[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      valid[u] = f0 + u < m.n_facets;
      cc[u] = valid[u] ? __ldg(f2c2 + f0 + u) : make_int2(0, -1);
    }
    int t0[kUnroll], t1[kUnroll];
    gather(cc, t0, t1);
    if (valid[0]) finish(cc, t0, t1, valid, f0);
  }
  cnt.add(n_conflict, 0);
  cnt.flush(counters, PHIFEM_CNT_FACET_CONFLICT, 1);
}

// ---- candidate records of the one-sided measures (mesh_scripts.py:137-192) -------------------------
// One thread per facet; the slots of a warp's records come from ONE atomicAdd (ballot + popc): 0.5 M increments of a
// single address took 275 us per pass at config E -- four passes per compute_tags_measures call.
__global__ void k_entity_records(phifem_mesh m, int nf_per_cell, const int8_t* __restrict__ ctags,
                                 const int8_t* __restrict__ ftags, int facet_tag, unsigned int cell_mask,
                                 int64_t* records, int64_t capacity, unsigned long long* n_records) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool match = f < m.n_facets && ftags[f] == facet_tag;
  if (!__any_sync(0xffffffffu, match)) return;
  // `_reshape_map` (:195-214) lists the cells of a facet in reverse link order
  int cell_of_col[2] = {-1, -1};
  if (match) {
    const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + f);
    cell_of_col[0] = cc.y >= 0 ? cc.y : cc.x;
    cell_of_col[1] = cc.y >= 0 ? cc.x : -1;
#pragma unroll
    for (int col = 0; col < 2; ++col)
      if (cell_of_col[col] >= 0 && !((cell_mask >> ctags[cell_of_col[col]]) & 1u)) cell_of_col[col] = -1;
  }
  const unsigned int b0 = __ballot_sync(0xffffffffu, cell_of_col[0] >= 0);
  const unsigned int b1 = __ballot_sync(0xffffffffu, cell_of_col[1] >= 0);
  const int total = __popc(b0) + __popc(b1);
  if (total == 0) return;
  const int lane = threadIdx.x & 31;
  unsigned long long base = 0ull;
  if (lane == 0) base = atomicAdd(n_records, (unsigned long long)total);
  base = __shfl_sync(0xffffffffu, base, 0);
  const unsigned int lt = (1u << lane) - 1u;
  unsigned long long slot = base + __popc(b0 & lt) + __popc(b1 & lt);
#pragma unroll
  for (int col = 0; col < 2; ++col) {
    const int c = cell_of_col[col];
    if (c < 0) continue;
    if ((int64_t)slot < capacity) {
      int lf = 0;
      for (int i = 0; i < nf_per_cell; ++i)
        if (m.c2f[(int64_t)c * nf_per_cell + i] == (int32_t)f) lf = i;
      records[3 * slot + 0] = 2 * f + col;
      records[3 * slot + 1] = c;
      records[3 * slot + 2] = lf;
    }
    ++slot;
  }
}

template <int CT>
__global__ void k_cell_points(phifem_mesh m, const double* __restrict__ shape, int npts,
                              double* __restrict__ out) {
  using T = CellTraits<CT>;
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= m.n_cells) return;
  int v[LocalBounds<CT>::nv];
  double xc[LocalBounds<CT>::nv][3];
  load_cell<CT>(m, c, v, xc);
  for (int q = 0; q < npts; ++q)
    for (int d = 0; d < T::gdim; ++d)
      out[(c * npts + q) * T::gdim + d] = seq_dot(shape + q * T::nv, 1, &xc[0][d], 3, T::nv);
}

template <typename F>
int dispatch_cell_type(int ct, F&& fn) {
  switch (ct) {
    case PHIFEM_TRIANGLE: fn(std::integral_constant<int, PHIFEM_TRIANGLE>()); return 0;
    case PHIFEM_QUADRILATERAL: fn(std::integral_constant<int, PHIFEM_QUADRILATERAL>()); return 0;
    case PHIFEM_TETRAHEDRON: fn(std::integral_constant<int, PHIFEM_TETRAHEDRON>()); return 0;
    case PHIFEM_HEXAHEDRON: fn(std::integral_constant<int, PHIFEM_HEXAHEDRON>()); return 0;
  }
  return -1;
}

int check_mesh(const phifem_mesh* m, bool need_facets) {
  PHIFEM_CHECK_ARG(m != nullptr, "mesh is null");
  PHIFEM_CHECK_ARG(m->x && m->cells, "mesh.x / mesh.cells is null");
  PHIFEM_CHECK_ARG(m->n_cells >= 0 && m->n_vertices >= 0, "negative sizes");
  PHIFEM_CHECK_ARG(!need_facets || (m->c2f && m->f2c), "mesh.c2f / mesh.f2c is null");
  const int want = m->cell_type == PHIFEM_TETRAHEDRON || m->cell_type == PHIFEM_HEXAHEDRON ? 3 : 2;
  if (m->cell_type < 0 || m->cell_type > 3) {
    set_error("unsupported cell type %d", m->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(m->gdim == want, "gdim does not match the cell type");
  return PHIFEM_OK;
}

int check_levelset(const phifem_mesh* m, const phifem_levelset* ls, bool facets) {
  PHIFEM_CHECK_ARG(ls != nullptr, "levelset is null");
  const bool hex = m->cell_type == PHIFEM_HEXAHEDRON;
  if (ls->mode == 0) {
    PHIFEM_CHECK_ARG(ls->coeffs != nullptr, "levelset.coeffs is null");
    PHIFEM_CHECK_ARG(ls->n_dofs_per_cell >= 1 &&
                         ls->n_dofs_per_cell <= (hex ? LocalBounds<PHIFEM_HEXAHEDRON>::nd : kMaxDofs),
                     "levelset.n_dofs_per_cell out of range");
    PHIFEM_CHECK_ARG(!hex || ls->dofmap != nullptr || ls->n_dofs_per_cell == 8,
                     "levelset.dofmap is null and levelset.n_dofs_per_cell is not 8 (Q1 vertex dofs)");
    // a null cell_table selects the P1 vertex-dof kernel (checked again by the caller)
    PHIFEM_CHECK_ARG(!facets || ls->facet_table != nullptr, "levelset.facet_table is null");
  } else if (ls->mode == 1) {
    PHIFEM_CHECK_ARG(facets ? ls->facet_values != nullptr : ls->cell_values != nullptr,
                     "levelset point values are null");
  } else {
    PHIFEM_CHECK_ARG(false, "levelset.mode must be 0 or 1");
  }
  PHIFEM_CHECK_ARG(facets || m->cell_type != PHIFEM_QUADRILATERAL || ls->coord_grad != nullptr,
                   "levelset.coord_grad is required for quadrilaterals");
  PHIFEM_CHECK_ARG(!hex || ls->coord_grad != nullptr, "levelset.coord_grad is required for hexahedra");
  PHIFEM_CHECK_ARG(!hex || (ls->n_cell_points >= 1 && ls->n_facet_points >= 1),
                   "levelset.n_cell_points / levelset.n_facet_points must be positive for hexahedra");
  return PHIFEM_OK;
}

}  // namespace
}  // namespace phifem

using namespace phifem;

extern "C" int phifem_cell_points(const phifem_mesh* mesh, const double* shape, int32_t n_points,
                                  double* out, void* stream) {
  if (int rc = check_mesh(mesh, false)) return rc;
  PHIFEM_CHECK_ARG(shape && out && n_points > 0, "null pointer / no points");
  if (mesh->n_cells == 0) return PHIFEM_OK;
  const int grid = (int)((mesh->n_cells + kBlock - 1) / kBlock);
  dispatch_cell_type(mesh->cell_type, [&](auto ct) {
    k_cell_points<decltype(ct)::value><<<grid, kBlock, 0, (cudaStream_t)stream>>>(*mesh, shape, n_points, out);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

namespace {
// PHIFEM_FACETS_KERNEL=ldg / PHIFEM_CELLS_KERNEL=ldg select the per-thread vector-load kernels (A/B runs; read at
// every call so that one process can compare the two)
bool facet_kernel_staged() {
  const char* e = getenv("PHIFEM_FACETS_KERNEL");
  return !(e && e[0] == 'l');
}
bool boundary_kernel_records() {  // PHIFEM_BOUNDARY_KERNEL=walk: ignore the per-mesh records (A/B runs, tests)
  const char* e = getenv("PHIFEM_BOUNDARY_KERNEL");
  return !(e && e[0] == 'w');
}
bool cell_kernel_staged() {
  const char* e = getenv("PHIFEM_CELLS_KERNEL");
  return !(e && e[0] == 'l');
}
}  // namespace

extern "C" int phifem_tag_cells(const phifem_mesh* mesh, const phifem_levelset* ls,
                                int32_t single_layer_cut, int32_t* cell_tags, int8_t* cell_tags8,
                                uint8_t* vertex_scratch, int64_t* counters, void* stream) {
  if (int rc = check_mesh(mesh, false)) return rc;
  if (int rc = check_levelset(mesh, ls, false)) return rc;
  PHIFEM_CHECK_ARG(cell_tags8 && counters, "output pointer is null");
  PHIFEM_CHECK_ARG(vertex_scratch, "vertex_scratch is null (uint8[n_vertices + 3])");
  const bool exact_zero_den = (single_layer_cut & 2) != 0;
  single_layer_cut &= 1;
  if (mesh->n_cells == 0) return PHIFEM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int ct = mesh->cell_type;
  const int nv = ct == PHIFEM_TRIANGLE ? 3 : (ct == PHIFEM_HEXAHEDRON ? 8 : 4);
  const bool simplex = ct == PHIFEM_TRIANGLE || ct == PHIFEM_TETRAHEDRON;
  // P1 fast kernel: vertex dofs, identity table (detection degree 1 puts the points on the vertices)
  const bool p1 = simplex && ls->mode == 0 && ls->dofmap == nullptr && ls->n_dofs_per_cell == nv &&
                  ls->n_cell_points == nv && ls->cell_table == nullptr;
  const int grid = grid_for(mesh->n_cells, kBlock, 8);
  if (p1) {
    const bool have_bounds = mesh->detj_min >= 1e-150 && mesh->detj_max <= 1e150 &&
                             mesh->detj_min <= mesh->detj_max;
    // without bounds on |det J| the magnitude bits stay clear and the denominators are evaluated exactly
    k_vertex_class<<<grid_for((mesh->n_vertices + 3) / 4, kBlock, 8), kBlock, 0, st>>>(
        ls->coeffs, mesh->n_vertices, have_bounds ? mesh->detj_min : 0.0,
        have_bounds ? mesh->detj_max : 1e300, vertex_scratch);
    const bool exact = exact_zero_den || !have_bounds;
    const int64_t tiles = (mesh->n_cells + kBlock * kUnroll - 1) / (kBlock * kUnroll);
    const bool staged = cell_kernel_staged() && (reinterpret_cast<uintptr_t>(mesh->cells) & 15) == 0 &&
                        (reinterpret_cast<uintptr_t>(cell_tags8) & 3) == 0;
    auto launch_staged = [&](auto c) {
      constexpr int CT = decltype(c)::value;
      constexpr size_t smem = staged_cells_smem<CT>();
      auto kernel = k_tag_cells_p1_staged<CT>;
      static bool attr_set[64] = {};
      int dev = 0;
      cudaGetDevice(&dev);
      if (!attr_set[dev & 63]) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_set[dev & 63] = true;
      }
      int per_sm = 0, sms = kNumSMs;
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem) != cudaSuccess || per_sm < 1)
        per_sm = 1;
      const int64_t cap = (int64_t)sms * per_sm;
      const int grid = (int)(tiles < cap ? tiles : cap);
      kernel<<<grid, kBlock, smem, st>>>(*mesh, ls->coeffs, vertex_scratch, exact, cell_tags, cell_tags8, counters);
    };
    if (staged && ct == PHIFEM_TRIANGLE)
      launch_staged(std::integral_constant<int, PHIFEM_TRIANGLE>());
    else if (staged)
      launch_staged(std::integral_constant<int, PHIFEM_TETRAHEDRON>());
    else if (ct == PHIFEM_TRIANGLE)
      k_tag_cells_p1<PHIFEM_TRIANGLE><<<persistent_grid(k_tag_cells_p1<PHIFEM_TRIANGLE>, kBlock, tiles),
                                        kBlock, 0, st>>>(*mesh, ls->coeffs, vertex_scratch, exact, cell_tags,
                                                         cell_tags8, counters);
    else
      k_tag_cells_p1<PHIFEM_TETRAHEDRON><<<persistent_grid(k_tag_cells_p1<PHIFEM_TETRAHEDRON>, kBlock, tiles),
                                           kBlock, 0, st>>>(*mesh, ls->coeffs, vertex_scratch, exact, cell_tags,
                                                            cell_tags8, counters);
  } else {
    PHIFEM_CHECK_ARG(ls->mode != 0 || ls->cell_table != nullptr, "levelset.cell_table is null");
    dispatch_cell_type(ct, [&](auto c) {
      k_tag_cells_generic<decltype(c)::value><<<grid, kBlock, 0, st>>>(*mesh, *ls, cell_tags, cell_tags8,
                                                                      counters);
    });
  }
  PHIFEM_CHECK_LAUNCH();
  if (single_layer_cut) {
    cudaMemsetAsync(vertex_scratch, 0, (size_t)mesh->n_vertices, st);
    const int g = (int)((mesh->n_cells + kBlock - 1) / kBlock);
    k_single_layer_mark<<<g, kBlock, 0, st>>>(mesh->cells, nv, mesh->n_cells, cell_tags8, vertex_scratch);
    k_single_layer_apply<<<g, kBlock, 0, st>>>(mesh->cells, nv, mesh->n_cells, cell_tags, cell_tags8,
                                               vertex_scratch, counters);
    PHIFEM_CHECK_LAUNCH();
  }
  return PHIFEM_OK;
}

namespace {
// one side stream + fork/join events per device (created on first use, never destroyed)
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  bool ok = false;
};
SideStream& side_stream() {
  static SideStream per_device[64];
  int dev = 0;
  cudaGetDevice(&dev);
  SideStream& s = per_device[dev & 63];
  if (!s.stream) {
    s.ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess &&
           cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) == cudaSuccess;
  }
  return s;
}
}  // namespace


extern "C" int phifem_tag_facets(const phifem_mesh* mesh, const phifem_levelset* ls,
                                 const int8_t* cell_tags8, int32_t* facet_tags, int8_t* facet_tags8,
                                 int64_t* counters, void* stream) {
  return phifem_tag_facets_phase(mesh, ls, cell_tags8, facet_tags, facet_tags8, counters,
                                 PHIFEM_FACETS_INTERIOR | PHIFEM_FACETS_BOUNDARY, stream);
}

extern "C" int phifem_tag_facets_phase(const phifem_mesh* mesh, const phifem_levelset* ls,
                                       const int8_t* cell_tags8, int32_t* facet_tags, int8_t* facet_tags8,
                                       int64_t* counters, int32_t phases, void* stream) {
  if (int rc = check_mesh(mesh, true)) return rc;
  if (int rc = check_levelset(mesh, ls, true)) return rc;
  PHIFEM_CHECK_ARG(cell_tags8 && facet_tags8 && counters, "null pointer");
  if (mesh->n_facets == 0) return PHIFEM_OK;
  const int64_t tiles = (mesh->n_facets + kBlock * kUnroll - 1) / (kBlock * kUnroll);
  cudaStream_t st = (cudaStream_t)stream;
  const bool two_pass = mesh->boundary_facets != nullptr;
  const bool both = (phases & 3) == 3;
  PHIFEM_CHECK_ARG((phases & 3) != 0, "phases selects nothing");
  PHIFEM_CHECK_ARG(both || two_pass, "phases need mesh.boundary_facets");
  // interior facets of a mesh that lists its boundary facets: f2c staged by TMA (needs a 16-byte aligned f2c; the
  // per-thread vector-load kernel otherwise, or with PHIFEM_FACETS_KERNEL=ldg for A/B runs)
  auto launch_interior = [&](auto c, bool beside_boundary = false) {
    constexpr int CT = decltype(c)::value;
    if (facet_kernel_staged() && (reinterpret_cast<uintptr_t>(mesh->f2c) & 15) == 0) {
      int grid = persistent_grid(k_tag_facets_staged<CT>, kBlock, tiles);
      // Beside the forked mesh-boundary kernel the persistent grid gives up one CTA per SM (5 of 6): the streaming
      // kernel alone is 7 % slower that way (0.161 against 0.150 ms at config E) but the latency-bound boundary kernel
      // then runs entirely under it: both phases 0.168 against 0.178 ms (4 per SM: 0.187), measured with a grid-size
      // override that has since been removed (it is in the history).
      int per_sm = grid / kNumSMs;
      if (beside_boundary && per_sm >= 4 && grid % kNumSMs == 0) grid -= kNumSMs;
      k_tag_facets_staged<CT><<<grid, kBlock, 0, st>>>(*mesh, cell_tags8, facet_tags, facet_tags8, counters);
    } else {
      const int grid = persistent_grid(k_tag_facets<CT, false>, kBlock, tiles);
      k_tag_facets<CT, false><<<grid, kBlock, 0, st>>>(*mesh, *ls, cell_tags8, facet_tags, facet_tags8, counters);
    }
  };
  auto launch_boundary = [&](auto c, cudaStream_t bs) {
    constexpr int CT = decltype(c)::value;
    const int g2 = (int)((mesh->n_boundary_facets + kBlock - 1) / kBlock);
    if constexpr (CT == PHIFEM_HEXAHEDRON) {  // no per-mesh records for hexahedra
      k_tag_boundary_facets<CT><<<g2, kBlock, 0, bs>>>(*mesh, *ls, cell_tags8, facet_tags, facet_tags8, counters);
    } else {
      if (mesh->boundary_owner && mesh->boundary_scale && CT != PHIFEM_QUADRILATERAL && boundary_kernel_records())
        k_tag_boundary_facets_rec<CT><<<g2, kBlock, 0, bs>>>(*mesh, *ls, cell_tags8, facet_tags, facet_tags8,
                                                             counters);
      else
        k_tag_boundary_facets<CT><<<g2, kBlock, 0, bs>>>(*mesh, *ls, cell_tags8, facet_tags, facet_tags8, counters);
    }
  };
  dispatch_cell_type(mesh->cell_type, [&](auto c) {
    constexpr int CT = decltype(c)::value;
    if (!both) {  // one phase alone, on the caller's stream (the caller orders them, e.g. around an all-reduce)
      if (phases & PHIFEM_FACETS_INTERIOR) {
        launch_interior(c);
      } else if (mesh->n_boundary_facets > 0) {
        launch_boundary(c, st);
      }
    } else if (two_pass) {
      // The mesh-boundary facets (a chain of dependent gathers over few threads: latency-bound) run on a
      // side stream forked from / joined to the caller's stream, concurrently with the streaming kernel;
      // the two kernels write disjoint facets.
      SideStream& ss = side_stream();
      const bool fork = mesh->n_boundary_facets > 0 && ss.ok;
      if (fork) {
        cudaEventRecord(ss.fork, st);
        cudaStreamWaitEvent(ss.stream, ss.fork, 0);
        launch_boundary(c, ss.stream);
        cudaEventRecord(ss.join, ss.stream);
      }
      launch_interior(c, fork);
      if (fork) {
        cudaStreamWaitEvent(st, ss.join, 0);
      } else if (mesh->n_boundary_facets > 0) {
        launch_boundary(c, st);
      }
    } else {
      const int grid = persistent_grid(k_tag_facets<CT, true>, kBlock, tiles);
      k_tag_facets<CT, true><<<grid, kBlock, 0, st>>>(*mesh, *ls, cell_tags8, facet_tags, facet_tags8,
                                                      counters);
    }
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_boundary_records(const phifem_mesh* mesh, uint32_t* boundary_owner, double* boundary_scale,
                                       void* stream) {
  if (int rc = check_mesh(mesh, true)) return rc;
  PHIFEM_CHECK_ARG(mesh->n_boundary_facets == 0 || mesh->boundary_facets, "mesh.boundary_facets is null");
  PHIFEM_CHECK_ARG(mesh->n_boundary_facets == 0 || (boundary_owner && boundary_scale), "output pointer is null");
  if (mesh->cell_type == PHIFEM_HEXAHEDRON) {  // 6 local facets do not fit the 2-bit fields of the meta word
    set_error("phifem_boundary_records: no per-mesh boundary records for hexahedra");
    return PHIFEM_ERR_UNSUPPORTED;
  }
  if (mesh->n_boundary_facets == 0) return PHIFEM_OK;
  const int g = (int)((mesh->n_boundary_facets + kBlock - 1) / kBlock);
  dispatch_cell_type(mesh->cell_type, [&](auto c) {
    constexpr int CT = decltype(c)::value;
    if constexpr (CT != PHIFEM_HEXAHEDRON)
      k_boundary_records<CT><<<g, kBlock, 0, (cudaStream_t)stream>>>(*mesh, boundary_owner, boundary_scale);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_entity_records(const phifem_mesh* mesh, const int8_t* cell_tags8,
                                     const int8_t* facet_tags8, int32_t facet_tag, uint32_t cell_mask,
                                     int64_t* records, int64_t capacity, int64_t* n_records,
                                     void* stream) {
  if (int rc = check_mesh(mesh, true)) return rc;
  PHIFEM_CHECK_ARG(cell_tags8 && facet_tags8 && n_records && (records || capacity == 0), "null pointer");
  if (mesh->n_facets == 0) return PHIFEM_OK;
  const int nf = mesh->cell_type == PHIFEM_TRIANGLE ? 3 : (mesh->cell_type == PHIFEM_HEXAHEDRON ? 6 : 4);
  const int grid = (int)((mesh->n_facets + kBlock - 1) / kBlock);
  k_entity_records<<<grid, kBlock, 0, (cudaStream_t)stream>>>(
      *mesh, nf, cell_tags8, facet_tags8, facet_tag, cell_mask, records, capacity,
      reinterpret_cast<unsigned long long*>(n_records));
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}
