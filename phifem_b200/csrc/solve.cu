// CSR sparse matrix-vector product for the Krylov solve that follows the assembly (SURVEY.md section 8f-3).
//
// The reference hands the assembled system to PETSc KSP "preonly" + MUMPS LU with null-pivot detection
// (demo/strong-dirichlet/flower/main.py:138-157, demo/weak-dirichlet/flower/main.py:161-184).  On the GPU the
// system stays where the assembly left it and is solved by Jacobi-preconditioned BiCGStab
// (phifem_b200/solve.py); this file provides its one bandwidth-bound building block.  phi-FEM rows are short
// (15 entries for P1 tetrahedra, 7 for P1 triangles), so a row is reduced by a group of 8 lanes: 4 rows per
// warp, coalesced 64-byte segments of `data` / `indices`, x gathered through the read-only path.
#include "common.cuh"

namespace phifem {
namespace {

constexpr int kSpmvBlock = 256;
constexpr int kLanesPerRow = 8;

__global__ void __launch_bounds__(kSpmvBlock) k_csr_spmv(int64_t n_rows, const int32_t* __restrict__ indptr,
                                                         const int32_t* __restrict__ indices,
                                                         const double* __restrict__ data,
                                                         const double* __restrict__ x, double* __restrict__ y) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = t / kLanesPerRow;
  const int sub = (int)(t % kLanesPerRow);
  double acc = 0.0;
  if (row < n_rows) {
    const int lo = __ldg(indptr + row), hi = __ldg(indptr + row + 1);
    for (int k = lo + sub; k < hi; k += kLanesPerRow) acc += __ldg(data + k) * __ldg(x + __ldg(indices + k));
  }
#pragma unroll
  for (int off = kLanesPerRow / 2; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off, kLanesPerRow);
  if (row < n_rows && sub == 0) y[row] = acc;
}

}  // namespace
}  // namespace phifem

using namespace phifem;

extern "C" int phifem_csr_spmv(int64_t n_rows, const int32_t* indptr, const int32_t* indices,
                               const double* data, const double* x, double* y, void* stream) {
  PHIFEM_CHECK_ARG(n_rows >= 0 && indptr && x && y, "null pointer");
  if (n_rows == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(indices && data, "null CSR arrays");
  const int64_t threads = n_rows * kLanesPerRow;
  k_csr_spmv<<<(unsigned)((threads + kSpmvBlock - 1) / kSpmvBlock), kSpmvBlock, 0, (cudaStream_t)stream>>>(
      n_rows, indptr, indices, data, x, y);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

// ---- fused Jacobi-BiCGStab iteration on the ACTIVE rows ------------------------------------------------------------------
// The torch-op iteration of round 1 ran ~25 elementwise / reduction kernels per iteration over full-length vectors
// (8.6 M rows in box mode, 3.4 M of them active): 1.6 ms per iteration at config E, of which the two products take 0.4.
// Here the unknowns are compacted to the active rows (the vectors then fit the L2: 27 MB each), the matrix is read in
// place through the row list and a column array remapped once per solve, and an iteration is FIVE kernels + three
// one-block scalar updates with every scalar in device memory:
//   p = r + beta (p - omega v), y = M^-1 p | v = A y, rhat.v | s = r - alpha v, z = M^-1 s | t = A z, t.s, t.t |
//   x += alpha y + omega z, r = s - omega t, rhat.r, r.r
// Dot products are per-block partial sums reduced in a fixed order by the scalar kernel: bitwise reproducible.
namespace phifem {
namespace {

constexpr int kVecBlock = 256;
enum { kRho = 0, kAlpha = 1, kOmega = 2, kBeta = 3, kRR = 4, kRhoNew = 5 };  // slots of the state vector

__device__ __forceinline__ double block_sum(double v, double* sh) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) sh[w] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += sh[i];
  __syncthreads();
  return s;  // valid in thread 0
}

// y[i] = sum_k data[k] x[cols[k]] over row rows[i] of the ORIGINAL matrix (cols = column ids remapped to the compact
// numbering, inactive columns -> n_act, where x holds 0); partial sums of w[i] y[i] and y[i]^2 per block
template <int L>
__global__ void __launch_bounds__(kSpmvBlock) k_spmv_rows_dot(int64_t n_act, const int32_t* __restrict__ rows,
                                                              const int32_t* __restrict__ indptr,
                                                              const int32_t* __restrict__ cols,
                                                              const double* __restrict__ data,
                                                              const double* __restrict__ x, const double* __restrict__ w,
                                                              double* __restrict__ y, double* __restrict__ partials) {
  __shared__ double sh[2][kSpmvBlock / 32];
  const int sub = (int)(threadIdx.x % L);
  const int64_t groups_per_pass = (int64_t)gridDim.x * (kSpmvBlock / L);
  double wy = 0.0, yy = 0.0;
  // persistent grid (at most 8 CTAs per SM): the number of partial sums the one-block scalar kernel has to add stays
  // ~1 000 whatever the size of the system; every lane group walks its rows with the same trip count as its warp
  const int64_t n_pass = (n_act + groups_per_pass - 1) / groups_per_pass;
  for (int64_t pass = 0; pass < n_pass; ++pass) {
    const int64_t i = pass * groups_per_pass + (int64_t)blockIdx.x * (kSpmvBlock / L) + threadIdx.x / L;
    double acc = 0.0;
    if (i < n_act) {
      const int row = __ldg(rows + i);
      const int lo = __ldg(indptr + row), hi = __ldg(indptr + row + 1);
      // kBatch entries per lane at a time: their column ids and values are requested together, then the gathers of x,
      // then the products -- a lane's trip through a 15-entry row is one batch instead of four dependent
      // load -> load -> fma rounds (430 iterations at config E: 193.5 ms with one entry at a time, 182.2 with two,
      // 180.3 with four; DESIGN.md §4)
      constexpr int kBatch = 4;
      for (int k0 = lo + sub; k0 < hi; k0 += kBatch * L) {
        int c[kBatch];
        double a[kBatch], xv[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
          const int k = k0 + u * L;
          const bool in = k < hi;
          c[u] = in ? __ldg(cols + k) : (int)n_act;   // x[n_act] = 0 by contract (the slot of the inactive columns)
          a[u] = in ? __ldg(data + k) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < kBatch; ++u) xv[u] = __ldg(x + c[u]);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) acc += a[u] * xv[u];
      }
    }
#pragma unroll
    for (int off = L / 2; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off, L);
    if (i < n_act && sub == 0) {
      y[i] = acc;
      wy += __ldg(w + i) * acc;
      yy += acc * acc;
    }
  }
  const double s0 = block_sum(wy, sh[0]);
  const double s1 = block_sum(yy, sh[1]);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = s0;
    partials[2 * blockIdx.x + 1] = s1;
  }
}

// one block: reduce the partial sums in a fixed order and update the scalars.  kind 0: rho_new = sum(p0), beta;
// kind 1: alpha = rho_new / sum(p0); kind 2: omega = sum(p0) / sum(p1); after kind 0 rho <- rho_new is deferred to kind 2
__global__ void __launch_bounds__(kVecBlock) k_bicgstab_scalars(int kind, const double* __restrict__ partials,
                                                               int n_blocks, double* __restrict__ st) {
  __shared__ double sh[2][kVecBlock / 32];
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < n_blocks; i += blockDim.x) {
    a += partials[2 * i];
    b += partials[2 * i + 1];
  }
  const double s0 = block_sum(a, sh[0]);
  const double s1 = block_sum(b, sh[1]);
  if (threadIdx.x != 0) return;
  const double tiny = 1e-300;
  if (kind == 0) {
    st[kRhoNew] = s0;
    st[kRR] = s1;
    st[kBeta] = (s0 / (st[kRho] + tiny)) * (st[kAlpha] / (st[kOmega] + tiny));
  } else if (kind == 1) {
    st[kAlpha] = st[kRhoNew] / (s0 + tiny);
  } else {
    st[kOmega] = s0 / (s1 + tiny);
    st[kRho] = st[kRhoNew];
  }
}

__global__ void __launch_bounds__(kVecBlock) k_bicgstab_p(int64_t n, const double* __restrict__ r,
                                                         const double* __restrict__ v, const double* __restrict__ minv,
                                                         const double* __restrict__ st, double* __restrict__ p,
                                                         double* __restrict__ y) {
  const double beta = st[kBeta], omega = st[kOmega];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double pi = r[i] + beta * (p[i] - omega * v[i]);
    p[i] = pi;
    y[i] = pi * minv[i];
  }
}

__global__ void __launch_bounds__(kVecBlock) k_bicgstab_s(int64_t n, const double* __restrict__ r,
                                                         const double* __restrict__ v, const double* __restrict__ minv,
                                                         const double* __restrict__ st, double* __restrict__ s,
                                                         double* __restrict__ z) {
  const double alpha = st[kAlpha];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double si = r[i] - alpha * v[i];
    s[i] = si;
    z[i] = si * minv[i];
  }
}

// x += alpha y + omega z, r = s - omega t; partial sums of rhat.r and r.r (grid = n_blocks blocks exactly)
__global__ void __launch_bounds__(kVecBlock) k_bicgstab_x(int64_t n, const double* __restrict__ y,
                                                         const double* __restrict__ z, const double* __restrict__ s,
                                                         const double* __restrict__ t, const double* __restrict__ rhat,
                                                         const double* __restrict__ st, double* __restrict__ x,
                                                         double* __restrict__ r, double* __restrict__ partials) {
  __shared__ double sh[2][kVecBlock / 32];
  const double alpha = st[kAlpha], omega = st[kOmega];
  double a = 0.0, b = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    x[i] += alpha * y[i] + omega * z[i];
    const double ri = s[i] - omega * t[i];
    r[i] = ri;
    a += rhat[i] * ri;
    b += ri * ri;
  }
  const double s0 = block_sum(a, sh[0]);
  const double s1 = block_sum(b, sh[1]);
  if (threadIdx.x == 0) {
    partials[2 * blockIdx.x] = s0;
    partials[2 * blockIdx.x + 1] = s1;
  }
}

}  // namespace
}  // namespace phifem

// set-up of the solve in two passes over the matrix instead of torch temporaries of nnz int64 entries:
// diagonal and largest magnitude of every row (the relative null-pivot test), and the column ids in the compact numbering
namespace phifem {
namespace {
__global__ void __launch_bounds__(256) k_row_scan(int64_t n_rows, const int32_t* __restrict__ indptr,
                                                 const int32_t* __restrict__ indices, const double* __restrict__ data,
                                                 double* __restrict__ diag, double* __restrict__ rowmax) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = t >> 2;
  const int sub = (int)(t & 3);
  double d = 0.0, mx = 0.0;
  if (row < n_rows) {
    const int lo = __ldg(indptr + row), hi = __ldg(indptr + row + 1);
    for (int k = lo + sub; k < hi; k += 4) {
      const double a = __ldg(data + k);
      if (__ldg(indices + k) == (int32_t)row) d = a;
      mx = fmax(mx, fabs(a));
    }
  }
#pragma unroll
  for (int off = 2; off > 0; off >>= 1) {
    const double od = __shfl_down_sync(0xffffffffu, d, off, 4);
    const double om = __shfl_down_sync(0xffffffffu, mx, off, 4);
    if (od != 0.0) d = od;
    mx = fmax(mx, om);
  }
  if (row < n_rows && sub == 0) {
    diag[row] = d;
    rowmax[row] = mx;
  }
}
__global__ void __launch_bounds__(256) k_remap_columns(int64_t nnz, const int32_t* __restrict__ indices,
                                                      const int32_t* __restrict__ cmap, int32_t* __restrict__ cols) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x)
    cols[k] = __ldg(cmap + __ldg(indices + k));
}
}  // namespace
}  // namespace phifem

extern "C" int phifem_csr_row_scan(int64_t n_rows, const int32_t* indptr, const int32_t* indices, const double* data,
                                   double* diag, double* rowmax, void* stream) {
  if (n_rows == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(n_rows > 0 && indptr && indices && data && diag && rowmax, "null pointer");
  const int64_t threads = n_rows * 4;
  k_row_scan<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n_rows, indptr, indices, data, diag,
                                                                                 rowmax);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_remap_columns(int64_t nnz, const int32_t* indices, const int32_t* cmap, int32_t* cols, void* stream) {
  if (nnz == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(nnz > 0 && indices && cmap && cols, "null pointer");
  k_remap_columns<<<8 * kNumSMs, 256, 0, (cudaStream_t)stream>>>(nnz, indices, cmap, cols);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

// lanes per row by the average row length (measured at config E, 15 entries per row, one BiCGStab iteration: 2 lanes 0.45 ms,
// 4: 0.45, 8: 0.55, 16: 0.89)
static int spmv_lanes(int64_t n_act, int64_t nnz_hint) {
  const int64_t avg = n_act > 0 ? nnz_hint / n_act : 0;
  return avg <= 24 ? 4 : (avg <= 48 ? 8 : (avg <= 96 ? 16 : 32));
}
static int spmv_rows_grid(int64_t n_act, int lanes) {
  const int64_t need = (n_act * lanes + kSpmvBlock - 1) / kSpmvBlock;
  const int64_t cap = 8 * (int64_t)kNumSMs;
  return (int)(need < cap ? need : cap);
}
static void launch_spmv_rows(int lanes, int grid, cudaStream_t st, int64_t n_act, const int32_t* rows, const int32_t* indptr,
                             const int32_t* cols, const double* data, const double* x, const double* w, double* y,
                             double* partials) {
  switch (lanes) {
    case 4: k_spmv_rows_dot<4><<<grid, kSpmvBlock, 0, st>>>(n_act, rows, indptr, cols, data, x, w, y, partials); break;
    case 8: k_spmv_rows_dot<8><<<grid, kSpmvBlock, 0, st>>>(n_act, rows, indptr, cols, data, x, w, y, partials); break;
    case 16: k_spmv_rows_dot<16><<<grid, kSpmvBlock, 0, st>>>(n_act, rows, indptr, cols, data, x, w, y, partials); break;
    default: k_spmv_rows_dot<32><<<grid, kSpmvBlock, 0, st>>>(n_act, rows, indptr, cols, data, x, w, y, partials); break;
  }
}

// y = A x on the compact system (rows / cols as below); partials: scratch of 2 * 8 * 148 doubles
extern "C" int phifem_csr_spmv_rows(int64_t n_act, int64_t nnz, const int32_t* rows, const int32_t* indptr,
                                    const int32_t* cols, const double* data, const double* x, double* y, double* partials,
                                    void* stream) {
  if (n_act == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(n_act > 0 && rows && indptr && cols && data && x && y && partials, "null pointer");
  const int lanes = spmv_lanes(n_act, nnz);
  launch_spmv_rows(lanes, spmv_rows_grid(n_act, lanes), (cudaStream_t)stream, n_act, rows, indptr, cols, data, x, x, y,
                   partials);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

// `iterations` BiCGStab iterations on the compact system, no host synchronisation: the caller reads state[4] = r.r when
// it wants to test convergence.  rows [n_act]: the active rows of the CSR matrix (indptr, data as assembled); cols [nnz]:
// its column ids in the compact numbering, inactive columns -> n_act.  Vectors of length n_act; y and z have one more
// slot (index n_act) that must hold 0.  state: 8 doubles {rho, alpha, omega, beta, r.r, rho_new, -, -}, set to
// {1, 1, 1, 0, ...} before the first call; partials: 2 * 8 * 148 doubles whose first *n_partials pairs hold
// partial sums of (rhat.r, r.r) of the current residual (first call: one pair); *n_partials is updated for the next call.
extern "C" int phifem_bicgstab_iterate(int64_t n_act, int64_t nnz, const int32_t* rows, const int32_t* indptr,
                                       const int32_t* cols, const double* data, const double* minv, const double* rhat, double* x, double* r,
                                       double* p, double* v, double* s, double* t, double* y, double* z, double* state,
                                       double* partials, int32_t* n_partials, int32_t iterations, void* stream) {
  PHIFEM_CHECK_ARG(n_act > 0 && rows && indptr && cols && data && minv && rhat && x && r && p && v && s && t && y && z &&
                       state && partials && n_partials,
                   "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int lanes = spmv_lanes(n_act, nnz);
  const int spmv_grid = spmv_rows_grid(n_act, lanes);
  int vec_grid = (int)((n_act + kVecBlock - 1) / kVecBlock);
  if (vec_grid > 8 * kNumSMs) vec_grid = 8 * kNumSMs;
  int ready = *n_partials;
  PHIFEM_CHECK_ARG(ready >= 1 && ready <= spmv_grid + vec_grid, "n_partials out of range");
  for (int it = 0; it < iterations; ++it) {
    k_bicgstab_scalars<<<1, kVecBlock, 0, st>>>(0, partials, ready, state);
    k_bicgstab_p<<<vec_grid, kVecBlock, 0, st>>>(n_act, r, v, minv, state, p, y);
    launch_spmv_rows(lanes, spmv_grid, st, n_act, rows, indptr, cols, data, y, rhat, v, partials);
    k_bicgstab_scalars<<<1, kVecBlock, 0, st>>>(1, partials, spmv_grid, state);
    k_bicgstab_s<<<vec_grid, kVecBlock, 0, st>>>(n_act, r, v, minv, state, s, z);
    launch_spmv_rows(lanes, spmv_grid, st, n_act, rows, indptr, cols, data, z, s, t, partials);
    k_bicgstab_scalars<<<1, kVecBlock, 0, st>>>(2, partials, spmv_grid, state);
    k_bicgstab_x<<<vec_grid, kVecBlock, 0, st>>>(n_act, y, z, s, t, rhat, state, x, r, partials);
    ready = vec_grid;
  }
  // r.r of the last iterate into state[4] (rho_new / beta are recomputed identically by a continuation)
  k_bicgstab_scalars<<<1, kVecBlock, 0, st>>>(0, partials, ready, state);
  *n_partials = ready;
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}
