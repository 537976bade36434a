// K2+K4, cell-once form of the cell pass: strong-Dirichlet phi-FEM operator, P1 on triangles / tetrahedra.
//
// Forms of reference demo/strong-dirichlet/flower/main.py:105,107-112 (bilinear, cells) and :126-128 (linear),
// closed forms of SURVEY.md Appendix B.  The row-gather pass (csrc/assemble_rows.cu) evaluates a cell once per
// VERTEX: cofactors, determinant and reciprocal 4 times per tetrahedron, ~146 fp64 instructions per (row, cell)
// record = ~580 per tetrahedron against ~190 for the whole 4x4 tensor evaluated once -- and the B200 retires only 64
// fp64 lanes per clock per SM.  Here a CTA owns a TILE of R consecutive listed rows (spatially compact: the rows are
// listed along a space-filling curve) and works through the cells touching the tile in CHUNKS of R cells:
//   evaluate  thread t takes the cell in slot t of the chunk, gathers its vertices, evaluates the WHOLE element
//             tensor and load vector once and parks the (D+1)^2 + (D+1) values in shared memory, entry-major
//             (buf[e * R + t]: conflict-free);
//   pull      after one barrier the thread of row l walks l's records of this chunk -- (slot, cell-local index of the
//             row's vertex, positions of the other vertices inside the row's column list) -- and adds the row of the
//             parked tensor to its private accumulators (diagonal and load entry in registers, off-diagonals in the
//             column acc[k * R + l] of shared memory, as in the row-gather kernel).
// Two tensor buffers alternate, so a chunk costs ONE barrier and the rows without records in a chunk go straight to the
// next evaluation.  A cell touching several tiles is evaluated once per tile (recompute factor ~1.6 at R = 256 on a
// Kuhn mesh instead of 4).  No atomics, no zero-fill; the cells of a tile are listed in ascending cell index, so every
// row sums its cells in mesh order: bitwise reproducible and independent of the tiling.
#include "common.cuh"
#include "p1_forms.cuh"

namespace phifem {
namespace {

// CTAs per SM of the tile kernels at R = 256 / 128 threads
constexpr int kTilesMinBlocks = 2;
constexpr int kTilesMinBlocks128 = 4;

// Whole element tensor of simplex X: K[i * NV + j] at out[(i * NV + j) * stride], b[i] at out[(NV * NV + i) * stride].
//   K_ij = |K|/((d+1)(d+2)) [ |g|^2 (1 + delta_ij) + a_i (P + p_j) + (P + p_i) a_j + G_i.G_j mu ] + 4 sigma h^2 |K| a_i a_j
//   b_i  = |K| d!/(d+3)! [ F P + sum f_k p_k + f_i (P + 2 p_i) + F p_i ] - 2 sigma h^2 |K| mean(f) a_i
// with g = grad(phi), a_j = g.G_j, P = sum p, mu = P^2 + sum p^2, F = sum f; every gradient is left scaled by det
// (G = R / det) so that one reciprocal serves the cell.
template <int D>
__device__ __forceinline__ void cell_tensor(const double (&X)[D + 1][D], const double (&p)[D + 1],
                                            const double (&fv)[D + 1], bool is_cut, double sigma,
                                            double* __restrict__ out, int stride) {
  constexpr int NV = D + 1;
  constexpr double dfact = D == 2 ? 2.0 : 6.0;
  double R[NV][D], det;
  simplex_cofactors<D>(X, R, det);
  const double inv = 1.0 / det;
  double gR[D];  // det * grad(phi)
#pragma unroll
  for (int d = 0; d < D; ++d) {
    double s = (p[1] - p[0]) * R[1][d];
#pragma unroll
    for (int k = 2; k < NV; ++k) s += (p[k] - p[0]) * R[k][d];
    gR[d] = s;
  }
  double aR[NV];  // det^2 * a_j
#pragma unroll
  for (int j = 0; j < NV; ++j) aR[j] = dot<D>(gR, R[j]);
  const double ggR = dot<D>(gR, gR);
  double P = p[0], S2 = p[0] * p[0], F = fv[0], FP = fv[0] * p[0];
#pragma unroll
  for (int k = 1; k < NV; ++k) {
    P += p[k];
    S2 += p[k] * p[k];
    F += fv[k];
    FP += fv[k] * p[k];
  }
  const double ainv = fabs(inv), adet = fabs(det);
  const double w = ainv * (1.0 / (dfact * (D + 1) * (D + 2)));
  const double wmu = w * (P * P + S2), wgg = w * ggR;
  double q[NV], wa[NV], sa[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    q[j] = P + p[j];
    wa[j] = w * aR[j];
    sa[j] = 0.0;
  }
  double sh2i = 0.0;  // sigma h_T^2 / det^2 on cut cells
  if (is_cut) {
    sh2i = sigma * diameter2<D>(X) * (inv * inv);
    const double sc = (4.0 / dfact) * sh2i * ainv;  // 4 sigma h^2 |K| / det^4
#pragma unroll
    for (int j = 0; j < NV; ++j) sa[j] = sc * aR[j];
  }
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int j = i; j < NV; ++j) {
      const double c = dot<D>(R[i], R[j]);
      double k = fma(c, wmu, i == j ? 2.0 * wgg : wgg);
      k = fma(wa[i], q[j], k);
      k = fma(q[i], wa[j], k);
      k = fma(sa[i], aR[j], k);
      out[(i * NV + j) * stride] = k;
      if (j != i) out[(j * NV + i) * stride] = k;
    }
  constexpr double fact_d3 = D == 2 ? 120.0 : 720.0;
  const double c3 = adet * (1.0 / fact_d3), base = F * P + FP;
  const double cs = adet * (2.0 / (dfact * NV)) * sh2i * F;
#pragma unroll
  for (int i = 0; i < NV; ++i)
    out[(NV * NV + i) * stride] = c3 * (base + fv[i] * (P + 2.0 * p[i]) + F * p[i]) - cs * aR[i];
}

// position of K_ij inside the packed symmetric tensor (i <= j: i * NV - i (i - 1) / 2 + j - i), 4 bits per (i, j)
template <int NV> __host__ __device__ constexpr uint64_t sym_lut() {
  uint64_t lut = 0;
  for (int i = 0; i < NV; ++i)
    for (int j = 0; j < NV; ++j) {
      const int a = i < j ? i : j, c = i < j ? j : i;
      lut |= (uint64_t)(a * NV - a * (a - 1) / 2 + c - a) << (4 * (i * 4 + j));
    }
  return lut;
}

__device__ __forceinline__ void cp_async4(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Software pipeline over the chunks of a tile: while a chunk's tensors are pulled, the vertex data of the NEXT chunk's
// cell is already on its way into registers, that chunk's records stream into shared memory with cp.async and the
// vertex ids of the chunk after it are being fetched -- the only global latency left on the critical path of a chunk is
// the barrier itself.
template <int D, int R>
__global__ void __launch_bounds__(R, R == 128 ? kTilesMinBlocks128 : kTilesMinBlocks) k_assemble_tiles_p1(
    const double* __restrict__ x, const double* __restrict__ phi, const double* __restrict__ f, double sigma,
    const int32_t* __restrict__ indptr, phifem_cell_tiles tl, int max_row_nnz, double* __restrict__ data,
    double* __restrict__ b) {
  constexpr int NV = D + 1, NS = NV * (NV + 1) / 2, NE = NS + NV;   // packed symmetric tensor + load vector
  constexpr uint64_t LUT = sym_lut<NV>();
  extern __shared__ double sm[];
  double* acc_s = sm;                                   // [max_row_nnz][R]
  double* buf_s = sm + (size_t)max_row_nnz * R;         // [2][NE][R]
  uint32_t* rec_s = reinterpret_cast<uint32_t*>(buf_s + 2 * NE * R);  // [2][NV * R]
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  const int64_t li = (int64_t)tile * R + tid;
  const bool has_row = li < tl.n_listed;
  int r = 0, start = 0, nnz = 0, dpos = 0;
  if (has_row) {
    r = __ldg(tl.rows + li);
    start = __ldg(indptr + r);
    nnz = __ldg(indptr + r + 1) - start;
    dpos = __ldg(tl.diag_pos + li);
  }
  double* acc = acc_s + tid;
  for (int k = 0; k < nnz; ++k) acc[k * R] = 0.0;
  double diag = 0.0, br = 0.0;
  const int c0 = __ldg(tl.chunk_ptr + tile), c1 = __ldg(tl.chunk_ptr + tile + 1);
  const int4* __restrict__ slots = reinterpret_cast<const int4*>(tl.slot_verts);
  const int4 none = make_int4(-1, 0, 0, 0);

  double X[NV][D], p[NV], fv[NV];
  auto gather = [&](const int4& sv) {  // issue the loads of a cell's vertex data (no use until the next evaluation)
    if (sv.x < 0) return;
    const int v[4] = {sv.x, sv.y & 0x7fffffff, sv.z, sv.w};
#pragma unroll
    for (int k = 0; k < NV; ++k) {
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = __ldg(x + (int64_t)v[k] * D + d);
      p[k] = __ldg(phi + v[k]);
      fv[k] = __ldg(f + v[k]);
    }
  };
  auto stream_records = [&](int c) {   // records of chunk c -> rec_s[c & 1] (asynchronous)
    const int rb = __ldg(tl.rec_base + c), nrec = __ldg(tl.rec_base + c + 1) - rb;
    uint32_t* dst = rec_s + ((c - c0) & 1) * (NV * R);
    for (int j = tid; j < nrec; j += R) cp_async4(dst + j, tl.rec + rb + j);
    cp_async_commit();
  };
  auto offsets = [&](int c, int& o0, int& o1) {
    const uint16_t* off = tl.rec_off + (int64_t)c * (R + 1);
    o0 = has_row ? (int)__ldg(off + tid) : 0;
    o1 = has_row ? (int)__ldg(off + tid + 1) : 0;
  };

  int4 sv = c0 < c1 ? __ldg(slots + (int64_t)c0 * R + tid) : none;           // cell evaluated in this chunk
  int4 sv1 = c0 + 1 < c1 ? __ldg(slots + (int64_t)(c0 + 1) * R + tid) : none;  // ... in the next one
  int o0 = 0, o1 = 0;
  if (c0 < c1) {
    stream_records(c0);
    offsets(c0, o0, o1);
    gather(sv);
  }
  for (int c = c0; c < c1; ++c) {
    const int sel = (c - c0) & 1;
    double* buf = buf_s + sel * (NE * R);
    const uint32_t* recs = rec_s + sel * (NV * R);
    if (sv.x >= 0) {   // evaluate: whole tensor of this thread's cell, packed symmetric, entry-major
      double out[NV * NV + NV];
      cell_tensor<D>(X, p, fv, sv.y < 0, sigma, out, 1);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
#pragma unroll
        for (int j = i; j < NV; ++j) buf[(int)((LUT >> (4 * (i * 4 + j))) & 0xf) * R + tid] = out[i * NV + j];
        buf[(NS + i) * R + tid] = out[NV * NV + i];
      }
    }
    // next chunk: vertex data into the registers just consumed, vertex ids of the chunk after it, record offsets
    sv = sv1;
    gather(sv);
    sv1 = c + 2 < c1 ? __ldg(slots + (int64_t)(c + 2) * R + tid) : none;
    const int q0 = o0, q1 = o1;
    if (c + 1 < c1) offsets(c + 1, o0, o1);
    cp_async_wait_all();   // this chunk's records (issued one chunk ago) have landed
    __syncthreads();
    if (c + 1 < c1) stream_records(c + 1);   // every thread is past the pull of chunk c - 1: its record buffer is free
    // pull: this row's records of the chunk; the parked values of record k + 1 are requested before record k is added
    int k = q0;
    uint32_t w = 0;
    double t[NV + 1];
    auto fetch = [&](int kk, uint32_t& ww, double (&tt)[NV + 1]) {
      ww = recs[kk];
      const int s = ww & 0xff, i = (ww >> 8) & 3;
      const double* src = buf + s;
#pragma unroll
      for (int j = 0; j < NV; ++j) tt[j] = src[(int)((LUT >> (4 * (i * 4 + j))) & 0xf) * R];
      tt[NV] = src[(NS + i) * R];
    };
    if (k < q1) fetch(k, w, t);
    while (k < q1) {
      const uint32_t wc = w;
      double tc[NV + 1];
#pragma unroll
      for (int j = 0; j <= NV; ++j) tc[j] = t[j];
      if (++k < q1) fetch(k, w, t);
      const int i = (wc >> 8) & 3;
      br += tc[NV];
      double a[D];
      double* dst[D];
#pragma unroll
      for (int m = 0; m < D; ++m) {   // the D other vertices of a cell sit at D distinct positions of the row
        dst[m] = acc + ((wc >> (10 + 7 * m)) & 0x7f) * R;
        a[m] = *dst[m];
      }
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        if (j == i) diag += tc[j];
      }
#pragma unroll
      for (int m = 0; m < D; ++m) {
        const int j = m + (m >= i);
        double v = tc[0];
#pragma unroll
        for (int jj = 1; jj < NV; ++jj)
          if (jj == j) v = tc[jj];
        *dst[m] = a[m] + v;
      }
    }
  }
  if (has_row) {
    acc[dpos * R] += diag;
    for (int k = 0; k < nnz; ++k) data[start + k] = acc[k * R];
    b[r] = br;
  }
}

// Cell-once PUSH form (plan option cell_pass="push"): same tiles, same cell list, but no parked tensors and no pull.
// The thread that evaluated a cell adds the rows of the tensor that belong to the tile's own rows straight into the
// tile's accumulators in shared memory -- acc[pos * R + l] for row l of the tile, its diagonal in dacc[l], its load
// entry in bacc[l].  A tile's cells share vertices, so the updates are shared-memory fp64 atomics (a compare-and-swap
// loop on sm_100: conflicts are rare, the loop usually runs once); nothing orders them, so the sum of a row is NOT in
// mesh order: results agree with the row-gather pass to rounding, not bit for bit.  No barrier between the cells of a
// tile: a thread walks slots tid, tid + R, ... with the next slot's vertex data in flight while it pushes.
//   push[q][i] (one word per cell-local vertex i of slot q): bit 8 = the vertex's row belongs to this tile,
//   bits 0-7 = its index l in the tile, 7 bits from bit 10 + 7 m = position inside row l's column list of the cell's
//   m-th OTHER vertex (ascending cell-local order).
template <int D, int R>
__global__ void __launch_bounds__(R, R == 128 ? kTilesMinBlocks128 : kTilesMinBlocks) k_assemble_push_p1(
    const double* __restrict__ x, const double* __restrict__ phi, const double* __restrict__ f, double sigma,
    const int32_t* __restrict__ indptr, phifem_cell_tiles tl, int max_row_nnz, double* __restrict__ data,
    double* __restrict__ b) {
  constexpr int NV = D + 1;
  extern __shared__ double sm[];
  double* acc_s = sm;                                   // [max_row_nnz][R]
  double* dacc = sm + (size_t)max_row_nnz * R;          // [R] diagonal entries
  double* bacc = dacc + R;                              // [R] load vector
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  const int64_t li = (int64_t)tile * R + tid;
  const bool has_row = li < tl.n_listed;
  int r = 0, start = 0, nnz = 0, dpos = 0;
  if (has_row) {
    r = __ldg(tl.rows + li);
    start = __ldg(indptr + r);
    nnz = __ldg(indptr + r + 1) - start;
    dpos = __ldg(tl.diag_pos + li);
  }
  for (int k = 0; k < nnz; ++k) acc_s[k * R + tid] = 0.0;
  dacc[tid] = 0.0;
  bacc[tid] = 0.0;
  const int64_t q0 = (int64_t)__ldg(tl.chunk_ptr + tile) * R, q1 = (int64_t)__ldg(tl.chunk_ptr + tile + 1) * R;
  const int4* __restrict__ slots = reinterpret_cast<const int4*>(tl.slot_verts);
  const uint4* __restrict__ pushw = reinterpret_cast<const uint4*>(tl.push);
  const int4 none = make_int4(-1, 0, 0, 0);

  double X[NV][D], p[NV], fv[NV];
  auto gather = [&](const int4& sv) {
    if (sv.x < 0) return;
    const int v[4] = {sv.x, sv.y & 0x7fffffff, sv.z, sv.w};
#pragma unroll
    for (int k = 0; k < NV; ++k) {
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = __ldg(x + (int64_t)v[k] * D + d);
      p[k] = __ldg(phi + v[k]);
      fv[k] = __ldg(f + v[k]);
    }
  };
  int64_t q = q0 + tid;
  int4 sv = q < q1 ? __ldg(slots + q) : none;
  int4 sv1 = q + R < q1 ? __ldg(slots + q + R) : none;
  uint4 pw = q < q1 ? __ldg(pushw + q) : make_uint4(0, 0, 0, 0);
  gather(sv);
  __syncthreads();   // accumulators are zero
  for (; q < q1; q += R) {
    const bool live = sv.x >= 0;
    const bool is_cut = sv.y < 0;
    double out[NV * NV + NV];
    if (live) cell_tensor<D>(X, p, fv, is_cut, sigma, out, 1);
    const uint4 pc = pw;
    // next slot: vertex data into the registers just consumed, ids of the slot after it, its push words
    sv = sv1;
    gather(sv);
    sv1 = q + 2 * R < q1 ? __ldg(slots + q + 2 * R) : none;
    if (q + R < q1) pw = __ldg(pushw + q + R);
    if (live) {
      const uint32_t w4[4] = {pc.x, pc.y, pc.z, pc.w};
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const uint32_t w = w4[i];
        if (w & 0x100u) {
          const int l = w & 0xff;
          double* dst[D + 2];
          double v[D + 2];
          dst[0] = dacc + l;
          v[0] = out[i * NV + i];
          dst[1] = bacc + l;
          v[1] = out[NV * NV + i];
#pragma unroll
          for (int m = 0; m < D; ++m) {
            const int j = m + (m >= i);
            dst[2 + m] = acc_s + ((w >> (10 + 7 * m)) & 0x7f) * R + l;
            v[2 + m] = out[i * NV + j];
          }
          // the D + 2 updates of a row as ONE batch: loads, sums, compare-and-swaps issued back to back (a
          // compiler-generated atomicAdd is a dependent LDS -> DADD -> CAS chain each); the rare loser retries alone.
          // Plain atomicAdd loops measured 2.582 against 2.846 ms at R = 256 (DESIGN.md §4, K2'').
          unsigned long long seen[D + 2], want[D + 2];
#pragma unroll
          for (int e = 0; e < D + 2; ++e) seen[e] = *reinterpret_cast<volatile unsigned long long*>(dst[e]);
#pragma unroll
          for (int e = 0; e < D + 2; ++e) want[e] = __double_as_longlong(__longlong_as_double(seen[e]) + v[e]);
#pragma unroll
          for (int e = 0; e < D + 2; ++e)
            want[e] = atomicCAS(reinterpret_cast<unsigned long long*>(dst[e]), seen[e], want[e]);
#pragma unroll
          for (int e = 0; e < D + 2; ++e)
            if (want[e] != seen[e]) atomicAdd(dst[e], v[e]);
        }
      }
    }
  }
  __syncthreads();
  if (has_row) {
    double* acc = acc_s + tid;
    acc[dpos * R] += dacc[tid];
    for (int k = 0; k < nnz; ++k) data[start + k] = acc[k * R];
    b[r] = bacc[tid];
  }
}

template <int D, int R>
cudaError_t launch_push(const phifem_mesh* mesh, const double* phi, const double* f, double sigma, const int32_t* indptr,
                        const phifem_cell_tiles& tl, int max_row_nnz, double* data, double* b, cudaStream_t st) {
  const size_t smem = ((size_t)max_row_nnz * R + 2 * R) * sizeof(double);
  auto kernel = k_assemble_push_p1<D, R>;
  cudaError_t err = cudaSuccess;
  if (smem > 48 * 1024) err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  kernel<<<(unsigned)tl.n_tiles, R, smem, st>>>(mesh->x, phi, f, sigma, indptr, tl, max_row_nnz, data, b);
  return cudaGetLastError();
}

template <int D, int R>
cudaError_t launch(const phifem_mesh* mesh, const double* phi, const double* f, double sigma, const int32_t* indptr,
                   const phifem_cell_tiles& tl, int max_row_nnz, double* data, double* b, cudaStream_t st) {
  constexpr int NV = D + 1, NE = NV * (NV + 1) / 2 + NV;
  const size_t smem = ((size_t)max_row_nnz * R + 2 * NE * R) * sizeof(double) + 2 * NV * R * sizeof(uint32_t);
  auto kernel = k_assemble_tiles_p1<D, R>;
  cudaError_t err = cudaSuccess;
  if (smem > 48 * 1024) err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  kernel<<<(unsigned)tl.n_tiles, R, smem, st>>>(mesh->x, phi, f, sigma, indptr, tl, max_row_nnz, data, b);
  return cudaGetLastError();
}

}  // namespace

// Cell pass over the tiles of `tl`; called by phifem_assemble_rows_p1 (csrc/assemble_rows.cu) in place of the row-gather
// cell pass when the plan carries tiles.  Returns cudaErrorInvalidValue for a malformed plan.
cudaError_t launch_cell_tiles_p1(const phifem_mesh* mesh, const double* phi, const double* f, double sigma,
                                 const int32_t* indptr, const phifem_cell_tiles* tl, int max_row_nnz, double* data,
                                 double* b, cudaStream_t st) {
  if (tl->n_tiles <= 0) return cudaSuccess;
  if (!(tl->rows && tl->diag_pos && tl->chunk_ptr && tl->slot_verts &&
        (tl->push || (tl->rec_base && tl->rec_off && tl->rec))) ||
      max_row_nnz > 128 || (tl->rows_per_tile != 128 && tl->rows_per_tile != 256))
    return cudaErrorInvalidValue;
  const bool tri = mesh->cell_type == PHIFEM_TRIANGLE;
  if (tl->push) {   // push form: atomics into the tile's shared-memory accumulators
    if (tl->rows_per_tile == 128)
      return tri ? launch_push<2, 128>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st)
                 : launch_push<3, 128>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st);
    return tri ? launch_push<2, 256>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st)
               : launch_push<3, 256>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st);
  }
  if (tl->rows_per_tile == 128)
    return tri ? launch<2, 128>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st)
               : launch<3, 128>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st);
  return tri ? launch<2, 256>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st)
             : launch<3, 256>(mesh, phi, f, sigma, indptr, *tl, max_row_nnz, data, b, st);
}

}  // namespace phifem
