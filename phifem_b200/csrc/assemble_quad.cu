// The Neumann phi-FEM operator of assemble_pk.cu on QUADRILATERALS, the cell type of the reference demo
// demo/neumann/square/main.py:103-158: mixed space (u, y, p) in Q1 x Q1^2 x DG0, Q1 or Q2 level set.
//
// The cell map x(xi, eta) = sum_a N_a(xi, eta) x_a is bilinear (vertices in tensor order v0 = (0,0), v1 = (1,0),
// v2 = (0,1), v3 = (1,1)), so nothing is affine: J, |det J| and J^-T are evaluated at every quadrature point, and even
// the u-u block of the interior cells is integrated by the cell rule (no closed form).  The rules are host tables
// (phifem_quadrature): cell points in reference coordinates (xi, eta), weights summing to 1 (the Gauss product rule
// of phifem_b200/quadrature.py rules_for_neumann_quad); facet points on the segment, weights summing to 1.
// Convex cells of either orientation (|det J|); a non-convex quadrilateral is outside the method and not checked.
//
// The entry points stay phifem_assemble_neumann_{cells,boundary,ghost} (assemble_pk.cu): they validate the arguments
// and call the launchers at the end of this file when mesh->cell_type == PHIFEM_QUADRILATERAL.
//
// The same file holds the strong-Dirichlet operator (demo/strong-dirichlet/flower/main.py:104-128) for a Q1 trial /
// test space and a Q1 or Q2 level set, behind phifem_assemble_{cells,boundary,ghost}_pk; its Hessian terms need the
// second derivative of the bilinear map (see k_quad_cells_strong).
#include "common.cuh"
#include "pk_common.cuh"

namespace phifem {
namespace quad {
using pk::dotd;
using pk::kBlockPk;
using pk::kMaxQuadPoints;

constexpr int NV = 4;            // vertices of a quadrilateral
constexpr int NM = NV * 3 + 1;   // cell-local mixed dofs [u x4, y node-major x8, p] = 13

// tensor-order reference vertex k = (k & 1, k >> 1); local facets (0,1), (0,2), (1,3), (2,3)
__host__ __device__ constexpr int facet_vertex(int f, int s) { return CellTraits<PHIFEM_QUADRILATERAL>::fv(f, s); }

// Lagrange Q_K on the GLL nodes of fem._GLL ({0, 1} / {0, 1/2, 1}), dolfinx-local order (vertices, the 4 edges in
// LOCAL_EDGES["quadrilateral"] order, interior): dof k is the tensor product L_ix(xi) L_iy(eta) of the 1-D node indices
template <int K>
__host__ __device__ constexpr int tensor_index(int k, int axis) {
  if (K == 1) {
    return axis == 0 ? (k & 1) : (k >> 1);
  } else {
    constexpr int t[9][2] = {{0, 0}, {2, 0}, {0, 2}, {2, 2}, {1, 0}, {0, 1}, {2, 1}, {1, 2}, {1, 1}};
    return t[k][axis];
  }
}

template <int K>
struct QSpace {
  static constexpr int ND = (K + 1) * (K + 1);
};

// 1-D Lagrange basis on the nodes {0, 1} (K = 1) or {0, 1/2, 1} (K = 2): values and derivatives at t
template <int K>
__device__ __forceinline__ void lagrange_1d(double t, double (&L)[K + 1], double (&dL)[K + 1]) {
  if constexpr (K == 1) {
    L[0] = 1.0 - t;  L[1] = t;
    dL[0] = -1.0;    dL[1] = 1.0;
  } else {
    L[0] = (1.0 - t) * (1.0 - 2.0 * t);  L[1] = 4.0 * t * (1.0 - t);  L[2] = t * (2.0 * t - 1.0);
    dL[0] = 4.0 * t - 3.0;                dL[1] = 4.0 - 8.0 * t;       dL[2] = 4.0 * t - 1.0;
  }
}

// vertex coordinates of one cell and h^2 (UFL CellDiameter of a degree-1 coordinate element: the largest of the
// 6 vertex-pair distances)
struct Cell {
  double X[NV][2], h2;
};

__device__ __forceinline__ void load_cell(const phifem_mesh& m, int64_t c, Cell& g) {
  const int4 q = __ldg(reinterpret_cast<const int4*>(m.cells) + c);
  const int v[NV] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const double2 p = __ldg(reinterpret_cast<const double2*>(m.x) + v[k]);
    g.X[k][0] = p.x;
    g.X[k][1] = p.y;
  }
  double h2 = 0.0;
#pragma unroll
  for (int a = 0; a < NV; ++a)
#pragma unroll
    for (int b = a + 1; b < NV; ++b) {
      const double dx = g.X[a][0] - g.X[b][0], dy = g.X[a][1] - g.X[b][1];
      h2 = fmax(h2, dx * dx + dy * dy);
    }
  g.h2 = h2;
}

// at reference point (xi, eta): Q1 values N, physical gradients G = J^-T grad_ref N, Jit = J^-T; returns |det J|
__device__ __forceinline__ double map_point(const Cell& g, double xi, double eta, double (&N)[NV], double (&G)[NV][2],
                                            double (&Jit)[2][2]) {
  const double dxi[NV] = {-(1.0 - eta), 1.0 - eta, -eta, eta};
  const double deta[NV] = {-(1.0 - xi), -xi, 1.0 - xi, xi};
  N[0] = (1.0 - xi) * (1.0 - eta);
  N[1] = xi * (1.0 - eta);
  N[2] = (1.0 - xi) * eta;
  N[3] = xi * eta;
  double J00 = 0.0, J01 = 0.0, J10 = 0.0, J11 = 0.0;   // J[r][c] = d x_r / d ref_c
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    J00 += g.X[k][0] * dxi[k];
    J01 += g.X[k][0] * deta[k];
    J10 += g.X[k][1] * dxi[k];
    J11 += g.X[k][1] * deta[k];
  }
  const double det = J00 * J11 - J01 * J10;
  const double inv = 1.0 / det;
  Jit[0][0] = J11 * inv;
  Jit[0][1] = -J10 * inv;
  Jit[1][0] = -J01 * inv;
  Jit[1][1] = J00 * inv;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    G[k][0] = Jit[0][0] * dxi[k] + Jit[0][1] * deta[k];
    G[k][1] = Jit[1][0] * dxi[k] + Jit[1][1] * deta[k];
  }
  return fabs(det);
}

// phi_h and grad(phi_h) of a Q_K level set at (xi, eta)
template <int K>
__device__ __forceinline__ void eval_phi(double xi, double eta, const double (&Jit)[2][2],
                                         const double (&pc)[QSpace<K>::ND], double& ph, double (&gph)[2]) {
  double Lx[K + 1], dLx[K + 1], Ly[K + 1], dLy[K + 1];
  lagrange_1d<K>(xi, Lx, dLx);
  lagrange_1d<K>(eta, Ly, dLy);
  double gr0 = 0.0, gr1 = 0.0;   // reference gradient
  ph = 0.0;
#pragma unroll
  for (int k = 0; k < QSpace<K>::ND; ++k) {
    const int ix = tensor_index<K>(k, 0), iy = tensor_index<K>(k, 1);
    ph += pc[k] * Lx[ix] * Ly[iy];
    gr0 += pc[k] * dLx[ix] * Ly[iy];
    gr1 += pc[k] * Lx[ix] * dLy[iy];
  }
  gph[0] = Jit[0][0] * gr0 + Jit[0][1] * gr1;
  gph[1] = Jit[1][0] * gr0 + Jit[1][1] * gr1;
}

template <int K>
__device__ __forceinline__ void load_phi(const phifem_mesh& m, const phifem_pk_space& sp,
                                         const double* __restrict__ phi, int64_t c, double (&pc)[QSpace<K>::ND]) {
  constexpr int ND = QSpace<K>::ND;
  const int32_t* dm = sp.dofmap ? sp.dofmap + c * ND : m.cells + c * ND;   // NULL: Q1 with vertex dofs
#pragma unroll
  for (int k = 0; k < ND; ++k) pc[k] = __ldg(phi + __ldg(dm + k));
}

// the tuple (u, grad u, s1, s2, s3) of mixed basis function mi at a point: s1 = y + grad u, s2 = div y + u,
// s3 = y.grad phi - kappa |grad phi| u + h^-1 p phi  (as neumann_basis of assemble_pk.cu, with 4 vertices)
__device__ __forceinline__ void mixed_basis(int mi, const double (&N)[NV], const double (&G)[NV][2],
                                            const double (&gph)[2], double ph_over_h, double kappa_ngp, double& U,
                                            double (&GU)[2], double (&S1)[2], double& S2, double& S3) {
  U = S2 = S3 = 0.0;
  GU[0] = GU[1] = S1[0] = S1[1] = 0.0;
  if (mi == NM - 1) {   // p: piecewise constant
    S3 = ph_over_h;
    return;
  }
  const bool is_u = mi < NV;
  const int node = is_u ? mi : (mi - NV) >> 1, comp = is_u ? -1 : (mi - NV) & 1;
  double nj = 0.0, Gj[2] = {0.0, 0.0};
#pragma unroll
  for (int k = 0; k < NV; ++k)
    if (k == node) {
      nj = N[k];
      Gj[0] = G[k][0];
      Gj[1] = G[k][1];
    }
  if (is_u) {
    U = S2 = nj;
    S3 = -kappa_ngp * nj;
    GU[0] = S1[0] = Gj[0];
    GU[1] = S1[1] = Gj[1];
  } else {
#pragma unroll
    for (int d = 0; d < 2; ++d)
      if (d == comp) {
        S1[d] = nj;
        S2 = Gj[d];
        S3 = nj * gph[d];
      }
  }
}

// Interior cells (tag 1): int grad u.grad v + u v and int f v by the cell rule; one thread per (active cell, u test
// dof a); cut cells are left to k_quad_cells_neumann.
__global__ void __launch_bounds__(kBlockPk) k_quad_interior_neumann(
    phifem_mesh m, const double* __restrict__ qpt_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ f, const int8_t* __restrict__ ctags, const int32_t* __restrict__ active,
    int64_t n_active, const int32_t* __restrict__ slots, const int32_t* __restrict__ mixed_dofmap,
    double* __restrict__ data, double* __restrict__ b) {
  __shared__ double qpt[kMaxQuadPoints * 2], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * 2; i += blockDim.x) qpt[i] = qpt_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_active * NV) return;
  const int64_t e = t / NV;
  const int a = (int)(t - e * NV);
  const int64_t c = __ldg(active + e);
  if (ctags[c] == 2) return;
  Cell g;
  load_cell(m, c, g);
  double fc[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) fc[k] = __ldg(f + __ldg(m.cells + c * NV + k));
  double A[NV], bv = 0.0;
#pragma unroll
  for (int j = 0; j < NV; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double N[NV], G[NV][2], Jit[2][2];
    const double w = qw[q] * map_point(g, qpt[2 * q], qpt[2 * q + 1], N, G, Jit);
    double fq = 0.0, na = N[0], ga0 = G[0][0], ga1 = G[0][1];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      fq += fc[k] * N[k];
      if (k == a) {
        na = N[k];
        ga0 = G[k][0];
        ga1 = G[k][1];
      }
    }
    bv += w * fq * na;
#pragma unroll
    for (int j = 0; j < NV; ++j) A[j] += w * (ga0 * G[j][0] + ga1 * G[j][1] + na * N[j]);
  }
  atomicAdd(b + __ldg(mixed_dofmap + c * NM + a), bv);
#pragma unroll
  for (int j = 0; j < NV; ++j) atomicAdd(data + __ldg(slots + (int64_t)(a * NM + j) * n_active + e), A[j]);
}

// Cut cells (tag 2): all 13 x 13 entries and the 13 load entries; one thread per (cut cell, mixed test dof a).
template <int KP>
__global__ void __launch_bounds__(kBlockPk) k_quad_cells_neumann(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qpt_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const double* __restrict__ f, const double* __restrict__ un,
    const int32_t* __restrict__ active, int64_t n_active, const int32_t* __restrict__ cut_positions, int64_t n_cut,
    const int32_t* __restrict__ slots, const int32_t* __restrict__ mixed_dofmap, double gamma, double kappa,
    double* __restrict__ data, double* __restrict__ b) {
  constexpr int NDP = QSpace<KP>::ND;
  __shared__ double qpt[kMaxQuadPoints * 2], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * 2; i += blockDim.x) qpt[i] = qpt_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cut * NM) return;
  const int64_t ec = t / NM;
  const int a = (int)(t - ec * NM);
  const int64_t e = __ldg(cut_positions + ec);
  const int64_t c = __ldg(active + e);
  Cell g;
  load_cell(m, c, g);
  double pc[NDP], fc[NV], uc[NV];
  load_phi<KP>(m, sp, phi, c, pc);
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int v = __ldg(m.cells + c * NV + k);
    fc[k] = __ldg(f + v);
    uc[k] = __ldg(un + v);
  }
  const double rh = 1.0 / sqrt(g.h2), rh2 = 1.0 / g.h2;
  double A[NM], bv = 0.0;
#pragma unroll
  for (int j = 0; j < NM; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double xi = qpt[2 * q], eta = qpt[2 * q + 1];
    double N[NV], G[NV][2], Jit[2][2];
    const double w = qw[q] * map_point(g, xi, eta, N, G, Jit);
    double ph, gph[2];
    eval_phi<KP>(xi, eta, Jit, pc, ph, gph);
    double fq = 0.0, uq = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      fq += fc[k] * N[k];
      uq += uc[k] * N[k];
    }
    const double ngp = sqrt(gph[0] * gph[0] + gph[1] * gph[1]);
    double Ua, GUa[2], S1a[2], S2a, S3a;
    mixed_basis(a, N, G, gph, ph * rh, kappa * ngp, Ua, GUa, S1a, S2a, S3a);
    bv += w * (fq * Ua + gamma * (fq * S2a - rh2 * uq * ngp * S3a));
#pragma unroll
    for (int bb = 0; bb < NM; ++bb) {
      double Ub, GUb[2], S1b[2], S2b, S3b;
      mixed_basis(bb, N, G, gph, ph * rh, kappa * ngp, Ub, GUb, S1b, S2b, S3b);
      A[bb] += w * (dotd<2>(GUa, GUb) + Ua * Ub + gamma * (dotd<2>(S1a, S1b) + S2a * S2b + rh2 * S3a * S3b));
    }
  }
  atomicAdd(b + __ldg(mixed_dofmap + c * NM + a), bv);
#pragma unroll
  for (int bb = 0; bb < NM; ++bb) atomicAdd(data + __ldg(slots + (int64_t)(a * NM + bb) * n_active + e), A[bb]);
}

// outward unit normal and length of local facet o (straight edge: constant normal); the side of the edge's line the
// vertex centroid lies on is the inside of a convex cell
__device__ __forceinline__ void edge_normal(const Cell& g, int o, double (&n)[2], double& len) {
  const int la = facet_vertex(o, 0), lb = facet_vertex(o, 1);
  double xa[2] = {g.X[0][0], g.X[0][1]}, xb[2] = {g.X[0][0], g.X[0][1]};
#pragma unroll
  for (int k = 1; k < NV; ++k) {
    if (k == la) { xa[0] = g.X[k][0]; xa[1] = g.X[k][1]; }
    if (k == lb) { xb[0] = g.X[k][0]; xb[1] = g.X[k][1]; }
  }
  const double tx = xb[0] - xa[0], ty = xb[1] - xa[1];
  len = sqrt(tx * tx + ty * ty);
  double nx = ty / len, ny = -tx / len;
  const double cx = 0.25 * (g.X[0][0] + g.X[1][0] + g.X[2][0] + g.X[3][0]);
  const double cy = 0.25 * (g.X[0][1] + g.X[1][1] + g.X[2][1] + g.X[3][1]);
  if (nx * (xa[0] - cx) + ny * (xa[1] - cy) < 0.0) {
    nx = -nx;
    ny = -ny;
  }
  n[0] = nx;
  n[1] = ny;
}

// int_{ds(100)} (y.n) v on (cell, local facet) pairs: Q1 restricted to the straight edge is linear, so the entry
// (u_i, y_(j,c)) is n_c |F| (1 + delta_ij) / 6 for i, j the edge's two vertices.  One thread per (entity, u test dof i).
__global__ void __launch_bounds__(kBlockPk) k_quad_boundary_neumann(
    phifem_mesh m, const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ slots,
    double* __restrict__ data) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * NV) return;
  const int64_t e = t / NV;
  const int i = (int)(t - e * NV);
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  const int la = facet_vertex(o, 0), lb = facet_vertex(o, 1);
  if (i != la && i != lb) return;   // v_i vanishes on the edge
  Cell g;
  load_cell(m, c, g);
  double n[2], len;
  edge_normal(g, o, n, len);
  const double cF = len * (1.0 / 6.0);
  for (int s = 0; s < 2; ++s) {
    const int j = s == 0 ? la : lb;
    const double mij = cF * (i == j ? 2.0 : 1.0);
#pragma unroll
    for (int cc = 0; cc < 2; ++cc)
      atomicAdd(data + __ldg(slots + (e * NM + i) * NM + NV + j * 2 + cc), n[cc] * mij);
  }
}

// sigma avg(h) int_F [grad u.n][grad v.n] over interior facets, into the (2 NM)^2 macro slots [mixed dofs of cell +
// (f2c[f][0]), of cell -].  The facet parameter runs from the edge's lower-global-id vertex to the higher one and is
// mapped into each side's reference coordinates, so that a quadrature point is the same physical point from both
// cells.  One thread per (facet, u dof a of either side: a / 4 = side).
__global__ void __launch_bounds__(kBlockPk) k_quad_ghost_neumann(
    phifem_mesh m, const double* __restrict__ qfp_g, const double* __restrict__ qw_g, int nq,
    const int32_t* __restrict__ facets, int64_t n_facets, const int32_t* __restrict__ slots, double sigma,
    double* __restrict__ data) {
  constexpr int NU = 2 * NV;
  __shared__ double qt[kMaxQuadPoints], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) {
    qt[i] = qfp_g[2 * i + 1];   // segment point (1 - t, t): the parameter t
    qw[i] = qw_g[i];
  }
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets * NU) return;
  const int64_t e = t / NU;
  const int a = (int)(t - e * NU);
  const int32_t fct = __ldg(facets + e);
  const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
  Cell g[2];
  double n[2][2], len = 0.0, r0[2][2], r1[2][2];   // per side: normal, reference end points of the parameter
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int64_t c = s == 0 ? cc.x : cc.y;
    load_cell(m, c, g[s]);
    int o = 0;
#pragma unroll
    for (int k = 0; k < NV; ++k)
      if (__ldg(m.c2f + c * NV + k) == fct) o = k;
    int la = facet_vertex(o, 0), lb = facet_vertex(o, 1);
    if (__ldg(m.cells + c * NV + la) > __ldg(m.cells + c * NV + lb)) {
      const int tmp = la;
      la = lb;
      lb = tmp;
    }
    r0[s][0] = la & 1; r0[s][1] = la >> 1;
    r1[s][0] = lb & 1; r1[s][1] = lb >> 1;
    double l;
    edge_normal(g[s], o, n[s], l);
    if (s == 0) len = l;
  }
  const double coef = sigma * 0.5 * (sqrt(g[0].h2) + sqrt(g[1].h2)) * len;
  double E[NU];
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) E[bb] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double tq = qt[q];
    double J[NU];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      double N[NV], G[NV][2], Jit[2][2];
      map_point(g[s], (1.0 - tq) * r0[s][0] + tq * r1[s][0], (1.0 - tq) * r0[s][1] + tq * r1[s][1], N, G, Jit);
#pragma unroll
      for (int k = 0; k < NV; ++k) J[s * NV + k] = G[k][0] * n[s][0] + G[k][1] * n[s][1];
    }
    const double wa = qw[q] * coef * pk::pick<NU>(J, a);
#pragma unroll
    for (int bb = 0; bb < NU; ++bb) E[bb] += wa * J[bb];
  }
  const int ma = (a / NV) * NM + (a % NV);
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) {
    const int mb = (bb / NV) * NM + (bb % NV);
    atomicAdd(data + __ldg(slots + (e * 2 * NM + ma) * 2 * NM + mb), E[bb]);
  }
}

// ==== strong-Dirichlet phi-FEM operator (reference demo/strong-dirichlet/flower/main.py:104-128) on Q1 =============
//   a = int_{dx(1,2)} grad(phi w).grad(phi v) - int_{ds(100)} (grad(phi w).n) phi v
//       + sigma int_{dS(2,3)} avg(h) [grad(phi w).n][grad(phi v).n] + sigma h^2 int_{dx(2)} lap(phi w) lap(phi v)
//   L = int_{dx(1,2)} f phi v - sigma h^2 int_{dx(2)} f lap(phi v)
// The physical Hessian on the bilinear cell: with K = J^-1 and c = d^2 x / dxi deta = X0 - X1 - X2 + X3 (the map's only
// second derivative), H u = K^T (H_ref u - (c.grad u) E) K, E = [[0, 1], [1, 0]].  Only its trace is needed:
// lap u = M00 P00 + 2 M01 P01 + M11 P11 with M = H_ref u - (c.grad u) E and P = K K^T.

// 1-D Lagrange basis of lagrange_1d with second derivatives
template <int K>
__device__ __forceinline__ void lagrange_1d_d2(double t, double (&L)[K + 1], double (&dL)[K + 1],
                                               double (&d2L)[K + 1]) {
  lagrange_1d<K>(t, L, dL);
  if constexpr (K == 1) {
    d2L[0] = d2L[1] = 0.0;
  } else {
    d2L[0] = 4.0;  d2L[1] = -8.0;  d2L[2] = 4.0;
  }
}

// eval_phi with the reference Hessian hr = (phi_xixi, phi_xieta, phi_etaeta)
template <int K>
__device__ __forceinline__ void eval_phi_hess(double xi, double eta, const double (&Jit)[2][2],
                                              const double (&pc)[QSpace<K>::ND], double& ph, double (&gph)[2],
                                              double (&hr)[3]) {
  double Lx[K + 1], dLx[K + 1], d2Lx[K + 1], Ly[K + 1], dLy[K + 1], d2Ly[K + 1];
  lagrange_1d_d2<K>(xi, Lx, dLx, d2Lx);
  lagrange_1d_d2<K>(eta, Ly, dLy, d2Ly);
  double gr0 = 0.0, gr1 = 0.0;
  ph = hr[0] = hr[1] = hr[2] = 0.0;
#pragma unroll
  for (int k = 0; k < QSpace<K>::ND; ++k) {
    const int ix = tensor_index<K>(k, 0), iy = tensor_index<K>(k, 1);
    ph += pc[k] * Lx[ix] * Ly[iy];
    gr0 += pc[k] * dLx[ix] * Ly[iy];
    gr1 += pc[k] * Lx[ix] * dLy[iy];
    hr[1] += pc[k] * dLx[ix] * dLy[iy];
    if (K == 2) {
      hr[0] += pc[k] * d2Lx[ix] * Ly[iy];
      hr[2] += pc[k] * Lx[ix] * d2Ly[iy];
    }
  }
  gph[0] = Jit[0][0] * gr0 + Jit[0][1] * gr1;
  gph[1] = Jit[1][0] * gr0 + Jit[1][1] * gr1;
}

// Cells of dx(1,2): row a of the 4 x 4 element tensor and b_a, the Hessian terms on cut cells only.  One thread per
// (active cell, test dof a); slots entry-major ([16, n_active]).
template <int KP>
__global__ void __launch_bounds__(kBlockPk) k_quad_cells_strong(
    phifem_mesh m, phifem_pk_space sw, phifem_pk_space sp, const double* __restrict__ qpt_g,
    const double* __restrict__ qw_g, int nq, const double* __restrict__ phi, const double* __restrict__ f,
    const int8_t* __restrict__ ctags, const int32_t* __restrict__ active, int64_t n_active,
    const int32_t* __restrict__ slots, double sigma, double* __restrict__ data, double* __restrict__ b) {
  constexpr int NDP = QSpace<KP>::ND;
  __shared__ double qpt[kMaxQuadPoints * 2], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * 2; i += blockDim.x) qpt[i] = qpt_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_active * NV) return;
  const int64_t e = t / NV;
  const int a = (int)(t - e * NV);
  const int64_t c = __ldg(active + e);
  Cell g;
  load_cell(m, c, g);
  double pc[NDP], fc[NV];
  load_phi<KP>(m, sp, phi, c, pc);
  const int32_t* dm = sw.dofmap ? sw.dofmap + c * NV : m.cells + c * NV;
#pragma unroll
  for (int k = 0; k < NV; ++k) fc[k] = __ldg(f + __ldg(dm + k));
  const bool cut = ctags[c] == 2;
  const double sh2 = sigma * g.h2;
  const double c0 = g.X[0][0] - g.X[1][0] - g.X[2][0] + g.X[3][0];   // c = d^2 x / dxi deta
  const double c1 = g.X[0][1] - g.X[1][1] - g.X[2][1] + g.X[3][1];
  const double sa = (a == 0 || a == 3) ? 1.0 : -1.0;                // H_ref psi_a = s_a E
  double A[NV], bv = 0.0;
#pragma unroll
  for (int j = 0; j < NV; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double xi = qpt[2 * q], eta = qpt[2 * q + 1];
    double N[NV], G[NV][2], Jit[2][2];
    const double w = qw[q] * map_point(g, xi, eta, N, G, Jit);
    double ph, gph[2], hr[3];
    eval_phi_hess<KP>(xi, eta, Jit, pc, ph, gph, hr);
    double fq = 0.0, na = N[0], ga[2] = {G[0][0], G[0][1]};
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      fq += fc[k] * N[k];
      if (k == a) {
        na = N[k];
        ga[0] = G[k][0];
        ga[1] = G[k][1];
      }
    }
    double gu[NV][2];
#pragma unroll
    for (int j = 0; j < NV; ++j)
#pragma unroll
      for (int d = 0; d < 2; ++d) gu[j][d] = N[j] * gph[d] + ph * G[j][d];
    double wga[2];
#pragma unroll
    for (int d = 0; d < 2; ++d) wga[d] = w * (na * gph[d] + ph * ga[d]);
    bv += w * fq * ph * na;
#pragma unroll
    for (int j = 0; j < NV; ++j) A[j] += dotd<2>(wga, gu[j]);
    if (cut) {
      const double P00 = Jit[0][0] * Jit[0][0] + Jit[1][0] * Jit[1][0];   // P = K K^T, K^T = Jit
      const double P01 = Jit[0][0] * Jit[0][1] + Jit[1][0] * Jit[1][1];
      const double P11 = Jit[0][1] * Jit[0][1] + Jit[1][1] * Jit[1][1];
      const double lph = hr[0] * P00 + 2.0 * (hr[1] - (c0 * gph[0] + c1 * gph[1])) * P01 + hr[2] * P11;
      double lu[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const double sj = (j == 0 || j == 3) ? 1.0 : -1.0;
        const double lpsi = 2.0 * P01 * (sj - (c0 * G[j][0] + c1 * G[j][1]));
        lu[j] = N[j] * lph + 2.0 * (gph[0] * G[j][0] + gph[1] * G[j][1]) + ph * lpsi;
      }
      const double lua = na * lph + 2.0 * dotd<2>(gph, ga) + ph * 2.0 * P01 * (sa - (c0 * ga[0] + c1 * ga[1]));
      const double ws = w * sh2 * lua;
      bv -= ws * fq;
#pragma unroll
      for (int j = 0; j < NV; ++j) A[j] += ws * lu[j];
    }
  }
  atomicAdd(b + __ldg(dm + a), bv);
#pragma unroll
  for (int j = 0; j < NV; ++j) atomicAdd(data + __ldg(slots + (int64_t)(a * NV + j) * n_active + e), A[j]);
}

// -int_{ds(100)} (grad(phi w).n) phi v on (cell, local facet) pairs, along the straight edge with its constant normal.
// One thread per (entity, test dof i); v_i vanishes on an edge without vertex i.  Slots entity-major ([n, 16]).
template <int KP>
__global__ void __launch_bounds__(kBlockPk) k_quad_boundary_strong(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qfp_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const int32_t* __restrict__ entities, int64_t n_entities,
    const int32_t* __restrict__ slots, double* __restrict__ data) {
  constexpr int NDP = QSpace<KP>::ND;
  __shared__ double qt[kMaxQuadPoints], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) {
    qt[i] = qfp_g[2 * i + 1];   // segment point (1 - t, t): the parameter t
    qw[i] = qw_g[i];
  }
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * NV) return;
  const int64_t e = t / NV;
  const int i = (int)(t - e * NV);
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  const int la = facet_vertex(o, 0), lb = facet_vertex(o, 1);
  if (i != la && i != lb) return;
  Cell g;
  load_cell(m, c, g);
  double pc[NDP];
  load_phi<KP>(m, sp, phi, c, pc);
  double n[2], len;
  edge_normal(g, o, n, len);
  const double r0[2] = {(double)(la & 1), (double)(la >> 1)}, r1[2] = {(double)(lb & 1), (double)(lb >> 1)};
  double A[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double tq = qt[q];
    const double xi = (1.0 - tq) * r0[0] + tq * r1[0], eta = (1.0 - tq) * r0[1] + tq * r1[1];
    double N[NV], G[NV][2], Jit[2][2];
    map_point(g, xi, eta, N, G, Jit);
    double ph, gph[2];
    eval_phi<KP>(xi, eta, Jit, pc, ph, gph);
    const double gpn = dotd<2>(gph, n);
    const double ui = -qw[q] * len * ph * pk::pick<NV>(N, i);
#pragma unroll
    for (int j = 0; j < NV; ++j) A[j] += ui * (N[j] * gpn + ph * dotd<2>(G[j], n));
  }
#pragma unroll
  for (int j = 0; j < NV; ++j) atomicAdd(data + __ldg(slots + (e * NV + i) * NV + j), A[j]);
}

// sigma avg(h) int_F [grad(phi w).n][grad(phi v).n] over interior facets, into the 8 x 8 macro slots [dofs of cell +
// (f2c[f][0]), of cell -].  The edge parameter runs from the lower- to the higher-global-id vertex (as in
// k_quad_ghost_neumann), so both sides evaluate the same physical points; each side evaluates phi and grad(phi) from
// its own cell's dofs.  One thread per (facet, macro dof a: a / 4 = side).
template <int KP>
__global__ void __launch_bounds__(kBlockPk) k_quad_ghost_strong(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qfp_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const int32_t* __restrict__ facets, int64_t n_facets,
    const int32_t* __restrict__ slots, double sigma, double* __restrict__ data) {
  constexpr int NDP = QSpace<KP>::ND, NU = 2 * NV;
  __shared__ double qt[kMaxQuadPoints], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) {
    qt[i] = qfp_g[2 * i + 1];
    qw[i] = qw_g[i];
  }
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets * NU) return;
  const int64_t e = t / NU;
  const int a = (int)(t - e * NU);
  const int32_t fct = __ldg(facets + e);
  const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
  Cell g[2];
  double pc[2][NDP], n[2][2], len = 0.0, r0[2][2], r1[2][2];
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int64_t c = s == 0 ? cc.x : cc.y;
    load_cell(m, c, g[s]);
    load_phi<KP>(m, sp, phi, c, pc[s]);
    int o = 0;
#pragma unroll
    for (int k = 0; k < NV; ++k)
      if (__ldg(m.c2f + c * NV + k) == fct) o = k;
    int la = facet_vertex(o, 0), lb = facet_vertex(o, 1);
    if (__ldg(m.cells + c * NV + la) > __ldg(m.cells + c * NV + lb)) {
      const int tmp = la;
      la = lb;
      lb = tmp;
    }
    r0[s][0] = la & 1; r0[s][1] = la >> 1;
    r1[s][0] = lb & 1; r1[s][1] = lb >> 1;
    double l;
    edge_normal(g[s], o, n[s], l);
    if (s == 0) len = l;
  }
  const double coef = sigma * 0.5 * (sqrt(g[0].h2) + sqrt(g[1].h2)) * len;
  double E[NU];
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) E[bb] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double tq = qt[q];
    double J[NU];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const double xi = (1.0 - tq) * r0[s][0] + tq * r1[s][0], eta = (1.0 - tq) * r0[s][1] + tq * r1[s][1];
      double N[NV], G[NV][2], Jit[2][2];
      map_point(g[s], xi, eta, N, G, Jit);
      double ph, gph[2];
      eval_phi<KP>(xi, eta, Jit, pc[s], ph, gph);
      const double gpn = dotd<2>(gph, n[s]);
#pragma unroll
      for (int k = 0; k < NV; ++k) J[s * NV + k] = N[k] * gpn + ph * dotd<2>(G[k], n[s]);
    }
    const double wa = qw[q] * coef * pk::pick<NU>(J, a);
#pragma unroll
    for (int bb = 0; bb < NU; ++bb) E[bb] += wa * J[bb];
  }
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) atomicAdd(data + __ldg(slots + (e * NU + a) * NU + bb), E[bb]);
}

inline unsigned blocks(int64_t threads) { return (unsigned)((threads + kBlockPk - 1) / kBlockPk); }

}  // namespace quad

// ---- launchers (arguments validated by the entry points in assemble_pk.cu) ------------------------------------------
int quad_neumann_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                       const double* phi, const double* f, const double* u_n, const int8_t* cell_tags8,
                       const int32_t* active, int64_t n_active, const int32_t* cut_positions, int64_t n_cut,
                       const int32_t* slots, const int32_t* mixed_dofmap, double gamma, double robin_coef,
                       double* data, double* b, cudaStream_t st) {
  using namespace quad;
  const double *qp = quad_rule->cell_points, *qw = quad_rule->cell_weights;
  const int nq = quad_rule->n_cell_points;
  k_quad_interior_neumann<<<blocks(n_active * NV), kBlockPk, 0, st>>>(*mesh, qp, qw, nq, f, cell_tags8, active,
                                                                       n_active, slots, mixed_dofmap, data, b);
  if (n_cut > 0) {
    if (space_phi->n_dofs_per_cell == QSpace<1>::ND)
      k_quad_cells_neumann<1><<<blocks(n_cut * NM), kBlockPk, 0, st>>>(
          *mesh, *space_phi, qp, qw, nq, phi, f, u_n, active, n_active, cut_positions, n_cut, slots, mixed_dofmap,
          gamma, robin_coef, data, b);
    else
      k_quad_cells_neumann<2><<<blocks(n_cut * NM), kBlockPk, 0, st>>>(
          *mesh, *space_phi, qp, qw, nq, phi, f, u_n, active, n_active, cut_positions, n_cut, slots, mixed_dofmap,
          gamma, robin_coef, data, b);
  }
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

int quad_neumann_boundary(const phifem_mesh* mesh, const int32_t* entities, int64_t n_entities, const int32_t* slots,
                          double* data, cudaStream_t st) {
  using namespace quad;
  k_quad_boundary_neumann<<<blocks(n_entities * NV), kBlockPk, 0, st>>>(*mesh, entities, n_entities, slots, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

int quad_neumann_ghost(const phifem_mesh* mesh, const phifem_quadrature* quad_rule, const int32_t* facets,
                       int64_t n_facets, const int32_t* slots, double sigma, double* data, cudaStream_t st) {
  using namespace quad;
  k_quad_ghost_neumann<<<blocks(n_facets * 2 * NV), kBlockPk, 0, st>>>(
      *mesh, quad_rule->facet_points, quad_rule->facet_weights, quad_rule->n_facet_points, facets, n_facets, slots,
      sigma, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

int quad_strong_cells(const phifem_mesh* mesh, const phifem_pk_space* space_w, const phifem_pk_space* space_phi,
                      const phifem_quadrature* quad_rule, const double* phi, const double* f, const int8_t* cell_tags8,
                      const int32_t* active, int64_t n_active, const int32_t* slots, double sigma, double* data,
                      double* b, cudaStream_t st) {
  using namespace quad;
  const double *qp = quad_rule->cell_points, *qw = quad_rule->cell_weights;
  const int nq = quad_rule->n_cell_points;
  if (space_phi->n_dofs_per_cell == QSpace<1>::ND)
    k_quad_cells_strong<1><<<blocks(n_active * NV), kBlockPk, 0, st>>>(
        *mesh, *space_w, *space_phi, qp, qw, nq, phi, f, cell_tags8, active, n_active, slots, sigma, data, b);
  else
    k_quad_cells_strong<2><<<blocks(n_active * NV), kBlockPk, 0, st>>>(
        *mesh, *space_w, *space_phi, qp, qw, nq, phi, f, cell_tags8, active, n_active, slots, sigma, data, b);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

int quad_strong_boundary(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                         const double* phi, const int32_t* entities, int64_t n_entities, const int32_t* slots,
                         double* data, cudaStream_t st) {
  using namespace quad;
  const double *qp = quad_rule->facet_points, *qw = quad_rule->facet_weights;
  const int nq = quad_rule->n_facet_points;
  if (space_phi->n_dofs_per_cell == QSpace<1>::ND)
    k_quad_boundary_strong<1><<<blocks(n_entities * NV), kBlockPk, 0, st>>>(*mesh, *space_phi, qp, qw, nq, phi,
                                                                             entities, n_entities, slots, data);
  else
    k_quad_boundary_strong<2><<<blocks(n_entities * NV), kBlockPk, 0, st>>>(*mesh, *space_phi, qp, qw, nq, phi,
                                                                             entities, n_entities, slots, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

int quad_strong_ghost(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                      const double* phi, const int32_t* facets, int64_t n_facets, const int32_t* slots, double sigma,
                      double* data, cudaStream_t st) {
  using namespace quad;
  const double *qp = quad_rule->facet_points, *qw = quad_rule->facet_weights;
  const int nq = quad_rule->n_facet_points;
  if (space_phi->n_dofs_per_cell == QSpace<1>::ND)
    k_quad_ghost_strong<1><<<blocks(n_facets * 2 * NV), kBlockPk, 0, st>>>(*mesh, *space_phi, qp, qw, nq, phi, facets,
                                                                            n_facets, slots, sigma, data);
  else
    k_quad_ghost_strong<2><<<blocks(n_facets * 2 * NV), kBlockPk, 0, st>>>(*mesh, *space_phi, qp, qw, nq, phi, facets,
                                                                            n_facets, slots, sigma, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

}  // namespace phifem
