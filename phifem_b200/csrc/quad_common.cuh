// Helpers of the bilinear quadrilateral cell (vertices in tensor order v0 = (0,0), v1 = (1,0), v2 = (0,1), v3 = (1,1)),
// shared by the quadrilateral kernels of assemble_quad.cu and assemble_elasticity.cu: the cell's vertices and diameter,
// the map and J^-T at a reference point, Q1 / Q2 level sets, and the outward normal of a straight edge.
#pragma once
#include "common.cuh"

namespace phifem {
namespace quad {

constexpr int NV = 4;            // vertices of a quadrilateral

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

}  // namespace quad
}  // namespace phifem
