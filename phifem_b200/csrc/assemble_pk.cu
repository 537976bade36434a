// K2/K3/K4 for Lagrange P1 / P2 trial-test spaces and P1 / P2 level sets on triangles / tetrahedra:
// the strong-Dirichlet phi-FEM operator of reference demo/strong-dirichlet/flower/main.py:104-128 with
// `fe_degree`, `levelset_degree` in {1, 2} (main.py:37-41), evaluated by quadrature.
//
// dolfinx would JIT one FFCx `tabulate_tensor` per integral and call it once per entity
// (main.py:121-123,130-131); here one thread evaluates a block of rows of one element tensor with every
// loop over basis functions unrolled at compile time (accumulators in registers), the quadrature rule
// staged in shared memory, and adds the entries into CSR through a precomputed entity -> slot map.
// The rules are host-provided tables (phifem_quadrature): the symbolic side picks rules exact for the
// polynomial degree of each integrand (2 (kw + kphi - 1) on cells, 2 (kw + kphi) - 1 on facets).
#include <type_traits>

#include "common.cuh"
#include "pk_common.cuh"

namespace phifem {
using namespace pk;
namespace {

// Does exactly ONE cell of a conforming simplicial mesh contribute to the CSR entry (dof i, dof j) of a cell?  True when
// the vertices the two dofs sit on (a vertex dof: itself; a P2 edge dof: the edge's two vertices) are all D + 1 vertices
// of the cell between them AND no facet contains them all -- in 2D: two different edge dofs, or a vertex dof and the
// dof of the opposite edge (12 of the 36 entries of a P2 triangle); in 3D: the dofs of two opposite edges (6 of 100).
// Such entries are written with a plain store after the zero-fill instead of an fp64 reduction: the P2 cell kernel of
// config C is bound by the rate of its reductions (42 per triangle), not by occupancy (8 or 12 warps per SM: same time).
template <int D, int K>
__host__ __device__ constexpr bool single_contributor(int i, int j) {
  constexpr int NV = D + 1;
  unsigned mask = 0;
  for (int t = 0; t < 2; ++t) {
    const int dof = t == 0 ? i : j;
    if (dof < NV) mask |= 1u << dof;
    else if (K == 2) mask |= (1u << ev<D>(dof - NV, 0)) | (1u << ev<D>(dof - NV, 1));
  }
  return mask == (1u << NV) - 1u;   // all vertices of the simplex: no facet (a proper subset of them) holds both dofs
}

// ---- cells: rows [I0, I1) of the symmetric element matrix (columns j >= i) and of the load vector ----
//   A_ij = int grad(phi psi_i).grad(phi psi_j) + [cut] sigma h^2 int lap(phi psi_i) lap(phi psi_j)   (main.py:105-112)
//   b_i  = int f phi psi_i - [cut] sigma h^2 int f lap(phi psi_i)                                     (:126-128)
template <int D, int KW, int KP, int I0, int I1>
__device__ __forceinline__ void cell_rows(const Geometry<D>& g, const double (&pc)[Space<D, KP>::ND],
                                          const double (&fc)[Space<D, KW>::ND], bool is_cut, double sigma,
                                          const double* __restrict__ qlam, const double* __restrict__ qw,
                                          int nq, const int32_t* __restrict__ slots, int64_t stride,
                                          const int32_t* __restrict__ dofs, double* __restrict__ data,
                                          double* __restrict__ b) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NDP = Space<D, KP>::ND, NR = I1 - I0;
  double A[NR][ND], bv[NR];
#pragma unroll
  for (int i = 0; i < NR; ++i) {
    bv[i] = 0.0;
#pragma unroll
    for (int j = 0; j < ND; ++j) A[i][j] = 0.0;
  }
  double wl[ND], lph = 0.0;
  laplacians<D, KW>(g.G, wl);
  {
    double pl[NDP];
    laplacians<D, KP>(g.G, pl);
#pragma unroll
    for (int k = 0; k < NDP; ++k) lph += pc[k] * pl[k];
  }
  const double sh2 = is_cut ? sigma * g.h2 : 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) lam[k] = qlam[q * NV + k];
    const double w = qw[q] * g.vol;
    double wv[ND], wg[ND][D];
    tabulate<D, KW>(lam, g.G, wv, wg);
    double ph, gph[D];
    eval_phi<D, KW, KP>(lam, g.G, wv, wg, pc, ph, gph);
    double fq = 0.0;
#pragma unroll
    for (int k = 0; k < ND; ++k) fq += fc[k] * wv[k];
    double gu[ND][D];
#pragma unroll
    for (int j = I0; j < ND; ++j)
#pragma unroll
      for (int d = 0; d < D; ++d) gu[j][d] = wv[j] * gph[d] + ph * wg[j][d];
    const double wf = w * fq;
#pragma unroll
    for (int i = I0; i < I1; ++i) {
      bv[i - I0] += wf * ph * wv[i];
      double wgi[D];
#pragma unroll
      for (int d = 0; d < D; ++d) wgi[d] = w * gu[i][d];
#pragma unroll
      for (int j = i; j < ND; ++j) A[i - I0][j] += dotd<D>(wgi, gu[j]);
    }
    if (is_cut) {
      double lu[ND];
#pragma unroll
      for (int j = I0; j < ND; ++j) lu[j] = wv[j] * lph + 2.0 * dotd<D>(gph, wg[j]) + ph * wl[j];
      const double ws = w * sh2;
#pragma unroll
      for (int i = I0; i < I1; ++i) {
        bv[i - I0] -= ws * fq * lu[i];
        const double wli = ws * lu[i];
#pragma unroll
        for (int j = i; j < ND; ++j) A[i - I0][j] += wli * lu[j];
      }
    }
  }
#pragma unroll
  for (int i = I0; i < I1; ++i) {
    atomicAdd(b + dofs[i], bv[i - I0]);
#pragma unroll
    for (int j = i; j < ND; ++j) {
      const double v = A[i - I0][j];
      const int32_t sij = __ldg(slots + (int64_t)(i * ND + j) * stride);
      const int32_t sji = __ldg(slots + (int64_t)(j * ND + i) * stride);
      if (single_contributor<D, KW>(i, j)) {
        data[sij] = v;
        data[sji] = v;
      } else {
        atomicAdd(data + sij, v);
        if (j != i) atomicAdd(data + sji, v);
      }
    }
  }
}

// row ranges of the passes (blockIdx.y): the accumulators of one pass must fit the register file
template <int ND> struct Passes { static constexpr int N = 1; };
template <> struct Passes<10> { static constexpr int N = 3; };

// measured on the B200 at config C (16 M P2 triangles, cell kernel): 128 threads x 3 CTAs per SM 1.252 ms, x 2 CTAs 1.252,
// x 4 CTAs (spills) 1.268; 64 threads x 6 CTAs 1.214; + the slot lines prefetched into L1 before the quadrature loop 1.188;
// 64 x 4 (226 registers, nothing spilled) 1.174; the quadrature loop unrolled by two: 1.172 (64 x 4), 1.274 (64 x 6).
// A persistent version with the next cells' loads pipelined through cp.async measured 1.331 against 1.175 ms: the kernel
// is bound by the number of its scattered reductions, not by the latency in front of them (DESIGN.md §4, K2p).
constexpr int kBlockPkCells = 64;
constexpr int kPkCellsMinBlocks2D = 4;

template <int D, int KW, int KP>
__global__ void __launch_bounds__(kBlockPkCells, D == 2 ? kPkCellsMinBlocks2D : 256 / kBlockPkCells) k_assemble_cells_pk(
    phifem_mesh m, phifem_pk_space sw, phifem_pk_space sp, const double* __restrict__ qlam_g,
    const double* __restrict__ qw_g, int nq, const double* __restrict__ phi, const double* __restrict__ f,
    const int8_t* __restrict__ ctags, const int32_t* __restrict__ active, int64_t n_active,
    const int32_t* __restrict__ slots, double sigma, double* __restrict__ data, double* __restrict__ b) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NDP = Space<D, KP>::ND;
  __shared__ double qlam[kMaxQuadPoints * NV], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * NV; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_active) return;
  const int64_t c = __ldg(active + e);
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double pc[NDP], fc[ND];
  load_dofs<D, KP>(m, sp, phi, c, pc);
  load_dofs<D, KW>(m, sw, f, c, fc);
  int32_t dofs[ND];
  {
    const int32_t* dm = sw.dofmap ? sw.dofmap + c * ND : m.cells + c * ND;
#pragma unroll
    for (int k = 0; k < ND; ++k) dofs[k] = __ldg(dm + k);
  }
  const bool is_cut = ctags[c] == 2;
  const int32_t* sl = slots + e;
  // the slot lines of the final scatter (entry-major: one coalesced line per entry and warp) are requested now, so that
  // the ND^2 dependent load -> reduction pairs at the end find them in L1
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < ND * ND; ++k) asm volatile("prefetch.global.L1 [%0];" ::"l"(sl + (int64_t)k * n_active));
  }
  if constexpr (ND == 10) {
    if (blockIdx.y == 0)
      cell_rows<D, KW, KP, 0, 2>(g, pc, fc, is_cut, sigma, qlam, qw, nq, sl, n_active, dofs, data, b);
    else if (blockIdx.y == 1)
      cell_rows<D, KW, KP, 2, 5>(g, pc, fc, is_cut, sigma, qlam, qw, nq, sl, n_active, dofs, data, b);
    else
      cell_rows<D, KW, KP, 5, 10>(g, pc, fc, is_cut, sigma, qlam, qw, nq, sl, n_active, dofs, data, b);
  } else {
    cell_rows<D, KW, KP, 0, ND>(g, pc, fc, is_cut, sigma, qlam, qw, nq, sl, n_active, dofs, data, b);
  }
}

// ---- one-sided boundary term: one thread per (entity, test dof i) ------------------------------------------
//   A_ij = -int_F (grad(phi psi_j).n) phi psi_i    (main.py:106), n = outward normal of the entity's cell
template <int D, int KW, int KP>
__global__ void __launch_bounds__(kBlockPk) k_assemble_boundary_pk(
    phifem_mesh m, phifem_pk_space sw, phifem_pk_space sp, const double* __restrict__ qlam_g,
    const double* __restrict__ qw_g, int nq, const double* __restrict__ phi,
    const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ slots,
    double* __restrict__ data) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NDP = Space<D, KP>::ND;
  __shared__ double qlam[kMaxQuadPoints * D], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * D; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * ND) return;
  const int64_t e = t / ND;
  const int i = (int)(t - e * ND);
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double pc[NDP];
  load_dofs<D, KP>(m, sp, phi, c, pc);
  double n[D], area;
  facet_normal<D>(g, o, n, area);
  double A[ND];
#pragma unroll
  for (int j = 0; j < ND; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
    facet_to_cell<D>(qlam + q * D, o, lam);
    double wv[ND], wg[ND][D];
    tabulate<D, KW>(lam, g.G, wv, wg);
    double ph, gph[D];
    eval_phi<D, KW, KP>(lam, g.G, wv, wg, pc, ph, gph);
    const double gpn = dotd<D>(gph, n);
    const double ui = -qw[q] * area * ph * pick<ND>(wv, i);
#pragma unroll
    for (int j = 0; j < ND; ++j) A[j] += ui * (wv[j] * gpn + ph * dotd<D>(wg[j], n));
  }
#pragma unroll
  for (int j = 0; j < ND; ++j) atomicAdd(data + __ldg(slots + (e * ND + i) * ND + j), A[j]);
}

// value and gradient of ONE basis function (run-time index i) of the P_K Lagrange basis at barycentric point lam
template <int D, int K>
__device__ __forceinline__ void basis_one(const double (&lam)[D + 1], const double (&G)[D + 1][D], int i,
                                          double& val, double (&grad)[D]) {
  constexpr int NV = D + 1;
  // vertex a (and, for an edge function, vertex b) the function belongs to
  int a = i, b = -1;
  if (K == 2 && i >= NV) {
    a = 0;
    b = 0;
#pragma unroll
    for (int e = 0; e < Space<D, K>::NE; ++e)
      if (e == i - NV) {
        a = ev<D>(e, 0);
        b = ev<D>(e, 1);
      }
  }
  double la = 0.0, lb = 0.0, Ga[D], Gb[D];
#pragma unroll
  for (int d = 0; d < D; ++d) Ga[d] = Gb[d] = 0.0;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    if (k == a) {
      la = lam[k];
#pragma unroll
      for (int d = 0; d < D; ++d) Ga[d] = G[k][d];
    }
    if (k == b) {
      lb = lam[k];
#pragma unroll
      for (int d = 0; d < D; ++d) Gb[d] = G[k][d];
    }
  }
  if (K == 1) {
    val = la;
#pragma unroll
    for (int d = 0; d < D; ++d) grad[d] = Ga[d];
  } else if (b < 0) {
    val = la * (2.0 * la - 1.0);
#pragma unroll
    for (int d = 0; d < D; ++d) grad[d] = (4.0 * la - 1.0) * Ga[d];
  } else {
    val = 4.0 * la * lb;
#pragma unroll
    for (int d = 0; d < D; ++d) grad[d] = 4.0 * (la * Gb[d] + lb * Ga[d]);
  }
}

// ---- ghost penalty: the 2 ND threads of a facet cooperate --------------------------------------------------------
//   E_ab = sigma avg(h_T) int_F J_a J_b,  J_a = grad(phi psi_a).n of the side dof a lives on   (main.py:113-118)
// macro dofs = [dofs of cell + (= f2c[f][0]), dofs of cell -]: 2 ND rows/columns, shared dofs appear twice
// and add into the same CSR entry, as in dolfinx's interior-facet assembly.  Thread (facet, a) tabulates ITS jump
// J_a at every facet point into shared memory; after one barrier it accumulates row a of E from the facet's table.
template <int D, int KW>
struct GhostLayout {
  static constexpr int NM = 2 * Space<D, KW>::ND;
  static constexpr int FPB = kBlockPk / NM;      // facets per block (the facet rule holds at most 32 points: 16 for P2 / P2)
};

template <int D, int KW, int KP>
__global__ void __launch_bounds__(kBlockPk) k_assemble_ghost_pk(
    phifem_mesh m, phifem_pk_space sw, phifem_pk_space sp, const double* __restrict__ qlam_g,
    const double* __restrict__ qw_g, int nq, const double* __restrict__ phi,
    const int32_t* __restrict__ facets, int64_t n_facets, const int32_t* __restrict__ slots, double sigma,
    double* __restrict__ data) {
  using L = GhostLayout<D, KW>;
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NDP = Space<D, KP>::ND, NM = L::NM, FPB = L::FPB, NP = NV + 2;
  // dynamic shared memory: the rule, the jumps Js[FPB][nq][NM] and -- evaluated ONCE per (facet, side, point) instead of
  // once per thread -- the point in the side's barycentric coordinates, phi and grad(phi).n there: Pq[FPB][2][nq][NV + 2]
  // (the P2 tetrahedron: 20 threads per facet each re-evaluated the 10 P2 basis functions of phi at 16 points;
  // 1.30 -> 1.04 ms for the 141 750 ghost facets of the 3d-p2 configuration -- what remains is the scatter: 400 fp64
  // reductions per facet, 196 of them onto entries another thread of the same facet also adds to)
  extern __shared__ double sm_ghost[];
  double* qlam = sm_ghost;
  double* qw = qlam + nq * D;
  double* Js = qw + nq;
  double* Pq = Js + (size_t)FPB * nq * NM;
  for (int i = threadIdx.x; i < nq * D; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int fl = threadIdx.x / NM, a = threadIdx.x % NM;
  const int64_t e = (int64_t)blockIdx.x * FPB + fl;
  const bool live = fl < FPB && e < n_facets;
  const bool minus = a >= ND;                 // the side this thread's dof lives on
  const int al = minus ? a - ND : a;          // its index among the side's dofs
  double coef = 0.0;
  double G[NV][D], n[D];  // geometry of this thread's side (selected value by value: stays in registers)
  if (live) {
    const int32_t fct = __ldg(facets + e);
    const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
    Geometry<D> gp, gm;
    load_geometry<D>(m, cc.x, gp);
    load_geometry<D>(m, cc.y, gm);
    int op = 0, om = 0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (__ldg(m.c2f + (int64_t)cc.x * NV + k) == fct) op = k;
      if (__ldg(m.c2f + (int64_t)cc.y * NV + k) == fct) om = k;
    }
    double pc[NDP];
    load_dofs<D, KP>(m, sp, phi, minus ? cc.y : cc.x, pc);
    double np_[D], nm_[D], area, area_m;
    facet_normal<D>(gp, op, np_, area);
    facet_normal<D>(gm, om, nm_, area_m);
    coef = sigma * 0.5 * (sqrt(gp.h2) + sqrt(gm.h2)) * area;
#pragma unroll
    for (int k = 0; k < NV; ++k)
#pragma unroll
      for (int d = 0; d < D; ++d) G[k][d] = minus ? gm.G[k][d] : gp.G[k][d];
#pragma unroll
    for (int d = 0; d < D; ++d) n[d] = minus ? nm_[d] : np_[d];
    // phase 0: the ND threads of a side share the side's nq points
    double* pq_side = Pq + ((size_t)(fl * 2 + (minus ? 1 : 0)) * nq) * NP;
    for (int q = al; q < nq; q += ND) {
      double lam[NV];
      facet_to_cell<D>(qlam + q * D, op, lam);
      if (minus) {  // the same physical point in the barycentric coordinates of cell -
        double xq[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < NV; ++k) s += lam[k] * gp.X[k][d];
          xq[d] = s - gm.X[0][d];
        }
#pragma unroll
        for (int k = 0; k < NV; ++k) lam[k] = (k == 0 ? 1.0 : 0.0) + dotd<D>(gm.G[k], xq);
      }
      double ph, gph[D];
      eval_phi_only<D, KP>(lam, G, pc, ph, gph);
#pragma unroll
      for (int k = 0; k < NV; ++k) pq_side[q * NP + k] = lam[k];
      pq_side[q * NP + NV] = ph;
      pq_side[q * NP + NV + 1] = dotd<D>(gph, n);
    }
  }
  __syncthreads();
  if (live) {  // phase 1: this thread's jump at every point
    const double* pq_side = Pq + ((size_t)(fl * 2 + (minus ? 1 : 0)) * nq) * NP;
    for (int q = 0; q < nq; ++q) {
      double lam[NV];
#pragma unroll
      for (int k = 0; k < NV; ++k) lam[k] = pq_side[q * NP + k];
      double val, grad[D];
      basis_one<D, KW>(lam, G, al, val, grad);
      Js[((size_t)fl * nq + q) * NM + a] = val * pq_side[q * NP + NV + 1] + pq_side[q * NP + NV] * dotd<D>(grad, n);
    }
  }
  __syncthreads();
  double E[NM];
#pragma unroll
  for (int bb = 0; bb < NM; ++bb) E[bb] = 0.0;
  if (live) {
    for (int q = 0; q < nq; ++q) {
      const double* jq = Js + ((size_t)fl * nq + q) * NM;
      const double wa = qw[q] * coef * jq[a];
#pragma unroll
      for (int bb = 0; bb < NM; ++bb) E[bb] += wa * jq[bb];
    }
  }
  // Adding the facet's duplicate entries up in shared memory first (400 -> 196 reductions per P2 tetrahedron facet)
  // measured 1.253 against 1.040 ms at 3d-p2: the pass is not bound by its reductions (DESIGN.md §4, K2p).
  if (!live) return;
#pragma unroll
  for (int bb = 0; bb < NM; ++bb) atomicAdd(data + __ldg(slots + (e * NM + a) * NM + bb), E[bb]);
}

// ==== weak-Dirichlet (dual) phi-FEM operator on the mixed space (u, p) in P_KW x P_KW ========================
// reference demo/weak-dirichlet/flower/main.py:112-151 (BASELINE.json configs[0]):
//   a = int_{dx(1,2)} grad u.grad v - int_ds (grad u.n) v + gamma h^-2 int_{dx(2)} (u - h^-1 phi p)(v - h^-1 phi q)
//       + sigma h^2 int_{dx(2)} lap u lap v + sigma int_{dS(2,3)} avg(h) [grad u.n][grad v.n]
//   L = int_{dx(1,2)} f v + gamma h^-2 int_{dx(2)} u_D (v - h^-1 phi q) - sigma h^2 int_{dx(2)} f lap v
// Cell-local mixed dofs: [u dofs, p dofs] (NM = 2 ND); one thread per (entity, mixed test dof).

template <int D, int KW, int KP>
__global__ void __launch_bounds__(kBlockPk) k_assemble_cells_weak_pk(
    phifem_mesh m, phifem_pk_space sw, phifem_pk_space sp, const double* __restrict__ qlam_g,
    const double* __restrict__ qw_g, int nq, const double* __restrict__ phi, const double* __restrict__ f,
    const double* __restrict__ ud, const int8_t* __restrict__ ctags, const int32_t* __restrict__ active,
    int64_t n_active, const int32_t* __restrict__ slots, const int32_t* __restrict__ mixed_dofmap,
    double gamma, double sigma, double* __restrict__ data, double* __restrict__ b) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NDP = Space<D, KP>::ND, NM = 2 * ND;
  __shared__ double qlam[kMaxQuadPoints * NV], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * NV; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_active * NM) return;
  const int64_t e = t / NM;
  const int a = (int)(t - e * NM);
  const bool test_q = a >= ND;  // mixed test function (0, psi_i) instead of (psi_i, 0)
  const int i = test_q ? a - ND : a;
  const int64_t c = __ldg(active + e);
  const bool is_cut = ctags[c] == 2;
  if (test_q && !is_cut) return;  // rows of q only carry the penalty term of cut cells
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double pc[NDP], fc[ND], uc[ND];
  load_dofs<D, KP>(m, sp, phi, c, pc);
  load_dofs<D, KW>(m, sw, f, c, fc);
  load_dofs<D, KW>(m, sw, ud, c, uc);
  double wl[ND];
  laplacians<D, KW>(g.G, wl);
  const double wli = pick<ND>(wl, i);
  const double h = sqrt(g.h2);
  const double pen = is_cut ? gamma / g.h2 : 0.0, stab = is_cut ? sigma * g.h2 : 0.0, rh = 1.0 / h;
  double A[NM], bv = 0.0;
#pragma unroll
  for (int j = 0; j < NM; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) lam[k] = qlam[q * NV + k];
    const double w = qw[q] * g.vol;
    double wv[ND], wg[ND][D];
    tabulate<D, KW>(lam, g.G, wv, wg);
    double ph, gph[D];
    eval_phi<D, KW, KP>(lam, g.G, wv, wg, pc, ph, gph);
    double fq = 0.0, uq = 0.0;
#pragma unroll
    for (int k = 0; k < ND; ++k) {
      fq += fc[k] * wv[k];
      uq += uc[k] * wv[k];
    }
    const double psi = pick<ND>(wv, i);
    if (!test_q) {
      double gi[D];
#pragma unroll
      for (int d = 0; d < D; ++d) {
        double v = wg[0][d];
#pragma unroll
        for (int k = 1; k < ND; ++k)
          if (k == i) v = wg[k][d];
        gi[d] = v;
      }
      bv += w * (fq * psi - stab * fq * wli);
#pragma unroll
      for (int j = 0; j < ND; ++j) A[j] += w * (dotd<D>(wg[j], gi) + stab * wl[j] * wli);
    }
    if (is_cut) {
      const double pr = -ph * rh;                   // p-part of the combination  u - h^-1 phi p
      const double T = (test_q ? pr * psi : psi) * w * pen;
      bv += uq * T;
#pragma unroll
      for (int j = 0; j < ND; ++j) {
        A[j] += wv[j] * T;
        A[ND + j] += pr * wv[j] * T;
      }
    }
  }
  atomicAdd(b + __ldg(mixed_dofmap + c * NM + a), bv);
#pragma unroll
  for (int j = 0; j < NM; ++j)
    if (j < ND || is_cut) atomicAdd(data + __ldg(slots + (int64_t)(a * NM + j) * n_active + e), A[j]);
}

template <int D, int KW>
__global__ void __launch_bounds__(kBlockPk) k_assemble_boundary_weak_pk(
    phifem_mesh m, const double* __restrict__ qlam_g, const double* __restrict__ qw_g, int nq,
    const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ slots,
    double* __restrict__ data) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NM = 2 * ND;
  __shared__ double qlam[kMaxQuadPoints * D], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * D; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * ND) return;
  const int64_t e = t / ND;
  const int i = (int)(t - e * ND);
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double n[D], area;
  facet_normal<D>(g, o, n, area);
  double A[ND];
#pragma unroll
  for (int j = 0; j < ND; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
    facet_to_cell<D>(qlam + q * D, o, lam);
    double wv[ND], wg[ND][D];
    tabulate<D, KW>(lam, g.G, wv, wg);
    const double vi = -qw[q] * area * pick<ND>(wv, i);
#pragma unroll
    for (int j = 0; j < ND; ++j) A[j] += vi * dotd<D>(wg[j], n);
  }
#pragma unroll
  for (int j = 0; j < ND; ++j) atomicAdd(data + __ldg(slots + (e * NM + i) * NM + j), A[j]);
}

template <int D, int KW, int NMIX = 2 * Space<D, KW>::ND>
__global__ void __launch_bounds__(kBlockPk) k_assemble_ghost_weak_pk(
    phifem_mesh m, const double* __restrict__ qlam_g, const double* __restrict__ qw_g, int nq,
    const int32_t* __restrict__ facets, int64_t n_facets, const int32_t* __restrict__ slots, double sigma,
    double* __restrict__ data) {
  constexpr int NV = D + 1, ND = Space<D, KW>::ND, NM = NMIX, NU = 2 * ND;  // NU: u dofs of both sides
  __shared__ double qlam[kMaxQuadPoints * D], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * D; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets * NU) return;
  const int64_t e = t / NU;
  const int a = (int)(t - e * NU);  // u dof a of side a / ND
  const int32_t fct = __ldg(facets + e);
  const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
  Geometry<D> gp, gm;
  load_geometry<D>(m, cc.x, gp);
  load_geometry<D>(m, cc.y, gm);
  int op = 0, om = 0;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    if (__ldg(m.c2f + (int64_t)cc.x * NV + k) == fct) op = k;
    if (__ldg(m.c2f + (int64_t)cc.y * NV + k) == fct) om = k;
  }
  double np_[D], nm_[D], area, area_m;
  facet_normal<D>(gp, op, np_, area);
  facet_normal<D>(gm, om, nm_, area_m);
  const double coef = sigma * 0.5 * (sqrt(gp.h2) + sqrt(gm.h2)) * area;
  double E[NU];
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) E[bb] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV], J[NU];
    facet_to_cell<D>(qlam + q * D, op, lam);
    {
      double wv[ND], wg[ND][D];
      tabulate<D, KW>(lam, gp.G, wv, wg);
#pragma unroll
      for (int j = 0; j < ND; ++j) J[j] = dotd<D>(wg[j], np_);
    }
    double xq[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
      double s = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) s += lam[k] * gp.X[k][d];
      xq[d] = s - gm.X[0][d];
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) lam[k] = (k == 0 ? 1.0 : 0.0) + dotd<D>(gm.G[k], xq);
    {
      double wv[ND], wg[ND][D];
      tabulate<D, KW>(lam, gm.G, wv, wg);
#pragma unroll
      for (int j = 0; j < ND; ++j) J[ND + j] = dotd<D>(wg[j], nm_);
    }
    const double wa = qw[q] * coef * pick<NU>(J, a);
#pragma unroll
    for (int bb = 0; bb < NU; ++bb) E[bb] += wa * J[bb];
  }
  // macro mixed index of u dof j of side s: s * NM + j
  const int ma = (a / ND) * NM + (a % ND);
#pragma unroll
  for (int bb = 0; bb < NU; ++bb) {
    const int mb = (bb / ND) * NM + (bb % ND);
    atomicAdd(data + __ldg(slots + (e * 2 * NM + ma) * 2 * NM + mb), E[bb]);
  }
}

// ==== Neumann phi-FEM operator on the mixed space (u, y, p) in P1 x P1^D x DG0 =====================================
// reference demo/neumann/square/main.py:103-158 (BASELINE.json configs[1]):
//   a = int_{dx(1,2)} (grad u.grad v + u v) + int_ds (y.n) v
//       + gamma int_{dx(2)} [ (y + grad u).(z + grad v) + (div y + u)(div z + v)
//                             + h^-2 (y.grad phi + h^-1 p phi)(z.grad phi + h^-1 q phi) ]
//       + sigma int_{dS(3)} avg(h) [grad u.n][grad v.n]
//   L = int_{dx(1,2)} f v + gamma int_{dx(2)} [ -h^-2 u_N |grad phi| (z.grad phi + h^-1 q phi) + f (div z + v) ]
// Cell-local mixed dofs: [u at the D+1 vertices, y node-major (vertex i, component c -> NV + i D + c), p]:
// NM = (D+1)(D+1) + 1.  Every basis function X carries  s1 = y + grad u, s2 = div y + u,
// s3 = y.grad phi + h^-1 p phi;  the cut-cell integrand is s1_b.s1_a + s2_b s2_a + h^-2 s3_b s3_a.
// One thread per (cell, mixed test dof a).
template <int D>
struct NeumannSpace {
  static constexpr int NV = D + 1;
  static constexpr int NM = NV * (1 + D) + 1;
};

// the tuple (u, grad u, s1, s2, s3) of mixed basis function m at a point (lam = P1 basis values, G their gradients)
template <int D>
__device__ __forceinline__ void neumann_basis(int m, const double (&lam)[D + 1], const double (&G)[D + 1][D],
                                              const double (&gph)[D], double ph_over_h, double kappa_ngp, double& U,
                                              double (&GU)[D], double (&S1)[D], double& S2, double& S3) {
  constexpr int NV = D + 1, NM = NeumannSpace<D>::NM;
  U = 0.0;
  S2 = 0.0;
  S3 = 0.0;
#pragma unroll
  for (int d = 0; d < D; ++d) GU[d] = S1[d] = 0.0;
  if (m == NM - 1) {  // p: piecewise constant
    S3 = ph_over_h;
    return;
  }
  const bool is_u = m < NV;
  const int node = is_u ? m : (m - NV) / D, comp = is_u ? -1 : (m - NV) % D;
  double lj = 0.0, Gj[D];
#pragma unroll
  for (int d = 0; d < D; ++d) Gj[d] = 0.0;
#pragma unroll
  for (int k = 0; k < NV; ++k)
    if (k == node) {
      lj = lam[k];
#pragma unroll
      for (int d = 0; d < D; ++d) Gj[d] = G[k][d];
    }
  if (is_u) {
    U = lj;
    S2 = lj;
    S3 = -kappa_ngp * lj;  // Robin: s3 = y.grad phi - |grad phi| kappa u + h^-1 p phi (demo/robin/square/main.py:124-133)
#pragma unroll
    for (int d = 0; d < D; ++d) GU[d] = S1[d] = Gj[d];
  } else {
#pragma unroll
    for (int d = 0; d < D; ++d)
      if (d == comp) {
        S1[d] = lj;
        S2 = Gj[d];
        S3 = lj * gph[d];
      }
  }
}

// Interior cells (tag 1) carry int grad u.grad v + u v and int f v only: the P1 stiffness and mass matrices in closed
// form, one light thread per (active cell, u test dof) -- kept apart from the cut-cell kernel, whose register footprint
// would otherwise set the occupancy of these latency-bound threads.
template <int D>
__global__ void __launch_bounds__(kBlockPk) k_assemble_interior_neumann(
    phifem_mesh m, const double* __restrict__ f, const int8_t* __restrict__ ctags, const int32_t* __restrict__ active,
    int64_t n_active, const int32_t* __restrict__ slots, const int32_t* __restrict__ mixed_dofmap,
    double* __restrict__ data, double* __restrict__ b) {
  constexpr int NV = D + 1, NM = NeumannSpace<D>::NM;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_active * NV) return;
  const int64_t e = t / NV;
  const int a = (int)(t - e * NV);
  const int64_t c = __ldg(active + e);
  if (ctags[c] == 2) return;
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  constexpr double mm = 1.0 / ((D + 1) * (D + 2));
  double Ga[D];
#pragma unroll
  for (int d = 0; d < D; ++d) Ga[d] = g.G[0][d];
#pragma unroll
  for (int k = 1; k < NV; ++k)
    if (k == a)
#pragma unroll
      for (int d = 0; d < D; ++d) Ga[d] = g.G[k][d];
  double s = 0.0;
#pragma unroll
  for (int k = 0; k < NV; ++k) s += __ldg(f + __ldg(m.cells + c * NV + k)) * (k == a ? 2.0 : 1.0);
  atomicAdd(b + __ldg(mixed_dofmap + c * NM + a), g.vol * mm * s);
#pragma unroll
  for (int bb = 0; bb < NV; ++bb)
    atomicAdd(data + __ldg(slots + (int64_t)(a * NM + bb) * n_active + e),
              g.vol * (dotd<D>(Ga, g.G[bb]) + (bb == a ? 2.0 * mm : mm)));
}

// Cut cells (tag 2): `cut_positions` [n_cut] = their positions in the active list.  One thread per (cut cell, mixed dof).
template <int D, int KP>
__global__ void __launch_bounds__(kBlockPk) k_assemble_cells_neumann(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qlam_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const double* __restrict__ f, const double* __restrict__ un,
    const int32_t* __restrict__ active, int64_t n_active, const int32_t* __restrict__ cut_positions, int64_t n_cut,
    const int32_t* __restrict__ slots, const int32_t* __restrict__ mixed_dofmap, double gamma, double kappa,
    double* __restrict__ data, double* __restrict__ b) {
  constexpr int NV = D + 1, NDP = Space<D, KP>::ND, NM = NeumannSpace<D>::NM;
  __shared__ double qlam[kMaxQuadPoints * NV], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * NV; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cut * NM) return;
  const int64_t ec = t / NM;
  const int a = (int)(t - ec * NM);
  const int64_t e = __ldg(cut_positions + ec);
  const int64_t c = __ldg(active + e);
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double pc[NDP], fc[NV], uc[NV];
  load_dofs<D, KP>(m, sp, phi, c, pc);
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int v = __ldg(m.cells + c * NV + k);
    fc[k] = __ldg(f + v);
    uc[k] = __ldg(un + v);
  }
  const double h = sqrt(g.h2), rh = 1.0 / h, rh2 = 1.0 / g.h2;
  const double pen = gamma;
  double A[NM], bv = 0.0;
#pragma unroll
  for (int j = 0; j < NM; ++j) A[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) lam[k] = qlam[q * NV + k];
    const double w = qw[q] * g.vol;
    double ph, gph[D];
    eval_phi_only<D, KP>(lam, g.G, pc, ph, gph);
    double fq = 0.0, uq = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      fq += fc[k] * lam[k];
      uq += uc[k] * lam[k];
    }
    const double ngp = sqrt(dotd<D>(gph, gph));
    double Ua, GUa[D], S1a[D], S2a, S3a;
    neumann_basis<D>(a, lam, g.G, gph, ph * rh, kappa * ngp, Ua, GUa, S1a, S2a, S3a);
    bv += w * (fq * Ua + pen * (fq * S2a - rh2 * uq * ngp * S3a));
#pragma unroll
    for (int bb = 0; bb < NM; ++bb) {
      double Ub, GUb[D], S1b[D], S2b, S3b;
      neumann_basis<D>(bb, lam, g.G, gph, ph * rh, kappa * ngp, Ub, GUb, S1b, S2b, S3b);
      A[bb] += w * (dotd<D>(GUa, GUb) + Ua * Ub + pen * (dotd<D>(S1a, S1b) + S2a * S2b + rh2 * S3a * S3b));
    }
  }
  atomicAdd(b + __ldg(mixed_dofmap + c * NM + a), bv);
#pragma unroll
  for (int bb = 0; bb < NM; ++bb)
    atomicAdd(data + __ldg(slots + (int64_t)(a * NM + bb) * n_active + e), A[bb]);
}

// int_{ds(100)} (y.n) v: one thread per (entity, u test dof i); columns y_(j,c)
template <int D>
__global__ void __launch_bounds__(kBlockPk) k_assemble_boundary_neumann(
    phifem_mesh m, const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ slots,
    double* __restrict__ data) {
  constexpr int NV = D + 1, NM = NeumannSpace<D>::NM;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * NV) return;
  const int64_t e = t / NV;
  const int i = (int)(t - e * NV);
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  if (i == o) return;  // v_i vanishes on the facet opposite vertex i
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double n[D], area;
  facet_normal<D>(g, o, n, area);
  const double cF = area * (1.0 / (D * (D + 1)));  // facet mass matrix |F| (1 + delta_ij) / (D (D+1))
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    if (j == o) continue;
    const double mij = cF * (i == j ? 2.0 : 1.0);
#pragma unroll
    for (int cc = 0; cc < D; ++cc)
      atomicAdd(data + __ldg(slots + (e * NM + i) * NM + NV + j * D + cc), n[cc] * mij);
  }
}

int check_pk(const phifem_mesh* m, const phifem_pk_space* sw, const phifem_pk_space* sp,
             const double* points, const double* weights, int nq) {
  PHIFEM_CHECK_ARG(m != nullptr && m->x && m->cells, "mesh is null");
  if (m->cell_type != PHIFEM_TRIANGLE && m->cell_type != PHIFEM_TETRAHEDRON) {
    set_error("P_k assembly supports triangles and tetrahedra, got cell type %d", m->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  const int D = m->cell_type == PHIFEM_TRIANGLE ? 2 : 3;
  PHIFEM_CHECK_ARG(m->gdim == D, "gdim mismatch");
  PHIFEM_CHECK_ARG(sw && sp, "function spaces are null");
  for (const phifem_pk_space* s : {sw, sp}) {
    if (s->degree != 1 && s->degree != 2) {
      set_error("P_k assembly implements degrees 1 and 2, got %d", s->degree);
      return PHIFEM_ERR_UNSUPPORTED;
    }
    const int nd = s->degree == 1 ? D + 1 : (D + 1) + D * (D + 1) / 2;
    PHIFEM_CHECK_ARG(s->n_dofs_per_cell == nd, "n_dofs_per_cell does not match the degree");
    PHIFEM_CHECK_ARG(s->dofmap || s->degree == 1, "a P2 space needs its dofmap");
  }
  PHIFEM_CHECK_ARG(points && weights && nq > 0 && nq <= kMaxQuadPoints, "quadrature rule (1..128 points)");
  return PHIFEM_OK;
}

// the strong-Dirichlet operator on quadrilaterals: a Q1 trial / test space, a Q1 or Q2 level set
int check_quad_strong(const phifem_mesh* m, const phifem_pk_space* sw, const phifem_pk_space* sp,
                      const double* points, const double* weights, int nq) {
  PHIFEM_CHECK_ARG(m->x && m->cells && m->gdim == 2, "quadrilateral mesh needs x, cells and gdim 2");
  PHIFEM_CHECK_ARG(sw && sp, "function spaces are null");
  if (sw->degree != 1) {
    set_error("the strong-Dirichlet operator on quadrilaterals implements a Q1 trial space, got degree %d", sw->degree);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(sw->n_dofs_per_cell == 4, "space_w->n_dofs_per_cell must be 4 (Q1) on quadrilaterals");
  PHIFEM_CHECK_ARG(sp->n_dofs_per_cell == 4 || sp->n_dofs_per_cell == 9,
                   "space_phi->n_dofs_per_cell must be 4 (Q1) or 9 (Q2) on quadrilaterals");
  PHIFEM_CHECK_ARG(sp->degree == (sp->n_dofs_per_cell == 4 ? 1 : 2),
                   "space_phi->degree does not match n_dofs_per_cell on quadrilaterals");
  PHIFEM_CHECK_ARG(sp->dofmap || sp->degree == 1, "a Q2 level set on quadrilaterals needs its dofmap");
  PHIFEM_CHECK_ARG(points && weights && nq > 0 && nq <= kMaxQuadPoints, "quadrature rule (1..128 points)");
  return PHIFEM_OK;
}

// instantiate kernel<D, KW, KP> for the runtime (cell type, degrees)
template <typename F>
void dispatch(int cell_type, int kw, int kp, F&& f) {
  auto with_d = [&](auto d) {
    constexpr int D = decltype(d)::value;
    if (kw == 1 && kp == 1) f(d, std::integral_constant<int, 1>{}, std::integral_constant<int, 1>{});
    else if (kw == 1) f(d, std::integral_constant<int, 1>{}, std::integral_constant<int, 2>{});
    else if (kp == 1) f(d, std::integral_constant<int, 2>{}, std::integral_constant<int, 1>{});
    else f(d, std::integral_constant<int, 2>{}, std::integral_constant<int, 2>{});
    (void)D;
  };
  if (cell_type == PHIFEM_TRIANGLE) with_d(std::integral_constant<int, 2>{});
  else with_d(std::integral_constant<int, 3>{});
}

}  // namespace

// the Neumann operator on quadrilaterals (bilinear cell map): csrc/assemble_quad.cu
int quad_neumann_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                       const double* phi, const double* f, const double* u_n, const int8_t* cell_tags8,
                       const int32_t* active, int64_t n_active, const int32_t* cut_positions, int64_t n_cut,
                       const int32_t* slots, const int32_t* mixed_dofmap, double gamma, double robin_coef,
                       double* data, double* b, cudaStream_t st);
int quad_neumann_boundary(const phifem_mesh* mesh, const int32_t* entities, int64_t n_entities, const int32_t* slots,
                          double* data, cudaStream_t st);
int quad_neumann_ghost(const phifem_mesh* mesh, const phifem_quadrature* quad_rule, const int32_t* facets,
                       int64_t n_facets, const int32_t* slots, double sigma, double* data, cudaStream_t st);
// the strong-Dirichlet operator on quadrilaterals (Q1 trial / test space): csrc/assemble_quad.cu
int quad_strong_cells(const phifem_mesh* mesh, const phifem_pk_space* space_w, const phifem_pk_space* space_phi,
                      const phifem_quadrature* quad_rule, const double* phi, const double* f, const int8_t* cell_tags8,
                      const int32_t* active, int64_t n_active, const int32_t* slots, double sigma, double* data,
                      double* b, cudaStream_t st);
int quad_strong_boundary(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                         const double* phi, const int32_t* entities, int64_t n_entities, const int32_t* slots,
                         double* data, cudaStream_t st);
int quad_strong_ghost(const phifem_mesh* mesh, const phifem_pk_space* space_phi, const phifem_quadrature* quad_rule,
                      const double* phi, const int32_t* facets, int64_t n_facets, const int32_t* slots, double sigma,
                      double* data, cudaStream_t st);
}  // namespace phifem

using namespace phifem;

extern "C" int phifem_assemble_cells_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                        const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                        const double* phi, const double* f, const int8_t* cell_tags8,
                                        const int32_t* active, int64_t n_active, const int32_t* slots,
                                        double sigma, double* data, double* b, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (mesh != nullptr && mesh->cell_type == PHIFEM_QUADRILATERAL) {
    if (int rc = check_quad_strong(mesh, space_w, space_phi, quad->cell_points, quad->cell_weights,
                                   quad->n_cell_points))
      return rc;
    if (n_active == 0) return PHIFEM_OK;
    PHIFEM_CHECK_ARG(phi && f && cell_tags8 && data && b && active && slots, "null pointer");
    return quad_strong_cells(mesh, space_w, space_phi, quad, phi, f, cell_tags8, active, n_active, slots, sigma, data,
                             b, (cudaStream_t)stream);
  }
  if (int rc = check_pk(mesh, space_w, space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points))
    return rc;
  if (n_active == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && f && cell_tags8 && data && b, "null pointer");
  PHIFEM_CHECK_ARG(active && slots, "null active / slots");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, space_phi->degree, [&](auto d, auto kw, auto kp) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value, KP = decltype(kp)::value;
    const dim3 grid((unsigned)((n_active + kBlockPkCells - 1) / kBlockPkCells), Passes<Space<D, KW>::ND>::N);
    k_assemble_cells_pk<D, KW, KP><<<grid, kBlockPkCells, 0, st>>>(
        *mesh, *space_w, *space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points, phi, f,
        cell_tags8, active, n_active, slots, sigma, data, b);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_boundary_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                           const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                           const double* phi, const int32_t* entities, int64_t n_entities,
                                           const int32_t* slots, double* data, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (mesh != nullptr && mesh->cell_type == PHIFEM_QUADRILATERAL) {
    if (int rc = check_quad_strong(mesh, space_w, space_phi, quad->facet_points, quad->facet_weights,
                                   quad->n_facet_points))
      return rc;
    if (n_entities == 0) return PHIFEM_OK;
    PHIFEM_CHECK_ARG(phi && data && entities && slots, "null pointer");
    return quad_strong_boundary(mesh, space_phi, quad, phi, entities, n_entities, slots, data, (cudaStream_t)stream);
  }
  if (int rc = check_pk(mesh, space_w, space_phi, quad->facet_points, quad->facet_weights, quad->n_facet_points))
    return rc;
  if (n_entities == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && data, "null pointer");
  PHIFEM_CHECK_ARG(entities && slots, "null entities / slots");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, space_phi->degree, [&](auto d, auto kw, auto kp) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value, KP = decltype(kp)::value;
    const int64_t threads = n_entities * Space<D, KW>::ND;
    k_assemble_boundary_pk<D, KW, KP><<<(unsigned)((threads + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, *space_w, *space_phi, quad->facet_points, quad->facet_weights, quad->n_facet_points, phi,
        entities, n_entities, slots, data);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_ghost_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                        const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                        const double* phi, const int32_t* facets, int64_t n_facets,
                                        const int32_t* slots, double sigma, double* data, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (mesh != nullptr && mesh->cell_type == PHIFEM_QUADRILATERAL) {
    if (int rc = check_quad_strong(mesh, space_w, space_phi, quad->facet_points, quad->facet_weights,
                                   quad->n_facet_points))
      return rc;
    if (n_facets == 0) return PHIFEM_OK;
    PHIFEM_CHECK_ARG(phi && data && mesh->c2f && mesh->f2c && facets && slots, "null pointer");
    return quad_strong_ghost(mesh, space_phi, quad, phi, facets, n_facets, slots, sigma, data, (cudaStream_t)stream);
  }
  if (int rc = check_pk(mesh, space_w, space_phi, quad->facet_points, quad->facet_weights, quad->n_facet_points))
    return rc;
  if (n_facets == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && data && mesh->c2f && mesh->f2c, "null pointer");
  PHIFEM_CHECK_ARG(facets && slots, "null facets / slots");
  PHIFEM_CHECK_ARG(quad->n_facet_points <= 32, "the ghost-penalty kernel holds at most 32 facet points");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, space_phi->degree, [&](auto d, auto kw, auto kp) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value, KP = decltype(kp)::value;
    constexpr int FPB = GhostLayout<D, KW>::FPB, NM = GhostLayout<D, KW>::NM;
    const int nq = quad->n_facet_points;
    const size_t smem = sizeof(double) * ((size_t)nq * (D + 1) + (size_t)FPB * nq * (NM + 2 * (D + 3)));
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(k_assemble_ghost_pk<D, KW, KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_assemble_ghost_pk<D, KW, KP><<<(unsigned)((n_facets + FPB - 1) / FPB), kBlockPk, smem, st>>>(
        *mesh, *space_w, *space_phi, quad->facet_points, quad->facet_weights, quad->n_facet_points, phi,
        facets, n_facets, slots, sigma, data);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

// ---- weak-Dirichlet operator (demo/weak-dirichlet/flower/main.py:112-151) ---------------------------------------
extern "C" int phifem_assemble_weak_cells_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                             const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                             const double* phi, const double* f, const double* u_d,
                                             const int8_t* cell_tags8, const int32_t* active, int64_t n_active,
                                             const int32_t* slots, const int32_t* mixed_dofmap, double gamma,
                                             double sigma, double* data, double* b, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (int rc = check_pk(mesh, space_w, space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points))
    return rc;
  if (n_active == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && f && u_d && cell_tags8 && data && b && mixed_dofmap, "null pointer");
  PHIFEM_CHECK_ARG(active && slots, "null active / slots");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, space_phi->degree, [&](auto d, auto kw, auto kp) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value, KP = decltype(kp)::value;
    const int64_t threads = n_active * 2 * Space<D, KW>::ND;
    k_assemble_cells_weak_pk<D, KW, KP><<<(unsigned)((threads + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, *space_w, *space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points, phi, f, u_d,
        cell_tags8, active, n_active, slots, mixed_dofmap, gamma, sigma, data, b);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_weak_boundary_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                                const phifem_quadrature* quad, const int32_t* entities,
                                                int64_t n_entities, const int32_t* slots, double* data,
                                                void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (int rc = check_pk(mesh, space_w, space_w, quad->facet_points, quad->facet_weights, quad->n_facet_points))
    return rc;
  if (n_entities == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(data != nullptr, "null pointer");
  PHIFEM_CHECK_ARG(entities && slots, "null entities / slots");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, 1, [&](auto d, auto kw, auto) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value;
    const int64_t threads = n_entities * Space<D, KW>::ND;
    k_assemble_boundary_weak_pk<D, KW><<<(unsigned)((threads + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, quad->facet_points, quad->facet_weights, quad->n_facet_points, entities, n_entities, slots, data);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_weak_ghost_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                             const phifem_quadrature* quad, const int32_t* facets,
                                             int64_t n_facets, const int32_t* slots, double sigma, double* data,
                                             void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (int rc = check_pk(mesh, space_w, space_w, quad->facet_points, quad->facet_weights, quad->n_facet_points))
    return rc;
  if (n_facets == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(data && mesh->c2f && mesh->f2c, "null pointer");
  PHIFEM_CHECK_ARG(facets && slots, "null facets / slots");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, space_w->degree, 1, [&](auto d, auto kw, auto) {
    constexpr int D = decltype(d)::value, KW = decltype(kw)::value;
    const int64_t threads = n_facets * 2 * Space<D, KW>::ND;
    k_assemble_ghost_weak_pk<D, KW><<<(unsigned)((threads + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, quad->facet_points, quad->facet_weights, quad->n_facet_points, facets, n_facets, slots, sigma,
        data);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

// ---- Neumann operator (demo/neumann/square/main.py:103-158) --------------------------------------------------------
extern "C" int phifem_assemble_neumann_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi,
                                             const phifem_quadrature* quad, const double* phi, const double* f,
                                             const double* u_n, const int8_t* cell_tags8, const int32_t* active,
                                             int64_t n_active, const int32_t* cut_positions, int64_t n_cut,
                                             const int32_t* slots, const int32_t* mixed_dofmap, double gamma,
                                             double robin_coef, double* data, double* b, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr && space_phi != nullptr, "quadrature / level-set space is null");
  if (mesh != nullptr && mesh->cell_type == PHIFEM_QUADRILATERAL) {
    PHIFEM_CHECK_ARG(mesh->x && mesh->cells && mesh->gdim == 2, "quadrilateral mesh needs x, cells and gdim 2");
    PHIFEM_CHECK_ARG(space_phi->n_dofs_per_cell == 4 || space_phi->n_dofs_per_cell == 9,
                     "space_phi->n_dofs_per_cell must be 4 (Q1) or 9 (Q2) on quadrilaterals");
    PHIFEM_CHECK_ARG(space_phi->degree == (space_phi->n_dofs_per_cell == 4 ? 1 : 2),
                     "space_phi->degree does not match n_dofs_per_cell");
    PHIFEM_CHECK_ARG(space_phi->dofmap || space_phi->degree == 1, "a Q2 level set needs its dofmap");
    PHIFEM_CHECK_ARG(quad->cell_points && quad->cell_weights && quad->n_cell_points > 0 &&
                         quad->n_cell_points <= kMaxQuadPoints, "quadrature rule (1..128 points)");
    if (n_active == 0) return PHIFEM_OK;
    PHIFEM_CHECK_ARG(phi && f && u_n && cell_tags8 && data && b && mixed_dofmap && active && slots, "null pointer");
    PHIFEM_CHECK_ARG(n_cut >= 0 && n_cut <= n_active && (n_cut == 0 || cut_positions), "cut-cell positions");
    return quad_neumann_cells(mesh, space_phi, quad, phi, f, u_n, cell_tags8, active, n_active, cut_positions, n_cut,
                              slots, mixed_dofmap, gamma, robin_coef, data, b, (cudaStream_t)stream);
  }
  phifem_pk_space p1{1, mesh && mesh->cell_type == PHIFEM_TRIANGLE ? 3 : 4, 0, nullptr};
  if (int rc = check_pk(mesh, &p1, space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points)) return rc;
  if (n_active == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && f && u_n && cell_tags8 && data && b && mixed_dofmap && active && slots, "null pointer");
  PHIFEM_CHECK_ARG(n_cut >= 0 && n_cut <= n_active && (n_cut == 0 || cut_positions), "cut-cell positions");
  cudaStream_t st = (cudaStream_t)stream;
  dispatch(mesh->cell_type, 1, space_phi->degree, [&](auto d, auto, auto kp) {
    constexpr int D = decltype(d)::value, KP = decltype(kp)::value;
    const int64_t light = n_active * (D + 1);
    k_assemble_interior_neumann<D><<<(unsigned)((light + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, f, cell_tags8, active, n_active, slots, mixed_dofmap, data, b);
    if (n_cut == 0) return;
    const int64_t threads = n_cut * NeumannSpace<D>::NM;
    k_assemble_cells_neumann<D, KP><<<(unsigned)((threads + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, *space_phi, quad->cell_points, quad->cell_weights, quad->n_cell_points, phi, f, u_n, active, n_active,
        cut_positions, n_cut, slots, mixed_dofmap, gamma, robin_coef, data, b);
  });
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_neumann_boundary(const phifem_mesh* mesh, const int32_t* entities,
                                                int64_t n_entities, const int32_t* slots, double* data,
                                                void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->x && mesh->cells, "mesh is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON &&
      mesh->cell_type != PHIFEM_QUADRILATERAL) {
    set_error("the Neumann operator supports triangles, quadrilaterals and tetrahedra, got cell type %d",
              mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  if (n_entities == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(entities && slots && data, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (mesh->cell_type == PHIFEM_QUADRILATERAL) {
    PHIFEM_CHECK_ARG(mesh->gdim == 2, "gdim mismatch");
    return quad_neumann_boundary(mesh, entities, n_entities, slots, data, st);
  }
  if (mesh->cell_type == PHIFEM_TRIANGLE)
    k_assemble_boundary_neumann<2><<<(unsigned)((n_entities * 3 + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, entities, n_entities, slots, data);
  else
    k_assemble_boundary_neumann<3><<<(unsigned)((n_entities * 4 + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, entities, n_entities, slots, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_neumann_ghost(const phifem_mesh* mesh, const phifem_quadrature* quad,
                                             const int32_t* facets, int64_t n_facets, const int32_t* slots,
                                             double sigma, double* data, void* stream) {
  PHIFEM_CHECK_ARG(quad != nullptr, "quadrature is null");
  if (mesh != nullptr && mesh->cell_type == PHIFEM_QUADRILATERAL) {
    PHIFEM_CHECK_ARG(mesh->x && mesh->cells && mesh->gdim == 2, "quadrilateral mesh needs x, cells and gdim 2");
    PHIFEM_CHECK_ARG(quad->facet_points && quad->facet_weights && quad->n_facet_points > 0 &&
                         quad->n_facet_points <= kMaxQuadPoints, "quadrature rule (1..128 points)");
    if (n_facets == 0) return PHIFEM_OK;
    PHIFEM_CHECK_ARG(data && mesh->c2f && mesh->f2c && facets && slots, "null pointer");
    return quad_neumann_ghost(mesh, quad, facets, n_facets, slots, sigma, data, (cudaStream_t)stream);
  }
  phifem_pk_space p1{1, mesh && mesh->cell_type == PHIFEM_TRIANGLE ? 3 : 4, 0, nullptr};
  if (int rc = check_pk(mesh, &p1, &p1, quad->facet_points, quad->facet_weights, quad->n_facet_points)) return rc;
  if (n_facets == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(data && mesh->c2f && mesh->f2c && facets && slots, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (mesh->cell_type == PHIFEM_TRIANGLE) {
    constexpr int NM = NeumannSpace<2>::NM;
    k_assemble_ghost_weak_pk<2, 1, NM><<<(unsigned)((n_facets * 6 + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, quad->facet_points, quad->facet_weights, quad->n_facet_points, facets, n_facets, slots, sigma, data);
  } else {
    constexpr int NM = NeumannSpace<3>::NM;
    k_assemble_ghost_weak_pk<3, 1, NM><<<(unsigned)((n_facets * 8 + kBlockPk - 1) / kBlockPk), kBlockPk, 0, st>>>(
        *mesh, quad->facet_points, quad->facet_weights, quad->n_facet_points, facets, n_facets, slots, sigma, data);
  }
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}
