// K2+K3+K4 fused, row-gather form: strong-Dirichlet phi-FEM operator, P1 on triangles / tetrahedra,
// one thread per CSR row.
//
// Forms of reference demo/strong-dirichlet/flower/main.py:104-128 (closed-form element tensors of
// SURVEY.md Appendix B).  dolfinx loops over cells and ADDs 4x4 blocks into PETSc AIJ rows
// (main.py:121-123); a GPU doing the same issues 20 fp64 reductions per tetrahedron, and the SM retires
// less than one reduction lane per clock (profiles/: 1.74 ms for 19.8 M cells, fp64 pipe 14 % busy).
// Here the loop is turned around: the thread owning row r walks the entities touching vertex r and
// evaluates only ITS row of each element tensor (1.8x the fp64 work of the cell loop, which the idle
// fp64 pipe absorbs), accumulating in registers (diagonal, load vector) and in a private, bank-conflict
// free column of shared memory (off-diagonals).  One plain store per CSR entry at the end: no atomics,
// no zero-fill, bitwise reproducible, and every rank of a multi-GPU run can own rows outright.
//
// Connectivity comes from the CSR pattern itself: a record holds the positions inside row r's column
// list of the entity's other vertices, so `indices[start + pos]` names them (include/phifem_b200.h).
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "p1_forms.cuh"

namespace phifem {
namespace {

// 64 threads x 8 CTAs per SM (the same 16 warps and 128 registers as 128 x 4): cell pass 1.200 -> 1.174 ms at config E
// (profiles/round2_i_rows_variants.md, tools/r3_run_h.sh) -- half the accumulator slab per CTA, finer-grained tail
constexpr int kRowsBlock = 64;
constexpr int kRowsMinBlocks = 512 / kRowsBlock;
constexpr uint32_t kPad = 0xffffffffu;

// Row 0 of the cell tensor of simplex X (local vertex 0 = the row's vertex): dx((1,2)) stiffness,
// dx(2) stabilisation (main.py:105,107-112) and entry 0 of the load vector (:126-128).
// Appendix B closed forms with every gradient left scaled by det (G = R / det), so that one reciprocal
// and ~125 fp64 operations give the row:
//   K_j = |K|/((d+1)(d+2)) [ |g|^2 (1 + delta_0j) + a_0 (P + p_j) + (P + p_0) a_j + G_0.G_j mu ]
//         + 4 sigma h^2 |K| a_0 a_j,     g = grad(phi), a_j = g.G_j, P = sum p, mu = P^2 + sum p^2.
template <int D>
__device__ __forceinline__ void cell_row(const double (&X)[D + 1][D], const double (&p)[D + 1],
                                         const double (&fv)[D + 1], bool is_cut, double sigma,
                                         double (&K)[D + 1], double& b0) {
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
  double aR[NV], c0[NV];  // det^2 * a_j, det^2 * G_0.G_j
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    aR[j] = dot<D>(gR, R[j]);
    c0[j] = dot<D>(R[0], R[j]);
  }
  const double ggR = dot<D>(gR, gR);
  double P = p[0], S2 = p[0] * p[0], F = fv[0], FP = fv[0] * p[0];
#pragma unroll
  for (int k = 1; k < NV; ++k) {
    P += p[k];
    S2 += p[k] * p[k];
    F += fv[k];
    FP += fv[k] * p[k];
  }
  const double mu = P * P + S2;
  const double ainv = fabs(inv), adet = fabs(det);
  const double w = ainv * (1.0 / (dfact * (D + 1) * (D + 2)));
  const double P0 = P + p[0];
  double sh2 = 0.0;  // sigma h_T^2 on cut cells
  if (is_cut) sh2 = sigma * diameter2<D>(X);
  const double sR = (4.0 / dfact) * sh2 * ainv * (inv * inv) * aR[0];  // 4 sigma h^2 |K| a_0 / det^2
#pragma unroll
  for (int j = 0; j < NV; ++j)
    K[j] = w * (ggR * (j == 0 ? 2.0 : 1.0) + aR[0] * (P + p[j]) + P0 * aR[j] + c0[j] * mu) + sR * aR[j];
  constexpr double fact_d3 = D == 2 ? 120.0 : 720.0;
  b0 = adet * ((1.0 / fact_d3) * ((F * P + FP) + fv[0] * P + F * p[0] + 2.0 * fv[0] * p[0]) -
               (2.0 / (dfact * NV)) * sh2 * F * aR[0] * (inv * inv));
}

// The same row from cached geometry (phifem_rows_plan.cell_geom): the forms see the cell only through its P1
// stiffness matrix S_ab = |K| grad(lambda_a).grad(lambda_b), |K| and h_T^2, which depend on the mesh alone and are
// tabulated once per plan: 8 doubles per active cell = [S_ab for a < b in lexicographic order, |K|, h_T^2, pad].
// With A_j = |K| grad(phi).grad(lambda_j) = sum_k (p_k - p_j) S_kj (rows of S sum to zero) and gg = |K| |grad(phi)|^2
// = sum_j p_j A_j:
//   K_j = [ gg (1 + delta_0j) + A_0 (P + p_j) + (P + p_0) A_j + S_0j mu ] / ((d+1)(d+2)) + 4 sigma h^2 A_0 A_j / |K|,
//   b_0 = |K| d!/(d+3)! [ F P + sum f_k p_k + f_0 P + F p_0 + 2 f_0 p_0 ] - 2 sigma h^2 F A_0 / (d+1),
// ~85 fp64 instructions instead of ~146 (no cofactors, no reciprocal off the cut cells), no coordinate gathers.
// MEASURED SLOWER on the B200 at config E (cell pass 1.74 ms against 1.20 ms; profiles/round2_a_geometry_kernel.md): the
// fp64 pipe falls from 56 % to 17 % busy, but the warp-instruction count does not (706 M against 734 M: selects for
// the row permutation, register moves) and the 64-byte table record of a cell -- read by D + 1 rows that run far apart in
// time -- misses L1 (hit rate 42 % against 88 % for the coordinates, which neighbouring rows share), so every record
// waits for an L2 round trip with one record of lead (long-scoreboard stalls 6.6 per issue against 0.9).  Requesting the
// table line 6 records ahead with prefetch.global.L2 made it 2.05 ms.  Kept as an option of the plan
// (`geometry=True`), off by default.
// Slot order: slot 0 = the row's vertex = cell-local vertex i, slot s >= 1 = the (s-1)-th other vertex in ascending
// local order (the order of the record's position bytes).
template <int NV> __host__ __device__ constexpr int geom_slot_to_local(int i, int s) {
  return s == 0 ? i : (s - 1 < i ? s - 1 : s);
}
template <int NV> __host__ __device__ constexpr int geom_stored(int x, int y) {  // index of S_xy, x != y
  return x < y ? x * (2 * NV - x - 1) / 2 + (y - x - 1) : y * (2 * NV - y - 1) / 2 + (x - y - 1);
}

template <int D>
__device__ __forceinline__ void cell_row_geom(const double (&g)[8], int i, const double (&p)[D + 1],
                                              const double (&fv)[D + 1], bool is_cut, double sigma,
                                              double (&K)[D + 1], double& b0) {
  constexpr int NV = D + 1, NO = NV * D / 2;
  double S[NV][NV];
#pragma unroll
  for (int a = 0; a < NV; ++a)
#pragma unroll
    for (int c = a + 1; c < NV; ++c) {
      double v = g[geom_stored<NV>(geom_slot_to_local<NV>(0, a), geom_slot_to_local<NV>(0, c))];
#pragma unroll
      for (int ii = 1; ii < NV; ++ii)
        if (i == ii) v = g[geom_stored<NV>(geom_slot_to_local<NV>(ii, a), geom_slot_to_local<NV>(ii, c))];
      S[a][c] = v;
    }
  const double vol = g[NO], h2 = g[NO + 1];
  double dp[NV][NV];  // p_a - p_c, a < c
#pragma unroll
  for (int a = 0; a < NV; ++a)
#pragma unroll
    for (int c = a + 1; c < NV; ++c) dp[a][c] = p[a] - p[c];
  double A[NV];
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (k < j) s += dp[k][j] * S[k][j];
      if (k > j) s -= dp[j][k] * S[j][k];
    }
    A[j] = s;
  }
  double gg = p[0] * A[0], P = p[0], S2 = p[0] * p[0], F = fv[0], FP = fv[0] * p[0], S00 = S[0][1];
#pragma unroll
  for (int k = 1; k < NV; ++k) {
    gg += p[k] * A[k];
    P += p[k];
    S2 += p[k] * p[k];
    F += fv[k];
    FP += fv[k] * p[k];
    if (k > 1) S00 += S[0][k];
  }
  const double mu = P * P + S2, P0 = P + p[0];
  constexpr double cm = 1.0 / ((D + 1) * (D + 2));
  constexpr double cb = D == 2 ? 1.0 / 60.0 : 1.0 / 120.0;  // d!/(d+3)!
  double sR = 0.0, sb = 0.0;
  if (is_cut) {
    const double sh2 = sigma * h2;
    sR = 4.0 * sh2 * A[0] / vol;
    sb = (2.0 / NV) * sh2 * F * A[0];
  }
  K[0] = cm * (2.0 * gg + 2.0 * A[0] * P0 - S00 * mu) + sR * A[0];
#pragma unroll
  for (int j = 1; j < NV; ++j) K[j] = cm * (gg + A[0] * (P + p[j]) + P0 * A[j] + S[0][j] * mu) + sR * A[j];
  b0 = vol * cb * ((F * P + FP) + fv[0] * P + F * p[0] + 2.0 * fv[0] * p[0]) - sb;
}

__device__ __forceinline__ double alpha3(int a, int b, int c) {
  return (double)((1 + (a == b)) * (1 + (a == c) + (b == c)));
}

// One-sided term -int_F (grad(phi w).n) phi v (main.py:106) on a (cell, local facet) entity of ds(100), in the same two
// phases as the ghost penalty.  Entity-once (k_surface_once_p1): with the cell's vertices listed as
// [facet vertices 0..D-1, opposite vertex], n = the outward normal of THIS cell (tests/test_one_sided_integral.py pins
// it), cF = |F| (D-1)!/(D+2)!, the thread stores cF grad(phi).n, cF grad(lambda_j).n for the D + 1 vertices and phi at
// the facet vertices: 2 D + 2 doubles.  Per row (facet vertex t): with the facet vertices rotated so that the row's
// vertex comes first, entry (0, j) = -[ (cF gn) W_j + (cF Gn_j) Q ],  W_j = sum_k phi_k alpha(j,k,0) for j on the
// facet (0 for the opposite vertex), Q = sum_kl phi_k phi_l alpha(l,k,0), alpha = the multiplicity factor of
// int lambda_a lambda_b lambda_c over the facet.
template <int D>
__device__ __forceinline__ void entity_record(const double (&X)[D + 1][D], const double (&p)[D + 1],
                                              double* __restrict__ w) {
  constexpr int NV = D + 1;
  double G[NV][D], det;
  simplex_gradients<D>(X, G, det);
  const double vol = fabs(det) * volume_factor<D>();
  const double gnorm = sqrt(dot<D>(G[D], G[D]));
  double n[D], g[D];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    n[d] = -G[D][d] / gnorm;
    double s = p[0] * G[0][d];
#pragma unroll
    for (int k = 1; k < NV; ++k) s += p[k] * G[k][d];
    g[d] = s;
  }
  constexpr double cfac = D == 2 ? 1.0 / 24.0 : 2.0 / 120.0;  // (d-1)!/(d+2)!
  const double cF = D * vol * gnorm * cfac;
  w[0] = cF * dot<D>(g, n);
#pragma unroll
  for (int j = 0; j < NV; ++j) w[1 + j] = cF * dot<D>(G[j], n);
#pragma unroll
  for (int k = 0; k < D; ++k) w[2 + D + k] = p[k];
  if (D == 2) w[6] = w[7] = 0.0;
}

// Row of facet vertex t from the entity's record: K[0] = diagonal, K[1..D-1] = facet vertices (t + j) % D,
// K[D] = the opposite vertex.
template <int D>
__device__ __forceinline__ void entity_row(const double (&wk)[8], int t, double (&K)[D + 1]) {
  double p[D], Gn[D];
#pragma unroll
  for (int k = 0; k < D; ++k) {  // rotate: index k <- (t + k) % D
    double pv = wk[2 + D + k], gv = wk[1 + k];
#pragma unroll
    for (int s = 1; s < D; ++s)
      if (t == s) {
        pv = wk[2 + D + (k + s) % D];
        gv = wk[1 + (k + s) % D];
      }
    p[k] = pv;
    Gn[k] = gv;
  }
  double Q = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k)
#pragma unroll
    for (int l = 0; l < D; ++l) Q += p[k] * p[l] * alpha3(l, k, 0);
#pragma unroll
  for (int j = 0; j < D; ++j) {
    double W = 0.0;
#pragma unroll
    for (int k = 0; k < D; ++k) W += p[k] * alpha3(j, k, 0);
    K[j] = -(wk[0] * W + Gn[j] * Q);
  }
  K[D] = -wk[1 + D] * Q;
}

// Ghost penalty sigma avg(h_T) int_F jump.jump (main.py:113-118) over the facet macro element
// M = [facet vertices 0..D-1 (as ordered in cell A = f2c[f][0]), opposite vertex of cell A, opposite vertex of
// cell B].  Two phases, both without atomics:
//   facet-once (k_surface_once_p1): with N = the facet's cofactor vector (normal scaled by (D-1)! |F|, the same
//     for both cells) the normal derivative of lambda_a seen from cell s is Gn_a = -(R_a . N) / (|det_s| |N|);
//     the jump of grad(phi w_m).n at a point of F is  lambda_m [m on F] gsum + phi c_m  with
//     gsum = sum_s grad(phi).n_s and c_m = sum_s Gn_m (sum_m c_m = 0: the barycentric gradients of a cell sum
//     to zero).  With s = sqrt(|sigma| avg(h) |F| / (D (D+1))) the thread stores s c_0..s c_D, s gsum and phi at
//     the facet vertices: 8 doubles = 64 bytes per facet (two 256-bit loads for a row), 93 MB for the 1.45 M
//     ghost facets of config E;
//   per row (k_assemble_rows_p1<D, kSurface>): the facet mass matrix |F| (1 + delta_kl) / (D (D+1)) gives
//     entry (a, m) = sign(sigma) [ (ga + c_a Pf)(gm + c_m Pf) + c_a c_m Sf2 + ga c_m phi_a + c_a gm phi_m
//                                  + ga gm delta_am ],  ga = s gsum if a lies on F else 0, Pf = sum phi_k,
//     Sf2 = sum phi_k^2 over the facet vertices: ~50 fp64 operations per row instead of ~300.
// The pass is bound by the L1 request rate of the per-lane record gathers (ncu: 6 x 128-bit loads per record
// cost 0.20 ms, 3 x 256-bit 0.16 ms), hence the compact record.
template <int D> constexpr int kGhostWork = 8;  // D + 1 jump coefficients, gsum, D facet values (+ pad in 2D)

// sm_100 256-bit read-only load (LDG.E.256): one L1 request per 32-byte sector instead of two
__device__ __forceinline__ void ldg256(const double* p, double& a, double& b, double& c, double& d) {
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}

template <int D>
__global__ void __launch_bounds__(kRowsBlock, 1) k_surface_once_p1(
    const double* __restrict__ x, const double* __restrict__ phi, double sigma,
    const int32_t* __restrict__ macro, int64_t n_facets, const int32_t* __restrict__ entity_macro,
    int64_t n_entities, double* __restrict__ work) {
  constexpr int NV = D + 1, NG = D + 2, W = kGhostWork<D>;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_facets + n_entities) return;
  if (g >= n_facets) {  // one-sided entity: record index n_facets + e
    const int64_t e = g - n_facets;
    double X[NV][D], p[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = __ldg(entity_macro + e * NV + k);
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = __ldg(x + (int64_t)v * D + d);
      p[k] = __ldg(phi + v);
    }
    entity_record<D>(X, p, work + g * W);
    return;
  }
  double M[NG][D], pm[NG];
#pragma unroll
  for (int m = 0; m < NG; ++m) {
    const int v = __ldg(macro + g * NG + m);
#pragma unroll
    for (int d = 0; d < D; ++d) M[m][d] = __ldg(x + (int64_t)v * D + d);
    pm[m] = __ldg(phi + v);
  }
  double c[NG], N[D], nn = 0.0, rn = 0.0, gsum = 0.0, hsum = 0.0;
#pragma unroll
  for (int m = 0; m < NG; ++m) c[m] = 0.0;
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    double X[NV][D], p[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int m = k < D ? k : D + side;
      p[k] = pm[m];
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = M[m][d];
    }
    double R[NV][D], det;
    simplex_cofactors<D>(X, R, det);
    if (side == 0) {
#pragma unroll
      for (int d = 0; d < D; ++d) N[d] = R[D][d];
      nn = dot<D>(N, N);
      rn = rsqrt(nn);
    }
    const double scale = -rn / fabs(det);
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      const double Gn = dot<D>(R[a], N) * scale;
      gsum += p[a] * Gn;
      c[a < D ? a : D + side] += Gn;
    }
    hsum += sqrt(diameter2<D>(X));
  }
  const double area = nn * rn * (D == 2 ? 1.0 : 0.5);  // |N| / (D-1)!
  const double sc = sqrt(fabs(sigma) * 0.5 * hsum * area * (1.0 / (D * (D + 1))));
  double* w = work + g * W;
#pragma unroll
  for (int m = 0; m <= D; ++m) w[m] = sc * c[m];
  w[D + 1] = sc * gsum;
#pragma unroll
  for (int k = 0; k < D; ++k) w[D + 2 + k] = pm[k];
  if (D == 2) w[6] = w[7] = 0.0;
}

// ---- the facet-once records from a per-plan STATIC table ---------------------------------------------------------------
// Everything k_surface_once_p1 computes from the coordinates is a property of the mesh and the tags: the jump
// coefficients c_m of a ghost facet and the scale sqrt(avg(h) |F| / (D (D+1))), the normal derivatives cF grad(lambda_j).n
// of a one-sided entity.  What depends on the level set is LINEAR in it with exactly these coefficients:
//   s gsum = sum_m phi_m (s c_m)  (grad(phi).n on a side = sum_a phi_a grad(lambda_a).n),   cF grad(phi).n = sum_j phi_j (cF Gn_j).
// k_surface_static_p1 tabulates the coefficients once per plan (8 doubles per facet / entity, sigma left out);
// k_surface_fill_p1 then builds the work record of a step from one 64-byte read, the vertex list and D + 2 gathers of phi
// -- no coordinate gathers, no cofactors, no square roots: 83 -> ~15 us for the 1.7 M records of config E.
template <int D>
__global__ void __launch_bounds__(kRowsBlock) k_surface_static_p1(
    const double* __restrict__ x, const int32_t* __restrict__ macro, int64_t n_facets,
    const int32_t* __restrict__ entity_macro, int64_t n_entities, double* __restrict__ table) {
  constexpr int NV = D + 1, NG = D + 2, W = kGhostWork<D>;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_facets + n_entities) return;
  double* t = table + g * W;
  if (g >= n_facets) {  // one-sided entity: cF grad(lambda_j).n, j = 0..D (entity_record with phi = 0 writes them)
    const int64_t e = g - n_facets;
    double X[NV][D], p[NV], w[W];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int v = __ldg(entity_macro + e * NV + k);
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = __ldg(x + (int64_t)v * D + d);
      p[k] = 0.0;
    }
    entity_record<D>(X, p, w);
#pragma unroll
    for (int j = 0; j < W; ++j) t[j] = j < NV ? w[1 + j] : 0.0;
    return;
  }
  double M[NG][D];
#pragma unroll
  for (int m = 0; m < NG; ++m) {
    const int v = __ldg(macro + g * NG + m);
#pragma unroll
    for (int d = 0; d < D; ++d) M[m][d] = __ldg(x + (int64_t)v * D + d);
  }
  double c[NG], N[D], nn = 0.0, rn = 0.0, hsum = 0.0;
#pragma unroll
  for (int m = 0; m < NG; ++m) c[m] = 0.0;
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    double X[NV][D];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int m = k < D ? k : D + side;
#pragma unroll
      for (int d = 0; d < D; ++d) X[k][d] = M[m][d];
    }
    double R[NV][D], det;
    simplex_cofactors<D>(X, R, det);
    if (side == 0) {
#pragma unroll
      for (int d = 0; d < D; ++d) N[d] = R[D][d];
      nn = dot<D>(N, N);
      rn = rsqrt(nn);
    }
    const double scale = -rn / fabs(det);
#pragma unroll
    for (int a = 0; a < NV; ++a) c[a < D ? a : D + side] += dot<D>(R[a], N) * scale;
    hsum += sqrt(diameter2<D>(X));
  }
  const double area = nn * rn * (D == 2 ? 1.0 : 0.5);  // |N| / (D-1)!
  const double s0 = sqrt(0.5 * hsum * area * (1.0 / (D * (D + 1))));
#pragma unroll
  for (int j = 0; j < W; ++j) t[j] = j < NG ? s0 * c[j] : 0.0;
}

template <int D>
__global__ void __launch_bounds__(kRowsBlock) k_surface_fill_p1(
    const double* __restrict__ phi, double sigma, const int32_t* __restrict__ macro, int64_t n_facets,
    const int32_t* __restrict__ entity_macro, int64_t n_entities, const double* __restrict__ table,
    double* __restrict__ work) {
  constexpr int NV = D + 1, NG = D + 2, W = kGhostWork<D>;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_facets + n_entities) return;
  double t[W];
  ldg256(table + g * W, t[0], t[1], t[2], t[3]);
  ldg256(table + g * W + 4, t[4], t[5], t[6], t[7]);
  double* w = work + g * W;
  if (g >= n_facets) {
    const int64_t e = g - n_facets;
    double p[NV], gn = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      p[k] = __ldg(phi + __ldg(entity_macro + e * NV + k));
      gn += p[k] * t[k];
    }
    w[0] = gn;
#pragma unroll
    for (int j = 0; j < NV; ++j) w[1 + j] = t[j];
#pragma unroll
    for (int k = 0; k < D; ++k) w[2 + D + k] = p[k];
    if (D == 2) w[6] = w[7] = 0.0;
    return;
  }
  const double sq = sqrt(fabs(sigma));
  double pm[NG], gs = 0.0;
#pragma unroll
  for (int m = 0; m < NG; ++m) {
    pm[m] = __ldg(phi + __ldg(macro + g * NG + m));
    gs += pm[m] * t[m];
  }
#pragma unroll
  for (int m = 0; m <= D; ++m) w[m] = sq * t[m];
  w[D + 1] = sq * gs;
#pragma unroll
  for (int k = 0; k < D; ++k) w[D + 2 + k] = pm[k];
  if (D == 2) w[6] = w[7] = 0.0;
}

// Row a of the macro tensor from the facet's work record; pr = phi at the row's own vertex, sg = sign(sigma).
template <int D>
__device__ __forceinline__ void ghost_row(const double (&wk)[kGhostWork<D>], int a, double pr, double sg,
                                          double (&K)[D + 2]) {
  constexpr int NG = D + 2;
  double c[NG], csum = 0.0;
#pragma unroll
  for (int m = 0; m <= D; ++m) {
    c[m] = wk[m];
    csum += wk[m];
  }
  c[D + 1] = -csum;
  const double gsum = wk[D + 1];
  double Pf = wk[D + 2], Sf2 = wk[D + 2] * wk[D + 2];
#pragma unroll
  for (int k = 1; k < D; ++k) {
    Pf += wk[D + 2 + k];
    Sf2 += wk[D + 2 + k] * wk[D + 2 + k];
  }
  double ca = c[0];
#pragma unroll
  for (int m = 1; m < NG; ++m)
    if (m == a) ca = c[m];
  const bool onf = a < D;  // the row's vertex lies on the facet
  const double ga = onf ? gsum : 0.0;
  const double Jsa = sg * (ga + ca * Pf), cs = sg * ca, gs = sg * ga;
#pragma unroll
  for (int m = 0; m < NG; ++m) {
    const double gm = m < D ? gsum : 0.0;
    const double Jsm = gm + c[m] * Pf;
    double cross = cs * c[m] * Sf2 + gs * c[m] * pr;
    if (m < D) cross += cs * gm * wk[D + 2 + m];
    if (m == a) cross += gs * gm;
    K[m] = Jsa * Jsm + cross;
  }
}

// X4: x is the mesh's padded coordinate table (phifem_mesh.x4, 4 doubles per vertex, 32-byte aligned): one 256-bit
// gather and one address per vertex instead of three 64-bit ones, and a vertex never straddles two sectors
template <int D, bool X4 = false>
__device__ __forceinline__ void load_vertex(const double* __restrict__ x, const double* __restrict__ phi,
                                            int v, double (&xv)[D], double& p) {
  if constexpr (X4 && D == 3) {
    double pad;
    ldg256(x + (int64_t)v * 4, xv[0], xv[1], xv[2], pad);
  } else {
#pragma unroll
    for (int d = 0; d < D; ++d) xv[d] = __ldg(x + (int64_t)v * D + d);
  }
  p = __ldg(phi + v);
}

enum { kCells = 0, kSurface = 1, kCellsGeom = 2, kCellsX4 = 3 };

// coordinates, phi and f of the D other vertices of a cell record
template <int D>
struct Others {
  double X[D][D], p[D], f[D];
};
// cached geometry of the record's cell, phi and f of its D other vertices
template <int D>
struct OthersGeom {
  double g[8], p[D], f[D];
};

// One pass over one row list.  KIND == kCells writes data / b of its rows, the surface passes add to them.
template <int D, int KIND>
__global__ void __launch_bounds__(kRowsBlock, kRowsMinBlocks) k_assemble_rows_p1(
    const double* __restrict__ x, const double* __restrict__ phi, const double* __restrict__ f,
    double sigma, const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
    phifem_row_list rl, const double* __restrict__ surface_work, double* __restrict__ data,
    double* __restrict__ b) {  // surface_work: facet-once records (kSurface) / cached cell geometry (kCellsGeom)
  constexpr int NV = D + 1, NG = D + 2;
  extern __shared__ double acc_s[];  // accumulator k of thread t at acc_s[k * kRowsBlock + t]
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t li = (int64_t)blockIdx.x * kRowsBlock + tid;
  const int slice = (int)(li >> 5);
  if (li >= rl.n_listed) return;  // no block-wide barrier below
  const int r = __ldg(rl.rows + li);
  const int start = __ldg(indptr + r);
  const int nnz = __ldg(indptr + r + 1) - start;
  const int dpos = __ldg(rl.diag_pos + li);
  const int32_t* __restrict__ cols = indices + start;
  double* acc = acc_s + tid;
  for (int k = 0; k < nnz; ++k) acc[k * kRowsBlock] = 0.0;
  double xr[D], pr;
  load_vertex<D, KIND == kCellsX4>(x, phi, r, xr, pr);
  double diag = 0.0, br = 0.0;
  const int kb = __ldg(rl.ptr + slice), ke = __ldg(rl.ptr + slice + 1);

  if constexpr (KIND == kCells || KIND == kCellsX4) {  // cells tagged 1 / 2 containing vertex r
    // Four records in flight per thread, one per dependent-load level: while record k is evaluated the
    // vertex data of record k+1 is arriving, the column indices of record k+2 have been requested and so
    // has the word of record k+3.  The two data buffers swap roles (loop unrolled by two) so that no
    // register-to-register copies are needed.
    const double fr = __ldg(f + r);
    auto fetch_rec = [&](int k) { return k < ke ? __ldg(rl.rec + (int64_t)k * 32 + lane) : kPad; };
    auto fetch_idx = [&](uint32_t rec, int (&v)[D]) {
      const uint32_t q = rec == kPad ? 0u : rec;  // pads gather the row's first column: harmless
#pragma unroll
      for (int j = 0; j < D; ++j) v[j] = __ldg(cols + ((q >> (8 * j)) & 0xff));
    };
    auto fetch_data = [&](const int (&v)[D], Others<D>& o) {
#pragma unroll
      for (int j = 0; j < D; ++j) {
        load_vertex<D, KIND == kCellsX4>(x, phi, v[j], o.X[j], o.p[j]);
        o.f[j] = __ldg(f + v[j]);
      }
    };
    uint32_t w0 = fetch_rec(kb), w1 = fetch_rec(kb + 1), w2 = fetch_rec(kb + 2);
    int v1[D];
    Others<D> A, B;
    if (kb < ke) {
      fetch_idx(w0, v1);
      fetch_data(v1, A);
      fetch_idx(w1, v1);
    }
    // on entry: `cur` holds the data of record k (word w0), v1 the column indices of record k+1 (word w1),
    // w2 the word of record k+2
    auto body = [&](int k, const Others<D>& cur, Others<D>& nxt) {
      fetch_data(v1, nxt);
      fetch_idx(w2, v1);
      const uint32_t w3 = fetch_rec(k + 3);
      if (w0 != kPad) {
        double X[NV][D], p[NV], fv[NV];
#pragma unroll
        for (int d = 0; d < D; ++d) X[0][d] = xr[d];
        p[0] = pr;
        fv[0] = fr;
#pragma unroll
        for (int j = 0; j < D; ++j) {
#pragma unroll
          for (int d = 0; d < D; ++d) X[j + 1][d] = cur.X[j][d];
          p[j + 1] = cur.p[j];
          fv[j + 1] = cur.f[j];
        }
        double K[NV], b0;
        cell_row<D>(X, p, fv, (w0 >> 24) & 1u, sigma, K, b0);
        diag += K[0];
        br += b0;
#pragma unroll
        for (int j = 0; j < D; ++j) acc[((w0 >> (8 * j)) & 0xff) * kRowsBlock] += K[j + 1];
      }
      w0 = w1;
      w1 = w2;
      w2 = w3;
    };
    for (int k = kb; k < ke; k += 2) {
      body(k, A, B);
      if (k + 1 < ke) body(k + 1, B, A);
    }
  } else if constexpr (KIND == kCellsGeom) {  // the cell pass on cached geometry: two words per record
    // word 0 = position bytes | cut << 24 | (cell-local index of the row's vertex) << 25, word 1 = the cell's index
    // in the geometry table.  Same four-deep pipeline as above; the cell's 64-byte geometry record arrives with two
    // 256-bit loads instead of 3 D coordinate loads.
    const double fr = __ldg(f + r);
    const uint2* __restrict__ recs = reinterpret_cast<const uint2*>(rl.rec);
    const uint2 pad2 = make_uint2(0u, kPad);
    auto fetch_rec = [&](int k) { return k < ke ? __ldg(recs + (int64_t)k * 32 + lane) : pad2; };
    auto fetch_idx = [&](uint2 rec, int (&v)[D]) {
      const uint32_t q = rec.y == kPad ? 0u : rec.x;
#pragma unroll
      for (int j = 0; j < D; ++j) v[j] = __ldg(cols + ((q >> (8 * j)) & 0xff));
    };
    auto fetch_data = [&](const int (&v)[D], uint2 rec, OthersGeom<D>& o) {
      const double* src = surface_work + (rec.y == kPad ? 0 : (int64_t)rec.y * 8);
      ldg256(src, o.g[0], o.g[1], o.g[2], o.g[3]);
      ldg256(src + 4, o.g[4], o.g[5], o.g[6], o.g[7]);
#pragma unroll
      for (int j = 0; j < D; ++j) {
        o.p[j] = __ldg(phi + v[j]);
        o.f[j] = __ldg(f + v[j]);
      }
    };
    uint2 w0 = fetch_rec(kb), w1 = fetch_rec(kb + 1), w2 = fetch_rec(kb + 2);
    int v1[D];
    OthersGeom<D> A, B;
    if (kb < ke) {
      fetch_idx(w0, v1);
      fetch_data(v1, w0, A);
      fetch_idx(w1, v1);
    }
    auto body = [&](int k, const OthersGeom<D>& cur, OthersGeom<D>& nxt) {
      fetch_data(v1, w1, nxt);
      fetch_idx(w2, v1);
      const uint2 w3 = fetch_rec(k + 3);
      if (w0.y != kPad) {
        double p[NV], fv[NV];
        p[0] = pr;
        fv[0] = fr;
#pragma unroll
        for (int j = 0; j < D; ++j) {
          p[j + 1] = cur.p[j];
          fv[j + 1] = cur.f[j];
        }
        double K[NV], b0;
        cell_row_geom<D>(cur.g, (int)((w0.x >> 25) & 3u), p, fv, (w0.x >> 24) & 1u, sigma, K, b0);
        diag += K[0];
        br += b0;
#pragma unroll
        for (int j = 0; j < D; ++j) acc[((w0.x >> (8 * j)) & 0xff) * kRowsBlock] += K[j + 1];
      }
      w0 = w1;
      w1 = w2;
      w2 = w3;
    };
    for (int k = kb; k < ke; k += 2) {
      body(k, A, B);
      if (k + 1 < ke) body(k + 1, B, A);
    }
  } else {  // surface pass: ghost-penalty facets and one-sided entities whose vertices include r
    // ghost record = {positions of the other macro vertices (macro order, the row's own index skipped),
    //                 facet index in the plan's ghost list | macro index of the row's vertex << 28};
    // one-sided record = {positions of [opposite vertex, facet vertices (t + 1) % D, ...],
    //                     (n_ghost_facets + entity index) | t << 28 | 1 << 31};
    // the facet's work record (L2-resident) of record k+1 is requested before record k is evaluated
    constexpr int W = kGhostWork<D>;
    const uint2* __restrict__ recs = reinterpret_cast<const uint2*>(rl.rec);
    const uint2 pad2 = make_uint2(0u, kPad);
    auto fetch_rec = [&](int k) { return k < ke ? __ldg(recs + (int64_t)k * 32 + lane) : pad2; };
    auto fetch_work = [&](uint2 rec, double (&wk)[W]) {
      const int64_t g = rec.y == kPad ? 0 : (int64_t)(rec.y & 0x0fffffffu);  // ghost facet or n_ghost + entity
      const double* src = surface_work + g * W;
#pragma unroll
      for (int q = 0; q < W / 4; ++q) ldg256(src + 4 * q, wk[4 * q], wk[4 * q + 1], wk[4 * q + 2], wk[4 * q + 3]);
    };
    // record words are streamed from HBM (read once): kept 5 deep so that the word naming the NEXT facet has
    // arrived when its work record is requested
    const double sg = sigma < 0.0 ? -1.0 : 1.0;
    auto evaluate = [&](const uint2 rec, const double (&cur)[W]) {
      if (rec.y == kPad) return;
      if (rec.y >> 31) {  // one-sided entity: byte 0 = the opposite vertex, byte j = facet vertex (t + j) % D
        double Kb[NV];
        entity_row<D>(cur, (int)((rec.y >> 28) & 7u), Kb);
        diag += Kb[0];
        acc[(rec.x & 0xff) * kRowsBlock] += Kb[D];
#pragma unroll
        for (int j = 1; j < D; ++j) acc[((rec.x >> (8 * j)) & 0xff) * kRowsBlock] += Kb[j];
        return;
      }
      const int a = (int)(rec.y >> 28);
      double K[NG];
      ghost_row<D>(cur, a, pr, sg, K);
      double Ka = K[0];
#pragma unroll
      for (int m = 1; m < NG; ++m)
        if (m == a) Ka = K[m];
      diag += Ka;
#pragma unroll
      for (int j = 0; j < NG - 1; ++j)  // j-th other macro vertex = macro index j (j < a) or j + 1
        acc[((rec.x >> (8 * j)) & 0xff) * kRowsBlock] += j < a ? K[j] : K[j + 1];
    };
    // a third work buffer (the records of two facets in flight) measured 0.242 against 0.236 ms: the pass is not bound
    // by the latency of these gathers (DESIGN.md §4, K2+K3+K4)
    double wa[W], wb[W];
    uint2 w0 = fetch_rec(kb), w1 = fetch_rec(kb + 1), w2 = fetch_rec(kb + 2), w3 = fetch_rec(kb + 3),
          w4 = fetch_rec(kb + 4);
    if (kb < ke) fetch_work(w0, wa);
    auto body = [&](int k, const double (&cur)[W], double (&nxt)[W]) {
      const uint2 rec = w0;
      fetch_work(w1, nxt);
      w0 = w1;
      w1 = w2;
      w2 = w3;
      w3 = w4;
      w4 = fetch_rec(k + 5);
      evaluate(rec, cur);
    };
    for (int k = kb; k < ke; k += 2) {
      body(k, wa, wb);
      if (k + 1 < ke) body(k + 1, wb, wa);
    }
  }
  acc[dpos * kRowsBlock] += diag;
  if constexpr (KIND != kSurface) {
    for (int k = 0; k < nnz; ++k) data[start + k] = acc[k * kRowsBlock];
    b[r] = br;
  } else {
    for (int k = 0; k < nnz; ++k) data[start + k] += acc[k * kRowsBlock];
  }
}

}  // namespace
}  // namespace phifem

using namespace phifem;

namespace phifem {  // csrc/assemble_tiles.cu
cudaError_t launch_cell_tiles_p1(const phifem_mesh* mesh, const double* phi, const double* f, double sigma,
                                 const int32_t* indptr, const phifem_cell_tiles* tl, int max_row_nnz, double* data,
                                 double* b, cudaStream_t st);
}

namespace {
bool list_ok(const phifem_row_list& l) {
  return l.n_listed == 0 || (l.rows && l.diag_pos && l.ptr && l.rec);
}
// one side stream + fork / join events per device (created on first use, never destroyed)
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

extern "C" int phifem_assemble_rows_p1(const phifem_mesh* mesh, const double* phi, const double* f,
                                       double sigma, const phifem_rows_plan* plan, double* data,
                                       double* b, void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->x, "mesh is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON) {
    set_error("P1 assembly supports triangles and tetrahedra, got cell type %d", mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(mesh->gdim == (mesh->cell_type == PHIFEM_TRIANGLE ? 2 : 3), "gdim mismatch");
  PHIFEM_CHECK_ARG(plan != nullptr, "plan is null");
  const phifem_cell_tiles* tiles = plan->tiles && plan->tiles->n_tiles > 0 ? plan->tiles : nullptr;
  if (plan->cells.n_listed == 0 && plan->surface.n_listed == 0 && !tiles) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(phi && f && data && b, "null pointer");
  PHIFEM_CHECK_ARG(plan->indptr && plan->indices, "CSR pattern is null");
  PHIFEM_CHECK_ARG(list_ok(plan->cells) && list_ok(plan->surface), "row list arrays are null");
  PHIFEM_CHECK_ARG(plan->max_row_nnz > 0 && plan->max_row_nnz <= 255, "plan.max_row_nnz out of range");
  const int64_t n_once = plan->surface.n_listed ? plan->n_ghost_facets + plan->n_entities : 0;
  PHIFEM_CHECK_ARG(plan->surface.n_listed == 0 ||
                       (n_once > 0 && n_once < (1 << 28) && plan->surface_work &&
                        (plan->n_ghost_facets == 0 || plan->ghost_macro) &&
                        (plan->n_entities == 0 || plan->entity_macro)),
                   "surface arrays (n_ghost_facets + n_entities < 2^28, ghost_macro, entity_macro, surface_work)");
  const size_t smem = (size_t)plan->max_row_nnz * kRowsBlock * sizeof(double);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t err = cudaSuccess;
  auto launch = [&](auto kernel, const phifem_row_list& rl, const double* work, const double* coords = nullptr) {
    if (rl.n_listed == 0 || err != cudaSuccess) return;
    if (smem > 48 * 1024)
      err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t grid = (rl.n_listed + kRowsBlock - 1) / kRowsBlock;
    if (err == cudaSuccess)
      kernel<<<(unsigned)grid, kRowsBlock, smem, st>>>(coords ? coords : mesh->x, phi, f, sigma, plan->indptr,
                                                       plan->indices, rl, work, data, b);
  };
  // the padded coordinate table is an option of the mesh (NULL by default: -2 % on the structured mesh, +2 % on the
  // renumbered unstructured one at config E)
  const bool use_x4 = mesh->x4 != nullptr;
  const bool geom = plan->cell_geom != nullptr;
  auto cell_tiles = [&]() {  // cell-once form of the cell pass
    if (err == cudaSuccess)
      err = launch_cell_tiles_p1(mesh, phi, f, sigma, plan->indptr, tiles, plan->max_row_nnz, data, b, st);
  };
  // The facet-once kernel (latency-bound gathers, 2 % of the work) is forked onto a side stream so that it shares
  // the SMs with the fp64-bound cell pass; the surface row pass waits for both.
  SideStream& ss = side_stream();
  const bool fork = n_once > 0 && (plan->cells.n_listed > 0 || tiles) && ss.ok;
  cudaStream_t once_stream = fork ? ss.stream : st;
  auto once = [&](auto dim) {
    constexpr int D = decltype(dim)::value;
    if (n_once == 0) return;
    if (fork) {
      cudaEventRecord(ss.fork, st);
      cudaStreamWaitEvent(ss.stream, ss.fork, 0);
    }
    const unsigned grid = (unsigned)((n_once + kRowsBlock - 1) / kRowsBlock);
    if (plan->surface_static)  // coefficients tabulated once per plan (phifem_surface_static_p1): the light kernel
      k_surface_fill_p1<D><<<grid, kRowsBlock, 0, once_stream>>>(phi, sigma, plan->ghost_macro, plan->n_ghost_facets,
                                                                 plan->entity_macro, plan->n_entities,
                                                                 plan->surface_static, plan->surface_work);
    else
      k_surface_once_p1<D><<<grid, kRowsBlock, 0, once_stream>>>(mesh->x, phi, sigma, plan->ghost_macro,
                                                                 plan->n_ghost_facets, plan->entity_macro,
                                                                 plan->n_entities, plan->surface_work);
    if (fork) cudaEventRecord(ss.join, ss.stream);
  };
  if (mesh->cell_type == PHIFEM_TRIANGLE) {
    once(std::integral_constant<int, 2>());
    if (tiles) cell_tiles();
    else if (geom) launch(k_assemble_rows_p1<2, kCellsGeom>, plan->cells, plan->cell_geom);
    else launch(k_assemble_rows_p1<2, kCells>, plan->cells, nullptr);
    if (fork) cudaStreamWaitEvent(st, ss.join, 0);
    launch(k_assemble_rows_p1<2, kSurface>, plan->surface, plan->surface_work);
  } else {
    once(std::integral_constant<int, 3>());
    if (tiles) cell_tiles();
    else if (geom) launch(k_assemble_rows_p1<3, kCellsGeom>, plan->cells, plan->cell_geom);
    else if (use_x4) launch(k_assemble_rows_p1<3, kCellsX4>, plan->cells, nullptr, mesh->x4);
    else launch(k_assemble_rows_p1<3, kCells>, plan->cells, nullptr);
    if (fork) cudaStreamWaitEvent(st, ss.join, 0);
    launch(k_assemble_rows_p1<3, kSurface>, plan->surface, plan->surface_work);
  }
  if (err != cudaSuccess) {
    set_error("phifem_assemble_rows_p1: launch failed (%zu bytes of shared memory per row-gather CTA%s): %s", smem,
              tiles ? ", cell tiles" : "", cudaGetErrorString(err));
    return PHIFEM_ERR_CUDA;
  }
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_surface_static_p1(const phifem_mesh* mesh, const phifem_rows_plan* plan, void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->x && plan != nullptr, "mesh / plan is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON) {
    set_error("P1 assembly supports triangles and tetrahedra, got cell type %d", mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  const int64_t n_once = plan->n_ghost_facets + plan->n_entities;
  if (n_once == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(plan->surface_static != nullptr, "plan.surface_static is null");
  PHIFEM_CHECK_ARG((plan->n_ghost_facets == 0 || plan->ghost_macro) && (plan->n_entities == 0 || plan->entity_macro),
                   "ghost_macro / entity_macro");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned grid = (unsigned)((n_once + kRowsBlock - 1) / kRowsBlock);
  if (mesh->cell_type == PHIFEM_TRIANGLE)
    k_surface_static_p1<2><<<grid, kRowsBlock, 0, st>>>(mesh->x, plan->ghost_macro, plan->n_ghost_facets,
                                                        plan->entity_macro, plan->n_entities, plan->surface_static);
  else
    k_surface_static_p1<3><<<grid, kRowsBlock, 0, st>>>(mesh->x, plan->ghost_macro, plan->n_ghost_facets,
                                                        plan->entity_macro, plan->n_entities, plan->surface_static);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}
