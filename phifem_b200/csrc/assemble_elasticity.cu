// Interface-elasticity phi-FEM operator (reference demo/interface-elasticity/main.py:152-274, BASELINE.json
// configs[3]) on the mixed space (u_in, u_out, y_in, y_out, p) in P1^D x P1^D x P1^(DxD) x P1^(DxD) x P1^D on
// triangles / tetrahedra, with a P1 or P2 level set:
//   a =   int_{dx(1,2)} sigma_in(u_in):eps(v_in) + int_{dx(2,3)} sigma_out(u_out):eps(v_out)            (:186-187)
//       + gamma int_{dx(2)} [ c_out (y_in + sigma_in(u_in)):(z_in + sigma_in(v_in))
//                           + c_in (y_out + sigma_out(u_out)):(z_out + sigma_out(v_out))
//                           + h^-2 ((y_in - y_out) grad phi).((z_in - z_out) grad phi)
//                           + h^-2 (u_in - u_out + h^-1 p phi).(v_in - v_out + h^-1 q phi) ]             (:189-205)
//       + sigma_s int_{dx(2)} h^2 (div y_in.div z_in + div y_out.div z_out)                             (:213-219)
//       + sigma_s int_{dS(3)} avg(h) [sigma_in(u_in) n].[sigma_in(v_in) n]  (and out over dS(4))        (:207-225)
//       + int_{ds(100)} (y_in n).v_in + int_{ds(101)} (y_out n).v_out                                  (:183-184)
//   L =   int_{dx(1,2)} f.v_in + int_{dx(2,3)} f.v_out + sigma_s int_{dx(2)} h^2 f.(div z_in + div z_out) (:254-269)
//
// Every field is nodal P1, so the mixed space has NB = 3 D + 2 D^2 dofs per vertex (global dof = NB vertex + o;
// o: u_in c -> c, u_out c -> D + c, y_in (r,s) -> 2D + r D + s, y_out (r,s) -> 2D + D^2 + r D + s, p c -> 2D + 2D^2 + c)
// and the CSR matrix is the vertex graph with dense NB x NB blocks: the entry (NB r + a, NB s + b) lives at
// NB (NB vptr[r] + a deg(r) + pos) + b, pos = rank of s in r's sorted vertex-neighbour list.  The only slot map
// is therefore the scalar one (NV^2 ints per cell instead of (NV NB)^2).
//
// Cut cells: one thread per (cell, test node k, trial node j, trial offset b).  The trial function's quantities
// (T_in = y_in + sigma_in(u_in), T_out, R = (y_in - y_out) grad phi, S = u_in - u_out + p phi / h, div y_in, div y_out)
// are a small runtime bundle; the NB test offsets are unrolled at compile time, so that each contraction holds only the
// non-zero terms of its field.  Consecutive threads write consecutive CSR entries.
//
// Quadrilaterals (gdim 2, vertices in tensor order): every field is Q1 on the bilinear cell (NB = 14, 4 vertices per
// cell, the same global numbering) and the level set Q1 or Q2.  The quadrature rule's cell_points are reference
// coordinates (xi, eta) on [0, 1]^2 and integrate the cut cells (quadrature.rules_for_elasticity_quad: (kphi + 2)^2
// Gauss points); the uncut cells use a fixed 2 x 2 Gauss rule and the stress jump a fixed 2-point Gauss rule on the edge,
// both compile-time constants; the one-sided terms have a closed form.  The bundle and the contractions above serve both
// cell types: they take point values and physical gradients of a nodal basis.
#include <utility>

#include "common.cuh"
#include "pk_common.cuh"
#include "quad_common.cuh"

namespace phifem {
using namespace pk;
namespace {

constexpr int kBlockEl = 128;

template <int D>
struct ES {
  static constexpr int NV = D + 1;
  static constexpr int UI = 0, UO = D, YI = 2 * D, YO = 2 * D + D * D, PP = 2 * D + 2 * D * D;
  static constexpr int NB = 3 * D + 2 * D * D;
  __host__ __device__ static constexpr int field(int o) { return o < UO ? 0 : o < YI ? 1 : o < YO ? 2 : o < PP ? 3 : 4; }
  __host__ __device__ static constexpr int base(int fld) { return fld == 0 ? UI : fld == 1 ? UO : fld == 2 ? YI : fld == 3 ? YO : PP; }
};

// does the cut-cell form couple test field fa with trial field fb?  (u_in,y_out), (u_out,y_in), (y,p) do not
__host__ __device__ constexpr bool couples(int fa, int fb) {
  if (fa > fb) { const int t = fa; fa = fb; fb = t; }
  if (fa == 0) return fb != 3;
  if (fa == 1) return fb != 2;
  if (fa == 2 || fa == 3) return fb != 4;
  return true;
}

template <int D>
struct Bundle {
  double TI[D][D], TO[D][D], R[D], S[D], DI[D], DO[D];
};

struct CellCoefs {
  double lmbda_in, mu_in, lmbda_out, mu_out;
  double w_in, w_out;      // stiffness switches: tag in (1,2) / (2,3)
  double pen_in, pen_out;  // gamma c_out, gamma c_in on cut cells (the weights of T_in:T_in and T_out:T_out)
  double pen_h2;           // gamma h^-2 on cut cells
  double stab;             // sigma_s h^2 on cut cells
};

// quantities of the mixed basis function (node with P1 value l and gradient Gn, offset o) at a point
template <int D>
__device__ __forceinline__ void trial_bundle(int o, double l, const double (&Gn)[D], const double (&gph)[D],
                                             double ph_over_h, const CellCoefs& cf, Bundle<D>& B) {
  using S_ = ES<D>;
#pragma unroll
  for (int r = 0; r < D; ++r) {
    B.R[r] = B.S[r] = B.DI[r] = B.DO[r] = 0.0;
#pragma unroll
    for (int s = 0; s < D; ++s) B.TI[r][s] = B.TO[r][s] = 0.0;
  }
  const int fld = S_::field(o);
  const int loc = o - S_::base(fld);
  if (fld <= 1) {  // u_in / u_out, component c: sigma(u) = lmbda G[c] I + mu (e_c x G + G x e_c)
    const int c = loc;
    const double lm = fld == 0 ? cf.lmbda_in : cf.lmbda_out, mu = fld == 0 ? cf.mu_in : cf.mu_out;
    double gc = 0.0;
#pragma unroll
    for (int s = 0; s < D; ++s)
      if (s == c) gc = Gn[s];
#pragma unroll
    for (int r = 0; r < D; ++r)
#pragma unroll
      for (int s = 0; s < D; ++s) {
        const double v = (r == s ? lm * gc : 0.0) + (r == c ? mu * Gn[s] : 0.0) + (s == c ? mu * Gn[r] : 0.0);
        if (fld == 0) B.TI[r][s] = v;
        else B.TO[r][s] = v;
      }
#pragma unroll
    for (int s = 0; s < D; ++s)
      if (s == c) B.S[s] = fld == 0 ? l : -l;
  } else if (fld <= 3) {  // y_in / y_out, entry (r0, s0)
    const int r0 = loc / D, s0 = loc - r0 * D;
    double gs = 0.0, Gs = 0.0;
#pragma unroll
    for (int s = 0; s < D; ++s)
      if (s == s0) {
        gs = gph[s];
        Gs = Gn[s];
      }
#pragma unroll
    for (int r = 0; r < D; ++r) {
      if (r != r0) continue;
#pragma unroll
      for (int s = 0; s < D; ++s)
        if (s == s0) {
          if (fld == 2) B.TI[r][s] = l;
          else B.TO[r][s] = l;
        }
      B.R[r] = fld == 2 ? l * gs : -l * gs;
      if (fld == 2) B.DI[r] = Gs;
      else B.DO[r] = Gs;
    }
  } else {  // p, component c
#pragma unroll
    for (int s = 0; s < D; ++s)
      if (s == loc) B.S[s] = l * ph_over_h;
  }
}

// integrand (without the quadrature weight) of test offset A at node (lk, Gk) against the trial bundle
template <int D, int A>
__device__ __forceinline__ double contract(const Bundle<D>& B, int fld_b, double lk, const double (&Gk)[D],
                                           const double (&gph)[D], double ph_over_h, const CellCoefs& cf) {
  using S_ = ES<D>;
  constexpr int fa = S_::field(A), loc = A - S_::base(fa);
  if constexpr (fa <= 1) {
    constexpr int c = loc;
    const double(&T)[D][D] = fa == 0 ? B.TI : B.TO;
    const double lm = fa == 0 ? cf.lmbda_in : cf.lmbda_out, mu = fa == 0 ? cf.mu_in : cf.mu_out;
    double tg = 0.0, tgt = 0.0, tr = 0.0;
#pragma unroll
    for (int s = 0; s < D; ++s) {
      tg += T[c][s] * Gk[s];
      tgt += T[s][c] * Gk[s];
      tr += T[s][s];
    }
    // sigma(u_b):eps(v_a) = (sigma(u_b) G_k)[c]; T_b:sigma(v_a) = lmbda G_k[c] tr(T_b) + mu (T_b G_k + T_b^T G_k)[c]
    const double stiff = fld_b == fa ? (fa == 0 ? cf.w_in : cf.w_out) * tg : 0.0;
    const double pen = (fa == 0 ? cf.pen_in : cf.pen_out) * (lm * Gk[c] * tr + mu * (tg + tgt));
    const double sv = cf.pen_h2 * B.S[c] * lk;
    return stiff + pen + (fa == 0 ? sv : -sv);
  } else if constexpr (fa <= 3) {
    constexpr int r = loc / D, s = loc % D;
    const double t = fa == 2 ? cf.pen_in * B.TI[r][s] : cf.pen_out * B.TO[r][s];
    const double rv = cf.pen_h2 * B.R[r] * gph[s];
    const double dv = cf.stab * (fa == 2 ? B.DI[r] : B.DO[r]) * Gk[s];
    return lk * (t + (fa == 2 ? rv : -rv)) + dv;
  } else {
    return cf.pen_h2 * B.S[loc] * lk * ph_over_h;
  }
}

template <int D, int... As>
__device__ __forceinline__ void accumulate(std::integer_sequence<int, As...>, double (&acc)[ES<D>::NB], double w,
                                           const Bundle<D>& B, int fld_b, double lk, const double (&Gk)[D],
                                           const double (&gph)[D], double ph_over_h, const CellCoefs& cf) {
  ((acc[As] += w * contract<D, As>(B, fld_b, lk, Gk, gph, ph_over_h, cf)), ...);
}

__device__ __forceinline__ int64_t block_address(const int32_t* __restrict__ vptr, int row_vertex, int a, int pos, int b,
                                                 int nb) {
  const int64_t p0 = __ldg(vptr + row_vertex), deg = __ldg(vptr + row_vertex + 1) - p0;
  return (int64_t)nb * ((int64_t)nb * p0 + (int64_t)a * deg + pos) + b;
}

// Cells tagged 1 (resp. 3) carry the stiffness block of u_in (resp. u_out) and its load only, constant integrands:
//   int sigma(u_b):eps(v_a) = |K| (lmbda G_k[c] G_j[c'] + mu (delta_cc' G_k.G_j + G_j[c] G_k[c'])),
//   int f_c lambda_k = |K| sum_l f_l[c] (1 + delta_lk) / ((D+1)(D+2)).        One thread per (cell, k, j).
template <int D>
__global__ void __launch_bounds__(kBlockEl) k_elasticity_uncut(
    phifem_mesh m, const double* __restrict__ f, const int8_t* __restrict__ ctags, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_cells, phifem_elasticity_params prm, double* __restrict__ data,
    double* __restrict__ b) {
  using S_ = ES<D>;
  constexpr int NV = S_::NV, NB = S_::NB;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m.n_cells * (NV * NV)) return;
  const int64_t c = t / (NV * NV);
  const int rem = (int)(t - c * (NV * NV));
  const int k = rem / NV, j = rem - k * NV;
  const int tag = ctags[c];
  if (tag != 1 && tag != 3) return;
  const double lm = tag == 1 ? prm.lmbda_in : prm.lmbda_out, mu = tag == 1 ? prm.mu_in : prm.mu_out;
  const int ou = tag == 1 ? S_::UI : S_::UO;
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double Gk[D], Gj[D];
#pragma unroll
  for (int d = 0; d < D; ++d) Gk[d] = Gj[d] = 0.0;
#pragma unroll
  for (int n = 0; n < NV; ++n) {
    if (n == k)
#pragma unroll
      for (int d = 0; d < D; ++d) Gk[d] = g.G[n][d];
    if (n == j)
#pragma unroll
      for (int d = 0; d < D; ++d) Gj[d] = g.G[n][d];
  }
  const double gg = mu * dotd<D>(Gk, Gj);
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_cells + c * (NV * NV) + rem);
#pragma unroll
  for (int ca = 0; ca < D; ++ca)
#pragma unroll
    for (int cb = 0; cb < D; ++cb)
      atomicAdd(data + block_address(vptr, vk, ou + ca, pos, ou + cb, NB),
                g.vol * (lm * Gk[ca] * Gj[cb] + mu * Gj[ca] * Gk[cb] + (ca == cb ? gg : 0.0)));
  if (j == k) {
#pragma unroll
    for (int ca = 0; ca < D; ++ca) {
      double s = 0.0;
#pragma unroll
      for (int l = 0; l < NV; ++l) s += __ldg(f + (int64_t)__ldg(m.cells + c * NV + l) * D + ca) * (l == k ? 2.0 : 1.0);
      atomicAdd(b + (int64_t)NB * vk + ou + ca, g.vol * s * (1.0 / ((D + 1) * (D + 2))));
    }
  }
}

template <int D, int KP>
__global__ void __launch_bounds__(kBlockEl, 3) k_elasticity_cells(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qlam_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const double* __restrict__ f, const int32_t* __restrict__ cut_cells,
    int64_t n_cut, const int32_t* __restrict__ vptr, const int32_t* __restrict__ pos_cells,
    phifem_elasticity_params prm, double* __restrict__ data, double* __restrict__ b) {
  using S_ = ES<D>;
  constexpr int NV = S_::NV, NB = S_::NB, NDP = Space<D, KP>::ND;
  __shared__ double qlam[kMaxQuadPoints * NV], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * NV; i += blockDim.x) qlam[i] = qlam_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cut * (NV * NV * NB)) return;
  const int64_t e = t / (NV * NV * NB);
  int rem = (int)(t - e * (NV * NV * NB));
  const int k = rem / (NV * NB);
  rem -= k * (NV * NB);
  const int j = rem / NB, ob = rem - j * NB;
  const int64_t c = __ldg(cut_cells + e);
  const int fld_b = S_::field(ob);
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  const double h = sqrt(g.h2);
  CellCoefs cf;
  cf.lmbda_in = prm.lmbda_in; cf.mu_in = prm.mu_in; cf.lmbda_out = prm.lmbda_out; cf.mu_out = prm.mu_out;
  cf.w_in = cf.w_out = 1.0;
  cf.pen_in = prm.gamma * prm.coef_out;
  cf.pen_out = prm.gamma * prm.coef_in;
  cf.pen_h2 = prm.gamma / g.h2;
  cf.stab = prm.sigma_s * g.h2;
  double Gk[D], Gj[D];
#pragma unroll
  for (int d = 0; d < D; ++d) Gk[d] = Gj[d] = 0.0;
#pragma unroll
  for (int n = 0; n < NV; ++n) {
    if (n == k)
#pragma unroll
      for (int d = 0; d < D; ++d) Gk[d] = g.G[n][d];
    if (n == j)
#pragma unroll
      for (int d = 0; d < D; ++d) Gj[d] = g.G[n][d];
  }
  double acc[NB];
#pragma unroll
  for (int a = 0; a < NB; ++a) acc[a] = 0.0;
  double pc[NDP];
  load_dofs<D, KP>(m, sp, phi, c, pc);
  for (int q = 0; q < nq; ++q) {
    double lam[NV];
#pragma unroll
    for (int n = 0; n < NV; ++n) lam[n] = qlam[q * NV + n];
    double ph, gph[D];
    eval_phi_only<D, KP>(lam, g.G, pc, ph, gph);
    const double lk = pick<NV>(lam, k), lj = pick<NV>(lam, j);
    Bundle<D> B;
    trial_bundle<D>(ob, lj, Gj, gph, ph / h, cf, B);
    accumulate<D>(std::make_integer_sequence<int, NB>{}, acc, qw[q] * g.vol, B, fld_b, lk, Gk, gph, ph / h, cf);
  }
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_cells + c * (NV * NV) + k * NV + j);
  const int64_t p0 = __ldg(vptr + vk), deg = __ldg(vptr + vk + 1) - p0;
  const int64_t base = (int64_t)NB * ((int64_t)NB * p0 + pos) + ob;
#pragma unroll
  for (int a = 0; a < NB; ++a) {
    if (couples(S_::field(a), fld_b)) atomicAdd(data + base + (int64_t)NB * a * deg, acc[a]);
  }
  // load vector: the threads with j == k own b[(k, ob)]
  if (j == k) {
    const int loc = ob - S_::base(fld_b);
    double bv = 0.0;
    if (fld_b <= 1) {  // int f_c lambda_k = |K| sum_l f_l[c] (1 + delta_lk) / ((D+1)(D+2))
      double s = 0.0;
#pragma unroll
      for (int l = 0; l < NV; ++l) s += __ldg(f + (int64_t)__ldg(m.cells + c * NV + l) * D + loc) * (l == k ? 2.0 : 1.0);
      bv = (fld_b == 0 ? cf.w_in : cf.w_out) * g.vol * s * (1.0 / ((D + 1) * (D + 2)));
    } else if (fld_b <= 3) {  // sigma_s h^2 int f.div z, div z = G_k[s] e_r
      const int r = loc / D, s0 = loc - r * D;
      double s = 0.0;
#pragma unroll
      for (int l = 0; l < NV; ++l) s += __ldg(f + (int64_t)__ldg(m.cells + c * NV + l) * D + r);
      bv = cf.stab * g.vol * pick<D>(Gk, s0) * s * (1.0 / NV);
    }
    if (fld_b <= 3) atomicAdd(b + (int64_t)NB * vk + ob, bv);
  }
}

// sigma_s avg(h) int_F [sigma(u) n].[sigma(v) n] over dS(3) (side 0: in) / dS(4) (side 1: out): sigma(u) is constant
// on each cell, so the jump is one vector per macro basis function.  One thread per (facet, trial side, node, component).
template <int D>
__global__ void __launch_bounds__(kBlockEl) k_elasticity_facets(
    phifem_mesh m, const int32_t* __restrict__ facets, int64_t n_facets, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_facets, int side, phifem_elasticity_params prm, double* __restrict__ data) {
  using S_ = ES<D>;
  constexpr int NV = S_::NV, NB = S_::NB, NT = 2 * NV * D;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets * NT) return;
  const int64_t e = t / NT;
  int rem = (int)(t - e * NT);
  const int sb = rem / (NV * D);
  rem -= sb * (NV * D);
  const int j = rem / D, cb = rem - j * D;
  const int32_t fct = __ldg(facets + e);
  const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
  const double lm = side == 0 ? prm.lmbda_in : prm.lmbda_out, mu = side == 0 ? prm.mu_in : prm.mu_out;
  const int ou = side == 0 ? S_::UI : S_::UO;
  Geometry<D> gs[2];
  load_geometry<D>(m, cc.x, gs[0]);
  load_geometry<D>(m, cc.y, gs[1]);
  double nrm[2][D], area[2];
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int64_t cell = s == 0 ? cc.x : cc.y;
    int o = 0;
#pragma unroll
    for (int n = 0; n < NV; ++n)
      if (__ldg(m.c2f + cell * NV + n) == fct) o = n;
    facet_normal<D>(gs[s], o, nrm[s], area[s]);
  }
  const double coef = prm.sigma_s * 0.5 * (sqrt(gs[0].h2) + sqrt(gs[1].h2)) * area[0];
  // J(s, n, c) = sigma(u) n_s = lmbda G[c] n + mu (e_c (G.n) + G n[c])
  auto jump = [&](int s, int n, int c, double (&J)[D]) {
    double Gn[D], ns[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
      Gn[d] = s == 0 ? gs[0].G[0][d] : gs[1].G[0][d];
      ns[d] = s == 0 ? nrm[0][d] : nrm[1][d];
    }
#pragma unroll
    for (int q = 1; q < NV; ++q)
      if (q == n)
#pragma unroll
        for (int d = 0; d < D; ++d) Gn[d] = s == 0 ? gs[0].G[q][d] : gs[1].G[q][d];
    const double gn = dotd<D>(Gn, ns);
    double gc = 0.0, nc = 0.0;
#pragma unroll
    for (int d = 0; d < D; ++d)
      if (d == c) {
        gc = Gn[d];
        nc = ns[d];
      }
#pragma unroll
    for (int d = 0; d < D; ++d) J[d] = lm * gc * ns[d] + mu * (Gn[d] * nc + (d == c ? gn : 0.0));
  };
  double Jb[D];
  jump(sb, j, cb, Jb);
  const int colslot = sb * NV + j;
#pragma unroll
  for (int sa = 0; sa < 2; ++sa)
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vk = __ldg(m.cells + (int64_t)(sa == 0 ? cc.x : cc.y) * NV + k);
      const int pos = __ldg(pos_facets + (e * (2 * NV) + sa * NV + k) * (2 * NV) + colslot);
#pragma unroll
      for (int ca = 0; ca < D; ++ca) {
        double Ja[D];
        jump(sa, k, ca, Ja);
        atomicAdd(data + block_address(vptr, vk, ou + ca, pos, ou + cb, NB), coef * dotd<D>(Ja, Jb));
      }
    }
}

// int_{ds(100)} (y_in n).v_in (side 0) / int_{ds(101)} (y_out n).v_out (side 1): one thread per (entity, k, j)
template <int D>
__global__ void __launch_bounds__(kBlockEl) k_elasticity_boundary(
    phifem_mesh m, const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_boundary, int side, double* __restrict__ data) {
  using S_ = ES<D>;
  constexpr int NV = S_::NV, NB = S_::NB;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * NV * NV) return;
  const int64_t e = t / (NV * NV);
  const int rem = (int)(t - e * NV * NV);
  const int k = rem / NV, j = rem - k * NV;
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  if (k == o || j == o) return;
  Geometry<D> g;
  load_geometry<D>(m, c, g);
  double n[D], area;
  facet_normal<D>(g, o, n, area);
  const double mkj = area * (k == j ? 2.0 : 1.0) * (1.0 / (D * (D + 1)));
  const int ou = side == 0 ? S_::UI : S_::UO, oy = side == 0 ? S_::YI : S_::YO;
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_boundary + e * (NV * NV) + rem);
#pragma unroll
  for (int cc = 0; cc < D; ++cc)
#pragma unroll
    for (int s = 0; s < D; ++s)
      atomicAdd(data + block_address(vptr, vk, ou + cc, pos, oy + cc * D + s, NB), n[s] * mkj);
}

// ==== quadrilaterals: bilinear cells, every field Q1 (NB = 14 dofs per vertex, 4 vertices per cell) ==================
// Nothing is affine, so every integral is a quadrature at reference points (xi, eta) mapped by quad::map_point.  The
// uncut cells and the stress jump use fixed Gauss rules, exact on a parallelogram: 2 x 2 points on the cell (the
// stiffness and the load have degree 2 per reference direction) and 2 on the edge (sigma(u) n is linear along it).
constexpr double kGauss2Lo = 0.21132486540518711775, kGauss2Hi = 0.78867513459481288225;   // (1 -+ 1/sqrt(3)) / 2

// row n of G [4][2] at a runtime index, without local memory
__device__ __forceinline__ void pick_row(const double (&G)[quad::NV][2], int n, double (&out)[2]) {
  out[0] = G[0][0];
  out[1] = G[0][1];
#pragma unroll
  for (int q = 1; q < quad::NV; ++q)
    if (q == n) {
      out[0] = G[q][0];
      out[1] = G[q][1];
    }
}

// sigma(N e_c) n = lmbda G[c] n + mu (G n[c] + e_c (G.n)) for the gradient G of a scalar nodal function N
__device__ __forceinline__ void stress_normal(const double (&Gn)[2], const double (&ns)[2], int c, double lm, double mu,
                                              double (&J)[2]) {
  const double gn = Gn[0] * ns[0] + Gn[1] * ns[1];
  const double gc = c == 0 ? Gn[0] : Gn[1], nc = c == 0 ? ns[0] : ns[1];
#pragma unroll
  for (int d = 0; d < 2; ++d) J[d] = lm * gc * ns[d] + mu * (Gn[d] * nc + (d == c ? gn : 0.0));
}

// Cells tagged 1 (resp. 3): the stiffness block of u_in (resp. u_out) and its load int f.v, by the 2 x 2 Gauss rule.
// One thread per (cell, k, j); the j == k threads write the load.
__global__ void __launch_bounds__(kBlockEl) k_elasticity_quad_uncut(
    phifem_mesh m, const double* __restrict__ f, const int8_t* __restrict__ ctags, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_cells, phifem_elasticity_params prm, double* __restrict__ data,
    double* __restrict__ b) {
  using S_ = ES<2>;
  constexpr int NV = quad::NV, NB = S_::NB;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m.n_cells * (NV * NV)) return;
  const int64_t c = t / (NV * NV);
  const int rem = (int)(t - c * (NV * NV));
  const int k = rem / NV, j = rem - k * NV;
  const int tag = ctags[c];
  if (tag != 1 && tag != 3) return;
  const double lm = tag == 1 ? prm.lmbda_in : prm.lmbda_out, mu = tag == 1 ? prm.mu_in : prm.mu_out;
  const int ou = tag == 1 ? S_::UI : S_::UO;
  quad::Cell g;
  quad::load_cell(m, c, g);
  double K[2][2] = {{0.0, 0.0}, {0.0, 0.0}}, M[NV];   // M[l] = int N_k N_l (the j == k threads)
#pragma unroll
  for (int l = 0; l < NV; ++l) M[l] = 0.0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    double N[NV], G[NV][2], Jit[2][2], Gk[2], Gj[2];
    const double w = 0.25 * quad::map_point(g, (q & 1) ? kGauss2Hi : kGauss2Lo, (q >> 1) ? kGauss2Hi : kGauss2Lo, N, G,
                                            Jit);
    pick_row(G, k, Gk);
    pick_row(G, j, Gj);
    const double gg = mu * (Gk[0] * Gj[0] + Gk[1] * Gj[1]);
#pragma unroll
    for (int ca = 0; ca < 2; ++ca)
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) K[ca][cb] += w * (lm * Gk[ca] * Gj[cb] + mu * Gj[ca] * Gk[cb] + (ca == cb ? gg : 0.0));
    const double wk = w * pick<NV>(N, k);
#pragma unroll
    for (int l = 0; l < NV; ++l) M[l] += wk * N[l];
  }
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_cells + c * (NV * NV) + rem);
#pragma unroll
  for (int ca = 0; ca < 2; ++ca)
#pragma unroll
    for (int cb = 0; cb < 2; ++cb) atomicAdd(data + block_address(vptr, vk, ou + ca, pos, ou + cb, NB), K[ca][cb]);
  if (j == k) {
#pragma unroll
    for (int ca = 0; ca < 2; ++ca) {
      double s = 0.0;
#pragma unroll
      for (int l = 0; l < NV; ++l) s += __ldg(f + (int64_t)__ldg(m.cells + c * NV + l) * 2 + ca) * M[l];
      atomicAdd(b + (int64_t)NB * vk + ou + ca, s);
    }
  }
}

// Cut cells (tag 2): every term of a and L by the cell rule of phifem_quadrature (reference points (xi, eta)).  One thread
// per (cut cell, test node k, trial node j, trial offset b) = 224 per cell; the trial bundle and the contractions are the
// simplex kernel's, at the point values and physical gradients of the Q1 basis.
template <int KP>
__global__ void __launch_bounds__(kBlockEl, 3) k_elasticity_quad_cells(
    phifem_mesh m, phifem_pk_space sp, const double* __restrict__ qpt_g, const double* __restrict__ qw_g, int nq,
    const double* __restrict__ phi, const double* __restrict__ f, const int32_t* __restrict__ cut_cells,
    int64_t n_cut, const int32_t* __restrict__ vptr, const int32_t* __restrict__ pos_cells,
    phifem_elasticity_params prm, double* __restrict__ data, double* __restrict__ b) {
  using S_ = ES<2>;
  constexpr int NV = quad::NV, NB = S_::NB, NDP = quad::QSpace<KP>::ND;
  __shared__ double qpt[kMaxQuadPoints * 2], qw[kMaxQuadPoints];
  for (int i = threadIdx.x; i < nq * 2; i += blockDim.x) qpt[i] = qpt_g[i];
  for (int i = threadIdx.x; i < nq; i += blockDim.x) qw[i] = qw_g[i];
  __syncthreads();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cut * (NV * NV * NB)) return;
  const int64_t e = t / (NV * NV * NB);
  int rem = (int)(t - e * (NV * NV * NB));
  const int k = rem / (NV * NB);
  rem -= k * (NV * NB);
  const int j = rem / NB, ob = rem - j * NB;
  const int64_t c = __ldg(cut_cells + e);
  const int fld_b = S_::field(ob);
  const int loc = ob - S_::base(fld_b);
  quad::Cell g;
  quad::load_cell(m, c, g);
  const double h = sqrt(g.h2);
  CellCoefs cf;
  cf.lmbda_in = prm.lmbda_in; cf.mu_in = prm.mu_in; cf.lmbda_out = prm.lmbda_out; cf.mu_out = prm.mu_out;
  cf.w_in = cf.w_out = 1.0;
  cf.pen_in = prm.gamma * prm.coef_out;
  cf.pen_out = prm.gamma * prm.coef_in;
  cf.pen_h2 = prm.gamma / g.h2;
  cf.stab = prm.sigma_s * g.h2;
  double acc[NB], L[NV];   // L[l]: the load of offset ob at node k per unit nodal value of f at node l (j == k threads)
#pragma unroll
  for (int a = 0; a < NB; ++a) acc[a] = 0.0;
#pragma unroll
  for (int l = 0; l < NV; ++l) L[l] = 0.0;
  double pc[NDP];
  quad::load_phi<KP>(m, sp, phi, c, pc);
  for (int q = 0; q < nq; ++q) {
    const double xi = qpt[2 * q], eta = qpt[2 * q + 1];
    double N[NV], G[NV][2], Jit[2][2], Gk[2], Gj[2];
    const double w = qw[q] * quad::map_point(g, xi, eta, N, G, Jit);
    double ph, gph[2];
    quad::eval_phi<KP>(xi, eta, Jit, pc, ph, gph);
    pick_row(G, k, Gk);
    pick_row(G, j, Gj);
    const double lk = pick<NV>(N, k), lj = pick<NV>(N, j);
    Bundle<2> B;
    trial_bundle<2>(ob, lj, Gj, gph, ph / h, cf, B);
    accumulate<2>(std::make_integer_sequence<int, NB>{}, acc, w, B, fld_b, lk, Gk, gph, ph / h, cf);
    if (j == k) {   // u: int f_loc N_k;  y (r, s0): sigma_s h^2 int f_r d_s0 N_k
      const double wl = w * (fld_b <= 1 ? lk : (loc % 2 == 0 ? Gk[0] : Gk[1]));
#pragma unroll
      for (int l = 0; l < NV; ++l) L[l] += wl * N[l];
    }
  }
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_cells + c * (NV * NV) + k * NV + j);
  const int64_t p0 = __ldg(vptr + vk), deg = __ldg(vptr + vk + 1) - p0;
  const int64_t base = (int64_t)NB * ((int64_t)NB * p0 + pos) + ob;
#pragma unroll
  for (int a = 0; a < NB; ++a) {
    if (couples(S_::field(a), fld_b)) atomicAdd(data + base + (int64_t)NB * a * deg, acc[a]);
  }
  if (j == k && fld_b <= 3) {
    const int comp = fld_b <= 1 ? loc : loc / 2;
    double s = 0.0;
#pragma unroll
    for (int l = 0; l < NV; ++l) s += __ldg(f + (int64_t)__ldg(m.cells + c * NV + l) * 2 + comp) * L[l];
    atomicAdd(b + (int64_t)NB * vk + ob, fld_b <= 1 ? s : cf.stab * s);
  }
}

// sigma_s avg(h) int_F [sigma(u) n].[sigma(v) n] over dS(3) (side 0: in) / dS(4) (side 1: out), by the 2-point Gauss
// rule on the edge.  The edge parameter runs from the lower- to the higher-global-id vertex in both cells (as
// k_quad_ghost_neumann), so both sides evaluate the same physical points.  One thread per (facet, trial side, node,
// component) = 16 per facet, each summing the 16 test entries of its column.
__global__ void __launch_bounds__(kBlockEl) k_elasticity_quad_facets(
    phifem_mesh m, const int32_t* __restrict__ facets, int64_t n_facets, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_facets, int side, phifem_elasticity_params prm, double* __restrict__ data) {
  using S_ = ES<2>;
  constexpr int NV = quad::NV, NB = S_::NB, NT = 2 * NV * 2;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_facets * NT) return;
  const int64_t e = t / NT;
  int rem = (int)(t - e * NT);
  const int sb = rem / (NV * 2);
  rem -= sb * (NV * 2);
  const int j = rem / 2, cb = rem - j * 2;
  const int32_t fct = __ldg(facets + e);
  const int2 cc = __ldg(reinterpret_cast<const int2*>(m.f2c) + fct);
  const double lm = side == 0 ? prm.lmbda_in : prm.lmbda_out, mu = side == 0 ? prm.mu_in : prm.mu_out;
  const int ou = side == 0 ? S_::UI : S_::UO;
  quad::Cell g[2];
  double n[2][2], len = 0.0, r0[2][2], r1[2][2];   // per side: normal, reference end points of the parameter
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int64_t c = s == 0 ? cc.x : cc.y;
    quad::load_cell(m, c, g[s]);
    int o = 0;
#pragma unroll
    for (int k = 0; k < NV; ++k)
      if (__ldg(m.c2f + c * NV + k) == fct) o = k;
    int la = quad::facet_vertex(o, 0), lb = quad::facet_vertex(o, 1);
    if (__ldg(m.cells + c * NV + la) > __ldg(m.cells + c * NV + lb)) {
      const int tmp = la;
      la = lb;
      lb = tmp;
    }
    r0[s][0] = la & 1; r0[s][1] = la >> 1;
    r1[s][0] = lb & 1; r1[s][1] = lb >> 1;
    double l;
    quad::edge_normal(g[s], o, n[s], l);
    if (s == 0) len = l;
  }
  const double coef = prm.sigma_s * 0.5 * (sqrt(g[0].h2) + sqrt(g[1].h2)) * len * 0.5;   // 0.5: the Gauss weight
  double E[2][NV][2];
#pragma unroll
  for (int sa = 0; sa < 2; ++sa)
#pragma unroll
    for (int k = 0; k < NV; ++k) E[sa][k][0] = E[sa][k][1] = 0.0;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const double tq = q == 0 ? kGauss2Lo : kGauss2Hi;
    double G[2][NV][2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      double N[NV], Jit[2][2];
      quad::map_point(g[s], (1.0 - tq) * r0[s][0] + tq * r1[s][0], (1.0 - tq) * r0[s][1] + tq * r1[s][1], N, G[s],
                      Jit);
    }
    double Gb[2] = {G[0][0][0], G[0][0][1]}, nb[2] = {n[0][0], n[0][1]}, Jb[2];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
      for (int k = 0; k < NV; ++k)
        if (s == sb && k == j) {
          Gb[0] = G[s][k][0];
          Gb[1] = G[s][k][1];
          nb[0] = n[s][0];
          nb[1] = n[s][1];
        }
    stress_normal(Gb, nb, cb, lm, mu, Jb);
#pragma unroll
    for (int sa = 0; sa < 2; ++sa)
#pragma unroll
      for (int k = 0; k < NV; ++k)
#pragma unroll
        for (int ca = 0; ca < 2; ++ca) {
          double Ja[2];
          stress_normal(G[sa][k], n[sa], ca, lm, mu, Ja);
          E[sa][k][ca] += coef * (Ja[0] * Jb[0] + Ja[1] * Jb[1]);
        }
  }
  const int colslot = sb * NV + j;
#pragma unroll
  for (int sa = 0; sa < 2; ++sa)
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vk = __ldg(m.cells + (int64_t)(sa == 0 ? cc.x : cc.y) * NV + k);
      const int pos = __ldg(pos_facets + (e * (2 * NV) + sa * NV + k) * (2 * NV) + colslot);
#pragma unroll
      for (int ca = 0; ca < 2; ++ca)
        atomicAdd(data + block_address(vptr, vk, ou + ca, pos, ou + cb, NB), E[sa][k][ca]);
    }
}

// int_{ds(100)} (y_in n).v_in (side 0) / int_{ds(101)} (y_out n).v_out (side 1) on quadrilaterals: Q1 restricted to the
// straight edge is linear, so the entry (v_(k,c), y_(j,(c,s))) is n_s |F| (1 + delta_kj) / 6 for k, j the edge's two
// vertices (as k_quad_boundary_neumann).  One thread per (entity, k, j).
__global__ void __launch_bounds__(kBlockEl) k_elasticity_quad_boundary(
    phifem_mesh m, const int32_t* __restrict__ entities, int64_t n_entities, const int32_t* __restrict__ vptr,
    const int32_t* __restrict__ pos_boundary, int side, double* __restrict__ data) {
  using S_ = ES<2>;
  constexpr int NV = quad::NV, NB = S_::NB;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_entities * NV * NV) return;
  const int64_t e = t / (NV * NV);
  const int rem = (int)(t - e * NV * NV);
  const int k = rem / NV, j = rem - k * NV;
  const int64_t c = __ldg(entities + 2 * e);
  const int o = __ldg(entities + 2 * e + 1);
  const int la = quad::facet_vertex(o, 0), lb = quad::facet_vertex(o, 1);
  if ((k != la && k != lb) || (j != la && j != lb)) return;   // N_k or N_j vanishes on the edge
  quad::Cell g;
  quad::load_cell(m, c, g);
  double n[2], len;
  quad::edge_normal(g, o, n, len);
  const double mkj = len * (k == j ? 2.0 : 1.0) * (1.0 / 6.0);
  const int ou = side == 0 ? S_::UI : S_::UO, oy = side == 0 ? S_::YI : S_::YO;
  const int vk = __ldg(m.cells + c * NV + k);
  const int pos = __ldg(pos_boundary + e * (NV * NV) + rem);
#pragma unroll
  for (int cc = 0; cc < 2; ++cc)
#pragma unroll
    for (int s = 0; s < 2; ++s)
      atomicAdd(data + block_address(vptr, vk, ou + cc, pos, oy + cc * 2 + s, NB), n[s] * mkj);
}

// Dirichlet conditions on an assembled CSR system, one warp per row: rows and columns of constrained dofs zeroed,
// their diagonal 1, b <- b - A g on the free rows, b = g on the constrained ones
// (dolfinx assemble_matrix(bcs=) + apply_lifting + bc.set: main.py:238, 271-274)
__global__ void __launch_bounds__(256) k_apply_dirichlet(int64_t n_rows, const int32_t* __restrict__ indptr,
                                                         const int32_t* __restrict__ indices,
                                                         const int8_t* __restrict__ marker,
                                                         const double* __restrict__ values, double* __restrict__ data,
                                                         double* __restrict__ b) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = warp; row < n_rows; row += n_warps) {
    const bool rbc = marker[row] != 0;
    double lift = 0.0;
    const int end = __ldg(indptr + row + 1);
    for (int i = __ldg(indptr + row) + lane; i < end; i += 32) {
      const int col = __ldg(indices + i);
      const bool cbc = marker[col] != 0;
      if (rbc || cbc) {
        if (!rbc) lift += data[i] * __ldg(values + col);
        data[i] = (rbc && col == row) ? 1.0 : 0.0;
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) lift += __shfl_xor_sync(0xffffffffu, lift, s);
    if (lane == 0) b[row] = rbc ? __ldg(values + row) : b[row] - lift;
  }
}

// The same on a STRUCTURALLY SYMMETRIC pattern (every operator of this library: one space for trial and test functions),
// driven by the list of constrained dofs: one warp per constrained dof c zeroes row c (diagonal 1, b[c] = g[c]) and, for
// every entry (c, j) with j free, finds the mirrored entry (j, c) by binary search in row j, lifts it into b[j] and zeroes
// it.  Work O(sum of the constrained rows' lengths) instead of a pass over the whole matrix (3.8 ms of the 6.3 ms step
// of the 2 M-triangle elasticity operator: 1.4e9 entries for 8 000 constrained dofs).  Parity-tested on small systems
// only so far (its first large run hit an int32 overflow in the bisection, fixed above, when the GPU budget of the round
// ran out): opt-in (`symmetric_bc=True`) until it has been timed at scale.
__global__ void __launch_bounds__(256) k_apply_dirichlet_list(const int32_t* __restrict__ indptr,
                                                              const int32_t* __restrict__ indices,
                                                              const int32_t* __restrict__ bc_dofs, int64_t n_bc,
                                                              const int8_t* __restrict__ marker,
                                                              const double* __restrict__ values,
                                                              double* __restrict__ data, double* __restrict__ b) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t w = warp; w < n_bc; w += n_warps) {
    const int c = __ldg(bc_dofs + w);
    const double g = __ldg(values + c);
    const int end = __ldg(indptr + c + 1);
    for (int i = __ldg(indptr + c) + lane; i < end; i += 32) {
      const int col = __ldg(indices + i);
      data[i] = col == c ? 1.0 : 0.0;
      if (marker[col] != 0) continue;  // a constrained row zeroes itself
      int lo = __ldg(indptr + col), hi = __ldg(indptr + col + 1);
      while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);  // (lo + hi) overflows int32 beyond 2^30 entries
        if (__ldg(indices + mid) < c) lo = mid + 1;
        else hi = mid;
      }
      if (lo < __ldg(indptr + col + 1) && __ldg(indices + lo) == c) {
        const double v = data[lo];
        if (v != 0.0) atomicAdd(b + col, -v * g);
        data[lo] = 0.0;
      }
    }
    if (lane == 0) b[c] = g;
  }
}

// the cell type: triangles (D = 2), tetrahedra (D = 3) and quadrilaterals (D = 2, is_quad)
int check_mesh(const phifem_mesh* m, int& D, bool& is_quad) {
  PHIFEM_CHECK_ARG(m != nullptr && m->x && m->cells, "mesh is null");
  if (m->cell_type != PHIFEM_TRIANGLE && m->cell_type != PHIFEM_TETRAHEDRON && m->cell_type != PHIFEM_QUADRILATERAL) {
    set_error("the interface-elasticity operator supports triangles, quadrilaterals and tetrahedra, got cell type %d",
              m->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  is_quad = m->cell_type == PHIFEM_QUADRILATERAL;
  D = m->cell_type == PHIFEM_TETRAHEDRON ? 3 : 2;
  PHIFEM_CHECK_ARG(m->gdim == D, "gdim mismatch");
  return PHIFEM_OK;
}

}  // namespace
}  // namespace phifem

using namespace phifem;

extern "C" int phifem_assemble_elasticity_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi,
                                                const phifem_quadrature* quad, const double* phi, const double* f,
                                                const int8_t* cell_tags8, const int32_t* cut_cells, int64_t n_cut,
                                                const int32_t* vptr, const int32_t* pos_cells,
                                                const phifem_elasticity_params* prm, double* data, double* b,
                                                void* stream) {
  int D = 0;
  bool is_quad = false;
  if (int rc = check_mesh(mesh, D, is_quad)) return rc;
  if (mesh->n_cells == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(space_phi && quad && prm, "space / quadrature / parameters are null");
  if (space_phi->degree != 1 && space_phi->degree != 2) {
    set_error("level-set degree %d: degrees 1 and 2 are implemented", space_phi->degree);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  if (is_quad) {
    PHIFEM_CHECK_ARG(space_phi->n_dofs_per_cell == 4 || space_phi->n_dofs_per_cell == 9,
                     "space_phi->n_dofs_per_cell must be 4 (Q1) or 9 (Q2) on quadrilaterals");
    PHIFEM_CHECK_ARG(space_phi->degree == (space_phi->n_dofs_per_cell == 4 ? 1 : 2),
                     "space_phi->degree does not match n_dofs_per_cell on quadrilaterals");
  }
  PHIFEM_CHECK_ARG(space_phi->dofmap || space_phi->degree == 1, "a P2 level set needs its dofmap");
  PHIFEM_CHECK_ARG(quad->cell_points && quad->cell_weights && quad->n_cell_points > 0 &&
                       quad->n_cell_points <= kMaxQuadPoints, "cell quadrature rule (1..128 points)");
  PHIFEM_CHECK_ARG(phi && f && cell_tags8 && vptr && pos_cells && data && b, "null array");
  PHIFEM_CHECK_ARG(n_cut >= 0 && (n_cut == 0 || cut_cells), "cut-cell list");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nv = is_quad ? quad::NV : D + 1, nb = 3 * D + 2 * D * D;
  {
    const int64_t blocks = (mesh->n_cells * (int64_t)(nv * nv) + kBlockEl - 1) / kBlockEl;
    PHIFEM_CHECK_ARG(blocks < (1ll << 31), "too many cells for one launch");
    if (is_quad) k_elasticity_quad_uncut<<<(unsigned)blocks, kBlockEl, 0, st>>>(*mesh, f, cell_tags8, vptr, pos_cells, *prm, data, b);
    else if (D == 2) k_elasticity_uncut<2><<<(unsigned)blocks, kBlockEl, 0, st>>>(*mesh, f, cell_tags8, vptr, pos_cells, *prm, data, b);
    else k_elasticity_uncut<3><<<(unsigned)blocks, kBlockEl, 0, st>>>(*mesh, f, cell_tags8, vptr, pos_cells, *prm, data, b);
    PHIFEM_CHECK_LAUNCH();
  }
  if (n_cut == 0) return PHIFEM_OK;
  const int64_t blocks = (n_cut * (int64_t)(nv * nv * nb) + kBlockEl - 1) / kBlockEl;
  PHIFEM_CHECK_ARG(blocks < (1ll << 31), "too many cut cells for one launch");
  const unsigned grid = (unsigned)blocks;
#define PHIFEM_EL_LAUNCH(DD, KK)                                                                                    \
  k_elasticity_cells<DD, KK><<<grid, kBlockEl, 0, st>>>(*mesh, *space_phi, quad->cell_points, quad->cell_weights,     \
                                                        quad->n_cell_points, phi, f, cut_cells, n_cut, vptr, pos_cells, \
                                                        *prm, data, b)
#define PHIFEM_EL_QUAD_LAUNCH(KK)                                                                                    \
  k_elasticity_quad_cells<KK><<<grid, kBlockEl, 0, st>>>(*mesh, *space_phi, quad->cell_points, quad->cell_weights,     \
                                                        quad->n_cell_points, phi, f, cut_cells, n_cut, vptr, pos_cells, \
                                                        *prm, data, b)
  if (is_quad && space_phi->degree == 1) PHIFEM_EL_QUAD_LAUNCH(1);
  else if (is_quad) PHIFEM_EL_QUAD_LAUNCH(2);
  else if (D == 2 && space_phi->degree == 1) PHIFEM_EL_LAUNCH(2, 1);
  else if (D == 2) PHIFEM_EL_LAUNCH(2, 2);
  else if (space_phi->degree == 1) PHIFEM_EL_LAUNCH(3, 1);
  else PHIFEM_EL_LAUNCH(3, 2);
#undef PHIFEM_EL_LAUNCH
#undef PHIFEM_EL_QUAD_LAUNCH
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_elasticity_facets(const phifem_mesh* mesh, const int32_t* facets, int64_t n_facets,
                                                 const int32_t* vptr, const int32_t* pos_facets, int32_t side,
                                                 const phifem_elasticity_params* prm, double* data, void* stream) {
  int D = 0;
  bool is_quad = false;
  if (int rc = check_mesh(mesh, D, is_quad)) return rc;
  if (n_facets == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(mesh->c2f && mesh->f2c, "mesh without facet connectivity");
  PHIFEM_CHECK_ARG(facets && vptr && pos_facets && prm && data, "null array");
  PHIFEM_CHECK_ARG(side == 0 || side == 1, "side must be 0 (in) or 1 (out)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t threads = n_facets * 2 * (is_quad ? quad::NV : D + 1) * D;
  const unsigned grid = (unsigned)((threads + kBlockEl - 1) / kBlockEl);
  if (is_quad) k_elasticity_quad_facets<<<grid, kBlockEl, 0, st>>>(*mesh, facets, n_facets, vptr, pos_facets, side, *prm, data);
  else if (D == 2) k_elasticity_facets<2><<<grid, kBlockEl, 0, st>>>(*mesh, facets, n_facets, vptr, pos_facets, side, *prm, data);
  else k_elasticity_facets<3><<<grid, kBlockEl, 0, st>>>(*mesh, facets, n_facets, vptr, pos_facets, side, *prm, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_assemble_elasticity_boundary(const phifem_mesh* mesh, const int32_t* entities,
                                                   int64_t n_entities, const int32_t* vptr,
                                                   const int32_t* pos_boundary, int32_t side, double* data,
                                                   void* stream) {
  int D = 0;
  bool is_quad = false;
  if (int rc = check_mesh(mesh, D, is_quad)) return rc;
  if (n_entities == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(entities && vptr && pos_boundary && data, "null array");
  PHIFEM_CHECK_ARG(side == 0 || side == 1, "side must be 0 (in) or 1 (out)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nv = is_quad ? quad::NV : D + 1;
  const int64_t threads = n_entities * nv * nv;
  const unsigned grid = (unsigned)((threads + kBlockEl - 1) / kBlockEl);
  if (is_quad) k_elasticity_quad_boundary<<<grid, kBlockEl, 0, st>>>(*mesh, entities, n_entities, vptr, pos_boundary, side, data);
  else if (D == 2) k_elasticity_boundary<2><<<grid, kBlockEl, 0, st>>>(*mesh, entities, n_entities, vptr, pos_boundary, side, data);
  else k_elasticity_boundary<3><<<grid, kBlockEl, 0, st>>>(*mesh, entities, n_entities, vptr, pos_boundary, side, data);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_apply_dirichlet(int64_t n_rows, const int32_t* indptr, const int32_t* indices,
                                      const int8_t* bc_marker, const double* bc_values, double* data, double* b,
                                      void* stream) {
  if (n_rows == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(n_rows > 0 && indptr && indices && bc_marker && bc_values && data && b, "null array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(n_rows * 32, 256, 8);
  k_apply_dirichlet<<<grid, 256, 0, st>>>(n_rows, indptr, indices, bc_marker, bc_values, data, b);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}

extern "C" int phifem_apply_dirichlet_symmetric(int64_t n_rows, const int32_t* indptr, const int32_t* indices,
                                                const int32_t* bc_dofs, int64_t n_bc, const int8_t* bc_marker,
                                                const double* bc_values, double* data, double* b, void* stream) {
  if (n_rows == 0 || n_bc == 0) return PHIFEM_OK;
  PHIFEM_CHECK_ARG(n_rows > 0 && n_bc > 0 && indptr && indices && bc_dofs && bc_marker && bc_values && data && b,
                   "null array");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(n_bc * 32, 256, 8);
  k_apply_dirichlet_list<<<grid, 256, 0, st>>>(indptr, indices, bc_dofs, n_bc, bc_marker, bc_values, data, b);
  PHIFEM_CHECK_LAUNCH();
  return PHIFEM_OK;
}
