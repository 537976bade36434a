// A host without Python for the mixed-space operators: cut-cell tags, CSR pattern and assembly of the weak-Dirichlet
// (P1 x P1, demo/weak-dirichlet/flower) and Neumann (P1 x P1^2 x DG0, demo/neumann/square) phi-FEM operators through the
// C ABI of libphifem_b200.so alone (include/phifem_b200.h): tags -> phifem_integration_entities ->
// phifem_pk_pattern_create over the caller's mixed dofmap -> phifem_assemble_weak_*_pk / phifem_assemble_neumann_*.
// The mesh is a unit square of 2 n^2 triangles built on the host, the level set P1.
//
//   nvcc -O2 -std=c++17 -gencode arch=compute_100a,code=sm_100a examples/capi_host_pk.cu -Iinclude \
//        -Lphifem_b200 -lphifem_b200 -Xlinker -rpath=$PWD/phifem_b200 -o capi_host_pk && ./capi_host_pk 48
//
// Prints key=value pairs: tag counts, then per operator (prefix weak_ / neumann_) nnz, n_active, n_cut, n_ghost,
// n_entities, a checksum of the column indices, sum |data| and sum b.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include "phifem_b200.h"

#define CHECK(call)                                                                   \
  do {                                                                                \
    int rc__ = (call);                                                                \
    if (rc__ != 0) {                                                                  \
      std::fprintf(stderr, "%s failed (%d): %s\n", #call, rc__, phifem_last_error()); \
      return 1;                                                                       \
    }                                                                                 \
  } while (0)

template <typename T>
T* to_device(const std::vector<T>& v) {
  T* d = nullptr;
  cudaMalloc(&d, std::max<size_t>(1, v.size()) * sizeof(T));
  cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
  return d;
}

// Quadrature tables of phifem_b200/quadrature.py for triangles (barycentric points, weights summing to 1):
// rules_for_weak(2, 1, 1) and rules_for_neumann(2, 1) share the 6-point cell rule of degree 4.
const std::vector<double> kCellPoints = {
    0.10810301816807033, 0.44594849091596483, 0.44594849091596483, 0.44594849091596483, 0.10810301816807033,
    0.44594849091596483, 0.44594849091596483, 0.44594849091596483, 0.10810301816807033, 0.09157621350977066,
    0.09157621350977066, 0.8168475729804587,  0.09157621350977066, 0.8168475729804587,  0.09157621350977066,
    0.8168475729804587,  0.09157621350977066, 0.09157621350977066};
const std::vector<double> kCellWeights = {0.22338158967801153, 0.22338158967801153, 0.22338158967801153,
                                          0.1099517436553218,  0.1099517436553218,  0.1099517436553218};
// facets: rules_for_weak(2, 1, 1) = the 1-point segment rule, rules_for_neumann(2, 1) = the 2-point Gauss rule
const std::vector<double> kWeakFacetPoints = {0.5, 0.5};
const std::vector<double> kWeakFacetWeights = {1.0};
const std::vector<double> kNeumannFacetPoints = {0.7886751345948129, 0.21132486540518713, 0.21132486540518713,
                                                 0.7886751345948129};
const std::vector<double> kNeumannFacetWeights = {0.4999999999999999, 0.4999999999999999};

struct Sums {
  long long idx_sum = 0;
  double abs_sum = 0.0, b_sum = 0.0;
};

// checksums of an assembled system (after a device synchronisation)
static int sums_of(const phifem_pk_pattern_view& v, const double* data, const double* b, Sums* s) {
  if (cudaDeviceSynchronize() != cudaSuccess) {
    std::fprintf(stderr, "CUDA error: %s\n", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }
  std::vector<double> h_data(v.nnz), h_b(v.n_rows);
  std::vector<int32_t> h_idx(v.nnz);
  cudaMemcpy(h_data.data(), data, v.nnz * sizeof(double), cudaMemcpyDeviceToHost);
  cudaMemcpy(h_b.data(), b, v.n_rows * sizeof(double), cudaMemcpyDeviceToHost);
  cudaMemcpy(h_idx.data(), v.indices, v.nnz * sizeof(int32_t), cudaMemcpyDeviceToHost);
  for (int64_t i = 0; i < v.nnz; ++i) {
    s->abs_sum += std::fabs(h_data[i]);
    s->idx_sum += (long long)h_idx[i] * (i % 7 + 1);
  }
  for (double t : h_b) s->b_sum += t;
  return 0;
}

static void print_sums(const char* name, const phifem_pk_pattern_view& v, const Sums& s) {
  std::printf("%s_nnz=%lld %s_n_active=%lld %s_n_cut=%lld %s_n_ghost=%lld %s_n_entities=%lld "
              "%s_indices_checksum=%lld %s_data_abs_sum=%.17g %s_b_sum=%.17g\n",
              name, (long long)v.nnz, name, (long long)v.n_active, name, (long long)v.n_cut, name,
              (long long)v.n_ghost, name, (long long)v.n_entities, name, s.idx_sum, name, s.abs_sum, name, s.b_sum);
}

int main(int argc, char** argv) {
  const int n = argc > 1 ? std::atoi(argv[1]) : 32;
  // mesh: vertex (i, j) -> i (n + 1) + j at (i / n, j / n); every square split along its "right" diagonal
  const int nvx = (n + 1) * (n + 1), nc = 2 * n * n;
  std::vector<double> x(2 * (size_t)nvx), phi(nvx), f(nvx), g(nvx);
  for (int i = 0; i <= n; ++i)
    for (int j = 0; j <= n; ++j) {
      const int v = i * (n + 1) + j;
      x[2 * v] = (double)i / n;
      x[2 * v + 1] = (double)j / n;
    }
  for (int v = 0; v < nvx; ++v) {
    const double dx = x[2 * v] - 0.503, dy = x[2 * v + 1] - 0.497;
    phi[v] = dx * dx + dy * dy - 0.3 * 0.3;
    f[v] = 1.0 + x[2 * v] + 2.0 * x[2 * v + 1];
    g[v] = x[2 * v] - 0.5 * x[2 * v + 1];  // Dirichlet data u_D (weak) and Neumann data u_N
  }
  std::vector<int32_t> cells(3 * (size_t)nc);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      const int v00 = i * (n + 1) + j, v10 = v00 + n + 1, v01 = v00 + 1, v11 = v10 + 1, c = 2 * (i * n + j);
      const int t[6] = {v00, v10, v11, v00, v01, v11};
      std::copy(t, t + 6, cells.begin() + 3 * (size_t)c);
    }
  // facets = lexicographic rank of the sorted vertex pair (dolfinx serial numbering); local facet i opposite vertex i
  std::map<std::array<int, 2>, int> facet_of;
  for (int c = 0; c < nc; ++c)
    for (int i = 0; i < 3; ++i) {
      std::array<int, 2> e = {cells[3 * c + (i + 1) % 3], cells[3 * c + (i + 2) % 3]};
      if (e[0] > e[1]) std::swap(e[0], e[1]);
      facet_of.emplace(e, 0);
    }
  int nf = 0;
  for (auto& kv : facet_of) kv.second = nf++;
  std::vector<int32_t> c2f(3 * (size_t)nc), f2c(2 * (size_t)nf, -1), bfacets;
  for (int c = 0; c < nc; ++c)
    for (int i = 0; i < 3; ++i) {
      std::array<int, 2> e = {cells[3 * c + (i + 1) % 3], cells[3 * c + (i + 2) % 3]};
      if (e[0] > e[1]) std::swap(e[0], e[1]);
      const int fc = facet_of[e];
      c2f[3 * c + i] = fc;
      f2c[2 * fc + (f2c[2 * fc] < 0 ? 0 : 1)] = c;  // cells ascending: c grows
    }
  for (int fc = 0; fc < nf; ++fc)
    if (f2c[2 * fc + 1] < 0) bfacets.push_back(fc);

  phifem_mesh mesh = {};
  mesh.cell_type = PHIFEM_TRIANGLE;
  mesh.gdim = 2;
  mesh.n_vertices = nvx;
  mesh.n_cells = nc;
  mesh.n_facets = nf;
  mesh.x = to_device(x);
  mesh.cells = to_device(cells);
  mesh.c2f = to_device(c2f);
  mesh.f2c = to_device(f2c);
  mesh.boundary_facets = to_device(bfacets);
  mesh.n_boundary_facets = (int64_t)bfacets.size();
  {  // once per mesh: the static part of the ds detection on the mesh-boundary facets
    uint32_t* owner = nullptr;
    double* scale = nullptr;
    cudaMalloc(&owner, std::max<size_t>(1, bfacets.size()) * 2 * sizeof(uint32_t));
    cudaMalloc(&scale, std::max<size_t>(1, bfacets.size()) * 4 * sizeof(double));
    CHECK(phifem_boundary_records(&mesh, owner, scale, nullptr));
    mesh.boundary_owner = owner;
    mesh.boundary_scale = scale;
  }
  double* d_phi = to_device(phi);
  double* d_f = to_device(f);
  double* d_g = to_device(g);

  // P1 level set, detection degree 1: the detection points are the vertices (identity tables)
  const double ftab_h[3][2][3] = {{{0, 1, 0}, {0, 0, 1}}, {{1, 0, 0}, {0, 0, 1}}, {{1, 0, 0}, {0, 1, 0}}};
  std::vector<double> ftab(&ftab_h[0][0][0], &ftab_h[0][0][0] + 18);
  phifem_levelset ls = {};
  ls.mode = 0;
  ls.n_dofs_per_cell = 3;
  ls.n_cell_points = 3;
  ls.n_facet_points = 2;
  ls.coeffs = d_phi;
  ls.facet_table = to_device(ftab);

  int32_t *cell_tags, *facet_tags;
  int8_t *cell_tags8, *facet_tags8;
  uint8_t* scratch;
  int64_t* counters;
  cudaMalloc(&cell_tags, nc * sizeof(int32_t));
  cudaMalloc(&cell_tags8, nc);
  cudaMalloc(&facet_tags, nf * sizeof(int32_t));
  cudaMalloc(&facet_tags8, nf);
  cudaMalloc(&scratch, nvx + 3);
  cudaMalloc(&counters, PHIFEM_N_COUNTERS * sizeof(int64_t));
  cudaMemset(counters, 0, PHIFEM_N_COUNTERS * sizeof(int64_t));
  CHECK(phifem_tag_cells(&mesh, &ls, 0, cell_tags, cell_tags8, scratch, counters, nullptr));
  CHECK(phifem_tag_facets(&mesh, &ls, cell_tags8, facet_tags, facet_tags8, counters, nullptr));
  int64_t cnt[PHIFEM_N_COUNTERS];
  cudaMemcpy(cnt, counters, sizeof(cnt), cudaMemcpyDeviceToHost);
  std::printf("interior=%lld cut=%lld exterior=%lld\n", (long long)cnt[PHIFEM_CNT_INTERIOR],
              (long long)cnt[PHIFEM_CNT_CUT], (long long)cnt[PHIFEM_CNT_EXTERIOR]);

  // ds(100): Gamma_h facets (tag 4) seen from the cells tagged 1 / 2
  int64_t n_ent = 0;
  int32_t* ents = nullptr;
  CHECK(phifem_integration_entities(&mesh, cell_tags8, facet_tags8, 4, (1u << 1) | (1u << 2), nullptr, 0, &n_ent, nullptr));
  cudaMalloc(&ents, std::max<int64_t>(1, n_ent) * 2 * sizeof(int32_t));
  CHECK(phifem_integration_entities(&mesh, cell_tags8, facet_tags8, 4, (1u << 1) | (1u << 2), ents, n_ent, &n_ent, nullptr));

  // the scalar P1 space (u, p, f, u_D of the weak form) and the P1 level-set space: vertex dofs
  phifem_pk_space p1 = {1, 3, nvx, mesh.cells};

  {  // weak Dirichlet on (u, p) in P1 x P1: u at vertex s -> 2 s, p -> 2 s + 1; cell-local order [u dofs, p dofs]
    std::vector<int32_t> mixed(6 * (size_t)nc);
    for (int c = 0; c < nc; ++c)
      for (int i = 0; i < 3; ++i) {
        mixed[6 * c + i] = 2 * cells[3 * c + i];
        mixed[6 * c + 3 + i] = 2 * cells[3 * c + i] + 1;
      }
    int32_t* d_mixed = to_device(mixed);
    phifem_pk_pattern* pat = nullptr;
    CHECK(phifem_pk_pattern_create(&mesh, d_mixed, 6, 2 * (int64_t)nvx, cell_tags8, facet_tags8, (1u << 2) | (1u << 3),
                                   ents, n_ent, &pat, nullptr));
    phifem_pk_pattern_view v;
    CHECK(phifem_pk_pattern_view_of(pat, &v));
    phifem_quadrature q = {6, 1, to_device(kCellPoints), to_device(kCellWeights), to_device(kWeakFacetPoints),
                           to_device(kWeakFacetWeights)};
    double *data, *b;
    cudaMalloc(&data, std::max<int64_t>(1, v.nnz) * sizeof(double));
    cudaMalloc(&b, v.n_rows * sizeof(double));
    cudaMemset(data, 0, v.nnz * sizeof(double));
    cudaMemset(b, 0, v.n_rows * sizeof(double));
    const double gamma = 1.0, sigma = 1.0;  // pen_coef, stab_coef of the demo
    if (v.n_active)
      CHECK(phifem_assemble_weak_cells_pk(&mesh, &p1, &p1, &q, d_phi, d_f, d_g, cell_tags8, v.active, v.n_active,
                                          v.slots_cells, d_mixed, gamma, sigma, data, b, nullptr));
    if (v.n_entities)
      CHECK(phifem_assemble_weak_boundary_pk(&mesh, &p1, &q, ents, v.n_entities, v.slots_boundary, data, nullptr));
    if (v.n_ghost)
      CHECK(phifem_assemble_weak_ghost_pk(&mesh, &p1, &q, v.ghost, v.n_ghost, v.slots_ghost, sigma, data, nullptr));
    Sums s;
    if (sums_of(v, data, b, &s)) return 1;
    print_sums("weak", v, s);
    phifem_pk_pattern_destroy(pat);
  }

  {  // Neumann on (u, y, p) in P1 x P1^2 x DG0: u at vertex s -> 3 s, y_c -> 3 s + 1 + c, p of cell k -> 3 Nv + k;
     // cell-local order [u x3, y node-major x6, p]
    std::vector<int32_t> mixed(10 * (size_t)nc);
    for (int c = 0; c < nc; ++c) {
      for (int i = 0; i < 3; ++i) {
        const int s = cells[3 * c + i];
        mixed[10 * c + i] = 3 * s;
        mixed[10 * c + 3 + 2 * i] = 3 * s + 1;
        mixed[10 * c + 3 + 2 * i + 1] = 3 * s + 2;
      }
      mixed[10 * c + 9] = 3 * nvx + c;
    }
    int32_t* d_mixed = to_device(mixed);
    phifem_pk_pattern* pat = nullptr;
    CHECK(phifem_pk_pattern_create(&mesh, d_mixed, 10, 3 * (int64_t)nvx + nc, cell_tags8, facet_tags8, 1u << 3, ents,
                                   n_ent, &pat, nullptr));
    phifem_pk_pattern_view v;
    CHECK(phifem_pk_pattern_view_of(pat, &v));
    phifem_quadrature q = {6, 2, to_device(kCellPoints), to_device(kCellWeights), to_device(kNeumannFacetPoints),
                           to_device(kNeumannFacetWeights)};
    double *data, *b;
    cudaMalloc(&data, std::max<int64_t>(1, v.nnz) * sizeof(double));
    cudaMalloc(&b, v.n_rows * sizeof(double));
    cudaMemset(data, 0, v.nnz * sizeof(double));
    cudaMemset(b, 0, v.n_rows * sizeof(double));
    const double gamma = 1.0, sigma = 1.0;
    if (v.n_active)
      CHECK(phifem_assemble_neumann_cells(&mesh, &p1, &q, d_phi, d_f, d_g, cell_tags8, v.active, v.n_active,
                                          v.cut_positions, v.n_cut, v.slots_cells, d_mixed, gamma, 0.0, data, b,
                                          nullptr));
    if (v.n_entities)
      CHECK(phifem_assemble_neumann_boundary(&mesh, ents, v.n_entities, v.slots_boundary, data, nullptr));
    if (v.n_ghost)
      CHECK(phifem_assemble_neumann_ghost(&mesh, &q, v.ghost, v.n_ghost, v.slots_ghost, sigma, data, nullptr));
    Sums s;
    if (sums_of(v, data, b, &s)) return 1;
    print_sums("neumann", v, s);
    phifem_pk_pattern_destroy(pat);
  }
  return 0;
}
