// A host without Python for the interface-elasticity operator (demo/interface-elasticity): cut-cell tags, the blocked
// CSR pattern and the assembly of the phi-FEM operator on the mixed space (u_in, u_out, y_in, y_out, p) through the
// C ABI of libphifem_b200.so alone (include/phifem_b200.h): tags -> phifem_integration_entities for ds(100) / ds(101)
// -> phifem_elasticity_pattern_create -> phifem_assemble_elasticity_{cells,facets,boundary} ->
// phifem_apply_dirichlet_symmetric on the u_in / u_out dofs of the mesh-boundary vertices.
// The mesh is a unit square of 2 n^2 triangles built on the host, the level set P1.
//
//   nvcc -O2 -std=c++17 -gencode arch=compute_100a,code=sm_100a examples/capi_host_elasticity.cu -Iinclude \
//        -Lphifem_b200 -lphifem_b200 -Xlinker -rpath=$PWD/phifem_b200 -o capi_host_elasticity && \
//   ./capi_host_elasticity 48
//
// Prints key=value pairs: tag counts, nnz, n_pairs, n_cut, n_facets_in, n_facets_out, n_entities_in, n_entities_out,
// n_bc, a checksum of the column indices, sum |data| and sum b.
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

// The cut-cell rule of phifem_b200/quadrature.py rules_for_neumann(2, 1) for triangles (barycentric points, weights
// summing to 1): the 6-point rule of degree 4.
const std::vector<double> kCellPoints = {
    0.10810301816807033, 0.44594849091596483, 0.44594849091596483, 0.44594849091596483, 0.10810301816807033,
    0.44594849091596483, 0.44594849091596483, 0.44594849091596483, 0.10810301816807033, 0.09157621350977066,
    0.09157621350977066, 0.8168475729804587,  0.09157621350977066, 0.8168475729804587,  0.09157621350977066,
    0.8168475729804587,  0.09157621350977066, 0.09157621350977066};
const std::vector<double> kCellWeights = {0.22338158967801153, 0.22338158967801153, 0.22338158967801153,
                                          0.1099517436553218,  0.1099517436553218,  0.1099517436553218};

// ds entities (cell, local facet) of the Gamma_h facets tagged `facet_tag`, seen from the cells of `cell_mask`
static int entities_of(const phifem_mesh& mesh, const int8_t* c8, const int8_t* f8, int facet_tag, uint32_t cell_mask,
                       int32_t** ents, int64_t* n) {
  *n = 0;
  CHECK(phifem_integration_entities(&mesh, c8, f8, facet_tag, cell_mask, nullptr, 0, n, nullptr));
  cudaMalloc(ents, std::max<int64_t>(1, *n) * 2 * sizeof(int32_t));
  CHECK(phifem_integration_entities(&mesh, c8, f8, facet_tag, cell_mask, *ents, *n, n, nullptr));
  return 0;
}

int main(int argc, char** argv) {
  const int n = argc > 1 ? std::atoi(argv[1]) : 32;
  // mesh: vertex (i, j) -> i (n + 1) + j at (i / n, j / n); every square split along its "right" diagonal
  const int nvx = (n + 1) * (n + 1), nc = 2 * n * n;
  std::vector<double> x(2 * (size_t)nvx), phi(nvx), f(2 * (size_t)nvx);
  for (int i = 0; i <= n; ++i)
    for (int j = 0; j <= n; ++j) {
      const int v = i * (n + 1) + j;
      x[2 * v] = (double)i / n;
      x[2 * v + 1] = (double)j / n;
    }
  for (int v = 0; v < nvx; ++v) {
    const double dx = x[2 * v] - 0.503, dy = x[2 * v + 1] - 0.497;
    phi[v] = dx * dx + dy * dy - 0.3 * 0.3;
    f[2 * v] = 1.0 + x[2 * v] + 2.0 * x[2 * v + 1];  // the P1 vector source f [Nv, 2]
    f[2 * v + 1] = x[2 * v] - 0.5 * x[2 * v + 1];
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
  std::vector<char> on_boundary(nvx, 0);
  for (const auto& kv : facet_of)
    if (f2c[2 * kv.second + 1] < 0) {
      bfacets.push_back(kv.second);
      on_boundary[kv.first[0]] = on_boundary[kv.first[1]] = 1;
    }

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

  // ds(100): Gamma_h facets (tag 4) seen from the cells tagged 1 / 2; ds(101): facets tagged 3 seen from cells 2 / 3
  int32_t *ents_in = nullptr, *ents_out = nullptr;
  int64_t n_in = 0, n_out = 0;
  if (entities_of(mesh, cell_tags8, facet_tags8, 4, (1u << 1) | (1u << 2), &ents_in, &n_in)) return 1;
  if (entities_of(mesh, cell_tags8, facet_tags8, 3, (1u << 2) | (1u << 3), &ents_out, &n_out)) return 1;

  phifem_elasticity_pattern* pat = nullptr;
  CHECK(phifem_elasticity_pattern_create(&mesh, cell_tags8, facet_tags8, ents_in, n_in, ents_out, n_out, &pat, nullptr));
  phifem_elasticity_pattern_view v;
  CHECK(phifem_elasticity_pattern_view_of(pat, &v));

  // the demo's materials (data.py:13-22) and penalty weights (main.py:189-190), pen_coef = stab_coef = 1
  const double E_in = 1.0, nu_in = 0.3, E_out = 0.001, nu_out = 0.3;
  phifem_elasticity_params prm;
  prm.lmbda_in = E_in * nu_in / (1.0 + nu_in) / (1.0 - 2.0 * nu_in);
  prm.mu_in = E_in / 2.0 / (1.0 + nu_in);
  prm.lmbda_out = E_out * nu_out / (1.0 + nu_out) / (1.0 - 2.0 * nu_out);
  prm.mu_out = E_out / 2.0 / (1.0 + nu_out);
  prm.coef_in = std::pow(E_in / (E_in + E_out), 2);
  prm.coef_out = std::pow(E_out / (E_in + E_out), 2);
  prm.gamma = 1.0;
  prm.sigma_s = 1.0;

  phifem_pk_space p1 = {1, 3, nvx, mesh.cells};  // the P1 level-set space: vertex dofs
  phifem_quadrature q = {6, 0, to_device(kCellPoints), to_device(kCellWeights), nullptr, nullptr};
  double *data, *b;
  cudaMalloc(&data, std::max<int64_t>(1, v.nnz) * sizeof(double));
  cudaMalloc(&b, v.n_rows * sizeof(double));
  cudaMemset(data, 0, v.nnz * sizeof(double));
  cudaMemset(b, 0, v.n_rows * sizeof(double));
  CHECK(phifem_assemble_elasticity_cells(&mesh, &p1, &q, d_phi, d_f, cell_tags8, v.cut_cells, v.n_cut, v.vptr,
                                         v.pos_cells, &prm, data, b, nullptr));
  if (v.n_facets_in)
    CHECK(phifem_assemble_elasticity_facets(&mesh, v.facets_in, v.n_facets_in, v.vptr, v.pos_facets_in, 0, &prm, data,
                                            nullptr));
  if (v.n_facets_out)
    CHECK(phifem_assemble_elasticity_facets(&mesh, v.facets_out, v.n_facets_out, v.vptr, v.pos_facets_out, 1, &prm,
                                            data, nullptr));
  if (n_in)
    CHECK(phifem_assemble_elasticity_boundary(&mesh, ents_in, n_in, v.vptr, v.pos_entities_in, 0, data, nullptr));
  if (n_out)
    CHECK(phifem_assemble_elasticity_boundary(&mesh, ents_out, n_out, v.vptr, v.pos_entities_out, 1, data, nullptr));

  // Dirichlet conditions u_in = u_out = g on the mesh-boundary vertices, g = (x - y, x + 0.5 y); dofs NB v + o with
  // o = c for u_in and 2 + c for u_out (the list ascending, without duplicates)
  const int nb = v.nb;
  std::vector<int32_t> bc_dofs;
  std::vector<int8_t> marker(v.n_rows, 0);
  std::vector<double> values(v.n_rows, 0.0);
  for (int s = 0; s < nvx; ++s) {
    if (!on_boundary[s]) continue;
    const double g[2] = {x[2 * s] - x[2 * s + 1], x[2 * s] + 0.5 * x[2 * s + 1]};
    for (int o = 0; o < 4; ++o) {
      const int dof = nb * s + o;
      bc_dofs.push_back(dof);
      marker[dof] = 1;
      values[dof] = g[o % 2];
    }
  }
  CHECK(phifem_apply_dirichlet_symmetric(v.n_rows, v.indptr, v.indices, to_device(bc_dofs), (int64_t)bc_dofs.size(),
                                         to_device(marker), to_device(values), data, b, nullptr));
  if (cudaDeviceSynchronize() != cudaSuccess) {
    std::fprintf(stderr, "CUDA error: %s\n", cudaGetErrorString(cudaGetLastError()));
    return 1;
  }

  std::vector<double> h_data(v.nnz), h_b(v.n_rows);
  std::vector<int32_t> h_idx(v.nnz);
  cudaMemcpy(h_data.data(), data, v.nnz * sizeof(double), cudaMemcpyDeviceToHost);
  cudaMemcpy(h_b.data(), b, v.n_rows * sizeof(double), cudaMemcpyDeviceToHost);
  cudaMemcpy(h_idx.data(), v.indices, v.nnz * sizeof(int32_t), cudaMemcpyDeviceToHost);
  long long idx_sum = 0;
  double abs_sum = 0.0, b_sum = 0.0;
  for (int64_t i = 0; i < v.nnz; ++i) {
    abs_sum += std::fabs(h_data[i]);
    idx_sum += (long long)h_idx[i] * (i % 7 + 1);
  }
  for (double t : h_b) b_sum += t;
  std::printf("nnz=%lld n_pairs=%lld n_cut=%lld n_facets_in=%lld n_facets_out=%lld n_entities_in=%lld "
              "n_entities_out=%lld n_bc=%lld indices_checksum=%lld data_abs_sum=%.17g b_sum=%.17g\n",
              (long long)v.nnz, (long long)v.n_pairs, (long long)v.n_cut, (long long)v.n_facets_in,
              (long long)v.n_facets_out, (long long)v.n_entities_in, (long long)v.n_entities_out,
              (long long)bc_dofs.size(), idx_sum, abs_sum, b_sum);
  phifem_elasticity_pattern_destroy(pat);
  return 0;
}
