// Symbolic phase of the P1 strong-Dirichlet operator behind the C ABI: what dolfinx does in
// `create_sparsity_pattern` + `create_matrix` when `assemble_matrix(form(a))` is first called
// (reference demo/strong-dirichlet/flower/main.py:121-123) -- the CSR pattern of the dofs coupled by the cells of
// dx((1,2)) and by the macro elements of the interior facets of dS((2,3)) [dep-knowledge, SURVEY.md C.3] -- plus the
// entity -> CSR-slot maps the per-entity kernels (phifem_assemble_{cells,boundary,ghost}_p1) scatter through.
// The Python package builds the same arrays with torch sort / unique (phifem_b200/assemble.py); this file lets a host
// without Python (a C++ / PETSc code base) run tags -> pattern -> assembly with the shared library alone.
//
// Device algorithm: stream compaction of the active cells and ghost facets (cub::DeviceSelect), one 64-bit key
// row * n_vertices + col per coupled vertex pair, radix sort + unique (cub) = the pattern, binary searches for the row
// pointers and the slot maps.  The same steps serve the quadrature-kernel operators (phifem_pk_pattern_create, over a
// caller-given dofmap) and the interface-elasticity operator (phifem_elasticity_pattern_create: the vertex graph, then
// its expansion into dense NB x NB blocks).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "common.cuh"

struct phifem_pattern {
  phifem_pattern_view v;
  void* owned[8];
  int n_owned;
};

struct phifem_pk_pattern {
  phifem_pk_pattern_view v;
  void* owned[8];
  int n_owned;
};

struct phifem_elasticity_pattern {
  phifem_elasticity_pattern_view v;
  void* owned[12];
  int n_owned;
};

namespace phifem {
// A private stream-ordered pool per device whose memory stays cached between calls (release threshold = max): the
// default pool hands its memory back to the driver at every synchronisation, and re-allocating the ~10 GB of sort
// scratch of config E costs ten times the sort.  phifem_pattern_release_scratch() trims it.
cudaMemPool_t g_pools[64] = {};
cudaMemPool_t scratch_pool() {  // also used by csrc/rows_plan.cu
  int dev = 0;
  cudaGetDevice(&dev);
  cudaMemPool_t& pool = g_pools[dev & 63];
  if (!pool) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    if (cudaMemPoolCreate(&pool, &props) != cudaSuccess) {
      pool = nullptr;
      return nullptr;
    }
    uint64_t keep = 6ull << 30;  // cached between calls up to 6 GiB (the row-gather plan of 50 M tetrahedra needs ~3);
                                 // anything above goes back to the driver at the next synchronisation
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  return pool;
}

namespace {

constexpr int kBlockSym = 256;

struct IsActiveCell {
  const int8_t* tags;
  __device__ bool operator()(int c) const { return tags[c] == 1 || tags[c] == 2; }
};
struct IsGhostFacet {
  const int8_t* tags;
  const int32_t* f2c;
  __device__ bool operator()(int f) const { return (tags[f] == 2 || tags[f] == 3) && f2c[2 * (int64_t)f + 1] >= 0; }
};

// macro vertex list of an interior facet: [facet vertices in the local order of cell + (= f2c[f][0]), opposite vertex of
// cell +, opposite vertex of cell -] (include/phifem_b200.h, phifem_assemble_ghost_p1)
__global__ void k_macro_vertices(phifem_mesh m, int nv, const int32_t* __restrict__ facets, int64_t n,
                                 int32_t* __restrict__ macro) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const int32_t f = facets[e];
  int32_t* out = macro + e * (nv + 1);
  int k = 0;
  for (int side = 0; side < 2; ++side) {
    const int64_t c = m.f2c[2 * (int64_t)f + side];
    int opposite = -1;
    for (int i = 0; i < nv; ++i) {
      const int32_t v = m.cells[c * nv + i];
      if (m.c2f[c * nv + i] == f) opposite = v;  // local facet i is opposite local vertex i
      else if (side == 0) out[k++] = v;
    }
    out[nv - 1 + side] = opposite;
  }
}

// keys row * n_vertices + col of every ordered vertex pair of every listed entity; verts[e * w + i]
__global__ void k_pair_keys(const int32_t* __restrict__ verts, int64_t n, int w, int64_t n_vertices,
                            int64_t* __restrict__ keys) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * w * w) return;
  const int64_t e = t / (w * w);
  const int r = (int)(t - e * w * w);
  keys[t] = (int64_t)verts[e * w + r / w] * n_vertices + verts[e * w + r % w];
}

// the same with an indirection: entity e = cells row list[e * stride] (active cells, one-sided entities)
__global__ void k_cell_pair_keys(const int32_t* __restrict__ cells, int nv, const int32_t* __restrict__ list,
                                 int stride, int64_t n, int64_t n_vertices, int64_t* __restrict__ keys) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * nv * nv) return;
  const int64_t e = t / (nv * nv);
  const int r = (int)(t - e * nv * nv);
  const int64_t c = list[e * stride];
  keys[t] = (int64_t)cells[c * nv + r / nv] * n_vertices + cells[c * nv + r % nv];
}

__device__ __forceinline__ int64_t lower_bound(const int64_t* __restrict__ a, int64_t n, int64_t key) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void k_slots(const int64_t* __restrict__ uniq, int64_t nnz, const int64_t* __restrict__ keys, int64_t n,
                        int32_t* __restrict__ slots) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) slots[t] = (int32_t)lower_bound(uniq, nnz, keys[t]);
}

__global__ void k_row_pointers(const int64_t* __restrict__ uniq, int64_t nnz, int64_t n_rows,
                               int32_t* __restrict__ indptr) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r <= n_rows) indptr[r] = (int32_t)lower_bound(uniq, nnz, r * n_rows);
}

__global__ void k_columns(const int64_t* __restrict__ uniq, int64_t nnz, int64_t n_rows,
                          int32_t* __restrict__ indices) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nnz) indices[t] = (int32_t)(uniq[t] % n_rows);
}

inline unsigned blocks_for(int64_t n) { return (unsigned)((n + kBlockSym - 1) / kBlockSym); }

// ---- quadrature-kernel operators (phifem_pk_pattern_create): the same keys over a caller-given pattern dofmap

struct IsMaskedGhostFacet {  // interior facets whose tag t has bit t set in `mask`
  const int8_t* tags;
  const int32_t* f2c;
  uint32_t mask;
  __device__ bool operator()(int f) const {
    const int t = tags[f];
    return t >= 0 && t < 7 && ((mask >> t) & 1u) && f2c[2 * (int64_t)f + 1] >= 0;
  }
};
struct IsCutPosition {  // positions in `active` of the cells tagged 2
  const int8_t* tags;
  const int32_t* active;
  __device__ bool operator()(int p) const { return tags[active[p]] == 2; }
};

// input checks: dofmap entries outside [0, n_rows), entities outside the active cells or their local facets
__global__ void k_count_dofs_out_of_range(const int32_t* __restrict__ dofmap, int64_t n, int64_t n_rows,
                                          unsigned long long* __restrict__ bad) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n && (dofmap[t] < 0 || dofmap[t] >= n_rows)) atomicAdd(bad, 1ull);
}
__global__ void k_count_bad_entities(const int32_t* __restrict__ entities, int64_t n, const int8_t* __restrict__ tags,
                                     int64_t n_cells, int n_local_facets, unsigned long long* __restrict__ bad) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int32_t c = entities[2 * t], lf = entities[2 * t + 1];
  if (c < 0 || c >= n_cells || lf < 0 || lf >= n_local_facets || (tags[c] != 1 && tags[c] != 2)) atomicAdd(bad, 1ull);
}

// keys of the active cells' dof pairs, entry-major: keys[r * n + e] = pair r = (i, j) of cell list[e], so that the slots
// k_slots writes come out as [nd*nd, n] (the layout of phifem_assemble_cells_pk)
__global__ void k_cell_pair_keys_entry_major(const int32_t* __restrict__ dofmap, int nd,
                                             const int32_t* __restrict__ list, int64_t n, int64_t n_rows,
                                             int64_t* __restrict__ keys) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * nd * nd) return;
  const int r = (int)(t / n);
  const int64_t c = list[t - r * n];
  keys[t] = (int64_t)dofmap[c * nd + r / nd] * n_rows + dofmap[c * nd + r % nd];
}

// macro dofs of an interior facet: [dofs of f2c[f][0], dofs of f2c[f][1]]
__global__ void k_macro_dofs(const int32_t* __restrict__ f2c, const int32_t* __restrict__ dofmap, int nd,
                             const int32_t* __restrict__ facets, int64_t n, int32_t* __restrict__ macro) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 2 * nd) return;
  const int64_t e = t / (2 * nd);
  const int k = (int)(t - e * 2 * nd);
  const int64_t c = f2c[2 * (int64_t)facets[e] + k / nd];
  macro[t] = dofmap[c * nd + k % nd];
}

// ordering of `_compute_integration_entities` (mesh_scripts.py:137-192): cells in first-appearance order of the
// candidate records (key = 2 facet + column), the local facets of a cell ascending
__global__ void k_entity_first_key(const int64_t* __restrict__ rec, int64_t n, unsigned long long* __restrict__ first) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) atomicMin(first + rec[3 * t + 1], (unsigned long long)rec[3 * t]);
}
__global__ void k_entity_sort_keys(const int64_t* __restrict__ rec, int64_t n,
                                   const unsigned long long* __restrict__ first, int64_t* __restrict__ skey,
                                   int64_t* __restrict__ sval) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int64_t cell = rec[3 * t + 1], lf = rec[3 * t + 2];
  skey[t] = (int64_t)first[cell] * 8 + lf;
  sval[t] = cell * 8 + lf;
}
__global__ void k_entity_unpack(const int64_t* __restrict__ sval, int64_t n, int32_t* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  out[2 * t] = (int32_t)(sval[t] >> 3);
  out[2 * t + 1] = (int32_t)(sval[t] & 7);
}

// ---- interface elasticity (phifem_elasticity_pattern_create): the vertex graph, expanded into dense NB x NB blocks

struct IsMaskedCell {  // cells whose tag t has bit t set in `mask`
  const int8_t* tags;
  uint32_t mask;
  __device__ bool operator()(int c) const {
    const int t = tags[c];
    return t >= 0 && t < 7 && ((mask >> t) & 1u);
  }
};

// input check of the one-sided entities: cell outside the mesh or not tagged in `cell_mask`, local facet out of range
__global__ void k_count_entities_outside(const int32_t* __restrict__ entities, int64_t n,
                                         const int8_t* __restrict__ tags, int64_t n_cells, int n_local_facets,
                                         uint32_t cell_mask, unsigned long long* __restrict__ bad) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int32_t c = entities[2 * t], lf = entities[2 * t + 1];
  if (c < 0 || c >= n_cells || lf < 0 || lf >= n_local_facets) atomicAdd(bad, 1ull);
  else if (tags[c] < 0 || tags[c] > 6 || !((cell_mask >> tags[c]) & 1u)) atomicAdd(bad, 1ull);
}

// position of a vertex pair = its slot minus the row's first slot = rank of the column among the row's neighbours;
// keys[e * w + i] -> pos[scatter[e] * w + i] (scatter null: pos[e * w + i])
__global__ void k_positions(const int64_t* __restrict__ uniq, int64_t nnz, const int32_t* __restrict__ vptr,
                            int64_t n_vertices, const int64_t* __restrict__ keys, int64_t n, int w,
                            const int32_t* __restrict__ scatter, int32_t* __restrict__ pos) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * w) return;
  const int64_t key = keys[t];
  const int32_t p = (int32_t)(lower_bound(uniq, nnz, key) - vptr[key / n_vertices]);
  if (scatter) {
    const int64_t e = t / w;
    pos[(int64_t)scatter[e] * w + (t - e * w)] = p;
  } else {
    pos[t] = p;
  }
}

// blocked row NB r + a starts at NB (NB vptr[r] + a deg(r)); the last entry (r = n_vertices, a = 0) is NB^2 vptr[Nv]
__global__ void k_blocked_row_pointers(const int32_t* __restrict__ vptr, int64_t n_vertices, int nb,
                                       int32_t* __restrict__ indptr) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > nb * n_vertices) return;
  const int64_t r = t / nb, a = t - r * nb;
  const int64_t deg = r < n_vertices ? vptr[r + 1] - vptr[r] : 0;
  indptr[t] = (int32_t)(nb * (nb * (int64_t)vptr[r] + a * deg));
}

// column indices of the blocked matrix: the NB rows of vertex r are NB copies of the same run of L = NB deg(r) words,
// word j = NB vcol[vptr[r] + j / NB] + j % NB, and they are contiguous from NB^2 vptr[r] on.  One warp per vertex walks
// that block of NB L words with consecutive lanes on consecutive words (the stores coalesce); j = w mod L is carried
// from one step to the next.  Bound by its stores: 4 NB^2 bytes per vertex pair, every address 64-bit.
template <int NB>
__global__ void k_expand_blocks(const int32_t* __restrict__ vptr, const int32_t* __restrict__ vcols,
                                int64_t n_vertices, int32_t* __restrict__ indices) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (r >= n_vertices) return;
  const int lane = threadIdx.x & 31;
  const int64_t beg = vptr[r];
  const int L = NB * (int)(vptr[r + 1] - beg);
  if (L == 0) return;
  const int32_t* __restrict__ cols = vcols + beg;
  int32_t* __restrict__ out = indices + NB * NB * beg;
  const int64_t total = (int64_t)NB * L;
  int j = lane;
  while (j >= L) j -= L;
  for (int64_t w = lane; w < total; w += 32) {
    const int p = j / NB;
    out[w] = NB * cols[p] + (j - p * NB);
    j += 32;
    while (j >= L) j -= L;
  }
}

struct Scratch {  // device allocations freed on scope exit (stream-ordered)
  cudaStream_t st;
  cudaMemPool_t pool;
  void* p[16];
  int n = 0;
  Scratch(cudaStream_t s, cudaMemPool_t pl) : st(s), pool(pl) {}
  void* get(size_t bytes) {
    void* q = nullptr;
    if (cudaMallocFromPoolAsync(&q, bytes ? bytes : 1, pool, st) != cudaSuccess) return nullptr;
    p[n++] = q;
    return q;
  }
  ~Scratch() {
    for (int i = 0; i < n; ++i) cudaFreeAsync(p[i], st);
  }
};

}  // namespace
}  // namespace phifem

using namespace phifem;

namespace phifem {
void plan_block_cache_release();  // csrc/rows_plan.cu: parked arrays of destroyed row-gather plans
}
extern "C" void phifem_pattern_release_scratch(void) {
  int dev = 0;
  cudaGetDevice(&dev);
  if (g_pools[dev & 63]) cudaMemPoolTrimTo(g_pools[dev & 63], 0);
  plan_block_cache_release();
}

extern "C" void phifem_pattern_destroy(phifem_pattern* p) {
  if (!p) return;
  for (int i = 0; i < p->n_owned; ++i) cudaFree(p->owned[i]);
  delete p;
}

extern "C" int phifem_pattern_view_of(const phifem_pattern* p, phifem_pattern_view* out) {
  PHIFEM_CHECK_ARG(p && out, "null pointer");
  *out = p->v;
  return PHIFEM_OK;
}

extern "C" int phifem_pattern_create_p1(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                                        const int32_t* entities, int64_t n_entities, phifem_pattern** out,
                                        void* stream) {
  PHIFEM_CHECK_ARG(out != nullptr, "out is null");
  *out = nullptr;
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->cells && mesh->c2f && mesh->f2c, "mesh / facet connectivity is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON) {
    set_error("P1 assembly supports triangles and tetrahedra, got cell type %d", mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(cell_tags8 && facet_tags8, "tag arrays are null");
  PHIFEM_CHECK_ARG(n_entities >= 0 && (n_entities == 0 || entities), "entity list");
  PHIFEM_CHECK_ARG(mesh->n_cells < (1ll << 31) && mesh->n_facets < (1ll << 31) && mesh->n_vertices < (1ll << 31),
                   "int32 index width");
  const int nv = mesh->cell_type == PHIFEM_TRIANGLE ? 3 : 4, nm = nv + 1;
  const int64_t n_rows = mesh->n_vertices;
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemPool_t pool = scratch_pool();
  if (!pool) {
    set_error("phifem_pattern_create_p1: cannot create the scratch memory pool");
    return PHIFEM_ERR_CUDA;
  }
  Scratch tmp(st, pool);
  phifem_pattern* pat = new phifem_pattern();
  pat->n_owned = 0;
  auto own = [&](size_t bytes) -> void* {
    void* q = nullptr;
    if (cudaMalloc(&q, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    pat->owned[pat->n_owned++] = q;
    return q;
  };
  auto fail = [&](const char* what) {
    set_error("phifem_pattern_create_p1: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
    phifem_pattern_destroy(pat);
    return PHIFEM_ERR_CUDA;
  };

  // 1. active cells (tags 1 / 2) and ghost-penalty facets (interior facets tagged 2 / 3), ascending
  int32_t* active_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_cells);
  int32_t* ghost_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_facets);
  int64_t* counts = (int64_t*)tmp.get(2 * sizeof(int64_t));
  if (!active_full || !ghost_full || !counts) return fail("scratch allocation");
  {
    thrust::counting_iterator<int> it(0);
    size_t b1 = 0, b2 = 0;
    cub::DeviceSelect::If(nullptr, b1, it, active_full, counts, (int)mesh->n_cells, IsActiveCell{cell_tags8}, st);
    cub::DeviceSelect::If(nullptr, b2, it, ghost_full, counts + 1, (int)mesh->n_facets,
                          IsGhostFacet{facet_tags8, mesh->f2c}, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceSelect::If(ws, b1, it, active_full, counts, (int)mesh->n_cells, IsActiveCell{cell_tags8}, st);
    cub::DeviceSelect::If(ws, b2, it, ghost_full, counts + 1, (int)mesh->n_facets,
                          IsGhostFacet{facet_tags8, mesh->f2c}, st);
  }
  int64_t h_counts[2] = {0, 0};
  if (cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("compaction");
  const int64_t na = h_counts[0], ng = h_counts[1];
  int32_t* active = (int32_t*)own(sizeof(int32_t) * na);
  int32_t* ghost = (int32_t*)own(sizeof(int32_t) * ng);
  if (!active || !ghost) return fail("output allocation");
  cudaMemcpyAsync(active, active_full, sizeof(int32_t) * na, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(ghost, ghost_full, sizeof(int32_t) * ng, cudaMemcpyDeviceToDevice, st);

  // 2. keys of every coupled pair: cells, ghost macro elements, one-sided entities (the latter lie inside active cells:
  //    they add no pattern entry but need slots)
  const int64_t kc = na * nv * nv, kg = ng * nm * nm, kb = n_entities * nv * nv;
  int64_t* keys = (int64_t*)tmp.get(sizeof(int64_t) * (kc + kg + kb));
  int32_t* macro = (int32_t*)tmp.get(sizeof(int32_t) * ng * nm);
  if (!keys || !macro) return fail("scratch allocation");
  if (kc) k_cell_pair_keys<<<blocks_for(kc), kBlockSym, 0, st>>>(mesh->cells, nv, active, 1, na, n_rows, keys);
  if (ng) {
    k_macro_vertices<<<blocks_for(ng), kBlockSym, 0, st>>>(*mesh, nv, ghost, ng, macro);
    k_pair_keys<<<blocks_for(kg), kBlockSym, 0, st>>>(macro, ng, nm, n_rows, keys + kc);
  }
  if (kb)
    k_cell_pair_keys<<<blocks_for(kb), kBlockSym, 0, st>>>(mesh->cells, nv, entities, 2, n_entities, n_rows,
                                                          keys + kc + kg);

  // 3. pattern = sorted unique keys of the cells and macro elements
  const int64_t nk = kc + kg;
  if (nk >= (1ll << 31)) {
    set_error("phifem_pattern_create_p1: %lld coupled pairs (limit 2^31): shard the mesh", (long long)nk);
    phifem_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  }
  int64_t* sorted = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  int64_t* uniq = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  int64_t* d_nnz = (int64_t*)tmp.get(sizeof(int64_t));
  if (!sorted || !uniq || !d_nnz) return fail("scratch allocation");
  int64_t nnz = 0;
  if (nk) {
    int end_bit = 1;
    while (end_bit < 63 && (1ll << end_bit) < n_rows * n_rows) ++end_bit;
    size_t b1 = 0, b2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(nullptr, b2, sorted, uniq, d_nnz, (int)nk, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceRadixSort::SortKeys(ws, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(ws, b2, sorted, uniq, d_nnz, (int)nk, st);
    if (cudaMemcpyAsync(&nnz, d_nnz, sizeof(nnz), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
      return fail("sort / unique");
  }

  // 4. CSR arrays and slot maps
  int32_t* indptr = (int32_t*)own(sizeof(int32_t) * (n_rows + 1));
  int32_t* indices = (int32_t*)own(sizeof(int32_t) * nnz);
  // three allocations: the kernels read their slot rows with vector loads (cudaMalloc alignment)
  int32_t* slots_c = (int32_t*)own(sizeof(int32_t) * kc);
  int32_t* slots_g = (int32_t*)own(sizeof(int32_t) * kg);
  int32_t* slots_b = (int32_t*)own(sizeof(int32_t) * kb);
  if (!indptr || !indices || !slots_c || !slots_g || !slots_b) return fail("output allocation");
  k_row_pointers<<<blocks_for(n_rows + 1), kBlockSym, 0, st>>>(uniq, nnz, n_rows, indptr);
  if (nnz) k_columns<<<blocks_for(nnz), kBlockSym, 0, st>>>(uniq, nnz, n_rows, indices);
  if (kc) k_slots<<<blocks_for(kc), kBlockSym, 0, st>>>(uniq, nnz, keys, kc, slots_c);
  if (kg) k_slots<<<blocks_for(kg), kBlockSym, 0, st>>>(uniq, nnz, keys + kc, kg, slots_g);
  if (kb) k_slots<<<blocks_for(kb), kBlockSym, 0, st>>>(uniq, nnz, keys + kc + kg, kb, slots_b);
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail("pattern kernels");

  pat->v.n_rows = n_rows;
  pat->v.nnz = nnz;
  pat->v.n_active = na;
  pat->v.n_ghost = ng;
  pat->v.n_entities = n_entities;
  pat->v.indptr = indptr;
  pat->v.indices = indices;
  pat->v.active = active;
  pat->v.ghost = ghost;
  pat->v.slots_cells = slots_c;
  pat->v.slots_ghost = slots_g;
  pat->v.slots_boundary = slots_b;
  *out = pat;
  return PHIFEM_OK;
}

extern "C" void phifem_pk_pattern_destroy(phifem_pk_pattern* p) {
  if (!p) return;
  for (int i = 0; i < p->n_owned; ++i) cudaFree(p->owned[i]);
  delete p;
}

extern "C" int phifem_pk_pattern_view_of(const phifem_pk_pattern* p, phifem_pk_pattern_view* out) {
  PHIFEM_CHECK_ARG(p && out, "null pointer");
  *out = p->v;
  return PHIFEM_OK;
}

// The arrays of PkAssemblyPlan (phifem_b200/assemble_pk.py), bit for bit: pattern = sorted unique keys
// row * n_rows + col of the active cells' nd x nd dof pairs and of the ghost macro elements' (2 nd) x (2 nd) pairs, slot =
// position of a key in that list (the entities' keys are looked up, they add no entry).
extern "C" int phifem_pk_pattern_create(const phifem_mesh* mesh, const int32_t* dofmap, int32_t nd, int64_t n_rows,
                                        const int8_t* cell_tags8, const int8_t* facet_tags8, uint32_t ghost_tag_mask,
                                        const int32_t* entities, int64_t n_entities, phifem_pk_pattern** out,
                                        void* stream) {
  PHIFEM_CHECK_ARG(out != nullptr, "out is null");
  *out = nullptr;
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->cells && mesh->c2f && mesh->f2c, "mesh / facet connectivity is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON &&
      mesh->cell_type != PHIFEM_QUADRILATERAL) {
    set_error("phifem_pk_pattern_create: the quadrature-kernel operators assemble on triangles, quadrilaterals and "
              "tetrahedra, got cell type %d", mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(dofmap != nullptr, "dofmap is null");
  PHIFEM_CHECK_ARG(cell_tags8 && facet_tags8, "tag arrays are null");
  PHIFEM_CHECK_ARG(nd >= 1 && nd <= 32, "nd (dofs per cell) must lie in 1..32");
  PHIFEM_CHECK_ARG(n_rows >= 1 && n_rows < (1ll << 31), "n_rows must lie in 1..2^31-1");
  PHIFEM_CHECK_ARG(n_entities >= 0 && (n_entities == 0 || entities), "entity list");
  PHIFEM_CHECK_ARG((ghost_tag_mask >> 7) == 0, "ghost_tag_mask sets bits outside the tag values 0..6");
  PHIFEM_CHECK_ARG(mesh->n_cells < (1ll << 31) && mesh->n_facets < (1ll << 31), "int32 index width");
  const int n_local_facets = mesh->cell_type == PHIFEM_TRIANGLE ? 3 : 4;
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemPool_t pool = scratch_pool();
  if (!pool) {
    set_error("phifem_pk_pattern_create: cannot create the scratch memory pool");
    return PHIFEM_ERR_CUDA;
  }
  Scratch tmp(st, pool);
  phifem_pk_pattern* pat = new phifem_pk_pattern();
  pat->n_owned = 0;
  auto own = [&](size_t bytes) -> void* {
    void* q = nullptr;
    if (cudaMalloc(&q, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    pat->owned[pat->n_owned++] = q;
    return q;
  };
  auto fail = [&](const char* what) {
    set_error("phifem_pk_pattern_create: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
    phifem_pk_pattern_destroy(pat);
    return PHIFEM_ERR_CUDA;
  };
  auto refuse = [&](const char* what) {
    set_error("phifem_pk_pattern_create: %s", what);
    phifem_pk_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  };

  // 1. active cells (tags 1 / 2) and ghost-penalty facets (interior facets whose tag is in the mask), ascending; the
  //    input checks count into the same block: {n_active, n_ghost, bad dofs, bad entities, n_cut, nnz}
  int32_t* active_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_cells);
  int32_t* ghost_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_facets);
  int64_t* counts = (int64_t*)tmp.get(6 * sizeof(int64_t));
  if (!active_full || !ghost_full || !counts) return fail("scratch allocation");
  cudaMemsetAsync(counts, 0, 6 * sizeof(int64_t), st);
  {
    thrust::counting_iterator<int> it(0);
    const IsMaskedGhostFacet is_ghost{facet_tags8, mesh->f2c, ghost_tag_mask};
    size_t b1 = 0, b2 = 0;
    cub::DeviceSelect::If(nullptr, b1, it, active_full, counts, (int)mesh->n_cells, IsActiveCell{cell_tags8}, st);
    cub::DeviceSelect::If(nullptr, b2, it, ghost_full, counts + 1, (int)mesh->n_facets, is_ghost, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceSelect::If(ws, b1, it, active_full, counts, (int)mesh->n_cells, IsActiveCell{cell_tags8}, st);
    cub::DeviceSelect::If(ws, b2, it, ghost_full, counts + 1, (int)mesh->n_facets, is_ghost, st);
  }
  unsigned long long* bad = (unsigned long long*)(counts + 2);
  if (mesh->n_cells)
    k_count_dofs_out_of_range<<<blocks_for(mesh->n_cells * nd), kBlockSym, 0, st>>>(dofmap, mesh->n_cells * nd,
                                                                                    n_rows, bad);
  if (n_entities)
    k_count_bad_entities<<<blocks_for(n_entities), kBlockSym, 0, st>>>(entities, n_entities, cell_tags8, mesh->n_cells,
                                                                       n_local_facets, bad + 1);
  int64_t h_counts[4] = {0, 0, 0, 0};
  if (cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("compaction");
  if (h_counts[2]) return refuse("dofmap has entries outside [0, n_rows)");
  if (h_counts[3])
    return refuse("entities: an entity's cell is not tagged 1 or 2, or its local facet is out of range");
  const int64_t na = h_counts[0], ng = h_counts[1];
  const int64_t kc = na * nd * nd, kg = ng * 4 * nd * nd, kb = n_entities * nd * nd, nk = kc + kg;
  if (nk >= (1ll << 31)) {
    set_error("phifem_pk_pattern_create: %lld coupled pairs (limit 2^31): shard the mesh", (long long)nk);
    phifem_pk_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  }
  int32_t* active = (int32_t*)own(sizeof(int32_t) * na);
  int32_t* ghost = (int32_t*)own(sizeof(int32_t) * ng);
  if (!active || !ghost) return fail("output allocation");
  cudaMemcpyAsync(active, active_full, sizeof(int32_t) * na, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(ghost, ghost_full, sizeof(int32_t) * ng, cudaMemcpyDeviceToDevice, st);

  // 2. cut cells: positions in `active` of the cells tagged 2 (their count comes back with nnz)
  int32_t* cut_full = (int32_t*)tmp.get(sizeof(int32_t) * na);
  if (!cut_full) return fail("scratch allocation");
  if (na) {
    thrust::counting_iterator<int> it(0);
    const IsCutPosition is_cut{cell_tags8, active};
    size_t b = 0;
    cub::DeviceSelect::If(nullptr, b, it, cut_full, counts + 4, (int)na, is_cut, st);
    void* ws = tmp.get(b);
    if (!ws) return fail("scratch allocation");
    cub::DeviceSelect::If(ws, b, it, cut_full, counts + 4, (int)na, is_cut, st);
  }

  // 3. keys: active cells (entry-major), ghost macro elements, one-sided entities (looked up only)
  int64_t* keys = (int64_t*)tmp.get(sizeof(int64_t) * (nk + kb));
  int32_t* macro = (int32_t*)tmp.get(sizeof(int32_t) * ng * 2 * nd);
  if (!keys || !macro) return fail("scratch allocation");
  if (kc) k_cell_pair_keys_entry_major<<<blocks_for(kc), kBlockSym, 0, st>>>(dofmap, nd, active, na, n_rows, keys);
  if (ng) {
    k_macro_dofs<<<blocks_for(ng * 2 * nd), kBlockSym, 0, st>>>(mesh->f2c, dofmap, nd, ghost, ng, macro);
    k_pair_keys<<<blocks_for(kg), kBlockSym, 0, st>>>(macro, ng, 2 * nd, n_rows, keys + kc);
  }
  if (kb) k_cell_pair_keys<<<blocks_for(kb), kBlockSym, 0, st>>>(dofmap, nd, entities, 2, n_entities, n_rows, keys + nk);

  // 4. pattern = sorted unique keys of the cells and macro elements
  int64_t* sorted = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  int64_t* uniq = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  if (!sorted || !uniq) return fail("scratch allocation");
  if (nk) {
    int end_bit = 1;
    while (end_bit < 63 && (1ll << end_bit) < n_rows * n_rows) ++end_bit;
    size_t b1 = 0, b2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(nullptr, b2, sorted, uniq, counts + 5, (int)nk, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceRadixSort::SortKeys(ws, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(ws, b2, sorted, uniq, counts + 5, (int)nk, st);
  }
  int64_t h_sizes[2] = {0, 0};  // n_cut, nnz
  if (cudaMemcpyAsync(h_sizes, counts + 4, sizeof(h_sizes), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("sort / unique");
  const int64_t n_cut = h_sizes[0], nnz = h_sizes[1];

  // 5. CSR arrays and slot maps
  int32_t* cut = (int32_t*)own(sizeof(int32_t) * n_cut);
  int32_t* indptr = (int32_t*)own(sizeof(int32_t) * (n_rows + 1));
  int32_t* indices = (int32_t*)own(sizeof(int32_t) * nnz);
  // three allocations: the kernels read their slot rows with vector loads (cudaMalloc alignment)
  int32_t* slots_c = (int32_t*)own(sizeof(int32_t) * kc);
  int32_t* slots_g = (int32_t*)own(sizeof(int32_t) * kg);
  int32_t* slots_b = (int32_t*)own(sizeof(int32_t) * kb);
  if (!cut || !indptr || !indices || !slots_c || !slots_g || !slots_b) return fail("output allocation");
  cudaMemcpyAsync(cut, cut_full, sizeof(int32_t) * n_cut, cudaMemcpyDeviceToDevice, st);
  k_row_pointers<<<blocks_for(n_rows + 1), kBlockSym, 0, st>>>(uniq, nnz, n_rows, indptr);
  if (nnz) k_columns<<<blocks_for(nnz), kBlockSym, 0, st>>>(uniq, nnz, n_rows, indices);
  if (kc) k_slots<<<blocks_for(kc), kBlockSym, 0, st>>>(uniq, nnz, keys, kc, slots_c);
  if (kg) k_slots<<<blocks_for(kg), kBlockSym, 0, st>>>(uniq, nnz, keys + kc, kg, slots_g);
  if (kb) k_slots<<<blocks_for(kb), kBlockSym, 0, st>>>(uniq, nnz, keys + nk, kb, slots_b);
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail("pattern kernels");

  pat->v.n_rows = n_rows;
  pat->v.nnz = nnz;
  pat->v.nd = nd;
  pat->v.n_active = na;
  pat->v.n_cut = n_cut;
  pat->v.n_ghost = ng;
  pat->v.n_entities = n_entities;
  pat->v.indptr = indptr;
  pat->v.indices = indices;
  pat->v.active = active;
  pat->v.cut_positions = cut;
  pat->v.ghost = ghost;
  pat->v.slots_cells = slots_c;
  pat->v.slots_ghost = slots_g;
  pat->v.slots_boundary = slots_b;
  *out = pat;
  return PHIFEM_OK;
}

extern "C" void phifem_elasticity_pattern_destroy(phifem_elasticity_pattern* p) {
  if (!p) return;
  for (int i = 0; i < p->n_owned; ++i) cudaFree(p->owned[i]);
  delete p;
}

extern "C" int phifem_elasticity_pattern_view_of(const phifem_elasticity_pattern* p,
                                                 phifem_elasticity_pattern_view* out) {
  PHIFEM_CHECK_ARG(p && out, "null pointer");
  *out = p->v;
  return PHIFEM_OK;
}

// The arrays of ElasticityPlan (phifem_b200/elasticity.py), bit for bit: vertex graph = sorted unique keys
// row * Nv + col of the vertex pairs of every cell tagged 1..3 and of the macro elements of the interior facets tagged
// 3 / 4, blocked CSR = that graph with dense NB x NB blocks, positions = ranks of the column vertices in their rows.
extern "C" int phifem_elasticity_pattern_create(const phifem_mesh* mesh, const int8_t* cell_tags8,
                                                const int8_t* facet_tags8, const int32_t* entities_in, int64_t n_in,
                                                const int32_t* entities_out, int64_t n_out,
                                                phifem_elasticity_pattern** out, void* stream) {
  PHIFEM_CHECK_ARG(out != nullptr, "out is null");
  *out = nullptr;
  PHIFEM_CHECK_ARG(mesh != nullptr && mesh->cells && mesh->c2f && mesh->f2c, "mesh / facet connectivity is null");
  if (mesh->cell_type != PHIFEM_TRIANGLE && mesh->cell_type != PHIFEM_TETRAHEDRON &&
      mesh->cell_type != PHIFEM_QUADRILATERAL) {
    set_error("phifem_elasticity_pattern_create: the interface-elasticity operator assembles on triangles, "
              "quadrilaterals and tetrahedra, got cell type %d", mesh->cell_type);
    return PHIFEM_ERR_UNSUPPORTED;
  }
  PHIFEM_CHECK_ARG(cell_tags8 && facet_tags8, "tag arrays are null");
  PHIFEM_CHECK_ARG(n_in >= 0 && (n_in == 0 || entities_in), "entities_in list");
  PHIFEM_CHECK_ARG(n_out >= 0 && (n_out == 0 || entities_out), "entities_out list");
  const int d = mesh->cell_type == PHIFEM_TETRAHEDRON ? 3 : 2;
  const int nv = mesh->cell_type == PHIFEM_TRIANGLE ? 3 : 4, n_local_facets = nv, nm = 2 * nv;
  const int nb = 3 * d + 2 * d * d;
  const int64_t n_vertices = mesh->n_vertices;
  PHIFEM_CHECK_ARG(mesh->n_cells < (1ll << 31) && mesh->n_facets < (1ll << 31) && n_vertices >= 0 &&
                       nb * n_vertices < (1ll << 31),
                   "int32 index width");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemPool_t pool = scratch_pool();
  if (!pool) {
    set_error("phifem_elasticity_pattern_create: cannot create the scratch memory pool");
    return PHIFEM_ERR_CUDA;
  }
  Scratch tmp(st, pool);
  phifem_elasticity_pattern* pat = new phifem_elasticity_pattern();
  pat->n_owned = 0;
  auto own = [&](size_t bytes) -> void* {
    void* q = nullptr;
    if (cudaMalloc(&q, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    pat->owned[pat->n_owned++] = q;
    return q;
  };
  auto fail = [&](const char* what) {
    set_error("phifem_elasticity_pattern_create: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
    phifem_elasticity_pattern_destroy(pat);
    return PHIFEM_ERR_CUDA;
  };
  auto refuse = [&](const char* what) {
    set_error("phifem_elasticity_pattern_create: %s", what);
    phifem_elasticity_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  };

  // 1. tagged cells (1..3), cut cells (2), interior facets tagged 3 and 4, ascending; the entity check counts into the
  //    same block: {n_tagged, n_cut, n_facets_in, n_facets_out, bad entities, n_pairs}
  const int64_t n_cells = mesh->n_cells;
  int32_t* tagged_full = (int32_t*)tmp.get(sizeof(int32_t) * n_cells);
  int32_t* cut_full = (int32_t*)tmp.get(sizeof(int32_t) * n_cells);
  int32_t* fin_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_facets);
  int32_t* fout_full = (int32_t*)tmp.get(sizeof(int32_t) * mesh->n_facets);
  int64_t* counts = (int64_t*)tmp.get(6 * sizeof(int64_t));
  if (!tagged_full || !cut_full || !fin_full || !fout_full || !counts) return fail("scratch allocation");
  cudaMemsetAsync(counts, 0, 6 * sizeof(int64_t), st);
  {
    thrust::counting_iterator<int> it(0);
    const IsMaskedCell is_tagged{cell_tags8, (1u << 1) | (1u << 2) | (1u << 3)}, is_cut{cell_tags8, 1u << 2};
    const IsMaskedGhostFacet is_in{facet_tags8, mesh->f2c, 1u << 3}, is_out{facet_tags8, mesh->f2c, 1u << 4};
    size_t b1 = 0, b2 = 0;
    cub::DeviceSelect::If(nullptr, b1, it, tagged_full, counts, (int)n_cells, is_tagged, st);
    cub::DeviceSelect::If(nullptr, b2, it, fin_full, counts + 2, (int)mesh->n_facets, is_in, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceSelect::If(ws, b1, it, tagged_full, counts, (int)n_cells, is_tagged, st);
    cub::DeviceSelect::If(ws, b1, it, cut_full, counts + 1, (int)n_cells, is_cut, st);
    cub::DeviceSelect::If(ws, b2, it, fin_full, counts + 2, (int)mesh->n_facets, is_in, st);
    cub::DeviceSelect::If(ws, b2, it, fout_full, counts + 3, (int)mesh->n_facets, is_out, st);
  }
  unsigned long long* bad = (unsigned long long*)(counts + 4);
  const uint32_t tagged_mask = (1u << 1) | (1u << 2) | (1u << 3);
  if (n_in)
    k_count_entities_outside<<<blocks_for(n_in), kBlockSym, 0, st>>>(entities_in, n_in, cell_tags8, n_cells,
                                                                     n_local_facets, tagged_mask, bad);
  if (n_out)
    k_count_entities_outside<<<blocks_for(n_out), kBlockSym, 0, st>>>(entities_out, n_out, cell_tags8, n_cells,
                                                                      n_local_facets, tagged_mask, bad);
  int64_t h_counts[5] = {0, 0, 0, 0, 0};
  if (cudaMemcpyAsync(h_counts, counts, sizeof(h_counts), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("compaction");
  if (h_counts[4])
    return refuse("entities: an entity's cell is not tagged 1, 2 or 3, or its local facet is out of range");
  const int64_t nt = h_counts[0], n_cut = h_counts[1], nfi = h_counts[2], nfo = h_counts[3];
  const int64_t kc = nt * nv * nv, kfi = nfi * nm * nm, kfo = nfo * nm * nm, nk = kc + kfi + kfo;
  const int64_t kei = n_in * nv * nv, keo = n_out * nv * nv;
  if (nk >= (1ll << 31)) {
    set_error("phifem_elasticity_pattern_create: %lld coupled vertex pairs (limit 2^31): shard the mesh", (long long)nk);
    phifem_elasticity_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  }
  int32_t* cut = (int32_t*)own(sizeof(int32_t) * n_cut);
  int32_t* fin = (int32_t*)own(sizeof(int32_t) * nfi);
  int32_t* fout = (int32_t*)own(sizeof(int32_t) * nfo);
  if (!cut || !fin || !fout) return fail("output allocation");
  cudaMemcpyAsync(cut, cut_full, sizeof(int32_t) * n_cut, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(fin, fin_full, sizeof(int32_t) * nfi, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(fout, fout_full, sizeof(int32_t) * nfo, cudaMemcpyDeviceToDevice, st);

  // 2. keys: tagged cells, the macro elements [vertices of f2c[f][0], of f2c[f][1]] of both facet lists, both entity
  //    lists (looked up only: their cells are tagged, so they add no pair)
  int64_t* keys = (int64_t*)tmp.get(sizeof(int64_t) * (nk + kei + keo));
  int32_t* macro = (int32_t*)tmp.get(sizeof(int32_t) * (nfi + nfo) * nm);
  if (!keys || !macro) return fail("scratch allocation");
  if (kc) k_cell_pair_keys<<<blocks_for(kc), kBlockSym, 0, st>>>(mesh->cells, nv, tagged_full, 1, nt, n_vertices, keys);
  if (nfi) {
    k_macro_dofs<<<blocks_for(nfi * nm), kBlockSym, 0, st>>>(mesh->f2c, mesh->cells, nv, fin, nfi, macro);
    k_pair_keys<<<blocks_for(kfi), kBlockSym, 0, st>>>(macro, nfi, nm, n_vertices, keys + kc);
  }
  if (nfo) {
    k_macro_dofs<<<blocks_for(nfo * nm), kBlockSym, 0, st>>>(mesh->f2c, mesh->cells, nv, fout, nfo, macro + nfi * nm);
    k_pair_keys<<<blocks_for(kfo), kBlockSym, 0, st>>>(macro + nfi * nm, nfo, nm, n_vertices, keys + kc + kfi);
  }
  if (kei)
    k_cell_pair_keys<<<blocks_for(kei), kBlockSym, 0, st>>>(mesh->cells, nv, entities_in, 2, n_in, n_vertices,
                                                           keys + nk);
  if (keo)
    k_cell_pair_keys<<<blocks_for(keo), kBlockSym, 0, st>>>(mesh->cells, nv, entities_out, 2, n_out, n_vertices,
                                                           keys + nk + kei);

  // 3. vertex graph = sorted unique keys of the cells and macro elements
  int64_t* sorted = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  int64_t* uniq = (int64_t*)tmp.get(sizeof(int64_t) * nk);
  if (!sorted || !uniq) return fail("scratch allocation");
  if (nk) {
    int end_bit = 1;
    while (end_bit < 63 && (1ll << end_bit) < n_vertices * n_vertices) ++end_bit;
    size_t b1 = 0, b2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(nullptr, b2, sorted, uniq, counts + 5, (int)nk, st);
    void* ws = tmp.get(b1 > b2 ? b1 : b2);
    if (!ws) return fail("scratch allocation");
    cub::DeviceRadixSort::SortKeys(ws, b1, keys, sorted, (int)nk, 0, end_bit, st);
    cub::DeviceSelect::Unique(ws, b2, sorted, uniq, counts + 5, (int)nk, st);
  }
  int64_t n_pairs = 0;
  if (cudaMemcpyAsync(&n_pairs, counts + 5, sizeof(n_pairs), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail("sort / unique");
  const int64_t nnz = (int64_t)nb * nb * n_pairs;
  if (nnz >= (1ll << 31)) {
    set_error("phifem_elasticity_pattern_create: %lld blocked entries (%d^2 x %lld vertex pairs; limit 2^31 - 1): "
              "shard the mesh", (long long)nnz, nb, (long long)n_pairs);
    phifem_elasticity_pattern_destroy(pat);
    return PHIFEM_ERR_ARGUMENT;
  }

  // 4. vertex row pointers, positions, blocked CSR
  const int64_t n_rows = nb * n_vertices;
  int32_t* vptr = (int32_t*)own(sizeof(int32_t) * (n_vertices + 1));
  int32_t* indptr = (int32_t*)own(sizeof(int32_t) * (n_rows + 1));
  int32_t* indices = (int32_t*)own(sizeof(int32_t) * nnz);
  int32_t* pos_c = (int32_t*)own(sizeof(int32_t) * n_cells * nv * nv);
  int32_t* pos_fi = (int32_t*)own(sizeof(int32_t) * kfi);
  int32_t* pos_fo = (int32_t*)own(sizeof(int32_t) * kfo);
  int32_t* pos_ei = (int32_t*)own(sizeof(int32_t) * kei);
  int32_t* pos_eo = (int32_t*)own(sizeof(int32_t) * keo);
  int32_t* vcols = (int32_t*)tmp.get(sizeof(int32_t) * n_pairs);
  if (!vptr || !indptr || !indices || !pos_c || !pos_fi || !pos_fo || !pos_ei || !pos_eo) return fail("output allocation");
  if (!vcols) return fail("scratch allocation");
  k_row_pointers<<<blocks_for(n_vertices + 1), kBlockSym, 0, st>>>(uniq, n_pairs, n_vertices, vptr);
  if (n_pairs) k_columns<<<blocks_for(n_pairs), kBlockSym, 0, st>>>(uniq, n_pairs, n_vertices, vcols);
  cudaMemsetAsync(pos_c, 0, sizeof(int32_t) * n_cells * nv * nv, st);  // cells not tagged 1..3 keep 0
  if (kc)
    k_positions<<<blocks_for(kc), kBlockSym, 0, st>>>(uniq, n_pairs, vptr, n_vertices, keys, nt, nv * nv, tagged_full,
                                                      pos_c);
  if (kfi)
    k_positions<<<blocks_for(kfi), kBlockSym, 0, st>>>(uniq, n_pairs, vptr, n_vertices, keys + kc, nfi, nm * nm,
                                                       nullptr, pos_fi);
  if (kfo)
    k_positions<<<blocks_for(kfo), kBlockSym, 0, st>>>(uniq, n_pairs, vptr, n_vertices, keys + kc + kfi, nfo, nm * nm,
                                                       nullptr, pos_fo);
  if (kei)
    k_positions<<<blocks_for(kei), kBlockSym, 0, st>>>(uniq, n_pairs, vptr, n_vertices, keys + nk, n_in, nv * nv,
                                                       nullptr, pos_ei);
  if (keo)
    k_positions<<<blocks_for(keo), kBlockSym, 0, st>>>(uniq, n_pairs, vptr, n_vertices, keys + nk + kei, n_out,
                                                       nv * nv, nullptr, pos_eo);
  k_blocked_row_pointers<<<blocks_for(n_rows + 1), kBlockSym, 0, st>>>(vptr, n_vertices, nb, indptr);
  if (nnz) {
    const unsigned grid = (unsigned)((n_vertices + kBlockSym / 32 - 1) / (kBlockSym / 32));  // one warp per vertex
    if (nb == 14) k_expand_blocks<14><<<grid, kBlockSym, 0, st>>>(vptr, vcols, n_vertices, indices);
    else k_expand_blocks<27><<<grid, kBlockSym, 0, st>>>(vptr, vcols, n_vertices, indices);
  }
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) return fail("pattern kernels");

  pat->v.n_vertices = n_vertices;
  pat->v.nb = nb;
  pat->v.n_rows = n_rows;
  pat->v.nnz = nnz;
  pat->v.n_pairs = n_pairs;
  pat->v.n_cells = n_cells;
  pat->v.n_cut = n_cut;
  pat->v.n_facets_in = nfi;
  pat->v.n_facets_out = nfo;
  pat->v.n_entities_in = n_in;
  pat->v.n_entities_out = n_out;
  pat->v.vptr = vptr;
  pat->v.indptr = indptr;
  pat->v.indices = indices;
  pat->v.cut_cells = cut;
  pat->v.facets_in = fin;
  pat->v.facets_out = fout;
  pat->v.pos_cells = pos_c;
  pat->v.pos_facets_in = pos_fi;
  pat->v.pos_facets_out = pos_fo;
  pat->v.pos_entities_in = pos_ei;
  pat->v.pos_entities_out = pos_eo;
  *out = pat;
  return PHIFEM_OK;
}

extern "C" int phifem_integration_entities_count(const phifem_mesh* mesh, const int8_t* cell_tags8,
                                                 const int8_t* facet_tags8, int32_t facet_tag, uint32_t cell_mask,
                                                 int64_t* n_entities_dev, void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr && n_entities_dev != nullptr, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(n_entities_dev, 0, sizeof(int64_t), st);
  if (mesh->n_facets == 0) return PHIFEM_OK;
  return phifem_entity_records(mesh, cell_tags8, facet_tags8, facet_tag, cell_mask, nullptr, 0, n_entities_dev, stream);
}

extern "C" int phifem_integration_entities_fill(const phifem_mesh* mesh, const int8_t* cell_tags8,
                                                const int8_t* facet_tags8, int32_t facet_tag, uint32_t cell_mask,
                                                int32_t* entities, int64_t n, void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr, "null pointer");
  PHIFEM_CHECK_ARG(n >= 0 && (n == 0 || entities), "entity buffer");
  if (n == 0 || mesh->n_facets == 0) return PHIFEM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemPool_t pool = scratch_pool();
  if (!pool) {
    set_error("phifem_integration_entities_fill: cannot create the scratch memory pool");
    return PHIFEM_ERR_CUDA;
  }
  Scratch tmp(st, pool);
  auto fail = [&](const char* what) {
    set_error("phifem_integration_entities_fill: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
    return PHIFEM_ERR_CUDA;
  };
  int64_t* d_n = (int64_t*)tmp.get(sizeof(int64_t));
  int64_t* rec = (int64_t*)tmp.get(sizeof(int64_t) * 3 * n);
  unsigned long long* first = (unsigned long long*)tmp.get(sizeof(unsigned long long) * mesh->n_cells);
  int64_t* skey = (int64_t*)tmp.get(sizeof(int64_t) * n);
  int64_t* sval = (int64_t*)tmp.get(sizeof(int64_t) * n);
  int64_t* skey2 = (int64_t*)tmp.get(sizeof(int64_t) * n);
  int64_t* sval2 = (int64_t*)tmp.get(sizeof(int64_t) * n);
  if (!d_n || !rec || !first || !skey || !sval || !skey2 || !sval2) return fail("scratch allocation");
  cudaMemsetAsync(d_n, 0, sizeof(int64_t), st);
  if (int rc = phifem_entity_records(mesh, cell_tags8, facet_tags8, facet_tag, cell_mask, rec, n, d_n, stream))
    return rc;
  cudaMemsetAsync(first, 0xff, sizeof(unsigned long long) * mesh->n_cells, st);
  k_entity_first_key<<<blocks_for(n), kBlockSym, 0, st>>>(rec, n, first);
  k_entity_sort_keys<<<blocks_for(n), kBlockSym, 0, st>>>(rec, n, first, skey, sval);
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, skey, skey2, sval, sval2, (int)n, 0, 40, st);
  void* ws = tmp.get(bytes);
  if (!ws) return fail("scratch allocation");
  cub::DeviceRadixSort::SortPairs(ws, bytes, skey, skey2, sval, sval2, (int)n, 0, 40, st);  // keys < 2^(32 + 1 + 3)
  k_entity_unpack<<<blocks_for(n), kBlockSym, 0, st>>>(sval2, n, entities);
  if (cudaGetLastError() != cudaSuccess) return fail("ordering kernels");
  return PHIFEM_OK;
}

extern "C" int phifem_integration_entities(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                                           int32_t facet_tag, uint32_t cell_mask, int32_t* entities, int64_t capacity,
                                           int64_t* n_entities, void* stream) {
  PHIFEM_CHECK_ARG(mesh != nullptr && n_entities != nullptr, "null pointer");
  PHIFEM_CHECK_ARG(capacity >= 0 && (capacity == 0 || entities), "entity buffer");
  *n_entities = 0;
  if (mesh->n_facets == 0) return PHIFEM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemPool_t pool = scratch_pool();
  if (!pool) {
    set_error("phifem_integration_entities: cannot create the scratch memory pool");
    return PHIFEM_ERR_CUDA;
  }
  int64_t n = 0;
  {
    Scratch tmp(st, pool);
    int64_t* d_n = (int64_t*)tmp.get(sizeof(int64_t));
    if (!d_n) {
      set_error("phifem_integration_entities: scratch allocation: %s", cudaGetErrorString(cudaGetLastError()));
      return PHIFEM_ERR_CUDA;
    }
    if (int rc = phifem_integration_entities_count(mesh, cell_tags8, facet_tags8, facet_tag, cell_mask, d_n, stream))
      return rc;
    if (cudaMemcpyAsync(&n, d_n, sizeof(n), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
      set_error("phifem_integration_entities: counting: %s", cudaGetErrorString(cudaGetLastError()));
      return PHIFEM_ERR_CUDA;
    }
  }
  *n_entities = n;
  if (n == 0 || n > capacity) return PHIFEM_OK;  // the caller retries with a buffer of *n_entities pairs
  if (int rc = phifem_integration_entities_fill(mesh, cell_tags8, facet_tags8, facet_tag, cell_mask, entities, n, stream))
    return rc;
  if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) {
    set_error("phifem_integration_entities: ordering kernels: %s", cudaGetErrorString(cudaGetLastError()));
    return PHIFEM_ERR_CUDA;
  }
  return PHIFEM_OK;
}
