/*
 * phifem_b200 -- C ABI of the B200-native phi-FEM hot path.
 *
 * The reference (PhiFEM/phiFEM) is pure Python on top of dolfinx; it has NO native FFI for this
 * path.  The functions below are the device-side replacements of the Python/dolfinx calls named in
 * each comment (paths relative to the reference tree).  INTEGRATION.md shows the ctypes binding a
 * maintainer would add on the reference side.
 *
 * Conventions
 *   - every `const T*` / `T*` is a DEVICE pointer unless the comment says HOST;
 *   - indices are int32, values fp64, row-major arrays;
 *   - the last argument is the CUDA stream (cudaStream_t passed as void*); calls are asynchronous;
 *   - return value: 0 on success, negative `phifem_status` otherwise; `phifem_last_error()` returns
 *     a thread-local message for the last failure on the calling thread.
 */
#ifndef PHIFEM_B200_H
#define PHIFEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PHIFEM_B200_ABI_VERSION 1

typedef enum phifem_status {
  PHIFEM_OK = 0,
  PHIFEM_ERR_ARGUMENT = -1,    /* bad argument (null pointer, unsupported size) */
  PHIFEM_ERR_CUDA = -2,        /* CUDA runtime error, see phifem_last_error() */
  PHIFEM_ERR_UNSUPPORTED = -3  /* cell type / degree outside the implemented path */
} phifem_status;

typedef enum phifem_cell_type {
  PHIFEM_TRIANGLE = 0,
  PHIFEM_QUADRILATERAL = 1,
  PHIFEM_TETRAHEDRON = 2,
  PHIFEM_HEXAHEDRON = 3        /* vertices in tensor order; tagging and the one-sided measures only */
} phifem_cell_type;

/* Mesh arrays resident in HBM (what a dolfinx `Mesh` + its topology connectivities hold;
 * src/phifem/mesh_scripts.py:151-153,308-315,419-422). */
typedef struct phifem_mesh {
  int32_t cell_type;      /* phifem_cell_type */
  int32_t gdim;           /* 2 or 3 */
  int64_t n_vertices;
  int64_t n_cells;
  int64_t n_facets;
  const double* x;        /* [n_vertices, gdim] */
  const int32_t* cells;   /* [n_cells, nvpc] cell -> vertex, dolfinx local order */
  const int32_t* c2f;     /* [n_cells, nfpc] cell -> facet (local facet i opposite vertex i) */
  const int32_t* f2c;     /* [n_facets, 2]   facet -> cells ascending, -1 pad */
  double detj_min;        /* optional bounds of |det J| over the mesh (0,0 = unknown): */
  double detj_max;        /* lets the P1 classifier skip the coordinate gather on uncut cells */
  const int32_t* boundary_facets; /* optional [n_boundary_facets]: facets with one cell, ascending; */
  int64_t n_boundary_facets;      /* lets the facet classifier run its ds detection as a second pass */
  /* optional, filled once per mesh by phifem_boundary_records (both or neither): what the ds detection of
   * mesh_scripts.py:434-452 needs of the mesh, so that the per-step pass over the mesh-boundary facets only gathers
   * the level set.  boundary_owner[i] = {owner cell of boundary_facets[i], meta}; meta = n | lf_0 << 4 | lf_1 << 6 |
   * lf_2 << 8 | lf_3 << 10 | first << 12 with n = number of mesh-boundary facets of the owner, lf_k their local
   * indices in ascending facet index, first = 1 iff boundary_facets[i] is the smallest of them;
   * boundary_scale[i][k] = integration scale (edge length / twice the triangle area) of local facet lf_k. */
  const uint32_t* boundary_owner; /* [n_boundary_facets, 2] */
  const double* boundary_scale;   /* [n_boundary_facets, 4] */
  /* optional (tetrahedra): the coordinates padded to 4 doubles per vertex, 32-byte aligned -- the row-gather cell pass
   * then fetches a vertex with one 256-bit load (one address, one sector) instead of three 64-bit ones */
  const double* x4;               /* [n_vertices, 4] = {x, y, z, 0} */
} phifem_mesh;

/* Discrete level set as seen by the detection forms (src/phifem/mesh_scripts.py:95-134).
 * mode 0: P_k coefficients + dofmap + basis tabulated at the detection points;
 * mode 1: values already evaluated at the detection points (UFL-expression mode of
 *         tests/test_compute_meshtags.py:160-161). */
typedef struct phifem_levelset {
  int32_t mode;
  int32_t n_dofs_per_cell;      /* nd (mode 0) */
  int32_t n_cell_points;        /* npts */
  int32_t n_facet_points;       /* nq */
  const double* coeffs;         /* [n_dofs]              (mode 0) */
  const int32_t* dofmap;        /* [n_cells, nd]; NULL => mesh.cells (P1)   (mode 0) */
  const double* cell_table;     /* [npts, nd] basis at the cell detection points   (mode 0) */
  const double* facet_table;    /* [nfpc, nq, nd] basis at the facet detection points (mode 0) */
  const double* cell_values;    /* [n_cells, npts]       (mode 1) */
  const double* facet_values;   /* [n_cells, nfpc, nq]   (mode 1) */
  const double* coord_grad;     /* reference gradients of the coordinate element:
                                   quadrilaterals: [npts, 4, 2] at the cell detection points (required by
                                   phifem_tag_cells);
                                   hexahedra: [npts + nfpc * nq, 8, 3] at the cell detection points, then at the
                                   facet detection points of local facets 0..5 (required by phifem_tag_cells and
                                   phifem_tag_facets*, which then also read n_cell_points); the scale of a cell point
                                   is |det J|, that of a facet point |dx/ds x dx/dt| (faces need not be planar).
                                   Hexahedral level sets: n_dofs_per_cell <= 27 (Q1 without dofmap: 8). */
} phifem_levelset;

/* Slots of the int64 counter block written by the tag kernels. */
enum {
  PHIFEM_CNT_INTERIOR = 0,     /* cells tagged 1 */
  PHIFEM_CNT_CUT = 1,          /* cells tagged 2 */
  PHIFEM_CNT_EXTERIOR = 2,     /* cells tagged 3 */
  PHIFEM_CNT_UNTAGGED = 3,     /* cells with NaN ratio */
  PHIFEM_CNT_ZERO_DEN = 4,     /* cells whose dx-denominator is ~0 (RuntimeWarning, :129-133) */
  PHIFEM_CNT_ZERO_DEN_AMBIGUOUS = 5, /* uncut cells whose ~0 test was skipped by the P1 fast path: if slot 4
                                  is 0 and this one is not, call again with bit 1 of single_layer_cut set */
  PHIFEM_CNT_FACET_ZERO_DEN = 11, /* cells whose ds-denominator is ~0 */
  PHIFEM_CNT_FACET_CONFLICT = 12, /* facets the reference algebra would emit twice */
  PHIFEM_CNT_BOUNDARY_OWNERS = 13, /* cells owning at least one mesh-boundary facet */
  PHIFEM_CNT_CALLER0 = 14,     /* slots 14, 15: never written by the tag kernels; the Python host parks the two */
  PHIFEM_CNT_CALLER1 = 15,     /* one-sided entity counts here so that ONE device -> host copy returns everything */
  PHIFEM_N_COUNTERS = 16
};

const char* phifem_last_error(void);
int phifem_abi_version(void);

/* n_words (<= 4096) 64-bit words of device memory -> page-locked host memory (cudaHostAlloc / cudaHostRegister'ed,
 * device-mapped: every such allocation is under unified addressing), written by a kernel over PCIe instead of a copy
 * engine: the counter block of phifem_tag_cells / phifem_tag_facets reaches the host without queueing behind a large
 * download issued on another stream.  Complete once an event recorded on `stream` after the call has completed.
 * Replaces the implicit device -> host reads of the reference's numpy views (src/phifem/mesh_scripts.py:129-133,
 * :360-374: warnings and debug checks on assembled arrays). */
int phifem_post_to_host(const int64_t* device_words, int64_t* pinned_host_words, int32_t n_words, void* stream);

/* Do these tags still belong to an assembly plan?  `cell_signature` = a copy of the one-byte cell tags the plan was
 * built from, `facet_signature` = the facet classes it depends on (1 = facet tag 2 or 3: ghost penalty, 2 = tag 4:
 * Gamma_h, 0 otherwise).  One pass; *mismatches (device int64, zeroed by the call) is non-zero afterwards iff a cell
 * tag or a facet class differs.  What a moving-interface loop asks after every classification before it reuses the
 * plan; the reference rebuilds its forms and matrices at every step (demo/strong-dirichlet/flower/main.py:59-66,
 * 121-123). */
int phifem_tags_match(const int8_t* cell_tags8, const int8_t* cell_signature, int64_t n_cells,
                      const int8_t* facet_tags8, const int8_t* facet_signature, int64_t n_facets,
                      int64_t* mismatches, void* stream);

/* Physical coordinates of reference points in every cell: out[n_cells, n_points, gdim].
 * `shape` [n_points, nvpc] = coordinate-element basis at the points.  Used to evaluate an
 * expression level set where the reference evaluates a UFL expression of SpatialCoordinate. */
int phifem_cell_points(const phifem_mesh* mesh, const double* shape, int32_t n_points,
                       double* out, void* stream);

/* Replaces `_compute_detection_vector` (:95-134) + `_tag_cells` (:284-390) for the `dx` detection
 * measure: cell_tags[n_cells] in {1 interior, 2 cut, 3 exterior, 0 untagged}; cell_tags8 is the
 * same as int8 (consumed by the facet / assembly kernels).  cell_tags may be NULL: only the int8 array is written then
 * (a quarter of the output bytes; widen it where an int32 `MeshTags.values` is asked for).  `counters` (int64[PHIFEM_N_COUNTERS])
 * must be zeroed by the caller; slots 0..5 are accumulated.  single_layer_cut: bit 0 applies
 * :349-358; bit 1 makes the P1 fast path evaluate every denominator exactly (see slot 5).  `vertex_scratch` (uint8[n_vertices + 3], any content) holds the per-vertex class bytes of
 * the P1 classifier (sign of phi, evaluated once per vertex) and the flags of single_layer_cut. */
int phifem_tag_cells(const phifem_mesh* mesh, const phifem_levelset* ls, int32_t single_layer_cut,
                     int32_t* cell_tags, int8_t* cell_tags8, uint8_t* vertex_scratch,
                     int64_t* counters, void* stream);

/* Replaces `_tag_facets` (:393-558) including its `ds` detection pass (:434-452):
 * facet_tags[n_facets] in 1..6 (may be NULL like cell_tags: int8 output only).  Reads counters[PHIFEM_CNT_EXTERIOR] on the device (the "no exterior
 * cell" branch :469-470), accumulates slots 11..13. */
int phifem_tag_facets(const phifem_mesh* mesh, const phifem_levelset* ls, const int8_t* cell_tags8,
                      int32_t* facet_tags, int8_t* facet_tags8, int64_t* counters, void* stream);

/* The same in two separately launchable phases, for callers that must make `counters[PHIFEM_CNT_EXTERIOR]` global
 * (an all-reduce across ranks) between the cell and facet kernels: the tags of interior facets do not depend on that
 * flag, so PHIFEM_FACETS_INTERIOR can run while the reduction is in flight and PHIFEM_FACETS_BOUNDARY (the mesh-boundary
 * facets, which do read it; needs mesh.boundary_facets) after it.  phases = both bits == phifem_tag_facets. */
enum { PHIFEM_FACETS_INTERIOR = 1, PHIFEM_FACETS_BOUNDARY = 2 };

/* Once per mesh: the static part of the ds detection on the mesh-boundary facets (mesh.boundary_owner /
 * mesh.boundary_scale, see phifem_mesh; needs mesh.boundary_facets).  The scales are computed by the same device
 * function, in the same operation order, as the pass that evaluates them on the fly: tags and counters do not depend
 * on whether the records are present. */
int phifem_boundary_records(const phifem_mesh* mesh, uint32_t* boundary_owner, double* boundary_scale, void* stream);
int phifem_tag_facets_phase(const phifem_mesh* mesh, const phifem_levelset* ls, const int8_t* cell_tags8,
                            int32_t* facet_tags, int8_t* facet_tags8, int64_t* counters, int32_t phases,
                            void* stream);

/* Candidate records of `_compute_integration_entities` (:137-192): for every facet with
 * facet_tags == facet_tag and every adjacent cell whose tag bit is set in cell_mask
 * (bit t set => cells tagged t allowed), append (key = 2*facet + column, cell, local facet) to
 * records[capacity, 3] (int64) in unspecified order; *n_records counts all candidates (may exceed
 * capacity => caller retries).  Column = position of the cell in the reversed facet->cell list. */
int phifem_entity_records(const phifem_mesh* mesh, const int8_t* cell_tags8,
                          const int8_t* facet_tags8, int32_t facet_tag, uint32_t cell_mask,
                          int64_t* records, int64_t capacity, int64_t* n_records, void* stream);

/* `_compute_integration_entities` (:137-192) complete: the flat (cell, local facet) pairs of every facet tagged
 * `facet_tag` seen from the cells whose tag bit is set in cell_mask, cells in first-appearance order, the local facets
 * of a cell ascending -- the `subdomain_data` of ds(100) (facet_tag 4, cell_mask 1<<1 | 1<<2) and ds(101) (facet_tag 3,
 * cell_mask 1<<2 | 1<<3), :617-626.  entities[capacity, 2] (device); *n_entities (HOST) = number of pairs; nothing is
 * written when it exceeds capacity (call again with a larger buffer).  Synchronises the stream. */
int phifem_integration_entities(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                                int32_t facet_tag, uint32_t cell_mask, int32_t* entities, int64_t capacity,
                                int64_t* n_entities, void* stream);

/* The two halves of phifem_integration_entities WITHOUT host synchronisation, for callers that read several counts
 * (and the tag counters) back with one device -> host copy: _count writes the number of pairs to *n_entities_dev
 * (DEVICE, int64); _fill writes exactly n pairs, n being that count as read back by the caller. */
int phifem_integration_entities_count(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                                      int32_t facet_tag, uint32_t cell_mask, int64_t* n_entities_dev, void* stream);
int phifem_integration_entities_fill(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                                     int32_t facet_tag, uint32_t cell_mask, int32_t* entities, int64_t n, void* stream);

/* ---- strong-Dirichlet phi-FEM operator, P1 on triangles / tetrahedra --------------------------
 * Forms: demo/strong-dirichlet/flower/main.py:104-128.  dof = vertex.  `data` (CSR values) and `b`
 * must be zeroed by the caller; contributions are ADDED (PETSc ADD_VALUES semantics, :121-123). */

/* (Slot maps are read with vector loads: pass 16-byte aligned arrays, e.g. separate cudaMalloc allocations.) */

/* dx((1,2)) stiffness + dx(2) stabilisation (:105,107-112) and the load vector (:126-128).
 * active[n_active] = cells tagged 1 or 2; slots[n_active, nv*nv] = CSR position of entry
 * (row = local test vertex i, col = local trial vertex j) at slots[e*nv*nv + i*nv + j]. */
int phifem_assemble_cells_p1(const phifem_mesh* mesh, const double* phi, const double* f,
                             const int8_t* cell_tags8, const int32_t* active, int64_t n_active,
                             const int32_t* slots, double sigma, double* data, double* b,
                             void* stream);

/* -int_{ds(100)} (grad(phi w).n) phi v (:106): entities[n_entities, 2] = (cell, local facet),
 * slots[n_entities, nv*nv]. */
int phifem_assemble_boundary_p1(const phifem_mesh* mesh, const double* phi, const int32_t* entities,
                                int64_t n_entities, const int32_t* slots, double* data,
                                void* stream);

/* sigma avg(h_T) jump.jump over dS((2,3)) (:113-118): facets[n_facets] interior facets tagged 2/3.
 * The 2nv macro dofs [cell+ vertices, cell- vertices] (cell+ = f2c[f][0]) hold nv+1 distinct vertices;
 * the two halves of a shared vertex are summed before the scatter, so slots[n_facets, (nv+1)^2] runs
 * over the vertex list [facet vertices in the local order of cell+, opposite vertex of cell+, opposite
 * vertex of cell-] (row-major, row = test).  Same sparsity as the (2nv)^2 macro block of dolfinx. */
int phifem_assemble_ghost_p1(const phifem_mesh* mesh, const double* phi, const int32_t* facets,
                             int64_t n_facets, const int32_t* slots, double sigma, double* data,
                             void* stream);

/* ---- owner-computes assembly (no atomics, no zero-fill, bitwise reproducible) ---------------------
 * Rows are grouped into spatially compact blocks; one CTA per block evaluates every cell / ghost facet /
 * one-sided entity touching the block's rows (an entity is listed once per block it touches: an
 * "instance"), parks each entry whose row the block owns in shared memory at a precomputed position,
 * then one thread per CSR entry (or load-vector row) sums its contiguous segment and stores it.
 * All arrays are built by the symbolic phase (phifem_b200/blocked.py). */
#define PHIFEM_BLOCK_DESC_INTS 12
typedef struct phifem_blocked_plan {
  int32_t n_blocks;
  int32_t capacity;            /* max contributions of any block = shared-memory doubles, <= 32767 */
  int32_t max_segments;        /* max padded segment count of any block (multiple of 8) */
  int32_t reserved;
  const int32_t* block_desc;   /* [n_blocks, 12]: n_contrib, seg_begin (multiple of 8), n_seg_padded
                                  (multiple of 8, > number of segments), cell_begin, cell_end,
                                  ghost_begin, ghost_end, bnd_begin, bnd_end, 0, 0, 0 */
  const int16_t* seg_start;    /* per block, at seg_begin: first buffer position of each segment
                                  (block-local), then pad entries equal to n_contrib */
  const int32_t* seg_dest;     /* same indexing: >= 0: CSR slot in `data`; < 0: row (dest & 0x7fffffff)
                                  of b; pads: 0 */
  int64_t n_cell_inst;
  const int32_t* cell_verts;   /* [n_cell_inst, 4] vertex ids (triangles: 4th unused); sign bit of the
                                  first id = cell is cut (tag 2) */
  const int16_t* cell_pos;     /* column-major words: entry e of instance i is the int16 at
                                  ((e/2) * n_cell_inst + i) * 2 + e%2; entries: nv*nv matrix (row-major,
                                  row = test) then nv load-vector entries; < 0 = row not owned */
  int64_t n_ghost_inst;
  const int32_t* ghost_facet;  /* [n_ghost_inst] facet id */
  const int16_t* ghost_pos;    /* same layout, (nv+1)^2 entries over the distinct vertices of the macro element */
  int64_t n_bnd_inst;
  const int32_t* bnd_entity;   /* [n_bnd_inst, 2] (cell, local facet) */
  const int16_t* bnd_pos;      /* same layout, nv*nv entries */
} phifem_blocked_plan;

/* Replaces phifem_assemble_{cells,boundary,ghost}_p1 in one launch; `data` and `b` need NOT be zeroed
 * (every CSR entry of the pattern and every active row of b is written exactly once; rows of b without
 * contributions are left untouched). */
int phifem_assemble_blocked_p1(const phifem_mesh* mesh, const double* phi, const double* f, double sigma,
                               const phifem_blocked_plan* plan, double* data, double* b, void* stream);

/* ---- row-gather assembly: one thread per CSR row (owner computes; no atomics, no zero-fill of `data`,
 * bitwise reproducible) ---------------------------------------------------------------------------
 * What dolfinx does as "loop over cells, MatSetValuesLocal(ADD_VALUES)" (demo/strong-dirichlet/flower/
 * main.py:121-123,130-131) is turned around: every listed row walks the cells, ghost-penalty facets and
 * one-sided entities that touch its vertex, evaluates ONLY its own row of each element tensor and keeps
 * the row's entries in shared-memory accumulators until one plain store per CSR entry.  An entity is not
 * named by its id: a record holds the positions, inside the row's own column list, of the entity's other
 * vertices (uint8 each), so the CSR pattern itself is the connectivity the kernel reads.
 * Records are stored as sliced ELLPACK over warps: slice s = listed rows [32 s, 32 s + 32), record k of
 * lane l at rec[((ptr[s] + k) * 32 + l) * words]; ptr[] counts records per lane, pads are all-ones.
 * The surface terms have their own list of rows (they touch only rows near the surface; walking them in the
 * cell pass would leave most lanes of every warp idle). */
typedef struct phifem_row_list {
  int64_t n_listed;            /* rows of this list, in processing order */
  const int32_t* rows;         /* [n_listed] row (= vertex) ids, each row at most once */
  const uint8_t* diag_pos;     /* [n_listed] position of the diagonal entry inside the row */
  const int32_t* ptr;          /* [ceil(n_listed / 32) + 1] */
  const uint32_t* rec;         /* records, see phifem_rows_plan */
} phifem_row_list;

/* Cell-once form of the cell pass (csrc/assemble_tiles.cu).  The row-gather pass evaluates a cell once per vertex
 * (the cofactors, the determinant and its reciprocal four times per tetrahedron); here a CTA owns a TILE of
 * `rows_per_tile` consecutive listed rows, evaluates every cell touching the tile ONCE (the whole element tensor),
 * parks the tensors of `rows_per_tile` cells (a CHUNK, one cell per thread) in shared memory and lets the thread of
 * each row pull its own entries -- in a fixed order, without atomics.  A cell touching several tiles is evaluated
 * once per tile (recompute factor ~1.6 for 256 spatially compact rows of a tetrahedral mesh instead of 4).
 *   slot q = chunk * rows_per_tile + lane holds one cell: slot_verts[q] = its vertex ids (cell-local order; v[0] < 0
 *   marks an empty slot, bit 31 of v[1] the cut cells; triangles leave v[3] unused).  The cells of a tile appear in
 *   ascending cell index, so every row sums its cells in mesh order whatever the tiling.
 *   Row l of the tile pulls, in chunk c, the records rec[rec_base[c] + rec_off[c][l] .. rec_base[c] + rec_off[c][l+1]):
 *   word = slot lane (bits 0-7) | cell-local index of the row's vertex (bits 8-9) | positions, inside the row's
 *   column list, of the cell's other vertices in ascending cell-local order (7 bits each from bit 10). */
typedef struct phifem_cell_tiles {
  int32_t rows_per_tile;       /* 128 or 256 (= threads per CTA = cells per chunk) */
  int32_t n_tiles;
  int64_t n_listed;            /* listed rows; tile t owns rows[t * rows_per_tile ...] */
  const int32_t* rows;         /* [n_listed] row (= vertex) ids in processing order */
  const uint8_t* diag_pos;     /* [n_listed] position of the diagonal entry inside the row */
  const int32_t* chunk_ptr;    /* [n_tiles + 1] chunks of tile t = [chunk_ptr[t], chunk_ptr[t + 1]) */
  const int32_t* slot_verts;   /* [n_chunks * rows_per_tile, 4] (16-byte aligned) */
  const int32_t* rec_base;     /* [n_chunks + 1] */
  const uint16_t* rec_off;     /* [n_chunks, rows_per_tile + 1] */
  const uint32_t* rec;         /* [rec_base[n_chunks]] */
  /* Optional [n_chunks * rows_per_tile, 4] (16-byte aligned): PUSH form of the pass.  When set, the thread that
   * evaluated the cell of slot q adds the tensor's rows to the tile's shared-memory accumulators itself (fp64
   * shared-memory atomics; rec_base / rec_off / rec are not read): push[q][i], i = cell-local vertex: bit 8 = the
   * vertex's row belongs to this tile, bits 0-7 = its index inside the tile, 7 bits from bit 10 + 7 m = position,
   * inside that row's column list, of the cell's m-th other vertex (ascending cell-local order).  The sum of a row is
   * then not in mesh order: equal to the pull form to rounding, not bit for bit. */
  const uint32_t* push;
} phifem_cell_tiles;

typedef struct phifem_rows_plan {
  const int32_t* indptr;       /* [n_rows + 1] CSR row pointers */
  const int32_t* indices;      /* [nnz] CSR column indices */
  int32_t max_row_nnz;         /* longest row (accumulators per thread), <= 255 */
  int32_t reserved;
  /* every row with pattern entries; one word per record: byte j < d = position of other vertex j of a
   * cell tagged 1/2 containing the row's vertex; bit 24: the cell is cut (tag 2).  This pass WRITES the
   * rows (data and b); rows listed here without records are written as zeros. */
  phifem_row_list cells;
  /* rows touched by the surface terms: interior facets tagged 2/3 (ghost penalty) and the one-sided entities of
   * ds(100).  A facet-once kernel first writes 8 doubles per ghost facet / entity into surface_work (jump
   * coefficients resp. normal derivatives, see csrc/assemble_rows.cu); this pass then ADDS each row's entries to the
   * rows written by the cell pass.  Two words per record:
   *   ghost facet g, macro element ghost_macro[g] = [facet vertices as ordered in cell A = f2c[f][0], opposite
   *     vertex of cell A, opposite vertex of cell B]: word 0 byte j = position of the j-th OTHER macro vertex
   *     (macro order, the row's own index skipped); word 1 = g | (macro index of the row's vertex << 28);
   *   one-sided entity e, entity_macro[e] = [facet vertices in ascending local order, opposite vertex]: the row's
   *     vertex is facet vertex t; word 0 byte 0 = position of the opposite vertex, byte j = position of facet
   *     vertex (t + j) % d; word 1 = (n_ghost_facets + e) | (t << 28) | (1 << 31). */
  phifem_row_list surface;
  int64_t n_ghost_facets;      /* n_ghost_facets + n_entities < 2^28 */
  const int32_t* ghost_macro;  /* [n_ghost_facets, d + 2] vertex ids */
  int64_t n_entities;
  const int32_t* entity_macro; /* [n_entities, d + 1] vertex ids */
  double* surface_work;        /* [n_ghost_facets + n_entities, 8] scratch (32-byte aligned), rewritten by every call */
  /* Optional cached geometry of the cell pass (NULL: the kernel gathers the coordinates and evaluates the cofactors per
   * record).  The forms see a cell only through its P1 stiffness matrix S_ab = |K| grad(lambda_a).grad(lambda_b), |K|
   * and h_T^2 -- mesh data, tabulated once per plan: 8 doubles per cell (32-byte aligned) = [S_ab for a < b in
   * lexicographic order (3 / 6 values), |K|, h_T^2, padding].  With it the records of `cells` hold TWO words: word 0 as
   * above plus (cell-local index of the row's vertex) << 25, word 1 = the cell's index in this table; the other vertices
   * of word 0 are in ascending cell-local order. */
  const double* cell_geom;
  /* Optional cell-once form of the cell pass (NULL: the row list `cells` above is walked).  When set, `cells` may be
   * empty; the rows of tiles->rows are written (data and b) exactly as the row-gather cell pass writes its rows. */
  const phifem_cell_tiles* tiles;
  /* Optional [n_ghost_facets + n_entities, 8], filled once per plan by phifem_surface_static_p1: the part of the
   * facet-once records that depends on the mesh alone -- per ghost facet s0 c_0 .. s0 c_{d+1} (jump coefficients of the
   * macro vertices, s0 = sqrt(avg(h) |F| / (d (d+1))), sigma left out), per one-sided entity cF grad(lambda_j).n for the
   * d + 1 vertices of entity_macro.  The per-step records are then LINEAR in the level set with these coefficients and a
   * light kernel builds them (no coordinate gathers); NULL: they are evaluated from the coordinates at every call. */
  double* surface_static;
} phifem_rows_plan;

/* Same operator as phifem_assemble_{cells,boundary,ghost}_p1: the facet-once kernel (forked onto an internal side
 * stream, joined before the surface pass), the cell pass and the surface pass.  `data` need NOT be zeroed (every entry of a listed row is written by the cell
 * pass); b[row] is written for listed rows only. */
int phifem_assemble_rows_p1(const phifem_mesh* mesh, const double* phi, const double* f, double sigma,
                            const phifem_rows_plan* plan, double* data, double* b, void* stream);

/* ---- strong-Dirichlet phi-FEM operator by quadrature: Lagrange P1 / P2 trial-test space (`fe_degree`,
 * demo/strong-dirichlet/flower/main.py:37) and P1 / P2 level set (`levelset_degree`, :39) on triangles and
 * tetrahedra.  Same forms and ADD semantics as the *_p1 entry points; `data` and `b` zeroed by the caller. */
typedef struct phifem_pk_space {
  int32_t degree;              /* 1 or 2 */
  int32_t n_dofs_per_cell;     /* nd: nv (P1) or nv + number of edges (P2) */
  int64_t n_dofs;
  const int32_t* dofmap;       /* [n_cells, nd], cell-local order = vertices, then edges in dolfinx local edge
                                  order (triangle (1,2),(0,2),(0,1); tetrahedron (2,3),(1,3),(1,2),(0,3),(0,2),
                                  (0,1)); NULL => mesh.cells (P1 with vertex dofs) */
} phifem_pk_space;

/* Quadrature tables (barycentric points, weights summing to 1); what dolfinx takes from basix for the
 * estimated degree of each integrand: cells 2 (kw + kphi - 1), facets 2 (kw + kphi) - 1.  At most 128 points. */
typedef struct phifem_quadrature {
  int32_t n_cell_points;
  int32_t n_facet_points;
  const double* cell_points;   /* [n_cell_points, nv] */
  const double* cell_weights;  /* [n_cell_points] */
  const double* facet_points;  /* [n_facet_points, nv - 1], facet vertices in ascending local order */
  const double* facet_weights; /* [n_facet_points] */
} phifem_quadrature;

/* Quadrilaterals (mesh->cell_type == PHIFEM_QUADRILATERAL, vertices in tensor order): the three entry points below
 * assemble the same forms with the bilinear cell map evaluated at every quadrature point (csrc/assemble_quad.cu); the
 * Hessian terms use the map's second derivative d^2 x / dxi deta.  There
 *   - space_w must be Q1 (degree 1, 4 dofs per cell): degree 2 returns PHIFEM_ERR_UNSUPPORTED;
 *   - space_phi->n_dofs_per_cell must be 4 (Q1) or 9 (Q2, with its dofmap, in the order of the Neumann entry points);
 *     any other value, or a degree that does not match, returns PHIFEM_ERR_ARGUMENT;
 *   - cell_points holds REFERENCE coordinates (xi, eta) [n_cell_points, 2] on [0,1]^2 (phifem_b200/quadrature.py
 *     rules_for_strong_quad); the facet table is the segment rule [n_facet_points, 2] = (1 - t, t);
 *   - cells must be convex (either orientation). */
/* dx((1,2)) + dx(2) terms and the load vector (:105,107-112,126-128).  slots[nd*nd, n_active]: CSR position of
 * entry (test dof i, trial dof j) of active cell e at slots[(i*nd + j) * n_active + e] (entry-major, so that
 * consecutive threads read consecutive words).  `f` lives in the trial/test space. */
int phifem_assemble_cells_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                             const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                             const double* phi, const double* f, const int8_t* cell_tags8,
                             const int32_t* active, int64_t n_active, const int32_t* slots, double sigma,
                             double* data, double* b, void* stream);

/* -int_{ds(100)} (grad(phi w).n) phi v (:106); slots[n_entities, nd*nd] (row = test dof). */
int phifem_assemble_boundary_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                const double* phi, const int32_t* entities, int64_t n_entities,
                                const int32_t* slots, double* data, void* stream);

/* Ghost penalty over dS((2,3)) (:113-118); macro dofs = [dofs of cell + (f2c[f][0]), dofs of cell -];
 * slots[n_facets, (2nd)^2] (row = test dof). */
int phifem_assemble_ghost_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                             const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                             const double* phi, const int32_t* facets, int64_t n_facets,
                             const int32_t* slots, double sigma, double* data, void* stream);

/* ---- weak-Dirichlet (dual) phi-FEM operator on the mixed space (u, p) in P_k x P_k, k = 1, 2:
 * demo/weak-dirichlet/flower/main.py:112-151 (`assemble_matrix(form(a))` :137-139, `assemble_vector(form(L))`
 * :153-154).  Cell-local mixed dof order [u dofs, p dofs] (nm = 2 nd); the global mixed numbering is the
 * caller's (`mixed_dofmap` [n_cells, nm]; phifem_b200/assemble_pk.py numbers u at scalar dof s as 2 s, p as
 * 2 s + 1).  space_w = the scalar P_k space of u, p, f and u_D; space_phi = the level-set space.  Slot maps over
 * the mixed tensors: cells entry-major [nm*nm, n_active], one-sided entities [n, nm*nm], ghost facets
 * [n, (2 nm)^2] with macro order [mixed dofs of cell +, mixed dofs of cell -].  ADD semantics; `data` / `b` zeroed by the caller. */
int phifem_assemble_weak_cells_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                  const phifem_pk_space* space_phi, const phifem_quadrature* quad,
                                  const double* phi, const double* f, const double* u_d,
                                  const int8_t* cell_tags8, const int32_t* active, int64_t n_active,
                                  const int32_t* slots, const int32_t* mixed_dofmap, double gamma,
                                  double sigma, double* data, double* b, void* stream);

/* -int_{ds(100)} (grad u.n) v (:114). */
int phifem_assemble_weak_boundary_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                     const phifem_quadrature* quad, const int32_t* entities,
                                     int64_t n_entities, const int32_t* slots, double* data, void* stream);

/* sigma avg(h_T) [grad u.n][grad v.n] over dS((2,3)) (:129-134). */
int phifem_assemble_weak_ghost_pk(const phifem_mesh* mesh, const phifem_pk_space* space_w,
                                  const phifem_quadrature* quad, const int32_t* facets, int64_t n_facets,
                                  const int32_t* slots, double sigma, double* data, void* stream);

/* ---- the step after the path (SURVEY.md 8f-3): y = A x for the CSR operator the assembly produced.  Building
 * block of the Jacobi-preconditioned BiCGStab in phifem_b200/solve.py, which stands where the reference calls
 * PETSc KSP preonly + MUMPS LU (demo/strong-dirichlet/flower/main.py:138-157). */
int phifem_csr_spmv(int64_t n_rows, const int32_t* indptr, const int32_t* indices, const double* data,
                    const double* x, double* y, void* stream);

/* The Krylov iteration itself, fused (csrc/solve.cu): Jacobi-preconditioned BiCGStab on the ACTIVE rows of an assembled
 * CSR system (rows with a usable diagonal; the others are MUMPS's null pivots, ICNTL(24), main.py:150-157).
 *   nnz           entries of the matrix (picks the lanes per row of the product); rows [n_act]  the active rows (ascending); cols [nnz] the matrix's column ids in the compact numbering, inactive
 *                 columns -> n_act; indptr / data: the matrix as assembled (read in place);
 *   vectors       length n_act (minv = 1 / diagonal, rhat = the shadow residual, x, r, p, v, s, t) and n_act + 1 with
 *                 a trailing 0 (y, z: what the products multiply);
 *   state [8]     {rho, alpha, omega, beta, r.r, rho_new, -, -}: {1, 1, 1, 0, ...} before the first call; state[4] = |r|^2
 *                 of the current iterate after every call;
 *   partials      at least 2 * 8 * 148 doubles (the products and the vector update write at most 8 * 148 pairs) and
 *                 2 * *n_partials; on entry its first *n_partials pairs hold partial sums of (rhat.r, r.r) (first
 *                 call: one pair); *n_partials (HOST) is updated for a continuation.  *n_partials below 1 or above the
 *                 product's grid + the vector grid (each at most 8 * 148 blocks) returns PHIFEM_ERR_ARGUMENT.
 * No host synchronisation; five kernels and three one-block scalar updates per iteration, bitwise reproducible. */
/* Set-up passes of the solve: diag[r] = a_rr (0 when the pattern has no diagonal entry) and rowmax[r] = max_c |a_rc| of
 * every row; cols[k] = cmap[indices[k]] (the column ids in the compact numbering of the active rows). */
int phifem_csr_row_scan(int64_t n_rows, const int32_t* indptr, const int32_t* indices, const double* data, double* diag,
                        double* rowmax, void* stream);
int phifem_remap_columns(int64_t nnz, const int32_t* indices, const int32_t* cmap, int32_t* cols, void* stream);
int phifem_csr_spmv_rows(int64_t n_act, int64_t nnz, const int32_t* rows, const int32_t* indptr, const int32_t* cols,
                         const double* data, const double* x, double* y, double* partials, void* stream);
int phifem_bicgstab_iterate(int64_t n_act, int64_t nnz, const int32_t* rows, const int32_t* indptr, const int32_t* cols,
                            const double* data, const double* minv, const double* rhat, double* x, double* r, double* p,
                            double* v, double* s, double* t, double* y, double* z, double* state, double* partials,
                            int32_t* n_partials, int32_t iterations, void* stream);

/* ---- Neumann phi-FEM operator on the mixed space (u, y, p) in P1 x P1^d x DG0: demo/neumann/square/main.py:103-158
 * (`assemble_matrix(form(a))` :141-143, `assemble_vector(form(L))` :160-161), triangles and tetrahedra, P1 or P2 level
 * set.  Cell-local mixed dof order [u at the vertices, y node-major (vertex i, component c -> nv + i d + c), p]
 * (nm = nv (1 + d) + 1); the global mixed numbering is the caller's (`mixed_dofmap` [n_cells, nm];
 * phifem_b200/assemble_pk.py numbers u at vertex s as (d+1) s, y_c as (d+1) s + 1 + c, p of cell k as (d+1) Nv + k).
 * `f` and `u_n` are P1 (vertex values).  robin_coef != 0 turns the penalty combination into
 * y.grad phi - |grad phi| robin_coef u + h^-1 p phi: the Robin operator of demo/robin/square/main.py:118-174 (u_n = the
 * Robin data; its ghost penalty runs over dS(2): pass those facets to phifem_assemble_neumann_ghost).  Slot maps: cells entry-major [nm*nm, n_active], one-sided entities
 * [n, nm*nm], interior facets tagged 3 [n, (2 nm)^2] (macro order [mixed dofs of cell +, of cell -]).  ADD semantics.
 *
 * Quadrilaterals (mesh->cell_type == PHIFEM_QUADRILATERAL, vertices in tensor order, the demo's own mesh): the mixed
 * space is Q1 x Q1^2 x DG0 (nm = 13: [u x4, y node-major x8, p]) and the bilinear cell map is evaluated at every
 * quadrature point (csrc/assemble_quad.cu).  There
 *   - phifem_quadrature.cell_points holds REFERENCE coordinates (xi, eta) [n_cell_points, 2] on [0,1]^2, weights summing
 *     to 1 (phifem_b200/quadrature.py rules_for_neumann_quad); the facet table stays the segment rule
 *     [n_facet_points, 2] = (1 - t, t), t running from the edge's lower-global-id vertex to the higher one;
 *   - space_phi->n_dofs_per_cell must be 4 (Q1, degree 1, dofmap may be NULL) or 9 (Q2, degree 2, dolfinx-local order:
 *     vertices, the edges (0,1),(0,2),(1,3),(2,3), interior); any other value returns PHIFEM_ERR_ARGUMENT;
 *   - every interior cell is integrated by the cell rule too (no closed form on a non-affine cell);
 *   - cells must be convex (either orientation); a non-convex quadrilateral is outside the method and not checked. */
/* `cut_positions` [n_cut]: positions in `active` of the cells tagged 2 (every term of the form, by quadrature); the
 * other active cells carry the P1 stiffness + mass block of u only (closed form, a separate light kernel). */
int phifem_assemble_neumann_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi,
                                  const phifem_quadrature* quad, const double* phi, const double* f,
                                  const double* u_n, const int8_t* cell_tags8, const int32_t* active,
                                  int64_t n_active, const int32_t* cut_positions, int64_t n_cut, const int32_t* slots,
                                  const int32_t* mixed_dofmap, double gamma, double robin_coef, double* data,
                                  double* b, void* stream);

/* int_{ds(100)} (y.n) v (:120). */
int phifem_assemble_neumann_boundary(const phifem_mesh* mesh, const int32_t* entities, int64_t n_entities,
                                     const int32_t* slots, double* data, void* stream);

/* sigma avg(h_T) [grad u.n][grad v.n] over dS(3) (:136-139). */
int phifem_assemble_neumann_ghost(const phifem_mesh* mesh, const phifem_quadrature* quad, const int32_t* facets,
                                  int64_t n_facets, const int32_t* slots, double sigma, double* data, void* stream);

/* ---- interface-elasticity phi-FEM operator on the mixed space (u_in, u_out, y_in, y_out, p) in
 * P1^d x P1^d x P1^(d x d) x P1^(d x d) x P1^d: demo/interface-elasticity/main.py:152-274 (`assemble_matrix(form(a), bcs)`
 * :238-240, `assemble_vector(form(L))` :271, `apply_lifting` / `bc.set` :273-275), triangles, quadrilaterals and
 * tetrahedra, P1 (Q1) or P2 (Q2) level set.  Every field is nodal, so the mixed space has NB = 3 d + 2 d^2 dofs per vertex: global dof = NB vertex + o,
 * o: u_in c -> c, u_out c -> d + c, y_in (r,s) -> 2d + r d + s, y_out (r,s) -> 2d + d^2 + r d + s, p c -> 2d + 2d^2 + c.
 * The CSR matrix is the vertex graph (`vptr` [n_vertices + 1], sorted neighbour lists: vertex pairs of every tagged cell
 * and of the macro elements of the interior facets tagged 3 / 4) with dense NB x NB blocks: entry (NB r + a, NB s + b)
 * at NB (NB vptr[r] + a deg(r) + pos) + b, pos = rank of s among r's neighbours.  Slot maps hold `pos` per vertex pair:
 * cells [n_cells, nv*nv], facets [n, (2 nv)^2] (macro order [vertices of cell +, of cell -]), entities [n, nv*nv]
 * (row = test vertex).  `f` is a P1 vector field [n_vertices, d].  ADD semantics; `data` / `b` zeroed by the caller.
 *
 * Quadrilaterals (mesh->cell_type == PHIFEM_QUADRILATERAL, gdim 2, vertices in tensor order): every field is Q1 on the
 * bilinear cell (NB = 14, nv = 4 in the slot maps) and `f` is Q1 (vertex values).  There
 *   - phifem_quadrature.cell_points holds REFERENCE coordinates (xi, eta) [n_cell_points, 2] on [0,1]^2, weights summing
 *     to 1: the rule of the cut cells (phifem_b200/quadrature.py rules_for_elasticity_quad, (kphi + 2)^2 Gauss points);
 *   - the cells tagged 1 / 3 are integrated by a fixed 2 x 2 Gauss rule, the stress jump by a fixed 2-point Gauss rule on
 *     the edge (compile-time constants, exact on parallelograms), the one-sided terms in closed form;
 *   - space_phi->n_dofs_per_cell must be 4 (Q1, degree 1) or 9 (Q2, degree 2, dolfinx-local order); any other value
 *     returns PHIFEM_ERR_ARGUMENT;
 *   - cells must be convex (either orientation); a non-convex quadrilateral is outside the method and not checked. */
typedef struct phifem_elasticity_params {
  double lmbda_in, mu_in;    /* Lame coefficients of data.py:5-22 */
  double lmbda_out, mu_out;
  double coef_in, coef_out;  /* (E_in / (E_in + E_out))^2, (E_out / (E_in + E_out))^2 (main.py:189-190) */
  double gamma;              /* penalization_coefficient */
  double sigma_s;            /* stabilization_coefficient */
} phifem_elasticity_params;

/* All cell integrals of `a` and `L` (dx((1,2)), dx((2,3)), dx(2)).  Cells tagged 1 / 3 (one closed-form stiffness block
 * each) are found through cell_tags8, cells with another tag skipped; `cut_cells` [n_cut] lists the cells tagged 2, which
 * carry every term of the form and are integrated by quadrature. */
int phifem_assemble_elasticity_cells(const phifem_mesh* mesh, const phifem_pk_space* space_phi,
                                     const phifem_quadrature* quad, const double* phi, const double* f,
                                     const int8_t* cell_tags8, const int32_t* cut_cells, int64_t n_cut,
                                     const int32_t* vptr, const int32_t* pos_cells,
                                     const phifem_elasticity_params* prm, double* data, double* b, void* stream);

/* sigma_s avg(h_T) [sigma(u) n].[sigma(v) n] over the given interior facets: side 0 = sigma_in / u_in over dS(3)
 * (:207-211), side 1 = sigma_out / u_out over dS(4) (:221-225). */
int phifem_assemble_elasticity_facets(const phifem_mesh* mesh, const int32_t* facets, int64_t n_facets,
                                      const int32_t* vptr, const int32_t* pos_facets, int32_t side,
                                      const phifem_elasticity_params* prm, double* data, void* stream);

/* int (y n).v over one-sided entities [cell, local facet]: side 0 = (y_in, v_in) over ds(100), side 1 = (y_out, v_out)
 * over ds(101) (:183-184, 235-236). */
int phifem_assemble_elasticity_boundary(const phifem_mesh* mesh, const int32_t* entities, int64_t n_entities,
                                        const int32_t* vptr, const int32_t* pos_boundary, int32_t side, double* data,
                                        void* stream);

/* Dirichlet conditions on an assembled CSR system (dolfinx `assemble_matrix(a, bcs)` + `apply_lifting` + `bc.set`,
 * main.py:238, 273-275): rows and columns of the marked dofs are zeroed (entries stay in the pattern), their diagonal
 * is 1, b <- b - A g on the free rows, b = g on the marked ones.  bc_marker int8 [n_rows], bc_values [n_rows]. */
int phifem_apply_dirichlet(int64_t n_rows, const int32_t* indptr, const int32_t* indices, const int8_t* bc_marker,
                           const double* bc_values, double* data, double* b, void* stream);
/* The same for a structurally symmetric pattern (one space for trial and test functions: every operator here), driven
 * by the list bc_dofs[n_bc] of the marked dofs: the mirrored entry (j, c) of every entry (c, j) of a marked row is found by
 * binary search, so the work is the marked rows' lengths instead of a pass over the matrix.  The lifting adds into b
 * with fp64 reductions (order not fixed).
 * PRECONDITIONS the call does not check: column indices sorted inside every row (the bisection), a structurally
 * symmetric pattern (entry (j, c) exists whenever (c, j) does), and bc_dofs free of duplicates (two warps on the same
 * row would lift twice; the Python wrapper passes torch.unique(bc_dofs)).  Opt-in: parity-tested on small systems only. */
int phifem_apply_dirichlet_symmetric(int64_t n_rows, const int32_t* indptr, const int32_t* indices,
                                     const int32_t* bc_dofs, int64_t n_bc, const int8_t* bc_marker,
                                     const double* bc_values, double* data, double* b, void* stream);

/* ---- symbolic phase of the P1 strong-Dirichlet operator on the device: what dolfinx does in `create_sparsity_pattern` /
 * `create_matrix` under `assemble_matrix(form(a))` (demo/strong-dirichlet/flower/main.py:121-123).  For hosts without
 * Python: tags (phifem_tag_cells / phifem_tag_facets) -> phifem_pattern_create_p1 -> phifem_assemble_{cells,boundary,
 * ghost}_p1 run the whole path with this library alone (the Python package builds the same arrays with torch sort /
 * unique and adds the row-gather plan on top).  The pattern object owns its device arrays (cudaMalloc); the call
 * synchronises the stream twice (two sizes come back to the host). */
typedef struct phifem_pattern phifem_pattern;
typedef struct phifem_pattern_view {
  int64_t n_rows, nnz;           /* rows = vertices; nnz < 2^31 */
  int64_t n_active, n_ghost, n_entities;
  const int32_t* indptr;         /* [n_rows + 1] */
  const int32_t* indices;        /* [nnz] sorted per row; structural zeros kept, rows without contributions empty */
  const int32_t* active;         /* [n_active] cells tagged 1 / 2, ascending */
  const int32_t* ghost;          /* [n_ghost] interior facets tagged 2 / 3, ascending */
  const int32_t* slots_cells;    /* [n_active, nv*nv]      as phifem_assemble_cells_p1 expects */
  const int32_t* slots_ghost;    /* [n_ghost, (nv+1)^2]    as phifem_assemble_ghost_p1 expects */
  const int32_t* slots_boundary; /* [n_entities, nv*nv]    as phifem_assemble_boundary_p1 expects */
} phifem_pattern_view;

/* entities[n_entities, 2] = the (cell, local facet) pairs of ds(100) (may be empty). */
int phifem_pattern_create_p1(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                             const int32_t* entities, int64_t n_entities, phifem_pattern** out, void* stream);
int phifem_pattern_view_of(const phifem_pattern* pattern, phifem_pattern_view* out);
void phifem_pattern_destroy(phifem_pattern* pattern);
/* The sort scratch of phifem_pattern_create_p1 (about 200 bytes per active cell) lives in a private stream-ordered memory
 * pool that stays cached between calls; this returns it to the driver. */
void phifem_pattern_release_scratch(void);

/* ---- the row-gather plan itself, built on the device (csrc/rows_plan.cu): CSR pattern (indptr, indices), active cells,
 * ghost facets and the two row lists of phifem_rows_plan, from the vertex -> cell adjacency (one radix sort of
 * n_active * nv keys, per-row merges) instead of one key per coupled vertex pair.  Every array equals what
 * phifem_b200/assemble.py + rows.py build with torch ops, bit for bit.  The handle owns its device arrays (cudaMalloc);
 * the call synchronises the stream a few times (sizes come back to the host).
 *   row_mask      optional [n_vertices] bytes: list only these rows (the rows a rank owns); NULL = every row;
 *   morton_cells  != 0: the rows of the cell pass are listed along the Morton curve of their vertices instead of
 *                 ascending (the surface rows always are, then balanced by record count in chunks of 4096). */
typedef struct phifem_rows_plan_handle phifem_rows_plan_handle;
typedef struct phifem_rows_plan_info {
  int64_t n_rows, nnz;
  int64_t n_active, n_ghost, n_entities;
  const int32_t* active;            /* [n_active] cells tagged 1 / 2, ascending */
  const int32_t* ghost;             /* [n_ghost] interior facets tagged 2 / 3, ascending */
  int64_t n_cell_records;           /* n_active * nv (records of unlisted rows included) */
  int64_t n_surface_records;        /* records of the surface list */
  int64_t cells_record_slots;       /* words of plan.cells.rec (pads included) */
  int64_t surface_record_slots;     /* uint2 slots of plan.surface.rec (pads included) */
} phifem_rows_plan_info;

/* Once per plan (after its ghost_macro / entity_macro lists exist): fills plan->surface_static. */
int phifem_surface_static_p1(const phifem_mesh* mesh, const phifem_rows_plan* plan, void* stream);

int phifem_rows_plan_create(const phifem_mesh* mesh, const int8_t* cell_tags8, const int8_t* facet_tags8,
                            const int32_t* entities, int64_t n_entities, const uint8_t* row_mask, int32_t morton_cells,
                            phifem_rows_plan_handle** out, void* stream);
/* plan: ready for phifem_assemble_rows_p1 (its pointers stay valid until the handle is destroyed). */
int phifem_rows_plan_view(const phifem_rows_plan_handle* handle, phifem_rows_plan* plan, phifem_rows_plan_info* info);
void phifem_rows_plan_destroy(phifem_rows_plan_handle* handle);

/* ---- the exchange step of a sharded classification over NVLink peer memory (csrc/peer.cu).  `_tag_facets` needs
 * "is there any exterior cell" GLOBALLY (reference src/phifem/mesh_scripts.py:469-474): every rank publishes its count of
 * tag-3 cells after phifem_tag_cells by storing (epoch, count) into a slot of every peer's memory (CUDA IPC mapping, one
 * 8-byte store per peer), runs phifem_tag_facets_phase(PHIFEM_FACETS_INTERIOR), then collects the sum from the slots in
 * its own memory and runs the PHIFEM_FACETS_BOUNDARY phase.  One process per GPU on one node, world <= 64.
 *   create   allocates the rank's slots and returns their 64-byte IPC handle;
 *   connect  takes the handles of ALL ranks ([world][64] bytes, gathered by the host code, e.g. MPI_Allgather) and maps them;
 *   publish  value: device pointer to the rank's count; every call starts a new epoch (kept in device memory: the two
 *            calls can be captured in a CUDA graph and replayed);
 *   collect  value_out (device) = sum over ranks of the counts of the current epoch (each clamped to 2^32 - 1); waits
 *            for peers that are late, gives up after ~1 s (phifem_peer_flags_error then returns 1). */
typedef struct phifem_peer_flags phifem_peer_flags;
int phifem_peer_flags_create(int32_t world, int32_t rank, phifem_peer_flags** out, void* handle64);
int phifem_peer_flags_connect(phifem_peer_flags* flags, const void* handles);
int phifem_peer_flags_publish(phifem_peer_flags* flags, const int64_t* value, void* stream);
int phifem_peer_flags_collect(phifem_peer_flags* flags, int64_t* value_out, void* stream);
int phifem_peer_flags_error(phifem_peer_flags* flags);
void phifem_peer_flags_destroy(phifem_peer_flags* flags);

/* ---- halo exchange of CSR / load-vector contributions over NVLink peer memory (csrc/peer.cu): SURVEY.md 8(b) export (5).
 * The reference's only parallel hook is the MPI communicator of its mesh (demo/strong-dirichlet/flower/main.py:49): PETSc
 * adds off-process contributions to their owner's rows inside `assemble_matrix` / `assemble_vector` + ghost updates
 * (main.py:121-131).  Here a rank that assembled contributions to rows owned by a peer pushes them into that peer's
 * receive buffer (CUDA IPC mapping, remote stores), publishes an epoch flag, waits for the flags of its own peers and
 * adds what it received into `dst` through a slot list -- ONE kernel, no pack, no collective library, CUDA-graph
 * capturable.  One process per GPU on one node.
 *   create   allocates the receive buffer ([2][capacity] doubles, capacity the same on every rank) and returns its
 *            64-byte CUDA IPC handle in handle64 (HOST);
 *   connect  handles (HOST) = the world handles in rank order; remote_offset[q] (HOST) = where this rank's values start
 *            inside peer q's receive buffer; send_ptr[world + 1] (HOST) = value range of peer q in this rank's send
 *            list; send_src[q] (HOST) = first element of peer q's CONTIGUOUS segment of `src` (used when the exchange is
 *            called without a send_index); n_recv = values this rank receives per exchange;
 *   exchange value j of peer q = src[send_index[send_ptr[q] + j]] (send_index DEVICE, may be NULL: src[send_src[q] + j]);
 *            on arrival dst[recv_index[i]] += received[i] (recv_index DEVICE [n_recv], fp64 reductions);
 *   error    synchronises; 1 = a receive waited ~1 s for a peer that never pushed. */
typedef struct phifem_halo phifem_halo;
int phifem_halo_create(int32_t world, int32_t rank, int64_t capacity, phifem_halo** out, void* handle64);
int phifem_halo_connect(phifem_halo* halo, const void* handles, const int64_t* remote_offset, const int64_t* send_ptr,
                        const int64_t* send_src, int64_t n_recv);
int phifem_halo_exchange(phifem_halo* halo, const double* src, const int64_t* send_index, const int64_t* recv_index,
                         double* dst, void* stream);
int phifem_halo_error(phifem_halo* halo);
void phifem_halo_destroy(phifem_halo* halo);

#ifdef __cplusplus
}
#endif
#endif /* PHIFEM_B200_H */
