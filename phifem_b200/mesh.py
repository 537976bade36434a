"""Mesh, topology and mesh tags: the data model of the hot path.

Stand-ins for the dolfinx objects the reference API exchanges (`dolfinx.mesh.Mesh`,
`MeshTags`, `AdjacencyList_int32`; reference src/phifem/mesh_scripts.py:12-15,151-153,386).
A `Mesh` owns its arrays on ONE device (HBM-resident for the whole life of the mesh, like a
dolfinx mesh lives in host memory); host copies are made lazily and only for the
duck-typed dolfinx-style accessors.

Layout in HBM (row-major, int32 indices, fp64 coordinates):
    x      [Nv, gdim]   vertex coordinates
    cells  [Nc, nvpc]   cell -> vertex (dolfinx local order)
    c2f    [Nc, nfpc]   cell -> facet, local facet i opposite local vertex i on simplices, _geometry.LOCAL_FACETS order
    f2c    [Nf, 2]      facet -> cells ascending, -1 pad on the mesh boundary
    fverts [Nf, nvpf]   facet -> sorted vertex tuple

Facet numbering = lexicographic rank of the sorted vertex tuple (what dolfinx 0.9 produces in
serial [probed on the reference's golden tag files, SURVEY.md C.2]).  The topology builder
is sort/unique plumbing written with torch ops so it runs where the mesh lives.
"""
import numpy as np
import torch

from . import _geometry as G


def default_device():
    return torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() \
        else torch.device("cpu")


class AdjacencyList:
    """Minimal `dolfinx.graph.AdjacencyList_int32` look-alike (host arrays)."""

    def __init__(self, array, offsets):
        self.array = np.ascontiguousarray(array, dtype=np.int32)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int32)

    def links(self, i):
        return self.array[self.offsets[i]:self.offsets[i + 1]]

    @property
    def num_nodes(self):
        return len(self.offsets) - 1


class _CellType:
    def __init__(self, name):
        self.name = name


class Topology:
    def __init__(self, mesh):
        self._mesh = mesh
        self.dim = G.TDIM[mesh.cell_type]
        self.cell_type = _CellType(mesh.cell_type)
        self._conn = {}

    def cell_name(self):
        return self._mesh.cell_type

    def create_connectivity(self, d0, d1):
        if (d0, d1) in self._conn:
            return
        m, tdim = self._mesh, self.dim
        if (d0, d1) == (tdim, 0):
            c = m.cells_host
            adj = AdjacencyList(c.ravel(), np.arange(0, c.size + 1, c.shape[1]))
        elif (d0, d1) == (tdim, tdim - 1):
            c2f = m.c2f.cpu().numpy()
            adj = AdjacencyList(c2f.ravel(), np.arange(0, c2f.size + 1, c2f.shape[1]))
        elif (d0, d1) == (tdim - 1, tdim):
            f2c = m.f2c.cpu().numpy()
            cnt = (f2c >= 0).sum(axis=1)
            adj = AdjacencyList(f2c[f2c >= 0], np.r_[0, np.cumsum(cnt)])
        elif (d0, d1) == (tdim - 1, 0):
            fv = m.facet_vertices.cpu().numpy()
            adj = AdjacencyList(fv.ravel(), np.arange(0, fv.size + 1, fv.shape[1]))
        elif (d0, d1) == (0, tdim):
            c = m.cells_host
            order = np.argsort(c.ravel(), kind="stable")
            cnt = np.bincount(c.ravel(), minlength=m.num_vertices)
            adj = AdjacencyList((order // c.shape[1]), np.r_[0, np.cumsum(cnt)])
        else:
            raise NotImplementedError("connectivity (%d, %d)" % (d0, d1))
        self._conn[(d0, d1)] = adj

    def connectivity(self, d0, d1):
        return self._conn.get((d0, d1))


class _Geometry:
    def __init__(self, mesh):
        self._mesh = mesh

    @property
    def x(self):
        x = self._mesh.x_host
        out = np.zeros((len(x), 3))
        out[:, :x.shape[1]] = x
        return out


def morton_keys(pts, bits=21):
    """Morton (Z-order) key of each point: coordinates quantised to `bits` bits per axis over the bounding box, bits
    interleaved (axis 0 least significant)."""
    d = pts.shape[1]
    bits = min(bits, 63 // d)
    lo, hi = pts.min(dim=0).values, pts.max(dim=0).values
    q = ((pts - lo) / (hi - lo).clamp(min=1e-300) * (2 ** bits - 1)).long().clamp_(0, 2 ** bits - 1)
    key = torch.zeros(pts.shape[0], dtype=torch.int64, device=pts.device)
    for bit in range(bits):
        for k in range(d):
            key |= ((q[:, k] >> bit) & 1) << (bit * d + k)
    return key


class Mesh:
    """Unstructured mesh of triangles, quadrilaterals, tetrahedra or hexahedra on one device (quadrilaterals and
    hexahedra with their vertices in tensor order)."""

    def __init__(self, x, cells, cell_type, device=None):
        if cell_type not in G.CELL_TYPES:
            raise NotImplementedError("unsupported cell type '%s'" % cell_type)
        self.cell_type = cell_type
        self.device = torch.device(device) if device is not None else default_device()
        self.x = torch.as_tensor(x, dtype=torch.float64).to(self.device).contiguous()
        self.cells = torch.as_tensor(cells).to(torch.int32).to(self.device).contiguous()
        if self.cells.ndim != 2 or self.cells.shape[1] != G.NVPC[cell_type]:
            raise ValueError("cells must have shape [Nc, %d]" % G.NVPC[cell_type])
        self.gdim = int(self.x.shape[1])
        self.num_vertices = int(self.x.shape[0])
        self.num_cells = int(self.cells.shape[0])
        self._topo = None
        self._host = {}
        self.sfc_ordered = False            # numbered along a space-filling curve (see `reordered`)
        self.original_cell_index = None
        self.input_global_indices = None
        self.topology = Topology(self)
        self.geometry = _Geometry(self)

    @staticmethod
    def from_xdmf(x, cells_file_order, cell_type, device=None):
        """XDMF stores quadrilaterals cyclically; dolfinx uses tensor order [a,b,d,c]
        [probed, SURVEY.md A.1]."""
        cells = np.asarray(cells_file_order)
        if cell_type == "quadrilateral":
            cells = cells[:, [0, 1, 3, 2]]
        return Mesh(x, cells, cell_type, device)

    def structured_fraction(self):
        """Share of the vertices that have the most common number of cells around them, relative to the interior share of
        a grid with as many vertices: ~1 for a mesh with the connectivity of a tensor grid (whatever its numbering and
        however its vertices were moved), ~0.1 for a Delaunay mesh.  Decides the renumbering of `reordered(curve="auto")`."""
        val = torch.bincount(self.cells.reshape(-1).long(), minlength=self.num_vertices)
        modal = float(torch.bincount(val).max()) / max(1, self.num_vertices)
        # the vertices on the boundary of a grid have fewer cells: compare with the interior share of an m^d grid
        m = max(3.0, self.num_vertices ** (1.0 / self.gdim))
        return min(1.0, modal / ((m - 2.0) / m) ** self.gdim)

    def reordered(self, curve="auto"):
        """The same mesh renumbered for data locality: curve="morton": vertices by the Morton key of their coordinates,
        cells by the Morton key of their centroid; curve="pencil": count-balanced slabs / pencils / lines (see
        `_reordered_pencils`); curve="auto" (default): pencils for a mesh with grid connectivity (`structured_fraction`
        >= 0.8), the Morton curve otherwise -- measured on the B200 (DESIGN.md section 5): scrambled grid of config E 1.86 ms
        per step in pencils against 2.16 ms along the Morton curve, Delaunay mesh of a random point cloud 0.242 ms against
        0.219 ms for the cell pass.  The cell-local vertex order is kept, so local facets and orientations are
        unchanged.  This is the data-locality reordering dolfinx applies when it builds a mesh (`create_mesh` reorders
        cells and vertices and keeps `topology.original_cell_index` / `geometry.input_global_indices` [dep-knowledge]);
        like there, everything downstream -- facet numbering, tags, dofs, CSR rows -- lives in the NEW numbering and the
        two maps translate user data:
            new.original_cell_index[c_new] = c_old        new.input_global_indices[v_new] = v_old
        so per-vertex data of the old mesh becomes `data[new.input_global_indices]`."""
        if curve not in ("auto", "morton", "pencil"):
            raise ValueError("curve must be 'auto', 'morton' or 'pencil'")
        if curve == "auto":
            curve = "pencil" if self.structured_fraction() >= 0.8 else "morton"
        if curve == "pencil":
            return self._reordered_pencils()
        vperm = torch.argsort(morton_keys(self.x), stable=True)                 # new -> old
        vinv = torch.empty_like(vperm)
        vinv[vperm] = torch.arange(self.num_vertices, device=self.device)
        step = 1 << 24
        ckey = torch.empty(self.num_cells, dtype=torch.int64, device=self.device)
        lo, hi = self.x.min(dim=0).values, self.x.max(dim=0).values
        box = torch.stack([lo, hi])
        for s0 in range(0, self.num_cells, step):
            cen = self.x[self.cells[s0:s0 + step].long()].mean(dim=1)
            ckey[s0:s0 + step] = morton_keys(torch.cat([box, cen]))[2:]         # same bounding box for every slab
        cperm = torch.argsort(ckey, stable=True)
        del ckey
        new = Mesh(self.x[vperm], vinv[self.cells[cperm].long()].to(torch.int32), self.cell_type, self.device)
        new.sfc_ordered = True
        new.reorder_curve = "morton"
        new.original_cell_index = cperm
        new.input_global_indices = vperm
        return new

    def _reordered_pencils(self):
        """curve="pencil": vertices in slabs of equal COUNT along axis 0, each slab in pencils of equal count along axis
        1 (3D), each pencil sorted along the last axis; cells by their lowest new vertex.  Parameter-free (no mesh size
        enters) and, on a mesh whose vertices sit near the points of a tensor grid (the jittered variant of SURVEY.md
        8d: jitter below half a spacing), exactly the lexicographic numbering of that grid -- the numbering under which
        the rows of a warp of the row-gather kernels are neighbours along a line and their gathers coalesce (cell pass at
        config E: 1.20 ms lexicographic, 1.55 ms Morton)."""
        nv, d, dev = self.num_vertices, self.gdim, self.device
        m = max(1, round(nv ** (1.0 / d)))
        per = [m ** (d - 1 - k) if m ** d == nv else int(-(-nv ** ((d - 1 - k) / d) // 1)) for k in range(d - 1)]
        group = torch.zeros(nv, dtype=torch.int64, device=dev)     # slab, then (slab, pencil) index of each vertex
        for k in range(d - 1):
            rank = torch.empty(nv, dtype=torch.int64, device=dev)
            rank[torch.argsort(self.x[:, k], stable=True)] = torch.arange(nv, device=dev)
            order = torch.argsort(group * nv + rank)                # vertices grouped, sorted along axis k inside
            start = torch.zeros(int(group.max()) + 2, dtype=torch.int64, device=dev)
            start[1:] = torch.cumsum(torch.bincount(group, minlength=start.numel() - 1), dim=0)
            pos = torch.empty(nv, dtype=torch.int64, device=dev)
            pos[order] = torch.arange(nv, device=dev)
            sub = (pos - start[group]) // max(1, per[k])
            width = int(sub.max()) + 1
            group = group * width + sub
        rank = torch.empty(nv, dtype=torch.int64, device=dev)
        rank[torch.argsort(self.x[:, d - 1], stable=True)] = torch.arange(nv, device=dev)
        vperm = torch.argsort(group * nv + rank)                    # new -> old
        vinv = torch.empty_like(vperm)
        vinv[vperm] = torch.arange(nv, device=dev)
        cells_new = vinv[self.cells.long()]
        cperm = torch.argsort(cells_new.min(dim=1).values, stable=True)
        new = Mesh(self.x[vperm], cells_new[cperm].to(torch.int32), self.cell_type, self.device)
        new.sfc_ordered = True
        new.reorder_curve = "pencil"
        new.original_cell_index = cperm
        new.input_global_indices = vperm
        return new

    # ---- host mirrors (lazy) -------------------------------------------------------------
    @property
    def x_host(self):
        if "x" not in self._host:
            self._host["x"] = self.x.cpu().numpy()
        return self._host["x"]

    @property
    def cells_host(self):
        if "cells" not in self._host:
            self._host["cells"] = self.cells.cpu().numpy()
        return self._host["cells"]

    # ---- facet topology (lazy, on the mesh's device) ----------------------------------------
    def _build(self):
        if self._topo is None:
            self._topo = build_facet_topology(self.cells, self.cell_type, self.num_vertices)
        return self._topo

    @property
    def c2f(self):
        return self._build()[0]

    @property
    def f2c(self):
        return self._build()[1]

    @property
    def facet_vertices(self):
        return self._build()[2]

    @property
    def num_facets(self):
        return int(self.f2c.shape[0])

    @property
    def boundary_facets(self):
        """Facets with a single cell (ascending int32 list), cached: a property of the mesh."""
        if "bfacets" not in self._host:
            self._host["bfacets"] = torch.nonzero(self.f2c[:, 1] < 0).reshape(-1).to(torch.int32).contiguous()
        return self._host["bfacets"]

    @property
    def x4(self):
        """Coordinates padded to 4 doubles per vertex (tetrahedra, cached): one 256-bit gather per vertex in the row-gather
        cell pass (phifem_mesh.x4)."""
        if "x4" not in self._host:
            x4 = torch.zeros((self.num_vertices, 4), dtype=torch.float64, device=self.device)
            x4[:, :self.gdim] = self.x
            self._host["x4"] = x4
        return self._host["x4"]

    def boundary_records(self):
        """(owner + meta [nb, 2] uint32 as int32 storage, scales [nb, 4]) of the mesh-boundary facets, cached: the static
        part of the ds detection of reference mesh_scripts.py:434-452 (csrc/tags.cu, k_boundary_records).  CUDA meshes
        only; None on the host."""
        if "brec" not in self._host:
            if self.device.type != "cuda":
                self._host["brec"] = (None, None)
            else:
                from . import _lib
                nb = int(self.boundary_facets.numel())
                owner = torch.zeros((max(nb, 1), 2), dtype=torch.int32, device=self.device)
                scale = torch.zeros((max(nb, 1), 4), dtype=torch.float64, device=self.device)
                _lib.check(_lib.load().phifem_boundary_records(
                    _lib.c_mesh(self, with_records=False), _lib.ptr(owner), _lib.ptr(scale), _lib.stream()))
                self._host["brec"] = (owner, scale)
        return self._host["brec"]

    def detj_bounds(self):
        """(min, max) of |det J| over the simplices of the mesh, cached ((0, 0) = unknown on other cells).  A property of the mesh
        alone: lets the P1 classifier decide uncut cells from the signs of phi without gathering
        coordinates (csrc/tags.cu, k_tag_cells_p1)."""
        if "detj" not in self._host:
            if self.cell_type not in G.SIMPLICES or self.num_cells == 0:
                self._host["detj"] = (0.0, 0.0)
            else:
                lo, hi = float("inf"), 0.0
                step = 1 << 24
                for s in range(0, self.num_cells, step):
                    xc = self.x[self.cells[s:s + step].long()]
                    e = xc[:, 1:, :] - xc[:, :1, :]
                    if e.shape[1] == 2:
                        det = e[:, 0, 0] * e[:, 1, 1] - e[:, 0, 1] * e[:, 1, 0]
                    else:
                        det = (e[:, 0] * torch.linalg.cross(e[:, 1], e[:, 2], dim=1)).sum(dim=1)
                    det = det.abs()
                    lo, hi = min(lo, float(det.min())), max(hi, float(det.max()))
                # widen: the kernel's own |det J| may differ from this one in the last bits
                self._host["detj"] = (lo * (1 - 1e-9), hi * (1 + 1e-9))
        return self._host["detj"]


def _unique_inverse(keys):
    uniq, inv = torch.unique(keys, sorted=True, return_inverse=True)
    return uniq, inv


def build_facet_topology(cells, cell_type, num_vertices):
    """Number the facets and build c2f / f2c / facet->vertices with sort-unique passes.

    Replaces `mesh.topology.create_connectivity(tdim, tdim-1)` / `(tdim-1, tdim)` as used at
    reference mesh_scripts.py:151-153,419-422.  Works on any torch device.
    """
    lfs = G.LOCAL_FACETS[cell_type]
    nc, nfpc, nvpf = cells.shape[0], len(lfs), len(lfs[0])
    c64 = cells.to(torch.int64)
    nv = int(num_vertices)
    # sorted vertex tuples of every (cell, local facet) instance, cell-major
    cols = []
    for lf in lfs:
        t, _ = torch.sort(c64[:, list(lf)], dim=1)
        cols.append(t)
    inst = torch.stack(cols, dim=1).reshape(nc * nfpc, nvpf)
    del cols
    key = inst[:, 0] * nv + inst[:, 1]
    if nvpf == 2:
        uniq, inv = _unique_inverse(key)
        fverts = torch.stack([uniq // nv, uniq % nv], dim=1)
    elif nvpf == 3:
        upair, pinv = _unique_inverse(key)          # rank of the leading pair keeps lexicographic order
        key = pinv * nv + inst[:, 2]
        del pinv
        uniq, inv = _unique_inverse(key)
        pair = upair[uniq // nv]
        fverts = torch.stack([pair // nv, pair % nv, uniq % nv], dim=1)
        del upair, pair
    else:
        # hexahedron faces: one more round; the rank of the leading triple keeps the order lexicographic
        upair, pinv = _unique_inverse(key)
        key = pinv * nv + inst[:, 2]
        del pinv
        utrip, tinv = _unique_inverse(key)
        key = tinv * nv + inst[:, 3]
        del tinv
        uniq, inv = _unique_inverse(key)
        trip = utrip[uniq // nv]
        pair = upair[trip // nv]
        fverts = torch.stack([pair // nv, pair % nv, trip % nv, uniq % nv], dim=1)
        del upair, utrip, trip, pair
    del inst, key
    nf = int(uniq.shape[0])
    c2f = inv.reshape(nc, nfpc).to(torch.int32)
    owner = torch.arange(nc, device=cells.device, dtype=torch.int32).repeat_interleave(nfpc)
    lo = torch.full((nf,), nc, dtype=torch.int32, device=cells.device)
    hi = torch.full((nf,), -1, dtype=torch.int32, device=cells.device)
    lo.scatter_reduce_(0, inv, owner, reduce="amin")
    hi.scatter_reduce_(0, inv, owner, reduce="amax")
    hi = torch.where(hi == lo, torch.full_like(hi, -1), hi)
    f2c = torch.stack([lo, hi], dim=1).contiguous()
    return c2f.contiguous(), f2c, fverts.to(torch.int32).contiguous()


class MeshTags:
    """`dolfinx.mesh.MeshTags` look-alike: `dim`, sorted int32 `indices`, int32 `values`, `find`.

    Tags live on the device (`values_dev` holds one entry per entity, 0 = untagged); the host
    views `indices` / `values` are materialised on first access (one D2H copy)."""

    def __init__(self, mesh, dim, values_dev=None, indices=None, values=None, tags8=None):
        self.mesh = mesh
        self.dim = dim
        self._values_dev = values_dev
        if tags8 is not None:     # the one-byte array the kernels wrote (computed tags fit a byte)
            self.tags8 = tags8
            self.tags8_exact = True
        self._indices = None if indices is None else np.ascontiguousarray(indices, dtype=np.int32)
        self._values = None if values is None else np.ascontiguousarray(values, dtype=np.int32)

    @property
    def values_dev(self):
        """Dense int32 tags on the device (the dtype of the reference's MeshTags.values); widened from the kernels'
        one-byte array on first access when only that was written."""
        if self._values_dev is None:
            self._values_dev = self.tags8.to(torch.int32)
        return self._values_dev

    @values_dev.setter
    def values_dev(self, v):
        self._values_dev = v

    @staticmethod
    def from_lists(mesh, dim, indices, values):
        """Like `dolfinx.mesh.meshtags(mesh, dim, indices, values)`."""
        indices = np.asarray(indices, dtype=np.int32)
        values = np.asarray(values, dtype=np.int32)
        n = mesh.num_cells if dim == mesh.topology.dim else mesh.num_facets
        dense = torch.zeros(n, dtype=torch.int32)
        dense[torch.from_numpy(indices.astype(np.int64))] = torch.from_numpy(values)
        return MeshTags(mesh, dim, dense.to(mesh.device), indices, values)

    def _materialise(self):
        if self._indices is None:
            # computed tags fit one byte: move the int8 copy the kernels wrote (4x fewer PCIe bytes) and
            # widen on the host; user-overwritten tags (`tags8_exact` unset) go through the int32 array
            t8 = getattr(self, "tags8", None)
            src = t8 if (t8 is not None and getattr(self, "tags8_exact", False)) else self.values_dev
            dense = src.cpu().numpy()
            idx = np.nonzero(dense)[0].astype(np.int32)
            self._indices, self._values = idx, dense[idx].astype(np.int32)

    @property
    def indices(self):
        self._materialise()
        return self._indices

    @property
    def values(self):
        self._materialise()
        return self._values

    def find(self, value):
        self._materialise()
        return self._indices[self._values == value]


class Measure:
    """What the reference returns as `ufl.Measure("ds", subdomain_data=[(100, e), (101, e)])`
    (mesh_scripts.py:631-633): calling it with an id selects the flat `[cell, local_facet, ...]`
    entity list of that id."""

    def __init__(self, integral_type, domain, subdomain_data=None):
        self.integral_type = integral_type
        self.domain = domain
        self.subdomain_data = subdomain_data

    def __call__(self, subdomain_id):
        return MeasureRestriction(self, subdomain_id)

    def entities(self, subdomain_id, device=False):
        if self.subdomain_data is None:
            raise ValueError("measure without subdomain data")
        for sid, ents in self.subdomain_data:
            if sid == subdomain_id:
                return ents if device else ents.cpu().numpy()
        raise KeyError(subdomain_id)


class MeasureRestriction:
    def __init__(self, measure, subdomain_id):
        self.measure = measure
        self.subdomain_id = subdomain_id

    @property
    def integration_entities(self):
        return self.measure.entities(self.subdomain_id)

    @property
    def integration_entities_dev(self):
        return self.measure.entities(self.subdomain_id, device=True)
