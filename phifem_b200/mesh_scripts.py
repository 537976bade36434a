"""Drop-in for `phifem.mesh_scripts` (reference src/phifem/mesh_scripts.py) on B200.

Same public function, argument meaning, tag values, measure ids and error behaviour as the
reference; underneath, the classification runs as hand-written CUDA kernels (csrc/tags.cu)
called through the C ABI of include/phifem_b200.h.  There is no CPU path: a mesh that does
not live on a CUDA device raises.

Public API (reference :571-653):

    cells_tags, facets_tags, submesh, boundaries_measure, submesh_maps = compute_tags_measures(
        mesh, discrete_levelset, detection_degree, box_mode=False, single_layer_cut=False,
        overwrite_tags={})

`mesh` is a `phifem_b200.mesh.Mesh` of triangles, quadrilaterals, tetrahedra or hexahedra (the last two are
extensions: the reference stops at 2D); `discrete_levelset` is a `phifem_b200.fem.Function`
(P1..P3, Q1..Q3, Q1 / Q2 on hexahedra) or a callable of the physical coordinates `f(x)` with `x` of shape (gdim, npoints)
(the stand-in for the reference's UFL expression of `SpatialCoordinate`).
"""
import os
import ctypes
import threading
import warnings

import numpy as np
import torch

from . import _geometry as G
from . import _lib
from .fem import Function
from .mesh import Measure, Mesh, MeshTags

debug_mode = os.environ.get("MODE") == "debug"  # reference :22-25

_reference_segment_points = G.reference_segment_points
_reference_triangle_boundary_points = G.reference_triangle_boundary_points
_reference_square_boundary_points = G.reference_square_boundary_points

_ZERO_WARNING = ("The detection function is zero everywhere on a cell. We mark it as 'cut' but this "
                 "can be incorrect and should be carefully checked.")


class _DeviceLevelset:
    """Level set staged for the kernels: owns the device buffers the C struct points to."""

    def __init__(self, mesh, levelset, detection_degree):
        ct, dev = mesh.cell_type, mesh.device
        pts = G.cell_detection_points(ct, detection_degree)       # raises NotImplementedError like :326-329
        fpts = G.facet_detection_points(ct, detection_degree)     # [nfpc, nq, tdim]
        self.npts, self.nq = len(pts), fpts.shape[1]
        self.keep = []
        f64 = dict(dtype=torch.float64, device=dev)
        coord_grad = None
        if ct == "quadrilateral":
            coord_grad = torch.as_tensor(G.coordinate_basis_grad(ct, pts), **f64).contiguous()
        elif ct == "hexahedron":
            # [npts + nfpc nq, 8, 3]: the trilinear map's gradients at the cell points, then at the facet points --
            # the kernels take |det J| and the face scale |dx/ds x dx/dt| per point from them
            grads = np.concatenate([G.coordinate_basis_grad(ct, pts),
                                    G.coordinate_basis_grad(ct, fpts.reshape(-1, fpts.shape[-1]))])
            coord_grad = torch.as_tensor(grads, **f64).contiguous()
        self.c = _lib.CLevelset()
        self.c.n_cell_points, self.c.n_facet_points = self.npts, self.nq
        self.c.coord_grad = _lib.ptr(coord_grad)
        self.keep.append(coord_grad)
        if isinstance(levelset, Function):
            V = levelset.function_space
            if V.mesh is not mesh:
                raise ValueError("the level set is defined on another mesh")
            coeffs = levelset.x.array
            coeffs = coeffs if torch.is_tensor(coeffs) else torch.from_numpy(np.ascontiguousarray(coeffs))
            coeffs = coeffs.to(dev, dtype=torch.float64, non_blocking=True).contiguous()
            nd = V.element.ndofs
            simplex_p1 = (V.degree == 1 and detection_degree == 1 and ct in G.SIMPLICES)
            self.c.mode, self.c.n_dofs_per_cell = 0, nd
            self.c.coeffs = _lib.ptr(coeffs)
            ftab = torch.as_tensor(V.element.tabulate(fpts), **f64).contiguous()
            self.c.facet_table = _lib.ptr(ftab)
            self.keep += [coeffs, ftab]
            if simplex_p1:
                # vertex dofs, points on the vertices: identity table => fast kernel (dofmap = cells)
                self.c.dofmap, self.c.cell_table = None, None
            else:
                dm = V.dofmap_dev
                ctab = torch.as_tensor(V.element.tabulate(pts), **f64).contiguous()
                self.c.dofmap, self.c.cell_table = _lib.ptr(dm), _lib.ptr(ctab)
                self.keep += [ctab, dm]
        elif callable(levelset):
            vals = self._evaluate(mesh, levelset, pts)
            fvals = self._evaluate(mesh, levelset, fpts.reshape(-1, fpts.shape[-1]))
            self.c.mode = 1
            self.c.cell_values, self.c.facet_values = _lib.ptr(vals), _lib.ptr(fvals)
            self.keep += [vals, fvals]
        else:
            raise TypeError("discrete_levelset must be a phifem_b200.fem.Function or a callable f(x)")

    @staticmethod
    def _evaluate(mesh, func, ref_pts):
        """phi at the push-forward of reference points: the points are computed on the device
        (phifem_cell_points), the user's Python expression is evaluated on the host."""
        shape = torch.as_tensor(G.coordinate_basis(mesh.cell_type, ref_pts), dtype=torch.float64,
                                device=mesh.device).contiguous()
        npts = len(ref_pts)
        xq = torch.empty((mesh.num_cells, npts, mesh.gdim), dtype=torch.float64, device=mesh.device)
        cm = _lib.c_mesh(mesh, with_facets=False)
        _lib.check(_lib.load().phifem_cell_points(cm, _lib.ptr(shape), npts, _lib.ptr(xq), _lib.stream()))
        pts = xq.reshape(-1, mesh.gdim).T.cpu().numpy()
        with np.errstate(all="ignore"):
            vals = np.asarray(func(pts), dtype=np.float64).reshape(mesh.num_cells, npts)
        return torch.from_numpy(np.ascontiguousarray(vals)).to(mesh.device)


class TagWorkspace:
    """Device buffers of one classification (reused across calls on the same mesh)."""

    def __init__(self, mesh, int32=False):
        """int32=True: the kernels also write the tags as int32 arrays (the dtype of the reference's MeshTags);
        by default only the one-byte arrays the facet / assembly kernels consume are written -- a quarter of the output
        bytes of the tag kernels -- and `MeshTags.values_dev` widens them when somebody asks."""
        dev = mesh.device
        self.cell_tags32 = torch.empty(mesh.num_cells, dtype=torch.int32, device=dev) if int32 else None
        self.cell_tags8 = torch.empty(mesh.num_cells, dtype=torch.int8, device=dev)
        self.facet_tags32 = torch.empty(mesh.num_facets, dtype=torch.int32, device=dev) if int32 else None
        self.facet_tags8 = torch.empty(mesh.num_facets, dtype=torch.int8, device=dev)
        self.counters = torch.zeros(_lib.N_COUNTERS, dtype=torch.int64, device=dev)
        self.vertex_scratch = None

    @property
    def cell_tags(self):
        """int32 view of the cell tags (widened on demand when the kernels wrote int8 only)."""
        return self.cell_tags32 if self.cell_tags32 is not None else self.cell_tags8.to(torch.int32)

    @property
    def facet_tags(self):
        return self.facet_tags32 if self.facet_tags32 is not None else self.facet_tags8.to(torch.int32)


_host_counters = threading.local()


def _read_counters(ws):
    """The counter block on the host: THE host synchronisation of a `compute_tags_measures` call.  A kernel posts the
    128 bytes into page-locked host memory (`phifem_post_to_host`) and the host waits for an event on the calling
    stream only -- a `counters.cpu()` would be a copy-engine transfer, which queues behind whatever download another
    stream has in flight (the CSR values of the previous step, in a pipeline with two steps in flight)."""
    key = ws.counters.device.index
    bufs = getattr(_host_counters, "bufs", None)
    if bufs is None:
        bufs = _host_counters.bufs = {}
    if key not in bufs:
        bufs[key] = (torch.zeros(_lib.N_COUNTERS, dtype=torch.int64).pin_memory(), torch.cuda.Event())
    host, event = bufs[key]
    _lib.check(_lib.load().phifem_post_to_host(_lib.ptr(ws.counters), host.data_ptr(), _lib.N_COUNTERS, _lib.stream()))
    event.record()
    event.synchronize()
    return host.numpy().copy()


def classify_cells(mesh, dls, ws, single_layer_cut=False, exact_zero_den=False):
    """K1 on the current stream: zero the counters, tag the cells (no host synchronisation).
    exact_zero_den: evaluate the isclose(den, 0) test of reference :129 on every cell instead of
    counting the inconclusive ones in counters[CNT_ZERO_DEN_AMBIGUOUS] (the tags do not depend on it)."""
    ws.counters.zero_()
    if ws.vertex_scratch is None:   # vertex class bytes of the P1 classifier, flags of single_layer_cut
        ws.vertex_scratch = torch.empty(mesh.num_vertices + 3, dtype=torch.uint8, device=mesh.device)
    _lib.check(_lib.load().phifem_tag_cells(
        _lib.c_mesh(mesh), dls.c, int(bool(single_layer_cut)) | (2 if exact_zero_den else 0),
        _lib.ptr(ws.cell_tags32),
        _lib.ptr(ws.cell_tags8), _lib.ptr(ws.vertex_scratch), _lib.ptr(ws.counters), _lib.stream()))


FACETS_INTERIOR, FACETS_BOUNDARY = 1, 2


def classify_facets(mesh, dls, ws, phases=FACETS_INTERIOR | FACETS_BOUNDARY):
    """Facet tags from the cell tags of `ws` on the current stream (no host synchronisation).  `phases`: run only
    the interior facets (independent of the global "any exterior cell" flag) or only the mesh-boundary facets
    (which read it) -- the sharded classifiers put their all-reduce between the two."""
    _lib.check(_lib.load().phifem_tag_facets_phase(
        _lib.c_mesh(mesh), dls.c, _lib.ptr(ws.cell_tags8), _lib.ptr(ws.facet_tags32),
        _lib.ptr(ws.facet_tags8), _lib.ptr(ws.counters), int(phases), _lib.stream()))


def classify_sharded(mesh, dls, ws, group=None, world=1, mark=None, single_layer_cut=False, peer=None):
    """Cells, then the interior facets WHILE the exterior-cell counts of the ranks travel, then the mesh-boundary facets
    (reference :469-474 makes their tags depend on the global "any exterior cell" flag).  The exchange is either
    `peer` (phifem_b200/peer.py: 8-byte stores into the peers' HBM over NVLink after the cell kernel, a read of the own
    slots before the facet kernels: two one-warp kernels) or, without it, an 8-byte `torch.distributed` all-reduce
    overlapped with the interior-facet kernel.  `mark` (optional callable) is invoked after the cell kernel and at the
    end (bench.py records CUDA events there)."""
    import torch.distributed as dist
    mark = mark or (lambda: None)
    classify_cells(mesh, dls, ws, single_layer_cut)
    mark()
    count = ws.counters[_lib.CNT_EXTERIOR:_lib.CNT_EXTERIOR + 1]
    if world > 1 and peer is not None:
        # the ranks run in lockstep, so the peers' stores are there (or microseconds away) when this rank's cell kernel
        # ends: collect at once and let the two facet kernels overlap on their fork / join streams as on one GPU
        peer.publish(count)
        peer.collect(count)
        classify_facets(mesh, dls, ws)
    elif world > 1:
        work = dist.all_reduce(count, group=group, async_op=True)
        classify_facets(mesh, dls, ws, FACETS_INTERIOR)
        work.wait()
        classify_facets(mesh, dls, ws, FACETS_BOUNDARY)
    else:
        classify_facets(mesh, dls, ws)
    mark()
    return ws


def classify(mesh, dls, single_layer_cut=False, ws=None, exact_zero_den=False):
    """Run the tag kernels (cells, then facets) on the current stream; returns the workspace."""
    ws = ws or TagWorkspace(mesh)
    classify_cells(mesh, dls, ws, single_layer_cut, exact_zero_den)
    classify_facets(mesh, dls, ws)
    return ws


def _cell_mask(cell_tag_values):
    mask = 0
    for t in cell_tag_values:
        mask |= 1 << int(t)
    return mask


# the two one-sided measures of box mode (reference :617-626): (facet tag, cell tags, counter slot of the count)
_DS_OUT = (4, (1, 2), _lib.CNT_CALLER0)
_DS_IN = (3, (2, 3), _lib.CNT_CALLER1)


def _count_entities(mesh, ws, cell_tags8, facet_tags8):
    """Queue the counting passes of ds(100) / ds(101) behind the tag kernels; the counts land in the two caller slots
    of the counter block, so that the ONE device -> host copy that fetches the counters brings them along."""
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    for facet_tag, cell_values, slot in (_DS_OUT, _DS_IN):
        _lib.check(lib.phifem_integration_entities_count(
            cm, _lib.ptr(cell_tags8), _lib.ptr(facet_tags8), facet_tag, _cell_mask(cell_values),
            ws.counters.data_ptr() + 8 * slot, _lib.stream()))


def _integration_entities_dev(mesh, cell_tags8, facet_tags8, facet_tag, cell_tag_values, n_known=None):
    """Device version of `_compute_integration_entities` (reference :137-192): flat int32
    [cell, local_facet, ...] tensor, cells in first-appearance order, local facets ascending.
    n_known: the number of pairs when the caller has already read it back (no host synchronisation then)."""
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    mask = _cell_mask(cell_tag_values)
    # candidates, first-appearance ordering and the sort all happen behind the C ABI (csrc/symbolic.cu)
    if n_known is not None:
        ents = torch.empty((int(n_known), 2), dtype=torch.int32, device=mesh.device)
        _lib.check(lib.phifem_integration_entities_fill(cm, _lib.ptr(cell_tags8), _lib.ptr(facet_tags8), facet_tag,
                                                        mask, _lib.ptr(ents), int(n_known), _lib.stream()))
        return ents.reshape(-1)
    n = ctypes.c_int64(0)
    capacity = max(1024, int(4 * mesh.num_facets ** (1 - 1.0 / mesh.topology.dim)))
    while True:
        ents = torch.empty((capacity, 2), dtype=torch.int32, device=mesh.device)
        _lib.check(lib.phifem_integration_entities(cm, _lib.ptr(cell_tags8), _lib.ptr(facet_tags8), facet_tag, mask,
                                                   _lib.ptr(ents), capacity, ctypes.byref(n), _lib.stream()))
        if n.value <= capacity:
            break
        capacity = int(n.value)
    return ents[:n.value].reshape(-1).contiguous()


def _narrow_tags(values_dev):
    """One-byte copy of dense int32 tags for the kernels.  The kernels and the plans only ever compare with the
    computed values 1..6; a user tag of `overwrite_tags` may be any other integer (reference :606-615 reserves only
    1..6 / 100 / 101), and a plain int8 cast would wrap 257 -> 1, 260 -> 4: everything outside 0..6 becomes 0
    ("matches nothing"), exactly as `find(4)` of the reference does not match 260."""
    v = values_dev
    return torch.where((v >= 0) & (v <= 6), v, torch.zeros_like(v)).to(torch.int8).contiguous()


def _tags_from_workspace(mesh, ws):
    tdim = mesh.topology.dim
    return (MeshTags(mesh, tdim, ws.cell_tags32, tags8=ws.cell_tags8),
            MeshTags(mesh, tdim - 1, ws.facet_tags32, tags8=ws.facet_tags8))


def _overwrite_tags(mesh, tags_to_overwrite, new_tags):
    """Reference :561-568: the user's tags win where both are defined."""
    dense = tags_to_overwrite.values_dev.clone()
    idx = torch.from_numpy(np.asarray(new_tags.indices, dtype=np.int64)).to(dense.device)
    dense[idx] = torch.from_numpy(np.asarray(new_tags.values, dtype=np.int32)).to(dense.device)
    return MeshTags(mesh, tags_to_overwrite.dim, dense)


def _check_debug(counters, facet_tags8):
    """MODE=debug assertions of reference :360-374 and :499-521 that apply to dense tag arrays."""
    if counters[_lib.CNT_INTERIOR] == 0:
        raise ValueError("No interior cells (1)!")
    if counters[_lib.CNT_CUT] == 0:
        print("WARNING: no cut cells computed in the partition.")
    ft = torch.bincount(facet_tags8.to(torch.int64), minlength=7)[1:7].cpu().numpy()
    if ft[0] == 0:
        raise ValueError("No interior facets (1)!")
    if ft[1] == 0:
        print("WARNING: no cut facet computed in the partition.")
    if ft[3] == 0:
        raise ValueError("No boundary facets (4)!")
    if counters[_lib.CNT_FACET_CONFLICT] != 0:
        raise ValueError("facet sets have a non-empty intersection!")


def compute_tags_measures(mesh, discrete_levelset, detection_degree, box_mode=False,
                          single_layer_cut=False, overwrite_tags={}):
    """Compute the mesh (cells and facets) tags as well as the discrete boundary measures.

    Same contract as reference src/phifem/mesh_scripts.py:571-653.  Cells: 1 inside, 2 cut,
    3 outside (:290-293).  Facets: 1 interior, 2 cut, 3 inside/cut interface, 4 Gamma_h,
    5 exterior, 6 direct inside/outside interface (:399-405).  box_mode=True returns tags on the
    input mesh and a `ds` measure whose id 100 / 101 hold the one-sided entities (:617-634);
    box_mode=False returns the submesh of Omega_h, tags re-indexed on it and its maps (:635-645).
    """
    if not isinstance(mesh, Mesh):
        raise TypeError("mesh must be a phifem_b200.mesh.Mesh")
    _lib.require_cuda(mesh)
    dls = _DeviceLevelset(mesh, discrete_levelset, detection_degree)
    ws = classify(mesh, dls, single_layer_cut)
    # box mode without user tags: the counting passes of ds(100) / ds(101) go behind the tag kernels, and the single
    # device -> host copy below (warnings, debug checks) returns their counts too -- ONE host synchronisation per call
    counted = box_mode and not overwrite_tags
    if counted:
        _count_entities(mesh, ws, ws.cell_tags8, ws.facet_tags8)
    counters = _read_counters(ws)
    if counters[_lib.CNT_ZERO_DEN] == 0 and counters[_lib.CNT_ZERO_DEN_AMBIGUOUS] > 0:
        # no cell settled the RuntimeWarning of :129-133 and some were left undecided: evaluate them
        ws = classify(mesh, dls, single_layer_cut, ws=ws, exact_zero_den=True)
        if counted:
            _count_entities(mesh, ws, ws.cell_tags8, ws.facet_tags8)
        counters = _read_counters(ws)
    if counters[_lib.CNT_ZERO_DEN] > 0:           # :129-133 for the dx detection
        warnings.warn(_ZERO_WARNING, RuntimeWarning)
    if counters[_lib.CNT_FACET_ZERO_DEN] > 0 or counters[_lib.CNT_BOUNDARY_OWNERS] < mesh.num_cells:
        # the ds detection vector is zero on every cell without a mesh-boundary facet: the
        # reference warns here on essentially every mesh (SURVEY.md section 8b)
        warnings.warn(_ZERO_WARNING, RuntimeWarning)
    if debug_mode:
        _check_debug(counters, ws.facet_tags8)
    cells_tags, facets_tags = _tags_from_workspace(mesh, ws)
    cell_tags8, facet_tags8 = ws.cell_tags8, ws.facet_tags8

    if "cells" in overwrite_tags.keys():          # :606-610
        ow = overwrite_tags["cells"]
        if np.any(np.isin([1, 2, 3], ow.values)):
            raise ValueError("Cannot overwrite cells tags with values 1, 2 or 3.")
        cells_tags = _overwrite_tags(mesh, cells_tags, ow)
        cell_tags8 = _narrow_tags(cells_tags.values_dev)
    if "facets" in overwrite_tags.keys():         # :611-615
        ow = overwrite_tags["facets"]
        if np.any(np.isin([1, 2, 3, 4, 5, 6, 100, 101], ow.values)):
            raise ValueError("Cannot overwrite facets tags with values 1, 2, 3, 4, 5, 6, 100 or 101.")
        facets_tags = _overwrite_tags(mesh, facets_tags, ow)
        facet_tags8 = _narrow_tags(facets_tags.values_dev)

    if box_mode:                                   # :617-634
        ents_out = _integration_entities_dev(mesh, cell_tags8, facet_tags8, *_DS_OUT[:2],
                                             n_known=counters[_DS_OUT[2]] if counted else None)
        ents_in = _integration_entities_dev(mesh, cell_tags8, facet_tags8, *_DS_IN[:2],
                                            n_known=counters[_DS_IN[2]] if counted else None)
        measure = Measure("ds", mesh, subdomain_data=[(100, ents_out), (101, ents_in)])
        cells_tags.tags8, facets_tags.tags8 = cell_tags8, facet_tags8
        cells_tags.tags8_exact = "cells" not in overwrite_tags
        facets_tags.tags8_exact = "facets" not in overwrite_tags
        return cells_tags, facets_tags, None, measure, None

    # submesh of Omega_h = cells tagged 1 or 2 (:635-645)
    keep = torch.nonzero((cell_tags8 == 1) | (cell_tags8 == 2)).reshape(-1)
    sub_parent = mesh.cells[keep].long()
    v_map = torch.unique(sub_parent)
    renum = torch.full((mesh.num_vertices,), -1, dtype=torch.int64, device=mesh.device)
    renum[v_map] = torch.arange(len(v_map), device=mesh.device)
    submesh = Mesh(mesh.x[v_map], renum[sub_parent].to(torch.int32), mesh.cell_type, mesh.device)
    sub_cell = cells_tags.values_dev[keep].contiguous()
    parent_facet = torch.empty(submesh.num_facets, dtype=torch.int64, device=mesh.device)
    parent_facet[submesh.c2f.reshape(-1).long()] = mesh.c2f[keep].reshape(-1).long()   # :244-260
    sub_facet = facets_tags.values_dev[parent_facet].contiguous()
    tdim = mesh.topology.dim
    c_map = keep.to(torch.int32).cpu().numpy()
    v_map_h = v_map.to(torch.int32).cpu().numpy()
    return (MeshTags(submesh, tdim, sub_cell), MeshTags(submesh, tdim - 1, sub_facet), submesh,
            Measure("ds", submesh), [c_map, v_map_h, v_map_h.copy()])


# the reference's test file calls the function by this name (tests/test_compute_meshtags.py:122)
compute_meshtags = compute_tags_measures


def _tag_cells(mesh, discrete_levelset, detection_degree, single_layer_cut=False):
    """Reference :284-390 (cells only)."""
    return compute_tags_measures(mesh, discrete_levelset, detection_degree, box_mode=True,
                                 single_layer_cut=single_layer_cut)[0]


def _tag_facets(mesh, cells_tags, discrete_levelset, detection_degree):
    """Reference :393-558 for given cell tags."""
    _lib.require_cuda(mesh)
    dls = _DeviceLevelset(mesh, discrete_levelset, detection_degree)
    ws = TagWorkspace(mesh)
    ws.cell_tags8 = _narrow_tags(cells_tags.values_dev).contiguous()
    ws.counters[_lib.CNT_EXTERIOR] = int((ws.cell_tags8 == 3).sum())
    _lib.check(_lib.load().phifem_tag_facets(_lib.c_mesh(mesh), dls.c, _lib.ptr(ws.cell_tags8),
                                             _lib.ptr(ws.facet_tags32), _lib.ptr(ws.facet_tags8),
                                             _lib.ptr(ws.counters), _lib.stream()))
    return MeshTags(mesh, mesh.topology.dim - 1, ws.facet_tags32, tags8=ws.facet_tags8)


def _compute_integration_entities(mesh, integration_cells, integration_facets, ind):
    """Reference :137-192, for explicit index lists (host arrays)."""
    _lib.require_cuda(mesh)
    ct8 = torch.zeros(mesh.num_cells, dtype=torch.int8, device=mesh.device)
    ct8[torch.as_tensor(np.asarray(integration_cells, dtype=np.int64), device=mesh.device)] = 1
    ft8 = torch.zeros(mesh.num_facets, dtype=torch.int8, device=mesh.device)
    ft8[torch.as_tensor(np.asarray(integration_facets, dtype=np.int64), device=mesh.device)] = 1
    ents = _integration_entities_dev(mesh, ct8, ft8, 1, (1,))
    return [(ind, ents.cpu().numpy())]


def _reshape_map(connect):
    """Reference :195-214: padded dense map, columns in reverse link order."""
    counts = np.diff(connect.offsets)
    width = int(counts.max())
    out = -np.ones((len(counts), width), dtype=int)
    ends = connect.offsets[1:]
    for col in range(width):
        has = counts > col
        out[has, col] = connect.array[ends[has] - col - 1]
    return out, width


def _transfer_tags(source_mesh_tags, dest_mesh, cmap, source_mesh=None):
    """Reference :217-281: re-index cell or facet tags onto a submesh."""
    cdim = dest_mesh.topology.dim
    cmap_d = torch.as_tensor(np.asarray(cmap, dtype=np.int64), device=dest_mesh.device)
    if source_mesh_tags.dim == cdim:
        return MeshTags(dest_mesh, cdim, source_mesh_tags.values_dev[cmap_d].contiguous())
    if source_mesh_tags.dim == cdim - 1:
        if source_mesh is None:
            raise ValueError("You must pass a source_mesh to transfer facets tags.")
        parent = torch.empty(dest_mesh.num_facets, dtype=torch.int64, device=dest_mesh.device)
        parent[dest_mesh.c2f.reshape(-1).long()] = source_mesh.c2f[cmap_d].reshape(-1).long()
        return MeshTags(dest_mesh, cdim - 1, source_mesh_tags.values_dev[parent].contiguous())
    raise ValueError("The source_mesh_tags can only be cells tags or facets tags.")
