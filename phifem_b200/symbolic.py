"""The symbolic phase of the P1 strong-Dirichlet operator through the C ABI (csrc/symbolic.cu): CSR pattern and
entity -> slot maps built on the device with cub sort / unique, for hosts that do not go through the torch-based plan of
phifem_b200/assemble.py.  `DevicePattern` wraps the library-owned arrays as torch tensors (zero copy) and assembles with
the per-entity kernels.

    pat = symbolic.DevicePattern(mesh, cells_tags, facets_tags, ds_bdy(100))
    A, b = pat.assemble(phi, f, stab_coef=1.0)

`DevicePkPattern` does the same for the quadrature-kernel operators (strong / weak Dirichlet, Neumann, Robin;
phifem_pk_pattern_create): the arrays of `assemble_pk.PkAssemblyPlan` for a caller-given pattern dofmap.
`DeviceElasticityPattern` does it for the interface-elasticity operator (phifem_elasticity_pattern_create): the arrays
of `elasticity.ElasticityPlan`.
"""
import ctypes

import torch

from . import _lib
from .assemble import CSRMatrix, _device_vector, _plan_inputs


def _as_tensor(ptr, n, device):
    """int32 device array owned by the library -> torch view (kept alive by the DevicePattern)."""
    if n == 0:
        return torch.zeros(0, dtype=torch.int32, device=device)

    class _Holder:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i4", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(_Holder(), device=device)


class DevicePattern:
    def __init__(self, mesh, cells_tags, facets_tags, ds=None):
        _lib.require_cuda(mesh)
        c8, f8, ents = _plan_inputs(mesh, cells_tags, facets_tags, ds)
        self.mesh, self.cell_tags8 = mesh, c8
        self.entities = ents.reshape(-1, 2).to(torch.int32).contiguous()
        lib = _lib.load()
        handle = ctypes.c_void_p()
        _lib.check(lib.phifem_pattern_create_p1(_lib.c_mesh(mesh), _lib.ptr(c8), _lib.ptr(f8),
                                                _lib.ptr(self.entities) if self.entities.numel() else None,
                                                self.entities.shape[0], ctypes.byref(handle), _lib.stream()))
        self._handle = handle
        v = _lib.CPatternView()
        _lib.check(lib.phifem_pattern_view_of(handle, ctypes.byref(v)))
        nv = mesh.cells.shape[1]
        dev = mesh.device
        self.n_rows, self.nnz = int(v.n_rows), int(v.nnz)
        self.indptr = _as_tensor(v.indptr, v.n_rows + 1, dev)
        self.indices = _as_tensor(v.indices, v.nnz, dev)
        self.active = _as_tensor(v.active, v.n_active, dev)
        self.ghost = _as_tensor(v.ghost, v.n_ghost, dev)
        self.slots_cells = _as_tensor(v.slots_cells, v.n_active * nv * nv, dev).reshape(-1, nv * nv)
        self.slots_ghost = _as_tensor(v.slots_ghost, v.n_ghost * (nv + 1) ** 2, dev).reshape(-1, (nv + 1) ** 2)
        self.slots_boundary = _as_tensor(v.slots_boundary, v.n_entities * nv * nv, dev).reshape(-1, nv * nv)

    def __del__(self):
        h = getattr(self, "_handle", None)
        if h and _lib is not None:       # (module globals are gone at interpreter shutdown)
            try:
                _lib.load().phifem_pattern_destroy(h)
            except Exception:
                pass
            self._handle = None

    def assemble(self, phi_h, f_h, stab_coef=1.0):
        """A, b of reference demo/strong-dirichlet/flower/main.py:121-131 through the per-entity kernels."""
        mesh = self.mesh
        lib = _lib.load()
        cm = _lib.c_mesh(mesh)
        phi, f = _device_vector(mesh, phi_h), _device_vector(mesh, f_h)
        data = torch.zeros(self.nnz, dtype=torch.float64, device=mesh.device)
        b = torch.zeros(self.n_rows, dtype=torch.float64, device=mesh.device)
        st = _lib.stream()
        p = _lib.ptr
        if self.active.numel():
            _lib.check(lib.phifem_assemble_cells_p1(cm, p(phi), p(f), p(self.cell_tags8), p(self.active),
                                                    self.active.numel(), p(self.slots_cells), float(stab_coef),
                                                    p(data), p(b), st))
        if self.entities.shape[0]:
            _lib.check(lib.phifem_assemble_boundary_p1(cm, p(phi), p(self.entities), self.entities.shape[0],
                                                       p(self.slots_boundary), p(data), st))
        if self.ghost.numel():
            _lib.check(lib.phifem_assemble_ghost_p1(cm, p(phi), p(self.ghost), self.ghost.numel(),
                                                    p(self.slots_ghost), float(stab_coef), p(data), st))
        A = CSRMatrix(self.indptr, self.indices, data, (self.n_rows, self.n_rows))
        A._pattern = self          # indptr / indices are views of arrays this object owns
        return A, b


class DevicePkPattern:
    """The symbolic phase of the quadrature-kernel operators through the C ABI (phifem_pk_pattern_create): the arrays of
    `assemble_pk.PkAssemblyPlan` under the same names and shapes, built on the device and owned by the library.

        plan = assemble.build_plan_weak_dirichlet(mesh, cells_tags, facets_tags, ds(100))
        pat = symbolic.DevicePkPattern(mesh, cells_tags, facets_tags, ds(100), plan.pattern_dofmap, plan.n_rows)

    `pattern_dofmap` [n_cells, nd]: the cell-local dofs of the space being assembled; `ghost_tags`: the facet tags that
    carry the ghost penalty, (2, 3) for strong and weak Dirichlet, (3,) for the Neumann demo, (2,) for the Robin demo."""

    def __init__(self, mesh, cells_tags, facets_tags, ds, pattern_dofmap, n_rows, ghost_tags=(2, 3)):
        _lib.require_cuda(mesh)
        c8, f8, ents = _plan_inputs(mesh, cells_tags, facets_tags, ds)
        self.mesh, self.cell_tags8 = mesh, c8
        self.entities = ents.reshape(-1, 2).to(torch.int32).contiguous()
        dm = pattern_dofmap.to(device=mesh.device, dtype=torch.int32).contiguous()
        nd = int(dm.shape[1])
        mask = 0
        for t in ghost_tags:
            if not 0 <= int(t) <= 6:
                raise ValueError("ghost tag %r outside the tag values 0..6" % (t,))
            mask |= 1 << int(t)
        lib = _lib.load()
        self._handle = _PatternHandle("phifem_pk_pattern_destroy")
        _lib.check(lib.phifem_pk_pattern_create(_lib.c_mesh(mesh), _lib.ptr(dm), nd, int(n_rows), _lib.ptr(c8),
                                                _lib.ptr(f8), mask,
                                                _lib.ptr(self.entities) if self.entities.numel() else None,
                                                self.entities.shape[0], ctypes.byref(self._handle.h), _lib.stream()))
        v = _lib.CPkPatternView()
        _lib.check(lib.phifem_pk_pattern_view_of(self._handle.h, ctypes.byref(v)))
        dev, i32 = mesh.device, torch.int32

        def view(p, *shape):           # each tensor keeps the handle alive: the arrays outlive this object if need be
            return _lib.device_view(p, shape, i32, dev, owner=self._handle)
        self.n_rows, self.nnz = int(v.n_rows), int(v.nnz)
        self.indptr = view(v.indptr, v.n_rows + 1)
        self.indices = view(v.indices, v.nnz)
        self.active = view(v.active, v.n_active)
        self.cut_positions = view(v.cut_positions, v.n_cut)
        self.ghost = view(v.ghost, v.n_ghost)
        self.slots_cells = view(v.slots_cells, nd * nd, v.n_active)
        self.slots_ghost = view(v.slots_ghost, v.n_ghost, 4 * nd * nd)
        self.slots_boundary = view(v.slots_boundary, v.n_entities, nd * nd)


class DeviceElasticityPattern:
    """The symbolic phase of the interface-elasticity operator through the C ABI (phifem_elasticity_pattern_create): the
    arrays of `elasticity.ElasticityPlan` under the same names and shapes, built on the device and owned by the library.

        pat = symbolic.DeviceElasticityPattern(mesh, cells_tags, facets_tags, d_bdry)

    `d_bdry`: the measure of compute_tags_measures(box_mode=True), whose ids 100 and 101 are used, or a pair of entity
    arrays (ds100, ds101), as for `elasticity.build_plan_interface_elasticity`."""

    def __init__(self, mesh, cells_tags, facets_tags, d_bdry):
        from .mesh import Measure
        _lib.require_cuda(mesh)
        d100, d101 = (d_bdry(100), d_bdry(101)) if isinstance(d_bdry, Measure) else d_bdry
        c8, f8, e_in = _plan_inputs(mesh, cells_tags, facets_tags, d100)
        _, _, e_out = _plan_inputs(mesh, cells_tags, facets_tags, d101)
        self.mesh, self.cell_tags8 = mesh, c8
        self.entities_in = e_in.reshape(-1, 2).to(torch.int32).contiguous()
        self.entities_out = e_out.reshape(-1, 2).to(torch.int32).contiguous()
        lib = _lib.load()
        self._handle = _PatternHandle("phifem_elasticity_pattern_destroy")
        ents = [(_lib.ptr(e) if e.numel() else None, e.shape[0]) for e in (self.entities_in, self.entities_out)]
        _lib.check(lib.phifem_elasticity_pattern_create(_lib.c_mesh(mesh), _lib.ptr(c8), _lib.ptr(f8), *ents[0],
                                                        *ents[1], ctypes.byref(self._handle.h), _lib.stream()))
        v = _lib.CElasticityPatternView()
        _lib.check(lib.phifem_elasticity_pattern_view_of(self._handle.h, ctypes.byref(v)))
        dev, i32 = mesh.device, torch.int32
        nv = mesh.cells.shape[1]

        def view(p, *shape):           # each tensor keeps the handle alive: the arrays outlive this object if need be
            return _lib.device_view(p, shape, i32, dev, owner=self._handle)
        self.nb, self.n_rows, self.nnz = int(v.nb), int(v.n_rows), int(v.nnz)
        self.vptr = view(v.vptr, v.n_vertices + 1)
        self.indptr = view(v.indptr, v.n_rows + 1)
        self.indices = view(v.indices, v.nnz)
        self.cut_cells = view(v.cut_cells, v.n_cut)
        self.facets_in = view(v.facets_in, v.n_facets_in)
        self.facets_out = view(v.facets_out, v.n_facets_out)
        self.pos_cells = view(v.pos_cells, v.n_cells, nv * nv)
        self.pos_facets_in = view(v.pos_facets_in, v.n_facets_in, 4 * nv * nv)
        self.pos_facets_out = view(v.pos_facets_out, v.n_facets_out, 4 * nv * nv)
        self.pos_entities_in = view(v.pos_entities_in, v.n_entities_in, nv * nv)
        self.pos_entities_out = view(v.pos_entities_out, v.n_entities_out, nv * nv)


class _PatternHandle:
    """Owner of a library pattern handle, released by `destroy`: destroyed with the last tensor that views its
    arrays."""

    def __init__(self, destroy):
        self.h = ctypes.c_void_p()
        self.destroy = destroy

    def __del__(self):
        if self.h and _lib is not None:       # (module globals are gone at interpreter shutdown)
            try:
                getattr(_lib.load(), self.destroy)(self.h)
            except Exception:
                pass
            self.h = None
