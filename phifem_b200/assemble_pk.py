"""Strong-Dirichlet phi-FEM operator for Lagrange P1 / P2 trial-test spaces and P1 / P2 level sets
(`fe_degree`, `levelset_degree` of reference demo/strong-dirichlet/flower/main.py:37-41), assembled into CSR
by the quadrature kernels of csrc/assemble_pk.cu; on quadrilaterals Q1 trial-test spaces with a Q1 / Q2 level set
(csrc/assemble_quad.cu, the same C entry points).

    V, Vphi = fem.functionspace(mesh, 2), fem.functionspace(mesh, 2)
    plan = assemble.build_plan(mesh, cells_tags, facets_tags, ds_bdy(100), V=V, V_phi=Vphi)
    A, b = assemble.assemble_strong_dirichlet(plan, phi_h, f_h, stab_coef=1.0)

Symbolic phase (torch sort/unique on the mesh's device): CSR pattern = all dof pairs of every cell tagged
1/2 plus all pairs among the dofs of the two cells of every interior facet tagged 2/3 (dolfinx
create_sparsity_pattern [dep-knowledge, SURVEY.md C.3]); entity -> CSR-slot maps stored so that consecutive threads
read consecutive words: entry-major ([nd*nd, n_cells]) for the cell kernel (one thread per cell), entity-major
([n, nd*nd]) for the facet kernels (the threads of one entity work on its rows).
"""
import ctypes

import torch

from . import _lib, quadrature


class PkAssemblyPlan:
    method = "pk-atomic"
    rowsplan = None
    blocked = None

    def __init__(self, mesh, cell_tags8, facet_tags8, entities, V, V_phi, form="strong", ghost_tag=None):
        """form = "strong": strong-Dirichlet operator on V; form = "weak": weak-Dirichlet (dual) operator on
        the mixed space V x V, u at scalar dof s numbered 2 s, p numbered 2 s + 1 (cell-local order
        [u dofs, p dofs])."""
        if form not in ("strong", "weak", "neumann"):
            raise ValueError("form must be 'strong', 'weak' or 'neumann'")
        if form == "neumann" and V.degree != 1:
            raise NotImplementedError("the Neumann operator is implemented for P1 u and y (main.py:37-39)")
        self.form = form
        if mesh.cell_type == "quadrilateral":
            # bilinear cell map: the Neumann and strong-Dirichlet kernels of csrc/assemble_quad.cu (the latter for a Q1
            # trial / test space); the weak form is not implemented there
            if form == "weak":
                raise NotImplementedError("the weak-Dirichlet operator is not implemented on quadrilaterals")
            if form == "strong" and V.degree != 1:
                raise NotImplementedError("the strong-Dirichlet operator on quadrilaterals implements a Q1 trial "
                                          "space only")
        elif mesh.cell_type not in ("triangle", "tetrahedron"):
            raise NotImplementedError("P_k assembly supports triangles and tetrahedra")
        for sp in (V, V_phi):
            if sp.mesh is not mesh:
                raise ValueError("the function space is defined on another mesh")
            if sp.degree not in (1, 2):
                raise NotImplementedError("the CUDA assembly path implements Lagrange degrees 1 and 2")
        dev = mesh.device
        self.mesh, self.V, self.V_phi = mesh, V, V_phi
        self.cell_tags8 = cell_tags8
        self.dofmap = V.dofmap_dev
        self.dofmap_phi = V_phi.dofmap_dev
        self.nd = int(self.dofmap.shape[1])
        if form == "weak":
            self.pattern_dofmap = torch.cat([2 * self.dofmap, 2 * self.dofmap + 1], dim=1).contiguous()
            self.n_rows = n = 2 * int(V.num_dofs)
        elif form == "neumann":
            # mixed space (u, y, p) in P1 x P1^d x DG0 (Q1 x Q1^2 x DG0 on quadrilaterals): u at vertex s -> (d+1) s,
            # y_c -> (d+1) s + 1 + c, p of cell k -> (d+1) Nv + k; cell-local order [u, y node-major, p]
            d_, nvx = mesh.gdim, mesh.num_vertices
            c = mesh.cells.long()
            y = ((d_ + 1) * c[:, :, None] + 1 + torch.arange(d_, device=dev)[None, None, :]).reshape(c.shape[0], -1)
            pcol = (d_ + 1) * nvx + torch.arange(mesh.num_cells, device=dev)[:, None]
            self.pattern_dofmap = torch.cat([(d_ + 1) * c, y, pcol], dim=1).to(torch.int32).contiguous()
            self.n_rows = n = (d_ + 1) * nvx + mesh.num_cells
        else:
            self.pattern_dofmap = self.dofmap
            self.n_rows = n = int(V.num_dofs)
        nd = int(self.pattern_dofmap.shape[1])       # dofs per cell of the assembled (possibly mixed) space
        self.active = torch.nonzero((cell_tags8 == 1) | (cell_tags8 == 2)).reshape(-1).to(torch.int32)
        # positions in `active` of the cut cells (the Neumann kernels integrate them apart from the interior cells)
        self.cut_positions = torch.nonzero(cell_tags8[self.active.long()] == 2).reshape(-1).to(torch.int32)
        interior = mesh.f2c[:, 1] >= 0
        if form == "neumann":      # dS(3) for the Neumann demo, dS(2) for the Robin demo
            gmask = facet_tags8 == (3 if ghost_tag is None else int(ghost_tag))
        else:
            gmask = (facet_tags8 == 2) | (facet_tags8 == 3)
        self.ghost = torch.nonzero(gmask & interior).reshape(-1).to(torch.int32)   # dS(3) resp. dS((2,3))
        self.entities = entities.reshape(-1, 2).to(torch.int32).contiguous()

        def pair_keys(dm):  # [m, k] dofs -> [m, k*k] keys row*n+col, row-major (row = test)
            return (dm[:, :, None] * n + dm[:, None, :]).reshape(dm.shape[0], dm.shape[1] * dm.shape[1])

        pdm = self.pattern_dofmap
        keys_c = pair_keys(pdm[self.active.long()].long())
        g = self.ghost.long()
        mac = torch.cat([pdm[mesh.f2c[g, 0].long()], pdm[mesh.f2c[g, 1].long()]], dim=1).long()
        keys_g = pair_keys(mac)
        n_c = keys_c.numel()
        uniq, inv = torch.unique(torch.cat([keys_c.reshape(-1), keys_g.reshape(-1)]), sorted=True,
                                 return_inverse=True)
        del keys_c, keys_g
        inv = inv.to(torch.int32)
        self.slots_cells = inv[:n_c].reshape(-1, nd * nd).t().contiguous()
        # cells: entry-major (one thread per cell); facets / entities: entity-major (the threads of one entity read
        # consecutive words)
        self.slots_ghost = inv[n_c:].reshape(-1, 4 * nd * nd).contiguous()
        del inv
        keys_b = pair_keys(pdm[self.entities[:, 0].long()].long())
        self.slots_boundary = torch.searchsorted(uniq, keys_b.reshape(-1)).reshape(-1, nd * nd) \
            .to(torch.int32).contiguous()
        rows = uniq // n
        self.indices = (uniq - rows * n).to(torch.int32).contiguous()
        counts = torch.bincount(rows, minlength=n)
        indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        indptr[1:] = torch.cumsum(counts, dim=0)
        self.indptr = indptr.to(torch.int32).contiguous()
        self.nnz = int(uniq.numel())
        if self.nnz >= 2 ** 31:
            raise NotImplementedError("CSR pattern with %d entries: indptr / slot maps are int32" % self.nnz)

        # quadrature tables and C structs (kept alive with the plan)
        d = mesh.gdim
        if form == "neumann" and mesh.cell_type == "quadrilateral":
            (cl, cw), (fl, fw) = quadrature.rules_for_neumann_quad(V_phi.degree)   # cell points: (xi, eta)
        elif mesh.cell_type == "quadrilateral":
            (cl, cw), (fl, fw) = quadrature.rules_for_strong_quad(V_phi.degree)
        elif form == "neumann":
            (cl, cw), (fl, fw) = quadrature.rules_for_neumann(d, V_phi.degree)
        else:
            rules = quadrature.rules_for_weak if form == "weak" else quadrature.rules_for
            (cl, cw), (fl, fw) = rules(d, V.degree, V_phi.degree)
        f64 = dict(dtype=torch.float64, device=dev)
        self._q = [torch.as_tensor(a, **f64).contiguous() for a in (cl, cw, fl, fw)]
        self.n_cell_points, self.n_facet_points = len(cw), len(fw)
        self._cquad = self._cw = self._cp = None

    def c_structs(self):
        if self._cquad is None:
            p = _lib.ptr
            q = self._q
            self._cquad = _lib.CQuadrature(self.n_cell_points, self.n_facet_points, p(q[0]), p(q[1]), p(q[2]),
                                           p(q[3]))
            self._cw = _lib.CPkSpace(self.V.degree, self.nd, self.V.num_dofs, p(self.dofmap))
            self._cp = _lib.CPkSpace(self.V_phi.degree, int(self.dofmap_phi.shape[1]), self.V_phi.num_dofs,
                                     p(self.dofmap_phi))
        return self._cw, self._cp, self._cquad

    def new_outputs(self):
        dev = self.mesh.device
        return (torch.zeros(self.nnz, dtype=torch.float64, device=dev),
                torch.zeros(self.n_rows, dtype=torch.float64, device=dev))


def assemble_pk_into(plan, phi, f, sigma, data, b, marks=None):
    """Numeric phase on the current stream: zero `data` / `b`, then the cell, one-sided and ghost-penalty
    kernels.  All arguments are device tensors; nothing synchronises."""
    marks = marks or (lambda: None)
    mesh = plan.mesh
    _lib.require_cuda(mesh)
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    cw, cp, cq = plan.c_structs()
    head = (cm, ctypes.byref(cw), ctypes.byref(cp), ctypes.byref(cq))
    st = _lib.stream()
    data.zero_()
    b.zero_()
    marks()
    _lib.check(lib.phifem_assemble_cells_pk(
        *head, _lib.ptr(phi), _lib.ptr(f), _lib.ptr(plan.cell_tags8), _lib.ptr(plan.active),
        plan.active.numel(), _lib.ptr(plan.slots_cells), float(sigma), _lib.ptr(data), _lib.ptr(b), st))
    marks()
    _lib.check(lib.phifem_assemble_boundary_pk(
        *head, _lib.ptr(phi), _lib.ptr(plan.entities), plan.entities.shape[0],
        _lib.ptr(plan.slots_boundary), _lib.ptr(data), st))
    marks()
    _lib.check(lib.phifem_assemble_ghost_pk(
        *head, _lib.ptr(phi), _lib.ptr(plan.ghost), plan.ghost.numel(), _lib.ptr(plan.slots_ghost),
        float(sigma), _lib.ptr(data), st))
    marks()
    return data, b


def assemble_weak_into(plan, phi, f, u_d, gamma, sigma, data, b):
    """Numeric phase of the weak-Dirichlet operator (plan.form == "weak") on the current stream."""
    mesh = plan.mesh
    _lib.require_cuda(mesh)
    if plan.form != "weak":
        raise ValueError("the plan was built for the strong-Dirichlet operator")
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    cw, cp, cq = plan.c_structs()
    st = _lib.stream()
    data.zero_()
    b.zero_()
    _lib.check(lib.phifem_assemble_weak_cells_pk(
        cm, ctypes.byref(cw), ctypes.byref(cp), ctypes.byref(cq), _lib.ptr(phi), _lib.ptr(f), _lib.ptr(u_d),
        _lib.ptr(plan.cell_tags8), _lib.ptr(plan.active), plan.active.numel(), _lib.ptr(plan.slots_cells),
        _lib.ptr(plan.pattern_dofmap), float(gamma), float(sigma), _lib.ptr(data), _lib.ptr(b), st))
    _lib.check(lib.phifem_assemble_weak_boundary_pk(
        cm, ctypes.byref(cw), ctypes.byref(cq), _lib.ptr(plan.entities), plan.entities.shape[0],
        _lib.ptr(plan.slots_boundary), _lib.ptr(data), st))
    _lib.check(lib.phifem_assemble_weak_ghost_pk(
        cm, ctypes.byref(cw), ctypes.byref(cq), _lib.ptr(plan.ghost), plan.ghost.numel(),
        _lib.ptr(plan.slots_ghost), float(sigma), _lib.ptr(data), st))
    return data, b


def assemble_neumann_into(plan, phi, f, u_n, gamma, sigma, data, b, robin_coef=0.0):
    """Numeric phase of the Neumann operator (plan.form == "neumann") on the current stream."""
    mesh = plan.mesh
    _lib.require_cuda(mesh)
    if plan.form != "neumann":
        raise ValueError("the plan was not built by build_plan_neumann")
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    _, cp, cq = plan.c_structs()
    st = _lib.stream()
    data.zero_()
    b.zero_()
    _lib.check(lib.phifem_assemble_neumann_cells(
        cm, ctypes.byref(cp), ctypes.byref(cq), _lib.ptr(phi), _lib.ptr(f), _lib.ptr(u_n),
        _lib.ptr(plan.cell_tags8), _lib.ptr(plan.active), plan.active.numel(), _lib.ptr(plan.cut_positions),
        plan.cut_positions.numel(), _lib.ptr(plan.slots_cells), _lib.ptr(plan.pattern_dofmap), float(gamma),
        float(robin_coef), _lib.ptr(data), _lib.ptr(b), st))
    _lib.check(lib.phifem_assemble_neumann_boundary(
        cm, _lib.ptr(plan.entities), plan.entities.shape[0], _lib.ptr(plan.slots_boundary), _lib.ptr(data), st))
    _lib.check(lib.phifem_assemble_neumann_ghost(
        cm, ctypes.byref(cq), _lib.ptr(plan.ghost), plan.ghost.numel(), _lib.ptr(plan.slots_ghost), float(sigma),
        _lib.ptr(data), st))
    return data, b
