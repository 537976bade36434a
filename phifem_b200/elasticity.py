"""Interface-elasticity phi-FEM operator (reference demo/interface-elasticity/main.py:107-274, BASELINE.json configs[3])
assembled into CSR by the kernels of csrc/assemble_elasticity.cu.

    cells_tags, facets_tags, _, d_bdry, _ = compute_tags_measures(mesh, levelset, 1, box_mode=True)
    plan = elasticity.build_plan_interface_elasticity(mesh, cells_tags, facets_tags, d_bdry)
    bc_dofs = plan.dofs("u_in", plan.boundary_vertices())                       # main.py:160-179
    A, b = elasticity.assemble_interface_elasticity(plan, phi_h, f_h, Material(), pen_coef=1.0, stab_coef=1.0,
                                                    bcs=(bc_dofs, u_exact_at_those_dofs))
    u_in, u_out, y_in, y_out, p = plan.split(x)

Mixed space (`mixd_element`, main.py:127-129): (u_in, u_out, y_in, y_out, p), every field nodal P1, NB = 3 d + 2 d^2 dofs
per vertex, global dof = NB vertex + o with o: u_in c -> c, u_out c -> d + c, y_in (r, s) -> 2 d + r d + s,
y_out (r, s) -> 2 d + d^2 + r d + s, p c -> 2 d + 2 d^2 + c (our numbering; dolfinx's is an implementation detail of its
dofmap builder).  Sparsity (dolfinx create_sparsity_pattern [dep-knowledge, SURVEY.md C.3]): all dof pairs of every cell
of dx((1,2)) u dx((2,3)) u dx(2) -- every tagged cell -- and all pairs among the dofs of the two cells of every interior
facet of dS(3) u dS(4); with nodal fields that is the vertex graph with dense NB x NB blocks, which is how the kernels
address it (one scalar slot map).  Symbolic phase = torch sort/unique on the mesh's device.

On quadrilaterals every field is Q1 on the bilinear cell (NB = 14, the same numbering) with a Q1 or Q2 level set; the
integrals follow the rules of `quadrature.rules_for_elasticity_quad`.
"""
import ctypes

import numpy as np
import torch

from . import _lib, quadrature
from .assemble import CSRMatrix, _device_vector, _plan_inputs, refuse_hexahedra

FIELDS = ("u_in", "u_out", "y_in", "y_out", "p")


class Material:
    """E / nu of both materials (data.py:13-22), their Lame coefficients (data.py:5-10) and the penalty weights
    (main.py:189-190)."""

    def __init__(self, E_in=1.0, nu_in=0.3, E_out=0.001, nu_out=0.3):
        self.E_in, self.nu_in, self.E_out, self.nu_out = E_in, nu_in, E_out, nu_out
        self.lmbda_in, self.mu_in = E_in * nu_in / (1.0 + nu_in) / (1.0 - 2.0 * nu_in), E_in / 2.0 / (1.0 + nu_in)
        self.lmbda_out = E_out * nu_out / (1.0 + nu_out) / (1.0 - 2.0 * nu_out)
        self.mu_out = E_out / 2.0 / (1.0 + nu_out)
        self.coef_in = (E_in / (E_in + E_out)) ** 2
        self.coef_out = (E_out / (E_in + E_out)) ** 2


def field_layout(d):
    """offset and number of components of each field inside a vertex block; block size."""
    sizes = (d, d, d * d, d * d, d)
    off, lay = 0, {}
    for name, s in zip(FIELDS, sizes):
        lay[name] = (off, s)
        off += s
    return lay, off


class ElasticityPlan:
    form = "interface-elasticity"

    def __init__(self, mesh, cell_tags8, facet_tags8, ents_in, ents_out, V_phi):
        refuse_hexahedra(mesh, "ElasticityPlan")
        if mesh.cell_type not in ("triangle", "tetrahedron", "quadrilateral"):
            raise NotImplementedError("the interface-elasticity operator supports triangles, quadrilaterals and "
                                      "tetrahedra")
        if V_phi.mesh is not mesh:
            raise ValueError("the level-set space is defined on another mesh")
        if V_phi.degree not in (1, 2):
            raise NotImplementedError("the CUDA assembly path implements level sets of degree 1 and 2")
        dev = mesh.device
        self.mesh, self.V_phi = mesh, V_phi
        self.cell_tags8 = cell_tags8
        d = mesh.gdim
        self.layout, self.nb = field_layout(d)
        nb, nvx = self.nb, mesh.num_vertices
        self.n_rows = nb * nvx
        cells = mesh.cells.long()
        tagged = (cell_tags8 >= 1) & (cell_tags8 <= 3)
        self.cut_cells = torch.nonzero(cell_tags8 == 2).reshape(-1).to(torch.int32)                   # dx(2)
        interior = mesh.f2c[:, 1] >= 0
        self.facets_in = torch.nonzero((facet_tags8 == 3) & interior).reshape(-1).to(torch.int32)     # dS(3)
        self.facets_out = torch.nonzero((facet_tags8 == 4) & interior).reshape(-1).to(torch.int32)    # dS(4)
        self.entities_in = ents_in.reshape(-1, 2).to(torch.int32).contiguous()                        # ds(100)
        self.entities_out = ents_out.reshape(-1, 2).to(torch.int32).contiguous()                      # ds(101)

        def pair_keys(vs):   # [m, k] vertices -> [m, k*k] keys row * Nv + col (row = test vertex)
            return (vs[:, :, None] * nvx + vs[:, None, :]).reshape(vs.shape[0], vs.shape[1] * vs.shape[1])

        def macro(facets):
            g = facets.long()
            return torch.cat([cells[mesh.f2c[g, 0].long()], cells[mesh.f2c[g, 1].long()]], dim=1)

        keys_c = pair_keys(cells)
        keys_fi, keys_fo = pair_keys(macro(self.facets_in)), pair_keys(macro(self.facets_out))
        uniq = torch.unique(torch.cat([keys_c[tagged].reshape(-1), keys_fi.reshape(-1), keys_fo.reshape(-1)]),
                            sorted=True)
        rows = uniq // nvx
        vcols = uniq - rows * nvx
        vptr = torch.zeros(nvx + 1, dtype=torch.int64, device=dev)
        vptr[1:] = torch.cumsum(torch.bincount(rows, minlength=nvx), dim=0)
        nnz_v = int(uniq.numel())
        self.nnz = nb * nb * nnz_v
        if self.nnz >= 2 ** 31:
            raise NotImplementedError("CSR pattern with %d entries: indptr is int32" % self.nnz)

        def positions(keys, valid=None):   # rank of the column vertex among the row vertex's neighbours
            flat = keys.reshape(-1)
            at = torch.searchsorted(uniq, flat).clamp_(max=max(nnz_v - 1, 0))
            pos = at - vptr[flat // nvx]
            if valid is not None:
                pos = torch.where(valid.repeat_interleave(keys.shape[1]), pos, torch.zeros_like(pos))
            return pos.reshape(keys.shape).to(torch.int32).contiguous()

        self.pos_cells = positions(keys_c, tagged)
        self.pos_facets_in, self.pos_facets_out = positions(keys_fi), positions(keys_fo)
        self.pos_entities_in = positions(pair_keys(cells[self.entities_in[:, 0].long()]))
        self.pos_entities_out = positions(pair_keys(cells[self.entities_out[:, 0].long()]))
        self.vptr = vptr.to(torch.int32).contiguous()

        # CSR arrays of the blocked matrix: row NB r + a starts at NB (NB vptr[r] + a deg(r))
        deg = vptr[1:] - vptr[:-1]
        ar = torch.arange(nb, device=dev)
        indptr = torch.empty(self.n_rows + 1, dtype=torch.int64, device=dev)
        indptr[:-1] = (nb * (nb * vptr[:-1, None] + ar[None, :] * deg[:, None])).reshape(-1)
        indptr[-1] = self.nnz
        self.indptr = indptr.to(torch.int32).contiguous()
        indices = torch.empty(self.nnz, dtype=torch.int32, device=dev)
        chunk = max(1, (1 << 24) // (nb * nb))
        pos_e = torch.arange(nnz_v, device=dev) - vptr[rows]
        for s in range(0, nnz_v, chunk):
            r, c, p = rows[s:s + chunk], vcols[s:s + chunk], pos_e[s:s + chunk]
            addr = (nb * (nb * vptr[r] + p))[:, None, None] + (nb * deg[r])[:, None, None] * ar[None, :, None] \
                + ar[None, None, :]
            val = (nb * c)[:, None, None] + ar[None, None, :]
            indices[addr.reshape(-1)] = val.expand(-1, nb, -1).reshape(-1).to(torch.int32)
        self.indices = indices

        if mesh.cell_type == "quadrilateral":   # the cut-cell rule; the other rules are constants of the kernels
            (cl, cw), _, _ = quadrature.rules_for_elasticity_quad(V_phi.degree)
        else:
            (cl, cw), _ = quadrature.rules_for_neumann(d, V_phi.degree)   # degree 2 (kphi + 1): (lambda phi)^2
        f64 = dict(dtype=torch.float64, device=dev)
        self._q = [torch.as_tensor(a, **f64).contiguous() for a in (cl, cw)]
        self.n_cell_points = len(cw)
        self._c = None

    # ---- dof helpers -------------------------------------------------------------------------------------------
    def dofs(self, field, vertices=None):
        """Global dofs [n, ncomp] of `field` at `vertices` (default: all)."""
        off, size = self.layout[field]
        v = torch.arange(self.mesh.num_vertices, device=self.mesh.device) if vertices is None \
            else torch.as_tensor(vertices, device=self.mesh.device).long()
        return self.nb * v[:, None] + off + torch.arange(size, device=self.mesh.device)[None, :]

    def boundary_vertices(self):
        """Vertices of the mesh-boundary facets (what `locate_entities_boundary` + `locate_dofs_topological` reach,
        main.py:160-176, when the marker selects the whole boundary of the box)."""
        fv = self.mesh.facet_vertices[self.mesh.boundary_facets.long()]
        return torch.unique(fv.reshape(-1).long())

    def split(self, x):
        """(u_in [Nv, d], u_out [Nv, d], y_in [Nv, d, d], y_out [Nv, d, d], p [Nv, d]) views of a mixed vector."""
        d = self.mesh.gdim
        X = x.reshape(self.mesh.num_vertices, self.nb)
        out = []
        for name in FIELDS:
            off, size = self.layout[name]
            blk = X[:, off:off + size]
            out.append(blk.reshape(-1, d, d) if size == d * d else blk)
        return tuple(out)

    def c_structs(self):
        if self._c is None:
            p = _lib.ptr
            dm = self.V_phi.dofmap_dev
            self._c = (_lib.CPkSpace(self.V_phi.degree, int(dm.shape[1]), self.V_phi.num_dofs, p(dm)),
                       _lib.CQuadrature(self.n_cell_points, 0, p(self._q[0]), p(self._q[1]), None, None))
        return self._c

    def new_outputs(self):
        dev = self.mesh.device
        return (torch.zeros(self.nnz, dtype=torch.float64, device=dev),
                torch.zeros(self.n_rows, dtype=torch.float64, device=dev))


def build_plan_interface_elasticity(mesh, cells_tags, facets_tags, d_bdry, V_phi=None):
    """Symbolic phase for `a` and `L` of the interface-elasticity demo.  `d_bdry` = the measure returned by
    compute_tags_measures(box_mode=True) (ids 100 and 101 are both used, main.py:235-236) or a pair of flat entity
    arrays (ds100, ds101).  `V_phi`: the level-set space (main.py:134-135; default P1)."""
    from . import fem
    from .mesh import Measure
    V_phi = fem.functionspace(mesh, 1) if V_phi is None else V_phi
    if isinstance(d_bdry, Measure):
        d100, d101 = d_bdry(100), d_bdry(101)
    else:
        d100, d101 = d_bdry
    c8, f8, e_in = _plan_inputs(mesh, cells_tags, facets_tags, d100)
    _, _, e_out = _plan_inputs(mesh, cells_tags, facets_tags, d101)
    return ElasticityPlan(mesh, c8, f8, e_in, e_out, V_phi)


def assemble_interface_elasticity_into(plan, phi, f, material, gamma, sigma_s, data, b, bc_marker=None,
                                       bc_values=None, bc_dofs=None):
    """Numeric phase on the current stream: zero `data` / `b`, cells, interface facets, one-sided entities, Dirichlet
    conditions.  All arguments are device tensors; nothing synchronises."""
    mesh = plan.mesh
    _lib.require_cuda(mesh)
    lib = _lib.load()
    cm = _lib.c_mesh(mesh)
    cp, cq = plan.c_structs()
    prm = _lib.CElasticityParams(material.lmbda_in, material.mu_in, material.lmbda_out, material.mu_out,
                                 material.coef_in, material.coef_out, float(gamma), float(sigma_s))
    st = _lib.stream()
    p = _lib.ptr
    data.zero_()
    b.zero_()
    _lib.check(lib.phifem_assemble_elasticity_cells(
        cm, ctypes.byref(cp), ctypes.byref(cq), p(phi), p(f), p(plan.cell_tags8), p(plan.cut_cells),
        plan.cut_cells.numel(), p(plan.vptr), p(plan.pos_cells), ctypes.byref(prm), p(data), p(b), st))
    for side, (fac, pos) in enumerate(((plan.facets_in, plan.pos_facets_in), (plan.facets_out, plan.pos_facets_out))):
        _lib.check(lib.phifem_assemble_elasticity_facets(cm, p(fac), fac.numel(), p(plan.vptr), p(pos), side,
                                                         ctypes.byref(prm), p(data), st))
    for side, (ent, pos) in enumerate(((plan.entities_in, plan.pos_entities_in),
                                       (plan.entities_out, plan.pos_entities_out))):
        _lib.check(lib.phifem_assemble_elasticity_boundary(cm, p(ent), ent.shape[0], p(plan.vptr), p(pos), side,
                                                           p(data), st))
    if bc_marker is not None and bc_dofs is not None:   # the pattern is structurally symmetric: list-driven variant
        _lib.check(lib.phifem_apply_dirichlet_symmetric(plan.n_rows, p(plan.indptr), p(plan.indices), p(bc_dofs),
                                                        bc_dofs.numel(), p(bc_marker), p(bc_values), p(data), p(b), st))
    elif bc_marker is not None:
        _lib.check(lib.phifem_apply_dirichlet(plan.n_rows, p(plan.indptr), p(plan.indices), p(bc_marker),
                                              p(bc_values), p(data), p(b), st))
    return data, b


def assemble_interface_elasticity(plan, phi_h, f_h, material=None, pen_coef=1.0, stab_coef=1.0, bcs=None,
                                  symmetric_bc=True):
    """A (CSR over the mixed dofs) and b of main.py:227-275.  `f_h`: P1 vector field [Nv, d] (the demo's `f` is a UFL
    expression, :150; here its nodal interpolant).  `bcs` = (dofs, values): Dirichlet conditions as dolfinx applies them
    (assemble_matrix(bcs=) zeroes rows / columns and sets the diagonal to 1, apply_lifting, bc.set).  symmetric_bc
    (default): the list-driven pass, whose work is the constrained rows' lengths -- the plan's pattern is structurally
    symmetric with sorted rows by construction; False = the pass over the whole matrix (bitwise reproducible lifting)."""
    mesh = plan.mesh
    _lib.require_cuda(mesh)
    material = material or Material()
    phi = _device_vector(mesh, phi_h, plan.V_phi)
    f = f_h if torch.is_tensor(f_h) else torch.from_numpy(np.ascontiguousarray(f_h, dtype=np.float64))
    f = f.to(mesh.device, dtype=torch.float64).contiguous()
    if tuple(f.shape) != (mesh.num_vertices, mesh.gdim):
        raise ValueError("f_h must hold one vector per vertex: expected shape (%d, %d)" % (mesh.num_vertices, mesh.gdim))
    marker = values = bc_list = None
    if bcs is not None:
        dofs = torch.as_tensor(bcs[0], device=mesh.device).reshape(-1).long()
        vals = torch.as_tensor(bcs[1], device=mesh.device, dtype=torch.float64).reshape(-1)
        if dofs.numel() != vals.numel():
            raise ValueError("bcs: %d dofs but %d values" % (dofs.numel(), vals.numel()))
        marker = torch.zeros(plan.n_rows, dtype=torch.int8, device=mesh.device)
        values = torch.zeros(plan.n_rows, dtype=torch.float64, device=mesh.device)
        marker[dofs] = 1
        values[dofs] = vals
        if symmetric_bc:   # list-driven Dirichlet pass (phifem_apply_dirichlet_symmetric) instead of the full-matrix one
            bc_list = torch.unique(dofs).to(torch.int32).contiguous()
    data, b = plan.new_outputs()
    assemble_interface_elasticity_into(plan, phi, f, material, pen_coef, stab_coef, data, b, marker, values, bc_list)
    return CSRMatrix(plan.indptr, plan.indices, data, (plan.n_rows, plan.n_rows)), b
