"""Assembly of the strong-Dirichlet phi-FEM operator into CSR on the GPU.

What the reference demo does with UFL + `dolfinx.fem.petsc.assemble_matrix / assemble_vector`
(reference demo/strong-dirichlet/flower/main.py:92-131), for P1 on triangles and tetrahedra:

    plan = build_plan(mesh, cells_tags, facets_tags, ds_bdy(100))          # symbolic, per tag set
    A, b = assemble_strong_dirichlet(plan, phi_h, f_h, stab_coef=1.0)      # numeric, hot path

Symbolic phase (sort/unique plumbing, torch ops on the device): CSR pattern = union over the
integral domains -- all vertex pairs of every cell tagged 1/2, all pairs among the two cells of
every interior facet tagged 2/3 -- with structural zeros kept and rows without contributions
empty (dolfinx create_sparsity_pattern [dep-knowledge, SURVEY.md C.3]); plus the entity ->
CSR-slot maps the kernels scatter through.  Numeric phase: three hand-written kernels
(csrc/assemble.cu) adding into zeroed `data` / `b`.
"""
import numpy as np
import torch

from . import _lib
from .fem import Function
from .mesh import Measure


class CSRMatrix:
    """Assembled operator: `indptr` int32 [n+1], `indices` int32 [nnz], `data` float64 [nnz] on the
    device; `.to_scipy()` copies to the host."""

    def __init__(self, indptr, indices, data, shape):
        self.indptr, self.indices, self.data, self.shape = indptr, indices, data, shape

    def to_scipy(self):
        import scipy.sparse as sp
        return sp.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(),
                              self.indptr.cpu().numpy()), shape=self.shape)


def ghost_macro_vertices(mesh, facets):
    """[n, nv+1] distinct vertices of the macro element of interior facets, in the order the ghost-penalty
    kernel emits its tensor: facet vertices as ordered in cell + (= f2c[f][0]), opposite vertex of cell +,
    opposite vertex of cell -."""
    g = facets.long()
    nv = mesh.cells.shape[1]
    out = []
    for side in (0, 1):
        c = mesh.f2c[g, side].long()
        cv = mesh.cells[c].long()
        lf = (mesh.c2f[c].long() == g[:, None]).long().argmax(dim=1)
        if side == 0:
            keep = torch.arange(nv, device=g.device)[None, :] != lf[:, None]
            out.append(cv[keep].reshape(-1, nv - 1))
        out.append(cv.gather(1, lf[:, None]))
    return torch.cat(out, dim=1)


class AssemblyPlan:
    """Tag-dependent symbolic data of one operator (reused for every assembly with the same tags).

    method = "rows"   : row-gather kernel, one thread per CSR row (the default: no atomics, no zero-fill,
    bitwise reproducible; phifem_b200/rows.py); falls back to "atomic" when a row holds more than 200
    entries;
    method = "atomic" : one thread per entity, fp64 reductions through the entity -> CSR-slot maps;
    method = "blocked": owner-computes CTA per row block with a shared-memory segmented reduction
    (phifem_b200/blocked.py); falls back to "atomic" when a single row gathers more contributions than a
    shared-memory block can hold."""

    def __init__(self, mesh, cell_tags8, facet_tags8, entities, method="rows", capacity=None,
                 order="auto", row_mask=None, geometry=False, cell_pass="rows", rows_per_tile=256, symbolic="auto"):
        """symbolic: "torch" = sort / unique passes with torch ops (any device: the CPU tests); "native" = the device
        builder behind the C ABI (csrc/rows_plan.cu: same arrays, bit for bit, from the vertex -> cell adjacency);
        "auto" = native for a row-gather plan on a CUDA mesh, torch otherwise."""
        if mesh.cell_type not in ("triangle", "tetrahedron"):
            raise NotImplementedError("P1 assembly supports triangles and tetrahedra")
        dev = mesh.device
        self.mesh = mesh
        self.cell_tags8 = cell_tags8
        # what the plan depends on, kept as copies (the caller may rewrite its tag arrays in place): `matches`
        self._sig_cells = cell_tags8.clone()
        self._sig_facets = _facet_classes(facet_tags8)
        n = mesh.num_vertices
        nv = mesh.cells.shape[1]
        self.n_rows = n
        ents2 = entities.reshape(-1, 2)
        if ents2.shape[0]:
            # a one-sided entity must lie in a cell of dx((1,2)): its dof pairs are looked up in the pattern of those
            # cells, and an entity of ds(101) or of another tag set would silently land in a neighbouring CSR slot
            t = cell_tags8[ents2[:, 0].long()]
            if not bool(((t == 1) | (t == 2)).all()):
                raise ValueError("a (cell, local facet) entity names a cell that is not tagged 1 or 2: the strong-/weak-"
                                 "Dirichlet plans take the entities of ds(100) (Gamma_h seen from Omega_h)")
        if symbolic not in ("auto", "torch", "native"):
            raise ValueError("symbolic must be 'auto', 'torch' or 'native'")
        native_ok = (method == "rows" and cell_pass == "rows" and not geometry and dev.type == "cuda")
        if symbolic == "native" and not native_ok:
            raise ValueError("the native symbolic phase builds row-gather plans (method='rows', cell_pass='rows') on "
                             "CUDA meshes")
        self._slots = None
        if native_ok and symbolic in ("auto", "native"):
            from . import rows as rows_mod
            try:
                if order == "auto":
                    order = "natural"
                rp = rows_mod.NativeRowsPlan(mesh, cell_tags8, facet_tags8, entities, order=order, row_mask=row_mask)
            except NotImplementedError:
                if symbolic == "native":
                    raise
                rp = None                      # e.g. a row longer than 255 entries: the torch path decides
            if rp is not None:
                self.entities = entities.reshape(-1, 2).to(torch.int32).contiguous()
                self.active, self.ghost, self.indptr, self.indices, self.nnz = rp.active, rp.ghost, rp.indptr, \
                    rp.indices, rp.nnz
                self.blocked, self.rowsplan, self.method, self.symbolic = None, rp, "rows", "native"
                return
        self.symbolic = "torch"
        self.active = torch.nonzero((cell_tags8 == 1) | (cell_tags8 == 2)).reshape(-1).to(torch.int32)
        interior = mesh.f2c[:, 1] >= 0
        self.ghost = torch.nonzero(((facet_tags8 == 2) | (facet_tags8 == 3)) & interior) \
            .reshape(-1).to(torch.int32)
        self.entities = entities.reshape(-1, 2).to(torch.int32).contiguous()

        def pair_keys(dm):  # [m, k] dofs -> [m, k*k] keys row*n+col, row-major (row = test)
            return (dm[:, :, None] * n + dm[:, None, :]).reshape(dm.shape[0], dm.shape[1] * dm.shape[1])

        dm = mesh.cells[self.active.long()].long()
        keys_c = pair_keys(dm)
        mac = ghost_macro_vertices(mesh, self.ghost)
        keys_g = pair_keys(mac)
        n_c = keys_c.numel()
        uniq, inv = torch.unique(torch.cat([keys_c.reshape(-1), keys_g.reshape(-1)]), sorted=True,
                                 return_inverse=True)
        del keys_c, keys_g
        slots_cells = inv[:n_c].reshape(-1, nv * nv).to(torch.int32).contiguous()
        slots_ghost = inv[n_c:].reshape(-1, (nv + 1) ** 2).to(torch.int32).contiguous()
        del inv
        keys_b = pair_keys(mesh.cells[self.entities[:, 0].long()].long())
        slots_boundary = torch.searchsorted(uniq, keys_b.reshape(-1)).reshape(-1, nv * nv) \
            .to(torch.int32).contiguous()
        self._slots = (slots_cells, slots_ghost, slots_boundary)
        rows = uniq // n
        self.indices = (uniq - rows * n).to(torch.int32).contiguous()
        counts = torch.bincount(rows, minlength=n)
        self.indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        self.indptr[1:] = torch.cumsum(counts, dim=0)
        self.indptr = self.indptr.to(torch.int32).contiguous()
        self.nnz = int(uniq.numel())
        if self.nnz >= 2 ** 31:
            raise NotImplementedError("CSR pattern with %d entries: indptr / slot maps are int32 (PETSc's default "
                                      "index width too); shard the mesh (phifem_b200/partition.py)" % self.nnz)
        self.blocked, self.rowsplan, self.method = None, None, "atomic"
        if method == "rows" and self.nnz > 0:
            from . import rows as rows_mod
            try:
                self.rowsplan = rows_mod.RowsPlan(self, order=order, row_mask=row_mask, geometry=geometry,
                                                  cell_pass=cell_pass, rows_per_tile=rows_per_tile)
                self.method = "rows"
            except NotImplementedError:
                self.rowsplan = None
        elif method == "blocked" and self.active.numel() > 0:
            from . import blocked
            try:
                self.blocked = blocked.BlockedPlan(self, capacity or blocked.DEFAULT_CAPACITY)
                self.method = "blocked"
            except NotImplementedError:
                self.blocked = None
        elif method not in ("rows", "blocked", "atomic"):
            raise ValueError("method must be 'rows', 'blocked' or 'atomic'")

    # entity -> CSR-slot maps of the per-entity (atomic) kernels and of the CPU arm: built with the torch pattern, or on
    # first use from a natively built pattern (position of the key row * n + col in the sorted key list)
    def _slot_maps(self):
        if self._slots is None:
            n, nv = self.n_rows, self.mesh.cells.shape[1]
            ip = self.indptr.long()
            rows = torch.repeat_interleave(torch.arange(n, device=self.mesh.device), ip[1:] - ip[:-1])
            keys = rows * n + self.indices.long()
            del rows

            def slots(dm):
                k = (dm[:, :, None] * n + dm[:, None, :]).reshape(-1)
                return torch.searchsorted(keys, k).reshape(dm.shape[0], -1).to(torch.int32).contiguous()
            cells = self.mesh.cells
            self._slots = (slots(cells[self.active.long()].long()), slots(ghost_macro_vertices(self.mesh, self.ghost)),
                           slots(cells[self.entities[:, 0].long()].long()))
        return self._slots

    slots_cells = property(lambda self: self._slot_maps()[0])
    slots_ghost = property(lambda self: self._slot_maps()[1])
    slots_boundary = property(lambda self: self._slot_maps()[2])

    def new_outputs(self):
        dev = self.mesh.device
        return (torch.zeros(self.nnz, dtype=torch.float64, device=dev),
                torch.zeros(self.n_rows, dtype=torch.float64, device=dev))

    def matches(self, cells_tags, facets_tags):
        """Is this plan (pattern, row lists, slot maps) still the plan of these tags?  True iff the cells of dx((1,2)),
        the cut cells dx(2), the ghost-penalty facets dS((2,3)) and Gamma_h (facet tag 4, hence ds(100)) are the ones
        the plan was built from -- what a moving-interface loop asks after every `compute_tags_measures` before it
        either reuses the plan or pays the re-plan (reference demos rebuild everything at every refinement step,
        demo/strong-dirichlet/flower/main.py:59-66,121-123).  Two passes over the tag bytes and one host
        synchronisation (CPU tensors, as in the host-logic tests: torch passes)."""
        c8, f8, _ = _plan_inputs(self.mesh, cells_tags, facets_tags, None)
        if c8.numel() != self._sig_cells.numel() or f8.numel() != self._sig_facets.numel():
            return False
        if c8.is_cuda:      # one fused pass behind the C ABI (csrc/capi.cu phifem_tags_match)
            bad = torch.empty(1, dtype=torch.int64, device=c8.device)
            _lib.check(_lib.load().phifem_tags_match(_lib.ptr(c8), _lib.ptr(self._sig_cells), c8.numel(), _lib.ptr(f8),
                                                     _lib.ptr(self._sig_facets), f8.numel(), _lib.ptr(bad), _lib.stream()))
            return int(bad.item()) == 0
        return bool(torch.equal(c8, self._sig_cells)) and bool(torch.equal(_facet_classes(f8), self._sig_facets))


def refuse_hexahedra(mesh, what):
    """Hexahedral meshes can be tagged (`compute_tags_measures`); no operator assembles on them yet."""
    if mesh.cell_type == "hexahedron":
        raise NotImplementedError("%s: no operator assembles on cell type 'hexahedron' (hexahedral meshes can be "
                                  "tagged only)" % what)


def _facet_classes(facet_tags8):
    """What a plan sees of a facet tag: 1 = ghost-penalty facet (tags 2 and 3 alike), 2 = Gamma_h (tag 4), 0 otherwise."""
    return ((facet_tags8 == 2) | (facet_tags8 == 3)).to(torch.int8) + 2 * (facet_tags8 == 4).to(torch.int8)


def _plan_inputs(mesh, cells_tags, facets_tags, ds):
    """int8 tag arrays and the [m, 2] entity list of `ds` on the mesh's device."""
    from .mesh_scripts import _narrow_tags   # values outside 0..6 (user tags) must not wrap into 1..6
    c8 = getattr(cells_tags, "tags8", None)
    c8 = c8 if c8 is not None else _narrow_tags(cells_tags.values_dev)
    f8 = getattr(facets_tags, "tags8", None)
    f8 = f8 if f8 is not None else _narrow_tags(facets_tags.values_dev)
    if ds is None:
        ents = torch.zeros(0, dtype=torch.int32, device=mesh.device)
    elif isinstance(ds, Measure) and ds.subdomain_data is None:
        # plain `ufl.Measure("ds", domain=submesh)` of the demos' "sub" mode (main.py:66-70): every exterior facet
        # of the mesh, seen from its only cell
        bf = mesh.boundary_facets.long()
        owner = mesh.f2c[bf, 0].long()
        lf = (mesh.c2f[owner].long() == bf[:, None]).long().argmax(dim=1)
        ents = torch.stack([owner, lf], dim=1).reshape(-1).to(torch.int32)
    elif hasattr(ds, "integration_entities_dev"):
        ents = ds.integration_entities_dev
    elif torch.is_tensor(ds):
        ents = ds.to(mesh.device)
    else:
        ents = torch.as_tensor(np.asarray(ds, dtype=np.int32), device=mesh.device)
    return c8.contiguous(), f8.contiguous(), ents


def build_plan(mesh, cells_tags, facets_tags, ds=None, method="rows", capacity=None, order="auto",
               V=None, V_phi=None, geometry=False, cell_pass="rows", rows_per_tile=256, symbolic="auto"):
    """Symbolic phase for `a` and `L` of the strong-Dirichlet demo.  `ds` is what the demo passes as
    `ds_bdy(100)` (main.py:64): a MeasureRestriction, a flat entity array, or None (no boundary term).
    `V` / `V_phi`: the demo's `primal_space` / `levelset_space` (main.py:74-75); omitted or both of degree 1
    => the closed-form P1 kernels, otherwise the quadrature kernels for P1 / P2 (phifem_b200/assemble_pk.py).
    A quadrilateral mesh always takes the quadrature kernels, with V defaulting to Q1 and V_phi to V (a Q1 trial space
    and a Q1 or Q2 level set); method "blocked" / "atomic", geometry, cell_pass != "rows" and symbolic="native" raise
    ValueError there.
    cell_pass (row-gather plans): "rows" = one evaluation per (row, cell) record, "tiles" = the cell-once pass of
    csrc/assemble_tiles.cu.  geometry (row-gather plans): tabulate the cells' geometry factors once per plan (phifem_b200/rows.py; an
    option kept for the record, slower than the default on the B200)."""
    refuse_hexahedra(mesh, "build_plan")
    c8, f8, ents = _plan_inputs(mesh, cells_tags, facets_tags, ds)
    if mesh.cell_type == "quadrilateral":
        # the quadrature kernels of csrc/assemble_quad.cu (PkAssemblyPlan); the row-gather options have no
        # quadrilateral implementation
        if method not in ("rows", "pk"):
            raise ValueError("method=%r: quadrilateral meshes are assembled by the quadrature kernels only" % method)
        if geometry or cell_pass != "rows" or symbolic == "native":
            raise ValueError("geometry, cell_pass and symbolic='native' are options of the row-gather plans, which "
                             "have no quadrilateral implementation")
        from . import fem
        from .assemble_pk import PkAssemblyPlan
        V = fem.functionspace(mesh, 1) if V is None else V
        V_phi = V if V_phi is None else V_phi
        return PkAssemblyPlan(mesh, c8, f8, ents, V, V_phi)
    V_phi = V if V_phi is None else V_phi
    V = V_phi if V is None else V
    if V is not None and (V.degree != 1 or V_phi.degree != 1 or method == "pk"):
        from .assemble_pk import PkAssemblyPlan
        return PkAssemblyPlan(mesh, c8, f8, ents, V, V_phi)
    return AssemblyPlan(mesh, c8, f8, ents, method=method, capacity=capacity,
                        order=order, geometry=geometry, cell_pass=cell_pass, rows_per_tile=rows_per_tile,
                        symbolic=symbolic)


def _device_vector(mesh, v, space=None):
    """Coefficient vector on the device; `space` (P_k plans) names the space it must live in."""
    if isinstance(v, Function):
        if space is None and v.function_space.degree != 1:
            raise NotImplementedError("this plan was built for P1 (vertex dofs); pass V / V_phi to build_plan")
        if space is not None and v.function_space.degree != space.degree:
            raise ValueError("coefficient of degree %d given where the plan expects degree %d"
                             % (v.function_space.degree, space.degree))
        v = v.x.array
    t = v if torch.is_tensor(v) else torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64))
    t = t.to(mesh.device, dtype=torch.float64, non_blocking=True).contiguous()
    n = mesh.num_vertices if space is None else space.num_dofs
    if t.numel() != n:
        raise ValueError("expected %d dof values, got %d" % (n, t.numel()))
    return t


def assemble_into(plan, phi, f, sigma, data, b, marks=None):
    """Numeric phase on the current stream: zero `data`/`b`, run the cell, boundary and ghost-penalty
    kernels.  All arguments are device tensors; nothing synchronises.  `marks` (optional callable) is
    invoked after the zeroing and after each kernel (bench.py records CUDA events there)."""
    if getattr(plan, "V", None) is not None:
        from .assemble_pk import assemble_pk_into
        return assemble_pk_into(plan, phi, f, sigma, data, b, marks=marks)
    marks_given = marks is not None
    marks = marks or (lambda: None)
    _lib.require_cuda(plan.mesh)
    if getattr(plan, "rowsplan", None) is not None:
        from . import rows as rows_mod
        marks()
        if marks_given:      # bench.py's breakdown: one C call per pass so that the events separate them
            rows_mod.assemble_rows_into(plan.rowsplan, phi, f, sigma, data, b, passes=("cells",))
            marks()
            marks()          # (the one-sided term is part of the surface pass)
            rows_mod.assemble_rows_into(plan.rowsplan, phi, f, sigma, data, b, passes=("surface",))
            marks()
        else:
            rows_mod.assemble_rows_into(plan.rowsplan, phi, f, sigma, data, b)
        return data, b
    if getattr(plan, "blocked", None) is not None:
        from . import blocked
        marks()
        blocked.assemble_blocked_into(plan.blocked, phi, f, sigma, data, b)
        marks()
        marks()
        marks()
        return data, b
    lib = _lib.load()
    cm = _lib.c_mesh(plan.mesh)
    st = _lib.stream()
    data.zero_()
    b.zero_()
    marks()
    _lib.check(lib.phifem_assemble_cells_p1(
        cm, _lib.ptr(phi), _lib.ptr(f), _lib.ptr(plan.cell_tags8), _lib.ptr(plan.active),
        plan.active.numel(), _lib.ptr(plan.slots_cells), float(sigma), _lib.ptr(data), _lib.ptr(b), st))
    marks()
    _lib.check(lib.phifem_assemble_boundary_p1(
        cm, _lib.ptr(phi), _lib.ptr(plan.entities), plan.entities.shape[0],
        _lib.ptr(plan.slots_boundary), _lib.ptr(data), st))
    marks()
    _lib.check(lib.phifem_assemble_ghost_p1(
        cm, _lib.ptr(phi), _lib.ptr(plan.ghost), plan.ghost.numel(), _lib.ptr(plan.slots_ghost),
        float(sigma), _lib.ptr(data), st))
    marks()
    return data, b


def assemble_strong_dirichlet(plan, phi_h, f_h, stab_coef=1.0):
    """A (CSR) and b of reference demo/strong-dirichlet/flower/main.py:104-131."""
    mesh = plan.mesh
    if getattr(plan, "form", "strong") != "strong":
        raise ValueError("the plan was built for the %s operator; call assemble_weak_dirichlet / assemble_neumann"
                         % plan.form)
    if getattr(plan, "V", None) is not None:
        from .assemble_pk import assemble_pk_into
        phi = _device_vector(mesh, phi_h, plan.V_phi)
        f = _device_vector(mesh, f_h, plan.V)
        data, b = plan.new_outputs()
        assemble_pk_into(plan, phi, f, stab_coef, data, b)
        return CSRMatrix(plan.indptr, plan.indices, data, (plan.n_rows, plan.n_rows)), b
    phi = _device_vector(mesh, phi_h)
    f = _device_vector(mesh, f_h)
    data, b = plan.new_outputs()
    assemble_into(plan, phi, f, stab_coef, data, b)
    return CSRMatrix(plan.indptr, plan.indices, data, (plan.n_rows, plan.n_rows)), b


def build_plan_weak_dirichlet(mesh, cells_tags, facets_tags, ds=None, V=None, V_phi=None):
    """Symbolic phase for `a` and `L` of the weak-Dirichlet (dual) demo (reference
    demo/weak-dirichlet/flower/main.py:112-151): mixed space `V x V` (u, p) (`mixed_space`, main.py:76-82),
    level-set space `V_phi`; defaults: P1 on the mesh.  The mixed vector holds u at even, p at odd positions."""
    refuse_hexahedra(mesh, "build_plan_weak_dirichlet")
    from . import fem
    from .assemble_pk import PkAssemblyPlan
    V = fem.functionspace(mesh, 1) if V is None else V
    V_phi = V if V_phi is None else V_phi
    c8, f8, ents = _plan_inputs(mesh, cells_tags, facets_tags, ds)
    return PkAssemblyPlan(mesh, c8, f8, ents, V, V_phi, form="weak")


def assemble_weak_dirichlet(plan, phi_h, f_h, u_D=None, pen_coef=1.0, stab_coef=1.0):
    """A (CSR over the mixed dofs) and b of reference demo/weak-dirichlet/flower/main.py:112-154;
    `u_D` = Dirichlet data in the primal space (None = 0, as `dirichlet_data` of the demo)."""
    from .assemble_pk import assemble_weak_into
    mesh = plan.mesh
    phi = _device_vector(mesh, phi_h, plan.V_phi)
    f = _device_vector(mesh, f_h, plan.V)
    ud = torch.zeros_like(f) if u_D is None else _device_vector(mesh, u_D, plan.V)
    data, b = plan.new_outputs()
    assemble_weak_into(plan, phi, f, ud, pen_coef, stab_coef, data, b)
    return CSRMatrix(plan.indptr, plan.indices, data, (plan.n_rows, plan.n_rows)), b


def build_plan_neumann(mesh, cells_tags, facets_tags, ds=None, V_phi=None, ghost_tag=3):
    """Symbolic phase for `a` and `L` of the Neumann demo (reference demo/neumann/square/main.py:103-158): mixed space
    (u, y, p) in P1 x P1^d x DG0 (`mixed_space`, main.py:71-79) on triangles / tetrahedra, level-set space `V_phi`
    (P1 or P2; default P1).  On quadrilaterals (the demo's own mesh) the space is Q1 x Q1^2 x DG0 and `V_phi` is Q1 or
    Q2, integrated by the Gauss product rule of `quadrature.rules_for_neumann_quad` (convex cells of either
    orientation; a non-convex quadrilateral is outside the method).  Mixed vector layout: u at vertex s -> (d+1) s,
    y_c -> (d+1) s + 1 + c, p of cell k -> (d+1) Nv + k (`plan.split(x)` returns the three fields).  ghost_tag: facets
    of the gradient-jump term, dS(3) in the Neumann demo (main.py:136-139), dS(2) in the Robin demo
    (demo/robin/square/main.py:143-150)."""
    refuse_hexahedra(mesh, "build_plan_neumann")
    from . import fem
    from .assemble_pk import PkAssemblyPlan
    V = fem.functionspace(mesh, 1)
    V_phi = V if V_phi is None else V_phi
    c8, f8, ents = _plan_inputs(mesh, cells_tags, facets_tags, ds)
    plan = PkAssemblyPlan(mesh, c8, f8, ents, V, V_phi, form="neumann", ghost_tag=ghost_tag)
    d, nv = mesh.gdim, mesh.num_vertices
    plan.split = lambda x: (x[:(d + 1) * nv].reshape(nv, d + 1)[:, 0], x[:(d + 1) * nv].reshape(nv, d + 1)[:, 1:],
                            x[(d + 1) * nv:])
    return plan


def assemble_neumann(plan, phi_h, f_h, u_N, pen_coef=1.0, stab_coef=1.0, robin_coef=0.0):
    """A (CSR over the mixed dofs) and b of reference demo/neumann/square/main.py:117-161; `f_h`, `u_N` are P1 (Q1 on
    quadrilaterals: vertex values).
    robin_coef != 0 (with a plan built with ghost_tag=2): the Robin operator of demo/robin/square/main.py:118-174,
    `u_N` being the Robin data u_R."""
    from .assemble_pk import assemble_neumann_into
    mesh = plan.mesh
    phi = _device_vector(mesh, phi_h, plan.V_phi)
    f = _device_vector(mesh, f_h, plan.V)
    un = _device_vector(mesh, u_N, plan.V)
    data, b = plan.new_outputs()
    assemble_neumann_into(plan, phi, f, un, pen_coef, stab_coef, data, b, robin_coef=robin_coef)
    return CSRMatrix(plan.indptr, plan.indices, data, (plan.n_rows, plan.n_rows)), b
