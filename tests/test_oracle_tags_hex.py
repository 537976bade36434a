"""Hexahedral meshes on the CPU: topology, detection points, trilinear scales, Q1 / Q2 elements and the oracle's tags.

The scales are held to exact sympy values on random rational vertices; the oracle's tags to properties that follow
from the detection rule (a plane between grid lines cuts one layer; relabelling moves tags with their entities)."""
import fractions

import numpy as np
import pytest
import sympy as sp
import torch

from oracle import tags as OT
from oracle import tags_hex as OH
from phifem_b200 import _geometry as G
from phifem_b200 import fem, synthetic
from phifem_b200.mesh import Mesh, build_facet_topology


@pytest.mark.parametrize("n", [1, 2, 3, 5])
def test_hexahedron_mesh_topology_counts_and_oracle_numbering(n):
    mesh = synthetic.hexahedron_mesh(n, device="cpu")
    box = synthetic.box_mesh(n, device="cpu")
    assert torch.equal(mesh.x, box.x)
    assert mesh.num_cells == n ** 3
    assert mesh.num_facets == 3 * n * n * (n + 1)
    assert int((mesh.f2c[:, 1] < 0).sum()) == 6 * n * n == mesh.boundary_facets.numel()
    c2f, f2c, fverts = OH.build_topology(mesh.cells.numpy())
    assert np.array_equal(mesh.c2f.numpy(), c2f)
    assert np.array_equal(mesh.f2c.numpy(), f2c)
    assert np.array_equal(mesh.facet_vertices.numpy(), fverts)
    # the vertices of every cell sit at the corners of its cube in tensor order
    xc = mesh.x[mesh.cells.long()].numpy()
    h = 1.0 / n
    assert np.allclose(xc - xc[:, :1], G.REF_VERTICES["hexahedron"][None] * h, atol=1e-14)


def test_facet_topology_of_relabelled_mesh_matches_oracle():
    mesh = synthetic.unstructured_variant(synthetic.hexahedron_mesh(4, device="cpu"), jitter=0.2, seed=3)
    c2f, f2c, fverts = build_facet_topology(mesh.cells, "hexahedron", mesh.num_vertices)
    oc2f, of2c, ofv = OH.build_topology(mesh.cells.numpy())
    assert np.array_equal(c2f.numpy(), oc2f) and np.array_equal(f2c.numpy(), of2c)
    assert np.array_equal(fverts.numpy(), ofv)
    # facet vertex tuples are sorted and in lexicographic order
    fv = fverts.numpy().astype(np.int64)
    assert np.all(np.diff(fv, axis=1) > 0)
    assert np.all(np.diff(((fv[:, 0] * 10 ** 3 + fv[:, 1]) * 10 ** 3 + fv[:, 2]) * 10 ** 3 + fv[:, 3]) > 0)


@pytest.mark.parametrize("N", [0, 1, 2, 3, 4])
def test_detection_points_count_surface_and_oracle_agree(N):
    pts = G.cell_detection_points("hexahedron", N)
    assert np.array_equal(pts, OH.boundary_points(N))
    fpts = G.facet_detection_points("hexahedron", N)
    assert np.array_equal(fpts, OH.facet_points_in_cell(N))
    if N == 0:
        assert np.array_equal(pts, [[0.5, 0.5, 0.5]])
        return
    assert len(pts) == 8 + 12 * (N - 1) + 6 * (N - 1) ** 2
    assert len(np.unique(pts, axis=0)) == len(pts)
    on_surface = np.any((pts == 0.0) | (pts == 1.0), axis=1)
    assert on_surface.all() and np.all((pts >= 0) & (pts <= 1))
    assert np.array_equal(pts[:8], G.REF_VERTICES["hexahedron"])
    # facet points: the square's points on every face, which holds them
    assert fpts.shape == (6, 4 * N, 3)
    for lf, face in enumerate(G.LOCAL_FACETS["hexahedron"]):
        rv = G.REF_VERTICES["hexahedron"][list(face)]
        fixed = np.nonzero(np.all(rv == rv[0], axis=0))[0]
        assert len(fixed) == 1 and np.all(fpts[lf][:, fixed[0]] == rv[0, fixed[0]])


def _random_rational_hex(rng):
    """Unit cube corners moved by rationals of up to 1/5: convex, non-affine."""
    verts = []
    for v in range(8):
        corner = [(v >> d) & 1 for d in range(3)]
        verts.append([fractions.Fraction(int(c) * 10 + int(rng.integers(-2, 3)), 10) for c in corner])
    return verts


def _sympy_map(verts):
    X = sp.symbols("X0:3")
    x = [0, 0, 0]
    for v, p in enumerate(verts):
        w = sp.Integer(1)
        for d in range(3):
            w *= X[d] if (v >> d) & 1 else 1 - X[d]
        for d in range(3):
            x[d] += w * sp.Rational(p[d].numerator, p[d].denominator)
    return X, sp.Matrix(x)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_cell_and_facet_scales_match_exact_sympy_values(seed):
    rng = np.random.default_rng(seed)
    verts = _random_rational_hex(rng)
    X, xmap = _sympy_map(verts)
    J = xmap.jacobian(X)
    x = np.array([[float(c) for c in p] for p in verts])
    cells = np.arange(8)[None, :]
    pts = OH.boundary_points(3)
    got = OH.cell_scale(x, cells, pts)[0]
    # the product's coordinate element gives the same Jacobians
    g = G.coordinate_basis_grad("hexahedron", pts)
    detj = sp.lambdify(X, J.det(), "sympy")
    for q, p in enumerate(pts):
        exact = abs(detj(*[sp.Rational(fractions.Fraction(c).limit_denominator(10 ** 6)) for c in p]))
        assert abs(got[q] - float(exact)) <= 1e-15 * max(1.0, float(exact))
        Jq = np.einsum("vj,vi->ij", g[q], x)
        assert abs(abs(np.linalg.det(Jq)) - float(exact)) <= 1e-14
    fpts = OH.facet_points_in_cell(3)
    fs = OH.facet_scale(x, cells, fpts)[0]
    for lf in range(6):
        sa, ta = OH.face_axes(lf)
        cr = J[:, sa].cross(J[:, ta])
        area = sp.lambdify(X, cr.dot(cr), "sympy")
        for q, p in enumerate(fpts[lf]):
            exact = sp.sqrt(area(*[sp.Rational(fractions.Fraction(c).limit_denominator(10 ** 6)) for c in p]))
            assert abs(fs[lf, q] - float(exact)) <= 1e-15 * max(1.0, float(exact))


def test_physical_points_reproduce_the_trilinear_map():
    rng = np.random.default_rng(7)
    verts = _random_rational_hex(rng)
    X, xmap = _sympy_map(verts)
    x = np.array([[float(c) for c in p] for p in verts])
    pts = OH.boundary_points(2)
    got = OH.physical_points(x, np.arange(8)[None, :], pts)[0]
    f = sp.lambdify(X, xmap, "numpy")
    for q, p in enumerate(pts):
        assert np.allclose(got[q], np.asarray(f(*p), dtype=float).ravel(), atol=1e-15, rtol=0)


@pytest.mark.parametrize("k", [1, 2])
def test_q_elements_are_kronecker_and_reproduce_qk(k):
    e = fem.LagrangeElement("hexahedron", k)
    assert e.ndofs == (k + 1) ** 3
    assert np.array_equal(e.tabulate(e.nodes), np.eye(e.ndofs))
    rng = np.random.default_rng(k)
    pts = rng.random((40, 3))
    tab = e.tabulate(pts, snap=False)
    for a in range(k + 1):
        for b in range(k + 1):
            for c in range(k + 1):
                f = lambda p: p[:, 0] ** a * p[:, 1] ** b * p[:, 2] ** c  # noqa: E731
                assert np.allclose(tab @ f(e.nodes), f(pts), atol=1e-13)
    if k == 2:  # vertices, edge midpoints, face centres, centre
        assert np.array_equal(e.nodes[:8], G.REF_VERTICES["hexahedron"])
        for i, (a, b) in enumerate(G.HEX_EDGES):
            assert np.array_equal(e.nodes[8 + i], 0.5 * (e.nodes[a] + e.nodes[b]))
        for i, face in enumerate(G.LOCAL_FACETS["hexahedron"]):
            assert np.array_equal(e.nodes[20 + i], e.nodes[list(face)].mean(axis=0))
        assert np.array_equal(e.nodes[26], [0.5, 0.5, 0.5])


def test_degree_3_on_hexahedra_is_refused():
    with pytest.raises(NotImplementedError, match="hexahedra"):
        fem.LagrangeElement("hexahedron", 3)
    with pytest.raises(NotImplementedError):
        fem.functionspace(synthetic.hexahedron_mesh(1, device="cpu"), 3)


@pytest.mark.parametrize("n", [1, 2, 4])
def test_q2_dofmap_counts_and_interpolation(n):
    mesh = synthetic.unstructured_variant(synthetic.hexahedron_mesh(n, device="cpu"), jitter=0.15, seed=n)
    V2 = fem.functionspace(mesh, ("Lagrange", 2))
    assert V2.num_dofs == (2 * n + 1) ** 3
    dm = V2.dofmap
    assert dm.shape == (n ** 3, 27) and len(np.unique(dm)) == V2.num_dofs
    # a face shared by two cells carries the same dof in both
    c2f = mesh.c2f.numpy()
    face_dof = np.full(mesh.num_facets, -1)
    for lf in range(6):
        prev = face_dof[c2f[:, lf]]
        assert np.all((prev < 0) | (prev == dm[:, 20 + lf]))
        face_dof[c2f[:, lf]] = dm[:, 20 + lf]
    # interpolation reproduces functions of the coordinate space exactly (Q1 on the trilinear cells)
    f = lambda x: 1.0 + 2.0 * x[0] - x[1] + 0.5 * x[2]  # noqa: E731
    for k, V in ((1, fem.functionspace(mesh, 1)), (2, V2)):
        fn = fem.Function(V).interpolate(f)
        X = V.tabulate_dof_coordinates()
        assert np.allclose(fn.x.array, f(X.T), atol=1e-14)
        pts = np.random.default_rng(0).random((10, 3))
        vals = fn.x.array[V.dofmap] @ V.element.tabulate(pts).T          # [Nc, 10]
        phys = OH.physical_points(mesh.x.numpy(), mesh.cells.numpy(), pts)
        assert np.allclose(vals, f(np.moveaxis(phys, 2, 0)), atol=1e-13)


def _oracle_tags(mesh, levelset, N, box_mode=True, single=False):
    x, cells = mesh.x.numpy(), mesh.cells.numpy().astype(np.int64)
    phi_c = OH.point_values_expression(levelset, x, cells, OH.boundary_points(N))
    phi_f = OH.point_values_expression(levelset, x, cells, OH.facet_points_in_cell(N))
    return OH.compute_tags_measures(x, cells, phi_c, phi_f, N, box_mode=box_mode, single_layer_cut=single)


@pytest.mark.parametrize("N", [1, 2, 3])          # N = 0: one point per cell, no cell can be cut
@pytest.mark.parametrize("axis", [0, 1, 2])
def test_oracle_plane_cuts_exactly_its_layer(N, axis):
    n = 6
    a = 0.37                                           # between the grid lines 2/6 and 3/6
    mesh = synthetic.hexahedron_mesh(n, device="cpu")
    out = _oracle_tags(mesh, lambda x: x[axis] - a, N)
    lo = mesh.x[mesh.cells.long()].numpy()[:, 0, axis]
    layer = np.floor(lo * n + 0.5).astype(int)
    want = np.where(layer < 2, 1, np.where(layer == 2, 2, 3))
    assert np.array_equal(out["cell_tags"], want)
    # Gamma_h: the faces between the cut layer and the exterior; facets 3: between the interior and the cut layer
    ft = out["facet_tags"]
    fv = mesh.facet_vertices.numpy()
    xf = mesh.x.numpy()[fv][:, :, axis]
    plane = np.all(xf == xf[:, :1], axis=1)
    pos = np.round(xf[:, 0] * n).astype(int)
    assert np.all(ft[plane & (pos == 3)] == 4)
    assert np.all(ft[plane & (pos == 2)] == 3)
    assert len(out["duplicates"]) == 0


@pytest.mark.parametrize("N", [1, 2])
def test_oracle_tags_are_invariant_under_relabelling(N):
    base = synthetic.unstructured_variant(synthetic.hexahedron_mesh(5, device="cpu"), jitter=0.2, seed=11)
    x, cells = base.x.numpy(), base.cells.numpy().astype(np.int64)
    sphere = lambda p: (p[0] - 0.51) ** 2 + (p[1] - 0.48) ** 2 + (p[2] - 0.5) ** 2 - 0.33 ** 2  # noqa: E731
    ref = _oracle_tags(base, sphere, N)
    rng = np.random.default_rng(5)
    cperm = rng.permutation(len(cells))
    vrel = rng.permutation(len(x))
    xn = np.empty_like(x)
    xn[vrel] = x
    moved = Mesh(xn, vrel[cells[cperm]].astype(np.int32), "hexahedron", device="cpu")
    out = _oracle_tags(moved, sphere, N)
    assert np.array_equal(out["cell_tags"], ref["cell_tags"][cperm])
    key = lambda fv, relabel: [tuple(sorted(relabel[v] for v in f)) for f in fv]  # noqa: E731
    ref_faces = dict(zip(key(ref["facet_vertices"], vrel), ref["facet_tags"]))
    mine = dict(zip(key(out["facet_vertices"], np.arange(len(x))), out["facet_tags"]))
    assert mine == ref_faces
    assert set(np.unique(ref["cell_tags"])) == {1, 2, 3}


def test_oracle_scales_on_the_affine_mesh_are_the_cube_measures():
    n = 3
    mesh = synthetic.hexahedron_mesh(n, lo=(-1.0, 0.0, 2.0), hi=(2.0, 1.5, 2.75), device="cpu")
    x, cells = mesh.x.numpy(), mesh.cells.numpy()
    h = np.array([3.0, 1.5, 0.75]) / n
    assert np.allclose(OH.cell_scale(x, cells, OH.boundary_points(2)), h.prod(), rtol=1e-14)
    fs = OH.facet_scale(x, cells, OH.facet_points_in_cell(2))
    for lf in range(6):
        sa, ta = OH.face_axes(lf)
        assert np.allclose(fs[:, lf], h[sa] * h[ta], rtol=1e-14)
    ents = np.stack([np.arange(len(cells)), np.full(len(cells), 5)], axis=1)
    nrm, area = OH.outward_normals(x, cells, ents)
    assert np.allclose(nrm, [0.0, 0.0, 1.0]) and np.allclose(area, h[0] * h[1])
    ents[:, 1] = 2
    nrm, _ = OH.outward_normals(x, cells, ents)
    assert np.allclose(nrm, [-1.0, 0.0, 0.0])


def test_square_and_triangle_facet_points_unchanged():
    # the facet-point builder now loops over the reference facet's coordinates: the 2D / tetrahedron tables are the
    # oracle's as before
    for ct in ("triangle", "quadrilateral", "tetrahedron"):
        for N in range(4):
            assert np.array_equal(G.facet_detection_points(ct, N), OT.facet_points_in_cell(ct, N))


def test_every_assembly_constructor_refuses_hexahedra():
    from phifem_b200 import assemble, elasticity, partition
    mesh = synthetic.hexahedron_mesh(2, device="cpu")
    phi = torch.zeros(mesh.num_vertices, dtype=torch.float64)
    calls = [lambda: assemble.build_plan(mesh, None, None),
             lambda: assemble.build_plan_weak_dirichlet(mesh, None, None),
             lambda: assemble.build_plan_neumann(mesh, None, None),
             lambda: elasticity.ElasticityPlan(mesh, None, None, None, None, None),
             lambda: partition.PartitionedProblem(mesh, phi, phi, 0, 1)]
    for call in calls:
        with pytest.raises(NotImplementedError, match="hexahedron"):
            call()
