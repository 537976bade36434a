"""The quadrilateral pieces of the Neumann operator that need no GPU: the Gauss product rule, the synthetic
quadrilateral mesh, the oracle's element tensors (oracle/assembly_quad.py) against exact sympy integrals on
parallelograms, and the symbolic phase of `build_plan_neumann` on a CPU quadrilateral mesh."""
import itertools

import numpy as np
import pytest
import sympy as sp
import torch

from oracle import assembly as OA
from oracle import assembly_quad as OQ
from oracle import tags as OT
from phifem_b200 import assemble, fem, quadrature, synthetic
from phifem_b200.mesh import MeshTags


@pytest.mark.parametrize("m", [1, 2, 3, 4, 5])
def test_square_rule_integrates_monomials(m):
    pts, w = quadrature.square_rule(m)
    assert pts.shape == (m * m, 2) and abs(w.sum() - 1.0) < 1e-15 and np.all(w > 0)
    for a, b in itertools.product(range(2 * m), repeat=2):
        exact = 1.0 / ((a + 1) * (b + 1))
        assert abs(float((w * pts[:, 0] ** a * pts[:, 1] ** b).sum()) - exact) < 1e-15, (a, b)


def test_rules_for_neumann_quad():
    for kphi in (1, 2):
        (cp, cw), (fp, fw) = quadrature.rules_for_neumann_quad(kphi)
        assert cp.shape == ((kphi + 2) ** 2, 2) and fp.shape == (2, 2)
        assert abs(cw.sum() - 1.0) < 1e-15 and abs(fw.sum() - 1.0) < 1e-15


def _corner_dets(mesh):
    x, cells = mesh.x.cpu().numpy(), mesh.cells.cpu().numpy()
    return np.array([OQ.cell_map(x[c], OQ.REF_VERTICES)[2] for c in cells])   # [Nc, 4]


@pytest.mark.parametrize("n", [1, 3, 8])
def test_quadrilateral_mesh(n):
    m = synthetic.quadrilateral_mesh(n, device="cpu")
    assert m.cell_type == "quadrilateral"
    assert m.num_cells == n * n and m.num_vertices == (n + 1) ** 2 and m.num_facets == 2 * n * (n + 1)
    x = m.x.numpy()
    assert np.allclose(x.min(axis=0), [-1, -1]) and np.allclose(x.max(axis=0), [1, 1])
    i, j = 1 % (n + 1), n // 2     # vertex id i*(n+1)+j is the point (x_i, y_j), as in rectangle_mesh
    assert np.allclose(x[i * (n + 1) + j], [-1 + 2 * i / n, -1 + 2 * j / n])
    assert np.allclose(_corner_dets(m), (2.0 / n) ** 2)
    u = synthetic.unstructured_variant(m, jitter=0.2, seed=7)
    dets = _corner_dets(u)
    assert np.all(dets > 0) or np.all(dets < 0)
    assert u.cell_type == "quadrilateral" and u.num_facets == m.num_facets


# ---- element tensors on a parallelogram against sympy ------------------------------------------------------------
XI, ETA, HS, NG = sp.symbols("xi eta hs ng", positive=True)
R = sp.Rational
X0 = sp.Matrix([R(-1, 3), R(1, 5)])
E1 = sp.Matrix([R(1, 2), R(1, 7)])
E2 = sp.Matrix([R(-1, 6), R(2, 5)])
NQ1 = [(1 - XI) * (1 - ETA), XI * (1 - ETA), (1 - XI) * ETA, XI * ETA]


def _verts(x0, e1, e2):
    return [x0, x0 + e1, x0 + e2, x0 + e1 + e2]


def _h2(verts):
    return max(sum((verts[a][d] - verts[b][d]) ** 2 for d in range(2)) for a in range(4) for b in range(a + 1, 4))


def _integrate(expr):
    """Integral over the reference square of a polynomial in (xi, eta) (coefficients may hold HS / NG)."""
    p = sp.Poly(sp.expand(expr), XI, ETA)
    return sum(c / ((i + 1) * (j + 1)) for (i, j), c in p.terms())


def _sympy_cell(verts, phi_ref, f, un, gamma, with_un):
    J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
    det = abs(J.det())
    Jit = J.inv().T
    grad = lambda e: Jit * sp.Matrix([sp.diff(e, XI), sp.diff(e, ETA)])   # noqa: E731
    G = [grad(n) for n in NQ1]
    gph = grad(phi_ref)
    fq = sum(fk * n for fk, n in zip(f, NQ1))
    uq = sum(uk * n for uk, n in zip(un, NQ1))
    zero = sp.Matrix([0, 0])
    fields = []   # (U, GU, S1, S2, S3) of the 13 mixed basis functions
    for j in range(4):
        fields.append((NQ1[j], G[j], G[j], NQ1[j], 0))
    for j in range(4):
        for c in range(2):
            s1 = sp.Matrix([NQ1[j] if d == c else 0 for d in range(2)])
            fields.append((0, zero, s1, G[j][c], NQ1[j] * gph[c]))
    fields.append((0, zero, zero, 0, phi_ref / HS))
    A = np.zeros((13, 13))
    b = np.zeros(13)
    h = sp.sqrt(_h2(verts))
    sub = {HS: h, NG: sp.sqrt((gph.T * gph)[0]) if with_un else 0}
    for a in range(13):
        Ua, GUa, S1a, S2a, S3a = fields[a]
        lb = fq * Ua + gamma * (fq * S2a - (uq * NG * S3a / HS ** 2 if with_un else 0))
        b[a] = float(sp.N(_integrate(lb * det).subs(sub), 30))
        for bb in range(a, 13):
            Ub, GUb, S1b, S2b, S3b = fields[bb]
            e = (GUa.T * GUb)[0] + Ua * Ub + gamma * ((S1a.T * S1b)[0] + S2a * S2b + S3a * S3b / HS ** 2)
            A[a, bb] = A[bb, a] = float(sp.N(_integrate(e * det).subs(sub), 30))
    return A, b


def _interpolate(kphi, phi_ref):
    el = fem.LagrangeElement("quadrilateral", kphi)
    return np.array([float(phi_ref.subs({XI: p[0], ETA: p[1]})) for p in el.nodes])


@pytest.mark.parametrize("kphi,case", [(1, "poly"), (2, "poly"), (1, "linear"), (2, "linear")])
def test_cell_tensor_matches_sympy_on_parallelogram(kphi, case):
    """poly: a Q_kphi level set with every monomial, u_N = 0 (|grad phi| is not polynomial); linear: a level set
    affine in x on the cell (constant gradient), so the u_N |grad phi| load term is polynomial too."""
    verts = _verts(X0, E1, E2)
    if case == "poly":
        mons = [XI ** i * ETA ** j for i in range(kphi + 1) for j in range(kphi + 1)]
        phi_ref = sum(R(3 + 2 * k, 7 + k) * (-1) ** k * mon for k, mon in enumerate(mons)) - R(1, 3)
    else:
        phi_ref = R(1, 4) - R(2, 3) * XI + R(3, 5) * ETA   # affine map: affine in x
    f = [R(1, 3), R(-2, 5), R(3, 4), R(1, 7)]
    un = [R(2, 3), R(1, 2), R(-1, 4), R(5, 6)] if case == "linear" else [0, 0, 0, 0]
    gamma = R(13, 10)
    A_s, b_s = _sympy_cell(verts, phi_ref, f, un, gamma, with_un=case == "linear")
    x = np.array([[float(v[0]), float(v[1])] for v in verts])
    to_f = lambda v: np.array([float(t) for t in v])[None]   # noqa: E731
    A, b = OQ.cell_tensors(x, np.array([[0, 1, 2, 3]]), _interpolate(kphi, phi_ref)[None], to_f(f), to_f(un),
                           np.array([True]), 1.3, kphi)
    assert np.abs(A[0] - A_s).max() <= 1e-13 * np.abs(A_s).max()
    assert np.abs(b[0] - b_s).max() <= 1e-13 * np.abs(b_s).max()
    # the same cell untagged as cut: only grad u.grad v + u v and f v remain
    A1, b1 = OQ.cell_tensors(x, np.array([[0, 1, 2, 3]]), _interpolate(kphi, phi_ref)[None], to_f(f), to_f(un),
                             np.array([False]), 1.3, kphi)
    assert np.count_nonzero(A1[0][4:]) == 0 and np.count_nonzero(A1[0][:, 4:]) == 0 and np.all(b1[0][4:] == 0)
    assert np.all(np.abs(A1[0][:4, :4]) > 0)


def test_boundary_tensor_matches_closed_form():
    m = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(5, device="cpu"), jitter=0.2, seed=3)
    x, cells = m.x.numpy(), m.cells.numpy().astype(np.int64)
    ents = np.array([(c, o) for c in range(0, m.num_cells, 3) for o in range(4)])
    A = OQ.boundary_tensors(x, cells, ents)
    for e, (c, o) in enumerate(ents):
        la, lb = OQ.QUAD_FACETS[o]
        X = x[cells[c]]
        t = X[lb] - X[la]
        length = np.linalg.norm(t)
        n = np.array([t[1], -t[0]]) / length
        if n @ (X[la] - X.mean(axis=0)) < 0:
            n = -n
        ref = np.zeros((13, 13))
        for i in (la, lb):
            for j in (la, lb):
                ref[i, 4 + 2 * j:6 + 2 * j] = n * length * (2.0 if i == j else 1.0) / 6.0
        assert np.abs(A[e] - ref).max() <= 1e-14 * np.abs(ref).max()


def test_ghost_tensor_matches_sympy():
    """Two parallelograms sharing an edge, the second one mirrored (negative det J): the macro tensor of
    sigma avg(h) int_F [grad u.n][grad v.n] (grad u varies along the edge: Q1 holds xi eta)."""
    x0, e1, e2 = X0, E1, E2
    pts = [x0, x0 + e1, x0 + e2, x0 + e1 + e2, x0 + 2 * e1, x0 + 2 * e1 + e2]
    cells = np.array([[0, 1, 2, 3], [4, 1, 5, 3]])
    x = np.array([[float(p[0]), float(p[1])] for p in pts])
    c2f, f2c, _ = OT.build_topology(cells.astype(np.int32), "quadrilateral")
    shared = [f for f in range(len(f2c)) if f2c[f, 1] >= 0]
    assert len(shared) == 1
    E = OQ.ghost_tensors(x, cells, c2f, f2c, shared, 0.7)[0]
    # sympy: parameter s along the shared edge x1 -> x3; both cells see it at xi = 1, eta = s
    s = sp.symbols("s")
    jumps, hsum = [], 0
    for cell in cells:
        verts = [pts[k] for k in cell]
        J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
        Jit = J.inv().T
        n = Jit * sp.Matrix([1, 0])
        n = n / sp.sqrt((n.T * n)[0])
        for N in NQ1:
            g = Jit * sp.Matrix([sp.diff(N, XI), sp.diff(N, ETA)])
            jumps.append(((g.T * n)[0]).subs({XI: 1, ETA: s}))
        hsum += sp.sqrt(_h2(verts))
    coef = R(7, 10) * hsum / 2 * sp.sqrt((e2.T * e2)[0])
    ref = np.zeros((26, 26))
    mac = [k for k in range(4)] + [13 + k for k in range(4)]
    for a in range(8):
        for b in range(8):
            ref[mac[a], mac[b]] = float(sp.N(coef * sp.integrate(sp.expand(jumps[a] * jumps[b]), (s, 0, 1)), 30))
    assert np.abs(E - ref).max() <= 1e-13 * np.abs(ref).max()


def test_symbolic_phase_matches_oracle_pattern():
    m = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(9, device="cpu"), jitter=0.2, seed=5)
    x, cells = m.x.numpy(), m.cells.numpy().astype(np.int64)
    phi = ((x - np.array([0.03, -0.02])) ** 2).sum(axis=1) - 0.6 ** 2
    ct = "quadrilateral"
    ftab = np.asarray([OT.coordinate_basis(ct, p)[0] for p in OT.facet_points_in_cell(ct, 1)])
    out = OT.compute_tags_measures(x, cells, ct, phi[cells], OT.point_values_function(phi, cells, ftab),
                                   box_mode=True, detection_points=OT.cell_detection_points(ct, 1))
    ctags = MeshTags(m, 2, torch.from_numpy(out["cell_tags"]))
    ftags = MeshTags(m, 1, torch.from_numpy(out["facet_tags"]))
    for kphi, gtag in ((1, 3), (2, 2)):
        plan = assemble.build_plan_neumann(m, ctags, ftags, out["ds100"], V_phi=fem.functionspace(m, kphi),
                                           ghost_tag=gtag)
        assert plan.n_rows == 3 * m.num_vertices + m.num_cells and plan.pattern_dofmap.shape[1] == 13
        assert plan.cut_positions.numel() > 0 and plan.ghost.numel() > 0 and plan.entities.shape[0] > 0
        assert plan.n_cell_points == (kphi + 2) ** 2 and plan.n_facet_points == 2
        active = np.nonzero((out["cell_tags"] == 1) | (out["cell_tags"] == 2))[0]
        ghost = np.nonzero((out["facet_tags"] == gtag) & (out["f2c"][:, 1] >= 0))[0]
        mixed = OQ.neumann_mixed_dofmap_quad(cells, m.num_vertices)
        assert np.array_equal(plan.pattern_dofmap.numpy(), mixed)
        ip, ix = OA.sparsity_pattern(plan.n_rows, mixed, active, ghost, out["f2c"])
        assert np.array_equal(plan.indptr.numpy(), ip) and np.array_equal(plan.indices.numpy(), ix)
