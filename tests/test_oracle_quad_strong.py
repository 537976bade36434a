"""The strong-Dirichlet operator on quadrilaterals without a GPU: the oracle's element tensors
(oracle/assembly_quad_strong.py `assemble_strong_dirichlet_quad`) against exact sympy integrals on parallelograms, its
physical Hessian on a non-parallelogram cell against high-precision central differences of the pulled-back function
(the check on the map's second-derivative term), and the symbolic phase of `build_plan` on a CPU quadrilateral mesh."""
import mpmath
import numpy as np
import pytest
import sympy as sp
import torch

from oracle import assembly as OA
from oracle import assembly_quad as OQ
from oracle import assembly_quad_strong as OS
from oracle import tags as OT
from phifem_b200 import assemble, fem, quadrature, synthetic
from phifem_b200.mesh import MeshTags

XI, ETA, S = sp.symbols("xi eta s")
R = sp.Rational
X0 = sp.Matrix([R(-1, 3), R(1, 5)])
E1 = sp.Matrix([R(1, 2), R(1, 7)])
E2 = sp.Matrix([R(-1, 6), R(2, 5)])
NQ1 = [(1 - XI) * (1 - ETA), XI * (1 - ETA), (1 - XI) * ETA, XI * ETA]
SIGMA = R(7, 10)


def _verts(x0, e1, e2):
    return [x0, x0 + e1, x0 + e2, x0 + e1 + e2]


def _h(verts):
    return sp.sqrt(max(sum((verts[a][d] - verts[b][d]) ** 2 for d in range(2))
                       for a in range(4) for b in range(a + 1, 4)))


def _phi_ref(kphi, seed):
    mons = [XI ** i * ETA ** j for i in range(kphi + 1) for j in range(kphi + 1)]
    return sum(R(3 + 2 * k + seed, 7 + k) * (-1) ** (k + seed) * mon for k, mon in enumerate(mons)) - R(1, 3)


def _interpolate(kphi, phi_ref):
    el = fem.LagrangeElement("quadrilateral", kphi)
    return np.array([float(phi_ref.subs({XI: p[0], ETA: p[1]})) for p in el.nodes])


def _calculus(verts):
    """grad and Laplacian in physical coordinates of expressions in (xi, eta) on a parallelogram (constant J)."""
    J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
    Jit = J.inv().T

    def grad(e):
        return Jit * sp.Matrix([sp.diff(e, XI), sp.diff(e, ETA)])

    def lap(e):
        H = sp.Matrix([[sp.diff(e, XI, XI), sp.diff(e, XI, ETA)], [sp.diff(e, ETA, XI), sp.diff(e, ETA, ETA)]])
        return (Jit * H * Jit.T).trace()
    return J, grad, lap


def _integrate(expr):
    p = sp.Poly(sp.expand(expr), XI, ETA)
    return sum(c / ((i + 1) * (j + 1)) for (i, j), c in p.terms())


def _to_np(verts):
    return np.array([[float(v[0]), float(v[1])] for v in verts])


@pytest.mark.parametrize("kphi", [1, 2])
def test_cell_tensor_matches_sympy_on_parallelogram(kphi):
    verts = _verts(X0, E1, E2)
    J, grad, lap = _calculus(verts)
    det = abs(J.det())
    phi_ref = _phi_ref(kphi, 0)
    f = [R(1, 3), R(-2, 5), R(3, 4), R(1, 7)]
    fq = sum(fk * n for fk, n in zip(f, NQ1))
    sh2 = SIGMA * _h(verts) ** 2
    gu = [grad(phi_ref * n) for n in NQ1]
    lu = [lap(phi_ref * n) for n in NQ1]
    A_s, A_cut, b_s, b_cut = (np.zeros((4, 4)), np.zeros((4, 4)), np.zeros(4), np.zeros(4))
    for a in range(4):
        b_s[a] = float(_integrate(fq * phi_ref * NQ1[a] * det))
        b_cut[a] = b_s[a] - float(sp.N(sh2 * _integrate(fq * lu[a] * det), 30))
        for bb in range(4):
            A_s[a, bb] = float(_integrate((gu[a].T * gu[bb])[0] * det))
            A_cut[a, bb] = A_s[a, bb] + float(sp.N(sh2 * _integrate(lu[a] * lu[bb] * det), 30))
    x = _to_np(verts)
    phi = _interpolate(kphi, phi_ref)[None]
    fv = np.array([[float(t) for t in f]])
    for cut, A_ref, b_ref in ((True, A_cut, b_cut), (False, A_s, b_s)):
        A, b = OS.strong_cell_tensors(x, np.array([[0, 1, 2, 3]]), phi, fv, np.array([cut]), 0.7, kphi)
        assert np.abs(A[0] - A_ref).max() <= 1e-13 * np.abs(A_ref).max()
        assert np.abs(b[0] - b_ref).max() <= 1e-13 * np.abs(b_ref).max()
    assert np.abs(A_cut - A_s).max() > 1e-3 * np.abs(A_s).max()   # the Hessian terms are present


@pytest.mark.parametrize("kphi", [1, 2])
def test_boundary_tensor_matches_sympy_on_parallelogram(kphi):
    verts = _verts(X0, E1, E2)
    _, grad, _ = _calculus(verts)
    phi_ref = _phi_ref(kphi, 1)
    x = _to_np(verts)
    phi = _interpolate(kphi, phi_ref)
    ents = np.array([[0, o] for o in range(4)])
    A = OS.strong_boundary_tensors(x, np.array([[0, 1, 2, 3]]), np.tile(phi, (4, 1)), ents, kphi)
    cen = sum(verts, sp.zeros(2, 1)) / 4
    for o in range(4):
        la, lb = OQ.QUAD_FACETS[o]
        t = verts[lb] - verts[la]
        length = sp.sqrt((t.T * t)[0])
        n = sp.Matrix([t[1], -t[0]]) / length
        if (n.T * (verts[la] - cen))[0] < 0:
            n = -n
        ra, rb = OQ.REF_VERTICES[la], OQ.REF_VERTICES[lb]
        edge = {XI: (1 - S) * int(ra[0]) + S * int(rb[0]), ETA: (1 - S) * int(ra[1]) + S * int(rb[1])}
        ref = np.zeros((4, 4))
        for i in range(4):
            for j in range(4):
                e = -((grad(phi_ref * NQ1[j]).T * n)[0] * phi_ref * NQ1[i]).subs(edge)
                ref[i, j] = float(sp.N(length * sp.integrate(sp.expand(e), (S, 0, 1)), 30))
        assert np.abs(A[o] - ref).max() <= 1e-13 * np.abs(ref).max(), o
        assert np.count_nonzero(ref[[k for k in range(4) if k not in (la, lb)]]) == 0


@pytest.mark.parametrize("kphi", [1, 2])
def test_ghost_tensor_matches_sympy(kphi):
    """Two parallelograms sharing an edge, the second mirrored (negative det J), each with its own level-set dofs:
    the macro tensor of sigma avg(h) int_F [grad(phi w).n][grad(phi v).n]."""
    x0, e1, e2 = X0, E1, E2
    pts = [x0, x0 + e1, x0 + e2, x0 + e1 + e2, x0 + 2 * e1, x0 + 2 * e1 + e2]
    cells = np.array([[0, 1, 2, 3], [4, 1, 5, 3]])
    x = _to_np(pts)
    c2f, f2c, _ = OT.build_topology(cells.astype(np.int32), "quadrilateral")
    shared = [f for f in range(len(f2c)) if f2c[f, 1] >= 0]
    assert len(shared) == 1
    phis = [_phi_ref(kphi, 0), _phi_ref(kphi, 1)]
    nd = (kphi + 1) ** 2
    phi = np.concatenate([_interpolate(kphi, p) for p in phis])
    phi_dofmap = np.arange(2 * nd).reshape(2, nd)
    E = OS.strong_ghost_tensors(x, cells, phi, phi_dofmap, c2f, f2c, shared, 0.7, kphi)[0]
    # both cells see the shared edge x1 -> x3 at xi = 1, eta = s
    jumps, hsum = [], 0
    for cell, phr in zip(cells, phis):
        verts = [pts[k] for k in cell]
        _, grad, _ = _calculus(verts)
        J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
        n = J.inv().T * sp.Matrix([1, 0])
        n = n / sp.sqrt((n.T * n)[0])
        for N in NQ1:
            jumps.append(((grad(phr * N).T * n)[0]).subs({XI: 1, ETA: S}))
        hsum += _h(verts)
    coef = SIGMA * hsum / 2 * sp.sqrt((e2.T * e2)[0])
    ref = np.zeros((8, 8))
    for a in range(8):
        for b in range(8):
            ref[a, b] = float(sp.N(coef * sp.integrate(sp.expand(jumps[a] * jumps[b]), (S, 0, 1)), 30))
    assert np.abs(E - ref).max() <= 1e-13 * np.abs(ref).max()


# ---- the physical Hessian on a non-affine cell -------------------------------------------------------------------
QX = np.array([[-0.31, 0.12], [0.47, 0.05], [-0.22, 0.83], [0.86, 0.61]])   # convex, c = X0 - X1 - X2 + X3 != 0


def _mp_hessian(element, coeffs, X, p, h=mpmath.mpf("1e-15")):
    """Central differences at 60 digits of u(x) = sum_k coeffs_k psi_k(ref(x)), ref(x) by Newton on the bilinear
    map."""
    Xm = [[mpmath.mpf(float(v)) for v in row] for row in X]
    coef = [[mpmath.mpf(float(v)) for v in row] for row in element.coef]
    exps = element.exps

    def ref_of(px, py):
        r = [mpmath.mpf("0.5"), mpmath.mpf("0.5")]
        for _ in range(60):
            N = [(1 - r[0]) * (1 - r[1]), r[0] * (1 - r[1]), (1 - r[0]) * r[1], r[0] * r[1]]
            dxi = [-(1 - r[1]), 1 - r[1], -r[1], r[1]]
            deta = [-(1 - r[0]), -r[0], 1 - r[0], r[0]]
            F = [sum(N[k] * Xm[k][d] for k in range(4)) - (px, py)[d] for d in range(2)]
            J = [[sum(dxi[k] * Xm[k][d] for k in range(4)), sum(deta[k] * Xm[k][d] for k in range(4))]
                 for d in range(2)]
            det = J[0][0] * J[1][1] - J[0][1] * J[1][0]
            s0 = (J[1][1] * F[0] - J[0][1] * F[1]) / det
            s1 = (-J[1][0] * F[0] + J[0][0] * F[1]) / det
            r = [r[0] - s0, r[1] - s1]
            if max(abs(s0), abs(s1)) < mpmath.mpf("1e-55"):
                break
        return r

    def u(px, py):
        r = ref_of(px, py)
        mon = [r[0] ** e[0] * r[1] ** e[1] for e in exps]
        return sum(coeffs[k] * sum(mon[m] * coef[m][k] for m in range(len(exps))) for k in range(element.ndofs))

    px, py = p
    u0 = u(px, py)
    uxx = (u(px + h, py) - 2 * u0 + u(px - h, py)) / h ** 2
    uyy = (u(px, py + h) - 2 * u0 + u(px, py - h)) / h ** 2
    uxy = (u(px + h, py + h) - u(px + h, py - h) - u(px - h, py + h) + u(px - h, py - h)) / (4 * h ** 2)
    return np.array([[float(uxx), float(uxy)], [float(uxy), float(uyy)]])


@pytest.mark.parametrize("k", [1, 2])
def test_physical_hessian_on_bilinear_cell(k):
    mpmath.mp.dps = 60
    el = fem.LagrangeElement("quadrilateral", k)
    refs = np.array([[0.21, 0.37], [0.5, 0.5], [0.83, 0.14], [0.09, 0.91]])
    N, dN = OQ.tabulate(OQ._Q1, refs)
    HN = OS.tabulate_hessians(OQ._Q1, refs)
    xq, J, _ = OQ.cell_map(QX, refs)
    d2x = np.einsum("kr,qkij->qrij", QX, HN)
    assert np.linalg.norm(d2x[:, :, 0, 1], axis=1).min() > 0.3      # the c-term is present
    _, dref = OQ.tabulate(el, refs)
    H = OS.physical_hessians(J, d2x, dref, OS.tabulate_hessians(el, refs))     # [nq, nd, 2, 2]
    rng = np.random.default_rng(5)
    combos = [np.eye(el.ndofs)[j] for j in range(el.ndofs)] + [rng.uniform(-1, 1, el.ndofs)]
    for coeffs in combos:
        Hc = np.einsum("qkrs,k->qrs", H, coeffs)
        cm = [mpmath.mpf(float(v)) for v in coeffs]
        for q in range(len(refs)):
            ref = _mp_hessian(el, cm, QX, (mpmath.mpf(float(xq[q, 0])), mpmath.mpf(float(xq[q, 1]))))
            assert np.abs(Hc[q] - ref).max() <= 1e-12 * max(np.abs(ref).max(), 1.0), (coeffs, q, Hc[q], ref)


# ---- rules and the symbolic phase ------------------------------------------------------------------------------
def test_rules_for_strong_quad():
    for kphi in (1, 2):
        (cp, cw), (fp, fw) = quadrature.rules_for_strong_quad(kphi)
        assert cp.shape == ((kphi + 2) ** 2, 2) and fp.shape == (kphi + 2, 2)
        assert abs(cw.sum() - 1.0) < 1e-15 and abs(fw.sum() - 1.0) < 1e-15
        t = fp[:, 1]
        for deg in range(2 * kphi + 3):
            assert abs(float((fw * t ** deg).sum()) - 1.0 / (deg + 1)) < 1e-15


def _cpu_problem(n=9):
    m = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(n, device="cpu"), jitter=0.2, seed=5)
    x, cells = m.x.numpy(), m.cells.numpy().astype(np.int64)
    phi = ((x - np.array([0.03, -0.02])) ** 2).sum(axis=1) - 0.6 ** 2
    ct = "quadrilateral"
    ftab = np.asarray([OT.coordinate_basis(ct, p)[0] for p in OT.facet_points_in_cell(ct, 1)])
    out = OT.compute_tags_measures(x, cells, ct, phi[cells], OT.point_values_function(phi, cells, ftab),
                                   box_mode=True, detection_points=OT.cell_detection_points(ct, 1))
    return m, cells, out, MeshTags(m, 2, torch.from_numpy(out["cell_tags"])), \
        MeshTags(m, 1, torch.from_numpy(out["facet_tags"]))


def test_build_plan_on_quadrilaterals():
    m, cells, out, ctags, ftags = _cpu_problem()
    active = np.nonzero((out["cell_tags"] == 1) | (out["cell_tags"] == 2))[0]
    ghost = np.nonzero(((out["facet_tags"] == 2) | (out["facet_tags"] == 3)) & (out["f2c"][:, 1] >= 0))[0]
    ip, ix = OA.sparsity_pattern(m.num_vertices, cells, active, ghost, out["f2c"])
    for kphi in (1, 2):
        Vp = fem.functionspace(m, kphi)
        plan = assemble.build_plan(m, ctags, ftags, out["ds100"], V_phi=Vp)
        assert plan.form == "strong" and plan.V.degree == 1 and plan.V_phi is Vp
        assert plan.n_cell_points == (kphi + 2) ** 2 and plan.n_facet_points == kphi + 2
        assert plan.ghost.numel() > 0 and plan.entities.shape[0] > 0
        assert np.array_equal(plan.indptr.numpy(), ip) and np.array_equal(plan.indices.numpy(), ix)
    plan = assemble.build_plan(m, ctags, ftags, out["ds100"])      # V and V_phi default to Q1
    assert plan.V.degree == 1 and plan.V_phi.degree == 1 and plan.n_rows == m.num_vertices
    assert np.array_equal(plan.indptr.numpy(), ip) and np.array_equal(plan.indices.numpy(), ix)


def test_build_plan_refusals_on_quadrilaterals():
    m, _, out, ctags, ftags = _cpu_problem(5)
    ds = out["ds100"]
    with pytest.raises(NotImplementedError):                  # Q2 trial space
        assemble.build_plan(m, ctags, ftags, ds, V=fem.functionspace(m, 2))
    with pytest.raises(NotImplementedError):                  # weak-Dirichlet form
        assemble.build_plan_weak_dirichlet(m, ctags, ftags, ds)
    for kw in (dict(method="blocked"), dict(method="atomic"), dict(geometry=True), dict(cell_pass="tiles"),
               dict(symbolic="native")):
        with pytest.raises(ValueError):
            assemble.build_plan(m, ctags, ftags, ds, **kw)
