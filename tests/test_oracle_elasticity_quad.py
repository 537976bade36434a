"""The interface-elasticity operator on quadrilaterals without a GPU: the oracle's element tensors
(oracle/elasticity_quad.py `assemble_interface_elasticity_quad`) against exact sympy integrals of the literal integrands
on a sheared parallelogram, the uncut stiffness on a cell that is not a parallelogram against the rigid modes, and the
symbolic phase of `ElasticityPlan` on a CPU quadrilateral mesh."""
import numpy as np
import pytest
import sympy as sp
import torch

from oracle import assembly as OA
from oracle import assembly_quad as OQ
from oracle import elasticity as OE
from oracle import elasticity_quad as OEQ
from oracle import tags as OT
from phifem_b200 import elasticity, fem, quadrature, synthetic

XI, ETA, S = sp.symbols("xi eta s")
R = sp.Rational
X0 = sp.Matrix([R(-1, 3), R(1, 5)])
E1 = sp.Matrix([R(1, 2), R(1, 7)])
E2 = sp.Matrix([R(-1, 6), R(2, 5)])
NQ1 = [(1 - XI) * (1 - ETA), XI * (1 - ETA), (1 - XI) * ETA, XI * ETA]
E_IN, NU_IN, E_OUT, NU_OUT = R(1), R(3, 10), R(1, 20), R(27, 100)
GAMMA, SIGMA_S = R(13, 10), R(7, 10)
NB = 14
MAT = OE.Material(1.0, 0.3, 0.05, 0.27)


def _lame(E, nu):
    return E * nu / (1 + nu) / (1 - 2 * nu), E / 2 / (1 + nu)


LM_IN, MU_IN = _lame(E_IN, NU_IN)
LM_OUT, MU_OUT = _lame(E_OUT, NU_OUT)
C_IN, C_OUT = (E_IN / (E_IN + E_OUT)) ** 2, (E_OUT / (E_IN + E_OUT)) ** 2


def _verts(x0, e1, e2):
    return [x0, x0 + e1, x0 + e2, x0 + e1 + e2]


def _to_np(verts):
    return np.array([[float(v[0]), float(v[1])] for v in verts])


def _h2(verts):
    return max(sum((verts[a][d] - verts[b][d]) ** 2 for d in range(2)) for a in range(4) for b in range(a + 1, 4))


def _phi_ref(kphi, seed):
    mons = [XI ** i * ETA ** j for i in range(kphi + 1) for j in range(kphi + 1)]
    return sum(R(3 + 2 * k + seed, 7 + k) * (-1) ** (k + seed) * mon for k, mon in enumerate(mons)) - R(1, 3)


def _interpolate(kphi, phi_ref):
    el = fem.LagrangeElement("quadrilateral", kphi)
    return np.array([float(phi_ref.subs({XI: p[0], ETA: p[1]})) for p in el.nodes])


def _poly(e):
    return sp.Poly(sp.expand(e), XI, ETA)


def _integrate(p):
    return sum(c / ((i + 1) * (j + 1)) for (i, j), c in p.terms())


def _dot(a, b):
    """sum of products of two lists of Polys (None = 0)."""
    out = None
    for u, v in zip(a, b):
        if u is None or v is None:
            continue
        out = u * v if out is None else out + u * v
    return out


def _basis_fields(verts, phi_ref):
    """For every mixed basis function (k, o), node-major: the fields of the forms (u, sigma(u), eps(u), y, div y, p phi
    for each material) as flat lists of Polys in (xi, eta), None = 0, with grad = J^-T grad_ref on the parallelogram;
    also grad phi and |det J|."""
    J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
    Jit = J.inv().T

    def grad(e):
        return list(Jit * sp.Matrix([sp.diff(e, XI), sp.diff(e, ETA)]))

    gphi = [_poly(g) for g in grad(phi_ref)]
    pphi = _poly(phi_ref)
    zero4, zero2 = [None] * 4, [None] * 2
    out = []
    for k in range(4):
        N, G = _poly(NQ1[k]), [_poly(g) for g in grad(NQ1[k])]
        for o in range(NB):
            fd = dict(ui=zero2, uo=zero2, si=zero4, ei=zero4, so=zero4, eo=zero4, yi=zero4, yo=zero4, dyi=zero2,
                      dyo=zero2, p=zero2)
            if o < 4:   # u_in / u_out component c: grad(u)_ij = delta_ic G_j
                c, side = o % 2, ("i" if o < 2 else "o")
                lm, mu = (LM_IN, MU_IN) if side == "i" else (LM_OUT, MU_OUT)
                gu = [[G[j] if i == c else None for j in range(2)] for i in range(2)]
                eps = [[_sum_half(gu[i][j], gu[j][i]) for j in range(2)] for i in range(2)]
                sig = [[_add(_scale(G[c], lm) if i == j else None, _scale(eps[i][j], 2 * mu)) for j in range(2)]
                       for i in range(2)]
                fd["u" + side] = [N if i == c else None for i in range(2)]
                fd["s" + side] = [sig[i][j] for i in range(2) for j in range(2)]
                fd["e" + side] = [eps[i][j] for i in range(2) for j in range(2)]
            elif o < 12:   # y_in / y_out entry (r, s): div(y)_i = delta_ir G_s
                side, loc = ("i" if o < 8 else "o"), (o - 4) % 4
                r, s = loc // 2, loc % 2
                fd["y" + side] = [N if (i, j) == (r, s) else None for i in range(2) for j in range(2)]
                fd["dy" + side] = [G[s] if i == r else None for i in range(2)]
            else:
                c = o - 12
                fd["p"] = [N * pphi if i == c else None for i in range(2)]     # p phi
            out.append(fd)
    return out, gphi, abs(J.det())


def _scale(p, c):
    return None if p is None else p * c


def _add(a, b):
    if a is None:
        return b
    return a if b is None else a + b


def _sum_half(a, b):
    s = _add(a, b)
    return None if s is None else s * R(1, 2)


def _derived(fd, gphi):
    """T_in = y_in + sigma_in(u_in), T_out, U = u_in - u_out, R = (y_in - y_out) grad phi."""
    Ti = [_add(a, b) for a, b in zip(fd["yi"], fd["si"])]
    To = [_add(a, b) for a, b in zip(fd["yo"], fd["so"])]
    U = [_add(a, _scale(b, -1)) for a, b in zip(fd["ui"], fd["uo"])]
    dy = [_add(a, _scale(b, -1)) for a, b in zip(fd["yi"], fd["yo"])]
    Rv = [_add(_scale(dy[2 * i], gphi[0]), _scale(dy[2 * i + 1], gphi[1])) for i in range(2)]
    return Ti, To, U, Rv


def _val(p):
    return sp.Integer(0) if p is None else _integrate(p)


def _reference_cell(kphi, tag):
    verts = _verts(X0, E1, E2)
    phi_ref = _phi_ref(kphi, 0)
    fds, gphi, det = _basis_fields(verts, phi_ref)
    fv = [[R(1, 3), R(-2, 5)], [R(3, 4), R(1, 7)], [R(-1, 2), R(2, 9)], [R(5, 6), R(-3, 8)]]
    fq = [_poly(sum(fv[k][c] * NQ1[k] for k in range(4))) for c in range(2)]
    h2 = _h2(verts)
    hf = sp.sqrt(h2)
    ins, outs, cut = tag in (1, 2), tag in (2, 3), tag == 2
    der = [_derived(fd, gphi) for fd in fds]
    A = np.zeros((56, 56))
    b = np.zeros(56)
    for a in range(56):
        fa = fds[a]
        Tia, Toa, Ua, Ra = der[a]
        bv = sp.Integer(0)
        if ins:
            bv += _val(_dot(fq, fa["ui"]))
        if outs:
            bv += _val(_dot(fq, fa["uo"]))
        if cut:
            bv += SIGMA_S * h2 * (_val(_dot(fq, fa["dyi"])) + _val(_dot(fq, fa["dyo"])))
        b[a] = float(sp.N(det * bv, 30))
        for bb in range(56):
            fb = fds[bb]
            Tib, Tob, Ub, Rb = der[bb]
            g0 = sp.Integer(0)
            if ins:
                g0 += _val(_dot(fb["si"], fa["ei"]))
            if outs:
                g0 += _val(_dot(fb["so"], fa["eo"]))
            if cut:
                g0 += GAMMA * (C_OUT * _val(_dot(Tib, Tia)) + C_IN * _val(_dot(Tob, Toa)))
                m2 = GAMMA * (_val(_dot(Rb, Ra)) + _val(_dot(Ub, Ua)))
                m3 = GAMMA * (_val(_dot(Ub, fa["p"])) + _val(_dot(fb["p"], Ua)))
                m4 = GAMMA * _val(_dot(fb["p"], fa["p"]))
                p2 = SIGMA_S * (_val(_dot(fb["dyi"], fa["dyi"])) + _val(_dot(fb["dyo"], fa["dyo"])))
                g0 = g0 + m2 / h2 + m3 / (h2 * hf) + m4 / (h2 * h2) + p2 * h2
            A[a, bb] = float(sp.N(det * g0, 30))
    return A, b, _to_np(verts), _interpolate(kphi, phi_ref), np.array([[float(c) for c in r] for r in fv])


@pytest.mark.parametrize("kphi", [1, 2])
def test_cell_tensors_match_sympy_on_parallelogram(kphi):
    """Cut (tag 2) and uncut (tags 1, 3) element tensors and load vectors at the kernels' rules, against the exact
    integrals of the literal integrands of the forms."""
    (cp, cw), (up, uw), _ = quadrature.rules_for_elasticity_quad(kphi)
    for tag in (1, 2, 3):
        A_ref, b_ref, x, phi, fv = _reference_cell(kphi, tag)
        A, b = OEQ.cell_tensors(x, np.array([[0, 1, 2, 3]]), phi[None], fv[None], np.array([tag]), MAT, 1.3, 0.7,
                                kphi, rule=(cp, cw), uncut_rule=(up, uw))
        assert np.abs(A[0] - A_ref).max() <= 1e-13 * np.abs(A_ref).max(), tag
        assert np.abs(b[0] - b_ref).max() <= 1e-13 * np.abs(b_ref).max(), tag
        if tag == 2:   # the penalty terms in h^-3 and h^-4 (p phi) are present
            p_rows = [k * NB + 12 + c for k in range(4) for c in range(2)]
            assert np.abs(A_ref[p_rows]).max() > 1e-3 * np.abs(A_ref).max()


def test_boundary_tensors_match_sympy_on_parallelogram():
    verts = _verts(X0, E1, E2)
    x = _to_np(verts)
    ents = np.array([[0, o] for o in range(4)])
    cen = sum(verts, sp.zeros(2, 1)) / 4
    for side, ou, oy in (("in", 0, 4), ("out", 2, 8)):
        A = OEQ.boundary_tensors(x, np.array([[0, 1, 2, 3]]), ents, side)
        for o in range(4):
            la, lb = OQ.QUAD_FACETS[o]
            t = verts[lb] - verts[la]
            nl = sp.Matrix([t[1], -t[0]])                      # length * outward normal
            if (nl.T * (verts[la] - cen))[0] < 0:
                nl = -nl
            ra, rb = OQ.REF_VERTICES[la], OQ.REF_VERTICES[lb]
            edge = {XI: (1 - S) * int(ra[0]) + S * int(rb[0]), ETA: (1 - S) * int(ra[1]) + S * int(rb[1])}
            ref = np.zeros((56, 56))
            for k in range(4):
                for j in range(4):
                    m = sp.integrate(sp.expand((NQ1[k] * NQ1[j]).subs(edge)), (S, 0, 1))
                    for c in range(2):
                        for s in range(2):
                            ref[k * NB + ou + c, j * NB + oy + 2 * c + s] = float(nl[s] * m)
            assert np.abs(A[o] - ref).max() <= 1e-14 * np.abs(ref).max(), (side, o)


def test_facet_tensors_match_sympy():
    """Two parallelograms sharing an edge, the second mirrored (negative det J): the macro tensor of
    sigma_s avg(h) int_F [sigma(u) n].[sigma(v) n] on both sides."""
    x0, e1, e2 = X0, E1, E2
    pts = [x0, x0 + e1, x0 + e2, x0 + e1 + e2, x0 + 2 * e1, x0 + 2 * e1 + e2]
    cells = np.array([[0, 1, 2, 3], [4, 1, 5, 3]])
    x = _to_np(pts)
    c2f, f2c, _ = OT.build_topology(cells.astype(np.int32), "quadrilateral")
    shared = [f for f in range(len(f2c)) if f2c[f, 1] >= 0]
    assert len(shared) == 1
    for side, ou, lm, mu in (("in", 0, LM_IN, MU_IN), ("out", 2, LM_OUT, MU_OUT)):
        E = OEQ.facet_tensors(x, cells, c2f, f2c, shared, side, MAT, 0.7)[0]
        # both cells see the shared edge x1 -> x3 at xi = 1, eta = s
        jumps, cols, hsum = [], [], 0
        for sc, cell in enumerate(cells[f2c[shared[0]]]):
            verts = [pts[k] for k in cell]
            J = sp.Matrix.hstack(verts[1] - verts[0], verts[2] - verts[0])
            Jit = J.inv().T
            n = Jit * sp.Matrix([1, 0])
            n = n / sp.sqrt((n.T * n)[0])
            for k in range(4):
                G = Jit * sp.Matrix([sp.diff(NQ1[k], XI), sp.diff(NQ1[k], ETA)])
                for c in range(2):
                    gu = sp.zeros(2, 2)
                    gu[c, :] = G.T
                    sig = lm * gu.trace() * sp.eye(2) + mu * (gu + gu.T)
                    jumps.append((sig * n).subs({XI: 1, ETA: S}))
                    cols.append(sc * 56 + k * NB + ou + c)
            hsum += sp.sqrt(_h2(verts))
        coef = SIGMA_S * hsum / 2 * sp.sqrt((e2.T * e2)[0])
        ref = np.zeros((112, 112))
        for a in range(16):
            for bb in range(16):
                ref[cols[a], cols[bb]] = float(sp.N(coef * sp.integrate(sp.expand((jumps[a].T * jumps[bb])[0]),
                                                                       (S, 0, 1)), 30))
        assert np.abs(E - ref).max() <= 1e-13 * np.abs(ref).max(), side


QX = np.array([[-0.31, 0.12], [0.47, 0.05], [-0.22, 0.83], [0.86, 0.61]])   # convex, not a parallelogram


@pytest.mark.parametrize("tag", [1, 3])
def test_uncut_stiffness_annihilates_rigid_modes(tag):
    """The two translations and the rotation (-y, x) are in the isoparametric Q1 space: on any cell, zero strain."""
    A, _ = OEQ.cell_tensors(QX, np.array([[0, 1, 2, 3]]), np.zeros((1, 4)), np.zeros((1, 4, 2)), np.array([tag]), MAT,
                            1.3, 0.7)
    ou = 0 if tag == 1 else 2
    idx = np.array([k * NB + ou + c for k in range(4) for c in range(2)])
    K = A[0][np.ix_(idx, idx)]
    assert np.abs(A[0]).sum() == np.abs(K).sum() and np.abs(K).max() > 0   # only the one material's block
    modes = [np.tile([1.0, 0.0], 4), np.tile([0.0, 1.0], 4), np.stack([-QX[:, 1], QX[:, 0]], axis=1).ravel()]
    for v in modes:
        assert np.abs(K @ v).max() <= 1e-14 * np.abs(K).max() * np.abs(v).max()
    assert np.abs(K @ np.stack([QX[:, 0], 0 * QX[:, 0]], axis=1).ravel()).max() > 1e-3 * np.abs(K).max()


def test_rules_for_elasticity_quad():
    for kphi in (1, 2):
        (cp, cw), (up, uw), (fp, fw) = quadrature.rules_for_elasticity_quad(kphi)
        assert cp.shape == ((kphi + 2) ** 2, 2) and up.shape == (4, 2) and fp.shape == (2, 2)
        for w in (cw, uw, fw):
            assert abs(w.sum() - 1.0) < 1e-15
        # the oracle's defaults are these rules
        for (p, w), (p2, w2) in (((cp, cw), OQ.gauss_square(kphi + 2)), ((up, uw), OQ.gauss_square(2))):
            assert np.abs(p - p2).max() < 1e-15 and np.abs(w - w2).max() < 1e-15
        t, wt = OQ.gauss_segment(2)
        assert np.abs(fp[:, 1] - t).max() < 1e-15 and np.abs(fw - wt).max() < 1e-15


def _cpu_problem(n=9):
    m = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(n, device="cpu"), jitter=0.2, seed=5)
    x, cells = m.x.numpy(), m.cells.numpy().astype(np.int64)
    phi = ((x - np.array([0.03, -0.02])) ** 2).sum(axis=1) - 0.6 ** 2
    ct = "quadrilateral"
    ftab = np.asarray([OT.coordinate_basis(ct, p)[0] for p in OT.facet_points_in_cell(ct, 1)])
    out = OT.compute_tags_measures(x, cells, ct, phi[cells], OT.point_values_function(phi, cells, ftab),
                                   box_mode=True, detection_points=OT.cell_detection_points(ct, 1))
    return m, x, cells, out


@pytest.mark.parametrize("kphi", [1, 2])
def test_elasticity_quad_symbolic_phase_matches_oracle_pattern(kphi):
    mesh, x, cells, out = _cpu_problem()
    assert set(np.unique(out["cell_tags"])) == {1, 2, 3}
    o = OE.Offsets(2)
    ct8 = torch.from_numpy(out["cell_tags"].astype(np.int8))
    ft8 = torch.from_numpy(out["facet_tags"].astype(np.int8))
    e100 = torch.from_numpy(np.asarray(out["ds100"], dtype=np.int32))
    e101 = torch.from_numpy(np.asarray(out["ds101"], dtype=np.int32))
    plan = elasticity.ElasticityPlan(mesh, ct8, ft8, e100, e101, fem.functionspace(mesh, kphi))
    assert plan.n_cell_points == (kphi + 2) ** 2
    mixed = OE.mixed_dofmap(cells, 2)
    interior = out["f2c"][:, 1] >= 0
    fac = np.nonzero(((out["facet_tags"] == 3) | (out["facet_tags"] == 4)) & interior)[0]
    ip, ix = OA.sparsity_pattern(o.nb * len(x), mixed, np.arange(len(cells)), fac, out["f2c"])
    assert plan.n_rows == o.nb * len(x) and plan.nb == o.nb == NB
    assert np.array_equal(plan.indptr.numpy(), ip) and np.array_equal(plan.indices.numpy(), ix)
    # the scalar slot maps address the blocked CSR the way the kernels do
    vptr = plan.vptr.numpy().astype(np.int64)
    pos = plan.pos_cells.numpy().reshape(len(cells), 4, 4)
    rng = np.random.default_rng(1)
    for _ in range(50):
        c, k, j = rng.integers(len(cells)), rng.integers(4), rng.integers(4)
        a, b = rng.integers(o.nb), rng.integers(o.nb)
        r = cells[c, k]
        addr = o.nb * (o.nb * vptr[r] + a * (vptr[r + 1] - vptr[r]) + pos[c, k, j]) + b
        assert ip[o.nb * r + a] <= addr < ip[o.nb * r + a + 1] and ix[addr] == o.nb * cells[c, j] + b
    f2c = out["f2c"]
    for facs, posf in ((plan.facets_in.numpy(), plan.pos_facets_in.numpy()),
                       (plan.facets_out.numpy(), plan.pos_facets_out.numpy())):
        assert len(facs) > 0
        mac = np.concatenate([cells[f2c[facs, 0]], cells[f2c[facs, 1]]], axis=1)     # [n, 8]
        posf = posf.reshape(len(facs), 8, 8)
        for _ in range(20):
            e, k, j = rng.integers(len(facs)), rng.integers(8), rng.integers(8)
            r = mac[e, k]
            addr = o.nb * (o.nb * vptr[r] + posf[e, k, j])
            assert ix[addr] == o.nb * mac[e, j]
    assert np.array_equal(np.sort(plan.facets_in.numpy()), np.nonzero((out["facet_tags"] == 3) & interior)[0])
    assert np.array_equal(np.sort(plan.facets_out.numpy()), np.nonzero((out["facet_tags"] == 4) & interior)[0])


def test_elasticity_quad_plan_refuses_a_cubic_level_set():
    mesh, _, _, out = _cpu_problem(4)
    t = lambda a, dt: torch.from_numpy(np.asarray(a, dtype=dt))   # noqa: E731
    args = (t(out["cell_tags"], np.int8), t(out["facet_tags"], np.int8), t(out["ds100"], np.int32),
            t(out["ds101"], np.int32))
    with pytest.raises(NotImplementedError):
        elasticity.ElasticityPlan(mesh, *args, fem.functionspace(mesh, 3))
