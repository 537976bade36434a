"""CPU oracle, quadrilaterals: the interface-elasticity phi-FEM operator in CSR (TEST INFRASTRUCTURE ONLY).

The forms of `oracle.elasticity` (reference demo/interface-elasticity/main.py:152-274) on quadrilateral meshes, with every
field of the mixed space (u_in, u_out, y_in, y_out, p) Q1 on the bilinear cell and a Q1 or Q2 level set.  Restated
independently of the CUDA kernels (csrc/assemble_elasticity.cu), field by field at quadrature points:

  * the bilinear cell map, J and J^-T at every point, basis values and gradients from `fem.LagrangeElement`
    (`oracle.assembly_quad` helpers);
  * the one-sided terms (y n).v by quadrature along the edge with the normal J^-T n_ref (the kernels use the closed form);
  * the stress jumps at physical points of the shared edge, pulled back into each cell by Newton's method on the bilinear
    map (the kernels map one edge parameter into both cells).

On a non-affine cell no integrand is polynomial, so the rules are arguments.  Their defaults are the kernels' rules
(`phifem_b200.quadrature.rules_for_elasticity_quad`): (kphi + 2)^2 Gauss points on cut cells, 2 x 2 on uncut cells,
2 Gauss points on the edges of the stress jump.  tests/test_oracle_elasticity_quad.py holds the element tensors on a
parallelogram to exact sympy integrals.

Mixed numbering as `oracle.elasticity` (NB = 14 dofs per vertex, global dof = NB vertex + o); cell-local order
node-major (local vertex k, offset o) -> k NB + o.
"""
import numpy as np

from oracle.assembly import _scatter, sparsity_pattern
from oracle.assembly_quad import (_Q1, QUAD_FACETS, REF_NORMALS, REF_VERTICES, cell_diameter, cell_map, gauss_segment,
                                  gauss_square, physical_gradients, pull_back, tabulate)
from oracle.elasticity import Material, Offsets, _sigma, apply_dirichlet, mixed_dofmap
from phifem_b200 import fem

NV, D = 4, 2
_O = Offsets(D)
NM = NV * _O.nb     # 56


def _fields(N, G):
    """Every mixed basis function of one cell at nq points (N [nq, 4], physical gradients G [nq, 4, 2]):
    u_in [q, m, 2], grad u_in [q, m, 2, 2] (grad(u)_ij = d_j u_i), the same for u_out, y_in [q, m, 2, 2],
    div y_in [q, m, 2], the same for y_out, p [q, m, 2]."""
    nq = len(N)
    z = lambda *s: np.zeros((nq, NM) + s)        # noqa: E731
    ui, gui, uo, guo = z(D), z(D, D), z(D), z(D, D)
    yi, dyi, yo, dyo, p = z(D, D), z(D), z(D, D), z(D), z(D)
    o = _O
    for k in range(NV):
        for c in range(D):
            for (u, gu, off) in ((ui, gui, o.ui), (uo, guo, o.uo)):
                m = k * o.nb + off + c
                u[:, m, c] = N[:, k]
                gu[:, m, c, :] = G[:, k, :]
            p[:, k * o.nb + o.p + c, c] = N[:, k]
            for s in range(D):
                for (y, dy, off) in ((yi, dyi, o.yi), (yo, dyo, o.yo)):
                    m = k * o.nb + off + c * D + s
                    y[:, m, c, s] = N[:, k]
                    dy[:, m, c] = G[:, k, s]
    return ui, gui, uo, guo, yi, dyi, yo, dyo, p


def cell_tensors(x, cells, phi_dofs, f_dofs, tags, mat, gamma, sigma_s, kphi=1, rule=None, uncut_rule=None):
    """Element tensors [n, 56, 56] and loads [n, 56] of the cells (tags in {1, 2, 3}); phi_dofs [n, nd_phi] and
    f_dofs [n, 4, 2] cell-local.  `rule` integrates the cut cells (tag 2), `uncut_rule` the others (reference points
    [nq, 2], weights summing to 1)."""
    cut_pts, cut_w = gauss_square(kphi + 2) if rule is None else (np.asarray(rule[0]), np.asarray(rule[1]))
    unc_pts, unc_w = gauss_square(2) if uncut_rule is None else (np.asarray(uncut_rule[0]), np.asarray(uncut_rule[1]))
    phi_el = fem.LagrangeElement("quadrilateral", kphi)
    out_A, out_b = [], []
    for c in range(len(cells)):
        t = tags[c]
        pts, w = (cut_pts, cut_w) if t == 2 else (unc_pts, unc_w)
        X = x[cells[c]]
        N, dN = tabulate(_Q1, pts)
        _, J, det = cell_map(X, pts)
        G = physical_gradients(J, dN)
        ui, gui, uo, guo, yi, dyi, yo, dyo, p = _fields(N, G)
        wq = w * np.abs(det)
        fq = N @ f_dofs[c]                                      # [q, 2]
        si, ei = _sigma(gui, mat.lmbda_in, mat.mu_in)
        so, eo = _sigma(guo, mat.lmbda_out, mat.mu_out)
        A = np.zeros((NM, NM))
        b = np.zeros(NM)
        if t in (1, 2):
            A += np.einsum("q,qbij,qaij->ab", wq, si, ei)
            b += np.einsum("q,qi,qai->a", wq, fq, ui)
        if t in (2, 3):
            A += np.einsum("q,qbij,qaij->ab", wq, so, eo)
            b += np.einsum("q,qi,qai->a", wq, fq, uo)
        if t == 2:
            pv, pg = tabulate(phi_el, pts)
            ph = pv @ phi_dofs[c]
            gph = np.einsum("qkr,k->qr", physical_gradients(J, pg), phi_dofs[c])
            h = cell_diameter(X)
            Ti, To = yi + si, yo + so
            R = np.einsum("qmij,qj->qmi", yi - yo, gph)
            S = ui - uo + p * (ph / h)[:, None, None]
            A += gamma * (mat.coef_out * np.einsum("q,qbij,qaij->ab", wq, Ti, Ti)
                          + mat.coef_in * np.einsum("q,qbij,qaij->ab", wq, To, To)
                          + np.einsum("q,qbi,qai->ab", wq, R, R) / h ** 2
                          + np.einsum("q,qbi,qai->ab", wq, S, S) / h ** 2)
            A += sigma_s * h ** 2 * (np.einsum("q,qbi,qai->ab", wq, dyi, dyi)
                                     + np.einsum("q,qbi,qai->ab", wq, dyo, dyo))
            b += sigma_s * h ** 2 * np.einsum("q,qi,qai->a", wq, fq, dyi + dyo)
        out_A.append(A)
        out_b.append(b)
    return np.array(out_A).reshape(-1, NM, NM), np.array(out_b).reshape(-1, NM)


def boundary_tensors(x, cells, ents, side, facet_rule=None):
    """int_F (y n).v on (cell, local facet) pairs by quadrature along the edge; side "in" (ds(100)) or "out"
    (ds(101)).  `facet_rule` = (parameters t [nq], weights summing to 1); default 2 Gauss points."""
    ents = np.asarray(ents).reshape(-1, 2)
    t, w = gauss_segment(2) if facet_rule is None else facet_rule
    out = np.zeros((len(ents), NM, NM))
    for e, (c, o) in enumerate(ents):
        X = x[cells[c]]
        a, b = QUAD_FACETS[o]
        pts = (1.0 - t)[:, None] * REF_VERTICES[a] + t[:, None] * REF_VERTICES[b]
        N, dN = tabulate(_Q1, pts)
        _, J, _ = cell_map(X, pts)
        n = np.einsum("qcr,c->qr", np.linalg.inv(J), REF_NORMALS[o])
        n /= np.linalg.norm(n, axis=1)[:, None]
        ds = w * np.linalg.norm(np.einsum("qrc,c->qr", J, REF_VERTICES[b] - REF_VERTICES[a]), axis=1)
        ui, _, uo, _, yi, _, yo, _, _ = _fields(N, physical_gradients(J, dN))
        u, y = (ui, yi) if side == "in" else (uo, yo)
        yn = np.einsum("qmij,qj->qmi", y, n)
        out[e] = np.einsum("q,qbi,qai->ab", ds, yn, u)
    return out


def facet_tensors(x, cells, c2f, f2c, facets, side, mat, sigma_s, facet_rule=None):
    """sigma_s avg(h) int_F [sigma(u) n].[sigma(v) n] over the macro dofs [cell +, cell -]; side "in" (sigma_in, u_in)
    or "out".  Quadrature at physical points of the edge (from its lower- to its higher-global-id vertex), pulled back
    into each cell."""
    facets = np.asarray(facets)
    t, w = gauss_segment(2) if facet_rule is None else facet_rule
    lmbda, mu = (mat.lmbda_in, mat.mu_in) if side == "in" else (mat.lmbda_out, mat.mu_out)
    E = np.zeros((len(facets), 2 * NM, 2 * NM))
    for e, f in enumerate(facets):
        cc = f2c[f]
        o0 = int(np.argmax(c2f[cc[0]] == f))
        a, b = (cells[cc[0]][k] for k in QUAD_FACETS[o0])
        lo, hi = x[min(a, b)], x[max(a, b)]
        length = np.linalg.norm(hi - lo)
        hs = 0.0
        Jmp = np.zeros((len(t), 2 * NM, D))
        for s in (0, 1):
            X = x[cells[cc[s]]]
            o = int(np.argmax(c2f[cc[s]] == f))
            hs += cell_diameter(X)
            for q, tq in enumerate(t):
                r = pull_back(X, (1.0 - tq) * lo + tq * hi)
                N, dN = tabulate(_Q1, r[None])
                _, J, _ = cell_map(X, r[None])
                n = np.linalg.inv(J[0]).T @ REF_NORMALS[o]
                n /= np.linalg.norm(n)
                _, gui, _, guo, *_ = _fields(N, physical_gradients(J, dN))
                sg, _ = _sigma(gui if side == "in" else guo, lmbda, mu)
                Jmp[q, s * NM:(s + 1) * NM] = np.einsum("mij,j->mi", sg[0], n)
        E[e] = sigma_s * 0.5 * hs * length * np.einsum("q,qai,qbi->ab", w, Jmp, Jmp)
    return E


def assemble_interface_elasticity_quad(x, cells, phi, f, cell_tags, facet_tags, c2f, f2c, ds100, ds101, mat=None,
                                       gamma=1.0, sigma_s=1.0, kphi=1, phi_dofmap=None, bc_dofs=None, bc_values=None,
                                       rule=None, uncut_rule=None, facet_rule=None):
    """(indptr, indices, data, b) of the operator in box mode on a quadrilateral mesh (arguments as
    `oracle.elasticity.assemble_interface_elasticity`; phi [n_dofs of the Q_kphi space], f [Nv, 2] nodal).  `rule`,
    `uncut_rule`: (reference points [nq, 2], weights summing to 1) of the cut / uncut cells; `facet_rule`: (parameters
    t [nq], weights summing to 1) of the stress-jump edges."""
    mat = mat or Material()
    x, cells = np.asarray(x), np.asarray(cells, dtype=np.int64)
    nvtx = len(x)
    mixed = mixed_dofmap(cells, D)
    n_rows = _O.nb * nvtx
    allc = np.nonzero(np.isin(cell_tags, (1, 2, 3)))[0]
    interior = f2c[:, 1] >= 0
    f3 = np.nonzero((facet_tags == 3) & interior)[0]
    f4 = np.nonzero((facet_tags == 4) & interior)[0]
    indptr, indices = sparsity_pattern(n_rows, mixed, allc, np.concatenate([f3, f4]), f2c)
    data = np.zeros(len(indices))
    b = np.zeros(n_rows)
    pdm = cells if phi_dofmap is None else np.asarray(phi_dofmap, dtype=np.int64)
    A, be = cell_tensors(x, cells[allc], phi[pdm[allc]], f[cells[allc]], cell_tags[allc], mat, gamma, sigma_s, kphi,
                         rule=rule, uncut_rule=uncut_rule)
    dm = mixed[allc]
    _scatter(indptr, indices, data, np.repeat(dm, NM, axis=1).ravel(), np.tile(dm, (1, NM)).ravel(), A.ravel())
    np.add.at(b, dm.ravel(), be.ravel())
    for ents, side in ((ds100, "in"), (ds101, "out")):
        ents = np.asarray(ents).reshape(-1, 2)
        if len(ents):
            dmb = mixed[ents[:, 0]]
            _scatter(indptr, indices, data, np.repeat(dmb, NM, axis=1).ravel(), np.tile(dmb, (1, NM)).ravel(),
                     boundary_tensors(x, cells, ents, side).ravel())
    for fac, side in ((f3, "in"), (f4, "out")):
        if len(fac):
            mac = np.concatenate([mixed[f2c[fac, 0]], mixed[f2c[fac, 1]]], axis=1)
            _scatter(indptr, indices, data, np.repeat(mac, 2 * NM, axis=1).ravel(), np.tile(mac, (1, 2 * NM)).ravel(),
                     facet_tensors(x, cells, c2f, f2c, fac, side, mat, sigma_s, facet_rule).ravel())
    if bc_dofs is not None and len(bc_dofs):
        apply_dirichlet(indptr, indices, data, b, np.asarray(bc_dofs), np.asarray(bc_values))
    return indptr, indices, data, b
