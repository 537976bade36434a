"""CPU oracle, quadrilaterals: the strong-Dirichlet phi-FEM operator with Q1 trial / test functions and a Q1 or Q2 level
set (TEST INFRASTRUCTURE ONLY).

The forms of reference demo/strong-dirichlet/flower/main.py:104-128 on the bilinear cell map, restated independently of
the CUDA kernels (csrc/assemble_quad.cu) with the conventions of `oracle.assembly_quad` (tensor-order vertices, the
bilinear map and J^-T at every point, basis and gradients from `fem.LagrangeElement`, ghost points pulled back into each
cell by Newton's method).  The result depends on the rule on a non-affine cell, so `rule` (cell) and `facet_rule` are
arguments; tests/test_oracle_quad_strong.py holds the element tensors on parallelograms to exact sympy integrals and the
physical Hessian on a non-parallelogram cell to high-precision central differences.
"""
import numpy as np

from oracle.assembly import _scatter, sparsity_pattern
from oracle.assembly_quad import (NV, QUAD_FACETS, REF_NORMALS, REF_VERTICES, _Q1, cell_diameter, cell_map,
                                  gauss_segment, gauss_square, physical_gradients, pull_back, tabulate)
from phifem_b200 import fem

# ---- forms -----------------------------------------------------------------------------------------------------------
#   a = int_{dx(1,2)} grad(phi w).grad(phi v) - int_{ds(100)} (grad(phi w).n) phi v
#       + sigma int_{dS(2,3)} avg(h) [grad(phi w).n][grad(phi v).n] + sigma h^2 int_{dx(2)} lap(phi w) lap(phi v)
#   L = int_{dx(1,2)} f phi v - sigma h^2 int_{dx(2)} f lap(phi v)
# with w, v, f in Q1 (vertex dofs) and phi in Q_kphi.  Second derivatives: the reference Hessians of the basis from the
# element's monomial coefficients, the map's second derivatives from the Q1 coordinate element, and the chain rule
# H = K^T (H_ref - sum_r (d^2 x_r / dref dref) du/dx_r) K with K = J^-1 -- not the closed form of the kernels.

def tabulate_hessians(element, pts):
    """Reference Hessians [nq, nd, 2, 2] of a Lagrange element at reference points [nq, 2]."""
    pts = np.atleast_2d(np.asarray(pts, dtype=np.float64))
    H = np.zeros((len(pts), element.ndofs, 2, 2))
    for a0 in range(2):
        for a1 in range(2):
            dm = np.zeros((len(pts), len(element.exps)))
            for m, e in enumerate(element.exps):
                e = list(e)
                c = 1.0
                for ax in (a0, a1):
                    c *= e[ax]
                    e[ax] -= 1
                if c == 0.0:
                    continue
                term = c * np.ones(len(pts))
                for d in range(2):
                    if e[d]:
                        term = term * pts[:, d] ** e[d]
                dm[:, m] = term
            H[:, :, a0, a1] = dm @ element.coef
    return H


def physical_hessians(J, d2x, dref, href):
    """Physical Hessians [nq, nd, 2, 2] from J [nq, 2, 2], the map's second derivatives d2x [nq, 2 (x_r), 2, 2], the
    reference gradients [nq, nd, 2] and reference Hessians [nq, nd, 2, 2] of the functions."""
    K = np.linalg.inv(J)                                   # K[c, r] = dref_c / dx_r
    M = href - np.einsum("qrij,qkr->qkij", d2x, physical_gradients(J, dref))
    return np.einsum("qir,qkij,qjs->qkrs", K, M, K)


def _strong_fields(X, pts, el, phi_c):
    """At reference points of one cell: Q1 values N, grad(phi psi_k) [nq, 4, 2], lap(phi psi_k) [nq, 4], phi, the
    physical map (x, J, det J)."""
    N, dN = tabulate(_Q1, pts)
    HN = tabulate_hessians(_Q1, pts)
    pv, pg = tabulate(el, pts)
    ph_ref = tabulate_hessians(el, pts)
    xq, J, det = cell_map(X, pts)
    d2x = np.einsum("kr,qkij->qrij", X, HN)
    G = physical_gradients(J, dN)
    lw = np.trace(physical_hessians(J, d2x, dN, HN), axis1=2, axis2=3)
    ph = pv @ phi_c
    gph = np.einsum("qkr,k->qr", physical_gradients(J, pg), phi_c)
    lph = np.trace(np.einsum("qkrs,k->qrs", physical_hessians(J, d2x, pg, ph_ref), phi_c), axis1=1, axis2=2)
    GU = N[:, :, None] * gph[:, None, :] + ph[:, None, None] * G
    LU = N * lph[:, None] + 2.0 * np.einsum("qr,qkr->qk", gph, G) + ph[:, None] * lw
    return N, GU, LU, ph, gph, G, J, det


def strong_cell_tensors(x, cells, phi_dofs, f_dofs, cut, sigma, kphi, rule=None):
    """Element tensors [n, 4, 4] and loads [n, 4] of dx((1,2)) (+ the Hessian terms of dx(2) on cut cells) by `rule`
    (reference points [nq, 2], weights summing to 1; default: (kphi + 2)^2 Gauss-Legendre points)."""
    pts, w = gauss_square(kphi + 2) if rule is None else (np.asarray(rule[0]), np.asarray(rule[1]))
    el = fem.LagrangeElement("quadrilateral", kphi)
    out_A, out_b = [], []
    for c in range(len(cells)):
        X = x[cells[c]]
        N, GU, LU, ph, _, _, _, det = _strong_fields(X, pts, el, phi_dofs[c])
        wq = w * np.abs(det)
        fq = N @ f_dofs[c]
        A = np.einsum("q,qad,qbd->ab", wq, GU, GU)
        b = np.einsum("q,q,q,qa->a", wq, fq, ph, N)
        if cut[c]:
            sh2 = sigma * cell_diameter(X) ** 2
            A += sh2 * np.einsum("q,qa,qb->ab", wq, LU, LU)
            b -= sh2 * np.einsum("q,q,qa->a", wq, fq, LU)
        out_A.append(A)
        out_b.append(b)
    return np.array(out_A).reshape(-1, NV, NV), np.array(out_b).reshape(-1, NV)


def _edge_normal(J, o):
    n = np.einsum("qcr,c->qr", np.linalg.inv(J), REF_NORMALS[o])
    return n / np.linalg.norm(n, axis=1)[:, None]


def strong_boundary_tensors(x, cells, phi_dofs, ents, kphi, facet_rule=None):
    """-int_F (grad(phi w).n) phi v on (cell, local facet) pairs by quadrature along the edge; phi_dofs [n, nd] of the
    entities' cells."""
    ents = np.asarray(ents).reshape(-1, 2)
    t, w = gauss_segment(kphi + 2) if facet_rule is None else facet_rule
    el = fem.LagrangeElement("quadrilateral", kphi)
    A = np.zeros((len(ents), NV, NV))
    for e, (c, o) in enumerate(ents):
        X = x[cells[c]]
        a, b = QUAD_FACETS[o]
        pts = (1.0 - t)[:, None] * REF_VERTICES[a] + t[:, None] * REF_VERTICES[b]
        N, GU, _, ph, _, _, J, _ = _strong_fields(X, pts, el, phi_dofs[e])
        n = _edge_normal(J, o)
        ds = w * np.linalg.norm(np.einsum("qrc,c->qr", J, REF_VERTICES[b] - REF_VERTICES[a]), axis=1)
        gun = np.einsum("qjr,qr->qj", GU, n)
        A[e] = -np.einsum("q,q,qi,qj->ij", ds, ph, N, gun)
    return A


def strong_ghost_tensors(x, cells, phi, phi_dofmap, c2f, f2c, facets, sigma, kphi, facet_rule=None):
    """sigma avg(h) int_F [grad(phi w).n][grad(phi v).n] over macro dofs [Q1 dofs of cell +, of cell -] [n, 8, 8]; the
    edge points are pulled back into each cell by Newton's method, phi evaluated from each side's own dofs."""
    facets = np.asarray(facets)
    t, w = gauss_segment(kphi + 2) if facet_rule is None else facet_rule
    el = fem.LagrangeElement("quadrilateral", kphi)
    E = np.zeros((len(facets), 2 * NV, 2 * NV))
    for e, f in enumerate(facets):
        cc = f2c[f]
        o0 = int(np.argmax(c2f[cc[0]] == f))
        a, b = (cells[cc[0]][k] for k in QUAD_FACETS[o0])
        lo, hi = x[min(a, b)], x[max(a, b)]
        length = np.linalg.norm(hi - lo)
        hs = 0.0
        Jmp = np.zeros((len(t), 2 * NV))
        for side in (0, 1):
            X = x[cells[cc[side]]]
            o = int(np.argmax(c2f[cc[side]] == f))
            hs += cell_diameter(X)
            pts = np.array([pull_back(X, (1.0 - tq) * lo + tq * hi) for tq in t])
            _, GU, _, _, _, _, J, _ = _strong_fields(X, pts, el, phi[phi_dofmap[cc[side]]])
            Jmp[:, side * NV:(side + 1) * NV] = np.einsum("qjr,qr->qj", GU, _edge_normal(J, o))
        E[e] = sigma * 0.5 * hs * length * np.einsum("q,qa,qb->ab", w, Jmp, Jmp)
    return E


def assemble_strong_dirichlet_quad(x, cells, phi, f, cell_tags, facet_tags, c2f, f2c, ds100, sigma=1.0, kphi=1,
                                   phi_dofmap=None, rule=None, facet_rule=None):
    """(indptr, indices, data, b) of the strong-Dirichlet operator on a quadrilateral mesh in box mode, Q1 w / v / f
    (dof = vertex id), Q_kphi level set.  `rule` = (reference points [nq, 2], weights summing to 1) of the cells,
    `facet_rule` = (parameters t [nq], weights summing to 1) of the edges."""
    x, cells = np.asarray(x), np.asarray(cells, dtype=np.int64)
    n_rows = len(x)
    phi_dofmap = cells if phi_dofmap is None else np.asarray(phi_dofmap, dtype=np.int64)
    active = np.nonzero((cell_tags == 1) | (cell_tags == 2))[0]
    ghost = np.nonzero(((facet_tags == 2) | (facet_tags == 3)) & (f2c[:, 1] >= 0))[0]
    ents = np.asarray(ds100).reshape(-1, 2)
    indptr, indices = sparsity_pattern(n_rows, cells, active, ghost, f2c)
    data = np.zeros(len(indices))
    b = np.zeros(n_rows)
    A, be = strong_cell_tensors(x, cells[active], phi[phi_dofmap[active]], f[cells[active]], cell_tags[active] == 2,
                                sigma, kphi, rule=rule)
    dm = cells[active]
    _scatter(indptr, indices, data, np.repeat(dm, NV, axis=1).ravel(), np.tile(dm, (1, NV)).ravel(), A.ravel())
    np.add.at(b, dm.ravel(), be.ravel())
    if len(ents):
        Ab = strong_boundary_tensors(x, cells, phi[phi_dofmap[ents[:, 0]]], ents, kphi, facet_rule)
        dmb = cells[ents[:, 0]]
        _scatter(indptr, indices, data, np.repeat(dmb, NV, axis=1).ravel(), np.tile(dmb, (1, NV)).ravel(), Ab.ravel())
    if len(ghost):
        Eg = strong_ghost_tensors(x, cells, phi, phi_dofmap, c2f, f2c, ghost, sigma, kphi, facet_rule)
        mac = np.concatenate([cells[f2c[ghost, 0]], cells[f2c[ghost, 1]]], axis=1)
        _scatter(indptr, indices, data, np.repeat(mac, 2 * NV, axis=1).ravel(), np.tile(mac, (1, 2 * NV)).ravel(),
                 Eg.ravel())
    return indptr, indices, data, b
