"""CPU oracle, quadrilaterals: the Neumann phi-FEM operator on the mixed space (u, y, p) in Q1 x Q1^2 x DG0 with a Q1
or Q2 level set (TEST INFRASTRUCTURE ONLY).

Same forms as `oracle.assembly.assemble_neumann` (reference demo/neumann/square/main.py:103-158, Robin variant
demo/robin/square/main.py:118-174) on the demo's own cell type.  Restated independently of the CUDA kernels
(csrc/assemble_quad.cu):

  * the bilinear cell map, its Jacobian and J^-T at every point, from the Q1 coordinate element;
  * basis values AND reference gradients from `fem.LagrangeElement("quadrilateral", k)` (its monomial coefficients,
    differentiated here), not from hand-written tensor-product formulas;
  * the one-sided term (y.n) v by quadrature along the edge with the normal J^-T n_ref;
  * the ghost penalty at physical points of the shared edge, pulled back into each cell by Newton's method on the
    bilinear map (the kernels map one edge parameter into both cells instead).

On a non-affine cell no integrand is polynomial, and |grad phi_h| is not polynomial even for a Q1 level set: the
result depends on the rule, so `rule` (cell) and `facet_rule` are arguments; the tests pass the kernels' rules.
tests/test_oracle_quad.py holds the element tensors on parallelograms to exact sympy integrals.

Cell-local mixed order [u x4, y node-major x8, p] (NM = 13); global numbering u at vertex s -> 3 s, y_c -> 3 s + 1 + c,
p of cell k -> 3 Nv + k.  (`oracle.assembly.neumann_mixed_dofmap` derives d from cells.shape[1] and does not apply.)
"""
import numpy as np

from oracle.assembly import _scatter, sparsity_pattern
from phifem_b200 import fem

NV, NM = 4, 13
# local facets of the tensor-order quadrilateral and their reference outward normals
QUAD_FACETS = ((0, 1), (0, 2), (1, 3), (2, 3))
REF_NORMALS = np.array([[0.0, -1.0], [-1.0, 0.0], [1.0, 0.0], [0.0, 1.0]])
REF_VERTICES = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]])


def tabulate(element, pts):
    """Values [nq, nd] and reference gradients [nq, nd, 2] of a Lagrange element at reference points [nq, 2]."""
    pts = np.atleast_2d(np.asarray(pts, dtype=np.float64))
    vals = element.tabulate(pts, snap=False)
    grads = np.zeros((len(pts), element.ndofs, 2))
    for axis in range(2):
        dm = np.zeros((len(pts), len(element.exps)))
        for m, e in enumerate(element.exps):
            if e[axis] == 0:
                continue
            term = e[axis] * np.ones(len(pts))
            for d in range(2):
                p = e[d] - (1 if d == axis else 0)
                if p:
                    term = term * pts[:, d] ** p
            dm[:, m] = term
        grads[:, :, axis] = dm @ element.coef
    return vals, grads


_Q1 = fem.LagrangeElement("quadrilateral", 1)


def cell_map(X, pts):
    """Bilinear map of one cell (vertices X [4, 2], tensor order) at reference points [nq, 2]:
    (physical points [nq, 2], J [nq, 2, 2] with J[r, c] = dx_r / dref_c, det J [nq])."""
    N, dN = tabulate(_Q1, pts)
    J = np.einsum("kr,qkc->qrc", X, dN)
    return N @ X, J, np.linalg.det(J)


def physical_gradients(J, dref):
    """grad = J^-T grad_ref for reference gradients [nq, nd, 2]."""
    return np.einsum("qkc,qcr->qkr", dref, np.linalg.inv(J))


def cell_diameter(X):
    """UFL CellDiameter of a degree-1 coordinate element: the largest vertex-pair distance."""
    return max(np.linalg.norm(X[a] - X[b]) for a in range(NV) for b in range(a + 1, NV))


def gauss_square(m):
    t, w = np.polynomial.legendre.leggauss(m)
    t, w = 0.5 * (t + 1.0), 0.5 * w
    X, Y = np.meshgrid(t, t, indexing="xy")
    return np.stack([X.ravel(), Y.ravel()], axis=1), (w[None, :] * w[:, None]).ravel()


def gauss_segment(m=2):
    t, w = np.polynomial.legendre.leggauss(m)
    return 0.5 * (t + 1.0), 0.5 * w


def neumann_mixed_dofmap_quad(cells, n_vertices):
    c = np.asarray(cells, dtype=np.int64)
    u = 3 * c
    y = (3 * c[:, :, None] + 1 + np.arange(2)[None, None, :]).reshape(len(c), -1)
    p = 3 * n_vertices + np.arange(len(c), dtype=np.int64)[:, None]
    return np.concatenate([u, y, p], axis=1)


def _fields(N, G, ph, gph, h, kappa):
    """Per point and mixed basis function: u, grad u, s1 = y + grad u, s2 = div y + u,
    s3 = y.grad phi - kappa |grad phi| u + h^-1 p phi."""
    nq = len(N)
    U, S2, S3 = np.zeros((nq, NM)), np.zeros((nq, NM)), np.zeros((nq, NM))
    GU, S1 = np.zeros((nq, NM, 2)), np.zeros((nq, NM, 2))
    ngp = np.sqrt((gph ** 2).sum(axis=1))
    for j in range(NV):
        U[:, j] = N[:, j]
        GU[:, j] = G[:, j]
        S1[:, j] = G[:, j]
        S2[:, j] = N[:, j]
        S3[:, j] = -kappa * ngp * N[:, j]
        for c in range(2):
            k = NV + 2 * j + c
            S1[:, k, c] = N[:, j]
            S2[:, k] = G[:, j, c]
            S3[:, k] = N[:, j] * gph[:, c]
    S3[:, NM - 1] = ph / h
    return U, GU, S1, S2, S3, ngp


def cell_tensors(x, cells, phi_dofs, f_dofs, un_dofs, cut, gamma, kphi, rule=None, kappa=0.0):
    """Element tensors [n, 13, 13] and loads [n, 13] of dx((1,2)) (+ dx(2) for cut cells) by `rule` (reference points
    [nq, 2], weights summing to 1; default: (kphi + 2)^2 Gauss-Legendre points)."""
    pts, w = gauss_square(kphi + 2) if rule is None else (np.asarray(rule[0]), np.asarray(rule[1]))
    Nq, dN = tabulate(_Q1, pts)
    pv, pg = tabulate(fem.LagrangeElement("quadrilateral", kphi), pts)
    out_A, out_b = [], []
    for c in range(len(cells)):
        X = x[cells[c]]
        _, J, det = cell_map(X, pts)
        G = physical_gradients(J, dN)
        ph = pv @ phi_dofs[c]
        gph = np.einsum("qkr,k->qr", physical_gradients(J, pg), phi_dofs[c])
        h = cell_diameter(X)
        U, GU, S1, S2, S3, ngp = _fields(Nq, G, ph, gph, h, kappa)
        wq = w * np.abs(det)
        fq, uq = Nq @ f_dofs[c], Nq @ un_dofs[c]
        A = np.einsum("q,qad,qbd->ab", wq, GU, GU) + np.einsum("q,qa,qb->ab", wq, U, U)
        b = np.einsum("q,q,qa->a", wq, fq, U)
        if cut[c]:
            A += gamma * (np.einsum("q,qad,qbd->ab", wq, S1, S1) + np.einsum("q,qa,qb->ab", wq, S2, S2)
                          + np.einsum("q,qa,qb->ab", wq, S3, S3) / h ** 2)
            b += gamma * (-np.einsum("q,q,q,qa->a", wq, uq, ngp, S3) / h ** 2 + np.einsum("q,q,qa->a", wq, fq, S2))
        out_A.append(A)
        out_b.append(b)
    return np.array(out_A).reshape(-1, NM, NM), np.array(out_b).reshape(-1, NM)


def boundary_tensors(x, cells, ents, facet_rule=None):
    """int_F (y.n) v on (cell, local facet) pairs by quadrature along the edge: rows u_i, columns y_(j,c)."""
    ents = np.asarray(ents).reshape(-1, 2)
    t, w = gauss_segment(2) if facet_rule is None else facet_rule
    A = np.zeros((len(ents), NM, NM))
    for e, (c, o) in enumerate(ents):
        X = x[cells[c]]
        a, b = QUAD_FACETS[o]
        pts = (1.0 - t)[:, None] * REF_VERTICES[a] + t[:, None] * REF_VERTICES[b]
        N, _ = tabulate(_Q1, pts)
        _, J, _ = cell_map(X, pts)
        n = np.einsum("qcr,c->qr", np.linalg.inv(J), REF_NORMALS[o])
        n /= np.linalg.norm(n, axis=1)[:, None]
        ds = w * np.linalg.norm(np.einsum("qrc,c->qr", J, REF_VERTICES[b] - REF_VERTICES[a]), axis=1)
        for i in range(NV):
            for j in range(NV):
                for cc in range(2):
                    A[e, i, NV + 2 * j + cc] = np.sum(ds * n[:, cc] * N[:, i] * N[:, j])
    return A


def pull_back(X, p, iters=30):
    """Reference coordinates of the physical point p in the (convex) cell X: Newton on the bilinear map."""
    r = np.array([0.5, 0.5])
    for _ in range(iters):
        xr, J, _ = cell_map(X, r[None])
        step = np.linalg.solve(J[0], xr[0] - p)
        r = r - step
        if np.abs(step).max() < 1e-16:
            break
    return r


def ghost_tensors(x, cells, c2f, f2c, facets, sigma, facet_rule=None):
    """sigma avg(h) int_F [grad u.n][grad v.n] over macro dofs [mixed dofs of cell +, of cell -]; u-u entries only."""
    facets = np.asarray(facets)
    t, w = gauss_segment(2) if facet_rule is None else facet_rule
    E = np.zeros((len(facets), 2 * NM, 2 * NM))
    for e, f in enumerate(facets):
        cc = f2c[f]
        o0 = int(np.argmax(c2f[cc[0]] == f))
        a, b = (cells[cc[0]][k] for k in QUAD_FACETS[o0])
        lo, hi = x[min(a, b)], x[max(a, b)]
        length = np.linalg.norm(hi - lo)
        hs = 0.0
        Jmp = np.zeros((len(t), 2 * NM))
        for side in (0, 1):
            X = x[cells[cc[side]]]
            o = int(np.argmax(c2f[cc[side]] == f))
            hs += cell_diameter(X)
            for q, tq in enumerate(t):
                r = pull_back(X, (1.0 - tq) * lo + tq * hi)
                _, dN = tabulate(_Q1, r[None])
                _, J, _ = cell_map(X, r[None])
                n = np.linalg.inv(J[0]).T @ REF_NORMALS[o]
                n /= np.linalg.norm(n)
                Jmp[q, side * NM:side * NM + NV] = physical_gradients(J, dN)[0] @ n
        E[e] = sigma * 0.5 * hs * length * np.einsum("q,qa,qb->ab", w, Jmp, Jmp)
    return E


def assemble_neumann_quad(x, cells, phi, f, un, cell_tags, facet_tags, c2f, f2c, ds100, gamma=1.0, sigma=1.0, kphi=1,
                          phi_dofmap=None, rule=None, facet_rule=None, robin_coef=0.0, ghost_tag=3):
    """(indptr, indices, data, b) of the Neumann (robin_coef = 0, ghost_tag = 3) or Robin (ghost_tag = 2) operator on
    a quadrilateral mesh in box mode.  `rule` = (reference points [nq, 2], weights summing to 1) of the cells,
    `facet_rule` = (parameters t [nq], weights summing to 1) of the edges."""
    x, cells = np.asarray(x), np.asarray(cells, dtype=np.int64)
    nvtx = len(x)
    mixed = neumann_mixed_dofmap_quad(cells, nvtx)
    n_rows = 3 * nvtx + len(cells)
    phi_dofmap = cells if phi_dofmap is None else np.asarray(phi_dofmap, dtype=np.int64)
    active = np.nonzero((cell_tags == 1) | (cell_tags == 2))[0]
    ghost = np.nonzero((facet_tags == ghost_tag) & (f2c[:, 1] >= 0))[0]
    ents = np.asarray(ds100).reshape(-1, 2)
    indptr, indices = sparsity_pattern(n_rows, mixed, active, ghost, f2c)
    data = np.zeros(len(indices))
    b = np.zeros(n_rows)
    A, be = cell_tensors(x, cells[active], phi[phi_dofmap[active]], f[cells[active]], un[cells[active]],
                         cell_tags[active] == 2, gamma, kphi, rule=rule, kappa=robin_coef)
    dm = mixed[active]
    _scatter(indptr, indices, data, np.repeat(dm, NM, axis=1).ravel(), np.tile(dm, (1, NM)).ravel(), A.ravel())
    np.add.at(b, dm.ravel(), be.ravel())
    if len(ents):
        Ab = boundary_tensors(x, cells, ents, facet_rule)
        dmb = mixed[ents[:, 0]]
        _scatter(indptr, indices, data, np.repeat(dmb, NM, axis=1).ravel(), np.tile(dmb, (1, NM)).ravel(), Ab.ravel())
    if len(ghost):
        Eg = ghost_tensors(x, cells, c2f, f2c, ghost, sigma, facet_rule)
        mac = np.concatenate([mixed[f2c[ghost, 0]], mixed[f2c[ghost, 1]]], axis=1)
        _scatter(indptr, indices, data, np.repeat(mac, 2 * NM, axis=1).ravel(), np.tile(mac, (1, 2 * NM)).ravel(),
                 Eg.ravel())
    return indptr, indices, data, b
