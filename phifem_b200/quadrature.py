"""Quadrature rules on the reference simplices (barycentric points, weights summing to 1).

dolfinx takes its rules from basix for the degree UFL estimates for each integrand
(reference demo/strong-dirichlet/flower/main.py:121,130: `dfx.fem.form(a)` / `form(L)`); the P_k kernels of
csrc/assemble_pk.cu take them as tables (`phifem_quadrature`).  Any rule exact to the integrand's degree gives
the same element tensors up to rounding, so the rules are chosen for point count:

  * segments : Gauss-Legendre;
  * triangles: Dunavant's fully symmetric 12-point rule for degree <= 6 (3-, 6-, 7-point rules below that);
  * tetrahedra: Keast's fully symmetric 24-point rule for degree 6, Walkington's 14-point rule for degrees 3-5 (1- and
    4-point rules below that);
  * anything else: collapsed (Stroud conical product) Gauss-Jacobi rules of the required order.

Every rule is checked against the exact monomial integrals at import of its first use; the orbit parameters
of the symmetric rules are polished by Newton iterations on those moment equations first, so the constants
below only need to be good starting points.  numpy only (Golub-Welsch for the Gauss-Jacobi nodes).
"""
import itertools
import math

import numpy as np


def gauss_jacobi(n, alpha):
    """n-point Gauss-Jacobi rule on [0, 1] for the weight (1 - t)^alpha (alpha = 0, 1, 2), exact to degree
    2n - 1; weights sum to 1 / (alpha + 1)."""
    k = np.arange(n, dtype=np.float64)
    a, b = float(alpha), 0.0
    # three-term recurrence of the Jacobi polynomials P^(a,b) on [-1, 1] (Golub-Welsch)
    with np.errstate(invalid="ignore", divide="ignore"):
        diag = (b * b - a * a) / ((2 * k + a + b) * (2 * k + a + b + 2))
    if a + b == 0.0:
        diag[0] = (b - a) / (a + b + 2)
    kk = k[1:]
    off = 2.0 / (2 * kk + a + b) * np.sqrt(kk * (kk + a) * (kk + b) * (kk + a + b)
                                           / ((2 * kk + a + b - 1) * (2 * kk + a + b + 1)))
    if n > 1 and a + b == 0.0:
        off[0] = 2.0 / (2 + a + b) * math.sqrt((1 + a) * (1 + b) / (3 + a + b))
    T = np.diag(diag) + np.diag(off, 1) + np.diag(off, -1)
    x, V = np.linalg.eigh(T)
    mu0 = 2.0 ** (a + b + 1) * math.gamma(a + 1) * math.gamma(b + 1) / math.gamma(a + b + 2)
    w = mu0 * V[0, :] ** 2
    # map [-1, 1] -> [0, 1]: t = (1 + x) / 2, weight (1 - x)^a -> 2^a (1 - t)^a
    return 0.5 * (x + 1.0), w / 2.0 ** (a + 1)


def conical_rule(d, n):
    """Collapsed Gauss-Jacobi product rule on the d-simplex with n^d points, exact to degree 2n - 1."""
    if d == 1:
        t, w = gauss_jacobi(n, 0)
        return np.stack([1 - t, t], axis=1), w
    if d == 2:
        a, wa = gauss_jacobi(n, 0)
        b, wb = gauss_jacobi(n, 1)
        X = (a[:, None] * (1 - b[None, :])).ravel()
        Y = np.repeat(b[None, :], n, axis=0).ravel()
        W = (wa[:, None] * wb[None, :]).ravel() * 2.0
        return np.stack([1 - X - Y, X, Y], axis=1), W
    a, wa = gauss_jacobi(n, 0)
    b, wb = gauss_jacobi(n, 1)
    c, wc = gauss_jacobi(n, 2)
    A, B, C = np.meshgrid(a, b, c, indexing="ij")
    X = (A * (1 - B) * (1 - C)).ravel()
    Y = (B * (1 - C)).ravel()
    Z = C.ravel()
    W = (wa[:, None, None] * wb[None, :, None] * wc[None, None, :]).ravel() * 6.0
    return np.stack([1 - X - Y - Z, X, Y, Z], axis=1), W


def monomial_integral(exps):
    """Integral of prod lambda_k^e_k over the simplex, normalised to unit measure."""
    d = len(exps) - 1
    return math.prod(math.factorial(e) for e in exps) * math.factorial(d) / math.factorial(sum(exps) + d)


def _moment_exponents(d, degree):
    return [e for tot in range(degree + 1) for e in itertools.product(range(tot + 1), repeat=d + 1)
            if sum(e) == tot and all(e[i] >= e[i + 1] for i in range(d))]


def max_moment_error(lam, w, degree):
    d = lam.shape[1] - 1
    err = 0.0
    for e in _moment_exponents(d, degree):
        err = max(err, abs(float((w * np.prod(lam ** np.array(e), axis=1)).sum()) - monomial_integral(e)))
    return err


# orbit descriptions: (kind, weight, parameters); kinds: "c" centroid, "s21"/"s31" (a, .., 1 - k a),
# "s111" (a, b, 1 - a - b), "s22" (a, a, 1/2 - a, 1/2 - a), "s211" (a, a, b, 1 - 2a - b)
_SYMMETRIC = {
    (2, 1): [("c", 1.0, ())],
    (2, 2): [("s21", 1.0 / 3.0, (1.0 / 6.0,))],
    (2, 4): [("s21", 0.223381589678011, (0.445948490915965,)), ("s21", 0.109951743655322, (0.091576213509771,))],
    (2, 6): [("s21", 0.116786275726379, (0.249286745170910,)), ("s21", 0.050844906370207, (0.063089014491502,)),
             ("s111", 0.082851075618374, (0.053145049844817, 0.310352451033784))],
    (3, 1): [("c", 1.0, ())],
    (3, 2): [("s31", 0.25, (0.138196601125011,))],
    # Walkington's 14-point rule, degree 5, positive weights
    (3, 5): [("s31", 0.112687925718016, (0.310885919263301,)), ("s31", 0.073493043116362, (0.092735250310891,)),
             ("s22", 0.042546020777081, (0.045503704125650,))],
    (3, 6): [("s31", 0.039922750258168, (0.214602871259152,)), ("s31", 0.010077211055321, (0.040673958534611,)),
             ("s31", 0.055357181543654, (0.322337890142276,)),
             ("s211", 0.048214285714286, (0.063661001875018, 0.603005664791649))],
}


def _expand(d, orbits):
    pts, wts = [], []
    for kind, w, par in orbits:
        if kind == "c":
            base = (1.0 / (d + 1),) * (d + 1)
        elif kind in ("s21", "s31"):
            a = par[0]
            base = (a,) * d + (1.0 - d * a,)
        elif kind == "s111":
            base = (par[0], par[1], 1.0 - par[0] - par[1])
        elif kind == "s22":
            base = (par[0], par[0], 0.5 - par[0], 0.5 - par[0])
        elif kind == "s211":
            base = (par[0], par[0], par[1], 1.0 - 2.0 * par[0] - par[1])
        else:
            raise ValueError(kind)
        perms = sorted(set(itertools.permutations(base)))
        pts.extend(perms)
        wts.extend([w] * len(perms))
    return np.array(pts), np.array(wts)


def _polish(d, degree, orbits):
    """Newton / Gauss-Newton on the moment equations in the orbit parameters (weights and positions)."""
    shapes = [(kind, len(par)) for kind, _, par in orbits]
    p = np.array([v for _, w, par in orbits for v in (w,) + tuple(par)], dtype=np.float64)
    exps = _moment_exponents(d, degree)
    target = np.array([monomial_integral(e) for e in exps])

    def unpack(q):
        out, k = [], 0
        for kind, npar in shapes:
            out.append((kind, q[k], tuple(q[k + 1:k + 1 + npar])))
            k += 1 + npar
        return out

    def resid(q):
        lam, w = _expand(d, unpack(q))
        return np.array([(w * np.prod(lam ** np.array(e), axis=1)).sum() for e in exps]) - target

    for _ in range(6):
        r = resid(p)
        J = np.empty((len(r), len(p)))
        for k in range(len(p)):
            h = 1e-7
            q = p.copy()
            q[k] += h
            J[:, k] = (resid(q) - r) / h
        step = np.linalg.lstsq(J, -r, rcond=None)[0]
        if not np.all(np.isfinite(step)):
            break
        p_new = p + step
        if np.abs(resid(p_new)).max() <= np.abs(r).max():
            p = p_new
        else:
            break
    return unpack(p)


_CACHE = {}


def simplex_rule(d, degree):
    """(points [nq, d+1] barycentric, weights [nq] summing to 1) exact for polynomials of `degree` on the
    d-simplex (d = 1, 2, 3)."""
    key = (d, int(degree))
    if key in _CACHE:
        return _CACHE[key]
    degree = max(1, int(degree))
    rule = None
    if d in (2, 3):
        cands = sorted(k for (dd, k) in _SYMMETRIC if dd == d and k >= degree)
        if cands:
            orbits = _polish(d, cands[0], _SYMMETRIC[(d, cands[0])])
            lam, w = _expand(d, orbits)
            if max_moment_error(lam, w, cands[0]) < 5e-16 and np.all(w > 0) and np.all(lam > 0):
                rule = (lam, w)
    if rule is None:
        n = degree // 2 + 1
        lam, w = conical_rule(d, n)
        if max_moment_error(lam, w, degree) > 1e-14:
            raise RuntimeError("quadrature: conical rule failed its moment check")
        rule = (lam, w)
    rule = (np.ascontiguousarray(rule[0]), np.ascontiguousarray(rule[1]))
    _CACHE[key] = rule
    return rule


def rules_for(d, kw, kphi):
    """Cell and facet rules of the strong-Dirichlet forms for P_kw trial/test functions and a P_kphi level
    set: cells need degree 2 (kw + kphi - 1) (stiffness; the load term f phi v has 2 kw + kphi, the
    stabilisation 2 (kw + kphi - 2)), facets 2 (kw + kphi) - 1 (one-sided term; the ghost penalty has
    2 (kw + kphi - 1))."""
    cell_degree = max(2 * (kw + kphi - 1), 2 * kw + kphi)
    facet_degree = 2 * (kw + kphi) - 1
    return simplex_rule(d, cell_degree), simplex_rule(d - 1, facet_degree)


def rules_for_weak(d, kw, kphi):
    """Cell and facet rules of the weak-Dirichlet forms (demo/weak-dirichlet/flower/main.py:112-151): the
    penalty block phi^2 p q needs degree 2 (kw + kphi) on cells; the facet terms (grad u.n) v and the gradient
    jumps need 2 kw - 1."""
    return simplex_rule(d, 2 * (kw + kphi)), simplex_rule(d - 1, max(1, 2 * kw - 1))


def rules_for_neumann(d, kphi):
    """Cell and facet rules of the Neumann forms (demo/neumann/square/main.py:117-158) for P1 u / y and a P_kphi
    level set: the penalty block (y.grad phi + p phi / h)^2 has degree 2 (kphi + 1) at most (|grad phi_h| in the
    load term is not polynomial for kphi = 2: integrated by the same rule); the facet terms are constant / linear."""
    return simplex_rule(d, 2 * (kphi + 1)), simplex_rule(d - 1, 2)


def square_rule(m):
    """m x m Gauss-Legendre product rule on the reference square [0, 1]^2: (points [m^2, 2] in reference coordinates
    (xi, eta), xi fastest; weights [m^2] summing to 1), exact for xi^a eta^b with a, b <= 2m - 1."""
    t, w = gauss_jacobi(int(m), 0)
    X, Y = np.meshgrid(t, t, indexing="xy")
    W = w[None, :] * w[:, None]
    return np.ascontiguousarray(np.stack([X.ravel(), Y.ravel()], axis=1)), np.ascontiguousarray(W.ravel())


def rules_for_neumann_quad(kphi):
    """Cell and facet rules of the Neumann forms on quadrilaterals for Q1 u / y and a Q_kphi level set: on a
    parallelogram the worst polynomial term, (y.grad phi)^2, has degree 2 (kphi + 1) in each reference direction, so
    kphi + 2 Gauss points per direction integrate every polynomial term exactly.  |grad phi_h| is not polynomial even
    for kphi = 1, and on a non-affine cell no integrand is: the operator is defined at this rule.  Facets: the 2-point
    segment rule (Q1 restricted to a straight edge is linear; on a parallelogram the gradient jumps are too)."""
    return square_rule(kphi + 2), simplex_rule(1, 2)


def rules_for_strong_quad(kphi):
    """Cell and facet rules of the strong-Dirichlet forms on quadrilaterals for Q1 w / v and a Q_kphi level set: on a
    parallelogram every integrand (stiffness, Hessian products, one-sided term, gradient jumps) is a polynomial of degree
    at most 2 (kphi + 1) per reference direction, and the load f phi v of degree kphi + 2: kphi + 2 Gauss points per
    direction on cells and a degree 2 kphi + 2 rule on edges are exact.  On a non-affine cell no integrand is
    polynomial: the operator is defined at these rules."""
    return square_rule(kphi + 2), simplex_rule(1, 2 * kphi + 2)


def rules_for_elasticity_quad(kphi):
    """Rules of the interface-elasticity forms on quadrilaterals (demo/interface-elasticity/main.py:181-269) for Q1
    fields and a Q_kphi level set: (cut-cell rule, uncut-cell rule, edge rule).

      * cut cells (tag 2), every term of a and L: (kphi + 2)^2 Gauss points, passed to the kernels in
        `phifem_quadrature`.  On a parallelogram the worst terms, (h^-1 p phi)^2 and ((y_in - y_out) grad phi)^2, have
        degree 2 (kphi + 1) per reference direction, so the rule is exact there;
      * uncut cells (tags 1 and 3), the stiffness of the one material and int f.v: 2 x 2 Gauss points (degree 2 per
        direction on a parallelogram), compile-time constants of the kernel;
      * the stress jump sigma_s avg(h) int [sigma(u) n].[sigma(v) n] over dS(3) / dS(4): 2 Gauss points on the edge
        (sigma(u) n is linear along the edge of a parallelogram), compile-time constants of the kernel.  Segment points
        are (1 - t, t), t running from the edge's lower-global-id vertex to the higher one.

    The one-sided terms int (y n).v over ds(100) / ds(101) are exact in closed form (Q1 restricted to a straight edge is
    linear).  On a cell that is not a parallelogram no integrand is polynomial: the operator is defined by these rules."""
    return square_rule(kphi + 2), square_rule(2), simplex_rule(1, 2)
