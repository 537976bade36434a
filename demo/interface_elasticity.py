#!/usr/bin/env python
"""The reference's interface-elasticity demo on the GPU (BASELINE.json configs[3]):

    python demo/interface_elasticity.py [--mesh-size 0.2] [--iterations 4] [--solver direct|bicgstab]
                                        [--cell-type triangle|quadrilateral]

mirrors `python main.py param1` of reference demo/interface-elasticity/main.py with param1.yaml: background mesh of the
box [-1.5, 1.5]^2 (main.py:92-107), tags in box mode (:111-115), mixed space (u_in, u_out, y_in, y_out, p) (:119-129),
Dirichlet condition on u_in on the box boundary (:160-179), forms (:181-269), solve (:240-286), the two displacements
combined (:288-321), relative L2 / H1_0 errors against the exact solution of data.py:43-48 (:325-397; here by quadrature
on the cells instead of a P3 interpolant), uniform refinement between iterations.

The tags and the assembly (matrix, right-hand side, lifting) run on the GPU; the linear solve is the step after the
path: `direct` hands the CSR system to scipy's sparse LU on the host (the reference uses MUMPS), `bicgstab` keeps it on
the GPU (Jacobi-BiCGStab; the least-squares penalty terms make the system ill-conditioned, so expect many iterations).

--cell-type quadrilateral runs the same steps on n^2 quadrilaterals of the same box: every field of the mixed space and
the level set Q1; the errors are integrated by 4 x 4 Gauss points on the bilinear cells.
"""
import argparse
import os
import sys
import warnings

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phifem_b200 import elasticity, fem, quadrature, solve, synthetic  # noqa: E402
from phifem.mesh_scripts import compute_tags_measures  # noqa: E402


def levelset(x):
    """data.py:39-40 (x: [n, 2] tensor or array)."""
    return 1.0 - (x[:, 0] ** 2 + x[:, 1] ** 2)


def exact_solution(X, mat):
    """data.py:43-48, and its gradient d_j u (both components of u are equal)."""
    r = np.sqrt(X[:, 0] ** 2 + X[:, 1] ** 2)
    scale = np.where(r < 1.0, mat.E_in / mat.E_out, 1.0)
    val = (np.cos(r) - np.cos(1.0) / mat.E_in) * scale
    grad = (-np.sinc(r / np.pi) * scale)[:, None] * X        # sin(r) / r, finite at the origin
    return np.stack([val, val], axis=1), grad


def source_term(X, mat):
    """f = -div(sigma_in(cos_vec(x))) / E_in (main.py:148-150) for u = (cos r, cos r):
    (div sigma)_i = (lmbda + mu) d_i (d_x c + d_y c) + mu lap c."""
    r0 = np.sqrt(X[:, 0] ** 2 + X[:, 1] ** 2)
    r = np.maximum(r0, 1e-8)
    c1, c2 = -np.sin(r), -np.cos(r)
    H = np.empty((len(X), 2, 2))
    for i in range(2):
        for j in range(2):
            H[:, i, j] = c2 * X[:, i] * X[:, j] / r ** 2 + c1 * ((i == j) / r - X[:, i] * X[:, j] / r ** 3)
            H[r0 < 1e-8, i, j] = -float(i == j)              # the Hessian of cos(r) at the origin
    div = (mat.lmbda_in + mat.mu_in) * H.sum(axis=2) + mat.mu_in * (H[:, 0, 0] + H[:, 1, 1])[:, None]
    return -div / mat.E_in


def errors(mesh, tags, u_in, u_out, mat):
    """Relative L2 and H1_0 errors of the combined solution: u_in on the cells tagged 1, u_out on the cells tagged 3."""
    lam, wq = quadrature.simplex_rule(2, 4)
    X = mesh.x.cpu().numpy()
    cells = mesh.cells.cpu().numpy()
    l2 = h1 = n_l2 = n_h1 = 0.0
    for tag, uh in ((1, u_in), (3, u_out)):
        cc = cells[tags == tag]
        xc = X[cc]
        e = xc[:, 1:] - xc[:, :1]
        det = e[:, 0, 0] * e[:, 1, 1] - e[:, 0, 1] * e[:, 1, 0]
        area = 0.5 * np.abs(det)
        G = np.empty((len(cc), 3, 2))                       # grad(lambda_k)
        G[:, 1] = np.stack([e[:, 1, 1], -e[:, 1, 0]], axis=1) / det[:, None]
        G[:, 2] = np.stack([-e[:, 0, 1], e[:, 0, 0]], axis=1) / det[:, None]
        G[:, 0] = -G[:, 1] - G[:, 2]
        gh = np.einsum("mkc,mkj->mcj", uh[cc], G)           # d_j u_c, constant per cell
        xq = np.einsum("qv,mvd->qmd", lam, xc).reshape(-1, 2)
        ue, ge = exact_solution(xq, mat)
        ue, ge = ue.reshape(len(wq), len(cc), 2), ge.reshape(len(wq), len(cc), 2)
        uq = np.einsum("qv,mvc->qmc", lam, uh[cc])
        w = wq[:, None] * area[None, :]
        l2 += float((w[:, :, None] * (uq - ue) ** 2).sum())
        n_l2 += float((w[:, :, None] * ue ** 2).sum())
        h1 += float((w[:, :, None, None] * (gh[None] - ge[:, :, None, :]) ** 2).sum())
        n_h1 += float((w[:, :, None, None] * np.repeat(ge[:, :, None, :], 2, axis=2) ** 2).sum())
    return (l2 / n_l2) ** 0.5, (h1 / n_h1) ** 0.5


def errors_quad(mesh, tags, u_in, u_out, mat):
    """`errors` on a quadrilateral mesh: 4 x 4 Gauss points on each bilinear cell, Q1 values and physical gradients
    J^-T grad_ref at every point."""
    pts, wq = quadrature.square_rule(4)
    xi, eta = pts[:, 0], pts[:, 1]
    N = np.stack([(1 - xi) * (1 - eta), xi * (1 - eta), (1 - xi) * eta, xi * eta], axis=1)            # [q, 4]
    dN = np.stack([np.stack([-(1 - eta), 1 - eta, -eta, eta], axis=1),
                   np.stack([-(1 - xi), -xi, 1 - xi, xi], axis=1)], axis=2)                           # [q, 4, 2]
    X = mesh.x.cpu().numpy()
    cells = mesh.cells.cpu().numpy()
    l2 = h1 = n_l2 = n_h1 = 0.0
    for tag, uh in ((1, u_in), (3, u_out)):
        cc = cells[tags == tag]
        xc = X[cc]                                          # [m, 4, 2]
        J = np.einsum("mkr,qkc->mqrc", xc, dN)              # J[r, c] = d x_r / d ref_c
        det = J[..., 0, 0] * J[..., 1, 1] - J[..., 0, 1] * J[..., 1, 0]
        G = np.einsum("qkc,mqcr->mqkr", dN, np.linalg.inv(J))             # physical gradients of the Q1 basis
        xq = np.einsum("qk,mkd->mqd", N, xc).reshape(-1, 2)
        ue, ge = exact_solution(xq, mat)
        ue, ge = ue.reshape(len(cc), len(wq), 2), ge.reshape(len(cc), len(wq), 2)
        uq = np.einsum("qk,mkc->mqc", N, uh[cc])
        gh = np.einsum("mqkj,mkc->mqcj", G, uh[cc])         # d_j u_c
        w = wq[None, :] * np.abs(det)
        l2 += float((w[:, :, None] * (uq - ue) ** 2).sum())
        n_l2 += float((w[:, :, None] * ue ** 2).sum())
        h1 += float((w[:, :, None, None] * (gh - ge[:, :, None, :]) ** 2).sum())
        n_h1 += float((w[:, :, None, None] * np.repeat(ge[:, :, None, :], 2, axis=2) ** 2).sum())
    return (l2 / n_l2) ** 0.5, (h1 / n_h1) ** 0.5


def main(mesh_size=0.2, iterations=4, solver="direct", pen_coef=1.0, stab_coef=1.0, quiet=False,
         cell_type="triangle"):
    if cell_type not in ("triangle", "quadrilateral"):
        raise ValueError("cell_type must be 'triangle' or 'quadrilateral'")
    mat = elasticity.Material(E_in=1.0, nu_in=0.3, E_out=0.001, nu_out=0.3)            # data.py:13-22
    n = int(3.0 / mesh_size)                                                            # main.py:92-93
    results = {"dof": [], "L2 relative error": [], "H10 relative error": []}
    make_mesh = synthetic.quadrilateral_mesh if cell_type == "quadrilateral" else synthetic.rectangle_mesh
    error_norms = errors_quad if cell_type == "quadrilateral" else errors
    for _ in range(iterations):
        mesh = make_mesh(n, lo=(-1.5, -1.5), hi=(1.5, 1.5))
        V = fem.functionspace(mesh, ("Lagrange", 1))
        phi_h = fem.Function(V, levelset(mesh.x))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            cells_tags, facets_tags, _, d_bdry, _ = compute_tags_measures(mesh, phi_h, 1, box_mode=True)
        plan = elasticity.build_plan_interface_elasticity(mesh, cells_tags, facets_tags, d_bdry)
        X = mesh.x.cpu().numpy()
        bv = plan.boundary_vertices()
        u_dbc = exact_solution(X[bv.cpu().numpy()], mat)[0]
        bcs = (plan.dofs("u_in", bv).reshape(-1), torch.from_numpy(u_dbc.reshape(-1)))
        A, b = elasticity.assemble_interface_elasticity(plan, phi_h, source_term(X, mat), mat, pen_coef=pen_coef,
                                                        stab_coef=stab_coef, bcs=bcs)
        if solver == "bicgstab":
            sol, info = solve.bicgstab(A, b, rtol=1e-9, maxiter=20000)
            if not info.converged:
                raise RuntimeError("the linear solve did not converge (%r): use --solver direct" % info)
            sol = sol.cpu()
        else:
            import scipy.sparse.linalg as spla
            M = A.to_scipy().tocsr()
            keep = np.nonzero(np.asarray(abs(M).sum(axis=1)).ravel() > 0)[0]          # MUMPS ICNTL(24): null pivots
            s = np.zeros(M.shape[0])
            s[keep] = spla.spsolve(M[keep][:, keep].tocsc(), b.cpu().numpy()[keep])
            sol, info = torch.from_numpy(s), "direct (scipy LU on %d of %d rows)" % (len(keep), M.shape[0])
        u_in, u_out, *_ = plan.split(sol)
        tags = cells_tags.values_dev.cpu().numpy()
        l2, h1 = error_norms(mesh, tags, u_in.numpy(), u_out.numpy(), mat)
        results["dof"].append(2 * mesh.num_vertices)
        results["L2 relative error"].append(l2)
        results["H10 relative error"].append(h1)
        if not quiet:
            print("n %4d  cells %7d (in %d, cut %d, out %d)  mixed dofs %8d  nnz %10d  L2 %.3e  H10 %.3e  %s" % (
                n, mesh.num_cells, (tags == 1).sum(), (tags == 2).sum(), (tags == 3).sum(), plan.n_rows, plan.nnz,
                l2, h1, info))
        n *= 2
    return results


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh-size", type=float, default=0.2)
    ap.add_argument("--iterations", type=int, default=4)
    ap.add_argument("--solver", choices=("direct", "bicgstab"), default="direct")
    ap.add_argument("--cell-type", choices=("triangle", "quadrilateral"), default="triangle")
    a = ap.parse_args()
    main(a.mesh_size, a.iterations, a.solver, cell_type=a.cell_type)
