"""The step after the path on the GPU: CSR SpMV kernel and Jacobi-BiCGStab (phifem_b200/solve.py) against scipy,
and the two demos end to end."""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from phifem_b200 import assemble, fem, mesh_scripts, solve, synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _system(kind, n, form):
    if kind.startswith("tri"):
        mesh = synthetic.rectangle_mesh(n, device="cuda")
        center, radius = (0.013, -0.021), 0.62
    elif kind == "quad":
        mesh = synthetic.quadrilateral_mesh(n, device="cuda")
        center, radius = (0.013, -0.021), 0.62
    else:
        mesh = synthetic.unstructured_variant(synthetic.box_mesh(n, device="cuda"), jitter=0.15, seed=4)
        center, radius = synthetic.SPHERE_CENTER, 0.37
    V1 = fem.functionspace(mesh, 1)
    V = fem.functionspace(mesh, 2) if kind.endswith("p2") else V1
    phi1 = synthetic.sphere_levelset(mesh.x, center=center, radius=radius)
    phi = synthetic.sphere_levelset(V.dof_coordinates_dev(), center=center, radius=radius) if V is not V1 else phi1
    X = V.dof_coordinates_dev() if V is not V1 else mesh.x
    f = torch.cos(3.0 * X[:, 0]) + X[:, 1]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ct, ft, _, ds, _ = mesh_scripts.compute_tags_measures(mesh, fem.Function(V1, phi1), 1, box_mode=True)
    if form == "strong":
        plan = assemble.build_plan(mesh, ct, ft, ds(100), V=V, V_phi=V) if V is not V1 else \
            assemble.build_plan(mesh, ct, ft, ds(100))
        A, b = assemble.assemble_strong_dirichlet(plan, phi, f)
    else:
        plan = assemble.build_plan_weak_dirichlet(mesh, ct, ft, ds(100), V=V)
        A, b = assemble.assemble_weak_dirichlet(plan, phi, f)
    return A, b


def _lanes(A, keep):
    """Lanes per row of the fused iteration's product (csrc/solve.cu spmv_lanes: by nnz / active rows)."""
    avg = int(A.data.numel()) // len(keep)
    return 4 if avg <= 24 else (8 if avg <= 48 else (16 if avg <= 96 else 32))


# "form:option" runs solve.bicgstab with one of its options on the same system: x0 = the direct solution (converged
# with no iteration), maxiter not a multiple of check_every, int64 indptr / indices, b zero on every active row
@pytest.mark.parametrize("kind,n,form", [("tri", 64, "strong"), ("tet", 14, "strong"), ("tri", 48, "weak"),
                                         ("tet-p2", 7, "strong"), ("tri-p2", 32, "weak"), ("quad", 64, "strong"),
                                         ("tri", 64, "strong:x0"), ("tri", 64, "strong:maxiter"),
                                         ("tri", 64, "strong:int64"), ("tri", 64, "strong:zero-b")])
def test_spmv_and_bicgstab_match_scipy(kind, n, form):
    import scipy.sparse.linalg as spla
    form, _, option = form.partition(":")
    A, b = _system(kind, n, form)
    M = A.to_scipy().tocsr()
    x = torch.from_numpy(np.random.default_rng(3).uniform(-1, 1, M.shape[0])).cuda()
    y = solve.spmv(A, x).cpu().numpy()
    want = M @ x.cpu().numpy()
    assert np.abs(y - want).max() <= 1e-13 * np.abs(want).max()
    d = M.diagonal()
    rowmax = np.asarray(abs(M).max(axis=1).todense()).ravel()
    active = np.abs(d) > 1e-14 * rowmax                      # solve.bicgstab's null-pivot test (default pivot_tol)
    keep = np.nonzero(active)[0]
    print("%s-%d-%s: %d of %d rows active, %d lanes per row" % (kind, n, form, len(keep), M.shape[0], _lanes(A, keep)))
    ref = np.zeros(M.shape[0])
    ref[keep] = spla.spsolve(M[keep][:, keep].tocsc(), b.cpu().numpy()[keep])
    if option == "x0":
        x0 = torch.from_numpy(ref).cuda()
        sol, info = solve.bicgstab(A, b, x0=x0)
        assert info.converged and info.iterations == 0 and info.n_active == len(keep), info
        assert torch.equal(sol, x0)
        return
    if option == "maxiter":
        sol, info = solve.bicgstab(A, b, rtol=1e-14, maxiter=13, check_every=5)
        assert info.iterations == 13 and not info.converged, info
        sol1, info1 = solve.bicgstab(A, b, rtol=1e-14, maxiter=13, check_every=1)
        assert info1.iterations == 13 and torch.equal(sol, sol1)
        r = b.cpu().numpy()[keep] - M[keep] @ sol.cpu().numpy()
        assert abs(np.linalg.norm(r) / np.linalg.norm(b.cpu().numpy()[keep]) - info.residual) <= 1e-8 * info.residual
        return
    if option == "zero-b":
        assert not active.all()
        bz = torch.from_numpy(np.where(active, 0.0, 1.0)).cuda()   # zero on the active rows only
        sol, info = solve.bicgstab(A, bz)
        assert info.converged and info.iterations == 0 and info.n_active == len(keep), info
        assert float(sol.abs().max()) == 0.0
        return
    if option == "int64":
        A = assemble.CSRMatrix(A.indptr.long(), A.indices.long(), A.data, A.shape)
    sol, info = solve.bicgstab(A, b, rtol=1e-11)
    assert info.converged and info.residual < 1e-9, info
    assert info.n_active == len(keep)
    got = sol.cpu().numpy()
    assert np.all(got[~active] == 0.0)                      # null pivots: unknown set to zero
    assert np.linalg.norm(got - ref) <= 1e-7 * np.linalg.norm(ref)


def test_demos_run_end_to_end():
    sys.path.insert(0, os.path.join(ROOT, "demo"))
    import strong_dirichlet_flower
    import weak_dirichlet_flower
    u1, info1 = strong_dirichlet_flower.main(n=100, degree=1, quiet=True)
    u2, info2 = weak_dirichlet_flower.main(n=100, quiet=True)
    assert info1.converged and info2.converged
    # the two formulations discretise the same Poisson problem on the flower: both solutions are positive in the
    # petal holding the source and agree to discretisation accuracy
    assert float(u1.max()) > 0.05 and float(u2.max()) > 0.05
    assert abs(float(u1.max()) - float(u2.max())) < 0.25 * float(u1.max())
    u3, info3 = strong_dirichlet_flower.main(n=60, degree=2, quiet=True)
    assert info3.converged and abs(float(u3.max()) - float(u1.max())) < 0.25 * float(u1.max())
