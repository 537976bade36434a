"""GPU parity of the strong-Dirichlet phi-FEM operator on quadrilaterals (csrc/assemble_quad.cu behind the
phifem_assemble_*_pk entry points) against the oracle of oracle/assembly_quad_strong.py at the kernels' rules, and its
meaning: the solved system converges to a manufactured solution u = phi w of -lap u = f, u = 0 on {phi = 0}."""
import ctypes
import warnings

import numpy as np
import pytest
import torch

from oracle import assembly_quad as OQ
from oracle import assembly_quad_strong as OS
from phifem_b200 import _lib, assemble, fem, mesh_scripts, quadrature, solve, synthetic

pytestmark = pytest.mark.gpu
RTOL = 1e-12


def _row_scale(indptr, data):
    scale = np.zeros(len(indptr) - 1)
    rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
    np.maximum.at(scale, rows, np.abs(data))
    return scale, rows


def _mesh(kind):
    if kind == "quad":
        return synthetic.quadrilateral_mesh(14, device="cuda")
    return synthetic.unstructured_variant(synthetic.quadrilateral_mesh(10, device="cuda"), jitter=0.2, seed=7)


def _tags(mesh, phi_vertices):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return mesh_scripts.compute_tags_measures(mesh, fem.Function(fem.functionspace(mesh, 1), phi_vertices), 1,
                                                  box_mode=True)


def _oracle(mesh, plan, phi, f, ctags, ftags, ds, kphi, sigma):
    (cl, cw), (fl, fw) = quadrature.rules_for_strong_quad(kphi)
    return OS.assemble_strong_dirichlet_quad(
        mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64), phi.cpu().numpy(), f.cpu().numpy(),
        ctags.values_dev.cpu().numpy(), ftags.values_dev.cpu().numpy(), mesh.c2f.cpu().numpy(), mesh.f2c.cpu().numpy(),
        ds(100).integration_entities, sigma=sigma, kphi=kphi, phi_dofmap=plan.V_phi.dofmap, rule=(cl, cw),
        facet_rule=(fl[:, 1], fw))


def _check(A, b, ref):
    ip, ix, data, bo = ref
    assert np.array_equal(A.indptr.cpu().numpy(), ip) and np.array_equal(A.indices.cpu().numpy(), ix)
    scale, rows = _row_scale(ip, data)
    gs = np.abs(data).max()
    assert np.all(np.abs(A.data.cpu().numpy() - data) <= RTOL * np.maximum(scale[rows], 1e-300 * gs))
    assert np.all(np.abs(b.cpu().numpy() - bo) <= RTOL * np.abs(bo).max())


@pytest.mark.parametrize("kphi", [1, 2])
@pytest.mark.parametrize("kind", ["quad", "quad-unstructured"])
def test_strong_quad_operator_matches_oracle(kind, kphi):
    mesh = _mesh(kind)
    center, radius = (0.013, -0.021), 0.61
    ctags, ftags, _, ds, _ = _tags(mesh, synthetic.sphere_levelset(mesh.x, center=center, radius=radius))
    Vp = fem.functionspace(mesh, kphi)
    phi = synthetic.sphere_levelset(Vp.dof_coordinates_dev(), center=center, radius=radius)
    rng = np.random.default_rng(41)
    f = torch.from_numpy(rng.uniform(-1, 1, mesh.num_vertices)).cuda()
    plan = assemble.build_plan(mesh, ctags, ftags, ds(100), V=fem.functionspace(mesh, 1), V_phi=Vp)
    assert plan.ghost.numel() > 0 and plan.entities.shape[0] > 0 and bool((plan.cell_tags8 == 2).any())
    A, b = assemble.assemble_strong_dirichlet(plan, phi, f, stab_coef=0.7)
    assert A.shape == (mesh.num_vertices, mesh.num_vertices)
    _check(A, b, _oracle(mesh, plan, phi, f, ctags, ftags, ds, kphi, 0.7))


def test_strong_quad_default_route():
    """build_plan without V / V_phi on a quadrilateral mesh: the same operator as an explicit Q1 / Q1 plan."""
    mesh = _mesh("quad-unstructured")
    phi = synthetic.sphere_levelset(mesh.x, center=(0.013, -0.021), radius=0.61)
    ctags, ftags, _, ds, _ = _tags(mesh, phi)
    f = synthetic.ball_source(mesh.x)
    V = fem.functionspace(mesh, 1)
    A0, b0 = assemble.assemble_strong_dirichlet(assemble.build_plan(mesh, ctags, ftags, ds(100)), phi, f)
    A1, b1 = assemble.assemble_strong_dirichlet(assemble.build_plan(mesh, ctags, ftags, ds(100), V=V, V_phi=V), phi, f)
    assert torch.equal(A0.indptr, A1.indptr) and torch.equal(A0.indices, A1.indices)
    scale, rows = _row_scale(A1.indptr.cpu().numpy(), A1.data.cpu().numpy())
    assert np.all(np.abs(A0.data.cpu().numpy() - A1.data.cpu().numpy()) <= RTOL * scale[rows])
    assert np.abs((b0 - b1).cpu().numpy()).max() <= RTOL * np.abs(b1.cpu().numpy()).max()


def test_strong_quad_without_cut_cells():
    """The level set contains the mesh: empty cut and ghost lists; the one-sided term runs on the 4 n mesh-boundary
    facets (they become Gamma_h)."""
    n = 7
    mesh = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(n, device="cuda"), jitter=0.2, seed=3)
    phi = synthetic.sphere_levelset(mesh.x, center=(0.0, 0.0), radius=9.0)
    ctags, ftags, _, ds, _ = _tags(mesh, phi)
    assert bool((ctags.values_dev == 1).all())
    f = torch.from_numpy(np.random.default_rng(2).uniform(-1, 1, mesh.num_vertices)).cuda()
    plan = assemble.build_plan(mesh, ctags, ftags, ds(100))
    assert plan.ghost.numel() == 0 and plan.entities.shape[0] == 4 * n
    A, b = assemble.assemble_strong_dirichlet(plan, phi, f)
    _check(A, b, _oracle(mesh, plan, phi, f, ctags, ftags, ds, 1, 1.0))


R_DISC, C_DISC = 0.62, (0.013, -0.021)


def _exact(X):
    """u = phi * w with phi = |x - c|^2 - R^2, w = -exp(x0) cos(x1) (tests/test_gpu_convergence.py): f = -lap u."""
    x0, x1 = X[:, 0] - C_DISC[0], X[:, 1] - C_DISC[1]
    phi = x0 * x0 + x1 * x1 - R_DISC * R_DISC
    w = -torch.exp(x0) * torch.cos(x1)
    gw0, gw1 = w, torch.exp(x0) * torch.sin(x1)
    lap = 4.0 * w + 2.0 * (2.0 * x0 * gw0 + 2.0 * x1 * gw1)
    return phi * w, -lap


def _manufactured_system(n, kphi):
    mesh = synthetic.quadrilateral_mesh(n, device="cuda")
    ctags, ftags, _, ds, _ = _tags(mesh, synthetic.sphere_levelset(mesh.x, center=C_DISC, radius=R_DISC))
    Vp = fem.functionspace(mesh, kphi)
    phi = synthetic.sphere_levelset(Vp.dof_coordinates_dev(), center=C_DISC, radius=R_DISC)
    _, f = _exact(mesh.x)
    plan = assemble.build_plan(mesh, ctags, ftags, ds(100), V_phi=Vp)
    A, b = assemble.assemble_strong_dirichlet(plan, phi, f, stab_coef=1.0)
    return mesh, ctags, plan, phi, A, b


def _spsolve(A, b):
    import scipy.sparse.linalg as spla
    M = A.to_scipy().tocsr()
    keep = np.nonzero(np.diff(M.indptr) > 0)[0]
    sol = np.zeros(M.shape[0])
    sol[keep] = spla.spsolve(M[keep][:, keep].tocsc(), b.cpu().numpy()[keep])
    return sol, keep


def _strong_quad_error(n, kphi):
    mesh, ctags, plan, phi, A, b = _manufactured_system(n, kphi)
    w, _ = _spsolve(A, b)
    pts, wq = OQ.gauss_square(4)
    N, dN = OQ.tabulate(OQ._Q1, pts)
    pv, _ = OQ.tabulate(fem.LagrangeElement("quadrilateral", kphi), pts)
    inter = torch.nonzero(ctags.values_dev == 1).reshape(-1)
    cells = mesh.cells[inter].long().cpu().numpy()
    pdm = plan.V_phi.dofmap_dev[inter].long().cpu().numpy()
    xc = mesh.x.cpu().numpy()[cells]                                  # [m, 4, 2]
    xq = np.einsum("qk,mkd->mqd", N, xc)
    J = np.einsum("mkr,qkc->mqrc", xc, dN)
    det = np.abs(J[..., 0, 0] * J[..., 1, 1] - J[..., 0, 1] * J[..., 1, 0])
    ue = _exact(torch.from_numpy(xq.reshape(-1, 2)))[0].numpy().reshape(xq.shape[:2])
    uh = np.einsum("qk,mk->mq", pv, phi.cpu().numpy()[pdm]) * np.einsum("qk,mk->mq", N, w[cells])
    err2 = float((wq[None] * det * (uh - ue) ** 2).sum())
    nrm2 = float((wq[None] * det * ue ** 2).sum())
    return (err2 / nrm2) ** 0.5


@pytest.mark.parametrize("kphi,last_err", [(1, 1.2e-3), (2, 5e-5)])
def test_strong_quad_manufactured_solution_converges(kphi, last_err):
    """Second order in L2, as P1 on triangles.  The oracle's system solved with scipy gives, at n = 24, 48, 96:
    Q1 level set 2.87e-2, 4.53e-3, 8.51e-4 (rates 2.67, 2.41: the interpolation error of the quadratic level set
    still dominates and decays faster); Q2 level set 5.09e-4, 1.34e-4, 3.18e-5 (rates 1.92, 2.08)."""
    errs = [_strong_quad_error(n, kphi) for n in (24, 48, 96)]
    rates = [np.log2(errs[i] / errs[i + 1]) for i in range(2)]
    print("strong quad errors", kphi, errs, rates)
    assert errs[-1] < last_err and min(rates) > 1.8, (errs, rates)


def test_strong_quad_bicgstab_matches_spsolve():
    _, _, plan, _, A, b = _manufactured_system(32, 2)
    x, info = solve.bicgstab(A, b, rtol=1e-12, maxiter=20000)
    assert info.converged, info
    ref, keep = _spsolve(A, b)
    assert len(keep) > 0
    u = x.cpu().numpy()
    assert np.abs(u[keep] - ref[keep]).max() <= 1e-8 * np.abs(ref[keep]).max()


def _call_cells(plan, mesh, sw, sp):
    lib = _lib.load()
    _, _, cq = plan.c_structs()
    data, b = plan.new_outputs()
    t = torch.zeros(mesh.num_vertices, dtype=torch.float64, device="cuda")
    rc = lib.phifem_assemble_cells_pk(
        _lib.c_mesh(mesh), ctypes.byref(sw), ctypes.byref(sp), ctypes.byref(cq), _lib.ptr(t), _lib.ptr(t),
        _lib.ptr(plan.cell_tags8), _lib.ptr(plan.active), plan.active.numel(), _lib.ptr(plan.slots_cells), 1.0,
        _lib.ptr(data), _lib.ptr(b), _lib.stream())
    return rc, lib.phifem_last_error().decode()


def test_strong_quad_errors():
    mesh = synthetic.quadrilateral_mesh(6, device="cuda")
    phi = synthetic.sphere_levelset(mesh.x, center=(0.01, 0.02), radius=0.6)
    ctags, ftags, _, ds, _ = _tags(mesh, phi)
    plan = assemble.build_plan(mesh, ctags, ftags, ds(100))
    cw, cp, _ = plan.c_structs()
    # the C ABI: a level-set space of 6 dofs per cell is an argument error, a Q2 trial space is unsupported
    rc, msg = _call_cells(plan, mesh, cw, _lib.CPkSpace(2, 6, cp.n_dofs, cp.dofmap))
    assert rc == -1 and "quadrilateral" in msg, msg                  # PHIFEM_ERR_ARGUMENT
    V2 = fem.functionspace(mesh, 2)
    rc, msg = _call_cells(plan, mesh, _lib.CPkSpace(2, 9, V2.num_dofs, _lib.ptr(V2.dofmap_dev)), cp)
    assert rc == -3 and "quadrilateral" in msg, msg                  # PHIFEM_ERR_UNSUPPORTED
    # the row-gather options have no quadrilateral implementation
    for kw in (dict(method="blocked"), dict(method="atomic"), dict(geometry=True), dict(cell_pass="tiles"),
               dict(symbolic="native")):
        with pytest.raises(ValueError):
            assemble.build_plan(mesh, ctags, ftags, ds(100), **kw)
