"""GPU parity of the interface-elasticity phi-FEM operator on quadrilaterals (csrc/assemble_elasticity.cu behind the
phifem_assemble_elasticity_* entry points) against the oracle of oracle/elasticity_quad.py at the kernels' rules, with
and without Dirichlet conditions, and its meaning: the solved system converges to the demo's manufactured two-material
solution (reference demo/interface-elasticity/data.py:43-48)."""
import ctypes
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from oracle import elasticity as OE
from oracle import elasticity_quad as OEQ
from phifem_b200 import _lib, elasticity, fem, mesh_scripts, quadrature, synthetic

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "demo"))
import interface_elasticity as demo  # noqa: E402

pytestmark = pytest.mark.gpu
RTOL = 1e-12


def _row_scale(indptr, data):
    scale = np.zeros(len(indptr) - 1)
    rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
    np.maximum.at(scale, rows, np.abs(data))
    return scale, rows


def _tags(mesh, phi_vertices):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return mesh_scripts.compute_tags_measures(mesh, fem.Function(fem.functionspace(mesh, 1), phi_vertices), 1,
                                                  box_mode=True)


def _oracle(mesh, Vp, phi, f, ctags, ftags, d_bdry, kphi, mat, bc_dofs=None, bc_vals=None):
    (cp, cw), (up, uw), (fp, fw) = quadrature.rules_for_elasticity_quad(kphi)
    return OEQ.assemble_interface_elasticity_quad(
        mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64), phi.cpu().numpy(), f.cpu().numpy(),
        ctags.values_dev.cpu().numpy(), ftags.values_dev.cpu().numpy(), mesh.c2f.cpu().numpy(), mesh.f2c.cpu().numpy(),
        d_bdry(100).integration_entities, d_bdry(101).integration_entities, mat=mat, gamma=1.3, sigma_s=0.7,
        kphi=kphi, phi_dofmap=Vp.dofmap.astype(np.int64), bc_dofs=bc_dofs, bc_values=bc_vals, rule=(cp, cw),
        uncut_rule=(up, uw), facet_rule=(fp[:, 1], fw))


def _check(A, b, ref):
    ip, ix, data, bo = ref
    assert np.array_equal(A.indptr.cpu().numpy(), ip) and np.array_equal(A.indices.cpu().numpy(), ix)
    scale, rows = _row_scale(ip, data)
    gs = np.abs(data).max()
    assert np.all(np.abs(A.data.cpu().numpy() - data) <= RTOL * np.maximum(scale[rows], 1e-300 * gs))
    assert np.all(np.abs(b.cpu().numpy() - bo) <= RTOL * np.abs(bo).max())


@pytest.mark.parametrize("with_bc", [False, True])
@pytest.mark.parametrize("kphi", [1, 2])
@pytest.mark.parametrize("kind", ["quad", "quad-unstructured"])
def test_elasticity_quad_operator_matches_oracle(kind, kphi, with_bc):
    if kind == "quad":
        mesh = synthetic.quadrilateral_mesh(14, device="cuda")
    else:
        mesh = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(10, device="cuda"), jitter=0.2, seed=7)
    center, radius = (0.013, -0.021), 0.61
    ctags, ftags, _, d_bdry, _ = _tags(mesh, synthetic.sphere_levelset(mesh.x, center=center, radius=radius))
    Vp = fem.functionspace(mesh, kphi)
    phi = synthetic.sphere_levelset(Vp.dof_coordinates_dev(), center=center, radius=radius)
    rng = np.random.default_rng(77)
    f = torch.from_numpy(rng.uniform(-1, 1, (mesh.num_vertices, 2))).cuda()
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=Vp)
    assert plan.cut_cells.numel() > 0 and plan.facets_in.numel() > 0 and plan.facets_out.numel() > 0
    assert plan.entities_in.shape[0] > 0 and plan.entities_out.shape[0] > 0
    mat = elasticity.Material(1.0, 0.3, 0.05, 0.27)
    bcs = bc_dofs = bc_vals = None
    if with_bc:
        bc_dofs = plan.dofs("u_in", plan.boundary_vertices()).reshape(-1)
        bc_vals = torch.from_numpy(rng.uniform(-1, 1, bc_dofs.numel())).cuda()
        bcs = (bc_dofs, bc_vals)
        bc_dofs, bc_vals = bc_dofs.cpu().numpy(), bc_vals.cpu().numpy()
    A, b = elasticity.assemble_interface_elasticity(plan, phi, f, mat, pen_coef=1.3, stab_coef=0.7, bcs=bcs)
    if with_bc:   # the full-matrix Dirichlet pass gives the same system
        A2, b2 = elasticity.assemble_interface_elasticity(plan, phi, f, mat, pen_coef=1.3, stab_coef=0.7, bcs=bcs,
                                                          symmetric_bc=False)
        assert torch.allclose(A2.data, A.data, rtol=0, atol=1e-13 * float(A.data.abs().max()))
        assert torch.allclose(b2, b, rtol=0, atol=1e-12 * float(b.abs().max()))
    assert A.shape[0] == 14 * mesh.num_vertices
    _check(A, b, _oracle(mesh, Vp, phi, f, ctags, ftags, d_bdry, kphi, OE.Material(1.0, 0.3, 0.05, 0.27), bc_dofs,
                         bc_vals))


@pytest.mark.parametrize("where", ["outside", "inside"])
def test_elasticity_quad_without_cut_cells(where):
    """The interface misses the mesh: no cut cell, no interface facet; in box mode the mesh boundary becomes the
    one-sided boundary of the material inside.  Only the rows of that material's displacement are filled."""
    n = 7
    mesh = synthetic.unstructured_variant(synthetic.quadrilateral_mesh(n, device="cuda"), jitter=0.2, seed=3)
    r = 0.5 if where == "outside" else 9.0
    c = (5.0, 5.0) if where == "outside" else (0.0, 0.0)
    phi = synthetic.sphere_levelset(mesh.x, center=c, radius=r)
    ctags, ftags, _, d_bdry, _ = _tags(mesh, phi)
    tag = 3 if where == "outside" else 1
    assert bool((ctags.values_dev == tag).all())
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry)
    assert plan.cut_cells.numel() == 0 and plan.facets_in.numel() == 0 and plan.facets_out.numel() == 0
    assert plan.entities_out.shape[0] == 0 and plan.entities_in.shape[0] == (4 * n if where == "inside" else 0)
    f = torch.from_numpy(np.random.default_rng(5).uniform(-1, 1, (mesh.num_vertices, 2))).cuda()
    mat = elasticity.Material(1.0, 0.3, 0.05, 0.27)
    A, b = elasticity.assemble_interface_elasticity(plan, phi, f, mat, pen_coef=1.3, stab_coef=0.7)
    ref = _oracle(mesh, plan.V_phi, phi, f, ctags, ftags, d_bdry, 1, OE.Material(1.0, 0.3, 0.05, 0.27))
    _check(A, b, ref)
    ip, data = ref[0], ref[2]
    blk = np.repeat(np.arange(len(ip) - 1), np.diff(ip)) % plan.nb
    off = plan.layout["u_out" if where == "outside" else "u_in"][0]
    assert np.all(data[(blk < off) | (blk >= off + 2)] == 0.0) and np.abs(data).max() > 0


def _solve(A, b):
    import scipy.sparse.linalg as spla
    M = A.to_scipy().tocsr()
    keep = np.nonzero(np.asarray(abs(M).sum(axis=1)).ravel() > 0)[0]
    sol = np.zeros(M.shape[0])
    sol[keep] = spla.spsolve(M[keep][:, keep].tocsc(), b.cpu().numpy()[keep])
    return sol


def _interface_error(n, E_out):
    mat = elasticity.Material(1.0, 0.3, E_out, 0.3)
    mesh = synthetic.quadrilateral_mesh(n, lo=(-1.5, -1.5), hi=(1.5, 1.5), device="cuda")   # param1.yaml bbox
    X = mesh.x.cpu().numpy()
    phi = demo.levelset(mesh.x)
    ctags, ftags, _, d_bdry, _ = _tags(mesh, phi)
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry)
    bv = plan.boundary_vertices()
    bcs = (plan.dofs("u_in", bv).reshape(-1),
           torch.from_numpy(demo.exact_solution(X[bv.cpu().numpy()], mat)[0].reshape(-1)).cuda())
    A, b = elasticity.assemble_interface_elasticity(plan, phi, demo.source_term(X, mat), mat, bcs=bcs)
    u_in, u_out, *_ = plan.split(torch.from_numpy(_solve(A, b)))
    return demo.errors_quad(mesh, ctags.values_dev.cpu().numpy(), u_in.numpy(), u_out.numpy(), mat)[0]


# relative L2 errors of the oracle's system (oracle/elasticity_quad.py, CPU tags of oracle/tags.py) solved with scipy's
# spsolve, at n = 15, 31, 63
ORACLE_L2 = {0.1: (0.024089416356740986, 0.0057514548727481945, 0.0012788299148053612),
             0.001: (0.03325649768310988, 0.007808768187182887, 0.0019586578358263456)}


@pytest.mark.parametrize("E_out", [0.1, 0.001])
def test_interface_elasticity_quad_manufactured_solution_converges(E_out):
    """The demo's test case (bbox [-1.5, 1.5]^2, unit-disc interface) on quadrilaterals, E_out = 0.1 and the demo's
    0.001: the GPU-assembled system reproduces the oracle's errors (rates 2.07, 2.17 and 2.09, 2.00)."""
    errs = [_interface_error(n, E_out) for n in (15, 31, 63)]
    rates = [np.log2(errs[i] / errs[i + 1]) for i in range(2)]
    print("interface-elasticity quad errors", E_out, errs, rates)
    assert np.allclose(errs, ORACLE_L2[E_out], rtol=1e-6, atol=0), (errs, ORACLE_L2[E_out])
    assert errs[-1] < 2.5e-3 and min(rates) > 1.9, (errs, rates)


def test_interface_elasticity_quad_demo_runs_end_to_end():
    res = demo.main(mesh_size=0.2, iterations=3, quiet=True, cell_type="quadrilateral")
    l2, h1 = res["L2 relative error"], res["H10 relative error"]
    assert res["dof"] == [2 * 16 * 16, 2 * 31 * 31, 2 * 61 * 61]
    assert l2[-1] < 3e-3 and l2[0] / l2[-1] > 10.0, l2
    assert h1[-1] < 4e-2 and h1[0] / h1[-1] > 3.0, h1


def _call_cells(plan, mesh, space):
    lib = _lib.load()
    _, cq = plan.c_structs()
    data, b = plan.new_outputs()
    phi = torch.zeros(max(space.n_dofs, mesh.num_vertices), dtype=torch.float64, device="cuda")
    f = torch.zeros(mesh.num_vertices, 2, dtype=torch.float64, device="cuda")
    prm = _lib.CElasticityParams(1.0, 1.0, 1.0, 1.0, 0.5, 0.5, 1.0, 1.0)
    rc = lib.phifem_assemble_elasticity_cells(
        _lib.c_mesh(mesh), ctypes.byref(space), ctypes.byref(cq), _lib.ptr(phi), _lib.ptr(f), _lib.ptr(plan.cell_tags8),
        _lib.ptr(plan.cut_cells), plan.cut_cells.numel(), _lib.ptr(plan.vptr), _lib.ptr(plan.pos_cells),
        ctypes.byref(prm), _lib.ptr(data), _lib.ptr(b), _lib.stream())
    return rc, lib.phifem_last_error().decode()


def test_elasticity_quad_c_abi_errors():
    mesh = synthetic.quadrilateral_mesh(6, device="cuda")
    ctags, ftags, _, d_bdry, _ = _tags(mesh, synthetic.sphere_levelset(mesh.x, center=(0.01, 0.02), radius=0.6))
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry)
    cp, _ = plan.c_structs()
    # a level-set space of 6 dofs per cell is an argument error
    rc, msg = _call_cells(plan, mesh, _lib.CPkSpace(2, 6, cp.n_dofs, cp.dofmap))
    assert rc == -1 and "n_dofs_per_cell" in msg and "quadrilateral" in msg, msg     # PHIFEM_ERR_ARGUMENT
    # a Q3 level set is not implemented
    rc, _ = _call_cells(plan, mesh, _lib.CPkSpace(3, 16, cp.n_dofs, cp.dofmap))
    assert rc == -3                                                                      # PHIFEM_ERR_UNSUPPORTED
    # the Q1 level set of the plan passes the same checks
    rc, msg = _call_cells(plan, mesh, cp)
    assert rc == 0, msg
