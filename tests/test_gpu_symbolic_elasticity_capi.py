"""The symbolic phase of the interface-elasticity operator behind the C ABI (csrc/symbolic.cu,
phifem_elasticity_pattern_create) produces bit for bit the arrays of the torch-based ElasticityPlan
(phifem_b200/elasticity.py) -- vertex graph, blocked CSR, cut cells, interface facets, the five position maps -- on
triangles, quadrilaterals and tetrahedra; the operator assembled through those arrays equals the plan's; a host program
without Python (examples/capi_host_elasticity.cu) reproduces the checksums of the Python path."""
import copy
import os
import subprocess
import types
import warnings

import numpy as np
import pytest
import torch

from phifem_b200 import elasticity, fem, mesh_scripts, symbolic, synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("vptr", "indptr", "indices", "cut_cells", "facets_in", "facets_out", "entities_in", "entities_out",
         "pos_cells", "pos_facets_in", "pos_facets_out", "pos_entities_in", "pos_entities_out")


def _mesh(kind, n):
    if kind.startswith("tri"):
        mesh, center, radius = synthetic.rectangle_mesh(n, device="cuda"), (0.013, -0.021), 0.61
    elif kind.startswith("quad"):
        mesh, center, radius = synthetic.quadrilateral_mesh(n, device="cuda"), (0.013, -0.021), 0.61
    else:
        mesh, center, radius = synthetic.box_mesh(n, device="cuda"), synthetic.SPHERE_CENTER, 0.37
    if kind.endswith("unstructured"):
        mesh = synthetic.unstructured_variant(mesh, jitter=0.2, seed=7)
    return mesh, center, radius


def _problem(mesh, center, radius, kphi):
    """Tags and measures of the level set interpolated into the degree-kphi space (detection degree kphi)."""
    Vp = fem.functionspace(mesh, kphi)
    phi = synthetic.sphere_levelset(Vp.dof_coordinates_dev(), center=center, radius=radius)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, d_bdry, _ = mesh_scripts.compute_tags_measures(mesh, fem.Function(Vp, phi), kphi,
                                                                        box_mode=True)
    return ctags, ftags, d_bdry, Vp, phi


def _assert_same_arrays(pat, plan):
    assert pat.nnz == plan.nnz and pat.n_rows == plan.n_rows and pat.nb == plan.nb
    for name in NAMES:
        a, b = getattr(pat, name), getattr(plan, name)
        assert a.dtype == b.dtype == torch.int32 and a.shape == b.shape, name
        assert torch.equal(a, b), name


def _assemble(plan, phi, with_bc):
    rng = np.random.default_rng(77)
    mesh = plan.mesh
    f = torch.from_numpy(rng.uniform(-1, 1, (mesh.num_vertices, mesh.gdim))).cuda()
    bcs = None
    if with_bc:
        dofs = torch.cat([plan.dofs("u_in", plan.boundary_vertices()).reshape(-1),
                          plan.dofs("u_out", plan.boundary_vertices()).reshape(-1)])
        bcs = (dofs, torch.from_numpy(rng.uniform(-1, 1, dofs.numel())).cuda())
    A, b = elasticity.assemble_interface_elasticity(plan, phi, f, elasticity.Material(1.0, 0.3, 0.05, 0.27),
                                                    pen_coef=1.3, stab_coef=0.7, bcs=bcs)
    torch.cuda.synchronize()
    return A.data, b


def _assert_same_operator(plan, pat, phi, with_bc):
    """The plan with the native arrays assembles the plan's own operator (fp64 atomics reorder the sums)."""
    native = copy.copy(plan)
    for name in NAMES:
        setattr(native, name, getattr(pat, name))
    d0, b0 = _assemble(plan, phi, with_bc)
    d1, b1 = _assemble(native, phi, with_bc)
    rows = torch.repeat_interleave(torch.arange(plan.n_rows, device="cuda"),
                                   (plan.indptr[1:] - plan.indptr[:-1]).long())
    scale = torch.zeros(plan.n_rows, dtype=torch.float64, device="cuda").scatter_reduce(0, rows, d0.abs(), "amax")
    assert bool(((d1 - d0).abs() <= 1e-14 * scale[rows]).all())
    assert float((b1 - b0).abs().max()) <= 1e-14 * float(b0.abs().max())
    assert float(d0.abs().sum()) > 0 and float(b0.abs().sum()) > 0


CASES = [(kind, n, kphi) for kind, n in (("tri", 12), ("tri-unstructured", 9), ("quad", 12), ("quad-unstructured", 9),
                                         ("tet", 4), ("tet-unstructured", 4))
         for kphi in (1, 2)]


@pytest.mark.parametrize("kind,n,kphi", CASES)
def test_device_elasticity_pattern_equals_the_torch_plan(kind, n, kphi):
    mesh, center, radius = _mesh(kind, n)
    ctags, ftags, d_bdry, Vp, phi = _problem(mesh, center, radius, kphi)
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=Vp)
    assert plan.cut_cells.numel() and plan.facets_in.numel() and plan.facets_out.numel()
    assert plan.entities_in.shape[0] and plan.entities_out.shape[0]
    pat = symbolic.DeviceElasticityPattern(mesh, ctags, ftags, d_bdry)
    _assert_same_arrays(pat, plan)
    for with_bc in (False, True):
        _assert_same_operator(plan, pat, phi, with_bc)


def test_untagged_cells_have_zero_positions():
    """pos_cells covers every cell; the rows of cells not tagged 1..3 are 0, as the plan's."""
    mesh, center, radius = _mesh("tri", 10)
    ctags, ftags, d_bdry, Vp, _ = _problem(mesh, center, radius, 1)
    c8 = ctags.tags8.clone()
    c8[::5] = torch.where(c8[::5] == 3, torch.zeros_like(c8[::5]), c8[::5])   # some exterior cells left untagged
    untagged = types.SimpleNamespace(tags8=c8)
    ds101 = d_bdry(101).integration_entities_dev.reshape(-1, 2)
    ds101 = ds101[c8[ds101[:, 0].long()] != 0].reshape(-1)
    pair = (d_bdry(100), ds101)
    plan = elasticity.build_plan_interface_elasticity(mesh, untagged, ftags, pair, V_phi=Vp)
    pat = symbolic.DeviceElasticityPattern(mesh, untagged, ftags, pair)
    assert bool((c8 == 0).any())
    assert not bool(pat.pos_cells[c8 == 0].any())
    _assert_same_arrays(pat, plan)


@pytest.mark.parametrize("kind,where", [("tri", "inside"), ("tri", "outside"), ("quad-unstructured", "inside"),
                                        ("tet", "inside"), ("tet", "outside")])
def test_without_cut_cells(kind, where):
    """A level set negative (positive) everywhere: every cell tagged 1 (3), no cut cell, no facet tagged 4."""
    mesh, center, _ = _mesh(kind, 6 if kind.startswith("tet") else 8)
    radius = 100.0 if where == "inside" else 1e-3
    center = center if where == "inside" else tuple(50.0 for _ in center)
    ctags, ftags, d_bdry, Vp, phi = _problem(mesh, center, radius, 1)
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=Vp)
    pat = symbolic.DeviceElasticityPattern(mesh, ctags, ftags, d_bdry)
    assert pat.cut_cells.numel() == 0 and pat.facets_out.numel() == 0
    assert pat.nnz == plan.nnz > 0
    _assert_same_arrays(pat, plan)
    _assert_same_operator(plan, pat, phi, True)


def test_without_entities():
    """Empty ds(100) and ds(101)."""
    mesh, center, radius = _mesh("tri-unstructured", 10)
    ctags, ftags, _, Vp, phi = _problem(mesh, center, radius, 2)
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, (None, None), V_phi=Vp)
    pat = symbolic.DeviceElasticityPattern(mesh, ctags, ftags, (None, None))
    assert pat.pos_entities_in.shape == (0, 9) and pat.pos_entities_out.shape == (0, 9)
    assert pat.cut_cells.numel() > 0 and pat.facets_in.numel() > 0
    _assert_same_arrays(pat, plan)
    _assert_same_operator(plan, pat, phi, False)


def test_more_than_2_to_the_30_entries():
    """rectangle_mesh(900): over 2^30 blocked entries, so the expansion's addresses leave the 32-bit range of signed
    products of 32-bit operands."""
    mesh, center, radius = _mesh("tri", 900)
    ctags, ftags, d_bdry, Vp, _ = _problem(mesh, center, radius, 1)
    pat = symbolic.DeviceElasticityPattern(mesh, ctags, ftags, d_bdry)
    assert pat.nnz > 2 ** 30
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=Vp)
    _assert_same_arrays(pat, plan)
    assert int(pat.indptr[-1]) == pat.nnz


def test_device_refusals():
    mesh, center, radius = _mesh("tri", 10)
    ctags, ftags, d_bdry, Vp, _ = _problem(mesh, center, radius, 1)
    ds100 = d_bdry(100).integration_entities_dev.reshape(-1, 2)
    ds101 = d_bdry(101).integration_entities_dev.reshape(-1, 2)
    # an entity whose cell is re-tagged 0
    c8 = ctags.tags8.clone()
    c8[ds100[0, 0].long()] = 0
    with pytest.raises(ValueError, match="entity's cell is not tagged 1, 2 or 3"):
        symbolic.DeviceElasticityPattern(mesh, types.SimpleNamespace(tags8=c8), ftags, d_bdry)
    # a local facet out of range (3 on triangles), a cell id outside the mesh; in either list
    for extra in ([int(ds100[0, 0]), 3], [mesh.num_cells, 0], [int(ds101[0, 0]), -1]):
        bad = torch.cat([ds101, torch.tensor([extra], dtype=torch.int32, device="cuda")])
        with pytest.raises(ValueError, match="entity's cell is not tagged 1, 2 or 3"):
            symbolic.DeviceElasticityPattern(mesh, ctags, ftags, (ds100, bad))
        with pytest.raises(ValueError, match="entity's cell is not tagged 1, 2 or 3"):
            symbolic.DeviceElasticityPattern(mesh, ctags, ftags, (bad, ds101))
    # the library is usable after the refusals
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=Vp)
    _assert_same_arrays(symbolic.DeviceElasticityPattern(mesh, ctags, ftags, d_bdry), plan)


def test_hexahedra_are_refused():
    mesh = synthetic.hexahedron_mesh(3, device="cuda")
    c8 = torch.ones(mesh.num_cells, dtype=torch.int8, device="cuda")
    f8 = torch.ones(mesh.num_facets, dtype=torch.int8, device="cuda")
    with pytest.raises(NotImplementedError, match="cell type 3"):
        symbolic.DeviceElasticityPattern(mesh, types.SimpleNamespace(tags8=c8), types.SimpleNamespace(tags8=f8),
                                         (None, None))


def test_c_host_without_python_reproduces_the_python_path(tmp_path):
    """examples/capi_host_elasticity.cu: a unit-square triangle mesh built in C, tags -> entities -> pattern ->
    interface-elasticity assembly with Dirichlet conditions through the C ABI."""
    exe = tmp_path / "capi_host_elasticity"
    lib_dir = os.path.join(ROOT, "phifem_b200")
    subprocess.run(["nvcc", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    os.path.join(ROOT, "examples", "capi_host_elasticity.cu"), "-I", os.path.join(ROOT, "include"),
                    "-L", lib_dir, "-lphifem_b200", "-Xlinker", "-rpath=" + lib_dir, "-o", str(exe)], check=True)
    n = 48
    out = subprocess.run([str(exe), str(n)], check=True, capture_output=True, text=True).stdout
    got = dict(item.split("=") for item in out.split())
    # the same problem through the Python package
    mesh = synthetic.rectangle_mesh(n, lo=(0.0, 0.0), hi=(1.0, 1.0), device="cuda")
    X = mesh.x
    phi = (X[:, 0] - 0.503) ** 2 + (X[:, 1] - 0.497) ** 2 - 0.3 ** 2
    f = torch.stack([1.0 + X[:, 0] + 2.0 * X[:, 1], X[:, 0] - 0.5 * X[:, 1]], dim=1).contiguous()
    fn = fem.Function(fem.functionspace(mesh, 1), phi)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, d_bdry, _ = mesh_scripts.compute_tags_measures(mesh, fn, 1, box_mode=True)
    c8 = ctags.values_dev
    assert [int(got["interior"]), int(got["cut"]), int(got["exterior"])] == \
        [int((c8 == 1).sum()), int((c8 == 2).sum()), int((c8 == 3).sum())]
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry)
    bv = plan.boundary_vertices()
    g = torch.stack([X[bv, 0] - X[bv, 1], X[bv, 0] + 0.5 * X[bv, 1]], dim=1)
    dofs = torch.cat([plan.dofs("u_in", bv), plan.dofs("u_out", bv)], dim=1).reshape(-1)
    vals = torch.cat([g, g], dim=1).reshape(-1)
    A, b = elasticity.assemble_interface_elasticity(plan, phi, f, pen_coef=1.0, stab_coef=1.0, bcs=(dofs, vals))
    assert int(got["nnz"]) == plan.nnz and int(got["n_pairs"]) == int(plan.vptr[-1])
    assert int(got["n_cut"]) == plan.cut_cells.numel() > 0
    assert int(got["n_facets_in"]) == plan.facets_in.numel() > 0
    assert int(got["n_facets_out"]) == plan.facets_out.numel() > 0
    assert int(got["n_entities_in"]) == plan.entities_in.shape[0] > 0
    assert int(got["n_entities_out"]) == plan.entities_out.shape[0] > 0
    assert int(got["n_bc"]) == dofs.numel()
    weights = torch.arange(plan.nnz, device="cuda") % 7 + 1
    assert int(got["indices_checksum"]) == int((plan.indices.long() * weights).sum())
    abs_sum = float(A.data.abs().sum())
    assert abs(float(got["data_abs_sum"]) - abs_sum) <= 1e-12 * abs_sum
    assert abs(float(got["b_sum"]) - float(b.sum())) <= 1e-12 * float(b.abs().sum())
