"""The symbolic phase of the quadrature-kernel operators behind the C ABI (csrc/symbolic.cu, phifem_pk_pattern_create)
produces bit for bit the arrays of the torch-based PkAssemblyPlan (phifem_b200/assemble_pk.py) -- CSR pattern, active
cells, cut-cell positions, ghost-penalty facets, the three slot maps -- for strong / weak Dirichlet, Neumann and Robin on
triangles, tetrahedra and quadrilaterals; the operators assembled through those arrays equal the plan's; a host program
without Python (examples/capi_host_pk.cu) reproduces the weak-Dirichlet and Neumann checksums of the Python path."""
import copy
import os
import subprocess
import warnings

import numpy as np
import pytest
import torch

from phifem_b200 import assemble, fem, mesh_scripts, symbolic, synthetic
from phifem_b200.assemble_pk import assemble_neumann_into, assemble_pk_into, assemble_weak_into

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("indptr", "indices", "active", "cut_positions", "ghost", "entities", "slots_cells", "slots_ghost",
         "slots_boundary")


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


def _tags(mesh, center, radius):
    det = fem.Function(fem.functionspace(mesh, 1),
                       synthetic.sphere_levelset(mesh.x, center=center, radius=radius).cpu().numpy())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, ds, _ = mesh_scripts.compute_tags_measures(mesh, det, 1, box_mode=True)
    return ctags, ftags, ds


def _plan(form, mesh, ctags, ftags, ents, kw, kphi):
    V, Vp = fem.functionspace(mesh, kw), fem.functionspace(mesh, kphi)
    if form == "strong":
        return assemble.build_plan(mesh, ctags, ftags, ents, V=V, V_phi=Vp, method="pk"), (2, 3)
    if form == "weak":
        return assemble.build_plan_weak_dirichlet(mesh, ctags, ftags, ents, V=V, V_phi=Vp), (2, 3)
    gtag = 2 if form == "robin" else 3
    return assemble.build_plan_neumann(mesh, ctags, ftags, ents, V_phi=Vp, ghost_tag=gtag), (gtag,)


def _native(plan, mesh, ctags, ftags, ents, ghost_tags):
    return symbolic.DevicePkPattern(mesh, ctags, ftags, ents, plan.pattern_dofmap, plan.n_rows, ghost_tags=ghost_tags)


def _assert_same_arrays(pat, plan):
    assert pat.nnz == plan.nnz and pat.n_rows == plan.n_rows
    for name in NAMES:
        a, b = getattr(pat, name), getattr(plan, name)
        assert a.dtype == b.dtype == torch.int32 and a.shape == b.shape, name
        assert torch.equal(a, b), name


def _assemble(plan, form, mesh, center, radius):
    """data, b of the plan's operator: phi_h = the interpolated level set, seeded data."""
    rng = np.random.default_rng(5)
    cuda = lambda n: torch.from_numpy(rng.uniform(-1, 1, n)).cuda()  # noqa: E731
    phi = synthetic.sphere_levelset(plan.V_phi.dof_coordinates_dev(), center=center, radius=radius)
    data, b = plan.new_outputs()
    if form == "strong":
        assemble_pk_into(plan, phi, cuda(plan.V.num_dofs), 0.9, data, b)
    elif form == "weak":
        assemble_weak_into(plan, phi, cuda(plan.V.num_dofs), cuda(plan.V.num_dofs), 1.3, 0.7, data, b)
    else:
        assemble_neumann_into(plan, phi, cuda(mesh.num_vertices), cuda(mesh.num_vertices), 1.3, 0.7, data, b,
                              robin_coef=0.8 if form == "robin" else 0.0)
    torch.cuda.synchronize()
    return data, b


def _assert_same_operator(plan, pat, form, mesh, center, radius):
    """The plan with the native arrays assembles the plan's own operator (fp64 atomics reorder the sums)."""
    native = copy.copy(plan)
    for name in NAMES:
        setattr(native, name, getattr(pat, name))
    d0, b0 = _assemble(plan, form, mesh, center, radius)
    d1, b1 = _assemble(native, form, mesh, center, radius)
    rows = torch.repeat_interleave(torch.arange(plan.n_rows, device="cuda"),
                                   (plan.indptr[1:] - plan.indptr[:-1]).long())
    scale = torch.zeros(plan.n_rows, dtype=torch.float64, device="cuda").scatter_reduce(0, rows, d0.abs(), "amax")
    assert bool(((d1 - d0).abs() <= 1e-14 * scale[rows]).all())
    assert float((b1 - b0).abs().max()) <= 1e-14 * float(b0.abs().max())
    assert float(d0.abs().sum()) > 0 and float(b0.abs().sum()) > 0


CASES = [
    # form, mesh kind, n, kw (trial / test degree), kphi (level-set degree)
    ("strong", "tri", 14, 1, 2), ("strong", "tri", 14, 2, 2),
    ("strong", "tri-unstructured", 10, 1, 2), ("strong", "tri-unstructured", 10, 2, 2),
    ("strong", "tet", 5, 1, 2), ("strong", "tet", 5, 2, 2),
    ("strong", "tet-unstructured", 4, 1, 2), ("strong", "tet-unstructured", 4, 2, 2),
    ("weak", "tri", 14, 1, 1), ("weak", "tri", 14, 2, 2), ("weak", "tri-unstructured", 10, 2, 1),
    ("weak", "tet", 5, 1, 1), ("weak", "tet-unstructured", 4, 1, 2),
    ("neumann", "tri", 14, 1, 1), ("neumann", "tri", 14, 1, 2), ("neumann", "tri-unstructured", 10, 1, 2),
    ("neumann", "tet", 5, 1, 2), ("neumann", "tet-unstructured", 4, 1, 1),
    ("robin", "tri", 14, 1, 1), ("robin", "tet-unstructured", 4, 1, 2),
    ("strong", "quad", 14, 1, 1), ("strong", "quad", 14, 1, 2), ("strong", "quad-unstructured", 10, 1, 2),
    ("neumann", "quad", 14, 1, 2), ("neumann", "quad-unstructured", 10, 1, 2), ("robin", "quad", 14, 1, 2),
]


@pytest.mark.parametrize("form,kind,n,kw,kphi", CASES)
def test_device_pk_pattern_equals_the_torch_plan(form, kind, n, kw, kphi):
    mesh, center, radius = _mesh(kind, n)
    ctags, ftags, ds = _tags(mesh, center, radius)
    plan, gt = _plan(form, mesh, ctags, ftags, ds(100), kw, kphi)
    assert plan.active.numel() and plan.cut_positions.numel() and plan.ghost.numel() and plan.entities.shape[0]
    pat = _native(plan, mesh, ctags, ftags, ds(100), gt)
    _assert_same_arrays(pat, plan)
    _assert_same_operator(plan, pat, form, mesh, center, radius)


def test_weak_p2_tetrahedra_the_widest_pattern_dofmap():
    """nd = 20: the mixed P2 x P2 space on tetrahedra."""
    mesh, center, radius = _mesh("tet", 4)
    ctags, ftags, ds = _tags(mesh, center, radius)
    plan, gt = _plan("weak", mesh, ctags, ftags, ds(100), 2, 2)
    assert plan.pattern_dofmap.shape[1] == 20
    _assert_same_arrays(_native(plan, mesh, ctags, ftags, ds(100), gt), plan)


@pytest.mark.parametrize("form", ["strong", "weak", "neumann"])
def test_nothing_active(form):
    """A disc outside the mesh: no active cell, no ghost facet, no entity; empty arrays, indptr all zero."""
    mesh = synthetic.rectangle_mesh(6, device="cuda")
    ctags, ftags, ds = _tags(mesh, (5.0, 5.0), 0.5)
    plan, gt = _plan(form, mesh, ctags, ftags, ds(100), 1, 1)
    pat = _native(plan, mesh, ctags, ftags, ds(100), gt)
    assert pat.nnz == 0 and pat.active.numel() == 0 and pat.ghost.numel() == 0 and pat.entities.numel() == 0
    assert torch.equal(pat.indptr, torch.zeros(plan.n_rows + 1, dtype=torch.int32, device="cuda"))
    _assert_same_arrays(pat, plan)


@pytest.mark.parametrize("form", ["strong", "neumann"])
def test_without_entities(form):
    mesh, center, radius = _mesh("tri-unstructured", 10)
    ctags, ftags, _ = _tags(mesh, center, radius)
    plan, gt = _plan(form, mesh, ctags, ftags, None, 1, 2)
    pat = _native(plan, mesh, ctags, ftags, None, gt)
    assert pat.entities.shape == (0, 2) and pat.slots_boundary.numel() == 0 and pat.ghost.numel() > 0
    _assert_same_arrays(pat, plan)
    _assert_same_operator(plan, pat, form, mesh, center, radius)


def test_without_ghost_facets():
    """A disc covering the whole mesh: every cell interior, no cut cell, no ghost facet, no entity."""
    mesh, _, _ = _mesh("quad-unstructured", 8)
    ctags, ftags, ds = _tags(mesh, (0.0, 0.0), 10.0)
    plan, gt = _plan("neumann", mesh, ctags, ftags, ds(100), 1, 1)
    pat = _native(plan, mesh, ctags, ftags, ds(100), gt)
    assert pat.active.numel() == mesh.num_cells and pat.ghost.numel() == 0 and pat.cut_positions.numel() == 0
    assert pat.slots_ghost.shape == (0, 4 * 13 * 13)
    _assert_same_arrays(pat, plan)
    _assert_same_operator(plan, pat, "neumann", mesh, (0.0, 0.0), 10.0)


def test_a_ghost_mask_without_facets():
    """ghost_tags=() selects no facet; the rest of the pattern is the plan's minus the macro elements' entries."""
    mesh, center, radius = _mesh("tri", 10)
    ctags, ftags, ds = _tags(mesh, center, radius)
    plan, _ = _plan("strong", mesh, ctags, ftags, ds(100), 1, 1)
    pat = _native(plan, mesh, ctags, ftags, ds(100), ())
    assert pat.ghost.numel() == 0 and 0 < pat.nnz < plan.nnz
    assert torch.equal(pat.active, plan.active) and torch.equal(pat.cut_positions, plan.cut_positions)


def test_device_refusals():
    mesh, center, radius = _mesh("tri", 10)
    ctags, ftags, ds = _tags(mesh, center, radius)
    plan, gt = _plan("weak", mesh, ctags, ftags, ds(100), 1, 1)
    # a dofmap entry >= n_rows (the largest dof of the plan's dofmap is n_rows - 1)
    with pytest.raises(ValueError, match="dofmap has entries outside"):
        symbolic.DevicePkPattern(mesh, ctags, ftags, ds(100), plan.pattern_dofmap, plan.n_rows - 1, ghost_tags=gt)
    bad = plan.pattern_dofmap.clone()
    bad[0, 0] = -1
    with pytest.raises(ValueError, match="dofmap has entries outside"):
        symbolic.DevicePkPattern(mesh, ctags, ftags, ds(100), bad, plan.n_rows, ghost_tags=gt)
    # an entity whose cell is tagged 3 (as ds(101) may hold): its keys are not in the pattern
    c8 = ctags.values_dev
    ents = ds(100).integration_entities.reshape(-1, 2)
    exterior = int(torch.nonzero(c8 == 3)[0, 0])
    for extra in ([exterior, 0], [int(plan.active[0]), 3], [mesh.num_cells, 0]):   # tag 3, local facet, cell id
        with_bad = np.concatenate([np.asarray(ents), np.asarray([extra])]).astype(np.int32)
        with pytest.raises(ValueError, match="entity's cell is not tagged 1 or 2"):
            symbolic.DevicePkPattern(mesh, ctags, ftags, with_bad, plan.pattern_dofmap, plan.n_rows, ghost_tags=gt)
    ds101 = np.asarray(ds(101).integration_entities).reshape(-1, 2)
    if np.any(c8.cpu().numpy()[ds101[:, 0]] == 3):
        with pytest.raises(ValueError, match="entity's cell is not tagged 1 or 2"):
            symbolic.DevicePkPattern(mesh, ctags, ftags, ds(101), plan.pattern_dofmap, plan.n_rows, ghost_tags=gt)
    with pytest.raises(ValueError, match="ghost tag"):
        symbolic.DevicePkPattern(mesh, ctags, ftags, ds(100), plan.pattern_dofmap, plan.n_rows, ghost_tags=(7,))
    # the library is usable after the refusals
    _assert_same_arrays(_native(plan, mesh, ctags, ftags, ds(100), gt), plan)


def test_c_host_without_python_reproduces_the_python_path(tmp_path):
    """examples/capi_host_pk.cu: a unit-square triangle mesh built in C, tags -> entities -> pattern -> weak-Dirichlet
    and Neumann assembly through the C ABI."""
    exe = tmp_path / "capi_host_pk"
    lib_dir = os.path.join(ROOT, "phifem_b200")
    subprocess.run(["nvcc", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    os.path.join(ROOT, "examples", "capi_host_pk.cu"), "-I", os.path.join(ROOT, "include"),
                    "-L", lib_dir, "-lphifem_b200", "-Xlinker", "-rpath=" + lib_dir, "-o", str(exe)], check=True)
    n = 48
    out = subprocess.run([str(exe), str(n)], check=True, capture_output=True, text=True).stdout
    got = dict(item.split("=") for item in out.split())
    # the same problem through the Python package
    mesh = synthetic.rectangle_mesh(n, lo=(0.0, 0.0), hi=(1.0, 1.0), device="cuda")
    X = mesh.x
    phi = (X[:, 0] - 0.503) ** 2 + (X[:, 1] - 0.497) ** 2 - 0.3 ** 2
    f = 1.0 + X[:, 0] + 2.0 * X[:, 1]
    g = X[:, 0] - 0.5 * X[:, 1]
    fn = fem.Function(fem.functionspace(mesh, 1), phi)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, ds, _ = mesh_scripts.compute_tags_measures(mesh, fn, 1, box_mode=True)
    c8 = ctags.values_dev
    assert [int(got["interior"]), int(got["cut"]), int(got["exterior"])] == \
        [int((c8 == 1).sum()), int((c8 == 2).sum()), int((c8 == 3).sum())]
    weak = assemble.build_plan_weak_dirichlet(mesh, ctags, ftags, ds(100))
    Aw, bw = assemble.assemble_weak_dirichlet(weak, phi, f, u_D=g, pen_coef=1.0, stab_coef=1.0)
    neu = assemble.build_plan_neumann(mesh, ctags, ftags, ds(100), ghost_tag=3)
    An, bn = assemble.assemble_neumann(neu, phi, f, g, pen_coef=1.0, stab_coef=1.0)
    for name, plan, A, b in (("weak", weak, Aw, bw), ("neumann", neu, An, bn)):
        assert int(got[name + "_nnz"]) == plan.nnz
        assert int(got[name + "_n_active"]) == plan.active.numel()
        assert int(got[name + "_n_cut"]) == plan.cut_positions.numel() > 0
        assert int(got[name + "_n_ghost"]) == plan.ghost.numel() > 0
        assert int(got[name + "_n_entities"]) == plan.entities.shape[0] > 0
        weights = torch.arange(plan.nnz, device="cuda") % 7 + 1
        assert int(got[name + "_indices_checksum"]) == int((plan.indices.long() * weights).sum())
        abs_sum = float(A.data.abs().sum())
        assert abs(float(got[name + "_data_abs_sum"]) - abs_sum) <= 1e-11 * abs_sum
        assert abs(float(got[name + "_b_sum"]) - float(b.sum())) <= 1e-11 * float(b.abs().sum())
