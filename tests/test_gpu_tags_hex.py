"""GPU: hexahedral classification (csrc/tags.cu through the C ABI) against the CPU oracle (oracle/tags_hex.py).

Bit-exact bar, as for the other cell types: cell tags, facet tags, the ds(100) / ds(101) entity lists, the submesh
arrays and the counters of the tag kernels equal the oracle's."""
import ctypes
import itertools
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import tags as OT
from oracle import tags_hex as OH
from phifem_b200 import _lib, fem, mesh_scripts, synthetic
from phifem_b200.mesh import MeshTags

pytestmark = pytest.mark.gpu

CENTER = (0.5 + math.pi / 1000.0, 0.5 + math.e / 1000.0, 0.5 + math.sqrt(2.0) / 1000.0)


def sphere(x, r=0.33):
    return (x[0] - CENTER[0]) ** 2 + (x[1] - CENTER[1]) ** 2 + (x[2] - CENTER[2]) ** 2 - r * r


def _mesh(kind, n=6):
    mesh = synthetic.hexahedron_mesh(n, device="cuda")
    if kind == "jittered":     # convex, non-affine cells, random cell order and vertex labels
        mesh = synthetic.unstructured_variant(mesh, jitter=0.2, seed=4)
    return mesh


def _levelset(mesh, kind):
    """(what compute_tags_measures takes, phi at the oracle's points given the detection degree)."""
    x, cells = mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64)
    if kind == "expr":
        return sphere, lambda N: (OH.point_values_expression(sphere, x, cells, OH.boundary_points(N)),
                                  OH.point_values_expression(sphere, x, cells, OH.facet_points_in_cell(N)))
    V = fem.functionspace(mesh, ("Lagrange", 1 if kind == "Q1" else 2))
    fn = fem.Function(V).interpolate(sphere)
    tab = V.element.tabulate
    return fn, lambda N: (OT.point_values_function(fn.x.array, V.dofmap, tab(OH.boundary_points(N))),
                          OT.point_values_function(fn.x.array, V.dofmap, tab(OH.facet_points_in_cell(N))))


def _run(mesh, ls, N, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return mesh_scripts.compute_tags_measures(mesh, ls, N, **kw)


def _counters(mesh, ls, N, single):
    dls = mesh_scripts._DeviceLevelset(mesh, ls, N)
    ws = mesh_scripts.classify(mesh, dls, single)
    torch.cuda.synchronize()
    return ws.counters.cpu().numpy()


def _assert_tags(mine, want):
    idx = np.nonzero(want)[0]
    assert np.array_equal(mine.indices, idx)
    assert np.array_equal(mine.values, want[idx])


CASES = list(itertools.product(("structured", "jittered"), ("Q1", "Q2", "expr"), (0, 1, 2, 3), (True, False),
                               (False, True)))


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%s-%s-N%d-%s-%s" % (
    c[0], c[1], c[2], "box" if c[3] else "sub", "single" if c[4] else "multi"))
def test_cuda_hex_tags_match_oracle(case):
    mesh_kind, ls_kind, N, box, single = case
    mesh = _mesh(mesh_kind)
    ls, oracle_values = _levelset(mesh, ls_kind)
    ctags, ftags, sub, ds, maps = _run(mesh, ls, N, box_mode=box, single_layer_cut=single)
    x, cells = mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64)
    phi_c, phi_f = oracle_values(N)
    out = OH.compute_tags_measures(x, cells, phi_c, phi_f, N, box_mode=box, single_layer_cut=single)
    assert np.array_equal(mesh.c2f.cpu().numpy(), out["c2f"])
    assert np.array_equal(mesh.f2c.cpu().numpy(), out["f2c"])
    _assert_tags(ctags, out["cell_tags"])
    _assert_tags(ftags, out["facet_tags"])
    if box:
        assert sub is None and maps is None
        assert np.array_equal(ds(100).integration_entities, out["ds100"])
        assert np.array_equal(ds(101).integration_entities, out["ds101"])
    else:
        assert np.array_equal(maps[0], out["c_map"])
        assert np.array_equal(maps[1], out["v_map"])
        assert np.array_equal(sub.cells.cpu().numpy(), out["sub_cells"])
        assert np.array_equal(sub.x.cpu().numpy(), out["sub_x"])
        assert sub.cell_type == "hexahedron"
    cnt, want = _counters(mesh, ls, N, single), out["counts"]
    assert [cnt[_lib.CNT_INTERIOR], cnt[_lib.CNT_CUT], cnt[_lib.CNT_EXTERIOR], cnt[_lib.CNT_UNTAGGED]] == \
        [want["interior"], want["cut"], want["exterior"], want["untagged"]]
    assert cnt[_lib.CNT_FACET_CONFLICT] == want["facet_conflicts"]
    assert cnt[_lib.CNT_BOUNDARY_OWNERS] == want["boundary_owners"]
    if N >= 1:
        assert want["cut"] > 0 and want["interior"] > 0 and want["exterior"] > 0


@pytest.mark.parametrize("ls_kind", ["Q2", "expr"])
def test_cuda_hex_overwrite_tags_and_one_sided_measures(ls_kind):
    mesh = _mesh("jittered")
    ls, oracle_values = _levelset(mesh, ls_kind)
    N = 2
    ct0, ft0, *_ = _run(mesh, ls, N, box_mode=True)
    cut = ct0.find(2)[:5]
    gam = ft0.find(4)[:7]
    ow = {"cells": MeshTags.from_lists(mesh, 3, cut, np.full(len(cut), 7)),
          "facets": MeshTags.from_lists(mesh, 2, gam, np.full(len(gam), 260))}
    ctags, ftags, _, ds, _ = _run(mesh, ls, N, box_mode=True, overwrite_tags=ow)
    x, cells = mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64)
    out = OH.compute_tags_measures(x, cells, *oracle_values(N), N, box_mode=True)
    ct, ft = out["cell_tags"].copy(), out["facet_tags"].copy()
    ct[cut], ft[gam] = 7, 260
    _assert_tags(ctags, ct)
    _assert_tags(ftags, ft)
    # the one-sided measures follow the overwritten tags: 7 and 260 match nothing
    c2f, f2c = out["c2f"], out["f2c"]
    assert np.array_equal(ds(100).integration_entities,
                          OT.integration_entities(c2f, f2c, (ct == 1) | (ct == 2), ft == 4))
    assert np.array_equal(ds(101).integration_entities,
                          OT.integration_entities(c2f, f2c, (ct == 2) | (ct == 3), ft == 3))
    with pytest.raises(ValueError):
        _run(mesh, ls, N, box_mode=True,
             overwrite_tags={"cells": MeshTags.from_lists(mesh, 3, cut[:1], np.array([2]))})


@pytest.mark.parametrize("ls_kind,N", [("Q1", 1), ("Q2", 2), ("expr", 3)])
def test_cuda_hex_divergence_theorem_on_gamma_h(ls_kind, N):
    n = 12
    mesh = synthetic.hexahedron_mesh(n, device="cuda")
    ls, _ = _levelset(mesh, ls_kind)
    ctags, ftags, _, ds, _ = _run(mesh, ls, N, box_mode=True)
    ct, ft = ctags.values_dev.cpu().numpy(), ftags.values_dev.cpu().numpy()
    assert not np.any(ft == 6)          # no interior cell touches an exterior one: ds(100) closes around Omega_h
    assert not np.any(ft[mesh.boundary_facets.cpu().numpy()] == 4)
    x, cells = mesh.x.cpu().numpy(), mesh.cells.cpu().numpy().astype(np.int64)
    ents = ds(100).integration_entities.reshape(-1, 2)
    assert len(ents) > 0
    nrm, area = OH.outward_normals(x, cells, ents)
    xf = np.array([x[cells[c]][list(OH.LOCAL_FACETS[lf])].mean(axis=0) for c, lf in ents])
    total = area.sum()
    assert np.abs((area[:, None] * nrm).sum(axis=0)).max() <= 1e-12 * total
    volume = ((ct == 1) | (ct == 2)).sum() * (1.0 / n) ** 3
    flux = (area * (xf * nrm).sum(axis=1)).sum() / 3.0
    assert abs(flux - volume) <= 1e-12 * volume


def _c_levelset(mesh, N):
    fn = fem.Function(fem.functionspace(mesh, 2)).interpolate(sphere)
    return mesh_scripts._DeviceLevelset(mesh, fn, N)


def test_cuda_hex_capi_argument_errors():
    mesh = _mesh("structured", 3)
    lib = _lib.load()
    dls = _c_levelset(mesh, 2)
    ws = mesh_scripts.TagWorkspace(mesh)
    ws.vertex_scratch = torch.empty(mesh.num_vertices + 3, dtype=torch.uint8, device=mesh.device)
    cm = _lib.c_mesh(mesh)

    def tag_cells(ls):
        return lib.phifem_tag_cells(cm, ctypes.byref(ls), 0, None, _lib.ptr(ws.cell_tags8),
                                    _lib.ptr(ws.vertex_scratch), _lib.ptr(ws.counters), _lib.stream())

    def tag_facets(ls):
        return lib.phifem_tag_facets(cm, ctypes.byref(ls), _lib.ptr(ws.cell_tags8), None, _lib.ptr(ws.facet_tags8),
                                     _lib.ptr(ws.counters), _lib.stream())

    def copy(**fields):
        ls = _lib.CLevelset()
        ctypes.pointer(ls)[0] = dls.c
        for k, v in fields.items():
            setattr(ls, k, v)
        return ls

    assert tag_cells(dls.c) == 0 and tag_facets(dls.c) == 0
    for call in (tag_cells, tag_facets):
        assert call(copy(coord_grad=None)) == -1
        assert b"levelset.coord_grad" in lib.phifem_last_error()
        assert call(copy(n_dofs_per_cell=28)) == -1
        assert b"levelset.n_dofs_per_cell" in lib.phifem_last_error()
        assert call(copy(dofmap=None)) == -1
        assert b"levelset.dofmap" in lib.phifem_last_error()
    owner = torch.zeros((mesh.boundary_facets.numel(), 2), dtype=torch.int32, device=mesh.device)
    scale = torch.zeros((mesh.boundary_facets.numel(), 4), dtype=torch.float64, device=mesh.device)
    assert lib.phifem_boundary_records(cm, _lib.ptr(owner), _lib.ptr(scale), _lib.stream()) == -3
    assert b"hexahedra" in lib.phifem_last_error()
    assert lib.phifem_abi_version() == 1
    torch.cuda.synchronize()


def test_cuda_hex_several_million_cells_follow_the_vertex_sign_rule():
    n = 160                                             # 4.1 M hexahedra
    mesh = synthetic.unstructured_variant_device(synthetic.hexahedron_mesh(n, device="cuda"), jitter=0.2, seed=9)
    phi = synthetic.sphere_levelset(mesh.x, radius=0.41)
    fn = fem.Function(fem.functionspace(mesh, 1), phi)
    ctags, ftags, _, ds, _ = _run(mesh, fn, 1, box_mode=True)
    # Q1, N = 1: the points are the vertices and every scale |det J| > 0, so a cell is interior / exterior iff phi has
    # one sign on its 8 vertices, cut otherwise (no vertex value is 0)
    pv = phi[mesh.cells.long()]
    assert bool((pv != 0).all())
    want = torch.where((pv < 0).all(dim=1), 1, torch.where((pv > 0).all(dim=1), 3, 2)).to(torch.int8)
    assert torch.equal(ctags.tags8, want)
    counts = torch.bincount(want.long(), minlength=4).cpu().numpy()
    assert counts[2] > 10000 and counts[1] > 0 and counts[3] > 0
    # interior facets between an interior and a cut cell are tagged 3, between cut and exterior 4
    f2c = mesh.f2c.long()
    inner = f2c[:, 1] >= 0
    t0, t1 = want[f2c[inner, 0]], want[f2c[inner, 1]]
    ft = ftags.tags8[inner]
    assert torch.equal(ft[(t0 == 1) & (t1 == 2) | (t0 == 2) & (t1 == 1)].unique().cpu(),
                       torch.tensor([3], dtype=torch.int8))
    assert torch.equal(ft[(t0 == 3) & (t1 == 2) | (t0 == 2) & (t1 == 3)].unique().cpu(),
                       torch.tensor([4], dtype=torch.int8))
    assert len(ds(100).integration_entities) == 2 * int(((t0 == 3) & (t1 == 2) | (t0 == 2) & (t1 == 3)).sum())
