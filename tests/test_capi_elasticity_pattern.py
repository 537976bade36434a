"""CPU-only: phifem_elasticity_pattern_create (csrc/symbolic.cu) refuses bad arguments before any CUDA call, with
PHIFEM_ERR_ARGUMENT and a message naming the field, and refuses hexahedral meshes and unknown cell types with
PHIFEM_ERR_UNSUPPORTED."""
import ctypes

import pytest

from phifem_b200 import _lib

P = 16        # a non-null address the checks never dereference
ARG, UNSUPPORTED = -1, -3


def _mesh(cell_type=_lib.CELL_TYPE_ID["triangle"], cells=P, c2f=P, f2c=P, n_vertices=9, n_cells=8, n_facets=12):
    return _lib.CMesh(cell_type, 2, n_vertices, n_cells, n_facets, P, cells, c2f, f2c, 0.0, 0.0, None, 0)


def _call(mesh=None, c8=P, f8=P, e_in=None, n_in=0, e_out=None, n_out=0, out=True, use_default_mesh=True):
    lib = _lib.load()
    if mesh is None and use_default_mesh:
        mesh = _mesh()
    handle = ctypes.c_void_p()
    rc = lib.phifem_elasticity_pattern_create(ctypes.byref(mesh) if mesh is not None else None, c8, f8, e_in, n_in,
                                              e_out, n_out, ctypes.byref(handle) if out else None, None)
    assert not handle.value
    return rc, lib.phifem_last_error().decode()


@pytest.mark.parametrize("kwargs,text", [
    (dict(out=False), "out is null"),
    (dict(use_default_mesh=False), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(cells=None)), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(c2f=None)), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(f2c=None)), "mesh / facet connectivity is null"),
    (dict(c8=None), "tag arrays are null"),
    (dict(f8=None), "tag arrays are null"),
    (dict(n_in=-1), "entities_in list"),
    (dict(n_in=5), "entities_in list"),
    (dict(n_out=-1, e_in=P, n_in=3), "entities_out list"),
    (dict(n_out=5), "entities_out list"),
    (dict(mesh=_mesh(n_cells=2 ** 31)), "int32 index width"),
    (dict(mesh=_mesh(n_facets=2 ** 31)), "int32 index width"),
    (dict(mesh=_mesh(n_vertices=-1)), "int32 index width"),
    # the blocked dofs NB v + b must fit int32: NB = 14 on triangles
    (dict(mesh=_mesh(n_vertices=2 ** 31 // 14 + 1)), "int32 index width"),
    (dict(mesh=_mesh(cell_type=_lib.CELL_TYPE_ID["tetrahedron"], n_vertices=2 ** 31 // 27 + 1)), "int32 index width"),
])
def test_argument_errors_need_no_gpu(kwargs, text):
    rc, msg = _call(**kwargs)
    assert rc == ARG
    assert msg == "phifem_elasticity_pattern_create: " + text


@pytest.mark.parametrize("cell_type", ["quadrilateral", "tetrahedron"])
def test_quadrilaterals_and_tetrahedra_pass_the_cell_type_check(cell_type):
    rc, msg = _call(mesh=_mesh(cell_type=_lib.CELL_TYPE_ID[cell_type]), c8=None)
    assert rc == ARG and msg == "phifem_elasticity_pattern_create: tag arrays are null"


def test_hexahedra_are_unsupported():
    rc, msg = _call(mesh=_mesh(cell_type=_lib.CELL_TYPE_ID["hexahedron"]))
    assert rc == UNSUPPORTED
    assert "cell type 3" in msg and "triangles, quadrilaterals and tetrahedra" in msg


def test_unknown_cell_type_is_unsupported():
    rc, msg = _call(mesh=_mesh(cell_type=7))
    assert rc == UNSUPPORTED and "cell type 7" in msg


def test_view_and_destroy_accept_null():
    lib = _lib.load()
    assert lib.phifem_elasticity_pattern_view_of(None, None) == ARG
    assert "null pointer" in lib.phifem_last_error().decode()
    lib.phifem_elasticity_pattern_destroy(None)
