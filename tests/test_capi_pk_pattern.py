"""CPU-only: phifem_pk_pattern_create (csrc/symbolic.cu) refuses bad arguments before any CUDA call, with
PHIFEM_ERR_ARGUMENT and a message naming the field, and refuses hexahedral meshes with PHIFEM_ERR_UNSUPPORTED."""
import ctypes

import pytest

from phifem_b200 import _lib

P = 16        # a non-null address the checks never dereference
ARG, UNSUPPORTED = -1, -3


def _mesh(cell_type=_lib.CELL_TYPE_ID["triangle"], cells=P, c2f=P, f2c=P, n_cells=8, n_facets=12):
    return _lib.CMesh(cell_type, 2, 9, n_cells, n_facets, P, cells, c2f, f2c, 0.0, 0.0, None, 0)


def _call(mesh=None, dofmap=P, nd=3, n_rows=9, c8=P, f8=P, mask=(1 << 2) | (1 << 3), entities=None, n_entities=0,
          out=True, use_default_mesh=True):
    lib = _lib.load()
    if mesh is None and use_default_mesh:
        mesh = _mesh()
    handle = ctypes.c_void_p()
    rc = lib.phifem_pk_pattern_create(ctypes.byref(mesh) if mesh is not None else None, dofmap, nd, n_rows, c8, f8,
                                      mask, entities, n_entities, ctypes.byref(handle) if out else None, None)
    assert not handle.value
    return rc, lib.phifem_last_error().decode()


@pytest.mark.parametrize("kwargs,text", [
    (dict(out=False), "out is null"),
    (dict(use_default_mesh=False), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(cells=None)), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(c2f=None)), "mesh / facet connectivity is null"),
    (dict(mesh=_mesh(f2c=None)), "mesh / facet connectivity is null"),
    (dict(dofmap=None), "dofmap is null"),
    (dict(c8=None), "tag arrays are null"),
    (dict(f8=None), "tag arrays are null"),
    (dict(nd=0), "nd (dofs per cell) must lie in 1..32"),
    (dict(nd=33), "nd (dofs per cell) must lie in 1..32"),
    (dict(nd=-4), "nd (dofs per cell) must lie in 1..32"),
    (dict(n_rows=0), "n_rows must lie in 1..2^31-1"),
    (dict(n_rows=2 ** 31), "n_rows must lie in 1..2^31-1"),
    (dict(n_entities=-1), "entity list"),
    (dict(n_entities=5), "entity list"),
    (dict(mask=1 << 7), "ghost_tag_mask sets bits outside the tag values 0..6"),
    (dict(mask=0xFFFFFFFF), "ghost_tag_mask sets bits outside the tag values 0..6"),
    (dict(mesh=_mesh(n_cells=2 ** 31)), "int32 index width"),
])
def test_argument_errors_need_no_gpu(kwargs, text):
    rc, msg = _call(**kwargs)
    assert rc == ARG
    assert msg == "phifem_pk_pattern_create: " + text


def test_the_bounds_of_nd_and_n_rows_pass_the_host_checks():
    """nd = 32 and n_rows = 2^31 - 1 are accepted: the call gets as far as the mesh's index width."""
    rc, msg = _call(nd=32, n_rows=2 ** 31 - 1, mesh=_mesh(n_cells=2 ** 31))
    assert rc == ARG and msg == "phifem_pk_pattern_create: int32 index width"


@pytest.mark.parametrize("cell_type", ["quadrilateral", "tetrahedron"])
def test_quadrilaterals_and_tetrahedra_pass_the_cell_type_check(cell_type):
    rc, msg = _call(mesh=_mesh(cell_type=_lib.CELL_TYPE_ID[cell_type]), dofmap=None)
    assert rc == ARG and msg == "phifem_pk_pattern_create: dofmap is null"


def test_hexahedra_are_unsupported():
    rc, msg = _call(mesh=_mesh(cell_type=_lib.CELL_TYPE_ID["hexahedron"]))
    assert rc == UNSUPPORTED
    assert "cell type 3" in msg and "triangles, quadrilaterals and tetrahedra" in msg


def test_unknown_cell_type_is_unsupported():
    rc, msg = _call(mesh=_mesh(cell_type=7))
    assert rc == UNSUPPORTED and "cell type 7" in msg


def test_view_and_destroy_accept_null():
    lib = _lib.load()
    assert lib.phifem_pk_pattern_view_of(None, None) == ARG
    assert "null pointer" in lib.phifem_last_error().decode()
    lib.phifem_pk_pattern_destroy(None)
