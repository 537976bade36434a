"""ctypes binding of libphifem_b200.so (the C ABI declared in include/phifem_b200.h).

There is no fallback: if the shared library is missing or no CUDA device is present the hot
path raises.  Build the library with `python -m phifem_b200.build` (or `__graft_entry__.build()`).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PHIFEM_B200_LIB") or os.path.join(_HERE, "libphifem_b200.so")

CELL_TYPE_ID = {"triangle": 0, "quadrilateral": 1, "tetrahedron": 2, "hexahedron": 3}
_SIMPLICES = ("triangle", "tetrahedron")
N_COUNTERS = 16
CNT_INTERIOR, CNT_CUT, CNT_EXTERIOR, CNT_UNTAGGED, CNT_ZERO_DEN, CNT_ZERO_DEN_AMBIGUOUS = 0, 1, 2, 3, 4, 5
CNT_FACET_ZERO_DEN, CNT_FACET_CONFLICT, CNT_BOUNDARY_OWNERS = 11, 12, 13
CNT_CALLER0, CNT_CALLER1 = 14, 15

_vp = ctypes.c_void_p


class CMesh(ctypes.Structure):
    _fields_ = [("cell_type", ctypes.c_int32), ("gdim", ctypes.c_int32),
                ("n_vertices", ctypes.c_int64), ("n_cells", ctypes.c_int64),
                ("n_facets", ctypes.c_int64),
                ("x", _vp), ("cells", _vp), ("c2f", _vp), ("f2c", _vp),
                ("detj_min", ctypes.c_double), ("detj_max", ctypes.c_double),
                ("boundary_facets", _vp), ("n_boundary_facets", ctypes.c_int64),
                ("boundary_owner", _vp), ("boundary_scale", _vp), ("x4", _vp)]


class CLevelset(ctypes.Structure):
    _fields_ = [("mode", ctypes.c_int32), ("n_dofs_per_cell", ctypes.c_int32),
                ("n_cell_points", ctypes.c_int32), ("n_facet_points", ctypes.c_int32),
                ("coeffs", _vp), ("dofmap", _vp), ("cell_table", _vp), ("facet_table", _vp),
                ("cell_values", _vp), ("facet_values", _vp), ("coord_grad", _vp)]


class CBlockedPlan(ctypes.Structure):
    _fields_ = [("n_blocks", ctypes.c_int32), ("capacity", ctypes.c_int32),
                ("max_segments", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("block_desc", _vp), ("seg_start", _vp), ("seg_dest", _vp),
                ("n_cell_inst", ctypes.c_int64), ("cell_verts", _vp), ("cell_pos", _vp),
                ("n_ghost_inst", ctypes.c_int64), ("ghost_facet", _vp), ("ghost_pos", _vp),
                ("n_bnd_inst", ctypes.c_int64), ("bnd_entity", _vp), ("bnd_pos", _vp)]


class CRowList(ctypes.Structure):
    _fields_ = [("n_listed", ctypes.c_int64), ("rows", _vp), ("diag_pos", _vp), ("ptr", _vp), ("rec", _vp)]


class CCellTiles(ctypes.Structure):
    _fields_ = [("rows_per_tile", ctypes.c_int32), ("n_tiles", ctypes.c_int32), ("n_listed", ctypes.c_int64),
                ("rows", _vp), ("diag_pos", _vp), ("chunk_ptr", _vp), ("slot_verts", _vp), ("rec_base", _vp),
                ("rec_off", _vp), ("rec", _vp), ("push", _vp)]


class CRowsPlan(ctypes.Structure):
    _fields_ = [("indptr", _vp), ("indices", _vp), ("max_row_nnz", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("cells", CRowList), ("surface", CRowList),
                ("n_ghost_facets", ctypes.c_int64), ("ghost_macro", _vp), ("n_entities", ctypes.c_int64),
                ("entity_macro", _vp), ("surface_work", _vp), ("cell_geom", _vp),
                ("tiles", ctypes.POINTER(CCellTiles)), ("surface_static", _vp)]


class CRowsPlanInfo(ctypes.Structure):
    _fields_ = [("n_rows", ctypes.c_int64), ("nnz", ctypes.c_int64), ("n_active", ctypes.c_int64),
                ("n_ghost", ctypes.c_int64), ("n_entities", ctypes.c_int64), ("active", _vp), ("ghost", _vp),
                ("n_cell_records", ctypes.c_int64), ("n_surface_records", ctypes.c_int64),
                ("cells_record_slots", ctypes.c_int64), ("surface_record_slots", ctypes.c_int64)]


class CPkSpace(ctypes.Structure):
    _fields_ = [("degree", ctypes.c_int32), ("n_dofs_per_cell", ctypes.c_int32), ("n_dofs", ctypes.c_int64),
                ("dofmap", _vp)]


class CQuadrature(ctypes.Structure):
    _fields_ = [("n_cell_points", ctypes.c_int32), ("n_facet_points", ctypes.c_int32),
                ("cell_points", _vp), ("cell_weights", _vp), ("facet_points", _vp), ("facet_weights", _vp)]


class CPatternView(ctypes.Structure):
    _fields_ = [("n_rows", ctypes.c_int64), ("nnz", ctypes.c_int64), ("n_active", ctypes.c_int64),
                ("n_ghost", ctypes.c_int64), ("n_entities", ctypes.c_int64), ("indptr", _vp), ("indices", _vp),
                ("active", _vp), ("ghost", _vp), ("slots_cells", _vp), ("slots_ghost", _vp), ("slots_boundary", _vp)]


class CPkPatternView(ctypes.Structure):
    _fields_ = [("n_rows", ctypes.c_int64), ("nnz", ctypes.c_int64), ("nd", ctypes.c_int32),
                ("n_active", ctypes.c_int64), ("n_cut", ctypes.c_int64), ("n_ghost", ctypes.c_int64),
                ("n_entities", ctypes.c_int64), ("indptr", _vp), ("indices", _vp), ("active", _vp),
                ("cut_positions", _vp), ("ghost", _vp), ("slots_cells", _vp), ("slots_ghost", _vp),
                ("slots_boundary", _vp)]


class CElasticityPatternView(ctypes.Structure):
    _fields_ = [("n_vertices", ctypes.c_int64), ("nb", ctypes.c_int32), ("n_rows", ctypes.c_int64),
                ("nnz", ctypes.c_int64), ("n_pairs", ctypes.c_int64), ("n_cells", ctypes.c_int64),
                ("n_cut", ctypes.c_int64), ("n_facets_in", ctypes.c_int64), ("n_facets_out", ctypes.c_int64),
                ("n_entities_in", ctypes.c_int64), ("n_entities_out", ctypes.c_int64)] + \
        [(n, _vp) for n in ("vptr", "indptr", "indices", "cut_cells", "facets_in", "facets_out", "pos_cells",
                            "pos_facets_in", "pos_facets_out", "pos_entities_in", "pos_entities_out")]


class CElasticityParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_double) for n in ("lmbda_in", "mu_in", "lmbda_out", "mu_out", "coef_in", "coef_out",
                                               "gamma", "sigma_s")]


_PK_HEAD = [ctypes.POINTER(CMesh), ctypes.POINTER(CPkSpace), ctypes.POINTER(CPkSpace),
            ctypes.POINTER(CQuadrature)]

_SIGNATURES = {
    "phifem_last_error": (ctypes.c_char_p, []),
    "phifem_abi_version": (ctypes.c_int, []),
    "phifem_post_to_host": (ctypes.c_int, [_vp, _vp, ctypes.c_int32, _vp]),
    "phifem_tags_match": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, _vp, _vp, ctypes.c_int64, _vp, _vp]),
    "phifem_cell_points": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, ctypes.c_int32, _vp, _vp]),
    "phifem_tag_cells": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CLevelset),
                                        ctypes.c_int32, _vp, _vp, _vp, _vp, _vp]),
    "phifem_tag_facets": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CLevelset), _vp, _vp,
                                         _vp, _vp, _vp]),
    "phifem_boundary_records": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, _vp]),
    "phifem_tag_facets_phase": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CLevelset), _vp, _vp,
                                               _vp, _vp, ctypes.c_int32, _vp]),
    "phifem_entity_records": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int32,
                                             ctypes.c_uint32, _vp, ctypes.c_int64, _vp, _vp]),
    "phifem_assemble_cells_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, _vp, _vp,
                                                ctypes.c_int64, _vp, ctypes.c_double, _vp, _vp, _vp]),
    "phifem_assemble_boundary_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int64,
                                                   _vp, _vp, _vp]),
    "phifem_assemble_ghost_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int64, _vp,
                                                ctypes.c_double, _vp, _vp]),
    "phifem_assemble_blocked_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_double,
                                                  ctypes.POINTER(CBlockedPlan), _vp, _vp, _vp]),
    "phifem_assemble_rows_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_double,
                                               ctypes.POINTER(CRowsPlan), _vp, _vp, _vp]),
    "phifem_assemble_cells_pk": (ctypes.c_int, _PK_HEAD + [_vp, _vp, _vp, _vp, ctypes.c_int64, _vp,
                                                           ctypes.c_double, _vp, _vp, _vp]),
    "phifem_assemble_boundary_pk": (ctypes.c_int, _PK_HEAD + [_vp, _vp, ctypes.c_int64, _vp, _vp, _vp]),
    "phifem_assemble_ghost_pk": (ctypes.c_int, _PK_HEAD + [_vp, _vp, ctypes.c_int64, _vp, ctypes.c_double,
                                                           _vp, _vp]),
    "phifem_assemble_neumann_cells": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CPkSpace),
                                                     ctypes.POINTER(CQuadrature), _vp, _vp, _vp, _vp, _vp,
                                                     ctypes.c_int64, _vp, ctypes.c_int64, _vp, _vp, ctypes.c_double,
                                                     ctypes.c_double, _vp, _vp, _vp]),
    "phifem_assemble_neumann_boundary": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, ctypes.c_int64, _vp, _vp, _vp]),
    "phifem_assemble_neumann_ghost": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CQuadrature), _vp,
                                                     ctypes.c_int64, _vp, ctypes.c_double, _vp, _vp]),
    "phifem_csr_spmv": (ctypes.c_int, [ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "phifem_csr_row_scan": (ctypes.c_int, [ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "phifem_remap_columns": (ctypes.c_int, [ctypes.c_int64, _vp, _vp, _vp, _vp]),
    "phifem_csr_spmv_rows": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "phifem_bicgstab_iterate": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64] + [_vp] * 16 + [ctypes.POINTER(ctypes.c_int32),
                                                                          ctypes.c_int32, _vp]),
    "phifem_assemble_weak_cells_pk": (ctypes.c_int, _PK_HEAD + [_vp, _vp, _vp, _vp, _vp, ctypes.c_int64, _vp, _vp,
                                                                ctypes.c_double, ctypes.c_double, _vp, _vp, _vp]),
    "phifem_assemble_weak_boundary_pk": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CPkSpace),
                                                        ctypes.POINTER(CQuadrature), _vp, ctypes.c_int64, _vp,
                                                        _vp, _vp]),
    "phifem_assemble_weak_ghost_pk": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CPkSpace),
                                                     ctypes.POINTER(CQuadrature), _vp, ctypes.c_int64, _vp,
                                                     ctypes.c_double, _vp, _vp]),
    "phifem_assemble_elasticity_cells": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CPkSpace),
                                                        ctypes.POINTER(CQuadrature), _vp, _vp, _vp, _vp, ctypes.c_int64,
                                                        _vp, _vp, ctypes.POINTER(CElasticityParams), _vp, _vp, _vp]),
    "phifem_assemble_elasticity_facets": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, ctypes.c_int64, _vp, _vp,
                                                         ctypes.c_int32, ctypes.POINTER(CElasticityParams), _vp, _vp]),
    "phifem_assemble_elasticity_boundary": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, ctypes.c_int64, _vp, _vp,
                                                           ctypes.c_int32, _vp, _vp]),
    "phifem_apply_dirichlet": (ctypes.c_int, [ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "phifem_apply_dirichlet_symmetric": (ctypes.c_int, [ctypes.c_int64, _vp, _vp, _vp, ctypes.c_int64, _vp, _vp, _vp,
                                                        _vp, _vp]),
    "phifem_pattern_create_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, _vp, ctypes.c_int64,
                                                ctypes.POINTER(_vp), _vp]),
    "phifem_pattern_view_of": (ctypes.c_int, [_vp, ctypes.POINTER(CPatternView)]),
    "phifem_integration_entities": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int32, ctypes.c_uint32,
                                                   _vp, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), _vp]),
    "phifem_integration_entities_count": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int32,
                                                         ctypes.c_uint32, _vp, _vp]),
    "phifem_integration_entities_fill": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, ctypes.c_int32,
                                                        ctypes.c_uint32, _vp, ctypes.c_int64, _vp]),
    "phifem_pattern_destroy": (None, [_vp]),
    "phifem_pk_pattern_create": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, ctypes.c_int32, ctypes.c_int64, _vp, _vp,
                                                ctypes.c_uint32, _vp, ctypes.c_int64, ctypes.POINTER(_vp), _vp]),
    "phifem_pk_pattern_view_of": (ctypes.c_int, [_vp, ctypes.POINTER(CPkPatternView)]),
    "phifem_pk_pattern_destroy": (None, [_vp]),
    "phifem_elasticity_pattern_create": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, _vp, ctypes.c_int64, _vp,
                                                        ctypes.c_int64, ctypes.POINTER(_vp), _vp]),
    "phifem_elasticity_pattern_view_of": (ctypes.c_int, [_vp, ctypes.POINTER(CElasticityPatternView)]),
    "phifem_elasticity_pattern_destroy": (None, [_vp]),
    "phifem_surface_static_p1": (ctypes.c_int, [ctypes.POINTER(CMesh), ctypes.POINTER(CRowsPlan), _vp]),
    "phifem_rows_plan_create": (ctypes.c_int, [ctypes.POINTER(CMesh), _vp, _vp, _vp, ctypes.c_int64, _vp,
                                               ctypes.c_int32, ctypes.POINTER(_vp), _vp]),
    "phifem_rows_plan_view": (ctypes.c_int, [_vp, ctypes.POINTER(CRowsPlan), ctypes.POINTER(CRowsPlanInfo)]),
    "phifem_rows_plan_destroy": (None, [_vp]),
    "phifem_peer_flags_create": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(_vp), _vp]),
    "phifem_peer_flags_connect": (ctypes.c_int, [_vp, _vp]),
    "phifem_peer_flags_publish": (ctypes.c_int, [_vp, _vp, _vp]),
    "phifem_peer_flags_collect": (ctypes.c_int, [_vp, _vp, _vp]),
    "phifem_peer_flags_error": (ctypes.c_int, [_vp]),
    "phifem_peer_flags_destroy": (None, [_vp]),
    "phifem_halo_create": (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, ctypes.POINTER(_vp), _vp]),
    "phifem_halo_connect": (ctypes.c_int, [_vp, _vp, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
                                           ctypes.POINTER(ctypes.c_int64), ctypes.c_int64]),
    "phifem_halo_exchange": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "phifem_halo_error": (ctypes.c_int, [_vp]),
    "phifem_halo_destroy": (None, [_vp]),
    "phifem_pattern_release_scratch": (None, []),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """dlopen the C-ABI library (no GPU needed for this step)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "phifem_b200: %s is missing -- build it with `python -m phifem_b200.build`; "
                "there is no CPU fallback for the hot path" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.phifem_abi_version() != 1:
            raise RuntimeError("phifem_b200: ABI version mismatch")
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().phifem_last_error().decode()
        if rc == -3:
            raise NotImplementedError(msg)
        if rc == -1:
            raise ValueError(msg)
        raise RuntimeError("phifem_b200 (%d): %s" % (rc, msg))


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("phifem_b200: expected a CUDA tensor; the hot path has no CPU fallback")
    if not t.is_contiguous():
        raise ValueError("phifem_b200: tensor must be contiguous")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


class _DeviceArray:
    """Zero-copy view of device memory owned by a C handle (`__cuda_array_interface__`)."""

    def __init__(self, pointer, shape, typestr, owner):
        self.owner = owner      # torch keeps THIS object alive for as long as the tensor lives, hence the handle too
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(pointer), False),
                                         "version": 2, "strides": None}


def device_view(pointer, shape, dtype, device, owner=None):
    """torch tensor over `pointer` (no copy).  `owner`: the object whose destruction frees the memory; the tensor keeps
    it alive (a CSRMatrix outlives the plan it came from)."""
    typestr = {torch.int32: "<i4", torch.uint8: "|u1", torch.float64: "<f8", torch.int8: "|i1"}[dtype]
    n = 1
    for k in shape:
        n *= int(k)
    if n == 0 or not pointer:
        return torch.zeros(tuple(shape), dtype=dtype, device=device)
    return torch.as_tensor(_DeviceArray(pointer, shape, typestr, owner), device=device)


def require_cuda(mesh):
    if mesh.device.type != "cuda":
        raise RuntimeError(
            "phifem_b200: the mesh lives on '%s'; cut-cell classification and assembly run on a CUDA "
            "device only (no CPU fallback)" % mesh.device)
    load()


def c_mesh(mesh, with_facets=True, with_records=True):
    require_cuda(mesh)
    lo, hi = mesh.detj_bounds() if mesh.cell_type in _SIMPLICES else (0.0, 0.0)
    owner = scale = None
    if with_facets and with_records and mesh.cell_type in _SIMPLICES:
        owner, scale = mesh.boundary_records()
    return CMesh(CELL_TYPE_ID[mesh.cell_type], mesh.gdim, mesh.num_vertices, mesh.num_cells,
                 mesh.num_facets if with_facets else 0, ptr(mesh.x), ptr(mesh.cells),
                 ptr(mesh.c2f) if with_facets else None, ptr(mesh.f2c) if with_facets else None,
                 lo, hi, ptr(mesh.boundary_facets) if with_facets else None,
                 mesh.boundary_facets.numel() if with_facets else 0,
                 ptr(owner) if owner is not None else None, ptr(scale) if scale is not None else None,
                 # measured on the B200 at config E: cell pass 1.201 -> 1.175 ms on the structured mesh, 1.553 -> 1.584 ms
                 # on the Morton-renumbered unstructured one, for 32 more bytes per vertex: opt-in
                 ptr(mesh.x4) if mesh.cell_type == "tetrahedron" and os.environ.get("PHIFEM_ROWS_X4") == "1" else None)
