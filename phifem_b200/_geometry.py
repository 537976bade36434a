"""Reference-cell data of the hot path: detection points, local facets, coordinate element.

Host-side constants only (a few dozen doubles); they parameterise the CUDA kernels.
Follows reference src/phifem/mesh_scripts.py:28-92 (point generators) and the dolfinx 0.9
reference-cell conventions [dep-knowledge, SURVEY.md Appendix C].
"""
import numpy as np

CELL_TYPES = ("triangle", "quadrilateral", "tetrahedron", "hexahedron")
CELL_TYPE_ID = {name: i for i, name in enumerate(CELL_TYPES)}
TDIM = {"triangle": 2, "quadrilateral": 2, "tetrahedron": 3, "hexahedron": 3}
NVPC = {"triangle": 3, "quadrilateral": 4, "tetrahedron": 4, "hexahedron": 8}
SIMPLICES = ("triangle", "tetrahedron")
# simplex local facet i is opposite local vertex i; quadrilateral and hexahedron facets in tensor order
LOCAL_FACETS = {
    "triangle": ((1, 2), (0, 2), (0, 1)),
    "quadrilateral": ((0, 1), (0, 2), (1, 3), (2, 3)),
    "tetrahedron": ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2)),
    "hexahedron": ((0, 1, 2, 3), (0, 1, 4, 5), (0, 2, 4, 6), (1, 3, 5, 7), (2, 3, 6, 7), (4, 5, 6, 7)),
}
REF_VERTICES = {
    "triangle": np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0]]),
    "quadrilateral": np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]]),
    "tetrahedron": np.array([[0.0, 0, 0], [1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0]]),
    # tensor order: v = i + 2 j + 4 k sits at (i, j, k)
    "hexahedron": np.array([[i, j, k] for k in (0.0, 1.0) for j in (0.0, 1.0) for i in (0.0, 1.0)]),
}
TET_EDGES = ((0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3))
HEX_EDGES = ((0, 1), (0, 2), (0, 4), (1, 3), (1, 5), (2, 3), (2, 6), (3, 7), (4, 5), (4, 6), (5, 7), (6, 7))


def reference_segment_points(N):
    """Reference mesh_scripts.py:28-40."""
    if N > 0:
        return np.linspace(0, 1, N + 1).astype(np.float64)[:, None]
    return np.array([[0.5]])


def reference_triangle_boundary_points(N):
    """Reference mesh_scripts.py:43-65 (order: v0 -> v1 -> v2 -> back towards v0)."""
    if N <= 0:
        return np.array([[1.0 / 3.0, 1.0 / 3.0]])
    t = np.linspace(0, 1, N + 1)
    rows = [np.stack([t, np.zeros_like(t)], axis=1),
            np.stack([1 - t[1:], t[1:]], axis=1)]
    if N > 1:
        rows.append(np.stack([np.zeros_like(t[1:-1]), 1 - t[1:-1]], axis=1))
    return np.concatenate(rows, axis=0).astype(np.float64)


def reference_square_boundary_points(N):
    """Reference mesh_scripts.py:68-92."""
    if N <= 0:
        return np.array([[0.5, 0.5]])
    t = np.linspace(0, 1, N + 1)
    rows = [np.stack([t, np.zeros_like(t)], axis=1),
            np.stack([np.ones_like(t[1:]), t[1:]], axis=1),
            np.stack([1.0 - t[1:], np.ones_like(t[1:])], axis=1)]
    if N > 1:
        rows.append(np.stack([np.zeros_like(t[1:-1]), 1.0 - t[1:-1]], axis=1))
    return np.concatenate(rows, axis=0).astype(np.float64)


def reference_tetrahedron_boundary_points(N):
    """3D extension (the reference stops at 2D, mesh_scripts.py:326-329): order-N lattice points on
    the surface of the reference tetrahedron -- 4 vertices, edge-interior points (edges
    (0,1),(0,2),(0,3),(1,2),(1,3),(2,3) walked low->high), face-interior points of faces 0..3."""
    rv = REF_VERTICES["tetrahedron"]
    if N <= 0:
        return np.array([[0.25, 0.25, 0.25]])
    t = np.linspace(0, 1, N + 1)
    pts = [rv[i] for i in range(4)]
    for a, b in TET_EDGES:
        for s in t[1:-1]:
            pts.append((1 - s) * rv[a] + s * rv[b])
    for face in LOCAL_FACETS["tetrahedron"]:
        a, b, c = (rv[i] for i in face)
        for i in range(1, N):
            for j in range(1, N - i):
                pts.append(a + t[i] * (b - a) + t[j] * (c - a))
    return np.array(pts, dtype=np.float64)


def reference_hexahedron_boundary_points(N):
    """3D extension in the manner of `reference_tetrahedron_boundary_points`: order-N lattice points on the surface
    of the reference cube -- 8 vertices, the N - 1 interior points of each edge (HEX_EDGES order, walked low -> high
    vertex), the (N - 1)^2 interior points of each face (LOCAL_FACETS order, face (a, b, c, d) parametrised by
    v_a + s (v_b - v_a) + t (v_c - v_a), s fastest).  N = 0: the centroid."""
    rv = REF_VERTICES["hexahedron"]
    if N <= 0:
        return np.array([[0.5, 0.5, 0.5]])
    t = np.linspace(0, 1, N + 1)
    pts = [rv[i] for i in range(8)]
    for a, b in HEX_EDGES:
        for s in t[1:-1]:
            pts.append((1 - s) * rv[a] + s * rv[b])
    for face in LOCAL_FACETS["hexahedron"]:
        a, b, c = (rv[i] for i in face[:3])
        for j in range(1, N):
            for i in range(1, N):
                pts.append(a + t[i] * (b - a) + t[j] * (c - a))
    return np.array(pts, dtype=np.float64)


def cell_detection_points(cell_type, N):
    if cell_type == "triangle":
        return reference_triangle_boundary_points(N)
    if cell_type == "quadrilateral":
        return reference_square_boundary_points(N)
    if cell_type == "tetrahedron":
        return reference_tetrahedron_boundary_points(N)
    if cell_type == "hexahedron":
        return reference_hexahedron_boundary_points(N)
    raise NotImplementedError(
        "Mesh tags computation does not support other cell types than 'triangle', "
        "'quadrilateral', 'tetrahedron' or 'hexahedron'")


def facet_detection_points(cell_type, N):
    """Points on the reference facet, mapped onto every local facet -> [nfpc, nq, tdim].  A hexahedron face
    (a, b, c, d) takes the square's points (s, t) at v_a + s (v_b - v_a) + t (v_c - v_a)."""
    if cell_type == "tetrahedron":
        fp = reference_triangle_boundary_points(N)
    elif cell_type == "hexahedron":
        fp = reference_square_boundary_points(N)
    else:
        fp = reference_segment_points(N)
    rv = REF_VERTICES[cell_type]
    out = []
    for lf in LOCAL_FACETS[cell_type]:
        p = np.tile(rv[lf[0]], (len(fp), 1))
        for k in range(1, fp.shape[1] + 1):
            p = p + fp[:, k - 1:k] * (rv[lf[k]] - rv[lf[0]])
        out.append(p)
    return np.array(out)


def coordinate_basis(cell_type, pts):
    """P1 / Q1 (bilinear, trilinear) coordinate-element values at reference points -> [npts, nvpc]."""
    pts = np.asarray(pts, dtype=np.float64)
    if cell_type == "quadrilateral":
        X, Y = pts[:, 0], pts[:, 1]
        return np.stack([(1 - X) * (1 - Y), X * (1 - Y), (1 - X) * Y, X * Y], axis=1)
    if cell_type == "hexahedron":
        f = [(1 - pts[:, d], pts[:, d]) for d in range(3)]
        return np.stack([f[0][v & 1] * f[1][(v >> 1) & 1] * f[2][v >> 2] for v in range(8)], axis=1)
    return np.concatenate([(1 - pts.sum(axis=1))[:, None], pts], axis=1)


def coordinate_basis_grad(cell_type, pts):
    """Reference gradients [npts, nvpc, tdim] of the coordinate element."""
    pts = np.asarray(pts, dtype=np.float64)
    if cell_type == "quadrilateral":
        X, Y = pts[:, 0], pts[:, 1]
        dX = np.stack([-(1 - Y), (1 - Y), -Y, Y], axis=1)
        dY = np.stack([-(1 - X), -X, (1 - X), X], axis=1)
        return np.stack([dX, dY], axis=2)
    if cell_type == "hexahedron":
        f = [(1 - pts[:, d], pts[:, d]) for d in range(3)]
        df = [(-np.ones(len(pts)), np.ones(len(pts)))] * 3
        g = np.empty((len(pts), 8, 3))
        for v in range(8):
            b = (v & 1, (v >> 1) & 1, v >> 2)
            g[:, v, 0] = df[0][b[0]] * f[1][b[1]] * f[2][b[2]]
            g[:, v, 1] = f[0][b[0]] * df[1][b[1]] * f[2][b[2]]
            g[:, v, 2] = f[0][b[0]] * f[1][b[1]] * df[2][b[2]]
        return g
    tdim = TDIM[cell_type]
    g = np.zeros((len(pts), tdim + 1, tdim))
    g[:, 0, :] = -1.0
    for d in range(tdim):
        g[:, d + 1, d] = 1.0
    return g
