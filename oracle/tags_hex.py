"""CPU oracle, hexahedra: level-set cut-cell classification (TEST INFRASTRUCTURE ONLY).

The hexahedral counterpart of `oracle.tags`, restated with numpy and independent of `phifem_b200`.  Hexahedra are OUR
extension, like tetrahedra (the reference stops at 2D, mesh_scripts.py:326-329).  Conventions follow dolfinx / basix
[dep-knowledge]:

  vertices in tensor order    v = i + 2 j + 4 k sits at (i, j, k) of the reference cube
  local facets (tensor order) (0,1,2,3) (0,1,4,5) (0,2,4,6) (1,3,5,7) (2,3,6,7) (4,5,6,7)
  local edges                 (0,1) (0,2) (0,4) (1,3) (1,5) (2,3) (2,6) (3,7) (4,5) (4,6) (5,7) (6,7)

Detection rule (defined here, DESIGN.md section 2):
  * cell points of order N: the 8 vertices, the N - 1 interior points of each edge (edge order, walked from the lower
    to the higher local vertex), the (N - 1)^2 interior points of each face (facet order, face (a, b, c, d) at
    v_a + s (v_b - v_a) + t (v_c - v_a), s fastest); N = 0: the centroid;
  * facet points: the square's boundary points (s, t) of `oracle.tags.square_boundary_points`, on every face by the same
    map;
  * scales: |det J| of the trilinear map at every cell point; |dx/ds x dx/dt| at every facet point.  The faces of a
    perturbed hexahedron are not planar, so the facet scale has shape [Nc, nfpc, nq] (a quadrilateral's is one edge
    length per facet).

The tagging algebra is `oracle.tags` unchanged: the ds detection there multiplies phi_q by one scale per facet, so the
facet values are handed over premultiplied, phi_q * s_q, with a unit scale (x * 1.0 == x exactly).  Every sum is
sequential, left to right, without FMA contraction, like `oracle.tags`.
"""
import numpy as np

from oracle import tags as OT

LOCAL_FACETS = ((0, 1, 2, 3), (0, 1, 4, 5), (0, 2, 4, 6), (1, 3, 5, 7), (2, 3, 6, 7), (4, 5, 6, 7))
EDGES = ((0, 1), (0, 2), (0, 4), (1, 3), (1, 5), (2, 3), (2, 6), (3, 7), (4, 5), (4, 6), (5, 7), (6, 7))
REF_VERTICES = np.array([[i, j, k] for k in (0.0, 1.0) for j in (0.0, 1.0) for i in (0.0, 1.0)])


def boundary_points(N):
    """Cell detection points of order N: 8 + 12 (N - 1) + 6 (N - 1)^2 points on the surface of the cube."""
    if N <= 0:
        return np.array([[0.5, 0.5, 0.5]])
    t = np.linspace(0, 1, N + 1)
    rv = REF_VERTICES
    pts = [tuple(v) for v in rv]
    for a, b in EDGES:
        for ti in t[1:-1]:
            pts.append(tuple((1 - ti) * rv[a] + ti * rv[b]))
    for face in LOCAL_FACETS:
        a, b, c = (rv[i] for i in face[:3])
        for j in range(1, N):
            for i in range(1, N):
                pts.append(tuple(a + t[i] * (b - a) + t[j] * (c - a)))
    return np.array(pts, dtype=np.float64)


def facet_points_in_cell(N):
    """[6, nq, 3]: the square's detection points (s, t) at v_a + s (v_b - v_a) + t (v_c - v_a) on every face."""
    st = OT.square_boundary_points(N)
    out = []
    for face in LOCAL_FACETS:
        a, b, c = (REF_VERTICES[i] for i in face[:3])
        out.append(a + st[:, 0:1] * (b - a) + st[:, 1:2] * (c - a))
    return np.array(out)


def face_axes(lf):
    """Reference axes of v_b - v_a and v_c - v_a of local face lf (the directions of s and t)."""
    a, b, c = LOCAL_FACETS[lf][:3]
    return int(np.log2(b - a)), int(np.log2(c - a))


def coordinate_basis(pts):
    """Trilinear coordinate element: values [npts, 8] and reference gradients [npts, 8, 3]."""
    pts = np.asarray(pts, dtype=np.float64)
    n = len(pts)
    val = np.empty((n, 8))
    grad = np.empty((n, 8, 3))
    for v in range(8):
        f = [pts[:, d] if (v >> d) & 1 else 1 - pts[:, d] for d in range(3)]
        df = [np.ones(n) if (v >> d) & 1 else -np.ones(n) for d in range(3)]
        val[:, v] = f[0] * f[1] * f[2]
        grad[:, v, 0] = df[0] * f[1] * f[2]
        grad[:, v, 1] = f[0] * df[1] * f[2]
        grad[:, v, 2] = f[0] * f[1] * df[2]
    return val, grad


def physical_points(x, cells, ref_pts):
    """x_q = sum_v N_v(xi_q) x_v -> [Nc, npts, 3]."""
    val, _ = coordinate_basis(ref_pts)
    xc = x[cells]
    out = np.empty((len(cells), len(ref_pts), 3))
    for q in range(len(ref_pts)):
        for d in range(3):
            out[:, q, d] = OT._seq_dot(val[q], xc[:, :, d])
    return out


def _jacobian_column(grad_q, xc, ax):
    """d x / d X_ax at one point -> [Nc, 3]."""
    return np.stack([OT._seq_dot(grad_q[:, ax], xc[:, :, d]) for d in range(3)], axis=1)


def _det3(a, b, c):
    """det [a b c] by cofactors, the operation order of `oracle.tags.cell_scale` for tetrahedra."""
    return (a[:, 0] * (b[:, 1] * c[:, 2] - c[:, 1] * b[:, 2])
            - b[:, 0] * (a[:, 1] * c[:, 2] - c[:, 1] * a[:, 2])
            + c[:, 0] * (a[:, 1] * b[:, 2] - b[:, 1] * a[:, 2]))


def cell_scale(x, cells, ref_pts):
    """|det J| of the trilinear map at every detection point -> [Nc, npts]."""
    _, grad = coordinate_basis(ref_pts)
    xc = x[cells]
    out = np.empty((len(cells), len(ref_pts)))
    for q in range(len(ref_pts)):
        a, b, c = (_jacobian_column(grad[q], xc, ax) for ax in range(3))
        out[:, q] = np.abs(_det3(a, b, c))
    return out


def _cross(e1, e2):
    return (e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1],
            e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2],
            e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0])


def facet_scale(x, cells, fpts):
    """|dx/ds x dx/dt| at every facet detection point -> [Nc, 6, nq] (fpts = `facet_points_in_cell`)."""
    xc = x[cells]
    nq = fpts.shape[1]
    out = np.empty((len(cells), len(LOCAL_FACETS), nq))
    for lf in range(len(LOCAL_FACETS)):
        sa, ta = face_axes(lf)
        _, grad = coordinate_basis(fpts[lf])
        for q in range(nq):
            cx, cy, cz = _cross(_jacobian_column(grad[q], xc, sa), _jacobian_column(grad[q], xc, ta))
            out[:, lf, q] = np.sqrt(cx * cx + cy * cy + cz * cz)
    return out


def point_values_expression(func, x, cells, ref_pts):
    """phi at the physical images of reference points [..., npts, 3] -> [Nc, ..., npts]."""
    ref_pts = np.asarray(ref_pts)
    lead = ref_pts.shape[:-1]
    xq = physical_points(x, cells, ref_pts.reshape(-1, 3))
    with np.errstate(all="ignore"):
        vals = func(xq.reshape(-1, 3).T)
    return np.asarray(vals, dtype=np.float64).reshape((len(cells),) + lead)


def build_topology(cells):
    """c2f [Nc, 6], f2c [Nf, 2] (ascending cells, -1 pad), facet_vertices [Nf, 4]: faces numbered by the lexicographic
    rank of their sorted vertex 4-tuple."""
    cells = np.asarray(cells, dtype=np.int64)
    nc, nfl = len(cells), len(LOCAL_FACETS)
    keys = np.sort(np.stack([cells[:, list(lf)] for lf in LOCAL_FACETS], axis=1), axis=2)
    uniq, inv = np.unique(keys.reshape(nc * nfl, 4), axis=0, return_inverse=True)
    c2f = inv.reshape(nc, nfl).astype(np.int32)
    f2c = -np.ones((len(uniq), 2), dtype=np.int32)
    owner = np.repeat(np.arange(nc, dtype=np.int32), nfl)
    order = np.argsort(c2f.ravel(), kind="stable")
    fs, cs = c2f.ravel()[order], owner[order]
    first = np.r_[True, fs[1:] != fs[:-1]]
    f2c[fs[first], 0] = cs[first]
    f2c[fs[~first], 1] = cs[~first]
    return c2f, f2c, uniq.astype(np.int32)


def compute_tags_measures(x, cells, phi_cell, phi_facet, N, box_mode=False, single_layer_cut=False, warn=False):
    """mesh_scripts.py:571-653 on a hexahedral mesh.  phi_cell [Nc, npts] at `boundary_points(N)`, phi_facet
    [Nc, 6, nq] at `facet_points_in_cell(N)`.  Returns the dict of `oracle.tags.compute_tags_measures`, plus the
    counts of the tag kernels' counter block ("counts")."""
    c2f, f2c, fverts = build_topology(cells)
    scale = cell_scale(x, cells, boundary_points(N))
    fscale = facet_scale(x, cells, facet_points_in_cell(N))
    ct = OT.tag_cells(phi_cell, scale, cells, single_layer_cut, warn)
    with np.errstate(all="ignore"):
        weighted = phi_facet * fscale
    ft, dup, kcell = OT.tag_facets(ct, c2f, f2c, weighted, np.ones(c2f.shape), warn)
    counts = {"interior": int((ct == 1).sum()), "cut": int((ct == 2).sum()), "exterior": int((ct == 3).sum()),
              "untagged": int((ct == 0).sum()), "facet_conflicts": len(dup),
              "boundary_owners": len(np.unique(f2c[f2c[:, 1] < 0, 0]))}
    out = {"c2f": c2f, "f2c": f2c, "facet_vertices": fverts, "duplicates": dup, "counts": counts,
           "parent_cell_tags": ct, "parent_facet_tags": ft}
    if box_mode:
        out["cell_tags"], out["facet_tags"] = ct, ft
        out["ds100"] = OT.integration_entities(c2f, f2c, (ct == 1) | (ct == 2), ft == 4)
        out["ds101"] = OT.integration_entities(c2f, f2c, (ct == 2) | (ct == 3), ft == 3)
    else:
        keep = np.nonzero((ct == 1) | (ct == 2))[0]
        sx, scells, v_map = OT.submesh(x, cells, keep)
        sc2f, _, _ = build_topology(scells)
        out.update(cell_tags=ct[keep], facet_tags=OT.transfer_facet_tags(ft, c2f, sc2f, keep),
                   sub_x=sx, sub_cells=scells, c_map=keep.astype(np.int32), v_map=v_map)
    return out


def outward_normals(x, cells, entities):
    """Outward unit normal and area of each (cell, local_facet) entity whose face is planar -> ([m, 3], [m]): the
    normal of (v_b - v_a) x (v_c - v_a), the area of the parallelogram they span, the sign from the cell centroid."""
    ents = np.asarray(entities).reshape(-1, 2)
    xc = x[cells[ents[:, 0]]]
    n = np.zeros((len(ents), 3))
    area = np.zeros(len(ents))
    for i, (c, lf) in enumerate(ents):
        p = xc[i][list(LOCAL_FACETS[lf])]
        nn = np.cross(p[1] - p[0], p[2] - p[0])
        area[i] = np.linalg.norm(nn)
        nn = nn / area[i]
        if np.dot(nn, p.mean(axis=0) - xc[i].mean(axis=0)) < 0:
            nn = -nn
        n[i] = nn
    return n, area
