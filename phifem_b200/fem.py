"""Caller-side finite-element helpers: Lagrange function spaces and functions.

The reference takes its level set as a `dolfinx.fem.Function` (reference
src/phifem/mesh_scripts.py:571-577, tests/test_compute_meshtags.py:153-158).  dolfinx and
basix are not part of this framework, so this module is the stand-in the drop-in API
accepts: `functionspace(mesh, ("Lagrange", k))`, `Function(V)`, `Function.interpolate(f)`,
`Function.x.array`.  It is host-side numpy bookkeeping (dof numbering, node sets,
tabulation of the basis at the detection points); the hot path consumes its arrays on the
GPU.

Element definition (matches basix 0.9 defaults [dep-knowledge, SURVEY.md A.2/C.7]):
Lagrange with GLL-warped nodes (differs from equispaced from degree 3), cell-local dof order
= vertices, then edges in dolfinx local edge order, then faces, then interior.  Global dof
numbering is ours (vertices, then edges, faces, cells); the hot path takes the dofmap as an
input array, so any numbering works (SURVEY.md C.5).
"""
import itertools
import math

import numpy as np

from .mesh import Mesh

_GLL = {
    1: np.array([0.0, 1.0]),
    2: np.array([0.0, 0.5, 1.0]),
    3: np.array([0.0, (1.0 - 1.0 / math.sqrt(5.0)) / 2.0, (1.0 + 1.0 / math.sqrt(5.0)) / 2.0, 1.0]),
}

# dolfinx local edge order [dep-knowledge, SURVEY.md C.7]
LOCAL_EDGES = {
    "triangle": ((1, 2), (0, 2), (0, 1)),
    "quadrilateral": ((0, 1), (0, 2), (1, 3), (2, 3)),
    "tetrahedron": ((2, 3), (1, 3), (1, 2), (0, 3), (0, 2), (0, 1)),
    "hexahedron": ((0, 1), (0, 2), (0, 4), (1, 3), (1, 5), (2, 3), (2, 6), (3, 7), (4, 5), (4, 6), (5, 7), (6, 7)),
}
LOCAL_FACES = {"tetrahedron": ((1, 2, 3), (0, 2, 3), (0, 1, 3), (0, 1, 2)),
               "hexahedron": ((0, 1, 2, 3), (0, 1, 4, 5), (0, 2, 4, 6), (1, 3, 5, 7), (2, 3, 6, 7), (4, 5, 6, 7))}
REF_VERTICES = {
    "triangle": np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0]]),
    "quadrilateral": np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]]),
    "tetrahedron": np.array([[0.0, 0, 0], [1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0]]),
    "hexahedron": np.array([[i, j, k] for k in (0.0, 1.0) for j in (0.0, 1.0) for i in (0.0, 1.0)]),
}


def _monomial_exponents(cell_type, k):
    if cell_type == "quadrilateral":
        return [(i, j) for i in range(k + 1) for j in range(k + 1)]
    if cell_type == "hexahedron":
        return list(itertools.product(range(k + 1), repeat=3))
    tdim = 2 if cell_type == "triangle" else 3
    return [e for e in itertools.product(range(k + 1), repeat=tdim) if sum(e) <= k]


def _monomials(exps, pts):
    pts = np.asarray(pts, dtype=np.float64)
    out = np.ones((len(pts), len(exps)))
    for m, e in enumerate(exps):
        for d, p in enumerate(e):
            if p:
                out[:, m] *= pts[:, d] ** p
    return out


class LagrangeElement:
    """Reference Lagrange element of degree 1..3 on triangle / quadrilateral / tetrahedron, 1..2 on hexahedron
    (Q2 nodes: vertices, edge midpoints, face centres, centre)."""

    def __init__(self, cell_type, degree):
        if cell_type not in REF_VERTICES:
            raise NotImplementedError(cell_type)
        if degree not in (1, 2, 3):
            raise NotImplementedError("Lagrange degree %d" % degree)
        if cell_type == "hexahedron" and degree == 3:
            raise NotImplementedError("Lagrange degree 3 on hexahedra")
        self.cell_type, self.degree = cell_type, degree
        rv = REF_VERTICES[cell_type]
        k = degree
        inner = _GLL[k][1:-1]
        nodes = [v for v in rv]
        # entity bookkeeping: list of (kind, local entity, position)
        ents = [("v", i, 0) for i in range(len(rv))]
        for e, (a, b) in enumerate(LOCAL_EDGES[cell_type]):
            for j, s in enumerate(inner):
                nodes.append((1 - s) * rv[a] + s * rv[b])
                ents.append(("e", e, j))
        if (cell_type == "tetrahedron" and k == 3) or (cell_type == "hexahedron" and k == 2):
            for f, face in enumerate(LOCAL_FACES[cell_type]):
                nodes.append(rv[list(face)].mean(axis=0))
                ents.append(("f", f, 0))
        if cell_type == "triangle" and k == 3:
            nodes.append(rv.mean(axis=0))
            ents.append(("c", 0, 0))
        if cell_type == "quadrilateral":
            for j, (sy, sx) in enumerate(itertools.product(inner, inner)):
                nodes.append(np.array([sx, sy]))
                ents.append(("c", 0, j))
        if cell_type == "hexahedron" and k == 2:
            nodes.append(rv.mean(axis=0))
            ents.append(("c", 0, 0))
        self.nodes = np.array(nodes)
        self.entities = ents
        self.exps = _monomial_exponents(cell_type, k)
        assert len(self.exps) == len(self.nodes)
        self.coef = np.linalg.inv(_monomials(self.exps, self.nodes))  # [monomial, basis]
        self.ndofs = len(self.nodes)

    def tabulate(self, pts, snap=True):
        """Basis values [..., npts, ndofs] at reference points [..., npts, tdim]; entries within
        1e-9 of 0 / +-1 are snapped like FFCx does with its tables [dep-knowledge]."""
        pts = np.asarray(pts, dtype=np.float64)
        lead = pts.shape[:-1]
        tab = _monomials(self.exps, pts.reshape(-1, pts.shape[-1])) @ self.coef
        if snap:
            for target in (0.0, 1.0, -1.0):
                tab[np.abs(tab - target) < 1e-9] = target
        return tab.reshape(lead + (self.ndofs,))


def _unique_rows(keys):
    uniq, inv = np.unique(keys, axis=0, return_inverse=True)
    return uniq, inv.reshape(-1)


def simplex_dofmap_device(mesh, degree):
    """Dofmap [Nc, nd] (int32, on the mesh's device) and dof count of P1 / P2 Lagrange on triangles /
    tetrahedra, built with torch sort/unique where the mesh lives.  Same numbering as the host builder in
    `FunctionSpace`: vertex dofs = vertex ids, then one dof per edge, edges numbered by the lexicographic
    rank of their sorted vertex pair, cell-local edge order = LOCAL_EDGES."""
    import torch
    if degree == 1:
        return mesh.cells, mesh.num_vertices
    assert degree == 2 and mesh.cell_type in ("triangle", "tetrahedron")
    nv = mesh.num_vertices
    c = mesh.cells.long()
    edges = LOCAL_EDGES[mesh.cell_type]
    a = torch.stack([c[:, e[0]] for e in edges], dim=1)
    b = torch.stack([c[:, e[1]] for e in edges], dim=1)
    key = torch.minimum(a, b) * nv + torch.maximum(a, b)
    del a, b
    uniq, inv = torch.unique(key.reshape(-1), sorted=True, return_inverse=True)
    n_edges = int(uniq.numel())
    del uniq, key
    dm = torch.cat([c, nv + inv.reshape(c.shape[0], len(edges))], dim=1).to(torch.int32).contiguous()
    return dm, nv + n_edges


class FunctionSpace:
    def __init__(self, mesh, degree):
        self.mesh = mesh
        self.element = LagrangeElement(mesh.cell_type, degree)
        self.degree = degree
        self._dofmap_dev = None
        if degree <= 2 and mesh.cell_type in ("triangle", "tetrahedron"):
            # large meshes: sort/unique on the device, host copy made on first use
            self._dofmap_dev, self.num_dofs = simplex_dofmap_device(mesh, degree)
            self._dofmap = None
            return
        cells = mesh.cells_host.astype(np.int64)
        nc = len(cells)
        nv = mesh.num_vertices
        k = degree
        cols = [cells]
        offset = nv
        if k > 1:
            edges = LOCAL_EDGES[mesh.cell_type]
            pairs = np.stack([cells[:, list(e)] for e in edges], axis=1)      # [Nc, ne, 2]
            flip = pairs[:, :, 0] > pairs[:, :, 1]
            _, inv = _unique_rows(np.sort(pairs, axis=2).reshape(-1, 2))
            eid = inv.reshape(nc, len(edges))
            n_edges = int(eid.max()) + 1
            for e in range(len(edges)):
                for j in range(k - 1):
                    pos = np.where(flip[:, e], k - 2 - j, j)
                    cols.append((offset + eid[:, e] * (k - 1) + pos)[:, None])
            offset += n_edges * (k - 1)
        kinds = [ent[0] for ent in self.element.entities]
        if "f" in kinds:
            # one dof per face, faces numbered by the lexicographic rank of their sorted vertex tuple
            faces = LOCAL_FACES[mesh.cell_type]
            tup = np.sort(np.stack([cells[:, list(f)] for f in faces], axis=1), axis=2)
            _, inv = _unique_rows(tup.reshape(-1, len(faces[0])))
            fid = inv.reshape(nc, len(faces))
            for f in range(len(faces)):
                cols.append((offset + fid[:, f])[:, None])
            offset += int(fid.max()) + 1
        n_int = kinds.count("c")
        if n_int:
            base = offset + np.arange(nc)[:, None] * n_int
            cols.append(base + np.arange(n_int)[None, :])
            offset += nc * n_int
        self._dofmap = np.ascontiguousarray(np.concatenate(cols, axis=1).astype(np.int32))
        self.num_dofs = int(offset)
        assert self._dofmap.shape[1] == self.element.ndofs

    @property
    def dofmap(self):
        """Host dofmap [Nc, nd] int32."""
        if self._dofmap is None:
            self._dofmap = np.ascontiguousarray(self._dofmap_dev.cpu().numpy())
        return self._dofmap

    @property
    def dofmap_dev(self):
        """Dofmap on the mesh's device (int32 [Nc, nd])."""
        if self._dofmap_dev is None:
            import torch
            self._dofmap_dev = torch.from_numpy(self._dofmap).to(self.mesh.device).contiguous()
        return self._dofmap_dev

    def dof_coordinates_dev(self):
        """Dof coordinates [num_dofs, gdim] on the mesh's device (P1 / P2 on simplices): vertices, then edge
        midpoints -- what `tabulate_dof_coordinates` returns on the host."""
        import torch
        if self.degree > 2 or self.mesh.cell_type not in ("triangle", "tetrahedron"):
            return torch.from_numpy(self.tabulate_dof_coordinates()).to(self.mesh.device)
        mesh = self.mesh
        if self.degree == 1:
            return mesh.x
        out = torch.empty((self.num_dofs, mesh.gdim), dtype=torch.float64, device=mesh.device)
        out[:mesh.num_vertices] = mesh.x
        nvpc = mesh.cells.shape[1]
        dm = self.dofmap_dev.long()
        for e, (a, b) in enumerate(LOCAL_EDGES[mesh.cell_type]):
            out[dm[:, nvpc + e]] = 0.5 * mesh.x[dm[:, a]] + 0.5 * mesh.x[dm[:, b]]
        return out

    def tabulate_dof_coordinates(self):
        """Physical coordinates of the dofs [num_dofs, gdim] (affine / bilinear push-forward of the
        reference nodes, accumulated vertex by vertex)."""
        from . import _geometry
        mesh = self.mesh
        shape = _geometry.coordinate_basis(mesh.cell_type, self.element.nodes)  # [nd, nvpc]
        xc = mesh.x_host[mesh.cells_host]                                        # [Nc, nvpc, gdim]
        out = np.zeros((self.num_dofs, mesh.gdim))
        for i in range(self.element.ndofs):
            acc = None
            for v in range(xc.shape[1]):
                w = shape[i, v]
                if w == 0.0:
                    continue
                term = xc[:, v, :] if w == 1.0 else w * xc[:, v, :]
                acc = term if acc is None else acc + term
            out[self.dofmap[:, i]] = acc
        return out


class _Vector:
    def __init__(self, n, array=None):
        self.array = np.zeros(n, dtype=np.float64) if array is None else array


class Function:
    """A finite-element function: `function_space`, `x.array` (dof values).  `values` may be a numpy
    array (copied) or a torch tensor on any device (kept as is: device-resident coefficients)."""

    def __init__(self, V, values=None):
        self.function_space = V
        if values is not None and not isinstance(values, np.ndarray) and hasattr(values, "device"):
            if values.numel() != V.num_dofs:
                raise ValueError("expected %d dof values" % V.num_dofs)
            self.x = _Vector(V.num_dofs, values)
            return
        self.x = _Vector(V.num_dofs)
        if values is not None:
            self.x.array[:] = values

    def interpolate(self, f):
        """f receives coordinates as an array of shape (3, npoints), like dolfinx."""
        X = self.function_space.tabulate_dof_coordinates()
        x3 = np.zeros((3, len(X)))
        x3[:X.shape[1]] = X.T
        with np.errstate(all="ignore"):
            self.x.array[:] = np.asarray(f(x3), dtype=np.float64)
        return self


class P1Space:
    """P1 space with vertex dofs and dofmap == mesh.cells, without any host-side copies (what the
    large configurations use; `functionspace(mesh, 1)` builds the same numbering)."""

    def __init__(self, mesh):
        self.mesh, self.degree = mesh, 1
        self.element = LagrangeElement(mesh.cell_type, 1)
        self.num_dofs = mesh.num_vertices

    @property
    def dofmap(self):
        return self.mesh.cells_host


def functionspace_p1_device(mesh: Mesh):
    return P1Space(mesh)


def functionspace(mesh: Mesh, element):
    """`element` = ("Lagrange", degree) or an int degree."""
    degree = element[1] if isinstance(element, (tuple, list)) else int(element)
    return FunctionSpace(mesh, degree)
