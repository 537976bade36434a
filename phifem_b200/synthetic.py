"""Synthetic meshes and level sets of the benchmark configurations (SURVEY.md section 8d).

S-2D(n): n x n squares split by the "right" diagonal -> 2 n^2 triangles (what
`dolfinx.mesh.create_rectangle` gives the reference demos,
demo/strong-dirichlet/flower/main.py:48-49).  Q-2D(n): the same n x n squares as quadrilaterals (the cell type of
demo/neumann/square).  S-3D(n): n^3 cubes x 6 Kuhn tetrahedra; H-3D(n): the same n^3 cubes as hexahedra.
Vertices are numbered lexicographically; generated directly on the target device.
"""
import itertools
import math

import numpy as np
import torch

from .mesh import Mesh, default_device


def _grid_vertices(lo, hi, n, device):
    axes = [torch.linspace(float(a), float(b), n + 1, dtype=torch.float64, device=device)
            for a, b in zip(lo, hi)]
    grids = torch.meshgrid(*axes, indexing="ij")
    return torch.stack([g.reshape(-1) for g in grids], dim=1).contiguous()


def rectangle_mesh(n, lo=(-1.0, -1.0), hi=(1.0, 1.0), device=None):
    """2 n^2 triangles; vertex id = i*(n+1)+j for the point (x_i, y_j)."""
    device = torch.device(device) if device is not None else default_device()
    x = _grid_vertices(lo, hi, n, device)
    i = torch.arange(n, device=device, dtype=torch.int64)
    I, J = torch.meshgrid(i, i, indexing="ij")
    v00 = (I * (n + 1) + J).reshape(-1)
    v10, v01, v11 = v00 + (n + 1), v00 + 1, v00 + (n + 1) + 1
    t0 = torch.stack([v00, v10, v11], dim=1)
    t1 = torch.stack([v00, v01, v11], dim=1)
    cells = torch.stack([t0, t1], dim=1).reshape(-1, 3).to(torch.int32)
    return Mesh(x, cells, "triangle", device)


def quadrilateral_mesh(n, lo=(-1.0, -1.0), hi=(1.0, 1.0), device=None):
    """n^2 quadrilaterals in dolfinx tensor order (v0 = (x_i, y_j), v1 = (x_i+1, y_j), v2 = (x_i, y_j+1),
    v3 = (x_i+1, y_j+1)); vertex id = i*(n+1)+j for the point (x_i, y_j), as in `rectangle_mesh`."""
    device = torch.device(device) if device is not None else default_device()
    x = _grid_vertices(lo, hi, n, device)
    i = torch.arange(n, device=device, dtype=torch.int64)
    I, J = torch.meshgrid(i, i, indexing="ij")
    v00 = (I * (n + 1) + J).reshape(-1)
    cells = torch.stack([v00, v00 + (n + 1), v00 + 1, v00 + (n + 1) + 1], dim=1).to(torch.int32).contiguous()
    return Mesh(x, cells, "quadrilateral", device)


def box_mesh(n, lo=(0.0, 0.0, 0.0), hi=(1.0, 1.0, 1.0), device=None):
    """6 nx ny nz Kuhn tetrahedra (n = int or (nx, ny, nz)): each cube is split along the 6 monotone
    edge paths from its low corner to its high corner; vertex id = (i*(ny+1)+j)*(nz+1)+k; the 6
    tetrahedra of a cube are consecutive and cubes are ordered x-major."""
    device = torch.device(device) if device is not None else default_device()
    nx, ny, nz = (n, n, n) if isinstance(n, int) else n
    axes = [torch.linspace(float(a), float(b), m + 1, dtype=torch.float64, device=device)
            for a, b, m in zip(lo, hi, (nx, ny, nz))]
    grids = torch.meshgrid(*axes, indexing="ij")
    x = torch.stack([g.reshape(-1) for g in grids], dim=1).contiguous()
    I, J, K = torch.meshgrid(*[torch.arange(m, device=device, dtype=torch.int64) for m in (nx, ny, nz)],
                             indexing="ij")
    base = ((I * (ny + 1) + J) * (nz + 1) + K).reshape(-1)
    stride = [(ny + 1) * (nz + 1), nz + 1, 1]
    tets = []
    for perm in itertools.permutations(range(3)):
        offs, acc = [0], 0
        for a in perm:
            acc += stride[a]
            offs.append(acc)
        tets.append(base[:, None] + torch.tensor(offs, device=device, dtype=torch.int64)[None, :])
    cells = torch.stack(tets, dim=1).reshape(-1, 4).to(torch.int32)
    return Mesh(x, cells, "tetrahedron", device)


def hexahedron_mesh(n, lo=(0.0, 0.0, 0.0), hi=(1.0, 1.0, 1.0), device=None):
    """nx ny nz hexahedra (n = int or (nx, ny, nz)) in dolfinx tensor order (v0 = (x_i, y_j, z_k), v1 = +x, v2 = +y,
    v3 = +x+y, v4..v7 the same at z_k+1); the vertices and vertex ids of `box_mesh`, cubes ordered x-major, so that
    the two meshes can be compared cube by cube."""
    device = torch.device(device) if device is not None else default_device()
    nx, ny, nz = (n, n, n) if isinstance(n, int) else n
    axes = [torch.linspace(float(a), float(b), m + 1, dtype=torch.float64, device=device)
            for a, b, m in zip(lo, hi, (nx, ny, nz))]
    grids = torch.meshgrid(*axes, indexing="ij")
    x = torch.stack([g.reshape(-1) for g in grids], dim=1).contiguous()
    I, J, K = torch.meshgrid(*[torch.arange(m, device=device, dtype=torch.int64) for m in (nx, ny, nz)],
                             indexing="ij")
    base = ((I * (ny + 1) + J) * (nz + 1) + K).reshape(-1)
    sx, sy, sz = (ny + 1) * (nz + 1), nz + 1, 1
    offs = torch.tensor([i * sx + j * sy + k * sz for k in (0, 1) for j in (0, 1) for i in (0, 1)],
                        device=device, dtype=torch.int64)
    cells = (base[:, None] + offs[None, :]).to(torch.int32).contiguous()
    return Mesh(x, cells, "hexahedron", device)


def unstructured_variant(mesh, jitter=0.2, seed=0):
    """Interior-vertex jitter (uniform in +-jitter*h), random cell permutation and random vertex
    relabelling: the "unstructured" stress variant of SURVEY.md section 8d."""
    rng = np.random.default_rng(seed)
    x = mesh.x.cpu().numpy().copy()
    cells = mesh.cells.cpu().numpy().astype(np.int64)
    lo, hi = x.min(axis=0), x.max(axis=0)
    nv = len(x)
    n = round(nv ** (1.0 / x.shape[1])) - 1
    h = (hi - lo) / n
    interior = np.all((x > lo + 1e-12) & (x < hi - 1e-12), axis=1)
    x[interior] += rng.uniform(-jitter, jitter, size=(int(interior.sum()), x.shape[1])) * h
    cells = cells[rng.permutation(len(cells))]
    relabel = rng.permutation(nv)
    xn = np.empty_like(x)
    xn[relabel] = x
    return Mesh(xn, relabel[cells].astype(np.int32), mesh.cell_type, mesh.device)


def unstructured_variant_device(mesh, jitter=0.2, seed=0):
    """`unstructured_variant` with torch generators on the mesh's device (the 50 M-cell benchmark mesh is never copied
    to the host): jitter from seed, cell permutation from seed + 1, vertex relabelling from seed + 2 (SURVEY.md 8d)."""
    dev = mesh.device
    gens = [torch.Generator(device=dev).manual_seed(seed + k) for k in range(3)]
    x = mesh.x.clone()
    lo, hi = x.min(dim=0).values, x.max(dim=0).values
    nv = mesh.num_vertices
    n = round(nv ** (1.0 / x.shape[1])) - 1
    h = (hi - lo) / n
    interior = ((x > lo + 1e-12) & (x < hi - 1e-12)).all(dim=1)
    u = torch.rand(x.shape, generator=gens[0], device=dev, dtype=torch.float64) * 2.0 - 1.0
    x += torch.where(interior[:, None], u * (jitter * h), torch.zeros_like(u))
    del u
    cperm = torch.randperm(mesh.num_cells, generator=gens[1], device=dev)
    relabel = torch.randperm(nv, generator=gens[2], device=dev)
    xn = torch.empty_like(x)
    xn[relabel] = x
    cells = relabel[mesh.cells[cperm].long()].to(torch.int32)
    return Mesh(xn, cells, mesh.cell_type, dev)


SPHERE_CENTER = (0.5 + math.pi / 1000.0, 0.5 + math.e / 1000.0, 0.5 + math.sqrt(2.0) / 1000.0)
SPHERE_RADIUS = 0.45


def sphere_levelset(x, center=SPHERE_CENTER, radius=SPHERE_RADIUS):
    """phi = |x - c|^2 - r^2 at the rows of x (torch tensor [N, gdim]); the offsets keep every
    vertex value away from zero (SURVEY.md section 8d)."""
    c = torch.tensor(center[:x.shape[1]], dtype=torch.float64, device=x.device)
    d = x - c
    return (d * d).sum(dim=1) - radius * radius


def ball_source(x, center=SPHERE_CENTER, radius=0.2, value=10.0):
    """Nodal values of 10 * 1[ball], the analogue of the demos' source term
    (demo/strong-dirichlet/flower/data.py:54-62)."""
    c = torch.tensor(center[:x.shape[1]], dtype=torch.float64, device=x.device)
    d = x - c
    return torch.where((d * d).sum(dim=1) <= radius * radius, value, 0.0).to(torch.float64)


# ---- flower domain of the reference demos (demo/weak-dirichlet/flower/data.py:27-99, demo/strong-dirichlet/
# flower/data.py:16-62): a disc of radius 2 with eight petals.  numpy, x of shape (gdim | 3, npoints) like a dolfinx
# interpolation callback.  `flower_detection` is the non-smooth min used for the tags (data.py:57-82),
# `flower_levelset` the graded smooth-min used in the forms (:27-54), `flower_source` 10 on a small disc inside the
# first petal (:85-99).  Checked against the reference's own values in tests/golden/flower_demo.npz.
def _flower_parts(x):
    s = np.cos(np.pi / 8.0) + np.sin(np.pi / 8.0)
    rp = np.sqrt(2.0) * 2.0 * s * np.sin(np.pi / 8.0)
    yield x[0] ** 2 + x[1] ** 2 - 4.0
    for i in range(1, 9):
        cx, cy = 2.0 * s * np.cos(i * np.pi / 4.0), 2.0 * s * np.sin(i * np.pi / 4.0)
        yield (x[0] - cx) ** 2 + (x[1] - cy) ** 2 - rp ** 2


def flower_detection(x):
    val = None
    for part in _flower_parts(x):
        val = part if val is None else np.minimum(val, part)
    return val


def flower_levelset(x):
    r = np.sqrt(x[0] ** 2 + x[1] ** 2)
    k = (np.pi / 2.0 - np.arctan(50.0 * (r - 2.0))) / np.pi / 2.0          # graded smoothing width in (0, 1/2)
    val = None
    for part in _flower_parts(x):
        if val is None:
            val = part
            continue
        lo = np.minimum(val, part)
        val = np.maximum(k, lo) - np.sqrt(np.maximum(k - val, 0.0) ** 2 + np.maximum(k - part, 0.0) ** 2)
    return val


def flower_source(x):
    s = np.cos(np.pi / 8.0) + np.sin(np.pi / 8.0)
    r1 = np.sqrt(2.0) * 2.0 * s * np.sin(np.pi / 8.0)
    return np.where((x[0] - 2.0 * s) ** 2 + x[1] ** 2 <= r1 ** 2 / 2.0, 10.0, 0.0)
