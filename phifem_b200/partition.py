"""Owner-computes sharding of an ARBITRARY simplex mesh across ranks (SURVEY.md section 8e).

`dist.SlabProblem` shards the synthetic weak-scaling box by construction.  This module shards any
triangle / tetrahedron mesh the way the north star describes: cells are sorted along a space-filling
(Morton) curve of their centroids and cut into `world` contiguous ranges; a CSR row (= vertex) is owned by
the lowest rank owning a cell that touches it; every rank keeps its own range, the cells touching its rows and
the cells sharing a vertex with those (which covers their facet neighbours, the reach of the ghost penalty, without a
global facet numbering) -- plus, with `single_layer_cut`, one more such layer --, classifies them redundantly and runs the row-gather kernels on its own rows.  Nothing is exchanged in the numeric phase except the 8-byte "any exterior cell" all-reduce of
the facet algebra (reference src/phifem/mesh_scripts.py:469-474).

The local mesh keeps the global relative order of cells, vertices and hence facets (order-preserving
relabelling), so every owned row sums the same contributions in the same order as on one GPU: the stacked
ranks are bitwise identical to the single-GPU operator.

The partitioner is symbolic-phase plumbing (torch ops on the mesh's device; every rank derives its part from
the same global arrays, no communication), so it also runs on CPU tensors under `gloo`, which is how the CPU
tests cover it.  The reference has no counterpart: dolfinx partitions with a graph partitioner behind
`create_rectangle` / `read_mesh` (demo/strong-dirichlet/flower/main.py:48-49) and phifem carries a TODO for
parallel tag transfer (src/phifem/mesh_scripts.py:264).
"""
import torch

from . import assemble, mesh_scripts
from .mesh import Mesh


from .mesh import morton_keys  # noqa: E402  (63-bit Morton keys over the bounding box)


def partition_cells(mesh, world, weights=None):
    """cell_owner [Nc] int64: contiguous ranges of the Morton order of the cell centroids, of equal total
    weight (default weight 1 per cell)."""
    cent = mesh.x[mesh.cells.long()].mean(dim=1)
    order = torch.argsort(morton_keys(cent), stable=True)
    w = torch.ones(mesh.num_cells, dtype=torch.float64, device=mesh.device) if weights is None \
        else weights.to(mesh.device, torch.float64)
    cum = torch.cumsum(w[order], 0)
    part = torch.clamp(((cum - 0.5 * w[order]) / cum[-1] * world).long(), 0, world - 1)
    owner = torch.empty(mesh.num_cells, dtype=torch.int64, device=mesh.device)
    owner[order] = part
    return owner


def rank_share(mesh, cell_owner, vowner, rank, single_layer_cut=False):
    """Global ids (ascending) of the cells and vertices rank `rank` keeps: the cells touching a row it owns, the cells
    sharing a vertex with those (a superset of their facet neighbours -- the reach of the ghost penalty and of the
    one-sided entities -- that needs no global facet numbering), its own range of the curve, and with
    `single_layer_cut` (reference :349-358 re-tags a cut cell from every cell sharing a VERTEX with it) one more layer."""
    cells = mesh.cells.long()
    dev = mesh.device
    owned_v = vowner == rank
    keep = owned_v[cells].any(dim=1)
    for _ in range(2 if single_layer_cut else 1):
        vmark = torch.zeros(mesh.num_vertices, dtype=torch.bool, device=dev)
        vmark[cells[keep].reshape(-1)] = True
        keep = vmark[cells].any(dim=1)
    keep |= cell_owner == rank             # every cell's tag has one home
    gc = torch.nonzero(keep).reshape(-1)
    gv = torch.unique(cells[gc].reshape(-1))
    return gc, gv


class PartitionedProblem:
    """One rank's share of (mesh, phi, f): local mesh = cells touching owned rows + the cells around them.

    Attributes: `mesh` (local), `phi`, `f` (local vertex values), `global_vertex` / `global_cell` (ids of the
    local entities, ascending), `row_mask` (local vertices whose rows this rank owns), `cell_owned`.

    Two ways in: the constructor (every rank holds the global arrays and cuts its own share: the CPU tests) and
    `PartitionedProblem.scatter` (ONE rank holds the global mesh, computes the partition once and sends every rank its
    share only: symbolic time and memory of a rank shrink with the number of ranks)."""

    def __init__(self, mesh, phi, f, rank, world, group=None, weights=None, single_layer_cut=False):
        assemble.refuse_hexahedra(mesh, "PartitionedProblem")
        if mesh.cell_type not in ("triangle", "tetrahedron"):
            raise NotImplementedError("sharding supports triangles and tetrahedra")
        cell_owner, vowner = self.ownership(mesh, world, weights)
        self.vertex_owner_global = vowner
        gc, gv = rank_share(mesh, cell_owner, vowner, rank, single_layer_cut)
        self._from_share(rank, world, group, single_layer_cut, mesh.cell_type, mesh.num_vertices, gc, gv,
                         mesh.cells[gc].long(), mesh.x[gv], phi.to(mesh.device)[gv], f.to(mesh.device)[gv],
                         vowner[gv] == rank, cell_owner[gc] == rank)

    @staticmethod
    def ownership(mesh, world, weights=None):
        """(cell_owner [Nc], vertex_owner [Nv]): contiguous ranges of the Morton order of the cell centroids of equal
        weight; a vertex (= CSR row) belongs to the lowest rank owning a cell that touches it."""
        cells = mesh.cells.long()
        cell_owner = partition_cells(mesh, world, weights)
        vowner = torch.full((mesh.num_vertices,), world, dtype=torch.int64, device=mesh.device)
        vowner.scatter_reduce_(0, cells.reshape(-1), cell_owner.repeat_interleave(cells.shape[1]), reduce="amin")
        return cell_owner, vowner

    def _from_share(self, rank, world, group, single_layer_cut, cell_type, n_global_vertices, gc, gv, cells_global,
                    x, phi, f, row_mask, cell_owned):
        dev = x.device
        self.rank, self.world, self.group = rank, world, group
        self.single_layer_cut = bool(single_layer_cut)
        # order-preserving relabelling: local vertex k = k-th smallest global id
        local = torch.searchsorted(gv, cells_global.reshape(-1)).reshape(cells_global.shape)
        self.mesh = Mesh(x, local.to(torch.int32), cell_type, dev)
        self.global_cell, self.global_vertex = gc, gv
        self.n_global_vertices = int(n_global_vertices)
        self.row_mask = row_mask.to(torch.bool)
        self.cell_owned = cell_owned.to(torch.bool)
        self.n_owned_cells = int(self.cell_owned.sum())
        self.phi, self.f = phi.contiguous(), f.contiguous()
        self.plan = None
        self.peer = None

    @classmethod
    def scatter(cls, mesh, phi, f, rank, world, group=None, weights=None, single_layer_cut=False, src=0,
                device=None):
        """Rank `src` passes the global (mesh, phi, f) -- everybody else passes None -- computes the Morton partition
        ONCE and sends each rank its share: global ids, cell -> global vertex, coordinates, level set, source, owned
        rows, owned cells (point-to-point `torch.distributed` transfers: NCCL between GPUs, gloo on the CPU).  No rank
        but `src` ever holds the global arrays, and nobody builds the global facet numbering."""
        import torch.distributed as dist
        dev = torch.device(device) if device is not None else mesh.device
        i64 = dict(dtype=torch.int64, device=dev)
        names = ("gc", "gv", "cells", "x", "phi", "f", "row_mask", "cell_owned")
        dtypes = (torch.int64, torch.int64, torch.int64, torch.float64, torch.float64, torch.float64, torch.uint8,
                  torch.uint8)
        mine = None
        if rank == src:
            assemble.refuse_hexahedra(mesh, "PartitionedProblem.scatter")
            if mesh.cell_type not in ("triangle", "tetrahedron"):
                raise NotImplementedError("sharding supports triangles and tetrahedra")
            cell_owner, vowner = cls.ownership(mesh, world, weights)
            nv, gdim = mesh.cells.shape[1], mesh.gdim
            for r in range(world):
                gc, gv = rank_share(mesh, cell_owner, vowner, r, single_layer_cut)
                part = (gc, gv, mesh.cells[gc].long().reshape(-1), mesh.x[gv].reshape(-1), phi.to(dev)[gv],
                        f.to(dev)[gv], (vowner[gv] == r).to(torch.uint8), (cell_owner[gc] == r).to(torch.uint8))
                head = torch.tensor([gc.numel(), gv.numel(), mesh.num_vertices, nv, gdim], **i64)
                if r == src:
                    mine = (head, part)
                    continue
                dist.send(head, r, group=group)
                for t in part:
                    dist.send(t.contiguous(), r, group=group)
                del part
            head, part = mine
        else:
            head = torch.empty(5, **i64)
            dist.recv(head, src, group=group)
            nc, nvl, _, nv, gdim = (int(v) for v in head)
            sizes = (nc, nvl, nc * nv, nvl * gdim, nvl, nvl, nvl, nc)
            part = []
            for n, dt in zip(sizes, dtypes):
                t = torch.empty(n, dtype=dt, device=dev)
                dist.recv(t, src, group=group)
                part.append(t)
        nc, nvl, n_global, nv, gdim = (int(v) for v in head)
        p = dict(zip(names, part))
        self = cls.__new__(cls)
        self.vertex_owner_global = None
        self._from_share(rank, world, group, single_layer_cut, "triangle" if nv == 3 else "tetrahedron", n_global,
                         p["gc"], p["gv"], p["cells"].reshape(nc, nv), p["x"].reshape(nvl, gdim), p["phi"], p["f"],
                         p["row_mask"], p["cell_owned"])
        return self

    # ---- tags --------------------------------------------------------------------------------------
    def classify(self, dls, ws, mark=None):
        """Cells, interior facets overlapped with the 8-byte all-reduce of the exterior-cell count, mesh-boundary
        facets (all on the current stream; mesh_scripts.classify_sharded)."""
        return mesh_scripts.classify_sharded(self.mesh, dls, ws, group=self.group, world=self.world, mark=mark,
                                             single_layer_cut=self.single_layer_cut, peer=getattr(self, "peer", None))

    def enable_peer_flags(self):
        """Exchange the exterior-cell counts through NVLink peer memory (phifem_b200/peer.py) instead of an all-reduce;
        returns False (and keeps the all-reduce) where peer mapping is unavailable.  Collective: every rank calls it."""
        from . import peer
        self.peer = peer.try_create(self.rank, self.world, self.group)
        return self.peer is not None

    # ---- symbolic phase ----------------------------------------------------------------------------
    def build_plan(self, cell_tags8, facet_tags8, entities=None):
        mesh = self.mesh
        if entities is None:
            entities = mesh_scripts._integration_entities_dev(mesh, cell_tags8, facet_tags8, 4, (1, 2))
        plan = assemble.AssemblyPlan(mesh, cell_tags8.contiguous(), facet_tags8.contiguous(),
                                     entities.reshape(-1, 2), method="rows", row_mask=self.row_mask)
        if plan.method != "rows":
            raise NotImplementedError("owner-computes sharding needs the row-gather plan")
        ip = plan.indptr.long()
        rows = torch.nonzero(self.row_mask).reshape(-1)
        cnt = ip[rows + 1] - ip[rows]
        plan.owned_rows_local = rows
        plan.owned_rows_global = self.global_vertex[rows]
        plan.owned_indptr = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=mesh.device)
        plan.owned_indptr[1:] = torch.cumsum(cnt, 0)
        # CSR slots of the owned rows, row by row
        start = torch.repeat_interleave(ip[rows] - plan.owned_indptr[:-1], cnt)
        plan.owned_slots = start + torch.arange(int(plan.owned_indptr[-1]), device=mesh.device)
        plan.owned_cols = self.global_vertex[plan.indices[plan.owned_slots].long()]
        self.plan = plan
        self.data, self.b_local = plan.new_outputs()
        return plan

    # ---- numeric phase -----------------------------------------------------------------------------
    def assemble(self, sigma=1.0, marks=None, local_kernels=None):
        """Runs the row-gather kernels on the owned rows.  `local_kernels(plan, phi, f, sigma, data, b)`
        replaces the CUDA kernels in the CPU (gloo) tests only."""
        p = self.plan
        if local_kernels is None:
            assemble.assemble_into(p, self.phi, self.f, sigma, self.data, self.b_local, marks=marks)
        else:
            local_kernels(p, self.phi, self.f, sigma, self.data, self.b_local)
        return self.data, self.b_local

    def owned_csr(self):
        """(global row ids [m] ascending, indptr [m+1], global column ids, data, b) of the owned rows."""
        p = self.plan
        return (p.owned_rows_global, p.owned_indptr, p.owned_cols, self.data[p.owned_slots],
                self.b_local[p.owned_rows_local])
