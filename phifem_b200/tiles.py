"""Symbolic phase of the cell-once cell pass (csrc/assemble_tiles.cu, k_assemble_tiles_p1).

Arrays of `phifem_cell_tiles` (include/phifem_b200.h): the listed rows are cut into tiles of R consecutive rows (R =
threads per CTA); a tile's cells = the active cells touching one of its rows, in ascending cell index, R cells per chunk;
a record per (row, cell) names the cell's slot in its chunk and where the cell's other vertices sit in the row's column
list.  Sort / scatter plumbing with torch ops on the mesh's device (CPU tensors work: tests/test_tiles_symbolic.py).
"""
import torch

from . import _lib

ROWS_PER_TILE = 256
MAX_ROW_NNZ = 128            # positions are 7 bits


class CellTiles:
    def __init__(self, mesh, active, cut, slots_cells, indptr, rows, diag_pos, rows_per_tile=ROWS_PER_TILE, push=False):
        """active [Na] int: active cells ascending; cut [Na] 0/1; slots_cells [Na, nv*nv] CSR slot of (row i, col j);
        indptr [n+1] int64; rows [L] int64 listed rows in processing order; diag_pos [L] uint8."""
        if rows_per_tile not in (128, 256):
            raise ValueError("rows_per_tile must be 128 or 256")
        dev = rows.device
        i64 = dict(dtype=torch.int64, device=dev)
        R = self.rows_per_tile = int(rows_per_tile)
        nv = mesh.cells.shape[1]
        n = indptr.numel() - 1
        L = int(rows.numel())
        self.n_listed = L
        self.n_tiles = nt = (L + R - 1) // R
        self.rows = rows.to(torch.int32).contiguous()
        self.diag_pos = diag_pos.contiguous()
        li_of_row = torch.full((n,), -1, **i64)
        li_of_row[rows] = torch.arange(L, **i64)
        cells_act = mesh.cells[active.long()].long()                      # [Na, nv]
        na = int(cells_act.shape[0])
        li = li_of_row[cells_act]                                         # [Na, nv]; -1: row not listed here
        valid = li >= 0
        a_idx = torch.arange(na, **i64)[:, None].expand(na, nv)
        key = (li[valid] // R) * max(na, 1) + a_idx[valid]                # (tile, active cell) of each (cell, vertex)
        ukey = torch.unique(key)                                          # sorted: tile-major, cells ascending
        pt, pa = ukey // max(na, 1), ukey % max(na, 1)
        cnt = torch.bincount(pt, minlength=nt)
        chunks_of = (cnt + R - 1) // R
        chunk_ptr = torch.zeros(nt + 1, **i64)
        chunk_ptr[1:] = torch.cumsum(chunks_of, 0)
        self.n_chunks = nch = int(chunk_ptr[-1])
        self.n_cell_slots = int(ukey.numel())                             # cell evaluations per pass
        self.n_active = na
        first = torch.cumsum(cnt, 0) - cnt
        rank = torch.arange(ukey.numel(), **i64) - first[pt]
        slot = chunk_ptr[pt] * R + rank
        sv = torch.full((max(nch, 1) * R, 4), -1, **i64)
        verts = cells_act[pa]
        if nv == 3:
            verts = torch.cat([verts, torch.zeros((verts.shape[0], 1), **i64)], dim=1)
        verts = verts.clone()
        verts[:, 1] |= cut.long()[pa] << 31
        sv[slot] = verts
        sv = torch.where(sv >= 2 ** 31, sv - 2 ** 32, sv).to(torch.int32)  # same bits as uint32
        # ---- push words (cell_pass="push"): per slot and cell-local vertex, where the tensor's row goes -----------
        self.push = None
        if push:
            sl = slots_cells.long().reshape(na, nv, nv)
            rows_s = cells_act[pa]                                         # [S, nv] row of each local vertex
            li_s = li[pa]
            mine = (li_s >= 0) & ((li_s // R) == pt[:, None])
            words = torch.zeros((max(nch, 1) * R, 4), **i64)
            for i in range(nv):
                w = (li_s[:, i] % R) | (1 << 8)
                m = 0
                for j in range(nv):
                    if j == i:
                        continue
                    pos = sl[pa, i, j] - indptr[rows_s[:, i]]
                    assert pos.numel() == 0 or (int(pos.min()) >= 0 and int(pos.max()) < MAX_ROW_NNZ)
                    w = w | (pos << (10 + 7 * m))
                    m += 1
                words[slot, i] = torch.where(mine[:, i], w, torch.zeros_like(w))
            self.push = words.to(torch.int32).contiguous()                 # bits 0..30 only
            del sl, rows_s, li_s, mine, words
        # ---- records ------------------------------------------------------------------------------------------
        gslot = slot[torch.searchsorted(ukey, key)]                        # slot of the record's cell in ITS tile
        chunk, lane = gslot // R, gslot % R
        loc = torch.arange(nv, **i64)[None, :].expand(na, nv)[valid]       # cell-local index of the row's vertex
        arow = a_idx[valid]
        sl = slots_cells.long().reshape(na, nv, nv)
        row_id = cells_act[valid]
        word = lane | (loc << 8)
        for m in range(nv - 1):
            j = m + (m >= loc).long()                                      # m-th other vertex, ascending local order
            pos = sl[arow, loc, j] - indptr[row_id]
            assert pos.numel() == 0 or (int(pos.min()) >= 0 and int(pos.max()) < MAX_ROW_NNZ)
            word |= pos << (10 + 7 * m)
        rkey = chunk * R + (li[valid] % R)                                 # (chunk, row of the tile)
        order = torch.argsort(rkey, stable=True)                           # records of a row keep cell order
        self.n_records = int(word.numel())
        self.rec = word[order].to(torch.int32).contiguous()
        if self.rec.numel() == 0:
            self.rec = torch.zeros(1, dtype=torch.int32, device=dev)
        per = torch.bincount(rkey, minlength=max(nch, 1) * R).reshape(max(nch, 1), R)
        off = torch.zeros((max(nch, 1), R + 1), **i64)
        off[:, 1:] = torch.cumsum(per, dim=1)
        rec_base = torch.zeros(max(nch, 1) + 1, **i64)
        rec_base[1:] = torch.cumsum(off[:, -1], 0)
        if int(rec_base[-1]) >= 2 ** 31:
            raise NotImplementedError("cell tiles: more than 2^31 records")
        self.rec_off = off.to(torch.int16).contiguous()                    # <= R * nv <= 1024 per chunk
        self.rec_base = rec_base.to(torch.int32).contiguous()
        self.chunk_ptr = chunk_ptr.to(torch.int32).contiguous()
        self.slot_verts = sv.contiguous()
        self._c = None

    @property
    def recompute(self):
        """Cell evaluations per active cell (1 = every cell once; 4 = the row-gather pass on tetrahedra)."""
        return self.n_cell_slots / max(1, self.n_active)

    def nbytes(self):
        return int(sum(t.numel() * t.element_size() for t in (self.rows, self.diag_pos, self.chunk_ptr, self.slot_verts,
                                                             self.rec_base, self.rec_off, self.rec) + (
                                                                 (self.push,) if self.push is not None else ())))

    def c_struct(self):
        if self._c is None:
            p = _lib.ptr
            self._c = _lib.CCellTiles(self.rows_per_tile, self.n_tiles, self.n_listed, p(self.rows), p(self.diag_pos),
                                      p(self.chunk_ptr), p(self.slot_verts), p(self.rec_base), p(self.rec_off),
                                      p(self.rec), p(self.push) if self.push is not None else None)
        return self._c
