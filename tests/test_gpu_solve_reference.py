"""The kernels of csrc/solve.cu held to a high-precision reference at every launch shape they take.

`phifem_bicgstab_iterate` picks 4, 8, 16 or 32 lanes per row from nnz / n_act, caps the product's grid at 8 CTAs per SM
(then every lane group walks several rows: the persistent multi-pass loop) and caps the vector kernels' grid the same
way (then they stride).  The assembled operators of the other tests reach only a few of these shapes, so the synthetic
systems below are built to pick each one, and every case asserts the shape it claims from the host formulas of
solve.cu (`spmv_lanes`, `spmv_rows_grid`).

Oracles:
- products and dot products: the forward-error bound |y_i - ref_i| <= (n_i + 2) 2^-53 sum_k |a_ik x_k| against an
  extended-precision sum (np.longdouble), which holds for any summation order and fails by many orders of magnitude if
  an entry is dropped, doubled or read through the wrong column;
- the set-up passes (diagonal, row maximum, remapped columns) select and take maxima only: bit for bit;
- one fused BiCGStab iteration from a captured device state against the same iteration restated in np.longdouble
  (one step from the same state, so rounding differences cannot grow over iterations);
- reproducibility and continuation: bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

from phifem_b200 import _lib

NUM_SMS, SPMV_BLOCK, VEC_BLOCK = 148, 256, 256
GRID_CAP = 8 * NUM_SMS               # both capped grids: 8 CTAs per SM
U = 2.0 ** -53                       # unit roundoff of float64
LD = np.longdouble
EPS_LD = float(np.finfo(LD).eps)     # the reference's own roundoff (2^-64 for x87 extended precision)
SCALAR_RTOL = 1e-11
VECTOR_RTOL = 1e-11
PIVOT_TOL = 1e-14                    # solve.bicgstab's default


# ---- launch shape: the host formulas of csrc/solve.cu ------------------------------------------------------------------
def spmv_lanes(n_act, nnz):
    avg = nnz // n_act if n_act > 0 else 0
    return 4 if avg <= 24 else (8 if avg <= 48 else (16 if avg <= 96 else 32))


def spmv_rows_grid(n_act, lanes):
    return min((n_act * lanes + SPMV_BLOCK - 1) // SPMV_BLOCK, GRID_CAP)


def vec_grid(n_act):
    return min((n_act + VEC_BLOCK - 1) // VEC_BLOCK, GRID_CAP)


def launch_shape(n_act, nnz):
    """(lanes, product grid, vector grid, passes of the product's persistent loop)"""
    lanes = spmv_lanes(n_act, nnz)
    grid = spmv_rows_grid(n_act, lanes)
    groups = grid * (SPMV_BLOCK // lanes)
    return lanes, grid, vec_grid(n_act), (n_act + groups - 1) // groups


# ---- synthetic systems ---------------------------------------------------------------------------------------------------
ACTIVE, NO_DIAG, ZERO_DIAG, TINY_DIAG, EMPTY = 0, 1, 2, 3, 4


def _row_reduce(ufunc, vals, indptr):
    """ufunc.reduce over every CSR row (0 for an empty row), vectorised."""
    n = len(indptr) - 1
    out = np.zeros(n, dtype=vals.dtype)
    full = np.nonzero(indptr[1:] > indptr[:-1])[0]
    if len(full):
        out[full] = ufunc.reduceat(vals, indptr[:-1][full])
    return out


class System:
    """A CSR matrix (int32 indptr / indices) and the compact system of its active rows as solve.bicgstab derives it."""

    def __init__(self, indptr, indices, data, pivot_tol=PIVOT_TOL):
        self.indptr, self.indices, self.data = indptr.astype(np.int32), indices.astype(np.int32), data
        self.n, self.nnz = len(indptr) - 1, len(data)
        self.lengths = np.diff(indptr.astype(np.int64))
        self.compact(pivot_tol)

    @classmethod
    def synthetic(cls, n_act, per_row, lanes, seed):
        """A strictly dominant (non-symmetric) diagonal on the active rows, a sprinkling of inactive rows (no diagonal
        entry, an explicit 0.0 diagonal, a diagonal of 1e-15 * rowmax, empty rows), random columns (some into inactive
        rows), rows of exactly 1, 4 L and 4 L + 1 entries and rows of more than 300."""
        rng = np.random.default_rng(seed)
        n_inact = max(16, n_act // 64)
        n = n_act + n_inact
        kind = np.full(n, ACTIVE, np.int8)
        kind[rng.choice(n, n_inact, replace=False)] = NO_DIAG + np.arange(n_inact) % 4
        lengths = rng.integers(1, 2 * per_row, n)                   # mean per_row
        lengths[(kind != ACTIVE) & (lengths < 2)] = 2
        lengths[kind == EMPTY] = 0
        act = np.nonzero(kind == ACTIVE)[0]
        special = np.array([1, 4 * lanes, 4 * lanes + 1, 333])     # one-entry rows, the kBatch * L tail, > 300 entries
        lengths[act[:4]] = special
        lengths[act[-4:]] = special[::-1]
        indptr = np.zeros(n + 1, np.int64)
        np.cumsum(lengths, out=indptr[1:])
        nnz = int(indptr[-1])
        row_of = np.repeat(np.arange(n), lengths)
        indices = (row_of + 1 + rng.integers(0, n - 1, nnz)) % n    # never the diagonal
        data = rng.uniform(-1.0, 1.0, nnz) * 10.0 ** rng.uniform(-2, 2, n)[row_of]
        has_diag = np.isin(kind, (ACTIVE, ZERO_DIAG, TINY_DIAG))
        dr = np.nonzero(has_diag)[0]
        dpos = indptr[dr] + (rng.random(len(dr)) * lengths[dr]).astype(np.int64)
        indices[dpos] = dr
        off = np.abs(data)
        off[dpos] = 0.0
        offsum, offmax = _row_reduce(np.add, off, indptr), _row_reduce(np.maximum, off, indptr)
        diag = rng.choice([-1.0, 1.0], n) * ((1.5 + rng.random(n)) * offsum + 10.0 ** rng.uniform(-2, 2, n))
        diag[kind == ZERO_DIAG] = 0.0
        diag[kind == TINY_DIAG] = 1e-15 * offmax[kind == TINY_DIAG]
        data[dpos] = diag[dr]
        S = cls(indptr, indices, data)
        S.kind = kind
        S.diag_pos = np.full(n, -1, np.int64)
        S.diag_pos[dr] = dpos - indptr[dr]                          # position of the diagonal within its row
        return S

    def row_scan(self):
        """diag (0 where the row has no diagonal entry) and rowmax = max_c |a_rc|: what k_row_scan computes."""
        indptr = self.indptr.astype(np.int64)
        rows = np.repeat(np.arange(self.n), self.lengths)
        on = self.indices == rows
        diag = np.zeros(self.n)
        diag[rows[on]] = self.data[on]
        return diag, _row_reduce(np.maximum, np.abs(self.data), indptr)

    def compact(self, pivot_tol):
        diag, rowmax = self.row_scan()
        self.rows = np.nonzero(np.abs(diag) > pivot_tol * rowmax)[0]
        self.n_act = n_act = len(self.rows)
        self.cmap = np.full(self.n, n_act, np.int32)
        self.cmap[self.rows] = np.arange(n_act, dtype=np.int32)
        self.cols = self.cmap[self.indices]
        self.minv = 1.0 / diag[self.rows]
        # CSR of the active rows in the compact numbering (column n_act: an inactive column, where vectors hold 0)
        clen = self.lengths[self.rows]
        self.c_indptr = np.zeros(n_act + 1, np.int64)
        np.cumsum(clen, out=self.c_indptr[1:])
        gather = np.repeat(self.indptr[self.rows].astype(np.int64) - self.c_indptr[:-1], clen) + np.arange(
            self.c_indptr[-1])
        self.c_cols, self.c_data, self.c_len = self.cols[gather], self.data[gather], clen

    def matvec(self, x, dtype=LD):
        """y = A x on the compact system (x: n_act + 1 entries, the last 0) in `dtype`, and sum_k |a_ik x_k|."""
        prod = self.c_data.astype(dtype) * np.asarray(x, dtype)[self.c_cols]
        return np.add.reduceat(prod, self.c_indptr[:-1]), np.add.reduceat(np.abs(prod), self.c_indptr[:-1])

    def scipy_compact(self):
        import scipy.sparse as sp
        n_act = self.n_act
        return sp.csr_matrix((self.c_data, self.c_cols, self.c_indptr), shape=(n_act, n_act + 1))[:, :n_act]


# (name, lanes, n_act, mean entries per row); "multi": n_act * lanes > 8 * 148 * 256, the product's persistent loop
# takes several passes; "strided": n_act > 8 * 148 * 256, the vector kernels' grid-stride loops wrap too
CASES = [("L4-single", 4, 3000, 12), ("L4-multi", 4, 80000, 12),
         ("L8-single", 8, 3000, 36), ("L8-multi", 8, 42000, 36),
         ("L16-single", 16, 3000, 72), ("L16-multi", 16, 21000, 72),
         ("L32-single", 32, 3000, 110), ("L32-multi", 32, 11000, 110),
         ("L4-strided", 4, 310000, 6)]
CASE_IDS = [c[0] for c in CASES]
_SYSTEMS = {}


def system(name):
    if name not in _SYSTEMS:
        i = CASE_IDS.index(name)
        _, lanes, n_act, per_row = CASES[i]
        S = System.synthetic(n_act, per_row, lanes, seed=100 + i)
        assert S.n_act == n_act
        _SYSTEMS[name] = S
    return _SYSTEMS[name]


def claimed_shape(name):
    _, lanes, n_act, _ = CASES[CASE_IDS.index(name)]
    return lanes, name.endswith(("multi", "strided")), name.endswith("strided")


def test_cases_cover_every_launch_shape():
    """Each case has the shape its name claims; together they take every lane count single-pass and multi-pass, and the
    striding vector kernels.  A change of the thresholds in solve.cu that moved a case fails here."""
    seen = set()
    for name in CASE_IDS:
        S = system(name)
        lanes, multi, strided = claimed_shape(name)
        L, grid, vgrid, passes = launch_shape(S.n_act, S.nnz)
        assert L == lanes, (name, L)
        assert (passes > 1) == multi and (grid == GRID_CAP) == multi, (name, grid, passes)
        assert (S.n_act > GRID_CAP * VEC_BLOCK) == strided and (vgrid == GRID_CAP) == strided, (name, vgrid)
        assert S.nnz < 4_000_000
        # the edges the kernels must get right, present in every system
        for length in (1, 4 * L, 4 * L + 1):
            assert np.any(S.c_len == length), (name, length)
        assert S.c_len.max() > 300
        assert np.any(S.cols == S.n_act)                             # columns into inactive rows
        for k in (NO_DIAG, ZERO_DIAG, TINY_DIAG, EMPTY):
            assert np.any(S.kind == k)
        assert np.array_equal(S.rows, np.nonzero(S.kind == ACTIVE)[0])
        seen.add((L, passes > 1))
    assert seen == {(L, m) for L in (4, 8, 16, 32) for m in (False, True)}


# ---- the BiCGStab iteration, restated -----------------------------------------------------------------------------------
def _dot(a, b, dtype=LD):
    p = np.asarray(a, dtype) * np.asarray(b, dtype)
    return p.sum(), np.abs(p).sum()


def _ext(v, dtype):
    return np.concatenate([np.asarray(v, dtype), np.zeros(1, dtype)])


def reference_step(S, rhat, st, dtype=LD, wrong=None):
    """One right-preconditioned (Jacobi) BiCGStab iteration from state `st` = {x, r, p, v, rho, alpha, omega} (csrc/solve.cu:
    p = r + beta (p - omega v), y = M^-1 p | v = A y | s = r - alpha v, z = M^-1 s | t = A z | x += alpha y + omega z,
    r = s - omega t), with rho_new = rhat.r computed directly.  Returns the vectors, the scalars of the state after the
    call (rho <- rho_new, and beta / rho_new / r.r of the NEXT iteration, which the call's closing scalar update writes)
    and the condition number sum |a_i b_i| / |sum a_i b_i| of the worst dot product.  `wrong` selects a deliberately
    wrong restatement (the tests of the tolerance)."""
    c = lambda v: np.asarray(v, dtype)            # noqa: E731
    minv, rhat = c(S.minv), c(rhat)
    x, r, p, v = c(st["x"]), c(st["r"]), c(st["p"]), c(st["v"])
    rho, alpha, omega = c(st["rho"]), c(st["alpha"]), c(st["omega"])
    conds = []

    def dot(a, b):
        s, a_ = _dot(a, b, dtype)
        conds.append(float(a_ / abs(s)) if s != 0 else np.inf)
        return s

    rho_new = dot(rhat, r)
    beta = (rho_new / rho) * ((omega / alpha) if wrong == "beta-swapped" else (alpha / omega))
    p = r + beta * (p - omega * v)
    y = minv * p
    v = S.matvec(_ext(y, dtype), dtype)[0]
    alpha = rho_new / dot(rhat, v)
    s = r - alpha * v
    z = minv * s
    t = S.matvec(_ext(z, dtype), dtype)[0]
    omega = dot(t, s) / (dot(s, s) if wrong == "omega-over-ss" else dot(t, t))
    x = x + alpha * y + omega * z
    r = s - omega * t
    rho_out = rho if wrong == "rho-not-rotated" else rho_new
    rho_next = dot(rhat, r)
    rr = dot(r, r)
    beta_next = (rho_next / rho_out) * (alpha / omega)
    return dict(x=x, r=r, p=p, v=v, s=s, t=t, y=y, z=z, rho=rho_out, alpha=alpha, omega=omega, beta=beta_next, rr=rr,
                rho_new=rho_next), max(conds)


SCALARS = ("rho", "alpha", "omega", "beta", "rr", "rho_new")
VECTORS = ("x", "r", "p", "v", "s", "t", "y", "z")


def step_errors(got, ref, cond):
    """|got - ref| over its tolerance for every scalar and vector of a step: SCALAR_RTOL relative on a scalar,
    VECTOR_RTOL times the max-norm on a vector, both times `cond`, the largest sum |a_i b_i| / |sum a_i b_i| of the dot
    products of the step.  A dot product's rounding error is a multiple of sum |a_i b_i|, so its relative error (and that
    of every scalar and vector formed from it) scales with this condition number.  It is large for rhat.r: BiCGStab
    makes r nearly orthogonal to rhat as it converges (10^2 .. 10^6 after five iterations here, 1 .. 10^3 before)."""
    c = max(cond, 1.0)
    err = {}
    for k in SCALARS:
        ref_k = float(ref[k])
        err[k] = abs(float(got[k]) - ref_k) / (SCALAR_RTOL * c * max(abs(ref_k), 1e-300))
    for k in VECTORS:
        ref_k = np.asarray(ref[k], LD)
        scale = float(np.abs(ref_k).max())
        err[k] = float(np.abs(np.asarray(got[k], LD)[:len(ref_k)] - ref_k).max()) / (VECTOR_RTOL * c * max(scale, 1e-300))
    return err


def initial_state(S, seed):
    b = np.random.default_rng(seed).uniform(-1.0, 1.0, S.n_act) * 10.0 ** np.random.default_rng(seed + 1).uniform(
        -1, 1, S.n_act)
    zero = np.zeros(S.n_act)
    return b, dict(x=zero, r=b.copy(), p=zero, v=zero, rho=1.0, alpha=1.0, omega=1.0)


def _advance(S, rhat, st, steps, dtype=LD):
    for _ in range(steps):
        nxt, _ = reference_step(S, rhat, st, dtype)
        st = {k: nxt[k] for k in ("x", "r", "p", "v", "rho", "alpha", "omega")}
    return st


def test_reference_iteration_converges_to_spsolve():
    """The restatement itself, on the CPU: run to convergence on two synthetic systems and compare with scipy's direct
    solve of the compact system."""
    import scipy.sparse.linalg as spla
    for name in ("L4-single", "L32-single"):
        S = system(name)
        b, st = initial_state(S, seed=5)
        bn = np.linalg.norm(b)
        for it in range(200):
            st = _advance(S, b, st, 1)
            res = float(np.sqrt(_dot(st["r"], st["r"])[0])) / bn
            if res < 1e-13:
                break
        assert res < 1e-13, (name, it, res)
        ref = spla.spsolve(S.scipy_compact().tocsc(), b)
        assert np.abs(np.asarray(st["x"], float) - ref).max() <= 1e-11 * np.abs(ref).max(), name
        # the recurrence residual is the true residual
        true_r = b - S.scipy_compact() @ np.asarray(st["x"], float)
        assert np.linalg.norm(true_r) <= 1e-12 * bn


def test_step_tolerance_is_tight_and_not_vacuous():
    """A float64 restatement of the step (another summation order) passes the comparison with a margin of 10^2; three
    wrong restatements -- omega = t.s / s.s, rho not rotated, alpha and omega swapped in beta -- miss it by at least
    10^3 (by 10^6 .. 10^14 on every case and seed tried)."""
    for name in ("L8-single", "L32-single"):
        S = system(name)
        b, st0 = initial_state(S, seed=9)
        st = _advance(S, b, st0, 5)
        st64 = {k: np.asarray(v, np.float64) for k, v in st.items()}    # a captured device state is float64
        ref, cond = reference_step(S, b, st64)
        f64, _ = reference_step(S, b, st64, dtype=np.float64)
        assert max(step_errors(f64, ref, cond).values()) <= 1e-2, (name, step_errors(f64, ref, cond))
        for wrong in ("omega-over-ss", "rho-not-rotated", "beta-swapped"):
            bad, _ = reference_step(S, b, st64, wrong=wrong)
            assert max(step_errors(bad, ref, cond).values()) >= 1e3, (name, wrong)


# ---- the device side ----------------------------------------------------------------------------------------------------
def _d(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


class Device:
    """The compact system of `S` on the GPU, as solve.bicgstab lays it out."""

    def __init__(self, S):
        self.S = S
        self.indptr, self.indices, self.data = _d(S.indptr), _d(S.indices), _d(S.data)
        self.rows, self.cols, self.minv = _d(S.rows.astype(np.int32)), _d(S.cols), _d(S.minv)

    def partials(self):
        return torch.full((2 * (2 * GRID_CAP + 1),), float("nan"), dtype=torch.float64, device="cuda")

    def spmv_rows(self, x, y, partials):
        P = _lib.ptr
        _lib.check(_lib.load().phifem_csr_spmv_rows(self.S.n_act, self.S.nnz, P(self.rows), P(self.indptr), P(self.cols),
                                                    P(self.data), P(x), P(y), P(partials), _lib.stream()))

    def start(self, b):
        n_act = self.S.n_act
        z = lambda extra=0: torch.zeros(n_act + extra, dtype=torch.float64, device="cuda")    # noqa: E731
        r = _d(b)
        V = dict(rhat=r.clone(), x=z(1), r=r, p=z(), v=z(), s=z(), t=z(), y=z(1), z=z(1),
                 state=torch.tensor([1.0, 1.0, 1.0, 0.0, 0.0, 0.0, 0.0, 0.0], dtype=torch.float64, device="cuda"),
                 partials=self.partials())
        rr = torch.dot(r, r)
        V["partials"][0] = rr
        V["partials"][1] = rr
        V["n_partials"] = ctypes.c_int32(1)
        return V

    def iterate(self, V, iterations):
        return _lib.load().phifem_bicgstab_iterate(
            self.S.n_act, self.S.nnz, *[_lib.ptr(t) for t in (self.rows, self.indptr, self.cols, self.data, self.minv)],
            *[_lib.ptr(V[k]) for k in ("rhat", "x", "r", "p", "v", "s", "t", "y", "z", "state", "partials")],
            ctypes.byref(V["n_partials"]), iterations, _lib.stream())

    @staticmethod
    def snapshot(V):
        out = {k: (v.cpu().numpy().copy() if torch.is_tensor(v) else v.value) for k, v in V.items()}
        return out

    @staticmethod
    def restore(snap):
        V = {k: (_d(v) if isinstance(v, np.ndarray) else ctypes.c_int32(v)) for k, v in snap.items()}
        return V


def _check_product(S, x, y, partials, w):
    """y against A x row by row, and the two partial sums of the first grid pairs against w.y and y.y."""
    L, grid, _, _ = launch_shape(S.n_act, S.nnz)
    ref, absum = S.matvec(x)
    n_act = S.n_act
    bound = (S.c_len + 2) * U * absum + S.c_len * EPS_LD * absum
    err = np.abs(np.asarray(y[:n_act], LD) - ref)
    assert np.all(err <= bound), ("row", int(np.argmax(err - bound)), float((err / np.maximum(bound, 1e-300)).max()))
    pairs = partials[:2 * grid].reshape(grid, 2)
    assert np.all(np.isfinite(pairs)), "a block of the product did not write its partial sums"
    assert np.all(np.isnan(partials[2 * grid:])), "partial sums written beyond the grid"
    for got, (a, b) in ((pairs[:, 0], (w[:n_act], y[:n_act])), (pairs[:, 1], (y[:n_act], y[:n_act]))):
        want, aw = _dot(a, b)
        tol = (n_act + grid + 2) * U * aw + 2 * n_act * EPS_LD * aw
        assert abs(np.sum(got.astype(LD)) - want) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_spmv_rows_and_partials_match_reference(name):
    S = system(name)
    D = Device(S)
    rng = np.random.default_rng(17)
    x = np.zeros(S.n_act + 1)
    x[:-1] = rng.choice([-1.0, 1.0], S.n_act) * 10.0 ** rng.uniform(-8, 8, S.n_act)
    xd = _d(x)
    y = torch.full((S.n_act + 1,), float("nan"), dtype=torch.float64, device="cuda")
    partials = D.partials()
    D.spmv_rows(xd, y, partials)
    y_h, p_h = y.cpu().numpy(), partials.cpu().numpy()
    assert np.isnan(y_h[-1])                                      # only the n_act rows are written
    _check_product(S, x, y_h, p_h, x)


@pytest.mark.gpu
@pytest.mark.parametrize("n_rows,per_row", [(1, 3), (1, 400), (1000, 9), (4133, 40), (2500, 330)])
def test_plain_spmv_matches_reference(n_rows, per_row):
    """phifem_csr_spmv (8 lanes per row, every row of the matrix): one row, a row count that is not a multiple of 32,
    empty rows, rows of 300 and more entries, x spanning 1e-8 .. 1e8."""
    rng = np.random.default_rng(n_rows + per_row)
    lengths = rng.integers(0, 2 * per_row, n_rows)
    if n_rows > 1:
        lengths[rng.choice(n_rows, max(1, n_rows // 50), replace=False)] = 0      # empty rows
    else:
        lengths[:] = per_row
    indptr = np.zeros(n_rows + 1, np.int64)
    np.cumsum(lengths, out=indptr[1:])
    nnz = int(indptr[-1])
    n_cols = max(n_rows, 50)
    indices = rng.integers(0, n_cols, nnz).astype(np.int32)
    data = rng.uniform(-1, 1, nnz) * 10.0 ** rng.uniform(-3, 3, nnz)
    x = rng.choice([-1.0, 1.0], n_cols) * 10.0 ** rng.uniform(-8, 8, n_cols)
    y = torch.full((n_rows,), float("nan"), dtype=torch.float64, device="cuda")
    P = _lib.ptr
    # the device arrays stay referenced until the kernel has run: a temporary tensor's block goes back to the caching
    # allocator when its last reference dies, and the next upload would reuse it
    args = [_d(indptr.astype(np.int32)), _d(indices), _d(data), _d(x), y]
    _lib.check(_lib.load().phifem_csr_spmv(n_rows, *[P(t) for t in args], _lib.stream()))
    got = y.cpu().numpy()
    prod = data.astype(LD) * x[indices].astype(LD)
    want, absum = _row_reduce(np.add, prod, indptr), _row_reduce(np.add, np.abs(prod), indptr)
    bound = (lengths + 2) * U * absum + lengths * EPS_LD * absum
    assert np.all(got[lengths == 0] == 0.0)
    assert np.all(np.abs(np.asarray(got, LD) - want) <= bound)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["L4-multi", "L32-single"])
def test_row_scan_and_remap_are_exact(name):
    """k_row_scan: diagonal and row maximum bit for bit, with the diagonal at every position mod 4 of its row, missing,
    or stored as 0.0; k_remap_columns: cols == cmap[indices] bit for bit (on nnz > 8 * 148 * 256 its grid-stride loop
    wraps)."""
    S = system(name)
    pos = S.diag_pos[S.kind != NO_DIAG]
    assert set((pos[pos >= 0] % 4).tolist()) == {0, 1, 2, 3}
    D = Device(S)
    lib, P = _lib.load(), _lib.ptr
    diag = torch.full((S.n,), float("nan"), dtype=torch.float64, device="cuda")
    rowmax = diag.clone()
    _lib.check(lib.phifem_csr_row_scan(S.n, P(D.indptr), P(D.indices), P(D.data), P(diag), P(rowmax), _lib.stream()))
    want_d, want_m = S.row_scan()
    assert np.array_equal(diag.cpu().numpy(), want_d) and np.array_equal(rowmax.cpu().numpy(), want_m)
    cols = torch.full((S.nnz,), -7, dtype=torch.int32, device="cuda")
    cmap = _d(S.cmap)
    _lib.check(lib.phifem_remap_columns(S.nnz, P(D.indices), P(cmap), P(cols), _lib.stream()))
    assert np.array_equal(cols.cpu().numpy(), S.cmap[S.indices])
    if name == "L4-multi":
        assert S.nnz > GRID_CAP * 256


@pytest.mark.gpu
def test_bicgstab_active_set_is_the_relative_pivot_test():
    """solve.bicgstab's active rows are |a_rr| > pivot_tol * rowmax: a diagonal of 1e-15 * rowmax is a null pivot at the
    default tolerance and active at 1e-16.  With maxiter = 0 the returned x is x0 on the active rows and 0 elsewhere."""
    from phifem_b200 import assemble, solve
    S = system("L8-single")
    D = Device(S)
    A = assemble.CSRMatrix(D.indptr, D.indices, D.data, (S.n, S.n))
    b = torch.ones(S.n, dtype=torch.float64, device="cuda")
    x0 = torch.full((S.n,), 2.0, dtype=torch.float64, device="cuda")
    for tol, active in ((PIVOT_TOL, S.kind == ACTIVE), (1e-16, (S.kind == ACTIVE) | (S.kind == TINY_DIAG))):
        x, info = solve.bicgstab(A, b, maxiter=0, x0=x0, pivot_tol=tol)
        assert info.iterations == 0 and info.n_active == int(active.sum())
        assert np.array_equal(x.cpu().numpy() != 0.0, active)


def _step_case(S, k, b=None):
    """Run k iterations, capture everything, run one more; returns (S, captured, after)."""
    D = Device(S)
    if b is None:
        b, _ = initial_state(S, seed=3)
    V = D.start(b)
    _lib.check(D.iterate(V, k))
    cap = Device.snapshot(V)
    V = Device.restore(cap)
    _lib.check(D.iterate(V, 1))
    return S, cap, Device.snapshot(V)


def _compare_step(S, cap, after):
    n_act = S.n_act
    _, _, vgrid, _ = launch_shape(n_act, S.nnz)
    # the captured partial sums are those of (rhat.r, r.r) of the captured residual
    npart = cap["n_partials"]
    pairs = cap["partials"][:2 * npart].reshape(npart, 2).astype(LD).sum(axis=0)
    for got, (a, b) in ((pairs[0], (cap["rhat"], cap["r"])), (pairs[1], (cap["r"], cap["r"]))):
        want, aw = _dot(a, b)
        assert abs(got - want) <= (n_act + vgrid + 2) * U * aw + 2 * n_act * EPS_LD * aw
    st = cap["state"]
    ref, cond = reference_step(S, cap["rhat"], dict(x=cap["x"][:n_act], r=cap["r"], p=cap["p"], v=cap["v"],
                                                    rho=st[0], alpha=st[1], omega=st[2]))
    got = {k: after[k] for k in VECTORS}
    got.update(zip(("rho", "alpha", "omega", "beta", "rr", "rho_new"), after["state"][:6]))
    err = step_errors(got, ref, cond)
    assert max(err.values()) <= 1.0, err
    assert after["n_partials"] == vgrid
    for k in ("x", "y", "z"):                      # the trailing slot of the vectors with one more entry stays 0
        assert after[k][n_act] == 0.0, k
    return cond


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1, 5])
@pytest.mark.parametrize("name", CASE_IDS)
def test_one_fused_iteration_matches_reference(name, k):
    S, cap, after = _step_case(system(name), k)
    assert cap["n_partials"] == (1 if k == 0 else launch_shape(S.n_act, S.nnz)[2])
    cond = _compare_step(S, cap, after)
    assert cond < (1e4 if k <= 1 else 1e7), cond   # the tolerance stays far below what a wrong step misses it by


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["L32-multi", "L4-strided"])
def test_iteration_is_reproducible_and_continues_bitwise(name):
    """Two runs from the same inputs agree bit for bit, and one call of 10 iterations equals ten calls of one."""
    S = system(name)
    D = Device(S)
    b, _ = initial_state(S, seed=11)
    runs = []
    for calls in ((10,), (10,), (1,) * 10):
        V = D.start(b)
        for k in calls:
            _lib.check(D.iterate(V, k))
        runs.append(Device.snapshot(V))
    for other in runs[1:]:
        for k in ("x", "r", "p", "v", "s", "t", "state"):
            assert np.array_equal(runs[0][k], other[k]), k
        assert other["n_partials"] == runs[0]["n_partials"]


@pytest.mark.gpu
def test_bicgstab_check_every_does_not_change_the_iterate():
    """solve.bicgstab reading |r|^2 back every iteration or every 10: the same x, bit for bit, at the same count."""
    from phifem_b200 import assemble, solve
    S = system("L16-single")
    D = Device(S)
    A = assemble.CSRMatrix(D.indptr, D.indices, D.data, (S.n, S.n))
    b = torch.from_numpy(np.random.default_rng(2).uniform(-1, 1, S.n)).cuda()
    x1, i1 = solve.bicgstab(A, b, rtol=1e-10, check_every=1)
    assert i1.converged, i1
    x10, i10 = solve.bicgstab(A, b, rtol=1e-10, check_every=10, maxiter=i1.iterations)
    assert i10.converged and i10.iterations == i1.iterations, (i1, i10)
    assert torch.equal(x1, x10)


def _elasticity_system():
    """The interface-elasticity operator of tests/test_gpu_elasticity.py (triangles, n = 12, P1 level set, Dirichlet
    conditions on the outer boundary): ~100 entries per active row."""
    import warnings
    from phifem_b200 import elasticity, fem, mesh_scripts, synthetic
    mesh = synthetic.rectangle_mesh(12, device="cuda")
    center, radius = (0.013, -0.021), 0.61
    V1 = fem.functionspace(mesh, 1)
    phi = synthetic.sphere_levelset(mesh.x, center=center, radius=radius)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, d_bdry, _ = mesh_scripts.compute_tags_measures(mesh, fem.Function(V1, phi.cpu().numpy()), 1,
                                                                        box_mode=True)
    rng = np.random.default_rng(77)
    f = torch.from_numpy(rng.uniform(-1, 1, (mesh.num_vertices, 2))).cuda()
    plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, d_bdry, V_phi=V1)
    bc_dofs = plan.dofs("u_in", plan.boundary_vertices()).reshape(-1)
    bcs = (bc_dofs, torch.from_numpy(rng.uniform(-1, 1, bc_dofs.numel())).cuda())
    A, b = elasticity.assemble_interface_elasticity(plan, phi, f, elasticity.Material(1.0, 0.3, 0.05, 0.27),
                                                    pen_coef=1.3, stab_coef=0.7, bcs=bcs)
    S = System(A.indptr.cpu().numpy(), A.indices.cpu().numpy(), A.data.cpu().numpy())
    return S, b.cpu().numpy()[S.rows]


@pytest.mark.gpu
def test_elasticity_product_and_one_iteration_match_reference():
    """The real wide-row operator: the product and one fused iteration (from the start and after one iteration) against
    the reference.  Convergence of BiCGStab on it is not asserted (the demo solves it directly)."""
    S, b = _elasticity_system()
    shape = launch_shape(S.n_act, S.nnz)
    print("interface elasticity: n_act %d, nnz %d, (lanes, grid, vector grid, passes) %s" % (S.n_act, S.nnz, shape))
    D = Device(S)
    x = np.zeros(S.n_act + 1)
    x[:-1] = np.random.default_rng(4).uniform(-1, 1, S.n_act)
    y = torch.full((S.n_act + 1,), float("nan"), dtype=torch.float64, device="cuda")
    partials = D.partials()
    xd = _d(x)
    D.spmv_rows(xd, y, partials)
    _check_product(S, x, y.cpu().numpy(), partials.cpu().numpy(), x)
    for k in (0, 1):
        _, cap, after = _step_case(S, k, b)
        _compare_step(S, cap, after)


# ---- C ABI refusals: argument checks fire before any launch, so these need no GPU --------------------------------------
def _host_buffers():
    keep = [(ctypes.c_double * 64)() for _ in range(4)] + [(ctypes.c_int32 * 64)() for _ in range(3)]
    return keep, [ctypes.addressof(b) for b in keep]


def test_solve_entry_points_refuse_null_pointers():
    lib = _lib.load()
    keep, (d0, d1, d2, d3, i0, i1, i2) = _host_buffers()

    def refused(rc):
        return rc == -1 and b"null" in lib.phifem_last_error()

    args = [i0, i1, d0, d1, d2]
    for j in range(len(args)):
        a = list(args)
        a[j] = None
        assert refused(lib.phifem_csr_spmv(4, *a, None)), j
    args = [i0, i1, d0, d1, d2]
    for j in range(len(args)):
        a = list(args)
        a[j] = None
        assert refused(lib.phifem_csr_row_scan(4, *a, None)), j
    args = [i0, i1, i2]
    for j in range(len(args)):
        a = list(args)
        a[j] = None
        assert refused(lib.phifem_remap_columns(4, *a, None)), j
    args = [i0, i1, i2, d0, d1, d2, d3]
    for j in range(len(args)):
        a = list(args)
        a[j] = None
        assert refused(lib.phifem_csr_spmv_rows(4, 16, *a, None)), j
    args = [i0, i1, i2] + [d0] * 13
    n_partials = ctypes.c_int32(1)
    for j in range(len(args)):
        a = list(args)
        a[j] = None
        assert refused(lib.phifem_bicgstab_iterate(4, 16, *a, ctypes.byref(n_partials), 1, None)), j
    assert refused(lib.phifem_bicgstab_iterate(4, 16, *args, None, 1, None))
    del keep


def test_solve_entry_points_accept_empty_systems():
    lib = _lib.load()
    keep, (d0, d1, d2, d3, i0, i1, i2) = _host_buffers()
    assert lib.phifem_csr_spmv(0, i0, None, None, d0, d1, None) == 0
    assert lib.phifem_csr_row_scan(0, None, None, None, None, None, None) == 0
    assert lib.phifem_remap_columns(0, None, None, None, None) == 0
    assert lib.phifem_csr_spmv_rows(0, 0, None, None, None, None, None, None, None, None) == 0
    del keep


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["L8-single", "L4-strided"])
def test_iterate_refuses_n_partials_out_of_range(name):
    """*n_partials of 0 or above the product grid + vector grid is refused before any launch (the buffers here are large
    enough that a missing check would read only initialised memory)."""
    S = system(name)
    D = Device(S)
    _, grid, vgrid, _ = launch_shape(S.n_act, S.nnz)
    b, _ = initial_state(S, seed=1)
    for bad in (0, -1, grid + vgrid + 1):
        V = D.start(b)
        V["partials"].zero_()
        before = Device.snapshot(V)
        V["n_partials"].value = bad
        assert D.iterate(V, 1) == -1 and b"n_partials" in _lib.load().phifem_last_error()
        assert V["n_partials"].value == bad
        after = Device.snapshot(V)
        for k in ("x", "r", "state"):
            assert np.array_equal(before[k], after[k]), k
