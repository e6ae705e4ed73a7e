"""Iterative solve on the assembled CSR system (SURVEY.md 8(f).1).

The reference solves `A[inner, inner] x = b[inner]` with a dense `torch.linalg.solve`
(basis/abstract_basis.py:177-195), which cannot exist once the matrix is only representable as
CSR (config 2: 2.1 M unknowns).  Here the same reduced system is solved by Jacobi-preconditioned
conjugate gradients on the full-length vectors with the non-interior rows and columns masked out;
one iteration is three hand-written kernels (`tfem_cg_iteration`: SpMV + p.Ap, the vector updates
+ r.z, the new direction) with every dot product reduced in a fixed order and the scalars kept on
the device; the host looks at the residual only every `check_every` iterations.

`amg()` builds a smoothed-aggregation algebraic multigrid hierarchy once, on the device, and
`preconditioner=` replaces Jacobi by one V-cycle of it per iteration (`tfem_pcg_iteration`); the
Gram matrix of a training loop is fixed, so one hierarchy serves every step (DESIGN.md §8(f).1).
`amg(..., refreshable=True)` also keeps the symbolic data for `AmgHierarchy.refresh`, which recomputes
every value for a new matrix on the same pattern without re-aggregating (moving meshes, K + beta M).
"""

from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import torch

from . import ops


@dataclass
class CgInfo:
    iterations: int
    relative_residual: float
    converged: bool


def csr_diagonal(crow: torch.Tensor, col: torch.Tensor, val: torch.Tensor) -> torch.Tensor:
    """Diagonal of a CSR matrix (zeros where a row stores no diagonal entry)."""
    n = crow.shape[0] - 1
    counts = (crow[1:] - crow[:-1]).long()
    row_of = torch.repeat_interleave(torch.arange(n, device=col.device), counts)
    on_diag = col.long() == row_of
    diag = torch.zeros(n, dtype=val.dtype, device=val.device)
    diag[row_of[on_diag]] = val[on_diag]
    return diag


def cg(
    crow: torch.Tensor,
    col: torch.Tensor,
    val: torch.Tensor,
    rhs: torch.Tensor,
    keep: Optional[torch.Tensor] = None,
    x0: Optional[torch.Tensor] = None,
    rtol: float = 1e-10,
    max_iterations: Optional[int] = None,
    check_every: Optional[int] = None,
    use_graph: bool = True,
    fused: bool = True,
    preconditioner: Optional["AmgHierarchy"] = None,
):
    """Solve `(M A M) x = M rhs` for symmetric positive definite `M A M`, `M = diag(keep)`.

    crow/col int32, val/rhs float; keep bool/uint8 of length n or None (every row).  Returns
    `(x, CgInfo)`; x is zero where keep is 0.  On CUDA one iteration is captured in a CUDA graph
    and replayed (`use_graph=False` keeps the eager loop); `fused=False` uses torch vector
    updates around `tfem_csr_spmv` instead of the three-kernel `tfem_cg_iteration`.

    `preconditioner`: an `amg()` hierarchy of this matrix and keep mask (ValueError otherwise) replaces Jacobi by one
    V-cycle per iteration (`tfem_pcg_iteration`).  The residual is checked every `check_every` iterations: 50 with
    Jacobi, every iteration with AMG (which needs tens of iterations, not thousands)."""
    n = crow.shape[0] - 1
    b = rhs.reshape(-1).to(device=val.device, dtype=val.dtype)
    if b.shape[0] != n:
        raise ValueError("right-hand side length does not match the matrix")
    keep8 = None
    if keep is not None:
        keep8 = keep.reshape(-1).to(device=val.device, dtype=torch.uint8).contiguous()
        b = b * keep8.to(val.dtype)
    if preconditioner is not None:
        preconditioner.check(crow, val, keep8)
        inv_diag = None
    else:
        diag = csr_diagonal(crow, col, val)
        inv_diag = torch.where(diag != 0, 1.0 / diag, torch.ones_like(diag))
    if check_every is None:
        check_every = 50 if preconditioner is None else 1
    x = torch.zeros_like(b) if x0 is None else x0.reshape(-1).to(device=val.device, dtype=val.dtype).clone()
    if keep8 is not None:
        x = x * keep8.to(val.dtype)
    r = b - ops.csr_spmv(crow, col, val, x, keep8) if x0 is not None else b.clone()
    z = r * inv_diag if preconditioner is None else ops.amg_vcycle(preconditioner, r)
    p = z.clone()
    ap = torch.empty_like(p)
    rz = torch.dot(r, z).reshape(1)
    b_norm = float(torch.linalg.vector_norm(b))
    if b_norm == 0.0:
        return x, CgInfo(0, 0.0, True)
    # Conjugate gradients converge in at most n steps in exact arithmetic; 2 n + 100 leaves room for rounding
    # without turning a breakdown into millions of graph replays
    limit = max_iterations if max_iterations is not None else 2 * n + 100
    initial = float(torch.linalg.vector_norm(r)) / b_norm
    if initial <= rtol or limit <= 0:  # e.g. a converged x0: nothing to iterate
        return x, CgInfo(0, initial, initial <= rtol)
    tiny = torch.finfo(val.dtype).tiny
    spmv = getattr(ops, "csr_spmv_raw", None) if val.is_cuda else None

    def iteration():  # every tensor it touches is preallocated: one CUDA graph replays it
        if spmv is not None:
            spmv(crow, col, val, p, keep8, ap)
        else:
            ap.copy_(ops.csr_spmv(crow, col, val, p, keep8))
        alpha = rz / torch.dot(p, ap).clamp_min(tiny)
        x.addcmul_(p, alpha)
        r.addcmul_(ap, alpha, value=-1.0)
        if preconditioner is None:
            torch.mul(r, inv_diag, out=z)
        elif val.is_cuda:
            ops.amg_vcycle_raw(preconditioner, r, z)
        else:
            z.copy_(ops.amg_vcycle(preconditioner, r))
        rz_new = torch.dot(r, z).reshape(1)
        p.mul_(rz_new / rz.clamp_min(tiny)).add_(z)
        rz.copy_(rz_new)

    fused_step = getattr(ops, "cg_iteration_raw", None) if (val.is_cuda and fused) else None
    if fused_step is not None and preconditioner is not None:
        # five launch groups per iteration (tfem_pcg_iteration): SpMV + p.Ap | x, r updates | V-cycle | r.z | new direction
        blocks = 8 * torch.cuda.get_device_properties(val.device).multi_processor_count
        partial = torch.zeros(2 * blocks, dtype=val.dtype, device=val.device)
        scal = torch.cat([rz, rz]).contiguous()

        def iteration():  # noqa: F811
            ops.pcg_iteration_raw(crow, col, val, keep8, preconditioner, x, r, z, p, ap, partial, scal)

    elif fused_step is not None:
        # three launches per iteration (tfem_cg_iteration): SpMV + p.Ap | x, r, z updates + r.z | new direction
        blocks = 8 * torch.cuda.get_device_properties(val.device).multi_processor_count
        partial = torch.zeros(2 * blocks, dtype=val.dtype, device=val.device)
        scal = torch.cat([rz, rz]).contiguous()
        inv_diag = inv_diag.contiguous()

        def iteration():  # noqa: F811
            fused_step(crow, col, val, keep8, inv_diag, x, r, z, p, ap, partial, scal)

    step = iteration
    iterations = 0
    if val.is_cuda and use_graph:
        # the loop is launch-bound (a dozen small kernels per iteration): capture one iteration
        side = torch.cuda.Stream(device=val.device)
        side.wait_stream(torch.cuda.current_stream(val.device))
        with torch.cuda.stream(side):
            warm = min(3, limit)  # warm-up outside capture (allocator, lazy module loading); they are real iterations
            for _ in range(warm):
                iteration()
            iterations = warm
        torch.cuda.current_stream(val.device).wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):  # records the launches, does not run them
            iteration()
        step = graph.replay
    rel = float("inf")
    best, stalled = initial, 0
    while iterations < limit:
        step()
        iterations += 1
        if iterations % check_every == 0 or iterations >= limit:
            rel = float(torch.linalg.vector_norm(r)) / b_norm  # the only host synchronisation
            if rel <= rtol:
                break
            # breakdown: a non-SPD or singular reduced system gives p.Ap <= 0 and then inf / NaN, or a residual
            # that no longer decreases; stop and report instead of replaying to the iteration limit
            if rel != rel or rel == float("inf"):
                break
            if rel < 0.999 * best:
                best, stalled = rel, 0
            else:
                stalled += 1
                if stalled >= 20:
                    break
    if rel == float("inf") and iterations > 0:
        rel = float(torch.linalg.vector_norm(r)) / b_norm
    converged = rel == rel and rel <= rtol
    return x, CgInfo(iterations, rel, converged)


# ------------------------------------------------------------------------------------------------
# smoothed-aggregation AMG preconditioner
# ------------------------------------------------------------------------------------------------

POWER_ITERATIONS = 15
POWER_SALT = 0x10000  # hash salt of the power-iteration start vector (+ level); oracle/amg_oracle.py uses the same
MAX_DENSE_COARSE = 32768  # the coarsest operator is inverted densely (tfem_amg_vcycle's limit)


@dataclass
class AmgLevel:
    """One smoothed level: operator A, prolongator P, restriction R = P^T (CSR), omega D^-1 and work vectors."""

    n: int
    n_coarse: int
    a_crow: torch.Tensor
    a_col: torch.Tensor
    a_val: torch.Tensor
    p_crow: torch.Tensor
    p_col: torch.Tensor
    p_val: torch.Tensor
    r_crow: torch.Tensor
    r_col: torch.Tensor
    r_val: torch.Tensor
    wdinv: torch.Tensor
    agg: torch.Tensor
    rho: float
    omega: float
    x: torch.Tensor = field(init=False)
    rc: torch.Tensor = field(init=False)
    ec: torch.Tensor = field(init=False)

    def __post_init__(self):
        self.x = torch.zeros_like(self.wdinv)
        self.rc = self.wdinv.new_zeros(self.n_coarse)
        self.ec = self.wdinv.new_zeros(self.n_coarse)


@dataclass
class AmgLevelPattern:
    """What a refresh of one level needs beyond the level itself: the tentative prolongator T (its values depend only on
    the aggregates), the pattern and values of the intermediate A P, and r_map (R entry k is P entry r_map[k])."""

    t_crow: torch.Tensor
    t_col: torch.Tensor
    t_val: torch.Tensor
    ap_crow: torch.Tensor
    ap_col: torch.Tensor
    ap_val: torch.Tensor
    r_map: torch.Tensor


@dataclass
class AmgPattern:
    """The symbolic data of a refreshable hierarchy: the input pattern it was built for, the gather map src from input
    values to the finest operator (M A M) + (I - M) (-1: a masked diagonal, set to 1), each level's AmgLevelPattern and
    the coarsest operator as CSR."""

    crow: torch.Tensor
    col: torch.Tensor
    src: torch.Tensor
    levels: List[AmgLevelPattern]
    coarse_crow: torch.Tensor
    coarse_col: torch.Tensor
    coarse_val: torch.Tensor

    def tensors(self) -> List[torch.Tensor]:
        out = [self.crow, self.col, self.src, self.coarse_crow, self.coarse_col, self.coarse_val]
        for lev in self.levels:
            out += [lev.t_crow, lev.t_col, lev.t_val, lev.ap_crow, lev.ap_col, lev.ap_val, lev.r_map]
        return out


@dataclass
class AmgHierarchy:
    """The hierarchy `amg()` builds for one matrix and keep mask; pass it as `preconditioner=`.

    levels: the smoothed levels, finest first; coarse_inv: dense inverse of the coarsest operator."""

    levels: List[AmgLevel]
    coarse_inv: torch.Tensor
    coarse_nnz: int
    keep: torch.Tensor  # uint8 [n] (ones when built without a mask)
    nnz: int
    theta: float
    _struct: object = field(default=None, repr=False)
    pattern: Optional[AmgPattern] = field(default=None, repr=False)  # amg(..., refreshable=True) only

    @property
    def n(self) -> int:
        return self.levels[0].n if self.levels else self.coarse_inv.shape[0]

    @property
    def dtype(self) -> torch.dtype:
        return self.coarse_inv.dtype

    @property
    def device(self) -> torch.device:
        return self.coarse_inv.device

    @property
    def grid_sizes(self) -> List[int]:
        return [lev.n for lev in self.levels] + [self.coarse_inv.shape[0]]

    @property
    def operator_complexity(self) -> float:
        """Stored entries of every level's operator over those of the finest."""
        total = sum(lev.a_col.shape[0] for lev in self.levels) + self.coarse_nnz
        return total / (self.levels[0].a_col.shape[0] if self.levels else max(self.coarse_nnz, 1))

    @property
    def rho(self) -> List[float]:
        return [lev.rho for lev in self.levels]

    @property
    def omega(self) -> List[float]:
        return [lev.omega for lev in self.levels]

    @property
    def struct(self):
        """The host array of struct tfem_amg_level the V-cycle entry points read."""
        if self._struct is None:
            self._struct = ops.amg_levels_struct(self)
        return self._struct

    def summary(self) -> str:
        rows = ", ".join(f"{n}" for n in self.grid_sizes)
        rho = ", ".join(f"{r:.4f}" for r in self.rho)
        return (f"{len(self.grid_sizes)} levels (rows {rows}), operator complexity {self.operator_complexity:.3f}, "
                f"theta {self.theta}, rho(D^-1 A) per level [{rho}]")

    def check(self, crow: torch.Tensor, val: torch.Tensor, keep8: Optional[torch.Tensor]) -> None:
        """ValueError unless this hierarchy was built for a matrix of this size, nnz, dtype and device and this keep mask."""
        n = crow.shape[0] - 1
        if n != self.n or val.shape[0] != self.nnz or val.dtype != self.dtype or val.device != self.device:
            raise ValueError(f"the AMG hierarchy was built for a {self.n}-row {self.dtype} matrix with {self.nnz} entries on {self.device}, "
                             f"not for this {n}-row {val.dtype} matrix with {val.shape[0]} entries on {val.device}")
        keep = torch.ones(n, dtype=torch.uint8, device=val.device) if keep8 is None else keep8
        if not torch.equal(keep, self.keep):
            raise ValueError("the AMG hierarchy was built for another keep mask")

    def refresh(self, matrix: torch.Tensor) -> "AmgHierarchy":
        """Recompute every value of this hierarchy for new matrix values on the pattern it was built from; returns self.

        `matrix`: a sparse CSR tensor with the built pattern, or a 1-D array of values aligned with it (like
        `layout="values"`).  The aggregates, the keep mask and every sparsity pattern stay; per level the operator, its
        diagonal, rho (the same power iteration as the build), omega, omega D^-1, P = (I - omega D^-1 A) T, R = P^T, A P
        and A_c are recomputed, then the dense coarsest inverse.  Every device tensor keeps its storage, so the
        hierarchy stays valid wherever it is already passed as `preconditioner=`.  A refresh with the matrix of the
        build reproduces the build bit for bit.

        It does not re-aggregate: when the strength pattern of the new matrix differs completely (e.g. another
        anisotropy), build a new hierarchy instead.  A hierarchy refreshed between the forward and the backward of
        `solve` preconditions the adjoint solve with the new values; that solve still converges to the adjoint of the
        saved matrix, which it multiplies by.

        ValueError, with nothing modified, for a hierarchy built without `refreshable=True`, a matrix of another size,
        nnz, dtype, device or pattern, or a value array of the wrong length."""
        pat = self.pattern
        if pat is None:
            raise ValueError("the AMG hierarchy was not built with refreshable=True")
        if isinstance(matrix, torch.Tensor) and matrix.layout == torch.sparse_csr:
            crow, col, val = matrix.crow_indices(), matrix.col_indices(), matrix.values()
            self.check(crow, val, self.keep)
            if not (torch.equal(crow.to(torch.int32), pat.crow) and torch.equal(col.to(torch.int32), pat.col)):
                raise ValueError("the matrix has another sparsity pattern than the AMG hierarchy was built for")
        else:
            val = matrix
            if val.dim() != 1 or val.shape[0] != self.nnz or val.dtype != self.dtype or val.device != self.device:
                raise ValueError(f"a value array of the AMG hierarchy is a 1-D {self.dtype} tensor of {self.nnz} entries on {self.device}, "
                                 f"not a {val.dim()}-D {val.dtype} tensor of shape {tuple(val.shape)} on {val.device}")
        val = val.contiguous()
        missing = torch.zeros(1, dtype=torch.int32, device=self.device)
        ops.gather_fill(pat.src, val, 1.0, self.levels[0].a_val if self.levels else pat.coarse_val)
        for level, (lev, lp) in enumerate(zip(self.levels, pat.levels)):
            a = (lev.a_crow, lev.a_col, lev.a_val)
            diag = ops.amg_diag(*a)
            rho = _spectral_radius(*a, 1.0 / diag, level)
            omega = 4.0 / (3.0 * rho)
            s_val = torch.empty_like(lev.a_val)
            ops.amg_smoother(*a, diag, omega, lev.wdinv, s_val)
            p = (lev.p_crow, lev.p_col, lev.p_val)
            ops.csr_spgemm_numeric((lev.a_crow, lev.a_col, s_val), (lp.t_crow, lp.t_col, lp.t_val), lev.p_crow, lev.p_col, lev.p_val, missing)
            ops.gather_fill(lp.r_map, lev.p_val, 0.0, lev.r_val)
            ops.csr_spgemm_numeric(a, p, lp.ap_crow, lp.ap_col, lp.ap_val, missing)
            nxt = self.levels[level + 1] if level + 1 < len(self.levels) else None
            c = (nxt.a_crow, nxt.a_col, nxt.a_val) if nxt is not None else (pat.coarse_crow, pat.coarse_col, pat.coarse_val)
            ops.csr_spgemm_numeric((lev.r_crow, lev.r_col, lev.r_val), (lp.ap_crow, lp.ap_col, lp.ap_val), c[0], c[1], c[2], missing)
            lev.rho, lev.omega = rho, omega
        self.coarse_inv.copy_(_dense_inverse(pat.coarse_crow, pat.coarse_col, pat.coarse_val))
        if int(missing.item()) != 0:  # the patterns are those of the build: a product outside them is an internal error
            raise RuntimeError(f"AMG refresh: {int(missing.item())} products fell outside the hierarchy's patterns")
        return self


def _hash32(i: torch.Tensor, salt: int) -> torch.Tensor:
    """oracle/amg_oracle.py hash32 in int64 arithmetic (products wrap; the low 32 bits are exact)."""
    m = 0xFFFFFFFF
    h = (i * 0x9E3779B1 + (salt * 0x85EBCA77 + 0x165667B1)) & m
    h = h ^ (h >> 16)
    h = (h * 0x85EBCA6B) & m
    h = h ^ (h >> 13)
    h = (h * 0xC2B2AE35) & m
    return h ^ (h >> 16)


def _masked_operator(crow, col, val, keep8):
    """(M A M) + (I - M): masked rows and columns dropped, their diagonals set to 1."""
    if keep8 is None:
        return crow, col, val.clone()
    n = crow.shape[0] - 1
    row = torch.repeat_interleave(torch.arange(n, device=col.device), (crow[1:] - crow[:-1]).long())
    k = keep8 != 0
    on_diag = row == col.long()
    live = (k[row] & k[col.long()]) | on_diag
    v = torch.where(on_diag & ~k[row], torch.ones_like(val), val)
    counts = torch.bincount(row[live], minlength=n)
    new_crow = torch.cat([counts.new_zeros(1), torch.cumsum(counts, 0)]).to(torch.int32)
    return new_crow, col[live].contiguous(), v[live].contiguous()


def _masked_operator_map(crow, col, keep8):
    """src [nnz of the masked operator]: the input entry each entry of `_masked_operator` takes (-1: a masked
    diagonal, which is 1)."""
    index = torch.arange(col.shape[0], dtype=torch.int32, device=col.device)
    if keep8 is None:
        return index
    n = crow.shape[0] - 1
    row = torch.repeat_interleave(torch.arange(n, device=col.device), (crow[1:] - crow[:-1]).long())
    k = keep8 != 0
    on_diag = row == col.long()
    live = (k[row] & k[col.long()]) | on_diag
    src = torch.where(on_diag & ~k[row], torch.full_like(index, -1), index)
    return src[live].contiguous()


def _transpose_map(p_crow, p_col):
    """r_map: R = P^T entry k is P entry r_map[k] (a stable sort of P's (column, row) keys, R's CSR order)."""
    n = p_crow.shape[0] - 1
    row = torch.repeat_interleave(torch.arange(n, device=p_col.device), (p_crow[1:] - p_crow[:-1]).long())
    key = p_col.long() * n + row
    return torch.argsort(key, stable=True).to(torch.int32)


def _dense_inverse(a_crow, a_col, a_val):
    n_c = a_crow.shape[0] - 1
    dense = torch.zeros((n_c, n_c), dtype=a_val.dtype, device=a_val.device)
    dense[torch.repeat_interleave(torch.arange(n_c, device=a_val.device), (a_crow[1:] - a_crow[:-1]).long()), a_col.long()] = a_val
    return torch.linalg.inv(dense).contiguous()


def _spectral_radius(crow, col, val, inv_diag, level: int) -> float:
    """rho(D^-1 A) by power iteration from a hash-generated (reproducible) start vector."""
    n = crow.shape[0] - 1
    v = _hash32(torch.arange(n, device=val.device), POWER_SALT + level).to(val.dtype) / 4294967296.0 - 0.5
    rho = None
    for _ in range(POWER_ITERATIONS):
        w = inv_diag * ops.csr_spmv(crow, col, val, v)
        nw = torch.linalg.vector_norm(w)
        rho = nw / torch.linalg.vector_norm(v)
        v = w / nw
    return float(rho)


def amg(matrix: torch.Tensor, keep: Optional[torch.Tensor] = None, theta: float = 0.08, max_coarse: int = 1000,
        max_levels: int = 12, refreshable: bool = False) -> AmgHierarchy:
    """Smoothed-aggregation AMG hierarchy of the operator `cg` solves, (M A M) + (I - M), M = diag(keep), for a
    symmetric positive definite CSR `matrix`; one-time set-up on the device.

    Per level: strength |a_ij| >= theta sqrt(|a_ii a_jj|); aggregates by parallel MIS(2); tentative prolongator
    T = 1 / sqrt(|aggregate|) (nodes without strong connections stay unaggregated: the smoother alone handles them);
    rho(D^-1 A) by 15 power iterations; P = (I - omega D^-1 A) T, omega = 4 / (3 rho); R = P^T; A_c = R A P by the
    deterministic SpGEMM.  Coarsening stops at <= max_coarse rows or max_levels levels; the coarsest operator is
    inverted densely.  The result is reproducible run to run.

    `refreshable=True` also keeps what `AmgHierarchy.refresh` needs to recompute the values for a new matrix on the same
    pattern (the finest gather map, T, the pattern of A P and the R-from-P map per level, the coarsest pattern); the
    hierarchy itself is the same bit for bit."""
    crow, col, val = matrix.crow_indices().to(torch.int32), matrix.col_indices().to(torch.int32), matrix.values()
    n = crow.shape[0] - 1
    keep8 = None if keep is None else keep.reshape(-1).to(device=val.device, dtype=torch.uint8).contiguous()
    if keep8 is not None and keep8.shape[0] != n:
        raise ValueError("keep mask length does not match the matrix")
    a = _masked_operator(crow, col, val, keep8)
    levels: List[AmgLevel] = []
    patterns: List[AmgLevelPattern] = []
    while a[0].shape[0] - 1 > max_coarse and len(levels) + 1 < max_levels:
        level = len(levels)
        a_crow, a_col, a_val = a
        n_l = a_crow.shape[0] - 1
        diag, strong = ops.amg_strength(a_crow, a_col, a_val, theta)
        agg, n_agg = ops.amg_aggregate(a_crow, a_col, strong, level)
        if n_agg == 0 or n_agg >= n_l:
            break  # nothing left to coarsen: this operator is the coarsest
        live = agg >= 0
        size = torch.bincount(agg[live].long(), minlength=n_agg)
        t_crow = torch.cat([size.new_zeros(1), torch.cumsum(live.long(), 0)]).to(torch.int32)
        t_col = agg[live].contiguous()
        t_val = (1.0 / torch.sqrt(size[t_col.long()].to(a_val.dtype))).contiguous()
        inv_diag = 1.0 / diag
        rho = _spectral_radius(a_crow, a_col, a_val, inv_diag, level)
        omega = 4.0 / (3.0 * rho)
        wdinv = (omega / diag).contiguous()
        row = torch.repeat_interleave(torch.arange(n_l, device=a_val.device), (a_crow[1:] - a_crow[:-1]).long())
        s_val = ((row == a_col.long()).to(a_val.dtype) - wdinv[row] * a_val).contiguous()
        p = ops.csr_spgemm((a_crow, a_col, s_val), n_l, (t_crow, t_col, t_val), n_agg)
        r = ops.csr_spgemm(p, n_agg, transpose=True)
        ap = ops.csr_spgemm(a, n_l, p, n_agg)
        a_c = ops.csr_spgemm(r, n_l, ap, n_agg)
        levels.append(AmgLevel(n_l, n_agg, a_crow, a_col, a_val, *p, *r, wdinv, agg, rho, omega))
        if refreshable:
            r_map = _transpose_map(p[0], p[1])
            if not torch.equal(p[2][r_map.long()].view(_bits(p[2].dtype)), r[2].view(_bits(r[2].dtype))):
                raise RuntimeError("AMG set-up: R is not P^T gathered through the transpose map")
            patterns.append(AmgLevelPattern(t_crow, t_col, t_val, ap[0], ap[1], ap[2], r_map))
        a = a_c
    a_crow, a_col, a_val = a
    n_c = a_crow.shape[0] - 1
    if n_c > MAX_DENSE_COARSE:
        raise ValueError(f"coarsening stopped at {n_c} rows, more than the dense coarsest solve takes ({MAX_DENSE_COARSE}); "
                         "raise max_levels or lower theta")
    coarse_inv = _dense_inverse(a_crow, a_col, a_val)
    keep_all = torch.ones(n, dtype=torch.uint8, device=val.device) if keep8 is None else keep8.clone()
    pattern = None
    if refreshable:
        pattern = AmgPattern(crow, col, _masked_operator_map(crow, col, keep8), patterns, a_crow, a_col, a_val)
    return AmgHierarchy(levels, coarse_inv, a_col.shape[0], keep_all, val.shape[0], theta, pattern=pattern)


def _bits(dtype: torch.dtype) -> torch.dtype:
    return torch.int64 if dtype == torch.float64 else torch.int32


class _CgSolve(torch.autograd.Function):
    """x = (M A M)^-1 M b through `cg`, differentiable w.r.t. b: for symmetric A the adjoint is one more solve,
    b_bar = (M A M)^-1 M x_bar (the matrix is a constant of the optimisation, as the Gram matrix of
    examples/example_weak.py:84-86 is)."""

    @staticmethod
    def forward(ctx, b, crow, col, val, keep, rtol, max_iterations, preconditioner):
        x, info = cg(crow, col, val, b.detach(), keep, rtol=rtol, max_iterations=max_iterations, preconditioner=preconditioner)
        if not info.converged:
            raise RuntimeError(f"conjugate gradients stopped at relative residual {info.relative_residual:.3e} after {info.iterations} iterations")
        ctx.save_for_backward(crow, col, val)
        ctx.keep, ctx.rtol, ctx.max_iterations, ctx.shape = keep, rtol, max_iterations, b.shape
        ctx.preconditioner = preconditioner
        ctx.info = info
        return x.reshape(b.shape)

    @staticmethod
    def backward(ctx, x_bar):
        crow, col, val = ctx.saved_tensors
        if not bool(x_bar.any()):
            return torch.zeros(ctx.shape, dtype=x_bar.dtype, device=x_bar.device), None, None, None, None, None, None, None
        b_bar, info = cg(crow, col, val, x_bar.detach(), ctx.keep, rtol=ctx.rtol, max_iterations=ctx.max_iterations,
                         preconditioner=ctx.preconditioner)
        if not info.converged:
            raise RuntimeError(f"adjoint conjugate gradients stopped at relative residual {info.relative_residual:.3e}")
        return b_bar.reshape(ctx.shape), None, None, None, None, None, None, None


def solve(matrix: torch.Tensor, rhs: torch.Tensor, keep: Optional[torch.Tensor] = None, rtol: float = 1e-10,
          max_iterations: Optional[int] = None, preconditioner: Optional[AmgHierarchy] = None) -> torch.Tensor:
    """`A^-1 rhs` for a symmetric positive definite CSR matrix (rows / columns with keep == 0 masked out), usable inside
    a loss: gradients flow to `rhs` through a second conjugate-gradient solve.  `preconditioner`: an `amg(matrix, keep)`
    hierarchy, used by both solves."""
    return _CgSolve.apply(rhs, matrix.crow_indices().to(torch.int32), matrix.col_indices().to(torch.int32), matrix.values(), keep,
                          rtol, max_iterations, preconditioner)


class _QuadraticForm(torch.autograd.Function):
    """r^T A^-1 r with ONE solve for value and gradient: d/dr = 2 A^-1 r for symmetric A."""

    @staticmethod
    def forward(ctx, r, crow, col, val, keep, rtol, max_iterations, preconditioner):
        x, info = cg(crow, col, val, r.detach(), keep, rtol=rtol, max_iterations=max_iterations, preconditioner=preconditioner)
        if not info.converged:
            raise RuntimeError(f"conjugate gradients stopped at relative residual {info.relative_residual:.3e} after {info.iterations} iterations")
        x = x.reshape(r.shape)
        ctx.save_for_backward(x)
        masked = r.detach() if keep is None else r.detach() * keep.reshape(r.shape).to(r.dtype)
        return (masked * x).sum()

    @staticmethod
    def backward(ctx, loss_bar):
        (x,) = ctx.saved_tensors
        return 2.0 * loss_bar * x, None, None, None, None, None, None, None


def inverse_quadratic_form(matrix: torch.Tensor, residual: torch.Tensor, keep: Optional[torch.Tensor] = None, rtol: float = 1e-10,
                           max_iterations: Optional[int] = None, preconditioner: Optional[AmgHierarchy] = None) -> torch.Tensor:
    """The robust-VPINN loss `r^T G^-1 r` of examples/example_weak.py:84-86,138 on a CSR Gram matrix that cannot be
    inverted densely: one conjugate-gradient solve gives the value and, since G is symmetric, the gradient 2 G^-1 r.
    `preconditioner`: an `amg(matrix, keep)` hierarchy, built once and reused every training step."""
    return _QuadraticForm.apply(residual, matrix.crow_indices().to(torch.int32), matrix.col_indices().to(torch.int32), matrix.values(),
                                keep, rtol, max_iterations, preconditioner)
