"""torch.library custom ops over the C ABI of include/tfem_b200.h.

Each op allocates its outputs with torch (device memory is torch's job), passes raw device
pointers and the current CUDA stream to the C entry point, and raises on any failure.
There is no CPU implementation: calling an op with CPU tensors raises `TfemError`.

Differentiable ops (`quad_reduce`, `scatter`, `weak_residual`) register their adjoints, which
are again C-ABI kernels, so `loss.backward()` of the VPINN examples
(reference model/model.py:61-67 over examples/example_weak.py:132-152) stays on the CUDA path.
"""

from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import Bilinear, TfemError, call, check_cuda, make_source, ptr

NS = "tfem_b200"

TRI_NQ = {1: 1, 2: 3, 3: 4, 4: 6}
LINE_NQ = {2: 2, 3: 3}


def _nq_tri(order: int) -> int:
    if order not in TRI_NQ:
        raise NotImplementedError("Integration order not implemented")
    return TRI_NQ[order]


def _i32(t: Tensor) -> Tensor:
    return t if t.dtype == torch.int32 else t.to(torch.int32)


# ------------------------------------------------------------------------------------------------
# geometry (not differentiable: mesh coordinates are data)
# ------------------------------------------------------------------------------------------------


@torch.library.custom_op(f"{NS}::tri_geometry", mutates_args=())
def tri_geometry(
    coords: Tensor,
    conn: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """coords (V,2), conn (N,3) int32 -> inv_jac (N,2,d), v_grad (N,3,d), x_q (N,q,d), dx (N,q)."""
    device = check_cuda(coords, conn, frac_jac, frac_inv, frac_det, frac_t)
    n_q = _nq_tri(quad_order)
    n_el = conn.shape[0]
    d = 3 if frac_jac is not None else 2
    opts = dict(dtype=coords.dtype, device=device)
    inv_jac = torch.empty((n_el, 2, d), **opts)
    v_grad = torch.empty((n_el, 3, d), **opts)
    x_q = torch.empty((n_el, n_q, d), **opts)
    dx = torch.empty((n_el, n_q), **opts)
    call(
        "tfem_tri_p1_geometry", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
        quad_order, ptr(frac_jac), ptr(frac_inv), ptr(frac_det), ptr(frac_t), ptr(inv_jac), ptr(v_grad), ptr(x_q), ptr(dx),
    )
    return inv_jac, v_grad, x_q, dx


@tri_geometry.register_fake
def _(coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    n_el, n_q = conn.shape[0], TRI_NQ[quad_order]
    d = 3 if frac_jac is not None else 2
    return (coords.new_empty((n_el, 2, d)), coords.new_empty((n_el, 3, d)), coords.new_empty((n_el, n_q, d)), coords.new_empty((n_el, n_q)))


@torch.library.custom_op(f"{NS}::edge_geometry", mutates_args=())
def edge_geometry(
    edge_coords: Tensor,
    n_edge_per_mesh: int,
    quad_order: int,
    frac_jac: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """edge_coords (E,2,2) -> inv_jac (E,), v_grad (E,2), x_q (E,q,d), dx (E,q)."""
    device = check_cuda(edge_coords, frac_jac, frac_det, frac_t)
    if quad_order not in LINE_NQ:
        raise NotImplementedError("Integration order not implemented")
    n_q = LINE_NQ[quad_order]
    n_edge = edge_coords.shape[0]
    d = 3 if frac_jac is not None else 2
    opts = dict(dtype=edge_coords.dtype, device=device)
    inv_jac = torch.empty((n_edge,), **opts)
    v_grad = torch.empty((n_edge, 2), **opts)
    x_q = torch.empty((n_edge, n_q, d), **opts)
    dx = torch.empty((n_edge, n_q), **opts)
    call(
        "tfem_edge_p1_geometry", edge_coords.dtype, device, n_edge, n_edge_per_mesh, ptr(edge_coords), quad_order,
        ptr(frac_jac), ptr(frac_det), ptr(frac_t), ptr(inv_jac), ptr(v_grad), ptr(x_q), ptr(dx),
    )
    return inv_jac, v_grad, x_q, dx


@edge_geometry.register_fake
def _(edge_coords, n_edge_per_mesh, quad_order, frac_jac=None, frac_det=None, frac_t=None):
    n_edge, n_q = edge_coords.shape[0], LINE_NQ[quad_order]
    d = 3 if frac_jac is not None else 2
    return (edge_coords.new_empty((n_edge,)), edge_coords.new_empty((n_edge, 2)), edge_coords.new_empty((n_edge, n_q, d)), edge_coords.new_empty((n_edge, n_q)))


# ------------------------------------------------------------------------------------------------
# generic path: quadrature sum of a user integrand + deterministic scatter
# ------------------------------------------------------------------------------------------------


@torch.library.custom_op(f"{NS}::quad_reduce", mutates_args=())
def quad_reduce(integrand: Tensor, dx: Tensor) -> Tensor:
    """integrand (N,q|1,m) (a q-stride of 0 broadcasts), dx (N,q) -> (N,m): sum_q dx * f."""
    device = check_cuda(dx)
    if not integrand.is_cuda:
        raise TfemError("tfem_b200 kernels need CUDA tensors (there is no CPU fallback)")
    n_el, n_q = dx.shape
    m = integrand.shape[-1]
    if integrand.stride(-1) != 1 and m > 1:
        integrand = integrand.contiguous()
    stride_e = integrand.stride(0) if integrand.shape[0] > 1 else 0
    stride_q = integrand.stride(1) if integrand.shape[1] > 1 else 0
    if n_el > 1 and integrand.shape[0] == 1:
        stride_e = 0
    out = torch.empty((n_el, m), dtype=dx.dtype, device=device)
    call("tfem_quad_reduce", dx.dtype, device, n_el, n_q, m, ptr(integrand), stride_e, stride_q, ptr(dx), ptr(out))
    return out


@quad_reduce.register_fake
def _(integrand, dx):
    return dx.new_empty((dx.shape[0], integrand.shape[-1]))


def _quad_reduce_setup(ctx, inputs, output):
    integrand, dx = inputs
    ctx.save_for_backward(dx)
    ctx.shape = integrand.shape


def _quad_reduce_backward(ctx, grad_out):
    (dx,) = ctx.saved_tensors
    grad = dx.unsqueeze(-1) * grad_out.unsqueeze(1)  # (N,q,m)
    shape = ctx.shape
    if shape[1] == 1 and grad.shape[1] != 1:
        grad = grad.sum(1, keepdim=True)
    if shape[0] == 1 and grad.shape[0] != 1:
        grad = grad.sum(0, keepdim=True)
    return grad, None


quad_reduce.register_autograd(_quad_reduce_backward, setup_context=_quad_reduce_setup)


@torch.library.custom_op(f"{NS}::scatter", mutates_args=())
def scatter(local: Tensor, seg: Tensor, perm: Tensor, inverse: Tensor) -> Tensor:
    """out[p] = sum_{s in seg[p]:seg[p+1]} local.flat[perm[s]] in increasing s (deterministic).

    `inverse[k]` is the output entry that flat input k lands in (used by the adjoint)."""
    device = check_cuda(local, seg, perm)
    n_out = seg.shape[0] - 1
    out = torch.empty((n_out,), dtype=local.dtype, device=device)
    call("tfem_scatter_bilinear", local.dtype, device, n_out, ptr(seg), ptr(perm), ptr(local), ptr(out))
    return out


@scatter.register_fake
def _(local, seg, perm, inverse):
    return local.new_empty((seg.shape[0] - 1,))


@torch.library.custom_op(f"{NS}::gather", mutates_args=())
def gather(src: Tensor, idx: Tensor) -> Tensor:
    """buf[i] = src[idx[i]] (the interface pack kernel; also the adjoint of `scatter`)."""
    device = check_cuda(src, idx)
    out = torch.empty((idx.shape[0],), dtype=src.dtype, device=device)
    call("tfem_iface_pack", src.dtype, device, idx.shape[0], ptr(idx), ptr(src), ptr(out))
    return out


@gather.register_fake
def _(src, idx):
    return src.new_empty((idx.shape[0],))


def _scatter_setup(ctx, inputs, output):
    local, seg, perm, inverse = inputs
    ctx.save_for_backward(inverse)
    ctx.shape = local.shape


def _scatter_backward(ctx, grad_out):
    (inverse,) = ctx.saved_tensors
    return gather(grad_out.contiguous(), inverse).reshape(ctx.shape), None, None, None


scatter.register_autograd(_scatter_backward, setup_context=_scatter_setup)


@torch.library.custom_op(f"{NS}::unpack_add_", mutates_args=("dst",))
def unpack_add_(dst: Tensor, idx: Tensor, buf: Tensor) -> None:
    """dst[idx[i]] += buf[i] for unique idx (owner-side sum of interface rows)."""
    device = check_cuda(dst, idx, buf)
    call("tfem_iface_unpack_add", dst.dtype, device, idx.shape[0], ptr(idx), ptr(buf), ptr(dst))


def pack_into_raw(out: Tensor, src: Tensor, idx: Tensor) -> None:
    """out[i] = src[idx[i]] into a preallocated buffer: direct C-ABI call for per-step hot loops."""
    device = check_cuda(out, src, idx)
    call("tfem_iface_pack", src.dtype, device, idx.shape[0], ptr(idx), ptr(src), ptr(out))


def pack_after_raw(out: Tensor, src: Tensor, idx: Tensor, progress: Tensor, target: int) -> None:
    """`pack_into_raw` that starts early and waits on the device until the assembly kernel running
    beside it has bumped `progress` to `target` (see tfem_iface_pack_after)."""
    device = check_cuda(out, src, idx, progress)
    call("tfem_iface_pack_after", src.dtype, device, idx.shape[0], ptr(idx), ptr(src), ptr(out), ptr(progress), target & 0xFFFFFFFF)


def unpack_add_raw(dst: Tensor, idx: Tensor, buf: Tensor) -> None:
    """dst[idx[i]] += buf[i] (unique idx): direct C-ABI call for per-step hot loops."""
    device = check_cuda(dst, idx, buf)
    call("tfem_iface_unpack_add", dst.dtype, device, idx.shape[0], ptr(idx), ptr(buf), ptr(dst))


@torch.library.custom_op(f"{NS}::csr_spmv", mutates_args=())
def csr_spmv(crow: Tensor, col: Tensor, val: Tensor, x: Tensor, keep: Optional[Tensor] = None) -> Tensor:
    """y = A x for the CSR matrix (crow, col, val); rows with keep == 0 (uint8) give 0."""
    device = check_cuda(crow, col, val, x)
    n_rows = crow.shape[0] - 1
    y = torch.empty(n_rows, dtype=val.dtype, device=device)
    call("tfem_csr_spmv", val.dtype, device, n_rows, ptr(crow), ptr(col), ptr(val), ptr(x), ptr(keep) if keep is not None else None, ptr(y))
    return y


@csr_spmv.register_fake
def _(crow, col, val, x, keep=None):
    return val.new_empty(crow.shape[0] - 1)


def csr_spmv_raw(crow: Tensor, col: Tensor, val: Tensor, x: Tensor, keep: Optional[Tensor], out: Tensor) -> None:
    """`csr_spmv` into a preallocated vector: direct C-ABI call for solver inner loops (CUDA-graph capturable)."""
    device = check_cuda(crow, col, val, x, out)
    call("tfem_csr_spmv", val.dtype, device, crow.shape[0] - 1, ptr(crow), ptr(col), ptr(val), ptr(x),
         ptr(keep) if keep is not None else None, ptr(out))


def cg_iteration_raw(crow: Tensor, col: Tensor, val: Tensor, keep: Optional[Tensor], inv_diag: Tensor, x: Tensor, r: Tensor,
                     z: Tensor, p: Tensor, ap: Tensor, partial: Tensor, scal: Tensor) -> None:
    """One fused preconditioned-CG iteration on preallocated state (see tfem_cg_iteration); CUDA-graph capturable."""
    device = check_cuda(crow, col, val, inv_diag, x, r, z, p, ap, partial, scal)
    call("tfem_cg_iteration", val.dtype, device, crow.shape[0] - 1, ptr(crow), ptr(col), ptr(val),
         ptr(keep) if keep is not None else None, ptr(inv_diag), ptr(x), ptr(r), ptr(z), ptr(p), ptr(ap), ptr(partial),
         partial.shape[0] // 2, ptr(scal))


# ------------------------------------------------------------------------------------------------
# smoothed-aggregation AMG (set-up and V-cycle; sparse.amg builds the hierarchy)
# ------------------------------------------------------------------------------------------------


def amg_strength(crow: Tensor, col: Tensor, val: Tensor, theta: float) -> Tuple[Tensor, Tensor]:
    """(diag [n], strong [nnz] uint8): strength of connection |a_ij| >= theta sqrt(|a_ii a_jj|), i != j."""
    device = check_cuda(crow, col, val)
    n = crow.shape[0] - 1
    diag = torch.empty(n, dtype=val.dtype, device=device)
    strong = torch.empty(col.shape[0], dtype=torch.uint8, device=device)
    call("tfem_amg_strength", val.dtype, device, n, ptr(crow), ptr(col), ptr(val), float(theta), ptr(diag), ptr(strong))
    return diag, strong


def _workspace(name: str, *sizes) -> int:
    import ctypes

    need = ctypes.c_int64(0)
    status = getattr(_lib.load(), name)(*sizes, ctypes.byref(need))
    if status != 0:
        raise TfemError(f"{name} failed ({status})")
    return int(need.value)


def amg_aggregate(crow: Tensor, col: Tensor, strong: Tensor, level: int) -> Tuple[Tensor, int]:
    """(agg [n] int32, n_agg): parallel MIS(2) aggregation of the strength graph (-1: no strong connection).
    Set-up: the host reads the undecided count after every round."""
    device = check_cuda(crow, col, strong)
    n = crow.shape[0] - 1
    key = torch.empty(n, dtype=torch.int64, device=device)
    scratch = torch.empty(2 * n, dtype=torch.int64, device=device)
    counter = torch.zeros(1, dtype=torch.int32, device=device)
    for round_ in range(n + 1):  # every round decides at least the undecided node of the largest key
        call("tfem_amg_mis2_round", None, device, n, ptr(crow), ptr(col), ptr(strong), level, int(round_ == 0), ptr(key), ptr(scratch),
                    ptr(counter))
        if int(counter.item()) == 0:
            break
    else:
        raise TfemError("MIS(2) aggregation did not terminate")
    workspace = torch.empty(_workspace("tfem_amg_aggregate_workspace", n), dtype=torch.uint8, device=device)
    agg = torch.empty(n, dtype=torch.int32, device=device)
    call("tfem_amg_aggregate", None, device, n, ptr(crow), ptr(col), ptr(strong), ptr(key), ptr(workspace), workspace.numel(),
                ptr(agg), ptr(counter))
    return agg, int(counter.item())


def csr_spgemm(a: Tuple[Tensor, Tensor, Tensor], n_cols_a: int, b: Tuple[Tensor, Tensor, Tensor], n_cols_b: int) -> Tuple[Tensor, Tensor, Tensor]:
    """C = A B as CSR (crow, col, val) for A with n_cols_a columns and B with n_cols_b (tfem_csr_spgemm; the device
    product reads A's column count from B's row pointer)."""
    a_crow, a_col, a_val = a
    b_crow, b_col, b_val = b
    device = check_cuda(a_crow, a_col, a_val, b_crow, b_col, b_val)
    n_rows = a_crow.shape[0] - 1
    n_products = int((b_crow[1:] - b_crow[:-1]).long()[a_col.long()].sum())
    workspace = torch.empty(_workspace("tfem_csr_spgemm_workspace", n_rows, n_products), dtype=torch.uint8, device=device)
    c_crow = torch.empty(n_rows + 1, dtype=torch.int32, device=device)
    c_col = torch.empty(max(n_products, 1), dtype=torch.int32, device=device)
    c_val = torch.empty(max(n_products, 1), dtype=a_val.dtype, device=device)
    c_nnz = torch.zeros(1, dtype=torch.int64, device=device)
    call("tfem_csr_spgemm", a_val.dtype, device, n_rows, ptr(a_crow), ptr(a_col), ptr(a_val), 0, ptr(b_crow), ptr(b_col), ptr(b_val),
         n_rows, max(n_cols_b, 1), n_products, ptr(workspace), workspace.numel(), ptr(c_crow), ptr(c_col), ptr(c_val), ptr(c_nnz))
    nnz = int(c_nnz.item())
    return c_crow, c_col[:nnz].clone(), c_val[:nnz].clone()


def csr_spgemm_numeric(a: Tuple[Tensor, Tensor, Tensor], b: Tuple[Tensor, Tensor, Tensor], c_crow: Tensor, c_col: Tensor,
                       out: Optional[Tensor] = None, n_missing: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """(c_val, n_missing): the values of C = A B on the pattern (c_crow, c_col), bitwise those `csr_spgemm` gives on its
    own pattern (tfem_csr_spgemm_numeric).  `out` receives c_val in place; products outside the pattern are dropped and
    counted into the int32 device counter `n_missing` (a new zeroed one when None)."""
    a_crow, a_col, a_val = a
    b_crow, b_col, b_val = b
    device = check_cuda(a_crow, a_col, a_val, b_crow, b_col, b_val, c_crow, c_col, out, n_missing)
    if out is None:
        out = torch.empty(c_col.shape[0], dtype=a_val.dtype, device=device)
    if n_missing is None:
        n_missing = torch.zeros(1, dtype=torch.int32, device=device)
    # an empty A, B or C has no storage; the kernel reads nothing of it but the entry point wants a pointer
    a_col, a_val, b_col, b_val, c_col, c_val = (t if t.numel() else t.new_empty(1) for t in (a_col, a_val, b_col, b_val, c_col, out))
    call("tfem_csr_spgemm_numeric", a_val.dtype, device, a_crow.shape[0] - 1, ptr(a_crow), ptr(a_col), ptr(a_val), ptr(b_crow), ptr(b_col),
         ptr(b_val), ptr(c_crow), ptr(c_col), ptr(c_val), ptr(n_missing))
    return out, n_missing


def amg_diag(crow: Tensor, col: Tensor, val: Tensor) -> Tensor:
    """diag [n] of a CSR matrix (0 where a row stores none): the diagonal `amg_strength` returns."""
    device = check_cuda(crow, col, val)
    diag = torch.empty(crow.shape[0] - 1, dtype=val.dtype, device=device)
    call("tfem_amg_diag", val.dtype, device, crow.shape[0] - 1, ptr(crow), ptr(col), ptr(val), ptr(diag))
    return diag


def amg_smoother(crow: Tensor, col: Tensor, val: Tensor, diag: Tensor, omega: float, wdinv: Tensor, s_val: Tensor) -> None:
    """wdinv = omega / diag and s_val = I - wdinv A on A's pattern, in place, rounded as torch rounds those expressions."""
    device = check_cuda(crow, col, val, diag, wdinv, s_val)
    call("tfem_amg_smoother", val.dtype, device, crow.shape[0] - 1, ptr(crow), ptr(col), ptr(val), ptr(diag), float(omega), ptr(wdinv),
         ptr(s_val))


def gather_fill(src: Tensor, values: Tensor, fill: float, out: Tensor) -> Tensor:
    """out[k] = values[src[k]] where src[k] >= 0, else fill (src int32), in place (tfem_gather)."""
    device = check_cuda(src, values, out)
    if out.shape[0] != src.shape[0] or out.dtype != values.dtype:
        raise TfemError("gather_fill: out must have src's length and the values' dtype")
    call("tfem_gather", values.dtype, device, src.shape[0], ptr(src), ptr(values), float(fill), ptr(out))
    return out


def amg_levels_struct(hierarchy):
    """ctypes array of struct tfem_amg_level over the device tensors of an `sparse.AmgHierarchy` (kept alive by it)."""
    levels = hierarchy.levels
    array = (_lib.AmgLevel * max(len(levels), 1))()
    for slot, lev in zip(array, levels):
        slot.n, slot.n_coarse = lev.n, lev.n_coarse
        for name in ("a_crow", "a_col", "a_val", "p_crow", "p_col", "p_val", "r_crow", "r_col", "r_val", "wdinv", "x", "rc", "ec"):
            setattr(slot, name, ptr(getattr(lev, name)))
    return array


def amg_vcycle_raw(hierarchy, r: Tensor, z: Tensor) -> None:
    """z = M_AMG r (one V-cycle, tfem_amg_vcycle) into a preallocated vector; CUDA-graph capturable."""
    device = check_cuda(r, z, hierarchy.coarse_inv)
    call("tfem_amg_vcycle", r.dtype, device, hierarchy.struct, len(hierarchy.levels), ptr(hierarchy.coarse_inv),
         hierarchy.coarse_inv.shape[0], ptr(r), ptr(z))


def amg_vcycle(hierarchy, r: Tensor) -> Tensor:
    """z = M_AMG r."""
    z = torch.empty_like(r)
    amg_vcycle_raw(hierarchy, r, z)
    return z


def pcg_iteration_raw(crow: Tensor, col: Tensor, val: Tensor, keep: Optional[Tensor], hierarchy, x: Tensor, r: Tensor, z: Tensor,
                      p: Tensor, ap: Tensor, partial: Tensor, scal: Tensor) -> None:
    """One AMG-preconditioned CG iteration on preallocated state (see tfem_pcg_iteration); CUDA-graph capturable."""
    device = check_cuda(crow, col, val, x, r, z, p, ap, partial, scal, hierarchy.coarse_inv)
    call("tfem_pcg_iteration", val.dtype, device, crow.shape[0] - 1, ptr(crow), ptr(col), ptr(val),
         ptr(keep) if keep is not None else None, hierarchy.struct, len(hierarchy.levels), ptr(hierarchy.coarse_inv),
         hierarchy.coarse_inv.shape[0], ptr(x), ptr(r), ptr(z), ptr(p), ptr(ap), ptr(partial), partial.shape[0] // 2, ptr(scal))


# ------------------------------------------------------------------------------------------------
# fused named forms
# ------------------------------------------------------------------------------------------------


@torch.library.custom_op(f"{NS}::local_forms", mutates_args=())
def local_forms(
    coords: Tensor,
    conn: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    alpha: float,
    beta: float,
    want_matrix: bool,
    source_kind: int,
    source_p: List[float],
    f_q: Optional[Tensor] = None,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor]:
    """Per-element alpha*K + beta*M (N,3,3) and load (N,3) without intermediates."""
    device = check_cuda(coords, conn, f_q, frac_jac, frac_inv, frac_det, frac_t)
    _nq_tri(quad_order)
    n_el = conn.shape[0]
    opts = dict(dtype=coords.dtype, device=device)
    want_vec = source_kind != _lib.TFEM_SRC_NONE
    local_mat = torch.empty((n_el, 3, 3) if want_matrix else (0, 3, 3), **opts)
    local_vec = torch.empty((n_el, 3) if want_vec else (0, 3), **opts)
    form = Bilinear(alpha, beta)
    src = make_source(source_kind, source_p)
    call(
        "tfem_tri_p1_local_forms", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
        quad_order, ptr(frac_jac), ptr(frac_inv), ptr(frac_det), ptr(frac_t), form, src, ptr(f_q),
        ptr(local_mat) if want_matrix else None, ptr(local_vec) if want_vec else None,
    )
    return local_mat, local_vec


@local_forms.register_fake
def _(coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, alpha, beta, want_matrix, source_kind, source_p,
      f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    n_el = conn.shape[0]
    return coords.new_empty((n_el if want_matrix else 0, 3, 3)), coords.new_empty((n_el if source_kind else 0, 3))


@torch.library.custom_op(f"{NS}::weighted_local_forms", mutates_args=())
def weighted_local_forms(
    coords: Tensor,
    conn: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    alpha: float,
    beta: float,
    alpha_q: Optional[Tensor],
    beta_q: Optional[Tensor],
    source_kind: int,
    source_p: List[float],
    f_q: Optional[Tensor] = None,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor]:
    """Per-element K(alpha_q) + M(beta_q) (N,3,3) and load (N,3); alpha_q / beta_q (N, n_q) or None for the constants."""
    device = check_cuda(coords, conn, alpha_q, beta_q, f_q, frac_jac, frac_inv, frac_det, frac_t)
    n_q = _nq_tri(quad_order)
    n_el = conn.shape[0]
    for name, field in (("alpha_q", alpha_q), ("beta_q", beta_q)):
        if field is not None and (tuple(field.shape) != (n_el, n_q) or field.dtype != coords.dtype):
            raise TfemError(f"{name} must be ({n_el}, {n_q}) {coords.dtype}, got {tuple(field.shape)} {field.dtype}")
    opts = dict(dtype=coords.dtype, device=device)
    want_vec = source_kind != _lib.TFEM_SRC_NONE
    local_mat = torch.empty((n_el, 3, 3), **opts)
    local_vec = torch.empty((n_el, 3) if want_vec else (0, 3), **opts)
    call(
        "tfem_tri_p1_weighted_local_forms", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
        quad_order, ptr(frac_jac), ptr(frac_inv), ptr(frac_det), ptr(frac_t), Bilinear(alpha, beta),
        make_source(source_kind, source_p), ptr(f_q), ptr(alpha_q), ptr(beta_q), ptr(local_mat),
        ptr(local_vec) if want_vec else None,
    )
    return local_mat, local_vec


@weighted_local_forms.register_fake
def _(coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, alpha, beta, alpha_q, beta_q, source_kind, source_p,
      f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    n_el = conn.shape[0]
    return coords.new_empty((n_el, 3, 3)), coords.new_empty((n_el if source_kind else 0, 3))


def _tiled_struct(tile_list: Tensor, tile_desc: Tensor, inst_blob: Tensor, tpl_desc: Tensor, tpl_blob: Tensor, meta: List[int],
                  progress: Optional[Tensor]):
    """struct tfem_tile_plan from the plan's device arrays and its integer fields (TilePlan.op_args)."""
    s = _lib.TilePlan()
    s.n_tiles = int(tile_list.numel())
    s.tile_list, s.tile_desc, s.inst_blob = tile_list.data_ptr(), tile_desc.data_ptr(), inst_blob.data_ptr()
    s.tpl_desc, s.tpl_blob = tpl_desc.data_ptr(), tpl_blob.data_ptr()
    (s.max_vert, s.max_elem, s.max_inst_words, s.max_tb_words, s.max_tc_words, s.has_elem_ids, s.table_bytes,
     od0, od1, od2, s.consumer_threads, s.reserve_ctas, s.n_progress_tiles) = meta
    s.od_base[0], s.od_base[1], s.od_base[2] = od0, od1, od2
    s.progress = None if progress is None else progress.data_ptr()
    if progress is None:
        s.n_progress_tiles = 0
    return s


@torch.library.custom_op(f"{NS}::assemble_csr_tiled", mutates_args=("csr_val", "load"))
def assemble_csr_tiled_op(
    coords: Tensor, tile_list: Tensor, tile_desc: Tensor, inst_blob: Tensor, tpl_desc: Tensor, tpl_blob: Tensor, meta: List[int],
    quad_order: int, alpha: float, beta: float, source_kind: int, source_p: List[float], csr_val: Optional[Tensor] = None,
    load: Optional[Tensor] = None, f_q: Optional[Tensor] = None, n_el_per_mesh: int = 0, frac_metric: Optional[Tensor] = None,
    progress: Optional[Tensor] = None,
) -> None:
    """The fused tiled assembly (tfem_tri_p1_assemble_csr[_ex]) as a registered op: ONE kernel writes the CSR value
    array and / or the load vector in place.  The tile plan travels as its device arrays plus `meta`
    (`TilePlan.op_args()`); `f_q` (N, n_q) = source at the quadrature points (source_kind SAMPLED); `frac_metric`
    (n_mesh, 4) = (a00, a01, a11, det J_f) for fracture networks."""
    device = check_cuda(coords, tile_list, tile_desc, inst_blob, tpl_desc, tpl_blob, csr_val, load, f_q, frac_metric, progress)
    plan = _tiled_struct(tile_list, tile_desc, inst_blob, tpl_desc, tpl_blob, meta, progress)
    form = Bilinear(alpha, beta)
    src = make_source(source_kind, source_p)
    if f_q is None and frac_metric is None:
        call("tfem_tri_p1_assemble_csr", coords.dtype, device, plan, ptr(coords), quad_order, form, src, ptr(csr_val), ptr(load))
    else:
        call("tfem_tri_p1_assemble_csr_ex", coords.dtype, device, plan, ptr(coords), quad_order, form, src, ptr(f_q), n_el_per_mesh,
             ptr(frac_metric), ptr(csr_val), ptr(load))


def assemble_csr_tiled(plan, coords: Tensor, quad_order: int, alpha: float, beta: float, source_kind: int,
                       source_p, csr_val: Optional[Tensor], load: Optional[Tensor], f_q: Optional[Tensor] = None,
                       n_el_per_mesh: int = 0, frac_metric: Optional[Tensor] = None) -> None:
    """Fused tiled assembly into preallocated outputs (one kernel).  `plan`: a `tileplan.TilePlan` (dispatched through
    the registered op `torch_fem_b200::assemble_csr_tiled`) or its C struct (`TilePlan.c_struct()`: the bare C-ABI call,
    for per-step hot loops that cannot afford the dispatcher)."""
    if hasattr(plan, "op_args"):
        assemble_csr_tiled_op(coords, *plan.op_args(), quad_order, alpha, beta, source_kind, list(source_p), csr_val, load, f_q,
                              n_el_per_mesh, frac_metric, plan.progress)
        return
    device = check_cuda(coords, csr_val, load, f_q, frac_metric)
    form = Bilinear(alpha, beta)
    src = make_source(source_kind, source_p)
    if f_q is None and frac_metric is None:
        call("tfem_tri_p1_assemble_csr", coords.dtype, device, plan, ptr(coords), quad_order, form, src, ptr(csr_val), ptr(load))
    else:
        call("tfem_tri_p1_assemble_csr_ex", coords.dtype, device, plan, ptr(coords), quad_order, form, src, ptr(f_q), n_el_per_mesh,
             ptr(frac_metric), ptr(csr_val), ptr(load))


# ------------------------------------------------------------------------------------------------
# weak residual with autograd
# ------------------------------------------------------------------------------------------------


def _weak_residual_local_launch(grad_u, coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, source_kind,
                                source_p, f_q, frac_jac, frac_inv, frac_det, frac_t) -> Tensor:
    """The launch itself (shared by the stand-alone op and by `weak_residual`, which would otherwise pay a
    second custom-op dispatch per training step)."""
    device = check_cuda(grad_u, coords, conn, dof_conn, f_q, frac_jac, frac_inv, frac_det, frac_t)
    n_q = _nq_tri(quad_order)
    n_el = conn.shape[0]
    d = 3 if frac_inv is not None else 2
    if tuple(grad_u.shape) != (n_el, n_q, d):
        raise TfemError(f"grad_u must have shape {(n_el, n_q, d)}, got {tuple(grad_u.shape)}")
    out = torch.empty((n_el, 3), dtype=coords.dtype, device=device)
    src = make_source(source_kind, source_p)
    call(
        "tfem_weak_residual_local", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
        quad_order, ptr(frac_jac), ptr(frac_inv), ptr(frac_det), ptr(frac_t), src, ptr(f_q), ptr(grad_u), ptr(out),
    )
    return out


@torch.library.custom_op(f"{NS}::weak_residual_local", mutates_args=())
def weak_residual_local(
    grad_u: Tensor,
    coords: Tensor,
    conn: Tensor,
    dof_conn: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    source_kind: int,
    source_p: List[float],
    f_q: Optional[Tensor] = None,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tensor:
    """grad_u (N,q,d) -> per-element residual (N,3): sum_q dx (f phi_i - grad phi_i . grad_u)."""
    return _weak_residual_local_launch(grad_u, coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order,
                                       source_kind, source_p, f_q, frac_jac, frac_inv, frac_det, frac_t)


@weak_residual_local.register_fake
def _(grad_u, coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, source_kind, source_p,
      f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    return coords.new_empty((conn.shape[0], 3))


@torch.library.custom_op(f"{NS}::weak_residual_bwd", mutates_args=())
def weak_residual_bwd(
    r_bar: Tensor,
    coords: Tensor,
    conn: Tensor,
    dof_conn: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
) -> Tensor:
    """r_bar (n_dof,) -> grad_u_bar (N,q,d) = -dx * sum_i grad phi_i * r_bar[dof_conn[:,i]]."""
    device = check_cuda(r_bar, coords, conn, dof_conn, frac_jac, frac_inv, frac_det)
    n_q = _nq_tri(quad_order)
    n_el = conn.shape[0]
    d = 3 if frac_inv is not None else 2
    out = torch.empty((n_el, n_q, d), dtype=coords.dtype, device=device)
    call(
        "tfem_weak_residual_bwd", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
        ptr(dof_conn), quad_order, ptr(frac_jac), ptr(frac_inv), ptr(frac_det), ptr(r_bar), ptr(out),
    )
    return out


@weak_residual_bwd.register_fake
def _(r_bar, coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, frac_jac=None, frac_inv=None, frac_det=None):
    d = 3 if frac_inv is not None else 2
    return coords.new_empty((conn.shape[0], TRI_NQ[quad_order], d))


@torch.library.custom_op(f"{NS}::weak_residual", mutates_args=())
def weak_residual(
    grad_u: Tensor,
    coords: Tensor,
    conn: Tensor,
    dof_conn: Tensor,
    lin_seg: Tensor,
    lin_perm: Tensor,
    n_el_per_mesh: int,
    n_vert_per_mesh: int,
    quad_order: int,
    source_kind: int,
    source_p: List[float],
    f_q: Optional[Tensor] = None,
    frac_jac: Optional[Tensor] = None,
    frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None,
    frac_t: Optional[Tensor] = None,
) -> Tensor:
    """Global weak residual r (n_dof,): element kernel + deterministic scatter, two launches -- or ONE launch
    (`tfem_batched_weak_residual`) for batches of small meshes with mesh-private DOFs (patches)."""
    n_mesh = conn.shape[0] // n_el_per_mesh
    if (frac_inv is None and n_el_per_mesh <= 8 and n_vert_per_mesh <= 16 and n_mesh > 1
            and lin_seg.shape[0] - 1 == n_mesh * n_vert_per_mesh and n_mesh * n_el_per_mesh == conn.shape[0]):
        device = check_cuda(grad_u, coords, conn, f_q)
        n_q = _nq_tri(quad_order)
        if tuple(grad_u.shape) != (conn.shape[0], n_q, 2):
            raise TfemError(f"grad_u must have shape {(conn.shape[0], n_q, 2)}, got {tuple(grad_u.shape)}")
        out = torch.empty((n_mesh * n_vert_per_mesh,), dtype=coords.dtype, device=device)
        call("tfem_batched_weak_residual", coords.dtype, device, n_mesh, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn),
             quad_order, make_source(source_kind, source_p), ptr(f_q), ptr(grad_u), ptr(out))
        return out
    local = _weak_residual_local_launch(
        grad_u, coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, source_kind, source_p,
        f_q, frac_jac, frac_inv, frac_det, frac_t,
    )
    device = check_cuda(local, lin_seg, lin_perm)
    n_dof = lin_seg.shape[0] - 1
    out = torch.empty((n_dof,), dtype=local.dtype, device=device)
    call("tfem_scatter_linear", local.dtype, device, n_dof, ptr(lin_seg), ptr(lin_perm), ptr(local), ptr(out))
    return out


@weak_residual.register_fake
def _(grad_u, coords, conn, dof_conn, lin_seg, lin_perm, n_el_per_mesh, n_vert_per_mesh, quad_order, source_kind,
      source_p, f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    return coords.new_empty((lin_seg.shape[0] - 1,))


def _weak_residual_setup(ctx, inputs, output):
    (grad_u, coords, conn, dof_conn, lin_seg, lin_perm, n_el_per_mesh, n_vert_per_mesh, quad_order, source_kind,
     source_p, f_q, frac_jac, frac_inv, frac_det, frac_t) = inputs
    ctx.save_for_backward(coords, conn, dof_conn, frac_jac, frac_inv, frac_det)
    ctx.meta = (n_el_per_mesh, n_vert_per_mesh, quad_order)


def _weak_residual_backward(ctx, r_bar):
    coords, conn, dof_conn, frac_jac, frac_inv, frac_det = ctx.saved_tensors
    n_el_per_mesh, n_vert_per_mesh, quad_order = ctx.meta
    grad = weak_residual_bwd(
        r_bar.contiguous(), coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, frac_jac, frac_inv, frac_det
    )
    return (grad,) + (None,) * 15


weak_residual.register_autograd(_weak_residual_backward, setup_context=_weak_residual_setup)


@torch.library.custom_op(f"{NS}::weak_residual_tiled", mutates_args=())
def weak_residual_tiled(
    grad_u: Tensor, coords: Tensor, conn: Tensor, dof_conn: Tensor, tile_list: Tensor, tile_desc: Tensor, inst_blob: Tensor,
    tpl_desc: Tensor, tpl_blob: Tensor, meta: List[int], n_dof: int, n_el_per_mesh: int, n_vert_per_mesh: int, quad_order: int,
    f_q: Optional[Tensor] = None, frac_jac: Optional[Tensor] = None, frac_inv: Optional[Tensor] = None,
    frac_det: Optional[Tensor] = None, frac_metric: Optional[Tensor] = None,
) -> Tensor:
    """Global weak residual r (n_dof,) in ONE launch of the tiled kernel (`tfem_weak_residual_tiled`): no per-element
    tensor, no scatter pass.  The tile plan (built with element ids) travels as its device arrays plus `meta`; `f_q`
    (N, n_q) = f at the quadrature points or None (f = 0); fracture networks pass J_f^+ (`frac_inv`) and the plane
    metric (`frac_metric`).  `conn`, `dof_conn`, `frac_jac`, `frac_det` only serve the adjoint (`weak_residual_bwd`)."""
    device = check_cuda(grad_u, coords, tile_list, tile_desc, inst_blob, tpl_desc, tpl_blob, f_q, frac_inv, frac_metric)
    n_q = _nq_tri(quad_order)
    d = 3 if frac_inv is not None else 2
    if tuple(grad_u.shape) != (conn.shape[0], n_q, d):
        raise TfemError(f"grad_u must have shape {(conn.shape[0], n_q, d)}, got {tuple(grad_u.shape)}")
    plan = _tiled_struct(tile_list, tile_desc, inst_blob, tpl_desc, tpl_blob, meta, None)
    out = torch.empty((n_dof,), dtype=coords.dtype, device=device)
    call("tfem_weak_residual_tiled", coords.dtype, device, plan, ptr(coords), quad_order, ptr(f_q), ptr(grad_u), n_el_per_mesh,
         ptr(frac_inv), ptr(frac_metric), ptr(out))
    return out


@weak_residual_tiled.register_fake
def _(grad_u, coords, conn, dof_conn, tile_list, tile_desc, inst_blob, tpl_desc, tpl_blob, meta, n_dof, n_el_per_mesh,
      n_vert_per_mesh, quad_order, f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_metric=None):
    return coords.new_empty((n_dof,))


def _weak_residual_tiled_setup(ctx, inputs, output):
    (grad_u, coords, conn, dof_conn, _tl, _td, _ib, _pd, _pb, _meta, _n_dof, n_el_per_mesh, n_vert_per_mesh, quad_order,
     _f_q, frac_jac, frac_inv, frac_det, _metric) = inputs
    ctx.save_for_backward(coords, conn, dof_conn, frac_jac, frac_inv, frac_det)
    ctx.meta = (n_el_per_mesh, n_vert_per_mesh, quad_order)


def _weak_residual_tiled_backward(ctx, r_bar):
    coords, conn, dof_conn, frac_jac, frac_inv, frac_det = ctx.saved_tensors
    n_el_per_mesh, n_vert_per_mesh, quad_order = ctx.meta
    grad = weak_residual_bwd(
        r_bar.contiguous(), coords, conn, dof_conn, n_el_per_mesh, n_vert_per_mesh, quad_order, frac_jac, frac_inv, frac_det
    )
    return (grad,) + (None,) * 18


weak_residual_tiled.register_autograd(_weak_residual_tiled_backward, setup_context=_weak_residual_tiled_setup)


@torch.library.custom_op(f"{NS}::h1_error", mutates_args=())
def h1_error(u: Tensor, grad_u: Tensor, u_ex: Tensor, grad_ex: Tensor, coords: Tensor, conn: Tensor, n_el_per_mesh: int,
             n_vert_per_mesh: int, quad_order: int, frac_det: Optional[Tensor] = None) -> Tensor:
    """Per-element H1 error sum_q dx ((u_ex - u)^2 + |grad_ex - grad_u|^2): fields (N,q) / (N,q,d) -> (N,)."""
    device = check_cuda(u, grad_u, u_ex, grad_ex, coords, conn, frac_det)
    n_el, n_q, d = grad_u.shape
    if n_q != _nq_tri(quad_order) or tuple(u.shape) != (n_el, n_q) or u_ex.shape != u.shape or grad_ex.shape != grad_u.shape:
        raise TfemError("h1_error: fields must be (N, n_q) and (N, n_q, d) at the basis' quadrature points")
    out = torch.empty((n_el,), dtype=coords.dtype, device=device)
    call("tfem_h1_error", coords.dtype, device, n_el, n_el_per_mesh, n_vert_per_mesh, ptr(coords), ptr(conn), quad_order,
         ptr(frac_det), d, ptr(u), ptr(grad_u), ptr(u_ex), ptr(grad_ex), ptr(out))
    return out


@h1_error.register_fake
def _(u, grad_u, u_ex, grad_ex, coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, frac_det=None):
    return coords.new_empty((conn.shape[0],))


# ------------------------------------------------------------------------------------------------
# edge topology (SURVEY 8(f).2): integer, one-time; plain functions (nothing to differentiate)
# ------------------------------------------------------------------------------------------------
def half_edges(conn: Tensor, n_vert: int, local_pairs) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """conn (F,N,3) int32 -> (he_sorted (3FN,) int64, cell_sorted (3FN,) int32, unique keys (E,) int64, incidence counts
    (E,) int32) of the cell edges keyed `mesh * n_vert^2 + min * n_vert + max` (`tfem_half_edges`)."""
    import ctypes

    device = check_cuda(conn)
    n_mesh, n_cells, _ = conn.shape
    n_half = 3 * n_mesh * n_cells
    lib = _lib.load()
    need = ctypes.c_int64()
    if lib.tfem_half_edges_workspace(n_mesh, n_cells, ctypes.byref(need)) != 0:
        raise TfemError("tfem_half_edges_workspace failed")
    workspace = torch.empty(need.value, dtype=torch.uint8, device=device)
    he_sorted = torch.empty(n_half, dtype=torch.int64, device=device)
    cell_sorted = torch.empty(n_half, dtype=torch.int32, device=device)
    uniq = torch.empty(n_half, dtype=torch.int64, device=device)
    counts = torch.empty(n_half, dtype=torch.int32, device=device)
    n_unique = torch.zeros(1, dtype=torch.int64, device=device)
    pairs = (ctypes.c_int32 * 6)(*[int(v) for pair in local_pairs for v in pair])
    call("tfem_half_edges", None, device, n_mesh, n_cells, n_vert, ptr(conn), pairs, ptr(workspace), need.value, ptr(he_sorted),
         ptr(cell_sorted), ptr(uniq), ptr(counts), ptr(n_unique))
    n = int(n_unique.item())
    return he_sorted, cell_sorted, uniq[:n], counts[:n]


def edge_cells(edge_vertices: Tensor, n_vert: int, n_sides: int, he_sorted: Tensor, cell_sorted: Tensor) -> Tensor:
    """edge_vertices (F,E,2) int32 -> adjacent cells (F,E,n_sides) int32, sides in increasing cell id (`tfem_edge_cells`)."""
    device = check_cuda(edge_vertices, he_sorted, cell_sorted)
    n_mesh, n_edges, _ = edge_vertices.shape
    cells = torch.empty((n_mesh, n_edges, n_sides), dtype=torch.int32, device=device)
    status = torch.zeros(1, dtype=torch.int32, device=device)
    call("tfem_edge_cells", None, device, n_mesh, n_edges, n_vert, ptr(edge_vertices), n_sides, ptr(he_sorted), ptr(cell_sorted),
         he_sorted.numel(), ptr(cells), ptr(status))
    flags = int(status.item())
    if flags & 1:
        raise ValueError("an edge of the edge list belongs to no cell")
    if flags & 2:
        raise ValueError("an edge marked interior has a single adjacent cell")
    return cells


def interior_edge_geometry(coords: Tensor, conn: Tensor, edge_vertices: Tensor, cells: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """coords (F,V,2), conn (F,N,3) int32, interior edges (F,E,2) int32 and their cells (F,E,2) int32 -> end points
    (F,E,2,2), length (F,E,1,1), oriented unit normal (F,E,1,2) (`tfem_interior_edge_geometry`)."""
    device = check_cuda(coords, conn, edge_vertices, cells)
    n_mesh, n_edges, _ = edge_vertices.shape
    opts = dict(dtype=coords.dtype, device=device)
    x = torch.empty((n_mesh, n_edges, 2, 2), **opts)
    length = torch.empty((n_mesh, n_edges, 1, 1), **opts)
    normal = torch.empty((n_mesh, n_edges, 1, 2), **opts)
    call("tfem_interior_edge_geometry", coords.dtype, device, n_mesh, n_edges, coords.shape[1], conn.shape[1], ptr(coords), ptr(conn),
         ptr(edge_vertices), ptr(cells), ptr(x), ptr(length), ptr(normal))
    return x, length, normal


# ------------------------------------------------------------------------------------------------
# fused MLP producer (SURVEY 8(f).3)
# ------------------------------------------------------------------------------------------------
ACT_TANH, ACT_RELU = 0, 1
MLP_MAX_WIDTH, MLP_MAX_SQUARE_BWD = 32, 7


def mlp_param_count(d: int, width: int, n_square: int) -> int:
    return width * d + width + n_square * (width * width + width) + width + 1


@torch.library.custom_op(f"{NS}::mlp_value_grad", mutates_args=())
def mlp_value_grad(params: Tensor, x: Tensor, width: int, n_square: int, act: int) -> Tuple[Tensor, Tensor]:
    """N(x) (M,) and dN/dx (M,d) of the MLP Linear(d,w) act {Linear(w,w) act} x n_square Linear(w,1) whose parameters
    are packed in `params` (torch.nn.Linear layout, in network order), by forward-mode differentiation in ONE kernel
    (`tfem_mlp_value_grad`).  Differentiable with respect to `params` (not `x`: the points are quadrature points)."""
    device = check_cuda(params, x)
    n_pts, d = x.shape
    if params.numel() != mlp_param_count(d, width, n_square) or params.dtype != x.dtype:
        raise TfemError(f"mlp_value_grad: expected {mlp_param_count(d, width, n_square)} packed parameters of dtype {x.dtype}")
    value = torch.empty((n_pts,), dtype=x.dtype, device=device)
    grad = torch.empty((n_pts, d), dtype=x.dtype, device=device)
    call("tfem_mlp_value_grad", x.dtype, device, n_pts, d, width, n_square, act, ptr(params), ptr(x), ptr(value), ptr(grad))
    return value, grad


@mlp_value_grad.register_fake
def _(params, x, width, n_square, act):
    return x.new_empty((x.shape[0],)), x.new_empty(x.shape)


@torch.library.custom_op(f"{NS}::mlp_value_grad_bwd", mutates_args=())
def mlp_value_grad_bwd(params: Tensor, x: Tensor, value_bar: Tensor, grad_bar: Tensor, width: int, n_square: int, act: int) -> Tensor:
    """Adjoint of `mlp_value_grad` with respect to the packed parameters (`tfem_mlp_value_grad_bwd`)."""
    device = check_cuda(params, x, value_bar, grad_bar)
    n_pts, d = x.shape
    n_partial = _lib.load().tfem_sm_count()
    if n_partial <= 0:
        raise TfemError("tfem_sm_count failed")
    partial = torch.empty((n_partial, params.numel()), dtype=x.dtype, device=device)
    out = torch.empty_like(params)
    call("tfem_mlp_value_grad_bwd", x.dtype, device, n_pts, d, width, n_square, act, ptr(params), ptr(x), ptr(value_bar), ptr(grad_bar),
         ptr(partial), n_partial, ptr(out))
    return out


@mlp_value_grad_bwd.register_fake
def _(params, x, value_bar, grad_bar, width, n_square, act):
    return torch.empty_like(params)


def _mlp_setup(ctx, inputs, output):
    params, x, width, n_square, act = inputs
    ctx.save_for_backward(params, x)
    ctx.meta = (width, n_square, act)


def _mlp_backward(ctx, value_bar, grad_bar):
    params, x = ctx.saved_tensors
    width, n_square, act = ctx.meta
    if value_bar is None:
        value_bar = torch.zeros(x.shape[0], dtype=x.dtype, device=x.device)
    if grad_bar is None:
        grad_bar = torch.zeros_like(x)
    out = mlp_value_grad_bwd(params, x, value_bar.contiguous(), grad_bar.contiguous(), width, n_square, act)
    return out, None, None, None, None


mlp_value_grad.register_autograd(_mlp_backward, setup_context=_mlp_setup)


# ------------------------------------------------------------------------------------------------
# interpolation / jump
# ------------------------------------------------------------------------------------------------


@torch.library.custom_op(f"{NS}::interp_cells", mutates_args=())
def interp_cells(
    u: Tensor, dof_conn: Tensor, v_grad: Tensor, quad_order: int, seg: Optional[Tensor] = None,
    perm: Optional[Tensor] = None, inverse: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor]:
    """u (n_dof,), dof_conn (N,3), v_grad (N,3,d) -> values (N,q), gradients (N,d).

    `seg`/`perm`/`inverse` (the linear-form scatter maps of the basis) are only needed to
    differentiate w.r.t. `u`."""
    device = check_cuda(u, dof_conn, v_grad)
    n_q = _nq_tri(quad_order)
    n_el, _, d = v_grad.shape
    val = torch.empty((n_el, n_q), dtype=u.dtype, device=device)
    grad = torch.empty((n_el, d), dtype=u.dtype, device=device)
    call("tfem_interp_cells", u.dtype, device, n_el, ptr(dof_conn), ptr(v_grad), d, quad_order, ptr(u), ptr(val), ptr(grad))
    return val, grad


@interp_cells.register_fake
def _(u, dof_conn, v_grad, quad_order, seg=None, perm=None, inverse=None):
    return u.new_empty((v_grad.shape[0], TRI_NQ[quad_order])), u.new_empty((v_grad.shape[0], v_grad.shape[2]))


@torch.library.custom_op(f"{NS}::interp_cells_bwd", mutates_args=())
def interp_cells_bwd(val_bar: Tensor, grad_bar: Tensor, v_grad: Tensor, quad_order: int) -> Tensor:
    """Per-element part (N,3) of the adjoint of `interp_cells` w.r.t. u."""
    device = check_cuda(val_bar, grad_bar, v_grad)
    n_el, _, d = v_grad.shape
    local = torch.empty((n_el, 3), dtype=v_grad.dtype, device=device)
    call("tfem_interp_cells_bwd", v_grad.dtype, device, n_el, ptr(v_grad), d, quad_order, ptr(val_bar), ptr(grad_bar), ptr(local))
    return local


@interp_cells_bwd.register_fake
def _(val_bar, grad_bar, v_grad, quad_order):
    return v_grad.new_empty((v_grad.shape[0], 3))


def _interp_cells_setup(ctx, inputs, output):
    u, dof_conn, v_grad, quad_order, seg, perm, inverse = inputs
    ctx.save_for_backward(v_grad, seg, perm, inverse)
    ctx.quad_order = quad_order
    ctx.n_dof = u.shape[0]


def _interp_cells_backward(ctx, val_bar, grad_bar):
    v_grad, seg, perm, inverse = ctx.saved_tensors
    if seg is None:
        raise TfemError("differentiating interp_cells w.r.t. u needs the scatter maps (seg, perm, inverse)")
    local = interp_cells_bwd(val_bar.contiguous(), grad_bar.contiguous(), v_grad, ctx.quad_order)
    u_bar = scatter(local.reshape(-1), seg, perm, inverse)
    return u_bar, None, None, None, None, None, None


interp_cells.register_autograd(_interp_cells_backward, setup_context=_interp_cells_setup)


@torch.library.custom_op(f"{NS}::interp_edges", mutates_args=())
def interp_edges(
    u: Tensor,
    edge_cells: Tensor,
    conn: Tensor,
    first_vertex: Tensor,
    inv_jac: Tensor,
    x_q: Tensor,
    n_edge_per_mesh: int,
    n_el_per_mesh: int,
    seg: Optional[Tensor] = None,
    perm: Optional[Tensor] = None,
    inverse: Optional[Tensor] = None,
) -> Tuple[Tensor, Tensor]:
    """Both cells of every interior edge at the edge points: values (E,2,q), gradients (E,2,d).

    `seg`/`perm`/`inverse` (scatter maps of the (edge, side, local vertex) -> DOF relation) are
    only needed to differentiate w.r.t. `u`."""
    device = check_cuda(u, edge_cells, conn, first_vertex, inv_jac, x_q)
    n_edge, n_q, d = x_q.shape
    val = torch.empty((n_edge, 2, n_q), dtype=u.dtype, device=device)
    grad = torch.empty((n_edge, 2, d), dtype=u.dtype, device=device)
    call(
        "tfem_interp_edges", u.dtype, device, n_edge, n_edge_per_mesh, n_el_per_mesh, ptr(edge_cells), ptr(conn),
        ptr(first_vertex), ptr(inv_jac), d, ptr(x_q), n_q, ptr(u), ptr(val), ptr(grad),
    )
    return val, grad


@interp_edges.register_fake
def _(u, edge_cells, conn, first_vertex, inv_jac, x_q, n_edge_per_mesh, n_el_per_mesh, seg=None, perm=None, inverse=None):
    n_edge, n_q, d = x_q.shape
    return u.new_empty((n_edge, 2, n_q)), u.new_empty((n_edge, 2, d))


@torch.library.custom_op(f"{NS}::interp_edges_bwd", mutates_args=())
def interp_edges_bwd(
    val_bar: Tensor, grad_bar: Tensor, edge_cells: Tensor, first_vertex: Tensor, inv_jac: Tensor, x_q: Tensor,
    n_edge_per_mesh: int, n_el_per_mesh: int,
) -> Tensor:
    """Per-(edge, side) part (2E,3) of the adjoint of `interp_edges` w.r.t. u."""
    device = check_cuda(val_bar, grad_bar, edge_cells, first_vertex, inv_jac, x_q)
    n_edge, n_q, d = x_q.shape
    local = torch.empty((2 * n_edge, 3), dtype=x_q.dtype, device=device)
    call(
        "tfem_interp_edges_bwd", x_q.dtype, device, n_edge, n_edge_per_mesh, n_el_per_mesh, ptr(edge_cells),
        ptr(first_vertex), ptr(inv_jac), d, ptr(x_q), n_q, ptr(val_bar), ptr(grad_bar), ptr(local),
    )
    return local


@interp_edges_bwd.register_fake
def _(val_bar, grad_bar, edge_cells, first_vertex, inv_jac, x_q, n_edge_per_mesh, n_el_per_mesh):
    return x_q.new_empty((2 * x_q.shape[0], 3))


def _interp_edges_setup(ctx, inputs, output):
    u, edge_cells, conn, first_vertex, inv_jac, x_q, n_edge_per_mesh, n_el_per_mesh, seg, perm, inverse = inputs
    ctx.save_for_backward(edge_cells, first_vertex, inv_jac, x_q, seg, perm, inverse)
    ctx.sizes = (n_edge_per_mesh, n_el_per_mesh)


def _interp_edges_backward(ctx, val_bar, grad_bar):
    edge_cells, first_vertex, inv_jac, x_q, seg, perm, inverse = ctx.saved_tensors
    if seg is None:
        raise TfemError("differentiating interp_edges w.r.t. u needs the scatter maps (seg, perm, inverse)")
    local = interp_edges_bwd(val_bar.contiguous(), grad_bar.contiguous(), edge_cells, first_vertex, inv_jac, x_q, *ctx.sizes)
    u_bar = scatter(local.reshape(-1), seg, perm, inverse)
    return (u_bar,) + (None,) * 10


interp_edges.register_autograd(_interp_edges_backward, setup_context=_interp_edges_setup)


@torch.library.custom_op(f"{NS}::edge_jump", mutates_args=())
def edge_jump(grad_edges: Tensor, normals: Tensor, h_e: Tensor, dx: Tensor) -> Tensor:
    """eta_E = sum_q dx h_E (grad u+ . n + grad u- . (-n))^2; grad_edges (E,2,d) -> (E,)."""
    device = check_cuda(grad_edges, normals, h_e, dx)
    n_edge, _, d = grad_edges.shape
    eta = torch.empty((n_edge,), dtype=grad_edges.dtype, device=device)
    call("tfem_edge_jump", grad_edges.dtype, device, n_edge, d, dx.shape[1], ptr(grad_edges), ptr(normals), ptr(h_e), ptr(dx), ptr(eta))
    return eta


@edge_jump.register_fake
def _(grad_edges, normals, h_e, dx):
    return grad_edges.new_empty((grad_edges.shape[0],))


def _edge_jump_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _edge_jump_backward(ctx, eta_bar):
    # d eta / d grad(+/-) = +/- 2 h_E (sum_q dx) jump n : elementwise on (E,2,d), a few tiny torch ops
    grad_edges, normals, h_e, dx = ctx.saved_tensors
    jump = ((grad_edges[:, 0] - grad_edges[:, 1]) * normals).sum(-1)
    coef = (2.0 * h_e * dx.sum(-1) * jump * eta_bar).unsqueeze(-1) * normals
    return torch.stack([coef, -coef], dim=1), None, None, None


edge_jump.register_autograd(_edge_jump_backward, setup_context=_edge_jump_setup)


# ------------------------------------------------------------------------------------------------
# device policy
# ------------------------------------------------------------------------------------------------

SRC_NONE, SRC_SAMPLED, SRC_CONST, SRC_SINSIN = (
    _lib.TFEM_SRC_NONE,
    _lib.TFEM_SRC_SAMPLED,
    _lib.TFEM_SRC_CONST,
    _lib.TFEM_SRC_SINSIN,
)


def place_mesh(mesh):
    """The assembly path is CUDA-only: move a host mesh to the current GPU or fail loudly."""
    if mesh.device.type == "cuda":
        return mesh
    if not torch.cuda.is_available():
        raise TfemError(
            "pytorch_fem_solver_b200 needs a CUDA device: the element-assembly path has no CPU implementation"
        )
    _lib.load()  # fail now, not at the first integrate_* call, if the library is missing
    # a copy: building a basis must not turn the caller's CPU mesh into a CUDA mesh behind their back
    return mesh.copy_to(torch.device("cuda", torch.cuda.current_device()))
