"""The integration engine, re-designed around fused CUDA kernels.

API and tensor shapes follow the reference's `AbstractBasis`
(torch_fem/basis/abstract_basis.py:10-195; SURVEY.md Appendix A).  What differs:

* geometry (`v_grad`, `integration_points`, `_dx`, `_inv_map_jacobian`) comes from ONE kernel
  (`tfem_tri_p1_geometry`) and is produced lazily -- the fused assembly forms never need it;
* `integrate_*` reduce over quadrature points with `tfem_quad_reduce` and scatter with a
  deterministic segmented reduction into CSR values (`tfem_scatter_*`), not `index_put_` into a
  dense `(N_d, N_d)` zero matrix (reference :81-91);
* named forms from `pytorch_fem_solver_b200.forms` skip the integrand altogether;
* results are dense tensors of the reference's shapes when they are small, CSR otherwise
  (`layout=` chooses explicitly).
"""

from __future__ import annotations

import abc
from dataclasses import dataclass
from typing import Any, Callable, Optional, Tuple

import torch

from .. import csr as csr_mod
from .. import forms, ops
from ..element.abstract_element import AbstractElement
from ..mesh.abstract_mesh import AbstractMesh

DENSE_LIMIT = 8192  # largest n_dof returned as a dense (n_dof, n_dof) tensor by default


@dataclass
class CellLayout:
    """Flattened view of the (possibly batched) triangle mesh the kernels consume."""

    coords: torch.Tensor  # (V_total, 2)
    conn: torch.Tensor  # (N_total, 3) int32, ids local to each mesh
    n_el_per_mesh: int
    n_vert_per_mesh: int
    lead: Tuple[int, ...]  # leading shape of per-element results, e.g. (N,), (P,4), (F,N)
    frac: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]] = None  # jac, inv, det, t

    @property
    def d(self) -> int:
        return 3 if self.frac is not None else 2

    @property
    def n_total(self) -> int:
        return self.conn.shape[0]

    def frac_args(self):
        return self.frac if self.frac is not None else (None, None, None, None)


class AbstractBasis(abc.ABC):
    """P1 basis on a mesh: geometry, index maps and the integrate_* family."""

    def __init__(self, mesh: AbstractMesh, element: AbstractElement):
        self._element = element
        self.mesh = ops.place_mesh(mesh)
        self._geometry = None
        self._geometry_version = 0
        self._pattern = None
        self._scatter_inverse = {}
        self._tile_plans = {}
        self._layout = self._compute_layout(self.mesh, element)
        self.v = self._reference_shape_values(element)
        (
            self._coords4global_dofs,
            self._global_dofs4elements,
            self._nodes4boundary_dofs,
            self._coords4elements,
        ) = self._compute_dofs(self.mesh, element)
        self._basis_parameters = self._compute_basis_parameters(
            self._coords4global_dofs, self._global_dofs4elements, self._nodes4boundary_dofs
        )

    # ------------------------------------------------------------------ geometry (lazy)
    def _reference_shape_values(self, element):
        nodes = element.gaussian_nodes.to(device=self._layout.coords.device, dtype=self._layout.coords.dtype)
        return element.compute_barycentric_coordinates(nodes)

    def _compute_integral_values(self):
        """One kernel for v_grad / points / dx / J^-1 (reference :42-63 as a tensor program)."""
        lay = self._layout
        inv_jac, v_grad, x_q, dx = ops.tri_geometry(
            lay.coords, lay.conn, lay.n_el_per_mesh, lay.n_vert_per_mesh, self._element.integration_order, *lay.frac_args()
        )
        q, d = x_q.shape[1], lay.d
        self._geometry = {
            "v_grad": v_grad.reshape(*lay.lead, 1, 3, d),
            "integration_points": x_q.reshape(*lay.lead, q, 1, d),
            "_dx": dx.reshape(*lay.lead, q, 1, 1),
            "_inv_map_jacobian": inv_jac.reshape(*lay.lead, 1, 2, d),
        }

    def _geo(self, name):
        if self._geometry is None:
            self._compute_integral_values()
        return self._geometry[name]

    def _set_geo(self, name, value):
        if self._geometry is None:
            self._compute_integral_values()
        self._geometry[name] = value

    v_grad = property(lambda self: self._geo("v_grad"), lambda self, v: self._set_geo("v_grad", v))
    integration_points = property(
        lambda self: self._geo("integration_points"), lambda self, v: self._set_geo("integration_points", v)
    )
    _dx = property(lambda self: self._geo("_dx"), lambda self, v: self._set_geo("_dx", v))
    _inv_map_jacobian = property(
        lambda self: self._geo("_inv_map_jacobian"), lambda self, v: self._set_geo("_inv_map_jacobian", v)
    )

    @property
    def n_q(self) -> int:
        return self._element.gaussian_nodes.shape[0]

    @property
    def dtype(self) -> torch.dtype:
        return self._layout.coords.dtype

    @property
    def device(self) -> torch.device:
        return self._layout.coords.device

    # ------------------------------------------------------------------ symbolic structures
    def _dof_conn_flat(self) -> torch.Tensor:
        """(N_total,3) int32 global DOF of each element vertex (scatter target)."""
        return self._flat_dofs

    @property
    def n_dof_flat(self) -> int:
        return self._n_dof_flat

    @property
    def pattern(self) -> csr_mod.CsrPattern:
        """CSR pattern + COO->CSR permutation of `bilinear_form_idx`, built on first use."""
        if self._pattern is None:
            self._pattern = csr_mod.build_pattern(self._dof_conn_flat(), self.n_dof_flat)
        return self._pattern

    def _inverse(self, kind: str) -> torch.Tensor:
        """Flat COO index -> output entry (adjoint of the scatter), built on first use."""
        if kind not in self._scatter_inverse:
            pat = self.pattern
            seg, perm = (pat.seg, pat.perm) if kind == "bilinear" else (pat.lin_seg, pat.lin_perm)
            counts = (seg[1:] - seg[:-1]).long()
            owner = torch.repeat_interleave(torch.arange(seg.shape[0] - 1, device=seg.device), counts)
            inverse = torch.empty_like(perm)
            inverse[perm.long()] = owner.to(torch.int32)
            self._scatter_inverse[kind] = inverse
        return self._scatter_inverse[kind]

    def tile_plan(self, rows_per_tile: int = 336, ordering: str = "auto", elem_ids: Optional[bool] = None):
        """Row-tile plan of the fused assembly kernel, cached per setting.  `elem_ids`: the instances carry the
        global id of every tile element (sampled sources, fracture networks); default: only where needed."""
        lay = self._layout
        if elem_ids is None:
            elem_ids = lay.frac is not None
        key = (rows_per_tile, ordering, bool(elem_ids))
        if key not in self._tile_plans:
            offsets = (torch.arange(lay.n_total, device=lay.conn.device) // lay.n_el_per_mesh) * lay.n_vert_per_mesh
            geom_conn = lay.conn.long() + offsets[:, None]
            dof_conn = self._dof_conn_flat()
            points = torch.zeros((self.n_dof_flat, 2), dtype=lay.coords.dtype, device=lay.coords.device)
            local = lay.coords[geom_conn.reshape(-1)].clone()
            if lay.n_total > lay.n_el_per_mesh:  # batched meshes share one local frame: keep them apart when clustering rows
                span = float(lay.coords[:, 0].max() - lay.coords[:, 0].min())  # side by side, no gaps: the blocks stay full
                local[:, 0] += span * (offsets.repeat_interleave(3) // lay.n_vert_per_mesh).to(local.dtype)
            points[dof_conn.reshape(-1).long()] = local
            self._tile_plans[key] = csr_mod.build_tile_plan(geom_conn, dof_conn, self.pattern, points, rows_per_tile, ordering,
                                                            elem_ids=bool(elem_ids))
        return self._tile_plans[key]

    #: weak-residual path: "auto" = the one-launch tiled kernel from RESIDUAL_TILED_MIN elements on (below, the tile
    #: plan's set-up outweighs the saved pass), "tiled" / "two_pass" force one (tests, benchmarks)
    residual_path = "auto"
    RESIDUAL_TILED_MIN = 1 << 16

    def _residual_tiled(self, src) -> bool:
        lay = self._layout
        supported = src.kind in (ops.SRC_SAMPLED, ops.SRC_NONE) and getattr(self, "_tiled_residual_ok", True)
        if self.residual_path == "tiled":
            if not supported:
                raise NotImplementedError("the tiled weak residual takes a sampled source (or none) on Basis / FractureBasis")
            return True
        return self.residual_path == "auto" and supported and lay.n_total >= self.RESIDUAL_TILED_MIN

    def _fracture_metric(self) -> Optional[torch.Tensor]:
        """(n_mesh, 4) = (a00, a01, a11, det J_f) with a = J_f^+ J_f^+^T: the metric in which the planar element
        vectors give the tangential gradients' inner products (fracture_basis.py:20-26)."""
        lay = self._layout
        if lay.frac is None:
            return None
        if getattr(self, "_frac_metric", None) is None:
            inv, det = lay.frac[1], lay.frac[2]  # (F,2,3), (F,)
            a = inv @ inv.mT
            self._frac_metric = torch.stack([a[:, 0, 0], a[:, 0, 1], a[:, 1, 1], det.reshape(-1)], dim=1).to(self.dtype).contiguous()
        return self._frac_metric

    def _sampled_source(self, src) -> torch.Tensor:
        """f at this basis' quadrature points, (N_total, n_q).  The points of a basis are fixed, so the samples of
        a `forms.SampledSource` are evaluated once per (source object, basis, geometry) and reused by every later
        call -- a training loop calls the residual thousands of times with the same right-hand side
        (examples/example_weak.py:64-75).  `source.refresh()` drops them (a callable with changing state)."""
        lay = self._layout
        key = (id(self), self._geometry_version, self.dtype)
        cache = getattr(src, "_samples", None)
        if cache is None or cache[0] != key:
            with torch.no_grad():
                values = src(self.integration_points).to(self.dtype).expand(*lay.lead, self.n_q, 1, 1).reshape(lay.n_total, self.n_q).contiguous()
            cache = (key, values)
            try:
                src._samples = cache
            except AttributeError:  # a source type without attribute storage: evaluate every time
                pass
        return cache[1]

    # ------------------------------------------------------------------ integrate_*
    def _reduce_integrand(self, integrand: torch.Tensor) -> torch.Tensor:
        """`(f * dx).sum(-3)` -> (N_total, a*b) for an integrand broadcastable to (*lead, q, a, b)."""
        lay = self._layout
        n_lead = len(lay.lead)
        t = integrand.to(self.dtype) if integrand.dtype != self.dtype else integrand
        while t.dim() < n_lead + 3:
            t = t.unsqueeze(0)
        a, b = t.shape[-2], t.shape[-1]
        q_i = t.shape[-3]
        if q_i not in (1, self.n_q):
            raise ValueError(f"integrand has {q_i} quadrature points, the basis has {self.n_q}")
        if all(s == 1 for s in t.shape[:n_lead]):
            t3 = t.reshape(1, q_i, a * b)
        else:
            t3 = t.expand(*lay.lead, q_i, a, b).reshape(lay.n_total, q_i, a * b)
        return ops.quad_reduce(t3, self._dx.reshape(lay.n_total, self.n_q))

    def integrate_functional(self, function: Callable[..., torch.Tensor], *args: Any, **kwargs: Any) -> torch.Tensor:
        """Per-element integral `(f * dx).sum(-3).sum(-2)` -> (*lead, b) (reference :65-72)."""
        if isinstance(function, forms.H1Error) and len(args) == 2 and not kwargs:
            return self._h1_error_fused(function, *args)
        integrand = function(self, *args, **kwargs)
        a, b = integrand.shape[-2], integrand.shape[-1]
        local = self._reduce_integrand(integrand).reshape(*self._layout.lead, a, b)
        return local.sum(-2)

    def _h1_error_fused(self, form, u, gradient) -> torch.Tensor:
        """`forms.H1Error` in one kernel (`tfem_h1_error`): no integrand, no dx tensor."""
        lay = self._layout
        key = (id(self), self._geometry_version, self.dtype)
        if form._samples is None or form._samples[0] != key:
            with torch.no_grad():
                points = self.integration_points
                ue = form.exact(points).to(self.dtype).expand(*lay.lead, self.n_q, 1, 1).reshape(lay.n_total, self.n_q).contiguous()
                ge = form.exact_grad(points).to(self.dtype).expand(*lay.lead, self.n_q, 1, lay.d).reshape(lay.n_total, self.n_q, lay.d).contiguous()
            form._samples = (key, ue, ge)
        _, ue, ge = form._samples
        uv = form.field(self, u).to(self.dtype).expand(*lay.lead, self.n_q, 1, 1).reshape(lay.n_total, self.n_q).contiguous()
        gv = form.field(self, gradient).to(self.dtype).expand(*lay.lead, self.n_q, 1, lay.d).reshape(lay.n_total, self.n_q, lay.d).contiguous()
        frac_det = lay.frac_args()[2] if lay.frac is not None else None
        out = ops.h1_error(uv.detach(), gv.detach(), ue, ge, lay.coords, lay.conn, lay.n_el_per_mesh, lay.n_vert_per_mesh,
                           self._element.integration_order, frac_det)
        return out.reshape(*lay.lead, 1)

    def integrate_bilinear_form(
        self, function: Callable[..., torch.Tensor], *args: Any, layout: Optional[str] = None, **kwargs: Any
    ) -> torch.Tensor:
        """Global operator of a bilinear form (reference :74-93).

        `layout`: "dense" (reference shape), "csr" (torch sparse CSR), "values" (CSR value
        array aligned with `basis.pattern`), None = dense up to DENSE_LIMIT DOFs, CSR above."""
        pat = self.pattern
        if isinstance(function, forms.FusedBilinear) and not args and not kwargs:
            values = self._assemble_fused(function, None)[0]
        else:
            local = self._reduce_integrand(function(self, *args, **kwargs))  # (N_total, 9)
            values = ops.scatter(local.reshape(-1), pat.seg, pat.perm, self._inverse("bilinear"))
        return self._matrix_result(values, layout)

    def integrate_linear_form(self, function: Callable[..., torch.Tensor], *args: Any, **kwargs: Any) -> torch.Tensor:
        """Global vector of a linear form (reference :95-112)."""
        pat = self.pattern
        lay = self._layout
        if isinstance(function, forms.WeakResidual) and len(args) == 1 and not kwargs:
            src = function.source
            grad = forms.WeakResidual.field(self, args[0])
            f_q = self._sampled_source(src) if src.kind == ops.SRC_SAMPLED else None
            grad_q = grad.to(self.dtype).expand(*lay.lead, self.n_q, 1, lay.d).reshape(lay.n_total, self.n_q, lay.d).contiguous()
            if self._residual_tiled(src):
                # one launch of the tiled kernel: rows sum their elements' terms, no (N,3) tensor, no scatter pass
                plan = self.tile_plan(elem_ids=True)
                frac_jac, frac_inv, frac_det, _ = lay.frac_args()
                vec = ops.weak_residual_tiled(
                    grad_q, lay.coords, lay.conn, self._dof_conn_flat(), *plan.op_args(), pat.n_dof, lay.n_el_per_mesh,
                    lay.n_vert_per_mesh, self._element.integration_order, f_q, frac_jac, frac_inv, frac_det, self._fracture_metric(),
                )
            else:
                vec = ops.weak_residual(
                    grad_q, lay.coords, lay.conn, self._dof_conn_flat(), pat.lin_seg, pat.lin_perm, lay.n_el_per_mesh,
                    lay.n_vert_per_mesh, self._element.integration_order, src.kind, list(src.params), f_q, *lay.frac_args(),
                )
        elif isinstance(function, forms.Load) and not args and not kwargs:
            vec = self._assemble_fused(None, function.source)[1]
        else:
            local = self._reduce_integrand(function(self, *args, **kwargs))  # (N_total, 3)
            vec = ops.scatter(local.reshape(-1), pat.lin_seg, pat.lin_perm, self._inverse("linear"))
        return self._vector_result(vec)

    def assemble(self, bilinear: Optional[forms.FusedBilinear], load: Optional[forms.Load], layout: Optional[str] = None,
                 path: str = "auto"):
        """Matrix and load vector of named forms in one pass (BASELINE config 2).

        `path`: "tiled" = single fused kernel over row tiles, "two_pass" = local_forms +
        scatter kernels, "auto" = tiled for planar meshes with an analytic source."""
        values, vec = self._assemble_fused(bilinear, load.source if load is not None else None, path)
        return (
            self._matrix_result(values, layout) if values is not None else None,
            self._vector_result(vec) if vec is not None else None,
        )

    def assemble_from_host(self, coords_host: torch.Tensor, bilinear, load, values_out: Optional[torch.Tensor],
                           load_out: Optional[torch.Tensor], path: str = "auto"):
        """Re-assemble for new vertex coordinates held in (pinned) HOST memory.

        Copies `coords_host` over the basis' device coordinates, runs the fused assembly and copies
        the CSR value array / load vector back into the given host tensors; everything is enqueued
        on the current stream (synchronise before reading the outputs).  The mesh topology -- and
        with it the CSR pattern and tile plan -- is unchanged, so nothing symbolic is redone."""
        lay = self._layout
        lay.coords.copy_(coords_host.reshape(lay.coords.shape), non_blocking=True)
        self._geometry = None  # cached v_grad / points / dx belong to the old coordinates
        self._geometry_version += 1
        values, vec = self._assemble_fused(bilinear, load.source if load is not None else None, path)
        hook = getattr(self, "_post_assemble_hook", None)
        if hook is not None:
            hook(values, vec)
        if values_out is not None and values is not None:
            values_out.copy_(values, non_blocking=True)
        if load_out is not None and vec is not None:
            load_out.copy_(vec.reshape(load_out.shape), non_blocking=True)
        return values_out, load_out

    def host_pipeline(self, bilinear, load, depth: int = 2) -> "HostPipeline":
        """Stream of re-assemblies fed from / drained to HOST memory, `depth` steps in flight: the
        host->device copy of step i+1, the assembly of step i and the device->host copy of step i-1 run
        on three streams (PCIe is full duplex, so throughput is set by the larger copy alone)."""
        return HostPipeline(self, bilinear, load, depth)

    def _assemble_fused(self, bilinear, source, path: str = "auto"):
        lay = self._layout
        pat = self.pattern
        order = self._element.integration_order
        src = forms.as_source(source)
        want_mat = bilinear is not None
        want_vec = source is not None
        alpha, beta = (bilinear.alpha, bilinear.beta) if want_mat else (0.0, 0.0)
        sampled = want_vec and src.kind == ops.SRC_SAMPLED
        # one launch for everything but analytic (x, y) sources on fractures, which the kernels evaluate in 3-D
        tiled_ok = lay.frac is None or not want_vec or src.kind in (ops.SRC_SAMPLED, ops.SRC_CONST, ops.SRC_NONE)
        if path == "tiled" and not tiled_ok:
            raise NotImplementedError("tiled assembly on a fracture network needs a sampled or constant source")
        if path == "tiled" or (path == "auto" and tiled_ok):
            plan = self.tile_plan(elem_ids=sampled or lay.frac is not None)
            values = torch.empty(pat.nnz, dtype=self.dtype, device=self.device) if want_mat else None
            vec = torch.empty(pat.n_dof, dtype=self.dtype, device=self.device) if want_vec else None
            ops.assemble_csr_tiled(plan, lay.coords, order, alpha, beta, src.kind if want_vec else 0, src.params, values, vec,
                                   self._sampled_source(src) if sampled else None, lay.n_el_per_mesh, self._fracture_metric())
            return values, vec
        f_q = self._sampled_source(src) if want_vec and src.kind == ops.SRC_SAMPLED else None
        local_mat, local_vec = ops.local_forms(
            lay.coords, lay.conn, lay.n_el_per_mesh, lay.n_vert_per_mesh, order, alpha, beta, want_mat,
            src.kind if want_vec else 0, list(src.params), f_q, *lay.frac_args(),
        )
        values = ops.scatter(local_mat.reshape(-1), pat.seg, pat.perm, self._inverse("bilinear")) if want_mat else None
        vec = ops.scatter(local_vec.reshape(-1), pat.lin_seg, pat.lin_perm, self._inverse("linear")) if want_vec else None
        return values, vec

    def _matrix_result(self, values: torch.Tensor, layout: Optional[str]) -> torch.Tensor:
        pat = self.pattern
        if layout is None:
            layout = "dense" if pat.n_dof <= DENSE_LIMIT else "csr"
        if layout == "values":
            return values
        if layout == "csr":
            return pat.to_sparse_csr(values)
        if layout == "dense":
            return pat.to_dense(values)
        raise ValueError(f"unknown layout {layout!r}")

    def _vector_result(self, vec: torch.Tensor) -> torch.Tensor:
        return vec.reshape(-1, 1)

    # ------------------------------------------------------------------ dense helpers (unchanged behaviour)
    def reduce(self, tensor: torch.Tensor):
        """Restrict to interior DOFs (reference :114-117)."""
        idx = self._basis_parameters["inner_dofs"]
        if tensor.layout == torch.sparse_csr:
            return self._reduce_csr(tensor, idx)
        return tensor[idx, :][:, idx] if tensor.size(-1) != 1 else tensor[idx]

    @staticmethod
    def _reduce_csr(matrix: torch.Tensor, inner: torch.Tensor) -> torch.Tensor:
        """`A[inner][:, inner]` of a CSR matrix as a CSR matrix in the compact interior numbering (the dense
        fancy-indexing of the reference, abstract_basis.py:114-117, without densifying: config 2 would be 35 TB)."""
        n = matrix.shape[-1]
        crow, col, val = matrix.crow_indices(), matrix.col_indices(), matrix.values()
        rank = torch.full((n,), -1, dtype=torch.int64, device=col.device)
        rank[inner] = torch.arange(inner.numel(), device=col.device)
        row_of = torch.repeat_interleave(torch.arange(n, device=col.device), (crow[1:] - crow[:-1]).long())
        keep = (rank[row_of] >= 0) & (rank[col.long()] >= 0)
        new_row = rank[row_of[keep]]
        counts = torch.bincount(new_row, minlength=inner.numel())
        new_crow = torch.zeros(inner.numel() + 1, dtype=crow.dtype, device=col.device)
        new_crow[1:] = torch.cumsum(counts, 0)
        return torch.sparse_csr_tensor(new_crow, rank[col.long()[keep]].to(col.dtype), val[keep], size=(inner.numel(), inner.numel()),
                                       device=val.device)  # (explicit: a default-device context must not move the result)

    def reshape_for_assembly(self, local_matrices: torch.Tensor, form: str) -> torch.Tensor:
        """Flatten local matrices in COO order (reference :162-171)."""
        if form == "bilinear":
            return local_matrices.reshape(-1)
        if form == "linear":
            return local_matrices.reshape(-1, 1)
        raise NotImplementedError(f"Unknown form type: {form}")

    def solution_tensor(self) -> torch.Tensor:
        """Zero vector of shape (nb_dofs, 1) (reference :173-175)."""
        return torch.zeros(self._basis_parameters["linear_form_shape"], dtype=self.dtype, device=self.device)

    def inner_dofs_mask(self) -> torch.Tensor:
        """uint8 [nb_dofs]: 1 on the inner DOFs -- the keep mask of the CSR solve (build `sparse.amg` with it)."""
        keep = torch.zeros(self._basis_parameters["linear_form_shape"][0], dtype=torch.uint8, device=self.device)
        keep[self._basis_parameters["inner_dofs"]] = 1
        return keep

    def solve(self, matrix: torch.Tensor, solution: torch.Tensor, vector: torch.Tensor, only_inner_dofs: bool = True,
              rtol: float = 1e-10, max_iterations=None, preconditioner=None):
        """Solve the (reduced) system and add the result to `solution` (reference :177-195).

        Dense matrices take the reference's direct solve.  A CSR matrix too large to densify
        (more than DENSE_LIMIT unknowns) is solved by preconditioned conjugate gradients on the
        CSR arrays (`sparse.cg`, symmetric positive definite systems such as stiffness / mass);
        the run's `sparse.CgInfo` is kept in `self.last_solve_info`.  `preconditioner`: on that path, a
        `sparse.amg(matrix, self.inner_dofs_mask())` hierarchy (built with keep=None when
        only_inner_dofs is False) replaces Jacobi; the direct solve ignores it."""
        inner = self._basis_parameters["inner_dofs"]
        if matrix.layout == torch.sparse_csr and matrix.shape[-1] > DENSE_LIMIT:
            from .. import sparse

            keep = None
            if only_inner_dofs:
                keep = torch.zeros(matrix.shape[-1], dtype=torch.uint8, device=matrix.device)
                keep[inner] = 1
            x, info = sparse.cg(matrix.crow_indices().to(torch.int32), matrix.col_indices().to(torch.int32), matrix.values(),
                                vector, keep, rtol=rtol, max_iterations=max_iterations, preconditioner=preconditioner)
            self.last_solve_info = info
            if not info.converged:
                raise RuntimeError(f"conjugate gradients stopped at relative residual {info.relative_residual:.3e} "
                                   f"after {info.iterations} iterations")
            if only_inner_dofs:
                solution[inner] += x[inner].reshape(-1, 1)
            else:
                solution += x.reshape(solution.shape)
            return solution
        if only_inner_dofs:
            matrix = self.reduce(matrix)
            vector = self.reduce(vector)
        elif matrix.layout == torch.sparse_csr:
            matrix = matrix.to_dense()
        solution[inner] += torch.linalg.solve(matrix, vector)
        return solution

    # ------------------------------------------------------------------ subclass hooks
    @abc.abstractmethod
    def _compute_layout(self, mesh, element) -> CellLayout:
        raise NotImplementedError

    @abc.abstractmethod
    def _compute_dofs(self, mesh, element):
        raise NotImplementedError

    @abc.abstractmethod
    def _compute_basis_parameters(self, coords4global_dofs, global_dofs4elements, nodes4boundary_dofs) -> dict:
        raise NotImplementedError


class HostPipeline:
    """Double-buffered host -> assembly -> host pipeline of one basis (planar mesh, analytic source).

    `step(coords_host, values_host, load_host)` enqueues one re-assembly for new vertex coordinates in
    pinned host memory and returns immediately; results land in the given pinned host tensors in
    submission order.  `synchronize()` waits for everything submitted.  The mesh topology, CSR
    pattern and tile plan are those of the basis (nothing symbolic is redone)."""

    def __init__(self, basis: "AbstractBasis", bilinear, load, depth: int = 2):
        lay, pat = basis._layout, basis.pattern
        src = forms.as_source(load.source if load is not None else None)
        if lay.frac is not None or src.kind == ops.SRC_SAMPLED:
            raise NotImplementedError("the host pipeline drives the tiled kernel: planar mesh and analytic source")
        self.basis, self.depth = basis, max(int(depth), 1)
        self.want_mat, self.want_vec = bilinear is not None, load is not None
        self.alpha, self.beta = (bilinear.alpha, bilinear.beta) if self.want_mat else (0.0, 0.0)
        self.src = src
        self.order = basis._element.integration_order
        self.plan = basis.tile_plan()
        device, dtype = basis.device, basis.dtype
        self.coords = [torch.empty_like(lay.coords) for _ in range(self.depth)]
        self.values = [torch.empty(pat.nnz, dtype=dtype, device=device) if self.want_mat else None for _ in range(self.depth)]
        self.load = [torch.empty(pat.n_dof, dtype=dtype, device=device) if self.want_vec else None for _ in range(self.depth)]
        self.copy_in, self.compute, self.copy_out = (torch.cuda.Stream(device=device) for _ in range(3))
        self.in_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.compute_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.out_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.submitted = 0

    def step(self, coords_host: torch.Tensor, values_host: Optional[torch.Tensor], load_host: Optional[torch.Tensor]):
        k = self.submitted % self.depth
        recycled = self.submitted >= self.depth
        with torch.cuda.stream(self.copy_in):
            if recycled:
                self.copy_in.wait_event(self.compute_done[k])  # the assembly that read this coordinate buffer
            self.coords[k].copy_(coords_host.reshape(self.coords[k].shape), non_blocking=True)
            self.in_done[k].record(self.copy_in)
        with torch.cuda.stream(self.compute):
            self.compute.wait_event(self.in_done[k])
            if recycled:
                self.compute.wait_event(self.out_done[k])  # the copy that drained these output buffers
            ops.assemble_csr_tiled(self.plan.c_struct(), self.coords[k], self.order, self.alpha, self.beta,
                                   self.src.kind if self.want_vec else 0, self.src.params, self.values[k], self.load[k])
            self.compute_done[k].record(self.compute)
        with torch.cuda.stream(self.copy_out):
            self.copy_out.wait_event(self.compute_done[k])
            if values_host is not None and self.want_mat:
                values_host.copy_(self.values[k], non_blocking=True)
            if load_host is not None and self.want_vec:
                load_host.copy_(self.load[k].reshape(load_host.shape), non_blocking=True)
            self.out_done[k].record(self.copy_out)
        self.submitted += 1

    def synchronize(self):
        for stream in (self.copy_in, self.compute, self.copy_out):
            stream.synchronize()


class LazyParameters(dict):
    """dict whose expensive entries (the 9N-long COO index maps) are built on first access."""

    def __init__(self, eager: dict, lazy: dict):
        super().__init__(eager)
        self._lazy = lazy

    def __missing__(self, key):
        if key in self._lazy:
            self[key] = self._lazy[key]()
            return self[key]
        raise KeyError(key)

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in self._lazy
