"""Stiffness and mass forms with coefficient fields on the device (DESIGN.md section 8(g)): `tfem_tri_p1_weighted_local_forms`
against the generic route (callable integrand -> quad_reduce -> scatter), constant fields against the constant kernel,
the load vector, determinism, and AMG solves and refreshes on a high-contrast operator."""

import numpy as np
import pytest
import torch

import pytorch_fem_solver_b200 as tfem
from pytorch_fem_solver_b200 import forms, meshgen, sparse
from tests import api_checks
from tests.conftest import load_golden

pytestmark = pytest.mark.gpu

RTOL = {torch.float64: 1e-12, torch.float32: 1e-5}


def kappa_fn(points):
    return 1.0 + 3.0 * points[..., 0:1] ** 2 + points[..., 1:2]


def c_fn(points):
    return 2.0 + torch.sin(3.0 * points[..., 0:1]) * points[..., 1:2]


def _rel(actual, expected):
    return float((actual - expected).abs().max() / expected.abs().max())


def _bitwise(x, y):
    bits = torch.int64 if x.dtype == torch.float64 else torch.int32
    return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.contiguous().view(bits), y.contiguous().view(bits))


def _on_device(make, dtype):
    previous = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        with torch.device("cuda"):
            return make()
    finally:
        torch.set_default_dtype(previous)


def _fractures(g, order):
    n_f = g["in_vertices"].shape[0]
    keys = ["vertices", "triangles", "vertex_markers", "edges", "edge_markers", "neighbors"]
    meshes = [{k: g["in_" + k][f] for k in keys if "in_" + k in g} for f in range(n_f)]
    return tfem.FractureBasis(tfem.FracturesTri(meshes, torch.tensor(g["in_fractures_3d_data"])), tfem.ElementTri(1, order))


def _patches(g, order):
    return tfem.PatchesBasis(tfem.Patches(torch.tensor(g["in_centers"]), torch.tensor(g["in_radius"])), tfem.ElementTri(1, order))


MESHES = {
    "jittered": lambda o: tfem.Basis(tfem.MeshTri(meshgen.structured_rectangle(40, 30, jitter=0.25, seed=5, topology=False)),
                                     tfem.ElementTri(1, o)),
    "permuted": lambda o: tfem.Basis(tfem.MeshTri(meshgen.permute_mesh(meshgen.structured_rectangle(36, 28, jitter=0.25, seed=6,
                                                                                                    topology=False))),
                                     tfem.ElementTri(1, o)),
    "delaunay": lambda o: tfem.Basis(tfem.MeshTri(api_checks.mesh_dict(load_golden("delaunay60"))), tfem.ElementTri(1, o)),
    "batched": lambda o: tfem.PatchesBasis(tfem.MeshesTri([meshgen.structured_rectangle(6, 5, jitter=0.2, seed=s, topology=False)
                                                    for s in range(7)]), tfem.ElementTri(1, o)),
    "fractures": lambda o: _fractures(load_golden("fractures2_8x4"), o),
    "patches": lambda o: _patches(load_golden("patches_l2"), o),
}


def _kinds(basis):
    lay = basis._layout
    n, q, lead = lay.n_total, basis.n_q, lay.lead
    gen = torch.Generator(device="cuda").manual_seed(3)
    per_element = (0.5 + torch.rand(n, generator=gen, device="cuda", dtype=basis.dtype)).reshape(*lead, 1, 1, 1)
    per_point = (0.5 + torch.rand(n * q, generator=gen, device="cuda", dtype=basis.dtype)).reshape(*lead, q, 1, 1)
    kinds = {"callable": (kappa_fn, c_fn), "per_element": (per_element, 0.75), "per_point": (2.0, per_point),
             "mixed": (per_point, per_element)}
    if lay.frac is not None:
        f = lead[0]
        kinds["per_fracture"] = (torch.linspace(0.1, 10.0, f, device="cuda", dtype=basis.dtype).reshape(f, 1, 1, 1, 1), 1.0)
    return kinds


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("mesh", list(MESHES))
def test_parity_with_the_generic_route(mesh, order, dtype):
    basis = _on_device(lambda: MESHES[mesh](order), dtype)
    for kind, (alpha, beta) in _kinds(basis).items():
        form = forms.StiffnessMass(alpha, beta)
        fused = basis.assemble(form, None, layout="values")[0]
        generic = basis.integrate_bilinear_form(lambda b: form(b), layout="values")
        assert fused.dtype == dtype
        assert _rel(fused, generic) <= RTOL[dtype], (mesh, order, kind, _rel(fused, generic))


@pytest.mark.parametrize("mesh", ["jittered", "fractures", "batched"])
def test_constant_fields_match_the_constant_kernel(mesh):
    basis = _on_device(lambda: MESHES[mesh](3), torch.float64)
    lay = basis._layout
    a = torch.full((*lay.lead, 1, 1, 1), 2.5, device="cuda", dtype=torch.float64)
    b = torch.full((*lay.lead, basis.n_q, 1, 1), 0.75, device="cuda", dtype=torch.float64)
    fields = basis.assemble(forms.StiffnessMass(a, b), None, layout="values", path="two_pass")[0]
    constants = basis.assemble(forms.StiffnessMass(2.5, 0.75), None, layout="values", path="two_pass")[0]
    assert _rel(fields, constants) <= 1e-13


@pytest.mark.parametrize("source", ["sinsin", "const", "sampled"])
@pytest.mark.parametrize("mesh", ["jittered", "fractures"])
def test_load_vector_is_that_of_the_two_pass_path(mesh, source):
    basis = _on_device(lambda: MESHES[mesh](4), torch.float64)
    src = {"sinsin": forms.SinSinSource(), "const": forms.ConstSource(1.5), "sampled": forms.SampledSource(c_fn)}[source]
    _, vec = basis.assemble(forms.StiffnessMass(kappa_fn, c_fn), forms.Load(src))
    _, ref = basis.assemble(None, forms.Load(src), path="two_pass")
    assert _bitwise(vec, ref)


def test_two_runs_are_bitwise_equal():
    basis = _on_device(lambda: MESHES["permuted"](4), torch.float64)
    form = forms.StiffnessMass(kappa_fn, c_fn)
    first = basis.assemble(form, forms.Load(), layout="values")
    form.refresh()
    second = basis.assemble(form, forms.Load(), layout="values")
    assert _bitwise(first[0], second[0]) and _bitwise(first[1], second[1])


def checkerboard(contrast, blocks=8):
    def kappa(points):
        cell = torch.floor(points.clamp(0.0, 1.0 - 1e-12) * blocks)
        dark = (cell[..., 0:1] + cell[..., 1:2]) % 2 == 0
        return torch.where(dark, torch.full_like(cell[..., 0:1], contrast), torch.ones_like(cell[..., 0:1]))

    return kappa


def per_element(basis, kappa):
    """kappa at each element's centroid, (N, 1, 1, 1): a material table.  A discontinuous kappa sampled per point would
    meet the negative centroid weight of the 4-point rule and can make element matrices indefinite."""
    return kappa(basis.integration_points.mean(dim=-3, keepdim=True))


def _contrast_problem(nx, ny, contrast):
    def make():
        mesh = tfem.MeshTri(meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False))
        return tfem.Basis(mesh, tfem.ElementTri(1, 3))

    return _on_device(make, torch.float64)


AMG_ITERATIONS_512 = 60


def test_high_contrast_solve_with_amg():
    """-div(kappa grad u) = f, kappa = 1e4 on an 8 x 8 checkerboard (one value per element), 512 x 512, rtol 1e-9."""
    basis = _contrast_problem(512, 512, 1e4)
    a, load = basis.assemble(forms.Stiffness(per_element(basis, checkerboard(1e4))), forms.Load(), layout="csr")
    keep = basis.inner_dofs_mask()
    x_amg = basis.solve(a, basis.solution_tensor(), load, rtol=1e-9, preconditioner=sparse.amg(a, keep))
    amg_info = basis.last_solve_info
    x_jac = basis.solve(a, basis.solution_tensor(), load, rtol=1e-9, max_iterations=100000)
    jacobi_info = basis.last_solve_info
    assert amg_info.converged and amg_info.iterations <= AMG_ITERATIONS_512, amg_info
    assert jacobi_info.iterations > 5 * amg_info.iterations, (jacobi_info, amg_info)
    assert _rel(x_amg, x_jac) <= 1e-6


def _same_hierarchy(h, fresh):
    assert len(h.levels) == len(fresh.levels)
    assert _bitwise(h.coarse_inv, fresh.coarse_inv)
    for mine, ref in zip(h.levels, fresh.levels):
        for name in ("a_val", "p_val", "r_val", "wdinv"):
            assert _bitwise(getattr(mine, name), getattr(ref, name)), name
        for name in ("a_crow", "a_col", "p_crow", "p_col", "r_crow", "r_col", "agg"):
            assert torch.equal(getattr(mine, name), getattr(ref, name)), name


def test_refresh_after_a_coefficient_change():
    """Refresh the hierarchy of kappa = 1e4 (checkerboard) for new coefficients on the same pattern.  kappa -> 2 kappa keeps
    the strength graph, so the refreshed hierarchy is a fresh `amg()` of the new matrix bit for bit.  A contrast change
    to 1e2 changes the aggregation a fresh build would choose (the oracle shows it at 128 x 128), so there the refreshed
    hierarchy keeps the old aggregates and is checked by its convergence."""
    basis = _contrast_problem(512, 512, 1e4)
    keep = basis.inner_dofs_mask()
    kappa = per_element(basis, checkerboard(1e4))
    a0, load = basis.assemble(forms.Stiffness(kappa), forms.Load(), layout="csr")
    h = sparse.amg(a0, keep, refreshable=True)
    a2 = basis.assemble(forms.Stiffness(2.0 * kappa), None, layout="csr")[0]
    h.refresh(a2.values())
    _same_hierarchy(h, sparse.amg(a2, keep))
    a1 = basis.assemble(forms.Stiffness(per_element(basis, checkerboard(1e2))), None, layout="csr")[0]
    assert torch.equal(a1.crow_indices(), a0.crow_indices()) and torch.equal(a1.col_indices(), a0.col_indices())
    h.refresh(a1.values())
    basis.solve(a1, basis.solution_tensor(), load, rtol=1e-9, preconditioner=h)
    assert basis.last_solve_info.converged and basis.last_solve_info.iterations <= AMG_ITERATIONS_512
