"""Stiffness and mass forms with coefficient fields (DESIGN.md section 8(g)) without a GPU: the numpy restatement of the
weighted local forms against `FusedBilinear.__call__`, the host logic of `Basis.assemble` with field coefficients
through an oracle-backed stand-in for `ops.weighted_local_forms` (defined here; tests/cpu_shim.py covers the older
ops), every error case, C-ABI argument validation, and AMG iteration counts on a high-contrast problem.  The kernel
itself is checked in tests/test_coefficient_forms_gpu.py."""

import numpy as np
import pytest
import torch

import pytorch_fem_solver_b200 as tfem
from oracle import amg_oracle as ao
from oracle import fem_oracle as fo
from pytorch_fem_solver_b200 import _lib, forms, meshgen, ops
from tests import api_checks, cpu_shim
from tests import coefficient_oracle as co

CALLS = []


def _weighted_local_forms(coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, alpha, beta, alpha_q, beta_q,
                          source_kind, source_p, f_q=None, frac_jac=None, frac_inv=None, frac_det=None, frac_t=None):
    """Stand-in for ops.weighted_local_forms: the oracle's weighted forms; records its field arguments."""
    CALLS.append({"alpha": alpha, "beta": beta, "alpha_q": alpha_q, "beta_q": beta_q})
    c, k, n_mesh = cpu_shim._batched(coords, conn, n_el_per_mesh, n_vert_per_mesh)
    geo = fo.tri_geometry(c, k, quad_order, cpu_shim._frac(n_mesh, frac_jac, frac_inv, frac_det, frac_t))
    lead = geo["integration_points"].shape[:-2]
    field = lambda q, const: const if q is None else cpu_shim._np(q).reshape(lead + (1, 1))  # noqa: E731
    integrand = co.form_weighted_stiffness_mass(geo, field(alpha_q, alpha), field(beta_q, beta))
    mat = torch.from_numpy(fo.quad_reduce(integrand, geo["dx"]).reshape(-1, 3, 3)).to(coords.dtype)
    _, vec = cpu_shim.local_forms(coords, conn, n_el_per_mesh, n_vert_per_mesh, quad_order, 0.0, 0.0, False, source_kind,
                                  source_p, f_q, frac_jac, frac_inv, frac_det, frac_t)
    return mat, vec


def _install(monkeypatch):
    cpu_shim.install(monkeypatch)
    monkeypatch.setattr(ops, "weighted_local_forms", _weighted_local_forms)
    CALLS.clear()


def kappa_fn(points):
    return 1.0 + 3.0 * points[..., 0:1] ** 2 + points[..., 1:2]


def c_fn(points):
    return 2.0 + torch.sin(3.0 * points[..., 0:1]) * points[..., 1:2]


def _generic(basis, form):
    return basis.integrate_bilinear_form(lambda b: form(b), layout="dense")


def _single(g, order):
    return tfem.Basis(tfem.MeshTri(api_checks.mesh_dict(g)), tfem.ElementTri(1, order))


def _fractures(g, order=2):
    n_f = g["in_vertices"].shape[0]
    keys = ["vertices", "triangles", "vertex_markers", "edges", "edge_markers", "neighbors"]
    meshes = [{k: g["in_" + k][f] for k in keys if "in_" + k in g} for f in range(n_f)]
    return tfem.FractureBasis(tfem.FracturesTri(meshes, torch.tensor(g["in_fractures_3d_data"])), tfem.ElementTri(1, order))


# ---------------------------------------------------------------------------------------------- the numpy restatement
@pytest.mark.parametrize("name,order", [("structured4x4", 1), ("structured6x5_jitter", 3), ("delaunay60", 4), ("delaunay60", 2)])
def test_oracle_matches_the_generic_route(golden, monkeypatch, name, order):
    _install(monkeypatch)
    g = golden(name)
    with api_checks.default_device("cpu"):
        basis = _single(g, order)
        coords, conn = g["in_vertices"], g["in_triangles"].astype(np.int64)
        geo = fo.tri_geometry(coords, conn, order)
        pts = geo["integration_points"]
        a = kappa_fn(torch.from_numpy(pts)).numpy()
        b = c_fn(torch.from_numpy(pts)).numpy()
        expect = fo.scatter_bilinear_dense(fo.quad_reduce(co.form_weighted_stiffness_mass(geo, a, b), geo["dx"]), conn, coords.shape[0])
        api_checks.close(_generic(basis, forms.StiffnessMass(kappa_fn, c_fn)), expect, what="generic route")
        # constant fields restate the existing form
        ones = np.ones(pts.shape[:-1] + (1,))
        np.testing.assert_allclose(co.form_weighted_stiffness_mass(geo, ones, ones), fo.form_stiffness_mass(geo), rtol=1e-15, atol=0)


# ---------------------------------------------------------------------------------------------- host logic
def test_field_coefficients_reach_the_new_op(golden, monkeypatch):
    _install(monkeypatch)
    with api_checks.default_device("cpu"):
        basis = _single(golden("delaunay60"), 3)
        form = forms.StiffnessMass(kappa_fn, 0.5)
        mat, vec = basis.assemble(form, forms.Load(forms.SinSinSource()), layout="dense")
        assert len(CALLS) == 1
        call = CALLS[0]
        assert call["beta_q"] is None and call["beta"] == 0.5
        aq = call["alpha_q"]
        assert aq.shape == (basis._layout.n_total, basis.n_q) and aq.is_contiguous() and aq.dtype == basis.dtype
        api_checks.close(mat, api_checks.npy(_generic(basis, form)), what="fused vs generic")
        api_checks.close(vec, api_checks.npy(basis.assemble(None, forms.Load(forms.SinSinSource()), path="two_pass")[1]), rtol=0,
                         what="load")


def test_number_coefficients_never_reach_the_new_op(golden, monkeypatch):
    _install(monkeypatch)
    with api_checks.default_device("cpu"):
        basis = _single(golden("structured4x4"), 2)
        for form in (forms.StiffnessMass(2.0, 3.0), forms.Stiffness(np.float64(1.5)), forms.Mass(torch.tensor(0.25))):
            assert not form.has_field and isinstance(form.alpha, float) and isinstance(form.beta, float)
            for path in ("two_pass", "tiled", "auto"):
                basis.assemble(form, forms.Load(), path=path)
            basis.integrate_bilinear_form(form)
        assert CALLS == []


def test_callables_are_sampled_once_and_resampled_after_refresh_and_moves(golden, monkeypatch):
    _install(monkeypatch)
    count = {"n": 0}

    def kappa(points):
        count["n"] += 1
        return kappa_fn(points)

    with api_checks.default_device("cpu"):
        g = {k: v.copy() for k, v in golden("structured6x5_jitter").items()}  # the moved coordinates may alias the arrays
        basis = _single(g, 3)
        form = forms.Stiffness(kappa)
        first = basis.assemble(form, None, layout="values")[0]
        basis.assemble(form, None, layout="values")
        basis.integrate_bilinear_form(form, layout="values")
        assert count["n"] == 1
        samples = form.alpha._samples[1]
        form.refresh()
        basis.assemble(form, None, layout="values")
        assert count["n"] == 2
        assert torch.equal(form.alpha._samples[1], samples)
        # moved points: assemble_from_host bumps the geometry version, the samples are taken again
        coords = basis._layout.coords.clone()
        moved = coords * 1.1
        values = torch.empty_like(first)
        basis.assemble_from_host(moved, form, None, values, None, path="two_pass")
        assert count["n"] == 3
        assert not torch.equal(form.alpha._samples[1], samples)
        # a second form owns its own samples
        other = forms.Stiffness(kappa)
        basis.assemble(other, None)
        assert count["n"] == 4


def test_broadcast_tensor_coefficients(golden, monkeypatch):
    _install(monkeypatch)
    with api_checks.default_device("cpu"):
        basis = _single(golden("delaunay60"), 4)
        n, q = basis._layout.n_total, basis.n_q
        per_element = torch.linspace(1.0, 5.0, n).reshape(n, 1, 1, 1)
        per_point = torch.linspace(0.5, 2.0, n * q).reshape(n, q, 1, 1)
        for alpha, beta in ((per_element, per_point), (per_point, 1.5), (0.0, per_element), (per_element, 0.0)):
            form = forms.StiffnessMass(alpha, beta)
            CALLS.clear()
            mat = basis.assemble(form, None, layout="dense")[0]
            api_checks.close(mat, api_checks.npy(_generic(basis, form)), what="tensor fields")
            for got, given in ((CALLS[0]["alpha_q"], alpha), (CALLS[0]["beta_q"], beta)):
                if isinstance(given, torch.Tensor):
                    assert torch.equal(got, given.expand(n, q, 1, 1).reshape(n, q))
                else:
                    assert got is None


@pytest.mark.parametrize("name", ["fractures2_4x2", "fractures2_8x4"])
def test_per_fracture_coefficients(golden, monkeypatch, name):
    _install(monkeypatch)
    with api_checks.default_device("cpu"):
        basis = _fractures(golden(name))
        f, n = basis._layout.lead
        transmissivity = torch.tensor([3.0, 0.25][:f] + [1.0] * max(f - 2, 0)).reshape(f, 1, 1, 1, 1)
        form = forms.StiffnessMass(transmissivity, lambda pts: 1.0 + pts[..., 2:3] ** 2)
        mat, vec = basis.assemble(form, forms.Load(lambda pts: pts[..., 0:1]), layout="dense")
        api_checks.close(mat, api_checks.npy(_generic(basis, form)), what="per-fracture")
        assert CALLS[0]["alpha_q"].shape == (f * n, basis.n_q)
        assert torch.equal(CALLS[0]["alpha_q"][:n], torch.full((n, basis.n_q), 3.0))


def test_patches_and_batched_meshes(golden, monkeypatch):
    _install(monkeypatch)
    g = golden("patches_l2")
    with api_checks.default_device("cpu"):
        basis = tfem.PatchesBasis(tfem.Patches(torch.tensor(g["in_centers"]), torch.tensor(g["in_radius"])), tfem.ElementTri(1, 2))
        lead = basis._layout.lead
        form = forms.StiffnessMass(torch.linspace(1.0, 2.0, lead[0]).reshape(lead[0], 1, 1, 1, 1), c_fn)
        api_checks.close(basis.assemble(form, None, layout="dense")[0], api_checks.npy(_generic(basis, form)), what="patches")
        meshes = tfem.MeshesTri([meshgen.structured_rectangle(6, 5, jitter=0.2, seed=s, topology=False) for s in range(5)])
        batched = tfem.PatchesBasis(meshes, tfem.ElementTri(1, 3))
        form = forms.StiffnessMass(kappa_fn, torch.linspace(1.0, 2.0, 5).reshape(5, 1, 1, 1, 1))
        api_checks.close(batched.assemble(form, None, layout="dense")[0], api_checks.npy(_generic(batched, form)), what="batched")


# ---------------------------------------------------------------------------------------------- errors
def test_errors_raise_before_any_launch(golden, monkeypatch):
    _install(monkeypatch)
    with api_checks.default_device("cpu"):
        basis = _single(golden("structured4x4"), 3)
        n, q = basis._layout.n_total, basis.n_q
        with pytest.raises(ValueError, match="broadcast"):
            basis.assemble(forms.Stiffness(torch.ones(n + 1, 1, 1, 1)), None)
        with pytest.raises(ValueError, match="broadcast"):
            basis.assemble(forms.Mass(torch.ones(n, q + 1, 1, 1)), None)
        with pytest.raises(ValueError, match="broadcast"):
            basis.assemble(forms.Mass(torch.ones(n, q, 1, 2)), None)
        with pytest.raises(ValueError, match="on meta"):
            basis.assemble(forms.Mass(torch.ones(n, 1, 1, 1, device="meta")), None)
        grad = torch.ones(n, 1, 1, 1, requires_grad=True)
        with pytest.raises(ValueError, match="generic route"):
            basis.assemble(forms.Stiffness(grad), None)
        with torch.no_grad():
            basis.assemble(forms.Stiffness(grad), None)  # no grad mode: the values are taken as data
        with pytest.raises(NotImplementedError):
            basis.assemble(forms.Stiffness(kappa_fn), forms.Load(), path="tiled")
        with pytest.raises(NotImplementedError):
            basis.host_pipeline(forms.StiffnessMass(kappa_fn, 1.0), forms.Load())
        assert len(CALLS) == 1  # only the no-grad call launched
        # the generic route differentiates with respect to the coefficient
        out = basis.integrate_bilinear_form(lambda b: forms.Stiffness(grad)(b), layout="values")
        out.sum().backward()
        assert grad.grad is not None and grad.grad.shape == grad.shape


def test_distributed_assembly_rejects_field_coefficients():
    from pytorch_fem_solver_b200.distributed import PartitionedFractureAssembly

    assembly = object.__new__(PartitionedFractureAssembly)  # the check comes before any of its state is used
    with pytest.raises(NotImplementedError, match="constant coefficients"):
        assembly.step(forms.Stiffness(kappa_fn), None)


# ---------------------------------------------------------------------------------------------- C ABI
def test_argument_validation_of_the_weighted_entry_points():
    lib = _lib.load()
    fake = _lib.ctypes.addressof(_lib.ctypes.create_string_buffer(64))  # never dereferenced: the checks below fail first
    form = _lib.Bilinear(1.0, 1.0)
    src = _lib.make_source()
    for fn in (lib.tfem_tri_p1_weighted_local_forms_f64, lib.tfem_tri_p1_weighted_local_forms_f32):
        assert fn(4, 4, 6, None, None, 3, None, None, None, None, form, src, None, fake, fake, fake, None, None) == -1  # NULL coords
        assert fn(4, 4, 6, fake, fake, 7, None, None, None, None, form, src, None, fake, fake, fake, None, None) == -2  # order 7
        assert fn(-1, 4, 6, fake, fake, 3, None, None, None, None, form, src, None, fake, fake, fake, None, None) == -1  # n_el < 0
        assert fn(0, 4, 6, None, None, 3, None, None, None, None, form, src, None, None, None, None, None, None) == 0  # nothing to do
        assert fn(4, 4, 6, fake, fake, 3, None, None, None, None, None, src, None, None, fake, fake, None, None) == -1  # no alpha
        sampled = _lib.make_source(_lib.TFEM_SRC_SAMPLED)
        assert fn(4, 4, 6, fake, fake, 3, None, None, None, None, form, sampled, None, fake, fake, fake, fake, None) == -1  # no f_q
        assert fn(4, 4, 6, fake, fake, 3, None, None, fake, None, form, src, None, fake, fake, fake, None, None) == -1  # half a fracture


# ---------------------------------------------------------------------------------------------- AMG on a high-contrast operator
def test_amg_oracle_iterations_on_a_high_contrast_problem():
    """kappa = 1e4 on an 8 x 8 checkerboard, 1 elsewhere, 128 x 128: the oracle's V-cycle needs 31 iterations at rtol
    1e-9, Jacobi 753."""
    mesh = meshgen.structured_rectangle(128, 128, jitter=0.25, seed=3, topology=False)
    a, keep, b = co.high_contrast_poisson(mesh)
    levels, coarse_inv = ao.hierarchy(a, keep)
    _, iterations = ao.pcg(a, b, keep, lambda r: ao.vcycle(levels, coarse_inv, r), rtol=1e-9)
    _, jacobi = ao.pcg(a, b, keep, rtol=1e-9)
    assert iterations <= AMG_BOUND
    assert jacobi > 5 * iterations


AMG_BOUND = 40
