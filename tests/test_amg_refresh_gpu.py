"""Numeric-only refresh of an AMG hierarchy on the device (tfem_csr_spgemm_numeric, tfem_amg_diag, tfem_amg_smoother,
tfem_gather, `AmgHierarchy.refresh`): bitwise against tfem_csr_spgemm and a fresh build, against the refresh oracle
(tests/amg_refresh_oracle.py), and in the solves that take the refreshed hierarchy."""

import math

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import pytorch_fem_solver_b200 as tfem
from oracle import amg_oracle as ao
from pytorch_fem_solver_b200 import forms, meshgen, ops, sparse
from tests import amg_refresh_oracle as ro

pytestmark = pytest.mark.gpu


def _scipy(crow, col, val, n_cols):
    return sp.csr_matrix((val.double().cpu().numpy(), col.cpu().numpy().astype(np.int64), crow.cpu().numpy().astype(np.int64)),
                         shape=(crow.shape[0] - 1, n_cols))


def _cuda_csr(a, dtype=torch.float64):
    a = sp.csr_matrix(a)
    a.sort_indices()
    return (torch.from_numpy(a.indptr.astype(np.int32)).cuda(), torch.from_numpy(a.indices.astype(np.int32)).cuda(),
            torch.from_numpy(a.data).to(dtype).cuda())


def _cuda_matrix(a, dtype=torch.float64):
    crow, col, val = _cuda_csr(a, dtype)
    return torch.sparse_csr_tensor(crow, col, val, size=a.shape)


def _rel(a, b):
    return abs(a - b).max() / abs(b).max()


def _bitwise(x, y):
    bits = torch.int64 if x.dtype == torch.float64 else torch.int32
    return x.dtype == y.dtype and x.shape == y.shape and torch.equal(x.contiguous().view(bits), y.contiguous().view(bits))


def problem(nx, ny, seed=1234):
    mesh = meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=seed, topology=False)
    k, keep, load = ao.p1_poisson(mesh)
    return k, keep, load, ro.mass(mesh)


def hierarchy_tensors(h):
    out = [h.coarse_inv, h.keep]
    for lev in h.levels:
        out += [lev.a_crow, lev.a_col, lev.a_val, lev.p_crow, lev.p_col, lev.p_val, lev.r_crow, lev.r_col, lev.r_val, lev.wdinv, lev.agg,
                lev.x, lev.rc, lev.ec]
    return out


# ---------------------------------------------------------------------------------------------- tfem_csr_spgemm_numeric
def _random_csr(rows, cols, density, rng, empty_rows):
    m = sp.random(rows, cols, density=density, format="lil", random_state=rng, data_rvs=lambda n: rng.standard_normal(n))
    for r in empty_rows:
        m[r, :] = 0
    m = m.tocsr()
    m.eliminate_zeros()
    return m


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_numeric_spgemm_bitwise_on_random_products(dtype):
    """Rectangular products with empty rows in A and B, rows of C up to a few hundred entries (several passes)."""
    rng = np.random.default_rng(7)
    for rows, inner, cols, density in ((300, 200, 150, 0.03), (64, 500, 400, 0.4), (3, 7, 3, 0.9), (50, 40, 1, 0.2)):
        a = _random_csr(rows, inner, density, rng, empty_rows=[0, rows // 2])
        b = _random_csr(inner, cols, density, rng, empty_rows=[1, inner - 1])
        a_t, b_t = _cuda_csr(a, dtype), _cuda_csr(b, dtype)
        c_crow, c_col, c_val = ops.csr_spgemm(a_t, inner, b_t, cols)
        got, missing = ops.csr_spgemm_numeric(a_t, b_t, c_crow, c_col)
        assert int(missing.item()) == 0
        assert _bitwise(got, c_val), (rows, inner, cols)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_numeric_spgemm_bitwise_on_every_product_of_the_amg_build(dtype):
    """P = S T, A P and R (A P) of every level of a 512 x 512 build; the smoother kernel and the R gather as well."""
    k, keep, _, _ = problem(512, 512)
    h = sparse.amg(_cuda_matrix(k, dtype), torch.from_numpy(keep).cuda(), refreshable=True)
    assert len(h.levels) >= 3
    for level, (lev, lp) in enumerate(zip(h.levels, h.pattern.levels)):
        a = (lev.a_crow, lev.a_col, lev.a_val)
        diag = ops.amg_diag(*a)
        assert _bitwise(diag, ops.amg_strength(*a, 0.08)[0])
        wdinv, s_val = torch.empty_like(lev.wdinv), torch.empty_like(lev.a_val)
        ops.amg_smoother(*a, diag, lev.omega, wdinv, s_val)
        row = torch.repeat_interleave(torch.arange(lev.n, device="cuda"), (lev.a_crow[1:] - lev.a_crow[:-1]).long())
        assert _bitwise(wdinv, lev.wdinv) and _bitwise(wdinv, lev.omega / diag)
        assert _bitwise(s_val, (row == lev.a_col.long()).to(dtype) - wdinv[row] * lev.a_val)
        s = (lev.a_crow, lev.a_col, s_val)
        t = (lp.t_crow, lp.t_col, lp.t_val)
        p = (lev.p_crow, lev.p_col, lev.p_val)
        r = (lev.r_crow, lev.r_col, lev.r_val)
        ap = (lp.ap_crow, lp.ap_col, lp.ap_val)
        nxt = h.levels[level + 1] if level + 1 < len(h.levels) else None
        c = (nxt.a_crow, nxt.a_col, nxt.a_val) if nxt is not None else (h.pattern.coarse_crow, h.pattern.coarse_col, h.pattern.coarse_val)
        for left, right, out, n_cols in ((s, t, p, lev.n_coarse), (a, p, ap, lev.n_coarse), (r, ap, c, lev.n_coarse)):
            ref = ops.csr_spgemm(left, left[0].shape[0] - 1, right, n_cols)
            assert torch.equal(ref[0], out[0]) and torch.equal(ref[1], out[1])
            got, missing = ops.csr_spgemm_numeric(left, right, out[0], out[1])
            assert int(missing.item()) == 0 and _bitwise(got, ref[2]) and _bitwise(got, out[2]), level
        assert _bitwise(ops.gather_fill(lp.r_map, lev.p_val, 0.0, torch.empty_like(lev.r_val)), lev.r_val)


def test_numeric_spgemm_counts_products_outside_the_pattern():
    rng = np.random.default_rng(3)
    a, b = _random_csr(80, 60, 0.1, rng, [5]), _random_csr(60, 70, 0.1, rng, [9])
    a_t, b_t = _cuda_csr(a), _cuda_csr(b)
    c_crow, c_col, c_val = ops.csr_spgemm(a_t, 60, b_t, 70)
    lengths = (c_crow[1:] - c_crow[:-1]).cpu()
    row = int(torch.nonzero(lengths >= 2)[0])
    drop = int(c_crow[row]) + 1  # the second entry of that row leaves the pattern
    keep = torch.ones(c_col.shape[0], dtype=torch.bool, device="cuda")
    keep[drop] = False
    crow2 = c_crow.clone()
    crow2[row + 1:] -= 1
    got, missing = ops.csr_spgemm_numeric(a_t, b_t, crow2, c_col[keep].contiguous())
    dropped_products = int(((a[row] != 0).astype(np.int64) @ (b[:, int(c_col[drop])] != 0).astype(np.int64)).toarray().sum())
    assert dropped_products > 0 and int(missing.item()) == dropped_products
    assert _bitwise(got, c_val[keep])  # every other entry is untouched by the drop


# ---------------------------------------------------------------------------------------------- the refresh
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_refreshable_setup_builds_the_same_hierarchy(dtype):
    """amg(A) and amg(A, refreshable=True) give the same hierarchy bit for bit on the device (512 x 512)."""
    k, keep, _, _ = problem(512, 512)
    a, keep_t = _cuda_matrix(k, dtype), torch.from_numpy(keep).cuda()
    plain, kept = sparse.amg(a, keep_t), sparse.amg(a, keep_t, refreshable=True)
    assert plain.pattern is None and kept.pattern is not None
    assert len(plain.levels) == len(kept.levels) >= 3
    for t1, t2 in zip(hierarchy_tensors(plain), hierarchy_tensors(kept)):
        assert _bitwise(t1, t2) if t1.is_floating_point() else (t1.dtype == t2.dtype and torch.equal(t1, t2))
    assert plain.rho == kept.rho and plain.omega == kept.omega and plain.coarse_nnz == kept.coarse_nnz


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("masked", [True, False])
def test_refresh_with_twice_the_matrix_is_a_fresh_build(dtype, masked):
    """amg(A).refresh(2 A) == amg(2 A) bit for bit: scaling by 2 is exact and the strength test, the power iteration and
    omega are scale-invariant, so both aggregate alike; this pins the rounding and order of the whole refresh."""
    k, keep, _, m = problem(256, 256)
    keep_t = torch.from_numpy(keep).cuda() if masked else None
    k = k if masked else (k + m).tocsr()  # without the Dirichlet mask K alone is singular
    a = _cuda_matrix(k, dtype)
    a2 = _cuda_matrix(2.0 * k, dtype)
    h = sparse.amg(a, keep_t, refreshable=True).refresh(a2)
    fresh = sparse.amg(a2, keep_t)
    assert len(h.levels) == len(fresh.levels) >= 2
    assert torch.equal(h.keep, fresh.keep)
    for l1, l2 in zip(h.levels, fresh.levels):
        for name in ("a_crow", "a_col", "p_crow", "p_col", "r_crow", "r_col", "agg"):
            assert torch.equal(getattr(l1, name), getattr(l2, name)), name
        for name in ("a_val", "p_val", "r_val", "wdinv"):
            assert _bitwise(getattr(l1, name), getattr(l2, name)), name
        assert l1.rho == l2.rho and l1.omega == l2.omega
    assert _bitwise(h.coarse_inv, fresh.coarse_inv)


def test_identity_refresh_changes_nothing():
    k, keep, _, _ = problem(300, 200)
    a = _cuda_matrix(k)
    h = sparse.amg(a, torch.from_numpy(keep).cuda(), refreshable=True)
    struct = h.struct
    tensors = hierarchy_tensors(h)[:1] + [t for lev in h.levels for t in (lev.a_val, lev.p_val, lev.r_val, lev.wdinv)]
    before = [t.clone() for t in tensors]
    pointers = [t.data_ptr() for t in hierarchy_tensors(h) + h.pattern.tensors()]
    rho, omega = h.rho, h.omega
    h.refresh(a)
    h.refresh(a.values())
    assert all(_bitwise(t, b) for t, b in zip(tensors, before))
    assert [t.data_ptr() for t in hierarchy_tensors(h) + h.pattern.tensors()] == pointers and h.struct is struct
    assert h.rho == rho and h.omega == omega


@pytest.mark.parametrize("case", ["mass", "rejittered"])
def test_refresh_matches_oracle(case):
    """512 x 512: P, R, A_c of the refresh against the refresh oracle to 1e-13 and rho to 1e-12, for K0 + 1e4 M0 and for
    a re-jittered mesh of the same topology."""
    k0, keep, _, m0 = problem(512, 512)
    if case == "mass":
        a = (k0 + 1e4 * m0).tocsr()
    else:
        a = problem(512, 512, seed=99)[0]
        assert np.array_equal(a.indptr, k0.indptr) and np.array_equal(a.indices, k0.indices)
    h = sparse.amg(_cuda_matrix(k0), torch.from_numpy(keep).cuda(), refreshable=True)
    levels = [{"agg": lev.agg.cpu().numpy(), "n_agg": lev.n_coarse} for lev in h.levels]
    h.refresh(_cuda_matrix(a))
    ref, ref_inv = ro.refresh(levels, a, keep)
    for level, (ours, lev) in enumerate(zip(h.levels, ref)):
        assert abs(ours.rho - lev["rho"]) <= 1e-12 * lev["rho"]
        assert _rel(_scipy(ours.p_crow, ours.p_col, ours.p_val, ours.n_coarse), lev["P"]) <= 1e-13
        assert _rel(_scipy(ours.r_crow, ours.r_col, ours.r_val, ours.n), lev["R"]) <= 1e-13
        nxt = h.levels[level + 1] if level + 1 < len(h.levels) else None
        if nxt is not None:
            assert _rel(_scipy(nxt.a_crow, nxt.a_col, nxt.a_val, nxt.n), lev["Ac"]) <= 1e-13
    assert np.abs(h.coarse_inv.cpu().numpy() - ref_inv).max() <= 1e-10 * np.abs(ref_inv).max()


def _basis(nx, ny, seed=1234):
    previous = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.device("cuda"):
            mesh = tfem.MeshTri(meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=seed, topology=False))
            basis = tfem.Basis(mesh, tfem.ElementTri(1, 3))
    finally:
        torch.set_default_dtype(previous)
    return mesh, basis


def test_config2_solve_after_refresh():
    """Config 2: a hierarchy of the seed-1234 stiffness refreshed for a re-jittered mesh of the same topology converges
    within 5 iterations of a fresh build and meets the O(h^2) nodal bound."""
    _, basis0 = _basis(2048, 1024)
    k0 = basis0.integrate_bilinear_form(forms.Stiffness(), layout="csr")
    h = sparse.amg(k0, basis0.inner_dofs_mask(), refreshable=True)
    del basis0
    mesh, basis = _basis(2048, 1024, seed=99)
    k1, load = basis.assemble(forms.Stiffness(), forms.Load(forms.SinSinSource()), layout="csr")
    assert torch.equal(k1.crow_indices(), k0.crow_indices()) and torch.equal(k1.col_indices(), k0.col_indices())
    del k0
    counts = {}
    for name, pre in (("fresh", sparse.amg(k1, basis.inner_dofs_mask())), ("refreshed", h.refresh(k1))):
        solution = basis.solve(k1, basis.solution_tensor(), load.reshape(-1, 1), rtol=1e-9, preconditioner=pre)
        info = basis.last_solve_info
        assert info.converged, (name, info)
        counts[name] = info.iterations
        points = mesh["vertices", "coordinates"].reshape(-1, 2)
        exact = torch.sin(math.pi * points[:, 0]) * torch.sin(math.pi * points[:, 1])
        assert float((solution.reshape(-1) - exact).abs().max()) < 3.0 / 1024**2, name
    assert counts["refreshed"] <= counts["fresh"] + 5, counts


def test_rvpinn_loss_after_refresh():
    """r^T G^-1 r and G^-1 r with their gradients against the dense formulas, after refreshing the hierarchy of
    G = K + M for G = K + 25 M (another beta)."""
    _, basis = _basis(48, 48)
    keep = basis.inner_dofs_mask()
    h = sparse.amg(basis.integrate_bilinear_form(forms.StiffnessMass(), layout="csr"), keep, max_coarse=200, refreshable=True)
    assert len(h.levels) >= 2
    gram = basis.integrate_bilinear_form(forms.StiffnessMass(1.0, 25.0), layout="csr")
    h.refresh(gram)
    idx = torch.nonzero(keep, as_tuple=True)[0]
    dense = gram.to_dense()[idx][:, idx]
    n = gram.shape[0]
    rng = np.random.default_rng(11)
    theta = torch.tensor(rng.standard_normal(n), device="cuda", requires_grad=True)
    r = torch.sin(theta) + 0.3 * theta
    loss = sparse.inverse_quadratic_form(gram, r.reshape(-1, 1), keep, rtol=1e-13, preconditioner=h)
    (g,) = torch.autograd.grad(loss, theta, retain_graph=True)
    theta_ref = theta.detach().clone().requires_grad_(True)
    r_ref = (torch.sin(theta_ref) + 0.3 * theta_ref)[idx]
    loss_ref = r_ref @ torch.linalg.solve(dense, r_ref)
    (g_ref,) = torch.autograd.grad(loss_ref, theta_ref)
    assert abs(float(loss) - float(loss_ref)) <= 1e-10 * abs(float(loss_ref))
    assert float((g - g_ref).abs().max()) <= 1e-9 * float(g_ref.abs().max())
    x = sparse.solve(gram, r.reshape(-1, 1), keep, rtol=1e-13, preconditioner=h)
    w = torch.tensor(rng.standard_normal(n), device="cuda")
    (g2,) = torch.autograd.grad((x.reshape(-1) * w).sum(), theta)
    theta_ref2 = theta.detach().clone().requires_grad_(True)
    x_ref = torch.zeros(n, dtype=torch.float64, device="cuda")
    x_ref[idx] = torch.linalg.solve(dense, (torch.sin(theta_ref2) + 0.3 * theta_ref2)[idx])
    (g2_ref,) = torch.autograd.grad((x_ref * w).sum(), theta_ref2)
    assert float((g2 - g2_ref).abs().max()) <= 1e-9 * float(g2_ref.abs().max())
