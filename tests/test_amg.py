"""Smoothed-aggregation AMG preconditioner (sparse.amg, DESIGN.md §8(f).1) without a GPU: the oracle's invariants and
iteration counts, and the host logic of `sparse.amg` / `sparse.cg(..., preconditioner=)` with the new ops replaced by
oracle-backed stand-ins (installed here; tests/cpu_shim.py covers the older ops).  The kernels themselves are checked
against the same oracle in tests/test_amg_gpu.py."""

import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import amg_oracle as ao
from pytorch_fem_solver_b200 import _lib, meshgen, ops, sparse
from tests import cpu_shim
from tests.conftest import load_golden


# ---------------------------------------------------------------------------------------------- stand-ins for the new ops
def _csr(crow, col, val, n_cols):
    return sp.csr_matrix((val.numpy(), col.numpy().astype(np.int64), crow.numpy().astype(np.int64)), shape=(crow.shape[0] - 1, n_cols))


def _torch_csr(m, dtype):
    m = sp.csr_matrix(m)
    m.sort_indices()
    return (torch.from_numpy(m.indptr.astype(np.int32)), torch.from_numpy(m.indices.astype(np.int32)),
            torch.from_numpy(m.data.astype(np.float64)).to(dtype))


def _amg_strength(crow, col, val, theta):
    a = _csr(crow, col, val, crow.shape[0] - 1)
    return torch.from_numpy(a.diagonal()).to(val.dtype), torch.from_numpy(ao.strength(a, theta).astype(np.uint8))


def _amg_aggregate(crow, col, strong, level):
    a = _csr(crow, col, torch.ones(col.shape[0], dtype=torch.float64), crow.shape[0] - 1)
    agg, n_agg = ao.aggregate(a, strong.numpy() != 0, level)
    return torch.from_numpy(agg), n_agg


def _csr_spgemm(a, n_cols_a, b, n_cols_b):
    return _torch_csr(_csr(*a, n_cols_a) @ _csr(*b, n_cols_b), a[2].dtype)


def _amg_diag(crow, col, val):
    return torch.from_numpy(_csr(crow, col, val, crow.shape[0] - 1).diagonal()).to(val.dtype)


def _amg_smoother(crow, col, val, diag, omega, wdinv, s_val):
    row = torch.repeat_interleave(torch.arange(crow.shape[0] - 1), (crow[1:] - crow[:-1]).long())
    wdinv.copy_(omega / diag)
    s_val.copy_((row == col.long()).to(val.dtype) - wdinv[row] * val)


def _gather_fill(src, values, fill, out):
    out.copy_(torch.where(src >= 0, values[src.long().clamp_min(0)], torch.full_like(out, fill)))
    return out


def _levels_of(h):
    levels = []
    for lev in h.levels:
        levels.append({"A": _csr(lev.a_crow, lev.a_col, lev.a_val, lev.n), "P": _csr(lev.p_crow, lev.p_col, lev.p_val, lev.n_coarse),
                       "R": _csr(lev.r_crow, lev.r_col, lev.r_val, lev.n), "wdinv": lev.wdinv.numpy()})
    return levels


def _amg_vcycle(h, r):
    return torch.from_numpy(ao.vcycle(_levels_of(h), h.coarse_inv.numpy(), r.numpy())).to(r.dtype)


def install(monkeypatch):
    cpu_shim.install(monkeypatch)
    for name, fn in (("amg_strength", _amg_strength), ("amg_aggregate", _amg_aggregate), ("csr_spgemm", _csr_spgemm),
                     ("amg_smoother", _amg_smoother), ("gather_fill", _gather_fill), ("amg_vcycle", _amg_vcycle)):
        monkeypatch.setattr(ops, name, fn)


# ---------------------------------------------------------------------------------------------- problems
def jittered(nx, ny, seed=1234):
    return ao.p1_poisson(meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=seed, topology=False))


def delaunay():
    g = load_golden("delaunay60")
    return ao.p1_poisson({"vertices": g["in_vertices"], "triangles": g["in_triangles"], "vertex_markers": g["in_vertex_markers"]})


def as_matrix(a):
    crow, col, val = _torch_csr(a, torch.float64)
    return torch.sparse_csr_tensor(crow, col, val, size=a.shape)


# ---------------------------------------------------------------------------------------------- oracle invariants
@pytest.mark.parametrize("problem", ["jittered64", "delaunay"])
def test_aggregation_invariants(problem):
    a, keep, _ = jittered(64, 64) if problem == "jittered64" else delaunay()
    op = ao.masked_operator(a, keep)
    strong = ao.strength(op, 0.08)
    agg, n_agg = ao.aggregate(op, strong, 0)
    key, rounds = ao.mis2(op, strong, 0)
    assert rounds >= 1 and n_agg >= 1
    n = op.shape[0]
    rows = np.repeat(np.arange(n), np.diff(op.indptr))
    s = sp.csr_matrix((np.ones(int(strong.sum())), (rows[strong], op.indices[strong])), shape=(n, n))
    has = np.asarray(s.sum(axis=1)).reshape(-1) > 0
    assert np.all(agg[has] >= 0)  # every node with a strong connection is aggregated
    assert np.all(agg[~has] == -1)
    assert np.all(agg[~keep] == -1)  # Dirichlet identity rows stay with the smoother
    within2 = ((s + s @ s + sp.identity(n)) != 0).tocsr()
    roots = np.nonzero((key >> np.uint64(61)) == ao.STATE_IN)[0]
    assert roots.shape[0] == n_agg
    root_of = np.empty(n_agg, dtype=np.int64)
    root_of[agg[roots]] = roots
    assert np.array_equal(agg[roots], np.arange(n_agg))  # roots are ranked in index order
    live = np.nonzero(agg >= 0)[0]
    assert np.all(np.asarray(within2[live, root_of[agg[live]]]).reshape(-1))  # within distance 2 of the aggregate's root
    between = within2[roots][:, roots].toarray()
    assert np.array_equal(between, np.eye(roots.shape[0], dtype=bool))  # roots pairwise more than distance 2 apart


def test_operator_properties():
    a, keep, _ = jittered(64, 64)
    lev = ao.build_level(ao.masked_operator(a, keep), 0, 0.08)
    t = lev["T"]
    assert abs(t.T @ t - sp.identity(lev["n_agg"])).max() < 1e-14  # orthonormal columns
    p, ac = lev["P"], lev["Ac"]
    ref = (p.T @ lev["A"] @ p).toarray()
    assert np.abs(ac.toarray() - ref).max() <= 1e-13 * np.abs(ref).max()
    assert abs(ac - ac.T).max() <= 1e-13 * abs(ac).max()
    assert abs(lev["R"] - p.T).max() == 0.0
    assert 1.0 < lev["rho"] < 2.5 and abs(lev["omega"] - 4.0 / (3.0 * lev["rho"])) < 1e-15


def test_vcycle_is_symmetric_positive_definite():
    a, keep, _ = jittered(32, 32)
    levels, coarse_inv = ao.hierarchy(a, keep, max_coarse=50)
    assert len(levels) >= 2
    n = a.shape[0]
    m = np.stack([ao.vcycle(levels, coarse_inv, e) for e in np.eye(n)], axis=1)
    rng = np.random.default_rng(0)
    v, w = rng.standard_normal(n), rng.standard_normal(n)
    assert abs(w @ ao.vcycle(levels, coarse_inv, v) - v @ ao.vcycle(levels, coarse_inv, w)) <= 1e-12 * np.linalg.norm(v) * np.linalg.norm(w)
    assert np.abs(m - m.T).max() <= 1e-12 * np.abs(m).max()
    assert np.linalg.eigvalsh(0.5 * (m + m.T)).min() > 0.0


@pytest.mark.parametrize("nx, bound", [(64, 30), (256, 34)])
def test_oracle_iteration_counts(nx, bound):
    """The prototype's 25 (64 x 64) and 29 (256 x 256) iterations at rtol 1e-10, against Jacobi's hundreds."""
    a, keep, b = jittered(nx, nx)
    levels, coarse_inv = ao.hierarchy(a, keep)
    x, iterations = ao.pcg(a, b, keep, lambda r: ao.vcycle(levels, coarse_inv, r), rtol=1e-10)
    assert iterations <= bound
    x_jacobi, jacobi = ao.pcg(a, b, keep, rtol=1e-10)
    assert jacobi > 8 * iterations
    assert np.abs(x - x_jacobi).max() <= 1e-8 * np.abs(x_jacobi).max()


# ---------------------------------------------------------------------------------------------- host logic through the stand-ins
def test_amg_setup_host_logic_matches_oracle(monkeypatch):
    install(monkeypatch)
    a, keep, _ = jittered(48, 40)
    h = sparse.amg(as_matrix(a), torch.from_numpy(keep), max_coarse=100)
    levels, coarse_inv = ao.hierarchy(a, keep, max_coarse=100)
    assert h.grid_sizes == [lev["A"].shape[0] for lev in levels] + [coarse_inv.shape[0]]
    for ours, ref in zip(h.levels, levels):
        assert np.array_equal(ours.agg.numpy(), ref["agg"])
        for name in ("P", "R", "A"):
            got = _csr(getattr(ours, name.lower() + "_crow"), getattr(ours, name.lower() + "_col"), getattr(ours, name.lower() + "_val"),
                       ref[name].shape[1])
            assert abs(got - ref[name]).max() <= 1e-13 * abs(ref[name]).max()
        assert abs(ours.rho - ref["rho"]) <= 1e-12 * ref["rho"]
    assert np.abs(h.coarse_inv.numpy() - coarse_inv).max() <= 1e-10 * np.abs(coarse_inv).max()
    assert 1.0 < h.operator_complexity < 2.0
    assert "levels" in h.summary()


def test_preconditioned_cg_host_logic(monkeypatch):
    install(monkeypatch)
    a, keep, b = jittered(40, 36)
    matrix, keep_t, b_t = as_matrix(a), torch.from_numpy(keep), torch.from_numpy(b)
    h = sparse.amg(matrix, keep_t, max_coarse=100)
    args = (matrix.crow_indices(), matrix.col_indices(), matrix.values())
    x, info = sparse.cg(*args, b_t, keep_t, rtol=1e-10, preconditioner=h)
    assert info.converged and info.iterations <= 30
    inner = np.nonzero(keep)[0]
    ref = np.zeros(a.shape[0])
    ref[inner] = sp.linalg.spsolve(a[inner][:, inner].tocsc(), b[inner])
    assert np.abs(x.numpy() - ref).max() <= 1e-8 * np.abs(ref).max()
    assert float(x[~keep_t].abs().max()) == 0.0  # the keep mask
    _, again = sparse.cg(*args, b_t, keep_t, x0=x, rtol=1e-8, preconditioner=h)
    assert again.converged and again.iterations == 0  # a converged x0
    _, short = sparse.cg(*args, b_t, keep_t, rtol=1e-12, max_iterations=3, preconditioner=h)
    assert short.iterations == 3 and not short.converged
    # breakdown: a negative definite system gives p.Ap < 0 -> inf / NaN; the solve stops and reports
    neg = as_matrix(-a)
    h_neg = sparse.amg(neg, keep_t, max_coarse=100)
    _, broken = sparse.cg(neg.crow_indices(), neg.col_indices(), neg.values(), b_t, keep_t, rtol=1e-10, preconditioner=h_neg)
    assert not broken.converged and broken.iterations <= 2 * a.shape[0] + 100


def test_solve_and_quadratic_form_host_logic(monkeypatch):
    install(monkeypatch)
    a, keep, b = jittered(24, 20)
    m = (a + sp.identity(a.shape[0])).tocsr()  # stiffness plus a mass-like term
    matrix, keep_t = as_matrix(m), torch.from_numpy(keep.astype(np.uint8))
    h = sparse.amg(matrix, keep_t, max_coarse=60)
    inner = np.nonzero(keep)[0]
    dense = m.toarray()[np.ix_(inner, inner)]
    r = torch.tensor(b, requires_grad=True)
    loss = sparse.inverse_quadratic_form(matrix, r, keep_t, rtol=1e-12, preconditioner=h)
    (g,) = torch.autograd.grad(loss, r)
    sol = np.linalg.solve(dense, b[inner])
    assert abs(float(loss) - b[inner] @ sol) <= 1e-10 * abs(b[inner] @ sol)
    assert np.abs(g.numpy()[inner] - 2 * sol).max() <= 1e-9 * np.abs(sol).max()
    w = np.random.default_rng(4).standard_normal(a.shape[0])
    x = sparse.solve(matrix, r, keep_t, rtol=1e-12, preconditioner=h)
    (g2,) = torch.autograd.grad((x * torch.from_numpy(w)).sum(), r)
    assert np.abs(g2.numpy()[inner] - np.linalg.solve(dense, w[inner])).max() <= 1e-9 * np.abs(np.linalg.solve(dense, w[inner])).max()


def test_mismatched_hierarchy_raises(monkeypatch):
    install(monkeypatch)
    a, keep, b = jittered(24, 20)
    matrix, keep_t, b_t = as_matrix(a), torch.from_numpy(keep), torch.from_numpy(b)
    h = sparse.amg(matrix, keep_t, max_coarse=60)
    args = (matrix.crow_indices(), matrix.col_indices(), matrix.values())
    other_keep = keep_t.clone()
    other_keep[np.nonzero(keep)[0][0]] = False
    with pytest.raises(ValueError, match="keep mask"):
        sparse.cg(*args, b_t, other_keep, preconditioner=h)
    with pytest.raises(ValueError, match="keep mask"):
        sparse.cg(*args, b_t, None, preconditioner=h)
    with pytest.raises(ValueError, match="built for"):
        sparse.cg(args[0], args[1], args[2].float(), b_t, keep_t, preconditioner=h)
    small, small_keep, small_b = jittered(20, 20)
    with pytest.raises(ValueError, match="built for"):
        sparse.solve(as_matrix(small), torch.from_numpy(small_b), torch.from_numpy(small_keep), preconditioner=h)


def test_argument_validation_of_the_amg_entry_points():
    """Bad arguments of the AMG entry points come back as status codes from the host side (no launch, no GPU)."""
    lib = _lib.load()
    need = ctypes.c_int64(-1)
    fake = ctypes.addressof(ctypes.create_string_buffer(256))  # never dereferenced: the checks below fail first
    assert lib.tfem_amg_strength_f64(-1, None, None, None, 0.08, None, None, None) == -1
    assert lib.tfem_amg_strength_f64(0, None, None, None, 0.08, None, None, None) == 0
    assert lib.tfem_amg_strength_f32(5, None, None, None, 0.08, None, None, None) == -1
    assert lib.tfem_amg_strength_f64(5, fake, fake, fake, -0.5, fake, fake, None) == -1  # theta < 0
    assert lib.tfem_amg_mis2_round(-1, None, None, None, 0, 1, None, None, None, None) == -1
    assert lib.tfem_amg_mis2_round(5, None, None, None, 0, 1, None, None, None, None) == -1
    assert lib.tfem_amg_mis2_round(0, None, None, None, 0, 1, None, None, None, None) == 0
    assert lib.tfem_amg_aggregate_workspace(-1, ctypes.byref(need)) == -1
    assert lib.tfem_amg_aggregate_workspace(10, None) == -1
    assert lib.tfem_amg_aggregate_workspace(2**31, ctypes.byref(need)) == -4
    assert lib.tfem_amg_aggregate(0, None, None, None, None, None, 0, None, None, None) == -1
    assert lib.tfem_amg_aggregate(5, fake, fake, fake, fake, None, 0, fake, fake, None) == -1  # no workspace
    assert lib.tfem_csr_spgemm_workspace(-1, 10, ctypes.byref(need)) == -1
    assert lib.tfem_csr_spgemm_workspace(10, 2**31, ctypes.byref(need)) == -4
    args = [fake, fake, fake, 0, None, None, None, 5, 5, 12, fake, 0, fake, fake, fake, fake, None]
    assert lib.tfem_csr_spgemm_f64(-1, *args) == -1
    assert lib.tfem_csr_spgemm_f64(5, fake, fake, fake, 0, None, None, None, 5, 5, 12, None, 0, fake, fake, fake, fake, None) == -1
    assert lib.tfem_csr_spgemm_f64(5, fake, fake, fake, 2, *args[4:]) == -1  # transpose is 0 or 1
    assert lib.tfem_csr_spgemm_f32(5, fake, fake, fake, 0, fake, None, None, *args[7:]) == -1  # B without columns / values
    assert lib.tfem_csr_spgemm_f64(5, fake, fake, fake, 0, None, None, None, 5, 0, 12, fake, 0, fake, fake, fake, fake, None) == -1
    level = _lib.AmgLevel()
    assert lib.tfem_amg_vcycle_f64(None, 1, fake, 10, fake, fake, None) == -1  # levels missing
    assert lib.tfem_amg_vcycle_f64(None, 0, None, 10, fake, fake, None) == -1  # coarse inverse missing
    assert lib.tfem_amg_vcycle_f64(None, 0, fake, 40000, fake, fake, None) == -4  # too large for the dense coarse solve
    assert lib.tfem_amg_vcycle_f32(ctypes.byref(level), 1, fake, 10, fake, fake, None) == -1  # empty level
    level.n, level.n_coarse = 100, 20
    for name in ("a_crow", "a_col", "a_val", "p_crow", "p_col", "p_val", "r_crow", "r_col", "r_val", "wdinv", "x", "rc", "ec"):
        setattr(level, name, fake)
    assert lib.tfem_amg_vcycle_f64(ctypes.byref(level), 1, fake, 10, fake, fake, None) == -1  # n_coarse does not chain
    assert lib.tfem_amg_vcycle_f64(ctypes.byref(level), 1, fake, 20, None, fake, None) == -1  # r missing
    pcg = [fake] * 3 + [None, ctypes.byref(level), 1, fake, 20] + [fake] * 6 + [4, fake, None]
    assert lib.tfem_pcg_iteration_f64(99, *pcg) == -1  # the hierarchy of another system
    assert lib.tfem_pcg_iteration_f64(-1, *pcg) == -1
    assert lib.tfem_pcg_iteration_f32(0, *pcg) == 0
