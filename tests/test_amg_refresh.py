"""Numeric-only refresh of an AMG hierarchy (`sparse.amg(..., refreshable=True)`, `AmgHierarchy.refresh`) without a
GPU: the refresh oracle (tests/amg_refresh_oracle.py) and what a refresh buys in iterations, and the host logic of
`refresh` with the new ops replaced by oracle-backed stand-ins.  The kernels are checked in tests/test_amg_refresh_gpu.py."""

import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import amg_oracle as ao
from pytorch_fem_solver_b200 import _lib, meshgen, ops, sparse
from tests import amg_refresh_oracle as ro
from tests.test_amg import _csr, as_matrix
from tests.test_amg import install as install_amg


# ---------------------------------------------------------------------------------------------- stand-ins for the new ops
def _csr_spgemm_numeric(a, b, c_crow, c_col, out=None, n_missing=None):
    n_cols = int(max(int(b[1].max()) if b[1].numel() else 0, int(c_col.max()) if c_col.numel() else 0)) + 1
    left, right = _csr(*a, b[0].shape[0] - 1), _csr(*b, n_cols)
    rows = np.repeat(np.arange(c_crow.shape[0] - 1), np.diff(c_crow.numpy()))
    cols = c_col.numpy().astype(np.int64)
    values = np.asarray((left @ right)[rows, cols]).reshape(-1)
    ones = lambda m: sp.csr_matrix((np.ones_like(m.data), m.indices, m.indptr), shape=m.shape)  # noqa: E731
    counts = ones(left) @ ones(right)
    missing = int(counts.sum() - np.asarray(counts[rows, cols]).sum())
    out = torch.empty(c_col.shape[0], dtype=a[2].dtype) if out is None else out
    n_missing = torch.zeros(1, dtype=torch.int32) if n_missing is None else n_missing
    out.copy_(torch.from_numpy(values))
    n_missing += missing
    return out, n_missing


def _amg_diag(crow, col, val):
    return torch.from_numpy(_csr(crow, col, val, crow.shape[0] - 1).diagonal()).to(val.dtype)


def _amg_smoother(crow, col, val, diag, omega, wdinv, s_val):
    row = torch.repeat_interleave(torch.arange(crow.shape[0] - 1), (crow[1:] - crow[:-1]).long())
    wdinv.copy_(omega / diag)
    s_val.copy_((row == col.long()).to(val.dtype) - wdinv[row] * val)


def _gather_fill(src, values, fill, out):
    out.copy_(torch.where(src >= 0, values[src.long().clamp_min(0)], torch.full_like(out, fill)))
    return out


def install(monkeypatch):
    install_amg(monkeypatch)
    for name, fn in (("csr_spgemm_numeric", _csr_spgemm_numeric), ("amg_diag", _amg_diag), ("amg_smoother", _amg_smoother),
                     ("gather_fill", _gather_fill)):
        monkeypatch.setattr(ops, name, fn)


# ---------------------------------------------------------------------------------------------- problems
def mesh(nx, ny, seed=1234):
    return meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=seed, topology=False)


def problem(nx, ny, seed=1234):
    """(K, keep, load, M) of the jittered unit square."""
    m = mesh(nx, ny, seed)
    k, keep, load = ao.p1_poisson(m)
    return k, keep, load, ro.mass(m)


def same_pattern(a, b):
    return np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)


def hierarchy_tensors(h):
    out = [h.coarse_inv, h.keep]
    for lev in h.levels:
        out += [lev.a_crow, lev.a_col, lev.a_val, lev.p_crow, lev.p_col, lev.p_val, lev.r_crow, lev.r_col, lev.r_val, lev.wdinv, lev.agg]
    return out


# ---------------------------------------------------------------------------------------------- the oracle
def test_oracle_refresh_with_the_build_matrix_reproduces_the_build():
    a, keep, _, _ = problem(64, 64)
    levels, coarse_inv = ao.hierarchy(a, keep, max_coarse=100)
    again, again_inv = ro.refresh(levels, a, keep)
    assert len(again) == len(levels) >= 2
    for ours, ref in zip(again, levels):
        for name in ("P", "R", "Ac"):
            assert same_pattern(ours[name], ref[name]) and np.array_equal(ours[name].data, ref[name].data)
        assert ours["rho"] == ref["rho"] and ours["omega"] == ref["omega"]
    assert np.array_equal(again_inv, coarse_inv)


def test_refreshed_vcycle_is_symmetric_positive_definite():
    k, keep, _, m = problem(32, 32)
    levels, _ = ao.hierarchy(k, keep, max_coarse=50)
    a = (k + 1e4 * m).tocsr()
    new, coarse_inv = ro.refresh(levels, a, keep)
    n = a.shape[0]
    mat = np.stack([ao.vcycle(new, coarse_inv, e) for e in np.eye(n)], axis=1)
    assert np.abs(mat - mat.T).max() <= 1e-12 * np.abs(mat).max()
    assert np.linalg.eigvalsh(0.5 * (mat + mat.T)).min() > 0.0


@pytest.mark.parametrize("nx", [128, 256])
def test_refresh_converges_like_a_fresh_build(nx):
    """PCG iterations to rtol 1e-10: a refreshed hierarchy within 3 of a fresh build, a stale one at least 1.5x a fresh
    one, for the re-jittered mesh of the same topology and for K0 + 1e4 M0 (at 256 x 256: 28 / 30 / 58 and 20 / 20 / 129)."""
    k0, keep, b, m0 = problem(nx, nx)
    levels0, inv0 = ao.hierarchy(k0, keep)
    k1, _, _, _ = problem(nx, nx, seed=99)
    assert same_pattern(k1, k0)
    for a in (k1, (k0 + 1e4 * m0).tocsr()):
        counts = {}
        fresh = ao.hierarchy(a, keep)
        refreshed = ro.refresh(levels0, a, keep)
        stale = (levels0, inv0)
        for name, (levels, inv) in (("fresh", fresh), ("refreshed", refreshed), ("stale", stale)):
            _, counts[name] = ao.pcg(a, b, keep, lambda r, lv=levels, ci=inv: ao.vcycle(lv, ci, r), rtol=1e-10)
        assert counts["refreshed"] <= counts["fresh"] + 3, counts
        assert counts["stale"] >= 1.5 * counts["fresh"], counts


# ---------------------------------------------------------------------------------------------- host logic through the stand-ins
def _compare_with_oracle(h, ref_levels, ref_inv):
    assert len(h.levels) == len(ref_levels)
    for level, (ours, ref) in enumerate(zip(h.levels, ref_levels)):
        nxt = h.levels[level + 1] if level + 1 < len(h.levels) else None
        for name, got in (("P", _csr(ours.p_crow, ours.p_col, ours.p_val, ours.n_coarse)), ("R", _csr(ours.r_crow, ours.r_col, ours.r_val, ours.n)),
                          ("A", _csr(ours.a_crow, ours.a_col, ours.a_val, ours.n))):
            assert abs(got - ref[name]).max() <= 1e-13 * abs(ref[name]).max(), (level, name)
        if nxt is not None:
            got = _csr(nxt.a_crow, nxt.a_col, nxt.a_val, nxt.n)
            assert abs(got - ref["Ac"]).max() <= 1e-13 * abs(ref["Ac"]).max()
        assert abs(ours.rho - ref["rho"]) <= 1e-12 * ref["rho"]
        assert ours.omega == 4.0 / (3.0 * ours.rho)
        assert np.abs(ours.wdinv.numpy() - ref["wdinv"]).max() <= 1e-13 * np.abs(ref["wdinv"]).max()
    assert np.abs(h.coarse_inv.numpy() - ref_inv).max() <= 1e-10 * np.abs(ref_inv).max()


def test_refresh_host_logic_matches_oracle(monkeypatch):
    install(monkeypatch)
    k, keep, _, m = problem(48, 40)
    h = sparse.amg(as_matrix(k), torch.from_numpy(keep), max_coarse=100, refreshable=True)
    levels, _ = ao.hierarchy(k, keep, max_coarse=100)
    assert len(h.levels) >= 2
    pointers = [t.data_ptr() for t in hierarchy_tensors(h)]
    struct = h.struct
    for a in ((k + 1e2 * m).tocsr(), problem(48, 40, seed=99)[0]):
        assert same_pattern(a, k)
        assert h.refresh(as_matrix(a)) is h
        _compare_with_oracle(h, *ro.refresh(levels, a, keep))
        assert [t.data_ptr() for t in hierarchy_tensors(h)] == pointers and h.struct is struct
        assert [f"{r:.4f}" for r in h.rho] == [f"{lev['rho']:.4f}" for lev in ro.refresh(levels, a, keep)[0]]
        assert f"{h.rho[0]:.4f}" in h.summary()


@pytest.mark.parametrize("masked", [True, False])
def test_refresh_from_values_equals_refresh_from_csr(monkeypatch, masked):
    install(monkeypatch)
    k, keep, _, m = problem(40, 36)
    keep_t = torch.from_numpy(keep) if masked else None
    a = as_matrix((k + 1e3 * m).tocsr())
    h1 = sparse.amg(as_matrix(k), keep_t, max_coarse=100, refreshable=True).refresh(a)
    h2 = sparse.amg(as_matrix(k), keep_t, max_coarse=100, refreshable=True).refresh(a.values().clone())
    for t1, t2 in zip(hierarchy_tensors(h1), hierarchy_tensors(h2)):
        assert torch.equal(t1, t2)
    assert h1.rho == h2.rho and h1.omega == h2.omega
    fresh = sparse.amg(a, keep_t, max_coarse=100)  # the new matrix aggregates alike here: the refresh is a fresh build
    if all(torch.equal(l1.agg, l2.agg) for l1, l2 in zip(h1.levels, fresh.levels)):
        for t1, t2 in zip(hierarchy_tensors(h1), hierarchy_tensors(fresh)):
            assert torch.allclose(t1.double(), t2.double(), rtol=1e-12, atol=0.0)


def test_refresh_errors_leave_the_hierarchy_unchanged(monkeypatch):
    install(monkeypatch)
    k, keep, _, m = problem(24, 20)
    keep_t = torch.from_numpy(keep)
    matrix = as_matrix(k)
    plain = sparse.amg(matrix, keep_t, max_coarse=60)
    with pytest.raises(ValueError, match="refreshable"):
        plain.refresh(matrix)
    h = sparse.amg(matrix, keep_t, max_coarse=60, refreshable=True)
    before = [t.clone() for t in hierarchy_tensors(h)]
    rho = list(h.rho)
    small = as_matrix(problem(20, 20)[0])
    other = k.tolil()
    other[0, k.shape[0] - 1] = other[k.shape[0] - 1, 0] = -1e-3  # one more pair of entries: another nnz
    moved = matrix.col_indices().clone()
    row0 = slice(int(matrix.crow_indices()[0]), int(matrix.crow_indices()[1]))
    moved[row0] = torch.flip(moved[row0], [0])  # same n, nnz and crow, other col
    cases = [
        (small, "built for"),
        (as_matrix(other.tocsr()), "built for"),
        (torch.sparse_csr_tensor(matrix.crow_indices(), matrix.col_indices(), matrix.values().float(), size=matrix.shape), "built for"),
        (torch.sparse_csr_tensor(matrix.crow_indices(), moved, matrix.values(), size=matrix.shape), "pattern"),
        (matrix.values()[:-1].clone(), "value array"),
        (matrix.values().float(), "value array"),
        (matrix.values().reshape(-1, 1), "value array"),
    ]
    for bad, message in cases:
        with pytest.raises(ValueError, match=message):
            h.refresh(bad)
        assert all(torch.equal(t, b) for t, b in zip(hierarchy_tensors(h), before)) and h.rho == rho


@pytest.mark.parametrize("masked", [True, False])
def test_refreshable_false_builds_the_same_hierarchy(monkeypatch, masked):
    install(monkeypatch)
    k, keep, _, _ = problem(40, 36)
    keep_t = torch.from_numpy(keep) if masked else None
    plain = sparse.amg(as_matrix(k), keep_t, max_coarse=100)
    kept = sparse.amg(as_matrix(k), keep_t, max_coarse=100, refreshable=True)
    assert plain.pattern is None and kept.pattern is not None
    for t1, t2 in zip(hierarchy_tensors(plain), hierarchy_tensors(kept)):
        assert t1.dtype == t2.dtype and torch.equal(t1, t2)
    assert plain.rho == kept.rho and plain.omega == kept.omega and plain.coarse_nnz == kept.coarse_nnz
    before = [t.clone() for t in hierarchy_tensors(kept)]
    kept.refresh(as_matrix(k))  # the build's own matrix
    for t1, t2 in zip(hierarchy_tensors(kept), before):
        assert torch.allclose(t1.double(), t2.double(), rtol=1e-13, atol=0.0)


def test_argument_validation_of_the_refresh_entry_points():
    """Bad arguments of the refresh entry points come back as status codes from the host side (no launch, no GPU)."""
    lib = _lib.load()
    fake = ctypes.addressof(ctypes.create_string_buffer(256))  # never dereferenced: the checks below fail first
    spgemm = [fake] * 10 + [None]
    assert lib.tfem_csr_spgemm_numeric_f64(-1, *spgemm) == -1
    assert lib.tfem_csr_spgemm_numeric_f64(0, *([None] * 11)) == 0
    for missing in range(10):
        args = list(spgemm)
        args[missing] = None
        assert lib.tfem_csr_spgemm_numeric_f32(5, *args) == -1, missing
    assert lib.tfem_csr_spgemm_numeric_f64(2**27, *spgemm) == -4  # one warp per row: rows * 32 must fit int32
    assert lib.tfem_amg_diag_f64(-1, None, None, None, None, None) == -1
    assert lib.tfem_amg_diag_f64(0, None, None, None, None, None) == 0
    assert lib.tfem_amg_diag_f32(5, fake, fake, fake, None, None) == -1
    assert lib.tfem_amg_diag_f64(2**31, fake, fake, fake, fake, None) == -4
    assert lib.tfem_amg_smoother_f64(-1, None, None, None, None, 1.0, None, None, None) == -1
    assert lib.tfem_amg_smoother_f64(0, None, None, None, None, 1.0, None, None, None) == 0
    assert lib.tfem_amg_smoother_f64(5, fake, fake, fake, fake, float("nan"), fake, fake, None) == -1
    assert lib.tfem_amg_smoother_f32(5, fake, fake, fake, fake, 0.5, fake, None, None) == -1
    assert lib.tfem_gather_f64(-1, None, None, 0.0, None, None) == -1
    assert lib.tfem_gather_f64(0, None, None, 0.0, None, None) == 0
    assert lib.tfem_gather_f32(5, fake, None, 1.0, fake, None) == -1
    assert lib.tfem_gather_f64(2**31, fake, fake, 1.0, fake, None) == -4
