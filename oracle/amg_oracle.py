"""numpy / scipy restatement of the smoothed-aggregation AMG preconditioner (`sparse.amg`, DESIGN.md §8(f).1).

Test infrastructure only: the package never imports it.  Every step is the one the CUDA set-up runs
(csrc/amg.cu, csrc/symbolic.cu `tfem_csr_spgemm`, sparse.amg), with the same integer hash, so the
aggregation -- integer and deterministic -- is reproduced exactly, and the floating-point parts agree to
rounding:

1. operator (M A M) + (I - M), M = diag(keep): masked rows / columns dropped, their diagonals set to 1;
2. strength: (i, j), i != j, is strong when |a_ij| >= theta sqrt(|a_ii a_jj|);
3. aggregation: parallel MIS(2) on the strength graph with keys (state, hash, i), then every node joins the
   root of the largest key among its strong neighbours, or (distance 2) the aggregate of the assigned
   neighbour of the largest key; nodes without strong connections stay unaggregated (-1);
4. tentative prolongator T[i, agg(i)] = 1 / sqrt(|agg|);
5. rho(D^-1 A) by 15 power iterations from a hash-generated start vector;
6. P = (I - omega D^-1 A) T, omega = 4 / (3 rho);
7. R = P^T, A_c = R A P;
8. recursion until <= max_coarse rows; the coarsest operator is inverted densely.
"""

from __future__ import annotations

import numpy as np
import scipy.sparse as sp

M32 = np.uint64(0xFFFFFFFF)
STATE_OUT, STATE_UNDECIDED, STATE_IN = 0, 1, 2
POWER_ITERATIONS = 15
POWER_SALT = 0x10000  # hash salt of the power-iteration start vector (+ level); the MIS keys use the level itself


def hash32(i, salt: int) -> np.ndarray:
    """32-bit integer hash of (i, salt): the murmur3 finaliser of i * 0x9E3779B1 + salt * 0x85EBCA77 + 0x165667B1."""
    h = (np.asarray(i, dtype=np.uint64) * np.uint64(0x9E3779B1) + np.uint64(salt) * np.uint64(0x85EBCA77) + np.uint64(0x165667B1)) & M32
    h ^= h >> np.uint64(16)
    h = (h * np.uint64(0x85EBCA6B)) & M32
    h ^= h >> np.uint64(13)
    h = (h * np.uint64(0xC2B2AE35)) & M32
    h ^= h >> np.uint64(16)
    return h


def mis_key(state: np.ndarray, level: int) -> np.ndarray:
    """key = state << 61 | (hash32(i, level) >> 3) << 32 | i: tuple order (state, hash, i) in one unsigned 64-bit word."""
    i = np.arange(state.shape[0], dtype=np.uint64)
    return (state.astype(np.uint64) << np.uint64(61)) | ((hash32(i, level) >> np.uint64(3)) << np.uint64(32)) | i


def masked_operator(a: sp.csr_matrix, keep=None) -> sp.csr_matrix:
    """(M A M) + (I - M) with the masked off-diagonal entries dropped (stored order kept)."""
    a = sp.csr_matrix(a)
    n = a.shape[0]
    if keep is None:
        return a.copy()
    keep = np.asarray(keep).reshape(-1) != 0
    rows = np.repeat(np.arange(n), np.diff(a.indptr))
    cols = a.indices
    diag = rows == cols
    live = (keep[rows] & keep[cols]) | diag
    vals = np.where(diag & ~keep[rows], 1.0, a.data).astype(a.data.dtype)
    counts = np.bincount(rows[live], minlength=n)
    indptr = np.concatenate([[0], np.cumsum(counts)])
    return sp.csr_matrix((vals[live], cols[live], indptr), shape=a.shape)


def strength(a: sp.csr_matrix, theta: float) -> np.ndarray:
    """Per stored entry: True when strong."""
    n = a.shape[0]
    rows = np.repeat(np.arange(n), np.diff(a.indptr))
    d = a.diagonal()
    return (rows != a.indices) & (np.abs(a.data) >= theta * np.sqrt(np.abs(d[rows] * d[a.indices])))


def _strong_edges(a, strong):
    rows = np.repeat(np.arange(a.shape[0]), np.diff(a.indptr))
    return rows[strong], a.indices[strong].astype(np.int64)


def mis2(a: sp.csr_matrix, strong: np.ndarray, level: int):
    """Final MIS(2) keys and the number of rounds.  Each round: two sweeps t <- max(t, max over strong neighbours),
    each reading the previous buffer; an undecided node whose own key is the maximum becomes IN, one whose maximum
    is an IN node becomes OUT."""
    n = a.shape[0]
    sr, sc = _strong_edges(a, strong)
    has = np.bincount(sr, minlength=n) > 0
    key = mis_key(np.where(has, STATE_UNDECIDED, STATE_OUT), level)
    rounds = 0
    while True:
        state = key >> np.uint64(61)
        if not np.any(state == STATE_UNDECIDED):
            return key, rounds
        t = key
        for _ in range(2):
            nxt = t.copy()
            np.maximum.at(nxt, sr, t[sc])
            t = nxt
        und = state == STATE_UNDECIDED
        become_in = und & (t == key)
        become_out = und & ~become_in & ((t >> np.uint64(61)) == STATE_IN)
        low = key & ((np.uint64(1) << np.uint64(61)) - np.uint64(1))
        key = np.where(become_in, low | (np.uint64(STATE_IN) << np.uint64(61)), np.where(become_out, low, key))
        rounds += 1


def _best_neighbour(n, sr, sc, key, candidate):
    """Per row: index of the candidate strong neighbour with the largest key, or -1."""
    e = candidate[sc]
    best = np.full(n, -1, dtype=np.int64)
    np.maximum.at(best, sr[e], key[sc[e]].astype(np.int64))  # keys < 2^63
    return np.where(best >= 0, best & 0xFFFFFFFF, -1)


def aggregate(a: sp.csr_matrix, strong: np.ndarray, level: int):
    """(agg [n] int32, n_agg): aggregate of every node, -1 for nodes without a strong connection."""
    n = a.shape[0]
    key, _ = mis2(a, strong, level)
    sr, sc = _strong_edges(a, strong)
    has = np.bincount(sr, minlength=n) > 0
    root = (key >> np.uint64(61)) == STATE_IN
    ids = np.cumsum(root) - root
    agg1 = np.full(n, -2, dtype=np.int64)
    agg1[~has] = -1
    agg1[root] = ids[root]
    best = _best_neighbour(n, sr, sc, key, root)
    first = (agg1 == -2) & (best >= 0)
    agg1[first] = ids[best[first]]
    best2 = _best_neighbour(n, sr, sc, key, agg1 >= 0)
    agg = agg1.copy()
    pending = agg1 == -2
    agg[pending] = np.where(best2[pending] >= 0, agg1[np.maximum(best2[pending], 0)], -1)
    return agg.astype(np.int32), int(root.sum())


def tentative(agg: np.ndarray, n_agg: int, dtype=np.float64) -> sp.csr_matrix:
    n = agg.shape[0]
    live = agg >= 0
    size = np.bincount(agg[live], minlength=n_agg)
    indptr = np.concatenate([[0], np.cumsum(live)])
    return sp.csr_matrix(((1.0 / np.sqrt(size[agg[live]])).astype(dtype), agg[live], indptr), shape=(n, n_agg))


def start_vector(n: int, level: int) -> np.ndarray:
    return hash32(np.arange(n), POWER_SALT + level).astype(np.float64) / 4294967296.0 - 0.5


def spectral_radius(a: sp.csr_matrix, level: int) -> float:
    """rho(D^-1 A): 15 power iterations, rho = |D^-1 A v| / |v| of the last one."""
    dinv = 1.0 / a.diagonal()
    v = start_vector(a.shape[0], level)
    rho = 0.0
    for _ in range(POWER_ITERATIONS):
        w = dinv * (a @ v)
        nw = np.linalg.norm(w)
        rho = nw / np.linalg.norm(v)
        v = w / nw
    return float(rho)


def build_level(a: sp.csr_matrix, level: int, theta: float):
    """One level of the hierarchy from its operator: dict with agg, n_agg, T, rho, omega, P, R, Ac, wdinv."""
    a = sp.csr_matrix(a)
    agg, n_agg = aggregate(a, strength(a, theta), level)
    t = tentative(agg, n_agg, a.dtype)
    rho = spectral_radius(a, level)
    omega = 4.0 / (3.0 * rho)
    d = a.diagonal()
    s = sp.identity(a.shape[0], format="csr") - sp.diags(omega / d) @ a
    p = (s @ t).tocsr()
    r = p.T.tocsr()
    ac = (r @ (a @ p)).tocsr()
    for m in (p, r, ac):
        m.sort_indices()
    return {"A": a, "agg": agg, "n_agg": n_agg, "T": t, "rho": rho, "omega": omega, "P": p, "R": r, "Ac": ac, "wdinv": omega / d}


def hierarchy(a: sp.csr_matrix, keep=None, theta: float = 0.08, max_coarse: int = 1000, max_levels: int = 12):
    """(levels, coarse_inv): the smoothed levels, finest first, and the dense inverse of the coarsest operator."""
    op = masked_operator(a, keep)
    levels = []
    while op.shape[0] > max_coarse and len(levels) + 1 < max_levels:
        lev = build_level(op, len(levels), theta)
        if lev["n_agg"] == 0 or lev["n_agg"] >= op.shape[0]:
            break
        levels.append(lev)
        op = lev["Ac"]
    return levels, np.linalg.inv(op.toarray())


def vcycle(levels, coarse_inv, b: np.ndarray) -> np.ndarray:
    """z = M_AMG b: x = omega D^-1 b; b_c = R (b - A x); x += P (cycle on b_c); x += omega D^-1 (b - A x)."""

    def cycle(l, rhs):
        if l == len(levels):
            return coarse_inv @ rhs
        lev = levels[l]
        x = lev["wdinv"] * rhs
        e = cycle(l + 1, lev["R"] @ (rhs - lev["A"] @ x))
        x = x + lev["P"] @ e
        return x + lev["wdinv"] * (rhs - lev["A"] @ x)

    return cycle(0, np.asarray(b, dtype=np.float64))


def pcg(a: sp.csr_matrix, b: np.ndarray, keep=None, precondition=None, rtol: float = 1e-10, max_iterations: int = 10000):
    """Preconditioned CG on (M A M) x = M b; returns (x, iterations), checking |r| / |b| after every iteration."""
    n = a.shape[0]
    m = np.ones(n) if keep is None else (np.asarray(keep).reshape(-1) != 0).astype(np.float64)
    op = lambda v: m * (a @ (m * v))  # noqa: E731
    if precondition is None:
        d = a.diagonal()
        precondition = lambda r: r / np.where(d != 0, d, 1.0)  # noqa: E731
    b = m * np.asarray(b, dtype=np.float64).reshape(-1)
    x = np.zeros(n)
    r = b.copy()
    z = precondition(r)
    p = z.copy()
    rz = r @ z
    nb = np.linalg.norm(b)
    for it in range(1, max_iterations + 1):
        ap = op(p)
        alpha = rz / (p @ ap)
        x += alpha * p
        r -= alpha * ap
        if np.linalg.norm(r) / nb <= rtol:
            return x, it
        z = precondition(r)
        rz_new = r @ z
        p = z + (rz_new / rz) * p
        rz = rz_new
    return x, max_iterations


def p1_poisson(mesh: dict):
    """P1 stiffness (CSR, scipy), boundary keep mask and sin sin load of a mesh dict (host-side test problems)."""
    from oracle import fem_oracle as fo

    coords, conn = mesh["vertices"], mesh["triangles"].astype(np.int64)
    n = coords.shape[0]
    geo = fo.tri_geometry(coords, conn, 3)
    crow, col, vals = fo.scatter_bilinear_csr(fo.quad_reduce(fo.form_stiffness(geo), geo["dx"]), conn, n)
    load = fo.scatter_linear(fo.quad_reduce(fo.form_load(geo, fo.source_sinsin(geo["integration_points"])), geo["dx"]), conn, n)
    if "vertex_markers" in mesh:
        keep = np.asarray(mesh["vertex_markers"]).reshape(-1) == 0
    else:
        x = coords
        keep = ~((np.abs(x[:, 0]) < 1e-12) | (np.abs(x[:, 0] - 1) < 1e-12) | (np.abs(x[:, 1]) < 1e-12) | (np.abs(x[:, 1] - 1) < 1e-12))
    return sp.csr_matrix((vals, col, crow), shape=(n, n)), keep, load.reshape(-1)
