"""numpy / scipy restatement of the numeric-only refresh of an AMG hierarchy (`sparse.AmgHierarchy.refresh`): the
aggregates of an `oracle.amg_oracle.hierarchy` are kept and every value is recomputed for a new matrix -- the steps of
`amg_oracle.build_level` after the aggregation.  Test infrastructure only."""

from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from oracle import amg_oracle as ao


def rebuild_level(a: sp.csr_matrix, level: int, agg: np.ndarray, n_agg: int):
    """`ao.build_level` with the aggregates given instead of computed."""
    a = sp.csr_matrix(a)
    t = ao.tentative(agg, n_agg, a.dtype)
    rho = ao.spectral_radius(a, level)
    omega = 4.0 / (3.0 * rho)
    d = a.diagonal()
    s = sp.identity(a.shape[0], format="csr") - sp.diags(omega / d) @ a
    p = (s @ t).tocsr()
    r = p.T.tocsr()
    ac = (r @ (a @ p)).tocsr()
    for m in (p, r, ac):
        m.sort_indices()
    return {"A": a, "agg": agg, "n_agg": n_agg, "T": t, "rho": rho, "omega": omega, "P": p, "R": r, "Ac": ac, "wdinv": omega / d}


def refresh(levels, a: sp.csr_matrix, keep=None):
    """(levels, coarse_inv) of the hierarchy `levels` refreshed for the matrix `a`: aggregates kept, values recomputed."""
    op = ao.masked_operator(a, keep)
    out = []
    for level, lev in enumerate(levels):
        out.append(rebuild_level(op, level, lev["agg"], lev["n_agg"]))
        op = out[-1]["Ac"]
    return out, np.linalg.inv(op.toarray())


def mass(mesh: dict) -> sp.csr_matrix:
    """P1 mass matrix of a mesh dict, on the pattern of `ao.p1_poisson`'s stiffness."""
    from oracle import fem_oracle as fo

    coords, conn = mesh["vertices"], mesh["triangles"].astype(np.int64)
    n = coords.shape[0]
    geo = fo.tri_geometry(coords, conn, 3)
    crow, col, vals = fo.scatter_bilinear_csr(fo.quad_reduce(fo.form_mass(geo), geo["dx"]), conn, n)
    return sp.csr_matrix((vals, col, crow), shape=(n, n))
