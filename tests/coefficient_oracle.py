"""numpy restatement of the weighted local forms of `forms.StiffnessMass(alpha, beta)` with coefficient fields, built on
the unchanged FEM oracle (oracle/fem_oracle.py), and a high-contrast test problem for the AMG oracle."""

from __future__ import annotations

import numpy as np
import scipy.sparse as sp

from oracle import fem_oracle as fo


def form_weighted_stiffness_mass(geo, alpha_q, beta_q):
    """alpha_q grad(v) grad(v)^T + beta_q v v^T; alpha_q, beta_q broadcastable to (..., N, q, 1, 1)."""
    return alpha_q * fo.form_stiffness(geo) + beta_q * fo.form_mass(geo)


def checkerboard_kappa(centroids: np.ndarray, blocks: int = 8, contrast: float = 1e4) -> np.ndarray:
    """kappa = contrast on the dark squares of a blocks x blocks checkerboard of the unit square, 1 elsewhere."""
    cell = np.floor(np.clip(centroids, 0.0, 1.0 - 1e-12) * blocks).astype(np.int64)
    return np.where((cell[..., 0] + cell[..., 1]) % 2 == 0, contrast, 1.0)


def high_contrast_poisson(mesh: dict, contrast: float = 1e4, blocks: int = 8, order: int = 3):
    """P1 operator of -div(kappa grad u) with a per-element checkerboard kappa (CSR, scipy), boundary keep mask and the
    sin sin load, like amg_oracle.p1_poisson."""
    coords, conn = mesh["vertices"], mesh["triangles"].astype(np.int64)
    n = coords.shape[0]
    geo = fo.tri_geometry(coords, conn, order)
    kappa = checkerboard_kappa(coords[conn].mean(axis=1), blocks, contrast)[:, None, None, None]
    local = fo.quad_reduce(form_weighted_stiffness_mass(geo, kappa, 0.0), geo["dx"])
    crow, col, vals = fo.scatter_bilinear_csr(local, conn, n)
    load = fo.scatter_linear(fo.quad_reduce(fo.form_load(geo, fo.source_sinsin(geo["integration_points"])), geo["dx"]), conn, n)
    x = coords
    keep = ~((np.abs(x[:, 0]) < 1e-12) | (np.abs(x[:, 0] - 1) < 1e-12) | (np.abs(x[:, 1]) < 1e-12) | (np.abs(x[:, 1] - 1) < 1e-12))
    return sp.csr_matrix((vals, col, crow), shape=(n, n)), keep, load.reshape(-1)
