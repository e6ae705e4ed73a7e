#!/usr/bin/env python
"""Numeric-only refresh of the config-2 AMG hierarchy (2048 x 1024 jittered mesh, 2 100 225 unknowns) in one process:
the set-up of `amg()` with and without `refreshable=True`, the refresh (best of `REPEATS`, split into the numeric
SpGEMMs, the power iterations and the dense coarsest inverse), the extra resident bytes of a refreshable hierarchy, and
the iterations and solve time to rtol 1e-9 with a fresh, a refreshed and a stale hierarchy for two new matrices on the
same pattern: the stiffness of a re-jittered mesh of the same topology (seed 99) and K + 1e4 M.  Also the card's name,
power limit and clocks.

    python tools/time_amg_refresh.py [out.json] [nx ny]

Times are CUDA events around work that ends in a device synchronise (best of `REPEATS`)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import pytorch_fem_solver_b200 as tfem  # noqa: E402
from pytorch_fem_solver_b200 import forms, ops, sparse  # noqa: E402
from tools.time_amg import card, timed  # noqa: E402

REPEATS = 3


def basis_of(nx, ny, seed):
    with torch.device("cuda"):
        mesh = tfem.MeshTri(tfem.meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=seed, topology=False))
        return tfem.Basis(mesh, tfem.ElementTri(1, 3))


def refresh_split(h):
    """ms of the three parts of a refresh, each timed on its own over the hierarchy's current values."""
    pat = h.pattern
    missing = torch.zeros(1, dtype=torch.int32, device=h.device)

    def spgemms():
        for level, (lev, lp) in enumerate(zip(h.levels, pat.levels)):
            ops.csr_spgemm_numeric((lev.a_crow, lev.a_col, lev.a_val), (lp.t_crow, lp.t_col, lp.t_val), lev.p_crow, lev.p_col,
                                   torch.empty_like(lev.p_val), missing)  # S has A's pattern: same work as S T
            ops.csr_spgemm_numeric((lev.a_crow, lev.a_col, lev.a_val), (lev.p_crow, lev.p_col, lev.p_val), lp.ap_crow, lp.ap_col,
                                   torch.empty_like(lp.ap_val), missing)
            nxt = h.levels[level + 1] if level + 1 < len(h.levels) else None
            c = (nxt.a_crow, nxt.a_col) if nxt is not None else (pat.coarse_crow, pat.coarse_col)
            ops.csr_spgemm_numeric((lev.r_crow, lev.r_col, lev.r_val), (lp.ap_crow, lp.ap_col, lp.ap_val), c[0], c[1], None, missing)

    def power():
        for level, lev in enumerate(h.levels):
            sparse._spectral_radius(lev.a_crow, lev.a_col, lev.a_val, 1.0 / ops.amg_diag(lev.a_crow, lev.a_col, lev.a_val), level)

    def inverse():
        sparse._dense_inverse(pat.coarse_crow, pat.coarse_col, pat.coarse_val)

    return {"numeric_spgemm_ms": timed(spgemms)[0], "power_iteration_ms": timed(power)[0], "coarse_inverse_ms": timed(inverse)[0]}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    nx, ny = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (2048, 1024)
    torch.set_default_dtype(torch.float64)
    basis = basis_of(nx, ny, 1234)
    k0, load = basis.assemble(forms.Stiffness(), forms.Load(forms.SinSinSource()), layout="csr")
    keep = basis.inner_dofs_mask()
    kmass = basis.integrate_bilinear_form(forms.StiffnessMass(1.0, 1e4), layout="csr")
    k1 = basis_of(nx, ny, 99).integrate_bilinear_form(forms.Stiffness(), layout="csr")
    assert torch.equal(k1.crow_indices(), k0.crow_indices()) and torch.equal(k1.col_indices(), k0.col_indices())
    assert torch.equal(kmass.crow_indices(), k0.crow_indices()) and torch.equal(kmass.col_indices(), k0.col_indices())

    sparse.amg(k0, keep, refreshable=True).refresh(k1)  # warm-up: module loading, allocator
    setup_ms, _ = timed(lambda: sparse.amg(k0, keep))
    refreshable_setup_ms, _ = timed(lambda: sparse.amg(k0, keep, refreshable=True))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    plain = sparse.amg(k0, keep)
    plain_bytes = torch.cuda.memory_allocated() - base
    del plain
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    h = sparse.amg(k0, keep, refreshable=True)
    refreshable_bytes = torch.cuda.memory_allocated() - base
    own = {t.data_ptr() for lev in h.levels for t in (lev.a_crow, lev.a_col)} | {k0.crow_indices().data_ptr(), k0.col_indices().data_ptr()}
    pattern_bytes = sum(t.numel() * t.element_size() for t in h.pattern.tensors() if t.data_ptr() not in own)

    refresh_ms, _ = timed(lambda: h.refresh(k1))
    record = {"card": card(), "mesh": [nx, ny], "unknowns": k0.shape[0], "nnz": k0.values().numel(), "rtol": 1e-9,
              "amg_setup_ms": setup_ms, "refreshable_setup_ms": refreshable_setup_ms, "refresh_ms": refresh_ms,
              "refresh_split": refresh_split(h), "setup_over_refresh": setup_ms / refresh_ms,
              "hierarchy_allocated_bytes": plain_bytes, "refreshable_hierarchy_allocated_bytes": refreshable_bytes,
              "extra_resident_bytes": refreshable_bytes - plain_bytes, "pattern_tensor_bytes": pattern_bytes,
              "ap_entries_finest": h.pattern.levels[0].ap_col.numel(), "grid_sizes": h.grid_sizes}

    stale = sparse.amg(k0, keep)
    args_of = lambda a: (a.crow_indices().to(torch.int32), a.col_indices().to(torch.int32), a.values(), load.reshape(-1), keep)  # noqa: E731
    for case, a in (("rejittered", k1), ("stiffness_plus_1e4_mass", kmass)):
        fresh_ms, fresh = timed(lambda: sparse.amg(a, keep))
        h.refresh(a)
        entry = {"fresh_setup_ms": fresh_ms, "rho_fresh": fresh.rho, "rho_refreshed": h.rho}
        for name, pre in (("fresh", fresh), ("refreshed", h), ("stale", stale)):
            ms, (_, info) = timed(lambda: sparse.cg(*args_of(a), rtol=1e-9, preconditioner=pre))
            entry[name] = {"iterations": info.iterations, "relative_residual": info.relative_residual, "converged": info.converged,
                           "solve_ms": ms}
        record[case] = entry
        del fresh
    text = json.dumps(record, indent=1)
    print(text)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
