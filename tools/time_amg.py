#!/usr/bin/env python
"""Config-2 solve (2048 x 1024 jittered mesh, 2 100 225 unknowns) with both preconditioners in one process: Jacobi CG
and smoothed-aggregation AMG CG (set-up time, iterations, solve time, time per iteration), the hierarchy, the peak
SpGEMM workspace of the set-up, and the card's name and power limit.

    python tools/time_amg.py [out.json] [nx ny]

Times are CUDA events around work that ends in a device synchronise (best of `REPEATS`)."""
import json
import math
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import pytorch_fem_solver_b200 as tfem  # noqa: E402
from pytorch_fem_solver_b200 import forms, ops, sparse  # noqa: E402

REPEATS = 3


def card():
    query = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True)
    return query.stdout.strip().splitlines()[0] if query.returncode == 0 else torch.cuda.get_device_name()


def timed(fn):
    best, out = float("inf"), None
    for _ in range(REPEATS):
        torch.cuda.synchronize()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        out = fn()
        stop.record()
        torch.cuda.synchronize()
        best = min(best, start.elapsed_time(stop))
    return best, out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    nx, ny = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (2048, 1024)
    torch.set_default_dtype(torch.float64)
    with torch.device("cuda"):
        mesh = tfem.MeshTri(tfem.meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False))
        basis = tfem.Basis(mesh, tfem.ElementTri(1, 3))
    stiffness, load = basis.assemble(forms.Stiffness(), forms.Load(forms.SinSinSource()), layout="csr")
    keep = basis.inner_dofs_mask()
    args = (stiffness.crow_indices().to(torch.int32), stiffness.col_indices().to(torch.int32), stiffness.values(), load.reshape(-1), keep)

    peak = {"spgemm_workspace_bytes": 0}
    workspace = ops._workspace

    def tracked(name, *sizes):
        need = workspace(name, *sizes)
        if name == "tfem_csr_spgemm_workspace":
            peak["spgemm_workspace_bytes"] = max(peak["spgemm_workspace_bytes"], need)
        return need

    ops._workspace = tracked
    sparse.amg(stiffness, keep)  # warm-up: module loading, allocator
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    setup_ms, h = timed(lambda: sparse.amg(stiffness, keep))
    ops._workspace = workspace
    setup_peak = torch.cuda.max_memory_allocated() - base

    points = mesh["vertices", "coordinates"].reshape(-1, 2)
    exact = torch.sin(math.pi * points[:, 0]) * torch.sin(math.pi * points[:, 1])
    record = {"card": card(), "mesh": [nx, ny], "unknowns": stiffness.shape[0], "nnz": stiffness.values().numel(), "rtol": 1e-9,
              "amg_setup_ms": setup_ms, "amg_setup_peak_allocated_bytes": setup_peak, **peak,
              "hierarchy": {"grid_sizes": h.grid_sizes, "operator_complexity": h.operator_complexity, "rho": h.rho, "omega": h.omega}}
    for name, pre in (("jacobi", None), ("amg", h)):
        ms, (x, info) = timed(lambda: sparse.cg(*args, rtol=1e-9, preconditioner=pre))
        record[name] = {"iterations": info.iterations, "relative_residual": info.relative_residual, "converged": info.converged,
                        "solve_ms": ms, "ms_per_iteration": ms / max(info.iterations, 1),
                        "max_nodal_error": float((x - exact).abs().max())}
    record["speedup_solve"] = record["jacobi"]["solve_ms"] / record["amg"]["solve_ms"]
    record["speedup_setup_plus_solve"] = record["jacobi"]["solve_ms"] / (record["amg"]["solve_ms"] + setup_ms)
    text = json.dumps(record, indent=1)
    print(text)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
