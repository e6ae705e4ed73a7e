"""End-to-end Poisson solve at BASELINE config-2 size on one B200.

    python examples/poisson_config2.py [nx ny]

-Laplace u = 2 pi^2 sin(pi x) sin(pi y) on the unit square, u = 0 on the boundary, P1 elements on the
jittered nx x ny mesh (default 2048 x 1024: 4 194 304 triangles, 2 100 225 unknowns):
fused assembly of the stiffness matrix + load vector to CSR (one kernel launch), then
Jacobi-preconditioned conjugate gradients on the CSR arrays (`tfem_cg_iteration`), then the same
solve preconditioned by smoothed-aggregation AMG (`sparse.amg`, `tfem_pcg_iteration`).  The
reference's `Basis.solve` densifies the matrix (35 TB at this size); this is the same call on the
CSR result.
"""

import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import pytorch_fem_solver_b200 as tfem  # noqa: E402
from pytorch_fem_solver_b200 import forms  # noqa: E402


def main():
    nx = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
    ny = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
    torch.set_default_dtype(torch.float64)
    t0 = time.perf_counter()
    mesh_dict = tfem.meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False)
    with torch.device("cuda"):
        mesh = tfem.MeshTri(mesh_dict)
        basis = tfem.Basis(mesh, tfem.ElementTri(1, 3))
    basis.tile_plan()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    basis.assemble(forms.Stiffness(), forms.Load(forms.SinSinSource()), layout="csr")  # first call loads the kernel
    start.record()
    stiffness, load = basis.assemble(forms.Stiffness(), forms.Load(forms.SinSinSource()), layout="csr")
    stop.record()
    torch.cuda.synchronize()
    assemble_ms = start.elapsed_time(stop)
    t2 = time.perf_counter()
    solution = basis.solve(stiffness, basis.solution_tensor(), load.reshape(-1, 1), rtol=1e-9)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    info = basis.last_solve_info
    points = mesh["vertices", "coordinates"].reshape(-1, 2)
    exact = torch.sin(math.pi * points[:, 0]) * torch.sin(math.pi * points[:, 1])
    error = float((solution.reshape(-1) - exact).abs().max())
    print(f"mesh {nx} x {ny}: {2 * nx * ny} triangles, {stiffness.shape[0]} unknowns, nnz {stiffness.values().numel()}")
    print(f"set-up (mesh, topology, CSR pattern, tile plan): {t1 - t0:.2f} s")
    print(f"assembly K + load to CSR: {assemble_ms:.3f} ms (device)")
    print(f"CG: {info.iterations} iterations, relative residual {info.relative_residual:.2e}, {t3 - t2:.3f} s "
          f"({1e6 * (t3 - t2) / max(info.iterations, 1):.1f} us per iteration)")
    print(f"max nodal error vs sin(pi x) sin(pi y): {error:.3e}  (h^2 = {(1.0 / min(nx, ny)) ** 2:.3e})")
    assert error < 3.0 / min(nx, ny) ** 2

    t4 = time.perf_counter()
    hierarchy = tfem.sparse.amg(stiffness, basis.inner_dofs_mask())  # one-time set-up, reusable for every solve with K
    torch.cuda.synchronize()
    t5 = time.perf_counter()
    solution_amg = basis.solve(stiffness, basis.solution_tensor(), load.reshape(-1, 1), rtol=1e-9, preconditioner=hierarchy)
    torch.cuda.synchronize()
    t6 = time.perf_counter()
    info_amg = basis.last_solve_info
    error_amg = float((solution_amg.reshape(-1) - exact).abs().max())
    print(f"AMG set-up: {t5 - t4:.3f} s  ({hierarchy.summary()})")
    print(f"AMG-preconditioned CG: {info_amg.iterations} iterations, relative residual {info_amg.relative_residual:.2e}, "
          f"{t6 - t5:.3f} s ({1e6 * (t6 - t5) / max(info_amg.iterations, 1):.1f} us per iteration)")
    print(f"max nodal error (AMG solve): {error_amg:.3e}")
    assert error_amg < 3.0 / min(nx, ny) ** 2


if __name__ == "__main__":
    main()
