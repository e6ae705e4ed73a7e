#!/usr/bin/env python
"""Stiffness and mass forms with coefficient fields at config 2 (2048 x 1024 jittered mesh, 4 194 304 elements,
`ElementTri(1, 3)` = 4 points, fp64) in one process:

1. the weighted local-forms kernel alone (per-point kappa and c fields, SinSin load), with its algorithmic bytes over
   time against the HBM bandwidth measured here by a device-to-device copy;
2. `assemble(StiffnessMass(kappa, c), Load(SinSin), layout="values")` against the generic route (callable integrand
   -> quad_reduce -> scatter): time and `torch.cuda.max_memory_allocated` above the resident set-up;
3. constant `StiffnessMass` on the two-pass and tiled paths, as reference points;
4. -div(kappa grad u) = f with kappa = 1e4 on an 8 x 8 checkerboard, one value per element: AMG set-up, iterations and solve time against
   Jacobi to rtol 1e-9, then a contrast change to 1e2 with a re-assembly, a refresh and a solve.

    python tools/time_coefficient_forms.py [out.json] [nx ny]

Kernel and assembly times are CUDA events around one call, the L2 flushed (256 MiB write) before each, median of
`REPEATS`; solves and set-ups are best of three.  The card's name, power limit and clocks are read in the same run."""
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import pytorch_fem_solver_b200 as tfem  # noqa: E402
from pytorch_fem_solver_b200 import forms, ops, sparse  # noqa: E402
from tools.time_amg import card, timed  # noqa: E402

REPEATS = 20


def checkerboard(contrast, blocks=8):
    def kappa(points):
        cell = torch.floor(points.clamp(0.0, 1.0 - 1e-12) * blocks)
        dark = (cell[..., 0:1] + cell[..., 1:2]) % 2 == 0
        return torch.where(dark, torch.full_like(cell[..., 0:1], contrast), torch.ones_like(cell[..., 0:1]))

    return kappa


def flushed(fn, repeats=REPEATS):
    """Median ms of `fn` over `repeats` calls, each after an L2 flush that lies outside its event pair."""
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    fn()
    times = []
    for i in range(repeats):
        flush.fill_(float(i))
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        fn()
        stop.record()
        torch.cuda.synchronize()
        times.append(start.elapsed_time(stop))
    return statistics.median(times)


def hbm_copy_bandwidth():
    """Bytes/s of a 4 GiB device-to-device copy (read + write), best of REPEATS."""
    src = torch.empty(1 << 29, dtype=torch.float64, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    ms, _ = timed(lambda: dst.copy_(src))
    return 2 * src.numel() * 8 / (ms * 1e-3)


def peak_extra(fn, resident):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - resident
    del out
    return peak


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    nx, ny = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (2048, 1024)
    torch.set_default_dtype(torch.float64)
    with torch.device("cuda"):
        mesh = tfem.MeshTri(tfem.meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False))
        basis = tfem.Basis(mesh, tfem.ElementTri(1, 3))
    lay, pat = basis._layout, basis.pattern
    n_el, n_q = lay.n_total, basis.n_q
    result = {"card": card(), "workload": {"nx": nx, "ny": ny, "elements": n_el, "dofs": pat.n_dof, "nnz": pat.nnz, "n_q": n_q,
                                           "dtype": "float64"}}

    # 1. the kernel alone
    kappa = forms.StiffnessMass(lambda p: 1.0 + p[..., 0:1] * p[..., 1:2], lambda p: 2.0 + p[..., 0:1])
    alpha_q, beta_q = basis._coefficient_samples(kappa.alpha), basis._coefficient_samples(kappa.beta)
    src = forms.SinSinSource()

    def kernel():
        return ops.weighted_local_forms(lay.coords, lay.conn, lay.n_el_per_mesh, lay.n_vert_per_mesh, 3, 0.0, 0.0, alpha_q, beta_q,
                                        src.kind, list(src.params))

    kernel_ms = flushed(kernel)
    # coordinates (each vertex once), connectivity, two coefficient streams, local matrices and load vectors
    bytes_alg = lay.coords.numel() * 8 + n_el * 3 * 4 + 2 * n_el * n_q * 8 + n_el * (9 + 3) * 8
    hbm = hbm_copy_bandwidth()
    result["kernel"] = {"ms": round(kernel_ms, 4), "algorithmic_bytes": bytes_alg,
                        "achieved_GBps": round(bytes_alg / (kernel_ms * 1e-3) / 1e9, 1),
                        "measured_hbm_copy_GBps": round(hbm / 1e9, 1),
                        "share_of_measured_hbm": round(bytes_alg / (kernel_ms * 1e-3) / hbm, 3)}

    # 2. fused against the generic route (same callables, samples cached for the fused form as in a loop)
    form = forms.StiffnessMass(checkerboard(1e4), lambda p: 1.0 + p[..., 0:1])
    load = forms.Load(forms.SinSinSource())
    basis.assemble(form, load, layout="values")
    generic = lambda: (basis.integrate_bilinear_form(lambda b: form(b), layout="values"), basis.integrate_linear_form(load))  # noqa: E731
    fused = lambda: basis.assemble(form, load, layout="values")  # noqa: E731
    generic()
    torch.cuda.synchronize()
    resident = torch.cuda.memory_allocated()
    result["assembly"] = {
        "fused_ms": round(flushed(fused), 3),
        "generic_ms": round(flushed(generic, 5), 3),
        "fused_peak_extra_MB": round(peak_extra(fused, resident) / 1e6, 1),
        "generic_peak_extra_MB": round(peak_extra(generic, resident) / 1e6, 1),
        "fused_first_call_ms_with_sampling": round(timed(lambda: (form.refresh(), fused()))[0], 3),
    }
    a_f, _ = fused()
    a_g, _ = generic()
    result["assembly"]["max_rel_difference"] = float((a_f - a_g).abs().max() / a_g.abs().max())

    # 3. constant coefficients on both existing paths
    const = forms.StiffnessMass(1.0, 1.0)
    result["constant"] = {path + "_ms": round(flushed(lambda: basis.assemble(const, load, layout="values", path=path)), 3)
                          for path in ("two_pass", "tiled")}
    del a_f, a_g

    # 4. high-contrast solve, AMG against Jacobi, then a contrast change and a refresh
    keep = basis.inner_dofs_mask()
    # one kappa per element (its centroid's square): a discontinuous kappa sampled per point meets the negative centroid
    # weight of the 4-point rule and can make element matrices indefinite
    centroids = basis.integration_points.mean(dim=-3, keepdim=True)
    a0, rhs = basis.assemble(forms.Stiffness(checkerboard(1e4)(centroids)), load, layout="csr")
    setup_ms, h = timed(lambda: sparse.amg(a0, keep, refreshable=True))

    def solve(matrix, pre, cap=None):
        """Iterations, convergence and best-of-3 ms of Basis.solve to rtol 1e-9; non-convergence is recorded, not raised."""
        def run():
            try:
                basis.solve(matrix, basis.solution_tensor(), rhs, rtol=1e-9, max_iterations=cap, preconditioner=pre)
            except RuntimeError:
                pass
        ms, _ = timed(run)
        info = basis.last_solve_info
        return {"iterations": info.iterations, "converged": bool(info.converged), "relative_residual": float(info.relative_residual),
                "solve_ms": round(ms, 1)}

    result["high_contrast_solve"] = out = {"rtol": 1e-9, "amg_setup_ms": round(setup_ms, 1), "amg": solve(a0, h),
                                           "jacobi": solve(a0, None, 200000)}
    assemble_ms, (a1, _) = timed(lambda: basis.assemble(forms.Stiffness(checkerboard(1e2)(centroids)), None, layout="csr"))
    refresh_ms, _ = timed(lambda: h.refresh(a1.values()))
    out["after_contrast_change_1e2"] = {"assemble_ms": round(assemble_ms, 2), "refresh_ms": round(refresh_ms, 1), "refreshed": solve(a1, h),
                                        "fresh_build": solve(a1, sparse.amg(a1, keep)), "jacobi": solve(a1, None, 200000)}

    text = json.dumps(result, indent=1)
    print(text)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
