#!/usr/bin/env python
"""Headline benchmark: P1 stiffness+mass and load assembly to CSR (BASELINE.json config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

One "step" = one full assembly of the synthetic structured mesh (nx=2048, ny=1024 squares ->
4 194 304 triangles per GPU, fp64, 4-point quadrature, bilinear form grad u.grad v + u v and
load f = 2 pi^2 sin(pi x) sin(pi y)) into CSR values + load vector.  Prints ONE JSON line.

* `value`     elements/s, device-timed (CUDA events around every step, L2 flushed in between),
              inputs resident in HBM, max over ranks;
* `e2e`       the same through the public API with HOST buffers: pinned coordinates copied
              host->device, assembly, CSR values + load copied device->host, every step;
* `roofline`  algorithmic bytes (SURVEY.md 8(d): 12 N_e + 16 N_v + 8 nnz + 8 N_v) / kernel time
              against the measured HBM copy bandwidth of MEASURED_PEAKS.json;
* `cpu_baseline`  the reference's own tensor program (oracle/torch_cpu_port.py) on the host cores.

`--impl reference` times that CPU port alone (the reference is pure Python and does not exist on
the GPU box; see DESIGN.md).  Multi-GPU (`torchrun`, one rank per GPU): weak scaling, each rank
assembles its own 4.19 M-element strip of a mesh that is N times taller; interface rows travel
over NVLink peer memory while the interior assembles (DESIGN.md section 6).

`--dump-outputs DIR` writes the CSR values and the load vector of the last timed step to DIR (see
`dump_outputs`), so that two builds can be compared output for output on the same seeded mesh.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

NX, NY = 2048, 1024
QUAD_ORDER = 3
METRIC = "elements assembled/sec to CSR (P1, fp64)"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--nx", type=int, default=NX)
    p.add_argument("--ny", type=int, default=NY)
    p.add_argument("--path", default="tiled", choices=["tiled", "two_pass"])
    p.add_argument("--rows-per-tile", type=int, default=336)
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="multi-GPU runs: weak = one nx x ny strip PER GPU (default), strong = the ONE nx x ny mesh cut into N element ranges")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--permuted", action="store_true",
                   help="locality stress (SURVEY.md 8(d)): random renumbering of vertices and elements, default_rng(7); N=1 only")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the CSR values and load vector of the last timed step as DIR/csr_values.npy and DIR/load.npy; one GPU only")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def measured_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(args):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/roofline_traffic.json); only valid for the configuration that was profiled."""
    path = os.path.join(REPO, "profiles", "roofline_traffic.json")
    if args.path != "tiled" or (args.nx, args.ny) != (NX, NY) or args.permuted or args.rows_per_tile != 336 or not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh).get("traffic_bytes_per_launch")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML; only samples taken while `active`
    (the timed region) are reported."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.active = False
        self.ready = threading.Event()
        self._stop_event = threading.Event()

    def run(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            # NVML enumerates physical GPUs: honour CUDA_VISIBLE_DEVICES when it lists indices
            visible = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in visible.split(",") if v.strip().isdigit()]
            physical = int(ids[self.index]) if self.index < len(ids) else self.index
            handle = pynvml.nvmlDeviceGetHandleByIndex(physical)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            getter = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._stop_event.is_set():
                clock = pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)
                mask = getter(handle)
                self.ready.set()
                if self.active:
                    self.samples.append(clock)
                    for name, bit in names.items():
                        if mask & bit:
                            self.reasons.add(name)
                time.sleep(0.0005)
        except Exception as exc:  # NVML missing: report it, never fail the bench
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")
            self.ready.set()

    def stop(self):
        self._stop_event.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        ordered = sorted(self.samples)
        return {"sm_mhz": ordered[len(ordered) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(ordered)}


DUMP_MAX_BYTES = 64_000_000  # both files together, .npy headers included
# per array: half the budget, less room for its .npy header (128 bytes for a 1-D float64 array)
DUMP_MAX_ELEMENTS = (DUMP_MAX_BYTES // 2 - 4096) // 8


def dump_outputs(directory, values, load):
    """Write the CSR values and the load vector as DIR/csr_values.npy and DIR/load.npy (1-D float64).

    An array longer than DUMP_MAX_ELEMENTS is replaced by its entries at the sorted indices of
    `numpy.random.default_rng(0).choice(length, DUMP_MAX_ELEMENTS, replace=False)`: the same entries on every run
    of the same mesh, so the dumps of two builds (or of `--impl ours` and `--impl reference`, whose CSR patterns
    are the same) compare entry for entry."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, array in (("csr_values", values), ("load", load)):
        flat = array.detach().reshape(-1).cpu().numpy().astype(np.float64, copy=False)
        if flat.size > DUMP_MAX_ELEMENTS:
            flat = flat[np.sort(np.random.default_rng(0).choice(flat.size, DUMP_MAX_ELEMENTS, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), flat)


def cpu_reference_run(nx, ny, repeats=1):
    """Time the CPU port of the reference pipeline; returns (elements/s, description, timings)."""
    import torch

    from oracle.torch_cpu_port import reference_assembly_cpu
    from pytorch_fem_solver_b200 import meshgen

    small = meshgen.structured_rectangle(64, 64, jitter=0.25, topology=False)
    reference_assembly_cpu(torch.from_numpy(small["vertices"]), torch.from_numpy(small["triangles"]), QUAD_ORDER)
    mesh = meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False)
    coords, conn = torch.from_numpy(mesh["vertices"]), torch.from_numpy(mesh["triangles"])
    best, best_t = None, None
    for _ in range(repeats):
        timings = {}
        reference_assembly_cpu(coords, conn, QUAD_ORDER, timings)
        if best is None or timings["total"] < best:
            best, best_t = timings["total"], timings
    n_el = conn.shape[0]
    return n_el / best, f"{n_el} elements (nx={nx}, ny={ny}), best of {repeats}", {k: round(v, 4) for k, v in best_t.items()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    # torchrun exports OMP_NUM_THREADS=1 for every rank; the reference arm runs on rank 0 alone and may
    # use every host core
    torch.set_num_threads(len(os.sched_getaffinity(0)))
    # the full workload of the repo arm: one step = the whole nx x ny mesh (about two seconds on 16 host cores)
    nx, ny = args.nx, args.ny
    from oracle.torch_cpu_port import reference_assembly_cpu
    from pytorch_fem_solver_b200 import meshgen

    mesh = meshgen.structured_rectangle(nx, ny, jitter=0.25, seed=1234, topology=False)
    coords, conn = torch.from_numpy(mesh["vertices"]), torch.from_numpy(mesh["triangles"])
    n_el = conn.shape[0]
    for _ in range(args.warmup):
        reference_assembly_cpu(coords, conn, QUAD_ORDER)
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = reference_assembly_cpu(coords, conn, QUAD_ORDER)
        if i + 1 < args.steps:
            last = None  # only the last step's outputs are kept
    elapsed = time.perf_counter() - t0
    if args.dump_outputs:
        matrix, load = last
        dump_outputs(args.dump_outputs, matrix.values(), load)
    value = n_el * args.steps / elapsed
    cores = torch.get_num_threads()
    sample = f"all {n_el} elements per step (nx={nx}, ny={ny}); {args.warmup} warm-up + {args.steps} timed steps"
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": "elements/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * elapsed / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "elements/s", "cores": cores, "kind": "port", "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": "elements/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    strong = world > 1 and getattr(args, "scaling", "weak") == "strong"
    per_gpu = 2 * args.nx * args.ny // world if strong else 2 * args.nx * args.ny
    return {
        "workload": f"BASELINE config 2: structured unit-square P1 triangle mesh nx={args.nx} ny={args.ny} "
        + (f"cut into {world} element ranges" if strong else "per GPU")
        + f" ({2 * args.nx * args.ny} elements), interior vertices jittered U(-0.25h,0.25h) seed 1234, fp64, "
        "ElementTri(1,3) 4-point quadrature, grad u.grad v + u v to CSR values + load 2pi^2 sin(pi x) sin(pi y)",
        "elements_per_gpu": per_gpu,
        "path": args.path,
        "l2": "flushed between timed steps (256 MiB write)",
        "symbolic": "CSR pattern + tile plan built once, outside the timed region",
        "multi_gpu": ("strong scaling: the one mesh is cut into contiguous element ranges, one per GPU; " if strong else
                      "weak scaling: one strip of the same size per GPU; ")
        + "interface rows are packed straight into the owner's "
        "receive buffer over NVLink peer memory (signal-pad handshake; TFEM_EXCHANGE=nccl selects one all_gather instead) "
        "and added by their owners on a side stream while the interior tiles assemble",
    }


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one GPU: run it with --gpus 1")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    import pytorch_fem_solver_b200 as tfem
    from pytorch_fem_solver_b200 import _lib, forms, ops

    torch.set_default_dtype(torch.float64)
    bilinear, load_form = forms.StiffnessMass(1.0, 1.0), forms.Load(forms.SinSinSource())

    if world == 1:
        mesh_dict = tfem.meshgen.structured_rectangle(args.nx, args.ny, jitter=0.25, seed=1234, topology=False)
        if args.permuted:
            mesh_dict = tfem.meshgen.permute_mesh(mesh_dict, seed=7)
        with torch.device(device):
            basis = tfem.Basis(tfem.MeshTri(mesh_dict), tfem.ElementTri(1, QUAD_ORDER))
        assembler = None
    else:
        from pytorch_fem_solver_b200 import distributed

        if args.scaling == "strong":
            global_mesh = tfem.meshgen.structured_rectangle(args.nx, args.ny, jitter=0.25, seed=1234, topology=False)
            assembler = distributed.PartitionedAssembly.from_mesh(global_mesh, rank, world, device, quad_order=QUAD_ORDER,
                                                                  rows_per_tile=args.rows_per_tile)
            del global_mesh
        else:
            assembler = distributed.StripAssembly(args.nx, args.ny, rank, world, device, QUAD_ORDER, rows_per_tile=args.rows_per_tile)
        basis = assembler.basis
        mesh_dict = assembler.mesh_dict

    # one-time symbolic phase (CSR pattern: sort/unique of the COO keys; tile plan), timed separately
    torch.cuda.synchronize()
    t_symbolic = time.perf_counter()
    pat = basis.pattern
    torch.cuda.synchronize()
    symbolic_pattern_s = time.perf_counter() - t_symbolic
    lay = basis._layout
    n_el, n_v, nnz = lay.n_total, pat.n_dof, pat.nnz
    src = load_form.source
    values = torch.empty(nnz, dtype=torch.float64, device=device)
    load = torch.empty(n_v, dtype=torch.float64, device=device)
    symbolic_plan_s = None
    symbolic_warm = None
    if args.path == "tiled":
        t_symbolic = time.perf_counter()
        plan = basis.tile_plan(args.rows_per_tile)
        torch.cuda.synchronize()
        symbolic_plan_s = time.perf_counter() - t_symbolic
        plan_struct = plan.c_struct()
        if assembler is None:
            # the same symbolic phase once more, warm (the first call also pays CUDA module loading and allocator growth)
            from pytorch_fem_solver_b200 import csr as csr_mod

            torch.cuda.synchronize()
            t_symbolic = time.perf_counter()
            warm_pattern = csr_mod.build_pattern(basis._dof_conn_flat(), pat.n_dof)
            torch.cuda.synchronize()
            symbolic_warm = [time.perf_counter() - t_symbolic]
            t_symbolic = time.perf_counter()
            csr_mod.build_tile_plan(lay.conn, basis._dof_conn_flat(), warm_pattern, lay.coords, args.rows_per_tile, "auto")
            torch.cuda.synchronize()
            symbolic_warm.append(time.perf_counter() - t_symbolic)
            del warm_pattern

        def local_step():
            ops.assemble_csr_tiled(plan_struct, lay.coords, QUAD_ORDER, 1.0, 1.0, src.kind, src.params, values, load)

        kernels_per_step = 1
    else:
        plan = None

        def local_step():
            return basis._assemble_fused(bilinear, src, "two_pass")

        kernels_per_step = 3

    if assembler is not None and args.path == "tiled":
        # interface tiles first, then interior tiles while the NCCL exchange runs on a side stream
        # the whole step (assembly launch + side-stream exchange) replayed from CUDA graphs where it can be captured
        captured = assembler.capture()
        step = assembler.replay if captured else assembler.step
        kernels_per_step = 2 + assembler.fused_exchange.n_kernels
        exchange_kind = type(assembler.fused_exchange).__name__ + (" (step replayed from CUDA graphs)" if captured else "")
    elif assembler is not None:

        def step():
            local_step()
            assembler.exchange(values, load)

    else:
        step = local_step

    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- device-timed steps (value) ------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(timeout=10)
    launches_before = sum(_lib.LAUNCHES.values())
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    barrier()
    sampler.active = True
    for i in range(args.steps):
        flush.fill_(float(i))  # evict L2 (126 MB) between timed steps; outside the event pair
        starts[i].record()
        last = step()
        ends[i].record()
        if i + 1 < args.steps:
            last = None  # only the last step's outputs are kept; earlier ones go back to the allocator as before
    barrier()
    sampler.active = False
    gpu_launches = sum(_lib.LAUNCHES.values()) - launches_before
    times_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = sum(times_ms)
    clocks = sampler.stop()
    # the tiled step writes into `values` / `load`, the two-pass step returns fresh arrays; a device copy is
    # written to disk after every timed phase, so the host work of the dump cannot idle the GPU between them
    dumped = None
    if args.dump_outputs:
        if args.path == "two_pass":
            dumped = [t.clone() for t in last]
        else:
            dumped = [values.clone(), load.clone()]
    del last

    # kernel-only time of the dominant kernel (roofline numerator), same stream, same flush
    k_ms = []
    for i in range(min(args.steps, 20)):
        flush.fill_(float(i))
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        local_step()
        e.record()
        e.synchronize()
        k_ms.append(s.elapsed_time(e))
    kernel_ms = sum(k_ms) / len(k_ms)

    # ---- end-to-end through the public API with host buffers (e2e) ----------------------------
    e2e = None
    if not args.no_e2e:
        coords_host = torch.from_numpy(mesh_dict["vertices"]).pin_memory()
        values_host = torch.empty(nnz, dtype=torch.float64).pin_memory()
        load_host = torch.empty((n_v, 1), dtype=torch.float64).pin_memory()

        if assembler is not None and args.path == "tiled":

            strip_pipeline = distributed.StripHostPipeline(assembler, depth=2)

            def e2e_step():  # host coordinates in, distributed assembly, owned values + load back to the host; 2 steps in flight
                strip_pipeline.step(coords_host, values_host, load_host)

        elif assembler is None and args.path == "tiled":
            # two steps in flight: H2D of step i+1, assembly of step i and D2H of step i-1 on three streams
            pipeline = basis.host_pipeline(bilinear, load_form, depth=2)
            e2e_api = ("Basis.host_pipeline(StiffnessMass, Load, depth=2).step(pinned coords, pinned values, pinned load): "
                       "every step copies its coordinates in and its CSR values + load out; consecutive steps overlap")

            def e2e_step():
                pipeline.step(coords_host, values_host, load_host)

        else:
            if assembler is not None:
                basis._post_assemble_hook = assembler.exchange  # interface rows summed before the device->host copy

            def e2e_step():
                basis.assemble_from_host(coords_host, bilinear, load_form, values_host, load_host, path=args.path)

        for _ in range(3):
            e2e_step()
        barrier()
        e2e_steps = max(min(args.steps, 20), 1)
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e = {"seconds": e2e_s, "steps": e2e_steps, "h2d": coords_host.numel() * 8, "d2h": (values_host.numel() + load_host.numel()) * 8}
        if assembler is None and args.path == "tiled":
            # for reference: the same step done one at a time (copy in, assemble, copy out, wait)
            basis.assemble_from_host(coords_host, bilinear, load_form, values_host, load_host, path=args.path)  # (first use of the registered op)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                basis.assemble_from_host(coords_host, bilinear, load_form, values_host, load_host, path=args.path)
                torch.cuda.synchronize()
            e2e["serial_ms"] = (time.perf_counter() - t0) / 5 * 1e3
            e2e["api"] = e2e_api

    # ---- reduce over ranks -----------------------------------------------------------------------
    stats = torch.tensor([total_ms, kernel_ms, e2e["seconds"] / e2e["steps"] if e2e else 0.0], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    total_ms, kernel_ms, e2e_step_s = stats.tolist()
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped)
    strong = world > 1 and args.scaling == "strong"
    total_elements = 2 * args.nx * args.ny if strong else n_el * world

    if rank == 0:
        peak, peak_source = measured_peak()
        algorithmic = 12 * n_el + 16 * n_v + 8 * nnz + 8 * n_v
        achieved = algorithmic / (kernel_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC,
            "value": total_elements * args.steps / (total_ms * 1e-3),
            "unit": "elements/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps,
            "higher_is_better": True,
            "scaling": "strong" if strong else "weak",
            "vs_baseline": None,
            "dtype": "f64",
            "data": "synthetic",
            "config": workload_config(args),
            "clocks": clocks,
            "gpu_launches": gpu_launches,
            "roofline": {
                "bound": "hbm",
                "achieved": achieved,
                "peak": peak,
                "unit": "GB/s",
                "frac": achieved / peak,
                "traffic": ncu_traffic(args),
                "traffic_source": "static: one `ncu --set full` capture of this kernel on this configuration, committed as "
                "profiles/roofline_traffic.json (not re-measured in this run; DRAM writes still in L2 at kernel end are not in it)",
                "peak_source": peak_source,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "kernel": ("assemble_tiled_kernel<double,384,3,SINSIN,true,false>" if os.environ.get("TFEM_TILED_CONSUMERS") == "384" else "assemble_tiled_ws_kernel<double,12,12,3,SINSIN,true,false>") if args.path == "tiled" else "local_forms + segment_reduce x2",
                "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": algorithmic,
                "bytes_per_element": algorithmic / n_el,
            },
        }
        line["config"]["symbolic_seconds"] = {"csr_pattern": round(symbolic_pattern_s, 3),
                                              "tile_plan": None if symbolic_plan_s is None else round(symbolic_plan_s, 3)}
        if symbolic_warm is not None:
            line["config"]["symbolic_seconds"]["note"] = "first call (CUDA module loading, allocator growth); *_warm = the same phase repeated"
            line["config"]["symbolic_seconds"]["csr_pattern_warm"] = round(symbolic_warm[0], 4)
            line["config"]["symbolic_seconds"]["tile_plan_warm"] = round(symbolic_warm[1], 4)
        if args.permuted:
            line["config"]["workload"] += "; vertices and elements randomly renumbered (default_rng(7)): locality stress, NOT the headline layout"
        if assembler is not None and args.path == "tiled":
            line["config"]["exchange"] = exchange_kind
        if plan is not None:
            line["config"]["tile_plan"] = {"tiles": plan.n_tiles, "rows_per_tile": args.rows_per_tile, "halo_factor": round(plan.halo_factor, 4),
                                           "index_bytes": plan.index_bytes, "max_vert": plan.max_vert, "max_elem": plan.max_elem, "templates": plan.n_templates,
                                           "lattice": plan.lattice}
        if e2e:
            line["e2e"] = {
                "value": total_elements / e2e_step_s,
                "unit": "elements/s",
                "h2d_bytes_per_step": e2e["h2d"],
                "d2h_bytes_per_step": e2e["d2h"],
                "ms_per_step": e2e_step_s * 1e3,
                "api": e2e.get("api") or ("Basis.assemble_from_host(pinned coords, StiffnessMass, Load, pinned values, pinned load)" if world == 1
                else "StripHostPipeline(StripAssembly, depth=2).step(pinned coords, pinned values, pinned load): every step copies its coordinates in and its CSR values + load out; consecutive steps overlap"),
            }
            if "serial_ms" in e2e:
                line["e2e"]["ms_per_step_one_at_a_time"] = e2e["serial_ms"]
        if world == 1 and not args.no_cpu_baseline:
            cpu_value, sample, timings = cpu_reference_run(args.nx, args.ny, repeats=2)
            line["cpu_baseline"] = {"value": cpu_value, "unit": "elements/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": sample, "host_cpus": os.cpu_count(), "stage_seconds": timings}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line of the contract, on the process's original stdout."""
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    global _REAL_STDOUT
    # Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is exactly one
    # JSON line on stdout, so everything else is sent to stderr.
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
