#!/usr/bin/env python
"""bench.py -- element-assembly throughput of libpetiga_cuda on BASELINE.json's headline configuration.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--path auto|quadrature] [--mesh 128] [--dump-outputs DIR]

Workload (config.workload): demo/Poisson3D of the reference, p=3 C2, 128^3 elements, dof=1, AIJ, Dirichlet 1.0 on
all six faces, one `IGAComputeSystem` per step (zero -> integrate -> fix-up -> scatter -> fully assembled).
metric = assembled Mnnz/s (scalar nonzeros of the assembled matrix / time of one assembly); elements/s is reported
beside it.  N > 1 (torchrun, one rank per GPU): the same global mesh split by the reference's box partition
(strong scaling), value = global nnz / max-over-ranks time.

--impl reference times the CPU restatement of the reference's assembly (oracle/, "port": the reference needs
PETSc+MPI+gfortran and cannot be built here) on all host cores, one emulated MPI rank per core.

--dump-outputs DIR (one process) writes what the last timed step computed, so that two builds can be compared output for
output on identical inputs: DIR/rhs.npy + rhs_index.npy (right-hand side at a fixed seeded sample of 2^21 positions, all of
them when it is shorter) and DIR/matrix_values.npy + matrix_rows.npy + matrix_cols.npy (2^20 sampled nonzeros of the
assembled matrix with their row and column), all float64: 56 MiB at most.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NNZ_FULL, NEL_FULL = 741217625, 128 ** 3       # SURVEY.md 8: cfg 2
W_E = 64 * (4096 * 7 + 64 * 3)                 # algorithmic FLOP per element, SURVEY.md 8(d)
FP64_NOMINAL_TFLOPS = 37.2                     # 148 SM x 64 DFMA lanes x 2 x 1.965 GHz


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for (ts, line) in self.rows:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def build_case(mesh, p=3, geometry=None):
    from petiga_b200.cases import Case
    geo = None if geometry in (None, "identity") else ("perturbed", 0.05)     # SURVEY 8d cfg 2g
    return Case(3, p=p, N=mesh, bcv=[(d, s, 0, 1.0) for d in range(3) for s in range(2)], geometry=geo)


# ------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, threads=None, per_rank=12):
    """The reference's CPU assembly algorithm on the host cores (oracle/cpu_reference.py; the only place this file executes
    oracle/): T emulated MPI ranks on T threads, reference box partition, ghost rows through a stash + assembly-end sum,
    library rebuilt with -march=native on this box."""
    from oracle.cpu_reference import run_cfg2_sample
    r = run_cfg2_sample(steps, warmup, T=threads, per_rank=per_rank, native=True)
    r["mnnz_per_s"] = r["elements_per_s"] * NNZ_FULL / NEL_FULL / 1e6
    return r


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    r = cpu_reference_run(args.steps, args.warmup, threads=args.cpu_threads)
    line = {
        "impl": "reference", "metric": "assembled_Mnnz_per_s", "value": r["mnnz_per_s"], "unit": "Mnnz/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "elements_per_s": r["elements_per_s"],
        "config": {"workload": "demo/Poisson3D p=3 C2 128^3 dof=1 AIJ IGAComputeSystem (CPU sample, see cpu_baseline.sample)"},
        "cpu_baseline": {"value": r["mnnz_per_s"], "unit": "Mnnz/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                         "cpu_model": r["cpu_model"], "ghost_row_sum": True, "stash_entries_per_step": r["stash_entries"]},
        "e2e": {"value": r["mnnz_per_s"], "unit": "Mnnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)
    return 0


# ------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  NCCL (NCCL_DEBUG=VERSION on the GPU boxes) and other native libraries write
    to fd 1 directly, so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--path", default="auto", choices=["auto", "quadrature"])
    ap.add_argument("--mesh", type=int, default=128)
    ap.add_argument("--geometry", default="identity", choices=["identity", "perturbed"])
    ap.add_argument("--quad-impl", type=int, default=-1, help="-1 = library choice, 0 = sum-factorised (v2), 1 = pair-loop, 2 = generic, 3 = persistent DMMA kernel (v3)")
    ap.add_argument("--cpu-threads", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-quad", action="store_true")
    ap.add_argument("--no-solve", action="store_true", help="skip the assemble + device CG solve figure (e2e_solve)")
    ap.add_argument("--no-parity", action="store_true", help="skip the golden-vector parity cases run before the timed region")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary BASELINE configurations (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's matrix and right-hand side "
                                                           "as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the GPU path, not of --impl reference")
        return main_reference(args)

    import ctypes as C
    import numpy as np
    import torch
    import petiga_b200 as pb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libpetiga_cuda has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one process: run it with --gpus 1")
    torch.cuda.set_device(local)
    L = pb.load_cuda()
    nccl = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            raw = (C.c_ubyte * 128)()
            assert L.petiga_cuda_comm_unique_id(raw) == 0, L.petiga_cuda_last_error()
            idbuf.copy_(torch.tensor(list(raw), dtype=torch.uint8))
        dist.broadcast(idbuf, 0)
        raw = (C.c_ubyte * 128)(*idbuf.cpu().tolist())
        comm = C.c_void_p()
        assert L.petiga_cuda_comm_init(C.byref(comm), world, rank, raw, local) == 0, L.petiga_cuda_last_error()
        nccl = comm.value

    # -------- parity on the live communicator, before anything is timed: small cases against committed golden vectors
    #          (CPU-oracle outputs in natural numbering, tests/golden/multirank_cases.npz; no oracle code runs here) --------
    parity = None
    if not args.no_parity:
        from petiga_b200.parity import check_cases

        def _allgather(a):
            if world == 1:
                return [a]
            t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            sizes = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
            dist.all_gather(sizes, torch.tensor([t.numel()], dtype=torch.int64, device="cuda"))
            mx = int(max(int(x.item()) for x in sizes))
            pad = torch.zeros(mx, dtype=t.dtype, device="cuda"); pad[:t.numel()] = t
            outs = [torch.zeros(mx, dtype=t.dtype, device="cuda") for _ in range(world)]
            dist.all_gather(outs, pad)
            return [o[:int(n.item())].cpu().numpy() for o, n in zip(outs, sizes)]

        def _allreduce(a):
            if world == 1:
                return a
            t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()
            dist.all_reduce(t)
            return t.cpu().numpy()
        parity = check_cases(rank, world, nccl, local, _allgather, _allreduce)

    stream = torch.cuda.Stream()
    case = build_case(args.mesh, geometry=args.geometry)
    g = case.product(rank=rank, size=world, nccl=nccl, device=local, setup=False)
    g.SetStream(stream.cuda_stream)
    g.SetUp()
    g.SetOption("path", {"auto": 0, "quadrature": 1}[args.path])
    g.SetOption("quad_impl", args.quad_impl)
    g.SetForm("SYSTEM", "POISSON")
    A, B = g.CreateMat(), g.CreateVec()          # IGACreateMat: pattern built once, outside the timed region
    nnz_local, nvec_local = A.nnz, B.size
    nnz_t = torch.tensor([nnz_local], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(nnz_t)
    nnz_global = int(nnz_t.item())
    nel_global = args.mesh ** 3

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            g.ComputeSystem(A, B)
        path_used = int(g.GetStat("last_path"))
        quad_flops = g.GetStat("last_flops")
        quad_kernel_label = kernel_name(g, {1: "quadrature", 2: "kronecker"}.get(path_used, "?"), mapped=args.geometry != "identity")
        # -------- timed region: device-resident (inputs already in HBM) --------
        sampler = ClockSampler(local)
        sampler.start()
        time.sleep(0.3)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # kernel time of the dominant kernel: a few synchronous steps (last_kernel_ms needs the step's events complete)
        kern_ms = 0.0
        for _ in range(5):
            g.ComputeSystem(A, B)
            kern_ms += g.GetStat("last_kernel_ms") / 5
        barrier()
        # the K timed steps are enqueued back to back on the IGA's stream (device-resident hand-off, no host wait per step)
        g.SetOption("async", 1)
        l0 = g.GetStat("launches")
        t0 = time.time()
        e0.record(stream)
        for _ in range(args.steps):
            g.ComputeSystem(A, B)
        e1.record(stream)
        barrier()
        t1 = time.time()
        g.SetOption("async", 0)
        ms = e0.elapsed_time(e1) / args.steps
        launches = int(g.GetStat("launches") - l0)
        snapshot = snapshot_outputs(g, A, B) if args.dump_outputs else None     # before the calls below overwrite A and B
        if t1 - t0 < 1.0:      # too short for nvidia-smi to see: keep the same kernel busy ~1.5 s for the clock record only
            tend = time.time() + 1.5
            while time.time() < tend:
                g.ComputeSystem(A, B)
            t1 = time.time()
        clocks = sampler.stop(t0, t1)
    if snapshot is not None:
        write_outputs(args.dump_outputs, snapshot)
        snapshot = None

    # -------- the per-element quadrature path on the same workload (reported beside the headline, not as it) --------
    quad = None
    if args.path == "auto" and path_used == 2 and not args.no_quad:
        g.SetOption("path", 1)
        with torch.cuda.stream(stream):
            for _ in range(2):
                g.ComputeSystem(A, B)
            barrier()
            e0.record(stream)
            qsteps, qk = 3, 0.0
            ql0 = g.GetStat("launches")
            for _ in range(qsteps):
                g.ComputeSystem(A, B)
                qk += g.GetStat("last_kernel_ms")
            e1.record(stream)
            barrier()
            qflops, qlabel, qlaunch = g.GetStat("last_flops"), kernel_name(g, "quadrature", mapped=args.geometry != "identity"), (g.GetStat("launches") - ql0) / qsteps
        qt = torch.tensor([e0.elapsed_time(e1) / qsteps, qk / qsteps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(qt, op=dist.ReduceOp.MAX)
        quad = {"ms_per_step": float(qt[0]), "kernel_ms": float(qt[1]), "steps": qsteps, "flops": qflops, "kernel": qlabel, "launches": qlaunch}
        g.SetOption("path", 0)
        g.ComputeSystem(A, B)

    ms_t = torch.tensor([ms, kern_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms, kern_ms = float(ms_t[0]), float(ms_t[1])

    # -------- end-to-end through the C-ABI with HOST buffers (pinned), D2H of the assembled system inside --------
    e2e = None
    if not args.no_e2e:
        plan = g.plan()
        nval, nvec = A.nnz, B.size
        hv, hr = C.c_void_p(), C.c_void_p()
        assert L.petiga_cuda_host_alloc(C.byref(hv), C.c_size_t(nval * 8)) == 0
        assert L.petiga_cuda_host_alloc(C.byref(hr), C.c_size_t(nvec * 8)) == 0
        ksteps = max(2, min(args.steps, 5))
        L.petiga_cuda_compute_host.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
        bc = _bc_struct(case)
        with torch.cuda.stream(stream):
            for it in range(1 + ksteps):
                if it == 1:
                    barrier()
                    e0.record(stream)
                rc = L.petiga_cuda_set_bc(plan, C.byref(bc))          # this step's inputs: the BC tables, host -> device
                assert rc == 0
                rc = L.petiga_cuda_compute_host(plan, 2, 0, 0.0, None, 0.0, None, hv, hr)
                assert rc == 0, L.petiga_cuda_last_error()
            e1.record(stream)
            barrier()
        ms_e = torch.tensor([e0.elapsed_time(e1) / ksteps], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms_e, op=dist.ReduceOp.MAX)
        chk = float(np.ctypeslib.as_array(C.cast(hr, C.POINTER(C.c_double)), shape=(nvec,))[:8].sum())
        e2e = {"value": nnz_global / (float(ms_e[0]) * 1e-3) / 1e6, "unit": "Mnnz/s", "ms_per_step": float(ms_e[0]),
               "h2d_bytes_per_step": C.sizeof(bc), "d2h_bytes_per_step": (nval + nvec) * 8, "steps": ksteps, "rhs_checksum8": chk}
        L.petiga_cuda_host_free(hv); L.petiga_cuda_host_free(hr)

    # -------- assemble + solve with the matrix never leaving the device (SURVEY 8 f-4): IGAComputeSystem, then CG + Jacobi on the
    #          device CSR (IGACreateKSP / KSPSolve of the host mirror), then ONLY the solution vector goes to the host --------
    e2e_solve = None
    if not args.no_solve and args.geometry == "identity":
        X = g.CreateVec()
        with torch.cuda.stream(stream):
            g.SetOption("path", 0)
            g.ComputeSystem(A, B)
            g.Solve(A, B, X, rtol=1e-8, maxits=20)                # warm-up: allocations, NCCL channels
            barrier()
            e0.record(stream)
            g.ComputeSystem(A, B)
            em = torch.cuda.Event(enable_timing=True)
            em.record(stream)
            its, rel = g.Solve(A, B, X, rtol=1e-8, maxits=5000)
            xh = X.get()                                           # device -> host: the solution, nothing else
            e1.record(stream)
            barrier()
        t_all = torch.tensor([e0.elapsed_time(e1), em.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
        e2e_solve = {"ms": float(t_all[0]), "solve_ms": float(t_all[1]), "cg_iterations": int(its), "relative_residual": float(rel),
                     "rtol": 1e-8, "preconditioner": "jacobi", "d2h_bytes": int(nvec_local * 8), "h2d_bytes": 0, "matrix_bytes_over_pcie": 0,
                     "ms_per_iteration": float(t_all[1]) / max(int(its), 1),
                     "spmv_GBps_per_gpu": 12.0 * nnz_local / (float(t_all[1]) / max(int(its), 1) * 1e-3) / 1e9,
                     "solution_checksum": float(np.abs(xh).sum()),
                     "note": "IGAComputeSystem + KSPSolve (CG, Jacobi) with the CSR consumed in place on the device; spmv_GBps counts 12 B per nonzero "
                             "(value + column index) over the whole iteration time (SpMV + 2 dot products + 2 vector updates)"}
        X.destroy()

    # -------- the other BASELINE configurations, one GPU, device-resident (secondary rows of SURVEY 8d) --------
    configs = None
    if world == 1 and not args.no_configs and args.mesh == 128 and args.geometry == "identity":
        A.destroy(); B.destroy(); g.Destroy()
        A = B = g = None
        torch.cuda.empty_cache()
        configs = sweep_configs(stream, measured_peaks())

    if rank != 0:
        return 0
    peaks = measured_peaks()
    # FP64 FMA peak measured on this device (DFMA micro-benchmark inside libpetiga_cuda; SURVEY 8d): MEASURED_PEAKS.json has none
    fb, fs = C.c_double(0.0), C.c_double(0.0)
    fp64 = {"nominal_tflops": FP64_NOMINAL_TFLOPS}
    if L.petiga_cuda_measure_fp64(local, C.c_double(1.0), C.byref(fb), C.byref(fs)) == 0 and fb.value > 0:
        fp64.update(measured_burst_tflops=fb.value, measured_sustained_tflops=fs.value)
    fp64_peak = fp64.get("measured_sustained_tflops", FP64_NOMINAL_TFLOPS)
    fp64_src = ("measured DFMA micro-benchmark (petiga_cuda_measure_fp64, sustained 1 s; burst %.1f; nominal %.1f)" % (fb.value, FP64_NOMINAL_TFLOPS)
                if "measured_sustained_tflops" in fp64 else "nominal FP64 FMA peak (148 SM x 64 lanes x 2 x 1.965 GHz)")
    sec = ms * 1e-3
    value = nnz_global / sec / 1e6
    if path_used == 2:     # separable path: one write-once kernel per step, HBM bound (SURVEY 8d)
        alg_bytes = 8.0 * (nnz_local + nvec_local)
        # launch duration = CUDA-event time of the timed region / K (each step is exactly one launch of this kernel; the
        # inter-launch gaps are inside, so this is the conservative figure); kernel_ms_sync = the plan's own per-launch events
        roof = {"bound": "hbm", "achieved": alg_bytes / (ms * 1e-3) / 1e9, "peak": peaks.get("hbm_gbs", 6650.0), "unit": "GB/s",
                "traffic": None, "kernel": "kron_rows_kernel", "kernel_ms": ms, "kernel_ms_sync": kern_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s"}
    else:                  # quadrature path: FP64 bound; achieved = the FP64 operations the kernels EXECUTE (library stat) / kernel time
        roof = {"bound": "fp64", "achieved": quad_flops / (kern_ms * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                "traffic": None, "kernel": quad_kernel_label, "kernel_ms": kern_ms, "executed_flop_per_launch": quad_flops,
                "algorithmic_flop_W_e": float(W_E) * (nel_global / world), "peak_source": fp64_src,
                "hbm_floor_ms": 8.0 * (nnz_local + nvec_local) / (peaks.get("hbm_gbs", 6650.0) * 1e9) * 1e3}
    roof["frac"] = roof["achieved"] / roof["peak"]
    try:    # dram bytes per launch from the committed ncu --set full capture of the same kernel (profiles/)
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "kron_rows_kernel" if path_used == 2 else quad_kernel_label.split(" ")[0]
        if world == 1 and args.mesh == prof[key]["mesh"] and args.geometry == "identity":
            roof["traffic"] = prof[key]["dram_bytes_per_launch"]
            roof["traffic_source"] = prof[key]["source"]
    except Exception:
        pass
    line = {
        "metric": "assembled_Mnnz_per_s", "value": value, "unit": "Mnnz/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "elements_per_s": nel_global / sec,
        "config": {"workload": "demo/Poisson3D p=3 C2 %d^3 dof=1 AIJ IGAComputeSystem%s" % (args.mesh, "" if args.geometry == "identity" else " on a mapped geometry (cfg 2g)"),
                   "elements": nel_global, "nnz": nnz_global,
                   "path": {1: "quadrature", 2: "kronecker"}.get(path_used, str(path_used)),
                   "l2": "each step rewrites the %.2f GB value array (> 126 MB L2)" % (nnz_local * 8 / 1e9),
                   "parallelism": "box partition, %d rank(s)" % world},
        "clocks": clocks, "gpu_launches": launches, "roofline": roof, "fp64_peak": fp64,
    }
    if quad:
        tf = quad["flops"] / (quad["kernel_ms"] * 1e-3) / 1e12
        line["quadrature_path"] = {"ms_per_step": quad["ms_per_step"], "value": nnz_global / (quad["ms_per_step"] * 1e-3) / 1e6, "unit": "Mnnz/s",
                                   "elements_per_s": nel_global / (quad["ms_per_step"] * 1e-3), "kernel": quad["kernel"],
                                   "kernel_ms": quad["kernel_ms"], "launches_per_step": quad["launches"],
                                   "roofline": {"bound": "fp64", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
                                                "peak_source": fp64_src, "executed_flop_per_step": quad["flops"],
                                                "algorithmic_flop_W_e": float(W_E) * (nel_global / world),
                                                "speedup_over_reference_loop_nest_flops": float(W_E) * (nel_global / world) / max(quad["flops"], 1.0),
                                                "hbm_floor_ms": 8.0 * (nnz_local + nvec_local) / (peaks.get("hbm_gbs", 6650.0) * 1e9) * 1e3,
                                                "note": "achieved = FP64 operations the kernels execute (sum factorisation + FP64 tensor cores: "
                                                        "far fewer than SURVEY 8(d)'s W_e) / kernel time; the binding floors of this path are the "
                                                        "red.global.add.f64 rate and shared-memory bandwidth (DESIGN.md 3.2b), not the FP64 pipe"}}
    if e2e:
        line["e2e"] = e2e
    if e2e_solve:
        line["e2e_solve"] = e2e_solve
    if parity is not None:
        line["parity"] = parity
    if configs is not None:
        line["configs"] = configs
    if world == 1 and not args.no_cpu_baseline:
        # the reference's CPU algorithm on ALL host cores (a bounded sample of the same workload: ~10-20 s of CPU work), with the
        # ghost-row sum; cfg 1 at its full size on one core beside it (BASELINE.json configs[0] is the CPU-runnable case)
        r = cpu_reference_run(2, 1, threads=args.cpu_threads, per_rank=12)
        line["cpu_baseline"] = {"value": r["mnnz_per_s"], "unit": "Mnnz/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
                                "elements_per_s": r["elements_per_s"], "cpu_model": r["cpu_model"], "ghost_row_sum": True}
        try:
            from oracle.cpu_reference import run_cfg1_full
            c1 = run_cfg1_full()
            line["cpu_baseline"]["cfg1_full_size_1core"] = {"value": c1["mnnz_per_s"], "unit": "Mnnz/s", "ms": c1["seconds"] * 1e3,
                                                             "elements_per_s": c1["elements_per_s"]}
        except Exception as e:      # the headline must not die on the side figure
            line["cpu_baseline"]["cfg1_full_size_1core"] = {"error": str(e)}
    _emit(line)
    return 0


def sweep_configs(stream, peaks):
    """cfg 1, 2g, 3, 4, 5 of BASELINE.json on one GPU: per config the path and kernel that ran, CUDA-event ms per call,
    Mnnz/s, elements/s and the roofline fraction of its bound (HBM for the write-once path: 8 B per stored value; FP64 for
    the quadrature kernels: the flops the kernel EXECUTES, reported by the library, over the measured DFMA peak)."""
    import numpy as np
    import torch
    import petiga_b200 as pb
    from petiga_b200.cases import baseline_config, state_vectors
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        traffic = {}
    out = []
    hbm = peaks.get("hbm_gbs", 6650.0)
    for name, steps in (("cfg1", 20), ("cfg2g", 3), ("cfg3", 5), ("cfg4", 5), ("cfg5", 20), ("cfg5f", 20)):
        case, slot, form, prm, w_e, state = baseline_config(name)
        g = case.product(setup=False)
        g.SetStream(stream.cuda_stream)
        g.SetUp()
        g.SetForm(slot, form, prm)
        A = g.CreateMat() if slot in ("SYSTEM", "IJACOBIAN") else None
        B = g.CreateVec() if slot in ("SYSTEM", "IFUNCTION") else None
        U = V = None
        if state:
            t = g.CreateVec(); n = t.size; t.destroy()
            u, v = state_vectors(n)
            U, V = g.CreateVec(), g.CreateVec()
            U.set(u); V.set(v)

        def call():
            if slot == "SYSTEM": g.ComputeSystem(A, B)
            elif slot == "IJACOBIAN": g.ComputeIJacobian(1.0e3, V, 0.0, U, A)
            else: g.ComputeIFunction(1.0e3, V, 0.0, U, B)
        with torch.cuda.stream(stream):
            for _ in range(3):
                call()
            torch.cuda.synchronize()
            g.SetOption("async", 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = g.GetStat("launches")
            e0.record(stream)
            for _ in range(steps):
                call()
            e1.record(stream)
            torch.cuda.synchronize()
            g.SetOption("async", 0)
        ms = e0.elapsed_time(e1) / steps
        nel = int(np.prod(g.info()["nel"]))
        nnz = (A.nnz * (case.dof ** 2 if A.baij else 1)) if A is not None else 0
        nvec = B.size if B is not None else 0
        path = {1: "quadrature", 2: "kronecker"}.get(int(g.GetStat("last_path")), "?")
        hybrid = path == "kronecker" and form == "L2PROJECTION"       # matrix by the separable path, load vector by a quadrature kernel
        row = {"config": name, "workload": WORKLOADS[name], "path": path, "kernel": kernel_name(g, path, mapped=case.geometry is not None) + (" + " + kernel_name(g, "quadrature") if hybrid else ""), "ms_per_call": ms, "steps": steps,
               "launches_per_call": (g.GetStat("launches") - l0) / steps, "elements": nel, "nnz": nnz,
               "elements_per_s": nel / (ms * 1e-3), "value": (nnz / (ms * 1e-3) / 1e6) if nnz else None, "unit": "Mnnz/s"}
        bytes_alg = 8.0 * (nnz + nvec * (1 + (2 if state else 0))) + (8.0 * 3 * g.info()["nnp"][0] * g.info()["nnp"][1] * g.info()["nnp"][2] if case.geometry else 0.0)
        hb = {"bound": "hbm", "achieved": bytes_alg / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "algorithmic_bytes": bytes_alg}
        hb["frac"] = hb["achieved"] / hb["peak"]
        if path == "kronecker":      # write-once matrix (+ the small load-vector kernel of the hybrid case): HBM bound
            row["roofline"] = hb
        else:
            fl = g.GetStat("last_flops")
            fp = {"bound": "fp64", "achieved": fl / (ms * 1e-3) / 1e12, "peak": peaks.get("fp64_tflops_measured", 34.1), "unit": "TFLOP/s",
                  "executed_flop_per_call": fl, "algorithmic_flop_W_e": float(w_e) * nel,
                  "note": "achieved counts the FP64 operations the kernel executes (library stat last_flops), not SURVEY 8(d)'s W_e"}
            fp["frac"] = fp["achieved"] / fp["peak"]
            row["roofline"] = fp
            row["roofline_hbm"] = hb
        key = "%s/%s" % (name, path)
        row["traffic"] = traffic.get(key, {}).get("dram_bytes_per_launch")
        out.append(row)
        for x in (A, B, U, V):
            if x is not None:
                x.destroy()
        g.Destroy()
        torch.cuda.empty_cache()
    return out


WORKLOADS = {
    "cfg1": "demo/Poisson2D p=2 C1 64x64 dof=1 AIJ IGAComputeSystem",
    "cfg2": "demo/Poisson3D p=3 C2 128^3 dof=1 AIJ IGAComputeSystem",
    "cfg2g": "demo/Poisson3D p=3 C2 128^3 on a mapped geometry (Greville + 0.05 sin sin sin), IGAComputeSystem",
    "cfg3": "demo/L2Projection 3-D p=4 C3 64^3 dof=1 AIJ IGAComputeSystem (-function linear)",
    "cfg4": "demo/Elasticity3D p=2 C1 96^3 dof=3 BAIJ IGAComputeSystem",
    "cfg5": "demo/CahnHilliard2D p=2 C1 512^2 periodic IGAComputeIJacobian (shift 1e3, seed 20261017 state)",
    "cfg5f": "demo/CahnHilliard2D p=2 C1 512^2 periodic IGAComputeIFunction",
}


def kernel_name(g, path, mapped=False):
    if path == "kronecker":
        return "kron_rows_kernel"
    impl = int(g.GetStat("last_impl"))
    if impl == 3:      # matrix kernel + the kernel that integrates the element vectors (and D' on mapped geometry)
        return ("quad_sf3r_kernel" if int(g.GetStat("last_sf3_variant")) == 0 else "quad_sf3_kernel") + (" (+ sf3_geom_kernel)" if mapped else " (+ quad_vec3_kernel)")
    return {0: "quad_sf_kernel", 1: "quad_kernel", 2: "quad_gen_kernel", 4: "quad_vec3_kernel"}.get(impl, "?")


def _bc_struct(case):
    import ctypes as C

    class BC(C.Structure):
        _fields_ = [("vcount", (C.c_int * 2) * 3), ("vfield", ((C.c_int * 64) * 2) * 3), ("vvalue", ((C.c_double * 64) * 2) * 3),
                    ("lcount", (C.c_int * 2) * 3), ("lfield", ((C.c_int * 64) * 2) * 3), ("lvalue", ((C.c_double * 64) * 2) * 3),
                    ("fixtableU", C.c_void_p)]
    bc = BC()
    for (a, s, f, v) in case.bcv:
        k = bc.vcount[a][s]
        bc.vfield[a][s][k] = f
        bc.vvalue[a][s][k] = v
        bc.vcount[a][s] = k + 1
    return bc


DUMP_SEED = 20261017
DUMP_MATRIX_ENTRIES, DUMP_RHS_ENTRIES = 1 << 20, 1 << 21      # 3 x 8 MiB + 2 x 16 MiB of float64


def _sample(n, k):
    """Sorted positions of a fixed seeded sample of k of n entries (all of them when n <= k)."""
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=k, replace=False))


def _device_array(ptr, n, typestr):
    """Zero-copy torch view of n elements of device memory owned by libpetiga_cuda."""
    import types
    import torch
    cai = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}
    return torch.as_tensor(types.SimpleNamespace(__cuda_array_interface__=cai), device="cuda")


def snapshot_outputs(g, A, B):
    """Device copies of a seeded sample of what the last ComputeSystem left in A and B: right-hand side entries with their
    positions, matrix values with their row and column (the AIJ pattern of IGACreateMat)."""
    import ctypes as C
    import torch
    import petiga_b200 as pb
    g.Synchronize()
    L = pb.load_cuda()
    L.petiga_cuda_plan_pattern.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 4
    nrows, nnz, rp, ci = C.c_int(), C.c_int64(), C.c_void_p(), C.c_void_p()
    assert L.petiga_cuda_plan_pattern(g.plan(), 0, C.byref(nrows), C.byref(nnz), C.byref(rp), C.byref(ci)) == 0, L.petiga_cuda_last_error()
    assert not A.baij and nnz.value == A.nnz
    pos = torch.from_numpy(_sample(A.nnz, DUMP_MATRIX_ENTRIES)).cuda()
    rowptr = _device_array(rp.value, nrows.value + 1, "<i4").long()
    idx = torch.from_numpy(_sample(B.size, DUMP_RHS_ENTRIES)).cuda()
    return {"matrix_values": _device_array(A.device_ptr(), A.nnz, "<f8")[pos],
            "matrix_rows": torch.searchsorted(rowptr, pos, right=True) - 1,
            "matrix_cols": _device_array(ci.value, A.nnz, "<i4")[pos],
            "rhs": _device_array(B.device_ptr(), B.size, "<f8")[idx], "rhs_index": idx}


def write_outputs(out_dir, snapshot):
    """DIR/<name>.npy, float64 throughout (row, column and position indices are exact in it)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in snapshot.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


if __name__ == "__main__":
    sys.exit(main())
