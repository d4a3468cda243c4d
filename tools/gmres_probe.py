"""Device GMRES(30) + Jacobi on the cfg-5 CahnHilliard2D IJacobian (512^2 by default): time per iteration.

    python tools/gmres_probe.py [--mesh 512] [--shift 1e3 1e7] [--maxit 300] [--restart 30]

For each shift: the IJacobian is assembled on the device at the seeded cfg-5 state, one warm-up solve runs, then one solve with
a fixed maxit is timed with CUDA events on the IGA's stream.  Prints one JSON line per shift.  The bytes-per-iteration model is
12 nnz (matrix values + column indices) + 16 (k+1) n (the basis read twice, by the multi-dot and by the update, for the k-th
Arnoldi step) averaged over a restart cycle + O(n); at 512^2 the basis (31 vectors, ~67 MB) is largely L2-resident, so the TB/s
figure is the model over the time, not HBM traffic.  The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        out["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.TimeoutExpired):
        out["power_limit_and_max_sm_clock"] = "nvidia-smi unavailable"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mesh", type=int, default=512)
    ap.add_argument("--shift", type=float, nargs="+", default=[1e3, 1e7])
    ap.add_argument("--maxit", type=int, default=300)
    ap.add_argument("--restart", type=int, default=30)
    args = ap.parse_args()
    import numpy as np
    import torch
    from petiga_b200.cases import baseline_config, state_vectors
    print(json.dumps(card()), flush=True)
    case, slot, form, prm, _, _ = baseline_config("cfg5", mesh=args.mesh)
    stream = torch.cuda.Stream()
    g = case.product(setup=False)
    g.SetStream(stream.cuda_stream)
    g.SetUp()
    g.SetForm(slot, form, prm)
    n = args.mesh * args.mesh
    U, V = state_vectors(n)
    vU, vV, A, B, X = g.CreateVec(), g.CreateVec(), g.CreateMat(), g.CreateVec(), g.CreateVec()
    vU.set(U); vV.set(V)
    B.set(np.random.default_rng(1).standard_normal(n))
    m = args.restart
    for shift in args.shift:
        g.ComputeIJacobian(shift, vV, 0.0, vU, A)
        g.Synchronize()
        g.Solve(A, B, X, rtol=1e-10, maxits=min(args.maxit, 2 * m), ksp_type="gmres", restart=m)      # warm-up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        its, rel, reason = g.Solve(A, B, X, rtol=1e-10, maxits=args.maxit, ksp_type="gmres", restart=m, return_reason=True)
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        # bytes per iteration, averaged over the Arnoldi steps k = 0..its-1 of the restart cycles
        ks = np.arange(its) % m
        bytes_it = 12.0 * A.nnz + 16.0 * float(np.mean(ks + 1)) * n + 6 * 8.0 * n
        print(json.dumps({"mesh": args.mesh, "n": n, "nnz": A.nnz, "shift": shift, "restart": m, "maxit": args.maxit, "iterations": its,
                          "reason": reason, "relres": rel, "solve_ms": round(ms, 3), "ms_per_iteration": round(ms / max(its, 1), 4),
                          "model_bytes_per_iteration": bytes_it, "model_TBps": round(bytes_it / (ms / max(its, 1) * 1e-3) / 1e12, 3)}),
              flush=True)
    for v in (vU, vV, A, B, X):
        v.destroy()
    g.Destroy()


if __name__ == "__main__":
    main()
