"""Time IGAComputeSystem with Laplace collocation on the device: 3-D p = 3 at 128^3 and 2-D p = 2 at 512^2 by default.

    python tools/colloc_probe.py [--case 3:3:128 2:2:512 ...] [--steps 50] [--warmup 5]

--case dim:p:N.  Every face carries a boundary value (identity rows), identity geometry.  The system is assembled once as a
warm-up, then `steps` assemblies are enqueued back to back on the IGA's stream (async mode) between two CUDA events.  The
collocation kernel is write-bound: the model counts (p+1)^dim * 8 B of values per row plus 8 B of right-hand side (the 1-D tables
and row bases it reads stay in L1/L2); TB/s is that model over the measured time per assembly, not measured HBM traffic.  The
value array of one assembly (above 126 MB at the default sizes) does not fit the L2.  The GPU name and power limit are read in
the same run and printed first."""
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
    ap.add_argument("--case", nargs="+", default=["3:3:128", "2:2:512"])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    import petiga_b200 as pb
    print(json.dumps(card()), flush=True)
    for spec in args.case:
        dim, p, N = (int(v) for v in spec.split(":"))
        stream = torch.cuda.Stream()
        g = pb.IGA(dim, 1)
        g.SetUseCollocation(True)
        for d in range(dim):
            g.AxisInitUniform(d, p, N)
        g.SetStream(stream.cuda_stream)
        g.SetUp()
        for d in range(dim):
            for s in range(2):
                g.SetBoundaryValue(d, s, 0, 0.0)
        g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
        A, B = g.CreateMat(), g.CreateVec()
        for _ in range(args.warmup):
            g.ComputeSystem(A, B)
        kernel_ms = g.GetStat("last_kernel_ms")
        g.SetOption("async", 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            g.ComputeSystem(A, B)
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        g.SetOption("async", 0)
        g.Synchronize()
        rows = B.size
        model = 8.0 * A.nnz + 8.0 * rows
        print(json.dumps({"dim": dim, "p": p, "N": N, "rows": rows, "nnz": A.nnz, "steps": args.steps,
                          "ms_per_assembly": round(ms, 4), "last_kernel_ms_warmup": round(kernel_ms, 4),
                          "model_bytes": model, "model_bytes_per_ms": round(model / ms, 1),
                          "model_TBps": round(model / (ms * 1e-3) / 1e12, 3)}), flush=True)
        A.destroy()
        B.destroy()
        g.Destroy()


if __name__ == "__main__":
    main()
