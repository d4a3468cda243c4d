"""Time IGAComputeFunction and IGAComputeJacobian of Bratu collocation next to IGAComputeSystem of Laplace collocation on the same
3-D p = 3 plan (128^3 by default).

    python tools/colloc_state_probe.py [--case 3:3:128 ...] [--steps 50] [--warmup 5]

--case dim:p:N.  Every face carries a boundary value, identity geometry, lambda = 1, a seeded state U.  Each driver runs `warmup`
times, then `steps` times back to back on the IGA's stream (async mode) between two CUDA events.  Bytes models (what the kernel
must move; the 1-D tables and row bases stay in L1/L2):
  System:   (p+1)^dim * 8 B of values + 8 B of right-hand side per row (written)
  Jacobian: (p+1)^dim * 8 B of values per row (written) + the ghost-box state read once (8 B per node)
  Function: 8 B written + 8 B of state read per row
TB/s is the model over the measured time per call, not measured HBM traffic.  The GPU name and power limit are read in the same
run and printed first."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.colloc_probe import card   # noqa: E402


def timed(g, stream, steps, warmup, call):
    import torch
    for _ in range(warmup):
        call()
    g.Synchronize()
    g.SetOption("async", 1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        call()
    e1.record(stream)
    e1.synchronize()
    g.SetOption("async", 0)
    g.Synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="+", default=["3:3:128"])
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
        g.SetForm("FUNCTION", "BRATU_COLLOCATION", (1.0,))
        g.SetForm("JACOBIAN", "BRATU_COLLOCATION", (1.0,))
        A, B, U = g.CreateMat(), g.CreateVec(), g.CreateVec()
        rows = B.size
        U.set(np.random.default_rng(0).uniform(0.0, 0.5, rows))
        res = {"dim": dim, "p": p, "N": N, "rows": rows, "nnz": A.nnz, "steps": args.steps}
        models = {"system": 8.0 * A.nnz + 8.0 * rows, "jacobian": 8.0 * A.nnz + 8.0 * rows, "function": 16.0 * rows}
        calls = {"system": lambda: g.ComputeSystem(A, B), "jacobian": lambda: g.ComputeJacobian(U, A), "function": lambda: g.ComputeFunction(U, B)}
        for name in ("system", "jacobian", "function"):
            ms = timed(g, stream, args.steps, args.warmup, calls[name])
            res[name] = {"ms": round(ms, 4), "model_bytes": models[name], "model_TBps": round(models[name] / (ms * 1e-3) / 1e12, 3)}
        print(json.dumps(res), flush=True)
        for o in (A, B, U):
            o.destroy()
        g.Destroy()


if __name__ == "__main__":
    main()
