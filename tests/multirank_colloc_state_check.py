"""Multi-rank check of Bratu by collocation, run under torchrun (one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tests/multirank_colloc_state_check.py
Every rank gathers the state on its collocation ghost box (NCCL state halo) and computes the Function/IFunction entries and the
Jacobian/IJacobian rows of the nodes it owns; they are compared with the rows of the reference's global operators
(tests/colloc_state_ref.py, permuted to the global numbering).  Then a distributed Newton solve (device F, J and GMRES + Jacobi)
is compared with scipy's Newton solution of the reference system."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    import petiga_b200 as pb
    from oracle.oracle import partition
    from tests.colloc_ref import Axis, Space
    from tests.colloc_state_ref import jacobian, newton, operators, residual

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = pb.load_cuda()
    idbuf = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        raw = (C.c_ubyte * 128)()
        assert L.petiga_cuda_comm_unique_id(raw) == 0
        idbuf.copy_(torch.tensor(list(raw), dtype=torch.uint8))
    dist.broadcast(idbuf, 0)
    raw = (C.c_ubyte * 128)(*idbuf.cpu().tolist())
    comm = C.c_void_p()
    assert L.petiga_cuda_comm_init(C.byref(comm), world, rank, raw, local) == 0, L.petiga_cuda_last_error()

    cases = [   # name, dim, degrees, elements (a 2-D or 3-D processor grid: ghost boxes reach up to 4 or 8 owners)
        ("bratu 2d p3", 2, (3, 3), (16, 14)),
        ("bratu 2d p2/p4", 2, (2, 4), (18, 12)),
        ("bratu 3d p3", 3, (3, 3, 3), (8, 8, 8)),
    ]
    lam, shift = 1.5, 3.0
    nfail = 0
    for name, dim, ps, Ns in cases:
        g = pb.IGA(dim, 1, rank=rank, size=world, nccl=comm.value, device=local)
        g.SetUseCollocation(True)
        for d in range(dim):
            g.AxisInitUniform(d, ps[d], Ns[d])
        g.SetUp()
        values = {(d, s): 0.0 for d in range(dim) for s in range(2)}
        for (d, s), v in values.items():
            g.SetBoundaryValue(d, s, 0, v)
        for slot in ("FUNCTION", "JACOBIAN", "IFUNCTION", "IJACOBIAN"):
            g.SetForm(slot, "BRATU_COLLOCATION", (lam,))
        axes = [Axis(ps[d], g.AxisGetKnots(d)) for d in range(dim)]
        grid, _ = partition(world, 0, dim, [len(a.span_off) for a in axes])
        space = Space(axes, grid)
        ops = operators(axes)
        n = ops[0].shape[0]
        nodes = np.indices([a.nnp for a in axes][::-1]).reshape(dim, -1)[::-1].T
        glob = np.array([space.global_of(tuple(w)) for w in nodes])     # natural -> global
        nat = np.empty(n, dtype=np.int64)
        nat[glob] = np.arange(n)
        r0, r1 = space.rank_start[rank], space.rank_start[rank + 1]
        rng = np.random.default_rng(7)
        Un, Vn = rng.uniform(-0.4, 0.6, n), rng.uniform(-1, 1, n)       # natural numbering, the same on every rank
        Uv, Vv, F, J = g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateMat()
        Uv.set(Un[nat][r0:r1])
        Vv.set(Vn[nat][r0:r1])
        rp, ci = J.pattern()
        errs = []
        for slot in ("FUNCTION", "IFUNCTION", "JACOBIAN", "IJACOBIAN"):
            tr = slot.startswith("I")
            if slot.endswith("FUNCTION"):
                if tr:
                    g.ComputeIFunction(shift, Vv, 0.0, Uv, F)
                else:
                    g.ComputeFunction(Uv, F)
                ref = residual(ops, Un, lam, V=Vn if tr else None, values=values, axes=axes)[nat][r0:r1]
                errs.append(np.linalg.norm(F.get() - ref) / np.linalg.norm(ref))
            else:
                if tr:
                    g.ComputeIJacobian(shift, Vv, 0.0, Uv, J)
                else:
                    g.ComputeJacobian(Uv, J)
                Jg = jacobian(ops, Un, lam, shift=shift if tr else 0.0, values=values, axes=axes)[nat][:, nat].tocsr()
                Jg.sort_indices()
                blk = Jg[r0:r1]
                same = np.array_equal(rp, blk.indptr) and np.array_equal(ci, blk.indices)
                errs.append(np.linalg.norm(J.values().reshape(-1) - blk.data) / np.linalg.norm(blk.data) if same else np.inf)
        # distributed Newton from U = 0
        dU = g.CreateVec()
        Uv.set(np.zeros(r1 - r0))
        hist = []
        for _ in range(8):
            g.ComputeFunction(Uv, F)
            f2 = torch.tensor([float(np.sum(F.get() ** 2))], dtype=torch.float64, device="cuda")
            dist.all_reduce(f2)
            hist.append(float(np.sqrt(f2.item())))
            if hist[-1] <= 1e-10:
                break
            g.ComputeJacobian(Uv, J)
            its, rel, reason = g.Solve(J, F, dU, rtol=1e-11, ksp_type="gmres", restart=100, maxits=20000, return_reason=True)
            Uv.set(Uv.get() - dU.get())
        Ur, _ = newton(ops, lam, values, axes)
        e_newton = np.abs(Uv.get() - Ur[nat][r0:r1]).max() / np.abs(Ur).max()
        ok = all(e <= 1e-12 for e in errs) and hist[-1] <= 1e-10 and len(hist) <= 7 and e_newton <= 1e-9
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        if rank == 0:
            print("%-16s %s F=%.1e IF=%.1e J=%.1e IJ=%.1e newton steps=%d |F|=%.1e err=%.1e" %
                  (name, "ok " if flag.item() == 0 else "FAIL", *errs, len(hist) - 1, hist[-1], e_newton), flush=True)
        nfail += int(flag.item() != 0)
        for v in (Uv, Vv, F, J, dU):
            v.destroy()
        g.Destroy()
    dist.barrier()
    if rank == 0:
        print("COLLOCATION STATE MULTIRANK %s: %d failures on %d ranks" % ("PASS" if nfail == 0 else "FAIL", nfail, world), flush=True)
    L.petiga_cuda_comm_destroy(comm)
    dist.destroy_process_group()
    return 1 if nfail else 0


if __name__ == "__main__":
    sys.exit(main())
