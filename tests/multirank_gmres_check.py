"""Multi-rank check of the device GMRES solve, run under torchrun (one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tests/multirank_gmres_check.py
Every rank assembles its rows of a non-symmetric Jacobian on its GPU and solves with GMRES + Jacobi (operand gathered and dot
products summed over NCCL); the owned part of the solution is compared with scipy's direct solve of the oracle's global matrix."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CH = [1.5, 3000.0]
PF = [1.0, 0.0045, 0.5, 1.0, 0.899, -0.910, -0.899, 0.020, 0.200]


def main():
    import torch
    import torch.distributed as dist
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    import petiga_b200 as pb
    from tests.common import Case, state_vectors

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

    pf = lambda mattype: Case(2, dof=2, p=2, N=(16, 12), limits=(-1.0, 1.0), periodic=True, mattype=mattype)
    cases = [
        ("cahnhilliard N=32", Case(2, p=2, N=32, C=1, periodic=True), "IJACOBIAN", "CAHNHILLIARD2D", CH, 1e7),
        ("cahnhilliard N=48", Case(2, p=2, N=48, C=1, periodic=True), "IJACOBIAN", "CAHNHILLIARD2D", CH, 1e7),
        ("patternform baij", pf(None), "IEJACOBIAN", "PATTERNFORMATION", PF, 2.5),
        ("patternform aij", pf("aij"), "IEJACOBIAN", "PATTERNFORMATION", PF, 2.5),
    ]
    nfail = 0
    for name, case, slot, form, prm, shift in cases:
        o = case.oracle()
        o.setup()
        rp, ci, rs = o.pattern(world)
        dof = case.dof
        n = (len(rp) - 1) * dof
        U, V = state_vectors(n)
        W = np.random.default_rng(8).random(n) if slot == "IEJACOBIAN" else None
        Ko, _ = o.assemble(slot, form, prm, size=world, shift=shift, V=V, t=0.3, U=U, W=W, t0=0.2)
        M = (sp.bsr_matrix((Ko.reshape(-1, dof, dof), ci, rp), shape=(n, n)) if dof > 1 else sp.csr_matrix((Ko.reshape(-1), ci, rp), shape=(n, n))).tocsc()
        b = np.random.default_rng(1).standard_normal(n)
        xs = spla.spsolve(M, b)
        r0, r1 = int(rs[rank]) * dof, int(rs[rank + 1]) * dof
        g = case.product(rank=rank, size=world, nccl=comm.value, device=local)
        g.SetForm(slot, form, prm)
        A, B, X, vU, vV, vW = g.CreateMat(), g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateVec()
        vU.set(U[r0:r1]); vV.set(V[r0:r1]); B.set(b[r0:r1])
        if W is not None:
            vW.set(W[r0:r1])
            g.ComputeIEJacobian(shift, vV, 0.3, vU, 0.2, vW, A)
        else:
            g.ComputeIJacobian(shift, vV, 0.3, vU, A)
        its, rel, reason = g.Solve(A, B, X, rtol=1e-10, ksp_type="gmres", return_reason=True)
        e_x = np.linalg.norm(X.get() - xs[r0:r1]) / np.linalg.norm(xs)
        ok = e_x <= 1e-8 and rel <= 1e-10 and reason == pb.iga.KSP_CONVERGED_RTOL
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        if rank == 0:
            print("%-20s gmres %s x=%.1e its=%d rel=%.1e reason=%d" % (name, "ok " if flag.item() == 0 else "FAIL", e_x, its, rel, reason), flush=True)
        nfail += int(flag.item() != 0)
        for v in (A, B, X, vU, vV, vW):
            v.destroy()
        g.Destroy()
    dist.barrier()
    if rank == 0:
        print("GMRES MULTIRANK %s: %d failures on %d ranks" % ("PASS" if nfail == 0 else "FAIL", nfail, world), flush=True)
    L.petiga_cuda_comm_destroy(comm)
    dist.destroy_process_group()
    return 1 if nfail else 0


if __name__ == "__main__":
    sys.exit(main())
