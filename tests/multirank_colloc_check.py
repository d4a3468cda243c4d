"""Multi-rank check of collocation, run under torchrun (one rank per GPU):
   python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tests/multirank_colloc_check.py
Every rank assembles the rows of the nodes it owns (no exchange); its CSR block and right-hand side are compared with the rows of
the reference's global system (tests/colloc_ref.py, permuted to the global numbering), and the distributed GMRES + Jacobi solution
with scipy's direct solve of that global system."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    import scipy.sparse.linalg as spla
    import petiga_b200 as pb
    from oracle.oracle import partition
    from tests.colloc_ref import Axis, Space, assemble

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

    cases = [   # name, dim, degrees, elements, form, params
        ("laplace 2d p2", 2, (2, 2), (16, 12), "LAPLACE_COLLOCATION", ()),
        ("convtest 2d p3/p2", 2, (3, 2), (14, 16), "CONVTEST_COLLOCATION", (1.0, 1.0)),
        ("convtest 3d p3", 3, (3, 3, 3), (8, 8, 8), "CONVTEST_COLLOCATION", (2.0, 0.5)),
    ]
    nfail = 0
    for name, dim, ps, Ns, form, prm in cases:
        g = pb.IGA(dim, 1, rank=rank, size=world, nccl=comm.value, device=local)
        g.SetUseCollocation(True)
        for d in range(dim):
            g.AxisInitUniform(d, ps[d], Ns[d])
        g.SetUp()
        values = {(d, s): 0.5 * s for d in range(dim) for s in range(2)}
        for (d, s), v in values.items():
            g.SetBoundaryValue(d, s, 0, v)
        g.SetForm("SYSTEM", form, prm)
        A, B, X = g.CreateMat(), g.CreateVec(), g.CreateVec()
        g.ComputeSystem(A, B)
        axes = [Axis(ps[d], g.AxisGetKnots(d)) for d in range(dim)]
        grid, _ = partition(world, 0, dim, [len(a.span_off) for a in axes])
        space = Space(axes, grid)
        An, Fn = assemble(axes, form, prm, values=values)
        n = An.shape[0]
        nodes = np.indices([a.nnp for a in axes][::-1]).reshape(dim, -1)[::-1].T
        glob = np.array([space.global_of(tuple(w)) for w in nodes])     # natural -> global
        nat = np.empty(n, dtype=np.int64)
        nat[glob] = np.arange(n)
        Ag = An[nat][:, nat].tocsr()
        Ag.sort_indices()
        Fg = Fn[nat]
        r0, r1 = space.rank_start[rank], space.rank_start[rank + 1]
        blk = Ag[r0:r1]
        rp, ci = A.pattern()
        vals = A.values().reshape(-1)
        e_pat = np.array_equal(rp, blk.indptr) and np.array_equal(ci, blk.indices)
        e_K = np.linalg.norm(vals - blk.data) / np.linalg.norm(blk.data) if e_pat else np.inf
        e_F = np.linalg.norm(B.get() - Fg[r0:r1]) / max(np.linalg.norm(Fg[r0:r1]), 1e-300)
        its, rel, reason = g.Solve(A, B, X, rtol=1e-11, ksp_type="gmres", maxits=20000, return_reason=True)
        xs = spla.spsolve(Ag.tocsc(), Fg)
        e_x = np.linalg.norm(X.get() - xs[r0:r1]) / np.linalg.norm(xs)
        ok = e_pat and e_K <= 1e-12 and (e_F <= 1e-12 or np.linalg.norm(Fg[r0:r1]) == 0) and e_x <= 1e-8 and reason == pb.iga.KSP_CONVERGED_RTOL
        flag = torch.tensor([0 if ok else 1], device="cuda")
        dist.all_reduce(flag)
        if rank == 0:
            print("%-20s %s K=%.1e F=%.1e x=%.1e its=%d reason=%d" % (name, "ok " if flag.item() == 0 else "FAIL", e_K, e_F, e_x, its, reason), flush=True)
        nfail += int(flag.item() != 0)
        for v in (A, B, X):
            v.destroy()
        g.Destroy()
    dist.barrier()
    if rank == 0:
        print("COLLOCATION MULTIRANK %s: %d failures on %d ranks" % ("PASS" if nfail == 0 else "FAIL", nfail, world), flush=True)
    L.petiga_cuda_comm_destroy(comm)
    dist.destroy_process_group()
    return 1 if nfail else 0


if __name__ == "__main__":
    sys.exit(main())
