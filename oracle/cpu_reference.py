"""CPU timing of the reference's assembly algorithm on the host cores (bench.py's cpu_baseline / --impl reference legs).

TEST/BENCH INFRASTRUCTURE: this is the oracle (oracle/petiga_oracle.c, kind "port": the reference itself needs PETSc + MPI +
gfortran, none of which exist in the image) run the way `mpiexec -n T` runs PetIGA: T emulated ranks of the reference's own
box partition, one host thread each (ctypes releases the GIL), every rank looping over its element box
(src/petigaksp.c:149-202), adding the rows it owns straight into the global CSR and the rows of other ranks into its stash;
then the receiving side of MatAssemblyEnd/VecAssemblyEnd adds the stashes (src/petigaksp.c:197-200).  The library is
rebuilt with -march=native on the box it runs on (oracle.build(native=True), in a temporary directory)."""
import os
import threading
import time

import numpy as np

from . import oracle as orc


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


class ReferenceRun:
    """T emulated ranks on T threads over one global system (shared CSR arrays)."""

    def __init__(self, dim, dof, p, mesh, bcv, slot, form, params, T, C=-1, periodic=False, native=True, state=False, shift=0.0):
        self.T, self.slot, self.form, self.params, self.dof, self.shift = T, slot, form, list(params), dof, shift
        self.objs = []
        for r in range(T):
            o = orc.OracleIGA(dim, dof, native=native)
            for d in range(dim):
                o.axis_uniform(d, p, mesh[d], 0.0, 1.0, C, periodic)
            for (a, s, f, v) in bcv:
                o.boundary_value(a, s, f, v)
            self.objs.append(o)
        self.rp, self.ci, self.rs = self.objs[0].pattern(T)
        self.pat = self.objs[0]._pat[T]                     # read-only during assembly: shared by every rank
        n, nnz = len(self.rp) - 1, len(self.ci)
        self.want_mat = slot in ("MATRIX", "SYSTEM", "JACOBIAN", "IJACOBIAN")
        self.want_vec = slot in ("VECTOR", "SYSTEM", "FUNCTION", "IFUNCTION")
        self.vals = np.zeros((nnz, dof, dof)) if self.want_mat else None
        self.rhs = np.zeros((n, dof)) if self.want_vec else None
        self.U = self.V = None
        if state:
            from petiga_b200.cases import state_vectors     # plain numpy helper (seeded synthetic state of SURVEY 8d)
            self.U, self.V = state_vectors(n * dof)
        L = self.objs[0].L
        self.stash = [L.oiga_stash_create() for _ in range(T)]
        self.nel = int(np.prod(mesh))
        self.nnz_scalar = nnz * dof * dof
        self.stash_entries = 0

    def step(self):
        """One IGACompute<slot>: zero, element loops, stash exchange.  Returns wall seconds."""
        T, L = self.T, self.objs[0].L
        prm = np.ascontiguousarray(self.params + [0.0] * 4, dtype=np.float64)
        bar = threading.Barrier(T)
        errs = []
        d = orc._d

        def work(r):
            try:
                o = self.objs[r]
                r0, r1 = int(self.rs[r]), int(self.rs[r + 1])
                if self.want_mat:
                    self.vals[self.rp[r0]:self.rp[r1]] = 0.0          # MatZeroEntries, each rank its rows
                if self.want_vec:
                    self.rhs[r0:r1] = 0.0
                bar.wait()
                rc = L.oiga_assemble_rank_stash(o.h, T, r, orc.SLOT[self.slot], orc.FORM[self.form], d(prm), self.shift, d(self.V), 0.0,
                                                d(self.U), self.pat, d(self.vals), d(self.rhs), self.stash[r])
                assert rc == 0, rc
                bar.wait()                                            # MatAssemblyBegin: all stashes complete
                for s in range(T):                                    # MatAssemblyEnd: add what the others stashed for me
                    if s != r:
                        L.oiga_stash_apply(self.stash[s], self.dof, self.pat, r, d(self.vals), d(self.rhs))
            except Exception as e:      # pragma: no cover
                errs.append(e)
                bar.abort()

        t0 = time.perf_counter()
        th = [threading.Thread(target=work, args=(r,)) for r in range(T)]
        for x in th:
            x.start()
        for x in th:
            x.join()
        dt = time.perf_counter() - t0
        if errs:
            raise errs[0]
        self.stash_entries = sum(int(L.oiga_stash_count(s)) for s in self.stash)
        return dt

    def close(self):
        L = self.objs[0].L
        for s in self.stash:
            L.oiga_stash_destroy(s)
        self.stash = []


def run_cfg2_sample(steps, warmup, T=None, per_rank=12, native=True):
    """BASELINE cfg 2 (Poisson3D p=3 C2, Dirichlet 1.0 on six faces, IGAComputeSystem) on a bounded sample: per_rank^3
    elements for each of T emulated ranks, arranged by the reference's own processor grid."""
    T = T or host_threads()
    grid, _ = orc.partition(T, 0, 3, [per_rank * T] * 3)
    mesh = [per_rank * g for g in grid]
    bcv = [(a, s, 0, 1.0) for a in range(3) for s in range(2)]
    run = ReferenceRun(3, 1, 3, mesh, bcv, "SYSTEM", "POISSON", [], T, native=native)
    times = []
    for it in range(warmup + steps):
        dt = run.step()
        if it >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    out = dict(seconds=sec, elements=run.nel, elements_per_s=run.nel / sec, cores=T, mesh=mesh, stash_entries=run.stash_entries,
               nnz_sample=run.nnz_scalar, checksum=float(run.rhs.sum()), cpu_model=orc.cpu_model(),
               sample="Poisson3D p=3 C2 IGAComputeSystem on a %dx%dx%d sub-mesh = %d^3 elements for each of %d emulated MPI ranks "
                      "(reference box partition %s, one host thread per rank, ghost rows through a PETSc-style stash and added in "
                      "an assembly-end phase; %d stashed entries per step); CPU: %s; Mnnz/s = elements/s x (741217625 nnz / 2097152 "
                      "elements of the full 128^3 mesh), i.e. extrapolated linearly in elements" %
                      (mesh[0], mesh[1], mesh[2], per_rank, T, "x".join(map(str, grid)), run.stash_entries, orc.cpu_model()))
    run.close()
    return out


def run_cfg1_full(T=1, native=True, repeats=3):
    """BASELINE cfg 1 at its FULL size (Poisson2D p=2 64x64, IGAComputeSystem, 1 MPI rank as BASELINE.json states)."""
    bcv = [(a, s, 0, 1.0) for a in range(2) for s in range(2)]
    run = ReferenceRun(2, 1, 2, [64, 64], bcv, "SYSTEM", "POISSON", [], T, native=native)
    run.step()
    sec = min(run.step() for _ in range(repeats))
    out = dict(seconds=sec, elements=run.nel, nnz=run.nnz_scalar, mnnz_per_s=run.nnz_scalar / sec / 1e6, elements_per_s=run.nel / sec, cores=T)
    run.close()
    return out
