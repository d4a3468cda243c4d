"""Isogeometric collocation on the device: the collocation kernel against the reference restatement (tests/colloc_ref.py) on
identity, mapped and rational geometry, in AIJ and BAIJ; a large identity-geometry case against scipy's Kronecker sum; bitwise
repeatability; GMRES solves of the assembled systems; the unsupported combinations of the C ABI; and the kernel's ptxas budget."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

import petiga_b200 as pb
from oracle.oracle import read_iga_file
from tests.colloc_ref import Axis, Space, assemble, l2_error_2d, scipy_laplace_kron
from tests.common import Case, rel_frobenius
from tests.geomutil import refine_annulus
from tests.test_host_collocation import CASES, make_iga

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_FACES = lambda dim, v: {(d, s): v for d in range(dim) for s in range(2)}   # noqa: E731


def _assemble_device(g, form, params, values, baij):
    """IGAComputeSystem on a collocation IGA (boundary values set here) -> (rowptr, colidx, values, rhs)."""
    if baij:
        g.SetMatType("baij")
    for (d, s), v in (values or {}).items():
        g.SetBoundaryValue(d, s, 0, v)
    g.SetForm("SYSTEM", form, params)
    A, B = g.CreateMat(), g.CreateVec()
    g.ComputeSystem(A, B)
    assert int(g.GetStat("last_path")) == 3          # PETIGA_PATH_COLLOCATION
    rp, ci = A.pattern()
    out = rp, ci, A.values().reshape(-1), B.get()
    A.destroy()
    B.destroy()
    return out


def _compare(g, axes, form, params, values, baij, X=None, W=None):
    rp, ci, vals, rhs = _assemble_device(g, form, params, values, baij)
    s = Space(axes)
    rpr, cir = s.pattern(0)
    assert np.array_equal(rp, rpr) and np.array_equal(ci, cir)
    Ar, Fr = assemble(axes, form, params, X=X, W=W, values=values)
    assert np.array_equal(Ar.indptr, rpr) and np.array_equal(Ar.indices, cir)
    assert rel_frobenius(vals, Ar.data) <= 1e-12
    if np.linalg.norm(Fr) == 0:
        assert np.abs(rhs).max() == 0
    else:
        assert rel_frobenius(rhs, Fr) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s_%s" % (c[0], "".join(map(str, c[1])), c[3]))
def test_identity_geometry(case, baij):
    dim, ps, Ns, Cs = case
    g = make_iga(dim, ps, Ns, Cs)
    axes = [Axis(ps[d], g.AxisGetKnots(d)) for d in range(dim)]
    _compare(g, axes, "LAPLACE_COLLOCATION", (), ALL_FACES(dim, 0.5), baij)
    g2 = make_iga(dim, ps, Ns, Cs)
    _compare(g2, axes, "CONVTEST_COLLOCATION", (1.5, 0.7), {(0, 0): 0.25, (dim - 1, 1): -1.0}, baij)


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
@pytest.mark.parametrize("form,params", [("LAPLACE_COLLOCATION", ()), ("CONVTEST_COLLOCATION", (1.0, 2.0))])
def test_mapped_geometry(form, params, baij):
    axes_f, nsd, X, W, rational = read_iga_file(os.path.join(GOLD, "cube_perturbed.dat"))
    assert not rational
    g = pb.IGA(3, 1)
    g.SetUseCollocation(True)
    for d, (p, U) in enumerate(axes_f):
        g.AxisSetKnots(d, p, U)
    g.SetGeometryArrays(X)
    g.SetUp()
    axes = [Axis(p, U) for p, U in axes_f]
    _compare(g, axes, form, params, ALL_FACES(3, 1.0), baij, X=X)


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
@pytest.mark.parametrize("height", [None, (3, 0.5)], ids=["2d", "3d"])
@pytest.mark.parametrize("form,params", [("LAPLACE_COLLOCATION", ()), ("CONVTEST_COLLOCATION", (0.5, 1.0))])
def test_rational_geometry(form, params, height, baij):
    class ColIGA(pb.IGA):
        def __init__(self, dim, dof):
            super().__init__(dim, dof)
            self.SetUseCollocation(True)
    g, X, W = refine_annulus(ColIGA, N=(5, 6), p=2, height=height)
    g.SetUp()
    dim = 2 if height is None else 3
    axes = [Axis(2, g.AxisGetKnots(d)) for d in range(dim)]
    _compare(g, axes, form, params, {(0, 0): 1.0, (1, 1): 2.0}, baij, X=X, W=W)


def _geometry_iga(kind):
    """collocation IGA on the perturbed cube (mapped) or the 3-D quarter annulus (NURBS) + its natural X"""
    if kind == "mapped":
        axes_f, nsd, X, W, rational = read_iga_file(os.path.join(GOLD, "cube_perturbed.dat"))
        g = pb.IGA(3, 1)
        g.SetUseCollocation(True)
        for d, (p, U) in enumerate(axes_f):
            g.AxisSetKnots(d, p, U)
        g.SetGeometryArrays(X)
    else:
        class ColIGA(pb.IGA):
            def __init__(self, dim, dof):
                super().__init__(dim, dof)
                self.SetUseCollocation(True)
        g, X, W = refine_annulus(ColIGA, N=(5, 6), p=2, height=(3, 0.5))
    g.SetUp()
    return g, X


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mapped", "rational"])
def test_laplacian_of_the_geometry_vanishes(kind):
    """An independent pin of the order-2 push-forward: on isoparametric geometry x_i = sum_b X_bi R_b, so the Laplace collocation
    matrix (no boundary rows) applied to each column of control-point coordinates is zero at every point."""
    g, X = _geometry_iga(kind)
    g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
    A, B = g.CreateMat(), g.CreateVec()
    g.ComputeSystem(A, B)
    rp, ci = A.pattern()
    M = sp.csr_matrix((A.values().reshape(-1), ci, rp), shape=(len(rp) - 1,) * 2)
    Xn = np.asarray(X).reshape(-1, 3)
    scale = abs(M).max() * np.abs(Xn).max()
    for i in range(3):
        assert np.abs(M @ Xn[:, i]).max() <= 1e-11 * scale, (kind, i, np.abs(M @ Xn[:, i]).max() / scale)
    A.destroy()
    B.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("slot", ["MATRIX", "VECTOR"])
def test_matrix_and_vector_slots(slot):
    """IGAComputeMatrix / IGAComputeVector through the C ABI: the same rows as the reference without boundary rows (these
    drivers never fix), the other output untouched."""
    import torch
    L = pb.load_cuda()
    L.petiga_cuda_compute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.petiga_cuda_form_select.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.petiga_cuda_finish.argtypes = [C.c_void_p]
    g, X = _geometry_iga("rational")
    for (d, s), v in ALL_FACES(3, 3.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    axes = [Axis(2, g.AxisGetKnots(d)) for d in range(3)]
    Ar, Fr = assemble(axes, "CONVTEST_COLLOCATION", (1.5, 0.5), X=X, W=_geometry_weights())
    plan = g.plan()
    slot_id = {"VECTOR": 0, "MATRIX": 1}[slot]
    prm = (C.c_double * 2)(1.5, 0.5)
    assert L.petiga_cuda_form_select(plan, slot_id, 17, prm, 2) == 0       # PETIGA_FORM_CONVTEST_COLLOCATION
    vals = torch.full((Ar.nnz,), 7.0, dtype=torch.float64, device="cuda")
    rhs = torch.full((Ar.shape[0],), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    assert L.petiga_cuda_compute(plan, slot_id, 0, 0.0, None, 0.0, None, C.c_void_p(vals.data_ptr()), C.c_void_p(rhs.data_ptr())) == 0
    assert L.petiga_cuda_finish(plan) == 0
    v, f = vals.cpu().numpy(), rhs.cpu().numpy()
    if slot == "MATRIX":
        assert rel_frobenius(v, Ar.data) <= 1e-12 and np.all(f == 7.0)
    else:
        assert rel_frobenius(f, Fr) <= 1e-12 and np.all(v == 7.0)


def _geometry_weights():
    return refine_annulus(_Rec, N=(5, 6), p=2, height=(3, 0.5))[2]


class _Rec:
    def __init__(self, dim, dof):
        pass

    def axis_knots(self, *a):
        pass

    def geometry(self, *a):
        pass


@pytest.mark.gpu
def test_large_kronecker_pin():
    """3-D p = 3, N = 48 (132651 rows): the device matrix against scipy's Kronecker sum, compared on the device."""
    import torch
    p, N = 3, 48
    g = make_iga(3, (p, p, p), (N, N, N), None)
    for (d, s), v in ALL_FACES(3, 0.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
    A, B = g.CreateMat(), g.CreateVec()
    g.ComputeSystem(A, B)
    rp, ci = A.pattern()
    axes = [Axis(p, g.AxisGetKnots(d)) for d in range(3)]
    K = scipy_laplace_kron(axes).tocsr()
    rows = np.repeat(np.arange(len(rp) - 1), np.diff(rp))
    expect = np.asarray(K[rows, ci]).ravel()
    ref = torch.tensor(expect, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    d2, r2 = C.c_double(), C.c_double()
    L = pb.load_cuda()
    rc = L.petiga_cuda_diff_norm2(C.c_void_p(A.device_ptr()), C.c_void_p(ref.data_ptr()), C.c_size_t(len(expect)), C.byref(d2), C.byref(r2))
    assert rc == 0
    assert np.sqrt(d2.value / r2.value) <= 1e-13
    # the pattern holds every nonzero of the Kronecker sum: the entries read at its positions carry all of K's norm
    K.eliminate_zeros()
    assert abs(np.sqrt(r2.value) - np.linalg.norm(K.data)) <= 1e-14 * np.linalg.norm(K.data)
    assert K.nnz <= len(ci)
    A.destroy()
    B.destroy()


@pytest.mark.gpu
def test_bitwise_repeatable():
    g = make_iga(3, (3, 2, 4), (5, 6, 4), None)
    for (d, s), v in ALL_FACES(3, 0.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    g.SetForm("SYSTEM", "CONVTEST_COLLOCATION", (1.0, 1.0))
    A, B = g.CreateMat(), g.CreateVec()
    g.ComputeSystem(A, B)
    v1, f1 = A.values().copy(), B.get().copy()
    g.ComputeSystem(A, B)
    v2, f2 = A.values(), B.get()
    assert v1.tobytes() == v2.tobytes() and f1.tobytes() == f2.tobytes()


@pytest.mark.gpu
def test_gmres_laplace_constant():
    g = make_iga(3, (3, 3, 3), (8, 8, 8), None)
    for (d, s), v in ALL_FACES(3, 1.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
    A, b, x = g.CreateMat(), g.CreateVec(), g.CreateVec()
    g.ComputeSystem(A, b)
    its, rn, reason = g.Solve(A, b, x, rtol=1e-12, ksp_type="gmres", maxits=5000, return_reason=True)
    assert reason == pb.iga.KSP_CONVERGED_RTOL, (its, rn, reason)
    assert np.abs(x.get() - 1.0).max() <= 1e-9


@pytest.mark.gpu
def test_gmres_convtest_error_matches_direct_solve():
    """ConvTest collocation, p = 2, N = 64: GMRES(30) + Jacobi reaches rtol 1e-10 within 200 iterations, and its L2 error
    (IGAComputeErrorNorm on the Galerkin IGA of the same axes: same numbering) is within 1 % of a direct solve's."""
    p, N = 2, 64
    g = make_iga(2, (p, p), (N, N), None)
    for (d, s), v in ALL_FACES(2, 0.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    g.SetForm("SYSTEM", "CONVTEST_COLLOCATION", (1.0, 1.0))
    A, b, x = g.CreateMat(), g.CreateVec(), g.CreateVec()
    g.ComputeSystem(A, b)
    its, rn, reason = g.Solve(A, b, x, rtol=1e-10, ksp_type="gmres", restart=30, maxits=200, return_reason=True)
    assert reason == pb.iga.KSP_CONVERGED_RTOL and its <= 200, (its, rn, reason)
    rp, ci = A.pattern()
    M = sp.csr_matrix((A.values().reshape(-1), ci, rp), shape=(len(rp) - 1,) * 2)
    u_direct = spl.spsolve(M.tocsc(), b.get())
    gal = make_iga(2, (p, p), (N, N), None, colloc=False)
    errs = []
    for u in (x.get(), u_direct):
        v = gal.CreateVec()
        v.set(u)
        errs.append(gal.ComputeErrorNorm(0, v, "ConvTest")[0])
        v.destroy()
    assert abs(errs[0] - errs[1]) <= 0.01 * errs[1], errs
    axes = [Axis(p, g.AxisGetKnots(d)) for d in range(2)]
    assert abs(errs[1] - l2_error_2d(axes, u_direct)) <= 1e-3 * errs[1]


@pytest.mark.gpu
def test_unsupported_combinations_leave_the_device_usable():
    """The library's own checks (C ABI, below the host mirror): a Galerkin form on a collocation plan, a collocation form on a
    Galerkin plan, and compute_scalar on a collocation plan are PETIGA_CUDA_ERR_SUP with no sticky CUDA error; a Galerkin
    assembly afterwards still matches the oracle."""
    import torch
    from tests.gpu_common import check_against_oracle
    L = pb.load_cuda()
    L.petiga_cuda_compute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.petiga_cuda_form_select.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.petiga_cuda_compute_scalar.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    buf = torch.zeros(1 << 16, dtype=torch.float64, device="cuda")
    rhs = torch.zeros(1 << 12, dtype=torch.float64, device="cuda")
    col = make_iga(2, (2, 2), (4, 4), None)
    plan = col.plan()
    assert L.petiga_cuda_form_select(plan, 2, 1, None, 0) == 0            # PETIGA_FORM_LAPLACE (Galerkin)
    assert L.petiga_cuda_compute(plan, 2, 0, 0.0, None, 0.0, None, C.c_void_p(buf.data_ptr()), C.c_void_p(rhs.data_ptr())) == 3
    S = (C.c_double * 1)()
    prm = (C.c_double * 3)(0.0, 4.0, 0.0)
    assert L.petiga_cuda_compute_scalar(plan, 0, prm, 3, None, 1, S) == 3
    gal = Case(2, p=2, N=4).product()
    gplan = gal.plan()
    assert L.petiga_cuda_form_select(gplan, 2, 16, None, 0) == 0           # PETIGA_FORM_LAPLACE_COLLOCATION
    assert L.petiga_cuda_compute(gplan, 2, 0, 0.0, None, 0.0, None, C.c_void_p(buf.data_ptr()), C.c_void_p(rhs.data_ptr())) == 3
    torch.cuda.synchronize()
    check_against_oracle(Case(2, p=2, N=4), "SYSTEM", "POISSON")


def test_colloc_kernel_register_budget():
    """ptxas -v of the in-tree build: no stack frame, no spills; the identity-geometry kernels keep 64 registers or fewer (4 CTAs
    of 256 threads per SM), the geometry kernels stay at their CUDA 12.9 counts."""
    libdir = pb.lib_dir()
    path = os.path.join(libdir, "pc_colloc.ptxas.log")
    if not os.path.exists(path):
        pytest.skip("library not built in-tree")
    txt = open(path).read()
    budget = {(1, 0): 64, (2, 0): 64, (3, 0): 64, (1, 1): 96, (2, 1): 128, (3, 1): 168}
    seen = 0
    for (dim, geo), cap in budget.items():
        sym = "colloc_kernelILi%dELb%dE" % (dim, geo)
        m = re.search(r"Function properties for [^\n]*%s[^\n]*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                      r"[^\n]*Used (\d+) registers" % re.escape(sym), txt)
        assert m, sym
        stack, st, ld, regs = map(int, m.groups())
        assert stack == 0 and st == 0 and ld == 0, (sym, stack, st, ld)
        assert regs <= cap, (sym, regs)
        seen += 1
    assert seen == 6


@pytest.mark.gpu
def test_multirank_collocation():
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(root, "tests", "multirank_colloc_check.py")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    print(out.stdout[-4000:])
    assert "COLLOCATION MULTIRANK PASS" in out.stdout
