"""GMRES(m) with right Jacobi preconditioning on the device (petiga_cuda_solve_gmres, KSPSetType(ksp, KSPGMRES)): the
non-symmetric Jacobians of the nonlinear and time-dependent forms solved where they were assembled.  Every solve is checked
against scipy's direct solve of the same device-assembled matrix."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import petiga_b200 as pb
from petiga_b200.iga import (KSP_CONVERGED_ATOL, KSP_CONVERGED_RTOL, KSP_DIVERGED_ITS, KSP_DIVERGED_NANORINF)
from tests.common import Case, state_vectors

pytestmark = pytest.mark.gpu

CH = [1.5, 3000.0]                                                   # demo/CahnHilliard2D.c {theta, alpha}
PF = [1.0, 0.0045, 0.5, 1.0, 0.899, -0.910, -0.899, 0.020, 0.200]    # demo/PatternFormation.c AppCtx (IMPLICIT)
PETSC_ERR_SUP, PETSC_ERR_ARG_IDN, PETSC_ERR_ARG_OUTOFRANGE = 56, 61, 63


def scipy_matrix(A, dof):
    rp, ci = A.pattern()
    vals = A.values()
    bs = dof if A.baij else 1
    n = (len(rp) - 1) * bs
    if A.baij:
        return sp.bsr_matrix((vals.reshape(-1, bs, bs), ci, rp), shape=(n, n)).tocsr()
    return sp.csr_matrix((vals, ci, rp), shape=(n, n))


def ch_jacobian(N, shift, mattype=None):
    """CahnHilliard2D IJacobian (p = 2, C^1, periodic) at the seeded cfg-5 state."""
    case = Case(2, p=2, N=N, C=1, periodic=True, mattype=mattype)
    g = case.product()
    g.SetForm("IJACOBIAN", "CAHNHILLIARD2D", CH)
    U, V = state_vectors(N * N)
    vU, vV, A = g.CreateVec(), g.CreateVec(), g.CreateMat()
    vU.set(U); vV.set(V)
    g.ComputeIJacobian(shift, vV, 0.0, vU, A)
    return g, A, 1


def pf_jacobian(mattype=None):
    """PatternFormation IEJacobian, dof 2, N = (16, 12), shift 2.5 (BAIJ bs 2 by default)."""
    case = Case(2, dof=2, p=2, N=(16, 12), limits=(-1.0, 1.0), periodic=True, mattype=mattype)
    g = case.product()
    g.SetForm("IEJACOBIAN", "PATTERNFORMATION", PF)
    n = 16 * 12 * 2
    U, V = state_vectors(n)
    U0 = np.random.default_rng(8).random(n)
    vU, vV, vW, A = g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateMat()
    vU.set(U); vV.set(V); vW.set(U0)
    g.ComputeIEJacobian(2.5, vV, 0.3, vU, 0.2, vW, A)
    return g, A, 2


def system(case, form, prm=()):
    g = case.product()
    g.SetForm("SYSTEM", form, prm)
    A, B = g.CreateMat(), g.CreateVec()
    g.ComputeSystem(A, B)
    return g, A, B


def solve_and_check(g, A, dof, rtol=1e-10, restart=30, seed=1):
    M = scipy_matrix(A, dof)
    b = np.random.default_rng(seed).standard_normal(M.shape[0])
    xs = spla.spsolve(M.tocsc(), b)
    B, X = g.CreateVec(), g.CreateVec()
    B.set(b)
    its, rel, reason = g.Solve(A, B, X, rtol=rtol, ksp_type="gmres", restart=restart, return_reason=True)
    x = X.get()
    assert reason == KSP_CONVERGED_RTOL and rel <= rtol, (its, rel, reason)
    assert np.linalg.norm(x - xs) <= 1e-8 * np.linalg.norm(xs), (its, np.linalg.norm(x - xs) / np.linalg.norm(xs))
    return its, x


@pytest.mark.parametrize("N", [32, 48])
def test_cahnhilliard_ijacobian(N):
    g, A, dof = ch_jacobian(N, 1e7)
    M = scipy_matrix(A, dof)
    assert spla.norm(M - M.T) > 1e-3 * spla.norm(M)          # the matrix is not symmetric
    its, _ = solve_and_check(g, A, dof)
    assert 0 < its < 200


@pytest.mark.parametrize("mattype", [None, "aij"])
def test_patternformation_iejacobian(mattype):
    g, A, dof = pf_jacobian(mattype)
    assert A.baij == (mattype is None)
    solve_and_check(g, A, dof)


@pytest.mark.parametrize("case,form,prm", [
    (Case(3, dof=3, p=2, N=4, bcv=[(0, 0, c, 0.0) for c in range(3)] + [(0, 1, 0, 1.0)]), "ELASTICITY3D", (1.0, 1.0)),   # BAIJ bs 3
    (Case(2, dof=4, p=2, N=(6, 5)), "MASS", ()),                                                                          # BAIJ bs 4
])
def test_block_systems_match_cg(case, form, prm):
    g, A, B = system(case, form, prm)
    M = scipy_matrix(A, case.dof)
    xs = spla.spsolve(M.tocsc(), B.get())
    Xg, Xc = g.CreateVec(), g.CreateVec()
    its, rel, reason = g.Solve(A, B, Xg, rtol=1e-12, ksp_type="gmres", return_reason=True)
    assert reason == KSP_CONVERGED_RTOL and rel <= 1e-12
    g.Solve(A, B, Xc, rtol=1e-12)                                        # CG on the same system
    xg, xc = Xg.get(), Xc.get()
    assert np.linalg.norm(xg - xs) <= 1e-8 * np.linalg.norm(xs)
    assert np.linalg.norm(xg - xc) <= 1e-8 * np.linalg.norm(xc)


def test_restart_lengths_agree():
    g, A, dof = ch_jacobian(32, 1e7)
    _, x5 = solve_and_check(g, A, dof, restart=5)
    _, x30 = solve_and_check(g, A, dof, restart=30)
    assert np.linalg.norm(x5 - x30) <= 1e-8 * np.linalg.norm(x30)


@pytest.mark.parametrize("dim", [1, 2])
def test_identity_system_happy_breakdown(dim):
    """Poisson with every node Dirichlet (p = 1, one element): the matrix is the identity, the first Arnoldi step breaks down."""
    case = Case(dim, p=1, N=1, bcv=[(d, s, 0, 1.0 + d + 2 * s) for d in range(dim) for s in range(2)])
    g, A, B = system(case, "POISSON")
    M = scipy_matrix(A, 1)
    assert np.array_equal(M.toarray(), np.eye(M.shape[0]))
    X = g.CreateVec()
    its, rel, reason = g.Solve(A, B, X, rtol=1e-10, ksp_type="gmres", return_reason=True)
    x, b = X.get(), B.get()
    assert its == 1 and reason in (KSP_CONVERGED_RTOL, KSP_CONVERGED_ATOL)
    assert np.all(np.isfinite(x)) and np.allclose(x, b, rtol=1e-14, atol=0)


def test_maxit_reports_diverged_its():
    """At the bench's shift Jacobi is too weak for CahnHilliard: the solve stops at maxit with rc 0 and says so."""
    g, A, dof = ch_jacobian(32, 1e3)
    M = scipy_matrix(A, dof)
    b = np.random.default_rng(1).standard_normal(M.shape[0])
    B, X = g.CreateVec(), g.CreateVec()
    B.set(b)
    its, rel, reason = g.Solve(A, B, X, rtol=1e-10, maxits=60, ksp_type="gmres", return_reason=True)
    x = X.get()
    assert reason == KSP_DIVERGED_ITS and its == 60
    assert np.all(np.isfinite(x))
    true = np.linalg.norm(b - M @ x) / np.linalg.norm(b)
    assert abs(rel - true) <= 1e-12 * true, (rel, true)


def _abi_solve(g, A, b_ptr, x_ptr, restart=30, rtol=1e-10, maxit=100, outputs=True):
    L = pb.load_cuda()
    its, rel, reason = C.c_int(-1), C.c_double(-1.0), C.c_int(99)
    args = (C.byref(its), C.byref(rel), C.byref(reason)) if outputs else (None, None, None)
    rc = L.petiga_cuda_solve_gmres(g.plan(), int(A.baij), C.c_void_p(A.device_ptr()), C.c_void_p(b_ptr), C.c_void_p(x_ptr), int(restart),
                                   C.c_double(rtol), C.c_double(1e-50), int(maxit), *args)
    return rc, its.value, rel.value, reason.value


def test_zero_rhs_and_argument_errors():
    g, A, dof = ch_jacobian(16, 1e7)
    B, X = g.CreateVec(), g.CreateVec()
    B.set(np.zeros(B.size))
    X.set(np.random.default_rng(2).standard_normal(X.size))             # a nonzero initial guess: b = 0 still gives x = 0
    rc, its, rel, reason = _abi_solve(g, A, B.device_ptr(), X.device_ptr())
    assert (rc, its, rel, reason) == (0, 0, 0.0, KSP_CONVERGED_ATOL)
    assert np.array_equal(X.get(), np.zeros(X.size))
    its, rel, reason = g.Solve(A, B, X, ksp_type="gmres", return_reason=True)
    assert (its, reason) == (0, KSP_CONVERGED_ATOL)
    # C ABI: b is x, restart < 1, maxit < 0, NULL outputs
    B.set(np.ones(B.size))
    assert _abi_solve(g, A, B.device_ptr(), B.device_ptr())[0] == 1
    assert _abi_solve(g, A, B.device_ptr(), X.device_ptr(), restart=0)[0] == 1
    assert _abi_solve(g, A, B.device_ptr(), X.device_ptr(), maxit=-1)[0] == 1
    assert _abi_solve(g, A, B.device_ptr(), X.device_ptr(), outputs=False)[0] == 1
    # host mirror
    with pytest.raises(pb.IGAError) as e:
        g.Solve(A, B, B, ksp_type="gmres")
    assert e.value.code == PETSC_ERR_ARG_IDN
    with pytest.raises(pb.IGAError) as e:
        g.Solve(A, B, X, ksp_type="gmres", restart=0)
    assert e.value.code == PETSC_ERR_ARG_OUTOFRANGE
    with pytest.raises(pb.IGAError) as e:
        g.Solve(A, B, X, ksp_type="bicg")
    assert e.value.code == PETSC_ERR_SUP and "bicg" in str(e.value)
    # BAIJ beyond bs 4 has no block product: PETSC_ERR_SUP, as for CG
    g5, A5, B5 = system(Case(2, dof=5, p=2, N=4), "MASS")
    with pytest.raises(pb.IGAError) as e:
        g5.Solve(A5, B5, g5.CreateVec(), ksp_type="gmres")
    assert e.value.code == PETSC_ERR_SUP


def test_restart_is_ignored_by_cg_and_cg_reports_a_reason():
    g, A, B = system(Case(2, p=2, N=8, bcv=[(d, s, 0, 1.0) for d in range(2) for s in range(2)]), "POISSON")
    X = g.CreateVec()
    its, rel, reason = g.Solve(A, B, X, rtol=1e-10, restart=5, return_reason=True)
    assert rel <= 1e-10 and reason == KSP_CONVERGED_RTOL
    its, rel, reason = g.Solve(A, B, X, rtol=1e-14, maxits=2, return_reason=True)
    assert its == 2 and reason == KSP_DIVERGED_ITS


def test_non_finite_values_stop_with_nanorinf():
    """An entry of 1e300 makes |A D^-1 v_0|^2 overflow in the first Arnoldi step: rc 0, DIVERGED_NANORINF, x the last finite
    iterate (the zero initial guess).  A NaN in b is caught before any iteration."""
    g, A, dof = ch_jacobian(16, 1e7)
    rp, ci = A.pattern()
    row = 40
    k = next(k for k in range(rp[row], rp[row + 1]) if ci[k] != row)
    big = C.c_double(1e300)
    L = pb.load_cuda()
    assert L.petiga_cuda_memcpy_h2d(C.c_void_p(A.device_ptr() + 8 * k), C.byref(big), C.c_size_t(8)) == 0
    B, X = g.CreateVec(), g.CreateVec()
    B.set(np.random.default_rng(1).standard_normal(B.size))
    its, rel, reason = g.Solve(A, B, X, ksp_type="gmres", return_reason=True)
    assert reason == KSP_DIVERGED_NANORINF and its == 1
    assert np.array_equal(X.get(), np.zeros(X.size)) and rel == 1.0
    b = np.ones(B.size); b[7] = np.nan
    B.set(b)
    its, rel, reason = g.Solve(A, B, X, ksp_type="gmres", return_reason=True)
    assert reason == KSP_DIVERGED_NANORINF and its == 0 and np.all(np.isfinite(X.get()))


def test_deterministic():
    g, A, dof = ch_jacobian(32, 1e7)
    b = np.random.default_rng(1).standard_normal(32 * 32)
    B, X1, X2 = g.CreateVec(), g.CreateVec(), g.CreateVec()
    B.set(b)
    r1 = g.Solve(A, B, X1, rtol=1e-10, ksp_type="gmres", return_reason=True)
    r2 = g.Solve(A, B, X2, rtol=1e-10, ksp_type="gmres", return_reason=True)
    assert r1 == r2
    assert X1.get().tobytes() == X2.get().tobytes()


def test_newton_backward_euler_step():
    """One backward-Euler step of CahnHilliard2D (shift a = 1e7, V = a (U - U0)): four Newton iterations with IFunction,
    IJacobian and GMRES on the device, and the same iterations with scipy's direct solve on the host."""
    N, a = 32, 1e7
    case = Case(2, p=2, N=N, C=1, periodic=True)
    g = case.product()
    g.SetForm("IFUNCTION", "CAHNHILLIARD2D", CH)
    g.SetForm("IJACOBIAN", "CAHNHILLIARD2D", CH)
    U0, _ = state_vectors(N * N)
    vU, vV, F, dU, J = g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateMat()

    def residual_and_jacobian(U):
        vU.set(U); vV.set(a * (U - U0))
        g.ComputeIFunction(a, vV, 0.0, vU, F)
        g.ComputeIJacobian(a, vV, 0.0, vU, J)
        return F.get()

    Ud, Uh = U0.copy(), U0.copy()
    norms = []
    for _ in range(4):
        f = residual_and_jacobian(Ud)
        norms.append(np.linalg.norm(f))
        its, rel, reason = g.Solve(J, F, dU, rtol=1e-10, ksp_type="gmres", return_reason=True)
        assert reason in (KSP_CONVERGED_RTOL, KSP_CONVERGED_ATOL)
        Ud = Ud - dU.get()
        fh = residual_and_jacobian(Uh)
        Uh = Uh - spla.spsolve(scipy_matrix(J, 1).tocsc(), fh)
        assert np.linalg.norm(Ud - Uh) <= 1e-8 * np.linalg.norm(Uh)
    norms.append(np.linalg.norm(residual_and_jacobian(Ud)))
    for k in range(4):
        # |F| falls at every iteration until it reaches the rounding level of the assembled residual
        assert norms[k + 1] < norms[k] or norms[k] <= 1e-10 * norms[0], norms
    assert norms[-1] <= 1e-8 * norms[0], norms


def test_multirank_gmres():
    import os
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29531", os.path.join(root, "tests", "multirank_gmres_check.py")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    print(out.stdout[-4000:])
    assert "GMRES MULTIRANK PASS" in out.stdout
