"""Bratu by collocation on the device (IGAComputeFunction/Jacobian/IFunction/IJacobian with BRATU_COLLOCATION): the state kernel
against tests/colloc_state_ref.py on identity, mapped and rational geometry in AIJ and BAIJ; bitwise repeatability; the lambda = 0
Jacobian against the Laplace collocation matrix; Newton solves with every piece on the device (2-D, and the 1-D exact-solution
rates); the kernel's ptxas budget; and the multi-rank check under torchrun."""
import os
import re

import numpy as np
import pytest

import petiga_b200 as pb
from oracle.oracle import read_iga_file
from tests.colloc_ref import Axis, Space
from tests.colloc_state_ref import bratu_1d_exact, jacobian, newton, operators, residual
from tests.common import rel_frobenius
from tests.geomutil import refine_annulus
from tests.test_host_collocation import CASES, make_iga

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_FACES = lambda dim, v: {(d, s): v for d in range(dim) for s in range(2)}   # noqa: E731
SLOTS = ("FUNCTION", "JACOBIAN", "IFUNCTION", "IJACOBIAN")


def _vec(g, arr):
    v = g.CreateVec()
    v.set(np.ascontiguousarray(arr, dtype=np.float64))
    return v


def _device_slots(g, lam, U, V, shift, values, baij):
    """all four slots on one collocation IGA -> {slot: F or (rowptr, colidx, values)}"""
    if baij:
        g.SetMatType("baij")
    for (d, s), v in (values or {}).items():
        g.SetBoundaryValue(d, s, 0, v)
    for slot in SLOTS:
        g.SetForm(slot, "BRATU_COLLOCATION", (lam,))
    Uv, Vv, F, J = _vec(g, U), _vec(g, V), g.CreateVec(), g.CreateMat()
    out = {}
    g.ComputeFunction(Uv, F)
    assert int(g.GetStat("last_path")) == 3          # PETIGA_PATH_COLLOCATION
    out["FUNCTION"] = F.get().copy()
    g.ComputeIFunction(shift, Vv, 0.25, Uv, F)
    out["IFUNCTION"] = F.get().copy()
    rp, ci = J.pattern()
    g.ComputeJacobian(Uv, J)
    out["JACOBIAN"] = (rp, ci, J.values().reshape(-1).copy())
    g.ComputeIJacobian(shift, Vv, 0.25, Uv, J)
    out["IJACOBIAN"] = (rp, ci, J.values().reshape(-1).copy())
    for o in (Uv, Vv, F, J):
        o.destroy()
    return out


def _compare(g, axes, X=None, W=None, values=None, baij=False, lam=1.3, shift=4.5):
    n = int(np.prod([a.nnp for a in axes]))
    rng = np.random.default_rng(n)
    U, V = rng.uniform(-0.4, 0.7, n), rng.uniform(-1.0, 1.0, n)
    got = _device_slots(g, lam, U, V, shift, values, baij)
    ops = operators(axes, X=X, W=W)
    rpr, cir = Space(axes).pattern(0)
    for slot in SLOTS:
        tr = slot.startswith("I")
        if slot.endswith("FUNCTION"):
            ref = residual(ops, U, lam, V=V if tr else None, values=values, axes=axes)
            assert rel_frobenius(got[slot], ref) <= 1e-12, slot
        else:
            Jr = jacobian(ops, U, lam, shift=shift if tr else 0.0, values=values, axes=axes)
            rp, ci, vals = got[slot]
            assert np.array_equal(rp, rpr) and np.array_equal(ci, cir) and np.array_equal(Jr.indices, cir)
            assert rel_frobenius(vals, Jr.data) <= 1e-12, slot


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s_%s" % (c[0], "".join(map(str, c[1])), c[3]))
def test_identity_geometry(case, baij):
    dim, ps, Ns, Cs = case
    g = make_iga(dim, ps, Ns, Cs)
    axes = [Axis(ps[d], g.AxisGetKnots(d)) for d in range(dim)]
    _compare(g, axes, values={(0, 0): 0.25, (dim - 1, 1): -0.5}, baij=baij)


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
def test_mapped_geometry(baij):
    axes_f, nsd, X, W, rational = read_iga_file(os.path.join(GOLD, "cube_perturbed.dat"))
    g = pb.IGA(3, 1)
    g.SetUseCollocation(True)
    for d, (p, U) in enumerate(axes_f):
        g.AxisSetKnots(d, p, U)
    g.SetGeometryArrays(X)
    g.SetUp()
    _compare(g, [Axis(p, U) for p, U in axes_f], X=X, values=ALL_FACES(3, 0.1), baij=baij)


class _ColIGA(pb.IGA):
    def __init__(self, dim, dof):
        super().__init__(dim, dof)
        self.SetUseCollocation(True)


@pytest.mark.gpu
@pytest.mark.parametrize("baij", [False, True], ids=["aij", "baij"])
@pytest.mark.parametrize("height", [None, (3, 0.5)], ids=["2d", "3d"])
def test_rational_geometry(height, baij):
    g, X, W = refine_annulus(_ColIGA, N=(5, 6), p=2, height=height)
    g.SetUp()
    dim = 2 if height is None else 3
    _compare(g, [Axis(2, g.AxisGetKnots(d)) for d in range(dim)], X=X, W=W, values={(0, 0): 1.0, (1, 1): 0.5}, baij=baij)


@pytest.mark.gpu
def test_bitwise_repeatable():
    g = make_iga(3, (3, 2, 4), (5, 6, 4), None)
    n = int(np.prod(g.info()["nnp"]))
    rng = np.random.default_rng(1)
    U, V = rng.uniform(-0.5, 0.5, n), rng.uniform(-1, 1, n)
    a = _device_slots(g, 2.0, U, V, 3.0, ALL_FACES(3, 0.0), False)
    b = _device_slots(g, 2.0, U, V, 3.0, None, False)    # same IGA, same boundary values (already set)
    for slot in SLOTS:
        x, y = (a[slot], b[slot]) if slot.endswith("FUNCTION") else (a[slot][2], b[slot][2])
        assert x.tobytes() == y.tobytes(), slot


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["identity", "rational"])
def test_lambda_zero_jacobian_is_the_laplace_matrix(kind):
    """lambda = 0: the Jacobian is -Lap R_b, the LAPLACE_COLLOCATION system matrix of the same IGA and boundary values"""
    mats = []
    for form in ("BRATU_COLLOCATION", "LAPLACE_COLLOCATION"):
        if kind == "identity":
            g = make_iga(3, (3, 3, 2), (6, 5, 7), None)
        else:
            g, X, W = refine_annulus(_ColIGA, N=(5, 6), p=2, height=(3, 0.5))
            g.SetUp()
        for (d, s), v in ALL_FACES(3, 0.5).items():
            g.SetBoundaryValue(d, s, 0, v)
        A = g.CreateMat()
        if form == "LAPLACE_COLLOCATION":
            B = g.CreateVec()
            g.SetForm("SYSTEM", form)
            g.ComputeSystem(A, B)
            B.destroy()
        else:
            n = int(np.prod(g.info()["nnp"]))
            Uv = _vec(g, np.random.default_rng(5).uniform(-1, 1, n))
            g.SetForm("JACOBIAN", form, (0.0,))
            g.ComputeJacobian(Uv, A)
            Uv.destroy()
        mats.append(A.values().reshape(-1).copy())
        A.destroy()
    J, K = mats
    assert np.abs(J - K).max() <= 1e-15 * np.abs(K).max()


def _newton_device(g, lam, tol, maxit=8):
    """Newton with IGAComputeFunction + IGAComputeJacobian + GMRES/Jacobi on the device; returns (U, |F| history)"""
    g.SetForm("FUNCTION", "BRATU_COLLOCATION", (lam,))
    g.SetForm("JACOBIAN", "BRATU_COLLOCATION", (lam,))
    U, F, dU, J = g.CreateVec(), g.CreateVec(), g.CreateVec(), g.CreateMat()
    U.set(np.zeros(U.size))
    hist = []
    for _ in range(maxit):
        g.ComputeFunction(U, F)
        hist.append(float(np.linalg.norm(F.get())))
        if hist[-1] <= tol:
            break
        g.ComputeJacobian(U, J)
        its, rn, reason = g.Solve(J, F, dU, rtol=1e-11, ksp_type="gmres", restart=100, maxits=20000, return_reason=True)
        assert reason == pb.iga.KSP_CONVERGED_RTOL, (its, rn, reason)
        U.set(U.get() - dU.get())
    u = U.get().copy()
    for o in (U, F, dU, J):
        o.destroy()
    return u, hist


@pytest.mark.gpu
def test_newton_2d_bratu():
    """lambda = 1, p = 3, N = 32, u = 0 on every face: |F| falls quadratically to 1e-10 within 6 steps, and the result is the
    scipy Newton solution of the reference system"""
    p, N = 3, 32
    g = make_iga(2, (p, p), (N, N), None)
    for (d, s), v in ALL_FACES(2, 0.0).items():
        g.SetBoundaryValue(d, s, 0, v)
    u, hist = _newton_device(g, 1.0, 1e-10)
    assert hist[-1] <= 1e-10 and len(hist) - 1 <= 6, hist
    for k in range(1, len(hist) - 1):     # quadratic: each step at least squares the relative residual (up to a constant)
        assert hist[k + 1] <= 10 * hist[k] ** 2 / hist[0] or hist[k + 1] <= 1e-10, hist
    axes = [Axis(p, g.AxisGetKnots(d)) for d in range(2)]
    ur, _ = newton(operators(axes), 1.0, ALL_FACES(2, 0.0), axes)
    assert np.abs(u - ur).max() <= 1e-9 * np.abs(ur).max()


@pytest.mark.gpu
def test_newton_1d_exact_solution_rates():
    """u'' + e^u = 0 on (0, 1) by device Newton: L2 rates 2, 2 and about 4 for p = 2, 3, 4 (N = 16 -> 32 -> 64)"""
    from scipy.interpolate import BSpline
    th, exact = bratu_1d_exact(1.0)
    xs = np.linspace(0, 1, 4001)
    for p, want in ((2, 1.9), (3, 1.9), (4, 3.8)):
        errs = []
        for N in (16, 32, 64):
            g = make_iga(1, (p,), (N,), None)
            g.SetBoundaryValue(0, 0, 0, 0.0)
            g.SetBoundaryValue(0, 1, 0, 0.0)
            u, hist = _newton_device(g, 1.0, 1e-10)
            assert hist[-1] <= 1e-10, hist
            errs.append(np.sqrt(np.mean((BSpline(np.array(g.AxisGetKnots(0)), u, p)(xs) - exact(xs)) ** 2)))
        rates = np.log2(np.array(errs[:-1]) / np.array(errs[1:]))
        assert np.all(rates >= want), (p, errs, rates)


def test_colloc_state_kernel_register_budget():
    """ptxas -v of the in-tree build: no stack frame (exp() included), no spills, and the CUDA 12.9 counts as caps"""
    path = os.path.join(pb.lib_dir(), "pc_colloc.ptxas.log")
    if not os.path.exists(path):
        pytest.skip("library not built in-tree")
    txt = open(path).read()
    budget = {(1, 0): 48, (2, 0): 56, (3, 0): 60, (1, 1): 78, (2, 1): 98, (3, 1): 143}
    for (dim, geo), cap in budget.items():
        sym = "colloc_state_kernelILi%dELb%dE" % (dim, geo)
        m = re.search(r"Function properties for [^\n]*%s[^\n]*\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                      r"[^\n]*Used (\d+) registers" % re.escape(sym), txt)
        assert m, sym
        stack, st, ld, regs = map(int, m.groups())
        assert stack == 0 and st == 0 and ld == 0, (sym, stack, st, ld)
        assert regs <= cap, (sym, regs)


@pytest.mark.gpu
def test_multirank_collocation_state():
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tests", "multirank_colloc_state_check.py")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    print(out.stdout[-4000:])
    assert "COLLOCATION STATE MULTIRANK PASS" in out.stdout
