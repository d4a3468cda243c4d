"""Device memory of a plan: every buffer a plan sizes lazily (separable tables, pair-product tables, D' scratch, mapped-face areas,
compute_host staging, CG and GMRES workspaces, scalar partials, collocation tables) is freed when the IGA is destroyed, and a fix
table whose halo fails leaves nothing behind.  Free device memory is read with cudaMemGetInfo; the first round of each test loads
the kernels it launches (their code stays resident), so the comparisons are between rounds that launch the same kernels."""
import ctypes as C

import numpy as np
import pytest

import petiga_b200 as pb
from petiga_b200.cases import perturbed_identity
from tests.common import Case

pytestmark = pytest.mark.gpu


def _cudart():
    for name in ("libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
        try:
            return C.CDLL(name)
        except OSError:
            pass
    return None


_RT = _cudart()


def _device_count():
    n = C.c_int(0)
    return n.value if _RT is not None and _RT.cudaGetDeviceCount(C.byref(n)) == 0 else 0


needs_device = pytest.mark.skipif(_device_count() == 0, reason="needs a CUDA device")


def free_bytes():
    free, total = C.c_size_t(), C.c_size_t()
    assert _RT.cudaSetDevice(0) == 0 and _RT.cudaDeviceSynchronize() == 0
    assert _RT.cudaMemGetInfo(C.byref(free), C.byref(total)) == 0
    return free.value


def _galerkin_round():
    """one 3-D p = 3 IGA through every lazily sized buffer of a Galerkin plan, then destroyed"""
    N = 6
    case = Case(3, p=3, N=N, bcv=[(d, 0, 0, 1.0) for d in range(3)])
    g = case.product()
    g.SetForm("SYSTEM", "POISSON")
    A, B, x = g.CreateMat(), g.CreateVec(), g.CreateVec()
    for path, impl in ((2, -1), (1, 0), (1, 3)):    # separable tables, pair products of the v2 and of the v3 kernel
        g.SetOption("path", path)
        g.SetOption("quad_impl", impl)
        g.ComputeSystem(A, B)
        assert int(g.GetStat("last_path")) == path and (path == 2 or int(g.GetStat("last_impl")) == impl)
    g.Solve(A, B, x, rtol=1e-6)                     # CG workspace
    g.Solve(A, B, x, rtol=1e-6, ksp_type="gmres")   # GMRES workspace
    assert np.isfinite(g.ComputeErrorNorm(0, x, None)).all()   # compute_scalar partials
    # compute_host: values and rhs staging, then U and V staging
    L = pb.load_cuda()
    f = L.petiga_cuda_compute_host
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    vals, rhs = np.empty(A.nnz), np.empty(B.size)
    assert f(g.plan(), 2, 0, 0.0, None, 0.0, None, vals.ctypes.data, rhs.ctypes.data) == 0, L.petiga_cuda_last_error()
    U, V = np.full(B.size, 0.1), np.full(B.size, -0.2)
    g.SetOption("path", 0)
    g.SetOption("quad_impl", -1)
    g.SetForm("IFUNCTION", "BRATU", [2.0])
    vU, vV, F = g.CreateVec(), g.CreateVec(), g.CreateVec()
    vU.set(U); vV.set(V)
    g.ComputeIFunction(1.5, vV, 0.5, vU, F)        # hands the form to the plan
    assert f(g.plan(), 5, 0, 1.5, V.ctypes.data, 0.5, U.ctypes.data, None, rhs.ctypes.data) == 0, L.petiga_cuda_last_error()
    assert np.allclose(rhs, F.get(), rtol=1e-13, atol=1e-13)
    # mapped geometry with face loads: D' of the third-generation kernel and the BoundaryArea factors of the loaded faces
    g.SetGeometryArrays(perturbed_identity(3, 3, N, 0.05))
    for d in range(3):
        g.SetBoundaryLoad(d, 1, 0, 0.25 * (d + 1))
    g.SetForm("SYSTEM", "LAPLACE")
    g.SetOption("path", 1)
    g.SetOption("quad_impl", 3)
    g.ComputeSystem(A, B)
    assert int(g.GetStat("last_impl")) == 3
    for o in (A, B, x, vU, vV, F):
        o.destroy()
    g.Destroy()


def _collocation_round():
    """a collocation plan (state numbering, state halo buffers) through a Bratu Jacobian"""
    g = pb.IGA(2, 1)
    g.SetUseCollocation(True)
    for d in range(2):
        g.AxisInitUniform(d, 3, 8)
    g.SetUp()
    g.SetForm("JACOBIAN", "BRATU_COLLOCATION", (1.0,))
    U, J = g.CreateVec(), g.CreateMat()
    U.set(np.linspace(0.0, 0.5, U.size))
    g.ComputeJacobian(U, J)
    assert int(g.GetStat("last_path")) == 3
    U.destroy(); J.destroy()
    g.Destroy()


@needs_device
def test_lazy_buffers_freed_with_the_plan():
    free = []
    for _ in range(3):
        _galerkin_round()
        _collocation_round()
        free.append(free_bytes())
    assert free[1] == free[0] and free[2] == free[0], free


def _failed_fixtable_round():
    """rank 0 of a two-rank IGA without a communicator: the fix table's halo fails, so the assembly fails with an error"""
    g = Case(2, p=2, N=8, bcv=[(0, 0, 0, 1.0)]).product(rank=0, size=2)
    g.SetForm("SYSTEM", "POISSON")
    A, B, T = g.CreateMat(), g.CreateVec(), g.CreateVec()
    T.set(np.ones(T.size))
    g.SetFixTable(T)
    with pytest.raises(pb.IGAError):
        g.ComputeSystem(A, B)
    for o in (A, B, T):
        o.destroy()
    g.Destroy()


@needs_device
def test_failed_fixtable_leaves_nothing_behind():
    _failed_fixtable_round()
    before = free_bytes()
    _failed_fixtable_round()
    assert free_bytes() == before
