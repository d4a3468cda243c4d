"""ctypes binding of libpetiga_host.so: the reference's IGA API names, one method per C function."""
import ctypes as C
import os

import numpy as np

from .build import lib_dir

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_host = None
_cuda = None

FORMS = {
    # name -> {slot name: exported sentinel symbol}
    "POISSON": {"SYSTEM": "IGADeviceForm_Poisson_System", "FUNCTION": "IGADeviceForm_Poisson_Function",
                "JACOBIAN": "IGADeviceForm_Poisson_Jacobian"},
    "LAPLACE": {"SYSTEM": "IGADeviceForm_Laplace_System"},
    "L2PROJECTION": {"SYSTEM": "IGADeviceForm_L2Projection_System"},
    "BOUNDARYINTEGRAL": {"SYSTEM": "IGADeviceForm_BoundaryIntegral_System"},
    "NEUMANN": {"SYSTEM": "IGADeviceForm_Neumann_SystemGalerkin"},
    "CONVTEST": {"SYSTEM": "IGADeviceForm_ConvTest_Galerkin"},
    # collocation forms (SetUseCollocation(True)): the strong form at the Greville points
    "LAPLACE_COLLOCATION": {"SYSTEM": "IGADeviceForm_Laplace_SystemCollocation"},
    "CONVTEST_COLLOCATION": {"SYSTEM": "IGADeviceForm_ConvTest_Collocation"},
    "MASS": {"SYSTEM": "IGADeviceForm_Mass_System", "MATRIX": "IGADeviceForm_Mass_Matrix", "VECTOR": "IGADeviceForm_Mass_Vector"},
    "ELASTICITY3D": {"SYSTEM": "IGADeviceForm_Elasticity3D_System"},
    "ELASTICITY": {"SYSTEM": "IGADeviceForm_Elasticity_System"},
    "CAHNHILLIARD2D": {"IFUNCTION": "IGADeviceForm_CahnHilliard2D_Residual", "IJACOBIAN": "IGADeviceForm_CahnHilliard2D_Tangent"},
    "CAHNHILLIARD3D": {"IFUNCTION": "IGADeviceForm_CahnHilliard3D_Residual", "IJACOBIAN": "IGADeviceForm_CahnHilliard3D_Tangent"},
    "BRATU": {"FUNCTION": "IGADeviceForm_Bratu_Function", "JACOBIAN": "IGADeviceForm_Bratu_Jacobian",
              "IFUNCTION": "IGADeviceForm_Bratu_IFunction", "IJACOBIAN": "IGADeviceForm_Bratu_IJacobian",
              "RHSFUNCTION": "IGADeviceForm_Bratu_RHSFunction", "RHSJACOBIAN": "IGADeviceForm_Bratu_RHSJacobian"},
    "NITSCHE": {"SYSTEM": "IGADeviceForm_Nitsche_System"},
    "SNES2D": {"FUNCTION": "IGADeviceForm_SNES2D_Function", "JACOBIAN": "IGADeviceForm_SNES2D_Jacobian"},
    "PATTERNFORMATION": {"IEFUNCTION": "IGADeviceForm_PatternFormation_IEFunction", "IEJACOBIAN": "IGADeviceForm_PatternFormation_IEJacobian"},
    "ELASTICROD": {"I2FUNCTION": "IGADeviceForm_ElasticRod_I2Function", "I2JACOBIAN": "IGADeviceForm_ElasticRod_I2Jacobian"},
}
_SETTERS = {"VECTOR": "IGASetFormVector", "MATRIX": "IGASetFormMatrix", "SYSTEM": "IGASetFormSystem",
            "FUNCTION": "IGASetFormFunction", "JACOBIAN": "IGASetFormJacobian", "IFUNCTION": "IGASetFormIFunction",
            "IJACOBIAN": "IGASetFormIJacobian", "IEFUNCTION": "IGASetFormIEFunction", "IEJACOBIAN": "IGASetFormIEJacobian",
            "RHSFUNCTION": "IGASetFormRHSFunction", "RHSJACOBIAN": "IGASetFormRHSJacobian", "I2FUNCTION": "IGASetFormI2Function",
            "I2JACOBIAN": "IGASetFormI2Jacobian"}


# KSPConvergedReason values (PETSc's; include/petiga_host.h)
KSP_CONVERGED_ITERATING, KSP_CONVERGED_RTOL, KSP_CONVERGED_ATOL = 0, 2, 3
KSP_DIVERGED_ITS, KSP_DIVERGED_BREAKDOWN, KSP_DIVERGED_NANORINF = -3, -5, -9


class IGAComm(C.Structure):
    _fields_ = [("rank", C.c_int), ("size", C.c_int), ("nccl", C.c_void_p), ("device", C.c_int)]


class IGAError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("PetscErrorCode %d: %s" % (code, msg))
        self.code = code


def load_cuda():
    """libpetiga_cuda.so (the product).  Raises if it has not been built -- there is no fallback."""
    global _cuda
    if _cuda is None:
        path = os.path.join(lib_dir(), "libpetiga_cuda.so")
        if not os.path.exists(path):
            raise RuntimeError("libpetiga_cuda.so not built (run __graft_entry__.build()); petiga_b200 has no CPU fallback")
        _cuda = C.CDLL(path, mode=C.RTLD_GLOBAL)
        _cuda.petiga_cuda_strerror.restype = C.c_char_p
        _cuda.petiga_cuda_last_error.restype = C.c_char_p
    return _cuda


def load_host():
    global _host
    if _host is None:
        load_cuda()
        path = os.path.join(lib_dir(), "libpetiga_host.so")
        if not os.path.exists(path):
            raise RuntimeError("libpetiga_host.so not built (run __graft_entry__.build())")
        _host = C.CDLL(path)
        _host.IGAGetLastErrorMessage.restype = C.c_char_p
        _host.IGAGetLayout.restype = C.c_void_p
        _host.IGAGetLayout.argtypes = [C.c_void_p]
    return _host


def _chk(rc):
    if rc:
        raise IGAError(rc, load_host().IGAGetLastErrorMessage().decode())


def iga_partition(size, rank, dim, N):
    H = load_host()
    Na = (C.c_int * 3)(*(list(N) + [1, 1, 1])[:3])
    n = (C.c_int * 3)(-1, -1, -1)
    i = (C.c_int * 3)(0, 0, 0)
    _chk(H.IGA_Partition(size, rank, dim, Na, n, i))
    return list(n)[:dim], list(i)[:dim]


def _vp(handle):
    """Handles cross ctypes as c_void_p objects: a bare Python int is converted to a 32-bit C int and would truncate a
    64-bit pointer (ADVICE r1: it only worked while malloc returned addresses below 4 GB)."""
    if isinstance(handle, C.c_void_p):
        return handle
    return C.c_void_p(handle)


class Vec:
    def __init__(self, iga, handle):
        self.iga, self.h = iga, _vp(handle)

    @property
    def size(self):
        n = C.c_int()
        _chk(load_host().VecGetLocalSize(self.h, C.byref(n)))
        return n.value

    def get(self):
        out = np.empty(self.size)
        _chk(load_host().VecGetArrayHost(self.h, out.ctypes.data_as(_dp)))
        return out

    def set(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float64).reshape(-1)
        assert arr.size == self.size
        _chk(load_host().VecSetArrayHost(self.h, arr.ctypes.data_as(_dp)))

    def device_ptr(self):
        p = C.c_void_p()
        _chk(load_host().VecGetArrayDevice(self.h, C.byref(p)))
        return p.value

    def destroy(self):
        if self.h:
            load_host().VecDestroy(C.byref(self.h))
            self.h = C.c_void_p()


class Mat:
    def __init__(self, iga, handle):
        self.iga, self.h = iga, _vp(handle)
        n, nnz, bs, baij = C.c_int(), C.c_int64(), C.c_int(), C.c_int()
        _chk(load_host().MatGetSizesIGA(self.h, C.byref(n), C.byref(nnz), C.byref(bs), C.byref(baij)))
        self.nrows_scalar, self.nnz, self.bs, self.baij = n.value, nnz.value, bs.value, bool(baij.value)
        self.nrows = self.nrows_scalar // self.bs if self.baij else self.nrows_scalar

    def pattern(self):
        rp = np.empty(self.nrows + 1, dtype=np.int32)
        ci = np.empty(self.nnz, dtype=np.int32)
        _chk(load_host().MatGetCSRHost(self.h, rp.ctypes.data_as(_ip), ci.ctypes.data_as(_ip), None))
        return rp, ci

    def values(self):
        """AIJ: [nnz] scalars; BAIJ: [nnz_blocks, bs, bs] with PETSc's column-major block storage undone
        (returned as row-major blocks [i][j])."""
        n = self.nnz * self.bs * self.bs if self.baij else self.nnz
        v = np.empty(n)
        _chk(load_host().MatGetCSRHost(self.h, None, None, v.ctypes.data_as(_dp)))
        if self.baij:
            return v.reshape(self.nnz, self.bs, self.bs).transpose(0, 2, 1).copy()
        return v

    def device_ptr(self):
        p = C.c_void_p()
        _chk(load_host().MatGetValuesDevice(self.h, C.byref(p)))
        return p.value

    def destroy(self):
        if self.h:
            load_host().MatDestroy(C.byref(self.h))
            self.h = C.c_void_p()


class IGA:
    """Thin object wrapper; method names are the reference's C function names minus the IGA prefix."""

    def __init__(self, dim=None, dof=None, rank=0, size=1, nccl=None, device=0):
        self.H = load_host()
        self.h = C.c_void_p()
        self.dim, self.dof = dim, dof
        comm = IGAComm(rank, size, nccl, device)
        _chk(self.H.IGACreate(comm, C.byref(self.h)))
        self._keep = []
        if dim is not None:
            self.SetDim(dim)
        if dof is not None:
            self.SetDof(dof)

    def __del__(self):
        try:
            self.Destroy()
        except Exception:
            pass

    def Destroy(self):
        if self.h:
            self.H.IGADestroy(C.byref(self.h))
            self.h = C.c_void_p()

    def SetDim(self, dim):
        _chk(self.H.IGASetDim(self.h, dim)); self.dim = dim

    def SetDof(self, dof):
        _chk(self.H.IGASetDof(self.h, dof)); self.dof = dof

    def SetOrder(self, order):
        _chk(self.H.IGASetOrder(self.h, order))

    def SetProcessors(self, i, n):
        _chk(self.H.IGASetProcessors(self.h, i, n))

    def SetRuleSize(self, i, q):
        _chk(self.H.IGASetRuleSize(self.h, i, q))

    def SetMatType(self, t):
        _chk(self.H.IGASetMatType(self.h, t.encode()))

    def SetUseCollocation(self, flag=True):
        """IGASetUseCollocation: assemble by collocation at the Greville points instead of Galerkin (before SetUp)."""
        _chk(self.H.IGASetUseCollocation(self.h, int(bool(flag))))

    def GetUseCollocation(self):
        f = C.c_int()
        _chk(self.H.IGAGetUseCollocation(self.h, C.byref(f)))
        return bool(f.value)

    def _axis(self, i):
        ax = C.c_void_p()
        _chk(self.H.IGAGetAxis(self.h, i, C.byref(ax)))
        return ax

    def AxisInitUniform(self, i, p, N, Ui=0.0, Uf=1.0, C_=-1, periodic=False):
        ax = self._axis(i)
        _chk(self.H.IGAAxisSetPeriodic(ax, int(periodic)))
        _chk(self.H.IGAAxisSetDegree(ax, p))
        _chk(self.H.IGAAxisInitUniform(ax, N, C.c_double(Ui), C.c_double(Uf), C_))

    def AxisSetKnots(self, i, p, U, periodic=False):
        ax = self._axis(i)
        U = np.ascontiguousarray(U, dtype=np.float64)
        _chk(self.H.IGAAxisSetPeriodic(ax, int(periodic)))
        _chk(self.H.IGAAxisSetDegree(ax, p))
        _chk(self.H.IGAAxisSetKnots(ax, len(U) - 1, U.ctypes.data_as(_dp)))

    def AxisInitBreaks(self, i, p, breaks, C_=-1, periodic=False):
        ax = self._axis(i)
        u = np.ascontiguousarray(breaks, dtype=np.float64)
        _chk(self.H.IGAAxisSetPeriodic(ax, int(periodic)))
        _chk(self.H.IGAAxisSetDegree(ax, p))
        _chk(self.H.IGAAxisInitBreaks(ax, len(u), u.ctypes.data_as(_dp), C_))

    def AxisGetKnots(self, i):
        ax = self._axis(i)
        m, U = C.c_int(), _dp()
        _chk(self.H.IGAAxisGetKnots(ax, C.byref(m), C.byref(U)))
        return np.ctypeslib.as_array(U, shape=(m.value + 1,)).copy()

    def AxisGetSpans(self, i):
        ax = self._axis(i)
        n, sp = C.c_int(), _ip()
        _chk(self.H.IGAAxisGetSpans(ax, C.byref(n), C.byref(sp)))
        return np.ctypeslib.as_array(sp, shape=(n.value,)).copy()

    # oracle-compatible aliases so that fixtures can build either object
    def axis_uniform(self, axis, p, N, Ui=0.0, Uf=1.0, C=-1, periodic=False):
        self.AxisInitUniform(axis, p, N, Ui, Uf, C, periodic)

    def axis_knots(self, axis, p, U, periodic=False):
        self.AxisSetKnots(axis, p, U, periodic)

    def geometry(self, X, W=None):
        self.SetGeometryArrays(X, W)

    def SetGeometryArrays(self, X, W=None):
        X = np.ascontiguousarray(X, dtype=np.float64)
        Wp = None
        if W is not None:
            W = np.ascontiguousarray(W, dtype=np.float64)
            Wp = W.ctypes.data_as(_dp)
        _chk(self.H.IGASetGeometryArrays(self.h, X.shape[-1], X.ctypes.data_as(_dp), Wp))

    def SetUp(self):
        _chk(self.H.IGASetUp(self.h))

    def SetBoundaryValue(self, axis, side, field, value):
        _chk(self.H.IGASetBoundaryValue(self.h, axis, side, field, C.c_double(value)))

    def SetBoundaryLoad(self, axis, side, field, value):
        _chk(self.H.IGASetBoundaryLoad(self.h, axis, side, field, C.c_double(value)))

    def SetBoundaryForm(self, axis, side, flag=True):
        _chk(self.H.IGASetBoundaryForm(self.h, axis, side, int(bool(flag))))

    def SetFixTable(self, vec):
        _chk(self.H.IGASetFixTable(self.h, vec.h if vec is not None else None))

    def SetForm(self, slot, form, params=()):
        """IGASetForm<slot>(iga, IGADeviceForm_<form>_<slot>, &ctx)"""
        sym = FORMS[form][slot]
        fn = C.cast(getattr(self.H, sym), C.c_void_p)
        ctx = (C.c_double * max(1, len(params)))(*params)
        if form == "PATTERNFORMATION" and len(params):      # the demo's AppCtx starts with a PetscBool (demo/PatternFormation.c:14-24)
            C.cast(ctx, C.POINTER(C.c_int))[0] = int(params[0] != 0)
            C.cast(ctx, C.POINTER(C.c_int))[1] = 0
        self._keep.append(ctx)
        _chk(getattr(self.H, _SETTERS[slot])(self.h, fn, C.cast(ctx, C.c_void_p) if len(params) else None))

    def SetFormRaw(self, slot, fnptr):
        _chk(getattr(self.H, _SETTERS[slot])(self.h, fnptr, None))

    def CreateMat(self):
        m = C.c_void_p()
        _chk(self.H.IGACreateMat(self.h, C.byref(m)))
        return Mat(self, m)

    def CreateVec(self):
        v = C.c_void_p()
        _chk(self.H.IGACreateVec(self.h, C.byref(v)))
        return Vec(self, v)

    def ComputeVector(self, B):
        _chk(self.H.IGAComputeVector(self.h, B.h))

    def ComputeMatrix(self, A):
        _chk(self.H.IGAComputeMatrix(self.h, A.h))

    def ComputeSystem(self, A, B):
        _chk(self.H.IGAComputeSystem(self.h, A.h, B.h))

    def ComputeFunction(self, U, F):
        _chk(self.H.IGAComputeFunction(self.h, U.h, F.h))

    def ComputeJacobian(self, U, J):
        _chk(self.H.IGAComputeJacobian(self.h, U.h, J.h))

    def ComputeIFunction(self, a, V, t, U, F):
        _chk(self.H.IGAComputeIFunction(self.h, C.c_double(a), V.h, C.c_double(t), U.h, F.h))

    def ComputeIJacobian(self, a, V, t, U, J):
        _chk(self.H.IGAComputeIJacobian(self.h, C.c_double(a), V.h, C.c_double(t), U.h, J.h))

    def ComputeIEFunction(self, a, V, t, U, t0, U0, F):
        _chk(self.H.IGAComputeIEFunction(self.h, C.c_double(a), V.h, C.c_double(t), U.h, C.c_double(t0), U0.h, F.h))

    def ComputeIEJacobian(self, a, V, t, U, t0, U0, J):
        _chk(self.H.IGAComputeIEJacobian(self.h, C.c_double(a), V.h, C.c_double(t), U.h, C.c_double(t0), U0.h, J.h))

    def ComputeRHSFunction(self, t, U, F):
        _chk(self.H.IGAComputeRHSFunction(self.h, C.c_double(t), U.h, F.h))

    def ComputeRHSJacobian(self, t, U, J):
        _chk(self.H.IGAComputeRHSJacobian(self.h, C.c_double(t), U.h, J.h))

    def ComputeI2Function(self, a, A, v, V, t, U, F):
        _chk(self.H.IGAComputeI2Function(self.h, C.c_double(a), A.h, C.c_double(v), V.h, C.c_double(t), U.h, F.h))

    def ComputeI2Jacobian(self, a, A, v, V, t, U, J):
        _chk(self.H.IGAComputeI2Jacobian(self.h, C.c_double(a), A.h, C.c_double(v), V.h, C.c_double(t), U.h, J.h))

    def GetOwnedNaturalIndices(self):
        inf = self.info()
        n = int(np.prod(inf["node_lwidth"]))
        out = np.empty(n, dtype=np.int32)
        _chk(self.H.IGAGetOwnedNaturalIndices(self.h, out.ctypes.data_as(_ip)))
        return out

    def Synchronize(self):
        _chk(self.H.IGASynchronize(self.h))

    # ---- files (src/petigaio.c) ----
    def Read(self, filename):
        _chk(self.H.IGARead(self.h, filename.encode()))
        d = C.c_int()
        _chk(self.H.IGAGetDim(self.h, C.byref(d)))
        self.dim = d.value

    def Write(self, filename):
        _chk(self.H.IGAWrite(self.h, filename.encode()))

    def ReadVec(self, vec, filename):
        _chk(self.H.IGAReadVec(self.h, vec.h, filename.encode()))

    def WriteVec(self, vec, filename):
        _chk(self.H.IGAWriteVec(self.h, vec.h, filename.encode()))

    def GetGeometryArrays(self):
        sizes, nsd, rat = (C.c_int * 3)(), C.c_int(), C.c_int()
        _chk(self.H.IGAGetGeometryArrays(self.h, sizes, C.byref(nsd), C.byref(rat), None, None))
        n = sizes[0] * sizes[1] * sizes[2]
        if nsd.value == 0:
            return list(sizes), 0, False, None, None
        X, W = np.zeros(n * nsd.value), np.zeros(n)
        _chk(self.H.IGAGetGeometryArrays(self.h, sizes, C.byref(nsd), C.byref(rat), X.ctypes.data_as(_dp), W.ctypes.data_as(_dp)))
        return list(sizes), nsd.value, bool(rat.value), X.reshape(n, nsd.value), W

    def ComputeScalar(self, U, n, scalar="CahnHilliard2D_Stats", ctx=()):
        """IGAComputeScalar (src/petigacomp.c:35-96) with a device Scalar sentinel; ctx = the demo's AppCtx reals."""
        fn = C.cast(getattr(self.H, "IGADeviceScalar_" + scalar), C.c_void_p)
        S = (C.c_double * n)()
        cx = (C.c_double * max(1, len(ctx)))(*ctx)
        _chk(self.H.IGAComputeScalar(self.h, (U.h if U is not None else None), n, S, fn, C.cast(cx, C.c_void_p)))
        return np.array(list(S))

    def ComputeErrorNorm(self, k, U=None, exact=None, ctx=()):
        """IGAComputeErrorNorm (src/petigacomp.c:155-186); exact: None | "ErrNormTest" | "L2Projection"."""
        fn = C.cast(getattr(self.H, "IGADeviceExact_" + exact), C.c_void_p) if exact else C.c_void_p(None)
        out = (C.c_double * self.dof)()
        cx = (C.c_double * max(1, len(ctx)))(*ctx)
        _chk(self.H.IGAComputeErrorNorm(self.h, k, (U.h if U is not None else None), fn, out, C.cast(cx, C.c_void_p)))
        return np.array(list(out))

    # ---- introspection ----
    def info(self):
        buf = (C.c_int * 46)()
        _chk(self.H.IGAGetInfoArray(self.h, buf))
        keys = ["p", "m", "nnp", "nel", "nqp", "nen", "proc_size", "proc_rank", "elem_start", "elem_width",
                "node_lstart", "node_lwidth", "node_gstart", "node_gwidth", "geom_size"]
        out = {"order": buf[0]}
        for k, key in enumerate(keys):
            out[key] = [buf[1 + 15 * i + k] for i in range(3)]
        return out

    def tables(self, axis):
        inf = self.info()
        nel, nqp, nen, m = inf["nel"][axis], inf["nqp"][axis], inf["nen"][axis], inf["m"][axis]

        def get(which, n):
            out = np.empty(n)
            _chk(self.H.IGAGetBasisTable(self.h, axis, which, out.ctypes.data_as(_dp)))
            return out
        return dict(value=get(0, nel * nqp * nen * 5).reshape(nel, nqp, nen, 5), weight=get(1, nel * nqp).reshape(nel, nqp),
                    point=get(2, nel * nqp).reshape(nel, nqp), detJac=get(3, nel), U=get(4, m + 1))

    def lgmap(self):
        n = int(np.prod(self.info()["node_gwidth"]))
        out = np.empty(n, dtype=np.int32)
        _chk(self.H.IGAGetLGMapHost(self.h, out.ctypes.data_as(_ip)))
        return out

    def layout(self):
        return Layout(self.H.IGAGetLayout(self.h))

    def SetStream(self, stream_ptr):
        _chk(self.H.IGASetStream(self.h, C.c_void_p(stream_ptr)))

    def MatMult(self, A, x, y):
        _chk(self.H.MatMult(A.h, x.h, y.h))

    def Solve(self, A, b, x, rtol=1e-8, atol=1e-50, maxits=10000, ksp_type="cg", restart=30, return_reason=False):
        """IGACreateKSP + KSPSetType + KSPSetOperators + KSPSetTolerances + KSPSolve (demo/Poisson3D.c:73-83) on the device with
        the Jacobi preconditioner: ksp_type "cg" (symmetric positive definite A) or "gmres" (GMRES(restart), any A with a nonzero
        diagonal).  Returns (iterations, |b - A x| / |b|), or (iterations, |b - A x| / |b|, KSPConvergedReason value) with
        return_reason=True."""
        ksp = C.c_void_p()
        _chk(self.H.IGACreateKSP(self.h, C.byref(ksp)))
        try:
            if ksp_type != "cg":
                _chk(self.H.KSPSetType(ksp, C.c_char_p(ksp_type.encode())))
            if restart != 30:
                _chk(self.H.KSPGMRESSetRestart(ksp, int(restart)))
            _chk(self.H.KSPSetOperators(ksp, A.h, A.h))
            _chk(self.H.KSPSetTolerances(ksp, C.c_double(rtol), C.c_double(atol), C.c_double(1e5), int(maxits)))
            _chk(self.H.KSPSolve(ksp, b.h, x.h))
            its, rn, reason = C.c_int(), C.c_double(), C.c_int()
            _chk(self.H.KSPGetIterationNumber(ksp, C.byref(its)))
            _chk(self.H.KSPGetResidualNorm(ksp, C.byref(rn)))
            if return_reason:
                _chk(self.H.KSPGetConvergedReason(ksp, C.byref(reason)))
                return its.value, rn.value, reason.value
            return its.value, rn.value
        finally:
            self.H.KSPDestroy(C.byref(ksp))

    def SetOption(self, name, value):
        _chk(self.H.IGASetOption(self.h, name.encode(), C.c_double(value)))

    def GetStat(self, name):
        v = C.c_double()
        _chk(self.H.IGAGetStat(self.h, name.encode(), C.byref(v)))
        return v.value

    def plan(self):
        p = C.c_void_p()
        _chk(self.H.IGAGetPlan(self.h, C.byref(p)))
        return p


class Layout:
    """Host-only layout object (petiga_layout_* of include/petiga_cuda.h); needs no GPU."""

    def __init__(self, handle):
        self.h = C.c_void_p(handle)
        self.L = load_cuda()

    def sizes(self):
        a, b, c, d, e = C.c_int(), C.c_int(), C.c_int(), C.c_int64(), C.c_int64()
        assert self.L.petiga_layout_sizes(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)) == 0
        return dict(nown=a.value, nghostbox=b.value, nloc=c.value, nnz_own=d.value, nnz_loc=e.value)

    def pattern(self, block, dof):
        s = self.sizes()
        bs = 1 if block else dof
        rp = np.empty(s["nown"] * bs + 1, dtype=np.int32)
        ci = np.empty(s["nnz_own"] * bs * bs, dtype=np.int32)
        rc = self.L.petiga_layout_pattern(self.h, int(block), rp.ctypes.data_as(_ip), ci.ctypes.data_as(_ip))
        assert rc == 0, rc
        return rp, ci

    def localrow(self):
        out = np.empty(self.sizes()["nghostbox"], dtype=np.int32)
        assert self.L.petiga_layout_localrow(self.h, out.ctypes.data_as(_ip)) == 0
        return out

    def lgmap(self):
        out = np.empty(self.sizes()["nghostbox"], dtype=np.int32)
        assert self.L.petiga_layout_lgmap(self.h, out.ctypes.data_as(_ip)) == 0
        return out

    def rowbase(self):
        out = np.empty(self.sizes()["nloc"] + 1, dtype=np.int64)
        assert self.L.petiga_layout_rowbase(self.h, out.ctypes.data_as(C.POINTER(C.c_int64))) == 0
        return out

    def position(self, ga, hb):
        g = (C.c_int * 3)(*ga)
        h = (C.c_int * 3)(*hb)
        pos = C.c_int64()
        rc = self.L.petiga_layout_position(self.h, g, h, C.byref(pos))
        assert rc == 0, rc
        return pos.value

    def exchange(self, kind):
        n = C.c_int()
        assert self.L.petiga_layout_exchange(self.h, kind, C.byref(n), None, 0) == 0
        out = np.zeros((max(n.value, 1), 4), dtype=np.int64)
        assert self.L.petiga_layout_exchange(self.h, kind, C.byref(n), out.ctypes.data_as(C.POINTER(C.c_int64)), n.value) == 0
        return out[:n.value]

    def recv_rows(self, peer_index, n):
        rows = np.empty(n, dtype=np.int32)
        assert self.L.petiga_layout_recv_rows(self.h, peer_index, rows.ctypes.data_as(_ip), n) == 0
        return rows
