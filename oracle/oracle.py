"""ctypes front-end of the CPU oracle (TEST INFRASTRUCTURE ONLY -- see oracle/petiga_oracle.c).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
The product package petiga_b200 never does.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

SLOT = dict(VECTOR=0, MATRIX=1, SYSTEM=2, FUNCTION=3, JACOBIAN=4, IFUNCTION=5, IJACOBIAN=6,
            IEFUNCTION=7, IEJACOBIAN=8, RHSFUNCTION=9, RHSJACOBIAN=10, I2FUNCTION=11, I2JACOBIAN=12)
MAT_SLOTS = ("MATRIX", "SYSTEM", "JACOBIAN", "IJACOBIAN", "IEJACOBIAN", "RHSJACOBIAN", "I2JACOBIAN")
VEC_SLOTS = ("VECTOR", "SYSTEM", "FUNCTION", "IFUNCTION", "IEFUNCTION", "RHSFUNCTION", "I2FUNCTION")
FORM = dict(POISSON=0, LAPLACE=1, L2PROJECTION=2, ELASTICITY3D=3, ELASTICITY=4, CAHNHILLIARD2D=5, BRATU=6, MASS=7,
            BOUNDARYINTEGRAL=8, NEUMANN=9, CAHNHILLIARD3D=10, CONVTEST=11, SNES2D=12, PATTERNFORMATION=13, ELASTICROD=14, NITSCHE=15)
SCALAR = dict(ERRNORM=0, CH_STATS=1)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def build(native=False):
    """Compile the oracle with gcc (a few seconds).  The portable library sits beside the source, mtime-guarded, so calling
    this every time is cheap.  native=True adds -march=native (CPU-baseline timing): that binary is only valid on the CPU it
    was built for and the tree may be read-only where the benchmark runs, so it goes to a fresh temporary directory."""
    src = os.path.join(_HERE, "petiga_oracle.c")
    hdr = os.path.join(_HERE, "gauss_tables.h")
    if native:
        tmpdir = tempfile.mkdtemp(prefix="petiga_oracle_")
        out = os.path.join(tmpdir, "libpetiga_oracle_native.so")
        try:
            subprocess.check_call(["gcc", "-O2", "-march=native", "-fPIC", "-shared", "-o", out, src, "-lm"], cwd=_HERE)
        except Exception:
            shutil.rmtree(tmpdir)
            raise
        return out
    out = os.path.join(_HERE, "libpetiga_oracle.so")
    if os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(src), os.path.getmtime(hdr)):
        return out
    tmp = out + ".tmp%d" % os.getpid()      # several ranks / xdist workers may build at once: write aside, then rename
    cmd = ["gcc", "-O2", "-march=x86-64-v2", "-fPIC", "-shared", "-o", tmp, src, "-lm"]
    subprocess.check_call(cmd, cwd=_HERE)
    os.replace(tmp, out)
    return out


_NATIVE = None


def lib(native=False):
    global _LIB, _NATIVE
    if native and _NATIVE is not None:
        return _NATIVE
    if _LIB is not None and not native:
        return _LIB
    try:
        path = build(native)     # always: a stale binary must never be compared against (ADVICE r1)
    except Exception:
        if native:
            return lib(False)
        raise
    L = C.CDLL(path)
    if native:
        shutil.rmtree(os.path.dirname(path))     # the loaded mapping outlives the file: nothing is left behind
    L.oiga_create.restype = C.c_void_p
    L.oiga_create.argtypes = [C.c_int, C.c_int]
    L.oiga_destroy.argtypes = [C.c_void_p]
    L.oiga_axis_init_uniform.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int]
    L.oiga_axis_set_knots.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, C.c_int]
    L.oiga_set_rule_size.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.oiga_set_order.argtypes = [C.c_void_p, C.c_int]
    L.oiga_set_boundary_value.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double]
    L.oiga_set_boundary_load.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double]
    L.oiga_set_boundary_form.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.oiga_tabulate_boundary.argtypes = [C.c_void_p, _ip, C.c_int, C.c_int, _ip] + [_dp] * 6
    L.oiga_set_geometry.argtypes = [C.c_void_p, C.c_int, _dp, _dp]
    L.oiga_set_fixtable.argtypes = [C.c_void_p, _dp, C.c_long]
    L.oiga_setup.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.oiga_get_info.argtypes = [C.c_void_p, _ip]
    L.oiga_set_aux.argtypes = [C.c_void_p, C.c_double, C.c_double, _dp]
    for name, rt in [("oiga_knots", _dp), ("oiga_spans", _ip), ("oiga_basis_offset", _ip), ("oiga_basis_detJac", _dp),
                     ("oiga_basis_weight", _dp), ("oiga_basis_point", _dp), ("oiga_basis_value", _dp)]:
        getattr(L, name).restype = rt
        getattr(L, name).argtypes = [C.c_void_p, C.c_int]
    L.oiga_lgmap.restype = _ip
    L.oiga_lgmap.argtypes = [C.c_void_p]
    L.oiga_partition.argtypes = [C.c_int, C.c_int, C.c_int, _ip, _ip, _ip]
    L.oiga_pattern_create.restype = C.c_void_p
    L.oiga_pattern_create.argtypes = [C.c_void_p, C.c_int]
    L.oiga_pattern_destroy.argtypes = [C.c_void_p]
    L.oiga_pattern_nrows.argtypes = [C.c_void_p]
    L.oiga_pattern_nnz.restype = C.c_long
    L.oiga_pattern_nnz.argtypes = [C.c_void_p]
    for name in ("oiga_pattern_rowptr", "oiga_pattern_colidx", "oiga_pattern_rank_rowstart"):
        getattr(L, name).restype = _ip
        getattr(L, name).argtypes = [C.c_void_p]
    L.oiga_assemble.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, C.c_double, _dp, C.c_double, _dp,
                                C.c_void_p, _dp, _dp]
    L.oiga_assemble_rank.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_double, _dp, C.c_double, _dp,
                                     C.c_void_p, _dp, _dp]
    L.oiga_assemble_range.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_double, _dp, C.c_double, _dp,
                                      C.c_void_p, _dp, _dp]
    L.oiga_stash_create.restype = C.c_void_p
    L.oiga_stash_destroy.argtypes = [C.c_void_p]
    L.oiga_stash_count.restype = C.c_long
    L.oiga_stash_count.argtypes = [C.c_void_p]
    L.oiga_assemble_rank_stash.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _dp, C.c_double, _dp, C.c_double, _dp,
                                           C.c_void_p, _dp, _dp, C.c_void_p]
    L.oiga_stash_apply.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, _dp, _dp]
    L.oiga_compute_scalar.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp, C.c_int, _dp]
    L.oiga_tabulate_element.argtypes = [C.c_void_p, _ip, _ip, _ip] + [_dp] * 12
    if not native:
        _LIB = L
    else:
        _NATIVE = L
    return L


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


class OracleIGA:
    """Mirror of the reference's IGA object restricted to what the assembly path reads."""

    def __init__(self, dim, dof=1, native=False):
        self.L = lib(native)
        self.dim, self.dof = dim, dof
        self.h = self.L.oiga_create(dim, dof)
        self._pat = {}

    def __del__(self):
        try:
            for p in self._pat.values():
                self.L.oiga_pattern_destroy(p)
            self.L.oiga_destroy(self.h)
        except Exception:
            pass

    # -- discretisation ---------------------------------------------------------------------
    def axis_uniform(self, axis, p, N, Ui=0.0, Uf=1.0, C=-1, periodic=False):
        assert self.L.oiga_axis_init_uniform(self.h, axis, p, N, Ui, Uf, C, int(periodic)) == 0

    def axis_knots(self, axis, p, U, periodic=False):
        U = np.ascontiguousarray(U, dtype=np.float64)
        assert self.L.oiga_axis_set_knots(self.h, axis, p, len(U) - 1, _d(U), int(periodic)) == 0

    def rule_size(self, axis, q):
        self.L.oiga_set_rule_size(self.h, axis, q)

    def order(self, k):
        self.L.oiga_set_order(self.h, k)

    def boundary_value(self, axis, side, field, value):
        self.L.oiga_set_boundary_value(self.h, axis, side, field, value)

    def boundary_load(self, axis, side, field, value):
        self.L.oiga_set_boundary_load(self.h, axis, side, field, value)

    def boundary_form(self, axis, side, flag=True):
        """IGASetBoundaryForm: visit the face with the boundary-integral pass (src/petigaelem.c:427-447)."""
        self.L.oiga_set_boundary_form(self.h, axis, side, int(bool(flag)))

    def tabulate_boundary(self, ID, axis, side):
        inf = self.info()
        nqp = int(np.prod([inf["nqp"][d] for d in range(self.dim) if d != axis])) if self.dim > 1 else 1
        nen = int(np.prod(inf["nen"]))
        o = dict(weight=np.zeros(nqp), detJac=np.zeros(nqp), detS=np.zeros(nqp), normal=np.zeros((nqp, self.dim)),
                 X0=np.zeros((nqp, self.dim)), shape0=np.zeros((nqp, nen)))
        ID3 = (C.c_int * 3)(*(list(ID) + [0, 0, 0])[:3])
        q = C.c_int()
        self.L.oiga_tabulate_boundary(self.h, ID3, axis, side, C.byref(q), *[_d(o[k]) for k in ("weight", "detJac", "detS", "normal", "X0", "shape0")])
        assert q.value == nqp
        return o

    def geometry(self, X, W=None):
        X = np.ascontiguousarray(X, dtype=np.float64)
        nsd = X.shape[-1]
        Wc = None if W is None else np.ascontiguousarray(W, dtype=np.float64)
        self.L.oiga_set_geometry(self.h, nsd, _d(X), _d(Wc))

    def fixtable(self, U):
        if U is None:
            self.L.oiga_set_fixtable(self.h, None, 0)
        else:
            U = np.ascontiguousarray(U, dtype=np.float64)
            self.L.oiga_set_fixtable(self.h, _d(U), U.size)

    def setup(self, size=1, rank=0):
        rc = self.L.oiga_setup(self.h, size, rank)
        assert rc == 0, rc
        return self.info()

    def info(self):
        buf = (C.c_int * 46)()
        self.L.oiga_get_info(self.h, buf)
        keys = ["p", "m", "nnp", "nel", "nqp", "nen", "proc_size", "proc_rank", "elem_start", "elem_width",
                "node_lstart", "node_lwidth", "node_gstart", "node_gwidth", "geom_size"]
        out = {"order": buf[0]}
        for k, key in enumerate(keys):
            out[key] = [buf[1 + 15 * i + k] for i in range(3)]
        return out

    def tables(self, axis):
        inf = self.info()
        nel, nqp, nen, m = inf["nel"][axis], inf["nqp"][axis], inf["nen"][axis], inf["m"][axis]
        g = lambda f, n, dt: np.ctypeslib.as_array(f(self.h, axis), shape=(n,)).astype(dt, copy=True)
        return dict(
            U=g(self.L.oiga_knots, m + 1, np.float64), span=g(self.L.oiga_spans, nel, np.int32),
            offset=g(self.L.oiga_basis_offset, nel, np.int32), detJac=g(self.L.oiga_basis_detJac, nel, np.float64),
            weight=g(self.L.oiga_basis_weight, nel * nqp, np.float64).reshape(nel, nqp),
            point=g(self.L.oiga_basis_point, nel * nqp, np.float64).reshape(nel, nqp),
            value=g(self.L.oiga_basis_value, nel * nqp * nen * 5, np.float64).reshape(nel, nqp, nen, 5))

    def lgmap(self):
        inf = self.info()
        n = int(np.prod(inf["node_gwidth"]))
        return np.ctypeslib.as_array(self.L.oiga_lgmap(self.h), shape=(n,)).copy()

    # -- pattern + assembly -----------------------------------------------------------------
    def pattern(self, size=1):
        """Global block-CSR pattern in PETSc numbering: (rowptr, colidx, rank_rowstart)."""
        if size not in self._pat:
            p = self.L.oiga_pattern_create(self.h, size)
            assert p
            self._pat[size] = p
        p = self._pat[size]
        n, nnz = self.L.oiga_pattern_nrows(p), self.L.oiga_pattern_nnz(p)
        rp = np.ctypeslib.as_array(self.L.oiga_pattern_rowptr(p), shape=(n + 1,)).copy()
        ci = np.ctypeslib.as_array(self.L.oiga_pattern_colidx(p), shape=(nnz,)).copy()
        rs = np.ctypeslib.as_array(self.L.oiga_pattern_rank_rowstart(p), shape=(size + 1,)).copy()
        return rp, ci, rs

    def assemble_rank(self, slot, form, params, size, rank, vals, rhs, shift=0.0, V=None, t=0.0, U=None):
        """Element loop of one emulated rank into preallocated global arrays (CPU-baseline timing)."""
        self.pattern(size)
        prm = np.ascontiguousarray(list(params) + [0.0] * 4, dtype=np.float64)
        rc = self.L.oiga_assemble_rank(self.h, size, rank, SLOT[slot], FORM[form], _d(prm), shift, _d(V), t, _d(U),
                                       self._pat[size], _d(vals), _d(rhs))
        assert rc == 0, rc

    def assemble(self, slot, form, params=(), size=1, shift=0.0, V=None, t=0.0, U=None, W=None, shift2=0.0, t0=0.0):
        """Returns (values[nnzb, dof, dof] or None, rhs[nrows, dof] or None) of one full assembly.
        W, shift2, t0: third vector / second shift / second time of the IE (U0, t0) and I2 (A, shiftV) drivers."""
        rp, ci, _ = self.pattern(size)
        p = self._pat[size]
        n, nnz, dof = len(rp) - 1, len(ci), self.dof
        slot_i = SLOT[slot]
        want_mat = slot in MAT_SLOTS
        want_vec = slot in VEC_SLOTS
        vals = np.zeros((nnz, dof, dof)) if want_mat else None
        rhs = np.zeros((n, dof)) if want_vec else None
        prm = np.ascontiguousarray(list(params) + [0.0] * 4, dtype=np.float64)
        Uc = None if U is None else np.ascontiguousarray(U, dtype=np.float64)
        Vc = None if V is None else np.ascontiguousarray(V, dtype=np.float64)
        Wc = None if W is None else np.ascontiguousarray(W, dtype=np.float64)
        self.L.oiga_set_aux(self.h, shift2, t0, _d(Wc))
        rc = self.L.oiga_assemble(self.h, size, slot_i, FORM[form], _d(prm), shift, _d(Vc), t, _d(Uc), p, _d(vals), _d(rhs))
        assert rc == 0, "oracle assemble failed rc=%d" % rc
        return vals, rhs

    def compute_scalar(self, scalar, params, n, U=None, size=1):
        """IGAComputeScalar (src/petigacomp.c:35-96) with a built-in Scalar callback: 'ERRNORM' (ErrorSqr :103-124,
        params = [k, exact id, choice]) or 'CH_STATS' (demo/CahnHilliard2D.c:43-58, params = [theta, alpha, cbar])."""
        prm = np.ascontiguousarray(list(params) + [0.0] * 4, dtype=np.float64)
        Uc = None if U is None else np.ascontiguousarray(U, dtype=np.float64)
        S = np.zeros(n)
        rc = self.L.oiga_compute_scalar(self.h, size, SCALAR[scalar], _d(prm), _d(Uc), n, _d(S))
        assert rc == 0, "oracle compute_scalar failed rc=%d" % rc
        return S

    def error_norm(self, k, U=None, exact=1, choice=0, size=1):
        """IGAComputeErrorNorm (src/petigacomp.c:155-186)."""
        return np.sqrt(self.compute_scalar("ERRNORM", [k, exact, choice], self.dof, U=U, size=size))

    def tabulate(self, ID, order=3):
        inf = self.info()
        nqp, nen = int(np.prod(inf["nqp"])), int(np.prod(inf["nen"]))
        dim = self.dim
        nsd = dim
        o = dict(weight=np.zeros(nqp), detJac=np.zeros(nqp), detX=np.zeros(nqp), point=np.zeros((nqp, dim)),
                 X0=np.zeros((nqp, nsd)), X1=np.zeros((nqp, nsd, dim)), X2=np.zeros((nqp, nsd, dim, dim)),
                 X3=np.zeros((nqp, nsd, dim, dim, dim)), shape0=np.zeros((nqp, nen)), shape1=np.zeros((nqp, nen, nsd)),
                 shape2=np.zeros((nqp, nen, nsd, nsd)), shape3=np.zeros((nqp, nen, nsd, nsd, nsd)))
        ID3 = (C.c_int * 3)(*(list(ID) + [0, 0, 0])[:3])
        q, a = C.c_int(), C.c_int()
        self.L.oiga_tabulate_element(self.h, ID3, C.byref(q), C.byref(a), *[_d(o[k]) for k in
                                     ("weight", "detJac", "detX", "point", "X0", "X1", "X2", "X3",
                                      "shape0", "shape1", "shape2", "shape3")])
        return o


def read_iga_file(filename):
    """IGALoad + IGALoadGeometry (src/petigaio.c:11-73,201-286) restated with numpy: returns
    (axes [(p, U)], nsd, X natural [..][nsd] or None, W natural or None, rational).  PETSc binary files are big-endian;
    the geometry Vec holds (w*x, w) per control point in natural order and is de-homogenised on load (:259-266)."""
    raw = open(filename, "rb").read()
    pos = [0]

    def ints(n):
        v = np.frombuffer(raw, dtype=">i4", count=n, offset=pos[0]).astype(np.int64)
        pos[0] += 4 * n
        return v

    def reals(n):
        v = np.frombuffer(raw, dtype=">f8", count=n, offset=pos[0]).astype(np.float64)
        pos[0] += 8 * n
        return v

    classid, info, dim = ints(3)
    if classid != 1211299:                      # IGA_FILE_CLASSID (include/petiga.h:394)
        raise ValueError("Not an IGA in file")  # :32
    axes = []
    for _ in range(dim):
        p, m1 = ints(2)
        axes.append((int(p), reals(int(m1))))
    if not (info & 1):
        return axes, 0, None, None, False
    nsd = int(ints(1)[0])
    vid, n = ints(2)
    if vid != 1211214:                          # VEC_FILE_CLASSID
        raise ValueError("Not a vector next in file")
    sizes = [len(U) - 1 - p for p, U in axes]   # geom_sizes = m - p control points per axis
    if n != int(np.prod(sizes)) * (nsd + 1):
        raise ValueError("Vector in file different size than input vector")
    Xw = reals(int(n)).reshape(-1, nsd + 1)
    W = Xw[:, nsd].copy()
    X = Xw[:, :nsd].copy()
    nz = np.abs(W) > 0
    X[nz] /= W[nz][:, None]                     # :262-264
    rational = bool(W.max() - W.min() > 100 * np.finfo(float).eps)   # :251-253
    shape = tuple(sizes[::-1])
    return axes, nsd, X.reshape(shape + (nsd,)), W.reshape(shape), rational


def oracle_from_file(filename, dof=1):
    """An OracleIGA with the axes and geometry of an IGA file (what IGARead leaves behind)."""
    axes, nsd, X, W, rational = read_iga_file(filename)
    o = OracleIGA(len(axes), dof)
    for d, (p, U) in enumerate(axes):
        o.axis_knots(d, p, U)
    if X is not None:
        o.geometry(X, W)
    return o


def partition(size, rank, dim, N):
    L = lib()
    Na = (C.c_int * 3)(*(list(N) + [1, 1, 1])[:3])
    n = (C.c_int * 3)(0, 0, 0)
    i = (C.c_int * 3)(0, 0, 0)
    rc = L.oiga_partition(size, rank, dim, Na, n, i)
    assert rc == 0, rc
    return list(n)[:dim], list(i)[:dim]
