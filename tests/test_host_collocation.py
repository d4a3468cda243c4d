"""Isogeometric collocation on the host side (no GPU): tables, boxes, numbering and pattern of IGASetUseCollocation against the
reference restatement in tests/colloc_ref.py; the reference's matrices against scipy's B-splines; known answers of the reference
system; and the argument / order / scope errors the host mirror raises before any device call."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse.linalg as spl

import petiga_b200 as pb
from oracle.oracle import partition
from tests.colloc_ref import Axis, Space, assemble, l2_error_2d, scipy_laplace_kron

PETSC_ERR_SUP, PETSC_ERR_ARG_WRONGSTATE = 56, 73

# (dim, degrees, elements, continuity or knot vectors)
CASES = [
    (1, (2,), (7,), None),
    (1, (4,), (9,), None),
    (2, (2, 2), (6, 5), None),
    (2, (3, 3), (5, 7), None),
    (2, (4, 2), (6, 4), None),                      # mixed degrees
    (2, (2, 3), (5, 4), (0, 1)),                    # C0 on axis 0: Greville points on knots
    (2, (3, 2), "nonuniform", None),
    (3, (2, 2, 2), (4, 3, 5), None),
    (3, (3, 2, 4), (3, 4, 3), None),
    (3, (4, 4, 4), (3, 3, 3), (2, 3, 1)),
]
NONUNIFORM = [np.array([0, 0, 0, 0, 0.1, 0.15, 0.4, 0.7, 0.72, 1, 1, 1, 1.0]), np.array([0, 0, 0, 0.3, 0.35, 0.5, 0.9, 1, 1, 1.0])]


def make_iga(dim, ps, Ns, Cs, rank=0, size=1, colloc=True):
    g = pb.IGA(dim, 1, rank=rank, size=size)
    if colloc:
        g.SetUseCollocation(True)
    for d in range(dim):
        if Ns == "nonuniform":
            g.AxisSetKnots(d, ps[d], NONUNIFORM[d])
        else:
            g.AxisInitUniform(d, ps[d], Ns[d], C_=(Cs[d] if Cs else -1))
    g.SetUp()
    return g


def ref_space(g, dim, ps, size=1):
    axes = [Axis(ps[d], g.AxisGetKnots(d)) for d in range(dim)]
    try:
        grid, _ = partition(size, 0, dim, [len(a.span_off) for a in axes])
    except AssertionError:
        pytest.skip("partition too fine for this mesh")
    return Space(axes, grid)


@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s_%s_%s" % (c[0], "".join(map(str, c[1])), c[2] if isinstance(c[2], str) else "x".join(map(str, c[2])), c[3]))
def test_tables_bit_exact(case):
    dim, ps, Ns, Cs = case
    g = make_iga(dim, ps, Ns, Cs)
    assert g.GetUseCollocation()
    s = ref_space(g, dim, ps)
    inf = g.info()
    for d in range(dim):
        a = s.axes[d]
        assert inf["nel"][d] == a.nnp and inf["nqp"][d] == 1
        t = g.tables(d)
        assert np.array_equal(t["point"][:, 0], a.point)
        assert np.array_equal(t["value"][:, 0], a.value)
        assert np.all(t["weight"] == 1.0) and np.all(t["detJac"] == 1.0)


@pytest.mark.parametrize("size", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s" % (c[0], "".join(map(str, c[1]))))
def test_boxes_lgmap_pattern(case, size):
    dim, ps, Ns, Cs = case
    g0 = make_iga(dim, ps, Ns, Cs)
    s = ref_space(g0, dim, ps, size)
    ngal = [len(a.span_off) for a in s.axes]
    if any(n < P for n, P in zip(ngal, s.grid)):
        pytest.skip("partition too fine for this mesh")
    for rank in range(size):
        g = make_iga(dim, ps, Ns, Cs, rank=rank, size=size)
        gal = make_iga(dim, ps, Ns, Cs, rank=rank, size=size, colloc=False)
        inf, infg = g.info(), gal.info()
        boxes = s.info(rank)
        for d in range(dim):
            es, ew, ls, lw, gs, gw = boxes[d]
            assert (inf["elem_start"][d], inf["elem_width"][d]) == (es, ew)
            assert (inf["node_lstart"][d], inf["node_lwidth"][d]) == (ls, lw)
            assert (inf["node_gstart"][d], inf["node_gwidth"][d]) == (gs, gw)
            # the owned boxes (hence the numbering) are the Galerkin ones
            assert (infg["node_lstart"][d], infg["node_lwidth"][d]) == (ls, lw)
        L = g.layout()
        sz = L.sizes()
        assert sz["nloc"] == sz["nown"]                               # no ghost rows
        assert np.array_equal(L.lgmap(), s.lgmap(rank))
        assert np.array_equal(g.lgmap(), s.lgmap(rank))
        rp, ci = s.pattern(rank)
        for block in (0, 1):
            rpl, cil = L.pattern(block, 1)
            assert np.array_equal(rpl, rp) and np.array_equal(cil, ci)
        assert all(e.size == 0 for e in (L.exchange(0), L.exchange(1)))


@pytest.mark.parametrize("dim,p,N", [(2, 2, 6), (2, 3, 5), (2, 4, 4), (3, 2, 3), (3, 3, 3)])
def test_reference_matrix_is_kronecker_sum(dim, p, N):
    """The reference's identity-geometry Laplace matrix equals, in natural order, the Kronecker sum of 1-D scipy collocation
    matrices with identity rows on the boundary (1e-13 relative)."""
    U = pb.cases.uniform_knots(p, N)
    axes = [Axis(p, U) for _ in range(dim)]
    A, _ = assemble(axes, values={(d, s): 0.0 for d in range(dim) for s in range(2)})
    B = scipy_laplace_kron(axes)
    assert abs(A - B).max() <= 1e-13 * abs(B).max()


@pytest.mark.parametrize("dim,p,N", [(2, 2, 8), (2, 3, 6), (3, 2, 4), (3, 4, 3)])
def test_laplace_constant_solution(dim, p, N):
    axes = [Axis(p, pb.cases.uniform_knots(p, N)) for _ in range(dim)]
    A, F = assemble(axes, values={(d, s): 1.0 for d in range(dim) for s in range(2)})
    u = spl.spsolve(A.tocsc(), F)
    assert np.abs(u - 1.0).max() <= 1e-12


@pytest.mark.parametrize("p", [2, 3, 4])
def test_convtest_orders(p):
    """Greville collocation converges with order p for even p and p - 1 for odd p (L2, N = 16 -> 32 -> 64)."""
    errs = []
    for N in (16, 32, 64):
        axes = [Axis(p, pb.cases.uniform_knots(p, N)) for _ in range(2)]
        A, F = assemble(axes, "CONVTEST_COLLOCATION", (1.0, 1.0), values={(d, s): 0.0 for d in range(2) for s in range(2)})
        errs.append(l2_error_2d(axes, spl.spsolve(A.tocsc(), F)))
    rates = np.log2(np.array(errs[:-1]) / np.array(errs[1:]))
    want = p - 0.2 if p % 2 == 0 else p - 1.2
    assert np.all(rates >= want), (errs, rates)


def test_set_use_collocation_order():
    g = make_iga(2, (2, 2), (4, 4), None)
    g.SetUseCollocation(True)                     # unchanged: allowed
    with pytest.raises(pb.IGAError) as e:
        g.SetUseCollocation(False)
    assert e.value.code == PETSC_ERR_ARG_WRONGSTATE
    h = make_iga(2, (2, 2), (4, 4), None, colloc=False)
    with pytest.raises(pb.IGAError) as e:
        h.SetUseCollocation(True)
    assert e.value.code == PETSC_ERR_ARG_WRONGSTATE


def test_setup_scope_errors():
    g = pb.IGA(2, 1)
    g.SetUseCollocation(True)
    g.AxisInitUniform(0, 2, 4, periodic=True)
    g.AxisInitUniform(1, 2, 4)
    with pytest.raises(pb.IGAError) as e:
        g.SetUp()
    assert e.value.code == PETSC_ERR_SUP and "periodic" in str(e.value)
    g = pb.IGA(2, 1)
    g.SetUseCollocation(True)
    g.AxisInitUniform(0, 1, 4)
    g.AxisInitUniform(1, 2, 4)
    with pytest.raises(pb.IGAError) as e:
        g.SetUp()
    assert e.value.code == PETSC_ERR_SUP and "degree" in str(e.value)


def _dummy(cls, iga):
    """A non-NULL Mat/Vec handle for the checks that run before the handle is looked at (never dereferenced)."""
    buf = C.create_string_buffer(64)
    obj = cls.__new__(cls)
    obj.iga, obj.h, obj._buf = iga, C.c_void_p(C.addressof(buf)), buf
    return obj


def _compute_system(g):
    A, B = _dummy(pb.Mat, g), _dummy(pb.Vec, g)
    g.ComputeSystem(A, B)


@pytest.mark.parametrize("what", ["galerkin_form", "load", "boundary_form", "kronecker", "slot", "colloc_form_on_galerkin"])
def test_compute_scope_errors(what):
    """Every unsupported combination is PETSC_ERR_SUP before the first device call (no CPU fallback, no device needed)."""
    g = make_iga(2, (2, 2), (4, 4), None, colloc=(what != "colloc_form_on_galerkin"))
    form = "LAPLACE_COLLOCATION"
    if what == "galerkin_form":
        form = "LAPLACE"
    elif what == "load":
        g.SetBoundaryLoad(0, 1, 0, 1.0)
    elif what == "boundary_form":
        g.SetBoundaryForm(1, 0, True)
    elif what == "kronecker":
        g.SetOption("path", 2)
    if what == "slot":
        g.SetForm("FUNCTION", "POISSON")
        with pytest.raises(pb.IGAError) as e:
            g.ComputeFunction(_dummy(pb.Vec, g), _dummy(pb.Vec, g))
        assert e.value.code == PETSC_ERR_SUP
        return
    g.SetForm("SYSTEM", form)
    with pytest.raises(pb.IGAError) as e:
        _compute_system(g)
    assert e.value.code == PETSC_ERR_SUP


def test_fixtable_is_unsupported():
    g = make_iga(2, (2, 2), (4, 4), None)
    g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
    g.H.IGASetFixTable(g.h, C.c_void_p(C.addressof(C.create_string_buffer(8))))
    with pytest.raises(pb.IGAError) as e:
        _compute_system(g)
    assert e.value.code == PETSC_ERR_SUP


def test_collocation_compute_needs_the_device():
    """A supported collocation system reaches the device: on a CPU box that is an error, never a host computation."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    g = make_iga(2, (2, 2), (4, 4), None)
    g.SetForm("SYSTEM", "LAPLACE_COLLOCATION")
    with pytest.raises(pb.IGAError) as e:
        g.CreateMat()
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


class _Space(C.Structure):
    """petiga_cuda_space of include/petiga_cuda.h"""
    _fields_ = ([("dim", C.c_int), ("dof", C.c_int), ("order", C.c_int)] +
                [(n, C.c_int * 3) for n in ("p", "m", "nel", "nnp", "periodic", "nqp1")] +
                [(n, C.c_void_p * 3) for n in ("U", "offset", "detJac", "weight", "point", "value")] +
                [(n, C.c_int * 3) for n in ("proc_sizes", "proc_ranks", "elem_start", "elem_width", "node_lstart", "node_lwidth",
                                            "node_gstart", "node_gwidth")] +
                [("collocation", C.c_int)])


@pytest.mark.parametrize("nel_from", ["axis", "basis", "wrong"])
def test_layout_accepts_the_axis_element_count(nel_from):
    """A caller that fills petiga_cuda_space from PetIGA's structures, as integration/petiga_cuda_glue.c does, passes the axis's
    element count (IGAAxis.nel) in nel; the table length IGABasis.nel (= nnp) is accepted too; anything else is an argument error."""
    dim, ps, Ns = 2, (2, 3), (5, 4)
    g = make_iga(dim, ps, Ns, None, rank=1, size=2)
    inf = g.info()
    sp_ = _Space()
    sp_.dim, sp_.dof, sp_.order, sp_.collocation = dim, 1, inf["order"], 1
    keep = []
    for d in range(3):
        t = g.tables(d)
        for name, arr in (("U", t["U"]), ("detJac", t["detJac"]), ("weight", t["weight"]), ("point", t["point"]), ("value", t["value"])):
            a = np.ascontiguousarray(arr, dtype=np.float64)
            keep.append(a)
            getattr(sp_, name)[d] = a.ctypes.data
        ax = Axis(inf["p"][d], t["U"]) if d < dim else None
        off = np.ascontiguousarray(ax.offset if ax else [0], dtype=np.int32)
        keep.append(off)
        sp_.offset[d] = off.ctypes.data
        nel_axis = len(ax.span_off) if ax else 1
        sp_.p[d], sp_.m[d], sp_.nnp[d], sp_.nqp1[d] = inf["p"][d], inf["m"][d], inf["nnp"][d], 1
        sp_.nel[d] = {"axis": nel_axis, "basis": inf["nnp"][d], "wrong": inf["nnp"][d] - 1 if d < dim else 1}[nel_from]
        for f in ("elem_start", "elem_width", "node_lstart", "node_lwidth", "node_gstart", "node_gwidth"):
            getattr(sp_, f)[d] = inf[f][d]
        sp_.proc_sizes[d], sp_.proc_ranks[d] = inf["proc_size"][d], inf["proc_rank"][d]
    L = pb.load_cuda()
    h = C.c_void_p()
    rc = L.petiga_layout_create(C.byref(h), C.byref(sp_), 1, 2)
    if nel_from == "wrong":
        assert rc == 1      # PETIGA_CUDA_ERR_ARG
        return
    assert rc == 0, L.petiga_cuda_last_error()
    try:
        mine, ref = pb.iga.Layout(h.value), g.layout()
        assert mine.sizes() == ref.sizes()
        assert np.array_equal(mine.lgmap(), ref.lgmap())
        for a, b in zip(mine.pattern(1, 1), ref.pattern(1, 1)):
            assert np.array_equal(a, b)
    finally:
        L.petiga_layout_destroy(h)
