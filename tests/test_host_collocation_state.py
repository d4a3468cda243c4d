"""Bratu by collocation on the host side (no GPU): the collocation state halo of the layout (state numbering and halo lists on 1-8
ranks against a numpy restatement, and driven with real messages over gloo), the scope errors of the nonlinear collocation slots,
and the reference of tests/colloc_state_ref.py pinned independently (scipy Kronecker products, the exact 1-D solution, finite
differences of F)."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import petiga_b200 as pb
from oracle.oracle import read_iga_file
from tests.colloc_ref import Axis, scipy_laplace_kron
from tests.colloc_state_ref import bratu_1d_exact, fixed_rows, jacobian, newton, operators, residual
from tests.geomutil import refine_annulus
from tests.test_host_collocation import CASES, PETSC_ERR_SUP, _dummy, make_iga, ref_space

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_FACES = lambda dim, v: {(d, s): v for d in range(dim) for s in range(2)}   # noqa: E731


def state_halo_ref(s, rank):
    """numpy restatement for `rank` of Space s: (staterow, nstate, [(owner, first, count)], [(neighbour, rows)])"""
    lg = s.lgmap(rank)
    r0, r1 = s.rank_start[rank], s.rank_start[rank + 1]
    nown = r1 - r0
    own = (lg >= r0) & (lg < r1)
    foreign = np.unique(lg[~own])
    staterow = np.where(own, lg - r0, nown + np.searchsorted(foreign, lg))
    owners = np.searchsorted(s.rank_start, foreign, side="right") - 1
    runs = [(int(q), nown + int(np.argmax(owners == q)), int((owners == q).sum())) for q in np.unique(owners)]
    reads = []
    for q in range(s.size):
        if q == rank:
            continue
        theirs = s.lgmap(q)
        mine = np.unique(theirs[(theirs >= r0) & (theirs < r1)]) - r0
        if mine.size:
            reads.append((q, mine))
    return staterow, nown + foreign.size, runs, reads


@pytest.mark.parametrize("size", [1, 2, 3, 4, 8])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s" % (c[0], "".join(map(str, c[1]))))
def test_state_halo_lists(case, size):
    dim, ps, Ns, Cs = case
    g0 = make_iga(dim, ps, Ns, Cs)
    s = ref_space(g0, dim, ps, size)
    if any(len(a.span_off) < P for a, P in zip(s.axes, s.grid)):
        pytest.skip("partition too fine for this mesh")
    for rank in range(size):
        g = make_iga(dim, ps, Ns, Cs, rank=rank, size=size)          # keeps the layout alive
        L = g.layout()
        staterow, nstate, runs, reads = state_halo_ref(s, rank)
        got, n = L.staterow()
        assert np.array_equal(got, staterow) and n == nstate
        assert [tuple(r[:3]) for r in L.exchange(2)] == runs and np.all(L.exchange(2)[:, 3] == 0)
        k3 = L.exchange(3)
        assert [int(r[0]) for r in k3] == [q for q, _ in reads]
        for i, (q, rows) in enumerate(reads):
            assert k3[i][1] == rows[0] and k3[i][2] == rows.size and k3[i][3] == 0
            assert np.array_equal(L.recv_rows(i, rows.size), rows)
        # the matrix side is what it was: no ghost rows, kinds 0 and 1 empty, the nodes of other ranks have no local row
        assert all(e.size == 0 for e in (L.exchange(0), L.exchange(1)))
        sz = L.sizes()
        assert sz["nloc"] == sz["nown"]
        assert np.array_equal(L.localrow() >= 0, staterow < sz["nown"])
        if size == 1:
            assert np.array_equal(staterow, np.arange(sz["nown"])[s.lgmap(0)]) and nstate == sz["nown"]


def test_galerkin_layout_has_no_state_halo():
    g = make_iga(2, (2, 2), (6, 5), None, rank=1, size=4, colloc=False)
    L = g.layout()
    assert L.exchange(2).size == 0 and L.exchange(3).size == 0
    assert L.exchange(0).size and L.exchange(1).size
    n = C.c_int()
    assert L.L.petiga_layout_staterow(L.h, C.byref(n), None) == 1     # PETIGA_CUDA_ERR_ARG


def _halo_worker(rank, world, port, case, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dim, ps, Ns = case
        g = make_iga(dim, ps, Ns, None, rank=rank, size=world)           # host logic only: no GPU touched
        L = g.layout()
        lg = L.lgmap()
        staterow, nstate = L.staterow()
        nown = L.sizes()["nown"]
        ntot = int(np.prod([g.info()["nnp"][d] for d in range(dim)]))
        glob = np.sin(np.arange(ntot) * 0.37) + 1e-3 * np.arange(ntot)   # a global vector in the global numbering
        r0 = int(lg[staterow == 0][0]) if nown else 0
        loc = np.full(nstate, np.nan)
        loc[:nown] = glob[r0:r0 + nown]
        reqs, bufs = [], []
        for i, (peer, _, nrows, _) in enumerate(L.exchange(3)):           # owners send what each neighbour reads
            t = torch.from_numpy(loc[L.recv_rows(i, int(nrows))].copy())
            reqs.append(dist.isend(t, int(peer), tag=7))
            bufs.append(t)
        incoming = []
        for (peer, first, nrows, _) in L.exchange(2):                     # one run per owner
            t = torch.zeros(int(nrows), dtype=torch.float64)
            reqs.append(dist.irecv(t, int(peer), tag=7))
            incoming.append((int(first), t))
        for r in reqs:
            r.wait()
        for first, t in incoming:
            loc[first:first + t.numel()] = t.numpy()
        out[rank] = bool(np.array_equal(loc[staterow], glob[lg])) and len(L.exchange(2)) >= (3 if world == 4 else 1)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,case", [(2, (3, (3, 2, 2), (5, 4, 4))), (4, (2, (3, 3), (9, 10))), (4, (3, (2, 2, 2), (6, 6, 6)))])
def test_state_halo_over_gloo(world, case):
    """Every rank's halo-filled state equals the global vector at its ghost-box nodes (on 4 ranks each ghost box reaches three
    other owners)."""
    import random
    port = 29900 + random.randint(0, 90)
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_halo_worker, args=(world, port, case, out), nprocs=world, join=True)
    assert all(out.get(r, False) for r in range(world)), dict(out)


# ---- scope errors of the nonlinear collocation slots (before any device call) ----
def _call(g, slot):
    V = lambda: _dummy(pb.Vec, g)        # noqa: E731
    M = lambda: _dummy(pb.Mat, g)        # noqa: E731
    {"FUNCTION": lambda: g.ComputeFunction(V(), V()), "JACOBIAN": lambda: g.ComputeJacobian(V(), M()),
     "IFUNCTION": lambda: g.ComputeIFunction(1.0, V(), 0.0, V(), V()), "IJACOBIAN": lambda: g.ComputeIJacobian(1.0, V(), 0.0, V(), M()),
     "RHSFUNCTION": lambda: g.ComputeRHSFunction(0.0, V(), V())}[slot]()


@pytest.mark.parametrize("what", ["on_galerkin", "galerkin_bratu", "rhs_slot", "dof2", "load", "boundary_form", "kronecker", "fixtable"])
@pytest.mark.parametrize("slot", ["FUNCTION", "JACOBIAN", "IFUNCTION", "IJACOBIAN"])
def test_state_scope_errors(what, slot):
    if what == "dof2":
        g = pb.IGA(2, 2)
        g.SetUseCollocation(True)
        for d in range(2):
            g.AxisInitUniform(d, 2, 4)
        g.SetUp()
    else:
        g = make_iga(2, (2, 2), (4, 4), None, colloc=(what != "on_galerkin"))
    form = "BRATU" if what == "galerkin_bratu" else "BRATU_COLLOCATION"
    if what == "rhs_slot":
        if slot != "FUNCTION":
            pytest.skip("one RHS case is enough")
        g.SetForm("RHSFUNCTION", "BRATU", (1.0,))
        slot = "RHSFUNCTION"
    else:
        g.SetForm(slot, form, (1.0,))
    if what == "load":
        g.SetBoundaryLoad(0, 1, 0, 1.0)
    elif what == "boundary_form":
        g.SetBoundaryForm(1, 0, True)
    elif what == "kronecker":
        g.SetOption("path", 2)
    elif what == "fixtable":
        g.H.IGASetFixTable(g.h, C.c_void_p(C.addressof(C.create_string_buffer(8))))
    with pytest.raises(pb.IGAError) as e:
        _call(g, slot)
    assert e.value.code == PETSC_ERR_SUP, str(e.value)


def test_state_forms_need_the_device():
    """A supported nonlinear collocation call reaches the device: on a CPU box that is an error, never a host computation."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    g = make_iga(2, (2, 2), (4, 4), None)
    g.SetForm("FUNCTION", "BRATU_COLLOCATION", (1.0,))
    with pytest.raises(pb.IGAError) as e:
        g.CreateVec()
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


# ---- independent pins of tests/colloc_state_ref.py ----
def _scipy_ops(axes):
    """B = Kronecker product of BSpline.design_matrix at the Greville points, -L = the Kronecker sum of the second-derivative
    collocation matrices (natural order, axis 0 fastest)"""
    from scipy.interpolate import BSpline
    B = None
    for a in axes[::-1]:
        U = np.array(a.U)
        gv = np.array([np.mean(U[i + 1:i + a.p + 1]) for i in range(a.nnp)])
        b0 = BSpline.design_matrix(gv, U, a.p)
        B = b0 if B is None else sp.kron(B, b0)
    return B.tocsr(), scipy_laplace_kron(axes, values_on_all_faces=False)


@pytest.mark.parametrize("dim,p,N", [(1, 3, 12), (2, 2, 6), (2, 3, 5), (3, 2, 3), (3, 4, 3)])
def test_reference_against_scipy(dim, p, N):
    """F(U) = -L U - lambda exp(B U) and J = -L - lambda diag(exp(B U)) B on the unfixed rows (1e-13); the fixed rows are U - value
    and identity rows."""
    axes = [Axis(p, pb.cases.uniform_knots(p, N)) for _ in range(dim)]
    Bs, Ls = _scipy_ops(axes)
    ops = operators(axes)
    rng = np.random.default_rng(dim * 10 + p)
    U = rng.uniform(-0.5, 0.8, Bs.shape[0])
    lam, values = 1.7, ALL_FACES(dim, 0.25)
    mask, fval = fixed_rows(axes, values)
    F = residual(ops, U, lam, values=values, axes=axes)
    J = jacobian(ops, U, lam, values=values, axes=axes).toarray()
    Fs = Ls @ U - lam * np.exp(Bs @ U)
    Js = (Ls - sp.diags(lam * np.exp(Bs @ U)) @ Bs).toarray()
    assert np.abs(F - Fs)[~mask].max() <= 1e-13 * np.abs(Fs).max()
    assert np.abs(J - Js)[~mask].max() <= 1e-13 * np.abs(Js).max()
    assert np.array_equal(F[mask], U[mask] - fval[mask])
    assert np.array_equal(J[mask], np.eye(len(U))[mask])


def test_reference_1d_exact_solution_rates():
    """u'' + e^u = 0, u(0) = u(1) = 0: the Newton solution of the reference converges to the exact solution at rate 2 for p = 2, 3 and
    about 4 for p = 4 (L2, N = 16 -> 32 -> 64): the p / p - 1 Greville pattern of ConvTest."""
    from scipy.interpolate import BSpline
    th, exact = bratu_1d_exact(1.0)
    assert abs(th - 1.5171645990508) <= 1e-12 and abs(exact(0.5) - 0.14053921440048) <= 1e-12
    xs = np.linspace(0, 1, 4001)
    for p, want in ((2, 1.9), (3, 1.9), (4, 3.8)):
        errs = []
        for N in (16, 32, 64):
            axes = [Axis(p, pb.cases.uniform_knots(p, N))]
            U, hist = newton(operators(axes), 1.0, ALL_FACES(1, 0.0), axes)
            assert len(hist) <= 6 and hist[-1] <= 1e-12 * hist[0], hist
            errs.append(np.sqrt(np.mean((BSpline(np.array(axes[0].U), U, p)(xs) - exact(xs)) ** 2)))
        rates = np.log2(np.array(errs[:-1]) / np.array(errs[1:]))
        assert np.all(rates >= want), (p, errs, rates)


class _Rec:
    """records what refine_annulus sets on an IGA"""
    def __init__(self, dim, dof):
        self.knots = {}

    def axis_knots(self, d, p, U):
        self.knots[d] = (p, U)

    def geometry(self, X, W):
        pass


def geometry_case(kind):
    """(axes, X, W) of the perturbed cube (mapped) or the 2-D quarter annulus (NURBS)"""
    if kind == "mapped":
        axes_f, nsd, X, W, rational = read_iga_file(os.path.join(GOLD, "cube_perturbed.dat"))
        return [Axis(p, U) for p, U in axes_f], X, None
    o, X, W = refine_annulus(_Rec, N=(5, 6), p=2)
    return [Axis(*o.knots[d]) for d in range(2)], X, W


@pytest.mark.parametrize("transient", [False, True], ids=["jacobian", "ijacobian"])
@pytest.mark.parametrize("kind", ["mapped", "rational"])
def test_reference_jacobian_is_the_derivative_of_f(kind, transient):
    """central differences of F (IFunction with V = V0 + shift (U - U0)) along random directions agree with J to ~1e-7"""
    axes, X, W = geometry_case(kind)
    ops = operators(axes, X=X, W=W)
    n = ops[0].shape[0]
    rng = np.random.default_rng(3)
    U0, V0 = rng.uniform(-0.3, 0.6, n), rng.uniform(-1, 1, n)
    lam, shift, values = 2.0, (7.5 if transient else 0.0), {(0, 0): 0.5, (1, 1): -0.25}

    def F(U):
        V = V0 + shift * (U - U0) if transient else None
        return residual(ops, U, lam, V=V, values=values, axes=axes)
    J = jacobian(ops, U0, lam, shift=shift, values=values, axes=axes)
    h = 1e-5
    for _ in range(4):
        w = rng.standard_normal(n)
        fd = (F(U0 + h * w) - F(U0 - h * w)) / (2 * h)
        Jw = J @ w
        assert np.linalg.norm(fd - Jw) <= 1e-7 * np.linalg.norm(Jw), np.linalg.norm(fd - Jw) / np.linalg.norm(Jw)
