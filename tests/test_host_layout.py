"""CPU tests of the product's host logic against the oracle: 1-D tables, partition, numbering (lgmap) and the
closed-form CSR pattern must be bit-exact (SURVEY 8a L1-L3, T1-T4).  No GPU needed: petiga_layout_* is host code."""
import ctypes as C
import os

import numpy as np
import pytest

import petiga_b200 as pb
from oracle.oracle import partition as oracle_partition
from tests.common import Case

CASES = [
    Case(1, p=1, N=5), Case(1, p=2, N=7, C=0), Case(1, p=3, N=16, periodic=True), Case(1, p=4, N=9, C=1),
    Case(2, p=2, N=(8, 5)), Case(2, p=3, N=6, C=(2, 0)), Case(2, p=2, N=10, periodic=True), Case(2, p=(2, 3), N=(7, 6)),
    Case(2, dof=3, p=2, N=(10, 5), periodic=(True, False)), Case(3, p=2, N=6), Case(3, p=3, N=(5, 4, 6)), Case(3, p=1, N=4),
    Case(3, dof=3, p=2, N=4), Case(3, p=2, N=(6, 10, 6), periodic=(False, True, False)), Case(3, p=4, N=5, C=2),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "d%d_p%s_N%s_C%s_w%s_dof%d" % (c.dim, c.p, c.N, c.C, c.periodic, c.dof))
@pytest.mark.parametrize("size", [1, 2, 3, 4, 8])
def test_tables_numbering_pattern_bit_exact(case, size):
    o = case.oracle()
    Nel = [case.N[d] if isinstance(case.N, tuple) else case.N for d in range(case.dim)]
    try:
        grid, _ = oracle_partition(size, 0, case.dim, Nel)
    except AssertionError:
        pytest.skip("partition too fine")
    if any(isinstance(case.periodic, tuple) and case.periodic[d] or case.periodic is True for d in range(case.dim)):
        # a periodic axis needs every rank box wider than the stencil; skip over-decomposed tiny meshes
        if any(Nel[d] // grid[d] < 2 * (case.p[d] if isinstance(case.p, tuple) else case.p) + 1 for d in range(case.dim)) and size > 1:
            pytest.skip("periodic mesh too small for this rank count")
    rp_o, ci_o, rs_o = o.pattern(size)
    for rank in range(size):
        inf_o = o.setup(size, rank)
        g = case.product(rank=rank, size=size)
        inf_p = g.info()
        assert inf_p == inf_o
        assert pb.iga_partition(size, rank, case.dim, Nel) == oracle_partition(size, rank, case.dim, Nel)
        for d in range(case.dim):
            to, tp = o.tables(d), g.tables(d)
            for k in ("U", "detJac", "weight", "point"):
                assert np.array_equal(to[k], tp[k]), k          # bit-exact knots / rule / Jacobians
            assert np.array_equal(to["value"], tp["value"])      # same algorithm, same operation order
        assert np.array_equal(g.lgmap(), o.lgmap())
        L = g.layout()
        assert np.array_equal(L.lgmap(), o.lgmap())
        # block pattern of this rank's rows == the oracle's rows [rs[rank], rs[rank+1])
        rp, ci = L.pattern(1, case.dof)
        r0, r1 = rs_o[rank], rs_o[rank + 1]
        assert len(rp) - 1 == r1 - r0
        assert np.array_equal(rp, rp_o[r0:r1 + 1] - rp_o[r0])
        assert np.array_equal(ci, ci_o[rp_o[r0]:rp_o[r1]])
        if case.dof > 1:   # AIJ expansion: UnblockIndices (petigamat.c:303-314)
            rps, cis = L.pattern(0, case.dof)
            dof = case.dof
            assert len(rps) - 1 == (r1 - r0) * dof
            for r in range(0, r1 - r0, max(1, (r1 - r0) // 7)):
                cols = ci[rp[r]:rp[r + 1]]
                exp = (cols[:, None] * dof + np.arange(dof)[None, :]).reshape(-1)
                for c in range(dof):
                    row = r * dof + c
                    assert np.array_equal(cis[rps[row]:rps[row + 1]], exp)


def test_exchange_lists_are_consistent():
    """Ghost rows sent by rank s to rank r must be exactly the rows r expects from s, in the same order."""
    case, size = Case(3, p=2, N=6), 8
    lays, infos = [], []
    for rank in range(size):
        g = case.product(rank=rank, size=size)
        lays.append((g, g.layout()))
    for r, (g, L) in enumerate(lays):
        lg, lr = L.lgmap(), L.localrow()
        nown = L.sizes()["nown"]
        glob_of_local = {}
        for gnode, row in zip(lg, lr):
            glob_of_local[row] = gnode
        for (peer, first, nrows, nblocks) in L.exchange(0):
            Lp = lays[peer][1]
            recv = Lp.exchange(1)
            idx = [i for i in range(len(recv)) if recv[i][0] == r]
            assert len(idx) == 1
            rows = Lp.recv_rows(idx[0], int(recv[idx[0]][2]))
            assert len(rows) == nrows and recv[idx[0]][3] == nblocks
            peer_start = None
            # global ids must match one to one
            lgp, lrp = Lp.lgmap(), Lp.localrow()
            own_glob = {row: gn for gn, row in zip(lgp, lrp) if row < Lp.sizes()["nown"]}
            for t in range(nrows):
                assert glob_of_local[first + t] == own_glob[rows[t]]


def test_c_abi_exports_every_declared_symbol():
    """The shared library must export every function include/petiga_cuda.h declares (no compute calls here)."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    L = pb.load_cuda()
    H = pb.load_host()
    names = re.findall(r"\b(petiga_(?:cuda|layout)_\w+)\s*\(", open(os.path.join(root, "include", "petiga_cuda.h")).read())
    assert len(set(names)) >= 30
    for n in set(names):
        assert hasattr(L, n), n
    hnames = re.findall(r"^PetscErrorCode\s+(\w+)\s*\(", open(os.path.join(root, "include", "petiga_host.h")).read(), re.M)
    assert len(set(hnames)) >= 50
    for n in set(hnames):
        assert hasattr(H, n), n
    assert L.petiga_cuda_version() == 100


def test_error_behaviour_matches_reference_checks():
    g = pb.IGA()
    with pytest.raises(pb.IGAError) as e:
        g.SetUp()                                   # "Must call IGASetDim() first" (petiga.c:1458)
    assert e.value.code == 73
    g.SetDim(2)
    with pytest.raises(pb.IGAError):
        g.SetDim(4)
    with pytest.raises(pb.IGAError) as e:
        g.AxisInitUniform(0, 2, 0)                  # petigaaxis.c:414
    assert e.value.code == 62
    with pytest.raises(pb.IGAError) as e:
        g.SetBoundaryValue(3, 0, 0, 1.0)            # IGAFormCheckArg (petigaform.c:95-99)
    assert e.value.code == 63
    # a host callback cannot be a device form
    CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)
    cb = CB(lambda p, K, F, ctx: 0)
    with pytest.raises(pb.IGAError) as e:
        g.SetFormRaw("SYSTEM", cb)
    assert e.value.code == 56


def test_no_cpu_fallback_without_gpu():
    """On a box without a GPU every device entry point must fail loudly, never compute on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    g = Case(2, p=2, N=4).product()
    g.SetForm("SYSTEM", "POISSON")
    with pytest.raises(pb.IGAError) as e:
        g.CreateMat()
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


def test_hot_kernel_register_budget():
    """Occupancy guard (ptxas -v logs of the in-tree build): the sum-factorised kernel of cfg 2 must keep 3 CTAs of 256
    threads per SM (<= 85 registers) and the separable kernel 4 (<= 64).  An inlined helper once pushed the former to 122
    registers and cost 37 % at cfg 2 without failing any parity test."""
    import os
    import re
    import petiga_b200
    libdir = petiga_b200.lib_dir()

    def regs(log, symbol_part):
        txt = open(os.path.join(libdir, log)).read()
        m = re.search(r"Compiling entry function '[^']*%s[^']*' for 'sm_100a'.*?Used (\d+) registers" % re.escape(symbol_part), txt, re.S)
        assert m, symbol_part
        return int(m.group(1))

    if not os.path.exists(os.path.join(libdir, "pc_quad2.ptxas.log")):
        pytest.skip("library not built in-tree")
    assert regs("pc_quad2.ptxas.log", "quad_sf_kernelILi3ELi3ELi1ELi4ELi1") <= 85
    assert regs("pc_quad2.ptxas.log", "quad_sf_kernelILi3ELi3ELi1ELi4ELi4") <= 64
    assert regs("pc_kron.ptxas.log", "kron_rows_kernelILi1ELi3ELi4") <= 64      # short pencils: 4 CTAs per SM
    assert regs("pc_kron.ptxas.log", "kron_rows_kernelILi1ELi3ELi3") <= 85      # long pencils: 3 CTAs per SM
    assert regs("pc_kron.ptxas.log", "kron_rows_kernelILi3ELi0ELi2") <= 128     # cfg 4 (BAIJ bs=3): 2 CTAs per SM (each warp stages a whole row in shared memory)
    # cfg 5, the third-generation kernels and cfg 3's vector kernel, held at their counts with CUDA 12.9
    assert regs("pc_quad.ptxas.log", "quad_kernelILi2ELi2ELi1ELi3E") <= 124     # cfg 5
    assert regs("pc_quad3.ptxas.log", "quad_sf3r_kernelILi0E") <= 168
    assert regs("pc_quad3.ptxas.log", "quad_sf3r_kernelILi1E") <= 168
    assert regs("pc_quad3.ptxas.log", "quad_sf3r_kernelILi2E") <= 162
    assert regs("pc_quad3.ptxas.log", "sf3_geom_kernel") <= 72
    assert regs("pc_quad3.ptxas.log", "quad_vec3_kernelILi4ELb0E") <= 48     # cfg 3


def test_functional_and_boundary_form_argument_checks():
    """Argument / state checks of the added drivers follow the reference (no GPU needed: they fire before any device work)."""
    import ctypes as C
    g = pb.IGA(2, 1)
    g.AxisInitUniform(0, 2, 4)
    g.AxisInitUniform(1, 2, 4)
    with pytest.raises(pb.IGAError) as e:
        g.ComputeErrorNorm(0)                       # IGACheckSetUp (petigacomp.c:164)
    assert e.value.code == 73
    g.SetUp()
    with pytest.raises(pb.IGAError) as e:
        g.ComputeErrorNorm(-1)                      # "Derivative index must be nonnegative" (petigacomp.c:170)
    assert e.value.code == 63
    for axis, side in ((3, 0), (-1, 0), (0, 2), (0, -1)):
        with pytest.raises(pb.IGAError) as e:
            g.SetBoundaryForm(axis, side, True)     # IGAFormCheckArg (petigaform.c:95-99)
        assert e.value.code == 63
    # a host callback cannot run on the device: PETSC_ERR_SUP, never a silent CPU fallback
    CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p)
    host_cb = CB(lambda p, U, n, S, ctx: 0)
    S = (C.c_double * 3)()
    rc = g.H.IGAComputeScalar(g.h, None, 3, S, host_cb, None)
    assert rc == 56
    EX = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p)
    out = (C.c_double * 1)()
    rc = g.H.IGAComputeErrorNorm(g.h, 0, None, EX(lambda p, k, V, ctx: 0), out, None)
    assert rc == 56


@pytest.mark.parametrize("p,C,periodic", [(2, 1, False), (3, 0, False), (3, 2, True), (4, 1, False)])
def test_axis_init_breaks_matches_oracle_tables(p, C, periodic):
    """IGAAxisInitBreaks (src/petigaaxis.c:323-382) on a graded mesh: knots, spans and the 1-D basis tables of the mirror are
    bit-identical to the oracle's built from the same knot vector; uniform breaks reproduce IGAAxisInitUniform bit for bit."""
    from oracle.oracle import OracleIGA
    breaks = np.array([0.0, 0.1, 0.25, 0.3, 0.55, 0.7, 0.85, 0.9, 1.0]) ** 1.5
    g = pb.IGA(1, 1)
    g.AxisInitBreaks(0, p, breaks, C, periodic)
    U = g.AxisGetKnots(0)
    s = p - C
    assert len(U) == 2 * (p + 1) + (len(breaks) - 2) * s                      # m + 1
    assert np.array_equal(np.unique(U[p:len(U) - p]), breaks)
    assert np.array_equal(g.AxisGetSpans(0), p + s * np.arange(len(breaks) - 1))
    g.SetUp()
    o = OracleIGA(1, 1)
    o.axis_knots(0, p, U, periodic)
    o.setup()
    to, tg = o.tables(0), g.tables(0)
    for key in ("U", "detJac", "weight", "point", "value"):
        assert np.array_equal(np.asarray(to[key]), np.asarray(tg[key])), key
    assert g.info()["nnp"][0] == o.info()["nnp"][0] and g.info()["nel"][0] == len(breaks) - 1
    # uniform breaks: identical to IGAAxisInitUniform when the breaks are the values it computes
    N = 7
    gu = pb.IGA(1, 1)
    gu.AxisInitUniform(0, p, N, 0.5, 2.0, C, periodic)
    Uu = gu.AxisGetKnots(0)
    gb = pb.IGA(1, 1)
    gb.AxisInitBreaks(0, p, np.unique(Uu[p:len(Uu) - p]), C, periodic)
    assert np.array_equal(gb.AxisGetKnots(0), Uu)
    with pytest.raises(pb.IGAError) as e:
        gb.AxisInitBreaks(0, p, [0.0, 0.5, 0.5, 1.0], C)        # strictly increasing (petigaaxis.c:337-339)
    assert e.value.code == 63


def test_headers_are_plain_c_and_the_readme_example_links(tmp_path):
    """include/*.h are the C boundary: a C99 translation unit (tests/csrc/readme_example.c, the README's snippet) must compile
    and link against the two shared libraries with gcc.  Without a GPU it stops at IGACreateMat with an error code (exit 3) --
    there is no CPU fallback; on a GPU box it runs through (exit 0)."""
    import shutil
    import subprocess
    import petiga_b200
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "readme_example")
    lib = petiga_b200.lib_dir()
    import torch
    for src in ("readme_example.c", "boundary_integral_example.c"):     # the second follows demo/BoundaryIntegral.c's main()
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "csrc", src),
                               "-L", lib, "-lpetiga_host", "-lpetiga_cuda", "-Wl,-rpath," + lib, "-o", exe])
        rc = subprocess.run([exe]).returncode
        assert rc == (0 if torch.cuda.is_available() else 3), (src, rc)


def test_handles_survive_ctypes_above_4gb():
    """ADVICE r1: Vec/Mat handles must cross ctypes as 64-bit pointers.  A bare Python int is converted to a C int and a
    pointer such as 0x55aa12345678 would arrive truncated; the wrappers keep c_void_p objects."""
    import ctypes as C
    from petiga_b200.iga import Mat, Vec, _vp
    big = 0x55AA12345678
    v = Vec(None, big)
    assert isinstance(v.h, C.c_void_p) and v.h.value == big
    labs = C.CDLL(None).labs
    labs.restype = C.c_long
    assert labs(v.h) == big              # what a library function receives when handed the wrapper's handle
    assert labs(_vp(C.c_void_p(big))) == big
    m = Mat.__new__(Mat)
    m.h = _vp(big)
    assert m.h.value == big


def test_glue_compiles():
    """SURVEY 7 step 2: the replacement bodies of the reference's drivers (integration/petiga_cuda_glue.c, written against the
    reference's <petiga.h>) are valid C against the C-ABI header; PETSc/PetIGA are absent, so a stub header stands in for them."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I" + os.path.join(root, "integration", "stub"),
                        "-I" + os.path.join(root, "include"), os.path.join(root, "integration", "petiga_cuda_glue.c")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
