"""Reference semantics of Bratu by collocation (PETIGA_FORM_BRATU_COLLOCATION), restated with numpy/scipy for the tests.

At the Greville point x_a of row a, with u = sum_b R_b U_b and v = sum_b R_b V_b over the row's (p+1)^dim columns:
  Function   F_a = -Lap u(x_a) - lambda e^u(x_a)              Jacobian   J_ab = -Lap R_b(x_a) - lambda e^u(x_a) R_b(x_a)
  IFunction  F_a = v(x_a) - Lap u(x_a) - lambda e^u(x_a)       IJacobian  J_ab = shift R_b(x_a) - Lap R_b(x_a) - lambda e^u(x_a) R_b(x_a)
A node with a boundary value (IGASetBoundaryValue) has F_a = U_a - value and an identity row.

Everything is in natural numbering.  The two operators B[a][b] = R_b(x_a) and L[a][b] = -Lap R_b(x_a) come from
tests/colloc_ref.py (identity, mapped and rational geometry), which is itself pinned against scipy's B-splines; this module
only adds the state.  tests/test_host_collocation_state.py pins it independently (scipy Kronecker products, an exact
solution, finite differences)."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spl

from tests.colloc_ref import assemble


def operators(axes, X=None, W=None):
    """(B, L): B[a][b] = R_b(x_a), L[a][b] = -Lap R_b(x_a), CSR with the collocation pattern (the same for both)."""
    B, _ = assemble(axes, "CONVTEST_COLLOCATION", (1.0, 0.0), X=X, W=W)     # c R_b - 0 Lap R_b
    L, _ = assemble(axes, "LAPLACE_COLLOCATION", (), X=X, W=W)
    assert np.array_equal(B.indptr, L.indptr) and np.array_equal(B.indices, L.indices)
    return B, L


def fixed_rows(axes, values):
    """(mask, value) of the natural rows that carry a boundary value; faces in axis/side order, the last one wins."""
    n = [a.nnp for a in axes]
    D = len(axes)
    node = np.indices(n[::-1]).reshape(D, -1)[::-1]
    mask = np.zeros(int(np.prod(n)), dtype=bool)
    fval = np.zeros(mask.size)
    for d in range(D):
        for s in range(2):
            if (d, s) in (values or {}):
                on = node[d] == (n[d] - 1 if s else 0)
                mask |= on
                fval[on] = values[(d, s)]
    return mask, fval


def residual(ops, U, lam, V=None, values=None, axes=None):
    """F(U) (Function), or the IFunction with V given; rows with a boundary value are U_a - value (needs axes)."""
    B, L = ops
    F = L @ U - lam * np.exp(B @ U)
    if V is not None:
        F = F + B @ V
    if values:
        mask, fval = fixed_rows(axes, values)
        F = np.where(mask, U - fval, F)
    return F


def jacobian(ops, U, lam, shift=0.0, values=None, axes=None):
    """J(U) (shift = 0: Jacobian; otherwise the IJacobian) as CSR with exactly the collocation pattern."""
    B, L = ops
    e = lam * np.exp(B @ U)
    rows = np.repeat(np.arange(B.shape[0]), np.diff(B.indptr))
    data = L.data + (shift - e[rows]) * B.data
    if values:
        mask, _ = fixed_rows(axes, values)
        data = np.where(mask[rows], (B.indices == rows).astype(np.float64), data)
    return sp.csr_matrix((data, B.indices.copy(), B.indptr.copy()), shape=B.shape)


def newton(ops, lam, values, axes, U0=None, rtol=1e-12, maxit=30):
    """Newton on F(U) = 0 with a direct solve per step until |F| <= rtol |F(U0)|; returns (U, list of |F| before every step)."""
    U = np.zeros(ops[0].shape[0]) if U0 is None else np.array(U0, dtype=np.float64)
    hist = []
    for _ in range(maxit):
        F = residual(ops, U, lam, values=values, axes=axes)
        hist.append(float(np.linalg.norm(F)))
        if hist[-1] <= rtol * hist[0]:
            break
        U = U - spl.spsolve(jacobian(ops, U, lam, values=values, axes=axes).tocsc(), F)
    return U, hist


def bratu_1d_exact(lam=1.0):
    """(theta, u): the smaller solution of u'' + lambda e^u = 0 on (0, 1), u(0) = u(1) = 0:
    u = -2 ln[cosh((x - 1/2) theta / 2) / cosh(theta / 4)], theta = sqrt(2 lambda) cosh(theta / 4)."""
    from scipy.optimize import brentq
    th = brentq(lambda t: t - np.sqrt(2 * lam) * np.cosh(t / 4), 0.1, 4.0, xtol=1e-15)
    return th, lambda x: -2 * np.log(np.cosh((np.asarray(x) - 0.5) * th / 2) / np.cosh(th / 4))
