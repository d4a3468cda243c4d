"""Reference semantics of isogeometric collocation (IGASetUseCollocation), restated with numpy/scipy for the tests.

What it computes, from the knot vectors alone:
  * the 1-D tables: Greville abscissae, FindSpan offsets and the basis functions with their derivatives there (The NURBS Book
    A2.1 / A2.3, in the operation order of the host mirror's tabulation, so the tables compare bit for bit);
  * the boxes of every rank: the Galerkin partition of the knot spans, element box = owned node box, ghost box = the union of
    the owned rows' stencils; the global numbering, the lgmap and the pattern (columns [offset, offset + p] per axis);
  * the collocation system in natural numbering for identity, mapped and rational geometry: K[a][b] = c N_b - k Lap_x N_b at
    x_a, F = fscale prod sin(pi x_i), identity rows (F = the value) on faces that carry a boundary value.
The matrix part is checked independently of this module against scipy's B-splines (tests/test_host_collocation.py)."""
import numpy as np
import scipy.sparse as sp


def bspline_ders(span, u, p, nd, U):
    """Basis functions and derivatives 0..nd at u (The NURBS Book A2.3); out[a][k], k < 5."""
    ndu = [[0.0] * 9 for _ in range(9)]
    left, right = [0.0] * 9, [0.0] * 9
    ndu[0][0] = 1.0
    for j in range(1, p + 1):
        left[j] = u - U[span + 1 - j]
        right[j] = U[span + j] - u
        saved = 0.0
        for r in range(j):
            ndu[j][r] = right[r + 1] + left[j - r]
            temp = ndu[r][j - 1] / ndu[j][r]
            ndu[r][j] = saved + right[r + 1] * temp
            saved = left[j - r] * temp
        ndu[j][j] = saved
    out = [[0.0] * 5 for _ in range(p + 1)]
    for r in range(p + 1):
        out[r][0] = ndu[r][p]
    a = [[0.0] * 9, [0.0] * 9]
    for r in range(p + 1):
        s1, s2 = 0, 1
        a[0][0] = 1.0
        for k in range(1, nd + 1):
            d = 0.0
            rk, pk = r - k, p - k
            if r >= k:
                a[s2][0] = a[s1][0] / ndu[pk + 1][rk]
                d = a[s2][0] * ndu[rk][pk]
            j1 = 1 if rk >= -1 else -rk
            j2 = k - 1 if r - 1 <= pk else p - r
            for j in range(j1, j2 + 1):
                a[s2][j] = (a[s1][j] - a[s1][j - 1]) / ndu[pk + 1][rk + j]
                d += a[s2][j] * ndu[rk + j][pk]
            if r <= pk:
                a[s2][k] = -a[s1][k - 1] / ndu[pk + 1][r]
                d += a[s2][k] * ndu[r][pk]
            out[r][k] = d
            s1, s2 = s2, s1
    fac = p
    for k in range(1, nd + 1):
        for r in range(p + 1):
            out[r][k] *= fac
        fac *= (p - k)
    return out


class Axis:
    """One parametric axis: knot vector U (open, non-periodic) of degree p."""

    def __init__(self, p, U):
        self.p, self.U = int(p), [float(u) for u in U]
        m = len(U) - 1
        n = m - p - 1
        self.nnp = n + 1
        self.span_off = [k - p for k in range(p, n + 1) if U[k] < U[k + 1]]   # Galerkin elements
        self.point, self.offset, self.value = [], [], []
        nd = min(p, 4)
        for i in range(self.nnp):
            u = 0.0
            for j in range(1, p + 1):
                u += self.U[i + j]
            u /= p
            k = n
            if u < self.U[n + 1]:
                k = p
                while k < n and self.U[k + 1] <= u:
                    k += 1
            self.point.append(u)
            self.offset.append(k - p)
            self.value.append(bspline_ders(k, u, p, nd, self.U))
        self.point = np.array(self.point)
        self.offset = np.array(self.offset, dtype=np.int64)
        self.value = np.array(self.value)          # [nnp][p+1][5]

    def boxes(self, P, r):
        """(es, ew, ls, lw, gs, gw) of processor coordinate r of P along this axis."""
        N, p = len(self.span_off), self.p
        ew = N // P + ((N % P) > r)
        es = r * (N // P) + (r if (N % P) > r else N % P)
        ef, el = es, es + ew - 1
        ls = self.span_off[ef]
        le = self.span_off[el + 1] if el < N - 1 else self.span_off[el] + p + 1
        lw = self.nnp - ls if r == P - 1 else le - ls
        gs = int(self.offset[ls])
        gw = int(self.offset[ls + lw - 1]) + p + 1 - gs
        return ls, lw, ls, lw, gs, gw


class Space:
    """A collocation IGA over `axes` (list of Axis, len = dim) distributed on `size` ranks with processor grid `grid`."""

    def __init__(self, axes, grid=None):
        self.axes, self.dim = axes, len(axes)
        self.grid = list(grid or [1] * self.dim) + [1] * (3 - self.dim)
        self.size = int(np.prod(self.grid))
        P = self.grid
        self.own = [np.zeros(a.nnp, dtype=np.int64) for a in axes]
        self.lbox = [[a.boxes(P[d], r)[2:4] for r in range(P[d])] for d, a in enumerate(axes)]
        for d, a in enumerate(axes):
            for r, (ls, lw) in enumerate(self.lbox[d]):
                self.own[d][ls:ls + lw] = r
        self.rank_start = [0]
        for q in range(self.size):
            c = self.coords(q)
            vol = 1
            for d in range(self.dim):
                vol *= self.lbox[d][c[d]][1]
            self.rank_start.append(self.rank_start[-1] + vol)

    def coords(self, q):
        P = self.grid
        return [q % P[0], (q // P[0]) % P[1], q // (P[0] * P[1])][:self.dim]

    def global_of(self, w):
        """global id of node w = (w0, w1, w2)"""
        r = [int(self.own[d][w[d]]) for d in range(self.dim)] + [0] * (3 - self.dim)
        q = r[0] + self.grid[0] * (r[1] + self.grid[1] * r[2])
        gid, mul = self.rank_start[q], 1
        for d in range(self.dim):
            ls, lw = self.lbox[d][r[d]]
            gid += (w[d] - ls) * mul
            mul *= lw
        return gid

    def info(self, rank):
        c = self.coords(rank)
        return [self.axes[d].boxes(self.grid[d], c[d]) for d in range(self.dim)]

    def _box_nodes(self, starts, widths):
        rng = [range(starts[d], starts[d] + widths[d]) for d in range(self.dim)]
        if self.dim == 1:
            return [(i,) for i in rng[0]]
        if self.dim == 2:
            return [(i, j) for j in rng[1] for i in rng[0]]
        return [(i, j, k) for k in rng[2] for j in rng[1] for i in rng[0]]

    def lgmap(self, rank):
        b = self.info(rank)
        return np.array([self.global_of(w) for w in self._box_nodes([x[4] for x in b], [x[5] for x in b])], dtype=np.int64)

    def pattern(self, rank):
        """owned rows of `rank` (local order) -> ascending global columns; (rowptr, colidx) of the node (BAIJ / dof 1) pattern"""
        b = self.info(rank)
        rowptr, colidx = [0], []
        for w in self._box_nodes([x[2] for x in b], [x[3] for x in b]):
            firsts = [int(self.axes[d].offset[w[d]]) for d in range(self.dim)]
            cols = self._box_nodes(firsts, [self.axes[d].p + 1 for d in range(self.dim)])
            colidx.extend(sorted(self.global_of(c) for c in cols))
            rowptr.append(len(colidx))
        return np.array(rowptr, dtype=np.int64), np.array(colidx, dtype=np.int64)


def _tensor(factors):
    """factors[d]: [n_d, e_d] -> [n_{D-1}..n_0, e_{D-1}..e_0] (rows natural, columns axis-0 fastest)"""
    D = len(factors)
    rows, cols = "ijk"[:D], "abc"[:D]
    spec = ",".join(rows[d] + cols[d] for d in range(D)) + "->" + rows[::-1] + cols[::-1]
    return np.einsum(spec, *factors)


def _sym_pairs(D):
    return [(a, b) for a in range(D) for b in range(a, D)]


def assemble(axes, form="LAPLACE_COLLOCATION", params=(), X=None, W=None, values=None):
    """The collocation system in natural numbering (scipy CSR, F).  X: natural [..][dim] or None; W: natural weights or None;
    values: {(axis, side): value} of IGASetBoundaryValue (identity rows, applied in axis/side order: the last face wins)."""
    D = len(axes)
    n = [a.nnp for a in axes]
    e = [a.p + 1 for a in axes]
    V = [a.value for a in axes]
    comp = lambda d, k: V[d][:, :, k]     # noqa: E731
    N0 = _tensor([comp(d, 0) for d in range(D)])
    N1 = [_tensor([comp(d, 1 if d == c else 0) for d in range(D)]) for c in range(D)]
    N2 = {}
    for a, b in _sym_pairs(D):
        N2[(a, b)] = _tensor([comp(d, (d == a) + (d == b)) for d in range(D)])
    # gather of node data at the columns of every row
    idx = [axes[d].offset[:, None] + np.arange(e[d])[None, :] for d in range(D)]

    def gather(arr):        # arr natural [n_{D-1}..n_0, ...] -> [rows..., cols..., ...]
        ix = []
        for d in range(D):  # array axis D-1-d holds axis d
            shape = [1] * (2 * D)
            shape[D - 1 - d] = n[d]
            shape[2 * D - 1 - d] = e[d]
            ix.append(idx[d].reshape(shape))
        return arr[tuple(ix[::-1])]
    csum = tuple(range(D, 2 * D))
    R0, R1, R2 = N0, N1, N2
    if W is not None:
        Wc = gather(np.asarray(W, dtype=np.float64).reshape(n[::-1]))
        W0 = (Wc * N0).sum(axis=csum, keepdims=True)
        W1 = [(Wc * N1[c]).sum(axis=csum, keepdims=True) for c in range(D)]
        W2 = {s: (Wc * N2[s]).sum(axis=csum, keepdims=True) for s in N2}
        R0 = Wc * N0 / W0
        R1 = [(Wc * N1[c] - R0 * W1[c]) / W0 for c in range(D)]
        R2 = {(a, b): (Wc * N2[(a, b)] - R0 * W2[(a, b)] - R1[a] * W1[b] - R1[b] * W1[a]) / W0 for a, b in N2}
    x = [None] * D
    if X is not None:
        Xc = gather(np.asarray(X, dtype=np.float64).reshape(tuple(n[::-1]) + (D,)))
        X0 = [(Xc[..., i] * R0).sum(axis=csum) for i in range(D)]
        X1 = np.stack([np.stack([(Xc[..., i] * R1[c]).sum(axis=csum) for c in range(D)], -1) for i in range(D)], -2)  # [rows, i, d]
        X2 = {s: np.stack([(Xc[..., i] * R2[s]).sum(axis=csum) for i in range(D)], -1) for s in R2}            # [rows, i]
        E = np.linalg.inv(X1)                                     # E[.., d, i] = du_d / dx_i
        g = {(a, b): (E[..., a, :] * E[..., b, :]).sum(-1) for a, b in R2}
        hk = sum((1.0 if a == b else 2.0) * X2[(a, b)] * g[(a, b)][..., None] for a, b in R2)   # [rows, k]
        h = [-(E[..., c, :] * hk).sum(-1) for c in range(D)]
        ex = tuple([slice(None)] * D + [None] * D)
        lap = sum((1.0 if a == b else 2.0) * R2[(a, b)] * g[(a, b)][ex] for a, b in R2) + sum(R1[c] * h[c][ex] for c in range(D))
        x = X0
    else:
        lap = sum(R2[(c, c)] for c in range(D))
        grids = np.meshgrid(*[a.point for a in axes[::-1]], indexing="ij")    # [n_{D-1}..n_0]
        x = grids[::-1]
    c, k = (0.0, 1.0) if form == "LAPLACE_COLLOCATION" else (float(params[0]), float(params[1]))
    fscale = 0.0 if form == "LAPLACE_COLLOCATION" else c + k * D * np.pi ** 2
    K = c * R0 - k * lap                                          # [rows..., cols...]
    F = fscale * np.prod([np.sin(np.pi * xi) for xi in x], axis=0) if fscale != 0.0 else np.zeros(tuple(n[::-1]))
    nrow = int(np.prod(n))
    ncol = int(np.prod(e))
    K = K.reshape(nrow, ncol)
    F = np.array(F, dtype=np.float64).reshape(nrow)
    # natural column ids
    colnat = np.zeros([1] * D + [1] * D, dtype=np.int64)
    mul = 1
    for d in range(D):
        shape = [1] * (2 * D)
        shape[D - 1 - d] = n[d]
        shape[2 * D - 1 - d] = e[d]
        colnat = colnat + idx[d].reshape(shape) * mul
        mul *= n[d]
    colnat = np.broadcast_to(colnat, tuple(n[::-1]) + tuple(e[::-1])).reshape(nrow, ncol)
    rows = np.repeat(np.arange(nrow), ncol)
    if values:
        node = np.indices(n[::-1]).reshape(D, -1)[::-1]           # node[d][row]
        fixed = np.zeros(nrow, dtype=bool)
        fval = np.zeros(nrow)
        for d in range(D):
            for s in range(2):
                if (d, s) in values:
                    on = node[d] == (n[d] - 1 if s else 0)
                    fixed |= on
                    fval[on] = values[(d, s)]
        K = np.where(fixed[:, None], (colnat == np.arange(nrow)[:, None]).astype(np.float64), K)
        F = np.where(fixed, fval, F)
    A = sp.csr_matrix((K.reshape(-1), (rows, colnat.reshape(-1))), shape=(nrow, nrow))
    A.sort_indices()
    return A, F


def scipy_laplace_kron(axes, values_on_all_faces=True):
    """-Lap by Kronecker sums of 1-D scipy collocation matrices (BSpline.design_matrix and its second derivative at the
    Greville points), natural order, identity rows on the boundary: an independent statement of the identity-geometry matrix."""
    from scipy.interpolate import BSpline
    B0, B2 = [], []
    for a in axes:
        U, p = np.array(a.U), a.p
        g = np.array([np.mean(U[i + 1:i + p + 1]) for i in range(a.nnp)])
        b0 = BSpline.design_matrix(g, U, p).toarray()
        b2 = np.zeros_like(b0)
        for j in range(a.nnp):
            cvec = np.zeros(a.nnp)
            cvec[j] = 1.0
            b2[:, j] = BSpline(U, cvec, p).derivative(2)(g)
        B0.append(sp.csr_matrix(b0))
        B2.append(sp.csr_matrix(b2))
    D = len(axes)
    A = None
    for c in range(D):
        term = None
        for d in range(D - 1, -1, -1):
            M = B2[d] if d == c else B0[d]
            term = M if term is None else sp.kron(term, M)
        A = term if A is None else A + term
    A = (-A).tolil()
    if values_on_all_faces:
        n = [a.nnp for a in axes]
        node = np.indices(n[::-1]).reshape(D, -1)[::-1]
        bnd = np.zeros(A.shape[0], dtype=bool)
        for d in range(D):
            bnd |= (node[d] == 0) | (node[d] == n[d] - 1)
        for r in np.where(bnd)[0]:
            A.rows[r] = [r]
            A.data[r] = [1.0]
    A = A.tocsr()
    A.sort_indices()
    return A


def l2_error_2d(axes, coef):
    """L2 error of the 2-D spline with natural coefficients `coef` against prod sin(pi x_i) (Gauss rule of p+2 points per span)."""
    from scipy.interpolate import BSpline
    Bs, ws = [], []
    for a in axes:
        U = np.array(a.U)
        xg, wg = np.polynomial.legendre.leggauss(a.p + 2)
        br = np.unique(U)
        pts = np.concatenate([(br[i + 1] - br[i]) / 2 * xg + (br[i + 1] + br[i]) / 2 for i in range(len(br) - 1)])
        wts = np.concatenate([(br[i + 1] - br[i]) / 2 * wg for i in range(len(br) - 1)])
        Bs.append((BSpline.design_matrix(pts, U, a.p).toarray(), pts))
        ws.append(wts)
    C = np.asarray(coef).reshape(axes[1].nnp, axes[0].nnp)      # [j][i]
    uh = Bs[1][0] @ C @ Bs[0][0].T                               # [qy][qx]
    ue = np.sin(np.pi * Bs[1][1])[:, None] * np.sin(np.pi * Bs[0][1])[None, :]
    return float(np.sqrt(np.sum(ws[1][:, None] * ws[0][None, :] * (uh - ue) ** 2)))
