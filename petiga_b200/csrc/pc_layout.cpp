// pc_layout.cpp -- see pc_layout.h
#include "pc_layout.h"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace pc {

// IGA_NextKnot: src/petigaaxis.c:482-494
static int next_knot(int m, const double* U, int k, int direction) {
  if (direction >= 0) {
    if (k < 0) return 0;
    for (int j = k + 1; j < m; j++)
      if (U[j] > U[k]) return j;
    return m;
  }
  if (k > m) return m;
  for (int j = k - 1; j > 0; j--)
    if (U[j] < U[k]) return j;
  return 0;
}

// Stencil(): src/petigamat.c:197-233.  Collocation branch: the p+1 basis functions that do not vanish at the row's point,
// [offset[i], offset[i] + p] of the collocation table.
static void stencil(const AxisLayout& a, const double* U, const int* offset, int collocation, int i, int& first, int& last) {
  if (collocation) {
    first = offset[i];
    last = offset[i] + a.p;
    return;
  }
  const int p = a.p, m = a.m, n = m - p - 1;
  first = next_knot(m, U, i, +1) - p - 1;
  last = next_knot(m, U, i + p + 1, -1);
  if (!a.periodic) {
    if (i <= p) first = 0;
    if (i >= n - p) last = n;
  } else if (i == 0) {
    int k = n + 1, j = next_knot(m, U, k, +1), s = j - k, C = p - s, nnp = n - C;
    k = next_knot(m, U, nnp, +1) - nnp;
    first = k - p - 1;
  }
}

static inline int wrap(int i, int n) { return i < 0 ? n + i : (i >= n ? i % n : i); }  // petigagrid.c:160-163

static int fail(Layout& L, int code, const std::string& msg) {
  L.error = msg;
  return code;
}

int build_layout(const petiga_cuda_space& sp, int rank, int nranks, Layout& L) {
  L = Layout();
  L.dim = sp.dim;
  L.dof = sp.dof;
  L.rank = rank;
  L.nranks = nranks;
  L.collocation = sp.collocation ? 1 : 0;
  if (sp.dim < 1 || sp.dim > 3) return fail(L, PETIGA_CUDA_ERR_ARG, "dim must be in [1,3]");
  if (sp.dof < 1 || sp.dof > 64) return fail(L, PETIGA_CUDA_ERR_ARG, "dof must be in [1,64]");
  int nprocs = 1;
  for (int d = 0; d < 3; d++) nprocs *= sp.proc_sizes[d];
  if (nprocs != nranks) return fail(L, PETIGA_CUDA_ERR_ARG, "prod(proc_sizes) != nranks");
  {  // rank -> (i,j,k), i fastest: src/petigapart.c:161-166
    int rr = rank;
    for (int d = 0; d < 3; d++) {
      int c = rr % sp.proc_sizes[d];
      rr /= sp.proc_sizes[d];
      if (c != sp.proc_ranks[d]) return fail(L, PETIGA_CUDA_ERR_ARG, "proc_ranks inconsistent with rank");
    }
  }
  for (int d = 0; d < 3; d++) {
    AxisLayout& a = L.ax[d];
    a.p = sp.p[d]; a.m = sp.m[d]; a.nel = sp.nel[d]; a.nnp = sp.nnp[d]; a.periodic = sp.periodic[d]; a.nqp = sp.nqp1[d];
    a.P = sp.proc_sizes[d]; a.r = sp.proc_ranks[d];
    if (a.p < 0 || a.p > kMaxP) return fail(L, PETIGA_CUDA_ERR_SUP, "degree must be <= 8 on the device path");
    if (d >= sp.dim && (a.p != 0 || a.nel != 1 || a.nnp != 1)) return fail(L, PETIGA_CUDA_ERR_ARG, "unused axes must be reset axes");
    if (!sp.U[d] || !sp.offset[d]) return fail(L, PETIGA_CUDA_ERR_ARG, "missing axis tables");
    const double* U = sp.U[d];
    const int* off = sp.offset[d];
    // The partition runs on the Galerkin elements (the knot spans).  A collocation table holds one entry per node instead, so
    // the Galerkin offsets are recovered from the knot vector: span k of every nonzero knot interval, offset k - p.
    std::vector<int> span_off;
    if (L.collocation) {
      if (a.periodic) return fail(L, PETIGA_CUDA_ERR_SUP, "collocation: periodic axes are not supported on the device path");
      if (d < sp.dim && a.p < 2) return fail(L, PETIGA_CUDA_ERR_SUP, "collocation: degree must be in [2,8] (second derivatives at the points)");
      for (int k = a.p; k <= a.m - a.p - 1; k++)
        if (U[k] < U[k + 1]) span_off.push_back(k - a.p);
      if (span_off.empty()) return fail(L, PETIGA_CUDA_ERR_ARG, "collocation: knot vector without a nonzero span");
      // nel may be the table length (IGABasis.nel = nnp) or the axis's element count (IGAAxis.nel); the tables always hold nnp
      if ((a.nel != a.nnp && a.nel != (int)span_off.size()) || a.nqp != 1)
        return fail(L, PETIGA_CUDA_ERR_ARG, "collocation: nel must be nnp (table length) or the number of knot spans, and nqp 1");
      a.nel = a.nnp;
      for (int i = 0; i < a.nnp; i++)
        if (off[i] < 0 || off[i] + a.p >= a.nnp) return fail(L, PETIGA_CUDA_ERR_ARG, "collocation: offset table out of range");
    }
    const int* eoff = L.collocation ? span_off.data() : off;
    const int nelp = L.collocation ? (int)span_off.size() : a.nel;
    a.first.resize(a.nnp); a.last.resize(a.nnp); a.own.assign(a.nnp, -1);
    for (int i = 0; i < a.nnp; i++) stencil(a, U, off, L.collocation, i, a.first[i], a.last[i]);
    a.box_es.resize(a.P); a.box_ew.resize(a.P); a.box_ls.resize(a.P); a.box_lw.resize(a.P); a.box_gs.resize(a.P); a.box_gw.resize(a.P);
    if (nelp < a.P) return fail(L, PETIGA_CUDA_ERR_ARG, "partition too fine");
    for (int r = 0; r < a.P; r++) {  // IGA_Dist1D (petigapart.c:170-176) + node boxes (petiga.c:1160-1209)
      int N = nelp, ew = N / a.P + ((N % a.P) > r), es = r * (N / a.P) + (((N % a.P) > r) ? r : (N % a.P));
      int efirst = es, elast = es + ew - 1;
      int gs = eoff[efirst], ge = eoff[elast] + a.p + 1, ls = gs;
      int le = (elast < N - 1) ? eoff[elast + 1] : eoff[elast] + a.p + 1;
      int lw = le - ls;
      if (r == a.P - 1) lw = a.nnp - ls;
      if (L.collocation) {   // element box = owned node box; ghost box = the stencils of the owned rows
        es = ls; ew = lw;
        if (lw < 1) return fail(L, PETIGA_CUDA_ERR_SUP, "a rank owns no nodes along an axis");
        gs = a.first[ls]; ge = a.last[ls + lw - 1] + 1;
      }
      a.box_es[r] = es; a.box_ew[r] = ew; a.box_ls[r] = ls; a.box_lw[r] = lw; a.box_gs[r] = gs; a.box_gw[r] = ge - gs;
      for (int i = ls; i < ls + lw; i++)
        if (i >= 0 && i < a.nnp) a.own[i] = r;
    }
    for (int i = 0; i < a.nnp; i++)
      if (a.own[i] < 0) return fail(L, PETIGA_CUDA_ERR_ARG, "node without owner (empty rank box?)");
    a.es = a.box_es[a.r]; a.ew = a.box_ew[a.r]; a.ls = a.box_ls[a.r]; a.lw = a.box_lw[a.r]; a.gs = a.box_gs[a.r]; a.gw = a.box_gw[a.r];
    if (a.es != sp.elem_start[d] || a.ew != sp.elem_width[d] || a.ls != sp.node_lstart[d] || a.lw != sp.node_lwidth[d] ||
        a.gs != sp.node_gstart[d] || a.gw != sp.node_gwidth[d])
      return fail(L, PETIGA_CUDA_ERR_ARG, "boxes in petiga_cuda_space disagree with IGA_Distribute arithmetic");
    if (a.lw < 1) return fail(L, PETIGA_CUDA_ERR_SUP, "a rank owns no nodes along an axis");
    a.wrapped.resize(a.gw); a.W.resize(a.gw); a.lo.resize(a.gw); a.simple.assign(a.gw, 1); a.seg.assign((size_t)a.gw * kMaxW, 0);
    for (int g = 0; g < a.gw; g++) {
      int w = wrap(a.gs + g, a.nnp);
      a.wrapped[g] = w;
      int W = a.last[w] - a.first[w] + 1;
      if (W < 1 || W > kMaxW) return fail(L, PETIGA_CUDA_ERR_SUP, "1-D stencil wider than 2p+1");
      a.W[g] = W;
      a.lo[g] = w - a.first[w];
      int key_own[kMaxW], key_idx[kMaxW];
      for (int c = 0; c < W; c++) {
        int wc = wrap(a.first[w] + c, a.nnp);
        key_idx[c] = wc;
        key_own[c] = a.own[wc];
      }
      for (int c = 0; c < W; c++) {
        int B = 0, S = 0, Lc = 0;
        for (int e = 0; e < W; e++) {
          if (e != c && key_idx[e] == key_idx[c])
            return fail(L, PETIGA_CUDA_ERR_SUP, "periodic axis too short: stencil wraps onto itself");
          if (key_own[e] < key_own[c]) B++;
          if (key_own[e] == key_own[c]) { S++; if (key_idx[e] < key_idx[c]) Lc++; }
        }
        a.seg[(size_t)g * kMaxW + c] = (uint32_t)B | ((uint32_t)S << 8) | ((uint32_t)Lc << 16);
        if (B != 0 || S != W || Lc != c) a.simple[g] = 0;
      }
    }
  }
  const AxisLayout &A0 = L.ax[0], &A1 = L.ax[1], &A2 = L.ax[2];
  // global numbering: rank r owns [rank_start[r], rank_start[r+1])
  L.rank_start.resize(nranks + 1);
  L.rank_start[0] = 0;
  for (int q = 0; q < nranks; q++) {
    int c0 = q % A0.P, c1 = (q / A0.P) % A1.P, c2 = q / (A0.P * A1.P);
    int64_t vol = (int64_t)A0.box_lw[c0] * A1.box_lw[c1] * A2.box_lw[c2];
    if ((int64_t)L.rank_start[q] + vol > INT32_MAX) return fail(L, PETIGA_CUDA_ERR_SUP, "more than 2^31 nodes");
    L.rank_start[q + 1] = L.rank_start[q] + (int)vol;
  }
  auto global_of = [&](int w0, int w1, int w2) {
    int r0 = A0.own[w0], r1 = A1.own[w1], r2 = A2.own[w2];
    int q = r0 + A0.P * (r1 + A1.P * r2);
    return L.rank_start[q] + (w0 - A0.box_ls[r0]) + A0.box_lw[r0] * ((w1 - A1.box_ls[r1]) + A1.box_lw[r1] * (w2 - A2.box_ls[r2]));
  };
  const int ng = A0.gw * A1.gw * A2.gw;
  L.nown = A0.lw * A1.lw * A2.lw;
  L.lgmap.resize(ng);
  L.localrow.resize(ng);
  std::vector<int> ghosts;  // global ids of the nodes I see but do not own
  const int my_lo = L.rank_start[rank], my_hi = L.rank_start[rank + 1];
  for (int k = 0, g = 0; k < A2.gw; k++)
    for (int j = 0; j < A1.gw; j++)
      for (int i = 0; i < A0.gw; i++, g++) {
        int gid = global_of(A0.wrapped[i], A1.wrapped[j], A2.wrapped[k]);
        L.lgmap[g] = gid;
        if (gid < my_lo || gid >= my_hi) ghosts.push_back(gid);
      }
  std::sort(ghosts.begin(), ghosts.end());
  ghosts.erase(std::unique(ghosts.begin(), ghosts.end()), ghosts.end());
  std::vector<int> foreign;   // collocation: every row is computed by the rank that owns its point, so the nodes of other
  if (L.collocation) foreign.swap(ghosts);   // ranks are state only (the halo), never rows
  L.nghostrows = (int)ghosts.size();
  L.nloc = L.nown + L.nghostrows;
  for (int g = 0; g < ng; g++) {
    int gid = L.lgmap[g];
    if (gid >= my_lo && gid < my_hi) L.localrow[g] = gid - my_lo;
    else if (L.collocation) L.localrow[g] = -1;
    else L.localrow[g] = L.nown + (int)(std::lower_bound(ghosts.begin(), ghosts.end(), gid) - ghosts.begin());
  }
  if (L.collocation) {
    L.nstate = L.nown + (int)foreign.size();
    L.staterow.resize(ng);
    for (int g = 0; g < ng; g++) {
      const int gid = L.lgmap[g];
      L.staterow[g] = (gid >= my_lo && gid < my_hi) ? gid - my_lo
                                                    : L.nown + (int)(std::lower_bound(foreign.begin(), foreign.end(), gid) - foreign.begin());
    }
  }
  // per-row node coordinates and widths, row bases
  for (int d = 0; d < 3; d++) { L.rowW[d].assign(L.nloc, 0); L.rowG[d].assign(L.nloc, 0); }
  for (int k = 0, g = 0; k < A2.gw; k++)
    for (int j = 0; j < A1.gw; j++)
      for (int i = 0; i < A0.gw; i++, g++) {
        int r = L.localrow[g];
        if (r < 0) continue;
        L.rowW[0][r] = A0.W[i]; L.rowW[1][r] = A1.W[j]; L.rowW[2][r] = A2.W[k];
        L.rowG[0][r] = A0.wrapped[i]; L.rowG[1][r] = A1.wrapped[j]; L.rowG[2][r] = A2.wrapped[k];
      }
  L.rowbase.resize((size_t)L.nloc + 1);
  L.rowbase[0] = 0;
  for (int r = 0; r < L.nloc; r++) {
    if (L.rowW[0][r] == 0) return fail(L, PETIGA_CUDA_ERR_ARG, "internal: owned node outside the ghost box");
    L.rowbase[r + 1] = L.rowbase[r] + (int64_t)L.rowW[0][r] * L.rowW[1][r] * L.rowW[2][r];
  }
  L.nnz_own = L.rowbase[L.nown];
  L.nnz_loc = L.rowbase[L.nloc];
  // ghost rows (collocation: foreign state nodes) -> owners (contiguous runs because both lists are sorted by global id)
  auto owner_runs = [&](const std::vector<int>& ids, bool rows, std::vector<Layout::Peer>& out) {
    const int n = (int)ids.size();
    for (int t = 0; t < n;) {
      int q = (int)(std::upper_bound(L.rank_start.begin(), L.rank_start.end(), ids[t]) - L.rank_start.begin()) - 1;
      int t1 = t;
      while (t1 < n && ids[t1] < L.rank_start[q + 1]) t1++;
      Layout::Peer pr;
      pr.rank = q; pr.first_row = L.nown + t; pr.nrows = t1 - t;
      pr.first_block = rows ? L.rowbase[L.nown + t] : 0; pr.nblocks = rows ? L.rowbase[L.nown + t1] - pr.first_block : 0;
      out.push_back(pr);
      t = t1;
    }
  };
  owner_runs(ghosts, true, L.send);
  owner_runs(foreign, false, L.state_send);
  // rows other ranks hold for me (collocation: read as state), in *their* order (ascending global id == ascending local index here)
  std::vector<Layout::Recv>& held = L.collocation ? L.state_recv : L.recv;
  for (int s = 0; s < nranks; s++) {
    if (s == rank) continue;
    int c[3] = {s % A0.P, (s / A0.P) % A1.P, s / (A0.P * A1.P)};
    std::vector<int> mine[3];
    bool any = true;
    for (int d = 0; d < 3; d++) {
      const AxisLayout& a = L.ax[d];
      for (int g = 0; g < a.box_gw[c[d]]; g++) {
        int w = wrap(a.box_gs[c[d]] + g, a.nnp);
        if (a.own[w] == a.r) mine[d].push_back(w);
      }
      std::sort(mine[d].begin(), mine[d].end());
      mine[d].erase(std::unique(mine[d].begin(), mine[d].end()), mine[d].end());
      if (mine[d].empty()) { any = false; break; }
    }
    if (!any) continue;
    Layout::Recv rv;
    rv.rank = s; rv.nblocks = 0;
    for (int w2 : mine[2]) for (int w1 : mine[1]) for (int w0 : mine[0]) {
      int row = (w0 - A0.ls) + A0.lw * ((w1 - A1.ls) + A1.lw * (w2 - A2.ls));
      rv.rows.push_back(row);
      if (!L.collocation) rv.nblocks += L.rowbase[row + 1] - L.rowbase[row];
    }
    held.push_back(std::move(rv));
  }
  return 0;
}

int host_pattern(const Layout& L, int block, std::vector<int>& rowptr, std::vector<int>& colidx) {
  const AxisLayout &A0 = L.ax[0], &A1 = L.ax[1], &A2 = L.ax[2];
  const int bs = block ? 1 : L.dof;
  if (L.nnz_own * bs * bs > INT32_MAX) return PETIGA_CUDA_ERR_SUP;
  rowptr.assign((size_t)L.nown * bs + 1, 0);
  colidx.assign((size_t)L.nnz_own * bs * bs, -1);
  for (int k = 0, row = 0; k < A2.lw; k++)
    for (int j = 0; j < A1.lw; j++)
      for (int i = 0; i < A0.lw; i++, row++) {
        int g[3] = {A0.ls + i - A0.gs, A1.ls + j - A1.gs, A2.ls + k - A2.gs};
        int Wi = A0.W[g[0]], Wj = A1.W[g[1]], Wk = A2.W[g[2]], W = Wi * Wj * Wk;
        int64_t base = L.rowbase[row];
        for (int r = 0; r < bs; r++) rowptr[(size_t)row * bs + r + 1] = (int)(base * bs * bs + (int64_t)(r + 1) * W * bs);
        for (int ck = 0; ck < Wk; ck++) for (int cj = 0; cj < Wj; cj++) for (int ci = 0; ci < Wi; ci++) {
          int c[3] = {ci, cj, ck};
          int64_t pos = col_position(L, g, c);
          int w0 = wrap(A0.first[A0.wrapped[g[0]]] + ci, A0.nnp), w1 = wrap(A1.first[A1.wrapped[g[1]]] + cj, A1.nnp),
              w2 = wrap(A2.first[A2.wrapped[g[2]]] + ck, A2.nnp);
          int r0 = A0.own[w0], r1 = A1.own[w1], r2 = A2.own[w2];
          int q = r0 + A0.P * (r1 + A1.P * r2);
          int gid = L.rank_start[q] + (w0 - A0.box_ls[r0]) + A0.box_lw[r0] * ((w1 - A1.box_ls[r1]) + A1.box_lw[r1] * (w2 - A2.box_ls[r2]));
          for (int r = 0; r < bs; r++)
            for (int cc = 0; cc < bs; cc++) colidx[(size_t)(base * bs * bs + (int64_t)r * W * bs + pos * bs + cc)] = gid * bs + cc;
        }
      }
  return 0;
}

}  // namespace pc
