// pc_kron.cu -- the separable ("Kronecker") assembly path.
//
// When the geometry map is the identity and the form's coefficient tensor is constant (Poisson, Laplace,
// mass/L2, elasticity: every linear BASELINE config), the sum over elements of the element matrices of the
// reference's quadrature loop (src/petigaksp.c:149-202) factorises over the axes:
//
//   A[(A,i),(B,j)] = sum_{al,be} C[i][j][al][be] * prod_d M_d^{(r_d,s_d)}[A_d][B_d],
//   M_d^{(r,s)}[a][b] = sum_{e in supp(a) & supp(b)} sum_q w_q J_e N_a^{(r)}(u_q) N_b^{(s)}(u_q)      (1-D, banded)
//
// with r_d = 1 iff component al is the derivative along axis d.  So every CSR value can be *written once*
// from three tiny 1-D tables: no per-element work, no zeroing pass, no atomics, no ghost-row exchange (each rank
// writes exactly its owned rows).  The kernel is bound by the 8 bytes it stores per nonzero (HBM roofline).
//
// The reference's per-element Dirichlet/Neumann fix-up (IGAElementFixSystem, src/petigaelem.c:1360-1389) is
// reproduced in aggregate: a boundary node is fixed in every element that contains it, so after ADD_VALUES
//   fixed row    -> zero, diagonal = number of elements containing the node, rhs = that count * value
//   fixed column -> zero, its unfixed entry times the value is subtracted from the row's rhs
//   loads        -> rhs += value * sum over the face elements of BoundaryArea (petigaelem.c:1118-1131)
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "pc_plan.h"

namespace pc {

namespace {

constexpr int kMaxTerms = 40;
constexpr int kKronP = 4;               // the separable path keeps its pencil tables in static shared memory: degree <= 4
constexpr int kMaxWW = (2 * kKronP + 1) * (2 * kKronP + 1);
constexpr int kStageCap = 32 * 16 + 192;         // dof > 1: doubles of dynamic shared memory per warp (one p = 2 BAIJ row of 125 3x3 blocks + its coefficients)

struct KronTerm { unsigned char ij, rs0, rs1, rs2; double c; };
struct KronVTerm { unsigned char i, r0, r1, r2; double c; };

struct KronParams {
  const double* M[3];     // [4][nnp][kMaxW]  1-D matrices, rs = 2*r+s major
  const double* mv[3];    // [2][nnp]         1-D load vectors  sum_e sum_q wJ N^{(r)}
  const int* nsup[3];     // [nnp]            elements containing basis i
  const double* lsum[3];  // [nnp]            sum over those elements of detJac/nen
  const double* rsum[3];  // [4][nnp]         row sums of M (all columns of the row)
  const int* first[3];    // [nnp]
  const int* Wg[3];       // [gw] widths by ghost coordinate
  const int* lo[3];       // [gw]
  const uint32_t* seg[3]; // [gw][kMaxW]
  const int* simp[3];     // [gw] columns of this 1-D row are already in storage order
  int ls[3], lw[3], gs[3], nnp[3], periodic[3];
  const int64_t* rowbase;
  const int* localrow;    // ghost box -> local row (for the fix table)
  const double* fixtable; // [ghost box][dof] or NULL
  int gw[3];
  int dim, dof, block, slot, simple, wfull0;
  int nterms, nvterms, rsmask0;
  int fast_lo, fast_hi;   // axis-0 local row range [lo,hi) of full-width, storage-ordered, unconstrained rows (multiple of 4 long)
  int rsmask_ij[9];       // per (i,j) block: which axis-0 order pairs occur
  int ncombo;             // distinct (axis-0 order pair, block entry) combinations; terms are sorted by combination
  unsigned char combo_rs0[36], combo_ij[36], combo_first[37];
  signed char slotA[9], slotB[9];   // ... as (at most) two order-pair indices per block entry, -1 = none; two_slot = 0 when an entry has more
  int two_slot;
  int minb_rows;          // scalar case: pencils at least this long run the 3-CTA (80-register) instantiation
  int bulk;               // dof 1 fast passes: rows staged in shared memory and written by cp.async.bulk (TMA) stores
  KronTerm terms[kMaxTerms];
  KronVTerm vterms[8];
  FixSide bc[3][2];
  int any_bc;
  double* values;
  double* rhs;
};

__device__ __forceinline__ int wrapi(int i, int n) { return i < 0 ? n + i : (i >= n ? i % n : i); }

// 1-D tables: one thread per (axis-local) output; deterministic summation order (elements ascending)
__global__ void kron_1d_kernel(DevAxis ax, const int* __restrict__ first, double* __restrict__ M, double* __restrict__ mv,
                               int* __restrict__ nsup, double* __restrict__ lsum) {
  const int nnp = ax.nnp, nen = ax.nen, nq = ax.nqp;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = nnp * kMaxW * 4;
  if (t < total) {
    const int rs = t / (nnp * kMaxW), rem = t - rs * nnp * kMaxW, i = rem / kMaxW, c = rem - i * kMaxW;
    const int r = rs >> 1, s = rs & 1;
    const int col = wrapi(first[i] + c, nnp);
    double acc = 0.0;
    // a 1-D row has at most 2p+1 columns; beyond them (the table rows are kMaxW wide) and, without periodicity, beyond the last
    // node the entry is zero -- a wrapped index must not fold back into the row's support on short axes
    const bool exists = c <= 2 * ax.p && (ax.periodic || first[i] + c < nnp);
    for (int e = 0; e < (exists ? ax.nel : 0); e++) {
      int a = -1, b = -1;
      for (int l = 0; l < nen; l++) {
        int node = wrapi(ax.offset[e] + l, nnp);
        if (node == i) a = l;
        if (node == col) b = l;
      }
      // the unwrapped column must be the one this element sees: first+c - i == b - a  (guards short periodic axes)
      if (a < 0 || b < 0) continue;
      const double J = ax.detJac[e];
      double se = 0.0;
      for (int q = 0; q < nq; q++) {
        const double* va = ax.value + ((size_t)(e * nq + q) * nen + a) * 5;
        const double* vb = ax.value + ((size_t)(e * nq + q) * nen + b) * 5;
        se += (ax.weight[e * nq + q] * J) * va[r] * vb[s];
      }
      acc += se;
    }
    M[t] = acc;
  }
  if (t < nnp * 2) {
    const int r = t / nnp, i = t - r * nnp;
    double acc = 0.0, ls = 0.0;
    int cnt = 0;
    for (int e = 0; e < ax.nel; e++) {
      int a = -1;
      for (int l = 0; l < nen; l++) if (wrapi(ax.offset[e] + l, nnp) == i) a = l;
      if (a < 0) continue;
      const double J = ax.detJac[e];
      double se = 0.0;
      for (int q = 0; q < nq; q++) se += (ax.weight[e * nq + q] * J) * ax.value[((size_t)(e * nq + q) * nen + a) * 5 + r];
      acc += se;
      cnt++;
      ls += J / (double)nen;
    }
    mv[t] = acc;
    if (r == 0) { nsup[i] = cnt; lsum[i] = ls; }
  }
}

__global__ void kron_rowsum_kernel(const double* __restrict__ M, double* __restrict__ rsum, int nnp) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;   // t = rs*nnp + i
  if (t >= 4 * nnp) return;
  double acc = 0.0;
  for (int c = 0; c < kMaxW; c++) acc += M[(size_t)t * kMaxW + c];
  rsum[t] = acc;
}

// Dirichlet data of a node from its per-axis boundary codes (0 interior, 1 side 0, 2 side 1): the last face in the
// reference's order (axis ascending, side 0 then 1) wins (AddFixa overwrites, petigaelem.c:1166-1189).
template <int DOF>
__device__ __forceinline__ void node_fix(const KronParams& kp, int c0, int c1, int c2, bool fixed[DOF], double val[DOF]) {
#pragma unroll
  for (int c = 0; c < DOF; c++) { fixed[c] = false; val[c] = 0.0; }
  const int code[3] = {c0, c1, c2};
#pragma unroll
  for (int d = 0; d < 3; d++) {
    if (d >= kp.dim || !code[d]) continue;
    const FixSide& fs = kp.bc[d][code[d] - 1];
    for (int k = 0; k < fs.vcount; k++)
#pragma unroll
      for (int c = 0; c < DOF; c++)
        if (fs.vfield[k] == c) { fixed[c] = true; val[c] = fs.vvalue[k]; }
  }
}

__device__ __forceinline__ int bcode(int col, int nnp, int periodic) { return periodic ? 0 : ((col == 0) ? 1 : ((col == nnp - 1) ? 2 : 0)); }

// One CTA per (A_j, A_k) pencil of owned rows; warps walk the rows A_i of the pencil; lanes walk the entries of a
// row in storage order, so every store instruction writes 256 contiguous bytes.
// PF > 0: all axes have degree PF, so a full-width interior row has compile-time extents and its loop unrolls completely
// MINB: resident CTAs per SM the register budget is set for.  Scalar case, measured (tools/kron_probe.py): 3 CTAs of 80 registers are
// 3 % faster than 4 of 64 on long pencils (128^3: 0.986 vs 1.011 ms) and 5 % slower on short ones (64^3, an 8-GPU share), where the
// latency-bound prologue and boundary rows want more warps; the launcher picks by pencil length.  dof > 1: 2 (128 registers).
template <int DOF, int PF, int MINB>
__global__ void __launch_bounds__(256, MINB) kron_rows_kernel(const __grid_constant__ KronParams kp) {
  extern __shared__ __align__(16) double dynstage[];   // dof > 1: kStageCap doubles per warp
  __shared__ double G[4][DOF * DOF][kMaxWW];     // G^{rs0}_{ij}[cjk] = sum_terms c * M_j^{rs1}[A_j][cj] * M_k^{rs2}[A_k][ck]
  __shared__ int jkinfo[kMaxWW];                 // code_j | code_k<<2 | diag<<4 | P2<<8 | P3<<16   (P1 in jkp1)
  __shared__ int jkp1[kMaxWW];
  __shared__ double jkval[kMaxWW];
  __shared__ double Gm[2][kMaxWW];               // DOF == 1: G0/G3 with the Dirichlet (j,k) columns zeroed; Hs = sum over those columns of G*value
  __shared__ double Hs[2];
  __shared__ int fast_ctr;                       // next 4-row pass of the interior stretch (dynamic hand-out)               // DOF == 1: Dirichlet value of a column fixed by a j or k face (jkinfo bit 5)
  const int pencil = (int)blockIdx.x;
  const int Aj = kp.ls[1] + pencil % kp.lw[1], Ak = kp.ls[2] + pencil / kp.lw[1];
  const int gj = Aj - kp.gs[1], gk = Ak - kp.gs[2];
  const int Wj = kp.Wg[1][gj], Wk = kp.Wg[2][gk], Wjk = Wj * Wk;
  const int fj = kp.first[1][Aj], fk = kp.first[2][Ak];
  const bool fixing = kp.any_bc && kp.slot == PETIGA_SLOT_SYSTEM;
  // pencil tables: the 1-D rows of axes 1 and 2 first (one global load per thread), then one thread per (combination, column):
  // a pencil's prologue used to be 25-49 threads walking all terms with two dependent global loads each (27 terms for
  // elasticity: ~10 000 cycles per CTA, two thirds of a cfg-4 CTA's life)
  __shared__ double sM[2][4][kMaxW];
  __shared__ uint32_t sSeg[2][kMaxW];            // packed (B, S, L) bytes of this pencil's axis-1 / axis-2 rows
  for (int t = threadIdx.x; t < 2 * 4 * kMaxW; t += blockDim.x) {
    const int d = t / (4 * kMaxW), rs = (t / kMaxW) & 3, cc = t % kMaxW;
    (&sM[0][0][0])[t] = kp.M[1 + d][((size_t)rs * kp.nnp[1 + d] + (d ? Ak : Aj)) * kMaxW + cc];
  }
  if (threadIdx.x < 2 * kMaxW) {
    const int d = threadIdx.x / kMaxW, cc = threadIdx.x % kMaxW;
    sSeg[d][cc] = kp.seg[1 + d][(d ? gk : gj) * kMaxW + cc];
  }
  for (int t = threadIdx.x; t < 4 * DOF * DOF * kMaxWW; t += blockDim.x) (&G[0][0][0])[t] = 0.0;
  if (threadIdx.x == 0) fast_ctr = 0;
  __syncthreads();
  for (int w = threadIdx.x; w < kp.ncombo * Wjk; w += blockDim.x) {
    const int k = w / Wjk, t = w - k * Wjk, cj = t % Wj, ck = t / Wj;
    double acc = 0.0;
    for (int n = kp.combo_first[k]; n < kp.combo_first[k + 1]; n++) {
      const KronTerm tm = kp.terms[n];
      acc += tm.c * sM[0][tm.rs1][cj] * sM[1][tm.rs2][ck];
    }
    G[kp.combo_rs0[k]][kp.combo_ij[k]][t] = acc;
  }
  bool jk_boundary = false;
  for (int t = threadIdx.x; t < Wjk; t += blockDim.x) {
    const int cj = t % Wj, ck = t / Wj;
    int info = bcode(fj + cj, kp.nnp[1], kp.periodic[1]) | (bcode(fk + ck, kp.nnp[2], kp.periodic[2]) << 2);
    if (cj == Aj - fj && ck == Ak - fk) info |= 16;
    int p1 = 0;
    {
      const uint32_t s1 = sSeg[0][cj], s2 = sSeg[1][ck];
      const int Bj = s1 & 255, Sj = (s1 >> 8) & 255, Lj = (s1 >> 16) & 255;
      const int Bk = s2 & 255, Sk = (s2 >> 8) & 255, Lk = (s2 >> 16) & 255;
      p1 = Bk * Wj + Sk * Bj;
      info |= (Sk * Sj) << 8;
      info |= (Lk * Sj + Lj) << 16;
    }
    if (DOF == 1 && fixing && (info & 15)) {   // "last face wins": k over j over i (AddFixa overwrites, petigaelem.c:1166-1189)
      bool f[1]; double fv[1];
      node_fix<1>(kp, 0, info & 3, (info >> 2) & 3, f, fv);
      if (f[0]) { info |= 32; jkval[t] = fv[0]; }
    }
    jkinfo[t] = info;
    jkp1[t] = p1;
  }
  // does any column of this pencil touch a (j,k) boundary face?  (uniform over the CTA)
  // (only faces that carry Dirichlet values matter: cfg 4 constrains the two axis-0 faces only)
  jk_boundary = fixing && ((!kp.periodic[1] && ((fj == 0 && kp.bc[1][0].vcount) || (fj + Wj == kp.nnp[1] && kp.bc[1][1].vcount))) ||
                           (!kp.periodic[2] && ((fk == 0 && kp.bc[2][0].vcount) || (fk + Wk == kp.nnp[2] && kp.bc[2][1].vcount))));
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const bool want_mat = kp.values != nullptr, want_vec = kp.rhs != nullptr;
  const int rcj = bcode(Aj, kp.nnp[1], kp.periodic[1]), rck = bcode(Ak, kp.nnp[2], kp.periodic[2]);
  // everything the row loop needs, in registers (the parameter block lives in constant memory)
  const int lw0 = kp.lw[0], ls0 = kp.ls[0], gs0 = kp.gs[0], nnp0 = kp.nnp[0], per0 = kp.periodic[0];
  const int* __restrict__ Wg0 = kp.Wg[0];
  const int* __restrict__ first0 = kp.first[0];
  const double* __restrict__ M0 = kp.M[0];
  const int64_t* __restrict__ rowbase = kp.rowbase;
  double* __restrict__ values = kp.values;
  double* __restrict__ rhs = kp.rhs;
  const int rsmask0 = kp.rsmask0;
  const int lr0 = lw0 * ((Aj - kp.ls[1]) + kp.lw[1] * (Ak - kp.ls[2]));
  const bool simple_jk = kp.simp[1][gj] && kp.simp[2][gk];
  const int* __restrict__ simple0 = kp.simp[0];
  const bool fast_ok = (DOF == 1) && !(rsmask0 & 6) && want_mat;
  // right-hand side of an unconstrained row when the load is a single separable term (Poisson, mass)
  const bool vsimple = want_vec && DOF == 1 && kp.nvterms == 1;
  const double vjk = vsimple ? kp.vterms[0].c * kp.mv[1][kp.vterms[0].r1 * kp.nnp[1] + Aj] * kp.mv[2][kp.vterms[0].r2 * kp.nnp[2] + Ak] : 0.0;
  const double* __restrict__ mv0 = kp.mv[0] + (vsimple ? kp.vterms[0].r0 * nnp0 : 0);
  // full-width rows (W_i = 2p+1, all but the first/last p rows of a pencil): lane -> (column offset, group) fixed per warp
  const int WiF = kp.wfull0, ngrpF = 32 / WiF, grpF = lane / WiF, ciF = lane - grpF * WiF;
  const int ostepF = ngrpF * WiF, offF = grpF * WiF + ciF, nfullF = Wjk / ngrpF;   // every group runs nfullF full iterations
  // ---- interior stretch of a pencil whose own node is not on a Dirichlet face: 4 rows per warp pass share the G loads;
  //      no per-row tests.  Columns on Dirichlet (j,k) faces are handled by the masked tables Gm (stored value 0) and their
  //      contribution to the right-hand side is separable:  -rowsum(M0^{00})*H0 - rowsum(M0^{11})*H3 ----
  int nfast = 0;
  const int fast_lo = kp.fast_lo;
  bool pencil_fast = false;
  if (PF > 0) {
    constexpr int WIC = 2 * PF + 1, WJKC = WIC * WIC;
    pencil_fast = fast_ok && simple_jk && !(fixing && (rcj || rck)) && Wjk == WJKC && WiF == WIC && kp.fast_hi > fast_lo &&
                  !(jk_boundary && (kp.fixtable || !want_vec));
    if (pencil_fast) {
      if (jk_boundary) {   // uniform over the CTA
        if (warp == 0) {
          double h0 = 0.0, h3 = 0.0;
          for (int t = lane; t < Wjk; t += 32) {
            const bool fx = jkinfo[t] & 32;
            const double g0 = G[0][0][t], g3 = G[3][0][t];
            if (fx) { h0 = fma(g0, jkval[t], h0); h3 = fma(g3, jkval[t], h3); }
            Gm[0][t] = fx ? 0.0 : g0;
            Gm[1][t] = fx ? 0.0 : g3;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) { h0 += __shfl_xor_sync(0xffffffffu, h0, o); h3 += __shfl_xor_sync(0xffffffffu, h3, o); }
          if (lane == 0) { Hs[0] = h0; Hs[1] = h3; }
        }
        __syncthreads();
      }
      nfast = kp.fast_hi - fast_lo;
    }
  }
  // ---- dof > 1, interior stretch of a pencil (the same row range as the scalar fast passes): see the register-direct passes after
  //      the general loop ----
  constexpr int DD = DOF * DOF;
  bool blk_fast = false;
  if constexpr (DOF > 1 && PF > 0) {
    constexpr int WIC = 2 * PF + 1;
    const bool row_jk_bc = fixing && ((rcj && (kp.bc[1][rcj - 1].vcount || kp.bc[1][rcj - 1].lcount)) || (rck && (kp.bc[2][rck - 1].vcount || kp.bc[2][rck - 1].lcount)));
    blk_fast = want_mat && kp.two_slot && kp.dim == 3 && simple_jk && !jk_boundary && !row_jk_bc && Wjk <= WIC * WIC && WiF == WIC &&
               kp.fast_hi > fast_lo && (nwarps & 1) == 0;           // (pencils next to a j/k end have fewer columns: same code, shorter rows)
    if (blk_fast) nfast = kp.fast_hi - fast_lo;
  }
  const int nslow = lw0 - nfast;   // the general loop walks the remaining rows (compacted index)
  // per-row parameters are prefetched one row ahead (registers), so that their L2 latency overlaps the stores of the
  // current row instead of stalling every row (ncu r1_ncu_kron_rows_mesh128_v3: long_scoreboard was the top stall)
  struct RowP { int Wi, fi, simple; int64_t base; double a0, a3; };
  auto load_row = [&](int il_) {
    RowP r;
    const int Ai_ = ls0 + il_, gi_ = Ai_ - gs0;
    r.Wi = __ldg(Wg0 + gi_); r.fi = __ldg(first0 + Ai_); r.simple = __ldg(simple0 + gi_);
    r.base = __ldg(rowbase + il_ + lr0);
    r.a0 = r.a3 = 0.0;
    if (DOF == 1) { r.a0 = __ldg(M0 + (size_t)Ai_ * kMaxW + ciF); r.a3 = __ldg(M0 + ((size_t)3 * nnp0 + Ai_) * kMaxW + ciF); }   // only the scalar fast paths use them
    return r;
  };
  RowP cur, nxt;
  memset(&cur, 0, sizeof(cur));
  nxt = cur;
  auto row_of = [&](int idx) { return (idx < fast_lo || nfast == 0) ? idx : idx + nfast; };
  if (warp < nslow) cur = load_row(row_of(warp));
  for (int idx = warp; idx < nslow; idx += nwarps, cur = nxt) {
    if (idx + nwarps < nslow) nxt = load_row(row_of(idx + nwarps));
    const int il = row_of(idx);
    const int Ai = ls0 + il, gi = Ai - gs0;
    const int Wi = cur.Wi, fi = cur.fi, W = Wi * Wjk;
    const int lr = il + lr0;
    const int64_t base = cur.base;
    const bool SIMPLE = simple_jk && cur.simple;
    if (fast_ok) {
      const bool rowb = fixing && ((!per0 && (Ai == 0 || Ai == nnp0 - 1)) || rcj || rck);
      const bool colb = jk_boundary || (fixing && !per0 && (fi == 0 || fi + Wi == nnp0));
      if (!rowb && !colb) {
        // interior row: out[cjk*Wi + ci] = M00_i[ci]*G0[cjk] + M11_i[ci]*G3[cjk]; lane = (ci, group), groups stride cjk
        constexpr int WIC = 2 * PF + 1, WJKC = WIC * WIC, NGRP = 32 / WIC, NITER = (WJKC + NGRP - 1) / NGRP, OSTEP = NGRP * WIC;
        if (!SIMPLE) {   // columns owned by several ranks / periodic wrap: same values, closed-form position per entry
          const unsigned inv = (65536u + Wi - 1) / Wi;
          const int grp = (int)((lane * inv) >> 16), ci = lane - grp * Wi, ngrp = (int)((32u * inv) >> 16);
          if (grp < ngrp) {
            const double a0 = __ldg(M0 + (size_t)Ai * kMaxW + ci), a3 = __ldg(M0 + ((size_t)3 * nnp0 + Ai) * kMaxW + ci);
            const uint32_t s0 = __ldg(kp.seg[0] + gi * kMaxW + ci);
            const int Bi = s0 & 255, Si = (s0 >> 8) & 255, Li = (s0 >> 16) & 255;
            double* __restrict__ rowp = values + base;
            for (int cjk = grp; cjk < Wjk; cjk += ngrp) {
              const int info = jkinfo[cjk];
              const int pos = jkp1[cjk] * Wi + ((info >> 8) & 255) * Bi + ((info >> 16) & 255) * Si + Li;
              rowp[pos] = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
            }
          }
        } else if (PF > 0 && Wi == WIC && Wjk == WJKC) {   // full-width row of an interior pencil: everything but (a0, a3, base) is static
          if (grpF < NGRP) {
            const double a0 = cur.a0, a3 = cur.a3;
            double* __restrict__ rowp = values + base + offF;
            const double* __restrict__ g0 = &G[0][0][grpF];
            const double* __restrict__ g3 = &G[3][0][grpF];
#pragma unroll
            for (int k = 0; k < NITER; k++)
              if ((k + 1) * NGRP <= WJKC || grpF + k * NGRP < WJKC) rowp[k * OSTEP] = fma(a3, g3[k * NGRP], a0 * g0[k * NGRP]);
          }
        } else if (Wi == WiF) {   // full-width row: lane mapping and trip count hoisted out of the row loop
          if (grpF < ngrpF) {
            const double a0 = cur.a0, a3 = cur.a3;
            double* __restrict__ rowp = values + base + offF;
            int cjk = grpF;
            for (int it = 0; it < nfullF; ++it) {
              *rowp = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
              rowp += ostepF; cjk += ngrpF;
            }
            if (cjk < Wjk) *rowp = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
          }
        } else {
          const unsigned inv = (65536u + Wi - 1) / Wi;
          const int grp = (int)((lane * inv) >> 16), ci = lane - grp * Wi, ngrp = (int)((32u * inv) >> 16);
          if (grp < ngrp) {
            const double a0 = __ldg(M0 + (size_t)Ai * kMaxW + ci), a3 = __ldg(M0 + ((size_t)3 * nnp0 + Ai) * kMaxW + ci);
            double* out = values + base + grp * Wi + ci;
            const int ostep = ngrp * Wi;
            for (int cjk = grp; cjk < Wjk; cjk += ngrp) {
              *out = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
              out += ostep;
            }
          }
        }
        if (want_vec && lane == 0) {
          if (vsimple) rhs[lr] = vjk * __ldg(mv0 + Ai);
          else {
            double F = 0.0;
            for (int n = 0; n < kp.nvterms; n++) {
              const KronVTerm vt = kp.vterms[n];
              F += vt.c * kp.mv[0][vt.r0 * nnp0 + Ai] * kp.mv[1][vt.r1 * kp.nnp[1] + Aj] * kp.mv[2][vt.r2 * kp.nnp[2] + Ak];
            }
            rhs[lr] = F;
          }
        }
        continue;
      }
      if (!kp.fixtable) {
        // boundary rows of the scalar case (constant Dirichlet values): column fix data is per-lane (axis 0) and
        // per-cjk (shared memory), so an entry costs a flag test instead of a walk over the face tables
        const int rci0 = bcode(Ai, nnp0, per0);
        bool rf[1]; double rv[1];
        node_fix<1>(kp, rci0, rcj, rck, rf, rv);
        const double nel = (double)(kp.nsup[0][Ai] * kp.nsup[1][Aj] * kp.nsup[2][Ak]);
        double* __restrict__ rowp = values + base;
        double racc0 = 0.0;
        if (rowb && rf[0]) {
          // fixed row: zero except the diagonal, which counts the elements containing the node (petigaelem.c:1377-1387)
          const int cjkd = (Ak - fk) * Wj + (Aj - fj), cid = Ai - fi;
          int ediag = cjkd * Wi + cid;
          if (!SIMPLE) {
            const uint32_t s0 = __ldg(kp.seg[0] + gi * kMaxW + cid);
            const int info = jkinfo[cjkd];
            ediag = jkp1[cjkd] * Wi + ((info >> 8) & 255) * (int)(s0 & 255) + ((info >> 16) & 255) * (int)((s0 >> 8) & 255) + (int)((s0 >> 16) & 255);
          }
          for (int e = lane; e < W; e += 32) rowp[e] = (e == ediag) ? nel : 0.0;
          if (want_vec && lane == 0) rhs[lr] = nel * rv[0];
          continue;
        }
        {  // free row with columns on Dirichlet faces: those entries move to the right-hand side
          const unsigned inv = (65536u + Wi - 1) / Wi;
          const int grp = (int)((lane * inv) >> 16), ci = lane - grp * Wi, ngrp = (int)((32u * inv) >> 16);
          if (grp < ngrp) {
            const double a0 = __ldg(M0 + (size_t)Ai * kMaxW + ci), a3 = __ldg(M0 + ((size_t)3 * nnp0 + Ai) * kMaxW + ci);
            bool cfi[1]; double cvi[1];
            node_fix<1>(kp, bcode(fi + ci, nnp0, per0), 0, 0, cfi, cvi);
            const bool ifix = cfi[0];
            const double ival = cvi[0];
            if (SIMPLE) {
              double* out = rowp + grp * Wi + ci;
              const int ostep = ngrp * Wi;
              for (int cjk = grp; cjk < Wjk; cjk += ngrp) {
                double v = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
                if (jkinfo[cjk] & 32) { racc0 = fma(-v, jkval[cjk], racc0); v = 0.0; }
                else if (ifix) { racc0 = fma(-v, ival, racc0); v = 0.0; }
                *out = v;
                out += ostep;
              }
            } else {
              const uint32_t s0 = __ldg(kp.seg[0] + gi * kMaxW + ci);
              const int Bi = s0 & 255, Si = (s0 >> 8) & 255, Li = (s0 >> 16) & 255;
              for (int cjk = grp; cjk < Wjk; cjk += ngrp) {
                double v = fma(a3, G[3][0][cjk], a0 * G[0][0][cjk]);
                const int info = jkinfo[cjk];
                if (info & 32) { racc0 = fma(-v, jkval[cjk], racc0); v = 0.0; }
                else if (ifix) { racc0 = fma(-v, ival, racc0); v = 0.0; }
                rowp[jkp1[cjk] * Wi + ((info >> 8) & 255) * Bi + ((info >> 16) & 255) * Si + Li] = v;
              }
            }
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) racc0 += __shfl_xor_sync(0xffffffffu, racc0, o);
          if (want_vec && lane == 0) {
            double F = vsimple ? vjk * __ldg(mv0 + Ai) : 0.0;
            if (!vsimple)
              for (int n = 0; n < kp.nvterms; n++) {
                const KronVTerm vt = kp.vterms[n];
                F += vt.c * kp.mv[0][vt.r0 * nnp0 + Ai] * kp.mv[1][vt.r1 * kp.nnp[1] + Aj] * kp.mv[2][vt.r2 * kp.nnp[2] + Ak];
              }
            if (rowb) {   // loads on the faces this (unfixed) node lies on
              const int rcode[3] = {rci0, rcj, rck};
              for (int d = 0; d < kp.dim; d++) {
                if (!rcode[d]) continue;
                const FixSide& fs = kp.bc[d][rcode[d] - 1];
                if (!fs.lcount) continue;
                double A = 1.0;
                if (kp.dim > 1) {
                  const int An[3] = {Ai, Aj, Ak};
                  for (int e2 = 0; e2 < kp.dim; e2++) if (e2 != d) A *= kp.lsum[e2][An[e2]];
                  A *= (kp.dim == 2) ? 2 : 4;
                }
                for (int k = 0; k < fs.lcount; k++) if (fs.lfield[k] == 0) F += fs.lvalue[k] * A;
              }
            }
            rhs[lr] = F + racc0;
          }
          continue;
        }
      }
    }
    const int rci = bcode(Ai, kp.nnp[0], kp.periodic[0]);
    const bool row_boundary = fixing && (rci | rcj | rck);
    const bool col_boundary = jk_boundary || (fixing && !kp.periodic[0] && (fi == 0 || fi + Wi == kp.nnp[0]));
    double racc[DOF];
#pragma unroll
    for (int c = 0; c < DOF; c++) racc[c] = 0.0;
    bool rfix[DOF];
    double rval[DOF];
#pragma unroll
    for (int c = 0; c < DOF; c++) { rfix[c] = false; rval[c] = 0.0; }
    const double nelem = (double)(kp.nsup[0][Ai] * kp.nsup[1][Aj] * kp.nsup[2][Ak]);
    if (row_boundary) {
      node_fix<DOF>(kp, rci, rcj, rck, rfix, rval);
      if (kp.fixtable) {
        const int gidx = gi + kp.gw[0] * (gj + kp.gw[1] * gk);
#pragma unroll
        for (int c = 0; c < DOF; c++) if (rfix[c]) rval[c] = kp.fixtable[(size_t)gidx * DOF + c];
      }
    }
    if (want_mat || col_boundary) {
      // lane -> (fixed column offset ci along axis 0, group); a group walks cjk with stride ngrp, so one warp store
      // covers ngrp*Wi consecutive entries of the row
      const int ngrp = 32 / Wi, grp = lane / Wi, ci = lane - grp * Wi;
      const bool slow = row_boundary || col_boundary;
      double a[4];
#pragma unroll
      for (int rs = 0; rs < 4; rs++) a[rs] = ((kp.rsmask0 >> rs) & 1) ? kp.M[0][((size_t)rs * kp.nnp[0] + Ai) * kMaxW + ci] : 0.0;
      int Bi = 0, Si = 1, Li = ci;
      if (!SIMPLE) { const uint32_t s0 = kp.seg[0][gi * kMaxW + ci]; Bi = s0 & 255; Si = (s0 >> 8) & 255; Li = (s0 >> 16) & 255; }
      const int cci = slow ? bcode(fi + ci, kp.nnp[0], kp.periodic[0]) : 0;
      const bool diag_i = (ci == Ai - fi);
      // BAIJ blocks of the ngrp*Wi entries a warp produces per iteration are contiguous in memory when the row is in
      // storage order: stage them in shared memory and write them back with full 256-byte warp stores
      const bool staged = (DOF > 1) && want_mat && kp.block && SIMPLE;
      double* stg = (DOF > 1) ? dynstage + (threadIdx.x >> 5) * kStageCap : nullptr;
      for (int cjk0 = 0; cjk0 < Wjk; cjk0 += ngrp) {
        const int cjk = cjk0 + grp;
        const bool act = grp < ngrp && cjk < Wjk;
        if (!act && !staged) continue;
        double v[DOF * DOF];
#pragma unroll
        for (int ij = 0; ij < DOF * DOF; ij++) v[ij] = 0.0;
        if (act) {
#pragma unroll
        for (int ij = 0; ij < DOF * DOF; ij++) {
          const int m = kp.rsmask_ij[ij];      // uniform: skip the order pairs this block never uses
          double x = 0.0;
          if (m & 1) x = a[0] * G[0][ij][cjk];
          if (m & 8) x = fma(a[3], G[3][ij][cjk], x);
          if (m & 2) x = fma(a[1], G[1][ij][cjk], x);
          if (m & 4) x = fma(a[2], G[2][ij][cjk], x);
          v[ij] = x;
        }
        int pos = cjk * Wi + ci;
        if (!SIMPLE || slow) {
          const int info = jkinfo[cjk];
          if (!SIMPLE) pos = jkp1[cjk] * Wi + ((info >> 8) & 255) * Bi + ((info >> 16) & 255) * Si + Li;
          if (slow && (row_boundary || cci || (info & 15))) {   // fixed row, or a column node on a Dirichlet face
            bool cfix[DOF];
            double cval[DOF];
            node_fix<DOF>(kp, cci, info & 3, (info >> 2) & 3, cfix, cval);
            if (kp.fixtable && (cci | (info & 15))) {
              const int cj = cjk % Wj, ck = cjk / Wj;
              const int hi = wrapi(fi + ci, kp.nnp[0]) - kp.gs[0], hj = wrapi(fj + cj, kp.nnp[1]) - kp.gs[1], hk = wrapi(fk + ck, kp.nnp[2]) - kp.gs[2];
              const int gidx = hi + kp.gw[0] * (hj + kp.gw[1] * hk);
#pragma unroll
              for (int c = 0; c < DOF; c++) if (cfix[c]) cval[c] = kp.fixtable[(size_t)gidx * DOF + c];
            }
            const bool isdiag = (info & 16) && diag_i;
#pragma unroll
            for (int i = 0; i < DOF; i++)
#pragma unroll
              for (int j = 0; j < DOF; j++) {
                double x = v[i * DOF + j];
                if (rfix[i]) x = (isdiag && i == j) ? nelem : 0.0;
                else if (cfix[j]) { racc[i] -= x * cval[j]; x = 0.0; }
                v[i * DOF + j] = x;
              }
          }
        }
        if (want_mat && !staged) {
          if (DOF == 1) kp.values[(size_t)(base + pos)] = v[0];
          else {
#pragma unroll
            for (int i = 0; i < DOF; i++)
#pragma unroll
              for (int j = 0; j < DOF; j++) {
                size_t off;
                if (kp.block) off = (size_t)(base + pos) * DOF * DOF + j * DOF + i;
                else off = (size_t)base * DOF * DOF + (size_t)i * W * DOF + (size_t)pos * DOF + j;
                kp.values[off] = v[i * DOF + j];
              }
          }
        }
        }   // act
        if (staged) {   // uniform over the warp
          const int e0 = cjk0 * Wi, ne = min(ngrp * Wi, W - e0);          // entries [e0, e0+ne) of the row, contiguous blocks
          if (act) {
#pragma unroll
            for (int i = 0; i < DOF; i++)
#pragma unroll
              for (int j = 0; j < DOF; j++) stg[lane * DOF * DOF + j * DOF + i] = v[i * DOF + j];   // column-major block
          }
          __syncwarp();
          double* dst = kp.values + (size_t)(base + e0) * DOF * DOF;
          for (int t = lane; t < ne * DOF * DOF; t += 32) dst[t] = stg[t];
          __syncwarp();
        }
      }
    }
    if (want_vec) {
      if (col_boundary) {
#pragma unroll
        for (int c = 0; c < DOF; c++) {
          double r = racc[c];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
          racc[c] = r;
        }
      }
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < DOF; c++) {
          double F = 0.0;
          for (int n = 0; n < kp.nvterms; n++) {
            const KronVTerm vt = kp.vterms[n];
            if (vt.i != c) continue;
            F += vt.c * kp.mv[0][vt.r0 * kp.nnp[0] + Ai] * kp.mv[1][vt.r1 * kp.nnp[1] + Aj] * kp.mv[2][vt.r2 * kp.nnp[2] + Ak];
          }
          if (row_boundary) {
            // AddFlux: loads on the faces this node lies on, summed over the face elements that contain it
            const int rcode[3] = {rci, rcj, rck};
            for (int d = 0; d < kp.dim; d++) {
              if (!rcode[d]) continue;
              const FixSide& fs = kp.bc[d][rcode[d] - 1];
              if (!fs.lcount) continue;
              double A = 1.0;
              if (kp.dim > 1) {
                const int An[3] = {Ai, Aj, Ak};
                for (int e2 = 0; e2 < kp.dim; e2++) if (e2 != d) A *= kp.lsum[e2][An[e2]];
                A *= (kp.dim == 2) ? 2 : 4;
              }
              for (int k = 0; k < fs.lcount; k++) if (fs.lfield[k] == c) F += fs.lvalue[k] * A;
            }
          }
          F += racc[c];
          if (rfix[c]) F = nelem * rval[c];
          kp.rhs[(size_t)lr * DOF + c] = F;
        }
      }
    }
  }
  // ---- dof > 1: register-direct rows.  A row of the interior stretch is WR blocks of DD doubles, contiguous in memory.  A lane owns
  //      the output positions t = 32 k + lane of HALF a row (two warps per row); the G factors of its positions do not depend on
  //      the axis-0 row, so they live in registers for the whole pencil (2 x KH doubles); per row only the 2 x WIC x DD axis-0 factors
  //      are staged (90 doubles at p = 2, loaded one row ahead), and every store instruction writes 256 contiguous bytes.
  //      Was (ncu r2_ncu_kron_cfg4_v2): the row built in shared memory and copied out -- 302 LSU wavefronts per 9 000-byte row
  //      against 220 cycles at HBM rate. ----
  if constexpr (DOF > 1 && PF > 0) {
    if (blk_fast) {
      constexpr int NSPLIT = 2;                                   // warps per row (measured: 4 warps per row at 3 CTAs per SM spills and is 10 % slower)
      constexpr int WIC = 2 * PF + 1, WJKC = WIC * WIC, KT = (WIC * WJKC * DD + 31) / 32, KH = (KT + NSPLIT - 1) / NSPLIT;
      constexpr int NACV = (WIC * DD * 2 + 31) / 32;
      const int WR = WIC * Wjk, NV = WR * DD;                     // blocks / doubles of a full-width row of THIS pencil
      const int h = warp % NSPLIT, pairi = warp / NSPLIT, npair = nwarps / NSPLIT;
      double gA[KH], gB[KH];
      int aoff[KH];
#pragma unroll
      for (int k = 0; k < KH; k++) {
        const int t = 32 * (h * KH + k) + lane;
        gA[k] = gB[k] = 0.0; aoff[k] = 0;
        if (t < NV) {
          int blk, i, j;
          if (kp.block) { blk = t / DD; const int e = t - blk * DD; j = e / DOF; i = e - j * DOF; }          // column-major blocks
          else { i = t / (WR * DOF); const int r2 = t - i * (WR * DOF); blk = r2 / DOF; j = r2 - blk * DOF; }   // DOF scalar rows
          const int ij = i * DOF + j, cjk = blk / WIC, ci = blk - cjk * WIC;
          if (kp.slotA[ij] >= 0) gA[k] = G[kp.slotA[ij]][ij][cjk];
          if (kp.slotB[ij] >= 0) gB[k] = G[kp.slotB[ij]][ij][cjk];
          // the staged table is ordered like the outputs (BAIJ: q = position inside the column-major block), so that consecutive
          // lanes read consecutive 16-byte entries: no bank conflicts
          aoff[k] = (ci * DD + (kp.block ? j * DOF + i : ij)) * 2;
        }
      }
      int acg[NACV];                                             // this lane's entries of the staged table ac[ci][ij][2] -> offsets into M0
#pragma unroll
      for (int k = 0; k < NACV; k++) {
        acg[k] = -1;
        const int t = lane + 32 * k;
        if (t < WIC * DD * 2) {
          const int ci = t / (DD * 2), r2 = t - ci * (DD * 2), q = r2 >> 1;
          const int ij = kp.block ? (q % DOF) * DOF + q / DOF : q;
          const int rs = (r2 & 1) ? kp.slotB[ij] : kp.slotA[ij];
          if (rs >= 0) acg[k] = rs * nnp0 * kMaxW + ci;
        }
      }
      double* acs = dynstage + warp * kStageCap + 32 * DD;       // (the general path's staging area comes first)
      double acv[NACV];
      int il = fast_lo + pairi;
#pragma unroll
      for (int k = 0; k < NACV; k++) acv[k] = (il < kp.fast_hi && acg[k] >= 0) ? __ldg(M0 + acg[k] + (size_t)(ls0 + il) * kMaxW) : 0.0;
      int64_t base_n = il < kp.fast_hi ? __ldg(rowbase + lr0 + il) : 0;
      for (; il < kp.fast_hi; il += npair) {
        const int Ai = ls0 + il, lr = il + lr0;
        const int64_t base = base_n;                             // (row parameters are loaded one row ahead)
        if (il + npair < kp.fast_hi) base_n = __ldg(rowbase + lr + npair);
#pragma unroll
        for (int k = 0; k < NACV; k++) { const int t = lane + 32 * k; if (t < WIC * DD * 2) acs[t] = acv[k]; }
        const int iln = il + npair;
#pragma unroll
        for (int k = 0; k < NACV; k++) acv[k] = (iln < kp.fast_hi && acg[k] >= 0) ? __ldg(M0 + acg[k] + (size_t)(ls0 + iln) * kMaxW) : 0.0;
        __syncwarp();
        double* __restrict__ dst = values + (size_t)base * DD + 32 * (h * KH) + lane;
        constexpr int KB = (KH + 2) / 3;                        // three batches: all loads of a batch issue before its stores
#pragma unroll
        for (int b3 = 0; b3 < 3; b3++) {
          double2 a2[KB];
#pragma unroll
          for (int kk = 0; kk < KB; kk++) { const int k = b3 * KB + kk; if (k < KH) a2[kk] = *reinterpret_cast<const double2*>(acs + aoff[k]); }
#pragma unroll
          for (int kk = 0; kk < KB; kk++) {
            const int k = b3 * KB + kk;
            if (k < KH && 32 * (h * KH + k) + lane < NV) dst[32 * k] = fma(a2[kk].y, gB[k], a2[kk].x * gA[k]);
          }
        }
        __syncwarp();
        if (want_vec && h == 0 && lane == 0) {
#pragma unroll
          for (int cc = 0; cc < DOF; cc++) {
            double F = 0.0;
            for (int n = 0; n < kp.nvterms; n++) {
              const KronVTerm vt = kp.vterms[n];
              if (vt.i != cc) continue;
              F += vt.c * kp.mv[0][vt.r0 * nnp0 + Ai] * kp.mv[1][vt.r1 * kp.nnp[1] + Aj] * kp.mv[2][vt.r2 * kp.nnp[2] + Ak];
            }
            rhs[(size_t)lr * DOF + cc] = F;
          }
        }
      }
    }
  }
  // ---- the 4-row passes, handed out dynamically: warps that had a (slower) general row above join later, so the CTA's
  //      warps finish together instead of leaving a low-parallelism tail ----
  if (PF > 0 && pencil_fast) {
    constexpr int WIC = 2 * PF + 1, WJKC = WIC * WIC, NGRP = 32 / WIC, NITER = (WJKC + NGRP - 1) / NGRP, OSTEP = NGRP * WIC, RW = WIC * WJKC, R = 4;
    const int64_t base_lo = __ldg(rowbase + lr0 + fast_lo);
    const double* __restrict__ g0 = jk_boundary ? &Gm[0][grpF] : &G[0][0][grpF];
    const double* __restrict__ g3 = jk_boundary ? &Gm[1][grpF] : &G[3][0][grpF];
    const double H0 = jk_boundary ? Hs[0] : 0.0, H3 = jk_boundary ? Hs[1] : 0.0;
    for (;;) {
      int grab = 0;
      if (lane == 0) grab = atomicAdd(&fast_ctr, 1);
      grab = __shfl_sync(0xffffffffu, grab, 0);
      const int il = fast_lo + grab * R;
      if (il >= kp.fast_hi) break;
      if (kp.bulk) {
        // the R rows of this pass are one contiguous run of R*RW doubles: build it in shared memory and let the TMA engine write it
        // (cp.async.bulk shared -> global, SASS UBLKCP) instead of 13 x R partial-width (28 of 32 lanes, 224-byte) warp stores.
        // Source, destination and size must be 16-byte aligned: the run is staged with the parity of its global start, the odd
        // first / last element goes out with a plain store.
        double* sb = dynstage + warp * (R * RW + 4);
        const int64_t gstart = base_lo + (int64_t)(il - fast_lo) * RW;
        const int par = (int)(gstart & 1);
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");          // the previous run of this warp has left the buffer
        __syncwarp();
        if (grpF < NGRP) {
          double a0[R], a3[R];
#pragma unroll
          for (int r = 0; r < R; r++) {
            a0[r] = __ldg(M0 + (size_t)(ls0 + il + r) * kMaxW + ciF);
            a3[r] = __ldg(M0 + ((size_t)3 * nnp0 + ls0 + il + r) * kMaxW + ciF);
          }
          double* __restrict__ rowp = sb + par + offF;
#pragma unroll
          for (int k = 0; k < NITER; k++)
            if ((k + 1) * NGRP <= WJKC || grpF + k * NGRP < WJKC) {
              const double x0 = g0[k * NGRP], x3 = g3[k * NGRP];
#pragma unroll
              for (int r = 0; r < R; r++) rowp[r * RW + k * OSTEP] = fma(a3[r], x3, a0[r] * x0);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");           // generic-proxy writes -> visible to the async proxy
        __syncwarp();
        if (lane == 0) {
          const uint32_t nbytes = (uint32_t)(R * RW - 2 * par) * 8u;            // R*RW is even: both parities leave a multiple of 16 bytes
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                       ::"l"(__cvta_generic_to_global(values + gstart + par)), "r"((uint32_t)__cvta_generic_to_shared(sb + 2 * par)), "r"(nbytes) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          if (par) { values[gstart] = sb[1]; values[gstart + R * RW - 1] = sb[R * RW]; }
        }
      } else
      if (grpF < NGRP) {
        double a0[R], a3[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
          a0[r] = __ldg(M0 + (size_t)(ls0 + il + r) * kMaxW + ciF);
          a3[r] = __ldg(M0 + ((size_t)3 * nnp0 + ls0 + il + r) * kMaxW + ciF);
        }
        double* __restrict__ rowp = values + base_lo + (int64_t)(il - fast_lo) * RW + offF;
#pragma unroll
        for (int k = 0; k < NITER; k++)
          if ((k + 1) * NGRP <= WJKC || grpF + k * NGRP < WJKC) {
            const double x0 = g0[k * NGRP], x3 = g3[k * NGRP];
#pragma unroll
            for (int r = 0; r < R; r++) rowp[r * RW + k * OSTEP] = fma(a3[r], x3, a0[r] * x0);
          }
      }
      if (want_vec && lane < R) {
        const int Ai = ls0 + il + lane;
        double F;
        if (vsimple) F = vjk * __ldg(mv0 + Ai);
        else {
          F = 0.0;
          for (int n = 0; n < kp.nvterms; n++) {
            const KronVTerm vt = kp.vterms[n];
            F += vt.c * kp.mv[0][vt.r0 * nnp0 + Ai] * kp.mv[1][vt.r1 * kp.nnp[1] + Aj] * kp.mv[2][vt.r2 * kp.nnp[2] + Ak];
          }
        }
        if (jk_boundary) F -= __ldg(kp.rsum[0] + Ai) * H0 + __ldg(kp.rsum[0] + (size_t)3 * nnp0 + Ai) * H3;
        rhs[lr0 + il + lane] = F;
      }
    }
    if (kp.bulk) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");       // all bulk stores of this thread have completed
  }
}

template <int DIM, int DOF>
void host_terms(int form, int slot, const double* prm, const FormInfo& fi, KronParams& kp) {
  const int NA = fi.mc1 - fi.mc0, NV = fi.vc1 - fi.vc0;
  std::vector<double> C((size_t)DOF * DOF * std::max(NA, 1) * std::max(NA, 1), 0.0), fv((size_t)DOF * std::max(NV, 1), 0.0);
  QPoint q;
  memset(&q, 0, sizeof(q));
  form_coefficients<DIM, DOF>(form, slot, prm, 0.0, 0.0, q, NA, NV, NA ? C.data() : nullptr, (NV && fi.constant_f) ? fv.data() : nullptr);
  kp.nterms = kp.nvterms = kp.rsmask0 = 0;
  for (int k = 0; k < 9; k++) kp.rsmask_ij[k] = 0;
  for (int i = 0; i < DOF; i++)
    for (int j = 0; j < DOF; j++)
      for (int al = 0; al < NA; al++)
        for (int be = 0; be < NA; be++) {
          double c = C[(((size_t)i * DOF + j) * NA + al) * NA + be];
          if (c == 0.0) continue;
          KronTerm t;
          const int ca = al + fi.mc0, cb = be + fi.mc0;
          unsigned char rs[3];
          for (int d = 0; d < 3; d++) rs[d] = (unsigned char)(((ca == 1 + d) ? 2 : 0) + ((cb == 1 + d) ? 1 : 0));
          t.ij = (unsigned char)(i * DOF + j); t.rs0 = rs[0]; t.rs1 = rs[1]; t.rs2 = rs[2]; t.c = c;
          if (kp.nterms < kMaxTerms) kp.terms[kp.nterms] = t;
          kp.nterms++;
          kp.rsmask0 |= 1 << rs[0];
          kp.rsmask_ij[i * DOF + j] |= 1 << rs[0];
        }
  for (int i = 0; i < DOF; i++)
    for (int al = 0; al < NV; al++) {
      double c = fv[(size_t)i * NV + al];
      if (c == 0.0) continue;
      const int ca = al + fi.vc0;
      KronVTerm t;
      t.i = (unsigned char)i; t.r0 = (ca == 1); t.r1 = (ca == 2); t.r2 = (ca == 3); t.c = c;
      if (kp.nvterms < 8) kp.vterms[kp.nvterms] = t;
      kp.nvterms++;
    }
}

}  // namespace

static int launch_kron_kernel(petiga_cuda_plan* P, const KronParams& kp) {
  const Layout& L = P->L;
  const int blocks = L.ax[1].lw * L.ax[2].lw;
  int threads = std::min(256, std::max(32, ((L.ax[0].lw + 0) * 32)));
  if (const char* e = getenv("PETIGA_KRON_THREADS")) threads = std::max(32, std::min(256, atoi(e) / 32 * 32));   // tuning knob
  int pf = L.ax[0].p;
  for (int d = 1; d < L.dim; d++) if (L.ax[d].p != pf) pf = 0;
  if (L.dim < 3 || (L.dof != 1 && pf > 2)) pf = 0;
  size_t dyn = L.dof > 1 ? (size_t)(threads / 32) * kStageCap * sizeof(double) : 0;
  if (L.dof == 1 && kp.bulk && pf > 0) dyn = (size_t)(threads / 32) * (4 * (2 * pf + 1) * (2 * pf + 1) * (2 * pf + 1) + 4) * sizeof(double);
  const int minb = L.dof > 1 ? 2 : (L.ax[0].lw >= kp.minb_rows ? 3 : 4);
#define KL(DOF_, PF_, MB_) if (L.dof == DOF_ && pf == PF_ && minb == MB_) { \
    if (dyn) PC_CUDA(cudaFuncSetAttribute(kron_rows_kernel<DOF_, PF_, MB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn)); \
    kron_rows_kernel<DOF_, PF_, MB_><<<blocks, threads, dyn, P->stream>>>(kp); }
  KL(1, 0, 3) KL(1, 1, 3) KL(1, 2, 3) KL(1, 3, 3) KL(1, 4, 3) KL(1, 0, 4) KL(1, 1, 4) KL(1, 2, 4) KL(1, 3, 4) KL(1, 4, 4)
  KL(2, 0, 2) KL(3, 0, 2) KL(2, 1, 2) KL(2, 2, 2) KL(3, 1, 2) KL(3, 2, 2)
#undef KL
  PC_CUDA(cudaGetLastError());
  P->launches++;
  return 0;
}

bool kron_applicable(const petiga_cuda_plan* P, int slot, int form) {
  const Layout& L = P->L;
  if (slot != PETIGA_SLOT_VECTOR && slot != PETIGA_SLOT_MATRIX && slot != PETIGA_SLOT_SYSTEM) return false;
  if (P->d_X) return false;                                  // mapped geometry: coefficients vary per point
  FormInfo fi = form_info(form, slot, L.dim, L.dof);
  if (!fi.valid || !fi.mat_const) return false;
  if (!fi.constant_f) {
    // point-wise load: the matrix can still be written by this path and the vector integrated by the quadrature kernel,
    // provided no Dirichlet/Neumann fix-up couples them (IGAComputeMatrix/Vector never fix)
    if (slot == PETIGA_SLOT_VECTOR) return false;
    if (slot == PETIGA_SLOT_SYSTEM && P->has_bc) return false;
  }
  if (L.dof > 3) return false;
  for (int d = 0; d < L.dim; d++) if (L.ax[d].p > kKronP) return false;
  if (P->d_fixtable && L.nranks > 1) return false;          // table values of off-box columns are not local
  for (int d = 0; d < L.dim; d++)
    if (L.ax[d].periodic && L.ax[d].nnp < 2 * L.ax[d].p + 1) return false;
  return true;
}

int launch_kronecker(petiga_cuda_plan* P, int slot, int block, double* values, double* rhs) {
  const Layout& L = P->L;
  const int form = P->slots[slot].form;
  FormInfo fi = form_info(form, slot, L.dim, L.dof);
  if (!P->d_kronrow[0]) {   // 1-D tables, once per plan
    for (int d = 0; d < 3; d++) {
      const int nnp = L.ax[d].nnp;
      void* buf = nullptr;
      const size_t nM = (size_t)4 * nnp * kMaxW, nmv = (size_t)2 * nnp;
      PC_CUDA(cudaMalloc(&buf, (nM + nmv + nnp + (size_t)4 * nnp) * sizeof(double) + (size_t)nnp * sizeof(int)));
      P->allocs.push_back(buf);
      P->d_kronrow[d] = (double*)buf;
      double* M = (double*)buf; double* mv = M + nM; double* lsum = mv + nmv; double* rsum = lsum + nnp; int* nsup = (int*)(rsum + (size_t)4 * nnp);
      const int total = (int)nM;
      kron_1d_kernel<<<(total + 127) / 128, 128, 0, P->stream>>>(P->dax[d], P->d_first[d], M, mv, nsup, lsum);
      PC_CUDA(cudaGetLastError());
      kron_rowsum_kernel<<<(4 * nnp + 127) / 128, 128, 0, P->stream>>>(M, rsum, nnp);
      PC_CUDA(cudaGetLastError());
      P->launches += 2;
    }
  }
  // the parameter block only depends on (slot, form, parameters, block layout, boundary conditions): build it once and
  // reuse it, so that a repeated assembly costs one kernel launch on the host side
  if (P->kron_cache.size() == sizeof(KronParams) && P->kron_cache_slot == slot && P->kron_cache_block == block &&
      P->kron_cache_version == P->config_version) {
    KronParams kc;
    memcpy(&kc, P->kron_cache.data(), sizeof(kc));
    kc.values = values; kc.rhs = rhs;
    return launch_kron_kernel(P, kc);
  }
  KronParams kp;
  memset(&kp, 0, sizeof(kp));
  bool simple = (L.nranks == 1);
  for (int d = 0; d < 3; d++) {
    const int nnp = L.ax[d].nnp;
    const size_t nM = (size_t)4 * nnp * kMaxW, nmv = (size_t)2 * nnp;
    kp.M[d] = P->d_kronrow[d]; kp.mv[d] = kp.M[d] + nM; kp.lsum[d] = kp.mv[d] + nmv; kp.rsum[d] = kp.lsum[d] + nnp; kp.nsup[d] = (const int*)(kp.rsum[d] + (size_t)4 * nnp);
    kp.first[d] = P->d_first[d]; kp.Wg[d] = P->dax[d].W; kp.lo[d] = P->dax[d].lo; kp.seg[d] = P->dax[d].seg; kp.simp[d] = P->dax[d].simple;
    kp.ls[d] = L.ax[d].ls; kp.lw[d] = L.ax[d].lw; kp.gs[d] = L.ax[d].gs; kp.gw[d] = L.ax[d].gw; kp.nnp[d] = nnp; kp.periodic[d] = L.ax[d].periodic;
    if (L.ax[d].periodic) simple = false;
  }
  kp.rowbase = P->d_rowbase; kp.localrow = P->d_localrow; kp.fixtable = P->d_fixtable;
  kp.dim = L.dim; kp.dof = L.dof; kp.block = block; kp.slot = slot; kp.simple = simple; kp.wfull0 = 2 * L.ax[0].p + 1;
  kp.bulk = P->kron_bulk;
  kp.minb_rows = P->kron_minb_rows;
  kp.values = values; kp.rhs = rhs;
  const double* prm = P->slots[slot].prm;
#define HT(DIM_, DOF_) if (L.dim == DIM_ && L.dof == DOF_) host_terms<DIM_, DOF_>(form, slot, prm, fi, kp);
  HT(1, 1) HT(1, 2) HT(1, 3) HT(2, 1) HT(2, 2) HT(2, 3) HT(3, 1) HT(3, 2) HT(3, 3)
#undef HT
  if (kp.nterms > kMaxTerms || kp.nvterms > 8) { set_error("separable path: too many coefficient terms"); return PETIGA_CUDA_ERR_SUP; }
  {  // terms grouped by (axis-0 order pair, block entry), original order kept inside a group (same summation order as before)
    std::stable_sort(kp.terms, kp.terms + kp.nterms, [](const KronTerm& a, const KronTerm& b) { return a.rs0 * 16 + a.ij < b.rs0 * 16 + b.ij; });
    kp.ncombo = 0;
    for (int n = 0; n < kp.nterms; n++) {
      if (n == 0 || kp.terms[n].rs0 != kp.terms[n - 1].rs0 || kp.terms[n].ij != kp.terms[n - 1].ij) {
        kp.combo_rs0[kp.ncombo] = kp.terms[n].rs0; kp.combo_ij[kp.ncombo] = kp.terms[n].ij; kp.combo_first[kp.ncombo] = (unsigned char)n;
        kp.ncombo++;
      }
    }
    kp.combo_first[kp.ncombo] = (unsigned char)kp.nterms;
  }
  kp.two_slot = 1;
  for (int ij = 0; ij < 9; ij++) {
    kp.slotA[ij] = kp.slotB[ij] = -1;
    int n = 0;
    for (int rs = 0; rs < 4; rs++)
      if ((kp.rsmask_ij[ij] >> rs) & 1) { if (n == 0) kp.slotA[ij] = (signed char)rs; else if (n == 1) kp.slotB[ij] = (signed char)rs; n++; }
    if (n > 2) kp.two_slot = 0;
  }
  if (slot == PETIGA_SLOT_SYSTEM) {
    fill_fix_sides(P, true, kp.bc);
    for (int d = 0; d < L.dim; d++)
      for (int s = 0; s < 2; s++)
        if (!L.ax[d].periodic && (kp.bc[d][s].vcount || kp.bc[d][s].lcount)) kp.any_bc = 1;
  }
  {  // longest run of axis-0 rows that are full-width, in storage order and free of Dirichlet rows/columns
    const AxisLayout& a0 = L.ax[0];
    const bool fixing0 = kp.any_bc && slot == PETIGA_SLOT_SYSTEM && !a0.periodic;
    int best_lo = 0, best_hi = 0, run_lo = -1;
    for (int il = 0; il <= a0.lw; il++) {
      bool ok = false;
      if (il < a0.lw) {
        const int Ai = a0.ls + il, gi = Ai - a0.gs, Wi = a0.W[gi], fi = a0.first[Ai];
        ok = (Wi == 2 * a0.p + 1) && a0.simple[gi];
        if (ok && fixing0 && (Ai == 0 || Ai == a0.nnp - 1 || fi == 0 || fi + Wi == a0.nnp)) ok = false;
      }
      if (ok) { if (run_lo < 0) run_lo = il; }
      else if (run_lo >= 0) { if (il - run_lo > best_hi - best_lo) { best_lo = run_lo; best_hi = il; } run_lo = -1; }
    }
    kp.fast_lo = best_lo;
    kp.fast_hi = best_lo + (best_hi - best_lo) / 4 * 4;
  }
  P->kron_cache.resize(sizeof(KronParams));
  memcpy(P->kron_cache.data(), &kp, sizeof(kp));
  P->kron_cache_slot = slot; P->kron_cache_block = block; P->kron_cache_version = P->config_version;
  return launch_kron_kernel(P, kp);
}

}  // namespace pc
