// pc_colloc.cu -- isogeometric collocation (IGASetUseCollocation): one matrix row per owned node, evaluated at the node's
// Greville point.
//
// There is no quadrature and no element loop.  The rank that owns a node computes its whole row, so every value is written
// exactly once with a plain store: no atomics, no ghost rows, no exchange, the same bits on every run, and no zeroing pass
// (the (p+1)^dim entries of a row are exactly its pattern).  Per row, on a group of G lanes (G = 4..32, the smallest power of
// two >= (p+1)^dim that fits a warp; wider rows give each lane several columns):
//
//   1-D tables at the point: IGABasis.value of the row's node (N, N', N'' of the p+1 functions that do not vanish there)
//   tensor products N, dN/du, d2N/du2 of the row's columns
//   rational weights: W, dW, d2W summed over the columns (group shuffles), Rationalize orders 0..2   (petigarat.f90.in:24-46)
//   geometry: X0, X1, X2 summed likewise; InverseMap orders 1..2                                    (petigamapinv.f90.in:28-52)
//   physical Laplacian of every column (petigamapshf.f90.in:36-61), the form, the closed-form position (seg_position)
//   A node that carries an IGASetBoundaryValue gets an identity row and F = the value (IGAComputeSystem only).
//
// Bytes: (p+1)^dim * 8 B of values per row plus 8 B of right-hand side; the tables read are a few hundred bytes per row and
// stay in L1/L2 (DESIGN 3.9).  Degrees are run-time values: one instantiation per (dim, geometry / no geometry).
#include <algorithm>

#include "pc_element.cuh"
#include "pc_plan.h"

namespace pc {

struct CollocParams {
  DevAxis ax[3];
  int ls[3], lw[3];          // owned node box
  int nown;
  const int64_t* rowbase;    // [nown+1]
  double* values;            // owned rows, or NULL (no matrix)
  double* rhs;               // [nown], or NULL (no vector)
  const double* X;           // geometry [ghost box][dim] or NULL
  const double* Wt;          // rational weights [ghost box] or NULL
  double c, k;               // K[a] = c N_a - k Lap N_a
  double fscale;             // F = fscale * prod sin(pi x_i)
  int fix;                   // identity rows on the faces with a value
  int vfix[3][2];
  double vval[3][2];
  int G;                     // lanes per row
};

// symmetric second-derivative slot (a <= b): (0,0),(1,1),(2,2) first, then (0,1),(0,2),(1,2) -- gen_sym_index of pc_quadg.cuh
template <int DIM>
__device__ __forceinline__ int colloc_sym(int a, int b) {
  if (a > b) { const int t = a; a = b; b = t; }
  if (a == b) return a;
  if (DIM == 2) return 2;
  return (a == 0) ? (b == 1 ? 3 : 4) : 5;
}

template <int N>
__device__ __forceinline__ void group_sum(double (&v)[N], int G) {
  for (int o = G >> 1; o > 0; o >>= 1)
#pragma unroll
    for (int i = 0; i < N; i++) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
}

template <int DIM, bool GEO>
__global__ void __launch_bounds__(256) colloc_kernel(const __grid_constant__ CollocParams cp) {
  constexpr int NS = DIM * (DIM + 1) / 2;
  const int G = cp.G, sub = threadIdx.x & (G - 1), rows_per_cta = 256 / G;
  int nA[3];
#pragma unroll
  for (int d = 0; d < 3; d++) nA[d] = d < DIM ? cp.ax[d].p + 1 : 1;
  const int nen = nA[0] * nA[1] * nA[2];
  // every group of a CTA runs the same number of iterations, so the full-warp shuffles below always see all 32 lanes
  for (int row0 = blockIdx.x * rows_per_cta; row0 < cp.nown; row0 += gridDim.x * rows_per_cta) {
    const int row = row0 + (int)threadIdx.x / G;
    const bool active = row < cp.nown;
    const int rr = active ? row : cp.nown - 1;   // inactive groups shadow the last row and store nothing
    int node[3], off[3], gr[3], W[3];
    const double* tb[3];
    {
      const int i0 = rr % cp.lw[0], i1 = (rr / cp.lw[0]) % cp.lw[1], i2 = rr / (cp.lw[0] * cp.lw[1]);
      node[0] = cp.ls[0] + i0; node[1] = cp.ls[1] + i1; node[2] = cp.ls[2] + i2;
    }
#pragma unroll
    for (int d = 0; d < 3; d++) {
      off[d] = cp.ax[d].offset[node[d]];
      gr[d] = node[d] - cp.ax[d].gs;
      W[d] = cp.ax[d].W[gr[d]];
      tb[d] = cp.ax[d].value + (size_t)node[d] * nA[d] * 5;   // nqp = 1: the table row of the node's own point
    }
    // parametric N, dN, d2N of column b
    auto basis = [&](int b, double& N0, double (&N1)[3], double (&N2)[6]) {
      const int a[3] = {b % nA[0], (b / nA[0]) % nA[1], b / (nA[0] * nA[1])};
      double v0[3] = {1, 1, 1}, v1[3] = {0, 0, 0}, v2[3] = {0, 0, 0};
#pragma unroll
      for (int d = 0; d < DIM; d++) { const double* t = tb[d] + a[d] * 5; v0[d] = t[0]; v1[d] = t[1]; v2[d] = t[2]; }
      N0 = v0[0] * v0[1] * v0[2];
#pragma unroll
      for (int d = 0; d < DIM; d++) {
        double g = (d == 0 ? v1[0] : v0[0]);
        if (DIM > 1) g *= (d == 1 ? v1[1] : v0[1]);
        if (DIM > 2) g *= (d == 2 ? v1[2] : v0[2]);
        N1[d] = g;
      }
#pragma unroll
      for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
        for (int b1 = a1; b1 < DIM; b1++) {
          double h = 1.0;
#pragma unroll
          for (int d = 0; d < DIM; d++) {
            const int cnt = (d == a1) + (d == b1);
            h *= (cnt == 0) ? v0[d] : (cnt == 1 ? v1[d] : v2[d]);
          }
          N2[colloc_sym<DIM>(a1, b1)] = h;
        }
    };
    auto gindex = [&](int b) {
      const int a0 = b % nA[0], a1 = (b / nA[0]) % nA[1], a2 = b / (nA[0] * nA[1]);
      return (off[0] + a0 - cp.ax[0].gs) + cp.ax[0].gw * ((off[1] + a1 - cp.ax[1].gs) + cp.ax[1].gw * (off[2] + a2 - cp.ax[2].gs));
    };

    // ---- Dirichlet: identity row (last face wins, as AddFixa) ----
    int fixed = 0;
    double fval = 0.0;
    if (cp.fix) {
#pragma unroll
      for (int d = 0; d < DIM; d++)
#pragma unroll
        for (int s = 0; s < 2; s++)
          if (cp.vfix[d][s] && node[d] == (s ? cp.ax[d].nnp - 1 : 0)) { fixed = 1; fval = cp.vval[d][s]; }
    }

    // ---- rational weights and geometry at the point (sums over the row's columns) ----
    double Wsum[1 + DIM + NS] = {};
    double Xs[GEO ? DIM : 1][1 + DIM + NS];
    double E[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, gs[6] = {0, 0, 0, 0, 0, 0}, hc[3] = {0, 0, 0};
    const bool rational = GEO && cp.Wt != nullptr, mapped = GEO && cp.X != nullptr;
    // rationalised R0, R1, R2 of column b (parametric derivatives)
    auto rbasis = [&](int b, double& R0, double (&R1)[3], double (&R2)[6]) {
      basis(b, R0, R1, R2);
      if (!rational) return;
      const double w = cp.Wt[gindex(b)], W0 = Wsum[0];
      const double r0 = w * R0 / W0;
      double r1[3] = {0, 0, 0};
#pragma unroll
      for (int d = 0; d < DIM; d++) r1[d] = (w * R1[d] - r0 * Wsum[1 + d]) / W0;
#pragma unroll
      for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
        for (int b1 = a1; b1 < DIM; b1++) {
          const int s = colloc_sym<DIM>(a1, b1);
          R2[s] = (w * R2[s] - r0 * Wsum[1 + DIM + s] - r1[a1] * Wsum[1 + b1] - r1[b1] * Wsum[1 + a1]) / W0;
        }
      R0 = r0;
#pragma unroll
      for (int d = 0; d < DIM; d++) R1[d] = r1[d];
    };
    double x[3] = {0, 0, 0};
#pragma unroll
    for (int d = 0; d < DIM; d++) x[d] = cp.ax[d].point[node[d]];
    if (GEO) {   // also on identity rows: the shuffles need every lane of the warp
      if (rational) {
#pragma unroll
        for (int i = 0; i < 1 + DIM + NS; i++) Wsum[i] = 0.0;
        for (int b = sub; b < nen; b += G) {
          double N0, N1[3], N2[6];
          basis(b, N0, N1, N2);
          const double w = cp.Wt[gindex(b)];
          Wsum[0] += w * N0;
#pragma unroll
          for (int d = 0; d < DIM; d++) Wsum[1 + d] += w * N1[d];
#pragma unroll
          for (int s = 0; s < NS; s++) Wsum[1 + DIM + s] += w * N2[s];
        }
        group_sum(Wsum, G);
      }
      if (mapped) {
#pragma unroll
        for (int i = 0; i < DIM; i++)
#pragma unroll
          for (int c = 0; c < 1 + DIM + NS; c++) Xs[i][c] = 0.0;
        for (int b = sub; b < nen; b += G) {
          double R0, R1[3], R2[6];
          rbasis(b, R0, R1, R2);
          const int gi = gindex(b);
#pragma unroll
          for (int i = 0; i < DIM; i++) {
            const double xb = cp.X[(size_t)gi * DIM + i];
            Xs[i][0] += xb * R0;
#pragma unroll
            for (int d = 0; d < DIM; d++) Xs[i][1 + d] += xb * R1[d];
#pragma unroll
            for (int s = 0; s < NS; s++) Xs[i][1 + DIM + s] += xb * R2[s];
          }
        }
#pragma unroll
        for (int i = 0; i < DIM; i++) group_sum(Xs[i], G);
        double X1[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
#pragma unroll
        for (int i = 0; i < DIM; i++) {
          x[i] = Xs[i][0];
#pragma unroll
          for (int d = 0; d < DIM; d++) X1[i][d] = Xs[i][1 + d];
        }
        inverse_map<DIM>(X1, E);
        // g[s] = sum_i E[a][i] E[b][i];  h[c] = - sum_k E[c][k] sum_{a,b} X2[k][a][b] g[a][b]   (petigamapinv.f90.in:47-52)
#pragma unroll
        for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
          for (int b1 = a1; b1 < DIM; b1++) {
            double s = 0.0;
#pragma unroll
            for (int i = 0; i < DIM; i++) s += E[a1][i] * E[b1][i];
            gs[colloc_sym<DIM>(a1, b1)] = s;
          }
        double hk[3] = {0, 0, 0};
#pragma unroll
        for (int kk = 0; kk < DIM; kk++) {
          double s = 0.0;
#pragma unroll
          for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
            for (int b1 = a1; b1 < DIM; b1++) {
              const int si = colloc_sym<DIM>(a1, b1);
              s += (a1 == b1 ? 1.0 : 2.0) * Xs[kk][1 + DIM + si] * gs[si];
            }
          hk[kk] = s;
        }
#pragma unroll
        for (int c = 0; c < DIM; c++) {
          double s = 0.0;
#pragma unroll
          for (int kk = 0; kk < DIM; kk++) s -= E[c][kk] * hk[kk];
          hc[c] = s;
        }
      }
    }
    if (!active) continue;

    // ---- the row: values at the closed-form positions, then the right-hand side ----
    if (cp.values) {
      const int64_t base = cp.rowbase[rr];
      const int self = (node[0] - off[0]) + nA[0] * ((node[1] - off[1]) + nA[1] * (node[2] - off[2]));
      for (int b = sub; b < nen; b += G) {
        const int a0 = b % nA[0], a1 = (b / nA[0]) % nA[1], a2 = b / (nA[0] * nA[1]);
        double v;
        if (fixed) v = (b == self) ? 1.0 : 0.0;
        else {
          double R0, R1[3], R2[6];
          if (GEO) rbasis(b, R0, R1, R2);
          else basis(b, R0, R1, R2);
          double lap = 0.0;
          if (mapped) {
#pragma unroll
            for (int p1 = 0; p1 < DIM; p1++)
#pragma unroll
              for (int q1 = p1; q1 < DIM; q1++) {
                const int s = colloc_sym<DIM>(p1, q1);
                lap += (p1 == q1 ? 1.0 : 2.0) * R2[s] * gs[s];
              }
#pragma unroll
            for (int d = 0; d < DIM; d++) lap += R1[d] * hc[d];
          } else {
#pragma unroll
            for (int d = 0; d < DIM; d++) lap += R2[d];
          }
          v = cp.c * R0 - cp.k * lap;
        }
        const int pos = seg_position(cp.ax[0].seg[gr[0] * kMaxW + a0], cp.ax[1].seg[gr[1] * kMaxW + a1], cp.ax[2].seg[gr[2] * kMaxW + a2], W[0], W[1]);
        cp.values[base + pos] = v;
      }
    }
    if (cp.rhs && sub == 0) {
      double f = fval;
      if (!fixed) {
        f = cp.fscale;
        if (f != 0.0)
#pragma unroll
          for (int d = 0; d < DIM; d++) f *= sinpi(x[d]);   // sin(pi x) without the stack frame of sin()'s large-argument reduction
      }
      cp.rhs[rr] = f;
    }
  }
}

int launch_collocation(petiga_cuda_plan* P, int slot, int form, double* values, double* rhs) {
  const Layout& L = P->L;
  CollocParams cp;
  memset(&cp, 0, sizeof(cp));
  for (int d = 0; d < 3; d++) { cp.ax[d] = P->dax[d]; cp.ls[d] = L.ax[d].ls; cp.lw[d] = L.ax[d].lw; }
  cp.nown = L.nown;
  cp.rowbase = P->d_rowbase;
  cp.values = slot_has_mat(slot) ? values : nullptr;
  cp.rhs = slot_has_vec(slot) ? rhs : nullptr;
  cp.X = P->d_X; cp.Wt = P->d_W;
  const double* prm = P->slots[slot].prm;
  if (form == PETIGA_FORM_LAPLACE_COLLOCATION) { cp.c = 0.0; cp.k = 1.0; cp.fscale = 0.0; }
  else { cp.c = prm[0]; cp.k = prm[1]; cp.fscale = prm[0] + prm[1] * L.dim * M_PI * M_PI; }
  cp.fix = 0;
  if (slot == PETIGA_SLOT_SYSTEM && P->has_bc) {   // IGAComputeVector/Matrix never fix (petigaksp.c:33-139)
    FixSide fs[3][2];
    memset(fs, 0, sizeof(fs));
    fill_fix_sides(P, false, fs);
    for (int d = 0; d < L.dim; d++)
      for (int s = 0; s < 2; s++)
        for (int k = 0; k < fs[d][s].vcount; k++)
          if (fs[d][s].vfield[k] == 0) { cp.vfix[d][s] = 1; cp.vval[d][s] = fs[d][s].vvalue[k]; cp.fix = 1; }
  }
  int nen = 1;
  for (int d = 0; d < L.dim; d++) nen *= L.ax[d].p + 1;
  int G = 4;
  while (G < nen && G < 32) G *= 2;
  cp.G = G;
  if (L.nown == 0) return 0;
  const int rows_per_cta = 256 / G;
  const int blocks = std::max(1, std::min((L.nown + rows_per_cta - 1) / rows_per_cta, P->num_sms * 16));
  const bool geo = P->d_X || P->d_W;
  switch (L.dim * 2 + (geo ? 1 : 0)) {
    case 2: colloc_kernel<1, false><<<blocks, 256, 0, P->stream>>>(cp); break;
    case 3: colloc_kernel<1, true><<<blocks, 256, 0, P->stream>>>(cp); break;
    case 4: colloc_kernel<2, false><<<blocks, 256, 0, P->stream>>>(cp); break;
    case 5: colloc_kernel<2, true><<<blocks, 256, 0, P->stream>>>(cp); break;
    case 6: colloc_kernel<3, false><<<blocks, 256, 0, P->stream>>>(cp); break;
    default: colloc_kernel<3, true><<<blocks, 256, 0, P->stream>>>(cp); break;
  }
  PC_CUDA(cudaGetLastError());
  P->launches++;
  return 0;
}

}  // namespace pc
