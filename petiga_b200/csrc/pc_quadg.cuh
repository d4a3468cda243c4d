// pc_quadg.cuh -- the generic quadrature kernel: everything about an element is a run-time quantity.
//
// The two tuned kernels (pc_quad.cuh, pc_quad2.cuh) are instantiated for one degree on all axes (p <= 4), dof <= 3, first
// derivatives on mapped geometry and the seven KSP/SNES/TS drivers.  The reference has none of these limits
// (test/makefile:23-40 sweeps dof 1..8 and mixed degrees; src/petigamapinv.f90.in:47-67, src/petigamapshf.f90.in:3-83 and
// src/petigarat.f90.in:3-57 carry second derivatives through NURBS and mapped geometry; src/petigats.c:182-477 and
// src/petigats2.c:23-175 add the IE/RHS/I2 drivers; src/petigaelem.c:427-447 visits boundary faces with full forms).  This
// kernel closes those holes with one CTA per element and the reference's own loop nest executed in parallel:
//
//   header     closure, gathers, Dirichlet/Neumann lists                (src/petigaelem.c:693-755,1166-1283)
//   per chunk of quadrature points:
//     tabulate parametric N, dN, d2N from the 1-D tables (or IGABasis.bnd_value on the face axis of a visited face)
//                                                                        (src/petiga3d.F90:32-233, src/petigaelem.c:788-868)
//     rationalize orders 0..2                                            (src/petigarat.f90.in:24-46)
//     geometry map X0, X1, X2; inverse map E1 and the contracted E2; unit normal, detS on a face
//                                                                        (petigamapgeo/petigamapinv.f90.in, src/petigaval.F90:45-99)
//     shape functions: N, grad_x N, Laplacian_x N                        (src/petigamapshf.f90.in:36-61)
//     state fields u, v, w, grad u, Laplacian u                          (src/petigaval.F90:182-251)
//     the form's coefficient tensors (pc_forms.cuh) and K_e += Psi^T (JW C Psi), F_e += Psi^T (JW f)   (src/petigapoint.c:451-465)
//   fix-up + closed-form scatter with red.global.add.f64                 (src/petigaelem.c:1360-1559)
//
// K_e lives in shared memory; when (nen*dof)^2 doubles do not fit, the element is processed in column panels (the chunk
// loop is repeated per panel).  It is a coverage kernel: correctness first, one element per CTA.
#pragma once
#include "pc_element.cuh"

namespace pc {

constexpr int kGenThreads = 256;
constexpr int kGenMaxN1 = 9;        // p <= 8 per axis
constexpr int kGenGeo = 72;         // doubles per quadrature point of geometry scratch

struct GenParams {
  KParams k;
  int pw;          // K_e panel width in columns (nen*dof when the whole element matrix fits)
  int ncomp;       // physical components kept: 1 + dim (+1: Laplacian)
  int nct;         // tabulated slots per (point, node): ncomp, or 1 + dim + dim(dim+1)/2 when full second derivatives are needed
  int full2;       // second derivatives go through the geometry / NURBS chain
  int nface0, nface1;   // face mode: element extents of the two face axes inside this rank's box
};

// shared-memory carve-up (offsets in doubles); same arithmetic on host and device
struct GenSmem {
  int tab, tb, cq, fq, jw, xq, geo, sq, ke, fe, ue, ve, we, xe, wn, fixval, flux, ufix, ints, total;
  __host__ __device__ GenSmem(int nen, int dof, int dim, int nct, int NA, int NV, int QC, int pw, int want_mat) {
    const int R = nen * dof;
    int o = 0;
    tab = o; o += QC * nct * nen;
    tb = o; o += want_mat ? QC * NA * nen * dof * dof : 0;
    cq = o; o += QC * dof * dof * (NA > 0 ? NA * NA : 1);
    fq = o; o += QC * dof * (NV > 0 ? NV : 1);
    jw = o; o += QC;
    xq = o; o += QC * 3;
    geo = o; o += QC * kGenGeo;
    sq = o; o += QC * dof * (3 + dim + 1);          // u, v, w, grad u, lap u
    ke = o; o += want_mat ? R * pw : 0;
    fe = o; o += R;
    ue = o; o += R; ve = o; o += R; we = o; o += R;
    xe = o; o += nen * dim; wn = o; o += nen;
    fixval = o; o += R; flux = o; o += R; ufix = o; o += R;
    ints = o; o += (nen + R + 3 * kGenMaxN1 * kGenMaxN1 + 3 * kGenMaxN1 + 8) / 2 + 2;
    total = o;
  }
};

__host__ __device__ inline int gen_nsym(int dim) { return dim * (dim + 1) / 2; }
// symmetric pair index (a <= b) -> slot; slot -> pair
__host__ __device__ inline int gen_sym_index(int dim, int a, int b) {
  if (a > b) { int t = a; a = b; b = t; }
  // order: (0,0),(1,1),(2,2),(0,1),(0,2),(1,2): diagonal first, so that slot d is d2/du_d2
  if (a == b) return a;
  if (dim == 2) return 2;
  return (a == 0) ? (b == 1 ? 3 : 4) : 5;
}

template <int DIM>
__global__ void __launch_bounds__(kGenThreads) quad_gen_kernel(const __grid_constant__ GenParams gp) {
  const KParams& prm = gp.k;
  extern __shared__ double sm[];
  const int T = kGenThreads, lt = threadIdx.x;
  const int dof = prm.dof;
  int nA[3], nQ[3];
#pragma unroll
  for (int d = 0; d < 3; d++) { nA[d] = prm.ax[d].nen; nQ[d] = prm.ax[d].nqp; }
  const int fax = prm.face_axis, fsd = prm.face_side;
  const bool face = fax >= 0;
  if (face) nQ[fax] = 1;                                   // nqp /= NQ[axis]; NQ[axis] = 1 (petigaelem.c:813-817)
  const int nen = nA[0] * nA[1] * nA[2], nqp = nQ[0] * nQ[1] * nQ[2], R = nen * dof;
  const int NA = prm.mc1 - prm.mc0, NV = prm.vc1 - prm.vc0, QC = prm.qc, pw = gp.pw, nct = gp.nct, ncomp = gp.ncomp;
  const bool want_mat = NA > 0 && slot_has_mat(prm.slot), want_vec = slot_has_vec(prm.slot);
  const GenSmem lay(nen, dof, DIM, nct, NA, NV, QC, pw, want_mat);
  double *Tab = sm + lay.tab, *Tb = sm + lay.tb, *Cq = sm + lay.cq, *Fq = sm + lay.fq, *JW = sm + lay.jw, *Xq = sm + lay.xq, *Geo = sm + lay.geo;
  double *Sq = sm + lay.sq, *Ke = sm + lay.ke, *Fe = sm + lay.fe, *Ue = sm + lay.ue, *Ve = sm + lay.ve, *We = sm + lay.we, *Xe = sm + lay.xe;
  double *Wn = sm + lay.wn, *FixVal = sm + lay.fixval, *Flux = sm + lay.flux, *UFix = sm + lay.ufix;
  int* lrow = reinterpret_cast<int*>(sm + lay.ints);
  int* fixflag = lrow + nen;
  uint32_t* segs = reinterpret_cast<uint32_t*>(fixflag + R);          // [3][kGenMaxN1*kGenMaxN1]
  int* Wd = reinterpret_cast<int*>(segs + 3 * kGenMaxN1 * kGenMaxN1);   // [3][kGenMaxN1]

  const bool mapped = prm.X != nullptr, rational = prm.Wt != nullptr;
  const bool state = prm.needs_state && prm.U != nullptr;
  const bool hasV = slot_has_v(prm.slot) && prm.V != nullptr, hasW = slot_has_w(prm.slot) && prm.Wv != nullptr;
  const bool i2 = slot_is_i2(prm.slot);
  const int fixkind = slot_fix_kind(prm.slot);
  const int nsym = gen_nsym(DIM);
  const bool order2 = ncomp > DIM + 1, full2 = gp.full2 != 0;

  // ---- element: IGANextElement (interior) or the elements of the visited face inside this rank's box ----
  int ID[3] = {0, 0, 0};
  {
    int idx = blockIdx.x;
    if (!face) element_id(prm.ax, idx, ID);
    else {
#pragma unroll
      for (int d = 0; d < 3; d++) {
        if (d == fax) { ID[d] = fsd ? prm.ax[d].nel - 1 : 0; continue; }
        const int c = idx % prm.ax[d].ew; idx /= prm.ax[d].ew; ID[d] = c + prm.ax[d].es;
      }
    }
  }
  const double Lax[3] = {prm.ax[0].detJac[ID[0]], prm.ax[1].detJac[ID[1]], prm.ax[2].detJac[ID[2]]};   // IGAPointFormScale

  // ---------------- header ----------------
  for (int a = lt; a < nen; a += T) {
    const int ai[3] = {a % nA[0], (a / nA[0]) % nA[1], a / (nA[0] * nA[1])};
    int gidx = 0, mul = 1;
#pragma unroll
    for (int d = 0; d < 3; d++) { gidx += (prm.ax[d].offset[ID[d]] + ai[d] - prm.ax[d].gs) * mul; mul *= prm.ax[d].gw; }
    const int lr = prm.localrow[gidx];
    lrow[a] = lr;
    if (mapped) {
#pragma unroll
      for (int i = 0; i < DIM; i++) Xe[a * DIM + i] = prm.X[(size_t)gidx * DIM + i];
    }
    Wn[a] = rational ? prm.Wt[gidx] : 1.0;
    int onfix[kMaxDof];
    double vfix[kMaxDof], vflux[kMaxDof];
    for (int c = 0; c < dof; c++) { onfix[c] = 0; vfix[c] = 0.0; vflux[c] = 0.0; }
    if (prm.any_bc) {   // BuildFix / AddFixa / AddFlux (petigaelem.c:1166-1283): last face wins for values, loads accumulate
#pragma unroll
      for (int d = 0; d < DIM; d++) {
        if (prm.ax[d].periodic) continue;
        for (int s = 0; s < 2; s++) {
          const FixSide& fs = prm.bc[d][s];
          if (!(fs.vcount || fs.lcount)) continue;
          if (ID[d] != (s ? prm.ax[d].nel - 1 : 0)) continue;
          if (ai[d] != (s ? nA[d] - 1 : 0)) continue;
          for (int k = 0; k < fs.vcount; k++) {
            const int c = fs.vfield[k];
            onfix[c] = 1;
            vfix[c] = prm.fixtable ? prm.fixtable[(size_t)gidx * dof + c] : fs.vvalue[k];
          }
          if (fs.lcount) {
            double A = 1.0;
            if (DIM > 1) {
              for (int e = 0; e < DIM; e++) if (e != d) A *= prm.ax[e].detJac[ID[e]] / (double)nA[e];
              if (prm.face_dS[d][s]) {
                const int f0 = (d == 0) ? 1 : 0, f1 = (d == 2) ? 1 : 2;
                const int fidx = (ID[f0] - prm.ax[f0].es) + ((DIM > 2) ? prm.ax[f0].ew * (ID[f1] - prm.ax[f1].es) : 0);
                A *= prm.face_dS[d][s][fidx];
              } else A *= (DIM == 2) ? 2.0 : 4.0;
            }
            for (int k = 0; k < fs.lcount; k++) vflux[fs.lfield[k]] += fs.lvalue[k] * A;
          }
        }
      }
    }
    for (int c = 0; c < dof; c++) {
      const int idx = a * dof + c;
      double u = 0.0, v = 0.0, w = 0.0;
      if (state) u = prm.U[(size_t)lr * dof + c];
      if (hasV) v = prm.V[(size_t)lr * dof + c];
      if (hasW) w = prm.Wv[(size_t)lr * dof + c];
      fixflag[idx] = onfix[c]; FixVal[idx] = vfix[c]; Flux[idx] = vflux[c]; UFix[idx] = u;
      if (onfix[c]) {   // FixValues(U) / DelValues(V); third vector: DelValues(A) for I2 (petigats2.c:68), FixValues(U0) for IE (petigats.c:228)
        u = vfix[c]; v = 0.0; w = i2 ? 0.0 : vfix[c];
      }
      Ue[idx] = u; Ve[idx] = v; We[idx] = w; Fe[idx] = 0.0;
    }
  }
  for (int t = lt; t < 3 * kGenMaxN1 * kGenMaxN1; t += T) {
    const int d = t / (kGenMaxN1 * kGenMaxN1), r = t - d * kGenMaxN1 * kGenMaxN1, ia = r / kGenMaxN1, ib = r - ia * kGenMaxN1;
    uint32_t s = 0x00000100u;
    if (d < DIM && ia < nA[d] && ib < nA[d]) {
      const int g = prm.ax[d].offset[ID[d]] + ia - prm.ax[d].gs;
      s = prm.ax[d].seg[g * kMaxW + ib - ia + prm.ax[d].lo[g]];
      if (ib == 0) Wd[d * kGenMaxN1 + ia] = prm.ax[d].W[g];
    } else if (ib == 0 && ia < kGenMaxN1) Wd[d * kGenMaxN1 + ia] = 1;
    segs[t] = s;
  }
  __syncthreads();

  // 1-D table of axis d at local point q: IGABasis.value, or bnd_value on the face axis (one point)
  auto tab1 = [&](int d, int q, int a) -> const double* {
    if (face && d == fax) return prm.bnd_value[d][fsd] + (size_t)a * 5;
    return prm.ax[d].value + ((size_t)(ID[d] * prm.ax[d].nqp + q) * nA[d] + a) * 5;
  };

  const int Ccols = R;
  for (int pc0 = 0; pc0 < (want_mat ? Ccols : 1); pc0 += pw) {      // column panels of K_e (one pass when it fits)
    const int pcols = want_mat ? min(pw, Ccols - pc0) : 0;
    const bool first_panel = (pc0 == 0);
    if (want_mat) for (int t = lt; t < R * pcols; t += T) Ke[t] = 0.0;
    __syncthreads();
    for (int q0 = 0; q0 < nqp; q0 += QC) {
      const int nq = min(QC, nqp - q0);
      // ---- (1) parametric tabulation ----
      for (int t = lt; t < nq * nen; t += T) {
        const int ql = t / nen, a = t - ql * nen, q = q0 + ql;
        const int qi[3] = {q % nQ[0], (q / nQ[0]) % nQ[1], q / (nQ[0] * nQ[1])};
        const int ai[3] = {a % nA[0], (a / nA[0]) % nA[1], a / (nA[0] * nA[1])};
        double v0[3] = {1, 1, 1}, v1[3] = {0, 0, 0}, v2[3] = {0, 0, 0};
#pragma unroll
        for (int d = 0; d < DIM; d++) { const double* tb = tab1(d, qi[d], ai[d]); v0[d] = tb[0]; v1[d] = tb[1]; v2[d] = tb[2]; }
        double* out = Tab + (size_t)ql * nct * nen + a;
        out[0] = v0[0] * v0[1] * v0[2];
#pragma unroll
        for (int d = 0; d < DIM; d++) {
          double g = (d == 0 ? v1[0] : v0[0]);
          if (DIM > 1) g *= (d == 1 ? v1[1] : v0[1]);
          if (DIM > 2) g *= (d == 2 ? v1[2] : v0[2]);
          out[(1 + d) * nen] = g;
        }
        if (order2) {
          if (!full2) {
            double lap = v2[0] * v0[1] * v0[2];
            if (DIM > 1) lap += v0[0] * v2[1] * v0[2];
            if (DIM > 2) lap += v0[0] * v0[1] * v2[2];
            out[(1 + DIM) * nen] = lap;
          } else {
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
                out[(1 + DIM + gen_sym_index(DIM, a1, b1)) * nen] = h;
              }
          }
        }
      }
      __syncthreads();
      double* G0 = Geo;   // per point ql: Geo[ql*kGenGeo + ...]
      // layout inside a point's scratch: [0] W0, [1..3] W1, [4..9] W2, [10..18] X1 (then E), [19..36] X2[i][s], [37..42] g[s], [43..45] h[c],
      //                                  [46] detX, [47..49] normal, [50] detS, [51] hn
      if (rational) {   // ---- (2) Rationalize (petigarat.f90.in:24-46) ----
        const int nsum = 1 + DIM + (full2 ? nsym : 0);
        for (int t = lt; t < nq * nsum; t += T) {
          const int ql = t / nsum, c = t - ql * nsum;
          const double* ps = Tab + ((size_t)ql * nct + c) * nen;
          double s = 0.0;
          for (int a = 0; a < nen; a++) s += Wn[a] * ps[a];
          G0[ql * kGenGeo + (c == 0 ? 0 : (c <= DIM ? c : 4 + (c - 1 - DIM)))] = s;
        }
        __syncthreads();
        for (int t = lt; t < nq * nen; t += T) {
          const int ql = t / nen, a = t - ql * nen;
          double* ps = Tab + (size_t)ql * nct * nen + a;
          const double* gq = G0 + ql * kGenGeo;
          const double w = Wn[a], W0 = gq[0];
          const double R0 = w * ps[0] / W0;
          double R1[3] = {0, 0, 0};
#pragma unroll
          for (int d = 0; d < DIM; d++) R1[d] = (w * ps[(1 + d) * nen] - R0 * gq[1 + d]) / W0;
          if (full2) {
#pragma unroll
            for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
              for (int b1 = a1; b1 < DIM; b1++) {
                const int s = gen_sym_index(DIM, a1, b1);
                ps[(1 + DIM + s) * nen] = (w * ps[(1 + DIM + s) * nen] - R0 * gq[4 + s] - R1[a1] * gq[1 + b1] - R1[b1] * gq[1 + a1]) / W0;
              }
          }
          ps[0] = R0;
#pragma unroll
          for (int d = 0; d < DIM; d++) ps[(1 + d) * nen] = R1[d];
        }
        __syncthreads();
      }
      if (mapped) {   // ---- (3) GeometryMap: X0, X1, X2 (petigamapgeo.f90.in:28-57) ----
        const int per = 1 + DIM + (full2 ? nsym : 0);
        for (int t = lt; t < nq * DIM * per; t += T) {
          const int ql = t / (DIM * per), r = t - ql * DIM * per, i = r / per, c = r - i * per;
          const double* ps = Tab + ((size_t)ql * nct + c) * nen;
          double s = 0.0;
          for (int a = 0; a < nen; a++) s += Xe[a * DIM + i] * ps[a];
          double* gq = G0 + ql * kGenGeo;
          if (c == 0) Xq[ql * 3 + i] = s;
          else if (c <= DIM) gq[10 + i * DIM + (c - 1)] = s;          // X1[i][d]
          else gq[19 + i * 6 + (c - 1 - DIM)] = s;                   // X2[i][s]
        }
        __syncthreads();
      }
      // ---- (4) per point: inverse map, contracted second-order terms, normal, weights ----
      for (int ql = lt; ql < nq; ql += T) {
        const int q = q0 + ql;
        const int qi[3] = {q % nQ[0], (q / nQ[0]) % nQ[1], q / (nQ[0] * nQ[1])};
        double* gq = G0 + ql * kGenGeo;
        double w = 1.0, J = 1.0, x[3] = {0, 0, 0};
#pragma unroll
        for (int d = 0; d < DIM; d++) {
          if (face && d == fax) { x[d] = prm.bnd_point[d][fsd]; continue; }     // bnd_weight = bnd_detJac = 1 (petigaelem.c:788)
          w *= prm.ax[d].weight[ID[d] * prm.ax[d].nqp + qi[d]];
          J *= Lax[d];
          x[d] = prm.ax[d].point[ID[d] * prm.ax[d].nqp + qi[d]];
        }
        double E[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}, nrm[3] = {0, 0, 0}, dS = 1.0, det = 1.0;
        if (mapped) {
          double X1[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
#pragma unroll
          for (int i = 0; i < DIM; i++)
#pragma unroll
            for (int d = 0; d < DIM; d++) X1[i][d] = gq[10 + i * DIM + d];
          det = inverse_map<DIM>(X1, E);
#pragma unroll
          for (int i = 0; i < DIM; i++) x[i] = Xq[ql * 3 + i];
          if (face) {   // IGA_GetNormal (src/petigaval.F90:45-99)
            if (DIM == 1) { nrm[0] = 1.0; dS = 1.0; }
            else if (DIM == 2) {
              const int dd = (fax == 0) ? 1 : 0; const double sg = (fax == 0) ? 1.0 : -1.0;
              const double t0 = sg * X1[0][dd], t1 = sg * X1[1][dd];
              nrm[0] = t1; nrm[1] = -t0;
              dS = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1]); nrm[0] /= dS; nrm[1] /= dS;
            } else {
              const int ds = (fax + 1) % 3, dt = (fax + 2) % 3;
              const double s0 = X1[0][ds], s1 = X1[1][ds], s2 = X1[2][ds], t0 = X1[0][dt], t1 = X1[1][dt], t2 = X1[2][dt];
              nrm[0] = s1 * t2 - s2 * t1; nrm[1] = s2 * t0 - s0 * t2; nrm[2] = s0 * t1 - s1 * t0;
              dS = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1] + nrm[2] * nrm[2]); nrm[0] /= dS; nrm[1] /= dS; nrm[2] /= dS;
            }
            if (fsd == 0) { nrm[0] = -nrm[0]; nrm[1] = -nrm[1]; nrm[2] = -nrm[2]; }
          }
        } else if (face) { nrm[fax] = fsd ? 1.0 : -1.0; }      // petigaelem.c:1018-1021
        // detJac *= detX in the interior, *= detS on a face (petigaelem.c:1024-1029)
        JW[ql] = (J * (mapped ? (face ? dS : det) : 1.0)) * w;
#pragma unroll
        for (int d = 0; d < 3; d++) Xq[ql * 3 + d] = x[d];
#pragma unroll
        for (int a = 0; a < 3; a++)
#pragma unroll
          for (int i = 0; i < 3; i++) gq[10 + a * 3 + i] = E[a][i];          // E[a][i] = du_a/dx_i, stride 3 from here on
        if (full2 && mapped) {
          // g[s] = sum_i E[a][i] E[b][i];  h[c] = sum_i E2(i,i,c) = - sum_k E[c][k] sum_{a,b} X2[k][a][b] g[a][b]   (petigamapinv.f90.in:47-52)
          double gs[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
          for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
            for (int b1 = a1; b1 < DIM; b1++) {
              double s = 0.0;
#pragma unroll
              for (int i = 0; i < DIM; i++) s += E[a1][i] * E[b1][i];
              gs[gen_sym_index(DIM, a1, b1)] = s;
            }
          double hk[3] = {0, 0, 0};
#pragma unroll
          for (int k = 0; k < DIM; k++) {
            double s = 0.0;
#pragma unroll
            for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
              for (int b1 = a1; b1 < DIM; b1++) {
                const int si = gen_sym_index(DIM, a1, b1);
                s += (a1 == b1 ? 1.0 : 2.0) * gq[19 + k * 6 + si] * gs[si];
              }
            hk[k] = s;
          }
#pragma unroll
          for (int c = 0; c < DIM; c++) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < DIM; k++) s -= E[c][k] * hk[k];
            gq[43 + c] = s;
          }
#pragma unroll
          for (int s = 0; s < 6; s++) gq[37 + s] = gs[s];
        }
        gq[46] = det;
        gq[47] = nrm[0]; gq[48] = nrm[1]; gq[49] = nrm[2]; gq[50] = dS;
        {   // NormalMeshSize (demo/NitscheMethod.c:58-67): G = E / L (IGAPointFormInvGradGeomMap), h = 2 / |G n|
          double nn = 0.0;
#pragma unroll
          for (int a = 0; a < DIM; a++) {
            double s = 0.0;
#pragma unroll
            for (int i = 0; i < DIM; i++) s += E[a][i] / Lax[a] * nrm[i];
            nn += s * s;
          }
          gq[51] = face ? 2.0 / sqrt(nn) : 0.0;
        }
      }
      __syncthreads();
      // ---- (5) ShapeFunctions orders 1 and (contracted) 2 (petigamapshf.f90.in:36-61) ----
      if (mapped) {
        for (int t = lt; t < nq * nen; t += T) {
          const int ql = t / nen, a = t - ql * nen;
          double* ps = Tab + (size_t)ql * nct * nen + a;
          const double* gq = G0 + ql * kGenGeo;
          double r1[3] = {0, 0, 0}, gx[3] = {0, 0, 0};
#pragma unroll
          for (int d = 0; d < DIM; d++) r1[d] = ps[(1 + d) * nen];
#pragma unroll
          for (int i = 0; i < DIM; i++)
#pragma unroll
            for (int d = 0; d < DIM; d++) gx[i] += r1[d] * gq[10 + d * 3 + i];
          if (full2) {
            double lap = 0.0;
#pragma unroll
            for (int a1 = 0; a1 < DIM; a1++)
#pragma unroll
              for (int b1 = a1; b1 < DIM; b1++) {
                const int s = gen_sym_index(DIM, a1, b1);
                lap += (a1 == b1 ? 1.0 : 2.0) * ps[(1 + DIM + s) * nen] * gq[37 + s];
              }
#pragma unroll
            for (int d = 0; d < DIM; d++) lap += r1[d] * gq[43 + d];
            ps[(1 + DIM) * nen] = lap;
          }
#pragma unroll
          for (int i = 0; i < DIM; i++) ps[(1 + i) * nen] = gx[i];
        }
        __syncthreads();
      }
      // ---- (6) fields at the points (petigaval.F90:182-251) ----
      const int per = 3 + DIM + 1;     // u, v, w, grad, lap
      if (state) {
        for (int t = lt; t < nq * dof * per; t += T) {
          const int ql = t / (dof * per), r = t - ql * dof * per, i = r / per, wsel = r - i * per;
          const int comp = (wsel <= 2) ? 0 : (wsel - 2);
          double s = 0.0;
          if (comp < ncomp) {
            const double* ps = Tab + ((size_t)ql * nct + comp) * nen;
            const double* src = (wsel == 1) ? Ve : (wsel == 2 ? We : Ue);
            for (int a = 0; a < nen; a++) s += ps[a] * src[a * dof + i];
          }
          Sq[ql * dof * per + r] = s;
        }
        __syncthreads();
      }
      // ---- (7) coefficient tensors of the form at the points ----
      for (int ql = lt; ql < nq; ql += T) {
        const double* gq = G0 + ql * kGenGeo;
        QPoint qp;
        qp.atboundary = face ? 1 : 0;
        qp.maxdeg = prm.maxdeg;
        qp.hn = gq[51];
#pragma unroll
        for (int d = 0; d < 3; d++) { qp.x[d] = Xq[ql * 3 + d]; qp.normal[d] = gq[47 + d]; }
        for (int i = 0; i < dof; i++) {
          qp.u[i] = qp.v[i] = qp.w[i] = qp.d2u[i] = 0.0;
          qp.gu[i][0] = qp.gu[i][1] = qp.gu[i][2] = 0.0;
          if (state) {
            const double* s = Sq + ql * dof * per + i * per;
            qp.u[i] = s[0]; qp.v[i] = s[1]; qp.w[i] = s[2];
#pragma unroll
            for (int d = 0; d < DIM; d++) qp.gu[i][d] = s[3 + d];
            qp.d2u[i] = s[3 + DIM];
          }
        }
        double* C = Cq + (size_t)ql * dof * dof * (NA > 0 ? NA * NA : 1);
        double* fv = Fq + (size_t)ql * dof * (NV > 0 ? NV : 1);
        for (int k = 0; k < dof * dof * NA * NA; k++) C[k] = 0.0;
        for (int k = 0; k < dof * NV; k++) fv[k] = 0.0;
        form_coefficients_rt<DIM>(prm.form, prm.slot, prm.prm, prm.shift, prm.t, qp, dof, NA, NV, NA ? C : nullptr, NV ? fv : nullptr);
      }
      __syncthreads();
      // ---- (8) B operand T[(q,al)][(b,j,i)] = JW_q sum_be C_q[i][j][al][be] Psi_be(b,q); element vector ----
      if (want_mat) {
        const int N = nen * dof * dof;
        for (int t = lt; t < nq * N; t += T) {
          const int ql = t / N, n = t - ql * N;
          const int b = n / (dof * dof), j = (n / dof) % dof, i = n % dof;
          const double* C = Cq + (size_t)ql * dof * dof * NA * NA + (size_t)(i * dof + j) * NA * NA;
          const double* ps = Tab + ((size_t)ql * nct + prm.mc0) * nen + b;
          const double jw = JW[ql];
          double* out = Tb + (size_t)ql * NA * N + n;
          for (int al = 0; al < NA; al++) {
            double s = 0.0;
            for (int be = 0; be < NA; be++) s += C[al * NA + be] * ps[be * nen];
            out[al * N] = s * jw;
          }
        }
      }
      if (want_vec && NV > 0 && first_panel)
        for (int t = lt; t < R; t += T) {
          const int a = t / dof, i = t - a * dof;
          double s = 0.0;
          for (int ql = 0; ql < nq; ql++) {
            const double* fv = Fq + (size_t)ql * dof * NV + i * NV;
            const double* ps = Tab + ((size_t)ql * nct + prm.vc0) * nen + a;
            double sq = 0.0;
            for (int al = 0; al < NV; al++) sq += ps[al * nen] * fv[al];
            s += sq * JW[ql];
          }
          Fe[t] += s;
        }
      __syncthreads();
      // ---- (9) K_e(panel) += Psi^T T over this chunk: a thread owns the entries t, t + T, ... of the panel ----
      if (want_mat) {
        const int N = nen * dof * dof;
        for (int t = lt; t < R * pcols; t += T) {
          const int r = t / pcols, cl = t - r * pcols, c = pc0 + cl;
          const int a = r / dof, i = r - a * dof, b = c / dof, j = c - b * dof;
          const int n = (b * dof + j) * dof + i;
          double s = 0.0;
          for (int ql = 0; ql < nq; ql++) {
            const double* pa = Tab + ((size_t)ql * nct + prm.mc0) * nen + a;
            const double* pb = Tb + (size_t)ql * NA * N + n;
            for (int al = 0; al < NA; al++) s += pa[al * nen] * pb[al * N];
          }
          Ke[t] += s;
        }
      }
      __syncthreads();
    }
    // ---------------- fix-up (petigaelem.c:1360-1389,1483-1501) + scatter (:1525-1559) of this panel ----------------
    if (want_mat) {
      const bool fixing = (fixkind == 1 || fixkind == 3) && prm.any_bc;
      for (int t = lt; t < R * pcols; t += T) {
        const int r = t / pcols, cl = t - r * pcols, c = pc0 + cl;
        const int a = r / dof, i = r - a * dof, b = c / dof, j = c - b * dof;
        double v = Ke[t];
        if (fixing) {
          const bool fr = fixflag[r], fc = fixflag[c];
          if (fr || fc) {
            if (fixkind == 1 && fc && !fr) atomicAdd(&Fe[r], -v * FixVal[c]);
            v = (r == c && !face) ? 1.0 : 0.0;       // a visited face adds to the element the interior pass already fixed
          }
        }
        if (v == 0.0) continue;
        const int ai[3] = {a % nA[0], (a / nA[0]) % nA[1], a / (nA[0] * nA[1])};
        const int bi[3] = {b % nA[0], (b / nA[0]) % nA[1], b / (nA[0] * nA[1])};
        const int W0 = Wd[ai[0]], W1 = Wd[kGenMaxN1 + ai[1]], W2 = Wd[2 * kGenMaxN1 + ai[2]];
        const int pos = seg_position(segs[ai[0] * kGenMaxN1 + bi[0]], segs[kGenMaxN1 * kGenMaxN1 + ai[1] * kGenMaxN1 + bi[1]],
                                     segs[2 * kGenMaxN1 * kGenMaxN1 + ai[2] * kGenMaxN1 + bi[2]], W0, W1);
        const int lr = lrow[a];
        int64_t base = prm.rowbase[lr];
        double* dst = prm.values;
        if (lr >= prm.nown) { dst = prm.ghost_values; base -= prm.nnz_own; }
        atomicAdd(dst + value_offset(base, pos, dof, prm.block, i, j, W0 * W1 * W2), v);
      }
    }
    __syncthreads();
  }
  if (want_vec) {
    for (int t = lt; t < R; t += T) {
      const int a = t / dof, i = t - a * dof;
      double F = Fe[t];
      if (fixkind == 1) { if (!face) F += Flux[t]; if (fixflag[t]) F = face ? 0.0 : FixVal[t]; }
      else if (fixkind == 2) { if (!face) F -= Flux[t]; if (fixflag[t]) F = face ? 0.0 : UFix[t] - FixVal[t]; }
      if (F != 0.0) atomicAdd(&prm.rhs[(size_t)lrow[a] * dof + i], F);
    }
  }
}

}  // namespace pc
