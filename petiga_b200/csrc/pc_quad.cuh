// pc_quad.cuh -- the per-element quadrature kernel (the reference's formulation, re-designed for an SM).
//
// Replaces, for a batch of elements per CTA, the whole body of the reference's element loop:
//   IGANextElement/BuildClosure   src/petigaelem.c:375-410,693-755    -> header phase (closure, gathers)
//   IGAElementBuildFix            src/petigaelem.c:1166-1283          -> fix lists, one thread per local dof
//   IGAElementBuildTabulation     src/petigaelem.c:794-1033 + src/petiga{1,2,3}d.F90 (K2-K7)
//                                                                     -> tabulate/rationalize/geometry phases,
//                                                                        only the components the form reads
//   form callback + IGAPointAddMat src/petigapoint.c:414-492 (K9)     -> coefficient tensors (pc_forms.cuh) and one
//                                                                        register-tiled FP64 contraction
//                                                                        K_e = Psi^T (JW C Psi)  from shared memory
//   IGAElementFix{System,Function,Jacobian} src/petigaelem.c:1360-1501 -> applied on the register tiles
//   IGAElementAssembleMat/Vec (MatSetValuesLocal ADD_VALUES) :1525-1559 -> closed-form CSR position + red.global.add.f64
#pragma once
#include "pc_element.cuh"

namespace pc {

__host__ __device__ constexpr int ipow(int b, int e) { return e <= 0 ? 1 : b * ipow(b, e - 1); }

template <int DIM, int P, int DOF, int TM>
struct QCfg {
  static constexpr int NEN1 = P + 1;
  static constexpr int NEN = ipow(NEN1, DIM);
  static constexpr int M = NEN;
  static constexpr int N = NEN * DOF * DOF;
  static constexpr int TN = TM * DOF;
  static constexpr int GM = M / TM, GN = N / TN, G = GM * GN;
  static_assert(M % TM == 0 && N % TN == 0, "tile must divide the element matrix");
  // Columns of a thread's tile are interleaved across the GN threads of a tile row in chunks of CH doubles, so that the
  // threads of a warp read consecutive 8/16-byte words of the B operand (no shared-memory bank conflicts).
  static constexpr int CH = (TN % 2 == 0) ? 2 : 1;
  __host__ __device__ static constexpr int col(int tx, int j) { return ((j / CH) * GN + tx) * CH + (j % CH); }
};

// shared-memory carve-up of one element slot (offsets in doubles); identical on host and device
struct QSmem {
  int psi, bs, cq, fq, jw, geo, xq, sq, fe, ue, ve, xe, we, fixval, flux, ufix, ints, total;
  __host__ __device__ QSmem(int M, int N, int dim, int dof, int NC, int NA, int NV, int QC, int nen1, int G = 0) {
    int o = 0;
    psi = o; o += QC * NC * M;
    bs = o; o += QC * NA * N;
    cq = o; o += QC * dof * dof * NA * NA;
    fq = o; o += QC * dof * (NV > 0 ? NV : 1);
    jw = o; o += QC;
    geo = o; o += QC * (dim * dim + 1 + 1 + dim);       // X1 (then E1), detX, W0, W1[dim]
    xq = o; o += QC * 3;
    sq = o; o += QC * dof * (2 + dim + 1);              // u, v, grad u, lap u
    fe = o; o += M * dof;
    ue = o; o += M * dof;
    ve = o; o += M * dof;
    xe = o; o += M * dim;
    we = o; o += M;
    fixval = o; o += M * dof;
    flux = o; o += M * dof;
    ufix = o; o += M * dof;
    ints = o; o += (M + M * dof + 3 * nen1 * nen1 + 3 * nen1 + 8 + 1) / 2 + 1;   // lrow, fixflag, segs, Wd, ID
    total = o;
    // several small elements share a CTA, G threads each: with a slot stride = G (mod 16 doubles) the threads of a warp that
    // belong to consecutive elements hit consecutive banks, as if the per-element arrays were packed back to back
    // (ncu r1_ncu_quad_kernel_cfg5: the T-builder's loads/stores ran at 2x their ideal wavefronts with the unpadded stride)
    if (G > 0 && G < 32) while (total % 16 != G % 16) total++;
  }
};

__device__ __forceinline__ double atomic_add_shared(double* addr, double v) { return atomicAdd(addr, v); }

template <int DIM, int P, int DOF, int TM>
__global__ void __launch_bounds__((QCfg<DIM, P, DOF, TM>::G > 256) ? ((QCfg<DIM, P, DOF, TM>::G + 31) / 32 * 32) : 256)
quad_kernel(const __grid_constant__ KParams prm) {
  using Cfg = QCfg<DIM, P, DOF, TM>;
  constexpr int NEN1 = Cfg::NEN1, M = Cfg::M, N = Cfg::N, TN = Cfg::TN, GN = Cfg::GN, G = Cfg::G;
  extern __shared__ double smem_all[];
  const int NC = prm.c1 - prm.c0, NA = prm.mc1 - prm.mc0, NV = prm.vc1 - prm.vc0, QC = prm.qc;
  const QSmem lay(M, N, DIM, DOF, NC, NA, NV, QC, NEN1, G);
  const int grp = threadIdx.x / G, lt = threadIdx.x - grp * G;
  const bool ingrp = grp < prm.epb;
  const int elem = blockIdx.x * prm.epb + grp;
  const bool valid = ingrp && elem < prm.nelem;
  double* sm = smem_all + (size_t)(ingrp ? grp : 0) * lay.total;
  double *Psi = sm + lay.psi, *Bs = sm + lay.bs, *Cq = sm + lay.cq, *Fq = sm + lay.fq, *JW = sm + lay.jw, *Geo = sm + lay.geo;
  double *Xq = sm + lay.xq, *Sq = sm + lay.sq, *Fe = sm + lay.fe, *Ue = sm + lay.ue, *Ve = sm + lay.ve, *Xe = sm + lay.xe;
  double *We = sm + lay.we, *FixVal = sm + lay.fixval, *Flux = sm + lay.flux, *UFix = sm + lay.ufix;
  int* lrow = reinterpret_cast<int*>(sm + lay.ints);
  int* fixflag = lrow + M;
  uint32_t* segs = reinterpret_cast<uint32_t*>(fixflag + M * DOF);
  int* Wd = reinterpret_cast<int*>(segs + 3 * NEN1 * NEN1);
  int* IDs = Wd + 3 * NEN1;

  const bool mapped = prm.X != nullptr, rational = prm.Wt != nullptr;
  const bool want_mat = NA > 0, want_vec = (prm.slot != PETIGA_SLOT_MATRIX && prm.slot != PETIGA_SLOT_JACOBIAN && prm.slot != PETIGA_SLOT_IJACOBIAN);
  const bool state = prm.needs_state && prm.U != nullptr;
  const bool transient = (prm.slot == PETIGA_SLOT_IFUNCTION || prm.slot == PETIGA_SLOT_IJACOBIAN);

  int ID[3] = {0, 0, 0}, nq1[3] = {1, 1, 1}, nqp = 1;
  if (valid) element_id(prm.ax, elem, ID);
#pragma unroll
  for (int d = 0; d < 3; d++) { nq1[d] = prm.ax[d].nqp; nqp *= nq1[d]; }

  // ---------------- header: closure, gathers, position tables, fix lists ----------------
  if (valid) {
    for (int a = lt; a < M; a += G) {
      int ia = a % NEN1, ja = (DIM > 1) ? (a / NEN1) % NEN1 : 0, ka = (DIM > 2) ? a / (NEN1 * NEN1) : 0;
      const int ai[3] = {ia, ja, ka};
      int gidx = closure_index<DIM>(prm.ax, ID, ai);
      int lr = prm.localrow[gidx];
      lrow[a] = lr;
      if (mapped) {
#pragma unroll
        for (int i = 0; i < DIM; i++) Xe[a * DIM + i] = prm.X[(size_t)gidx * DIM + i];
        if (rational) We[a] = prm.Wt[gidx];
      }
      // fix lists: BuildFix/AddFixa/AddFlux (petigaelem.c:1166-1283), "last face wins" for values, loads accumulate
      int onfix[DOF];
      double vfix[DOF], vflux[DOF];
#pragma unroll
      for (int c = 0; c < DOF; c++) { onfix[c] = 0; vfix[c] = 0.0; vflux[c] = 0.0; }
      if (prm.any_bc) {
#pragma unroll
        for (int d = 0; d < DIM; d++) {
          if (prm.ax[d].periodic) continue;
          for (int s = 0; s < 2; s++) {
            const FixSide& fs = prm.bc[d][s];
            if (!(fs.vcount || fs.lcount)) continue;
            if (ID[d] != (s ? prm.ax[d].nel - 1 : 0)) continue;
            if (ai[d] != (s ? NEN1 - 1 : 0)) continue;
            for (int k = 0; k < fs.vcount; k++) {
              int c = fs.vfield[k];
              onfix[c] = 1;
              vfix[c] = prm.fixtable ? prm.fixtable[(size_t)gidx * DOF + c] : fs.vvalue[k];
            }
            if (fs.lcount) {  // BoundaryArea, unmapped branch (petigaelem.c:1118-1131)
              double A = 1.0;
              if (DIM > 1) {
                for (int e = 0; e < DIM; e++)
                  if (e != d) A *= prm.ax[e].detJac[ID[e]] / (double)NEN1;
                if (prm.face_dS[d][s]) {   // mapped geometry: surface Jacobian integrated over the face (face_area_kernel, pc_api.cu)
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
#pragma unroll
      for (int c = 0; c < DOF; c++) {
        int idx = a * DOF + c;
        double u = 0.0, v = 0.0;
        if (state) {
          u = prm.U[(size_t)lr * DOF + c];
          if (transient && prm.V) v = prm.V[(size_t)lr * DOF + c];
        }
        fixflag[idx] = onfix[c];
        FixVal[idx] = vfix[c];
        Flux[idx] = vflux[c];
        UFix[idx] = u;                      // FixValues keeps the old value (petigaelem.c:1343-1358)
        if (onfix[c]) { u = vfix[c]; v = 0.0; }   // FixValues / DelValues (:1327-1341)
        Ue[idx] = u;
        Ve[idx] = v;
        Fe[idx] = 0.0;
      }
    }
    for (int t = lt; t < 3 * NEN1 * NEN1; t += G) {
      int d = t / (NEN1 * NEN1), r = t - d * NEN1 * NEN1, ia = r / NEN1, ib = r - ia * NEN1;
      uint32_t s = 0x00000100u;   // unused axis: B=0,S=1,L=0
      if (d < DIM) {
        int g = prm.ax[d].offset[ID[d]] + ia - prm.ax[d].gs;
        int c = ib - ia + prm.ax[d].lo[g];
        s = prm.ax[d].seg[g * kMaxW + c];
        if (ib == 0) Wd[d * NEN1 + ia] = prm.ax[d].W[g];
      } else if (ib == 0) Wd[d * NEN1 + ia] = 1;
      segs[t] = s;
    }
    if (lt == 0) { IDs[0] = ID[0]; IDs[1] = ID[1]; IDs[2] = ID[2]; }
  }
  __syncthreads();

  // register tile of K_e: rows a in [row0,row0+TM), columns n=(b,j,i) in [col0,col0+TN)
  const int ty = lt / GN, tx = lt - ty * GN;
  const int row0 = ty * TM;
  double acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; i++)
#pragma unroll
    for (int j = 0; j < TN; j++) acc[i][j] = 0.0;

  // ---------------- quadrature loop in chunks of QC points ----------------
  for (int q0 = 0; q0 < nqp; q0 += QC) {
    const int nq = min(QC, nqp - q0);
    if (valid) {
      // K2/K3: tensor-product tabulation of the components the form reads (petiga3d.F90:1-233)
      for (int t = lt; t < nq * M; t += G) {
        int ql = t / M, a = t - ql * M, q = q0 + ql;
        int qi[3] = {q % nq1[0], (q / nq1[0]) % nq1[1], q / (nq1[0] * nq1[1])};
        int ai[3] = {a % NEN1, (DIM > 1) ? (a / NEN1) % NEN1 : 0, (DIM > 2) ? a / (NEN1 * NEN1) : 0};
        double v0[3] = {1, 1, 1}, v1[3] = {0, 0, 0}, v2[3] = {0, 0, 0};
#pragma unroll
        for (int d = 0; d < DIM; d++) {
          const double* tab = prm.ax[d].value + ((size_t)(ID[d] * nq1[d] + qi[d]) * NEN1 + ai[d]) * 5;
          v0[d] = tab[0]; v1[d] = tab[1]; v2[d] = tab[2];
        }
        double* out = Psi + (size_t)ql * NC * M + a;
        if (prm.c0 == 0) out[0] = v0[0] * v0[1] * v0[2];
#pragma unroll
        for (int d = 0; d < DIM; d++) {
          int c = 1 + d;
          if (c >= prm.c0 && c < prm.c1) {
            double g = (d == 0 ? v1[0] : v0[0]);
            if (DIM > 1) g *= (d == 1 ? v1[1] : v0[1]);
            if (DIM > 2) g *= (d == 2 ? v1[2] : v0[2]);
            out[(c - prm.c0) * M] = g;
          }
        }
        if (DIM + 1 < prm.c1) {
          double lap = v2[0] * v0[1] * v0[2];
          if (DIM > 1) lap += v0[0] * v2[1] * v0[2];
          if (DIM > 2) lap += v0[0] * v0[1] * v2[2];
          out[(DIM + 1 - prm.c0) * M] = lap;
        }
      }
    }
    __syncthreads();
    if (mapped) {
      double* X1 = Geo;                       // [QC][DIM*DIM]   X1[i][d] = dX_i/du_d
      double* detX = Geo + QC * DIM * DIM;    // [QC]
      double* W0 = detX + QC;                 // [QC]
      double* W1 = W0 + QC;                   // [QC][DIM]
      if (rational) {  // K4 Rationalize, orders 0-1 (petigarat.f90.in:24-35)
        if (valid)
          for (int t = lt; t < nq * (1 + DIM); t += G) {
            int ql = t / (1 + DIM), c = t - ql * (1 + DIM);
            const double* ps = Psi + ((size_t)ql * NC + c) * M;
            double s = 0.0;
            for (int a = 0; a < M; a++) s += We[a] * ps[a];
            if (c == 0) W0[ql] = s; else W1[ql * DIM + c - 1] = s;
          }
        __syncthreads();
        if (valid)
          for (int t = lt; t < nq * M; t += G) {
            int ql = t / M, a = t - ql * M;
            double* ps = Psi + (size_t)ql * NC * M + a;
            double w0 = W0[ql], R0 = We[a] * ps[0] / w0;
#pragma unroll
            for (int d = 0; d < DIM; d++) ps[(1 + d) * M] = (We[a] * ps[(1 + d) * M] - R0 * W1[ql * DIM + d]) / w0;
            ps[0] = R0;
          }
        __syncthreads();
      }
      if (valid) {  // K5 GeometryMap (petigamapgeo.f90.in:28-43)
        for (int t = lt; t < nq * DIM * (DIM + 1); t += G) {
          int ql = t / (DIM * (DIM + 1)), r = t - ql * DIM * (DIM + 1), i = r / (DIM + 1), c = r - i * (DIM + 1);
          const double* ps = Psi + ((size_t)ql * NC + c) * M;
          double s = 0.0;
          for (int a = 0; a < M; a++) s += Xe[a * DIM + i] * ps[a];
          if (c == 0) Xq[ql * 3 + i] = s; else X1[(ql * DIM + i) * DIM + c - 1] = s;
        }
      }
      __syncthreads();
      if (valid) for (int ql = lt; ql < nq; ql += G) {  // K6 InverseMap order 1 (petigamapinv.f90.in:28-31, petigadet/inv.f90.in)
        double* J = X1 + ql * DIM * DIM;   // J[i][d]
        double E[DIM * DIM], det;
        if (DIM == 1) { det = J[0]; E[0] = 1.0 / det; }
        else if (DIM == 2) {
          det = J[0] * J[3] - J[1] * J[2];
          E[0] = J[3] / det; E[1] = -J[1] / det; E[2] = -J[2] / det; E[3] = J[0] / det;   // E[d][i] = du_d/dx_i
        } else {
          double a00 = J[0], a01 = J[1], a02 = J[2], a10 = J[3], a11 = J[4], a12 = J[5], a20 = J[6], a21 = J[7], a22 = J[8];
          det = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
          E[0] = (a11 * a22 - a12 * a21) / det; E[1] = -(a01 * a22 - a02 * a21) / det; E[2] = (a01 * a12 - a02 * a11) / det;
          E[3] = -(a10 * a22 - a12 * a20) / det; E[4] = (a00 * a22 - a02 * a20) / det; E[5] = -(a00 * a12 - a02 * a10) / det;
          E[6] = (a10 * a21 - a11 * a20) / det; E[7] = -(a00 * a21 - a01 * a20) / det; E[8] = (a00 * a11 - a01 * a10) / det;
        }
        detX[ql] = det;
#pragma unroll
        for (int k = 0; k < DIM * DIM; k++) J[k] = E[k];
      }
      __syncthreads();
      if (valid)  // K7 ShapeFunctions order 1: R1_i = sum_d N1_d * du_d/dx_i (petigamapshf.f90.in:36-43)
        for (int t = lt; t < nq * M; t += G) {
          int ql = t / M, a = t - ql * M;
          double* ps = Psi + (size_t)ql * NC * M + a;
          const double* E = X1 + ql * DIM * DIM;
          double g[DIM], r[DIM];
#pragma unroll
          for (int d = 0; d < DIM; d++) g[d] = ps[(1 + d) * M];
#pragma unroll
          for (int i = 0; i < DIM; i++) {
            r[i] = 0.0;
#pragma unroll
            for (int d = 0; d < DIM; d++) r[i] += g[d] * E[d * DIM + i];
          }
#pragma unroll
          for (int i = 0; i < DIM; i++) ps[(1 + i) * M] = r[i];
        }
      __syncthreads();
    }
    // K12 field evaluation at the points (petigaval.F90:182-251)
    if (state) {
      const int per = DOF * (2 + DIM + 1);
      if (valid)
        for (int t = lt; t < nq * per; t += G) {
          int ql = t / per, r = t - ql * per, i = r / (2 + DIM + 1), w = r - i * (2 + DIM + 1);
          // w: 0 = u, 1 = v, 2..1+DIM = grad, 2+DIM = laplacian
          int comp = (w <= 1) ? 0 : (w - 1);
          double s = 0.0;
          if (comp >= prm.c0 && comp < prm.c1) {
            const double* ps = Psi + ((size_t)ql * NC + comp - prm.c0) * M;
            const double* src = (w == 1) ? Ve : Ue;
            for (int a = 0; a < M; a++) s += ps[a] * src[a * DOF + i];
          }
          Sq[ql * per + r] = s;
        }
      __syncthreads();
    }
    // per-point weights and coefficient tensors
    if (valid) for (int ql = lt; ql < nq; ql += G) {
      int q = q0 + ql;
      int qi[3] = {q % nq1[0], (q / nq1[0]) % nq1[1], q / (nq1[0] * nq1[1])};
      double w = 1.0, J = 1.0;
      QPoint qp;
      qp.atboundary = 0;
#pragma unroll
      for (int d = 0; d < 3; d++) qp.x[d] = 0.0;
#pragma unroll
      for (int d = 0; d < DIM; d++) {  // IGA_Quadrature_3D: W = iW*jW*kW, J = iJ*jJ*kJ (petiga3d.F90:22-28)
        w *= prm.ax[d].weight[ID[d] * nq1[d] + qi[d]];
        J *= prm.ax[d].detJac[ID[d]];
        qp.x[d] = prm.ax[d].point[ID[d] * nq1[d] + qi[d]];
      }
      if (mapped) {
        J *= Geo[QC * DIM * DIM + ql];      // detJac *= detX (petigaelem.c:1024-1029)
#pragma unroll
        for (int d = 0; d < DIM; d++) qp.x[d] = Xq[ql * 3 + d];
      }
      const double jw = J * w;              // IGAPointAddArray: JW = detJac*weight (petigapoint.c:461)
      JW[ql] = jw;
      if (prm.per_qp || q0 == 0) {
        if (state) {
          const int per = DOF * (2 + DIM + 1);
#pragma unroll
          for (int i = 0; i < DOF; i++) {
            const double* s = Sq + ql * per + i * (2 + DIM + 1);
            qp.u[i] = s[0]; qp.v[i] = s[1];
#pragma unroll
            for (int d = 0; d < DIM; d++) qp.gu[i][d] = s[2 + d];
            qp.d2u[i] = s[2 + DIM];
          }
        }
        double* C = Cq + (size_t)ql * DOF * DOF * NA * NA;
        double* fv = Fq + (size_t)ql * DOF * (NV > 0 ? NV : 1);
        for (int k = 0; k < DOF * DOF * NA * NA; k++) C[k] = 0.0;
        for (int k = 0; k < DOF * NV; k++) fv[k] = 0.0;
        form_coefficients<DIM, DOF>(prm.form, prm.slot, prm.prm, prm.shift, prm.t, qp, NA, NV, NA ? C : nullptr, NV ? fv : nullptr);
      }
    }
    __syncthreads();
    if (valid) {
      // B operand: T[(q,al)][(b,j,i)] = JW_q * sum_be C_q[i][j][al][be] * Psi_be(b,q); a thread keeps its column n
      if (want_mat) {
        constexpr int PARTS = (G >= N) ? G / N : 1;
        for (int t = lt; t < PARTS * N; t += G) {
          const int n = t % N, part = t / N;
          const int b = n / (DOF * DOF), j = (n / DOF) % DOF, i = n % DOF;
          const double* Cij = Cq + (size_t)(i * DOF + j) * NA * NA;
          const double* psb = Psi + (size_t)(prm.mc0 - prm.c0) * M + b;
          for (int ql = part; ql < nq; ql += PARTS) {
            const double* C = Cij + (prm.per_qp ? (size_t)ql * DOF * DOF * NA * NA : 0);
            const double* ps = psb + (size_t)ql * NC * M;
            const double jw = JW[ql];
            double* out = Bs + (size_t)ql * NA * N + n;
            for (int al = 0; al < NA; al++) {
              double sacc = 0.0;
              for (int be = 0; be < NA; be++) sacc += C[al * NA + be] * ps[be * M];
              out[al * N] = sacc * jw;
            }
          }
        }
      }
      // element vector: F_e[a,i] += sum_q JW_q sum_al Psi_al(a,q) f_q[i][al]
      if (want_vec && NV > 0)
        for (int t = lt; t < M * DOF; t += G) {
          int a = t / DOF, i = t - a * DOF;
          double s = 0.0;
          for (int ql = 0; ql < nq; ql++) {
            const double* fv = Fq + (size_t)(prm.per_qp ? ql : 0) * DOF * NV + i * NV;
            const double* ps = Psi + ((size_t)ql * NC + prm.vc0 - prm.c0) * M + a;
            double sq = 0.0;
            for (int al = 0; al < NV; al++) sq += ps[al * M] * fv[al];
            s += sq * JW[ql];
          }
          Fe[t] += s;
        }
    }
    __syncthreads();
    // K9: the contraction K_e += Psi^T T over this chunk, register tiled from shared memory
    if (valid && want_mat) {
      for (int ql = 0; ql < nq; ql++) {
        const double* pa = Psi + ((size_t)ql * NC + prm.mc0 - prm.c0) * M + row0;
        const double* pb = Bs + (size_t)ql * NA * N;
        for (int al = 0; al < NA; al++) {
          double af[TM], bf[TN];
#pragma unroll
          for (int i = 0; i < TM; i++) af[i] = pa[al * M + i];
#pragma unroll
          for (int j = 0; j < TN; j++) bf[j] = pb[al * N + Cfg::col(tx, j)];
#pragma unroll
          for (int i = 0; i < TM; i++)
#pragma unroll
            for (int j = 0; j < TN; j++) acc[i][j] = fma(af[i], bf[j], acc[i][j]);
        }
      }
    }
    __syncthreads();
  }

  // ---------------- fix-up on the tiles (petigaelem.c:1360-1389, :1483-1501) ----------------
  const bool fix_mat = (prm.slot == PETIGA_SLOT_SYSTEM || prm.slot == PETIGA_SLOT_JACOBIAN || prm.slot == PETIGA_SLOT_IJACOBIAN);
  if (valid && want_mat && fix_mat && prm.any_bc) {
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
      for (int j = 0; j < TN; j++) {
        int a = row0 + i, n = Cfg::col(tx, j);
        int b = n / (DOF * DOF), jj = (n / DOF) % DOF, ii = n % DOF;
        int ra = a * DOF + ii, cb = b * DOF + jj;
        bool fr = fixflag[ra], fc = fixflag[cb];
        if (fr || fc) {
          if (prm.slot == PETIGA_SLOT_SYSTEM && fc && !fr) atomic_add_shared(&Fe[ra], -acc[i][j] * FixVal[cb]);
          acc[i][j] = (ra == cb) ? 1.0 : 0.0;
        }
      }
  }
  __syncthreads();
  if (valid && want_vec) {  // FixSystem / FixFunction vector part, then VecSetValuesLocal(ADD_VALUES)
    for (int t = lt; t < M * DOF; t += G) {
      int a = t / DOF, i = t - a * DOF;
      double F = Fe[t];
      if (prm.slot == PETIGA_SLOT_SYSTEM) { F += Flux[t]; if (fixflag[t]) F = FixVal[t]; }
      else if (prm.slot == PETIGA_SLOT_FUNCTION || prm.slot == PETIGA_SLOT_IFUNCTION) { F -= Flux[t]; if (fixflag[t]) F = UFix[t] - FixVal[t]; }
      if (F != 0.0) atomicAdd(&prm.rhs[(size_t)lrow[a] * DOF + i], F);
    }
  }
  // ---------------- scatter: closed-form CSR position + FP64 reduction (K10) ----------------
  if (valid && want_mat) {
#pragma unroll
    for (int i = 0; i < TM; i++) {
      const int a = row0 + i;
      const int ia = a % NEN1, ja = (DIM > 1) ? (a / NEN1) % NEN1 : 0, ka = (DIM > 2) ? a / (NEN1 * NEN1) : 0;
      const int lr = lrow[a];
      const int W0 = Wd[ia], W1 = Wd[NEN1 + ja], W2 = Wd[2 * NEN1 + ka];
      int64_t base = prm.rowbase[lr];
      double* dst = prm.values;
      if (lr >= prm.nown) { dst = prm.ghost_values; base -= prm.nnz_own; }
#pragma unroll
      for (int j = 0; j < TN; j++) {
        const double v = acc[i][j];
        if (v == 0.0) continue;   // adding an exact zero cannot change the sum
        const int n = Cfg::col(tx, j);
        const int b = n / (DOF * DOF), jj = (n / DOF) % DOF, ii = n % DOF;
        const int ib = b % NEN1, jb = (DIM > 1) ? (b / NEN1) % NEN1 : 0, kb = (DIM > 2) ? b / (NEN1 * NEN1) : 0;
        const int pos = seg_position(segs[ia * NEN1 + ib], segs[NEN1 * NEN1 + ja * NEN1 + jb], segs[2 * NEN1 * NEN1 + ka * NEN1 + kb], W0, W1);
        atomicAdd(dst + value_offset(base, pos, DOF, prm.block, ii, jj, W0 * W1 * W2), v);
      }
    }
  }
}

}  // namespace pc
