// pc_bnd.cu -- the boundary-integral pass of the element loop (SURVEY.md 8f-2).
//
// Reference: IGAElementNextForm visits, before the interior, every face of a boundary element that was enabled with
// IGASetBoundaryForm (src/petigaelem.c:427-447); IGAElementBuildTabulation then tabulates on the face: the face axis uses
// the one-point "rule" (bnd_point, weight 1, detJac 1) and the end-point basis table bnd_value (IGA_Quadrature_BNDR /
// IGA_BasisFuns_BNDR, :788-792,813-868), the normal and the surface Jacobian detS come from IGA_GetNormal
// (src/petigaval.F90:45-99) and detJac *= detS (:1012-1029).  The user callback sees p->atboundary.
//
// The built-in boundary terms are vector terms  F[a][i] += N_a * g_i(face, x, n)  (demo/BoundaryIntegral.c:41-57), so the
// pass is one small kernel after the interior kernel: a warp per face element; phase 1, a lane per face quadrature point
// (geometry jets -> x, detS, normal, JW*g); phase 2, a lane per local node (sum over the points).  Dofs that the element
// fixes (IGAElementFixSystem overwrites F[k] = v, :1377-1387) are skipped; everything else is linear, so adding the face
// terms after the interior kernel's own fix-up gives the reference's element vector.
#include <cstring>

#include "pc_plan.h"

namespace pc {

namespace {

constexpr int kWarps = 4;
constexpr int kMaxFaceQ = 100;     // face quadrature points per element (10 x 10 rule)

struct BndParams {
  DevAxis ax[3];
  const double* bnd_value[3][2];   // [nen][5] end-point tables (IGABasis.bnd_value, include/petiga.h:134-139)
  double bnd_point[3][2];
  int dim, dof, dir, side, n0, n1; // face (dir, side); n0 x n1 face elements in this rank's box
  const int* localrow;
  const double* X;
  const double* Wt;
  double* rhs;                     // unified local vector [nloc*dof]
  FixSide bc[3][2];
  int apply_fix;                   // slot SYSTEM with Dirichlet values: skip the dofs the element fixes
  int form, slot;
  double prm[8];
};

// g_i of the built-in forms:  F[a][i] += N_a * g_i   on the face (dir, side) at physical point x with outward normal n
template <int DIM>
__device__ inline bool boundary_vector_coefficients(int form, const double* prm, int dir, int side, const double* x, const double* n, int dof, double* g) {
  (void)prm; (void)dir; (void)side; (void)x; (void)n;
  switch (form) {
    case PETIGA_FORM_BOUNDARYINTEGRAL:   // demo/BoundaryIntegral.c:41-49  Neumann(): F[a] = N0[a] * 1.0
      for (int i = 0; i < dof; i++) g[i] = 1.0;
      return true;
  }
  return false;
}

template <int DIM>
__global__ void __launch_bounds__(kWarps * 32) bnd_vec_kernel(const __grid_constant__ BndParams bp) {
  __shared__ double sJW[kWarps][kMaxFaceQ];
  __shared__ double sG[kWarps][kMaxFaceQ][kMaxDof];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int fe = blockIdx.x * kWarps + warp;
  if (fe >= bp.n0 * bp.n1) return;
  const int dir = bp.dir, side = bp.side;
  int fa[2] = {0, 0}, nfa = 0;
  for (int i = 0; i < DIM; i++) if (i != dir) fa[nfa++] = i;
  int ID[3] = {0, 0, 0};
  ID[dir] = side ? bp.ax[dir].nel - 1 : 0;
  if (DIM > 1) ID[fa[0]] = bp.ax[fa[0]].es + fe % bp.n0;
  if (DIM > 2) ID[fa[1]] = bp.ax[fa[1]].es + fe / bp.n0;
  int nq[3] = {1, 1, 1}, nen1[3] = {1, 1, 1};
  for (int d = 0; d < DIM; d++) { nq[d] = (d == dir) ? 1 : bp.ax[d].nqp; nen1[d] = bp.ax[d].nen; }
  const int nqf = nq[0] * nq[1] * nq[2], nen = nen1[0] * nen1[1] * nen1[2];
  const bool mapped = bp.X != nullptr, rational = bp.Wt != nullptr;

  auto table = [&](int d, int q) -> const double* {   // 1-D values of axis d at the face point's d-th coordinate
    return (d == dir) ? bp.bnd_value[d][side] : bp.ax[d].value + (size_t)(ID[d] * bp.ax[d].nqp + q) * nen1[d] * 5;
  };
  int gbase[3];
  for (int d = 0; d < 3; d++) gbase[d] = (d < DIM) ? bp.ax[d].offset[ID[d]] - bp.ax[d].gs : 0;

  // ---- phase 1: a lane per face quadrature point ----
  for (int q = lane; q < nqf; q += 32) {
    const int qi[3] = {q % nq[0], (q / nq[0]) % nq[1], q / (nq[0] * nq[1])};
    double JW = 1.0, x[3] = {0, 0, 0}, nrm[3] = {0, 0, 0};
    for (int d = 0; d < DIM; d++) {
      if (d == dir) { x[d] = bp.bnd_point[d][side]; continue; }              // weight 1, detJac 1 (IGA_Quadrature_BNDR)
      JW *= bp.ax[d].weight[ID[d] * bp.ax[d].nqp + qi[d]] * bp.ax[d].detJac[ID[d]];
      x[d] = bp.ax[d].point[ID[d] * bp.ax[d].nqp + qi[d]];
    }
    nrm[dir] = side ? 1.0 : -1.0;
    if (mapped) {
      const double* t0 = table(0, qi[0]);
      const double* t1 = (DIM > 1) ? table(1, qi[1]) : nullptr;
      const double* t2 = (DIM > 2) ? table(2, qi[2]) : nullptr;
      // jets (value + parametric gradient) of w, w*x_i
      double w0 = 0, w1[3] = {0, 0, 0}, X0[3] = {0, 0, 0}, X1[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
      for (int ka = 0; ka < nen1[2]; ka++) {
        const double k0 = (DIM > 2) ? t2[ka * 5] : 1.0, k1 = (DIM > 2) ? t2[ka * 5 + 1] : 0.0;
        for (int ja = 0; ja < nen1[1]; ja++) {
          const double j0 = (DIM > 1) ? t1[ja * 5] : 1.0, j1 = (DIM > 1) ? t1[ja * 5 + 1] : 0.0;
          for (int ia = 0; ia < nen1[0]; ia++) {
            const int gidx = (gbase[0] + ia) + bp.ax[0].gw * ((gbase[1] + ja) + bp.ax[1].gw * (gbase[2] + ka));
            const double wa = rational ? bp.Wt[gidx] : 1.0;
            const double N = t0[ia * 5] * j0 * k0;
            const double dN[3] = {t0[ia * 5 + 1] * j0 * k0, t0[ia * 5] * j1 * k0, t0[ia * 5] * j0 * k1};
            w0 = fma(wa, N, w0);
            for (int d = 0; d < DIM; d++) w1[d] = fma(wa, dN[d], w1[d]);
            for (int i = 0; i < DIM; i++) {
              const double xa = wa * bp.X[(size_t)gidx * DIM + i];
              X0[i] = fma(xa, N, X0[i]);
              for (int d = 0; d < DIM; d++) X1[i][d] = fma(xa, dN[d], X1[i][d]);
            }
          }
        }
      }
      if (rational)   // quotient rule (petigarat.f90.in:24-35 applied to the sums)
        for (int i = 0; i < DIM; i++) {
          X0[i] /= w0;
          for (int d = 0; d < DIM; d++) X1[i][d] = (X1[i][d] - X0[i] * w1[d]) / w0;
        }
      for (int i = 0; i < DIM; i++) x[i] = X0[i];
      // IGA_GetNormal (petigaval.F90:45-99): F(d,:) = dx/du_d
      double dS = 1.0;
      if (DIM == 1) nrm[0] = 1.0;
      else if (DIM == 2) {
        const int dd = (dir == 0) ? 1 : 0;
        const double sg = (dir == 0) ? 1.0 : -1.0, tx = sg * X1[0][dd], ty = sg * X1[1][dd];
        nrm[0] = ty; nrm[1] = -tx;
        dS = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1]);
        nrm[0] /= dS; nrm[1] /= dS;
      } else {
        const int ds = (dir + 1) % 3, dt = (dir + 2) % 3;
        const double s0 = X1[0][ds], s1 = X1[1][ds], s2 = X1[2][ds], u0 = X1[0][dt], u1 = X1[1][dt], u2 = X1[2][dt];
        nrm[0] = s1 * u2 - s2 * u1; nrm[1] = s2 * u0 - s0 * u2; nrm[2] = s0 * u1 - s1 * u0;
        dS = sqrt(nrm[0] * nrm[0] + nrm[1] * nrm[1] + nrm[2] * nrm[2]);
        nrm[0] /= dS; nrm[1] /= dS; nrm[2] /= dS;
      }
      if (side == 0) for (int i = 0; i < DIM; i++) nrm[i] = -nrm[i];
      JW *= dS;   // detJac *= detS (petigaelem.c:1027-1028)
    }
    double g[kMaxDof] = {0, 0, 0, 0};
    boundary_vector_coefficients<DIM>(bp.form, bp.prm, dir, side, x, nrm, bp.dof, g);
    sJW[warp][q] = JW;
    for (int i = 0; i < bp.dof; i++) sG[warp][q][i] = g[i];
  }
  __syncwarp();
  // ---- phase 2: a lane per local node: F[a][i] = sum_q JW_q g_q[i] R_a(q); R = rationalised basis ----
  for (int a = lane; a < nen; a += 32) {
    const int ai[3] = {a % nen1[0], (a / nen1[0]) % nen1[1], a / (nen1[0] * nen1[1])};
    const int gidx = (gbase[0] + ai[0]) + bp.ax[0].gw * ((gbase[1] + ai[1]) + bp.ax[1].gw * (gbase[2] + ai[2]));
    const double wa = rational ? bp.Wt[gidx] : 1.0;
    double F[kMaxDof] = {0, 0, 0, 0};
    for (int q = 0; q < nqf; q++) {
      const int qi[3] = {q % nq[0], (q / nq[0]) % nq[1], q / (nq[0] * nq[1])};
      double N = table(0, qi[0])[ai[0] * 5];
      if (DIM > 1) N *= table(1, qi[1])[ai[1] * 5];
      if (DIM > 2) N *= table(2, qi[2])[ai[2] * 5];
      if (rational) {   // R0 = W N / sum W N
        double w0 = 0.0;
        for (int kb = 0; kb < nen1[2]; kb++)
          for (int jb = 0; jb < nen1[1]; jb++)
            for (int ib = 0; ib < nen1[0]; ib++) {
              const int gb = (gbase[0] + ib) + bp.ax[0].gw * ((gbase[1] + jb) + bp.ax[1].gw * (gbase[2] + kb));
              double Nb = table(0, qi[0])[ib * 5];
              if (DIM > 1) Nb *= table(1, qi[1])[jb * 5];
              if (DIM > 2) Nb *= table(2, qi[2])[kb * 5];
              w0 = fma(bp.Wt[gb], Nb, w0);
            }
        N = wa * N / w0;
      }
      const double s = sJW[warp][q] * N;
      for (int i = 0; i < bp.dof; i++) F[i] = fma(s, sG[warp][q][i], F[i]);
    }
    // dofs fixed by this element (BuildFix: node on a Dirichlet face of a boundary element, petigaelem.c:1214-1283)
    bool fixed[kMaxDof] = {false, false, false, false};
    if (bp.apply_fix)
      for (int d = 0; d < DIM; d++) {
        if (bp.ax[d].periodic) continue;
        for (int s = 0; s < 2; s++) {
          const FixSide& fs = bp.bc[d][s];
          if (!fs.vcount || ID[d] != (s ? bp.ax[d].nel - 1 : 0) || ai[d] != (s ? nen1[d] - 1 : 0)) continue;
          for (int k = 0; k < fs.vcount; k++) fixed[fs.vfield[k]] = true;
        }
      }
    const int lr = bp.localrow[gidx];
    for (int i = 0; i < bp.dof; i++)
      if (!fixed[i] && F[i] != 0.0) atomicAdd(&bp.rhs[(size_t)lr * bp.dof + i], F[i]);
  }
}

}  // namespace

bool form_has_boundary_term(int form) { return form == PETIGA_FORM_BOUNDARYINTEGRAL; }

// the boundary pass of one compute call: adds the face terms of every visited face into rhs (unified local vector)
int launch_boundary_pass(petiga_cuda_plan* P, int slot, int form, const double* prm, double* rhs, bool apply_fix) {
  const Layout& L = P->L;
  for (int d = 0; d < L.dim; d++)
    for (int s = 0; s < 2; s++) {
      if (!P->visit[d][s] || L.ax[d].periodic) continue;
      // does this rank's element box touch the face?
      const int face_e = s ? L.ax[d].nel - 1 : 0;
      if (face_e < L.ax[d].es || face_e >= L.ax[d].es + L.ax[d].ew) continue;
      if (!P->d_bnd_value[d][s]) { set_error("boundary form: end-point basis tables not set (petiga_cuda_set_boundary_tables)"); return PETIGA_CUDA_ERR_ORDER; }
      BndParams bp;
      memset(&bp, 0, sizeof(bp));
      for (int i = 0; i < 3; i++) {
        bp.ax[i] = P->dax[i];
        for (int t = 0; t < 2; t++) { bp.bnd_value[i][t] = P->d_bnd_value[i][t].get(); bp.bnd_point[i][t] = P->bnd_point[i][t]; }
      }
      int fa[2] = {0, 0}, nfa = 0;
      for (int i = 0; i < L.dim; i++) if (i != d) fa[nfa++] = i;
      bp.dim = L.dim; bp.dof = L.dof; bp.dir = d; bp.side = s;
      bp.n0 = (L.dim > 1) ? L.ax[fa[0]].ew : 1; bp.n1 = (L.dim > 2) ? L.ax[fa[1]].ew : 1;
      bp.localrow = P->d_localrow.get(); bp.X = P->d_X.get(); bp.Wt = P->d_W.get(); bp.rhs = rhs;
      bp.apply_fix = apply_fix ? 1 : 0; bp.form = form; bp.slot = slot;
      memcpy(bp.prm, prm, sizeof(bp.prm));
      int nqf = 1;
      for (int i = 0; i < L.dim; i++) if (i != d) nqf *= L.ax[i].nqp;
      if (nqf > kMaxFaceQ) { set_error("boundary form: more than 100 quadrature points per face element"); return PETIGA_CUDA_ERR_SUP; }
      if (apply_fix) fill_fix_sides(P, false, bp.bc);
      const int nfe = bp.n0 * bp.n1, blocks = (nfe + kWarps - 1) / kWarps;
      if (L.dim == 1) bnd_vec_kernel<1><<<blocks, kWarps * 32, 0, P->stream>>>(bp);
      else if (L.dim == 2) bnd_vec_kernel<2><<<blocks, kWarps * 32, 0, P->stream>>>(bp);
      else bnd_vec_kernel<3><<<blocks, kWarps * 32, 0, P->stream>>>(bp);
      PC_CUDA(cudaGetLastError());
      P->launches++;
    }
  return 0;
}

}  // namespace pc

using namespace pc;

extern "C" int petiga_cuda_set_boundary_tables(petiga_cuda_plan* P, int axis, const double* bnd_value0, const double* bnd_value1,
                                               double bnd_point0, double bnd_point1) {
  if (!P || axis < 0 || axis > 2 || !bnd_value0 || !bnd_value1) return PETIGA_CUDA_ERR_ARG;
  PC_CUDA(cudaSetDevice(P->device));
  const size_t n = (size_t)(P->L.ax[axis].p + 1) * 5;
  const double* src[2] = {bnd_value0, bnd_value1};
  for (int s = 0; s < 2; s++) {   // a table whose copy failed is dropped, so the face passes report it as not set
    DevBuf<double>& b = P->d_bnd_value[axis][s];
    int rc = b.reserve(n);
    if (rc) return rc;
    const cudaError_t e = cudaMemcpy(b.get(), src[s], n * sizeof(double), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { b.reset(); return cuda_fail(e, "set_boundary_tables"); }
  }
  P->bnd_point[axis][0] = bnd_point0; P->bnd_point[axis][1] = bnd_point1;
  return 0;
}

extern "C" int petiga_cuda_set_boundary_form(petiga_cuda_plan* P, int axis, int side, int flag) {
  if (!P || axis < 0 || axis > 2 || side < 0 || side > 1) return PETIGA_CUDA_ERR_ARG;
  P->visit[axis][side] = flag ? 1 : 0;
  P->config_version++;
  return 0;
}
