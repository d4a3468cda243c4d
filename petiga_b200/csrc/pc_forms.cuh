// pc_forms.cuh -- built-in device forms as per-quadrature-point coefficient tensors.
//
// The reference calls a host callback per quadrature point that fills K[a][i][b][j] and F[a][i] with an
// O(nen^2) double loop (e.g. demo/Poisson3D.c:3-23).  Every built-in form is bilinear in the tabulated
// shape quantities Psi = (N, dN/dx_0.., Laplacian N) of the test function a and the trial function b:
//      K_q[a,i,b,j] = sum_{al,be} Psi_al(a) * C_q[i][j][al][be] * Psi_be(b)
//      F_q[a,i]     = sum_{al}    Psi_al(a) * f_q[i][al]
// so on the device a form is only the small generator of (C_q, f_q); the O(nen^2 nqp) work is one
// form-independent FP64 contraction (pc_quad.cuh).  The algebra is the reference's expression
// re-associated; parity is checked to 1e-12 relative Frobenius error, not bit-wise.
//
// Psi component numbering: 0 = N, 1..DIM = first derivatives, DIM+1 = Laplacian.
#pragma once
#include <cuda_runtime.h>

#include "../../include/petiga_cuda.h"

namespace pc {

constexpr int kMaxComp = 5;   // N, 3 derivatives, Laplacian
constexpr int kMaxDof = 8;    // test/IGACreate.c sweeps dof 1..8 (test/makefile:23-40)
constexpr int kMaxPrm = 12;   // reals of the largest AppCtx (demo/PatternFormation.c:14-24: flag + 8)

// which IGACompute* a slot stands for (include/petiga.h:837-851, src/petigats.c:182-477, src/petigats2.c:23-175)
__host__ __device__ inline bool slot_has_mat(int s) {
  return s == PETIGA_SLOT_MATRIX || s == PETIGA_SLOT_SYSTEM || s == PETIGA_SLOT_JACOBIAN || s == PETIGA_SLOT_IJACOBIAN ||
         s == PETIGA_SLOT_IEJACOBIAN || s == PETIGA_SLOT_RHSJACOBIAN || s == PETIGA_SLOT_I2JACOBIAN;
}
__host__ __device__ inline bool slot_has_vec(int s) {
  return s == PETIGA_SLOT_VECTOR || s == PETIGA_SLOT_SYSTEM || s == PETIGA_SLOT_FUNCTION || s == PETIGA_SLOT_IFUNCTION ||
         s == PETIGA_SLOT_IEFUNCTION || s == PETIGA_SLOT_RHSFUNCTION || s == PETIGA_SLOT_I2FUNCTION;
}
__host__ __device__ inline bool slot_has_state(int s) { return s >= PETIGA_SLOT_FUNCTION; }            // reads U
__host__ __device__ inline bool slot_has_w(int s) {                                                     // third vector: U0 (IE) / A (I2)
  return s == PETIGA_SLOT_IEFUNCTION || s == PETIGA_SLOT_IEJACOBIAN || s == PETIGA_SLOT_I2FUNCTION || s == PETIGA_SLOT_I2JACOBIAN;
}
__host__ __device__ inline bool slot_has_v(int s) { return s == PETIGA_SLOT_IFUNCTION || s == PETIGA_SLOT_IJACOBIAN || slot_has_w(s); }
__host__ __device__ inline bool slot_is_i2(int s) { return s == PETIGA_SLOT_I2FUNCTION || s == PETIGA_SLOT_I2JACOBIAN; }
// element fix-up applied after the quadrature loop: 0 none (IGAComputeVector/Matrix), 1 FixSystem, 2 FixFunction, 3 FixJacobian
__host__ __device__ inline int slot_fix_kind(int s) {
  if (s == PETIGA_SLOT_SYSTEM) return 1;
  if (!slot_has_state(s)) return 0;
  return slot_has_vec(s) ? 2 : 3;
}

// static description of a (form, slot) pair: which Psi components the matrix / vector parts read
struct FormInfo {
  int valid;          // form provides this slot
  int mc0, mc1;       // matrix component range [mc0, mc1)
  int vc0, vc1;       // vector component range [vc0, vc1)
  int per_qp;         // coefficients depend on the quadrature point (state / position)
  int needs_x;        // reads the physical point
  int needs_state;    // reads U (and V for transient slots)
  int order;          // highest derivative read (0, 1 or 2)
  int constant_f;     // vector coefficient is a constant (eligible for the separable path)
  int mat_const;      // matrix coefficient tensor does not depend on the point
  int bnd_mat, bnd_vec;   // the callback has a p->atboundary branch that adds matrix / vector terms on visited faces
  int colloc;         // a collocation form (pc_colloc.cu): runs on collocation plans only, and nothing else runs there
};

__host__ __device__ inline FormInfo form_info(int form, int slot, int dim, int dof) {
  FormInfo f = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  const bool lin = (slot == PETIGA_SLOT_VECTOR || slot == PETIGA_SLOT_MATRIX || slot == PETIGA_SLOT_SYSTEM);
  const bool fun = (slot == PETIGA_SLOT_FUNCTION || slot == PETIGA_SLOT_IFUNCTION);
  const bool jac = (slot == PETIGA_SLOT_JACOBIAN || slot == PETIGA_SLOT_IJACOBIAN);
  switch (form) {
    case PETIGA_FORM_POISSON:
      if (dof != 1) break;
      if (lin) { f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 1; f.order = 1; f.constant_f = 1; }
      else if (slot == PETIGA_SLOT_FUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 1 + dim; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      else if (slot == PETIGA_SLOT_JACOBIAN) { f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.order = 1; }
      break;
    case PETIGA_FORM_LAPLACE:
      if (dof != 1 || !lin) break;
      f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 0; f.order = 1; f.constant_f = 1;
      break;
    case PETIGA_FORM_L2PROJECTION:
      if (dof != 1 || !lin) break;
      f.valid = 1; f.mc0 = 0; f.mc1 = 1; f.vc0 = 0; f.vc1 = 1; f.per_qp = 1; f.needs_x = 1; f.order = 0;
      break;
    case PETIGA_FORM_BOUNDARYINTEGRAL:   // interior part = Laplace; the face term is added by the boundary pass (pc_bnd.cu)
      if (dof != 1 || slot != PETIGA_SLOT_SYSTEM) break;
      f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 0; f.order = 1; f.constant_f = 1;
      break;
    case PETIGA_FORM_NEUMANN:
      if (dof != 1 || slot != PETIGA_SLOT_SYSTEM) break;
      f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 1; f.per_qp = 1; f.needs_x = 1; f.order = 1;
      break;
    case PETIGA_FORM_CONVTEST:
      if (dof != 1 || slot != PETIGA_SLOT_SYSTEM) break;
      f.valid = 1; f.mc0 = 0; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 1; f.per_qp = 1; f.needs_x = 1; f.order = 1;
      break;
    case PETIGA_FORM_MASS:
      if (!lin || dof > kMaxDof) break;
      f.valid = 1; f.mc0 = 0; f.mc1 = 1; f.vc0 = 0; f.vc1 = 1; f.order = 0; f.constant_f = 1;
      break;
    case PETIGA_FORM_ELASTICITY3D:
      if (!lin || dim != 3 || dof != 3) break;
      f.valid = 1; f.mc0 = 1; f.mc1 = 4; f.vc0 = 0; f.vc1 = 0; f.order = 1; f.constant_f = 1;
      break;
    case PETIGA_FORM_ELASTICITY:
      if (!lin || dof != dim) break;
      f.valid = 1; f.mc0 = 1; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 0; f.order = 1; f.constant_f = 1;
      break;
    case PETIGA_FORM_CAHNHILLIARD2D:
      if (dim != 2 || dof != 1) break;
      if (slot == PETIGA_SLOT_IFUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 4; f.per_qp = 1; f.needs_state = 1; f.order = 2; }
      if (slot == PETIGA_SLOT_IJACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 4; f.per_qp = 1; f.needs_state = 1; f.order = 2; }
      break;
    case PETIGA_FORM_CAHNHILLIARD3D:
      if (dim != 3 || dof != 1) break;
      if (slot == PETIGA_SLOT_IFUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 5; f.per_qp = 1; f.needs_state = 1; f.order = 2; }
      if (slot == PETIGA_SLOT_IJACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 5; f.per_qp = 1; f.needs_state = 1; f.order = 2; }
      break;
    case PETIGA_FORM_BRATU:
      if (dof != 1) break;
      if (fun || slot == PETIGA_SLOT_RHSFUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 1 + dim; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      if (jac || slot == PETIGA_SLOT_RHSJACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 1 + dim; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      break;
    case PETIGA_FORM_SNES2D:            // test/Test_SNES_2D.c:12-72 (dof 4, dim 2)
      if (dim != 2 || dof != 4) break;
      if (slot == PETIGA_SLOT_FUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 3; f.per_qp = 1; f.needs_state = 1; f.needs_x = 1; f.order = 1; }
      if (slot == PETIGA_SLOT_JACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 3; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      break;
    case PETIGA_FORM_PATTERNFORMATION:  // demo/PatternFormation.c:26-141 (dof 2, dim 2)
      if (dim != 2 || dof != 2) break;
      if (slot == PETIGA_SLOT_IEFUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 3; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      if (slot == PETIGA_SLOT_IEJACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 3; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      break;
    case PETIGA_FORM_ELASTICROD:        // demo/ElasticRodFJ.F90
      if (dof != 1) break;
      if (slot == PETIGA_SLOT_I2FUNCTION) { f.valid = 1; f.vc0 = 0; f.vc1 = 1 + dim; f.per_qp = 1; f.needs_state = 1; f.order = 1; }
      if (slot == PETIGA_SLOT_I2JACOBIAN) { f.valid = 1; f.mc0 = 0; f.mc1 = 1 + dim; f.order = 1; }
      break;
    case PETIGA_FORM_LAPLACE_COLLOCATION:    // demo/Laplace.c SystemCollocation
      if (dof != 1 || !lin) break;
      f.valid = 1; f.colloc = 1; f.order = 2; f.constant_f = 1;
      break;
    case PETIGA_FORM_CONVTEST_COLLOCATION:   // strong form of test/ConvTest.c
      if (dof != 1 || !lin) break;
      f.valid = 1; f.colloc = 1; f.order = 2; f.needs_x = 1;
      break;
    case PETIGA_FORM_NITSCHE:           // demo/NitscheMethod.c:70-119: interior Poisson (f = -2 dim) + face terms
      if (dof != 1 || slot != PETIGA_SLOT_SYSTEM) break;
      f.valid = 1; f.mc0 = 0; f.mc1 = 1 + dim; f.vc0 = 0; f.vc1 = 1 + dim; f.per_qp = 1; f.needs_x = 1; f.order = 1; f.bnd_mat = 1; f.bnd_vec = 1;
      break;
  }
  if (form == PETIGA_FORM_BOUNDARYINTEGRAL && f.valid) f.bnd_vec = 1;
  f.mat_const = !f.per_qp || form == PETIGA_FORM_L2PROJECTION || form == PETIGA_FORM_NEUMANN || form == PETIGA_FORM_CONVTEST ||
                form == PETIGA_FORM_NITSCHE;
  if (slot == PETIGA_SLOT_VECTOR) { f.mc0 = f.mc1 = 0; }
  if (slot == PETIGA_SLOT_MATRIX) { f.vc0 = f.vc1 = 0; }
  return f;
}

// demo/L2Projection.c:3-61
__host__ __device__ inline double l2_function(int choice, int dim, const double* x) {
  double f = 0;
  switch (choice) {
    case 0: for (int i = 0; i < dim; i++) f += x[i]; return f;
    case 1: for (int i = 0; i < dim; i++) f += x[i] * x[i]; return f;
    case 2: for (int i = 0; i < dim; i++) f += x[i] * x[i] * x[i]; return f;
    case 3: for (int i = 0; i < dim; i++) f += x[i] * x[i] * x[i] * x[i]; return f;
    case 4: {
      double X = 2.5 * x[0] + 1, Y = 2.0 * (dim > 1 ? x[1] : 0.0) + 0;
      return exp(-X * X - Y * Y) + 0.5 * exp(-(X - 2) * (X - 2) - (Y - 0.5) * (Y - 0.5));
    }
    case 5: {
      double X = x[0] * 3, Y = (dim > 1 ? x[1] : 0.0) * 3;
      return 3 * pow(1 - X, 2) * exp(-pow(X, 2) - pow(Y + 1, 2)) - 10 * (X / 5 - pow(X, 3) - pow(Y, 5)) * exp(-pow(X, 2) - pow(Y, 2)) -
             1.0 / 3 * exp(-pow(X + 1, 2) - pow(Y, 2));
    }
    case 6: f = 1; for (int i = 0; i < dim; i++) f *= sin(M_PI * x[i]); return f;
    case 7: for (int i = 0; i < dim; i++) f += (x[i] < 0.0) ? -1.0 : +1.0; return f;
  }
  return 0;
}

// What a form sees at one quadrature point (the device "IGAPoint": include/petiga.h:644-703)
struct QPoint {
  double x[3];          // physical point (IGAPointFormGeomMap)
  double u[kMaxDof];    // IGAPointFormValue(U)
  double v[kMaxDof];    // IGAPointFormValue(V)
  double gu[kMaxDof][3];// IGAPointFormGrad(U)
  double d2u[kMaxDof];  // IGAPointFormDel2(U)
  double w[kMaxDof];    // IGAPointFormValue of the third vector: U0 (IE drivers) or A (I2 drivers)
  // boundary-integral pass (p->atboundary, include/petiga.h:645-647,668): only the generic kernel's face mode sets these
  int atboundary;
  double normal[3];     // outward unit normal (IGA_GetNormal, src/petigaval.F90:45-99)
  double hn;            // demo/NitscheMethod.c:58-67 NormalMeshSize: 2 / |G^T n|, G = IGAPointFormInvGradGeomMap
  int maxdeg;           // max axis degree (Degree(), :48-56)
};

// Fill the coefficient tensors of one quadrature point.
//   C : [DOF][DOF][NA][NA]  (NA = mc1-mc0), index ((i*DOF+j)*NA+al)*NA+be, components relative to mc0
//   fv: [DOF][NV]           (NV = vc1-vc0), index i*NV+al, components relative to vc0
// Both are pre-zeroed by the caller.
template <int DIM>
__host__ __device__ __forceinline__ void form_coefficients_rt(int form, int slot, const double* prm, double shift, double t, const QPoint& q,
                                                              const int DOF, int NA, int NV, double* C, double* fv) {
  (void)t;
  switch (form) {
    case PETIGA_FORM_POISSON:   // demo/Poisson3D.c:18,20 ; residual/tangent of the same problem for SNES slots
      if (C && NA) for (int d = 0; d < DIM; d++) C[d * NA + d] = 1.0;
      if (fv && NV) {
        if (slot == PETIGA_SLOT_FUNCTION) { fv[0] = -1.0; for (int d = 0; d < DIM; d++) fv[1 + d] = q.gu[0][d]; }
        else fv[0] = 1.0;
      }
      break;
    case PETIGA_FORM_LAPLACE:   // demo/Laplace.c:44-45
      if (C && NA) for (int d = 0; d < DIM; d++) C[d * NA + d] = 1.0;
      break;
    case PETIGA_FORM_BOUNDARYINTEGRAL:   // demo/BoundaryIntegral.c:27-39 Laplace()
      if (C && NA) for (int d = 0; d < DIM; d++) C[d * NA + d] = 1.0;
      break;
    case PETIGA_FORM_NEUMANN: {   // demo/Neumann.c:10-13,28-45
      if (C && NA) for (int d = 0; d < DIM; d++) C[d * NA + d] = 1.0;
      if (fv && NV) fv[0] = 4 * M_PI * M_PI * (sin(2 * M_PI * q.x[0]) + sin(2 * M_PI * q.x[1]) + sin(2 * M_PI * q.x[2]));
      break;
    }
    case PETIGA_FORM_CONVTEST: {   // test/ConvTest.c:30-69: c N_a N_b + k grad N_a . grad N_b ; f = (c + k dim pi^2) prod sin(pi x_i)
      const double c = prm[0], k = prm[1];
      if (C && NA) { C[0] = c; for (int d = 0; d < DIM; d++) C[(1 + d) * NA + (1 + d)] = k; }
      if (fv && NV) { double f = c + k * DIM * M_PI * M_PI; for (int d = 0; d < DIM; d++) f *= sin(M_PI * q.x[d]); fv[0] = f; }
      break;
    }
    case PETIGA_FORM_L2PROJECTION:  // demo/L2Projection.c:81-85
      if (C && NA) C[0] = 1.0;
      if (fv && NV) fv[0] = l2_function((int)prm[0], DIM, q.x);
      break;
    case PETIGA_FORM_MASS:      // test/IGACreate.c:24-41
      if (C && NA) for (int i = 0; i < DOF; i++) C[(i * DOF + i) * NA * NA] = 1.0;
      if (fv && NV) for (int i = 0; i < DOF; i++) fv[i * NV] = 1.0;
      break;
    case PETIGA_FORM_ELASTICITY3D: {  // demo/Elasticity3D.c:33-41, literal (note the mu*mu of :37)
      if (!(C && NA) || DIM != 3 || DOF != 3) break;
      const double la = prm[0], mu = prm[1];
#define CE(i, j, al, be) C[(((i) * DOF + (j)) * NA + (al)) * NA + (be)]
      CE(0, 0, 0, 0) = la + 2 * mu; CE(0, 0, 1, 1) = mu; CE(0, 0, 2, 2) = mu;
      CE(0, 1, 0, 1) = la; CE(0, 1, 1, 0) = mu;
      CE(0, 2, 0, 2) = la; CE(0, 2, 2, 0) = mu;
      CE(1, 0, 0, 1) = mu; CE(1, 0, 1, 0) = la;
      CE(1, 1, 1, 1) = la + 2 * mu; CE(1, 1, 2, 2) = mu; CE(1, 1, 0, 0) = mu * mu;
      CE(1, 2, 1, 2) = la; CE(1, 2, 2, 1) = mu;
      CE(2, 0, 0, 2) = mu; CE(2, 0, 2, 0) = la;
      CE(2, 1, 1, 2) = mu; CE(2, 1, 2, 1) = la;
      CE(2, 2, 0, 0) = mu; CE(2, 2, 1, 1) = mu; CE(2, 2, 2, 2) = la + 2 * mu;
      break;
    }
    case PETIGA_FORM_ELASTICITY: {    // demo/Elasticity.c:36-44
      if (!(C && NA) || DOF != DIM) break;
      const double la = prm[0], mu = prm[1];
      for (int i = 0; i < DOF; i++)
        for (int j = 0; j < DOF; j++)
          for (int al = 0; al < DIM; al++)
            for (int be = 0; be < DIM; be++)
              CE(i, j, al, be) = (i == j && al == be ? mu : 0.0) + (al == i && be == j ? la : 0.0) + (al == j && be == i ? mu : 0.0);
      break;
    }
#undef CE
    case PETIGA_FORM_CAHNHILLIARD2D:    // demo/CahnHilliard2D.c:9-32,84-197  (chemical potential scaled by 3*alpha)
    case PETIGA_FORM_CAHNHILLIARD3D: {  // demo/CahnHilliard3D.c:11-52,54-169 (scaled by L0^2/lambda); same residual/tangent in DIM dims
      const double theta = prm[0];
      const double scale = (form == PETIGA_FORM_CAHNHILLIARD2D) ? 3 * prm[1] : prm[1] * prm[1] / prm[2];
      const double c = q.u[0], c_t = q.v[0], del2_c = q.d2u[0];
      const double M = c * (1 - c), dM = 1 - 2 * c, d2M = -2;
      double dmu = 0.5 / theta * 1 / (c * (1 - c)) - 2; dmu *= scale;
      const double t1 = M * dmu + dM * del2_c;
      if (fv && NV) {
        fv[0] = c_t;
        for (int d = 0; d < DIM; d++) fv[1 + d] = q.gu[0][d] * t1;
        fv[1 + DIM] = M * del2_c;
      }
      if (C && NA) {
        double d2mu = 0.5 / theta * (2 * c - 1) / (c * c * (1 - c) * (1 - c)); d2mu *= scale;
        const double t2 = (dM * dmu + M * d2mu + d2M * del2_c);
        C[0 * NA + 0] = shift;
        for (int d = 0; d < DIM; d++) {
          C[(1 + d) * NA + (1 + d)] = t1;
          C[(1 + d) * NA + 0] = q.gu[0][d] * t2;
          C[(1 + d) * NA + (1 + DIM)] = q.gu[0][d] * dM;
        }
        C[(1 + DIM) * NA + 0] = dM * del2_c;
        C[(1 + DIM) * NA + (1 + DIM)] = M;
      }
      break;
    }
    case PETIGA_FORM_BRATU: {   // demo/BratuFJ.F90:22-62 (Function), :64-114 (Jacobian), :118-150 (IFunction), IJacobian
      const double lam = prm[0], eu = exp(q.u[0]);
      if (slot == PETIGA_SLOT_RHSFUNCTION || slot == PETIGA_SLOT_RHSJACOBIAN) {
        // explicit form u_t = lap u + lambda exp(u): G_a = -grad N_a . grad u + N_a lambda exp(u) (no reference demo registers an
        // RHSFunction; this exercises IGAComputeRHSFunction/RHSJacobian, src/petigats.c:357-477)
        if (fv && NV) { fv[0] = lam * eu; for (int d = 0; d < DIM; d++) fv[1 + d] = -q.gu[0][d]; }
        if (C && NA) { C[0] = lam * eu; for (int d = 0; d < DIM; d++) C[(1 + d) * NA + (1 + d)] = -1.0; }
        break;
      }
      const bool tr = (slot == PETIGA_SLOT_IFUNCTION || slot == PETIGA_SLOT_IJACOBIAN);
      if (fv && NV) { fv[0] = (tr ? q.v[0] : 0.0) - lam * eu; for (int d = 0; d < DIM; d++) fv[1 + d] = q.gu[0][d]; }
      if (C && NA) { C[0] = (tr ? shift : 0.0) - lam * eu; for (int d = 0; d < DIM; d++) C[(1 + d) * NA + (1 + d)] = 1.0; }
      break;
    }
    case PETIGA_FORM_SNES2D: {   // test/Test_SNES_2D.c:12-72: L2 projection of Peaks, Poisson, reaction-diffusion, Bratu
      if (DIM != 2 || DOF != 4) break;
      if (fv && NV) {
        fv[0 * NV + 0] = q.u[0] - l2_function(5, 2, q.x);
        fv[1 * NV + 0] = -1.0; fv[1 * NV + 1] = q.gu[1][0]; fv[1 * NV + 2] = q.gu[1][1];
        fv[2 * NV + 0] = q.u[2] - 1.0; fv[2 * NV + 1] = q.gu[2][0]; fv[2 * NV + 2] = q.gu[2][1];
        fv[3 * NV + 0] = -1.0 * exp(q.u[3]); fv[3 * NV + 1] = q.gu[3][0]; fv[3 * NV + 2] = q.gu[3][1];
      }
      if (C && NA) {
#define CD(i, al, be) C[(((i) * DOF + (i)) * NA + (al)) * NA + (be)]
        CD(0, 0, 0) = 1.0;
        CD(1, 1, 1) = 1.0; CD(1, 2, 2) = 1.0;
        CD(2, 0, 0) = 1.0; CD(2, 1, 1) = 1.0; CD(2, 2, 2) = 1.0;
        CD(3, 1, 1) = 1.0; CD(3, 2, 2) = 1.0; CD(3, 0, 0) = -1.0 * exp(q.u[3]);
#undef CD
      }
      break;
    }
    case PETIGA_FORM_PATTERNFORMATION: {   // demo/PatternFormation.c:26-141; prm = {IMPLICIT, delta, D1, D2, alpha, beta, gamma, tau1, tau2}
      if (DIM != 2 || DOF != 2) break;
      const bool impl = prm[0] != 0.0;
      const double delta = prm[1], D1 = prm[2], D2 = prm[3], alpha = prm[4], beta = prm[5], gamma = prm[6], tau1 = prm[7], tau2 = prm[8];
      const double u = impl ? q.u[0] : q.w[0], v = impl ? q.u[1] : q.w[1];
      if (fv && NV) {
        const double f = alpha * u * (1 - tau1 * v * v) + v * (1 - tau2 * u);
        const double g = beta * v * (1 + alpha * tau1 / beta * u * v) + u * (gamma + tau2 * v);
        fv[0 * NV + 0] = q.v[0] - f; fv[0 * NV + 1] = delta * D1 * q.gu[0][0]; fv[0 * NV + 2] = delta * D1 * q.gu[0][1];
        fv[1 * NV + 0] = q.v[1] - g; fv[1 * NV + 1] = delta * D2 * q.gu[1][0]; fv[1 * NV + 2] = delta * D2 * q.gu[1][1];
      }
      if (C && NA) {
#define CB(i, j, al, be) C[(((i) * DOF + (j)) * NA + (al)) * NA + (be)]
        CB(0, 0, 0, 0) = shift; CB(0, 0, 1, 1) = delta * D1; CB(0, 0, 2, 2) = delta * D1;
        CB(1, 1, 0, 0) = shift; CB(1, 1, 1, 1) = delta * D2; CB(1, 1, 2, 2) = delta * D2;
        if (impl) {
          const double uu = q.u[0], vv = q.u[1];
          CB(0, 0, 0, 0) -= alpha * (1 - tau1 * vv * vv) - tau2 * vv;
          CB(0, 1, 0, 0) -= -2 * alpha * tau1 * uu * vv + (1 - tau2 * uu);
          CB(1, 0, 0, 0) -= alpha * tau1 * vv * vv + (gamma + tau2 * vv);
          CB(1, 1, 0, 0) -= (beta + 2 * alpha * tau1 * uu * vv) + tau2 * uu;
        }
#undef CB
      }
      break;
    }
    case PETIGA_FORM_ELASTICROD: {   // demo/ElasticRodFJ.F90:19-95; prm = {rho, E}; shift = shiftA
      const double rho = prm[0], E = prm[1];
      if (fv && NV) { fv[0] = rho * q.w[0]; for (int d = 0; d < DIM; d++) fv[1 + d] = E * q.gu[0][d]; }
      if (C && NA) { C[0] = shift * rho; for (int d = 0; d < DIM; d++) C[(1 + d) * NA + (1 + d)] = E; }
      break;
    }
    case PETIGA_FORM_NITSCHE: {   // demo/NitscheMethod.c:70-119
      if (!q.atboundary) {
        if (C && NA) for (int d = 0; d < DIM; d++) C[(1 + d) * NA + (1 + d)] = 1.0;
        if (fv && NV) fv[0] = -2.0 * DIM;
      } else {
        double g = 0.0;
        for (int d = 0; d < DIM; d++) g += q.x[d] * q.x[d];
        const double alpha = 5 * (q.maxdeg + 1) / q.hn;
        if (C && NA) {
          C[0] = alpha;
          for (int d = 0; d < DIM; d++) { C[0 * NA + (1 + d)] = -q.normal[d]; C[(1 + d) * NA + 0] = -q.normal[d]; }
        }
        if (fv && NV) { fv[0] = alpha * g; for (int d = 0; d < DIM; d++) fv[1 + d] = -q.normal[d] * g; }
      }
      break;
    }
  }
}

// compile-time dof front end of the tuned kernels (same code after inlining)
template <int DIM, int DOF>
__host__ __device__ __forceinline__ void form_coefficients(int form, int slot, const double* prm, double shift, double t, const QPoint& q,
                                                           int NA, int NV, double* C, double* fv) {
  form_coefficients_rt<DIM>(form, slot, prm, shift, t, q, DOF, NA, NV, C, fv);
}

}  // namespace pc
