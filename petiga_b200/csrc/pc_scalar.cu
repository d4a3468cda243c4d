// pc_scalar.cu -- IGAComputeScalar / IGAComputeErrorNorm on the device (SURVEY.md 8f-1).
//
// Replaces the element/point loop of src/petigacomp.c:35-96: per quadrature point a Scalar callback produces n
// numbers which are accumulated with the weight detJac*weight (IGAPointAddArray, src/petigapoint.c:451-465), then
// MPI_Allreduce(SUM) -> here a two-stage deterministic reduction (per-CTA partials in a fixed order, then one warp)
// followed by ncclAllReduce over the ranks.  The built-in callbacks are
//   PETIGA_SCALAR_ERRNORM   ErrorSqr of IGAComputeErrorNorm (src/petigacomp.c:103-124): |D^k u_exact - D^k u_h|^2 per field
//   PETIGA_SCALAR_CH_STATS  the CahnHilliard monitor (demo/CahnHilliard2D.c:36-58): free energy, 2nd and 3rd moments
//
// A thread owns a quadrature point.  The reference evaluates D^k u_h by contracting U with the k-th order *shape
// functions* of every node (IGAPointEvaluate, src/petigapoint.c:387-412), which needs the rationalised and
// pushed-forward basis (K4-K7).  Here the same numbers come from the *field* side: the parametric jets of
// w = sum W_a N_a, w*x and w*u are accumulated once from the 1-D tables, the NURBS quotient rule and the geometry
// push-forward  H_x = E1^T (H_xi - sum_m (grad_x u)_m X2_m) E1  are applied to the 3+dof fields instead of the nen
// basis functions.  Degrees may differ per axis; derivative order 0..2, identity, mapped and rational geometry.
#include <cmath>
#include <cstring>

#include "pc_element.cuh"
#include "pc_plan.h"

namespace pc {

namespace {

constexpr int kMaxS = 8;          // scalars per call
constexpr int kThreads = 128;

struct ScalarParams {
  DevAxis ax[3];
  int dim, dof, nelem;
  const int* localrow;     // ghost box -> local row
  const double* U;         // unified local state [nloc*dof] or NULL
  const double* X;         // [ghost box][dim] or NULL
  const double* Wt;        // [ghost box] or NULL
  int sid, n, kmax;
  double prm[8];
  double* partial;         // [gridDim.x][n]
};

// jet of one field in DIM parametric directions: value, gradient, symmetric Hessian (packed upper triangle)
template <int DIM>
struct Jet {
  static constexpr int NH = DIM * (DIM + 1) / 2;
  double v, g[DIM], h[NH];
  __device__ void zero() { v = 0; for (int d = 0; d < DIM; d++) g[d] = 0; for (int k = 0; k < NH; k++) h[k] = 0; }
};
__device__ __forceinline__ int hidx(int DIM, int a, int b) { if (a > b) { int t = a; a = b; b = t; } return a * DIM - a * (a - 1) / 2 + (b - a); }

// test/IGAErrNorm.c:26-52 (id 1, four fields) and demo/L2Projection.c:3-61 (id 2, value only): D^k of field i at x
template <int DIM>
__device__ void exact_field(int id, int choice, int i, const double* x, int k, double* out) {
  const int n = (k == 0) ? 1 : (k == 1 ? DIM : DIM * DIM);
  for (int c = 0; c < n; c++) out[c] = 0.0;
  if (id == 1) {
    double prod = 1.0;
    for (int d = 0; d < DIM; d++) prod *= x[d];
    if (k == 0) {
      double s1 = 0, s2 = 0;
      for (int d = 0; d < DIM; d++) { s1 += x[d]; s2 += x[d] * x[d]; }
      out[0] = (i == 0) ? 1.0 : (i == 1 ? s1 : (i == 2 ? s2 : prod));
    } else if (k == 1) {
      for (int d = 0; d < DIM; d++) out[d] = (i == 0) ? 0.0 : (i == 1 ? 1.0 : (i == 2 ? 2 * x[d] : prod / x[d]));
    } else {
      for (int a = 0; a < DIM; a++)
        for (int b = 0; b < DIM; b++)
          out[a * DIM + b] = (i == 2) ? ((a == b) ? 2.0 : 0.0) : (i == 3 ? ((a == b) ? 0.0 : prod / (x[a] * x[b])) : 0.0);
    }
  } else if (id == 2 && k == 0) {
    double xx[3] = {0, 0, 0};
    for (int d = 0; d < DIM; d++) xx[d] = x[d];
    out[0] = l2_function(choice, DIM, xx);
  } else if (id == 4 && k <= 1) {   // test/ConvTest.c:8-28 Solution: prod sin(pi x_i) and its gradient
    if (k == 0) { double v = 1.0; for (int d = 0; d < DIM; d++) v *= sin(M_PI * x[d]); out[0] = v; }
    else
      for (int a = 0; a < DIM; a++) {
        double g = 1.0;
        for (int b = 0; b < DIM; b++) g *= (a == b) ? M_PI * cos(M_PI * x[b]) : sin(M_PI * x[b]);
        out[a] = g;
      }
  } else if (id == 3 && k == 0) {   // demo/Neumann.c:5-8 Solution (x has zeros above DIM)
    double xx[3] = {0, 0, 0};
    for (int d = 0; d < DIM; d++) xx[d] = x[d];
    out[0] = sin(2 * M_PI * xx[0]) + sin(2 * M_PI * xx[1]) + sin(2 * M_PI * xx[2]);
  }
}

// accumulate the parametric jet of sum_a coef[a] N_a at one quadrature point from the 1-D tables
template <int DIM>
__device__ __forceinline__ void accumulate(const ScalarParams& sp, const int* ID, const int* qi, const double* coef, int stride, int kmax,
                                           Jet<DIM>& J) {
  J.zero();
  const int n0 = sp.ax[0].nen, n1 = (DIM > 1) ? sp.ax[1].nen : 1, n2 = (DIM > 2) ? sp.ax[2].nen : 1;
  const double* t0 = sp.ax[0].value + (size_t)(ID[0] * sp.ax[0].nqp + qi[0]) * n0 * 5;
  const double* t1 = (DIM > 1) ? sp.ax[1].value + (size_t)(ID[1] * sp.ax[1].nqp + qi[1]) * n1 * 5 : nullptr;
  const double* t2 = (DIM > 2) ? sp.ax[2].value + (size_t)(ID[2] * sp.ax[2].nqp + qi[2]) * n2 * 5 : nullptr;
  for (int ka = 0; ka < n2; ka++) {
    const double k0 = (DIM > 2) ? t2[ka * 5] : 1.0, k1 = (DIM > 2) ? t2[ka * 5 + 1] : 0.0, k2 = (DIM > 2) ? t2[ka * 5 + 2] : 0.0;
    for (int ja = 0; ja < n1; ja++) {
      const double j0 = (DIM > 1) ? t1[ja * 5] : 1.0, j1 = (DIM > 1) ? t1[ja * 5 + 1] : 0.0, j2 = (DIM > 1) ? t1[ja * 5 + 2] : 0.0;
      // line sums along axis 0
      double s0 = 0, s1 = 0, s2 = 0;
      const double* c = coef + (size_t)(ka * n1 + ja) * n0 * stride;
      for (int ia = 0; ia < n0; ia++) {
        const double u = c[ia * stride];
        s0 = fma(t0[ia * 5], u, s0);
        if (kmax >= 1) s1 = fma(t0[ia * 5 + 1], u, s1);
        if (kmax >= 2) s2 = fma(t0[ia * 5 + 2], u, s2);
      }
      const double jk00 = j0 * k0;
      J.v = fma(s0, jk00, J.v);
      if (kmax >= 1) {
        J.g[0] = fma(s1, jk00, J.g[0]);
        if (DIM > 1) J.g[1] = fma(s0, j1 * k0, J.g[1]);
        if (DIM > 2) J.g[2] = fma(s0, j0 * k1, J.g[2]);
      }
      if (kmax >= 2) {
        J.h[hidx(DIM, 0, 0)] = fma(s2, jk00, J.h[hidx(DIM, 0, 0)]);
        if (DIM > 1) {
          J.h[hidx(DIM, 0, 1)] = fma(s1, j1 * k0, J.h[hidx(DIM, 0, 1)]);
          J.h[hidx(DIM, 1, 1)] = fma(s0, j2 * k0, J.h[hidx(DIM, 1, 1)]);
        }
        if (DIM > 2) {
          J.h[hidx(DIM, 0, 2)] = fma(s1, j0 * k1, J.h[hidx(DIM, 0, 2)]);
          J.h[hidx(DIM, 1, 2)] = fma(s0, j1 * k1, J.h[hidx(DIM, 1, 2)]);
          J.h[hidx(DIM, 2, 2)] = fma(s0, j0 * k2, J.h[hidx(DIM, 2, 2)]);
        }
      }
    }
  }
}

// NURBS quotient rule on a field jet A = jet(sum c_a W_a N_a) with w = jet(sum W_a N_a) (petigarat.f90.in:24-45 applied to the sum)
template <int DIM>
__device__ __forceinline__ void quotient(Jet<DIM>& A, const Jet<DIM>& w, int kmax) {
  const double iw = 1.0 / w.v;
  A.v *= iw;
  if (kmax >= 1)
    for (int d = 0; d < DIM; d++) A.g[d] = (A.g[d] - A.v * w.g[d]) * iw;
  if (kmax >= 2)
    for (int a = 0; a < DIM; a++)
      for (int b = a; b < DIM; b++) {
        const int k = hidx(DIM, a, b);
        A.h[k] = (A.h[k] - A.g[a] * w.g[b] - A.g[b] * w.g[a] - A.v * w.h[k]) * iw;
      }
}

template <int DIM>
__global__ void __launch_bounds__(kThreads) scalar_kernel(const __grid_constant__ ScalarParams sp) {
  extern __shared__ double sm[];
  const int nen = sp.ax[0].nen * sp.ax[1].nen * sp.ax[2].nen, dof = sp.dof;
  double* Ue = sm;                       // [nen][dof]   (times W_a when rational)
  double* Xe = Ue + nen * dof;           // [nen][DIM]   (times W_a when rational)
  double* We = Xe + nen * DIM;           // [nen]
  __shared__ double red[kThreads / 32][kMaxS];
  const bool mapped = sp.X != nullptr, rational = sp.Wt != nullptr;
  const int kmax = sp.kmax, n = sp.n;
  int nq1[3], nqp = 1;
  for (int d = 0; d < 3; d++) { nq1[d] = sp.ax[d].nqp; nqp *= nq1[d]; }
  double S[kMaxS];
#pragma unroll
  for (int k = 0; k < kMaxS; k++) S[k] = 0.0;

  for (int elem = blockIdx.x; elem < sp.nelem; elem += gridDim.x) {
    int ID[3];
    element_id(sp.ax, elem, ID);
    __syncthreads();
    for (int a = threadIdx.x; a < nen; a += blockDim.x) {   // closure + IGAElementGetValues (petigaelem.c:693-755,1074-1100)
      const int n0 = sp.ax[0].nen, n1 = sp.ax[1].nen;
      const int ia = a % n0, ja = (a / n0) % n1, ka = a / (n0 * n1);
      const int g0 = sp.ax[0].offset[ID[0]] + ia - sp.ax[0].gs;
      const int g1 = sp.ax[1].offset[ID[1]] + ja - sp.ax[1].gs;
      const int g2 = sp.ax[2].offset[ID[2]] + ka - sp.ax[2].gs;
      const int gidx = g0 + sp.ax[0].gw * (g1 + sp.ax[1].gw * g2);
      const double w = rational ? sp.Wt[gidx] : 1.0;
      if (rational) We[a] = w;
      if (mapped) for (int i = 0; i < DIM; i++) Xe[a * DIM + i] = w * sp.X[(size_t)gidx * DIM + i];
      if (sp.U) {
        const int lr = sp.localrow[gidx];
        for (int i = 0; i < dof; i++) Ue[a * dof + i] = w * sp.U[(size_t)lr * dof + i];
      }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < nqp; q += blockDim.x) {
      const int qi[3] = {q % nq1[0], (q / nq1[0]) % nq1[1], q / (nq1[0] * nq1[1])};
      double JW = 1.0, x[3] = {0, 0, 0};
#pragma unroll
      for (int d = 0; d < DIM; d++) {   // IGA_Quadrature_*: W = prod w, J = prod detJac (petiga3d.F90:22-28)
        JW *= sp.ax[d].weight[ID[d] * nq1[d] + qi[d]] * sp.ax[d].detJac[ID[d]];
        x[d] = sp.ax[d].point[ID[d] * nq1[d] + qi[d]];
      }
      Jet<DIM> w;
      double E[DIM][DIM];              // E[d][i] = d xi_d / d x_i
      Jet<DIM> Xj[DIM];
      if (rational) accumulate<DIM>(sp, ID, qi, We, 1, kmax, w);
      if (mapped) {
        for (int i = 0; i < DIM; i++) {
          accumulate<DIM>(sp, ID, qi, Xe + i, DIM, kmax > 1 ? kmax : 1, Xj[i]);
          if (rational) quotient<DIM>(Xj[i], w, kmax > 1 ? kmax : 1);
          x[i] = Xj[i].v;
        }
        double det;   // InverseMap, order 1 (petigamapinv.f90.in:28-31)
        if (DIM == 1) { det = Xj[0].g[0]; E[0][0] = 1.0 / det; }
        else if (DIM == 2) {
          const double a = Xj[0].g[0], b = Xj[0].g[DIM > 1 ? 1 : 0], c = Xj[DIM > 1 ? 1 : 0].g[0], d = Xj[DIM > 1 ? 1 : 0].g[DIM > 1 ? 1 : 0];
          det = a * d - b * c;
          E[0][0] = d / det; E[0][DIM > 1 ? 1 : 0] = -b / det; E[DIM > 1 ? 1 : 0][0] = -c / det; E[DIM > 1 ? 1 : 0][DIM > 1 ? 1 : 0] = a / det;
        } else {
          constexpr int I1 = DIM > 1 ? 1 : 0, I2 = DIM > 2 ? 2 : 0;
          const double a00 = Xj[0].g[0], a01 = Xj[0].g[I1], a02 = Xj[0].g[I2], a10 = Xj[I1].g[0], a11 = Xj[I1].g[I1], a12 = Xj[I1].g[I2],
                       a20 = Xj[I2].g[0], a21 = Xj[I2].g[I1], a22 = Xj[I2].g[I2];
          det = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
          E[0][0] = (a11 * a22 - a12 * a21) / det; E[0][I1] = -(a01 * a22 - a02 * a21) / det; E[0][I2] = (a01 * a12 - a02 * a11) / det;
          E[I1][0] = -(a10 * a22 - a12 * a20) / det; E[I1][I1] = (a00 * a22 - a02 * a20) / det; E[I1][I2] = -(a00 * a12 - a02 * a10) / det;
          E[I2][0] = (a10 * a21 - a11 * a20) / det; E[I2][I1] = -(a00 * a21 - a01 * a20) / det; E[I2][I2] = (a00 * a11 - a01 * a10) / det;
        }
        JW *= det;   // detJac *= detX (petigaelem.c:1024-1029)
      }
      for (int i = 0; i < dof; i++) {
        Jet<DIM> u;
        u.zero();
        if (sp.U) {
          accumulate<DIM>(sp, ID, qi, Ue + i, dof, kmax, u);
          if (rational) quotient<DIM>(u, w, kmax);
        }
        double gu[DIM], hu[DIM][DIM];
        for (int a = 0; a < DIM; a++) { gu[a] = 0; for (int b = 0; b < DIM; b++) hu[a][b] = 0; }
        if (kmax >= 1) {
          if (mapped) { for (int m = 0; m < DIM; m++) { double s = 0; for (int d = 0; d < DIM; d++) s = fma(u.g[d], E[d][m], s); gu[m] = s; } }
          else for (int d = 0; d < DIM; d++) gu[d] = u.g[d];
        }
        if (kmax >= 2) {
          if (mapped) {   // H_x = E^T (H_xi - sum_m gu_m X2_m) E   (ShapeFunctions order 2 + InverseMap E2, applied to the field)
            double T[DIM][DIM];
            for (int a = 0; a < DIM; a++)
              for (int b = 0; b < DIM; b++) {
                double s = u.h[hidx(DIM, a, b)];
                for (int m = 0; m < DIM; m++) s = fma(-gu[m], Xj[m].h[hidx(DIM, a, b)], s);
                T[a][b] = s;
              }
            for (int ii = 0; ii < DIM; ii++)
              for (int jj = 0; jj < DIM; jj++) {
                double s = 0;
                for (int a = 0; a < DIM; a++)
                  for (int b = 0; b < DIM; b++) s = fma(E[a][ii] * E[b][jj], T[a][b], s);
                hu[ii][jj] = s;
              }
          } else
            for (int a = 0; a < DIM; a++)
              for (int b = 0; b < DIM; b++) hu[a][b] = u.h[hidx(DIM, a, b)];
        }
        // ---- the Scalar callbacks ----
        if (sp.sid == PETIGA_SCALAR_ERRNORM) {   // ErrorSqr (petigacomp.c:103-124)
          const int k = (int)sp.prm[0], ex = (int)sp.prm[1];
          double ev[9];
          exact_field<DIM>(ex, (int)sp.prm[2], i, x, k, ev);
          double e2 = 0.0;
          if (k == 0) { const double e = fabs(ev[0] - u.v); e2 = e * e; }
          else if (k == 1) for (int d = 0; d < DIM; d++) { const double e = fabs(ev[d] - gu[d]); e2 += e * e; }
          else for (int a = 0; a < DIM; a++) for (int b = 0; b < DIM; b++) { const double e = fabs(ev[a * DIM + b] - hu[a][b]); e2 += e * e; }
#pragma unroll
          for (int c = 0; c < kMaxDof; c++) if (c == i) S[c] = fma(e2, JW, S[c]);
        } else if (sp.sid == PETIGA_SCALAR_CH_STATS) {   // demo/CahnHilliard2D.c:36-58
          const double theta = sp.prm[0], alpha = sp.prm[1], diff = u.v - sp.prm[2], c = u.v;
          const double g2 = gu[0] * gu[0] + gu[DIM > 1 ? 1 : 0] * gu[DIM > 1 ? 1 : 0];
          const double Efree = c * log(c) + (1 - c) * log(1 - c) + 2 * theta * c * (1 - c) + theta / (3 * alpha) * g2;
          S[0] = fma(Efree, JW, S[0]);
          S[1] = fma(diff * diff, JW, S[1]);
          S[2] = fma(diff * diff * diff, JW, S[2]);
        }
      }
    }
  }
  // deterministic block reduction: shuffle tree inside a warp, warps summed in order by thread 0
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kMaxS; k++) {
    double v = S[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < n) {
    double v = 0.0;
    for (int w = 0; w < kThreads / 32; w++) v += red[w][threadIdx.x];
    sp.partial[(size_t)blockIdx.x * n + threadIdx.x] = v;
  }
}

// second stage: one warp per scalar, fixed-order strided sums + shuffle tree
__global__ void scalar_reduce_kernel(const double* __restrict__ partial, int nblocks, int n, double* __restrict__ out) {
  const int k = blockIdx.x, lane = threadIdx.x;
  double v = 0.0;
  for (int b = lane; b < nblocks; b += 32) v += partial[(size_t)b * n + k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if (lane == 0) out[k] = v;
}

}  // namespace

int allreduce_sum(petiga_cuda_plan* P, double* d_buf, int n);   // pc_comm.cu

}  // namespace pc

using namespace pc;

extern "C" int petiga_cuda_compute_scalar(petiga_cuda_plan* P, int scalar_id, const double* params, int nparams, const double* U, int n,
                                          double* S_host) {
  if (!P || !S_host || n < 1 || n > kMaxS || nparams < 0 || nparams > 8 || (nparams && !params)) { set_error("compute_scalar: bad argument"); return PETIGA_CUDA_ERR_ARG; }
  const Layout& L = P->L;
  if (L.collocation) { set_error("compute_scalar: a collocation plan has no quadrature rule; integrate on the Galerkin plan of the same axes (same numbering)"); return PETIGA_CUDA_ERR_SUP; }
  ScalarParams sp;
  memset(&sp, 0, sizeof(sp));
  for (int k = 0; k < nparams; k++) sp.prm[k] = params[k];
  int kmax = 0;
  if (scalar_id == PETIGA_SCALAR_ERRNORM) {
    const int k = (int)sp.prm[0], ex = (int)sp.prm[1];
    if (k < 0) { set_error("IGAComputeErrorNorm: derivative index must be nonnegative"); return PETIGA_CUDA_ERR_ARG; }   // petigacomp.c:170
    if (k > 2) { set_error("compute_scalar: error norms above the H2 seminorm are not available on the device path"); return PETIGA_CUDA_ERR_SUP; }
    if (n != L.dof || L.dof > kMaxDof) { set_error("compute_scalar: ERRNORM produces dof (<= 4) scalars"); return PETIGA_CUDA_ERR_ARG; }
    if (ex < 0 || ex > 4 || (ex == 1 && L.dof != 4) || ((ex == 2 || ex == 3) && k != 0) || (ex == 4 && k > 1)) { set_error("compute_scalar: exact solution id not applicable"); return PETIGA_CUDA_ERR_SUP; }
    kmax = k;
  } else if (scalar_id == PETIGA_SCALAR_CH_STATS) {
    if (L.dim != 2 || L.dof != 1 || n != 3 || !U) { set_error("compute_scalar: CH_STATS needs dim 2, dof 1, n 3 and a state vector"); return PETIGA_CUDA_ERR_ARG; }
    kmax = 1;
  } else { set_error("compute_scalar: unknown scalar functional"); return PETIGA_CUDA_ERR_ARG; }
  if (kmax > P->order) { set_error("compute_scalar: functional reads derivatives above IGASetOrder"); return PETIGA_CUDA_ERR_ARG; }
  PC_CUDA(cudaSetDevice(P->device));
  const double* U_k = U;
  if (L.nranks > 1 && U) {   // IGAGetLocalVecArray: G2L halo (petigavec.c:256-269)
    int rc = halo_state(P, L.send, L.recv, U, P->d_U_loc.get());
    if (rc) return rc;
    U_k = P->d_U_loc.get();
  }
  for (int d = 0; d < 3; d++) sp.ax[d] = P->dax[d];
  sp.dim = L.dim; sp.dof = L.dof; sp.nelem = L.ax[0].ew * L.ax[1].ew * L.ax[2].ew;
  sp.localrow = P->d_localrow.get(); sp.U = U_k; sp.X = P->d_X.get(); sp.Wt = P->d_W.get();
  sp.sid = scalar_id; sp.n = n; sp.kmax = kmax;
  const int nen = (L.ax[0].p + 1) * (L.ax[1].p + 1) * (L.ax[2].p + 1);
  const size_t smem = (size_t)nen * (L.dof + L.dim + 1) * sizeof(double);
  if (smem > 200 * 1024) { set_error("compute_scalar: element does not fit shared memory"); return PETIGA_CUDA_ERR_SUP; }
  const int blocks = std::max(1, std::min(sp.nelem, P->num_sms * 8));
  if (int rc = P->d_scalar.reserve((size_t)(blocks + 1) * kMaxS)) return rc;
  sp.partial = P->d_scalar.get() + kMaxS;
  cudaEventRecord(P->ev0, P->stream);
#define SK(DIM_)                                                                                                        \
  if (L.dim == DIM_) {                                                                                                  \
    PC_CUDA(cudaFuncSetAttribute(scalar_kernel<DIM_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));         \
    scalar_kernel<DIM_><<<blocks, kThreads, smem, P->stream>>>(sp);                                                     \
  }
  SK(1) SK(2) SK(3)
#undef SK
  PC_CUDA(cudaGetLastError());
  scalar_reduce_kernel<<<n, 32, 0, P->stream>>>(sp.partial, blocks, n, P->d_scalar.get());
  PC_CUDA(cudaGetLastError());
  P->launches += 2;
  cudaEventRecord(P->ev1, P->stream);
  if (L.nranks > 1) {   // MPI_Allreduce(localS, S, n, SUM) (petigacomp.c:90)
    int rc = allreduce_sum(P, P->d_scalar.get(), n);
    if (rc) return rc;
  }
  PC_CUDA(cudaMemcpyAsync(S_host, P->d_scalar.get(), (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, P->stream));
  return petiga_cuda_finish(P);
}
