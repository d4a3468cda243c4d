// iga_host.cpp -- PETSc-free host mirror of PetIGA's IGA API around the assembly path (include/petiga_host.h).
//
// Host work done here (one-time set-up, integer/table work the reference also does on the CPU):
//   knot vectors        IGAAxisInitUniform / IGAAxisSetKnots   (ref: src/petigaaxis.c:401-480)
//   Gauss rule + 1-D basis tables  IGABasisInitQuadrature      (ref: src/petigabasis.c:83-219, petigabsb.f90.in)
//   processor grid + boxes         IGA_Partition / Stage1      (ref: src/petigapart.c, src/petiga.c:1111-1209)
//   collocation tables + boxes     IGASetUseCollocation: one point per basis function, its Greville abscissa
// Everything per-element runs on the GPU through libpetiga_cuda; there is no CPU assembly path here.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <set>
#include <string>
#include <vector>

#include "../../include/petiga_cuda.h"
#include "../../include/petiga_host.h"
#include "gauss_tables.h"

namespace {

thread_local std::string g_msg;
PetscErrorCode fail(PetscErrorCode code, const std::string& m) { g_msg = m; return code; }
PetscErrorCode from_cuda(int rc) {
  if (!rc) return 0;
  g_msg = std::string(petiga_cuda_strerror(rc)) + ": " + petiga_cuda_last_error();
  switch (rc) {
    case PETIGA_CUDA_ERR_ARG: return PETSC_ERR_ARG_OUTOFRANGE;
    case PETIGA_CUDA_ERR_ORDER: return PETSC_ERR_ORDER;
    case PETIGA_CUDA_ERR_SUP: return PETSC_ERR_SUP;
    case PETIGA_CUDA_ERR_MEM: return PETSC_ERR_MEM;
    default: return PETSC_ERR_LIB;
  }
}

}  // namespace

struct _n_IGAAxis {
  int p = 0, m = 1, periodic = 0, nnp = 1, nel = 1;
  std::vector<double> U{-0.5, 0.5};
  std::vector<int> span{0};
  IGA owner = nullptr;
};

// Mat/Vec borrow plan-owned device tables (the CSR pattern); `gen` is the IGA's plan generation at creation, so that a Mat or
// Vec that outlives its set-up (IGARead, IGASetRuleSize, IGADestroy) is refused instead of reading freed device memory.
struct _p_Vec {
  IGA iga; int n; double* d; long gen; };
struct _p_Mat {
  IGA iga; int baij; int bs; int nrows; int64_t nnz; const int* d_rowptr; const int* d_colidx; double* d_values; long gen; };

struct _p_KSP {      // IGACreateKSP: conjugate gradients (petiga_cuda_solve_cg) or GMRES (petiga_cuda_solve_gmres) + Jacobi on the device
  IGA iga; Mat A; double rtol, abstol; int maxits, its; double rnorm;
  bool gmres = false; int restart = 30; KSPConvergedReason reason = KSP_CONVERGED_ITERATING; };

struct _p_IGA {
  IGAComm comm;
  int dim = -1, dof = -1, order = -1, setup = 0;
  int collocation = 0;   // IGASetUseCollocation
  _n_IGAAxis axis[3];
  int rule_nqp[3] = {0, 0, 0};
  int proc_user[3] = {-1, -1, -1};
  std::string mattype;
  // tables
  int nqp[3] = {1, 1, 1};
  std::vector<int> offset[3];
  std::vector<double> detJac[3], weight[3], point[3], value[3];
  // partition
  int proc_sizes[3] = {1, 1, 1}, proc_ranks[3] = {0, 0, 0};
  int elem_start[3] = {0, 0, 0}, elem_width[3] = {1, 1, 1};
  int node_lstart[3] = {0, 0, 0}, node_lwidth[3] = {1, 1, 1}, node_gstart[3] = {0, 0, 0}, node_gwidth[3] = {1, 1, 1};
  int geom_sizes[3] = {1, 1, 1};
  // geometry (natural) and bc
  int nsd = 0; std::vector<double> geomX, geomW; bool rational = false;
  std::vector<double> geomW_all;   // weights as given (kept even when constant, as iga->rationalW is; written back by IGAWrite)
  petiga_cuda_bc bc;
  Vec fixtable = nullptr;
  std::vector<double> fixtable_local;
  bool bc_dirty = true, geom_dirty = true;
  struct Slot { int form = -1; double prm[12] = {0}; int nprm = 0; bool dirty = false; } slots[PETIGA_NSLOTS];
  petiga_layout* layout = nullptr;
  petiga_cuda_plan* plan = nullptr;
  void* stream = nullptr;
  std::vector<std::pair<std::string, double>> options;
  int visit[3][2] = {{0, 0}, {0, 0}, {0, 0}};   // IGASetBoundaryForm
  std::vector<double> bnd_value[3][2]; double bnd_point[3][2] = {{0, 0}, {0, 0}, {0, 0}};   // IGABasis.bnd_* (petigabasis.c:208-217)
  bool async = false;   // IGASetOption("async",1): the drivers only enqueue; IGASynchronize / host getters wait
  long plan_gen = 0;    // bumped whenever the plan is destroyed (Mat/Vec created before that become stale)
};

namespace {

std::set<IGA>& live_igas() { static std::set<IGA> s; return s; }
void drop_plan(IGA g) {
  if (g->plan) { petiga_cuda_plan_destroy(g->plan); g->plan = nullptr; }
  g->plan_gen++;
}
template <class Obj>
PetscErrorCode check_owner(Obj* o, IGA g, const char* what) {
  if (!live_igas().count(o->iga)) return fail(PETSC_ERR_ARG_WRONGSTATE, std::string(what) + ": its IGA was destroyed");
  if (g && o->iga != g) return fail(PETSC_ERR_ARG_WRONG, std::string(what) + " was created by a different IGA");            // PetscCheckSameComm-style
  if (o->gen != o->iga->plan_gen) return fail(PETSC_ERR_ARG_WRONGSTATE, std::string(what) + " predates the current IGASetUp(); create it again");
  return 0;
}

// ---- knots ----
int next_knot(int m, const double* U, int k, int dir) {
  if (dir >= 0) { if (k < 0) return 0; for (int j = k + 1; j < m; j++) if (U[j] > U[k]) return j; return m; }
  if (k > m) return m;
  for (int j = k - 1; j > 0; j--) if (U[j] < U[k]) return j;
  return 0;
}

void axis_finish(_n_IGAAxis* ax) {   // spans + node count from the knot vector (IGAAxisSetUp semantics)
  const int p = ax->p, m = ax->m, n = m - p - 1;
  ax->span.clear();
  for (int k = p; (k = next_knot(m, ax->U.data(), k, 1)) <= n + 1;) ax->span.push_back(k - 1);
  ax->nel = (int)ax->span.size();
  if (ax->periodic) {
    int k = n + 1, j = next_knot(m, ax->U.data(), k, 1), s = j - k, C = p - s;
    ax->nnp = n - C;
  } else ax->nnp = n + 1;
}

// ---- B-spline basis functions and derivatives at one point (Cox-de Boor triangle + derivative
//      recurrences: The NURBS Book A2.3, the algorithm behind src/petigabsb.f90.in:3-63).
//      out[a][k], a = 0..p, k = 0..4 (entries above nd zero). ----
void bspline_ders(int span, double u, int p, int nd, const double* U, double out[][5]) {
  double ndu[9][9], left[9], right[9], a[2][9];
  ndu[0][0] = 1.0;
  for (int j = 1; j <= p; j++) {
    left[j] = u - U[span + 1 - j];
    right[j] = U[span + j] - u;
    double saved = 0.0;
    for (int r = 0; r < j; r++) {
      ndu[j][r] = right[r + 1] + left[j - r];
      double temp = ndu[r][j - 1] / ndu[j][r];
      ndu[r][j] = saved + right[r + 1] * temp;
      saved = left[j - r] * temp;
    }
    ndu[j][j] = saved;
  }
  for (int r = 0; r <= p; r++) { for (int k = 0; k < 5; k++) out[r][k] = 0.0; out[r][0] = ndu[r][p]; }
  for (int r = 0; r <= p; r++) {
    int s1 = 0, s2 = 1;
    a[0][0] = 1.0;
    for (int k = 1; k <= nd; k++) {
      double d = 0.0;
      const int rk = r - k, pk = p - k;
      if (r >= k) { a[s2][0] = a[s1][0] / ndu[pk + 1][rk]; d = a[s2][0] * ndu[rk][pk]; }
      const int j1 = (rk >= -1) ? 1 : -rk, j2 = (r - 1 <= pk) ? k - 1 : p - r;
      for (int j = j1; j <= j2; j++) { a[s2][j] = (a[s1][j] - a[s1][j - 1]) / ndu[pk + 1][rk + j]; d += a[s2][j] * ndu[rk + j][pk]; }
      if (r <= pk) { a[s2][k] = -a[s1][k - 1] / ndu[pk + 1][r]; d += a[s2][k] * ndu[r][pk]; }
      out[r][k] = d;
      std::swap(s1, s2);
    }
  }
  int fac = p;
  for (int k = 1; k <= nd; k++) { for (int r = 0; r <= p; r++) out[r][k] *= fac; fac *= (p - k); }
}

// ---- processor grid (IGA_Partition: src/petigapart.c:12-168; same integer/double arithmetic) ----
int cut2(int M, int N, int m, int n) { return M * (n - 1) + N * (m - 1); }
int cut3(int M, int N, int P, int m, int n, int p) { return N * P * (m - 1) + M * P * (n - 1) + M * N * (p - 1); }
int part2_inner(int size, int M, int N, int& m, int& n) {
  m = (int)(0.5 + std::sqrt(((double)M) / ((double)N) * ((double)size)));
  if (m == 0) m = 1;
  while (m > 0 && size % m) m--;
  n = size / m;
  return cut2(M, N, m, n);
}
void part2(int size, int M, int N, int& m, int& n) {
  int m1, n1, m2, n2;
  int a = part2_inner(size, M, N, m1, n1), b = part2_inner(size, N, M, n2, m2);
  if (a < b) { m = m1; n = n1; } else { m = m2; n = n2; }
  if (M == N && n < m) std::swap(m, n);
}
int part3_inner(int size, int M, int N, int P, int& m, int& n, int& p) {
  m = (int)(0.5 + std::pow(((double)M * (double)M) / ((double)N * (double)P) * (double)size, 1. / 3.));
  if (m == 0) m = 1;
  while (m > 0 && size % m) m--;
  part2(size / m, N, P, n, p);
  int C = cut3(M, N, P, m, n, p), mm, nn, pp, CC;
  for (mm = m; mm >= 1; mm--) { if (size % mm) continue; part2(size / mm, N, P, nn, pp); CC = cut3(M, N, P, mm, nn, pp); if (CC < C) { m = mm; n = nn; p = pp; C = CC; } }
  for (nn = n; nn >= 1; nn--) { if (size % nn) continue; part2(size / nn, M, P, mm, pp); CC = cut3(M, N, P, mm, nn, pp); if (CC < C) { m = mm; n = nn; p = pp; C = CC; } }
  for (pp = p; pp >= 1; pp--) { if (size % pp) continue; part2(size / pp, M, N, mm, nn); CC = cut3(M, N, P, mm, nn, pp); if (CC < C) { m = mm; n = nn; p = pp; C = CC; } }
  return cut3(M, N, P, m, n, p);
}
void part3(int size, int M, int N, int P, int& mo, int& no, int& po) {
  int m[3], n[3], p[3], C[3], best = 0;
  C[0] = part3_inner(size, M, N, P, m[0], n[0], p[0]);
  C[1] = part3_inner(size, N, M, P, n[1], m[1], p[1]);
  C[2] = part3_inner(size, P, M, N, p[2], m[2], n[2]);
  for (int k = 1; k < 3; k++) if (C[k] < C[best]) best = k;
  if (M == N && n[best] < m[best]) std::swap(m[best], n[best]);
  if (M == P && p[best] < m[best]) std::swap(m[best], p[best]);
  if (N == P && p[best] < n[best]) std::swap(n[best], p[best]);
  mo = m[best]; no = n[best]; po = p[best];
}

PetscErrorCode check(IGA iga) { return iga ? 0 : fail(PETSC_ERR_ARG_NULL, "Null IGA"); }

PetscErrorCode fill_space(IGA g, petiga_cuda_space& sp) {
  memset(&sp, 0, sizeof(sp));
  sp.dim = g->dim; sp.dof = g->dof; sp.order = g->order;
  for (int d = 0; d < 3; d++) {
    const _n_IGAAxis& ax = g->axis[d];
    sp.p[d] = ax.p; sp.m[d] = ax.m; sp.nel[d] = g->collocation ? ax.nnp : ax.nel; sp.nnp[d] = ax.nnp; sp.periodic[d] = ax.periodic; sp.nqp1[d] = g->nqp[d];
    sp.U[d] = ax.U.data(); sp.offset[d] = g->offset[d].data(); sp.detJac[d] = g->detJac[d].data();
    sp.weight[d] = g->weight[d].data(); sp.point[d] = g->point[d].data(); sp.value[d] = g->value[d].data();
    sp.proc_sizes[d] = g->proc_sizes[d]; sp.proc_ranks[d] = g->proc_ranks[d];
    sp.elem_start[d] = g->elem_start[d]; sp.elem_width[d] = g->elem_width[d];
    sp.node_lstart[d] = g->node_lstart[d]; sp.node_lwidth[d] = g->node_lwidth[d];
    sp.node_gstart[d] = g->node_gstart[d]; sp.node_gwidth[d] = g->node_gwidth[d];
  }
  sp.collocation = g->collocation;
  return 0;
}

PetscErrorCode ensure_plan(IGA g) {
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  if (!g->plan) {
    petiga_cuda_space sp;
    fill_space(g, sp);
    int rc = petiga_cuda_plan_create(&g->plan, &sp, g->comm.rank, g->comm.size, g->comm.nccl, g->stream, g->comm.device);
    if (rc) return from_cuda(rc);
    g->bc_dirty = g->geom_dirty = true;
    for (auto& s : g->slots) s.dirty = (s.form >= 0);
    for (auto& o : g->options) { rc = petiga_cuda_set_option(g->plan, o.first.c_str(), o.second); if (rc) return from_cuda(rc); }
    for (int d = 0; d < g->dim; d++) {
      rc = petiga_cuda_set_boundary_tables(g->plan, d, g->bnd_value[d][0].data(), g->bnd_value[d][1].data(), g->bnd_point[d][0], g->bnd_point[d][1]);
      if (rc) return from_cuda(rc);
      for (int sd = 0; sd < 2; sd++) { rc = petiga_cuda_set_boundary_form(g->plan, d, sd, g->visit[d][sd]); if (rc) return from_cuda(rc); }
    }
  }
  if (g->geom_dirty) {
    if (g->nsd) {   // ghost-box slice of the natural arrays (src/petigaio.c:255-286)
      const int *gs = g->node_gstart, *gw = g->node_gwidth, *sz = g->geom_sizes;
      std::vector<double> X((size_t)gw[0] * gw[1] * gw[2] * g->nsd), W;
      if (g->rational) W.resize((size_t)gw[0] * gw[1] * gw[2]);
      size_t pos = 0;
      for (int k = gs[2]; k < gs[2] + gw[2]; k++)
        for (int j = gs[1]; j < gs[1] + gw[1]; j++)
          for (int i = gs[0]; i < gs[0] + gw[0]; i++, pos++) {
            size_t nat = (size_t)i + (size_t)sz[0] * ((size_t)j + (size_t)sz[1] * k);
            for (int c = 0; c < g->nsd; c++) X[pos * g->nsd + c] = g->geomX[nat * g->nsd + c];
            if (g->rational) W[pos] = g->geomW[nat];
          }
      int rc = petiga_cuda_set_geometry(g->plan, g->nsd, X.data(), g->rational ? W.data() : nullptr);
      if (rc) return from_cuda(rc);
    } else {
      int rc = petiga_cuda_set_geometry(g->plan, 0, nullptr, nullptr);
      if (rc) return from_cuda(rc);
    }
    g->geom_dirty = false;
  }
  if (g->bc_dirty) {
    petiga_cuda_bc bc = g->bc;
    bc.fixtableU = nullptr;
    int rc = petiga_cuda_set_bc(g->plan, &bc);
    if (rc) return from_cuda(rc);
    if (g->fixtable) {   // IGASetFixTable -> IGAGlobalToLocal: the library scatters the device vector (NCCL halo when distributed)
      rc = petiga_cuda_set_fixtable_device(g->plan, g->fixtable->d);
      if (rc) return from_cuda(rc);
    }
    g->bc_dirty = false;
  }
  for (int s = 0; s < PETIGA_NSLOTS; s++)
    if (g->slots[s].dirty) {
      int rc = petiga_cuda_form_select(g->plan, s, g->slots[s].form, g->slots[s].prm, g->slots[s].nprm);
      if (rc) return from_cuda(rc);
      g->slots[s].dirty = false;
    }
  return 0;
}

// swap01 = 1: AppCtx is {mu, lambda} (demo/Elasticity.c); swap01 = 2: AppCtx starts with a PetscBool (demo/PatternFormation.c:14-24)
struct FormEntry { const void* fn; int slot; int form; int nprm; int swap01; };
#define FN(f) ((const void*)(f))
const FormEntry* lookup_form(const void* fn, int slot) {
  static const FormEntry table[] = {
      {FN(IGADeviceForm_Poisson_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_POISSON, 0, 0},
      {FN(IGADeviceForm_Poisson_Function), PETIGA_SLOT_FUNCTION, PETIGA_FORM_POISSON, 0, 0},
      {FN(IGADeviceForm_Poisson_Jacobian), PETIGA_SLOT_JACOBIAN, PETIGA_FORM_POISSON, 0, 0},
      {FN(IGADeviceForm_Laplace_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_LAPLACE, 0, 0},
      {FN(IGADeviceForm_L2Projection_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_L2PROJECTION, 1, 0},
      {FN(IGADeviceForm_Mass_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_MASS, 0, 0},
      {FN(IGADeviceForm_BoundaryIntegral_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_BOUNDARYINTEGRAL, 0, 0},
      {FN(IGADeviceForm_Neumann_SystemGalerkin), PETIGA_SLOT_SYSTEM, PETIGA_FORM_NEUMANN, 0, 0},
      {FN(IGADeviceForm_ConvTest_Galerkin), PETIGA_SLOT_SYSTEM, PETIGA_FORM_CONVTEST, 2, 0},
      {FN(IGADeviceForm_Laplace_SystemCollocation), PETIGA_SLOT_SYSTEM, PETIGA_FORM_LAPLACE_COLLOCATION, 0, 0},
      {FN(IGADeviceForm_ConvTest_Collocation), PETIGA_SLOT_SYSTEM, PETIGA_FORM_CONVTEST_COLLOCATION, 2, 0},
      {FN(IGADeviceForm_Mass_Matrix), PETIGA_SLOT_MATRIX, PETIGA_FORM_MASS, 0, 0},
      {FN(IGADeviceForm_Mass_Vector), PETIGA_SLOT_VECTOR, PETIGA_FORM_MASS, 0, 0},
      {FN(IGADeviceForm_Elasticity3D_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_ELASTICITY3D, 2, 0},
      {FN(IGADeviceForm_Elasticity_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_ELASTICITY, 2, 1},
      {FN(IGADeviceForm_CahnHilliard2D_Residual), PETIGA_SLOT_IFUNCTION, PETIGA_FORM_CAHNHILLIARD2D, 2, 0},
      {FN(IGADeviceForm_CahnHilliard2D_Tangent), PETIGA_SLOT_IJACOBIAN, PETIGA_FORM_CAHNHILLIARD2D, 2, 0},
      {FN(IGADeviceForm_CahnHilliard3D_Residual), PETIGA_SLOT_IFUNCTION, PETIGA_FORM_CAHNHILLIARD3D, 3, 0},
      {FN(IGADeviceForm_CahnHilliard3D_Tangent), PETIGA_SLOT_IJACOBIAN, PETIGA_FORM_CAHNHILLIARD3D, 3, 0},
      {FN(IGADeviceForm_Bratu_Function), PETIGA_SLOT_FUNCTION, PETIGA_FORM_BRATU, 1, 0},
      {FN(IGADeviceForm_Bratu_Jacobian), PETIGA_SLOT_JACOBIAN, PETIGA_FORM_BRATU, 1, 0},
      {FN(IGADeviceForm_Bratu_IFunction), PETIGA_SLOT_IFUNCTION, PETIGA_FORM_BRATU, 1, 0},
      {FN(IGADeviceForm_Bratu_IJacobian), PETIGA_SLOT_IJACOBIAN, PETIGA_FORM_BRATU, 1, 0},
      {FN(IGADeviceForm_Nitsche_System), PETIGA_SLOT_SYSTEM, PETIGA_FORM_NITSCHE, 0, 0},
      {FN(IGADeviceForm_SNES2D_Function), PETIGA_SLOT_FUNCTION, PETIGA_FORM_SNES2D, 0, 0},
      {FN(IGADeviceForm_SNES2D_Jacobian), PETIGA_SLOT_JACOBIAN, PETIGA_FORM_SNES2D, 0, 0},
      {FN(IGADeviceForm_PatternFormation_IEFunction), PETIGA_SLOT_IEFUNCTION, PETIGA_FORM_PATTERNFORMATION, 9, 2},
      {FN(IGADeviceForm_PatternFormation_IEJacobian), PETIGA_SLOT_IEJACOBIAN, PETIGA_FORM_PATTERNFORMATION, 9, 2},
      {FN(IGADeviceForm_ElasticRod_I2Function), PETIGA_SLOT_I2FUNCTION, PETIGA_FORM_ELASTICROD, 2, 0},
      {FN(IGADeviceForm_ElasticRod_I2Jacobian), PETIGA_SLOT_I2JACOBIAN, PETIGA_FORM_ELASTICROD, 2, 0},
      {FN(IGADeviceForm_Bratu_RHSFunction), PETIGA_SLOT_RHSFUNCTION, PETIGA_FORM_BRATU, 1, 0},
      {FN(IGADeviceForm_Bratu_RHSJacobian), PETIGA_SLOT_RHSJACOBIAN, PETIGA_FORM_BRATU, 1, 0},
  };
  for (const auto& e : table) if (e.fn == fn && e.slot == slot) return &e;
  return nullptr;
}

PetscErrorCode set_form(IGA g, int slot, const void* fn, void* ctx) {
  if (PetscErrorCode e = check(g)) return e;
  auto& s = g->slots[slot];
  if (!fn) { s.form = -1; s.nprm = 0; s.dirty = true; return 0; }   // a cleared callback reaches the plan too (form_select(-1))
  const FormEntry* fe = lookup_form(fn, slot);
  if (!fe) return fail(PETSC_ERR_SUP, "IGASetForm*: host callbacks cannot run on the GPU; pass one of the IGADeviceForm_* sentinels");
  if (fe->nprm && !ctx) return fail(PETSC_ERR_ARG_NULL, "IGASetForm*: this form needs its AppCtx");   // nothing committed yet
  s.form = fe->form; s.nprm = fe->nprm; s.dirty = true;
  memset(s.prm, 0, sizeof(s.prm));
  if (fe->swap01 == 2) {   // {PetscBool flag; PetscReal ...}: the flag occupies the first 8-byte slot of the struct
    s.prm[0] = (double)(*(const int*)ctx != 0);
    for (int k = 1; k < fe->nprm; k++) s.prm[k] = ((const double*)ctx)[k];
  } else {
    for (int k = 0; k < fe->nprm; k++) s.prm[k] = ((const double*)ctx)[k];
    if (fe->swap01 == 1) std::swap(s.prm[0], s.prm[1]);   // demo/Elasticity.c AppCtx is {mu, lambda}
  }
  return 0;
}

PetscErrorCode host_sentinel() { return fail(PETSC_ERR_SUP, "device form sentinel called on the host"); }

}  // namespace

extern "C" {

const char* IGAGetLastErrorMessage(void) { return g_msg.c_str(); }

#define SENT3(name) PetscErrorCode name(IGAPoint, PetscScalar*, void*) { return host_sentinel(); }
#define SENT4(name) PetscErrorCode name(IGAPoint, PetscScalar*, PetscScalar*, void*) { return host_sentinel(); }
#define SENTF(name) PetscErrorCode name(IGAPoint, const PetscScalar*, PetscScalar*, void*) { return host_sentinel(); }
#define SENTI(name) PetscErrorCode name(IGAPoint, PetscReal, const PetscScalar*, PetscReal, const PetscScalar*, PetscScalar*, void*) { return host_sentinel(); }
SENT4(IGADeviceForm_Poisson_System) SENTF(IGADeviceForm_Poisson_Function) SENTF(IGADeviceForm_Poisson_Jacobian)
SENT4(IGADeviceForm_Laplace_System) SENT4(IGADeviceForm_L2Projection_System) SENT4(IGADeviceForm_Mass_System)
SENT3(IGADeviceForm_Mass_Matrix) SENT3(IGADeviceForm_Mass_Vector)
SENT4(IGADeviceForm_BoundaryIntegral_System) SENT4(IGADeviceForm_Neumann_SystemGalerkin) SENT4(IGADeviceForm_ConvTest_Galerkin)
SENT4(IGADeviceForm_Laplace_SystemCollocation) SENT4(IGADeviceForm_ConvTest_Collocation)
PetscErrorCode IGADeviceExact_ConvTest(IGAPoint, PetscInt, PetscScalar*, void*) { return host_sentinel(); }
PetscErrorCode IGADeviceExact_Neumann(IGAPoint, PetscInt, PetscScalar*, void*) { return host_sentinel(); }
SENT4(IGADeviceForm_Elasticity3D_System) SENT4(IGADeviceForm_Elasticity_System)
SENTI(IGADeviceForm_CahnHilliard2D_Residual) SENTI(IGADeviceForm_CahnHilliard2D_Tangent)
SENTI(IGADeviceForm_CahnHilliard3D_Residual) SENTI(IGADeviceForm_CahnHilliard3D_Tangent)
PetscErrorCode IGADeviceScalar_CahnHilliard2D_Stats(IGAPoint, const PetscScalar*, PetscInt, PetscScalar*, void*) { return host_sentinel(); }
PetscErrorCode IGADeviceExact_ErrNormTest(IGAPoint, PetscInt, PetscScalar*, void*) { return host_sentinel(); }
PetscErrorCode IGADeviceExact_L2Projection(IGAPoint, PetscInt, PetscScalar*, void*) { return host_sentinel(); }
SENTF(IGADeviceForm_Bratu_Function) SENTF(IGADeviceForm_Bratu_Jacobian) SENTI(IGADeviceForm_Bratu_IFunction) SENTI(IGADeviceForm_Bratu_IJacobian)
SENT4(IGADeviceForm_Nitsche_System) SENTF(IGADeviceForm_SNES2D_Function) SENTF(IGADeviceForm_SNES2D_Jacobian)
#define SENT3V(name) PetscErrorCode name(IGAPoint, PetscReal, const PetscScalar*, PetscReal, const PetscScalar*, PetscReal, const PetscScalar*, PetscScalar*, void*) { return host_sentinel(); }
#define SENTR(name) PetscErrorCode name(IGAPoint, PetscReal, const PetscScalar*, PetscScalar*, void*) { return host_sentinel(); }
SENT3V(IGADeviceForm_PatternFormation_IEFunction) SENT3V(IGADeviceForm_PatternFormation_IEJacobian)
SENT3V(IGADeviceForm_ElasticRod_I2Function) SENT3V(IGADeviceForm_ElasticRod_I2Jacobian)
SENTR(IGADeviceForm_Bratu_RHSFunction) SENTR(IGADeviceForm_Bratu_RHSJacobian)

PetscErrorCode IGA_Partition(PetscInt size, PetscInt rank, PetscInt dim, const PetscInt N[], PetscInt n[], PetscInt i[]) {
  if (size < 1) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of partitions must be positive");
  if (i && (rank < 0 || rank >= size)) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Partition index out of range");
  switch (dim) {
    case 3:
      if (n[0] < 1 && n[1] < 1 && n[2] < 1) part3(size, N[0], N[1], N[2], n[0], n[1], n[2]);
      else if (n[0] < 1 && n[1] < 1) part2(size / n[2], N[0], N[1], n[0], n[1]);
      else if (n[0] < 1 && n[2] < 1) part2(size / n[1], N[0], N[2], n[0], n[2]);
      else if (n[1] < 1 && n[2] < 1) part2(size / n[0], N[1], N[2], n[1], n[2]);
      else if (n[0] < 1) n[0] = size / (n[1] * n[2]);
      else if (n[1] < 1) n[1] = size / (n[0] * n[2]);
      else if (n[2] < 1) n[2] = size / (n[0] * n[1]);
      break;
    case 2:
      if (n[0] < 1 && n[1] < 1) part2(size, N[0], N[1], n[0], n[1]);
      else if (n[0] < 1) n[0] = size / n[1];
      else if (n[1] < 1) n[1] = size / n[0];
      break;
    case 1: if (n[0] < 1) n[0] = size; break;
    default: return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of dimensions must be in range [1,3]");
  }
  int prod = 1;
  for (int k = 0; k < dim; k++) prod *= n[k];
  if (prod != size) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Bad partition");
  for (int k = 0; k < dim; k++) if (N[k] < n[k]) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Partition is too fine");
  if (i) for (int k = 0; k < dim; k++) { i[k] = rank % n[k]; rank -= i[k]; rank /= n[k]; }
  return 0;
}

PetscErrorCode IGACreate(IGAComm comm, IGA* iga) {
  if (!iga) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (comm.size < 1 || comm.rank < 0 || comm.rank >= comm.size) return fail(PETSC_ERR_ARG_OUTOFRANGE, "bad communicator");
  IGA g = new _p_IGA();
  g->comm = comm;
  memset(&g->bc, 0, sizeof(g->bc));
  for (int d = 0; d < 3; d++) g->axis[d].owner = g;
  live_igas().insert(g);
  *iga = g;
  return 0;
}

PetscErrorCode IGADestroy(IGA* iga) {
  if (!iga || !*iga) return 0;
  IGA g = *iga;
  drop_plan(g);
  if (g->layout) petiga_layout_destroy(g->layout);
  live_igas().erase(g);
  delete g;
  *iga = nullptr;
  return 0;
}

PetscErrorCode IGASetDim(IGA g, PetscInt dim) {
  if (PetscErrorCode e = check(g)) return e;
  if (dim < 1 || dim > 3) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of parametric dimensions must be in range [1,3]");
  if (g->dim > 0 && g->dim != dim) return fail(PETSC_ERR_ARG_WRONGSTATE, "Cannot change IGA dim after it was set");
  g->dim = dim;
  return 0;
}
PetscErrorCode IGAGetDim(IGA g, PetscInt* dim) { if (PetscErrorCode e = check(g)) return e; *dim = g->dim; return 0; }
PetscErrorCode IGASetDof(IGA g, PetscInt dof) {
  if (PetscErrorCode e = check(g)) return e;
  if (dof < 1) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of DOFs per node must be greater than one");
  if (g->dof > 0 && g->dof != dof) return fail(PETSC_ERR_ARG_WRONGSTATE, "Cannot change number of DOFs after it was set");
  g->dof = dof;
  return 0;
}
PetscErrorCode IGAGetDof(IGA g, PetscInt* dof) { if (PetscErrorCode e = check(g)) return e; *dof = g->dof; return 0; }
PetscErrorCode IGASetOrder(IGA g, PetscInt order) {
  if (PetscErrorCode e = check(g)) return e;
  if (order < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Order must be nonnegative");
  g->order = order < 1 ? 1 : (order > 4 ? 4 : order);   // PetscClipInterval(order,1,4): src/petiga.c:470
  return 0;
}
PetscErrorCode IGASetProcessors(IGA g, PetscInt i, PetscInt processors) {
  if (PetscErrorCode e = check(g)) return e;
  if (i < 0 || i > 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Index must be in [0,2]");
  if (g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Cannot call after IGASetUp()");
  g->proc_user[i] = processors;
  return 0;
}
PetscErrorCode IGAGetAxis(IGA g, PetscInt i, IGAAxis* axis) {
  if (PetscErrorCode e = check(g)) return e;
  if (i < 0 || i > 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Index must be in [0,2]");
  *axis = &g->axis[i];
  return 0;
}
PetscErrorCode IGASetRuleSize(IGA g, PetscInt i, PetscInt nqp) {
  if (PetscErrorCode e = check(g)) return e;
  if (i < 0 || i > 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Index must be in [0,2]");
  if (nqp < 1 || nqp > 10) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of quadrature points not implemented");
  g->rule_nqp[i] = nqp;
  g->setup = 0;   // IGASetRuleSize resets the setup stage in the reference
  drop_plan(g);
  return 0;
}
// include/petiga.h IGASetUseCollocation (src/petiga.c): chooses the discretisation before IGASetUp
PetscErrorCode IGASetUseCollocation(IGA g, PetscBool flag) {
  if (PetscErrorCode e = check(g)) return e;
  const int c = flag ? 1 : 0;
  if (g->setup && c != g->collocation) return fail(PETSC_ERR_ARG_WRONGSTATE, "Cannot change collocation after IGASetUp()");
  g->collocation = c;
  return 0;
}
PetscErrorCode IGAGetUseCollocation(IGA g, PetscBool* flag) {
  if (PetscErrorCode e = check(g)) return e;
  if (!flag) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  *flag = g->collocation ? PETSC_TRUE : PETSC_FALSE;
  return 0;
}
PetscErrorCode IGASetMatType(IGA g, const char* t) {
  if (PetscErrorCode e = check(g)) return e;
  if (!t || (strcmp(t, "aij") && strcmp(t, "baij"))) return fail(PETSC_ERR_SUP, "device path assembles MATAIJ and MATBAIJ only");
  g->mattype = t;
  return 0;
}

PetscErrorCode IGAAxisSetPeriodic(IGAAxis ax, PetscBool periodic) { if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis"); ax->periodic = periodic ? 1 : 0; return 0; }
PetscErrorCode IGAAxisSetDegree(IGAAxis ax, PetscInt p) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (p < 1) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Polynomial degree must be greater than zero");
  ax->p = p;
  return 0;
}
PetscErrorCode IGAAxisSetKnots(IGAAxis ax, PetscInt m, const PetscReal U[]) {
  if (!ax || !U) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (ax->p < 1) return fail(PETSC_ERR_ORDER, "Must call IGAAxisSetDegree() first");
  if (m < 2 * ax->p + 1) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of knots must be at least 2*(p+1)");
  for (int k = 1; k <= m; k++) if (U[k - 1] > U[k]) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Knot sequence must be non-decreasing");
  ax->m = m;
  ax->U.assign(U, U + m + 1);
  axis_finish(ax);
  return 0;
}
// src/petigaaxis.c:323-382: open knot vector through the given breaks, each interior break repeated p-C times
PetscErrorCode IGAAxisInitBreaks(IGAAxis ax, PetscInt nu, const PetscReal u[], PetscInt C) {
  if (!ax || !u) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (C == PETSC_DECIDE) C = ax->p - 1;
  if (ax->p < 1) return fail(PETSC_ERR_ORDER, "Must call IGAAxisSetDegree() first");
  if (nu < 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of breaks must be at least two");
  for (int i = 1; i < nu; i++) if (u[i - 1] >= u[i]) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Break sequence must be strictly increasing");
  if (C < 0 || C >= ax->p) return fail(PETSC_ERR_ARG_WRONG, "Continuity must be in range [0,p-1]");
  const int p = ax->p, s = p - C, r = nu - 1, m = 2 * (p + 1) + (r - 1) * s - 1, n = m - p - 1;
  ax->m = m;
  ax->U.assign(m + 1, 0.0);
  double* U = ax->U.data();
  int k = 0;
  for (; k <= p; k++) { U[k] = u[0]; U[m - k] = u[r]; }
  for (int i = 1; i <= r - 1; i++)
    for (int j = 0; j < s; j++) U[k++] = u[i];
  if (ax->periodic)
    for (k = 0; k <= C; k++) { U[C - k] = U[p] - U[m - p] + U[n - k]; U[m - C + k] = U[m - p] - U[p] + U[p + 1 + k]; }
  ax->nel = r;
  ax->span.resize(r);
  for (int i = 0; i < r; i++) ax->span[i] = p + i * s;
  ax->nnp = ax->periodic ? n - C : n + 1;
  return 0;
}
// getters: src/petigaaxis.c:155-310
PetscErrorCode IGAAxisGetPeriodic(IGAAxis ax, PetscBool* periodic) { if (!ax || !periodic) return fail(PETSC_ERR_ARG_NULL, "Null pointer"); *periodic = ax->periodic ? PETSC_TRUE : PETSC_FALSE; return 0; }
PetscErrorCode IGAAxisGetDegree(IGAAxis ax, PetscInt* p) { if (!ax || !p) return fail(PETSC_ERR_ARG_NULL, "Null pointer"); *p = ax->p; return 0; }
PetscErrorCode IGAAxisGetKnots(IGAAxis ax, PetscInt* m, PetscReal* U[]) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (m) *m = ax->m;
  if (U) *U = ax->U.data();
  return 0;
}
PetscErrorCode IGAAxisGetLimits(IGAAxis ax, PetscReal* Ui, PetscReal* Uf) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (Ui) *Ui = ax->U[ax->p];
  if (Uf) *Uf = ax->U[ax->m - ax->p];
  return 0;
}
PetscErrorCode IGAAxisGetSpans(IGAAxis ax, PetscInt* nel, PetscInt* span[]) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (nel) *nel = ax->nel;
  if (span) *span = ax->span.data();
  return 0;
}

PetscErrorCode IGAAxisInitUniform(IGAAxis ax, PetscInt N, PetscReal Ui, PetscReal Uf, PetscInt C) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (C == PETSC_DECIDE) C = ax->p - 1;
  if (ax->p < 1) return fail(PETSC_ERR_ORDER, "Must call IGAAxisSetDegree() first");
  if (N < 1) return fail(PETSC_ERR_ARG_WRONG, "Number of elements must be greater than zero");
  if (Ui >= Uf) return fail(PETSC_ERR_ARG_WRONG, "Initial value must be less than final value");
  if (C < 0 || C >= ax->p) return fail(PETSC_ERR_ARG_WRONG, "Continuity must be in range [0,p-1]");
  const int p = ax->p, s = p - C, m = 2 * (p + 1) + (N - 1) * s - 1, n = m - p - 1;
  ax->m = m;
  ax->U.assign(m + 1, 0.0);
  double* U = ax->U.data();
  int k = 0;
  for (; k <= p; k++) { U[k] = Ui; U[m - k] = Uf; }
  for (int i = 1; i <= N - 1; i++)
    for (int j = 1; j <= s; j++) U[k++] = Ui + (PetscReal)i / (PetscReal)N * (Uf - Ui);   // operation order of petigaaxis.c:439
  if (ax->periodic)
    for (k = 0; k <= C; k++) { U[C - k] = U[p] - U[m - p] + U[n - k]; U[m - C + k] = U[m - p] - U[p] + U[p + 1 + k]; }
  ax->nel = N;
  ax->span.resize(N);
  for (int i = 0; i < N; i++) ax->span[i] = p + i * s;
  ax->nnp = ax->periodic ? n - C : n + 1;
  return 0;
}
PetscErrorCode IGAAxisGetSizes(IGAAxis ax, PetscInt* nel, PetscInt* nnp) {
  if (!ax) return fail(PETSC_ERR_ARG_NULL, "Null axis");
  if (nel) *nel = ax->nel;
  if (nnp) *nnp = ax->nnp;
  return 0;
}

PetscErrorCode IGASetUp(IGA g) {
  if (PetscErrorCode e = check(g)) return e;
  if (g->setup) return 0;
  if (g->dim < 1) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetDim() first");
  if (g->dof < 1) g->dof = 1;
  for (int d = 0; d < g->dim; d++) {
    if (g->axis[d].p < 1) return fail(PETSC_ERR_ORDER, "Must call IGAAxisSetDegree() first");
    if (g->axis[d].m < 2 * g->axis[d].p + 1) return fail(PETSC_ERR_ORDER, "Must call IGAAxisSetKnots() first");
  }
  for (int d = g->dim; d < 3; d++) { g->axis[d] = _n_IGAAxis(); g->axis[d].owner = g; }   // IGAAxisReset
  if (g->order < 0) {
    int o = 0;
    for (int d = 0; d < g->dim; d++) o = std::max(o, g->axis[d].p);
    g->order = o < 1 ? 1 : (o > 4 ? 4 : o);
  }
  // Stage 1: processor grid and boxes
  int N[3] = {1, 1, 1}, n[3], c[3] = {0, 0, 0};
  for (int d = 0; d < g->dim; d++) N[d] = g->axis[d].nel;
  for (int d = 0; d < 3; d++) n[d] = d < g->dim ? g->proc_user[d] : 1;
  if (PetscErrorCode e = IGA_Partition(g->comm.size, g->comm.rank, g->dim, N, n, c)) return e;
  for (int d = 0; d < 3; d++) {
    const _n_IGAAxis& ax = g->axis[d];
    const int P = d < g->dim ? n[d] : 1, r = d < g->dim ? c[d] : 0, nel = ax.nel, p = ax.p;
    g->proc_sizes[d] = P; g->proc_ranks[d] = r;
    const int ew = nel / P + ((nel % P) > r), es = r * (nel / P) + (((nel % P) > r) ? r : (nel % P));
    const int efirst = es, elast = es + ew - 1;
    const int gstart = ax.span[efirst] - p, gend = ax.span[elast] + 1, lstart = gstart;
    const int lend = (elast < nel - 1) ? ax.span[elast + 1] - p : ax.span[elast] + 1;
    g->elem_start[d] = es; g->elem_width[d] = ew;
    g->node_lstart[d] = lstart; g->node_lwidth[d] = (r == P - 1) ? ax.nnp - lstart : lend - lstart;
    g->node_gstart[d] = gstart; g->node_gwidth[d] = gend - gstart;
    g->geom_sizes[d] = ax.span[nel - 1] + 1;
  }
  // Stage 3: rule + 1-D tables
  for (int d = 0; d < 3 && g->collocation; d++) {   // collocation: one point per basis function, its Greville abscissa
    const _n_IGAAxis& ax = g->axis[d];
    const int p = ax.p, nnp = ax.nnp, nen = p + 1, n = ax.m - p - 1, nd = std::min(p, 4);
    if (p > 8) return fail(PETSC_ERR_SUP, "degree > 8");
    g->nqp[d] = 1;
    g->offset[d].assign(nnp, 0); g->detJac[d].assign(nnp, 1.0);
    g->weight[d].assign(nnp, 1.0); g->point[d].assign(nnp, 0.0);
    g->value[d].assign((size_t)nnp * nen * 5, 0.0);
    for (int i = 0; i < nnp; i++) {
      double u = 0.0;
      if (p > 0) {
        for (int j = 1; j <= p; j++) u += ax.U[i + j];
        u /= p;
      }
      int k = n;   // FindSpan (The NURBS Book A2.1): the largest k with U[k] <= u < U[k+1]; k = n at the right end
      if (u < ax.U[n + 1]) { k = p; while (k < n && ax.U[k + 1] <= u) k++; }
      g->offset[d][i] = k - p;
      g->point[d][i] = u;
      double ders[9][5];
      bspline_ders(k, u, p, nd, ax.U.data(), ders);
      for (int a = 0; a < nen; a++) for (int dd = 0; dd < 5; dd++) g->value[d][((size_t)i * nen + a) * 5 + dd] = ders[a][dd];
    }
    // element box = owned node box; ghost box = union of the owned rows' stencils [offset, offset + p]
    g->elem_start[d] = g->node_lstart[d]; g->elem_width[d] = g->node_lwidth[d];
    const int lo = g->offset[d][g->node_lstart[d]], hi = g->offset[d][g->node_lstart[d] + g->node_lwidth[d] - 1] + p + 1;
    g->node_gstart[d] = lo; g->node_gwidth[d] = hi - lo;
  }
  for (int d = 0; d < 3 && !g->collocation; d++) {
    const _n_IGAAxis& ax = g->axis[d];
    const int p = ax.p, nel = ax.nel, nen = p + 1, nd = std::min(p, 4);
    int q = (d < g->dim) ? g->rule_nqp[d] : 0;
    if (q < 1) q = p + 1;
    if (q > 10) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of quadrature points not implemented");
    if (p > 8) return fail(PETSC_ERR_SUP, "degree > 8");
    g->nqp[d] = q;
    g->offset[d].assign(nel, 0); g->detJac[d].assign(nel, 0.0);
    g->weight[d].assign((size_t)nel * q, 0.0); g->point[d].assign((size_t)nel * q, 0.0);
    g->value[d].assign((size_t)nel * q * nen * 5, 0.0);
    for (int e = 0; e < nel; e++) {
      const int k = ax.span[e];
      const double u0 = ax.U[k], u1 = ax.U[k + 1], J = (u1 - u0) / 2;
      g->offset[d][e] = k - p;
      g->detJac[d][e] = J;
      for (int iq = 0; iq < q; iq++) {
        const double u = (GAUSS_X[q][iq] + 1) * J + u0;
        g->weight[d][(size_t)e * q + iq] = GAUSS_W[q][iq];
        g->point[d][(size_t)e * q + iq] = u;
        double ders[9][5];
        bspline_ders(k, u, p, nd, ax.U.data(), ders);
        for (int a = 0; a < nen; a++) for (int dd = 0; dd < 5; dd++) g->value[d][(((size_t)e * q + iq) * nen + a) * 5 + dd] = ders[a][dd];
      }
    }
  }
  for (int d = 0; d < 3; d++) {   // boundary tables: k0 = p, u0 = U[k0]; k1 = n, u1 = U[k1+1] (src/petigabasis.c:208-217)
    const _n_IGAAxis& ax = g->axis[d];
    const int p = ax.p, n = ax.m - p - 1, nd = std::min(p, 4);
    const int kb[2] = {p, n};
    const double ub[2] = {ax.U[p], ax.U[n + 1]};
    for (int s = 0; s < 2; s++) {
      double ders[9][5];
      memset(ders, 0, sizeof(ders));
      bspline_ders(kb[s], ub[s], p, nd, ax.U.data(), ders);
      g->bnd_value[d][s].assign((size_t)(p + 1) * 5, 0.0);
      for (int a = 0; a <= p; a++) for (int dd = 0; dd < 5; dd++) g->bnd_value[d][s][(size_t)a * 5 + dd] = ders[a][dd];
      g->bnd_point[d][s] = ub[s];
    }
  }
  if (g->layout) { petiga_layout_destroy(g->layout); g->layout = nullptr; }
  petiga_cuda_space sp;
  fill_space(g, sp);
  int rc = petiga_layout_create(&g->layout, &sp, g->comm.rank, g->comm.size);
  if (rc) return from_cuda(rc);
  if (g->nsd) {
    size_t need = (size_t)g->geom_sizes[0] * g->geom_sizes[1] * g->geom_sizes[2];
    if (g->geomX.size() != need * g->nsd) return fail(PETSC_ERR_ARG_WRONGSTATE, "geometry array size does not match the knot vectors");
  }
  g->setup = 1;
  return 0;
}

PetscErrorCode IGASetGeometryArrays(IGA g, PetscInt nsd, const PetscReal* X, const PetscReal* W) {
  if (PetscErrorCode e = check(g)) return e;
  if (!X) { g->nsd = 0; g->geomX.clear(); g->geomW.clear(); g->rational = false; g->geom_dirty = true; return 0; }
  if (g->dim < 1) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetDim() first");
  size_t n = 1;
  for (int d = 0; d < g->dim; d++) n *= (size_t)(g->axis[d].m - g->axis[d].p);
  g->nsd = nsd;
  g->geomX.assign(X, X + n * nsd);
  g->rational = false;
  g->geomW.clear();
  g->geomW_all.clear();
  if (W) g->geomW_all.assign(W, W + n);
  if (W) {
    double lo = W[0], hi = W[0];
    for (size_t k = 0; k < n; k++) { lo = std::min(lo, W[k]); hi = std::max(hi, W[k]); }
    g->rational = std::fabs(hi - lo) > 100 * 2.220446049250313e-16;   // src/petigaio.c:251-253
    if (g->rational) g->geomW.assign(W, W + n);
  }
  g->geom_dirty = true;
  return 0;
}

static PetscErrorCode set_bc_entry(IGA g, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value, bool load) {
  if (PetscErrorCode e = check(g)) return e;
  if (axis < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "axis must be nonnegative");
  if (axis >= 3) return fail(PETSC_ERR_ARG_OUTOFRANGE, "axis must be less than 3");
  if (side < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "side must be nonnegative");
  if (side >= 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "side must be less than 2");
  if (field < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "field must be nonnegative");
  if (field >= 64) return fail(PETSC_ERR_ARG_OUTOFRANGE, "field must be less than 64");
  int* cnt = load ? &g->bc.lcount[axis][side] : &g->bc.vcount[axis][side];
  int* fld = load ? g->bc.lfield[axis][side] : g->bc.vfield[axis][side];
  double* val = load ? g->bc.lvalue[axis][side] : g->bc.vvalue[axis][side];
  int k = 0;
  for (; k < *cnt; k++) if (fld[k] == field) break;   // IGAFormBCSetEntry: src/petigaform.c:102-110
  if (k == *cnt) (*cnt)++;
  fld[k] = field; val[k] = value;
  g->bc_dirty = true;
  return 0;
}
PetscErrorCode IGASetBoundaryValue(IGA g, PetscInt a, PetscInt s, PetscInt f, PetscScalar v) { return set_bc_entry(g, a, s, f, v, false); }
PetscErrorCode IGASetBoundaryLoad(IGA g, PetscInt a, PetscInt s, PetscInt f, PetscScalar v) { return set_bc_entry(g, a, s, f, v, true); }
// IGAForm object API (include/petiga.h:270-289, src/petigaform.c): in the mirror the form lives inside the IGA, so the handle
// is the IGA itself behind an opaque type; every function forwards to the IGASet* entry of the same meaning
static inline IGA form_iga(IGAForm f) { return reinterpret_cast<IGA>(f); }
PetscErrorCode IGAGetForm(IGA g, IGAForm* form) {
  if (PetscErrorCode e = check(g)) return e;
  if (!form) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  *form = reinterpret_cast<IGAForm>(g);
  return 0;
}
PetscErrorCode IGAFormSetBoundaryValue(IGAForm f, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value) { return IGASetBoundaryValue(form_iga(f), axis, side, field, value); }
PetscErrorCode IGAFormSetBoundaryLoad(IGAForm f, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value) { return IGASetBoundaryLoad(form_iga(f), axis, side, field, value); }
PetscErrorCode IGAFormSetBoundaryForm(IGAForm f, PetscInt axis, PetscInt side, PetscBool flag) { return IGASetBoundaryForm(form_iga(f), axis, side, flag); }
PetscErrorCode IGAFormClearBoundary(IGAForm f, PetscInt axis, PetscInt side) {   // src/petigaform.c: value/load counts and the visit flag of one face
  IGA g = form_iga(f);
  if (PetscErrorCode e = check(g)) return e;
  if (axis < 0 || axis >= 3 || side < 0 || side >= 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "axis/side out of range");
  g->bc.vcount[axis][side] = 0; g->bc.lcount[axis][side] = 0; g->visit[axis][side] = 0;
  g->bc_dirty = true;
  if (g->plan) return from_cuda(petiga_cuda_set_boundary_form(g->plan, axis, side, 0));
  return 0;
}
PetscErrorCode IGAFormSetVector(IGAForm f, IGAFormVector fn, void* ctx) { return IGASetFormVector(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetMatrix(IGAForm f, IGAFormMatrix fn, void* ctx) { return IGASetFormMatrix(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetSystem(IGAForm f, IGAFormSystem fn, void* ctx) { return IGASetFormSystem(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetFunction(IGAForm f, IGAFormFunction fn, void* ctx) { return IGASetFormFunction(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetJacobian(IGAForm f, IGAFormJacobian fn, void* ctx) { return IGASetFormJacobian(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetIFunction(IGAForm f, IGAFormIFunction fn, void* ctx) { return IGASetFormIFunction(form_iga(f), fn, ctx); }
PetscErrorCode IGAFormSetIJacobian(IGAForm f, IGAFormIJacobian fn, void* ctx) { return IGASetFormIJacobian(form_iga(f), fn, ctx); }

// include/petiga.h:300, src/petigaform.c IGAFormSetBoundaryForm
PetscErrorCode IGASetBoundaryForm(IGA g, PetscInt axis, PetscInt side, PetscBool flag) {
  if (PetscErrorCode e = check(g)) return e;
  if (axis < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "axis must be nonnegative");
  if (axis >= 3) return fail(PETSC_ERR_ARG_OUTOFRANGE, "axis must be less than 3");
  if (side < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "side must be nonnegative");
  if (side >= 2) return fail(PETSC_ERR_ARG_OUTOFRANGE, "side must be less than 2");
  g->visit[axis][side] = flag ? 1 : 0;
  if (g->plan) return from_cuda(petiga_cuda_set_boundary_form(g->plan, axis, side, g->visit[axis][side]));
  return 0;
}
PetscErrorCode IGASetFixTable(IGA g, Vec table) { if (PetscErrorCode e = check(g)) return e; g->fixtable = table; g->bc_dirty = true; return 0; }

PetscErrorCode IGASetFormVector(IGA g, IGAFormVector f, void* ctx) { return set_form(g, PETIGA_SLOT_VECTOR, (const void*)f, ctx); }
PetscErrorCode IGASetFormMatrix(IGA g, IGAFormMatrix f, void* ctx) { return set_form(g, PETIGA_SLOT_MATRIX, (const void*)f, ctx); }
PetscErrorCode IGASetFormSystem(IGA g, IGAFormSystem f, void* ctx) { return set_form(g, PETIGA_SLOT_SYSTEM, (const void*)f, ctx); }
PetscErrorCode IGASetFormFunction(IGA g, IGAFormFunction f, void* ctx) { return set_form(g, PETIGA_SLOT_FUNCTION, (const void*)f, ctx); }
PetscErrorCode IGASetFormJacobian(IGA g, IGAFormJacobian f, void* ctx) { return set_form(g, PETIGA_SLOT_JACOBIAN, (const void*)f, ctx); }
PetscErrorCode IGASetFormIFunction(IGA g, IGAFormIFunction f, void* ctx) { return set_form(g, PETIGA_SLOT_IFUNCTION, (const void*)f, ctx); }
PetscErrorCode IGASetFormIJacobian(IGA g, IGAFormIJacobian f, void* ctx) { return set_form(g, PETIGA_SLOT_IJACOBIAN, (const void*)f, ctx); }

PetscErrorCode IGASetFormI2Function(IGA g, IGAFormI2Function f, void* ctx) { return set_form(g, PETIGA_SLOT_I2FUNCTION, (const void*)f, ctx); }
PetscErrorCode IGASetFormI2Jacobian(IGA g, IGAFormI2Jacobian f, void* ctx) { return set_form(g, PETIGA_SLOT_I2JACOBIAN, (const void*)f, ctx); }
PetscErrorCode IGASetFormIEFunction(IGA g, IGAFormIEFunction f, void* ctx) { return set_form(g, PETIGA_SLOT_IEFUNCTION, (const void*)f, ctx); }
PetscErrorCode IGASetFormIEJacobian(IGA g, IGAFormIEJacobian f, void* ctx) { return set_form(g, PETIGA_SLOT_IEJACOBIAN, (const void*)f, ctx); }
PetscErrorCode IGASetFormRHSFunction(IGA g, IGAFormRHSFunction f, void* ctx) { return set_form(g, PETIGA_SLOT_RHSFUNCTION, (const void*)f, ctx); }
PetscErrorCode IGASetFormRHSJacobian(IGA g, IGAFormRHSJacobian f, void* ctx) { return set_form(g, PETIGA_SLOT_RHSJACOBIAN, (const void*)f, ctx); }

PetscErrorCode IGACreateMat(IGA g, Mat* mat) {
  if (PetscErrorCode e = check(g)) return e;
  if (!mat) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (PetscErrorCode e = ensure_plan(g)) return e;
  const bool baij = g->mattype.empty() ? (g->dof > 1) : (g->mattype == "baij");   // src/petiga.c:1326-1330
  Mat A = new _p_Mat();
  A->iga = g; A->baij = baij; A->bs = g->dof; A->gen = g->plan_gen;
  int nrows; int64_t nnz;
  int rc = petiga_cuda_plan_pattern(g->plan, baij ? 1 : 0, &nrows, &nnz, &A->d_rowptr, &A->d_colidx);
  if (rc) { delete A; return from_cuda(rc); }
  A->nrows = nrows; A->nnz = nnz;
  int nown, ng; int64_t nnzb;
  petiga_cuda_plan_sizes(g->plan, &nown, &ng, &nnzb);
  const size_t nval = (size_t)nnzb * g->dof * g->dof;
  petiga_cuda_plan_activate(g->plan);   // allocate on the plan's device, not on whichever is current
  rc = petiga_cuda_malloc((void**)&A->d_values, nval * sizeof(double));
  if (rc) { delete A; return from_cuda(rc); }
  *mat = A;
  return 0;
}
PetscErrorCode MatDestroy(Mat* mat) { if (mat && *mat) { petiga_cuda_free((*mat)->d_values); delete *mat; *mat = nullptr; } return 0; }
PetscErrorCode IGACreateVec(IGA g, Vec* vec) {
  if (PetscErrorCode e = check(g)) return e;
  if (!vec) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (PetscErrorCode e = ensure_plan(g)) return e;
  int nown, ng; int64_t nnzb;
  petiga_cuda_plan_sizes(g->plan, &nown, &ng, &nnzb);
  Vec v = new _p_Vec();
  v->iga = g; v->n = nown * g->dof; v->gen = g->plan_gen;
  petiga_cuda_plan_activate(g->plan);
  int rc = petiga_cuda_malloc((void**)&v->d, (size_t)v->n * sizeof(double));
  if (rc) { delete v; return from_cuda(rc); }
  std::vector<double> z(v->n, 0.0);
  petiga_cuda_memcpy_h2d(v->d, z.data(), z.size() * sizeof(double));
  *vec = v;
  return 0;
}
PetscErrorCode VecDestroy(Vec* vec) { if (vec && *vec) { petiga_cuda_free((*vec)->d); delete *vec; *vec = nullptr; } return 0; }
PetscErrorCode MatGetSizesIGA(Mat A, PetscInt* nrows, int64_t* nnz, PetscInt* bs, PetscBool* baij) {
  if (!A) return fail(PETSC_ERR_ARG_NULL, "Null Mat");
  if (nrows) *nrows = A->iga->dof * (A->baij ? A->nrows : A->nrows / A->iga->dof);
  if (nnz) *nnz = A->nnz;
  if (bs) *bs = A->bs;
  if (baij) *baij = A->baij;
  return 0;
}
PetscErrorCode MatGetCSRHost(Mat A, PetscInt* rowptr, PetscInt* colidx, PetscScalar* values) {
  if (!A) return fail(PETSC_ERR_ARG_NULL, "Null Mat");
  if (PetscErrorCode e = check_owner(A, nullptr, "Mat")) return e;
  int rc = A->iga->plan ? petiga_cuda_finish(A->iga->plan) : 0;
  if (rc) return from_cuda(rc);
  if (A->iga->plan) petiga_cuda_plan_activate(A->iga->plan);
  if (rowptr) rc = petiga_cuda_memcpy_d2h(rowptr, A->d_rowptr, ((size_t)A->nrows + 1) * sizeof(int));
  if (!rc && colidx) rc = petiga_cuda_memcpy_d2h(colidx, A->d_colidx, (size_t)A->nnz * sizeof(int));
  if (!rc && values) {
    const size_t nval = A->baij ? (size_t)A->nnz * A->bs * A->bs : (size_t)A->nnz;
    rc = petiga_cuda_memcpy_d2h(values, A->d_values, nval * sizeof(double));
  }
  return from_cuda(rc);
}
PetscErrorCode MatGetValuesDevice(Mat A, PetscScalar** d) { if (!A || !d) return fail(PETSC_ERR_ARG_NULL, "Null"); *d = A->d_values; return 0; }
PetscErrorCode VecGetLocalSize(Vec v, PetscInt* n) { if (!v || !n) return fail(PETSC_ERR_ARG_NULL, "Null"); *n = v->n; return 0; }
PetscErrorCode VecGetArrayHost(Vec v, PetscScalar* out) { if (!v || !out) return fail(PETSC_ERR_ARG_NULL, "Null"); if (PetscErrorCode e = check_owner(v, nullptr, "Vec")) return e; if (v->iga->plan) { petiga_cuda_finish(v->iga->plan); petiga_cuda_plan_activate(v->iga->plan); } return from_cuda(petiga_cuda_memcpy_d2h(out, v->d, (size_t)v->n * sizeof(double))); }
PetscErrorCode VecSetArrayHost(Vec v, const PetscScalar* in) { if (!v || !in) return fail(PETSC_ERR_ARG_NULL, "Null"); if (PetscErrorCode e = check_owner(v, nullptr, "Vec")) return e; if (v->iga->plan) petiga_cuda_plan_activate(v->iga->plan); return from_cuda(petiga_cuda_memcpy_h2d(v->d, in, (size_t)v->n * sizeof(double))); }
PetscErrorCode VecGetArrayDevice(Vec v, PetscScalar** d) { if (!v || !d) return fail(PETSC_ERR_ARG_NULL, "Null"); *d = v->d; return 0; }

// what the collocation kernel supports, checked before any device work (the library repeats the checks for direct callers)
static PetscErrorCode check_collocation(IGA g, int slot) {
  const int f = g->slots[slot].form;
  const bool cform = f == PETIGA_FORM_LAPLACE_COLLOCATION || f == PETIGA_FORM_CONVTEST_COLLOCATION;
  if (!g->collocation) {
    if (cform) return fail(PETSC_ERR_SUP, "a collocation form needs IGASetUseCollocation(iga, PETSC_TRUE)");
    return 0;
  }
  if (slot != PETIGA_SLOT_VECTOR && slot != PETIGA_SLOT_MATRIX && slot != PETIGA_SLOT_SYSTEM)
    return fail(PETSC_ERR_SUP, "collocation: only IGAComputeVector/Matrix/System run on the device");
  if (!cform) return fail(PETSC_ERR_SUP, "collocation: pass one of the IGADeviceForm_*Collocation sentinels (Galerkin forms integrate)");
  if (g->dof != 1) return fail(PETSC_ERR_SUP, "collocation: the device forms have dof 1");
  for (int d = 0; d < g->dim; d++)
    for (int s = 0; s < 2; s++) {
      if (g->bc.lcount[d][s]) return fail(PETSC_ERR_SUP, "collocation: IGASetBoundaryLoad is not supported");
      if (g->visit[d][s]) return fail(PETSC_ERR_SUP, "collocation: IGASetBoundaryForm is not supported");
    }
  if (g->fixtable) return fail(PETSC_ERR_SUP, "collocation: IGASetFixTable is not supported");
  for (auto& o : g->options)
    if (o.first == "path" && (int)o.second == PETIGA_PATH_KRONECKER) return fail(PETSC_ERR_SUP, "collocation: the separable path does not apply");
  return 0;
}

static PetscErrorCode run(IGA g, int slot, PetscReal a, Vec V, PetscReal t, Vec U, Mat A, Vec B, PetscReal a2 = 0, Vec W = nullptr, PetscReal t0 = 0) {
  if (PetscErrorCode e = check(g)) return e;
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");                     // IGACheckSetUp
  if (g->slots[slot].form < 0) return fail(PETSC_ERR_USER, "Must call IGASetForm*() first");
  if (PetscErrorCode e = check_collocation(g, slot)) return e;
  if (PetscErrorCode e = ensure_plan(g)) return e;
  if (A) if (PetscErrorCode e = check_owner(A, g, "Mat")) return e;
  for (Vec x : {V, U, B, W}) if (x) if (PetscErrorCode e = check_owner(x, g, "Vec")) return e;
  int rc = petiga_cuda_compute_ext(g->plan, slot, A ? A->baij : 0, a, V ? V->d : nullptr, t, U ? U->d : nullptr, a2, W ? W->d : nullptr, t0,
                                   A ? A->d_values : nullptr, B ? B->d : nullptr);
  if (rc) return from_cuda(rc);
  if (g->async) return 0;                          // device-resident hand-off: ordered on the IGA's stream, no host wait
  return from_cuda(petiga_cuda_finish(g->plan));   // Mat/VecAssemblyEnd: fully assembled on return
}
PetscErrorCode IGASynchronize(IGA g) {
  if (PetscErrorCode e = check(g)) return e;
  return g->plan ? from_cuda(petiga_cuda_finish(g->plan)) : 0;
}

// ---- the step after the path: MatMult and a KSP that stays on the device (src/petiga.c:856-885 IGACreateKSP; demo/Poisson3D.c:73-83) ----
PetscErrorCode MatMult(Mat A, Vec x, Vec y) {
  if (!A || !x || !y) return fail(PETSC_ERR_ARG_NULL, "Null Mat/Vec");
  if (PetscErrorCode e = check_owner(A, nullptr, "Mat")) return e;
  if (PetscErrorCode e = check_owner(x, A->iga, "Vec")) return e;
  if (PetscErrorCode e = check_owner(y, A->iga, "Vec")) return e;
  if (x == y) return fail(PETSC_ERR_ARG_IDN, "x and y must be different vectors");
  IGA g = A->iga;
  if (int rc = petiga_cuda_spmv(g->plan, A->baij, A->d_values, x->d, y->d)) return from_cuda(rc);
  return g->async ? 0 : from_cuda(petiga_cuda_finish(g->plan));
}
PetscErrorCode IGACreateKSP(IGA g, KSP* ksp) {
  if (PetscErrorCode e = check(g)) return e;
  if (!ksp) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  *ksp = new _p_KSP{g, nullptr, 1e-5, 1e-50, 10000, 0, 0.0};      // PETSc's default tolerances (KSPSetTolerances man page)
  return 0;
}
PetscErrorCode KSPSetOperators(KSP ksp, Mat A, Mat P) {
  if (!ksp || !A) return fail(PETSC_ERR_ARG_NULL, "Null KSP/Mat");
  if (P && P != A) return fail(PETSC_ERR_SUP, "KSPSetOperators: the preconditioner is the Jacobi diagonal of A; pass P = A");
  if (PetscErrorCode e = check_owner(A, ksp->iga, "Mat")) return e;
  ksp->A = A;
  return 0;
}
PetscErrorCode KSPSetTolerances(KSP ksp, PetscReal rtol, PetscReal abstol, PetscReal dtol, PetscInt maxits) {
  (void)dtol;
  if (!ksp) return fail(PETSC_ERR_ARG_NULL, "Null KSP");
  if (rtol < 0 || abstol < 0 || maxits < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Tolerances and iteration count must be nonnegative");
  ksp->rtol = rtol; ksp->abstol = abstol; ksp->maxits = maxits;
  return 0;
}
PetscErrorCode KSPSolve(KSP ksp, Vec b, Vec x) {
  if (!ksp || !b || !x) return fail(PETSC_ERR_ARG_NULL, "Null KSP/Vec");
  if (!ksp->A) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call KSPSetOperators() first");
  if (PetscErrorCode e = check_owner(ksp->A, ksp->iga, "Mat")) return e;
  if (PetscErrorCode e = check_owner(b, ksp->iga, "Vec")) return e;
  if (PetscErrorCode e = check_owner(x, ksp->iga, "Vec")) return e;
  if (b == x) return fail(PETSC_ERR_ARG_IDN, "b and x must be different vectors");
  IGA g = ksp->iga;
  // KSPSolve starts from x = 0 unless KSPSetInitialGuessNonzero was called (not mirrored)
  ksp->reason = KSP_CONVERGED_ITERATING;
  if (ksp->gmres) {
    if (int rc = petiga_cuda_memset_async(g->plan, x->d, 0, (size_t)x->n * sizeof(double))) return from_cuda(rc);
    int reason = 0;
    if (int rc = petiga_cuda_solve_gmres(g->plan, ksp->A->baij, ksp->A->d_values, b->d, x->d, ksp->restart, ksp->rtol, ksp->abstol, ksp->maxits,
                                         &ksp->its, &ksp->rnorm, &reason)) return from_cuda(rc);
    ksp->reason = (KSPConvergedReason)reason;
    return 0;
  }
  if (int rc = petiga_cuda_memset(x->d, 0, (size_t)x->n * sizeof(double))) return from_cuda(rc);
  if (int rc = petiga_cuda_solve_cg(g->plan, ksp->A->baij, ksp->A->d_values, b->d, x->d, ksp->rtol, ksp->abstol, ksp->maxits, &ksp->its, &ksp->rnorm))
    return from_cuda(rc);
  ksp->reason = ksp->rnorm <= ksp->rtol ? KSP_CONVERGED_RTOL : ksp->its < ksp->maxits ? KSP_CONVERGED_ATOL : KSP_DIVERGED_ITS;
  return 0;
}
PetscErrorCode KSPSetType(KSP ksp, KSPType type) {
  if (!ksp || !type) return fail(PETSC_ERR_ARG_NULL, "Null KSP/KSPType");
  if (!strcmp(type, KSPCG)) ksp->gmres = false;
  else if (!strcmp(type, KSPGMRES)) ksp->gmres = true;
  else return fail(PETSC_ERR_SUP, std::string("KSPSetType: unsupported type \"") + type + "\" (the device provides \"cg\" and \"gmres\")");
  return 0;
}
PetscErrorCode KSPGMRESSetRestart(KSP ksp, PetscInt restart) {
  if (!ksp) return fail(PETSC_ERR_ARG_NULL, "Null KSP");
  if (restart < 1) return fail(PETSC_ERR_ARG_OUTOFRANGE, "KSPGMRESSetRestart: restart must be at least 1");
  ksp->restart = restart;
  return 0;
}
PetscErrorCode KSPGetConvergedReason(KSP ksp, KSPConvergedReason* reason) {
  if (!ksp || !reason) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  *reason = ksp->reason;
  return 0;
}
PetscErrorCode KSPGetIterationNumber(KSP ksp, PetscInt* its) { if (!ksp || !its) return fail(PETSC_ERR_ARG_NULL, "Null pointer"); *its = ksp->its; return 0; }
PetscErrorCode KSPGetResidualNorm(KSP ksp, PetscReal* rnorm) { if (!ksp || !rnorm) return fail(PETSC_ERR_ARG_NULL, "Null pointer"); *rnorm = ksp->rnorm; return 0; }
PetscErrorCode KSPDestroy(KSP* ksp) { if (ksp && *ksp) { delete *ksp; *ksp = nullptr; } return 0; }
PetscErrorCode IGAComputeVector(IGA g, Vec B) { if (!B) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_VECTOR, 0, nullptr, 0, nullptr, nullptr, B); }
PetscErrorCode IGAComputeMatrix(IGA g, Mat A) { if (!A) return fail(PETSC_ERR_ARG_NULL, "Null Mat"); return run(g, PETIGA_SLOT_MATRIX, 0, nullptr, 0, nullptr, A, nullptr); }
PetscErrorCode IGAComputeSystem(IGA g, Mat A, Vec B) { if (!A || !B) return fail(PETSC_ERR_ARG_NULL, "Null Mat/Vec"); return run(g, PETIGA_SLOT_SYSTEM, 0, nullptr, 0, nullptr, A, B); }
PetscErrorCode IGAComputeFunction(IGA g, Vec U, Vec F) { if (!U || !F) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_FUNCTION, 0, nullptr, 0, U, nullptr, F); }
PetscErrorCode IGAComputeJacobian(IGA g, Vec U, Mat J) { if (!U || !J) return fail(PETSC_ERR_ARG_NULL, "Null Vec/Mat"); return run(g, PETIGA_SLOT_JACOBIAN, 0, nullptr, 0, U, J, nullptr); }
PetscErrorCode IGAComputeIFunction(IGA g, PetscReal a, Vec V, PetscReal t, Vec U, Vec F) { if (!V || !U || !F) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_IFUNCTION, a, V, t, U, nullptr, F); }
PetscErrorCode IGAComputeIJacobian(IGA g, PetscReal a, Vec V, PetscReal t, Vec U, Mat J) { if (!V || !U || !J) return fail(PETSC_ERR_ARG_NULL, "Null Vec/Mat"); return run(g, PETIGA_SLOT_IJACOBIAN, a, V, t, U, J, nullptr); }

// src/petigats.c:182-477 and src/petigats2.c:23-175: same skeleton, a third vector (U0 / A) and a second time / shift
PetscErrorCode IGAComputeIEFunction(IGA g, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Vec F) { if (!V || !U || !U0 || !F) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_IEFUNCTION, a, V, t, U, nullptr, F, 0, U0, t0); }
PetscErrorCode IGAComputeIEJacobian(IGA g, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Mat J) { if (!V || !U || !U0 || !J) return fail(PETSC_ERR_ARG_NULL, "Null Vec/Mat"); return run(g, PETIGA_SLOT_IEJACOBIAN, a, V, t, U, J, nullptr, 0, U0, t0); }
PetscErrorCode IGAComputeRHSFunction(IGA g, PetscReal t, Vec U, Vec F) { if (!U || !F) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_RHSFUNCTION, 0, nullptr, t, U, nullptr, F); }
PetscErrorCode IGAComputeRHSJacobian(IGA g, PetscReal t, Vec U, Mat J) { if (!U || !J) return fail(PETSC_ERR_ARG_NULL, "Null Vec/Mat"); return run(g, PETIGA_SLOT_RHSJACOBIAN, 0, nullptr, t, U, J, nullptr); }
PetscErrorCode IGAComputeI2Function(IGA g, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Vec F) { if (!A || !V || !U || !F) return fail(PETSC_ERR_ARG_NULL, "Null Vec"); return run(g, PETIGA_SLOT_I2FUNCTION, a, V, t, U, nullptr, F, v, A, 0); }
PetscErrorCode IGAComputeI2Jacobian(IGA g, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Mat J) { if (!A || !V || !U || !J) return fail(PETSC_ERR_ARG_NULL, "Null Vec/Mat"); return run(g, PETIGA_SLOT_I2JACOBIAN, a, V, t, U, J, nullptr, v, A, 0); }

// src/petigacomp.c:35-96
PetscErrorCode IGAComputeScalar(IGA g, Vec vecU, PetscInt n, PetscScalar S[], IGAFormScalar Scalar, void* ctx) {
  if (PetscErrorCode e = check(g)) return e;
  if (!S) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  if (Scalar != IGADeviceScalar_CahnHilliard2D_Stats)
    return fail(PETSC_ERR_SUP, "IGAComputeScalar: host callbacks cannot run on the GPU; pass one of the IGADeviceScalar_* sentinels");
  if (!ctx) return fail(PETSC_ERR_ARG_NULL, "IGAComputeScalar: this functional needs its AppCtx");
  if (PetscErrorCode e = ensure_plan(g)) return e;
  return from_cuda(petiga_cuda_compute_scalar(g->plan, PETIGA_SCALAR_CH_STATS, (const double*)ctx, 3, vecU ? vecU->d : nullptr, n, S));
}
// src/petigacomp.c:155-186
PetscErrorCode IGAComputeErrorNorm(IGA g, PetscInt k, Vec vecU, IGAFormExact Exact, PetscReal enorm[], void* ctx) {
  if (PetscErrorCode e = check(g)) return e;
  if (!enorm) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  if (k < 0) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Derivative index must be nonnegative");   // :170
  double prm[3] = {(double)k, 0.0, 0.0};
  if (Exact == IGADeviceExact_ErrNormTest) prm[1] = 1;
  else if (Exact == IGADeviceExact_Neumann) prm[1] = 3;
  else if (Exact == IGADeviceExact_ConvTest) prm[1] = 4;
  else if (Exact == IGADeviceExact_L2Projection) { prm[1] = 2; if (!ctx) return fail(PETSC_ERR_ARG_NULL, "IGADeviceExact_L2Projection needs {choice}"); prm[2] = *(const double*)ctx; }
  else if (Exact) return fail(PETSC_ERR_SUP, "IGAComputeErrorNorm: host callbacks cannot run on the GPU; pass one of the IGADeviceExact_* sentinels or NULL");
  if (PetscErrorCode e = ensure_plan(g)) return e;
  double errsqr[8];
  if (g->dof > 8) return fail(PETSC_ERR_SUP, "IGAComputeErrorNorm: dof > 8");
  int rc = petiga_cuda_compute_scalar(g->plan, PETIGA_SCALAR_ERRNORM, prm, 3, vecU ? vecU->d : nullptr, g->dof, errsqr);
  if (rc) return from_cuda(rc);
  for (int i = 0; i < g->dof; i++) enorm[i] = sqrt(errsqr[i]);   // :180
  return 0;
}

PetscErrorCode IGAGetInfoArray(IGA g, PetscInt info[46]) {
  if (PetscErrorCode e = check(g)) return e;
  int k = 0;
  info[k++] = g->order;
  for (int d = 0; d < 3; d++) {   // nel: entries of the basis tables (nnp under collocation, as IGABasis.nel)
    info[k++] = g->axis[d].p; info[k++] = g->axis[d].m; info[k++] = g->axis[d].nnp; info[k++] = (g->collocation && g->setup) ? g->axis[d].nnp : g->axis[d].nel;
    info[k++] = g->nqp[d]; info[k++] = g->axis[d].p + 1; info[k++] = g->proc_sizes[d]; info[k++] = g->proc_ranks[d];
    info[k++] = g->elem_start[d]; info[k++] = g->elem_width[d]; info[k++] = g->node_lstart[d]; info[k++] = g->node_lwidth[d];
    info[k++] = g->node_gstart[d]; info[k++] = g->node_gwidth[d]; info[k++] = g->geom_sizes[d];
  }
  return 0;
}
PetscErrorCode IGAGetBasisTable(IGA g, PetscInt axis, PetscInt which, PetscReal* out) {
  if (PetscErrorCode e = check(g)) return e;
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  const std::vector<double>* src = nullptr;
  switch (which) {
    case 0: src = &g->value[axis]; break;
    case 1: src = &g->weight[axis]; break;
    case 2: src = &g->point[axis]; break;
    case 3: src = &g->detJac[axis]; break;
    case 4: src = &g->axis[axis].U; break;
    default: return fail(PETSC_ERR_ARG_OUTOFRANGE, "which");
  }
  memcpy(out, src->data(), src->size() * sizeof(double));
  return 0;
}
PetscErrorCode IGAGetLGMapHost(IGA g, PetscInt* lgmap) {
  if (PetscErrorCode e = check(g)) return e;
  if (!g->layout) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  return from_cuda(petiga_layout_lgmap(g->layout, lgmap));
}
PetscErrorCode IGASetOption(IGA g, const char* name, PetscReal value) {
  if (PetscErrorCode e = check(g)) return e;
  if (!strcmp(name, "async")) { g->async = value != 0; return 0; }
  for (auto& o : g->options) if (o.first == name) { o.second = value; goto done; }
  g->options.emplace_back(name, value);
done:
  if (g->plan) return from_cuda(petiga_cuda_set_option(g->plan, name, value));
  return 0;
}
PetscErrorCode IGAGetStat(IGA g, const char* name, PetscReal* value) {
  if (PetscErrorCode e = check(g)) return e;
  if (!g->plan) return fail(PETSC_ERR_ARG_WRONGSTATE, "no plan yet");
  return from_cuda(petiga_cuda_get_stat(g->plan, name, value));
}
PetscErrorCode IGAGetPlan(IGA g, void** plan) {
  if (PetscErrorCode e = check(g)) return e;
  if (PetscErrorCode e = ensure_plan(g)) return e;
  *plan = g->plan;
  return 0;
}
void* IGAGetLayout(IGA g) { return g ? g->layout : nullptr; }
PetscErrorCode IGASetStream(IGA g, void* stream) {
  if (PetscErrorCode e = check(g)) return e;
  if (g->plan) return fail(PETSC_ERR_ORDER, "IGASetStream must be called before the first IGACreateMat/Vec/Compute");
  g->stream = stream;
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// Geometry / vector files: the PETSc binary format the reference reads and writes (src/petigaio.c).  Everything is
// big-endian (PetscBinaryRead/Write swap on little-endian hosts): PetscInt = int32, PetscReal/PetscScalar = float64.
//   IGA file  (IGASave :75-139):  int IGA_FILE_CLASSID=1211299 | int info (bit0 geometry, bit1 property) | int dim |
//                                 per axis { int p, int m+1, real U[m+1] } | [ int nsd | Vec ] | [ int npd | Vec ]
//   Vec       (VecView binary):   int VEC_FILE_CLASSID=1211214 | int n | scalar[n]
//   geometry Vec (:288-369):      natural order (i fastest) over the geom_sizes grid, per control point
//                                 (w*x_0 .. w*x_{nsd-1}, w); IGALoadGeometry de-homogenises (:259-266)
// ---------------------------------------------------------------------------------------------------------------
namespace {
constexpr int kIGAFileClassId = 1211299, kVecFileClassId = 1211214;

struct BinFile {
  FILE* f = nullptr;
  ~BinFile() { if (f) fclose(f); }
  bool open(const char* name, const char* mode) { f = fopen(name, mode); return f != nullptr; }
  static uint32_t swap32(uint32_t v) { return __builtin_bswap32(v); }
  static uint64_t swap64(uint64_t v) { return __builtin_bswap64(v); }
  bool read_int(int* v) { uint32_t u; if (fread(&u, 4, 1, f) != 1) return false; u = swap32(u); memcpy(v, &u, 4); return true; }
  bool read_reals(double* v, size_t n) {
    if (fread(v, 8, n, f) != n) return false;
    for (size_t k = 0; k < n; k++) { uint64_t u; memcpy(&u, v + k, 8); u = swap64(u); memcpy(v + k, &u, 8); }
    return true;
  }
  bool write_int(int v) { uint32_t u; memcpy(&u, &v, 4); u = swap32(u); return fwrite(&u, 4, 1, f) == 1; }
  bool write_reals(const double* v, size_t n) {
    for (size_t k = 0; k < n; k++) { uint64_t u; memcpy(&u, v + k, 8); u = swap64(u); if (fwrite(&u, 8, 1, f) != 1) return false; }
    return true;
  }
};

void reset_iga(IGA g) {   // IGAReset (src/petiga.c) as far as the mirror holds state
  drop_plan(g);
  if (g->layout) { petiga_layout_destroy(g->layout); g->layout = nullptr; }
  g->setup = 0;
  g->nsd = 0; g->geomX.clear(); g->geomW.clear(); g->geomW_all.clear(); g->rational = false; g->geom_dirty = true;
  g->fixtable = nullptr; g->fixtable_local.clear(); g->bc.fixtableU = nullptr; g->bc_dirty = true;
}
}  // namespace

extern "C" {

// IGARead -> IGALoad (src/petigaio.c:535-569, :11-73)
PetscErrorCode IGARead(IGA g, const char filename[]) {
  if (PetscErrorCode e = check(g)) return e;
  if (!filename) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  BinFile bf;
  if (!bf.open(filename, "rb")) return fail(PETSC_ERR_FILE_OPEN, std::string("Cannot open file ") + filename);
  int classid = 0, info = 0, dim = 0;
  if (!bf.read_int(&classid)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
  if (classid != kIGAFileClassId) return fail(PETSC_ERR_ARG_WRONG, "Not an IGA in file");          // :32
  if (!bf.read_int(&info) || !bf.read_int(&dim)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
  const bool geometry = info & 0x1, property = info & 0x2;
  reset_iga(g);
  g->dim = -1;
  if (PetscErrorCode e = IGASetDim(g, dim)) return e;
  for (int i = 0; i < dim; i++) {
    int p = 0, m1 = 0;
    if (!bf.read_int(&p) || !bf.read_int(&m1) || m1 < 2 || m1 > (1 << 28)) return fail(PETSC_ERR_FILE_READ, "Bad axis record");
    std::vector<double> U((size_t)m1);
    if (!bf.read_reals(U.data(), U.size())) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
    IGAAxis ax = &g->axis[i];
    ax->periodic = 0;                                       // IGAAxisInit: degree + knots; files carry no periodicity
    ax->p = 0;
    if (PetscErrorCode e = IGAAxisSetDegree(ax, p)) return e;
    if (PetscErrorCode e = IGAAxisSetKnots(ax, m1 - 1, U.data())) return e;
  }
  for (int i = dim; i < 3; i++) { g->axis[i] = _n_IGAAxis(); g->axis[i].owner = g; }
  if (geometry) {   // IGALoadGeometry :201-286
    int nsd = 0;
    if (!bf.read_int(&nsd)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
    if (nsd < 1 || nsd > 3) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of space dimensions must be in range [1,3]");
    if (nsd < dim) return fail(PETSC_ERR_ARG_OUTOFRANGE, "Number of space dimensions must greater than or equal to dim");
    int vid = 0, n = 0;
    if (!bf.read_int(&vid) || !bf.read_int(&n)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
    if (vid != kVecFileClassId) return fail(PETSC_ERR_ARG_WRONG, "Not a vector next in file");
    size_t npts = 1;
    for (int i = 0; i < dim; i++) npts *= (size_t)(g->axis[i].m - g->axis[i].p);
    if ((size_t)n != npts * (nsd + 1)) return fail(PETSC_ERR_FILE_UNEXPECTED, "Vector in file different size than input vector");
    std::vector<double> Xw((size_t)n), X(npts * nsd), W(npts);
    if (!bf.read_reals(Xw.data(), Xw.size())) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
    for (size_t a = 0, pos = 0; a < npts; a++) {
      for (int i = 0; i < nsd; i++) X[i + a * nsd] = Xw[pos++];
      W[a] = Xw[pos++];
      if (std::fabs(W[a]) > 0) for (int i = 0; i < nsd; i++) X[i + a * nsd] /= W[a];          // :262-264
    }
    if (PetscErrorCode e = IGASetGeometryArrays(g, nsd, X.data(), W.data())) return e;          // rational iff max(w)-min(w) > 100 eps (:251-253)
  }
  if (property) return fail(PETSC_ERR_SUP, "IGARead: property fields are not part of the device path");
  return 0;
}

PetscErrorCode IGAGetGeometryArrays(IGA g, PetscInt sizes[3], PetscInt* nsd, PetscBool* rational, PetscReal* X, PetscReal* W) {
  if (PetscErrorCode e = check(g)) return e;
  for (int d = 0; d < 3; d++) if (sizes) sizes[d] = d < g->dim ? g->axis[d].m - g->axis[d].p : 1;
  if (nsd) *nsd = g->nsd;
  if (rational) *rational = g->rational ? PETSC_TRUE : PETSC_FALSE;
  if (X && g->nsd) memcpy(X, g->geomX.data(), g->geomX.size() * sizeof(double));
  if (W && g->nsd) { const size_t n = g->geomX.size() / g->nsd; for (size_t a = 0; a < n; a++) W[a] = g->geomW_all.empty() ? 1.0 : g->geomW_all[a]; }
  return 0;
}

// IGAWrite -> IGASave (src/petigaio.c:571-597, :75-139); the file is written by rank 0 (every rank of the mirror holds the
// full natural geometry arrays)
PetscErrorCode IGAWrite(IGA g, const char filename[]) {
  if (PetscErrorCode e = check(g)) return e;
  if (!filename) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");          // IGACheckSetUpStage2
  if (g->comm.rank != 0) return 0;
  BinFile bf;
  if (!bf.open(filename, "wb")) return fail(PETSC_ERR_FILE_OPEN, std::string("Cannot open file ") + filename);
  bool ok = bf.write_int(kIGAFileClassId) && bf.write_int(g->nsd ? 0x1 : 0x0) && bf.write_int(g->dim);
  for (int i = 0; ok && i < g->dim; i++) {
    const _n_IGAAxis& ax = g->axis[i];
    ok = bf.write_int(ax.p) && bf.write_int(ax.m + 1) && bf.write_reals(ax.U.data(), (size_t)ax.m + 1);
  }
  if (ok && g->nsd) {   // IGASaveGeometry :288-369
    const int nsd = g->nsd;
    const size_t npts = g->geomX.size() / nsd;
    std::vector<double> Xw(npts * (nsd + 1));
    for (size_t a = 0, pos = 0; a < npts; a++) {
      const bool hasW = !g->geomW_all.empty();
      const double w = (hasW && std::fabs(g->geomW_all[a]) > 0) ? g->geomW_all[a] : 1.0;
      for (int i = 0; i < nsd; i++) Xw[pos++] = g->geomX[i + a * nsd] * w;
      Xw[pos++] = hasW ? g->geomW_all[a] : 1.0;
    }
    ok = bf.write_int(nsd) && bf.write_int(kVecFileClassId) && bf.write_int((int)Xw.size()) && bf.write_reals(Xw.data(), Xw.size());
  }
  if (!ok) return fail(PETSC_ERR_FILE_WRITE, "Error writing to file");
  return 0;
}

// natural index (i fastest over the global node grid) of this rank's owned nodes, in owned order
static void owned_natural(IGA g, std::vector<size_t>& nat) {
  const int* ls = g->node_lstart; const int* lw = g->node_lwidth;
  const size_t n0 = g->axis[0].nnp, n1 = g->axis[1].nnp;
  nat.clear();
  for (int k = 0; k < lw[2]; k++) for (int j = 0; j < lw[1]; j++) for (int i = 0; i < lw[0]; i++)
    nat.push_back((size_t)(ls[0] + i) + n0 * ((size_t)(ls[1] + j) + n1 * (size_t)(ls[2] + k)));
}

// natural (i fastest over the global node grid) index of every owned node, in this rank's owned = PETSc-global order
PetscErrorCode IGAGetOwnedNaturalIndices(IGA g, PetscInt* nat) {
  if (PetscErrorCode e = check(g)) return e;
  if (!nat) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  std::vector<size_t> v;
  owned_natural(g, v);
  for (size_t a = 0; a < v.size(); a++) nat[a] = (PetscInt)v[a];
  return 0;
}

// IGAReadVec -> IGALoadVec (src/petigaio.c:685-709, :644-662): file holds the natural vector; every rank reads its part
PetscErrorCode IGAReadVec(IGA g, Vec vec, const char filename[]) {
  if (PetscErrorCode e = check(g)) return e;
  if (!vec || !filename) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  BinFile bf;
  if (!bf.open(filename, "rb")) return fail(PETSC_ERR_FILE_OPEN, std::string("Cannot open file ") + filename);
  int vid = 0, n = 0;
  if (!bf.read_int(&vid) || !bf.read_int(&n)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
  if (vid != kVecFileClassId) return fail(PETSC_ERR_ARG_WRONG, "Not a vector next in file");
  const size_t ntot = (size_t)g->axis[0].nnp * g->axis[1].nnp * g->axis[2].nnp * g->dof;
  if ((size_t)n != ntot) return fail(PETSC_ERR_FILE_UNEXPECTED, "Vector in file different size than input vector");
  std::vector<double> nat_v(ntot), own((size_t)vec->n);
  if (!bf.read_reals(nat_v.data(), ntot)) return fail(PETSC_ERR_FILE_READ, "Read past end of file");
  std::vector<size_t> nat;
  owned_natural(g, nat);
  for (size_t a = 0; a < nat.size(); a++) for (int c = 0; c < g->dof; c++) own[a * g->dof + c] = nat_v[nat[a] * g->dof + c];
  return VecSetArrayHost(vec, own.data());
}

// IGAWriteVec -> IGASaveVec (src/petigaio.c:711-735, :664-683)
PetscErrorCode IGAWriteVec(IGA g, Vec vec, const char filename[]) {
  if (PetscErrorCode e = check(g)) return e;
  if (!vec || !filename) return fail(PETSC_ERR_ARG_NULL, "Null pointer");
  if (!g->setup) return fail(PETSC_ERR_ARG_WRONGSTATE, "Must call IGASetUp() first");
  if (g->comm.size > 1) return fail(PETSC_ERR_SUP, "IGAWriteVec: gathering a distributed vector to the natural ordering is not available in the mirror");
  std::vector<double> own((size_t)vec->n);
  if (PetscErrorCode e = VecGetArrayHost(vec, own.data())) return e;
  BinFile bf;
  if (!bf.open(filename, "wb")) return fail(PETSC_ERR_FILE_OPEN, std::string("Cannot open file ") + filename);
  if (!(bf.write_int(kVecFileClassId) && bf.write_int(vec->n) && bf.write_reals(own.data(), own.size())))
    return fail(PETSC_ERR_FILE_WRITE, "Error writing to file");
  return 0;
}

}  // extern "C"
