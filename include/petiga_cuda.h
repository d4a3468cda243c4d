/*
 * petiga_cuda.h -- C ABI of libpetiga_cuda: the B200-native element-assembly path of PetIGA.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  Everything behind it is CUDA for sm_100a; there is
 * no CPU fallback: every entry point returns PETIGA_CUDA_ERR_NODEVICE when no CUDA device is usable.
 * Signatures use plain C scalars, pointers and sizes only -- no PETSc, torch or C++ types -- so the
 * same library serves (a) PetIGA's own drivers re-written against include/petiga.h (INTEGRATION.md
 * shows the glue), (b) the PETSc-free host mirror in include/petiga_host.h and (c) ctypes.
 *
 * What each entry point replaces in the reference (/root/reference = dalcinl/PetIGA):
 *   petiga_cuda_plan_create   <- what IGASetUp leaves in `struct _p_IGA` (include/petiga.h:327-391;
 *                                src/petiga.c:1111-1493) + IGAElementInit (src/petigaelem.c:140-263)
 *   petiga_cuda_plan_pattern  <- IGACreateMat's preallocation pattern (src/petigamat.c:345-549)
 *   petiga_cuda_form_select   <- IGASetForm{Vector,Matrix,System,Function,Jacobian,IFunction,IJacobian}
 *                                (include/petiga.h:302-308, src/petigaform.c:155-263): a host
 *                                function pointer cannot run on the GPU, so a built-in device form id
 *                                + parameter block stands in for (fnptr, ctx)
 *   petiga_cuda_set_bc        <- IGASetBoundaryValue/Load + IGASetFixTable (include/petiga.h:297-300)
 *   petiga_cuda_set_geometry  <- iga->geometryX / iga->rationalW (include/petiga.h:348-353)
 *   petiga_cuda_compute       <- the bodies of IGAComputeVector/Matrix/System (src/petigaksp.c:33-202),
 *                                IGAComputeFunction/Jacobian (src/petigasnes.c:23-139),
 *                                IGAComputeIFunction/IJacobian (src/petigats.c:23-159), including the
 *                                zeroing, the G2L halo of the state (src/petigavec.c:147-169,256-269),
 *                                the per-element Dirichlet/Neumann fix-up (src/petigaelem.c:1263-1501),
 *                                the ADD_VALUES scatter (src/petigaelem.c:1525-1559) and the off-rank
 *                                row exchange of MatAssemblyBegin/End (src/petigaksp.c:197-200)
 *   petiga_cuda_finish        <- the synchronisation point of MatAssemblyEnd/VecAssemblyEnd
 *
 * All functions return int: 0 on success, else a PETIGA_CUDA_ERR_* code (petiga_cuda_strerror()).
 * They never throw and never call exit().  Work is enqueued on the plan's stream; only
 * petiga_cuda_finish and the *_host helpers synchronise.  A plan is not thread-safe (neither is the
 * reference's element iterator: one per IGA, src/petigaelem.c:264-272).
 */
#ifndef PETIGA_CUDA_H
#define PETIGA_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PETIGA_CUDA_VERSION 100

enum {
  PETIGA_CUDA_OK = 0,
  PETIGA_CUDA_ERR_ARG = 1,       /* bad argument (PETSC_ERR_ARG_OUTOFRANGE / ARG_WRONG analogue)      */
  PETIGA_CUDA_ERR_ORDER = 2,     /* call sequence wrong (PETSC_ERR_ORDER / ARG_WRONGSTATE analogue)   */
  PETIGA_CUDA_ERR_SUP = 3,       /* configuration not supported on the device (PETSC_ERR_SUP)         */
  PETIGA_CUDA_ERR_MEM = 4,       /* device or host allocation failed                                  */
  PETIGA_CUDA_ERR_CUDA = 5,      /* CUDA runtime error (message via petiga_cuda_last_error)           */
  PETIGA_CUDA_ERR_NODEVICE = 6,  /* no usable CUDA device: there is no CPU fallback                   */
  PETIGA_CUDA_ERR_NCCL = 7       /* NCCL error / NCCL not loadable                                    */
};

/* the seven driver slots (which IGACompute* is being replaced) */
enum {
  PETIGA_SLOT_VECTOR = 0, PETIGA_SLOT_MATRIX = 1, PETIGA_SLOT_SYSTEM = 2, PETIGA_SLOT_FUNCTION = 3,
  PETIGA_SLOT_JACOBIAN = 4, PETIGA_SLOT_IFUNCTION = 5, PETIGA_SLOT_IJACOBIAN = 6,
  /* the implicit-explicit, explicit and second-order TS drivers (src/petigats.c:182-477, src/petigats2.c:23-175) */
  PETIGA_SLOT_IEFUNCTION = 7, PETIGA_SLOT_IEJACOBIAN = 8, PETIGA_SLOT_RHSFUNCTION = 9, PETIGA_SLOT_RHSJACOBIAN = 10,
  PETIGA_SLOT_I2FUNCTION = 11, PETIGA_SLOT_I2JACOBIAN = 12, PETIGA_NSLOTS = 13
};

/* built-in device forms = the user callbacks of the reference's demos/tests */
enum {
  PETIGA_FORM_POISSON = 0,        /* demo/Poisson{1,2,3}D.c:3-23 System; as Function/Jacobian: its residual/tangent */
  PETIGA_FORM_LAPLACE = 1,        /* demo/Laplace.c:35-48 SystemGalerkin                                            */
  PETIGA_FORM_L2PROJECTION = 2,   /* demo/L2Projection.c:67-88; params[0] = function choice 0..7 (:3-61)            */
  PETIGA_FORM_ELASTICITY3D = 3,   /* demo/Elasticity3D.c:13-46; params = {lambda, mu}                               */
  PETIGA_FORM_ELASTICITY = 4,     /* demo/Elasticity.c:22-52 (dof == dim); params = {lambda, mu}                    */
  PETIGA_FORM_CAHNHILLIARD2D = 5, /* demo/CahnHilliard2D.c:84-197 Residual/Tangent; params = {theta, alpha}         */
  PETIGA_FORM_BRATU = 6,          /* demo/BratuFJ.F90 Function/Jacobian/IFunction/IJacobian; params = {lambda}      */
  PETIGA_FORM_MASS = 7,           /* test/IGACreate.c:10-64 Vector/Matrix/System (block mass, any dof)              */
  PETIGA_FORM_BOUNDARYINTEGRAL = 8, /* demo/BoundaryIntegral.c:27-57 System: Laplace inside, F = N*1.0 on the faces
                                     enabled with petiga_cuda_set_boundary_form (p->atboundary branch)               */
  PETIGA_FORM_NEUMANN = 9,        /* demo/Neumann.c:28-45 SystemGalerkin: Laplace + f = 4 pi^2 sum_i sin(2 pi x_i)   */
  PETIGA_FORM_CAHNHILLIARD3D = 10, /* demo/CahnHilliard3D.c:54-169 Residual/Tangent; params = {theta, L0, lambda}          */
  PETIGA_FORM_CONVTEST = 11,      /* test/ConvTest.c:30-69 Galerkin (reaction-diffusion); params = {c, k}                */
  PETIGA_FORM_SNES2D = 12,        /* test/Test_SNES_2D.c:12-72 Function/Jacobian (dim 2, dof 4)                            */
  PETIGA_FORM_PATTERNFORMATION = 13, /* demo/PatternFormation.c:26-141 IEFunction/IEJacobian (dim 2, dof 2);
                                        params = {IMPLICIT, delta, D1, D2, alpha, beta, gamma, tau1, tau2}                 */
  PETIGA_FORM_ELASTICROD = 14,    /* demo/ElasticRodFJ.F90 I2Function/I2Jacobian; params = {rho, E}                        */
  PETIGA_FORM_NITSCHE = 15,       /* demo/NitscheMethod.c:70-119 System: Poisson inside, Nitsche matrix + vector terms on the
                                     faces enabled with petiga_cuda_set_boundary_form                                       */
  /* isogeometric collocation (petiga_cuda_space.collocation = 1): the strong form at the Greville points; slots VECTOR, MATRIX,
     SYSTEM, dof 1.  A Galerkin form on a collocation plan, or one of these on a Galerkin plan, is PETIGA_CUDA_ERR_SUP */
  PETIGA_FORM_LAPLACE_COLLOCATION = 16,   /* demo/Laplace.c SystemCollocation: K[a] = -Lap N_a, F = 0                                 */
  PETIGA_FORM_CONVTEST_COLLOCATION = 17,  /* strong form of test/ConvTest.c: K[a] = c N_a - k Lap N_a,
                                             F = (c + k dim pi^2) prod sin(pi x_i); params = {c, k}                                 */
  PETIGA_NFORMS = 18              /* PETIGA_FORM_BRATU also provides RHSFunction/RHSJacobian (its explicit form)            */
};

/* built-in Scalar callbacks of petiga_cuda_compute_scalar (IGAComputeScalar, src/petigacomp.c:35-96) */
enum {
  PETIGA_SCALAR_ERRNORM = 0,      /* ErrorSqr of IGAComputeErrorNorm (src/petigacomp.c:103-124): n = dof squared errors;
                                     params = {k (0..2), exact id, choice}; exact id 0 = NULL, 1 = test/IGAErrNorm.c:26-52
                                     (dof 4), 2 = demo/L2Projection.c:3-61 function `choice` (k = 0), 3 = demo/Neumann.c:5-8
                                     Solution (k = 0), 4 = test/ConvTest.c:8-28 prod sin(pi x_i) (k = 0, 1)                */
  PETIGA_SCALAR_CH_STATS = 1,     /* demo/CahnHilliard2D.c:36-58 monitor: n = 3 (free energy, 2nd, 3rd moment);
                                     params = {theta, alpha, cbar}                                                          */
  PETIGA_NSCALARS = 2
};

/* assembly algorithm selection (petiga_cuda_set_option "path") */
enum {
  PETIGA_PATH_AUTO = 0,           /* Kronecker row-gather when the form/geometry is separable, else quadrature     */
  PETIGA_PATH_QUADRATURE = 1,     /* always the per-element quadrature kernels (the reference's formulation)       */
  PETIGA_PATH_KRONECKER = 2,      /* force the separable path; PETIGA_CUDA_ERR_SUP when not applicable             */
  PETIGA_PATH_COLLOCATION = 3     /* stat "last_path" only: the collocation kernel of a collocation plan ran              */
};
/* quadrature kernel selection (petiga_cuda_set_option "quad_impl"): -1 = by element size; 0 = sum-factorised; 1 = pair loop;
   2 = generic runtime-degree kernel (mixed degrees, degree <= 8, dof <= 8, second derivatives on mapped / NURBS geometry,
   the IE/RHS/I2 drivers, boundary-integral matrix terms) */

typedef struct petiga_cuda_plan petiga_cuda_plan;

/* What IGASetUp computed (host pointers; copied at plan creation).  Axes >= dim must be the reference's
   "reset" axis: p=0, m=1, U={-0.5,0.5}, nel=nnp=1, one quadrature point (src/petigaaxis.c:44-66). */
typedef struct {
  int dim, dof, order;                 /* order: highest derivative a form may read (1..3)                 */
  int p[3], m[3], nel[3], nnp[3], periodic[3], nqp1[3];
  const double *U[3];                  /* knot vectors [m+1]            (IGAAxis.U,      petiga.h:50-60)   */
  const int    *offset[3];             /* [nel]                         (IGABasis.offset petiga.h:122-141) */
  const double *detJac[3];             /* [nel]                                                             */
  const double *weight[3];             /* [nel][nqp1]                                                       */
  const double *point[3];              /* [nel][nqp1]                                                       */
  const double *value[3];              /* [nel][nqp1][p+1][5]                                               */
  int proc_sizes[3], proc_ranks[3];    /* IGA_Partition                 (src/petigapart.c:136-168)         */
  int elem_start[3], elem_width[3];    /* this rank's element box       (src/petigapart.c:170-202)         */
  int node_lstart[3], node_lwidth[3];  /* owned node box                (src/petiga.c:1186-1209)           */
  int node_gstart[3], node_gwidth[3];  /* ghost node box                                                   */
  int collocation;                     /* IGASetUseCollocation (0 = Galerkin).  The tables then hold one point per basis
                                          function -- its Greville abscissa: nnp entries, nqp1 = 1, offset[i] = span - p,
                                          weight = detJac = 1, value = the basis and its derivatives there -- and the element box
                                          is the owned node box.  The partition and numbering stay the Galerkin ones (from the
                                          knot spans); the ghost box is the union of the owned rows' stencils.  nel may be
                                          the table length nnp (IGABasis.nel) or the axis's element count (IGAAxis.nel). */
} petiga_cuda_space;   /* the boxes of the other ranks follow from (nel, offset, proc_sizes) by the same arithmetic */

/* IGAFormBC tables (include/petiga.h:221-225) + the fix table */
typedef struct {
  int    vcount[3][2]; int vfield[3][2][64]; double vvalue[3][2][64];   /* IGASetBoundaryValue */
  int    lcount[3][2]; int lfield[3][2][64]; double lvalue[3][2][64];   /* IGASetBoundaryLoad  */
  const double *fixtableU;             /* host, ghost-box local [gw_k][gw_j][gw_i][dof] or NULL (IGASetFixTable) */
} petiga_cuda_bc;

/* ---- library ---- */
int         petiga_cuda_version(void);
const char *petiga_cuda_strerror(int code);
const char *petiga_cuda_last_error(void);             /* detail of the last failure on this thread          */
int         petiga_cuda_device_count(int *count);

/* Measured FP64 FMA throughput of the device in TFLOP/s (DFMA micro-benchmark: best single launch = burst, back-to-back
   launches for `seconds` = sustained).  The roofline denominator of the quadrature kernels (SURVEY.md 8d). */
int         petiga_cuda_measure_fp64(int device, double seconds, double *tflops_burst, double *tflops_sustained);

/* ---- plan ---- */
/* stream: a cudaStream_t (NULL = the plan creates its own non-blocking stream).
   nccl_comm: an ncclComm_t spanning `nranks` ranks, or NULL when nranks == 1 (or to let the plan use
   petiga_cuda_comm_* below). device: CUDA device ordinal. */
int petiga_cuda_plan_create(petiga_cuda_plan **plan, const petiga_cuda_space *space, int rank, int nranks,
                            void *nccl_comm, void *stream, int device);
int petiga_cuda_plan_destroy(petiga_cuda_plan *plan);
/* options: "path" (0 auto, 1 quadrature, 2 separable), "quad_impl" (-1 library's choice, 0 sum-factorised, 1 pair loop, 2 generic,
            3 third generation), "sf3_variant" (0 rows carried in the DMMA accumulators where the axis-0 rows advance one per element,
            1 shared-memory window always), "sf3_static" (1 use the compiled-in form structures when the run-time lists match),
            "kron_minb_rows" (scalar separable kernel: pencil length from which the 3-CTA build runs), "kron_bulk" (1: cp.async.bulk row
            stores, measured slower), "scatter" (99: integrate but skip the global reductions, profiling only)
   A collocation plan (petiga_cuda_space.collocation) always runs the collocation kernel; "path" = 2 is PETIGA_CUDA_ERR_SUP there.
   stats:   "launches", "last_path", "last_impl", "last_sf3_variant", "last_sf3_static", "last_kernel_ms", "last_flops", "num_sms",
            "nghostrows", "nnz_loc" */
int petiga_cuda_set_option(petiga_cuda_plan *plan, const char *name, double value);
int petiga_cuda_get_stat(petiga_cuda_plan *plan, const char *name, double *value);

/* geometry: host ghost-box arrays X[gw_k][gw_j][gw_i][nsd], W[gw_k][gw_j][gw_i] (W may be NULL);
   nsd must equal dim.  Pass X == NULL to return to the identity map. */
int petiga_cuda_set_geometry(petiga_cuda_plan *plan, int nsd, const double *X, const double *W);
int petiga_cuda_set_bc(petiga_cuda_plan *plan, const petiga_cuda_bc *bc);
/* Boundary-integral pass (IGASetBoundaryForm, src/petigaform.c; element side src/petigaelem.c:427-447,813-868,1012-1029):
   set_boundary_tables hands over IGABasis.bnd_value[0..1] ([p+1][5] each) and bnd_point[0..1] of one axis
   (include/petiga.h:134-139, src/petigabasis.c:208-217); set_boundary_form switches the pass on for a face.  A form
   without a boundary term (everything except PETIGA_FORM_BOUNDARYINTEGRAL) makes petiga_cuda_compute return
   PETIGA_CUDA_ERR_SUP while a face is enabled. */
int petiga_cuda_set_boundary_tables(petiga_cuda_plan *plan, int axis, const double *bnd_value0, const double *bnd_value1,
                                    double bnd_point0, double bnd_point1);
int petiga_cuda_set_boundary_form(petiga_cuda_plan *plan, int axis, int side, int flag);
/* IGASetFixTable with the table as a *global device vector* (this rank's owned part [owned nodes * dof]): the library does
   the global-to-local scatter itself (NCCL halo on more than one rank).  Call after petiga_cuda_set_bc; NULL clears it. */
int petiga_cuda_set_fixtable_device(petiga_cuda_plan *plan, const double *table_own);
/* form_id = -1 clears the slot (IGASetForm*(iga, NULL, NULL)); compute on it then fails with PETIGA_CUDA_ERR_ORDER */
int petiga_cuda_form_select(petiga_cuda_plan *plan, int slot, int form_id, const double *params, int nparams);

/* ---- pattern (IGACreateMat) ----
   block = 0: scalar AIJ CSR (rows = owned nodes * dof); block = 1: BAIJ block CSR (rows = owned nodes).
   Column ids are global (PETSc numbering), ascending in every row.  The arrays live on the device and are
   owned by the plan; *_host copies them out.  nnz counts scalars (block=0) or blocks (block=1). */
int petiga_cuda_plan_pattern(petiga_cuda_plan *plan, int block, int *nrows, int64_t *nnz,
                             const int **d_rowptr, const int **d_colidx);
int petiga_cuda_plan_pattern_host(petiga_cuda_plan *plan, int block, int *rowptr, int *colidx);
int petiga_cuda_plan_sizes(petiga_cuda_plan *plan, int *nown_nodes, int *nghost_nodes, int64_t *nnz_blocks);
int petiga_cuda_plan_lgmap_host(petiga_cuda_plan *plan, int *lgmap);   /* ghost node -> global node   */

/* ---- compute ----
   values: device array to assemble into, laid out as the pattern of `block` says
           (block=0: [nnz_scalar]; block=1: [nnz_blocks][dof*dof] column-major blocks as MATBAIJ stores them);
   rhs:    device array [owned nodes * dof].   Either may be NULL when the slot does not produce it.
   U, V:   device arrays [owned nodes * dof] (global vectors, this rank's part) or NULL.
   Outputs are zeroed first and fully assembled (ghost-row contributions exchanged) after
   petiga_cuda_finish, exactly as the reference drivers leave their Mat/Vec. */
int petiga_cuda_compute(petiga_cuda_plan *plan, int slot, int block, double shift, const double *V, double t,
                        const double *U, double *values, double *rhs);
/* The drivers with a third vector and a second shift / time (slots 7..12):
     IEFunction/IEJacobian (shift, V, t, U, t0, W = U0)      src/petigats.c:182-355
     RHSFunction/RHSJacobian (t, U)                           src/petigats.c:357-477
     I2Function/I2Jacobian (shift = shiftA, W = A, shift2 = shiftV, V, t, U)   src/petigats2.c:23-175
   Slots 0..6 ignore the extra arguments (petiga_cuda_compute is this call with them zero). */
int petiga_cuda_compute_ext(petiga_cuda_plan *plan, int slot, int block, double shift, const double *V, double t,
                            const double *U, double shift2, const double *W, double t0, double *values, double *rhs);
int petiga_cuda_finish(petiga_cuda_plan *plan);

/* ---- the step after the path (SURVEY.md 8 f-4): device-resident consumers of the assembled CSR ----
   In the reference the assembled Mat goes to PETSc: IGACreateKSP (src/petiga.c:856-885), KSPSetOperators + KSPSolve
   (demo/Poisson3D.c:73-83; the demo targets run -ksp_type cg -pc_type jacobi).  These two entry points keep that step on the
   device, so that assemble + solve moves no matrix byte over PCIe.  `block` and `values` as in petiga_cuda_compute; x, y, b are
   device vectors of the owned rows (nown * dof).  Multi-rank plans gather the operand over NCCL (rank-major global numbering).
   petiga_cuda_spmv      <- MatMult
   petiga_cuda_solve_cg  <- KSPSolve with KSPCG + PCJACOBI: x is the initial guess on entry; stops at |r| <= max(rtol |b|, atol)
                            or maxit; *iters and *relres (= |r| / |b|) report the outcome.  The matrix must be symmetric positive
                            definite (Poisson, Laplace, mass, elasticity systems).
   petiga_cuda_solve_gmres <- KSPSolve with KSPGMRES + PCJACOBI (-ksp_pc_side right; PETSc's default side for GMRES is left):
                            restarted GMRES(restart), classical Gram-Schmidt without refinement, the Jacobi diagonal applied on the
                            right (A D^-1 u = b, x = D^-1 u), so that rtol, atol and relres mean what they mean for CG.  Any square
                            matrix with a nonzero diagonal: the IJacobians of the nonlinear and time-dependent forms are not
                            symmetric.  x is the initial guess on entry; stops at |b - A x| <= max(rtol |b|, atol) or maxit.
                            Convergence is decided on the true residual, recomputed at the end of every cycle; *iters, *relres
                            (= |b - A x| / |b| at exit) and *reason (PETIGA_KSP_*, PETSc's KSPConvergedReason values) report the
                            outcome.  Stopping at maxit, a breakdown or a non-finite value returns 0 with the reason set; x then holds
                            the last finite iterate.  b = 0 gives x = 0, 0 iterations and PETIGA_KSP_CONVERGED_ATOL.
                            PETIGA_CUDA_ERR_ARG: a NULL pointer, b == x, restart < 1 or maxit < 0; PETIGA_CUDA_ERR_SUP: BAIJ with
                            dof > 4 (as petiga_cuda_spmv).  Deterministic: two solves of the same system give the same bits. */
enum {
  PETIGA_KSP_CONVERGED_ITERATING = 0, PETIGA_KSP_CONVERGED_RTOL = 2, PETIGA_KSP_CONVERGED_ATOL = 3,
  PETIGA_KSP_DIVERGED_ITS = -3, PETIGA_KSP_DIVERGED_BREAKDOWN = -5, PETIGA_KSP_DIVERGED_NANORINF = -9
};
int petiga_cuda_spmv(petiga_cuda_plan *plan, int block, const double *values, const double *x, double *y);
int petiga_cuda_solve_cg(petiga_cuda_plan *plan, int block, const double *values, const double *b, double *x,
                         double rtol, double atol, int maxit, int *iters, double *relres);
int petiga_cuda_solve_gmres(petiga_cuda_plan *plan, int block, const double *values, const double *b, double *x, int restart,
                            double rtol, double atol, int maxit, int *iters, double *relres, int *reason);

/* IGAComputeScalar (src/petigacomp.c:35-96): S[k] = sum over all ranks, elements and quadrature points of
   detJac*weight * Scalar_k(point, U).  U: device [owned nodes * dof] or NULL (a NULL state evaluates as zero, which is how
   IGAComputeErrorNorm(iga,k,NULL,Exact,..) yields the norms of the exact solution).  S_host receives the n global sums on
   every rank (the reference's MPI_Allreduce); the call synchronises the plan's stream.  Sums are deterministic. */
int petiga_cuda_compute_scalar(petiga_cuda_plan *plan, int scalar_id, const double *params, int nparams,
                               const double *U, int n, double *S_host);

/* host-buffer convenience (the end-to-end call: H2D of U/V, compute, D2H of values/rhs, synchronous) */
int petiga_cuda_compute_host(petiga_cuda_plan *plan, int slot, int block, double shift, const double *V_host,
                             double t, const double *U_host, double *values_host, double *rhs_host);

/* ---- device memory helpers for C callers without a CUDA runtime of their own.  They act on the CURRENT device:
        petiga_cuda_plan_activate makes the plan's device current (cudaSetDevice) ---- */
int petiga_cuda_plan_activate(petiga_cuda_plan *plan);
int petiga_cuda_malloc(void **ptr, size_t bytes);
int petiga_cuda_free(void *ptr);
int petiga_cuda_memcpy_h2d(void *dst, const void *src, size_t bytes);
int petiga_cuda_memcpy_d2h(void *dst, const void *src, size_t bytes);
int petiga_cuda_memset(void *dst, int value, size_t bytes);
int petiga_cuda_memset_async(petiga_cuda_plan *plan, void *dst, int value, size_t bytes);   /* enqueued on the plan's stream */
int petiga_cuda_host_alloc(void **ptr, size_t bytes);   /* pinned */
int petiga_cuda_host_free(void *ptr);
/* sum (a-b)^2 and sum b^2 over n device doubles on the current device (deterministic; synchronous): lets a caller compare two
   assembled value arrays (e.g. the two assembly paths at full size) without copying 2 x 5.9 GB to the host */
int petiga_cuda_diff_norm2(const double *d_a, const double *d_b, size_t n, double *diff2, double *ref2);

/* ---- NCCL bootstrap (one rank per GPU; the id travels over the caller's own channel, e.g. MPI_Bcast
        in PetIGA or torch.distributed in the test harness) ---- */
int petiga_cuda_comm_unique_id(void *id128);                       /* 128 bytes, call on rank 0        */
int petiga_cuda_comm_init(void **nccl_comm, int nranks, int rank, const void *id128, int device);
int petiga_cuda_comm_destroy(void *nccl_comm);

/* exchange plan introspection (host logic; usable without a GPU run): for this rank, the neighbours and
   the ghost-row / halo lists.  kind = 0: ghost rows sent to owners (matrix/vector assembly),
   kind = 1: rows received from lower neighbours.  Returns the count; when out != NULL fills
   out[3*i+0] = peer rank, out[3*i+1] = first row (local id), out[3*i+2] = number of rows. */
int petiga_cuda_plan_exchange_info(petiga_cuda_plan *plan, int kind, int *count, int *out, int capacity);

/* ---- host-only layout logic (needs no GPU): the integer work of IGASetUp_Stage2 + IGACreateMat
        (numbering, closed-form CSR positions, exchange lists) as a standalone object, so that it can be
        unit-tested on a CPU box and inspected by a caller.  The device plan uses the same tables. ---- */
typedef struct petiga_layout petiga_layout;
int petiga_layout_create(petiga_layout **layout, const petiga_cuda_space *space, int rank, int nranks);
int petiga_layout_destroy(petiga_layout *layout);
int petiga_layout_sizes(const petiga_layout *layout, int *nown, int *nghostbox, int *nloc, int64_t *nnz_own, int64_t *nnz_loc);
int petiga_layout_lgmap(const petiga_layout *layout, int *lgmap);          /* [nghostbox] */
int petiga_layout_localrow(const petiga_layout *layout, int *localrow);    /* [nghostbox] */
int petiga_layout_rowbase(const petiga_layout *layout, int64_t *rowbase);  /* [nloc+1]    */
int petiga_layout_pattern(const petiga_layout *layout, int block, int *rowptr, int *colidx);
/* closed-form position of column node (unwrapped ghost coordinates hb) in the row of ghost node ga */
int petiga_layout_position(const petiga_layout *layout, const int ga[3], const int hb[3], int64_t *pos);
/* kind 0: ghost rows I send (peer, first local row, nrows, nblocks); kind 1: rows I receive.
   out[4*i..]; for kind 1 the row list of peer i is returned by petiga_layout_recv_rows. */
int petiga_layout_exchange(const petiga_layout *layout, int kind, int *count, int64_t *out, int capacity);
int petiga_layout_recv_rows(const petiga_layout *layout, int peer_index, int *rows, int capacity);

#ifdef __cplusplus
}
#endif
#endif /* PETIGA_CUDA_H */
