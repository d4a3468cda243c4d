/*
 * petiga_host.h -- PETSc-free host mirror of the slice of PetIGA's public API (include/petiga.h of the
 * reference) that surrounds the element-assembly path, implemented on top of the C ABI in petiga_cuda.h.
 *
 * Why it exists: the reference is a PETSc library and this image has no PETSc/MPI, so the reference's own
 * drivers cannot be linked here.  This mirror keeps the reference's names, argument meaning and error
 * behaviour (PetscErrorCode returns, "must call X first" state checks) so that the parity tests read like
 * the reference's demos (demo/Poisson3D.c:26-67 etc.).  With PETSc present, the same calls are made from
 * PetIGA's re-written driver bodies instead (INTEGRATION.md).
 *
 * Differences forced by the missing dependencies (each is marked below):
 *   - MPI_Comm  -> IGAComm {rank, size, nccl communicator, device}
 *   - Mat / Vec -> minimal device-resident CSR / array objects with the AIJ / BAIJ value layouts
 *   - form callbacks are host function pointers in the reference; the GPU cannot call them, so the
 *     IGASetForm* setters accept only the exported IGADeviceForm_* sentinels (same signatures as
 *     include/petiga.h:153-171) and fail with PETSC_ERR_SUP for any other pointer.
 */
#ifndef PETIGA_HOST_H
#define PETIGA_HOST_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int PetscErrorCode;
typedef int PetscInt;
typedef double PetscReal;
typedef double PetscScalar;
typedef int PetscBool;
#define PETSC_TRUE 1
#define PETSC_FALSE 0
#define PETSC_DECIDE (-1)

/* PETSc error codes used by the mirrored functions (petscerror.h values) */
#define PETSC_ERR_MEM 55
#define PETSC_ERR_SUP 56
#define PETSC_ERR_ORDER 58
#define PETSC_ERR_ARG_OUTOFRANGE 63
#define PETSC_ERR_ARG_IDN 61
#define PETSC_ERR_ARG_WRONG 62
#define PETSC_ERR_ARG_WRONGSTATE 73
#define PETSC_ERR_LIB 76
#define PETSC_ERR_USER 83
#define PETSC_ERR_ARG_NULL 85
#define PETSC_ERR_FILE_OPEN 65
#define PETSC_ERR_FILE_READ 66
#define PETSC_ERR_FILE_WRITE 67
#define PETSC_ERR_FILE_UNEXPECTED 79

typedef struct { int rank, size; void *nccl; int device; } IGAComm;   /* stands in for MPI_Comm */

typedef struct _p_IGA *IGA;
typedef struct _n_IGAAxis *IGAAxis;
typedef struct _n_IGAPoint *IGAPoint;       /* opaque here: forms run on the device */
typedef struct _n_IGAForm *IGAForm;         /* include/petiga.h:220-268; opaque handle of the IGA's form */
typedef struct _p_Mat *Mat;
typedef struct _p_KSP *KSP;
typedef struct _p_Vec *Vec;

/* callback signatures of include/petiga.h:153-171 */
typedef PetscErrorCode (*IGAFormVector)(IGAPoint p, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormMatrix)(IGAPoint p, PetscScalar *K, void *ctx);
typedef PetscErrorCode (*IGAFormSystem)(IGAPoint p, PetscScalar *K, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormFunction)(IGAPoint p, const PetscScalar *U, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormJacobian)(IGAPoint p, const PetscScalar *U, PetscScalar *J, void *ctx);
typedef PetscErrorCode (*IGAFormIFunction)(IGAPoint p, PetscReal a, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormIJacobian)(IGAPoint p, PetscReal a, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscScalar *J, void *ctx);

/* include/petiga.h:172-197: second-order (I2), implicit-explicit (IE) and explicit (RHS) TS callbacks */
typedef PetscErrorCode (*IGAFormI2Function)(IGAPoint p, PetscReal a, const PetscScalar *A, PetscReal v, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormI2Jacobian)(IGAPoint p, PetscReal a, const PetscScalar *A, PetscReal v, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscScalar *J, void *ctx);
typedef PetscErrorCode (*IGAFormIEFunction)(IGAPoint p, PetscReal a, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscReal t0, const PetscScalar *U0, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormIEJacobian)(IGAPoint p, PetscReal a, const PetscScalar *V, PetscReal t, const PetscScalar *U, PetscReal t0, const PetscScalar *U0, PetscScalar *J, void *ctx);
typedef PetscErrorCode (*IGAFormRHSFunction)(IGAPoint p, PetscReal t, const PetscScalar *U, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormRHSJacobian)(IGAPoint p, PetscReal t, const PetscScalar *U, PetscScalar *J, void *ctx);

typedef PetscErrorCode (*IGAFormScalar)(IGAPoint p, const PetscScalar *U, PetscInt n, PetscScalar *S, void *ctx);   /* petiga.h:172 */
typedef PetscErrorCode (*IGAFormExact)(IGAPoint p, PetscInt k, PetscScalar V[], void *ctx);                          /* petiga.h:173 */

/* ---- device-form sentinels: pass these where the reference passes the demo's callback; ctx points at the
        demo's AppCtx (its leading PetscReal members are the parameters).  Calling them on the host fails. ---- */
PetscErrorCode IGADeviceForm_Poisson_System(IGAPoint, PetscScalar *, PetscScalar *, void *);            /* demo/Poisson{1,2,3}D.c System      */
PetscErrorCode IGADeviceForm_Poisson_Function(IGAPoint, const PetscScalar *, PetscScalar *, void *);    /* residual of the same problem        */
PetscErrorCode IGADeviceForm_Poisson_Jacobian(IGAPoint, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_Laplace_System(IGAPoint, PetscScalar *, PetscScalar *, void *);            /* demo/Laplace.c SystemGalerkin       */
PetscErrorCode IGADeviceForm_L2Projection_System(IGAPoint, PetscScalar *, PetscScalar *, void *);       /* ctx: {PetscReal choice}             */
PetscErrorCode IGADeviceForm_Mass_System(IGAPoint, PetscScalar *, PetscScalar *, void *);               /* test/IGACreate.c System             */
PetscErrorCode IGADeviceForm_Mass_Matrix(IGAPoint, PetscScalar *, void *);                              /* test/IGACreate.c Matrix             */
PetscErrorCode IGADeviceForm_Mass_Vector(IGAPoint, PetscScalar *, void *);                              /* test/IGACreate.c Vector             */
PetscErrorCode IGADeviceForm_BoundaryIntegral_System(IGAPoint, PetscScalar *, PetscScalar *, void *);   /* demo/BoundaryIntegral.c:50-57 System (Laplace + face term) */
PetscErrorCode IGADeviceForm_Neumann_SystemGalerkin(IGAPoint, PetscScalar *, PetscScalar *, void *);    /* demo/Neumann.c:28-45                                       */
PetscErrorCode IGADeviceForm_ConvTest_Galerkin(IGAPoint, PetscScalar *, PetscScalar *, void *);         /* test/ConvTest.c:51-69; ctx: {c, k}                         */
/* collocation forms (IGASetUseCollocation): the strong form at each Greville point, K[a] and F of one row per node */
PetscErrorCode IGADeviceForm_Laplace_SystemCollocation(IGAPoint, PetscScalar *, PetscScalar *, void *);  /* demo/Laplace.c SystemCollocation: -Lap N_a */
PetscErrorCode IGADeviceForm_ConvTest_Collocation(IGAPoint, PetscScalar *, PetscScalar *, void *);      /* c N_a - k Lap N_a, F = (c + k dim pi^2) prod sin(pi x_i); ctx: {c, k} */
PetscErrorCode IGADeviceForm_Elasticity3D_System(IGAPoint, PetscScalar *, PetscScalar *, void *);       /* ctx: {lambda, mu}                   */
PetscErrorCode IGADeviceForm_Elasticity_System(IGAPoint, PetscScalar *, PetscScalar *, void *);         /* ctx: {mu, lambda} as demo/Elasticity.c:10-13 */
PetscErrorCode IGADeviceForm_CahnHilliard2D_Residual(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *); /* ctx: {theta, alpha} */
PetscErrorCode IGADeviceForm_CahnHilliard2D_Tangent(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_CahnHilliard3D_Residual(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *); /* demo/CahnHilliard3D.c:54-107; ctx: {theta, L0, lambda} */
PetscErrorCode IGADeviceForm_CahnHilliard3D_Tangent(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_Bratu_Function(IGAPoint, const PetscScalar *, PetscScalar *, void *);      /* ctx: {lambda}                       */
PetscErrorCode IGADeviceForm_Bratu_Jacobian(IGAPoint, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_Bratu_IFunction(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_Bratu_IJacobian(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);

PetscErrorCode IGADeviceForm_Nitsche_System(IGAPoint, PetscScalar *, PetscScalar *, void *);             /* demo/NitscheMethod.c:70-119 (interior + face terms) */
PetscErrorCode IGADeviceForm_SNES2D_Function(IGAPoint, const PetscScalar *, PetscScalar *, void *);     /* test/Test_SNES_2D.c:12-46 (dim 2, dof 4) */
PetscErrorCode IGADeviceForm_SNES2D_Jacobian(IGAPoint, const PetscScalar *, PetscScalar *, void *);     /* test/Test_SNES_2D.c:48-72 */
/* demo/PatternFormation.c:26-141; ctx: the demo's AppCtx {PetscBool IMPLICIT; PetscReal delta, D1, D2, alpha, beta, gamma, tau1, tau2} */
PetscErrorCode IGADeviceForm_PatternFormation_IEFunction(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_PatternFormation_IEJacobian(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
/* demo/ElasticRodFJ.F90 (ElasticRod_IFunction / ElasticRod_IJacobian); ctx: {rho, E} */
PetscErrorCode IGADeviceForm_ElasticRod_I2Function(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_ElasticRod_I2Jacobian(IGAPoint, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscReal, const PetscScalar *, PetscScalar *, void *);
/* explicit form of the transient Bratu problem (no reference demo registers an RHSFunction); ctx: {lambda} */
PetscErrorCode IGADeviceForm_Bratu_RHSFunction(IGAPoint, PetscReal, const PetscScalar *, PetscScalar *, void *);
PetscErrorCode IGADeviceForm_Bratu_RHSJacobian(IGAPoint, PetscReal, const PetscScalar *, PetscScalar *, void *);

/* Scalar / Exact sentinels for IGAComputeScalar and IGAComputeErrorNorm (src/petigacomp.c:35-186) */
PetscErrorCode IGADeviceScalar_CahnHilliard2D_Stats(IGAPoint, const PetscScalar *, PetscInt, PetscScalar *, void *);  /* demo/CahnHilliard2D.c:43-58; ctx: {theta, alpha, cbar} */
PetscErrorCode IGADeviceExact_ErrNormTest(IGAPoint, PetscInt, PetscScalar *, void *);     /* test/IGAErrNorm.c:26-52 (dof 4: 1, sum x, sum x^2, prod x) */
PetscErrorCode IGADeviceExact_ConvTest(IGAPoint, PetscInt, PetscScalar *, void *);        /* test/ConvTest.c:104-111 (k = 0, 1)                            */
PetscErrorCode IGADeviceExact_Neumann(IGAPoint, PetscInt, PetscScalar *, void *);         /* demo/Neumann.c:80-86 (k = 0)                                  */
PetscErrorCode IGADeviceExact_L2Projection(IGAPoint, PetscInt, PetscScalar *, void *);    /* demo/L2Projection.c:3-61; ctx: {PetscReal choice}; k = 0     */

/* ---- IGA object: include/petiga.h:393-460 ---- */
PetscErrorCode IGACreate(IGAComm comm, IGA *iga);
PetscErrorCode IGADestroy(IGA *iga);
PetscErrorCode IGASetDim(IGA iga, PetscInt dim);
PetscErrorCode IGAGetDim(IGA iga, PetscInt *dim);
PetscErrorCode IGASetDof(IGA iga, PetscInt dof);
PetscErrorCode IGAGetDof(IGA iga, PetscInt *dof);
PetscErrorCode IGASetOrder(IGA iga, PetscInt order);
PetscErrorCode IGASetProcessors(IGA iga, PetscInt i, PetscInt processors);
PetscErrorCode IGAGetAxis(IGA iga, PetscInt i, IGAAxis *axis);
PetscErrorCode IGASetRuleSize(IGA iga, PetscInt i, PetscInt nqp);
PetscErrorCode IGASetMatType(IGA iga, const char *mattype);            /* "aij" or "baij" (petiga.c:1326-1330 default) */
/* Isogeometric collocation instead of Galerkin (-iga_collocation).  Before IGASetUp; changing it afterwards is
   PETSC_ERR_ARG_WRONGSTATE.  IGASetUp then tabulates one point per basis function (its Greville abscissa, nel = nnp, one
   point, weight = detJac = 1), keeps the Galerkin partition and numbering, takes the owned node box as the element box and the
   union of the owned rows' stencils as the ghost box.  Collocation runs the collocation forms (IGADeviceForm_*Collocation) in
   the VECTOR, MATRIX and SYSTEM slots, dof 1, degree 2..8, non-periodic axes; IGAComputeSystem replaces the row of a node that
   carries an IGASetBoundaryValue by an identity row with F = the value.  Boundary loads, boundary forms, fix tables and the
   separable path are PETSC_ERR_SUP.  The matrix is not symmetric: solve it with KSPGMRES. */
PetscErrorCode IGASetUseCollocation(IGA iga, PetscBool collocation);
PetscErrorCode IGAGetUseCollocation(IGA iga, PetscBool *collocation);
PetscErrorCode IGASetUp(IGA iga);
/* geometry in natural ordering, i fastest, (n_d+1) control points per axis: X[..][nsd], W[..] or NULL.
   Stands in for IGALoadGeometry (src/petigaio.c:201-286), which reads the same arrays from a PETSc binary file. */
PetscErrorCode IGASetGeometryArrays(IGA iga, PetscInt nsd, const PetscReal *X, const PetscReal *W);

/* geometry / vector files in the reference's PETSc binary format (src/petigaio.c:11-139,201-369,535-735) */
PetscErrorCode IGARead(IGA iga, const char filename[]);
PetscErrorCode IGAWrite(IGA iga, const char filename[]);
PetscErrorCode IGAReadVec(IGA iga, Vec vec, const char filename[]);
PetscErrorCode IGAWriteVec(IGA iga, Vec vec, const char filename[]);
/* the geometry the IGA holds, natural ordering: sizes[3] control points per axis, nsd, rational flag; X/W may be NULL */
PetscErrorCode IGAGetGeometryArrays(IGA iga, PetscInt sizes[3], PetscInt *nsd, PetscBool *rational, PetscReal *X, PetscReal *W);

/* ---- axis: include/petiga.h:62-89 ---- */
PetscErrorCode IGAAxisSetPeriodic(IGAAxis axis, PetscBool periodic);
PetscErrorCode IGAAxisSetDegree(IGAAxis axis, PetscInt p);
PetscErrorCode IGAAxisSetKnots(IGAAxis axis, PetscInt m, const PetscReal U[]);
PetscErrorCode IGAAxisInitUniform(IGAAxis axis, PetscInt N, PetscReal Ui, PetscReal Uf, PetscInt C);
PetscErrorCode IGAAxisInitBreaks(IGAAxis axis, PetscInt nu, const PetscReal u[], PetscInt C);   /* src/petigaaxis.c:323-382 */
PetscErrorCode IGAAxisGetPeriodic(IGAAxis axis, PetscBool *periodic);
PetscErrorCode IGAAxisGetDegree(IGAAxis axis, PetscInt *p);
PetscErrorCode IGAAxisGetKnots(IGAAxis axis, PetscInt *m, PetscReal *U[]);
PetscErrorCode IGAAxisGetLimits(IGAAxis axis, PetscReal *Ui, PetscReal *Uf);
PetscErrorCode IGAAxisGetSpans(IGAAxis axis, PetscInt *nel, PetscInt *span[]);
PetscErrorCode IGAAxisGetSizes(IGAAxis axis, PetscInt *nel, PetscInt *nnp);

/* ---- boundary conditions and forms: include/petiga.h:297-308 ---- */
PetscErrorCode IGASetBoundaryValue(IGA iga, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value);
PetscErrorCode IGASetBoundaryLoad(IGA iga, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value);
PetscErrorCode IGASetBoundaryForm(IGA iga, PetscInt axis, PetscInt side, PetscBool flag);   /* boundary-integral pass on that face */
PetscErrorCode IGASetFixTable(IGA iga, Vec table);
PetscErrorCode IGASetFormVector(IGA iga, IGAFormVector Vector, void *ctx);
PetscErrorCode IGASetFormMatrix(IGA iga, IGAFormMatrix Matrix, void *ctx);
PetscErrorCode IGASetFormSystem(IGA iga, IGAFormSystem System, void *ctx);
PetscErrorCode IGASetFormFunction(IGA iga, IGAFormFunction Function, void *ctx);
PetscErrorCode IGASetFormJacobian(IGA iga, IGAFormJacobian Jacobian, void *ctx);
PetscErrorCode IGASetFormIFunction(IGA iga, IGAFormIFunction IFunction, void *ctx);
PetscErrorCode IGASetFormIJacobian(IGA iga, IGAFormIJacobian IJacobian, void *ctx);
PetscErrorCode IGASetFormI2Function(IGA iga, IGAFormI2Function IFunction, void *ctx);      /* include/petiga.h:309-314 */
PetscErrorCode IGASetFormI2Jacobian(IGA iga, IGAFormI2Jacobian IJacobian, void *ctx);
PetscErrorCode IGASetFormIEFunction(IGA iga, IGAFormIEFunction IEFunction, void *ctx);
PetscErrorCode IGASetFormIEJacobian(IGA iga, IGAFormIEJacobian IEJacobian, void *ctx);
PetscErrorCode IGASetFormRHSFunction(IGA iga, IGAFormRHSFunction RHSFunction, void *ctx);
PetscErrorCode IGASetFormRHSJacobian(IGA iga, IGAFormRHSJacobian RHSJacobian, void *ctx);

/* the IGAForm object API of the demos that use it (demo/BoundaryIntegral.c:163-172): include/petiga.h:270-289 */
PetscErrorCode IGAGetForm(IGA iga, IGAForm *form);
PetscErrorCode IGAFormSetBoundaryValue(IGAForm form, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value);
PetscErrorCode IGAFormSetBoundaryLoad(IGAForm form, PetscInt axis, PetscInt side, PetscInt field, PetscScalar value);
PetscErrorCode IGAFormSetBoundaryForm(IGAForm form, PetscInt axis, PetscInt side, PetscBool flag);
PetscErrorCode IGAFormClearBoundary(IGAForm form, PetscInt axis, PetscInt side);
PetscErrorCode IGAFormSetVector(IGAForm form, IGAFormVector Vector, void *ctx);
PetscErrorCode IGAFormSetMatrix(IGAForm form, IGAFormMatrix Matrix, void *ctx);
PetscErrorCode IGAFormSetSystem(IGAForm form, IGAFormSystem System, void *ctx);
PetscErrorCode IGAFormSetFunction(IGAForm form, IGAFormFunction Function, void *ctx);
PetscErrorCode IGAFormSetJacobian(IGAForm form, IGAFormJacobian Jacobian, void *ctx);
PetscErrorCode IGAFormSetIFunction(IGAForm form, IGAFormIFunction IFunction, void *ctx);
PetscErrorCode IGAFormSetIJacobian(IGAForm form, IGAFormIJacobian IJacobian, void *ctx);

/* ---- Mat / Vec: src/petigamat.c:345-549, src/petigavec.c:78-113 ---- */
PetscErrorCode IGACreateMat(IGA iga, Mat *mat);
PetscErrorCode IGACreateVec(IGA iga, Vec *vec);
PetscErrorCode MatDestroy(Mat *mat);
PetscErrorCode VecDestroy(Vec *vec);
/* sizes: local rows (scalar), local nnz in the matrix's own layout (scalars for AIJ, blocks for BAIJ), block size */
PetscErrorCode MatGetSizesIGA(Mat mat, PetscInt *nrows, int64_t *nnz, PetscInt *bs, PetscBool *baij);
PetscErrorCode MatGetCSRHost(Mat mat, PetscInt *rowptr, PetscInt *colidx, PetscScalar *values);   /* any may be NULL */
PetscErrorCode MatGetValuesDevice(Mat mat, PetscScalar **d_values);
PetscErrorCode VecGetLocalSize(Vec vec, PetscInt *n);
PetscErrorCode VecGetArrayHost(Vec vec, PetscScalar *out);
PetscErrorCode VecSetArrayHost(Vec vec, const PetscScalar *in);
PetscErrorCode VecGetArrayDevice(Vec vec, PetscScalar **d_array);

/* ---- the seven drivers: include/petiga.h:837-851 ---- */
PetscErrorCode IGAComputeVector(IGA iga, Vec B);
PetscErrorCode IGAComputeMatrix(IGA iga, Mat A);
PetscErrorCode IGAComputeSystem(IGA iga, Mat A, Vec B);
PetscErrorCode IGAComputeFunction(IGA iga, Vec U, Vec F);
PetscErrorCode IGAComputeJacobian(IGA iga, Vec U, Mat J);
PetscErrorCode IGAComputeIFunction(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, Vec F);
PetscErrorCode IGAComputeIJacobian(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, Mat J);
/* the IE / RHS / I2 drivers: include/petiga.h:852-877, src/petigats.c:182-477, src/petigats2.c:23-175 */
PetscErrorCode IGAComputeIEFunction(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Vec F);
PetscErrorCode IGAComputeIEJacobian(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Mat J);
PetscErrorCode IGAComputeRHSFunction(IGA iga, PetscReal t, Vec U, Vec F);
PetscErrorCode IGAComputeRHSJacobian(IGA iga, PetscReal t, Vec U, Mat J);
PetscErrorCode IGAComputeI2Function(IGA iga, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Vec F);
PetscErrorCode IGAComputeI2Jacobian(IGA iga, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Mat J);

/* ---- functionals: src/petigacomp.c:35-186.  vecU may be NULL; Scalar/Exact must be one of the sentinels above
        (Exact may be NULL: norms of the discrete field) ---- */
PetscErrorCode IGAComputeScalar(IGA iga, Vec vecU, PetscInt n, PetscScalar S[], IGAFormScalar Scalar, void *ctx);
PetscErrorCode IGAComputeErrorNorm(IGA iga, PetscInt k, Vec vecU, IGAFormExact Exact, PetscReal enorm[], void *ctx);

/* ---- introspection used by the tests / bench ---- */
PetscErrorCode IGAGetInfoArray(IGA iga, PetscInt info[46]);     /* same layout as the oracle's oiga_get_info */
PetscErrorCode IGAGetBasisTable(IGA iga, PetscInt axis, PetscInt which, PetscReal *out);  /* 0 value,1 weight,2 point,3 detJac,4 knots */
PetscErrorCode IGAGetLGMapHost(IGA iga, PetscInt *lgmap);
PetscErrorCode IGAGetOwnedNaturalIndices(IGA iga, PetscInt *nat);   /* [owned nodes]: the natural<->global map of IGAReadVec (src/petigavec.c n2g) */
PetscErrorCode IGASetOption(IGA iga, const char *name, PetscReal value);     /* forwarded to petiga_cuda_set_option; "async" = 1:
                                                                                 IGACompute* only enqueue on the IGA's stream (device-
                                                                                 resident hand-off to a GPU solve, SURVEY 8f-4) */
PetscErrorCode IGAGetStat(IGA iga, const char *name, PetscReal *value);
/* ---- the step after the path (SURVEY.md 8 f-4): the assembled Mat stays on the device and is consumed there ----
   IGACreateKSP: src/petiga.c:856-885; use as demo/Poisson3D.c:73-83 does.  The preconditioner is always the Jacobi diagonal
   (-pc_type jacobi).  Two Krylov methods (KSPSetType):
     KSPCG     conjugate gradients, for the symmetric positive definite systems of the linear demos.  The default of
               IGACreateKSP here (PETSc's default is GMRES).
     KSPGMRES  restarted GMRES (KSPGMRESSetRestart, default 30; classical Gram-Schmidt) for any matrix with a nonzero diagonal,
               e.g. the non-symmetric IJacobians of the nonlinear and time-dependent forms.  The diagonal is applied on the
               right (-ksp_pc_side right; PETSc's default side for GMRES is left), so the residual tested is |b - A x|.
   KSPGetResidualNorm returns |b - A x| / |b|; KSPGetConvergedReason says why the solve stopped.  For CG the reason is derived
   from what the CG kernel returns: |r| / |b| <= rtol gives RTOL, else fewer than maxits iterations gives ATOL, else
   DIVERGED_ITS; so a CG solve that meets atol in its last allowed burst of iterations is reported as DIVERGED_ITS.
   MatMult is the product the solvers iterate with. */
typedef const char *KSPType;
#define KSPCG "cg"
#define KSPGMRES "gmres"
typedef enum {
  KSP_CONVERGED_ITERATING = 0, KSP_CONVERGED_RTOL = 2, KSP_CONVERGED_ATOL = 3,
  KSP_DIVERGED_ITS = -3, KSP_DIVERGED_BREAKDOWN = -5, KSP_DIVERGED_NANORINF = -9
} KSPConvergedReason;
PetscErrorCode MatMult(Mat A, Vec x, Vec y);
PetscErrorCode IGACreateKSP(IGA iga, KSP *ksp);
PetscErrorCode KSPSetType(KSP ksp, KSPType type);                   /* KSPCG or KSPGMRES; any other name: PETSC_ERR_SUP */
PetscErrorCode KSPGMRESSetRestart(KSP ksp, PetscInt restart);       /* >= 1; ignored by CG */
PetscErrorCode KSPSetOperators(KSP ksp, Mat A, Mat P);
PetscErrorCode KSPSetTolerances(KSP ksp, PetscReal rtol, PetscReal abstol, PetscReal dtol, PetscInt maxits);
PetscErrorCode KSPSolve(KSP ksp, Vec b, Vec x);
PetscErrorCode KSPGetIterationNumber(KSP ksp, PetscInt *its);
PetscErrorCode KSPGetResidualNorm(KSP ksp, PetscReal *rnorm);
PetscErrorCode KSPGetConvergedReason(KSP ksp, KSPConvergedReason *reason);
PetscErrorCode KSPDestroy(KSP *ksp);

PetscErrorCode IGASynchronize(IGA iga);                                        /* wait for the IGA's stream (after IGASetOption(iga,"async",1)) */
PetscErrorCode IGASetStream(IGA iga, void *cuda_stream);                      /* stream all device work is enqueued on */
void *IGAGetLayout(IGA iga);                                                 /* the petiga_layout behind the IGA */
PetscErrorCode IGAGetPlan(IGA iga, void **plan);                             /* the petiga_cuda_plan behind the IGA */
const char *IGAGetLastErrorMessage(void);
/* pure host logic (no GPU needed): partition of src/petigapart.c */
PetscErrorCode IGA_Partition(PetscInt size, PetscInt rank, PetscInt dim, const PetscInt N[], PetscInt n[], PetscInt i[]);

#ifdef __cplusplus
}
#endif
#endif /* PETIGA_HOST_H */
