/* petiga_cuda_glue.c -- what a PetIGA maintainer adds to bind libpetiga_cuda: replacement bodies of the assembly drivers
 *   IGAComputeVector/Matrix/System        src/petigaksp.c:33-202
 *   IGAComputeFunction/Jacobian           src/petigasnes.c:23-139
 *   IGAComputeIFunction/IJacobian         src/petigats.c:23-159
 *   IGAComputeIEFunction/IEJacobian, RHSFunction/RHSJacobian   src/petigats.c:182-477
 *   IGAComputeI2Function/I2Jacobian       src/petigats2.c:23-175
 *   IGAComputeErrorNorm                   src/petigacomp.c:127-186
 * written against the reference's <petiga.h>.  PETSc, MPI and PetIGA are not in this image, so the file is syntax-checked against
 * integration/stub/petiga.h (tests/test_host_layout.py::test_glue_compiles), not linked.  Everything else in PetIGA stays as it is:
 * the element loop, the Fortran kernels and MatSetValuesLocal are simply no longer reached from these drivers.
 * Value arrays: the library writes one CSR per rank with global column ids ascending in every row (petiga_cuda_plan_pattern) --
 * create the Mat with MatSetPreallocationCOO from that pattern or use a SeqAIJCUSPARSE/BAIJ matrix preallocated by IGACreateMat
 * (INTEGRATION.md 4, note on MPIAIJ). */
#include <petiga.h>
#include <petiga_cuda.h>

static PetscErrorCode IGACudaPlanDestroy(void *p) { return petiga_cuda_plan_destroy((petiga_cuda_plan *)p) ? PETSC_ERR_LIB : PETSC_SUCCESS; }

/* one plan per IGASetUp, composed on the IGA object */
static PetscErrorCode IGAGetCudaPlan(IGA iga, petiga_cuda_plan **plan)
{
  PetscContainer c = NULL;
  PetscFunctionBegin;
  PetscCall(PetscObjectQuery((PetscObject)iga, "petiga_cuda_plan", (PetscObject *)&c));
  if (!c) {
    petiga_cuda_space sp;
    PetscMPIInt       rank, size;
    PetscInt          i, s, ngpus = 8;
    MPI_Comm          comm;
    void             *nccl = NULL;
    unsigned char     id[128];
    PetscCall(PetscMemzero(&sp, sizeof(sp)));
    PetscCall(IGAGetComm(iga, &comm));
    PetscCallMPI(MPI_Comm_rank(comm, &rank));
    PetscCallMPI(MPI_Comm_size(comm, &size));
    sp.dim = iga->dim; sp.dof = iga->dof; sp.order = iga->order;                       /* include/petiga.h:337-339 */
    for (i = 0; i < 3; i++) {
      IGAAxis  ax = iga->axis[i];                                                       /* :341-343 */
      IGABasis b  = iga->basis[i];
      sp.p[i] = ax->p; sp.m[i] = ax->m; sp.nel[i] = ax->nel; sp.nnp[i] = ax->nnp; sp.periodic[i] = ax->periodic;
      sp.U[i] = ax->U; sp.nqp1[i] = b->nqp;
      sp.offset[i] = b->offset; sp.detJac[i] = b->detJac; sp.weight[i] = b->weight; sp.point[i] = b->point; sp.value[i] = b->value;
      sp.proc_sizes[i] = iga->proc_sizes[i]; sp.proc_ranks[i] = iga->proc_ranks[i];    /* :358-376 */
      sp.elem_start[i] = iga->elem_start[i]; sp.elem_width[i] = iga->elem_width[i];
      sp.node_lstart[i] = iga->node_lstart[i]; sp.node_lwidth[i] = iga->node_lwidth[i];
      sp.node_gstart[i] = iga->node_gstart[i]; sp.node_gwidth[i] = iga->node_gwidth[i];
    }
    sp.collocation = iga->collocation;                                                  /* IGASetUseCollocation: the basis tables
                                                                                           and boxes above are then the collocation ones
                                                                                           (nnp entries; nel = ax->nel is accepted) */
    if (size > 1) {                                                                     /* one rank per GPU; the id travels over MPI */
      if (!rank) PetscCheck(!petiga_cuda_comm_unique_id(id), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
      PetscCallMPI(MPI_Bcast(id, 128, MPI_BYTE, 0, comm));
      PetscCheck(!petiga_cuda_comm_init(&nccl, size, rank, id, rank % ngpus), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
    }
    PetscCheck(!petiga_cuda_plan_create(plan, &sp, rank, size, nccl, NULL, rank % ngpus), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
    if (iga->geometry)                                                                  /* ghost-box arrays, :348-353 */
      PetscCheck(!petiga_cuda_set_geometry(*plan, iga->geometry, iga->geometryX, iga->rational ? iga->rationalW : NULL), comm, PETSC_ERR_SUP, "%s", petiga_cuda_last_error());
    for (i = 0; i < iga->dim; i++) {                                                    /* IGABasis.bnd_value / bnd_point, :134-139 */
      IGABasis b = iga->basis[i];
      PetscCheck(!petiga_cuda_set_boundary_tables(*plan, i, b->bnd_value[0], b->bnd_value[1], b->bnd_point[0], b->bnd_point[1]), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
      for (s = 0; s < 2; s++) PetscCheck(!petiga_cuda_set_boundary_form(*plan, i, s, iga->form->visit[i][s]), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
    }
    PetscCall(PetscContainerCreate(comm, &c));
    PetscCall(PetscContainerSetPointer(c, *plan));
    PetscCall(PetscContainerSetUserDestroy(c, IGACudaPlanDestroy));
    PetscCall(PetscObjectCompose((PetscObject)iga, "petiga_cuda_plan", (PetscObject)c));
    PetscCall(PetscContainerDestroy(&c));
  } else PetscCall(PetscContainerGetPointer(c, (void **)plan));
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* IGASetBoundaryValue/Load + IGASetFixTable state of the form (include/petiga.h:221-268) -> the plan, before every compute */
static PetscErrorCode IGACudaPushBC(IGA iga, petiga_cuda_plan *plan)
{
  petiga_cuda_bc bc;
  PetscInt       i, s, k;
  MPI_Comm       comm;
  PetscFunctionBegin;
  PetscCall(IGAGetComm(iga, &comm));
  PetscCall(PetscMemzero(&bc, sizeof(bc)));
  for (i = 0; i < iga->dim; i++)
    for (s = 0; s < 2; s++) {
      IGAFormBC v = iga->form->value[i][s], l = iga->form->load[i][s];
      bc.vcount[i][s] = v->count;
      for (k = 0; k < v->count; k++) { bc.vfield[i][s][k] = v->field[k]; bc.vvalue[i][s][k] = v->value[k]; }
      bc.lcount[i][s] = l->count;
      for (k = 0; k < l->count; k++) { bc.lfield[i][s][k] = l->field[k]; bc.lvalue[i][s][k] = l->value[k]; }
    }
  bc.fixtableU = iga->fixtable ? iga->fixtableU : NULL;
  PetscCheck(!petiga_cuda_set_bc(plan, &bc), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
  PetscFunctionReturn(PETSC_SUCCESS);
}

/* the common body: state vectors in, Mat values and/or Vec out, all device pointers */
static PetscErrorCode IGACudaCompute(IGA iga, int slot, PetscLogEvent event, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal a2, Vec W, PetscReal t0, Mat J, Vec F)
{
  petiga_cuda_plan  *plan;
  const PetscScalar *u = NULL, *v = NULL, *w = NULL;
  PetscScalar       *vals = NULL, *f = NULL;
  PetscBool          baij = PETSC_FALSE;
  MPI_Comm           comm;
  PetscFunctionBegin;
  IGACheckSetUp(iga, 1);
  PetscCall(IGAGetComm(iga, &comm));
  PetscCall(IGAGetCudaPlan(iga, &plan));
  PetscCall(IGACudaPushBC(iga, plan));
  PetscCall(PetscLogEventBegin(event, iga, V, U, J ? (void *)J : (void *)F));            /* same events as the reference drivers */
  if (U) PetscCall(VecGetArrayReadAndMemType(U, &u, NULL));                              /* owned part; the G2L halo is inside the library */
  if (V) PetscCall(VecGetArrayReadAndMemType(V, &v, NULL));
  if (W) PetscCall(VecGetArrayReadAndMemType(W, &w, NULL));
  if (J) {
    PetscCall(PetscObjectTypeCompareAny((PetscObject)J, &baij, "seqbaij", "mpibaij", ""));
    PetscCall(MatSeqAIJCUSPARSEGetArrayWrite(J, &vals));
  }
  if (F) PetscCall(VecGetArrayWriteAndMemType(F, &f, NULL));
  PetscCheck(!petiga_cuda_compute_ext(plan, slot, baij, a, v, t, u, a2, w, t0, vals, f), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
  PetscCheck(!petiga_cuda_finish(plan), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());   /* == Mat/VecAssemblyEnd */
  if (F) PetscCall(VecRestoreArrayWriteAndMemType(F, &f));
  if (J) PetscCall(MatSeqAIJCUSPARSERestoreArrayWrite(J, &vals));
  if (W) PetscCall(VecRestoreArrayReadAndMemType(W, &w));
  if (V) PetscCall(VecRestoreArrayReadAndMemType(V, &v));
  if (U) PetscCall(VecRestoreArrayReadAndMemType(U, &u));
  PetscCall(PetscLogEventEnd(event, iga, V, U, J ? (void *)J : (void *)F));
  PetscFunctionReturn(PETSC_SUCCESS);
}

PetscErrorCode IGAComputeVector(IGA iga, Vec B) { return IGACudaCompute(iga, PETIGA_SLOT_VECTOR, IGA_FormVector, 0, NULL, 0, NULL, 0, NULL, 0, NULL, B); }
PetscErrorCode IGAComputeMatrix(IGA iga, Mat A) { return IGACudaCompute(iga, PETIGA_SLOT_MATRIX, IGA_FormMatrix, 0, NULL, 0, NULL, 0, NULL, 0, A, NULL); }
PetscErrorCode IGAComputeSystem(IGA iga, Mat A, Vec B) { return IGACudaCompute(iga, PETIGA_SLOT_SYSTEM, IGA_FormSystem, 0, NULL, 0, NULL, 0, NULL, 0, A, B); }
PetscErrorCode IGAComputeFunction(IGA iga, Vec U, Vec F) { return IGACudaCompute(iga, PETIGA_SLOT_FUNCTION, IGA_FormFunction, 0, NULL, 0, U, 0, NULL, 0, NULL, F); }
PetscErrorCode IGAComputeJacobian(IGA iga, Vec U, Mat J) { return IGACudaCompute(iga, PETIGA_SLOT_JACOBIAN, IGA_FormJacobian, 0, NULL, 0, U, 0, NULL, 0, J, NULL); }
PetscErrorCode IGAComputeIFunction(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, Vec F) { return IGACudaCompute(iga, PETIGA_SLOT_IFUNCTION, IGA_FormIFunction, a, V, t, U, 0, NULL, 0, NULL, F); }
PetscErrorCode IGAComputeIJacobian(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, Mat J) { return IGACudaCompute(iga, PETIGA_SLOT_IJACOBIAN, IGA_FormIJacobian, a, V, t, U, 0, NULL, 0, J, NULL); }
/* src/petigats.c:182-477: U0 at time t0 is the third vector */
PetscErrorCode IGAComputeIEFunction(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Vec F) { return IGACudaCompute(iga, PETIGA_SLOT_IEFUNCTION, IGA_FormIFunction, a, V, t, U, 0, U0, t0, NULL, F); }
PetscErrorCode IGAComputeIEJacobian(IGA iga, PetscReal a, Vec V, PetscReal t, Vec U, PetscReal t0, Vec U0, Mat J) { return IGACudaCompute(iga, PETIGA_SLOT_IEJACOBIAN, IGA_FormIJacobian, a, V, t, U, 0, U0, t0, J, NULL); }
PetscErrorCode IGAComputeRHSFunction(IGA iga, PetscReal t, Vec U, Vec F) { return IGACudaCompute(iga, PETIGA_SLOT_RHSFUNCTION, IGA_FormFunction, 0, NULL, t, U, 0, NULL, 0, NULL, F); }
PetscErrorCode IGAComputeRHSJacobian(IGA iga, PetscReal t, Vec U, Mat J) { return IGACudaCompute(iga, PETIGA_SLOT_RHSJACOBIAN, IGA_FormJacobian, 0, NULL, t, U, 0, NULL, 0, J, NULL); }
/* src/petigats2.c:23-175: shift a on A (third vector), shift v on V */
PetscErrorCode IGAComputeI2Function(IGA iga, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Vec F) { return IGACudaCompute(iga, PETIGA_SLOT_I2FUNCTION, IGA_FormIFunction, a, V, t, U, v, A, 0, NULL, F); }
PetscErrorCode IGAComputeI2Jacobian(IGA iga, PetscReal a, Vec A, PetscReal v, Vec V, PetscReal t, Vec U, Mat J) { return IGACudaCompute(iga, PETIGA_SLOT_I2JACOBIAN, IGA_FormIJacobian, a, V, t, U, v, A, 0, J, NULL); }

/* The exact-solution callback is a host pointer (include/petiga.h:171); the library exports sentinels with that signature
   (include/petiga_host.h:122-124) and evaluates the matching built-in on the device. */
extern PetscErrorCode IGADeviceExact_ErrNormTest(void *, PetscInt, PetscScalar *, void *);
extern PetscErrorCode IGADeviceExact_L2Projection(void *, PetscInt, PetscScalar *, void *);
static int IGACudaExactId(IGAFormExact Exact) { return Exact == IGADeviceExact_ErrNormTest ? 1 : Exact == IGADeviceExact_L2Projection ? 2 : 0; }

/* src/petigacomp.c:127-186: the element loop + MPI_Allreduce (:63-90) is one call; the sums arrive on every rank */
PetscErrorCode IGAComputeErrorNorm(IGA iga, PetscInt k, Vec vecU, IGAFormExact Exact, PetscReal enorm[], void *ctx)
{
  petiga_cuda_plan  *plan;
  const PetscScalar *u = NULL;
  PetscScalar        errsqr[64];
  double             prm[3];
  PetscInt           i, dof = iga->dof;
  MPI_Comm           comm;
  PetscFunctionBegin;
  IGACheckSetUp(iga, 1);
  PetscCall(IGAGetComm(iga, &comm));
  PetscCall(IGAGetCudaPlan(iga, &plan));
  prm[0] = (double)k;
  prm[1] = (double)IGACudaExactId(Exact);          /* 0 = no exact solution (norms of U itself) */
  prm[2] = ctx ? *(PetscReal *)ctx : 0.0;
  if (vecU) PetscCall(VecGetArrayReadAndMemType(vecU, &u, NULL));
  PetscCall(PetscLogEventBegin(IGA_FormScalar, iga, vecU, 0, 0));
  PetscCheck(!petiga_cuda_compute_scalar(plan, PETIGA_SCALAR_ERRNORM, prm, 3, u, dof, errsqr), comm, PETSC_ERR_LIB, "%s", petiga_cuda_last_error());
  PetscCall(PetscLogEventEnd(IGA_FormScalar, iga, vecU, 0, 0));
  if (vecU) PetscCall(VecRestoreArrayReadAndMemType(vecU, &u));
  for (i = 0; i < dof; i++) enorm[i] = PetscSqrtReal(PetscRealPart(errsqr[i]));       /* :180 */
  PetscFunctionReturn(PETSC_SUCCESS);
}
