/* STUB of the few PETSc / PetIGA declarations that integration/petiga_cuda_glue.c touches -- for a syntax check only
 * (tests/test_host_layout.py::test_glue_compiles): PETSc, MPI and PetIGA's own headers are not in this image.  Field and function
 * names follow the reference's include/petiga.h:122-141 (IGABasis), :95-110 (IGAAxis), :221-268 (IGAForm), :327-391 (struct _p_IGA)
 * and the PETSc manual pages; nothing here is compiled into the product.  A real build includes the reference's <petiga.h>. */
#ifndef STUB_PETIGA_H
#define STUB_PETIGA_H
#include <stddef.h>
typedef int PetscErrorCode, PetscInt, PetscMPIInt, PetscBool, PetscMemType, PetscLogEvent;
typedef double PetscReal, PetscScalar;
typedef struct _p_Mat *Mat;
typedef struct _p_Vec *Vec;
typedef struct _p_PetscObject *PetscObject;
typedef struct _p_PetscContainer *PetscContainer;
typedef int MPI_Comm;
#define PETSC_SUCCESS 0
#define PETSC_ERR_LIB 76
#define PETSC_ERR_SUP 56
#define PETSC_TRUE 1
#define PETSC_FALSE 0
#define MPI_BYTE 1
#define PetscFunctionBegin
#define PetscFunctionReturn(x) return (x)
#define PetscCall(x) do { PetscErrorCode ierr_ = (x); if (ierr_) return ierr_; } while (0)
#define PetscCallMPI(x) PetscCall(x)
#define PetscCheck(cond, comm, code, ...) do { if (!(cond)) return (code); } while (0)
#define SETERRQ(comm, code, ...) return (code)
#define PetscSqrtReal(x) __builtin_sqrt(x)
#define PetscRealPart(x) (x)
typedef struct { PetscInt p, m, nel, nnp; PetscBool periodic; PetscReal *U; } *IGAAxis;
typedef struct { PetscInt nqp, nen; PetscInt *offset; PetscReal *detJac, *weight, *point, *value, *bnd_value[2], bnd_point[2]; } *IGABasis;
typedef struct { PetscInt count, field[64]; PetscScalar value[64]; } *IGAFormBC;
typedef PetscErrorCode (*IGAFormSystem)(void *p, PetscScalar *K, PetscScalar *F, void *ctx);
typedef PetscErrorCode (*IGAFormExact)(void *p, PetscInt k, PetscScalar *u, void *ctx);
typedef struct { struct { void *System, *Function, *Jacobian, *IFunction, *IJacobian, *Vector, *Matrix, *SysCtx, *FunCtx, *JacCtx, *IFunCtx, *IJacCtx, *VecCtx, *MatCtx; } *ops;
                 IGAFormBC value[3][2], load[3][2]; PetscBool visit[3][2]; } *IGAForm;
struct _p_IGA { PetscInt dim, dof, order; IGAAxis axis[3]; IGABasis basis[3]; IGAForm form;
                PetscInt proc_sizes[3], proc_ranks[3], elem_start[3], elem_width[3], node_lstart[3], node_lwidth[3], node_gstart[3], node_gwidth[3];
                PetscInt geometry; PetscBool rational, fixtable; PetscReal *geometryX, *rationalW; PetscScalar *fixtableU;
                PetscBool collocation; };
typedef struct _p_IGA *IGA;
extern PetscLogEvent IGA_FormSystem, IGA_FormFunction, IGA_FormJacobian, IGA_FormIFunction, IGA_FormIJacobian, IGA_FormVector, IGA_FormMatrix, IGA_FormScalar;
PetscErrorCode IGAGetComm(IGA, MPI_Comm *);
PetscErrorCode MPI_Comm_rank(MPI_Comm, PetscMPIInt *), MPI_Comm_size(MPI_Comm, PetscMPIInt *), MPI_Bcast(void *, int, int, int, MPI_Comm);
PetscErrorCode PetscObjectQuery(PetscObject, const char *, PetscObject *), PetscObjectCompose(PetscObject, const char *, PetscObject);
PetscErrorCode PetscContainerCreate(MPI_Comm, PetscContainer *), PetscContainerSetPointer(PetscContainer, void *), PetscContainerGetPointer(PetscContainer, void **);
PetscErrorCode PetscContainerSetUserDestroy(PetscContainer, PetscErrorCode (*)(void *)), PetscContainerDestroy(PetscContainer *);
PetscErrorCode PetscLogEventBegin(PetscLogEvent, void *, void *, void *, void *), PetscLogEventEnd(PetscLogEvent, void *, void *, void *, void *);
PetscErrorCode MatSeqAIJCUSPARSEGetArrayWrite(Mat, PetscScalar **), MatSeqAIJCUSPARSERestoreArrayWrite(Mat, PetscScalar **);
PetscErrorCode MatGetBlockSize(Mat, PetscInt *), PetscObjectTypeCompareAny(PetscObject, PetscBool *, const char *, ...);
PetscErrorCode VecGetArrayWriteAndMemType(Vec, PetscScalar **, PetscMemType *), VecRestoreArrayWriteAndMemType(Vec, PetscScalar **);
PetscErrorCode VecGetArrayReadAndMemType(Vec, const PetscScalar **, PetscMemType *), VecRestoreArrayReadAndMemType(Vec, const PetscScalar **);
PetscErrorCode PetscMemzero(void *, size_t);
#define IGACheckSetUp(iga, arg) do { } while (0)
#endif
