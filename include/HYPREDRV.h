/* HYPREDRV.h -- public C API of hypredrive_b200: the drop-in boundary.
 *
 * Same names, argument meaning, uint32_t error-bitfield convention and ownership rules as
 * the reference's include/HYPREDRV.h (line numbers below refer to that file).  Behind it the
 * solve path (BoomerAMG-preconditioned PCG/GMRES on a ParCSR matrix) runs entirely in
 * hand-written sm_100a CUDA kernels (include/hdk.h); there is no CPU fallback.  Entry points
 * outside the hot path named by SURVEY.md section 8 are exported too and fail with an error
 * bit and a message instead of being absent.
 *
 * Return value: the process-global sticky error bitfield; 0 == HYPREDRV_SUCCESS.  Callers
 * must serialise all HYPREDRV_* calls (reference include/HYPREDRV.h:66-70).
 */
#ifndef HYPREDRV_HEADER
#define HYPREDRV_HEADER

#include <mpi.h>
#include <stdint.h>

#include <HYPRE.h>
#include <HYPRE_IJ_mv.h>
#include <HYPRE_config.h>
#include <HYPRE_krylov.h>
#include <HYPRE_parcsr_ls.h>
#include <HYPRE_parcsr_mv.h>
#include <HYPRE_utilities.h>

#include "HYPREDRV_config.h"

#ifdef __cplusplus
extern "C" {
#endif

#define HYPREDRV_EXPORT_SYMBOL __attribute__((visibility("default")))
#define HYPREDRV_SUCCESS ((uint32_t)0u)

/* error bits (reference include/internal/error.h:16-47; ABI-visible through `code & BIT`) */
#define HYPREDRV_ERROR_YAML_INVALID_INDENT 0x00000001u
#define HYPREDRV_ERROR_YAML_INVALID_BASE_INDENT 0x00000002u
#define HYPREDRV_ERROR_YAML_INCONSISTENT_INDENT 0x00000004u
#define HYPREDRV_ERROR_YAML_INVALID_DIVISOR 0x00000008u
#define HYPREDRV_ERROR_YAML_TREE_NULL 0x00000010u
#define HYPREDRV_ERROR_YAML_TREE_INVALID 0x00000020u
#define HYPREDRV_ERROR_YAML_MIXED_INDENT 0x00000040u
#define HYPREDRV_ERROR_YAML_INVALID_INDENT_JUMP 0x00000080u
#define HYPREDRV_ERROR_INVALID_KEY 0x00000100u
#define HYPREDRV_ERROR_INVALID_VAL 0x00000200u
#define HYPREDRV_ERROR_UNEXPECTED_VAL 0x00000400u
#define HYPREDRV_ERROR_MAYBE_INVALID_VAL 0x00000800u
#define HYPREDRV_ERROR_MISSING_KEY 0x00001000u
#define HYPREDRV_ERROR_EXTRA_KEY 0x00002000u
#define HYPREDRV_ERROR_MISSING_SOLVER 0x00004000u
#define HYPREDRV_ERROR_MISSING_PRECON 0x00008000u
#define HYPREDRV_ERROR_MISSING_DOFMAP 0x00010000u
#define HYPREDRV_ERROR_INVALID_SOLVER 0x00020000u
#define HYPREDRV_ERROR_INVALID_PRECON 0x00040000u
#define HYPREDRV_ERROR_FILE_NOT_FOUND 0x00080000u
#define HYPREDRV_ERROR_FILE_UNEXPECTED_ENTRY 0x00100000u
#define HYPREDRV_ERROR_UNKNOWN_HYPREDRV_OBJ 0x00200000u
#define HYPREDRV_ERROR_HYPREDRV_NOT_INITIALIZED 0x00400000u
#define HYPREDRV_ERROR_UNKNOWN_TIMING 0x00800000u
#define HYPREDRV_ERROR_HYPRE_INTERNAL 0x01000000u
#define HYPREDRV_ERROR_MISSING_LIB 0x02000000u
#define HYPREDRV_ERROR_ALLOCATION 0x20000000u
#define HYPREDRV_ERROR_OUT_OF_BOUNDS 0x40000000u
#define HYPREDRV_ERROR_UNKNOWN 0x80000000u

struct hypredrv_struct;
typedef struct hypredrv_struct *HYPREDRV_t;

/* ---- lifecycle and error handling -------------------------------------------------------- */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_Initialize(void);                                     /* :112 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_Finalize(void);                                       /* :138 */
HYPREDRV_EXPORT_SYMBOL void     HYPREDRV_ErrorCodeDescribe(uint32_t error_code);               /* :170 */
HYPREDRV_EXPORT_SYMBOL void     HYPREDRV_ErrorCodeClear(void);                                 /* :187 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_ErrorInvalidValue(const char *message);               /* :199 */
HYPREDRV_EXPORT_SYMBOL void     HYPREDRV_SafeCallHandleError(uint32_t error_code, MPI_Comm comm, const char *file,
                                                             int line, const char *func);      /* :221 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_Create(MPI_Comm comm, HYPREDRV_t *hypredrv_ptr);      /* :257 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_Destroy(HYPREDRV_t *hypredrv_ptr);                    /* :289 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PrintLibInfo(MPI_Comm comm, int print_datetime);      /* :311 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PrintSystemInfo(MPI_Comm comm);                       /* :333 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PrintExitInfo(MPI_Comm comm, const char *argv0);      /* :358 */

/* ---- configuration (YAML text / file / presets) ----------------------------------------- */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsParse(int argc, char **argv, HYPREDRV_t hypredrv); /* :391 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_SetLibraryMode(HYPREDRV_t hypredrv);                  /* :427 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_ObjectSetName(HYPREDRV_t hypredrv, const char *name);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsGetWarmup(HYPREDRV_t hypredrv, int *warmup); /* :465 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsGetNumRepetitions(HYPREDRV_t hypredrv, int *num_reps);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsGetNumLinearSystems(HYPREDRV_t hypredrv, int *num_ls);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsGetNumPreconVariants(HYPREDRV_t hypredrv, int *num_variants);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsSetPreconVariant(HYPREDRV_t hypredrv, int variant_idx); /* :545 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsSetPreconPreset(HYPREDRV_t hypredrv, const char *preset); /* :570 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_InputArgsSetSolverPreset(HYPREDRV_t hypredrv, const char *preset); /* :596 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_SolverPresetRegister(const char *name, const char *yaml_text, const char *help);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconPresetRegister(const char *name, const char *yaml_text, const char *help);

/* ---- linear system ------------------------------------------------------------------------ */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemBuild(HYPREDRV_t hypredrv);               /* :669 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemReadMatrix(HYPREDRV_t hypredrv);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetMatrix(HYPREDRV_t hypredrv, HYPRE_Matrix mat_A); /* :728 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetRHS(HYPREDRV_t hypredrv, HYPRE_Vector vec);      /* :821 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetMatrixFromCSR(HYPREDRV_t hypredrv, HYPRE_BigInt row_start,
                                                                      HYPRE_BigInt row_end, const HYPRE_BigInt *indptr,
                                                                      const HYPRE_BigInt *col_indices,
                                                                      const HYPRE_Real *data);            /* :882 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetRHSFromArray(HYPREDRV_t hypredrv, HYPRE_BigInt row_start,
                                                                     HYPRE_BigInt row_end, const HYPRE_Real *values); /* :918 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetInitialGuess(HYPREDRV_t hypredrv, HYPRE_Vector vec); /* :956 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetSolution(HYPREDRV_t hypredrv, HYPRE_Vector vec);     /* :988 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetReferenceSolution(HYPREDRV_t hypredrv, HYPRE_Vector vec);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemResetInitialGuess(HYPREDRV_t hypredrv);                 /* :1052 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetPrecMatrix(HYPREDRV_t hypredrv, HYPRE_Matrix mat);   /* :1092 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetSolutionValues(HYPREDRV_t hypredrv, HYPRE_Complex **sol_data); /* :1369 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetSolutionLength(HYPREDRV_t hypredrv, HYPRE_BigInt *length);     /* :1382 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetSolutionNorm(HYPREDRV_t hypredrv, const char *norm_type,
                                                                     double *norm);                          /* :1409 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetSolution(HYPREDRV_t hypredrv, HYPRE_Vector *vec);    /* :1436 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetRHSValues(HYPREDRV_t hypredrv, HYPRE_Complex **rhs_data);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetRHS(HYPREDRV_t hypredrv, HYPRE_Vector *vec);         /* :1493 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetMatrix(HYPREDRV_t hypredrv, HYPRE_Matrix *mat);      /* :1518 */

/* B200 extension (additive): assemble one of the reference example stencils directly in HBM
 * (kind 7 / 27 / 107, see hdk_csr_stencil) instead of host assembly + upload, and install it
 * together with its right-hand side.  c = {cx,cy,cz} or {kappa,umax,dt}. */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetStencil(HYPREDRV_t hypredrv, int kind, int nx, int ny, int nz,
                                                                const double *c, HYPRE_BigInt row_start,
                                                                HYPRE_BigInt row_end);
/* B200 extension (additive): device pointer of the working solution / rhs (no D2H copy). */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemGetDevicePointers(HYPREDRV_t hypredrv, double **x_d, double **b_d);
/* B200 extension (additive): opaque device handles for roofline instrumentation (bench.py). */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_GetDeviceHandles(HYPREDRV_t hypredrv, void **hdk_matrix, void **hdk_amg);
/* B200 extension (additive): the hdk_amg_params block (include/hdk.h) the next AMG setup passes to
 * the device, after the same option checks (error bits set for unsupported combinations). */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconGetDeviceParams(HYPREDRV_t hypredrv, void *hdk_amg_params);

/* ---- preconditioner / solver lifecycle --------------------------------------------------- */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconCreate(HYPREDRV_t hypredrv);                    /* :1719 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverCreate(HYPREDRV_t hypredrv);              /* :1743 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconSetup(HYPREDRV_t hypredrv);                     /* :1771 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverSetup(HYPREDRV_t hypredrv);               /* :1798 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverApply(HYPREDRV_t hypredrv);               /* :1822 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconApply(HYPREDRV_t hypredrv, HYPRE_Vector vec_b, HYPRE_Vector vec_x); /* :1852 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_PreconDestroy(HYPREDRV_t hypredrv);                   /* :1878 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverDestroy(HYPREDRV_t hypredrv);             /* :1905 */

/* ---- statistics / annotations ------------------------------------------------------------- */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StatsPrint(HYPREDRV_t hypredrv);                      /* :1932 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_AnnotateBegin(HYPREDRV_t hypredrv, const char *name, int id); /* :1996 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_AnnotateEnd(HYPREDRV_t hypredrv, const char *name, int id);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_AnnotateLevelBegin(HYPREDRV_t hypredrv, int level, const char *name, int id);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_AnnotateLevelEnd(HYPREDRV_t hypredrv, int level, const char *name, int id);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverGetNumIter(HYPREDRV_t hypredrv, int *iters);        /* :2126 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverGetConverged(HYPREDRV_t hypredrv, int *converged);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverGetFinalRelativeResidualNorm(HYPREDRV_t hypredrv, double *norm);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverGetSetupTime(HYPREDRV_t hypredrv, double *seconds);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSolverGetSolveTime(HYPREDRV_t hypredrv, double *seconds); /* :2207 */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StatsLevelGetCount(HYPREDRV_t hypredrv, int level, int *count);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StatsLevelGetEntry(HYPREDRV_t hypredrv, int level, int index, int *entry_id,
                                                            int *num_solves, int *linear_iters, double *setup_time,
                                                            double *solve_time);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StatsLevelPrint(HYPREDRV_t hypredrv, int level);

/* ---- outside the hot path (SURVEY.md section 8): exported, fail with an error bit + message */
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetDiscreteGradient(HYPREDRV_t hypredrv, HYPRE_Matrix G);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetDiscreteCurl(HYPREDRV_t hypredrv, HYPRE_Matrix C);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetCoordinates(HYPREDRV_t hypredrv, HYPRE_Vector x, HYPRE_Vector y,
                                                                    HYPRE_Vector z);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetDofmap(HYPREDRV_t hypredrv, int size, const int *dofmap);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetInterleavedDofmap(HYPREDRV_t hypredrv, int num_local_blocks,
                                                                          int num_dof_types);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetContiguousDofmap(HYPREDRV_t hypredrv, int num_local_blocks,
                                                                         int num_dof_types);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemReadDofmap(HYPREDRV_t hypredrv);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemPrintDofmap(HYPREDRV_t hypredrv, const char *filename);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemPrint(HYPREDRV_t hypredrv);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetNearNullSpace(HYPREDRV_t hypredrv, int num_entries,
                                                                      int num_components, const HYPRE_Complex *values);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemSetNullSpace(HYPREDRV_t hypredrv, int num_entries,
                                                                  int num_components, const HYPRE_Complex *values);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StateVectorSet(HYPREDRV_t hypredrv, int nstates, HYPRE_IJVector *vecs);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StateVectorGetValues(HYPREDRV_t hypredrv, int index, HYPRE_Complex **data_ptr);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StateVectorCopy(HYPREDRV_t hypredrv, int index_in, int index_out);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StateVectorUpdateAll(HYPREDRV_t hypredrv);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_StateVectorApplyCorrection(HYPREDRV_t hypredrv, int state_idx);
HYPREDRV_EXPORT_SYMBOL uint32_t HYPREDRV_LinearSystemComputeEigenspectrum(HYPREDRV_t hypredrv);

/* scalar widths of this build (the reference's Python bridge queries the same three,
 * interfaces/python/src/HYPREDRV_python.h:27-43) */
HYPREDRV_EXPORT_SYMBOL int HYPREDRV_SizeofBigInt(void);
HYPREDRV_EXPORT_SYMBOL int HYPREDRV_SizeofReal(void);
HYPREDRV_EXPORT_SYMBOL int HYPREDRV_SizeofInt(void);

#ifdef __cplusplus
}
#endif
#endif /* HYPREDRV_HEADER */
