/* csr_ingest.c -- unit test of HYPREDRV_LinearSystemSetMatrixFromCSR / SetRHSFromArray through
 * the C API: malformed input sets HYPREDRV_ERROR_INVALID_VAL without touching memory it was not
 * given, rows without entries are accepted, the library keeps its own copy of CSR input while a
 * caller's HYPRE_IJ objects stay the caller's across matrix replacements, and small systems (also
 * from an offset slab of indptr) solve to their known answers.  The sticky error state is handled
 * through the error-module entry points that hypredrive's own unit tests bind.
 * Prints one line per check and exits non-zero if any failed. */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include "HYPREDRV.h"
#include "HYPREDRV_utils.h"

/* hypredrive's internal error module (include/internal/error.h upstream), exported by the library */
void     hypredrv_ErrorCodeSet(uint32_t bits);
uint32_t hypredrv_ErrorCodeGet(void);
int      hypredrv_ErrorCodeActive(void);
void     hypredrv_ErrorCodeReset(uint32_t bits);
void     hypredrv_ErrorCodeResetAll(void);
void     hypredrv_ErrorMsgClear(void);

static const char *CONFIG = "general:\n  statistics: off\n"
                            "solver:\n  pcg:\n    max_iter: 100\n    relative_tol: 1.0e-8\n    print_level: 0\n"
                            "preconditioner:\n  amg:\n    print_level: 0\n";

static int failures = 0;

static void check(int ok, const char *what)
{
   printf("%s: %s\n", ok ? "ok" : "FAILED", what);
   failures += !ok;
}

/* the call fails with the INVALID_VAL bit, which the sticky state also holds until it is cleared */
static void expect_invalid(uint32_t code, const char *what)
{
   check((code & HYPREDRV_ERROR_INVALID_VAL) != 0 && (hypredrv_ErrorCodeGet() & HYPREDRV_ERROR_INVALID_VAL) != 0 &&
            hypredrv_ErrorCodeActive(), what);
   hypredrv_ErrorCodeResetAll();
   hypredrv_ErrorMsgClear();
   check(!hypredrv_ErrorCodeActive() && hypredrv_ErrorCodeGet() == 0, "error state cleared");
}

static void expect_solution(HYPREDRV_t obj, double a, double b, const char *what)
{
   HYPRE_Complex *x = NULL;
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemGetSolutionValues(obj, &x));
   check(x && fabs(x[0] - a) < 1e-6 && fabs(x[1] - b) < 1e-6, what);
}

static HYPREDRV_t create(void)
{
   HYPREDRV_t obj      = NULL;
   char      *argv[1]  = {(char *)CONFIG};
   HYPREDRV_SAFE_CALL(HYPREDRV_Create(MPI_COMM_WORLD, &obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_SetLibraryMode(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_InputArgsParse(1, argv, obj));
   return obj;
}

static void solve(HYPREDRV_t obj)
{
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetInitialGuess(obj, NULL));
   HYPREDRV_SAFE_CALL(HYPREDRV_PreconCreate(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverCreate(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverSetup(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverApply(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_PreconDestroy(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverDestroy(obj));
}

int main(int argc, char **argv)
{
   MPI_Init(&argc, &argv);
   HYPREDRV_SAFE_CALL(HYPREDRV_Initialize());
   HYPREDRV_t obj = create();

   /* ---- error module: bits accumulate and are cleared one by one or all at once ---- */
   hypredrv_ErrorCodeSet(HYPREDRV_ERROR_INVALID_VAL);
   hypredrv_ErrorCodeSet(HYPREDRV_ERROR_FILE_NOT_FOUND);
   check(hypredrv_ErrorCodeGet() == (HYPREDRV_ERROR_INVALID_VAL | HYPREDRV_ERROR_FILE_NOT_FOUND), "error bits accumulate");
   hypredrv_ErrorCodeReset(HYPREDRV_ERROR_INVALID_VAL);
   check(hypredrv_ErrorCodeGet() == HYPREDRV_ERROR_FILE_NOT_FOUND && hypredrv_ErrorCodeActive(), "one bit reset");
   hypredrv_ErrorCodeResetAll();
   check(hypredrv_ErrorCodeGet() == 0 && !hypredrv_ErrorCodeActive(), "all bits reset");

   /* ---- malformed input ---- */
   const HYPRE_BigInt ip2[3] = {0, 1, 2}, cols2[2] = {0, 1}, ip_dec[3] = {0, 2, 1}, ip_neg[2] = {-1, 0};
   const HYPRE_Real   diag2[2] = {2.0, 4.0};
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, NULL, cols2, diag2), "NULL indptr");
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 1, 0, ip2, cols2, diag2), "row_end < row_start");
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 0, ip_neg, cols2, diag2), "negative indptr[0]");
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip_dec, cols2, diag2), "decreasing indptr");
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip2, NULL, diag2), "NULL col_indices with entries");
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip2, cols2, NULL), "NULL data with entries");
   /* a row count beyond HYPRE_Int is refused before indptr[n] is read (indptr has two entries) */
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 2147483647LL, ip2, cols2, diag2), "row count overflow");
   const HYPRE_BigInt ip_big[2] = {0, 2147483648LL};
   expect_invalid(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 0, ip_big, cols2, diag2), "nonzero count overflow");
   const HYPRE_Real rhs2[2] = {8.0, 16.0};
   expect_invalid(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 1, rhs2), "right-hand side before the matrix");

   /* ---- rows without entries are accepted (row 1 of this 3 x 3 matrix is empty) ---- */
   const HYPRE_BigInt ip_empty[4] = {0, 1, 1, 2}, cols_empty[2] = {0, 2};
   const HYPRE_Real   vals_empty[2] = {1.0, 1.0};
   check(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 2, ip_empty, cols_empty, vals_empty) == HYPREDRV_SUCCESS,
         "matrix with an empty row");
   HYPREDRV_SAFE_CALL(HYPREDRV_Destroy(&obj));

   /* ---- known answers: diag(2, 4) x = (8, 16) -> x = (4, 4); then diag(4, 8) -> (2, 2) ---- */
   obj = create();
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip2, cols2, diag2));
   expect_invalid(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 2, rhs2), "right-hand side row range mismatch");
   expect_invalid(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 1, NULL), "NULL right-hand side values");
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 1, rhs2));
   solve(obj);
   expect_solution(obj, 4.0, 4.0, "diag(2, 4) x = (8, 16)");

   /* ---- ownership: CSR input is copied (the caller frees it right after the call) ---- */
   HYPRE_BigInt *ip_h = malloc(3 * sizeof(HYPRE_BigInt)), *cols_h = malloc(2 * sizeof(HYPRE_BigInt));
   HYPRE_Real   *vals_h = malloc(2 * sizeof(HYPRE_Real)), *rhs_h = malloc(2 * sizeof(HYPRE_Real));
   for (int i = 0; i < 3; i++) ip_h[i] = ip2[i];
   cols_h[0] = 0; cols_h[1] = 1; vals_h[0] = 4.0; vals_h[1] = 8.0; rhs_h[0] = 8.0; rhs_h[1] = 16.0;
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip_h, cols_h, vals_h));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 1, rhs_h));
   free(ip_h); free(cols_h); free(vals_h); free(rhs_h);
   solve(obj);
   expect_solution(obj, 2.0, 2.0, "replaced matrix diag(4, 8) from freed CSR arrays");

   /* ---- ownership: a caller's IJ matrix and vector replace the library's copy, and back ---- */
   HYPRE_IJMatrix A_ij;
   HYPRE_IJVector b_ij;
   HYPRE_IJMatrixCreate(MPI_COMM_WORLD, 0, 1, 0, 1, &A_ij);
   HYPRE_IJMatrixSetObjectType(A_ij, HYPRE_PARCSR);
   HYPRE_IJMatrixInitialize(A_ij);
   HYPRE_IJVectorCreate(MPI_COMM_WORLD, 0, 1, &b_ij);
   HYPRE_IJVectorSetObjectType(b_ij, HYPRE_PARCSR);
   HYPRE_IJVectorInitialize(b_ij);
   for (HYPRE_BigInt r = 0; r < 2; r++)
   {
      int           one = 1;
      HYPRE_Complex a = 1.0 + r, rhs = 8.0;
      HYPRE_IJMatrixSetValues(A_ij, 1, &one, &r, &r, &a);
      HYPRE_IJVectorSetValues(b_ij, 1, &r, &rhs);
   }
   HYPRE_IJMatrixAssemble(A_ij);
   HYPRE_IJVectorAssemble(b_ij);
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrix(obj, (HYPRE_Matrix)A_ij));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHS(obj, (HYPRE_Vector)b_ij));
   solve(obj);
   expect_solution(obj, 8.0, 4.0, "caller's IJ matrix diag(1, 2) x = (8, 8)");
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 1, ip2, cols2, diag2));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 1, rhs2));
   solve(obj);
   expect_solution(obj, 4.0, 4.0, "CSR matrix after the IJ matrix");
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrix(obj, (HYPRE_Matrix)A_ij));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHS(obj, (HYPRE_Vector)b_ij));
   solve(obj);
   expect_solution(obj, 8.0, 4.0, "the same IJ matrix again");
   HYPREDRV_SAFE_CALL(HYPREDRV_Destroy(&obj));
   /* the library never took the caller's objects: they are still valid and the caller frees them */
   HYPRE_BigInt lo = -1, hi = -1;
   check(HYPRE_IJMatrixGetLocalRange(A_ij, &lo, &hi, NULL, NULL) == 0 && lo == 0 && hi == 1, "IJ matrix still the caller's");
   check(HYPRE_IJMatrixDestroy(A_ij) == 0 && HYPRE_IJVectorDestroy(b_ij) == 0, "caller destroys its IJ objects");

   /* ---- offset slab: indptr = {2, 3} selects the third entry, 3 x = 6 -> ||x|| = 2 ---- */
   obj = create();
   const HYPRE_BigInt ip_off[2] = {2, 3}, cols_off[3] = {99, 99, 0};
   const HYPRE_Real   vals_off[3] = {0.0, 0.0, 3.0}, rhs1 = 6.0;
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrixFromCSR(obj, 0, 0, ip_off, cols_off, vals_off));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHSFromArray(obj, 0, 0, &rhs1));
   solve(obj);
   double norm = 0.0;
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemGetSolutionNorm(obj, "l2", &norm));
   check(fabs(norm - 2.0) < 1e-6, "offset indptr slab 3 x = 6");
   HYPREDRV_SAFE_CALL(HYPREDRV_Destroy(&obj));

   HYPREDRV_SAFE_CALL(HYPREDRV_Finalize());
   MPI_Finalize();
   printf("%d failure(s)\n", failures);
   return failures ? 1 : 0;
}
