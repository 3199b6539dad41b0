/* laplacian.c -- example driver of the HYPREDRV_* C API in the manner of hypredrive's C_laplacian
 * example: the 7-point Poisson problem on an nx x ny x nz grid (coefficients 1), right-hand side 1
 * on the y = 0 plane and 0 elsewhere, assembled on the host through the HYPRE_IJ interface and
 * solved five times with AMG-PCG; rank 0 prints the statistics table.
 *   laplacian [-n nx ny nz] [-P px py pz]
 * -n is the global grid, -P the process grid (px * py * pz ranks of the launcher environment).
 * As in the hypredrive example, the processes form a Cartesian communicator (MPI_Cart_*), each owns
 * one block of the grid, and rows are numbered block by block in rank order (x fastest inside a
 * block), so every rank owns a contiguous range of rows.  With px = py = 1 that is the
 * lexicographic numbering of the whole grid. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "HYPREDRV.h"
#include "HYPREDRV_utils.h"

/* first index and extent of block c of n points split into p blocks */
static long long blk_lo(int n, int p, int c) { return (long long)n * c / p; }
static long long blk_len(int n, int p, int c) { return blk_lo(n, p, c + 1) - blk_lo(n, p, c); }

/* global row of grid point g (inside the domain) given every rank's first row */
static HYPRE_BigInt global_row(MPI_Comm cart, const int n[3], const int P[3], const HYPRE_BigInt *first,
                               const long long g[3])
{
   int c[3], q = 0;
   long long lo[3], len[3];
   for (int d = 0; d < 3; d++)
   {
      c[d] = 0;
      while (blk_lo(n[d], P[d], c[d] + 1) <= g[d]) c[d]++;
      lo[d] = blk_lo(n[d], P[d], c[d]);
      len[d] = blk_len(n[d], P[d], c[d]);
   }
   MPI_Cart_rank(cart, c, &q);
   return first[q] + ((g[2] - lo[2]) * len[1] + (g[1] - lo[1])) * len[0] + (g[0] - lo[0]);
}

static const char *CONFIG = "solver: pcg\npreconditioner: amg\n";

int main(int argc, char **argv)
{
   MPI_Comm comm = MPI_COMM_WORLD;
   int      myid = 0, nprocs = 1;
   int      n[3] = {10, 10, 10}, P[3] = {1, 1, 1};
   const int num_solves = 5;
   MPI_Init(&argc, &argv);
   for (int i = 1; i < argc; i++)
   {
      int *dst = !strcmp(argv[i], "-n") ? n : (!strcmp(argv[i], "-P") ? P : NULL);
      if (!dst || i + 3 >= argc)
      {
         fprintf(stderr, "usage: %s [-n nx ny nz] [-P px py pz]\n", argv[0]);
         return 1;
      }
      for (int d = 0; d < 3; d++) dst[d] = atoi(argv[++i]);
   }
   HYPREDRV_SAFE_CALL(HYPREDRV_Initialize());
   HYPREDRV_t obj = NULL;
   HYPREDRV_SAFE_CALL(HYPREDRV_Create(comm, &obj));
   MPI_Comm_rank(comm, &myid);
   MPI_Comm_size(comm, &nprocs);
   if (n[0] < 1 || n[1] < 1 || n[2] < 1 || P[0] < 1 || P[1] < 1 || P[2] < 1 || P[0] > n[0] || P[1] > n[1] ||
       P[2] > n[2])
   {
      if (!myid) fprintf(stderr, "%s: need a positive grid and at most one process per grid plane\n", argv[0]);
      return 1;
   }
   const int periods[3] = {0, 0, 0};
   MPI_Comm  cart;
   if (MPI_Cart_create(comm, 3, P, periods, 0, &cart) != MPI_SUCCESS)
   {
      if (!myid) fprintf(stderr, "%s: -P %d %d %d does not match %d processes\n", argv[0], P[0], P[1], P[2], nprocs);
      return 1;
   }
   /* the topology as the communicator reports it: the last rank sits at the far corner */
   int corner[3];
   MPI_Cart_coords(cart, nprocs - 1, 3, corner);
   if (!myid)
   {
      printf("Grid dimensions:      %d x %d x %d\n", n[0], n[1], n[2]);
      printf("Processor topology:   %d x %d x %d\n", corner[0] + 1, corner[1] + 1, corner[2] + 1);
      printf("Diffusion coeffs:     (%.2e, %.2e, %.2e)\n", 1.0, 1.0, 1.0);
      printf("Discretization:       7-point stencil\n");
      printf("Number of solves:     %d\n", num_solves);
      fflush(stdout);
   }
   char *cfg_argv[1] = {(char *)CONFIG};
   HYPREDRV_SAFE_CALL(HYPREDRV_SetLibraryMode(obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_InputArgsParse(1, cfg_argv, obj));

   /* every rank's first row (block sizes in rank order), this rank's block and its neighbours */
   HYPRE_BigInt *first = malloc((size_t)(nprocs + 1) * sizeof(HYPRE_BigInt));
   first[0] = 0;
   for (int q = 0; q < nprocs; q++)
   {
      int c[3];
      MPI_Cart_coords(cart, q, 3, c);
      first[q + 1] = first[q] + blk_len(n[0], P[0], c[0]) * blk_len(n[1], P[1], c[1]) * blk_len(n[2], P[2], c[2]);
   }
   int       me[3], lower[3], upper[3];
   long long lo[3], hi[3];
   MPI_Cart_coords(cart, myid, 3, me);
   for (int d = 0; d < 3; d++)
   {
      MPI_Cart_shift(cart, d, 1, &lower[d], &upper[d]);
      lo[d] = blk_lo(n[d], P[d], me[d]);
      hi[d] = blk_lo(n[d], P[d], me[d] + 1);
   }
   const HYPRE_BigInt ilower = first[myid], iupper = first[myid + 1] - 1;
   HYPRE_IJMatrix A;
   HYPRE_IJVector b;
   HYPRE_IJMatrixCreate(comm, ilower, iupper, ilower, iupper, &A);
   HYPRE_IJMatrixSetObjectType(A, HYPRE_PARCSR);
   HYPRE_IJMatrixInitialize(A);
   HYPRE_IJVectorCreate(comm, ilower, iupper, &b);
   HYPRE_IJVectorSetObjectType(b, HYPRE_PARCSR);
   HYPRE_IJVectorInitialize(b);
   /* neighbours in the order -z, -y, -x, +x, +y, +z after the diagonal */
   static const int dir[6][2] = {{2, -1}, {1, -1}, {0, -1}, {0, 1}, {1, 1}, {2, 1}};
   for (long long gz = lo[2]; gz < hi[2]; gz++)
      for (long long gy = lo[1]; gy < hi[1]; gy++)
         for (long long gx = lo[0]; gx < hi[0]; gx++)
         {
            const long long g[3] = {gx, gy, gz};
            HYPRE_BigInt    row = global_row(cart, n, P, first, g), cols[7];
            HYPRE_Complex   vals[7], rhs = (gy == 0) ? 1.0 : 0.0;
            int             k = 0;
            cols[k] = row; vals[k++] = 6.0;
            for (int e = 0; e < 6; e++)
            {
               long long h[3] = {gx, gy, gz};
               const int d = dir[e][0];
               h[d] += dir[e][1];
               if (h[d] < 0 || h[d] >= n[d]) continue;                   /* Dirichlet boundary */
               /* a point outside this block belongs to the neighbour MPI_Cart_shift named */
               if ((h[d] < lo[d] && lower[d] == MPI_PROC_NULL) || (h[d] >= hi[d] && upper[d] == MPI_PROC_NULL))
               {
                  fprintf(stderr, "%s: no neighbour process in direction %d\n", argv[0], d);
                  return 1;
               }
               cols[k] = global_row(cart, n, P, first, h); vals[k++] = -1.0;
            }
            HYPRE_IJMatrixSetValues(A, 1, &k, &row, cols, vals);
            HYPRE_IJVectorSetValues(b, 1, &row, &rhs);
         }
   HYPRE_IJMatrixAssemble(A);
   HYPRE_IJVectorAssemble(b);
   free(first);

   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetMatrix(obj, (HYPRE_Matrix)A));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetRHS(obj, (HYPRE_Vector)b));
   HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemSetInitialGuess(obj, NULL));
   for (int i = 0; i < num_solves; i++)
   {
      HYPREDRV_SAFE_CALL(HYPREDRV_LinearSystemResetInitialGuess(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_PreconCreate(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverCreate(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverSetup(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverApply(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_PreconDestroy(obj));
      HYPREDRV_SAFE_CALL(HYPREDRV_LinearSolverDestroy(obj));
   }
   HYPREDRV_SAFE_CALL(HYPREDRV_StatsPrint(obj));
   HYPRE_IJMatrixDestroy(A);
   HYPRE_IJVectorDestroy(b);
   MPI_Comm_free(&cart);
   HYPREDRV_SAFE_CALL(HYPREDRV_Destroy(&obj));
   HYPREDRV_SAFE_CALL(HYPREDRV_Finalize());
   MPI_Finalize();
   return 0;
}
