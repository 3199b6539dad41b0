/* hdk.h -- thin C-ABI over the hand-written sm_100a CUDA kernels of hypredrive_b200.
 *
 * The HYPREDRV_* host layer (include/HYPREDRV.h, plain C) drives the device through these
 * entry points only: opaque handles, plain pointers and sizes, no C++/torch types.  Each
 * entry replaces one hypre call that the reference makes on the hot path; the reference
 * file:line it stands in for is quoted next to it.  All functions return 0 on success and a
 * non-zero code on failure; hdk_last_error() returns the message.  There is NO CPU
 * fallback: without a CUDA device every compute entry fails with HDK_ERR_NO_DEVICE.
 *
 * Pointers named *_d are DEVICE pointers, *_h HOST pointers.
 */
#ifndef HDK_H
#define HDK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HDK_OK 0
#define HDK_ERR_NO_DEVICE 1
#define HDK_ERR_CUDA 2
#define HDK_ERR_INVALID 3
#define HDK_ERR_ALLOC 4
#define HDK_ERR_UNSUPPORTED 5
#define HDK_ERR_COMM 6

typedef struct hdk_csr_s hdk_csr; /* device ParCSR block pair (diag + offd) of one rank */
typedef struct hdk_amg_s hdk_amg; /* device BoomerAMG hierarchy */

/* ---- runtime (reference: HYPRE_Initialize / HYPRE_Finalize, src/internal/runtime.c:101-133) */
int         hdk_init(int device);        /* device < 0: LOCAL_RANK env or current device */
int         hdk_finalize(void);
int         hdk_device_count(void);      /* 0 when no CUDA device is usable */
const char *hdk_last_error(void);
int         hdk_sync(void);              /* synchronise the compute stream */
void       *hdk_stream(void);            /* cudaStream_t of the compute stream */

/* ---- communicator (reference: MPI_Comm passed to HYPREDRV_Create, src/HYPREDRV.c:1014-1043).
 * One process per GPU.  The 128-byte NCCL unique id is produced on rank 0 and broadcast by
 * the host program (torch.distributed / any launcher) before hdk_comm_init. */
int hdk_comm_unique_id(void *id128_h);
int hdk_comm_init(int rank, int nranks, const void *id128_h);
/* the same from the launcher's environment alone (RANK, WORLD_SIZE, MASTER_ADDR/PORT): rank 0 publishes
 * the id through a file (HDK_NCCL_ID_FILE); used by HYPREDRV_Create when WORLD_SIZE > 1 and the host
 * program has not called hdk_comm_init itself */
int hdk_comm_init_from_env(void);
/* halo exchange in use: 0 = single rank, 1 = NCCL send/recv on a communication stream,
 * 2 = peer-memory stores over NVLink (CUDA IPC arena; HDK_HALO_IPC=0 disables) */
int hdk_comm_halo_mode(void);
int hdk_comm_rank(void);
int hdk_comm_size(void);
int hdk_comm_finalize(void);
/* max / sum of one 64-bit integer over all ranks (control plane: global sizes) */
int hdk_comm_max_i64(int64_t local, int64_t *global);
int hdk_comm_sum_i64(int64_t local, int64_t *global);

/* ---- device vectors (reference: HYPRE_IJVector / hypre_ParVector, src/internal/linsys.c:1412-1491) */
int hdk_vec_alloc(int64_t n, double **x_d);
int hdk_vec_free(double *x_d);
/* page-locked host buffers for the library-owned host views of device vectors (full PCIe rate) */
int hdk_host_alloc(size_t bytes, void **p_h);
int hdk_host_free(void *p_h);
int hdk_vec_h2d(double *x_d, const double *x_h, int64_t n);
int hdk_vec_d2h(double *x_h, const double *x_d, int64_t n);
int hdk_vec_fill(double *x_d, double value, int64_t n);
int hdk_vec_copy(double *dst_d, const double *src_d, int64_t n);
int hdk_vec_axpy(double alpha, const double *x_d, double *y_d, int64_t n);
int hdk_vec_scale(double alpha, double *x_d, int64_t n);
/* global (all-rank) inner product and norms; kind: 0 = L1, 1 = L2, 2 = Linf
 * (reference: hypre_ParVectorInnerProd, src/internal/linsys.c:2815-2924) */
int hdk_vec_dot(const double *x_d, const double *y_d, int64_t n, double *result_h);
int hdk_vec_norm(const double *x_d, int64_t n, int kind, double *result_h);
/* HYPRE_ParVectorSetRandomValues-compatible fill: x_i = 2 hypre_Rand() - 1 from the Park-Miller
 * stream seeded with `seed`, element i taken at position global_offset + i (identical to hypre on
 * one rank; partition-invariant on several) (reference: src/internal/linsys.c:1810-1838, 2050-2060) */
int hdk_vec_random(double *x_d, int64_t n, int64_t global_offset, int seed);

/* ---- matrix (reference: HYPRE_IJMatrixCreate/SetValues/Assemble,
 *      src/internal/linsys.c:1287-1388; HYPREDRV_LinearSystemSetMatrixFromCSR, src/HYPREDRV.c:2141) */
/* Build the rank-local ParCSR from host CSR with GLOBAL 64-bit columns.  Rows
 * [row_start,row_end] inclusive; indptr[0] may be a non-zero offset.  The diagonal entry is
 * swapped to the front of each row as hypre's IJ assembly does. */
int hdk_csr_from_host(int64_t row_start, int64_t row_end, int64_t global_rows,
                      const int64_t *indptr_h, const int64_t *cols_h, const double *vals_h,
                      hdk_csr **A);
/* Same, from arrays already resident on the device (device-side assembly path). */
int hdk_csr_from_device(int64_t row_start, int64_t row_end, int64_t global_rows,
                        const int64_t *indptr_d, const int64_t *cols_d, const double *vals_d,
                        hdk_csr **A);
int hdk_csr_destroy(hdk_csr *A);
int hdk_csr_info(const hdk_csr *A, int64_t *local_rows, int64_t *global_rows,
                 int64_t *local_nnz, int64_t *global_nnz);
/* copy the local diag block back in storage order (host buffers sized by hdk_csr_info) */
int hdk_csr_get_diag(const hdk_csr *A, int32_t *rowptr_h, int32_t *col_h, double *val_h);

/* y = alpha*A*x + beta*y with halo exchange (reference: HYPRE_ParCSRMatrixMatvec,
 * src/internal/linsys.c:1835, 3031). x_d, y_d hold the rank-local slices. */
int hdk_csr_matvec(const hdk_csr *A, double alpha, const double *x_d, double beta, double *y_d);
/* r = b - A x (reference: hypredrv_LinearSystemComputeResidualNorm, src/internal/linsys.c:3030-3032) */
int hdk_csr_residual(const hdk_csr *A, const double *x_d, const double *b_d, double *r_d);
/* which SpMV kernel the row-length statistics selected: 0 = stream (short rows),
 * 1 = warp-per-row vector kernel; also returns the statistics */
int hdk_csr_spmv_kind(const hdk_csr *A, int *kind, double *avg_row, int *max_row);

/* ---- synthetic stencil assembly on the device (reference generators:
 *      examples/src/C_laplacian/laplacian.c:720-921, 1138-1356; C_convdif/convdif.c:782-990).
 * kind: 7 = 7-pt Laplacian, 27 = 27-pt Laplacian, 107 = upwind convection-diffusion.
 * The global grid nx*ny*nz is numbered x-fastest; this rank owns rows [row_start,row_end].
 * c = {cx,cy,cz} (Laplacians) or {kappa,umax,dt} (conv-diff).  b_d receives the RHS. */
int hdk_csr_stencil(int kind, int nx, int ny, int nz, const double c[3], int64_t row_start,
                    int64_t row_end, hdk_csr **A, double *b_d);

/* ---- BoomerAMG (reference: hypredrv_AMGCreate, src/internal/amg.c:863-1035;
 *      HYPRE_BoomerAMGSetup/Solve, src/internal/precon.c:107-108) */
typedef struct
{
   int    coarsen_type;    /* 8 = PMIS (the device coarsening); 10 (HMIS) is mapped to PMIS */
   double strong_th;       /* 0.25 */
   double max_row_sum;     /* 0.9 */
   int    max_coarse_size; /* 64 */
   int    min_coarse_size; /* 0 */
   int    max_levels;      /* 25 */
   int    interp_type;     /* 6 = extended+i */
   int    max_nnz_row;     /* 4 */
   double trunc_factor;    /* 0 */
   int    relax_down, relax_up, relax_coarse; /* 18 l1-Jacobi, 7 Jacobi, 11/12 two-stage GS, 16 Chebyshev, 9 GE */
   int    sweeps_down, sweeps_up, sweeps_coarse;
   double relax_weight, outer_weight;
   int    rand_seed;       /* 2747 */
   int    keep_transpose;  /* 1: store R = P^T explicitly */
   int    print_level;
   /* systems AMG, unknown approach (hypre num_functions / dof_func): > 1 keeps strength and
    * interpolation inside each function.  dof_func: host array of this rank's row labels in
    * [0, num_functions), read during the setup only; NULL = interleaved (global row % num_functions) */
   int            num_functions; /* 1 */
   const int32_t *dof_func;      /* NULL */
   /* aggressive coarsening (hypre agg_num_levels ...): on levels l < agg_num_levels a second PMIS
    * stage runs on the C points over the paths of length <= 2 (at least agg_num_paths of them), and
    * P is multipass interpolation (agg_interp_type 4, the only type with a device kernel), each pass
    * truncated by agg_trunc_factor / agg_max_nnz_row (0: no limit).  Needs num_functions == 1. */
   int    agg_num_levels;   /* 0 */
   int    agg_num_paths;    /* 1 */
   int    agg_interp_type;  /* 4 = multipass */
   int    agg_max_nnz_row;  /* 0 */
   double agg_trunc_factor; /* 0 */
   /* Chebyshev smoothing (relax 16, hypre HYPRE_BoomerAMGSetCheby*): per level, the eigenvalue bounds of
    * C A (C = D^{-1}, D = diag|a_ii|, when scaled; C = I otherwise) from cheby_eig_est CG-Lanczos steps
    * (0: Gershgorin bounds), the interval [lower, 1.1 max] with lower = min + fraction (1.1 max - min),
    * and the monomial coefficients of the order-cheby_order polynomial; rule in DESIGN.md section 4 */
   int    cheby_order;     /* 2: passes over A per sweep, 1..4 */
   double cheby_fraction;  /* 0.3: (0, 1] */
   int    cheby_eig_est;   /* 10: CG steps of the eigenvalue estimate, 0 = Gershgorin */
   int    cheby_variant;   /* 0 (1 has no device implementation and is rejected) */
   int    cheby_scale;     /* 1: smooth with D^{-1/2} A D^{-1/2}; 0: with A */
} hdk_amg_params;

void hdk_amg_default_params(hdk_amg_params *p);
int  hdk_amg_setup(const hdk_csr *A, const hdk_amg_params *p, hdk_amg **M);
int  hdk_amg_destroy(hdk_amg *M);
/* z = M^{-1} r : one V-cycle from a zero initial guess (reference: PreconSolveDispatch,
 * src/internal/solver.c:314-329; HYPREDRV_PreconApply, src/HYPREDRV.c:3345) */
int  hdk_amg_apply(hdk_amg *M, const double *r_d, double *z_d);
/* one V-cycle from the initial guess held in u_d */
int  hdk_amg_vcycle(hdk_amg *M, const double *f_d, double *u_d);

/* hierarchy introspection (parity tests, statistics) */
int hdk_amg_num_levels(const hdk_amg *M);
int hdk_amg_num_dist_levels(const hdk_amg *M); /* N > 1: leading levels that are row-distributed (the rest is replicated) */
int hdk_amg_level_info(const hdk_amg *M, int level, int64_t *rows, int64_t *nnz_A, int64_t *nnz_P);
/* which: 0 = A_l, 1 = P_l, 2 = R_l, 3 = S_l (pattern; val_h may be NULL) -- local diag block;
 * 4 = S2_l, the second-stage strength of an aggressive level over its first-stage C points (pattern,
 * amg_keep_debug only, like S_l).  col_h == NULL copies the row pointers alone (S2 can hold more
 * entries than A_l, so a caller sizes the column buffer from them). */
int hdk_amg_get_matrix(const hdk_amg *M, int level, int which, int32_t *rowptr_h,
                       int32_t *col_h, double *val_h);
/* N > 1 (row-distributed setup), tunable amg_keep_debug set before the setup: this rank's rows of
 * A_l (which = 0) or P_l (which = 1) with GLOBAL 64-bit columns in the serial storage order, so the
 * slabs of all ranks concatenate to the one-rank matrix.  Any output pointer may be NULL. */
int hdk_amg_get_rows(const hdk_amg *M, int level, int which, int64_t *row0, int64_t *nrows, int64_t *nnz,
                     int64_t *indptr_h, int64_t *cols_h, double *vals_h);
int hdk_amg_get_cf(const hdk_amg *M, int level, int32_t *cf_h);
/* function labels of this rank's rows of level l (hierarchies built with num_functions > 1) */
int hdk_amg_get_dof_func(const hdk_amg *M, int level, int32_t *dof_h);
int hdk_amg_get_measure(const hdk_amg *M, int level, double *measure_h);
int hdk_amg_get_l1(const hdk_amg *M, int level, double *l1_h);
/* Chebyshev data of level l (a level whose sweeps use relax 16): eig_h[0] = max_eig, eig_h[1] = min_eig,
 * coefs_h[0..cheby_order) the polynomial coefficients c_0.., ds_h (may be NULL) this rank's D^{-1/2}
 * (all ones when cheby_scale = 0) */
int hdk_amg_get_cheby(const hdk_amg *M, int level, double *eig_h, double *coefs_h, double *ds_h);
double hdk_amg_operator_complexity(const hdk_amg *M);
/* algorithmic HBM bytes moved by one V-cycle (sum over levels, see DESIGN.md) */
double hdk_amg_vcycle_bytes(const hdk_amg *M);

/* stand-alone setup stages (parity tests against the oracle, one rank) */
int hdk_amg_strength(const hdk_csr *A, double theta, double max_row_sum, int64_t *nnz_S,
                     int32_t **rowptr_d, int32_t **col_d);
int hdk_amg_pmis(int64_t n, const int32_t *S_rowptr_d, const int32_t *S_col_d, int seed,
                 int64_t global_offset, int32_t *cf_d, double *measure_d, int *iterations);
int hdk_free_device(void *p_d);
int hdk_copy_d2h(void *dst_h, const void *src_d, size_t bytes);
int hdk_copy_h2d(void *dst_d, const void *src_h, size_t bytes);
int hdk_malloc_device(void **p_d, size_t bytes);

/* ---- Krylov (reference: HYPRE_ParCSRPCGSolve / HYPRE_ParCSRGMRESSolve,
 *      src/internal/solver.c:211, 223, 614; options src/internal/pcg.c:15-25, gmres.c:16-27) */
typedef struct
{
   int    max_iter;
   double rel_tol, abs_tol;
   int    krylov_dim;          /* GMRES restart length */
   int    min_iter;            /* GMRES */
   int    skip_real_res_check; /* GMRES */
   /* results */
   int    iters, converged;
   double rel_res_norm;        /* recurrence residual norm / ||b|| */
   double solve_ms;            /* CUDA-event time of the solve region */
} hdk_krylov;

int hdk_pcg(const hdk_csr *A, hdk_amg *M /* NULL: none */, const double *b_d, double *x_d,
            hdk_krylov *k);
int hdk_gmres(const hdk_csr *A, hdk_amg *M, const double *b_d, double *x_d, hdk_krylov *k);
/* "next" row 8f-3: the other Krylov callers of the same kernels (reference src/internal/solver.c:229-252) */
int hdk_fgmres(const hdk_csr *A, hdk_amg *M, const double *b_d, double *x_d, hdk_krylov *k);
int hdk_bicgstab(const hdk_csr *A, hdk_amg *M, const double *b_d, double *x_d, hdk_krylov *k);

/* ---- measurement helpers: average kernel time in ms over `reps` back-to-back launches of
 * one hot kernel on the compute stream, CUDA-event timed (bench.py roofline leg).
 * kernel: 0 = SpMV y=Ax, 1 = l1-Jacobi sweep fused with residual, 2 = residual r=b-Ax,
 *         3 = PCG fused x/r update + <r,r> + first V-cycle sweep (the 64 B/row variant the solve runs),
 *         4 = V-cycle, 5 = PCG p = z + beta p, 6 = one fused two-stage Gauss-Seidel sweep (relax 11/12),
 *         9 = one Chebyshev sweep (relax 16) on the fine level of M */
int hdk_time_kernel(const hdk_csr *A, hdk_amg *M, int kernel, int reps, double *avg_ms,
                    double *algorithmic_bytes);
/* number of kernel launches issued by this library since the last call (and reset) */
int64_t hdk_launch_count_reset(void);
/* kernel-selection tunables for matrices analysed after the call (same names as the HDK_*
 * environment variables, lower case without the prefix): spmv_rows_mult, spmv_tgt_max, spmv_lpr,
 * sell_min_rows, sell_min_rows_dist, sell_min_avg, sell_sort, export_max_rows (N > 1: operators with more
 * rows pack their halo instead of folding the export into the producer), graph_rows (V-cycle levels with at most
 * this many rows are replayed from a CUDA graph; 0 = off), replicate_rows (N > 1: levels with
 * at most this many global rows are replicated on every rank), amg_keep_debug (keep the strength
 * pattern and PMIS measures of every level for hdk_amg_get_matrix(...,'S') / get_measure).
 * Unknown key -> HDK_ERR_INVALID. */
int hdk_tune(const char *key, double value);
/* cudaProfilerStart (1) / cudaProfilerStop (0) for `ncu --profile-from-start off` */
int hdk_profiler_range(int start);

#ifdef __cplusplus
}
#endif
#endif
