/* hd_api.c -- the HYPREDRV_* public API of hypredrive_b200 (plain C host code).
 * Re-implements the lifecycle subset of the reference's src/HYPREDRV.c for the hot path
 * (citations per function) on top of the hdk_* device C-ABI.  All numerical work happens in
 * CUDA kernels; this file only validates, tracks ownership/state and keeps statistics. */
#include "hd_internal.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define HD_OBJ_MAGIC 0x48445256u
#define HD_MAX_LIVE 256

struct hypredrv_struct
{
   uint32_t  magic;
   MPI_Comm  comm;
   int       rank, nprocs;
   bool      lib_mode;
   hd_args  *args;
   hdk_csr  *A;
   hdk_csr  *A_prec;  /* preconditioner reuse: the (older) matrix the live hierarchy was built on */
   int       ls_index; /* 0-based index of the installed linear system (-1: none yet) */
   int64_t   row_start, row_end, n;
   double   *b_d, *x0_d, *x_d;
   double   *x_prev_d;            /* solution of the system that was replaced (init_guess_mode previous) */
   int64_t   x_prev_rs, x_prev_re;
   double   *x_host, *b_host;
   hdk_amg  *precon;
   bool      precon_created, precon_is_setup, solver_created;
   hd_stats *stats;
   int       iters, converged;
   double    final_res, setup_time, solve_time;
   double    pending_build;
   bool      have_pending_build;
   struct hypre_IJVector_struct *sol_handle, *rhs_handle;
};

static bool       g_initialized = false;
static HYPREDRV_t g_live[HD_MAX_LIVE];

/* ------------------------------------------------------------------------------------- */
static uint32_t fail(uint32_t bit, const char *fmt, const char *arg)
{
   hd_err_set(bit);
   if (fmt) hd_err_msg(fmt, arg ? arg : "");
   return hd_err_get();
}

static uint32_t hdk_fail(int rc)
{
   if (rc == HDK_OK) return hd_err_get();
   hd_err_set(rc == HDK_ERR_ALLOC ? HYPREDRV_ERROR_ALLOCATION : HYPREDRV_ERROR_HYPRE_INTERNAL);
   hd_err_msg("hdk: %s", hdk_last_error());
   return hd_err_get();
}

static bool is_live(HYPREDRV_t h)
{
   if (!h) return false;
   for (int i = 0; i < HD_MAX_LIVE; i++)
      if (g_live[i] == h) return h->magic == HD_OBJ_MAGIC;
   return false;
}

#define CHECK_INIT()                                                                   \
   do {                                                                                \
      if (!g_initialized) return fail(HYPREDRV_ERROR_HYPREDRV_NOT_INITIALIZED, NULL, NULL); \
   } while (0)
#define CHECK_OBJ(h)                                                                   \
   do {                                                                                \
      CHECK_INIT();                                                                    \
      if (!is_live(h)) return fail(HYPREDRV_ERROR_UNKNOWN_HYPREDRV_OBJ, NULL, NULL);   \
   } while (0)
#define CHECK_ARGS(h)                                                                  \
   do {                                                                                \
      CHECK_OBJ(h);                                                                    \
      if (!(h)->args) return fail(HYPREDRV_ERROR_MISSING_KEY, "%s", "input arguments were not parsed (HYPREDRV_InputArgsParse)"); \
   } while (0)

/* ------------------------------------------------------------------------------------- */
uint32_t HYPREDRV_Initialize(void)
{
   /* reference src/HYPREDRV.c:916 -> runtime.c:101 (HYPRE_Initialize).  The device context
    * is created lazily on the first call that needs the GPU, so configuration-only use of the
    * API works on a machine without one. */
   g_initialized = true;
   return hd_err_get();
}

uint32_t HYPREDRV_Finalize(void)
{
   if (!g_initialized) return hd_err_get();
   for (int i = 0; i < HD_MAX_LIVE; i++)
      if (g_live[i]) { HYPREDRV_t h = g_live[i]; HYPREDRV_Destroy(&h); } /* leaked objects, src/HYPREDRV.c:931-943 */
   hdk_finalize();
   g_initialized = false;
   return hd_err_get();
}

void HYPREDRV_ErrorCodeDescribe(uint32_t error_code) { hd_err_describe(error_code); hd_err_clear_msgs(); }
void HYPREDRV_ErrorCodeClear(void) { hd_err_reset(); }

uint32_t HYPREDRV_ErrorInvalidValue(const char *message)
{
   hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
   if (message) hd_err_msg("%s", message);
   return hd_err_get();
}

void HYPREDRV_SafeCallHandleError(uint32_t error_code, MPI_Comm comm, const char *file, int line, const char *func)
{
   if (!error_code) return;
   fprintf(stderr, "At %s:%d in %s():\n", file, line, func);
   HYPREDRV_ErrorCodeDescribe(error_code);
   const char *dbg = getenv("HYPREDRV_DEBUG");
   if (dbg && !strcmp(dbg, "1")) { abort(); }
   int status = (int)(error_code & 0xffu);
   MPI_Abort(comm, status ? status : EXIT_FAILURE);
}

uint32_t HYPREDRV_Create(MPI_Comm comm, HYPREDRV_t *out)
{
   CHECK_INIT();
   if (!out) return fail(HYPREDRV_ERROR_UNKNOWN_HYPREDRV_OBJ, NULL, NULL);
   HYPREDRV_t h = calloc(1, sizeof(*h));
   if (!h) return fail(HYPREDRV_ERROR_ALLOCATION, NULL, NULL);
   h->magic = HD_OBJ_MAGIC;
   h->comm  = comm;
   /* several processes (launcher exported WORLD_SIZE > 1) and no communicator yet: bring NCCL up from the
    * environment, or fail clearly -- never run as N independent single-rank solves */
   if (comm != MPI_COMM_SELF && getenv("WORLD_SIZE") && atoi(getenv("WORLD_SIZE")) > 1 && hdk_comm_size() <= 1 &&
       hdk_device_count() > 0)
   {
      int rc = hdk_comm_init_from_env();
      if (rc) { free(h); return hdk_fail(rc); }
   }
   MPI_Comm_rank(comm, &h->rank);
   MPI_Comm_size(comm, &h->nprocs);
   h->stats     = hd_stats_create();
   h->ls_index  = -1;
   h->row_end   = -1;
   int slot = -1;
   for (int i = 0; i < HD_MAX_LIVE; i++) if (!g_live[i]) { slot = i; break; }
   if (slot < 0) { free(h->stats); free(h); return fail(HYPREDRV_ERROR_ALLOCATION, "%s", "too many live HYPREDRV objects"); }
   g_live[slot] = h;
   *out = h;
   return hd_err_get();
}

static void drop_precon(HYPREDRV_t h)
{
   if (h->precon) { hdk_amg_destroy(h->precon); h->precon = NULL; }
   if (h->A_prec) { hdk_csr_destroy(h->A_prec); h->A_prec = NULL; }
   h->precon_is_setup = false;
}

/* static reuse policy (reference src/internal/precon_reuse.c:780-830): may the live hierarchy
 * serve linear system `ls_id`? */
static bool precon_reusable_for(HYPREDRV_t h, int ls_id)
{
   return h->precon && h->precon_is_setup && h->args && h->args->reuse.enabled &&
          !hd_reuse_should_rebuild(&h->args->reuse, ls_id);
}

/* init_guess_mode 'previous' (reference linsys.c:2044-2063): the solution of the system that is being
 * replaced survives as the candidate initial guess of the next one */
static void stash_previous_solution(HYPREDRV_t h)
{
   if (!h->x_d || !h->args || h->args->ls.init_guess_mode != 4) return;
   if (h->x_prev_d) hdk_vec_free(h->x_prev_d);
   h->x_prev_d = h->x_d; h->x_prev_rs = h->row_start; h->x_prev_re = h->row_end;
   h->x_d = NULL;
}

static void free_system(HYPREDRV_t h)
{
   drop_precon(h);
   if (h->A) { hdk_csr_destroy(h->A); h->A = NULL; }
   if (h->b_d) { hdk_vec_free(h->b_d); h->b_d = NULL; }
   if (h->x0_d) { hdk_vec_free(h->x0_d); h->x0_d = NULL; }
   if (h->x_d) { hdk_vec_free(h->x_d); h->x_d = NULL; }
   hdk_host_free(h->x_host); h->x_host = NULL;
   hdk_host_free(h->b_host); h->b_host = NULL;
}

uint32_t HYPREDRV_Destroy(HYPREDRV_t *hp)
{
   CHECK_INIT();
   if (!hp || !is_live(*hp)) return fail(HYPREDRV_ERROR_UNKNOWN_HYPREDRV_OBJ, NULL, NULL);
   HYPREDRV_t h = *hp;
   free_system(h);
   if (h->x_prev_d) { hdk_vec_free(h->x_prev_d); h->x_prev_d = NULL; }
   if (h->sol_handle) { h->sol_handle->data = NULL; free(h->sol_handle); }
   if (h->rhs_handle) { h->rhs_handle->data = NULL; free(h->rhs_handle); }
   free(h->args);
   free(h->stats);
   for (int i = 0; i < HD_MAX_LIVE; i++) if (g_live[i] == h) g_live[i] = NULL;
   h->magic = 0;
   free(h);
   *hp = NULL;
   return hd_err_get();
}

uint32_t HYPREDRV_PrintLibInfo(MPI_Comm comm, int print_datetime)
{
   CHECK_INIT();
   int rank = 0, size = 1;
   MPI_Comm_rank(comm, &rank);
   MPI_Comm_size(comm, &size);
   if (rank == 0)
   {
      if (print_datetime)
      {
         time_t t = time(NULL);
         char   buf[64];
         strftime(buf, sizeof(buf), "%Y-%m-%d %H:%M:%S", localtime(&t));
         printf("Date and time: %s\n", buf);
      }
      printf("\nUsing HYPREDRV_DEVELOP_STRING: %s (B200-native CUDA backend, sm_100a)\n\n", HYPREDRV_RELEASE_VERSION);
      printf("Running on %d MPI rank%s\n", size, size > 1 ? "s" : "");
      fflush(stdout);
   }
   return hd_err_get();
}

uint32_t HYPREDRV_PrintSystemInfo(MPI_Comm comm)
{
   CHECK_INIT();
   int rank = 0;
   MPI_Comm_rank(comm, &rank);
   if (rank == 0) { printf("CUDA devices visible: %d\n", hdk_device_count()); fflush(stdout); }
   return hd_err_get();
}

uint32_t HYPREDRV_PrintExitInfo(MPI_Comm comm, const char *argv0)
{
   CHECK_INIT();
   int rank = 0;
   MPI_Comm_rank(comm, &rank);
   if (rank == 0)
   {
      time_t t = time(NULL);
      char   buf[64];
      strftime(buf, sizeof(buf), "%Y-%m-%d %H:%M:%S", localtime(&t));
      printf("Date and time: %s\n%s done!\n", buf, argv0 ? argv0 : "hypredrive");
      fflush(stdout);
   }
   return hd_err_get();
}

/* ---- configuration ------------------------------------------------------------------- */
static bool looks_like_yaml_text(const char *s)
{
   /* inline YAML: contains a newline or a "key:" pattern (reference args.c:1294-1313) */
   if (strchr(s, '\n')) return true;
   const char *c = strchr(s, ':');
   size_t      n = strlen(s);
   bool        file_ext = (n > 4 && (!strcmp(s + n - 4, ".yml") || (n > 5 && !strcmp(s + n - 5, ".yaml"))));
   return c != NULL && !file_ext;
}

uint32_t HYPREDRV_InputArgsParse(int argc, char **argv, HYPREDRV_t h)
{
   CHECK_OBJ(h);
   if (argc < 1 || !argv || !argv[0]) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "no configuration given");
   /* find the configuration source: argv[0] (library / legacy form) or the first *.yml token
    * before -a/--args (driver form) */
   int cfg = 0;
   if (!looks_like_yaml_text(argv[0]))
   {
      size_t n0 = strlen(argv[0]);
      bool   is_file = (n0 > 4 && (!strcmp(argv[0] + n0 - 4, ".yml") || (n0 > 5 && !strcmp(argv[0] + n0 - 5, ".yaml"))));
      if (!is_file)
         for (int i = 1; i < argc; i++)
         {
            if (!strcmp(argv[i], "-a") || !strcmp(argv[i], "--args")) break;
            size_t n = strlen(argv[i]);
            if (n > 4 && (!strcmp(argv[i] + n - 4, ".yml") || (n > 5 && !strcmp(argv[i] + n - 5, ".yaml")))) { cfg = i; break; }
         }
   }
   char *text = NULL, dir[2048] = ".";
   if (looks_like_yaml_text(argv[cfg])) text = strdup(argv[cfg]);
   else
   {
      FILE *fp = fopen(argv[cfg], "rb");
      if (!fp) return fail(HYPREDRV_ERROR_FILE_NOT_FOUND, "cannot open configuration file '%s'", argv[cfg]);
      fseek(fp, 0, SEEK_END);
      long sz = ftell(fp);
      fseek(fp, 0, SEEK_SET);
      text = malloc((size_t)sz + 1);
      size_t rd = fread(text, 1, (size_t)sz, fp);
      text[rd] = 0;
      fclose(fp);
      snprintf(dir, sizeof(dir), "%s", argv[cfg]);
      char *slash = strrchr(dir, '/');
      if (slash) *slash = 0; else strcpy(dir, ".");
   }
   hd_args *a = hd_args_parse(text, dir, argc - cfg - 1, argv + cfg + 1, h->lib_mode, h->rank == 0);
   free(text);
   if (!a) return hd_err_get();
   free(h->args);
   h->args = a;
   h->stats->use_millisec = a->general.use_millisec;
   snprintf(h->stats->name, sizeof(h->stats->name), "%s", a->general.name);
   return hd_err_get();
}

uint32_t HYPREDRV_SetLibraryMode(HYPREDRV_t h)
{
   CHECK_OBJ(h);
   h->lib_mode = true;
   if (h->args) { h->args->lib_mode = true; h->args->general.print_config_params = 0; }
   return hd_err_get();
}

uint32_t HYPREDRV_ObjectSetName(HYPREDRV_t h, const char *name)
{
   CHECK_OBJ(h);
   snprintf(h->stats->name, sizeof(h->stats->name), "%s", name ? name : "");
   return hd_err_get();
}

uint32_t HYPREDRV_InputArgsGetWarmup(HYPREDRV_t h, int *v) { CHECK_ARGS(h); if (v) *v = h->args->general.warmup; return hd_err_get(); }
uint32_t HYPREDRV_InputArgsGetNumRepetitions(HYPREDRV_t h, int *v) { CHECK_ARGS(h); if (v) *v = h->args->general.num_repetitions; return hd_err_get(); }
uint32_t HYPREDRV_InputArgsGetNumLinearSystems(HYPREDRV_t h, int *v) { CHECK_ARGS(h); if (v) *v = h->args->ls.num_systems; return hd_err_get(); }
uint32_t HYPREDRV_InputArgsGetNumPreconVariants(HYPREDRV_t h, int *v) { CHECK_ARGS(h); if (v) *v = h->args->num_precon_variants; return hd_err_get(); }

uint32_t HYPREDRV_InputArgsSetPreconVariant(HYPREDRV_t h, int idx)
{
   CHECK_ARGS(h);
   if (idx < 0 || idx >= h->args->num_precon_variants) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "preconditioner variant index out of range");
   h->args->active_precon_variant = idx;
   return hd_err_get();
}

static void ensure_args(HYPREDRV_t h)
{
   if (!h->args)
   {
      h->args = calloc(1, sizeof(hd_args));
      hd_args_defaults(h->args, h->lib_mode);
   }
}

uint32_t HYPREDRV_InputArgsSetPreconPreset(HYPREDRV_t h, const char *preset)
{
   CHECK_OBJ(h);
   if (!preset) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "Preconditioner preset name cannot be NULL");
   ensure_args(h);
   drop_precon(h); h->precon_created = false;
   hd_args_apply_precon_preset(h->args, preset);
   return hd_err_get();
}

uint32_t HYPREDRV_InputArgsSetSolverPreset(HYPREDRV_t h, const char *preset)
{
   CHECK_OBJ(h);
   if (!preset) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "Solver preset name cannot be NULL");
   ensure_args(h);
   hd_args_apply_solver_preset(h->args, preset);
   return hd_err_get();
}

uint32_t HYPREDRV_SolverPresetRegister(const char *name, const char *yaml_text, const char *help)
{
   if (hd_preset_register(1, name, yaml_text, help)) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "invalid solver preset");
   return hd_err_get();
}
uint32_t HYPREDRV_PreconPresetRegister(const char *name, const char *yaml_text, const char *help)
{
   if (hd_preset_register(0, name, yaml_text, help)) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "invalid preconditioner preset");
   return hd_err_get();
}

/* ---- linear system ------------------------------------------------------------------- */
static uint32_t read_vector_into(HYPREDRV_t h, const char *fname, double **dst);
static uint32_t alloc_vec(double **p, int64_t n);

static void build_timer_add(HYPREDRV_t h, double t0)
{
   hdk_sync();
   h->pending_build += hd_wtime() - t0;
   h->have_pending_build = true;
}

static uint32_t install_matrix(HYPREDRV_t h, hdk_csr *A, int64_t rs, int64_t re)
{
   const int next = h->ls_index + 1;
   stash_previous_solution(h);
   if (precon_reusable_for(h, next) && h->row_start == rs && h->row_end == re)
   {
      /* keep the hierarchy (and the matrix its level 0 refers to) for the new system */
      hdk_amg  *M = h->precon;
      hdk_csr  *Ap = h->A_prec ? h->A_prec : h->A;
      if (h->A_prec) hdk_csr_destroy(h->A);
      h->A = NULL; h->precon = NULL; h->A_prec = NULL;
      free_system(h);
      h->precon = M; h->A_prec = Ap; h->precon_is_setup = true;
      h->A = A; h->row_start = rs; h->row_end = re; h->n = re - rs + 1;
      h->ls_index = next;
      return hd_err_get();
   }
   free_system(h);
   h->A = A; h->row_start = rs; h->row_end = re; h->n = re - rs + 1;
   h->precon_created = false; h->solver_created = false;
   h->ls_index = next;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetMatrixFromCSR(HYPREDRV_t h, HYPRE_BigInt row_start, HYPRE_BigInt row_end,
                                               const HYPRE_BigInt *indptr, const HYPRE_BigInt *col_indices,
                                               const HYPRE_Real *data)
{
   /* reference src/HYPREDRV.c:2141-2191 -> src/internal/linsys.c:1190-1405 */
   CHECK_OBJ(h);
   if (!indptr) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "indptr cannot be NULL");
   if (row_end < row_start) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "row_end must be >= row_start");
   /* row and entry counts must fit HYPRE_Int (32 bit here), reference linsys.c:1226-1262; checked
    * before indptr[n] is touched (tests/test_setmatrix_from_csr.c:373-384 passes a 2-entry indptr) */
   if ((long long)row_end - (long long)row_start >= 2147483647LL)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "local row count does not fit HYPRE_Int");
   int64_t n = (int64_t)(row_end - row_start + 1);
   if (indptr[0] < 0) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "indptr[0] must be nonnegative");
   if (n == 1 && (long long)indptr[1] - (long long)indptr[0] > 2147483647LL)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "local nonzero count does not fit HYPRE_Int");
   for (int64_t i = 0; i < n; i++)
      if (indptr[i + 1] < indptr[i]) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "indptr must be nondecreasing");
   if ((long long)indptr[n] - (long long)indptr[0] > 2147483647LL)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "local nonzero count does not fit HYPRE_Int");
   if (indptr[n] > indptr[0] && (!col_indices || !data))
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "col_indices and data cannot be NULL when nnz > 0");
   double   t0 = hd_wtime();
   int64_t  grows = 0;
   int      rc = hdk_init(-1);
   if (rc) return hdk_fail(rc);
   rc = hdk_comm_max_i64((int64_t)row_end + 1, &grows);
   if (rc) return hdk_fail(rc);
   hdk_csr *A = NULL;
   rc = hdk_csr_from_host(row_start, row_end, grows, (const int64_t *)indptr, (const int64_t *)col_indices, data, &A);
   if (rc) return hdk_fail(rc);
   install_matrix(h, A, row_start, row_end);
   build_timer_add(h, t0);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetMatrix(HYPREDRV_t h, HYPRE_Matrix mat_A)
{
   /* reference src/HYPREDRV.c:1998-2017: adopt a caller-built IJ matrix (NULL: read from file) */
   CHECK_OBJ(h);
   struct hypre_IJMatrix_struct *ij = (struct hypre_IJMatrix_struct *)mat_A;
   if (!ij) return HYPREDRV_LinearSystemReadMatrix(h);
   if (ij->magic != HD_IJMAT_MAGIC) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "matrix handle is not a HYPRE_IJMatrix");
   if (hd_ij_matrix_flatten(ij)) return fail(HYPREDRV_ERROR_ALLOCATION, NULL, NULL);
   return HYPREDRV_LinearSystemSetMatrixFromCSR(h, ij->ilower, ij->iupper, (const HYPRE_BigInt *)ij->indptr, ij->cols, ij->vals);
}

uint32_t HYPREDRV_LinearSystemSetStencil(HYPREDRV_t h, int kind, int nx, int ny, int nz, const double *c,
                                         HYPRE_BigInt row_start, HYPRE_BigInt row_end)
{
   CHECK_OBJ(h);
   if (!c || nx < 1 || ny < 1 || nz < 1) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "invalid stencil arguments");
   if (row_end < row_start) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "row_end must be >= row_start");
   double t0 = hd_wtime();
   int    rc = hdk_init(-1);
   if (rc) return hdk_fail(rc);
   double *b = NULL;
   rc = hdk_vec_alloc(row_end - row_start + 1, &b);
   if (rc) return hdk_fail(rc);
   hdk_csr *A = NULL;
   rc = hdk_csr_stencil(kind, nx, ny, nz, c, row_start, row_end, &A, b);
   if (rc) { hdk_vec_free(b); return hdk_fail(rc); }
   install_matrix(h, A, row_start, row_end);
   h->b_d = b;
   build_timer_add(h, t0);
   return hd_err_get();
}

static uint32_t alloc_vec(double **p, int64_t n)
{
   if (*p) return hd_err_get();
   int rc = hdk_vec_alloc(n, p);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetRHSFromArray(HYPREDRV_t h, HYPRE_BigInt row_start, HYPRE_BigInt row_end, const HYPRE_Real *values)
{
   /* reference src/HYPREDRV.c:2198-2255 */
   CHECK_OBJ(h);
   if (row_end < row_start) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "row_end must be >= row_start");
   if (!values) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "values cannot be NULL");
   if (!h->A) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "the matrix must be set before the right-hand side");
   if (row_start != h->row_start || row_end != h->row_end)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "RHS row range must match the matrix row range");
   double t0 = hd_wtime();
   if (alloc_vec(&h->b_d, h->n)) return hd_err_get();
   int rc = hdk_vec_h2d(h->b_d, values, h->n);
   if (rc) return hdk_fail(rc);
   build_timer_add(h, t0);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetRHS(HYPREDRV_t h, HYPRE_Vector vec)
{
   /* reference src/HYPREDRV.c:2101-2134; NULL -> generated RHS per linear_system.rhs_mode
    * (src/internal/linsys.c:1778-1840) */
   CHECK_OBJ(h);
   struct hypre_IJVector_struct *v = (struct hypre_IJVector_struct *)vec;
   if (v)
   {
      if (v->magic != HD_IJVEC_MAGIC) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "vector handle is not a HYPRE_IJVector");
      return HYPREDRV_LinearSystemSetRHSFromArray(h, v->jlower, v->jupper, v->data);
   }
   if (!h->A) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "the matrix must be set before the right-hand side");
   int mode = h->args ? h->args->ls.rhs_mode : 2;
   if (mode == 2)
   {
      if (h->args && h->args->ls.rhs_filename[0])
      {
         double   t0 = hd_wtime();
         uint32_t e = read_vector_into(h, h->args->ls.rhs_filename, &h->b_d);
         if (!e) build_timer_add(h, t0);
         return e;
      }
      if (h->b_d) return hd_err_get(); /* e.g. installed together with a device stencil */
      return fail(HYPREDRV_ERROR_FILE_NOT_FOUND, "%s", "rhs_mode 'file' but linear_system.rhs_filename is empty");
   }
   double t0 = hd_wtime();
   if (alloc_vec(&h->b_d, h->n)) return hd_err_get();
   int rc = HDK_OK;
   if (mode == 0) rc = hdk_vec_fill(h->b_d, 0.0, h->n);
   else if (mode == 1) rc = hdk_vec_fill(h->b_d, 1.0, h->n);
   else if (mode == 3) rc = hdk_vec_random(h->b_d, h->n, h->row_start, 2023);
   else
   {
      double *xr = NULL; /* randsol: b = A * x_rand */
      rc = hdk_vec_alloc(h->n, &xr);
      if (!rc) rc = hdk_vec_random(xr, h->n, h->row_start, 2023);
      if (!rc) rc = hdk_csr_matvec(h->A, 1.0, xr, 0.0, h->b_d);
      hdk_vec_free(xr);
   }
   if (rc) return hdk_fail(rc);
   build_timer_add(h, t0);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetInitialGuess(HYPREDRV_t h, HYPRE_Vector vec)
{
   /* reference src/HYPREDRV.c:2333-2368 -> src/internal/linsys.c:1974-2104: builds x0 per
    * init_guess_mode and a zeroed working solution */
   CHECK_OBJ(h);
   if (!h->A) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "the matrix must be set before the initial guess");
   const bool had_x = (h->x_d != NULL); /* a solve of THIS system already produced a solution */
   if (alloc_vec(&h->x0_d, h->n) || alloc_vec(&h->x_d, h->n)) return hd_err_get();
   int rc = HDK_OK;
   struct hypre_IJVector_struct *v = (struct hypre_IJVector_struct *)vec;
   if (v)
   {
      if (v->magic != HD_IJVEC_MAGIC || v->n != h->n) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "initial guess vector does not match the system");
      rc = hdk_vec_h2d(h->x0_d, v->data, h->n);
   }
   else
   {
      int mode = h->args ? h->args->ls.init_guess_mode : 0;
      if (mode == 1) rc = hdk_vec_fill(h->x0_d, 1.0, h->n);
      else if (mode == 3) rc = hdk_vec_random(h->x0_d, h->n, h->row_start, 2023);
      else if (mode == 4)
      {
         /* previous solution: of this system if it was solved before, else of the system it replaced
          * when the row range is the same; otherwise zeros (reference linsys.c:2044-2063) */
         if (had_x) rc = hdk_vec_copy(h->x0_d, h->x_d, h->n);
         else if (h->x_prev_d && h->x_prev_rs == h->row_start && h->x_prev_re == h->row_end) rc = hdk_vec_copy(h->x0_d, h->x_prev_d, h->n);
         else rc = hdk_vec_fill(h->x0_d, 0.0, h->n); /* no compatible previous solution; using zeros */
      }
      else if (mode == 2)
      {
         if (!h->args->ls.x0_filename[0]) return fail(HYPREDRV_ERROR_FILE_NOT_FOUND, "%s", "init_guess_mode 'file' but linear_system.x0_filename is empty");
         uint32_t e = read_vector_into(h, h->args->ls.x0_filename, &h->x0_d);
         if (e) return e;
      }
      else rc = hdk_vec_fill(h->x0_d, 0.0, h->n);
   }
   if (!rc && (!h->args || h->args->ls.init_guess_mode != 4)) rc = hdk_vec_fill(h->x_d, 0.0, h->n);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetSolution(HYPREDRV_t h, HYPRE_Vector vec)
{
   CHECK_OBJ(h);
   if (!h->A) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "the matrix must be set first");
   if (alloc_vec(&h->x_d, h->n)) return hd_err_get();
   struct hypre_IJVector_struct *v = (struct hypre_IJVector_struct *)vec;
   int rc = v ? hdk_vec_h2d(h->x_d, v->data, h->n) : hdk_vec_fill(h->x_d, 0.0, h->n);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_LinearSystemResetInitialGuess(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:2454 -> src/internal/linsys.c:2185-2227: x <- x0 */
   CHECK_OBJ(h);
   if (!h->x_d || !h->x0_d)
   {
      uint32_t e = HYPREDRV_LinearSystemSetInitialGuess(h, NULL);
      if (e) return e;
   }
   int rc = hdk_vec_copy(h->x_d, h->x0_d, h->n);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_LinearSystemSetPrecMatrix(HYPREDRV_t h, HYPRE_Matrix mat)
{
   CHECK_OBJ(h);
   if (mat && (void *)mat != (void *)h->A)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "a preconditioning matrix different from A is not supported on the B200 path");
   return hd_err_get(); /* NULL => M := A (reference src/HYPREDRV.c) */
}

uint32_t HYPREDRV_LinearSystemBuild(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:1933-1990 (file-driven) */
   CHECK_ARGS(h);
   uint32_t e = HYPREDRV_LinearSystemReadMatrix(h);
   if (e) return e;
   if ((e = HYPREDRV_LinearSystemSetRHS(h, NULL))) return e;
   if ((e = HYPREDRV_LinearSystemSetInitialGuess(h, NULL))) return e;
   return HYPREDRV_LinearSystemSetPrecMatrix(h, NULL);
}

static void join_path(char *out, size_t cap, const char *dir, const char *name)
{
   if (dir && dir[0] && name[0] != '/') snprintf(out, cap, "%s/%s", dir, name);
   else snprintf(out, cap, "%s", name);
}

uint32_t HYPREDRV_LinearSystemReadMatrix(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:1940 -> linsys.c:946-977: IJ parts "<name>.%05d[.bin]" */
   CHECK_ARGS(h);
   if (!h->args->ls.matrix_filename[0]) return fail(HYPREDRV_ERROR_FILE_NOT_FOUND, "%s", "linear_system.matrix_filename is empty");
   char path[2048];
   join_path(path, sizeof(path), h->args->ls.dirname, h->args->ls.matrix_filename);
   double         t0 = hd_wtime();
   HYPRE_IJMatrix ij = NULL;
   if (hd_read_ij_matrix(path, h->rank, &ij)) return hd_err_get();
   if (hd_ij_matrix_flatten(ij)) { HYPRE_IJMatrixDestroy(ij); return fail(HYPREDRV_ERROR_ALLOCATION, NULL, NULL); }
   uint32_t e = HYPREDRV_LinearSystemSetMatrixFromCSR(h, ij->ilower, ij->iupper, (const HYPRE_BigInt *)ij->indptr, ij->cols, ij->vals);
   HYPRE_IJMatrixDestroy(ij);
   if (e) return e;
   h->pending_build += hd_wtime() - t0 - 0.0; /* file parsing counts as LS build time */
   if (h->rank == 0)
   {
      int64_t lr, gr, ln, gn;
      hdk_csr_info(h->A, &lr, &gr, &ln, &gn);
      printf("====================================================================================\n");
      printf("Solving linear system #%d with %lld rows and %lld nonzeros...\n", h->stats->ls_id + 1, (long long)gr, (long long)gn);
      /* the closing rule is printed by the statistics summary (reference stats.c:1231) */
      fflush(stdout);
   }
   h->stats->ls_id++;
   return hd_err_get();
}

static uint32_t read_vector_into(HYPREDRV_t h, const char *fname, double **dst)
{
   char path[2048];
   join_path(path, sizeof(path), h->args->ls.dirname, fname);
   HYPRE_IJVector v = NULL;
   if (hd_read_ij_vector(path, h->rank, &v)) return hd_err_get();
   if (v->n != h->n) { HYPRE_IJVectorDestroy(v); return fail(HYPREDRV_ERROR_FILE_UNEXPECTED_ENTRY, "vector file %s does not match the matrix row range", path); }
   if (alloc_vec(dst, h->n)) { HYPRE_IJVectorDestroy(v); return hd_err_get(); }
   int rc = hdk_vec_h2d(*dst, v->data, h->n);
   HYPRE_IJVectorDestroy(v);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetSolutionValues(HYPREDRV_t h, HYPRE_Complex **sol_data)
{
   /* reference src/HYPREDRV.c:2479-2492: library-owned HOST pointer */
   CHECK_OBJ(h);
   if (!sol_data) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "sol_data cannot be NULL");
   if (!h->x_d) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "no solution vector is available");
   int rc = h->x_host ? HDK_OK : hdk_host_alloc(sizeof(double) * (size_t)(h->n > 0 ? h->n : 1), (void **)&h->x_host);
   if (!rc) rc = hdk_vec_d2h(h->x_host, h->x_d, h->n);
   if (rc) return hdk_fail(rc);
   *sol_data = h->x_host;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetRHSValues(HYPREDRV_t h, HYPRE_Complex **rhs_data)
{
   CHECK_OBJ(h);
   if (!rhs_data) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "rhs_data cannot be NULL");
   if (!h->b_d) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "no right-hand side is available");
   int rc = h->b_host ? HDK_OK : hdk_host_alloc(sizeof(double) * (size_t)(h->n > 0 ? h->n : 1), (void **)&h->b_host);
   if (!rc) rc = hdk_vec_d2h(h->b_host, h->b_d, h->n);
   if (rc) return hdk_fail(rc);
   *rhs_data = h->b_host;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetSolutionLength(HYPREDRV_t h, HYPRE_BigInt *length)
{
   CHECK_OBJ(h);
   if (!length) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "length cannot be NULL");
   *length = h->A ? (HYPRE_BigInt)h->n : 0;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetSolutionNorm(HYPREDRV_t h, const char *norm_type, double *norm)
{
   /* reference src/HYPREDRV.c:2505-2561 -> src/internal/linsys.c:2815-2924 */
   CHECK_OBJ(h);
   if (!norm_type || !norm) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "norm_type and norm cannot be NULL");
   if (!h->x_d) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "no solution vector is available");
   int kind;
   if (!strcmp(norm_type, "L1") || !strcmp(norm_type, "l1")) kind = 0;
   else if (!strcmp(norm_type, "L2") || !strcmp(norm_type, "l2")) kind = 1;
   else if (!strcmp(norm_type, "inf") || !strcmp(norm_type, "Linf") || !strcmp(norm_type, "linf")) kind = 2;
   else return fail(HYPREDRV_ERROR_INVALID_VAL, "unknown norm type '%s' (L1, L2, inf)", norm_type);
   int rc = hdk_vec_norm(h->x_d, h->n, kind, norm);
   return rc ? hdk_fail(rc) : hd_err_get();
}

static struct hypre_IJVector_struct *view_handle(struct hypre_IJVector_struct **slot, HYPREDRV_t h, double *host)
{
   if (!*slot) { *slot = calloc(1, sizeof(**slot)); (*slot)->magic = HD_IJVEC_MAGIC; }
   (*slot)->jlower = h->row_start; (*slot)->jupper = h->row_end; (*slot)->n = h->n; (*slot)->data = host;
   return *slot;
}

uint32_t HYPREDRV_LinearSystemGetSolution(HYPREDRV_t h, HYPRE_Vector *vec)
{
   CHECK_OBJ(h);
   HYPRE_Complex *p;
   uint32_t       e = HYPREDRV_LinearSystemGetSolutionValues(h, &p);
   if (e) return e;
   if (vec) *vec = (HYPRE_Vector)view_handle(&h->sol_handle, h, p);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetRHS(HYPREDRV_t h, HYPRE_Vector *vec)
{
   CHECK_OBJ(h);
   HYPRE_Complex *p;
   uint32_t       e = HYPREDRV_LinearSystemGetRHSValues(h, &p);
   if (e) return e;
   if (vec) *vec = (HYPRE_Vector)view_handle(&h->rhs_handle, h, p);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetMatrix(HYPREDRV_t h, HYPRE_Matrix *mat)
{
   CHECK_OBJ(h);
   if (mat) *mat = (HYPRE_Matrix)h->A; /* opaque device handle */
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSystemGetDevicePointers(HYPREDRV_t h, double **x_d, double **b_d)
{
   CHECK_OBJ(h);
   if (x_d) *x_d = h->x_d;
   if (b_d) *b_d = h->b_d;
   return hd_err_get();
}

uint32_t HYPREDRV_GetDeviceHandles(HYPREDRV_t h, void **A, void **M)
{
   CHECK_OBJ(h);
   if (A) *A = h->A;
   if (M) *M = h->precon;
   return hd_err_get();
}

/* ---- preconditioner / solver lifecycle ---------------------------------------------- */
uint32_t HYPREDRV_PreconCreate(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:2793 -> precon.c:461 -> amg.c:863: options only; the hierarchy
    * is built by Setup */
   CHECK_ARGS(h);
   hd_err_reset();
   if (precon_reusable_for(h, h->ls_index)) { h->precon_created = true; return hd_err_get(); } /* reference HYPREDRV.c:2814-2833 */
   drop_precon(h);
   h->precon_created = true; h->precon_is_setup = false;
   return hd_err_get();
}

uint32_t HYPREDRV_PreconGetDeviceParams(HYPREDRV_t h, void *params)
{
   CHECK_ARGS(h);
   if (!params) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "null parameter block");
   if (hd_amg_check(&h->args->amg)) return hd_err_get();
   hd_amg_to_hdk(&h->args->amg, (hdk_amg_params *)params);
   return hd_err_get();
}

static uint32_t do_precon_setup(HYPREDRV_t h)
{
   if (!h->A) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "the matrix must be set before the preconditioner setup");
   if (precon_reusable_for(h, h->ls_index)) { h->setup_time = 0.0; return hd_err_get(); } /* reuse: no rebuild for this system */
   drop_precon(h);
   hdk_sync();
   double t0 = hd_wtime();
   if (h->args->precon_method == HD_PRECON_AMG)
   {
      hdk_amg_params p;
      if (hd_amg_check(&h->args->amg)) return hd_err_get();
      hd_amg_to_hdk(&h->args->amg, &p);
      if (p.coarsen_type != 8)
      {
         /* said once per process, whatever the print level: the CPU-default chain (HMIS) is inherently
          * sequential; results then follow the reference's GPU-build defaults, not its CPU goldens */
         static int warned = 0;
         if (h->rank == 0 && !warned++)
            fprintf(stderr, "hypredrive_b200: warning: coarsening type %d has no device kernel; using PMIS (8), "
                            "the reference's HYPRE_USING_GPU default\n", p.coarsen_type);
         p.coarsen_type = 8;
      }
      int rc = hdk_amg_setup(h->A, &p, &h->precon);
      if (rc) return hdk_fail(rc);
   }
   hdk_sync();
   h->setup_time      = hd_wtime() - t0;
   h->precon_is_setup = true;
   return hd_err_get();
}

static void stats_new_entry(HYPREDRV_t h)
{
   hd_stats *s = h->stats;
   if (s->counter + 1 >= HD_STATS_MAX) return;
   s->counter++;
   int i = s->counter;
   s->has_solve[i] = 0; s->setup[i] = 0; s->solve[i] = 0; s->iters[i] = 0; s->r0[i] = 0; s->rr[i] = 0;
   s->has_build[i] = h->have_pending_build;
   s->build[i]     = h->pending_build;
   h->have_pending_build = false; h->pending_build = 0.0;
}

uint32_t HYPREDRV_PreconSetup(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:2961 -> precon.c:709 -> HYPRE_BoomerAMGSetup */
   CHECK_ARGS(h);
   hd_err_reset();
   if (!h->precon_created) return fail(HYPREDRV_ERROR_INVALID_PRECON, "%s", "preconditioner was not created");
   return do_precon_setup(h);
}

uint32_t HYPREDRV_LinearSolverCreate(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:2897-2932: creates the preconditioner too when none exists */
   CHECK_ARGS(h);
   hd_err_reset();
   if (!h->precon_created)
   {
      h->precon_created = true;
      if (!precon_reusable_for(h, h->ls_index)) drop_precon(h); /* else: kept from an earlier system (reuse) */
   }
   h->solver_created = true;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSolverSetup(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:3001 -> solver.c:457-546: the Krylov setup calls back into the
    * preconditioner setup ("prec" timer, solver.c:288-302) */
   CHECK_ARGS(h);
   hd_err_reset();
   if (!h->solver_created) return fail(HYPREDRV_ERROR_INVALID_SOLVER, "%s", "solver was not created");
   stats_new_entry(h);
   uint32_t e = do_precon_setup(h);
   if (e) return e;
   if (h->stats->counter >= 0) h->stats->setup[h->stats->counter] = h->setup_time;
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSolverApply(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:3126 -> solver.c:627-693: r0 (untimed), Krylov solve ("solve"
    * timer), iterations, true relative residual (untimed) */
   CHECK_ARGS(h);
   hd_err_reset();
   if (!h->solver_created) return fail(HYPREDRV_ERROR_INVALID_SOLVER, "%s", "solver was not created");
   if (!h->precon_is_setup) return fail(HYPREDRV_ERROR_INVALID_PRECON, "%s", "preconditioner is not set up (call HYPREDRV_LinearSolverSetup)");
   if (!h->A || !h->b_d) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "matrix and right-hand side must be set before the solve");
   if (!h->x_d) { uint32_t e = HYPREDRV_LinearSystemResetInitialGuess(h); if (e) return e; }
   hd_stats *s = h->stats;
   if (s->counter < 0 || s->has_solve[s->counter]) stats_new_entry(h);
   int     i = s->counter;
   double *r = NULL, rn = 0.0, bn = 0.0;
   int     rc = hdk_vec_alloc(h->n, &r);
   if (!rc) rc = hdk_csr_residual(h->A, h->x_d, h->b_d, r);
   if (!rc) rc = hdk_vec_norm(r, h->n, 1, &rn);
   if (rc) { hdk_vec_free(r); return hdk_fail(rc); }
   double r0 = rn;
   hdk_krylov k;
   memset(&k, 0, sizeof(k));
   if (h->args->solver_method == HD_SOLVER_PCG)
   {
      k.max_iter = h->args->pcg.max_iter; k.rel_tol = h->args->pcg.relative_tol; k.abs_tol = h->args->pcg.absolute_tol;
      rc = hdk_pcg(h->A, h->precon, h->b_d, h->x_d, &k);
   }
   else
   {
      k.max_iter = h->args->gmres.max_iter; k.rel_tol = h->args->gmres.relative_tol; k.abs_tol = h->args->gmres.absolute_tol;
      k.krylov_dim = h->args->gmres.krylov_dim; k.min_iter = h->args->gmres.min_iter;
      k.skip_real_res_check = h->args->gmres.skip_real_res_check;
      if (h->args->solver_method == HD_SOLVER_FGMRES) rc = hdk_fgmres(h->A, h->precon, h->b_d, h->x_d, &k);
      else if (h->args->solver_method == HD_SOLVER_BICGSTAB) rc = hdk_bicgstab(h->A, h->precon, h->b_d, h->x_d, &k);
      else rc = hdk_gmres(h->A, h->precon, h->b_d, h->x_d, &k);
   }
   if (rc) { hdk_vec_free(r); return hdk_fail(rc); }
   h->iters = k.iters; h->converged = k.converged; h->final_res = k.rel_res_norm; h->solve_time = 1e-3 * k.solve_ms;
   /* true final residual ||b - A x|| / ||b|| (||b|| = 0 -> 1) */
   rc = hdk_csr_residual(h->A, h->x_d, h->b_d, r);
   if (!rc) rc = hdk_vec_norm(r, h->n, 1, &rn);
   if (!rc) rc = hdk_vec_norm(h->b_d, h->n, 1, &bn);
   hdk_vec_free(r);
   if (rc) return hdk_fail(rc);
   if (i >= 0 && i < HD_STATS_MAX)
   {
      s->has_solve[i] = 1; s->solve[i] = h->solve_time; s->iters[i] = k.iters; s->r0[i] = r0;
      s->rr[i] = rn / (bn > 0.0 ? bn : 1.0);
      if (s->setup[i] == 0.0 && h->setup_time > 0.0 && i == 0) s->setup[i] = h->setup_time;
   }
   return hd_err_get();
}

uint32_t HYPREDRV_PreconApply(HYPREDRV_t h, HYPRE_Vector vec_b, HYPRE_Vector vec_x)
{
   /* reference src/HYPREDRV.c:3345 -> precon.c:804 -> HYPRE_BoomerAMGSolve (x is the guess) */
   CHECK_ARGS(h);
   hd_err_reset();
   struct hypre_IJVector_struct *b = (struct hypre_IJVector_struct *)vec_b, *x = (struct hypre_IJVector_struct *)vec_x;
   if (!b || !x || b->magic != HD_IJVEC_MAGIC || x->magic != HD_IJVEC_MAGIC || b->n != h->n || x->n != h->n)
      return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "PreconApply needs IJ vectors matching the system");
   if (!h->precon_is_setup) return fail(HYPREDRV_ERROR_INVALID_PRECON, "%s", "preconditioner is not set up");
   double *bd = NULL, *xd = NULL;
   int     rc = hdk_vec_alloc(h->n, &bd);
   if (!rc) rc = hdk_vec_alloc(h->n, &xd);
   if (!rc) rc = hdk_vec_h2d(bd, b->data, h->n);
   if (!rc) rc = hdk_vec_h2d(xd, x->data, h->n);
   if (!rc) rc = h->precon ? hdk_amg_vcycle(h->precon, bd, xd) : hdk_vec_copy(xd, bd, h->n);
   if (!rc) rc = hdk_vec_d2h(x->data, xd, h->n);
   hdk_vec_free(bd); hdk_vec_free(xd);
   return rc ? hdk_fail(rc) : hd_err_get();
}

uint32_t HYPREDRV_PreconDestroy(HYPREDRV_t h)
{
   CHECK_OBJ(h);
   h->precon_created = false;
   if (precon_reusable_for(h, h->ls_index + 1)) return hd_err_get(); /* the next system reuses it */
   drop_precon(h);
   return hd_err_get();
}

uint32_t HYPREDRV_LinearSolverDestroy(HYPREDRV_t h)
{
   /* reference src/HYPREDRV.c:3463: also releases the preconditioner it created */
   CHECK_OBJ(h);
   h->solver_created = false;
   return HYPREDRV_PreconDestroy(h);
}

/* ---- statistics / getters ------------------------------------------------------------ */
uint32_t HYPREDRV_StatsPrint(HYPREDRV_t h)
{
   CHECK_OBJ(h);
   if (h->rank == 0 && (!h->args || h->args->general.statistics)) hd_stats_print(h->stats, stdout);
   return hd_err_get();
}
uint32_t HYPREDRV_AnnotateBegin(HYPREDRV_t h, const char *name, int id) { CHECK_OBJ(h); (void)name; (void)id; return hd_err_get(); }
uint32_t HYPREDRV_AnnotateEnd(HYPREDRV_t h, const char *name, int id) { CHECK_OBJ(h); (void)name; (void)id; return hd_err_get(); }
uint32_t HYPREDRV_AnnotateLevelBegin(HYPREDRV_t h, int level, const char *name, int id) { CHECK_OBJ(h); (void)level; (void)name; (void)id; return hd_err_get(); }
uint32_t HYPREDRV_AnnotateLevelEnd(HYPREDRV_t h, int level, const char *name, int id) { CHECK_OBJ(h); (void)level; (void)name; (void)id; return hd_err_get(); }

uint32_t HYPREDRV_LinearSolverGetNumIter(HYPREDRV_t h, int *iters) { CHECK_OBJ(h); if (!iters) return fail(HYPREDRV_ERROR_INVALID_VAL, NULL, NULL); *iters = h->iters; return hd_err_get(); }
uint32_t HYPREDRV_LinearSolverGetConverged(HYPREDRV_t h, int *c) { CHECK_OBJ(h); if (!c) return fail(HYPREDRV_ERROR_INVALID_VAL, NULL, NULL); *c = h->converged; return hd_err_get(); }
uint32_t HYPREDRV_LinearSolverGetFinalRelativeResidualNorm(HYPREDRV_t h, double *n) { CHECK_OBJ(h); if (!n) return fail(HYPREDRV_ERROR_INVALID_VAL, NULL, NULL); *n = h->final_res; return hd_err_get(); }
uint32_t HYPREDRV_LinearSolverGetSetupTime(HYPREDRV_t h, double *s) { CHECK_OBJ(h); if (!s) return fail(HYPREDRV_ERROR_INVALID_VAL, NULL, NULL); *s = h->setup_time; return hd_err_get(); }
uint32_t HYPREDRV_LinearSolverGetSolveTime(HYPREDRV_t h, double *s) { CHECK_OBJ(h); if (!s) return fail(HYPREDRV_ERROR_INVALID_VAL, NULL, NULL); *s = h->solve_time; return hd_err_get(); }

uint32_t HYPREDRV_StatsLevelGetCount(HYPREDRV_t h, int level, int *count)
{
   CHECK_OBJ(h);
   if (level != 0 || !count) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "only statistics level 0 exists");
   int c = 0;
   for (int i = 0; i <= h->stats->counter; i++) c += h->stats->has_solve[i];
   *count = c;
   return hd_err_get();
}
uint32_t HYPREDRV_StatsLevelGetEntry(HYPREDRV_t h, int level, int index, int *entry_id, int *num_solves, int *linear_iters,
                                     double *setup_time, double *solve_time)
{
   CHECK_OBJ(h);
   if (level != 0 || index < 0 || index > h->stats->counter) return fail(HYPREDRV_ERROR_INVALID_VAL, "%s", "statistics entry out of range");
   if (entry_id) *entry_id = index;
   if (num_solves) *num_solves = h->stats->has_solve[index];
   if (linear_iters) *linear_iters = h->stats->iters[index];
   if (setup_time) *setup_time = h->stats->setup[index];
   if (solve_time) *solve_time = h->stats->solve[index];
   return hd_err_get();
}
uint32_t HYPREDRV_StatsLevelPrint(HYPREDRV_t h, int level) { (void)level; return HYPREDRV_StatsPrint(h); }

int HYPREDRV_SizeofBigInt(void) { return (int)sizeof(HYPRE_BigInt); }
int HYPREDRV_SizeofReal(void) { return (int)sizeof(HYPRE_Real); }
int HYPREDRV_SizeofInt(void) { return (int)sizeof(HYPRE_Int); }

/* ---- outside the hot path: exported, fail loudly -------------------------------------- */
#define OUT_OF_SCOPE(what)                                                                             \
   do {                                                                                                \
      CHECK_OBJ(hypredrv);                                                                             \
      return fail(HYPREDRV_ERROR_UNKNOWN, "%s is outside the B200 hot path (SURVEY.md section 8)", what); \
   } while (0)

uint32_t HYPREDRV_LinearSystemSetReferenceSolution(HYPREDRV_t hypredrv, HYPRE_Vector v) { (void)v; OUT_OF_SCOPE("reference solutions"); }
uint32_t HYPREDRV_LinearSystemSetDiscreteGradient(HYPREDRV_t hypredrv, HYPRE_Matrix G) { (void)G; OUT_OF_SCOPE("discrete gradient (AMS)"); }
uint32_t HYPREDRV_LinearSystemSetDiscreteCurl(HYPREDRV_t hypredrv, HYPRE_Matrix C) { (void)C; OUT_OF_SCOPE("discrete curl (ADS)"); }
uint32_t HYPREDRV_LinearSystemSetCoordinates(HYPREDRV_t hypredrv, HYPRE_Vector x, HYPRE_Vector y, HYPRE_Vector z) { (void)x; (void)y; (void)z; OUT_OF_SCOPE("coordinate vectors"); }
uint32_t HYPREDRV_LinearSystemSetDofmap(HYPREDRV_t hypredrv, int size, const int *dofmap) { (void)size; (void)dofmap; OUT_OF_SCOPE("dofmaps (MGR)"); }
uint32_t HYPREDRV_LinearSystemSetInterleavedDofmap(HYPREDRV_t hypredrv, int a, int b) { (void)a; (void)b; OUT_OF_SCOPE("dofmaps (MGR)"); }
uint32_t HYPREDRV_LinearSystemSetContiguousDofmap(HYPREDRV_t hypredrv, int a, int b) { (void)a; (void)b; OUT_OF_SCOPE("dofmaps (MGR)"); }
uint32_t HYPREDRV_LinearSystemReadDofmap(HYPREDRV_t hypredrv) { OUT_OF_SCOPE("dofmaps (MGR)"); }
uint32_t HYPREDRV_LinearSystemPrintDofmap(HYPREDRV_t hypredrv, const char *f) { (void)f; OUT_OF_SCOPE("dofmaps (MGR)"); }
uint32_t HYPREDRV_LinearSystemPrint(HYPREDRV_t hypredrv) { OUT_OF_SCOPE("linear-system dumps"); }
uint32_t HYPREDRV_LinearSystemSetNearNullSpace(HYPREDRV_t hypredrv, int a, int b, const HYPRE_Complex *v) { (void)a; (void)b; (void)v; OUT_OF_SCOPE("near-null-space vectors"); }
uint32_t HYPREDRV_LinearSystemSetNullSpace(HYPREDRV_t hypredrv, int a, int b, const HYPRE_Complex *v) { (void)a; (void)b; (void)v; OUT_OF_SCOPE("null-space vectors"); }
uint32_t HYPREDRV_StateVectorSet(HYPREDRV_t hypredrv, int n, HYPRE_IJVector *v) { (void)n; (void)v; OUT_OF_SCOPE("state vectors"); }
uint32_t HYPREDRV_StateVectorGetValues(HYPREDRV_t hypredrv, int i, HYPRE_Complex **p) { (void)i; (void)p; OUT_OF_SCOPE("state vectors"); }
uint32_t HYPREDRV_StateVectorCopy(HYPREDRV_t hypredrv, int a, int b) { (void)a; (void)b; OUT_OF_SCOPE("state vectors"); }
uint32_t HYPREDRV_StateVectorUpdateAll(HYPREDRV_t hypredrv) { OUT_OF_SCOPE("state vectors"); }
uint32_t HYPREDRV_StateVectorApplyCorrection(HYPREDRV_t hypredrv, int i) { (void)i; OUT_OF_SCOPE("state vectors"); }
uint32_t HYPREDRV_LinearSystemComputeEigenspectrum(HYPREDRV_t hypredrv) { OUT_OF_SCOPE("eigenspectrum analysis"); }
