/* hd_internal.h -- host-side (plain C) internals of the HYPREDRV_* layer of hypredrive_b200.
 * Mirrors the roles of the reference's src/internal/{error,yaml,args,amg,pcg,gmres,stats,
 * linsys}.h for the hot-path subset; written from scratch around the hdk_* device C-ABI. */
#ifndef HD_INTERNAL_H
#define HD_INTERNAL_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "HYPREDRV.h"
#include "hdk.h"

/* ---------------------------------------------------------------- errors (hd_error.c) */
void     hd_err_set(uint32_t bits);
uint32_t hd_err_get(void);
void     hd_err_reset(void);
void     hd_err_msg(const char *fmt, ...);
void     hd_err_print_msgs(void);
void     hd_err_clear_msgs(void);
void     hd_err_describe(uint32_t code);
int      hd_err_msg_count(void);
const char *hd_err_msg_get(int i);

/* ---------------------------------------------------------------- YAML tree (hd_yaml.c) */
typedef struct hd_node
{
   char           *key;
   char           *val;        /* trimmed, unquoted, lower-cased unless key contains "name" */
   char           *raw_val;    /* original spelling */
   int             level;
   int             is_seq_item; /* came from a "- " line */
   int             used;       /* consumed by a schema */
   int             invalid;    /* 1 = unknown key, 2 = bad value */
   struct hd_node *child, *next, *parent;
} hd_node;

hd_node *hd_yaml_parse(const char *text, const char *base_dir); /* NULL + error bits on failure */
void     hd_yaml_free(hd_node *root);
hd_node *hd_yaml_find(hd_node *parent, const char *key);
int      hd_yaml_override(hd_node *root, const char *path, const char *value);
void     hd_yaml_print(const hd_node *root, FILE *fp);

/* ---------------------------------------------------------------- options (hd_args.c) */
typedef enum { HD_SOLVER_PCG = 0, HD_SOLVER_GMRES = 1, HD_SOLVER_FGMRES = 2, HD_SOLVER_BICGSTAB = 3 } hd_solver_t;
typedef enum { HD_PRECON_AMG = 0, HD_PRECON_NONE = 1 } hd_precon_t;

typedef struct
{
   char   name[256];
   char   statistics_filename[1024];
   int    warmup, statistics, print_config_params, use_millisec, device_lazy_init, exec_policy;
   int    use_vendor_spgemm, use_vendor_spmv, num_repetitions;
   double dev_pool_size, uvm_pool_size, host_pool_size, pinned_pool_size;
} hd_general_args;

typedef struct
{
   char matrix_filename[1024], rhs_filename[1024], x0_filename[1024], dirname[1024];
   int  init_guess_mode; /* zeros 0, ones 1, file 2, random 3, previous 4 */
   int  rhs_mode;        /* zeros 0, ones 1, file 2, random 3, randsol 4 */
   int  type, num_systems, exec_policy;
} hd_ls_args;

typedef struct
{
   int    max_iter, two_norm, stop_crit, rel_change, print_level, recompute_res;
   double relative_tol, absolute_tol, residual_tol, conv_fac_tol;
} hd_pcg_args;

typedef struct
{
   int    min_iter, max_iter, stop_crit, skip_real_res_check, krylov_dim, rel_change, logging, print_level;
   double relative_tol, absolute_tol, conv_fac_tol;
} hd_gmres_args;

typedef struct
{
   int    max_iter, print_level;
   double tolerance;
   /* interpolation */
   int    prolongation_type, restriction_type, max_nnz_row;
   double trunc_factor, restrict_strong_th, restrict_filter_th;
   /* coarsening */
   int    coarsen_type, rap2, mod_rap2, keep_transpose, sabs, num_functions, filter_functions, nodal, seq_amg_th;
   int    min_coarse_size, max_coarse_size, max_levels;
   double max_row_sum, strong_th;
   /* aggressive */
   int    agg_num_levels, agg_num_paths, agg_prolongation_type, agg_max_nnz_row;
   double agg_trunc_factor, agg_P12_max_elements, agg_P12_trunc_factor;
   /* relaxation */
   int    relax_type, down_type, up_type, coarse_type, down_sweeps, up_sweeps, coarse_sweeps, num_sweeps, order, points;
   double weight, outer_weight;
   /* relaxation:chebyshev (hypre HYPRE_BoomerAMGSetCheby{Order,Fraction,EigEst,Variant,Scale}) */
   int    cheby_order, cheby_eig_est, cheby_variant, cheby_scale;
   double cheby_fraction;
   /* complex smoother */
   int    smooth_type, smooth_num_levels, smooth_num_sweeps;
} hd_amg_args;

/* preconditioner.reuse, static policy (reference src/internal/precon_reuse.c:780-830,
 * docs/usrman-src/input_structure.rst "Static reuse") */
#define HD_REUSE_MAX_IDS 256
typedef struct
{
   int enabled, frequency, n_ids;
   int ids[HD_REUSE_MAX_IDS];
} hd_reuse_args;

typedef struct
{
   hd_general_args general;
   hd_ls_args      ls;
   hd_solver_t     solver_method;
   hd_pcg_args     pcg;
   hd_gmres_args   gmres;
   hd_precon_t     precon_method;
   hd_amg_args     amg;
   hd_reuse_args   reuse;
   int             num_precon_variants, active_precon_variant;
   bool            lib_mode;
} hd_args;

void hd_args_defaults(hd_args *a, bool lib_mode);
void hd_amg_defaults(hd_amg_args *a);
void hd_pcg_defaults(hd_pcg_args *a);
void hd_gmres_defaults(hd_gmres_args *a);
/* text: YAML text; overrides: argc/argv pairs "--a:b:c value" (may start with -a/--args) */
hd_args *hd_args_parse(const char *yaml_text, const char *base_dir, int n_over, char **over, bool lib_mode,
                       bool print_tree);
int  hd_args_apply_precon_preset(hd_args *a, const char *preset);
int  hd_args_apply_solver_preset(hd_args *a, const char *preset);
int  hd_preset_register(int kind, const char *name, const char *text, const char *help);
void hd_amg_to_hdk(const hd_amg_args *a, hdk_amg_params *p);
int  hd_amg_check(const hd_amg_args *a); /* 1 (error bit and message set): an option combination without a device path */
/* 1 if the preconditioner must be rebuilt for the 0-based linear system `ls_id` */
int  hd_reuse_should_rebuild(const hd_reuse_args *r, int ls_id);

/* ---------------------------------------------------------------- statistics (hd_stats.c) */
#define HD_STATS_MAX 4096
typedef struct
{
   int    counter;            /* current entry (-1 before the first system) */
   int    ls_id;
   double build[HD_STATS_MAX], setup[HD_STATS_MAX], solve[HD_STATS_MAX];
   double r0[HD_STATS_MAX], rr[HD_STATS_MAX];
   int    iters[HD_STATS_MAX], has_solve[HD_STATS_MAX], has_build[HD_STATS_MAX];
   double t_open[8];
   int    use_millisec;
   char   name[256];
} hd_stats;

hd_stats *hd_stats_create(void);
void      hd_stats_print(const hd_stats *s, FILE *fp);
double    hd_wtime(void);

/* ---------------------------------------------------------------- IJ containers (hd_ij.c) */
struct hypre_IJMatrix_struct
{
   uint32_t      magic;
   HYPRE_BigInt  ilower, iupper, jlower, jupper;
   int64_t       nrows;
   int64_t      *row_len, *row_cap;
   HYPRE_BigInt **row_cols;
   double      **row_vals;
   int           assembled;
   /* flattened after assemble */
   int64_t      *indptr;
   HYPRE_BigInt *cols;
   double       *vals;
};
struct hypre_IJVector_struct
{
   uint32_t     magic;
   HYPRE_BigInt jlower, jupper;
   int64_t      n;
   double      *data;
};
#define HD_IJMAT_MAGIC 0x494a4d41u
#define HD_IJVEC_MAGIC 0x494a5645u
int hd_ij_matrix_flatten(struct hypre_IJMatrix_struct *A);

/* ---------------------------------------------------------------- file readers (hd_io.c) */
int hd_read_ij_matrix(const char *prefix, int rank, HYPRE_IJMatrix *out);
int hd_read_ij_vector(const char *prefix, int rank, HYPRE_IJVector *out);

#endif
