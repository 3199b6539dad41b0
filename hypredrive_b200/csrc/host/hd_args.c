/* hd_args.c -- table-driven mapping of the YAML tree onto solver options.
 * Keys, defaults and name<->integer maps follow the reference:
 *   general          src/internal/args.c:31-104
 *   linear_system    src/internal/linsys.c:361-431
 *   solver: pcg      src/internal/pcg.c:15-25      gmres  src/internal/gmres.c:16-27
 *   preconditioner: amg  src/internal/amg.c:23-90 (schema), :120-238 (defaults under
 *                    HYPRE_USING_GPU -- this library IS the GPU build: PMIS, l1-Jacobi,
 *                    mod_rap2, keep_transpose), :245-458 (maps)
 * A map accepts the name or its integer (src/internal/containers.c:752-794); booleans accept
 * on/yes/true/1 and off/no/false/0 (containers.c:691-702). */
#include "hd_internal.h"
#include <ctype.h>
#include <stdlib.h>
#include <string.h>

typedef struct { const char *name; int value; } hd_map;
typedef enum { F_INT, F_DBL, F_STR, F_MAP, F_GB, F_IGNORE } hd_ftype;
typedef struct
{
   const char   *key;
   hd_ftype      type;
   size_t        off;
   const hd_map *map;
   size_t        cap; /* F_STR */
} hd_field;

#define MAP_END {NULL, 0}
static const hd_map map_onoff[] = {{"on", 1}, {"yes", 1}, {"true", 1}, {"1", 1}, {"off", 0}, {"no", 0}, {"false", 0}, {"0", 0}, MAP_END};
static const hd_map map_stats[] = {{"off", 0}, {"no", 0}, {"false", 0}, {"0", 0}, {"on", 1}, {"yes", 1}, {"true", 1}, {"1", 1}, {"2", 2}, MAP_END};
static const hd_map map_exec[]  = {{"host", 0}, {"device", 1}, MAP_END};
static const hd_map map_lstype[] = {{"online", 0}, {"ij", 1}, {"parcsr", 2}, {"mtx", 3}, MAP_END};
static const hd_map map_rhs[]   = {{"zeros", 0}, {"ones", 1}, {"file", 2}, {"random", 3}, {"randsol", 4}, MAP_END};
static const hd_map map_x0[]    = {{"zeros", 0}, {"ones", 1}, {"file", 2}, {"random", 3}, {"previous", 4}, MAP_END};
static const hd_map map_interp[] = {{"mod_classical", 0}, {"least_squares", 1}, {"mod_classical_he", 2}, {"direct_sep_weights", 3},
   {"multipass", 4}, {"multipass_sep_weights", 5}, {"extended+i", 6}, {"extended+i_c", 7}, {"standard", 8},
   {"standard_sep_weights", 9}, {"blk_classical", 10}, {"blk_classical_diag", 11}, {"f_f", 12}, {"f_f1", 13},
   {"extended", 14}, {"mm_extended", 16}, {"mm_extended+i", 17}, {"mm-ext+i", 17}, {"mm_extended+e", 18},
   {"mm-ext+e", 18}, {"blk_direct", 24}, {"one_point", 100}, MAP_END};
static const hd_map map_restr[] = {{"p_transpose", 0}, {"air_1", 1}, {"air_2", 2}, {"neumann_air_0", 3}, {"neumann_air_1", 4},
   {"neumann_air_2", 5}, {"air_1.5", 15}, MAP_END};
static const hd_map map_coarsen[] = {{"cljp", 0}, {"rs", 1}, {"rs3", 3}, {"falgout", 6}, {"pmis", 8}, {"hmis", 10}, MAP_END};
static const hd_map map_relax[] = {{"jacobi_non_mv", 0}, {"forward-hgs", 3}, {"backward-hgs", 4}, {"chaotic-hgs", 5}, {"hsgs", 6},
   {"jacobi", 7}, {"l1-hsgs", 8}, {"forward-solve", 10}, {"2gs-it1", 11}, {"2gs-it2", 12}, {"forward-hl1gs", 13},
   {"backward-hl1gs", 14}, {"cg", 15}, {"chebyshev", 16}, {"l1-jacobi", 18}, {"l1sym-hgs", 89}, MAP_END};
static const hd_map map_coarse[] = {{"jacobi_non_mv", 0}, {"hsgs", 6}, {"jacobi", 7}, {"l1-hsgs", 8}, {"ge", 9}, {"2gs-it1", 11},
   {"2gs-it2", 12}, {"forward-hl1gs", 13}, {"backward-hl1gs", 14}, {"cg", 15}, {"chebyshev", 16}, {"l1-jacobi", 18},
   {"l1sym-hgs", 89}, {"lu_piv", 99}, {"lu_inv", 199}, MAP_END};
static const hd_map map_points[] = {{"all", 0}, {"air", 1}, MAP_END};
static const hd_map map_aggint[] = {{"2_stage_extended+i", 1}, {"2_stage_standard", 2}, {"2_stage_extended", 3}, {"multipass", 4},
   {"mm_extended", 5}, {"mm_extended+i", 6}, {"mm_extended+e", 7}, MAP_END};
static const hd_map map_smooth[] = {{"fsai", 4}, {"ilu", 5}, {"schwarz", 6}, {"pilut", 7}, {"parasails", 8}, {"euclid", 9}, MAP_END};

#define OFF(T, f) offsetof(T, f)
#define FI(T, f) {#f, F_INT, OFF(T, f), NULL, 0}
#define FD(T, f) {#f, F_DBL, OFF(T, f), NULL, 0}
#define FM(T, f, m) {#f, F_MAP, OFF(T, f), m, 0}
#define FS(T, f) {#f, F_STR, OFF(T, f), NULL, sizeof(((T *)0)->f)}
#define FG(T, f) {#f, F_GB, OFF(T, f), NULL, 0}
#define FX(k) {k, F_IGNORE, 0, NULL, 0}
#define FEND {NULL, F_INT, 0, NULL, 0}

static const hd_field f_general[] = {
   FS(hd_general_args, name), FS(hd_general_args, statistics_filename), FM(hd_general_args, warmup, map_onoff),
   FM(hd_general_args, statistics, map_stats), FM(hd_general_args, print_config_params, map_onoff),
   FM(hd_general_args, use_millisec, map_onoff), FM(hd_general_args, device_lazy_init, map_onoff),
   FM(hd_general_args, exec_policy, map_exec), FM(hd_general_args, use_vendor_spgemm, map_onoff),
   FM(hd_general_args, use_vendor_spmv, map_onoff), FI(hd_general_args, num_repetitions),
   FG(hd_general_args, dev_pool_size), FG(hd_general_args, uvm_pool_size), FG(hd_general_args, host_pool_size),
   FG(hd_general_args, pinned_pool_size), FEND};

static const hd_field f_ls[] = {
   FS(hd_ls_args, matrix_filename), FS(hd_ls_args, rhs_filename), FS(hd_ls_args, x0_filename), FS(hd_ls_args, dirname),
   FM(hd_ls_args, init_guess_mode, map_x0), FM(hd_ls_args, rhs_mode, map_rhs), FM(hd_ls_args, type, map_lstype),
   FM(hd_ls_args, exec_policy, map_exec), FI(hd_ls_args, num_systems),
   FX("sequence_filename"), FX("matrix_basename"), FX("precmat_filename"), FX("precmat_basename"), FX("rhs_basename"),
   FX("xref_filename"), FX("xref_basename"), FX("timestep_filename"), FX("sol_filename"), FX("dofmap_filename"),
   FX("dofmap_basename"), FX("digits_suffix"), FX("init_suffix"), FX("last_suffix"), FX("set_suffix"),
   FX("print_system"), FX("eigspec"), FX("dof_labels"), FEND};

static const hd_field f_pcg[] = {
   FI(hd_pcg_args, max_iter), FM(hd_pcg_args, two_norm, map_onoff), FM(hd_pcg_args, stop_crit, map_onoff),
   FM(hd_pcg_args, rel_change, map_onoff), FI(hd_pcg_args, print_level), FI(hd_pcg_args, recompute_res),
   FD(hd_pcg_args, relative_tol), FD(hd_pcg_args, absolute_tol), FD(hd_pcg_args, residual_tol),
   FD(hd_pcg_args, conv_fac_tol), FEND};

static const hd_field f_gmres[] = {
   FI(hd_gmres_args, min_iter), FI(hd_gmres_args, max_iter), FI(hd_gmres_args, stop_crit),
   FM(hd_gmres_args, skip_real_res_check, map_onoff), FI(hd_gmres_args, krylov_dim), FM(hd_gmres_args, rel_change, map_onoff),
   FI(hd_gmres_args, logging), FI(hd_gmres_args, print_level), FD(hd_gmres_args, relative_tol),
   FD(hd_gmres_args, absolute_tol), FD(hd_gmres_args, conv_fac_tol), FEND};

/* fgmres (src/internal/fgmres.c:14-21) and bicgstab (src/internal/bicgstab.c:14-22) share the
 * gmres option record: their keys are subsets of it */
static const hd_field f_fgmres[] = {
   FI(hd_gmres_args, min_iter), FI(hd_gmres_args, max_iter), FI(hd_gmres_args, krylov_dim), FI(hd_gmres_args, logging),
   FI(hd_gmres_args, print_level), FD(hd_gmres_args, relative_tol), FD(hd_gmres_args, absolute_tol), FEND};
static const hd_field f_bicgstab[] = {
   FI(hd_gmres_args, min_iter), FI(hd_gmres_args, max_iter), FI(hd_gmres_args, stop_crit), FI(hd_gmres_args, logging),
   FI(hd_gmres_args, print_level), FD(hd_gmres_args, relative_tol), FD(hd_gmres_args, absolute_tol),
   FD(hd_gmres_args, conv_fac_tol), FEND};

static const hd_field f_amg[] = {FI(hd_amg_args, max_iter), FI(hd_amg_args, print_level), FD(hd_amg_args, tolerance), FEND};
static const hd_field f_amg_int[] = {
   FM(hd_amg_args, prolongation_type, map_interp), FM(hd_amg_args, restriction_type, map_restr), FI(hd_amg_args, max_nnz_row),
   FD(hd_amg_args, trunc_factor), FD(hd_amg_args, restrict_strong_th), FD(hd_amg_args, restrict_filter_th), FEND};
static const hd_field f_amg_csn[] = {
   {"type", F_MAP, OFF(hd_amg_args, coarsen_type), map_coarsen, 0}, FM(hd_amg_args, rap2, map_onoff),
   FM(hd_amg_args, mod_rap2, map_onoff), FM(hd_amg_args, keep_transpose, map_onoff), FI(hd_amg_args, sabs),
   FI(hd_amg_args, num_functions), FM(hd_amg_args, filter_functions, map_onoff), FM(hd_amg_args, nodal, map_onoff),
   FI(hd_amg_args, seq_amg_th), FI(hd_amg_args, min_coarse_size), FI(hd_amg_args, max_coarse_size),
   FI(hd_amg_args, max_levels), FD(hd_amg_args, max_row_sum), FD(hd_amg_args, strong_th), FEND};
static const hd_field f_amg_agg[] = {
   {"num_levels", F_INT, OFF(hd_amg_args, agg_num_levels), NULL, 0}, {"num_paths", F_INT, OFF(hd_amg_args, agg_num_paths), NULL, 0},
   {"prolongation_type", F_MAP, OFF(hd_amg_args, agg_prolongation_type), map_aggint, 0},
   {"max_nnz_row", F_INT, OFF(hd_amg_args, agg_max_nnz_row), NULL, 0},
   {"trunc_factor", F_DBL, OFF(hd_amg_args, agg_trunc_factor), NULL, 0},
   {"P12_max_elements", F_DBL, OFF(hd_amg_args, agg_P12_max_elements), NULL, 0},
   {"P12_trunc_factor", F_DBL, OFF(hd_amg_args, agg_P12_trunc_factor), NULL, 0}, FEND};
static const hd_field f_amg_rlx[] = {
   FM(hd_amg_args, down_type, map_relax), FM(hd_amg_args, up_type, map_relax), FM(hd_amg_args, coarse_type, map_coarse),
   FI(hd_amg_args, down_sweeps), FI(hd_amg_args, up_sweeps), FI(hd_amg_args, coarse_sweeps), FI(hd_amg_args, num_sweeps),
   FI(hd_amg_args, order), FM(hd_amg_args, points, map_points), FD(hd_amg_args, weight), FD(hd_amg_args, outer_weight),
   FEND};
static const hd_field f_amg_cheby[] = {
   {"order", F_INT, OFF(hd_amg_args, cheby_order), NULL, 0}, {"fraction", F_DBL, OFF(hd_amg_args, cheby_fraction), NULL, 0},
   {"eig_est", F_INT, OFF(hd_amg_args, cheby_eig_est), NULL, 0}, {"variant", F_INT, OFF(hd_amg_args, cheby_variant), NULL, 0},
   {"scale", F_INT, OFF(hd_amg_args, cheby_scale), NULL, 0}, FEND};
static const hd_field f_amg_smt[] = {
   {"type", F_MAP, OFF(hd_amg_args, smooth_type), map_smooth, 0}, {"num_levels", F_INT, OFF(hd_amg_args, smooth_num_levels), NULL, 0},
   {"num_sweeps", F_INT, OFF(hd_amg_args, smooth_num_sweeps), NULL, 0}, FX("fsai"), FX("ilu"), FEND};

/* ------------------------------------------------------------------------------------- */
static int map_lookup(const hd_map *m, const char *s, int *out)
{
   for (const hd_map *e = m; e->name; e++)
      if (!strcmp(e->name, s)) { *out = e->value; return 1; }
   /* also accept the integer code of any entry */
   char *end;
   long  v = strtol(s, &end, 10);
   if (*s && !*end)
      for (const hd_map *e = m; e->name; e++)
         if (e->value == (int)v) { *out = (int)v; return 1; }
   return 0;
}

static void mark_invalid(hd_node *n, int kind, const char *section)
{
   n->invalid = kind;
   if (kind == 1) { hd_err_set(HYPREDRV_ERROR_INVALID_KEY); hd_err_msg("unknown key '%s' under '%s'", n->key, section); }
   else { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("invalid value '%s' for key '%s' under '%s'", n->raw_val, n->key, section); }
}

/* set every child of `blk` that `tab` knows; unknown children are errors unless a later table
 * (nested sections) claims them -- callers pass `nested` names to skip */
static void apply_fields(hd_node *blk, const hd_field *tab, void *base, const char *section, const char **nested)
{
   for (hd_node *c = blk ? blk->child : NULL; c; c = c->next)
   {
      int skip = 0;
      for (const char **s = nested; s && *s; s++) if (!strcmp(*s, c->key)) skip = 1;
      if (skip) continue;
      const hd_field *f = NULL;
      for (const hd_field *t = tab; t->key; t++) if (!strcmp(t->key, c->key)) { f = t; break; }
      if (!f) { mark_invalid(c, 1, section); continue; }
      c->used = 1;
      char *p = (char *)base + f->off, *end;
      switch (f->type)
      {
         case F_INT:
         {
            long v = strtol(c->val, &end, 10);
            if (!c->val[0] || *end) { int b; if (map_lookup(map_onoff, c->val, &b)) v = b; else { mark_invalid(c, 2, section); break; } }
            *(int *)p = (int)v;
            break;
         }
         case F_DBL:
         case F_GB:
         {
            double v = strtod(c->val, &end);
            if (!c->val[0] || *end) { mark_invalid(c, 2, section); break; }
            *(double *)p = f->type == F_GB ? v * 1073741824.0 : v;
            break;
         }
         case F_STR: snprintf(p, f->cap, "%s", c->raw_val); break;
         case F_MAP:
         {
            int v;
            if (!map_lookup(f->map, c->val, &v)) mark_invalid(c, 2, section);
            else *(int *)p = v;
            break;
         }
         case F_IGNORE: break;
      }
   }
}

void hd_pcg_defaults(hd_pcg_args *a)
{
   a->max_iter = 100; a->two_norm = 1; a->stop_crit = 0; a->rel_change = 0; a->print_level = 1; a->recompute_res = 0;
   a->relative_tol = 1.0e-6; a->absolute_tol = 0.0; a->residual_tol = 0.0; a->conv_fac_tol = 0.0;
}

void hd_gmres_defaults(hd_gmres_args *a)
{
   a->min_iter = 0; a->max_iter = 300; a->stop_crit = 0; a->skip_real_res_check = 0; a->krylov_dim = 30; a->rel_change = 0;
   a->logging = 1; a->print_level = 1; a->relative_tol = 1.0e-6; a->absolute_tol = 0.0; a->conv_fac_tol = 0.0;
}

void hd_amg_defaults(hd_amg_args *a)
{
   memset(a, 0, sizeof(*a));
   a->max_iter = 1; a->print_level = 0; a->tolerance = 0.0;
   a->prolongation_type = 6; a->restriction_type = 0; a->max_nnz_row = 4; a->trunc_factor = 0.0;
   a->restrict_strong_th = 0.25; a->restrict_filter_th = 0.0;
   a->rap2 = 0; a->mod_rap2 = 1; a->keep_transpose = 1; a->coarsen_type = 8; /* HYPRE_USING_GPU defaults */
   a->num_functions = 1; a->sabs = 0; a->filter_functions = 0; a->nodal = 0; a->seq_amg_th = 0;
   a->min_coarse_size = 0; a->max_coarse_size = 64; a->max_levels = 25; a->max_row_sum = 0.9; a->strong_th = 0.25;
   a->agg_num_levels = 0; a->agg_num_paths = 1; a->agg_prolongation_type = 4; a->agg_max_nnz_row = 0;
   a->relax_type = -1; a->down_type = 18; a->up_type = 18; a->coarse_type = 9;
   a->down_sweeps = -1; a->up_sweeps = -1; a->coarse_sweeps = 1; a->num_sweeps = 1; a->order = 0; a->points = 0;
   a->weight = 1.0; a->outer_weight = 1.0;
   a->cheby_order = 2; a->cheby_fraction = 0.3; a->cheby_eig_est = 10; a->cheby_variant = 0; a->cheby_scale = 1;
   a->smooth_type = 5; a->smooth_num_levels = 0; a->smooth_num_sweeps = 1;
}

void hd_args_defaults(hd_args *a, bool lib_mode)
{
   memset(a, 0, sizeof(*a));
   a->lib_mode = lib_mode;
   hd_general_args *gnl = &a->general;
   gnl->warmup = 0; gnl->statistics = 1; gnl->print_config_params = lib_mode ? 0 : 1; gnl->use_millisec = 0;
   gnl->device_lazy_init = 0; gnl->exec_policy = 1; gnl->use_vendor_spgemm = 1; gnl->use_vendor_spmv = 1;
   gnl->num_repetitions = 1;
   gnl->dev_pool_size = gnl->uvm_pool_size = gnl->host_pool_size = 2.0 * 1073741824.0;
   gnl->pinned_pool_size = 0.1 * 1073741824.0;
   a->ls.init_guess_mode = 0; a->ls.rhs_mode = 2; a->ls.type = 1; a->ls.num_systems = 1; a->ls.exec_policy = 1;
   a->solver_method = HD_SOLVER_PCG;
   hd_pcg_defaults(&a->pcg);
   hd_gmres_defaults(&a->gmres);
   a->precon_method = HD_PRECON_AMG;
   hd_amg_defaults(&a->amg);
   a->num_precon_variants = 1; a->active_precon_variant = 0;
}

static void amg_alias(hd_amg_args *a, const char *name)
{
   /* "jacobi" / "gauss-seidel" = one-level AMG (reference src/internal/precon.c:255-288) */
   int rt = -1;
   if (!strcmp(name, "jacobi")) rt = 0;
   else if (!strcmp(name, "gauss-seidel")) rt = 3;
   if (rt < 0) return;
   a->max_levels = 1; a->relax_type = rt; a->down_type = rt; a->coarse_type = rt;
   a->down_sweeps = 1; a->up_sweeps = 0; a->coarse_sweeps = 1;
}

static void parse_amg_block(hd_node *blk, hd_amg_args *a)
{
   static const char *nested[] = {"interpolation", "aggressive", "coarsening", "relaxation", "smoother", NULL};
   apply_fields(blk, f_amg, a, "amg", nested);
   hd_node *s;
   if ((s = hd_yaml_find(blk, "interpolation"))) { s->used = 1; apply_fields(s, f_amg_int, a, "amg:interpolation", NULL); }
   if ((s = hd_yaml_find(blk, "coarsening"))) { s->used = 1; apply_fields(s, f_amg_csn, a, "amg:coarsening", NULL); }
   if ((s = hd_yaml_find(blk, "aggressive"))) { s->used = 1; apply_fields(s, f_amg_agg, a, "amg:aggressive", NULL); }
   if ((s = hd_yaml_find(blk, "relaxation")))
   {
      static const char *rlx_nested[] = {"chebyshev", NULL};
      s->used = 1;
      apply_fields(s, f_amg_rlx, a, "amg:relaxation", rlx_nested);
      hd_node *c;
      if ((c = hd_yaml_find(s, "chebyshev"))) { c->used = 1; apply_fields(c, f_amg_cheby, a, "amg:relaxation:chebyshev", NULL); }
   }
   if ((s = hd_yaml_find(blk, "smoother"))) { s->used = 1; apply_fields(s, f_amg_smt, a, "amg:smoother", NULL); }
}

/* ---- presets (reference src/internal/presets.c:17-33) --------------------------------- */
typedef struct { int kind; char *name, *text, *help; } hd_preset;
static hd_preset *g_user = NULL;
static int        g_nuser = 0;

int hd_preset_register(int kind, const char *name, const char *text, const char *help)
{
   if (!name || !text) return 1;
   g_user = realloc(g_user, sizeof(hd_preset) * (size_t)(g_nuser + 1));
   g_user[g_nuser].kind = kind; g_user[g_nuser].name = strdup(name); g_user[g_nuser].text = strdup(text);
   g_user[g_nuser].help = strdup(help ? help : "");
   g_nuser++;
   return 0;
}

static int parse_precon_text(hd_args *a, const char *text);
static int parse_solver_text(hd_args *a, const char *text);

int hd_args_apply_precon_preset(hd_args *a, const char *preset)
{
   static const struct { const char *name, *text; } builtin[] = {
      {"poisson", "amg"},
      {"elasticity_2d", "amg:\n  coarsening:\n    num_functions: 2\n    strong_th: 0.8"},
      {"elasticity_3d", "amg:\n  coarsening:\n    num_functions: 3\n    strong_th: 0.8"},
   };
   for (int i = 0; i < g_nuser; i++)
      if (g_user[i].kind == 0 && !strcmp(g_user[i].name, preset)) return parse_precon_text(a, g_user[i].text);
   for (size_t i = 0; i < sizeof(builtin) / sizeof(builtin[0]); i++)
      if (!strcmp(builtin[i].name, preset)) return parse_precon_text(a, builtin[i].text);
   /* a bare method name is accepted as a preset too ("amg") */
   if (!strcmp(preset, "amg") || !strcmp(preset, "jacobi") || !strcmp(preset, "gauss-seidel") || !strcmp(preset, "none"))
      return parse_precon_text(a, preset);
   hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
   hd_err_msg("unknown preconditioner preset '%s'", preset);
   return 1;
}

int hd_args_apply_solver_preset(hd_args *a, const char *preset)
{
   for (int i = 0; i < g_nuser; i++)
      if (g_user[i].kind == 1 && !strcmp(g_user[i].name, preset)) return parse_solver_text(a, g_user[i].text);
   return parse_solver_text(a, preset);
}

static int set_solver_method(hd_args *a, const char *name)
{
   if (!strcmp(name, "pcg")) { a->solver_method = HD_SOLVER_PCG; return 0; }
   if (!strcmp(name, "gmres")) { a->solver_method = HD_SOLVER_GMRES; return 0; }
   if (!strcmp(name, "fgmres")) { a->solver_method = HD_SOLVER_FGMRES; return 0; }
   if (!strcmp(name, "bicgstab")) { a->solver_method = HD_SOLVER_BICGSTAB; return 0; }
   hd_err_set(HYPREDRV_ERROR_INVALID_SOLVER);
   hd_err_msg("unknown solver '%s' (supported: pcg, gmres, fgmres, bicgstab)", name);
   return 1;
}

static int set_precon_method(hd_args *a, const char *name)
{
   hd_amg_defaults(&a->amg);
   if (!strcmp(name, "amg")) { a->precon_method = HD_PRECON_AMG; return 0; }
   if (!strcmp(name, "jacobi") || !strcmp(name, "gauss-seidel")) { a->precon_method = HD_PRECON_AMG; amg_alias(&a->amg, name); return 0; }
   if (!strcmp(name, "none")) { a->precon_method = HD_PRECON_NONE; return 0; }
   hd_err_set(HYPREDRV_ERROR_INVALID_PRECON);
   hd_err_msg("preconditioner '%s' is outside the B200 hot path (supported: amg, jacobi, none)", name);
   return 1;
}

static int parse_solver_node(hd_args *a, hd_node *n)
{
   n->used = 1;
   if (!n->child)
   {
      /* value-only form: per-method defaults, print_level forced 0 (reference args.c:374-401) */
      if (!n->val[0]) { hd_err_set(HYPREDRV_ERROR_MISSING_SOLVER); hd_err_msg("empty solver section"); return 1; }
      if (set_solver_method(a, n->val)) { n->invalid = 2; return 1; }
      hd_pcg_defaults(&a->pcg); hd_gmres_defaults(&a->gmres);
      if (a->solver_method == HD_SOLVER_BICGSTAB) a->gmres.max_iter = 100;
      a->pcg.print_level = 0; a->gmres.print_level = 0;
      return 0;
   }
   hd_node *method = NULL;
   for (hd_node *c = n->child; c; c = c->next)
   {
      if (!strcmp(c->key, "scaling")) { c->used = 1; continue; } /* optional sibling, off by default */
      if (method) { hd_err_set(HYPREDRV_ERROR_EXTRA_KEY); hd_err_msg("solver section must name exactly one method"); c->invalid = 1; return 1; }
      method = c;
   }
   if (!method) { hd_err_set(HYPREDRV_ERROR_MISSING_SOLVER); return 1; }
   if (set_solver_method(a, method->key)) { method->invalid = 1; return 1; }
   method->used = 1;
   if (a->solver_method == HD_SOLVER_PCG) { hd_pcg_defaults(&a->pcg); apply_fields(method, f_pcg, &a->pcg, "solver:pcg", NULL); }
   else
   {
      hd_gmres_defaults(&a->gmres);
      if (a->solver_method == HD_SOLVER_GMRES) apply_fields(method, f_gmres, &a->gmres, "solver:gmres", NULL);
      else if (a->solver_method == HD_SOLVER_FGMRES) apply_fields(method, f_fgmres, &a->gmres, "solver:fgmres", NULL);
      else { a->gmres.max_iter = 100; apply_fields(method, f_bicgstab, &a->gmres, "solver:bicgstab", NULL); }
   }
   return 0;
}

/* preconditioner.reuse: `reuse: <frequency>` | `reuse: yes/no` | block {enabled, policy, frequency,
 * linear_system_ids (alias linear_solver_ids), per_timestep}.  Only the static policy exists
 * here; `adaptive` and `per_timestep: yes` are rejected (reference precon_reuse.c:2290-2400). */
static int parse_bool_word(const char *v, int *out)
{
   if (!strcmp(v, "yes") || !strcmp(v, "on") || !strcmp(v, "true") || !strcmp(v, "1")) { *out = 1; return 0; }
   if (!strcmp(v, "no") || !strcmp(v, "off") || !strcmp(v, "false") || !strcmp(v, "0")) { *out = 0; return 0; }
   return 1;
}

static int parse_reuse_node(hd_args *a, hd_node *n)
{
   hd_reuse_args *r = &a->reuse;
   n->used = 1;
   if (!n->child)
   {
      char *end = NULL;
      long  f = strtol(n->val, &end, 10);
      int   b;
      if (n->val[0] && end && !*end && f >= 0) { r->enabled = 1; r->frequency = (int)f; return 0; }
      if (!parse_bool_word(n->val, &b)) { r->enabled = b; return 0; }
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("preconditioner.reuse: '%s' is not supported (static reuse only: a frequency, yes/no or a block)", n->val);
      n->invalid = 2;
      return 1;
   }
   int seen_freq = 0, seen_ids = 0;
   for (hd_node *c = n->child; c; c = c->next)
   {
      c->used = 1;
      if (!strcmp(c->key, "enabled"))
      {
         if (parse_bool_word(c->val, &r->enabled)) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("Invalid value for preconditioner.reuse.enabled: '%s'", c->val); c->invalid = 2; return 1; }
      }
      else if (!strcmp(c->key, "frequency"))
      {
         char *end = NULL;
         long  f = strtol(c->val, &end, 10);
         if (!c->val[0] || !end || *end || f < 0) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("Invalid value for preconditioner.reuse.frequency: '%s'", c->val); c->invalid = 2; return 1; }
         r->frequency = (int)f; seen_freq = 1;
      }
      else if (!strcmp(c->key, "linear_system_ids") || !strcmp(c->key, "linear_solver_ids"))
      {
         /* flow list "[0, 5, 10]" or a block sequence of "- id" items */
         r->n_ids = 0;
         const char *p = c->val;
         for (hd_node *it = c->child; it; it = it->next)
         {
            it->used = 1;
            if (r->n_ids < HD_REUSE_MAX_IDS) r->ids[r->n_ids++] = atoi(it->val[0] ? it->val : it->key);
         }
         while (*p)
         {
            while (*p && (*p < '0' || *p > '9') && *p != '-') p++;
            if (!*p) break;
            char *end = NULL;
            long  v = strtol(p, &end, 10);
            if (end == p) break;
            if (v < 0 || r->n_ids >= HD_REUSE_MAX_IDS) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("Failed to parse preconditioner.reuse.linear_system_ids"); c->invalid = 2; return 1; }
            r->ids[r->n_ids++] = (int)v;
            p = end;
         }
         if (r->n_ids == 0) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("Failed to parse preconditioner.reuse.linear_system_ids"); c->invalid = 2; return 1; }
         seen_ids = 1;
      }
      else if (!strcmp(c->key, "policy"))
      {
         if (strcmp(c->val, "static")) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("preconditioner.reuse.policy '%s' is not supported (static only)", c->val); c->invalid = 2; return 1; }
      }
      else if (!strcmp(c->key, "per_timestep"))
      {
         int b = 0;
         if (parse_bool_word(c->val, &b) || b) { hd_err_set(HYPREDRV_ERROR_INVALID_VAL); hd_err_msg("preconditioner.reuse.per_timestep is not supported"); c->invalid = 2; return 1; }
      }
      else
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_KEY);
         hd_err_msg("unknown key 'preconditioner.reuse.%s'", c->key);
         c->invalid = 1;
         return 1;
      }
   }
   if (seen_freq && seen_ids)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("preconditioner.reuse: do not combine linear_system_ids with frequency");
      return 1;
   }
   return 0;
}

int hd_reuse_should_rebuild(const hd_reuse_args *r, int ls_id)
{
   /* reference precon_reuse.c:780-830 */
   if (ls_id < 0) ls_id = 0;
   if (!r || !r->enabled) return 1;
   if (r->n_ids > 0)
   {
      for (int i = 0; i < r->n_ids; i++) if (r->ids[i] == ls_id) return 1;
      return 0;
   }
   int freq = r->frequency < 0 ? 0 : r->frequency;
   return (ls_id % (freq + 1)) == 0;
}

static int parse_precon_node(hd_args *a, hd_node *n)
{
   n->used = 1;
   if (!n->child)
   {
      if (!n->val[0]) { hd_err_set(HYPREDRV_ERROR_MISSING_PRECON); hd_err_msg("empty preconditioner section"); return 1; }
      if (set_precon_method(a, n->val)) { n->invalid = 2; return 1; }
      return 0;
   }
   hd_node *method = NULL;
   for (hd_node *c = n->child; c; c = c->next)
   {
      if (!strcmp(c->key, "reuse")) { if (parse_reuse_node(a, c)) return 1; continue; }
      if (!strcmp(c->key, "preset")) { c->used = 1; if (hd_args_apply_precon_preset(a, c->val)) { c->invalid = 2; return 1; } method = c; continue; }
      if (method) { hd_err_set(HYPREDRV_ERROR_EXTRA_KEY); hd_err_msg("preconditioner section must name exactly one method"); c->invalid = 1; return 1; }
      method = c;
      if (set_precon_method(a, c->key)) { c->invalid = 1; return 1; }
      c->used = 1;
      if (a->precon_method == HD_PRECON_AMG)
      {
         hd_node *blk = c;
         /* a sequence under the method lists variants (reference args.c:928-953) */
         int nvar = 0;
         for (hd_node *it = c->child; it; it = it->next) if (it->is_seq_item) nvar++;
         if (nvar > 0)
         {
            a->num_precon_variants = nvar;
            int k = 0;
            for (hd_node *it = c->child; it; it = it->next)
               if (it->is_seq_item) { if (k == a->active_precon_variant) blk = it; it->used = 1; k++; }
         }
         parse_amg_block(blk, &a->amg);
      }
   }
   if (!method) { hd_err_set(HYPREDRV_ERROR_MISSING_PRECON); return 1; }
   return 0;
}

static int parse_precon_text(hd_args *a, const char *text)
{
   /* preset text is either a bare method name or a "method:\n  ..." block */
   char *wrapped;
   if (!strchr(text, ':')) { size_t n = strlen(text) + 32; wrapped = malloc(n); snprintf(wrapped, n, "preconditioner: %s\n", text); }
   else
   {
      size_t n = 2 * strlen(text) + 64;
      wrapped  = malloc(n);
      char *w  = wrapped + snprintf(wrapped, n, "preconditioner:\n  ");
      for (const char *p = text; *p; p++) { *w++ = *p; if (*p == '\n') { *w++ = ' '; *w++ = ' '; } }
      *w++ = '\n'; *w = 0;
   }
   hd_node *root = hd_yaml_parse(wrapped, ".");
   free(wrapped);
   if (!root) return 1;
   int rc = parse_precon_node(a, hd_yaml_find(root, "preconditioner"));
   hd_yaml_free(root);
   return rc || (hd_err_get() != 0);
}

static int parse_solver_text(hd_args *a, const char *text)
{
   char *wrapped;
   if (!strchr(text, ':')) { size_t n = strlen(text) + 32; wrapped = malloc(n); snprintf(wrapped, n, "solver: %s\n", text); }
   else
   {
      size_t n = 2 * strlen(text) + 64;
      wrapped  = malloc(n);
      char *w  = wrapped + snprintf(wrapped, n, "solver:\n  ");
      for (const char *p = text; *p; p++) { *w++ = *p; if (*p == '\n') { *w++ = ' '; *w++ = ' '; } }
      *w++ = '\n'; *w = 0;
   }
   hd_node *root = hd_yaml_parse(wrapped, ".");
   free(wrapped);
   if (!root) return 1;
   int rc = parse_solver_node(a, hd_yaml_find(root, "solver"));
   hd_yaml_free(root);
   return rc || (hd_err_get() != 0);
}

hd_args *hd_args_parse(const char *yaml_text, const char *base_dir, int n_over, char **over, bool lib_mode, bool print_tree)
{
   hd_node *root = hd_yaml_parse(yaml_text, base_dir);
   if (!root) return NULL;
   /* CLI overrides: optional leading -a/--args, then pairs */
   int i0 = 0;
   if (n_over > 0 && (!strcmp(over[0], "-a") || !strcmp(over[0], "--args"))) i0 = 1;
   if ((n_over - i0) % 2 != 0)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("override arguments must come in '--path:to:key value' pairs");
      hd_yaml_free(root);
      return NULL;
   }
   for (int i = i0; i + 1 < n_over; i += 2) hd_yaml_override(root, over[i], over[i + 1]);

   hd_args *a = calloc(1, sizeof(hd_args));
   hd_args_defaults(a, lib_mode);
   /* duplicate / unknown top-level keys */
   static const char *top[] = {"general", "linear_system", "solver", "preconditioner", NULL};
   for (hd_node *c = root->child; c; c = c->next)
   {
      int known = 0;
      for (const char **t = top; *t; t++) if (!strcmp(*t, c->key)) known = 1;
      if (!known) mark_invalid(c, 1, "<top level>");
      for (hd_node *d = c->next; d; d = d->next)
         if (!strcmp(c->key, d->key)) { hd_err_set(HYPREDRV_ERROR_EXTRA_KEY); hd_err_msg("duplicate top-level key '%s'", c->key); d->invalid = 1; }
   }
   hd_node *n;
   if ((n = hd_yaml_find(root, "general"))) { n->used = 1; apply_fields(n, f_general, &a->general, "general", NULL); }
   if ((n = hd_yaml_find(root, "linear_system"))) { n->used = 1; apply_fields(n, f_ls, &a->ls, "linear_system", NULL); }
   if ((n = hd_yaml_find(root, "solver"))) parse_solver_node(a, n);
   if ((n = hd_yaml_find(root, "preconditioner"))) parse_precon_node(a, n);
   else { hd_err_set(HYPREDRV_ERROR_MISSING_KEY); hd_err_msg("missing mandatory key 'preconditioner'"); }

   if (hd_err_get())
   {
      hd_err_set(HYPREDRV_ERROR_YAML_TREE_INVALID);
      fprintf(stderr, "Invalid configuration:\n");
      hd_yaml_print(root, stderr);
      hd_yaml_free(root);
      free(a);
      return NULL;
   }
   if (print_tree && a->general.print_config_params)
   {
      printf("------------------------------------------------------------------------------------\n");
      hd_yaml_print(root, stdout);
      printf("------------------------------------------------------------------------------------\n");
   }
   hd_yaml_free(root);
   return a;
}

/* options struct -> device parameter block (reference hypredrv_AMGCreate, amg.c:863-1035) */
void hd_amg_to_hdk(const hd_amg_args *a, hdk_amg_params *p)
{
   hdk_amg_default_params(p);
   p->coarsen_type = a->coarsen_type; p->strong_th = a->strong_th; p->max_row_sum = a->max_row_sum;
   p->max_coarse_size = a->max_coarse_size; p->min_coarse_size = a->min_coarse_size; p->max_levels = a->max_levels;
   p->interp_type = a->prolongation_type; p->max_nnz_row = a->max_nnz_row; p->trunc_factor = a->trunc_factor;
   p->relax_down = a->down_type; p->relax_up = a->up_type; p->relax_coarse = a->coarse_type;
   p->sweeps_down = a->down_sweeps > -1 ? a->down_sweeps : a->num_sweeps;
   p->sweeps_up = a->up_sweeps > -1 ? a->up_sweeps : a->num_sweeps;
   p->sweeps_coarse = a->coarse_sweeps > -1 ? a->coarse_sweeps : a->num_sweeps;
   p->relax_weight = a->weight; p->outer_weight = a->outer_weight;
   p->keep_transpose = a->keep_transpose; p->print_level = a->print_level;
   p->num_functions = a->num_functions;
   p->agg_num_levels = a->agg_num_levels; p->agg_num_paths = a->agg_num_paths;
   p->agg_interp_type = a->agg_prolongation_type; p->agg_max_nnz_row = a->agg_max_nnz_row;
   p->agg_trunc_factor = a->agg_trunc_factor;
   p->cheby_order = a->cheby_order; p->cheby_fraction = a->cheby_fraction; p->cheby_eig_est = a->cheby_eig_est;
   p->cheby_variant = a->cheby_variant; p->cheby_scale = a->cheby_scale;
}

/* systems AMG (num_functions > 1) runs hypre's unknown approach only: the nodal approach and
 * filter_functions would otherwise be ignored silently, so they are rejected; so are the aggressive
 * coarsening options the device setup cannot honour */
int hd_amg_check(const hd_amg_args *a)
{
   int bad = 0;
   if (a->num_functions < 1)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("amg:coarsening:num_functions must be at least 1 (got %d)", a->num_functions);
      bad = 1;
   }
   if (a->num_functions > 1 && a->nodal)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("amg:coarsening:nodal is not supported with num_functions = %d: only the unknown approach (nodal: 0) has a device setup", a->num_functions);
      bad = 1;
   }
   if (a->num_functions > 1 && a->filter_functions)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("amg:coarsening:filter_functions is not supported with num_functions = %d", a->num_functions);
      bad = 1;
   }
   /* aggressive coarsening: the keys only matter with num_levels > 0 */
   if (a->agg_num_levels < 0)
   {
      hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
      hd_err_msg("amg:aggressive:num_levels must be at least 0 (got %d)", a->agg_num_levels);
      bad = 1;
   }
   if (a->agg_num_levels > 0)
   {
      if (a->agg_num_paths < 1)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:aggressive:num_paths must be at least 1 (got %d)", a->agg_num_paths);
         bad = 1;
      }
      if (a->agg_max_nnz_row < 0)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:aggressive:max_nnz_row must be at least 0 (got %d)", a->agg_max_nnz_row);
         bad = 1;
      }
      if (!(a->agg_trunc_factor >= 0.0 && a->agg_trunc_factor < 1.0))
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:aggressive:trunc_factor must be in [0, 1) (got %g)", a->agg_trunc_factor);
         bad = 1;
      }
      if (a->agg_prolongation_type != 4)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:aggressive:prolongation_type %d is not supported: only multipass (4) has a device setup", a->agg_prolongation_type);
         bad = 1;
      }
      if (a->num_functions > 1)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:aggressive:num_levels = %d is not supported with num_functions = %d", a->agg_num_levels, a->num_functions);
         bad = 1;
      }
   }
   /* Chebyshev smoothing: the keys only matter when a phase relaxes with type 16 */
   if (a->down_type == 16 || a->up_type == 16 || a->coarse_type == 16)
   {
      if (a->cheby_order < 1 || a->cheby_order > 4)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:order must be in 1..4 (got %d)", a->cheby_order);
         bad = 1;
      }
      if (!(a->cheby_fraction > 0.0 && a->cheby_fraction <= 1.0))
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:fraction must be in (0, 1] (got %g)", a->cheby_fraction);
         bad = 1;
      }
      if (a->cheby_eig_est < 0)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:eig_est must be at least 0 (got %d)", a->cheby_eig_est);
         bad = 1;
      }
      if (a->cheby_variant == 1)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:variant 1 is not supported: only variant 0 has a device implementation");
         bad = 1;
      }
      else if (a->cheby_variant != 0)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:variant must be 0 or 1 (got %d)", a->cheby_variant);
         bad = 1;
      }
      if (a->cheby_scale != 0 && a->cheby_scale != 1)
      {
         hd_err_set(HYPREDRV_ERROR_INVALID_VAL);
         hd_err_msg("amg:relaxation:chebyshev:scale must be 0 or 1 (got %d)", a->cheby_scale);
         bad = 1;
      }
   }
   return bad;
}
