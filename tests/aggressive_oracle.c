/* aggressive_oracle.c -- CPU restatement of aggressive coarsening with multipass interpolation
 * (BoomerAMG agg_num_levels > 0, agg_interp_type 4); TEST INFRASTRUCTURE ONLY.
 *
 * Built on the parity oracle (oracle/oracle.h, liboracle.so): strength, PMIS, RAP, the transpose,
 * the l1 norms, the coarse solve and the Krylov methods are the oracle's own functions.  What
 * aggressive coarsening adds on a level l < agg_num_levels is restated here (after hypre's
 * hypre_BoomerAMGCreate2ndS, hypre_BoomerAMGCorrectCFMarker2 and hypre_BoomerAMGBuildModMultipass;
 * hypre parity is not pinned, this file is the rule the device is compared with):
 *   - S2: for first-stage C points i != j, paths(i,j) = [j in S_i] + |{k in S_i : cf1[k] != C,
 *     j in S_k}|; row c(i) holds c(j) for paths(i,j) >= num_paths, ascending, never c(i);
 *   - a second PMIS on S2 (the oracle's oamg_pmis); a first-stage C point that it makes F becomes -2;
 *   - multipass interpolation: pass numbers by breadth-first sweeps along S from the C points,
 *     pass-2 rows from the strong C neighbours, pass-p rows (p >= 3) as the weighted sum of the
 *     truncated pass-(p-1) rows of the strong neighbours, each pass truncated before the next.
 * Other levels follow oracle/amg_setup.c line for line, so with agg_num_levels == 0 the result is
 * the oracle's oamg_setup. */
#include "oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define C_PT 1
#define F_PT -1
#define Z_PT -2
#define SF_PT -3

typedef struct
{
   int    num_levels;   /* agg_num_levels */
   int    num_paths;    /* agg_num_paths */
   int    max_nnz_row;  /* agg_max_nnz_row (0: no limit) */
   double trunc_factor; /* agg_trunc_factor */
} oagg_params;

typedef struct
{
   oamg *h;                    /* a hierarchy in the oracle's own layout: oamg_destroy frees it */
   ocsr *S2[OAMG_MAX_LEVELS];  /* second-stage strength of the aggressive levels (NULL elsewhere) */
   int  *pass[OAMG_MAX_LEVELS];
} oagg;

static int cmp_int(const void *a, const void *b)
{
   int x = *(const int *)a, y = *(const int *)b;
   return (x > y) - (x < y);
}

/* second-stage strength over the first-stage C points (cf1 == 1), numbered in row order */
ocsr *oagg_s2(const ocsr *S, const int *cf1, int num_paths)
{
   int  n   = S->nrows;
   int *c   = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   int  nc1 = 0;
   for (int i = 0; i < n; i++) c[i] = (cf1[i] == C_PT) ? nc1++ : -1;
   int  *cnt  = (int *)calloc((size_t)nc1 + 1, sizeof(int));
   int  *list = (int *)malloc(sizeof(int) * ((size_t)nc1 + 1));
   int  *ia   = (int *)calloc((size_t)nc1 + 1, sizeof(int));
   int   cap  = 1024, nnz = 0;
   int  *ja   = (int *)malloc(sizeof(int) * (size_t)cap);
   for (int i = 0; i < n; i++)
   {
      if (c[i] < 0) continue;
      int m = 0;
      for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
      {
         int j = S->ja[k];
         if (cf1[j] == C_PT) { if (cnt[c[j]]++ == 0) list[m++] = c[j]; }
         else
            for (int kk = S->ia[j]; kk < S->ia[j + 1]; kk++)
            {
               int j2 = S->ja[kk];
               if (cf1[j2] == C_PT && j2 != i && cnt[c[j2]]++ == 0) list[m++] = c[j2];
            }
      }
      int row0 = nnz;
      for (int t = 0; t < m; t++)
      {
         if (cnt[list[t]] >= num_paths)
         {
            if (nnz == cap) { cap *= 2; ja = (int *)realloc(ja, sizeof(int) * (size_t)cap); }
            ja[nnz++] = list[t];
         }
         cnt[list[t]] = 0;
      }
      qsort(ja + row0, (size_t)(nnz - row0), sizeof(int), cmp_int);
      ia[c[i] + 1] = nnz;
   }
   ocsr *S2 = ocsr_alloc(nc1, nc1, nnz, 0);
   memcpy(S2->ia, ia, sizeof(int) * ((size_t)nc1 + 1));
   if (nnz) memcpy(S2->ja, ja, sizeof(int) * (size_t)nnz);
   free(c); free(cnt); free(list); free(ia); free(ja);
   return S2;
}

/* first-stage C points that the second PMIS makes F become -2; every other point keeps cf1 */
void oagg_combine(int n, const int *cf1, const int *cf2, int *cf)
{
   for (int i = 0, ic = 0; i < n; i++)
   {
      cf[i] = cf1[i];
      if (cf1[i] == C_PT) { if (cf2[ic] == F_PT) cf[i] = Z_PT; ic++; }
   }
}

/* pass[i] = 1 for C points, p + 1 for a point with a strong neighbour in pass p (breadth first),
 * 0 for points no sweep reaches; returns the largest pass */
int oagg_pass(const ocsr *S, const int *cf, int *pass)
{
   int n = S->nrows, p = 1, assigned = 1;
   for (int i = 0; i < n; i++) pass[i] = (cf[i] == C_PT) ? 1 : 0;
   while (assigned)
   {
      assigned = 0;
      for (int i = 0; i < n; i++)
      {
         if (pass[i] != 0) continue;
         for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
            if (pass[S->ja[k]] == p) { pass[i] = p + 1; assigned++; break; }
      }
      if (assigned) p++;
   }
   return p;
}

/* hypre_qsort2abs (utilities/qsort.c), as in oracle/amg_setup.c */
static void swap2(int *v, double *w, int i, int j)
{
   int    t = v[i]; v[i] = v[j]; v[j] = t;
   double d = w[i]; w[i] = w[j]; w[j] = d;
}
static void qsort2abs(int *v, double *w, int left, int right)
{
   if (left >= right) return;
   swap2(v, w, left, (left + right) / 2);
   int last = left;
   for (int i = left + 1; i <= right; i++)
      if (fabs(w[i]) > fabs(w[left])) swap2(v, w, ++last, i);
   swap2(v, w, left, last);
   qsort2abs(v, w, left, last - 1);
   qsort2abs(v, w, last + 1, right);
}

/* the truncation loop of oamg_extpi_interp on one row; returns the new length */
static int trunc_row(int *pj, double *pd, int len, double trunc_factor, int max_elmts)
{
   if (trunc_factor > 0.0 && len > 0)
   {
      double maxc = 0.0, row_sum = 0.0, scale = 0.0;
      for (int k = 0; k < len; k++) if (fabs(pd[k]) > maxc) maxc = fabs(pd[k]);
      maxc *= trunc_factor;
      int w = 0;
      for (int k = 0; k < len; k++)
      {
         row_sum += pd[k];
         if (!(fabs(pd[k]) < maxc)) { scale += pd[k]; pj[w] = pj[k]; pd[w] = pd[k]; w++; }
      }
      if (scale != 0.0 && scale != row_sum)
      {
         scale = row_sum / scale;
         for (int k = 0; k < w; k++) pd[k] *= scale;
      }
      len = w;
   }
   if (max_elmts > 0 && len > max_elmts)
   {
      double row_sum = 0.0, scale = 0.0;
      for (int k = 0; k < len; k++) row_sum += pd[k];
      qsort2abs(pj, pd, 0, len - 1);
      for (int k = 0; k < max_elmts; k++) scale += pd[k];
      if (scale != 0.0 && scale != row_sum)
      {
         scale = row_sum / scale;
         for (int k = 0; k < max_elmts; k++) pd[k] *= scale;
      }
      len = max_elmts;
   }
   return len;
}

/* multipass interpolation (after hypre_BoomerAMGBuildModMultipass).  a_ij of a strong neighbour j
 * is the entry of A that S took it from: S keeps A's column order, so both rows are walked together.
 * On return SF_PT (-3) entries of cf are reset to F_PT (-1); -2 stays. */
ocsr *oagg_multipass(const ocsr *A, const ocsr *S, int *cf, const int *pass, int max_elmts, double trunc_factor,
                     int *n_coarse_out)
{
   int  n   = A->nrows;
   int *f2c = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   int  nc  = 0;
   for (int i = 0; i < n; i++) f2c[i] = (cf[i] == C_PT) ? nc++ : -1;
   int     nnzS = S->ia[n];
   double *sval = (double *)malloc(sizeof(double) * ((size_t)nnzS + 1));
   for (int i = 0; i < n; i++)
   {
      int ka = A->ia[i] + 1;
      for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
      {
         while (A->ja[ka] != S->ja[k]) ka++;
         sval[k] = A->a[ka++];
      }
   }
   int maxp = 0;
   for (int i = 0; i < n; i++) if (pass[i] > maxp) maxp = pass[i];
   int    **rc  = (int **)calloc((size_t)n + 1, sizeof(int *));
   double **rv  = (double **)calloc((size_t)n + 1, sizeof(double *));
   int     *rl  = (int *)calloc((size_t)n + 1, sizeof(int));
   int     *mark = (int *)malloc(sizeof(int) * ((size_t)nc + 1));
   for (int c = 0; c < nc; c++) mark[c] = -1;
   for (int i = 0; i < n; i++)
      if (pass[i] == 1)
      {
         rc[i] = (int *)malloc(sizeof(int)); rv[i] = (double *)malloc(sizeof(double));
         rc[i][0] = f2c[i]; rv[i][0] = 1.0; rl[i] = 1;
      }
   for (int p = 2; p <= maxp; p++)
      for (int i = 0; i < n; i++)
      {
         if (pass[i] != p) continue;
         double nneg = 0.0, npos = 0.0, cneg = 0.0, cpos = 0.0;
         for (int k = A->ia[i] + 1; k < A->ia[i + 1]; k++)
         {
            if (A->a[k] < 0) nneg += A->a[k];
            else npos += A->a[k];
         }
         for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
            if (pass[S->ja[k]] == p - 1)
            {
               if (sval[k] < 0) cneg += sval[k];
               else cpos += sval[k];
            }
         double d = A->a[A->ia[i]];
         if (cpos == 0.0) d += npos;
         if (d == 0.0) continue; /* empty row */
         double alfa = cneg != 0.0 ? nneg / cneg / d : 0.0;
         double beta = cpos != 0.0 ? npos / cpos / d : 0.0;
         int     len = 0, cap = 0;
         int    *pj  = NULL;
         double *pd  = NULL;
         for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
         {
            int j = S->ja[k];
            if (pass[j] != p - 1) continue;
            double w = sval[k] < 0 ? -(alfa * sval[k]) : -(beta * sval[k]);
            if (p == 2)
            {
               if (len == cap) { cap = cap ? 2 * cap : 8; pj = (int *)realloc(pj, sizeof(int) * (size_t)cap); pd = (double *)realloc(pd, sizeof(double) * (size_t)cap); }
               pj[len] = f2c[j]; pd[len] = w; len++;
               continue;
            }
            for (int t = 0; t < rl[j]; t++)
            {
               int    col  = rc[j][t];
               double prod = w * rv[j][t];
               if (mark[col] < 0)
               {
                  if (len == cap) { cap = cap ? 2 * cap : 8; pj = (int *)realloc(pj, sizeof(int) * (size_t)cap); pd = (double *)realloc(pd, sizeof(double) * (size_t)cap); }
                  mark[col] = len; pj[len] = col; pd[len] = prod; len++;
               }
               else pd[mark[col]] += prod;
            }
         }
         for (int t = 0; t < len; t++) mark[pj[t]] = -1;
         rl[i] = trunc_row(pj, pd, len, trunc_factor, max_elmts);
         rc[i] = pj; rv[i] = pd;
      }
   int tot = 0;
   for (int i = 0; i < n; i++) tot += rl[i];
   ocsr *P = ocsr_alloc(n, nc, tot, 1);
   int   w = 0;
   for (int i = 0; i < n; i++)
   {
      P->ia[i] = w;
      for (int t = 0; t < rl[i]; t++) { P->ja[w] = rc[i][t]; P->a[w] = rv[i][t]; w++; }
      free(rc[i]); free(rv[i]);
   }
   P->ia[n] = w;
   for (int i = 0; i < n; i++) if (cf[i] == SF_PT) cf[i] = F_PT;
   if (n_coarse_out) *n_coarse_out = nc;
   free(rc); free(rv); free(rl); free(mark); free(sval); free(f2c);
   return P;
}

static int relax_l1_option(int type)
{
   if (type == 18) return 1;
   if (type == 8 || type == 13 || type == 14) return 4;
   return 5;
}

/* oamg_setup (oracle/amg_setup.c) with aggressive coarsening on levels l < agg->num_levels */
oagg *oagg_setup(const ocsr *Ain, const oamg_params *prm, const oagg_params *agg)
{
   oagg *s = (oagg *)calloc(1, sizeof(oagg));
   oamg *h = (oamg *)calloc(1, sizeof(oamg));
   s->h = h;
   h->prm = *prm;
   ocsr *A0 = ocsr_from_arrays(Ain->nrows, Ain->ncols, Ain->ia, Ain->ja, Ain->a);
   ocsr_diag_first(A0);
   h->A[0] = A0;
   int level = 0, not_finished = prm->max_levels > 1;
   while (not_finished)
   {
      ocsr   *A    = h->A[level];
      int     n    = A->nrows;
      ocsr   *S    = oamg_strength(A, prm->strong_th, prm->max_row_sum);
      int    *cf   = (int *)calloc((size_t)n + 1, sizeof(int));
      double *meas = (double *)calloc((size_t)n + 1, sizeof(double));
      const int aggressive = level < agg->num_levels;
      if (aggressive)
      {
         oamg_pmis(S, prm->rand_seed, 0, cf, meas);
         int nc1 = 0;
         for (int i = 0; i < n; i++) nc1 += (cf[i] == C_PT);
         if (nc1 > 0)
         {
            ocsr *S2  = oagg_s2(S, cf, agg->num_paths);
            int  *cf2 = (int *)calloc((size_t)nc1 + 1, sizeof(int));
            oamg_pmis(S2, prm->rand_seed, 0, cf2, NULL);
            oagg_combine(n, cf, cf2, cf);
            free(cf2);
            s->S2[level] = S2;
         }
      }
      else if (prm->coarsen_type == 10)
      {
         oamg_rs_first_pass(S, cf);
         oamg_pmis(S, prm->rand_seed, 1, cf, meas);
      }
      else oamg_pmis(S, prm->rand_seed, 0, cf, meas);
      int nc = 0;
      for (int i = 0; i < n; i++) nc += (cf[i] == 1);
      h->S[level] = S; h->measure[level] = meas;
      h->cf_raw[level] = (int *)malloc(sizeof(int) * ((size_t)n + 1));
      memcpy(h->cf_raw[level], cf, sizeof(int) * (size_t)n);
      h->cf[level] = cf;
      if (nc == 0 || nc == n || nc < prm->min_coarse_size) break;
      int nc2;
      if (aggressive)
      {
         s->pass[level] = (int *)malloc(sizeof(int) * ((size_t)n + 1));
         oagg_pass(S, cf, s->pass[level]);
         h->P[level] = oagg_multipass(A, S, cf, s->pass[level], agg->max_nnz_row, agg->trunc_factor, &nc2);
      }
      else h->P[level] = oamg_extpi_interp(A, S, cf, prm->max_nnz_row, prm->trunc_factor, &nc2);
      h->R[level]     = ocsr_transpose(h->P[level]);
      h->A[level + 1] = oamg_rap(h->R[level], A, h->P[level]);
      level++;
      if (level == prm->max_levels - 1 || nc <= prm->max_coarse_size) not_finished = 0;
      if (level >= OAMG_MAX_LEVELS - 1) not_finished = 0;
   }
   h->nlev = level + 1;
   for (int l = 0; l < h->nlev; l++)
   {
      int n = h->A[l]->nrows;
      h->l1_down[l] = (double *)malloc(sizeof(double) * ((size_t)n + 1));
      h->l1_up[l]   = (double *)malloc(sizeof(double) * ((size_t)n + 1));
      oamg_l1_norms(h->A[l], relax_l1_option(prm->relax_down), h->l1_down[l]);
      oamg_l1_norms(h->A[l], relax_l1_option(prm->relax_up), h->l1_up[l]);
      h->u[l]  = (double *)calloc((size_t)n + 1, sizeof(double));
      h->f[l]  = (double *)calloc((size_t)n + 1, sizeof(double));
      h->t[l]  = (double *)calloc((size_t)n + 1, sizeof(double));
      h->t2[l] = (double *)calloc((size_t)n + 1, sizeof(double));
   }
   if (prm->relax_coarse == 9 || prm->relax_coarse == 99 || h->nlev == 1)
   {
      ocsr *Ac = h->A[h->nlev - 1];
      int   n  = Ac->nrows;
      if ((double)n * n < 2.0e8)
      {
         h->ge_n = n;
         h->ge   = (double *)calloc((size_t)n * n + 1, sizeof(double));
         for (int i = 0; i < n; i++)
            for (int k = Ac->ia[i]; k < Ac->ia[i + 1]; k++) h->ge[(size_t)i * n + Ac->ja[k]] += Ac->a[k];
      }
   }
   return s;
}

oamg *oagg_hierarchy(oagg *s) { return s->h; }
ocsr *oagg_s2_of(const oagg *s, int level) { return (level >= 0 && level < OAMG_MAX_LEVELS) ? s->S2[level] : NULL; }
const int *oagg_pass_of(const oagg *s, int level) { return (level >= 0 && level < OAMG_MAX_LEVELS) ? s->pass[level] : NULL; }

void oagg_destroy(oagg *s)
{
   if (!s) return;
   oamg_destroy(s->h);
   for (int l = 0; l < OAMG_MAX_LEVELS; l++) { ocsr_free(s->S2[l]); free(s->pass[l]); }
   free(s);
}
