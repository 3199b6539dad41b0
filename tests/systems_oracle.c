/* systems_oracle.c -- CPU restatement of BoomerAMG's systems setup, num_functions > 1 with the
 * unknown approach (nodal = 0); TEST INFRASTRUCTURE ONLY.
 *
 * Built on the parity oracle (oracle/oracle.h, liboracle.so): PMIS, RAP, the transpose, the l1
 * norms, the coarse solve and the Krylov methods are the oracle's own functions.  What changes
 * with num_functions > 1 is restated here (hypre: parcsr_ls/par_strength.c num_functions > 1
 * branch, par_lr_interp.c hypre_BoomerAMGBuildExtPIInterp, par_coarse_parms.c):
 *   - strength: row_scale and row_sum over the off-diagonals of the row's own function only; an
 *     entry is strong only if it passes the threshold and couples equal functions;
 *   - extended+i: a weak coupling to another function is dropped instead of lumped into the
 *     diagonal (C-hat comes from S, which has no cross-function entry);
 *   - coarse labels: the labels of the C points in coarse order.
 * The level loop, interpolation and truncation otherwise follow oracle/amg_setup.c line for line,
 * so with num_functions == 1 the result is the oracle's oamg_setup. */
#include "oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define C_PT 1
#define F_PT -1
#define SF_PT -3

typedef struct
{
   oamg *h;                     /* a hierarchy in the oracle's own layout: oamg_destroy frees it */
   int   num_functions;
   int  *dof[OAMG_MAX_LEVELS];  /* function label of every row of level l */
} osys;

ocsr *osys_strength(const ocsr *A, double theta, double max_row_sum, int nf, const int *dof)
{
   int   n    = A->nrows;
   int  *cnt  = (int *)calloc((size_t)n + 1, sizeof(int));
   char *keep = (char *)malloc((size_t)(A->ia[n] > 0 ? A->ia[n] : 1));
#pragma omp parallel for schedule(static)
   for (int i = 0; i < n; i++)
   {
      int b = A->ia[i], e = A->ia[i + 1];
      int c = 0;
      if (e > b)
      {
         double diag = A->a[b], row_scale = 0.0, row_sum = diag;
         for (int k = b + 1; k < e; k++)
         {
            if (nf > 1 && dof[A->ja[k]] != dof[i]) continue;
            double v = A->a[k];
            if (diag < 0) row_scale = row_scale > v ? row_scale : v;
            else row_scale = row_scale < v ? row_scale : v;
            row_sum += v;
         }
         keep[b] = 0;
         if (fabs(row_sum) > fabs(diag) * max_row_sum && max_row_sum < 1.0)
         {
            for (int k = b + 1; k < e; k++) keep[k] = 0;
         }
         else
         {
            for (int k = b + 1; k < e; k++)
            {
               int strong = (diag < 0) ? !(A->a[k] <= theta * row_scale) : !(A->a[k] >= theta * row_scale);
               keep[k]    = strong && (nf == 1 || dof[A->ja[k]] == dof[i]);
               c += keep[k];
            }
         }
      }
      cnt[i + 1] = c;
   }
   for (int i = 0; i < n; i++) cnt[i + 1] += cnt[i];
   ocsr *S = ocsr_alloc(n, n, cnt[n], 0);
   memcpy(S->ia, cnt, sizeof(int) * ((size_t)n + 1));
#pragma omp parallel for schedule(static)
   for (int i = 0; i < n; i++)
   {
      int p = S->ia[i];
      for (int k = A->ia[i] + 1; k < A->ia[i + 1]; k++)
         if (keep[k]) S->ja[p++] = A->ja[k];
   }
   free(cnt);
   free(keep);
   return S;
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

/* oamg_extpi_interp (oracle/amg_setup.c) with the systems weak-connection branch */
static ocsr *osys_extpi_interp(const ocsr *A, const ocsr *S, int *cf, int max_elmts, double trunc_factor,
                               int *n_coarse_out, int nf, const int *dof)
{
   int  n   = A->nrows;
   int *f2c = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   int *pi  = (int *)calloc((size_t)n + 1, sizeof(int));
   int  nc  = 0;
   for (int i = 0; i < n; i++) f2c[i] = (cf[i] >= 0) ? nc++ : -1;

#pragma omp parallel
   {
      int *mark = (int *)malloc(sizeof(int) * ((size_t)n + 1));
      for (int i = 0; i < n; i++) mark[i] = -1;
#pragma omp for schedule(static)
      for (int i = 0; i < n; i++)
      {
         int c = 0;
         if (cf[i] >= 0) c = 1;
         else if (cf[i] != SF_PT)
         {
            for (int jj = S->ia[i]; jj < S->ia[i + 1]; jj++)
            {
               int i1 = S->ja[jj];
               if (cf[i1] >= 0) { if (mark[i1] != i) { mark[i1] = i; c++; } }
               else if (cf[i1] != SF_PT)
                  for (int kk = S->ia[i1]; kk < S->ia[i1 + 1]; kk++)
                  {
                     int k1 = S->ja[kk];
                     if (cf[k1] >= 0 && mark[k1] != i) { mark[k1] = i; c++; }
                  }
            }
         }
         pi[i + 1] = c;
      }
      free(mark);
   }
   for (int i = 0; i < n; i++) pi[i + 1] += pi[i];
   int     nnzP = pi[n];
   int    *pj   = (int *)malloc(sizeof(int) * ((size_t)nnzP + 1));
   double *pd   = (double *)malloc(sizeof(double) * ((size_t)nnzP + 1));

#pragma omp parallel
   {
      int *mark = (int *)malloc(sizeof(int) * ((size_t)n + 1));
      for (int i = 0; i < n; i++) mark[i] = -1;
#pragma omp for schedule(static)
      for (int i = 0; i < n; i++)
      {
         int jb = pi[i], jc = pi[i];
         if (cf[i] >= 0) { pj[jc] = f2c[i]; pd[jc] = 1.0; continue; }
         if (cf[i] == SF_PT) continue;
         const int sfm = -2 - i;
         for (int jj = S->ia[i]; jj < S->ia[i + 1]; jj++)
         {
            int i1 = S->ja[jj];
            if (cf[i1] >= 0)
            {
               if (mark[i1] < jb) { mark[i1] = jc; pj[jc] = f2c[i1]; pd[jc] = 0.0; jc++; }
            }
            else if (cf[i1] != SF_PT)
            {
               mark[i1] = sfm;
               for (int kk = S->ia[i1]; kk < S->ia[i1 + 1]; kk++)
               {
                  int k1 = S->ja[kk];
                  if (cf[k1] >= 0 && mark[k1] < jb) { mark[k1] = jc; pj[jc] = f2c[k1]; pd[jc] = 0.0; jc++; }
               }
            }
         }
         int    je       = jc;
         double diagonal = A->a[A->ia[i]];
         for (int jj = A->ia[i] + 1; jj < A->ia[i + 1]; jj++)
         {
            int i1 = A->ja[jj];
            if (mark[i1] >= jb && mark[i1] < je) pd[mark[i1]] += A->a[jj];
            else if (mark[i1] == sfm)
            {
               double sum = 0.0;
               int    sgn = A->a[A->ia[i1]] < 0 ? -1 : 1;
               for (int j1 = A->ia[i1] + 1; j1 < A->ia[i1 + 1]; j1++)
               {
                  int i2 = A->ja[j1];
                  if (((mark[i2] >= jb && mark[i2] < je) || i2 == i) && sgn * A->a[j1] < 0) sum += A->a[j1];
               }
               if (sum != 0)
               {
                  double distribute = A->a[jj] / sum;
                  for (int j1 = A->ia[i1] + 1; j1 < A->ia[i1 + 1]; j1++)
                  {
                     int i2 = A->ja[j1];
                     if (mark[i2] >= jb && mark[i2] < je && sgn * A->a[j1] < 0)
                        pd[mark[i2]] += distribute * A->a[j1];
                     if (i2 == i && sgn * A->a[j1] < 0) diagonal += distribute * A->a[j1];
                  }
               }
               else diagonal += A->a[jj];
            }
            else if (cf[i1] != SF_PT && (nf == 1 || dof[i] == dof[i1])) diagonal += A->a[jj];
         }
         if (diagonal != 0.0)
            for (int jj = jb; jj < je; jj++) pd[jj] /= -diagonal;
      }
      free(mark);
   }

   int *newlen = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   for (int i = 0; i < n; i++)
   {
      int b = pi[i], e = pi[i + 1], len = e - b;
      if (trunc_factor > 0.0 && len > 0)
      {
         double maxc = 0.0, row_sum = 0.0, scale = 0.0;
         for (int k = b; k < e; k++) if (fabs(pd[k]) > maxc) maxc = fabs(pd[k]);
         maxc *= trunc_factor;
         int w = b;
         for (int k = b; k < e; k++)
         {
            row_sum += pd[k];
            if (!(fabs(pd[k]) < maxc)) { scale += pd[k]; pj[w] = pj[k]; pd[w] = pd[k]; w++; }
         }
         if (scale != 0.0 && scale != row_sum)
         {
            scale = row_sum / scale;
            for (int k = b; k < w; k++) pd[k] *= scale;
         }
         len = w - b;
         e   = w;
      }
      if (max_elmts > 0 && len > max_elmts)
      {
         double row_sum = 0.0, scale = 0.0;
         for (int k = b; k < e; k++) row_sum += pd[k];
         qsort2abs(pj + b, pd + b, 0, len - 1);
         for (int k = 0; k < max_elmts; k++) scale += pd[b + k];
         if (scale != 0.0 && scale != row_sum)
         {
            scale = row_sum / scale;
            for (int k = 0; k < max_elmts; k++) pd[b + k] *= scale;
         }
         len = max_elmts;
      }
      newlen[i] = len;
   }
   int tot = 0;
   for (int i = 0; i < n; i++) tot += newlen[i];
   ocsr *P = ocsr_alloc(n, nc, tot, 1);
   int   w = 0;
   for (int i = 0; i < n; i++)
   {
      P->ia[i] = w;
      for (int k = 0; k < newlen[i]; k++) { P->ja[w] = pj[pi[i] + k]; P->a[w] = pd[pi[i] + k]; w++; }
   }
   P->ia[n] = w;
   for (int i = 0; i < n; i++) if (cf[i] == SF_PT) cf[i] = F_PT;
   if (n_coarse_out) *n_coarse_out = nc;
   free(newlen); free(pj); free(pd); free(pi); free(f2c);
   return P;
}

static int relax_l1_option(int type)
{
   if (type == 18) return 1;
   if (type == 8 || type == 13 || type == 14) return 4;
   return 5;
}

/* oamg_setup (oracle/amg_setup.c) with labels: dof_func labels the rows of A (NULL: hypre's
 * interleaved default, row % num_functions). */
osys *osys_setup(const ocsr *Ain, const oamg_params *prm, int num_functions, const int *dof_func)
{
   osys *s = (osys *)calloc(1, sizeof(osys));
   oamg *h = (oamg *)calloc(1, sizeof(oamg));
   s->h = h;
   s->num_functions = num_functions;
   h->prm = *prm;
   ocsr *A0 = ocsr_from_arrays(Ain->nrows, Ain->ncols, Ain->ia, Ain->ja, Ain->a);
   ocsr_diag_first(A0);
   h->A[0]   = A0;
   s->dof[0] = (int *)malloc(sizeof(int) * ((size_t)A0->nrows + 1));
   for (int i = 0; i < A0->nrows; i++) s->dof[0][i] = dof_func ? dof_func[i] : i % num_functions;
   int level = 0, not_finished = prm->max_levels > 1;
   while (not_finished)
   {
      ocsr   *A    = h->A[level];
      int     n    = A->nrows;
      ocsr   *S    = osys_strength(A, prm->strong_th, prm->max_row_sum, num_functions, s->dof[level]);
      int    *cf   = (int *)calloc((size_t)n + 1, sizeof(int));
      double *meas = (double *)calloc((size_t)n + 1, sizeof(double));
      if (prm->coarsen_type == 10)
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
      h->P[level] = osys_extpi_interp(A, S, cf, prm->max_nnz_row, prm->trunc_factor, &nc2, num_functions, s->dof[level]);
      s->dof[level + 1] = (int *)malloc(sizeof(int) * ((size_t)nc2 + 1));
      for (int i = 0, ic = 0; i < n; i++)
         if (cf[i] == C_PT) s->dof[level + 1][ic++] = s->dof[level][i];
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

oamg *osys_hierarchy(osys *s) { return s->h; }
const int *osys_dof(const osys *s, int level) { return (level >= 0 && level < OAMG_MAX_LEVELS) ? s->dof[level] : NULL; }

void osys_destroy(osys *s)
{
   if (!s) return;
   oamg_destroy(s->h);
   for (int l = 0; l < OAMG_MAX_LEVELS; l++) free(s->dof[l]);
   free(s);
}
