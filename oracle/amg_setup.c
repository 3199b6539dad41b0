/* amg_setup.c -- CPU restatement of the BoomerAMG setup phase (TEST INFRASTRUCTURE ONLY).
 *
 * Reference trigger: HYPRE_BoomerAMGSetup via src/internal/solver.c:296 /
 * src/internal/precon.c:107, options from src/internal/amg.c:863-1035.
 * The algorithms restate hypre (third-party, not vendored): parcsr_ls/par_strength.c,
 * par_coarsen.c (PMIS/HMIS, Ruge first pass), par_indepset.c, par_lr_interp.c
 * (extended+i), par_interp.c (truncation), utilities/qsort.c (hypre_qsort2abs),
 * par_rap.c (hypre_BoomerAMGBuildCoarseOperatorKT), par_amg_setup.c (level loop),
 * parcsr_ls/ams.c (hypre_ParCSRComputeL1Norms).  Single partition (one rank).
 */
#include "oracle.h"
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define C_PT 1
#define F_PT -1
#define Z_PT -2
#define SF_PT -3

void oamg_default_params(oamg_params *p, int gpu_defaults)
{
   /* src/internal/amg.c:120-238 */
   p->coarsen_type    = gpu_defaults ? 8 : 10;
   p->strong_th       = 0.25;
   p->max_row_sum     = 0.9;
   p->max_coarse_size = 64;
   p->min_coarse_size = 0;
   p->max_levels      = 25;
   p->interp_type     = 6;
   p->max_nnz_row     = 4;
   p->trunc_factor    = 0.0;
   p->relax_down      = gpu_defaults ? 18 : 13;
   p->relax_up        = gpu_defaults ? 18 : 14;
   p->relax_coarse    = 9;
   p->sweeps_down = p->sweeps_up = p->sweeps_coarse = 1;
   p->relax_weight = p->outer_weight = 1.0;
   p->rand_seed                      = 2747;
}

/* hypre_BoomerAMGCreateS (par_strength.c), num_functions == 1.  A has its diagonal first.
 * S keeps A's column order, excludes the diagonal, pattern only. */
ocsr *oamg_strength(const ocsr *A, double theta, double max_row_sum)
{
   int  n   = A->nrows;
   int *cnt = (int *)calloc((size_t)n + 1, sizeof(int));
   char *keep = (char *)malloc((size_t)(A->ia[n] > 0 ? A->ia[n] : 1));
#pragma omp parallel for schedule(static)
   for (int i = 0; i < n; i++)
   {
      int    b = A->ia[i], e = A->ia[i + 1];
      int    c = 0;
      if (e > b)
      {
         double diag = A->a[b], row_scale = 0.0, row_sum = diag;
         for (int k = b + 1; k < e; k++)
         {
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
         else if (diag < 0)
         {
            for (int k = b + 1; k < e; k++) { keep[k] = !(A->a[k] <= theta * row_scale); c += keep[k]; }
         }
         else
         {
            for (int k = b + 1; k < e; k++) { keep[k] = !(A->a[k] >= theta * row_scale); c += keep[k]; }
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

/* hypre_BoomerAMGCoarsenPMIS (par_coarsen.c) + hypre_BoomerAMGIndepSetInit /
 * hypre_BoomerAMGIndepSet (par_indepset.c), one rank.
 * cf_init == 1 is the second stage of HMIS (cf holds the Ruge first-pass result). */
void oamg_pmis(const ocsr *S, int seed, int cf_init, int *cf, double *measure_out)
{
   int     n       = S->nrows;
   double *measure = (double *)calloc((size_t)n > 0 ? n : 1, sizeof(double));
   double *rnd     = (double *)malloc(sizeof(double) * ((size_t)n > 0 ? n : 1));
   int    *graph   = (int *)malloc(sizeof(int) * ((size_t)n > 0 ? n : 1));
   int     gsize   = 0;

   /* measure = |{k : i in S_k}| + hypre_Rand() in row order */
   for (int k = 0; k < S->ia[n]; k++) measure[S->ja[k]] += 1.0;
   oracle_rand_stream(seed, n, rnd);
   for (int i = 0; i < n; i++) measure[i] += rnd[i];
   if (measure_out) memcpy(measure_out, measure, sizeof(double) * (size_t)n);

   if (cf_init)
   {
      for (int i = 0; i < n; i++)
      {
         int rowlen = S->ia[i + 1] - S->ia[i];
         if (cf[i] == F_PT) cf[i] = 0; /* (offd rows too in parallel) */
         if (cf[i] == Z_PT)
         {
            if (measure[i] >= 1.0 || rowlen > 0) { cf[i] = 0; graph[gsize++] = i; }
            else cf[i] = F_PT;
         }
         else if (cf[i] == SF_PT) measure[i] = 0;
         else graph[gsize++] = i;
      }
   }
   else
   {
      for (int i = 0; i < n; i++)
      {
         cf[i] = 0;
         if (S->ia[i + 1] - S->ia[i] == 0) { cf[i] = SF_PT; measure[i] = 0; }
         else graph[gsize++] = i;
      }
   }

   int iter = 0;
   while (gsize > 0)
   {
      if (!cf_init || iter)
      {
         /* hypre_BoomerAMGIndepSet */
         for (int g = 0; g < gsize; g++)
         {
            int i = graph[g];
            if (measure[i] > 1) cf[i] = 1;
         }
         for (int g = 0; g < gsize; g++)
         {
            int i = graph[g];
            if (measure[i] > 1)
               for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
               {
                  int j = S->ja[k];
                  if (measure[j] > 1)
                  {
                     if (measure[i] > measure[j]) cf[j] = 0;
                     else if (measure[j] > measure[i]) cf[i] = 0;
                  }
               }
         }
      }
      iter++;
      /* set C and F points */
      for (int g = 0; g < gsize; g++)
      {
         int i = graph[g];
         if (measure[i] < 1) cf[i] = F_PT; /* influences nobody */
         if (cf[i] > 0) cf[i] = C_PT;
         else
            for (int k = S->ia[i]; k < S->ia[i + 1]; k++)
               if (cf[S->ja[k]] > 0) cf[i] = F_PT;
      }
      /* update subgraph */
      for (int g = 0; g < gsize; g++)
      {
         int i = graph[g];
         if (cf[i] != 0)
         {
            measure[i] = 0;
            graph[g]   = graph[gsize - 1];
            gsize--;
            g--;
         }
      }
   }
   free(measure);
   free(rnd);
   free(graph);
}

/* First pass of classical Ruge-Stueben coarsening (hypre_BoomerAMGCoarsenRuge with
 * coarsen_type 10, the first stage of HMIS): bucket lists ordered by measure, FIFO inside
 * a bucket (hypre_enter_on_lists appends at the tail, the head of the top list is taken). */
typedef struct { int *next, *prev, *head, *tail; int maxm; } rs_lists;

static void rs_enter(rs_lists *L, int m, int i)
{
   L->next[i] = -1;
   L->prev[i] = L->tail[m];
   if (L->tail[m] >= 0) L->next[L->tail[m]] = i;
   else L->head[m] = i;
   L->tail[m] = i;
   if (m > L->maxm) L->maxm = m;
}
static void rs_remove(rs_lists *L, int m, int i)
{
   if (L->prev[i] >= 0) L->next[L->prev[i]] = L->next[i];
   else L->head[m] = L->next[i];
   if (L->next[i] >= 0) L->prev[L->next[i]] = L->prev[i];
   else L->tail[m] = L->prev[i];
}

void oamg_rs_first_pass(const ocsr *S, int *cf)
{
   int   n  = S->nrows;
   ocsr *ST = ocsr_transpose(S);
   int  *m  = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   int   mmax = 0;
   for (int i = 0; i < n; i++) { m[i] = ST->ia[i + 1] - ST->ia[i]; if (m[i] > mmax) mmax = m[i]; }
   /* a measure grows by at most |S^T_i| (once per dependent that turns F): bound 2*mmax */
   int      cap = 4 * mmax + 64;
   rs_lists L;
   L.next = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   L.prev = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   L.head = (int *)malloc(sizeof(int) * (size_t)cap);
   L.tail = (int *)malloc(sizeof(int) * (size_t)cap);
   L.maxm = 0;
   for (int k = 0; k < cap; k++) L.head[k] = L.tail[k] = -1;

   int num_left = n;
   for (int j = 0; j < n; j++) cf[j] = 0;
   for (int j = 0; j < n; j++)
   {
      if (S->ia[j + 1] == S->ia[j] && m[j] == 0) { cf[j] = SF_PT; num_left--; }
   }
   for (int j = 0; j < n; j++)
   {
      if (cf[j] == SF_PT) continue;
      if (m[j] > 0) rs_enter(&L, m[j], j);
      else
      {
         cf[j] = Z_PT; /* f_pnt for HMIS */
         for (int k = S->ia[j]; k < S->ia[j + 1]; k++)
         {
            int nb = S->ja[k];
            if (cf[nb] != SF_PT)
            {
               if (nb < j)
               {
                  if (m[nb] > 0) rs_remove(&L, m[nb], nb);
                  m[nb]++;
                  rs_enter(&L, m[nb], nb);
               }
               else m[nb]++;
            }
         }
         num_left--;
      }
   }
   while (num_left > 0)
   {
      while (L.maxm > 0 && L.head[L.maxm] < 0) L.maxm--;
      if (L.maxm <= 0) break;
      int idx = L.head[L.maxm];
      cf[idx] = C_PT;
      rs_remove(&L, m[idx], idx);
      m[idx] = 0;
      num_left--;
      for (int j = ST->ia[idx]; j < ST->ia[idx + 1]; j++)
      {
         int nb = ST->ja[j];
         if (cf[nb] == 0)
         {
            cf[nb] = F_PT;
            rs_remove(&L, m[nb], nb);
            num_left--;
            for (int k = S->ia[nb]; k < S->ia[nb + 1]; k++)
            {
               int n2 = S->ja[k];
               if (cf[n2] == 0)
               {
                  rs_remove(&L, m[n2], n2);
                  m[n2]++;
                  if (m[n2] >= cap) { fprintf(stderr, "oracle: RS measure overflow\n"); abort(); }
                  rs_enter(&L, m[n2], n2);
               }
            }
         }
      }
      for (int j = S->ia[idx]; j < S->ia[idx + 1]; j++)
      {
         int nb = S->ja[j];
         if (cf[nb] == 0)
         {
            rs_remove(&L, m[nb], nb);
            m[nb]--;
            if (m[nb] > 0) rs_enter(&L, m[nb], nb);
            else
            {
               cf[nb] = F_PT;
               num_left--;
               for (int k = S->ia[nb]; k < S->ia[nb + 1]; k++)
               {
                  int n2 = S->ja[k];
                  if (cf[n2] == 0)
                  {
                     rs_remove(&L, m[n2], n2);
                     m[n2]++;
                     rs_enter(&L, m[n2], n2);
                  }
               }
            }
         }
      }
   }
   free(L.next); free(L.prev); free(L.head); free(L.tail);
   free(m);
   ocsr_free(ST);
}

/* hypre_qsort2abs (utilities/qsort.c): sort v, w in DEcreasing order of |w|; the tie order
 * this particular quicksort produces decides which equal-weight entries survive truncation. */
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

/* hypre_BoomerAMGBuildExtPIInterp (par_lr_interp.c) followed by
 * hypre_BoomerAMGInterpTruncation (par_interp.c), one rank.  On return SF_PT (-3) entries
 * of cf are reset to F_PT (-1) as hypre does. */
ocsr *oamg_extpi_interp(const ocsr *A, const ocsr *S, int *cf, int max_elmts,
                        double trunc_factor, int *n_coarse_out)
{
   int  n   = A->nrows;
   int *f2c = (int *)malloc(sizeof(int) * ((size_t)n + 1));
   int *pi  = (int *)calloc((size_t)n + 1, sizeof(int));
   int  nc  = 0;
   for (int i = 0; i < n; i++) f2c[i] = (cf[i] >= 0) ? nc++ : -1;

   /* pass 1: row sizes of the untruncated P (|C-hat_i|) */
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

   /* pass 2: weights */
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
         const int sfm = -2 - i; /* unique "strong F neighbour of row i" marker (< -1) */
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
            else if (cf[i1] != SF_PT) diagonal += A->a[jj];
         }
         if (diagonal != 0.0)
            for (int jj = jb; jj < je; jj++) pd[jj] /= -diagonal;
      }
      free(mark);
   }
   /* NOTE: the per-thread `mark` test uses (>= jb && < je): with one marker array per row
    * sweep this equals hypre's `P_marker[i1] >= jj_begin_row` because later rows have not
    * been visited yet in the sequential code. */

   /* truncation: trunc_factor, then keep the max_elmts largest |w| (sorted order), rescale */
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

/* hypre_BoomerAMGBuildCoarseOperatorKT (par_rap.c), one rank: RAP = R A P with R = P^T.
 * Row ic: diagonal first, then columns in order of discovery of the loop nest
 * (i1 in R_ic) x (i2 in A_i1) x (i3 in P_i2); value = sum of (r*a)*p in that order. */
ocsr *oamg_rap(const ocsr *R, const ocsr *A, const ocsr *P)
{
   int  nc  = R->nrows;
   int *cia = (int *)calloc((size_t)nc + 1, sizeof(int));
   /* symbolic */
#pragma omp parallel
   {
      int *mark = (int *)malloc(sizeof(int) * ((size_t)nc + 1));
      for (int i = 0; i < nc; i++) mark[i] = -1;
#pragma omp for schedule(dynamic, 256)
      for (int ic = 0; ic < nc; ic++)
      {
         int c    = 1;
         mark[ic] = ic;
         for (int j1 = R->ia[ic]; j1 < R->ia[ic + 1]; j1++)
         {
            int i1 = R->ja[j1];
            for (int j2 = A->ia[i1]; j2 < A->ia[i1 + 1]; j2++)
            {
               int i2 = A->ja[j2];
               for (int j3 = P->ia[i2]; j3 < P->ia[i2 + 1]; j3++)
               {
                  int i3 = P->ja[j3];
                  if (mark[i3] != ic) { mark[i3] = ic; c++; }
               }
            }
         }
         cia[ic + 1] = c;
      }
      free(mark);
   }
   for (int i = 0; i < nc; i++) cia[i + 1] += cia[i];
   ocsr *C = ocsr_alloc(nc, nc, cia[nc], 1);
   memcpy(C->ia, cia, sizeof(int) * ((size_t)nc + 1));
#pragma omp parallel
   {
      int *mark = (int *)malloc(sizeof(int) * ((size_t)nc + 1));
      for (int i = 0; i < nc; i++) mark[i] = -1;
#pragma omp for schedule(dynamic, 256)
      for (int ic = 0; ic < nc; ic++)
      {
         int b = C->ia[ic], c = b;
         mark[ic] = c; C->ja[c] = ic; C->a[c] = 0.0; c++;
         for (int j1 = R->ia[ic]; j1 < R->ia[ic + 1]; j1++)
         {
            int    i1 = R->ja[j1];
            double r  = R->a[j1];
            for (int j2 = A->ia[i1]; j2 < A->ia[i1 + 1]; j2++)
            {
               int    i2 = A->ja[j2];
               double ra = r * A->a[j2];
               for (int j3 = P->ia[i2]; j3 < P->ia[i2 + 1]; j3++)
               {
                  int    i3  = P->ja[j3];
                  double rap = ra * P->a[j3];
                  if (mark[i3] < b) { mark[i3] = c; C->ja[c] = i3; C->a[c] = rap; c++; }
                  else C->a[mark[i3]] += rap;
               }
            }
         }
      }
      free(mark);
   }
   free(cia);
   return C;
}

/* hypre_ParCSRComputeL1Norms (parcsr_ls/ams.c), one rank (offd block empty):
 * option 1: full l1 row norm (relax 18); option 4: truncated l1 (relax 8/13/14) = |a_ii| on
 * one rank; option 5: the diagonal itself (relax 7).  Sign follows the diagonal. */
void oamg_l1_norms(const ocsr *A, int option, double *l1)
{
#pragma omp parallel for schedule(static)
   for (int i = 0; i < A->nrows; i++)
   {
      double d = A->ia[i + 1] > A->ia[i] ? A->a[A->ia[i]] : 0.0;
      double v;
      if (option == 1)
      {
         v = 0.0;
         for (int k = A->ia[i]; k < A->ia[i + 1]; k++) v += fabs(A->a[k]);
         if (d < 0) v = -v;
      }
      else if (option == 4)
      {
         v = fabs(d);
         if (d < 0) v = -v;
      }
      else v = d;
      l1[i] = v;
   }
}

static int relax_l1_option(int type)
{
   if (type == 18) return 1;
   if (type == 8 || type == 13 || type == 14) return 4;
   return 5;
}

/* hypre_BoomerAMGSetup level loop (par_amg_setup.c). */
oamg *oamg_setup(const ocsr *Ain, const oamg_params *prm)
{
   oamg *h = (oamg *)calloc(1, sizeof(oamg));
   h->prm  = *prm;
   ocsr *A0 = ocsr_from_arrays(Ain->nrows, Ain->ncols, Ain->ia, Ain->ja, Ain->a);
   ocsr_diag_first(A0);
   h->A[0]  = A0;
   int level = 0, not_finished = prm->max_levels > 1;
   while (not_finished)
   {
      ocsr *A = h->A[level];
      int   n = A->nrows;
      ocsr *S = oamg_strength(A, prm->strong_th, prm->max_row_sum);
      int  *cf = (int *)calloc((size_t)n + 1, sizeof(int));
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
      h->P[level]     = oamg_extpi_interp(A, S, cf, prm->max_nnz_row, prm->trunc_factor, &nc2);
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
   /* coarsest level: dense copy for Gaussian elimination (hypre_GaussElimSetup, which has no size
    * limit; the n^2 < 2e8 cap bounds the copy to 1.6 GB and is the device's limit too) */
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
   return h;
}

void oamg_destroy(oamg *h)
{
   if (!h) return;
   for (int l = 0; l < OAMG_MAX_LEVELS; l++)
   {
      ocsr_free(h->A[l]); ocsr_free(h->P[l]); ocsr_free(h->R[l]); ocsr_free(h->S[l]);
      free(h->cf[l]); free(h->cf_raw[l]); free(h->l1_down[l]); free(h->l1_up[l]); free(h->measure[l]);
      free(h->u[l]); free(h->f[l]); free(h->t[l]); free(h->t2[l]);
   }
   free(h->ge);
   free(h);
}
