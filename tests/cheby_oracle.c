/* cheby_oracle.c -- CPU restatement of Chebyshev smoothing (BoomerAMG relax_type 16, cheby_variant 0);
 * TEST INFRASTRUCTURE ONLY.
 *
 * Built on the parity oracle (oracle/oracle.h, liboracle.so): the hierarchy comes from the oracle (or
 * from the systems / aggressive restatements, which produce an oracle hierarchy), the other smoothers
 * are the oracle's oamg_relax and the Krylov methods are the oracle's own krylov.c, compiled here a
 * second time against this file's preconditioner.  What Chebyshev smoothing adds is restated after
 * hypre's hypre_ParCSRRelax_Cheby_Setup / _Solve and hypre_ParCSRMaxEigEstimate(CG); hypre parity is not
 * pinned, this file is the rule the device is compared with (DESIGN.md section 4):
 *   1. ds_i = 1 / sqrt|a_ii| (scale = 1), else 1;
 *   2. eigenvalue bounds of C A, C = D^{-1} (scaled) or I: Gershgorin (eig_est = 0) or eig_est steps of
 *      CG-Lanczos from b = ovec_set_random(seed 1), eigenvalues of the tridiagonal by tql1;
 *   3. interval [lower, upper] and theta, delta; 4. monomial coefficients of the order-k polynomial;
 *   sweep: r = ds (f - A u); v = c_{k-1} r; v = c_i r + ds (A (ds v)), i = k-2..0; u = u + ds v.
 * Every product and sum is rounded separately (compiled with -ffp-contract=off). */
#include "oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef struct
{
   int    order;    /* 1..4 */
   double fraction; /* (0, 1] */
   int    eig_est;  /* CG steps, 0 = Gershgorin */
   int    scale;    /* 1: D^{-1/2} A D^{-1/2} */
} ocheby_params;

typedef struct
{
   oamg         *h; /* borrowed */
   ocheby_params cp;
   int           has[OAMG_MAX_LEVELS];
   double       *ds[OAMG_MAX_LEVELS];
   double        eig[OAMG_MAX_LEVELS][2]; /* max, min */
   double        c[OAMG_MAX_LEVELS][4];
   double       *r, *v, *t;               /* sweep work, level-0 size */
} ocheby;

/* ---- 1 + 2a: scaling and Gershgorin bounds; -1 for a zero diagonal with scale = 1 ---------- */
int ocheby_gershgorin(const ocsr *A, int scale, double *ds, double *eig)
{
   double hi = -INFINITY, nlo = -INFINITY;
   int    bad = 0;
   for (int i = 0; i < A->nrows; i++)
   {
      double d = 0.0, R = 0.0;
      for (int k = A->ia[i]; k < A->ia[i + 1]; k++)
      {
         if (A->ja[k] == i) d = d + A->a[k];
         else R = R + fabs(A->a[k]);
      }
      double ad = fabs(d);
      if (scale && ad == 0.0) { bad = 1; ds[i] = 0.0; continue; }
      ds[i]    = scale ? 1.0 / sqrt(ad) : 1.0;
      double h = scale ? (ad + R) / ad : ad + R;
      double l = scale ? (ad - R) / ad : ad - R;
      hi       = fmax(hi, h);
      nlo      = fmax(nlo, -l);
   }
   eig[0] = hi;
   eig[1] = -nlo;
   return bad ? -1 : 0;
}

/* ---- tql1 (hypre_LINPACKcgtql1): eigenvalues of the symmetric tridiagonal, ascending ------- */
static double pythag(double a, double b)
{
   double p = fmax(fabs(a), fabs(b));
   if (p == 0.0) return 0.0;
   double q = fmin(fabs(a), fabs(b)) / p;
   return p * sqrt(1.0 + q * q);
}
static int tql1(int n, double *d, double *e)
{
   if (n == 1) return 0;
   for (int i = 1; i < n; i++) e[i - 1] = e[i];
   e[n - 1] = 0.0;
   double f = 0.0, tst1 = 0.0;
   for (int l = 0; l < n; l++)
   {
      int    it = 0, m;
      double h = fabs(d[l]) + fabs(e[l]);
      if (tst1 < h) tst1 = h;
      for (m = l; m < n; m++)
         if (tst1 + fabs(e[m]) == tst1) break;
      if (m > l)
      {
         for (;;)
         {
            if (it++ == 30) return -1;
            int    l1 = l + 1;
            double g = d[l];
            double p = (d[l1] - g) / (2.0 * e[l]);
            double r = pythag(p, 1.0);
            double sr = (p >= 0.0) ? fabs(r) : -fabs(r);
            d[l]  = e[l] / (p + sr);
            d[l1] = e[l] * (p + sr);
            double dl1 = d[l1];
            h = g - d[l];
            for (int i = l1 + 1; i < n; i++) d[i] -= h;
            f += h;
            p = d[m];
            double c = 1.0, c2 = c, c3 = c, el1 = e[l1], s = 0.0, s2 = 0.0;
            for (int i = m - 1; i >= l; i--)
            {
               c3 = c2; c2 = c; s2 = s;
               g = c * e[i];
               h = c * p;
               r = pythag(p, e[i]);
               e[i + 1] = s * r;
               s = e[i] / r;
               c = p / r;
               p = c * d[i] - s * g;
               d[i + 1] = h + s * (c * g + s * d[i]);
            }
            p = -s * s2 * c3 * el1 * e[l] / dl1;
            e[l] = s * p;
            d[l] = c * p;
            if (!(tst1 + fabs(e[l]) > tst1)) break;
         }
      }
      double p = d[l] + f;
      int    i = l;
      for (; i > 0 && p < d[i - 1]; i--) d[i] = d[i - 1];
      d[i] = p;
   }
   return 0;
}

/* ---- 2b: CG-Lanczos bounds; returns the number of completed steps (0: no estimate) --------- */
int ocheby_cg_eig(const ocsr *A, int scale, int k, double *eig)
{
   int     n = A->nrows;
   double *r = (double *)malloc(sizeof(double) * ((size_t)n + 1)), *z = (double *)malloc(sizeof(double) * ((size_t)n + 1));
   double *p = (double *)malloc(sizeof(double) * ((size_t)n + 1)), *s = (double *)malloc(sizeof(double) * ((size_t)n + 1));
   double *dabs = (double *)malloc(sizeof(double) * ((size_t)n + 1));
   double *al = (double *)calloc((size_t)k + 1, sizeof(double)), *be = (double *)calloc((size_t)k + 2, sizeof(double));
   for (int i = 0; i < n; i++)
   {
      double d = 0.0;
      for (int q = A->ia[i]; q < A->ia[i + 1]; q++)
         if (A->ja[q] == i) d = d + A->a[q];
      dabs[i] = fabs(d);
   }
   ovec_set_random(1, n, r);
   for (int i = 0; i < n; i++) { z[i] = scale ? r[i] / dabs[i] : r[i]; p[i] = z[i]; }
   double gamma = ovec_dot(n, r, z);
   int    m = 0;
   for (int j = 0; j < k; j++)
   {
      ocsr_matvec(1.0, A, p, 0.0, s);
      double sp = ovec_dot(n, s, p);
      if (!(sp > 0.0)) break;
      double alpha = gamma / sp;
      al[j] = alpha;
      m = j + 1;
      for (int i = 0; i < n; i++)
      {
         r[i] = r[i] - alpha * s[i];
         z[i] = scale ? r[i] / dabs[i] : r[i];
      }
      double gn = ovec_dot(n, r, z);
      if (!(gn > 0.0)) break;
      double beta = gn / gamma;
      be[j + 1] = beta;
      gamma = gn;
      for (int i = 0; i < n; i++) p[i] = z[i] + beta * p[i];
   }
   if (m > 0)
   {
      /* T_jj = 1/alpha_j + beta_j/alpha_{j-1}, T_{j,j+1} = sqrt(beta_{j+1})/alpha_j */
      double *d = (double *)malloc(sizeof(double) * (size_t)m), *e = (double *)calloc((size_t)m, sizeof(double));
      for (int j = 0; j < m; j++)
      {
         d[j] = (j == 0) ? 1.0 / al[0] : 1.0 / al[j] + be[j] / al[j - 1];
         if (j > 0) e[j] = sqrt(be[j]) / al[j - 1];
      }
      if (tql1(m, d, e) != 0) m = 0;
      else { eig[0] = d[m - 1]; eig[1] = d[0]; }
      free(d); free(e);
   }
   free(r); free(z); free(p); free(s); free(dabs); free(al); free(be);
   return m;
}

/* ---- 3 + 4: interval and coefficients; -1 for a degenerate interval ----------------------- */
int ocheby_coefs(double max_eig, double min_eig, double fraction, int order, double *c)
{
   double upper, lower;
   if (min_eig >= 0.0) { upper = 1.1 * max_eig; lower = (upper - min_eig) * fraction + min_eig; }
   else if (max_eig <= 0.0) { upper = 1.1 * min_eig; lower = max_eig - (max_eig - upper) * fraction; }
   else { const double mn = 0.0; upper = 1.1 * max_eig; lower = (upper - mn) * fraction + mn; }
   const double theta = (upper + lower) / 2.0, delta = (upper - lower) / 2.0;
   if (theta == 0.0 || !isfinite(theta) || !isfinite(delta)) return -1;
   const double t2 = theta * theta, d2 = delta * delta;
   if (order == 1) c[0] = 1.0 / theta;
   else if (order == 2)
   {
      const double den = d2 - 2.0 * t2;
      c[0] = -4.0 * theta / den; c[1] = 2.0 / den;
   }
   else if (order == 3)
   {
      const double den = 4.0 * t2 * theta - 3.0 * d2 * theta;
      c[0] = (12.0 * t2 - 3.0 * d2) / den; c[1] = -12.0 * theta / den; c[2] = 4.0 / den;
   }
   else
   {
      const double den = 8.0 * t2 * t2 - 8.0 * d2 * t2 + d2 * d2;
      c[0] = (32.0 * t2 * theta - 16.0 * d2 * theta) / den; c[1] = -(48.0 * t2 - 8.0 * d2) / den;
      c[2] = 32.0 * theta / den; c[3] = -8.0 / den;
   }
   for (int i = 0; i < order; i++)
      if (!isfinite(c[i])) return -1;
   return 0;
}

/* ---- one sweep ---------------------------------------------------------------------------- */
void ocheby_sweep(const ocsr *A, const double *ds, const double *c, int order, const double *f, double *u,
                  double *r, double *v, double *t)
{
   int n = A->nrows;
   for (int i = 0; i < n; i++)
   {
      double res = f[i];
      for (int k = A->ia[i]; k < A->ia[i + 1]; k++) res -= A->a[k] * u[A->ja[k]];
      r[i] = ds[i] * res;
   }
   for (int i = 0; i < n; i++) v[i] = c[order - 1] * r[i];
   for (int m = order - 2; m >= 0; m--)
   {
      for (int i = 0; i < n; i++) t[i] = ds[i] * v[i];
      for (int i = 0; i < n; i++)
      {
         double acc = 0.0;
         for (int k = A->ia[i]; k < A->ia[i + 1]; k++) acc += A->a[k] * t[A->ja[k]];
         v[i] = c[m] * r[i] + ds[i] * acc;
      }
   }
   for (int i = 0; i < n; i++) u[i] = u[i] + ds[i] * v[i];
}

/* ---- hierarchy ---------------------------------------------------------------------------- */
void ocheby_destroy(ocheby *ch)
{
   if (!ch) return;
   for (int l = 0; l < OAMG_MAX_LEVELS; l++) free(ch->ds[l]);
   free(ch->r); free(ch->v); free(ch->t);
   free(ch);
}

/* Chebyshev data for every level of h on which a type-16 sweep runs.  eigs (2 per level, may be NULL):
 * bounds to use instead of the estimate where eigs[2l] is not NaN.  status: 0, or -(1 + level) of the
 * first level whose setup is rejected (zero diagonal, failed estimate, degenerate interval). */
ocheby *ocheby_attach(oamg *h, const ocheby_params *cp, const double *eigs, int *status)
{
   ocheby *ch = (ocheby *)calloc(1, sizeof(ocheby));
   ch->h  = h;
   ch->cp = *cp;
   *status = 0;
   int n0 = h->A[0]->nrows;
   ch->r = (double *)malloc(sizeof(double) * ((size_t)n0 + 1));
   ch->v = (double *)malloc(sizeof(double) * ((size_t)n0 + 1));
   ch->t = (double *)malloc(sizeof(double) * ((size_t)n0 + 1));
   for (int l = 0; l < h->nlev && *status == 0; l++)
   {
      int fine = l < h->nlev - 1;
      int on   = fine ? (h->prm.relax_down == 16 || h->prm.relax_up == 16) : (h->prm.relax_coarse == 16);
      if (!on) continue;
      const ocsr *A = h->A[l];
      ch->has[l]    = 1;
      ch->ds[l]     = (double *)malloc(sizeof(double) * ((size_t)A->nrows + 1));
      double ge[2];
      if (ocheby_gershgorin(A, cp->scale, ch->ds[l], ge) != 0) { *status = -(1 + l); break; }
      ch->eig[l][0] = ge[0]; ch->eig[l][1] = ge[1];
      if (eigs && !isnan(eigs[2 * l])) { ch->eig[l][0] = eigs[2 * l]; ch->eig[l][1] = eigs[2 * l + 1]; }
      else if (cp->eig_est > 0 && ocheby_cg_eig(A, cp->scale, cp->eig_est, ch->eig[l]) == 0) { *status = -(1 + l); break; }
      if (ocheby_coefs(ch->eig[l][0], ch->eig[l][1], cp->fraction, cp->order, ch->c[l]) != 0) { *status = -(1 + l); break; }
   }
   return ch;
}

/* hypre_gselim (the oracle's copy is file-local) */
static void gselim(double *A, double *x, int n)
{
   if (n == 1) { if (A[0] != 0.0) x[0] /= A[0]; return; }
   for (int k = 0; k < n - 1; k++)
      if (A[(size_t)k * n + k] != 0.0)
         for (int j = k + 1; j < n; j++)
            if (A[(size_t)j * n + k] != 0.0)
            {
               double factor = A[(size_t)j * n + k] / A[(size_t)k * n + k];
               for (int m = k + 1; m < n; m++) A[(size_t)j * n + m] -= factor * A[(size_t)k * n + m];
               x[j] -= factor * x[k];
            }
   for (int k = n - 1; k > 0; --k)
   {
      if (A[(size_t)k * n + k] != 0.0)
      {
         x[k] /= A[(size_t)k * n + k];
         for (int j = 0; j < k; j++)
            if (A[(size_t)j * n + k] != 0.0) x[j] -= x[k] * A[(size_t)j * n + k];
      }
   }
   if (A[0] != 0.0) x[0] /= A[0];
}

static void relax(ocheby *ch, int l, int type, const double *l1, const double *f, double *u)
{
   oamg *h = ch->h;
   if (type == 16) ocheby_sweep(h->A[l], ch->ds[l], ch->c[l], ch->cp.order, f, u, ch->r, ch->v, ch->t);
   else oamg_relax(h->A[l], f, u, type, h->prm.relax_weight, l1, h->t[l], h->t2[l]);
}

void ocheby_sweep_level(ocheby *ch, int l, const double *f, double *u)
{
   ocheby_sweep(ch->h->A[l], ch->ds[l], ch->c[l], ch->cp.order, f, u, ch->r, ch->v, ch->t);
}

/* oamg_vcycle (hypre_BoomerAMGCycle, V, relax_order 0) with the type-16 sweeps of this file */
void ocheby_vcycle(ocheby *ch, const double *f, double *u)
{
   oamg *h = ch->h;
   int   n0 = h->A[0]->nrows, L = h->nlev - 1;
   memcpy(h->f[0], f, sizeof(double) * (size_t)n0);
   memcpy(h->u[0], u, sizeof(double) * (size_t)n0);
   for (int l = 0; l < L; l++)
   {
      for (int s = 0; s < h->prm.sweeps_down; s++) relax(ch, l, h->prm.relax_down, h->l1_down[l], h->f[l], h->u[l]);
      ocsr_residual(h->A[l], h->u[l], h->f[l], h->t[l]);
      ocsr_matvec(1.0, h->R[l], h->t[l], 0.0, h->f[l + 1]);
      memset(h->u[l + 1], 0, sizeof(double) * (size_t)h->A[l + 1]->nrows);
   }
   int n = h->A[L]->nrows;
   if (h->ge && h->ge_n == n && (h->prm.relax_coarse == 9 || h->prm.relax_coarse == 99))
   {
      double *M = (double *)malloc(sizeof(double) * ((size_t)n * n + 1));
      memcpy(M, h->ge, sizeof(double) * (size_t)n * n);
      memcpy(h->u[L], h->f[L], sizeof(double) * (size_t)n);
      gselim(M, h->u[L], n);
      free(M);
   }
   else
      for (int s = 0; s < h->prm.sweeps_coarse; s++) relax(ch, L, h->prm.relax_coarse, h->l1_down[L], h->f[L], h->u[L]);
   for (int l = L - 1; l >= 0; l--)
   {
      const ocsr *P = h->P[l];
      double     *uf = h->u[l], *uc = h->u[l + 1];
      for (int i = 0; i < P->nrows; i++)
      {
         double s = uf[i];
         for (int k = P->ia[i]; k < P->ia[i + 1]; k++) s += P->a[k] * uc[P->ja[k]];
         uf[i] = s;
      }
      for (int s = 0; s < h->prm.sweeps_up; s++) relax(ch, l, h->prm.relax_up, h->l1_up[l], h->f[l], h->u[l]);
   }
   memcpy(u, h->u[0], sizeof(double) * (size_t)n0);
}

void ocheby_precond(ocheby *ch, const double *r, double *z)
{
   memset(z, 0, sizeof(double) * (size_t)ch->h->A[0]->nrows);
   ocheby_vcycle(ch, r, z);
}

/* the oracle's Krylov methods, compiled against this preconditioner (they hand the `oamg *` they are
 * given to oamg_precond only, so an ocheby handle travels through them unchanged) */
static void ocheby_precond_cb(oamg *M, const double *r, double *z) { ocheby_precond((ocheby *)(void *)M, r, z); }
#define oamg_precond ocheby_precond_cb
#define opcg ocheby_pcg
#define ogmres ocheby_gmres
#define ofgmres ocheby_fgmres
#define obicgstab ocheby_bicgstab
#include "krylov.c"
