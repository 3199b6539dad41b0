// hdk_amg_solve.cu -- BoomerAMG V-cycle on the device (north-star item 2).
// Stands in for HYPRE_BoomerAMGSolve / hypre_BoomerAMGCycle (cycle_type 1, relax_order 0,
// max_iter 1, tol 0) reached from PreconSolveDispatch (reference src/internal/solver.c:314-329)
// and HYPREDRV_PreconApply (src/HYPREDRV.c:3345).  Per level: l1-Jacobi (18) / Jacobi (7) /
// two-stage Gauss-Seidel (11, 12) sweeps fused with their residual evaluation, explicit
// R = P^T restriction, P prolongation fused with the correction, dense coarsest solve kept
// on the GPU (pre-inverted operator, one matvec).
#include "hdk_amg.cuh"

namespace hdk {

// u = Ainv f: one warp per row of the dense inverse (any n; size_t row offsets)
__global__ void __launch_bounds__(256) k_dense_apply(const double *__restrict__ Ainv, const double *__restrict__ f,
                                                     double *__restrict__ u, int n)
{
   int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
   if (row >= n) return;
   double acc = 0.0;
   for (int j = lane; j < n; j += 32) acc += Ainv[(size_t)row * n + j] * f[j];
   acc = warp_sum(acc);
   if (lane == 0) u[row] = acc;
}

static bool is_jacobi(int t) { return t == 18 || t == 7 || t == 0; }

// One Chebyshev sweep (relax 16, hypre_ParCSRRelax_Cheby_Solve, scaled form; DESIGN.md section 4):
//   r = ds (f - A u);  v = c_{k-1} r;  v = c_i r + ds (A (ds v)) for i = k-2..0;  out = u + ds v
// The passes carry w = ds v, so every pass is one product with a fused epilogue: START (r and w),
// STEP (w), FIN (out, optionally with the fused dot <f, out>); order 1 is the single pass ONE.
// in == nullptr: zero initial guess, the first pass is element-wise (f - A 0 = f).  Levels whose
// off-rank part is added by a correction kernel run each pass as a plain product + element-wise epilogue.
static int cheby_sweep(hdk_amg_s *M, int l, const double *f, const double *in, double *out, int fin, double *fin_out,
                       const hdk_csr_s *export_to = nullptr)
{
   AmgLevel &L = M->lev[(size_t)l];
   if (!L.cheb_ds) return set_error(HDK_ERR_INVALID, "level %d has no Chebyshev data", l);
   const int     k = M->prm.cheby_order, n = L.n;
   const bool    fused = parcsr_single_kernel(*L.A);
   const double *c = L.cheb_c;
   SpmvArgs      a;
   a.d = L.cheb_ds;
   if (k == 1)
   {
      a.b = f; a.alpha = c[0]; a.uo = in; a.y = out;
      if (!in) HDK_TRY(cheb_epilogue_pass(SPMV_CHEB_ONE, n, f, a));
      else if (fused)
      {
         a.x = in; a.export_to = export_to;
         if (fin != FIN_NONE) { a.dotv = f; a.fin = fin; a.fin_out = fin_out; fin = FIN_NONE; }
         HDK_TRY(parcsr_matvec(*L.A, SPMV_CHEB_ONE, a));
      }
      else
      {
         SpmvArgs rr;
         rr.x = in; rr.b = f; rr.y = L.cheb_r;
         HDK_TRY(parcsr_matvec(*L.A, SPMV_RESIDUAL, rr));
         HDK_TRY(cheb_epilogue_pass(SPMV_CHEB_ONE, n, L.cheb_r, a));
      }
   }
   else
   {
      double *cur = L.cheb_v[0], *nxt = L.cheb_v[1];
      // START: r = ds (f - A u), w = ds (c_{k-1} r)
      a.b = f; a.alpha = c[k - 1]; a.y = cur; a.y2 = L.cheb_r;
      if (!in) HDK_TRY(cheb_epilogue_pass(SPMV_CHEB_START, n, f, a));
      else if (fused)
      {
         a.x = in; a.export_to = L.A;
         HDK_TRY(parcsr_matvec(*L.A, SPMV_CHEB_START, a));
      }
      else
      {
         SpmvArgs rr;
         rr.x = in; rr.b = f; rr.y = nxt;
         HDK_TRY(parcsr_matvec(*L.A, SPMV_RESIDUAL, rr));
         HDK_TRY(cheb_epilogue_pass(SPMV_CHEB_START, n, nxt, a));
      }
      for (int i = k - 2; i >= 0; i--)
      {
         // STEP: w' = ds (c_i r + ds (A w)); the last one (i = 0) is FIN: out = u + ds (c_0 r + ds (A w))
         const int mode = (i == 0) ? SPMV_CHEB_FIN : SPMV_CHEB_STEP;
         SpmvArgs  b2;
         b2.d = L.cheb_ds; b2.b = L.cheb_r; b2.alpha = c[i];
         b2.y = (i == 0) ? out : nxt;
         b2.uo = in;
         if (fused)
         {
            b2.x = cur; b2.export_to = (i == 0) ? export_to : L.A;
            if (i == 0 && fin != FIN_NONE) { b2.dotv = f; b2.fin = fin; b2.fin_out = fin_out; fin = FIN_NONE; }
            HDK_TRY(parcsr_matvec(*L.A, mode, b2));
         }
         else
         {
            SpmvArgs pr;
            pr.x = cur; pr.y = b2.y;
            HDK_TRY(parcsr_matvec(*L.A, SPMV_SET, pr));
            HDK_TRY(cheb_epilogue_pass(mode, n, b2.y, b2));
         }
         std::swap(cur, nxt);
      }
   }
   if (fin != FIN_NONE) HDK_TRY(vec_dot_dev(f, out, n, fin, fin_out));
   return HDK_OK;
}

// one smoothing sweep u_new = S(u_old); result written to `out` (out != in)
// export_to: the matrix whose product reads `out` next (its halo is filled by this sweep's kernel)
static int relax_sweep(hdk_amg_s *M, int l, int type, const double *l1, const double *f, const double *in,
                       double *out, int fin, double *fin_out, const hdk_csr_s *export_to = nullptr)
{
   if (type == 16) return cheby_sweep(M, l, f, in, out, fin, fin_out, export_to);
   AmgLevel &L = M->lev[(size_t)l];
   SpmvArgs  a;
   a.x = in; a.y = out; a.b = f; a.d = l1; a.w = M->prm.relax_weight;
   if (is_jacobi(type))
   {
      if (fin != FIN_NONE) { a.dotv = f; a.fin = fin; a.fin_out = fin_out; }
      a.export_to = export_to;
      return parcsr_matvec(*L.A, SPMV_JACOBI, a);
   }
   if (type == 11 || type == 12)
   {
      // two-stage GS (hypre_BoomerAMGRelaxTwoStageGaussSeidel): r = w D^{-1}(f - A u); u += r; then
      // k = 1..inner: r <- D^{-1} L r, u += (-1)^k r.  Fused: ONE pass over A produces both r and
      // u + r, and each inner step is one pass over the strict lower triangle whose epilogue divides
      // by the diagonal and applies the signed update -- 2 (type 11) or 3 (type 12) kernels per sweep,
      // no scratch allocation.  (hypre applies L in place bottom-up, which reads only entries not yet
      // updated, i.e. the same Jacobi-type product as this out-of-place form.)
      const int inner = (type == 11) ? 1 : 2;
      if (L.gs1 && parcsr_single_kernel(*L.A))
      {
         a.y = out; a.y2 = L.gs1;
         HDK_TRY(parcsr_matvec(*L.A, SPMV_JACOBI2, a));
         double *cur = L.gs1, *nxt = L.gs2;
         double  mult = 1.0;
         for (int it = 0; it < inner; it++)
         {
            mult = -mult;
            SpmvArgs b2;
            b2.x = cur; b2.y = out; b2.d = l1; b2.alpha = mult;
            b2.y2 = (it + 1 < inner) ? nxt : nullptr;
            HDK_TRY(spmv_launch(L.L, SPMV_GS_STEP, b2));
            double *tmp = cur; cur = nxt; nxt = tmp;
         }
      }
      else
      {
         // rows whose off-rank part is added by a separate correction kernel: unfused form
         double *r, *r2;
         HDK_TRY(dalloc(&r, (size_t)L.n + 8));
         HDK_TRY(dalloc(&r2, (size_t)L.n + 8));
         a.y = r;                                 // r = w D^{-1} (f - A u_old)
         HDK_TRY(parcsr_matvec(*L.A, SPMV_JACOBI_R, a));
         HDK_TRY(vec_copy(out, in, L.n));         // out = u_old
         HDK_TRY(vec_axpy(1.0, r, out, L.n));     // out = u_old + r
         double mult  = 1.0;
         double *cur = r, *nxt = r2;
         for (int it = 0; it < inner; it++)
         {
            SpmvArgs b2;
            b2.x = cur; b2.y = nxt;
            HDK_TRY(spmv_launch(L.L, SPMV_SET, b2));
            HDK_TRY(vec_scaled_div(nxt, nxt, l1, 1.0, L.n));
            mult = -mult;
            HDK_TRY(vec_axpy(mult, nxt, out, L.n));
            double *tmp = cur; cur = nxt; nxt = tmp;
         }
         dfree(r); dfree(r2);
      }
      if (fin != FIN_NONE) HDK_TRY(vec_dot_dev(f, out, L.n, fin, fin_out));
      return HDK_OK;
   }
   return set_error(HDK_ERR_UNSUPPORTED, "relaxation type %d has no device kernel (use 18, 7, 0, 11, 12 or 16)", type);
}

static int coarse_solve(hdk_amg_s *M, int l, const double *f, double *u, double *alt, bool zero_guess, double **result)
{
   AmgLevel &L = M->lev[(size_t)l];
   *result     = u;
   if (M->ge_inv && M->ge_n == L.n)
   {
      k_dense_apply<<<cdiv(L.n, 8), 256, 0, g.stream>>>(M->ge_inv, f, u, L.n);
      HDK_LAUNCH_CHECK();
      return HDK_OK;
   }
   // no dense factor (operator too large or smoother requested): relaxation sweeps
   int     type = (M->prm.relax_coarse == 9 || M->prm.relax_coarse == 99) ? 18 : M->prm.relax_coarse;
   double *cur = u, *oth = alt;
   int     sweeps = M->prm.sweeps_coarse < 1 ? 1 : M->prm.sweeps_coarse;
   for (int s = 0; s < sweeps; s++)
   {
      if (s == 0 && zero_guess && is_jacobi(type))
      {
         HDK_TRY(vec_scaled_div(cur, f, L.l1_down, M->prm.relax_weight, L.n));
      }
      else
      {
         if (s == 0 && zero_guess && type == 16) HDK_TRY(cheby_sweep(M, l, f, nullptr, oth, FIN_NONE, nullptr));
         else
         {
            if (s == 0 && zero_guess) HDK_TRY(vec_fill(cur, 0.0, L.n));
            HDK_TRY(relax_sweep(M, l, type, L.l1_down, f, cur, oth, FIN_NONE, nullptr));
         }
         double *tmp = cur; cur = oth; oth = tmp;
      }
   }
   *result = cur;
   return HDK_OK;
}

// buffer in which a cycle over levels [l0, nlev) entered with vectors (f, u0) keeps its iterate at
// the start: chosen so that the result lands in u0 without a copy (default sweeps)
static double *cycle_start_buffer(hdk_amg_s *M, int l0, double *u0, bool zero_guess)
{
   const hdk_amg_params &p = M->prm;
   const int nfine = M->tail ? M->nlev : M->nlev - 1;
   int       oop;
   if (nfine <= l0) oop = 0;
   else
   {
      int down_oop = zero_guess && is_jacobi(p.relax_down) ? (p.sweeps_down > 0 ? p.sweeps_down - 1 : 0) : p.sweeps_down;
      oop          = down_oop + p.sweeps_up;
   }
   const bool start_in_u0 = zero_guess ? (oop % 2 == 0) : true;
   return start_in_u0 ? u0 : M->lev[(size_t)l0].t;
}

// ---- CUDA graphs for the latency-bound part of the cycle ------------------------------------------
// The levels with few rows are a chain of ~20 small dependent kernels (6-40 us each, launch-latency
// bound).  All their operands are hierarchy-owned buffers, so the sub-cycle from the first small level
// down to the coarsest solve and back is captured ONCE into a CUDA graph (same kernels, same order:
// results are bit-identical) and replayed with one launch per V-cycle.  Tunable graph_rows
// (HDK_GRAPH_ROWS): levels with at most that many rows are replayed from a graph, 0 disables.
static int amg_cycle_impl(hdk_amg_s *M, const double *f0, double *u0, bool zero_guess, int fin, double *fin_out, int l0, int kg);

static int first_graph_level(hdk_amg_s *M, int l0)
{
   if (M->tail || M->graph_off) return -1;               // distributed levels take changing kernel arguments
   const int64_t rows = tune_graph_rows();
   if (rows <= 0) return -1;
   const hdk_amg_params &p = M->prm;
   // (two-stage GS may allocate scratch; Chebyshev sweeps use preallocated buffers only)
   if (!(is_jacobi(p.relax_down) || p.relax_down == 16) || !(is_jacobi(p.relax_up) || p.relax_up == 16)) return -1;
   for (int l = l0; l < M->nlev; l++)
      if (M->lev[(size_t)l].n <= rows) return l;
   return -1;
}

// run the cycle over [kg, nlev) with vectors (f, u) from a graph captured on first use
static int cycle_graph_run(hdk_amg_s *M, const double *f, double *u, bool zero_guess, bool prefilled, int kg)
{
   for (auto &G : M->graphs)
      if (G.f == f && G.u == u && G.zero_guess == zero_guess && G.prefilled == prefilled && G.level == kg)
      {
         HDK_CUDA(cudaGraphLaunch((cudaGraphExec_t)G.exec, g.stream));
         g.launches += G.nodes;
         return HDK_OK;
      }
   // capture (the launches below are recorded, not executed)
   const int64_t before = g.launches;
   cudaGraph_t   graph = nullptr;
   if (cudaStreamBeginCapture(g.stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess)
   {
      cudaGetLastError();
      M->graph_off = true;
      M->prefilled_at = prefilled ? kg : -1;
      return amg_cycle_impl(M, f, u, zero_guess, FIN_NONE, nullptr, kg, -1);
   }
   M->prefilled_at = prefilled ? kg : -1;
   int         rc = amg_cycle_impl(M, f, u, zero_guess, FIN_NONE, nullptr, kg, -1);
   cudaError_t e = cudaStreamEndCapture(g.stream, &graph);
   cudaGraphExec_t exec = nullptr;
   if (rc == HDK_OK && e == cudaSuccess && graph) e = cudaGraphInstantiate(&exec, graph, 0);
   if (graph) cudaGraphDestroy(graph);
   if (rc != HDK_OK || e != cudaSuccess || !exec)
   {
      // not capturable here: run directly from now on
      cudaGetLastError();
      M->graph_off = true;
      if (rc != HDK_OK) return rc;
      M->prefilled_at = prefilled ? kg : -1;
      return amg_cycle_impl(M, f, u, zero_guess, FIN_NONE, nullptr, kg, -1);
   }
   hdk_amg_s::CycleGraph G;
   G.f = f; G.u = u; G.zero_guess = zero_guess; G.prefilled = prefilled; G.level = kg; G.exec = exec;
   G.nodes = (int)(g.launches - before);
   g.launches = before;
   M->graphs.push_back(G);
   HDK_CUDA(cudaGraphLaunch(exec, g.stream));
   g.launches += G.nodes;
   return HDK_OK;
}

// One V-cycle over levels [l0, nlev) of M.  Level-l0 vectors are the caller's (f, u); u is also
// used as scratch.  With a replicated tail (N > 1) every level of M is a "fine" level and the
// coarsest stage is: sum the restricted right-hand side over ranks, run the serial tail cycle.
int amg_cycle(hdk_amg_s *M, const double *f0, double *u0, bool zero_guess, int fin, double *fin_out, int l0)
{
   int kg = first_graph_level(M, l0);
   if (kg == l0)
   {
      // the whole cycle is small: one graph, unless a fused dot has to come out of its last kernel
      if (fin == FIN_NONE)
      {
         const bool pf = (M->prefilled_at == l0) && zero_guess;
         M->prefilled_at = -1;
         return cycle_graph_run(M, f0, u0, zero_guess, pf, l0);
      }
      kg = (l0 + 1 < M->nlev) ? l0 + 1 : -1;
   }
   return amg_cycle_impl(M, f0, u0, zero_guess, fin, fin_out, l0, kg);
}

// kg > l0: the levels [kg, nlev) run as a sub-cycle replayed from a CUDA graph; kg < 0: all levels here
static int amg_cycle_impl(hdk_amg_s *M, const double *f0, double *u0, bool zero_guess, int fin, double *fin_out, int l0, int kg)
{
   const int             nl = M->nlev;
   const bool            has_tail = (M->tail != nullptr);
   const int             nfine = has_tail ? nl : nl - 1; // levels [l0, nfine) smooth + restrict
   const hdk_amg_params &p = M->prm;
   std::vector<double *> cur((size_t)nl + 1, nullptr), alt((size_t)nl + 1, nullptr);
   std::vector<const double *> rhs((size_t)nl + 1, nullptr);
   bool                  fin_done = false;
   if (has_tail && nl == 0)
   {
      // the whole hierarchy is replicated: gather the right-hand side, cycle, take my slice
      HDK_TRY(vec_fill(M->full_f, 0.0, M->tail_n));
      HDK_TRY(vec_copy(M->full_f + M->tail_off, f0, M->tail_cnt));
      HDK_TRY(allreduce_dev(M->full_f, (int)M->tail_n));
      if (!zero_guess)
      {
         HDK_TRY(vec_fill(M->full_u, 0.0, M->tail_n));
         HDK_TRY(vec_copy(M->full_u + M->tail_off, u0, M->tail_cnt));
         HDK_TRY(allreduce_dev(M->full_u, (int)M->tail_n));
      }
      HDK_TRY(amg_cycle(M->tail, M->full_f, M->full_u, zero_guess, FIN_NONE, nullptr, M->tail_level));
      HDK_TRY(vec_copy(u0, M->full_u + M->tail_off, M->tail_cnt));
      if (fin != FIN_NONE) HDK_TRY(vec_dot_dev(f0, u0, M->tail_cnt, fin, fin_out));
      return HDK_OK;
   }
   // level-l0 buffer parity so that the result lands in u0 without a copy (default sweeps)
   {
      AmgLevel &L0 = M->lev[(size_t)l0];
      cur[(size_t)l0] = cycle_start_buffer(M, l0, u0, zero_guess);
      alt[(size_t)l0] = (cur[(size_t)l0] == u0) ? L0.t : u0;
      rhs[(size_t)l0] = f0;
   }
   for (int l = l0 + 1; l < nl; l++) { cur[(size_t)l] = M->lev[(size_t)l].u; alt[(size_t)l] = M->lev[(size_t)l].t; rhs[(size_t)l] = M->lev[(size_t)l].f; }

   // the first pre-smoothing sweep of a level entered with a zero guess is u = (w f)/d: it is
   // produced by the kernel that produces f (the restriction of the level above, or the PCG
   // residual update for level l0), so it costs no pass of its own
   bool prefilled = (M->prefilled_at == l0) && zero_guess;
   M->prefilled_at = -1;
   const bool sub = (kg > l0 && kg < nl);              // levels [kg, nl) replayed from a graph
   const int  ndown = sub ? kg : nfine;                // levels [l0, ndown) smooth + restrict here
   if (sub) cur[(size_t)kg] = cycle_start_buffer(M, kg, M->lev[(size_t)kg].u, true); // where the sub-cycle expects its first sweep
   for (int l = l0; l < ndown; l++)
   {
      AmgLevel &L = M->lev[(size_t)l];
      bool      zg = (l > l0) || zero_guess;
      for (int s = 0; s < p.sweeps_down; s++)
      {
         if (s == 0 && zg && is_jacobi(p.relax_down))
         {
            // (the next product on this level -- another sweep or the residual -- reads this vector)
            tl_mark(l, 5);
            if (!prefilled) HDK_TRY(vec_scaled_div(cur[(size_t)l], rhs[(size_t)l], L.l1_down, p.relax_weight, L.n, L.A));
         }
         else
         {
            tl_mark(l, 10);
            if (s == 0 && zg && p.relax_down == 16) // Chebyshev from a zero guess: no fill, no residual product
               HDK_TRY(cheby_sweep(M, l, rhs[(size_t)l], nullptr, alt[(size_t)l], FIN_NONE, nullptr, L.A));
            else
            {
               if (s == 0 && zg) HDK_TRY(vec_fill(cur[(size_t)l], 0.0, L.n));
               HDK_TRY(relax_sweep(M, l, p.relax_down, L.l1_down, rhs[(size_t)l], cur[(size_t)l], alt[(size_t)l], FIN_NONE, nullptr, L.A));
            }
            std::swap(cur[(size_t)l], alt[(size_t)l]);
         }
      }
      if (p.sweeps_down == 0 && zg) HDK_TRY(vec_fill(cur[(size_t)l], 0.0, L.n));
      // residual into the spare buffer, restrict to the next level
      if (p.sweeps_down == 0 && zg)
      {
         HDK_TRY(vec_copy(alt[(size_t)l], rhs[(size_t)l], L.n));
      }
      else
      {
         SpmvArgs a;
         a.x = cur[(size_t)l]; a.y = alt[(size_t)l]; a.b = rhs[(size_t)l];
         a.export_to = L.R;                                    // the restriction reads the residual next
         tl_mark(l, 1);
         HDK_TRY(parcsr_matvec(*L.A, SPMV_RESIDUAL, a));
      }
      SpmvArgs rr;
      tl_mark(l, 2);
      rr.x = alt[(size_t)l];
      prefilled = false;
      if (l + 1 < nl) rr.y = M->lev[(size_t)l + 1].f;
      else
      {
         // first replicated level: my rows of the coarse right-hand side go into the full vector
         if (M->gather.on) rr.y = ipc_gather_buffer(M->gather) + M->tail_off; // every slice is overwritten by its owner
         else
         {
            HDK_TRY(vec_fill(M->full_f, 0.0, M->tail_n));
            rr.y = M->full_f + M->tail_off;
         }
      }
      if (l + 1 < nfine && p.sweeps_down > 0 && is_jacobi(p.relax_down))
      {
         // f_{l+1} = R r  and  u_{l+1} = (w f_{l+1})/d_{l+1}  in one kernel
         rr.y2 = cur[(size_t)l + 1]; rr.d = M->lev[(size_t)l + 1].l1_down; rr.w = p.relax_weight;
         if (!(sub && l + 1 == kg)) { rr.export_to = M->lev[(size_t)l + 1].A; rr.export_y2 = true; } // its first product reads the sweep
         HDK_TRY(parcsr_matvec(*L.R, SPMV_SET_DIV, rr));
         prefilled = true;
      }
      else HDK_TRY(parcsr_matvec(*L.R, SPMV_SET, rr));
   }
   // coarsest stage
   const double *coarse_sol = nullptr; // solution feeding the prolongation of level nfine-1
   tl_mark(ndown, 6);
   if (sub)
   {
      AmgLevel &Lk = M->lev[(size_t)kg];
      HDK_TRY(cycle_graph_run(M, Lk.f, Lk.u, true, prefilled, kg));
      cur[(size_t)kg] = Lk.u;                          // the sub-cycle leaves its result in u
   }
   else if (has_tail)
   {
      // the ranks own disjoint slices of the coarse right-hand side: with the peer-memory arena each
      // rank stores its slice into every peer's copy (one kernel + a flag wait), else NCCL sums the
      // zero-padded vectors
      const double *tf = M->full_f;
      if (M->gather.on)
      {
         HDK_TRY(ipc_gather(M->gather, M->tail_off, M->tail_cnt));
         tf = M->gather.buf[M->gather.seq & 1];
      }
      else HDK_TRY(allreduce_dev(M->full_f, (int)M->tail_n));
      HDK_TRY(amg_cycle(M->tail, tf, M->full_u, true, FIN_NONE, nullptr, M->tail_level));
      coarse_sol = M->full_u;
   }
   else
   {
      const int Lc = nl - 1;
      double   *res;
      bool      zg = (Lc > l0) || zero_guess;
      HDK_TRY(coarse_solve(M, Lc, rhs[(size_t)Lc], cur[(size_t)Lc], alt[(size_t)Lc], zg, &res));
      if (res != cur[(size_t)Lc]) std::swap(cur[(size_t)Lc], alt[(size_t)Lc]);
      coarse_sol = cur[(size_t)Lc];
   }
   for (int l = ndown - 1; l >= l0; l--)
   {
      AmgLevel &L = M->lev[(size_t)l];
      // u += P e_c
      tl_mark(l, 3);
      SpmvArgs a;
      a.x = (l + 1 < nl) ? cur[(size_t)l + 1] : coarse_sol;
      a.y = cur[(size_t)l];
      if (p.sweeps_up > 0) a.export_to = L.A;                  // the post-smoothing sweep reads the corrected iterate
      else if (l > l0) a.export_to = M->lev[(size_t)l - 1].P;
      HDK_TRY(parcsr_matvec(*L.P, SPMV_ADD, a));
      for (int s = 0; s < p.sweeps_up; s++)
      {
         bool last = (l == l0 && s == p.sweeps_up - 1);
         int  f_   = (last && fin != FIN_NONE) ? fin : FIN_NONE;
         // reader of this sweep's result: the next sweep, or the prolongation of the level above
         const hdk_csr_s *next = (s + 1 < p.sweeps_up) ? L.A : (l > l0 ? M->lev[(size_t)l - 1].P : nullptr);
         tl_mark(l, 4);
         HDK_TRY(relax_sweep(M, l, p.relax_up, L.l1_up, rhs[(size_t)l], cur[(size_t)l], alt[(size_t)l], f_, fin_out, next));
         std::swap(cur[(size_t)l], alt[(size_t)l]);
         if (f_ != FIN_NONE) fin_done = true;
      }
   }
   tl_mark(l0, 0);
   if (cur[(size_t)l0] != u0) HDK_TRY(vec_copy(u0, cur[(size_t)l0], M->lev[(size_t)l0].n));
   if (fin != FIN_NONE && !fin_done) HDK_TRY(vec_dot_dev(f0, u0, M->lev[(size_t)l0].n, fin, fin_out));
   return HDK_OK;
}

// For a caller that can produce u0 = (w r)/d itself (PCG's fused x/r update): the buffer the
// V-cycle expects it in, the diagonal and the weight.  false: the cycle does not start that way.
bool amg_prefill_target(hdk_amg_s *M, double *z, double **buf, const double **d, double *w, const hdk_csr_s **reader)
{
   if (reader) *reader = (M->nlev > 0) ? M->lev[0].A : nullptr; // the matrix whose product reads the first sweep
   const hdk_amg_params &p = M->prm;
   const bool has_tail = (M->tail != nullptr);
   const int  nl = M->nlev, nfine = has_tail ? nl : nl - 1;
   if (nl == 0 || nfine <= 0 || p.sweeps_down <= 0 || !is_jacobi(p.relax_down)) return false;
   const int  oop = (p.sweeps_down - 1) + p.sweeps_up;
   *buf = (oop % 2 == 0) ? z : M->lev[0].t;
   *d   = M->lev[0].l1_down;
   *w   = p.relax_weight;
   return true;
}

int amg_precond(hdk_amg_s *M, const double *r, double *z, int fin, double *fin_out)
{
   return amg_cycle(M, r, z, true, fin, fin_out, 0);
}

} // namespace hdk

using namespace hdk;

extern "C" {

int hdk_amg_apply(hdk_amg *M, const double *r_d, double *z_d)
{
   HDK_TRY(require_init());
   if (!M) return set_error(HDK_ERR_INVALID, "null hierarchy");
   return amg_precond(M, r_d, z_d, FIN_NONE, nullptr);
}

int hdk_amg_vcycle(hdk_amg *M, const double *f_d, double *u_d)
{
   HDK_TRY(require_init());
   if (!M) return set_error(HDK_ERR_INVALID, "null hierarchy");
   return amg_cycle(M, f_d, u_d, false, FIN_NONE, nullptr, 0);
}

// CUDA-event timing of one hot kernel, `reps` back-to-back launches (bench.py roofline leg)
int hdk_time_kernel(const hdk_csr *A, hdk_amg *M, int kernel, int reps, double *avg_ms, double *bytes)
{
   HDK_TRY(require_init());
   if (!A) return set_error(HDK_ERR_INVALID, "null matrix");
   const int64_t n = A->diag.nrows;
   const double  nnz = (double)A->diag.nnz + A->offd.nnz;
   double *x, *y, *b, *d, *z;
   HDK_TRY(dalloc(&x, (size_t)n + 8)); HDK_TRY(dalloc(&y, (size_t)n + 8));
   HDK_TRY(dalloc(&b, (size_t)n + 8)); HDK_TRY(dalloc(&d, (size_t)n + 8));
   HDK_TRY(dalloc(&z, (size_t)n + 8));
   HDK_TRY(hdk_vec_random(x, n, A->row_start, 1));
   HDK_TRY(hdk_vec_random(b, n, A->row_start, 2));
   HDK_TRY(vec_fill(d, 6.0, n));
   HDK_TRY(vec_fill(y, 0.0, n));
   double by = 0.0;
   int    rc = HDK_OK;
   for (int pass = 0; pass < 2 && rc == HDK_OK; pass++)
   {
      int count = pass == 0 ? 3 : reps; // warm-up, then timed
      if (pass == 1) HDK_CUDA(cudaEventRecord(g.ev_a, g.stream));
      for (int it = 0; it < count && rc == HDK_OK; it++)
      {
         SpmvArgs a;
         a.x = x; a.y = y; a.b = b; a.d = d;
         switch (kernel)
         {
            case 0: rc = parcsr_matvec(*A, SPMV_SET, a); by = 12.0 * nnz + 4.0 * (n + 1) + 16.0 * n; break;
            case 1: rc = parcsr_matvec(*A, SPMV_JACOBI, a); by = 12.0 * nnz + 4.0 * (n + 1) + 32.0 * n; break;
            case 2: rc = parcsr_matvec(*A, SPMV_RESIDUAL, a); by = 12.0 * nnz + 4.0 * (n + 1) + 24.0 * n; break;
            case 3: // the variant the PCG solve runs: x/r update + <r,r> + the V-cycle's first sweep z0 = (w r)/l1
               rc = vec_fill(g.dscal + S_ALPHA, 1e-3, 1);
               if (rc == HDK_OK) rc = pcg_update_xr(y, b, x, d, n, g.dscal, FIN_IPROD, nullptr, z, d, 1.0);
               by = 64.0 * n; break;
            case 5: // p = z + beta p
               rc = vec_fill(g.dscal + S_BETA, 0.5, 1);
               if (rc == HDK_OK) rc = pcg_update_p(y, x, n, g.dscal);
               by = 24.0 * n; break;
            case 4:
               if (!M) rc = set_error(HDK_ERR_INVALID, "V-cycle timing needs a hierarchy");
               else { rc = amg_precond(M, b, y, FIN_NONE, nullptr); by = M->vcycle_bytes; }
               break;
            case 6: // one two-stage Gauss-Seidel sweep on the fine level (hierarchy set up with relax 11 or 12)
               if (!M || M->nlev < 1 || !M->lev[0].L.rowptr) rc = set_error(HDK_ERR_INVALID, "two-stage GS timing needs a hierarchy set up with relaxation 11 or 12");
               else
               {
                  const int    type = (M->prm.relax_down == 12 || M->prm.relax_up == 12) ? 12 : 11;
                  const double nnzL = (double)M->lev[0].L.nnz;
                  rc = relax_sweep(M, 0, type, M->lev[0].l1_down, b, x, y, FIN_NONE, nullptr);
                  // stage 1 reads A, u, f, d and writes r, u+r; every inner step reads L, r, d, u and writes u (and r)
                  by = 12.0 * nnz + 4.0 * (n + 1) + 40.0 * n + (type == 11 ? 1 : 2) * (12.0 * nnzL + 4.0 * (n + 1) + 32.0 * n) + (type == 12 ? 8.0 * n : 0.0);
               }
               break;
            case 9: // one Chebyshev sweep on the fine level (hierarchy set up with relaxation 16)
               if (!M || M->nlev < 1 || !M->lev[0].cheb_ds) rc = set_error(HDK_ERR_INVALID, "Chebyshev timing needs a hierarchy whose fine level smooths with relaxation 16");
               else
               {
                  const int    k = M->prm.cheby_order;
                  const double pass = 12.0 * nnz + 4.0 * (n + 1);
                  rc = cheby_sweep(M, 0, b, x, y, FIN_NONE, nullptr);
                  // START reads u, f, ds and writes r, w; each STEP reads w, r, ds and writes w; FIN also reads u_old
                  by = (k == 1) ? pass + 32.0 * n : k * pass + 40.0 * n + (k - 2) * 32.0 * n + 40.0 * n;
               }
               break;
            case 7: rc = halo_exchange_begin(*A, x); by = 8.0 * A->halo.n_send; break; // the halo exchange alone (N > 1)
            case 8: // the product without its exchange (N > 1: what the fused off-diagonal part costs)
               dbg_skip_exchange(true);
               rc = parcsr_matvec(*A, SPMV_SET, a); by = 12.0 * nnz + 4.0 * (n + 1) + 16.0 * n;
               dbg_skip_exchange(false);
               break;
            default: rc = set_error(HDK_ERR_INVALID, "unknown kernel id %d", kernel);
         }
      }
   }
   if (rc == HDK_OK)
   {
      HDK_CUDA(cudaEventRecord(g.ev_b, g.stream));
      HDK_CUDA(cudaEventSynchronize(g.ev_b));
      float ms = 0.f;
      HDK_CUDA(cudaEventElapsedTime(&ms, g.ev_a, g.ev_b));
      if (avg_ms) *avg_ms = (double)ms / (reps > 0 ? reps : 1);
      if (bytes) *bytes = by;
   }
   dfree(x); dfree(y); dfree(b); dfree(d); dfree(z);
   return rc;
}

} // extern "C"
