// hdk_spmv.cu -- the fused CSR SpMV family (north-star items 1 and 2):
//   y = A x | r = b - A x | l1-Jacobi sweep fused with its residual | y += A x | axpby
// each optionally fused with a dot product of the result (PCG <Ap,p>, <r,z>).
// Stands in for hypre_ParCSRMatrixMatvec / hypre_ParCSRMatrixMatvecOutOfPlace and
// hypre_BoomerAMGRelax (types 7, 18) -- reference call sites src/internal/linsys.c:1835, 3031,
// src/internal/solver.c:614 (every Krylov iteration) and the V-cycle behind solver.c:314-329.
//
// Kernel choice by measured row-length statistics (csr_analyze):
//  * STREAM (max_row <= 1024): persistent CTAs walk nnz-balanced row blocks (about one row per
//    thread).  One elected thread issues 1-D TMA bulk copies (cp.async.bulk -> UBLKCP) of the
//    block's contiguous val / col ranges into one of two shared-memory stages, tracked by an
//    mbarrier; while block i+1 is in flight, block i is consumed one row per thread: col/val
//    come from shared memory (conflict-free for odd row lengths), x is gathered through L1 --
//    coalesced across the rows of a warp on stencil matrices -- and the row is accumulated
//    sequentially in CSR order with separately rounded multiply and add, so results are
//    bit-identical to the CPU oracle.  HBM sees only perfectly contiguous bulk reads.
//  * VECTOR (longer rows): one warp per row, shuffle reduction.
#include "hdk_internal.cuh"
#include "hdk_amg.cuh"
#include <stdlib.h>
#include <string.h>
#include <map>

namespace hdk {

constexpr int ST       = 256;   // threads per CTA
constexpr int S_TGT_LO = 1024;  // non-zeros per block: bounds
constexpr int S_TGT_HI = 8192;
constexpr int S_MAXR   = 1024;  // longest row the stream kernel accepts

// kernel-selection tunables: defaults, overridden by environment variables at first use and by
// hdk_tune() at any time (they apply to matrices analysed afterwards)
struct Tune
{
   double rows_mult     = 1.0;      // HDK_SPMV_ROWS_MULT   rows per thread of a stream-kernel block
   double tgt_max       = 3072;     // HDK_SPMV_TGT_MAX     non-zeros per stream-kernel block (cap)
   double lpr           = 0;        // HDK_SPMV_LPR         force lanes per row (0 = by row length)
   double sell_min_rows = 200000;   // HDK_SELL_MIN_ROWS    sliced-ELL for matrices with at least this many rows
   double sell_min_rows_dist = 30000;  // HDK_SELL_MIN_ROWS_DIST  the same for slabs with off-rank entries (fused off-rank block)
   double sell_min_avg  = 0.0;      // HDK_SELL_MIN_AVG     ... and more than this many non-zeros per row
   double sell_sort     = 1;        // HDK_SELL_SORT        sort the columns of coarse operators in the slices
   double amg_keep_debug = 0;       // HDK_AMG_KEEP_DEBUG   keep S and the PMIS measures of every level (introspection)
   double replicate_rows = 262144;  // HDK_REPLICATE_ROWS   N > 1: levels with at most this many global rows form the replicated tail
   double export_max_rows = 1e18;   // HDK_EXPORT_MAX_ROWS  N > 1: operators with more rows pack their halo instead of folding the export
   double graph_rows    = 150000;   // HDK_GRAPH_ROWS       V-cycle levels with at most this many rows are replayed from a CUDA graph (0: off)
   bool   env_read      = false;
};
static Tune tune;
static const struct { const char *key, *env; double Tune::*field; } tune_keys[] = {
   {"spmv_rows_mult", "HDK_SPMV_ROWS_MULT", &Tune::rows_mult}, {"spmv_tgt_max", "HDK_SPMV_TGT_MAX", &Tune::tgt_max},
   {"spmv_lpr", "HDK_SPMV_LPR", &Tune::lpr},                   {"sell_min_rows", "HDK_SELL_MIN_ROWS", &Tune::sell_min_rows},
   {"sell_min_rows_dist", "HDK_SELL_MIN_ROWS_DIST", &Tune::sell_min_rows_dist},
   {"amg_keep_debug", "HDK_AMG_KEEP_DEBUG", &Tune::amg_keep_debug},
   {"replicate_rows", "HDK_REPLICATE_ROWS", &Tune::replicate_rows},
   {"graph_rows", "HDK_GRAPH_ROWS", &Tune::graph_rows},
   {"export_max_rows", "HDK_EXPORT_MAX_ROWS", &Tune::export_max_rows},
   {"sell_min_avg", "HDK_SELL_MIN_AVG", &Tune::sell_min_avg},  {"sell_sort", "HDK_SELL_SORT", &Tune::sell_sort}};
static Tune &tunables()
{
   if (!tune.env_read)
   {
      tune.env_read = true;
      for (const auto &k : tune_keys)
      {
         const char *e = getenv(k.env);
         if (e && *e) tune.*(k.field) = atof(e);
      }
   }
   return tune;
}
bool tune_amg_keep_debug() { return tunables().amg_keep_debug != 0.0; }
int64_t tune_replicate_rows() { return (int64_t)tunables().replicate_rows; }
int64_t tune_graph_rows() { return (int64_t)tunables().graph_rows; }

int tune_set(const char *key, double value)
{
   Tune &t = tunables();
   for (const auto &k : tune_keys)
      if (!strcmp(key, k.key)) { t.*(k.field) = value; return HDK_OK; }
   return set_error(HDK_ERR_INVALID, "unknown tunable '%s'", key);
}

struct SpmvDev
{
   const int    *rowptr, *col, *blk_row;
   const double *val;
   const double *x, *b, *d, *dotv;
   double       *y, *y2;
   double        w, alpha, beta;
   int           nrows, fin;
   double       *fin_out, *scal, *partials;
   unsigned     *ticket;
   // sliced-ELL operands (kind 2)
   const int    *sl_off, *sl_meta, *sl_col;
   const double *sl_val;
   int           nslice;
   // fused off-rank block (N > 1, see OffdFuse): CSR arrays of the block and the halo buffer; has_halo
   // selects the multi-rank kernel variants
   const int    *orp, *ocol;
   const double *oval, *xh;
   int           has_halo;

   // halo of the NEXT product filled by this kernel (see HaloExport); exp_y2: the exported vector is y2
   HaloExport    exp;
   int           exp_y2;
   const double *uo; // Chebyshev finish: the iterate the correction is added to (nullptr: zero)
};

// ---- PTX helpers: mbarrier + 1-D bulk tensor-memory-accelerator copies -------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
   asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
   asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
   asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
   asm volatile("{\n"
                ".reg .pred P1;\n"
                "LAB_WAIT:\n"
                "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
                "@P1 bra DONE;\n"
                "bra LAB_WAIT;\n"
                "DONE:\n"
                "}" ::"r"(bar), "r"(parity) : "memory");
}

// second output of SPMV_SET_DIV: the zero-guess l1-Jacobi sweep of the next level, u = (w*f)/d
// (same expression as k_scaled_div)
// writes the outputs of row r and returns the value of y (what a fused dot multiplies).  `v` is the
// result of the row epilogue: y for most modes, the correction w(b - Ax)/d for JACOBI2, A x for GS_STEP.
// The row of the output that feeds the next product is also handed to the halo export.
template <int MODE, bool EXP = false>
__device__ __forceinline__ double store_out(const SpmvDev &a, int r, double v, double dd, double xo, int &nexp)
{
   double yn = v, y2 = 0.0;
   if (MODE == SPMV_JACOBI2)
   {
      yn = __dadd_rn(xo, v);
      y2 = v;
      a.y2[r] = y2;
   }
   else if (MODE == SPMV_GS_STEP)
   {
      y2 = (dd != 0.0) ? __ddiv_rn(v, dd) : 0.0;
      yn = __dadd_rn(a.y[r], __dmul_rn(a.alpha, y2));
      if (a.y2) a.y2[r] = y2;
   }
   else if (MODE == SPMV_SET_DIV)
   {
      y2 = (dd != 0.0) ? __ddiv_rn(__dmul_rn(a.w, v), dd) : 0.0;
      a.y2[r] = y2;
   }
   else if (MODE == SPMV_CHEB_START)
   {
      // v = r = ds (f - A u): kept for the later passes; y = ds (c r) is what the next product gathers
      y2 = v;
      a.y2[r] = y2;
      yn = __dmul_rn(dd, __dmul_rn(a.alpha, v));
   }
   a.y[r] = yn;
   // (compiled only into the multi-rank sliced-ELL variants: the plain kernels keep their 32 registers)
   if (EXP && a.exp.seq) nexp += export_row(a.exp, r, a.exp_y2 ? y2 : yn);
   return yn;
}

template <int MODE>
__device__ __forceinline__ double store_out(const SpmvDev &a, int r, double v, double dd, double xo)
{
   int none = 0;
   return store_out<MODE, false>(a, r, v, dd, xo, none);
}

struct BlkMeta { int r0, r1, k0, k1; };
__device__ __forceinline__ BlkMeta blk_meta(const SpmvDev &a, int b)
{
   BlkMeta m;
   m.r0 = __ldg(a.blk_row + b);
   m.r1 = __ldg(a.blk_row + b + 1);
   m.k0 = __ldg(a.rowptr + m.r0);
   m.k1 = __ldg(a.rowptr + m.r1);
   return m;
}

// per-row operands of the epilogue, loaded before the wait on the bulk copy
struct RowOps
{
   int    s, e;
   double b, d, xo, yo, dv;
};

// Chebyshev epilogues (relax 16), every product and sum rounded separately in the order of the
// polynomial loop (DESIGN.md section 4): o.d = ds, o.b = f (START, ONE: acc is already f - A u) or the
// scaled residual r (STEP, FIN: acc = A w), o.yo = u_old, alpha = the coefficient of this pass
template <int MODE>
__device__ __forceinline__ double cheb_epilogue(const SpmvDev &a, const RowOps &o, double acc)
{
   if (MODE == SPMV_CHEB_START) return __dmul_rn(o.d, acc);
   if (MODE == SPMV_CHEB_ONE) return __dadd_rn(o.yo, __dmul_rn(o.d, __dmul_rn(a.alpha, __dmul_rn(o.d, acc))));
   const double v = __dadd_rn(__dmul_rn(a.alpha, o.b), __dmul_rn(o.d, acc));
   if (MODE == SPMV_CHEB_STEP) return __dmul_rn(o.d, v);
   return __dadd_rn(o.yo, __dmul_rn(o.d, v));
}
template <int MODE>
__device__ __forceinline__ void cheb_load(const SpmvDev &a, int r, RowOps &o)
{
   o.b = a.b[r];
   o.d = a.d[r];
   if (MODE == SPMV_CHEB_FIN || MODE == SPMV_CHEB_ONE) o.yo = a.uo ? a.uo[r] : 0.0;
}

template <int MODE, bool DOT>
__device__ __forceinline__ void row_load(const SpmvDev &a, int r, int ka, RowOps &o)
{
   o.s = __ldg(a.rowptr + r) - ka;
   o.e = __ldg(a.rowptr + r + 1) - ka;
   if (MODE == SPMV_RESIDUAL || MODE == SPMV_JACOBI || MODE == SPMV_JACOBI_R || MODE == SPMV_JACOBI2) o.b = a.b[r];
   if (MODE == SPMV_JACOBI || MODE == SPMV_JACOBI_R || MODE == SPMV_SET_DIV || MODE == SPMV_JACOBI2 || MODE == SPMV_GS_STEP) o.d = a.d[r];
   if (MODE == SPMV_JACOBI || MODE == SPMV_JACOBI2) o.xo = a.x[r];
   if (MODE == SPMV_ADD || MODE == SPMV_AXPBY) o.yo = a.y[r];
   if (MODE >= SPMV_CHEB_START) cheb_load<MODE>(a, r, o);
   if (DOT) o.dv = a.dotv[r];
}

// one row: sequential accumulation in CSR order from the staged val / col, fused epilogue
template <int MODE>
__device__ __forceinline__ double row_compute(const SpmvDev &a, const RowOps &o, const double *vs, const int *cs)
{
   constexpr bool SUB = (MODE == SPMV_RESIDUAL || MODE == SPMV_JACOBI || MODE == SPMV_JACOBI_R || MODE == SPMV_JACOBI2 ||
                         MODE == SPMV_CHEB_START || MODE == SPMV_CHEB_ONE);
   double acc = SUB ? o.b : ((MODE == SPMV_ADD) ? o.yo : 0.0);
   int    k = o.s;
   // groups of four: issue the gathers together, then accumulate in order
   for (; k + 4 <= o.e; k += 4)
   {
      int    c0 = cs[k], c1 = cs[k + 1], c2 = cs[k + 2], c3 = cs[k + 3];
      double x0 = __ldg(a.x + c0), x1 = __ldg(a.x + c1), x2 = __ldg(a.x + c2), x3 = __ldg(a.x + c3);
      double p0 = __dmul_rn(vs[k], x0), p1 = __dmul_rn(vs[k + 1], x1);
      double p2 = __dmul_rn(vs[k + 2], x2), p3 = __dmul_rn(vs[k + 3], x3);
      if (SUB) { acc = __dadd_rn(acc, -p0); acc = __dadd_rn(acc, -p1); acc = __dadd_rn(acc, -p2); acc = __dadd_rn(acc, -p3); }
      else { acc = __dadd_rn(acc, p0); acc = __dadd_rn(acc, p1); acc = __dadd_rn(acc, p2); acc = __dadd_rn(acc, p3); }
   }
   if (k < o.e)
   {
      // tail of 1..3 entries, gathers issued together
      int    c0 = cs[k], c1 = (k + 1 < o.e) ? cs[k + 1] : c0, c2 = (k + 2 < o.e) ? cs[k + 2] : c0;
      double x0 = __ldg(a.x + c0), x1 = __ldg(a.x + c1), x2 = __ldg(a.x + c2);
      double p0 = __dmul_rn(vs[k], x0);
      acc       = __dadd_rn(acc, SUB ? -p0 : p0);
      if (k + 1 < o.e) { double p1 = __dmul_rn(vs[k + 1], x1); acc = __dadd_rn(acc, SUB ? -p1 : p1); }
      if (k + 2 < o.e) { double p2 = __dmul_rn(vs[k + 2], x2); acc = __dadd_rn(acc, SUB ? -p2 : p2); }
   }
   if (MODE >= SPMV_CHEB_START) return cheb_epilogue<MODE>(a, o, acc);
   if (MODE == SPMV_SET || MODE == SPMV_SET_DIV || MODE == SPMV_ADD || MODE == SPMV_RESIDUAL || MODE == SPMV_GS_STEP) return acc;
   if (MODE == SPMV_AXPBY)
      return (a.beta == 0.0) ? __dmul_rn(a.alpha, acc) : __dadd_rn(__dmul_rn(a.alpha, acc), __dmul_rn(a.beta, o.yo));
   if (MODE == SPMV_JACOBI)
      return (o.d != 0.0) ? __dadd_rn(o.xo, __ddiv_rn(__dmul_rn(a.w, acc), o.d)) : o.xo;
   /* SPMV_JACOBI_R, SPMV_JACOBI2: the correction */
   return (o.d != 0.0) ? __ddiv_rn(__dmul_rn(a.w, acc), o.d) : 0.0;
}

// several lanes per row (long rows): lane `sub` of LPR sums entries s+sub, s+sub+LPR, ...;
// the LPR partials are combined by a fixed-order butterfly (deterministic, but not the
// sequential CSR order -- fp parity with the oracle within tolerance)
template <int LPR>
__device__ __forceinline__ double row_partial(const SpmvDev &a, int k, int e, const double *vs, const int *cs)
{
   double acc = 0.0;
   for (; k + 3 * LPR < e; k += 4 * LPR)
   {
      int    c0 = cs[k], c1 = cs[k + LPR], c2 = cs[k + 2 * LPR], c3 = cs[k + 3 * LPR];
      double x0 = __ldg(a.x + c0), x1 = __ldg(a.x + c1), x2 = __ldg(a.x + c2), x3 = __ldg(a.x + c3);
      acc = __dadd_rn(acc, __dmul_rn(vs[k], x0));
      acc = __dadd_rn(acc, __dmul_rn(vs[k + LPR], x1));
      acc = __dadd_rn(acc, __dmul_rn(vs[k + 2 * LPR], x2));
      acc = __dadd_rn(acc, __dmul_rn(vs[k + 3 * LPR], x3));
   }
   for (; k < e; k += LPR) acc = __dadd_rn(acc, __dmul_rn(vs[k], __ldg(a.x + cs[k])));
   return acc;
}

template <int MODE>
__device__ __forceinline__ double row_finish(const SpmvDev &a, const RowOps &o, double total)
{
   if (MODE >= SPMV_CHEB_START)
      return cheb_epilogue<MODE>(a, o, (MODE == SPMV_CHEB_START || MODE == SPMV_CHEB_ONE) ? __dadd_rn(o.b, -total) : total);
   if (MODE == SPMV_SET || MODE == SPMV_SET_DIV || MODE == SPMV_GS_STEP) return total;
   if (MODE == SPMV_ADD) return __dadd_rn(o.yo, total);
   if (MODE == SPMV_AXPBY)
      return (a.beta == 0.0) ? __dmul_rn(a.alpha, total) : __dadd_rn(__dmul_rn(a.alpha, total), __dmul_rn(a.beta, o.yo));
   double res = __dadd_rn(o.b, -total);
   if (MODE == SPMV_RESIDUAL) return res;
   if (MODE == SPMV_JACOBI)
      return (o.d != 0.0) ? __dadd_rn(o.xo, __ddiv_rn(__dmul_rn(a.w, res), o.d)) : o.xo;
   return (o.d != 0.0) ? __ddiv_rn(__dmul_rn(a.w, res), o.d) : 0.0;
}

template <int MODE, bool DOT, int LPR>
__global__ void __launch_bounds__(ST, 4) k_spmv_tma(SpmvDev a, int nblk, int cap)
{
   constexpr int PF  = 2;        // row rounds whose operands are prefetched
   constexpr int RPB = ST / LPR; // rows per round
   extern __shared__ __align__(128) unsigned char smem_raw[];
   __shared__ double red[ST / 32];
   __shared__ int    flag;
   double *vbuf = reinterpret_cast<double *>(smem_raw + 128);
   int    *cbuf = reinterpret_cast<int *>(smem_raw + 128 + (size_t)2 * cap * sizeof(double));
   const uint32_t bar0 = smem_u32(smem_raw), bar1 = bar0 + 8;
   const int tid = threadIdx.x, G = gridDim.x;
   if (tid == 0)
   {
      mbar_init(bar0, 1);
      mbar_init(bar1, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
   }
   __syncthreads();
   int      b = blockIdx.x, nb = b + G;
   int      stage = 0;
   uint32_t ph0 = 0u, ph1 = 0u;
   double   dacc = 0.0;
   BlkMeta  cur = BlkMeta{0, 0, 0, 0}, nxt = BlkMeta{0, 0, 0, 0};
   if (b < nblk)
   {
      cur = blk_meta(a, b);
      int ka = cur.k0 & ~3, len4 = (cur.k1 - ka + 3) & ~3;
      if (tid == 0 && len4 > 0)
      {
         mbar_expect_tx(bar0, (uint32_t)len4 * 12u);
         tma_load_1d(smem_u32(vbuf), a.val + ka, (uint32_t)len4 * 8u, bar0);
         tma_load_1d(smem_u32(cbuf), a.col + ka, (uint32_t)len4 * 4u, bar0);
      }
   }
   if (nb < nblk) nxt = blk_meta(a, nb);
   while (b < nblk)
   {
      // 1. bulk copies of the next block into the other stage (its readers passed the barrier
      //    that closed the previous iteration)
      if (nb < nblk && tid == 0)
      {
         int ka = nxt.k0 & ~3, len4 = (nxt.k1 - ka + 3) & ~3;
         if (len4 > 0)
         {
            const uint32_t bar = stage ? bar0 : bar1;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar, (uint32_t)len4 * 12u);
            tma_load_1d(smem_u32(vbuf + (size_t)(stage ^ 1) * cap), a.val + ka, (uint32_t)len4 * 8u, bar);
            tma_load_1d(smem_u32(cbuf + (size_t)(stage ^ 1) * cap), a.col + ka, (uint32_t)len4 * 4u, bar);
         }
      }
      // 2. metadata two blocks ahead, 3. per-row operands of this block (plain global loads)
      const int nnb = nb + G;
      BlkMeta   nn  = BlkMeta{0, 0, 0, 0};
      if (nnb < nblk) nn = blk_meta(a, nnb);
      const int ka = cur.k0 & ~3, len = cur.k1 - ka;
      RowOps    ro[PF];
#pragma unroll
      for (int j = 0; j < PF; ++j)
      {
         int r = cur.r0 + tid / LPR + j * RPB;
         if (r < cur.r1) row_load<MODE, DOT>(a, r, ka, ro[j]);
      }
      // 4. wait for this block's val / col
      const double *vs = vbuf + (size_t)stage * cap;
      const int    *cs = cbuf + (size_t)stage * cap;
      if (len > 0)
      {
         if (stage) { mbar_wait(bar1, ph1); ph1 ^= 1u; }
         else { mbar_wait(bar0, ph0); ph0 ^= 1u; }
      }
      // 5. one row per thread (LPR == 1, exact CSR order) or per group of LPR lanes
      if (LPR == 1)
      {
#pragma unroll
         for (int j = 0; j < PF; ++j)
         {
            int r = cur.r0 + tid + j * ST;
            if (r < cur.r1)
            {
               double yn = store_out<MODE>(a, r, row_compute<MODE>(a, ro[j], vs, cs), ro[j].d, ro[j].xo);
               if (DOT) dacc += ro[j].dv * yn;
            }
         }
         for (int r = cur.r0 + tid + PF * ST; r < cur.r1; r += ST)
         {
            RowOps o;
            row_load<MODE, DOT>(a, r, ka, o);
            double yn = store_out<MODE>(a, r, row_compute<MODE>(a, o, vs, cs), o.d, o.xo);
            if (DOT) dacc += o.dv * yn;
         }
      }
      else
      {
         const int sub = tid % LPR, rl = tid / LPR;
#pragma unroll
         for (int j = 0; j < PF; ++j)
         {
            int    r = cur.r0 + rl + j * RPB;
            bool   valid = r < cur.r1;
            double part = valid ? row_partial<LPR>(a, ro[j].s + sub, ro[j].e, vs, cs) : 0.0;
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, o));
            if (valid && sub == 0)
            {
               double yn = store_out<MODE>(a, r, row_finish<MODE>(a, ro[j], part), ro[j].d, ro[j].xo);
               if (DOT) dacc += ro[j].dv * yn;
            }
         }
         for (int base = cur.r0 + PF * RPB; base < cur.r1; base += RPB) // uniform trip count
         {
            int    r = base + rl;
            bool   valid = r < cur.r1;
            RowOps o;
            o.s = o.e = 0;
            if (valid) row_load<MODE, DOT>(a, r, ka, o);
            double part = valid ? row_partial<LPR>(a, o.s + sub, o.e, vs, cs) : 0.0;
#pragma unroll
            for (int w = LPR / 2; w > 0; w >>= 1) part = __dadd_rn(part, __shfl_xor_sync(0xffffffffu, part, w));
            if (valid && sub == 0)
            {
               double yn = store_out<MODE>(a, r, row_finish<MODE>(a, o, part), o.d, o.xo);
               if (DOT) dacc += o.dv * yn;
            }
         }
      }
      __syncthreads(); // stage may be overwritten by the copies issued in the next iteration
      b = nb; nb = nnb; cur = nxt; nxt = nn; stage ^= 1;
   }
   if (DOT)
   {
      double bs = block_sum<ST>(dacc, red);
      __syncthreads();
      grid_finish<ST>(bs, a.partials, a.ticket, a.fin, a.fin_out, a.scal, red, &flag);
   }
}

// ---------------------------------------------------------------------------------------
// Sliced-ELL kernel for the irregular operators of the hierarchy (coarse A, P, R).
// Slices of 32 consecutive rows are stored column-major (entry k of the 32 rows is one
// contiguous 256-byte / 128-byte segment), rows ordered by decreasing length inside the slice
// so that the active lanes of every column load are a prefix.  One warp owns a slice, one lane
// a row: val / col loads are perfectly coalesced streaming loads straight from HBM (no
// shared-memory staging, no bank conflicts), the x gathers of a warp instruction touch the
// same stencil position of 32 neighbouring rows, and every row is accumulated sequentially in
// its stored order with separately rounded multiply and add.
// ---------------------------------------------------------------------------------------
constexpr int SELL_T = 256;
constexpr int SELL_OFFD_BIT = 32; // sl_meta = len << 6 | row has off-rank entries << 5 | row offset in the slice

template <int MODE>
__device__ __forceinline__ double row_epilogue(const SpmvDev &a, const RowOps &o, double acc)
{
   if (MODE >= SPMV_CHEB_START) return cheb_epilogue<MODE>(a, o, acc);
   if (MODE == SPMV_SET || MODE == SPMV_SET_DIV || MODE == SPMV_ADD || MODE == SPMV_RESIDUAL || MODE == SPMV_GS_STEP) return acc;
   if (MODE == SPMV_AXPBY)
      return (a.beta == 0.0) ? __dmul_rn(a.alpha, acc) : __dadd_rn(__dmul_rn(a.alpha, acc), __dmul_rn(a.beta, o.yo));
   if (MODE == SPMV_JACOBI)
      return (o.d != 0.0) ? __dadd_rn(o.xo, __ddiv_rn(__dmul_rn(a.w, acc), o.d)) : o.xo;
   return (o.d != 0.0) ? __ddiv_rn(__dmul_rn(a.w, acc), o.d) : 0.0;
}

// x gathers of the sliced-ELL kernel.  HDK_XHINT builds tag them with an L2 evict_last policy (the
// val / col stream is evict_first already): on the big coarse levels the gathered vector is re-read
// from HBM ~10x because the 1.8 GB operator stream pushes it out of L2 between its first and last use.
#ifdef HDK_XHINT
__device__ __forceinline__ uint64_t x_policy()
{
   uint64_t pol;
   asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
   return pol;
}
__device__ __forceinline__ double ld_x(const double *p, uint64_t pol)
{
   double v;
   asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
   return v;
}
#define LDX(p) ld_x((p), xpol)
#else
#define LDX(p) __ldg(p)
#endif
// EXP: the halo export of the next product is folded into this kernel (multi-rank variants only)
template <int MODE, bool DOT, bool OFFD, bool EXP>
__device__ __forceinline__ void sell_body(const SpmvDev &a)
{
#ifdef HDK_XHINT
   const uint64_t xpol = x_policy();
#endif
   constexpr bool SUB  = (MODE == SPMV_RESIDUAL || MODE == SPMV_JACOBI || MODE == SPMV_JACOBI_R || MODE == SPMV_JACOBI2 ||
                          MODE == SPMV_CHEB_START || MODE == SPMV_CHEB_ONE);
   constexpr bool DIAG = (MODE == SPMV_JACOBI || MODE == SPMV_JACOBI_R || MODE == SPMV_SET_DIV || MODE == SPMV_JACOBI2 || MODE == SPMV_GS_STEP);
   constexpr bool XOLD = (MODE == SPMV_JACOBI || MODE == SPMV_JACOBI2);
   __shared__ double red[SELL_T / 32];
   __shared__ int    flag;
   const int lane = threadIdx.x & 31;
   const int wpb  = SELL_T / 32;
   // fused dot: the per-thread partial lives in shared memory, not in a register pair that would be
   // live across the streaming loop (the loop's register budget decides the occupancy)
   __shared__ double s_dot[DOT ? SELL_T : 1];
   if (DOT) s_dot[threadIdx.x] = 0.0;
   int nexp = 0; // send-list entries this lane stored (EXP variants)
   for (int s = blockIdx.x * wpb + (threadIdx.x >> 5); s < a.nslice; s += gridDim.x * wpb)
   {
      const int  meta  = __ldg(a.sl_meta + (size_t)s * 32 + lane);
      const int  len   = meta >> 6;
      const int  r     = s * 32 + (meta & 31);
      const bool valid = r < a.nrows;
      const size_t base = (size_t)__ldg(a.sl_off + s) * 32 + lane;
      RowOps o;
      o.b = o.d = o.xo = o.yo = o.dv = 0.0;
      // (which operands are fetched before and which after the streaming loop is chosen by the
      // register count ptxas ends up with: 32 = 8 CTAs per SM, 33-40 = 6, 41-48 = 5)
      constexpr bool LATE = DOT; // fused-dot variants: smoother operands after the loop as well
      // Chebyshev: the residual passes (START, ONE) fetch like the Jacobi modes, the others after the loop
      constexpr bool CHEB_EARLY = MODE >= SPMV_CHEB_START && SUB && !LATE;
      if (valid)
      {
         if (CHEB_EARLY) cheb_load<MODE>(a, r, o);
         if (SUB) o.b = a.b[r];
         if (!LATE && DIAG) o.d = a.d[r];
         if (!LATE && XOLD) o.xo = a.x[r];
         if (MODE == SPMV_AXPBY) o.yo = a.y[r];
      }
      double        acc = SUB ? o.b : 0.0;
      const int    *cp  = a.sl_col + base;
      const double *vp  = a.sl_val + base;
      // software pipeline: the val / col loads of group k+1 are in flight while the gathers of
      // group k complete, so every lane keeps 8 streaming loads + 4 gathers outstanding
      int    c0 = 0, c1 = 0, c2 = 0, c3 = 0;
      double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
      if (0 < len) { c0 = __ldcs(cp); v0 = __ldcs(vp); }
      if (1 < len) { c1 = __ldcs(cp + 32); v1 = __ldcs(vp + 32); }
      if (2 < len) { c2 = __ldcs(cp + 64); v2 = __ldcs(vp + 64); }
      if (3 < len) { c3 = __ldcs(cp + 96); v3 = __ldcs(vp + 96); }
#pragma unroll 1 // unrolled copies of this software-pipelined body double the register count (occupancy)
      for (int k = 0; k < len; k += 4)
      {
         const double x0 = LDX(a.x + c0), x1 = LDX(a.x + c1), x2 = LDX(a.x + c2), x3 = LDX(a.x + c3);
         const size_t q  = (size_t)(k + 4) * 32;
         int          n0 = 0, n1 = 0, n2 = 0, n3 = 0;
         double       w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
         if (k + 4 < len) { n0 = __ldcs(cp + q); w0 = __ldcs(vp + q); }
         if (k + 5 < len) { n1 = __ldcs(cp + q + 32); w1 = __ldcs(vp + q + 32); }
         if (k + 6 < len) { n2 = __ldcs(cp + q + 64); w2 = __ldcs(vp + q + 64); }
         if (k + 7 < len) { n3 = __ldcs(cp + q + 96); w3 = __ldcs(vp + q + 96); }
         const double p0 = __dmul_rn(v0, x0), p1 = __dmul_rn(v1, x1), p2 = __dmul_rn(v2, x2), p3 = __dmul_rn(v3, x3);
         acc = __dadd_rn(acc, SUB ? -p0 : p0);
         if (k + 1 < len) acc = __dadd_rn(acc, SUB ? -p1 : p1);
         if (k + 2 < len) acc = __dadd_rn(acc, SUB ? -p2 : p2);
         if (k + 3 < len) acc = __dadd_rn(acc, SUB ? -p3 : p3);
         c0 = n0; c1 = n1; c2 = n2; c3 = n3;
         v0 = w0; v1 = w1; v2 = w2; v3 = w3;
      }
      if (OFFD && (meta & SELL_OFFD_BIT))
      {
         // row with off-rank entries: continue the row's sum in stored order with the halo values.  The
         // exchange is complete before this kernel starts (the pack / exporting kernel of this rank ends
         // with the wait for the neighbours' flags) and buffer reuse is ordered by the next exchange, so
         // this kernel has no system-scope synchronisation at all.
         for (int k = __ldg(a.orp + r), e = __ldg(a.orp + r + 1); k < e; ++k)
         {
            const double p0 = __dmul_rn(__ldg(a.oval + k), __ldcg(a.xh + __ldg(a.ocol + k)));
            acc = __dadd_rn(acc, SUB ? -p0 : p0);
         }
      }
      if (valid)
      {
         if (LATE && DIAG) o.d = a.d[r];
         if (LATE && XOLD) o.xo = a.x[r];
         if (MODE >= SPMV_CHEB_START && !CHEB_EARLY) cheb_load<MODE>(a, r, o);
         if (DOT) o.dv = a.dotv[r];
         // y += A x: y is read only now (live across the loop it costs 10 registers = 3 CTAs per SM),
         // so the sum is y + (a_0 x_0 + a_1 x_1 + ...) -- rounding-level difference to the CSR-order sum
         if (MODE == SPMV_ADD) acc = __dadd_rn(a.y[r], acc);
         double yn = store_out<MODE, EXP>(a, r, row_epilogue<MODE>(a, o, acc), o.d, o.xo, nexp);
         if (DOT) s_dot[threadIdx.x] += o.dv * yn;
      }
   }
   if (EXP) export_finish(a.exp, nexp);
   if (DOT)
   {
      double bs = block_sum<SELL_T>(s_dot[threadIdx.x], red);
      __syncthreads();
      grid_finish<SELL_T>(bs, a.partials, a.ticket, a.fin, a.fin_out, a.scal, red, &flag);
   }
}

// Kernel entry point.  The kernel lives on memory-level parallelism across warps, so occupancy
// matters: 32 registers (8 CTAs per SM) for the plain variants, 40-48 with a fused dot, 48-64 with
// the fused off-diagonal block.
template <int MODE, bool DOT, bool OFFD, bool EXP>
__global__ void __launch_bounds__(SELL_T) k_spmv_sell(SpmvDev a) { sell_body<MODE, DOT, OFFD, EXP>(a); }

// slice metadata: lanes ranked by decreasing row length (ties by row), slice width = longest row
__global__ void k_sell_meta(const int *rowptr, int nrows, int nslice, int *meta, int *width, int *max_slice_nnz,
                            const int *offd_rowptr)
{
   const int lane = threadIdx.x & 31;
   const int s    = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
   if (s >= nslice) return;
   const int r   = s * 32 + lane;
   const int len = (r < nrows) ? rowptr[r + 1] - rowptr[r] : 0;
   const int key = (r < nrows) ? len : -1;
   int       rank = 0, w = 0;
   for (int j = 0; j < 32; ++j)
   {
      int kj = __shfl_sync(0xffffffffu, key, j);
      rank += (kj > key) || (kj == key && j < lane);
      w = kj > w ? kj : w;
   }
   const int ob = (offd_rowptr && r < nrows && offd_rowptr[r + 1] > offd_rowptr[r]) ? SELL_OFFD_BIT : 0;
   meta[(size_t)s * 32 + rank] = (len << 6) | lane | ob;
   if (lane == 0)
   {
      width[s] = w;
      int hi   = s * 32 + 32;
      if (hi > nrows) hi = nrows;
      atomicMax(max_slice_nnz, rowptr[hi] - rowptr[s * 32]);
   }
}

// copy CSR rows into the slices through shared memory (coalesced on both sides); with `sort`
// the entries of a row after a leading diagonal are ordered by column, which lines up the
// gathers of neighbouring rows
template <bool SORT>
__global__ void k_sell_fill(const int *rowptr, const int *col, const double *val, int nrows, int nslice, const int *sl_off,
                            const int *meta, int *scol, double *sval, int cap)
{
   extern __shared__ __align__(16) unsigned char sm_raw[];
   const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
   double   *vs = reinterpret_cast<double *>(sm_raw) + (size_t)w * cap;
   int      *cs = reinterpret_cast<int *>(sm_raw + (size_t)nw * cap * sizeof(double)) + (size_t)w * cap;
   const int s  = blockIdx.x * nw + w;
   if (s >= nslice) return;
   int hi = s * 32 + 32;
   if (hi > nrows) hi = nrows;
   const int k0 = rowptr[s * 32], k1 = rowptr[hi];
   for (int k = k0 + lane; k < k1; k += 32) { cs[k - k0] = col[k]; vs[k - k0] = val[k]; }
   __syncwarp();
   const int m = meta[(size_t)s * 32 + lane], len = m >> 6, r = s * 32 + (m & 31);
   if (r >= nrows || len == 0) return;
   const int rs = rowptr[r] - k0;
   if (SORT)
   {
      const int b = rs + ((cs[rs] == r) ? 1 : 0), e = rs + len;
      for (int k = b + 1; k < e; ++k)
      {
         int    c = cs[k];
         double v = vs[k];
         int    j = k - 1;
         while (j >= b && cs[j] > c) { cs[j + 1] = cs[j]; vs[j + 1] = vs[j]; --j; }
         cs[j + 1] = c; vs[j + 1] = v;
      }
   }
   const size_t base = (size_t)sl_off[s] * 32 + lane;
   for (int k = 0; k < len; ++k)
   {
      scol[base + (size_t)k * 32] = cs[rs + k];
      sval[base + (size_t)k * 32] = vs[rs + k];
   }
}

template <int MODE, bool DOT, bool OFFD, bool EXP>
static int launch_sell_v(const DevCSR &A, const SpmvDev &d)
{
   static int occ = 0;
   if (!occ)
   {
      HDK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_spmv_sell<MODE, DOT, OFFD, EXP>, SELL_T, 0));
      if (occ < 1) occ = 1;
   }
   int grid = cdiv(A.nslice, SELL_T / 32);
   int cap  = g.sm_count * occ;
   if (grid > cap) grid = cap;
   k_spmv_sell<MODE, DOT, OFFD, EXP><<<grid, SELL_T, 0, g.stream>>>(d);
   return HDK_OK;
}
template <int MODE, bool DOT>
static int launch_sell(const DevCSR &A, const SpmvDev &d)
{
   if (!d.has_halo) return launch_sell_v<MODE, DOT, false, false>(A, d);
   return d.exp.seq ? launch_sell_v<MODE, DOT, true, true>(A, d) : launch_sell_v<MODE, DOT, true, false>(A, d);
}

// one warp per row; lanes stride the row with scalar loads (rows here are long, so each warp
// reads whole 128-byte lines).  Summation order differs from the oracle (tolerance parity).
template <int MODE, bool DOT>
__global__ void __launch_bounds__(ST) k_spmv_vector(SpmvDev a)
{
   __shared__ double red[ST / 32];
   __shared__ int    flag;
   const int lane = threadIdx.x & 31;
   const int wpb  = ST / 32;
   double    dacc = 0.0;
   for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < a.nrows; r += gridDim.x * wpb)
   {
      int    s = a.rowptr[r], e = a.rowptr[r + 1];
      double acc = 0.0;
      for (int k = s + lane; k < e; k += 32) acc += __ldg(a.val + k) * __ldg(a.x + __ldg(a.col + k));
      acc = warp_sum(acc);
      if (lane == 0 && MODE >= SPMV_CHEB_START)
      {
         RowOps o;
         cheb_load<MODE>(a, r, o);
         double yn = cheb_epilogue<MODE>(a, o, (MODE == SPMV_CHEB_START || MODE == SPMV_CHEB_ONE) ? __dadd_rn(o.b, -acc) : acc);
         yn = store_out<MODE>(a, r, yn, o.d, 0.0);
         if (DOT) dacc += a.dotv[r] * yn;
      }
      else if (lane == 0)
      {
         double yn;
         if (MODE == SPMV_SET || MODE == SPMV_SET_DIV || MODE == SPMV_GS_STEP) yn = acc;
         else if (MODE == SPMV_AXPBY) yn = (a.beta == 0.0) ? a.alpha * acc : a.alpha * acc + a.beta * a.y[r];
         else if (MODE == SPMV_ADD) yn = a.y[r] + acc;
         else
         {
            double res = a.b[r] - acc;
            if (MODE == SPMV_RESIDUAL) yn = res;
            else
            {
               double dd = a.d[r];
               if (MODE == SPMV_JACOBI) yn = (dd != 0.0) ? a.x[r] + (a.w * res) / dd : a.x[r];
               else yn = (dd != 0.0) ? (a.w * res) / dd : 0.0;
            }
         }
         constexpr bool NEED_D = (MODE == SPMV_SET_DIV || MODE == SPMV_GS_STEP);
         yn = store_out<MODE>(a, r, yn, NEED_D ? a.d[r] : 0.0, MODE == SPMV_JACOBI2 ? a.x[r] : 0.0);
         if (DOT) dacc += a.dotv[r] * yn;
      }
   }
   if (DOT)
   {
      double bs = block_sum<ST>(dacc, red);
      __syncthreads();
      grid_finish<ST>(bs, a.partials, a.ticket, a.fin, a.fin_out, a.scal, red, &flag);
   }
}

template <int MODE, bool DOT, int LPR>
static int launch_tma(const DevCSR &A, const SpmvDev &d)
{
   static bool                  attr_set = false;
   static std::map<size_t, int> occ_cache; // per template instantiation: smem bytes -> CTAs/SM
   size_t                       smem = 128 + (size_t)2 * A.cap * 12;
   if (!attr_set)
   {
      HDK_CUDA(cudaFuncSetAttribute(k_spmv_tma<MODE, DOT, LPR>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
      attr_set = true;
   }
   auto it = occ_cache.find(smem);
   if (it == occ_cache.end())
   {
      int occ = 0;
      HDK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_spmv_tma<MODE, DOT, LPR>, ST, smem));
      if (occ < 1) occ = 1;
      it = occ_cache.emplace(smem, occ).first;
   }
   int grid = g.sm_count * it->second;
   if (grid > A.nblk) grid = A.nblk;
   k_spmv_tma<MODE, DOT, LPR><<<grid, ST, smem, g.stream>>>(d, A.nblk, A.cap);
   return HDK_OK;
}

template <int MODE>
static int launch_mode(const DevCSR &A, const SpmvDev &d, bool dot)
{
   if (A.kind == 0)
   {
      switch (A.lpr)
      {
         case 2: if (dot) HDK_TRY((launch_tma<MODE, true, 2>(A, d))); else HDK_TRY((launch_tma<MODE, false, 2>(A, d))); break;
         case 4: if (dot) HDK_TRY((launch_tma<MODE, true, 4>(A, d))); else HDK_TRY((launch_tma<MODE, false, 4>(A, d))); break;
         case 8: if (dot) HDK_TRY((launch_tma<MODE, true, 8>(A, d))); else HDK_TRY((launch_tma<MODE, false, 8>(A, d))); break;
         default: if (dot) HDK_TRY((launch_tma<MODE, true, 1>(A, d))); else HDK_TRY((launch_tma<MODE, false, 1>(A, d))); break;
      }
   }
   else if (A.kind == 2)
   {
      if (dot) HDK_TRY((launch_sell<MODE, true>(A, d))); else HDK_TRY((launch_sell<MODE, false>(A, d)));
   }
   else
   {
      int grid = cdiv(A.nrows, ST / 32);
      int cap  = g.sm_count * 16;
      if (grid > cap) grid = cap;
      if (grid < 1) grid = 1;
      if (dot) k_spmv_vector<MODE, true><<<grid, ST, 0, g.stream>>>(d);
      else k_spmv_vector<MODE, false><<<grid, ST, 0, g.stream>>>(d);
   }
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}

int spmv_launch(const DevCSR &A, int mode, const SpmvArgs &s, const OffdFuse *of)
{
   if (A.nrows <= 0) return HDK_OK;
   SpmvDev d;
   d.rowptr = A.rowptr; d.col = A.col; d.val = A.val; d.blk_row = A.blk_row;
   d.x = s.x; d.b = s.b; d.d = s.d; d.dotv = s.dotv; d.y = s.y; d.y2 = s.y2;
   d.w = s.w; d.alpha = s.alpha; d.beta = s.beta;
   d.nrows = A.nrows; d.fin = s.fin; d.fin_out = s.fin_out;
   d.scal = g.dscal; d.partials = g.partials; d.ticket = g.counters;
   d.sl_off = A.sl_off; d.sl_meta = A.sl_meta; d.sl_col = A.sl_col; d.sl_val = A.sl_val; d.nslice = A.nslice;
   d.orp = nullptr; d.ocol = nullptr; d.oval = nullptr; d.xh = nullptr; d.has_halo = 0;
   if (of)
   {
      if (A.kind != 2 || !A.sl_offd_flags) return set_error(HDK_ERR_INVALID, "fused off-rank block needs the sliced-ELL layout with flagged rows");
      d.orp = of->orp; d.ocol = of->ocol; d.oval = of->oval; d.xh = of->xh;
      d.has_halo = 1;
   }
   d.exp = HaloExport();
   d.exp_y2 = s.export_y2 ? 1 : 0;
   d.uo = s.uo;
   // Folding the export into this kernel saves the consumer's pack kernel (~13 us).  The exporting variants
   // compile to the same register budget as the non-exporting multi-rank ones (32 for SET / RESIDUAL /
   // ADD, 40 for the rest -- guarded by tests/test_abi_and_host.py), so every product folds; the tunable
   // export_max_rows makes operators above a size pack instead (experiments).
   if (s.export_to && of && (double)A.nrows <= tunables().export_max_rows) halo_export_begin(*s.export_to, &d.exp);
   bool dot = (s.fin != FIN_NONE && s.dotv != nullptr);
   switch (mode)
   {
      case SPMV_SET: return launch_mode<SPMV_SET>(A, d, dot);
      case SPMV_RESIDUAL: return launch_mode<SPMV_RESIDUAL>(A, d, dot);
      case SPMV_JACOBI: return launch_mode<SPMV_JACOBI>(A, d, dot);
      case SPMV_ADD: return launch_mode<SPMV_ADD>(A, d, dot);
      case SPMV_AXPBY: return launch_mode<SPMV_AXPBY>(A, d, dot);
      case SPMV_JACOBI_R: return launch_mode<SPMV_JACOBI_R>(A, d, dot);
      case SPMV_SET_DIV: return launch_mode<SPMV_SET_DIV>(A, d, dot);
      case SPMV_JACOBI2: return launch_mode<SPMV_JACOBI2>(A, d, dot);
      case SPMV_GS_STEP: return launch_mode<SPMV_GS_STEP>(A, d, dot);
      case SPMV_CHEB_START: return launch_mode<SPMV_CHEB_START>(A, d, dot);
      case SPMV_CHEB_STEP: return launch_mode<SPMV_CHEB_STEP>(A, d, dot);
      case SPMV_CHEB_FIN: return launch_mode<SPMV_CHEB_FIN>(A, d, dot);
      case SPMV_CHEB_ONE: return launch_mode<SPMV_CHEB_ONE>(A, d, dot);
   }
   return set_error(HDK_ERR_INVALID, "unknown spmv mode %d", mode);
}

// Chebyshev epilogue on a finished row result (levels whose off-rank part is added by a correction
// kernel, and the zero-guess start where f - A 0 = f): the expressions of the fused kernels
template <int MODE>
__global__ void __launch_bounds__(ST) k_cheb_epi(SpmvDev a, const double *__restrict__ acc)
{
   for (int r = blockIdx.x * ST + threadIdx.x; r < a.nrows; r += gridDim.x * ST)
   {
      RowOps o;
      o.yo = 0.0;
      cheb_load<MODE>(a, r, o);
      store_out<MODE>(a, r, cheb_epilogue<MODE>(a, o, acc[r]), o.d, 0.0);
   }
}

int cheb_epilogue_pass(int mode, int n, const double *acc, const SpmvArgs &s)
{
   if (n <= 0) return HDK_OK;
   SpmvDev d;
   memset(&d, 0, sizeof(d));
   d.b = s.b; d.d = s.d; d.y = s.y; d.y2 = s.y2; d.alpha = s.alpha; d.uo = s.uo; d.nrows = n;
   int grid = cdiv(n, ST);
   if (grid > g.sm_count * 8) grid = g.sm_count * 8;
   switch (mode)
   {
      case SPMV_CHEB_START: k_cheb_epi<SPMV_CHEB_START><<<grid, ST, 0, g.stream>>>(d, acc); break;
      case SPMV_CHEB_STEP: k_cheb_epi<SPMV_CHEB_STEP><<<grid, ST, 0, g.stream>>>(d, acc); break;
      case SPMV_CHEB_FIN: k_cheb_epi<SPMV_CHEB_FIN><<<grid, ST, 0, g.stream>>>(d, acc); break;
      case SPMV_CHEB_ONE: k_cheb_epi<SPMV_CHEB_ONE><<<grid, ST, 0, g.stream>>>(d, acc); break;
      default: return set_error(HDK_ERR_INVALID, "unknown Chebyshev epilogue %d", mode);
   }
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}

// ---------------------------------------------------------------------------------------
// analysis: row-length statistics and the nnz-balanced row blocks of the stream kernel
// ---------------------------------------------------------------------------------------
__global__ void k_row_stats(const int *rowptr, int nrows, int *max_row)
{
   int m = 0;
   for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += gridDim.x * blockDim.x)
   {
      int l = rowptr[r + 1] - rowptr[r];
      m     = l > m ? l : m;
   }
   for (int o = 16; o > 0; o >>= 1) { int t = __shfl_down_sync(0xffffffffu, m, o); m = t > m ? t : m; }
   if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(max_row, m);
}

__global__ void k_blk_rows(const int *rowptr, int nrows, int nblk, int tgt, int *blk_row)
{
   int b = blockIdx.x * blockDim.x + threadIdx.x;
   if (b > nblk) return;
   if (b == nblk) { blk_row[b] = nrows; return; }
   int target = b * tgt;
   int lo = 0, hi = nrows; // first i in [0,nrows] with rowptr[i] >= target
   while (lo < hi)
   {
      int mid = (lo + hi) >> 1;
      if (rowptr[mid] >= target) hi = mid; else lo = mid + 1;
   }
   blk_row[b] = lo;
}

static void sell_free(DevCSR &A)
{
   dfree(A.sl_off); dfree(A.sl_meta); dfree(A.sl_col); dfree(A.sl_val);
   A.sl_off = A.sl_meta = A.sl_col = nullptr; A.sl_val = nullptr; A.nslice = 0;
}

// build the sliced-ELL copy; leaves A.kind untouched (and no copy) when the layout does not pay:
// too much padding or slices that do not fit the staging buffer of the fill kernel
static int sell_build(DevCSR &A)
{
   const bool sort = tunables().sell_sort != 0.0 && A.coarse_op;
   const int ns = cdiv(A.nrows, 32);
   int      *width = nullptr, *dmax = reinterpret_cast<int *>(g.dscal + S_TMP3);
   HDK_TRY(dalloc(&A.sl_meta, (size_t)ns * 32));
   HDK_TRY(dalloc(&A.sl_off, (size_t)ns + 1));
   HDK_TRY(dalloc(&width, (size_t)ns + 1));
   HDK_CUDA(cudaMemsetAsync(width + ns, 0, sizeof(int), g.stream));
   HDK_CUDA(cudaMemsetAsync(dmax, 0, sizeof(int), g.stream));
   // N > 1: rows with off-rank entries are flagged, the multi-rank kernel variants add those entries
   // (HDK_FUSE_OFFD=0: no flags, a second kernel adds them)
   static int fuse_on = -1;
   if (fuse_on < 0) { const char *e = getenv("HDK_FUSE_OFFD"); fuse_on = (e && atoi(e) == 0) ? 0 : 1; }
   const int *orp = fuse_on ? A.offd_rowptr : nullptr;
   k_sell_meta<<<cdiv(ns, 8), 256, 0, g.stream>>>(A.rowptr, A.nrows, ns, A.sl_meta, width, dmax, orp);
   A.sl_offd_flags = (orp != nullptr);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_int(width, A.sl_off, ns + 1));
   int h[2] = {0, 0};
   HDK_CUDA(cudaMemcpyAsync(&h[0], A.sl_off + ns, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaMemcpyAsync(&h[1], dmax, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   dfree(width);
   const int64_t padded = (int64_t)h[0] * 32;
   const int     cap    = (h[1] + 3) & ~3;
   int           nw     = 4;
   while (nw > 1 && (size_t)nw * cap * 12 > 200 * 1024) nw >>= 1;
   if (padded > 3 * (int64_t)A.nnz + 4096 || (size_t)nw * cap * 12 > 200 * 1024) { sell_free(A); return HDK_OK; }
   HDK_TRY(dalloc(&A.sl_col, (size_t)padded + 32));
   HDK_TRY(dalloc(&A.sl_val, (size_t)padded + 32));
   const size_t smem = (size_t)nw * cap * 12;
   const bool   do_sort = sort && A.nrows == A.ncols;
   if (do_sort)
   {
      HDK_CUDA(cudaFuncSetAttribute(k_sell_fill<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      k_sell_fill<true><<<cdiv(ns, nw), nw * 32, smem, g.stream>>>(A.rowptr, A.col, A.val, A.nrows, ns, A.sl_off, A.sl_meta,
                                                                    A.sl_col, A.sl_val, cap);
   }
   else
   {
      HDK_CUDA(cudaFuncSetAttribute(k_sell_fill<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      k_sell_fill<false><<<cdiv(ns, nw), nw * 32, smem, g.stream>>>(A.rowptr, A.col, A.val, A.nrows, ns, A.sl_off, A.sl_meta,
                                                                     A.sl_col, A.sl_val, cap);
   }
   HDK_LAUNCH_CHECK();
   A.nslice = ns;
   A.kind   = 2;
   return HDK_OK;
}

int csr_analyze(DevCSR &A)
{
   if (A.blk_row) { dfree(A.blk_row); A.blk_row = nullptr; }
   sell_free(A);
   A.nblk = 0; A.kind = 0; A.max_row = 0; A.avg_row = 0.0;
   if (A.nrows <= 0) return HDK_OK;
   int *dmax = reinterpret_cast<int *>(g.dscal + S_TMP3);
   HDK_CUDA(cudaMemsetAsync(dmax, 0, sizeof(int), g.stream));
   int grid = cdiv(A.nrows, 256);
   if (grid > g.sm_count * 8) grid = g.sm_count * 8;
   k_row_stats<<<grid, 256, 0, g.stream>>>(A.rowptr, A.nrows, dmax);
   HDK_LAUNCH_CHECK();
   int hmax = 0;
   HDK_CUDA(cudaMemcpyAsync(&hmax, dmax, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   A.max_row = hmax;
   A.avg_row = (double)A.nnz / (double)A.nrows;
   A.kind    = (hmax <= S_MAXR) ? 0 : 1;
   if (A.kind == 0 && A.val)
   {
      // large operators go to the sliced-ELL kernel; small ones are latency-bound and do better
      // with several lanes per row in the stream kernel
      const Tune &t = tunables();
      const double min_rows = A.offd_rowptr ? t.sell_min_rows_dist : t.sell_min_rows;
      if ((double)A.nrows >= min_rows && A.avg_row > t.sell_min_avg) HDK_TRY(sell_build(A));
   }
   if (A.kind == 0)
   {
      // non-zeros per block: about one row per thread (`mult` x 256 rows), 64-aligned
      const Tune &t = tunables();
      double mult = t.rows_mult > 0 ? t.rows_mult : 1.0;
      int    thi  = (int)t.tgt_max;
      if (thi < S_TGT_LO) thi = S_TGT_LO;
      if (thi > S_TGT_HI) thi = S_TGT_HI;
      // lanes per row from the average row length (1 keeps the exact sequential CSR order)
      const int lpr_force = (int)t.lpr;
      int lpr = A.avg_row <= 12.0 ? 1 : (A.avg_row <= 24.0 ? 2 : (A.avg_row <= 56.0 ? 4 : 8));
      if (lpr_force == 1 || lpr_force == 2 || lpr_force == 4 || lpr_force == 8) lpr = lpr_force;
      A.lpr   = lpr;
      int tgt = ((int)(A.avg_row * (256.0 / lpr) * mult) / 64) * 64;
      if (tgt < S_TGT_LO) tgt = S_TGT_LO;
      if (tgt > thi) tgt = thi;
      A.tgt  = tgt;
      A.cap  = (tgt + hmax + 8 + 3) & ~3; // shared-memory entries per stage
      A.nblk = A.nnz / tgt + 1;
      if (A.nblk > PARTIALS_CAP) return set_error(HDK_ERR_UNSUPPORTED, "matrix too large for the reduction scratch");
      HDK_TRY(dalloc(&A.blk_row, (size_t)A.nblk + 1));
      k_blk_rows<<<cdiv(A.nblk + 1, 256), 256, 0, g.stream>>>(A.rowptr, A.nrows, A.nblk, tgt, A.blk_row);
      HDK_LAUNCH_CHECK();
   }
   return HDK_OK;
}

int csr_alloc(DevCSR &A, int nrows, int ncols, int nnz, bool values)
{
   A.nrows = nrows; A.ncols = ncols; A.nnz = nnz; A.owns = true;
   HDK_TRY(dalloc(&A.rowptr, (size_t)nrows + 1));
   HDK_TRY(dalloc(&A.col, (size_t)nnz + 8));
   HDK_CUDA(cudaMemsetAsync(A.col + nnz, 0, sizeof(int) * 8, g.stream));
   if (values)
   {
      HDK_TRY(dalloc(&A.val, (size_t)nnz + 8));
      HDK_CUDA(cudaMemsetAsync(A.val + nnz, 0, sizeof(double) * 8, g.stream));
   }
   else A.val = nullptr;
   return HDK_OK;
}

void csr_free(DevCSR &A)
{
   if (A.owns) { dfree(A.rowptr); dfree(A.col); dfree(A.val); }
   dfree(A.blk_row);
   sell_free(A);
   A = DevCSR();
}

// wait budget / error flag of this translation unit's copy of the flag-wait globals
int wait_globals_spmv(long long tmo, int *err)
{
   return wait_globals_set(tmo, err) == cudaSuccess ? HDK_OK : set_error(HDK_ERR_CUDA, "cannot set the wait budget");
}

} // namespace hdk
