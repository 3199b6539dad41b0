// hdk_amg_setup.cu -- BoomerAMG setup on the device (north-star item 4):
// strength of connection, PMIS coarsening, extended+i interpolation with truncation,
// R = P^T, Galerkin RAP with hash accumulators, l1 norms, dense coarsest inverse.
// Stands in for HYPRE_BoomerAMGSetup (reference trigger src/internal/solver.c:296,
// src/internal/precon.c:107; options src/internal/amg.c:863-1035).
//
// Parity contract: integer results (S, C/F splitting, sparsity of P and of every coarse
// operator, including the storage order inside rows) are bit-identical to the CPU oracle
// (oracle/amg_setup.c), and so are the floating-point values, because every row is
// accumulated by one thread in the oracle's order with separately rounded multiply/add.
#include "hdk_amg.cuh"
#include <algorithm>
#include <math.h>
#include <stdlib.h>
#include <time.h>

namespace hdk {

#define C_PT 1
#define F_PT -1
#define SF_PT -3

// HDK_SETUP_TIMING=1: synchronise and print the wall time of every setup stage
static double g_t_last = 0.0;
static bool   g_timing = false;
static double wall_now()
{
   struct timespec ts;
   clock_gettime(CLOCK_MONOTONIC, &ts);
   return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
static void stage_mark(const char *name, int level)
{
   if (!g_timing) return;
   cudaStreamSynchronize(g.stream);
   double t = wall_now();
   if (name) fprintf(stderr, "[hdk setup] level %d %-12s %8.3f ms\n", level, name, 1e3 * (t - g_t_last));
   g_t_last = t;
}

void setup_stage_mark(const char *name, int level) { stage_mark(name, level); }

static const int64_t SCRATCH_BUDGET = (int64_t)1 << 30; // hash slots per chunk (4-8 GB)

// ---- work sharing of the replicated multi-rank setup --------------------------------------
// While the global hierarchy is built on every rank (setup_distributed), the row-parallel
// stages (interpolation, Galerkin product) compute only this rank's share of the rows of the
// GLOBAL matrices and the ranks exchange their row segments (grouped NCCL broadcasts), so the
// result on every rank is the same bit-identical global level at 1/nranks of the work.
static bool g_share = false;
static int  g_share_min_rows = 65536; // smaller levels: the exchange latency exceeds the saving
static bool share_on(int n) { return g_share && g.nranks > 1 && n >= g_share_min_rows; }
static void share_range(int n, int &lo, int &hi)
{
   lo = 0; hi = n;
   if (!share_on(n)) return;
   lo = (int)((int64_t)n * g.rank / g.nranks);
   hi = (int)((int64_t)n * (g.rank + 1) / g.nranks);
}
// exchange a per-row array (elem bytes per row) computed for the shares of [0,n)
static int share_rows(void *base, size_t elem, int n)
{
   if (!share_on(n)) return HDK_OK;
   std::vector<int64_t> offs((size_t)g.nranks + 1);
   for (int r = 0; r <= g.nranks; r++) offs[(size_t)r] = (int64_t)((int64_t)n * r / g.nranks) * (int64_t)elem;
   return allgatherv_bytes(base, offs.data());
}
// exchange per-entry arrays of a CSR whose rows were computed by shares; rowptr is complete
static int share_entries(const int *rowptr_d, int n, void *a, size_t ea, void *b, size_t eb)
{
   if (!share_on(n)) return HDK_OK;
   std::vector<int>     bnd((size_t)g.nranks + 1);
   std::vector<int64_t> offs((size_t)g.nranks + 1);
   for (int r = 0; r <= g.nranks; r++)
      HDK_CUDA(cudaMemcpyAsync(&bnd[(size_t)r], rowptr_d + (int64_t)n * r / g.nranks, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   if (a) { for (int r = 0; r <= g.nranks; r++) offs[(size_t)r] = (int64_t)bnd[(size_t)r] * (int64_t)ea; HDK_TRY(allgatherv_bytes(a, offs.data())); }
   if (b) { for (int r = 0; r <= g.nranks; r++) offs[(size_t)r] = (int64_t)bnd[(size_t)r] * (int64_t)eb; HDK_TRY(allgatherv_bytes(b, offs.data())); }
   return HDK_OK;
}

// =====================================================================================
// small utilities
// =====================================================================================
// sum of n non-negative ints in 64 bits: the row counts of a product must fit the int32 row
// pointers before they are scanned (a 640^3 7-point problem overflows at level 1)
__global__ void k_sum_i64(const int *v, int n, unsigned long long *out)
{
   unsigned long long s = 0;
   for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += (unsigned long long)(v[i] > 0 ? v[i] : 0);
   for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
   if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}
static int check_fits_int32(const int *cnt, int n, const char *what)
{
   unsigned long long *d = reinterpret_cast<unsigned long long *>(g.dscal + S_TMP2), h = 0;
   HDK_CUDA(cudaMemsetAsync(d, 0, sizeof(unsigned long long), g.stream));
   int grid = cdiv(n, 256);
   if (grid > g.sm_count * 8) grid = g.sm_count * 8;
   if (grid < 1) grid = 1;
   k_sum_i64<<<grid, 256, 0, g.stream>>>(cnt, n, d);
   HDK_LAUNCH_CHECK();
   HDK_CUDA(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   if (h > 2000000000ULL)
      return set_error(HDK_ERR_UNSUPPORTED, "%s would have %llu non-zeros: more than the int32 row pointers of this setup hold", what, h);
   return HDK_OK;
}

__global__ void k_chunk_bounds(const int64_t *off, int n, int64_t budget, int nchunks, int *bounds)
{
   int c = blockIdx.x * blockDim.x + threadIdx.x;
   if (c > nchunks) return;
   if (c == nchunks) { bounds[c] = n; return; }
   int64_t target = (int64_t)c * budget;
   int lo = 0, hi = n;
   while (lo < hi) { int mid = (lo + hi) >> 1; if (off[mid] >= target) hi = mid; else lo = mid + 1; }
   bounds[c] = lo;
}

// rows [bounds[c], bounds[c+1]) use at most `maxsz` scratch slots
static int plan_chunks(const int64_t *off_d, int n, std::vector<int> &bounds, int64_t &maxsz)
{
   int64_t total = 0;
   HDK_CUDA(cudaMemcpyAsync(&total, off_d + n, sizeof(int64_t), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   if (total <= SCRATCH_BUDGET) { bounds = {0, n}; maxsz = total; return HDK_OK; }
   int  nch = (int)((total + SCRATCH_BUDGET - 1) / SCRATCH_BUDGET);
   int *bd;
   HDK_TRY(dalloc(&bd, (size_t)nch + 1));
   k_chunk_bounds<<<cdiv(nch + 1, 128), 128, 0, g.stream>>>(off_d, n, SCRATCH_BUDGET, nch, bd);
   HDK_LAUNCH_CHECK();
   bounds.resize((size_t)nch + 1);
   HDK_CUDA(cudaMemcpyAsync(bounds.data(), bd, sizeof(int) * ((size_t)nch + 1), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   dfree(bd);
   bounds.erase(std::unique(bounds.begin(), bounds.end()), bounds.end());
   maxsz = 0;
   for (size_t c = 0; c + 1 < bounds.size(); c++)
   {
      int64_t o[2];
      HDK_CUDA(cudaMemcpyAsync(&o[0], off_d + bounds[c], sizeof(int64_t), cudaMemcpyDeviceToHost, g.stream));
      HDK_CUDA(cudaMemcpyAsync(&o[1], off_d + bounds[c + 1], sizeof(int64_t), cudaMemcpyDeviceToHost, g.stream));
      HDK_CUDA(cudaStreamSynchronize(g.stream));
      if (o[1] - o[0] > maxsz) maxsz = o[1] - o[0];
   }
   return HDK_OK;
}

__device__ __forceinline__ int pow2ceil(int v)
{
   if (v < 4) return 4;
   return 1 << (32 - __clz(v - 1));
}

// open-addressing tables living in global scratch, one per row, keys initialised to -1
__device__ __forceinline__ unsigned hslot(int key, int cap) { return ((unsigned)key * 2654435761u) >> (__clz(cap) + 1); }

__device__ __forceinline__ bool hset_insert(int *keys, int cap, int key)
{
   unsigned h = hslot(key, cap), mask = (unsigned)cap - 1;
   while (true)
   {
      int k = keys[h];
      if (k == key) return false;
      if (k == -1) { keys[h] = key; return true; }
      h = (h + 1) & mask;
   }
}
__device__ __forceinline__ int hmap_find(const int2 *tab, int cap, int key)
{
   unsigned h = hslot(key, cap), mask = (unsigned)cap - 1;
   while (true)
   {
      int2 e = tab[h];
      if (e.x == key) return e.y;
      if (e.x == -1) return -1;
      h = (h + 1) & mask;
   }
}
// returns the stored value if present, else stores `val` and returns -1
__device__ __forceinline__ int hmap_insert(int2 *tab, int cap, int key, int val)
{
   unsigned h = hslot(key, cap), mask = (unsigned)cap - 1;
   while (true)
   {
      int2 e = tab[h];
      if (e.x == key) return e.y;
      if (e.x == -1) { tab[h] = make_int2(key, val); return -1; }
      h = (h + 1) & mask;
   }
}

// shared-memory table shared by the lanes of one warp: concurrent inserts of DISTINCT keys
__device__ __forceinline__ int wt_find_or_insert(int *keys, int cap, int key, bool &isnew)
{
   unsigned h = hslot(key, cap), mask = (unsigned)cap - 1;
   while (true)
   {
      int k = keys[h];
      if (k == key) { isnew = false; return (int)h; }
      if (k == -1)
      {
         int old = atomicCAS(keys + h, -1, key);
         if (old == -1) { isnew = true; return (int)h; }
         if (old == key) { isnew = false; return (int)h; }
      }
      h = (h + 1) & mask;
   }
}

// =====================================================================================
// strength of connection (hypre_BoomerAMGCreateS)
// =====================================================================================
struct RowS { double diag, thr; bool weak_all; };

__device__ __forceinline__ RowS row_strength(const int *rp, const double *val, const int *orp, const double *oval,
                                             int i, double theta, double mrs)
{
   RowS   r;
   int    b = rp[i], e = rp[i + 1];
   double diag = val[b], row_scale = 0.0, row_sum = diag;
   for (int k = b + 1; k < e; k++)
   {
      double v = val[k];
      if (diag < 0) row_scale = row_scale > v ? row_scale : v;
      else row_scale = row_scale < v ? row_scale : v;
      row_sum = __dadd_rn(row_sum, v);
   }
   if (orp)
      for (int k = orp[i]; k < orp[i + 1]; k++)
      {
         double v = oval[k];
         if (diag < 0) row_scale = row_scale > v ? row_scale : v;
         else row_scale = row_scale < v ? row_scale : v;
         row_sum = __dadd_rn(row_sum, v);
      }
   r.diag     = diag;
   r.thr      = __dmul_rn(theta, row_scale);
   r.weak_all = (fabs(row_sum) > __dmul_rn(fabs(diag), mrs)) && (mrs < 1.0);
   return r;
}

template <bool FILL>
__global__ void k_strength(const int *rp, const int *col, const double *val, const int *orp, const double *oval,
                           int n, double theta, double mrs, int *cnt, const int *srp, int *scol)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   if (i == n) { if (!FILL) cnt[n] = 0; return; }
   int b = rp[i], e = rp[i + 1], c = 0;
   int p = FILL ? srp[i] : 0;
   if (e > b)
   {
      RowS r = row_strength(rp, val, orp, oval, i, theta, mrs);
      if (!r.weak_all)
         for (int k = b + 1; k < e; k++)
         {
            double v      = val[k];
            bool   strong = (r.diag < 0) ? !(v <= r.thr) : !(v >= r.thr);
            if (strong) { if (FILL) scol[p++] = col[k]; else c++; }
         }
   }
   if (!FILL) cnt[i] = c;
}

int build_strength_csr(const DevCSR &D, const int *orp, const double *ov, double theta, double mrs, DevCSR &S)
{
   int n = D.nrows;
   int *cnt, *srp;
   HDK_TRY(dalloc(&cnt, (size_t)n + 1));
   HDK_TRY(dalloc(&srp, (size_t)n + 1));
   k_strength<false><<<cdiv(n + 1, 256), 256, 0, g.stream>>>(D.rowptr, D.col, D.val, orp, ov, n, theta, mrs, cnt, nullptr, nullptr);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_int(cnt, srp, n + 1));
   int nnzS = 0;
   HDK_CUDA(cudaMemcpyAsync(&nnzS, srp + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   dfree(cnt);
   S = DevCSR();
   S.nrows = n; S.ncols = n; S.nnz = nnzS; S.rowptr = srp; S.owns = true;
   HDK_TRY(dalloc(&S.col, (size_t)nnzS + 8));
   k_strength<true><<<cdiv(n + 1, 256), 256, 0, g.stream>>>(D.rowptr, D.col, D.val, orp, ov, n, theta, mrs, nullptr, srp, S.col);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}

static int build_strength(const hdk_csr_s &A, double theta, double mrs, DevCSR &S)
{
   const int    *orp = A.offd.nnz > 0 ? A.offd.rowptr : nullptr;
   const double *ov  = A.offd.nnz > 0 ? A.offd.val : nullptr;
   return build_strength_csr(A.diag, orp, ov, theta, mrs, S);
}

// =====================================================================================
// PMIS (hypre_BoomerAMGCoarsenPMIS + hypre_BoomerAMGIndepSet), measures from the
// Park-Miller stream of hypre_Rand() reached by skip-ahead: seed_k = seed0 * 16807^k mod (2^31-1)
// =====================================================================================
__device__ __forceinline__ uint32_t mulmod31(uint32_t a, uint32_t b)
{
   const uint64_t M = 2147483647ull;
   uint64_t p = (uint64_t)a * b;
   uint64_t r = (p & M) + (p >> 31);
   r          = (r & M) + (r >> 31);
   if (r >= M) r -= M;
   return (uint32_t)r;
}

__global__ void k_count_cols(const int *col, int nnz, int *cnt)
{
   int k = blockIdx.x * blockDim.x + threadIdx.x;
   if (k < nnz) atomicAdd(cnt + col[k], 1);
}

__global__ void k_measure(const int *cnt, int n, uint32_t seed0, int64_t goff, double *measure)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   uint64_t e = (uint64_t)(goff + i) + 1; // number of hypre_Rand() calls up to and including row i
   uint32_t base = 16807u, acc = seed0;
   while (e)
   {
      if (e & 1) acc = mulmod31(acc, base);
      base = mulmod31(base, base);
      e >>= 1;
   }
   measure[i] = __dadd_rn((double)cnt[i], __ddiv_rn((double)acc, 2147483647.0));
}

__global__ void k_pmis_init(const int *srp, int n, int *cf, double *measure)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   if (srp[i + 1] == srp[i]) { cf[i] = SF_PT; measure[i] = 0.0; }
   else cf[i] = 0;
}

__global__ void k_pmis_mark(int n, int *cf, const double *measure)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n && cf[i] == 0 && measure[i] > 1.0) cf[i] = 1;
}

__global__ void k_pmis_elim(const int *srp, const int *scol, int n, int *cf, const double *measure, int row0)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   i += row0; // rows [row0, row0 + n)
   double mi = measure[i];
   if (!(mi > 1.0)) return;
   for (int k = srp[i]; k < srp[i + 1]; k++)
   {
      int    j  = scol[k];
      double mj = measure[j];
      if (mj > 1.0)
      {
         if (mi > mj) cf[j] = 0;
         else if (mj > mi) cf[i] = 0;
      }
   }
}

__global__ void k_pmis_set(const int *srp, const int *scol, int n, int *cf, double *measure, int *remaining, int row0)
{
   int  i = blockIdx.x * blockDim.x + threadIdx.x;
   bool undecided = false;
   if (i < n)
   {
      i += row0; // rows [row0, row0 + n)
      double mi = measure[i];
      if (mi > 0.0) // still in the graph
      {
         int c = cf[i];
         if (mi < 1.0) c = F_PT;
         if (c > 0) c = C_PT;
         else
            for (int k = srp[i]; k < srp[i + 1]; k++)
               if (cf[scol[k]] > 0) { c = F_PT; break; }
         cf[i] = c;
         if (c != 0) measure[i] = 0.0; else undecided = true;
      }
   }
   int cnt = __syncthreads_count(undecided);
   if (threadIdx.x == 0 && cnt) atomicAdd(remaining, cnt);
}

static int run_pmis(const DevCSR &S, int seed, int64_t goff, int *cf, double *measure, double *measure_keep, int *iters_out)
{
   int  n = S.nrows;
   int *cnt;
   HDK_TRY(dalloc(&cnt, (size_t)n + 1));
   HDK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)n + 1), g.stream));
   if (S.nnz > 0) { k_count_cols<<<cdiv(S.nnz, 256), 256, 0, g.stream>>>(S.col, S.nnz, cnt); HDK_LAUNCH_CHECK(); }
   uint32_t s0 = seed < 1 ? 1u : (seed >= 2147483647 ? 2147483646u : (uint32_t)seed);
   k_measure<<<cdiv(n, 256), 256, 0, g.stream>>>(cnt, n, s0, goff, measure);
   HDK_LAUNCH_CHECK();
   dfree(cnt);
   if (measure_keep) HDK_CUDA(cudaMemcpyAsync(measure_keep, measure, sizeof(double) * (size_t)n, cudaMemcpyDeviceToDevice, g.stream));
   k_pmis_init<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, n, cf, measure);
   HDK_LAUNCH_CHECK();
   int *rem = reinterpret_cast<int *>(g.dscal + S_TMP2);
   int  iters = 0, hrem = 1;
   while (hrem > 0 && iters < 1000)
   {
      HDK_CUDA(cudaMemsetAsync(rem, 0, sizeof(int), g.stream));
      k_pmis_mark<<<cdiv(n, 256), 256, 0, g.stream>>>(n, cf, measure);
      HDK_LAUNCH_CHECK();
      k_pmis_elim<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, S.col, n, cf, measure, 0);
      HDK_LAUNCH_CHECK();
      k_pmis_set<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, S.col, n, cf, measure, rem, 0);
      HDK_LAUNCH_CHECK();
      HDK_CUDA(cudaMemcpyAsync(&hrem, rem, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
      HDK_CUDA(cudaStreamSynchronize(g.stream));
      iters++;
   }
   if (iters_out) *iters_out = iters;
   return HDK_OK;
}

// stage launchers used by the distributed driver (hdk_amg_dist.cu): same kernels, rows [row0, row0+n)
__global__ void k_count_cols_rows(const int *srp, const int *scol, int row0, int n, int *cnt)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   for (int k = srp[row0 + i]; k < srp[row0 + i + 1]; k++) atomicAdd(cnt + scol[k], 1);
}
int pmis_count_cols(const DevCSR &S, int row0, int n, int *cnt)
{
   if (n <= 0) return HDK_OK;
   k_count_cols_rows<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, S.col, row0, n, cnt);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}
int pmis_measure(const int *cnt, int n, int seed, int64_t goff, double *measure)
{
   if (n <= 0) return HDK_OK;
   uint32_t s0 = seed < 1 ? 1u : (seed >= 2147483647 ? 2147483646u : (uint32_t)seed);
   k_measure<<<cdiv(n, 256), 256, 0, g.stream>>>(cnt, n, s0, goff, measure);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}
int pmis_init(const DevCSR &S, int row0, int n, int *cf, double *measure)
{
   if (n <= 0) return HDK_OK;
   k_pmis_init<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr + row0, n, cf + row0, measure + row0);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}
int pmis_mark(int n, int *cf, const double *measure)
{
   if (n <= 0) return HDK_OK;
   k_pmis_mark<<<cdiv(n, 256), 256, 0, g.stream>>>(n, cf, measure);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}
int pmis_elim(const DevCSR &S, int row0, int n, int *cf, const double *measure)
{
   if (n <= 0) return HDK_OK;
   k_pmis_elim<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, S.col, n, cf, measure, row0);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}
int pmis_set(const DevCSR &S, int row0, int n, int *cf, double *measure, int *remaining)
{
   if (n <= 0) return HDK_OK;
   k_pmis_set<<<cdiv(n, 256), 256, 0, g.stream>>>(S.rowptr, S.col, n, cf, measure, remaining, row0);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}

__global__ void k_cf_flag(const int *cf, int n, int *flag)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   flag[i] = (i < n && cf[i] > 0) ? 1 : 0;
}

// =====================================================================================
// extended+i interpolation (hypre_BoomerAMGBuildExtPIInterp) + truncation
// (hypre_BoomerAMGInterpTruncation with hypre_qsort2abs): one thread per row
// =====================================================================================
__global__ void k_interp_cap(const int *srp, const int *scol, const int *cf, int n, int *cap, const int *slow)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   int c = 0;
   if (i < n && slow[i] && cf[i] < 0 && cf[i] != SF_PT)
   {
      int ub = 0;
      for (int k = srp[i]; k < srp[i + 1]; k++)
      {
         int j = scol[k];
         if (cf[j] > 0) ub++;
         else if (cf[j] != SF_PT) ub += srp[j + 1] - srp[j];
      }
      c = pow2ceil(2 * ub);
   }
   cap[i] = c;
}

__global__ void k_interp_count(const int *srp, const int *scol, const int *cf, int row0, int row1,
                               const int64_t *off, int *keys, int max_elmts, int *cnt, int *rowlen, const int *slow)
{
   int i = row0 + blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= row1 || !slow[i]) return;
   int c = 0;
   if (cf[i] > 0) c = 1;
   else if (cf[i] != SF_PT)
   {
      int *tab = keys + (off[i] - off[row0]);
      int  cap = (int)(off[i + 1] - off[i]);
      for (int k = srp[i]; k < srp[i + 1]; k++)
      {
         int i1 = scol[k];
         if (cf[i1] > 0) { if (hset_insert(tab, cap, i1)) c++; }
         else if (cf[i1] != SF_PT)
            for (int kk = srp[i1]; kk < srp[i1 + 1]; kk++)
            {
               int k1 = scol[kk];
               if (cf[k1] > 0 && hset_insert(tab, cap, k1)) c++;
            }
      }
   }
   cnt[i]    = c;
   rowlen[i] = (max_elmts > 0 && c > max_elmts) ? max_elmts : c;
}

__global__ void k_interp_cap2(const int *srp, const int *cf, const int *cnt, int n, int *cap2, const int *slow)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   int c = 0;
   if (i < n && slow[i] && cf[i] < 0 && cf[i] != SF_PT) c = pow2ceil(2 * (cnt[i] + (srp[i + 1] - srp[i])));
   cap2[i] = c;
}

__device__ __forceinline__ void swap2(int *v, double *w, int i, int j)
{
   int t = v[i]; v[i] = v[j]; v[j] = t;
   double d = w[i]; w[i] = w[j]; w[j] = d;
}

// hypre_qsort2abs without recursion: the partition of every sub-range is independent of the
// order sub-ranges are visited in, so an explicit stack gives the identical arrangement.
// `keep`: only positions [0, keep) of the result are used by the caller (interpolation truncation keeps
// the max_elmts largest |w|).  A sub-range that starts at or beyond `keep` can never move an element
// into [0, keep), so it is not sorted at all -- the leading positions end up exactly as the full
// quicksort leaves them (ties included) at O(n + keep log keep) instead of O(n log n) swaps.
__device__ void qsort2abs_dev(int *v, double *w, int n, int keep)
{
   int stl[40], str[40], sp = 0;
   stl[0] = 0; str[0] = n - 1; sp = 1;
   while (sp > 0)
   {
      sp--;
      int left = stl[sp], right = str[sp];
      while (left < right && left < keep)
      {
         swap2(v, w, left, (left + right) / 2);
         int last = left;
         for (int i = left + 1; i <= right; i++)
            if (fabs(w[i]) > fabs(w[left])) swap2(v, w, ++last, i);
         swap2(v, w, left, last);
         // recurse on the smaller part first (bounded stack), loop on the other
         int l1 = left, r1 = last - 1, l2 = last + 1, r2 = right;
         if (r1 - l1 < r2 - l2)
         {
            if (l2 < r2 && l2 < keep) { stl[sp] = l2; str[sp] = r2; sp++; }
            left = l1; right = r1;
         }
         else
         {
            if (l1 < r1 && l1 < keep) { stl[sp] = l1; str[sp] = r1; sp++; }
            left = l2; right = r2;
         }
      }
   }
}

__global__ void k_interp_fill(const int *arp, const int *acol, const double *aval, const int *srp, const int *scol,
                              const int *cf, const int *f2c, int row0, int row1, const int *cnt,
                              const int64_t *hoff, int2 *htab, const int64_t *loff, int *lcol, double *lval,
                              int max_elmts, const int *prp, int *pcol, double *pval, const int *slow)
{
   int i = row0 + blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= row1 || !slow[i]) return;
   int p0 = prp[i];
   if (cf[i] > 0) { pcol[p0] = f2c[i]; pval[p0] = 1.0; return; }
   if (cf[i] == SF_PT) return;
   int2   *tab = htab + (hoff[i] - hoff[row0]);
   int     cap = (int)(hoff[i + 1] - hoff[i]);
   int    *lc  = lcol + (loff[i] - loff[row0]);
   double *lv  = lval + (loff[i] - loff[row0]);
   int     nC  = 0;
   // discovery of C-hat_i in hypre's order; strong F neighbours are tagged with -2
   for (int k = srp[i]; k < srp[i + 1]; k++)
   {
      int i1 = scol[k];
      if (cf[i1] > 0)
      {
         if (hmap_insert(tab, cap, i1, nC) == -1) { lc[nC] = i1; lv[nC] = 0.0; nC++; }
      }
      else if (cf[i1] != SF_PT)
      {
         hmap_insert(tab, cap, i1, -2);
         for (int kk = srp[i1]; kk < srp[i1 + 1]; kk++)
         {
            int k1 = scol[kk];
            if (cf[k1] > 0 && hmap_insert(tab, cap, k1, nC) == -1) { lc[nC] = k1; lv[nC] = 0.0; nC++; }
         }
      }
   }
   double diagonal = aval[arp[i]];
   for (int jj = arp[i] + 1; jj < arp[i + 1]; jj++)
   {
      int    i1 = acol[jj];
      double a  = aval[jj];
      int    m  = hmap_find(tab, cap, i1);
      if (m >= 0) lv[m] = __dadd_rn(lv[m], a);
      else if (m == -2)
      {
         double sum = 0.0;
         double sgn = aval[arp[i1]] < 0 ? -1.0 : 1.0;
         for (int j1 = arp[i1] + 1; j1 < arp[i1 + 1]; j1++)
         {
            int    i2 = acol[j1];
            double v  = aval[j1];
            if (sgn * v < 0 && (i2 == i || hmap_find(tab, cap, i2) >= 0)) sum = __dadd_rn(sum, v);
         }
         if (sum != 0.0)
         {
            double distribute = __ddiv_rn(a, sum);
            for (int j1 = arp[i1] + 1; j1 < arp[i1 + 1]; j1++)
            {
               int    i2 = acol[j1];
               double v  = aval[j1];
               if (sgn * v < 0)
               {
                  int m2 = hmap_find(tab, cap, i2);
                  if (m2 >= 0) lv[m2] = __dadd_rn(lv[m2], __dmul_rn(distribute, v));
                  if (i2 == i) diagonal = __dadd_rn(diagonal, __dmul_rn(distribute, v));
               }
            }
         }
         else diagonal = __dadd_rn(diagonal, a);
      }
      else if (cf[i1] != SF_PT) diagonal = __dadd_rn(diagonal, a);
   }
   if (diagonal != 0.0)
   {
      double nd = -diagonal;
      for (int k = 0; k < nC; k++) lv[k] = __ddiv_rn(lv[k], nd);
   }
   int len = nC;
   if (max_elmts > 0 && nC > max_elmts)
   {
      double row_sum = 0.0, scale = 0.0;
      for (int k = 0; k < nC; k++) row_sum = __dadd_rn(row_sum, lv[k]);
      qsort2abs_dev(lc, lv, nC, max_elmts);
      for (int k = 0; k < max_elmts; k++) scale = __dadd_rn(scale, lv[k]);
      if (scale != 0.0 && scale != row_sum)
      {
         scale = __ddiv_rn(row_sum, scale);
         for (int k = 0; k < max_elmts; k++) lv[k] = __dmul_rn(lv[k], scale);
      }
      len = max_elmts;
   }
   for (int k = 0; k < len; k++) { pcol[p0 + k] = f2c[lc[k]]; pval[p0 + k] = lv[k]; }
}

// ---- one thread per row, C-hat in thread-local arrays (short rows: the stencil levels) -----------
// Single pass like k_interp_warp<true, true>: discovery, weights and truncation of a row in one go, the
// result in slot i * max_elmts of the staging buffer, cnt / rowlen / slow set for the later passes.
// C-hat of a 7-point row has at most ~20 members, so a linear search over a local array replaces the
// hash table in global scratch (round 2 before: 8.6 GB of tables for 256^3, 10.7 GB of DRAM traffic
// and a counting pass).  Slots are assigned in discovery order, exactly like the tables' indices, so
// every sum is accumulated in the same order.  Rows that do not fit the arrays are flagged slow.
constexpr int IS_CAP = 48; // |C-hat| handled here
constexpr int IS_F   = 24; // strong F neighbours handled here
__device__ __forceinline__ int is_find(const int *key, int n, int k)
{
   for (int j = 0; j < n; j++)
      if (key[j] == k) return j;
   return -1;
}
__global__ void __launch_bounds__(128) k_interp_small(const int *arp, const int *acol, const double *aval, const int *srp,
                                                      const int *scol, const int *cf, const int *f2c, int row_lo, int row_hi,
                                                      int max_elmts, int *cnt, int *rowlen, int *slow, int *scol_out, double *sval_out)
{
   const int i = row_lo + blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= row_hi) return;
   const int       ci = cf[i];
   const long long p0 = (long long)i * max_elmts;
   if (ci > 0) { cnt[i] = 1; rowlen[i] = 1; slow[i] = 0; scol_out[p0] = f2c[i]; sval_out[p0] = 1.0; return; }
   if (ci == SF_PT) { cnt[i] = 0; rowlen[i] = 0; slow[i] = 0; return; }
   int    lc[IS_CAP], fk[IS_F];
   double lv[IS_CAP];
   int    nC = 0, nF = 0;
   bool   overflow = false;
   // discovery of C-hat_i in hypre's order
   for (int k = srp[i]; k < srp[i + 1] && !overflow; k++)
   {
      const int i1 = scol[k], c1 = cf[i1];
      if (c1 > 0)
      {
         if (is_find(lc, nC, i1) < 0) { if (nC < IS_CAP) { lc[nC] = i1; lv[nC] = 0.0; nC++; } else overflow = true; }
      }
      else if (c1 != SF_PT)
      {
         if (nF < IS_F) fk[nF++] = i1; else overflow = true;
         for (int kk = srp[i1]; kk < srp[i1 + 1] && !overflow; kk++)
         {
            const int k1 = scol[kk];
            if (cf[k1] > 0 && is_find(lc, nC, k1) < 0) { if (nC < IS_CAP) { lc[nC] = k1; lv[nC] = 0.0; nC++; } else overflow = true; }
         }
      }
   }
   if (overflow) { cnt[i] = 0; rowlen[i] = 0; slow[i] = 1; return; } // (the table-based path does this row)
   cnt[i] = nC; rowlen[i] = (nC > max_elmts) ? max_elmts : nC; slow[i] = 0;
   // weights: the row of A in stored order
   double diagonal = aval[arp[i]];
   for (int jj = arp[i] + 1; jj < arp[i + 1]; jj++)
   {
      const int    i1 = acol[jj];
      const double a  = aval[jj];
      const int    m  = is_find(lc, nC, i1);
      if (m >= 0) lv[m] = __dadd_rn(lv[m], a);
      else if (is_find(fk, nF, i1) >= 0)
      {
         double       sum = 0.0;
         const int    b1 = arp[i1] + 1, e1 = arp[i1 + 1];
         const double sgn = aval[b1 - 1] < 0 ? -1.0 : 1.0;
         for (int j1 = b1; j1 < e1; j1++)
         {
            const int    i2 = acol[j1];
            const double v  = aval[j1];
            if (sgn * v < 0 && (i2 == i || is_find(lc, nC, i2) >= 0)) sum = __dadd_rn(sum, v);
         }
         if (sum != 0.0)
         {
            const double distribute = __ddiv_rn(a, sum);
            for (int j1 = b1; j1 < e1; j1++)
            {
               const int    i2 = acol[j1];
               const double v  = aval[j1];
               if (sgn * v < 0)
               {
                  const int m2 = is_find(lc, nC, i2);
                  if (m2 >= 0) lv[m2] = __dadd_rn(lv[m2], __dmul_rn(distribute, v));
                  if (i2 == i) diagonal = __dadd_rn(diagonal, __dmul_rn(distribute, v));
               }
            }
         }
         else diagonal = __dadd_rn(diagonal, a);
      }
      else if (cf[i1] != SF_PT) diagonal = __dadd_rn(diagonal, a);
   }
   if (diagonal != 0.0)
   {
      const double nd = -diagonal;
      for (int k = 0; k < nC; k++) lv[k] = __ddiv_rn(lv[k], nd);
   }
   int len = nC;
   if (nC > max_elmts)
   {
      double row_sum = 0.0, scale = 0.0;
      for (int k = 0; k < nC; k++) row_sum = __dadd_rn(row_sum, lv[k]);
      qsort2abs_dev(lc, lv, nC, max_elmts);
      for (int k = 0; k < max_elmts; k++) scale = __dadd_rn(scale, lv[k]);
      if (scale != 0.0 && scale != row_sum)
      {
         scale = __ddiv_rn(row_sum, scale);
         for (int k = 0; k < max_elmts; k++) lv[k] = __dmul_rn(lv[k], scale);
      }
      len = max_elmts;
   }
   for (int k = 0; k < len; k++) { scol_out[p0 + k] = f2c[lc[k]]; sval_out[p0 + k] = lv[k]; }
}

// ---- warp-per-row extended+i interpolation (shared-memory hash + candidate list) ----------
// Same sequence of operations as the one-thread version (and the oracle): C-hat is discovered
// in hypre's order (chunks of 32 candidates, slots assigned in lane order), the weight loop
// runs sequentially over the row of A, lanes only parallelise the hash look-ups of the inner
// loops, and every floating-point sum is accumulated in CSR order.
constexpr int IW_CAP   = 256; // hash slots per warp: C-hat plus the strong F neighbours
constexpr int IW_LIST  = 120; // longest C-hat handled here
constexpr int IW_WARPS = 8;

__device__ __forceinline__ int wt_find(const int *keys, const int *idx, int cap, int key)
{
   unsigned h = hslot(key, cap), mask = (unsigned)cap - 1;
   while (true)
   {
      int k = keys[h];
      if (k == key) return idx[h];
      if (k == -1) return -1;
      h = (h + 1) & mask;
   }
}

// STAGE (single-pass interpolation, max_elmts > 0): discovery AND weights in one launch; the truncated
// row (at most max_elmts entries) goes to slot i * max_elmts of a staging buffer and cnt / rowlen / slow
// are set like the counting pass does, so no row is traversed twice.
template <bool FILL, bool STAGE = false>
__global__ void __launch_bounds__(32 * IW_WARPS) k_interp_warp(const int *arp, const int *acol, const double *aval,
                                                               const int *srp, const int *scol, const int *cf,
                                                               const int *f2c, int n, int max_elmts, int *cnt, int *rowlen,
                                                               int *slow, const int *prp, int *pcol, double *pval, int force_slow,
                                                               int row_lo)
{
   __shared__ int    s_keys[IW_WARPS][IW_CAP];
   __shared__ int    s_idx[IW_WARPS][IW_CAP];
   __shared__ int    s_lc[IW_WARPS][IW_LIST + 8];
   __shared__ double s_lv[IW_WARPS][IW_LIST + 8];
   const int      lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
   const unsigned FULL = 0xffffffffu, LT = (1u << lane) - 1u;
   const int      i = row_lo + blockIdx.x * IW_WARPS + wid; // rows [row_lo, n)
   if (i >= n) return;
   const int ci = cf[i];
   if (ci > 0)
   {
      if (lane == 0)
      {
         if (!FILL || STAGE) { cnt[i] = 1; rowlen[i] = 1; slow[i] = 0; }
         if (FILL) { const int p1 = STAGE ? i * max_elmts : prp[i]; pcol[p1] = f2c[i]; pval[p1] = 1.0; }
      }
      return;
   }
   if (ci == SF_PT) { if ((!FILL || STAGE) && lane == 0) { cnt[i] = 0; rowlen[i] = 0; slow[i] = 0; } return; }
   if (FILL && !STAGE && slow[i]) return;
   if (!FILL && force_slow) { if (lane == 0) { slow[i] = 1; cnt[i] = 0; rowlen[i] = 0; } return; }
   int *keys = s_keys[wid], *idx = s_idx[wid], *lc = s_lc[wid];
   double *lv = s_lv[wid];
   for (int h = lane; h < IW_CAP; h += 32) keys[h] = -1;
   __syncwarp();
   int  nC = 0, nins = 0;
   bool overflow = false;
   // ---- discovery of C-hat_i; strong F neighbours are tagged with idx = -2.  The row overflows once
   // |C-hat| > IW_LIST or the inserts (C-hat plus strong F neighbours) exceed IW_INS; the count is
   // checked after every insert (of at most 32 keys), so the table never holds more than IW_INS + 32
   // keys and never fills: in a full open-addressing table wt_find_or_insert would probe forever.
   constexpr int IW_INS = (IW_CAP * 3) / 4;
   for (int jj = srp[i]; jj < srp[i + 1] && !overflow; jj++)
   {
      const int i1 = scol[jj], c1 = cf[i1];
      if (c1 > 0)
      {
         bool isnew = false;
         int  h = 0;
         if (lane == 0) h = wt_find_or_insert(keys, IW_CAP, i1, isnew);
         unsigned nm = __ballot_sync(FULL, lane == 0 && isnew);
         if (nm)
         {
            if (nC >= IW_LIST) overflow = true;
            else if (lane == 0) { idx[h] = nC; lc[nC] = i1; lv[nC] = 0.0; }
            nC++; nins++;
            if (nins > IW_INS) overflow = true;
         }
      }
      else if (c1 != SF_PT)
      {
         if (lane == 0) { bool nw; int h = wt_find_or_insert(keys, IW_CAP, i1, nw); idx[h] = -2; }
         nins++;
         if (nins > IW_INS) overflow = true;
         __syncwarp();
         for (int base = srp[i1]; base < srp[i1 + 1] && !overflow; base += 32)
         {
            const int  kk = base + lane;
            const int  k1 = kk < srp[i1 + 1] ? scol[kk] : -1;
            const bool act = k1 >= 0 && cf[k1] > 0;
            bool       isnew = false;
            int        h = 0;
            if (act) h = wt_find_or_insert(keys, IW_CAP, k1, isnew);
            const unsigned nm = __ballot_sync(FULL, act && isnew);
            const int      add = __popc(nm);
            if (nC + add > IW_LIST || nins + add > IW_INS) overflow = true;
            else if (act && isnew) { int s = nC + __popc(nm & LT); idx[h] = s; lc[s] = k1; lv[s] = 0.0; }
            nC += add; nins += add;
            __syncwarp();
         }
      }
      __syncwarp();
   }
   if (!FILL || STAGE)
   {
      if (lane == 0)
      {
         slow[i]   = overflow ? 1 : 0;
         cnt[i]    = overflow ? 0 : nC;
         rowlen[i] = overflow ? 0 : ((max_elmts > 0 && nC > max_elmts) ? max_elmts : nC);
      }
      if (!FILL || overflow) return; // (single pass: a row this table cannot hold goes to the one-thread path)
   }
   // ---- weights: sequential over the row of A (hypre's order), lanes over the inner look-ups.
   // The per-entry operands (column, value, table look-up, and for strong F neighbours the row
   // bounds and diagonal sign of A_{i1}) are fetched by 32 lanes at once and broadcast with
   // shuffles, so the sequential loop has no chain of dependent global loads.
   const int rs = arp[i], re = arp[i + 1];
   double    diagonal = aval[rs];
   for (int cb = rs + 1; cb < re; cb += 32)
   {
      const int    jl = cb + lane;
      const bool   vl = jl < re;
      const int    p_i1 = vl ? acol[jl] : -1;
      const double p_a  = vl ? aval[jl] : 0.0;
      int          p_m = -1, p_b1 = 0, p_e1 = 0, p_cf = 0;
      double       p_sgn = 1.0;
      if (vl)
      {
         p_m = wt_find(keys, idx, IW_CAP, p_i1);
         if (p_m == -2)
         {
            const int d1 = arp[p_i1];
            p_e1  = arp[p_i1 + 1];
            p_sgn = aval[d1] < 0 ? -1.0 : 1.0;
            p_b1  = d1 + 1;
         }
         else if (p_m < 0) p_cf = cf[p_i1];
      }
      const int nchunk = (re - cb) < 32 ? (re - cb) : 32;
      for (int t = 0; t < nchunk; t++)
      {
         const double a = __shfl_sync(FULL, p_a, t);
         const int    m = __shfl_sync(FULL, p_m, t);
         if (m >= 0) { if (lane == 0) lv[m] = __dadd_rn(lv[m], a); }
         else if (m == -2)
         {
            const double sgn = __shfl_sync(FULL, p_sgn, t);
            const int    b1 = __shfl_sync(FULL, p_b1, t), e1 = __shfl_sync(FULL, p_e1, t);
            double       sum = 0.0;
            if (e1 - b1 <= 32)
            {
               // the neighbour's row fits one chunk (the usual case): its entries, signs and table
               // look-ups are fetched ONCE and serve both the ordered sum and the distribution
               const int    j1 = b1 + lane;
               const bool   v1 = j1 < e1;
               const int    i2 = v1 ? acol[j1] : -1;
               const double v  = v1 ? aval[j1] : 0.0;
               const bool   neg = v1 && (sgn * v < 0);
               const int    m2 = neg ? wt_find(keys, idx, IW_CAP, i2) : -1;
               unsigned     rem = __ballot_sync(FULL, neg && (i2 == i || m2 >= 0));
               while (rem) { int src = __ffs(rem) - 1; sum = __dadd_rn(sum, __shfl_sync(FULL, v, src)); rem &= rem - 1u; }
               if (sum != 0.0)
               {
                  const double tt = __dmul_rn(__ddiv_rn(a, sum), v);
                  if (neg && m2 >= 0) lv[m2] = __dadd_rn(lv[m2], tt);
                  const unsigned dm = __ballot_sync(FULL, neg && i2 == i);
                  if (dm) diagonal = __dadd_rn(diagonal, __shfl_sync(FULL, tt, __ffs(dm) - 1));
               }
               else diagonal = __dadd_rn(diagonal, a);
               __syncwarp();
               continue;
            }
            for (int base = b1; base < e1; base += 32)
            {
               const int    j1 = base + lane;
               const bool   v1 = j1 < e1;
               const int    i2 = v1 ? acol[j1] : -1;
               const double v  = v1 ? aval[j1] : 0.0;
               const bool   q  = v1 && (sgn * v < 0) && (i2 == i || wt_find(keys, idx, IW_CAP, i2) >= 0);
               unsigned     rem = __ballot_sync(FULL, q);
               while (rem) { int src = __ffs(rem) - 1; sum = __dadd_rn(sum, __shfl_sync(FULL, v, src)); rem &= rem - 1u; }
            }
            if (sum != 0.0)
            {
               const double distribute = __ddiv_rn(a, sum);
               for (int base = b1; base < e1; base += 32)
               {
                  const int    j1 = base + lane;
                  const bool   v1 = j1 < e1;
                  const int    i2 = v1 ? acol[j1] : -1;
                  const double v  = v1 ? aval[j1] : 0.0;
                  const bool   neg = v1 && (sgn * v < 0);
                  const int    m2 = neg ? wt_find(keys, idx, IW_CAP, i2) : -1;
                  const double tt = __dmul_rn(distribute, v);
                  if (neg && m2 >= 0) lv[m2] = __dadd_rn(lv[m2], tt);
                  const unsigned dm = __ballot_sync(FULL, neg && i2 == i);
                  if (dm) diagonal = __dadd_rn(diagonal, __shfl_sync(FULL, tt, __ffs(dm) - 1));
               }
            }
            else diagonal = __dadd_rn(diagonal, a);
         }
         else if (__shfl_sync(FULL, p_cf, t) != SF_PT) diagonal = __dadd_rn(diagonal, a);
         __syncwarp();
      }
   }
   if (diagonal != 0.0)
   {
      const double nd = -diagonal;
      for (int k = lane; k < nC; k += 32) lv[k] = __ddiv_rn(lv[k], nd);
   }
   __syncwarp();
   int len = nC;
   if (max_elmts > 0 && nC > max_elmts)
   {
      if (lane == 0)
      {
         double row_sum = 0.0, scale = 0.0;
         for (int k = 0; k < nC; k++) row_sum = __dadd_rn(row_sum, lv[k]);
         qsort2abs_dev(lc, lv, nC, max_elmts);
         for (int k = 0; k < max_elmts; k++) scale = __dadd_rn(scale, lv[k]);
         if (scale != 0.0 && scale != row_sum)
         {
            scale = __ddiv_rn(row_sum, scale);
            for (int k = 0; k < max_elmts; k++) lv[k] = __dmul_rn(lv[k], scale);
         }
      }
      len = max_elmts;
      __syncwarp();
   }
   const int p0 = STAGE ? i * max_elmts : prp[i];
   for (int k = lane; k < len; k += 32) { pcol[p0 + k] = f2c[lc[k]]; pval[p0 + k] = lv[k]; }
}

// staged rows (slot i * stride) -> CSR position; rows of the one-thread path are filled by k_interp_fill
__global__ void k_interp_compact(const int *rowlen, const int *slow, const int *prp, const int *scol, const double *sval, int stride,
                                 int row_lo, int row_hi, int *pcol, double *pval)
{
   int i = row_lo + blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= row_hi || slow[i]) return;
   const int len = rowlen[i], p0 = prp[i];
   const long long s0 = (long long)i * stride;
   for (int k = 0; k < len; k++) { pcol[p0 + k] = scol[s0 + k]; pval[p0 + k] = sval[s0 + k]; }
}

__global__ void k_mask_cnt(const int *cnt, const int *slow, int n, int *out)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i <= n) out[i] = (i < n && slow[i]) ? cnt[i] : 0;
}

__global__ void k_cf_reset_sf(int *cf, int n)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n && cf[i] == SF_PT) cf[i] = F_PT;
}

// hypre_BoomerAMGInterpTruncation as a post-pass (used when trunc_factor > 0; with trunc_factor
// = 0 the max_elmts stage is fused into the interpolation kernels): per row, drop the weights
// below trunc_factor * max|w| and rescale the rest to the old row sum, then keep the max_elmts
// largest |w| (hypre_qsort2abs order) and rescale again.  One thread per row, in place.
__global__ void k_trunc_rows(const int *rp, int *col, double *val, int n, double tf, int max_elmts, int *newlen)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   if (i == n) { newlen[i] = 0; return; }
   int b = rp[i], e = rp[i + 1], len = e - b;
   if (tf > 0.0 && len > 0)
   {
      double maxc = 0.0, row_sum = 0.0, scale = 0.0;
      for (int k = b; k < e; k++) if (fabs(val[k]) > maxc) maxc = fabs(val[k]);
      maxc  = __dmul_rn(maxc, tf);
      int w = b;
      for (int k = b; k < e; k++)
      {
         double v = val[k];
         row_sum  = __dadd_rn(row_sum, v);
         if (!(fabs(v) < maxc)) { scale = __dadd_rn(scale, v); col[w] = col[k]; val[w] = v; w++; }
      }
      if (scale != 0.0 && scale != row_sum)
      {
         scale = __ddiv_rn(row_sum, scale);
         for (int k = b; k < w; k++) val[k] = __dmul_rn(val[k], scale);
      }
      len = w - b;
      e   = w;
   }
   if (max_elmts > 0 && len > max_elmts)
   {
      double row_sum = 0.0, scale = 0.0;
      for (int k = b; k < e; k++) row_sum = __dadd_rn(row_sum, val[k]);
      qsort2abs_dev(col + b, val + b, len, max_elmts);
      for (int k = 0; k < max_elmts; k++) scale = __dadd_rn(scale, val[b + k]);
      if (scale != 0.0 && scale != row_sum)
      {
         scale = __ddiv_rn(row_sum, scale);
         for (int k = 0; k < max_elmts; k++) val[b + k] = __dmul_rn(val[b + k], scale);
      }
      len = max_elmts;
   }
   newlen[i] = len;
}
__global__ void k_compact_rows(const int *rp, const int *col, const double *val, const int *nrp, int n, int *ncol, double *nval)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   int b = rp[i], nb = nrp[i], len = nrp[i + 1] - nb;
   for (int k = 0; k < len; k++) { ncol[nb + k] = col[b + k]; nval[nb + k] = val[b + k]; }
}
static int interp_truncate(DevCSR &P, double trunc_factor, int max_elmts)
{
   const int n = P.nrows;
   int *newlen, *nrp;
   HDK_TRY(dalloc(&newlen, (size_t)n + 1));
   HDK_TRY(dalloc(&nrp, (size_t)n + 1));
   k_trunc_rows<<<cdiv(n + 1, 128), 128, 0, g.stream>>>(P.rowptr, P.col, P.val, n, trunc_factor, max_elmts, newlen);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_int(newlen, nrp, n + 1));
   int nnz = 0;
   HDK_CUDA(cudaMemcpyAsync(&nnz, nrp + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   DevCSR Q;
   Q.nrows = n; Q.ncols = P.ncols; Q.nnz = nnz; Q.rowptr = nrp; Q.owns = true;
   HDK_TRY(dalloc(&Q.col, (size_t)nnz + 8));
   HDK_TRY(dalloc(&Q.val, (size_t)nnz + 8));
   HDK_CUDA(cudaMemsetAsync(Q.col + nnz, 0, sizeof(int) * 8, g.stream));
   HDK_CUDA(cudaMemsetAsync(Q.val + nnz, 0, sizeof(double) * 8, g.stream));
   k_compact_rows<<<cdiv(n, 128), 128, 0, g.stream>>>(P.rowptr, P.col, P.val, nrp, n, Q.col, Q.val);
   HDK_LAUNCH_CHECK();
   dfree(newlen);
   csr_free(P);
   P = Q;
   return HDK_OK;
}

// rows [row_lo, row_hi) only (row_lo < 0: all rows, or this rank's share of a work-shared global level)
int build_interp(const DevCSR &A, const DevCSR &S, int *cf, const int *f2c, int nc, int max_elmts_in, double trunc_factor,
                 DevCSR &P, int row_lo, int row_hi)
{
   // with a truncation factor the rows are built complete and truncated by the post-pass
   const int max_elmts = (trunc_factor > 0.0) ? 0 : max_elmts_in;
   int  n = A.nrows;
   int *cap, *cnt, *rowlen, *prp;
   int64_t *off;
   HDK_TRY(dalloc(&cap, (size_t)n + 1));
   HDK_TRY(dalloc(&cnt, (size_t)n + 1));
   HDK_TRY(dalloc(&rowlen, (size_t)n + 1));
   HDK_TRY(dalloc(&prp, (size_t)n + 1));
   HDK_TRY(dalloc(&off, (size_t)n + 1));
   int *slow;
   HDK_TRY(dalloc(&slow, (size_t)n + 1));
   // short rows (fine stencil levels): one thread per row beats one warp per row
   static double slow_avg = -1.0; // HDK_INTERP_THREAD_AVG: rows up to this average length go one thread per row
   if (slow_avg < 0.0) { const char *e = getenv("HDK_INTERP_THREAD_AVG"); slow_avg = e ? atof(e) : 10.0; }
   const int force_slow = ((double)A.nnz / (n > 0 ? n : 1)) <= slow_avg ? 1 : 0;
   // this rank's share of the rows (all of them unless the multi-rank setup shares the work);
   // rows outside it keep slow = cnt = rowlen = 0, which every later kernel skips
   int lo, hi;
   share_range(n, lo, hi);
   if (row_lo >= 0) { lo = row_lo; hi = row_hi; }
   if (share_on(n) || lo != 0 || hi != n)
   {
      HDK_CUDA(cudaMemsetAsync(slow, 0, sizeof(int) * ((size_t)n + 1), g.stream));
      HDK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)n + 1), g.stream));
      HDK_CUDA(cudaMemsetAsync(rowlen, 0, sizeof(int) * ((size_t)n + 1), g.stream));
   }
   // Single-pass interpolation (rows of at most max_elmts entries): discovery and weights in ONE launch
   // into a fixed-stride staging buffer, row lengths from the same launch -- one warp per row with a
   // shared-memory table, or one thread per row with thread-local arrays on the stencil levels.  The
   // counting pass below is only needed when rows are unbounded (no truncation) or for flagged rows.
   static int interp_single = -1;
   if (interp_single < 0) { const char *e = getenv("HDK_INTERP_SINGLE"); interp_single = (e && atoi(e) == 0) ? 0 : 1; }
   const bool staged = interp_single == 1 && max_elmts > 0 && (long long)n * max_elmts < 2000000000LL;
   int    *stg_col = nullptr;
   double *stg_val = nullptr;
   if (staged)
   {
      HDK_TRY(dalloc(&stg_col, (size_t)n * max_elmts + 8));
      HDK_TRY(dalloc(&stg_val, (size_t)n * max_elmts + 8));
      if (force_slow) // short rows: one thread per row with thread-local tables
      {
         if (hi > lo)
            k_interp_small<<<cdiv(hi - lo, 128), 128, 0, g.stream>>>(A.rowptr, A.col, A.val, S.rowptr, S.col, cf, f2c, lo, hi, max_elmts,
                                                                     cnt, rowlen, slow, stg_col, stg_val);
      }
      else
         k_interp_warp<true, true><<<cdiv(hi - lo, IW_WARPS), 32 * IW_WARPS, 0, g.stream>>>(A.rowptr, A.col, A.val, S.rowptr, S.col, cf, f2c, hi,
                                                                                            max_elmts, cnt, rowlen, slow, nullptr, stg_col, stg_val, 0, lo);
      HDK_LAUNCH_CHECK();
   }
   else
   {
      // pass 1a: |C-hat_i| by the warp kernel (shared-memory hash); rows it cannot hold are flagged
      k_interp_warp<false><<<cdiv(hi - lo, IW_WARPS), 32 * IW_WARPS, 0, g.stream>>>(A.rowptr, A.col, A.val, S.rowptr, S.col, cf, f2c, hi,
                                                                                   max_elmts, cnt, rowlen, slow, nullptr, nullptr, nullptr, force_slow, lo);
      HDK_LAUNCH_CHECK();
   }
   // pass 1b: flagged rows, one thread per row, hash sets in global scratch (chunked)
   k_interp_cap<<<cdiv(n + 1, 256), 256, 0, g.stream>>>(S.rowptr, S.col, cf, n, cap, slow);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_i64(cap, off, n + 1));
   std::vector<int> bounds;
   int64_t          maxsz;
   HDK_TRY(plan_chunks(off, n, bounds, maxsz));
   {
      int *keys;
      HDK_TRY(dalloc(&keys, (size_t)maxsz + 4));
      for (size_t c = 0; c + 1 < bounds.size(); c++)
      {
         int r0 = bounds[c], r1 = bounds[c + 1];
         if (r1 <= r0) continue;
         HDK_CUDA(cudaMemsetAsync(keys, 0xFF, sizeof(int) * ((size_t)maxsz + 4), g.stream));
         k_interp_count<<<cdiv(r1 - r0, 128), 128, 0, g.stream>>>(S.rowptr, S.col, cf, r0, r1, off, keys, max_elmts, cnt, rowlen, slow);
         HDK_LAUNCH_CHECK();
      }
      dfree(keys);
   }
   HDK_CUDA(cudaMemsetAsync(rowlen + n, 0, sizeof(int), g.stream));
   HDK_CUDA(cudaMemsetAsync(cnt + n, 0, sizeof(int), g.stream));
   HDK_TRY(share_rows(rowlen, sizeof(int), n)); // row lengths of the other ranks' shares
   HDK_TRY(check_fits_int32(rowlen, n, "the interpolation operator"));
   HDK_TRY(exclusive_scan_int(rowlen, prp, n + 1));
   int nnzP = 0;
   HDK_CUDA(cudaMemcpyAsync(&nnzP, prp + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   P = DevCSR();
   P.nrows = n; P.ncols = nc; P.nnz = nnzP; P.rowptr = prp; P.owns = true;
   HDK_TRY(dalloc(&P.col, (size_t)nnzP + 8));
   HDK_TRY(dalloc(&P.val, (size_t)nnzP + 8));
   HDK_CUDA(cudaMemsetAsync(P.col + nnzP, 0, sizeof(int) * 8, g.stream));
   HDK_CUDA(cudaMemsetAsync(P.val + nnzP, 0, sizeof(double) * 8, g.stream));
   // pass 2: weights.  hash maps sized from the exact counts, candidate lists in scratch
   int64_t *loff;
   HDK_TRY(dalloc(&loff, (size_t)n + 1));
   if (staged)
   {
      k_interp_compact<<<cdiv(hi - lo, 256), 256, 0, g.stream>>>(rowlen, slow, prp, stg_col, stg_val, max_elmts, lo, hi, P.col, P.val);
      HDK_LAUNCH_CHECK();
      dfree(stg_col); dfree(stg_val);
   }
   else
   {
      k_interp_warp<true><<<cdiv(hi - lo, IW_WARPS), 32 * IW_WARPS, 0, g.stream>>>(A.rowptr, A.col, A.val, S.rowptr, S.col, cf, f2c, hi,
                                                                                  max_elmts, cnt, rowlen, slow, prp, P.col, P.val, force_slow, lo);
      HDK_LAUNCH_CHECK();
   }
   k_interp_cap2<<<cdiv(n + 1, 256), 256, 0, g.stream>>>(S.rowptr, cf, cnt, n, cap, slow);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_i64(cap, off, n + 1));
   k_mask_cnt<<<cdiv(n + 1, 256), 256, 0, g.stream>>>(cnt, slow, n, rowlen); // candidate lists only for the fallback rows
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_i64(rowlen, loff, n + 1));
   HDK_TRY(plan_chunks(off, n, bounds, maxsz));
   {
      int64_t maxl = 0;
      for (size_t c = 0; c + 1 < bounds.size(); c++)
      {
         int64_t o[2];
         HDK_CUDA(cudaMemcpyAsync(&o[0], loff + bounds[c], sizeof(int64_t), cudaMemcpyDeviceToHost, g.stream));
         HDK_CUDA(cudaMemcpyAsync(&o[1], loff + bounds[c + 1], sizeof(int64_t), cudaMemcpyDeviceToHost, g.stream));
         HDK_CUDA(cudaStreamSynchronize(g.stream));
         if (o[1] - o[0] > maxl) maxl = o[1] - o[0];
      }
      int2   *htab;
      int    *lcol;
      double *lval;
      HDK_TRY(dalloc(&htab, (size_t)maxsz + 4));
      HDK_TRY(dalloc(&lcol, (size_t)maxl + 4));
      HDK_TRY(dalloc(&lval, (size_t)maxl + 4));
      for (size_t c = 0; c + 1 < bounds.size(); c++)
      {
         int r0 = bounds[c], r1 = bounds[c + 1];
         if (r1 <= r0) continue;
         HDK_CUDA(cudaMemsetAsync(htab, 0xFF, sizeof(int2) * ((size_t)maxsz + 4), g.stream));
         k_interp_fill<<<cdiv(r1 - r0, 128), 128, 0, g.stream>>>(A.rowptr, A.col, A.val, S.rowptr, S.col, cf, f2c, r0, r1,
                                                                cnt, off, htab, loff, lcol, lval, max_elmts, prp, P.col, P.val, slow);
         HDK_LAUNCH_CHECK();
      }
      dfree(htab); dfree(lcol); dfree(lval);
   }
   HDK_TRY(share_entries(prp, n, P.col, sizeof(int), P.val, sizeof(double)));
   k_cf_reset_sf<<<cdiv(n, 256), 256, 0, g.stream>>>(cf, n);
   HDK_LAUNCH_CHECK();
   dfree(cap); dfree(cnt); dfree(rowlen); dfree(off); dfree(loff); dfree(slow);
   if (trunc_factor > 0.0) HDK_TRY(interp_truncate(P, trunc_factor, max_elmts_in));
   return HDK_OK;
}

// =====================================================================================
// R = P^T (hypre_CSRMatrixTranspose order: ascending fine row inside each coarse row)
// =====================================================================================
// Counting transpose: per-column counts (atomics on distinct addresses), scan, scatter through
// per-column cursors, then every row of the transpose is put in ascending order of the source row
// by the thread that owns it (interpolation transposes have ~10-30 entries per row; the source
// rows are unique inside a row, so the result is deterministic whatever order the atomics ran in).
__global__ void k_tr_count(const int *col, int nnz, int *cnt)
{
   int k = blockIdx.x * blockDim.x + threadIdx.x;
   if (k < nnz) atomicAdd(cnt + col[k], 1);
}
__global__ void k_tr_place(const int *rp, const int *col, const double *val, int n, const int *trp, int *cursor, int *tcol, double *tval)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   for (int k = rp[i]; k < rp[i + 1]; k++)
   {
      int c = col[k];
      int p = trp[c] + atomicAdd(cursor + c, 1);
      tcol[p] = i;
      if (val) tval[p] = val[k];
   }
}
__global__ void k_tr_sort_rows(const int *trp, int nrows, int *tcol, double *tval)
{
   int r = blockIdx.x * blockDim.x + threadIdx.x;
   if (r >= nrows) return;
   int b = trp[r], e = trp[r + 1];
   for (int a = b + 1; a < e; a++)
   {
      int    c = tcol[a];
      double v = tval ? tval[a] : 0.0;
      int    j = a - 1;
      while (j >= b && tcol[j] > c) { tcol[j + 1] = tcol[j]; if (tval) tval[j + 1] = tval[j]; j--; }
      tcol[j + 1] = c;
      if (tval) tval[j + 1] = v;
   }
}

int csr_transpose(const DevCSR &A, DevCSR &T)
{
   int nnz = A.nnz;
   HDK_TRY(csr_alloc(T, A.ncols, A.nrows, nnz, A.val != nullptr));
   if (nnz == 0) { HDK_CUDA(cudaMemsetAsync(T.rowptr, 0, sizeof(int) * ((size_t)T.nrows + 1), g.stream)); return HDK_OK; }
   int *cnt, *cursor;
   HDK_TRY(dalloc(&cnt, (size_t)T.nrows + 1));
   HDK_TRY(dalloc(&cursor, (size_t)T.nrows + 1));
   HDK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)T.nrows + 1), g.stream));
   HDK_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)T.nrows + 1), g.stream));
   k_tr_count<<<cdiv(nnz, 256), 256, 0, g.stream>>>(A.col, nnz, cnt);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_int(cnt, T.rowptr, T.nrows + 1));
   k_tr_place<<<cdiv(A.nrows, 256), 256, 0, g.stream>>>(A.rowptr, A.col, A.val, A.nrows, T.rowptr, cursor, T.col, T.val);
   HDK_LAUNCH_CHECK();
   k_tr_sort_rows<<<cdiv(T.nrows, 128), 128, 0, g.stream>>>(T.rowptr, T.nrows, T.col, T.val);
   HDK_LAUNCH_CHECK();
   dfree(cnt); dfree(cursor);
   return HDK_OK;
}

// =====================================================================================
// Galerkin product (hypre_BoomerAMGBuildCoarseOperatorKT order): one thread per coarse row,
// hash accumulators in scratch; row = diagonal first, then columns in discovery order of
// (i1 in R_ic) x (i2 in A_i1) x (i3 in P_i2); value = sum (r*a)*p in that order.
// =====================================================================================
// ---- warp-per-row Galerkin product with shared-memory hash accumulators -------------------
// A warp walks the product stream of one coarse row in hypre's loop order, 32 products at a
// time.  Lanes that hit the same column in one chunk are grouped with match.any; the group
// leader inserts / looks up the column (new columns get slots in lane order = discovery
// order) and adds the group's products in lane order, so both the column order and every
// floating-point sum equal the sequential loop bit for bit.
constexpr int RW_CAP   = 512;  // hash slots per warp
constexpr int RW_LIMIT = 320;  // longest row handled here; longer rows fall back to k_rap_count/fill
constexpr int RW_WARPS = 8;

// BUMP (single-pass product): the finished row goes to a bump-allocated position of a staging buffer
// (one atomicAdd per row) and cnt / rowoff record its length and position; rows that do not fit this
// table size are flagged (cnt = -1) for the next larger table, a full staging buffer is reported as
// cnt = -2 (the host then falls back to the two-pass product).
template <bool FILL, int CAP, bool BUMP = false>
__global__ void __launch_bounds__(32 * RW_WARPS) k_rap_warp(const int *rrp, const int *rcol, const double *rval,
                                                            const int *arp, const int *acol, const double *aval,
                                                            const int *prp, const int *pcol, const double *pval,
                                                            int nc, int *cnt, const int *crp, int *ccol, double *cval,
                                                            int row_lo, int len_lo, int len_hi,
                                                            unsigned long long *bump_cursor = nullptr, long long bump_cap = 0,
                                                            long long *rowoff = nullptr, int only_flagged = 0)
{
   extern __shared__ __align__(16) unsigned char rw_smem[];
   const int      lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
   const unsigned FULL = 0xffffffffu;
   const int      ic = row_lo + blockIdx.x * RW_WARPS + wid; // rows [row_lo, nc)
   if (ic >= nc) return;
   constexpr int LIMIT = BUMP ? (((CAP * 5) / 8 < RW_LIMIT) ? (CAP * 5) / 8 : RW_LIMIT) : RW_LIMIT; // longest row this table takes
   if (FILL && !BUMP) { const int c = cnt[ic]; if (c > RW_LIMIT || c <= len_lo || c > len_hi) return; } // rows of this table size
   if (BUMP && only_flagged && cnt[ic] != -1) return;                                             // rows the smaller table gave up on
   int    *keys = reinterpret_cast<int *>(rw_smem) + (size_t)wid * CAP;
   int    *idx  = reinterpret_cast<int *>(rw_smem) + (size_t)RW_WARPS * CAP + (size_t)wid * CAP;
   double *vals = reinterpret_cast<double *>(rw_smem + (size_t)2 * RW_WARPS * CAP * sizeof(int)) + (size_t)wid * CAP;
   for (int h = lane; h < CAP; h += 32) keys[h] = -1;
   __syncwarp();
   int  count = 1;
   bool overflow = false;
   if (lane == 0)
   {
      bool nw;
      int  h = wt_find_or_insert(keys, CAP, ic, nw);
      if (FILL) { idx[h] = 0; vals[h] = 0.0; }
   }
   __syncwarp();
   // The loop nest is hypre's (R row -> A rows -> P rows) and is walked in its order, 32 entries
   // of an A row ("chunk") at a time.  Latency hiding: the R row with the bounds of its A rows is
   // fetched 32 entries at once and broadcast by shuffles, and the operands of chunk k+1 (A
   // entries and their P row bounds) are loaded before chunk k is processed.
   const int rend = rrp[ic + 1];
   for (int rb = rrp[ic]; rb < rend && !overflow; rb += 32)
   {
      const int    jr = rb + lane;
      const bool   vr = jr < rend;
      const int    p_i1 = vr ? rcol[jr] : 0;
      const double p_r  = (FILL && vr) ? rval[jr] : 0.0;
      const int    p_a0 = vr ? arp[p_i1] : 0, p_a1 = vr ? arp[p_i1 + 1] : 0;
      const int    nR = (rend - rb) < 32 ? (rend - rb) : 32;
      int          t = 0, base = __shfl_sync(FULL, p_a0, 0);
      // operands of the current chunk
      int    i2, ps, pl;
      double ra;
      {
         const int    a1 = __shfl_sync(FULL, p_a1, 0);
         const double r  = __shfl_sync(FULL, p_r, 0);
         const int    j2 = base + lane;
         const bool   v2 = j2 < a1;
         i2 = v2 ? acol[j2] : 0;
         ra = (FILL && v2) ? __dmul_rn(r, aval[j2]) : 0.0;
         ps = v2 ? prp[i2] : 0;
         pl = v2 ? prp[i2 + 1] - ps : 0;
      }
      while (t < nR && !overflow)
      {
         // coordinates and operands of the next chunk
         int nt = t, nbase = base + 32;
         if (nbase >= __shfl_sync(FULL, p_a1, t)) { nt = t + 1; nbase = __shfl_sync(FULL, p_a0, nt & 31); }
         int    n_i2 = 0, n_ps = 0, n_pl = 0;
         double n_ra = 0.0;
         if (nt < nR)
         {
            const int    a1 = __shfl_sync(FULL, p_a1, nt);
            const double r  = __shfl_sync(FULL, p_r, nt);
            const int    j2 = nbase + lane;
            const bool   v2 = j2 < a1;
            n_i2 = v2 ? acol[j2] : 0;
            n_ra = (FILL && v2) ? __dmul_rn(r, aval[j2]) : 0.0;
            n_ps = v2 ? prp[n_i2] : 0;
            n_pl = v2 ? prp[n_i2 + 1] - n_ps : 0;
         }
         // process the current chunk
         int incl = pl;
#pragma unroll
         for (int o = 1; o < 32; o <<= 1) { int u = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += u; }
         const int excl = incl - pl, Tc = __shfl_sync(FULL, incl, 31);
         for (int q0 = 0; q0 < Tc; q0 += 32)
         {
            const int  q = q0 + lane;
            const bool act = q < Tc;
            int lo = 0, hi = 31; // smallest m with incl[m] > q
#pragma unroll
            for (int s = 0; s < 5; s++)
            {
               int mid = (lo + hi) >> 1;
               int v   = __shfl_sync(FULL, incl, mid);
               if (v > q) hi = mid; else lo = mid + 1;
            }
            const int    m   = lo;
            const int    j3  = q - __shfl_sync(FULL, excl, m);
            const int    psm = __shfl_sync(FULL, ps, m);
            const double ram = __shfl_sync(FULL, ra, m);
            const int    key = act ? pcol[psm + j3] : (-2 - lane);
            const double rap = (FILL && act) ? __dmul_rn(ram, pval[psm + j3]) : 0.0;
            const unsigned grp = __match_any_sync(FULL, key);
            const bool leader = act && (lane == __ffs(grp) - 1);
            bool isnew = false;
            int  h = 0;
            if (leader) h = wt_find_or_insert(keys, CAP, key, isnew);
            const unsigned newmask = __ballot_sync(FULL, leader && isnew);
            if (FILL && leader && isnew) idx[h] = count + __popc(newmask & ((1u << lane) - 1u));
            count += __popc(newmask);
            if (count > LIMIT) overflow = true;
            if (FILL)
            {
               const int maxc = (int)__reduce_max_sync(FULL, leader ? (unsigned)__popc(grp) : 0u);
               double    acc = 0.0;
               bool      first = true;
               unsigned  rem = leader ? grp : 0u;
               for (int s = 0; s < maxc; s++)
               {
                  int    src = rem ? (__ffs(rem) - 1) : lane;
                  double v   = __shfl_sync(FULL, rap, src);
                  if (rem)
                  {
                     if (first) { acc = isnew ? v : __dadd_rn(vals[h], v); first = false; }
                     else acc = __dadd_rn(acc, v);
                     rem &= rem - 1u;
                  }
               }
               if (leader) vals[h] = acc;
            }
            __syncwarp();
            if (overflow) break;
         }
         t = nt; base = nbase;
         i2 = n_i2; ra = n_ra; ps = n_ps; pl = n_pl;
      }
   }
   if (!FILL) { if (lane == 0) cnt[ic] = overflow ? -1 : count; return; }
   if (BUMP)
   {
      if (overflow) { if (lane == 0) cnt[ic] = -1; return; }
      long long off = 0;
      if (lane == 0) off = (long long)atomicAdd(bump_cursor, (unsigned long long)count);
      off = __shfl_sync(FULL, off, 0);
      if (off + count > bump_cap) { if (lane == 0) cnt[ic] = -2; return; }
      for (int h = lane; h < CAP; h += 32)
         if (keys[h] >= 0) { int s = idx[h]; ccol[off + s] = keys[h]; cval[off + s] = vals[h]; }
      if (lane == 0) { cnt[ic] = count; rowoff[ic] = off; }
      return;
   }
   const int b = crp[ic];
   for (int h = lane; h < CAP; h += 32)
      if (keys[h] >= 0) { int s = idx[h]; ccol[b + s] = keys[h]; cval[b + s] = vals[h]; }
}

// staging buffer -> final CSR position (one warp per row; rows longer than RW_LIMIT come from k_rap_fill)
__global__ void k_rap_compact(const int *cnt, const long long *rowoff, const int *crp, const int *bcol, const double *bval,
                              int row_lo, int row_hi, int *ccol, double *cval)
{
   const int lane = threadIdx.x & 31;
   const int ic = row_lo + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
   if (ic >= row_hi) return;
   const int c = cnt[ic];
   if (c <= 0 || c > RW_LIMIT) return;
   const long long o = rowoff[ic];
   const int       b = crp[ic];
   for (int k = lane; k < c; k += 32) { ccol[b + k] = bcol[o + k]; cval[b + k] = bval[o + k]; }
}
__global__ void k_any_equal(const int *v, int n, int key, int *out)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i < n && v[i] == key) *out = 1;
}

__global__ void k_max_int(const int *v, int n, int *out)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   int m = i < n ? v[i] : 0;
   for (int o = 16; o > 0; o >>= 1) { int t = __shfl_down_sync(0xffffffffu, m, o); m = t > m ? t : m; }
   if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

__global__ void k_rap_q(const int *arp, const int *acol, const int *prp, int n, int *q)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   int s = 0;
   for (int k = arp[i]; k < arp[i + 1]; k++) { int j = acol[k]; s += prp[j + 1] - prp[j]; }
   q[i] = s;
}
__global__ void k_rap_cap(const int *rrp, const int *rcol, const int *q, int nc, int *cap, const int *cnt)
{
   int ic = blockIdx.x * blockDim.x + threadIdx.x;
   if (ic > nc) return;
   if (ic == nc || cnt[ic] != -1) { cap[ic] = 0; return; } // only rows the warp kernel gave up on
   long long ub = 1;
   for (int k = rrp[ic]; k < rrp[ic + 1]; k++) ub += q[rcol[k]];
   if (ub > nc) ub = nc;
   cap[ic] = pow2ceil((int)(2 * ub));
}
__global__ void k_rap_count(const int *rrp, const int *rcol, const int *arp, const int *acol, const int *prp,
                            const int *pcol, int row0, int row1, const int64_t *off, int *keys, int *cnt)
{
   int ic = row0 + blockIdx.x * blockDim.x + threadIdx.x;
   if (ic >= row1) return;
   int *tab = keys + (off[ic] - off[row0]);
   int  cap = (int)(off[ic + 1] - off[ic]);
   if (cap == 0) return;
   int  c   = 1;
   hset_insert(tab, cap, ic);
   for (int j1 = rrp[ic]; j1 < rrp[ic + 1]; j1++)
   {
      int i1 = rcol[j1];
      for (int j2 = arp[i1]; j2 < arp[i1 + 1]; j2++)
      {
         int i2 = acol[j2];
         for (int j3 = prp[i2]; j3 < prp[i2 + 1]; j3++)
            if (hset_insert(tab, cap, pcol[j3])) c++;
      }
   }
   cnt[ic] = c;
}
__global__ void k_rap_cap2(const int *cnt, int nc, int *cap2, int lo, int hi)
{
   int ic = blockIdx.x * blockDim.x + threadIdx.x;
   if (ic > nc) return;
   cap2[ic] = (ic >= lo && ic < hi && cnt[ic] > RW_LIMIT) ? pow2ceil(2 * cnt[ic]) : 0; // rows too long for the warp kernel
}
__global__ void k_rap_fill(const int *rrp, const int *rcol, const double *rval, const int *arp, const int *acol,
                           const double *aval, const int *prp, const int *pcol, const double *pval, int row0,
                           int row1, const int64_t *off, int2 *htab, const int *crp, int *ccol, double *cval)
{
   int ic = row0 + blockIdx.x * blockDim.x + threadIdx.x;
   if (ic >= row1) return;
   int2 *tab = htab + (off[ic] - off[row0]);
   int   cap = (int)(off[ic + 1] - off[ic]);
   if (cap == 0) return;
   int   b = crp[ic], c = b;
   hmap_insert(tab, cap, ic, c);
   ccol[c] = ic; cval[c] = 0.0; c++;
   for (int j1 = rrp[ic]; j1 < rrp[ic + 1]; j1++)
   {
      int    i1 = rcol[j1];
      double r  = rval[j1];
      for (int j2 = arp[i1]; j2 < arp[i1 + 1]; j2++)
      {
         int    i2 = acol[j2];
         double ra = __dmul_rn(r, aval[j2]);
         for (int j3 = prp[i2]; j3 < prp[i2 + 1]; j3++)
         {
            int    i3  = pcol[j3];
            double rap = __dmul_rn(ra, pval[j3]);
            int    m   = hmap_insert(tab, cap, i3, c);
            if (m == -1) { ccol[c] = i3; cval[c] = rap; c++; }
            else cval[m] = __dadd_rn(cval[m], rap);
         }
      }
   }
}

// coarse rows [row_lo, row_hi) only (row_lo < 0: all rows, or this rank's share of a work-shared global level)
int build_rap(const DevCSR &R, const DevCSR &A, const DevCSR &P, DevCSR &C, int row_lo, int row_hi)
{
   stage_mark(nullptr, -1);
   int nc = R.nrows, n = A.nrows;
   if (row_lo >= 0 && row_hi <= row_lo)
   {
      // no row to compute here (a rank of the distributed setup that owns no coarse point)
      HDK_TRY(csr_alloc(C, nc, nc, 0));
      HDK_CUDA(cudaMemsetAsync(C.rowptr, 0, sizeof(int) * ((size_t)nc + 1), g.stream));
      return HDK_OK;
   }
   int *q, *cap, *cnt, *crp;
   int64_t *off;
   HDK_TRY(dalloc(&q, (size_t)n + 1));
   HDK_TRY(dalloc(&cap, (size_t)nc + 1));
   HDK_TRY(dalloc(&cnt, (size_t)nc + 1));
   HDK_TRY(dalloc(&crp, (size_t)nc + 1));
   HDK_TRY(dalloc(&off, (size_t)nc + 1));
   k_rap_q<<<cdiv(n, 256), 256, 0, g.stream>>>(A.rowptr, A.col, P.rowptr, n, q);
   HDK_LAUNCH_CHECK();
   // this rank's share of the coarse rows (all of them unless the multi-rank setup shares the work)
   int lo, hi;
   share_range(nc, lo, hi);
   if (row_lo >= 0) { lo = row_lo; hi = row_hi; }
   if (share_on(nc) || lo != 0 || hi != nc) HDK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)nc + 1), g.stream));
   // Single-pass product (default; HDK_RAP_SINGLE=0 selects count + fill): every row is computed ONCE into
   // a staging buffer, 256-slot tables first, the rows those cannot hold with 512-slot tables; the
   // row lengths fall out of the same pass, then the rows are copied to their CSR position.  Rows
   // longer than RW_LIMIT take the one-thread-per-row path below either way.
   static int rap_single = -1;
   if (rap_single < 0) { const char *e = getenv("HDK_RAP_SINGLE"); rap_single = (e && atoi(e) == 0) ? 0 : 1; }
   int       *bcol = nullptr;
   double    *bval = nullptr;
   long long *rowoff = nullptr;
   bool       single = rap_single == 1;
   if (single)
   {
      const long long bump_cap = 2LL * (long long)A.nnz + (1LL << 22);
      unsigned long long *cursor = reinterpret_cast<unsigned long long *>(g.dscal + S_TMP2);
      int *flag = reinterpret_cast<int *>(g.dscal + S_TMP3);
      if (bump_cap > 2000000000LL) single = false;
      if (single)
      {
         static bool attr_b = false;
         if (!attr_b)
         {
            HDK_CUDA(cudaFuncSetAttribute(k_rap_warp<true, 256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RW_WARPS * 256 * 16));
            HDK_CUDA(cudaFuncSetAttribute(k_rap_warp<true, RW_CAP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, RW_WARPS * RW_CAP * 16));
            attr_b = true;
         }
         HDK_TRY(dalloc(&bcol, (size_t)bump_cap + 8));
         HDK_TRY(dalloc(&bval, (size_t)bump_cap + 8));
         HDK_TRY(dalloc(&rowoff, (size_t)nc + 1));
         HDK_CUDA(cudaMemsetAsync(cursor, 0, sizeof(unsigned long long), g.stream));
         HDK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), g.stream));
         const int nb = cdiv(hi - lo, RW_WARPS);
         k_rap_warp<true, 256, true><<<nb, 32 * RW_WARPS, (size_t)RW_WARPS * 256 * 16, g.stream>>>(
            R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, nullptr, bcol, bval, lo, 0, 0,
            cursor, bump_cap, rowoff, 0);
         HDK_LAUNCH_CHECK();
         k_any_equal<<<cdiv(hi - lo, 256), 256, 0, g.stream>>>(cnt + lo, hi - lo, -1, flag);
         HDK_LAUNCH_CHECK();
         int hflag = 0;
         HDK_CUDA(cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
         HDK_CUDA(cudaStreamSynchronize(g.stream));
         if (hflag)
         {
            k_rap_warp<true, RW_CAP, true><<<nb, 32 * RW_WARPS, (size_t)RW_WARPS * RW_CAP * 16, g.stream>>>(
               R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, nullptr, bcol, bval, lo, 0, 0,
               cursor, bump_cap, rowoff, 1);
            HDK_LAUNCH_CHECK();
         }
         // staging buffer exhausted somewhere? then start over with the two-pass product
         HDK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), g.stream));
         k_any_equal<<<cdiv(hi - lo, 256), 256, 0, g.stream>>>(cnt + lo, hi - lo, -2, flag);
         HDK_LAUNCH_CHECK();
         HDK_CUDA(cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
         HDK_CUDA(cudaStreamSynchronize(g.stream));
         if (hflag)
         {
            single = false;
            dfree(bcol); dfree(bval); dfree(rowoff);
            bcol = nullptr; bval = nullptr; rowoff = nullptr;
            if (lo != 0 || hi != nc) HDK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * ((size_t)nc + 1), g.stream));
         }
      }
      stage_mark("  rap.single", -1);
   }
   if (!single)
   {
      // pass 1a: exact row lengths by the warp kernel (rows longer than RW_LIMIT are flagged -1)
      k_rap_warp<false, RW_CAP><<<cdiv(hi - lo, RW_WARPS), 32 * RW_WARPS, (size_t)RW_WARPS * RW_CAP * sizeof(int), g.stream>>>(
         R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, nullptr, nullptr, nullptr, lo, 0, 0);
      HDK_LAUNCH_CHECK();
      stage_mark("  rap.warp1", -1);
   }
   // pass 1b: flagged rows through the one-thread-per-row kernel with hash sets in global scratch
   k_rap_cap<<<cdiv(nc + 1, 256), 256, 0, g.stream>>>(R.rowptr, R.col, q, nc, cap, cnt);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_i64(cap, off, nc + 1));
   std::vector<int> bounds;
   int64_t          maxsz;
   HDK_TRY(plan_chunks(off, nc, bounds, maxsz));
   {
      int *keys;
      HDK_TRY(dalloc(&keys, (size_t)maxsz + 4));
      for (size_t c = 0; c + 1 < bounds.size(); c++)
      {
         int r0 = bounds[c], r1 = bounds[c + 1];
         if (r1 <= r0) continue;
         HDK_CUDA(cudaMemsetAsync(keys, 0xFF, sizeof(int) * ((size_t)maxsz + 4), g.stream));
         k_rap_count<<<cdiv(r1 - r0, 128), 128, 0, g.stream>>>(R.rowptr, R.col, A.rowptr, A.col, P.rowptr, P.col, r0, r1, off, keys, cnt);
         HDK_LAUNCH_CHECK();
      }
      dfree(keys);
   }
   stage_mark("  rap.thr1", -1);
   HDK_CUDA(cudaMemsetAsync(cnt + nc, 0, sizeof(int), g.stream));
   HDK_TRY(share_rows(cnt, sizeof(int), nc)); // row lengths of the other ranks' shares
   HDK_TRY(check_fits_int32(cnt, nc, "the coarse-grid operator"));
   HDK_TRY(exclusive_scan_int(cnt, crp, nc + 1));
   int nnzC = 0;
   HDK_CUDA(cudaMemcpyAsync(&nnzC, crp + nc, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   C = DevCSR();
   C.nrows = nc; C.ncols = nc; C.nnz = nnzC; C.rowptr = crp; C.owns = true;
   HDK_TRY(dalloc(&C.col, (size_t)nnzC + 8));
   HDK_TRY(dalloc(&C.val, (size_t)nnzC + 8));
   HDK_CUDA(cudaMemsetAsync(C.col + nnzC, 0, sizeof(int) * 8, g.stream));
   HDK_CUDA(cudaMemsetAsync(C.val + nnzC, 0, sizeof(double) * 8, g.stream));
   if (single)
   {
      k_rap_compact<<<cdiv(hi - lo, 8), 256, 0, g.stream>>>(cnt, rowoff, crp, bcol, bval, lo, hi, C.col, C.val);
      HDK_LAUNCH_CHECK();
      dfree(bcol); dfree(bval); dfree(rowoff);
      stage_mark("  rap.compact", -1);
   }
   else
   {
      // small tables (more resident warps) when every row of the level is short
      int *dmax = reinterpret_cast<int *>(g.dscal + S_TMP3), hmax = 0;
      HDK_CUDA(cudaMemsetAsync(dmax, 0, sizeof(int), g.stream));
      k_max_int<<<cdiv(nc, 256), 256, 0, g.stream>>>(cnt, nc, dmax);
      HDK_LAUNCH_CHECK();
      HDK_CUDA(cudaMemcpyAsync(&hmax, dmax, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
      HDK_CUDA(cudaStreamSynchronize(g.stream));
      static bool attr = false;
      size_t      smem = (size_t)RW_WARPS * RW_CAP * (2 * sizeof(int) + sizeof(double));
      if (!attr) { HDK_CUDA(cudaFuncSetAttribute(k_rap_warp<true, RW_CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); attr = true; }
      // the table size is a static share of shared memory, so it sets the occupancy: rows are
      // served by the smallest table that holds them (load factor <= 5/8), one launch per size
      static bool attr256 = false;
      if (!attr256) { HDK_CUDA(cudaFuncSetAttribute(k_rap_warp<true, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, RW_WARPS * 256 * 16)); attr256 = true; }
      const int nb = cdiv(hi - lo, RW_WARPS);
      k_rap_warp<true, 128><<<nb, 32 * RW_WARPS, (size_t)RW_WARPS * 128 * 16, g.stream>>>(
         R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, crp, C.col, C.val, lo, 0, 80);
      HDK_LAUNCH_CHECK();
      if (hmax > 80)
      {
         k_rap_warp<true, 256><<<nb, 32 * RW_WARPS, (size_t)RW_WARPS * 256 * 16, g.stream>>>(
            R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, crp, C.col, C.val, lo, 80, 160);
         HDK_LAUNCH_CHECK();
      }
      if (hmax > 160)
         k_rap_warp<true, RW_CAP><<<nb, 32 * RW_WARPS, smem, g.stream>>>(
            R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col, P.val, hi, cnt, crp, C.col, C.val, lo, 160, RW_LIMIT);
      HDK_LAUNCH_CHECK();
      stage_mark("  rap.warp2", -1);
   }
   k_rap_cap2<<<cdiv(nc + 1, 256), 256, 0, g.stream>>>(cnt, nc, cap, lo, hi);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_i64(cap, off, nc + 1));
   HDK_TRY(plan_chunks(off, nc, bounds, maxsz));
   {
      int2 *htab;
      HDK_TRY(dalloc(&htab, (size_t)maxsz + 4));
      for (size_t c = 0; c + 1 < bounds.size(); c++)
      {
         int r0 = bounds[c], r1 = bounds[c + 1];
         if (r1 <= r0) continue;
         HDK_CUDA(cudaMemsetAsync(htab, 0xFF, sizeof(int2) * ((size_t)maxsz + 4), g.stream));
         k_rap_fill<<<cdiv(r1 - r0, 128), 128, 0, g.stream>>>(R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, P.rowptr, P.col,
                                                             P.val, r0, r1, off, htab, crp, C.col, C.val);
         HDK_LAUNCH_CHECK();
      }
      dfree(htab);
   }
   HDK_TRY(share_entries(crp, nc, C.col, sizeof(int), C.val, sizeof(double)));
   dfree(q); dfree(cap); dfree(cnt); dfree(off);
   return HDK_OK;
}

// =====================================================================================
// l1 norms (hypre_ParCSRComputeL1Norms): option 1 full row l1 norm (relax 18);
// option 4 truncated l1 = |a_ii| + 0.5*sum_offd|a_ij| (relax 8/13/14); option 5 diagonal
// =====================================================================================
__global__ void k_l1(const int *rp, const double *val, const int *orp, const double *oval, int n, int option, double *l1)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   int    b = rp[i], e = rp[i + 1];
   double d = e > b ? val[b] : 0.0, v;
   if (option == 1)
   {
      v = 0.0;
      for (int k = b; k < e; k++) v = __dadd_rn(v, fabs(val[k]));
      if (orp) for (int k = orp[i]; k < orp[i + 1]; k++) v = __dadd_rn(v, fabs(oval[k]));
      if (d < 0) v = -v;
   }
   else if (option == 4)
   {
      double od = 0.0;
      if (orp) for (int k = orp[i]; k < orp[i + 1]; k++) od = __dadd_rn(od, fabs(oval[k]));
      v = __dadd_rn(fabs(d), __dmul_rn(0.5, od));
      if (v <= (4.0 / 3.0) * fabs(d)) v = fabs(d);
      if (d < 0) v = -v;
   }
   else v = d;
   l1[i] = v;
}

static int relax_l1_option(int type)
{
   if (type == 18) return 1;
   if (type == 8 || type == 13 || type == 14) return 4;
   return 5;
}

static int build_l1(const hdk_csr_s &A, int option, double **out)
{
   int n = A.diag.nrows;
   HDK_TRY(dalloc(out, (size_t)n + 8));
   const int    *orp = A.offd.nnz > 0 ? A.offd.rowptr : nullptr;
   const double *ov  = A.offd.nnz > 0 ? A.offd.val : nullptr;
   k_l1<<<cdiv(n, 256), 256, 0, g.stream>>>(A.diag.rowptr, A.diag.val, orp, ov, n, option, *out);
   HDK_LAUNCH_CHECK();
   return HDK_OK;
}

// strict lower triangle (two-stage Gauss-Seidel)
template <bool FILL>
__global__ void k_lower(const int *rp, const int *col, const double *val, int n, int *cnt, const int *lrp, int *lcol, double *lval)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i > n) return;
   if (i == n) { if (!FILL) cnt[n] = 0; return; }
   int c = 0, p = FILL ? lrp[i] : 0;
   for (int k = rp[i]; k < rp[i + 1]; k++)
      if (col[k] < i) { if (FILL) { lcol[p] = col[k]; lval[p] = val[k]; p++; } else c++; }
   if (!FILL) cnt[i] = c;
}

static int build_lower(const DevCSR &A, DevCSR &L)
{
   int  n = A.nrows;
   int *cnt, *lrp;
   HDK_TRY(dalloc(&cnt, (size_t)n + 1));
   HDK_TRY(dalloc(&lrp, (size_t)n + 1));
   k_lower<false><<<cdiv(n + 1, 256), 256, 0, g.stream>>>(A.rowptr, A.col, A.val, n, cnt, nullptr, nullptr, nullptr);
   HDK_LAUNCH_CHECK();
   HDK_TRY(exclusive_scan_int(cnt, lrp, n + 1));
   int nnz = 0;
   HDK_CUDA(cudaMemcpyAsync(&nnz, lrp + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   dfree(cnt);
   HDK_TRY(csr_alloc(L, n, n, nnz));
   dfree(L.rowptr); L.rowptr = lrp;
   k_lower<true><<<cdiv(n + 1, 256), 256, 0, g.stream>>>(A.rowptr, A.col, A.val, n, nullptr, lrp, L.col, L.val);
   HDK_LAUNCH_CHECK();
   return csr_analyze(L);
}

// =====================================================================================
// coarsest level: dense inverse by Gauss-Jordan with partial pivoting (one CTA up to GJ_ONE_CTA rows)
// =====================================================================================
__global__ void k_dense_fill(const int *rp, const int *col, const double *val, int n, double *M /* n x 2n */)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i >= n) return;
   for (int k = rp[i]; k < rp[i + 1]; k++) M[(size_t)i * 2 * n + col[k]] += val[k];
   M[(size_t)i * 2 * n + n + i] = 1.0;
}

__global__ void __launch_bounds__(1024) k_gauss_jordan(double *M, int n, double *inv)
{
   __shared__ double sval[32];
   __shared__ int    sidx[32];
   __shared__ int    piv;
   __shared__ double pivval;
   const int tid = threadIdx.x, nt = blockDim.x, w = 2 * n;
   for (int k = 0; k < n; k++)
   {
      // pivot search in column k
      double best = -1.0; int bi = k;
      for (int r = k + tid; r < n; r += nt) { double v = fabs(M[(size_t)r * w + k]); if (v > best) { best = v; bi = r; } }
      for (int o = 16; o > 0; o >>= 1)
      {
         double ov = __shfl_down_sync(0xffffffffu, best, o); int oi = __shfl_down_sync(0xffffffffu, bi, o);
         if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
      }
      if ((tid & 31) == 0) { sval[tid >> 5] = best; sidx[tid >> 5] = bi; }
      __syncthreads();
      if (tid == 0)
      {
         double b = sval[0]; int i2 = sidx[0];
         for (int q = 1; q < (nt + 31) / 32; q++) if (sval[q] > b || (sval[q] == b && sidx[q] < i2)) { b = sval[q]; i2 = sidx[q]; }
         piv = i2; pivval = M[(size_t)i2 * w + k];
      }
      __syncthreads();
      int    pr = piv;
      double pv = pivval;
      if (pv != 0.0)
      {
         if (pr != k)
            for (int j = tid; j < w; j += nt) { double t = M[(size_t)k * w + j]; M[(size_t)k * w + j] = M[(size_t)pr * w + j]; M[(size_t)pr * w + j] = t; }
         __syncthreads();
         for (int j = tid; j < w; j += nt) M[(size_t)k * w + j] /= pv;
         __syncthreads();
         // eliminate column k from every other row
         for (int idx = tid; idx < n * w; idx += nt)
         {
            int r = idx / w, j = idx - r * w;
            if (r != k && j != k)
            {
               double f = M[(size_t)r * w + k];
               if (f != 0.0) M[(size_t)r * w + j] -= f * M[(size_t)k * w + j];
            }
         }
         __syncthreads();
         for (int r = tid; r < n; r += nt) if (r != k) M[(size_t)r * w + k] = 0.0;
      }
      __syncthreads();
   }
   for (int idx = tid; idx < n * n; idx += nt) { int r = idx / n, j = idx - r * n; inv[idx] = M[(size_t)r * w + n + j]; }
}

// The same elimination for coarsest operators of more than GJ_ONE_CTA rows, two launches per pivot
// step over the whole grid: k_gj_pivot (one CTA) picks, swaps and scales the pivot row and saves
// the multipliers of column k in f; k_gj_eliminate updates every other row.  Each entry sees the
// same operations in the same order as in k_gauss_jordan.  Left of column k the pivot row is zero.
constexpr int GJ_ONE_CTA = 1024;
__global__ void __launch_bounds__(1024) k_gj_pivot(double *M, int n, int k, double *f)
{
   __shared__ double sval[32];
   __shared__ int    sidx[32];
   __shared__ int    piv;
   __shared__ double pivval;
   const int tid = threadIdx.x, nt = blockDim.x, w = 2 * n;
   double best = -1.0; int bi = k;
   for (int r = k + tid; r < n; r += nt) { double v = fabs(M[(size_t)r * w + k]); if (v > best) { best = v; bi = r; } }
   for (int o = 16; o > 0; o >>= 1)
   {
      double ov = __shfl_down_sync(0xffffffffu, best, o); int oi = __shfl_down_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
   }
   if ((tid & 31) == 0) { sval[tid >> 5] = best; sidx[tid >> 5] = bi; }
   __syncthreads();
   if (tid == 0)
   {
      double b = sval[0]; int i2 = sidx[0];
      for (int q = 1; q < (nt + 31) / 32; q++) if (sval[q] > b || (sval[q] == b && sidx[q] < i2)) { b = sval[q]; i2 = sidx[q]; }
      piv = i2; pivval = M[(size_t)i2 * w + k];
   }
   __syncthreads();
   const int    pr = piv;
   const double pv = pivval;
   if (pv != 0.0)
   {
      if (pr != k)
         for (int j = tid; j < w; j += nt) { double t = M[(size_t)k * w + j]; M[(size_t)k * w + j] = M[(size_t)pr * w + j]; M[(size_t)pr * w + j] = t; }
      __syncthreads();
      for (int j = tid; j < w; j += nt) M[(size_t)k * w + j] /= pv;
   }
   // a zero pivot column leaves the step out: no multipliers
   for (int r = tid; r < n; r += nt) f[r] = (pv != 0.0 && r != k) ? M[(size_t)r * w + k] : 0.0;
}

__global__ void k_gj_eliminate(double *M, int n, int k, const double *f)
{
   const int    r = blockIdx.y, w = 2 * n;
   const double fr = f[r];
   if (fr == 0.0) return; // (also the pivot row)
   for (int j = k + blockIdx.x * blockDim.x + threadIdx.x; j < w; j += gridDim.x * blockDim.x)
   {
      if (j == k) M[(size_t)r * w + k] = 0.0;
      else M[(size_t)r * w + j] -= fr * M[(size_t)k * w + j];
   }
}

__global__ void k_gj_extract(const double *M, int n, double *inv)
{
   const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
   if (idx >= (int64_t)n * n) return;
   const int64_t r = idx / n, j = idx - r * n;
   inv[idx] = M[r * 2 * n + n + j];
}

static int build_dense_inverse(const DevCSR &A, double **inv)
{
   int     n = A.nrows;
   double *M;
   HDK_TRY(dalloc(&M, (size_t)n * 2 * n + 8));
   if (int rc = dalloc(inv, (size_t)n * n + 8)) { dfree(M); return rc; }
   HDK_CUDA(cudaMemsetAsync(M, 0, sizeof(double) * ((size_t)n * 2 * n), g.stream));
   k_dense_fill<<<cdiv(n, 128), 128, 0, g.stream>>>(A.rowptr, A.col, A.val, n, M);
   HDK_LAUNCH_CHECK();
   if (n <= GJ_ONE_CTA)
   {
      k_gauss_jordan<<<1, 1024, 0, g.stream>>>(M, n, *inv);
      HDK_LAUNCH_CHECK();
   }
   else
   {
      double *f;
      if (int rc = dalloc(&f, (size_t)n + 8)) { dfree(M); return rc; }
      for (int k = 0; k < n; k++)
      {
         k_gj_pivot<<<1, 1024, 0, g.stream>>>(M, n, k, f);
         k_gj_eliminate<<<dim3(cdiv(2 * n - k, 256), n), 256, 0, g.stream>>>(M, n, k, f);
      }
      HDK_LAUNCH_CHECK();
      k_gj_extract<<<(unsigned)(((int64_t)n * n + 255) / 256), 256, 0, g.stream>>>(M, n, *inv);
      HDK_LAUNCH_CHECK();
      dfree(f);
   }
   dfree(M);
   return HDK_OK;
}

// wrap a rank-local DevCSR as a ParCSR object with an empty offd block
hdk_csr_s *wrap_local(DevCSR &D, int64_t grows)
{
   hdk_csr_s *A  = new hdk_csr_s();
   A->row_start  = 0; A->row_end = (int64_t)D.nrows - 1; A->global_rows = grows; A->global_nnz = D.nnz;
   A->diag       = D;
   D             = DevCSR();
   return A;
}

void destroy_local(hdk_csr_s *A)
{
   if (!A) return;
   csr_free(A->diag); csr_free(A->offd);
   halo_plan_free(A->halo);
   dfree(A->offd_rows);
   delete A;
}

} // namespace hdk

using namespace hdk;

extern "C" {

void hdk_amg_default_params(hdk_amg_params *p)
{
   /* GPU-build defaults of the reference: src/internal/amg.c:120-238 under HYPRE_USING_GPU */
   p->coarsen_type = 8; p->strong_th = 0.25; p->max_row_sum = 0.9;
   p->max_coarse_size = 64; p->min_coarse_size = 0; p->max_levels = 25;
   p->interp_type = 6; p->max_nnz_row = 4; p->trunc_factor = 0.0;
   p->relax_down = 18; p->relax_up = 18; p->relax_coarse = 9;
   p->sweeps_down = p->sweeps_up = p->sweeps_coarse = 1;
   p->relax_weight = p->outer_weight = 1.0;
   p->rand_seed = 2747; p->keep_transpose = 1; p->print_level = 0;
}

int hdk_amg_destroy(hdk_amg *M)
{
   if (!M) return HDK_OK;
   if (g.inited)
   {
      for (auto &L : M->lev)
      {
         if (L.owns_A) destroy_local(L.A);
         destroy_local(L.P); destroy_local(L.R);
         csr_free(L.S); csr_free(L.L);
         dfree(L.cf); dfree(L.measure); dfree(L.f2c);
         if (L.l1_up != L.l1_down) dfree(L.l1_up);
         dfree(L.l1_down);
         dfree(L.u); dfree(L.f); dfree(L.t); dfree(L.gs1); dfree(L.gs2);
         for (int w = 0; w < 2; w++) { dfree(L.dbg_ip[w]); dfree(L.dbg_col[w]); dfree(L.dbg_val[w]); }
      }
      dfree(M->ge_inv); dfree(M->full_f); dfree(M->full_u);
      ipc_gather_free(M->gather);
      for (auto &G : M->graphs) if (G.exec) cudaGraphExecDestroy((cudaGraphExec_t)G.exec);
      M->graphs.clear();
   }
   if (M->tail) hdk_amg_destroy(M->tail);
   delete M;
   return HDK_OK;
}

// per-level solve data: smoother diagonals, work vectors, (two-stage GS) lower triangles, and the
// algorithmic byte count of one V-cycle
int finalize_levels(hdk_amg_s *M, const hdk_amg_params *prm, int64_t live_max_rows)
{
   int    rc = HDK_OK;
   double bytes = 0.0;
   for (int l = 0; l < M->nlev && rc == HDK_OK; l++)
   {
      AmgLevel &L = M->lev[(size_t)l];
      int       n = L.n;
      if (live_max_rows >= 0 && n > live_max_rows) continue; // global level that is only sliced, never cycled
      if ((rc = build_l1(*L.A, relax_l1_option(prm->relax_down), &L.l1_down))) break;
      if (relax_l1_option(prm->relax_up) == relax_l1_option(prm->relax_down)) L.l1_up = L.l1_down;
      else if ((rc = build_l1(*L.A, relax_l1_option(prm->relax_up), &L.l1_up))) break;
      if ((rc = dalloc(&L.t, (size_t)n + 8))) break;
      if (l > 0)
      {
         if ((rc = dalloc(&L.u, (size_t)n + 8))) break;
         if ((rc = dalloc(&L.f, (size_t)n + 8))) break;
      }
      bool tsgs = (prm->relax_down == 11 || prm->relax_down == 12 || prm->relax_up == 11 || prm->relax_up == 12);
      if (tsgs && (rc = build_lower(L.A->diag, L.L))) break;
      if (tsgs && ((rc = dalloc(&L.gs1, (size_t)n + 8)) || (rc = dalloc(&L.gs2, (size_t)n + 8)))) break;
      // algorithmic bytes of one V-cycle (DESIGN.md): zero-guess pre-smooth 24n, residual,
      // restriction, prolongation, post-smooth
      double nnzA = (double)L.A->diag.nnz + L.A->offd.nnz;
      if (L.P)
      {
         double nnzP = (double)L.P->diag.nnz + L.P->offd.nnz, ncl = (double)L.P->diag.ncols;
         bytes += 24.0 * n;                                       // u = w f / d
         bytes += 12.0 * nnzA + 4.0 * (n + 1) + 24.0 * n;         // r = f - A u
         bytes += 12.0 * nnzP + 4.0 * (ncl + 1) + 8.0 * n + 8.0 * ncl; // f_c = R r
         bytes += 12.0 * nnzP + 4.0 * (n + 1) + 16.0 * n + 8.0 * ncl;  // u += P e
         bytes += 12.0 * nnzA + 4.0 * (n + 1) + 32.0 * n;         // post-smooth
      }
      else bytes += 8.0 * (double)n * n + 16.0 * n;
   }
   M->vcycle_bytes = bytes;
   return rc;
}

// live_max_rows >= 0: the hierarchy is the global one of a multi-rank setup; levels with more
// rows are only sliced into slabs afterwards, so they get no SpMV analysis and no solve data
int setup_serial(const hdk_csr_s *A0, const hdk_amg_params *prm, hdk_amg_s **out, bool keep_f2c,
                 int64_t live_max_rows)
{
   hdk_amg_s *M = new hdk_amg_s();
   M->prm       = *prm;
   M->keep_f2c  = keep_f2c;
   M->keep_debug = tune_amg_keep_debug();
   int rc       = HDK_OK;
   M->lev.emplace_back();
   M->lev[0].A = const_cast<hdk_csr_s *>(A0);
   M->lev[0].owns_A = false;
   M->lev[0].n = A0->diag.nrows;
   int  level = 0;
   bool more  = prm->max_levels > 1;
   double nnz0 = (double)A0->diag.nnz + A0->offd.nnz, nnz_sum = nnz0;
   while (more && rc == HDK_OK)
   {
      AmgLevel        &L = M->lev[(size_t)level];
      const hdk_csr_s &A = *L.A;
      int              n = L.n;
      stage_mark(nullptr, level);
      if ((rc = build_strength(A, prm->strong_th, prm->max_row_sum, L.S))) break;
      stage_mark("strength", level);
      if ((rc = dalloc(&L.cf, (size_t)n + 1))) break;
      double *meas, *keep = nullptr;
      if ((rc = dalloc(&meas, (size_t)n + 1))) break;
      if (M->keep_debug) { if ((rc = dalloc(&keep, (size_t)n + 1))) break; }
      L.measure = keep;
      int64_t goff = (level == 0) ? A.row_start : 0;
      rc = run_pmis(L.S, prm->rand_seed, goff, L.cf, meas, keep, nullptr);
      stage_mark("pmis", level);
      dfree(meas);
      if (rc) break;
      int *flag, *f2c;
      if ((rc = dalloc(&flag, (size_t)n + 1))) break;
      if ((rc = dalloc(&f2c, (size_t)n + 1))) break;
      k_cf_flag<<<cdiv(n + 1, 256), 256, 0, g.stream>>>(L.cf, n, flag);
      g.launches++;
      if ((rc = exclusive_scan_int(flag, f2c, n + 1))) break;
      int nc = 0;
      cudaMemcpyAsync(&nc, f2c + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream);
      cudaStreamSynchronize(g.stream);
      dfree(flag);
      if (nc == 0 || nc == n || nc < prm->min_coarse_size) { dfree(f2c); break; }
      DevCSR P, R, C;
      rc = build_interp(A.diag, L.S, L.cf, f2c, nc, prm->max_nnz_row, prm->trunc_factor, P, -1, -1);
      stage_mark("interp", level);
      if (keep_f2c) L.f2c = f2c; else dfree(f2c);
      if (rc) break;
      if ((rc = csr_transpose(P, R))) break;
      stage_mark("transpose", level);
      if ((rc = build_rap(R, A.diag, P, C, -1, -1))) break;
      stage_mark("rap", level);
      C.coarse_op = true;
      if (live_max_rows < 0 || n <= live_max_rows)
      {
         if ((rc = csr_analyze(P))) break;
         if ((rc = csr_analyze(R))) break;
      }
      if (live_max_rows < 0 || nc <= live_max_rows)
      {
         if ((rc = csr_analyze(C))) break;
      }
      stage_mark("analyze", level);
      nnz_sum += C.nnz;
      L.P = wrap_local(P, n);
      L.R = wrap_local(R, nc);
      M->lev.emplace_back();
      AmgLevel &N = M->lev.back();
      N.A = wrap_local(C, nc); N.owns_A = true; N.n = nc;
      level++;
      if (level == prm->max_levels - 1 || nc <= prm->max_coarse_size) more = false;
      if (!M->keep_debug) csr_free(M->lev[(size_t)level - 1].S);
   }
   if (rc == HDK_OK)
   {
      M->nlev = level + 1;
      M->op_complexity = nnz_sum / (nnz0 > 0 ? nnz0 : 1.0);
      rc = finalize_levels(M, prm, live_max_rows);
   }
   if (rc == HDK_OK)
   {
      AmgLevel &Lc = M->lev[(size_t)M->nlev - 1];
      bool      want_ge = (prm->relax_coarse == 9 || prm->relax_coarse == 99 || prm->relax_coarse == 19);
      // hypre_GaussElimSetup builds the dense coarse matrix whatever its size; both this library and
      // the CPU oracle cap it at n^2 < 2e8 (1.6 GB, about 14 000 rows) and relax above that
      if (want_ge && (double)Lc.n * Lc.n < 2.0e8 && Lc.n > 0 && Lc.A->offd.nnz == 0)
      {
         rc = build_dense_inverse(Lc.A->diag, &M->ge_inv);
         M->ge_n = Lc.n;
      }
   }
   if (rc == HDK_OK) rc = (cudaStreamSynchronize(g.stream) == cudaSuccess) ? HDK_OK : set_error(HDK_ERR_CUDA, "setup sync failed: %s", cudaGetErrorString(cudaGetLastError()));
   if (rc != HDK_OK) { hdk_amg_destroy(M); return rc; }
   *out = M;
   return HDK_OK;
}

// ------------------------------------------------------------------------------------------
// N > 1.  Round-1 design: every rank reassembles the GLOBAL operator (NCCL broadcasts of the row
// slabs), runs the serial device setup on it -- so the hierarchy is bit-identical to the
// single-GPU one for any partition -- then keeps only its row slabs of A_l, P_l, R_l for the
// large levels (ParCSR with halo plans) and the complete small levels (replicated "tail").
// The solve phase is fully distributed; the setup does not scale yet (DESIGN.md section 5).
// ------------------------------------------------------------------------------------------
__global__ void k_shift_i64(const int64_t *in, int64_t *out, int64_t n, int64_t shift)
{
   int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
   if (i < n) out[i] = in[i] + shift;
}
__global__ void k_slice_indptr(const int *rp, int r0, int n, int64_t *out)
{
   int i = blockIdx.x * blockDim.x + threadIdx.x;
   if (i <= n) out[i] = (int64_t)rp[r0 + i] - (int64_t)rp[r0];
}
__global__ void k_slice_entries(const int *col, const double *val, int64_t k0, int64_t cnt, int64_t *ocol, double *oval)
{
   int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
   if (k < cnt) { ocol[k] = col[k0 + k]; oval[k] = val[k0 + k]; }
}

// rows [r0, r1) of a serial block -> ParCSR slab (distributed) or local block over all columns
static int slice_rows(const DevCSR &D, int r0, int r1, int64_t cs, int64_t ce, int64_t grows, int64_t gcols,
                      bool square, bool distributed, hdk_csr_s **out)
{
   int      n = r1 - r0;
   int      k[2];
   HDK_CUDA(cudaMemcpyAsync(&k[0], D.rowptr + r0, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaMemcpyAsync(&k[1], D.rowptr + r1, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   int64_t  cnt = (int64_t)k[1] - k[0];
   int64_t *ip, *cj;
   double  *va;
   HDK_TRY(dalloc(&ip, (size_t)n + 1));
   HDK_TRY(dalloc(&cj, (size_t)cnt + 1));
   HDK_TRY(dalloc(&va, (size_t)cnt + 1));
   k_slice_indptr<<<cdiv(n + 1, 256), 256, 0, g.stream>>>(D.rowptr, r0, n, ip);
   HDK_LAUNCH_CHECK();
   if (cnt > 0)
   {
      k_slice_entries<<<cdiv(cnt, 256), 256, 0, g.stream>>>(D.col, D.val, k[0], cnt, cj, va);
      HDK_LAUNCH_CHECK();
   }
   int rc = parcsr_build(r0, (int64_t)r1 - 1, cs, ce, grows, gcols, square, distributed, false, ip, cj, va, out);
   dfree(ip); dfree(cj); dfree(va);
   return rc;
}

static int setup_distributed(const hdk_csr_s *A0, const hdk_amg_params *prm, hdk_amg_s **out)
{
   const int R = g.nranks, me = g.rank;
   stage_mark(nullptr, -2);
   if (!A0->orig_indptr) return set_error(HDK_ERR_INVALID, "distributed setup needs the matrix to be built at N > 1");
   // 1. sizes and offsets of every rank's slab
   std::vector<int64_t> rows_all, nnz_all;
   HDK_TRY(allgather_i64_host(A0->diag.nrows, rows_all));
   HDK_TRY(allgather_i64_host(A0->orig_nnz, nnz_all));
   std::vector<int64_t> roff((size_t)R + 1, 0), koff((size_t)R + 1, 0);
   for (int r = 0; r < R; r++) { roff[(size_t)r + 1] = roff[(size_t)r] + rows_all[(size_t)r]; koff[(size_t)r + 1] = koff[(size_t)r] + nnz_all[(size_t)r]; }
   const int64_t N = roff[(size_t)R], NNZ = koff[(size_t)R];
   if (N > 2000000000LL || NNZ > 2000000000LL)
      return set_error(HDK_ERR_UNSUPPORTED, "global problem (%lld rows, %lld nnz) exceeds the int32 limits of the replicated setup", (long long)N, (long long)NNZ);
   if (roff[(size_t)me] != A0->row_start) return set_error(HDK_ERR_INVALID, "row partition is not contiguous in rank order");
   // 2. reassemble the global operator on every rank
   int64_t *gip, *gcj;
   double  *gva;
   HDK_TRY(dalloc(&gip, (size_t)N + 1));
   HDK_TRY(dalloc(&gcj, (size_t)NNZ + 1));
   HDK_TRY(dalloc(&gva, (size_t)NNZ + 1));
   {
      int64_t n = rows_all[(size_t)me];
      k_shift_i64<<<cdiv(n, 256), 256, 0, g.stream>>>(A0->orig_indptr, gip + roff[(size_t)me], n, koff[(size_t)me]);
      HDK_LAUNCH_CHECK();
      HDK_CUDA(cudaMemcpyAsync(gcj + koff[(size_t)me], A0->orig_cols, sizeof(int64_t) * (size_t)A0->orig_nnz, cudaMemcpyDeviceToDevice, g.stream));
      HDK_CUDA(cudaMemcpyAsync(gva + koff[(size_t)me], A0->orig_vals, sizeof(double) * (size_t)A0->orig_nnz, cudaMemcpyDeviceToDevice, g.stream));
      HDK_CUDA(cudaMemcpyAsync(gip + N, &NNZ, sizeof(int64_t), cudaMemcpyHostToDevice, g.stream));
   }
   for (int r = 0; r < R; r++)
   {
      HDK_TRY(bcast_bytes(gip + roff[(size_t)r], sizeof(int64_t) * (size_t)rows_all[(size_t)r], r));
      HDK_TRY(bcast_bytes(gcj + koff[(size_t)r], sizeof(int64_t) * (size_t)nnz_all[(size_t)r], r));
      HDK_TRY(bcast_bytes(gva + koff[(size_t)r], sizeof(double) * (size_t)nnz_all[(size_t)r], r));
   }
   const int64_t rep_rows = tune_replicate_rows();
   hdk_csr_s *G = nullptr;
   int rc = parcsr_build(0, N - 1, 0, N - 1, N, N, true, false, false, gip, gcj, gva, &G, N <= rep_rows);
   dfree(gip); dfree(gcj); dfree(gva);
   if (rc) return rc;
   // 3. the global hierarchy (serial algorithm, identical on every rank)
   stage_mark("gather A", -2);
   hdk_amg_s *Mg = nullptr;
   g_share = !(getenv("HDK_SETUP_SHARE") && atoi(getenv("HDK_SETUP_SHARE")) == 0);
   if (getenv("HDK_SHARE_MIN_ROWS")) g_share_min_rows = atoi(getenv("HDK_SHARE_MIN_ROWS"));
   rc = setup_serial(G, prm, &Mg, true, rep_rows);
   g_share = false;
   if (rc) { destroy_local(G); return rc; }
   Mg->lev[0].owns_A = true; // G belongs to the global hierarchy
   stage_mark("global setup", -2);
   // 4. fine ranges of every rank on every level; first replicated level
   const int nl = Mg->nlev;
   std::vector<std::vector<int64_t>> starts((size_t)nl); // starts[l][r], r = 0..R
   starts[0] = roff;
   int tail_level = nl - 1;
   for (int l = 0; l < nl; l++)
   {
      bool empty = false;
      for (int r = 0; r < R; r++) if (starts[(size_t)l][(size_t)r + 1] <= starts[(size_t)l][(size_t)r]) empty = true;
      if (Mg->lev[(size_t)l].n <= rep_rows || empty) { tail_level = l; break; }
      if (l + 1 < nl)
      {
         // coarse ranges = f2c at the fine range boundaries
         std::vector<int64_t> nxt((size_t)R + 1, 0);
         for (int r = 0; r <= R; r++)
         {
            int v = 0;
            HDK_CUDA(cudaMemcpyAsync(&v, Mg->lev[(size_t)l].f2c + starts[(size_t)l][(size_t)r], sizeof(int), cudaMemcpyDeviceToHost, g.stream));
            HDK_CUDA(cudaStreamSynchronize(g.stream));
            nxt[(size_t)r] = v;
         }
         starts[(size_t)l + 1] = nxt;
      }
   }
   // 5. distributed levels [0, tail_level): slabs of A_l, P_l, R_l
   hdk_amg_s *M = new hdk_amg_s();
   M->prm = *prm;
   M->tail = Mg; M->tail_level = tail_level;
   M->op_complexity = Mg->op_complexity;
   for (int l = 0; l < tail_level && rc == HDK_OK; l++)
   {
      AmgLevel &Lg = Mg->lev[(size_t)l];
      M->lev.emplace_back();
      AmgLevel &L = M->lev.back();
      const int64_t fs = starts[(size_t)l][(size_t)me], fe = starts[(size_t)l][(size_t)me + 1];
      const int64_t cs = starts[(size_t)l + 1][(size_t)me], ce = starts[(size_t)l + 1][(size_t)me + 1];
      const int64_t nf = Lg.n, nc = Mg->lev[(size_t)l + 1].n;
      L.n = (int)(fe - fs);
      if (l == 0) { L.A = const_cast<hdk_csr_s *>(A0); L.owns_A = false; }
      else
      {
         if ((rc = slice_rows(Lg.A->diag, (int)fs, (int)fe, fs, fe - 1, nf, nf, true, true, &L.A))) break;
         L.owns_A = true;
      }
      if (l + 1 < tail_level)
      {
         if ((rc = slice_rows(Lg.P->diag, (int)fs, (int)fe, cs, ce - 1, nf, nc, false, true, &L.P))) break;
      }
      else
      {
         // the next level is replicated: P reads the complete coarse vector, no halo
         if ((rc = slice_rows(Lg.P->diag, (int)fs, (int)fe, 0, nc - 1, nf, nc, false, false, &L.P))) break;
      }
      if ((rc = slice_rows(Lg.R->diag, (int)cs, (int)ce, fs, fe - 1, nc, nf, false, true, &L.R))) break;
   }
   stage_mark("slice", -2);
   if (rc == HDK_OK)
   {
      M->nlev = tail_level;
      M->tail_n   = Mg->lev[(size_t)tail_level].n;
      M->tail_off = starts[(size_t)tail_level][(size_t)me];
      M->tail_cnt = starts[(size_t)tail_level][(size_t)me + 1] - M->tail_off;
      rc = finalize_levels(M, prm, -1);
      double vb = M->vcycle_bytes;
      // per-rank byte count: distributed levels (local) + replicated tail
      for (int l = tail_level; l < nl; l++)
      {
         AmgLevel &Lg = Mg->lev[(size_t)l];
         double    n = Lg.n, nnzA = Lg.A->diag.nnz;
         if (Lg.P) { double nnzP = Lg.P->diag.nnz, ncl = Lg.P->diag.ncols; vb += 24.0 * n + 2 * (12.0 * nnzA + 4.0 * n) + 56.0 * n + 2 * (12.0 * nnzP) + 28.0 * n + 16.0 * ncl; }
         else vb += 8.0 * n * n + 16.0 * n;
      }
      M->vcycle_bytes = vb;
   }
   if (rc == HDK_OK) rc = dalloc(&M->full_f, (size_t)M->tail_n + 8);
   if (rc == HDK_OK) rc = dalloc(&M->full_u, (size_t)M->tail_n + 8);
   // 6. drop the global copies of the distributed levels
   if (rc == HDK_OK)
   {
      for (int l = 0; l < tail_level; l++)
      {
         AmgLevel &Lg = Mg->lev[(size_t)l];
         if (Lg.owns_A) { destroy_local(Lg.A); Lg.A = nullptr; Lg.owns_A = false; }
         destroy_local(Lg.P); Lg.P = nullptr;
         destroy_local(Lg.R); Lg.R = nullptr;
         csr_free(Lg.S); csr_free(Lg.L);
         dfree(Lg.cf); Lg.cf = nullptr; dfree(Lg.measure); Lg.measure = nullptr; dfree(Lg.f2c); Lg.f2c = nullptr;
         if (Lg.l1_up != Lg.l1_down) dfree(Lg.l1_up);
         dfree(Lg.l1_down); Lg.l1_down = Lg.l1_up = nullptr;
         dfree(Lg.u); dfree(Lg.f); dfree(Lg.t); Lg.u = Lg.f = Lg.t = nullptr;
      }
      HDK_CUDA(cudaStreamSynchronize(g.stream));
   }
   stage_mark("finalize", -2);
   if (rc != HDK_OK) { hdk_amg_destroy(M); return rc; }
   *out = M;
   return HDK_OK;
}

int hdk_amg_setup(const hdk_csr *A0, const hdk_amg_params *prm, hdk_amg **out)
{
   HDK_TRY(require_init());
   if (!A0 || !prm || !out) return set_error(HDK_ERR_INVALID, "hdk_amg_setup: null argument");
   if (prm->interp_type != 6) return set_error(HDK_ERR_UNSUPPORTED, "interpolation type %d: only extended+i (6) has a device kernel", prm->interp_type);
   if (prm->trunc_factor < 0.0 || prm->trunc_factor >= 1.0) return set_error(HDK_ERR_INVALID, "interpolation trunc_factor must be in [0, 1)");
   g_timing = getenv("HDK_SETUP_TIMING") && atoi(getenv("HDK_SETUP_TIMING")) == 1;
   // row-distributed setup (hdk_amg_dist.cu); HDK_SETUP_REPLICATED=1 selects the round-1 scheme that
   // rebuilds the global hierarchy on every rank (kept for comparison)
   const bool replicated = getenv("HDK_SETUP_REPLICATED") && atoi(getenv("HDK_SETUP_REPLICATED")) == 1;
   const bool force_dist = getenv("HDK_SETUP_DIST_FORCE") && atoi(getenv("HDK_SETUP_DIST_FORCE")) == 1;
   if (g.nranks > 1 && replicated) return setup_distributed(A0, prm, out);
   if (g.nranks > 1 || (force_dist && A0->orig_indptr)) return setup_distributed_rows(A0, prm, out);
   return setup_serial(A0, prm, out, false, -1);
}

int hdk_amg_num_levels(const hdk_amg *M) { return M ? M->nlev + (M->tail ? M->tail->nlev - M->tail_level : 0) : 0; }
int hdk_amg_num_dist_levels(const hdk_amg *M) { return (M && M->tail) ? M->nlev : 0; } // N > 1: row-distributed levels
double hdk_amg_operator_complexity(const hdk_amg *M) { return M ? M->op_complexity : 0.0; }
double hdk_amg_vcycle_bytes(const hdk_amg *M) { return M ? M->vcycle_bytes : 0.0; }

// levels [0, nlev) are this rank's slabs of the distributed levels; the following ones live in the
// replicated tail hierarchy
static const hdk_amg_s *resolve_level(const hdk_amg *M, int &level)
{
   if (M && M->tail && level >= M->nlev) { level = level - M->nlev + M->tail_level; return M->tail; }
   return M;
}

int hdk_amg_level_info(const hdk_amg *M, int level, int64_t *rows, int64_t *nnz_A, int64_t *nnz_P)
{
   M = resolve_level(M, level);
   if (!M || level < 0 || level >= M->nlev) return set_error(HDK_ERR_INVALID, "level out of range");
   const AmgLevel &L = M->lev[(size_t)level];
   if (rows) *rows = L.n;
   if (nnz_A) *nnz_A = (int64_t)L.A->diag.nnz + L.A->offd.nnz;
   if (nnz_P) *nnz_P = L.P ? L.P->diag.nnz : 0;
   return HDK_OK;
}

int hdk_amg_get_matrix(const hdk_amg *M, int level, int which, int32_t *rowptr_h, int32_t *col_h, double *val_h)
{
   HDK_TRY(require_init());
   M = resolve_level(M, level);
   if (!M || level < 0 || level >= M->nlev) return set_error(HDK_ERR_INVALID, "level out of range");
   const AmgLevel &L = M->lev[(size_t)level];
   const DevCSR   *D = nullptr;
   if (which == 0) D = &L.A->diag;
   else if (which == 1 && L.P) D = &L.P->diag;
   else if (which == 2 && L.R) D = &L.R->diag;
   else if (which == 3 && L.S.rowptr) D = &L.S;
   if (!D) return set_error(HDK_ERR_INVALID, "matrix %d not available on level %d", which, level);
   if (rowptr_h) HDK_CUDA(cudaMemcpyAsync(rowptr_h, D->rowptr, sizeof(int) * ((size_t)D->nrows + 1), cudaMemcpyDeviceToHost, g.stream));
   if (col_h && D->nnz) HDK_CUDA(cudaMemcpyAsync(col_h, D->col, sizeof(int) * (size_t)D->nnz, cudaMemcpyDeviceToHost, g.stream));
   if (val_h && D->val && D->nnz) HDK_CUDA(cudaMemcpyAsync(val_h, D->val, sizeof(double) * (size_t)D->nnz, cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   return HDK_OK;
}

static int get_level_array(const hdk_amg *M, int level, const void *src, size_t bytes, void *dst)
{
   HDK_TRY(require_init());
   if (!M || level < 0 || level >= M->nlev || !src) return set_error(HDK_ERR_INVALID, "array not available on level %d", level);
   return hdk_copy_d2h(dst, src, bytes);
}
int hdk_amg_get_cf(const hdk_amg *M, int level, int32_t *cf_h)
{
   M = resolve_level(M, level);
   if (!M || level < 0 || level >= M->nlev) return set_error(HDK_ERR_INVALID, "level out of range");
   return get_level_array(M, level, M->lev[(size_t)level].cf, sizeof(int) * (size_t)M->lev[(size_t)level].n, cf_h);
}
int hdk_amg_get_measure(const hdk_amg *M, int level, double *m_h)
{
   M = resolve_level(M, level);
   if (!M || level < 0 || level >= M->nlev) return set_error(HDK_ERR_INVALID, "level out of range");
   return get_level_array(M, level, M->lev[(size_t)level].measure, sizeof(double) * (size_t)M->lev[(size_t)level].n, m_h);
}
int hdk_amg_get_l1(const hdk_amg *M, int level, double *l1_h)
{
   M = resolve_level(M, level);
   if (!M || level < 0 || level >= M->nlev) return set_error(HDK_ERR_INVALID, "level out of range");
   return get_level_array(M, level, M->lev[(size_t)level].l1_down, sizeof(double) * (size_t)M->lev[(size_t)level].n, l1_h);
}

int hdk_amg_strength(const hdk_csr *A, double theta, double max_row_sum, int64_t *nnz_S, int32_t **rowptr_d, int32_t **col_d)
{
   HDK_TRY(require_init());
   if (!A) return set_error(HDK_ERR_INVALID, "null matrix");
   DevCSR S;
   HDK_TRY(build_strength(*A, theta, max_row_sum, S));
   *nnz_S = S.nnz; *rowptr_d = S.rowptr; *col_d = S.col;
   return HDK_OK;
}

int hdk_amg_pmis(int64_t n, const int32_t *S_rowptr_d, const int32_t *S_col_d, int seed, int64_t global_offset,
                 int32_t *cf_d, double *measure_d, int *iterations)
{
   HDK_TRY(require_init());
   DevCSR S;
   S.nrows = (int)n; S.ncols = (int)n; S.rowptr = const_cast<int *>(S_rowptr_d); S.col = const_cast<int *>(S_col_d);
   HDK_CUDA(cudaMemcpyAsync(&S.nnz, S_rowptr_d + n, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
   HDK_CUDA(cudaStreamSynchronize(g.stream));
   double *work;
   HDK_TRY(dalloc(&work, (size_t)n + 1));
   int rc = run_pmis(S, seed, global_offset, cf_d, work, measure_d, iterations);
   dfree(work);
   return rc;
}

} // extern "C"
