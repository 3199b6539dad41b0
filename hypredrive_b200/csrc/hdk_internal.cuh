// hdk_internal.cuh -- shared device-side plumbing of the hdk kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "hdk.h"

namespace hdk {

struct Ctx
{
   bool         inited = false;
   int          device = 0;
   int          sm_count = 148;
   cudaStream_t stream = nullptr;     // compute stream
   cudaStream_t comm_stream = nullptr; // halo exchange stream
   cudaEvent_t  ev_a = nullptr, ev_b = nullptr, ev_scal = nullptr, ev_halo = nullptr, ev_pack = nullptr;
   int          rank = 0, nranks = 1;
   void        *nccl = nullptr;        // ncclComm_t
   int64_t      launches = 0;
   // reduction scratch
   double      *partials = nullptr;    // device, PARTIALS_CAP doubles
   unsigned    *counters = nullptr;    // device, 64 tickets (zero-initialised, self-resetting)
   double      *dscal = nullptr;       // device scalar block (64 doubles)
   double      *hscal = nullptr;       // pinned host mirror (64 doubles)
   char         err[1024] = {0};
};

extern Ctx g;
constexpr int PARTIALS_CAP = 1 << 20;

int  set_error(int code, const char *fmt, ...);
int  require_init();

#define HDK_CUDA(call)                                                                     \
   do {                                                                                    \
      cudaError_t e__ = (call);                                                            \
      if (e__ != cudaSuccess)                                                              \
         return hdk::set_error(HDK_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,  \
                               cudaGetErrorString(e__));                                   \
   } while (0)

#define HDK_TRY(call)                  \
   do {                                \
      int rc__ = (call);               \
      if (rc__ != HDK_OK) return rc__; \
   } while (0)

#define HDK_LAUNCH_CHECK()                                                                  \
   do {                                                                                     \
      hdk::g.launches++;                                                                    \
      cudaError_t e__ = cudaGetLastError();                                                 \
      if (e__ != cudaSuccess)                                                               \
         return hdk::set_error(HDK_ERR_CUDA, "%s:%d launch -> %s", __FILE__, __LINE__,      \
                               cudaGetErrorString(e__));                                    \
   } while (0)

// stream-ordered allocation from the device memory pool (cached between calls)
template <class T>
inline int dalloc(T **p, size_t n)
{
   *p = nullptr;
   if (n == 0) n = 1;
   cudaError_t e = cudaMallocAsync((void **)p, n * sizeof(T), g.stream);
   if (e != cudaSuccess)
      return set_error(HDK_ERR_ALLOC, "cudaMallocAsync(%zu bytes) -> %s", n * sizeof(T),
                       cudaGetErrorString(e));
   return HDK_OK;
}
inline void dfree(void *p)
{
   if (p) cudaFreeAsync(p, g.stream);
}

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------
// One CSR block on the device.  rowptr/col are int32 (hypre HYPRE_Int), values fp64.
// col/val are allocated with 8 slack entries (col = 0, val = 0) so 128-bit loads that
// start at a 4-entry aligned index never leave the allocation.
// ---------------------------------------------------------------------------------------
struct DevCSR
{
   int     nrows = 0, ncols = 0;
   int     nnz = 0;
   int    *rowptr = nullptr;
   int    *col = nullptr;
   double *val = nullptr;
   // SpMV analysis (row-length statistics -> kernel choice)
   int     kind = 0;          // 0 stream, 1 vector (warp per row), 2 sliced-ELL
   int     max_row = 0;
   double  avg_row = 0.0;
   int     tgt = 0, cap = 0;  // stream kernel: non-zeros per CTA, shared-memory entries per stage
   int     lpr = 1;           // stream kernel: lanes per row (1, 2, 4, 8)
   int     nblk = 0;          // stream kernel: number of nnz-balanced row blocks
   int    *blk_row = nullptr; // nblk+1 first rows
   // sliced-ELL copy (kind 2): slices of 32 rows stored column-major, see hdk_spmv.cu
   int     nslice = 0;
   int    *sl_off = nullptr;  // nslice+1 prefix sums of slice widths (units of 32 entries)
   int    *sl_meta = nullptr; // nslice*32: row length << 6 | has-offd flag << 5 | row offset inside the slice
   int    *sl_col = nullptr;
   double *sl_val = nullptr;
   const int *offd_rowptr = nullptr; // set before csr_analyze: rows with off-rank entries get flagged in sl_meta
   bool    sl_offd_flags = false;
   bool    coarse_op = false; // Galerkin operator of the hierarchy: its stored column order may be changed
   bool    owns = true;
};

int  csr_alloc(DevCSR &A, int nrows, int ncols, int nnz, bool values = true);
void csr_free(DevCSR &A);
int  csr_analyze(DevCSR &A);
int  tune_set(const char *key, double value);
bool tune_amg_keep_debug();
int64_t tune_replicate_rows();
int64_t tune_graph_rows();

// epilogue selectors of the fused SpMV family (see hdk_spmv.cu)
enum SpmvMode
{
   SPMV_SET = 0,      // y = A x
   SPMV_RESIDUAL = 1, // y = b - A x        (res = b; res -= a*x in CSR order)
   SPMV_JACOBI = 2,   // y = x + w*(b - A x)/d
   SPMV_ADD = 3,      // y = y + A x        (s = y; s += a*x in CSR order)
   SPMV_AXPBY = 4,    // y = alpha*(A x) + beta*y
   SPMV_JACOBI_R = 5, // y = w*(b - A x)/d  (two-stage GS first stage)
   SPMV_SET_DIV = 6,  // y = A x ; y2 = w*y/d  (restriction fused with the next level's first l1-Jacobi sweep)
   SPMV_JACOBI2 = 7,  // y2 = w*(b - A x)/d ; y = x + y2   (two-stage GS, first stage: correction AND updated iterate)
   SPMV_GS_STEP = 8,  // t = (A x)/d ; y2 = t ; y = y + alpha*t   (two-stage GS inner step on the strict lower triangle)
   // Chebyshev sweep (relax 16), d = ds = |a_ii|^{-1/2}, alpha = the polynomial coefficient c, b = f or r
   SPMV_CHEB_START = 10, // y2 = r = d (b - A x) ; y = d (c r)                   (first pass of an order >= 2 sweep)
   SPMV_CHEB_STEP = 11,  // y = d (c b + d (A x))                                (b = r)
   SPMV_CHEB_FIN = 12,   // y = uo + d (c b + d (A x))                           (b = r; uo = u_old, nullptr = 0)
   SPMV_CHEB_ONE = 13    // y = uo + d (c (d (b - A x)))                         (order 1: the whole sweep)
};

// what the last block does with a fused dot product
enum FinOp
{
   FIN_NONE = 0,
   FIN_STORE = 1,  // out[0] = v
   FIN_SDOTP = 2,  // PCG: sdotp = v; alpha = gamma / v
   FIN_IPROD = 3,  // PCG: i_prod = v
   FIN_GAMMA = 4   // PCG: gamma_old = gamma; gamma = v; beta = v / gamma_old
};

// layout of the device scalar block used by the Krylov drivers
enum ScalIdx
{
   S_BIPROD = 0, S_GAMMA = 1, S_GAMMA_OLD = 2, S_SDOTP = 3, S_IPROD = 4, S_ALPHA = 5, S_BETA = 6,
   S_TMP0 = 8, S_TMP1 = 9, S_TMP2 = 10, S_TMP3 = 11, S_H0 = 16 /* 16..63: GMRES h column */
};

} // namespace hdk
struct hdk_csr_s;
namespace hdk {
struct SpmvArgs
{
   const double *x = nullptr;   // input vector (gathered)
   double       *y = nullptr;   // output
   const double *b = nullptr;   // rhs (RESIDUAL / JACOBI)
   const double *d = nullptr;   // diagonal scaling (JACOBI)
   const double *xo = nullptr;  // halo part of x (offd block), appended columns
   double       *y2 = nullptr;  // second output of SPMV_SET_DIV
   double        w = 1.0, alpha = 1.0, beta = 0.0;
   const double *uo = nullptr;  // iterate the Chebyshev finish adds to (SPMV_CHEB_FIN / _ONE; nullptr: zero)
   // fused dot: sum_i dotv[i]*y_new[i]  (dotv may alias x or b)
   const double *dotv = nullptr;
   int           fin = FIN_NONE;
   double       *fin_out = nullptr;
   // the matrix whose next product reads this kernel's output (y, or y2 with export_y2): its halo is
   // filled by this kernel (see HaloExport) when the peer-memory path is on
   const struct ::hdk_csr_s *export_to = nullptr;
   bool          export_y2 = false;
};


// vector kernels (hdk_vec.cu)
int vec_fill(double *x, double v, int64_t n);
int vec_copy(double *dst, const double *src, int64_t n);
int vec_axpy(double a, const double *x, double *y, int64_t n);
int vec_scale(double a, double *x, int64_t n);
int vec_dot_dev(const double *x, const double *y, int64_t n, int fin, double *out_d); // device result
int vec_dot_host(const double *x, const double *y, int64_t n, double *out_h);         // + allreduce
int vec_scaled_div(double *u, const double *f, const double *d, double w, int64_t n,    // u = w f / d
                   const struct ::hdk_csr_s *export_to = nullptr);                          // (+ halo of export_to's next product)
int pcg_update_xr(double *x, double *r, const double *p, const double *s, int64_t n, double *scal,
                  int fin = FIN_IPROD, double *fin_out = nullptr, // <r,r> -> fin (FIN_STORE at N > 1)
                  double *z0 = nullptr, const double *zd = nullptr, double zw = 1.0, // optional z0 = (zw r)/zd
                  const struct ::hdk_csr_s *export_z0_to = nullptr);
int pcg_update_p(double *p, const double *z, int64_t n, const double *scal, const struct ::hdk_csr_s *export_to = nullptr);
int vec_copy_dot(double *z, const double *r, int64_t n, int fin, double *out_d);      // z=r, <r,r>
int allreduce_dev(double *buf_d, int count);                                          // sum over ranks (no-op on 1 rank)
int allreduce_fin_dev(double *buf_d, int count, int fin, double *fin_out);            // ... + Krylov scalar recurrence, one kernel

// ---------------------------------------------------------------------------------------
// ParCSR of one rank: diag + offd blocks, halo bookkeeping
// ---------------------------------------------------------------------------------------
// Peer-memory halo exchange (CUDA IPC over NVLink): the pack kernel stores the boundary values
// straight into the neighbours' halo buffers and raises a sequence flag there; the kernel that
// consumes the halo waits for the flags itself.  See hdk_comm.cu.
constexpr int IPC_MAXP = 8; // neighbours per direction handled by the peer-memory path
struct IpcSendArgs
{
   double             *dst[IPC_MAXP];   // remote segment of x_halo (current half) per send neighbour
   int                 off[IPC_MAXP + 1];
   int                 npeer;           // send neighbours
   unsigned long long *flag[IPC_MAXP];  // remote "sequence reached" slot of EVERY neighbour (send or receive)
   const unsigned long long *rflag;     // my own slots, one per neighbour: the last CTA waits for them,
   int                 nflag;           // so the exchange is complete when the kernel ends
   unsigned long long  seq;
   unsigned           *ticket;
};
// Halo export folded into the PRODUCER of a vector: the kernel that writes x stores the rows its
// neighbours need straight into their halo buffers (peer stores over NVLink); the warp whose stores
// complete the send list raises the sequence flags and waits for this rank's own halo, so the
// consumer's exchange costs no kernel of its own.  dir: direct table over the rows outside the
// export-free middle range -> index of the exported row (or -1); ptr / slot: per exported row, its
// positions in the concatenated send list (a row may go to several neighbours).
struct HaloExport
{
   const int          *dir = nullptr, *ptr = nullptr, *slot = nullptr;
   int                 total = 0;          // entries of the send list: the export is complete when all are stored
   int                 lo_end = 0, hi_begin = 0; // rows in [lo_end, hi_begin) are never exported (quick reject)
   double             *dst[IPC_MAXP];
   int                 off[IPC_MAXP + 1];
   int                 npeer = 0;
   unsigned long long *flag[IPC_MAXP];     // as in IpcSendArgs
   const unsigned long long *rflag = nullptr;
   int                 nflag = 0;
   unsigned long long  seq = 0;            // 0: export off
   unsigned           *ticket = nullptr;
};

// off-rank block fused into the sliced-ELL kernel: rows flagged in sl_meta continue their sum with
// the block's entries (CSR arrays) and the values of the finished exchange (xh)
struct OffdFuse
{
   const int    *orp = nullptr, *ocol = nullptr;
   const double *oval = nullptr, *xh = nullptr;
};
int spmv_launch(const DevCSR &A, int mode, const SpmvArgs &a, const OffdFuse *of = nullptr);

struct IpcHalo
{
   bool                on = false;
   int64_t             region_off = -1;
   size_t              region_bytes = 0;
   double             *xh[2] = {nullptr, nullptr}; // local halves of x_halo
   unsigned long long *data_flag = nullptr;         // local slots, one per neighbour (send or receive)
   double             *dst[2][IPC_MAXP];            // per send neighbour
   unsigned long long *nbr_flag[IPC_MAXP];          // my slot in every neighbour's region
   int                 nnbr = 0;
   unsigned long long  seq = 0;
   unsigned           *tickets = nullptr; // two device counters: pack, export
   // inverse of the send list for exports folded into the producer kernel
   int                *exp_dir = nullptr, *exp_ptr = nullptr, *exp_slot = nullptr;
   int                 exp_lo_end = 0, exp_hi_begin = 0;
   bool                preposted = false;  // the current sequence was filled by the producer: no pack kernel
};

#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p)
{
   unsigned long long v;
   asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
   return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v)
{
   asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Wait for a neighbour's sequence flag.  The wait is bounded by a configurable budget
// (HDK_IPC_TIMEOUT_S, default 300 s, 0 = unbounded): when it runs out the kernel raises an
// error flag in device memory and carries on with whatever the buffer holds -- the CUDA context stays
// usable, the host reports HDK_ERR_COMM at the end of the operation (comm_check_error) and later
// waits return at once.  No trap: a trap would poison the context of this rank and hang its peers.
// Budget and flag live in per-translation-unit device globals (set by wait_globals_set at communicator
// creation), not in kernel arguments: two more arguments on the out-of-line wait cost the sliced-ELL
// kernel 8 registers = 2 CTAs per SM.
static __device__ long long d_wait_tmo = 0;
static __device__ int      *d_wait_err = nullptr;
static __device__ __noinline__ void wait_seq_slow(const unsigned long long *p, unsigned long long want)
{
   const long long t0 = clock64(), tmo = d_wait_tmo;
   int            *err = d_wait_err;
   unsigned        spins = 0;
   while (ld_acquire_sys_u64(p) < want)
   {
      __nanosleep(64);
      if (tmo > 0 && (++spins & 1023u) == 0)
      {
         // the flag lives in device memory: an L2 hit for the other waiters, which give up with it
         if (clock64() - t0 > tmo) { if (err) *(volatile int *)err = 1; return; }
         if (err && *(volatile int *)err) return;
      }
   }
}
__device__ __forceinline__ void wait_seq_sys(const unsigned long long *p, unsigned long long want, long long = 0, int * = nullptr)
{
   if (ld_acquire_sys_u64(p) >= want) return;
   wait_seq_slow(p, want); // out of line: keeps the waiting kernels' register count down
}
// one call per translation unit that contains waiting kernels (each has its own copy of the globals)
static inline cudaError_t wait_globals_set(long long tmo, int *err)
{
   cudaError_t e = cudaMemcpyToSymbol(d_wait_tmo, &tmo, sizeof(tmo));
   if (e == cudaSuccess) e = cudaMemcpyToSymbol(d_wait_err, &err, sizeof(err));
   return e;
}
// Producer side of a folded halo exchange: row r of the vector just got value v.  Returns the number
// of send-list entries stored (summed per thread and handed to export_finish).
// Buffer reuse needs no acknowledgement: every exchange is two-way between neighbours (a rank raises
// its flag at EVERY neighbour, also one it sends no values to) and the kernel that starts exchange s
// (pack or exporting producer) does not end before all neighbours' flags have reached s.  A neighbour's
// flag s was raised after -- in its stream -- the product that read exchange s - 1, so when my exchange
// s + 1 starts overwriting the half of s - 1, that product is finished.
__device__ __forceinline__ int export_row(const HaloExport &e, int r, double v)
{
   if (e.seq == 0 || (r >= e.lo_end && r < e.hi_begin)) return 0;
   // direct table over the two row ranges outside [lo_end, hi_begin): index into ptr, or -1
   const int i = e.dir[r < e.lo_end ? r : e.lo_end + (r - e.hi_begin)];
   if (i < 0) return 0;
   const int k0 = e.ptr[i], k1 = e.ptr[i + 1];
   for (int k = k0; k < k1; k++)
   {
      const int s = e.slot[k];
      int       p = 0;
      while (p + 1 < e.npeer && s >= e.off[p + 1]) p++;
      e.dst[p][s - e.off[p]] = v;
   }
   return k1 - k0;
}
// raise my flag at every neighbour, then wait until all of theirs have reached the same sequence: the
// exchange is complete when the kernel that calls this ends, and consumers need no synchronisation.
// (Measured against waiting in the consumer -- per boundary lane, or thread 0 of every CTA at kernel
// start -- this is ~0.5 ms per 256^3 solve faster at N = 2: one thread polls, once, at a kernel's tail.)
__device__ __forceinline__ void exchange_complete(unsigned long long *const *flag, const unsigned long long *rflag, int nflag,
                                                  unsigned long long seq)
{
   __threadfence_system();
   for (int p = 0; p < nflag; p++) st_release_sys_u64(flag[p], seq);
   for (int p = 0; p < nflag; p++) wait_seq_sys(rflag + p, seq);
}
// End of the producer kernel, executed by every warp with all 32 lanes (cnt: what the lane's
// export_row calls returned).  Warps that exported nothing pay one warp reduction; an exporting warp
// orders its lanes' peer stores with ONE system-scope fence (lane 0, after the warp barrier of the
// reduction) and adds its count to the ticket; the warp that completes the send list finishes the
// exchange.  No CTA barrier, no per-CTA atomics.
__device__ __forceinline__ void export_finish(const HaloExport &e, int cnt)
{
   if (e.seq == 0) return;
   const unsigned tot = __reduce_add_sync(0xffffffffu, (unsigned)cnt);
   __syncwarp(); // (the reduction itself is no memory barrier) orders the lanes' peer stores before lane 0's fence
   if (tot == 0 || (threadIdx.x & 31) != 0) return;
   __threadfence_system();
   const unsigned before = atomicAdd(e.ticket, tot);
   if (before + tot == (unsigned)e.total)
   {
      *e.ticket = 0u; // every contribution is in: re-arm for the next exchange (kernels of one plan are stream-ordered)
      exchange_complete(e.flag, e.rflag, e.nflag, e.seq);
   }
}
#endif

// all-gather of a replicated vector's slices through peer stores (hdk_comm.cu)
struct IpcGather
{
   bool                on = false;
   int64_t             n = 0, region_off = -1;
   size_t              region_bytes = 0;
   unsigned long long  seq = 0;
   unsigned long long *flags = nullptr;        // my flag slots, one per source rank
   double             *buf[2] = {nullptr, nullptr};
   double             *peer_buf[2][16];
   unsigned long long *peer_flag[16];
   unsigned           *ticket = nullptr;
};
int     ipc_gather_alloc(IpcGather &G, int64_t n); // collective; G.on stays false without the peer-memory arena
void    ipc_gather_free(IpcGather &G);
double *ipc_gather_buffer(IpcGather &G);
int     ipc_gather(IpcGather &G, int64_t off, int64_t cnt);

struct HaloPlan
{
   IpcHalo             ipc;
   int                 n_halo = 0;         // number of offd columns (size of x_halo)
   int64_t            *col_map = nullptr;  // device, sorted global ids of offd columns
   std::vector<int>     recv_rank, recv_off, recv_cnt; // per neighbour (host)
   std::vector<int>     send_rank, send_off, send_cnt;
   int                 n_send = 0;
   int                *send_idx = nullptr; // device, local row ids to pack
   double             *send_buf = nullptr; // device
   double             *x_halo = nullptr;   // device
};

} // namespace hdk

struct hdk_csr_s
{
   int64_t       row_start = 0, row_end = -1, global_rows = 0, global_nnz = 0;
   int64_t       col_start = 0, col_end = -1, global_cols = 0; // this rank's share of the column space
   int64_t      *orig_indptr = nullptr, *orig_cols = nullptr;  // N > 1: caller's rows, global columns
   double       *orig_vals = nullptr;
   int64_t       orig_nnz = 0;
   int          *offd_rows = nullptr; // rows with off-rank entries
   int           n_offd_rows = 0;
   hdk::DevCSR   diag, offd;
   hdk::HaloPlan halo;
   std::vector<int64_t> row_starts; // partition (nranks+1), host
};

namespace hdk {
int parcsr_matvec(const hdk_csr_s &A, int mode, SpmvArgs a); // halo exchange + diag + offd
bool parcsr_single_kernel(const hdk_csr_s &A);
int parcsr_build(int64_t rs, int64_t re, int64_t cs, int64_t ce, int64_t grows, int64_t gcols, bool square,
                 bool distributed, bool keep_orig, const int64_t *indptr, const int64_t *cols, const double *vals,
                 hdk_csr_s **out, bool analyze = true);
int allreduce_max_dev(double *buf_d, int count);
int bcast_bytes(void *buf_d, size_t bytes, int root);                 // NCCL broadcast on the compute stream
int allgather_i64_host(int64_t mine, std::vector<int64_t> &all);
int allgather_i32_host(const int *mine, int cnt, std::vector<int> &all); // all[r*cnt + i]
int allreduce_i32_dev(int *buf_d, int count);
int alltoallv_bytes(const void *send_d, const int64_t *soff /* nranks+1 */, void *recv_d, const int64_t *roff /* nranks+1 */);
int allgatherv_bytes(void *base_d, const int64_t *byte_offs /* nranks+1 */); // in place, compute stream
void halo_plan_free(HaloPlan &H);
const double *halo_buffer(const hdk_csr_s &A); // after halo_exchange_begin: where this exchange's values are
int halo_exchange_begin(const hdk_csr_s &A, const double *x);
void dbg_skip_exchange(bool on);
void tl_mark(int level, int op); // diagnostics timeline (hdk_runtime.cu)
int halo_exchange_end(const hdk_csr_s &A);
// producer-side exchange: fills *e for the kernel that writes the vector A's next product reads and
// marks the plan as served; false (and e->seq == 0) when the plan is not on the peer-memory path
bool halo_export_begin(const hdk_csr_s &A, HaloExport *e);
void halo_export_cancel(const hdk_csr_s &A); // the exported vector will not be consumed after all
int comm_check_error(); // HDK_ERR_COMM when a peer-memory wait ran out of its budget since the last call
int wait_globals_spmv(long long tmo, int *err); // per-translation-unit setters of the wait budget / error flag
int wait_globals_csr(long long tmo, int *err);
int wait_globals_vec(long long tmo, int *err);

// ---------------------------------------------------------------------------------------
// device reduction helper: block sum -> partials -> last block finishes (deterministic)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
   for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
   return v;
}

template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double *sm /* THREADS/32 */)
{
   int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
   v = warp_sum(v);
   if (lane == 0) sm[w] = v;
   __syncthreads();
   double r = 0.0;
   if (w == 0)
   {
      r = (lane < THREADS / 32) ? sm[lane] : 0.0;
      r = warp_sum(r);
   }
   return r; // valid in thread 0
}

__device__ __forceinline__ void apply_fin(int fin, double v, double *out, double *scal)
{
   switch (fin)
   {
      case FIN_STORE: out[0] = v; break;
      // <Ap,p> = 0 is a breakdown (hypre_PCGSolve stops before the update): alpha = 0 leaves x and r
      // untouched, the host sees S_SDOTP == 0 and ends the iteration
      case FIN_SDOTP: scal[S_SDOTP] = v; scal[S_ALPHA] = (v != 0.0) ? scal[S_GAMMA] / v : 0.0; break;
      case FIN_IPROD: scal[S_IPROD] = v; break;
      case FIN_GAMMA:
      {
         double go = scal[S_GAMMA];
         scal[S_GAMMA_OLD] = go; scal[S_GAMMA] = v; scal[S_BETA] = v / go;
         break;
      }
      default: break;
   }
}

// Every block calls this with its (thread-0 valid) block sum.  The last block to arrive adds
// the partials in a fixed order and applies `fin`.  ticket counters wrap back to zero.
template <int THREADS>
__device__ __forceinline__ void grid_finish(double blocksum, double *partials, unsigned *ticket,
                                            int fin, double *out, double *scal, double *sm,
                                            int *flag_sm)
{
   if (threadIdx.x == 0)
   {
      partials[blockIdx.x] = blocksum;
      __threadfence();
      unsigned t = atomicInc(ticket, gridDim.x - 1);
      *flag_sm   = (t == gridDim.x - 1);
   }
   __syncthreads();
   if (*flag_sm)
   {
      __threadfence();
      double s = 0.0;
      for (unsigned i = threadIdx.x; i < gridDim.x; i += THREADS) s += __ldcg(partials + i);
      __syncthreads();
      s = block_sum<THREADS>(s, sm);
      if (threadIdx.x == 0) apply_fin(fin, s, out, scal);
   }
}

} // namespace hdk
