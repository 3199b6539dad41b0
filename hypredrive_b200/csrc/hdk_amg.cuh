// hdk_amg.cuh -- device BoomerAMG hierarchy (internal).
#pragma once
#include "hdk_internal.cuh"

namespace hdk {

struct AmgLevel
{
   hdk_csr_s *A = nullptr;  // level operator (level 0 is borrowed from the caller)
   bool       owns_A = false;
   hdk_csr_s *P = nullptr;  // n_l x n_{l+1}
   hdk_csr_s *R = nullptr;  // n_{l+1} x n_l  (P^T stored explicitly: keep_transpose)
   DevCSR     S;            // strength pattern (diag block)
   DevCSR     S2;           // aggressive levels: second-stage strength over the first-stage C points
   int       *cf = nullptr;
   int       *f2c = nullptr; // exclusive scan of (cf > 0), n+1 entries (kept for the N > 1 slicing)
   double    *measure = nullptr;
   int       *dof = nullptr;     // function labels of the rows (systems AMG, num_functions > 1)
   double    *l1_down = nullptr, *l1_up = nullptr; // smoother diagonals (may alias)
   double    *u = nullptr, *f = nullptr, *t = nullptr;
   double    *gs1 = nullptr, *gs2 = nullptr; // two-stage GS: correction vectors of the inner steps
   DevCSR     L;            // strict lower triangle (two-stage GS only)
   // Chebyshev smoothing (relax 16): D^{-1/2} (ones when unscaled), the sweep's scaled residual and the
   // two alternating polynomial states; eigenvalue bounds (max, min) and coefficients c_0..c_{order-1}
   double    *cheb_ds = nullptr, *cheb_r = nullptr, *cheb_v[2] = {nullptr, nullptr};
   double     cheb_eig[2] = {0.0, 0.0}, cheb_c[4] = {0.0, 0.0, 0.0, 0.0};
   int        n = 0;
   // distributed setup, amg_keep_debug: my rows of P_l and A_l with GLOBAL columns in the serial
   // storage order (what the parity tests compare with the oracle, slab by slab)
   int64_t   *dbg_ip[2] = {nullptr, nullptr}, *dbg_col[2] = {nullptr, nullptr}; // [0] = A_l, [1] = P_l
   double    *dbg_val[2] = {nullptr, nullptr};
   int64_t    dbg_nnz[2] = {0, 0}, row0 = 0;
};

} // namespace hdk

struct hdk_amg_s
{
   hdk_amg_params             prm;
   std::vector<hdk::AmgLevel> lev;
   int                        nlev = 0;
   double                    *ge_inv = nullptr; // dense inverse of the coarsest operator
   int                        ge_n = 0;
   double                     op_complexity = 0.0;
   double                     vcycle_bytes = 0.0;
   bool                       keep_debug = false; // keep S / measure for introspection (tunable amg_keep_debug)
   int                        prefilled_at = -1; // next zero-guess cycle from this level: its first sweep is already in place
   // sub-cycles over the small levels captured into CUDA graphs (hdk_amg_solve.cu)
   struct CycleGraph { const double *f; double *u; bool zero_guess, prefilled; int level; void *exec; int nodes; };
   std::vector<CycleGraph>    graphs;
   bool                       graph_off = false;
   bool                       keep_f2c = false;
   // N > 1: levels [0, nlev) are row-distributed; from level `tail_level` on, the hierarchy is
   // replicated on every rank (`tail`, a serial hierarchy of the GLOBAL problem) and the
   // restricted right-hand side is summed over ranks into `full_f`
   hdk_amg_s                 *tail = nullptr;
   int                        tail_level = 0;   // level of `tail` that continues this hierarchy
   int64_t                    tail_off = 0, tail_cnt = 0, tail_n = 0; // my slice of the first replicated level
   double                    *full_f = nullptr, *full_u = nullptr;
   hdk::IpcGather             gather;   // peer-memory all-gather of the slices of full_f (replaces the all-reduce)
};

// pieces of the serial setup (hdk_amg_setup.cu) that the distributed driver (hdk_amg_dist.cu) reuses
extern "C" {
int finalize_levels(hdk_amg_s *M, const hdk_amg_params *prm, int64_t live_max_rows);
// dof0_d: device labels of the rows of A0 (systems AMG); nullptr: prm->dof_func or interleaved labels
int setup_serial(const hdk_csr_s *A0, const hdk_amg_params *prm, hdk_amg_s **out, bool keep_f2c, int64_t live_max_rows,
                 const int *dof0_d = nullptr);
int setup_distributed_rows(const hdk_csr_s *A0, const hdk_amg_params *prm, hdk_amg_s **out); // hdk_amg_dist.cu
}

namespace hdk {
int build_strength_csr(const DevCSR &D, const int *orp, const double *ov, double theta, double mrs, DevCSR &S,
                       const int *dof = nullptr);
int pmis_count_cols(const DevCSR &S, int row0, int n, int *cnt);
int pmis_measure(const int *cnt, int n, int seed, int64_t goff, double *measure);
int pmis_init(const DevCSR &S, int row0, int n, int *cf, double *measure);
int pmis_mark(int n, int *cf, const double *measure);
int pmis_elim(const DevCSR &S, int row0, int n, int *cf, const double *measure);
int pmis_set(const DevCSR &S, int row0, int n, int *cf, double *measure, int *remaining);
int build_interp(const DevCSR &A, const DevCSR &S, int *cf, const int *f2c, int nc, int max_elmts_in, double trunc_factor,
                 DevCSR &P, int row_lo, int row_hi, const int *dof = nullptr);
int build_rap(const DevCSR &R, const DevCSR &A, const DevCSR &P, DevCSR &C, int row_lo, int row_hi);
int csr_transpose(const DevCSR &A, DevCSR &T);
hdk_csr_s *wrap_local(DevCSR &D, int64_t grows);
void destroy_local(hdk_csr_s *A);
void setup_stage_mark(const char *name, int level);

// z = M^{-1} r (one V-cycle from a zero guess); if fin != FIN_NONE the last kernel also
// produces <r,z> and applies `fin`
int amg_precond(hdk_amg_s *M, const double *r, double *z, int fin, double *fin_out);
// V-cycle over levels [l0, nlev) of M; level l0 uses the caller's vectors
int amg_cycle(hdk_amg_s *M, const double *f, double *u, bool zero_guess, int fin, double *fin_out, int l0 = 0);
int exclusive_scan_int(const int *in, int *out, int n);       // hdk_csr.cu (hand-written reduce-then-scan)
int exclusive_scan_i64(const int *in, int64_t *out, int n);
int exclusive_scan_i64_i64(const int64_t *in, int64_t *out, int64_t n);
// Chebyshev (hdk_spmv.cu): y = the epilogue of `mode` (SPMV_CHEB_*) applied to a finished row result
// acc (A x, or b - A x for START / ONE), element-wise; the unfused form and the zero-guess start
int cheb_epilogue_pass(int mode, int n, const double *acc, const SpmvArgs &a);
bool amg_prefill_target(hdk_amg_s *M, double *z, double **buf, const double **d, double *w, const hdk_csr_s **reader = nullptr);
} // namespace hdk
