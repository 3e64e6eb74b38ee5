// kb_internal.h -- internal C++ interfaces of libkrylov_b200.
//
// Layering (mirrors Krylov.jl's L1..L3, SURVEY.md section 1):
//   Ctx           one CUDA stream + reduction scratch + pinned scalar mailbox
//   blas1.cu      k* primitives on device vectors   (src/krylov_utils.jl:309-349)
//   spmv.cu       CSR operator: plain and TMA-staged SpMV (kmul!, krylov_utils.jl:305)
//   cg_fused.cu   two-launch CG iteration               (src/cg.jl:195-268)
//   fused_phases.cu  fused iteration phases of bicgstab!/minres!/gmres! (+ the Arnoldi step fom!/fgmres! share)
//   solvers.cu    host control flow of cg!/gmres!/bicgstab!/minres! on the primitives
//   siblings.cu   cgs!, cg_lanczos!, fom!, fgmres!, dqgmres!, diom!, cr! on the same kernels (SURVEY.md 8f-3)
//   block.cu      block_gmres! on row-major device panels (8f-2; block.h)
//   mtx.cu        Matrix Market ingestion, transposed operator (8f-4; mtx.h)
//   capi.cu       the C ABI (include/krylov_b200.h)
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "common.cuh"
#include "dist.cuh"

namespace kb {

// ---------------------------------------------------------------------------
// Execution context: everything a solve needs besides its vectors.
// ---------------------------------------------------------------------------
struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  void* partials = nullptr;      // kMaxPartials * 4 doubles of reduction scratch
  unsigned* tickets = nullptr;   // 8 tickets (zero-initialised, self re-arming)
  void* dscal = nullptr;         // 16 device scalars (doubles) written by reductions
  void* hscal = nullptr;         // pinned mirror of dscal
  long long launches = 0;        // kernels launched through this context (bench: gpu_launches)
  DistComm* dcomm = nullptr;     // device-resident communicator of a row-partitioned solve (nullptr: single GPU)
  DistExchange* dex = nullptr;   // host-side plan of the general x-halo exchange (nullptr: single GPU)

  void init(int dev);
  void destroy();
  void sync() { KB_CUDA(cudaStreamSynchronize(stream)); }
};

template <class T> T* dev_alloc(size_t n);                // cudaMalloc, n elements (+ 64 B pad)
void dev_free(void* p);

// ---------------------------------------------------------------------------
// BLAS-1 on device vectors.  Scalars that solvers consume on the host are
// returned by value (one pinned read-back + stream sync), exactly like the
// reference's kdot/knorm; the *_dev variants leave the result in ctx.dscal[slot].
// ---------------------------------------------------------------------------
template <class T> T    k_dot(Ctx& c, int n, const T* x, const T* y);
template <class T> T    k_nrm2(Ctx& c, int n, const T* x);
template <class T> T    k_cg_prologue(Ctx& c, int n, const T* b, T* x, T* r, T* p);   // x = 0, r = p = b, returns <b, b>
template <class T> void k_dot2(Ctx& c, int n, const T* a, const T* b, const T* u, const T* v, T* r1, T* r2);
template <class T> void k_dot_dev(Ctx& c, int n, const T* x, const T* y, int slot);
template <class T> void k_axpy(Ctx& c, int n, T s, const T* x, T* y);                 // y += s x
template <class T> void k_axpby(Ctx& c, int n, T s, const T* x, T t, T* y);           // y = s x + t y
template <class T> void k_scal(Ctx& c, int n, T s, T* x);                             // x *= s
template <class T> void k_copy(Ctx& c, int n, T* y, const T* x);                      // y = x
template <class T> void k_scalcopy(Ctx& c, int n, T* y, T s, const T* x);             // y = s x
template <class T> void k_divcopy(Ctx& c, int n, T* y, const T* x, T s);              // y = x / s
template <class T> void k_fill(Ctx& c, int n, T* x, T v);
template <class T> void k_diagmul(Ctx& c, int n, T* y, const T* d, const T* x, bool ldiv);  // y = d.*x or x./d
template <class T> void k_blockdiag_mul(Ctx& c, int n, int bs, const T* blocks, const T* x, T* y);   // y = blockdiag(B_k) x
template <class T> void k_blockdiag_invert(Ctx& c, int n, int bs, const T* blocks, T* inv, int* singular);  // per-block inverse
// row-partitioned solves (no-ops on a single GPU)
double k_dist_sum(Ctx& c, double v);                                   // sum of a host scalar over all ranks
void dist_agree_on_exit(Ctx& c, bool& user_exit, bool& overtimed);     // OR the exit flags over the ranks
void dist_check_alive(Ctx& c);                                         // throws once a reduction has timed out
// A NaN scalar read back on a row-partitioned workspace may be the mark of a dead communicator (every reduction
// returns NaN from then on): raise at once instead of iterating on NaNs until itmax.
inline void dist_nan_guard(Ctx& c, double v) { if (c.dcomm && v != v) dist_check_alive(c); }

// ---------------------------------------------------------------------------
// CSR operator resident in HBM (int32 indices, 0-based, columns ascending).
// ---------------------------------------------------------------------------
constexpr int kTileRows = 256;   // rows per TMA-staged tile (= consumer threads per CTA)

template <class T>
struct Csr {
  int n = 0;
  long long nnz = 0;
  int* rowptr = nullptr;    // n+1 (+ pad)
  int* colind = nullptr;    // nnz (+ pad)
  T* val = nullptr;         // nnz (+ pad)
  // TMA staging plan (filled by plan()):
  int ntiles = 0;
  int tile_cap = 0;         // max nnz of any kTileRows-row tile
  int max_row = 0;          // longest row
  int max_col = -1;         // largest column index (validated against the number of columns when a solve starts)
  bool tma_ok = false;      // tile fits the shared-memory stage budget
  int stages = 0;           // pipeline depth chosen for tile_cap
  size_t smem_bytes = 0;    // dynamic smem of the staged kernels
  int grid = 0;             // persistent grid (multiple of the SM count)
  int ctas_per_sm = 0;      // resident CTAs per SM the ring was sized for
  // Dictionary encoding (built by plan() when the operator has at most kDictMax distinct (column - row, value)
  // pairs, as stencil and structured-grid operators do).  The staged SpMV and the persistent CG kernel then stream
  // one code byte per nonzero instead of colind + val; every other kernel keeps reading the CSR arrays above.
  uint8_t* code = nullptr;  // nnz (+ pad): index into the dictionary of each nonzero, in the stored order
  void* dict = nullptr;     // kDictMax int32 column offsets, then kDictMax T values (sorted by offset, bit pattern)
  int ndict = 0;            // dictionary entries in use; 0: no encoding
  int dict_stages = 0;      // ring depth of the encoded pipeline (same grid and CTAs per SM as the CSR plan)
  size_t dict_smem_bytes = 0;
};
constexpr int kDictMax = 256;

template <class T> void csr_upload(Ctx& c, Csr<T>& A, int n, long long nnz, const void* rowptr, const void* colind,
                                   const T* val, int index_base, int index_bytes, bool on_device);
template <class T> void csr_free(Csr<T>& A);
template <class T> void csr_plan(Ctx& c, Csr<T>& A);
// y = A x.  variant: 0 auto (TMA-staged when the plan allows), 1 force row-per-thread LDG, 2 force TMA-staged
template <class T> void k_spmv(Ctx& c, const Csr<T>& A, const T* x, T* y, int variant = 0);
// Row-partitioned operators: send this rank's boundary entries of x to the peers' halo buffers and meet in the
// in-kernel barrier (no-op on a single GPU).  Every y = A x on a distributed workspace is preceded by one.
template <class T> void k_halo_exchange(Ctx& c, const T* x);

// ---------------------------------------------------------------------------
// Operators as the solvers see them (A, M, N of the reference's kwargs).
// ---------------------------------------------------------------------------
typedef void (*MatvecFn)(const void* x, void* y, void* userdata);

template <class T>
struct LinOp {
  enum Kind { NONE, CSR, DIAG, BDIAG, HOST_CB, DEV_CB } kind = NONE;
  const Csr<T>* csr = nullptr;
  const T* diag = nullptr;       // DIAG: y = diag .* x (or x ./ diag with ldiv)
  const T* blocks = nullptr;     // BDIAG: dense bs x bs diagonal blocks, row-major, ceil(n / bs) of them (block-Jacobi)
  const T* blocks_inv = nullptr; //        their inverses (ldiv = true applies these)
  int bs = 0;
  MatvecFn fn = nullptr;         // callbacks: host pointers (HOST_CB) or device pointers (DEV_CB)
  void* userdata = nullptr;
  T* hx = nullptr;               // pinned staging for HOST_CB
  T* hy = nullptr;
  int n = 0;
  bool is_identity() const { return kind == NONE; }
};
template <class T> void op_apply(Ctx& c, const LinOp<T>& op, const T* x, T* y, bool ldiv = false);

// ---------------------------------------------------------------------------
// Solver options / statistics (kwargs of cg!/gmres!/bicgstab!/minres!;
// SimpleStats, src/krylov_stats.jl:24-36).
// ---------------------------------------------------------------------------
struct SolveOpts {
  double atol = -1, rtol = -1;      // <0 => sqrt(eps(T))
  int itmax = 0;                    // 0 => 2n
  double timemax = 1.0 / 0.0;
  int verbose = 0;
  bool history = false;
  double radius = 0;                // CG
  bool linesearch = false;          // CG, MINRES
  double lambda = 0;                // MINRES
  double etol = -1, conlim = -1;    // MINRES (<0 => defaults)
  bool restart = false;             // GMRES, FOM, FGMRES
  bool reorthogonalization = false; // GMRES, FOM, FGMRES
  bool check_curvature = false;     // CG-Lanczos
  double cr_gamma = -1;             // CR: kwarg γ (<0 => sqrt(eps(T)))
  bool ldiv = false;
  int (*callback)(void* ws, void* user) = nullptr;   // returns nonzero => user-requested exit
  void* callback_user = nullptr;
  int fused = 1;                    // 0 => force the generic primitive path
  int batch = 0;                    // fused CG: iterations enqueued per host poll (0 => default)
  int time_kernels = 0;             // fused CG: bracket the first launches of K1/K2 with CUDA events
  int persist = 1;                  // fused CG: 0 => keep the two-launch kernels instead of the persistent one
};

struct Stats {
  int niter = 0;
  bool solved = false, inconsistent = false, indefinite = false;
  int npcCount = 0;
  std::vector<double> residuals, Aresiduals, Acond;
  double allocation_timer = 0, timer = 0;
  double Anorm = NAN;                  // LanczosStats (cg_lanczos!)
  std::string status = "unknown";
  void reset() { residuals.clear(); Aresiduals.clear(); Acond.clear(); indefinite = false; npcCount = 0; }
};

// values of KrylovSolverType (interfaces/include/krylov.h:48-83); cg_lanczos has no slot in the reference's C enum
enum SolverKind { S_CG = 0, S_CR = 1, S_MINRES = 3, S_DIOM = 5, S_DQGMRES = 6, S_FOM = 7, S_GMRES = 8, S_FGMRES = 9, S_BICGSTAB = 10,
                  S_CGS = 11, S_CG_LANCZOS = 100 };

// One workspace per (solver, dtype): owns every device vector of the solver
// (src/krylov_workspaces.jl; SURVEY.md appendix B for fields and aliasing).
template <class T>
struct Workspace {
  SolverKind kind;
  int m = 0, n = 0;
  Ctx ctx;
  Stats stats;
  bool warm_start = false;
  // device vectors (nullptr == Julia's length-0 vector)
  T *x = nullptr, *dx = nullptr;
  T *r = nullptr, *p = nullptr, *Ap = nullptr, *z = nullptr, *npc_dir = nullptr;      // CG
  T *p2 = nullptr;                                                                   // CG fused: second p buffer
  T *v = nullptr, *s = nullptr, *qd = nullptr, *t = nullptr, *yz = nullptr;           // BiCGSTAB (+ r, p)
  T *r1 = nullptr, *r2 = nullptr, *w1 = nullptr, *w2 = nullptr, *y = nullptr, *vv = nullptr;  // MINRES
  T *w = nullptr, *q = nullptr, *pp = nullptr;                                        // GMRES / FOM / FGMRES (+ V)
  T *u = nullptr, *ts = nullptr, *vw = nullptr;                                       // CGS (+ r, p, q, yz)
  T *Mv = nullptr, *Mv_prev = nullptr, *Mv_next = nullptr;                            // CG-Lanczos (+ p, vv)
  std::vector<T*> V;
  std::vector<T*> Z;                   // FGMRES: Z[k] = N_k V[k];  DQGMRES / DIOM: the direction stack P
  std::vector<T> c, sgiv, zg, R;       // GMRES host-side Givens data
  std::vector<T> err_vec;              // MINRES window
  int memory = 20, window = 5;
  int inner_iter = 0;
  const T* mdiag_fused = nullptr;      // diagonal of M for the fused CG kernels (set per solve; nullptr: M = I)
  const T* mblocks_fused = nullptr;    // block-Jacobi M for the persistent CG kernel (set per solve; nullptr: none)
  int mbs_fused = 0;
  double k1_ms = 0, k2_ms = 0;         // average event-timed duration of the fused kernels (time_kernels)
  int timed_pairs = 0;
  void* fused_state = nullptr;         // device scalar block of the fused paths
  void* fused_host = nullptr;          // pinned mirror (2 slots)
  cudaEvent_t fused_ev[2] = {nullptr, nullptr};   // fused CG: one event per read-back slot
  unsigned long long fused_seq = 0;               // persistent CG: sequence number of the last launch (host-polled report)
  T* bbuf = nullptr;                   // device copies of host b / c for the C ABI
  T* cbuf = nullptr;
  // row-partitioned (multi-GPU) state; world == 1 means single GPU
  struct Dist {
    int rank = 0, world = 1;
    HaloMap halo{0, 0, nullptr, nullptr};      // device arrays
    void* mailbox = nullptr;                    // local mailbox allocation (values + flags)
    T* bufA_peer[kMaxRanks] = {};               // every rank's `p` allocation (as created)
    T* bufB_peer[kMaxRanks] = {};               // every rank's `p2` allocation
    T* r_peer[kMaxRanks] = {};
    std::vector<void*> opened;                  // cudaIpcOpenMemHandle results to close
    bool swapped = false;                       // ws.p currently points at the bufB allocation
    T* halo_buf = nullptr;                      // local halo buffers [r | p(bufA) | p(bufB)], nhalo entries each
    T* halo_buf_peer[kMaxRanks] = {};           // every rank's halo_buf
    int nhalo_peer[kMaxRanks] = {};             // every rank's halo length (section stride inside its halo_buf)
    void* dummy[3] = {nullptr, nullptr, nullptr};  // placeholder IPC exports of the non-CG solvers
    T* xhalo = nullptr;                         // general x-halo buffer (2 sections) of k_halo_exchange
    T* xhalo_peer[kMaxRanks] = {};
    int nsend = 0;                              // send list of the general exchange (device arrays)
    int* send_row = nullptr; int* send_peer = nullptr; int* send_slot = nullptr;
    long long nglobal = 0;                      // global number of rows (default itmax = 2 n)
    int npush = 0;                              // > 0: push mode (contiguous send ranges), else pull mode
    int* tile_order = nullptr;                  // persistent CG: interior tiles first, halo tiles last (device)
    const void* tile_order_for = nullptr;       // ... built for this operator
    int tile_order_n = 0;
    int tile_order_interior = 0;                // number of tiles without halo columns (they come first)
    PushRange push[kMaxPushRanges];
  } dist;
};

template <class T> Workspace<T>* ws_create(SolverKind kind, int m, int n, int memory, int window, int device);
template <class T> void ws_destroy(Workspace<T>* ws);
template <class T> void ws_warm_start(Workspace<T>* ws, const T* x0_dev);

// Solver drivers (device pointers for b, c).  Throw std::runtime_error where
// the reference calls error(...).
template <class T> void cg_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const SolveOpts& o);
template <class T> void gmres_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void bicgstab_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const T* c, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void minres_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const SolveOpts& o);
// Sibling solvers on the same kernels (siblings.cu; SURVEY.md 8f-3)
template <class T> void cgs_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const T* c, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void cg_lanczos_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const SolveOpts& o);
template <class T> void fom_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void fgmres_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void dqgmres_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void diom_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const LinOp<T>& N, const SolveOpts& o);
template <class T> void cr_solve(Workspace<T>& ws, const LinOp<T>& A, const T* b, const LinOp<T>& M, const SolveOpts& o);

// Fused CG (cg_fused.cu).  Returns false if the configuration is not eligible
// (caller falls back to the generic primitive path, still on the GPU).
template <class T> bool cg_fused_eligible(const LinOp<T>& A, const LinOp<T>& M, const SolveOpts& o);
template <class T> void cg_dist_push_r(Workspace<T>& ws);
template <class T> void cg_fused_prepare(Workspace<T>& ws);   // device/pinned scalar blocks, p2, events (ws_create)
constexpr size_t kFusedBlockBytes = 4096;
template <class T> void cg_fused_loop(Workspace<T>& ws, const Csr<T>& A, const SolveOpts& o, T gamma0, T eps_tol, int itmax,
                                      double start_time, bool& solved, bool& tired, bool& zero_curvature,
                                      bool& inconsistent, bool& user_exit, bool& overtimed, int& iter);

// Fused iteration phases of BiCGSTAB / MINRES / GMRES (fused_phases.cu); eligible when A is a CSR operator,
// M = N = I (and for GMRES no reorthogonalization).
template <class T> void bicgstab_fused_iteration(Workspace<T>& ws, const Csr<T>& A, const T* cvec, bool first, T rho_in, T* alpha,
                                                 T* omega, T* next_rho, T* rNorm);
template <class T> void minres_fused_lanczos(Workspace<T>& ws, const Csr<T>& A, int iter, T lambda, T beta, T oldbeta, T cs, T sn,
                                             T deltabar, T eps_rot, T* w, T* alpha, T* beta2);
template <class T> T minres_fused_update(Workspace<T>& ws, T* w, T gamma, T phi);
// xin: vector the operator is applied to (default V[k]; FGMRES passes Z[k])
template <class T> void gmres_fused_arnoldi(Workspace<T>& ws, const Csr<T>& A, int k, T* h_out, T* Hbis, const T* xin = nullptr);
template <class T> void fused_multi_axpy(Workspace<T>& ws, T* xr, int k, const T* y, T* const* vecs);
// sibling solvers (fused_phases.cu): grouped passes with host-side scalars
template <class T> void fused_orth_chain(Workspace<T>& ws, const Csr<T>& A, const T* xin, T* q, const T* const* vecs, int cnt, T* h_out, T* Hbis);
template <class T> void trunc_fused_direction(Workspace<T>& ws, T* pp, int cnt, T* const* pvecs, const T* coefs, const T* z, T h0, T step);
template <class T> T cgs_fused_sigma(Workspace<T>& ws, const Csr<T>& A, const T* cvec);
template <class T> void cgs_fused_update(Workspace<T>& ws, const Csr<T>& A, const T* cvec, T alpha, T* rho_next, T* rr);
template <class T> void cgs_fused_directions(Workspace<T>& ws, T beta);
template <class T> T lanczos_fused_delta(Workspace<T>& ws, const Csr<T>& A);
template <class T> T lanczos_fused_recur(Workspace<T>& ws, T delta, T beta, bool later);
template <class T> void lanczos_fused_update(Workspace<T>& ws, T beta, T gamma, T sigma, T omega);
template <class T> void cr_fused_step(Workspace<T>& ws, const Csr<T>& A, T alpha, T* xx, T* rr, T* ArAr, T* rAr);
template <class T> T cr_fused_directions(Workspace<T>& ws, T beta);
template <class T> void gmres_fused_update_x(Workspace<T>& ws, T* xr, int k, const T* y);
int gmres_fused_max();

double now_seconds();

}  // namespace kb
