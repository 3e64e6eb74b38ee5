// capi.cu -- the C ABI declared in include/krylov_b200.h.
//
// Part 1 mirrors interfaces/src/LibKrylov.jl (entry points) and
// interfaces/src/c_stores.jl (handle store, option mapping) of the reference:
// never propagate exceptions, log to stderr, return -1; -2 for unknown
// (solver, dtype); free returns 1 for an unknown handle.  Unlike the reference
// (global typed Dicts, documented as not thread-safe) the handle table is a
// single mutex-protected map.
#include <cmath>
#include <cstring>
#include <memory>
#include <mutex>
#include <unordered_map>

#include "../../include/krylov_b200.h"
#include "kb_internal.h"
#include "block.h"
#include "mtx.h"
#include "dense_small.h"

using namespace kb;

namespace {

thread_local std::string g_last_error;
int g_device = -1;

struct CsrAny {
  int dtype = 1;
  Csr<double> d;
  Csr<float> f;
  Ctx* owner_ctx = nullptr;
  ~CsrAny() { csr_free(d); csr_free(f); }
};

struct Handle {
  int solver = 0, dtype = 1, device_kind = 0;
  bool block = false;                  // ws is a BlockWorkspace (krylov_block_* entry points)
  int p = 0;
  void* ws = nullptr;
  std::shared_ptr<CsrAny> csr;
  void* Mdiag = nullptr;
  void* Ndiag = nullptr;
  void* Pblk[2] = {nullptr, nullptr};      // block-Jacobi M / N: dense diagonal blocks (device) ...
  void* Pblk_inv[2] = {nullptr, nullptr};  // ... and their inverses (ldiv = true)
  int Pbs[2] = {0, 0};
  KrylovB200Options ext;
  void *hx = nullptr, *hy = nullptr;   // pinned staging for host callbacks
};

std::mutex g_mu;
std::unordered_map<void*, Handle*> g_handles;

Handle* lookup_any(void* p) {
  std::lock_guard<std::mutex> lk(g_mu);
  auto it = g_handles.find(p);
  return it == g_handles.end() ? nullptr : it->second;
}
// single-RHS entry points only accept single-RHS handles, block entry points only block handles
Handle* lookup(void* p) { Handle* h = lookup_any(p); return (h && !h->block) ? h : nullptr; }
Handle* lookup_block(void* p) { Handle* h = lookup_any(p); return (h && h->block) ? h : nullptr; }

int fail(const char* where, const std::exception& e) {
  g_last_error = std::string(where) + ": " + e.what();
  fprintf(stderr, "[krylov_b200] %s\n", g_last_error.c_str());
  return -1;
}
int fail(const char* where, const char* msg) {
  g_last_error = std::string(where) + ": " + msg;
  fprintf(stderr, "[krylov_b200] %s\n", g_last_error.c_str());
  return -1;
}

bool supported_solver(int s) {
  return s == S_CG || s == S_MINRES || s == S_GMRES || s == S_BICGSTAB || s == S_FOM || s == S_FGMRES || s == S_CGS ||
         s == S_CG_LANCZOS || s == S_CR || s == S_DIOM || s == S_DQGMRES;
}

int pick_device() {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt <= 0) {
    cudaGetLastError();
    throw std::runtime_error("no usable CUDA device: libkrylov_b200 has no CPU compute path");
  }
  int dev = g_device;
  if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
  if (dev >= cnt) throw std::runtime_error("device index out of range");
  cudaDeviceProp prop;
  KB_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major < 10) throw std::runtime_error("libkrylov_b200 is built for sm_100a only");
  return dev;
}

template <class T> Workspace<T>* W(Handle* h) { return reinterpret_cast<Workspace<T>*>(h->ws); }
template <class T> BlockWorkspace<T>* BW(Handle* h) { return reinterpret_cast<BlockWorkspace<T>*>(h->ws); }
// what the entry points shared by both handle kinds need
Ctx& ctx_of(Handle* h) {
  if (h->block) return h->dtype == KRYLOV_FLOAT64 ? BW<double>(h)->ctx : BW<float>(h)->ctx;
  return h->dtype == KRYLOV_FLOAT64 ? W<double>(h)->ctx : W<float>(h)->ctx;
}
int n_of(Handle* h) {
  if (h->block) return h->dtype == KRYLOV_FLOAT64 ? BW<double>(h)->n : BW<float>(h)->n;
  return h->dtype == KRYLOV_FLOAT64 ? W<double>(h)->n : W<float>(h)->n;
}
template <class T> Csr<T>& csr_of(CsrAny& a);
template <> Csr<double>& csr_of<double>(CsrAny& a) { return a.d; }
template <> Csr<float>& csr_of<float>(CsrAny& a) { return a.f; }

template <class T> void destroy_handle(Handle* h) {
  Workspace<T>* ws = W<T>(h);
  if (ws) {
    KB_CUDA(cudaSetDevice(ws->ctx.device));
    if (ws->ctx.stream) cudaStreamSynchronize(ws->ctx.stream);
  }
  h->csr.reset();
  dev_free(h->Mdiag); dev_free(h->Ndiag);
  for (int w = 0; w < 2; w++) { dev_free(h->Pblk[w]); dev_free(h->Pblk_inv[w]); }
  if (h->hx) cudaFreeHost(h->hx);
  if (h->hy) cudaFreeHost(h->hy);
  ws_destroy<T>(ws);
  delete h;
}

// Bring a caller vector (host or device, per device_kind) into a device buffer.
template <class T> const T* stage_in(Handle* h, Workspace<T>* ws, const void* src, T*& buf) {
  if (!src) return nullptr;
  if (h->device_kind == KRYLOV_CUDA) return (const T*)src;
  if (!buf) buf = dev_alloc<T>((size_t)ws->n);
  KB_CUDA(cudaMemcpyAsync(buf, src, sizeof(T) * (size_t)ws->n, cudaMemcpyHostToDevice, ws->ctx.stream));
  return buf;
}

template <class T> LinOp<T> make_cb_op(Handle* h, Workspace<T>* ws, KrylovMatvec fn, void* ud) {
  LinOp<T> op;
  op.n = ws->n;
  if (!fn) return op;
  op.fn = fn; op.userdata = ud;
  if (h->device_kind == KRYLOV_CUDA) { op.kind = LinOp<T>::DEV_CB; return op; }
  op.kind = LinOp<T>::HOST_CB;
  if (!h->hx) {
    KB_CUDA(cudaHostAlloc(&h->hx, sizeof(T) * (size_t)ws->n, cudaHostAllocDefault));
    KB_CUDA(cudaHostAlloc(&h->hy, sizeof(T) * (size_t)ws->n, cudaHostAllocDefault));
  }
  op.hx = (T*)h->hx; op.hy = (T*)h->hy;
  return op;
}

// _opts_kw + per-family kwargs (interfaces/src/c_stores.jl:255-260, 288-300 CG,
// 303-315 MINRES, 334-354 BiCGSTAB, 377-398 GMRES)
SolveOpts map_opts(const Handle* h, const KrylovOptions* o) {
  SolveOpts s;
  KrylovOptions d = krylov_default_options();
  if (!o) o = &d;
  s.atol = std::isnan(o->atol) ? -1 : o->atol;
  s.rtol = std::isnan(o->rtol) ? -1 : o->rtol;
  s.itmax = o->itmax;
  s.verbose = o->verbose;
  s.timemax = std::isnan(o->timemax) ? INFINITY : o->timemax;
  if (h->solver == S_CG || h->solver == S_CR) { s.radius = o->radius; s.linesearch = o->linesearch != 0; }   // _typed_solve_cg!
  if (h->solver == S_DIOM || h->solver == S_DQGMRES) s.reorthogonalization = o->reorthogonalization != 0;      // _typed_solve_mn_reorth!
  s.cr_gamma = std::isnan(h->ext.cr_gamma) ? -1 : h->ext.cr_gamma;
  if (h->solver == S_MINRES) { s.lambda = o->lambda; s.linesearch = o->linesearch != 0; }
  // _typed_solve_gmres! serves GMRES, FGMRES and FOM (c_stores.jl:376-398)
  if (h->solver == S_GMRES || h->solver == S_FGMRES || h->solver == S_FOM) {
    s.restart = o->restart != 0; s.reorthogonalization = o->reorthogonalization != 0;
  }
  s.check_curvature = h->ext.check_curvature != 0;
  s.history = h->ext.history != 0;
  s.ldiv = h->ext.ldiv != 0;
  s.etol = std::isnan(h->ext.etol) ? -1 : h->ext.etol;
  s.conlim = std::isnan(h->ext.conlim) ? -1 : h->ext.conlim;
  s.fused = h->ext.fused;
  s.persist = h->ext.fused != 2;       // fused == 2: fused CG keeps the two-launch kernels (A/B measurements, tests)
  s.batch = h->ext.batch;
  s.callback = h->ext.callback;
  s.callback_user = h->ext.callback_user;
  s.time_kernels = h->ext.time_kernels;
  return s;
}

template <class T>
int do_solve(Handle* h, KrylovMatvec fA, KrylovMatvec fM, KrylovMatvec fN, const void* b, const void* c, void* ud,
             const KrylovOptions* opts) {
  Workspace<T>* ws = W<T>(h);
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  SolveOpts so = map_opts(h, opts);
  LinOp<T> A;
  if (fA) A = make_cb_op<T>(h, ws, fA, ud);
  else if (h->csr) {
    A.kind = LinOp<T>::CSR; A.csr = &csr_of<T>(*h->csr); A.n = ws->n;
    // columns: n local ones plus, row-partitioned, the halo entries -- anything beyond is an out-of-bounds gather
    const long long ncols = (long long)ws->n + (ws->dist.world > 1 ? ws->dist.halo.nhalo : 0);
    if (A.csr->n != ws->n || A.csr->max_col >= ncols)
      throw std::runtime_error("CSR operator: size or column index inconsistent with the workspace (n = " + std::to_string(ws->n) +
                               ", operator rows = " + std::to_string(A.csr->n) + ", largest column = " + std::to_string(A.csr->max_col) + ")");
  }
  else throw std::runtime_error("no operator: pass matvec_A or attach one with krylov_b200_set_operator_csr");
  if (A.kind == LinOp<T>::CSR && A.csr->n != ws->n) throw std::runtime_error("(workspace.m, workspace.n) is inconsistent with size(A)");
  LinOp<T> M = make_cb_op<T>(h, ws, fM, ud), N = make_cb_op<T>(h, ws, fN, ud);
  if (!fM && h->Mdiag) { M.kind = LinOp<T>::DIAG; M.diag = (const T*)h->Mdiag; }
  if (!fN && h->Ndiag) { N.kind = LinOp<T>::DIAG; N.diag = (const T*)h->Ndiag; }
  if (!fM && !h->Mdiag && h->Pblk[0]) { M.kind = LinOp<T>::BDIAG; M.blocks = (const T*)h->Pblk[0]; M.blocks_inv = (const T*)h->Pblk_inv[0]; M.bs = h->Pbs[0]; M.n = ws->n; }
  if (!fN && !h->Ndiag && h->Pblk[1]) { N.kind = LinOp<T>::BDIAG; N.blocks = (const T*)h->Pblk[1]; N.blocks_inv = (const T*)h->Pblk_inv[1]; N.bs = h->Pbs[1]; N.n = ws->n; }
  if (!b) throw std::runtime_error("b is NULL");
  const T* bd = stage_in<T>(h, ws, b, ws->bbuf);
  dist_check_alive(ws->ctx);             // row-partitioned: refuse to start on a dead communicator
  switch (h->solver) {
    case S_CG: cg_solve<T>(*ws, A, bd, M, so); break;
    case S_MINRES: minres_solve<T>(*ws, A, bd, M, so); break;
    case S_GMRES: gmres_solve<T>(*ws, A, bd, M, N, so); break;
    case S_FOM: fom_solve<T>(*ws, A, bd, M, N, so); break;
    case S_FGMRES: fgmres_solve<T>(*ws, A, bd, M, N, so); break;
    case S_CG_LANCZOS: cg_lanczos_solve<T>(*ws, A, bd, M, so); break;
    case S_CR: cr_solve<T>(*ws, A, bd, M, so); break;
    case S_DQGMRES: dqgmres_solve<T>(*ws, A, bd, M, N, so); break;
    case S_DIOM: diom_solve<T>(*ws, A, bd, M, N, so); break;
    case S_CGS: {
      const T* cd = stage_in<T>(h, ws, c, ws->cbuf);
      cgs_solve<T>(*ws, A, bd, cd, M, N, so);
      break;
    }
    case S_BICGSTAB: {
      // the reference's C layer never forwards `c` for BiCGSTAB (c = b); we accept it when given
      const T* cd = stage_in<T>(h, ws, c, ws->cbuf);
      bicgstab_solve<T>(*ws, A, bd, cd, M, N, so);
      break;
    }
  }
  dist_check_alive(ws->ctx);             // a reduction timed out during the solve: raise instead of returning NaNs
  return 0;
}

template <class T> int do_get_x(Handle* h, void* x, int n) {
  Workspace<T>* ws = W<T>(h);
  if (n > ws->n) n = ws->n;
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  KB_CUDA(cudaMemcpyAsync(x, ws->x, sizeof(T) * (size_t)n,
                          h->device_kind == KRYLOV_CUDA ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ws->ctx.stream));
  ws->ctx.sync();
  return 0;
}

template <class T> int do_warm_start(Handle* h, const void* x0, int n) {
  Workspace<T>* ws = W<T>(h);
  if (n != ws->n) throw std::runtime_error("x0 should have size n");
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  // c_stores.jl:218-229: allocate dx if empty, copy, set the flag
  if (!ws->dx) ws->dx = dev_alloc<T>((size_t)ws->n);
  KB_CUDA(cudaMemcpyAsync(ws->dx, x0, sizeof(T) * (size_t)n,
                          h->device_kind == KRYLOV_CUDA ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ws->ctx.stream));
  ws->ctx.sync();
  ws->warm_start = true;
  return 0;
}

template <class T> Stats& stats_of(Handle* h) { return W<T>(h)->stats; }
Stats& stats_any(Handle* h) {
  if (h->block) return h->dtype == KRYLOV_FLOAT64 ? BW<double>(h)->stats : BW<float>(h)->stats;
  return h->dtype == KRYLOV_FLOAT64 ? stats_of<double>(h) : stats_of<float>(h);
}

template <class T> void* vec_by_name(Workspace<T>* ws, const char* nm) {
  struct { const char* n; T* p; } tab[] = {
      {"x", ws->x}, {"dx", ws->dx}, {"r", ws->r}, {"p", ws->p}, {"Ap", ws->Ap}, {"z", ws->z}, {"npc_dir", ws->npc_dir},
      {"v", ws->kind == S_MINRES ? (ws->vv ? ws->vv : ws->r2) : ws->v}, {"s", ws->s}, {"qd", ws->qd}, {"t", ws->t}, {"yz", ws->yz},
      {"r1", ws->r1}, {"r2", ws->r2}, {"w1", ws->w1}, {"w2", ws->w2}, {"y", ws->y}, {"w", ws->w}, {"q", ws->q},
      {"u", ws->u}, {"ts", ws->ts}, {"vw", ws->vw}, {"Mv", ws->Mv}, {"Mv_prev", ws->Mv_prev}, {"Mv_next", ws->Mv_next}};
  for (auto& e : tab) if (!strcmp(e.n, nm)) return e.p;
  if (nm[0] == 'P' && nm[1]) { int i = atoi(nm + 1); if (i >= 1 && i <= (int)ws->Z.size()) return ws->Z[i - 1]; return nullptr; }
  if (!strcmp(nm, "Ar")) return ws->Ap;
  if (!strcmp(nm, "Mq")) return ws->z;
  if (nm[0] == 'Z') { int i = atoi(nm + 1); if (i >= 1 && i <= (int)ws->Z.size()) return ws->Z[i - 1]; return nullptr; }
  if (nm[0] == 'V') { int i = atoi(nm + 1); if (i >= 1 && i <= (int)ws->V.size()) return ws->V[i - 1]; }
  return nullptr;
}

}  // namespace

extern "C" {

// ------------------------------- part 1 -----------------------------------
int krylov_workspace_create(KrylovSolverType solver, int m, int n, KrylovDataType dtype, KrylovDeviceType device,
                            const KrylovWorkspaceOptions* wopts, void** ws_out) {
  try {
    if (!supported_solver((int)solver) || (dtype != KRYLOV_FLOAT32 && dtype != KRYLOV_FLOAT64)) return -2;
    if (device != KRYLOV_CPU && device != KRYLOV_CUDA) return fail("krylov_workspace_create", "unknown device");
    if (!ws_out) return fail("krylov_workspace_create", "ws_out is NULL");
    if (m < 0 || n < 0) return fail("krylov_workspace_create", "negative dimension");
    const int dev = pick_device();
    const int memory = wopts ? wopts->memory : 0, window = wopts ? wopts->window : 0;   // 0 -> 20 / 5 (c_stores.jl:1799-1800)
    Handle* h = new Handle();
    h->solver = (int)solver; h->dtype = (int)dtype; h->device_kind = (int)device;
    h->ext = krylov_b200_default_options();
    try {
      if (dtype == KRYLOV_FLOAT64) h->ws = ws_create<double>((SolverKind)solver, m, n, memory, window, dev);
      else h->ws = ws_create<float>((SolverKind)solver, m, n, memory, window, dev);
    } catch (...) { delete h; throw; }
    {
      std::lock_guard<std::mutex> lk(g_mu);
      g_handles[h] = h;
    }
    *ws_out = h;
    return 0;
  } catch (const std::exception& e) { return fail("krylov_workspace_create", e); }
}

KrylovWorkspaceOptions krylov_default_workspace_options(void) { KrylovWorkspaceOptions w = {0, 0}; return w; }

KrylovOptions krylov_default_options(void) {
  KrylovOptions o;
  o.atol = NAN; o.rtol = NAN; o.itmax = 0; o.verbose = 0; o.lambda = 0.0; o.tau = NAN; o.nu = NAN;
  o.timemax = NAN; o.radius = 0.0; o.restart = 0; o.reorthogonalization = 0; o.linesearch = 0;
  return o;
}

void krylov_get_version(int* major, int* minor, int* patch) {
  if (major) *major = KRYLOV_VERSION_MAJOR;
  if (minor) *minor = KRYLOV_VERSION_MINOR;
  if (patch) *patch = KRYLOV_VERSION_PATCH;
}

int krylov_solve(void* ws, KrylovMatvec matvec_A, KrylovMatvec matvec_At, KrylovMatvec matvec_M, KrylovMatvec matvec_N,
                 const void* b, const void* c, void* userdata, const KrylovOptions* opts) {
  (void)matvec_At;   // none of CG / MINRES / GMRES / BiCGSTAB uses the adjoint
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_solve", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? do_solve<double>(h, matvec_A, matvec_M, matvec_N, b, c, userdata, opts)
                                      : do_solve<float>(h, matvec_A, matvec_M, matvec_N, b, c, userdata, opts);
  } catch (const std::exception& e) { return fail("krylov_solve", e); }
}

int krylov_get_x(void* ws, void* x, int n) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_get_x", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? do_get_x<double>(h, x, n) : do_get_x<float>(h, x, n);
  } catch (const std::exception& e) { return fail("krylov_get_x", e); }
}

int krylov_get_y(void* ws, void* y, int m) {
  (void)y; (void)m;
  Handle* h = lookup(ws);
  if (!h) return fail("krylov_get_y", "unknown workspace handle");
  return -2;   // solution_count == 1 for the four solvers (c_stores.jl:211-216)
}

int krylov_is_solved(void* ws) { Handle* h = lookup(ws); return h ? (stats_any(h).solved ? 1 : 0) : -1; }
int krylov_niter(void* ws) { Handle* h = lookup(ws); return h ? stats_any(h).niter : -1; }
double krylov_elapsed_time(void* ws) { Handle* h = lookup(ws); return h ? stats_any(h).timer : -1.0; }

int krylov_warm_start(void* ws, const void* x0, int n) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_warm_start", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? do_warm_start<double>(h, x0, n) : do_warm_start<float>(h, x0, n);
  } catch (const std::exception& e) { return fail("krylov_warm_start", e); }
}

int krylov_warm_start2(void* ws, const void* x0, const void* y0, int nx, int ny) {
  (void)x0; (void)y0; (void)nx; (void)ny;
  Handle* h = lookup(ws);
  if (!h) return fail("krylov_warm_start2", "unknown workspace handle");
  return -2;
}

// One destroy routine for both handle kinds: sets the handle's device, drops the operator and the preconditioner
// diagonals, frees the pinned callback staging and the workspace.
static void destroy_any(Handle* h) {
  if (h->block) {
    Ctx& c = ctx_of(h);
    KB_CUDA(cudaSetDevice(c.device));
    if (c.stream) cudaStreamSynchronize(c.stream);
    h->csr.reset();
    dev_free(h->Mdiag); dev_free(h->Ndiag);
    if (h->hx) cudaFreeHost(h->hx);
    if (h->hy) cudaFreeHost(h->hy);
    if (h->dtype == KRYLOV_FLOAT64) block_ws_destroy<double>(BW<double>(h)); else block_ws_destroy<float>(BW<float>(h));
    delete h;
  } else if (h->dtype == KRYLOV_FLOAT64) {
    destroy_handle<double>(h);
  } else {
    destroy_handle<float>(h);
  }
}

// Frees a single-RHS workspace; a block handle passed here is forwarded to the block destroy path (the reference
// keeps one key store for both kinds, c_stores.jl:1652-1655).  Unknown handle -> 1 (double free is safe).
int krylov_workspace_free(void* ws) {
  Handle* h = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_handles.find(ws);
    if (it == g_handles.end()) return 1;
    h = it->second;
    g_handles.erase(it);
  }
  try {
    destroy_any(h);
  } catch (const std::exception& e) { fail("krylov_workspace_free", e); }
  return 0;
}

// Block solvers: outside the path (SURVEY.md section 8f-2).
// Block solvers (interfaces/src/LibKrylov.jl block entry points; krylov.h:246-285).  block_gmres only:
// KRYLOV_BLOCK_MINRES answers -2.  B, X, X0 are the reference's column-major n x p blocks.
int krylov_block_workspace_create(KrylovBlockSolverType solver, int m, int n, int p, KrylovDataType dtype, KrylovDeviceType device,
                                  const KrylovWorkspaceOptions* wopts, void** ws_out) {
  try {
    if (solver != KRYLOV_BLOCK_GMRES || (dtype != KRYLOV_FLOAT32 && dtype != KRYLOV_FLOAT64)) return -2;
    if (device != KRYLOV_CPU && device != KRYLOV_CUDA) return fail("krylov_block_workspace_create", "unknown device");
    if (!ws_out) return fail("krylov_block_workspace_create", "ws_out is NULL");
    if (m < 0 || n < 0 || p < 1) return fail("krylov_block_workspace_create", "bad dimensions");
    const int dev = pick_device();
    const int memory = wopts ? wopts->memory : 0;
    Handle* h = new Handle();
    h->block = true; h->p = p; h->solver = (int)solver; h->dtype = (int)dtype; h->device_kind = (int)device;
    h->ext = krylov_b200_default_options();
    try {
      if (dtype == KRYLOV_FLOAT64) h->ws = block_ws_create<double>(m, n, p, memory, dev);
      else h->ws = block_ws_create<float>(m, n, p, memory, dev);
    } catch (...) { delete h; throw; }
    {
      std::lock_guard<std::mutex> lk(g_mu);
      g_handles[h] = h;
    }
    *ws_out = h;
    return 0;
  } catch (const std::exception& e) { return fail("krylov_block_workspace_create", e); }
}

}  // extern "C" (templates below need C++ linkage)
namespace {
template <class T> BlockOp<T> make_block_cb(Handle* h, KrylovBlockMatvec fn, void* ud) {
  BlockOp<T> op;
  if (!fn) return op;
  op.fn = fn; op.userdata = ud;
  op.kind = h->device_kind == KRYLOV_CUDA ? BlockOp<T>::DEV_CB : BlockOp<T>::HOST_CB;
  return op;
}
// caller block (host or device, column-major) -> device column-major staging in ws.tmp2
template <class T> const T* stage_block(Handle* h, BlockWorkspace<T>* ws, const void* src) {
  if (h->device_kind == KRYLOV_CUDA) return (const T*)src;
  const size_t np = (size_t)ws->n * ws->p;
  if (!ws->tmp2) ws->tmp2 = dev_alloc<T>(np);
  KB_CUDA(cudaMemcpyAsync(ws->tmp2, src, sizeof(T) * np, cudaMemcpyHostToDevice, ws->ctx.stream));
  return ws->tmp2;
}
template <class T> int do_block_solve(Handle* h, KrylovBlockMatvec fA, KrylovBlockMatvec fM, KrylovBlockMatvec fN, const void* B,
                                      void* ud, const KrylovOptions* opts) {
  BlockWorkspace<T>* ws = BW<T>(h);
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  SolveOpts so = map_opts(h, opts);
  KrylovOptions d = krylov_default_options();
  const KrylovOptions* o = opts ? opts : &d;
  so.restart = o->restart != 0; so.reorthogonalization = o->reorthogonalization != 0;
  BlockOp<T> A = make_block_cb<T>(h, fA, ud);
  if (!fA) {
    if (!h->csr) throw std::runtime_error("no operator: pass matvec_A or attach one with krylov_b200_set_operator_csr");
    A.kind = BlockOp<T>::CSR; A.csr = &csr_of<T>(*h->csr);
    if (A.csr->n != ws->n) throw std::runtime_error("(workspace.m, workspace.n) is inconsistent with size(A)");
  }
  BlockOp<T> M = make_block_cb<T>(h, fM, ud), N = make_block_cb<T>(h, fN, ud);
  if (!fM && h->Mdiag) { M.kind = BlockOp<T>::DIAG; M.diag = (const T*)h->Mdiag; }
  if (!fN && h->Ndiag) { N.kind = BlockOp<T>::DIAG; N.diag = (const T*)h->Ndiag; }
  if (!B) throw std::runtime_error("B is NULL");
  const T* Bd = stage_block<T>(h, ws, B);
  block_gmres_solve<T>(*ws, A, Bd, M, N, so);
  return 0;
}
template <class T> int do_block_get_X(Handle* h, void* X, int n, int p) {
  BlockWorkspace<T>* ws = BW<T>(h);
  if (n != ws->n || p != ws->p) throw std::runtime_error("X should have size n x p");
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  const size_t np = (size_t)n * p;
  if (h->device_kind == KRYLOV_CUDA) { block_get_X<T>(*ws, (T*)X); return 0; }
  block_get_X<T>(*ws, ws->tmp);
  KB_CUDA(cudaMemcpyAsync(X, ws->tmp, sizeof(T) * np, cudaMemcpyDeviceToHost, ws->ctx.stream));
  ws->ctx.sync();
  return 0;
}
template <class T> int do_block_warm_start(Handle* h, const void* X0, int n, int p) {
  BlockWorkspace<T>* ws = BW<T>(h);
  if (n != ws->n || p != ws->p) throw std::runtime_error("X0 should have size n x p");
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  block_warm_start<T>(*ws, stage_block<T>(h, ws, X0));
  return 0;
}
}  // namespace
extern "C" {

int krylov_block_solve(void* ws, KrylovBlockMatvec matvec_A, KrylovBlockMatvec matvec_M, KrylovBlockMatvec matvec_N, const void* B,
                       void* userdata, const KrylovOptions* opts) {
  try {
    Handle* h = lookup_block(ws);
    if (!h) return fail("krylov_block_solve", "unknown block workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? do_block_solve<double>(h, matvec_A, matvec_M, matvec_N, B, userdata, opts)
                                      : do_block_solve<float>(h, matvec_A, matvec_M, matvec_N, B, userdata, opts);
  } catch (const std::exception& e) { return fail("krylov_block_solve", e); }
}
int krylov_block_get_X(void* ws, void* X, int n, int p) {
  try {
    Handle* h = lookup_block(ws);
    if (!h || !X) return fail("krylov_block_get_X", "bad arguments");
    return h->dtype == KRYLOV_FLOAT64 ? do_block_get_X<double>(h, X, n, p) : do_block_get_X<float>(h, X, n, p);
  } catch (const std::exception& e) { return fail("krylov_block_get_X", e); }
}
int krylov_block_is_solved(void* ws) { Handle* h = lookup_block(ws); return h ? (stats_any(h).solved ? 1 : 0) : -1; }
int krylov_block_niter(void* ws) { Handle* h = lookup_block(ws); return h ? stats_any(h).niter : -1; }
double krylov_block_elapsed_time(void* ws) { Handle* h = lookup_block(ws); return h ? stats_any(h).timer : -1.0; }
int krylov_block_warm_start(void* ws, const void* x0, int n, int p) {
  try {
    Handle* h = lookup_block(ws);
    if (!h || !x0) return fail("krylov_block_warm_start", "bad arguments");
    return h->dtype == KRYLOV_FLOAT64 ? do_block_warm_start<double>(h, x0, n, p) : do_block_warm_start<float>(h, x0, n, p);
  } catch (const std::exception& e) { return fail("krylov_block_warm_start", e); }
}
long long krylov_b200_block_qr_fallbacks(void* ws) {
  Handle* h = lookup_block(ws);
  if (!h) return -1;
  return h->dtype == KRYLOV_FLOAT64 ? BW<double>(h)->qr_fallbacks : BW<float>(h)->qr_fallbacks;
}
int krylov_block_workspace_free(void* ws) {
  try {
    Handle* h = lookup_block(ws);
    if (!h) return 1;
    {
      std::lock_guard<std::mutex> lk(g_mu);
      g_handles.erase(ws);
    }
    destroy_any(h);
    return 0;
  } catch (const std::exception& e) { return fail("krylov_block_workspace_free", e); }
}

// ------------------------------- part 2 -----------------------------------
int krylov_b200_device_count(void) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess) { cudaGetLastError(); return 0; }
  return cnt;
}
int krylov_b200_set_device(int device) { g_device = device; return 0; }
const char* krylov_b200_last_error(void) { return g_last_error.c_str(); }

int krylov_b200_set_operator_csr(void* ws, int n, long long nnz, const void* rowptr, const void* colind, const void* values,
                                 int index_base, int index_bytes, int location) {
  try {
    Handle* h = lookup_any(ws);
    if (!h) return fail("krylov_b200_set_operator_csr", "unknown workspace handle");
    auto a = std::make_shared<CsrAny>();
    a->dtype = h->dtype;
    Ctx& cx = ctx_of(h);
    KB_CUDA(cudaSetDevice(cx.device));
    if (n != n_of(h)) throw std::runtime_error("(workspace.m, workspace.n) is inconsistent with size(A)");
    if (h->dtype == KRYLOV_FLOAT64)
      csr_upload<double>(cx, a->d, n, nnz, rowptr, colind, (const double*)values, index_base, index_bytes, location != 0);
    else
      csr_upload<float>(cx, a->f, n, nnz, rowptr, colind, (const float*)values, index_base, index_bytes, location != 0);
    h->csr = a;
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_set_operator_csr", e); }
}

int krylov_b200_share_operator(void* ws, void* src) {
  Handle* h = lookup_any(ws); Handle* s = lookup_any(src);
  if (!h || !s) return fail("krylov_b200_share_operator", "unknown workspace handle");
  if (!s->csr || s->dtype != h->dtype) return fail("krylov_b200_share_operator", "source has no CSR operator of this dtype");
  h->csr = s->csr;
  return 0;
}

int krylov_b200_attach_csr(void* ws, void* csr) {
  Handle* h = lookup_any(ws);
  if (!h || !csr) return fail("krylov_b200_attach_csr", "bad arguments");
  CsrAny* a = (CsrAny*)csr;
  if (a->dtype != h->dtype) return fail("krylov_b200_attach_csr", "dtype mismatch");
  h->csr = std::shared_ptr<CsrAny>(std::shared_ptr<CsrAny>(), a);   // non-owning alias
  return 0;
}

int krylov_b200_operator_encoding(void* ws) {
  Handle* h = lookup_any(ws);
  if (!h) return fail("krylov_b200_operator_encoding", "unknown workspace handle");
  if (!h->csr) return fail("krylov_b200_operator_encoding", "no CSR operator attached");
  return h->dtype == KRYLOV_FLOAT64 ? h->csr->d.ndict : h->csr->f.ndict;
}

int krylov_b200_set_preconditioner_diag(void* ws, int which, const void* d, int location) {
  try {
    Handle* h = lookup_any(ws);
    if (!h) return fail("krylov_b200_set_preconditioner_diag", "unknown workspace handle");
    void*& slot = which == 0 ? h->Mdiag : h->Ndiag;
    if (!d) { dev_free(slot); slot = nullptr; return 0; }
    const size_t esz = h->dtype == KRYLOV_FLOAT64 ? 8 : 4;
    const int n = n_of(h);
    KB_CUDA(cudaSetDevice(ctx_of(h).device));
    if (!slot) slot = dev_alloc<char>(esz * (size_t)n);
    KB_CUDA(cudaMemcpy(slot, d, esz * (size_t)n, location ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_set_preconditioner_diag", e); }
}

// Block-Jacobi preconditioner (SURVEY.md 8f-1; docs/src/preconditioners.md:33,159): dense bs x bs diagonal blocks,
// row-major, ceil(n / bs) of them.  The inverses are formed once here so that ldiv = true is a product as well.
int krylov_b200_set_preconditioner_blockdiag(void* ws, int which, int bs, const void* blocks, int location) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_set_preconditioner_blockdiag", "unknown (single right-hand side) workspace handle");
    if (which != 0 && which != 1) return fail("krylov_b200_set_preconditioner_blockdiag", "which must be 0 (M) or 1 (N)");
    dev_free(h->Pblk[which]); dev_free(h->Pblk_inv[which]);
    h->Pblk[which] = h->Pblk_inv[which] = nullptr; h->Pbs[which] = 0;
    if (!blocks) return 0;
    if (bs < 2 || bs > 8) return fail("krylov_b200_set_preconditioner_blockdiag", "block size must be in 2..8");
    const size_t esz = h->dtype == KRYLOV_FLOAT64 ? 8 : 4;
    const int n = n_of(h);
    const size_t cnt = (size_t)((n + bs - 1) / bs) * bs * bs;
    Ctx& c = ctx_of(h);
    KB_CUDA(cudaSetDevice(c.device));
    h->Pblk[which] = dev_alloc<char>(esz * cnt);
    h->Pblk_inv[which] = dev_alloc<char>(esz * cnt);
    h->Pbs[which] = bs;
    KB_CUDA(cudaMemcpyAsync(h->Pblk[which], blocks, esz * cnt, location ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c.stream));
    int* dsing = nullptr;
    KB_CUDA(cudaMalloc((void**)&dsing, sizeof(int)));
    KB_CUDA(cudaMemsetAsync(dsing, 0, sizeof(int), c.stream));
    if (h->dtype == KRYLOV_FLOAT64) k_blockdiag_invert<double>(c, n, bs, (const double*)h->Pblk[which], (double*)h->Pblk_inv[which], dsing);
    else k_blockdiag_invert<float>(c, n, bs, (const float*)h->Pblk[which], (float*)h->Pblk_inv[which], dsing);
    int sing = 0;
    KB_CUDA(cudaMemcpyAsync(&sing, dsing, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    cudaFree(dsing);
    if (sing) fprintf(stderr, "[krylov_b200] warning: a diagonal block of the block-Jacobi preconditioner is singular (its inverse, used by ldiv = true, is zero)\n");
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_set_preconditioner_blockdiag", e); }
}

KrylovB200Options krylov_b200_default_options(void) {
  KrylovB200Options o;
  memset(&o, 0, sizeof(o));
  o.etol = NAN; o.conlim = NAN; o.fused = 1; o.cr_gamma = NAN;
  return o;
}

int krylov_b200_set_options(void* ws, const KrylovB200Options* opts) {
  Handle* h = lookup_any(ws);
  if (!h) return fail("krylov_b200_set_options", "unknown workspace handle");
  h->ext = opts ? *opts : krylov_b200_default_options();
  return 0;
}

int krylov_b200_get_stats(void* ws, KrylovB200Stats* out) {
  Handle* h = lookup_any(ws);
  if (!h || !out) return fail("krylov_b200_get_stats", "unknown workspace handle");
  const Stats& s = stats_any(h);
  memset(out, 0, sizeof(*out));
  out->niter = s.niter; out->solved = s.solved; out->inconsistent = s.inconsistent; out->indefinite = s.indefinite;
  out->npcCount = s.npcCount; out->nresiduals = (int)s.residuals.size(); out->nAresiduals = (int)s.Aresiduals.size();
  out->nAcond = (int)s.Acond.size(); out->allocation_timer = s.allocation_timer; out->timer = s.timer;
  strncpy(out->status, s.status.c_str(), sizeof(out->status) - 1);
  out->Anorm = s.Anorm;
  return 0;
}

int krylov_b200_get_history(void* ws, int which, double* out, int cap) {
  Handle* h = lookup_any(ws);
  if (!h) return fail("krylov_b200_get_history", "unknown workspace handle");
  if (!out || cap < 0) return fail("krylov_b200_get_history", "bad arguments (out is NULL or cap < 0)");
  const Stats& s = stats_any(h);
  const std::vector<double>& v = which == 0 ? s.residuals : which == 1 ? s.Aresiduals : s.Acond;
  int k = (int)v.size() < cap ? (int)v.size() : cap;
  for (int i = 0; i < k; i++) out[i] = v[i];
  return k;
}

int krylov_b200_get_vector(void* ws, const char* name, void** dev_ptr) {
  Handle* h = lookup(ws);
  if (!h || !name || !dev_ptr) return fail("krylov_b200_get_vector", "bad arguments");
  void* p = h->dtype == KRYLOV_FLOAT64 ? vec_by_name<double>(W<double>(h), name) : vec_by_name<float>(W<float>(h), name);
  *dev_ptr = p;
  return p ? 0 : -2;
}

int krylov_b200_get_kernel_times(void* ws, double* out) {
  Handle* h = lookup(ws);
  if (!h || !out) return fail("krylov_b200_get_kernel_times", "bad arguments");
  if (h->dtype == KRYLOV_FLOAT64) { auto* w = W<double>(h); out[0] = w->k1_ms; out[1] = w->k2_ms; out[2] = w->timed_pairs; }
  else { auto* w = W<float>(h); out[0] = w->k1_ms; out[1] = w->k2_ms; out[2] = w->timed_pairs; }
  return 0;
}

long long krylov_b200_launch_count(void* ws) {
  Handle* h = lookup_any(ws);
  if (!h) return -1;
  return ctx_of(h).launches;
}

void* krylov_b200_stream(void* ws) {
  Handle* h = lookup_any(ws);
  if (!h) return nullptr;
  return (void*)ctx_of(h).stream;
}

int krylov_b200_wait_stream(void* ws, void* producer_stream) {
  try {
    Handle* h = lookup_any(ws);
    if (!h) return fail("krylov_b200_wait_stream", "unknown workspace handle");
    Ctx& c = ctx_of(h);
    KB_CUDA(cudaSetDevice(c.device));
    cudaEvent_t ev;
    KB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e1 = cudaEventRecord(ev, (cudaStream_t)producer_stream);
    cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(c.stream, ev, 0) : e1;
    cudaEventDestroy(ev);            // released once the wait has been satisfied
    if (e2 != cudaSuccess) throw std::runtime_error(cudaGetErrorString(e2));
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_wait_stream", e); }
}

// ------------------------------ row-partitioned solves --------------------
}  // extern "C" (templates below need C++ linkage)
namespace {
constexpr int kIpcHandles = 6;   // r, p, p2, mailbox, halo_buf, xhalo
constexpr size_t kMailBytes = kMailWords * sizeof(unsigned long long);

template <class T> int dist_init_t(Handle* h, int rank, int world, int nhalo, const int* halo_rank, const int* halo_off) {
  Workspace<T>* ws = W<T>(h);
  if (world < 1 || world > kMaxRanks || rank < 0 || rank >= world) throw std::runtime_error("bad rank/world");
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  if (h->solver == S_CG) {
    // r and the two direction buffers get a TAIL of nhalo entries: the persistent kernel stages the halo there and
    // gathers column nloc + h as element nloc + h of the same array (cg_fused.cu)
    KB_CUDA(cudaStreamSynchronize(ws->ctx.stream));
    const size_t len = (size_t)ws->n + (size_t)(nhalo > 0 ? nhalo : 0);
    T** bufs[3] = {&ws->r, &ws->p, &ws->p2};
    for (T** b : bufs) {
      dev_free(*b);
      *b = dev_alloc<T>(len);
      KB_CUDA(cudaMemset(*b, 0, sizeof(T) * len));
    }
  }
  ws->dist.rank = rank; ws->dist.world = world;
  int *dr = nullptr, *dof = nullptr;
  KB_CUDA(cudaMalloc((void**)&dr, sizeof(int) * (size_t)(nhalo > 0 ? nhalo : 1)));
  KB_CUDA(cudaMalloc((void**)&dof, sizeof(int) * (size_t)(nhalo > 0 ? nhalo : 1)));
  if (nhalo > 0) {
    KB_CUDA(cudaMemcpy(dr, halo_rank, sizeof(int) * (size_t)nhalo, cudaMemcpyHostToDevice));
    KB_CUDA(cudaMemcpy(dof, halo_off, sizeof(int) * (size_t)nhalo, cudaMemcpyHostToDevice));
  }
  ws->dist.halo = HaloMap{ws->n, nhalo, dr, dof};
  KB_CUDA(cudaMalloc(&ws->dist.mailbox, kMailBytes));
  KB_CUDA(cudaMemset(ws->dist.mailbox, 0, kMailBytes));
  // local halo buffers of the push mode: [r | p(bufA) | p(bufB)]
  ws->dist.halo_buf = dev_alloc<T>(3 * (size_t)(nhalo > 0 ? nhalo : 1));
  KB_CUDA(cudaMemset(ws->dist.halo_buf, 0, sizeof(T) * 3 * (size_t)(nhalo > 0 ? nhalo : 1)));
  ws->dist.npush = 0;
  // general x-halo exchange (all solvers): two sections of nhalo entries
  ws->dist.xhalo = dev_alloc<T>(2 * (size_t)(nhalo > 0 ? nhalo : 1));
  KB_CUDA(cudaMemset(ws->dist.xhalo, 0, sizeof(T) * 2 * (size_t)(nhalo > 0 ? nhalo : 1)));
  ws->dist.nglobal = ws->n;
  if (h->solver != S_CG) for (int i = 0; i < 3; i++) KB_CUDA(cudaMalloc(&ws->dist.dummy[i], 256));
  return 0;
}

template <class T> int dist_export_t(Handle* h, void* out) {
  Workspace<T>* ws = W<T>(h);
  if (!ws->dist.mailbox) throw std::runtime_error("call krylov_b200_dist_init first");
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  cudaIpcMemHandle_t* hs = (cudaIpcMemHandle_t*)out;
  // CG exports r/p/p2 for its in-kernel halo pull; the other solvers export three small placeholder allocations
  void* vr = ws->kind == S_CG ? (void*)ws->r : ws->dist.dummy[0];
  void* vp = ws->kind == S_CG ? (void*)ws->p : ws->dist.dummy[1];
  void* vp2 = ws->kind == S_CG ? (void*)ws->p2 : ws->dist.dummy[2];
  void* ptrs[kIpcHandles] = {vr, vp, vp2, ws->dist.mailbox, ws->dist.halo_buf, ws->dist.xhalo};
  for (int i = 0; i < kIpcHandles; i++) KB_CUDA(cudaIpcGetMemHandle(&hs[i], ptrs[i]));
  return 0;
}

template <class T> int dist_import_t(Handle* h, const void* all) {
  Workspace<T>* ws = W<T>(h);
  auto& D = ws->dist;
  KB_CUDA(cudaSetDevice(ws->ctx.device));
  const cudaIpcMemHandle_t* hs = (const cudaIpcMemHandle_t*)all;
  DistComm hc;
  memset(&hc, 0, sizeof(hc));
  hc.rank = D.rank; hc.world = D.world;
  {
    // spin budget of one cross-GPU reduction; a peer that stays away longer is treated as dead (dist.cuh)
    const char* es = getenv("KB200_DIST_TIMEOUT_S");
    double secs = es ? atof(es) : 30.0;
    if (!(secs > 0)) secs = 30.0;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ws->ctx.device);
    hc.timeout_cycles = (long long)(secs * 1e3 * (khz > 0 ? khz : 1965000));
  }
  for (int k = 0; k < D.world; k++) {
    void* ptr[kIpcHandles];
    if (k == D.rank) {
      ptr[0] = ws->r; ptr[1] = ws->p; ptr[2] = ws->p2; ptr[3] = D.mailbox; ptr[4] = D.halo_buf; ptr[5] = D.xhalo;
    } else {
      for (int i = 0; i < kIpcHandles; i++) {
        KB_CUDA(cudaIpcOpenMemHandle(&ptr[i], hs[k * kIpcHandles + i], cudaIpcMemLazyEnablePeerAccess));
        D.opened.push_back(ptr[i]);
      }
    }
    D.r_peer[k] = (T*)ptr[0]; D.bufA_peer[k] = (T*)ptr[1]; D.bufB_peer[k] = (T*)ptr[2];
    D.halo_buf_peer[k] = (T*)ptr[4];
    D.xhalo_peer[k] = (T*)ptr[5];
    hc.mail[k] = (unsigned long long*)ptr[3];
  }
  D.swapped = false;
  // plan of the general x-halo exchange (k_halo_exchange)
  DistExchange* ex = ws->ctx.dex ? ws->ctx.dex : new DistExchange();
  memset(ex, 0, sizeof(*ex));
  ex->nsend = D.nsend; ex->send_row = D.send_row; ex->send_peer = D.send_peer; ex->send_slot = D.send_slot;
  for (int k = 0; k < D.world; k++) { ex->xhalo_peer[k] = D.xhalo_peer[k]; ex->nhalo_peer[k] = D.nhalo_peer[k]; }
  ex->xhalo = D.xhalo; ex->nhalo = D.halo.nhalo; ex->nloc = ws->n; ex->count = 0;
  ws->ctx.dex = ex;
  if (!ws->ctx.dcomm) KB_CUDA(cudaMalloc((void**)&ws->ctx.dcomm, sizeof(DistComm)));
  KB_CUDA(cudaMemcpy(ws->ctx.dcomm, &hc, sizeof(DistComm), cudaMemcpyHostToDevice));
  return 0;
}
}  // namespace
extern "C" {

int krylov_b200_dist_handle_bytes(void) { return (int)(kIpcHandles * sizeof(cudaIpcMemHandle_t)); }

int krylov_b200_dist_init(void* ws, int rank, int world, int nhalo, const int* halo_rank, const int* halo_off) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_dist_init", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? dist_init_t<double>(h, rank, world, nhalo, halo_rank, halo_off)
                                      : dist_init_t<float>(h, rank, world, nhalo, halo_rank, halo_off);
  } catch (const std::exception& e) { return fail("krylov_b200_dist_init", e); }
}
int krylov_b200_dist_set_sendlist(void* ws, int nsend, const int* rows, const int* peers, const int* slots,
                                  const int* nhalo_all, long long nglobal) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_dist_set_sendlist", "unknown workspace handle");
    auto apply = [&](auto* w) {
      KB_CUDA(cudaSetDevice(w->ctx.device));
      auto up = [&](const int* src) {
        int* d = nullptr;
        KB_CUDA(cudaMalloc((void**)&d, sizeof(int) * (size_t)(nsend > 0 ? nsend : 1)));
        if (nsend > 0) KB_CUDA(cudaMemcpy(d, src, sizeof(int) * (size_t)nsend, cudaMemcpyHostToDevice));
        return d;
      };
      w->dist.send_row = up(rows); w->dist.send_peer = up(peers); w->dist.send_slot = up(slots);
      w->dist.nsend = nsend;
      for (int k = 0; k < w->dist.world; k++) w->dist.nhalo_peer[k] = nhalo_all[k];
      w->dist.nglobal = nglobal;
    };
    if (h->dtype == KRYLOV_FLOAT64) apply(W<double>(h)); else apply(W<float>(h));
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_dist_set_sendlist", e); }
}
int krylov_b200_dist_set_push(void* ws, int nranges, const int* ranges4, const int* nhalo_all) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_dist_set_push", "unknown workspace handle");
    if (nranges < 0 || nranges > kMaxPushRanges) return fail("krylov_b200_dist_set_push", "too many ranges (pull mode stays on)");
    auto apply = [&](auto* w) {
      for (int q = 0; q < nranges; q++) w->dist.push[q] = PushRange{ranges4[4 * q], ranges4[4 * q + 1], ranges4[4 * q + 2], ranges4[4 * q + 3]};
      for (int k = 0; k < w->dist.world; k++) w->dist.nhalo_peer[k] = nhalo_all[k];
      w->dist.npush = nranges;
    };
    if (h->dtype == KRYLOV_FLOAT64) apply(W<double>(h)); else apply(W<float>(h));
    return 0;
  } catch (const std::exception& e) { return fail("krylov_b200_dist_set_push", e); }
}
int krylov_b200_dist_export(void* ws, void* handles_out) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_dist_export", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? dist_export_t<double>(h, handles_out) : dist_export_t<float>(h, handles_out);
  } catch (const std::exception& e) { return fail("krylov_b200_dist_export", e); }
}
int krylov_b200_dist_import(void* ws, const void* all_handles) {
  try {
    Handle* h = lookup(ws);
    if (!h) return fail("krylov_b200_dist_import", "unknown workspace handle");
    return h->dtype == KRYLOV_FLOAT64 ? dist_import_t<double>(h, all_handles) : dist_import_t<float>(h, all_handles);
  } catch (const std::exception& e) { return fail("krylov_b200_dist_import", e); }
}

// ------------------------------ flat primitives ---------------------------
void* kb200_ctx_create(int device) {
  try {
    if (device < 0) device = pick_device();
    Ctx* c = new Ctx();
    c->init(device);
    return c;
  } catch (const std::exception& e) { fail("kb200_ctx_create", e); return nullptr; }
}
void kb200_ctx_destroy(void* ctx) {
  Ctx* c = (Ctx*)ctx;
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  c->destroy();
  delete c;
}
int kb200_sync(void* ctx) {
  try { ((Ctx*)ctx)->sync(); return 0; } catch (const std::exception& e) { return fail("kb200_sync", e); }
}
void* kb200_alloc(long long bytes) {
  try { return dev_alloc<char>((size_t)bytes); } catch (const std::exception& e) { fail("kb200_alloc", e); return nullptr; }
}
int kb200_free(void* p) { dev_free(p); return 0; }
int kb200_h2d(void* dst, const void* src, long long bytes) {
  return cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyHostToDevice) == cudaSuccess ? 0 : fail("kb200_h2d", "cudaMemcpy failed");
}
int kb200_d2h(void* dst, const void* src, long long bytes) {
  return cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : fail("kb200_d2h", "cudaMemcpy failed");
}

#define FLAT(name, body_d, body_f)                                                        \
  try {                                                                                   \
    Ctx& c = *(Ctx*)ctx;                                                                  \
    if (dtype == KRYLOV_FLOAT64) { typedef double T; (void)sizeof(T); body_d; }           \
    else if (dtype == KRYLOV_FLOAT32) { typedef float T; (void)sizeof(T); body_f; }       \
    else return -2;                                                                       \
    return 0;                                                                             \
  } catch (const std::exception& e) { return fail(name, e); }

int kb200_dot(void* ctx, int dtype, int n, const void* x, const void* y, double* result) {
  FLAT("kb200_dot", *result = k_dot<T>(c, n, (const T*)x, (const T*)y), *result = k_dot<T>(c, n, (const T*)x, (const T*)y))
}
int kb200_nrm2(void* ctx, int dtype, int n, const void* x, double* result) {
  FLAT("kb200_nrm2", *result = k_nrm2<T>(c, n, (const T*)x), *result = k_nrm2<T>(c, n, (const T*)x))
}
int kb200_axpy(void* ctx, int dtype, int n, double s, const void* x, void* y) {
  FLAT("kb200_axpy", k_axpy<T>(c, n, (T)s, (const T*)x, (T*)y), k_axpy<T>(c, n, (T)s, (const T*)x, (T*)y))
}
int kb200_axpby(void* ctx, int dtype, int n, double s, const void* x, double t, void* y) {
  FLAT("kb200_axpby", k_axpby<T>(c, n, (T)s, (const T*)x, (T)t, (T*)y), k_axpby<T>(c, n, (T)s, (const T*)x, (T)t, (T*)y))
}
int kb200_scal(void* ctx, int dtype, int n, double s, void* x) {
  FLAT("kb200_scal", k_scal<T>(c, n, (T)s, (T*)x), k_scal<T>(c, n, (T)s, (T*)x))
}
int kb200_copy(void* ctx, int dtype, int n, void* y, const void* x) {
  FLAT("kb200_copy", k_copy<T>(c, n, (T*)y, (const T*)x), k_copy<T>(c, n, (T*)y, (const T*)x))
}
int kb200_scalcopy(void* ctx, int dtype, int n, void* y, double s, const void* x) {
  FLAT("kb200_scalcopy", k_scalcopy<T>(c, n, (T*)y, (T)s, (const T*)x), k_scalcopy<T>(c, n, (T*)y, (T)s, (const T*)x))
}
int kb200_divcopy(void* ctx, int dtype, int n, void* y, const void* x, double s) {
  FLAT("kb200_divcopy", k_divcopy<T>(c, n, (T*)y, (const T*)x, (T)s), k_divcopy<T>(c, n, (T*)y, (const T*)x, (T)s))
}
int kb200_fill(void* ctx, int dtype, int n, void* x, double v) {
  FLAT("kb200_fill", k_fill<T>(c, n, (T*)x, (T)v), k_fill<T>(c, n, (T*)x, (T)v))
}

void* kb200_csr_create(void* ctx, int dtype, int n, long long nnz, const void* rowptr, const void* colind, const void* values,
                       int index_base, int index_bytes, int location) {
  try {
    Ctx& c = *(Ctx*)ctx;
    CsrAny* a = new CsrAny();
    a->dtype = dtype; a->owner_ctx = &c;
    try {
      if (dtype == KRYLOV_FLOAT64) csr_upload<double>(c, a->d, n, nnz, rowptr, colind, (const double*)values, index_base, index_bytes, location != 0);
      else if (dtype == KRYLOV_FLOAT32) csr_upload<float>(c, a->f, n, nnz, rowptr, colind, (const float*)values, index_base, index_bytes, location != 0);
      else throw std::runtime_error("unsupported dtype");
    } catch (...) { delete a; throw; }
    return a;
  } catch (const std::exception& e) { fail("kb200_csr_create", e); return nullptr; }
}
void kb200_csr_destroy(void* csr) { delete (CsrAny*)csr; }

// Matrix Market ingestion and the transposed operator (mtx.cu)
void* kb200_csr_read_mtx(void* ctx, const char* path, int dtype) {
  try {
    if (!ctx || !path) throw std::runtime_error("bad arguments");
    Ctx& c = *(Ctx*)ctx;
    HostCsr h;
    read_matrix_market(path, h);
    CsrAny* a = new CsrAny();
    a->dtype = dtype; a->owner_ctx = &c;
    try {
      if (dtype == KRYLOV_FLOAT64) csr_from_host<double>(c, a->d, h);
      else if (dtype == KRYLOV_FLOAT32) csr_from_host<float>(c, a->f, h);
      else throw std::runtime_error("unsupported dtype");
    } catch (...) { delete a; throw; }
    return a;
  } catch (const std::exception& e) { fail("kb200_csr_read_mtx", e); return nullptr; }
}

void* kb200_csr_transpose(void* ctx, void* csr) {
  try {
    if (!ctx || !csr) throw std::runtime_error("bad arguments");
    Ctx& c = *(Ctx*)ctx;
    CsrAny* src = (CsrAny*)csr;
    HostCsr h, ht;
    if (src->dtype == KRYLOV_FLOAT64) csr_to_host<double>(c, src->d, h); else csr_to_host<float>(c, src->f, h);
    transpose_csr(h, ht);
    CsrAny* a = new CsrAny();
    a->dtype = src->dtype; a->owner_ctx = &c;
    try {
      if (a->dtype == KRYLOV_FLOAT64) csr_from_host<double>(c, a->d, ht); else csr_from_host<float>(c, a->f, ht);
    } catch (...) { delete a; throw; }
    return a;
  } catch (const std::exception& e) { fail("kb200_csr_transpose", e); return nullptr; }
}

int kb200_csr_info(void* csr, int* n, long long* nnz) {
  CsrAny* a = (CsrAny*)csr;
  if (!a) return -1;
  if (n) *n = a->dtype == KRYLOV_FLOAT64 ? a->d.n : a->f.n;
  if (nnz) *nnz = a->dtype == KRYLOV_FLOAT64 ? a->d.nnz : a->f.nnz;
  return 0;
}

int kb200_csr_download(void* ctx, void* csr, int* rowptr, int* colind, void* values) {
  try {
    if (!ctx || !csr) throw std::runtime_error("bad arguments");
    Ctx& c = *(Ctx*)ctx;
    CsrAny* a = (CsrAny*)csr;
    HostCsr h;
    if (a->dtype == KRYLOV_FLOAT64) csr_to_host<double>(c, a->d, h); else csr_to_host<float>(c, a->f, h);
    if (rowptr) for (size_t i = 0; i < h.rowptr.size(); i++) rowptr[i] = (int)h.rowptr[i];
    if (colind) for (size_t i = 0; i < h.colind.size(); i++) colind[i] = (int)h.colind[i];
    if (values) {
      if (a->dtype == KRYLOV_FLOAT64) std::memcpy(values, h.val.data(), sizeof(double) * h.val.size());
      else for (size_t i = 0; i < h.val.size(); i++) ((float*)values)[i] = (float)h.val[i];
    }
    return 0;
  } catch (const std::exception& e) { return fail("kb200_csr_download", e); }
}

// ---- host-side pieces, callable without a GPU (tests/test_host_logic.py) ---------------------------------------
int kb200_mtx_read(const char* path, int* n, long long* nnz, int* rowptr, int* colind, double* values) {
  try {
    if (!path) throw std::runtime_error("path is NULL");
    HostCsr h;
    read_matrix_market(path, h);
    if (n) *n = h.n;
    if (nnz) *nnz = (long long)h.colind.size();
    if (rowptr) for (size_t i = 0; i < h.rowptr.size(); i++) rowptr[i] = (int)h.rowptr[i];
    if (colind) for (size_t i = 0; i < h.colind.size(); i++) colind[i] = (int)h.colind[i];
    if (values) std::memcpy(values, h.val.data(), sizeof(double) * h.val.size());
    return 0;
  } catch (const std::exception& e) { return fail("kb200_mtx_read", e); }
}

int kb200_host_householder(int m, int k, double* Q, double* R, double* tau, int compact) {
  if (!Q || !R || !tau || m < k || k < 1) return fail("kb200_host_householder", "bad arguments");
  dense::householder_compact<double>(m, k, Q, R, tau);
  if (!compact) dense::org2r<double>(m, k, Q, m, tau);
  return 0;
}

int kb200_host_cholqr_factors(int p, const double* G, double* R, double* Rinv) {
  if (!G || !R || !Rinv || p < 1) return fail("kb200_host_cholqr_factors", "bad arguments");
  if (!dense::cholesky_upper<double>(p, G, R)) return 1;
  dense::inv_upper<double>(p, R, Rinv);
  return 0;
}

int kb200_host_householder_signs(int p, const double* top, double* s) {
  if (!top || !s || p < 1) return fail("kb200_host_householder_signs", "bad arguments");
  std::vector<double> W(top, top + (size_t)p * p);
  dense::householder_signs<double>(p, W.data(), s);
  return 0;
}

int kb200_spmv_csr(void* ctx, void* csr, const void* x, void* y, int variant) {
  try {
    Ctx& c = *(Ctx*)ctx;
    CsrAny* a = (CsrAny*)csr;
    if (a->dtype == KRYLOV_FLOAT64) k_spmv<double>(c, a->d, (const double*)x, (double*)y, variant);
    else k_spmv<float>(c, a->f, (const float*)x, (float*)y, variant);
    return 0;
  } catch (const std::exception& e) { return fail("kb200_spmv_csr", e); }
}

int kb200_csr_plan(void* csr, long long* out) {
  CsrAny* a = (CsrAny*)csr;
  if (!a || !out) return -1;
  if (a->dtype == KRYLOV_FLOAT64) {
    const Csr<double>& A = a->d;
    out[0] = A.ntiles; out[1] = A.tile_cap; out[2] = A.max_row; out[3] = A.tma_ok; out[4] = A.stages; out[5] = A.grid; out[6] = (long long)A.smem_bytes;
  } else {
    const Csr<float>& A = a->f;
    out[0] = A.ntiles; out[1] = A.tile_cap; out[2] = A.max_row; out[3] = A.tma_ok; out[4] = A.stages; out[5] = A.grid; out[6] = (long long)A.smem_bytes;
  }
  return 0;
}

}  // extern "C"
