/*
 * krylov_b200.h -- C ABI of libkrylov_b200.so, the B200 (sm_100a) drop-in for
 * the inner-iteration path of Krylov.jl's cg!/gmres!/bicgstab!/minres!.
 *
 * PART 1 is binary-compatible with the reference's libkrylov
 * (interfaces/include/krylov.h @ Krylov.jl v0.10.8): same symbol names, same
 * struct layouts (interfaces/src/c_enums.jl:30-62), same enum values
 * (interfaces/scripts/solver_table.jl:5-42), same return-code conventions
 * (docs/src/interfaces/reference.md:144-170).  A C/Fortran program written
 * against krylov.h links against this library unchanged.
 *
 * PART 2 is additive: the CUDA device id, a device-resident CSR operator (so
 * the SpMV can be fused with the BLAS-1 work instead of crossing back into a
 * host callback once per product), statistics the reference keeps in
 * SimpleStats, and the flat per-primitive entry points a Julia `ccall` shim
 * binds (krylov.jl_b200/julia/KrylovB200.jl).
 *
 * Where vectors live: every workspace vector lives in HBM and every vector
 * operation runs on the GPU.  `device` only says where the CALLER's buffers
 * are: KRYLOV_CPU  -> b, c, x0, x and the matvec callbacks use host pointers
 * (the library stages them); KRYLOV_CUDA -> they are device pointers.
 * There is no CPU compute path: without a usable GPU, create returns -1.
 */
#ifndef KRYLOV_B200_H
#define KRYLOV_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ======================= PART 1: the libkrylov ABI ======================= */

#ifndef KRYLOV_H /* allow inclusion next to the reference header */

#define KRYLOV_VERSION_MAJOR 0
#define KRYLOV_VERSION_MINOR 10
#define KRYLOV_VERSION_PATCH 8

/* element type of every vector (krylov.h:37-42) */
typedef enum { KRYLOV_FLOAT32 = 0, KRYLOV_FLOAT64 = 1, KRYLOV_COMPLEX32 = 2, KRYLOV_COMPLEX64 = 3 } KrylovDataType;

/* krylov.h:44-46 has KRYLOV_CPU only; KRYLOV_CUDA is this library's addition */
typedef enum { KRYLOV_CPU = 0, KRYLOV_CUDA = 1 } KrylovDeviceType;

/* positional, frozen (krylov.h:48-83).  Implemented here: CG, MINRES, GMRES, BICGSTAB (the hot path) and the
 * siblings CR, DIOM, DQGMRES, FOM, FGMRES, CGS that run on the same kernels; every other value returns -2. */
typedef enum {
  KRYLOV_CG = 0, KRYLOV_CR = 1, KRYLOV_SYMMLQ = 2, KRYLOV_MINRES = 3, KRYLOV_MINRES_QLP = 4, KRYLOV_DIOM = 5,
  KRYLOV_DQGMRES = 6, KRYLOV_FOM = 7, KRYLOV_GMRES = 8, KRYLOV_FGMRES = 9, KRYLOV_BICGSTAB = 10, KRYLOV_CGS = 11,
  KRYLOV_BILQ = 12, KRYLOV_QMR = 13, KRYLOV_USYMLQ = 14, KRYLOV_USYMQR = 15, KRYLOV_TRICG = 16, KRYLOV_TRIMR = 17,
  KRYLOV_TRILQR = 18, KRYLOV_BILQR = 19, KRYLOV_LSLQ = 20, KRYLOV_LSQR = 21, KRYLOV_LSMR = 22, KRYLOV_USYMLQR = 23,
  KRYLOV_CGLS = 24, KRYLOV_CRLS = 25, KRYLOV_CGNE = 26, KRYLOV_CRMR = 27, KRYLOV_CRAIG = 28, KRYLOV_CRAIGMR = 29,
  KRYLOV_LNLQ = 30, KRYLOV_GPMR = 31, KRYLOV_CAR = 32, KRYLOV_MINARES = 33
} KrylovSolverType;

typedef enum { KRYLOV_BLOCK_GMRES = 0, KRYLOV_BLOCK_MINRES = 1 } KrylovBlockSolverType;

/* y = A x, y = A^H x, or y = M^-1 x.  The library owns x and y; they are
 * valid only during the call (reference.md:57-61). */
typedef void (*KrylovMatvec)(const void *x, void *y, void *userdata);
typedef void (*KrylovBlockMatvec)(const void *X, void *Y, int p, void *userdata);

/* construction-time options; 0 = solver default (memory 20, window 5) */
typedef struct {
  int memory;
  int window;
} KrylovWorkspaceOptions;

/* solve-time options; NaN / 0 = solver default (c_stores.jl:255-260) */
typedef struct {
  double atol;
  double rtol;
  int itmax;
  int verbose;
  double lambda;
  double tau;
  double nu;
  double timemax;
  double radius;
  int restart;
  int reorthogonalization;
  int linesearch;
} KrylovOptions;

#endif /* KRYLOV_H */

/* 0 ok | -1 error (message on stderr, *ws_out untouched) | -2 unknown/unsupported (solver, dtype) */
int krylov_workspace_create(KrylovSolverType solver, int m, int n, KrylovDataType dtype, KrylovDeviceType device,
                            const KrylovWorkspaceOptions *wopts, void **ws_out);
KrylovWorkspaceOptions krylov_default_workspace_options(void);
KrylovOptions krylov_default_options(void);
void krylov_get_version(int *major, int *minor, int *patch);
/* 0 ok | -1 error.  matvec_A may be NULL once a CSR operator is attached (part 2). */
int krylov_solve(void *ws, KrylovMatvec matvec_A, KrylovMatvec matvec_At, KrylovMatvec matvec_M, KrylovMatvec matvec_N,
                 const void *b, const void *c, void *userdata, const KrylovOptions *opts);
int krylov_get_x(void *ws, void *x, int n);
int krylov_get_y(void *ws, void *y, int m); /* -2: single-solution solver */
int krylov_is_solved(void *ws);             /* 1 | 0 | -1 */
int krylov_niter(void *ws);
double krylov_elapsed_time(void *ws);
int krylov_warm_start(void *ws, const void *x0, int n);
int krylov_warm_start2(void *ws, const void *x0, const void *y0, int nx, int ny); /* -2 here */
int krylov_workspace_free(void *ws); /* 0 | 1 if the handle is unknown (double free is safe) */

/* Block solvers (krylov.h:250-285): KRYLOV_BLOCK_GMRES is implemented (p <= 32, Float32 / Float64; the tall-skinny
 * panel products of Float64 p = 8 / 16 / 32 run on the FP64 tensor cores); KRYLOV_BLOCK_MINRES answers -2. */
int krylov_block_workspace_create(KrylovBlockSolverType solver, int m, int n, int p, KrylovDataType dtype,
                                  KrylovDeviceType device, const KrylovWorkspaceOptions *wopts, void **ws_out);
int krylov_block_solve(void *ws, KrylovBlockMatvec matvec_A, KrylovBlockMatvec matvec_M, KrylovBlockMatvec matvec_N,
                       const void *B, void *userdata, const KrylovOptions *opts);
int krylov_block_get_X(void *ws, void *X, int n, int p);
int krylov_block_is_solved(void *ws);
int krylov_block_niter(void *ws);
double krylov_block_elapsed_time(void *ws);
int krylov_block_warm_start(void *ws, const void *x0, int n, int p);
int krylov_block_workspace_free(void *ws);
/* Number of panel QR factorizations of this block workspace that left the fast path: a Gram matrix that is not
 * numerically positive definite (rank-deficient block of right-hand sides or Krylov block) makes CholQR2 impossible,
 * and that ONE panel is then factorized by LAPACK's Householder algorithm run as 4p passes of the panel kernels
 * (still on the device).  0 on well-posed blocks. */
long long krylov_b200_block_qr_fallbacks(void *ws);

/* ===================== PART 2: B200 additions (additive) ===================== */

/* Number of usable CUDA devices (0 when there is no GPU / no driver). */
int krylov_b200_device_count(void);
/* Device used by subsequently created workspaces (default: current device). */
int krylov_b200_set_device(int device);
/* Last error message of the calling thread ("" if none). */
const char *krylov_b200_last_error(void);

/* Attach a CSR matrix as the operator A of `ws`: replaces mul!(y, A, x) at
 * cg.jl:196, gmres.jl:257, bicgstab.jl:221,228, minres.jl:289.
 *   rowptr[n+1], colind[nnz], values[nnz] (element type = workspace dtype);
 *   index_base 0|1, index_bytes 4|8 (Julia's SparseMatrixCSC{T,Int64} passes
 *   1 and 8 -- for a symmetric matrix its CSC arrays ARE the CSR arrays);
 *   location 0 = host arrays, 1 = device arrays.
 * The library keeps its own int32 / 0-based device copy. */
int krylov_b200_set_operator_csr(void *ws, int n, long long nnz, const void *rowptr, const void *colind,
                                 const void *values, int index_base, int index_bytes, int location);
/* Share the CSR operator already attached to `src` (no copy). */
int krylov_b200_share_operator(void *ws, void *src);
/* Attach a CSR object made by kb200_csr_create (not owned: keep it alive while `ws` uses it). */
int krylov_b200_attach_csr(void *ws, void *csr);
/* How the staged SpMV and the persistent CG kernel stream the attached CSR operator: the number of entries of its
 * (column - row, value) dictionary when it is stored as one code byte per nonzero, 0 when they stream the CSR
 * arrays (more than 256 distinct pairs, a non-default tile plan, or KB200_CSR_DICT=0 at upload), -1 on error. */
int krylov_b200_operator_encoding(void *ws);
/* Diagonal preconditioner: which = 0 -> M, 1 -> N; d[n] holds the diagonal of
 * the operator the solver applies (P^-1 with the default ldiv=false). NULL detaches. */
int krylov_b200_set_preconditioner_diag(void *ws, int which, const void *d, int location);
/* Block-Jacobi preconditioner (docs/src/preconditioners.md:33,159): which = 0 -> M, 1 -> N; blocks[ceil(n/bs)][bs][bs]
 * (row-major dense diagonal blocks, 2 <= bs <= 8, element type = workspace dtype; a last block of n % bs rows uses
 * its leading part) of the operator the solver applies (P^-1 with the default ldiv = false; with ldiv = true the
 * blocks are P and their inverses, formed once here, are applied).  cg! with M block-diagonal runs the persistent
 * fused kernel (z = M r formed block by block in the r-update phase); every other solver applies it as one extra
 * kernel per product.  A diagonal set with krylov_b200_set_preconditioner_diag takes precedence.  NULL detaches. */
int krylov_b200_set_preconditioner_blockdiag(void *ws, int which, int bs, const void *blocks, int location);

/* cg_lanczos! (src/cg_lanczos.jl) has no slot in the reference's KrylovSolverType; this value selects it in
 * krylov_workspace_create.  Options: M, check_curvature (KrylovB200Options), the common tolerances. */
#define KRYLOV_B200_CG_LANCZOS 100

/* Extra solve-time switches not present in KrylovOptions. */
typedef struct {
  int history;        /* 1: record residual history (kwarg `history`)              */
  int ldiv;           /* 1: preconditioners are applied with ldiv! (kwarg `ldiv`)   */
  double etol;        /* MINRES; NaN -> sqrt(eps)                                   */
  double conlim;      /* MINRES; NaN -> 1/sqrt(eps)                                 */
  int fused;          /* 1 (default): fused kernels when eligible (CG: one persistent cooperative launch per
                       * batch of iterations); 2: fused CG as two launches per iteration; 0: primitives */
  int batch;          /* fused CG: iterations enqueued per host poll; 0 -> default  */
  int (*callback)(void *ws, void *user); /* kwarg `callback`; nonzero return = stop */
  void *callback_user;
  int time_kernels;   /* fused CG: time the two phases of the iteration (see krylov_b200_get_kernel_times) */
  int check_curvature; /* CG-Lanczos: kwarg `check_curvature` (src/cg_lanczos.jl:94)                            */
  double cr_gamma;     /* CR: kwarg `γ` (src/cr.jl:112); NaN -> sqrt(eps)                                        */
} KrylovB200Options;
KrylovB200Options krylov_b200_default_options(void);
int krylov_b200_set_options(void *ws, const KrylovB200Options *opts);

/* SimpleStats (src/krylov_stats.jl:24-36) */
typedef struct {
  int niter;
  int solved;
  int inconsistent;
  int indefinite;
  int npcCount;
  int nresiduals;
  int nAresiduals;
  int nAcond;
  double allocation_timer;
  double timer;
  char status[96];
  double Anorm;       /* LanczosStats.Anorm (cg_lanczos!); NaN for the other solvers */
} KrylovB200Stats;
int krylov_b200_get_stats(void *ws, KrylovB200Stats *out);
/* which: 0 residuals, 1 Aresiduals, 2 Acond.  Returns the number copied (<= cap) or -1. */
int krylov_b200_get_history(void *ws, int which, double *out, int cap);
/* Device pointer of a workspace vector by its reference field name
 * ("x","r","p","Ap","z","npc_dir","v","s","qd","r1","r2","w1","w2","y","w","dx","V1".."Vk"). */
int krylov_b200_get_vector(void *ws, const char *name, void **dev_ptr);
/* Average durations (ms) of the fused kernels measured with CUDA events on the workspace stream during the
 * last solve run with time_kernels = 1: out[0] = K1 (SpMV + p update + <p,Ap>), out[1] = K2 (x, r update + <r,r>),
 * out[2] = number of timed iterations. */
int krylov_b200_get_kernel_times(void *ws, double *out3);
/* Kernels launched so far through this workspace's stream. */
long long krylov_b200_launch_count(void *ws);
/* The CUDA stream (cudaStream_t) all of this workspace's work is ordered on.  It is a private NON-BLOCKING stream:
 * nothing orders it against the caller's streams implicitly.  STREAM CONTRACT for device-pointer inputs (KRYLOV_CUDA
 * workspaces: b, c, x0; location = 1 arrays of krylov_b200_set_operator_csr / set_preconditioner_diag): the data
 * must be complete when the call is made, OR the producer must be ordered before this stream with
 * krylov_b200_wait_stream (or cudaStreamWaitEvent on krylov_b200_stream(ws)).  Outputs need no care: every solve
 * returns after synchronising its stream. */
void *krylov_b200_stream(void *ws);
/* Make the workspace's stream wait for everything enqueued so far on `producer_stream` (a cudaStream_t; NULL = the
 * legacy default stream): records an event there and waits for it on krylov_b200_stream(ws).  Returns 0 / -1. */
int krylov_b200_wait_stream(void *ws, void *producer_stream);

/* ---- row-partitioned solves: one process per GPU, one workspace per process ----
 * The workspace is created with n = number of LOCAL rows; its CSR operator has
 * n rows and n + nhalo columns: column j < n is local, column n + h is the halo
 * entry h, owned by rank halo_rank[h] at offset halo_off[h] of that rank's local
 * vectors.  Peers' vectors are mapped with CUDA IPC: every rank calls dist_init,
 * dist_export (fills krylov_b200_dist_handle_bytes() bytes), the caller gathers
 * the blobs of all ranks in rank order (e.g. torch.distributed.all_gather) and
 * passes the concatenation to dist_import.  Afterwards krylov_solve on a CG
 * workspace runs the fused path with in-kernel NVLink halo loads and in-kernel
 * all-reduces of the dot products (csrc/dist.cuh).  All ranks must call
 * krylov_solve with the same options. */
int krylov_b200_dist_handle_bytes(void);
int krylov_b200_dist_init(void *ws, int rank, int world, int nhalo, const int *halo_rank, const int *halo_off);
/* Optional push mode (after dist_init, any time before the first solve): `ranges4` holds nranges (<= 4) quadruples
 * (first local row, count, peer rank, first slot in the peer's halo) describing which contiguous blocks of this
 * rank's rows each peer needs; nhalo_all[world] = every rank's halo length.  The producing kernels then store
 * those entries directly into the peers' halo buffers and nobody issues fine-grained P2P loads. */
int krylov_b200_dist_set_push(void *ws, int nranges, const int *ranges4, const int *nhalo_all);
/* Send list of the general x-halo exchange that precedes every y = A x of a distributed workspace (all four
 * solvers): entry e sends local row rows[e] to slot slots[e] of rank peers[e]'s halo.  nhalo_all[world] = every
 * rank's halo length, nglobal = global number of rows.  Call after dist_init and before dist_export/import. */
int krylov_b200_dist_set_sendlist(void *ws, int nsend, const int *rows, const int *peers, const int *slots,
                                  const int *nhalo_all, long long nglobal);
int krylov_b200_dist_export(void *ws, void *handles_out);
int krylov_b200_dist_import(void *ws, const void *all_handles);

/* ---- flat primitives: the k* wrappers of src/krylov_utils.jl:305-349 ----
 * dtype selects float/double; all pointers are device pointers; scalars by
 * value as double; results by pointer.  `ctx` comes from kb200_ctx_create. */
void *kb200_ctx_create(int device);
void kb200_ctx_destroy(void *ctx);
int kb200_sync(void *ctx);
void *kb200_alloc(long long bytes);
int kb200_free(void *p);
int kb200_h2d(void *dst, const void *src, long long bytes);
int kb200_d2h(void *dst, const void *src, long long bytes);
int kb200_dot(void *ctx, int dtype, int n, const void *x, const void *y, double *result);
int kb200_nrm2(void *ctx, int dtype, int n, const void *x, double *result);
int kb200_axpy(void *ctx, int dtype, int n, double s, const void *x, void *y);
int kb200_axpby(void *ctx, int dtype, int n, double s, const void *x, double t, void *y);
int kb200_scal(void *ctx, int dtype, int n, double s, void *x);
int kb200_copy(void *ctx, int dtype, int n, void *y, const void *x);
int kb200_scalcopy(void *ctx, int dtype, int n, void *y, double s, const void *x);
int kb200_divcopy(void *ctx, int dtype, int n, void *y, const void *x, double s);
int kb200_fill(void *ctx, int dtype, int n, void *x, double v);
/* CSR operator objects for the flat API (same arguments as set_operator_csr). */
void *kb200_csr_create(void *ctx, int dtype, int n, long long nnz, const void *rowptr, const void *colind,
                       const void *values, int index_base, int index_bytes, int location);
void kb200_csr_destroy(void *csr);
/* Data formats either side of the path (SURVEY.md 8f-4).  kb200_csr_read_mtx: Matrix Market `matrix coordinate
 * {real|integer|pattern} {general|symmetric|skew-symmetric}` (what benchmark/benchmarks.jl:23-33 reads through
 * MatrixMarket.jl), duplicates summed, symmetric storage expanded; NULL on error (krylov_b200_last_error).
 * kb200_csr_transpose: a new object holding A^T (= A^H for the real types here, docs/src/matrix_free.md:36-44). */
void *kb200_csr_read_mtx(void *ctx, const char *path, int dtype);
void *kb200_csr_transpose(void *ctx, void *csr);
int kb200_csr_info(void *csr, int *n, long long *nnz);
/* rowptr[n+1], colind[nnz] (0-based int32), values[nnz] in the object's dtype; any pointer may be NULL */
int kb200_csr_download(void *ctx, void *csr, int *rowptr, int *colind, void *values);
/* Host-side pieces, callable without a GPU (they make no CUDA call): the Matrix Market parser behind
 * kb200_csr_read_mtx (pass NULL arrays to query n / nnz first) and the small dense algebra of the block path --
 * LAPACK-style Householder QR (householder!, src/block_krylov_utils.jl:201-208: Q m x k column-major in/out, R k x k,
 * compact = 1 keeps the reflectors), the Cholesky factor / inverse of a Gram matrix (1: not positive definite
 * enough for CholQR2), and the Householder-sign reconstruction from the top p x p block of an orthonormal factor. */
int kb200_mtx_read(const char *path, int *n, long long *nnz, int *rowptr, int *colind, double *values);
int kb200_host_householder(int m, int k, double *Q, double *R, double *tau, int compact);
int kb200_host_cholqr_factors(int p, const double *G, double *R, double *Rinv);
int kb200_host_householder_signs(int p, const double *top, double *s);
/* y = A x.  variant: 0 auto, 1 row-per-thread LDG kernel, 2 TMA-staged kernel. */
int kb200_spmv_csr(void *ctx, void *csr, const void *x, void *y, int variant);
/* staging plan of a CSR object: out[0]=ntiles out[1]=tile_cap out[2]=max_row out[3]=tma_ok out[4]=stages out[5]=grid out[6]=smem_bytes */
int kb200_csr_plan(void *csr, long long *out7);

#ifdef __cplusplus
}
#endif
#endif /* KRYLOV_B200_H */
