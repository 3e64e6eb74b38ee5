// cg_fused.cu -- the CG hot loop (src/cg.jl:195-268) with every scalar recurrence on the device.
//
//   phase A / K1  p <- z + beta p   (cg.jl:259, applied on the fly while gathering)
//                 Ap <- A p         (cg.jl:196)
//                 pAp <- <p, Ap>    (cg.jl:197)   -> curvature test + alpha (cg.jl:198-213)
//                 x += alpha_prev p_prev          (cg.jl:239 of the PREVIOUS iteration; p_prev is in a register here)
//   phase B / K2  r -= alpha Ap                   (cg.jl:240)
//                 gamma' <- <r, r>  (cg.jl:242)   -> rNorm, stop tests, beta, pNorm2 (cg.jl:244-258)
//
// Two implementations of the same arithmetic:
//   * cg_persist (default): ONE cooperative, co-resident kernel runs a batch of 32 iterations; the phases are
//     separated by grid-wide barriers that carry the dot-product reductions, the TMA producer prefetches the next
//     iteration's first tiles across the barrier, the kernel reports its scalar block into pinned host memory when
//     it ends.  Row-partitioned (MODE = kDist): the halo of r and p is staged over NVLink into the tails of the
//     local vectors at the start of phase A and both barriers end in a warp-parallel cross-GPU all-reduce
//     (dist.cuh).  Block-Jacobi M (MODE = kBlockJac): z = M r is formed block by block in phase B.
//   * cg_k1_tma / cg_k1_rows + cg_k2: two launches per iteration, used when x must be current after every
//     iteration (callbacks, verbose, timemax), when the operator has no TMA tile plan, and as the A/B reference
//     (fused = 2, KB200_PERSIST=0).  Their row-partitioned variant pulls halo entries nonzero by nonzero.
//
// The host only enqueues launches and polls the scalar block (one read-back per batch of iterations); launches
// enqueued past the stopping point see `done` and return immediately, so niter, x, r, p at exit are those of the
// reference loop.  p is double-buffered because phase A reads the old direction of neighbouring rows while
// writing the new one.
#include "solver_common.h"
#include "spmv_tiles.cuh"

namespace kb {

constexpr int kHist = 64;

template <class T>
struct CgState {
  T gamma, pAp, alpha, beta, pNorm2, rNorm, eps_tol, pad0;
  int iter, itmax, done, linesearch;
  int solved, tired, zero_curvature, inconsistent;
  int npc, not_spd, comm_error, pad2;
  T hist[kHist];
};

static_assert(sizeof(CgState<double>) % 8 == 0 && sizeof(CgState<float>) % 8 == 0, "CgState is copied as 8-byte words");

template <class T>
struct CgPeers {           // peers' vectors for the halo gather (DIST only)
  HaloMap halo;
  const T* r[kMaxRanks];
  const T* p_old[kMaxRanks];
  const T* mdiag;          // diagonal of M (nullptr: M = I); rides along in this kernel-parameter block
  const T* r_halo;         // push mode: LOCAL halo copies kept current by the peers' K2 / K1 (nullptr: pull mode)
  const T* p_halo_old;
  PushPlan<T> push_p;      // where this rank's new p entries go (peers' p_halo of the new parity)
};

template <class T>
__device__ __forceinline__ void cg_k1_finalize(CgState<T>* st, T pAp) {
  st->pAp = pAp;
  const T lim = mul_rn(Eps<T>::v, st->pNorm2);
  if (pAp <= lim) {                       // radius == 0 on this path (cg.jl:198)
    if (fabs(pAp) <= lim) { st->zero_curvature = 1; st->inconsistent = !st->linesearch; }
    if (st->linesearch) { st->npc = 1; st->solved = 1; }
    if (st->zero_curvature || st->solved) { st->done = 1; return; }
  }
  st->alpha = div_rn(st->gamma, pAp);      // cg.jl:213
}

template <class T>
__device__ __forceinline__ void cg_k2_finalize(CgState<T>* st, T gamma_next) {
  if (!(gamma_next >= T(0))) { st->not_spd = 1; st->done = 1; return; }   // cg.jl:243
  const T rNorm = sqrt_rn(gamma_next);
  st->rNorm = rNorm;
  const int it1 = st->iter + 1;
  st->hist[it1 % kHist] = rNorm;
  const bool solved = (rNorm <= st->eps_tol) || (add_rn(rNorm, T(1)) <= T(1));   // cg.jl:249-253
  if (!solved) {                                                                // cg.jl:255-258
    const T beta = div_rn(gamma_next, st->gamma);
    st->beta = beta;
    st->pNorm2 = add_rn(gamma_next, mul_rn(mul_rn(beta, beta), st->pNorm2));
    st->gamma = gamma_next;
  }
  st->iter = it1;
  st->solved = solved;
  st->tired = it1 >= st->itmax;
  st->done = solved || st->tired;
}

// Global (all ranks) value of a finished local reduction; flags a dead peer.
template <class T>
__device__ __forceinline__ bool cg_global_sum(CgState<T>* st, DistComm* dc, T& v) {
  if (dc) {
    v = dist_reduce(dc, v);
    if (dc->error) { st->comm_error = 1; st->done = 1; return false; }
  }
  return true;
}

// MODE is a compile-time variant so that the plain path carries no dead branches inside the 8-deep gather batch
// (a run-time `if (mdiag)` between the loads cost 11 % of K1: profiles/r1_ab.txt):
//   0 = single GPU, M = I      1 = row-partitioned (halo columns)      2 = single GPU, Diagonal M (Jacobi)
//   3 = single GPU, block-diagonal M (block-Jacobi; z = M r is materialised block by block in phase B)
constexpr int kPlain = 0, kDist = 1, kJacobi = 2, kBlockJac = 3;   // kBlockJac: persistent kernel only

template <class T, int MODE>
struct PVal {               // p_j = z_j + beta p_j, for local and (kDist) halo columns
  const T* r; const T* p_old; T beta; const CgPeers<T>* peers;
  const T* mdiag;           // Jacobi / Diagonal M (cg.jl:241 z = M r applied on the fly); nullptr: M = I, z == r
  __device__ __forceinline__ T operator()(int j) const {
    if (MODE == kDist && j >= peers->halo.nloc) {
      const int h = j - peers->halo.nloc;
      if (peers->r_halo)     // push mode: the owners stored these entries into my halo buffers
        return add_rn(__ldg(&peers->r_halo[h]), mul_rn(beta, __ldg(&peers->p_halo_old[h])));
      const int rk = __ldg(&peers->halo.src_rank[h]), off = __ldg(&peers->halo.src_off[h]);
      return add_rn(__ldg(&peers->r[rk][off]), mul_rn(beta, __ldg(&peers->p_old[rk][off])));
    }
    T z = __ldg(&r[j]);
    if (MODE == kJacobi) z = mul_rn(__ldg(&mdiag[j]), z);
    return add_rn(z, mul_rn(beta, __ldg(&p_old[j])));
  }
};

// ---- K1, TMA-staged -------------------------------------------------------
// MINB = 4 caps the kernel at 56 registers so four CTAs fit on an SM (a few bytes of spill); MINB = 1 leaves
// ptxas free (72 registers, three CTAs).  The plan's CTAs-per-SM choice selects the variant.
//
// XUP: K1 of iteration k also applies the PREVIOUS iteration's solution update x += alpha_{k-1} p_{k-1}
// (cg.jl:239).  K1 holds p_{k-1}[row] in a register anyway (it forms p_k = z + beta p_{k-1}), so moving the update
// here removes K2's read of p: one vector pass less per iteration (the 9nv of SURVEY's B_cg instead of 10nv).
// The arithmetic is unchanged (same add/mul on the same operands); the update of the LAST iteration is applied
// by the host loop at exit.  Not used when a callback must see a current x after every iteration.
template <class T> struct RowPre { T pn, po, xr; };

template <class T, int MODE, int MINB, bool XUP>
__global__ void __launch_bounds__(kTileThreads, MINB) cg_k1_tma(Csr<T> A, const T* __restrict__ r, const T* __restrict__ p_old,
                                                          T* __restrict__ p_new, T* __restrict__ Ap, CgState<T>* st,
                                                          T* part, unsigned* ticket, DistComm* dc, CgPeers<T> peers,
                                                          T* __restrict__ x) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ T sm[32];
  if (*(volatile int*)&st->done) return;
  T dacc = T(0);
  bool sent = false;
  const T beta = st->beta, alpha_prev = st->alpha;
  const bool xup = XUP && st->iter > 0;            // nothing pending before the first iteration
  const PVal<T, MODE> pval{r, p_old, beta, &peers, peers.mdiag};
  auto row_begin = [&](int row) {
    RowPre<T> q;
    q.po = __ldg(&p_old[row]);
    T z = __ldg(&r[row]);
    if (MODE == kJacobi) z = mul_rn(__ldg(&peers.mdiag[row]), z);
    q.pn = add_rn(z, mul_rn(beta, q.po));
    q.xr = xup ? x[row] : T(0);
    return q;
  };
  spmv_tiles_run<T>(A, smem, pval, row_begin, [&](int row, T acc, RowPre<T> q) {
    p_new[row] = q.pn;
    if (MODE == kDist) sent |= peers.push_p(row, q.pn);
    Ap[row] = acc;
    if (xup) x[row] = add_rn(q.xr, mul_rn(alpha_prev, q.po));
    dacc += q.pn * acc;
  });
  if (MODE == kDist && sent) __threadfence_system();   // pushed halo entries visible to the peers before the all-reduce
  T mine[1] = {block_sum(dacc, sm)}, tot[1];
  if (grid_sum_last<T, 1>(mine, part, ticket, sm, tot) && threadIdx.x == 0) {
    if (cg_global_sum(st, MODE == kDist ? dc : nullptr, tot[0])) cg_k1_finalize(st, tot[0]);
  }
}

// ---- K1, row-per-thread LDG (when the tile plan does not fit) --------------
template <class T, int MODE, bool XUP>
__global__ void __launch_bounds__(kBlock) cg_k1_rows(Csr<T> A, const T* __restrict__ r, const T* __restrict__ p_old,
                                                     T* __restrict__ p_new, T* __restrict__ Ap, CgState<T>* st, T* part,
                                                     unsigned* ticket, DistComm* dc, CgPeers<T> peers, T* __restrict__ x) {
  __shared__ T sm[32];
  if (*(volatile int*)&st->done) return;
  T dacc = T(0);
  bool sent = false;
  const T alpha_prev = st->alpha;
  const bool xup = XUP && st->iter > 0;
  const PVal<T, MODE> pval{r, p_old, st->beta, &peers, peers.mdiag};
  const int stride = gridDim.x * blockDim.x;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < A.n; row += stride) {
    const int kb = A.rowptr[row], ke = A.rowptr[row + 1];
    T acc = T(0);
    for (int k = kb; k < ke; k++) acc = add_rn(acc, mul_rn(A.val[k], pval(A.colind[k])));
    const T pn = pval(row);
    p_new[row] = pn;
    if (MODE == kDist) sent |= peers.push_p(row, pn);
    Ap[row] = acc;
    if (xup) x[row] = add_rn(x[row], mul_rn(alpha_prev, __ldg(&p_old[row])));
    dacc += pn * acc;
  }
  if (MODE == kDist && sent) __threadfence_system();
  T mine[1] = {block_sum(dacc, sm)}, tot[1];
  if (grid_sum_last<T, 1>(mine, part, ticket, sm, tot) && threadIdx.x == 0) {
    if (cg_global_sum(st, MODE == kDist ? dc : nullptr, tot[0])) cg_k1_finalize(st, tot[0]);
  }
}

// ---- K2 -------------------------------------------------------------------
// XK2 = true: K2 also applies x += alpha p (cg.jl:239) -- used when K1 runs without XUP (callbacks / verbose).
template <class T, int MODE, bool XK2>   // MODE: kPlain | kDist (push_r may be active) | kJacobi
__global__ void __launch_bounds__(kBlock) cg_k2(int n, T* __restrict__ x, T* __restrict__ r, const T* __restrict__ p,
                                                const T* __restrict__ Ap, CgState<T>* st, T* part, unsigned* ticket,
                                                DistComm* dc, const T* __restrict__ mdiag, PushPlan<T> push_r) {
  __shared__ T sm[32];
  if (*(volatile int*)&st->done) return;
  const T alpha = st->alpha, nalpha = -alpha;
  T acc = T(0);
  bool sent = false;
  // (Measured and rejected, profiles/r1_sweep_k1.txt: walking K2 downwards with evict-first x accesses to reuse
  //  the L2 tails left by K1 made K2 13 % and the following K1 8 % SLOWER -- ascending plain accesses stay.)
  const int stride = gridDim.x * blockDim.x;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    T xv[4], rv[4], pv[4], av[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int j = i + u * stride;
      rv[u] = r[j]; av[u] = __ldg(&Ap[j]);
      if (XK2) { xv[u] = x[j]; pv[u] = __ldg(&p[j]); }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int j = i + u * stride;
      if (XK2) x[j] = add_rn(xv[u], mul_rn(alpha, pv[u]));
      const T rn = add_rn(rv[u], mul_rn(nalpha, av[u]));
      r[j] = rn;
      if (MODE == kDist) sent |= push_r(j, rn);                             // row-partitioned: neighbours' halo copy of r
      acc += rn * (MODE == kJacobi ? mul_rn(__ldg(&mdiag[j]), rn) : rn);   // <r, z>, z = M r (cg.jl:241-242)
    }
  }
  for (; i < n; i += stride) {
    const int j = i;
    if (XK2) x[j] = add_rn(x[j], mul_rn(alpha, p[j]));
    const T rn = add_rn(r[j], mul_rn(nalpha, Ap[j]));
    r[j] = rn;
    if (MODE == kDist) sent |= push_r(j, rn);
    acc += rn * (MODE == kJacobi ? mul_rn(__ldg(&mdiag[j]), rn) : rn);
  }
  if (MODE == kDist && sent) __threadfence_system();
  T mine[1] = {block_sum(acc, sm)}, tot[1];
  if (grid_sum_last<T, 1>(mine, part, ticket, sm, tot) && threadIdx.x == 0) {
    if (cg_global_sum(st, dc, tot[0])) cg_k2_finalize(st, tot[0]);
  }
}

// ===========================================================================
// Persistent cooperative variant: ONE launch runs a whole batch of iterations.
//
// Same arithmetic as cg_k1_tma + cg_k2 (phase A = K1 with the x update riding along, phase B = K2), but the two
// kernel boundaries of an iteration become two grid-wide barriers inside a co-resident grid:
//   * no launch gap / ramp-down / ramp-up between the phases;
//   * the TMA producer warp runs AHEAD of the barrier: as soon as the consumers release the last ring slots of
//     phase A it streams the first tiles of the NEXT iteration's phase A (the matrix does not change), so after
//     the beta barrier the consumers find their first tiles already in shared memory;
//   * each barrier carries its reduction: CTAs publish their partial, the last one to arrive re-reduces all
//     partials in index order (deterministic), runs the scalar recurrence (cg_k1_finalize / cg_k2_finalize) and,
//     row-partitioned, the cross-GPU all-reduce with a full warp, then releases the others.
// Row-partitioned (MODE = kDist): the halo is STAGED instead of being pulled nonzero by nonzero.  At the start of
// phase A every CTA's producer warp fetches its share of the halo list from the owners' r and p buffers with
// coalesced system-scope loads (all in flight at once: one NVLink round trip) and stores the entries into the
// TAILS of the local r and p buffers (nloc + nhalo entries each), so that the gather is the single-GPU code with
// no halo branch at all; tiles with halo columns are ordered LAST in every CTA's tile sequence (tile_order) and
// wait for the staging counter, so the exchange hides behind the interior tiles.
//
// Memory model: vectors written in one phase are read in the next through plain (coherent) loads after the
// barrier's acquire; nothing that changes during the launch is read through the non-coherent path (__ldg).
// ===========================================================================
struct GridBar { unsigned count, gen, halo_ready, timed_iters; unsigned long long ns_a, ns_b; };

__device__ __forceinline__ unsigned ld_acquire_gpu_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ double ld_sys(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_sys(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}

// Grid-wide barrier that also sums one value per thread over the whole grid.  `fin(total)` runs in warp 0 of the
// LAST CTA to arrive (total valid in every lane of that warp) before anyone is released.  Returns false (in every
// thread) if the wait timed out: the caller must leave the kernel.
// The iteration scalars every thread needs after a barrier, broadcast through shared memory: ONE thread per CTA
// reads them from the device block (four independent loads, one L2 round trip) instead of every thread doing four or
// five dependent volatile reads per iteration.
template <class T> struct CgScal { T alpha, beta; int iter, done; };
template <class T>
__device__ __forceinline__ void cg_load_scal(const CgState<T>* st, CgScal<T>* sc) {
  const volatile CgState<T>* v = st;
  const T al = v->alpha, be = v->beta;
  const int it = v->iter, dn = v->done;
  sc->alpha = al; sc->beta = be; sc->iter = it; sc->done = dn;
}

template <class T, class Fin>
__device__ __forceinline__ bool grid_reduce_barrier(GridBar* gb, T v, T* part, T* sm, unsigned* sflag, const CgState<T>* st,
                                                    CgScal<T>* sc, Fin fin) {
  const T mine = block_sum(v, sm);
  if (threadIdx.x == 0) {
    const unsigned g = *(volatile unsigned*)&gb->gen;      // read BEFORE arriving
    __stcg(&part[blockIdx.x], mine);
    __threadfence();
    const unsigned t = atomicAdd(&gb->count, 1u);
    sflag[0] = (t == gridDim.x - 1);
    sflag[1] = g;
  }
  __syncthreads();
  const bool last = sflag[0] != 0;
  const unsigned g = sflag[1];
  bool ok = true;
  if (last) {
    if (threadIdx.x < 32) {
      // warp 0 alone re-reduces the partials (fixed order: lane-strided, then the shuffle tree): no CTA-wide
      // synchronisation on the critical path of the release
      __threadfence();
      T acc = T(0);
      for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) acc += __ldcg(&part[i]);
      const T tot = warp_sum(acc);          // valid in every lane
      fin(tot);
      __syncwarp();
      if (threadIdx.x == 0) {
        cg_load_scal<T>(st, sc);             // after this thread's own finalize
        gb->count = 0u;                      // ordered before the release below (st.release covers this thread's prior writes)
        st_release_gpu_u32(&gb->gen, g + 1u);
      }
    }
  } else if (threadIdx.x == 0) {
    const long long t0 = clock64();
    while (ld_acquire_gpu_u32(&gb->gen) == g) {
      if (clock64() - t0 > 120000000000LL) { sflag[0] = 2; break; }     // ~1 minute: the grid is wedged
    }
    cg_load_scal<T>(st, sc);
  }
  __syncthreads();
  if (sflag[0] == 2) ok = false;
  __syncthreads();           // sflag is rewritten by the next barrier
  return ok;
}

template <class T>
struct CgPeerTab {          // device-resident table of the peers' buffers (row-partitioned solves)
  const T* r[kMaxRanks];
  const T* p[2][kMaxRanks];  // in the order of CgPersistArgs::P
};

template <class T>
struct CgPersistArgs {
  T* r; T* P0; T* P1; T* Ap; T* x;     // P0 / P1: direction buffers; iteration k reads P[k & 1], writes the other
  const T* mdiag;            // kJacobi
  T* z;                      // kBlockJac: z = M r, written in phase B, gathered in phase A in place of r
  const T* mblocks;          //            dense bs x bs diagonal blocks of M, row-major
  int mbs;
  HaloMap halo;              // kDist ...
  const CgPeerTab<T>* tab;
  const int* tile_order;     // interior tiles first, tiles with halo columns last (bit 31 set)
  int n_interior;            // number of interior tiles = first halo position of tile_order
  int max_iters;
  int timed;                 // accumulate phase durations (CTA 0, %globaltimer) into the GridBar block
  // Zero-copy report: when the launch ends, CTA 0 copies the scalar block into pinned HOST memory and then stores the
  // launch's sequence number there.  The host polls that word instead of an event behind a D2H copy, so consecutive
  // persistent launches sit back to back on the stream (a copy between two kernels costs two engine hand-offs).
  CgState<T>* hsnap;
  unsigned long long* hseq;
  unsigned long long seq;
};

template <class T>
__device__ __forceinline__ void cg_report_to_host(const CgPersistArgs<T>& a, const CgState<T>* st) {
  if (blockIdx.x != 0 || threadIdx.x >= 32 || a.hsnap == nullptr) return;
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(st);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(a.hsnap);
  for (int w = threadIdx.x; w < (int)(sizeof(CgState<T>) / 8); w += 32) dst[w] = __ldcg(&src[w]);
  __threadfence_system();
  __syncwarp();
  if (threadIdx.x == 0) { *(volatile unsigned long long*)a.hseq = a.seq; __threadfence_system(); }
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// Phase B with a block-Jacobi M (cg.jl:240-242): one thread per diagonal block updates r, forms z = M_blk r on the
// spot (the block's rows are all in this thread's registers) and accumulates <r, z>.  BS = 0: run-time block size.
template <class T, int BS>
__device__ __forceinline__ T cg_phase_b_block(int n, int bs_rt, T nalpha, T* r, const T* Ap, T* z, const T* __restrict__ B, int first, int stride) {
  const int bs = BS ? BS : bs_rt;
  const int nb = (n + bs - 1) / bs;
  T acc = T(0);
  for (int blk = first; blk < nb; blk += stride) {
    const int r0 = blk * bs, rows = min(bs, n - r0);
    T rn[BS ? BS : 8];
#pragma unroll
    for (int i = 0; i < (BS ? BS : 8); i++)
      if (i < rows) { rn[i] = add_rn(r[r0 + i], mul_rn(nalpha, Ap[r0 + i])); r[r0 + i] = rn[i]; }
    const T* Bk = B + (size_t)blk * bs * bs;
#pragma unroll
    for (int i = 0; i < (BS ? BS : 8); i++) {
      if (i < rows) {
        T zi = T(0);
#pragma unroll
        for (int j = 0; j < (BS ? BS : 8); j++)
          if (j < rows) zi = add_rn(zi, mul_rn(__ldg(&Bk[i * bs + j]), rn[j]));
        z[r0 + i] = zi;
        acc += rn[i] * zi;
      }
    }
  }
  return acc;
}

// Halo staging of the row-partitioned persistent kernel (one warp per CTA): this CTA's share of the halo list, all
// loads in flight at once.  The halo entries of r and of the old direction land in the TAILS of the local vectors
// (r and the p buffers of a row-partitioned workspace hold nloc + nhalo entries), so the gather of phase A is
// exactly the single-GPU code: column j >= nloc is simply element j of the same array.  The CONSUMER threads do
// it, one entry per thread and trip, before their first tile: the share of a CTA is usually <= 256 entries, i.e.
// one NVLink round trip for the whole CTA, while the producer warp keeps the tile ring full.  (First version: the
// producer warp staged, 7 dependent round trips per lane during which it issued no tiles -- the consumers starved
// for ~15 us per iteration at 2 GPUs.  An explicit 8-deep unroll made ptxas schedule the gather batches of the same
// kernel as load -> use chains, so the loop is left to the compiler.)
template <class T>
__device__ __forceinline__ void cg_stage_halo(HaloMap halo, const CgPeerTab<T>* tab, T* r, T* p_old, int pb, int G, int tid, int nthreads) {
  const int nh = halo.nhalo, nloc = halo.nloc;
  const int per = (nh + G - 1) / G;
  const int h0 = (int)blockIdx.x * per, h1 = min(nh, h0 + per);
  for (int h = h0 + tid; h < h1; h += nthreads) {
    const int rk = __ldg(&halo.src_rank[h]), off = __ldg(&halo.src_off[h]);
    const T rv = ld_sys(tab->r[rk] + off);
    const T pv = ld_sys(tab->p[pb][rk] + off);
    __stcg(&r[nloc + h], rv);
    __stcg(&p_old[nloc + h], pv);
  }
}

// DICT: the matrix streams as the operator's dictionary codes (Csr::code); kPlain and kJacobi at 3 CTAs per SM.
template <class T, int MODE, int MINB, int DEPTH, bool DICT>
__global__ void __launch_bounds__(kTileThreads, MINB) cg_persist(Csr<T> A, CgPersistArgs<T> a, CgState<T>* st, T* part,
                                                                GridBar* gb, DistComm* dc) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ T sm[32];
  __shared__ unsigned sflag[2];
  __shared__ CgScal<T> sc;
  volatile CgState<T>* vst = st;
  if (vst->done) { cg_report_to_host<T>(a, st); return; }    // uniform: st only changes inside the barriers below
  if (threadIdx.x == 0) cg_load_scal<T>(st, &sc);            // published by the __syncthreads of P.init below
  TilePipe<T, DICT> P;
  P.init(A, smem);
  const int G = gridDim.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cnt = (A.ntiles - (int)blockIdx.x + G - 1) / G;         // grid <= ntiles: cnt >= 1
  auto tile_at = [&](int j) -> int {
    const int q = blockIdx.x + j * G;
    return MODE == kDist ? __ldg(&a.tile_order[q]) : q;
  };
  // row-partitioned: positions >= n_interior of the tile order are halo tiles; this CTA owns positions b + j G
  const int cnt_int = MODE == kDist ? max(0, min(cnt, (a.n_interior - (int)blockIdx.x + G - 1) / G)) : cnt;
  const unsigned pre = (unsigned)min(P.S, cnt);
  const uint64_t pol = l2_evict_first_policy();
  unsigned ppos = 0, cpos = 0;
  int passes = 0;
  const int n = A.n;
  for (int k = 0; k < a.max_iters; k++) {
    const int iter = sc.iter;
    const T beta = sc.beta, alpha_prev = sc.alpha;
    const bool xup = iter > 0;                 // x += alpha_{k-1} p_{k-1} rides in phase A (cg.jl:239)
    T* p_old = (iter & 1) ? a.P1 : a.P0;
    T* p_new = (iter & 1) ? a.P0 : a.P1;
    T dacc = T(0);
    const bool timing = a.timed && blockIdx.x == 0 && tid == 0;
    unsigned long long t0 = 0, t1 = 0;
    if (timing) t0 = globaltimer_ns();
    // ------------------------------ phase A (= K1) ------------------------------
    if (warp == kConsumerWarps) {
      if (lane == 0) {
        const unsigned target = (unsigned)(k + 1) * (unsigned)cnt + (k + 1 < a.max_iters ? pre : 0u);
        tile_issue_until<T, DICT>(A, P, ppos, target, cnt, tile_at, pol);
      }
    } else {
      const T* r = MODE == kBlockJac ? a.z : a.r;      // block-Jacobi: gather z = M r (materialised by phase B)
      const T* mdiag = a.mdiag;
      auto gather = [&](int j) -> T {          // p_j = z_j + beta p_j (cg.jl:259 applied on the fly); row-partitioned:
        T z = r[j];                            // j >= nloc reads the staged tail of the same arrays
        if (MODE == kJacobi) z = mul_rn(__ldg(&mdiag[j]), z);
        return add_rn(z, mul_rn(beta, p_old[j]));
      };
      auto row_begin = [&](int row) {
        RowPre<T> q;
        q.po = p_old[row];
        T z = r[row];
        if (MODE == kJacobi) z = mul_rn(__ldg(&mdiag[row]), z);
        q.pn = add_rn(z, mul_rn(beta, q.po));
        q.xr = xup ? a.x[row] : T(0);
        return q;
      };
      auto row_done = [&](int row, T acc, RowPre<T> q) {
        p_new[row] = q.pn;
        a.Ap[row] = acc;
        if (xup) a.x[row] = add_rn(q.xr, mul_rn(alpha_prev, q.po));
        dacc += q.pn * acc;
      };
      if (MODE == kDist) {
        cg_stage_halo<T>(a.halo, a.tab, a.r, p_old, iter & 1, G, tid, kTileRows);
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicAdd(&gb->halo_ready, 1u);       // 8 consumer warps per CTA report
        // interior tiles first; the tiles with halo columns (last in this CTA's sequence) only after every CTA's
        // producer warp has staged its share of the halo
        tile_consume_pass<T, DEPTH, DICT>(A, P, cpos, 0, cnt_int, tile_at, gather, row_begin, row_done);
        if (cnt_int < cnt) {
          if (lane == 0) { while (ld_acquire_gpu_u32(&gb->halo_ready) < (unsigned)(G * kConsumerWarps)) { } }
          __syncwarp();
          tile_consume_pass<T, DEPTH, DICT>(A, P, cpos, cnt_int, cnt, tile_at, gather, row_begin, row_done);
        }
      } else {
        tile_consume_pass<T, DEPTH, DICT>(A, P, cpos, 0, cnt, tile_at, gather, row_begin, row_done);
      }
    }
    passes = k + 1;
    bool ok = grid_reduce_barrier<T>(gb, dacc, part, sm, sflag, st, &sc, [&](T tot) {
      if (MODE == kDist) {
        tot = (T)dist_allreduce_sum_warp<T>(dc, (double)tot);
        if (*(volatile int*)&dc->error) { if (lane == 0) { st->comm_error = 1; st->done = 1; } return; }
      }
      if (lane == 0) cg_k1_finalize(st, tot);
    });
    if (!ok || sc.done) break;
    if (timing) t1 = globaltimer_ns();
    // ------------------------------ phase B (= K2) ------------------------------
    {
      const T alpha = sc.alpha, nalpha = -alpha;
      T* r = a.r;
      const T* Ap = a.Ap;
      const T* mdiag = a.mdiag;
      T acc = T(0);
      const int stride = G * kTileThreads;
      int i = (int)blockIdx.x * kTileThreads + tid;
      if (MODE == kBlockJac) {
        if (a.mbs == 4) acc = cg_phase_b_block<T, 4>(n, 4, nalpha, r, Ap, a.z, a.mblocks, i, stride);
        else if (a.mbs == 2) acc = cg_phase_b_block<T, 2>(n, 2, nalpha, r, Ap, a.z, a.mblocks, i, stride);
        else if (a.mbs == 8) acc = cg_phase_b_block<T, 8>(n, 8, nalpha, r, Ap, a.z, a.mblocks, i, stride);
        else acc = cg_phase_b_block<T, 0>(n, a.mbs, nalpha, r, Ap, a.z, a.mblocks, i, stride);
        i = n;                                  // the element loops below are skipped
      }
      for (; i + 3 * stride < n; i += 4 * stride) {
        T rv[4], av[4];
#pragma unroll
        for (int u = 0; u < 4; u++) { rv[u] = r[i + u * stride]; av[u] = Ap[i + u * stride]; }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int j = i + u * stride;
          const T rn = add_rn(rv[u], mul_rn(nalpha, av[u]));
          r[j] = rn;
          acc += rn * (MODE == kJacobi ? mul_rn(__ldg(&mdiag[j]), rn) : rn);
        }
      }
      for (; i < n; i += stride) {
        const T rn = add_rn(r[i], mul_rn(nalpha, Ap[i]));
        r[i] = rn;
        acc += rn * (MODE == kJacobi ? mul_rn(__ldg(&mdiag[i]), rn) : rn);
      }
      ok = grid_reduce_barrier<T>(gb, acc, part, sm, sflag, st, &sc, [&](T tot) {
        if (MODE == kDist) {
          tot = (T)dist_allreduce_sum_warp<T>(dc, (double)tot);
          if (*(volatile int*)&dc->error) { if (lane == 0) { st->comm_error = 1; st->done = 1; } return; }
        }
        if (lane == 0) {
          cg_k2_finalize(st, tot);
          gb->halo_ready = 0u;                 // every consumer is past phase A: re-arm the staging counter
        }
      });
      if (timing) {
        const unsigned long long t2 = globaltimer_ns();
        gb->ns_a += t1 - t0; gb->ns_b += t2 - t1; gb->timed_iters += 1;
      }
      if (!ok || sc.done) break;
    }
  }
  if (warp == kConsumerWarps && lane == 0) tile_drain<T, DICT>(P, (unsigned)passes * (unsigned)cnt, ppos);
  cg_report_to_host<T>(a, st);                 // st is final: every CTA left the loop after the same barrier
}

// Prologue of a row-partitioned solve in push mode: send the boundary entries of r_0 to the neighbours' halo
// buffers.  The all-reduce of the prologue's <r,z> (launched next on the same stream) orders it before any K1.
template <class T>
__global__ void push_ranges_kernel(const T* __restrict__ v, PushPlan<T> plan) {
  const int stride = gridDim.x * blockDim.x, tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (int q = 0; q < plan.nranges; q++)
    for (int d = tid; d < plan.rg[q].count; d += stride) plan.dst[q][plan.rg[q].slot + d] = v[plan.rg[q].start + d];
  __threadfence_system();
}

template <class T> void cg_dist_push_r(Workspace<T>& ws) {
  if (ws.dist.world <= 1 || ws.dist.npush <= 0) return;
  PushPlan<T> plan;
  memset(&plan, 0, sizeof(plan));
  plan.nranges = ws.dist.npush;
  for (int q = 0; q < ws.dist.npush; q++) { plan.rg[q] = ws.dist.push[q]; plan.dst[q] = ws.dist.halo_buf_peer[plan.rg[q].peer]; }
  push_ranges_kernel<T><<<sm_count(), kBlock, 0, ws.ctx.stream>>>(ws.r, plan);
  KB_CUDA(cudaGetLastError());
  ws.ctx.launches++;
}

// ---------------------------------------------------------------------------
// Everything the fused loops need besides the solver's vectors is allocated when the workspace is created
// (ws_create) -- the in-place call allocates nothing (test/test_allocations.jl:54-57).
constexpr size_t kOffGridBar = 1024, kOffPeerTab = 2048, kOffHostSeq = 3072;     // layout of the 4 KB device / pinned blocks

template <class T> void cg_fused_prepare(Workspace<T>& ws) {
  static_assert(sizeof(CgState<T>) <= kOffGridBar && sizeof(CgPeerTab<T>) <= kFusedBlockBytes - kOffPeerTab, "block layout");
  if (!ws.fused_state) {
    KB_CUDA(cudaMalloc(&ws.fused_state, kFusedBlockBytes));
    KB_CUDA(cudaMemset(ws.fused_state, 0, kFusedBlockBytes));
    KB_CUDA(cudaHostAlloc(&ws.fused_host, kFusedBlockBytes, cudaHostAllocPortable | cudaHostAllocMapped));
    memset(ws.fused_host, 0, kFusedBlockBytes);
  }
  if (!ws.p2) ws.p2 = dev_alloc<T>((size_t)ws.n);
  for (int i = 0; i < 2; i++)
    if (!ws.fused_ev[i]) KB_CUDA(cudaEventCreateWithFlags(&ws.fused_ev[i], cudaEventDisableTiming));
}

// Row-partitioned persistent CG: order of the row tiles -- tiles without halo columns first, tiles that gather
// halo entries last (bit 31 set), so that every CTA reaches its halo tiles at the END of phase A, long after the
// halo staging of that iteration has finished.
template <class T>
__global__ void tile_halo_flags_kernel(Csr<T> A, int nloc, int* flags) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nw = (gridDim.x * blockDim.x) >> 5;
  for (int t = warp; t < A.ntiles; t += nw) {
    const int k0 = A.rowptr[t * kTileRows], k1 = A.rowptr[min(t * kTileRows + kTileRows, A.n)];
    bool any = false;
    for (int k = k0 + lane; k < k1; k += 32) any |= A.colind[k] >= nloc;
    any = __any_sync(0xffffffffu, any);
    if (lane == 0) flags[t] = any ? 1 : 0;
  }
}

template <class T> void cg_dist_tile_order(Workspace<T>& ws, const Csr<T>& A) {
  if (ws.dist.tile_order && ws.dist.tile_order_for == (const void*)A.rowptr && ws.dist.tile_order_n == A.ntiles) return;
  Ctx& c = ws.ctx;
  if (ws.dist.tile_order) { cudaFree(ws.dist.tile_order); ws.dist.tile_order = nullptr; }
  const int nt = A.ntiles;
  KB_CUDA(cudaMalloc((void**)&ws.dist.tile_order, sizeof(int) * (size_t)(nt > 0 ? nt : 1)));
  if (nt > 0) {
    tile_halo_flags_kernel<T><<<sm_count() * 4, 256, 0, c.stream>>>(A, ws.n, ws.dist.tile_order);
    KB_CUDA(cudaGetLastError());
    std::vector<int> fl(nt), ord;
    KB_CUDA(cudaMemcpyAsync(fl.data(), ws.dist.tile_order, sizeof(int) * nt, cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    ord.reserve(nt);
    for (int t = 0; t < nt; t++) if (!fl[t]) ord.push_back(t);
    ws.dist.tile_order_interior = (int)ord.size();
    for (int t = 0; t < nt; t++) if (fl[t]) ord.push_back((int)((unsigned)t | 0x80000000u));
    KB_CUDA(cudaMemcpyAsync(ws.dist.tile_order, ord.data(), sizeof(int) * nt, cudaMemcpyHostToDevice, c.stream));
    c.sync();
  }
  ws.dist.tile_order_for = (const void*)A.rowptr;
  ws.dist.tile_order_n = nt;
}

// ---------------------------------------------------------------------------
template <class T> bool cg_fused_eligible(const LinOp<T>& A, const LinOp<T>& M, const SolveOpts& o) {
  // M = I, or a Diagonal M applied with mul! (the Jacobi case of SURVEY.md 8f-1), folded into the two kernels
  const bool m_ok = M.is_identity() || (M.kind == LinOp<T>::DIAG && !o.ldiv);
  if (o.fused && A.kind == LinOp<T>::CSR && M.kind == LinOp<T>::BDIAG && !o.ldiv && o.radius == 0) {
    // block-Jacobi M: only the persistent kernel carries it (phase B forms z = M r block by block)
    const char* epers = getenv("KB200_PERSIST");
    const bool single_step = (o.callback != nullptr) || (o.timemax < 1e300) || o.verbose > 0;
    return A.csr->tma_ok && o.persist != 0 && !single_step && !(epers && atoi(epers) == 0);
  }
  return o.fused && A.kind == LinOp<T>::CSR && m_ok && o.radius == 0;
}

template <class T>
void cg_fused_loop(Workspace<T>& ws, const Csr<T>& A, const SolveOpts& o, T gamma0, T eps_tol, int itmax, double start_time,
                   bool& solved, bool& tired, bool& zero_curvature, bool& inconsistent, bool& user_exit, bool& overtimed,
                   int& iter) {
  Ctx& c = ws.ctx;
  const int n = ws.n;
  typedef CgState<T> St;
  const bool dist = ws.dist.world > 1;
  cg_fused_prepare<T>(ws);                      // no-op: done at workspace creation
  St* dst = (St*)ws.fused_state;
  St* hst = (St*)ws.fused_host;                 // two read-back slots, kOffGridBar apart
  auto hslot = [&](int i) -> St* { return (St*)((char*)hst + (size_t)i * kOffGridBar); };

  St init;
  memset(&init, 0, sizeof(init));
  init.gamma = gamma0; init.pNorm2 = gamma0; init.beta = T(0); init.eps_tol = eps_tol;
  init.rNorm = sqrt(gamma0); init.itmax = itmax; init.linesearch = o.linesearch ? 1 : 0;
  *hslot(0) = init;
  KB_CUDA(cudaMemcpyAsync(dst, hslot(0), sizeof(St), cudaMemcpyHostToDevice, c.stream));
  KB_CUDA(cudaMemsetAsync((char*)ws.fused_state + kOffGridBar, 0, sizeof(GridBar), c.stream));
  // (no sync: the copy reads slot 0 in stream order before any kernel or read-back of this solve writes it)

  const bool jac = ws.mdiag_fused != nullptr;
  const bool single_step = (o.callback != nullptr) || (o.timemax < 1e300) || o.verbose > 0;
  // x += alpha p moves from K2 into the next K1 (one vector pass less) unless x must be current after every
  // iteration (callbacks, verbose, time limits) -- KB200_XUP=0 keeps the update in K2 for A/B measurements.
  const char* exu = getenv("KB200_XUP");
  const bool xup = !single_step && !(exu && atoi(exu) == 0);
  // All variants share one signature: pick the kernel once.
  typedef void (*K1Fn)(Csr<T>, const T*, const T*, T*, T*, CgState<T>*, T*, unsigned*, DistComm*, CgPeers<T>, T*);
  typedef void (*K2Fn)(int, T*, T*, const T*, const T*, CgState<T>*, T*, unsigned*, DistComm*, const T*, PushPlan<T>);
  K1Fn k1 = nullptr;
  K2Fn k2 = nullptr;
  if (A.tma_ok) {
    if (dist) k1 = xup ? cg_k1_tma<T, kDist, 3, true> : cg_k1_tma<T, kDist, 3, false>;
    else if (jac) k1 = xup ? cg_k1_tma<T, kJacobi, 3, true> : cg_k1_tma<T, kJacobi, 3, false>;
    else if (A.ctas_per_sm >= 4) k1 = xup ? cg_k1_tma<T, kPlain, 4, true> : cg_k1_tma<T, kPlain, 4, false>;
    else if (A.ctas_per_sm == 3) k1 = xup ? cg_k1_tma<T, kPlain, 3, true> : cg_k1_tma<T, kPlain, 3, false>;
    else k1 = xup ? cg_k1_tma<T, kPlain, 1, true> : cg_k1_tma<T, kPlain, 1, false>;
  } else {
    if (dist) k1 = xup ? cg_k1_rows<T, kDist, true> : cg_k1_rows<T, kDist, false>;
    else if (jac) k1 = xup ? cg_k1_rows<T, kJacobi, true> : cg_k1_rows<T, kJacobi, false>;
    else k1 = xup ? cg_k1_rows<T, kPlain, true> : cg_k1_rows<T, kPlain, false>;
  }
  if (dist) k2 = xup ? cg_k2<T, kDist, false> : cg_k2<T, kDist, true>;
  else if (jac) k2 = xup ? cg_k2<T, kJacobi, false> : cg_k2<T, kJacobi, true>;
  else k2 = xup ? cg_k2<T, kPlain, false> : cg_k2<T, kPlain, true>;
  // The persistent grid must equal what is actually co-resident: a register count that silently drops the
  // occupancy below the plan's CTAs/SM would otherwise run the tiles in 1.5 waves (measured: K1 2.2x slower).
  int k1_grid = A.grid;
  if (A.tma_ok) {
    ensure_dyn_smem((const void*)k1, 220 * 1024);
    int occ = 0;
    KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k1, kTileThreads, A.smem_bytes));
    if (occ < 1) throw std::runtime_error("cg_k1_tma does not fit on an SM with the planned shared-memory ring");
    const int resident = std::min(occ, A.ctas_per_sm) * sm_count();
    k1_grid = std::min(resident, std::max(1, A.ntiles));
  }
  const int g2 = stream_grid(n, 4, 8);
  const int g1r = stream_grid(n, 1, 8);
  T* P[2] = {ws.p, ws.p2};   // ws.p holds z (= r) from the prologue: with beta = 0, K1 forms p = r + 0*p
  T* part = (T*)c.partials;
  // peers' direction buffers in the same order as P[]
  CgPeers<T> peersP[2];
  memset(peersP, 0, sizeof(peersP));
  const T* md = ws.mdiag_fused;
  peersP[0].mdiag = md; peersP[1].mdiag = md;
  PushPlan<T> push_r;
  memset(&push_r, 0, sizeof(push_r));
  if (dist) {
    for (int b = 0; b < 2; b++) {
      peersP[b].halo = ws.dist.halo;
      const bool wantB = (b == 1) != ws.dist.swapped;     // P[b] is the bufB allocation?
      for (int k = 0; k < ws.dist.world; k++) {
        peersP[b].r[k] = ws.dist.r_peer[k];
        peersP[b].p_old[k] = wantB ? ws.dist.bufB_peer[k] : ws.dist.bufA_peer[k];
      }
      if (ws.dist.npush > 0) {
        // push mode: halo_buf = [r | p(bufA) | p(bufB)], nhalo entries each (every rank with its own nhalo)
        const size_t nh = (size_t)ws.dist.halo.nhalo;
        peersP[b].r_halo = ws.dist.halo_buf;
        peersP[b].p_halo_old = ws.dist.halo_buf + (wantB ? 2 : 1) * nh;
        peersP[b].push_p.nranges = ws.dist.npush;
        for (int q = 0; q < ws.dist.npush; q++) {
          const PushRange& rg = ws.dist.push[q];
          peersP[b].push_p.rg[q] = rg;
          // K1 with p_old = P[b] writes P[b^1]: the OTHER allocation's section of the peer's halo buffer
          peersP[b].push_p.dst[q] = ws.dist.halo_buf_peer[rg.peer] + (wantB ? 1 : 2) * (size_t)ws.dist.nhalo_peer[rg.peer];
          push_r.rg[q] = rg;
          push_r.dst[q] = ws.dist.halo_buf_peer[rg.peer];
        }
        push_r.nranges = ws.dist.npush;
      }
    }
  }

  static const char* ebatch = getenv("KB200_BATCH");            // A/B measurements of the per-launch fixed cost
  int batch = o.batch > 0 ? o.batch : (single_step ? 1 : (ebatch && atoi(ebatch) > 0 ? atoi(ebatch) : 32));   // iterations per launch / host poll
  if (batch > kHist / 2) batch = kHist / 2;
  if (single_step) batch = 1;

  // Persistent cooperative variant (one launch per batch of iterations): whenever the tile plan is staged and x
  // need not be current after every iteration.  KB200_PERSIST=0 keeps the two-launch kernels (A/B measurements).
  const char* epers = getenv("KB200_PERSIST");
  const bool persist = A.tma_ok && xup && !(epers && atoi(epers) == 0) && o.persist != 0;
  const bool bjac = ws.mblocks_fused != nullptr;
  if (bjac && !persist) throw std::runtime_error("block-Jacobi M reached the fused CG loop without the persistent kernel");
  typedef void (*KpFn)(Csr<T>, CgPersistArgs<T>, CgState<T>*, T*, GridBar*, DistComm*);
  KpFn kp = nullptr;
  int pgrid = 0;
  size_t psmem = 0;
  CgPersistArgs<T> pa;
  memset(&pa, 0, sizeof(pa));
  GridBar* gbar = (GridBar*)((char*)ws.fused_state + kOffGridBar);
  if (persist) {
    // register budget follows the plan's CTAs per SM: 3 (72 registers, the default plan) or 2 (112 registers: all 16
    // loads of an 8-nonzero gather batch in flight per thread; selected with KB200_CTAS_PER_SM=2 / large tiles)
    static const char* edep = getenv("KB200_GATHER_DEPTH");
    const int depth = edep ? atoi(edep) : 0;
    // The dictionary-encoded operator streams ~1 byte per nonzero instead of 12 (DESIGN.md section 3); the plan only
    // builds it for the default 3-CTA/SM ring, and the encoded kernel runs the same grid, so the dot-product trees and
    // with them every iterate are those of the CSR kernel.
    const bool dict = A.ndict > 0 && !dist && !bjac && depth != 4;
    if (dict) {
      kp = jac ? cg_persist<T, kJacobi, 3, 8, true> : cg_persist<T, kPlain, 3, 8, true>;
    } else if (A.ctas_per_sm >= 3) {
      // measured on cfg2 (profiles/README.md, round 2): 8-deep batches 3825 it/s, 4-deep 3691 it/s
      if (bjac) kp = cg_persist<T, kBlockJac, 2, 8, false>;   // the block code of phase B needs the 96-register budget (2 CTAs per SM)
      else if (depth == 4) kp = dist ? cg_persist<T, kDist, 3, 4, false> : (jac ? cg_persist<T, kJacobi, 3, 4, false> : cg_persist<T, kPlain, 3, 4, false>);
      else kp = dist ? cg_persist<T, kDist, 3, 8, false> : (jac ? cg_persist<T, kJacobi, 3, 8, false> : cg_persist<T, kPlain, 3, 8, false>);
    } else {
      if (bjac) kp = cg_persist<T, kBlockJac, 2, 8, false>;
      else if (depth == 4) kp = dist ? cg_persist<T, kDist, 2, 4, false> : (jac ? cg_persist<T, kJacobi, 2, 4, false> : cg_persist<T, kPlain, 2, 4, false>);
      else kp = dist ? cg_persist<T, kDist, 2, 8, false> : (jac ? cg_persist<T, kJacobi, 2, 8, false> : cg_persist<T, kPlain, 2, 8, false>);
    }
    psmem = dict ? A.dict_smem_bytes : A.smem_bytes;
    ensure_dyn_smem((const void*)kp, 220 * 1024);
    int occ = 0;
    KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kp, kTileThreads, psmem));
    if (occ < 1) throw std::runtime_error("cg_persist does not fit on an SM with the planned shared-memory ring");
    pgrid = std::min(std::min(occ, A.ctas_per_sm) * sm_count(), std::max(1, A.ntiles));
    pa.r = ws.r; pa.P0 = ws.p; pa.P1 = ws.p2; pa.Ap = ws.Ap; pa.x = ws.x;
    pa.mdiag = md;
    pa.z = ws.z; pa.mblocks = ws.mblocks_fused; pa.mbs = ws.mbs_fused;
    pa.max_iters = batch;
    pa.timed = o.time_kernels ? 1 : 0;
    if (dist) {
      cg_dist_tile_order<T>(ws, A);
      CgPeerTab<T>* htab = (CgPeerTab<T>*)((char*)ws.fused_host + kOffPeerTab);
      memset(htab, 0, sizeof(*htab));
      for (int b = 0; b < 2; b++) {
        const bool wantB = (b == 1) != ws.dist.swapped;
        for (int k = 0; k < ws.dist.world; k++) {
          htab->r[k] = ws.dist.r_peer[k];
          htab->p[b][k] = wantB ? ws.dist.bufB_peer[k] : ws.dist.bufA_peer[k];
        }
      }
      CgPeerTab<T>* dtab = (CgPeerTab<T>*)((char*)ws.fused_state + kOffPeerTab);
      KB_CUDA(cudaMemcpyAsync(dtab, htab, sizeof(*htab), cudaMemcpyHostToDevice, c.stream));
      pa.halo = ws.dist.halo;
      pa.tab = dtab;
      pa.tile_order = ws.dist.tile_order;
      pa.n_interior = ws.dist.tile_order_interior;
    }
  }

  cudaEvent_t* ev = ws.fused_ev;
  int enq = 0;
  // optional per-kernel timing (bench.py roofline breakdown): events around launches 8..39
  constexpr int kTimedFirst = 8, kTimedCount = 32;
  std::vector<cudaEvent_t> tev;
  if (o.time_kernels) {
    tev.resize(3 * kTimedCount);
    for (auto& e : tev) KB_CUDA(cudaEventCreate(&e));
  }
  // persistent launches report into pinned host memory (cg_report_to_host): poll the sequence word; every ~1000 polls
  // make sure the stream is still alive so that a faulted kernel raises instead of hanging the host
  unsigned long long* hseq = (unsigned long long*)((char*)ws.fused_host + kOffHostSeq);
  unsigned long long expect[2] = {0, 0};
  auto wait_report = [&](int slot) {
    long spins = 0;
    while (__atomic_load_n(&hseq[slot], __ATOMIC_ACQUIRE) != expect[slot]) {
      if ((++spins & 1023) == 0) {
        const cudaError_t q = cudaStreamQuery(c.stream);
        if (q != cudaSuccess && q != cudaErrorNotReady) throw CudaError(std::string("persistent CG kernel failed: ") + cudaGetErrorString(q));
        if (q == cudaSuccess && __atomic_load_n(&hseq[slot], __ATOMIC_ACQUIRE) != expect[slot])
          throw std::runtime_error("persistent CG kernel finished without reporting its state");
      }
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
    }
  };
  auto enqueue = [&](int slot) {
    if (persist) {
      DistComm* dcm = dist ? c.dcomm : nullptr;
      Csr<T> Acopy = A;
      T* partp = part;
      pa.hsnap = hslot(slot);
      pa.hseq = hseq + slot;
      pa.seq = expect[slot] = ++ws.fused_seq;
      void* args[] = {(void*)&Acopy, (void*)&pa, (void*)&dst, (void*)&partp, (void*)&gbar, (void*)&dcm};
      KB_CUDA(cudaLaunchCooperativeKernel((const void*)kp, dim3(pgrid), dim3(kTileThreads), args, psmem, c.stream));
      c.launches += 1;
      enq += batch;
      return;                                   // the kernel reports into pinned host memory itself
    }
    for (int b = 0; !persist && b < batch; b++, enq++) {
      T* p_old = P[enq & 1];
      T* p_new = P[(enq + 1) & 1];
      const CgPeers<T>& pe = peersP[enq & 1];
      const int ti = enq - kTimedFirst;
      const bool timed = o.time_kernels && ti >= 0 && ti < kTimedCount;
      if (timed) KB_CUDA(cudaEventRecord(tev[3 * ti], c.stream));
      DistComm* dcm = dist ? c.dcomm : nullptr;
      if (A.tma_ok) k1<<<k1_grid, kTileThreads, A.smem_bytes, c.stream>>>(A, ws.r, p_old, p_new, ws.Ap, dst, part, c.tickets + 2, dcm, pe, ws.x);
      else k1<<<g1r, kBlock, 0, c.stream>>>(A, ws.r, p_old, p_new, ws.Ap, dst, part, c.tickets + 2, dcm, pe, ws.x);
      if (timed) KB_CUDA(cudaEventRecord(tev[3 * ti + 1], c.stream));
      k2<<<g2, kBlock, 0, c.stream>>>(n, ws.x, ws.r, p_new, ws.Ap, dst, part, c.tickets + 3, dcm, md, push_r);
      if (timed) KB_CUDA(cudaEventRecord(tev[3 * ti + 2], c.stream));
      c.launches += 2;
    }
    KB_CUDA(cudaGetLastError());
    KB_CUDA(cudaMemcpyAsync(hslot(slot), dst, sizeof(St), cudaMemcpyDeviceToHost, c.stream));
    KB_CUDA(cudaEventRecord(ev[slot], c.stream));
  };

  int cur = 0, seen = 0;   // seen: iterations whose rNorm has been pushed to the history
  St last;
  enqueue(0);
  for (;;) {
    if (!single_step) enqueue(cur ^ 1);           // keep the GPU busy while the host inspects `cur`
    if (persist) wait_report(cur);
    else KB_CUDA(cudaEventSynchronize(ev[cur]));
    last = *hslot(cur);
    for (int k = seen + 1; k <= last.iter; k++) {
      if (o.history) ws.stats.residuals.push_back((double)last.hist[k % kHist]);
    }
    seen = last.iter;
    if (last.done) break;
    if (single_step) {
      if (o.verbose > 0 && (last.iter % o.verbose == 0))
        fprintf(stdout, "%5d  %7.1e  %8.1e  %8.1e\n", last.iter, (double)last.rNorm, (double)last.pAp, (double)last.alpha);
      if (o.callback) {
        // the callback may read ws.x / ws.r: the stream is idle here, data is current
        ws.stats.niter = last.iter;
        user_exit = o.callback(&ws, o.callback_user) != 0;
      }
      overtimed = (now_seconds() - start_time) > o.timemax;
      agree_exit(ws, o, user_exit, overtimed);      // row-partitioned: same decision on every rank
      if (user_exit || overtimed) break;
      enqueue(cur);
    } else {
      cur ^= 1;
    }
  }
  c.sync();   // drain speculative no-op launches
  if (o.time_kernels && persist) {
    // phase durations measured inside the kernel (%globaltimer of CTA 0, barriers included)
    GridBar hb;
    KB_CUDA(cudaMemcpy(&hb, gbar, sizeof(hb), cudaMemcpyDeviceToHost));
    ws.timed_pairs = (int)hb.timed_iters;
    ws.k1_ms = hb.timed_iters ? 1e-6 * (double)hb.ns_a / hb.timed_iters : 0;
    ws.k2_ms = hb.timed_iters ? 1e-6 * (double)hb.ns_b / hb.timed_iters : 0;
    for (auto& e : tev) cudaEventDestroy(e);
  } else if (o.time_kernels) {
    const int pairs = std::min(kTimedCount, std::max(0, std::min(enq, last.iter) - kTimedFirst));
    double s1 = 0, s2 = 0;
    for (int i = 0; i < pairs; i++) {
      float a = 0, b = 0;
      cudaEventElapsedTime(&a, tev[3 * i], tev[3 * i + 1]);
      cudaEventElapsedTime(&b, tev[3 * i + 1], tev[3 * i + 2]);
      s1 += a; s2 += b;
    }
    ws.timed_pairs = pairs;
    ws.k1_ms = pairs ? s1 / pairs : 0;
    ws.k2_ms = pairs ? s2 / pairs : 0;
    for (auto& e : tev) cudaEventDestroy(e);
  }
  if (last.comm_error) throw std::runtime_error("cross-GPU all-reduce timed out: a peer rank is not participating");
  if (last.not_spd) throw std::runtime_error("The linear operator `A` or the preconditioner `M` is not symmetric positive definite.");

  iter = last.iter;
  solved = last.solved != 0;
  tired = last.tired != 0;
  zero_curvature = last.zero_curvature != 0;
  inconsistent = last.inconsistent != 0;
  // Which buffer holds the current direction?  K1 of iteration k writes P[(k+1)&1].
  // Normal exit after K2 of iteration iter-1: p = P[iter & 1].  Exit from K1's
  // curvature test at iteration `iter` (iter not incremented): p = P[(iter+1) & 1].
  const bool k1_exit = zero_curvature || last.npc;
  T* pcur = k1_exit ? P[(iter + 1) & 1] : P[iter & 1];
  if (pcur != ws.p) { T* tmp = ws.p; ws.p = ws.p2; ws.p2 = tmp; ws.dist.swapped = !ws.dist.swapped; }
  // XUP: the x update of the last completed iteration has not been applied yet (the K1 that would have done it
  // saw `done`).  A K1 exit applied its predecessor's update during its own pass, so nothing is pending then.
  if (xup && !k1_exit && iter > 0) k_axpy<T>(c, n, last.alpha, ws.p, ws.x);
  if (last.npc) {                                   // linesearch branch, cg.jl:203-209
    if (iter == 0) k_copy<T>(c, n, ws.x, ws.p);
    k_copy<T>(c, n, ws.npc_dir, ws.p);
    ws.stats.npcCount = 1;
    ws.stats.indefinite = true;
  }
}

#define INST(T)                                                                                              \
  template bool cg_fused_eligible<T>(const LinOp<T>&, const LinOp<T>&, const SolveOpts&);                    \
  template void cg_fused_prepare<T>(Workspace<T>&);                                                          \
  template void cg_dist_push_r<T>(Workspace<T>&);                                                            \
  template void cg_fused_loop<T>(Workspace<T>&, const Csr<T>&, const SolveOpts&, T, T, int, double, bool&, bool&, \
                                 bool&, bool&, bool&, bool&, int&);
INST(double)
INST(float)
#undef INST

}  // namespace kb
