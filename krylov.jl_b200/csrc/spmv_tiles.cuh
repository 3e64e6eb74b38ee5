// spmv_tiles.cuh -- TMA-staged CSR row-tile pipeline (sm_100a).
//
// A persistent CTA walks tiles of kTileRows consecutive rows.  One producer
// warp streams each tile's row-pointer slice, column indices and values from
// HBM into a shared-memory ring with 1-D bulk TMA copies (cp.async.bulk ->
// SASS UBLKCP) that complete on an mbarrier; eight consumer warps wait on the
// barrier and reduce one row per thread from shared memory, gathering x
// through the read-only L1/L2 path.  Consumers hand the stage back through a
// second mbarrier.  The matrix (>= 80 % of the bytes of an SpMV) therefore
// moves as large asynchronous bursts with several KB in flight per SM and no
// register staging, while the irregular x gather stays on LDG.
// DICT = true (operators with a dictionary, Csr::code): the stage carries one code byte per nonzero instead of the
// values and column indices; column and value are looked up in the dictionary each CTA keeps in shared memory.
//
// Row sums accumulate left to right in ascending column order with the product
// rounded before the add -- the order SparseArrays' CSC mul! produces for every
// y[i] -- so y is bit-identical to the sequential CPU oracle.  (The gathers of
// up to kGatherDepth nonzeros are ISSUED together to overlap their latencies;
// the additions are still performed in column order.)
#pragma once
#include "common.cuh"
#include "kb_internal.h"

namespace kb {

constexpr int kConsumerWarps = kTileRows / 32;            // 8
constexpr int kTileThreads = kTileRows + 32;              // + 1 producer warp
constexpr int kGatherDepth = 8;                           // gathers in flight per thread
#ifndef KB_CLAMP_GATHER
#define KB_CLAMP_GATHER 1                                 // 0: guarded gathers of round 1 (A/B builds)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
  unsigned ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
// 1-D bulk TMA copy global -> shared, completion counted in bytes on `bar`.
// The matrix streams are read once per SpMV: tag them evict-first in L2 so the
// gathered vectors (re-read by neighbouring rows) keep their lines.
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, unsigned bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
// x gather (y = A x) through the read-only path, single GPU.  The kernels are compiled once per gather type:
// the pointer select of the row-partitioned variant below costs the single-GPU fused phases 6-17 % when it is
// only disabled at run time (profiles/README.md), so it is a compile-time choice like the CG kernels' MODE.
template <class T>
struct XPlain {
  const T* __restrict__ x;
  __device__ __forceinline__ T operator()(int j) const { return __ldg(&x[j]); }
};

// Row-partitioned operators: column j >= nloc is halo entry j - nloc of the local halo buffer (filled by
// k_halo_exchange); the source is chosen by a pointer select, not a branch, so the batch of gathers stays a
// straight line of loads.
template <class T>
struct XGather {
  const T* x;
  const T* xh_minus_nloc;   // halo buffer base shifted by -nloc (only dereferenced for j >= nloc)
  int nloc;
  __device__ __forceinline__ T operator()(int j) const {
    const T* base = j < nloc ? x : xh_minus_nloc;
    return __ldg(&base[j]);
  }
};

// The gather for vector x under context c (host side).
template <class T>
inline XGather<T> xgather_of(const Ctx& c, const T* x) {
  if (!c.dex) return XGather<T>{x, x, 2147483647};
  const DistExchange& d = *c.dex;
  const T* section = reinterpret_cast<const T*>(d.xhalo) + (size_t)((d.count + 1) & 1) * (size_t)d.nhalo;   // parity of the LAST exchange
  return XGather<T>{x, section - d.nloc, d.nloc};
}

__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// Shared-memory layout (all offsets multiples of 128 B): 128 B of mbarriers, the dictionary (DICT only), then the
// ring.  A CSR stage holds the tile's rowptr slice, values and column indices; a DICT stage the rowptr slice and
// one code byte per nonzero (about 3 KB instead of 23 KB for a 7-point stencil).
template <class T, bool DICT = false>
struct TileLayout {
  int cap;  // max nnz per tile
  __host__ __device__ static constexpr size_t align_up(size_t v) { return (v + 127) & ~size_t(127); }
  __host__ __device__ size_t rp_bytes() const { return align_up((kTileRows + 4) * sizeof(int)); }
  __host__ __device__ size_t val_bytes() const { return align_up((size_t)(cap + 16 / sizeof(T)) * sizeof(T)); }
  __host__ __device__ size_t col_bytes() const { return align_up((size_t)(cap + 8) * sizeof(int)); }
  __host__ __device__ size_t code_bytes() const { return align_up((size_t)cap + 32); }
  __host__ __device__ static constexpr size_t dict_bytes() { return DICT ? (size_t)kDictMax * (sizeof(int) + sizeof(T)) : 0; }
  __host__ __device__ size_t stage_bytes() const { return rp_bytes() + (DICT ? code_bytes() : val_bytes() + col_bytes()); }
  __host__ __device__ static constexpr size_t ring_offset() { return 128 + dict_bytes(); }
  __host__ __device__ size_t total_bytes(int stages) const { return ring_offset() + (size_t)stages * stage_bytes(); }
};

// Stage of tile t (nonzeros [k0, k1)) into ring slot `st`: the rowptr slice plus either the values and column
// indices (CSR) or the code bytes (DICT), completing on `bar`.  Bulk copies move multiples of 16 B from 16-B aligned
// addresses: the ranges are widened to that grain (the arrays are padded) and the consumers offset into them.
template <class T, bool DICT>
__device__ __forceinline__ void tile_stage_issue(const Csr<T>& A, const TileLayout<T, DICT>& L, unsigned char* st, uint64_t* bar,
                                                 int t, int k0, int k1, uint64_t pol) {
  const unsigned rp_b = (kTileRows + 4) * sizeof(int);
  if constexpr (DICT) {
    const int k0b = k0 & ~15, k1b = (k1 + 15) & ~15;
    const unsigned c_b = (unsigned)(k1b - k0b);
    mbar_expect_tx(bar, rp_b + c_b);
    tma_load_1d(st, A.rowptr + t * kTileRows, rp_b, bar, pol);
    if (c_b) tma_load_1d(st + L.rp_bytes(), A.code + k0b, c_b, bar, pol);
  } else {
    constexpr int VA = 16 / sizeof(T);
    const int k0v = k0 & ~(VA - 1), k1v = (k1 + VA - 1) & ~(VA - 1);
    const int k0c = k0 & ~3, k1c = (k1 + 3) & ~3;
    const unsigned v_b = (unsigned)(k1v - k0v) * sizeof(T);
    const unsigned c_b = (unsigned)(k1c - k0c) * sizeof(int);
    mbar_expect_tx(bar, rp_b + v_b + c_b);
    tma_load_1d(st, A.rowptr + t * kTileRows, rp_b, bar, pol);
    if (v_b) tma_load_1d(st + L.rp_bytes(), A.val + k0v, v_b, bar, pol);
    if (c_b) tma_load_1d(st + L.rp_bytes() + L.val_bytes(), A.colind + k0c, c_b, bar, pol);
  }
}

// DICT: copy the operator's dictionary into shared memory (every thread of the CTA; publish with a barrier).
template <class T>
__device__ __forceinline__ void dict_to_smem(const Csr<T>& A, unsigned char* smem) {
  constexpr int words = (int)(TileLayout<T, true>::dict_bytes() / sizeof(uint4));
  const uint4* src = reinterpret_cast<const uint4*>(A.dict);
  uint4* dst = reinterpret_cast<uint4*>(smem + 128);
  for (int i = threadIdx.x; i < words; i += blockDim.x) dst[i] = __ldg(&src[i]);
}

// DICT: sum of one row whose nonzeros are codes crow[kb .. ke) into the dictionary (doff, dval) in shared memory.
// Column = row + offset: all DEPTH gathers of a batch are issued (clamped indices, as in the CSR consumers) before
// the values are looked up, and the products are added left to right with the same roundings as the CSR path, so
// the row sum is bit-identical to it.
template <class T, int DEPTH, class Gather>
__device__ __forceinline__ T dict_row_sum(const uint8_t* crow, const int* doff, const T* dval, int row, int kb, int ke,
                                          Gather gather) {
  T acc = T(0);
  for (int k = kb; k < ke; k += DEPTH) {
    T xv[DEPTH];
#pragma unroll
    for (int u = 0; u < DEPTH; u++) xv[u] = gather(row + doff[crow[min(k + u, ke - 1)]]);
    asm volatile("" ::: "memory");        // keep the gathers above the value look-ups
#pragma unroll
    for (int u = 0; u < DEPTH; u++) {
      const T nx = add_rn(acc, mul_rn(dval[crow[min(k + u, ke - 1)]], xv[u]));
      acc = (k + u < ke) ? nx : acc;
    }
  }
  return acc;
}

struct NoRowBegin {
  __device__ __forceinline__ int operator()(int) const { return 0; }
};

// The producer of the tile pipeline (one elected lane): for every tile of this CTA, wait for a free ring slot and
// issue the bulk copies of its stage, which complete on the slot's `full` barrier.
template <class T, bool DICT = false>
__device__ __forceinline__ void tile_producer(const Csr<T>& A, const TileLayout<T, DICT>& L, int S, unsigned char* ring, uint64_t* full,
                                              uint64_t* empty) {
  const uint64_t pol = l2_evict_first_policy();
  int it = 0;
  int t = blockIdx.x;
  int k0 = 0, k1 = 0;
  if (t < A.ntiles) { k0 = __ldg(&A.rowptr[t * kTileRows]); k1 = __ldg(&A.rowptr[min(t * kTileRows + kTileRows, A.n)]); }
  for (; t < A.ntiles; t += gridDim.x, it++) {
    // start fetching the NEXT tile's nnz range before blocking on the ring slot
    const int tn = t + gridDim.x;
    int nk0 = 0, nk1 = 0;
    if (tn < A.ntiles) { nk0 = __ldg(&A.rowptr[tn * kTileRows]); nk1 = __ldg(&A.rowptr[min(tn * kTileRows + kTileRows, A.n)]); }
    const int s = it % S;
    mbar_wait(&empty[s], ((it / S) & 1) ^ 1);
    tile_stage_issue<T, DICT>(A, L, ring + (size_t)s * L.stage_bytes(), &full[s], t, k0, k1, pol);
    k0 = nk0; k1 = nk1;
  }
}

// Runs the tile pipeline.  Every thread of the CTA must call it (blockDim.x ==
// kTileThreads).  `gather(j)` returns the x value for column j; `row_begin(row)`
// is evaluated before the row's gathers (use it to start loads the epilogue
// needs) and its result is handed to `row_done(row, acc, pre)` with the
// finished row sum (consumer threads only, row < n).  DICT: stream the operator's code bytes (A.ndict > 0).
template <class T, bool DICT = false, class Gather, class RowBegin, class RowDone>
__device__ __forceinline__ void spmv_tiles_run(const Csr<T>& A, unsigned char* smem, Gather gather, RowBegin row_begin,
                                               RowDone row_done) {
  const TileLayout<T, DICT> L{A.tile_cap};
  const int S = DICT ? A.dict_stages : A.stages;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);        // [S]
  uint64_t* empty = full + S;                                // [S]   (S <= 8 -> 128 B header)
  unsigned char* ring = smem + L.ring_offset();
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int VA = 16 / sizeof(T);                         // values per 16 B

  if (DICT) dict_to_smem<T>(A, smem);
  if (tid == 0) {
    for (int s = 0; s < S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumerWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == kConsumerWarps) {
    // ------------------------------ producer ------------------------------
    // (Tried and removed, profiles/r1_sweep_k1.txt + r1_ab.txt: letting the whole producer warp walk the column
    //  indices of the queued tile and prefetch its x entries into L2 -- no gain at 3 stages, and the extra live
    //  state cost the kernel its 3-CTAs/SM register budget: 335 vs 299 us per iteration on the same GPU.)
    if (lane == 0) tile_producer<T, DICT>(A, L, S, ring, full, empty);
  } else {
    // ------------------------------ consumers -----------------------------
    int it = 0;
    for (int t = blockIdx.x; t < A.ntiles; t += gridDim.x, it++) {
      const int row = t * kTileRows + tid;
      auto pre = row_begin(row < A.n ? row : 0);               // independent of the tile: issue before waiting
      const int s = it % S;
      mbar_wait(&full[s], (it / S) & 1);
      const unsigned char* st = ring + (size_t)s * L.stage_bytes();
      const int* rp = reinterpret_cast<const int*>(st);
      if (DICT && row < A.n) {
        const uint8_t* crow = reinterpret_cast<const uint8_t*>(st + L.rp_bytes()) - (rp[0] & ~15);
        const int* doff = reinterpret_cast<const int*>(smem + 128);
        const T* dval = reinterpret_cast<const T*>(doff + kDictMax);
        row_done(row, dict_row_sum<T, kGatherDepth>(crow, doff, dval, row, rp[tid], rp[tid + 1], gather), pre);
      } else if (row < A.n) {
        const T* vs = reinterpret_cast<const T*>(st + L.rp_bytes());
        const int* cs = reinterpret_cast<const int*>(st + L.rp_bytes() + L.val_bytes());
        const int k0 = rp[0];
        const T* vrow = vs - (k0 & ~(VA - 1));
        const int* crow = cs - (k0 & ~3);
        const int kb = rp[tid], ke = rp[tid + 1];
        T acc = T(0);
        for (int k = kb; k < ke; k += kGatherDepth) {
          T xv[kGatherDepth], av[kGatherDepth];
#if KB_CLAMP_GATHER
          // clamped indices + selected sums: straight-line code, every gather of the batch is issued before the
          // first use (guarded loads compile to load -> use -> load chains: 2-3 loads in flight instead of 8)
#pragma unroll
          for (int u = 0; u < kGatherDepth; u++) {
            const int kk = min(k + u, ke - 1);
            av[u] = vrow[kk];
            xv[u] = gather(crow[kk]);
          }
          asm volatile("" ::: "memory");      // keep the loads above the sums (the optimiser would sink them)
#pragma unroll
          for (int u = 0; u < kGatherDepth; u++) {
            const T nx = add_rn(acc, mul_rn(av[u], xv[u]));
            acc = (k + u < ke) ? nx : acc;
          }
#else
#pragma unroll
          for (int u = 0; u < kGatherDepth; u++) {
            if (k + u < ke) { av[u] = vrow[k + u]; xv[u] = gather(crow[k + u]); }
          }
#pragma unroll
          for (int u = 0; u < kGatherDepth; u++) {
            if (k + u < ke) acc = add_rn(acc, mul_rn(av[u], xv[u]));
          }
#endif
        }
        row_done(row, acc, pre);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
    }
  }
}


// ---------------------------------------------------------------------------
// The same pipeline split into pieces for PERSISTENT kernels (cg_fused.cu: cg_persist) that run the tile pass
// many times inside one launch.  Ring positions are running counters (slot = pos % S, phase = (pos / S) & 1) that
// survive from one pass to the next, so the producer may already stream the first tiles of the NEXT pass (the
// matrix does not change between iterations) while the consumers sit in a grid-wide barrier.
// `tile_at(j)` maps the j-th tile of this CTA's sequence to a tile id; bit 31 set marks a tile whose gathers
// need data that `pre_tile()` must wait for (row-partitioned solves: halo columns).
// ---------------------------------------------------------------------------
template <class T, bool DICT = false>
struct TilePipe {
  TileLayout<T, DICT> L;
  int S;
  uint64_t* full;
  uint64_t* empty;
  unsigned char* ring;
  const int* doff;          // DICT: the dictionary in shared memory
  const T* dval;
  __device__ __forceinline__ void init(const Csr<T>& A, unsigned char* smem) {   // every thread of the CTA
    L = TileLayout<T, DICT>{A.tile_cap};
    S = DICT ? A.dict_stages : A.stages;
    full = reinterpret_cast<uint64_t*>(smem);
    empty = full + S;
    ring = smem + L.ring_offset();
    doff = reinterpret_cast<const int*>(smem + 128);
    dval = reinterpret_cast<const T*>(doff + kDictMax);
    if (DICT) dict_to_smem<T>(A, smem);
    if (threadIdx.x == 0) {
      for (int s = 0; s < S; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], kConsumerWarps); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
};

// Producer (one elected lane): issue ring positions [pos, target).  Position q carries tile tile_at(q % cnt).
template <class T, bool DICT, class TileAt>
__device__ __forceinline__ void tile_issue_until(const Csr<T>& A, const TilePipe<T, DICT>& P, unsigned& pos, unsigned target, int cnt,
                                                 TileAt tile_at, uint64_t pol) {
  if (pos >= target) return;
  int t = tile_at((int)(pos % (unsigned)cnt)) & 0x7fffffff;
  int k0 = __ldg(&A.rowptr[t * kTileRows]), k1 = __ldg(&A.rowptr[min(t * kTileRows + kTileRows, A.n)]);
  for (; pos < target; pos++) {
    int tn = 0, nk0 = 0, nk1 = 0;
    if (pos + 1 < target) {        // next tile's nnz range: fetch before blocking on the ring slot
      tn = tile_at((int)((pos + 1) % (unsigned)cnt)) & 0x7fffffff;
      nk0 = __ldg(&A.rowptr[tn * kTileRows]); nk1 = __ldg(&A.rowptr[min(tn * kTileRows + kTileRows, A.n)]);
    }
    const int s = (int)(pos % (unsigned)P.S);
    mbar_wait(&P.empty[s], ((pos / (unsigned)P.S) & 1) ^ 1);
    tile_stage_issue<T, DICT>(A, P.L, P.ring + (size_t)s * P.L.stage_bytes(), &P.full[s], t, k0, k1, pol);
    t = tn; k0 = nk0; k1 = nk1;
  }
}

// Producer at kernel exit: positions [consumed, pos) were issued but never consumed -- wait for their copies to
// land (a CTA must not retire with bulk copies in flight into its shared memory).
template <class T, bool DICT>
__device__ __forceinline__ void tile_drain(const TilePipe<T, DICT>& P, unsigned consumed, unsigned pos) {
  for (unsigned q = consumed; q < pos; q++) mbar_wait(&P.full[q % (unsigned)P.S], (q / (unsigned)P.S) & 1);
}

// Consumers (threads 0 .. kTileRows-1): tiles j0 <= j < j1 of this CTA's sequence (a pass is one call with
// [0, cnt), or two calls when something must happen between the interior tiles and the halo tiles).
template <class T, int DEPTH, bool DICT, class TileAt, class Gather, class RowBegin, class RowDone>
__device__ __forceinline__ void tile_consume_pass(const Csr<T>& A, const TilePipe<T, DICT>& P, unsigned& cpos, int j0, int j1, TileAt tile_at,
                                                  Gather gather, RowBegin row_begin, RowDone row_done) {
  constexpr int VA = 16 / sizeof(T);
  const int tid = threadIdx.x, lane = tid & 31;
  for (int j = j0; j < j1; j++, cpos++) {
    const int t = tile_at(j) & 0x7fffffff;
    const int row = t * kTileRows + tid;
    auto pre = row_begin(row < A.n ? row : 0);
    const int s = (int)(cpos % (unsigned)P.S);
    mbar_wait(&P.full[s], (cpos / (unsigned)P.S) & 1);
    const unsigned char* st = P.ring + (size_t)s * P.L.stage_bytes();
    const int* rp = reinterpret_cast<const int*>(st);
    if (DICT && row < A.n) {
      const uint8_t* crow = reinterpret_cast<const uint8_t*>(st + P.L.rp_bytes()) - (rp[0] & ~15);
      row_done(row, dict_row_sum<T, DEPTH>(crow, P.doff, P.dval, row, rp[tid], rp[tid + 1], gather), pre);
    } else if (row < A.n) {
      const T* vs = reinterpret_cast<const T*>(st + P.L.rp_bytes());
      const int* cs = reinterpret_cast<const int*>(st + P.L.rp_bytes() + P.L.val_bytes());
      const int k0 = rp[0];
      const T* vrow = vs - (k0 & ~(VA - 1));
      const int* crow = cs - (k0 & ~3);
      const int kb = rp[tid], ke = rp[tid + 1];
      T acc = T(0);
      // The gathers here are plain (coherent) loads, which the compiler will not speculate: guarded loads would
      // be chained load -> use -> load.  Clamp the index instead (every address is valid) and select the sum, so
      // the batch is straight-line code and all gathers of a row are issued together.
      for (int k = kb; k < ke; k += DEPTH) {
        T xv[DEPTH], av[DEPTH];
#pragma unroll
        for (int u = 0; u < DEPTH; u++) xv[u] = gather(crow[min(k + u, ke - 1)]);
        asm volatile("" ::: "memory");        // keep the gathers above everything else (the optimiser would sink them)
        // the matrix values come from shared memory (short latency): fetch them only now, so that the registers
        // of the batch hold gathered data instead -- at 72 registers per thread that is the difference between
        // 2 and 8 global loads in flight
#pragma unroll
        for (int u = 0; u < DEPTH; u++) av[u] = vrow[min(k + u, ke - 1)];
#pragma unroll
        for (int u = 0; u < DEPTH; u++) {
          const T nx = add_rn(acc, mul_rn(av[u], xv[u]));
          acc = (k + u < ke) ? nx : acc;
        }
      }
      row_done(row, acc, pre);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&P.empty[s]);
  }
}

}  // namespace kb
