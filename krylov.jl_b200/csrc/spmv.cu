// spmv.cu -- the CSR operator: upload/normalisation, staging plan, and the
// y = A x kernels that stand in for `kmul!(y, A, x)` = mul!(y, A, x)
// (src/krylov_utils.jl:305; call sites cg.jl:196, gmres.jl:257,
// bicgstab.jl:221,228, minres.jl:289).
#include "kb_internal.h"
#include "spmv_tiles.cuh"

#include <algorithm>
#include <type_traits>
#include <vector>

namespace kb {

// ---------------------------------------------------------------------------
// Upload: accept the caller's (rowptr, colind, val) with 0/1-based, 32/64-bit
// indices on host or device; store int32 0-based in padded device arrays.
// The bijection (shift by index_base, narrow to int32) keeps every
// (row, col, val) triplet of the input -- "bit-exact integer indexing".
// ---------------------------------------------------------------------------
template <class I>
__global__ void index_convert_kernel(long long cnt, const I* __restrict__ in, int* __restrict__ out, int base, int* bad) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < cnt; i += stride) {
    long long v = (long long)in[i] - base;
    if (v < 0 || v > 2147483647LL) atomicExch(bad, 1);
    out[i] = (int)v;
  }
}

__global__ void fill_int_kernel(int cnt, int* out, int v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cnt) out[i] = v;
}

template <class T>
void csr_upload(Ctx& c, Csr<T>& A, int n, long long nnz, const void* rowptr, const void* colind, const T* val,
                int index_base, int index_bytes, bool on_device) {
  if (n < 0 || nnz < 0 || nnz > 2147483647LL - 64) throw std::runtime_error("CSR operator: n/nnz out of int32 range");
  if (index_bytes != 4 && index_bytes != 8) throw std::runtime_error("CSR operator: index_bytes must be 4 or 8");
  if (index_base != 0 && index_base != 1) throw std::runtime_error("CSR operator: index_base must be 0 or 1");
  csr_free(A);
  A.n = n; A.nnz = nnz;
  const size_t rp_len = (size_t)n + 1, rp_pad = kTileRows + 16;
  A.rowptr = dev_alloc<int>(rp_len + rp_pad);
  A.colind = dev_alloc<int>((size_t)nnz + 16);
  A.val = dev_alloc<T>((size_t)nnz + 16);
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  KB_CUDA(cudaMemcpyAsync(A.val, val, sizeof(T) * (size_t)nnz, kind, c.stream));
  KB_CUDA(cudaMemsetAsync(A.val + nnz, 0, sizeof(T) * 16, c.stream));
  KB_CUDA(cudaMemsetAsync(A.colind + nnz, 0, sizeof(int) * 16, c.stream));
  int* bad = nullptr;
  KB_CUDA(cudaMalloc((void**)&bad, sizeof(int)));
  KB_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), c.stream));
  void* tmp_rp = nullptr; void* tmp_ci = nullptr;
  if (index_bytes == 4 && index_base == 0) {
    KB_CUDA(cudaMemcpyAsync(A.rowptr, rowptr, sizeof(int) * rp_len, kind, c.stream));
    KB_CUDA(cudaMemcpyAsync(A.colind, colind, sizeof(int) * (size_t)nnz, kind, c.stream));
  } else {
    const void* drp = rowptr; const void* dci = colind;
    if (!on_device) {
      KB_CUDA(cudaMalloc(&tmp_rp, (size_t)index_bytes * rp_len));
      KB_CUDA(cudaMalloc(&tmp_ci, (size_t)index_bytes * (size_t)(nnz ? nnz : 1)));
      KB_CUDA(cudaMemcpyAsync(tmp_rp, rowptr, (size_t)index_bytes * rp_len, cudaMemcpyHostToDevice, c.stream));
      KB_CUDA(cudaMemcpyAsync(tmp_ci, colind, (size_t)index_bytes * (size_t)nnz, cudaMemcpyHostToDevice, c.stream));
      drp = tmp_rp; dci = tmp_ci;
    }
    const int g = sm_count() * 8;
    if (index_bytes == 8) {
      index_convert_kernel<long long><<<g, 256, 0, c.stream>>>((long long)rp_len, (const long long*)drp, A.rowptr, index_base, bad);
      index_convert_kernel<long long><<<g, 256, 0, c.stream>>>(nnz, (const long long*)dci, A.colind, index_base, bad);
    } else {
      index_convert_kernel<int><<<g, 256, 0, c.stream>>>((long long)rp_len, (const int*)drp, A.rowptr, index_base, bad);
      index_convert_kernel<int><<<g, 256, 0, c.stream>>>(nnz, (const int*)dci, A.colind, index_base, bad);
    }
    KB_CUDA(cudaGetLastError());
  }
  // rows past n (read by the last tile's row-pointer slice) are empty
  fill_int_kernel<<<((int)rp_pad + 255) / 256, 256, 0, c.stream>>>((int)rp_pad, A.rowptr + rp_len, (int)nnz);
  KB_CUDA(cudaGetLastError());
  int hbad = 0;
  KB_CUDA(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  c.sync();
  cudaFree(bad);
  if (tmp_rp) cudaFree(tmp_rp);
  if (tmp_ci) cudaFree(tmp_ci);
  if (hbad) { csr_free(A); throw std::runtime_error("CSR operator: index outside int32 range after rebasing"); }
  try { csr_plan(c, A); } catch (...) { csr_free(A); throw; }
}

template <class T> void csr_free(Csr<T>& A) {
  dev_free(A.rowptr); dev_free(A.colind); dev_free(A.val); dev_free(A.code); dev_free(A.dict);
  A = Csr<T>();
}

// ---------------------------------------------------------------------------
// Staging plan: largest tile (nnz of kTileRows consecutive rows) and longest
// row decide whether the TMA ring fits, how deep it is, and the grid.
// ---------------------------------------------------------------------------
__global__ void plan_kernel(int n, int ntiles, const int* __restrict__ rowptr,
                            int* out /* [0]=tile_cap [1]=max_row [2]=unsorted [3]=rowptr not monotone [4]=max col [5]=negative col */,
                            const int* __restrict__ colind, long long nnz) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int stride = gridDim.x * blockDim.x;
  int cap = 0, mr = 0, uns = 0, bad = 0, mc = -1, neg = 0;
  for (int i = t; i < n; i += stride) {
    const int kb = rowptr[i], ke = rowptr[i + 1];
    // validation (a malformed matrix must be an error, not an out-of-bounds read in the SpMV): row pointers
    // non-decreasing and inside [0, nnz] -- only then are the column indices of the row looked at
    if (kb > ke || kb < 0 || (long long)ke > nnz) { bad = 1; continue; }
    mr = max(mr, ke - kb);
    for (int k = kb; k < ke; k++) { const int cj = colind[k]; mc = max(mc, cj); neg |= cj < 0; }
    // halo columns (index >= n, row-partitioned operators) keep their global position in the row: skip them
    for (int k = kb + 1; k < ke; k++) uns |= (colind[k] <= colind[k - 1]) && colind[k] < n && colind[k - 1] < n;
  }
  if (bad) atomicExch(&out[3], 1);
  __syncthreads();
  for (int i = t; i < ntiles; i += stride) {
    const int r0 = i * kTileRows, r1 = min(r0 + kTileRows, n);
    cap = max(cap, rowptr[r1] - rowptr[r0]);
  }
  atomicMax(&out[0], cap);
  atomicMax(&out[1], mr);
  atomicMax(&out[4], mc);
  if (uns) atomicExch(&out[2], 1);
  if (neg) atomicExch(&out[5], 1);
}

// ---------------------------------------------------------------------------
// Dictionary encoding: every nonzero k of row i is the pair (colind[k] - i, bit pattern of val[k]).  Operators with at
// most kDictMax distinct pairs (stencils, structured grids) are stored once more as one code byte per nonzero; the
// values are compared by bit pattern, so 0.0 / -0.0 stay distinct and decoding is exact.
//   pass 1 (dict_collect_kernel): each warp keeps a table of the pairs it has seen (de-duplicated with
//           __match_any_sync), the warps of a CTA merge theirs, dict_merge_kernel merges the CTAs' tables.  Any table
//           outgrowing kDictMax raises `overflow`, which every warp polls: a general matrix is rejected after a
//           fraction of one pass.
//   host:   sort the pairs by (offset, bits) -- code numbering independent of the scheduling, encoding deterministic.
//   pass 2 (dict_encode_kernel): binary search of each pair in the sorted table.
// ---------------------------------------------------------------------------
template <class T> using DictBits = typename std::conditional<sizeof(T) == 8, unsigned long long, unsigned>::type;
__device__ __forceinline__ unsigned long long dict_bits(double v) { return (unsigned long long)__double_as_longlong(v); }
__device__ __forceinline__ unsigned dict_bits(float v) { return __float_as_uint(v); }

// Lanes with `have` add (off, bits) to the warp's table [0, cnt) unless it is there.  Returns the new count (warp-
// uniform); entries past kDictMax are counted but not stored.
template <class B>
__device__ __forceinline__ int dict_warp_insert(int* toff, B* tbits, int cnt, bool have, int off, B bits) {
  const int lane = threadIdx.x & 31;
  bool need = have;
  for (int e = 0; need && e < cnt; e++) need = !(toff[e] == off && tbits[e] == bits);
  const unsigned needm = __ballot_sync(0xffffffffu, need);
  if (!needm) return cnt;
  const unsigned same = __match_any_sync(0xffffffffu, off) & __match_any_sync(0xffffffffu, bits) & needm;
  const bool lead = need && (__ffs(same) - 1 == lane);
  const unsigned leads = __ballot_sync(0xffffffffu, lead);
  const int slot = cnt + __popc(leads & ((1u << lane) - 1u));
  if (lead && slot < kDictMax) { toff[slot] = off; tbits[slot] = bits; }
  __syncwarp();
  return cnt + __popc(leads);
}

constexpr int kDictWarps = 8;

template <class T>
__global__ void __launch_bounds__(kDictWarps * 32) dict_collect_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ colind,
                                                                     const T* __restrict__ val, int* cta_off, DictBits<T>* cta_bits,
                                                                     int* cta_cnt, int* overflow) {
  typedef DictBits<T> B;
  __shared__ int soff[kDictWarps][kDictMax];
  __shared__ B sbits[kDictWarps][kDictMax];
  __shared__ int scnt[kDictWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stride = gridDim.x * kDictWarps * 32;
  int cnt = 0;
  for (int base = (blockIdx.x * kDictWarps + warp) * 32; base < n && cnt <= kDictMax; base += stride) {
    if (__any_sync(0xffffffffu, *(volatile int*)overflow != 0)) break;     // another warp has already seen too many
    const int row = base + lane;
    int kb = 0, ke = 0;
    if (row < n) { kb = rowptr[row]; ke = rowptr[row + 1]; }
    const int len = __reduce_max_sync(0xffffffffu, (unsigned)(ke - kb));
    for (int j = 0; j < len && cnt <= kDictMax; j++) {
      const bool have = kb + j < ke;
      const int off = have ? colind[kb + j] - row : 0;
      const B bits = have ? dict_bits(val[kb + j]) : B(0);
      cnt = dict_warp_insert<B>(soff[warp], sbits[warp], cnt, have, off, bits);
    }
  }
  if (lane == 0) { scnt[warp] = cnt; if (cnt > kDictMax) atomicExch(overflow, 1); }
  __syncthreads();
  if (warp != 0) return;
  for (int w = 1; w < kDictWarps && cnt <= kDictMax; w++) {
    const int m = min(scnt[w], kDictMax);
    for (int e0 = 0; e0 < m && cnt <= kDictMax; e0 += 32) {
      const int e = e0 + lane;
      cnt = dict_warp_insert<B>(soff[0], sbits[0], cnt, e < m, e < m ? soff[w][e] : 0, e < m ? sbits[w][e] : B(0));
    }
  }
  if (cnt > kDictMax) { if (lane == 0) atomicExch(overflow, 1); }
  for (int e = lane; e < min(cnt, kDictMax); e += 32) {
    cta_off[blockIdx.x * kDictMax + e] = soff[0][e];
    cta_bits[blockIdx.x * kDictMax + e] = sbits[0][e];
  }
  if (lane == 0) cta_cnt[blockIdx.x] = cnt;
}

// One warp: merge the CTAs' tables into out_* ([0] of out_cnt: number of pairs, kDictMax + 1 when there are more).
template <class B>
__global__ void dict_merge_kernel(int ncta, const int* cta_off, const B* cta_bits, const int* cta_cnt, const int* overflow,
                                  int* out_off, B* out_bits, int* out_cnt) {
  __shared__ int soff[kDictMax];
  __shared__ B sbits[kDictMax];
  const int lane = threadIdx.x;
  int cnt = *(volatile const int*)overflow ? kDictMax + 1 : 0;
  for (int b = 0; b < ncta && cnt <= kDictMax; b++) {
    const int m = cta_cnt[b];
    for (int e0 = 0; e0 < m && cnt <= kDictMax; e0 += 32) {
      const int e = e0 + lane;
      const bool have = e < m;
      cnt = dict_warp_insert<B>(soff, sbits, cnt, have, have ? cta_off[b * kDictMax + e] : 0, have ? cta_bits[b * kDictMax + e] : B(0));
    }
  }
  for (int e = lane; e < min(cnt, kDictMax); e += 32) { out_off[e] = soff[e]; out_bits[e] = sbits[e]; }
  if (lane == 0) *out_cnt = min(cnt, kDictMax + 1);
}

// code[k] = position of nonzero k's pair in the sorted dictionary (kDictMax offsets, then kDictMax values).
template <class T>
__global__ void __launch_bounds__(kBlock) dict_encode_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ colind,
                                                            const T* __restrict__ val, const void* dict, int ndict,
                                                            uint8_t* __restrict__ code, int* missing) {
  typedef DictBits<T> B;
  __shared__ int soff[kDictMax];
  __shared__ B sbits[kDictMax];
  for (int e = threadIdx.x; e < ndict; e += blockDim.x) {
    soff[e] = reinterpret_cast<const int*>(dict)[e];
    sbits[e] = dict_bits(reinterpret_cast<const T*>(reinterpret_cast<const int*>(dict) + kDictMax)[e]);
  }
  __syncthreads();
  const int stride = gridDim.x * blockDim.x;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += stride) {
    const int ke = rowptr[row + 1];
    for (int k = rowptr[row]; k < ke; k++) {
      const int off = colind[k] - row;
      const B bits = dict_bits(val[k]);
      int lo = 0, hi = ndict;                 // first entry >= (off, bits)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (soff[mid] < off || (soff[mid] == off && sbits[mid] < bits)) lo = mid + 1;
        else hi = mid;
      }
      if (lo < ndict && soff[lo] == off && sbits[lo] == bits) code[k] = (uint8_t)lo;
      else atomicExch(missing, 1);
    }
  }
}

// Builds A.code / A.dict / A.ndict when the operator has at most kDictMax distinct pairs (else leaves ndict = 0).
template <class T> static void csr_dict_build(Ctx& c, Csr<T>& A) {
  typedef DictBits<T> B;
  const int ncta = sm_count() * 2;
  char* tmp = nullptr;
  const size_t tab = (size_t)ncta * kDictMax;
  const size_t bytes = tab * (sizeof(int) + sizeof(B)) + (size_t)ncta * sizeof(int) + kDictMax * (sizeof(int) + sizeof(B)) + 4 * sizeof(int);
  KB_CUDA(cudaMalloc((void**)&tmp, bytes));
  B* cta_bits = (B*)tmp;
  B* out_bits = cta_bits + tab;
  int* cta_off = (int*)(out_bits + kDictMax);
  int* out_off = cta_off + tab;
  int* cta_cnt = out_off + kDictMax;
  int* flags = cta_cnt + ncta;                 // [0] overflow  [1] pairs found  [2] pair missing from the table
  int h[3] = {0, 0, 0};
  std::vector<int> hoff(kDictMax);
  std::vector<B> hbits(kDictMax);
  try {
    KB_CUDA(cudaMemsetAsync(flags, 0, 4 * sizeof(int), c.stream));
    dict_collect_kernel<T><<<ncta, kDictWarps * 32, 0, c.stream>>>(A.n, A.rowptr, A.colind, A.val, cta_off, cta_bits, cta_cnt, flags);
    dict_merge_kernel<B><<<1, 32, 0, c.stream>>>(ncta, cta_off, cta_bits, cta_cnt, flags, out_off, out_bits, flags + 1);
    KB_CUDA(cudaGetLastError());
    KB_CUDA(cudaMemcpyAsync(h, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    KB_CUDA(cudaMemcpyAsync(hoff.data(), out_off, kDictMax * sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    KB_CUDA(cudaMemcpyAsync(hbits.data(), out_bits, kDictMax * sizeof(B), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    const int nd = h[1];
    if (nd >= 1 && nd <= kDictMax) {
      std::vector<std::pair<int, B>> pairs(nd);
      for (int e = 0; e < nd; e++) pairs[e] = {hoff[e], hbits[e]};
      std::sort(pairs.begin(), pairs.end());
      std::vector<char> hd(TileLayout<T, true>::dict_bytes(), 0);
      int* doff = (int*)hd.data();
      T* dval = (T*)(doff + kDictMax);
      for (int e = 0; e < nd; e++) { doff[e] = pairs[e].first; memcpy(&dval[e], &pairs[e].second, sizeof(T)); }
      A.dict = dev_alloc<char>(hd.size());
      A.code = reinterpret_cast<uint8_t*>(dev_alloc<char>((size_t)A.nnz + 64));       // the bulk copies read whole 16-B granules past nnz
      KB_CUDA(cudaMemcpyAsync(A.dict, hd.data(), hd.size(), cudaMemcpyHostToDevice, c.stream));
      KB_CUDA(cudaMemsetAsync(A.code + A.nnz, 0, 64, c.stream));
      dict_encode_kernel<T><<<sm_count() * 4, kBlock, 0, c.stream>>>(A.n, A.rowptr, A.colind, A.val, A.dict, nd, A.code, flags + 2);
      KB_CUDA(cudaGetLastError());
      KB_CUDA(cudaMemcpyAsync(&h[2], flags + 2, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
      c.sync();
      if (h[2]) throw std::runtime_error("CSR operator: dictionary encoding lost a (column offset, value) pair");
      A.ndict = nd;
    }
  } catch (...) {
    cudaFree(tmp);
    throw;
  }
  cudaFree(tmp);
}

template <class T> void csr_plan(Ctx& c, Csr<T>& A) {
  A.ntiles = (A.n + kTileRows - 1) / kTileRows;
  int* dout = nullptr;
  KB_CUDA(cudaMalloc((void**)&dout, 6 * sizeof(int)));
  KB_CUDA(cudaMemsetAsync(dout, 0, 6 * sizeof(int), c.stream));
  int h[6] = {0, 0, 0, 0, -1, 0};
  int ends[2] = {0, (int)A.nnz};
  if (A.n > 0) {
    KB_CUDA(cudaMemcpyAsync(dout + 4, &h[4], sizeof(int), cudaMemcpyHostToDevice, c.stream));
    plan_kernel<<<sm_count() * 4, 256, 0, c.stream>>>(A.n, A.ntiles, A.rowptr, dout, A.colind, A.nnz);
    KB_CUDA(cudaGetLastError());
    KB_CUDA(cudaMemcpyAsync(&ends[0], A.rowptr, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    KB_CUDA(cudaMemcpyAsync(&ends[1], A.rowptr + A.n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
  }
  KB_CUDA(cudaMemcpyAsync(h, dout, sizeof(h), cudaMemcpyDeviceToHost, c.stream));
  c.sync();
  cudaFree(dout);
  // the reference would throw a BoundsError on such input; here it must not reach the kernels
  if (ends[0] != 0 || (long long)ends[1] != A.nnz || h[3])
    throw std::runtime_error("CSR operator: row pointers must start at 0 (after rebasing), be non-decreasing and end at nnz");
  if (h[5]) throw std::runtime_error("CSR operator: negative column index (after rebasing)");
  A.max_col = h[4];
  if (h[2]) fprintf(stderr, "[krylov_b200] warning: CSR column indices are not strictly ascending within rows; "
                            "results remain correct but are no longer bit-comparable to SparseArrays' order\n");
  A.tile_cap = h[0];
  A.max_row = h[1];
  // Ring sizing: prefer 2 CTAs/SM (<= 110 KB each) with up to 4 stages; fall
  // back to 1 CTA/SM (<= 220 KB) with >= 2 stages; otherwise no TMA staging.
  TileLayout<T> L{A.tile_cap};
  const size_t two_cta = 110 * 1024, one_cta = 220 * 1024;
  A.tma_ok = false;
  int per_sm = 2;
  // tuning overrides (profiles/sweep_k1.py): KB200_STAGES, KB200_CTAS_PER_SM
  const char* es = getenv("KB200_STAGES");
  const char* ec = getenv("KB200_CTAS_PER_SM");
  if (es && ec) {
    const int s = atoi(es), cps = atoi(ec);
    if (s >= 1 && s <= 8 && cps >= 1 && cps <= 8 && L.total_bytes(s) * cps <= 226 * 1024) { A.tma_ok = true; A.stages = s; per_sm = cps; }
  }
  // default: 3 CTAs/SM x 2 stages when it fits.  Measured on cfg2 (profiles/r1_sweep_k1.txt): K1 = 219 us at
  // 2 stages x 3 CTAs, 227 us at 3x3, 284-298 us at any depth with 2 CTAs: the gather latency wants 27 warps/SM,
  // and a shallower ring leaves more of the 228 KB to L1 for the gathered vectors.
  if (!A.tma_ok && L.total_bytes(2) * 3 <= 226 * 1024) { A.tma_ok = true; A.stages = 2; per_sm = 3; }
  for (int s = 4; s >= 2 && !A.tma_ok; s--)
    if (L.total_bytes(s) <= two_cta) { A.tma_ok = true; A.stages = s; per_sm = 2; }
  for (int s = 4; s >= 2 && !A.tma_ok; s--)
    if (L.total_bytes(s) <= one_cta) { A.tma_ok = true; A.stages = s; per_sm = 1; }
  const bool default_plan = A.tma_ok && per_sm == 3 && !(es && ec);
  if (A.tma_ok) {
    A.smem_bytes = L.total_bytes(A.stages);
    int g = sm_count() * per_sm;
    A.grid = g < A.ntiles ? g : (A.ntiles > 0 ? A.ntiles : 1);
    A.ctas_per_sm = per_sm;
  } else {
    A.stages = 0; A.smem_bytes = 0; A.grid = 0;
  }
  // Dictionary codes for the default ring (3 CTAs/SM, the same grid: the encoded kernels reduce in the same order).
  // A stage shrinks from ~23 KB to ~3 KB (cfg2), so the encoded ring is 4 deep -- the producer runs further ahead
  // across the persistent kernel's grid barriers -- and what the CTAs leave of the 228 KB goes to L1 for the gathers.
  // KB200_CSR_DICT=0 keeps the CSR stream (A/B runs and tests on one build).
  const char* ed = getenv("KB200_CSR_DICT");
  if (default_plan && A.nnz > 0 && !(ed && atoi(ed) == 0)) {
    const TileLayout<T, true> Ld{A.tile_cap};
    for (int s = 4; s >= 2 && !A.dict_stages; s--)
      if (Ld.total_bytes(s) * 3 <= 226 * 1024) A.dict_stages = s;
    if (A.dict_stages) {
      csr_dict_build<T>(c, A);
      if (A.ndict) A.dict_smem_bytes = Ld.total_bytes(A.dict_stages);
      else A.dict_stages = 0;
    }
  }
}

// ---------------------------------------------------------------------------
// Kernels
// ---------------------------------------------------------------------------
// Row-per-thread LDG kernel: always valid (any row length), used when the
// staging plan does not fit and as an independent check of the staged kernel.
template <class T, bool DOT, class G>
__global__ void __launch_bounds__(kBlock) spmv_rows_kernel(Csr<T> A, G xg, T* __restrict__ y, T* part,
                                                           unsigned* ticket, T* out) {
  __shared__ T sm[32];
  T dacc = T(0);
  const int stride = gridDim.x * blockDim.x;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < A.n; row += stride) {
    const int kb = A.rowptr[row], ke = A.rowptr[row + 1];
    T acc = T(0);
    for (int k = kb; k < ke; k++) acc = add_rn(acc, mul_rn(A.val[k], xg(A.colind[k])));
    y[row] = acc;
    if (DOT) dacc += __ldg(&xg.x[row]) * acc;
  }
  if (DOT) {
    T mine[1] = {block_sum(dacc, sm)}, tot[1];
    if (grid_sum_last<T, 1>(mine, part, ticket, sm, tot) && threadIdx.x == 0) out[0] = tot[0];
  }
}

template <class T, bool DOT, class G, bool DICT>
__global__ void __launch_bounds__(kTileThreads, 3) spmv_tma_kernel(Csr<T> A, G xg, T* __restrict__ y, T* part,
                                                                unsigned* ticket, T* out) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ T sm[32];
  T dacc = T(0);
  spmv_tiles_run<T, DICT>(
      A, smem, xg, [&](int row) { return DOT ? __ldg(&xg.x[row]) : T(0); },
      [&](int row, T acc, T xr) {
        y[row] = acc;
        if (DOT) dacc += xr * acc;
      });
  if (DOT) {
    T mine[1] = {block_sum(dacc, sm)}, tot[1];
    if (grid_sum_last<T, 1>(mine, part, ticket, sm, tot) && threadIdx.x == 0) out[0] = tot[0];
  }
}

template <class T, bool DOT, class G>
static void spmv_launch_g(Ctx& c, const Csr<T>& A, G xg, T* y, int slot, int variant) {
  T* out = reinterpret_cast<T*>(reinterpret_cast<double*>(c.dscal) + slot);
  const bool staged = variant == 2 || (variant == 0 && A.tma_ok);
  if (staged) {
    if (!A.tma_ok) throw std::runtime_error("TMA-staged SpMV requested but the tile plan does not fit shared memory");
    // the dictionary-encoded stream when the operator has one (single GPU: the row-partitioned gather stays on CSR)
    auto kern = spmv_tma_kernel<T, DOT, G, false>;
    size_t smem = A.smem_bytes;
    if constexpr (std::is_same<G, XPlain<T>>::value) {
      if (A.ndict > 0) { kern = spmv_tma_kernel<T, DOT, G, true>; smem = A.dict_smem_bytes; }
    }
    ensure_dyn_smem((const void*)kern, 220 * 1024);
    int occ = 0;   // persistent grid = what is really co-resident (never more than one wave)
    KB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kTileThreads, smem));
    if (occ < 1) throw std::runtime_error("spmv_tma_kernel does not fit on an SM with the planned shared-memory ring");
    const int grid = std::min(std::min(occ, A.ctas_per_sm) * sm_count(), std::max(1, A.ntiles));
    kern<<<grid, kTileThreads, smem, c.stream>>>(A, xg, y, (T*)c.partials, c.tickets + 1, out);
  } else {
    const int grid = stream_grid(A.n, 1, 8);
    spmv_rows_kernel<T, DOT, G><<<grid, kBlock, 0, c.stream>>>(A, xg, y, (T*)c.partials, c.tickets + 1, out);
  }
  KB_CUDA(cudaGetLastError());
  c.launches++;
}

template <class T, bool DOT>
static void spmv_launch(Ctx& c, const Csr<T>& A, const T* x, T* y, int slot, int variant) {
  if (A.n <= 0) return;
  if (c.dex) spmv_launch_g<T, DOT, XGather<T>>(c, A, xgather_of<T>(c, x), y, slot, variant);   // row-partitioned: [local | halo]
  else spmv_launch_g<T, DOT, XPlain<T>>(c, A, XPlain<T>{x}, y, slot, variant);
}

template <class T> void k_spmv(Ctx& c, const Csr<T>& A, const T* x, T* y, int variant) { spmv_launch<T, false>(c, A, x, y, 1, variant); }

// ---------------------------------------------------------------------------
// General x-halo exchange of row-partitioned operators (dist.cuh: DistExchange)
// ---------------------------------------------------------------------------
template <class T> struct ExchangeDst { T* p[kMaxRanks]; };

template <class T>
__global__ void __launch_bounds__(kBlock) halo_exchange_kernel(const T* __restrict__ x, int nsend, const int* __restrict__ row,
                                                               const int* __restrict__ peer, const int* __restrict__ slot,
                                                               ExchangeDst<T> dst, unsigned* ticket, DistComm* dc) {
  __shared__ bool is_last;
  const int stride = gridDim.x * blockDim.x;
  bool sent = false;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nsend; e += stride) {
    dst.p[peer[e]][slot[e]] = x[row[e]];
    sent = true;
  }
  if (sent) __threadfence_system();        // my stores are visible to the peers before the barrier below
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
    if (is_last) *ticket = 0u;
  }
  __syncthreads();
  // the last CTA of this rank enters the cross-GPU barrier: when it returns, every rank has finished pushing
  if (is_last && threadIdx.x == 0) dist_allreduce_sum(dc, 0.0);
}

template <class T> void k_halo_exchange(Ctx& c, const T* x) {
  if (!c.dex) return;
  DistExchange& d = *c.dex;
  ExchangeDst<T> dst;
  const size_t par = (size_t)(d.count & 1);
  for (int k = 0; k < kMaxRanks; k++)
    dst.p[k] = d.xhalo_peer[k] ? reinterpret_cast<T*>(d.xhalo_peer[k]) + par * (size_t)d.nhalo_peer[k] : nullptr;
  const int grid = d.nsend > 0 ? std::min(sm_count(), (d.nsend + kBlock - 1) / kBlock) : 1;
  halo_exchange_kernel<T><<<grid, kBlock, 0, c.stream>>>(x, d.nsend, d.send_row, d.send_peer, d.send_slot, dst, c.tickets + 6, c.dcomm);
  KB_CUDA(cudaGetLastError());
  c.launches++;
  d.count++;
}

// ---------------------------------------------------------------------------
// Operator application (A, M, N as the solvers see them)
// ---------------------------------------------------------------------------
template <class T> void op_apply(Ctx& c, const LinOp<T>& op, const T* x, T* y, bool ldiv) {
  switch (op.kind) {
    case LinOp<T>::CSR:
      k_halo_exchange<T>(c, x);            // row-partitioned operators only; no-op on a single GPU
      k_spmv<T>(c, *op.csr, x, y, 0);
      break;
    case LinOp<T>::DIAG: k_diagmul<T>(c, op.n, y, op.diag, x, ldiv); break;
    case LinOp<T>::BDIAG: k_blockdiag_mul<T>(c, op.n, op.bs, ldiv ? op.blocks_inv : op.blocks, x, y); break;
    case LinOp<T>::DEV_CB:
      c.sync();                       // the callback may use its own stream
      op.fn(x, y, op.userdata);
      KB_CUDA(cudaDeviceSynchronize());
      break;
    case LinOp<T>::HOST_CB:
      // reference: ccall(op.fptr, ..., x, y, userdata) on host pointers
      // (interfaces/src/c_operator.jl:35-42); here x/y live in HBM, so stage.
      KB_CUDA(cudaMemcpyAsync(op.hx, x, sizeof(T) * (size_t)op.n, cudaMemcpyDeviceToHost, c.stream));
      c.sync();
      op.fn(op.hx, op.hy, op.userdata);
      KB_CUDA(cudaMemcpyAsync(y, op.hy, sizeof(T) * (size_t)op.n, cudaMemcpyHostToDevice, c.stream));
      break;
    case LinOp<T>::NONE: k_copy<T>(c, op.n, y, x); break;
  }
}

#define INST(T)                                                                                                  \
  template void csr_upload<T>(Ctx&, Csr<T>&, int, long long, const void*, const void*, const T*, int, int, bool); \
  template void csr_free<T>(Csr<T>&);                                                                            \
  template void csr_plan<T>(Ctx&, Csr<T>&);                                                                      \
  template void k_spmv<T>(Ctx&, const Csr<T>&, const T*, T*, int);                                               \
  template void k_halo_exchange<T>(Ctx&, const T*);                                                              \
  template void op_apply<T>(Ctx&, const LinOp<T>&, const T*, T*, bool);
INST(double)
INST(float)
#undef INST

}  // namespace kb
