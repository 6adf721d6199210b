// Affinity graph (reference models/mpti.py:717-756) and label propagation (models/mpti.py:758-776)
// in sparse form, plus the query loss / prediction / confusion counters.
#include <cooperative_groups.h>

#include "common.cuh"
#include "lp.cuh"

namespace cg = cooperative_groups;

// --------------------------------------------------------------------------------------------
// Per-row selection of the k nearest other valid nodes: 4-pass 8-bit radix select on the row's
// order-preserving integer keys in shared memory, then an ordered compaction (ties at the k-th
// distance -> lowest index).  One CTA per row.
// --------------------------------------------------------------------------------------------
#define SEL_THREADS 256

__global__ __launch_bounds__(SEL_THREADS) void knn_select_kernel(const float* __restrict__ D2,
                                                                 const uint8_t* __restrict__ valid,
                                                                 int nn, int k,
                                                                 int32_t* __restrict__ nbr) {
  extern __shared__ unsigned s_key[];  // [nn]
  __shared__ int s_hist[256];
  __shared__ unsigned s_prefix, s_mask;
  __shared__ int s_need;
  __shared__ int s_w[2][SEL_THREADS / 32];
  const int g = blockIdx.y, i = blockIdx.x;
  const uint8_t* vg = valid + (int64_t)g * nn;
  if (!vg[i]) return;
  const float* row = D2 + ((int64_t)g * nn + i) * nn;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int j = tid; j < nn; j += SEL_THREADS) {
    unsigned key = 0xffffffffu;
    if (j != i && vg[j]) {
      key = f2key(row[j]);
      if (key == 0xffffffffu) key = 0xfffffffeu;
    }
    s_key[j] = key;
  }
  if (tid == 0) {
    s_prefix = 0;
    s_mask = 0;
    s_need = k;
  }
  for (int pass = 3; pass >= 0; --pass) {
    const int shift = 8 * pass;
    s_hist[tid] = 0;  // SEL_THREADS == 256
    __syncthreads();
    const unsigned prefix = s_prefix, mask = s_mask;
    for (int j = tid; j < nn; j += SEL_THREADS) {
      const unsigned key = s_key[j];
      if ((key & mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 255], 1);
    }
    __syncthreads();
    if (w == 0) {
      // which bin holds the need-th smallest key: warp scan over 8 bins per lane (a single thread
      // walking the 256 bins was ~25 % of the kernel's instructions)
      int h[8], local = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        h[q] = s_hist[8 * lane + q];
        local += h[q];
      }
      int incl = local;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += a;
      }
      const int need = s_need, excl = incl - local;
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      // first bin b (< 255) with cum(b) + hist[b] >= need, else b = 255 — as the serial walk
      bool mine = excl < need && need <= incl;
      if (total < need) mine = lane == 31;
      __syncwarp();
      if (mine) {
        int cum = excl, b = 8 * lane;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (b == 255 || cum + h[q] >= need) break;
          cum += h[q];
          ++b;
        }
        s_need = need - cum;
        s_prefix = prefix | ((unsigned)b << shift);
        s_mask = mask | (255u << shift);
      }
    }
    __syncthreads();
  }
  const unsigned T = s_prefix;
  const int need_eq = s_need;
  int32_t* out = nbr + ((int64_t)g * nn + i) * k;
  // ordered compaction with two barriers: every thread owns a contiguous run of `per` keys (odd
  // stride -> conflict-free), counts its (< T) and (== T) keys, a block-wide exclusive scan gives
  // its output offset and its rank among the ties, then it writes its selected indices in order.
  int per = (nn + SEL_THREADS - 1) / SEL_THREADS;
  per |= 1;
  const int j0 = tid * per, j1 = min(nn, j0 + per);
  int c_lt = 0, c_eq = 0;
  for (int j = j0; j < j1; ++j) {
    const unsigned key = s_key[j];
    c_lt += key < T;
    c_eq += key == T;
  }
  // warp inclusive scans
  int s_lt = c_lt, s_eq = c_eq;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, s_lt, o), b2 = __shfl_up_sync(0xffffffffu, s_eq, o);
    if (lane >= o) {
      s_lt += a;
      s_eq += b2;
    }
  }
  if (lane == 31) {
    s_w[0][w] = s_lt;
    s_w[1][w] = s_eq;
  }
  __syncthreads();
  int off_lt = s_lt - c_lt, off_eq = s_eq - c_eq;
  for (int q = 0; q < w; ++q) {
    off_lt += s_w[0][q];
    off_eq += s_w[1][q];
  }
  // output position of my first selected key = (#lt before me) + min(#eq before me, need_eq)
  int pos = off_lt + min(off_eq, need_eq);
  int eq_rank = off_eq;
  for (int j = j0; j < j1; ++j) {
    const unsigned key = s_key[j];
    bool sel = key < T;
    if (key == T) {
      sel = eq_rank < need_eq;
      ++eq_rank;
    }
    if (sel) {
      if (pos < k) out[pos] = j;
      ++pos;
    }
  }
}

// Same selection, one WARP per row with the row's keys in registers (KPL per lane, j = lane + 32 t):
// the k-th smallest key is found by narrowing [lo, hi] eight bits at a time from the row's actual
// key range (the top radix digits of distances that span two or three binades carry no
// information), stopping as soon as the boundary bin is taken whole; the ordered compaction is a
// ballot per 32 keys.  No block barrier anywhere.  Output identical to knn_select_kernel.
#define SELW_WARPS 8

template <int KPL>
__global__ __launch_bounds__(SELW_WARPS * 32) void knn_select_warp_kernel(
    const float* __restrict__ D2, const uint8_t* __restrict__ valid, int nn, int k,
    int32_t* __restrict__ nbr) {
  __shared__ int s_hist[SELW_WARPS][256];
  __shared__ unsigned s_vbits[KPL];  // validity of the graph's nodes, one bit per node
  const int g = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * SELW_WARPS + w;
  const uint8_t* vg = valid + (int64_t)g * nn;
  for (int t = w; t < KPL; t += SELW_WARPS) {
    const int j = lane + 32 * t;
    const unsigned bits = __ballot_sync(0xffffffffu, j < nn && vg[j] != 0);
    if (lane == 0) s_vbits[t] = bits;
  }
  __syncthreads();
  if (i >= nn) return;
  if (!((s_vbits[i >> 5] >> (i & 31)) & 1u)) return;
  const float* row = D2 + ((int64_t)g * nn + i) * nn;
  int* hist = s_hist[w];
  // every load of the row is issued before the first use (no load sits behind a validity branch)
  float v[KPL];
#pragma unroll
  for (int t = 0; t < KPL; ++t) v[t] = __ldcs(row + min(lane + 32 * t, nn - 1));
  unsigned key[KPL];
  unsigned lo = 0xffffffffu, hi = 0u;
  int n_real = 0;
#pragma unroll
  for (int t = 0; t < KPL; ++t) {
    const int j = lane + 32 * t;
    unsigned kk = f2key(v[t]);
    if (kk == 0xffffffffu) kk = 0xfffffffeu;
    const bool real = ((s_vbits[t] >> lane) & 1u) && j != i;
    lo = real ? min(lo, kk) : lo;
    hi = real ? max(hi, kk) : hi;
    n_real += real;
    key[t] = real ? kk : 0xffffffffu;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    n_real += __shfl_xor_sync(0xffffffffu, n_real, o);
  }
  unsigned T;
  int need_eq;
  if (n_real < k) {  // every real key, then the lowest-index fillers
    T = 0xffffffffu;
    need_eq = k - n_real;
  } else {
    int need = k;
    while (true) {
      const unsigned range = hi - lo;
      if (range == 0) {
        T = lo;
        need_eq = need;
        break;
      }
      const int sh = max(0, 24 - (int)__clz(range));  // (key - lo) >> sh  in [0, 255]
#pragma unroll
      for (int q = 0; q < 8; ++q) hist[lane + 32 * q] = 0;
      __syncwarp();
#pragma unroll
      for (int t = 0; t < KPL; ++t)
        if (key[t] >= lo && key[t] <= hi) atomicAdd(&hist[(key[t] - lo) >> sh], 1);
      __syncwarp();
      int h[8], local = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        h[q] = hist[8 * lane + q];
        local += h[q];
      }
      int incl = local;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += a;
      }
      const int excl = incl - local;
      const bool mine = excl < need && need <= incl;  // exactly one lane: total >= need
      int b = 0, cum = 0, hb = 0;
      if (mine) {
        cum = excl;
        b = 8 * lane;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          hb = h[q];
          if (cum + h[q] >= need) break;
          cum += h[q];
          ++b;
        }
      }
      const unsigned owner = __ballot_sync(0xffffffffu, mine);
      const int src = __ffs(owner) - 1;
      b = __shfl_sync(0xffffffffu, b, src);
      cum = __shfl_sync(0xffffffffu, cum, src);
      hb = __shfl_sync(0xffffffffu, hb, src);
      __syncwarp();
      need -= cum;
      const unsigned nlo = lo + ((unsigned)b << sh);
      const unsigned nhi = min(hi, nlo + ((1u << sh) - 1u));
      if (hb == need) {  // the whole boundary bin is taken: nothing ties at the cut
        T = nhi + 1u;    // nhi <= 0xfffffffe
        need_eq = 0;
        break;
      }
      if (sh == 0) {     // the bin is a single key value
        T = nlo;
        need_eq = need;
        break;
      }
      lo = nlo;
      hi = nhi;
    }
  }
  int32_t* out = nbr + ((int64_t)g * nn + i) * k;
  const unsigned lt_mask = (1u << lane) - 1u;
  int pos = 0, eq_seen = 0;
#pragma unroll
  for (int t = 0; t < KPL; ++t) {
    const bool is_eq = key[t] == T && (lane + 32 * t) < nn;
    const unsigned eqb = __ballot_sync(0xffffffffu, is_eq);
    bool sel = key[t] < T;
    if (is_eq) sel = eq_seen + __popc(eqb & lt_mask) < need_eq;
    const unsigned sb = __ballot_sync(0xffffffffu, sel);
    if (sel) {
      const int p = pos + __popc(sb & lt_mask);
      if (p < k) out[p] = lane + 32 * t;
    }
    pos += __popc(sb);
    eq_seen += __popc(eqb);
  }
}

// Rows too long for one warp's registers (nn up to 31 * 256): one CTA per row, every thread keeps a
// contiguous run of the row's keys in registers (staged through shared memory so the global loads
// stay coalesced), the same range narrowing with ONE barrier per pass (three rotating histograms,
// every warp scans the bins for itself), then the ordered compaction of knn_select_kernel.
template <int KPT, int NT = SEL_THREADS>
__global__ __launch_bounds__(NT, (KPT <= 20 ? 1024 : 512) / NT) void knn_select_reg_kernel(
    const float* __restrict__ D2, const uint8_t* __restrict__ valid, int nn, int k,
    int32_t* __restrict__ nbr) {
  extern __shared__ unsigned s_key[];  // [nn]
  __shared__ int s_hist[3][256];
  __shared__ unsigned s_lo[NT / 32], s_hi[NT / 32];
  __shared__ int s_cnt[NT / 32];
  __shared__ int s_w[2][NT / 32];
  const int g = blockIdx.y, i = blockIdx.x;
  const uint8_t* vg = valid + (int64_t)g * nn;
  if (!vg[i]) return;
  const float* row = D2 + ((int64_t)g * nn + i) * nn;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  unsigned lo = 0xffffffffu, hi = 0u;
  int n_real = 0;
  for (int j = tid; j < nn; j += NT) {
    const float v = __ldcs(row + j);
    const bool real = vg[j] != 0 && j != i;
    unsigned kk = f2key(v);
    if (kk == 0xffffffffu) kk = 0xfffffffeu;
    lo = real ? min(lo, kk) : lo;
    hi = real ? max(hi, kk) : hi;
    n_real += real;
    s_key[j] = real ? kk : 0xffffffffu;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    n_real += __shfl_xor_sync(0xffffffffu, n_real, o);
  }
  if (lane == 0) {
    s_lo[w] = lo;
    s_hi[w] = hi;
    s_cnt[w] = n_real;
  }
  if (tid < 256) s_hist[0][tid] = 0;
  __syncthreads();
  n_real = 0;
#pragma unroll
  for (int q = 0; q < NT / 32; ++q) {
    lo = min(lo, s_lo[q]);
    hi = max(hi, s_hi[q]);
    n_real += s_cnt[q];
  }
  // my contiguous run (odd length -> conflict-free shared-memory reads)
  int per = (nn + NT - 1) / NT;
  per |= 1;
  const int j0 = tid * per;
  unsigned key[KPT];
#pragma unroll
  for (int t = 0; t < KPT; ++t) key[t] = (t < per && j0 + t < nn) ? s_key[j0 + t] : 0xffffffffu;
  unsigned T;
  int need_eq;
  if (n_real < k) {
    T = 0xffffffffu;
    need_eq = k - n_real;
  } else {
    int need = k, p = 0;
    while (true) {
      const unsigned range = hi - lo;
      if (range == 0) {
        T = lo;
        need_eq = need;
        break;
      }
      const int sh = max(0, 24 - (int)__clz(range));
      int* hist = s_hist[p % 3];
      if (tid < 256) s_hist[(p + 1) % 3][tid] = 0;  // last read two passes ago
#pragma unroll
      for (int t = 0; t < KPT; ++t)
        if (key[t] >= lo && key[t] <= hi) atomicAdd(&hist[(key[t] - lo) >> sh], 1);
      __syncthreads();
      int h[8], local = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        h[q] = hist[8 * lane + q];
        local += h[q];
      }
      int incl = local;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += a;
      }
      const int excl = incl - local;
      const bool mine = excl < need && need <= incl;
      int b = 0, cum = 0, hb = 0;
      if (mine) {
        cum = excl;
        b = 8 * lane;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          hb = h[q];
          if (cum + h[q] >= need) break;
          cum += h[q];
          ++b;
        }
      }
      const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
      b = __shfl_sync(0xffffffffu, b, src);
      cum = __shfl_sync(0xffffffffu, cum, src);
      hb = __shfl_sync(0xffffffffu, hb, src);
      need -= cum;
      const unsigned nlo = lo + ((unsigned)b << sh);
      const unsigned nhi = min(hi, nlo + ((1u << sh) - 1u));
      if (hb == need) {
        T = nhi + 1u;
        need_eq = 0;
        break;
      }
      if (sh == 0) {
        T = nlo;
        need_eq = need;
        break;
      }
      lo = nlo;
      hi = nhi;
      ++p;
    }
  }
  int32_t* out = nbr + ((int64_t)g * nn + i) * k;
  int c_lt = 0, c_eq = 0;
#pragma unroll
  for (int t = 0; t < KPT; ++t) {
    const bool in = t < per && j0 + t < nn;
    c_lt += in && key[t] < T;
    c_eq += in && key[t] == T;
  }
  int s_lt = c_lt, s_eq = c_eq;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, s_lt, o), b2 = __shfl_up_sync(0xffffffffu, s_eq, o);
    if (lane >= o) {
      s_lt += a;
      s_eq += b2;
    }
  }
  if (lane == 31) {
    s_w[0][w] = s_lt;
    s_w[1][w] = s_eq;
  }
  __syncthreads();
  int off_lt = s_lt - c_lt, off_eq = s_eq - c_eq;
  for (int q = 0; q < w; ++q) {
    off_lt += s_w[0][q];
    off_eq += s_w[1][q];
  }
  int pos = off_lt + min(off_eq, need_eq);
  int eq_rank = off_eq;
#pragma unroll
  for (int t = 0; t < KPT; ++t) {
    if (t < per && j0 + t < nn) {
      bool sel = key[t] < T;
      if (key[t] == T) {
        sel = eq_rank < need_eq;
        ++eq_rank;
      }
      if (sel) {
        if (pos < k) out[pos] = j0 + t;
        ++pos;
      }
    }
  }
}

// --------------------------------------------------------------------------------------------
// Bounded selection: the same neighbour lists from the distance GEMM's group minima (AFF_GROUP
// contiguous columns per group, tc_gemm_tma.cu) and one pass over the row.
//
// Why the bound holds: let tau be the k-th smallest group minimum.  The k groups with the smallest
// minima each hold a distinct real column whose key is <= tau, so the k-th smallest real key T
// satisfies T <= tau.  Every selected column has a key <= T <= tau, and so does every column whose
// key equals T.  The candidates (real columns with key <= tau), kept in column order, therefore
// hold all the columns the select can pick and every tie at T, in the order that sends ties to the
// lowest index: the exact select on the candidates is the exact select on the row.
//
// One warp per row: tau by range narrowing over the ~nn / AFF_GROUP group minima; the row streamed
// once in 16-byte loads, the candidates ballot-compacted into the warp's shared buffer; the exact
// select (T, ties, ordered list) on the candidates.  A row without a bound (fewer than k groups hold
// a real column) or with more than SELB_CAP candidates takes the same exact select on the whole row,
// read again from global memory.  Needs nn % 4 == 0 and a 4-byte aligned `valid`.
// --------------------------------------------------------------------------------------------
#define SELB_WARPS 4
#define SELB_CAP 1024  // candidates per row (see bounded_select_pays)
#define SELB_LOADS 8    // 16-byte loads in flight per lane

// the k-th smallest (k >= 1) of the keys key_at(0 .. n-1) that are not 0xffffffff, as T and the
// number need_eq of keys equal to T among the k smallest; with fewer than k such keys, T = 0xffffffff
// and need_eq = k - their count.  The range narrowing of knn_select_warp_kernel.  Whole warp.
template <class KeyAt>
__device__ __forceinline__ void warp_kth_key(int n, int k, KeyAt key_at, int* hist, int lane,
                                             unsigned& T, int& need_eq) {
  unsigned lo = 0xffffffffu, hi = 0u;
  int n_real = 0;
  for (int j = lane; j < n; j += 32) {
    const unsigned kk = key_at(j);
    const bool real = kk != 0xffffffffu;
    lo = real ? min(lo, kk) : lo;
    hi = real ? max(hi, kk) : hi;
    n_real += real;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    n_real += __shfl_xor_sync(0xffffffffu, n_real, o);
  }
  if (n_real < k) {
    T = 0xffffffffu;
    need_eq = k - n_real;
    return;
  }
  int need = k;
  while (true) {
    const unsigned range = hi - lo;
    if (range == 0) {
      T = lo;
      need_eq = need;
      return;
    }
    const int sh = max(0, 24 - (int)__clz(range));
#pragma unroll
    for (int q = 0; q < 8; ++q) hist[lane + 32 * q] = 0;
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
      const unsigned kk = key_at(j);
      if (kk >= lo && kk <= hi) atomicAdd(&hist[(kk - lo) >> sh], 1);
    }
    __syncwarp();
    int h[8], local = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      h[q] = hist[8 * lane + q];
      local += h[q];
    }
    int incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += a;
    }
    const int excl = incl - local;
    const bool mine = excl < need && need <= incl;
    int b = 0, cum = 0, hb = 0;
    if (mine) {
      cum = excl;
      b = 8 * lane;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        hb = h[q];
        if (cum + h[q] >= need) break;
        cum += h[q];
        ++b;
      }
    }
    const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
    b = __shfl_sync(0xffffffffu, b, src);
    cum = __shfl_sync(0xffffffffu, cum, src);
    hb = __shfl_sync(0xffffffffu, hb, src);
    __syncwarp();
    need -= cum;
    const unsigned nlo = lo + ((unsigned)b << sh);
    const unsigned nhi = min(hi, nlo + ((1u << sh) - 1u));
    if (hb == need) {
      T = nhi + 1u;
      need_eq = 0;
      return;
    }
    if (sh == 0) {
      T = nlo;
      need_eq = need;
      return;
    }
    lo = nlo;
    hi = nhi;
  }
}

// out[0 .. k-1] = col_at(j) of the keys < T and of the first need_eq keys == T, in the order of j
template <class KeyAt, class ColAt>
__device__ __forceinline__ void warp_emit_selected(int n, int k, KeyAt key_at, ColAt col_at,
                                                   unsigned T, int need_eq, int lane, int32_t* out) {
  const unsigned lt_mask = (1u << lane) - 1u;
  int pos = 0, eq_seen = 0;
  for (int j0 = 0; j0 < n && pos < k; j0 += 32) {
    const int j = j0 + lane;
    const unsigned kk = j < n ? key_at(j) : 0u;
    const bool is_eq = j < n && kk == T;
    const unsigned eqb = __ballot_sync(0xffffffffu, is_eq);
    bool sel = j < n && kk < T;
    if (is_eq) sel = eq_seen + __popc(eqb & lt_mask) < need_eq;
    const unsigned sb = __ballot_sync(0xffffffffu, sel);
    if (sel) {
      const int p = pos + __popc(sb & lt_mask);
      if (p < k) out[p] = col_at(j);
    }
    pos += __popc(sb);
    eq_seen += __popc(eqb);
  }
}

__global__ __launch_bounds__(SELB_WARPS * 32) void knn_select_bounded_kernel(
    const float* __restrict__ D2, const uint8_t* __restrict__ valid,
    const unsigned* __restrict__ gmin, int nn, int k, int32_t* __restrict__ nbr) {
  __shared__ unsigned s_key[SELB_WARPS][SELB_CAP];
  __shared__ uint16_t s_col[SELB_WARPS][SELB_CAP];
  __shared__ int s_hist[SELB_WARPS][256];
  const int g = blockIdx.y, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * SELB_WARPS + w;  // no block barrier below: a warp may leave
  if (i >= nn) return;
  const uint8_t* vg = valid + (int64_t)g * nn;
  if (!vg[i]) return;
  const float* row = D2 + ((int64_t)g * nn + i) * nn;
  int32_t* out = nbr + ((int64_t)g * nn + i) * k;
  int* hist = s_hist[w];
  unsigned* ck = s_key[w];
  uint16_t* cc = s_col[w];
  const int ngrp = (nn + AFF_GROUP - 1) / AFF_GROUP;
  const unsigned* gr = gmin + ((int64_t)g * nn + i) * aff_gstride(nn);
  // tau: any key with at least k group minima at or below it bounds the cut; T - 1 when exactly k
  // minima lie below T
  unsigned T;
  int need_eq;
  warp_kth_key(ngrp, k, [&](int j) { return __ldg(gr + j); }, hist, lane, T, need_eq);
  int cnt = 0;
  if (T != 0xffffffffu) {
    const unsigned tau = need_eq == 0 ? T - 1u : T;
    const float4* row4 = reinterpret_cast<const float4*>(row);
    const uint32_t* vw = reinterpret_cast<const uint32_t*>(vg);
    const unsigned lt_mask = (1u << lane) - 1u;
    const int nq = nn / 4;
    // SELB_LOADS 16-byte loads per lane are issued before any of them is used: the compaction's
    // ballots and shared-memory stores would otherwise hold every load back behind the last one
    for (int q0 = 0; q0 < nq; q0 += 32 * SELB_LOADS) {
      float4 vv[SELB_LOADS];
      uint32_t vbs[SELB_LOADS];
#pragma unroll
      for (int u = 0; u < SELB_LOADS; ++u) {
        const int q = q0 + 32 * u + lane;
        vv[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        vbs[u] = 0;
        if (q < nq) {
          vv[u] = __ldcs(row4 + q);
          vbs[u] = __ldg(vw + q);
        }
      }
#pragma unroll
      for (int u = 0; u < SELB_LOADS; ++u) {
        const int q = q0 + 32 * u + lane;  // columns 4 q .. 4 q + 3
        const float e[4] = {vv[u].x, vv[u].y, vv[u].z, vv[u].w};
        bool c[4];
        int nc = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          c[t] = ((vbs[u] >> (8 * t)) & 0xffu) && 4 * q + t != i && dist_key(e[t]) <= tau;
          nc += c[t];
        }
        // ordered compaction: exclusive prefix of the lanes' counts (0..4) from three bit ballots
        const unsigned m0 = __ballot_sync(0xffffffffu, nc & 1),
                       m1 = __ballot_sync(0xffffffffu, nc & 2),
                       m2 = __ballot_sync(0xffffffffu, nc & 4);
        int p = cnt + __popc(m0 & lt_mask) + 2 * __popc(m1 & lt_mask) + 4 * __popc(m2 & lt_mask);
#pragma unroll
        for (int t = 0; t < 4; ++t)
          if (c[t]) {
            if (p < SELB_CAP) {
              ck[p] = dist_key(e[t]);
              cc[p] = (uint16_t)(4 * q + t);
            }
            ++p;
          }
        cnt += __popc(m0) + 2 * __popc(m1) + 4 * __popc(m2);
      }
    }
    __syncwarp();
  }
  if (T != 0xffffffffu && cnt <= SELB_CAP) {
    warp_kth_key(cnt, k, [&](int j) { return ck[j]; }, hist, lane, T, need_eq);
    warp_emit_selected(cnt, k, [&](int j) { return ck[j]; }, [&](int j) { return (int)cc[j]; }, T,
                       need_eq, lane, out);
  } else {
    auto key_at = [&](int j) {
      return (vg[j] && j != i) ? dist_key(__ldcg(row + j)) : 0xffffffffu;
    };
    warp_kth_key(nn, k, key_at, hist, lane, T, need_eq);
    warp_emit_selected(nn, k, key_at, [](int j) { return j; }, T, need_eq, lane, out);
  }
}

// --------------------------------------------------------------------------------------------
// Gaussian similarity of the kept edges (models/mpti.py:745-746) with torch<=1.8
// pairwise_distance: dist = || f_i - f_j + 1e-6 ||_2 by direct differences, sim = exp(-0.5 (dist/sigma)^2).
// One warp per node, 8 lanes per neighbour.  VEC: the feature rows are 16-byte aligned (read as
// float4); otherwise each float4 is assembled from four scalar loads.
// --------------------------------------------------------------------------------------------
#define LP_MAX_F4 8

template <bool VEC>
__device__ __forceinline__ float4 ld_f4(const float* p) {
  if (VEC) return *reinterpret_cast<const float4*>(p);
  return make_float4(p[0], p[1], p[2], p[3]);
}

template <bool VEC>
__global__ __launch_bounds__(256) void edge_sim_kernel(const float* __restrict__ F,
                                                       int64_t graph_rows, int64_t row_off, int nn,
                                                       int D, const uint8_t* __restrict__ valid,
                                                       const int32_t* __restrict__ nbr, int k,
                                                       float sigma, float* __restrict__ sim) {
  const int g = blockIdx.y;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= nn) return;
  if (!valid[(int64_t)g * nn + i]) return;
  const int lane = threadIdx.x & 31, sub = lane & 7, grp = lane >> 3;
  const float* Fg = F + ((int64_t)g * graph_rows + row_off) * D;
  const int D4 = D >> 2;
  float4 xf[LP_MAX_F4];
  const float* xrow = Fg + (int64_t)i * D;
#pragma unroll
  for (int u = 0; u < LP_MAX_F4; ++u) {
    int c4 = sub + 8 * u;
    xf[u] = (c4 < D4) ? ld_f4<VEC>(xrow + 4 * c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const int32_t* nb = nbr + ((int64_t)g * nn + i) * k;
  float* so = sim + ((int64_t)g * nn + i) * k;
  for (int t0 = 0; t0 < k; t0 += 4) {
    const int t = t0 + grp;
    const bool ok = t < k;
    const int j = ok ? nb[t] : i;
    const float* yrow = Fg + (int64_t)j * D;
    float acc = 0.f;
#pragma unroll
    for (int u = 0; u < LP_MAX_F4; ++u) {
      int c4 = sub + 8 * u;
      if (c4 < D4) {
        float4 y = ld_f4<VEC>(yrow + 4 * c4);
        float d0 = __fadd_rn(xf[u].x - y.x, 1e-6f), d1 = __fadd_rn(xf[u].y - y.y, 1e-6f),
              d2 = __fadd_rn(xf[u].z - y.z, 1e-6f), d3 = __fadd_rn(xf[u].w - y.w, 1e-6f);
        acc = fmaf(d0, d0, acc);
        acc = fmaf(d1, d1, acc);
        acc = fmaf(d2, d2, acc);
        acc = fmaf(d3, d3, acc);
      }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    acc += __shfl_xor_sync(0xffffffffu, acc, 4);
    if (ok && sub == 0) {
      const float tt = sqrtf(acc) / sigma;
      so[t] = expf(-0.5f * (tt * tt));
    }
  }
}

// --------------------------------------------------------------------------------------------
// In-edge lists (the A^T half of W = A + A^T, models/mpti.py:752): count, scan, fill, then sort
// each column's list by source so the result does not depend on atomic ordering.
// --------------------------------------------------------------------------------------------
__global__ void in_count_kernel(const int32_t* __restrict__ nbr, const uint8_t* __restrict__ valid,
                                int nn, int k, int32_t* __restrict__ in_cnt) {
  const int g = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nn * k) return;
  const int i = (int)(e / k);
  if (!valid[(int64_t)g * nn + i]) return;
  const int j = nbr[(int64_t)g * nn * k + e];
  atomicAdd(&in_cnt[(int64_t)g * nn + j], 1);
}

// exclusive scan of in_cnt -> in_ptr (nn + 1 entries per graph); also zeroes the fill cursors
__global__ __launch_bounds__(1024) void in_scan_kernel(int32_t* __restrict__ in_cnt, int nn,
                                                       int32_t* __restrict__ in_ptr) {
  __shared__ int s_part[1024];
  const int g = blockIdx.x, tid = threadIdx.x;
  int32_t* cnt = in_cnt + (int64_t)g * nn;
  int32_t* ptr = in_ptr + (int64_t)g * (nn + 1);
  const int per = (nn + 1023) / 1024;
  const int lo = min(nn, tid * per), hi = min(nn, lo + per);
  int s = 0;
  for (int i = lo; i < hi; ++i) s += cnt[i];
  s_part[tid] = s;
  __syncthreads();
  // Hillis-Steele inclusive scan over 1024 partials
  for (int o = 1; o < 1024; o <<= 1) {
    int v = tid >= o ? s_part[tid - o] : 0;
    __syncthreads();
    s_part[tid] += v;
    __syncthreads();
  }
  int run = tid == 0 ? 0 : s_part[tid - 1];
  for (int i = lo; i < hi; ++i) {
    ptr[i] = run;
    run += cnt[i];
    cnt[i] = 0;  // reused as the fill cursor
  }
  if (tid == 1023) ptr[nn] = s_part[1023];
}

__global__ void in_fill_kernel(const int32_t* __restrict__ nbr, const float* __restrict__ sim,
                               const uint8_t* __restrict__ valid, int nn, int k,
                               const int32_t* __restrict__ in_ptr, int32_t* __restrict__ cursor,
                               int32_t* __restrict__ in_src, float* __restrict__ in_w) {
  const int g = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nn * k) return;
  const int i = (int)(e / k);
  if (!valid[(int64_t)g * nn + i]) return;
  const int64_t ge = (int64_t)g * nn * k + e;
  const int j = nbr[ge];
  const int pos = in_ptr[(int64_t)g * (nn + 1) + j] + atomicAdd(&cursor[(int64_t)g * nn + j], 1);
  in_src[(int64_t)g * nn * k + pos] = i;
  in_w[(int64_t)g * nn * k + pos] = sim[ge];
}

// Sort-free variant of the same lists.  The transposed adjacency is first written as a BIT matrix
// (bits[j] has bit i set when i -> j; atomicOr is order-independent), a row's word-prefix popcounts
// give every in-edge its rank among the sources of its column, and the fill writes (source,
// weight) straight to that rank: the lists come out sorted by source with no atomics on the
// position and nothing to sort afterwards.
__global__ void in_bits_kernel(const int32_t* __restrict__ nbr, const uint8_t* __restrict__ valid,
                               int nn, int k, int W, uint32_t* __restrict__ bits) {
  const int g = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nn * k) return;
  const int i = (int)(e / k);
  if (!valid[(int64_t)g * nn + i]) return;
  const int j = nbr[(int64_t)g * nn * k + e];
  atomicOr(&bits[((int64_t)g * nn + j) * W + (i >> 5)], 1u << (i & 31));
}

// one warp per column j: exclusive popcount prefix of its words -> pre (uint16), total -> in_cnt
__global__ __launch_bounds__(256) void in_rank_kernel(const uint32_t* __restrict__ bits, int nn,
                                                      int W, uint16_t* __restrict__ pre,
                                                      int32_t* __restrict__ in_cnt) {
  const int g = blockIdx.y, lane = threadIdx.x & 31;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (j >= nn) return;
  const uint32_t* b = bits + ((int64_t)g * nn + j) * W;
  uint16_t* p = pre + ((int64_t)g * nn + j) * W;
  int base = 0;
  for (int w0 = 0; w0 < W; w0 += 32) {
    const int w = w0 + lane;
    const int c = w < W ? __popc(b[w]) : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += a;
    }
    if (w < W) p[w] = (uint16_t)(base + incl - c);
    base += __shfl_sync(0xffffffffu, incl, 31);
  }
  if (lane == 0) in_cnt[(int64_t)g * nn + j] = base;
}

__global__ void in_fill_rank_kernel(const int32_t* __restrict__ nbr, const float* __restrict__ sim,
                                    const uint8_t* __restrict__ valid, int nn, int k, int W,
                                    const uint32_t* __restrict__ bits,
                                    const uint16_t* __restrict__ pre,
                                    const int32_t* __restrict__ in_ptr,
                                    int32_t* __restrict__ in_src, float* __restrict__ in_w) {
  const int g = blockIdx.y;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)nn * k) return;
  const int i = (int)(e / k);
  if (!valid[(int64_t)g * nn + i]) return;
  const int64_t ge = (int64_t)g * nn * k + e;
  const int j = nbr[ge];
  const int64_t o = ((int64_t)g * nn + j) * W + (i >> 5);
  const int rank = (int)pre[o] + __popc(bits[o] & ((1u << (i & 31)) - 1u));
  const int pos = in_ptr[(int64_t)g * (nn + 1) + j] + rank;
  in_src[(int64_t)g * nn * k + pos] = i;
  in_w[(int64_t)g * nn * k + pos] = sim[ge];
}

// Launched twice: a small-capacity pass (segments up to `cap_hi` entries, little shared memory ->
// many resident CTAs) and a large-capacity pass for the few hub columns (cap_lo < L <= cap_hi).
__global__ __launch_bounds__(256) void in_sort_kernel(const int32_t* __restrict__ in_ptr, int nn,
                                                      int k, int32_t* __restrict__ in_src,
                                                      float* __restrict__ in_w, int cap_lo,
                                                      int cap_hi) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  const int g = blockIdx.y, j = blockIdx.x;
  const int32_t* ptr = in_ptr + (int64_t)g * (nn + 1);
  const int lo = ptr[j], L = ptr[j + 1] - lo;
  if (L <= 1 || L <= cap_lo || L > cap_hi) return;
  int P = 2;
  while (P < L) P <<= 1;
  int* s_src = reinterpret_cast<int*>(s_raw);
  float* s_val = reinterpret_cast<float*>(s_raw) + P;
  int32_t* src = in_src + (int64_t)g * nn * k + lo;
  float* val = in_w + (int64_t)g * nn * k + lo;
  const int tid = threadIdx.x;
  for (int t = tid; t < P; t += 256) {
    s_src[t] = t < L ? src[t] : 0x7fffffff;
    s_val[t] = t < L ? val[t] : 0.f;
  }
  __syncthreads();
  for (int ksz = 2; ksz <= P; ksz <<= 1)
    for (int jj = ksz >> 1; jj > 0; jj >>= 1) {
      for (int t = tid; t < P; t += 256) {
        const int x = t ^ jj;
        if (x > t) {
          const bool up = (t & ksz) == 0;
          const int a = s_src[t], b = s_src[x];
          if ((a > b) == up) {
            s_src[t] = b;
            s_src[x] = a;
            const float va = s_val[t];
            s_val[t] = s_val[x];
            s_val[x] = va;
          }
        }
      }
      __syncthreads();
    }
  for (int t = tid; t < L; t += 256) {
    src[t] = s_src[t];
    val[t] = s_val[t];
  }
}

// Lists of up to 256 in-edges (the common case: the mean in-degree equals k = 200): one WARP per
// list, 8 (source, weight) pairs per lane in registers, bitonic network with shuffles for partner
// distances < 32 and register swaps above — no block barriers, 8 lists per CTA.
__global__ __launch_bounds__(256) void in_sort_warp_kernel(const int32_t* __restrict__ in_ptr, int nn,
                                                           int k, int32_t* __restrict__ in_src,
                                                           float* __restrict__ in_w) {
  const int g = blockIdx.y, lane = threadIdx.x & 31;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (j >= nn) return;
  const int32_t* ptr = in_ptr + (int64_t)g * (nn + 1);
  const int lo = ptr[j], L = ptr[j + 1] - lo;
  if (L <= 1 || L > 256) return;
  int32_t* src = in_src + (int64_t)g * nn * k + lo;
  float* val = in_w + (int64_t)g * nn * k + lo;
  int key[8];
  float w[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {  // element t = 32 r + lane
    const int t = 32 * r + lane;
    key[r] = t < L ? src[t] : 0x7fffffff;
    w[r] = t < L ? val[t] : 0.f;
  }
#pragma unroll
  for (int ksz = 2; ksz <= 256; ksz <<= 1) {
#pragma unroll
    for (int jj = ksz >> 1; jj > 0; jj >>= 1) {
      if (jj >= 32) {
        const int dr = jj >> 5;  // partner = same lane, register r ^ dr
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const int pr = r ^ dr;
          if (pr > r) {
            const bool up = ((32 * r) & ksz) == 0;  // bits >= 5 of t come from r alone
            if ((key[r] > key[pr]) == up) {
              const int tk = key[r]; key[r] = key[pr]; key[pr] = tk;
              const float tw = w[r]; w[r] = w[pr]; w[pr] = tw;
            }
          }
        }
      } else {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const int t = 32 * r + lane;
          const int ok = __shfl_xor_sync(0xffffffffu, key[r], jj);
          const float ow = __shfl_xor_sync(0xffffffffu, w[r], jj);
          const bool up = (t & ksz) == 0;
          const bool lower = (lane & jj) == 0;  // this lane holds the lower index of the pair
          // ascending pair (up): lower index keeps the smaller key; descending: the larger
          const bool take = lower ? ((key[r] > ok) == up) : ((ok > key[r]) == up);
          if (take) {
            key[r] = ok;
            w[r] = ow;
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int t = 32 * r + lane;
    if (t < L) {
      src[t] = key[r];
      val[t] = w[r];
    }
  }
}

// --------------------------------------------------------------------------------------------
// Merged symmetric rows: W = A + A^T (models/mpti.py:752) stored once per row as (col u16, val)
// with the mutual pairs combined (W_ij = a_ij + a_ji, exactly the reference's sum).  Row i =
// its k out-edges in index order (mutual in-weights added in), then the non-mutual in-edges in
// source order.  One warp per row; each in-edge is looked up in the sorted out-list by bisection.
// Row segments are handed out with an atomic cursor: their placement may differ run to run, the
// contents (and so every sum taken over a row) do not.  A graph owns lp_rowcap(k) entries per node.
// --------------------------------------------------------------------------------------------
__global__ __launch_bounds__(256) void merge_rows_kernel(
    const int32_t* __restrict__ nbr, const float* __restrict__ sim,
    const int32_t* __restrict__ in_ptr, const int32_t* __restrict__ in_src,
    const float* __restrict__ in_w, const uint8_t* __restrict__ valid, int nn, int k,
    int32_t* __restrict__ cursor, int32_t* __restrict__ rowptr, int32_t* __restrict__ rowlen,
    uint16_t* __restrict__ mcol, float* __restrict__ mval) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  const int g = blockIdx.y, wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + wi;
  int* s_idx = reinterpret_cast<int*>(s_raw) + wi * k;
  float* s_val = reinterpret_cast<float*>(s_raw) + 8 * k + wi * k;
  if (i >= nn) return;
  const int64_t vb = (int64_t)g * nn;
  if (!valid[vb + i]) {
    if (lane == 0) {
      rowptr[vb + i] = 0;
      rowlen[vb + i] = 0;
    }
    return;
  }
  const int64_t ob = (vb + i) * k;
  for (int t = lane; t < k; t += 32) {
    s_idx[t] = nbr[ob + t];
    s_val[t] = sim[ob + t];
  }
  __syncwarp();
  const int32_t* ptr = in_ptr + (int64_t)g * (nn + 1);
  const int64_t ib = vb * k;
  const int e0 = ptr[i], e1 = ptr[i + 1];
  // pass 1: how many in-edges are not mutual
  int keep = 0;
  for (int t0 = e0; t0 < e1; t0 += 32) {
    const int t = t0 + lane;
    bool kp = false;
    if (t < e1) {
      const int s = in_src[ib + t];
      int lo = 0, hi = k;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (s_idx[mid] < s) lo = mid + 1; else hi = mid;
      }
      kp = !(lo < k && s_idx[lo] == s);
    }
    keep += __popc(__ballot_sync(0xffffffffu, kp));
  }
  const int total = k + keep;
  // segments are multiples of 4 entries (the solver reads a row as uint2 + float4 groups); the
  // pad entries are (column 0, weight 0) and lie beyond rowlen
  const int padded = (total + 3) & ~3;
  int start = 0;
  if (lane == 0) start = atomicAdd(&cursor[g], padded);
  start = __shfl_sync(0xffffffffu, start, 0);
  const int64_t mb = vb * lp_rowcap(k) + start;
  // pass 2: fold mutual in-weights into the out entries, append the rest
  int run = 0;
  for (int t0 = e0; t0 < e1; t0 += 32) {
    const int t = t0 + lane;
    bool kp = false;
    int s = 0;
    float wv = 0.f;
    if (t < e1) {
      s = in_src[ib + t];
      wv = in_w[ib + t];
      int lo = 0, hi = k;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (s_idx[mid] < s) lo = mid + 1; else hi = mid;
      }
      if (lo < k && s_idx[lo] == s) s_val[lo] += wv; else kp = true;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, kp);
    if (kp) {
      const int pos = k + run + __popc(bal & ((1u << lane) - 1));
      mcol[mb + pos] = (uint16_t)s;
      mval[mb + pos] = wv;
    }
    run += __popc(bal);
  }
  __syncwarp();
  for (int t = lane; t < k; t += 32) {
    mcol[mb + t] = (uint16_t)s_idx[t];
    mval[mb + t] = s_val[t];
  }
  if (lane < padded - total) {
    mcol[mb + total + lane] = 0;
    mval[mb + total + lane] = 0.f;
  }
  if (lane == 0) {
    rowptr[vb + i] = start;
    rowlen[vb + i] = total;
  }
}

// D = rowsum(W) ; D^-1/2 = sqrt(1 / (D + eps))      (models/mpti.py:767-770)
__global__ __launch_bounds__(256) void degree_merged_kernel(const int32_t* __restrict__ rowptr,
                                                            const int32_t* __restrict__ rowlen,
                                                            const float* __restrict__ mval, int nn,
                                                            int k, float* __restrict__ dinv) {
  const int g = blockIdx.y;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= nn) return;
  const int lane = threadIdx.x & 31;
  const int64_t vb = (int64_t)g * nn;
  const int L = rowlen[vb + i];
  float d = 0.f;
  if (L > 0) {
    const float* v = mval + vb * lp_rowcap(k) + rowptr[vb + i];
    for (int t = lane; t < L; t += 32) d += v[t];
    d = warp_sum(d);
    d = sqrtf(1.0f / (d + 2.220446049250313e-16f));
  }
  if (lane == 0) dinv[vb + i] = d;
}

// S = D^-1/2 W D^-1/2 on the stored pattern (models/mpti.py:772)
__global__ void normalize_merged_kernel(const int32_t* __restrict__ rowptr,
                                        const int32_t* __restrict__ rowlen,
                                        const uint16_t* __restrict__ mcol, float* __restrict__ mval,
                                        const float* __restrict__ dinv, int nn, int k) {
  const int g = blockIdx.y;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= nn) return;
  const int lane = threadIdx.x & 31;
  const int64_t vb = (int64_t)g * nn;
  const int L = rowlen[vb + i];
  const float* dg = dinv + vb;
  const float di = dg[i];
  const int64_t mb = vb * lp_rowcap(k) + rowptr[vb + i];
  for (int t = lane; t < L; t += 32) mval[mb + t] = (di * mval[mb + t]) * dg[mcol[mb + t]];
}

// --------------------------------------------------------------------------------------------
// Label propagation: (I - alpha S) Z = Y by conjugate gradients, all n_cls right-hand sides at
// once, one thread-block CLUSTER per graph (16 CTAs when the device grants it, else 8).
//   - rows are sliced over the cluster's CTAs; X, R, AP of a slice are private to its CTA;
//   - the search direction P is the only vector other CTAs read: it lives in global memory (L2),
//     and every CTA stages the whole of it (n x NCV floats) in shared memory once per iteration,
//     so the 2 x k x n gathers of the sparse product hit shared memory, not L2;
//   - the matrix (out-edge list + in-edge list) streams from L2 once per iteration;
//   - dot products are exchanged through distributed shared memory and summed in rank order, so
//     every CTA sees bit-identical scalars and the control flow stays cluster-uniform.
// --------------------------------------------------------------------------------------------
#define CG_THREADS 1024
#define CGC_MAXT 1024     // cluster kernel: up to 32 warps, ONE CTA per SM, one matrix row per thread
#define CG_CL_MAX 16
#define CG_MAXC 8
#define CG_MAXPASS 3      // matrix rows (or row segments) per thread -> at most 3072 per CTA
#define CG_SEGR 48        // residue ranks per row segment: 8 * 48 = 384 entries = 96 rounds
#define CG_MAXPART 1024   // segments of split rows a CTA can combine through shared memory
#define CG_TAB_HDR 4      // lo, hi, passes, segments of split rows
#define CG_TAB_INTS (CG_TAB_HDR + 32 * CG_MAXPASS * 2 + CG_MAXPASS * CGC_MAXT * 2)
#define CG_PK_SMEM (4096 * 4 + 8192 * 4 * 2)
#define CG_SMEM_MAX (200 * 1024)  // dynamic shared memory of lp_cg_kernel: P + split-row partials

struct CgExchange {
  float slot[2][CG_CL_MAX][CG_MAXC];
};

template <int NCV>
__device__ __forceinline__ void cg_allreduce(cg::cluster_group& cluster, CgExchange* ex,
                                             float* s_warp, const float* part, int& xcnt,
                                             float* total) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int rank = cluster.block_rank(), CL = cluster.num_blocks();
  const int n_warps = blockDim.x >> 5;
  float v[NCV];
#pragma unroll
  for (int c = 0; c < NCV; ++c) v[c] = warp_sum(part[c]);
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < NCV; ++c) s_warp[w * CG_MAXC + c] = v[c];
  }
  __syncthreads();
  const int par = xcnt & 1;
  if (tid < NCV) {
    float s = 0.f;
    for (int q = 0; q < n_warps; ++q) s += s_warp[q * CG_MAXC + tid];
    for (int r = 0; r < CL; ++r) {
      float* dst = cluster.map_shared_rank(&ex->slot[par][rank][tid], r);
      *dst = s;
    }
  }
  cluster.sync();
#pragma unroll
  for (int c = 0; c < NCV; ++c) {
    float s = 0.f;
    for (int r = 0; r < CL; ++r) s += ex->slot[par][r][c];
    total[c] = s;
  }
  ++xcnt;
}

// --------------------------------------------------------------------------------------------
// Packing for the cluster kernel below, once per solve.
//
// The product y = S p gathers one float4 of the shared-memory copy of p per matrix entry.  The
// first versions walked a row with a whole warp (entries in arbitrary order: 9.3 wavefronts per
// LDS.128 instead of 4, a shuffle reduction per row, ~130 instructions per 128 entries) and ran at
// one entry per clock per SM however the loads were arranged.  Here ONE THREAD OWNS ONE ROW:
//   * no reduction, ~35 instructions per 128 entries;
//   * the 32 rows of a warp are stored interleaved (lane-major groups of 4 entries: one uint2 of
//     columns + one float4 of weights per lane and round): a warp streams 768 contiguous bytes per
//     round;
//   * bank conflicts are designed out: the row owned by lane l is re-ordered so that its entry
//     number t has column residue (l + t) mod 8 — at every step the 8 lanes of a quarter-warp
//     gather from 8 different 16-byte bank groups.  Missing residues are padded with
//     (column (l + t) mod 8, weight 0), which adds 0 to the sum;
//   * row lengths range from 200 to 3 000 entries (hub prototypes), so a row is cut into SEGMENTS
//     of at most 384 entries (48 ranks of every residue); the segments of a split row are added
//     in order through shared memory.  Segments are sorted by length before they are dealt to the
//     threads, so the 32 segments of a warp are equally long, and the CTAs of a cluster own
//     contiguous row ranges with (almost) the same number of segments.
// A graph that does not fit its share of the scratch area (very skewed residues) is flagged and
// solved by the plain warp-per-row path of the kernel.
//   tab[(g * CL + rank)] = {lo, hi, passes, split segments} | slice[32 warps][CG_MAXPASS]{first
//   group, rounds} | thread[CG_MAXPASS][1024]{row - lo << 8 | segment, segments << 16 | part slot}
// --------------------------------------------------------------------------------------------
__global__ __launch_bounds__(256) void cg_hist_kernel(const int32_t* __restrict__ rowptr,
                                                      const int32_t* __restrict__ rowlen,
                                                      const uint8_t* __restrict__ valid,
                                                      const uint16_t* __restrict__ mcol, int nn,
                                                      int k, int32_t* __restrict__ rowmax) {
  const int g = blockIdx.y;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= nn) return;
  const int lane = threadIdx.x & 31;
  const int64_t vb = (int64_t)g * nn;
  int mx = 0;
  if (valid[vb + i]) {
    const int L = rowlen[vb + i];
    const uint16_t* c = mcol + vb * lp_rowcap(k) + rowptr[vb + i];
    int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int t0 = 0; t0 < L; t0 += 32) {
      const int t = t0 + lane;
      const int res = t < L ? (int)(c[t] & 7) : -1;
#pragma unroll
      for (int b = 0; b < 8; ++b) cnt[b] += __popc(__ballot_sync(0xffffffffu, res == b));
    }
#pragma unroll
    for (int b = 0; b < 8; ++b) mx = max(mx, cnt[b]);
  }
  if (lane == 0) rowmax[vb + i] = mx;  // largest residue class of the row (0: invalid node)
}

__global__ __launch_bounds__(1024) void cg_pack_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ rowlen,
    const int32_t* __restrict__ rowmax, const uint16_t* __restrict__ mcol,
    const float* __restrict__ mval, int nn, int k, int64_t pk_cap, int32_t* __restrict__ tab_all,
    int32_t* __restrict__ flags, uint2* __restrict__ pcol, float4* __restrict__ pval) {
  extern __shared__ __align__(16) unsigned char pk_smem[];
  uint32_t* s_key = reinterpret_cast<uint32_t*>(pk_smem);  // [4096] rounds << 21 | row - lo << 8 | seg
  int* s_pre = reinterpret_cast<int*>(s_key + 4096);       // [nn] segments before row i (whole graph)
  int* s_prx = s_pre + 8192;                               // [nn] segments of split rows before row i
  __shared__ int s_scan[2][32];
  __shared__ int s_tot[2];
  __shared__ int s_rng[2];
  __shared__ int s_wtot[32], s_wbase[32];
  const int CL = gridDim.x, rank = blockIdx.x, g = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t vb = (int64_t)g * nn;
  const int32_t* rp = rowptr + vb;
  const int32_t* rl = rowlen + vb;
  const int32_t* rmx = rowmax + vb;
  const uint16_t* mc = mcol + vb * lp_rowcap(k);
  const float* mv = mval + vb * lp_rowcap(k);
  int32_t* tab = tab_all + (size_t)(g * CL + rank) * CG_TAB_INTS;
  for (int e = tid; e < CG_TAB_HDR + 32 * CG_MAXPASS * 2; e += 1024) tab[e] = 0;
  // ---- segments per row, prefix over the whole graph (8 rows per thread, nn <= 8192)
  {
    int nseg[8], run = 0, runx = 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = tid * 8 + u;
      nseg[u] = i < nn ? (rmx[i] + CG_SEGR - 1) / CG_SEGR : 0;
      run += nseg[u];
      runx += nseg[u] > 1 ? nseg[u] : 0;
    }
    int inc = run, incx = runx;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int a = __shfl_up_sync(0xffffffffu, inc, o), ax = __shfl_up_sync(0xffffffffu, incx, o);
      if (lane >= o) {
        inc += a;
        incx += ax;
      }
    }
    if (lane == 31) {
      s_scan[0][w] = inc;
      s_scan[1][w] = incx;
    }
    __syncthreads();
    if (w == 0) {
      int v = s_scan[0][lane], vx = s_scan[1][lane];
      int i2 = v, ix2 = vx;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int a = __shfl_up_sync(0xffffffffu, i2, o), ax = __shfl_up_sync(0xffffffffu, ix2, o);
        if (lane >= o) {
          i2 += a;
          ix2 += ax;
        }
      }
      s_scan[0][lane] = i2 - v;
      s_scan[1][lane] = ix2 - vx;
      if (lane == 31) {
        s_tot[0] = i2;
        s_tot[1] = ix2;
      }
    }
    if (tid == 0) {
      s_rng[0] = nn;
      s_rng[1] = 0;
    }
    __syncthreads();
    int pre = s_scan[0][w] + inc - run, prex = s_scan[1][w] + incx - runx;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = tid * 8 + u;
      if (i < nn) {
        s_pre[i] = pre;
        s_prx[i] = prex;
      }
      pre += nseg[u];
      prex += nseg[u] > 1 ? nseg[u] : 0;
    }
  }
  __syncthreads();
  // ---- this CTA's contiguous row range: rows whose first segment falls into its share
  const int NV = s_tot[0];
  for (int i = tid; i < nn; i += 1024) {
    const int owner = NV > 0 ? min(CL - 1, (int)((int64_t)s_pre[i] * CL / NV)) : (i * CL) / nn;
    if (owner == rank) {
      atomicMin(&s_rng[0], i);
      atomicMax(&s_rng[1], i + 1);
    }
  }
  __syncthreads();
  const int lo = min(s_rng[0], s_rng[1]), hi = s_rng[1];
  const int pre_lo = lo < nn ? s_pre[lo] : NV, prx_lo = lo < nn ? s_prx[lo] : s_tot[1];
  const int nv = (hi < nn ? s_pre[hi] : NV) - pre_lo;           // segments of this CTA
  const int nx = (hi < nn ? s_prx[hi] : s_tot[1]) - prx_lo;    // ... of which belong to split rows
  const int passes = (nv + CGC_MAXT - 1) / CGC_MAXT;
  const int64_t share = pk_cap / CL;
  bool bad = passes > CG_MAXPASS || nx > CG_MAXPART || hi - lo > 8191;
  // ---- keys of the segments, sorted by length (descending)
  int npow = 32;
  while (npow < nv) npow <<= 1;
  if (!bad) {
    for (int i = tid; i < npow; i += 1024) s_key[i] = 0;
    __syncthreads();
    for (int i = lo + tid; i < hi; i += 1024) {
      const int mx = rmx[i];
      const int ns = (mx + CG_SEGR - 1) / CG_SEGR;
      if (ns > 255) bad = true;
      for (int sg = 0; sg < ns && sg < 256; ++sg) {
        const int ranks = min(CG_SEGR, mx - sg * CG_SEGR);
        s_key[s_pre[i] - pre_lo + sg] =
            ((uint32_t)(2 * ranks) << 21) | ((uint32_t)(i - lo) << 8) | (uint32_t)sg;
      }
    }
  }
  bad = __syncthreads_or(bad);
  if (!bad) {
    for (int ksz = 2; ksz <= npow; ksz <<= 1)
      for (int j = ksz >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < npow; i += 1024) {
          const int ixj = i ^ j;
          if (ixj > i) {
            const uint32_t x = s_key[i], y = s_key[ixj];
            const bool desc = (i & ksz) == 0;
            if (desc ? x < y : x > y) {
              s_key[i] = y;
              s_key[ixj] = x;
            }
          }
        }
        __syncthreads();
      }
    // slices: (pass, warp) holds sorted segments pass * 1024 + warp * 32 + lane; as long as its first
    if (tid < 32) {
      int tot = 0;
      for (int p = 0; p < passes; ++p) {
        const int i0 = p * CGC_MAXT + tid * 32;
        tot += i0 < nv ? (int)(s_key[i0] >> 21) * 32 : 0;
      }
      s_wtot[tid] = tot;
    }
    __syncthreads();
    if (tid == 0) {
      int run = 0;
      for (int q = 0; q < 32; ++q) {
        s_wbase[q] = run;
        run += s_wtot[q];
      }
      s_tot[0] = run;
    }
    __syncthreads();
    if (s_tot[0] > share) bad = true;
  }
  if (tid == 0) {
    tab[0] = lo;
    tab[1] = hi;
    tab[2] = bad ? 0 : passes;
    tab[3] = nx;
    if (bad) atomicOr(&flags[g], 1);
  }
  if (bad) return;
  // ---- per-thread table: which segment thread t works on in pass p
  for (int e = tid; e < CG_MAXPASS * CGC_MAXT; e += 1024) {
    const int p = e / CGC_MAXT, t = e % CGC_MAXT;
    const int i = p * CGC_MAXT + t;
    int m0 = -1, m1 = 0;
    if (p < passes && i < nv) {
      const uint32_t key = s_key[i];
      const int rloc = (int)((key >> 8) & 0x1fffu), sg = (int)(key & 0xffu);
      const int ns = (rmx[lo + rloc] + CG_SEGR - 1) / CG_SEGR;
      m0 = (rloc << 8) | sg;
      m1 = (ns << 16) | (ns > 1 ? s_prx[lo + rloc] - prx_lo : 0);
    }
    tab[CG_TAB_HDR + 32 * CG_MAXPASS * 2 + 2 * e + 0] = m0;
    tab[CG_TAB_HDR + 32 * CG_MAXPASS * 2 + 2 * e + 1] = m1;
  }
  // ---- every pack warp fills and scatters the slices of the consumer warp with its number
  uint2* gc = pcol + (int64_t)g * pk_cap + rank * share;
  float4* gv = pval + (int64_t)g * pk_cap + rank * share;
  int base = s_wbase[w];
  for (int p = 0; p < passes; ++p) {
    const int i0 = p * CGC_MAXT + w * 32;
    const int rounds = i0 < nv ? (int)(s_key[i0] >> 21) : 0;
    if (lane == 0) {
      tab[CG_TAB_HDR + (w * CG_MAXPASS + p) * 2 + 0] = (int)(rank * share) + base;
      tab[CG_TAB_HDR + (w * CG_MAXPASS + p) * 2 + 1] = rounds;
    }
    // pads everywhere first: entry t of lane l has column (l + t) mod 8 and weight 0
    for (int r = 0; r < rounds; ++r) {
      const unsigned t0 = (unsigned)(lane + 4 * r);
      uint2 c2;
      c2.x = (t0 & 7u) | (((t0 + 1) & 7u) << 16);
      c2.y = ((t0 + 2) & 7u) | (((t0 + 3) & 7u) << 16);
      gc[base + r * 32 + lane] = c2;
      gv[base + r * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();
    uint16_t* c16 = reinterpret_cast<uint16_t*>(gc + base);
    float* v32 = reinterpret_cast<float*>(gv + base);
    // metadata of the slice's 32 segments: lane l fetches segment l's, the loop broadcasts them
    int my_L = 0, my_ptr = 0, my_sg = 0;
    if (i0 + lane < nv) {
      const uint32_t key = s_key[i0 + lane];
      const int row = lo + (int)((key >> 8) & 0x1fffu);
      my_L = rl[row];
      my_ptr = rp[row];
      my_sg = (int)(key & 0xffu);
    }
    const int n_here = min(32, nv - i0);
    for (int l = 0; l < n_here; ++l) {  // the segment owned by lane l of the consumer warp
      const int L = __shfl_sync(0xffffffffu, my_L, l), sg = __shfl_sync(0xffffffffu, my_sg, l);
      const int ptr = __shfl_sync(0xffffffffu, my_ptr, l);
      const int r_lo = sg * CG_SEGR, r_hi = r_lo + CG_SEGR;  // ranks of every residue in this segment
      const uint16_t* c = mc + ptr;
      const float* v = mv + ptr;
      int seen[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      // one chunk of 32 entries ahead in flight
      int col_n = lane < L ? (int)c[lane] : -1;
      float val_n = lane < L ? v[lane] : 0.f;
      for (int t0 = 0; t0 < L; t0 += 32) {
        const int col = col_n;
        const float val = val_n;
        const int tn = t0 + 32 + lane;
        col_n = tn < L ? (int)c[tn] : -1;
        val_n = tn < L ? v[tn] : 0.f;
        const int res = col >= 0 ? (col & 7) : -1;
        int rho = -1;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const uint32_t m = __ballot_sync(0xffffffffu, res == b);
          if (res == b) rho = seen[b] + __popc(m & ((1u << lane) - 1));
          seen[b] += __popc(m);
        }
        if (rho >= r_lo && rho < r_hi) {
          const int step = 8 * (rho - r_lo) + ((res - l) & 7);  // residue (l + step) mod 8 == res
          const int64_t d = ((int64_t)(step >> 2) * 32 + l) * 4 + (step & 3);
          c16[d] = (uint16_t)col;
          v32[d] = val;
        }
        // every residue class is past this segment: the rest of the row belongs to later segments
        int done_all = 1;
#pragma unroll
        for (int b = 0; b < 8; ++b) done_all &= seen[b] >= r_hi;
        if (done_all) break;
      }
    }
    __syncwarp();
    base += rounds * 32;
  }
}

// Vectors are stored padded to NCV columns (NCV = 4 or 8) so a node's row is one or two float4.
template <int NCV>
__global__ __launch_bounds__(CGC_MAXT, 1) void lp_cg_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ rowlen,
    const uint16_t* __restrict__ mcol, const float* __restrict__ mval,
    const uint8_t* __restrict__ valid, int nn, int k,
    const float* __restrict__ Y, int nc, float alpha, float tol, int max_iter,
    float* __restrict__ Z, float* __restrict__ X, float* __restrict__ R, float* __restrict__ Pv,
    float* __restrict__ AP, int32_t* __restrict__ iters_out, float* __restrict__ resid_out,
    const int32_t* __restrict__ tab_all, const int32_t* __restrict__ flags,
    const uint2* __restrict__ pcol, const float4* __restrict__ pval, int64_t pk_cap) {
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = cluster.num_blocks(), rank = cluster.block_rank();
  const int g = blockIdx.y;
  extern __shared__ __align__(16) float Ps[];  // [nn][NCV] staged copy of P
  __shared__ CgExchange ex;
  __shared__ float s_warp[(CGC_MAXT / 32) * CG_MAXC];
  float* s_split = Ps + (size_t)nn * NCV;  // [CG_MAXPART][NCV] partial sums of split rows
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, T = blockDim.x;
  const int64_t vb = (int64_t)g * nn;
  const uint8_t* vg = valid + vb;
  const float* Yg = Y + vb * nc;
  float* Zg = Z + vb * nc;
  float* Xg = X + vb * NCV;
  float* Rg = R + vb * NCV;
  float* Pg = Pv + vb * NCV;
  float* APg = AP + vb * NCV;
  // this CTA's contiguous row range (cg_pack_kernel balanced the ranges by row segments)
  const int32_t* tab = tab_all + (size_t)(g * CL + rank) * CG_TAB_INTS;
  const int lo = tab[0], hi = tab[1];
  const int nloc = hi - lo;  // this CTA's rows: lo + j
  int xcnt = 0;

  float part[NCV], bb[NCV], rs[NCV], tot[NCV];
#pragma unroll
  for (int c = 0; c < NCV; ++c) part[c] = 0.f;
  for (int jj = tid; jj < nloc; jj += T) {
    const int row = lo + jj;
    const bool ok = vg[row];
#pragma unroll
    for (int c = 0; c < NCV; ++c) {
      const float y = (ok && c < nc) ? Yg[(int64_t)row * nc + c] : 0.f;
      Xg[(int64_t)row * NCV + c] = 0.f;
      Rg[(int64_t)row * NCV + c] = y;
      Pg[(int64_t)row * NCV + c] = y;
      APg[(int64_t)row * NCV + c] = 0.f;
      part[c] = fmaf(y, y, part[c]);
    }
  }
  cg_allreduce<NCV>(cluster, &ex, s_warp, part, xcnt, bb);
  bool done[NCV];
  bool all_done = true;
#pragma unroll
  for (int c = 0; c < NCV; ++c) {
    rs[c] = bb[c];
    done[c] = !(bb[c] > 0.f);
    all_done = all_done && done[c];
  }
  const float tol2 = tol * tol;
  // ---- this thread's row segments (cg_pack_kernel): one per pass
  const bool packed = flags[g] == 0;
  const int passes = packed ? tab[2] : 0;
  const bool any_split = packed && tab[3] > 0;
  // (the per-pass entries of the table are re-read from L1/L2 where they are used: keeping them in
  // registers for the whole solve spills at the 64-register cap of a 1024-thread CTA)
  const int32_t* t_slice = tab + CG_TAB_HDR + w * CG_MAXPASS * 2;
  const int32_t* t_thread = tab + CG_TAB_HDR + 32 * CG_MAXPASS * 2 + 2 * tid;
  const uint2* gc = pcol + (int64_t)g * pk_cap;
  const float4* gv = pval + (int64_t)g * pk_cap;
  int it = 0;
  while (!all_done && it < max_iter) {
    // ---- stage P (written by every CTA of the cluster, published by the last cluster.sync)
    {
      const float4* src = reinterpret_cast<const float4*>(Pg);
      float4* dst = reinterpret_cast<float4*>(Ps);
      const int n4 = nn * (NCV / 4);
      for (int i = tid; i < n4; i += T) dst[i] = __ldcg(src + i);
    }
    __syncthreads();
    // ---- AP = P - alpha * S P  on my rows; partial P.AP
#pragma unroll
    for (int c = 0; c < NCV; ++c) part[c] = 0.f;
    if (packed) {
      constexpr unsigned SH = NCV == 4 ? 4 : 5;  // node -> byte offset of its row of P
      const unsigned char* Pb = reinterpret_cast<const unsigned char*>(Ps);
#pragma unroll
      for (int p = 0; p < passes; ++p) {
        const int rounds = __ldg(t_slice + 2 * p + 1);
        if (rounds == 0) continue;  // warp-uniform
        const int sbase = __ldg(t_slice + 2 * p);
        const uint2* c2 = gc + sbase + lane;
        const float4* v4 = gv + sbase + lane;
        float acc[NCV];
#pragma unroll
        for (int c = 0; c < NCV; ++c) acc[c] = 0.f;
        auto fma4 = [&](float wgt, unsigned byte_off) {
#pragma unroll
          for (int q = 0; q < NCV / 4; ++q) {
            const float4 p4 = *reinterpret_cast<const float4*>(Pb + byte_off + 16 * q);
            acc[4 * q + 0] = fmaf(wgt, p4.x, acc[4 * q + 0]);
            acc[4 * q + 1] = fmaf(wgt, p4.y, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(wgt, p4.z, acc[4 * q + 2]);
            acc[4 * q + 3] = fmaf(wgt, p4.w, acc[4 * q + 3]);
          }
        };
        auto consume = [&](const uint2& c, const float4& v) {
          fma4(v.x, (c.x & 0xffffu) << SH);
          fma4(v.y, (c.x >> 16) << SH);
          fma4(v.z, (c.y & 0xffffu) << SH);
          fma4(v.w, (c.y >> 16) << SH);
        };
        // rounds is even (padded lengths are multiples of 8): two rounds in flight, two consumed
        uint2 ca = __ldcs(c2), cb = __ldcs(c2 + 32);
        float4 va = __ldcs(v4), vb4 = __ldcs(v4 + 32);
        for (int r = 2; r < rounds; r += 2) {
          const uint2 na = __ldcs(c2 + r * 32), nb = __ldcs(c2 + r * 32 + 32);
          const float4 wa = __ldcs(v4 + r * 32), wb = __ldcs(v4 + r * 32 + 32);
          consume(ca, va);
          consume(cb, vb4);
          ca = na;
          cb = nb;
          va = wa;
          vb4 = wb;
        }
        consume(ca, va);
        consume(cb, vb4);
        const int m0 = __ldg(t_thread + 2 * p * CGC_MAXT), m1 = __ldg(t_thread + 2 * p * CGC_MAXT + 1);
        if (m0 >= 0) {
          if ((m1 >> 16) == 1) {  // a whole row: done
            const int row = lo + (m0 >> 8);
#pragma unroll
            for (int c = 0; c < NCV; ++c) {
              const float pv = Ps[(size_t)row * NCV + c];
              const float ap = pv - alpha * acc[c];
              APg[(int64_t)row * NCV + c] = ap;
              part[c] = fmaf(pv, ap, part[c]);
            }
          } else {  // a segment of a split row: parked in shared memory, added in order below
            float* dst = s_split + (size_t)((m1 & 0xffff) + (m0 & 0xff)) * NCV;
#pragma unroll
            for (int c = 0; c < NCV; ++c) dst[c] = acc[c];
          }
        }
      }
      if (any_split) {  // CTA-uniform
        __syncthreads();
        for (int p = 0; p < passes; ++p) {
          const int m0 = __ldg(t_thread + 2 * p * CGC_MAXT), m1 = __ldg(t_thread + 2 * p * CGC_MAXT + 1);
          if (m0 >= 0 && (m1 >> 16) > 1 && (m0 & 0xff) == 0) {  // owner of segment 0
            const int row = lo + (m0 >> 8), ns = m1 >> 16;
            const float* src = s_split + (size_t)(m1 & 0xffff) * NCV;
#pragma unroll
            for (int c = 0; c < NCV; ++c) {
              float sum = 0.f;
              for (int sg = 0; sg < ns; ++sg) sum += src[sg * NCV + c];
              const float pv = Ps[(size_t)row * NCV + c];
              const float ap = pv - alpha * sum;
              APg[(int64_t)row * NCV + c] = ap;
              part[c] = fmaf(pv, ap, part[c]);
            }
          }
        }
      }
    } else {
      // plain path (a graph whose packed rows did not fit): a warp per row over the merged lists
      const int32_t* rp = rowptr + vb;
      const int32_t* rl = rowlen + vb;
      const uint16_t* mc = mcol + vb * lp_rowcap(k);
      const float* mv = mval + vb * lp_rowcap(k);
      for (int row = lo + w; row < hi; row += T >> 5) {
        if (!vg[row]) continue;
        float acc[NCV];
#pragma unroll
        for (int c = 0; c < NCV; ++c) acc[c] = 0.f;
        const int L = rl[row];
        const uint16_t* crow = mc + rp[row];
        const float* vrow = mv + rp[row];
        for (int t = lane; t < L; t += 32) {
          const int cj = (int)crow[t];
          const float cv = vrow[t];
#pragma unroll
          for (int c = 0; c < NCV; ++c) acc[c] = fmaf(cv, Ps[(size_t)cj * NCV + c], acc[c]);
        }
#pragma unroll
        for (int c = 0; c < NCV; ++c) {
          const float sum = warp_sum(acc[c]);
          const float pv = Ps[(size_t)row * NCV + c];
          const float ap = pv - alpha * sum;
          if (lane == 0) {
            APg[(int64_t)row * NCV + c] = ap;
            part[c] = fmaf(pv, ap, part[c]);
          }
        }
      }
    }
    cg_allreduce<NCV>(cluster, &ex, s_warp, part, xcnt, tot);
    float a[NCV];
#pragma unroll
    for (int c = 0; c < NCV; ++c) a[c] = (!done[c] && tot[c] > 0.f) ? rs[c] / tot[c] : 0.f;
    // ---- X += a P ; R -= a AP ; partial R.R      (own rows; P from the staged copy)
#pragma unroll
    for (int c = 0; c < NCV; ++c) part[c] = 0.f;
    for (int jj = tid; jj < nloc; jj += T) {
      const int row = lo + jj;
#pragma unroll
      for (int c = 0; c < NCV; ++c) {
        const int64_t o = (int64_t)row * NCV + c;
        const float r = Rg[o] - a[c] * APg[o];
        Xg[o] = fmaf(a[c], Ps[o], Xg[o]);
        Rg[o] = r;
        part[c] = fmaf(r, r, part[c]);
      }
    }
    cg_allreduce<NCV>(cluster, &ex, s_warp, part, xcnt, tot);
    float beta[NCV];
    all_done = true;
#pragma unroll
    for (int c = 0; c < NCV; ++c) {
      beta[c] = (!done[c] && rs[c] > 0.f) ? tot[c] / rs[c] : 0.f;
      if (!done[c]) {
        rs[c] = tot[c];
        if (tot[c] <= tol2 * bb[c]) done[c] = true;
      }
      all_done = all_done && done[c];
    }
    // ---- P = R + beta P   (frozen for finished columns)
    for (int jj = tid; jj < nloc; jj += T) {
      const int row = lo + jj;
#pragma unroll
      for (int c = 0; c < NCV; ++c)
        if (!done[c]) {
          const int64_t o = (int64_t)row * NCV + c;
          Pg[o] = fmaf(beta[c], Ps[o], Rg[o]);
        }
    }
    ++it;
    cluster.sync();  // publish P (and make sure nobody still reads Ps before it is restaged)
  }
  // Z (unpadded) from my rows
  for (int jj = tid; jj < nloc; jj += T) {
    const int row = lo + jj;
    for (int c = 0; c < nc; ++c) Zg[(int64_t)row * nc + c] = Xg[(int64_t)row * NCV + c];
  }
  if (rank == 0 && tid == 0) {
    if (iters_out) iters_out[g] = it;
    if (resid_out) {
      float m = 0.f;
#pragma unroll
      for (int c = 0; c < NCV; ++c)
        if (bb[c] > 0.f) m = fmaxf(m, sqrtf(rs[c] / bb[c]));
      resid_out[g] = m;
    }
  }
  cluster.sync();
}

template <int NCV>
static int launch_cg(int CL, int G, size_t smem, cudaStream_t st, const int32_t* rowptr,
                     const int32_t* rowlen, const uint16_t* mcol, const float* mval,
                     const uint8_t* valid, int nn, int k, const float* Y, int nc,
                     float alpha, float tol, int max_iter, float* Z, float* X, float* R, float* P,
                     float* AP, int32_t* iters_out, float* resid_out, void* scratch,
                     size_t scratch_bytes) {
  cudaError_t e = cudaFuncSetAttribute(lp_cg_kernel<NCV>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, CG_SMEM_MAX);
  if (e != cudaSuccess) return (int)e;
  if (CL > 8) {
    e = cudaFuncSetAttribute(lp_cg_kernel<NCV>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return (int)e;
  }
  const int T = CGC_MAXT;
  smem += sizeof(float) * (size_t)CG_MAXPART * NCV;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CL, G, 1);
  cfg.blockDim = dim3(T, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  {  // can the device co-schedule a cluster of this size at all?
    int n_clusters = 0;
    e = cudaOccupancyMaxActiveClusters(&n_clusters, lp_cg_kernel<NCV>, &cfg);
    if (e != cudaSuccess || n_clusters < 1) {
      (void)cudaGetLastError();
      return -1000;
    }
  }
  // scratch: per-CTA tables | per-graph flags + row maxima | packed columns | packed weights
  const int64_t pk_cap = lp_pack_groups(nn, k);  // groups of 4 entries per graph
  const size_t tab_bytes = align_up(sizeof(int32_t) * (size_t)G * CL * CG_TAB_INTS, 256);
  const size_t flg_bytes = align_up(sizeof(int32_t) * (size_t)G * (1 + nn), 256);
  const size_t col_bytes = align_up(sizeof(uint2) * (size_t)G * pk_cap, 256);
  const size_t val_bytes = align_up(sizeof(float4) * (size_t)G * pk_cap, 256);
  if (!scratch || scratch_bytes < tab_bytes + flg_bytes + col_bytes + val_bytes)
    return R3DFS_E_WORKSPACE;
  unsigned char* sp = reinterpret_cast<unsigned char*>(scratch);
  int32_t* tab = reinterpret_cast<int32_t*>(sp);
  int32_t* flags = reinterpret_cast<int32_t*>(sp + tab_bytes);
  uint2* pcol = reinterpret_cast<uint2*>(sp + tab_bytes + flg_bytes);
  float4* pval = reinterpret_cast<float4*>(sp + tab_bytes + flg_bytes + col_bytes);
  e = cudaMemsetAsync(flags, 0, sizeof(int32_t) * (size_t)G, st);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(cg_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CG_PK_SMEM);
  if (e != cudaSuccess) return (int)e;
  int32_t* rowmax = flags + G;
  cg_hist_kernel<<<dim3((nn + 7) / 8, G), 256, 0, st>>>(rowptr, rowlen, valid, mcol, nn, k, rowmax);
  R3DFS_CHECK_LAUNCH();
  cg_pack_kernel<<<dim3(CL, G), 1024, CG_PK_SMEM, st>>>(rowptr, rowlen, rowmax, mcol, mval, nn, k,
                                                       pk_cap, tab, flags, pcol, pval);
  R3DFS_CHECK_LAUNCH();
  const int32_t* tabc = tab;
  const int32_t* flc = flags;
  const uint2* pc = pcol;
  const float4* pv = pval;
  e = cudaLaunchKernelEx(&cfg, lp_cg_kernel<NCV>, rowptr, rowlen, mcol, mval, valid, nn, k, Y, nc,
                         alpha, tol, max_iter, Z, X, R, P, AP, iters_out, resid_out, tabc, flc, pc,
                         pv, pk_cap);
  if (e != cudaSuccess) return (int)e;
  ++r3dfs_launches;
  return 0;
}

// --------------------------------------------------------------------------------------------
// Same solve, matrix resident in SHARED memory.  The grid is one CTA per SM, cut into groups of GS
// CTAs; a group solves one graph at a time (graphs group, group + n_groups, ...).  A CTA owns a
// slice of the rows and copies their (col, val) lists into its shared memory once — with 37 CTAs
// per 4416-node graph that is ~190 KB per CTA, so the 60-odd sparse products of the solve never
// touch L2/HBM again (the cluster kernel streams ~7 MB per graph per iteration and is bound by
// exactly that).  Rows that do not fit stay in global memory and are streamed as before.
//   - x, r, Ap of the slice live in shared memory; only P goes through global memory (each CTA
//     publishes its rows, all CTAs restage the whole vector);
//   - CTAs of a group meet at a counter barrier in global memory (co-residency comes from the
//     cooperative launch); dot products go through per-CTA slots and are summed in rank order by
//     every CTA, so all CTAs see bit-identical scalars and the control flow stays group-uniform.
// --------------------------------------------------------------------------------------------
#define GCG_SLOT 8  // floats per CTA slot
#define GCG_MAX_GS 160

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void group_barrier(unsigned* cnt, unsigned& target, int GS) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += (unsigned)GS;
    __threadfence();
    atomicAdd(cnt, 1u);
    while (ld_acquire_u32(cnt) < target) {
    }
    __threadfence();
  }
  __syncthreads();
}

// sum of every thread's part[] over the CTA -> slot of this CTA; barrier; total over the group
template <int NCV>
__device__ __forceinline__ void group_allreduce(float* s_warp, float* s_slot, const float* part,
                                                float* slots, int rank, int GS, unsigned* cnt,
                                                unsigned& target, int& phase, float* total) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  float v[NCV];
#pragma unroll
  for (int c = 0; c < NCV; ++c) v[c] = warp_sum(part[c]);
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < NCV; ++c) s_warp[w * CG_MAXC + c] = v[c];
  }
  __syncthreads();
  float* my = slots + ((size_t)(phase & 1) * GS + rank) * GCG_SLOT;
  if (tid < NCV) {
    float s = 0.f;
    for (int q = 0; q < CG_THREADS / 32; ++q) s += s_warp[q * CG_MAXC + tid];
    __stcg(my + tid, s);
  }
  group_barrier(cnt, target, GS);
  // one L2 round trip: thread r fetches CTA r's slot, then everybody sums the copies in rank order
  const float* all = slots + (size_t)(phase & 1) * GS * GCG_SLOT;
  if (tid < GS) {
#pragma unroll
    for (int q = 0; q < NCV / 4; ++q)
      reinterpret_cast<float4*>(s_slot + tid * GCG_SLOT)[q] =
          __ldcg(reinterpret_cast<const float4*>(all + (size_t)tid * GCG_SLOT) + q);
  }
  __syncthreads();
#pragma unroll
  for (int c = 0; c < NCV; ++c) total[c] = 0.f;
  for (int r = 0; r < GS; ++r) {
#pragma unroll
    for (int q = 0; q < NCV / 4; ++q) {
      const float4 t4 = reinterpret_cast<const float4*>(s_slot + r * GCG_SLOT)[q];
      total[4 * q + 0] += t4.x;
      total[4 * q + 1] += t4.y;
      total[4 * q + 2] += t4.z;
      total[4 * q + 3] += t4.w;
    }
  }
  ++phase;
}

template <int NCV, bool SMEM>
__device__ __forceinline__ void cg_row_product(const uint16_t* crow, const float* vrow, int L,
                                               int lane, const float* Ps, float* acc) {
  int t0 = 0;
  for (; t0 + 256 <= L; t0 += 256) {
    int cj[8];
    float cv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int t = t0 + lane + 32 * u;
      cj[u] = (int)crow[t];
      cv[u] = vrow[t];
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
#pragma unroll
      for (int q = 0; q < NCV / 4; ++q) {
        const float4 p4 = *reinterpret_cast<const float4*>(Ps + (int64_t)cj[u] * NCV + 4 * q);
        acc[4 * q + 0] = fmaf(cv[u], p4.x, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(cv[u], p4.y, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(cv[u], p4.z, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(cv[u], p4.w, acc[4 * q + 3]);
      }
    }
  }
  // remainder in ONE predicated round: a warp owns only a couple of rows per iteration here, so the
  // 32-entry steps of a row are a latency chain (in the batched cluster kernel, where 16 warps keep
  // the memory system busy, the same change cost 5 %: there the extra predicated work is what shows)
  if (t0 < L) {
    const int nU = (L - t0 + 31) >> 5;
    int cj[8];
    float cv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int t = t0 + lane + 32 * u;
      const bool ok = u < nU && t < L;
      cj[u] = ok ? (int)crow[t] : 0;
      cv[u] = ok ? vrow[t] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (u < nU) {
#pragma unroll
        for (int q = 0; q < NCV / 4; ++q) {
          const float4 p4 = *reinterpret_cast<const float4*>(Ps + (int64_t)cj[u] * NCV + 4 * q);
          acc[4 * q + 0] = fmaf(cv[u], p4.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(cv[u], p4.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(cv[u], p4.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(cv[u], p4.w, acc[4 * q + 3]);
        }
      }
    }
  }
}

template <int NCV>
__global__ __launch_bounds__(CG_THREADS, 1) void lp_cg_group_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ rowlen,
    const uint16_t* __restrict__ mcol, const float* __restrict__ mval,
    const uint8_t* __restrict__ valid, int G, int nn, int k, const float* __restrict__ Y, int nc,
    float alpha, float tol, int max_iter, float* __restrict__ Z, float* __restrict__ Pv,
    unsigned* __restrict__ counters, float* __restrict__ slots_all, int GS, int rows_max,
    int cache_entries, int32_t* __restrict__ iters_out, float* __restrict__ resid_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // [Ps nn*NCV f32][xs rows_max*NCV][rs rows_max*NCV][aps rows_max*NCV][off rows_max i32]
  // [vals cache_entries f32][cols cache_entries u16]
  float* Ps = reinterpret_cast<float*>(smem_raw);
  float* xs = Ps + (size_t)nn * NCV;
  float* rsm = xs + (size_t)rows_max * NCV;
  float* aps = rsm + (size_t)rows_max * NCV;
  int* s_off = reinterpret_cast<int*>(aps + (size_t)rows_max * NCV);
  float* c_val = reinterpret_cast<float*>(s_off + rows_max);
  uint16_t* c_col = reinterpret_cast<uint16_t*>(c_val + cache_entries);
  __shared__ float s_warp[(CG_THREADS / 32) * CG_MAXC];
  __shared__ __align__(16) float s_slot[GCG_MAX_GS * GCG_SLOT];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int group = blockIdx.x / GS, rank = blockIdx.x % GS, n_groups = gridDim.x / GS;
  if (group >= n_groups) return;  // leftover CTAs (grid not a multiple of GS)
  unsigned* cnt = counters + group * 32;  // one counter per 128-byte line
  float* slots = slots_all + (size_t)group * 2 * GS * GCG_SLOT;
  unsigned target = 0;
  int phase = 0;
  const int chunk = (nn + GS - 1) / GS;
  const int lo = min(nn, rank * chunk), hi = min(nn, lo + chunk);
  const int nrows = hi - lo;
  const float tol2 = tol * tol;

  for (int g = group; g < G; g += n_groups) {
    const int64_t vb = (int64_t)g * nn;
    const uint8_t* vg = valid + vb;
    const float* Yg = Y + vb * nc;
    float* Zg = Z + vb * nc;
    float* Pg = Pv + vb * NCV;
    const int32_t* rp = rowptr + vb;
    const int32_t* rl = rowlen + vb;
    const uint16_t* mc = mcol + vb * lp_rowcap(k);
    const float* mv = mval + vb * lp_rowcap(k);
    // ---- cache my rows' lists: offsets by one warp's scan, then a cooperative copy
    if (w == 0) {
      int base = 0;
      for (int r0 = 0; r0 < nrows; r0 += 32) {
        const int r = r0 + lane;
        const int L = (r < nrows && vg[lo + r]) ? rl[lo + r] : 0;
        int incl = L;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int a = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += a;
        }
        const int off = base + incl - L;
        if (r < nrows) s_off[r] = (off + L <= cache_entries) ? off : -1;
        base += __shfl_sync(0xffffffffu, incl, 31);
      }
    }
    __syncthreads();
    for (int r = w; r < nrows; r += CG_THREADS / 32) {
      const int off = s_off[r];
      if (off < 0 || !vg[lo + r]) continue;
      const int L = rl[lo + r];
      const uint16_t* crow = mc + rp[lo + r];
      const float* vrow = mv + rp[lo + r];
      for (int t = lane; t < L; t += 32) {
        c_col[off + t] = crow[t];
        c_val[off + t] = vrow[t];
      }
    }
    // ---- x = 0, r = p = y
    float part[NCV], bb[NCV], rs[NCV], tot[NCV];
#pragma unroll
    for (int c = 0; c < NCV; ++c) part[c] = 0.f;
    for (int r = tid; r < nrows; r += CG_THREADS) {
      const int row = lo + r;
      const bool ok = vg[row];
      float y[NCV];
#pragma unroll
      for (int c = 0; c < NCV; ++c) {
        y[c] = (ok && c < nc) ? Yg[(int64_t)row * nc + c] : 0.f;
        xs[r * NCV + c] = 0.f;
        rsm[r * NCV + c] = y[c];
        aps[r * NCV + c] = 0.f;
        part[c] = fmaf(y[c], y[c], part[c]);
      }
#pragma unroll
      for (int q = 0; q < NCV / 4; ++q)
        __stcg(reinterpret_cast<float4*>(Pg + (int64_t)row * NCV) + q,
               make_float4(y[4 * q], y[4 * q + 1], y[4 * q + 2], y[4 * q + 3]));
    }
    group_allreduce<NCV>(s_warp, s_slot, part, slots, rank, GS, cnt, target, phase, bb);  // publishes P too
    bool done[NCV];
    bool all_done = true;
#pragma unroll
    for (int c = 0; c < NCV; ++c) {
      rs[c] = bb[c];
      done[c] = !(bb[c] > 0.f);
      all_done = all_done && done[c];
    }
    int it = 0;
    while (!all_done && it < max_iter) {
      {  // stage P
        const float4* src = reinterpret_cast<const float4*>(Pg);
        float4* dst = reinterpret_cast<float4*>(Ps);
        const int n4 = nn * (NCV / 4);
        for (int i4 = tid; i4 < n4; i4 += CG_THREADS) dst[i4] = __ldcg(src + i4);
      }
      __syncthreads();
#pragma unroll
      for (int c = 0; c < NCV; ++c) part[c] = 0.f;
      for (int r = w; r < nrows; r += CG_THREADS / 32) {
        const int row = lo + r;
        if (!vg[row]) continue;
        float acc[NCV];
#pragma unroll
        for (int c = 0; c < NCV; ++c) acc[c] = 0.f;
        const int L = rl[row];
        const int off = s_off[r];
        if (off >= 0)
          cg_row_product<NCV, true>(c_col + off, c_val + off, L, lane, Ps, acc);
        else
          cg_row_product<NCV, false>(mc + rp[row], mv + rp[row], L, lane, Ps, acc);
#pragma unroll
        for (int c = 0; c < NCV; ++c) {
          const float s = warp_sum(acc[c]);
          const float p = Ps[(int64_t)row * NCV + c];
          const float ap = p - alpha * s;
          if (lane == 0) {
            aps[r * NCV + c] = ap;
            part[c] = fmaf(p, ap, part[c]);
          }
        }
      }
      group_allreduce<NCV>(s_warp, s_slot, part, slots, rank, GS, cnt, target, phase, tot);
      float a[NCV];
#pragma unroll
      for (int c = 0; c < NCV; ++c) a[c] = (!done[c] && tot[c] > 0.f) ? rs[c] / tot[c] : 0.f;
#pragma unroll
      for (int c = 0; c < NCV; ++c) part[c] = 0.f;
      for (int r = tid; r < nrows; r += CG_THREADS) {
#pragma unroll
        for (int c = 0; c < NCV; ++c) {
          const int o = r * NCV + c;
          const float rr = rsm[o] - a[c] * aps[o];
          xs[o] = fmaf(a[c], Ps[(int64_t)(lo + r) * NCV + c], xs[o]);
          rsm[o] = rr;
          part[c] = fmaf(rr, rr, part[c]);
        }
      }
      group_allreduce<NCV>(s_warp, s_slot, part, slots, rank, GS, cnt, target, phase, tot);
      float beta[NCV];
      all_done = true;
#pragma unroll
      for (int c = 0; c < NCV; ++c) {
        beta[c] = (!done[c] && rs[c] > 0.f) ? tot[c] / rs[c] : 0.f;
        if (!done[c]) {
          rs[c] = tot[c];
          if (tot[c] <= tol2 * bb[c]) done[c] = true;
        }
        all_done = all_done && done[c];
      }
      ++it;
      if (all_done || it >= max_iter) break;  // group-uniform: nobody needs the next P
      for (int r = tid; r < nrows; r += CG_THREADS) {
        const int row = lo + r;
        float pn[NCV];
#pragma unroll
        for (int c = 0; c < NCV; ++c) {
          const float pold = Ps[(int64_t)row * NCV + c];
          pn[c] = done[c] ? pold : fmaf(beta[c], pold, rsm[r * NCV + c]);
        }
#pragma unroll
        for (int q = 0; q < NCV / 4; ++q)
          __stcg(reinterpret_cast<float4*>(Pg + (int64_t)row * NCV) + q,
                 make_float4(pn[4 * q], pn[4 * q + 1], pn[4 * q + 2], pn[4 * q + 3]));
      }
      group_barrier(cnt, target, GS);  // publish P
    }
    for (int r = tid; r < nrows; r += CG_THREADS)
      for (int c = 0; c < nc; ++c) Zg[(int64_t)(lo + r) * nc + c] = xs[r * NCV + c];
    if (rank == 0 && tid == 0) {
      if (iters_out) iters_out[g] = it;
      if (resid_out) {
        float m = 0.f;
#pragma unroll
        for (int c = 0; c < NCV; ++c)
          if (bb[c] > 0.f) m = fmaxf(m, sqrtf(rs[c] / bb[c]));
        resid_out[g] = m;
      }
    }
    __syncthreads();  // the slice buffers are reused by the next graph
  }
}

// scratch (global): 32 counters lines + slots; taken from the AP buffer the cluster kernel uses
template <int NCV>
static int launch_cg_group(int G, cudaStream_t st, const int32_t* rowptr, const int32_t* rowlen,
                           const uint16_t* mcol, const float* mval, const uint8_t* valid, int nn,
                           int k, const float* Y, int nc, float alpha, float tol, int max_iter,
                           float* Z, float* P, float* scratch, size_t scratch_floats,
                           int32_t* iters_out, float* resid_out) {
  static int n_sm = 0, coop = 0, smem_max = 0;
  if (n_sm == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  }
  if (!coop || n_sm < 8) return -1000;
  // CTAs per graph: as few as keep (almost) the whole matrix in shared memory, so that as many
  // graphs as possible are in flight; never more groups than graphs
  // measured on the single graph of a training step (4416 nodes): 74 CTAs beat 37, 110 and 148 —
  // more CTAs shorten the row slices but every CTA restages the whole of P and joins every barrier
  const int n_groups = min(G, 4);
  const int GS = min(GCG_MAX_GS, min(74, n_sm / n_groups));
  const int rows_max = (nn + GS - 1) / GS;
  const size_t fixed = sizeof(float) * ((size_t)nn * NCV + 3 * (size_t)rows_max * NCV) +
                       sizeof(int) * (size_t)rows_max;
  const size_t smem = (size_t)smem_max - 8 * 1024;  // minus the kernel's static shared memory
  if (fixed + 6 * 1024 > smem) return -1000;
  const int cache_entries = (int)(((smem - fixed) / 6) & ~(size_t)7);
  const size_t need_scratch = 32 * 32 + (size_t)n_groups * 2 * GS * GCG_SLOT;
  if (need_scratch > scratch_floats) return -1000;
  cudaError_t e = cudaFuncSetAttribute(lp_cg_group_kernel<NCV>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemsetAsync(scratch, 0, 32 * 32 * sizeof(unsigned), st);
  if (e != cudaSuccess) return (int)e;
  unsigned* counters = reinterpret_cast<unsigned*>(scratch);
  float* slots = scratch + 32 * 32;
  int grid = n_groups * GS;
  void* args[] = {(void*)&rowptr, (void*)&rowlen, (void*)&mcol, (void*)&mval, (void*)&valid,
                  (void*)&G, (void*)&nn, (void*)&k, (void*)&Y, (void*)&nc, (void*)&alpha,
                  (void*)&tol, (void*)&max_iter, (void*)&Z, (void*)&P, (void*)&counters,
                  (void*)&slots, (void*)&GS, (void*)&rows_max, (void*)&cache_entries,
                  (void*)&iters_out, (void*)&resid_out};
  e = cudaLaunchCooperativeKernel((const void*)lp_cg_group_kernel<NCV>, dim3(grid), dim3(CG_THREADS),
                                  args, smem, st);
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return -1000;
  }
  ++r3dfs_launches;
  return 0;
}

// --------------------------------------------------------------------------------------------
// Query rows of Z -> logits, argmax prediction (models/mpti_learner.py:98) and the mean
// cross-entropy (models/mpti.py:571).  One CTA per episode, fixed-order reduction.
// --------------------------------------------------------------------------------------------
__global__ __launch_bounds__(1024) void query_head_kernel(const float* __restrict__ Z, int nn,
                                                          int q_off, int nq, int nc,
                                                          const int64_t* __restrict__ qy,
                                                          float* __restrict__ logits,
                                                          float* __restrict__ loss,
                                                          int32_t* __restrict__ pred) {
  __shared__ float s_red[32];
  const int g = blockIdx.x, tid = threadIdx.x;
  const float* Zg = Z + ((int64_t)g * nn + q_off) * nc;
  float part = 0.f;
  for (int i = tid; i < nq; i += 1024) {
    float mx = -INFINITY;
    int am = 0;
    for (int c = 0; c < nc; ++c) {
      const float v = Zg[(int64_t)i * nc + c];
      logits[((int64_t)g * nq + i) * nc + c] = v;
      if (v > mx) {
        mx = v;
        am = c;
      }
    }
    if (pred) pred[(int64_t)g * nq + i] = am;
    if (qy) {
      float se = 0.f;
      for (int c = 0; c < nc; ++c) se += expf(Zg[(int64_t)i * nc + c] - mx);
      const int y = (int)qy[(int64_t)g * nq + i];
      part += (mx + logf(se)) - Zg[(int64_t)i * nc + y];
    }
  }
  part = warp_sum(part);
  if ((tid & 31) == 0) s_red[tid >> 5] = part;
  __syncthreads();
  if (tid == 0 && loss) {
    float s = 0.f;
    for (int q = 0; q < 32; ++q) s += s_red[q];
    loss[g] = qy ? s / (float)nq : 0.f;
  }
}

// evaluate_metric counters (reference eval_noise.py:43-62)
__global__ void confusion_kernel(const int32_t* __restrict__ pred, const int64_t* __restrict__ gt,
                                 const int32_t* __restrict__ class_slot, int n_way,
                                 int64_t pts_per_episode, int64_t total, int n_slots,
                                 unsigned long long* __restrict__ counters) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t ep = e / pts_per_episode;
  const int g = (int)gt[e], p = pred[e];
  const int gi = g == 0 ? 0 : class_slot[ep * n_way + g - 1];
  const int pi = p == 0 ? 0 : class_slot[ep * n_way + p - 1];
  atomicAdd(&counters[gi], 1ull);
  atomicAdd(&counters[n_slots + pi], 1ull);
  if (g == p) atomicAdd(&counters[2 * n_slots + gi], 1ull);
}

// --------------------------------------------------------------------------------------------
// launchers
// --------------------------------------------------------------------------------------------
// The bounded select pays where a row's candidates fit the warp's buffer with room to spare.  Were
// the row's columns in random order, a group's minimum would lie below distance quantile p with
// probability 1 - (1 - p)^AFF_GROUP; the k-th smallest minimum sits where that equals k / groups,
// and about nn p columns lie below it.  That count must be at most half the buffer.  Rows that
// still overflow take the exact fallback.
static bool bounded_select_pays(int nn, int k) {
  const double groups = (nn + AFF_GROUP - 1) / AFF_GROUP;
  if (groups <= k) return false;
  return nn * (1.0 - pow(1.0 - k / groups, 1.0 / AFF_GROUP)) <= SELB_CAP / 2;
}

int launch_affinity(const float* F, int64_t graph_rows, int64_t row_off, const uint8_t* valid,
                    int G, int nn, int D, int k, float sigma, float* norms, float* D2,
                    unsigned* gmin, int32_t* nbr, float* sim, cudaStream_t st,
                    const StageRec* sr) {
  if (D % 4 != 0 || D > 32 * LP_MAX_F4 || k > 1024 || nn > 65535) return R3DFS_E_UNSUPPORTED;
  R3DFS_TRY(launch_row_norms_batched(F + row_off * D, graph_rows * D, G, nn, D, D, norms, st));
  // Squared-L2 matrix in Gram form (what faiss.IndexFlatL2 ranks by, models/mpti.py:733-735):
  // the TMEM-operand kernel (linear_ts_kernel<128, true>), which also writes the group minima that
  // bound the select; the register-fed one, without bounds, when TMA cannot address the feature
  // matrix, or under R3DFS_DIST_TC=1 in the measurement build
  static const bool sel_block = R3DFS_GETENV("R3DFS_SELECT_BLOCK") != nullptr;
  if (sel_block || !bounded_select_pays(nn, k) || nn % 4 != 0 ||
      (reinterpret_cast<uintptr_t>(valid) & 3) != 0)
    gmin = nullptr;
  static const bool dist_tc = R3DFS_GETENV("R3DFS_DIST_TC") != nullptr;
  int rc = dist_tc ? R3DFS_E_UNSUPPORTED
                   : launch_gram_dist_ts(F, graph_rows, row_off, G, nn, D, norms, D2, valid, gmin,
                                         st);
  if (rc == R3DFS_E_UNSUPPORTED) {
    gmin = nullptr;
    rc = launch_gram_dist_tc(F, graph_rows, row_off, G, nn, D, norms, D2, st);
  }
  R3DFS_TRY(rc);
  if (sr) sr->mark(R3DFS_ST_DIST, st);
  if (gmin) {
    knn_select_bounded_kernel<<<dim3((nn + SELB_WARPS - 1) / SELB_WARPS, G), SELB_WARPS * 32, 0,
                                st>>>(D2, valid, gmin, nn, k, nbr);
    R3DFS_CHECK_LAUNCH();
  } else if (nn <= 32 * 80 && !sel_block) {
    const dim3 gs((nn + SELW_WARPS - 1) / SELW_WARPS, G);
    if (nn <= 32 * 40)
      knn_select_warp_kernel<40><<<gs, SELW_WARPS * 32, 0, st>>>(D2, valid, nn, k, nbr);
    else
      knn_select_warp_kernel<80><<<gs, SELW_WARPS * 32, 0, st>>>(D2, valid, nn, k, nbr);
    R3DFS_CHECK_LAUNCH();
  } else if (nn <= 31 * SEL_THREADS && !sel_block) {
    const size_t smem = sizeof(unsigned) * (size_t)nn;  // <= 31 KB
    if (nn <= 19 * SEL_THREADS)
      knn_select_reg_kernel<20><<<dim3(nn, G), SEL_THREADS, smem, st>>>(D2, valid, nn, k, nbr);
    else  // 512 threads keep 20 keys per thread and 1024 threads per SM in flight (32 keys per
          // thread on 256 threads: half the occupancy)
      knn_select_reg_kernel<20, 512><<<dim3(nn, G), 512, smem, st>>>(D2, valid, nn, k, nbr);
    R3DFS_CHECK_LAUNCH();
  } else {
    size_t smem = sizeof(unsigned) * (size_t)nn;
    cudaError_t e = cudaFuncSetAttribute(knn_select_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    knn_select_kernel<<<dim3(nn, G), SEL_THREADS, smem, st>>>(D2, valid, nn, k, nbr);
    R3DFS_CHECK_LAUNCH();
  }
  if (sr) sr->mark(R3DFS_ST_SELECT, st);
  const dim3 gs((nn + 7) / 8, G);
  if ((reinterpret_cast<uintptr_t>(F) & 15) == 0)
    edge_sim_kernel<true><<<gs, 256, 0, st>>>(F, graph_rows, row_off, nn, D, valid, nbr, k, sigma,
                                              sim);
  else  // a feature matrix TMA could not address either (the register-fed GEMM ran)
    edge_sim_kernel<false><<<gs, 256, 0, st>>>(F, graph_rows, row_off, nn, D, valid, nbr, k, sigma,
                                               sim);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_SIM, st);
  return 0;
}

// Every CTA of lp_cg_kernel stages the whole of P (nn x NCV floats) and the partial sums of up to
// CG_MAXPART split-row segments (CG_MAXPART x NCV floats) in its CG_SMEM_MAX bytes of dynamic shared
// memory; cg_pack_kernel's row prefix and the 16-bit merged columns cap any graph at 8192 nodes.
// NCV = 4 (n_cls <= 4): 8192 nodes; NCV = 8 (n_cls 5..8): 204800 / 32 - 1024 = 5376 nodes.
int lp_max_nodes(int n_cls) {
  if (n_cls < 1 || n_cls > CG_MAXC) return 0;
  const int ncv = n_cls <= 4 ? 4 : 8;
  const int fit = (int)(CG_SMEM_MAX / (sizeof(float) * ncv)) - CG_MAXPART;
  return fit < 8192 ? fit : 8192;
}

// (I - alpha S) X = RHS on merged rows that are already built and normalised (the label-propagation
// solve itself, and its adjoint in the training backward: S is symmetric).
int launch_lp_solve(const int32_t* rowptr, const int32_t* rowlen, const uint16_t* mcol,
                    const float* mval, const uint8_t* valid, int G, int nn, int k, const float* Y,
                    int nc, float alpha, float tol, int max_iter, float* Z, float* X, float* R,
                    float* P, float* AP, int32_t* iters_out, float* resid_out, cudaStream_t st,
                    bool latency, void* scratch, size_t scratch_bytes) {
  if (nc > CG_MAXC || nc < 1 || nn > 8192) return R3DFS_E_UNSUPPORTED;
  // padded vector width: one or two float4 per node
  const int ncv = nc <= 4 ? 4 : 8;
  const size_t smem_cg = sizeof(float) * (size_t)nn * ncv;
  if (smem_cg > CG_SMEM_MAX) return R3DFS_E_UNSUPPORTED;
  int rc = -1000;
  if (latency) {  // matrix resident in shared memory, groups of CTAs (cooperative launch)
    const size_t scratch_floats = (size_t)G * nn * ncv;
    rc = ncv == 4 ? launch_cg_group<4>(G, st, rowptr, rowlen, mcol, mval, valid, nn, k, Y, nc, alpha,
                                       tol, max_iter, Z, P, AP, scratch_floats, iters_out, resid_out)
                  : launch_cg_group<8>(G, st, rowptr, rowlen, mcol, mval, valid, nn, k, Y, nc, alpha,
                                       tol, max_iter, Z, P, AP, scratch_floats, iters_out, resid_out);
    if (rc == 0) return 0;
    if (rc != -1000) return rc;
  }
  if (nn > lp_max_nodes(nc)) return R3DFS_E_UNSUPPORTED;  // the cluster solve's limit
  // One CTA per SM (the kernel keeps a queue of matrix rounds in 128 registers per thread), so a
  // batch of graphs gets as many CTAs per graph as keep ALL graphs in flight in one wave (25 graphs
  // on 148 SMs: clusters of 5); a handful of graphs gets 16.  A warp keeps the metadata of at most
  // 32 * CG_MJ rows in registers, which bounds the rows of a CTA from above.
  int dev = 0, n_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  const int rows_cta_max = CGC_MAXT * CG_MAXPASS;
  const int cl_need = (nn + rows_cta_max - 1) / rows_cta_max;
  const int cl_start = max(G <= 4 ? 16 : max(1, min(8, n_sm / G)), cl_need);
  for (int CL = cl_start; CL >= cl_need && CL >= 1 && rc == -1000;
       CL = (CL & (CL - 1)) ? (1 << (31 - __builtin_clz(CL))) : CL >> 1) {
    if (ncv == 4)
      rc = launch_cg<4>(CL, G, smem_cg, st, rowptr, rowlen, mcol, mval, valid, nn, k, Y, nc, alpha,
                        tol, max_iter, Z, X, R, P, AP, iters_out, resid_out, scratch, scratch_bytes);
    else
      rc = launch_cg<8>(CL, G, smem_cg, st, rowptr, rowlen, mcol, mval, valid, nn, k, Y, nc, alpha,
                        tol, max_iter, Z, X, R, P, AP, iters_out, resid_out, scratch, scratch_bytes);
  }
  if (rc != 0) return rc == -1000 ? R3DFS_E_UNSUPPORTED : rc;
  return 0;
}

int launch_label_propagate(const int32_t* nbr, float* sim, const uint8_t* valid, int G, int nn,
                           int k, const float* Y, int nc, float alpha, float tol, int max_iter,
                           int32_t* in_cnt, int32_t* in_ptr, int32_t* in_src, float* in_w,
                           float* dinv, int32_t* rowptr, int32_t* rowlen, int32_t* cursor,
                           uint16_t* mcol, float* mval, float* Z, float* X, float* R, float* P,
                           float* AP, int32_t* iters_out, float* resid_out, cudaStream_t st,
                           const StageRec* sr, void* scratch, size_t scratch_bytes, bool latency,
                           void* dense_scratch, int32_t* dense_info) {
  if (nc > CG_MAXC || nc < 1 || nn > 8192) return R3DFS_E_UNSUPPORTED;
  cudaError_t e;
  const int64_t edges = (int64_t)nn * k;
  dim3 ge((unsigned)((edges + 255) / 256), G);
  const int W = (nn + 31) / 32;
  const size_t bits_bytes = sizeof(uint32_t) * (size_t)G * nn * W;
  const size_t pre_bytes = sizeof(uint16_t) * (size_t)G * nn * W;
  static const bool force_sort = R3DFS_GETENV("R3DFS_INEDGE_SORT") != nullptr;
  if (scratch && scratch_bytes >= bits_bytes + pre_bytes && !force_sort) {
    // sort-free: bit matrix of the transposed adjacency -> ranks -> ordered fill
    uint32_t* bits = reinterpret_cast<uint32_t*>(scratch);
    uint16_t* pre = reinterpret_cast<uint16_t*>(reinterpret_cast<unsigned char*>(scratch) + bits_bytes);
    e = cudaMemsetAsync(bits, 0, bits_bytes, st);
    if (e != cudaSuccess) return (int)e;
    in_bits_kernel<<<ge, 256, 0, st>>>(nbr, valid, nn, k, W, bits);
    R3DFS_CHECK_LAUNCH();
    in_rank_kernel<<<dim3((nn + 7) / 8, G), 256, 0, st>>>(bits, nn, W, pre, in_cnt);
    R3DFS_CHECK_LAUNCH();
    in_scan_kernel<<<G, 1024, 0, st>>>(in_cnt, nn, in_ptr);
    R3DFS_CHECK_LAUNCH();
    in_fill_rank_kernel<<<ge, 256, 0, st>>>(nbr, sim, valid, nn, k, W, bits, pre, in_ptr, in_src,
                                            in_w);
    R3DFS_CHECK_LAUNCH();
  } else {
    e = cudaMemsetAsync(in_cnt, 0, sizeof(int32_t) * (size_t)G * nn, st);
    if (e != cudaSuccess) return (int)e;
    in_count_kernel<<<ge, 256, 0, st>>>(nbr, valid, nn, k, in_cnt);
    R3DFS_CHECK_LAUNCH();
    in_scan_kernel<<<G, 1024, 0, st>>>(in_cnt, nn, in_ptr);
    R3DFS_CHECK_LAUNCH();
    in_fill_kernel<<<ge, 256, 0, st>>>(nbr, sim, valid, nn, k, in_ptr, in_cnt, in_src, in_w);
    R3DFS_CHECK_LAUNCH();
    e = cudaFuncSetAttribute(in_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 8192);
    if (e != cudaSuccess) return (int)e;
    in_sort_warp_kernel<<<dim3((nn + 7) / 8, G), 256, 0, st>>>(in_ptr, nn, k, in_src, in_w);
    R3DFS_CHECK_LAUNCH();
    in_sort_kernel<<<dim3(nn, G), 256, 8 * 1024, st>>>(in_ptr, nn, k, in_src, in_w, 256, 1024);
    R3DFS_CHECK_LAUNCH();
    in_sort_kernel<<<dim3(nn, G), 256, 8 * 8192, st>>>(in_ptr, nn, k, in_src, in_w, 1024, 8192);
    R3DFS_CHECK_LAUNCH();
  }
  dim3 gr((nn + 7) / 8, G);
  e = cudaMemsetAsync(cursor, 0, sizeof(int32_t) * (size_t)G, st);
  if (e != cudaSuccess) return (int)e;
  const size_t smem_m = (size_t)8 * k * 8;
  e = cudaFuncSetAttribute(merge_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           (int)smem_m);
  if (e != cudaSuccess) return (int)e;
  merge_rows_kernel<<<gr, 256, smem_m, st>>>(nbr, sim, in_ptr, in_src, in_w, valid, nn, k, cursor,
                                            rowptr, rowlen, mcol, mval);
  R3DFS_CHECK_LAUNCH();
  degree_merged_kernel<<<gr, 256, 0, st>>>(rowptr, rowlen, mval, nn, k, dinv);
  R3DFS_CHECK_LAUNCH();
  normalize_merged_kernel<<<gr, 256, 0, st>>>(rowptr, rowlen, mcol, mval, dinv, nn, k);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_SYM, st);

  if (dense_scratch) {
    R3DFS_TRY(launch_lp_cholesky_solve(rowptr, rowlen, mcol, mval, valid, G, nn, k, Y, nc, alpha, Z,
                                       dense_scratch, dense_info, st));
    if (sr) sr->mark(R3DFS_ST_CG, st);
    return 0;
  }
  // the in-edge scratch (bit matrix, ranks) is dead by now: the solver re-uses it
  R3DFS_TRY(launch_lp_solve(rowptr, rowlen, mcol, mval, valid, G, nn, k, Y, nc, alpha, tol, max_iter,
                            Z, X, R, P, AP, iters_out, resid_out, st, latency, scratch,
                            scratch_bytes));
  if (sr) sr->mark(R3DFS_ST_CG, st);
  return 0;
}

int launch_query_head(const float* Z, int G, int nn, int q_off, int nq, int nc, const int64_t* qy,
                      float* logits, float* loss, int32_t* pred, cudaStream_t st) {
  query_head_kernel<<<G, 1024, 0, st>>>(Z, nn, q_off, nq, nc, qy, logits, loss, pred);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int launch_confusion(const int32_t* pred, const int64_t* gt, const int32_t* class_slot, int E,
                     int n_way, int64_t pts, int n_slots, int64_t* counters, cudaStream_t st) {
  const int64_t total = (int64_t)E * pts;
  confusion_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
      pred, gt, class_slot, n_way, pts, total, n_slots,
      reinterpret_cast<unsigned long long*>(counters));
  R3DFS_CHECK_LAUNCH();
  return 0;
}
