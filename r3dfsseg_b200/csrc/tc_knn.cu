// knn on the tensor cores: the pairwise-distance GEMM (3xTF32, tcgen05.mma, accumulators in TMEM)
// feeds a per-row top-k selection that reads the accumulator straight out of TMEM — the (N, N)
// matrix never exists in shared or global memory  (reference models/dgcnn.py:17-23).
//
// One CTA = 128 query points of one cloud, warp-specialised:
//   warps 4-7  load 128-candidate tiles (global -> TF32 hi/lo split -> K-major UMMA tiles in shared
//              memory, 2 stages); one of their threads issues the MMAs into one of two TMEM
//              accumulator buffers and commits to an mbarrier;
//   warps 0-3  own one TMEM lane (= query row) per thread: tcgen05.ld 32 columns at a time, form
//              the reference's ranking key, queue the candidates that beat the row's current k-th
//              best, then merge the queue into a sorted k-list kept in registers.
// While the selectors work on tile j the tensor core computes tile j+1 and the loaders fetch j+2.
#include <stdlib.h>

#include "common.cuh"
#include "tc.cuh"

#define KT_TQ 128
#define KT_TC 128
#define KT_THREADS 384  // warps 0-7 selectors (2 per TMEM lane quarter), warps 8-11 loaders

template <int KC4>
struct KnnTcSmem {
  static constexpr int TILE = tc::tile_bytes(128, KC4);  // one of hi / lo
  static constexpr int Q_OFF = 0;                        // Q hi, Q lo
  static constexpr int B_OFF = 2 * TILE;                 // 2 stages x (hi, lo)
  static constexpr int QV_OFF = B_OFF + 4 * TILE;        // queue values  [16][256] float
  static constexpr int QI_OFF = QV_OFF + 16 * 256 * 4;   // queue columns [16][256] uint8
  static constexpr int XS_OFF = QI_OFF + 16 * 256;       // |x_j|^2 of 4 tiles in flight [4][128]
  static constexpr int TOTAL = XS_OFF + 4 * 128 * 4 + 64;  // (the queue is reused for the final merge)
};

template <int KC4>
__device__ __forceinline__ void knn_store_tile(unsigned char* hi_base, unsigned char* lo_base,
                                               const float* __restrict__ x, int ld, int C,
                                               int64_t row0, int64_t rows_end, int t, int nthr,
                                               bool vec_ok) {
  constexpr int LBO = tc::tile_lbo(128);
  constexpr int CH = 128 * KC4;
  // a warp covers 32/KC4' rows x chunks; chunk index fastest so global reads are contiguous
  for (int c = t; c < CH; c += nthr) {
    const int r = c / KC4, kc = c % KC4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t row = row0 + r;
    const int k = 4 * kc;
    if (row < rows_end && k < C) {
      const float* p = x + row * (int64_t)ld + k;
      if (vec_ok && k + 3 < C) {
        v = *reinterpret_cast<const float4*>(p);
      } else {
        v.x = p[0];
        if (k + 1 < C) v.y = p[1];
        if (k + 2 < C) v.z = p[2];
        if (k + 3 < C) v.w = p[3];
      }
    }
    float4 hi, lo;
    tc::split4(v, hi, lo);
    *reinterpret_cast<float4*>(hi_base + kc * LBO + r * 16) = hi;
    *reinterpret_cast<float4*>(lo_base + kc * LBO + r * 16) = lo;
  }
}

// Candidate-tile loader split in two so that a thread's global loads of the NEXT tile are all in
// flight while the current tile is converted and the MMAs are issued (the straight loop above
// serialises one L2 round trip per 16-byte chunk, which is what used to bound the whole kernel).
template <int KC4, int ROWS, int NTHR>
struct TileRegs {
  static constexpr int NCH = ROWS * KC4 / NTHR;
  float4 v[NCH];
};

template <int KC4, int ROWS, int NTHR>
__device__ __forceinline__ void tile_load(TileRegs<KC4, ROWS, NTHR>& tr, const float* __restrict__ x,
                                          int ld, int C, int64_t row0, int64_t rows_end, int t,
                                          bool vec_ok) {
#pragma unroll
  for (int i = 0; i < TileRegs<KC4, ROWS, NTHR>::NCH; ++i) {
    const int c = t + i * NTHR;
    const int r = c / KC4, kc = c % KC4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t row = row0 + r;
    const int k = 4 * kc;
    if (row < rows_end && k < C) {
      const float* p = x + row * (int64_t)ld + k;
      if (vec_ok && k + 3 < C) {
        v = __ldg(reinterpret_cast<const float4*>(p));
      } else {
        v.x = __ldg(p);
        if (k + 1 < C) v.y = __ldg(p + 1);
        if (k + 2 < C) v.z = __ldg(p + 2);
        if (k + 3 < C) v.w = __ldg(p + 3);
      }
    }
    tr.v[i] = v;
  }
}

template <int KC4, int ROWS, int NTHR>
__device__ __forceinline__ void tile_store(const TileRegs<KC4, ROWS, NTHR>& tr,
                                           unsigned char* hi_base, unsigned char* lo_base, int t) {
  constexpr int LBO = tc::tile_lbo(ROWS);
#pragma unroll
  for (int i = 0; i < TileRegs<KC4, ROWS, NTHR>::NCH; ++i) {
    const int c = t + i * NTHR;
    const int r = c / KC4, kc = c % KC4;
    float4 hi, lo;
    tc::split4(tr.v[i], hi, lo);
    *reinterpret_cast<float4*>(hi_base + kc * LBO + r * 16) = hi;
    *reinterpret_cast<float4*>(lo_base + kc * LBO + r * 16) = lo;
  }
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}

// sorted (descending) insertion into a register-resident k-list; c[i] = key > lv[i]
template <int KL>
__device__ __forceinline__ void list_insert(float (&lv)[KL], int (&li)[KL], float key, int idx) {
#pragma unroll
  for (int i = KL - 1; i > 0; --i) {
    const bool up = key > lv[i - 1];  // everything from i-1 on moves down one slot
    const bool here = key > lv[i];
    const float nv = up ? lv[i - 1] : (here ? key : lv[i]);
    const int ni = up ? li[i - 1] : (here ? idx : li[i]);
    lv[i] = nv;
    li[i] = ni;
  }
  if (key > lv[0]) {
    lv[0] = key;
    li[0] = idx;
  }
}

template <int KC4, int KL>
__global__ __launch_bounds__(KT_THREADS, 1) void knn_tc_kernel(const float* __restrict__ x, int ld,
                                                               int C, const float* __restrict__ xx,
                                                               int N, int k,
                                                               int32_t* __restrict__ idx32,
                                                               int64_t* __restrict__ idx64) {
  extern __shared__ __align__(128) unsigned char smem[];
  using S = KnnTcSmem<KC4>;
  __shared__ uint64_t bar_full[2];   // accumulator buffer b ready (= MMAs of its tile complete)
  __shared__ uint64_t bar_tfree[2];  // accumulator buffer b drained by the 128 selector threads
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int b = blockIdx.y;
  const int q0 = blockIdx.x * KT_TQ;
  const int64_t base = (int64_t)b * N;
  constexpr int LBO = tc::tile_lbo(128);
  constexpr uint32_t IDESC = tc::make_idesc_tf32(128, KT_TC);
  const bool vec_ok = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  const int T = (N + KT_TC - 1) / KT_TC;
  const int ksteps = (min(C, 4 * KC4) + 7) / 8;

  if (tid == 0) {
    tc::mbar_init(&bar_full[0], 1);
    tc::mbar_init(&bar_full[1], 1);
    tc::mbar_init(&bar_tfree[0], 256);
    tc::mbar_init(&bar_tfree[1], 256);
    tc::mbar_fence_init();
  }
  if (w == 0) tc::tmem_alloc(&tmem_base_s, 2 * KT_TC);
  // query tile (all threads)
  knn_store_tile<KC4>(smem + S::Q_OFF, smem + S::Q_OFF + S::TILE, x, ld, C, base + q0, base + N,
                      tid, KT_THREADS, vec_ok);
  tc::fence_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  if (w >= 8) {
    // ------------------------------ loaders + MMA issue -------------------------------------
    const int lt = tid - 256;
    TileRegs<KC4, 128, 128> tr;
    float* xs = reinterpret_cast<float*>(smem + S::XS_OFF);
    tile_load(tr, x, ld, C, base, base + N, lt, vec_ok);
    float xn = lt < N ? __ldg(xx + base + lt) : 0.f;
    for (int j = 0; j < T; ++j) {
      const int st = j & 1;
      if (j >= 2) tc::mbar_wait(&bar_full[st], ((j >> 1) - 1) & 1);  // stage's previous MMAs done
      unsigned char* hi = smem + S::B_OFF + st * 2 * S::TILE;
      unsigned char* lo = hi + S::TILE;
      tile_store(tr, hi, lo, lt);
      // the tile's |x_j|^2 travel with it (ring of 4: slot j is rewritten by tile j + 4, whose
      // loaders have waited for MMA j + 2, which was issued after the selectors released tile j)
      xs[(j & 3) * KT_TC + lt] = xn;
      if (j + 1 < T) {
        tile_load(tr, x, ld, C, base + (int64_t)(j + 1) * KT_TC, base + N, lt, vec_ok);
        const int cn_ = (j + 1) * KT_TC + lt;
        xn = cn_ < N ? __ldg(xx + base + cn_) : 0.f;
      }
      tc::fence_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (lt == 0) {
        if (j >= 2) tc::mbar_wait(&bar_tfree[st], ((j >> 1) - 1) & 1);  // buffer drained
        tc::tc_fence_after();
        const uint32_t q_hi = tc::smem_u32(smem + S::Q_OFF), q_lo = q_hi + S::TILE;
        const uint32_t b_hi = tc::smem_u32(hi), b_lo = b_hi + S::TILE;
        const uint32_t d = tmem_d + st * KT_TC;
        // one descriptor per operand tile; k-step ks is a constant added to its address field
        const uint64_t dqh = tc::make_desc(q_hi, LBO, 128), dql = tc::make_desc(q_lo, LBO, 128);
        const uint64_t dbh = tc::make_desc(b_hi, LBO, 128), dbl = tc::make_desc(b_lo, LBO, 128);
        constexpr uint64_t KS = tc::desc_kstep(LBO);
        tc::mma_tf32_c<false>(d, dql, dbh, IDESC);
        tc::mma_tf32_c<true>(d, dqh, dbl, IDESC);
        tc::mma_tf32_c<true>(d, dqh, dbh, IDESC);
#pragma unroll
        for (int ks = 1; ks < 2 * KC4 / 4; ++ks) {
          if (ks < ksteps) {
            tc::mma_tf32_c<true>(d, dql + ks * KS, dbh + ks * KS, IDESC);
            tc::mma_tf32_c<true>(d, dqh + ks * KS, dbl + ks * KS, IDESC);
            tc::mma_tf32_c<true>(d, dqh + ks * KS, dbh + ks * KS, IDESC);
          }
        }
        tc::mma_commit(&bar_full[st]);
      }
    }
  } else {
    // ------------------------------ selectors ------------------------------------------------
    // thread = (query row, column half): warps w and w+4 share TMEM lane quarter w%4; warp w < 4
    // scans columns 0..63 of every tile, warp w >= 4 columns 64..127; the two partial k-lists of a
    // row are merged through shared memory at the end.
    float* qv = reinterpret_cast<float*>(smem + S::QV_OFF);
    unsigned char* qi = smem + S::QI_OFF;
    const int row = 32 * (w & 3) + lane;
    const int half = w >> 2;
    const int q = q0 + row;
    const float nq = (q < N) ? -xx[base + q] : 0.f;
    const float* xs = reinterpret_cast<const float*>(smem + S::XS_OFF);
    float lv[KL];
    int li[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) {
      lv[i] = -INFINITY;
      li[i] = 0;
    }
    for (int j = 0; j < T; ++j) {
      const int st = j & 1;
      tc::mbar_wait(&bar_full[st], (j >> 1) & 1);
      tc::tc_fence_after();
      const int c0 = j * KT_TC;
#pragma unroll 1
      for (int cc = 64 * half; cc < 64 * half + 64; cc += 32) {
        float v[32];
        tc::tmem_ld32(tmem_d + ((uint32_t)(32 * (w & 3)) << 16) + (uint32_t)(st * KT_TC + cc), v);
        // 16 columns at a time: queue what beats the current k-th best, then merge the queue
#pragma unroll
        for (int hh = 0; hh < 32; hh += 16) {
          const float thr = lv[KL - 1];
          int cnt = 0;
#pragma unroll
          for (int u = hh; u < hh + 16; u += 4) {
            const int cg = c0 + cc + u;
            const float4 cn = *reinterpret_cast<const float4*>(xs + (j & 3) * KT_TC + cc + u);
            const float cnv[4] = {cn.x, cn.y, cn.z, cn.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              // reference key: -xx_i - (-2 x_i.x_j) - xx_j
              const float key = fmaf(2.f, v[u + e], nq) - cnv[e];  // = (nq - (-2 v)) - cn exactly
              if (key > thr && cg + e < N) {
                qv[cnt * 256 + tid] = key;
                qi[cnt * 256 + tid] = (unsigned char)(cc + u + e);
                ++cnt;
              }
            }
          }
          const int mx = __reduce_max_sync(0xffffffffu, cnt);
          for (int e = 0; e < mx; ++e) {
            if (e < cnt) {
              const float key = qv[e * 256 + tid];
              if (key > lv[KL - 1]) list_insert<KL>(lv, li, key, c0 + (int)qi[e * 256 + tid]);
            }
          }
        }
      }
      tc::tc_fence_before();
      mbar_arrive(&bar_tfree[st]);
    }
    // merge: the upper-half warps publish their lists, the lower-half warps absorb them
    int* mi = reinterpret_cast<int*>(smem + S::B_OFF);  // loaders are done with the B stages by now
    asm volatile("bar.sync 2, 256;" ::: "memory");      // every selector has consumed its last tile
    if (half == 1) {
#pragma unroll
      for (int i = 0; i < KL; ++i) {
        qv[i * 128 + row] = lv[i];
        mi[i * 128 + row] = li[i];
      }
    }
    asm volatile("bar.sync 2, 256;" ::: "memory");
    if (half == 0) {
#pragma unroll 1
      for (int i = 0; i < KL; ++i) {
        const float key = qv[i * 128 + row];
        if (key > lv[KL - 1]) list_insert<KL>(lv, li, key, mi[i * 128 + row]);
      }
      if (q < N) {
#pragma unroll
        for (int i = 0; i < KL; ++i) {
          if (i < k) {
            const int64_t o = (base + q) * k + i;
            if (idx32) idx32[o] = li[i];
            if (idx64) idx64[o] = li[i];
          }
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (w == 0) tc::tmem_dealloc(tmem_d, 2 * KT_TC);
}


// ---------------------------------------------------------------------------------------------
// Two-pass variant (k <= 20, 1024 <= N <= 65535): the per-row selection above pays one
// warp-divergent 120-instruction list insertion for each of the ~k (1 + ln(N / k)) candidates that
// beat a running threshold.  Here the distance GEMM runs TWICE (it is cheap: the tensor pipe idles
// otherwise) and the first pass only produces a tight, exact lower bound of every row's k-th best
// key:  the row's candidates are cut into 64 groups, the k-th largest of the 64 group maxima is
// <= the k-th largest key, and only ~k (1 + 1/3) keys lie above it.  The second pass recomputes the
// keys (bit-identical), appends the few that reach the bound to a per-thread queue in shared
// memory, and the 20-lists are built once at the end, all lanes inserting together.
//   candidate tiles are 64 wide here (two 33 KB operand stages instead of 66 KB) to make room for
//   the queues; warps 0-7 = (TMEM lane quarter, 32-column half), warps 8-11 loaders + MMA issue.
// ---------------------------------------------------------------------------------------------
#define K2_TC 64
#define K2_CAP 56  // queue entries per selector thread; drained when fewer than 32 slots remain
#define K2_G 32    // group maxima per selector thread (64 per row)
#define K2_THREADS 416  // warps 0-7 selectors, 8-11 loaders, 12 MMA issue

template <int KC4>
struct Knn2Smem {
  static constexpr int TQ = tc::tile_bytes(128, KC4);
  static constexpr int TB = tc::tile_bytes(K2_TC, KC4);
  static constexpr int Q_OFF = 0;                            // Q hi, Q lo
  static constexpr int B_OFF = 2 * TQ;                       // 2 stages x (hi, lo)
  static constexpr int QK_OFF = B_OFF + 4 * TB;              // queue keys [CAP][256] float
  static constexpr int QC_OFF = QK_OFF + K2_CAP * 256 * 4;   // queue columns [CAP][256] u16
  static constexpr int XS_OFF = QC_OFF + K2_CAP * 256 * 2;   // |x_j|^2 of 4 tiles in flight [4][64]
  static constexpr int TOTAL = XS_OFF + 4 * K2_TC * 4 + 64;
};

template <int KC4, int ROWS>
__device__ __forceinline__ void knn_store_tile_r(unsigned char* hi_base, unsigned char* lo_base,
                                                 const float* __restrict__ x, int ld, int C,
                                                 int64_t row0, int64_t rows_end, int t, int nthr,
                                                 bool vec_ok) {
  constexpr int LBO = tc::tile_lbo(ROWS);
  constexpr int CH = ROWS * KC4;
  for (int c = t; c < CH; c += nthr) {
    const int r = c / KC4, kc = c % KC4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t row = row0 + r;
    const int k = 4 * kc;
    if (row < rows_end && k < C) {
      const float* p = x + row * (int64_t)ld + k;
      if (vec_ok && k + 3 < C) {
        v = *reinterpret_cast<const float4*>(p);
      } else {
        v.x = p[0];
        if (k + 1 < C) v.y = p[1];
        if (k + 2 < C) v.z = p[2];
        if (k + 3 < C) v.w = p[3];
      }
    }
    float4 hi, lo;
    tc::split4(v, hi, lo);
    *reinterpret_cast<float4*>(hi_base + kc * LBO + r * 16) = hi;
    *reinterpret_cast<float4*>(lo_base + kc * LBO + r * 16) = lo;
  }
}

// descending bitonic sort of 64 registers (fully unrolled: every index is a compile-time constant)
__device__ __forceinline__ void sort64_desc(float (&v)[64]) {
#pragma unroll
  for (int size = 2; size <= 64; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll
      for (int i = 0; i < 64; ++i) {
        const int j = i ^ stride;
        if (j > i) {
          const bool desc = (i & size) == 0;
          const float a = v[i], b = v[j];
          v[i] = desc ? fmaxf(a, b) : fminf(a, b);
          v[j] = desc ? fminf(a, b) : fmaxf(a, b);
        }
      }
    }
  }
}

// the reference's ranking keys of 32 consecutive candidates: -xx_i - (-2 x_i.x_j) - xx_j
__device__ __forceinline__ void knn_keys32(float (&v)[32], float nq, const float* xs32) {
#pragma unroll
  for (int u = 0; u < 32; u += 4) {
    const float4 cn = *reinterpret_cast<const float4*>(xs32 + u);
    // (nq - (-2 v)) - cn: the doubling is exact, so one FMA gives the reference's rounding
    v[u + 0] = fmaf(2.f, v[u + 0], nq) - cn.x;
    v[u + 1] = fmaf(2.f, v[u + 1], nq) - cn.y;
    v[u + 2] = fmaf(2.f, v[u + 2], nq) - cn.z;
    v[u + 3] = fmaf(2.f, v[u + 3], nq) - cn.w;
  }
}

template <int KC4>
__global__ __launch_bounds__(K2_THREADS, 1) void knn_tc2_kernel(const float* __restrict__ x, int ld,
                                                                int C, const float* __restrict__ xx,
                                                                int N, int k,
                                                                int32_t* __restrict__ idx32,
                                                                int64_t* __restrict__ idx64) {
  constexpr int KL = 20;
  extern __shared__ __align__(128) unsigned char smem[];
  using S = Knn2Smem<KC4>;
  __shared__ uint64_t bar_full[2];   // accumulator b ready = its MMAs done (also: operand stage b free)
  __shared__ uint64_t bar_tfree[2];  // accumulator b drained by the 256 selector threads
  __shared__ uint64_t bar_sfull[2];  // operand stage b written by the 128 loader threads
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int b = blockIdx.y;
  const int q0 = blockIdx.x * KT_TQ;
  const int64_t base = (int64_t)b * N;
  constexpr int LBOQ = tc::tile_lbo(128), LBOB = tc::tile_lbo(K2_TC);
  constexpr uint32_t IDESC = tc::make_idesc_tf32(128, K2_TC);
  const bool vec_ok = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  const int T = (N + K2_TC - 1) / K2_TC;
  const int ksteps = (min(C, 4 * KC4) + 7) / 8;

  if (tid == 0) {
    tc::mbar_init(&bar_full[0], 1);
    tc::mbar_init(&bar_full[1], 1);
    tc::mbar_init(&bar_tfree[0], 256);
    tc::mbar_init(&bar_tfree[1], 256);
    tc::mbar_init(&bar_sfull[0], 128);
    tc::mbar_init(&bar_sfull[1], 128);
    tc::mbar_fence_init();
  }
  if (w == 0) tc::tmem_alloc(&tmem_base_s, 2 * K2_TC);
  knn_store_tile_r<KC4, 128>(smem + S::Q_OFF, smem + S::Q_OFF + S::TQ, x, ld, C, base + q0,
                             base + N, tid, K2_THREADS, vec_ok);
  tc::fence_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  if (w == 12) {
    // ------------------------------ MMA issue: its own warp ------------------------------------
    // (when a loader thread issued the MMAs, the loaders stood still for as long as the tensor
    // pipe took to accept the 24 instructions of a tile, and the next tile's conversion could not
    // overlap them: MMA and operand staging ran back to back instead of side by side)
    if (lane == 0) {
      const uint32_t q_hi = tc::smem_u32(smem + S::Q_OFF), q_lo = q_hi + S::TQ;
      const uint64_t dqh = tc::make_desc(q_hi, LBOQ, 128), dql = tc::make_desc(q_lo, LBOQ, 128);
      constexpr uint64_t KQ = tc::desc_kstep(LBOQ), KB = tc::desc_kstep(LBOB);
      for (int j = 0; j < 2 * T; ++j) {
        const int st = j & 1;
        tc::mbar_wait(&bar_sfull[st], (j >> 1) & 1);                      // operands staged
        if (j >= 2) tc::mbar_wait(&bar_tfree[st], ((j >> 1) - 1) & 1);    // accumulator drained
        tc::tc_fence_after();
        const uint32_t b_hi = tc::smem_u32(smem + S::B_OFF + st * 2 * S::TB), b_lo = b_hi + S::TB;
        const uint32_t d = tmem_d + st * K2_TC;
        const uint64_t dbh = tc::make_desc(b_hi, LBOB, 128), dbl = tc::make_desc(b_lo, LBOB, 128);
        tc::mma_tf32_c<false>(d, dql, dbh, IDESC);
        tc::mma_tf32_c<true>(d, dqh, dbl, IDESC);
        tc::mma_tf32_c<true>(d, dqh, dbh, IDESC);
#pragma unroll
        for (int ks = 1; ks < 2 * KC4 / 4; ++ks) {
          if (ks < ksteps) {
            tc::mma_tf32_c<true>(d, dql + ks * KQ, dbh + ks * KB, IDESC);
            tc::mma_tf32_c<true>(d, dqh + ks * KQ, dbl + ks * KB, IDESC);
            tc::mma_tf32_c<true>(d, dqh + ks * KQ, dbh + ks * KB, IDESC);
          }
        }
        tc::mma_commit(&bar_full[st]);
      }
    }
  } else if (w >= 8) {
    // ------------------------------ loaders: every tile twice ----------------------------------
    // Two tiles of global loads are in flight per thread (two register sets, prefetch distance 2):
    // with one, every tile paid a full L2 round trip between "registers free again" and "data
    // there" (ncu: the loaders' first use of the loaded data was the hottest loader instruction and
    // the tensor pipe idled 70 % of the time waiting for operands).
    const int lt = tid - 256;
    TileRegs<KC4, K2_TC, 128> trA, trB;
    float* xs = reinterpret_cast<float*>(smem + S::XS_OFF);
    auto tile_of = [&](int j) { return j < T ? j : j - T; };
    auto norm_of = [&](int j) {
      const int cn_ = tile_of(j) * K2_TC + lt;
      return (lt < K2_TC && cn_ < N) ? __ldg(xx + base + cn_) : 0.f;
    };
    tile_load(trA, x, ld, C, base, base + N, lt, vec_ok);
    float xnA = norm_of(0), xnB = 0.f;
    if (2 * T > 1) {
      tile_load(trB, x, ld, C, base + (int64_t)tile_of(1) * K2_TC, base + N, lt, vec_ok);
      xnB = norm_of(1);
    }
    for (int j = 0; j < 2 * T; j += 2) {  // 2 T is even
      {
        const int st = 0;
        if (j >= 2) tc::mbar_wait(&bar_full[st], ((j >> 1) - 1) & 1);  // stage's previous MMAs done
        unsigned char* hi = smem + S::B_OFF + st * 2 * S::TB;
        unsigned char* lo = hi + S::TB;
        tile_store(trA, hi, lo, lt);
        if (lt < K2_TC) xs[(j & 3) * K2_TC + lt] = xnA;  // ring of 4, see knn_tc_kernel
        if (j + 2 < 2 * T) {
          tile_load(trA, x, ld, C, base + (int64_t)tile_of(j + 2) * K2_TC, base + N, lt, vec_ok);
          xnA = norm_of(j + 2);
        }
        tc::fence_async_smem();
        mbar_arrive(&bar_sfull[st]);
      }
      {
        const int st = 1, j1 = j + 1;
        if (j1 >= 2) tc::mbar_wait(&bar_full[st], ((j1 >> 1) - 1) & 1);
        unsigned char* hi = smem + S::B_OFF + st * 2 * S::TB;
        unsigned char* lo = hi + S::TB;
        tile_store(trB, hi, lo, lt);
        if (lt < K2_TC) xs[(j1 & 3) * K2_TC + lt] = xnB;
        if (j1 + 2 < 2 * T) {
          tile_load(trB, x, ld, C, base + (int64_t)tile_of(j1 + 2) * K2_TC, base + N, lt, vec_ok);
          xnB = norm_of(j1 + 2);
        }
        tc::fence_async_smem();
        mbar_arrive(&bar_sfull[st]);
      }
    }
  } else {
    // ------------------------------ selectors ------------------------------------------------
    float* qk = reinterpret_cast<float*>(smem + S::QK_OFF);
    unsigned short* qc = reinterpret_cast<unsigned short*>(smem + S::QC_OFF);
    const int row = 32 * (w & 3) + lane;
    const int half = w >> 2;
    const int q = q0 + row;
    const float nq = (q < N) ? -xx[base + q] : 0.f;
    const float* xs = reinterpret_cast<const float*>(smem + S::XS_OFF) + 32 * half;
    const uint32_t taddr = tmem_d + ((uint32_t)(32 * (w & 3)) << 16) + (uint32_t)(32 * half);
    // ---- pass 1: group maxima --------------------------------------------------------------
#pragma unroll 1
    for (int s = 0; s < K2_G; ++s) qk[s * 256 + tid] = -INFINITY;
#pragma unroll 1
    for (int j = 0; j < T; ++j) {
      const int st = j & 1;
      tc::mbar_wait(&bar_full[st], (j >> 1) & 1);
      tc::tc_fence_after();
      float v[32];
      tc::tmem_ld32(taddr + (uint32_t)(st * K2_TC), v);
      const int c0 = j * K2_TC + 32 * half;
      knn_keys32(v, nq, xs + (j & 3) * K2_TC);
      tc::tc_fence_before();
      mbar_arrive(&bar_tfree[st]);  // accumulator buffer and the tile's norms are consumed
      float m = -INFINITY;
      if (c0 + 32 <= N) {
#pragma unroll
        for (int e = 0; e < 32; ++e) m = fmaxf(m, v[e]);
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (c0 + e < N) m = fmaxf(m, v[e]);
      }
      float* g = qk + (j & (K2_G - 1)) * 256 + tid;
      *g = fmaxf(*g, m);
    }
    // ---- bound: k-th largest of the row's 64 group maxima ---------------------------------------
    asm volatile("bar.sync 2, 256;" ::: "memory");
    float tau;
    {
      float gm[64];
#pragma unroll
      for (int s = 0; s < K2_G; ++s) {
        gm[s] = qk[s * 256 + tid];
        gm[K2_G + s] = qk[s * 256 + (tid ^ 128)];
      }
      sort64_desc(gm);
      tau = gm[0];
#pragma unroll
      for (int i = 1; i < KL; ++i)
        if (i == k - 1) tau = gm[i];
    }
    asm volatile("bar.sync 2, 256;" ::: "memory");  // the maxima are read: the region becomes the queue
    // ---- pass 2: queue everything that reaches the bound, build the lists lazily -------------------
    float lv[KL];
    int li[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) {
      lv[i] = -INFINITY;
      li[i] = 0;
    }
    int qcnt = 0;
    auto drain = [&]() {
      const int mx = __reduce_max_sync(0xffffffffu, qcnt);
      for (int e = 0; e < mx; ++e) {
        if (e < qcnt) {
          const float key = qk[e * 256 + tid];
          if (key > lv[KL - 1]) list_insert<KL>(lv, li, key, (int)qc[e * 256 + tid]);
        }
      }
      qcnt = 0;
    };
#pragma unroll 1
    for (int j2 = 0; j2 < T; ++j2) {
      const int j = T + j2;
      const int st = j & 1;
      tc::mbar_wait(&bar_full[st], (j >> 1) & 1);
      tc::tc_fence_after();
      float v[32];
      tc::tmem_ld32(taddr + (uint32_t)(st * K2_TC), v);
      const int c0 = j2 * K2_TC + 32 * half;
      knn_keys32(v, nq, xs + (j & 3) * K2_TC);
      tc::tc_fence_before();
      mbar_arrive(&bar_tfree[st]);
      // one comparison per key: v >= tau and v > thr  <=>  v >= max(tau, next float above thr)
      const float thr = lv[KL - 1];
      const int tb = __float_as_int(thr);  // next float above thr (-inf -> -FLT_MAX, -0 -> denorm min)
      const float cut = fmaxf(tau, __int_as_float(tb >= 0 ? tb + 1 : (tb == (int)0x80000000 ? 1 : tb - 1)));
      const int nvalid = N - c0;
      if (nvalid >= 32) {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          if (v[e] >= cut) {
            qk[qcnt * 256 + tid] = v[e];
            qc[qcnt * 256 + tid] = (unsigned short)(c0 + e);
            ++qcnt;
          }
        }
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          if (v[e] >= cut && e < nvalid) {
            qk[qcnt * 256 + tid] = v[e];
            qc[qcnt * 256 + tid] = (unsigned short)(c0 + e);
            ++qcnt;
          }
        }
      }
      if (__any_sync(0xffffffffu, qcnt > K2_CAP - 32)) drain();
    }
    drain();
    // merge the two column halves of every row (as in knn_tc_kernel)
    float* qv = qk;
    int* mi = reinterpret_cast<int*>(smem + S::B_OFF);
    asm volatile("bar.sync 2, 256;" ::: "memory");
    if (half == 1) {
#pragma unroll
      for (int i = 0; i < KL; ++i) {
        qv[i * 128 + row] = lv[i];
        mi[i * 128 + row] = li[i];
      }
    }
    asm volatile("bar.sync 2, 256;" ::: "memory");
    if (half == 0) {
#pragma unroll 1
      for (int i = 0; i < KL; ++i) {
        const float key = qv[i * 128 + row];
        if (key > lv[KL - 1]) list_insert<KL>(lv, li, key, mi[i * 128 + row]);
      }
      if (q < N) {
#pragma unroll
        for (int i = 0; i < KL; ++i) {
          if (i < k) {
            const int64_t o = (base + q) * k + i;
            if (idx32) idx32[o] = li[i];
            if (idx64) idx64[o] = li[i];
          }
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (w == 0) tc::tmem_dealloc(tmem_d, 2 * K2_TC);
}

template <int KC4>
static int launch_knn_tc2_t(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                            int32_t* idx32, int64_t* idx64, cudaStream_t st) {
  using S = Knn2Smem<KC4>;
  cudaError_t e = cudaFuncSetAttribute(knn_tc2_kernel<KC4>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((N + KT_TQ - 1) / KT_TQ, (unsigned)B);
  knn_tc2_kernel<KC4><<<grid, K2_THREADS, S::TOTAL, st>>>(x, ld, C, xx, N, k, idx32, idx64);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// TMA-fed two-pass variant with the query operand in TMEM.
// What bounded knn_tc2_kernel (per-tile clock64 timeline of one CTA, scripts/microbench/knn_trace.cu,
// and scripts/microbench/mma_rate.cu):
//  * tcgen05.mma kind::tf32 with both operands in shared memory reads 32 B per operand row per
//    instruction: at N = 64 that is 6 KB in the 48 cycles the instruction takes alone — the whole
//    128 B/clk of the SM's shared memory — so every other shared-memory access (the loaders' tile
//    stores, the selectors' queue) stretched the MMAs to 59 (pass 1) / 80 (pass 2) cycles each;
//    and a 128x64x8 instruction never goes below ~45 cycles (1460 MAC/clk) whereas 128x128x8 runs
//    at 64 cycles = 2047 MAC/clk, the TF32 peak;
//  * the issuing thread is effectively synchronous (the accumulator is complete ~25 cycles after
//    the last issue returns), so its ~400 cycles of barrier round trips per tile idle the pipe;
//  * the four loader warps re-split every candidate tile in every one of a cloud's 16 CTAs, twice.
// Here:  the 128 query rows live in TMEM (hi and lo halves, written once with tcgen05.st) and are
// the MMA's A operand, so an instruction reads only its 4 KB B tile from shared memory; candidate
// tiles are 128 wide (full-rate MMAs, half as many barrier round trips per candidate); the split
// happens ONCE per point — knn_split_kernel writes every 128-candidate tile of a cloud to global
// memory exactly as the MMA wants it in shared memory (hi tile, lo tile, then the 128 squared
// norms) and one cp.async.bulk per stage brings it in: no loader warps.  Same split arithmetic,
// same accumulation order, same selection: neighbour lists are bit-identical to knn_tc2_kernel's.
//   warps 0-7 selectors (TMEM lane quarter, 64-column half), warp 8 lane 0 = copy producer,
//   warp 9 lane 0 = MMA issue; NST operand stages, 3 accumulators of 128 columns behind the
//   128 columns of Q (512 TMEM columns), norms in a ring of 8.
// ---------------------------------------------------------------------------------------------
// per-tile timestamps of one CTA (scripts/microbench/knn_trace.cu compiles this file with KNN_TRACE)
#ifdef KNN_TRACE
__device__ long long g_knn_trace[8 * 4096];
#define KNN_TR(slot, j) \
  do { if (blockIdx.x == KNN_TRACE_BX && blockIdx.y == KNN_TRACE_BY) g_knn_trace[(slot) * 4096 + (j)] = clock64(); } while (0)
#else
#define KNN_TR(slot, j) do { } while (0)
#endif
#define K3_THREADS 576  // warps 0-15 selectors, 16 copy producer, 17 MMA issue
#define K3_TC 128
#define K3_NACC 3
#define K3_NR 8
// single-product pass 1 pays where the MMAs dominate a tile (C = 64: 24 -> 8 per tile); at C <= 16 a
// tile has 6 MMAs anyway and the looser bound only adds candidates (knn0 1.47 -> 1.58 ms)
#define K3_APPROX1(kc4) ((kc4) >= 16)
#define K3_G 16   // group maxima per selector thread (64 per row)

template <int KC4>
struct KnnSplit {
  static constexpr int TB = tc::tile_bytes(K3_TC, KC4);
  static constexpr int NORMS = K3_TC * 4 + 16;  // 128 squared norms + their maximum
  static constexpr int BLK = 2 * TB + NORMS;    // hi, lo, norms
};

template <int KC4>
__global__ __launch_bounds__(256) void knn_split_kernel(const float* __restrict__ x, int ld, int C,
                                                        const float* __restrict__ xx, int N,
                                                        unsigned char* __restrict__ out) {
  extern __shared__ __align__(128) unsigned char sm[];
  using P = KnnSplit<KC4>;
  constexpr int LBO = tc::tile_lbo(K3_TC);
  const int t = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int T = gridDim.x;
  const int64_t base = (int64_t)b * N;
  const bool vec_ok = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  knn_store_tile_r<KC4, K3_TC>(sm, sm + P::TB, x, ld, C, base + (int64_t)t * K3_TC, base + N, tid,
                               256, vec_ok);
  if (tid < K3_TC) {
    const int cn = t * K3_TC + tid;
    const float nv = cn < N ? xx[base + cn] : 0.f;
    float* nrm = reinterpret_cast<float*>(sm + 2 * P::TB);
    nrm[tid] = nv;
    float mx = nv;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) nrm[K3_TC + (tid >> 5)] = mx;  // four partial maxima (the tile's 16 spare bytes)
  }
  if (tid < 2 * KC4)  // the 16 bytes of padding behind every chunk column (never read by the MMA)
    *reinterpret_cast<float4*>(sm + (tid / KC4) * P::TB + (tid % KC4) * LBO + K3_TC * 16) =
        make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  float4* dst = reinterpret_cast<float4*>(out + ((int64_t)b * T + t) * P::BLK);
  const float4* src = reinterpret_cast<const float4*>(sm);
  for (int i = tid; i < P::BLK / 16; i += 256) dst[i] = src[i];
}

template <int KC4, int NST, int CAP>
struct Knn3Smem {
  static constexpr int TB = tc::tile_bytes(K3_TC, KC4);
  static constexpr int B_OFF = 0;                            // NST stages x (hi, lo)
  static constexpr int XS_OFF = B_OFF + NST * 2 * TB;        // |x_j|^2 ring [K3_NR][128]
  static constexpr int QK_OFF = XS_OFF + K3_NR * (K3_TC * 4 + 16);  // queue keys [CAP][512] float
  static constexpr int QC_OFF = QK_OFF + CAP * 512 * 4;      // queue columns [CAP][512] u16
  static constexpr int TOTAL = QC_OFF + CAP * 512 * 2;
  static_assert(CAP >= K3_G + 1 && CAP >= 17, "queue region: pass-1 group maxima / half a chunk");
  static_assert(NST * 2 * TB >= 3 * 20 * 128 * 8, "the final merge borrows the operand stages");
};

// descending bitonic sort of 16 registers
__device__ __forceinline__ void sort16_desc(float (&v)[16]) {
#pragma unroll
  for (int size = 2; size <= 16; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int j = i ^ stride;
        if (j > i) {
          const bool desc = (i & size) == 0;
          const float a = v[i], b = v[j];
          v[i] = desc ? fmaxf(a, b) : fminf(a, b);
          v[j] = desc ? fminf(a, b) : fmaxf(a, b);
        }
      }
    }
  }
}

template <int KC4, int NST, int CAP>
__global__ __launch_bounds__(K3_THREADS, 1) void knn_tc3_kernel(
    const float* __restrict__ x, int ld, int C, const float* __restrict__ xx,
    const unsigned char* __restrict__ split, int N, int k, int32_t* __restrict__ idx32,
    int64_t* __restrict__ idx64) {
  constexpr int KL = 20;
  constexpr int QCOLS = 8 * KC4;  // TMEM columns of the query operand (hi + lo)
  constexpr int ACC0 = 128;       // first accumulator column
  extern __shared__ __align__(128) unsigned char smem[];
  using S = Knn3Smem<KC4, NST, CAP>;
  using P = KnnSplit<KC4>;
  static_assert(QCOLS <= ACC0, "query operand overlaps the accumulators");
  __shared__ uint64_t bar_sfull[NST];       // operand stage s landed (bulk-copy bytes)
  __shared__ uint64_t bar_sfree[NST];       // operand stage s read by its MMAs
  __shared__ uint64_t bar_full[K3_NACC];    // accumulator a complete
  __shared__ uint64_t bar_tfree[K3_NACC];   // accumulator a drained by the 512 selector threads
  __shared__ uint64_t bar_q[2];             // query tile landed / moved on into TMEM
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int b = blockIdx.y;
  const int q0 = blockIdx.x * KT_TQ;
  const int64_t base = (int64_t)b * N;
  constexpr int LBOB = tc::tile_lbo(K3_TC);
  constexpr uint32_t IDESC = tc::make_idesc_tf32(128, K3_TC);
  const int T = (N + K3_TC - 1) / K3_TC;
  const int ksteps = (min(C, 4 * KC4) + 7) / 8;
  if (tid == 0) KNN_TR(6, 4000);

  if (tid == 0) {
    for (int i = 0; i < NST; ++i) {
      tc::mbar_init(&bar_sfull[i], 1);
      tc::mbar_init(&bar_sfree[i], 1);
    }
    for (int i = 0; i < K3_NACC; ++i) {
      tc::mbar_init(&bar_full[i], 1);
      tc::mbar_init(&bar_tfree[i], 512);
    }
    tc::mbar_init(&bar_q[0], 1);
    tc::mbar_init(&bar_q[1], 128);
    tc::mbar_fence_init();
  }
  if (w == 0) tc::tmem_alloc(&tmem_base_s, 512);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;
  if (tid == 0) KNN_TR(6, 4001);

  if (w == 16) {
    // ------------------------------ copy producer: every tile twice --------------------------
    // The CTA's 128 query rows are candidate tile blockIdx.x of the same cloud: their pre-split
    // copy goes through the last operand stage on its way into TMEM (thread-per-row global loads
    // took 7000 cycles here; this takes the latency of one bulk copy).
    if (lane == 0) {
      const unsigned char* src0 = split + (int64_t)b * T * P::BLK;
      tc::mbar_arrive_expect_tx(&bar_q[0], (uint32_t)(2 * S::TB));
      tc::bulk_g2s(smem + S::B_OFF + (NST - 1) * 2 * S::TB, src0 + (int64_t)blockIdx.x * P::BLK,
                   2 * S::TB, &bar_q[0]);
      for (int j = 0; j < 2 * T; ++j) {
        const int s = j % NST;
        if (j >= NST) tc::mbar_wait(&bar_sfree[s], ((j / NST) - 1) & 1);
        if (j == NST - 1) tc::mbar_wait(&bar_q[1], 0);  // the query tile has left the stage
        KNN_TR(0, j);
        const unsigned char* src = src0 + (int64_t)(j < T ? j : j - T) * P::BLK;
        // pass 1 works on the single product Qhi.Bhi (see the MMA warp): only the hi tile travels
        const uint32_t tbytes = (K3_APPROX1(KC4) && j < T) ? S::TB : 2 * S::TB;
        tc::mbar_arrive_expect_tx(&bar_sfull[s], tbytes + P::NORMS);
        tc::bulk_g2s(smem + S::B_OFF + s * 2 * S::TB, src, tbytes, &bar_sfull[s]);
        // norm ring of 8: slot j is rewritten by tile j + 8, whose copy waits for MMA j + 8 - NST
        // (>= j + 4), which was issued after the selectors released tile j + 4 - K3_NACC >= j
        tc::bulk_g2s(smem + S::XS_OFF + (j & (K3_NR - 1)) * P::NORMS, src + 2 * S::TB, P::NORMS,
                     &bar_sfull[s]);
      }
    }
  } else if (w < 4) {  // query rows -> TMEM (a warp can only touch its own lane quarter)
    const int row = 32 * w + lane;
    const unsigned char* qh = smem + S::B_OFF + (NST - 1) * 2 * S::TB + row * 16;
    const uint32_t trow = tmem_d + ((uint32_t)(32 * w) << 16);
    tc::mbar_wait(&bar_q[0], 0);
#pragma unroll
    for (int c4 = 0; c4 < KC4; c4 += 4) {
      float hi[16], lo[16];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 h = *reinterpret_cast<const float4*>(qh + (c4 + u) * LBOB);
        const float4 l = *reinterpret_cast<const float4*>(qh + S::TB + (c4 + u) * LBOB);
        hi[4 * u] = h.x; hi[4 * u + 1] = h.y; hi[4 * u + 2] = h.z; hi[4 * u + 3] = h.w;
        lo[4 * u] = l.x; lo[4 * u + 1] = l.y; lo[4 * u + 2] = l.z; lo[4 * u + 3] = l.w;
      }
      tc::tmem_st16(trow + (uint32_t)(4 * c4), hi);
      tc::tmem_st16(trow + (uint32_t)(4 * KC4 + 4 * c4), lo);
    }
    mbar_arrive(&bar_q[1]);
    tc::tmem_st_wait();
  }
  if (w != 16) {  // all but the producer warp: the query operand is in TMEM
    tc::tc_fence_before();
    asm volatile("bar.sync 3, %0;" ::"n"(K3_THREADS - 32) : "memory");
    tc::tc_fence_after();
  }

  if (w == 16) {
    // (done above)
  } else if (w == 17) {
    // ------------------------------ MMA issue: the whole warp walks the loop, one elected lane
    // issues (tc::mma_tf32_ts_elect) ----------------------------------------------------------
    const uint32_t aq_hi = tmem_d, aq_lo = tmem_d + 4 * KC4;
    constexpr uint64_t KB = tc::desc_kstep(LBOB);
    for (int j = 0; j < 2 * T; ++j) {
      const int s = j % NST, a = j % K3_NACC;
      tc::mbar_wait(&bar_sfull[s], (j / NST) & 1);
      if (lane == 0) KNN_TR(1, j);
      if (j >= K3_NACC) tc::mbar_wait(&bar_tfree[a], ((j / K3_NACC) - 1) & 1);
      if (lane == 0) KNN_TR(2, j);
      tc::tc_fence_after();
      const uint32_t b_hi = tc::smem_u32(smem + S::B_OFF + s * 2 * S::TB), b_lo = b_hi + S::TB;
      const uint32_t d = tmem_d + ACC0 + a * K3_TC;
      const uint64_t dbh = tc::make_desc(b_hi, LBOB, 128), dbl = tc::make_desc(b_lo, LBOB, 128);
      if (K3_APPROX1(KC4) && j < T) {
        // pass 1 only has to bound the k-th best key: ONE TF32 product (a third of the MMAs, half
        // of the tile bytes); the selectors subtract a rigorous bound of what the two dropped
        // products can contribute
        tc::mma_tf32_ts_elect<false>(d, aq_hi, dbh, IDESC);
#pragma unroll
        for (int ks = 1; ks < 2 * KC4 / 4; ++ks)
          if (ks < ksteps) tc::mma_tf32_ts_elect<true>(d, aq_hi + 8 * ks, dbh + ks * KB, IDESC);
      } else {
        tc::mma_tf32_ts_elect<false>(d, aq_lo, dbh, IDESC);
        tc::mma_tf32_ts_elect<true>(d, aq_hi, dbl, IDESC);
        tc::mma_tf32_ts_elect<true>(d, aq_hi, dbh, IDESC);
#pragma unroll
        for (int ks = 1; ks < 2 * KC4 / 4; ++ks) {
          if (ks < ksteps) {
            tc::mma_tf32_ts_elect<true>(d, aq_lo + 8 * ks, dbh + ks * KB, IDESC);
            tc::mma_tf32_ts_elect<true>(d, aq_hi + 8 * ks, dbl + ks * KB, IDESC);
            tc::mma_tf32_ts_elect<true>(d, aq_hi + 8 * ks, dbh + ks * KB, IDESC);
          }
        }
      }
      tc::mma_commit_elect(&bar_sfree[s]);
      tc::mma_commit_elect(&bar_full[a]);
      if (lane == 0) KNN_TR(3, j);
    }
  } else {
    // ------------------------------ selectors --------------------------------------------------
    // thread = (query row, 32-column quarter of every 128-candidate tile): 16 warps, four per
    // scheduler — with eight the selection was latency-bound at half an instruction per cycle and
    // scheduler, and slower than the MMAs in pass 2
    float* qk = reinterpret_cast<float*>(smem + S::QK_OFF);
    unsigned short* qc = reinterpret_cast<unsigned short*>(smem + S::QC_OFF);
    const int row = 32 * (w & 3) + lane;
    const int cq = w >> 2;
    const int q = q0 + row;
    const float nq = (q < N) ? -xx[base + q] : 0.f;
    const unsigned char* xs_ring = smem + S::XS_OFF;  // slot stride P::NORMS
    const uint32_t taddr = tmem_d + ((uint32_t)(32 * (w & 3)) << 16) + (uint32_t)(ACC0 + 32 * cq);
    // ---- pass 1: group maxima (16 per thread, 64 per row) of the APPROXIMATE keys (Qhi.Bhi) ---
    float kmax2 = 0.f;  // largest squared candidate norm
#pragma unroll 1
    for (int s = 0; s < K3_G; ++s) qk[s * 512 + tid] = -INFINITY;
#pragma unroll 1
    for (int j = 0; j < T; ++j) {
      const int a = j % K3_NACC;
      if (tid == 0) KNN_TR(7, j);
      // (the tile's norms landed before its MMAs were issued: the issuing thread waited for the
      // copy barrier.  The selectors must NOT wait on that barrier themselves — a stage can be
      // refilled for tile j + NST before they reach tile j, and a parity wait two phases behind
      // never returns)
      tc::mbar_wait(&bar_full[a], (j / K3_NACC) & 1);
      if (tid == 0) KNN_TR(4, j);
      tc::tc_fence_after();
      float v[32];
      tc::tmem_ld32(taddr + (uint32_t)(a * K3_TC), v);
      if (tid == 0) KNN_TR(5, j);
      const int c0 = j * K3_TC + 32 * cq;
      {
        const float* xs = reinterpret_cast<const float*>(xs_ring + (j & (K3_NR - 1)) * P::NORMS);
        knn_keys32(v, nq, xs + 32 * cq);
        if (K3_APPROX1(KC4)) {
          const float4 tm = *reinterpret_cast<const float4*>(xs + K3_TC);
          kmax2 = fmaxf(kmax2, fmaxf(fmaxf(tm.x, tm.y), fmaxf(tm.z, tm.w)));
        }
      }
      tc::tc_fence_before();
      mbar_arrive(&bar_tfree[a]);  // accumulator and the tile's norms are consumed
      if (tid == 0) KNN_TR(6, j);
      float m = -INFINITY;
      if (c0 + 32 <= N) {
#pragma unroll
        for (int e = 0; e < 32; ++e) m = fmaxf(m, v[e]);
      } else {
#pragma unroll
        for (int e = 0; e < 32; ++e)
          if (c0 + e < N) m = fmaxf(m, v[e]);
      }
      float* g = qk + (j & (K3_G - 1)) * 512 + tid;
      *g = fmaxf(*g, m);
    }
    // ---- bound.  Any lower bound of the row's k-th best key is valid; the tightest one from the 64
    // group maxima is their k-th largest, but selecting it (a 64-element sort, or a 4-way merge of
    // the four threads' sorted runs) took 8000-9000 cycles in which the tensor pipe ran dry after
    // three tiles.  Branch-free instead: every thread sorts its 16 maxima, the two threads of a
    // 64-column half combine their runs into the ceil(k/2)-th largest of the half's 32 maxima
    // (k-th of two sorted runs = max_i min(A[i-1], B[k-i-1])), and tau = the smaller of the two
    // halves' values: 2 ceil(k/2) >= k keys lie at or above it.  ~17 % more candidates reach the
    // queue (28 instead of 24 per row at k = 20). ------------------------------------------------
    float tau;
    {
      float gm[K3_G];
#pragma unroll
      for (int s = 0; s < K3_G; ++s) gm[s] = qk[s * 512 + tid];
      sort16_desc(gm);
#pragma unroll
      for (int s = 0; s < K3_G; ++s) qk[s * 512 + tid] = gm[s];
      asm volatile("bar.sync 2, 512;" ::: "memory");
      const int kh = (k + 1) >> 1;          // <= 10
      const float* pb = qk + (tid ^ 128);   // the other 32-column quarter of this half, same row
      float th = -INFINITY;
#pragma unroll
      for (int i = 0; i <= (KL + 1) / 2; ++i) {
        if (i <= kh) {
          const float av = i == 0 ? INFINITY : gm[i - 1];
          const int bi = kh - i - 1;
          const float bv = bi < 0 ? INFINITY : pb[bi * 512];
          th = fmaxf(th, fminf(av, bv));
        }
      }
      float* tx = reinterpret_cast<float*>(qc);  // the column queue is idle until pass 2
      tx[tid] = th;
      asm volatile("bar.sync 2, 512;" ::: "memory");
      tau = fminf(th, tx[tid ^ 256]);
      // The bound came from keys with Qlo.Bhi + Qhi.Blo missing: |q_lo| <= 2^-11 |q| (TF32 round to
      // nearest), so the two dot products are below 2^-10 |q||k| (1 + 2^-11), the FP32 accumulation
      // of the 3 x 64 products differs by < 2e-5 |q||k|, and the key doubles the dot product:
      // |key - approximate key| < 2^-9 * 1.02 |q| max|k| (+ the rounding of the key's own two
      // operations).  k approximate keys are >= the approximate bound, so k exact keys are >= it
      // minus the margin.
      const float q2 = -nq;
      if (K3_APPROX1(KC4))
        tau -= 1.05f * (1.0f / 512.0f) * sqrtf(q2 * kmax2) + (1.0f / 524288.0f) * (q2 + kmax2);
    }
    asm volatile("bar.sync 2, 512;" ::: "memory");  // the maxima are read: the region becomes the queue
    // ---- pass 2: queue everything that reaches the bound, build the lists lazily -------------------
    float lv[KL];
    int li[KL];
#pragma unroll
    for (int i = 0; i < KL; ++i) {
      lv[i] = -INFINITY;
      li[i] = 0;
    }
    int qcnt = 0;
    auto drain = [&]() {
      const int mx = __reduce_max_sync(0xffffffffu, qcnt);
      for (int e = 0; e < mx; ++e) {
        if (e < qcnt) {
          const float key = qk[e * 512 + tid];
          if (key > lv[KL - 1]) list_insert<KL>(lv, li, key, (int)qc[e * 512 + tid]);
        }
      }
      qcnt = 0;
    };
#pragma unroll 1
    for (int j2 = 0; j2 < T; ++j2) {
      const int j = T + j2;
      const int a = j % K3_NACC;
      if (tid == 0) KNN_TR(7, j);
      tc::mbar_wait(&bar_full[a], (j / K3_NACC) & 1);
      if (tid == 0) KNN_TR(4, j);
      tc::tc_fence_after();
      float v[32];
      tc::tmem_ld32(taddr + (uint32_t)(a * K3_TC), v);
      if (tid == 0) KNN_TR(5, j);
      const int c0 = j2 * K3_TC + 32 * cq;
      knn_keys32(v, nq, reinterpret_cast<const float*>(xs_ring + (j & (K3_NR - 1)) * P::NORMS) + 32 * cq);
      tc::tc_fence_before();
      mbar_arrive(&bar_tfree[a]);
      if (tid == 0) KNN_TR(6, j);
      const int nvalid = N - c0;
#pragma unroll
      for (int hh = 0; hh < 32; hh += 16) {  // a queue holds half a chunk at least
        if (__any_sync(0xffffffffu, qcnt > CAP - 16)) drain();
        // one comparison per key: v >= tau and v > thr  <=>  v >= max(tau, next float above thr)
        const float thr = lv[KL - 1];
        const int tb = __float_as_int(thr);  // next float above thr (-inf -> -FLT_MAX, -0 -> denorm min)
        const float cut = fmaxf(tau, __int_as_float(tb >= 0 ? tb + 1 : (tb == (int)0x80000000 ? 1 : tb - 1)));
        if (nvalid >= 32) {
#pragma unroll
          for (int e = hh; e < hh + 16; ++e) {
            if (v[e] >= cut) {
              qk[qcnt * 512 + tid] = v[e];
              qc[qcnt * 512 + tid] = (unsigned short)(c0 + e);
              ++qcnt;
            }
          }
        } else {
#pragma unroll
          for (int e = hh; e < hh + 16; ++e) {
            if (v[e] >= cut && e < nvalid) {
              qk[qcnt * 512 + tid] = v[e];
              qc[qcnt * 512 + tid] = (unsigned short)(c0 + e);
              ++qcnt;
            }
          }
        }
      }
    }
    if (tid == 0) KNN_TR(6, 4002);
    drain();
    if (tid == 0) KNN_TR(6, 4003);
    // merge the four column quarters of every row, pairwise (1 -> 0 and 3 -> 2, then 2 -> 0); the
    // published lists are sorted, so a merge stops at the first entry that does not make the list.
    // Every copy has landed and every MMA has completed by now: the operand stages are free.
    float* mv = reinterpret_cast<float*>(smem + S::B_OFF);      // [3][KL][128]
    int* mi = reinterpret_cast<int*>(smem + S::B_OFF) + 3 * KL * 128;
    asm volatile("bar.sync 2, 512;" ::: "memory");
    if (cq & 1) {
#pragma unroll
      for (int i = 0; i < KL; ++i) {
        mv[((cq >> 1) * KL + i) * 128 + row] = lv[i];
        mi[((cq >> 1) * KL + i) * 128 + row] = li[i];
      }
    }
    asm volatile("bar.sync 2, 512;" ::: "memory");
    if (!(cq & 1)) {
#pragma unroll 1
      for (int i = 0; i < KL; ++i) {
        const float key = mv[((cq >> 1) * KL + i) * 128 + row];
        if (!(key > lv[KL - 1])) break;
        list_insert<KL>(lv, li, key, mi[((cq >> 1) * KL + i) * 128 + row]);
      }
      if (cq == 2) {
#pragma unroll
        for (int i = 0; i < KL; ++i) {
          mv[(2 * KL + i) * 128 + row] = lv[i];
          mi[(2 * KL + i) * 128 + row] = li[i];
        }
      }
    }
    asm volatile("bar.sync 2, 512;" ::: "memory");
    if (cq == 0) {
#pragma unroll 1
      for (int i = 0; i < KL; ++i) {
        const float key = mv[(2 * KL + i) * 128 + row];
        if (!(key > lv[KL - 1])) break;
        list_insert<KL>(lv, li, key, mi[(2 * KL + i) * 128 + row]);
      }
      if (q < N) {
#pragma unroll
        for (int i = 0; i < KL; ++i) {
          if (i < k) {
            const int64_t o = (base + q) * k + i;
            if (idx32) idx32[o] = li[i];
            if (idx64) idx64[o] = li[i];
          }
        }
      }
    }
  }
  if (tid == 0) KNN_TR(6, 4004);
  tc::tc_fence_before();
  __syncthreads();
  if (w == 0) tc::tmem_dealloc(tmem_d, 512);
  if (tid == 0) KNN_TR(6, 4005);
}

template <int KC4, int NST, int CAP>
static int launch_knn_tc3_t(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                            int32_t* idx32, int64_t* idx64, void* split_ws, cudaStream_t st) {
  using S = Knn3Smem<KC4, NST, CAP>;
  using P = KnnSplit<KC4>;
  static_assert(S::TOTAL <= 232448 - 256, "shared memory budget");
  const int T = (N + K3_TC - 1) / K3_TC;
  cudaError_t e = cudaFuncSetAttribute(knn_split_kernel<KC4>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, P::BLK);
  if (e != cudaSuccess) return (int)e;
  knn_split_kernel<KC4><<<dim3(T, (unsigned)B), 256, P::BLK, st>>>(x, ld, C, xx, N,
                                                                   (unsigned char*)split_ws);
  R3DFS_CHECK_LAUNCH();
  e = cudaFuncSetAttribute(knn_tc3_kernel<KC4, NST, CAP>,
                           cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((N + KT_TQ - 1) / KT_TQ, (unsigned)B);
  knn_tc3_kernel<KC4, NST, CAP><<<grid, K3_THREADS, S::TOTAL, st>>>(
      x, ld, C, xx, (const unsigned char*)split_ws, N, k, idx32, idx64);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// bytes of the pre-split candidate tiles of B clouds of N points (0: shape not served by the
// TMA-fed kernel)
size_t knn_split_bytes(int C, int64_t B, int N, int k) {
  if (k < 1 || k > 20 || C > 64 || N < 1024 || N > 65535 || N < k) return 0;
  const size_t T = (size_t)(N + K3_TC - 1) / K3_TC;
  const size_t blk = C <= 16 ? KnnSplit<4>::BLK : KnnSplit<16>::BLK;
  return (size_t)B * T * blk;
}

template <int KC4, int KL>
static int launch_knn_tc_t(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                           int32_t* idx32, int64_t* idx64, cudaStream_t st) {
  using S = KnnTcSmem<KC4>;
  cudaError_t e = cudaFuncSetAttribute(knn_tc_kernel<KC4, KL>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((N + KT_TQ - 1) / KT_TQ, (unsigned)B);
  knn_tc_kernel<KC4, KL><<<grid, KT_THREADS, S::TOTAL, st>>>(x, ld, C, xx, N, k, idx32, idx64);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

static bool knn_tc2_forced() {  // A/B switch: R3DFS_KNN_TC2=1 (register-fed two-pass kernel)
  static const bool v = [] {
    const char* e = R3DFS_GETENV("R3DFS_KNN_TC2");
    return e && e[0] == '1';
  }();
  return v;
}

// returns R3DFS_E_UNSUPPORTED for shapes the tensor-core kernel is not built for (C > 64)
int launch_knn_tc(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                  int32_t* idx32, int64_t* idx64, cudaStream_t st, void* split_ws,
                  size_t split_bytes) {
  if (k < 1 || k > 32 || C > 64 || N < k) return R3DFS_E_UNSUPPORTED;
  // TMA-fed kernel when the caller lends scratch for the pre-split tiles
  if (split_ws && !knn_tc2_forced()) {
    const size_t need = knn_split_bytes(C, B, N, k);
    if (need && split_bytes >= need && (reinterpret_cast<uintptr_t>(split_ws) & 15) == 0) {
      if (C <= 16)
        return launch_knn_tc3_t<4, 4, 30>(x, ld, C, xx, B, N, k, idx32, idx64, split_ws, st);
      return launch_knn_tc3_t<16, 2, 30>(x, ld, C, xx, B, N, k, idx32, idx64, split_ws, st);
    }
  }
  // two-pass selection (measured per 300 clouds of 2048 points: C = 9: 2.03 vs 3.05 ms single
  // pass, C = 64: 3.20 vs 3.43 ms)
  if (k <= 20 && N >= 1024 && N <= 65535) {
    if (C <= 16) return launch_knn_tc2_t<4>(x, ld, C, xx, B, N, k, idx32, idx64, st);
    return launch_knn_tc2_t<16>(x, ld, C, xx, B, N, k, idx32, idx64, st);
  }
  if (C <= 16) {
    if (k <= 20) return launch_knn_tc_t<4, 20>(x, ld, C, xx, B, N, k, idx32, idx64, st);
    return launch_knn_tc_t<4, 32>(x, ld, C, xx, B, N, k, idx32, idx64, st);
  }
  if (k <= 20) return launch_knn_tc_t<16, 20>(x, ld, C, xx, B, N, k, idx32, idx64, st);
  return launch_knn_tc_t<16, 32>(x, ld, C, xx, B, N, k, idx32, idx64, st);
}
