// linear layer on the tensor cores with TMA-fed operands:
//     Y[map(m)][n] = act(s[n] * sum_k X[m][k] W[n][k] + t[n])
// Same math as tc_gemm.cu (3xTF32 tcgen05.mma, TMEM accumulator); the difference is the feed:
//   - one thread issues cp.async.bulk.tensor (TMA) loads of raw FP32 tiles of X and W, 4 k-blocks
//     ahead, completing on mbarriers — no registers and no thread is blocked on global memory;
//   - warps 0-7 turn a landed raw tile into the TF32 hi / lo UMMA operand tiles (2 stages) and
//     hand the stage over through an mbarrier;
//   - one thread of warp 8 issues the TMA loads and the MMAs; tcgen05.commit releases the stage.
// Out-of-range rows / columns / k are zero-filled by the TMA unit itself.
#include <cuda.h>

#include "common.cuh"
#include "tc.cuh"

// per-k-block timestamps of one CTA (scripts/microbench/linear_trace.cu compiles this file with LIN_TRACE)
#ifdef LIN_TRACE
__device__ long long g_lin_trace[8 * 1024];
#define LIN_TR(slot, j) \
  do { if (blockIdx.x == LIN_TRACE_BX) g_lin_trace[(slot) * 1024 + (j)] = clock64(); } while (0)
#else
#define LIN_TR(slot, j) do { } while (0)
#endif
#define TM_BM 128
#define TM_BK 16
#define TM_KC4 (TM_BK / 4)
#define TM_THREADS 256       // operand converters / epilogue (warps 0-7)
#define TM_ALL_THREADS 288   // + warp 8: TMA and MMA issue
#define TM_RAW_STAGES 2

template <int BN>
struct TmaSmem {
  static constexpr int RAW_A = TM_BM * TM_BK * 4;  // 8 KB
  static constexpr int RAW_B = BN * TM_BK * 4;
  static constexpr int RAW_STAGE = RAW_A + RAW_B;
  static constexpr int OP_A = tc::tile_bytes(TM_BM, TM_KC4);
  static constexpr int OP_B = tc::tile_bytes(BN, TM_KC4);
  static constexpr int OP_STAGE = 2 * OP_A + 2 * OP_B;
  static constexpr int RAW_OFF = 0;
  static constexpr int OP_OFF = TM_RAW_STAGES * RAW_STAGE;
  static constexpr int TOTAL = OP_OFF + 2 * OP_STAGE + 1024;  // +1024: manual 1 KB alignment
};

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, "
      "%3}], [%4];" ::"r"(tc::smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(tc::smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc::smem_u32(bar)),
               "r"(bytes)
               : "memory");
}

template <int BN>
__global__ __launch_bounds__(TM_ALL_THREADS, 2) void linear_tma_kernel(
    const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
    const float* __restrict__ s, const float* __restrict__ t, int act, int64_t M, int K, int Nout,
    float* __restrict__ Y, int ldy, RowMap map) {
  extern __shared__ unsigned char smem_raw[];
  using S = TmaSmem<BN>;
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar_full[TM_RAW_STAGES];  // raw tile landed (TMA transaction bytes)
  __shared__ uint64_t bar_mma[2];                // operand stage's MMAs done -> stage free
  __shared__ uint64_t bar_op[2];                 // operand stage written by the 256 converters
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_sc[BN], s_sh[BN];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  // the n-tiles of one m-tile are neighbours in launch order, so the X tile they all read comes
  // from DRAM once and from L2 afterwards (with m fastest every n-tile re-read X from DRAM)
  const int n_tiles = (Nout + BN - 1) / BN;
  const int m0 = (blockIdx.x / n_tiles) * TM_BM;
  const int n0 = (blockIdx.x % n_tiles) * BN;
  constexpr int LBO_A = tc::tile_lbo(TM_BM), LBO_B = tc::tile_lbo(BN);
  constexpr uint32_t IDESC = tc::make_idesc_tf32(TM_BM, BN);
  constexpr int A_CH = TM_BM * TM_KC4 / TM_THREADS;  // 2
  constexpr int B_CH = BN * TM_KC4 / TM_THREADS;     // 2 (BN=128) or 1 (BN=64)
  const int KB = (K + TM_BK - 1) / TM_BK;
  if (tid == 0) LIN_TR(7, 2);

  if (tid < BN) {
    const int n = n0 + tid;
    s_sc[tid] = (s && n < Nout) ? s[n] : 1.f;
    s_sh[tid] = (t && n < Nout) ? t[n] : 0.f;
  }
  if (tid == 0) {
    for (int i = 0; i < TM_RAW_STAGES; ++i) tc::mbar_init(&bar_full[i], 1);
    tc::mbar_init(&bar_mma[0], 1);
    tc::mbar_init(&bar_mma[1], 1);
    tc::mbar_init(&bar_op[0], TM_THREADS);
    tc::mbar_init(&bar_op[1], TM_THREADS);
    tc::mbar_fence_init();
  }
  if (w == 0) tc::tmem_alloc(&tmem_base_s, BN);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  auto issue_tma = [&](int kb) {  // issue thread only
    const int rs = kb % TM_RAW_STAGES;
    unsigned char* ra = smem + S::RAW_OFF + rs * S::RAW_STAGE;
    mbar_expect_tx(&bar_full[rs], S::RAW_STAGE);
    tma_load_2d(ra, &tmX, kb * TM_BK, m0, &bar_full[rs]);
    tma_load_2d(ra + S::RAW_A, &tmW, kb * TM_BK, n0, &bar_full[rs]);
  };

  if (w == 8) {
    // ---- TMA + MMA issue: one thread of its own warp, so the converters never stand still while
    // the tensor pipe accepts a k-block's MMAs (they used to wait for the issuing thread at a
    // CTA-wide barrier every k-block)
    // (the whole warp walks the loop; lane 0 starts the copies, one elected lane issues the MMAs)
    {
      if (lane == 0)
        for (int kb = 0; kb < min(KB, TM_RAW_STAGES); ++kb) issue_tma(kb);
      __syncwarp();
      constexpr uint64_t KA = tc::desc_kstep(LBO_A), KBs = tc::desc_kstep(LBO_B);
      for (int kb = 0; kb < KB; ++kb) {
        const int os = kb & 1;
        tc::mbar_wait(&bar_op[os], (kb >> 1) & 1);  // stage converted; raw stage kb fully read
        if (lane == 0) LIN_TR(0, kb);
        tc::tc_fence_after();
        if (lane == 0 && kb + TM_RAW_STAGES < KB) issue_tma(kb + TM_RAW_STAGES);
        __syncwarp();
        unsigned char* a_hi = smem + S::OP_OFF + os * S::OP_STAGE;
        const uint32_t ah = tc::smem_u32(a_hi), al = ah + S::OP_A;
        const uint32_t bh = al + S::OP_A, bl = bh + S::OP_B;
        const uint64_t dah = tc::make_desc(ah, LBO_A, 128), dal = tc::make_desc(al, LBO_A, 128);
        const uint64_t dbh = tc::make_desc(bh, LBO_B, 128), dbl = tc::make_desc(bl, LBO_B, 128);
        const int ksteps = min(TM_BK, K - kb * TM_BK + 7) / 8;
        tc::mma_tf32_elect(tmem_d, dal, dbh, IDESC, kb != 0);
        tc::mma_tf32_elect(tmem_d, dah, dbl, IDESC, 1);
        tc::mma_tf32_elect(tmem_d, dah, dbh, IDESC, 1);
        if (ksteps > 1) {
          tc::mma_tf32_elect(tmem_d, dal + KA, dbh + KBs, IDESC, 1);
          tc::mma_tf32_elect(tmem_d, dah + KA, dbl + KBs, IDESC, 1);
          tc::mma_tf32_elect(tmem_d, dah + KA, dbh + KBs, IDESC, 1);
        }
        tc::mma_commit_elect(&bar_mma[os]);
        if (lane == 0) LIN_TR(1, kb);
      }
    }
  } else {
    // ---- converters: raw FP32 tile -> TF32 hi / lo UMMA operand tiles ----------------------------
    for (int kb = 0; kb < KB; ++kb) {
      const int rs = kb % TM_RAW_STAGES, os = kb & 1;
      if (tid == 0) LIN_TR(2, kb);
      tc::mbar_wait(&bar_full[rs], (kb / TM_RAW_STAGES) & 1);
      if (tid == 0) LIN_TR(3, kb);
      const unsigned char* ra = smem + S::RAW_OFF + rs * S::RAW_STAGE;
      const unsigned char* rb = ra + S::RAW_A;
      float4 av[A_CH], bv[B_CH];
#pragma unroll
      for (int i = 0; i < A_CH; ++i) {
        const int c = tid + i * TM_THREADS;  // raw tile is row-major [row][16 floats]
        av[i] = *reinterpret_cast<const float4*>(ra + c * 16);
      }
#pragma unroll
      for (int i = 0; i < B_CH; ++i) {
        const int c = tid + i * TM_THREADS;
        bv[i] = *reinterpret_cast<const float4*>(rb + c * 16);
      }
      if (tid == 0) LIN_TR(4, kb);
      if (kb >= 2) tc::mbar_wait(&bar_mma[os], ((kb >> 1) - 1) & 1);
      if (tid == 0) LIN_TR(5, kb);
      unsigned char* a_hi = smem + S::OP_OFF + os * S::OP_STAGE;
      unsigned char* a_lo = a_hi + S::OP_A;
      unsigned char* b_hi = a_lo + S::OP_A;
      unsigned char* b_lo = b_hi + S::OP_B;
#pragma unroll
      for (int i = 0; i < A_CH; ++i) {
        const int c = tid + i * TM_THREADS;
        const int r = c / TM_KC4, kc = c % TM_KC4;
        float4 hi, lo;
        tc::split4(av[i], hi, lo);
        *reinterpret_cast<float4*>(a_hi + kc * LBO_A + r * 16) = hi;
        *reinterpret_cast<float4*>(a_lo + kc * LBO_A + r * 16) = lo;
      }
#pragma unroll
      for (int i = 0; i < B_CH; ++i) {
        const int c = tid + i * TM_THREADS;
        const int r = c / TM_KC4, kc = c % TM_KC4;
        float4 hi, lo;
        tc::split4(bv[i], hi, lo);
        *reinterpret_cast<float4*>(b_hi + kc * LBO_B + r * 16) = hi;
        *reinterpret_cast<float4*>(b_lo + kc * LBO_B + r * 16) = lo;
      }
      tc::fence_async_smem();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(&bar_op[os]))
                   : "memory");
      if (tid == 0) LIN_TR(6, kb);
    }
  }
  tc::mbar_wait(&bar_mma[(KB - 1) & 1], ((KB - 1) >> 1) & 1);
  if (tid == 0) LIN_TR(7, 0);
  tc::tc_fence_after();
  if (w < 8) {
    // all MMAs are complete, so the operand stages are free: reuse them as per-warp transpose
    // buffers for coalesced stores
    float* wbuf = reinterpret_cast<float*>(smem + S::OP_OFF) + w * (32 * 33);
    const int rbase = 32 * (w & 3);
    constexpr int HALF = BN / 2;
    const int cbase = (w >> 2) * HALF;
    const bool vec_y = ((ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(Y) & 15) == 0);
#pragma unroll
    for (int cc = 0; cc < HALF; cc += 32) {
      float v[32];
      tc::tmem_ld32(tmem_d + ((uint32_t)rbase << 16) + (uint32_t)(cbase + cc), v);
      const int nb = n0 + cbase + cc;
#pragma unroll
      for (int j = 0; j < 32; ++j)
        v[j] = apply_act(fmaf(s_sc[cbase + cc + j], v[j], s_sh[cbase + cc + j]), act);
      tc::store_chunk_coalesced(wbuf, v, lane, Nout - nb, vec_y, [&](int r) -> float* {
        const int64_t m = (int64_t)m0 + rbase + r;
        return (m < M) ? Y + map(m) * (int64_t)ldy + nb : nullptr;
      });
    }
  }
  if (tid == 0) LIN_TR(7, 1);
  tc::tc_fence_before();
  __syncthreads();
  if (w == 0) tc::tmem_dealloc(tmem_d, BN);
}

// ---------------------------------------------------------------------------------------------
// Variant with the X operand in TMEM.  The per-k-block trace of linear_tma_kernel
// (scripts/microbench/linear_trace.cu) shows a CTA needing ~2100 cycles per k-block whose six
// MMAs take 384: two CTAs per SM move ~290 KB through shared memory per 2100 cycles — raw tiles
// in (TMA), out (converters), hi/lo operand tiles in again (with 2-way bank conflicts), and both
// operands out once more for every one of the three MMAs of a k-step — i.e. the SM's 128 B/clk.
// Here the converters write the X tile's hi / lo parts straight into TMEM (tcgen05.st, thread =
// row) and the MMA takes its A operand from there: no A operand tile in shared memory at all, and
// an MMA reads only its W tile.  The raw tiles are 64B-swizzled by the TMA unit so that
// thread-per-row reads are conflict-free, and the W tile is written row-contiguously (no bank
// conflicts).  Shared-memory traffic per k-block: 144 KB -> 72 KB.  Same split, same MMA order:
// bit-identical results.
//   TMEM (256 columns per CTA, two CTAs per SM): accumulator 0..BN-1, X stages at 128 + 32 s
//   (hi 16 columns, lo 16 columns).
// ---------------------------------------------------------------------------------------------
#define TS_RAW_STAGES 3
template <int BN>
struct TsSmem {
  static constexpr int RAW_A = TM_BM * TM_BK * 4;  // 8 KB, 64-byte rows, SWIZZLE_64B
  static constexpr int RAW_B = BN * TM_BK * 4;
  static constexpr int RAW_STAGE = RAW_A + RAW_B;
  static constexpr int OP_B = tc::tile_bytes(BN, TM_KC4);
  static constexpr int OP_STAGE = 2 * OP_B;  // W hi, W lo
  static constexpr int RAW_OFF = 0;
  static constexpr int OP_OFF = TS_RAW_STAGES * RAW_STAGE;
  static constexpr int TOTAL = OP_OFF + 2 * OP_STAGE + 1024;  // +1024: manual 1 KB alignment
  static_assert(TS_RAW_STAGES * RAW_STAGE >= 8 * 32 * 33 * 4, "epilogue transpose buffers");
};

// logical 16-byte chunk c of row r of a 64B-swizzled raw tile (64-byte rows, 512-byte aligned)
__device__ __forceinline__ float4 ts_raw_chunk(const unsigned char* tile, int r, int c) {
  return *reinterpret_cast<const float4*>(tile + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
}

// DIST = true is the squared-distance form of the affinity graph (the epilogue of
// linear_tc_kernel<128, true>, which this replaces): X = W = the node features of graph blockIdx.z
// (rows zrow * z + row0 .. of the matrix behind tmX), Y[m][n] = (s[m] + s[n]) - 2 acc with s the
// squared row norms; only the tiles on and above the diagonal are computed, an off-diagonal tile
// is stored twice (as is, and mirrored).  With gmin, every stored value also enters its row's
// group minimum: gmin[z][row][col / AFF_GROUP] (row stride aff_gstride(nn)) = min dist_key over the
// group's columns, where the row's own column and the columns of invalid nodes (valid[z][col] == 0)
// count as 0xffffffff.
template <int BN, bool DIST = false>
__global__ __launch_bounds__(TM_ALL_THREADS, 2) void linear_ts_kernel(
    const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
    const float* __restrict__ s, const float* __restrict__ t, int act, int64_t M, int K, int Nout,
    float* __restrict__ Y, int ldy, RowMap map, int64_t zrow = 0, int64_t row0 = 0,
    const uint8_t* __restrict__ valid = nullptr, unsigned* __restrict__ gmin = nullptr) {
  static_assert(!DIST || (BN == TM_BM && 32 % AFF_GROUP == 0), "DIST: square tiles, groups in a chunk");
  if (DIST && blockIdx.y < blockIdx.x) return;
  extern __shared__ unsigned char smem_raw[];
  using S = TsSmem<BN>;
  unsigned char* smem = reinterpret_cast<unsigned char*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar_full[TS_RAW_STAGES];  // raw tiles landed (TMA transaction bytes)
  __shared__ uint64_t bar_mma[2];                // operand stage's MMAs done -> stage free
  __shared__ uint64_t bar_op[2];                 // operand stage written by the 256 converters
  __shared__ uint32_t tmem_base_s;
  __shared__ float s_sc[BN], s_sh[BN];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int n_tiles = (Nout + BN - 1) / BN;
  const int m0 = DIST ? blockIdx.x * TM_BM : (blockIdx.x / n_tiles) * TM_BM;
  const int n0 = DIST ? blockIdx.y * BN : (blockIdx.x % n_tiles) * BN;
  // DIST: this graph's rows inside the feature matrix, its norms and its output matrix
  const int tma_row = DIST ? (int)(zrow * blockIdx.z + row0) : 0;
  if (DIST) {
    s += (int64_t)blockIdx.z * M;
    Y += (int64_t)blockIdx.z * M * (int64_t)ldy;
  }
  constexpr int LBO_B = tc::tile_lbo(BN);
  constexpr uint32_t IDESC = tc::make_idesc_tf32(TM_BM, BN);
  constexpr uint32_t COL_A = 128;
  const int KB = (K + TM_BK - 1) / TM_BK;

  if (tid < BN) {
    const int n = n0 + tid;
    if (DIST) {  // the column norms
      s_sc[tid] = n < Nout ? s[n] : 0.f;
    } else {
      s_sc[tid] = (s && n < Nout) ? s[n] : 1.f;
      s_sh[tid] = (t && n < Nout) ? t[n] : 0.f;
    }
  }
  if (tid == 0) {
    for (int i = 0; i < TS_RAW_STAGES; ++i) tc::mbar_init(&bar_full[i], 1);
    tc::mbar_init(&bar_mma[0], 1);
    tc::mbar_init(&bar_mma[1], 1);
    tc::mbar_init(&bar_op[0], TM_THREADS);
    tc::mbar_init(&bar_op[1], TM_THREADS);
    tc::mbar_fence_init();
  }
  if (w == 0) tc::tmem_alloc(&tmem_base_s, 256);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_d = tmem_base_s;

  auto issue_tma = [&](int kb) {  // one lane of the issue warp
    const int rs = kb % TS_RAW_STAGES;
    unsigned char* ra = smem + S::RAW_OFF + rs * S::RAW_STAGE;
    mbar_expect_tx(&bar_full[rs], S::RAW_STAGE);
    tma_load_2d(ra, &tmX, kb * TM_BK, tma_row + m0, &bar_full[rs]);
    tma_load_2d(ra + S::RAW_A, &tmW, kb * TM_BK, tma_row + n0, &bar_full[rs]);
  };

  if (w == 8) {
    // ---- TMA + MMA issue (the whole warp walks the loop; lane 0 starts the copies, one elected
    // lane issues the MMAs) ----------------------------------------------------------------------
    if (lane == 0)
      for (int kb = 0; kb < min(KB, TS_RAW_STAGES); ++kb) issue_tma(kb);
    __syncwarp();
    constexpr uint64_t KBs = tc::desc_kstep(LBO_B);
    for (int kb = 0; kb < KB; ++kb) {
      const int os = kb & 1;
      tc::mbar_wait(&bar_op[os], (kb >> 1) & 1);  // stage converted; raw stage kb fully read
      tc::tc_fence_after();
      if (lane == 0 && kb + TS_RAW_STAGES < KB) issue_tma(kb + TS_RAW_STAGES);
      __syncwarp();
      const uint32_t bh = tc::smem_u32(smem + S::OP_OFF + os * S::OP_STAGE), bl = bh + S::OP_B;
      const uint64_t dbh = tc::make_desc(bh, LBO_B, 128), dbl = tc::make_desc(bl, LBO_B, 128);
      const uint32_t ah = tmem_d + COL_A + os * 32, al = ah + 16;
      const int ksteps = min(TM_BK, K - kb * TM_BK + 7) / 8;
      tc::mma_tf32_ts_e(tmem_d, al, dbh, IDESC, kb != 0);
      tc::mma_tf32_ts_e(tmem_d, ah, dbl, IDESC, 1);
      tc::mma_tf32_ts_e(tmem_d, ah, dbh, IDESC, 1);
      if (ksteps > 1) {
        tc::mma_tf32_ts_e(tmem_d, al + 8, dbh + KBs, IDESC, 1);
        tc::mma_tf32_ts_e(tmem_d, ah + 8, dbl + KBs, IDESC, 1);
        tc::mma_tf32_ts_e(tmem_d, ah + 8, dbh + KBs, IDESC, 1);
      }
      tc::mma_commit_elect(&bar_mma[os]);
    }
  } else {
    // ---- converters: X rows -> TMEM (thread = row, 8 columns), W rows -> UMMA tile in shared memory
    const int ar = 32 * (w & 3) + lane;  // X row = TMEM lane
    const int acp = w >> 2;              // chunks 2 acp, 2 acp + 1 = columns 8 acp .. 8 acp + 7
    const uint32_t trow = tmem_d + ((uint32_t)(32 * (w & 3)) << 16) + COL_A + 8 * acp;
    constexpr int B_CH = BN * TM_KC4 / TM_THREADS;  // 2 (BN = 128) or 1 (BN = 64)
    const int br = tid % BN, bc0 = (tid / BN) * B_CH;
    for (int kb = 0; kb < KB; ++kb) {
      const int rs = kb % TS_RAW_STAGES, os = kb & 1;
      tc::mbar_wait(&bar_full[rs], (kb / TS_RAW_STAGES) & 1);
      const unsigned char* ra = smem + S::RAW_OFF + rs * S::RAW_STAGE;
      const unsigned char* rb = ra + S::RAW_A;
      const float4 a0 = ts_raw_chunk(ra, ar, 2 * acp), a1 = ts_raw_chunk(ra, ar, 2 * acp + 1);
      float4 bv[B_CH];
#pragma unroll
      for (int i = 0; i < B_CH; ++i) bv[i] = ts_raw_chunk(rb, br, bc0 + i);
      if (kb >= 2) tc::mbar_wait(&bar_mma[os], ((kb >> 1) - 1) & 1);
      tc::tc_fence_after();
      {
        float4 h0, l0, h1, l1;
        tc::split4(a0, h0, l0);
        tc::split4(a1, h1, l1);
        const float hi[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        const float lo[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
        tc::tmem_st8(trow + os * 32, hi);
        tc::tmem_st8(trow + os * 32 + 16, lo);
      }
      unsigned char* b_hi = smem + S::OP_OFF + os * S::OP_STAGE;
      unsigned char* b_lo = b_hi + S::OP_B;
#pragma unroll
      for (int i = 0; i < B_CH; ++i) {
        float4 hi, lo;
        tc::split4(bv[i], hi, lo);
        *reinterpret_cast<float4*>(b_hi + (bc0 + i) * LBO_B + br * 16) = hi;
        *reinterpret_cast<float4*>(b_lo + (bc0 + i) * LBO_B + br * 16) = lo;
      }
      tc::tmem_st_wait();
      tc::tc_fence_before();
      tc::fence_async_smem();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(&bar_op[os]))
                   : "memory");
    }
  }
  tc::mbar_wait(&bar_mma[(KB - 1) & 1], ((KB - 1) >> 1) & 1);
  tc::tc_fence_after();
  if (w < 8) {
    // all MMAs are complete and every raw tile has been read: the raw stages become the per-warp
    // transpose buffers of the coalesced stores
    float* wbuf = reinterpret_cast<float*>(smem + S::RAW_OFF) + w * (32 * 33);
    const int rbase = 32 * (w & 3);
    constexpr int HALF = BN / 2;
    const int cbase = (w >> 2) * HALF;
    const bool vec_y = ((ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(Y) & 15) == 0);
#pragma unroll
    for (int cc = 0; cc < HALF; cc += 32) {
      float v[32];
      tc::tmem_ld32(tmem_d + ((uint32_t)rbase << 16) + (uint32_t)(cbase + cc), v);
      const int nb = n0 + cbase + cc;
      if (DIST) {
        const int64_t m = (int64_t)m0 + rbase + lane;
        const float sm = (m < M) ? s[m] : 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = (sm + s_sc[cbase + cc + j]) - 2.f * v[j];
        if (blockIdx.y > blockIdx.x && m < M) {
          // mirrored tile: a lane holds one row, so for a fixed column the warp's 32 values are
          // consecutive in the transposed row — coalesced as they stand
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nb + j < Nout) Y[(int64_t)(nb + j) * ldy + m] = v[j];
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          v[j] = apply_act(fmaf(s_sc[cbase + cc + j], v[j], s_sh[cbase + cc + j]), act);
      }
      tc::store_chunk_coalesced(wbuf, v, lane, Nout - nb, vec_y, [&](int r) -> float* {
        const int64_t m = (int64_t)m0 + rbase + r;
        return (m < M) ? Y + map(m) * (int64_t)ldy + nb : nullptr;
      });
      if (DIST && gmin) {
        // group minima, read back from the transpose buffer the store just filled: wbuf[r][c] is
        // row m0 + rbase + r, column nb + c, and lane-indexed reads are conflict-free either way.
        // A lane stores the 4 minima of its row in this chunk as one 16-byte vector.
        static_assert(32 / AFF_GROUP == 4, "one uint4 of minima per row and chunk");
        const int gstride = aff_gstride(Nout);
        const uint8_t* vz = valid + (int64_t)blockIdx.z * M;
        uint4* gz = reinterpret_cast<uint4*>(gmin + (int64_t)blockIdx.z * M * gstride);
        const int64_t m = (int64_t)m0 + rbase + lane;
        const int self = (blockIdx.x == blockIdx.y) ? (int)(m - nb) : -1;
        unsigned cvalid = __ballot_sync(0xffffffffu, nb + lane < Nout && vz[nb + lane]);
        unsigned g4[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
#pragma unroll
        for (int c = 0; c < 32; ++c)
          g4[c / AFF_GROUP] = min(g4[c / AFF_GROUP], (((cvalid >> c) & 1u) && c != self)
                                                         ? dist_key(wbuf[lane * 33 + c])
                                                         : 0xffffffffu);
        if (m < M && nb < Nout)
          gz[(m * gstride + nb / AFF_GROUP) / 4] = make_uint4(g4[0], g4[1], g4[2], g4[3]);
        if (blockIdx.y > blockIdx.x) {  // mirrored: row nb + lane over the columns m0 + rbase + r
          const int64_t c0 = (int64_t)m0 + rbase;
          cvalid = __ballot_sync(0xffffffffu, m < M && vz[m]);
#pragma unroll
          for (int q = 0; q < 4; ++q) g4[q] = 0xffffffffu;
#pragma unroll
          for (int r = 0; r < 32; ++r)
            g4[r / AFF_GROUP] = min(g4[r / AFF_GROUP], ((cvalid >> r) & 1u)
                                                           ? dist_key(wbuf[r * 33 + lane])
                                                           : 0xffffffffu);
          if (nb + lane < Nout && c0 < M)
            gz[((int64_t)(nb + lane) * gstride + c0 / AFF_GROUP) / 4] =
                make_uint4(g4[0], g4[1], g4[2], g4[3]);
        }
        __syncwarp();  // the next chunk overwrites wbuf
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (w == 0) tc::tmem_dealloc(tmem_d, 256);
}

// ---- host side: tensor maps through the driver entry point (no link-time libcuda dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// 2-D fp32 tensor (rows x K, row stride ld floats), box = 16 (k) x box_rows
static bool make_map(CUtensorMap* m, const float* base, int64_t rows, int K, int64_t ld,
                     int box_rows, bool swizzle64 = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {TM_BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE,
            swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE,
            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int BN>
static int launch_tma_bn(const CUtensorMap& tx, const CUtensorMap& tw, const float* s,
                         const float* t, int act, int64_t M, int K, int Nout, float* Y, int ldy,
                         RowMap map, cudaStream_t st) {
  using S = TmaSmem<BN>;
  cudaError_t e = cudaFuncSetAttribute(linear_tma_kernel<BN>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)(((M + TM_BM - 1) / TM_BM) * ((Nout + BN - 1) / BN)));
  linear_tma_kernel<BN><<<grid, TM_ALL_THREADS, S::TOTAL, st>>>(tx, tw, s, t, act, M, K, Nout, Y, ldy,
                                                            map);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

template <int BN>
static int launch_ts_bn(const CUtensorMap& tx, const CUtensorMap& tw, const float* s, const float* t,
                        int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                        cudaStream_t st) {
  using S = TsSmem<BN>;
  cudaError_t e = cudaFuncSetAttribute(linear_ts_kernel<BN>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((unsigned)(((M + TM_BM - 1) / TM_BM) * ((Nout + BN - 1) / BN)));
  linear_ts_kernel<BN><<<grid, TM_ALL_THREADS, S::TOTAL, st>>>(tx, tw, s, t, act, M, K, Nout, Y, ldy,
                                                           map);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// D2[g][i][j] = |f_i|^2 + |f_j|^2 - 2 f_i.f_j for G graphs of nn nodes (rows of D floats) on the
// TMEM-operand kernel (+ the group minima of every row when gmin is given);
// R3DFS_E_UNSUPPORTED when TMA cannot address the feature matrix
int launch_gram_dist_ts(const float* F, int64_t graph_rows, int64_t row_off, int G, int nn, int D,
                        const float* norms, float* D2, const uint8_t* valid, unsigned* gmin,
                        cudaStream_t st) {
  if ((D & 3) != 0 || (reinterpret_cast<uintptr_t>(F) & 15) != 0 ||
      (int64_t)G * graph_rows >= (1ll << 31))
    return R3DFS_E_UNSUPPORTED;
  CUtensorMap tf;
  if (!make_map(&tf, F, (int64_t)G * graph_rows, D, D, TM_BM, true)) return R3DFS_E_UNSUPPORTED;
  using S = TsSmem<128>;
  cudaError_t e = cudaFuncSetAttribute(linear_ts_kernel<128, true>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, S::TOTAL);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((nn + TM_BM - 1) / TM_BM, (nn + 127) / 128, G);
  linear_ts_kernel<128, true><<<grid, TM_ALL_THREADS, S::TOTAL, st>>>(
      tf, tf, norms, nullptr, 0, nn, D, nn, D2, nn, identity_map(), graph_rows, row_off, valid,
      gmin);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

static bool linear_smem_a_forced() {  // A/B switch: R3DFS_LINEAR_SMEM_A=1 (X operand through shared memory)
  static const bool v = [] {
    const char* e = R3DFS_GETENV("R3DFS_LINEAR_SMEM_A");
    return e && e[0] == '1';
  }();
  return v;
}

// returns R3DFS_E_UNSUPPORTED when the operands do not meet TMA's alignment rules (the caller
// then uses the register-fed kernel of tc_gemm.cu)
int launch_linear_tma(const float* X, int ldx, const float* W, const float* s, const float* t,
                      int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                      cudaStream_t st) {
  if ((ldx & 3) != 0 || (K & 3) != 0 || (reinterpret_cast<uintptr_t>(X) & 15) != 0 ||
      (reinterpret_cast<uintptr_t>(W) & 15) != 0 || M >= (1ll << 31))
    return R3DFS_E_UNSUPPORTED;
  const int bn = (Nout > 64) ? 128 : 64;
  CUtensorMap tx, tw;
  if (!linear_smem_a_forced()) {
    if (!make_map(&tx, X, M, K, ldx, TM_BM, true) || !make_map(&tw, W, Nout, K, K, bn, true))
      return R3DFS_E_UNSUPPORTED;
    if (bn == 128) return launch_ts_bn<128>(tx, tw, s, t, act, M, K, Nout, Y, ldy, map, st);
    return launch_ts_bn<64>(tx, tw, s, t, act, M, K, Nout, Y, ldy, map, st);
  }
  if (!make_map(&tx, X, M, K, ldx, TM_BM) || !make_map(&tw, W, Nout, K, K, bn))
    return R3DFS_E_UNSUPPORTED;
  if (bn == 128) return launch_tma_bn<128>(tx, tw, s, t, act, M, K, Nout, Y, ldy, map, st);
  return launch_tma_bn<64>(tx, tw, s, t, act, M, K, Nout, Y, ldy, map, st);
}
