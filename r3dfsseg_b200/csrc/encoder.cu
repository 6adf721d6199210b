// DGCNN encoder kernels (reference models/dgcnn.py, models/attention.py, models/mpti.py:18-40).
// FP32 SIMT implementations: register-tiled GEMMs with XOR-swizzled shared-memory tiles.
#include "common.cuh"

// --------------------------------------------------------------------------------------------
// (B, C, N) strided  ->  point-major (B*N, C) contiguous
// --------------------------------------------------------------------------------------------
__global__ void to_point_major_kernel(const float* __restrict__ x, int64_t C, int64_t N, int64_t sb,
                                      int64_t sc, int64_t sn, float* __restrict__ out,
                                      int64_t total) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  int64_t c = e % C;
  int64_t r = e / C;
  int64_t n = r % N;
  int64_t b = r / N;
  out[e] = x[b * sb + c * sc + n * sn];
}

int launch_to_point_major(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                          int64_t sn, float* out, cudaStream_t st) {
  int64_t total = B * C * N;
  int threads = 256;
  int64_t blocks = (total + threads - 1) / threads;
  to_point_major_kernel<<<(unsigned)blocks, threads, 0, st>>>(x, C, N, sb, sc, sn, out, total);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// squared row norms: xx[r] = sum_c x[r][c]^2   (reference models/dgcnn.py:19)
// --------------------------------------------------------------------------------------------
__global__ void row_norms_kernel(const float* __restrict__ x, int64_t rows, int ld, int C,
                                 float* __restrict__ out) {
  int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* p = x + r * (int64_t)ld;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) {
    float v = p[c];
    s = fmaf(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) out[r] = s;
}

// the same for `batch` matrices `xs` floats apart (out: `rows` norms per matrix, dense) — one launch
__global__ void row_norms_batched_kernel(const float* __restrict__ x, int64_t xs, int64_t rows,
                                         int ld, int C, float* __restrict__ out) {
  int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* p = x + blockIdx.y * xs + r * (int64_t)ld;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) {
    float v = p[c];
    s = fmaf(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) out[blockIdx.y * rows + r] = s;
}

int launch_row_norms_batched(const float* x, int64_t xs, int batch, int64_t rows, int ld, int C,
                             float* out, cudaStream_t st) {
  row_norms_batched_kernel<<<dim3((unsigned)((rows + 7) / 8), batch), 256, 0, st>>>(x, xs, rows, ld,
                                                                                  C, out);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int launch_row_norms(const float* x, int64_t rows, int ld, int C, float* out, cudaStream_t st) {
  int threads = 256;
  int64_t blocks = (rows + 7) / 8;
  row_norms_kernel<<<(unsigned)blocks, threads, 0, st>>>(x, rows, ld, C, out);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// Transposed, swizzled tile load: global row-major [rows][ld] -> smem [KC][ROWS] with
// column index (row ^ ((kk & 7) << 2)).  Each warp iteration covers 4 rows x 8 kk, so global
// reads hit whole 32 B sectors and the 32 smem stores fall in 32 different banks.
// --------------------------------------------------------------------------------------------
template <int ROWS, int KC>
__device__ __forceinline__ void load_tile_T(float* __restrict__ dst, const float* __restrict__ src,
                                            int ld, int64_t row0, int64_t rows_end, int k0,
                                            int k_end) {
  constexpr int KG = KC / 8;
  constexpr int PAIRS = (ROWS / 4) * KG;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  const int r_lo = lane & 3, k_lo = lane >> 2;
  for (int p = w; p < PAIRS; p += nw) {
    int kg = p % KG, rg = p / KG;
    int row = 4 * rg + r_lo, kk = 8 * kg + k_lo;
    int64_t gr = row0 + row;
    int gk = k0 + kk;
    float v = 0.f;
    if (gr < rows_end && gk < k_end) v = src[gr * (int64_t)ld + gk];
    dst[kk * ROWS + (row ^ (k_lo << 2))] = v;
  }
}

// --------------------------------------------------------------------------------------------
// knn: pairwise "distance" tile (register-tiled FP32) feeding a warp-level sorted top-k list.
// Ranking key follows reference models/dgcnn.py:18-22:  pd = -xx_i - (-2 x_i.x_j) - xx_j, topk
// largest, so self comes first.  One CTA = 64 query points of one cloud; the (N, N) matrix is
// never written anywhere.
// --------------------------------------------------------------------------------------------
#define KNN_TQ 64
#define KNN_TC 64
#define KNN_KC 64

__global__ __launch_bounds__(256) void knn_kernel(const float* __restrict__ x, int ld, int C,
                                                  const float* __restrict__ xx, int N, int k,
                                                  int32_t* __restrict__ idx32,
                                                  int64_t* __restrict__ idx64) {
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;                        // [KC][TQ]
  float* Cs = Qs + KNN_KC * KNN_TQ;        // [KC][TC]
  float* Ds = Cs + KNN_KC * KNN_TC;        // [TQ][TC+1]
  float* qn = Ds + KNN_TQ * (KNN_TC + 1);  // [TQ]
  float* cn = qn + KNN_TQ;                 // [TC]

  const int b = blockIdx.y;
  const int q0 = blockIdx.x * KNN_TQ;
  const int64_t base = (int64_t)b * N;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;
  const int nchunks = (C + KNN_KC - 1) / KNN_KC;

  if (tid < KNN_TQ) qn[tid] = (q0 + tid < N) ? xx[base + q0 + tid] : 0.f;

  // per-warp sorted lists for its 8 query rows: lane l holds the l-th best (largest key)
  float lv[8];
  int li[8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    lv[r] = -INFINITY;
    li[r] = 0;
  }

  if (nchunks == 1) load_tile_T<KNN_TQ, KNN_KC>(Qs, x, ld, base + q0, base + N, 0, C);

  for (int c0 = 0; c0 < N; c0 += KNN_TC) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int ch = 0; ch < nchunks; ++ch) {
      const int k0 = ch * KNN_KC;
      __syncthreads();  // previous users of Cs / Ds / Qs are done
      if (nchunks > 1) load_tile_T<KNN_TQ, KNN_KC>(Qs, x, ld, base + q0, base + N, k0, C);
      load_tile_T<KNN_TC, KNN_KC>(Cs, x, ld, base + c0, base + N, k0, C);
      if (ch == 0 && tid < KNN_TC) cn[tid] = (c0 + tid < N) ? xx[base + c0 + tid] : 0.f;
      __syncthreads();
      const int kend = min(KNN_KC, C - k0);
#pragma unroll 8
      for (int kk = 0; kk < kend; ++kk) {
        const int sw = (kk & 7) << 2;
        float4 a = *reinterpret_cast<const float4*>(&Qs[kk * KNN_TQ + ((4 * ty) ^ sw)]);
        float4 c = *reinterpret_cast<const float4*>(&Cs[kk * KNN_TC + ((4 * tx) ^ sw)]);
        float av[4] = {a.x, a.y, a.z, a.w};
        float cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], cv[j], acc[i][j]);
      }
    }
    // keys -> smem tile
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = 4 * ty + i;
      const float nq = -qn[r];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 4 * tx + j;
        float inner = -2.f * acc[i][j];
        float pd = (nq - inner) - cn[c];
        if (c0 + c >= N) pd = -INFINITY;
        Ds[r * (KNN_TC + 1) + c] = pd;
      }
    }
    __syncthreads();
    // selection: warp w owns rows 8w .. 8w+7
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int row = 8 * w + r;
      float thr = __shfl_sync(0xffffffffu, lv[r], k - 1);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float d = Ds[row * (KNN_TC + 1) + lane + 32 * h];
        unsigned m = __ballot_sync(0xffffffffu, d > thr);
        while (m) {
          const int src = __ffs(m) - 1;
          m &= m - 1;
          const float dv = __shfl_sync(0xffffffffu, d, src);
          if (dv > thr) {  // thr may have risen since the ballot
            const int ci = c0 + 32 * h + src;
            const int pos = __popc(__ballot_sync(0xffffffffu, lv[r] >= dv));
            const float pv = __shfl_up_sync(0xffffffffu, lv[r], 1);
            const int pi = __shfl_up_sync(0xffffffffu, li[r], 1);
            if (lane > pos) {
              lv[r] = pv;
              li[r] = pi;
            } else if (lane == pos) {
              lv[r] = dv;
              li[r] = ci;
            }
            thr = __shfl_sync(0xffffffffu, lv[r], k - 1);
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int q = q0 + 8 * w + r;
    if (q < N && lane < k) {
      const int64_t o = (base + q) * k + lane;
      if (idx32) idx32[o] = li[r];
      if (idx64) idx64[o] = li[r];
    }
  }
}

static constexpr size_t KNN_SMEM =
    sizeof(float) * (KNN_KC * KNN_TQ + KNN_KC * KNN_TC + KNN_TQ * (KNN_TC + 1) + KNN_TQ + KNN_TC);

int launch_knn(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
               int32_t* idx32, int64_t* idx64, cudaStream_t st) {
  if (k < 1 || k > 32) return R3DFS_E_UNSUPPORTED;
  cudaError_t e = cudaFuncSetAttribute(knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)KNN_SMEM);
  if (e != cudaSuccess) return (int)e;
  dim3 grid((N + KNN_TQ - 1) / KNN_TQ, (unsigned)B);
  knn_kernel<<<grid, 256, KNN_SMEM, st>>>(x, ld, C, xx, N, k, idx32, idx64);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// linear:  Y[map(m)][n] = act(s[n] * sum_k X[m][k] W[n][k] + t[n])      (1x1 conv + folded BN)
// 128 x 64 tile, BK = 16, 256 threads, 8 x 4 micro-tile.
// --------------------------------------------------------------------------------------------
#define LIN_BM 128
#define LIN_BN 64
#define LIN_BK 16

__global__ __launch_bounds__(256) void linear_kernel(const float* __restrict__ X, int ldx,
                                                     const float* __restrict__ W,
                                                     const float* __restrict__ s,
                                                     const float* __restrict__ t, int act,
                                                     int64_t M, int K, int Nout,
                                                     float* __restrict__ Y, int ldy, RowMap map) {
  __shared__ __align__(16) float As[LIN_BK * LIN_BM];
  __shared__ __align__(16) float Bs[LIN_BK * LIN_BN];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int64_t m0 = (int64_t)blockIdx.x * LIN_BM;
  const int n0 = blockIdx.y * LIN_BN;

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += LIN_BK) {
    __syncthreads();
    load_tile_T<LIN_BM, LIN_BK>(As, X, ldx, m0, M, k0, K);
    load_tile_T<LIN_BN, LIN_BK>(Bs, W, K, n0, Nout, k0, K);
    __syncthreads();
    const int kend = min(LIN_BK, K - k0);
#pragma unroll 4
    for (int kk = 0; kk < kend; ++kk) {
      const int sw = (kk & 7) << 2;
      float4 a0 = *reinterpret_cast<const float4*>(&As[kk * LIN_BM + ((8 * ty) ^ sw)]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[kk * LIN_BM + ((8 * ty + 4) ^ sw)]);
      float4 bb = *reinterpret_cast<const float4*>(&Bs[kk * LIN_BN + ((4 * tx) ^ sw)]);
      float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t m = m0 + 8 * ty + i;
    if (m >= M) continue;
    float* yrow = Y + map(m) * (int64_t)ldy;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + 4 * tx + j;
      if (n < Nout) {
        float v = acc[i][j];
        float sc = s ? s[n] : 1.f;
        float sh = t ? t[n] : 0.f;
        yrow[n] = apply_act(fmaf(sc, v, sh), act);
      }
    }
  }
}

int launch_linear(const float* X, int ldx, const float* W, const float* s, const float* t, int act,
                  int64_t M, int K, int Nout, float* Y, int ldy, RowMap map, cudaStream_t st) {
  dim3 grid((unsigned)((M + LIN_BM - 1) / LIN_BM), (Nout + LIN_BN - 1) / LIN_BN);
  linear_kernel<<<grid, 256, 0, st>>>(X, ldx, W, s, t, act, M, K, Nout, Y, ldy, map);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// EdgeConv first-layer split (reference models/dgcnn.py:41,53):
//   W1 . cat(x_j - x_i, x_i) = W1a . x_j + (W1b - W1a) . x_i
// wpq (128, C) = [W1a ; W1b - W1a], spq = [s1 ; s1], tpq = [0 ; t1], so one per-point GEMM gives
// PQ[:, 0:64] = s1 * (W1a x)   and   PQ[:, 64:128] = s1 * ((W1b - W1a) x) + t1.
// --------------------------------------------------------------------------------------------
__global__ void fold_edge_w1_kernel(const float* __restrict__ w1, const float* __restrict__ s1,
                                    const float* __restrict__ t1, int C, float* __restrict__ wpq,
                                    float* __restrict__ spq, float* __restrict__ tpq) {
  const int total = 128 * C;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    int c = e / C, kk = e % C;
    float v;
    if (c < 64)
      v = w1[c * 2 * C + kk];
    else
      v = w1[(c - 64) * 2 * C + C + kk] - w1[(c - 64) * 2 * C + kk];
    wpq[e] = v;
  }
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 128) {
    spq[i] = s1[i & 63];
    tpq[i] = i < 64 ? 0.f : t1[i - 64];
  }
}

int launch_fold_edge_w1(const float* w1, const float* s1, const float* t1, int C, float* wpq,
                        float* spq, float* tpq, cudaStream_t st) {
  fold_edge_w1_kernel<<<8, 256, 0, st>>>(w1, s1, t1, C, wpq, spq, tpq);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// get_edge_feature (reference models/dgcnn.py:26-42), materialising: out (B, 2C, N, K) =
// cat(x_j - x_i, x_i).  Pure HBM write stream (the output is 2K x the input).  One thread owns 4
// consecutive (n, j) positions and walks over the channels: the neighbour indices are read once,
// every channel iteration issues two 128-bit streaming stores, and a warp writes 512 contiguous
// bytes per channel plane.
// --------------------------------------------------------------------------------------------
__global__ __launch_bounds__(256) void edge_feature_kernel(const float* __restrict__ x, int C,
                                                           int64_t N, int64_t sb, int64_t sc,
                                                           int64_t sn,
                                                           const int64_t* __restrict__ idx, int K,
                                                           float* __restrict__ out,
                                                           int64_t quads_per_plane) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= quads_per_plane) return;
  const int64_t b = blockIdx.y;
  const int64_t NK = N * K;
  const float* xb = x + b * sb;
  const int64_t* ib = idx + b * NK;
  int64_t nbo[4], cto[4];
  bool ok[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int64_t e = 4 * q + u;
    ok[u] = e < NK;
    const int64_t ee = ok[u] ? e : 0;
    cto[u] = (ee / K) * sn;
    nbo[u] = ib[ee] * sn;
  }
  const bool vec = (4 * q + 3 < NK) && ((NK & 3) == 0);
  float* o1 = out + (b * 2 * C) * NK + 4 * q;
  float* o2 = o1 + (int64_t)C * NK;
  for (int c = 0; c < C; ++c) {
    const float* xc = xb + c * sc;
    float d[4], ct[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ct[u] = xc[cto[u]];
      d[u] = xc[nbo[u]] - ct[u];
    }
    if (vec) {
      __stcs(reinterpret_cast<float4*>(o1), make_float4(d[0], d[1], d[2], d[3]));
      __stcs(reinterpret_cast<float4*>(o2), make_float4(ct[0], ct[1], ct[2], ct[3]));
    } else {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u]) {
          o1[u] = d[u];
          o2[u] = ct[u];
        }
    }
    o1 += NK;
    o2 += NK;
  }
}

// Row-gather variant (x point-major: channels contiguous).  One CTA = EF_EB consecutive (n, j)
// positions x all channels:
//   1. the neighbour rows x[nbr] (C contiguous floats, one or a few full sectors each) and the few
//      centre rows are gathered into a shared-memory tile, transposed to [channel][position];
//   2. every channel plane of the output receives EF_EB contiguous floats with 128-bit streaming
//      stores (a warp writes 512 contiguous bytes).
// The 4-byte random gathers of the kernel above (up to 32 L1 wavefronts per load instruction, the
// real limiter of this otherwise pure write stream) become a few conflict-light LDS.
#define EF_EB 128
#define EF_THREADS 256
#define EF_TS (EF_EB + 4)  // tile row stride: rows stay 16-byte aligned for the LDS.128 of step 2
// position of (channel c, slot e): the 16-byte groups of a row are XOR-swizzled with bits of c, so
// the transposing scalar stores of step 1 (16 lanes = 16 channel quads of one slot) fall in 8
// bank groups instead of 2, while a row's groups stay a permutation (step 2 is conflict-free)
__device__ __forceinline__ int ef_pos(int c, int e) {
  return c * EF_TS + ((((e >> 2) ^ ((c >> 3) & 7))) << 2) + (e & 3);
}

template <int CT>  // CT = 64: channel count known at compile time (shifts instead of divisions)
__global__ __launch_bounds__(EF_THREADS) void edge_feature_pm_kernel(
    const float* __restrict__ xp, int C_rt, int64_t N, int64_t sb, int64_t sn,
    const int64_t* __restrict__ idx, int K, float* __restrict__ out) {
  const int C = CT ? CT : C_rt;
  extern __shared__ __align__(16) float ef_smem[];
  float* T = ef_smem;                 // [C][EF_TS]     x[nbr] transposed
  float* Ct = T + (size_t)C * EF_TS;  // [C][EF_TS]     x[centre] transposed (per position)
  __shared__ int s_nb[EF_EB], s_ct[EF_EB];  // neighbour / centre point of every slot
  const int tid = threadIdx.x;
  const int64_t b = blockIdx.y;
  const int64_t NK = N * K;
  const int64_t e0 = (int64_t)blockIdx.x * EF_EB;
  const int ne = (int)min((int64_t)EF_EB, NK - e0);
  const float* xb = xp + b * sb;
  for (int e = tid; e < ne; e += EF_THREADS) {
    s_nb[e] = (int)idx[b * NK + e0 + e];
    s_ct[e] = (int)((e0 + e) / K);
  }
  __syncthreads();
  const bool vec_in = (C & 3) == 0 && (sn & 3) == 0 && (reinterpret_cast<uintptr_t>(xb) & 15) == 0;
  if (CT == 64 && vec_in && ne == EF_EB) {
    // full tile, 64 channels: every thread's 2 x 8 row chunks are in flight before the first one
    // is used (a plain loop would pay one L2 round trip per iteration)
    constexpr int R = EF_EB * 16 / EF_THREADS;
    float4 v[R], ct[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = tid + r * EF_THREADS, e = i >> 4, c4 = i & 15;
      v[r] = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)s_nb[e] * sn) + c4);
      ct[r] = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)s_ct[e] * sn) + c4);
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = tid + r * EF_THREADS, e = i >> 4, c4 = i & 15;
      const int p0 = ef_pos(4 * c4, e);
      T[p0] = v[r].x; T[p0 + EF_TS] = v[r].y; T[p0 + 2 * EF_TS] = v[r].z; T[p0 + 3 * EF_TS] = v[r].w;
      Ct[p0] = ct[r].x; Ct[p0 + EF_TS] = ct[r].y; Ct[p0 + 2 * EF_TS] = ct[r].z;
      Ct[p0 + 3 * EF_TS] = ct[r].w;
    }
  } else if (vec_in) {
    const int C4 = C >> 2;
    for (int i = tid; i < ne * C4; i += EF_THREADS) {
      const int e = i / C4, c4 = i - e * C4;
      const float4 v = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)s_nb[e] * sn) + c4);
      const float4 ct = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)s_ct[e] * sn) + c4);
      const int p0 = ef_pos(4 * c4, e);  // channels 4 c4 .. 4 c4 + 3 share (c >> 3): same swizzle
      T[p0] = v.x; T[p0 + EF_TS] = v.y; T[p0 + 2 * EF_TS] = v.z; T[p0 + 3 * EF_TS] = v.w;
      Ct[p0] = ct.x; Ct[p0 + EF_TS] = ct.y; Ct[p0 + 2 * EF_TS] = ct.z; Ct[p0 + 3 * EF_TS] = ct.w;
    }
  } else {
    for (int i = tid; i < ne * C; i += EF_THREADS) {
      const int e = i / C, c = i - e * C;
      T[ef_pos(c, e)] = __ldg(xb + (int64_t)s_nb[e] * sn + c);
      Ct[ef_pos(c, e)] = __ldg(xb + (int64_t)s_ct[e] * sn + c);
    }
  }
  __syncthreads();
  float* o1 = out + (b * 2 * C) * NK + e0;  // plane c: x_j - x_i ; plane C + c: x_i
  const bool vec = ne == EF_EB && (NK & 3) == 0;
  if (vec) {
    for (int i = tid; i < C * (EF_EB / 4); i += EF_THREADS) {
      const int c = i / (EF_EB / 4), q = i - c * (EF_EB / 4);
      const int p0 = ef_pos(c, 4 * q);
      const float4 t = *reinterpret_cast<const float4*>(T + p0);
      const float4 ct = *reinterpret_cast<const float4*>(Ct + p0);
      const float4 d = make_float4(t.x - ct.x, t.y - ct.y, t.z - ct.z, t.w - ct.w);
      __stcs(reinterpret_cast<float4*>(o1 + (int64_t)c * NK) + q, d);
      __stcs(reinterpret_cast<float4*>(o1 + (int64_t)(C + c) * NK) + q, ct);
    }
  } else {
    for (int i = tid; i < C * ne; i += EF_THREADS) {
      const int c = i / ne, e = i - c * ne;
      const float ct = Ct[ef_pos(c, e)];
      o1[(int64_t)c * NK + e] = T[ef_pos(c, e)] - ct;
      o1[(int64_t)(C + c) * NK + e] = ct;
    }
  }
}

size_t edge_feature_scratch_bytes(int64_t B, int64_t C, int64_t N) {
  return sizeof(float) * (size_t)B * C * N + 256;
}

// ws (may be NULL): scratch of edge_feature_scratch_bytes() used to bring a channel-major x into
// point-major form first.  Without it (or when the tile would not fit in shared memory) the
// 4-positions-per-thread kernel above runs on the strided input directly.
int launch_edge_feature(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                        int64_t sn, const int64_t* idx, int K, float* out, cudaStream_t st,
                        void* ws, size_t ws_bytes) {
  const size_t smem = sizeof(float) * 2 * (size_t)C * EF_TS;
  // whole-row gathers pay off for rows of >= 128 bytes (measured at B = 64, C = 64, k = 20, with
  // the transpose pass of a channel-major x included: N = 8192 2.36 -> 1.37 ms = 62 % of the HBM
  // copy peak, N = 2048 0.39 -> 0.36 ms = 59 %)
  const bool fits = smem <= 200 * 1024 && N * K < ((int64_t)1 << 31) * EF_EB && (C & 3) == 0 &&
                    C >= 32 && (sc == 1 || N >= 1024);
  const float* xp = nullptr;
  int64_t psb = 0, psn = 0;
  if (fits && sc == 1) {  // already point-major behind the view (the reference's collate layout)
    xp = x;
    psb = sb;
    psn = sn;
  } else if (fits && ws && ws_bytes >= edge_feature_scratch_bytes(B, C, N)) {
    float* t = reinterpret_cast<float*>(ws);
    R3DFS_TRY(launch_to_point_major(x, B, C, N, sb, sc, sn, t, st));
    xp = t;
    psb = N * C;
    psn = C;
  }
  if (xp) {
    dim3 grid((unsigned)((N * K + EF_EB - 1) / EF_EB), (unsigned)B);
    cudaError_t e;
    if (C == 64) {
      e = cudaFuncSetAttribute(edge_feature_pm_kernel<64>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      edge_feature_pm_kernel<64><<<grid, EF_THREADS, smem, st>>>(xp, 64, N, psb, psn, idx, K, out);
    } else {
      e = cudaFuncSetAttribute(edge_feature_pm_kernel<0>,
                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      edge_feature_pm_kernel<0><<<grid, EF_THREADS, smem, st>>>(xp, (int)C, N, psb, psn, idx, K, out);
    }
    R3DFS_CHECK_LAUNCH();
    return 0;
  }
  int64_t quads = (N * K + 3) / 4;
  dim3 grid((unsigned)((quads + 255) / 256), (unsigned)B);
  edge_feature_kernel<<<grid, 256, 0, st>>>(x, (int)C, N, sb, sc, sn, idx, K, out, quads);
  R3DFS_CHECK_LAUNCH();
  return 0;
}
