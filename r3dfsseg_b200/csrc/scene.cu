// Whole-scan segmentation (include/r3dfs.h, "Segmenting a whole scan"): cut an (M, 6) scan into
// overlapping xy blocks, split every block into chunks of n_points sampled points normalised as the
// reference's loader does, and merge the per-chunk logits back onto the scan's points.
//
// r3dfs_scene_support ("Support shots from a labelled scan") reads the same plan to cut support
// shots out of a labelled scan: per-block class counts, a seeded choice of blocks per class, and
// shot clouds built by the chunk clouds' code.
//
// r3dfs_scene_plan builds every index the other calls need and leaves it in the workspace:
//   bbox -> grid -> per-point membership counts -> scan -> one record (block << 32 | key, position)
//   per membership -> LSD radix sort -> block segments -> chunk counts -> scan -> (chunk, slot) of
//   every membership, stored back at its position in point order.
// Every step is integer arithmetic or a correctly rounded fp32 operation written out explicitly
// (__fsub_rn / __fdiv_rn), so that the numpy oracle of the tests reproduces it bit for bit, and no
// step uses a float atomic.
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int SCAN_T = 1024, SCAN_IPT = 4, SCAN_TILE = SCAN_T * SCAN_IPT;
constexpr int RS_T = 256, RS_WARPS = RS_T / 32, RS_IPT = 8, RS_TILE = RS_T * RS_IPT;
constexpr int BBOX_CTAS = 256;
constexpr int MAX_CLS = 8;

// device-side plan scalars
struct SceneHdr {
  float x0, y0, stride;
  int32_t ncx, ncy, nbx, nby;
  int32_t err;       // 1: x or y not finite, or the grid has 2^31 blocks or more
  int32_t T;         // memberships
  int32_t n_seg;     // non-empty blocks
  int32_t n_chunks;
  int32_t scratch;   // totals nobody reads
};

struct SceneWs {
  SceneHdr* hdr;
  float* bbox;          // (BBOX_CTAS, 5) partial min x, min y, max x, max y, non-finite flag
  int32_t* off;         // (M + 1) first membership of each point; off[M] = T
  int32_t* bsum;        // scan scratch: one sum per tile
  uint64_t* keys[2];    // (Tmax) records: block << 32 | key; padding = ~0
  int32_t* vals[2];     // (Tmax) membership position in point order
  int32_t* mem_point;   // (Tmax) point of each membership
  int32_t* seg;         // (Tmax + 1) exclusive scan of the block-start flags of the sorted records
  int32_t* seg_start;   // (Tmax + 1) first sorted record of each non-empty block; [n_seg] = T
  int32_t* chunk_off;   // (Tmax + 1) first chunk of each non-empty block; [n_seg] = n_chunks
  int32_t* chunk_seg;   // (Tmax) block segment of each chunk
  int32_t* mem_chunk;   // (Tmax) chunk of each membership (point order)
  int32_t* mem_slot;    // (Tmax) slot of each membership in its chunk
  int32_t* hist;        // (256 * radix tiles) radix digit counts
};

inline int64_t scene_tmax(int64_t M, int r) { return (int64_t)r * r * M; }
inline int64_t rs_tiles(int64_t n) { return (n + RS_TILE - 1) / RS_TILE; }
inline int64_t scan_tiles(int64_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE; }

void carve_scene(WsBump& ws, int64_t M, int r, SceneWs& w) {
  const int64_t T = scene_tmax(M, r);
  const int64_t scan_max = std::max(std::max(M + 1, T + 1), 256 * rs_tiles(T));
  w.hdr = ws.take<SceneHdr>(1);
  w.bbox = ws.take<float>(BBOX_CTAS * 5);
  w.off = ws.take<int32_t>(M + 1);
  w.bsum = ws.take<int32_t>(scan_tiles(scan_max) + 1);
  for (int i = 0; i < 2; ++i) {
    w.keys[i] = ws.take<uint64_t>(T);
    w.vals[i] = ws.take<int32_t>(T);
  }
  w.mem_point = ws.take<int32_t>(T);
  w.seg = ws.take<int32_t>(T + 1);
  w.seg_start = ws.take<int32_t>(T + 1);
  w.chunk_off = ws.take<int32_t>(T + 1);
  w.chunk_seg = ws.take<int32_t>(T);
  w.mem_chunk = ws.take<int32_t>(T);
  w.mem_slot = ws.take<int32_t>(T);
  w.hist = ws.take<int32_t>(256 * rs_tiles(T));
}

inline unsigned nblk(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

__host__ __device__ inline uint32_t lowbias32(uint32_t x) {
  x ^= x >> 16;
  x *= 0x7feb352du;
  x ^= x >> 15;
  x *= 0x846ca68bu;
  x ^= x >> 16;
  return x;
}

// cell of a coordinate: min(floor((x - x0) / stride), n_cells - 1); x >= x0, so the quotient is
// non-negative and bounded by the grid checked in scene_grid_kernel
__device__ __forceinline__ int cell_of(float x, float x0, float stride, int n_cells) {
  const float q = floorf(__fdiv_rn(__fsub_rn(x, x0), stride));
  return min((int)q, n_cells - 1);
}

// ---- scan: exclusive, in place, int32 values, int64 length -----------------------------------
__device__ __forceinline__ int block_excl_scan(int v, int* s_warp, int* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s_warp[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    int s = lane < nw ? s_warp[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += u;
    }
    s_warp[lane] = s;  // inclusive over warps
  }
  __syncthreads();
  const int excl = (wid ? s_warp[wid - 1] : 0) + inc - v;
  if (total) *total = s_warp[nw - 1];
  __syncthreads();
  return excl;
}

__global__ __launch_bounds__(SCAN_T) void scan_reduce_kernel(const int32_t* __restrict__ a,
                                                             int64_t n, int32_t* __restrict__ bsum) {
  __shared__ int s_warp[32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_IPT;
  int v = 0;
#pragma unroll
  for (int i = 0; i < SCAN_IPT; ++i)
    if (base + i < n) v += a[base + i];
  int total;
  block_excl_scan(v, s_warp, &total);
  if (threadIdx.x == 0) bsum[blockIdx.x] = total;
}

// one CTA: exclusive scan of the tile sums in place, grand total -> *total
__global__ __launch_bounds__(SCAN_T) void scan_tiles_kernel(int32_t* __restrict__ bsum,
                                                            int64_t nb, int32_t* __restrict__ total) {
  __shared__ int s_warp[32];
  int carry = 0;
  for (int64_t b0 = 0; b0 < nb; b0 += SCAN_T) {
    const int64_t i = b0 + threadIdx.x;
    const int v = i < nb ? bsum[i] : 0;
    int t;
    const int e = block_excl_scan(v, s_warp, &t);
    if (i < nb) bsum[i] = carry + e;
    carry += t;
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ __launch_bounds__(SCAN_T) void scan_apply_kernel(int32_t* __restrict__ a, int64_t n,
                                                            const int32_t* __restrict__ bsum) {
  __shared__ int s_warp[32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_IPT;
  int v[SCAN_IPT];
  int sum = 0;
#pragma unroll
  for (int i = 0; i < SCAN_IPT; ++i) {
    v[i] = base + i < n ? a[base + i] : 0;
    sum += v[i];
  }
  int run = bsum[blockIdx.x] + block_excl_scan(sum, s_warp, nullptr);
#pragma unroll
  for (int i = 0; i < SCAN_IPT; ++i) {
    if (base + i < n) a[base + i] = run;
    run += v[i];
  }
}

int scan_excl(int32_t* a, int64_t n, int32_t* bsum, int32_t* total, cudaStream_t st) {
  const int64_t nb = scan_tiles(n);
  scan_reduce_kernel<<<(unsigned)nb, SCAN_T, 0, st>>>(a, n, bsum);
  R3DFS_CHECK_LAUNCH();
  scan_tiles_kernel<<<1, SCAN_T, 0, st>>>(bsum, nb, total);
  R3DFS_CHECK_LAUNCH();
  scan_apply_kernel<<<(unsigned)nb, SCAN_T, 0, st>>>(a, n, bsum);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// ---- LSD radix sort of (u64 key, i32 value) pairs, 8 bits per pass, stable -------------------
__global__ __launch_bounds__(RS_T) void radix_hist_kernel(const uint64_t* __restrict__ keys,
                                                          int64_t n, int shift, int64_t ntiles,
                                                          int32_t* __restrict__ hist) {
  __shared__ int h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * RS_TILE;
  for (int i = threadIdx.x; i < RS_TILE; i += RS_T)
    if (base + i < n) atomicAdd(&h[(int)((keys[base + i] >> shift) & 255)], 1);
  __syncthreads();
  hist[(int64_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

// hist: exclusive scan (digit-major over tiles) = first output position of each (digit, tile).
// Warp w ranks elements [base + w*RS_IPT*32, +RS_IPT*32) in order, so a tile keeps input order
// among equal digits.
__global__ __launch_bounds__(RS_T) void radix_scatter_kernel(
    const uint64_t* __restrict__ kin, const int32_t* __restrict__ vin, uint64_t* __restrict__ kout,
    int32_t* __restrict__ vout, int64_t n, int shift, int64_t ntiles,
    const int32_t* __restrict__ hist) {
  __shared__ int s_cnt[RS_WARPS][256];
  __shared__ int s_base[256];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < RS_WARPS * 256; i += RS_T) (&s_cnt[0][0])[i] = 0;
  s_base[threadIdx.x] = hist[(int64_t)threadIdx.x * ntiles + blockIdx.x];
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * RS_TILE + (int64_t)wid * RS_IPT * 32;
  const unsigned lt = (1u << lane) - 1u;
  uint64_t key[RS_IPT];
  int32_t val[RS_IPT];
  int dig[RS_IPT], rank[RS_IPT];
#pragma unroll
  for (int s = 0; s < RS_IPT; ++s) {
    const int64_t i = base + s * 32 + lane;
    const bool ok = i < n;
    key[s] = ok ? kin[i] : 0;
    val[s] = ok ? vin[i] : 0;
    const int d = (int)((key[s] >> shift) & 255);
    dig[s] = ok ? d : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, ok ? d : 256 + lane);
    rank[s] = ok ? s_cnt[wid][d] + __popc(peers & lt) : 0;
    __syncwarp();
    if (ok && lane == __ffs(peers) - 1) s_cnt[wid][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  {
    const int d = threadIdx.x;
    int run = 0;
    for (int w = 0; w < RS_WARPS; ++w) {
      const int c = s_cnt[w][d];
      s_cnt[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int s = 0; s < RS_IPT; ++s) {
    if (dig[s] < 0) continue;
    const int64_t pos = (int64_t)s_base[dig[s]] + s_cnt[wid][dig[s]] + rank[s];
    kout[pos] = key[s];
    vout[pos] = val[s];
  }
}

// sorts keys[0]/vals[0] over n entries; 8 passes, so the result is back in keys[0]/vals[0]
int radix_sort(SceneWs& w, int64_t n, cudaStream_t st) {
  const int64_t nt = rs_tiles(n);
  for (int pass = 0; pass < 8; ++pass) {
    const int a = pass & 1, shift = 8 * pass;
    radix_hist_kernel<<<(unsigned)nt, RS_T, 0, st>>>(w.keys[a], n, shift, nt, w.hist);
    R3DFS_CHECK_LAUNCH();
    R3DFS_TRY(scan_excl(w.hist, 256 * nt, w.bsum, &w.hdr->scratch, st));
    radix_scatter_kernel<<<(unsigned)nt, RS_T, 0, st>>>(w.keys[a], w.vals[a], w.keys[a ^ 1],
                                                         w.vals[a ^ 1], n, shift, nt, w.hist);
    R3DFS_CHECK_LAUNCH();
  }
  return 0;
}

// ---- plan kernels ------------------------------------------------------------------------------
__global__ __launch_bounds__(256) void scene_bbox_kernel(const float* __restrict__ pts, int64_t M,
                                                         int64_t s_m, int64_t s_c,
                                                         float* __restrict__ part) {
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY, bad = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float x = pts[i * s_m], y = pts[i * s_m + s_c];
    if (!isfinite(x) || !isfinite(y)) bad = 1.f;
    mnx = fminf(mnx, x);
    mny = fminf(mny, y);
    mxx = fmaxf(mxx, x);
    mxy = fmaxf(mxy, y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
    mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
    bad = fmaxf(bad, __shfl_xor_sync(0xffffffffu, bad, o));
  }
  __shared__ float s[8][5];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) {
    s[wid][0] = mnx;
    s[wid][1] = mny;
    s[wid][2] = mxx;
    s[wid][3] = mxy;
    s[wid][4] = bad;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) {
      s[0][0] = fminf(s[0][0], s[w][0]);
      s[0][1] = fminf(s[0][1], s[w][1]);
      s[0][2] = fmaxf(s[0][2], s[w][2]);
      s[0][3] = fmaxf(s[0][3], s[w][3]);
      s[0][4] = fmaxf(s[0][4], s[w][4]);
    }
    for (int c = 0; c < 5; ++c) part[blockIdx.x * 5 + c] = s[0][c];
  }
}

// n_cells = max(1, floor(ext / stride + 0.5)) in fp32; 0 when it does not fit the grid's int32
__device__ int64_t n_cells_of(float ext, float stride) {
  const float q = floorf(__fadd_rn(__fdiv_rn(ext, stride), 0.5f));
  if (!(q < 2147483648.f)) return 0;
  return q < 1.f ? 1 : (int64_t)q;
}

__global__ void scene_grid_kernel(const float* __restrict__ part, float block_size, int r,
                                  SceneHdr* __restrict__ h) {
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY, bad = 0.f;
  for (int c = 0; c < BBOX_CTAS; ++c) {
    mnx = fminf(mnx, part[c * 5 + 0]);
    mny = fminf(mny, part[c * 5 + 1]);
    mxx = fmaxf(mxx, part[c * 5 + 2]);
    mxy = fmaxf(mxy, part[c * 5 + 3]);
    bad = fmaxf(bad, part[c * 5 + 4]);
  }
  const float stride = __fdiv_rn(block_size, (float)r);
  const int64_t ncx = n_cells_of(__fsub_rn(mxx, mnx), stride);
  const int64_t ncy = n_cells_of(__fsub_rn(mxy, mny), stride);
  const int64_t nbx = ncx > r ? ncx - r + 1 : 1, nby = ncy > r ? ncy - r + 1 : 1;
  const bool err = bad != 0.f || ncx == 0 || ncy == 0 || nbx * nby >= (int64_t)1 << 31;
  h->x0 = mnx;
  h->y0 = mny;
  h->stride = stride;
  h->ncx = err ? 1 : (int32_t)ncx;
  h->ncy = err ? 1 : (int32_t)ncy;
  h->nbx = err ? 1 : (int32_t)nbx;
  h->nby = err ? 1 : (int32_t)nby;
  h->err = err ? 1 : 0;
}

struct BlockRange {
  int lx, hx, ly, hy;
};

__device__ __forceinline__ BlockRange block_range(const float* __restrict__ pts, int64_t i,
                                                  int64_t s_m, int64_t s_c, const SceneHdr& h,
                                                  int r) {
  const int u = cell_of(pts[i * s_m], h.x0, h.stride, h.ncx);
  const int v = cell_of(pts[i * s_m + s_c], h.y0, h.stride, h.ncy);
  return BlockRange{max(0, u - r + 1), min(u, h.nbx - 1), max(0, v - r + 1), min(v, h.nby - 1)};
}

// off[i] = number of blocks containing point i (0 on a grid error); off[M] = 0
__global__ void scene_count_kernel(const float* __restrict__ pts, int64_t M, int64_t s_m,
                                   int64_t s_c, int r, const SceneHdr* __restrict__ hp,
                                   int32_t* __restrict__ off) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > M) return;
  const SceneHdr h = *hp;
  if (i == M || h.err) {
    off[i] = 0;
    return;
  }
  const BlockRange b = block_range(pts, i, s_m, s_c, h, r);
  off[i] = (b.hx - b.lx + 1) * (b.hy - b.ly + 1);
}

// one record per membership, in point order and, within a point, ascending block id
__global__ void scene_emit_kernel(const float* __restrict__ pts, int64_t M, int64_t s_m,
                                  int64_t s_c, int r, uint32_t seed_hash,
                                  const SceneHdr* __restrict__ hp, const int32_t* __restrict__ off,
                                  uint64_t* __restrict__ keys, int32_t* __restrict__ vals,
                                  int32_t* __restrict__ mem_point) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const SceneHdr h = *hp;
  if (h.err) return;
  const BlockRange b = block_range(pts, i, s_m, s_c, h, r);
  const uint64_t k = lowbias32((uint32_t)i ^ seed_hash);
  int32_t t = off[i];
  for (int ix = b.lx; ix <= b.hx; ++ix)
    for (int iy = b.ly; iy <= b.hy; ++iy, ++t) {
      keys[t] = ((uint64_t)((int64_t)ix * h.nby + iy) << 32) | k;
      vals[t] = t;
      mem_point[t] = (int32_t)i;
    }
}

// records past T sort last
__global__ void scene_pad_kernel(int64_t n, const SceneHdr* __restrict__ hp,
                                 uint64_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n || p < hp->T) return;
  keys[p] = ~0ull;
  vals[p] = (int32_t)p;
}

__device__ __forceinline__ bool block_starts(const uint64_t* __restrict__ keys, int64_t p) {
  return p == 0 || (keys[p] >> 32) != (keys[p - 1] >> 32);
}

// seg[p] = 1 where sorted record p opens a block (p < T), 0 elsewhere, over n + 1 entries
__global__ void scene_flag_kernel(int64_t n, const SceneHdr* __restrict__ hp,
                                  const uint64_t* __restrict__ keys, int32_t* __restrict__ seg) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p > n) return;
  seg[p] = p < hp->T && block_starts(keys, p) ? 1 : 0;
}

__global__ void scene_seg_start_kernel(int64_t n, const SceneHdr* __restrict__ hp,
                                       const uint64_t* __restrict__ keys,
                                       const int32_t* __restrict__ seg,
                                       int32_t* __restrict__ seg_start) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int32_t T = hp->T;
  if (p == 0) seg_start[hp->n_seg] = T;
  if (p < T && block_starts(keys, p)) seg_start[seg[p]] = (int32_t)p;
}

// chunk_off[s] = ceil(n_b / N) for the n_seg blocks, 0 up to n + 1 entries
__global__ void scene_block_chunks_kernel(int64_t n, int N, const SceneHdr* __restrict__ hp,
                                          const int32_t* __restrict__ seg_start,
                                          int32_t* __restrict__ chunk_off) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > n) return;
  int32_t c = 0;
  if (s < hp->n_seg) {
    const int32_t nb = seg_start[s + 1] - seg_start[s];
    c = (nb + N - 1) / N;
  }
  chunk_off[s] = c;
}

// member of rank rho of a block with C_b chunks -> chunk rho mod C_b, slot rho div C_b; stored at
// the membership's position in point order
__global__ void scene_member_kernel(int64_t n, int N, SceneHdr* __restrict__ hp,
                                    const uint64_t* __restrict__ keys,
                                    const int32_t* __restrict__ vals,
                                    const int32_t* __restrict__ seg,
                                    const int32_t* __restrict__ seg_start,
                                    const int32_t* __restrict__ chunk_off,
                                    int32_t* __restrict__ chunk_seg,
                                    int32_t* __restrict__ mem_chunk,
                                    int32_t* __restrict__ mem_slot, int64_t* __restrict__ n_chunks) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p == 0) *n_chunks = hp->err ? -1 : (int64_t)hp->n_chunks;
  if (p >= n || p >= hp->T) return;
  const int32_t s = block_starts(keys, p) ? seg[p] : seg[p] - 1;
  const int32_t rho = (int32_t)p - seg_start[s];
  const int32_t c0 = chunk_off[s], cb = chunk_off[s + 1] - c0;
  const int32_t c = c0 + rho % cb, slot = rho / cb;
  const int32_t t = vals[p];
  mem_chunk[t] = c;
  mem_slot[t] = slot;
  if (slot == 0) chunk_seg[c] = s;
}

// ---- chunk clouds ------------------------------------------------------------------------------
// A cloud of N slots over `count` members of one block: slot q holds the member of sorted record
// first + (q mod count) * stride + offset, normalised over those members.  One CTA of 256 threads.
__device__ __forceinline__ void scene_cloud(const float* __restrict__ pts, int64_t s_m, int64_t s_c,
                                            int N, const int32_t* __restrict__ vals,
                                            const int32_t* __restrict__ mem_point, int32_t first,
                                            int32_t stride, int32_t offset, int32_t count,
                                            float* __restrict__ out, int32_t* __restrict__ src) {
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int q = threadIdx.x; q < count; q += blockDim.x) {
    const int64_t i = mem_point[vals[first + (int64_t)q * stride + offset]];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float v = pts[i * s_m + k * s_c];
      mn[k] = fminf(mn[k], v);
      mx[k] = fmaxf(mx[k], v);
    }
  }
  __shared__ float s_mn[8][3], s_mx[8][3], s_min[3], s_e[3];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
      mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
    }
    if (lane == 0) {
      s_mn[wid][k] = mn[k];
      s_mx[wid][k] = mx[k];
    }
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int k = threadIdx.x;
    float a = s_mn[0][k], b = s_mx[0][k];
    for (int w = 1; w < 8; ++w) {
      a = fminf(a, s_mn[w][k]);
      b = fmaxf(b, s_mx[w][k]);
    }
    // max over the chunk of fl(x - m) is fl(max x - m): a correctly rounded subtraction is monotone
    s_min[k] = a;
    s_e[k] = __fsub_rn(b, a);
  }
  __syncthreads();
  for (int q = threadIdx.x; q < N; q += blockDim.x) {
    const int32_t i = mem_point[vals[first + (int64_t)(q % count) * stride + offset]];
    const float* pt = pts + (int64_t)i * s_m;
    float* o = out + (int64_t)q * 9;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float d = __fsub_rn(pt[k * s_c], s_min[k]);
      o[k] = d;
      o[6 + k] = s_e[k] > 0.f ? __fdiv_rn(d, s_e[k]) : 0.f;
      o[3 + k] = __fdiv_rn(pt[(3 + k) * s_c], 255.f);
    }
    src[q] = i;
  }
}

// a cloud with no members: zeros, src -1
__device__ __forceinline__ void scene_cloud_empty(int N, float* __restrict__ out,
                                                  int32_t* __restrict__ src) {
  for (int q = threadIdx.x; q < N; q += blockDim.x) {
    src[q] = -1;
    for (int k = 0; k < 9; ++k) out[(int64_t)q * 9 + k] = 0.f;
  }
}

// One CTA per chunk.  Slot q of chunk j of a block with n_b members in C_b chunks holds the member
// of rank (q mod count_j) * C_b + j, count_j = ceil((n_b - j) / C_b).
__global__ __launch_bounds__(256) void scene_chunk_kernel(
    const float* __restrict__ pts, int64_t s_m, int64_t s_c, int N,
    const SceneHdr* __restrict__ hp, const int32_t* __restrict__ vals,
    const int32_t* __restrict__ mem_point, const int32_t* __restrict__ seg_start,
    const int32_t* __restrict__ chunk_off, const int32_t* __restrict__ chunk_seg,
    float* __restrict__ chunk_x, int32_t* __restrict__ chunk_src) {
  const int64_t c = blockIdx.x;
  float* out = chunk_x + c * N * 9;
  int32_t* src = chunk_src + c * N;
  if (c >= hp->n_chunks) {  // more chunks asked for than the plan made
    scene_cloud_empty(N, out, src);
    return;
  }
  const int32_t s = chunk_seg[c], c0 = chunk_off[s], cb = chunk_off[s + 1] - c0;
  const int32_t j = (int32_t)c - c0, p0 = seg_start[s], nb = seg_start[s + 1] - p0;
  const int32_t cnt = (nb - j + cb - 1) / cb;
  scene_cloud(pts, s_m, s_c, N, vals, mem_point, p0, cb, j, cnt, out, src);
}

// ---- merge ---------------------------------------------------------------------------------------
// One thread per point: its memberships in ascending block id, sequential fp32 sums, one division.
__global__ void scene_merge_kernel(const float* __restrict__ logits, int64_t M, int N, int nc,
                                   int64_t n_chunks, const int32_t* __restrict__ off,
                                   const int32_t* __restrict__ mem_chunk,
                                   const int32_t* __restrict__ mem_slot, float* __restrict__ out,
                                   int32_t* __restrict__ pred, int32_t* __restrict__ coverage) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  float acc[MAX_CLS];
#pragma unroll
  for (int k = 0; k < MAX_CLS; ++k) acc[k] = 0.f;
  int cov = 0;
  for (int32_t t = off[i]; t < off[i + 1]; ++t) {
    const int32_t c = mem_chunk[t];
    if (c >= n_chunks) continue;
    const float* row = logits + ((int64_t)c * N + mem_slot[t]) * nc;
#pragma unroll
    for (int k = 0; k < MAX_CLS; ++k)
      if (k < nc) acc[k] = __fadd_rn(acc[k], row[k]);
    ++cov;
  }
  const float den = (float)cov;
  float mx = -INFINITY;
  int am = 0;
#pragma unroll
  for (int k = 0; k < MAX_CLS; ++k) {
    if (k >= nc) break;
    const float v = __fdiv_rn(acc[k], den);
    out[i * nc + k] = v;
    if (v > mx) {  // the episode head's rule (query_head_kernel): first maximum
      mx = v;
      am = k;
    }
  }
  if (pred) pred[i] = am;
  if (coverage) coverage[i] = cov;
}

// ---- support shots -----------------------------------------------------------------------------
// Each way keeps the eligible blocks with the 32 smallest keys (k_shot <= 32) as a sorted list of
// (key << 32 | segment), one entry per lane; keys are a bijection of the block id, so no two
// entries of a way are equal.  Empty entries are ~0.  A fixed grid of CTAs keeps one list per way
// and CTA; one CTA per way merges them.
constexpr int SUP_CTAS = 128, SUP_T = 256, SUP_WARPS = SUP_T / 32, SUP_U = 8;
constexpr int MAX_WAY = 7, MAX_SHOT = 32;
constexpr uint64_t TOP_EMPTY = ~0ull;

struct SupportSel {
  int32_t cls[MAX_WAY];
  uint32_t wkey[MAX_WAY];  // lowbias32(lowbias32(seed) + w + 1)
  int32_t n_way, min_points;
  double min_ratio;
};

struct SupportWs {
  uint64_t* part_top;  // (SUP_CTAS, n_way, 32) per-CTA lists
  int32_t* part_n;     // (SUP_CTAS, n_way) per-CTA eligible counts
  int32_t* shot_seg;   // (n_way, k_shot) segment of every shot, -1 = missing
};

void carve_support(WsBump& ws, int n_way, int k_shot, SupportWs& w) {
  w.part_top = ws.take<uint64_t>((size_t)SUP_CTAS * n_way * MAX_SHOT);
  w.part_n = ws.take<int32_t>((size_t)SUP_CTAS * n_way);
  w.shot_seg = ws.take<int32_t>((size_t)n_way * k_shot);
}

// v (warp-uniform) into the lane-distributed sorted list
__device__ __forceinline__ uint64_t top_insert(uint64_t list, uint64_t v) {
  const int lane = threadIdx.x & 31;
  const int pos = __popc(__ballot_sync(0xffffffffu, list < v));
  const uint64_t up = __shfl_up_sync(0xffffffffu, list, 1);
  return lane < pos ? list : lane == pos ? v : up;
}

// number of entries of the sorted 32-entry list x below v
__device__ __forceinline__ int count_below(const uint64_t* x, uint64_t v) {
  int n = 0;
#pragma unroll
  for (int st = 16; st > 0; st >>= 1)
    if (x[n + st - 1] < v) n += st;
  return n + (x[n] < v ? 1 : 0);
}

// out = the 32 smallest of the sorted lists a and b (shared memory; out may be a).  One warp.
__device__ __forceinline__ void top_merge(uint64_t* a, const uint64_t* b, uint64_t* out) {
  const int lane = threadIdx.x & 31;
  const uint64_t va = a[lane], vb = b[lane];
  const int ra = lane + count_below(b, va), rb = lane + count_below(a, vb);
  __syncwarp();
  if (ra < 32) out[ra] = va;
  if (rb < 32) out[rb] = vb;
  __syncwarp();
}

// One warp per block segment: counts its members of every way's class (vals -> mem_point ->
// labels, each membership read once), tests eligibility and inserts the block into the warp's
// lists; then the CTA merges its warps' lists.  Segment s goes to CTA s mod SUP_CTAS, so the few
// segments of a small scan spread over the SMs.
__global__ __launch_bounds__(SUP_T) void scene_support_count_kernel(
    const SceneHdr* __restrict__ hp, const uint64_t* __restrict__ keys,
    const int32_t* __restrict__ vals, const int32_t* __restrict__ mem_point,
    const int32_t* __restrict__ seg_start, const int32_t* __restrict__ labels, SupportSel sel,
    uint64_t* __restrict__ part_top, int32_t* __restrict__ part_n) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int32_t n_seg = hp->n_seg;
  uint64_t top[MAX_WAY];
  int n_el[MAX_WAY];
#pragma unroll
  for (int w = 0; w < MAX_WAY; ++w) {
    top[w] = TOP_EMPTY;
    n_el[w] = 0;
  }
  for (int32_t s = wid * SUP_CTAS + blockIdx.x; s < n_seg; s += SUP_CTAS * SUP_WARPS) {
    const int32_t p0 = seg_start[s], nb = seg_start[s + 1] - p0;
    int cnt[MAX_WAY];
#pragma unroll
    for (int w = 0; w < MAX_WAY; ++w) cnt[w] = 0;
    for (int32_t base = 0; base < nb; base += 32 * SUP_U) {
      int32_t t[SUP_U];
#pragma unroll
      for (int u = 0; u < SUP_U; ++u) {
        const int32_t q = base + u * 32 + lane;
        t[u] = q < nb ? vals[p0 + q] : -1;
      }
#pragma unroll
      for (int u = 0; u < SUP_U; ++u) t[u] = t[u] >= 0 ? mem_point[t[u]] : -1;
#pragma unroll
      for (int u = 0; u < SUP_U; ++u) {
        if (t[u] < 0) continue;
        const int32_t l = labels[t[u]];
#pragma unroll
        for (int w = 0; w < MAX_WAY; ++w) cnt[w] += (w < sel.n_way && l == sel.cls[w]) ? 1 : 0;
      }
    }
    // max(floor(n_b * min_ratio), min_points), the product in fp64 as Python's int(n_b * 0.05)
    const double thr = fmax(floor((double)nb * sel.min_ratio), (double)sel.min_points);
    const uint32_t b = (uint32_t)(keys[p0] >> 32);
#pragma unroll
    for (int w = 0; w < MAX_WAY; ++w) {
      if (w >= sel.n_way) continue;
      const int c = __reduce_add_sync(0xffffffffu, cnt[w]);
      if ((double)c > thr) {
        ++n_el[w];
        top[w] = top_insert(top[w], ((uint64_t)lowbias32(b ^ sel.wkey[w]) << 32) | (uint32_t)s);
      }
    }
  }
  __shared__ uint64_t s_top[SUP_WARPS][MAX_WAY][32];
  __shared__ int s_n[SUP_WARPS][MAX_WAY];
#pragma unroll
  for (int w = 0; w < MAX_WAY; ++w) {
    s_top[wid][w][lane] = top[w];
    if (lane == 0) s_n[wid][w] = n_el[w];
  }
  __syncthreads();
  if (wid >= sel.n_way) return;
  const int w = wid;
  for (int o = 1; o < SUP_WARPS; ++o) top_merge(s_top[0][w], s_top[o][w], s_top[0][w]);
  const int n = __reduce_add_sync(0xffffffffu, lane < SUP_WARPS ? s_n[lane][w] : 0);
  part_top[((int64_t)blockIdx.x * sel.n_way + w) * 32 + lane] = s_top[0][w][lane];
  if (lane == 0) part_n[blockIdx.x * sel.n_way + w] = n;
}

// One CTA per way: merges the SUP_CTAS lists, keeps the first k_shot entries as the way's shots.
__global__ __launch_bounds__(SUP_T) void scene_support_pick_kernel(
    const SceneHdr* __restrict__ hp, const uint64_t* __restrict__ keys,
    const int32_t* __restrict__ seg_start, const uint64_t* __restrict__ part_top,
    const int32_t* __restrict__ part_n, int n_way, int k_shot, int32_t* __restrict__ shot_seg,
    int32_t* __restrict__ shot_block, int32_t* __restrict__ n_eligible) {
  __shared__ uint64_t s_p[SUP_CTAS][32];
  __shared__ int s_n[SUP_WARPS];
  const int w = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < SUP_CTAS * 32; i += SUP_T)
    s_p[i >> 5][i & 31] = part_top[((int64_t)(i >> 5) * n_way + w) * 32 + (i & 31)];
  int n = 0;
  for (int g = threadIdx.x; g < SUP_CTAS; g += SUP_T) n += part_n[g * n_way + w];
  n = __reduce_add_sync(0xffffffffu, n);
  if (lane == 0) s_n[wid] = n;
  __syncthreads();
  for (int g = wid + SUP_WARPS; g < SUP_CTAS; g += SUP_WARPS) top_merge(s_p[wid], s_p[g], s_p[wid]);
  __syncthreads();
  if (wid != 0) return;
  for (int o = 1; o < SUP_WARPS; ++o) top_merge(s_p[0], s_p[o], s_p[0]);
  const bool err = hp->err != 0;
  if (lane < k_shot) {
    const uint64_t v = s_p[0][lane];
    const int32_t s = err || v == TOP_EMPTY ? -1 : (int32_t)(uint32_t)v;
    shot_seg[w * k_shot + lane] = s;
    shot_block[w * k_shot + lane] = s < 0 ? -1 : (int32_t)(keys[seg_start[s]] >> 32);
  }
  if (lane == 0) {
    int tot = 0;
    for (int i = 0; i < SUP_WARPS; ++i) tot += s_n[i];
    n_eligible[w] = err ? -1 : tot;
  }
}

// One CTA per shot: the block's first min(n_b, N) members in rank order, repeated to N slots, by
// the chunk clouds' code; mask = label == the way's class.
__global__ __launch_bounds__(256) void scene_support_cloud_kernel(
    const float* __restrict__ pts, int64_t s_m, int64_t s_c, int N,
    const int32_t* __restrict__ labels, const __grid_constant__ SupportSel sel, int k_shot,
    const int32_t* __restrict__ vals, const int32_t* __restrict__ mem_point,
    const int32_t* __restrict__ seg_start, const int32_t* __restrict__ shot_seg,
    float* __restrict__ support_x, int32_t* __restrict__ support_y,
    int32_t* __restrict__ support_src) {
  const int64_t g = blockIdx.x;
  float* out = support_x + g * N * 9;
  int32_t* src = support_src + g * N;
  int32_t* y = support_y + g * N;
  const int32_t s = shot_seg[g];
  if (s < 0) {
    scene_cloud_empty(N, out, src);
    for (int q = threadIdx.x; q < N; q += blockDim.x) y[q] = 0;
    return;
  }
  const int32_t p0 = seg_start[s], nb = seg_start[s + 1] - p0;
  scene_cloud(pts, s_m, s_c, N, vals, mem_point, p0, 1, 0, min(nb, N), out, src);
  const int32_t cls = sel.cls[g / k_shot];
  for (int q = threadIdx.x; q < N; q += blockDim.x) y[q] = labels[src[q]] == cls ? 1 : 0;
}

int scene_common_checks(int64_t M, int overlap, int n_points) {
  if (M <= 0) return R3DFS_E_BADARG;
  if (overlap < 1 || overlap > 4 || n_points < 64 || n_points > 65536) return R3DFS_E_UNSUPPORTED;
  if (scene_tmax(M, overlap) >= ((int64_t)1 << 31)) return R3DFS_E_UNSUPPORTED;
  return 0;
}

}  // namespace

extern "C" {

size_t r3dfs_scene_workspace(int64_t M, int overlap) {
  if (M <= 0 || overlap < 1 || overlap > 4 || scene_tmax(M, overlap) >= ((int64_t)1 << 31))
    return 0;
  WsBump ws(nullptr, 0);
  SceneWs w;
  carve_scene(ws, M, overlap, w);
  return align_up(ws.off, 256);
}

int r3dfs_scene_plan(const float* points, int64_t M, int64_t s_m, int64_t s_c, float block_size,
                     int overlap, uint32_t seed, int n_points, int64_t* n_chunks, void* wsp,
                     size_t ws_bytes, r3dfs_stream_t stream) {
  if (!points || !n_chunks || !wsp || !(block_size > 0.f) || !isfinite(block_size))
    return R3DFS_E_BADARG;
  R3DFS_TRY(scene_common_checks(M, overlap, n_points));
  if (ws_bytes < r3dfs_scene_workspace(M, overlap)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  SceneWs w;
  carve_scene(ws, M, overlap, w);
  const int64_t T = scene_tmax(M, overlap);
  scene_bbox_kernel<<<BBOX_CTAS, 256, 0, st>>>(points, M, s_m, s_c, w.bbox);
  R3DFS_CHECK_LAUNCH();
  scene_grid_kernel<<<1, 1, 0, st>>>(w.bbox, block_size, overlap, w.hdr);
  R3DFS_CHECK_LAUNCH();
  scene_count_kernel<<<nblk(M + 1), 256, 0, st>>>(points, M, s_m, s_c, overlap, w.hdr, w.off);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(scan_excl(w.off, M + 1, w.bsum, &w.hdr->T, st));
  scene_emit_kernel<<<nblk(M), 256, 0, st>>>(points, M, s_m, s_c, overlap, lowbias32(seed), w.hdr,
                                              w.off, w.keys[0], w.vals[0], w.mem_point);
  R3DFS_CHECK_LAUNCH();
  scene_pad_kernel<<<nblk(T), 256, 0, st>>>(T, w.hdr, w.keys[0], w.vals[0]);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(radix_sort(w, T, st));
  scene_flag_kernel<<<nblk(T + 1), 256, 0, st>>>(T, w.hdr, w.keys[0], w.seg);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(scan_excl(w.seg, T + 1, w.bsum, &w.hdr->n_seg, st));
  scene_seg_start_kernel<<<nblk(T), 256, 0, st>>>(T, w.hdr, w.keys[0], w.seg, w.seg_start);
  R3DFS_CHECK_LAUNCH();
  scene_block_chunks_kernel<<<nblk(T + 1), 256, 0, st>>>(T, n_points, w.hdr, w.seg_start,
                                                         w.chunk_off);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(scan_excl(w.chunk_off, T + 1, w.bsum, &w.hdr->n_chunks, st));
  scene_member_kernel<<<nblk(T), 256, 0, st>>>(T, n_points, w.hdr, w.keys[0], w.vals[0], w.seg,
                                                w.seg_start, w.chunk_off, w.chunk_seg, w.mem_chunk,
                                                w.mem_slot, n_chunks);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int r3dfs_scene_chunks(const float* points, int64_t M, int64_t s_m, int64_t s_c, int overlap,
                       int n_points, int64_t n_chunks, float* chunk_x, int32_t* chunk_src,
                       void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!points || !chunk_x || !chunk_src || !wsp || n_chunks <= 0) return R3DFS_E_BADARG;
  R3DFS_TRY(scene_common_checks(M, overlap, n_points));
  if (n_chunks > scene_tmax(M, overlap)) return R3DFS_E_BADARG;
  if (ws_bytes < r3dfs_scene_workspace(M, overlap)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  SceneWs w;
  carve_scene(ws, M, overlap, w);
  scene_chunk_kernel<<<(unsigned)n_chunks, 256, 0, st>>>(points, s_m, s_c, n_points, w.hdr,
                                                          w.vals[0], w.mem_point, w.seg_start,
                                                          w.chunk_off, w.chunk_seg, chunk_x,
                                                          chunk_src);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int r3dfs_scene_merge(const float* logits, int64_t M, int overlap, int n_points, int64_t n_chunks,
                      int n_cls, float* point_logits, int32_t* point_pred, int32_t* coverage,
                      void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!logits || !point_logits || !wsp || n_chunks <= 0) return R3DFS_E_BADARG;
  R3DFS_TRY(scene_common_checks(M, overlap, n_points));
  if (n_cls < 1 || n_cls > MAX_CLS) return R3DFS_E_UNSUPPORTED;
  if (n_chunks > scene_tmax(M, overlap)) return R3DFS_E_BADARG;
  if (ws_bytes < r3dfs_scene_workspace(M, overlap)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  SceneWs w;
  carve_scene(ws, M, overlap, w);
  scene_merge_kernel<<<nblk(M), 256, 0, st>>>(logits, M, n_points, n_cls, n_chunks, w.off,
                                               w.mem_chunk, w.mem_slot, point_logits, point_pred,
                                               coverage);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

size_t r3dfs_scene_support_workspace(int n_way, int k_shot) {
  if (n_way < 1 || n_way > MAX_WAY || k_shot < 1 || k_shot > MAX_SHOT) return 0;
  WsBump ws(nullptr, 0);
  SupportWs w;
  carve_support(ws, n_way, k_shot, w);
  return align_up(ws.off, 256);
}

int r3dfs_scene_support(const float* points, int64_t M, int64_t s_m, int64_t s_c,
                        const int32_t* labels, const int32_t* h_classes, int n_way, int k_shot,
                        int min_points, double min_ratio, uint32_t seed, int overlap, int n_points,
                        float* support_x, int32_t* support_y, int32_t* support_src,
                        int32_t* shot_block, int32_t* n_eligible, const void* plan_ws,
                        size_t plan_ws_bytes, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!points || !labels || !h_classes || !support_x || !support_y || !support_src ||
      !shot_block || !n_eligible || !plan_ws || !wsp)
    return R3DFS_E_BADARG;
  R3DFS_TRY(scene_common_checks(M, overlap, n_points));
  if (n_way < 1 || n_way > MAX_WAY || k_shot < 1 || k_shot > MAX_SHOT) return R3DFS_E_UNSUPPORTED;
  if (min_points < 0 || !(min_ratio >= 0.0 && min_ratio <= 1.0)) return R3DFS_E_BADARG;
  SupportSel sel{};
  for (int w = 0; w < n_way; ++w) {
    for (int v = 0; v < w; ++v)
      if (h_classes[v] == h_classes[w]) return R3DFS_E_BADARG;
    sel.cls[w] = h_classes[w];
    sel.wkey[w] = lowbias32(lowbias32(seed) + (uint32_t)w + 1u);
  }
  sel.n_way = n_way;
  sel.min_points = min_points;
  sel.min_ratio = min_ratio;
  if (plan_ws_bytes < r3dfs_scene_workspace(M, overlap)) return R3DFS_E_WORKSPACE;
  if (ws_bytes < r3dfs_scene_support_workspace(n_way, k_shot)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump pws(const_cast<void*>(plan_ws), plan_ws_bytes);
  SceneWs p;
  carve_scene(pws, M, overlap, p);
  WsBump ws(wsp, ws_bytes);
  SupportWs w;
  carve_support(ws, n_way, k_shot, w);
  scene_support_count_kernel<<<SUP_CTAS, SUP_T, 0, st>>>(p.hdr, p.keys[0], p.vals[0], p.mem_point,
                                                         p.seg_start, labels, sel, w.part_top,
                                                         w.part_n);
  R3DFS_CHECK_LAUNCH();
  scene_support_pick_kernel<<<n_way, SUP_T, 0, st>>>(p.hdr, p.keys[0], p.seg_start, w.part_top,
                                                     w.part_n, n_way, k_shot, w.shot_seg,
                                                     shot_block, n_eligible);
  R3DFS_CHECK_LAUNCH();
  scene_support_cloud_kernel<<<n_way * k_shot, 256, 0, st>>>(
      points, s_m, s_c, n_points, labels, sel, k_shot, p.vals[0], p.mem_point, p.seg_start,
      w.shot_seg, support_x, support_y, support_src);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
