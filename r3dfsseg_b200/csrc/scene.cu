// Whole-scan segmentation (include/r3dfs.h, "Segmenting a whole scan"): cut an (M, 6) scan into
// overlapping xy blocks, split every block into chunks of n_points sampled points normalised as the
// reference's loader does, and merge the per-chunk logits back onto the scan's points.
//
// r3dfs_scene_support ("Support shots from a labelled scan") reads the same plan to cut support
// shots out of a labelled scan: per-block class counts, a seeded choice of blocks per class, and
// shot clouds built by the chunk clouds' code.
//
// r3dfs_scene_index / r3dfs_scene_index_classes / r3dfs_scene_episodes ("Few-shot episodes from
// labelled scans") append planned scans to a dataset index (global blocks, members, class counts,
// per-class eligible lists) and sample few-shot episodes from it with the same shot clouds.
//
// r3dfs_scene_plan builds every index the other calls need and leaves it in the workspace:
//   bbox -> grid -> per-point membership counts -> scan -> one record (block << 32 | key, position)
//   per membership -> LSD radix sort -> block segments -> chunk counts -> scan -> (chunk, slot) of
//   every membership, stored back at its position in point order.
// Every step is integer arithmetic or a correctly rounded fp32 operation written out explicitly
// (__fsub_rn / __fdiv_rn), so that the numpy oracle of the tests reproduces it bit for bit, and no
// step uses a float atomic.
#include <algorithm>
#include <vector>

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
// Member q of a plan block: sorted record first + q * stride + offset.
struct PlanMembers {
  const int32_t* __restrict__ vals;
  const int32_t* __restrict__ mem_point;
  int32_t first, stride, offset;
  __device__ __forceinline__ int32_t operator()(int32_t q) const {
    return mem_point[vals[first + (int64_t)q * stride + offset]];
  }
};

// Member q of a dataset-index block: its q-th member in rank order.
struct IndexMembers {
  const int32_t* __restrict__ member;
  int64_t first;
  __device__ __forceinline__ int32_t operator()(int32_t q) const { return member[first + q]; }
};

// A cloud of N slots over `count` members of one block: slot q holds member q mod count,
// normalised over those members.  One CTA of 256 threads.
template <class Members>
__device__ __forceinline__ void scene_cloud(const float* __restrict__ pts, int64_t s_m, int64_t s_c,
                                            int N, const Members at, int32_t count,
                                            float* __restrict__ out, int32_t* __restrict__ src) {
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int q = threadIdx.x; q < count; q += blockDim.x) {
    const int64_t i = at(q);
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
    const int32_t i = at(q % count);
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
  scene_cloud(pts, s_m, s_c, N, PlanMembers{vals, mem_point, p0, cb, j}, cnt, out, src);
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
  scene_cloud(pts, s_m, s_c, N, PlanMembers{vals, mem_point, p0, 1, 0}, min(nb, N), out, src);
  const int32_t cls = sel.cls[g / k_shot];
  for (int q = threadIdx.x; q < N; q += blockDim.x) y[q] = labels[src[q]] == cls ? 1 : 0;
}

// ---- dataset index ----------------------------------------------------------------------------
constexpr int MAX_IDX_CLS = 64, IDX_T = 256, IDX_WARPS = IDX_T / 32;

struct IndexCls {
  int32_t id[MAX_IDX_CLS];  // class ids, ascending
  int32_t at[MAX_IDX_CLS];  // index of id[k] in the caller's class list
  int32_t n;
};

// block table and members of one planned scan, appended at (b0, m0)
__global__ void index_blocks_kernel(const SceneHdr* __restrict__ hp,
                                    const uint64_t* __restrict__ keys,
                                    const int32_t* __restrict__ seg_start, int32_t scan, int64_t b0,
                                    int64_t m0, int64_t* __restrict__ block_off,
                                    int32_t* __restrict__ block_scan,
                                    int32_t* __restrict__ block_id) {
  const int32_t s = blockIdx.x * blockDim.x + threadIdx.x, n_seg = hp->n_seg;
  if (s > n_seg) return;
  block_off[b0 + s] = m0 + seg_start[s];
  if (s == n_seg) return;
  block_scan[b0 + s] = scan;
  block_id[b0 + s] = (int32_t)(keys[seg_start[s]] >> 32);
}

__global__ void index_members_kernel(int64_t T, const int32_t* __restrict__ vals,
                                     const int32_t* __restrict__ mem_point, int64_t m0,
                                     int32_t point_base, int32_t* __restrict__ member) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < T) member[m0 + p] = point_base + mem_point[vals[p]];
}

// One warp per block: class counts of its members.  Lanes holding the same class are counted by
// their lowest lane (__match_any_sync), so no two lanes write one counter.
__global__ __launch_bounds__(IDX_T) void index_count_kernel(
    const SceneHdr* __restrict__ hp, const int32_t* __restrict__ vals,
    const int32_t* __restrict__ mem_point, const int32_t* __restrict__ seg_start,
    const int32_t* __restrict__ labels, const __grid_constant__ IndexCls cls, int64_t b0,
    int32_t* __restrict__ count) {
  __shared__ int s_cnt[IDX_WARPS][MAX_IDX_CLS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int32_t s = blockIdx.x * IDX_WARPS + wid;
  if (s >= hp->n_seg) return;
  for (int k = lane; k < MAX_IDX_CLS; k += 32) s_cnt[wid][k] = 0;
  __syncwarp();
  const int32_t p0 = seg_start[s], nb = seg_start[s + 1] - p0;
  for (int32_t base = 0; base < nb; base += 32) {
    int k = -1;
    if (base + lane < nb) {
      const int32_t l = labels[mem_point[vals[p0 + base + lane]]];
      int lo = 0, hi = cls.n;  // first id >= l
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cls.id[mid] < l) lo = mid + 1; else hi = mid;
      }
      if (lo < cls.n && cls.id[lo] == l) k = cls.at[lo];
    }
    const unsigned peers = __match_any_sync(0xffffffffu, k);
    if (k >= 0 && lane == __ffs(peers) - 1) s_cnt[wid][k] += __popc(peers);
    __syncwarp();
  }
  for (int k = lane; k < cls.n; k += 32) count[(b0 + s) * cls.n + k] = s_cnt[wid][k];
}

// flag[c * n_blocks + b] = block b is eligible for class c; flag[n_cls * n_blocks] = 0
__global__ void index_flag_kernel(const int64_t* __restrict__ block_off,
                                  const int32_t* __restrict__ count, int64_t n_blocks, int n_cls,
                                  int min_points, double min_ratio, int32_t* __restrict__ flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = n_blocks * n_cls;
  if (i > n) return;
  if (i == n) {
    flag[i] = 0;
    return;
  }
  const int64_t c = i / n_blocks, b = i - c * n_blocks;
  const int64_t nb = block_off[b + 1] - block_off[b];
  // max(floor(n_b * min_ratio), min_points), the rule of scene_support_count_kernel
  const double thr = fmax(floor((double)nb * min_ratio), (double)min_points);
  flag[i] = (double)count[b * n_cls + c] > thr ? 1 : 0;
}

// after the exclusive scan: entry i is eligible iff pos[i + 1] > pos[i]
__global__ void index_lists_kernel(const int32_t* __restrict__ pos, int64_t n_blocks, int n_cls,
                                   int32_t* __restrict__ elig_off,
                                   int32_t* __restrict__ elig_block) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = n_blocks * n_cls;
  if (i > n) return;
  if (i % n_blocks == 0) elig_off[i / n_blocks] = pos[i];
  if (i < n && pos[i + 1] > pos[i]) elig_block[pos[i]] = (int32_t)(i % n_blocks);
}

// ---- episodes ---------------------------------------------------------------------------------
enum { NOISE_NONE = 0, NOISE_OOD = 1, NOISE_SYM = 2, NOISE_PAIR = 3 };
constexpr int EP_T = 256, EP_WARPS = EP_T / 32;

struct EpisodeArgs {
  uint32_t seed_hash;  // lowbias32(seed)
  int64_t first, step;
  int n_way, k_shot, n_queries, n_cls, noise_type;
};

// the host arrays, copied into the workspace as one block of int32
struct EpisodeHost {
  int32_t* way;      // (E, n_way) class index of every way
  int32_t* n_noise;  // (E)
  int32_t* cls;      // (n_cls) class ids
  int32_t* pair;     // (n_cls) class index of pair[c]
};

struct EpisodeWs {
  int32_t* host;   // the EpisodeHost block
  int32_t* noisy;  // (E, n_way, k_shot) 1 = noisy shot
};

__host__ __device__ inline size_t ep_host_ints(int E, int n_way, int n_cls) {
  return (size_t)E * n_way + E + 2 * (size_t)n_cls;
}

__host__ __device__ inline EpisodeHost ep_host_view(int32_t* p, int E, int n_way, int n_cls) {
  EpisodeHost h;
  h.way = p;
  h.n_noise = h.way + (size_t)E * n_way;
  h.cls = h.n_noise + E;
  h.pair = h.cls + n_cls;
  return h;
}

void carve_episodes(WsBump& ws, int E, int n_way, int k_shot, int n_cls, EpisodeWs& w) {
  w.host = ws.take<int32_t>(ep_host_ints(E, n_way, n_cls));
  w.noisy = ws.take<int32_t>((size_t)E * n_way * k_shot);
}

__host__ __device__ inline uint32_t hkey(uint32_t a, uint32_t b) {
  return lowbias32(a ^ lowbias32(b));
}

// One CTA per (episode, way): the way's clean shots and query blocks (the smallest keys of its
// class's eligible list), the noise class and block of every noisy shot, and the keyed shuffle.
__global__ __launch_bounds__(EP_T) void episode_select_kernel(
    const int32_t* __restrict__ elig_off, const int32_t* __restrict__ elig_block,
    const EpisodeArgs a, const int32_t* __restrict__ hbuf, int E, int32_t* __restrict__ noisy,
    int32_t* __restrict__ shot_block, int32_t* __restrict__ support_flag,
    int32_t* __restrict__ query_block) {
  __shared__ uint64_t s_top[EP_WARPS][32];
  __shared__ int32_t s_range[MAX_IDX_CLS], s_perm[MAX_IDX_CLS], s_ncls[MAX_SHOT],
      s_nblk[MAX_SHOT], s_n_range;
  __shared__ uint32_t s_okey[MAX_SHOT];
  const EpisodeHost h = ep_host_view(const_cast<int32_t*>(hbuf), E, a.n_way, a.n_cls);
  const int e = blockIdx.x / a.n_way, w = blockIdx.x % a.n_way;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int n_noise = h.n_noise[e], k_clean = a.k_shot - n_noise;
  const int c = h.way[e * a.n_way + w];
  const uint32_t ke = hkey(a.seed_hash, (uint32_t)(a.first + (int64_t)e * a.step));
  const uint32_t kw = hkey(ke, (uint32_t)w + 1u);

  // clean shots and queries: the k_clean + n_queries smallest lowbias32(b ^ kw)
  const int32_t l0 = elig_off[c], ln = elig_off[c + 1] - l0;
  uint64_t top = TOP_EMPTY;
  for (int32_t base = wid * 32; base < ln; base += EP_T) {
    const int32_t q = base + lane;
    const uint64_t v = q < ln ? ((uint64_t)lowbias32((uint32_t)elig_block[l0 + q] ^ kw) << 32) |
                                    (uint32_t)elig_block[l0 + q]
                              : TOP_EMPTY;
    const uint64_t thr = __shfl_sync(0xffffffffu, top, 31);
    for (unsigned m = __ballot_sync(0xffffffffu, v < thr); m; m &= m - 1)
      top = top_insert(top, __shfl_sync(0xffffffffu, v, __ffs(m) - 1));
  }
  s_top[wid][lane] = top;

  // noise range: ood = the index's classes with an eligible block that no way holds, ascending;
  // sym = the other ways' classes in way order; pair = pair[c]
  if (threadIdx.x == 0) {
    int n = 0;
    if (a.noise_type == NOISE_OOD) {
      for (int k = 0; k < a.n_cls; ++k) {
        bool used = elig_off[k + 1] == elig_off[k];
        for (int v = 0; v < a.n_way; ++v) used |= h.way[e * a.n_way + v] == k;
        if (!used) s_range[n++] = k;
      }
    } else if (a.noise_type == NOISE_SYM) {
      for (int v = 0; v < a.n_way; ++v)
        if (v != w) s_range[n++] = h.way[e * a.n_way + v];
    } else if (a.noise_type == NOISE_PAIR) {
      s_range[n++] = h.pair[c];
    }
    s_n_range = n;
  }
  __syncthreads();
  const int nr = s_n_range;
  const bool single_use = k_clean - 1 == 1 && (a.noise_type == NOISE_OOD || a.noise_type == NOISE_SYM);
  if (single_use && threadIdx.x < nr) {  // pi: the range ranked by lowbias32(r ^ hkey(kw, 33))
    const uint32_t kp = hkey(kw, 33u), mine = lowbias32((uint32_t)threadIdx.x ^ kp);
    int rank = 0;
    for (int r = 0; r < nr; ++r) rank += lowbias32((uint32_t)r ^ kp) < mine ? 1 : 0;
    s_perm[rank] = threadIdx.x;
  }
  if (wid == 0) {
    for (int o = 1; o < EP_WARPS; ++o) top_merge(s_top[0], s_top[o], s_top[0]);
  }
  __syncthreads();
  if (threadIdx.x < n_noise) {
    const int j = threadIdx.x;
    s_ncls[j] = single_use ? s_range[s_perm[min(j, nr - 1)]]
                           : s_range[((uint64_t)hkey(kw, 64u + j) * (uint32_t)nr) >> 32];
  }
  __syncthreads();
  // noisy shot j: the smallest lowbias32(b ^ hkey(kw, 128 + j)) of its class's eligible list
  for (int j = wid; j < n_noise; j += EP_WARPS) {
    const int32_t o = elig_off[s_ncls[j]], n = elig_off[s_ncls[j] + 1] - o;
    const uint32_t kj = hkey(kw, 128u + j);
    uint64_t best = TOP_EMPTY;
    for (int32_t q = lane; q < n; q += 32) {
      const uint32_t b = (uint32_t)elig_block[o + q];
      const uint64_t v = ((uint64_t)lowbias32(b ^ kj) << 32) | b;
      best = v < best ? v : best;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const uint64_t u = __shfl_xor_sync(0xffffffffu, best, d);
      best = u < best ? u : best;
    }
    if (lane == 0) s_nblk[j] = (int32_t)(uint32_t)best;
  }
  const uint32_t ks = hkey(kw, 34u);
  if (threadIdx.x < a.k_shot) s_okey[threadIdx.x] = lowbias32((uint32_t)threadIdx.x ^ ks);
  __syncthreads();
  // shot t before the shuffle: clean shot t (t < k_clean) or noisy shot t - k_clean; it goes to
  // the slot of its rank under lowbias32(t ^ hkey(kw, 34))
  const int64_t ew = (int64_t)e * a.n_way + w;
  if (threadIdx.x < a.k_shot) {
    const int t = threadIdx.x;
    int slot = 0;
    for (int u = 0; u < a.k_shot; ++u) slot += s_okey[u] < s_okey[t] ? 1 : 0;
    const bool nz = t >= k_clean;
    const int32_t b = nz ? s_nblk[t - k_clean] : (int32_t)(uint32_t)s_top[0][t];
    const int32_t k = nz ? s_ncls[t - k_clean] : c;
    shot_block[ew * a.k_shot + slot] = b;
    support_flag[ew * a.k_shot + slot] = h.cls[k];
    noisy[ew * a.k_shot + slot] = nz ? 1 : 0;
  }
  if (threadIdx.x < a.n_queries)
    query_block[ew * a.n_queries + threadIdx.x] = (int32_t)(uint32_t)s_top[0][k_clean + threadIdx.x];
}

// One CTA per cloud: the support shots of every (episode, way), then the query clouds.  Slot s of
// a block's cloud holds member rank s mod min(n_b, N), normalised as a chunk cloud.
__global__ __launch_bounds__(256) void episode_cloud_kernel(
    const float* __restrict__ pts, int64_t s_m, int64_t s_c, int N,
    const int32_t* __restrict__ labels, const int64_t* __restrict__ block_off,
    const int32_t* __restrict__ member, const EpisodeArgs a, const int32_t* __restrict__ hbuf,
    int E, const int32_t* __restrict__ noisy, const int32_t* __restrict__ shot_block,
    const int32_t* __restrict__ support_flag, const int32_t* __restrict__ query_block,
    float* __restrict__ support_x, int32_t* __restrict__ support_y,
    int32_t* __restrict__ gt_support_y, int32_t* __restrict__ support_src,
    float* __restrict__ query_x, int64_t* __restrict__ query_y, int32_t* __restrict__ query_src) {
  const int64_t g = blockIdx.x, n_shots = (int64_t)E * a.n_way * a.k_shot;
  const bool shot = g < n_shots;
  const int64_t i = shot ? g : g - n_shots;
  const int32_t b = shot ? shot_block[i] : query_block[i];
  const int64_t m0 = block_off[b];
  const int32_t nb = (int32_t)(block_off[b + 1] - m0);
  float* out = (shot ? support_x : query_x) + i * N * 9;
  int32_t* src = (shot ? support_src : query_src) + i * N;
  scene_cloud(pts, s_m, s_c, N, IndexMembers{member, m0}, min(nb, N), out, src);
  if (shot) {
    const int32_t cls = support_flag[i], nz = noisy[i];
    for (int q = threadIdx.x; q < N; q += blockDim.x) {
      const int32_t y = labels[src[q]] == cls ? 1 : 0;
      support_y[i * N + q] = y;
      gt_support_y[i * N + q] = nz ? 0 : y;
    }
  } else {
    const EpisodeHost h = ep_host_view(const_cast<int32_t*>(hbuf), E, a.n_way, a.n_cls);
    const int64_t e = i / ((int64_t)a.n_way * a.n_queries);
    int32_t wc[MAX_WAY];
#pragma unroll
    for (int v = 0; v < MAX_WAY; ++v) wc[v] = v < a.n_way ? h.cls[h.way[e * a.n_way + v]] : 0;
    for (int q = threadIdx.x; q < N; q += blockDim.x) {
      const int32_t l = labels[src[q]];
      int64_t y = 0;
#pragma unroll
      for (int v = MAX_WAY - 1; v >= 0; --v)
        if (v < a.n_way && l == wc[v]) y = v + 1;
      query_y[i * N + q] = y;
    }
  }
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

int r3dfs_scene_index(const int32_t* labels, int64_t M, int overlap, const int32_t* h_classes,
                      int n_cls, int32_t scan, int64_t point_base, int64_t n_blocks,
                      int64_t n_members, int64_t block_cap, int64_t member_cap, int64_t* block_off,
                      int32_t* block_scan, int32_t* block_id, int32_t* member, int32_t* count,
                      int64_t* h_sizes, const void* plan_ws, size_t plan_ws_bytes,
                      r3dfs_stream_t stream) {
  if (!labels || !h_classes || !block_off || !block_scan || !block_id || !member || !count ||
      !h_sizes || !plan_ws || scan < 0 || point_base < 0 || n_blocks < 0 || n_members < 0)
    return R3DFS_E_BADARG;
  R3DFS_TRY(scene_common_checks(M, overlap, 64));
  if (n_cls < 1 || n_cls > MAX_IDX_CLS) return R3DFS_E_UNSUPPORTED;
  if (point_base + M > INT32_MAX) return R3DFS_E_UNSUPPORTED;
  IndexCls cls{};
  cls.n = n_cls;
  for (int k = 0; k < n_cls; ++k) {
    for (int v = 0; v < k; ++v)
      if (h_classes[v] == h_classes[k]) return R3DFS_E_BADARG;
    cls.at[k] = k;
  }
  std::sort(cls.at, cls.at + n_cls, [&](int32_t x, int32_t y) { return h_classes[x] < h_classes[y]; });
  for (int k = 0; k < n_cls; ++k) cls.id[k] = h_classes[cls.at[k]];
  if (plan_ws_bytes < r3dfs_scene_workspace(M, overlap)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump pws(const_cast<void*>(plan_ws), plan_ws_bytes);
  SceneWs p;
  carve_scene(pws, M, overlap, p);
  // the one host synchronisation per scan: the plan's block and membership counts
  SceneHdr hdr;
  cudaError_t e = cudaMemcpyAsync(&hdr, p.hdr, sizeof(hdr), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return (int)e;
  if (hdr.err) {
    h_sizes[0] = h_sizes[1] = -1;
    return R3DFS_E_BADARG;
  }
  h_sizes[0] = hdr.n_seg;
  h_sizes[1] = hdr.T;
  if (n_members + hdr.T >= ((int64_t)1 << 31)) return R3DFS_E_UNSUPPORTED;
  if (n_blocks + hdr.n_seg > block_cap || n_members + hdr.T > member_cap) return R3DFS_E_WORKSPACE;
  index_blocks_kernel<<<nblk(hdr.n_seg + 1), 256, 0, st>>>(p.hdr, p.keys[0], p.seg_start, scan,
                                                           n_blocks, n_members, block_off,
                                                           block_scan, block_id);
  R3DFS_CHECK_LAUNCH();
  if (hdr.T > 0) {
    index_members_kernel<<<nblk(hdr.T), 256, 0, st>>>(hdr.T, p.vals[0], p.mem_point, n_members,
                                                      (int32_t)point_base, member);
    R3DFS_CHECK_LAUNCH();
  }
  if (hdr.n_seg > 0) {
    index_count_kernel<<<nblk(hdr.n_seg, IDX_WARPS), IDX_T, 0, st>>>(
        p.hdr, p.vals[0], p.mem_point, p.seg_start, labels, cls, n_blocks, count);
    R3DFS_CHECK_LAUNCH();
  }
  return 0;
}

size_t r3dfs_scene_index_workspace(int64_t n_blocks, int n_cls) {
  if (n_blocks < 1 || n_cls < 1 || n_cls > MAX_IDX_CLS ||
      n_blocks * n_cls >= ((int64_t)1 << 31) - 1)
    return 0;
  const int64_t n = n_blocks * n_cls + 1;
  WsBump ws(nullptr, 0);
  ws.take<int32_t>(n);
  ws.take<int32_t>(scan_tiles(n) + 1);
  ws.take<int32_t>(1);
  return align_up(ws.off, 256);
}

int r3dfs_scene_index_classes(const int64_t* block_off, const int32_t* count, int64_t n_blocks,
                              int n_cls, int min_points, double min_ratio, int32_t* elig_off,
                              int32_t* elig_block, int32_t* h_elig_off, void* wsp, size_t ws_bytes,
                              r3dfs_stream_t stream) {
  if (!block_off || !count || !elig_off || !elig_block || !h_elig_off || !wsp)
    return R3DFS_E_BADARG;
  if (min_points < 0 || !(min_ratio >= 0.0 && min_ratio <= 1.0)) return R3DFS_E_BADARG;
  const size_t need = r3dfs_scene_index_workspace(n_blocks, n_cls);
  if (need == 0) return n_blocks < 1 ? R3DFS_E_BADARG : R3DFS_E_UNSUPPORTED;
  if (ws_bytes < need) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = n_blocks * n_cls + 1;
  WsBump ws(wsp, ws_bytes);
  int32_t* pos = ws.take<int32_t>(n);
  int32_t* bsum = ws.take<int32_t>(scan_tiles(n) + 1);
  int32_t* total = ws.take<int32_t>(1);
  index_flag_kernel<<<nblk(n), 256, 0, st>>>(block_off, count, n_blocks, n_cls, min_points,
                                             min_ratio, pos);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(scan_excl(pos, n, bsum, total, st));
  index_lists_kernel<<<nblk(n), 256, 0, st>>>(pos, n_blocks, n_cls, elig_off, elig_block);
  R3DFS_CHECK_LAUNCH();
  cudaError_t e = cudaMemcpyAsync(h_elig_off, elig_off, sizeof(int32_t) * (n_cls + 1),
                                  cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  return e == cudaSuccess ? 0 : (int)e;
}

size_t r3dfs_scene_episodes_workspace(int n_episodes, int n_way, int k_shot, int n_queries,
                                      int n_cls) {
  if (n_episodes < 1 || n_way < 1 || n_way > MAX_WAY || k_shot < 1 || k_shot > MAX_SHOT ||
      n_queries < 1 || n_queries > MAX_SHOT || n_cls < 1 || n_cls > MAX_IDX_CLS ||
      (int64_t)n_episodes * n_way * n_queries > 65535)
    return 0;
  WsBump ws(nullptr, 0);
  EpisodeWs w;
  carve_episodes(ws, n_episodes, n_way, k_shot, n_cls, w);
  return align_up(ws.off, 256);
}

int r3dfs_scene_episodes(const float* points, int64_t s_m, int64_t s_c, const int32_t* labels,
                         const int64_t* block_off, const int32_t* member, const int32_t* elig_off,
                         const int32_t* elig_block, const int32_t* h_elig_off,
                         const int32_t* h_classes, int n_cls, const int32_t* h_way_class,
                         const int32_t* h_n_noise, int noise_type, const int32_t* h_pair,
                         int n_episodes, int n_way, int k_shot, int n_queries, int n_points,
                         uint32_t seed, int64_t first, int64_t step, float* support_x,
                         int32_t* support_y, int32_t* gt_support_y, int32_t* support_flag,
                         float* query_x, int64_t* query_y, int32_t* shot_block,
                         int32_t* query_block, int32_t* support_src, int32_t* query_src,
                         void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!points || !labels || !block_off || !member || !elig_off || !elig_block || !h_elig_off ||
      !h_classes || !h_way_class || !h_n_noise || !support_x || !support_y || !gt_support_y ||
      !support_flag || !query_x || !query_y || !shot_block || !query_block || !support_src ||
      !query_src || !wsp)
    return R3DFS_E_BADARG;
  const size_t need = r3dfs_scene_episodes_workspace(n_episodes, n_way, k_shot, n_queries, n_cls);
  if (need == 0 || n_points < 64 || n_points > 65536) return R3DFS_E_UNSUPPORTED;
  if (noise_type < NOISE_NONE || noise_type > NOISE_PAIR || (noise_type == NOISE_PAIR && !h_pair))
    return R3DFS_E_BADARG;
  if (first < 0 || step < 1 || first + (int64_t)(n_episodes - 1) * step > (int64_t)UINT32_MAX)
    return R3DFS_E_BADARG;
  const int E = n_episodes;
  std::vector<int32_t> hb(ep_host_ints(E, n_way, n_cls));
  EpisodeHost h = ep_host_view(hb.data(), E, n_way, n_cls);
  auto index_of = [&](int32_t id) {
    for (int k = 0; k < n_cls; ++k)
      if (h_classes[k] == id) return k;
    return -1;
  };
  auto n_elig = [&](int k) { return h_elig_off[k + 1] - h_elig_off[k]; };
  for (int k = 0; k < n_cls; ++k) {
    if (index_of(h_classes[k]) != k) return R3DFS_E_BADARG;  // duplicate class id
    h.cls[k] = h_classes[k];
    h.pair[k] = k;
    if (noise_type == NOISE_PAIR && (h.pair[k] = index_of(h_pair[k])) < 0) return R3DFS_E_BADARG;
  }
  for (int e = 0; e < E; ++e) {
    const int nn = h_n_noise[e];
    if (nn < 0 || nn > k_shot || (noise_type == NOISE_NONE && nn > 0)) return R3DFS_E_BADARG;
    if (k_shot - nn + n_queries > MAX_SHOT) return R3DFS_E_UNSUPPORTED;
    h.n_noise[e] = nn;
    int n_ood = 0;
    int32_t* way = h.way + (size_t)e * n_way;
    for (int w = 0; w < n_way; ++w) {
      way[w] = index_of(h_way_class[(size_t)e * n_way + w]);
      if (way[w] < 0 || n_elig(way[w]) < k_shot - nn + n_queries) return R3DFS_E_BADARG;
      for (int v = 0; v < w; ++v)
        if (way[v] == way[w]) return R3DFS_E_BADARG;
    }
    for (int k = 0; k < n_cls; ++k)
      n_ood += n_elig(k) > 0 && std::find(way, way + n_way, k) == way + n_way ? 1 : 0;
    if (nn == 0) continue;
    if ((noise_type == NOISE_OOD && n_ood == 0) || (noise_type == NOISE_SYM && n_way < 2))
      return R3DFS_E_BADARG;
    if (noise_type == NOISE_PAIR)
      for (int w = 0; w < n_way; ++w)
        if (n_elig(h.pair[way[w]]) < 1) return R3DFS_E_BADARG;
  }
  if (ws_bytes < need) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_episodes(ws, E, n_way, k_shot, n_cls, w);
  cudaError_t ce = cudaMemcpyAsync(w.host, hb.data(), sizeof(int32_t) * hb.size(),
                                   cudaMemcpyHostToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  const EpisodeArgs a{lowbias32(seed), first, step, n_way, k_shot, n_queries, n_cls, noise_type};
  episode_select_kernel<<<E * n_way, EP_T, 0, st>>>(elig_off, elig_block, a, w.host, E, w.noisy,
                                                    shot_block, support_flag, query_block);
  R3DFS_CHECK_LAUNCH();
  const int64_t n_clouds = (int64_t)E * n_way * (k_shot + n_queries);
  episode_cloud_kernel<<<(unsigned)n_clouds, 256, 0, st>>>(
      points, s_m, s_c, n_points, labels, block_off, member, a, w.host, E, w.noisy, shot_block,
      support_flag, query_block, support_x, support_y, gt_support_y, support_src, query_x, query_y,
      query_src);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

}  // extern "C"
