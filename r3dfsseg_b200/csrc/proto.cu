// Multi-prototype generation (reference models/mpti.py:597-715) and the eval-time multi-scale
// degree-based noise suppression over support shots (models/mpti.py:87-223, 316-371).
#include <cooperative_groups.h>

#include "common.cuh"
#include "proto.cuh"

namespace cg = cooperative_groups;

// --------------------------------------------------------------------------------------------
// Farthest point sampling in feature space (torch_cluster.fps as called at models/mpti.py:613).
// One thread-block CLUSTER per set: the set's points are sliced across the cluster's CTAs, every
// CTA keeps the running min-distance of its slice in shared memory, 8 lanes share one point
// (float4 loads, 3 shuffles), and the per-pick argmax is exchanged through distributed shared
// memory with one cluster barrier per pick.  Distances are direct differences in FP32
// (sum (x - s)^2): the Gram form is not accurate enough to reproduce the pick sequence.
// --------------------------------------------------------------------------------------------
#define FPS_THREADS 512
#define FPS_MAX_CL 16
#define FPS_MAX_F4 8  // per-lane float4 fragments -> D <= 256

__device__ __forceinline__ int fps_target_count(int n, int k) {
  // m = ceil(fp32(n) * fp32(k / n))  (the ratio is a Python float, cast to the tensor dtype)
  float ratio = (float)((double)k / (double)n);
  float prod = __fmul_rn((float)n, ratio);
  return (int)ceilf(prod);
}

__global__ __launch_bounds__(FPS_THREADS) void fps_kernel(const float* __restrict__ feat, int D,
                                                          const int32_t* __restrict__ set_off,
                                                          const int32_t* __restrict__ set_n,
                                                          int m_max, int k_for_count,
                                                          int32_t* __restrict__ idx_out,
                                                          int32_t* __restrict__ cnt_out) {
  cg::cluster_group cluster = cg::this_cluster();
  const int CL = cluster.num_blocks();
  const int rank = cluster.block_rank();
  const int set = blockIdx.y;
  extern __shared__ __align__(16) float dist[];  // slice min-distances
  __shared__ float s_wv[FPS_THREADS / 32];
  __shared__ int s_wi[FPS_THREADS / 32];
  __shared__ float s_cv[2][FPS_MAX_CL];
  __shared__ int s_ci[2][FPS_MAX_CL];

  const int n = set_n[set];
  const int64_t row0 = set_off[set];
  int m;
  if (k_for_count > 0)
    m = (n > k_for_count) ? fps_target_count(n, k_for_count) : 0;
  else
    m = min(m_max, n);
  m = min(m, m_max);
  if (rank == 0 && threadIdx.x == 0 && cnt_out) cnt_out[set] = m;
  int32_t* out = idx_out + (int64_t)set * m_max;
  if (m <= 0) {  // uniform over the cluster: nobody reaches a barrier
    return;
  }
  int chunk = (n + CL - 1) / CL;
  chunk = (chunk + 3) & ~3;
  const int lo = min(n, rank * chunk), hi = min(n, lo + chunk);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int sub = lane & 7, grp = lane >> 3;
  const int D4 = D >> 2;
  for (int i = tid; i < hi - lo; i += FPS_THREADS) dist[i] = INFINITY;
  __syncthreads();

  int last = 0;
  if (rank == 0 && tid == 0) out[0] = 0;
  for (int pick = 1; pick < m; ++pick) {
    // seed fragments (same addresses across point groups -> broadcast)
    float4 sfrag[FPS_MAX_F4];
    const float4* srow = reinterpret_cast<const float4*>(feat + (row0 + last) * (int64_t)D);
#pragma unroll
    for (int u = 0; u < FPS_MAX_F4; ++u) {
      int c4 = sub + 8 * u;
      sfrag[u] = (c4 < D4) ? srow[c4] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float bv = -1.f;
    int bi = 0x7fffffff;
    for (int pb = lo + w * 4; pb < hi; pb += (FPS_THREADS / 32) * 4) {
      // warp-uniform trip count: the tail groups stay in the loop for the shuffles
      const int p = pb + grp;
      const bool valid = p < hi;
      float acc = 0.f;
      if (valid) {
        const float4* xrow = reinterpret_cast<const float4*>(feat + (row0 + p) * (int64_t)D);
#pragma unroll
        for (int u = 0; u < FPS_MAX_F4; ++u) {
          int c4 = sub + 8 * u;
          if (c4 < D4) {
            float4 x = xrow[c4];
            float d0 = x.x - sfrag[u].x, d1 = x.y - sfrag[u].y, d2 = x.z - sfrag[u].z,
                  d3 = x.w - sfrag[u].w;
            acc = fmaf(d0, d0, acc);
            acc = fmaf(d1, d1, acc);
            acc = fmaf(d2, d2, acc);
            acc = fmaf(d3, d3, acc);
          }
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (valid) {
        float nd = fminf(dist[p - lo], acc);
        if (sub == 0) dist[p - lo] = nd;
        if (nd > bv) {  // p increases within a thread: strict > keeps the lowest index
          bv = nd;
          bi = p;
        }
      }
    }
    // warp argmax (ties -> lowest index)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) {
        bv = ov;
        bi = oi;
      }
    }
    if (lane == 0) {
      s_wv[w] = bv;
      s_wi[w] = bi;
    }
    __syncthreads();
    const int par = pick & 1;
    if (tid == 0) {
      float cv = s_wv[0];
      int ci = s_wi[0];
      for (int i = 1; i < FPS_THREADS / 32; ++i) {
        if (s_wv[i] > cv || (s_wv[i] == cv && s_wi[i] < ci)) {
          cv = s_wv[i];
          ci = s_wi[i];
        }
      }
      for (int r = 0; r < CL; ++r) {
        float* rv = cluster.map_shared_rank(&s_cv[par][rank], r);
        int* ri = cluster.map_shared_rank(&s_ci[par][rank], r);
        *rv = cv;
        *ri = ci;
      }
    }
    cluster.sync();
    float gv = s_cv[par][0];
    int gi = s_ci[par][0];
    for (int r = 1; r < CL; ++r) {
      float v = s_cv[par][r];
      int i2 = s_ci[par][r];
      if (v > gv || (v == gv && i2 < gi)) {
        gv = v;
        gi = i2;
      }
    }
    if (gi == 0x7fffffff) gi = 0;
    last = gi;
    if (rank == 0 && tid == 0) out[pick] = gi;
  }
  // keep every CTA's shared memory alive until all remote writes/reads are done
  cluster.sync();
}

// CTAs per set.  A CTA streams its slice at only ~25-70 GB/s (one round of loads per warp in
// flight), so a set's sweep time is its bytes over (CTAs x that rate): with a batch of episodes
// 8-CTA clusters already fill every SM twice over and HBM is the limit, but the handful of sets of
// a single episode (the training step) leaves most SMs idle — those get 16-CTA clusters.
static int fps_cluster_size(int n_sets) { return n_sets <= 16 ? 16 : 8; }

// The streaming kernel above (every pick re-reads the set): few picks (the fps_k = 4 prototypes of
// the way-contrast loss), feature widths other than 192, callers without a spill area.
static int launch_fps_stream(const float* feat, int D, const int32_t* set_off,
                             const int32_t* set_n, int n_sets, int n_cap, int m_max,
                             int k_for_count, int32_t* idx_out, int32_t* cnt_out,
                             cudaStream_t st) {
  if (D % 4 != 0 || D > 32 * FPS_MAX_F4 || D <= 0) return R3DFS_E_UNSUPPORTED;
  int CL = fps_cluster_size(n_sets);
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  size_t smem = 0;
  cudaError_t e;
  for (;; CL = 8) {
    int chunk = (n_cap + CL - 1) / CL;
    chunk = (chunk + 3) & ~3;
    smem = sizeof(float) * (size_t)chunk;
    if (smem > 200 * 1024) return R3DFS_E_UNSUPPORTED;
    e = cudaFuncSetAttribute(fps_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return (int)e;
    if (CL > 8) {
      e = cudaFuncSetAttribute(fps_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      if (e != cudaSuccess) return (int)e;
    }
    cfg = {};
    cfg.gridDim = dim3(CL, n_sets, 1);
    cfg.blockDim = dim3(FPS_THREADS, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (CL <= 8) break;
    int n_clusters = 0;  // can the device co-schedule a 16-CTA cluster of this kernel at all?
    e = cudaOccupancyMaxActiveClusters(&n_clusters, fps_kernel, &cfg);
    if (e == cudaSuccess && n_clusters >= 1) break;
    (void)cudaGetLastError();
  }
  e = cudaLaunchKernelEx(&cfg, fps_kernel, feat, D, set_off, set_n, m_max, k_for_count, idx_out,
                         cnt_out);
  if (e != cudaSuccess) return (int)e;
  ++r3dfs_launches;
  return 0;
}

// impl: R3DFS_FPS_AUTO / _STREAM / _Q8.  The int8-filter kernel (fps_q8.cu) needs D = 192, a spill
// area of fps_q8_spill_bytes(total rows) and pays two extra passes over the set, so AUTO takes it
// from 16 picks up.  sets_per_group > 1 = the episode layout (set 0 of every group is the large
// background set, the others are per-way foreground sets): two launches with different cluster
// sizes, so that the small sets do not occupy 16 SMs each.
int launch_fps_ex(const float* feat, int D, const int32_t* set_off, const int32_t* set_n,
                  int n_sets, int n_cap, int m_max, int k_for_count, int32_t* idx_out,
                  int32_t* cnt_out, cudaStream_t st, uint8_t* spill, int sets_per_group,
                  int impl) {
  const bool q8_ok = spill != nullptr && D == 192;
  if (impl == R3DFS_FPS_Q8 && !q8_ok) return R3DFS_E_UNSUPPORTED;
  if (impl == R3DFS_FPS_STREAM || !q8_ok || (impl == R3DFS_FPS_AUTO && m_max < 16))
    return launch_fps_stream(feat, D, set_off, set_n, n_sets, n_cap, m_max, k_for_count, idx_out,
                             cnt_out, st);
  if (sets_per_group > 1 && n_sets % sets_per_group == 0) {
    const int groups = n_sets / sets_per_group, per = sets_per_group - 1;
    // background sets: cl = 0, the smallest cluster whose shared memory holds the set
    R3DFS_TRY(launch_fps_q8(feat, set_off, set_n, groups, 0, 1, sets_per_group, n_cap, 0, m_max,
                            k_for_count, spill, idx_out, cnt_out, st));
    // foreground sets: as many CTAs per set as keep all of them in ONE wave (rows beyond the
    // cluster's shared memory are swept from the spill area, still as bytes)
    int dev = 0, n_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    int cl = 8;
    while (cl > 1 && groups * per * cl > n_sm) cl >>= 1;
    return launch_fps_q8(feat, set_off, set_n, groups * per, 1, per, sets_per_group, n_cap, cl,
                         m_max, k_for_count, spill, idx_out, cnt_out, st);
  }
  return launch_fps_q8(feat, set_off, set_n, n_sets, 0, 1, 1, n_cap, 0, m_max, k_for_count, spill,
                       idx_out, cnt_out, st);
}

// --------------------------------------------------------------------------------------------
// `.unique()` of the FPS picks (models/mpti.py:613-614): sort ascending, drop duplicates.
// n <= k: every point is its own prototype (models/mpti.py:631-634) -> identity seeds.
// One warp-sized CTA per set; m <= 128.
// --------------------------------------------------------------------------------------------
__global__ void seeds_unique_kernel(const int32_t* __restrict__ picks,
                                    const int32_t* __restrict__ pick_cnt,
                                    const int32_t* __restrict__ set_n, int m_max, int k,
                                    int32_t* __restrict__ seeds, int32_t* __restrict__ proto_cnt) {
  __shared__ int s[128];
  __shared__ int cnt;
  const int set = blockIdx.x, tid = threadIdx.x;  // 128 threads
  const int n = set_n[set];
  int32_t* out = seeds + (int64_t)set * m_max;
  if (n <= k) {
    for (int i = tid; i < m_max; i += 128) out[i] = i < n ? i : -1;
    if (tid == 0) proto_cnt[set] = n;
    return;
  }
  const int m = pick_cnt[set];
  s[tid] = tid < m ? picks[(int64_t)set * m_max + tid] : 0x7fffffff;
  __syncthreads();
  for (int ksz = 2; ksz <= 128; ksz <<= 1)
    for (int j = ksz >> 1; j > 0; j >>= 1) {
      int ixj = tid ^ j;
      if (ixj > tid) {
        bool up = (tid & ksz) == 0;
        int a = s[tid], b = s[ixj];
        if ((a > b) == up) {
          s[tid] = b;
          s[ixj] = a;
        }
      }
      __syncthreads();
    }
  if (tid == 0) {
    int c = 0;
    for (int i = 0; i < m; ++i)
      if (i == 0 || s[i] != s[i - 1]) out[c++] = s[i];
    cnt = c;
    proto_cnt[set] = c;
  }
  __syncthreads();
  for (int i = cnt + tid; i < m_max; i += 128) out[i] = -1;
}

// --------------------------------------------------------------------------------------------
// Prototype = mean of its members (models/mpti.py:625-629), deterministic, in two steps:
//   1. one CTA per (set, chunk of 2048 points): thread d walks the chunk's points in order and
//      adds dimension d of each point to its prototype's accumulator in shared memory;
//   2. one CTA per (set, prototype): chunk partials are added in chunk order, divided by the count.
// Every feature row is read exactly once; no floating-point atomics.
// --------------------------------------------------------------------------------------------
#define MEAN_THREADS 256
#define PM_CHUNK 2048

__global__ __launch_bounds__(MEAN_THREADS) void proto_partial_kernel(
    const float* __restrict__ feat, int D, const int32_t* __restrict__ set_off,
    const int32_t* __restrict__ set_n, const int32_t* __restrict__ proto_cnt,
    const int32_t* __restrict__ assign, int m_max, int n_chunks, float* __restrict__ partial,
    int32_t* __restrict__ pcount) {
  extern __shared__ __align__(16) float s_acc[];  // [m_max][D] then [m_max] counts
  const int set = blockIdx.y, chunk = blockIdx.x;
  const int n = set_n[set];
  const int p0 = chunk * PM_CHUNK;
  if (p0 >= n) return;
  const int p1 = min(n, p0 + PM_CHUNK);
  const int m = proto_cnt[set];
  const int64_t row0 = set_off[set];
  const int tid = threadIdx.x;
  int* s_cnt = reinterpret_cast<int*>(s_acc + (size_t)m_max * D);
  for (int e = tid; e < m * D; e += MEAN_THREADS) s_acc[e] = 0.f;
  for (int e = tid; e < m; e += MEAN_THREADS) s_cnt[e] = 0;
  __syncthreads();
  if (tid < D) {
    const float* f = feat + (row0 + p0) * (int64_t)D + tid;
    const int32_t* a = assign + row0 + p0;
#pragma unroll 4
    for (int i = 0; i < p1 - p0; ++i) {
      const int p = a[i];
      s_acc[p * D + tid] += f[(int64_t)i * D];
    }
  } else if (tid == MEAN_THREADS - 1) {
    const int32_t* a = assign + row0 + p0;
    for (int i = 0; i < p1 - p0; ++i) s_cnt[a[i]] += 1;
  }
  __syncthreads();
  float* out = partial + ((int64_t)set * n_chunks + chunk) * m_max * D;
  for (int e = tid; e < m * D; e += MEAN_THREADS) out[e] = s_acc[e];
  int32_t* oc = pcount + ((int64_t)set * n_chunks + chunk) * m_max;
  for (int e = tid; e < m; e += MEAN_THREADS) oc[e] = s_cnt[e];
}

__global__ __launch_bounds__(MEAN_THREADS) void proto_reduce_kernel(
    const float* __restrict__ partial, const int32_t* __restrict__ pcount, int D,
    const int32_t* __restrict__ set_n, const int32_t* __restrict__ proto_cnt, int m_max,
    int n_chunks, int slot, int sets_per_group, int64_t group_rows, float* __restrict__ proto_out,
    int ld_out) {
  const int set = blockIdx.y, p = blockIdx.x;
  if (p >= proto_cnt[set]) return;
  const int nch = (set_n[set] + PM_CHUNK - 1) / PM_CHUNK;
  const int tid = threadIdx.x;
  if (tid >= D) return;
  float acc = 0.f;
  int count = 0;
  for (int c = 0; c < nch; ++c) {
    const int64_t b = (int64_t)set * n_chunks + c;
    acc += partial[(b * m_max + p) * D + tid];
    count += pcount[b * m_max + p];
  }
  const int64_t orow = (int64_t)(set / sets_per_group) * group_rows +
                       (int64_t)(set % sets_per_group) * slot + p;
  proto_out[orow * ld_out + tid] = acc / (float)count;
}

int multi_prototypes_chunks(int n_cap) { return (n_cap + PM_CHUNK - 1) / PM_CHUNK; }

int launch_multi_prototypes(const float* feat, int D, const int32_t* set_off,
                            const int32_t* set_n, int n_sets, int n_cap, int k, int32_t* picks,
                            int32_t* pick_cnt, int32_t* seeds, int32_t* proto_cnt,
                            int32_t* assign, float* partial, int32_t* pcount, float* seed_stats,
                            int sets_per_group, int64_t group_rows, float* proto_out, int ld_out,
                            cudaStream_t st, const StageRec* sr, uint8_t* fps_spill,
                            int fps_sets_per_group) {
  const int m_max = k + 1;
  if (m_max > 128 || D > MEAN_THREADS) return R3DFS_E_UNSUPPORTED;
  R3DFS_TRY(launch_fps_ex(feat, D, set_off, set_n, n_sets, n_cap, m_max, k, picks, pick_cnt, st,
                          fps_spill, fps_sets_per_group, R3DFS_FPS_AUTO));
  if (sr) sr->mark(R3DFS_ST_FPS, st);
  seeds_unique_kernel<<<n_sets, 128, 0, st>>>(picks, pick_cnt, set_n, m_max, k, seeds, proto_cnt);
  R3DFS_CHECK_LAUNCH();
  // tensor-core filter + exact verify (tc_assign.cu)
  R3DFS_TRY(launch_assign_tc(feat, D, set_off, set_n, seeds, proto_cnt, n_sets, n_cap, m_max, k,
                             seed_stats, seed_stats + (size_t)n_sets * 128, assign, st));
  const int n_chunks = multi_prototypes_chunks(n_cap);
  const size_t smem_p = sizeof(float) * (size_t)m_max * D + sizeof(int) * (size_t)m_max;
  cudaError_t e = cudaFuncSetAttribute(proto_partial_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p);
  if (e != cudaSuccess) return (int)e;
  proto_partial_kernel<<<dim3(n_chunks, n_sets), MEAN_THREADS, smem_p, st>>>(
      feat, D, set_off, set_n, proto_cnt, assign, m_max, n_chunks, partial, pcount);
  R3DFS_CHECK_LAUNCH();
  proto_reduce_kernel<<<dim3(m_max, n_sets), MEAN_THREADS, 0, st>>>(
      partial, pcount, D, set_n, proto_cnt, m_max, n_chunks, m_max, sets_per_group, group_rows,
      proto_out, ld_out);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// Support-set compaction for one batch of episodes (models/mpti.py:656-672, 703-705).
// Set 0 of an episode = background points of every way/shot (mask == 0), set 1+w = foreground
// points (mask != 0) of the kept shots of way w, both in (way, shot, point) order.
// --------------------------------------------------------------------------------------------
__global__ void fg_count_kernel(const int32_t* __restrict__ sy, int N, int32_t* __restrict__ cnt) {
  __shared__ int s[8];
  const int cloud = blockIdx.x;
  int c = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) c += sy[(int64_t)cloud * N + i] != 0;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += s[q];
    cnt[cloud] = t;
  }
}

// one thread per episode: set sizes/offsets and each cloud's start inside its sets
__global__ void set_layout_kernel(const int32_t* __restrict__ fg_cnt,
                                  const int32_t* __restrict__ keep, int E, int n_way, int k_shot,
                                  int N, int32_t* __restrict__ set_off, int32_t* __restrict__ set_n,
                                  int32_t* __restrict__ cloud_bg_off,
                                  int32_t* __restrict__ cloud_fg_off) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  const int S = n_way + 1, C = n_way * k_shot;
  const int cap = C * N;
  int bg = 0;
  for (int c = 0; c < C; ++c) bg += N - fg_cnt[e * C + c];
  int off = e * cap;
  set_off[e * S] = off;
  set_n[e * S] = bg;
  int run = off;
  for (int c = 0; c < C; ++c) {
    cloud_bg_off[e * C + c] = run;
    run += N - fg_cnt[e * C + c];
  }
  off += bg;
  for (int w = 0; w < n_way; ++w) {
    set_off[e * S + 1 + w] = off;
    int tot = 0;
    for (int s = 0; s < k_shot; ++s) {
      const int c = w * k_shot + s;
      if (keep[e * C + c]) {
        cloud_fg_off[e * C + c] = off + tot;
        tot += fg_cnt[e * C + c];
      } else {
        cloud_fg_off[e * C + c] = -1;
      }
    }
    set_n[e * S + 1 + w] = tot;
    off += tot;
  }
}

// CTA per support cloud: ordered compaction + row copy into the set buffer
__global__ __launch_bounds__(256) void set_gather_kernel(
    const float* __restrict__ F, int64_t ep_rows, int64_t sup_row_off, int clouds_per_ep, int N,
    int D, const int32_t* __restrict__ sy, const int32_t* __restrict__ cloud_bg_off,
    const int32_t* __restrict__ cloud_fg_off, float* __restrict__ setfeat) {
  __shared__ int s_dst[256];
  __shared__ int s_w[2][8];
  const int cloud = blockIdx.x;
  const int e = cloud / clouds_per_ep, c = cloud % clouds_per_ep;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  int bg_run = cloud_bg_off[cloud];
  const int fg0 = cloud_fg_off[cloud];
  int fg_run = fg0;
  const int64_t src0 = (int64_t)e * ep_rows + sup_row_off + (int64_t)c * N;
  const int D4 = D >> 2;
  for (int c0 = 0; c0 < N; c0 += 256) {
    const int i = c0 + tid;
    const bool in = i < N;
    const bool fg = in && sy[(int64_t)cloud * N + i] != 0;
    const bool bg = in && !fg;
    const unsigned bf = __ballot_sync(0xffffffffu, fg), bb = __ballot_sync(0xffffffffu, bg);
    if (lane == 0) {
      s_w[0][w] = __popc(bf);
      s_w[1][w] = __popc(bb);
    }
    __syncthreads();
    int offf = 0, offb = 0, totf = 0, totb = 0;
    for (int q = 0; q < 8; ++q) {
      if (q < w) {
        offf += s_w[0][q];
        offb += s_w[1][q];
      }
      totf += s_w[0][q];
      totb += s_w[1][q];
    }
    const unsigned lt = (1u << lane) - 1;
    int dst = -1;
    if (fg && fg0 >= 0) dst = fg_run + offf + __popc(bf & lt);
    if (bg) dst = bg_run + offb + __popc(bb & lt);
    s_dst[tid] = dst;
    __syncthreads();
    // copy rows: one warp per row
    const int cnt = min(256, N - c0);
    for (int r = w; r < cnt; r += 8) {
      const int d = s_dst[r];
      if (d < 0) continue;
      const float4* src = reinterpret_cast<const float4*>(F + (src0 + c0 + r) * (int64_t)D);
      float4* dp = reinterpret_cast<float4*>(setfeat + (int64_t)d * D);
      for (int q = lane; q < D4; q += 32) dp[q] = src[q];
    }
    fg_run += totf;
    bg_run += totb;
    __syncthreads();
  }
}

int launch_set_compaction(const float* F, int64_t ep_rows, int64_t sup_row_off, int E, int n_way,
                          int k_shot, int N, int D, const int32_t* sy, const int32_t* keep,
                          int32_t* fg_cnt, int32_t* set_off, int32_t* set_n, int32_t* cloud_bg_off,
                          int32_t* cloud_fg_off, float* setfeat, cudaStream_t st) {
  const int C = n_way * k_shot;
  fg_count_kernel<<<E * C, 256, 0, st>>>(sy, N, fg_cnt);
  R3DFS_CHECK_LAUNCH();
  set_layout_kernel<<<(E + 63) / 64, 64, 0, st>>>(fg_cnt, keep, E, n_way, k_shot, N, set_off, set_n,
                                                  cloud_bg_off, cloud_fg_off);
  R3DFS_CHECK_LAUNCH();
  set_gather_kernel<<<E * C, 256, 0, st>>>(F, ep_rows, sup_row_off, C, N, D, sy, cloud_bg_off,
                                           cloud_fg_off, setfeat);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

// --------------------------------------------------------------------------------------------
// MDNS step 1 — grid_sampling (models/mpti.py:316-371) for both scales of
// Mean_pl_support_y_multi_scale (:187-189): (1,1,1) -> cell 0, (2,2,1) -> cells 1..4 in the
// reference's loop order (x outer, y inner).  Cell bounds are inclusive on both sides and are
// formed with the reference's own FP32 operations (min + i*d, start + d).  One CTA per support
// cloud; 4 thread groups x D threads sum interleaved points, combined in fixed order.
// --------------------------------------------------------------------------------------------
#define MDNS_CELLS 5
#define MDNS_GROUPS 4

__global__ void mdns_cells_kernel(const float* __restrict__ sx, int64_t s_e, int64_t s_cloud,
                                  int64_t s_c, int64_t s_n, const int32_t* __restrict__ sy,
                                  const float* __restrict__ F, int64_t ep_rows,
                                  int64_t sup_row_off, int clouds_per_ep, int N, int D,
                                  float* __restrict__ cell_mean, int32_t* __restrict__ cell_cnt,
                                  uint8_t* __restrict__ cell_mask_out) {
  extern __shared__ unsigned char s_mask[];  // [N] cell bitmask per point
  __shared__ float s_red[6][32];
  __shared__ float s_bb[6];
  __shared__ int s_cnt[MDNS_CELLS];
  __shared__ float s_part[MDNS_GROUPS][MDNS_CELLS][256];
  const int cloud = blockIdx.x;
  const int e = cloud / clouds_per_ep, c = cloud % clouds_per_ep;
  const float* x = sx + e * s_e + c * s_cloud;
  const int32_t* y = sy + (int64_t)cloud * N;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  // bbox of the foreground points (y == 1, models/mpti.py:113)
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int i = tid; i < N; i += blockDim.x) {
    if (y[i] == 1) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        float v = x[a * s_c + i * s_n];
        mn[a] = fminf(mn[a], v);
        mx[a] = fmaxf(mx[a], v);
      }
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    if (lane == 0) {
      s_red[a][w] = mn[a];
      s_red[3 + a][w] = mx[a];
    }
  }
  if (tid < MDNS_CELLS) s_cnt[tid] = 0;
  __syncthreads();
  if (tid < 6) {
    float v = s_red[tid][0];
    for (int q = 1; q < nw; ++q) v = tid < 3 ? fminf(v, s_red[tid][q]) : fmaxf(v, s_red[tid][q]);
    s_bb[tid] = v;
  }
  __syncthreads();
  const float x_min = s_bb[0], y_min = s_bb[1], z_min = s_bb[2];
  const float x_max = s_bb[3], y_max = s_bb[4], z_max = s_bb[5];
  // scale (1,1,1): d = (max-min)/1 ; start = min + 0*d ; end = start + d
  const float dx1 = __fdiv_rn(x_max - x_min, 1.f), dy1 = __fdiv_rn(y_max - y_min, 1.f),
              dz1 = __fdiv_rn(z_max - z_min, 1.f);
  const float xs1 = __fadd_rn(x_min, __fmul_rn(0.f, dx1)), ys1 = __fadd_rn(y_min, __fmul_rn(0.f, dy1)),
              zs1 = __fadd_rn(z_min, __fmul_rn(0.f, dz1));
  const float xe1 = __fadd_rn(xs1, dx1), ye1 = __fadd_rn(ys1, dy1), ze1 = __fadd_rn(zs1, dz1);
  // scale (2,2,1)
  const float dx2 = __fdiv_rn(x_max - x_min, 2.f), dy2 = __fdiv_rn(y_max - y_min, 2.f);
  float xs2[2], xe2[2], ys2[2], ye2[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    xs2[i] = __fadd_rn(x_min, __fmul_rn((float)i, dx2));
    xe2[i] = __fadd_rn(xs2[i], dx2);
    ys2[i] = __fadd_rn(y_min, __fmul_rn((float)i, dy2));
    ye2[i] = __fadd_rn(ys2[i], dy2);
  }
  int lc[MDNS_CELLS] = {0, 0, 0, 0, 0};
  for (int i = tid; i < N; i += blockDim.x) {
    unsigned char m = 0;
    if (y[i] == 1) {
      const float px = x[i * s_n], py = x[s_c + i * s_n], pz = x[2 * s_c + i * s_n];
      const bool zin = pz >= zs1 && pz <= ze1;
      if (px >= xs1 && px <= xe1 && py >= ys1 && py <= ye1 && zin) m |= 1;
#pragma unroll
      for (int ix = 0; ix < 2; ++ix)
#pragma unroll
        for (int iy = 0; iy < 2; ++iy)
          if (px >= xs2[ix] && px <= xe2[ix] && py >= ys2[iy] && py <= ye2[iy] && zin)
            m |= (unsigned char)(2u << (ix * 2 + iy));
    }
    s_mask[i] = m;
    if (cell_mask_out) cell_mask_out[(int64_t)cloud * N + i] = m;
#pragma unroll
    for (int q = 0; q < MDNS_CELLS; ++q) lc[q] += (m >> q) & 1;
  }
#pragma unroll
  for (int q = 0; q < MDNS_CELLS; ++q) {
    int v = lc[q];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && v) atomicAdd(&s_cnt[q], v);
  }
  __syncthreads();
  // cell sums
  const int g = tid / D, d = tid % D;
  const int64_t src0 = (int64_t)e * ep_rows + sup_row_off + (int64_t)c * N;
  if (g < MDNS_GROUPS) {
    float acc[MDNS_CELLS] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int i = g; i < N; i += MDNS_GROUPS) {
      const unsigned m = s_mask[i];
      if (m) {
        const float v = F[(src0 + i) * (int64_t)D + d];
#pragma unroll
        for (int q = 0; q < MDNS_CELLS; ++q)
          if ((m >> q) & 1) acc[q] += v;
      }
    }
#pragma unroll
    for (int q = 0; q < MDNS_CELLS; ++q) s_part[g][q][d] = acc[q];
  }
  __syncthreads();
  if (tid < D) {
#pragma unroll
    for (int q = 0; q < MDNS_CELLS; ++q) {
      float sum = ((s_part[0][q][tid] + s_part[1][q][tid]) + s_part[2][q][tid]) + s_part[3][q][tid];
      const int cnt = s_cnt[q];
      cell_mean[((int64_t)cloud * MDNS_CELLS + q) * D + tid] = cnt > 0 ? sum / (float)cnt : 0.f;
    }
  }
  if (tid < MDNS_CELLS) cell_cnt[cloud * MDNS_CELLS + tid] = s_cnt[tid];
}

// --------------------------------------------------------------------------------------------
// MDNS step 2 — Mean_pl_support_y (models/mpti.py:124-166) at both scales + the multi-scale vote
// (:198-221).  One CTA per (episode, way).
// --------------------------------------------------------------------------------------------
#define MDNS_MAX_SEEDS 128

__global__ void mdns_vote_kernel(const float* __restrict__ cell_mean,
                                 const int32_t* __restrict__ cell_cnt,
                                 const int32_t* __restrict__ fg_cnt, int k_shot, int D,
                                 int32_t* __restrict__ keep, float* __restrict__ clean_flag,
                                 float* __restrict__ degree_out, float* __restrict__ scale_flag_out) {
  extern __shared__ __align__(16) float s_v[];  // [L][D] normalised seeds
  __shared__ float s_deg[MDNS_MAX_SEEDS];
  __shared__ int s_shot[MDNS_MAX_SEEDS];
  __shared__ int s_cell[MDNS_MAX_SEEDS];
  __shared__ float s_flag[2][32];
  __shared__ int s_L;
  const int ew = blockIdx.x;  // episode * n_way + way
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
  for (int scale = 0; scale < 2; ++scale) {
    __syncthreads();
    if (tid == 0) {
      int L = 0;
      for (int s = 0; s < k_shot; ++s) {
        const int cloud = ew * k_shot + s;
        const int c_lo = scale == 0 ? 0 : 1, c_hi = scale == 0 ? 1 : 5;
        for (int q = c_lo; q < c_hi; ++q)
          if (cell_cnt[cloud * MDNS_CELLS + q] > 0 && L < MDNS_MAX_SEEDS) {
            s_shot[L] = s;
            s_cell[L] = cloud * MDNS_CELLS + q;
            ++L;
          }
      }
      s_L = L;
    }
    __syncthreads();
    const int L = s_L;
    // F.normalize(p=2, dim=1): v / max(||v||, 1e-12)
    for (int i = w; i < L; i += nw) {
      const float* src = cell_mean + (int64_t)s_cell[i] * D;
      float ss = 0.f;
      for (int d = lane; d < D; d += 32) ss = fmaf(src[d], src[d], ss);
      ss = warp_sum(ss);
      const float nrm = fmaxf(sqrtf(ss), 1e-12f);
      for (int d = lane; d < D; d += 32) s_v[i * D + d] = src[d] / nrm;
    }
    __syncthreads();
    // degree_i = sum_{j != i} cos_ij (cubed at scale (1,1,1), models/mpti.py:135-136)
    for (int i = w; i < L; i += nw) {
      float deg = 0.f;
      for (int j = 0; j < L; ++j) {
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = fmaf(s_v[i * D + d], s_v[j * D + d], dot);
        dot = warp_sum(dot);
        if (j == i) dot = 0.f;
        if (scale == 0) dot = dot * dot * dot;
        deg += dot;
      }
      if (lane == 0) s_deg[i] = deg;
    }
    __syncthreads();
    if (degree_out)  // diagnostic: (way, scale, 4 * k_shot) degrees in seed order, NaN padded
      for (int i = tid; i < 4 * k_shot; i += blockDim.x)
        degree_out[((int64_t)ew * 2 + scale) * (4 * k_shot) + i] = i < L ? s_deg[i] : NAN;
    if (tid == 0) {
      float mean = 0.f;
      for (int i = 0; i < L; ++i) mean += s_deg[i];
      mean = mean / (float)L;
      for (int s = 0; s < k_shot; ++s) {
        int tot = 0, on = 0;
        for (int i = 0; i < L; ++i)
          if (s_shot[i] == s) {
            ++tot;
            on += s_deg[i] > mean;
          }
        // torch.mean(mask.float()) > 0.5 ; an empty shot gives nan > 0.5 = False
        s_flag[scale][s] = (tot > 0 && (float)on / (float)tot > 0.5f) ? 1.f : 0.f;
      }
    }
  }
  __syncthreads();
  if (scale_flag_out)
    for (int i = tid; i < 2 * k_shot; i += blockDim.x)
      scale_flag_out[(int64_t)ew * 2 * k_shot + i] = s_flag[i / k_shot][i % k_shot];
  if (tid == 0) {
    int kept_pts = 0;
    for (int s = 0; s < k_shot; ++s) {
      const float total = (s_flag[0][s] + s_flag[1][s]) / 2.f;
      const int kp = !(total < 0.5f);
      keep[ew * k_shot + s] = kp;
      if (kp) kept_pts += fg_cnt[ew * k_shot + s];
    }
    if (kept_pts == 0)  // every shot of the way was dropped -> reset (models/mpti.py:216-219)
      for (int s = 0; s < k_shot; ++s) keep[ew * k_shot + s] = 1;
    if (clean_flag)
      for (int s = 0; s < k_shot; ++s) clean_flag[ew * k_shot + s] = (float)keep[ew * k_shot + s];
  }
}

int launch_mdns(const float* sx, int64_t s_e, int64_t s_cloud, int64_t s_c, int64_t s_n,
                const int32_t* sy, const float* F, int64_t ep_rows, int64_t sup_row_off, int E,
                int n_way, int k_shot, int N, int D, float* cell_mean, int32_t* cell_cnt,
                int32_t* fg_cnt, int32_t* keep, float* clean_flag, cudaStream_t st,
                uint8_t* cell_mask_out, float* degree_out, float* scale_flag_out) {
  const int C = n_way * k_shot;
  if (D > 256 || k_shot > 32 || k_shot * 4 > MDNS_MAX_SEEDS) return R3DFS_E_UNSUPPORTED;
  fg_count_kernel<<<E * C, 256, 0, st>>>(sy, N, fg_cnt);
  R3DFS_CHECK_LAUNCH();
  const int threads = MDNS_GROUPS * D <= 1024 ? MDNS_GROUPS * D : 1024;
  if (threads < MDNS_GROUPS * D) return R3DFS_E_UNSUPPORTED;
  mdns_cells_kernel<<<E * C, threads, N, st>>>(sx, s_e, s_cloud, s_c, s_n, sy, F, ep_rows,
                                               sup_row_off, C, N, D, cell_mean, cell_cnt,
                                               cell_mask_out);
  R3DFS_CHECK_LAUNCH();
  size_t smem = sizeof(float) * (size_t)(4 * k_shot) * D;
  cudaError_t e = cudaFuncSetAttribute(mdns_vote_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  mdns_vote_kernel<<<E * n_way, 256, smem, st>>>(cell_mean, cell_cnt, fg_cnt, k_shot, D, keep,
                                                 clean_flag, degree_out, scale_flag_out);
  R3DFS_CHECK_LAUNCH();
  return 0;
}
