// Shared device/host helpers for libr3dfs (sm_100a).  Internal — the public surface is include/r3dfs.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/r3dfs.h"

#define R3DFS_FEAT_DIM 192
#define R3DFS_EC_WIDTH 64

extern thread_local long long r3dfs_launches;  // diagnostic: kernels launched by this thread

// A/B switches (predecessor kernels that tests pin the current ones to, DESIGN.md §6) exist only
// in the measurement build `libr3dfs_ab.so` (make ab: -DR3DFS_AB_SWITCHES); the shipped library
// reads no environment variable and keeps no configuration state.
#ifdef R3DFS_AB_SWITCHES
#include <stdlib.h>
#define R3DFS_GETENV(name) getenv(name)
#else
#define R3DFS_GETENV(name) ((const char*)nullptr)
#endif

#define R3DFS_CHECK_LAUNCH()                       \
  do {                                             \
    cudaError_t e__ = cudaGetLastError();          \
    if (e__ != cudaSuccess) return (int)e__;       \
    ++r3dfs_launches;                              \
  } while (0)

// optional stage-boundary events (r3dfs_episode_diag_t::h_stage_events)
struct StageRec {
  cudaEvent_t* ev;
  inline void mark(int stage, cudaStream_t st) const {
    if (ev && ev[stage]) cudaEventRecord(ev[stage], st);
  }
};

#define R3DFS_TRY(expr)                            \
  do {                                             \
    int rc__ = (expr);                             \
    if (rc__ != 0) return rc__;                    \
  } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// merged symmetric rows (lp.cu): entries a graph owns per node; row segments are multiples of 4
// (a graph's rows hold at most 2 k nn entries in total; every row is padded to a multiple of 4)
__host__ __device__ inline int lp_rowcap(int k) { return ((2 * k + 3) & ~3) + 4; }
// packed form of those rows for the cluster CG kernel (cg_pack_kernel): groups of 4 entries a graph
// may occupy — 1.6 x its entries (measured need: 1.34 x) plus 64 per node
__host__ __device__ inline int64_t lp_pack_groups(int64_t nn, int k) {
  return (nn * (int64_t)(2 * k) * 2 / 5 + 64 * nn + 63) / 64 * 64;
}
// bytes of solver scratch for G graphs (tables for up to 16 CTAs per graph + flags + packed lists)
static inline size_t lp_solver_scratch_bytes(size_t G, size_t nn, int k) {
  return G * 16 * (4 + 32 * 3 * 2 + 3 * 1024 * 2) * 4 + 256 + 4 * G * (1 + nn) + 256 +
         (8 + 16) * G * (size_t)lp_pack_groups(nn, k) + 512;
}

// Bump allocator over the caller's workspace.  Never owns memory.
struct WsBump {
  char* base;
  size_t cap;
  size_t off;
  __host__ WsBump(void* p, size_t c) : base((char*)p), cap(c), off(0) {}
  template <typename T>
  __host__ T* take(size_t n) {
    off = align_up(off, 256);
    T* r = (T*)(base + off);
    off += n * sizeof(T);
    return r;
  }
  __host__ bool ok() const { return off <= cap; }
};

// Row mapping for per-cloud outputs that land inside the per-episode node matrix:
// row(b, i) = (b / cpe) * ep_rows + row_off + (b % cpe) * n + i.   cpe == 0 -> identity b*n+i.
struct RowMap {
  int cpe;
  int n;
  int64_t ep_rows;
  int64_t row_off;
  __host__ __device__ inline int64_t operator()(int64_t m) const {
    if (cpe == 0) return m;
    int64_t b = m / n, i = m - b * n;
    return (b / cpe) * ep_rows + row_off + (b % cpe) * (int64_t)n + i;
  }
};
static inline RowMap identity_map() { return RowMap{0, 1, 0, 0}; }

enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_LRELU = 2 };

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == ACT_RELU) return fmaxf(v, 0.f);
  if (act == ACT_LRELU) return v > 0.f ? v : 0.2f * v;
  return v;
}

// Affinity graph (lp.cu, and the distance GEMM's epilogue in tc_gemm_tma.cu): squared distances are
// ranked by order-preserving integer keys.  0xffffffff is reserved for "not a real column" (the row's
// own node, an invalid node), so a real distance whose key would be 0xffffffff is clamped.
__device__ __forceinline__ unsigned f2key(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ unsigned dist_key(float f) {
  const unsigned kk = f2key(f);
  return kk == 0xffffffffu ? 0xfffffffeu : kk;
}
// The distance GEMM can also write, per row, the smallest key of every group of AFF_GROUP
// contiguous columns: the bound of the select (lp.cu).  Layout (graphs, nn, aff_gstride(nn)) u32,
// rows padded to whole 32-column chunks (the GEMM stores a chunk's minima as one 16-byte vector).
#define AFF_GROUP 8
__host__ __device__ inline int aff_gstride(int nn) { return (nn + 31) / 32 * (32 / AFF_GROUP); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// internal launchers (defined in the .cu files)
int launch_to_point_major(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                          int64_t sn, float* out, cudaStream_t st);
int launch_row_norms(const float* x, int64_t rows, int ld, int C, float* out, cudaStream_t st);
int launch_row_norms_batched(const float* x, int64_t xs, int batch, int64_t rows, int ld, int C,
                             float* out, cudaStream_t st);
int launch_knn(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
               int32_t* idx32, int64_t* idx64, cudaStream_t st);
int launch_knn_tc(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                  int32_t* idx32, int64_t* idx64, cudaStream_t st, void* split_ws = nullptr,
                  size_t split_bytes = 0);
// scratch the TMA-fed kNN kernel wants for the pre-split candidate tiles (0: shape not served)
size_t knn_split_bytes(int C, int64_t B, int N, int k);
// impl 0: tensor cores when C <= 64, CUDA cores otherwise; 1: CUDA cores; 2: tensor cores
int launch_knn_auto(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                    int32_t* idx32, int64_t* idx64, int impl, cudaStream_t st,
                    void* split_ws = nullptr, size_t split_bytes = 0);
int launch_linear(const float* X, int ldx, const float* W, const float* s, const float* t, int act,
                  int64_t M, int K, int Nout, float* Y, int ldy, RowMap map, cudaStream_t st);
int launch_linear_tc(const float* X, int ldx, const float* W, const float* s, const float* t,
                     int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                     cudaStream_t st);
int launch_linear_tma(const float* X, int ldx, const float* W, const float* s, const float* t,
                      int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                      cudaStream_t st);
// TMA-fed tensor-core kernel, or the register-fed one when TMA cannot address the operands
int launch_linear_auto(const float* X, int ldx, const float* W, const float* s, const float* t,
                       int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                       cudaStream_t st);
// gmin (optional): the group minima of every row, with the row's own column and the columns of
// invalid nodes (valid[g][j] == 0) counted as 0xffffffff
int launch_gram_dist_ts(const float* F, int64_t graph_rows, int64_t row_off, int G, int nn, int D,
                        const float* norms, float* D2, const uint8_t* valid, unsigned* gmin,
                        cudaStream_t st);
int launch_gram_dist_tc(const float* F, int64_t graph_rows, int64_t row_off, int G, int nn, int D,
                        const float* norms, float* D2, cudaStream_t st);
int launch_edge_mlp_tc(const float* PQ, const int32_t* idx, const float* w2, const float* s2,
                       const float* t2, int64_t B, int N, int k, float* Y, int ldy, RowMap map,
                       cudaStream_t st);
int launch_edge_feature(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                        int64_t sn, const int64_t* idx, int K, float* out, cudaStream_t st,
                        void* ws = nullptr, size_t ws_bytes = 0);
size_t edge_feature_scratch_bytes(int64_t B, int64_t C, int64_t N);
int launch_attention_tc(const float* qkv, int ld, int64_t B, int N, float* Y, int ldy, RowMap map,
                        cudaStream_t st, float* kmax_ws = nullptr, void* split_ws = nullptr,
                        size_t split_bytes = 0);
// scratch for the pre-split K / V^T tiles of the TMA-fed attention kernel
size_t attention_split_bytes(int64_t B, int N);
int launch_fold_edge_w1(const float* w1, const float* s1, const float* t1, int C, float* wpq,
                        float* spq, float* tpq, cudaStream_t st);

int launch_protonet_head(const float* F, int64_t ep_rows, int64_t sup_row_off, int64_t q_row_off,
                         int E, int n_way, int k_shot, int N, int nq, int D, const int32_t* sy,
                         const int32_t* keep, int method, float* fg, float* bg, float* proto,
                         float* Z, int nn, cudaStream_t st);

int launch_fps(const float* feat, int D, const int32_t* set_off, const int32_t* set_n, int n_sets,
               int m_max, int k_for_count, int32_t* idx_out, cudaStream_t st);
