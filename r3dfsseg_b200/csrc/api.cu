// C ABI of libr3dfs.so (include/r3dfs.h): argument checks, workspace carving, and the episode
// pipeline that chains the kernels of encoder.cu / proto.cu / lp.cu on one stream with no host
// synchronisation (every data-dependent size stays on the device).
#include <stdlib.h>

#include "common.cuh"
#include "lp.cuh"
#include "proto.cuh"
#include "episode.cuh"

// ---------------------------------------------------------------------------------------------
// small glue kernels
// ---------------------------------------------------------------------------------------------
// strided (groups, clouds_in, C, N) -> point-major rows of cloud  (grp * cpe_out + cloud_off + c)
__global__ void gather_clouds_kernel(const float* __restrict__ x, int clouds_in, int C, int N,
                                     int64_t s_g, int64_t s_cloud, int64_t s_c, int64_t s_n,
                                     int cpe_out, int cloud_off, float* __restrict__ out,
                                     int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int c = (int)(e % C);
  int64_t r = e / C;
  const int n = (int)(r % N);
  r /= N;
  const int cl = (int)(r % clouds_in);
  const int64_t grp = r / clouds_in;
  const int64_t ocloud = grp * cpe_out + cloud_off + cl;
  out[(ocloud * N + n) * C + c] = x[grp * s_g + cl * s_cloud + c * s_c + n * s_n];
}

__global__ void copy_cols_kernel(const float* __restrict__ src, int lds, int64_t M, int ncols,
                                 float* __restrict__ dst, int ldd, RowMap map) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int c4n = ncols >> 2;
  if (e >= M * c4n) return;
  const int64_t m = e / c4n;
  const int c4 = (int)(e % c4n);
  reinterpret_cast<float4*>(dst + map(m) * (int64_t)ldd)[c4] =
      reinterpret_cast<const float4*>(src + m * (int64_t)lds)[c4];
}

__global__ void fill_i32_kernel(int32_t* p, int64_t n, int32_t v) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) p[e] = v;
}

// valid mask + one-hot label matrix Y of the graph nodes (models/mpti.py:493-505): prototype slot
// s*slot + p is a node iff p < proto_cnt[s]; its label column is s (0 = background, 1+w = way w).
__global__ void graph_init_kernel(const int32_t* __restrict__ proto_cnt, int S, int slot, int ppad,
                                  int nn, int nc, uint8_t* __restrict__ valid,
                                  float* __restrict__ Y) {
  const int g = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nn) return;
  bool v = true;
  int lab = -1;
  if (i < ppad) {
    const int s = i / slot, p = i % slot;
    v = s < S && p < proto_cnt[g * S + s];
    lab = s;
  }
  valid[(int64_t)g * nn + i] = v ? 1 : 0;
  for (int c = 0; c < nc; ++c) Y[((int64_t)g * nn + i) * nc + c] = (v && c == lab) ? 1.f : 0.f;
}

// given prototypes -> prototype slots of the node matrix (the query half of a split episode): slot
// s*slot + p of episode e = row (s*slot + p) of proto + e*p_e when p < count, 0 otherwise, and 0 up
// to ppad; count = proto_count[e*c_e + s] clamped to [0, slot].  One float4 per thread.
__global__ void proto_rows_kernel(const float* __restrict__ proto, int64_t p_e,
                                  const int32_t* __restrict__ proto_count, int64_t c_e, int S,
                                  int slot, int ppad, int64_t f_rows, float* __restrict__ F,
                                  int32_t* __restrict__ proto_cnt) {
  constexpr int D4 = R3DFS_FEAT_DIM / 4;
  const int e = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S) proto_cnt[e * S + i] = min(max(proto_count[e * c_e + i], 0), slot);
  if (i >= ppad * D4) return;
  const int r = i / D4, s = r / slot;
  int cnt = 0;
  if (s < S) cnt = min(max(proto_count[e * c_e + s], 0), slot);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r - s * slot < cnt) v = reinterpret_cast<const float4*>(proto + e * p_e)[i];
  reinterpret_cast<float4*>(F + e * f_rows * R3DFS_FEAT_DIM)[i] = v;
}

__global__ void i32_to_i64_kernel(const int32_t* __restrict__ a, int64_t* __restrict__ b,
                                  int64_t n) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n) b[e] = a[e];
}

thread_local long long r3dfs_launches = 0;

bool simt_gemm_forced() {
  static const bool v = [] {
    const char* e = R3DFS_GETENV("R3DFS_SIMT_GEMM");
    return e && e[0] == '1';
  }();
  return v;
}

int launch_knn_auto(const float* x, int ld, int C, const float* xx, int64_t B, int N, int k,
                    int32_t* idx32, int64_t* idx64, int impl, cudaStream_t st, void* split_ws,
                    size_t split_bytes) {
  if (impl == 2)
    return launch_knn_tc(x, ld, C, xx, B, N, k, idx32, idx64, st, split_ws, split_bytes);
  if (impl == 0 && !simt_gemm_forced() && C <= 64)
    return launch_knn_tc(x, ld, C, xx, B, N, k, idx32, idx64, st, split_ws, split_bytes);
  return launch_knn(x, ld, C, xx, B, N, k, idx32, idx64, st);
}

int launch_edge_mlp_auto(const float* PQ, const int32_t* idx, const float* w2, const float* s2,
                         const float* t2, int64_t B, int N, int k, float* Y, int ldy, RowMap map,
                         cudaStream_t st) {
  if (simt_gemm_forced())
    return launch_edge_mlp(PQ, idx, w2, s2, t2, B, N, k, Y, ldy, map, nullptr, st);
  return launch_edge_mlp_tc(PQ, idx, w2, s2, t2, B, N, k, Y, ldy, map, st);
}

int launch_attention_auto(const float* qkv, int ld, int64_t B, int N, float* Y, int ldy,
                          RowMap map, cudaStream_t st, float* kmax_ws, void* split_ws,
                          size_t split_bytes) {
  if (simt_gemm_forced()) return launch_attention(qkv, ld, B, N, Y, ldy, map, st);
  return launch_attention_tc(qkv, ld, B, N, Y, ldy, map, st, kmax_ws, split_ws, split_bytes);
}

int launch_linear_auto(const float* X, int ldx, const float* W, const float* s, const float* t,
                       int act, int64_t M, int K, int Nout, float* Y, int ldy, RowMap map,
                       cudaStream_t st) {
  if (simt_gemm_forced())
    return launch_linear(X, ldx, W, s, t, act, M, K, Nout, Y, ldy, map, st);
  // TMA-fed kernel when the operands meet TMA's alignment rules, register-fed kernel otherwise
  const int rc = launch_linear_tma(X, ldx, W, s, t, act, M, K, Nout, Y, ldy, map, st);
  if (rc != R3DFS_E_UNSUPPORTED) return rc;
  return launch_linear_tc(X, ldx, W, s, t, act, M, K, Nout, Y, ldy, map, st);
}

static inline unsigned nblk(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

// ---------------------------------------------------------------------------------------------
// encoder (getFeatures): DGCNN + BaseLearner + SelfAttention
// ---------------------------------------------------------------------------------------------
void carve_encoder(WsBump& ws, int64_t M, int k, EncoderWs& e) {
  e.xx = ws.take<float>(M);
  e.idx = ws.take<int32_t>(M * k);
  e.wpq = ws.take<float>(128 * 64);
  e.spq = ws.take<float>(128);
  e.tpq = ws.take<float>(128);
  e.PQ = ws.take<float>(M * 128);
  e.ecat = ws.take<float>(M * 192);
  e.h512 = ws.take<float>(M * 512);
  e.l2 = ws.take<float>(M * 256);
  e.h128 = ws.take<float>(M * 128);
  e.qkv = ws.take<float>(M * 192);
}

int check_weights(const r3dfs_weights_t* w) {
  if (!w) return R3DFS_E_BADARG;
  if (w->in_dim < 1 || w->in_dim > 64 || w->dgcnn_k < 1 || w->dgcnn_k > 32)
    return R3DFS_E_UNSUPPORTED;
  for (int i = 0; i < 3; ++i)
    if (!w->ec_w1[i] || !w->ec_s1[i] || !w->ec_t1[i] || !w->ec_w2[i] || !w->ec_s2[i] ||
        !w->ec_t2[i])
      return R3DFS_E_BADARG;
  for (int i = 0; i < 2; ++i)
    if (!w->mlp_w[i] || !w->mlp_s[i] || !w->mlp_t[i] || !w->bl_w[i] || !w->bl_s[i] || !w->bl_t[i])
      return R3DFS_E_BADARG;
  if (!w->att_wqkv) return R3DFS_E_BADARG;
  return 0;
}

// xp: (B*N, in_dim) point-major.  F: feature rows (ld 192) addressed through `map`.
int encoder_forward(const r3dfs_weights_t* w, const float* xp, int64_t B, int N,
                           const EncoderWs& e, float* F, RowMap map, float* level2,
                           cudaStream_t st, const StageRec* sr) {
  const int64_t M = B * N;
  const int k = w->dgcnn_k;
  for (int i = 0; i < 3; ++i) {
    const float* in = i == 0 ? xp : e.ecat + 64 * (i - 1);
    const int ld = i == 0 ? w->in_dim : 192;
    const int C = i == 0 ? w->in_dim : 64;
    R3DFS_TRY(launch_row_norms(in, M, ld, C, e.xx, st));
    // h512 is idle until the MLP: it holds the kNN kernel's pre-split candidate tiles
    R3DFS_TRY(launch_knn_auto(in, ld, C, e.xx, B, N, k, e.idx, nullptr, 0, st, e.h512,
                              sizeof(float) * (size_t)M * 512));
    if (sr) sr->mark(R3DFS_ST_KNN0 + 3 * i, st);
    R3DFS_TRY(launch_fold_edge_w1(w->ec_w1[i], w->ec_s1[i], w->ec_t1[i], C, e.wpq, e.spq, e.tpq, st));
    R3DFS_TRY(launch_linear_auto(in, ld, e.wpq, e.spq, e.tpq, ACT_NONE, M, C, 128, e.PQ, 128,
                            identity_map(), st));
    if (sr) sr->mark(R3DFS_ST_PQ0 + 3 * i, st);
    R3DFS_TRY(launch_edge_mlp_auto(e.PQ, e.idx, w->ec_w2[i], w->ec_s2[i], w->ec_t2[i], B, N, k,
                                   e.ecat + 64 * i, 192, identity_map(), st));
    if (sr) sr->mark(R3DFS_ST_EDGE0 + 3 * i, st);
  }
  // level-1 feature = first EdgeConv output (models/dgcnn.py:127, models/mpti.py:586-589)
  copy_cols_kernel<<<nblk(M * 16), 256, 0, st>>>(e.ecat, 192, M, 64, F, 192, map);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(launch_linear_auto(e.ecat, 192, w->mlp_w[0], w->mlp_s[0], w->mlp_t[0], ACT_LRELU, M, 192,
                          512, e.h512, 512, identity_map(), st));
  R3DFS_TRY(launch_linear_auto(e.h512, 512, w->mlp_w[1], w->mlp_s[1], w->mlp_t[1], ACT_LRELU, M, 512,
                          256, e.l2, 256, identity_map(), st));
  if (sr) sr->mark(R3DFS_ST_MLP, st);
  if (level2) {
    cudaError_t ce = cudaMemcpyAsync(level2, e.l2, sizeof(float) * M * 256,
                                     cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return (int)ce;
  }
  R3DFS_TRY(launch_linear_auto(e.l2, 256, w->bl_w[0], w->bl_s[0], w->bl_t[0], ACT_RELU, M, 256, 128,
                          e.h128, 128, identity_map(), st));
  R3DFS_TRY(launch_linear_auto(e.h128, 128, w->bl_w[1], w->bl_s[1], w->bl_t[1], ACT_NONE, M, 128, 64,
                          F + 128, 192, map, st));
  if (sr) sr->mark(R3DFS_ST_BASE, st);
  R3DFS_TRY(launch_linear_auto(e.l2, 256, w->att_wqkv, nullptr, nullptr, ACT_NONE, M, 256, 192, e.qkv,
                          192, identity_map(), st));
  if (sr) sr->mark(R3DFS_ST_QKV, st);
  // xx: free scratch for the key-norm maxima; h512 (idle after the MLP) holds the pre-split K / V^T
  R3DFS_TRY(launch_attention_auto(e.qkv, 192, B, N, F + 64, 192, map, st, e.xx, e.h512,
                                  sizeof(float) * (size_t)M * 512));
  if (sr) sr->mark(R3DFS_ST_ATT, st);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// public entry points
// ---------------------------------------------------------------------------------------------
extern "C" {

int r3dfs_version(void) { return R3DFS_VERSION; }

long long r3dfs_launch_count(void) { return r3dfs_launches; }

const char* r3dfs_strerror(int code) {
  switch (code) {
    case R3DFS_OK: return "ok";
    case R3DFS_E_BADARG: return "bad argument (null pointer or non-positive size)";
    case R3DFS_E_UNSUPPORTED: return "shape not supported by the sm_100a kernels";
    case R3DFS_E_WORKSPACE: return "workspace too small";
    case R3DFS_E_ALIGN: return "pointer not 16-byte aligned";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "unknown error";
}

// ---- knn -------------------------------------------------------------------------------------
size_t r3dfs_knn_workspace(int64_t B, int64_t C, int64_t N, int k) {
  return align_up(sizeof(float) * B * N * C, 256) + align_up(sizeof(float) * B * N, 256) +
         align_up(knn_split_bytes((int)C, B, (int)N, k), 256) + 768;
}

int r3dfs_knn(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc, int64_t sn,
              int k, int64_t* idx_out, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  return r3dfs_knn_ex(x, B, C, N, sb, sc, sn, k, idx_out, 0, wsp, ws_bytes, stream);
}

int r3dfs_knn_ex(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                 int64_t sn, int k, int64_t* idx_out, int impl, void* wsp, size_t ws_bytes,
                 r3dfs_stream_t stream) {
  if (!x || !idx_out || !wsp || B <= 0 || C <= 0 || N <= 0) return R3DFS_E_BADARG;
  if (k < 1 || k > 32 || k > N) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_knn_workspace(B, C, N, k)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  float* xp = ws.take<float>(B * N * C);
  float* xx = ws.take<float>(B * N);
  const size_t split_bytes = knn_split_bytes((int)C, B, (int)N, k);
  unsigned char* split = split_bytes ? ws.take<unsigned char>(split_bytes) : nullptr;
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  R3DFS_TRY(launch_to_point_major(x, B, C, N, sb, sc, sn, xp, st));
  R3DFS_TRY(launch_row_norms(xp, B * N, (int)C, (int)C, xx, st));
  if (impl < 0 || impl > 2) return R3DFS_E_UNSUPPORTED;
  return launch_knn_auto(xp, (int)C, (int)C, xx, B, (int)N, k, nullptr, idx_out, impl, st, split,
                         split_bytes);
}

// ---- get_edge_feature --------------------------------------------------------------------------
size_t r3dfs_edge_feature_workspace(int64_t B, int64_t C, int64_t N) {
  return edge_feature_scratch_bytes(B, C, N);
}

int r3dfs_edge_feature(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                       int64_t sn, const int64_t* idx, int K, float* out, void* ws, size_t ws_bytes,
                       r3dfs_stream_t stream) {
  if (!x || !idx || !out || B <= 0 || C <= 0 || N <= 0 || K <= 0) return R3DFS_E_BADARG;
  if (C > 65535 || B > 65535) return R3DFS_E_UNSUPPORTED;
  if (((uintptr_t)out & 15) != 0) return R3DFS_E_ALIGN;
  return launch_edge_feature(x, B, C, N, sb, sc, sn, idx, K, out, (cudaStream_t)stream, ws, ws_bytes);
}

// ---- linear ---------------------------------------------------------------------------------
int r3dfs_linear_ex(const float* x, int64_t ldx, const float* w, const float* s, const float* t,
                    int act, int64_t M, int64_t K, int64_t Nout, float* y, int64_t ldy, int impl,
                    r3dfs_stream_t stream) {
  if (!x || !w || !y || M <= 0 || K <= 0 || Nout <= 0 || ldx < K || ldy < Nout)
    return R3DFS_E_BADARG;
  if (act < 0 || act > 2 || Nout > 65535 * 64 || impl < 0 || impl > 3) return R3DFS_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (impl == 1)
    return launch_linear(x, (int)ldx, w, s, t, act, M, (int)K, (int)Nout, y, (int)ldy,
                         identity_map(), st);
  if (impl == 2)
    return launch_linear_tc(x, (int)ldx, w, s, t, act, M, (int)K, (int)Nout, y, (int)ldy,
                            identity_map(), st);
  if (impl == 3)
    return launch_linear_tma(x, (int)ldx, w, s, t, act, M, (int)K, (int)Nout, y, (int)ldy,
                             identity_map(), st);
  return launch_linear_auto(x, (int)ldx, w, s, t, act, M, (int)K, (int)Nout, y, (int)ldy,
                            identity_map(), st);
}

int r3dfs_linear(const float* x, int64_t ldx, const float* w, const float* s, const float* t,
                 int act, int64_t M, int64_t K, int64_t Nout, float* y, int64_t ldy,
                 r3dfs_stream_t stream) {
  return r3dfs_linear_ex(x, ldx, w, s, t, act, M, K, Nout, y, ldy, 0, stream);
}

// ---- fused EdgeConv block ------------------------------------------------------------------------
size_t r3dfs_edgeconv_workspace(int64_t B, int64_t C, int64_t N, int k) {
  const int64_t M = B * N;
  return align_up(sizeof(float) * M * C, 256) + align_up(sizeof(float) * M, 256) +
         align_up(sizeof(int32_t) * M * k, 256) + align_up(sizeof(float) * 128 * C, 256) +
         2 * 512 + align_up(sizeof(float) * M * 128, 256) +
         align_up(knn_split_bytes((int)C, B, (int)N, k), 256) + 1280;
}

int r3dfs_edgeconv(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                   int64_t sn, int k, const float* w1, const float* s1, const float* t1,
                   const float* w2, const float* s2, const float* t2, float* y, int64_t* idx_out,
                   void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!x || !w1 || !s1 || !t1 || !w2 || !s2 || !t2 || !y || !wsp || B <= 0 || C <= 0 || N <= 0)
    return R3DFS_E_BADARG;
  if (k < 1 || k > 32 || k > N || B > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_edgeconv_workspace(B, C, N, k)) return R3DFS_E_WORKSPACE;
  if (((uintptr_t)y & 15) != 0) return R3DFS_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t M = B * N;
  WsBump ws(wsp, ws_bytes);
  float* xp = ws.take<float>(M * C);
  float* xx = ws.take<float>(M);
  int32_t* idx = ws.take<int32_t>(M * k);
  float* wpq = ws.take<float>(128 * C);
  float* spq = ws.take<float>(128);
  float* tpq = ws.take<float>(128);
  float* PQ = ws.take<float>(M * 128);
  const size_t split_bytes = knn_split_bytes((int)C, B, (int)N, k);
  unsigned char* split = split_bytes ? ws.take<unsigned char>(split_bytes) : nullptr;
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  R3DFS_TRY(launch_to_point_major(x, B, C, N, sb, sc, sn, xp, st));
  R3DFS_TRY(launch_row_norms(xp, M, (int)C, (int)C, xx, st));
  R3DFS_TRY(launch_knn_auto(xp, (int)C, (int)C, xx, B, (int)N, k, idx, idx_out, 0, st, split,
                            split_bytes));
  R3DFS_TRY(launch_fold_edge_w1(w1, s1, t1, (int)C, wpq, spq, tpq, st));
  R3DFS_TRY(launch_linear_auto(xp, (int)C, wpq, spq, tpq, ACT_NONE, M, (int)C, 128, PQ, 128,
                               identity_map(), st));
  return launch_edge_mlp_auto(PQ, idx, w2, s2, t2, B, (int)N, k, y, 64, identity_map(), st);
}

// ---- attention ----------------------------------------------------------------------------------
size_t r3dfs_attention_workspace(int64_t B, int64_t N) {
  return align_up(sizeof(float) * B * N * 192, 256) + align_up(sizeof(float) * B, 256) +
         align_up(attention_split_bytes(B, (int)N), 256) + 512;
}

int r3dfs_attention(const float* x, int64_t B, int64_t N, int64_t Cin, const float* wqkv, float* y,
                    void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!x || !wqkv || !y || !wsp || B <= 0 || N <= 0 || Cin <= 0) return R3DFS_E_BADARG;
  if (B > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_attention_workspace(B, N)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  float* qkv = ws.take<float>(B * N * 192);
  float* kmax = ws.take<float>(B);
  const size_t split_bytes = attention_split_bytes(B, (int)N);
  unsigned char* split = ws.take<unsigned char>(split_bytes);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  R3DFS_TRY(launch_linear_auto(x, (int)Cin, wqkv, nullptr, nullptr, ACT_NONE, B * N, (int)Cin, 192,
                               qkv, 192, identity_map(), st));
  return launch_attention_auto(qkv, 192, B, (int)N, y, 64, identity_map(), st, kmax, split,
                               split_bytes);
}

// ---- getFeatures --------------------------------------------------------------------------------
size_t r3dfs_features_workspace(int64_t B, int64_t N) {
  const int64_t M = B * N;
  // xp (<= 64 ch) + encoder buffers: xx 1, idx 32, PQ 128, ecat 192, h512, l2 256, h128, qkv 192
  return sizeof(float) * M * (64 + 1 + 32 + 128 + 192 + 512 + 256 + 128 + 192) + 128 * 64 * 4 +
         16 * 1024;
}

int r3dfs_features(const r3dfs_weights_t* w, const float* x, int64_t B, int64_t N, int64_t sb,
                   int64_t sc, int64_t sn, float* feat, float* level2, void* wsp, size_t ws_bytes,
                   r3dfs_stream_t stream) {
  R3DFS_TRY(check_weights(w));
  if (!x || !feat || !wsp || B <= 0 || N <= 0) return R3DFS_E_BADARG;
  if (B > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_features_workspace(B, N)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  float* xp = ws.take<float>(B * N * w->in_dim);
  EncoderWs e;
  carve_encoder(ws, B * N, w->dgcnn_k, e);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  R3DFS_TRY(launch_to_point_major(x, B, w->in_dim, N, sb, sc, sn, xp, st));
  return encoder_forward(w, xp, B, (int)N, e, feat, identity_map(), level2, st);
}

// ---- fps ----------------------------------------------------------------------------------------
int r3dfs_fps(const float* feat, int64_t D, const int32_t* set_off, const int32_t* set_n,
              int n_sets, int64_t n_cap, int m_max, int32_t* idx_out, r3dfs_stream_t stream) {
  if (!feat || !set_off || !set_n || !idx_out || n_sets <= 0 || m_max <= 0 || n_cap <= 0)
    return R3DFS_E_BADARG;
  if (n_sets > 65535) return R3DFS_E_UNSUPPORTED;
  return launch_fps_ex(feat, (int)D, set_off, set_n, n_sets, (int)n_cap, m_max, 0, idx_out,
                       nullptr, (cudaStream_t)stream);
}

size_t r3dfs_fps_workspace(int64_t total_rows) {
  return total_rows > 0 ? fps_q8_spill_bytes(total_rows) + 256 : 0;
}

int r3dfs_fps_ex(const float* feat, int64_t D, const int32_t* set_off, const int32_t* set_n,
                 int n_sets, int64_t n_cap, int64_t total_rows, int m_max, int impl,
                 int32_t* idx_out, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!feat || !set_off || !set_n || !idx_out || n_sets <= 0 || m_max <= 0 || n_cap <= 0 ||
      total_rows <= 0 || impl < R3DFS_FPS_AUTO || impl > R3DFS_FPS_Q8)
    return R3DFS_E_BADARG;
  if (n_sets > 65535) return R3DFS_E_UNSUPPORTED;
  uint8_t* spill = nullptr;
  if (impl != R3DFS_FPS_STREAM && wsp) {
    if (ws_bytes < r3dfs_fps_workspace(total_rows)) return R3DFS_E_WORKSPACE;
    WsBump ws(wsp, ws_bytes);
    spill = ws.take<uint8_t>(fps_q8_spill_bytes(total_rows));
  }
  return launch_fps_ex(feat, (int)D, set_off, set_n, n_sets, (int)n_cap, m_max, 0, idx_out,
                       nullptr, (cudaStream_t)stream, spill, 1, impl);
}

// ---- getMutiplePrototypes -------------------------------------------------------------------------
size_t r3dfs_multi_prototypes_workspace(int64_t total_rows, int n_sets, int k) {
  const size_t ch = multi_prototypes_chunks((int)total_rows);
  return align_up(fps_q8_spill_bytes(total_rows), 256) +
         align_up(sizeof(int32_t) * (size_t)n_sets * (k + 1), 256) +
         align_up(sizeof(int32_t) * (size_t)n_sets, 256) +
         align_up(sizeof(float) * (size_t)n_sets * ch * (k + 1) * 256, 256) +
         align_up(sizeof(int32_t) * (size_t)n_sets * ch * (k + 1), 256) +
         align_up(sizeof(float) * (size_t)n_sets * 256, 256) + 2048;
}

int r3dfs_multi_prototypes(const float* feat, int64_t D, const int32_t* set_off,
                           const int32_t* set_n, int n_sets, int64_t total_rows, int k,
                           float* proto_out, int32_t* proto_count, int32_t* assign_out,
                           int32_t* seed_idx_out, void* wsp, size_t ws_bytes,
                           r3dfs_stream_t stream) {
  if (!feat || !set_off || !set_n || !proto_out || !proto_count || !assign_out || !seed_idx_out ||
      !wsp || n_sets <= 0 || total_rows <= 0 || k <= 0)
    return R3DFS_E_BADARG;
  if (n_sets > 65535 || k > 127) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_multi_prototypes_workspace(total_rows, n_sets, k)) return R3DFS_E_WORKSPACE;
  WsBump ws(wsp, ws_bytes);
  int32_t* picks = ws.take<int32_t>((size_t)n_sets * (k + 1));
  int32_t* pick_cnt = ws.take<int32_t>(n_sets);
  const size_t ch = multi_prototypes_chunks((int)total_rows);
  float* partial = ws.take<float>((size_t)n_sets * ch * (k + 1) * D);
  int32_t* pcount = ws.take<int32_t>((size_t)n_sets * ch * (k + 1));
  float* seed_stats = ws.take<float>((size_t)n_sets * 256);
  uint8_t* fps_spill = ws.take<uint8_t>(fps_q8_spill_bytes(total_rows));
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  // n_cap: no set can be larger than the whole buffer
  return launch_multi_prototypes(feat, (int)D, set_off, set_n, n_sets, (int)total_rows, k, picks,
                                 pick_cnt, seed_idx_out, proto_count, assign_out, partial, pcount,
                                 seed_stats, n_sets,
                                 (int64_t)n_sets * (k + 1), proto_out, (int)D,
                                 (cudaStream_t)stream, nullptr, fps_spill);
}

// ---- multi-scale degree-based noise suppression ------------------------------------------------------
size_t r3dfs_mdns_workspace(int n_episodes, int n_way, int k_shot) {
  if (n_episodes <= 0 || n_way <= 0 || k_shot <= 0) return 0;
  return align_up(sizeof(int32_t) * (size_t)n_episodes * n_way * k_shot, 256) + 256;
}

int r3dfs_mdns(const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c, int64_t s_n,
               const int32_t* support_y, const float* support_feat, int n_episodes, int n_way,
               int k_shot, int64_t N, float* cell_mean, int32_t* cell_count, uint8_t* cell_mask,
               float* degree, float* scale_flag, int32_t* keep, float* clean_flag, void* wsp,
               size_t ws_bytes, r3dfs_stream_t stream) {
  if (!support_x || !support_y || !support_feat || !cell_mean || !cell_count || !keep || !wsp ||
      n_episodes <= 0 || n_way <= 0 || k_shot <= 0 || N <= 0)
    return R3DFS_E_BADARG;
  if (N > 200 * 1024) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mdns_workspace(n_episodes, n_way, k_shot)) return R3DFS_E_WORKSPACE;
  WsBump ws(wsp, ws_bytes);
  int32_t* fg_cnt = ws.take<int32_t>((size_t)n_episodes * n_way * k_shot);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  return launch_mdns(support_x, s_e, s_cloud, s_c, s_n, support_y, support_feat,
                     (int64_t)n_way * k_shot * N, 0, n_episodes, n_way, k_shot, (int)N,
                     R3DFS_FEAT_DIM, cell_mean, cell_count, fg_cnt, keep, clean_flag,
                     (cudaStream_t)stream, cell_mask, degree, scale_flag);
}

// ---- affinity + label propagation -------------------------------------------------------------------
size_t r3dfs_affinity_workspace(int n_graphs, int64_t n_max, int64_t D, int k) {
  (void)D;
  (void)k;
  return align_up(sizeof(float) * (size_t)n_graphs * n_max, 256) +
         align_up(sizeof(float) * (size_t)n_graphs * n_max * n_max, 256) + 512;
}

int r3dfs_affinity_knn(const float* node_feat, const uint8_t* valid, int n_graphs, int64_t n_max,
                       int64_t D, int k, float sigma, int32_t* nbr, float* sim, void* wsp,
                       size_t ws_bytes, r3dfs_stream_t stream) {
  if (!node_feat || !valid || !nbr || !sim || !wsp || n_graphs <= 0 || n_max <= 0 || k <= 0)
    return R3DFS_E_BADARG;
  if (k >= n_max || n_graphs > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_affinity_workspace(n_graphs, n_max, D, k)) return R3DFS_E_WORKSPACE;
  WsBump ws(wsp, ws_bytes);
  float* norms = ws.take<float>((size_t)n_graphs * n_max);
  float* D2 = ws.take<float>((size_t)n_graphs * n_max * n_max);
  return launch_affinity(node_feat, n_max, 0, valid, n_graphs, (int)n_max, (int)D, k, sigma, norms,
                         D2, nbr, sim, (cudaStream_t)stream);
}

// scratch shared by the sort-free in-edge build (bit matrix + rank prefixes) and, after it, by the
// solver (row schedule table of up to 16 CTAs per graph + the row lists re-packed in schedule order)
static size_t lp_scratch_bytes(size_t G, size_t n, int k) {
  const size_t inedge = 6 * G * n * ((n + 31) / 32);
  const size_t solver = lp_solver_scratch_bytes(G, n, k);
  return inedge > solver ? inedge : solver;
}

size_t r3dfs_label_propagate_workspace(int n_graphs, int64_t n_max, int k, int n_cls) {
  const size_t G = n_graphs, n = n_max;
  (void)n_cls;
  return align_up(4 * G * n * k, 256) * 3 + align_up(4 * G * (n + 1), 256) * 6 +
         align_up(4 * G * n * 8, 256) * 4 + align_up(6 * G * n * (size_t)lp_rowcap(k), 256) +
         align_up(lp_scratch_bytes(G, n, k), 256) + 8192;
}

int r3dfs_label_propagate(const int32_t* nbr, const float* sim, const uint8_t* valid, int n_graphs,
                          int64_t n_max, int k, const float* Y, int n_cls, float alpha, float tol,
                          int max_iter, float* Z, int32_t* iters_out, float* resid_out, void* wsp,
                          size_t ws_bytes, r3dfs_stream_t stream) {
  if (!nbr || !sim || !valid || !Y || !Z || !wsp || n_graphs <= 0 || n_max <= 0 || k <= 0)
    return R3DFS_E_BADARG;
  if (n_graphs > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_label_propagate_workspace(n_graphs, n_max, k, n_cls))
    return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t G = n_graphs, n = n_max;
  WsBump ws(wsp, ws_bytes);
  float* sv = ws.take<float>(G * n * k);
  int32_t* in_src = ws.take<int32_t>(G * n * k);
  float* in_w = ws.take<float>(G * n * k);
  int32_t* in_cnt = ws.take<int32_t>(G * (n + 1));
  int32_t* in_ptr = ws.take<int32_t>(G * (n + 1));
  float* dinv = ws.take<float>(G * (n + 1));
  int32_t* rowptr = ws.take<int32_t>(G * n);
  int32_t* rowlen = ws.take<int32_t>(G * n);
  int32_t* cursor = ws.take<int32_t>(G);
  uint16_t* mcol = ws.take<uint16_t>(G * n * lp_rowcap(k));
  float* mval = ws.take<float>(G * n * lp_rowcap(k));
  float* X = ws.take<float>(G * n * 8);
  float* R = ws.take<float>(G * n * 8);
  float* P = ws.take<float>(G * n * 8);
  float* AP = ws.take<float>(G * n * 8);
  const size_t scratch_bytes = lp_scratch_bytes(G, n, k);
  unsigned char* scratch = ws.take<unsigned char>(scratch_bytes);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  cudaError_t ce = cudaMemcpyAsync(sv, sim, sizeof(float) * G * n * k, cudaMemcpyDeviceToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  return launch_label_propagate(nbr, sv, valid, n_graphs, (int)n_max, k, Y, n_cls, alpha, tol,
                                max_iter, in_cnt, in_ptr, in_src, in_w, dinv, rowptr, rowlen, cursor,
                                mcol, mval, Z, X, R, P, AP, iters_out, resid_out, st, nullptr,
                                scratch, scratch_bytes);
}

// ---- dense FP64 Cholesky solve of the same system (cross-check of the CG solve) -----------------------
size_t r3dfs_lp_cholesky_workspace(int n_graphs, int64_t n_max, int k, int n_cls) {
  if (n_graphs <= 0 || n_max <= 0 || k <= 0) return 0;
  return r3dfs_label_propagate_workspace(n_graphs, n_max, k, n_cls) +
         lp_cholesky_scratch_bytes(n_graphs, (int)n_max) + 1024;
}

int r3dfs_lp_cholesky(const int32_t* nbr, const float* sim, const uint8_t* valid, int n_graphs,
                      int64_t n_max, int k, const float* Y, int n_cls, float alpha, float* Z,
                      int32_t* info_out, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!nbr || !sim || !valid || !Y || !Z || !wsp || n_graphs <= 0 || n_max <= 0 || k <= 0)
    return R3DFS_E_BADARG;
  if (n_graphs > 65535 || n_max > 8192) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_lp_cholesky_workspace(n_graphs, n_max, k, n_cls)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t G = n_graphs, n = n_max;
  WsBump ws(wsp, ws_bytes);
  float* sv = ws.take<float>(G * n * k);
  int32_t* in_src = ws.take<int32_t>(G * n * k);
  float* in_w = ws.take<float>(G * n * k);
  int32_t* in_cnt = ws.take<int32_t>(G * (n + 1));
  int32_t* in_ptr = ws.take<int32_t>(G * (n + 1));
  float* dinv = ws.take<float>(G * (n + 1));
  int32_t* rowptr = ws.take<int32_t>(G * n);
  int32_t* rowlen = ws.take<int32_t>(G * n);
  int32_t* cursor = ws.take<int32_t>(G);
  uint16_t* mcol = ws.take<uint16_t>(G * n * lp_rowcap(k));
  float* mval = ws.take<float>(G * n * lp_rowcap(k));
  const size_t scratch_bytes = lp_scratch_bytes(G, n, k);
  unsigned char* scratch = ws.take<unsigned char>(scratch_bytes);
  unsigned char* dense = ws.take<unsigned char>(lp_cholesky_scratch_bytes(n_graphs, (int)n_max));
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  cudaError_t ce = cudaMemcpyAsync(sv, sim, sizeof(float) * G * n * k, cudaMemcpyDeviceToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  return launch_label_propagate(nbr, sv, valid, n_graphs, (int)n_max, k, Y, n_cls, alpha, 0.f, 0,
                                in_cnt, in_ptr, in_src, in_w, dinv, rowptr, rowlen, cursor, mcol,
                                mval, Z, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, st,
                                nullptr, scratch, scratch_bytes, false, dense, info_out);
}

// ---- confusion counters ----------------------------------------------------------------------------
int r3dfs_confusion_accumulate(const int32_t* pred, const int64_t* gt, const int32_t* class_slot,
                               int n_episodes, int n_way, int64_t pts_per_episode, int n_slots,
                               int64_t* counters, r3dfs_stream_t stream) {
  if (!pred || !gt || !class_slot || !counters || n_episodes <= 0 || n_way <= 0 ||
      pts_per_episode <= 0 || n_slots <= 0)
    return R3DFS_E_BADARG;
  return launch_confusion(pred, gt, class_slot, n_episodes, n_way, pts_per_episode, n_slots,
                          counters, (cudaStream_t)stream);
}

// ---- whole episodes ---------------------------------------------------------------------------------
}  // extern "C"

int episode_dims(const r3dfs_episode_cfg_t* c, EpisodeDims& d) {
  if (!c) return R3DFS_E_BADARG;
  if (c->n_way < 1 || c->n_way > 7 || c->k_shot < 1 || c->k_shot > 32 || c->n_query < 1 ||
      c->n_points < 64 || c->n_subprototypes < 1 || c->n_subprototypes > 127 || c->k_connect < 1 ||
      c->k_connect > 1024)
    return R3DFS_E_UNSUPPORTED;
  d.S = c->n_way + 1;
  d.nc = c->n_way + 1;
  d.slot = c->n_subprototypes + 1;
  d.ppad = (d.S * d.slot + 63) / 64 * 64;
  d.nq_pts = c->n_query * c->n_points;
  d.nn = d.ppad + d.nq_pts;
  d.C = c->n_way * c->k_shot;
  d.ns_pts = d.C * c->n_points;
  d.cpe = c->n_query + d.C;
  d.ep_rows = (int64_t)d.nn + d.ns_pts;
  if (d.nn > 8192 || c->k_connect >= d.nq_pts) return R3DFS_E_UNSUPPORTED;
  return 0;
}

// buffers of the support part (noise suppression, set compaction, prototypes) for G episodes
static void carve_support_bufs(WsBump& ws, const EpisodeDims& d, size_t G, EpisodeWs& w) {
  w.fg_cnt = ws.take<int32_t>(G * d.C);
  w.keep = ws.take<int32_t>(G * d.C);
  w.set_off = ws.take<int32_t>(G * d.S);
  w.set_n = ws.take<int32_t>(G * d.S);
  w.cloud_bg_off = ws.take<int32_t>(G * d.C);
  w.cloud_fg_off = ws.take<int32_t>(G * d.C);
  w.setfeat = ws.take<float>(G * d.ns_pts * R3DFS_FEAT_DIM);
  w.fps_spill = ws.take<uint8_t>(fps_q8_spill_bytes((int64_t)G * d.ns_pts));
  w.picks = ws.take<int32_t>(G * d.S * d.slot);
  w.pick_cnt = ws.take<int32_t>(G * d.S);
  w.seeds = ws.take<int32_t>(G * d.S * d.slot);
  w.assign = ws.take<int32_t>(G * d.ns_pts);
  {
    const size_t ch = multi_prototypes_chunks(d.ns_pts);
    w.partial = ws.take<float>(G * d.S * ch * d.slot * R3DFS_FEAT_DIM);
    w.pcount = ws.take<int32_t>(G * d.S * ch * d.slot);
    w.seed_stats = ws.take<float>(G * d.S * 256);
  }
  w.cell_mean = ws.take<float>(G * d.C * 5 * R3DFS_FEAT_DIM);
  w.cell_cnt = ws.take<int32_t>(G * d.C * 5);
}

// buffers of the query part (graph, label propagation) for G episodes
static void carve_graph_bufs(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d,
                             size_t G, EpisodeWs& w) {
  const size_t nn = d.nn, k = c->k_connect;
  w.valid = ws.take<uint8_t>(G * nn);
  w.Y = ws.take<float>(G * nn * d.nc);
  w.norms = ws.take<float>(G * nn);
  // dense squared distances; afterwards scratch of the in-edge build and of the solver's packed rows
  w.D2 = ws.take<float>(episode_d2_floats(G, nn, k));
  w.nbr = ws.take<int32_t>(G * nn * k);
  w.sim = ws.take<float>(G * nn * k);
  w.in_cnt = ws.take<int32_t>(G * (nn + 1));
  w.in_ptr = ws.take<int32_t>(G * (nn + 1));
  w.in_src = ws.take<int32_t>(G * nn * k);
  w.in_w = ws.take<float>(G * nn * k);
  w.dinv = ws.take<float>(G * nn);
  w.rowptr = ws.take<int32_t>(G * nn);
  w.rowlen = ws.take<int32_t>(G * nn);
  w.cursor = ws.take<int32_t>(G);
  w.mcol = ws.take<uint16_t>(G * nn * lp_rowcap(k));
  w.mval = ws.take<float>(G * nn * lp_rowcap(k));
  w.Z = ws.take<float>(G * nn * d.nc);
  w.X = ws.take<float>(G * nn * 8);
  w.R = ws.take<float>(G * nn * 8);
  w.P = ws.take<float>(G * nn * 8);
  w.AP = ws.take<float>(G * nn * 8);
}

void carve_episode(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d, int E,
                          int in_dim, int dg_k, EpisodeWs& w) {
  const int64_t M = (int64_t)E * d.cpe * c->n_points;
  w.xp = ws.take<float>(M * in_dim);
  carve_encoder(ws, M, dg_k, w.enc);
  w.F = ws.take<float>((size_t)E * d.ep_rows * R3DFS_FEAT_DIM);
  carve_support_bufs(ws, d, E, w);
  w.proto_cnt = ws.take<int32_t>((size_t)E * d.S);
  carve_graph_bufs(ws, c, d, E, w);
}

// support call: the support clouds' encoder buffers, their feature rows (n_sets blocks of ns_pts
// rows) and the support part's buffers; no graph buffers (proto_cnt is the caller's output)
static void carve_support(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d,
                          int n_sets, int in_dim, int dg_k, EpisodeWs& w) {
  const int64_t M = (int64_t)n_sets * d.C * c->n_points;
  w = EpisodeWs{};
  w.xp = ws.take<float>(M * in_dim);
  carve_encoder(ws, M, dg_k, w.enc);
  w.F = ws.take<float>((size_t)n_sets * d.ns_pts * R3DFS_FEAT_DIM);
  carve_support_bufs(ws, d, n_sets, w);
}

// query call: the query clouds' encoder buffers, nodes-only feature blocks (nn rows per episode:
// prototype slots, then query points), the clamped prototype counts and the graph buffers
static void carve_query(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d, int E,
                        int in_dim, int dg_k, EpisodeWs& w) {
  const int64_t M = (int64_t)E * c->n_query * c->n_points;
  w = EpisodeWs{};
  w.xp = ws.take<float>(M * in_dim);
  carve_encoder(ws, M, dg_k, w.enc);
  w.F = ws.take<float>((size_t)E * d.nn * R3DFS_FEAT_DIM);
  w.proto_cnt = ws.take<int32_t>((size_t)E * d.S);
  carve_graph_bufs(ws, c, d, E, w);
}

// floats of the D2 area of G graphs: the n x n distance matrix, or the solver scratch if that is larger
size_t episode_d2_floats(size_t G, size_t nn, int k) {
  const size_t dense = G * nn * nn, solver = (lp_solver_scratch_bytes(G, nn, k) + 3) / 4;
  return dense > solver ? dense : solver;
}

size_t r3dfs_mpti_workspace(const r3dfs_episode_cfg_t* cfg, int n_episodes) {
  EpisodeDims d;
  if (episode_dims(cfg, d) != 0 || n_episodes <= 0) return 0;
  WsBump ws(nullptr, ~(size_t)0);
  EpisodeWs w;
  carve_episode(ws, cfg, d, n_episodes, 64, 32, w);
  return ws.off + 4096;
}

// support part of the episode (models/mpti.py:440-493): noise suppression, fg/bg sets, FPS seeds,
// assignment, prototype means.  F rows [sup_off, sup_off + ns_pts) of every f_rows-row block hold
// the support features; prototype p of set s of episode e is written to row
// e * proto_rows + s * slot + p of `proto` (rows p >= w.proto_cnt are not written).
static int episode_support_part(const r3dfs_episode_cfg_t* cfg, const EpisodeDims& d, int E,
                                const EpisodeWs& w, int64_t f_rows, int64_t sup_off,
                                const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                                int64_t s_n, const int32_t* support_y, float* proto,
                                int64_t proto_rows, float* clean_flag, cudaStream_t st,
                                const StageRec* sr) {
  const int N = cfg->n_points, D = R3DFS_FEAT_DIM;
  // noise suppression over support shots (eval only, models/mpti.py:440-442)
  if (cfg->mdns) {
    R3DFS_TRY(launch_mdns(support_x, s_e, s_cloud, s_c, s_n, support_y, w.F, f_rows, sup_off, E,
                          cfg->n_way, cfg->k_shot, N, D, w.cell_mean, w.cell_cnt, w.fg_cnt, w.keep,
                          clean_flag, st));
  } else {
    fill_i32_kernel<<<nblk((int64_t)E * d.C), 256, 0, st>>>(w.keep, (int64_t)E * d.C, 1);
    R3DFS_CHECK_LAUNCH();
  }
  if (sr) sr->mark(R3DFS_ST_MDNS, st);
  // prototype sets -> FPS seeds -> assignment -> means
  R3DFS_TRY(launch_set_compaction(w.F, f_rows, sup_off, E, cfg->n_way, cfg->k_shot, N, D,
                                  support_y, w.keep, w.fg_cnt, w.set_off, w.set_n, w.cloud_bg_off,
                                  w.cloud_fg_off, w.setfeat, st));
  if (sr) sr->mark(R3DFS_ST_SETS, st);
  R3DFS_TRY(launch_multi_prototypes(w.setfeat, D, w.set_off, w.set_n, E * d.S, d.ns_pts,
                                    cfg->n_subprototypes, w.picks, w.pick_cnt, w.seeds,
                                    w.proto_cnt, w.assign, w.partial, w.pcount, w.seed_stats, d.S,
                                    proto_rows, proto, D, st, sr, w.fps_spill, d.S));
  if (sr) sr->mark(R3DFS_ST_PROTO, st);
  return 0;
}

// query part of the episode (models/mpti.py:493-571): F holds, in blocks of f_rows rows per
// episode, the prototype slots (rows [0, ppad), zero where no prototype) and the query features
// (rows [ppad, nn)); w.proto_cnt the prototype count of every set.  Graph, label propagation, head.
static int episode_query_part(const r3dfs_episode_cfg_t* cfg, const EpisodeDims& d, int E,
                              const EpisodeWs& w, int64_t f_rows, const int64_t* query_y,
                              float* logits, float* loss, int32_t* pred,
                              const r3dfs_episode_diag_t* diag, cudaStream_t st,
                              const StageRec* sr, bool latency) {
  const int D = R3DFS_FEAT_DIM;
  // graph: nodes = [prototype slots | query points]
  graph_init_kernel<<<dim3(nblk(d.nn), E), 256, 0, st>>>(w.proto_cnt, d.S, d.slot, d.ppad, d.nn,
                                                         d.nc, w.valid, w.Y);
  R3DFS_CHECK_LAUNCH();
  R3DFS_TRY(launch_affinity(w.F, f_rows, 0, w.valid, E, d.nn, D, cfg->k_connect, cfg->sigma,
                            w.norms, w.D2, w.nbr, w.sim, st, sr));
  R3DFS_TRY(launch_label_propagate(w.nbr, w.sim, w.valid, E, d.nn, cfg->k_connect, w.Y, d.nc,
                                   cfg->alpha, cfg->cg_tol, cfg->cg_max_iter, w.in_cnt, w.in_ptr,
                                   w.in_src, w.in_w, w.dinv, w.rowptr, w.rowlen, w.cursor, w.mcol,
                                   w.mval, w.Z, w.X, w.R, w.P, w.AP,
                                   diag ? diag->cg_iters : nullptr,
                                   diag ? diag->cg_resid : nullptr, st, sr, w.D2,
                                   sizeof(float) * episode_d2_floats(E, d.nn, cfg->k_connect),  // D2 is dead here
                                   latency));
  // query rows -> logits / loss / prediction
  R3DFS_TRY(launch_query_head(w.Z, E, d.nn, d.ppad, d.nq_pts, d.nc, query_y, logits, loss, pred, st));
  if (sr) sr->mark(R3DFS_ST_HEAD, st);
  if (diag && diag->proto_count) {
    cudaError_t ce = cudaMemcpyAsync(diag->proto_count, w.proto_cnt,
                                     sizeof(int32_t) * (size_t)E * d.S, cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return (int)ce;
  }
  return 0;
}

// graph half of the episode: F already holds the query + support features (rows ppad.. of every
// episode block); everything after getFeatures in models/mpti.py:440-571.  The prototypes go
// straight into the prototype slots of F.
int episode_graph_half(const r3dfs_episode_cfg_t* cfg, const EpisodeDims& d, int E,
                              const EpisodeWs& w, const float* support_x, int64_t s_e,
                              int64_t s_cloud, int64_t s_c, int64_t s_n, const int32_t* support_y,
                              const int64_t* query_y, float* logits, float* loss, int32_t* pred,
                              const r3dfs_episode_diag_t* diag, cudaStream_t st, bool latency) {
  const int D = R3DFS_FEAT_DIM;
  StageRec srv{diag ? (cudaEvent_t*)diag->h_stage_events : nullptr};
  const StageRec* sr = srv.ev ? &srv : nullptr;
  cudaError_t ce = cudaMemset2DAsync(w.F, sizeof(float) * d.ep_rows * D, 0,
                                     sizeof(float) * (size_t)d.ppad * D, E, st);
  if (ce != cudaSuccess) return (int)ce;
  R3DFS_TRY(episode_support_part(cfg, d, E, w, d.ep_rows, d.nn, support_x, s_e, s_cloud, s_c, s_n,
                                 support_y, w.F, d.ep_rows, diag ? diag->clean_flag : nullptr, st,
                                 sr));
  return episode_query_part(cfg, d, E, w, d.ep_rows, query_y, logits, loss, pred, diag, st, sr,
                            latency);
}

size_t r3dfs_mpti_support_workspace(const r3dfs_episode_cfg_t* cfg, int n_sets) {
  EpisodeDims d;
  if (episode_dims(cfg, d) != 0 || n_sets <= 0) return 0;
  WsBump ws(nullptr, ~(size_t)0);
  EpisodeWs w;
  carve_support(ws, cfg, d, n_sets, 64, 32, w);
  return ws.off + 4096;
}

// the query call uses no k_shot: its dims are taken with k_shot = 1, so that neither the envelope
// check nor the workspace depends on it
static int query_dims(const r3dfs_episode_cfg_t* cfg, r3dfs_episode_cfg_t& qc, EpisodeDims& d) {
  if (!cfg) return R3DFS_E_BADARG;
  qc = *cfg;
  qc.k_shot = 1;
  qc.mdns = 0;
  return episode_dims(&qc, d);
}

size_t r3dfs_mpti_query_workspace(const r3dfs_episode_cfg_t* cfg, int n_episodes) {
  r3dfs_episode_cfg_t qc;
  EpisodeDims d;
  if (query_dims(cfg, qc, d) != 0 || n_episodes <= 0) return 0;
  WsBump ws(nullptr, ~(size_t)0);
  EpisodeWs w;
  carve_query(ws, &qc, d, n_episodes, 64, 32, w);
  return ws.off + 4096;
}

extern "C" {

int r3dfs_mpti_forward(const r3dfs_episode_cfg_t* cfg, const r3dfs_weights_t* hw, int E,
                       const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                       int64_t s_n, const int32_t* support_y, const float* query_x, int64_t q_e,
                       int64_t q_cloud, int64_t q_c, int64_t q_n, const int64_t* query_y,
                       float* logits, float* loss, int32_t* pred, const r3dfs_episode_diag_t* diag,
                       void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg, d));
  R3DFS_TRY(check_weights(hw));
  if (!support_x || !support_y || !query_x || !logits || !wsp || E <= 0) return R3DFS_E_BADARG;
  if ((int64_t)E * d.cpe > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mpti_workspace(cfg, E)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = cfg->n_points, in_dim = hw->in_dim;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_episode(ws, cfg, d, E, in_dim, hw->dgcnn_k, w);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  const int64_t B = (int64_t)E * d.cpe;
  StageRec srv{diag ? (cudaEvent_t*)diag->h_stage_events : nullptr};
  const StageRec* sr = srv.ev ? &srv : nullptr;
  if (sr) sr->mark(R3DFS_ST_BEGIN, st);
  // clouds -> point-major, episode-major order [queries | supports] (matches F's row layout)
  int64_t tq = (int64_t)E * cfg->n_query * N * in_dim;
  gather_clouds_kernel<<<nblk(tq), 256, 0, st>>>(query_x, cfg->n_query, in_dim, N, q_e, q_cloud,
                                                 q_c, q_n, d.cpe, 0, w.xp, tq);
  R3DFS_CHECK_LAUNCH();
  int64_t tsup = (int64_t)E * d.C * N * in_dim;
  gather_clouds_kernel<<<nblk(tsup), 256, 0, st>>>(support_x, d.C, in_dim, N, s_e, s_cloud, s_c,
                                                   s_n, d.cpe, cfg->n_query, w.xp, tsup);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_INPUT, st);
  // features of every cloud (models/mpti.py:433-437), written straight into the node matrix
  RowMap fmap{d.cpe, N, d.ep_rows, (int64_t)d.ppad};
  R3DFS_TRY(encoder_forward(hw, w.xp, B, N, w.enc, w.F, fmap, nullptr, st, sr));
  return episode_graph_half(cfg, d, E, w, support_x, s_e, s_cloud, s_c, s_n, support_y, query_y,
                            logits, loss, pred, diag, st);
}

int r3dfs_protonet_forward(const r3dfs_episode_cfg_t* cfg, const r3dfs_weights_t* hw, int E,
                           const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                           int64_t s_n, const int32_t* support_y, const float* query_x, int64_t q_e,
                           int64_t q_cloud, int64_t q_c, int64_t q_n, const int64_t* query_y,
                           int dist_method, float* logits, float* loss, int32_t* pred,
                           float* clean_flag, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg, d));
  R3DFS_TRY(check_weights(hw));
  if (!support_x || !support_y || !query_x || !logits || !wsp || E <= 0) return R3DFS_E_BADARG;
  if (dist_method != 0 || (int64_t)E * d.cpe > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mpti_workspace(cfg, E)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = cfg->n_points, in_dim = hw->in_dim, D = R3DFS_FEAT_DIM;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_episode(ws, cfg, d, E, in_dim, hw->dgcnn_k, w);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  const int64_t B = (int64_t)E * d.cpe;
  int64_t tq = (int64_t)E * cfg->n_query * N * in_dim;
  gather_clouds_kernel<<<nblk(tq), 256, 0, st>>>(query_x, cfg->n_query, in_dim, N, q_e, q_cloud,
                                                 q_c, q_n, d.cpe, 0, w.xp, tq);
  R3DFS_CHECK_LAUNCH();
  int64_t tsup = (int64_t)E * d.C * N * in_dim;
  gather_clouds_kernel<<<nblk(tsup), 256, 0, st>>>(support_x, d.C, in_dim, N, s_e, s_cloud, s_c,
                                                   s_n, d.cpe, cfg->n_query, w.xp, tsup);
  R3DFS_CHECK_LAUNCH();
  RowMap fmap{d.cpe, N, d.ep_rows, (int64_t)d.ppad};
  R3DFS_TRY(encoder_forward(hw, w.xp, B, N, w.enc, w.F, fmap, nullptr, st));
  const int32_t* keep = nullptr;
  if (cfg->mdns) {  // Mean_pl_support_y_multi_scale (models/protonet.py:491-536) = the MPTI kernels
    R3DFS_TRY(launch_mdns(support_x, s_e, s_cloud, s_c, s_n, support_y, w.F, d.ep_rows, d.nn, E,
                          cfg->n_way, cfg->k_shot, N, D, w.cell_mean, w.cell_cnt, w.fg_cnt, w.keep,
                          clean_flag, st));
    keep = w.keep;
  }
  // pooled vectors and prototypes live in the (otherwise unused) compacted-set buffer
  float* fg = w.setfeat;
  float* bg = fg + (size_t)E * d.C * D;
  float* proto = bg + (size_t)E * d.C * D;
  R3DFS_TRY(launch_protonet_head(w.F, d.ep_rows, d.nn, d.ppad, E, cfg->n_way, cfg->k_shot, N,
                                 d.nq_pts, D, support_y, keep, dist_method, fg, bg, proto, w.Z, d.nn,
                                 st));
  return launch_query_head(w.Z, E, d.nn, d.ppad, d.nq_pts, d.nc, query_y, logits, loss, pred, st);
}

int r3dfs_mpti_forward_features(const r3dfs_episode_cfg_t* cfg, int E, const float* support_x,
                                int64_t s_e, int64_t s_cloud, int64_t s_c, int64_t s_n,
                                const int32_t* support_y, const float* support_feat,
                                const float* query_feat, const int64_t* query_y, float* logits,
                                float* loss, int32_t* pred, const r3dfs_episode_diag_t* diag,
                                void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg, d));
  if (!support_x || !support_y || !support_feat || !query_feat || !logits || !wsp || E <= 0)
    return R3DFS_E_BADARG;
  if ((int64_t)E * d.cpe > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mpti_workspace(cfg, E)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int D = R3DFS_FEAT_DIM;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_episode(ws, cfg, d, E, 64, 32, w);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  const size_t pitch = sizeof(float) * d.ep_rows * D;
  cudaError_t ce = cudaMemcpy2DAsync(w.F + (size_t)d.ppad * D, pitch, query_feat,
                                     sizeof(float) * (size_t)d.nq_pts * D,
                                     sizeof(float) * (size_t)d.nq_pts * D, E,
                                     cudaMemcpyDeviceToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  ce = cudaMemcpy2DAsync(w.F + (size_t)d.nn * D, pitch, support_feat,
                         sizeof(float) * (size_t)d.ns_pts * D,
                         sizeof(float) * (size_t)d.ns_pts * D, E, cudaMemcpyDeviceToDevice, st);
  if (ce != cudaSuccess) return (int)ce;
  return episode_graph_half(cfg, d, E, w, support_x, s_e, s_cloud, s_c, s_n, support_y, query_y,
                            logits, loss, pred, diag, st);
}

// stage events a half does not run are recorded where it stands, so every interval is defined
static void mark_stages(const StageRec* sr, int first, int last, cudaStream_t st) {
  if (!sr) return;
  for (int i = first; i <= last; ++i) sr->mark(i, st);
}

int r3dfs_mpti_support(const r3dfs_episode_cfg_t* cfg, const r3dfs_weights_t* hw, int n_sets,
                       const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                       int64_t s_n, const int32_t* support_y, float* proto, int32_t* proto_count,
                       const r3dfs_episode_diag_t* diag, void* wsp, size_t ws_bytes,
                       r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg, d));
  R3DFS_TRY(check_weights(hw));
  if (!support_x || !support_y || !proto || !proto_count || !wsp || n_sets <= 0)
    return R3DFS_E_BADARG;
  if ((int64_t)n_sets * d.C > 65535) return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mpti_support_workspace(cfg, n_sets)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = cfg->n_points, in_dim = hw->in_dim, D = R3DFS_FEAT_DIM;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_support(ws, cfg, d, n_sets, in_dim, hw->dgcnn_k, w);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  w.proto_cnt = proto_count;
  StageRec srv{diag ? (cudaEvent_t*)diag->h_stage_events : nullptr};
  const StageRec* sr = srv.ev ? &srv : nullptr;
  if (sr) sr->mark(R3DFS_ST_BEGIN, st);
  const int64_t proto_rows = (int64_t)d.S * d.slot;
  cudaError_t ce = cudaMemsetAsync(proto, 0, sizeof(float) * (size_t)n_sets * proto_rows * D, st);
  if (ce != cudaSuccess) return (int)ce;
  const int64_t tsup = (int64_t)n_sets * d.C * N * in_dim;
  gather_clouds_kernel<<<nblk(tsup), 256, 0, st>>>(support_x, d.C, in_dim, N, s_e, s_cloud, s_c,
                                                   s_n, d.C, 0, w.xp, tsup);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_INPUT, st);
  // features of the support clouds only (models/mpti.py:433-435), ns_pts rows per set
  RowMap fmap{d.C, N, (int64_t)d.ns_pts, 0};
  R3DFS_TRY(encoder_forward(hw, w.xp, (int64_t)n_sets * d.C, N, w.enc, w.F, fmap, nullptr, st, sr));
  R3DFS_TRY(episode_support_part(cfg, d, n_sets, w, d.ns_pts, 0, support_x, s_e, s_cloud, s_c, s_n,
                                 support_y, proto, proto_rows, diag ? diag->clean_flag : nullptr,
                                 st, sr));
  mark_stages(sr, R3DFS_ST_DIST, R3DFS_ST_HEAD, st);
  return 0;
}

int r3dfs_mpti_query(const r3dfs_episode_cfg_t* cfg, const r3dfs_weights_t* hw, int E,
                     const float* proto, int64_t p_e, const int32_t* proto_count, int64_t c_e,
                     const float* query_x, int64_t q_e, int64_t q_cloud, int64_t q_c, int64_t q_n,
                     const int64_t* query_y, float* logits, float* loss, int32_t* pred,
                     const r3dfs_episode_diag_t* diag, void* wsp, size_t ws_bytes,
                     r3dfs_stream_t stream) {
  r3dfs_episode_cfg_t qc;
  EpisodeDims d;
  R3DFS_TRY(query_dims(cfg, qc, d));
  R3DFS_TRY(check_weights(hw));
  if (!proto || !proto_count || !query_x || !logits || !wsp || E <= 0 || p_e < 0 || c_e < 0)
    return R3DFS_E_BADARG;
  if ((int64_t)E * qc.n_query > 65535) return R3DFS_E_UNSUPPORTED;
  if (((uintptr_t)proto & 15) != 0 || (p_e & 3) != 0) return R3DFS_E_ALIGN;
  if (ws_bytes < r3dfs_mpti_query_workspace(cfg, E)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = qc.n_points, in_dim = hw->in_dim;
  WsBump ws(wsp, ws_bytes);
  EpisodeWs w;
  carve_query(ws, &qc, d, E, in_dim, hw->dgcnn_k, w);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  StageRec srv{diag ? (cudaEvent_t*)diag->h_stage_events : nullptr};
  const StageRec* sr = srv.ev ? &srv : nullptr;
  if (sr) sr->mark(R3DFS_ST_BEGIN, st);
  const int64_t tq = (int64_t)E * qc.n_query * N * in_dim;
  gather_clouds_kernel<<<nblk(tq), 256, 0, st>>>(query_x, qc.n_query, in_dim, N, q_e, q_cloud, q_c,
                                                 q_n, qc.n_query, 0, w.xp, tq);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_INPUT, st);
  // features of the query clouds only (models/mpti.py:436-437), after the prototype slots
  RowMap fmap{qc.n_query, N, (int64_t)d.nn, (int64_t)d.ppad};
  R3DFS_TRY(encoder_forward(hw, w.xp, (int64_t)E * qc.n_query, N, w.enc, w.F, fmap, nullptr, st,
                            sr));
  mark_stages(sr, R3DFS_ST_MDNS, R3DFS_ST_FPS, st);
  proto_rows_kernel<<<dim3(nblk((int64_t)d.ppad * (R3DFS_FEAT_DIM / 4)), E), 256, 0, st>>>(
      proto, p_e, proto_count, c_e, d.S, d.slot, d.ppad, d.nn, w.F, w.proto_cnt);
  R3DFS_CHECK_LAUNCH();
  if (sr) sr->mark(R3DFS_ST_PROTO, st);
  return episode_query_part(&qc, d, E, w, d.nn, query_y, logits, loss, pred, diag, st, sr, false);
}

}  // extern "C"
