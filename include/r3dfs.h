/*
 * r3dfs.h — C ABI of libr3dfs.so: the B200 (sm_100a) implementation of the R3DFSSeg / MPTI
 * episode hot path.  This is the drop-in boundary: plain pointers and sizes, no torch types.
 *
 * Conventions (all entry points)
 *   - every pointer is a DEVICE pointer unless the parameter name starts with `h_`;
 *   - the caller owns every buffer (inputs, outputs, workspace); the library never allocates,
 *     frees or keeps a pointer after the call returns, and has no global mutable state;
 *   - all work is enqueued on `stream`; no call synchronises the device;
 *   - return 0 on success, a negative R3DFS_E_* for bad arguments, a positive value =
 *     (int)cudaError_t when a launch failed.  Nothing throws or aborts;
 *   - results are bit-reproducible run to run (no floating-point atomics); the one exception is
 *     r3dfs_mpti_train_backward (two gather adjoints use float atomics, stated there);
 *   - "point-major" = a cloud stored as N rows of C contiguous floats.  The reference's collate
 *     (dataloaders/loader.py:1662-1684) hands over exactly this memory behind a transposed
 *     (B, C, N) view, so strided (B, C, N) inputs are accepted everywhere a cloud comes in.
 *
 * Reference interface each entry replaces is cited as file:line of Pixie8888/R3DFSSeg.
 */
#ifndef R3DFS_H_
#define R3DFS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R3DFS_VERSION 100

#define R3DFS_OK 0
#define R3DFS_E_BADARG (-1)      /* null pointer, non-positive size                          */
#define R3DFS_E_UNSUPPORTED (-2) /* shape outside what the kernels are built for (see each)  */
#define R3DFS_E_WORKSPACE (-3)   /* workspace too small: call the matching *_workspace()     */
#define R3DFS_E_ALIGN (-4)       /* pointer not aligned as required (16 B unless noted)      */

typedef void* r3dfs_stream_t; /* cudaStream_t */

int r3dfs_version(void);
const char* r3dfs_strerror(int code);

/* ------------------------------------------------------------------------------------------
 * DGCNN pieces (reference models/dgcnn.py)
 * ---------------------------------------------------------------------------------------- */

/* knn(x, k) — models/dgcnn.py:17-23.  x: (B, C, N) fp32 with element strides (sb, sc, sn).
 * idx_out: (B, N, k) int64, the k nearest points INCLUDING the point itself, nearest first
 * (ranking key = -|xi|^2 + 2 xi.xj - |xj|^2 exactly as the reference forms it).  1 <= k <= 32. */
size_t r3dfs_knn_workspace(int64_t B, int64_t C, int64_t N, int k);
int r3dfs_knn(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
              int64_t sn, int k, int64_t* idx_out, void* ws, size_t ws_bytes,
              r3dfs_stream_t stream);

/* Same with the implementation pinned: impl 0 = default (tcgen05 kernel when C <= 64), 1 = FP32
 * CUDA-core kernel, 2 = tensor-core kernel (R3DFS_E_UNSUPPORTED when C > 64). */
int r3dfs_knn_ex(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                 int64_t sn, int k, int64_t* idx_out, int impl, void* ws, size_t ws_bytes,
                 r3dfs_stream_t stream);

/* get_edge_feature(x, K, idx) — models/dgcnn.py:26-42.  Materialises the (B, 2C, N, K)
 * contiguous edge tensor cat(x_j - x_i, x_i).  idx: (B, N, K) int64 contiguous.
 * ws (optional, may be NULL / 0): r3dfs_edge_feature_workspace() bytes of scratch; with it a
 * channel-major x is first brought into point-major form so that the neighbour gathers read whole
 * rows (a point-major x behind a transposed view — the reference's collate layout — needs none). */
size_t r3dfs_edge_feature_workspace(int64_t B, int64_t C, int64_t N);
int r3dfs_edge_feature(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                       int64_t sn, const int64_t* idx, int K, float* out, void* ws, size_t ws_bytes,
                       r3dfs_stream_t stream);

/* Weights of the episode model, eval mode.  Every BatchNorm is folded by the host into a
 * per-channel (scale, shift) pair: y = act(scale * (W x) + shift)  (conv bias folded into shift).
 *   EdgeConv block i (models/dgcnn.py:45-61,116-119):  ec_w1[i] (64, 2*Cin_i) row-major,
 *       ec_w2[i] (64, 64); LeakyReLU(0.2) after both; Cin = {in_dim, 64, 64}.
 *   point MLP (models/dgcnn.py:121-122): mlp_w[0] (512, 192), mlp_w[1] (256, 512), LeakyReLU(0.2).
 *   BaseLearner (models/mpti.py:18-40): bl_w[0] (128, 256) + ReLU, bl_w[1] (64, 128) no act.
 *   SelfAttention (models/attention.py:32-48): att_wqkv (192, 256) = [q_map; k_map; v_map].
 * Widths are the reference defaults (eval_noise.py:198-217); other widths -> R3DFS_E_UNSUPPORTED. */
typedef struct r3dfs_weights {
  int32_t in_dim;  /* 9  */
  int32_t dgcnn_k; /* 20 */
  const float* ec_w1[3];
  const float* ec_s1[3];
  const float* ec_t1[3];
  const float* ec_w2[3];
  const float* ec_s2[3];
  const float* ec_t2[3];
  const float* mlp_w[2];
  const float* mlp_s[2];
  const float* mlp_t[2];
  const float* bl_w[2];
  const float* bl_s[2];
  const float* bl_t[2];
  const float* att_wqkv;
} r3dfs_weights_t;

/* 1x1 conv + folded BatchNorm + activation on point-major rows — the building block of the
 * reference's conv1d / conv2d stacks (models/dgcnn.py:45-80) and BaseLearner (models/mpti.py:31-39):
 *   y[m][n] = act(s[n] * sum_k x[m][k] w[n][k] + t[n]),  act: 0 none, 1 ReLU, 2 LeakyReLU(0.2).
 * x: (M, K) rows ldx floats apart; w: (Nout, K) row-major; s, t: (Nout) or NULL (= 1, 0);
 * y: (M, Nout) rows ldy floats apart. */
int r3dfs_linear(const float* x, int64_t ldx, const float* w, const float* s, const float* t,
                 int act, int64_t M, int64_t K, int64_t Nout, float* y, int64_t ldy,
                 r3dfs_stream_t stream);
/* Same, with the implementation pinned: impl 0 = default (tcgen05 3xTF32 tensor-core kernel),
 * 1 = FP32 CUDA-core kernel, 2 = tensor-core kernel fed through registers, 3 = tensor-core kernel
 * fed by TMA (R3DFS_E_UNSUPPORTED unless ldx % 4 == 0, K % 4 == 0 and 16-byte aligned pointers).
 * All are exact to FP32 rounding; the switch exists for A/B measurements and the parity tests. */
int r3dfs_linear_ex(const float* x, int64_t ldx, const float* w, const float* s, const float* t,
                    int act, int64_t M, int64_t K, int64_t Nout, float* y, int64_t ldy, int impl,
                    r3dfs_stream_t stream);

/* One fused EdgeConv block, eval BN: knn -> gather -> (W1, BN, LReLU) -> (W2, BN, LReLU) -> max
 * over k (models/dgcnn.py:115-118).  The (B, 2C, N, k) edge tensor is never formed.
 * x: (B, C, N) strided; y: (B, N, 64) point-major contiguous; idx_out: optional (B, N, k) int64. */
size_t r3dfs_edgeconv_workspace(int64_t B, int64_t C, int64_t N, int k);
int r3dfs_edgeconv(const float* x, int64_t B, int64_t C, int64_t N, int64_t sb, int64_t sc,
                   int64_t sn, int k, const float* w1, const float* s1, const float* t1,
                   const float* w2, const float* s2, const float* t2, float* y, int64_t* idx_out,
                   void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* getFeatures(x) — models/mpti.py:579-589 (use_attention=True): DGCNN (models/dgcnn.py:113-127)
 * + BaseLearner + SelfAttention, concatenated [level1(64) | attention(64) | base(64)].
 * x: (B, in_dim, N) strided.  feat: (B, N, 192) point-major contiguous.
 * level2 (optional, may be NULL): (B, N, 256) point-major = DGCNN's second output. */
size_t r3dfs_features_workspace(int64_t B, int64_t N);
int r3dfs_features(const r3dfs_weights_t* h_w, const float* x, int64_t B, int64_t N, int64_t sb,
                   int64_t sc, int64_t sn, float* feat, float* level2, void* ws, size_t ws_bytes,
                   r3dfs_stream_t stream);

/* SelfAttention.forward, eval (dropout off) — models/attention.py:32-48, out_channel = 64.
 * x: (B, N, Cin) point-major; wqkv: (192, Cin); y: (B, N, 64) point-major. */
size_t r3dfs_attention_workspace(int64_t B, int64_t N);
int r3dfs_attention(const float* x, int64_t B, int64_t N, int64_t Cin, const float* wqkv, float* y,
                    void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Multi-prototype generation (reference models/mpti.py:597-634)
 * ---------------------------------------------------------------------------------------- */

/* torch_cluster.fps(feat, None, ratio=m/n, random_start=False) as called at models/mpti.py:613,
 * for `n_sets` independent sets in one launch.  Set s = rows [set_off[s], set_off[s]+set_n[s])
 * of feat (rows of D contiguous floats, D % 4 == 0, D <= 256).  Start at local index 0;
 * dist_i = min(dist_i, sum_d (x_id - x_last,d)^2) in fp32 (direct differences);
 * next = argmax (lowest index on ties).  idx_out: (n_sets, m_max) int32 local indices in
 * selection order; count per set = min(m_max, n).  n_cap = host-known upper bound of every
 * set_n[s] (sizes the per-CTA shared-memory slice; set sizes themselves stay on the device). */
int r3dfs_fps(const float* feat, int64_t D, const int32_t* set_off, const int32_t* set_n,
              int n_sets, int64_t n_cap, int m_max, int32_t* idx_out, r3dfs_stream_t stream);

/* Same contract and the same picks, with a workspace and a choice of kernel.
 *   R3DFS_FPS_STREAM  every pick re-reads the FP32 rows of the set (r3dfs_fps);
 *   R3DFS_FPS_Q8      D = 192 only: rows are kept as bytes in the shared memory of the set's
 *                     thread-block cluster, an exact integer lower bound on the distance decides
 *                     which rows can change their running minimum, and only those (3-4 % per
 *                     pick) are re-read in FP32 — same arithmetic, same sequence;
 *   R3DFS_FPS_AUTO    Q8 when D = 192 and m_max >= 16, else STREAM.
 * total_rows = rows of feat (upper bound of set_off[s] + set_n[s]). */
#define R3DFS_FPS_AUTO 0
#define R3DFS_FPS_STREAM 1
#define R3DFS_FPS_Q8 2
size_t r3dfs_fps_workspace(int64_t total_rows);
int r3dfs_fps_ex(const float* feat, int64_t D, const int32_t* set_off, const int32_t* set_n,
                 int n_sets, int64_t n_cap, int64_t total_rows, int m_max, int impl,
                 int32_t* idx_out, void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* Multi-scale degree-based noise suppression over support shots, eval only — reference
 * models/mpti.py:87-223 (Mean_pl_support_y at scales (1,1,1) and (2,2,1), the two-scale vote) with
 * grid_sampling (:316-371): per shot the bounding box of the foreground xyz (channels 0-2 of
 * support_x, mask == 1), cells with INCLUSIVE bounds on both sides in the reference's FP32 bound
 * arithmetic (start = min + i * d, end = start + d), cell seed = mean feature of its points.
 * support_x: (E, n_way*k_shot, 9, N) by strides; support_y: (E, n_way*k_shot, N) int32;
 * support_feat: (E, n_way*k_shot*N, 192) point-major rows.
 * Cells per shot: index 0 = the single cell of scale (1,1,1); 1 + 2*ix + iy = cell (ix, iy) of
 * scale (2,2,1) (the reference's x-major loop order).
 *   cell_mean  (E*n_way*k_shot, 5, 192)  mean feature per cell (0 when empty)
 *   cell_count (E*n_way*k_shot, 5)       points per cell
 *   cell_mask  (E*n_way*k_shot, N) u8, nullable: bit q set = point lies in cell q (a point on a
 *              shared face lies in both cells; the reference's `assignments` keeps the later one)
 *   degree     (E*n_way, 2, 4*k_shot), nullable: row sums of the masked cosine map (cubed at scale
 *              (1,1,1)) in seed order (shot-major, non-empty cells only), NaN padded
 *   scale_flag (E*n_way, 2, k_shot), nullable: per-scale majority vote (mean(degree > mean) > 0.5)
 *   keep       (E*n_way*k_shot) int32: 1 = shot kept (mean of the two flags >= 0.5; a way that
 *              loses every shot keeps all of them);  clean_flag: same as float, nullable. */
size_t r3dfs_mdns_workspace(int n_episodes, int n_way, int k_shot);
int r3dfs_mdns(const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c, int64_t s_n,
               const int32_t* support_y, const float* support_feat, int n_episodes, int n_way,
               int k_shot, int64_t N, float* cell_mean, int32_t* cell_count, uint8_t* cell_mask,
               float* degree, float* scale_flag, int32_t* keep, float* clean_flag, void* ws,
               size_t ws_bytes, r3dfs_stream_t stream);

/* getMutiplePrototypes(feat, k) — models/mpti.py:597-634, for `n_sets` sets in one call:
 * m = ceil(fp32(n) * fp32(k / n)) FPS seeds (k or k+1), sorted + deduplicated (`.unique()`),
 * assignment = argmin_j || f - seed_j + 1e-6 ||_2 (torch<=1.8 pairwise_distance, first minimum),
 * prototype = mean of members; n <= k -> every point is its own prototype.
 * proto_out: (n_sets, k+1, D); proto_count: (n_sets) int32; assign_out: int32 per feat row (local
 * prototype index); seed_idx_out: (n_sets, k+1) int32 sorted local seed indices (-1 padded). */
size_t r3dfs_multi_prototypes_workspace(int64_t total_rows, int n_sets, int k);
int r3dfs_multi_prototypes(const float* feat, int64_t D, const int32_t* set_off,
                           const int32_t* set_n, int n_sets, int64_t total_rows, int k,
                           float* proto_out, int32_t* proto_count, int32_t* assign_out,
                           int32_t* seed_idx_out, void* ws, size_t ws_bytes,
                           r3dfs_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Affinity graph + label propagation (reference models/mpti.py:717-776)
 * ---------------------------------------------------------------------------------------- */

/* calculateLocalConstrainedAffinity (models/mpti.py:717-756) in sparse form, `n_graphs` graphs
 * per call, each with n_max node slots of which those with valid[g][i] != 0 exist.
 *   nbr: (n_graphs, n_max, k) int32 — the k nearest OTHER valid nodes by squared L2 (the
 *        faiss.IndexFlatL2 search of k+1 with column 0 = the node itself dropped, :733-736);
 *   sim: (n_graphs, n_max, k) fp32 — exp(-0.5 (||f_i - f_j + 1e-6||_2 / sigma)^2) (:745-746).
 * node_feat: (n_graphs, n_max, D) fp32, D % 4 == 0.  Requires k < #valid nodes, k <= 1024. */
size_t r3dfs_affinity_workspace(int n_graphs, int64_t n_max, int64_t D, int k);
int r3dfs_affinity_knn(const float* node_feat, const uint8_t* valid, int n_graphs, int64_t n_max,
                       int64_t D, int k, float sigma, int32_t* nbr, float* sim, void* ws,
                       size_t ws_bytes, r3dfs_stream_t stream);

/* label_propagate (models/mpti.py:758-776):  W = A + A^T with A the k-sparse matrix (nbr, sim),
 * zero diagonal; S = D^-1/2 W D^-1/2 with D = rowsum(W) + eps; solve (I - alpha S) Z = Y by FP32
 * conjugate gradients on the sparse graph (the reference inverts the dense matrix).
 * Y, Z: (n_graphs, n_max, n_cls) fp32, n_cls <= 8.  Rows of invalid nodes are written as 0.
 * n_max <= 8192 for n_cls <= 4 and n_max <= 5376 for n_cls 5..8 (the CG solve stages every node's
 * search direction in shared memory); larger graphs return R3DFS_E_UNSUPPORTED before any launch.
 * iters_out (n_graphs) int32 / resid_out (n_graphs) fp32: optional CG diagnostics (may be NULL). */
size_t r3dfs_label_propagate_workspace(int n_graphs, int64_t n_max, int k, int n_cls);
int r3dfs_label_propagate(const int32_t* nbr, const float* sim, const uint8_t* valid, int n_graphs,
                          int64_t n_max, int k, const float* Y, int n_cls, float alpha, float tol,
                          int max_iter, float* Z, int32_t* iters_out, float* resid_out, void* ws,
                          size_t ws_bytes, r3dfs_stream_t stream);

/* The same system (I - alpha S) Z = Y solved by a DENSE FP64 Cholesky factorisation on the GPU —
 * the in-library cross-check of the conjugate-gradient solve above (BASELINE.json north_star item 4;
 * the reference inverts the dense matrix, models/mpti.py:775).  Same graph inputs; Z (G, n, n_cls)
 * fp32 (rounded from the FP64 solution); info (G) int32, nullable: 0, or 1 + the first pivot that
 * was not positive.  n <= 8192; needs 8 n^2 bytes per graph: not meant for the timed path. */
size_t r3dfs_lp_cholesky_workspace(int n_graphs, int64_t n_max, int k, int n_cls);
int r3dfs_lp_cholesky(const int32_t* nbr, const float* sim, const uint8_t* valid, int n_graphs,
                      int64_t n_max, int k, const float* Y, int n_cls, float alpha, float* Z,
                      int32_t* info, void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Whole episode(s): MPTI_SelfAtten.forward, eval path (reference models/mpti.py:414-577)
 * ---------------------------------------------------------------------------------------- */

typedef struct r3dfs_episode_cfg {
  int32_t n_way;
  int32_t k_shot;
  int32_t n_query;         /* number of query clouds = n_way * n_queries                        */
  int32_t n_points;        /* 2048; multiple of 64                                               */
  int32_t n_subprototypes; /* 100  (<= 127)                                                     */
  int32_t k_connect;       /* 200                                                               */
  float sigma;             /* 1.0                                                               */
  float alpha;             /* 0.99 (models/mpti.py:758)                                         */
  int32_t mdns;            /* 1 = multi-scale degree-based noise suppression (forward eval=True) */
  int32_t cg_max_iter;     /* e.g. 200                                                          */
  float cg_tol;            /* relative residual, e.g. 1e-6                                      */
} r3dfs_episode_cfg_t;

/* Stage boundaries of r3dfs_mpti_forward, for profiling: when diag.stage_events is given, event i
 * is recorded on the stream when stage i has been enqueued completely (event 0 before any work),
 * so elapsed(event[i-1], event[i]) is the device time of stage i. */
enum r3dfs_stage {
  R3DFS_ST_BEGIN = 0,
  R3DFS_ST_INPUT,   /* clouds -> point-major                                        */
  R3DFS_ST_KNN0, R3DFS_ST_PQ0, R3DFS_ST_EDGE0, /* EdgeConv 1: kNN, per-point W1, gather+W2+max */
  R3DFS_ST_KNN1, R3DFS_ST_PQ1, R3DFS_ST_EDGE1,
  R3DFS_ST_KNN2, R3DFS_ST_PQ2, R3DFS_ST_EDGE2,
  R3DFS_ST_MLP,     /* point MLP 192 -> 512 -> 256                                  */
  R3DFS_ST_BASE,    /* BaseLearner                                                  */
  R3DFS_ST_QKV,     /* q/k/v projections                                            */
  R3DFS_ST_ATT,     /* attention                                                    */
  R3DFS_ST_MDNS,    /* multi-scale degree-based noise suppression                   */
  R3DFS_ST_SETS,    /* fg/bg set compaction                                         */
  R3DFS_ST_FPS,     /* farthest point sampling                                      */
  R3DFS_ST_PROTO,   /* seed sort/unique, assignment, cluster means                  */
  R3DFS_ST_DIST,    /* node distance matrix                                         */
  R3DFS_ST_SELECT,  /* k_connect nearest per node                                   */
  R3DFS_ST_SIM,     /* Gaussian similarities                                        */
  R3DFS_ST_SYM,     /* in-edge lists, degrees, normalisation                        */
  R3DFS_ST_CG,      /* conjugate-gradient solve                                     */
  R3DFS_ST_HEAD,    /* logits / loss / prediction                                   */
  R3DFS_N_STAGES
};

/* Device-side per-episode diagnostics (all optional: pass NULL to skip). */
typedef struct r3dfs_episode_diag {
  int32_t* proto_count; /* (E, n_way + 1): prototypes of [bg, way 0, ...]                      */
  float* clean_flag;    /* (E, n_way, k_shot): MDNS clean flag (1 = kept), models/mpti.py:201-221;
                           written only when cfg.mdns = 1                                       */
  int32_t* cg_iters;    /* (E)                                                                  */
  float* cg_resid;      /* (E)                                                                  */
  void** h_stage_events; /* HOST array of R3DFS_N_STAGES cudaEvent_t owned by the caller, or NULL */
} r3dfs_episode_diag_t;

/* Number of kernels this thread has launched through the library so far (diagnostic counter). */
long long r3dfs_launch_count(void);

/* Episode envelope (every episode entry point; the workspace queries return 0 outside it and the
 * calls R3DFS_E_UNSUPPORTED, before any launch): 1 <= n_way <= 7, 1 <= k_shot <= 32,
 * n_points >= 64, 1 <= n_subprototypes <= 127, 1 <= k_connect <= 1024, k_connect < n_query *
 * n_points, and graph nodes = roundup64((n_way + 1) * (n_subprototypes + 1)) + n_query * n_points
 * <= 8192, or <= 5376 when n_way >= 4 (the label-propagation limit at n_way + 1 classes). */
size_t r3dfs_mpti_workspace(const r3dfs_episode_cfg_t* h_cfg, int n_episodes);

/* E = n_episodes independent episodes in one call (reference: one per forward call).
 *   support_x: (E, n_way, k_shot, in_dim, N) with element strides (s_e, s_cloud, s_c, s_n) —
 *              clouds of an episode are n_way*k_shot consecutive `s_cloud` steps;
 *   support_y: (E, n_way, k_shot, N) int32 contiguous, non-zero = foreground;
 *   query_x:   (E, n_query, in_dim, N) strides (q_e, q_cloud, q_c, q_n);
 *   query_y:   (E, n_query, N) int64 contiguous in [0, n_way] (may be NULL -> loss not computed);
 *   logits:    (E, n_query, N, n_way+1) fp32 — Z rows of the query nodes (the reference returns
 *              this buffer viewed as (n_query, n_way+1, N), models/mpti.py:558-559);
 *   loss:      (E) fp32 cross-entropy of logits vs query_y (models/mpti.py:571);
 *   pred:      (E, n_query, N) int32 argmax labels (models/mpti_learner.py:98); may be NULL. */
int r3dfs_mpti_forward(const r3dfs_episode_cfg_t* h_cfg, const r3dfs_weights_t* h_w,
                       int n_episodes, const float* support_x, int64_t s_e, int64_t s_cloud,
                       int64_t s_c, int64_t s_n, const int32_t* support_y, const float* query_x,
                       int64_t q_e, int64_t q_cloud, int64_t q_c, int64_t q_n,
                       const int64_t* query_y, float* logits, float* loss, int32_t* pred,
                       const r3dfs_episode_diag_t* h_diag, void* ws, size_t ws_bytes,
                       r3dfs_stream_t stream);

/* The same episode(s) from precomputed features: everything after getFeatures
 * (models/mpti.py:440-571).  support_feat: (E, n_way*k_shot*N, 192) point-major rows in
 * (way, shot, point) order; query_feat: (E, n_query*N, 192).  support_x is still needed for the
 * xyz channels the noise suppression grids over (models/mpti.py:116).  Workspace and outputs as
 * r3dfs_mpti_forward.  Used by the stage-wise parity tests and by callers that cache features. */
int r3dfs_mpti_forward_features(const r3dfs_episode_cfg_t* h_cfg, int n_episodes,
                                const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                                int64_t s_n, const int32_t* support_y, const float* support_feat,
                                const float* query_feat, const int64_t* query_y, float* logits,
                                float* loss, int32_t* pred, const r3dfs_episode_diag_t* h_diag,
                                void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* One support set, many query clouds: r3dfs_mpti_forward cut into its two halves, so that the
 * part of an episode that depends on the support set alone runs once per set.  Chaining the two
 * calls on the same episodes returns what r3dfs_mpti_forward returns, bit for bit.  Both accept
 * the envelope of r3dfs_mpti_forward and return its error codes.
 *
 * Support half of MPTI_SelfAtten.forward, eval (models/mpti.py:433-435, 440-493): getFeatures of
 * the n_sets * n_way * k_shot support clouds only, MDNS when cfg->mdns, fg/bg sets, FPS seeds,
 * assignment, prototype means.  support_x / support_y as r3dfs_mpti_forward with n_sets sets.
 *   proto:       (n_sets, n_way+1, n_subprototypes+1, 192) fp32, classes [bg, way 0, ...];
 *                rows >= proto_count are zero
 *   proto_count: (n_sets, n_way+1) int32
 * h_diag: clean_flag and stage events as in r3dfs_mpti_forward (the graph stages are recorded
 * at the end, with no work between them); the other fields are ignored. */
size_t r3dfs_mpti_support_workspace(const r3dfs_episode_cfg_t* h_cfg, int n_sets);
int r3dfs_mpti_support(const r3dfs_episode_cfg_t* h_cfg, const r3dfs_weights_t* h_w, int n_sets,
                       const float* support_x, int64_t s_e, int64_t s_cloud, int64_t s_c,
                       int64_t s_n, const int32_t* support_y, float* proto, int32_t* proto_count,
                       const r3dfs_episode_diag_t* h_diag, void* ws, size_t ws_bytes,
                       r3dfs_stream_t stream);

/* Query half (models/mpti.py:436-437, 495-571): getFeatures of the E * n_query query clouds only,
 * then graph, label propagation and head against given prototypes (layout of r3dfs_mpti_support).
 * p_e / c_e = element stride between episodes in proto / proto_count; 0 = every episode uses the
 * same support set (no copy).  proto must be 16-byte aligned and p_e a multiple of 4.  Counts are
 * clamped to [0, n_subprototypes+1]; prototype rows at or past a set's count are read as zero.
 * Uses n_way, n_query, n_points, n_subprototypes, k_connect, sigma, alpha, cg_* of h_cfg; k_shot
 * and mdns are ignored, and the workspace does not depend on k_shot.  query_x, query_y, outputs
 * and h_diag as r3dfs_mpti_forward (proto_count: the clamped counts; clean_flag is not written;
 * the stages mdns, sets and fps are recorded with no work between them, proto = the copy of the
 * given prototypes into the graph). */
size_t r3dfs_mpti_query_workspace(const r3dfs_episode_cfg_t* h_cfg, int n_episodes);
int r3dfs_mpti_query(const r3dfs_episode_cfg_t* h_cfg, const r3dfs_weights_t* h_w, int n_episodes,
                     const float* proto, int64_t p_e, const int32_t* proto_count, int64_t c_e,
                     const float* query_x, int64_t q_e, int64_t q_cloud, int64_t q_c, int64_t q_n,
                     const int64_t* query_y, float* logits, float* loss, int32_t* pred,
                     const r3dfs_episode_diag_t* h_diag, void* ws, size_t ws_bytes,
                     r3dfs_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Segmenting a whole scan against one support set
 * ---------------------------------------------------------------------------------------- */

/* A scan of M points is cut into overlapping xy blocks, every block into chunks of N = n_points
 * points laid out as the reference's loader lays out a block (dataloaders/loader.py:201-219); the
 * chunks are segmented as 1-query episodes (r3dfs_mpti_query, n_query = 1, p_e = 0) and the chunk
 * logits are merged back onto the points.  Three calls share one workspace, which must not be
 * touched between them: plan -> chunks -> (query) -> merge.
 *
 *   points: (M, 6) fp32 by element strides (s_m, s_c): x y z in metres (any origin), r g b in
 *           0..255 (the S3DIS / ScanNet .npy convention).
 * Every operation below is an fp32 operation rounded to nearest, written out (no contraction).
 *
 * Grid.  Blocks are xy columns over the full height.  r = overlap (1..4), stride = block_size / r,
 *   x0 = min x, ext_x = max x - x0; n_cells_x = max(1, floor(ext_x / stride + 0.5)) (the last cell
 *   absorbs a remainder under half a stride); a point's cell u = min(floor((x - x0) / stride),
 *   n_cells_x - 1); n_bx = max(1, n_cells_x - r + 1); the point lies in every block
 *   ix in [max(0, u - r + 1), min(u, n_bx - 1)], the same in y; block id b = ix * n_by + iy.
 *   Every point lies in 1 to r^2 blocks.
 * Chunks.  Empty blocks make none; a block of n_b members makes C_b = ceil(n_b / N).  Members are
 *   ranked by k(i) = lowbias32(i ^ lowbias32(seed)) (i = point index; lowbias32(x): x ^= x >> 16;
 *   x *= 0x7feb352d; x ^= x >> 15; x *= 0x846ca68b; x ^= x >> 16 on uint32, a bijection: no ties).
 *   Rank rho goes to chunk rho mod C_b, slot rho div C_b, so every chunk is a uniform sample of the
 *   block.  Chunk j has count_j = ceil((n_b - j) / C_b) members; slot s >= count_j repeats slot
 *   s mod count_j (the loader's sampling with replacement of a small block).  Chunks are numbered
 *   by ascending block id, then j.
 * Chunk cloud (N, 9) point-major, over the chunk's own points: m = min xyz, xyz' = xyz - m,
 *   e = max xyz', XYZ = e > 0 ? xyz' / e : 0 per axis (the reference divides 0 by 0 on a flat axis),
 *   rgb' = rgb / 255; channels xyz' | rgb' | XYZ.
 * Merge.  A point's logits = the sum, in ascending block id, of the logits row at its own slot of
 *   each block that holds it (repeats excluded), sequential fp32 adds from 0, divided once by the
 *   number of contributions; pred = argmax (first maximum, as the episode head); coverage = the
 *   number of contributions (1..r^2).
 *
 * Limits: r^2 * M < 2^31, 64 <= N <= 65536 (R3DFS_E_UNSUPPORTED).  The chunks go through
 * r3dfs_mpti_query in batches of at most 65535 (its E * n_query limit). */
size_t r3dfs_scene_workspace(int64_t M, int overlap); /* 0 outside the limits; host only */

/* Builds the grid, the memberships and the chunk layout in the workspace and writes the number of
 * chunks to the DEVICE int64 *n_chunks: -1 when an x or y coordinate is not finite or the grid has
 * 2^31 blocks or more.  block_size > 0 and finite.  Reading n_chunks back is the one host
 * synchronisation a scene needs. */
int r3dfs_scene_plan(const float* points, int64_t M, int64_t s_m, int64_t s_c, float block_size,
                     int overlap, uint32_t seed, int n_points, int64_t* n_chunks, void* ws,
                     size_t ws_bytes, r3dfs_stream_t stream);

/* chunk_x: (n_chunks, N, 9) point-major chunk clouds; chunk_src: (n_chunks, N) int32, the point of
 * every slot.  n_chunks (host) = the value plan wrote; chunks past it are written as 0 / -1. */
int r3dfs_scene_chunks(const float* points, int64_t M, int64_t s_m, int64_t s_c, int overlap,
                       int n_points, int64_t n_chunks, float* chunk_x, int32_t* chunk_src,
                       void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* logits: (n_chunks, N, n_cls) fp32 (r3dfs_mpti_query's logits of the chunks in order), n_cls <= 8.
 * point_logits: (M, n_cls) fp32; point_pred (M) int32 and coverage (M) int32 may be NULL. */
int r3dfs_scene_merge(const float* logits, int64_t M, int overlap, int n_points, int64_t n_chunks,
                      int n_cls, float* point_logits, int32_t* point_pred, int32_t* coverage,
                      void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* Support shots from a labelled scan (the reference's class2scans index, dataloaders/s3dis.py /
 * scannet.py, and sample_pointcloud(..., support=True), dataloaders/loader.py:201-219), on a scan
 * planned by r3dfs_scene_plan with the same points, block_size, overlap, seed and N = n_points.
 *   labels: (M) int32 class of every point; h_classes: HOST array of n_way distinct class ids.
 * Counts.  For every non-empty block b with n_b members, count_w(b) = members i with
 *   labels[i] == classes[w].
 * Eligibility.  b is eligible for way w iff count_w(b) > max(floor(n_b * min_ratio), min_points),
 *   the product in fp64 (as Python's int(n_b * 0.05)); the reference uses min_points = 100,
 *   min_ratio = 0.05.  n_eligible[w] = the number of eligible blocks.
 * Choice.  Way w ranks its eligible blocks by lowbias32(b ^ lowbias32(lowbias32(seed) + w + 1))
 *   (uint32, wrapping): a bijection of the block id, different for every way.  Its shots are the
 *   k_shot eligible blocks with the smallest keys, in ascending key order; a block may serve
 *   several ways.  shot_block (n_way, k_shot) int32 = the block id of every shot.
 * Shot cloud.  The block's members in the plan's rank order k(i); slot s holds rank
 *   s mod min(n_b, N): for n_b >= N the N lowest-ranked members, each once (the reference's
 *   sampling without replacement), for a smaller block its members repeated.  For n_b <= N it is
 *   the block's single chunk of r3dfs_scene_chunks.  Normalised as a chunk cloud.
 *   support_x: (n_way, k_shot, N, 9) point-major; support_src (n_way, k_shot, N) int32 = the point
 *   of every slot; support_y (n_way, k_shot, N) int32 = labels[src] == classes[w].
 * Missing shots (n_eligible[w] < k_shot) are a zero cloud with src -1, block -1 and mask 0.  When
 *   the plan reported a grid error (n_chunks = -1), every n_eligible is -1.
 * The plan workspace is only read: chunks and merge on it return what they returned before.
 * Deterministic, no atomics, no host synchronisation.  ws: r3dfs_scene_support_workspace bytes
 * (under 1 MB, independent of M).  1 <= n_way <= 7 and 1 <= k_shot <= 32 (else
 * R3DFS_E_UNSUPPORTED); duplicate classes, min_points < 0, or min_ratio outside [0, 1] or not
 * finite give R3DFS_E_BADARG.  Every check happens before anything is launched. */
size_t r3dfs_scene_support_workspace(int n_way, int k_shot); /* 0 outside the limits; host only */
int r3dfs_scene_support(const float* points, int64_t M, int64_t s_m, int64_t s_c,
                        const int32_t* labels, const int32_t* h_classes, int n_way, int k_shot,
                        int min_points, double min_ratio, uint32_t seed, int overlap, int n_points,
                        float* support_x, int32_t* support_y, int32_t* support_src,
                        int32_t* shot_block, int32_t* n_eligible, const void* plan_ws,
                        size_t plan_ws_bytes, void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* Few-shot episodes from labelled scans (the reference's NoiseInMetaTest.generate_one_episode,
 * dataloaders/loader.py:648-890, over its class2scans lists).
 *
 * Dataset index.  A dataset is a list of labelled scans concatenated into one points and one labels
 * array; scan i starts at point point_base_i.  Every scan is planned by r3dfs_scene_plan on its own
 * slice (one block_size, overlap and seed for all) and appended by r3dfs_scene_index, which reads
 * the plan workspace (the workspace may be freed afterwards).  Global blocks are numbered in scan
 * order, then by ascending block id within the scan:
 *   block_off (n_blocks + 1) int64: first membership of each block in `member`;
 *   block_scan, block_id (n_blocks) int32: its scan and its block id in that scan;
 *   member (n_members) int32: the GLOBAL point of every member, in the plan's rank order k(i);
 *   count (n_blocks, n_cls) int32: members whose label is h_classes[k] (1..64 distinct ids; other
 *     labels count for no class).
 * r3dfs_scene_index appends one scan at (n_blocks, n_members), the sizes so far, and writes the
 * scan's block and membership counts to HOST h_sizes[0..1] (it synchronises the stream once).  When
 * the arrays' capacities (block_cap blocks, member_cap members) are too small it returns
 * R3DFS_E_WORKSPACE after writing h_sizes, with nothing written: grow them and call again.  A plan
 * that found no valid grid gives h_sizes = -1 and R3DFS_E_BADARG.  Limits: the plan's, point_base + M
 * < 2^31 and total memberships < 2^31 (R3DFS_E_UNSUPPORTED).
 * r3dfs_scene_index_classes, once after the last scan: block b is eligible for class k iff
 *   count(b, k) > max(floor(n_b * min_ratio), min_points), the product in fp64 (the rule of
 *   r3dfs_scene_support).  elig_off (n_cls + 1) and elig_block (room for n_blocks * n_cls) hold
 *   every class's eligible global blocks in ascending order (the reference's class2scans);
 *   h_elig_off (HOST, n_cls + 1) receives a copy (one stream synchronisation).  ws:
 *   r3dfs_scene_index_workspace bytes; n_blocks * n_cls < 2^31 - 1.
 *
 * Episodes.  r3dfs_scene_episodes builds E episodes of n_way ways, k_shot shots and n_queries query
 * blocks per way.  Host inputs: h_elig_off (from r3dfs_scene_index_classes), h_classes (the index's
 * n_cls ids), h_way_class (E, n_way) class ids, h_n_noise (E) noisy shots per way, noise_type
 * (0 none, 1 ood, 2 sym, 3 pair) and h_pair (n_cls) = pair[h_classes[k]] as class ids (pair only;
 * may map a class to itself).  Episode e has index g = first + e * step (uint32).  Every key is
 * integer hashing with lowbias32 (see "Segmenting a whole scan"), H(a, b) = lowbias32(a ^
 * lowbias32(b)) on uint32:
 *   K_e = H(lowbias32(seed), g);  way w: K_w = H(K_e, w + 1);  k_clean = k_shot - n_noise.
 *   Clean shots and queries.  The way's class list is ranked by lowbias32(b ^ K_w) over the global
 *     block index b (a bijection: no ties); the first k_clean blocks are the clean shots, the next
 *     n_queries the way's query blocks (distinct from its shots; blocks may repeat across ways).
 *   Noise range R.  ood: the index's classes with at least one eligible block that are not among
 *     the episode's ways, in index order; sym: the other ways' classes in way order; pair:
 *     [pair[c]].  Noisy shot j (0 <= j < n_noise) takes class R[(H(K_w, 64 + j) * |R|) >> 32]
 *     (64-bit product), except when k_clean - 1 == 1 for ood and sym, the reference's single-use
 *     rule: then it takes R[pi[min(j, |R| - 1)]], where pi lists 0..|R|-1 by ascending
 *     lowbias32(r ^ H(K_w, 33)).  Its block is the smallest lowbias32(b ^ H(K_w, 128 + j)) of
 *     that class's eligible list.
 *   Shuffle.  Shot t of the way (t < k_clean: clean shot t; else noisy shot t - k_clean) goes to
 *     slot rank_t, its rank among t = 0..k_shot-1 under lowbias32(t ^ H(K_w, 34)).
 *   Clouds.  Slot s of a block's cloud holds member rank s mod min(n_b, N), normalised as a chunk
 *     cloud (the shot clouds of r3dfs_scene_support).
 * Outputs (device): support_x (E, n_way, k_shot, N, 9) and query_x (E, n_way * n_queries, N, 9)
 *   point-major, query clouds way-major; support_y (E, n_way, k_shot, N) int32 = label == the
 *   shot's class; gt_support_y = support_y on clean shots, 0 on noisy ones; support_flag
 *   (E, n_way, k_shot) int32 class id of every shot; query_y (E, n_way * n_queries, N) int64 = w + 1
 *   where label == class of way w, else 0; shot_block (E, n_way, k_shot), query_block
 *   (E, n_way * n_queries) int32 global blocks; support_src / query_src int32 global point of
 *   every slot.  Every output is a function of (seed, g) and the index alone.
 * Deterministic, no atomics, no host synchronisation; the host arrays are copied into the
 * workspace (r3dfs_scene_episodes_workspace bytes).  Limits (R3DFS_E_UNSUPPORTED): 1 <= n_way <= 7,
 * 1 <= k_shot <= 32, n_queries >= 1, k_clean + n_queries <= 32, E * n_way * n_queries <= 65535,
 * 1 <= n_cls <= 64, 64 <= N <= 65536.  R3DFS_E_BADARG: an unknown or repeated class, a way class
 * with fewer than k_clean + n_queries eligible blocks, n_noise outside 0..k_shot or non-zero
 * without noise, an empty noise range (or a pair class without eligible blocks) where n_noise > 0,
 * first < 0, step < 1 or g past 2^32 - 1.  Every check happens before anything is launched. */
int r3dfs_scene_index(const int32_t* labels, int64_t M, int overlap, const int32_t* h_classes,
                      int n_cls, int32_t scan, int64_t point_base, int64_t n_blocks,
                      int64_t n_members, int64_t block_cap, int64_t member_cap, int64_t* block_off,
                      int32_t* block_scan, int32_t* block_id, int32_t* member, int32_t* count,
                      int64_t* h_sizes, const void* plan_ws, size_t plan_ws_bytes,
                      r3dfs_stream_t stream);
size_t r3dfs_scene_index_workspace(int64_t n_blocks, int n_cls); /* 0 outside the limits */
int r3dfs_scene_index_classes(const int64_t* block_off, const int32_t* count, int64_t n_blocks,
                              int n_cls, int min_points, double min_ratio, int32_t* elig_off,
                              int32_t* elig_block, int32_t* h_elig_off, void* ws, size_t ws_bytes,
                              r3dfs_stream_t stream);
size_t r3dfs_scene_episodes_workspace(int n_episodes, int n_way, int k_shot, int n_queries,
                                      int n_cls); /* 0 outside the limits; host only */
int r3dfs_scene_episodes(const float* points, int64_t s_m, int64_t s_c, const int32_t* labels,
                         const int64_t* block_off, const int32_t* member, const int32_t* elig_off,
                         const int32_t* elig_block, const int32_t* h_elig_off,
                         const int32_t* h_classes, int n_cls, const int32_t* h_way_class,
                         const int32_t* h_n_noise, int noise_type, const int32_t* h_pair,
                         int n_episodes, int n_way, int k_shot, int n_queries, int n_points,
                         uint32_t seed, int64_t first, int64_t step, float* support_x,
                         int32_t* support_y, int32_t* gt_support_y, int32_t* support_flag,
                         float* query_x, int64_t* query_y, int32_t* shot_block,
                         int32_t* query_block, int32_t* support_src, int32_t* query_src, void* ws,
                         size_t ws_bytes, r3dfs_stream_t stream);

/* ProtoNet + MDNS (reference models/protonet.py:357-945 ProtoNet_Contrast.forward, train=False):
 * same encoder and noise suppression as MPTI, then masked average pooling of the support
 * features (:878-890), one prototype per way from the kept shots + one background prototype
 * (:892-915) and the similarity of every query point to every prototype (:917-940).
 * dist_method 0 = 'cosine' (x 10), the only one that runs in the reference: 'euclidean' reduces
 * over the point axis and fails in the loss, the scripts' default 'gaussian' raises
 * NotImplementedError; anything else returns R3DFS_E_UNSUPPORTED.  Arguments, outputs and workspace
 * (r3dfs_mpti_workspace) as r3dfs_mpti_forward; cfg->mdns = 0 keeps every shot; clean_flag:
 * optional (E, n_way, k_shot) fp32 output of the noise suppression. */
int r3dfs_protonet_forward(const r3dfs_episode_cfg_t* h_cfg, const r3dfs_weights_t* h_w,
                           int n_episodes, const float* support_x, int64_t s_e, int64_t s_cloud,
                           int64_t s_c, int64_t s_n, const int32_t* support_y, const float* query_x,
                           int64_t q_e, int64_t q_cloud, int64_t q_c, int64_t q_n,
                           const int64_t* query_y, int dist_method, float* logits, float* loss,
                           int32_t* pred, float* clean_flag, void* ws, size_t ws_bytes,
                           r3dfs_stream_t stream);

/* evaluate_metric counters (reference eval_noise.py:35-62): for every query point, map the
 * episode-local label to its slot in the test-class list and accumulate gt / predicted /
 * true-positive counts.  class_slot: (E, n_way) int32 = test_classes.index(sampled_class) + 1.
 * counters: (3, n_slots) int64, accumulated in place (zero them before the first call); they
 * are what NCCL sum-all-reduces across ranks. */
int r3dfs_confusion_accumulate(const int32_t* pred, const int64_t* gt, const int32_t* class_slot,
                               int n_episodes, int n_way, int64_t pts_per_episode, int n_slots,
                               int64_t* counters, r3dfs_stream_t stream);


/* ------------------------------------------------------------------------------------------
 * Meta-training step (reference models/mpti_learner.py:50-79 around
 * MPTI_SelfAtten.forward(train=True), models/mpti.py:414-577, loss = lp + 0.1 * way-contrast)
 * ---------------------------------------------------------------------------------------- */

/* Trainable tensors, in the order of the reference's named_parameters(); every tensor keeps the
 * reference's shape, flattened row-major, and all of them live back to back in ONE flat fp32
 * buffer (376 896 floats at in_dim = 9) — the same buffer is the gradient bucket NCCL all-reduces
 * and the range the fused Adam kernel walks.  r3dfs_train_param_layout() gives the offsets. */
enum r3dfs_param {
  R3DFS_P_EC0_W1 = 0, /* encoder.edge_convs.0.layer.0.weight (64, 2*in_dim)                     */
  R3DFS_P_EC0_G1,     /* .layer.1.weight   (BatchNorm gamma)                                    */
  R3DFS_P_EC0_B1,     /* .layer.1.bias     (BatchNorm beta)                                     */
  R3DFS_P_EC0_W2,     /* .layer.3.weight (64, 64)                                               */
  R3DFS_P_EC0_G2,     /* .layer.4.weight                                                        */
  R3DFS_P_EC0_B2,     /* .layer.4.bias                                                          */
  /* edge_convs.1 and .2 follow with the same six entries each (W1 is (64, 128))               */
  R3DFS_P_MLP0_W = 18, /* encoder.conv.layer.0.weight (512, 192)                                */
  R3DFS_P_MLP0_G, R3DFS_P_MLP0_B,
  R3DFS_P_MLP1_W,      /* encoder.conv.layer.3.weight (256, 512)                                */
  R3DFS_P_MLP1_G, R3DFS_P_MLP1_B,
  R3DFS_P_BL0_W,       /* base_learner.convs.0.0.weight (128, 256)                              */
  R3DFS_P_BL0_BIAS, R3DFS_P_BL0_G, R3DFS_P_BL0_B,
  R3DFS_P_BL1_W,       /* base_learner.convs.1.0.weight (64, 128)                               */
  R3DFS_P_BL1_BIAS, R3DFS_P_BL1_G, R3DFS_P_BL1_B,
  R3DFS_P_ATT_Q,       /* att_learner.{q,k,v}_map.weight (64, 256) each, contiguous = (192, 256) */
  R3DFS_P_ATT_K, R3DFS_P_ATT_V,
  R3DFS_P_PROJ_W,      /* proj.weight (128, 192)                                                */
  R3DFS_P_PROJ_B,      /* proj.bias (128)                                                       */
  R3DFS_N_PARAMS
};
/* offsets[i] = first float of tensor i, offsets[R3DFS_N_PARAMS] = total; returns the index of
 * the first non-encoder tensor's offset (the learning-rate group boundary, mpti_learner.py:27). */
int64_t r3dfs_train_param_layout(int in_dim, int64_t* offsets);

/* BatchNorm layers in forward order: edge_convs.i.layer.{1,4} (i = 0..2), conv.layer.{1,4},
 * base_learner.convs.{0,1}.1.  Running statistics live in one flat buffer: for layer b with C_b
 * channels, floats [2*off_b, 2*off_b + C_b) = running_mean, the next C_b = running_var;
 * offsets[R3DFS_N_BN] = total channels (1344). */
#define R3DFS_N_BN 10
void r3dfs_train_bn_layout(int64_t* offsets);

/* Forward of one training episode.  BatchNorm uses batch statistics, separately over the support
 * clouds and over the query clouds (two getFeatures calls, models/mpti.py:434-436); bn_running
 * (may be NULL) is updated in place with momentum 0.1 for both.  Attention dropout
 * (models/attention.py:45): keep_support (n_way*k_shot, N, N) / keep_query (n_query, N, N) are
 * 0/1 keep masks (r3dfs_dropout_mask), NULL = no dropout; kept entries are scaled 1/(1-dropout_p).
 * support_flag: (n_way, k_shot) int32 absolute class of each shot (way-contrast labels).
 * losses[0] = label-propagation cross-entropy, losses[1] = way-contrast loss (fps_k = 4, temp 0.1).
 * cfg->mdns is ignored (noise suppression is eval-only, models/mpti.py:440).  The workspace keeps
 * every activation the backward needs: pass the SAME, untouched workspace to
 * r3dfs_mpti_train_backward. */
size_t r3dfs_mpti_train_workspace(const r3dfs_episode_cfg_t* h_cfg, int in_dim, int dgcnn_k);
int r3dfs_mpti_train_forward(const r3dfs_episode_cfg_t* h_cfg, int in_dim, int dgcnn_k,
                             const float* params, float* bn_running, const float* support_x,
                             int64_t s_cloud, int64_t s_c, int64_t s_n, const int32_t* support_y,
                             const int32_t* support_flag, const float* query_x, int64_t q_cloud,
                             int64_t q_c, int64_t q_n, const int64_t* query_y, float dropout_p,
                             const uint8_t* keep_support, const uint8_t* keep_query, float* logits,
                             float* losses, int32_t* cg_iters, void* ws, size_t ws_bytes,
                             r3dfs_stream_t stream);

/* Backward of w_lp * losses[0] + w_contrast * losses[1] wrt every trainable tensor: grads (flat,
 * same layout as params) is overwritten.  Gradients flow through the prototype means, the Gaussian
 * affinities, the degree normalisation and the label-propagation solve (adjoint by the same CG),
 * not through kNN / FPS / argmin indices — as under autograd in the reference.  The EdgeConv and
 * affinity gather adjoints use float atomics: results are reproducible to rounding, not bitwise. */
int r3dfs_mpti_train_backward(const r3dfs_episode_cfg_t* h_cfg, int in_dim, int dgcnn_k,
                              const float* params, const int32_t* support_y,
                              const int32_t* support_flag, const int64_t* query_y, float dropout_p,
                              const uint8_t* keep_support, const uint8_t* keep_query, float w_lp,
                              float w_contrast, float* grads, void* ws, size_t ws_bytes,
                              r3dfs_stream_t stream);

/* The reference's logging-only diagnostics of a training forward (models/mpti.py:514-552), from
 * the workspace of the last r3dfs_mpti_train_forward: ratios[0] = clean_ratio_LP_avg (foreground
 * support points whose prototype's propagated label agrees with the ground-truth mask, averaged
 * over ways), ratios[1] = clean_ratio_original_avg.  gt_support_y: (n_way, k_shot, N) int32. */
int r3dfs_mpti_train_clean_ratio(const r3dfs_episode_cfg_t* h_cfg, int in_dim, int dgcnn_k,
                                 const int32_t* support_y, const int32_t* gt_support_y,
                                 float* ratios, void* ws, size_t ws_bytes, r3dfs_stream_t stream);

/* Diagnostics for the parity tests: copies the discrete decisions of the last
 * r3dfs_mpti_train_forward out of its workspace, so that a reference implementation can be run
 * with the same neighbour lists / cluster assignments (they carry no gradient, but FP32 ties in
 * them make an end-to-end comparison chaotic).  Every pointer is a device buffer or NULL (skipped):
 *   knn_support[i] (n_way*k_shot*N*dgcnn_k) / knn_query[i] (n_query*N*dgcnn_k): EdgeConv i neighbours,
 *       cloud-local indices;
 *   set_off / set_n / proto_cnt (n_way+1): rows of the compacted support buffer holding the
 *       background set (0) and each way's foreground set (1+w), and their prototype counts;
 *   assign (n_way*k_shot*N): prototype of every compacted row (local index within its set);
 *   cloud_fg_off / fg_cnt / cproto_cnt (n_way*k_shot): each shot's foreground rows and the number
 *       of way-contrast prototypes;  cassign: as assign, for the way-contrast prototypes;
 *   nbr (nn * k_connect), valid (nn): affinity neighbours in node-slot numbering, with
 *       nn = roundup64((n_way+1)*(n_subprototypes+1)) + n_query*N; prototype p of set s is node
 *       s*(n_subprototypes+1) + p, query point q is node nn - n_query*N + q. */
typedef struct r3dfs_train_export {
  int32_t* knn_support[3];
  int32_t* knn_query[3];
  int32_t* set_off;
  int32_t* set_n;
  int32_t* proto_cnt;
  int32_t* assign;
  int32_t* cloud_fg_off;
  int32_t* fg_cnt;
  int32_t* cproto_cnt;
  int32_t* cassign;
  int32_t* nbr;
  uint8_t* valid;
} r3dfs_train_export_t;
int r3dfs_mpti_train_export(const r3dfs_episode_cfg_t* h_cfg, int in_dim, int dgcnn_k,
                            const r3dfs_train_export_t* h_out, void* ws, size_t ws_bytes,
                            r3dfs_stream_t stream);

/* torch.optim.Adam step (defaults of models/mpti_learner.py:26-32) over the flat buffers:
 * floats [0, n_group0) use lr0 (encoder, 1e-4), the rest lr1 (args.lr); step = 1, 2, ...;
 * grad_scale multiplies the gradient first (1 / world_size after a sum all-reduce). */
int r3dfs_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                    int64_t n_group0, float lr0, float lr1, float beta1, float beta2, float eps,
                    int64_t step, float grad_scale, r3dfs_stream_t stream);

/* Counter-based dropout keep mask: mask[i] = 1 iff u(seed, i) >= p. */
int r3dfs_dropout_mask(uint64_t seed, int64_t n, float p, uint8_t* mask, r3dfs_stream_t stream);

/* C (M, N; rows ldc apart) = alpha * A * B + beta * C in FP32 with element strides
 * A(m, k) = A[m*sAm + k*sAk], B(k, n) = B[k*sBk + n*sBn] — the gradient GEMM of the training path,
 * exposed for its parity test.  ws: sgemm scratch of at least ws_bytes (split-K partials). */
int r3dfs_sgemm(const float* A, int64_t sAm, int64_t sAk, const float* B, int64_t sBk, int64_t sBn,
                float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, float alpha, float beta,
                void* ws, size_t ws_bytes, r3dfs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* R3DFS_H_ */
