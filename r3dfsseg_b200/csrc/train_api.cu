// C ABI of the meta-training step (include/r3dfs.h, "Meta-training step"): one episode forward
// with batch-statistics BatchNorm, attention dropout and the way-contrast loss, and its backward
// into one flat gradient buffer.  Forward and backward share a workspace that keeps every saved
// activation; both carve it with the same deterministic layout.
#include "episode.cuh"
#include "lp.cuh"
#include "proto.cuh"
#include "train.cuh"

#define BN_EPS 1e-5f
#define BN_MOMENTUM 0.1f
#define CONTRAST_FPS_K 4
#define CONTRAST_TEMP 0.1f
#define SGEMM_PARTIAL_FLOATS ((size_t)8 << 20)
#define BN_SCRATCH_DOUBLES ((size_t)2 * 512 * BN_MAX_BLOCKS + 2 * 512)

static const int kBnChannels[R3DFS_N_BN] = {64, 64, 64, 64, 64, 64, 512, 256, 128, 64};

static void param_layout(int in_dim, int64_t* off) {
  int64_t o = 0;
  int i = 0;
  for (int l = 0; l < 3; ++l) {
    const int C = l == 0 ? in_dim : 64;
    const int64_t sz[6] = {64 * 2 * (int64_t)C, 64, 64, 64 * 64, 64, 64};
    for (int q = 0; q < 6; ++q) {
      off[i++] = o;
      o += sz[q];
    }
  }
  const int64_t rest[] = {512 * 192, 512, 512, 256 * 512, 256, 256,       // point MLP
                          128 * 256, 128, 128, 128, 64 * 128, 64, 64, 64,  // BaseLearner
                          64 * 256, 64 * 256, 64 * 256,                    // q, k, v
                          128 * 192, 128};                                 // proj
  for (int64_t s : rest) {
    off[i++] = o;
    o += s;
  }
  off[i] = o;
}

static void bn_layout(int64_t* off) {
  int64_t o = 0;
  for (int b = 0; b < R3DFS_N_BN; ++b) {
    off[b] = o;
    o += kBnChannels[b];
  }
  off[R3DFS_N_BN] = o;
}

// saved state of one getFeatures call (B clouds)
struct GroupWs {
  int64_t B, M, Ek;
  float* xp;
  int32_t* idx[3];
  float* h1pre[3];
  float* h2pre[3];
  uint8_t* arg[3];
  float *ecat, *h512pre, *a512, *l2pre, *l2, *bl0pre, *bl0a, *bl1pre, *qkv;
  float *P, *Pd;
  float* stats[R3DFS_N_BN];
};

struct TrainWs {
  EpisodeWs ep;
  GroupWs grp[2];  // 0 = support clouds, 1 = query clouds
  float* wpq[3];
  float *ones, *zeros;
  // transposed weights for the tensor-core input-gradient GEMMs: W2 of the 3 EdgeConvs, MLP0, MLP1,
  // BL1, Wqkv
  float* wT[7];
  // shared scratch
  float *xx, *PQ, *edgeA, *edgeB, *dS, *dqkv, *dl2, *d512, *decat, *d128, *d64, *dPQ, *dWf;
  double* bn_scratch;
  float* partial;
  // graph half
  float *dF, *dZ, *Gm, *dD, *gE;
  int32_t *members, *cmembers;
  // way-contrast
  int32_t *cpicks, *cpick_cnt, *cseeds, *cproto_cnt, *cassign, *cpcount;
  float *cpartial, *cseed_stats, *cproto, *dcproto, *loss_way;
};

static void carve_group(WsBump& ws, int64_t B, int N, int k, int in_dim, bool dropout, GroupWs& g) {
  g.B = B;
  g.M = B * N;
  g.Ek = g.M * k;
  g.xp = ws.take<float>(g.M * in_dim);
  for (int i = 0; i < 3; ++i) {
    g.idx[i] = ws.take<int32_t>(g.Ek);
    g.h1pre[i] = ws.take<float>(g.Ek * 64);
    g.h2pre[i] = ws.take<float>(g.Ek * 64);
    g.arg[i] = ws.take<uint8_t>(g.M * 64);
  }
  g.ecat = ws.take<float>(g.M * 192);
  g.h512pre = ws.take<float>(g.M * 512);
  g.a512 = ws.take<float>(g.M * 512);
  g.l2pre = ws.take<float>(g.M * 256);
  g.l2 = ws.take<float>(g.M * 256);
  g.bl0pre = ws.take<float>(g.M * 128);
  g.bl0a = ws.take<float>(g.M * 128);
  g.bl1pre = ws.take<float>(g.M * 64);
  g.qkv = ws.take<float>(g.M * 192);
  g.P = ws.take<float>((size_t)B * N * N);
  g.Pd = dropout ? ws.take<float>((size_t)B * N * N) : g.P;
  for (int b = 0; b < R3DFS_N_BN; ++b) g.stats[b] = ws.take<float>(2 * kBnChannels[b]);
}

static void carve_train(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d, int in_dim,
                        int dg_k, TrainWs& t) {
  const int N = c->n_points;
  carve_episode(ws, c, d, 1, in_dim, dg_k, t.ep);
  // dropout buffers are always carved so the layout does not depend on dropout_p
  carve_group(ws, d.C, N, dg_k, in_dim, true, t.grp[0]);
  carve_group(ws, c->n_query, N, dg_k, in_dim, true, t.grp[1]);
  const int64_t Bm = d.C > c->n_query ? d.C : c->n_query;
  const int64_t Mm = Bm * N, Em = Mm * dg_k;
  for (int i = 0; i < 3; ++i) t.wpq[i] = ws.take<float>(128 * 64);
  t.ones = ws.take<float>(512);
  t.zeros = ws.take<float>(512);
  {
    const size_t wt_sz[7] = {64 * 64, 64 * 64, 64 * 64, 512 * 192, 256 * 512, 64 * 128, 192 * 256};
    for (int i = 0; i < 7; ++i) t.wT[i] = ws.take<float>(wt_sz[i]);
  }
  t.xx = ws.take<float>(Mm);
  t.PQ = ws.take<float>(Mm * 128);
  t.edgeA = ws.take<float>(Em * 64);
  t.edgeB = ws.take<float>(Em * 64);
  t.dS = ws.take<float>((size_t)Bm * N * N);
  t.dqkv = ws.take<float>(Mm * 192);
  t.dl2 = ws.take<float>(Mm * 256);
  t.d512 = ws.take<float>(Mm * 512);
  t.decat = ws.take<float>(Mm * 192);
  t.d128 = ws.take<float>(Mm * 128);
  t.d64 = ws.take<float>(Mm * 64);
  t.dPQ = ws.take<float>(Mm * 128);
  t.dWf = ws.take<float>(128 * 64);
  t.bn_scratch = ws.take<double>(BN_SCRATCH_DOUBLES);
  t.partial = ws.take<float>(SGEMM_PARTIAL_FLOATS);
  t.dF = ws.take<float>((size_t)d.ep_rows * R3DFS_FEAT_DIM);
  t.dZ = ws.take<float>((size_t)d.nn * 8);
  t.Gm = ws.take<float>((size_t)d.nn * 8);
  t.dD = ws.take<float>(d.nn);
  t.gE = ws.take<float>((size_t)d.nn * c->k_connect);
  t.members = ws.take<int32_t>(d.S * d.slot);
  const int cslot = CONTRAST_FPS_K + 1;
  t.cmembers = ws.take<int32_t>(d.C * cslot);
  t.cpicks = ws.take<int32_t>(d.C * cslot);
  t.cpick_cnt = ws.take<int32_t>(d.C);
  t.cseeds = ws.take<int32_t>(d.C * cslot);
  t.cproto_cnt = ws.take<int32_t>(d.C);
  t.cassign = ws.take<int32_t>(d.ns_pts);
  const size_t ch = multi_prototypes_chunks(N);
  t.cpcount = ws.take<int32_t>(d.C * ch * cslot);
  t.cpartial = ws.take<float>(d.C * ch * cslot * R3DFS_FEAT_DIM);
  t.cseed_stats = ws.take<float>((size_t)d.C * 256);
  t.cproto = ws.take<float>((size_t)d.C * cslot * R3DFS_FEAT_DIM);
  t.dcproto = ws.take<float>((size_t)d.C * cslot * R3DFS_FEAT_DIM);
  t.loss_way = ws.take<float>(8);
}

static inline unsigned nblk(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

__global__ void gather_cloud_rows_kernel(const float* __restrict__ x, int C, int N, int64_t s_cloud,
                                         int64_t s_c, int64_t s_n, float* __restrict__ out,
                                         int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int c = (int)(e % C);
  const int64_t r = e / C;
  const int n = (int)(r % N);
  const int64_t cl = r / N;
  out[e] = x[cl * s_cloud + c * s_c + n * s_n];
}

__global__ void finish_losses_kernel(const float* __restrict__ lp, const float* __restrict__ loss_way,
                                     int n_way, float* __restrict__ losses) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    losses[0] = lp[0];
    float s = 0.f;
    for (int w = 0; w < n_way; ++w) s += loss_way[w];
    losses[1] = s / (float)n_way;
  }
}

struct TrainCtx {
  const float* params;
  const int64_t* off;   // parameter offsets
  float* grads;         // NULL in forward
  float* running;       // NULL -> not updated
  const int64_t* bnoff;
  int in_dim, k, N;
  cudaStream_t st;
  const float* P(int i) const { return params + off[i]; }
  float* G(int i) const { return grads + off[i]; }
  float* R(int b) const { return running ? running + 2 * bnoff[b] : nullptr; }
};

// y = x W^T (+ bias) on the tensor cores (3xTF32, exact to FP32 rounding)
static int lin_fwd(const TrainCtx& c, const float* x, int ldx, const float* W, const float* bias,
                   int64_t M, int K, int Nout, float* y, int ldy) {
  return launch_linear_auto(x, ldx, W, nullptr, bias, ACT_NONE, M, K, Nout, y, ldy, identity_map(),
                            c.st);
}

// dX (M x K) = dY (M x Nout) W (Nout x K), beta = 0/1
static int lin_bwd_x(const TrainCtx& c, const TrainWs& t, const float* dY, int ld_dy, const float* W,
                     int64_t M, int K, int Nout, float* dX, int ld_dx, float beta) {
  return launch_sgemm(dY, ld_dy, 1, 0, W, K, 1, 0, dX, ld_dx, 0, (int)M, K, Nout, 1, 1.f, beta, 1,
                      t.partial, c.st);
}

// dX (M x K) = dY (M x Nout) W with W^T (K x Nout, row-major) given: the forward tensor-core kernel
static int lin_bwd_x_tc(const TrainCtx& c, const float* dY, int ld_dy, const float* WT, int64_t M,
                        int K, int Nout, float* dX, int ld_dx) {
  return launch_linear_auto(dY, ld_dy, WT, nullptr, nullptr, ACT_NONE, M, Nout, K, dX, ld_dx,
                            identity_map(), c.st);
}

// dW (Nout x K) += dY^T X, reduced over M rows (split-K, fixed order)
static int lin_bwd_w(const TrainCtx& c, const TrainWs& t, const float* dY, int ld_dy, const float* X,
                     int ldx, int64_t M, int K, int Nout, float* dW) {
  // 3xTF32 tensor cores, split over the rows, fixed-order reduce
  const int max_splits = (int)(SGEMM_PARTIAL_FLOATS / ((size_t)Nout * K));
  if (max_splits >= 1) {
    int splits = 1;
    R3DFS_TRY(launch_gemm_tn_tc(dY, ld_dy, X, ldx, Nout, K, M, max_splits, t.partial, &splits, c.st));
    return launch_sgemm_reduce(t.partial, Nout, K, splits, 1.f, 1.f, dW, K, c.st);
  }
  const int splits = sgemm_splits(Nout, K, M, 1);
  if ((size_t)splits * Nout * K > SGEMM_PARTIAL_FLOATS) return R3DFS_E_WORKSPACE;
  return launch_sgemm(dY, 1, ld_dy, 0, X, ldx, 1, 0, dW, K, 0, Nout, K, (int)M, 1, 1.f, 1.f, splits,
                      t.partial, c.st);
}

static int bn_index_param(int b, int& gi, int& bi) {
  // BN layer b -> parameter indices of (gamma, beta)
  if (b < 6) {
    gi = 6 * (b / 2) + (b % 2 ? R3DFS_P_EC0_G2 : R3DFS_P_EC0_G1);
  } else if (b == 6) gi = R3DFS_P_MLP0_G;
  else if (b == 7) gi = R3DFS_P_MLP1_G;
  else if (b == 8) gi = R3DFS_P_BL0_G;
  else gi = R3DFS_P_BL1_G;
  bi = gi + 1;
  return 0;
}

static int bn_fwd(const TrainCtx& c, const TrainWs& t, const GroupWs& g, int b, const float* x,
                  int64_t ldx, int64_t rows, int act, float* y, int64_t ldy) {
  int gi, bi;
  bn_index_param(b, gi, bi);
  const int C = kBnChannels[b];
  R3DFS_TRY(launch_bn_stats(x, ldx, rows, C, BN_EPS, BN_MOMENTUM, c.R(b), g.stats[b], t.bn_scratch,
                            c.st));
  return launch_bn_act(x, ldx, rows, C, g.stats[b], c.P(gi), c.P(bi), act, y, ldy, c.st);
}

static int bn_bwd(const TrainCtx& c, const TrainWs& t, const GroupWs& g, int b, const float* dy,
                  int64_t ld_dy, const float* x, int64_t ldx, int64_t rows, int act, float* dx,
                  int64_t ld_dx) {
  int gi, bi;
  bn_index_param(b, gi, bi);
  return launch_bn_act_bwd(dy, ld_dy, x, ldx, rows, kBnChannels[b], g.stats[b], c.P(gi), c.P(bi), act,
                           dx, ld_dx, c.G(gi), c.G(bi), t.bn_scratch, c.st);
}

// getFeatures in training mode (models/mpti.py:579-589) for one group of clouds; Fout rows ld 192
static int group_forward(const TrainCtx& c, const TrainWs& t, const GroupWs& g, float dropout_p,
                         const uint8_t* keep, float* Fout) {
  const int N = c.N, k = c.k;
  const int64_t M = g.M, Ek = g.Ek;
  cudaStream_t st = c.st;
  for (int i = 0; i < 3; ++i) {
    const float* in = i == 0 ? g.xp : g.ecat + 64 * (i - 1);
    const int ld = i == 0 ? c.in_dim : 192;
    const int C = i == 0 ? c.in_dim : 64;
    const int pw = 6 * i;
    R3DFS_TRY(launch_row_norms(in, M, ld, C, t.xx, st));
    R3DFS_TRY(launch_knn_auto(in, ld, C, t.xx, g.B, N, k, g.idx[i], nullptr, 0, st));
    R3DFS_TRY(lin_fwd(c, in, ld, t.wpq[i], nullptr, M, C, 128, t.PQ, 128));
    R3DFS_TRY(launch_edge_pre(t.PQ, g.idx[i], g.B, N, k, g.h1pre[i], st));
    R3DFS_TRY(bn_fwd(c, t, g, 2 * i, g.h1pre[i], 64, Ek, ACT_LRELU, t.edgeA, 64));
    R3DFS_TRY(lin_fwd(c, t.edgeA, 64, c.P(pw + R3DFS_P_EC0_W2), nullptr, Ek, 64, 64, g.h2pre[i], 64));
    int gi, bi;
    bn_index_param(2 * i + 1, gi, bi);
    R3DFS_TRY(launch_bn_stats(g.h2pre[i], 64, Ek, 64, BN_EPS, BN_MOMENTUM, c.R(2 * i + 1),
                              g.stats[2 * i + 1], t.bn_scratch, st));
    R3DFS_TRY(launch_edge_max(g.h2pre[i], g.stats[2 * i + 1], c.P(gi), c.P(bi), M, k,
                              g.ecat + 64 * i, 192, g.arg[i], st));
  }
  R3DFS_TRY(launch_copy_cols_plain(g.ecat, 192, M, 64, Fout, 192, st));
  // point MLP 192 -> 512 -> 256 (models/dgcnn.py:121-122)
  R3DFS_TRY(lin_fwd(c, g.ecat, 192, c.P(R3DFS_P_MLP0_W), nullptr, M, 192, 512, g.h512pre, 512));
  R3DFS_TRY(bn_fwd(c, t, g, 6, g.h512pre, 512, M, ACT_LRELU, g.a512, 512));
  R3DFS_TRY(lin_fwd(c, g.a512, 512, c.P(R3DFS_P_MLP1_W), nullptr, M, 512, 256, g.l2pre, 256));
  R3DFS_TRY(bn_fwd(c, t, g, 7, g.l2pre, 256, M, ACT_LRELU, g.l2, 256));
  // BaseLearner (models/mpti.py:35-40)
  R3DFS_TRY(lin_fwd(c, g.l2, 256, c.P(R3DFS_P_BL0_W), c.P(R3DFS_P_BL0_BIAS), M, 256, 128, g.bl0pre, 128));
  R3DFS_TRY(bn_fwd(c, t, g, 8, g.bl0pre, 128, M, ACT_RELU, g.bl0a, 128));
  R3DFS_TRY(lin_fwd(c, g.bl0a, 128, c.P(R3DFS_P_BL1_W), c.P(R3DFS_P_BL1_BIAS), M, 128, 64, g.bl1pre, 64));
  R3DFS_TRY(bn_fwd(c, t, g, 9, g.bl1pre, 64, M, ACT_NONE, Fout + 128, 192));
  // SelfAttention (models/attention.py:39-48)
  R3DFS_TRY(lin_fwd(c, g.l2, 256, c.P(R3DFS_P_ATT_Q), nullptr, M, 256, 192, g.qkv, 192));
  const int64_t cs = (int64_t)N * 192, ps = (int64_t)N * N;
  R3DFS_TRY(launch_sgemm(g.qkv, 192, 1, cs, g.qkv + 64, 1, 192, cs, g.P, N, ps, N, N, 64, (int)g.B,
                         0.125f, 0.f, 1, t.partial, st));
  const bool drop = keep != nullptr && dropout_p > 0.f;
  R3DFS_TRY(launch_softmax_rows(g.P, g.B * N, N, drop ? keep : nullptr, dropout_p, g.Pd, st));
  const float* Pd = drop ? g.Pd : g.P;
  R3DFS_TRY(launch_sgemm(Pd, N, 1, ps, g.qkv + 128, 192, 1, cs, Fout + 64, 192, cs, N, 64, N,
                         (int)g.B, 1.f, 0.f, 1, t.partial, st));
  return 0;
}

// backward of group_forward given dF (rows ld 192); accumulates parameter gradients
static int group_backward(const TrainCtx& c, const TrainWs& t, const GroupWs& g, float dropout_p,
                          const uint8_t* keep, const float* dF) {
  const int N = c.N, k = c.k;
  const int64_t M = g.M, Ek = g.Ek;
  cudaStream_t st = c.st;
  const int64_t cs = (int64_t)N * 192, ps = (int64_t)N * N;
  const bool drop = keep != nullptr && dropout_p > 0.f;
  const float* Pd = drop ? g.Pd : g.P;
  // ---- attention: O = Pd V, Pd = dropout(softmax(Q K^T / 8)) ------------------------------------
  const float* dO = dF + 64;
  // dPd = dO V^T
  R3DFS_TRY(launch_sgemm(dO, 192, 1, cs, g.qkv + 128, 1, 192, cs, t.dS, N, ps, N, N, 64, (int)g.B,
                         1.f, 0.f, 1, t.partial, st));
  // dV = Pd^T dO
  R3DFS_TRY(launch_sgemm(Pd, 1, N, ps, dO, 192, 1, cs, t.dqkv + 128, 192, cs, N, 64, N, (int)g.B,
                         1.f, 0.f, 1, t.partial, st));
  R3DFS_TRY(launch_softmax_rows_bwd(g.P, t.dS, g.B * N, N, drop ? keep : nullptr, dropout_p, st));
  // dQ = dS K / 8 ; dK = dS^T Q / 8
  R3DFS_TRY(launch_sgemm(t.dS, N, 1, ps, g.qkv + 64, 192, 1, cs, t.dqkv, 192, cs, N, 64, N, (int)g.B,
                         0.125f, 0.f, 1, t.partial, st));
  R3DFS_TRY(launch_sgemm(t.dS, 1, N, ps, g.qkv, 192, 1, cs, t.dqkv + 64, 192, cs, N, 64, N, (int)g.B,
                         0.125f, 0.f, 1, t.partial, st));
  R3DFS_TRY(lin_bwd_w(c, t, t.dqkv, 192, g.l2, 256, M, 256, 192, c.G(R3DFS_P_ATT_Q)));
  R3DFS_TRY(lin_bwd_x_tc(c, t.dqkv, 192, t.wT[6], M, 256, 192, t.dl2, 256));
  // ---- BaseLearner ------------------------------------------------------------------------------
  R3DFS_TRY(bn_bwd(c, t, g, 9, dF + 128, 192, g.bl1pre, 64, M, ACT_NONE, t.d64, 64));
  R3DFS_TRY(lin_bwd_w(c, t, t.d64, 64, g.bl0a, 128, M, 128, 64, c.G(R3DFS_P_BL1_W)));
  R3DFS_TRY(launch_col_sum_acc(t.d64, 64, M, 64, c.G(R3DFS_P_BL1_BIAS), t.bn_scratch, st));
  R3DFS_TRY(lin_bwd_x_tc(c, t.d64, 64, t.wT[5], M, 128, 64, t.d128, 128));
  R3DFS_TRY(bn_bwd(c, t, g, 8, t.d128, 128, g.bl0pre, 128, M, ACT_RELU, t.d128, 128));
  R3DFS_TRY(lin_bwd_w(c, t, t.d128, 128, g.l2, 256, M, 256, 128, c.G(R3DFS_P_BL0_W)));
  R3DFS_TRY(launch_col_sum_acc(t.d128, 128, M, 128, c.G(R3DFS_P_BL0_BIAS), t.bn_scratch, st));
  R3DFS_TRY(lin_bwd_x(c, t, t.d128, 128, c.P(R3DFS_P_BL0_W), M, 256, 128, t.dl2, 256, 1.f));
  // ---- point MLP --------------------------------------------------------------------------------
  R3DFS_TRY(bn_bwd(c, t, g, 7, t.dl2, 256, g.l2pre, 256, M, ACT_LRELU, t.dl2, 256));
  R3DFS_TRY(lin_bwd_w(c, t, t.dl2, 256, g.a512, 512, M, 512, 256, c.G(R3DFS_P_MLP1_W)));
  R3DFS_TRY(lin_bwd_x_tc(c, t.dl2, 256, t.wT[4], M, 512, 256, t.d512, 512));
  R3DFS_TRY(bn_bwd(c, t, g, 6, t.d512, 512, g.h512pre, 512, M, ACT_LRELU, t.d512, 512));
  R3DFS_TRY(lin_bwd_w(c, t, t.d512, 512, g.ecat, 192, M, 192, 512, c.G(R3DFS_P_MLP0_W)));
  R3DFS_TRY(lin_bwd_x_tc(c, t.d512, 512, t.wT[3], M, 192, 512, t.decat, 192));
  R3DFS_TRY(launch_add_cols(dF, 192, M, 64, t.decat, 192, st));  // level-1 feature
  // ---- EdgeConv blocks, last to first -------------------------------------------------------------
  for (int i = 2; i >= 0; --i) {
    const float* in = i == 0 ? g.xp : g.ecat + 64 * (i - 1);
    const int ld = i == 0 ? c.in_dim : 192;
    const int C = i == 0 ? c.in_dim : 64;
    const int pw = 6 * i;
    R3DFS_TRY(launch_edge_max_bwd(t.decat + 64 * i, 192, g.arg[i], M, k, t.edgeB, st));
    R3DFS_TRY(bn_bwd(c, t, g, 2 * i + 1, t.edgeB, 64, g.h2pre[i], 64, Ek, ACT_LRELU, t.edgeB, 64));
    // a1 = LReLU(BN1(h1pre)) recomputed
    int gi, bi;
    bn_index_param(2 * i, gi, bi);
    R3DFS_TRY(launch_bn_act(g.h1pre[i], 64, Ek, 64, g.stats[2 * i], c.P(gi), c.P(bi), ACT_LRELU,
                            t.edgeA, 64, st));
    R3DFS_TRY(lin_bwd_w(c, t, t.edgeB, 64, t.edgeA, 64, Ek, 64, 64, c.G(pw + R3DFS_P_EC0_W2)));
    R3DFS_TRY(lin_bwd_x_tc(c, t.edgeB, 64, t.wT[i], Ek, 64, 64, t.edgeA, 64));
    R3DFS_TRY(bn_bwd(c, t, g, 2 * i, t.edgeA, 64, g.h1pre[i], 64, Ek, ACT_LRELU, t.edgeA, 64));
    R3DFS_TRY(launch_edge_pre_bwd(t.edgeA, g.idx[i], g.B, N, k, t.dPQ, st));
    // d[W1a ; W1b - W1a] = dPQ^T x, unfolded into dW1
    cudaError_t ce = cudaMemsetAsync(t.dWf, 0, sizeof(float) * 128 * C, st);
    if (ce != cudaSuccess) return (int)ce;
    R3DFS_TRY(lin_bwd_w(c, t, t.dPQ, 128, in, ld, M, C, 128, t.dWf));
    R3DFS_TRY(launch_unfold_w1_grad(t.dWf, C, c.G(pw + R3DFS_P_EC0_W1), st));
    if (i > 0)
      R3DFS_TRY(lin_bwd_x(c, t, t.dPQ, 128, t.wpq[i], M, 64, 128, t.decat + 64 * (i - 1), 192, 1.f));
  }
  return 0;
}

static int fold_weights(const TrainCtx& c, const TrainWs& t) {
  R3DFS_TRY(launch_fill_f32(t.ones, 512, 1.f, c.st));
  R3DFS_TRY(launch_fill_f32(t.zeros, 512, 0.f, c.st));
  for (int i = 0; i < 3; ++i) {
    const int C = i == 0 ? c.in_dim : 64;
    // spq / tpq outputs land in the (unused) eval-encoder scratch
    R3DFS_TRY(launch_fold_edge_w1(c.P(6 * i + R3DFS_P_EC0_W1), t.ones, t.zeros, C, t.wpq[i],
                                  t.ep.enc.spq, t.ep.enc.tpq, c.st));
  }
  return 0;
}

extern "C" {

int64_t r3dfs_train_param_layout(int in_dim, int64_t* offsets) {
  int64_t off[R3DFS_N_PARAMS + 1];
  param_layout(in_dim, off);
  if (offsets)
    for (int i = 0; i <= R3DFS_N_PARAMS; ++i) offsets[i] = off[i];
  return off[R3DFS_P_BL0_W];
}

void r3dfs_train_bn_layout(int64_t* offsets) { bn_layout(offsets); }

size_t r3dfs_mpti_train_workspace(const r3dfs_episode_cfg_t* cfg, int in_dim, int dgcnn_k) {
  EpisodeDims d;
  if (episode_dims(cfg, d) != 0 || in_dim < 1 || in_dim > 64 || dgcnn_k < 1 || dgcnn_k > 32) return 0;
  WsBump ws(nullptr, ~(size_t)0);
  TrainWs t;
  carve_train(ws, cfg, d, in_dim, dgcnn_k, t);
  return ws.off + 4096;
}

int r3dfs_mpti_train_forward(const r3dfs_episode_cfg_t* cfg_in, int in_dim, int dgcnn_k,
                             const float* params, float* bn_running, const float* support_x,
                             int64_t s_cloud, int64_t s_c, int64_t s_n, const int32_t* support_y,
                             const int32_t* support_flag, const float* query_x, int64_t q_cloud,
                             int64_t q_c, int64_t q_n, const int64_t* query_y, float dropout_p,
                             const uint8_t* keep_support, const uint8_t* keep_query, float* logits,
                             float* losses, int32_t* cg_iters, void* wsp, size_t ws_bytes,
                             r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg_in, d));
  if (!params || !support_x || !support_y || !support_flag || !query_x || !query_y || !logits ||
      !losses || !wsp)
    return R3DFS_E_BADARG;
  if (in_dim < 1 || in_dim > 64 || dgcnn_k < 1 || dgcnn_k > 32 || dropout_p < 0.f || dropout_p >= 1.f ||
      cfg_in->k_shot < 2)
    return R3DFS_E_UNSUPPORTED;
  if (ws_bytes < r3dfs_mpti_train_workspace(cfg_in, in_dim, dgcnn_k)) return R3DFS_E_WORKSPACE;
  r3dfs_episode_cfg_t cfg = *cfg_in;
  cfg.mdns = 0;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  TrainWs t;
  carve_train(ws, &cfg, d, in_dim, dgcnn_k, t);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  int64_t off[R3DFS_N_PARAMS + 1], bnoff[R3DFS_N_BN + 1];
  param_layout(in_dim, off);
  bn_layout(bnoff);
  TrainCtx c{params, off, nullptr, bn_running, bnoff, in_dim, dgcnn_k, cfg.n_points, st};
  const int N = cfg.n_points, D = R3DFS_FEAT_DIM;
  R3DFS_TRY(fold_weights(c, t));
  int64_t tot = (int64_t)d.C * N * in_dim;
  gather_cloud_rows_kernel<<<nblk(tot), 256, 0, st>>>(support_x, in_dim, N, s_cloud, s_c, s_n,
                                                      t.grp[0].xp, tot);
  R3DFS_CHECK_LAUNCH();
  tot = (int64_t)cfg.n_query * N * in_dim;
  gather_cloud_rows_kernel<<<nblk(tot), 256, 0, st>>>(query_x, in_dim, N, q_cloud, q_c, q_n,
                                                      t.grp[1].xp, tot);
  R3DFS_CHECK_LAUNCH();
  // two getFeatures calls, support first (models/mpti.py:433-436)
  R3DFS_TRY(group_forward(c, t, t.grp[0], dropout_p, keep_support, t.ep.F + (size_t)d.nn * D));
  R3DFS_TRY(group_forward(c, t, t.grp[1], dropout_p, keep_query, t.ep.F + (size_t)d.ppad * D));
  // prototypes -> affinity graph -> label propagation -> cross-entropy (models/mpti.py:484-571)
  r3dfs_episode_diag_t diag = {};
  diag.cg_iters = cg_iters;
  R3DFS_TRY(episode_graph_half(&cfg, d, 1, t.ep, support_x, 0, s_cloud, s_c, s_n, support_y, query_y,
                               logits, t.loss_way + 7, nullptr, &diag, st, /*latency=*/true));
  // way-contrast loss on fps_k = 4 prototypes of every shot's foreground (models/mpti.py:226-313);
  // the shots' foreground rows are contiguous sub-ranges of the compacted set buffer
  const int cslot = CONTRAST_FPS_K + 1;
  R3DFS_TRY(launch_multi_prototypes(t.ep.setfeat, D, t.ep.cloud_fg_off, t.ep.fg_cnt, d.C, N,
                                    CONTRAST_FPS_K, t.cpicks, t.cpick_cnt, t.cseeds, t.cproto_cnt,
                                    t.cassign, t.cpartial, t.cpcount, t.cseed_stats, d.C, 0, t.cproto,
                                    D, st));
  for (int w = 0; w < cfg.n_way; ++w)
    R3DFS_TRY(launch_contrast(t.cproto, t.cproto_cnt, cslot, D, support_flag, cfg.n_way, cfg.k_shot,
                              w, c.P(R3DFS_P_PROJ_W), c.P(R3DFS_P_PROJ_B), CONTRAST_TEMP, t.loss_way,
                              0, 0.f, nullptr, nullptr, nullptr, st));
  finish_losses_kernel<<<1, 32, 0, st>>>(t.loss_way + 7, t.loss_way, cfg.n_way, losses);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int r3dfs_mpti_train_backward(const r3dfs_episode_cfg_t* cfg_in, int in_dim, int dgcnn_k,
                              const float* params, const int32_t* support_y,
                              const int32_t* support_flag, const int64_t* query_y, float dropout_p,
                              const uint8_t* keep_support, const uint8_t* keep_query, float w_lp,
                              float w_contrast, float* grads, void* wsp, size_t ws_bytes,
                              r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg_in, d));
  if (!params || !support_y || !support_flag || !query_y || !grads || !wsp) return R3DFS_E_BADARG;
  if (ws_bytes < r3dfs_mpti_train_workspace(cfg_in, in_dim, dgcnn_k)) return R3DFS_E_WORKSPACE;
  r3dfs_episode_cfg_t cfg = *cfg_in;
  cfg.mdns = 0;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  TrainWs t;
  carve_train(ws, &cfg, d, in_dim, dgcnn_k, t);
  if (!ws.ok()) return R3DFS_E_WORKSPACE;
  int64_t off[R3DFS_N_PARAMS + 1], bnoff[R3DFS_N_BN + 1];
  param_layout(in_dim, off);
  bn_layout(bnoff);
  TrainCtx c{params, off, grads, nullptr, bnoff, in_dim, dgcnn_k, cfg.n_points, st};
  const int N = cfg.n_points, D = R3DFS_FEAT_DIM, nn = d.nn, nc = d.nc, kc = cfg.k_connect;
  const EpisodeWs& w = t.ep;
  cudaError_t ce = cudaMemsetAsync(grads, 0, sizeof(float) * off[R3DFS_N_PARAMS], st);
  if (ce != cudaSuccess) return (int)ce;
  ce = cudaMemsetAsync(t.dF, 0, sizeof(float) * (size_t)d.ep_rows * D, st);
  if (ce != cudaSuccess) return (int)ce;
  for (int i = 0; i < 3; ++i)
    R3DFS_TRY(launch_transpose(c.P(6 * i + R3DFS_P_EC0_W2), 64, 64, t.wT[i], st));
  R3DFS_TRY(launch_transpose(c.P(R3DFS_P_MLP0_W), 512, 192, t.wT[3], st));
  R3DFS_TRY(launch_transpose(c.P(R3DFS_P_MLP1_W), 256, 512, t.wT[4], st));
  R3DFS_TRY(launch_transpose(c.P(R3DFS_P_BL1_W), 64, 128, t.wT[5], st));
  R3DFS_TRY(launch_transpose(c.P(R3DFS_P_ATT_Q), 192, 256, t.wT[6], st));
  // cross-entropy -> dZ -> adjoint solve G = (I - alpha S)^-1 dZ -> per-edge gradients -> node rows
  R3DFS_TRY(launch_ce_grad(w.Z, nn, d.ppad, d.nq_pts, nc, query_y, w_lp, t.dZ, st));
  R3DFS_TRY(launch_lp_solve(w.rowptr, w.rowlen, w.mcol, w.mval, w.valid, 1, nn, kc, t.dZ, nc,
                            cfg.alpha, cfg.cg_tol, cfg.cg_max_iter, t.Gm, w.X, w.R, w.P, w.AP,
                            nullptr, nullptr, st, /*latency=*/true, w.D2,
                            sizeof(float) * episode_d2_floats(1, nn, kc)));
  R3DFS_TRY(launch_lp_adjoint_edges(w.rowptr, w.rowlen, w.mcol, w.mval, w.dinv, w.valid, w.nbr, w.sim,
                                    nn, kc, nc, w.Z, t.Gm, cfg.alpha, cfg.sigma, t.dD, t.gE, st));
  R3DFS_TRY(launch_sim_bwd(w.F, D, w.valid, w.nbr, t.gE, nn, kc, t.dF, st));
  // way-contrast backward into the per-shot prototypes and the projection head
  const int cslot = CONTRAST_FPS_K + 1;
  const bool with_contrast = w_contrast != 0.f;
  if (with_contrast) {
    ce = cudaMemsetAsync(t.dcproto, 0, sizeof(float) * (size_t)d.C * cslot * D, st);
    if (ce != cudaSuccess) return (int)ce;
    for (int wy = 0; wy < cfg.n_way; ++wy)
      R3DFS_TRY(launch_contrast(t.cproto, t.cproto_cnt, cslot, D, support_flag, cfg.n_way,
                                cfg.k_shot, wy, c.P(R3DFS_P_PROJ_W), c.P(R3DFS_P_PROJ_B),
                                CONTRAST_TEMP, t.loss_way, 1, w_contrast / (float)cfg.n_way,
                                c.G(R3DFS_P_PROJ_W), c.G(R3DFS_P_PROJ_B), t.dcproto, st));
    R3DFS_TRY(launch_proto_counts(t.cpcount, w.fg_cnt, t.cproto_cnt, d.C, cslot,
                                  multi_prototypes_chunks(N), t.cmembers, st));
  }
  // prototype means -> support points
  R3DFS_TRY(launch_proto_counts(w.pcount, w.set_n, w.proto_cnt, d.S, d.slot,
                                multi_prototypes_chunks(d.ns_pts), t.members, st));
  float* dFsup = t.dF + (size_t)nn * D;
  R3DFS_TRY(launch_support_grad(t.dF, d.slot, w.assign, t.members, with_contrast ? t.dcproto : nullptr,
                                cslot, t.cassign, t.cmembers, cfg.n_way, cfg.k_shot, N, D, support_y,
                                w.cloud_bg_off, w.cloud_fg_off, dFsup, st));
  R3DFS_TRY(group_backward(c, t, t.grp[0], dropout_p, keep_support, dFsup));
  R3DFS_TRY(group_backward(c, t, t.grp[1], dropout_p, keep_query, t.dF + (size_t)d.ppad * D));
  return 0;
}

// --------------------------------------------------------------------------------------------
// The reference's logging-only diagnostics of a training forward (models/mpti.py:514-552):
// per way, every foreground support point takes the label-propagation verdict of its prototype
// (argmax of the prototype's Z row == way + 1) and is compared with the ground-truth mask;
// clean_ratio_LP = fraction of agreeing points, clean_ratio_original = fraction whose GIVEN mask
// (always 1 on these points) agrees.  One CTA; integer counts, so the result is exact.
// --------------------------------------------------------------------------------------------
__global__ __launch_bounds__(1024) void clean_ratio_kernel(
    const int32_t* __restrict__ support_y, const int32_t* __restrict__ gt_support_y,
    const int32_t* __restrict__ cloud_fg_off, const int32_t* __restrict__ assign,
    const float* __restrict__ Z, int n_way, int k_shot, int N, int slot, int nc,
    float* __restrict__ out) {
  __shared__ int s_warp[32];
  __shared__ int s_cnt[3];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  float ratio_lp = 0.f, ratio_orig = 0.f;
  for (int way = 0; way < n_way; ++way) {
    int ok_lp = 0, ok_orig = 0, total = 0;
    for (int shot = 0; shot < k_shot; ++shot) {
      const int cloud = way * k_shot + shot;
      const int32_t* y = support_y + (int64_t)cloud * N;
      const int32_t* g = gt_support_y + (int64_t)cloud * N;
      int base = cloud_fg_off[cloud];  // row of the cloud's first foreground point in the set buffer
      for (int p0 = 0; p0 < N; p0 += 1024) {
        const int p = p0 + tid;
        const bool fg = p < N && y[p] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, fg);
        if (lane == 0) s_warp[w] = __popc(bal);
        __syncthreads();
        int before = 0, all = 0;
        for (int q = 0; q < 32; ++q) {
          const int c = s_warp[q];
          before += q < w ? c : 0;
          all += c;
        }
        if (fg) {
          const int row = base + before + __popc(bal & ((1u << lane) - 1));
          const float* z = Z + (int64_t)((1 + way) * slot + assign[row]) * nc;
          int arg = 0;
          float best = z[0];
          for (int c = 1; c < nc; ++c)
            if (z[c] > best) {
              best = z[c];
              arg = c;
            }
          const int gt = g[p];
          ok_lp += ((arg == way + 1) ? 1 : 0) == gt;
          ok_orig += 1 == gt;
          total += 1;
        }
        base += all;
        __syncthreads();
      }
    }
    // block sums
    int v[3] = {ok_lp, ok_orig, total};
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      for (int o = 16; o > 0; o >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
      if (lane == 0) s_warp[w] = v[q];
      __syncthreads();
      if (tid == 0) {
        int t = 0;
        for (int i = 0; i < 32; ++i) t += s_warp[i];
        s_cnt[q] = t;
      }
      __syncthreads();
    }
    ratio_lp += (float)s_cnt[0] / (float)s_cnt[2];   // 0/0 = nan, as in the reference
    ratio_orig += (float)s_cnt[1] / (float)s_cnt[2];
  }
  if (tid == 0) {
    out[0] = ratio_lp / (float)n_way;
    out[1] = ratio_orig / (float)n_way;
  }
}

int r3dfs_mpti_train_clean_ratio(const r3dfs_episode_cfg_t* cfg_in, int in_dim, int dgcnn_k,
                                 const int32_t* support_y, const int32_t* gt_support_y,
                                 float* ratios, void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg_in, d));
  if (!support_y || !gt_support_y || !ratios || !wsp) return R3DFS_E_BADARG;
  if (ws_bytes < r3dfs_mpti_train_workspace(cfg_in, in_dim, dgcnn_k)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  TrainWs t;
  carve_train(ws, cfg_in, d, in_dim, dgcnn_k, t);
  clean_ratio_kernel<<<1, 1024, 0, st>>>(support_y, gt_support_y, t.ep.cloud_fg_off, t.ep.assign,
                                         t.ep.Z, cfg_in->n_way, cfg_in->k_shot, cfg_in->n_points,
                                         d.slot, d.nc, ratios);
  R3DFS_CHECK_LAUNCH();
  return 0;
}

int r3dfs_mpti_train_export(const r3dfs_episode_cfg_t* cfg_in, int in_dim, int dgcnn_k,
                            const r3dfs_train_export_t* o, void* wsp, size_t ws_bytes,
                            r3dfs_stream_t stream) {
  EpisodeDims d;
  R3DFS_TRY(episode_dims(cfg_in, d));
  if (!o || !wsp) return R3DFS_E_BADARG;
  if (ws_bytes < r3dfs_mpti_train_workspace(cfg_in, in_dim, dgcnn_k)) return R3DFS_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  WsBump ws(wsp, ws_bytes);
  TrainWs t;
  carve_train(ws, cfg_in, d, in_dim, dgcnn_k, t);
  auto cp = [&](void* dst, const void* src, size_t bytes) -> int {
    if (!dst) return 0;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
    return e == cudaSuccess ? 0 : (int)e;
  };
  for (int i = 0; i < 3; ++i) {
    R3DFS_TRY(cp(o->knn_support[i], t.grp[0].idx[i], sizeof(int32_t) * t.grp[0].Ek));
    R3DFS_TRY(cp(o->knn_query[i], t.grp[1].idx[i], sizeof(int32_t) * t.grp[1].Ek));
  }
  R3DFS_TRY(cp(o->set_off, t.ep.set_off, sizeof(int32_t) * d.S));
  R3DFS_TRY(cp(o->set_n, t.ep.set_n, sizeof(int32_t) * d.S));
  R3DFS_TRY(cp(o->proto_cnt, t.ep.proto_cnt, sizeof(int32_t) * d.S));
  R3DFS_TRY(cp(o->assign, t.ep.assign, sizeof(int32_t) * d.ns_pts));
  R3DFS_TRY(cp(o->cloud_fg_off, t.ep.cloud_fg_off, sizeof(int32_t) * d.C));
  R3DFS_TRY(cp(o->fg_cnt, t.ep.fg_cnt, sizeof(int32_t) * d.C));
  R3DFS_TRY(cp(o->cproto_cnt, t.cproto_cnt, sizeof(int32_t) * d.C));
  R3DFS_TRY(cp(o->cassign, t.cassign, sizeof(int32_t) * d.ns_pts));
  R3DFS_TRY(cp(o->nbr, t.ep.nbr, sizeof(int32_t) * (size_t)d.nn * cfg_in->k_connect));
  R3DFS_TRY(cp(o->valid, t.ep.valid, (size_t)d.nn));
  return 0;
}

int r3dfs_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                    int64_t n_group0, float lr0, float lr1, float beta1, float beta2, float eps,
                    int64_t step, float grad_scale, r3dfs_stream_t stream) {
  if (!params || !grads || !exp_avg || !exp_avg_sq || n <= 0 || step < 1) return R3DFS_E_BADARG;
  // bias corrections in double, as torch.optim.Adam computes them (1 - 0.999^t loses ~6e-5
  // relative in FP32 powf at small t)
  const float bc1 = (float)(1.0 - pow((double)beta1, (double)step)),
              bc2 = (float)(1.0 - pow((double)beta2, (double)step));
  return launch_adam(params, grads, exp_avg, exp_avg_sq, n, n_group0, lr0, lr1, beta1, beta2, eps,
                     bc1, bc2, grad_scale, (cudaStream_t)stream);
}

int r3dfs_dropout_mask(uint64_t seed, int64_t n, float p, uint8_t* mask, r3dfs_stream_t stream) {
  if (!mask || n <= 0 || p < 0.f || p >= 1.f) return R3DFS_E_BADARG;
  return launch_dropout_mask(seed, n, p, mask, (cudaStream_t)stream);
}

int r3dfs_sgemm(const float* A, int64_t sAm, int64_t sAk, const float* B, int64_t sBk, int64_t sBn,
                float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, float alpha, float beta,
                void* wsp, size_t ws_bytes, r3dfs_stream_t stream) {
  if (!A || !B || !C || M <= 0 || N <= 0 || K <= 0) return R3DFS_E_BADARG;
  int splits = sgemm_splits((int)M, (int)N, K, 1);
  if (!wsp || (size_t)splits * M * N * sizeof(float) > ws_bytes) splits = 1;
  return launch_sgemm(A, sAm, sAk, 0, B, sBk, sBn, 0, C, ldc, 0, (int)M, (int)N, (int)K, 1, alpha,
                      beta, splits, (float*)wsp, (cudaStream_t)stream);
}

}  // extern "C"
