// Episode pipeline internals shared by api.cu (inference) and train_api.cu (meta-training).
#pragma once
#include "common.cuh"

struct EncoderWs {
  float* xx;
  int32_t* idx;
  float* wpq;
  float* spq;
  float* tpq;
  float* PQ;
  float* ecat;
  float* h512;
  float* l2;
  float* h128;
  float* qkv;
};


struct EpisodeDims {
  int S, slot, ppad, nq_pts, nn, ns_pts, cpe, C, nc;
  int64_t ep_rows;
};


struct EpisodeWs {
  float* xp;
  EncoderWs enc;
  float* F;
  int32_t *fg_cnt, *keep, *set_off, *set_n, *cloud_bg_off, *cloud_fg_off;
  float* setfeat;
  uint8_t* fps_spill;  // fps_q8_spill_bytes(all set rows)
  int32_t *picks, *pick_cnt, *seeds, *proto_cnt, *assign, *pcount;
  float *partial, *seed_stats;
  float* cell_mean;
  int32_t* cell_cnt;
  uint8_t* valid;
  float *Y, *norms, *D2;
  unsigned* gmin;  // group minima of the distance matrix (launch_affinity)
  int32_t* nbr;
  float* sim;
  int32_t *in_cnt, *in_ptr, *in_src;
  float *in_w, *dinv, *Z, *X, *R, *P, *AP;
  int32_t *rowptr, *rowlen, *cursor;
  uint16_t* mcol;
  float* mval;
};


void carve_encoder(WsBump& ws, int64_t M, int k, EncoderWs& e);
int check_weights(const r3dfs_weights_t* w);
int encoder_forward(const r3dfs_weights_t* w, const float* xp, int64_t B, int N, const EncoderWs& e,
                    float* F, RowMap map, float* level2, cudaStream_t st,
                    const StageRec* sr = nullptr);
int episode_dims(const r3dfs_episode_cfg_t* c, EpisodeDims& d);
size_t episode_d2_floats(size_t G, size_t nn, int k);
void carve_episode(WsBump& ws, const r3dfs_episode_cfg_t* c, const EpisodeDims& d, int E, int in_dim,
                   int dg_k, EpisodeWs& w);
// everything after getFeatures (models/mpti.py:440-571); F rows [ppad, nn) = query features,
// [nn, nn + ns_pts) = support features
int episode_graph_half(const r3dfs_episode_cfg_t* cfg, const EpisodeDims& d, int E,
                       const EpisodeWs& w, const float* support_x, int64_t s_e, int64_t s_cloud,
                       int64_t s_c, int64_t s_n, const int32_t* support_y, const int64_t* query_y,
                       float* logits, float* loss, int32_t* pred, const r3dfs_episode_diag_t* diag,
                       cudaStream_t st, bool latency = false);
