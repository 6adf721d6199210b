// internal launchers of lp.cu
#pragma once
#include "common.cuh"

// gmin: affinity_gmin_words(G, nn) u32 of scratch for the group minima that bound the select
int launch_affinity(const float* F, int64_t graph_rows, int64_t row_off, const uint8_t* valid,
                    int G, int nn, int D, int k, float sigma, float* norms, float* D2,
                    unsigned* gmin, int32_t* nbr, float* sim, cudaStream_t st,
                    const StageRec* sr = nullptr);
inline size_t affinity_gmin_words(size_t G, size_t nn) {
  return G * nn * (size_t)aff_gstride((int)nn);
}
int launch_label_propagate(const int32_t* nbr, float* sim, const uint8_t* valid, int G, int nn,
                           int k, const float* Y, int nc, float alpha, float tol, int max_iter,
                           int32_t* in_cnt, int32_t* in_ptr, int32_t* in_src, float* in_w,
                           float* dinv, int32_t* rowptr, int32_t* rowlen, int32_t* cursor,
                           uint16_t* mcol, float* mval, float* Z, float* X, float* R, float* P,
                           float* AP, int32_t* iters_out, float* resid_out, cudaStream_t st,
                           const StageRec* sr = nullptr, void* scratch = nullptr,
                           size_t scratch_bytes = 0, bool latency = false,
                           void* dense_scratch = nullptr, int32_t* dense_info = nullptr);
// dense_scratch (lp_cholesky_scratch_bytes(G, nn) bytes): solve by the dense FP64 Cholesky of
// lp_dense.cu instead of conjugate gradients (cross-check; dense_info[g] != 0: not positive definite)
size_t lp_cholesky_scratch_bytes(int G, int nn);
int launch_lp_cholesky_solve(const int32_t* rowptr, const int32_t* rowlen, const uint16_t* mcol,
                             const float* mval, const uint8_t* valid, int G, int nn, int k,
                             const float* Y, int nc, float alpha, float* Z, void* scratch,
                             int32_t* info_out, cudaStream_t st);
// scratch (optional): >= 6 * G * nn * ceil(nn / 32) bytes enables the sort-free in-edge build
int launch_lp_solve(const int32_t* rowptr, const int32_t* rowlen, const uint16_t* mcol,
                    const float* mval, const uint8_t* valid, int G, int nn, int k, const float* Y,
                    int nc, float alpha, float tol, int max_iter, float* Z, float* X, float* R,
                    float* P, float* AP, int32_t* iters_out, float* resid_out, cudaStream_t st,
                    bool latency = false, void* scratch = nullptr, size_t scratch_bytes = 0);
// Largest graph (nodes) the cluster CG solve of launch_lp_solve takes at n_cls classes (0 when n_cls
// is outside 1..8): 8192 for n_cls <= 4, 5376 for n_cls 5..8.
int lp_max_nodes(int n_cls);
// latency = true (a handful of graphs, e.g. the single episode of a training step): the whole GPU
// works on min(G, 4) graphs at a time with the matrix resident in shared memory (lp_cg_group_kernel);
// the default is one thread-block cluster per graph, which has the higher throughput on a batch.
// X, R, P, AP: (G, nn, 8) scratch; rowptr/rowlen: (G, nn); cursor: (G); mcol/mval: (G, 2*nn*k)
int launch_query_head(const float* Z, int G, int nn, int q_off, int nq, int nc, const int64_t* qy,
                      float* logits, float* loss, int32_t* pred, cudaStream_t st);
int launch_confusion(const int32_t* pred, const int64_t* gt, const int32_t* class_slot, int E,
                     int n_way, int64_t pts, int n_slots, int64_t* counters, cudaStream_t st);
