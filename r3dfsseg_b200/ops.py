"""Operator layer: torch tensors in, libr3dfs.so (hand-written sm_100a CUDA) underneath.

Every function takes CUDA tensors, allocates outputs/workspace with torch (device memory and
streams are torch's job here, nothing else), and enqueues the C-ABI call on the current stream.
CPU tensors are rejected — there is no fallback path.  The main entry points are also registered
as torch custom ops in the `r3dfs::` namespace (CUDA implementation only).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import EpisodeCfg, EpisodeDiag, Weights, check

ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2


def _need_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("r3dfsseg_b200 ops run on CUDA tensors only (no CPU fallback); "
                               f"got a tensor on {t.device}")
        dev = t.device
    return dev


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _ws(nbytes: int, dev: torch.device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t if t.dtype == torch.float32 else t.float()


# ------------------------------------------------------------------------------------------------
# DGCNN pieces
# ------------------------------------------------------------------------------------------------
def knn(x: torch.Tensor, k: int, impl: int = 0) -> torch.Tensor:
    """reference models/dgcnn.py:17-23 — (B, C, N) -> (B, N, k) int64, self first.
    impl: 0 default (tcgen05 when C <= 64), 1 FP32 CUDA cores, 2 tensor cores."""
    dev = _need_cuda(x)
    x = _f32(x)
    B, Cc, N = x.shape
    L = _lib.lib()
    idx = torch.empty((B, N, k), dtype=torch.int64, device=dev)
    nb = L.r3dfs_knn_workspace(B, Cc, N, k)
    ws = _ws(nb, dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_knn_ex(_p(x), B, Cc, N, x.stride(0), x.stride(1), x.stride(2), k, _p(idx),
                             impl, _p(ws), ws.numel(), _stream()), "r3dfs_knn")
    return idx


def get_edge_feature(x: torch.Tensor, K: int = 20, idx: Optional[torch.Tensor] = None) -> torch.Tensor:
    """reference models/dgcnn.py:26-42 — (B, C, N) -> (B, 2C, N, K) = cat(x_j - x_i, x_i)."""
    dev = _need_cuda(x, idx)
    x = _f32(x)
    B, Cc, N = x.shape
    if idx is None:
        idx = knn(x, K)
    idx = idx.to(torch.int64).contiguous()
    out = torch.empty((B, 2 * Cc, N, K), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = None if x.stride(1) == 1 else _ws(L.r3dfs_edge_feature_workspace(B, Cc, N), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_edge_feature(_p(x), B, Cc, N, x.stride(0), x.stride(1), x.stride(2), _p(idx),
                                   K, _p(out), _p(ws), 0 if ws is None else ws.numel(), _stream()),
              "r3dfs_edge_feature")
    return out


get_graph_feature = get_edge_feature  # name used by BASELINE.json's north_star


def linear(x_pm: torch.Tensor, w: torch.Tensor, s: Optional[torch.Tensor], t: Optional[torch.Tensor],
           act: int, impl: int = 0) -> torch.Tensor:
    """Point-major 1x1 conv + folded BN + activation: (M, K) -> (M, Nout).
    impl: 0 default (tcgen05 3xTF32), 1 FP32 CUDA cores, 2 tensor cores."""
    dev = _need_cuda(x_pm, w, s, t)
    x_pm = _f32(x_pm).contiguous()
    w = _f32(w).contiguous()
    M, K = x_pm.shape
    Nout = w.shape[0]
    y = torch.empty((M, Nout), dtype=torch.float32, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        check(L.r3dfs_linear_ex(_p(x_pm), K, _p(w), _p(s), _p(t), act, M, K, Nout, _p(y), Nout,
                                impl, _stream()), "r3dfs_linear")
    return y


def edgeconv(x: torch.Tensor, w1: torch.Tensor, s1: torch.Tensor, t1: torch.Tensor,
             w2: torch.Tensor, s2: torch.Tensor, t2: torch.Tensor, k: int,
             return_idx: bool = False):
    """One fused EdgeConv block (models/dgcnn.py:115-118, eval BN).  (B, C, N) -> (B, 64, N)
    (a transposed view of the point-major (B, N, 64) result)."""
    dev = _need_cuda(x, w1, s1, t1, w2, s2, t2)
    x = _f32(x)
    B, Cc, N = x.shape
    y = torch.empty((B, N, 64), dtype=torch.float32, device=dev)
    idx = torch.empty((B, N, k), dtype=torch.int64, device=dev) if return_idx else None
    L = _lib.lib()
    ws = _ws(L.r3dfs_edgeconv_workspace(B, Cc, N, k), dev)
    w1 = _f32(w1).reshape(64, 2 * Cc).contiguous()
    w2 = _f32(w2).reshape(64, 64).contiguous()
    with torch.cuda.device(dev):
        check(L.r3dfs_edgeconv(_p(x), B, Cc, N, x.stride(0), x.stride(1), x.stride(2), k, _p(w1),
                               _p(s1), _p(t1), _p(w2), _p(s2), _p(t2), _p(y), _p(idx), _p(ws),
                               ws.numel(), _stream()), "r3dfs_edgeconv")
    out = y.transpose(1, 2)
    return (out, idx) if return_idx else out


def attention(x_pm: torch.Tensor, wqkv: torch.Tensor) -> torch.Tensor:
    """SelfAttention eval (models/attention.py:32-48): (B, N, Cin) point-major -> (B, N, 64)."""
    dev = _need_cuda(x_pm, wqkv)
    x_pm = _f32(x_pm).contiguous()
    wqkv = _f32(wqkv).contiguous()
    B, N, Cin = x_pm.shape
    y = torch.empty((B, N, 64), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = _ws(L.r3dfs_attention_workspace(B, N), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_attention(_p(x_pm), B, N, Cin, _p(wqkv), _p(y), _p(ws), ws.numel(),
                                _stream()), "r3dfs_attention")
    return y


# ------------------------------------------------------------------------------------------------
# packed eval weights
# ------------------------------------------------------------------------------------------------
def fold_bn(bn: torch.nn.modules.batchnorm._BatchNorm, conv_bias: Optional[torch.Tensor] = None):
    """BatchNorm (eval, running stats) -> per-channel (scale, shift); a conv bias ahead of the BN
    is absorbed into the shift."""
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    if conv_bias is not None:
        shift = shift + conv_bias.detach().float() * scale
    return scale.contiguous(), shift.contiguous()


class PackedWeights:
    """Device-resident fp32 tensors + the r3dfs_weights_t that points at them."""

    def __init__(self, model: torch.nn.Module):
        enc, bl, att = model.encoder, model.base_learner, model.att_learner
        dev = next(model.parameters()).device
        _need_cuda(next(model.parameters()))
        keep: List[torch.Tensor] = []

        def hold(t: torch.Tensor) -> int:
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        w = Weights()
        w.in_dim = int(enc.edge_convs[0].layer[0].weight.shape[1] // 2)
        w.dgcnn_k = int(enc.k)
        if len(enc.edge_convs) != 3:
            raise NotImplementedError("libr3dfs is built for 3 EdgeConv blocks of widths [64, 64]")
        for i, blk in enumerate(enc.edge_convs):
            c1, b1, c2, b2 = blk.layer[0], blk.layer[1], blk.layer[3], blk.layer[4]
            if tuple(c1.weight.shape[:1]) != (64,) or tuple(c2.weight.shape[:2]) != (64, 64):
                raise NotImplementedError("EdgeConv widths other than [64, 64] are not supported")
            s1, t1 = fold_bn(b1)
            s2, t2 = fold_bn(b2)
            w.ec_w1[i] = hold(c1.weight.reshape(64, -1))
            w.ec_s1[i], w.ec_t1[i] = hold(s1), hold(t1)
            w.ec_w2[i] = hold(c2.weight.reshape(64, 64))
            w.ec_s2[i], w.ec_t2[i] = hold(s2), hold(t2)
        m1, mb1, m2, mb2 = enc.conv.layer[0], enc.conv.layer[1], enc.conv.layer[3], enc.conv.layer[4]
        if tuple(m1.weight.shape[:2]) != (512, 192) or tuple(m2.weight.shape[:2]) != (256, 512):
            raise NotImplementedError("dgcnn_mlp_widths other than [512, 256] are not supported")
        for i, (cv, bn) in enumerate(((m1, mb1), (m2, mb2))):
            s, t = fold_bn(bn)
            w.mlp_w[i] = hold(cv.weight.reshape(cv.weight.shape[0], -1))
            w.mlp_s[i], w.mlp_t[i] = hold(s), hold(t)
        if len(bl.convs) != 2 or bl.convs[0][0].weight.shape[0] != 128 or bl.convs[1][0].weight.shape[0] != 64:
            raise NotImplementedError("base_widths other than [128, 64] are not supported")
        for i, seq in enumerate(bl.convs):
            cv, bn = seq[0], seq[1]
            s, t = fold_bn(bn, cv.bias)
            w.bl_w[i] = hold(cv.weight.reshape(cv.weight.shape[0], -1))
            w.bl_s[i], w.bl_t[i] = hold(s), hold(t)
        if att.q_map.weight.shape[0] != 64:
            raise NotImplementedError("output_dim other than 64 is not supported")
        wqkv = torch.cat([att.q_map.weight, att.k_map.weight, att.v_map.weight], 0)
        w.att_wqkv = hold(wqkv.reshape(192, -1))
        self.struct = w
        self.device = dev
        self._keep = keep
        self.tensors = keep  # the 31 packed tensors in r3dfs_weights_t order (see _weights_struct)


def features(pw: PackedWeights, x: torch.Tensor, want_level2: bool = False):
    """getFeatures (models/mpti.py:579-589): (B, in_dim, N) -> (B, 192, N) (transposed view of the
    point-major result); optionally also DGCNN's 256-channel output as (B, 256, N)."""
    dev = _need_cuda(x)
    x = _f32(x)
    B, Cin, N = x.shape
    if Cin != pw.struct.in_dim:
        raise ValueError(f"expected {pw.struct.in_dim} input channels, got {Cin}")
    feat = torch.empty((B, N, 192), dtype=torch.float32, device=dev)
    lvl2 = torch.empty((B, N, 256), dtype=torch.float32, device=dev) if want_level2 else None
    L = _lib.lib()
    ws = _ws(L.r3dfs_features_workspace(B, N), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_features(C.byref(pw.struct), _p(x), B, N, x.stride(0), x.stride(1),
                               x.stride(2), _p(feat), _p(lvl2), _p(ws), ws.numel(), _stream()),
              "r3dfs_features")
    if want_level2:
        return feat.transpose(1, 2), lvl2.transpose(1, 2)
    return feat.transpose(1, 2)


# ------------------------------------------------------------------------------------------------
# prototypes / graph
# ------------------------------------------------------------------------------------------------
FPS_AUTO, FPS_STREAM, FPS_Q8 = 0, 1, 2


def fps(feat: torch.Tensor, set_off: torch.Tensor, set_n: torch.Tensor, m_max: int,
        n_cap: Optional[int] = None, impl: int = FPS_AUTO) -> torch.Tensor:
    """Farthest point sampling from local index 0 for several sets at once -> (n_sets, m_max) int32.
    impl: FPS_STREAM re-reads the FP32 rows for every pick, FPS_Q8 (D = 192) keeps byte rows on chip
    and re-reads only the rows an exact bound cannot decide; same picks either way."""
    dev = _need_cuda(feat, set_off, set_n)
    feat = _f32(feat).contiguous()
    set_off = set_off.to(torch.int32).contiguous()
    set_n = set_n.to(torch.int32).contiguous()
    n_sets = set_off.numel()
    if n_cap is None:
        n_cap = int(feat.shape[0])
    out = torch.full((n_sets, m_max), -1, dtype=torch.int32, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        if impl == FPS_STREAM:
            check(L.r3dfs_fps(_p(feat), feat.shape[1], _p(set_off), _p(set_n), n_sets, n_cap, m_max,
                              _p(out), _stream()), "r3dfs_fps")
        else:
            ws = torch.empty(L.r3dfs_fps_workspace(feat.shape[0]), dtype=torch.uint8, device=dev)
            check(L.r3dfs_fps_ex(_p(feat), feat.shape[1], _p(set_off), _p(set_n), n_sets, n_cap,
                                 feat.shape[0], m_max, impl, _p(out), _p(ws), ws.numel(),
                                 _stream()), "r3dfs_fps_ex")
    return out


def mdns(support_x: torch.Tensor, support_y: torch.Tensor, support_feat: torch.Tensor,
         want_internals: bool = False):
    """Multi-scale degree-based noise suppression (models/mpti.py:87-223, 316-371).
    support_x (E, n_way, k_shot, 9, N) any strides, support_y (E, n_way, k_shot, N),
    support_feat (E, n_way*k_shot*N, 192) -> dict(keep (E, n_way, k_shot) int32, clean_flag float,
    cell_mean (E, n_way, k_shot, 5, 192), cell_count (..., 5) [, cell_mask (E, n_way, k_shot, N) u8,
    degree (E, n_way, 2, 4*k_shot), scale_flag (E, n_way, 2, k_shot)])."""
    dev = _need_cuda(support_x, support_y, support_feat)
    E, n_way, k_shot, Cin, N = support_x.shape
    sx = _f32(support_x)
    if sx.stride(1) != k_shot * sx.stride(2):
        sx = sx.contiguous()
    sy = support_y.to(torch.int32).contiguous()
    sf = _f32(support_feat).contiguous()
    Cn = n_way * k_shot
    out = dict(keep=torch.empty((E, n_way, k_shot), dtype=torch.int32, device=dev),
               clean_flag=torch.empty((E, n_way, k_shot), dtype=torch.float32, device=dev),
               cell_mean=torch.empty((E, n_way, k_shot, 5, 192), dtype=torch.float32, device=dev),
               cell_count=torch.empty((E, n_way, k_shot, 5), dtype=torch.int32, device=dev))
    if want_internals:
        out.update(cell_mask=torch.empty((E, n_way, k_shot, N), dtype=torch.uint8, device=dev),
                   degree=torch.empty((E, n_way, 2, 4 * k_shot), dtype=torch.float32, device=dev),
                   scale_flag=torch.empty((E, n_way, 2, k_shot), dtype=torch.float32, device=dev))
    L = _lib.lib()
    ws = _ws(L.r3dfs_mdns_workspace(E, n_way, k_shot), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_mdns(_p(sx), sx.stride(0), sx.stride(2), sx.stride(3), sx.stride(4), _p(sy),
                           _p(sf), E, n_way, k_shot, N, _p(out["cell_mean"]), _p(out["cell_count"]),
                           _p(out.get("cell_mask")), _p(out.get("degree")),
                           _p(out.get("scale_flag")), _p(out["keep"]), _p(out["clean_flag"]),
                           _p(ws), ws.numel(), _stream()), "r3dfs_mdns")
    return out


def multi_prototypes(feat: torch.Tensor, set_off: torch.Tensor, set_n: torch.Tensor, k: int):
    """getMutiplePrototypes (models/mpti.py:597-634) for several sets at once.
    Returns (prototypes (n_sets, k+1, D), counts (n_sets), assignments (rows), seeds (n_sets, k+1))."""
    dev = _need_cuda(feat, set_off, set_n)
    feat = _f32(feat).contiguous()
    set_off = set_off.to(torch.int32).contiguous()
    set_n = set_n.to(torch.int32).contiguous()
    n_sets = set_off.numel()
    rows, D = feat.shape
    proto = torch.zeros((n_sets, k + 1, D), dtype=torch.float32, device=dev)
    cnt = torch.zeros((n_sets,), dtype=torch.int32, device=dev)
    assign = torch.full((rows,), -1, dtype=torch.int32, device=dev)
    seeds = torch.full((n_sets, k + 1), -1, dtype=torch.int32, device=dev)
    L = _lib.lib()
    ws = _ws(L.r3dfs_multi_prototypes_workspace(rows, n_sets, k), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_multi_prototypes(_p(feat), D, _p(set_off), _p(set_n), n_sets, rows, k,
                                       _p(proto), _p(cnt), _p(assign), _p(seeds), _p(ws),
                                       ws.numel(), _stream()), "r3dfs_multi_prototypes")
    return proto, cnt, assign, seeds


def affinity_knn(node_feat: torch.Tensor, valid: torch.Tensor, k: int, sigma: float):
    """calculateLocalConstrainedAffinity (models/mpti.py:717-756), sparse: (G, n, D) ->
    nbr (G, n, k) int32, sim (G, n, k) fp32."""
    dev = _need_cuda(node_feat, valid)
    node_feat = _f32(node_feat).contiguous()
    valid = valid.to(torch.uint8).contiguous()
    G, n, D = node_feat.shape
    nbr = torch.zeros((G, n, k), dtype=torch.int32, device=dev)
    sim = torch.zeros((G, n, k), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = _ws(L.r3dfs_affinity_workspace(G, n, D, k), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_affinity_knn(_p(node_feat), _p(valid), G, n, D, k, float(sigma), _p(nbr),
                                   _p(sim), _p(ws), ws.numel(), _stream()), "r3dfs_affinity_knn")
    return nbr, sim


def label_propagate(nbr: torch.Tensor, sim: torch.Tensor, valid: torch.Tensor, Y: torch.Tensor,
                    alpha: float = 0.99, tol: float = 1e-6, max_iter: int = 200):
    """label_propagate (models/mpti.py:758-776) by sparse CG.  Returns (Z, iters, resid)."""
    dev = _need_cuda(nbr, sim, valid, Y)
    nbr = nbr.to(torch.int32).contiguous()
    sim = _f32(sim).contiguous()
    valid = valid.to(torch.uint8).contiguous()
    Y = _f32(Y).contiguous()
    G, n, k = nbr.shape
    nc = Y.shape[-1]
    Z = torch.empty((G, n, nc), dtype=torch.float32, device=dev)
    iters = torch.zeros((G,), dtype=torch.int32, device=dev)
    resid = torch.zeros((G,), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = _ws(L.r3dfs_label_propagate_workspace(G, n, k, nc), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_label_propagate(_p(nbr), _p(sim), _p(valid), G, n, k, _p(Y), nc, float(alpha),
                                      float(tol), int(max_iter), _p(Z), _p(iters), _p(resid),
                                      _p(ws), ws.numel(), _stream()), "r3dfs_label_propagate")
    return Z, iters, resid


def lp_cholesky(nbr: torch.Tensor, sim: torch.Tensor, valid: torch.Tensor, Y: torch.Tensor,
                alpha: float = 0.99):
    """The label-propagation system solved by a dense FP64 Cholesky factorisation on the GPU — the
    cross-check of `label_propagate`'s conjugate gradients.  Returns (Z fp32, info int32 (G))."""
    dev = _need_cuda(nbr, sim, valid, Y)
    nbr = nbr.to(torch.int32).contiguous()
    sim = _f32(sim).contiguous()
    valid = valid.to(torch.uint8).contiguous()
    Y = _f32(Y).contiguous()
    G, n, k = nbr.shape
    nc = Y.shape[-1]
    Z = torch.empty((G, n, nc), dtype=torch.float32, device=dev)
    info = torch.zeros((G,), dtype=torch.int32, device=dev)
    L = _lib.lib()
    ws = _ws(L.r3dfs_lp_cholesky_workspace(G, n, k, nc), dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_lp_cholesky(_p(nbr), _p(sim), _p(valid), G, n, k, _p(Y), nc, float(alpha),
                                  _p(Z), _p(info), _p(ws), ws.numel(), _stream()),
              "r3dfs_lp_cholesky")
    return Z, info


# ------------------------------------------------------------------------------------------------
# whole episodes
# ------------------------------------------------------------------------------------------------
def make_cfg(n_way: int, k_shot: int, n_query: int, n_points: int, n_subprototypes: int = 100,
             k_connect: int = 200, sigma: float = 1.0, alpha: float = 0.99, mdns: bool = True,
             cg_max_iter: int = 200, cg_tol: float = 1e-6) -> EpisodeCfg:
    return EpisodeCfg(n_way, k_shot, n_query, n_points, n_subprototypes, k_connect, float(sigma),
                      float(alpha), int(bool(mdns)), int(cg_max_iter), float(cg_tol))


def _envelope_error(cfg: EpisodeCfg) -> "_lib.R3dfsError":
    """What a workspace query of 0 means for an episode configuration."""
    return _lib.R3dfsError(
        "episode configuration outside what libr3dfs is built for: n_way 1..7, k_shot 1..32, "
        "n_points >= 64, n_subprototypes 1..127, k_connect 1..1024 and < n_queries * n_points, "
        "graph nodes = roundup64((n_way + 1) * (n_subprototypes + 1)) + n_queries * n_points <= 8192 "
        "(the merged rows index columns with 16 bits and the CG kernels stage 8192 nodes); got "
        f"n_way={cfg.n_way} k_shot={cfg.k_shot} n_query={cfg.n_query} n_points={cfg.n_points} "
        f"n_subprototypes={cfg.n_subprototypes} k_connect={cfg.k_connect}")


def _stage_event_array(stage_events: Optional[Sequence["torch.cuda.Event"]]):
    """Raw cudaEvent_t handles of caller-owned torch events (created by a first record())."""
    if stage_events is None:
        return None
    if len(stage_events) != len(_lib.STAGES):
        raise ValueError(f"need {len(_lib.STAGES)} stage events")
    return (C.c_void_p * len(stage_events))(*[int(e.cuda_event) for e in stage_events])


def _mpti_forward_raw(pw: Optional[PackedWeights], cfg: EpisodeCfg, support_x: torch.Tensor,
                 support_y: torch.Tensor, query_x: torch.Tensor, query_y: Optional[torch.Tensor],
                 want_diag: bool = False, workspace: Optional[torch.Tensor] = None,
                 support_feat: Optional[torch.Tensor] = None,
                 query_feat: Optional[torch.Tensor] = None,
                 stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """E episodes in one call.
    support_x (E, n_way, k_shot, C, N) any strides with uniform cloud stride; support_y
    (E, n_way, k_shot, N) int32; query_x (E, n_query, C, N); query_y (E, n_query, N) int64.
    Returns dict(logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N) int32 [, diag])."""
    dev = _need_cuda(support_x, support_y, query_x, query_y)
    support_x, query_x = _f32(support_x), _f32(query_x)
    E, n_way, k_shot, Cin, N = support_x.shape
    nq = query_x.shape[1]
    if (n_way, k_shot, nq, N) != (cfg.n_way, cfg.k_shot, cfg.n_query, cfg.n_points):
        raise ValueError("episode tensors do not match the episode configuration")
    if support_x.stride(1) != k_shot * support_x.stride(2):
        support_x = support_x.contiguous()
    support_y = support_y.to(torch.int32).contiguous()
    if query_y is not None:
        query_y = query_y.to(torch.int64).contiguous()
    nc = n_way + 1
    logits = torch.empty((E, nq, N, nc), dtype=torch.float32, device=dev)
    loss = torch.zeros((E,), dtype=torch.float32, device=dev)
    pred = torch.empty((E, nq, N), dtype=torch.int32, device=dev)
    L = _lib.lib()
    need = L.r3dfs_mpti_workspace(C.byref(cfg), E)
    if need == 0:
        raise _envelope_error(cfg)
    ws = workspace if workspace is not None and workspace.numel() >= need else _ws(need, dev)
    diag = None
    dstruct = None
    ev_arr = _stage_event_array(stage_events)
    if want_diag or ev_arr is not None:
        dstruct = EpisodeDiag(None, None, None, None, None)
    if want_diag:
        diag = {
            "proto_count": torch.zeros((E, nc), dtype=torch.int32, device=dev),
            "clean_flag": torch.ones((E, n_way, k_shot), dtype=torch.float32, device=dev),
            "cg_iters": torch.zeros((E,), dtype=torch.int32, device=dev),
            "cg_resid": torch.zeros((E,), dtype=torch.float32, device=dev),
        }
        dstruct.proto_count = diag["proto_count"].data_ptr()
        dstruct.clean_flag = diag["clean_flag"].data_ptr()
        dstruct.cg_iters = diag["cg_iters"].data_ptr()
        dstruct.cg_resid = diag["cg_resid"].data_ptr()
    if ev_arr is not None:
        dstruct.h_stage_events = C.cast(ev_arr, C.POINTER(C.c_void_p))
    if support_feat is not None:
        # precomputed features (point-major (E, rows, 192)): graph half only
        support_feat = _f32(support_feat).contiguous()
        query_feat = _f32(query_feat).contiguous()
        assert support_feat.shape == (E, n_way * k_shot * N, 192)
        assert query_feat.shape == (E, nq * N, 192)
        with torch.cuda.device(dev):
            check(L.r3dfs_mpti_forward_features(
                C.byref(cfg), E, _p(support_x), support_x.stride(0), support_x.stride(2),
                support_x.stride(3), support_x.stride(4), _p(support_y), _p(support_feat),
                _p(query_feat), _p(query_y), _p(logits), _p(loss), _p(pred),
                C.byref(dstruct) if dstruct is not None else None, _p(ws), ws.numel(), _stream()),
                "r3dfs_mpti_forward_features")
        out = {"logits": logits, "loss": loss, "pred": pred}
        if diag is not None:
            out["diag"] = diag
        return out
    with torch.cuda.device(dev):
        check(L.r3dfs_mpti_forward(
            C.byref(cfg), C.byref(pw.struct), E,
            _p(support_x), support_x.stride(0), support_x.stride(2), support_x.stride(3),
            support_x.stride(4), _p(support_y),
            _p(query_x), query_x.stride(0), query_x.stride(1), query_x.stride(2), query_x.stride(3),
            _p(query_y), _p(logits), _p(loss), _p(pred),
            C.byref(dstruct) if dstruct is not None else None, _p(ws), ws.numel(), _stream()),
            "r3dfs_mpti_forward")
    out = {"logits": logits, "loss": loss, "pred": pred}
    if diag is not None:
        out["diag"] = diag
    return out


def protonet_forward(pw: PackedWeights, cfg: EpisodeCfg, support_x: torch.Tensor,
                     support_y: torch.Tensor, query_x: torch.Tensor,
                     query_y: Optional[torch.Tensor], dist_method: str = "cosine",
                     workspace: Optional[torch.Tensor] = None):
    """E ProtoNet(+MDNS when cfg.mdns) episodes in one call (reference models/protonet.py:780-858).
    Tensors as `mpti_forward`.  Returns dict(logits (E, n_query, N, n_way+1), loss (E),
    pred (E, n_query, N) int32, clean_flag (E, n_way, k_shot))."""
    if dist_method != "cosine":
        # the reference's 'euclidean' branch reduces over the point axis and fails in the loss; any
        # other name (the scripts' default is 'gaussian') raises there too (models/protonet.py:933-939)
        raise NotImplementedError(
            "Error! Distance computation method (%s) is unknown!" % dist_method)
    dev = _need_cuda(support_x, support_y, query_x, query_y)
    support_x, query_x = _f32(support_x), _f32(query_x)
    E, n_way, k_shot, Cin, N = support_x.shape
    nq = query_x.shape[1]
    if (n_way, k_shot, nq, N) != (cfg.n_way, cfg.k_shot, cfg.n_query, cfg.n_points):
        raise ValueError("episode tensors do not match the episode configuration")
    if support_x.stride(1) != k_shot * support_x.stride(2):
        support_x = support_x.contiguous()
    support_y = support_y.to(torch.int32).contiguous()
    if query_y is not None:
        query_y = query_y.to(torch.int64).contiguous()
    nc = n_way + 1
    logits = torch.empty((E, nq, N, nc), dtype=torch.float32, device=dev)
    loss = torch.zeros((E,), dtype=torch.float32, device=dev)
    pred = torch.empty((E, nq, N), dtype=torch.int32, device=dev)
    clean = torch.ones((E, n_way, k_shot), dtype=torch.float32, device=dev)
    L = _lib.lib()
    need = L.r3dfs_mpti_workspace(C.byref(cfg), E)
    if need == 0:
        raise _envelope_error(cfg)
    ws = workspace if workspace is not None and workspace.numel() >= need else _ws(need, dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_protonet_forward(
            C.byref(cfg), C.byref(pw.struct), E,
            _p(support_x), support_x.stride(0), support_x.stride(2), support_x.stride(3),
            support_x.stride(4), _p(support_y),
            _p(query_x), query_x.stride(0), query_x.stride(1), query_x.stride(2), query_x.stride(3),
            _p(query_y), 0, _p(logits), _p(loss), _p(pred), _p(clean), _p(ws), ws.numel(),
            _stream()), "r3dfs_protonet_forward")
    return {"logits": logits, "loss": loss, "pred": pred, "clean_flag": clean}


def _mpti_support_raw(pw: PackedWeights, cfg: EpisodeCfg, support_x: torch.Tensor,
                      support_y: torch.Tensor, want_diag: bool = False,
                      stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """The support half of S episodes in one call (r3dfs_mpti_support).
    support_x (S, n_way, k_shot, C, N) any strides with uniform cloud stride, support_y
    (S, n_way, k_shot, N).  Returns (proto (S, n_way+1, n_subprototypes+1, 192), proto_count
    (S, n_way+1) int32, clean_flag (S, n_way, k_shot) or None without want_diag)."""
    dev = _need_cuda(support_x, support_y)
    support_x = _f32(support_x)
    S, n_way, k_shot, Cin, N = support_x.shape
    if (n_way, k_shot, N) != (cfg.n_way, cfg.k_shot, cfg.n_points):
        raise ValueError("support tensors do not match the episode configuration")
    if support_x.stride(1) != k_shot * support_x.stride(2):
        support_x = support_x.contiguous()
    support_y = support_y.to(torch.int32).contiguous()
    nc = n_way + 1
    proto = torch.empty((S, nc, cfg.n_subprototypes + 1, 192), dtype=torch.float32, device=dev)
    count = torch.empty((S, nc), dtype=torch.int32, device=dev)
    clean = torch.ones((S, n_way, k_shot), dtype=torch.float32, device=dev) if want_diag else None
    L = _lib.lib()
    need = L.r3dfs_mpti_support_workspace(C.byref(cfg), S)
    if need == 0:
        raise _envelope_error(cfg)
    ws = _ws(need, dev)
    ev_arr = _stage_event_array(stage_events)
    dstruct = None
    if want_diag or ev_arr is not None:
        dstruct = EpisodeDiag(None, None if clean is None else clean.data_ptr(), None, None, None)
        if ev_arr is not None:
            dstruct.h_stage_events = C.cast(ev_arr, C.POINTER(C.c_void_p))
    with torch.cuda.device(dev):
        check(L.r3dfs_mpti_support(
            C.byref(cfg), C.byref(pw.struct), S,
            _p(support_x), support_x.stride(0), support_x.stride(2), support_x.stride(3),
            support_x.stride(4), _p(support_y), _p(proto), _p(count),
            C.byref(dstruct) if dstruct is not None else None, _p(ws), ws.numel(), _stream()),
            "r3dfs_mpti_support")
    return proto, count, clean


def _mpti_query_raw(pw: PackedWeights, cfg: EpisodeCfg, proto: torch.Tensor,
                    proto_count: torch.Tensor, query_x: torch.Tensor,
                    query_y: Optional[torch.Tensor] = None, shared: bool = False,
                    want_diag: bool = False, workspace: Optional[torch.Tensor] = None,
                    stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """The query half of E episodes in one call (r3dfs_mpti_query) against the prototypes of
    `mpti_support`.  proto (S, n_way+1, n_subprototypes+1, 192), proto_count (S, n_way+1):
    S == E (episode i uses set i), or S == 1 with shared=True (every episode uses set 0, read in
    place).  query_x (E, n_query, C, N) any strides, query_y (E, n_query, N) or None.
    Returns dict(logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N) int32 [, diag
    (proto_count, cg_iters, cg_resid)])."""
    dev = _need_cuda(proto, proto_count, query_x, query_y)
    query_x = _f32(query_x)
    E, nq, Cin, N = query_x.shape
    nc, slot = cfg.n_way + 1, cfg.n_subprototypes + 1
    if (nq, N) != (cfg.n_query, cfg.n_points):
        raise ValueError("query tensors do not match the episode configuration")
    proto = _f32(proto).contiguous()
    proto_count = proto_count.to(torch.int32).contiguous()
    S = proto.shape[0]
    if tuple(proto.shape[1:]) != (nc, slot, 192) or tuple(proto_count.shape) != (S, nc):
        raise ValueError("prototypes do not match the episode configuration")
    if S != (1 if shared else E):
        raise ValueError(f"{S} prototype sets for {E} episodes (shared={shared})")
    p_e, c_e = (0, 0) if shared else (nc * slot * 192, nc)
    if query_y is not None:
        query_y = query_y.to(torch.int64).contiguous()
    logits = torch.empty((E, nq, N, nc), dtype=torch.float32, device=dev)
    loss = torch.zeros((E,), dtype=torch.float32, device=dev)
    pred = torch.empty((E, nq, N), dtype=torch.int32, device=dev)
    L = _lib.lib()
    need = L.r3dfs_mpti_query_workspace(C.byref(cfg), E)
    if need == 0:
        raise _envelope_error(cfg)
    ws = workspace if workspace is not None and workspace.numel() >= need else _ws(need, dev)
    ev_arr = _stage_event_array(stage_events)
    diag = dstruct = None
    if want_diag or ev_arr is not None:
        dstruct = EpisodeDiag(None, None, None, None, None)
    if want_diag:
        diag = {"proto_count": torch.zeros((E, nc), dtype=torch.int32, device=dev),
                "cg_iters": torch.zeros((E,), dtype=torch.int32, device=dev),
                "cg_resid": torch.zeros((E,), dtype=torch.float32, device=dev)}
        dstruct.proto_count = diag["proto_count"].data_ptr()
        dstruct.cg_iters = diag["cg_iters"].data_ptr()
        dstruct.cg_resid = diag["cg_resid"].data_ptr()
    if ev_arr is not None:
        dstruct.h_stage_events = C.cast(ev_arr, C.POINTER(C.c_void_p))
    with torch.cuda.device(dev):
        check(L.r3dfs_mpti_query(
            C.byref(cfg), C.byref(pw.struct), E, _p(proto), p_e, _p(proto_count), c_e,
            _p(query_x), query_x.stride(0), query_x.stride(1), query_x.stride(2), query_x.stride(3),
            _p(query_y), _p(logits), _p(loss), _p(pred),
            C.byref(dstruct) if dstruct is not None else None, _p(ws), ws.numel(), _stream()),
            "r3dfs_mpti_query")
    out = {"logits": logits, "loss": loss, "pred": pred}
    if diag is not None:
        out["diag"] = diag
    return out


# ------------------------------------------------------------------------------------------------
# whole scans (r3dfs_scene_*: blocks -> chunks of n_points -> query episodes -> merge)
# ------------------------------------------------------------------------------------------------
@dataclass
class ScenePlan:
    """One scan planned by r3dfs_scene_plan: the workspace holding its chunk layout (read by
    `scene_chunks` and `scene_merge`, which must get the same points), and the chunk count as a
    (1,) int64 device tensor (-1: an x or y coordinate is not finite, or the grid is too large)."""
    points: torch.Tensor
    workspace: torch.Tensor
    n_chunks: torch.Tensor
    overlap: int
    n_points: int


def scene_plan(points: torch.Tensor, n_points: int, block_size: float = 1.0, overlap: int = 1,
               seed: int = 0) -> ScenePlan:
    """Grid, block memberships and chunk layout of an (M, 6) scan (x y z in metres, r g b in
    0..255; any strides) for chunks of n_points points.  Enqueued only: nothing is read back."""
    dev = _need_cuda(points)
    points = _f32(points)
    if points.dim() != 2 or points.shape[1] != 6:
        raise ValueError(f"points must be (M, 6) = x y z r g b; got {tuple(points.shape)}")
    M = int(points.shape[0])
    L = _lib.lib()
    need = L.r3dfs_scene_workspace(M, int(overlap))
    if need == 0:
        raise _lib.R3dfsError(f"scene of {M} points at overlap {overlap} is outside what libr3dfs "
                              "is built for: overlap 1..4 and overlap^2 * M < 2^31")
    ws = _ws(need, dev)
    n_chunks = torch.empty((1,), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(L.r3dfs_scene_plan(_p(points), M, points.stride(0), points.stride(1),
                                 float(block_size), int(overlap), int(seed), int(n_points),
                                 _p(n_chunks), _p(ws), ws.numel(), _stream()), "r3dfs_scene_plan")
    return ScenePlan(points, ws, n_chunks, int(overlap), int(n_points))


def scene_chunks(plan: ScenePlan, n_chunks: int):
    """-> chunk_x (n_chunks, N, 9) point-major chunk clouds, chunk_src (n_chunks, N) int32 (the
    scan point of every slot).  n_chunks = the plan's count, read back by the caller."""
    pts = plan.points
    N = plan.n_points
    chunk_x = torch.empty((n_chunks, N, 9), dtype=torch.float32, device=pts.device)
    chunk_src = torch.empty((n_chunks, N), dtype=torch.int32, device=pts.device)
    L = _lib.lib()
    with torch.cuda.device(pts.device):
        check(L.r3dfs_scene_chunks(_p(pts), pts.shape[0], pts.stride(0), pts.stride(1),
                                   plan.overlap, N, int(n_chunks), _p(chunk_x), _p(chunk_src),
                                   _p(plan.workspace), plan.workspace.numel(), _stream()),
              "r3dfs_scene_chunks")
    return chunk_x, chunk_src


def scene_merge(plan: ScenePlan, logits: torch.Tensor, n_chunks: int):
    """Chunk logits (n_chunks, N, n_cls) -> dict(logits (M, n_cls) = mean over the blocks holding
    each point, pred (M,) int32, coverage (M,) int32 = number of those blocks)."""
    dev = _need_cuda(logits)
    logits = _f32(logits).contiguous()
    if tuple(logits.shape[:2]) != (n_chunks, plan.n_points) or logits.dim() != 3:
        raise ValueError(f"expected chunk logits ({n_chunks}, {plan.n_points}, n_cls); got "
                         f"{tuple(logits.shape)}")
    M, nc = int(plan.points.shape[0]), int(logits.shape[2])
    out = {"logits": torch.empty((M, nc), dtype=torch.float32, device=dev),
           "pred": torch.empty((M,), dtype=torch.int32, device=dev),
           "coverage": torch.empty((M,), dtype=torch.int32, device=dev)}
    L = _lib.lib()
    with torch.cuda.device(dev):
        check(L.r3dfs_scene_merge(_p(logits), M, plan.overlap, plan.n_points, int(n_chunks), nc,
                                  _p(out["logits"]), _p(out["pred"]), _p(out["coverage"]),
                                  _p(plan.workspace), plan.workspace.numel(), _stream()),
              "r3dfs_scene_merge")
    return out


def scene_support(plan: ScenePlan, labels: torch.Tensor, classes: Sequence[int], k_shot: int,
                  seed: int = 0, min_points: int = 100, min_ratio: float = 0.05):
    """Support shots of a labelled scan (r3dfs_scene_support): for every class, the k_shot blocks
    with the smallest seeded keys among those holding more than max(floor(n_b * min_ratio),
    min_points) of its points, each sampled to the plan's n_points and normalised as a chunk.
    `plan` must come from scene_plan with the same seed; labels (M,) int32 or int64 class ids.
    Enqueued only.  Returns dict(support_x (n_way, k_shot, 9, N), a view over point-major memory
    that encode_support takes as it is; support_y (n_way, k_shot, N) int32 masks; src
    (n_way, k_shot, N) int32 scan point of every slot; block (n_way, k_shot) int32 block id, -1 for
    a missing shot; n_eligible (n_way,) int32 device tensor, -1 when the plan found no valid grid)."""
    pts = plan.points
    dev = _need_cuda(labels)
    M, N = int(pts.shape[0]), plan.n_points
    if tuple(labels.shape) != (M,):
        raise ValueError(f"labels must be ({M},); got {tuple(labels.shape)}")
    labels = labels.to(torch.int32).contiguous()
    n_way, k_shot = len(classes), int(k_shot)
    L = _lib.lib()
    need = L.r3dfs_scene_support_workspace(n_way, k_shot)
    if need == 0:
        raise _lib.R3dfsError(f"{n_way} classes x {k_shot} shots is outside what libr3dfs is built "
                              "for: 1..7 classes, 1..32 shots")
    ws = _ws(need, dev)
    x = torch.empty((n_way, k_shot, N, 9), dtype=torch.float32, device=dev)
    out = {"support_x": x.transpose(2, 3),
           "support_y": torch.empty((n_way, k_shot, N), dtype=torch.int32, device=dev),
           "src": torch.empty((n_way, k_shot, N), dtype=torch.int32, device=dev),
           "block": torch.empty((n_way, k_shot), dtype=torch.int32, device=dev),
           "n_eligible": torch.empty((n_way,), dtype=torch.int32, device=dev)}
    h_cls = (C.c_int32 * n_way)(*[int(c) for c in classes])
    with torch.cuda.device(dev):
        check(L.r3dfs_scene_support(
            _p(pts), M, pts.stride(0), pts.stride(1), _p(labels), h_cls, n_way, k_shot,
            int(min_points), float(min_ratio), int(seed), plan.overlap, N, _p(x),
            _p(out["support_y"]), _p(out["src"]), _p(out["block"]), _p(out["n_eligible"]),
            _p(plan.workspace), plan.workspace.numel(), _p(ws), ws.numel(), _stream()),
            "r3dfs_scene_support")
    return out


def confusion_accumulate(pred: torch.Tensor, gt: torch.Tensor, class_slot: torch.Tensor,
                         counters: torch.Tensor) -> None:
    """evaluate_metric counters (eval_noise.py:35-62), accumulated in place into the (3, n_slots)
    int64 `counters`.  pred (E, P) int32, gt (E, P) int64, class_slot (E, n_way) int32."""
    dev = _need_cuda(pred, gt, class_slot, counters)
    pred = pred.to(torch.int32).contiguous().reshape(pred.shape[0], -1)
    gt = gt.to(torch.int64).contiguous().reshape(gt.shape[0], -1)
    class_slot = class_slot.to(torch.int32).contiguous()
    assert counters.dtype == torch.int64 and counters.is_contiguous() and counters.shape[0] == 3
    E, P = pred.shape
    L = _lib.lib()
    with torch.cuda.device(dev):
        check(L.r3dfs_confusion_accumulate(_p(pred), _p(gt), _p(class_slot), E, class_slot.shape[1],
                                           P, counters.shape[1], _p(counters), _stream()),
              "r3dfs_confusion_accumulate")


# ------------------------------------------------------------------------------------------------
# torch custom ops (CUDA implementation only — a CPU tensor has nowhere to go)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("r3dfs::knn", mutates_args=(), device_types="cuda")
def _knn_op(x: torch.Tensor, k: int) -> torch.Tensor:
    return knn(x, k)


@_knn_op.register_fake
def _(x, k):
    return x.new_empty((x.shape[0], x.shape[2], k), dtype=torch.int64)


@torch.library.custom_op("r3dfs::edge_feature", mutates_args=(), device_types="cuda")
def _edge_feature_op(x: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    return get_edge_feature(x, idx.shape[-1], idx)


@_edge_feature_op.register_fake
def _(x, idx):
    return x.new_empty((x.shape[0], 2 * x.shape[1], x.shape[2], idx.shape[-1]))


@torch.library.custom_op("r3dfs::edgeconv", mutates_args=(), device_types="cuda")
def _edgeconv_op(x: torch.Tensor, w1: torch.Tensor, s1: torch.Tensor, t1: torch.Tensor,
                 w2: torch.Tensor, s2: torch.Tensor, t2: torch.Tensor, k: int) -> torch.Tensor:
    """-> POINT-MAJOR (B, N, 64) (the kernel's layout; module code takes the transposed view)."""
    return edgeconv(x, w1, s1, t1, w2, s2, t2, k).transpose(1, 2)


@_edgeconv_op.register_fake
def _(x, w1, s1, t1, w2, s2, t2, k):
    return x.new_empty((x.shape[0], x.shape[2], 64))


@torch.library.custom_op("r3dfs::linear", mutates_args=(), device_types="cuda")
def _linear_op(x: torch.Tensor, w: torch.Tensor, s: Optional[torch.Tensor],
               t: Optional[torch.Tensor], act: int) -> torch.Tensor:
    return linear(x, w, s, t, act)


@_linear_op.register_fake
def _(x, w, s, t, act):
    return x.new_empty((x.shape[0], w.shape[0]))


@torch.library.custom_op("r3dfs::attention", mutates_args=(), device_types="cuda")
def _attention_op(x_pm: torch.Tensor, wqkv: torch.Tensor) -> torch.Tensor:
    return attention(x_pm, wqkv)


@_attention_op.register_fake
def _(x_pm, wqkv):
    return x_pm.new_empty((x_pm.shape[0], x_pm.shape[1], 64))


def _weights_struct(tensors: Sequence[torch.Tensor], in_dim: int, dgcnn_k: int) -> Weights:
    """r3dfs_weights_t over the 31 packed tensors in PackedWeights order."""
    if len(tensors) != 31:
        raise ValueError("expected the 31 packed weight tensors of PackedWeights")
    w = Weights()
    w.in_dim, w.dgcnn_k = int(in_dim), int(dgcnn_k)
    it = iter(int(t.data_ptr()) for t in tensors)
    for i in range(3):
        w.ec_w1[i], w.ec_s1[i], w.ec_t1[i] = next(it), next(it), next(it)
        w.ec_w2[i], w.ec_s2[i], w.ec_t2[i] = next(it), next(it), next(it)
    for i in range(2):
        w.mlp_w[i], w.mlp_s[i], w.mlp_t[i] = next(it), next(it), next(it)
    for i in range(2):
        w.bl_w[i], w.bl_s[i], w.bl_t[i] = next(it), next(it), next(it)
    w.att_wqkv = next(it)
    return w


class _WeightsView:
    """What `features` / `mpti_forward` need of a PackedWeights, rebuilt from tensors inside an op."""

    def __init__(self, tensors, in_dim, dgcnn_k):
        self.struct = _weights_struct(tensors, in_dim, dgcnn_k)
        self._keep = list(tensors)


@torch.library.custom_op("r3dfs::features", mutates_args=(), device_types="cuda")
def _features_op(x: torch.Tensor, weights: Sequence[torch.Tensor], in_dim: int,
                 dgcnn_k: int) -> torch.Tensor:
    """getFeatures -> POINT-MAJOR (B, N, 192)."""
    return features(_WeightsView(weights, in_dim, dgcnn_k), x).transpose(1, 2)


@_features_op.register_fake
def _(x, weights, in_dim, dgcnn_k):
    return x.new_empty((x.shape[0], x.shape[2], 192))


@torch.library.custom_op("r3dfs::fps", mutates_args=(), device_types="cuda")
def _fps_op(feat: torch.Tensor, set_off: torch.Tensor, set_n: torch.Tensor, m_max: int,
            n_cap: int, impl: int) -> torch.Tensor:
    return fps(feat, set_off, set_n, m_max, n_cap if n_cap > 0 else None, impl)


@_fps_op.register_fake
def _(feat, set_off, set_n, m_max, n_cap, impl):
    return feat.new_empty((set_off.numel(), m_max), dtype=torch.int32)


@torch.library.custom_op("r3dfs::multi_prototypes", mutates_args=(), device_types="cuda")
def _multi_prototypes_op(feat: torch.Tensor, set_off: torch.Tensor, set_n: torch.Tensor,
                         k: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    return multi_prototypes(feat, set_off, set_n, k)


@_multi_prototypes_op.register_fake
def _(feat, set_off, set_n, k):
    n = set_off.numel()
    i32 = dict(dtype=torch.int32)
    return (feat.new_empty((n, k + 1, feat.shape[1])), feat.new_empty((n,), **i32),
            feat.new_empty((feat.shape[0],), **i32), feat.new_empty((n, k + 1), **i32))


@torch.library.custom_op("r3dfs::mdns", mutates_args=(), device_types="cuda")
def _mdns_op(support_x: torch.Tensor, support_y: torch.Tensor, support_feat: torch.Tensor
             ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    o = mdns(support_x, support_y, support_feat)
    return o["keep"], o["clean_flag"], o["cell_mean"], o["cell_count"]


@_mdns_op.register_fake
def _(support_x, support_y, support_feat):
    E, nw, ks = support_x.shape[:3]
    return (support_x.new_empty((E, nw, ks), dtype=torch.int32), support_x.new_empty((E, nw, ks)),
            support_x.new_empty((E, nw, ks, 5, 192)),
            support_x.new_empty((E, nw, ks, 5), dtype=torch.int32))


@torch.library.custom_op("r3dfs::affinity_knn", mutates_args=(), device_types="cuda")
def _affinity_knn_op(node_feat: torch.Tensor, valid: torch.Tensor, k: int,
                     sigma: float) -> Tuple[torch.Tensor, torch.Tensor]:
    return affinity_knn(node_feat, valid, k, sigma)


@_affinity_knn_op.register_fake
def _(node_feat, valid, k, sigma):
    G, n = node_feat.shape[:2]
    return node_feat.new_empty((G, n, k), dtype=torch.int32), node_feat.new_empty((G, n, k))


@torch.library.custom_op("r3dfs::label_propagate", mutates_args=(), device_types="cuda")
def _label_propagate_op(nbr: torch.Tensor, sim: torch.Tensor, valid: torch.Tensor, Y: torch.Tensor,
                        alpha: float, tol: float, max_iter: int
                        ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    return label_propagate(nbr, sim, valid, Y, alpha, tol, max_iter)


@_label_propagate_op.register_fake
def _(nbr, sim, valid, Y, alpha, tol, max_iter):
    G = nbr.shape[0]
    return (sim.new_empty(Y.shape), sim.new_empty((G,), dtype=torch.int32), sim.new_empty((G,)))


@torch.library.custom_op("r3dfs::lp_cholesky", mutates_args=(), device_types="cuda")
def _lp_cholesky_op(nbr: torch.Tensor, sim: torch.Tensor, valid: torch.Tensor, Y: torch.Tensor,
                    alpha: float) -> Tuple[torch.Tensor, torch.Tensor]:
    return lp_cholesky(nbr, sim, valid, Y, alpha)


@_lp_cholesky_op.register_fake
def _(nbr, sim, valid, Y, alpha):
    return sim.new_empty(Y.shape), sim.new_empty((nbr.shape[0],), dtype=torch.int32)


@torch.library.custom_op("r3dfs::mpti_forward", mutates_args=("workspace",), device_types="cuda")
def _mpti_forward_op(weights: Sequence[torch.Tensor], in_dim: int, dgcnn_k: int,
                     support_x: torch.Tensor, support_y: torch.Tensor, query_x: torch.Tensor,
                     query_y: torch.Tensor, n_subprototypes: int, k_connect: int, sigma: float,
                     alpha: float, mdns: bool, cg_max_iter: int, cg_tol: float,
                     workspace: Optional[torch.Tensor]
                     ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor,
                                torch.Tensor, torch.Tensor, torch.Tensor]:
    """The whole episode batch (reference models/mpti.py:414-577, eval) as ONE op:
    -> (logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N) int32, proto_count (E, n_way+1)
    int32, clean_flag (E, n_way, k_shot), cg_iters (E) int32, cg_resid (E))."""
    E, n_way, k_shot, _, N = support_x.shape
    cfg = make_cfg(n_way, k_shot, query_x.shape[1], N, n_subprototypes, k_connect, sigma, alpha,
                   mdns, cg_max_iter, cg_tol)
    out = _mpti_forward_raw(_WeightsView(weights, in_dim, dgcnn_k), cfg, support_x, support_y,
                            query_x, query_y, want_diag=True, workspace=workspace)
    d = out["diag"]
    return (out["logits"], out["loss"], out["pred"], d["proto_count"], d["clean_flag"],
            d["cg_iters"], d["cg_resid"])


@_mpti_forward_op.register_fake
def _(weights, in_dim, dgcnn_k, support_x, support_y, query_x, query_y, n_subprototypes, k_connect,
      sigma, alpha, mdns, cg_max_iter, cg_tol, workspace):
    E, n_way, k_shot, _, N = support_x.shape
    nq = query_x.shape[1]
    f, i32 = support_x.new_empty, dict(dtype=torch.int32)
    return (f((E, nq, N, n_way + 1)), f((E,)), f((E, nq, N), **i32), f((E, n_way + 1), **i32),
            f((E, n_way, k_shot)), f((E,), **i32), f((E,)))


@torch.library.custom_op("r3dfs::mpti_support", mutates_args=(), device_types="cuda")
def _mpti_support_op(weights: Sequence[torch.Tensor], in_dim: int, dgcnn_k: int,
                     support_x: torch.Tensor, support_y: torch.Tensor, n_query: int,
                     n_subprototypes: int, k_connect: int, mdns: bool
                     ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Support half of S episodes (reference models/mpti.py:433-435, 440-493, eval) as ONE op:
    -> (proto (S, n_way+1, n_subprototypes+1, 192), proto_count (S, n_way+1) int32,
    clean_flag (S, n_way, k_shot)).  n_query / k_connect only enter the envelope check."""
    S, n_way, k_shot, _, N = support_x.shape
    cfg = make_cfg(n_way, k_shot, n_query, N, n_subprototypes, k_connect, mdns=mdns)
    return _mpti_support_raw(_WeightsView(weights, in_dim, dgcnn_k), cfg, support_x, support_y,
                             want_diag=True)


@_mpti_support_op.register_fake
def _(weights, in_dim, dgcnn_k, support_x, support_y, n_query, n_subprototypes, k_connect, mdns):
    S, n_way, k_shot, _, N = support_x.shape
    f = support_x.new_empty
    return (f((S, n_way + 1, n_subprototypes + 1, 192)), f((S, n_way + 1), dtype=torch.int32),
            f((S, n_way, k_shot)))


@torch.library.custom_op("r3dfs::mpti_query", mutates_args=("workspace",), device_types="cuda")
def _mpti_query_op(weights: Sequence[torch.Tensor], in_dim: int, dgcnn_k: int, proto: torch.Tensor,
                   proto_count: torch.Tensor, query_x: torch.Tensor,
                   query_y: Optional[torch.Tensor], shared: bool, k_shot: int, k_connect: int,
                   sigma: float, alpha: float, cg_max_iter: int, cg_tol: float,
                   workspace: Optional[torch.Tensor]
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """Query half of E episodes (reference models/mpti.py:436-437, 495-571, eval) against given
    prototypes as ONE op: -> (logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N)
    int32, cg_iters (E) int32, cg_resid (E)).  n_way and n_subprototypes come from proto's shape;
    k_shot (of the support set) only appears in error messages, the query half does not use it."""
    E, nq, _, N = query_x.shape
    n_way, n_sub = proto.shape[1] - 1, proto.shape[2] - 1
    cfg = make_cfg(n_way, k_shot, nq, N, n_sub, k_connect, sigma, alpha, False, cg_max_iter, cg_tol)
    out = _mpti_query_raw(_WeightsView(weights, in_dim, dgcnn_k), cfg, proto, proto_count, query_x,
                          query_y, shared, want_diag=True, workspace=workspace)
    d = out["diag"]
    return out["logits"], out["loss"], out["pred"], d["cg_iters"], d["cg_resid"]


@_mpti_query_op.register_fake
def _(weights, in_dim, dgcnn_k, proto, proto_count, query_x, query_y, shared, k_shot, k_connect,
      sigma, alpha, cg_max_iter, cg_tol, workspace):
    E, nq, _, N = query_x.shape
    f, i32 = query_x.new_empty, dict(dtype=torch.int32)
    return (f((E, nq, N, proto.shape[1])), f((E,)), f((E, nq, N), **i32), f((E,), **i32), f((E,)))


# the registered ops, for module code (traceable by torch.compile / fake tensors)
op = torch.ops.r3dfs


def mpti_forward(pw: Optional[PackedWeights], cfg: EpisodeCfg, support_x: torch.Tensor,
                 support_y: torch.Tensor, query_x: torch.Tensor, query_y: Optional[torch.Tensor],
                 want_diag: bool = False, workspace: Optional[torch.Tensor] = None,
                 support_feat: Optional[torch.Tensor] = None,
                 query_feat: Optional[torch.Tensor] = None,
                 stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """E episodes in one call (see _mpti_forward_raw).  The plain case goes through the registered
    op `r3dfs::mpti_forward`; stage events and precomputed features are eager-only diagnostics."""
    if stage_events is not None or support_feat is not None or query_y is None or pw is None:
        return _mpti_forward_raw(pw, cfg, support_x, support_y, query_x, query_y, want_diag,
                                 workspace, support_feat, query_feat, stage_events)
    r = op.mpti_forward(pw.tensors, pw.struct.in_dim, pw.struct.dgcnn_k, support_x, support_y,
                        query_x, query_y, cfg.n_subprototypes, cfg.k_connect, cfg.sigma, cfg.alpha,
                        bool(cfg.mdns), cfg.cg_max_iter, cfg.cg_tol, workspace)
    out = {"logits": r[0], "loss": r[1], "pred": r[2]}
    if want_diag:
        out["diag"] = {"proto_count": r[3], "clean_flag": r[4], "cg_iters": r[5], "cg_resid": r[6]}
    return out


def mpti_support(pw: PackedWeights, cfg: EpisodeCfg, support_x: torch.Tensor,
                 support_y: torch.Tensor, want_diag: bool = False,
                 stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """Support half of S episodes, encoded once (see _mpti_support_raw): -> (proto, proto_count,
    clean_flag or None).  The plain case goes through the registered op `r3dfs::mpti_support`."""
    if stage_events is not None:
        return _mpti_support_raw(pw, cfg, support_x, support_y, want_diag, stage_events)
    proto, count, clean = op.mpti_support(pw.tensors, pw.struct.in_dim, pw.struct.dgcnn_k,
                                          support_x, support_y, cfg.n_query, cfg.n_subprototypes,
                                          cfg.k_connect, bool(cfg.mdns))
    return proto, count, clean if want_diag else None


def mpti_query(pw: PackedWeights, cfg: EpisodeCfg, proto: torch.Tensor, proto_count: torch.Tensor,
               query_x: torch.Tensor, query_y: Optional[torch.Tensor] = None, shared: bool = False,
               want_diag: bool = False, workspace: Optional[torch.Tensor] = None,
               stage_events: Optional[Sequence["torch.cuda.Event"]] = None):
    """Query half of E episodes against given prototypes (see _mpti_query_raw); returns the dict
    of `mpti_forward`.  The plain case goes through the registered op `r3dfs::mpti_query`."""
    if stage_events is not None:
        return _mpti_query_raw(pw, cfg, proto, proto_count, query_x, query_y, shared, want_diag,
                               workspace, stage_events)
    if (proto.shape[1], proto.shape[2]) != (cfg.n_way + 1, cfg.n_subprototypes + 1):
        raise ValueError("prototypes do not match the episode configuration")
    r = op.mpti_query(pw.tensors, pw.struct.in_dim, pw.struct.dgcnn_k, proto, proto_count, query_x,
                      query_y, bool(shared), cfg.k_shot, cfg.k_connect, cfg.sigma, cfg.alpha,
                      cfg.cg_max_iter, cfg.cg_tol, workspace)
    out = {"logits": r[0], "loss": r[1], "pred": r[2]}
    if want_diag:
        out["diag"] = {"cg_iters": r[3], "cg_resid": r[4]}
    return out
