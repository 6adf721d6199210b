"""Multi-prototype transductive inference with the reference's module surface
(reference models/mpti.py:18-40 BaseLearner, :45-85 and :414-577 MPTI_SelfAtten).

`forward(support_x, support_y, query_x, query_y, ...)` keeps the reference's signature and return
arity; in eval mode the whole episode — features, multi-scale degree-based noise suppression,
FPS multi-prototypes, k-NN Gaussian affinity graph, label propagation, loss — is ONE call into
libr3dfs.so (`r3dfs_mpti_forward`), with no host synchronisation inside.  `forward_episodes`
runs a batch of independent episodes through the same call.  `encode_support` / `segment` split
that call in two, so that a labelled support set is encoded once and any number of query clouds
are segmented against it (`r3dfs_mpti_support` / `r3dfs_mpti_query`).  `segment_scene` labels a
whole scan against such a set, and `support_from_scene` cuts the support clouds out of a labelled
scan (`r3dfs_scene_*`).  State-dict keys are the reference's.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from .attention import SelfAttention
from .dgcnn import DGCNN


def _need_eval(m: nn.Module) -> None:
    if m.training:
        raise NotImplementedError("r3dfsseg_b200: stand-alone call in training mode; use "
                                  "forward(..., train=True) for the training step or .eval()")


def packed_weights(model: nn.Module) -> ops.PackedWeights:
    """The model's weights as the kernels read them, packed lazily in eager mode and packed again
    when the signature of its parameters and buffers changed: the storage and version counter of
    each, which change with any in-place update (optimizer step, load_state_dict, BatchNorm
    statistics).  model._packed_sig is the signature of the packed weights."""
    if torch.compiler.is_compiling():
        # tracing (torch.compile / export): the packed tensors are graph inputs, built beforehand
        if model._packed is None:
            raise RuntimeError("call model.pack_weights() once before tracing the module")
        return model._packed
    sig = tuple((t.data_ptr(), t._version) for t in model.state_dict(keep_vars=True).values())
    if model._packed is None or sig != model._packed_sig:
        model._packed = ops.PackedWeights(model)
        model._packed_sig = sig
    return model._packed


def _check_scan(points, block_size, overlap, seed) -> None:
    if not isinstance(points, torch.Tensor) or not points.is_cuda:
        raise ValueError("points must be a CUDA tensor")
    if points.dim() != 2 or points.shape[1] != 6 or points.shape[0] == 0:
        raise ValueError(f"points must be (M, 6) with M > 0; got {tuple(points.shape)}")
    if int(overlap) != overlap or not 1 <= overlap <= 4:
        raise ValueError(f"overlap must be an integer in 1..4; got {overlap}")
    if not float(block_size) > 0.0 or float(block_size) == float("inf"):
        raise ValueError(f"block_size must be a positive number of metres; got {block_size}")
    if int(seed) != seed or not 0 <= seed < 2 ** 32:
        raise ValueError(f"seed must be a uint32; got {seed}")


class BaseLearner(nn.Module):
    """Conv1d(bias) + BatchNorm1d stack, ReLU between layers (reference models/mpti.py:18-40)."""

    def __init__(self, in_channels, params):
        super().__init__()
        self.num_convs = len(params)
        self.convs = nn.ModuleList()
        width = in_channels
        for out_dim in params:
            self.convs.append(nn.Sequential(nn.Conv1d(width, out_dim, 1), nn.BatchNorm1d(out_dim)))
            width = out_dim

    def forward(self, x):
        _need_eval(self)
        B, _, N = x.shape
        h = x.transpose(1, 2).reshape(B * N, -1)
        for i, seq in enumerate(self.convs):
            s, t = ops.fold_bn(seq[1], seq[0].bias)
            act = ops.ACT_RELU if i != self.num_convs - 1 else ops.ACT_NONE
            h = ops.op.linear(h.contiguous(), seq[0].weight.reshape(seq[0].weight.shape[0], -1), s, t, act)
        return h.reshape(B, N, -1).transpose(1, 2)


@dataclass
class SupportSet:
    """What `MPTI_SelfAtten.encode_support` keeps of S support sets: the prototypes
    (S, n_way+1, n_subprototypes+1, 192) of classes [bg, way 0, ...] (rows past a set's count are
    zero), their counts proto_count (S, n_way+1) int32, the noise-suppression flags clean_flag
    (S, n_way, k_shot) (1 = shot kept; all ones without MDNS), the configuration they were built
    with, and the signature of the weights and BatchNorm statistics they were encoded under."""
    prototypes: torch.Tensor
    proto_count: torch.Tensor
    clean_flag: torch.Tensor
    n_way: int
    k_shot: int
    n_points: int
    n_subprototypes: int
    mdns: bool
    weights_sig: Tuple

    @property
    def n_sets(self) -> int:
        return int(self.prototypes.shape[0])


class MPTI_SelfAtten(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.n_way = args.n_way
        self.k_shot = args.k_shot
        self.in_channels = args.pc_in_dim
        self.n_points = args.pc_npts
        self.use_attention = args.use_attention
        self.n_subprototypes = args.n_subprototypes
        self.k_connect = args.k_connect
        self.sigma = args.sigma
        self.n_classes = self.n_way + 1
        if not self.use_attention:
            raise NotImplementedError("only use_attention=True is built (the reference's optimiser "
                                      "has no other branch, models/mpti_learner.py:26-32)")
        self.encoder = DGCNN(args.edgeconv_widths, args.dgcnn_mlp_widths, args.pc_in_dim,
                             k=args.dgcnn_k)
        self.base_learner = BaseLearner(args.dgcnn_mlp_widths[-1], args.base_widths)
        self.att_learner = SelfAttention(args.dgcnn_mlp_widths[-1], args.output_dim)
        self.feat_dim = args.edgeconv_widths[0][-1] + args.output_dim + args.base_widths[-1]
        self.shot_seed = getattr(args, "shot_seed", 1)
        self.proj = nn.Linear(self.feat_dim, 128)  # way-contrast head (train only)
        # label-propagation solver settings (the reference inverts the dense system instead)
        self.lp_alpha = 0.99
        self.cg_tol = float(getattr(args, "cg_tol", 1e-6))
        self.cg_max_iter = int(getattr(args, "cg_max_iter", 200))
        self._packed = None
        self._packed_sig = None
        self._last_diag = None
        self._flat_state = None       # training: parameters as views of one flat buffer
        self._train_ws = None
        self._train_step = 0

    # ---------------------------------------------------------------------------------------
    _weights = packed_weights

    def pack_weights(self) -> ops.PackedWeights:
        """Folds the BatchNorm statistics into per-channel scale/shift and packs the 31 weight
        tensors the kernels read (done lazily in eager mode; call it once before torch.compile)."""
        self._packed = None
        return self._weights()

    def _cfg(self, n_query: int, mdns: bool):
        return ops.make_cfg(self.n_way, self.k_shot, n_query, self.n_points, self.n_subprototypes,
                            self.k_connect, self.sigma, self.lp_alpha, mdns, self.cg_max_iter,
                            self.cg_tol)

    def getFeatures(self, x):
        """(B, C_in, N) -> (B, 192, N)   (reference models/mpti.py:579-589)"""
        _need_eval(self)
        pw = self._weights()
        return ops.op.features(x, pw.tensors, self.in_channels, int(self.encoder.k)).transpose(1, 2)

    # ---------------------------------------------------------------------------------------
    def forward_episodes(self, support_x, support_y, query_x, query_y=None, eval=True,
                         want_diag=False, workspace=None, support_feat=None, query_feat=None,
                         stage_events=None):
        """Batch of E independent episodes (leading dim E on every tensor).
        Returns dict(logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N)).
        With `support_feat` (E, n_way*k_shot*N, 192) / `query_feat` (E, n_query*N, 192) given,
        the encoder is skipped and only the graph half runs on those features."""
        _need_eval(self)
        if support_feat is None and stage_events is None and query_y is not None:
            # the registered op r3dfs::mpti_forward (traceable: torch.compile, fake tensors)
            pw = self._weights()
            r = ops.op.mpti_forward(pw.tensors, self.in_channels, int(self.encoder.k), support_x,
                                    support_y, query_x, query_y, self.n_subprototypes,
                                    self.k_connect, float(self.sigma), self.lp_alpha, bool(eval),
                                    self.cg_max_iter, self.cg_tol, workspace)
            out = {"logits": r[0], "loss": r[1], "pred": r[2]}
            if want_diag:
                out["diag"] = {"proto_count": r[3], "clean_flag": r[4], "cg_iters": r[5],
                               "cg_resid": r[6]}
            return out
        # eager only (ctypes structs): stage events, precomputed features, no query labels
        cfg = self._cfg(query_x.shape[1], mdns=bool(eval))
        if support_feat is not None:
            return ops.mpti_forward_features(cfg, support_x, support_y, support_feat, query_feat,
                                             query_y, want_diag, workspace, stage_events)
        return ops.mpti_forward(self._weights(), cfg, support_x, support_y, query_x, query_y,
                                want_diag, workspace, stage_events)

    # ---------------------------------------------------------------------------------------
    def encode_support(self, support_x, support_y, eval=True) -> SupportSet:
        """Support half of forward (models/mpti.py:433-435, 440-493), run once for a labelled
        support set: (n_way, k_shot, C, N) / (n_way, k_shot, N) for one set, or a leading S for
        S sets.  eval=True runs the noise suppression, exactly as forward(eval=True).  The result
        is handed to `segment` as often as wanted."""
        _need_eval(self)
        if support_x.dim() == 4:
            support_x, support_y = support_x.unsqueeze(0), support_y.unsqueeze(0)
        if support_x.dim() != 5 or support_y.dim() != 4:
            raise ValueError("support_x must be (n_way, k_shot, C, N) or (S, n_way, k_shot, C, N)")
        S, n_way, k_shot, _, N = support_x.shape
        if (n_way, N) != (self.n_way, self.n_points):
            raise ValueError(f"support set of {n_way} ways x {N} points for a model of "
                             f"{self.n_way} ways x {self.n_points} points")
        pw = self._weights()
        sig = None if torch.compiler.is_compiling() else self._packed_sig
        # the envelope is checked for one query cloud per way (the reference's episodes)
        proto, count, clean = ops.op.mpti_support(pw.tensors, self.in_channels, int(self.encoder.k),
                                                  support_x, support_y, n_way,
                                                  self.n_subprototypes, self.k_connect, bool(eval))
        return SupportSet(proto, count, clean, int(n_way), int(k_shot), int(N),
                          int(self.n_subprototypes), bool(eval), sig)

    def _check_support(self, support: SupportSet) -> None:
        _need_eval(self)
        if (support.n_way, support.n_points, support.n_subprototypes) != \
                (self.n_way, self.n_points, self.n_subprototypes):
            raise ValueError(
                f"support set built for n_way={support.n_way} n_points={support.n_points} "
                f"n_subprototypes={support.n_subprototypes}; the model has n_way={self.n_way} "
                f"n_points={self.n_points} n_subprototypes={self.n_subprototypes}")

    def _support_weights(self, support: SupportSet) -> ops.PackedWeights:
        """The packed weights, refused when they are not those `support` was encoded under."""
        pw = self._weights()
        if not torch.compiler.is_compiling() and self._packed_sig != support.weights_sig:
            raise RuntimeError("the weights or BatchNorm statistics changed after the support set "
                               "was encoded: its prototypes are stale, call encode_support again")
        return pw

    def _query(self, pw: ops.PackedWeights, support: SupportSet, query_x, query_y=None, sel=None):
        """The registered op r3dfs::mpti_query (traceable) of E query episodes against `support`:
        episode i against set i, against the one set (read in place), or against set sel[i]."""
        proto, count = support.prototypes, support.proto_count
        if sel is not None:
            proto, count = proto.index_select(0, sel), count.index_select(0, sel)
        return ops.op.mpti_query(pw.tensors, self.in_channels, int(self.encoder.k), proto, count,
                                 query_x, query_y, sel is None and support.n_sets == 1,
                                 support.k_shot, self.k_connect, float(self.sigma), self.lp_alpha,
                                 self.cg_max_iter, self.cg_tol, None)

    def segment(self, support: SupportSet, query_x, query_y=None,
                set_index: Optional[Sequence[int]] = None):
        """Query half of forward (models/mpti.py:436-437, 495-571) against an encoded support set.
        query_x (E, n_query, C, N) [query_y (E, n_query, N)]: episode i uses set i when the
        support holds E sets, the one set when it holds one (read in place), or set set_index[i].
        Returns dict(logits (E, n_query, N, n_way+1), loss (E), pred (E, n_query, N)), equal bit
        for bit to forward_episodes on the same supports.  A 3-D query_x (n_query, C, N) is one
        episode and returns what forward returns: (query_pred (n_query, n_way+1, N), loss)."""
        self._check_support(support)
        single = query_x.dim() == 3
        if single:
            query_x = query_x.unsqueeze(0)
            query_y = None if query_y is None else query_y.unsqueeze(0)
        E, S = query_x.shape[0], support.n_sets
        sel = None
        if set_index is not None:
            idx = [int(i) for i in set_index]
            if len(idx) != E or any(i < 0 or i >= S for i in idx):
                raise ValueError(f"set_index must hold {E} indices in [0, {S}); got {idx}")
            sel = torch.tensor(idx, dtype=torch.int64, device=support.prototypes.device)
        elif S != 1 and S != E:
            raise ValueError(f"{S} support sets for {E} query episodes: pass set_index")
        r = self._query(self._support_weights(support), support, query_x, query_y, sel)
        if single:
            return r[0][0].transpose(1, 2), r[1][0]
        return {"logits": r[0], "loss": r[1], "pred": r[2]}

    def segment_scene(self, support: SupportSet, points, block_size=1.0, overlap=1, seed=0,
                      chunk_batch=64):
        """Labels every point of a whole scan against one encoded support set.
        points: (M, 6) CUDA tensor, x y z in metres (any origin) and r g b in 0..255, the S3DIS /
        ScanNet .npy convention.  The scan is cut into xy blocks of block_size metres that overlap
        `overlap`-fold per axis (1..4), every block into chunks of n_points points normalised as the
        reference's loader normalises a block, the chunks are segmented `chunk_batch` at a time as
        1-query episodes against `support` (r3dfs_mpti_query), and each point's logits are averaged
        over the blocks that hold it.  `seed` picks which points share a chunk.  The contract,
        exact to the bit, is in include/r3dfs.h ("Segmenting a whole scan").
        Returns dict(logits (M, n_way+1), pred (M,) int32, coverage (M,) int32 = blocks holding the
        point, n_chunks).  Eager only: the chunk count depends on the data and is read back once.
        Results are reproducible for a given chunk_batch; another chunk_batch can change the
        logits in the last bits, as the query kernels round differently at another batch size."""
        self._check_support(support)
        if support.n_sets != 1:
            raise ValueError(f"a scene is segmented against one support set; got {support.n_sets}")
        _check_scan(points, block_size, overlap, seed)
        if int(chunk_batch) < 1 or chunk_batch > 65535:
            raise ValueError(f"chunk_batch must be in 1..65535; got {chunk_batch}")
        pw = self._support_weights(support)
        N, nc = self.n_points, self.n_classes
        plan = ops.scene_plan(points, N, float(block_size), int(overlap), int(seed))
        E = int(plan.n_chunks.item())
        if E < 0:
            raise ValueError("points hold a non-finite x or y coordinate, or the scan spans 2^31 "
                             "blocks or more")
        chunk_x, _ = ops.scene_chunks(plan, E)
        query_x = chunk_x.view(E, 1, N, 9).transpose(2, 3)   # (E, 1, 9, N), point-major memory
        logits = torch.empty((E, N, nc), dtype=torch.float32, device=points.device)
        B = int(chunk_batch)
        for b0 in range(0, E, B):
            logits[b0:b0 + B] = self._query(pw, support, query_x[b0:b0 + B])[0][:, 0]
        out = ops.scene_merge(plan, logits, E)
        out["n_chunks"] = E
        return out

    def support_from_scene(self, points, labels, classes, k_shot=None, block_size=1.0, overlap=1,
                           seed=0, min_points=100, min_ratio=0.05):
        """Cuts a support set out of a labelled scan, as the reference's loader builds support
        shots (class2scans + sample_pointcloud(support=True)).
        points: (M, 6) CUDA tensor as for segment_scene; labels: (M,) int32 or int64 CUDA tensor of
        class ids; classes: the model's n_way distinct class ids, one per way.  The scan is cut into
        the blocks segment_scene uses (block_size, overlap, seed); a block can serve class c when it
        holds more than max(floor(n_b * min_ratio), min_points) points of c.  Each way takes the
        k_shot such blocks with the smallest seeded keys and samples n_points of each, normalised
        as a chunk cloud; the mask is label == c.  The contract is in include/r3dfs.h ("Support
        shots from a labelled scan").
        Returns dict(support_x (n_way, k_shot, 9, N), support_y (n_way, k_shot, N) int32, src,
        block (n_way, k_shot), n_eligible (n_way,)) for encode_support(s["support_x"],
        s["support_y"]).  Shots of several scans combine with torch.cat along dim 1.  Raises
        ValueError when a class has fewer than k_shot eligible blocks.  Eager only: n_eligible is
        read back once."""
        k_shot = self.k_shot if k_shot is None else k_shot
        _check_scan(points, block_size, overlap, seed)
        if not isinstance(labels, torch.Tensor) or labels.device != points.device or \
                labels.dtype not in (torch.int32, torch.int64) or \
                tuple(labels.shape) != (points.shape[0],):
            raise ValueError(f"labels must be an int32 or int64 ({points.shape[0]},) tensor on "
                             f"{points.device}")
        classes = list(classes)
        if len(classes) != self.n_way or any(int(c) != c or not -2 ** 31 <= c < 2 ** 31
                                             for c in classes) or len(set(classes)) != len(classes):
            raise ValueError(f"classes must be {self.n_way} distinct int32 class ids; got {classes}")
        if int(k_shot) != k_shot or not 1 <= k_shot <= 32:
            raise ValueError(f"k_shot must be an integer in 1..32; got {k_shot}")
        if int(min_points) != min_points or not 0 <= min_points < 2 ** 31:
            raise ValueError(f"min_points must be a non-negative int32; got {min_points}")
        if not 0.0 <= float(min_ratio) <= 1.0:
            raise ValueError(f"min_ratio must be in [0, 1]; got {min_ratio}")
        plan = ops.scene_plan(points, self.n_points, float(block_size), int(overlap), int(seed))
        out = ops.scene_support(plan, labels, [int(c) for c in classes], int(k_shot), int(seed),
                                int(min_points), float(min_ratio))
        n_el = out["n_eligible"].tolist()
        if any(n < 0 for n in n_el):
            raise ValueError("points hold a non-finite x or y coordinate, or the scan spans 2^31 "
                             "blocks or more")
        short = [f"class {c}: {n} eligible blocks" for c, n in zip(classes, n_el) if n < k_shot]
        if short:
            raise ValueError(f"too few blocks for k_shot={k_shot} ({'; '.join(short)}); lower "
                             "min_points / min_ratio or k_shot, or add shots from another scan")
        return out

    def forward(self, support_x, support_y, query_x, query_y, gt_support_y=None, gt_query_y=None,
                train=False, logger=None, step=None, path=None, sampled_classes=None,
                bg_pcd_x=None, bg_pcd_y=None, support_c=None, support_flag=None, pcd_1024=None,
                label_1024=None, pcd_cutout=None, label_cutout=None, eval=False):
        """Same contract as reference models/mpti.py:414-577.
        train=False: returns (query_pred (n_query, n_way+1, N), lp_loss).
        train=True (module in .train() mode): returns the reference's 7-tuple (query_pred, lp_loss,
        contrast_loss, query_acc_LP, query_acc_original, clean_ratio_LP_avg,
        clean_ratio_original_avg); lp_loss / contrast_loss carry gradients to the parameters through
        r3dfs_mpti_train_backward.  The two clean-ratio entries are logging-only diagnostics in the
        reference (:514-552); both come from r3dfs_mpti_train_clean_ratio (NaN without gt_support_y)."""
        if train:
            if not self.training:
                raise RuntimeError("forward(train=True) needs the module in .train() mode "
                                   "(reference models/mpti_learner.py:61)")
            if support_flag is None:
                raise ValueError("forward(train=True) needs support_flag (way-contrast labels)")
            from ..train import train_episode
            query_pred, lp_loss, contrast = train_episode(self, support_x, support_y, query_x,
                                                          query_y, support_flag)
            with torch.no_grad():
                pl = query_pred.argmax(1)
                gq = gt_query_y if gt_query_y is not None else query_y
                denom = float(self.n_way * self.n_points)
                acc_lp = (pl == gq).sum().float() / denom
                acc_orig = (query_y == gq).sum().float() / denom
                ratio_lp = ratio_orig = torch.full((), float("nan"), device=query_pred.device)
                if gt_support_y is not None:  # models/mpti.py:514-552 (logging-only diagnostics)
                    from ..train import clean_ratios
                    ratio_lp, ratio_orig = clean_ratios(self, support_y, gt_support_y)
            return query_pred, lp_loss, contrast, acc_lp, acc_orig, ratio_lp, ratio_orig
        if self.training:
            raise RuntimeError("call forward(..., train=True) in training mode, or .eval() first")
        sx = support_x.reshape(self.n_way, self.k_shot, self.in_channels, self.n_points) \
            if support_x.dim() != 4 else support_x
        out = self.forward_episodes(sx.unsqueeze(0), support_y.unsqueeze(0), query_x.unsqueeze(0),
                                    query_y.unsqueeze(0), eval=eval, want_diag=True)
        self._last_diag = out["diag"]
        query_pred = out["logits"][0].transpose(1, 2)
        return query_pred, out["loss"][0]

    # the reference sets these as plain attributes inside forward; reading them here syncs
    @property
    def num_prototypes(self) -> Optional[int]:
        return None if self._last_diag is None else int(self._last_diag["proto_count"][0].sum())

    @property
    def num_nodes(self) -> Optional[int]:
        p = self.num_prototypes
        return None if p is None else p + self.n_way * self.n_points

    def computeCrossEntropyLoss(self, query_logits, query_labels):
        return F.cross_entropy(query_logits, query_labels)
