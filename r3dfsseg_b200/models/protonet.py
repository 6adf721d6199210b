"""Prototypical network with noise suppression, eval path (reference models/protonet.py:357-945,
ProtoNet_Contrast: "protonet+CCNS+MDNS").

Same encoder, state-dict keys, `forward` signature and return arity as the reference.  In eval
(`train=False`) the episode — features, multi-scale degree-based noise suppression, masked average
pooling, one prototype per way from the kept shots plus a background prototype, cosine similarity
x 10 and the cross-entropy — is ONE call into libr3dfs.so (`r3dfs_protonet_forward`).  The
meta-training branch of this baseline (way-contrast on raw features, :410-489) is not built: the
training hot path of this repo is MPTI's (`r3dfsseg_b200.train`).
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from .attention import SelfAttention
from .dgcnn import DGCNN
from .mpti import BaseLearner, packed_weights


class ProtoNet_Contrast(nn.Module):
    def __init__(self, args):
        super().__init__()
        self.n_way = args.n_way
        self.k_shot = args.k_shot
        self.dist_method = args.dist_method
        self.in_channels = args.pc_in_dim
        self.n_points = args.pc_npts
        self.use_attention = args.use_attention
        if not self.use_attention:
            raise NotImplementedError("only use_attention=True is built")
        self.encoder = DGCNN(args.edgeconv_widths, args.dgcnn_mlp_widths, args.pc_in_dim,
                             k=args.dgcnn_k)
        self.base_learner = BaseLearner(args.dgcnn_mlp_widths[-1], args.base_widths)
        self.att_learner = SelfAttention(args.dgcnn_mlp_widths[-1], args.output_dim)
        self.feat_dim = 192
        self.proj = nn.Linear(self.feat_dim, 128)
        self.shot_level_clean_ratio = 0
        self.mdns = bool(getattr(args, "mdns", True))  # reference: always on in eval (:847)
        self._packed = None
        self._packed_sig = None
        self.clean_flag = None

    _weights = packed_weights

    def getFeatures(self, x):
        """(B, C_in, N) -> (B, 192, N)   (reference models/protonet.py:860-876)"""
        if self.training:
            raise NotImplementedError("ProtoNet_Contrast: eval path only; call .eval()")
        return ops.features(self._weights(), x)

    def forward_episodes(self, support_x, support_y, query_x, query_y=None, workspace=None):
        """Batch of E independent episodes (leading dim E on every tensor)."""
        if self.training:
            raise NotImplementedError("ProtoNet_Contrast: eval path only; call .eval()")
        cfg = ops.make_cfg(self.n_way, self.k_shot, query_x.shape[1], self.n_points, 100,
                           min(200, query_x.shape[1] * self.n_points - 1), 1.0, 0.99, self.mdns,
                           1, 1e-6)
        return ops.protonet_forward(self._weights(), cfg, support_x, support_y, query_x, query_y,
                                    dist_method=self.dist_method, workspace=workspace)

    def forward(self, support_x, support_y, query_x, query_y, gt_support_y=None, gt_query_y=None,
                train=False, logger=None, step=None, path=None, sampled_classes=None,
                bg_pcd_x=None, bg_pcd_y=None, support_c=None, support_flag=None, pcd_1024=None,
                label_1024=None, pcd_cutout=None, label_cutout=None):
        """train=False: (query_pred (n_queries, n_way+1, N), loss)  (reference :780-858)."""
        if train:
            raise NotImplementedError("ProtoNet_Contrast: the meta-training branch is not built")
        sx = support_x.reshape(self.n_way, self.k_shot, self.in_channels, self.n_points) \
            if support_x.dim() != 4 else support_x
        out = self.forward_episodes(sx.unsqueeze(0), support_y.unsqueeze(0), query_x.unsqueeze(0),
                                    query_y.unsqueeze(0))
        self.clean_flag = out["clean_flag"][0]
        if gt_support_y is not None and self.mdns:
            # shot-level clean ratio bookkeeping of the reference (:824-829), kept on the device
            gt_flag = (gt_support_y.sum(-1) > 0).float()
            self.shot_level_clean_ratio = self.shot_level_clean_ratio + \
                ((self.clean_flag * gt_flag).sum(-1) / self.clean_flag.sum(-1)).sum()
        return out["logits"][0].transpose(1, 2), out["loss"][0]

    def computeCrossEntropyLoss(self, query_logits, query_labels):
        return F.cross_entropy(query_logits, query_labels)
