"""numpy restatement of the support-shot contract of include/r3dfs.h ("Support shots from a labelled
scan") on top of the scene plan of tests/scene_oracle.py: per-block class counts, eligibility,
the seeded choice of blocks per way, and the shot clouds with their masks.  Counts and thresholds
are exact integers (the ratio product in float64), the clouds single float32 operations as the
chunk clouds, so the GPU results are compared with torch.equal."""
from __future__ import annotations

import numpy as np

from tests.scene_oracle import F32, lowbias32, plan


def blocks(points, n_points, block_size=1.0, overlap=1, seed=0):
    """-> (plan, block ids (n_seg,), members of every block in rank order (list of arrays))."""
    pl = plan(points, n_points, block_size, overlap, seed)
    P, B = pl["mem_point"], pl["mem_block"]
    key = lowbias32(P.astype(np.uint64) ^ lowbias32(int(seed) & 0xFFFFFFFF))
    srt = np.lexsort((key, B))                  # by (block, key): the plan's rank order
    ids, start, n_b = np.unique(B[srt], return_index=True, return_counts=True)
    members = [P[srt][s:s + n] for s, n in zip(start, n_b)]
    return pl, ids, members


def way_key(block_ids, seed, w):
    wk = lowbias32((int(lowbias32(int(seed) & 0xFFFFFFFF)) + w + 1) & 0xFFFFFFFF)
    return lowbias32(np.asarray(block_ids, np.uint64) ^ wk)


def normalise(pts, src):
    """(…, N) point indices -> (…, N, 9) clouds: xyz - min | rgb / 255 | (xyz - min) / max."""
    xyz = pts[src, 0:3]
    xyzp = xyz - xyz.min(-2, keepdims=True)
    e = xyzp.max(-2, keepdims=True)
    XYZ = np.where(e > 0, xyzp / np.where(e > 0, e, F32(1)), F32(0)).astype(F32)
    return np.concatenate([xyzp, pts[src, 3:6] / F32(255), XYZ], -1).astype(F32)


def support(points, labels, classes, k_shot, n_points, block_size=1.0, overlap=1, seed=0,
            min_points=100, min_ratio=0.05):
    """-> dict(support_x (n_way, k_shot, N, 9) float32 point-major, support_y / src
    (n_way, k_shot, N) int32, block (n_way, k_shot) int32, n_eligible (n_way,) int32,
    count (n_way, n_seg), threshold (n_seg,), block_ids (n_seg,))."""
    pts = np.asarray(points, dtype=F32)
    labels = np.asarray(labels)
    N, n_way = int(n_points), len(classes)
    _, ids, members = blocks(pts, N, block_size, overlap, seed)
    n_b = np.array([len(m) for m in members], np.int64)
    count = np.array([[int((labels[m] == c).sum()) for m in members] for c in classes], np.int64)
    thr = np.maximum(np.floor(n_b.astype(np.float64) * float(min_ratio)).astype(np.int64),
                     int(min_points))
    sx = np.zeros((n_way, k_shot, N, 9), F32)
    sy = np.zeros((n_way, k_shot, N), np.int32)
    src = np.full((n_way, k_shot, N), -1, np.int32)
    blk = np.full((n_way, k_shot), -1, np.int32)
    n_el = np.zeros(n_way, np.int32)
    for w, c in enumerate(classes):
        elig = np.nonzero(count[w] > thr)[0]
        n_el[w] = len(elig)
        chosen = elig[np.argsort(way_key(ids[elig], seed, w))][:k_shot]
        for j, s in enumerate(chosen):
            m = members[s]
            src[w, j] = m[np.arange(N) % min(len(m), N)]
            sx[w, j] = normalise(pts, src[w, j])
            sy[w, j] = labels[src[w, j]] == c
            blk[w, j] = ids[s]
    return dict(support_x=sx, support_y=sy, src=src, block=blk, n_eligible=n_el, count=count,
                threshold=thr, block_ids=ids)
