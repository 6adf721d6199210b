"""numpy restatement of the dataset index and the episode sampler of include/r3dfs.h ("Few-shot
episodes from labelled scans") on top of the scene plan (tests/scene_oracle.py) and the shot
clouds (tests/scene_support_oracle.py).  Keys are exact uint32 integers, counts and thresholds
exact (the ratio product in float64) and clouds single float32 operations, so the GPU results are
compared with torch.equal."""
from __future__ import annotations

import numpy as np

from tests.scene_oracle import F32, lowbias32
from tests.scene_support_oracle import blocks, normalise

NOISE = {None: 0, "ood": 1, "sym": 2, "pair": 3}


def H(a, b):
    return int(lowbias32(int(a) ^ int(lowbias32(int(b) & 0xFFFFFFFF))))


def index(scans, classes, n_points, block_size=1.0, overlap=1, seed=0, min_points=100,
          min_ratio=0.05):
    """scans: list of (points (M_i, 6), labels (M_i,)).  -> dict(points, labels (the concatenation),
    block_off, block_scan, block_id, member, count, elig (list of arrays per class), elig_off,
    elig_block)."""
    pts = np.concatenate([np.asarray(p, F32) for p, _ in scans]).astype(F32)
    lab = np.concatenate([np.asarray(l_, np.int64) for _, l_ in scans])
    off, bscan, bid, mem = [0], [], [], []
    base = 0
    for i, (p, _) in enumerate(scans):
        _, ids, members = blocks(np.asarray(p, F32), n_points, block_size, overlap, seed)
        for b, m in zip(ids, members):
            off.append(off[-1] + len(m))
            bscan.append(i)
            bid.append(int(b))
            mem.append(m + base)
        base += len(p)
    member = np.concatenate(mem).astype(np.int32)
    off = np.asarray(off, np.int64)
    n_b = np.diff(off)
    count = np.array([[int((lab[member[off[b]:off[b + 1]]] == c).sum()) for c in classes]
                      for b in range(len(n_b))], np.int64).reshape(len(n_b), len(classes))
    thr = np.maximum(np.floor(n_b.astype(np.float64) * float(min_ratio)).astype(np.int64),
                     int(min_points))
    elig = [np.nonzero(count[:, k] > thr)[0].astype(np.int32) for k in range(len(classes))]
    elig_off = np.concatenate([[0], np.cumsum([len(e) for e in elig])]).astype(np.int32)
    return dict(points=pts, labels=lab, classes=list(classes), block_off=off,
                block_scan=np.asarray(bscan, np.int32), block_id=np.asarray(bid, np.int32),
                member=member, count=count.astype(np.int32), threshold=thr, elig=elig,
                elig_off=elig_off, elig_block=np.concatenate(elig).astype(np.int32))


def _ranked(blocks_, key):
    return blocks_[np.argsort(lowbias32(blocks_.astype(np.uint64) ^ key), kind="stable")]


def _cloud(ix, b, N):
    m = ix["member"][ix["block_off"][b]:ix["block_off"][b + 1]]
    src = m[np.arange(N) % min(len(m), N)]
    return src, normalise(ix["points"], src)


def episodes(ix, way_classes, n_noise, noise_type, k_shot, n_queries, n_points, seed=0, first=0,
             step=1, pair=None):
    """way_classes (E, n_way) class ids; n_noise (E,); pair (n_cls) class ids or None.  -> the
    outputs of r3dfs_scene_episodes as numpy arrays, plus noisy (E, n_way, k_shot)."""
    classes = ix["classes"]
    at = {c: k for k, c in enumerate(classes)}
    wc = np.asarray(way_classes, np.int64).reshape(len(n_noise), -1)
    E, n_way = wc.shape
    N = int(n_points)
    nq = n_way * n_queries
    elig = ix["elig"]
    out = dict(support_x=np.zeros((E, n_way, k_shot, N, 9), F32),
               support_y=np.zeros((E, n_way, k_shot, N), np.int32),
               gt_support_y=np.zeros((E, n_way, k_shot, N), np.int32),
               support_flag=np.zeros((E, n_way, k_shot), np.int32),
               query_x=np.zeros((E, nq, N, 9), F32), query_y=np.zeros((E, nq, N), np.int64),
               shot_block=np.zeros((E, n_way, k_shot), np.int32),
               query_block=np.zeros((E, nq), np.int32),
               support_src=np.zeros((E, n_way, k_shot, N), np.int32),
               query_src=np.zeros((E, nq, N), np.int32), noisy=np.zeros((E, n_way, k_shot), bool))
    lab = ix["labels"]
    for e in range(E):
        g = (first + e * step) & 0xFFFFFFFF
        ke = H(int(lowbias32(int(seed) & 0xFFFFFFFF)), g)
        ways = [at[int(c)] for c in wc[e]]
        nn = int(n_noise[e])
        kc = k_shot - nn
        for w, c in enumerate(ways):
            kw = H(ke, w + 1)
            ranked = _ranked(elig[c], kw)
            clean, queries = ranked[:kc], ranked[kc:kc + n_queries]
            if noise_type == "ood":
                R = [k for k in range(len(classes)) if len(elig[k]) and k not in ways]
            elif noise_type == "sym":
                R = [ways[v] for v in range(n_way) if v != w]
            elif noise_type == "pair":
                R = [at[int(pair[c])]]
            else:
                R = []
            single = kc - 1 == 1 and noise_type in ("ood", "sym")
            if single and R:
                pi = np.argsort(lowbias32(np.arange(len(R), dtype=np.uint64) ^ H(kw, 33)),
                                kind="stable")
            ncls, nblk = [], []
            for j in range(nn):
                if single:
                    k = R[pi[min(j, len(R) - 1)]]
                else:
                    k = R[(H(kw, 64 + j) * len(R)) >> 32]
                ncls.append(k)
                nblk.append(int(_ranked(elig[k], H(kw, 128 + j))[0]))
            pre_b = [int(b) for b in clean] + nblk
            pre_c = [c] * kc + ncls
            okey = lowbias32(np.arange(k_shot, dtype=np.uint64) ^ H(kw, 34))
            slot = np.argsort(np.argsort(okey, kind="stable"), kind="stable")
            for t in range(k_shot):
                s = slot[t]
                b, cid = pre_b[t], classes[pre_c[t]]
                src, x = _cloud(ix, b, N)
                y = (lab[src] == cid).astype(np.int32)
                out["shot_block"][e, w, s] = b
                out["support_flag"][e, w, s] = cid
                out["noisy"][e, w, s] = t >= kc
                out["support_src"][e, w, s] = src
                out["support_x"][e, w, s] = x
                out["support_y"][e, w, s] = y
                out["gt_support_y"][e, w, s] = 0 if t >= kc else y
            for q, b in enumerate(queries):
                i = w * n_queries + q
                src, x = _cloud(ix, int(b), N)
                out["query_block"][e, i] = b
                out["query_src"][e, i] = src
                out["query_x"][e, i] = x
                y = np.zeros(N, np.int64)
                for v in range(n_way - 1, -1, -1):
                    y[lab[src] == classes[ways[v]]] = v + 1
                out["query_y"][e, i] = y
    return out
