"""Deterministic synthetic S3DIS/ScanNet-shape few-shot episodes.

The real datasets are not available (no network), so bench/tests use clouds that follow
the reference's input contract (reference `dataloaders/loader.py:201-219` channel layout
`xyz-min | rgb/255 | xyz/max`, `:626,1692` dtypes, `:1662-1684` collate transposes that
leave the cloud point-major in memory) and its noise model for out-of-distribution shots
(`dataloaders/loader.py:669-680,797-810`: `round(k_shot*ratio)` shots per way are whole
clouds whose foreground object is a class outside the sampled ways, their ground-truth
masks are zero, and shot order is shuffled per way; `make_episode` also has the reference's
"sym", "pair" and "partial" noise types).
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional

import numpy as np
import torch

N_POINTS = 2048

# class pools: 6 test classes per S3DIS fold (reference dataloaders/s3dis.py:30),
# 10 per ScanNet fold (reference dataloaders/scannet.py:23)
CLASS_POOL = {"s3dis": 6, "scannet": 10}


def _class_style(cls: int):
    """Fixed per-class appearance: rgb, blob sigma (anisotropic) and height."""
    r = np.random.default_rng(1000 + int(cls))
    rgb = r.uniform(0.1, 0.9, size=3)
    sigma = r.uniform(0.08, 0.2, size=3)
    height = r.uniform(0.3, 2.2)
    return rgb, sigma, height


def make_cloud(rng: np.random.Generator, objects: List[int], n_pts: int = N_POINTS):
    """One block of `n_pts` points: floor/clutter background + one Gaussian blob per
    entry of `objects`.  Returns (pts (n_pts, 9) float32, cls (n_pts,) int64) with cls=-1
    for background, in a random point order."""
    n_obj = len(objects)
    fracs = rng.uniform(0.15, 0.35, size=n_obj) / max(1, n_obj) ** 0.5
    counts = np.maximum(1, (fracs * n_pts).astype(np.int64))
    n_bg = n_pts - int(counts.sum())
    xyz = []
    rgb = []
    cls = []
    # background: floor slab, a wall, and uniform clutter
    n_floor = n_bg // 2
    n_wall = n_bg // 4
    n_clut = n_bg - n_floor - n_wall
    floor = np.stack([rng.uniform(0, 1, n_floor), rng.uniform(0, 1, n_floor),
                      np.abs(rng.normal(0, 0.01, n_floor))], 1)
    wall = np.stack([rng.uniform(0, 1, n_wall), np.abs(rng.normal(0, 0.01, n_wall)),
                     rng.uniform(0, 3, n_wall)], 1)
    clut = np.stack([rng.uniform(0, 1, n_clut), rng.uniform(0, 1, n_clut),
                     rng.uniform(0, 3, n_clut)], 1)
    xyz += [floor, wall, clut]
    rgb += [np.tile([0.55, 0.5, 0.45], (n_floor, 1)), np.tile([0.8, 0.8, 0.75], (n_wall, 1)),
            rng.uniform(0.2, 0.8, size=(n_clut, 3))]
    cls += [np.full(n_bg, -1, np.int64)]
    for c, cnt in zip(objects, counts):
        col, sig, h = _class_style(c)
        ctr = np.array([rng.uniform(0.2, 0.8), rng.uniform(0.2, 0.8), h])
        p = ctr + rng.normal(0, 1, size=(cnt, 3)) * sig
        p[:, 0:2] = np.clip(p[:, 0:2], 0, 1)
        p[:, 2] = np.clip(p[:, 2], 0, 3)
        xyz.append(p)
        rgb.append(np.tile(col, (cnt, 1)))
        cls.append(np.full(cnt, int(c), np.int64))
    xyz = np.concatenate(xyz, 0)
    rgb = np.clip(np.concatenate(rgb, 0) + rng.normal(0, 0.05, size=(n_pts, 3)), 0, 1)
    cls = np.concatenate(cls, 0)
    perm = rng.permutation(n_pts)
    xyz, rgb, cls = xyz[perm], rgb[perm], cls[perm]
    xyz = xyz - xyz.min(0)
    XYZ = xyz / np.maximum(xyz.max(0), 1e-6)
    pts = np.concatenate([xyz, rgb, XYZ], 1).astype(np.float32)
    return pts, cls


def make_scene(seed: int, size_xy=(6.0, 4.0), points_per_m2: float = 10000.0,
               classes: Optional[List[int]] = None, dataset: str = "s3dis"):
    """A synthetic room scan in the style of `make_cloud`: floor, four walls, uniform clutter and
    Gaussian blobs of the given classes (default: two per class of the dataset's pool), with
    x y z in metres from an arbitrary origin and r g b in 0..255 (the S3DIS / ScanNet .npy
    convention).  Returns (points (M, 6) float32, cls (M,) int64 with -1 = background), in a random
    point order; M = round(points_per_m2 * area)."""
    rng = np.random.default_rng(seed)
    sx, sy = float(size_xy[0]), float(size_xy[1])
    M = int(round(points_per_m2 * sx * sy))
    if classes is None:
        classes = list(range(CLASS_POOL[dataset])) * 2
    n_obj = int(0.25 * M) // max(1, len(classes)) if classes else 0
    n_floor = int(0.4 * M)
    n_wall = int(0.2 * M)
    n_clut = M - n_floor - n_wall - n_obj * len(classes)
    xyz, rgb, cls = [], [], []
    xyz.append(np.stack([rng.uniform(0, sx, n_floor), rng.uniform(0, sy, n_floor),
                         np.abs(rng.normal(0, 0.01, n_floor))], 1))
    rgb.append(np.tile([0.55, 0.5, 0.45], (n_floor, 1)))
    # walls: a point on the perimeter, pushed a little into the room
    t = rng.uniform(0, 2 * (sx + sy), n_wall)
    d = np.abs(rng.normal(0, 0.01, n_wall))
    wx = np.where(t < sx, t, np.where(t < sx + sy, sx - d, np.where(t < 2 * sx + sy,
                                                                    2 * sx + sy - t, d)))
    wy = np.where(t < sx, d, np.where(t < sx + sy, t - sx, np.where(t < 2 * sx + sy, sy - d,
                                                                    2 * (sx + sy) - t)))
    xyz.append(np.stack([wx, wy, rng.uniform(0, 3, n_wall)], 1))
    rgb.append(np.tile([0.8, 0.8, 0.75], (n_wall, 1)))
    xyz.append(np.stack([rng.uniform(0, sx, n_clut), rng.uniform(0, sy, n_clut),
                         rng.uniform(0, 3, n_clut)], 1))
    rgb.append(rng.uniform(0.2, 0.8, size=(n_clut, 3)))
    cls.append(np.full(n_floor + n_wall + n_clut, -1, np.int64))
    for c in classes:
        col, sig, h = _class_style(c)
        ctr = np.array([rng.uniform(0.5, sx - 0.5), rng.uniform(0.5, sy - 0.5), h])
        p = ctr + rng.normal(0, 1, size=(n_obj, 3)) * sig
        p[:, 0] = np.clip(p[:, 0], 0, sx)
        p[:, 1] = np.clip(p[:, 1], 0, sy)
        p[:, 2] = np.clip(p[:, 2], 0, 3)
        xyz.append(p)
        rgb.append(np.tile(col, (n_obj, 1)))
        cls.append(np.full(n_obj, int(c), np.int64))
    xyz = np.concatenate(xyz, 0) + rng.uniform(-50, 50, size=3)   # arbitrary origin
    rgb = np.clip(np.concatenate(rgb, 0) + rng.normal(0, 0.05, size=(M, 3)), 0, 1) * 255.0
    cls = np.concatenate(cls, 0)
    perm = rng.permutation(M)
    pts = np.concatenate([xyz, rgb], 1)[perm].astype(np.float32)
    return pts, cls[perm]


@dataclasses.dataclass
class Episode:
    """Host-side episode, laid out like the reference's collate output
    (`dataloaders/loader.py:1676-1684`)."""
    support_x: torch.Tensor      # (n_way, k_shot, 9, N) fp32, point-major memory (transposed view)
    support_y: torch.Tensor      # (n_way, k_shot, N) int32 0/1
    query_x: torch.Tensor        # (n_way*n_queries, 9, N) fp32, transposed view
    query_y: torch.Tensor        # (n_way*n_queries, N) int64 in [0, n_way]
    gt_support_y: torch.Tensor   # (n_way, k_shot, N) int32
    sampled_classes: np.ndarray  # (n_way,) int32
    support_flag: torch.Tensor   # (n_way, k_shot) int32 absolute class of each shot

    def as_test_data(self):
        """The 7-entry list `MPTILearner_V3.test` unpacks (`models/mpti_learner.py:92`)."""
        z = torch.zeros_like(self.support_y)
        zq = torch.zeros(self.query_y.shape, dtype=torch.int32)
        return [self.support_x, self.support_y, self.query_x, self.query_y, z, zq, self.gt_support_y]


NOISE_TYPES = ("ood", "sym", "pair", "partial")


def default_pair_dict(dataset: str):
    """A fixed class -> noise-class pairing over the fold's test classes, in the spirit of the
    reference's `noise_pair_dict` (dataloaders/loader.py:592-593, 735): mostly a cyclic shift, with one
    class mapped to itself ("some pair noise don't have noisy class", :797)."""
    pool = CLASS_POOL[dataset]
    d = {c: (c + 1) % pool for c in range(pool)}
    d[pool - 1] = pool - 1
    return d


def make_episode(seed: int, n_way: int = 2, k_shot: int = 5, n_queries: int = 1,
                 dataset: str = "s3dis", noise_ratio=0.0,
                 n_pts: int = N_POINTS, noise_type: str = "ood", pair_dict=None) -> Episode:
    """Synthetic counterpart of `NoiseInMetaTest.generate_one_episode` (reference
    dataloaders/loader.py:648-890).  `round(k_shot * noise_ratio)` shots per way are noisy (a list of
    ratios means "draw one per episode", the reference's train mode, :668-670); their ground-truth
    masks are zero (:798-802), shots are shuffled per way (:806-810) and `support_flag` records every
    shot's absolute class (:730,795).  noise_type (:675-686,734-747):
      "ood"     — the noisy shot's foreground object is a test class outside the sampled ways;
      "sym"     — it is one of the OTHER sampled ways;
      "pair"    — it is `pair_dict[class of the way]` (may be the class itself);
      "partial" — the shot shows the way's own class, but the given mask also covers one object of
                  another class (`sample_pointcloud(partial_noise=True)`, :241-257).
    A noise class is dropped from a way's range once it has supplied `k_shot - n_noise - 1` shots
    (:790-793; the reference re-creates its counter inside the loop, so this fires only when that
    number is 1 — mirrored as executed)."""
    if noise_type not in NOISE_TYPES:
        raise ValueError(f"noise_type must be one of {NOISE_TYPES}")
    pool = CLASS_POOL[dataset]
    rng = np.random.default_rng(seed)
    sampled = rng.choice(pool, size=n_way, replace=False)
    others = [c for c in range(pool) if c not in sampled]
    if isinstance(noise_ratio, (list, tuple)):
        noise_ratio = float(rng.choice(np.asarray(noise_ratio, dtype=np.float64)))
    n_noise = int(round(k_shot * noise_ratio))
    if noise_type == "pair" and pair_dict is None:
        pair_dict = default_pair_dict(dataset)
    sx, sy, gy, flag = [], [], [], []
    qx, qy = [], []
    for w, c in enumerate(sampled):
        # query clouds: the way's class plus (sometimes) another sampled class
        for _ in range(n_queries):
            objs = [int(c)]
            if rng.uniform() < 0.5 and n_way > 1:
                objs.append(int(rng.choice([s for s in sampled if s != c])))
            if rng.uniform() < 0.3 and others:
                objs.append(int(rng.choice(others)))
            pts, cls = make_cloud(rng, objs, n_pts)
            lab = np.zeros(n_pts, np.int64)
            for i, s in enumerate(sampled):
                lab[cls == s] = i + 1
            qx.append(pts)
            qy.append(lab)
        wx, wy, wg, wf = [], [], [], []
        if noise_type == "sym" and n_way > 1:
            noise_range = [int(s_) for s_ in sampled if s_ != c]
        elif noise_type == "pair":
            noise_range = [int(pair_dict[int(c)])]
        elif noise_type == "partial":
            noise_range = [int(c)]
        else:
            noise_range = list(others)
        single_use = (k_shot - n_noise - 1) == 1 and noise_type in ("ood", "sym")
        for k in range(k_shot):
            noisy = k >= k_shot - n_noise
            extra_mask_cls = None
            if noisy and noise_range:
                fg_cls = int(rng.choice(noise_range))
                if single_use and len(noise_range) > 1:
                    noise_range.remove(fg_cls)
            else:
                fg_cls = int(rng.choice(others)) if (noisy and others) else int(c)
            objs = [fg_cls]
            if noisy and noise_type == "partial":
                # needs a second object of another class in the block (:754-763)
                extra_mask_cls = int(rng.choice([x for x in range(pool) if x != fg_cls]))
                objs.append(extra_mask_cls)
            elif rng.uniform() < 0.3 and others:
                extra = int(rng.choice(others))
                if extra != fg_cls:
                    objs.append(extra)
            pts, cls = make_cloud(rng, objs, n_pts)
            m = (cls == fg_cls)
            if extra_mask_cls is not None:
                m = m | (cls == extra_mask_cls)
            m = m.astype(np.int32)
            wx.append(pts)
            wy.append(m)
            wg.append(np.zeros_like(m) if noisy else m.copy())
            wf.append(fg_cls)
        order = rng.permutation(k_shot)
        sx.append(np.stack(wx)[order])
        sy.append(np.stack(wy)[order])
        gy.append(np.stack(wg)[order])
        flag.append(np.asarray(wf, np.int32)[order])
    support = np.stack(sx)            # (n_way, k_shot, N, 9)
    query = np.stack(qx)              # (n_way*n_queries, N, 9)
    return Episode(
        support_x=torch.from_numpy(support).transpose(2, 3),
        support_y=torch.from_numpy(np.stack(sy)),
        query_x=torch.from_numpy(query).transpose(1, 2),
        query_y=torch.from_numpy(np.stack(qy).astype(np.int64)),
        gt_support_y=torch.from_numpy(np.stack(gy)),
        sampled_classes=sampled.astype(np.int32),
        support_flag=torch.from_numpy(np.stack(flag)),
    )


def default_args(n_way: int = 2, k_shot: int = 5, n_queries: int = 1, **over):
    """The reference's flag defaults the model reads (`eval_noise.py:176-217`,
    `models/mpti.py:49-78`), as an argparse-like Namespace."""
    import argparse
    a = argparse.Namespace(
        n_way=n_way, k_shot=k_shot, n_queries=n_queries, pc_in_dim=9, pc_npts=N_POINTS,
        use_attention=True, n_subprototypes=100, k_connect=200, sigma=1.0,
        edgeconv_widths=[[64, 64], [64, 64], [64, 64]], dgcnn_mlp_widths=[512, 256],
        dgcnn_k=20, base_widths=[128, 64], output_dim=64, shot_seed=1,
        lr=1e-3, step_size=5000, gamma=0.5, model_checkpoint_path=None,
        pretrain_checkpoint_path=None)
    for k, v in over.items():
        setattr(a, k, v)
    return a
