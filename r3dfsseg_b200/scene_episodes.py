"""Few-shot episodes sampled on the GPU from labelled scans, as the reference's
`NoiseInMetaTest.generate_one_episode` (dataloaders/loader.py:648-890) draws them from the blocks
of many rooms: per way, support and query blocks from the class's `class2scans` list, n_points
sampled and normalised per block, query labels remapped to 0..n_way, and round(k_shot * ratio)
noisy shots per way (ood, sym or pair noise), shuffled.

The sampler defines its own seeded contract (include/r3dfs.h, "Few-shot episodes from labelled
scans") instead of numpy's random stream: the same distributions, reproducible bit for bit, and
episode g is the same whichever batch it is sampled in.  Not covered: `partial` noise, the
reference's train-time augmentation (pc_augm), and reading dataset folders from disk.
"""
from __future__ import annotations

import itertools
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops

NOISE_TYPES = (None, "ood", "sym", "pair")


def _lowbias32(x: int) -> int:
    x &= 0xFFFFFFFF
    x ^= x >> 16
    x = (x * 0x7FEB352D) & 0xFFFFFFFF
    x ^= x >> 15
    x = (x * 0x846CA68B) & 0xFFFFFFFF
    return x ^ (x >> 16)


def _hkey(a: int, b: int) -> int:
    return _lowbias32(a ^ _lowbias32(b))


def episode_key(seed: int, g: int) -> int:
    """K_e of include/r3dfs.h: the key of episode index g."""
    return _hkey(_lowbias32(seed), g)


class SceneEpisodes:
    """A dataset of labelled scans, indexed once on the GPU, from which batches of episodes are
    sampled without leaving the device.

    scans      list of (points (M_i, 6), labels (M_i,)) CUDA tensors: x y z in metres, r g b in
               0..255 (the S3DIS / ScanNet .npy convention), int32 or int64 class ids
    classes    the fold's classes (1..64 distinct ids); other labels count for no class
    n_points, block_size, overlap, seed
               every scan is cut into the blocks of `segment_scene` (r3dfs_scene_plan); a block's
               cloud holds n_points of its points
    min_points, min_ratio
               a block serves class c when it holds more than max(floor(n_b * min_ratio),
               min_points) points of c (the reference's class2scans rule)

    `n_eligible` holds the size of every class's class2scans list."""

    def __init__(self, scans: Sequence[Tuple[torch.Tensor, torch.Tensor]], classes: Sequence[int],
                 n_points: int = 2048, block_size: float = 1.0, overlap: int = 1, seed: int = 0,
                 min_points: int = 100, min_ratio: float = 0.05):
        from .models.mpti import _check_scan
        if not scans:
            raise ValueError("scans must hold at least one (points, labels) pair")
        classes = [int(c) for c in classes]
        if not 1 <= len(classes) <= 64 or len(set(classes)) != len(classes) or \
                any(not -2 ** 31 <= c < 2 ** 31 for c in classes):
            raise ValueError(f"classes must be 1..64 distinct int32 ids; got {classes}")
        if int(n_points) != n_points or not 64 <= n_points <= 65536:
            raise ValueError(f"n_points must be in 64..65536; got {n_points}")
        if int(min_points) != min_points or not 0 <= min_points < 2 ** 31:
            raise ValueError(f"min_points must be a non-negative int32; got {min_points}")
        if not 0.0 <= float(min_ratio) <= 1.0:
            raise ValueError(f"min_ratio must be in [0, 1]; got {min_ratio}")
        for i, (p, lab) in enumerate(scans):
            _check_scan(p, block_size, overlap, seed)
            if not isinstance(lab, torch.Tensor) or lab.device != p.device or \
                    lab.dtype not in (torch.int32, torch.int64) or tuple(lab.shape) != (p.shape[0],):
                raise ValueError(f"labels of scan {i} must be an int32 or int64 ({p.shape[0]},) "
                                 f"tensor on {p.device}")
        self.classes = classes
        self.n_points, self.seed = int(n_points), int(seed)
        self.points = torch.cat([ops._f32(p) for p, _ in scans]).contiguous()
        self.labels = torch.cat([lab.to(torch.int32) for _, lab in scans]).contiguous()
        base = np.concatenate([[0], np.cumsum([int(p.shape[0]) for p, _ in scans])]).tolist()
        if base[-1] >= 2 ** 31:
            raise ValueError(f"the scans hold {base[-1]} points; at most 2^31 - 1 are indexed")
        plans, labs = [], []
        for i in range(len(scans)):
            plans.append(ops.scene_plan(self.points[base[i]:base[i + 1]], self.n_points,
                                        float(block_size), int(overlap), self.seed))
            labs.append(self.labels[base[i]:base[i + 1]])
        self.index = ops.scene_index(plans, labs, base[:-1], classes, int(min_points),
                                     float(min_ratio))
        off = self.index.h_elig_off
        self.n_eligible: Dict[int, int] = {c: off[k + 1] - off[k] for k, c in enumerate(classes)}

    # ---------------------------------------------------------------------------------------
    def test_classes(self, n_way: int, n_per_combination: int = 100) -> np.ndarray:
        """The reference's test set (MyTestDataset): every n_way-combination of the fold's classes,
        n_per_combination episodes each, as an (E, n_way) int32 array of way classes."""
        comb = list(itertools.combinations(self.classes, int(n_way)))
        return np.repeat(np.asarray(comb, np.int32).reshape(-1, int(n_way)), int(n_per_combination),
                         axis=0)

    def n_noise(self, k_shot: int, noise_ratio, first: int, n: int, step: int = 1) -> List[int]:
        """Noisy shots per way of episodes first, first + step, ...: round(k_shot * ratio); a list
        of ratios gives every episode the entry (H(K_e, 0) * len) >> 32 (the reference's train mode,
        loader.py:668-670)."""
        if isinstance(noise_ratio, (list, tuple, np.ndarray)):
            r = [float(x) for x in noise_ratio]
            if not r:
                raise ValueError("noise_ratio list is empty")
            pick = [r[(_hkey(episode_key(self.seed, first + i * step), 0) * len(r)) >> 32]
                    for i in range(n)]
        else:
            pick = [float(noise_ratio)] * n
        if any(not 0.0 <= x <= 1.0 for x in pick):
            raise ValueError(f"noise ratios must be in [0, 1]; got {noise_ratio}")
        return [int(round(k_shot * x)) for x in pick]

    def sample(self, way_classes, k_shot: int, n_queries: int = 1, first: int = 0,
               noise_type: Optional[str] = None, noise_ratio=0.0, pair_dict=None,
               step: int = 1) -> dict:
        """Samples E episodes on the device: episode i of the batch has index first + i * step and
        way classes way_classes[i] ((E, n_way) class ids, or (n_way,) for one episode).  Every
        output is a function of (seed, episode index) alone.
        noise_type None, "ood", "sym" or "pair"; noise_ratio a float or a list (one ratio drawn
        per episode); pair_dict maps a class to its pair-noise class (a class it lacks maps to
        itself).  Returns the batch as forward_episodes takes it: support_x (E, n_way, k_shot, 9, N)
        and query_x (E, n_way*n_queries, 9, N) views over point-major memory, support_y,
        gt_support_y (E, n_way, k_shot, N) int32, support_flag (E, n_way, k_shot) int32 class of
        every shot, query_y (E, n_way*n_queries, N) int64 in 0..n_way, sampled_classes (E, n_way)
        int32 numpy array, n_noise (E,), and the provenance: shot_block, query_block (global
        blocks of self.index), support_src, query_src (global points of every slot)."""
        wc = np.asarray(way_classes, dtype=np.int64)
        if wc.ndim == 1:
            wc = wc[None]
        if wc.ndim != 2 or wc.shape[0] < 1 or not 1 <= wc.shape[1] <= 7:
            raise ValueError(f"way_classes must be (E, n_way) with 1..7 ways; got {wc.shape}")
        E, n_way = wc.shape
        if int(k_shot) != k_shot or not 1 <= k_shot <= 32:
            raise ValueError(f"k_shot must be an integer in 1..32; got {k_shot}")
        if int(n_queries) != n_queries or n_queries < 1 or E * n_way * n_queries > 65535:
            raise ValueError(f"n_queries must be >= 1 with E * n_way * n_queries <= 65535; got "
                             f"{E} x {n_way} x {n_queries}")
        if noise_type not in NOISE_TYPES:
            raise ValueError(f"noise_type must be one of {NOISE_TYPES} ('partial' is not built)")
        if int(first) != first or int(step) != step or first < 0 or step < 1 or \
                first + (E - 1) * step >= 2 ** 32:
            raise ValueError(f"episode indices first={first}, step={step} must stay in 0..2^32-1")
        nn = self.n_noise(int(k_shot), noise_ratio, int(first), E, int(step))
        if noise_type is None and any(nn):
            raise ValueError("noise_ratio > 0 needs a noise_type")
        pair = None
        if noise_type == "pair":
            if pair_dict is None:
                raise ValueError("pair noise needs pair_dict")
            pair = [int(pair_dict.get(c, c)) for c in self.classes]
            bad = [p for p in pair if p not in self.n_eligible]
            if bad:
                raise ValueError(f"pair_dict maps to classes outside the dataset: {bad}")
        for e in range(E):
            row = [int(c) for c in wc[e]]
            unknown = [c for c in row if c not in self.n_eligible]
            if unknown or len(set(row)) != n_way:
                raise ValueError(f"episode {first + e * step}: ways {row} must be distinct classes "
                                 f"of {self.classes}")
            need = k_shot - nn[e] + n_queries
            if need > 32:
                raise ValueError(f"k_shot - n_noise + n_queries = {need} exceeds 32")
            short = [f"class {c}: {self.n_eligible[c]} eligible blocks" for c in row
                     if self.n_eligible[c] < need]
            if short:
                raise ValueError(f"too few blocks for {k_shot - nn[e]} clean shots + {n_queries} "
                                 f"queries ({'; '.join(short)}); lower min_points / min_ratio or "
                                 "add scans")
            if nn[e] and noise_type == "ood" and not any(
                    self.n_eligible[c] > 0 for c in self.classes if c not in row):
                raise ValueError(f"episode {first + e * step}: no class outside the ways {row} has "
                                 "an eligible block for ood noise")
            if nn[e] and noise_type == "sym" and n_way < 2:
                raise ValueError("sym noise needs at least two ways")
            if nn[e] and noise_type == "pair":
                empty = [pair[self.classes.index(c)] for c in row
                         if self.n_eligible[pair[self.classes.index(c)]] < 1]
                if empty:
                    raise ValueError(f"pair noise classes without eligible blocks: {empty}")
        out = ops.scene_episodes(self.index, self.points, self.labels, wc.tolist(), nn, noise_type,
                                 pair, int(k_shot), int(n_queries), self.n_points, self.seed,
                                 int(first), int(step))
        out["support_x"] = out["support_x"].transpose(3, 4)
        out["query_x"] = out["query_x"].transpose(2, 3)
        out["sampled_classes"] = wc.astype(np.int32)
        out["n_noise"] = np.asarray(nn, np.int32)
        return out
