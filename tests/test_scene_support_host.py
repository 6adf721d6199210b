"""CPU tests of support shots cut from a labelled scan: the numpy oracle of the contract in
include/r3dfs.h ("Support shots from a labelled scan") on hand-built scans (the eligibility
threshold at its edge, either term of it dominating, one block serving two ways, blocks smaller
than, equal to and larger than N, a flat axis, overlap 2, fewer eligible blocks than k_shot), and
the host side of r3dfs_scene_support (workspace query, argument checks before anything is
launched).  The GPU tests compare the kernels with the same oracle."""
import ctypes as C

import numpy as np
import pytest

from tests import scene_oracle as O
from tests import scene_support_oracle as S
from tests.test_scene_host import _key_order, _pts

N = 64


def _scan(n_per_block, labels_per_block, seed=0):
    """Blocks side by side along x (block i holds x in [i, i + 0.9]), y in [0, 0.9]; block i gets
    n_per_block[i] points whose first len(labels) points carry the given labels, the rest -1."""
    rng = np.random.default_rng(seed)
    xs, ls = [], []
    for i, (n, lab) in enumerate(zip(n_per_block, labels_per_block)):
        x = rng.uniform(i, i + 0.9, n)
        x[0] = i                                     # cells start at integers: block i = cell i
        xs.append(x)
        lab = np.asarray(lab, np.int64)
        ls.append(np.concatenate([lab, np.full(n - len(lab), -1, np.int64)]))
    x = np.concatenate(xs)
    pts = _pts(x, rng.uniform(0, 0.9, len(x)), rng.uniform(0, 2, len(x)),
               rng.uniform(0, 255, (len(x), 3)))
    return pts, np.concatenate(ls)


def test_threshold_is_strict():
    # n_b = 200, ratio 0.05 -> 10 > min_points 4: 10 points of the class are not enough, 11 are
    pts, lab = _scan([200, 200], [[1] * 10, [1] * 11])
    r = S.support(pts, lab, [1], 2, N, min_points=4, min_ratio=0.05)
    assert list(r["threshold"]) == [10, 10] and list(r["count"][0]) == [10, 11]
    assert list(r["n_eligible"]) == [1]
    assert list(r["block"][0]) == [1, -1]


@pytest.mark.parametrize("n_b, ratio_thr", [(1000, 50), (100, 5)])
def test_either_term_of_the_threshold_can_dominate(n_b, ratio_thr):
    thr = max(ratio_thr, 20)              # 1000 points: the ratio term; 100 points: min_points
    pts, lab = _scan([n_b, n_b], [[3] * thr, [3] * (thr + 1)])
    r = S.support(pts, lab, [3], 1, N, min_points=20, min_ratio=0.05)
    assert list(r["threshold"]) == [thr, thr]
    assert list(r["n_eligible"]) == [1] and list(r["block"][0]) == [1]


def test_ratio_product_is_float64():
    # int(n_b * 0.05) of Python: 0.05 as a double, not as a float32 (0.05f * 60 rounds the same,
    # the product is what the float64 rule pins)
    n_b = np.arange(1, 5000)
    thr = np.floor(n_b.astype(np.float64) * 0.05).astype(np.int64)
    assert np.array_equal(thr, np.array([int(n * 0.05) for n in n_b]))


def test_one_block_serves_two_ways():
    pts, lab = _scan([300, 300], [[5] * 40 + [7] * 40, [5] * 10])
    r = S.support(pts, lab, [7, 5], 1, N, min_points=20, min_ratio=0.0)
    assert list(r["n_eligible"]) == [1, 1]
    assert r["block"][0, 0] == r["block"][1, 0] == 0
    assert np.array_equal(r["src"][0, 0], r["src"][1, 0])           # the same cloud
    assert np.array_equal(r["support_x"][0, 0], r["support_x"][1, 0])
    assert np.array_equal(r["support_y"][0, 0], (lab[r["src"][0, 0]] == 7).astype(np.int32))
    assert np.array_equal(r["support_y"][1, 0], (lab[r["src"][1, 0]] == 5).astype(np.int32))


def test_blocks_smaller_equal_and_larger_than_n():
    sizes = [30, N, 100]
    pts, lab = _scan(sizes, [[2] * n for n in sizes], seed=4)
    r = S.support(pts, lab, [2], 3, N, min_points=0, min_ratio=0.0, seed=9)
    assert r["n_eligible"][0] == 3 and sorted(r["block"][0]) == [0, 1, 2]
    first = np.concatenate([[0], np.cumsum(sizes)])
    chunks = O.plan(pts, N, 1.0, 1, seed=9)
    for j, b in enumerate(r["block"][0]):
        src = r["src"][0, j]
        ranked = _key_order(np.arange(first[b], first[b + 1]), seed=9)
        assert list(src) == list(ranked[np.arange(N) % min(len(ranked), N)])
        if sizes[b] > N:
            assert len(set(src)) == N                                 # N distinct points
        else:
            assert len(set(src)) == sizes[b]
            # a block of at most N points is its single segment_scene chunk
            c = list(chunks["chunk_src"][:, 0]).index(src[0])
            assert np.array_equal(chunks["chunk_src"][c], src)
            assert np.array_equal(chunks["chunk_x"][c], r["support_x"][0, j])
        assert (r["support_y"][0, j] == 1).all()


def test_shots_follow_the_way_key():
    pts, lab = _scan([100] * 6, [[1] * 30 + [2] * 30] * 6, seed=2)
    r = S.support(pts, lab, [1, 2], 6, N, min_points=10, min_ratio=0.0, seed=11)
    for w in range(2):
        keys = S.way_key(r["block"][w], 11, w)
        assert sorted(r["block"][w]) == list(range(6)) and list(keys) == sorted(keys)
    assert list(r["block"][0]) != list(r["block"][1])                 # another key per way
    r2 = S.support(pts, lab, [1, 2], 2, N, min_points=10, min_ratio=0.0, seed=12)
    assert list(r2["n_eligible"]) == [6, 6]


def test_flat_axis():
    rng = np.random.default_rng(6)
    pts = _pts(rng.uniform(0, 0.9, 200), rng.uniform(0, 0.9, 200), 1.25,
               rng.uniform(0, 255, (200, 3)))
    lab = np.where(np.arange(200) < 150, 4, -1)
    r = S.support(pts, lab, [4], 1, N, min_points=0, min_ratio=0.5)
    x = r["support_x"][0, 0]
    assert not x[:, 2].any() and not x[:, 8].any()
    assert x[:, 0:2].min() == 0 and x[:, 6:8].max() == 1


def test_overlap_2_counts_every_membership():
    rng = np.random.default_rng(8)
    M = 6000
    pts = _pts(rng.uniform(0, 3.2, M), rng.uniform(0, 2.1, M), rng.uniform(0, 2, M))
    lab = rng.integers(-1, 3, M)
    r = S.support(pts, lab, [0, 2], 4, N, overlap=2, min_points=30, min_ratio=0.05, seed=3)
    pl = O.plan(pts, N, 1.0, 2, seed=3)
    for w, c in enumerate([0, 2]):
        for s, b in enumerate(r["block_ids"]):
            inside = pl["mem_point"][pl["mem_block"] == b]
            assert r["count"][w, s] == (lab[inside] == c).sum()
            assert r["threshold"][s] == max(int(len(inside) * 0.05), 30)
        assert r["n_eligible"][w] == (r["count"][w] > r["threshold"]).sum() >= 4
        for j, b in enumerate(r["block"][w]):
            assert set(r["src"][w, j]) <= set(pl["mem_point"][pl["mem_block"] == b])


def test_missing_shots_are_empty():
    pts, lab = _scan([200, 200, 200], [[1] * 50, [1] * 50, []])
    r = S.support(pts, lab, [1, 9], 3, N, min_points=20, min_ratio=0.05)
    assert list(r["n_eligible"]) == [2, 0]
    assert r["block"][0, 2] == -1 and (r["block"][1] == -1).all()
    for w, j in [(0, 2), (1, 0), (1, 1), (1, 2)]:
        assert not r["support_x"][w, j].any() and not r["support_y"][w, j].any()
        assert (r["src"][w, j] == -1).all()


# ---- the C call, host side ---------------------------------------------------------------------
def test_scene_support_workspace_is_a_pure_host_call():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    sizes = [L.r3dfs_scene_support_workspace(w, k) for w in range(1, 8) for k in (1, 5, 32)]
    assert all(0 < s < (1 << 20) for s in sizes)
    assert sizes == sorted(sizes)
    for w, k in [(0, 5), (8, 5), (2, 0), (2, 33)]:
        assert L.r3dfs_scene_support_workspace(w, k) == 0


def test_scene_support_checks_arguments_before_launching():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    BAD, UNS, WS = -1, -2, -3
    fake = C.c_void_p(4096)          # never dereferenced: every call below returns first
    null = C.c_void_p(0)
    n0 = L.r3dfs_launch_count()

    def call(pts=fake, M=1000, lab=fake, cls=(1, 2), n_way=None, k=5, mp=100, mr=0.05, r=1,
             N=2048, out=fake, pws=fake, pnb=1 << 40, ws=fake, nb=0):
        n_way = len(cls) if n_way is None else n_way
        h = None if cls is None else (C.c_int32 * max(1, len(cls)))(*cls)
        return L.r3dfs_scene_support(pts, M, 6, 1, lab, h, n_way, k, mp, mr, 0, r, N, out, out,
                                     out, out, out, pws, pnb, ws, nb, null)

    assert call() == WS                                        # everything else valid
    assert call(pnb=0, nb=1 << 20) == WS                       # plan workspace too small
    for kw in (dict(pts=null), dict(lab=null), dict(cls=None, n_way=2), dict(out=null), dict(pws=null),
               dict(ws=null), dict(M=0), dict(cls=(3, 3)), dict(cls=(1, 2, 1)), dict(mp=-1),
               dict(mr=-0.01), dict(mr=1.01), dict(mr=float("nan")), dict(mr=float("inf"))):
        assert call(**kw) == BAD, kw
    for kw in (dict(cls=(), n_way=0), dict(cls=tuple(range(8))), dict(k=0), dict(k=33),
               dict(r=0), dict(r=5), dict(N=63), dict(M=2 ** 31 // 16, r=4)):
        assert call(**kw) == UNS, kw
    assert call(mp=0, mr=0.0) == WS and call(mr=1.0) == WS    # edges of the ranges are valid
    assert L.r3dfs_launch_count() == n0


def test_support_from_scene_refuses_cpu_points():
    import torch
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(2, 5)).eval()
    with pytest.raises(ValueError):
        m.support_from_scene(torch.zeros(100, 6), torch.zeros(100, dtype=torch.int64), [1, 2])
