"""CPU tests of few-shot episodes sampled from labelled scans: the numpy oracle of the contract in
include/r3dfs.h ("Few-shot episodes from labelled scans") on hand-built multi-scan datasets, and
the host side of r3dfs_scene_index / r3dfs_scene_episodes (workspace queries, argument checks
before anything is launched).  The GPU tests compare the kernels with the same oracle."""
import ctypes as C

import numpy as np
import pytest

from tests import scene_episodes_oracle as X
from tests.test_scene_support_host import _scan

N = 64


def _dataset(seed=0):
    """three scans of 4, 3 and 5 blocks; classes 1..4 spread so that every class has 3+ blocks"""
    a = _scan([200] * 4, [[1] * 60 + [2] * 60, [1] * 60 + [3] * 60, [2] * 60 + [4] * 60,
                          [3] * 60 + [4] * 60], seed)
    b = _scan([150, 300, 200], [[1] * 40, [2] * 100 + [4] * 100, [3] * 80], seed + 1)
    c = _scan([250] * 5, [[1] * 70, [2] * 70, [3] * 70, [4] * 70, [1] * 30 + [2] * 30], seed + 2)
    return [a, b, c]


def _ix(**kw):
    return X.index(_dataset(), [1, 2, 3, 4], N, min_points=20, min_ratio=0.05, **kw)


def test_eligibility_at_the_threshold_edge():
    scans = [_scan([200, 200], [[1] * 10, [1] * 11]), _scan([200], [[1] * 11])]
    ix = X.index(scans, [1], N, min_points=4, min_ratio=0.05)
    assert list(ix["threshold"]) == [10, 10, 10]
    assert list(ix["count"][:, 0]) == [10, 11, 11]
    assert list(ix["elig"][0]) == [1, 2]


def test_global_block_numbering_and_ascending_class_lists():
    ix = _ix()
    assert list(ix["block_scan"]) == [0] * 4 + [1] * 3 + [2] * 5
    assert list(ix["block_id"]) == [0, 1, 2, 3, 0, 1, 2, 0, 1, 2, 3, 4]
    sizes = [200] * 4 + [150, 300, 200] + [250] * 5
    assert list(np.diff(ix["block_off"])) == sizes
    first = np.concatenate([[0], np.cumsum(sizes)])
    for b in range(12):                       # members are the block's own global points
        m = ix["member"][ix["block_off"][b]:ix["block_off"][b + 1]]
        assert sorted(m) == list(range(first[b], first[b + 1]))
    for e in ix["elig"]:
        assert list(e) == sorted(e) and len(e) >= 3
    assert list(ix["elig_off"]) == list(np.cumsum([0] + [len(e) for e in ix["elig"]]))


def _sample(ix, wc, nn, noise, k=5, nq=1, seed=3, first=0, pair=None):
    return X.episodes(ix, wc, nn, noise, k, nq, N, seed=seed, first=first, pair=pair)


def test_clean_shots_and_queries_of_a_way_are_distinct():
    ix = _ix()
    r = _sample(ix, [[1, 2]] * 6, [0] * 6, None, k=2, nq=1)
    for e in range(6):
        for w in range(2):
            blocks = list(r["shot_block"][e, w]) + [r["query_block"][e, w]]
            assert len(set(blocks)) == 3
            assert set(blocks) <= set(ix["elig"][w])
    assert len({tuple(r["shot_block"][e].ravel()) for e in range(6)}) > 1   # episodes differ


def test_noise_classes_follow_their_range():
    ix = _ix()
    wc = [[1, 2], [3, 4], [2, 3]] * 3
    r = _sample(ix, wc, [2] * 9, "ood", k=3)
    for e, row in enumerate(wc):
        for w in range(2):
            f = r["support_flag"][e, w][r["noisy"][e, w]]
            assert len(f) == 2 and not set(f) & set(row)
    r = _sample(ix, wc, [2] * 9, "sym", k=3)
    for e, row in enumerate(wc):
        for w in range(2):
            assert set(r["support_flag"][e, w][r["noisy"][e, w]]) == {row[1 - w]}
    pair = [2, 1, 3, 4]                       # 1 <-> 2, 3 and 4 map to themselves
    r = _sample(ix, wc, [1] * 9, "pair", k=3, pair=pair)
    for e, row in enumerate(wc):
        for w, c in enumerate(row):
            nz = r["noisy"][e, w]
            assert list(r["support_flag"][e, w][nz]) == [pair[c - 1]]
            blk = r["shot_block"][e, w][nz][0]
            assert blk in ix["elig"][pair[c - 1] - 1]


def test_single_use_rule_gives_distinct_noise_classes():
    # k_shot 5, ratio 0.6: 3 noisy shots, k_shot - n_noise - 1 == 1; with 1 way, 3 ood classes
    ix = _ix()
    r = _sample(ix, [[1]] * 8, [3] * 8, "ood", k=5)
    for e in range(8):
        f = r["support_flag"][e, 0][r["noisy"][e, 0]]
        assert sorted(f) == [2, 3, 4]
    # two ways: two ood classes for three shots -> both used, then the last one repeats
    r = _sample(ix, [[1, 2]] * 8, [3] * 8, "ood", k=5)
    for e in range(8):
        for w in range(2):
            f = list(r["support_flag"][e, w][r["noisy"][e, w]])
            assert set(f) == {3, 4}


def test_gt_mask_flag_shuffle_and_query_remap():
    ix = _ix()
    wc = [[2, 4], [1, 3]] * 4
    r = _sample(ix, wc, [2] * 8, "ood", k=4, nq=2)
    lab = ix["labels"]
    slots_seen = set()
    for e, row in enumerate(wc):
        for w, c in enumerate(row):
            nz = r["noisy"][e, w]
            assert nz.sum() == 2 and (r["support_flag"][e, w][~nz] == c).all()
            slots_seen.add(tuple(np.nonzero(nz)[0]))
            for s in range(4):
                y = (lab[r["support_src"][e, w, s]] == r["support_flag"][e, w, s]).astype(np.int32)
                assert np.array_equal(r["support_y"][e, w, s], y)
                assert np.array_equal(r["gt_support_y"][e, w, s], np.zeros_like(y) if nz[s] else y)
            for q in range(2):
                ql = lab[r["query_src"][e, w * 2 + q]]
                want = np.where(ql == row[0], 1, np.where(ql == row[1], 2, 0))
                assert np.array_equal(r["query_y"][e, w * 2 + q], want)
    assert len(slots_seen) > 1                # the noisy shots do not always sit last


def test_episode_alone_equals_its_entry_in_a_batch():
    ix = _ix()
    wc = [[1, 2], [3, 4], [2, 3], [4, 1]]
    batch = _sample(ix, wc, [1, 0, 2, 1], "sym", k=4, first=7)
    for i in range(4):
        one = _sample(ix, [wc[i]], [[1, 0, 2, 1][i]], "sym", k=4, first=7 + i)
        for k, v in one.items():
            assert np.array_equal(v[0], batch[k][i]), k


# ---- the C calls, host side ----------------------------------------------------------------------
def test_workspace_queries_are_pure_host_calls():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    assert 0 < L.r3dfs_scene_index_workspace(1000, 6) < L.r3dfs_scene_index_workspace(2000, 6)
    for nb, nc in [(0, 6), (100, 0), (100, 65), (2 ** 26, 64)]:
        assert L.r3dfs_scene_index_workspace(nb, nc) == 0
    ok = L.r3dfs_scene_episodes_workspace(16, 2, 5, 1, 6)
    assert 0 < ok < (1 << 20)
    for a in [(0, 2, 5, 1, 6), (1, 0, 5, 1, 6), (1, 8, 5, 1, 6), (1, 2, 0, 1, 6), (1, 2, 33, 1, 6),
              (1, 2, 5, 0, 6), (1, 2, 5, 1, 0), (1, 2, 5, 1, 65), (9363, 7, 1, 1, 6)]:
        assert L.r3dfs_scene_episodes_workspace(*a) == 0, a
    assert L.r3dfs_scene_episodes_workspace(9362, 7, 1, 1, 6) > 0     # 65534 query clouds


def test_scene_index_checks_arguments_before_launching():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    BAD, UNS, WS = -1, -2, -3
    fake, null = C.c_void_p(4096), C.c_void_p(0)
    sizes = (C.c_int64 * 2)()
    n0 = L.r3dfs_launch_count()

    def call(lab=fake, M=1000, r=1, cls=(1, 2), scan=0, pb=0, out=fake, sz=sizes, pws=fake, pnb=0):
        h = (C.c_int32 * max(1, len(cls)))(*cls)
        return L.r3dfs_scene_index(lab, M, r, h, len(cls), scan, pb, 0, 0, 10, 10, out, out, out,
                                   out, out, sz, pws, pnb, null)

    assert call() == WS                                        # plan workspace too small
    for kw in (dict(lab=null), dict(out=null), dict(pws=null), dict(M=0), dict(cls=(3, 3)),
               dict(scan=-1), dict(pb=-1)):
        assert call(**kw) == BAD, kw
    for kw in (dict(cls=()), dict(cls=tuple(range(65))), dict(r=5), dict(pb=2 ** 31 - 10)):
        assert call(**kw) == UNS, kw
    ws = L.r3dfs_scene_index_workspace(10, 2)

    def classes(off=fake, nb=10, nc=2, mp=0, mr=0.0, ws_bytes=ws, h=None):
        h = (C.c_int32 * 3)() if h is None else h
        return L.r3dfs_scene_index_classes(off, fake, nb, nc, mp, mr, fake, fake, h, fake,
                                           ws_bytes, null)

    assert classes(ws_bytes=ws - 1) == WS
    for kw in (dict(off=null), dict(nb=0), dict(mp=-1), dict(mr=1.5), dict(mr=float("nan"))):
        assert classes(**kw) == BAD, kw
    assert classes(nc=65) == UNS
    assert L.r3dfs_launch_count() == n0


def _episodes_call(L, **over):
    fake, null = C.c_void_p(4096), C.c_void_p(0)
    a = dict(elig=(0, 3, 6, 6, 9), cls=(1, 2, 3, 4), way=(1, 2), nn=(0,), noise=0, pair=None,
             E=1, n_way=2, k=2, nq=1, N=64, first=0, step=1, ws=None, out=fake)
    a.update(over)
    I32 = lambda v: (C.c_int32 * max(1, len(v)))(*v)  # noqa: E731
    ws = a["ws"] if a["ws"] is not None else L.r3dfs_scene_episodes_workspace(
        a["E"], a["n_way"], a["k"], a["nq"], len(a["cls"]))
    o = a["out"]
    return L.r3dfs_scene_episodes(
        fake, 6, 1, fake, fake, fake, fake, fake, I32(a["elig"]), I32(a["cls"]), len(a["cls"]),
        I32(a["way"]), I32(a["nn"]), a["noise"], None if a["pair"] is None else I32(a["pair"]),
        a["E"], a["n_way"], a["k"], a["nq"], a["N"], 0, a["first"], a["step"],
        o, o, o, o, o, o, o, o, o, o, fake, ws - 1 if a["ws"] is None else ws, null)


def test_scene_episodes_checks_arguments_before_launching():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    BAD, UNS, WS = -1, -2, -3
    n0 = L.r3dfs_launch_count()
    assert _episodes_call(L) == WS                             # everything else valid
    assert _episodes_call(L, noise=1, nn=(1,)) == WS          # ood: classes 2 and 4 are outside
    assert _episodes_call(L, noise=3, nn=(1,), pair=(2, 1, 3, 4)) == WS
    for kw in (dict(out=C.c_void_p(0)), dict(way=(1, 1)), dict(way=(1, 9)), dict(cls=(1, 2, 3, 1)),
               dict(way=(3, 1)),                               # class 3 has no eligible block
               dict(k=3),                                      # 3 + 1 > 3 eligible blocks
               dict(nn=(1,)),                                  # noise without a noise type
               dict(noise=1, nn=(3,)),                         # n_noise > k_shot
               dict(noise=1, nn=(-1,)), dict(noise=4), dict(noise=3, nn=(1,)),   # pair map missing
               dict(noise=3, nn=(1,), pair=(3, 1, 3, 4)),      # class 3 has no eligible block
               dict(noise=3, nn=(1,), pair=(9, 1, 3, 4)),      # unknown pair class
               dict(noise=2, nn=(1,), way=(1,), n_way=1),      # sym with one way
               dict(noise=1, nn=(1,), elig=(0, 3, 6, 6, 6)),   # ood: no other class eligible
               dict(first=-1), dict(step=0), dict(first=2 ** 32)):
        assert _episodes_call(L, **kw) == BAD, kw
    for kw in (dict(n_way=8, way=tuple(range(8)), cls=tuple(range(8)), elig=tuple(range(9))),
               dict(k=33), dict(nq=0), dict(N=63), dict(k=20, nq=13, elig=(0, 40, 80, 80, 120)),
               dict(E=32768, way=(1, 2) * 32768, nn=(0,) * 32768)):
        assert _episodes_call(L, **kw) == UNS, kw
    assert L.r3dfs_launch_count() == n0


def test_python_layer_names_the_short_class():
    import torch
    from r3dfsseg_b200.scene_episodes import SceneEpisodes
    ds = SceneEpisodes.__new__(SceneEpisodes)          # the checks need no device
    ds.classes, ds.seed, ds.n_points = [1, 2, 3], 0, 64
    ds.n_eligible = {1: 9, 2: 4, 3: 0}
    with pytest.raises(ValueError, match=r"class 2: 4 eligible"):
        ds.sample([[1, 2]], k_shot=5)
    with pytest.raises(ValueError, match=r"class 3: 0 eligible"):
        ds.sample([[3, 1]], k_shot=1)
    with pytest.raises(ValueError):
        ds.sample([[1, 1]], k_shot=1)
    with pytest.raises(ValueError):
        ds.sample([[1, 2]], k_shot=2, noise_type="partial")
    with pytest.raises(ValueError):
        ds.sample([[1, 2]], k_shot=2, noise_ratio=0.5)
    with pytest.raises(ValueError, match="ood"):
        ds.sample([[1, 2]], k_shot=2, noise_type="ood", noise_ratio=0.5)
    with pytest.raises(ValueError):
        SceneEpisodes([(torch.zeros(10, 6), torch.zeros(10, dtype=torch.int64))], [1])
