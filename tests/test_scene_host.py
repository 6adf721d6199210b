"""CPU tests of whole-scan segmentation: the numpy oracle of the contract in include/r3dfs.h on
hand-built scans (cell edges, remainder slivers, flat axes, blocks of N, N+1 and 1 points, scans
smaller than one chunk, overlap 2 and 4), and the host side of the r3dfs_scene_* calls (workspace
query, argument checks before anything is launched).  The GPU tests compare the kernels with the
same oracle."""
import ctypes as C

import numpy as np
import pytest

from tests import scene_oracle as O

F32 = np.float32


def _pts(x, y, z=None, rgb=None):
    x = np.asarray(x, F32)
    y = np.broadcast_to(np.asarray(y, F32), x.shape)
    z = np.zeros_like(x) if z is None else np.broadcast_to(np.asarray(z, F32), x.shape)
    rgb = np.full((len(x), 3), 128, F32) if rgb is None else np.asarray(rgb, F32)
    return np.concatenate([np.stack([x, y, z], 1), rgb], 1).astype(F32)


def _blocks_of(pl, i):
    return list(pl["mem_block"][pl["mem_point"] == i])


def test_points_on_cell_edges():
    p = _pts([0, 1, 2, 3], 0)
    pl = O.plan(p, 64, 1.0, 1)
    assert pl["cells"] == (3, 1) and pl["blocks"] == (3, 1)   # ext 3 = 3 cells, the last absorbs 3.0
    assert list(pl["cell"][0]) == [0, 1, 2, 2]
    assert [_blocks_of(pl, i) for i in range(4)] == [[0], [1], [2], [2]]
    pl = O.plan(p, 64, 1.0, 2)                                  # stride 0.5: 6 cells, 5 blocks
    assert pl["cells"] == (6, 1) and pl["blocks"] == (5, 1)
    assert list(pl["cell"][0]) == [0, 2, 4, 5]
    assert [_blocks_of(pl, i) for i in range(4)] == [[0], [1, 2], [3, 4], [4]]
    assert list(pl["coverage"]) == [1, 2, 2, 1]


@pytest.mark.parametrize("ext, cells", [(2.49, 2), (2.51, 3), (0.49, 1), (0.0, 1)])
def test_remainder_sliver(ext, cells):
    p = _pts([0.0, 0.3, ext], [0.0, 0.0, 0.0])
    pl = O.plan(p, 64, 1.0, 1)
    assert pl["cells"][0] == cells
    assert pl["cell"][0][2] == cells - 1            # the last point is in the last cell
    assert pl["coverage"].tolist() == [1, 1, 1]


def test_flat_axis_and_channels():
    rng = np.random.default_rng(0)
    p = _pts(rng.uniform(10, 10.9, 300), rng.uniform(-5, -4.2, 300), 1.5,
             rng.uniform(0, 255, (300, 3)))
    pl = O.plan(p, 128, 1.0, 1)
    x = pl["chunk_x"]
    assert x.dtype == np.float32 and x.shape == (pl["n_chunks"], 128, 9)
    assert not x[:, :, 2].any() and not x[:, :, 8].any()      # flat z: xyz' = 0 and XYZ = 0
    assert (x[:, :, 0:2].min(1) == 0).all() and (x[:, :, 6:8].max(1) == 1).all()
    src = pl["chunk_src"]
    assert np.array_equal(x[:, :, 3:6], p[src, 3:6] / F32(255))
    assert np.array_equal(x[:, :, 0:3], p[src, 0:3] - p[src, 0:3].min(1, keepdims=True))


def _key_order(idx, seed=0):
    idx = np.asarray(idx)
    return idx[np.argsort(O.lowbias32(idx.astype(np.uint64) ^ O.lowbias32(seed)))]


def test_blocks_of_n_n_plus_1_and_1_points():
    N = 64
    rng = np.random.default_rng(1)
    xa = rng.uniform(0.0, 0.99, N)           # block 0: N points   -> 1 chunk
    xa[0] = 0.0                              # x0 = 0, ext = 2.5: 3 cells
    xb = rng.uniform(1.0, 1.99, N + 1)       # block 1: N+1 points -> 2 chunks of 33 and 32
    xc = [2.5]                               # block 2: 1 point    -> 1 chunk of repeats
    p = _pts(np.concatenate([xa, xb, xc]), rng.uniform(0, 0.9, 2 * N + 2))
    pl = O.plan(p, N, 1.0, 1, seed=7)
    assert pl["cells"] == (3, 1) and pl["n_chunks"] == 4
    assert list(pl["count"]) == [N, 33, 32, 1]
    src = pl["chunk_src"]
    assert sorted(src[0]) == list(range(N))                               # no repeat
    ranked = _key_order(np.arange(N, 2 * N + 1), seed=7)                  # block 1 by key
    assert list(src[1][:33]) == list(ranked[0::2]) and list(src[2][:32]) == list(ranked[1::2])
    for c, n in ((1, 33), (2, 32)):                                       # padding repeats
        assert np.array_equal(src[c], src[c][np.arange(N) % n])
    assert (src[3] == 2 * N + 1).all()
    assert (pl["coverage"] == 1).all()


def test_scan_smaller_than_one_chunk():
    p = _pts(np.linspace(0, 0.5, 10), 0.2)
    pl = O.plan(p, 64, 1.0, 1, seed=3)
    assert pl["n_chunks"] == 1
    assert list(pl["chunk_src"][0]) == list(np.resize(_key_order(np.arange(10), 3), 64))


@pytest.mark.parametrize("r", [1, 2, 4])
def test_overlap_coverage_follows_the_r2_rule(r):
    rng = np.random.default_rng(r)
    p = _pts(rng.uniform(0, 5.3, 4000), rng.uniform(0, 3.7, 4000))
    pl = O.plan(p, 64, 1.0, r)
    cov = np.ones(len(p), np.int64)
    for a, (u, nb) in enumerate(zip(pl["cell"], pl["blocks"])):
        # block i covers cells i .. i + r - 1; a single block covers every cell
        blocks = np.arange(nb)[None, :]
        inside = (blocks <= u[:, None]) & ((u[:, None] <= blocks + r - 1) | (nb == 1))
        cov *= inside.sum(1)
    assert np.array_equal(pl["coverage"], cov)
    assert cov.min() >= 1 and cov.max() == r * r
    # every membership is one real (non-repeat) slot of a chunk of its block
    assert (pl["chunk_src"][pl["mem_chunk"], pl["mem_slot"]] == pl["mem_point"]).all()
    assert (pl["mem_slot"] < pl["count"][pl["mem_chunk"]]).all()
    real = np.arange(64)[None, :] < pl["count"][:, None]
    assert np.array_equal(np.bincount(pl["chunk_src"][real], minlength=len(p)), cov)


def test_seed_changes_chunks_not_memberships():
    rng = np.random.default_rng(5)
    p = _pts(rng.uniform(0, 2, 3000), rng.uniform(0, 2, 3000))
    a, b = O.plan(p, 64, 1.0, 2, seed=0), O.plan(p, 64, 1.0, 2, seed=1)
    assert a["n_chunks"] == b["n_chunks"] and np.array_equal(a["coverage"], b["coverage"])
    assert np.array_equal(a["mem_block"], b["mem_block"])
    assert not np.array_equal(a["chunk_src"], b["chunk_src"])


def test_merge_averages_over_blocks_in_block_order():
    p = _pts([0, 1, 2, 3], 0)
    pl = O.plan(p, 64, 1.0, 2)
    lg = np.zeros((pl["n_chunks"], 64, 2), F32)
    lg[pl["mem_chunk"], pl["mem_slot"]] = np.stack([pl["mem_block"], -pl["mem_block"]], 1)
    out, pred, cov = O.merge(lg, pl)
    assert out[:, 0].tolist() == [0.0, 1.5, 3.5, 4.0] and list(cov) == [1, 2, 2, 1]
    assert list(pred) == [0, 0, 0, 0]                       # tie at 0 -> first class


# ---- the C calls, host side -------------------------------------------------------------------
def test_scene_workspace_is_a_pure_host_call():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    for r in (1, 2, 3, 4):
        sizes = [L.r3dfs_scene_workspace(M, r) for M in (1, 1000, 10 ** 5, 10 ** 6)]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes) and len(set(sizes)) == 4
    for M in (1000, 10 ** 6):
        by_r = [L.r3dfs_scene_workspace(M, r) for r in (1, 2, 3, 4)]
        assert by_r == sorted(by_r) and len(set(by_r)) == 4
    assert L.r3dfs_scene_workspace(0, 1) == 0
    assert L.r3dfs_scene_workspace(1000, 0) == 0 and L.r3dfs_scene_workspace(1000, 5) == 0
    assert L.r3dfs_scene_workspace(2 ** 31 // 16, 4) == 0       # r^2 M = 2^31
    assert L.r3dfs_scene_workspace(2 ** 31 // 16 - 1, 4) > 0


def test_scene_calls_check_arguments_before_launching():
    from r3dfsseg_b200 import _lib
    L = _lib.lib()
    BAD, UNS, WS = -1, -2, -3
    fake = C.c_void_p(4096)          # never dereferenced: every call below returns first
    null = C.c_void_p(0)
    n0 = L.r3dfs_launch_count()

    def plan(pts=fake, M=1000, bs=1.0, r=1, N=2048, n=fake, ws=fake, nb=0):
        return L.r3dfs_scene_plan(pts, M, 6, 1, bs, r, 0, N, n, ws, nb, null)

    def chunks(pts=fake, M=1000, r=1, N=2048, E=5, x=fake, src=fake, ws=fake, nb=0):
        return L.r3dfs_scene_chunks(pts, M, 6, 1, r, N, E, x, src, ws, nb, null)

    def merge(lg=fake, M=1000, r=1, N=2048, E=5, nc=3, out=fake, ws=fake, nb=0):
        return L.r3dfs_scene_merge(lg, M, r, N, E, nc, out, fake, fake, ws, nb, null)

    for call in (plan, chunks, merge):
        assert call() == WS                                   # everything else valid
        assert call(ws=null) == BAD
        assert call(M=0) == BAD
        assert call(r=0) == UNS and call(r=5) == UNS
        assert call(N=63) == UNS and call(N=65537) == UNS
        assert call(M=2 ** 31 // 16, r=4) == UNS
    for kw in (dict(pts=null), dict(n=null), dict(bs=0.0), dict(bs=-1.0), dict(bs=float("nan")),
               dict(bs=float("inf"))):
        assert plan(**kw) == BAD, kw
    for kw in (dict(pts=null), dict(x=null), dict(src=null), dict(E=0), dict(E=1001)):
        assert chunks(**kw) == BAD, kw
    for kw in (dict(lg=null), dict(out=null), dict(E=0)):
        assert merge(**kw) == BAD, kw
    assert merge(nc=0) == UNS and merge(nc=9) == UNS
    assert L.r3dfs_launch_count() == n0


def test_segment_scene_refuses_cpu_points():
    import torch
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten
    from r3dfsseg_b200.models.mpti import SupportSet
    m = MPTI_SelfAtten(default_args(2, 5)).eval()
    sup = SupportSet(torch.zeros(1, 3, 101, 192), torch.zeros(1, 3, dtype=torch.int32),
                     torch.ones(1, 2, 5), 2, 5, 2048, 100, True, None)
    with pytest.raises(ValueError):
        m.segment_scene(sup, torch.zeros(100, 6))
    with pytest.raises(ValueError):                          # another configuration
        MPTI_SelfAtten(default_args(3, 5)).eval().segment_scene(sup, torch.zeros(100, 6))
