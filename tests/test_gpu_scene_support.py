"""Support shots cut from a labelled scan on the GPU: r3dfs_scene_support against the numpy oracle
of the contract (tests/scene_support_oracle.py), the plan it reads left as it was, encode_support
on the shots it returns, and MPTI_SelfAtten.support_from_scene.  Every comparison is exact
(torch.equal)."""
import numpy as np
import pytest
import torch

from r3dfsseg_b200 import ops
from r3dfsseg_b200.episodes import default_args, make_scene
from tests import scene_support_oracle as S
from tests.test_scene_support_host import _scan

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
KEYS = ("support_x", "support_y", "src", "block", "n_eligible")


def _gpu_support(pts, labels, classes, k_shot, N, block_size=1.0, overlap=1, seed=0, **kw):
    plan = ops.scene_plan(pts, N, block_size, overlap, seed)
    return plan, ops.scene_support(plan, labels, classes, k_shot, seed, **kw)


def _check(points, labels, classes, k_shot, N, block_size=1.0, overlap=1, seed=0, **kw):
    ref = S.support(points, labels, classes, k_shot, N, block_size, overlap, seed, **kw)
    _, got = _gpu_support(torch.from_numpy(points).to(DEV), torch.from_numpy(labels).to(DEV),
                          classes, k_shot, N, block_size, overlap, seed, **kw)
    assert got["support_x"].shape == (len(classes), k_shot, 9, N)
    assert torch.equal(got["support_x"].transpose(2, 3).cpu(), torch.from_numpy(ref["support_x"]))
    for k in KEYS[1:]:
        assert torch.equal(got[k].cpu(), torch.from_numpy(ref[k])), k
    return ref, got


@pytest.fixture(scope="module")
def room():
    return make_scene(11)             # 6 m x 4 m, 240 000 points, two blobs of each class


@pytest.mark.parametrize("overlap", [1, 2])
def test_shots_of_a_room_equal_the_oracle(room, overlap):
    pts, cls = room
    ref, _ = _check(pts, cls, [0, 3, 5], 5, 2048, 1.0, overlap, seed=5)
    assert (ref["n_eligible"] > 0).all()
    if overlap == 1:
        assert (ref["n_eligible"] < 5).any()          # missing shots are part of the comparison


def test_shots_of_a_translated_room_equal_its_oracle(room):
    pts, cls = room
    far = (pts + np.array([1000, 1000, 1000, 0, 0, 0], np.float32)).astype(np.float32)
    _check(far, cls, [1, 2, 4], 5, 2048, 1.0, 2, seed=5)


def _edge_cases():
    N = 64
    rng = np.random.default_rng(6)
    flat = (np.concatenate([rng.uniform(0, 0.9, (200, 2)), np.full((200, 1), 1.25),
                            rng.uniform(0, 255, (200, 3))], 1).astype(np.float32),
            np.where(np.arange(200) < 150, 4, -1))
    M = 6000
    ov2 = (np.concatenate([rng.uniform(0, 3.2, (M, 1)), rng.uniform(0, 2.1, (M, 1)),
                           rng.uniform(0, 2, (M, 1)), rng.uniform(0, 255, (M, 3))],
                          1).astype(np.float32), rng.integers(-1, 3, M))
    return {
        "threshold_edge": (_scan([200, 200], [[1] * 10, [1] * 11]), [1], 2, N, 1,
                           dict(min_points=4, min_ratio=0.05)),
        "ratio_dominates": (_scan([1000, 1000], [[3] * 50, [3] * 51]), [3], 1, N, 1,
                            dict(min_points=20, min_ratio=0.05)),
        "min_points_dominates": (_scan([100, 100], [[3] * 20, [3] * 21]), [3], 1, N, 1,
                                 dict(min_points=20, min_ratio=0.05)),
        "block_serves_two_ways": (_scan([300, 300], [[5] * 40 + [7] * 40, [5] * 10]), [7, 5], 1,
                                  N, 1, dict(min_points=20, min_ratio=0.0)),
        "smaller_equal_larger_than_n": (_scan([30, N, 100], [[2] * 30, [2] * N, [2] * 100],
                                              seed=4), [2], 3, N, 1,
                                        dict(min_points=0, min_ratio=0.0)),
        "flat_z": (flat, [4], 1, N, 1, dict(min_points=0, min_ratio=0.5)),
        "overlap2": (ov2, [0, 2], 4, N, 2, dict(min_points=30, min_ratio=0.05)),
        "fewer_than_k_shot": (_scan([200, 200, 200], [[1] * 50, [1] * 50, []]), [1, 9], 3, N, 1,
                              dict(min_points=20, min_ratio=0.05)),
        "seven_ways_32_shots": ((ov2[0], rng.integers(0, 7, M)), [6, 0, 1, 2, 3, 4, 5], 32, N,
                                2, dict(min_points=0, min_ratio=0.1)),
    }


@pytest.mark.parametrize("name", list(_edge_cases()))
def test_shots_of_edge_cases_equal_the_oracle(name):
    (pts, lab), classes, k, N, r, kw = _edge_cases()[name]
    _check(pts, lab, classes, k, N, 1.0, r, seed=9, **kw)


def test_strided_points_and_int64_labels(room):
    pts, cls = room
    wide = np.concatenate([pts, np.arange(len(pts), dtype=np.float32)[:, None]], 1)  # (M, 7)
    ref = S.support(pts, cls, [2, 5], 5, 2048, 1.0, 2, seed=1)
    t = torch.from_numpy(wide).to(DEV)[:, :6]
    lab = torch.from_numpy(cls).to(DEV)
    assert t.stride() == (7, 1) and lab.dtype == torch.int64
    _, got = _gpu_support(t, lab, [2, 5], 5, 2048, 1.0, 2, seed=1)
    assert torch.equal(got["support_x"].transpose(2, 3).cpu(), torch.from_numpy(ref["support_x"]))
    for k in KEYS[1:]:
        assert torch.equal(got[k].cpu(), torch.from_numpy(ref[k])), k


def test_plan_is_left_as_it_was(room):
    pts, cls = room
    p = torch.from_numpy(pts).to(DEV)
    plan = ops.scene_plan(p, 2048, 1.0, 2, 3)
    E = int(plan.n_chunks.item())
    lg = torch.randn((E, 2048, 3), generator=torch.Generator().manual_seed(0)).to(DEV)
    x0, src0 = ops.scene_chunks(plan, E)
    m0 = ops.scene_merge(plan, lg, E)
    ws0 = plan.workspace.clone()
    ops.scene_support(plan, torch.from_numpy(cls).to(DEV), [0, 1, 2, 3], 7, 3)
    assert torch.equal(plan.workspace, ws0)
    x1, src1 = ops.scene_chunks(plan, E)
    m1 = ops.scene_merge(plan, lg, E)
    assert torch.equal(x0, x1) and torch.equal(src0, src1)
    for k in ("logits", "pred", "coverage"):
        assert torch.equal(m0[k], m1[k]), k


def test_non_finite_x_gives_minus_one_eligible():
    pts, lab = _scan([200, 200], [[1] * 50, [1] * 50])
    pts[3, 0] = np.nan
    _, got = _gpu_support(torch.from_numpy(pts).to(DEV), torch.from_numpy(lab).to(DEV), [1, 2],
                          2, 64, min_points=0, min_ratio=0.0)
    assert got["n_eligible"].tolist() == [-1, -1]
    assert (got["block"] == -1).all() and (got["src"] == -1).all()
    assert not got["support_y"].any() and not got["support_x"].any()


# ---- encode_support and support_from_scene ----------------------------------------------------
def _model(fixture_sd, n_way, k_shot):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot))
    m.load_state_dict(fixture_sd)
    return m.to(DEV).eval()


ENCODE_CASES = {
    "s3dis_2way_5shot_mdns": dict(n_way=2, classes=[2, 7], scene=dict(seed=31,
                                                                      classes=[2] * 6 + [7] * 6)),
    "scannet_3way_5shot": dict(n_way=3, classes=[1, 4, 6],
                               scene=dict(seed=32, classes=[1] * 5 + [4] * 5 + [6] * 5,
                                          dataset="scannet")),
}


@pytest.mark.parametrize("name", list(ENCODE_CASES))
def test_encode_support_on_the_shots_equals_the_oracle_clouds(fixture_sd, name):
    c = ENCODE_CASES[name]
    m = _model(fixture_sd, c["n_way"], 5)
    pts, cls = make_scene(**c["scene"])
    ref = S.support(pts, cls, c["classes"], 5, 2048, 1.0, 2, seed=4)
    assert (ref["n_eligible"] >= 5).all()
    s = m.support_from_scene(torch.from_numpy(pts).to(DEV), torch.from_numpy(cls).to(DEV),
                             c["classes"], overlap=2, seed=4)
    assert s["support_x"].transpose(2, 3).is_contiguous()        # the view, no copy
    got = m.encode_support(s["support_x"], s["support_y"], eval=True)
    rx = torch.from_numpy(ref["support_x"]).permute(0, 1, 3, 2).contiguous().to(DEV)
    want = m.encode_support(rx, torch.from_numpy(ref["support_y"]).to(DEV), eval=True)
    assert torch.equal(got.prototypes, want.prototypes)
    assert torch.equal(got.proto_count, want.proto_count)
    assert torch.equal(got.clean_flag, want.clean_flag)


def test_support_from_scene_then_segment_scene(fixture_sd):
    m = _model(fixture_sd, 2, 5)
    a_pts, a_cls = make_scene(31, classes=[2] * 6 + [7] * 6)
    s = m.support_from_scene(torch.from_numpy(a_pts).to(DEV), torch.from_numpy(a_cls).to(DEV),
                             [2, 7])
    sup = m.encode_support(s["support_x"], s["support_y"])
    b = torch.from_numpy(make_scene(33, size_xy=(3.0, 2.0), points_per_m2=8000.0)[0]).to(DEV)
    out = m.segment_scene(sup, b, overlap=1)
    assert out["logits"].shape == (b.shape[0], 3) and torch.isfinite(out["logits"]).all()
    assert (out["coverage"] == 1).all()
    # 3 shots of one scan and 2 of another combine along the shot axis
    c_pts, c_cls = make_scene(34, classes=[2] * 4 + [7] * 4)
    sa = m.support_from_scene(torch.from_numpy(a_pts).to(DEV), torch.from_numpy(a_cls).to(DEV),
                              [2, 7], k_shot=3)
    sc = m.support_from_scene(torch.from_numpy(c_pts).to(DEV), torch.from_numpy(c_cls).to(DEV),
                              [2, 7], k_shot=2)
    assert torch.equal(sa["support_x"], s["support_x"][:, :3])     # a prefix of the 5 shots
    x = torch.cat([sa["support_x"], sc["support_x"]], 1)
    y = torch.cat([sa["support_y"], sc["support_y"]], 1)
    mixed = m.encode_support(x, y)
    assert torch.isfinite(m.segment_scene(mixed, b)["logits"]).all()


def test_support_from_scene_is_deterministic_and_seeded(fixture_sd):
    m = _model(fixture_sd, 2, 5)
    pts, cls = make_scene(31, classes=[2] * 6 + [7] * 6)
    p, lab = torch.from_numpy(pts).to(DEV), torch.from_numpy(cls).to(DEV)
    a = m.support_from_scene(p, lab, [2, 7], overlap=2, seed=0)
    b = m.support_from_scene(p, lab, [2, 7], overlap=2, seed=0)
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k
    c = m.support_from_scene(p, lab, [2, 7], overlap=2, seed=1)
    assert torch.equal(c["n_eligible"], a["n_eligible"])
    assert not torch.equal(c["block"], a["block"])


def test_support_from_scene_guards(fixture_sd):
    from r3dfsseg_b200 import _lib
    m = _model(fixture_sd, 2, 5)
    pts, cls = make_scene(31, classes=[2] * 6 + [7] * 6)
    p, lab = torch.from_numpy(pts).to(DEV), torch.from_numpy(cls).to(DEV)
    m.support_from_scene(p, lab, [2, 7])
    L = _lib.lib()
    torch.cuda.synchronize()
    n0 = L.r3dfs_launch_count()
    bad = [dict(points=p.cpu()), dict(points=p[:0]), dict(points=p[:, :5]),
           dict(labels=lab.cpu()), dict(labels=lab[:-1]), dict(labels=lab.float()),
           dict(classes=[2]), dict(classes=[2, 7, 1]), dict(classes=[2, 2]),
           dict(classes=[2, 2 ** 31]), dict(k_shot=0), dict(k_shot=33),
           dict(overlap=0), dict(overlap=5), dict(block_size=0.0), dict(block_size=float("nan")),
           dict(seed=-1), dict(min_points=-1), dict(min_ratio=-0.1), dict(min_ratio=1.5),
           dict(min_ratio=float("nan"))]
    for kw in bad:
        args = dict(points=p, labels=lab, classes=[2, 7])
        args.update(kw)
        with pytest.raises(ValueError):
            m.support_from_scene(**args)
    assert L.r3dfs_launch_count() == n0
    with pytest.raises(ValueError, match=r"class 9: 0 eligible"):          # a short class
        m.support_from_scene(p, lab, [2, 9])
    far = p.clone()
    far[0, 0] = float("inf")
    with pytest.raises(ValueError, match="non-finite"):
        m.support_from_scene(far, lab, [2, 7])
