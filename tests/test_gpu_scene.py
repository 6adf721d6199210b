"""Whole-scan segmentation on the GPU: the r3dfs_scene_* kernels against the numpy oracle of the
contract (tests/scene_oracle.py), and MPTI_SelfAtten.segment_scene against `segment` run on the
same chunks and merged by the oracle.  Every comparison is exact (torch.equal)."""
import numpy as np
import pytest
import torch

from r3dfsseg_b200 import ops
from r3dfsseg_b200.episodes import default_args, make_episode, make_scene
from tests import scene_oracle as O
from tests.test_scene_host import _pts

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _gpu_plan(points, N, block_size=1.0, overlap=1, seed=0):
    pts = torch.from_numpy(points).to(DEV)
    plan = ops.scene_plan(pts, N, block_size, overlap, seed)
    E = int(plan.n_chunks.item())
    x, src = ops.scene_chunks(plan, E)
    return plan, E, x, src


def _check_chunks(points, N, block_size=1.0, overlap=1, seed=0):
    ref = O.plan(points, N, block_size, overlap, seed)
    plan, E, x, src = _gpu_plan(points, N, block_size, overlap, seed)
    assert E == ref["n_chunks"]
    assert torch.equal(src.cpu(), torch.from_numpy(ref["chunk_src"]))
    assert torch.equal(x.cpu(), torch.from_numpy(ref["chunk_x"]))
    return ref, plan, E


@pytest.fixture(scope="module")
def room():
    return make_scene(11)[0]          # 6 m x 4 m, 240 000 points


@pytest.mark.parametrize("overlap", [1, 2])
def test_chunks_of_a_room_equal_the_oracle(room, overlap):
    assert room.shape[0] >= 200_000
    _check_chunks(room, 2048, 1.0, overlap, seed=5)


def test_chunks_of_a_translated_room_equal_its_oracle(room):
    far = (room + np.array([1000, 1000, 1000, 0, 0, 0], np.float32)).astype(np.float32)
    _check_chunks(far, 2048, 1.0, 2, seed=5)


def _edge_cases():
    rng = np.random.default_rng(3)
    N = 64
    xa = rng.uniform(0.0, 0.99, N)
    xa[0] = 0.0
    blocks = _pts(np.concatenate([xa, rng.uniform(1.0, 1.99, N + 1), [2.5]]),
                  rng.uniform(0, 0.9, 2 * N + 2), 0.0, rng.uniform(0, 255, (2 * N + 2, 3)))
    return {
        "cell_edges": (_pts([0, 1, 2, 3], [0, 1, 2, 3]), N, 2),
        "sliver_under": (_pts([0.0, 0.3, 2.49], 0.0), N, 1),
        "sliver_over": (_pts([0.0, 0.3, 2.51], 0.0), N, 1),
        "flat_z": (_pts(rng.uniform(10, 10.9, 300), rng.uniform(-5, -4.2, 300), 1.5,
                        rng.uniform(0, 255, (300, 3))), 128, 1),
        "n_n1_1_members": (blocks, N, 1),
        "fewer_than_n": (_pts(np.linspace(0, 0.5, 10), 0.2), N, 1),
        "overlap4": (_pts(rng.uniform(0, 5.3, 4000), rng.uniform(0, 3.7, 4000),
                          rng.uniform(0, 3, 4000)), N, 4),
    }


@pytest.mark.parametrize("name", list(_edge_cases()))
def test_chunks_of_edge_cases_equal_the_oracle(name):
    pts, N, r = _edge_cases()[name]
    _check_chunks(pts, N, 1.0, r, seed=7)


def test_merge_equals_the_oracle(room):
    ref, plan, E = _check_chunks(room, 2048, 1.0, 2, seed=1)
    lg = torch.randn((E, 2048, 3), generator=torch.Generator().manual_seed(0))
    out = ops.scene_merge(plan, lg.to(DEV), E)
    r_logits, r_pred, r_cov = O.merge(lg.numpy(), ref)
    assert torch.equal(out["logits"].cpu(), torch.from_numpy(r_logits))
    assert torch.equal(out["pred"].cpu(), torch.from_numpy(r_pred))
    assert torch.equal(out["coverage"].cpu(), torch.from_numpy(r_cov))


def test_non_finite_xy_is_reported_by_the_chunk_count():
    pts = _pts([0.0, 1.0, float("nan")], 0.0)
    plan = ops.scene_plan(torch.from_numpy(pts).to(DEV), 64)
    assert int(plan.n_chunks.item()) == -1


# ---- segment_scene ----------------------------------------------------------------------------
def _model(fixture_sd, n_way, k_shot):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot))
    m.load_state_dict(fixture_sd)
    return m.to(DEV).eval()


def _support(m, n_way, k_shot, **ep):
    e = make_episode(41, n_way, k_shot, **ep)
    return m.encode_support(e.support_x.to(DEV), e.support_y.to(DEV), eval=True)


SCENE_CASES = {
    "s3dis_2way_5shot_mdns": dict(n_way=2, k_shot=5, ep=dict(noise_ratio=0.4), overlap=2),
    "scannet_3way_5shot_ood": dict(n_way=3, k_shot=5, overlap=1,
                                   ep=dict(dataset="scannet", noise_ratio=0.4, noise_type="ood")),
}


@pytest.mark.parametrize("name", list(SCENE_CASES))
def test_segment_scene_equals_segment_on_the_chunks(fixture_sd, name):
    c = SCENE_CASES[name]
    m = _model(fixture_sd, c["n_way"], c["k_shot"])
    sup = _support(m, c["n_way"], c["k_shot"], **c["ep"])
    pts_np = make_scene(21, size_xy=(3.0, 2.0), points_per_m2=8000.0)[0]
    pts = torch.from_numpy(pts_np).to(DEV)
    ref = O.plan(pts_np, 2048, 1.0, c["overlap"], 3)
    E = ref["n_chunks"]
    qx = torch.from_numpy(ref["chunk_x"]).to(DEV).view(E, 1, 2048, 9).transpose(2, 3)
    outs = {}
    for b in (1, 7, E + 5):
        # segment on the oracle's chunks in the same batches: the query half's kernels are not
        # batch-invariant in the last bits, so the exact reference is batched as segment_scene is
        seg = torch.cat([m.segment(sup, qx[b0:b0 + b])["logits"][:, 0] for b0 in range(0, E, b)])
        r_logits, r_pred, r_cov = O.merge(seg.cpu().numpy(), ref)
        out = m.segment_scene(sup, pts, overlap=c["overlap"], seed=3, chunk_batch=b)
        assert out["n_chunks"] == E
        assert out["logits"].shape == (pts.shape[0], c["n_way"] + 1)
        assert torch.equal(out["logits"].cpu(), torch.from_numpy(r_logits))
        assert torch.equal(out["pred"].cpu(), torch.from_numpy(r_pred))
        assert torch.equal(out["coverage"].cpu(), torch.from_numpy(r_cov))
        outs[b] = out
    # across batch sizes: the same labels, logits within FP32 rounding of one another
    a = outs[E + 5]
    for b in (1, 7):
        rel = float((outs[b]["logits"] - a["logits"]).abs().max() / a["logits"].abs().max())
        agree = float((outs[b]["pred"] == a["pred"]).float().mean())
        assert rel < 1e-4 and agree >= 0.999, (b, rel, agree)


def test_segment_scene_is_deterministic_and_seeded(fixture_sd):
    m = _model(fixture_sd, 2, 5)
    sup = _support(m, 2, 5)
    pts = torch.from_numpy(make_scene(22, size_xy=(2.5, 2.0), points_per_m2=6000.0)[0]).to(DEV)
    a = m.segment_scene(sup, pts, overlap=2, seed=0)
    b = m.segment_scene(sup, pts, overlap=2, seed=0)
    for k in ("logits", "pred", "coverage"):
        assert torch.equal(a[k], b[k]), k
    pa = ops.scene_plan(pts, 2048, 1.0, 2, 0)
    pb = ops.scene_plan(pts, 2048, 1.0, 2, 1)
    E = int(pa.n_chunks.item())
    assert int(pb.n_chunks.item()) == E
    assert not torch.equal(ops.scene_chunks(pa, E)[1], ops.scene_chunks(pb, E)[1])
    c = m.segment_scene(sup, pts, overlap=2, seed=1)
    assert torch.equal(c["coverage"], a["coverage"])


def test_segment_scene_guards(fixture_sd):
    from r3dfsseg_b200 import _lib
    m = _model(fixture_sd, 2, 5)
    sup = _support(m, 2, 5)
    pts = torch.from_numpy(make_scene(23, size_xy=(1.5, 1.0), points_per_m2=3000.0)[0]).to(DEV)
    m.segment_scene(sup, pts)
    L = _lib.lib()
    torch.cuda.synchronize()
    n0 = L.r3dfs_launch_count()
    bad = [dict(points=pts.cpu()), dict(points=pts[:0]), dict(points=pts[:, :5]),
           dict(overlap=0), dict(overlap=5), dict(block_size=0.0), dict(block_size=-1.0),
           dict(seed=-1), dict(chunk_batch=0)]
    for kw in bad:
        args = dict(points=pts)
        args.update(kw)
        with pytest.raises(ValueError):
            m.segment_scene(sup, **args)
    assert L.r3dfs_launch_count() == n0
    with pytest.raises(ValueError):                                   # other configuration
        _model(fixture_sd, 3, 5).segment_scene(sup, pts)
    e = make_episode(42, 2, 5)
    two = m.encode_support(torch.stack([e.support_x] * 2).to(DEV),
                           torch.stack([e.support_y] * 2).to(DEV))
    with pytest.raises(ValueError):                                   # more than one set
        m.segment_scene(two, pts)
    with pytest.raises(ValueError):                                   # non-finite x
        far = pts.clone()
        far[0, 0] = float("inf")
        m.segment_scene(sup, far)
    m.load_state_dict(fixture_sd)                                     # stale prototypes
    with pytest.raises(RuntimeError, match="stale"):
        m.segment_scene(sup, pts)
    m.segment_scene(m.encode_support(e.support_x.to(DEV), e.support_y.to(DEV)), pts)
