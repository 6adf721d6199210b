"""Few-shot episodes sampled on the GPU from labelled scans: the dataset index and
r3dfs_scene_episodes against the numpy oracle of the contract (tests/scene_episodes_oracle.py),
the clouds against scene_chunks, EpisodeEvaluator.run_scenes against EpisodeEvaluator.run on the
same episodes, and a training step on a sampled episode.  Every comparison is exact
(torch.equal)."""
import numpy as np
import pytest
import torch

from r3dfsseg_b200 import ops
from r3dfsseg_b200.episodes import Episode, default_args, make_scene
from r3dfsseg_b200.scene_episodes import SceneEpisodes
from tests import scene_episodes_oracle as X

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
N = 2048
S3DIS = [0, 1, 2, 3, 4, 5]
SCANNET = list(range(10))
IX_KEYS = ("block_off", "block_scan", "block_id", "member", "count", "elig_off", "elig_block")
EP_KEYS = ("support_y", "gt_support_y", "support_flag", "query_y", "shot_block", "query_block",
           "support_src", "query_src")


def _rooms(n, dataset="s3dis", shift_last=True):
    rooms = [make_scene(40 + i, size_xy=(5.0, 4.0), points_per_m2=6000.0, dataset=dataset)
             for i in range(n)]
    if shift_last:
        p, c = rooms[-1]
        rooms[-1] = ((p + np.array([1000, 1000, 1000, 0, 0, 0], np.float32)).astype(np.float32), c)
    return rooms


def _ds(rooms, classes, overlap=1, seed=5, **kw):
    scans = [(torch.from_numpy(p).to(DEV), torch.from_numpy(c).to(DEV)) for p, c in rooms]
    ds = SceneEpisodes(scans, classes, N, 1.0, overlap, seed, **kw)
    ref = X.index(rooms, classes, N, 1.0, overlap, seed, **kw)
    return ds, ref


@pytest.fixture(scope="module")
def s3dis():
    return _ds(_rooms(3), S3DIS)


@pytest.fixture(scope="module")
def scannet():
    return _ds(_rooms(3, "scannet"), SCANNET)


@pytest.mark.parametrize("overlap", [1, 2])
def test_index_equals_the_oracle(overlap):
    ds, ref = _ds(_rooms(3), S3DIS, overlap=overlap)
    for k in IX_KEYS:
        assert torch.equal(getattr(ds.index, k).cpu(), torch.from_numpy(
            np.asarray(ref[k]).astype(getattr(ds.index, k).cpu().numpy().dtype))), k
    assert [ds.n_eligible[c] for c in S3DIS] == [len(e) for e in ref["elig"]]
    assert min(ds.n_eligible.values()) >= 6


def _check(ds, ref, wc, k_shot, n_queries=1, first=0, noise_type=None, noise_ratio=0.0,
           pair_dict=None):
    got = ds.sample(wc, k_shot, n_queries, first, noise_type, noise_ratio, pair_dict)
    pair = None if pair_dict is None else [pair_dict.get(c, c) for c in ds.classes]
    want = X.episodes(ref, got["sampled_classes"], got["n_noise"], noise_type, k_shot, n_queries,
                      N, seed=ds.seed, first=first, pair=pair)
    assert torch.equal(got["support_x"].transpose(3, 4).cpu(), torch.from_numpy(want["support_x"]))
    assert torch.equal(got["query_x"].transpose(2, 3).cpu(), torch.from_numpy(want["query_x"]))
    for k in EP_KEYS:
        assert torch.equal(got[k].cpu(), torch.from_numpy(want[k])), k
    return got, want


CASES = {
    "clean_2way_5shot": dict(pool="s3dis", wc=[[0, 3], [1, 2], [4, 5], [2, 0]], k=5),
    "ood_3way_5shot_scannet": dict(pool="scannet", wc=[[1, 4, 6], [0, 2, 9], [3, 5, 7]], k=5,
                                   noise_type="ood", noise_ratio=0.4),
    "sym_0.4": dict(pool="s3dis", wc=[[0, 3], [1, 2], [4, 5]], k=5, noise_type="sym",
                    noise_ratio=0.4),
    "pair_0.2": dict(pool="s3dis", wc=[[0, 3], [1, 5], [4, 2]], k=5, noise_type="pair",
                     noise_ratio=0.2, pair_dict={0: 1, 1: 2, 2: 3, 3: 4, 4: 5, 5: 5}),
    "ood_ratio_0.6": dict(pool="s3dis", wc=[[0, 3], [1, 2]], k=5, noise_type="ood",
                          noise_ratio=0.6),
    "ratio_list": dict(pool="s3dis", wc=[[0, 3], [1, 2], [4, 5], [2, 0], [1, 3]], k=5,
                       noise_type="sym", noise_ratio=[0.0, 0.2, 0.4, 0.6]),
    "two_queries": dict(pool="s3dis", wc=[[0, 3], [1, 2]], k=5, nq=2, noise_type="ood",
                        noise_ratio=0.2),
    "one_way": dict(pool="s3dis", wc=[[0], [3], [5]], k=5, noise_type="ood", noise_ratio=0.4),
    "one_episode": dict(pool="s3dis", wc=[[2, 4]], k=5, first=123),
}


@pytest.mark.parametrize("name", list(CASES))
def test_sampled_batches_equal_the_oracle(name, s3dis, scannet):
    c = CASES[name]
    ds, ref = s3dis if c["pool"] == "s3dis" else scannet
    _check(ds, ref, c["wc"], c["k"], c.get("nq", 1), c.get("first", 0), c.get("noise_type"),
           c.get("noise_ratio", 0.0), c.get("pair_dict"))


def test_37_episodes_from_a_non_zero_first_and_alone(s3dis):
    ds, ref = s3dis
    wc = ds.test_classes(2, 3)[:37]
    got, _ = _check(ds, ref, wc, 5, 1, 1000, "ood", 0.4)
    one = ds.sample(wc[17], 5, 1, 1017, "ood", 0.4)
    for k in EP_KEYS + ("support_x", "query_x"):
        assert torch.equal(one[k][0], got[k][17]), k


def test_clouds_equal_the_scene_chunks_of_their_block():
    pts, cls = make_scene(11)
    p, lab = torch.from_numpy(pts).to(DEV), torch.from_numpy(cls).to(DEV)
    ds = SceneEpisodes([(p, lab)], [0, 1, 2, 3, 4, 5], n_points=16384, seed=9)
    got = ds.sample([[0, 1], [2, 3], [4, 5]], 2, 1)
    plan = ops.scene_plan(p, 16384, 1.0, 1, 9)
    E = int(plan.n_chunks.item())
    cx, csrc = ops.scene_chunks(plan, E)
    first = {int(s[0]): i for i, s in enumerate(csrc.cpu())}
    nb = (ds.index.block_off[1:] - ds.index.block_off[:-1]).cpu()
    sx, qx = got["support_x"].transpose(3, 4), got["query_x"].transpose(2, 3)
    checked = 0
    for blocks, x, src in ((got["shot_block"], sx, got["support_src"]),
                           (got["query_block"], qx, got["query_src"])):
        for i in np.ndindex(*blocks.shape):
            if nb[int(blocks[i])] <= 16384:
                c = first[int(src[i][0])]
                assert torch.equal(src[i], csrc[c]) and torch.equal(x[i], cx[c])
                checked += 1
    assert checked > 5


def _model(fixture_sd, n_way, k_shot):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot))
    m.load_state_dict(fixture_sd)
    return m.to(DEV).eval()


def test_run_scenes_equals_run_on_the_same_episodes(fixture_sd, s3dis):
    from r3dfsseg_b200.evaluate import EpisodeEvaluator
    ds, _ = s3dis
    m = _model(fixture_sd, 2, 5)
    wc = ds.test_classes(2, 1)[:12]          # at most 3 batches of 4 per rank: run's 3 slots
    b = ds.sample(wc, 5, 1, 0, "ood", 0.4)
    eps = [Episode(b["support_x"][i].cpu(), b["support_y"][i].cpu(), b["query_x"][i].cpu(),
                   b["query_y"][i].cpu(), b["gt_support_y"][i].cpu(), b["sampled_classes"][i],
                   b["support_flag"][i].cpu()) for i in range(len(wc))]
    counters = {}
    for world in (1, 2):
        for rank in range(world):
            got = EpisodeEvaluator(m, S3DIS, batch=4).run_scenes(ds, wc, 5, 1, "ood", 0.4, rank,
                                                                 world)
            want = EpisodeEvaluator(m, S3DIS, batch=4).run(eps, rank, world)
            assert torch.equal(got["counters"], want["counters"])
            assert got["mean_loss"] == want["mean_loss"]
            assert got["n_episodes"] == want["n_episodes"] == len(range(rank, 12, world))
            counters[world, rank] = got["counters"]
    assert torch.equal(counters[2, 0] + counters[2, 1], counters[1, 0])
    assert counters[1, 0][0, 1:].sum() > 0


def test_a_sampled_episode_drives_a_training_step(fixture_sd, s3dis):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    ds, _ = s3dis
    m = MPTI_SelfAtten(default_args(2, 5))
    m.load_state_dict(fixture_sd)
    m = m.to(DEV).train()
    b = ds.sample([[1, 4]], 5, 1, 0, "ood", 0.4)
    out = m(b["support_x"][0], b["support_y"][0], b["query_x"][0], b["query_y"][0],
            gt_support_y=b["gt_support_y"][0], train=True, support_flag=b["support_flag"][0])
    (out[1] + 0.1 * out[2]).backward()
    assert torch.isfinite(out[1]) and torch.isfinite(out[2])
    grads = [p.grad for p in m.parameters() if p.grad is not None]
    assert grads and all(torch.isfinite(g).all() for g in grads)


def test_sampling_is_deterministic_and_seeded(s3dis):
    ds, _ = s3dis
    wc = [[0, 3], [1, 2], [4, 5]]
    a = ds.sample(wc, 5, 1, 0, "sym", 0.4)
    b = ds.sample(wc, 5, 1, 0, "sym", 0.4)
    for k in EP_KEYS + ("support_x", "query_x"):
        assert torch.equal(a[k], b[k]), k
    rooms = _rooms(3)
    other = SceneEpisodes([(torch.from_numpy(p).to(DEV), torch.from_numpy(c).to(DEV))
                           for p, c in rooms], S3DIS, N, 1.0, 1, seed=6)
    c = other.sample(wc, 5, 1, 0, "sym", 0.4)
    assert not torch.equal(c["shot_block"], a["shot_block"])
