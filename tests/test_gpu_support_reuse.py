"""One support set, many query clouds: MPTI_SelfAtten.encode_support + segment (the support and
query halves of r3dfs_mpti_forward) against forward_episodes on the same episodes.  The same
kernels run on the same rows, so the comparison is exact (torch.equal), not a tolerance."""
import pytest
import torch

from r3dfsseg_b200.episodes import default_args, make_episode

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def model(fixture_sd):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    ms = {}

    def get(n_way, k_shot, **over):
        key = (n_way, k_shot, tuple(sorted(over.items())))
        if key not in ms:
            m = MPTI_SelfAtten(default_args(n_way, k_shot, **over))
            m.load_state_dict(fixture_sd)
            ms[key] = m.to(DEV).eval()
        return ms[key]
    return get


def _fresh(fixture_sd, n_way=2, k_shot=5, **over):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot, **over))
    m.load_state_dict(fixture_sd)
    return m.to(DEV).eval()


def _batch(eps, n_query=None):
    """Episodes stacked on a leading E axis, in the point-major memory of the reference's collate."""
    sx = torch.stack([e.support_x.transpose(2, 3) for e in eps]).to(DEV).transpose(3, 4)
    sy = torch.stack([e.support_y for e in eps]).to(DEV)
    qx = torch.stack([e.query_x.transpose(1, 2) for e in eps]).to(DEV).transpose(2, 3)
    qy = torch.stack([e.query_y for e in eps]).to(DEV)
    if n_query is not None:
        qx, qy = qx[:, :n_query], qy[:, :n_query]
    return sx, sy, qx, qy


def _assert_same(got, ref):
    for k in ("logits", "loss", "pred"):
        assert torch.equal(got[k], ref[k]), k


def _few_fg(eps, keep=5):
    """Way 0 keeps `keep` foreground points per shot: a set smaller than n_subprototypes."""
    for e in eps:
        for s in range(e.support_y.shape[1]):
            fg = torch.nonzero(e.support_y[0, s]).flatten()
            e.support_y[0, s, fg[keep:]] = 0
    return eps


CASES = {
    "s3dis_2way_5shot_noisy": dict(n_way=2, k_shot=5, ev=True, ep=dict(noise_ratio=0.4)),
    "s3dis_2way_5shot_no_mdns": dict(n_way=2, k_shot=5, ev=False, ep=dict(noise_ratio=0.4)),
    "scannet_3way_5shot_ood": dict(n_way=3, k_shot=5, ev=True,
                                   ep=dict(dataset="scannet", noise_ratio=0.4, noise_type="ood")),
    "s3dis_2way_1shot": dict(n_way=2, k_shot=1, ev=True, ep={}),
    "ragged_512pts_20sub_1query": dict(n_way=2, k_shot=2, ev=True, ep=dict(n_pts=512),
                                       over=dict(pc_npts=512, n_subprototypes=20, k_connect=100),
                                       n_query=1, few_fg=True),
}


@pytest.mark.parametrize("name", list(CASES))
def test_split_equals_forward_bit_for_bit(model, name):
    c = CASES[name]
    m = model(c["n_way"], c["k_shot"], **c.get("over", {}))
    eps = [make_episode(300 + 7 * i + len(name), c["n_way"], c["k_shot"], **c["ep"])
           for i in range(3)]
    if c.get("few_fg"):
        eps = _few_fg(eps)
    sx, sy, qx, qy = _batch(eps, c.get("n_query"))
    ref = m.forward_episodes(sx, sy, qx, qy, eval=c["ev"], want_diag=True)
    sup = m.encode_support(sx, sy, eval=c["ev"])
    got = m.segment(sup, qx, qy)
    _assert_same(got, ref)
    assert torch.equal(sup.proto_count, ref["diag"]["proto_count"])
    assert torch.equal(sup.clean_flag, ref["diag"]["clean_flag"])
    assert sup.n_sets == 3 and sup.k_shot == c["k_shot"] and sup.mdns == c["ev"]
    if c.get("few_fg"):   # every foreground point of way 0 is its own prototype
        assert int(sup.proto_count[:, 1].max()) <= 5 * c["k_shot"]
    # rows past a set's count are zero
    slot = torch.arange(sup.prototypes.shape[2], device=DEV)
    pad = slot[None, None, :] >= sup.proto_count[:, :, None]
    assert not sup.prototypes[pad].any()
    # one-episode form: what forward returns
    pred, loss = m.segment(m.encode_support(sx[0], sy[0], eval=c["ev"]), qx[0], qy[0])
    assert torch.equal(pred, ref["logits"][0].transpose(1, 2)) and torch.equal(loss, ref["loss"][0])


def test_one_set_shared_by_many_episodes(model):
    m = model(2, 5)
    eps = [make_episode(400 + i, 2, 5, noise_ratio=0.4) for i in range(4)]
    sx, sy, qx, qy = _batch(eps)
    ref = m.forward_episodes(torch.cat([sx[:1]] * 4), torch.cat([sy[:1]] * 4), qx, qy, eval=True)
    sup = m.encode_support(sx[0], sy[0])           # one (n_way, k_shot, C, N) set
    assert sup.n_sets == 1
    _assert_same(m.segment(sup, qx, qy), ref)


def test_set_index_picks_the_set_of_each_episode(model):
    m = model(2, 5)
    eps = [make_episode(500 + i, 2, 5, noise_ratio=0.4) for i in range(3)]
    sx, sy, qx, qy = _batch(eps)
    sup = m.encode_support(sx[:2], sy[:2])
    idx = [1, 0, 1]
    ref = m.forward_episodes(sx[idx], sy[idx], qx, qy, eval=True)
    _assert_same(m.segment(sup, qx, qy, set_index=idx), ref)
    _assert_same(m.segment(sup, qx, qy, set_index=torch.tensor(idx)), ref)


def test_segment_is_deterministic(model):
    m = model(2, 5)
    sx, sy, qx, qy = _batch([make_episode(600 + i, 2, 5, noise_ratio=0.4) for i in range(3)])
    sup = m.encode_support(sx, sy)
    a, b = m.segment(sup, qx, qy), m.segment(sup, qx, qy)
    _assert_same(a, b)
    sup2 = m.encode_support(sx, sy)
    assert torch.equal(sup.prototypes, sup2.prototypes)


def test_stale_support_set_is_refused(fixture_sd):
    m = _fresh(fixture_sd)
    sx, sy, qx, qy = _batch([make_episode(700, 2, 5)])
    sup = m.encode_support(sx, sy)
    m.segment(sup, qx, qy)
    m.load_state_dict(fixture_sd)                  # same values, but new weights were loaded
    with pytest.raises(RuntimeError, match="stale"):
        m.segment(sup, qx, qy)
    sup = m.encode_support(sx, sy)
    m.segment(sup, qx, qy)
    with torch.no_grad():
        m.encoder.edge_convs[0].layer[1].running_mean.add_(0.01)   # a BatchNorm statistic
    with pytest.raises(RuntimeError, match="stale"):
        m.segment(sup, qx, qy)


def test_guards(model, fixture_sd):
    from r3dfsseg_b200 import _lib
    m = model(2, 5)
    sx, sy, qx, qy = _batch([make_episode(800 + i, 2, 5) for i in range(3)])
    sup = m.encode_support(sx[:2], sy[:2])
    # a model of another configuration
    for over in (dict(n_subprototypes=50), dict(pc_npts=1024)):
        other = model(2, 5, **over)
        with pytest.raises(ValueError):
            other.segment(sup, qx, qy)
    with pytest.raises(ValueError):
        model(3, 5).segment(sup, qx, qy)
    # set indices are checked on the host before anything is launched
    L = _lib.lib()
    torch.cuda.synchronize()
    n0 = L.r3dfs_launch_count()
    for bad in ([0, 1, 2], [0, -1, 1], [0, 1]):
        with pytest.raises(ValueError):
            m.segment(sup, qx, qy, set_index=bad)
    assert L.r3dfs_launch_count() == n0
    with pytest.raises(ValueError):           # 2 sets for 3 episodes and no set_index
        m.segment(sup, qx, qy)
    # CPU tensors
    with pytest.raises(RuntimeError):
        m.segment(sup, qx.cpu(), qy.cpu(), set_index=[0, 1, 0])
    with pytest.raises(RuntimeError):
        m.encode_support(sx.cpu(), sy.cpu())
    # outside the envelope: the same error as forward_episodes (4 queries of 2048 points make a
    # graph of more than 8192 nodes; 200 sub-prototypes exceed 127)
    q4x, q4y = torch.cat([qx, qx], 1), torch.cat([qy, qy], 1)
    with pytest.raises(_lib.R3dfsError) as ref:
        m.forward_episodes(sx, sy, q4x, q4y, eval=True)
    with pytest.raises(_lib.R3dfsError) as got:
        m.segment(m.encode_support(sx, sy), q4x, q4y)
    assert str(got.value) == str(ref.value)
    big = model(2, 5, n_subprototypes=200)
    with pytest.raises(_lib.R3dfsError) as ref:
        big.forward_episodes(sx, sy, qx, qy, eval=True)
    with pytest.raises(_lib.R3dfsError) as got:
        big.encode_support(sx, sy)
    assert str(got.value) == str(ref.value)
    # training mode
    t = _fresh(fixture_sd).train()
    with pytest.raises(NotImplementedError):
        t.encode_support(sx, sy)
    with pytest.raises(NotImplementedError):
        t.segment(sup, qx, qy)


def test_segment_traces_under_torch_compile_fullgraph(model):
    m = model(2, 5)
    sx, sy, qx, qy = _batch([make_episode(900 + i, 2, 5, noise_ratio=0.4) for i in range(3)])
    with torch.no_grad():
        m.pack_weights()
        sup = m.encode_support(sx, sy)
        ref = m.segment(sup, qx, qy)
        got = torch.compile(lambda a, b: m.segment(sup, a, b), fullgraph=True)(qx, qy)
    _assert_same(got, ref)
