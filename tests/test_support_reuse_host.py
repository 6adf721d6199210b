"""CPU tests of the split episode (one support set, many query clouds): the workspace queries of
r3dfs_mpti_support / r3dfs_mpti_query are pure host calls sized for their own half, and the two
custom ops have fake kernels.  No kernel is launched here."""
import torch


def test_split_workspace_queries_are_pure_host_calls():
    from r3dfsseg_b200 import _lib, ops
    L = _lib.lib()
    cfg = ops.make_cfg(2, 5, 2, 2048)
    for E in (1, 25):
        full = L.r3dfs_mpti_workspace(cfg, E)
        query = L.r3dfs_mpti_query_workspace(cfg, E)
        support = L.r3dfs_mpti_support_workspace(cfg, E)
        assert 0 < query < full
        assert 0 < support <= full
    # the query half carves nothing support-sized: its workspace ignores k_shot
    sizes = {L.r3dfs_mpti_query_workspace(ops.make_cfg(2, k, 2, 2048), 25) for k in (1, 2, 5, 32)}
    assert len(sizes) == 1
    # the support half carves nothing query-sized beyond the envelope check
    assert L.r3dfs_mpti_support_workspace(ops.make_cfg(2, 5, 2, 2048), 3) == \
        L.r3dfs_mpti_support_workspace(ops.make_cfg(2, 5, 3, 2048), 3)


def test_split_workspace_queries_reject_the_same_configs():
    from r3dfsseg_b200 import _lib, ops
    L = _lib.lib()
    outside = [ops.make_cfg(9, 5, 2, 2048),                      # n_way > 7
               ops.make_cfg(2, 5, 2, 2048, n_subprototypes=200),  # > 127 sub-prototypes
               ops.make_cfg(2, 5, 4, 2048),                      # graph of > 8192 nodes
               ops.make_cfg(2, 5, 2, 2048, k_connect=4096)]      # k_connect >= query points
    for cfg in outside:
        assert L.r3dfs_mpti_workspace(cfg, 1) == 0
        assert L.r3dfs_mpti_support_workspace(cfg, 1) == 0
        assert L.r3dfs_mpti_query_workspace(cfg, 1) == 0
    cfg = ops.make_cfg(2, 5, 2, 2048)
    assert L.r3dfs_mpti_support_workspace(cfg, 0) == 0
    assert L.r3dfs_mpti_query_workspace(cfg, 0) == 0


def test_split_ops_have_fake_kernels():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from r3dfsseg_b200 import ops  # noqa: F401  (registers the ops)
    op = torch.ops.r3dfs
    with FakeTensorMode():
        f = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device="cuda")
        S, E, nw, ks, N, nq = 2, 3, 2, 5, 2048, 2
        w = [f(4)] * 31
        proto, count, clean = op.mpti_support(w, 9, 20, f(S, nw, ks, 9, N),
                                              f(S, nw, ks, N, dt=torch.int32), nq, 100, 200, True)
        assert tuple(proto.shape) == (S, nw + 1, 101, 192) and proto.dtype == torch.float32
        assert tuple(count.shape) == (S, nw + 1) and count.dtype == torch.int32
        assert tuple(clean.shape) == (S, nw, ks)
        r = op.mpti_query(w, 9, 20, proto, count, f(E, nq, 9, N), f(E, nq, N, dt=torch.int64),
                          False, ks, 200, 1.0, 0.99, 200, 1e-6, None)
        assert [tuple(t.shape) for t in r] == [(E, nq, N, nw + 1), (E,), (E, nq, N), (E,), (E,)]
        assert r[2].dtype == torch.int32 and r[3].dtype == torch.int32
        assert r[0].device.type == "cuda"
        r = op.mpti_query(w, 9, 20, proto[:1], count[:1], f(E, nq, 9, N), None, True, ks, 200, 1.0,
                          0.99, 200, 1e-6, None)
        assert tuple(r[0].shape) == (E, nq, N, nw + 1)
