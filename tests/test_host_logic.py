"""CPU tests of the host-side logic: the C-ABI library loads and exports what include/r3dfs.h
declares, episode sharding + the counter all-reduce (gloo, world_size 2), mIoU arithmetic, the
synthetic episode contract.  No kernel is launched here."""
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from r3dfsseg_b200 import _lib
    header = open(os.path.join(ROOT, "include", "r3dfs.h")).read()
    declared = set(re.findall(r"\b(r3dfs_[a-z0-9_]+)\s*\(", header))
    assert "r3dfs_mpti_forward" in declared and "r3dfs_knn" in declared
    handle = _lib.lib()
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in r3dfs.h but not exported"
    for name in _lib.SIGNATURES:
        assert name in declared, f"{name} bound in _lib.py but not declared in r3dfs.h"
    assert handle.r3dfs_version() == 100
    assert b"workspace" in handle.r3dfs_strerror(-3)


def test_workspace_queries_are_pure_host_calls():
    from r3dfsseg_b200 import _lib, ops
    L = _lib.lib()
    cfg = ops.make_cfg(2, 5, 2, 2048)
    one = L.r3dfs_mpti_workspace(cfg, 1)
    many = L.r3dfs_mpti_workspace(cfg, 8)
    assert 0 < one < many <= 8 * one + (1 << 20)
    bad = ops.make_cfg(9, 5, 2, 2048)   # n_way > 7 is outside the kernels' range
    assert L.r3dfs_mpti_workspace(bad, 1) == 0
    assert L.r3dfs_knn_workspace(4, 9, 2048, 20) > 0


def test_episode_envelope_follows_the_cg_node_limit():
    """The episode workspace queries refuse a graph the CG solve cannot stage: 8192 nodes up to
    3 ways (n_cls <= 4), 5376 from 4 ways on (n_cls 5..8 pad P to 8 floats a node), where
    nodes = roundup64((n_way + 1) * (n_subprototypes + 1)) + n_query * n_points."""
    from r3dfsseg_b200 import _lib, ops
    L = _lib.lib()
    # the largest accepted: 4-way, 4 queries x 1216 points (512 + 4864 = 5376 nodes) and the
    # benchmark's 2-way episode with two 2048-point queries (320 + 4096 = 4416 nodes)
    for cfg in (ops.make_cfg(4, 1, 4, 1216), ops.make_cfg(2, 5, 2, 2048),
                ops.make_cfg(3, 1, 3, 2560), ops.make_cfg(7, 1, 7, 640)):
        assert L.r3dfs_mpti_workspace(cfg, 1) > 0
        assert L.r3dfs_mpti_query_workspace(cfg, 1) > 0
        assert L.r3dfs_mpti_support_workspace(cfg, 1) > 0
    # rejected: 4-way at 1536 points (512 + 6144 = 6656 nodes), a 4-way query of three 2048-point
    # clouds (512 + 6144), 4-way at 1280 points (512 + 5120 = 5632), and 3-way past 8192 nodes
    for cfg in (ops.make_cfg(4, 1, 4, 1536), ops.make_cfg(4, 1, 3, 2048),
                ops.make_cfg(4, 1, 4, 1280), ops.make_cfg(3, 1, 3, 2816)):
        assert L.r3dfs_mpti_workspace(cfg, 1) == 0
        assert L.r3dfs_mpti_query_workspace(cfg, 1) == 0
        assert L.r3dfs_mpti_support_workspace(cfg, 1) == 0
    # the stand-alone solve checks the same limit before it touches any buffer (these addresses
    # are never dereferenced): n_cls 5 at 5377 nodes, n_cls 4 past 8192, n_cls outside 1..8
    fake = 4096
    for n, nc in ((5377, 5), (5377, 8), (8193, 4), (1000, 9)):
        rc = L.r3dfs_label_propagate(fake, fake, fake, 1, n, 16, fake, nc, 0.99, 1e-6, 200, fake,
                                     None, None, fake, 1 << 62, None)
        assert rc == -2, (n, nc, rc)   # R3DFS_E_UNSUPPORTED


def test_product_path_rejects_cpu_tensors():
    from r3dfsseg_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.knn(torch.rand(1, 9, 64), 4)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.get_edge_feature(torch.rand(1, 9, 64), 4, torch.zeros(1, 64, 4, dtype=torch.long))


def test_module_state_dict_matches_reference_names(fixture_sd):
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(2, 5))
    assert set(m.state_dict().keys()) == set(fixture_sd.keys())
    m.load_state_dict(fixture_sd)          # strict
    assert sum(p.numel() for p in m.parameters()) == 376896   # SURVEY.md §8b
    with pytest.raises(NotImplementedError):
        m.train()
        m.getFeatures(torch.rand(1, 9, 2048))


def test_sharding_partitions_episodes():
    from r3dfsseg_b200.evaluate import shard_indices
    for world in (1, 2, 3, 4, 8):
        seen = sorted(i for r in range(world) for i in shard_indices(101, r, world))
        assert seen == list(range(101))
        sizes = [len(shard_indices(101, r, world)) for r in range(world)]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_indices(10, 2, 2)


def test_miou_matches_reference_metric():
    """evaluate_metric (reference eval_noise.py:23-72) restated by the oracle vs evaluate.py."""
    from oracle import mpti_oracle as O
    from r3dfsseg_b200.evaluate import class_slots, iou_from_counters
    rng = np.random.default_rng(0)
    test_classes = [3, 11, 10, 0, 8, 4]
    preds = [rng.integers(0, 3, (2, 512)) for _ in range(24)]
    gts = [rng.integers(0, 3, (2, 512)) for _ in range(24)]
    l2c = [rng.choice(test_classes, 2, replace=False) for _ in range(24)]
    counters = O.confusion_counts(preds, gts, l2c, test_classes)
    # brute-force restatement of the reference's per-point loop
    ref = np.zeros((3, 7), dtype=np.int64)
    for p, g, c in zip(preds, gts, l2c):
        slot = [0] + class_slots(c, test_classes)
        for pv, gv in zip(p.reshape(-1), g.reshape(-1)):
            ref[0, slot[gv]] += 1
            ref[1, slot[pv]] += 1
            ref[2, slot[gv]] += int(pv == gv)
    assert np.array_equal(counters, ref)
    res = iou_from_counters(torch.from_numpy(counters))
    assert (counters[0] > 0).all()
    assert abs(res["mean_iou"] - O.mean_iou(counters)) < 1e-12


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from oracle import mpti_oracle as O
    from r3dfsseg_b200.evaluate import all_reduce_eval_state, shard_indices
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(123)      # same stream on every rank
    test_classes = list(range(6))
    n = 25
    preds = [rng.integers(0, 3, (2, 256)) for _ in range(n)]
    gts = [rng.integers(0, 3, (2, 256)) for _ in range(n)]
    l2c = [rng.choice(test_classes, 2, replace=False) for _ in range(n)]
    losses = rng.random(n)
    mine = shard_indices(n, rank, world)
    part = O.confusion_counts([preds[i] for i in mine], [gts[i] for i in mine],
                              [l2c[i] for i in mine], test_classes)
    counters = torch.from_numpy(part.copy())
    loss_sum = torch.tensor(float(sum(losses[i] for i in mine)), dtype=torch.float64)
    cnt = torch.tensor(float(len(mine)), dtype=torch.float64)
    all_reduce_eval_state(counters, loss_sum, cnt)
    full = O.confusion_counts(preds, gts, l2c, test_classes)
    ok = bool(np.array_equal(counters.numpy(), full)) and abs(float(loss_sum) - losses.sum()) < 1e-9 \
        and int(cnt) == n
    q.put((rank, ok))
    dist.destroy_process_group()


def test_counter_allreduce_gloo_world2():
    """The N>1 path on CPU: shard, reduce, compare with the single-rank counters (exact ints)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(results) == [(0, True), (1, True)]


def test_synthetic_episode_contract():
    """Shapes / dtypes / strides the reference's collate produces (loader.py:1662-1684)."""
    from r3dfsseg_b200.episodes import make_episode
    ep = make_episode(3, 3, 5, dataset="scannet", noise_ratio=0.4)
    assert ep.support_x.shape == (3, 5, 9, 2048) and not ep.support_x.is_contiguous()
    assert ep.support_x.transpose(2, 3).is_contiguous()           # point-major memory
    assert ep.support_y.dtype == torch.int32 and ep.query_y.dtype == torch.int64
    assert ep.query_x.shape == (3, 9, 2048) and int(ep.query_y.max()) <= 3
    assert (ep.support_y.sum(-1) >= 1).all()                       # >= 1 fg point per shot
    noisy = (ep.gt_support_y.sum(-1) == 0).sum(1)
    assert (noisy == 2).all()                                      # round(5 * 0.4) OOD shots per way
    again = make_episode(3, 3, 5, dataset="scannet", noise_ratio=0.4)
    assert torch.equal(ep.support_x, again.support_x)


def test_train_parameter_layout_matches_reference_order(fixture_sd):
    """The flat parameter buffer of the training path = the reference's named_parameters() order and
    sizes (376 896 floats, encoder/rest learning-rate split at 261 504: models/mpti_learner.py:26-32)."""
    from r3dfsseg_b200 import train as T
    off, group0 = T.param_layout(9)
    names = [k for k in fixture_sd if not (k.endswith("running_mean") or k.endswith("running_var")
                                           or k.endswith("num_batches_tracked"))]
    assert names == T.PARAM_NAMES
    assert [off[i + 1] - off[i] for i in range(len(names))] == [fixture_sd[k].numel() for k in names]
    assert off[-1] == 376896 and group0 == 261504
    assert all(o % 4 == 0 for o in off)           # every tensor 16-byte aligned in the bucket
    bn = T.bn_layout()
    chans = [fixture_sd[p + ".running_mean"].numel() for p in T.BN_PREFIXES]
    assert [bn[i + 1] - bn[i] for i in range(len(chans))] == chans and bn[-1] == 1344


def _gloo_grad_worker(rank, world, port, q):
    import torch.distributed as dist
    from r3dfsseg_b200.train import all_reduce_gradients
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(5)
    per_rank = [torch.randn(376896, generator=g) for _ in range(world)]
    bucket = per_rank[rank].clone()
    scale = all_reduce_gradients(bucket)
    mean = torch.stack(per_rank).sum(0) / world
    q.put((rank, bool(torch.allclose(bucket * scale, mean, atol=1e-6)) and scale == 1.0 / world))
    dist.destroy_process_group()


def test_gradient_bucket_allreduce_gloo_world2():
    """Meta-training N>1 path on CPU: one flat bucket, sum all-reduce, mean folded into the scale."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_grad_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(results) == [(0, True), (1, True)]


def _gloo_replica_worker(rank, world, port, q):
    import torch.distributed as dist
    from r3dfsseg_b200.train import average_tensor, broadcast_tensors
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(100 + rank)           # every rank starts from OTHER values
    flat, running = torch.randn(376896, generator=g), torch.rand(2 * 1344, generator=g)
    broadcast_tensors((flat, running), 0)
    g0 = torch.Generator().manual_seed(100)
    same_start = torch.equal(flat, torch.randn(376896, generator=g0)) and \
        torch.equal(running, torch.rand(2 * 1344, generator=g0))
    # a step: every rank moves its running statistics by its own episode, then they are averaged
    delta = [torch.full((2 * 1344,), float(r + 1)) for r in range(world)]
    start = running.clone()
    running += delta[rank]
    average_tensor(running)
    ok_avg = torch.allclose(running, start + torch.stack(delta).mean(0))
    q.put((rank, bool(same_start and ok_avg)))
    dist.destroy_process_group()


def test_replica_state_broadcast_and_bn_average_gloo_world2():
    """Data-parallel replicas: parameters + BatchNorm statistics are broadcast from rank 0 when the
    optimiser is built, and the running statistics are averaged over the ranks after each step."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_replica_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(results) == [(0, True), (1, True)]


def test_raw_episode_container_round_trip_and_read_into(tmp_path):
    """`.r3ep`: the reference's eight datasets as one flat file that reader threads read straight
    into (pinned) staging rows; converting a folder of .npz/.h5 episodes keeps every array."""
    from r3dfsseg_b200 import episode_io as IO
    from r3dfsseg_b200.episodes import make_episode
    eps = [make_episode(s, 3, 5, dataset="scannet", noise_ratio=0.4) for s in (1, 2)]
    src, dst = tmp_path / "npz", tmp_path / "raw"
    src.mkdir()
    for i, e in enumerate(eps):
        IO.write_episode(str(src / ("%d.h5" % i)), IO.episode_arrays(e))
    assert IO.convert_folder(str(src), str(dst)) == 2
    a, b = IO.EpisodeFolder(str(src)), IO.EpisodeFolder(str(dst))
    assert all(n.endswith(IO.RAW_EXT) for n in b.file_names)
    for i in range(2):
        for x, y in zip(a[i], b[i]):
            assert x.dtype == y.dtype and np.array_equal(x, y)
        stage = {"support_ptclouds": np.zeros((4, 3, 5, 2048, 9), np.float32),
                 "query_labels": np.zeros((4, 3, 2048), np.int64)}
        for folder in (a, b):
            cls = folder.read_into(i, {k: v[2] for k, v in stage.items()})
            assert np.array_equal(cls, eps[i].sampled_classes)
            assert np.array_equal(stage["support_ptclouds"][2], a[i][0])
            assert np.array_equal(stage["query_labels"][2], a[i][3])
            assert not stage["support_ptclouds"][1].any()
    with pytest.raises(ValueError):
        b.read_into(0, {"support_ptclouds": np.zeros((2, 5, 2048, 9), np.float32)})


def test_episode_file_round_trip(tmp_path):
    """The reference's episode schema (dataloaders/loader.py:1687-1721) survives write -> read, and
    the collate leaves the clouds point-major behind (.., 9, N) views (loader.py:1676-1684)."""
    from r3dfsseg_b200 import episode_io as IO
    from r3dfsseg_b200.episodes import make_episode
    ep = make_episode(5, 2, 5, noise_ratio=0.4)
    arrays = IO.episode_arrays(ep)
    assert [a.dtype.name for a in arrays] == [IO.SCHEMA[k] for k in IO.ORDER]
    path = IO.write_episode(str(tmp_path / "0.h5"), arrays)
    back = IO.read_episode(path)
    for a, b in zip(arrays, back):
        assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b)
    data, classes = IO.collate_test(back)
    assert data[0].shape == (2, 5, 9, 2048) and data[0].transpose(2, 3).is_contiguous()
    assert data[2].shape == (2, 9, 2048) and data[3].dtype == torch.int64
    assert torch.equal(data[0], ep.support_x) and torch.equal(data[3], ep.query_y)
    assert np.array_equal(classes, ep.sampled_classes)
    folder = IO.EpisodeFolder(str(tmp_path))
    assert len(folder) == 1
    (d2, c2), = list(folder)
    assert torch.equal(d2[2], ep.query_x)
    sx, sy, qx, qy, cls = IO.stage_batch([back, back], pin=False)
    assert sx.shape == (2, 2, 5, 2048, 9) and qy.shape == (2, 2, 2048) and cls.shape == (2, 2)


def test_symmetric_noise_episode():
    """'sym' noise (reference dataloaders/loader.py:677-678): noisy shots show another sampled way."""
    from r3dfsseg_b200.episodes import make_episode
    ep = make_episode(9, 3, 5, dataset="scannet", noise_ratio=0.4, noise_type="sym")
    sampled = set(int(c) for c in ep.sampled_classes)
    noisy = ep.gt_support_y.sum(-1) == 0
    assert (noisy.sum(1) == 2).all()
    for w in range(3):
        for k in range(5):
            cls = int(ep.support_flag[w, k])
            if noisy[w, k]:
                assert cls in sampled and cls != int(ep.sampled_classes[w])
            else:
                assert cls == int(ep.sampled_classes[w])
    clean = make_episode(9, 3, 5, dataset="scannet", noise_ratio=0.4)   # default stays 'ood'
    assert not torch.equal(clean.support_flag, ep.support_flag)


def test_pair_and_partial_noise_and_ratio_list():
    """'pair' / 'partial' noise and the train-mode ratio list of the reference's episode sampler
    (dataloaders/loader.py:668-670, 734-747, 241-257, 790-802)."""
    from r3dfsseg_b200.episodes import default_pair_dict, make_episode
    pd = default_pair_dict("scannet")
    ep = make_episode(5, 3, 5, dataset="scannet", noise_ratio=0.4, noise_type="pair")
    noisy = ep.gt_support_y.sum(-1) == 0
    assert (noisy.sum(1) == 2).all()
    for w in range(3):
        c = int(ep.sampled_classes[w])
        for k in range(5):
            want = pd[c] if noisy[w, k] else c
            assert int(ep.support_flag[w, k]) == want
    # partial: the noisy shots show the way's own class, but their mask covers more than that object
    ep = make_episode(6, 2, 5, noise_ratio=0.4, noise_type="partial")
    noisy = ep.gt_support_y.sum(-1) == 0
    assert (noisy.sum(1) == 2).all()
    for w in range(2):
        assert (ep.support_flag[w] == int(ep.sampled_classes[w])).all()
    clean_frac = ep.support_y[~noisy].float().mean()
    noisy_frac = ep.support_y[noisy].float().mean()
    assert noisy_frac > clean_frac               # an extra object is marked foreground
    assert (ep.gt_support_y[~noisy] == ep.support_y[~noisy]).all()
    # a list of ratios draws one per episode (train mode); 0.0 and 0.4 both occur over seeds
    seen = set()
    for seed in range(12):
        e = make_episode(seed, 2, 5, noise_ratio=[0.0, 0.4])
        seen.add(int((e.gt_support_y.sum(-1) == 0).sum(1)[0]))
    assert seen == {0, 2}
    # k_shot - n_noise - 1 == 1: a noise class supplies at most one shot of a way (loader.py:790-793)
    e = make_episode(3, 2, 5, dataset="scannet", noise_ratio=0.6)
    noisy = e.gt_support_y.sum(-1) == 0
    for w in range(2):
        flags = e.support_flag[w][noisy[w]].tolist()
        assert len(flags) == 3 and len(set(flags)) == 3
    with pytest.raises(ValueError):
        make_episode(0, 2, 5, noise_type="bogus")


def test_checkpoint_formats_round_trip_with_the_reference_optimizer(tmp_path):
    """r3dfsseg_b200/checkpoint.py: the fused optimizer's flat moments <-> torch.optim.Adam.state_dict()
    over the reference's four parameter groups (models/mpti_learner.py:26-32), and the reference's
    checkpoint.tar / pre-training files (utils/checkpoint_util.py:10-45)."""
    from r3dfsseg_b200 import checkpoint as ck
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten
    from r3dfsseg_b200.train import PARAM_NAMES, param_layout
    torch.manual_seed(0)
    m = MPTI_SelfAtten(default_args(2, 5))
    named = dict(m.named_parameters())
    assert list(named) == PARAM_NAMES           # reference registration order = optimizer order
    params = [named[n] for n in PARAM_NAMES]
    # the reference's optimizer, stepped once on random gradients
    ref_opt = torch.optim.Adam([{"params": m.encoder.parameters(), "lr": 1e-4},
                                {"params": m.base_learner.parameters()},
                                {"params": m.att_learner.parameters()},
                                {"params": m.proj.parameters()}], lr=1e-3)
    for p in params:
        p.grad = torch.randn_like(p)
    ref_opt.step()
    sd = ref_opt.state_dict()
    offsets, _ = param_layout(9)
    shapes = [p.shape for p in params]
    like = torch.zeros(offsets[-1])
    ea, es, step, lrs = ck.adam_state_from_reference(sd, PARAM_NAMES, shapes, offsets, like)
    assert step == 1 and lrs == (1e-4, 1e-3)
    for i, (p, o) in enumerate(zip(params, offsets)):
        assert torch.equal(ea[o:o + p.numel()].view(p.shape), sd["state"][i]["exp_avg"])
        assert torch.equal(es[o:o + p.numel()].view(p.shape), sd["state"][i]["exp_avg_sq"])
    back = ck.adam_state_to_reference(ea, es, step, PARAM_NAMES, shapes, offsets, lrs)
    assert [g["params"] for g in back["param_groups"]] == [g["params"] for g in sd["param_groups"]]
    assert [g["lr"] for g in back["param_groups"]] == [1e-4, 1e-3, 1e-3, 1e-3]
    fresh = torch.optim.Adam([{"params": m.encoder.parameters(), "lr": 1e-4},
                              {"params": m.base_learner.parameters()},
                              {"params": m.att_learner.parameters()},
                              {"params": m.proj.parameters()}], lr=1e-3)
    fresh.load_state_dict(back)                  # torch accepts what we write
    fs = fresh.state_dict()["state"]
    assert all(torch.equal(fs[i]["exp_avg"], sd["state"][i]["exp_avg"]) for i in range(len(params)))
    assert int(float(fs[0]["step"])) == 1
    # files: checkpoint.tar and the pre-training file
    ck.save_model_checkpoint(m, ref_opt, str(tmp_path), iteration=7, iou=0.5)
    m2 = MPTI_SelfAtten(default_args(2, 5))
    ck.load_model_checkpoint(m2, str(tmp_path), mode="test")
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    pre = tmp_path / "pre.tar"
    torch.save({"params": m.encoder.state_dict()}, pre)
    m3 = MPTI_SelfAtten(default_args(2, 5))
    ck.load_pretrain_checkpoint(m3, str(pre))
    assert torch.equal(m3.encoder.state_dict()["conv.layer.0.weight"],
                       m.encoder.state_dict()["conv.layer.0.weight"])
    assert not torch.equal(m3.proj.weight, m.proj.weight)      # only the encoder is taken
    with pytest.raises(ValueError):
        ck.load_model_checkpoint(m2, str(tmp_path / "nowhere"), mode="test")
    with pytest.raises(ValueError):
        ck.load_pretrain_checkpoint(m3, None)


def test_custom_ops_have_fake_kernels_for_shape_inference():
    """Every op of the `r3dfs::` namespace carries a fake (meta) kernel, so the module code can be
    traced without touching a GPU: shapes/dtypes under FakeTensorMode with CUDA-device fakes."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from r3dfsseg_b200 import ops  # noqa: F401  (registers the ops)
    op = torch.ops.r3dfs
    with FakeTensorMode():
        dev = "cuda"
        f = lambda *s, dt=torch.float32: torch.empty(s, dtype=dt, device=dev)
        E, nw, ks, N, nq = 3, 2, 5, 2048, 2
        w = [f(4)] * 31
        r = op.mpti_forward(w, 9, 20, f(E, nw, ks, 9, N), f(E, nw, ks, N, dt=torch.int32),
                            f(E, nq, 9, N), f(E, nq, N, dt=torch.int64), 100, 200, 1.0, 0.99, True,
                            200, 1e-6, None)
        assert [tuple(t.shape) for t in r] == [(E, nq, N, 3), (E,), (E, nq, N), (E, 3), (E, nw, ks),
                                               (E,), (E,)]
        assert r[2].dtype == torch.int32 and r[0].device.type == "cuda"
        assert op.knn(f(4, 9, 100), 20).shape == (4, 100, 20)
        assert op.edge_feature(f(4, 9, 100), f(4, 100, 20, dt=torch.int64)).shape == (4, 18, 100, 20)
        assert op.edgeconv(f(4, 9, 100), f(64, 18), f(64), f(64), f(64, 64), f(64), f(64), 20).shape \
            == (4, 100, 64)
        assert op.linear(f(1000, 192), f(512, 192), f(512), f(512), 2).shape == (1000, 512)
        assert op.attention(f(4, 100, 256), f(192, 256)).shape == (4, 100, 64)
        assert op.features(f(4, 9, 100), w, 9, 20).shape == (4, 100, 192)
        i32 = torch.int32
        assert op.fps(f(500, 192), f(2, dt=i32), f(2, dt=i32), 101, 0, 0).shape == (2, 101)
        p, c, a, sd = op.multi_prototypes(f(500, 192), f(2, dt=i32), f(2, dt=i32), 100)
        assert p.shape == (2, 101, 192) and c.shape == (2,) and a.shape == (500,) and sd.shape == (2, 101)
        k, cf, cm, cc = op.mdns(f(E, nw, ks, 9, N), f(E, nw, ks, N, dt=i32), f(E, nw * ks * N, 192))
        assert k.shape == (E, nw, ks) and cm.shape == (E, nw, ks, 5, 192) and cc.dtype == i32
        nb, sm = op.affinity_knn(f(2, 700, 192), f(2, 700, dt=torch.uint8), 200, 1.0)
        assert nb.shape == (2, 700, 200) and nb.dtype == i32 and sm.shape == (2, 700, 200)
        z, it, rs = op.label_propagate(nb, sm, f(2, 700, dt=torch.uint8), f(2, 700, 3), 0.99, 1e-6, 200)
        assert z.shape == (2, 700, 3) and it.dtype == i32 and rs.shape == (2,)
