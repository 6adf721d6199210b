"""CPU: the oracle restatement (oracle/mpti_oracle.py) against the golden vectors that were
produced by the reference's own modules (oracle/make_golden.py)."""
import torch

from oracle import mpti_oracle as O
from r3dfsseg_b200.episodes import make_episode
from tests.helpers import knn_sets_match


def test_knn_matches_reference(golden_dgcnn):
    g = golden_dgcnn
    for key in ("x9", "x64"):
        x = g[key]
        idx = O.knn(x, 20)
        ok, bad = knn_sets_match(idx, g["knn_" + key], O.knn_scores(x), largest=True)
        assert ok, f"{key}: {bad} rows differ beyond ties"


def test_edge_feature_matches_reference(golden_dgcnn):
    g = golden_dgcnn
    e = O.get_edge_feature(g["x9"], 20, g["knn_x9"])
    assert torch.equal(e, g["edge_x9"])


def test_dgcnn_matches_reference(golden_dgcnn, fixture_sd):
    g = golden_dgcnn
    l1, l2 = O.dgcnn_forward(g["dgcnn_x"], fixture_sd)
    assert torch.allclose(l1, g["dgcnn_l1"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(l2, g["dgcnn_l2"], rtol=1e-5, atol=1e-6)


def test_fps_count_rule():
    # ceil(fp32(n) * fp32(k/n)) is k or k+1 (SURVEY.md §2.1)
    ks = {O.fps_count(n, 100) for n in range(101, 4000)}
    assert ks == {100, 101}
    assert all(O.fps_count(n, 4) == 4 for n in range(5, 3000))


import pytest


@pytest.mark.parametrize("name", ["s3dis_2way_1shot", "s3dis_2way_5shot_mdns",
                                  "s3dis_2way_5shot_noisy_mdns", "scannet_3way_5shot_ood_mdns"])
def test_episode_matches_reference(golden_episodes, fixture_sd, name):
    c = golden_episodes[name]
    ep = make_episode(c["seed"], c["n_way"], c["k_shot"], dataset=c["dataset"],
                      noise_ratio=c["noise_ratio"])
    with torch.no_grad():
        out = O.forward_episode(fixture_sd, ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                                eval_mdns=c["eval"])
    ref = c["query_pred"]
    assert out["num_prototypes"] == c["num_prototypes"]
    if c["eval"]:
        assert torch.equal(out["clean_flag"], c["clean_flag"])
    err = (out["query_pred"] - ref).abs().max() / ref.abs().max()
    assert err < 1e-3, err
    agree = (out["query_pred"].argmax(1) == ref.argmax(1)).float().mean()
    assert agree >= 0.999, agree
    assert abs(float(out["loss"]) - float(c["loss"])) < 1e-4


def test_train_oracle_vs_reference_golden(fixture_sd):
    """oracle/mpti_train_oracle.py (training forward + autograd) against the numbers the REFERENCE's
    own forward(train=True) + backward produced (oracle/make_golden_train.py)."""
    import os
    from oracle import mpti_train_oracle as TO
    torch.set_num_threads(os.cpu_count())
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "golden_train.pt"))
    name = "train_s3dis_2way_5shot_clean"
    g = gold[name]
    ep = make_episode(g["seed"], g["n_way"], g["k_shot"], dataset=g["dataset"],
                      noise_ratio=g["noise_ratio"])
    P, running = TO.split_state_dict(fixture_sd)
    out = TO.forward_train(P, ep.support_x, ep.support_y, ep.query_x, ep.query_y, ep.support_flag,
                           running=running)
    (out["lp_loss"] + 0.1 * out["contrast_loss"]).backward()
    assert abs(float(out["lp_loss"]) - float(g["lp_loss"])) < 1e-5
    assert abs(float(out["contrast_loss"]) - float(g["contrast_loss"])) < 1e-5
    for k, p in P.items():
        if k.endswith("0.bias") and k.startswith("base_learner"):
            continue  # exactly-zero gradient (bias ahead of batch-stat BN): rounding noise only
        s = p.grad.reshape(-1)[::29]
        ref = g["grad_sample"][k]
        assert float((s - ref).abs().max()) <= 2e-5 * float(ref.abs().max()) + 1e-8, k
    for k, v in running.items():
        if v.dtype.is_floating_point:
            ref = g["running"][k]
            assert float((v - ref).abs().max()) < 1e-5 * max(1.0, float(ref.abs().max())), k
        else:
            assert int(v) == int(g["running"][k])


@pytest.mark.parametrize("name", ["s3dis_2way_5shot_noisy", "scannet_3way_5shot_ood",
                                  "s3dis_2way_1shot"])
def test_protonet_oracle_matches_reference(fixture_sd, name):
    """oracle/protonet_oracle.py against the REFERENCE's ProtoNet_Contrast.forward (eval) outputs
    (models/protonet.py:780-858; written by `python -m oracle.make_golden protonet`)."""
    import os
    from oracle import protonet_oracle as PO
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "golden_protonet.pt"))
    c = gold[name]
    ep = make_episode(c["seed"], c["n_way"], c["k_shot"], dataset=c["dataset"],
                      noise_ratio=c["noise_ratio"])
    with torch.no_grad():
        out = PO.forward_episode(fixture_sd, ep.support_x, ep.support_y, ep.query_x, ep.query_y)
    assert torch.equal(out["clean_flag"], c["clean_flag"])
    ref = c["query_pred"]
    err = (out["query_pred"] - ref).abs().max() / ref.abs().max()
    assert err < 1e-5, err
    assert torch.equal(out["query_pred"].argmax(1), ref.argmax(1))
    assert abs(float(out["loss"]) - float(c["loss"])) < 1e-5


# ---------------------------------------------------------------------------------------------
# pins added in round 2
# ---------------------------------------------------------------------------------------------
def test_mdns_internals_pinned_to_reference():
    """O.grid_sampling / O.mdns_flags_one_scale / O.mdns_multi_scale against what the reference's
    own methods (models/mpti.py:316-371, 87-176, 178-223) return on support sets whose foreground
    points lie exactly on cell faces (inclusive bounds on both sides, later cells overwrite
    assignments); stored in tests/golden/golden_mdns.pt by `python -m oracle.make_golden mdns`."""
    import os
    from tests.helpers import mdns_case
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "golden_mdns.pt"))
    assert len(gold) == 3
    for g in gold.values():
        n_way, k_shot = g["n_way"], g["k_shot"]
        sx, sy, sf = mdns_case(g["seed"], n_way, k_shot)
        for (nx, ny, nz) in ((1, 1, 1), (2, 2, 1)):
            ref = g["scales"]["%dx%dx%d" % (nx, ny, nz)]
            for w in range(n_way):
                for k in range(k_shot):
                    fg = sy[w, k] == 1
                    sp, f = sx[w, k][:, fg].t(), sf[w, k][:, fg].t()
                    cell = ref["cells"][w * k_shot + k]
                    s, a, n = O.grid_sampling(sp, f, nx, ny, nz)
                    assert n == cell["count"] and torch.equal(a, cell["assign"].long())
                    assert torch.equal(s, cell["seeds"])
            assert torch.equal(O.mdns_flags_one_scale(sf, sy, sx, nx, ny, nz), ref["flag"])
        pl, clean = O.mdns_multi_scale(sf, sy, sx)
        assert torch.equal(clean, g["clean"])
        assert len(pl) == len(g["pl"]) and all(torch.equal(a, b) for a, b in zip(pl, g["pl"]))


def _metric_case(seed=0, n_eps=7, n_way=3, n_q=3, N=257, pool=6):
    import numpy as np
    r = np.random.default_rng(seed)
    test_classes = sorted(r.choice(13, size=pool, replace=False).tolist())
    preds, gts, l2c = [], [], []
    for _ in range(n_eps):
        l2c.append(r.choice(test_classes, size=n_way, replace=False))
        gts.append(r.integers(0, n_way + 1, size=(n_q, N)))
        p = gts[-1].copy()
        flip = r.uniform(size=p.shape) < 0.3
        p[flip] = r.integers(0, n_way + 1, size=int(flip.sum()))
        preds.append(p)
    return preds, gts, l2c, test_classes


def test_confusion_counts_golden():
    """O.confusion_counts + O.mean_iou == the reference's evaluate_metric (eval_noise.py:23-72),
    per-class IoU included (read from its log lines), from the committed numbers
    (tests/golden/golden_metric.json, written by `python -m oracle.make_golden metric`)."""
    import json
    import os
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_metric.json")))
    preds, gts, l2c, test_classes = _metric_case(**g["case"])
    assert test_classes == g["test_classes"]
    counters = O.confusion_counts(preds, gts, l2c, test_classes)
    assert abs(O.mean_iou(counters) - g["mean_iou"]) < 1e-12
    gt, pos, tp = counters.astype(float)
    assert len(g["iou"]) == counters.shape[1]
    for c, v in enumerate(g["iou"]):
        assert abs(tp[c] / (gt[c] + pos[c] - tp[c]) - v) < 1e-6


def test_trained_fixture_loss_matches_oracle(fixture_sd):
    """tests/golden/weights_fixture.pt was meta-trained by the CUDA training path
    (scripts/train_fixture.py).  The losses that path reported for one more training forward on a
    fixed episode (dropout off) must be what the CPU training oracle computes from the same weights."""
    import json
    import os
    from oracle import mpti_train_oracle as TO
    log = json.load(open(os.path.join(os.path.dirname(__file__), "golden",
                                      "weights_fixture_train_log.json")))
    assert log["eval_after"]["s3dis_2way_clean"][0] > 0.9 > 0.5 > log["eval_before"]["s3dis_2way_clean"][0]
    chk = log["check"]
    torch.set_num_threads(os.cpu_count())
    ep = make_episode(chk["seed"], 2, 5, noise_ratio=chk["noise_ratio"])
    P, running = TO.split_state_dict(fixture_sd)
    with torch.no_grad():
        out = TO.forward_train(P, ep.support_x, ep.support_y, ep.query_x, ep.query_y, ep.support_flag,
                               running=None)
    # free-running (kNN / FPS ties may flip): same bar as tests/test_gpu_train.py
    assert abs(float(out["lp_loss"]) - chk["lp_loss"]) < 2e-3 * max(1.0, abs(chk["lp_loss"]))
    assert abs(float(out["contrast_loss"]) - chk["contrast_loss"]) < 2e-3 * chk["contrast_loss"]
