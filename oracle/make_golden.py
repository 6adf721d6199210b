"""TEST INFRASTRUCTURE.  Generates tests/golden/*.pt by running the REFERENCE's own modules
(imported unmodified from /root/reference under oracle/ref_shims.py) on seeded synthetic inputs.
Build container only.  Run:  python -m oracle.make_golden

Files (small on purpose; episodes are regenerated from their seed, only outputs are stored):
  golden_dgcnn.pt      knn / get_edge_feature / DGCNN.forward on small random clouds
  golden_episodes.pt   MPTI_SelfAtten.forward outputs for the three episode configurations
  golden_protonet.pt   ProtoNet_Contrast.forward (eval) outputs; `python -m oracle.make_golden protonet`
                       writes only this file
  golden_metric.json   evaluate_metric on a seeded random case (`python -m oracle.make_golden metric`)
  golden_mdns.pt       grid_sampling / Mean_pl_support_y / Mean_pl_support_y_multi_scale on the
                       support sets of tests.helpers.mdns_case (`python -m oracle.make_golden mdns`).
                       The committed file was written through the oracle's restatements of those
                       three methods, which the reference's own methods matched bit for bit on
                       these inputs (the comparison was run live against the reference tree)
  golden_parity.pt     free-running parity cases (`python -m oracle.make_golden parity`): for the
                       four episode configurations above plus 10 seeds each of BASELINE.json
                       configs[2] (S3DIS-shape 2-way 5-shot) and configs[3] (ScanNet-shape 3-way
                       5-shot, 40 % OOD shots), the reference's FP32 logits and the FP64
                       adjudicator's logits (oracle.mpti_oracle.forward_episode_fp64)
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402
from r3dfsseg_b200.episodes import default_args, make_episode  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

EPISODE_CASES = [
    # name, seed, n_way, k_shot, dataset, noise_ratio, eval(MDNS)
    ("s3dis_2way_1shot", 0, 2, 1, "s3dis", 0.0, False),
    ("s3dis_2way_5shot_mdns", 1, 2, 5, "s3dis", 0.0, True),
    ("s3dis_2way_5shot_noisy_mdns", 3, 2, 5, "s3dis", 0.4, True),
    ("scannet_3way_5shot_ood_mdns", 2, 3, 5, "scannet", 0.4, True),
]


PROTONET_CASES = [
    ("s3dis_2way_5shot_noisy", 3, 2, 5, "s3dis", 0.4),
    ("scannet_3way_5shot_ood", 2, 3, 5, "scannet", 0.4),
    ("s3dis_2way_1shot", 0, 2, 1, "s3dis", 0.0),
]


def protonet(ref, sd):
    """ProtoNet_Contrast (models/protonet.py:357) in eval: query_pred, loss, clean flags."""
    out = {}
    for name, seed, n_way, k_shot, ds, noise in PROTONET_CASES:
        args = default_args(n_way, k_shot, dist_method="cosine")
        m = ref.protonet.ProtoNet_Contrast(args)
        m.load_state_dict(sd)
        m.eval()
        ep = make_episode(seed, n_way, k_shot, dataset=ds, noise_ratio=noise)
        with torch.no_grad(), ref_shims.quiet():
            pred, loss = m(ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                           gt_support_y=ep.gt_support_y)
            sf = m.getFeatures(ep.support_x.reshape(n_way * k_shot, 9, -1)).view(
                n_way, k_shot, 192, -1)
            _, clean = m.Mean_pl_support_y_multi_scale(sf, ep.support_y, ep.gt_support_y,
                                                       ep.support_x)
        out[name] = dict(seed=seed, n_way=n_way, k_shot=k_shot, dataset=ds, noise_ratio=noise,
                         query_pred=pred.contiguous().clone(), loss=loss.clone(),
                         clean_flag=clean.clone())
        print(name, "loss", float(loss), "acc",
              float((pred.argmax(1) == ep.query_y).float().mean()), "clean", clean.tolist())
    torch.save(out, os.path.join(GOLD, "golden_protonet.pt"))
    print("golden_protonet.pt written")


PARITY_CASES = list(EPISODE_CASES) \
    + [("s3dis_2way_5shot_seed%d" % s, s, 2, 5, "s3dis", 0.0, True) for s in range(100, 110)] \
    + [("scannet_3way_5shot_ood_seed%d" % s, s, 3, 5, "scannet", 0.4, True) for s in range(200, 210)]


def parity(ref, sd):
    """Reference FP32 logits + FP64 adjudicator logits per free-running parity case."""
    from oracle import mpti_oracle as O
    out = {}
    for name, seed, n_way, k_shot, ds, noise, ev in PARITY_CASES:
        m = ref.mpti.MPTI_SelfAtten(default_args(n_way, k_shot))
        m.load_state_dict(sd)
        m.eval()
        ep = make_episode(seed, n_way, k_shot, dataset=ds, noise_ratio=noise)
        with torch.no_grad(), ref_shims.quiet():
            pred, loss = m(ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                           gt_support_y=ep.gt_support_y, eval=ev)
            clean = None
            if ev:
                sf = m.getFeatures(ep.support_x.reshape(n_way * k_shot, 9, -1)).view(
                    n_way, k_shot, 192, -1)
                _, clean = m.Mean_pl_support_y_multi_scale(sf, ep.support_y, ep.gt_support_y,
                                                           ep.support_x)
            adj = O.forward_episode_fp64(sd, ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                                         eval_mdns=ev)
        p64 = adj["query_pred"]
        rel = float((pred.double() - p64).abs().max() / p64.abs().max())
        agree = float((pred.argmax(1) == p64.argmax(1)).float().mean())
        out[name] = dict(seed=seed, n_way=n_way, k_shot=k_shot, dataset=ds, noise_ratio=noise,
                         eval=ev, query_pred=pred.contiguous().clone(), loss=loss.clone(),
                         query_pred_fp64=p64.float().contiguous().clone(),
                         loss_fp64=adj["loss"].float().clone(),
                         clean_flag=clean, clean_flag_fp64=adj["clean_flag"],
                         proto_count_fp64=adj["proto_count"],
                         num_prototypes=int(m.num_prototypes))
        print(name, "loss", float(loss), "fp64", float(adj["loss"]), "ref32 vs fp64: max rel",
              "%.2e" % rel, "labels", "%.5f" % agree, "acc",
              float((pred.argmax(1) == ep.query_y).float().mean()), flush=True)
    torch.save(out, os.path.join(GOLD, "golden_parity.pt"))
    print("golden_parity.pt written")


def metric(ref):
    """evaluate_metric (eval_noise.py:23-72) on a seeded random case -> golden_metric.json."""
    import json
    import re
    from tests.test_oracle_golden import _metric_case
    case = dict(seed=0, n_eps=7, n_way=3, n_q=3, N=257, pool=6)
    preds, gts, l2c, test_classes = _metric_case(**case)

    class Log:
        lines = []

        def cprint(self, s):
            self.lines.append(s)

    miou = float(ref.evaluate_metric(Log(), preds, gts, l2c, test_classes))
    ious = [float(re.search(r"IoU: ([0-9.]+)", s).group(1)) for s in Log.lines if "IoU:" in s]
    with open(os.path.join(GOLD, "golden_metric.json"), "w") as f:
        json.dump(dict(case=case, test_classes=test_classes, mean_iou=miou, iou=ious), f)
    print("golden_metric.json written", miou)


MDNS_CASES = [(0, 2, 5), (1, 3, 5), (2, 2, 1)]  # (seed, n_way, k_shot) of tests.helpers.mdns_case
MDNS_SCALES = [(1, 1, 1), (2, 2, 1)]


def mdns(model_of):
    """Noise-suppression internals (models/mpti.py:87-223, 316-371) on support sets whose
    foreground points lie exactly on cell faces.  `model_of(n_way, k_shot)` returns an object with
    the reference's grid_sampling / Mean_pl_support_y / Mean_pl_support_y_multi_scale methods."""
    from tests.helpers import mdns_case
    out = {}
    for seed, n_way, k_shot in MDNS_CASES:
        sx, sy, sf = mdns_case(seed, n_way, k_shot)
        m = model_of(n_way, k_shot)
        case = dict(seed=seed, n_way=n_way, k_shot=k_shot, scales={})
        for scale in MDNS_SCALES:
            cells = []
            for w in range(n_way):
                for k in range(k_shot):
                    fg = sy[w, k] == 1
                    s, a, n = m.grid_sampling(sx[w, k][:, fg].t(), sf[w, k][:, fg].t(), *scale)
                    # cell indices < 4: int8 keeps the file small; tests compare after .long()
                    cells.append(dict(seeds=s.clone(), assign=a.to(torch.int8).cpu(), count=int(n)))
            with ref_shims.quiet():
                flag = m.Mean_pl_support_y(sf, sy, sy, sx, *scale)[1]
            case["scales"]["%dx%dx%d" % scale] = dict(cells=cells, flag=flag.clone())
        with ref_shims.quiet():
            pl, clean = m.Mean_pl_support_y_multi_scale(sf, sy, sy, sx)
        case.update(pl=[p.clone() for p in pl], clean=clean.clone())
        out["seed%d_%dway_%dshot" % (seed, n_way, k_shot)] = case
    torch.save(out, os.path.join(GOLD, "golden_mdns.pt"))
    print("golden_mdns.pt written")


def main():
    ref = ref_shims.load_reference()
    torch.set_num_threads(os.cpu_count())
    sd = torch.load(os.path.join(GOLD, "weights_fixture.pt"))
    if sys.argv[1:] == ["metric"]:
        return metric(ref)
    if sys.argv[1:] == ["mdns"]:
        return mdns(lambda n_way, k_shot: ref.mpti.MPTI_SelfAtten(default_args(n_way, k_shot)))
    if sys.argv[1:] == ["protonet"]:
        return protonet(ref, sd)
    if sys.argv[1:] == ["parity"]:
        return parity(ref, sd)

    # ---- DGCNN pieces -----------------------------------------------------------------------
    g = torch.Generator().manual_seed(7)
    x9 = torch.rand((2, 9, 256), generator=g)
    x64 = torch.randn((2, 64, 256), generator=g)
    out = {"x9": x9, "x64": x64}
    out["knn_x9"] = ref.dgcnn.knn(x9, 20)
    out["knn_x64"] = ref.dgcnn.knn(x64, 20)
    out["edge_x9"] = ref.dgcnn.get_edge_feature(x9, K=20, idx=out["knn_x9"])
    enc = ref.dgcnn.DGCNN([[64, 64]] * 3, [512, 256], 9, k=20)
    enc.load_state_dict({k[len("encoder."):]: v for k, v in sd.items() if k.startswith("encoder.")})
    enc.eval()
    xe = torch.rand((2, 9, 512), generator=g)
    with torch.no_grad():
        l1, l2 = enc(xe)
    out.update(dgcnn_x=xe, dgcnn_l1=l1, dgcnn_l2=l2)
    torch.save(out, os.path.join(GOLD, "golden_dgcnn.pt"))
    print("golden_dgcnn.pt written")

    # ---- episodes ---------------------------------------------------------------------------
    eps = {}
    for name, seed, n_way, k_shot, ds, noise, ev in EPISODE_CASES:
        args = default_args(n_way, k_shot)
        m = ref.mpti.MPTI_SelfAtten(args)
        m.load_state_dict(sd)
        m.eval()
        ep = make_episode(seed, n_way, k_shot, dataset=ds, noise_ratio=noise)
        with torch.no_grad(), ref_shims.quiet():
            pred, loss = m(ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                           gt_support_y=ep.gt_support_y, eval=ev)
            feat_q = m.getFeatures(ep.query_x[:1])
            clean = None
            if ev:
                sf = m.getFeatures(ep.support_x.reshape(n_way * k_shot, 9, -1)).view(
                    n_way, k_shot, 192, -1)
                _, clean = m.Mean_pl_support_y_multi_scale(sf, ep.support_y, ep.gt_support_y,
                                                           ep.support_x)
        eps[name] = dict(seed=seed, n_way=n_way, k_shot=k_shot, dataset=ds, noise_ratio=noise,
                         eval=ev, query_pred=pred.contiguous().clone(), loss=loss.clone(),
                         num_prototypes=int(m.num_prototypes), clean_flag=clean,
                         query0_feat_sub=feat_q[0, :, ::8].contiguous().clone())
        print(name, "loss", float(loss), "P", m.num_prototypes,
              "acc", float((pred.argmax(1) == ep.query_y).float().mean()),
              "clean", None if clean is None else clean.tolist())
    torch.save(eps, os.path.join(GOLD, "golden_episodes.pt"))
    print("golden_episodes.pt written")
    protonet(ref, sd)


if __name__ == "__main__":
    main()
