import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from r3dfsseg_b200.episodes import default_args, make_episode
from r3dfsseg_b200.models import MPTI_SelfAtten
sd = torch.load(os.path.join(ROOT, "tests/golden/weights_fixture.pt"))
gold = torch.load(os.path.join(ROOT, "tests/golden/golden_parity.pt"))
for name in ("s3dis_2way_1shot", "s3dis_2way_5shot_mdns"):
    c = gold[name]
    m = MPTI_SelfAtten(default_args(c["n_way"], c["k_shot"])); m.load_state_dict(sd); m = m.cuda().eval()
    ep = make_episode(c["seed"], c["n_way"], c["k_shot"], dataset=c["dataset"], noise_ratio=c["noise_ratio"])
    pred, loss = m(ep.support_x.cuda(), ep.support_y.cuda(), ep.query_x.cuda(), ep.query_y.cuda(), gt_support_y=ep.gt_support_y.cuda(), eval=c["eval"])
    ref = c["query_pred"]
    print(name, "err", float((pred.cpu() - ref).abs().max() / ref.abs().max()), "iters", int(m._last_diag["cg_iters"][0]), "resid", float(m._last_diag["cg_resid"][0]))
