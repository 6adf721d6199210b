"""Selection / in-edge kernels of the affinity graph on the same inputs under different A/B switches.
    python scripts/check_select.py run OUT.pt [n] [G] [case]     (one process per switch setting)
    python scripts/check_select.py cmp A.pt B.pt
    python scripts/check_select.py cand [n] [G] [case]     (candidates of the bounded select per row)
Graph 1 has fewer valid nodes than k (the filler path), graph 2 a block of invalid nodes.  Cases:
"base" (the default); "dup": 1200 equal feature rows in graph 0 (1199 keys tie at 0 in their rows,
more candidates than the bounded select's buffer holds); "exact_k": graph 1 has k valid nodes and
graph 2 k + 1 (every row has exactly k others)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

D, k = 192, 200


def inputs(n, G, case):
    g = torch.Generator().manual_seed(0)
    centers = torch.randn((6, D), generator=g) * 0.15
    feat = centers[torch.randint(0, 6, (G, n), generator=g)] + torch.randn((G, n, D), generator=g) * 0.06
    feat[0, 5] = feat[0, 900]          # exact duplicates -> ties at distance 0 and at the cut
    feat[0, 6] = feat[0, 900]
    valid = torch.ones((G, n), dtype=torch.uint8)
    valid[:, 300:320] = 0
    if G > 1:
        valid[1] = 0
        valid[1, 10:160] = 1           # 150 valid nodes < k
    if case == "dup":
        feat[0, 1000:2200] = feat[0, 1000]
    elif case == "exact_k":
        valid[1:3] = 0
        valid[1, 7:7 + k] = 1
        if G > 2:
            valid[2, 3:3 + 7 * (k + 1):7] = 1
    else:
        assert case == "base", case
    return feat, valid


mode = sys.argv[1]
if mode == "run":
    from r3dfsseg_b200 import ops
    out = sys.argv[2]
    n = int(sys.argv[3]) if len(sys.argv) > 3 else 2368
    G = int(sys.argv[4]) if len(sys.argv) > 4 else 25
    feat, valid = inputs(n, G, sys.argv[5] if len(sys.argv) > 5 else "base")
    feat, valid = feat.cuda(), valid.cuda()
    for _ in range(3):
        nbr, sim = ops.affinity_knn(feat, valid, k, 1.0)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(5):
        nbr, sim = ops.affinity_knn(feat, valid, k, 1.0)
    t1.record()
    torch.cuda.synchronize()
    Y = torch.zeros((G, n, 3), device="cuda")
    Y[:, :100, 0] = 1
    Y[:, 100:200, 1] = 1
    Y[:, 200:300, 2] = 1
    Z, iters, resid = ops.label_propagate(nbr, sim, valid, Y)
    print("affinity ms", t0.elapsed_time(t1) / 5, "cg iters", iters.tolist()[:4])
    torch.save({"nbr": nbr.cpu(), "sim": sim.cpu(), "valid": valid.cpu(), "Z": Z.cpu()}, out)
elif mode == "cand":
    # what the bounded select (csrc/lp.cu) keeps per row: the real columns whose distance is at most
    # the k-th smallest minimum over groups of 8 columns, with distances from an FP64 Gram matrix
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 4416
    G = int(sys.argv[3]) if len(sys.argv) > 3 else 25
    feat, valid = inputs(n, G, sys.argv[4] if len(sys.argv) > 4 else "base")
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    cnts, unbounded, rows = [], 0, 0
    for gi in range(G):
        f = feat[gi].to(dev, torch.float64)
        sq = (f * f).sum(1)
        d2 = sq[:, None] + sq[None, :] - 2.0 * f @ f.T
        real = valid[gi].to(dev).bool()[None, :].expand(n, n).clone()
        real.fill_diagonal_(False)
        d2 = torch.where(real, d2, torch.full_like(d2, float("inf")))
        gm = torch.nn.functional.pad(d2, (0, (-n) % 8), value=float("inf")).view(n, -1, 8).amin(2)
        tau = gm.kthvalue(k, dim=1).values if gm.shape[1] >= k else torch.full_like(sq, float("inf"))
        vr = valid[gi].to(dev).bool()
        ok = vr & torch.isfinite(tau)
        unbounded += int((vr & ~ok).sum())
        rows += int(vr.sum())
        cnts.append((d2 <= tau[:, None]).sum(1)[ok].cpu())
    c = torch.cat(cnts).double()
    q = torch.quantile(c, torch.tensor([0.5, 0.9, 0.99, 0.999], dtype=torch.float64))
    print(f"n {n} G {G}: rows {rows}, candidates per row mean {float(c.mean()):.1f} median "
          f"{float(q[0]):.0f} p90 {float(q[1]):.0f} p99 {float(q[2]):.0f} p99.9 {float(q[3]):.0f} "
          f"max {int(c.max())}; over 1024: {int((c > 1024).sum())}; no bound: {unbounded}")
else:
    a, b = torch.load(sys.argv[2]), torch.load(sys.argv[3])
    v = a["valid"].bool()
    same = (a["nbr"] == b["nbr"])[v]
    za, zb = torch.nan_to_num(a["Z"], nan=-1.0), torch.nan_to_num(b["Z"], nan=-1.0)
    ok = bool(same.all()) and torch.equal(a["sim"][v], b["sim"][v]) and torch.equal(za, zb)
    print("rows", int(v.sum()), "identical rows", int(same.all(-1).sum()),
          "sim equal", bool(torch.equal(a["sim"][v], b["sim"][v])), "Z equal", torch.equal(za, zb))
    sys.exit(0 if ok else 1)
