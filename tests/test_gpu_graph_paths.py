"""The graph half of an episode away from the benchmark's shapes, against FP64.

`launch_affinity` picks one of five kNN-200 selects and one of two distance GEMMs from n, k and the
alignment of its inputs; `launch_lp_solve` picks the padded class width (NCV = 4 or 8) and the
cluster size from n_cls, n and the batch; `cg_pack_kernel` decides per graph between the packed
rows and the plain warp-per-row product.  Every case here names the path it is there for, checks
under torch.profiler that the intended kernel ran where a kernel name tells the path apart, and
compares with a plain FP64 restatement of the same operation.  The episode cases run 4- to 7-way
episodes (n_cls 5..8) inside the node limit of the CG solve, and the boundary cases check that
configurations past it are refused before any kernel is launched."""
import math

import pytest
import torch

from oracle import mpti_oracle as O
from r3dfsseg_b200.episodes import default_args, make_episode
from tests.helpers import knn_sets_match

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# launch_affinity's constants (csrc/lp.cu, csrc/common.cuh)
AFF_GROUP, SELB_CAP, SEL_THREADS = 8, 1024, 256
# launch_lp_solve / cg_pack_kernel's constants (csrc/lp.cu)
CGC_MAXT, CG_MAXPASS, CG_SEGR, CG_MAXPART = 1024, 3, 48, 1024


def _launched(fn):
    """fn() under the profiler; returns (its result, the names of every event recorded)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _ran(names, kernel):
    return any(kernel in s for s in names)


# ---------------------------------------------------------------------------------------------
# affinity kNN
# ---------------------------------------------------------------------------------------------
SELECTS = {"warp40": "knn_select_warp_kernel<40>", "warp80": "knn_select_warp_kernel<80>",
           "reg256": "knn_select_reg_kernel<20, 256>", "reg512": "knn_select_reg_kernel<20, 512>",
           "radix": "knn_select_kernel(", "bounded": "knn_select_bounded_kernel"}


def _select_choice(n, k, valid_aligned=True, feat_aligned=True):
    """launch_affinity's choice of select, restated (the bounded one needs the group minima of
    the TMA distance GEMM, n % 4 == 0, a 4-byte aligned valid mask and bounded_select_pays)."""
    groups = (n + AFF_GROUP - 1) // AFF_GROUP
    pays = groups > k and n * (1.0 - (1.0 - k / groups) ** (1.0 / AFF_GROUP)) <= SELB_CAP / 2
    if pays and n % 4 == 0 and valid_aligned and feat_aligned:
        return "bounded"
    if n <= 32 * 80:
        return "warp40" if n <= 32 * 40 else "warp80"
    if n <= 31 * SEL_THREADS:
        return "reg256" if n <= 19 * SEL_THREADS else "reg512"
    return "radix"


def _graph_inputs(G, n, D, seed, n_valid):
    """G graphs of clustered features with distinct seeds.  Graph b has n_valid[b] valid nodes:
    an invalid block and an invalid tail, or (few valid nodes) valid nodes spread evenly.  Exact
    duplicates for ties: a block of 40 copies of one row and 30 pairs."""
    g = torch.Generator().manual_seed(seed)
    feat = torch.empty((G, n, D))
    valid = torch.zeros((G, n), dtype=torch.uint8)
    for b in range(G):
        centers = torch.randn((6, D), generator=g) * 0.15
        f = centers[torch.randint(0, 6, (n,), generator=g)] + torch.randn((n, D), generator=g) * 0.06
        f[100:140] = f[99]
        f[200:260:2] = f[201:261:2]
        feat[b] = f
        nv = n_valid[b]
        if 2 * nv < n:   # evenly spread: blocks of invalid nodes between the valid ones
            valid[b, torch.linspace(0, n - 1, nv).round().long()] = 1
        else:            # an invalid block [300, 300 + gap), then an invalid tail
            gap = min(96, n - nv)
            valid[b, :nv + gap] = 1
            valid[b, 300:300 + gap] = 0
        assert int(valid[b].sum()) == nv
    return feat, valid


AFF_CASES = [  # (n, k, sigma, expected select, variant)
    (1200, 200, 1.0, "warp40", None),
    (2370, 200, 0.5, "warp80", None),
    (4418, 200, 2.0, "reg256", None),
    (6546, 200, 1.0, "reg512", None),
    (8190, 200, 0.5, "radix", None),
    (4416, 200, 1.0, "bounded", None),
    (6544, 200, 2.0, "bounded", None),
    (8192, 200, 1.0, "bounded", None),
    (4416, 200, 0.5, "reg256", "valid+1"),
    (4416, 200, 2.0, "reg256", "feat+4"),
    (4416, 1000, 1.0, "reg256", None),
    (2560, 100, 2.0, "bounded", None),
]


@pytest.mark.parametrize("n,k,sigma,expect,variant", AFF_CASES)
def test_affinity_knn_paths_vs_fp64(n, k, sigma, expect, variant):
    """warp<40> / warp<80> / reg<20> / reg<20, 512> / radix / bounded select (and, for 'feat+4',
    the register-fed distance GEMM) against the FP64 exact kNN of each of 3 graphs."""
    from r3dfsseg_b200 import ops
    assert _select_choice(n, k, variant != "valid+1", variant != "feat+4") == expect
    G, D = 3, 192
    # graph 2 has fewer than k valid nodes: its rows hold every other valid node
    feat, valid = _graph_inputs(G, n, D, seed=n + k, n_valid=[n - 7, n - 300, min(150, k - 1)])
    feat_d, valid_d = feat.to(DEV), valid.to(DEV)
    if variant == "valid+1":   # a view one byte into a larger buffer
        buf = torch.zeros(G * n + 1, dtype=torch.uint8, device=DEV)
        valid_d = buf[1:].view(G, n)
        valid_d.copy_(valid)
    if variant == "feat+4":    # a view 4 bytes into a larger buffer: TMA cannot address it
        buf = torch.zeros(G * n * D + 1, device=DEV)
        feat_d = buf[1:].view(G, n, D)
        feat_d.copy_(feat)
    (nbr, sim), names = _launched(lambda: ops.affinity_knn(feat_d, valid_d, k, sigma))
    for key, kern in SELECTS.items():
        assert _ran(names, kern) == (key == expect), (key, expect, sorted(names))
    dist = "linear_tc_kernel<" if variant == "feat+4" else "linear_ts_kernel<"
    assert _ran(names, dist), (dist, sorted(names))
    for b in range(G):
        f = feat_d[b].double()
        v = valid_d[b].bool()
        vi = torch.nonzero(v).flatten()
        sq = (f * f).sum(1)
        d2 = (sq[:, None] + sq[None, :] - 2.0 * (f @ f.t())).clamp_min(0)
        d2[:, ~v] = float("inf")
        d2.fill_diagonal_(float("inf"))
        got = nbr[b, vi].long()
        keep = v[got] & (got != vi[:, None])          # valid neighbours other than the node
        if len(vi) <= k:   # fewer than k + 1 valid nodes (outside the k < #valid contract): the
            # row holds every other valid node once; the slots past them are not specified
            hits = torch.zeros((len(vi), n), device=DEV)
            hits.scatter_add_(1, got, keep.float())
            other = v[None, :].expand(len(vi), n).float().clone()
            other[torch.arange(len(vi), device=DEV), vi] = 0
            assert torch.equal(hits, other), b
        else:
            assert keep.all()                          # only valid neighbours, no self edges
            ref = torch.topk(d2[vi], k, dim=1, largest=False).indices
            diff = torch.nonzero((got.sort(1)[0] != ref.sort(1)[0]).any(1)).flatten()
            if len(diff):
                ok, bad = knn_sets_match(got[diff], ref[diff], d2[vi[diff]], largest=False)
                assert ok, f"graph {b}: {bad} rows differ beyond ties"
        # similarity of the pair the kernel returned: exp(-0.5 ||f_i - f_j + 1e-6||^2 / sigma^2),
        # compared on d2 = -2 sigma^2 log(sim) (FP32 rounding of the 192-term sum)
        rows = vi[:, None].expand_as(got)[keep]
        cols = got[keep]
        d2_ref = ((f[rows] - f[cols] + 1e-6) ** 2).sum(1)
        d2_got = -2.0 * sigma ** 2 * torch.log(sim[b, vi][keep].double())
        assert torch.allclose(d2_got, d2_ref, rtol=2e-5, atol=2e-5), \
            float((d2_got - d2_ref).abs().max())


# ---------------------------------------------------------------------------------------------
# label propagation
# ---------------------------------------------------------------------------------------------
def _lp_graph(n, k, seed, kind="random", n_invalid=0, hubs=150):
    """(nbr, sim, valid) of one graph on the GPU, nbr pointing at valid nodes only.
    random: k random valid neighbours; ring: the k nearest ring positions; hub: rows 0..hubs-1
    are in every row's list, the rest of the list random."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    valid = torch.ones(n, dtype=torch.uint8, device=DEV)
    if n_invalid:
        s = 500 + (seed * 37) % 200
        valid[s:s + n_invalid] = 0
    vb = valid.bool()
    idx = torch.arange(n, device=DEV)
    if kind == "ring":
        off = torch.cat([torch.arange(1, k // 2 + 1), -torch.arange(1, k // 2 + 1)]).to(DEV)
        nbr = (idx[:, None] + off[None, :]) % n
        assert vb.all()
    else:
        score = torch.rand((n, n), generator=g, device=DEV)
        if kind == "hub":
            score[:, :hubs] += 2.0
        score[:, ~vb] = -1.0
        score[idx, idx] = -1.0
        nbr = score.topk(k, dim=1).indices
        del score
    sim = 0.05 + 0.95 * torch.rand((n, k), generator=g, device=DEV)
    return nbr.to(torch.int32), sim, valid


def _lp_reference(nbr, sim, valid, alpha=0.99):
    """FP64 (I - alpha S) on the valid nodes (dense), its LU factors, and the valid index."""
    n, k = nbr.shape
    vi = torch.nonzero(valid.bool()).flatten()
    W = torch.zeros((n, n), dtype=torch.float64, device=DEV)
    rows = torch.arange(n, device=DEV)[:, None].expand(n, k)
    W.index_put_((rows[vi], nbr[vi].long()), sim[vi].double(), accumulate=True)
    W = W + W.t()
    W.fill_diagonal_(0)
    W = W[vi][:, vi]
    d = W.sum(1) + 2.220446049250313e-16
    dsi = d.rsqrt()
    M = torch.eye(len(vi), dtype=torch.float64, device=DEV) - alpha * (dsi[:, None] * W * dsi[None, :])
    return M, torch.linalg.lu_factor(M), vi


def _check_lp(Z, iters, resid, Ys, bases, owner, max_iter=200):
    """Every graph g of the batch against the FP64 solve of its base graph owner[g]."""
    for bi, (M, lu, vi, valid) in enumerate(bases):
        gs = [g for g in range(len(owner)) if owner[g] == bi]
        nc = Ys.shape[-1]
        Yv = torch.cat([Ys[g][vi].double() for g in gs], 1)          # (nv, len(gs) * nc)
        Z64 = torch.linalg.lu_solve(*lu, Yv)
        for t, g in enumerate(gs):
            z64 = Z64[:, t * nc:(t + 1) * nc]
            z = Z[g][vi].double()
            err = float((z - z64).abs().max() / z64.abs().max())
            agree = float((z.argmax(1) == z64.argmax(1)).float().mean())
            y = Ys[g][vi].double()
            ny = y.norm(dim=0)
            cols = ny > 0
            true_res = float(((y - M @ z).norm(dim=0)[cols] / ny[cols]).max())
            # the library normalises S = D^-1/2 W D^-1/2 in FP32: against the FP64 operator that
            # alone leaves 2e-6 to 3.6e-6 (B200, these graphs; rounding the exact Z to FP32 only
            # 3e-7 to 4e-7); a CG on the wrong operator (a dropped or misplaced row segment)
            # leaves the weight of the lost entries, a few per mille of a row and more
            info = (g, err, agree, true_res, int(iters[g]), float(resid[g]))
            assert err < 1e-4 and agree >= 0.999, info
            assert true_res <= 1e-5, info
            assert float(resid[g]) <= 1.1e-6 and int(iters[g]) < max_iter, info
            assert (Z[g][~valid.bool()] == 0).all(), info


def _labels(G, n, nc, seed):
    """Distinct Y per graph: one-hot rows on 5 % of the nodes, plus junk on every node that a
    solve must ignore where the node is invalid (set by the caller)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    Y = torch.zeros((G, n, nc), device=DEV)
    lab = torch.rand((G, n), generator=g, device=DEV) < 0.05
    cls = torch.randint(0, nc, (G, n), generator=g, device=DEV)
    Y.scatter_(2, cls[..., None], lab[..., None].float())
    Y[:, 0, :] = 0
    Y[:, 0, 0] = 1.0   # no all-zero graph
    return Y


def _lp_run(n, G, nc, k=200, kinds=("random",), n_distinct=3, seed=0):
    from r3dfsseg_b200 import ops
    graphs = [_lp_graph(n, k, seed + 17 * i, kinds[i % len(kinds)], n_invalid=0 if i == 0 else 40 + i)
              for i in range(min(n_distinct, G))]
    owner = [g % len(graphs) for g in range(G)]
    nbr = torch.stack([graphs[o][0] for o in owner])
    sim = torch.stack([graphs[o][1] for o in owner])
    valid = torch.stack([graphs[o][2] for o in owner])
    Y = _labels(G, n, nc, seed + 1)
    Y[valid == 0] = 0.5                         # must be ignored
    Z, iters, resid = ops.label_propagate(nbr, sim, valid, Y)
    bases = [(*_lp_reference(*gr), gr[2]) for gr in graphs]
    Yc = Y.clone()
    Yc[valid == 0] = 0
    _check_lp(Z, iters, resid, Yc, bases, owner)
    return graphs, owner


def _cluster_size(n, G):
    """launch_lp_solve's first cluster size (the one it runs whenever the device grants it)."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    cl_need = -(-n // (CGC_MAXT * CG_MAXPASS))
    return max(16 if G <= 4 else max(1, min(8, n_sm // G)), cl_need)


LP_CASES = [(n, G, nc) for n in (2368, 4416) for G in (1, 4, 5, 19, 25, 37, 150) for nc in (4, 8)] + \
    [(2368, 1, 2), (4416, 25, 2), (2368, 5, 5), (4416, 1, 5), (4416, 25, 5)]


@pytest.mark.parametrize("n,G,nc", LP_CASES)
def test_label_propagate_cluster_sizes_vs_fp64(n, G, nc):
    """lp_cg_kernel<4> / <8> at every cluster size the launcher picks for a batch of G graphs
    (16, 8, 7, 5, 4, 2, 1 on 148 SMs), three distinct graphs tiled with distinct labels."""
    _lp_run(n, G, nc, seed=n + 7 * G + nc)


@pytest.mark.parametrize("n,G,nc", [(6544, 1, 4), (8192, 1, 4), (6544, 60, 4), (8192, 60, 4),
                                    (5376, 1, 8), (5376, 6, 8), (5376, 1, 5)])
def test_label_propagate_largest_graphs_vs_fp64(n, G, nc):
    """The largest graphs of each padded width: 6544 and 8192 nodes at NCV = 4 (cl_need = 3, so
    60 graphs run clusters of 3), 5376 nodes at NCV = 8 (P + the split-row partials fill the
    200 KB of shared memory exactly)."""
    _lp_run(n, G, nc, n_distinct=2, seed=n + G + nc)


def _pack_plan(nbr, valid, CL):
    """cg_pack_kernel's per-CTA decision for one graph at cluster size CL, restated: the merged
    row of node i holds the distinct columns of W = A + A^T; it is cut into ceil(rowmax / 48)
    segments, rowmax = its largest column-residue (mod 8) class; CTAs own contiguous rows with
    about equal segment counts; a CTA with more than 3 passes of 1024 segments, more than
    CG_MAXPART segments of split rows, or packed rows beyond its share of the scratch marks the
    graph unpacked."""
    n, k = nbr.shape
    vb = valid.bool()
    r = torch.arange(n, device=DEV)[:, None].expand(n, k)[vb]
    c = nbr.long()[vb]
    key = torch.unique(torch.cat([r * n + c, c * n + r]))
    rr, cc = key // n, key % n
    rowmax = torch.bincount(rr * 8 + (cc & 7), minlength=8 * n).view(n, 8).max(1).values
    rowmax[~vb] = 0
    nseg = (rowmax + CG_SEGR - 1) // CG_SEGR
    pre = torch.cumsum(nseg, 0) - nseg
    prx = torch.cumsum(torch.where(nseg > 1, nseg, 0), 0) - torch.where(nseg > 1, nseg, 0)
    NV, NX = int(nseg.sum()), int(torch.where(nseg > 1, nseg, 0).sum())
    owner = torch.clamp(pre * CL // NV, max=CL - 1)
    pk_cap = (n * (2 * k) * 2 // 5 + 64 * n + 63) // 64 * 64
    share = pk_cap // CL
    plan = []
    for rank in range(CL):
        rows = torch.nonzero(owner == rank).flatten()
        lo, hi = int(rows.min()), int(rows.max()) + 1
        nv = (int(pre[hi]) if hi < n else NV) - int(pre[lo])
        nx = (int(prx[hi]) if hi < n else NX) - int(prx[lo])
        passes = -(-nv // CGC_MAXT)
        # segments sorted by length (2 * ranks rounds of 4 entries), dealt in slices of 32
        lens = []
        for i in range(lo, hi):
            mx = int(rowmax[i])
            lens += [2 * min(CG_SEGR, mx - s * CG_SEGR) for s in range(int(nseg[i]))]
        lens.sort(reverse=True)
        used = sum(lens[i0] * 32 for i0 in range(0, len(lens), 32))
        bad = passes > CG_MAXPASS or nx > CG_MAXPART or hi - lo > 8191 or used > share
        plan.append(dict(lo=lo, hi=hi, passes=passes, nx=nx, used=used, share=share, bad=bad))
    return plan


def test_label_propagate_ring_graph_takes_the_packed_rows():
    """Low-degree ring graph (k = 16, n = 4416, one graph: clusters of 16).  Each merged row holds
    the 16 ring columns i +- 1..8, 2 per residue class, so no row is split (nx = 0), every CTA
    runs one pass over its 276 rows, and the packed rows use a fraction of the share: the packed
    branch of lp_cg_kernel."""
    n, k, G, nc = 4416, 16, 1, 4
    graphs, _ = _lp_run(n, G, nc, k=k, kinds=("ring",), n_distinct=1, seed=5)
    plan = _pack_plan(graphs[0][0], graphs[0][2], _cluster_size(n, G))
    assert all(not p["bad"] and p["nx"] == 0 and p["passes"] == 1 for p in plan), plan


def test_label_propagate_hub_graph_takes_the_plain_rows():
    """Hub graph: rows 0..149 are in every row's list (k = 200, n = 4416), so each hub's merged
    row holds about 4416 columns, ~552 per residue class: 12 segments of 48 ranks, 1800 split
    segments for the 150 hubs, against ~1 segment for the ~4266 other rows (NV ~ 6000-7000).
    25 graphs get clusters of 5 (148 SMs // 25), so CTA 0 owns the first ~NV / 5 > 1024 segments,
    nearly all of them hub segments: more than CG_MAXPART split segments, and the graph is
    marked unpacked — lp_cg_kernel's warp-per-row branch.  The plan is derived below from the
    graph itself."""
    n, k, G, nc = 4416, 200, 25, 5
    graphs, _ = _lp_run(n, G, nc, k=k, kinds=("hub",), n_distinct=1, seed=9)
    CL = _cluster_size(n, G)
    plan = _pack_plan(graphs[0][0], graphs[0][2], CL)
    assert CL == 5 and plan[0]["nx"] > CG_MAXPART and plan[0]["bad"], (CL, plan)


# ---------------------------------------------------------------------------------------------
# 4- to 7-way episodes
# ---------------------------------------------------------------------------------------------
def _model(fixture_sd, n_way, k_shot, n_pts):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot, pc_npts=n_pts))
    m.load_state_dict(fixture_sd)
    return m.to(DEV).eval()


@pytest.mark.parametrize("n_way,k_shot,n_pts,dataset,noise", [
    (4, 1, 1216, "s3dis", 0.0),      # 512 + 4 x 1216 = 5376 nodes, the NCV = 8 limit
    (5, 2, 896, "s3dis", 0.5),       # one noisy shot per way
    (7, 1, 640, "scannet", 1.0),     # every shot an out-of-distribution one
])
def test_many_way_episode_vs_oracle(fixture_sd, n_way, k_shot, n_pts, dataset, noise):
    """Whole 4- to 7-way episodes (n_cls 5..8: lp_cg_kernel<8>, cg_pack_kernel at 8 floats a
    node) from raw clouds with MDNS, against the oracle's graph half on the CUDA features."""
    m = _model(fixture_sd, n_way, k_shot, n_pts)
    ep = make_episode(300 + n_way, n_way, k_shot, n_pts=n_pts, dataset=dataset, noise_ratio=noise)
    pred, loss = m(ep.support_x.to(DEV), ep.support_y.to(DEV), ep.query_x.to(DEV),
                   ep.query_y.to(DEV), eval=True)
    sf = m.getFeatures(ep.support_x.reshape(n_way * k_shot, 9, -1).to(DEV)).cpu()
    qf = m.getFeatures(ep.query_x.to(DEV)).cpu()
    with torch.no_grad():
        ref = O.forward_episode(fixture_sd, ep.support_x, ep.support_y, ep.query_x, ep.query_y,
                                eval_mdns=True, support_feat=sf, query_feat=qf)
    rp, pred = ref["query_pred"], pred.cpu()
    assert pred.shape == rp.shape == (n_way, n_way + 1, n_pts)
    assert m._last_diag["proto_count"][0].cpu().tolist() == ref["proto_count"]
    assert torch.equal(m._last_diag["clean_flag"][0].cpu(), ref["clean_flag"])
    err = float((pred - rp).abs().max() / rp.abs().max())
    agree = float((pred.argmax(1) == rp.argmax(1)).float().mean())
    assert err < 1e-3 and agree >= 0.999, (err, agree)
    assert abs(float(loss) - float(ref["loss"])) < 1e-4


def _stack(eps):
    sx = torch.stack([e.support_x for e in eps]).to(DEV)
    sy = torch.stack([e.support_y for e in eps]).to(DEV)
    qx = torch.stack([e.query_x for e in eps]).to(DEV)
    qy = torch.stack([e.query_y for e in eps]).to(DEV)
    return sx, sy, qx, qy


def test_four_way_episode_batch_and_segment(fixture_sd):
    """A batch of 6 4-way episodes at 5376 nodes (the batched NCV = 8 solve at clusters of 8)
    is deterministic and equals the single-episode calls (clusters of 16) to the CG tolerance;
    segment() against the encoded support equals forward_episodes bit for bit."""
    m = _model(fixture_sd, 4, 1, 1216)
    eps = [make_episode(400 + s, 4, 1, n_pts=1216, noise_ratio=0.0) for s in range(6)]
    sx, sy, qx, qy = _stack(eps)
    a = m.forward_episodes(sx, sy, qx, qy, eval=True)
    b = m.forward_episodes(sx, sy, qx, qy, eval=True)
    assert torch.equal(a["logits"], b["logits"]) and torch.equal(a["loss"], b["loss"])
    assert _cluster_size(5376, 6) == 8
    for i, e in enumerate(eps):
        pred, loss = m(e.support_x.to(DEV), e.support_y.to(DEV), e.query_x.to(DEV),
                       e.query_y.to(DEV), eval=True)
        got = a["logits"][i].transpose(1, 2)
        err = float((got - pred).abs().max() / pred.abs().max())
        agree = float((got.argmax(1) == pred.argmax(1)).float().mean())
        assert err < 1e-3 and agree >= 0.999 and abs(float(loss) - float(a["loss"][i])) < 1e-4, \
            (i, err, agree)
    sup = m.encode_support(sx[0], sy[0])
    pred, loss = m.segment(sup, qx[0], qy[0])
    one = m.forward_episodes(sx[:1], sy[:1], qx[:1], qy[:1], eval=True)
    assert torch.equal(pred, one["logits"][0].transpose(1, 2)) and torch.equal(loss, one["loss"][0])


# ---------------------------------------------------------------------------------------------
# the node limit of the CG solve
# ---------------------------------------------------------------------------------------------
def test_configurations_past_the_cg_node_limit_are_refused_before_any_launch(fixture_sd):
    """A 4-way episode at 1536 points (512 + 6144 = 6656 nodes > 5376), a 4-way segment() of
    three 2048-point queries (6656 nodes) and label_propagate at n_cls 5 on 5377 nodes raise
    before any kernel is launched; a valid 4-way episode right after still runs."""
    from r3dfsseg_b200 import _lib, ops
    from r3dfsseg_b200.models.mpti import SupportSet
    L = _lib.lib()
    big = _model(fixture_sd, 4, 1, 1536)
    ep = make_episode(500, 4, 1, n_pts=1536)
    wide = _model(fixture_sd, 4, 1, 2048)
    e2 = make_episode(501, 4, 1, n_pts=2048)
    # a 4-way support set of 2048-point shots, encoded under a one-query envelope (2560 nodes)
    pw = wide._weights()
    proto, count, clean = ops.op.mpti_support(pw.tensors, wide.in_channels, int(wide.encoder.k),
                                              e2.support_x[None].to(DEV), e2.support_y[None].to(DEV),
                                              1, wide.n_subprototypes, wide.k_connect, True)
    sup = SupportSet(proto, count, clean, 4, 1, 2048, wide.n_subprototypes, True, wide._packed_sig)
    nbr, sim, valid = _lp_graph(5377, 16, 3, "ring")
    torch.cuda.synchronize()
    n0 = L.r3dfs_launch_count()
    with pytest.raises(_lib.R3dfsError, match="outside what libr3dfs is built for"):
        big(ep.support_x.to(DEV), ep.support_y.to(DEV), ep.query_x.to(DEV), ep.query_y.to(DEV),
            eval=True)
    with pytest.raises(_lib.R3dfsError, match="outside what libr3dfs is built for"):
        wide.segment(sup, e2.query_x[:3][None].to(DEV))
    with pytest.raises(_lib.R3dfsError, match="not supported"):
        ops.label_propagate(nbr[None], sim[None], valid[None], torch.ones((1, 5377, 5), device=DEV))
    torch.cuda.synchronize()
    assert L.r3dfs_launch_count() == n0
    ok = _model(fixture_sd, 4, 1, 1216)
    e3 = make_episode(502, 4, 1, n_pts=1216)
    pred, loss = ok(e3.support_x.to(DEV), e3.support_y.to(DEV), e3.query_x.to(DEV),
                    e3.query_y.to(DEV), eval=True)
    torch.cuda.synchronize()
    assert torch.isfinite(pred).all() and math.isfinite(float(loss))
    assert int(ok._last_diag["cg_iters"][0]) < 200
