"""GPU parity of the meta-training step (SURVEY.md §8 A16/A17, config 5): the CUDA forward and
backward behind r3dfs_mpti_train_forward / _backward against the CPU oracle's autograd
(oracle/mpti_train_oracle.py, pinned to the reference by tests/golden/golden_train.pt).

The discrete decisions of an episode (EdgeConv neighbour lists, FPS/argmin cluster assignments,
affinity-graph neighbours) carry no gradient but FP32 ties in them make an end-to-end comparison
chaotic, so the strict test is TEACHER-FORCED: the oracle is run with the decisions the CUDA path
took (r3dfs_mpti_train_export) and losses / logits / every gradient tensor / BatchNorm running
statistics must then agree to FP32 rounding accumulated over the graph.  A second, free-running
test compares with the reference's own golden numbers at a statistical tolerance."""
import os

import pytest
import torch

from oracle import mpti_train_oracle as TO
from r3dfsseg_b200.episodes import default_args, make_episode

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# conv biases ahead of a batch-statistics BatchNorm have an exactly-zero gradient; both sides only
# produce rounding noise there
ZERO_GRAD = {"base_learner.convs.0.0.bias", "base_learner.convs.1.0.bias"}


def _model(sd, n_way=2, k_shot=5):
    from r3dfsseg_b200.models import MPTI_SelfAtten
    m = MPTI_SelfAtten(default_args(n_way, k_shot))
    m.load_state_dict(sd)
    return m.to(DEV).train()


def _run_cuda(m, ep, p_drop=0.0, ks=None, kq=None):
    from r3dfsseg_b200 import train as T
    qp, lp, ct = T.train_episode(m, ep.support_x.to(DEV), ep.support_y.to(DEV), ep.query_x.to(DEV),
                                 ep.query_y.to(DEV), ep.support_flag.to(DEV), dropout_p=p_drop,
                                 keep_support=ks, keep_query=kq)
    (lp + 0.1 * ct).backward()
    torch.cuda.synchronize()
    return qp.detach().cpu(), float(lp.detach()), float(ct.detach())


@pytest.mark.parametrize("seed,n_way,noise,p_drop", [(11, 2, 0.0, 0.0), (12, 2, 0.4, 0.1),
                                                     (13, 3, 0.4, 0.0)])
def test_train_step_teacher_forced(fixture_sd, seed, n_way, noise, p_drop):
    from r3dfsseg_b200 import train as T
    torch.set_num_threads(os.cpu_count())
    ds = "scannet" if n_way == 3 else "s3dis"
    ep = make_episode(seed, n_way, 5, dataset=ds, noise_ratio=noise)
    m = _model(fixture_sd, n_way, 5)
    ks = kq = None
    if p_drop > 0:
        ks = T.dropout_mask(1234, (n_way * 5, 2048, 2048), p_drop, DEV)
        kq = T.dropout_mask(99, (n_way, 2048, 2048), p_drop, DEV)
        assert abs(float(ks.float().mean()) - (1 - p_drop)) < 1e-3
    qp, lp, ct = _run_cuda(m, ep, p_drop, ks, kq)
    ratio_lp, ratio_orig = (float(x) for x in T.clean_ratios(m, ep.support_y, ep.gt_support_y))
    forced = T.export_decisions(m)
    P, running = TO.split_state_dict(fixture_sd)
    out = TO.forward_train(P, ep.support_x, ep.support_y, ep.query_x, ep.query_y, ep.support_flag,
                           running=running, keep_mask_support=None if ks is None else ks.cpu(),
                           keep_mask_query=None if kq is None else kq.cpu(), dropout_p=p_drop,
                           forced=forced, keep=True)
    (out["lp_loss"] + 0.1 * out["contrast_loss"]).backward()
    # the reference's logging diagnostics (models/mpti.py:514-552) from the oracle's Z and the
    # exported assignments: exact up to argmax ties on the prototype rows
    Zp, pc, acc_lp, acc_or = out["Z"].detach(), forced["proto_cnt"], [], []
    for w in range(n_way):
        rows = Zp[sum(pc[:1 + w]):sum(pc[:2 + w])]
        proto_pred = (rows.argmax(1) == w + 1).long()
        point_pred = proto_pred[forced["assign"][1 + w]]
        fg = ep.support_y[w].reshape(-1) == 1
        gt = ep.gt_support_y[w].reshape(-1)[fg].long()
        acc_lp.append(float((point_pred == gt).float().mean()))
        acc_or.append(float((gt == 1).float().mean()))
    assert abs(ratio_lp - sum(acc_lp) / n_way) < 2e-3, (ratio_lp, acc_lp)
    assert abs(ratio_orig - sum(acc_or) / n_way) < 1e-6, (ratio_orig, acc_or)
    assert abs(lp - float(out["lp_loss"])) <= 1e-4 * abs(float(out["lp_loss"]))
    assert abs(ct - float(out["contrast_loss"])) <= 1e-4 * abs(float(out["contrast_loss"]))
    ref_q = out["query_pred"].detach()
    assert float((qp - ref_q).abs().max() / ref_q.abs().max()) < 1e-3          # north_star tolerance
    assert float((qp.argmax(1) == ref_q.argmax(1)).float().mean()) >= 0.999
    named = dict(m.named_parameters())
    for k in T.PARAM_NAMES:
        g, r = named[k].grad.detach().cpu(), P[k].grad
        if k in ZERO_GRAD:
            assert float(g.abs().max()) < 1e-6
            continue
        err = float((g - r).abs().max()) / float(r.abs().max())
        assert err < 1e-2, (k, err)
        assert abs(float(g.norm()) - float(r.norm())) < 2e-3 * float(r.norm()), k
    for k, v in m.named_buffers():
        if v.dtype.is_floating_point:
            assert float((v.cpu() - running[k]).abs().max()) < 1e-4, k
        else:
            assert int(v) == int(running[k]), k


def test_forward_train_tuple_matches_reference_diagnostics(fixture_sd):
    """The drop-in 7-tuple of forward(train=True) (models/mpti.py:575): the four logging diagnostics
    against the numbers the reference itself printed for the same episode (golden_train.pt)."""
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "golden_train.pt"))
    g = gold["train_s3dis_2way_5shot_noisy"]
    ep = make_episode(g["seed"], g["n_way"], g["k_shot"], dataset=g["dataset"], noise_ratio=g["noise_ratio"])
    m = _model(fixture_sd)
    m.att_learner.dropout.p = 0.0
    out = m(ep.support_x.to(DEV), ep.support_y.to(DEV), ep.query_x.to(DEV), ep.query_y.to(DEV),
            gt_support_y=ep.gt_support_y.to(DEV), gt_query_y=ep.query_y.to(DEV), train=True,
            support_flag=ep.support_flag.to(DEV))
    assert len(out) == 7
    got = [float(x) for x in out[3:7]]
    assert not any(v != v for v in got)                       # no NaN placeholder any more
    for a, b in zip(got, g["diagnostics"]):
        assert abs(a - b) < 5e-3, (got, g["diagnostics"])     # free-running: ties may move a prototype


def test_train_step_free_running_vs_reference_golden(fixture_sd):
    """No teacher forcing: the reference's own numbers (oracle/make_golden_train.py).  Ties broken
    differently move kNN lists / FPS seeds, so this is a statistical bound, not an FP32 one."""
    from r3dfsseg_b200 import train as T
    gold = torch.load(os.path.join(os.path.dirname(__file__), "golden", "golden_train.pt"))
    for name, g in gold.items():
        ep = make_episode(g["seed"], g["n_way"], g["k_shot"], dataset=g["dataset"],
                          noise_ratio=g["noise_ratio"])
        m = _model(fixture_sd, g["n_way"], g["k_shot"])
        _, lp, ct = _run_cuda(m, ep)
        assert abs(lp - float(g["lp_loss"])) < 1e-2 * float(g["lp_loss"]), name
        assert abs(ct - float(g["contrast_loss"])) < 1e-2 * float(g["contrast_loss"]), name
        named = dict(m.named_parameters())
        tot = torch.sqrt(sum(named[k].grad.pow(2).sum() for k in T.PARAM_NAMES)).item()
        ref = torch.sqrt(sum(v.pow(2) for v in g["grad_norm"].values())).item()
        assert abs(tot - ref) < 0.05 * ref, (name, tot, ref)


@pytest.mark.parametrize("M,N,K,ta,tb", [(300, 70, 129, False, False), (64, 64, 50000, True, False),
                                         (2048, 2048, 64, False, True), (192, 256, 24576, True, False),
                                         (1000, 192, 512, False, False), (5, 3, 7, True, True)])
def test_sgemm_strided(M, N, K, ta, tb):
    """The gradient GEMM (generic element strides, split-K with a fixed-order reduce) vs float64."""
    import ctypes as C
    from r3dfsseg_b200 import _lib, ops
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn((K, M) if ta else (M, K), generator=g)
    B = torch.randn((N, K) if tb else (K, N), generator=g)
    C0 = torch.randn((M, N + 3), generator=g)
    Ad, Bd, Cd = A.to(DEV), B.to(DEV), C0.to(DEV)
    ws = torch.empty(32 << 20, dtype=torch.uint8, device=DEV)
    sAm, sAk = (1, M) if ta else (K, 1)
    sBk, sBn = (1, K) if tb else (N, 1)
    _lib.check(_lib.lib().r3dfs_sgemm(ops._p(Ad), sAm, sAk, ops._p(Bd), sBk, sBn, ops._p(Cd), N + 3, M,
                                      N, K, 0.5, 2.0, ops._p(ws), ws.numel(), ops._stream()), "sgemm")
    ref = 0.5 * ((A.t() if ta else A).double() @ (B.t() if tb else B).double()) + 2.0 * C0[:, :N].double()
    got = Cd.cpu()
    assert torch.equal(got[:, N:], C0[:, N:])  # padding columns untouched
    err = float((got[:, :N].double() - ref).abs().max() / ref.abs().max())
    assert err < 2e-6 * max(1.0, (K / 512) ** 0.5), err


def test_fused_adam_matches_torch(fixture_sd):
    """r3dfs_adam_step vs torch.optim.Adam with the reference's two learning-rate groups."""
    from r3dfsseg_b200 import train as T
    m = _model(fixture_sd)
    opt = T.FusedAdam(m, lr=1e-3)
    fs = T.flat_state(m)
    ref_p = [p.detach().cpu().clone().requires_grad_(True) for p in fs.params]
    enc = [p for n, p in zip(T.PARAM_NAMES, ref_p) if n.startswith("encoder.")]
    rest = [p for n, p in zip(T.PARAM_NAMES, ref_p) if not n.startswith("encoder.")]
    ropt = torch.optim.Adam([{"params": enc, "lr": 1e-4}, {"params": rest}], lr=1e-3)
    g = torch.Generator().manual_seed(3)
    for step in range(3):
        for p, rp in zip(fs.params, ref_p):
            gr = torch.randn(rp.shape, generator=g) * 0.01
            rp.grad = gr.clone()
            p.grad = gr.to(DEV)
        opt.step()
        ropt.step()
    for n, p, rp in zip(T.PARAM_NAMES, fs.params, ref_p):
        assert float((p.detach().cpu() - rp.detach()).abs().max()) < 2e-6, n


def test_learner_train_then_test(fixture_sd):
    """MPTILearner_V3 contract (reference models/mpti_learner.py:50-102): two optimisation steps
    move the parameters, the losses stay finite, and the eval path picks the new weights up."""
    from r3dfsseg_b200 import train as T
    from r3dfsseg_b200.models import MPTI_SelfAtten
    args = default_args(2, 5)
    model = MPTI_SelfAtten(args)
    model.load_state_dict(fixture_sd)
    learner = T.MPTILearner_V3(args, mode="train", model=model)
    before = T.flat_state(learner.model).flat.clone()
    nbt0 = int(fixture_sd["encoder.conv.layer.1.num_batches_tracked"])
    losses = []
    for seed in (21, 22):
        ep = make_episode(seed, 2, 5, noise_ratio=0.2)
        c = lambda t: t.to(DEV)
        zq = torch.zeros_like(ep.query_y)
        data = [c(ep.support_x), c(ep.support_y), c(ep.query_x), c(ep.query_y),
                c(torch.zeros_like(ep.support_y)), c(zq), c(ep.gt_support_y), c(ep.query_y), None,
                None, c(ep.support_flag)]
        out = learner.train(data, logger=None)
        assert len(out) == 8
        losses.append(float(out[0]))
        assert 0.0 <= out[3] <= 1.0
    assert all(map(lambda v: v == v and abs(v) < 1e3, losses))
    after = T.flat_state(learner.model).flat
    delta = (after - before).abs()
    assert float(delta.max()) > 1e-5 and float(delta.max()) < 1e-2   # |update| ~ lr per step
    for bn in T.flat_state(learner.model).bn:
        assert int(bn.num_batches_tracked) == nbt0 + 4   # two getFeatures calls per step
    ep = make_episode(30, 2, 5)
    pred, loss, acc = learner.test([t.to(DEV) if torch.is_tensor(t) else t
                                    for t in ep.as_test_data()], ep.sampled_classes, eval=True)
    assert pred.shape == (2, 2048) and float(loss) == float(loss) and 0.0 <= acc <= 1.0
    # the reference's state-dict keys survive the flat re-homing
    sd2 = learner.model.state_dict()
    assert set(sd2.keys()) == set(fixture_sd.keys())


def test_learner_resumes_from_reference_format_checkpoint(fixture_sd, tmp_path):
    """checkpoint.tar in the reference's layout (utils/checkpoint_util.py:26-45,
    mpti_train_noise.py:137-144): one step, save, resume in a new learner through
    `args.model_checkpoint_path` — weights, Adam moments, step count and learning rates come back
    bit for bit, torch.optim.Adam over the reference's four groups accepts the optimizer state, and
    the next step of the resumed learner equals the next step of the original."""
    from r3dfsseg_b200 import checkpoint as ck
    from r3dfsseg_b200 import train as T
    from r3dfsseg_b200.models import MPTI_SelfAtten

    def data_of(seed):
        ep = make_episode(seed, 2, 5, noise_ratio=0.2)
        c = lambda t: t.to(DEV)
        zq = torch.zeros_like(ep.query_y)
        return [c(ep.support_x), c(ep.support_y), c(ep.query_x), c(ep.query_y),
                c(torch.zeros_like(ep.support_y)), c(zq), c(ep.gt_support_y), c(ep.query_y), None,
                None, c(ep.support_flag)]

    args = default_args(2, 5)
    model = MPTI_SelfAtten(args)
    model.load_state_dict(fixture_sd)
    a = T.MPTILearner_V3(args, mode="train", model=model)
    a.train(data_of(41))
    ck.save_model_checkpoint(a.model, a.optimizer, str(tmp_path), iteration=1, iou=0.25)
    saved = torch.load(str(tmp_path / "checkpoint.tar"))
    assert set(saved) >= {"iteration", "IoU", "model_state_dict", "optimizer_state_dict"}
    ref_model = MPTI_SelfAtten(args)
    ref_opt = torch.optim.Adam([{"params": ref_model.encoder.parameters(), "lr": 1e-4},
                                {"params": ref_model.base_learner.parameters()},
                                {"params": ref_model.att_learner.parameters()},
                                {"params": ref_model.proj.parameters()}], lr=args.lr)
    ref_opt.load_state_dict(saved["optimizer_state_dict"])          # the reference side can resume
    args_b = default_args(2, 5, model_checkpoint_path=str(tmp_path))
    b = T.MPTILearner_V3(args_b, mode="train")
    assert torch.equal(T.flat_state(b.model).flat, T.flat_state(a.model).flat)
    assert torch.equal(T.flat_state(b.model).running, T.flat_state(a.model).running)
    assert torch.equal(b.optimizer.exp_avg, a.optimizer.exp_avg)
    assert torch.equal(b.optimizer.exp_avg_sq, a.optimizer.exp_avg_sq)
    assert b.optimizer.step_count == a.optimizer.step_count == 1
    b.model._train_step = a.model._train_step                      # same dropout counter
    la = a.train(data_of(42))
    lb = b.train(data_of(42))
    assert abs(float(la[0].detach()) - float(lb[0].detach())) <= 1e-4 * abs(float(la[0].detach()))
    # float atomics in the backward: the two runs are not bit-identical.  Parameters whose true
    # gradient is exactly zero (the conv biases ahead of a batch-statistics BatchNorm, 192 of 376 896)
    # receive pure rounding noise, which Adam normalises to steps of +-lr; everything else agrees
    # far below one update
    d = (T.flat_state(a.model).flat - T.flat_state(b.model).flat).abs()
    assert float((d < 1e-6).float().mean()) > 0.995, (float(d.max()), float((d < 1e-6).float().mean()))


def test_backward_after_a_second_forward_fails_loudly(fixture_sd):
    """All saved activations of a training forward live in ONE shared workspace; forward(A),
    forward(B), backward(A) would silently use B's activations — it must raise instead, while the
    usual forward -> backward per episode (and backward of the LATEST forward) keeps working."""
    from r3dfsseg_b200 import train as T
    m = _model(fixture_sd)
    eps = [make_episode(s, 2, 5, noise_ratio=0.2) for s in (31, 32)]
    outs = []
    for ep in eps:
        _, lp, ct = T.train_episode(m, ep.support_x.to(DEV), ep.support_y.to(DEV), ep.query_x.to(DEV),
                                    ep.query_y.to(DEV), ep.support_flag.to(DEV), dropout_p=0.0)
        outs.append(lp + 0.1 * ct)
    with pytest.raises(RuntimeError, match="overwritten"):
        outs[0].backward()
    outs[1].backward()                      # the latest forward is intact
    assert all(p.grad is not None for p in m.parameters())


def test_fused_adam_without_gradients_is_a_no_op(fixture_sd):
    """torch.optim.Adam skips parameters whose .grad is None; the fused step must not decay moments
    or move parameters with an all-zero stand-in gradient."""
    from r3dfsseg_b200 import train as T
    m = _model(fixture_sd)
    opt = T.FusedAdam(m, lr=1e-3)
    before = T.flat_state(m).flat.clone()
    opt.zero_grad(set_to_none=True)
    opt.step()
    assert opt.step_count == 0 and torch.equal(T.flat_state(m).flat, before)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_replicas_stay_identical_nccl_world2(tmp_path):
    """Two NCCL ranks built from DIFFERENT initial weights: after FusedAdam's broadcast and three
    training steps on different episodes, parameters and BatchNorm running statistics are equal
    bit for bit on both ranks (gradient all-reduce + running-statistics average)."""
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.dirname(__file__)), "scripts", "check_replicas.py")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
                        "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port",
                        str(29400 + os.getpid() % 500), script], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "REPLICAS_EQUAL" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
