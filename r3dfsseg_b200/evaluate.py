"""Sharded, batched evaluation driver: the reference's `test_few_shot` + `evaluate_metric`
(reference eval_noise.py:23-113) for many episodes per call and many GPUs.

Episodes are independent (eval_noise.py:85-106), so episode i belongs to rank i % world; every rank
runs its shard through `MPTI_SelfAtten.forward_episodes` in batches, accumulates the three
evaluate_metric counter rows (ground truth / predicted / true positive per test-class slot,
eval_noise.py:35-37) on the device, and ONE sum all-reduce of (3 x n_slots) int64 + the loss sum
ends the run.  Nothing else crosses GPUs.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np
import torch


def shard_indices(n_items: int, rank: int, world: int) -> List[int]:
    """Static round-robin sharding of independent episodes."""
    if not (0 <= rank < world):
        raise ValueError("rank must be in [0, world)")
    return list(range(rank, n_items, world))


def class_slots(sampled_classes: Sequence[int], test_classes: Sequence[int]) -> List[int]:
    """Episode-local label l (1-based) -> slot test_classes.index(sampled_classes[l-1]) + 1
    (reference eval_noise.py:48-59); slot 0 is the background."""
    tc = list(test_classes)
    return [tc.index(int(c)) + 1 for c in sampled_classes]


def iou_from_counters(counters) -> Dict[str, object]:
    """IoU_c = TP / (GT + Pred - TP); mean over the foreground slots (eval_noise.py:64-70)."""
    c = counters.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(counters) \
        else np.asarray(counters, dtype=np.float64)
    gt, pos, tp = c
    with np.errstate(divide="ignore", invalid="ignore"):
        iou = tp / (gt + pos - tp)
    return {"iou": iou, "mean_iou": float(np.mean(iou[1:]))}


def all_reduce_eval_state(counters: torch.Tensor, loss_sum: torch.Tensor, n_episodes: torch.Tensor):
    """Sum the per-rank partial results in place.  No-op without an initialised process group
    (single GPU).  Works with any backend (nccl on GPUs, gloo in the CPU tests)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
        dist.all_reduce(loss_sum, op=dist.ReduceOp.SUM)
        dist.all_reduce(n_episodes, op=dist.ReduceOp.SUM)
    return counters, loss_sum, n_episodes


class _Slot:
    """One in-flight batch: pinned host staging buffers (filled by the reader threads), their device
    twins, a workspace, a stream and partial results.  Hand-over: the producer fills the host side
    and queues the slot; the consumer enqueues the H2D copies + the forward on the slot's stream,
    records `copied` and sets `issued`; the producer waits for both before it refills the slot."""

    def __init__(self, model, batch, n_query, device):
        import threading
        nw, ks, N, C = model.n_way, model.k_shot, model.n_points, model.in_channels
        pin = dict(pin_memory=True)
        self.h_sx = torch.empty((batch, nw, ks, N, C), dtype=torch.float32, **pin)
        self.h_sy = torch.empty((batch, nw, ks, N), dtype=torch.int32, **pin)
        self.h_qx = torch.empty((batch, n_query, N, C), dtype=torch.float32, **pin)
        self.h_qy = torch.empty((batch, n_query, N), dtype=torch.int64, **pin)
        self.h_slot = torch.empty((batch, nw), dtype=torch.int32, **pin)
        # numpy views of the same pinned memory, keyed by the episode-file dataset names
        self.np = {"support_ptclouds": self.h_sx.numpy(), "support_masks": self.h_sy.numpy(),
                   "query_ptclouds": self.h_qx.numpy(), "query_labels": self.h_qy.numpy()}
        self.np_slot = self.h_slot.numpy()
        self.d = [torch.empty_like(t, device=device) for t in
                  (self.h_sx, self.h_sy, self.h_qx, self.h_qy, self.h_slot)]
        self.stream = torch.cuda.Stream(device=device)
        self.copied = torch.cuda.Event()
        self.issued = threading.Event()
        self.issued.set()
        self.ws = None
        self.counters = None   # per-slot partial results: slots run on different streams
        self.loss_sum = None


class EpisodeEvaluator:
    """Runs episodes through the model, `batch` per C-ABI call.

    model         r3dfsseg_b200.models.MPTI_SelfAtten on a CUDA device, eval mode
    test_classes  the fold's test class ids (defines the counter slots)
    batch         episodes per C-ABI call
    n_inflight    batches in flight: each has its own persistent pinned staging buffers, device
                  buffers, workspace and stream; reader threads fill the next batches' buffers
                  (straight from the episode files when the source can `read_into`) while the GPU
                  runs the previous ones
    """

    def __init__(self, model, test_classes: Sequence[int], batch: int = 16, eval_mdns: bool = True,
                 n_inflight: int = 3, n_readers: int = 6):
        self.model = model
        self.test_classes = list(test_classes)
        self.batch = int(batch)
        self.eval_mdns = eval_mdns
        self.device = next(model.parameters()).device
        self.n_inflight = max(2, int(n_inflight))
        self.n_readers = max(1, int(n_readers))
        self._slots = None
        self._slots_key = None

    # ---- staging --------------------------------------------------------------------------------
    def _get_slots(self, n_query):
        key = (self.batch, n_query, self.n_inflight)
        if self._slots is None or self._slots_key != key:
            self._slots = [_Slot(self.model, self.batch, n_query, self.device)
                           for _ in range(self.n_inflight)]
            self._slots_key = key
        return self._slots

    def _fill(self, slot: "_Slot", i: int, data, classes):
        """One episode (the reference's collate output, loader.py:1676-1684: (.., 9, N) views over
        point-major memory) into row i of the pinned staging buffers: plain memcpys."""
        nw, ks = self.model.n_way, self.model.k_shot
        sx = data[0].reshape(nw, ks, data[0].shape[-2], data[0].shape[-1])
        slot.h_sx[i].copy_(sx.transpose(2, 3))
        slot.h_sy[i].copy_(data[1].reshape(nw, ks, -1))
        slot.h_qx[i].copy_(data[2].transpose(1, 2))
        slot.h_qy[i].copy_(data[3])
        slot.np_slot[i] = class_slots(np.asarray(classes).reshape(-1), self.test_classes)

    def _read_into(self, source, slot: "_Slot", i: int, index: int):
        classes = source.read_into(index, {k: v[i] for k, v in slot.np.items()})
        slot.np_slot[i] = class_slots(classes, self.test_classes)

    def _produce(self, source, rank, world, n_query_hint, q):
        """Producer thread: this rank's shard, `batch` episodes at a time, into the slots in turn."""
        from concurrent.futures import ThreadPoolExecutor
        try:
            torch.cuda.set_device(self.device)  # this thread allocates pinned memory and streams
            slots, bi = None, 0

            def next_slot(n_query):
                nonlocal slots, bi
                if slots is None:
                    slots = self._get_slots(n_query)
                sl = slots[bi % len(slots)]
                bi += 1
                sl.issued.wait()            # the consumer has enqueued this slot's previous batch
                sl.copied.synchronize()     # ... and its H2D copies have left the host buffers
                sl.issued.clear()
                return sl

            if hasattr(source, "read_into") and hasattr(source, "__len__"):
                mine = shard_indices(len(source), rank, world)
                with ThreadPoolExecutor(self.n_readers) as pool:
                    for s in range(0, len(mine), self.batch):
                        idx = mine[s:s + self.batch]
                        sl = next_slot(n_query_hint(source, idx[0]))
                        list(pool.map(lambda t: self._read_into(source, sl, t[0], t[1]),
                                      enumerate(idx)))
                        q.put((sl, len(idx)))
            else:
                if hasattr(source, "item") and hasattr(source, "__len__"):
                    it = (source.item(i) for i in shard_indices(len(source), rank, world))
                else:
                    it = (item for i, item in enumerate(source) if i % world == rank)
                sl, n = None, 0
                for data, classes in it:
                    if sl is None:
                        sl, n = next_slot(int(data[2].shape[0])), 0
                    self._fill(sl, n, data, classes)
                    n += 1
                    if n == self.batch:
                        q.put((sl, n))
                        sl = None
                if sl is not None:
                    q.put((sl, n))
            q.put(None)
        except BaseException as e:  # surface reader errors in the consumer
            q.put(e)

    # ---- the loop ---------------------------------------------------------------------------------
    def run(self, episodes, rank: int = 0, world: int = 1, logger=None,
            log_every: int = 50) -> Dict[str, object]:
        """episodes: a sequence of Episode-like objects, an EpisodeFolder, or any iterable of
        (data, sampled_classes) as the reference's test loader yields them — consumed as a stream.
        logger: optional object with `.cprint(str)` (the reference's utils.logger); it gets the
        reference's progress line every `log_every` episodes (eval_noise.py:94-95) and the
        per-class IoU printout at the end (:64-68)."""
        import queue
        import threading
        from . import _lib, ops
        if isinstance(episodes, (list, tuple)) and episodes and hasattr(episodes[0], "support_x"):
            episodes = _EpisodeList(episodes)
        n_slots = len(self.test_classes) + 1
        dev = self.device
        counters = torch.zeros((3, n_slots), dtype=torch.int64, device=dev)
        loss_sum = torch.zeros((), dtype=torch.float64, device=dev)
        cg_bad = torch.zeros((), dtype=torch.float64, device=dev)
        cur = torch.cuda.current_stream(dev)
        q: "queue.Queue" = queue.Queue()

        def n_query_hint(source, index):
            return int(source[index][2].shape[0])  # query_ptclouds of the first episode

        with torch.cuda.device(dev):
            threading.Thread(target=self._produce, args=(episodes, rank, world, n_query_hint, q),
                             daemon=True).start()
        prepared, last_loss, done = set(), None, 0
        while True:
            got = q.get()
            if got is None:
                break
            if isinstance(got, BaseException):
                raise got
            sl, n = got
            if id(sl) not in prepared:   # first use in this run: workspace, zeroed partial results
                cfg = self.model._cfg(int(sl.h_qx.shape[1]), mdns=bool(self.eval_mdns))
                need = _lib.lib().r3dfs_mpti_workspace(cfg, self.batch)
                if sl.ws is None or sl.ws.numel() < need:
                    sl.ws = torch.empty(need, dtype=torch.uint8, device=dev)
                sl.counters = torch.zeros_like(counters)
                sl.loss_sum = torch.zeros_like(loss_sum)
                sl.cg_bad = None
                sl.stream.wait_stream(cur)
                prepared.add(id(sl))
            with torch.cuda.stream(sl.stream):
                for h, d in zip((sl.h_sx, sl.h_sy, sl.h_qx, sl.h_qy, sl.h_slot), sl.d):
                    d[:n].copy_(h[:n], non_blocking=True)
                sl.copied.record(sl.stream)
                sl.issued.set()
                sx, sy, qx, qy, slot = (d[:n] for d in sl.d)
                out = self.model.forward_episodes(sx.transpose(3, 4), sy, qx.transpose(2, 3), qy,
                                                  eval=self.eval_mdns, workspace=sl.ws,
                                                  want_diag=True)
                ops.confusion_accumulate(out["pred"], qy, slot, sl.counters)
                sl.loss_sum += out["loss"].double().sum()
                # label-propagation solves that hit cg_max_iter without reaching cg_tol (no sync:
                # counted on the device, reported with the result)
                nc_bad = (out["diag"]["cg_iters"] >= int(self.model.cg_max_iter)).sum().double()
                sl.cg_bad = nc_bad if getattr(sl, "cg_bad", None) is None else sl.cg_bad + nc_bad
                last_loss = out["loss"]
                for t in (out["pred"], out["loss"], out["logits"]):
                    t.record_stream(sl.stream)
            if logger is not None and (done + n) // log_every > done // log_every:
                from datetime import datetime
                logger.cprint("[Eval] Iter: %d | Loss: %.4f | %s" % (
                    done + n, float(last_loss[-1]), str(datetime.now())))
            done += n
        for sl in (self._slots or []):
            if id(sl) in prepared:
                cur.wait_stream(sl.stream)
                counters += sl.counters
                loss_sum += sl.loss_sum
                if getattr(sl, "cg_bad", None) is not None:
                    cg_bad += sl.cg_bad
        n = torch.tensor(float(done), dtype=torch.float64, device=dev)
        all_reduce_eval_state(counters, loss_sum, n)
        res = iou_from_counters(counters)
        res.update(counters=counters.cpu(), mean_loss=float(loss_sum / n), n_episodes=int(n),
                   cg_not_converged=int(cg_bad))
        if res["cg_not_converged"]:
            import warnings
            warnings.warn("%d label-propagation solve(s) on this rank stopped at cg_max_iter=%d "
                          "before reaching cg_tol=%g" % (res["cg_not_converged"],
                                                         self.model.cg_max_iter, self.model.cg_tol))
        if logger is not None and rank == 0:
            for c in range(n_slots):
                logger.cprint("class %d: iou %f" % (c, res["iou"][c]))
            logger.cprint("mean IoU: %f\n" % res["mean_iou"])
        return res

    def run_scenes(self, ds, way_classes, k_shot: int, n_queries: int = 1,
                   noise_type: Optional[str] = None, noise_ratio=0.0, rank: int = 0,
                   world: int = 1, pair_dict=None, first: int = 0, logger=None,
                   log_every: int = 50) -> Dict[str, object]:
        """`run` over episodes sampled on the device from a `SceneEpisodes` dataset: episode i has
        way classes way_classes[i] (e.g. ds.test_classes(n_way)) and index first + i, and belongs
        to rank i % world.  Each batch of this rank's episodes is sampled, run through
        forward_episodes and counted without leaving the device; the run ends with the same
        all-reduce as `run` and returns the same dict."""
        from . import _lib, ops
        wc = np.asarray(way_classes, dtype=np.int64)
        if wc.ndim == 1:
            wc = wc[None]
        mine = shard_indices(len(wc), rank, world)
        n_slots = len(self.test_classes) + 1
        dev = self.device
        counters = torch.zeros((3, n_slots), dtype=torch.int64, device=dev)
        loss_sum = torch.zeros((), dtype=torch.float64, device=dev)
        cg_bad = torch.zeros((), dtype=torch.float64, device=dev)
        slots = torch.tensor([class_slots(wc[i], self.test_classes) for i in mine],
                             dtype=torch.int32).reshape(len(mine), wc.shape[1]).to(dev)
        ws, done = None, 0
        for s in range(0, len(mine), self.batch):
            idx = mine[s:s + self.batch]
            b = ds.sample(wc[idx], k_shot, n_queries, first=first + idx[0], noise_type=noise_type,
                          noise_ratio=noise_ratio, pair_dict=pair_dict, step=world)
            if ws is None:
                cfg = self.model._cfg(int(b["query_x"].shape[1]), mdns=bool(self.eval_mdns))
                ws = torch.empty(_lib.lib().r3dfs_mpti_workspace(cfg, self.batch),
                                 dtype=torch.uint8, device=dev)
            out = self.model.forward_episodes(b["support_x"], b["support_y"], b["query_x"],
                                              b["query_y"], eval=self.eval_mdns, workspace=ws,
                                              want_diag=True)
            ops.confusion_accumulate(out["pred"], b["query_y"], slots[s:s + len(idx)], counters)
            loss_sum += out["loss"].double().sum()
            cg_bad += (out["diag"]["cg_iters"] >= int(self.model.cg_max_iter)).sum().double()
            if logger is not None and (done + len(idx)) // log_every > done // log_every:
                from datetime import datetime
                logger.cprint("[Eval] Iter: %d | Loss: %.4f | %s" % (
                    done + len(idx), float(out["loss"][-1]), str(datetime.now())))
            done += len(idx)
        n = torch.tensor(float(done), dtype=torch.float64, device=dev)
        all_reduce_eval_state(counters, loss_sum, n)
        res = iou_from_counters(counters)
        res.update(counters=counters.cpu(), mean_loss=float(loss_sum / n), n_episodes=int(n),
                   cg_not_converged=int(cg_bad))
        if res["cg_not_converged"]:
            import warnings
            warnings.warn("%d label-propagation solve(s) on this rank stopped at cg_max_iter=%d "
                          "before reaching cg_tol=%g" % (res["cg_not_converged"],
                                                         self.model.cg_max_iter, self.model.cg_tol))
        if logger is not None and rank == 0:
            for c in range(n_slots):
                logger.cprint("class %d: iou %f" % (c, res["iou"][c]))
            logger.cprint("mean IoU: %f\n" % res["mean_iou"])
        return res


class _EpisodeList:
    """Adapter: Episode-like objects (support_x, support_y, query_x, query_y, sampled_classes) as an
    indexable source of (data, sampled_classes)."""

    def __init__(self, eps):
        self.eps = eps

    def __len__(self):
        return len(self.eps)

    def item(self, i):
        e = self.eps[i]
        return [e.support_x, e.support_y, e.query_x, e.query_y], e.sampled_classes


def test_few_shot(test_loader, learner, logger, test_classes, path=None, eval=False, batch: int = 16,
                  n_inflight: int = 3):
    """Drop-in for reference eval_noise.py:75-113: same arguments, returns (mean_loss, mean_IoU).
    `test_loader` yields (data, sampled_classes) per episode exactly as the reference's DataLoader
    (batch_size 1, `batch_test_task_collate_test`); it is consumed as a STREAM (never materialised):
    background threads read/collate ahead into persistent pinned buffers, episodes run `batch` at a
    time through one C-ABI call each on `n_inflight` streams, and — under torch.distributed — are
    sharded over the ranks.  An `episode_io.EpisodeFolder` is read by several threads."""
    import torch.distributed as dist
    rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    learner.model.eval()
    ev = getattr(learner, "_evaluator", None)
    key = (tuple(test_classes), batch, bool(eval), n_inflight)
    if ev is None or getattr(learner, "_evaluator_key", None) != key:
        ev = EpisodeEvaluator(learner.model, test_classes, batch=batch, eval_mdns=bool(eval),
                              n_inflight=n_inflight)
        learner._evaluator, learner._evaluator_key = ev, key
    res = ev.run(test_loader, rank, world, logger=logger)
    return res["mean_loss"], res["mean_iou"]
