#!/usr/bin/env python
"""Time of sampling few-shot episodes from labelled scans on the GPU (SceneEpisodes: the dataset
index, r3dfs_scene_episodes) and its share of an evaluation run.

    python scripts/bench_scene_episodes.py --out DIR [--rooms 16] [--reps 10] [--warmup 2]

Datasets: --rooms make_scene rooms of 10 m x 10 m at 10 000 points per m^2 (1 000 000 points each,
16 000 000 for 16 rooms) with the S3DIS pool (6 classes, two blobs each per room), and as many with
the ScanNet pool (10 classes); 1 m blocks at overlap 1, 2048 points per cloud, the reference's
eligibility rule.  Measured, with CUDA events (a host clock around the index build, which
synchronises once per scan):
  index    SceneEpisodes(...): a plan per scan, r3dfs_scene_index, r3dfs_scene_index_classes
  sampler  --batch episodes per sample() call, alone: 2-way 5-shot clean on the S3DIS pool and
           3-way 5-shot with 40 % ood noise on the ScanNet pool; episodes/s and bytes written/s
  eval     EpisodeEvaluator.run_scenes over --n-eval 2-way 5-shot episodes (MDNS on) against the
           same loop over the same episodes pre-sampled and resident on the device; the legs
           alternate --reps times, and their difference is the sampler's share of the run
Every shape is warmed up first.  A 512 MiB write evicts the 126 MB L2 before every timed sampler
call.  One JSON line on stdout, also written to DIR/scene_episodes.json.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from scripts.bench_support_reuse import gpu_info  # noqa: E402

OUT_KEYS = ("support_x", "support_y", "gt_support_y", "support_flag", "query_x", "query_y",
            "shot_block", "query_block", "support_src", "query_src")


def build(dataset: str, n_rooms: int, dev: str):
    from r3dfsseg_b200.episodes import CLASS_POOL, make_scene
    from r3dfsseg_b200.scene_episodes import SceneEpisodes
    scans = []
    for i in range(n_rooms):
        p, c = make_scene(100 + i, size_xy=(10.0, 10.0), points_per_m2=10000.0, dataset=dataset)
        scans.append((torch.from_numpy(p).to(dev), torch.from_numpy(c).to(dev)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ds = SceneEpisodes(scans, list(range(CLASS_POOL[dataset])))
    torch.cuda.synchronize()
    return ds, time.perf_counter() - t0, sum(int(p.shape[0]) for p, _ in scans)


def time_sampler(ds, wc, k_shot, noise_type, ratio, reps, warmup, flush):
    for i in range(warmup):
        ds.sample(wc, k_shot, 1, i * len(wc), noise_type, ratio)
    ms = []
    for r in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = ds.sample(wc, k_shot, 1, (warmup + r) * len(wc), noise_type, ratio)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    nbytes = sum(out[k].numel() * out[k].element_size() for k in OUT_KEYS)
    med = float(np.median(ms))
    return {"episodes_per_call": len(wc), "ms_per_call_median": med,
            "ms_per_call_min": float(min(ms)), "episodes_per_s": len(wc) / med * 1e3,
            "bytes_written_per_call": nbytes, "gb_written_per_s": nbytes / med / 1e6}


def presampled_run(ev, batches, slots):
    """run_scenes' loop without the sampler: the batches are already on the device."""
    from r3dfsseg_b200 import _lib, ops
    m, dev = ev.model, ev.device
    counters = torch.zeros((3, len(ev.test_classes) + 1), dtype=torch.int64, device=dev)
    loss_sum = torch.zeros((), dtype=torch.float64, device=dev)
    cfg = m._cfg(int(batches[0]["query_x"].shape[1]), mdns=bool(ev.eval_mdns))
    ws = torch.empty(_lib.lib().r3dfs_mpti_workspace(cfg, ev.batch), dtype=torch.uint8, device=dev)
    for b, s in zip(batches, slots):
        out = m.forward_episodes(b["support_x"], b["support_y"], b["query_x"], b["query_y"],
                                 eval=ev.eval_mdns, workspace=ws, want_diag=True)
        ops.confusion_accumulate(out["pred"], b["query_y"], s, counters)
        loss_sum += out["loss"].double().sum()
    return counters, loss_sum


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for scene_episodes.json")
    ap.add_argument("--rooms", type=int, default=16, help="rooms per dataset")
    ap.add_argument("--batch", type=int, default=64, help="episodes per sample() call")
    ap.add_argument("--n-eval", type=int, default=256, help="episodes of the evaluation legs")
    ap.add_argument("--reps", type=int, default=10, help="timed repetitions")
    ap.add_argument("--warmup", type=int, default=2, help="warm-up repetitions")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene_episodes.py needs a CUDA device")
    dev = "cuda:0"
    torch.cuda.set_device(dev)
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.evaluate import EpisodeEvaluator, class_slots
    from r3dfsseg_b200.models import MPTI_SelfAtten
    res = {"gpu": gpu_info()}
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    s3dis, t_s, m_s = build("s3dis", a.rooms, dev)
    scannet, t_n, m_n = build("scannet", a.rooms, dev)
    res["index"] = {"s3dis": {"points": m_s, "blocks": s3dis.index.n_blocks, "seconds": t_s,
                              "n_eligible": s3dis.n_eligible},
                    "scannet": {"points": m_n, "blocks": scannet.index.n_blocks, "seconds": t_n,
                                "n_eligible": scannet.n_eligible}}
    rng = np.random.default_rng(0)
    wc2 = np.stack([rng.choice(6, 2, replace=False) for _ in range(a.batch)])
    wc3 = np.stack([rng.choice(10, 3, replace=False) for _ in range(a.batch)])
    res["sampler"] = {
        "s3dis_2way_5shot_clean": time_sampler(s3dis, wc2, 5, None, 0.0, a.reps, a.warmup, flush),
        "scannet_3way_5shot_ood_0.4": time_sampler(scannet, wc3, 5, "ood", 0.4, a.reps, a.warmup,
                                                   flush)}

    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    m = MPTI_SelfAtten(default_args(2, 5))
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    ev = EpisodeEvaluator(m, list(range(6)), batch=16)
    wce = np.repeat(s3dis.test_classes(2, 1), -(-a.n_eval // 15), axis=0)[:a.n_eval]
    batches = [s3dis.sample(wce[i:i + ev.batch], 5, 1, i) for i in range(0, len(wce), ev.batch)]
    slots = [torch.tensor([class_slots(c, ev.test_classes) for c in b["sampled_classes"]],
                          dtype=torch.int32, device=dev) for b in batches]
    legs = {"run_scenes": lambda: ev.run_scenes(s3dis, wce, 5, 1)["counters"],
            "presampled": lambda: presampled_run(ev, batches, slots)[0].cpu()}
    for f in legs.values():
        f()
    times = {k: [] for k in legs}
    counters = {}
    for _ in range(a.reps):
        for k, f in legs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            counters[k] = f()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    med = {k: float(np.median(v)) for k, v in times.items()}
    res["eval"] = {"episodes": len(wce), "batch": ev.batch, "mdns": True,
                   "seconds_median": med, "seconds_min": {k: min(v) for k, v in times.items()},
                   "episodes_per_s": {k: len(wce) / v for k, v in med.items()},
                   "sampler_share": (med["run_scenes"] - med["presampled"]) / med["run_scenes"],
                   "counters_equal": bool(torch.equal(counters["run_scenes"],
                                                      counters["presampled"]))}
    res["timing"] = ("sampler: CUDA events per sample() call, 512 MiB write before each; eval: "
                     "host clock around synchronised runs, legs alternating")
    line = json.dumps(res)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "scene_episodes.json"), "w") as f:
        f.write(line + "\n")
    print(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
