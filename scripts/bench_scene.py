#!/usr/bin/env python
"""Points/s of labelling a whole scan against one support set (MPTI_SelfAtten.segment_scene).

    python scripts/bench_scene.py --out DIR [--reps 5] [--warmup 2] [--chunk-batch 64]

Scene: one synthetic room of make_scene (10 m x 10 m, 10 000 points per m^2 = 1 000 000 points),
against one 2-way 5-shot S3DIS-shape support set (2048 points, 100 sub-prototypes, k_connect 200,
MDNS on), seeded fixture weights of tests/golden, 1 m blocks at overlap 1 and 2.
Every repetition runs the four phases of segment_scene with CUDA events between them:
  plan    r3dfs_scene_plan (grid, memberships, radix sort, chunk layout); then the one read-back
          of the chunk count (host time, reported apart)
  chunks  r3dfs_scene_chunks (the (E, N, 9) chunk clouds)
  query   r3dfs_mpti_query over the chunks, --chunk-batch 1-query episodes per call
  merge   r3dfs_scene_merge
A 512 MiB write evicts the 126 MB L2 before every timed repetition; --warmup repetitions per overlap
come first.  The phase-by-phase result is compared with segment_scene's (torch.equal).
One JSON line on stdout, also written to DIR/scene.json.  Needs a CUDA device.
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

import torch  # noqa: E402

from scripts.bench_support_reuse import gpu_info  # noqa: E402

N_WAY, K_SHOT, N_PTS = 2, 5, 2048
PHASES = ("plan", "chunks", "query", "merge")


def run_phases(model, support, pts, overlap, chunk_batch, seed=0):
    """segment_scene's steps with an event after each: -> (out, [events], readback_s, E)."""
    from r3dfsseg_b200 import ops
    pw = model._weights()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(PHASES) + 1)]
    ev[0].record()
    plan = ops.scene_plan(pts, N_PTS, 1.0, overlap, seed)
    ev[1].record()
    t0 = time.perf_counter()
    E = int(plan.n_chunks.item())
    readback = time.perf_counter() - t0
    chunk_x, _ = ops.scene_chunks(plan, E)
    ev[2].record()
    qx = chunk_x.view(E, 1, N_PTS, 9).transpose(2, 3)
    logits = torch.empty((E, N_PTS, N_WAY + 1), dtype=torch.float32, device=pts.device)
    for b0 in range(0, E, chunk_batch):
        logits[b0:b0 + chunk_batch] = model._query(pw, support, qx[b0:b0 + chunk_batch])[0][:, 0]
    ev[3].record()
    out = ops.scene_merge(plan, logits, E)
    ev[4].record()
    return out, ev, readback, E


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for scene.json")
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions per overlap")
    ap.add_argument("--warmup", type=int, default=2, help="warm-up repetitions per overlap")
    ap.add_argument("--chunk-batch", type=int, default=64)
    ap.add_argument("--size", type=float, default=10.0, help="room side in metres")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("bench_scene.py needs a CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2

    from r3dfsseg_b200.episodes import default_args, make_episode, make_scene
    from r3dfsseg_b200.models import MPTI_SelfAtten

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    model = MPTI_SelfAtten(default_args(N_WAY, K_SHOT))
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    ep = make_episode(20_000, N_WAY, K_SHOT)
    support = model.encode_support(ep.support_x.to(dev), ep.support_y.to(dev), eval=True)
    pts = torch.from_numpy(make_scene(7, size_xy=(args.size, args.size),
                                      points_per_m2=10000.0)[0]).to(dev)
    M = int(pts.shape[0])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    res = {"metric": "points/s labelling a whole scan against one support set",
           "scene": f"make_scene(7), {args.size:g} m x {args.size:g} m, {M} points, 1 m blocks",
           "config": f"{N_WAY}-way {K_SHOT}-shot, {N_PTS} points per chunk, 100 sub-prototypes, "
                     f"k_connect 200, MDNS on, fixture weights, chunk_batch {args.chunk_batch}",
           "timing": "CUDA events between phases; 512 MiB write before every timed repetition "
                     "evicts the L2", "reps": args.reps, "warmup": args.warmup}
    ok = True
    for overlap in (1, 2):
        for _ in range(args.warmup):
            run_phases(model, support, pts, overlap, args.chunk_batch)
        torch.cuda.synchronize()
        ph = {p: [] for p in PHASES}
        tot, rb = [], []
        for _ in range(args.reps):
            flush.zero_()
            out, ev, readback, E = run_phases(model, support, pts, overlap, args.chunk_batch)
            torch.cuda.synchronize()
            for i, p in enumerate(PHASES):
                ph[p].append(ev[i].elapsed_time(ev[i + 1]))
            tot.append(ev[0].elapsed_time(ev[-1]))
            rb.append(readback * 1e3)
        ref = model.segment_scene(support, pts, overlap=overlap, seed=0,
                                  chunk_batch=args.chunk_batch)
        equal = all(bool(torch.equal(out[k], ref[k])) for k in ("logits", "pred", "coverage"))
        ok &= equal
        mean = {p: sum(v) / len(v) for p, v in ph.items()}
        total = sum(tot) / len(tot)
        res[f"overlap{overlap}"] = {
            "n_chunks": E,
            "phase_ms": {p: round(v, 4) for p, v in mean.items()},
            "readback_host_ms": round(sum(rb) / len(rb), 4),
            "total_ms": round(total, 3), "total_min_ms": round(min(tot), 3),
            "total_max_ms": round(max(tot), 3),
            "points_per_s": round(M / (total / 1e3)),
            "share_outside_query": round(1.0 - mean["query"] / total, 4),
            "mean_coverage": round(float(ref["coverage"].float().mean()), 4),
            "equals_segment_scene": equal,
        }
    res.update(gpu_info())
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "scene.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
