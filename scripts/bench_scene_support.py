#!/usr/bin/env python
"""Time of cutting a support set out of a labelled scan (r3dfs_scene_support) and encoding it.

    python scripts/bench_scene_support.py --out DIR [--reps 20] [--warmup 3]

Scene: the room of scripts/bench_scene.py (make_scene(7), 10 m x 10 m, 10 000 points per m^2 =
1 000 000 points) with its per-point class labels, 1 m blocks at overlap 1 and 2, seed 0.  Support:
2-way 5-shot S3DIS-shape (2048 points, 100 sub-prototypes, k_connect 200, MDNS on), classes 2 and
3 (the classes of this room with at least 5 eligible blocks at overlap 1), the reference's
eligibility rule (more than max(int(0.05 n_b), 100) points of the class), seeded fixture weights of
tests/golden.  Every repetition times three phases with CUDA events:
  plan    r3dfs_scene_plan (grid, memberships, radix sort, chunk layout)
  cut     r3dfs_scene_support (per-block class counts, choice of the shots, shot clouds and masks)
  encode  encode_support on the returned shots (r3dfs_mpti_support)
Labels are converted to int32 once, outside the timed window.  A 512 MiB write evicts the 126 MB
L2 before every timed repetition; --warmup repetitions per overlap come first.  The cut is compared
with the numpy oracle of tests/scene_support_oracle.py for the same room (torch.equal), and
support_from_scene with the cut.  One JSON line on stdout, also written to DIR/scene_support.json.
Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scripts.bench_support_reuse import gpu_info  # noqa: E402

N_WAY, K_SHOT, N_PTS = 2, 5, 2048
CLASSES = [2, 3]
PHASES = ("plan", "cut", "encode")
KEYS = ("support_x", "support_y", "src", "block", "n_eligible")


def run_phases(model, pts, labels, overlap, seed=0):
    """plan -> cut -> encode with an event after each: -> (shots, support set, [events])."""
    from r3dfsseg_b200 import ops
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(PHASES) + 1)]
    ev[0].record()
    plan = ops.scene_plan(pts, N_PTS, 1.0, overlap, seed)
    ev[1].record()
    shots = ops.scene_support(plan, labels, CLASSES, K_SHOT, seed)
    ev[2].record()
    sup = model.encode_support(shots["support_x"], shots["support_y"], eval=True)
    ev[3].record()
    return shots, sup, ev


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for scene_support.json")
    ap.add_argument("--reps", type=int, default=20, help="timed repetitions per overlap")
    ap.add_argument("--warmup", type=int, default=3, help="warm-up repetitions per overlap")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print("bench_scene_support.py needs a CUDA device (there is no CPU fallback)",
              file=sys.stderr)
        return 2

    from r3dfsseg_b200.episodes import default_args, make_scene
    from r3dfsseg_b200.models import MPTI_SelfAtten
    from tests import scene_support_oracle as S

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    model = MPTI_SelfAtten(default_args(N_WAY, K_SHOT))
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    pts_np, cls_np = make_scene(7, size_xy=(10.0, 10.0), points_per_m2=10000.0)
    pts = torch.from_numpy(pts_np).to(dev)
    labels = torch.from_numpy(cls_np).to(dev).to(torch.int32)
    M = int(pts.shape[0])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    res = {"metric": "ms to cut a support set out of a labelled scan and encode it",
           "scene": f"make_scene(7), 10 m x 10 m, {M} points, 1 m blocks, seed 0",
           "config": f"{N_WAY}-way {K_SHOT}-shot, classes {CLASSES}, {N_PTS} points per shot, "
                     "min_points 100, min_ratio 0.05, 100 sub-prototypes, k_connect 200, MDNS on, "
                     "fixture weights",
           "timing": "CUDA events between phases; 512 MiB write before every timed repetition "
                     "evicts the L2", "reps": args.reps, "warmup": args.warmup}
    ok = True
    for overlap in (1, 2):
        for _ in range(args.warmup):
            run_phases(model, pts, labels, overlap)
        torch.cuda.synchronize()
        ph = {p: [] for p in PHASES}
        tot = []
        for _ in range(args.reps):
            flush.zero_()
            shots, sup, ev = run_phases(model, pts, labels, overlap)
            torch.cuda.synchronize()
            for i, p in enumerate(PHASES):
                ph[p].append(ev[i].elapsed_time(ev[i + 1]))
            tot.append(ev[0].elapsed_time(ev[-1]))
        ref = S.support(pts_np, cls_np, CLASSES, K_SHOT, N_PTS, 1.0, overlap, 0)
        oracle_equal = bool(torch.equal(shots["support_x"].transpose(2, 3).cpu(),
                                        torch.from_numpy(ref["support_x"])))
        for k in KEYS[1:]:
            oracle_equal &= bool(torch.equal(shots[k].cpu(), torch.from_numpy(ref[k])))
        api = model.support_from_scene(pts, labels, CLASSES, overlap=overlap, seed=0)
        api_equal = all(bool(torch.equal(api[k], shots[k])) for k in KEYS)
        ok &= oracle_equal and api_equal
        mean = {p: sum(v) / len(v) for p, v in ph.items()}
        total = sum(tot) / len(tot)
        res[f"overlap{overlap}"] = {
            "n_eligible": shots["n_eligible"].tolist(),
            "blocks": shots["block"].tolist(),
            "phase_ms": {p: round(v, 4) for p, v in mean.items()},
            "phase_min_ms": {p: round(min(v), 4) for p, v in ph.items()},
            "phase_max_ms": {p: round(max(v), 4) for p, v in ph.items()},
            "total_ms": round(total, 4),
            "cut_share": round(mean["cut"] / total, 4),
            "cut_equals_oracle": oracle_equal,
            "support_from_scene_equals_cut": api_equal,
            "proto_count": sup.proto_count.tolist(),
        }
    res.update(gpu_info())
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "scene_support.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
