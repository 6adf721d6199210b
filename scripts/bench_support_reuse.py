#!/usr/bin/env python
"""Episodes/s of segmenting query clouds against ONE labelled support set, two ways, in one run:

  leg A  forward_episodes in calls of --chunk episodes that all repeat the same support set: the
         support clouds are encoded, denoised and turned into prototypes again in every call;
  leg B  encode_support once, then segment in calls of --chunk episodes sharing that set (the
         query half reads the set's prototypes in place, episode stride 0).

    python scripts/bench_support_reuse.py --out DIR [--calls 20] [--warmup 10] [--chunk 25]

Shapes: BASELINE.json configs[2] (S3DIS-shape 2-way 5-shot, 2048 points, n_query 2, 100
sub-prototypes per way, k_connect 200, MDNS on), the seeded fixture weights of tests/golden.
The two legs alternate call by call after --warmup warm-up calls each; every timed call is timed
by CUDA events, and a 512 MiB write between timed calls evicts the 126 MB L2 (as bench.py does).
Per-stage device times of both calls come from a separate serialised run with stage events.
The outputs of the two legs on the timed inputs are compared with torch.equal.
One JSON line on stdout, also written to DIR/support_reuse.json.  Needs a CUDA device: there is
no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_WAY, K_SHOT, N_QUERY, N_PTS = 2, 5, 2, 2048


def gpu_info() -> dict:
    """Device name, power limit and maximum SM clock, read while the measurement runs."""
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = r.stdout.strip() if r.returncode == 0 else f"failed: {r.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired) as e:
        info["nvidia_smi"] = f"failed: {e}"
    return info


def stage_times(run, n_calls: int, flush: torch.Tensor) -> dict:
    """Mean device time per stage of `run(stage_events)` over n_calls serialised calls (ms)."""
    from r3dfsseg_b200 import _lib
    names = _lib.STAGES
    per_call = []
    for _ in range(n_calls):
        evs = [torch.cuda.Event(enable_timing=True) for _ in names]
        for e in evs:
            e.record()  # materialise the cudaEvent_t handles
        flush.zero_()
        run(evs)
        per_call.append(evs)
    torch.cuda.synchronize()
    return {names[i]: round(sum(evs[i - 1].elapsed_time(evs[i]) for evs in per_call) / n_calls, 4)
            for i in range(1, len(names))}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for support_reuse.json")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per leg (>= 20)")
    ap.add_argument("--warmup", type=int, default=10, help="warm-up calls per leg (>= 10)")
    ap.add_argument("--chunk", type=int, default=25, help="episodes per call")
    ap.add_argument("--seed", type=int, default=20_000)
    args = ap.parse_args()
    if args.calls < 20 or args.warmup < 10:
        ap.error("--calls must be >= 20 and --warmup >= 10")
    if not torch.cuda.is_available():
        print("bench_support_reuse.py needs a CUDA device (there is no CPU fallback)", file=sys.stderr)
        return 2

    from r3dfsseg_b200 import ops
    from r3dfsseg_b200.episodes import default_args, make_episode
    from r3dfsseg_b200.models import MPTI_SelfAtten

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    model = MPTI_SelfAtten(default_args(N_WAY, K_SHOT))
    model.load_state_dict(sd)
    model = model.to(dev).eval()

    # one labelled support set; E query episodes (N_QUERY clouds each) to segment against it
    E = args.chunk
    sup_ep = make_episode(args.seed, N_WAY, K_SHOT)
    q_eps = [make_episode(args.seed + 1 + i, N_WAY, K_SHOT) for i in range(E)]
    sx1 = sup_ep.support_x.transpose(2, 3).contiguous().to(dev).transpose(2, 3)  # point-major
    sy1 = sup_ep.support_y.to(dev)
    qx = torch.stack([e.query_x.transpose(1, 2) for e in q_eps]).to(dev).transpose(2, 3)
    qy = torch.stack([e.query_y for e in q_eps]).to(dev)
    # leg A: the support set repeated for every episode of a call, as forward_episodes takes it
    sxE = sx1.unsqueeze(0).expand(E, -1, -1, -1, -1).transpose(3, 4).contiguous().transpose(3, 4)
    syE = sy1.unsqueeze(0).expand(E, -1, -1, -1).contiguous()

    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    out = {}

    def leg_a():
        out["a"] = model.forward_episodes(sxE, syE, qx, qy, eval=True)

    support = model.encode_support(sx1, sy1, eval=True)

    def leg_b():
        out["b"] = model.segment(support, qx, qy)

    legs = {"a": leg_a, "b": leg_b}
    for _ in range(args.warmup):
        leg_a()
        leg_b()
    torch.cuda.synchronize()

    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(args.calls)] for k in legs}
    for i in range(args.calls):
        for k, run in legs.items():
            flush.zero_()
            ev[k][i][0].record()
            run()
            ev[k][i][1].record()
    torch.cuda.synchronize()
    ms = {k: [a.elapsed_time(b) for a, b in ev[k]] for k in legs}
    equal = {f: bool(torch.equal(out["a"][f], out["b"][f])) for f in ("logits", "loss", "pred")}

    # encode_support itself (once per labelled set in leg B; not part of its per-call time)
    enc_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(5)]
    for a, b in enc_ev:
        flush.zero_()
        a.record()
        model.encode_support(sx1, sy1, eval=True)
        b.record()
    torch.cuda.synchronize()
    enc_ms = sum(a.elapsed_time(b) for a, b in enc_ev) / len(enc_ev)

    # per-stage device times, serialised, in a run of their own
    pw, cfg = model._weights(), model._cfg(N_QUERY, mdns=True)
    stages_query = stage_times(
        lambda evs: ops.mpti_query(pw, cfg, support.prototypes, support.proto_count, qx, qy,
                                   shared=True, stage_events=evs), 10, flush)
    stages_forward = stage_times(
        lambda evs: model.forward_episodes(sxE, syE, qx, qy, eval=True, stage_events=evs), 10, flush)

    def summary(v):
        v = sorted(v)
        mean = sum(v) / len(v)
        return {"mean_ms": round(mean, 4), "median_ms": round(v[len(v) // 2], 4),
                "min_ms": round(v[0], 4), "max_ms": round(v[-1], 4),
                "episodes_per_s": round(E / (mean / 1e3), 2)}

    res = {
        "metric": "episodes/s segmenting against one support set (2-way 5-shot, 2048 pts)",
        "config": f"{N_WAY}-way {K_SHOT}-shot, {N_PTS} points, n_query {N_QUERY}, 100 "
                  "sub-prototypes, k_connect 200, MDNS on, fixture weights",
        "episodes_per_call": E, "timed_calls_per_leg": args.calls, "warmup_calls_per_leg": args.warmup,
        "timing": "CUDA events per call, legs alternating; 512 MiB write between timed calls "
                  "evicts the L2",
        "leg_a_forward_episodes": summary(ms["a"]),
        "leg_b_segment": summary(ms["b"]),
        "speedup_b_over_a": round(sum(ms["a"]) / sum(ms["b"]), 3),
        "encode_support_ms": round(enc_ms, 4),
        "outputs_equal": equal,
        "stage_ms_query_call": stages_query,
        "stage_ms_forward_call": stages_forward,
        **gpu_info(),
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "support_reuse.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res), flush=True)
    return 0 if all(equal.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
