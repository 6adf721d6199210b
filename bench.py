#!/usr/bin/env python
"""bench.py — MPTI episodes/s (2-way 5-shot, 2048 pts) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" = one pass of the episode hot path over one batch of `--episodes` (default 100) synthetic
S3DIS-shape 2-way 5-shot episodes (BASELINE.json configs[2]), fed to the C ABI in chunks of
`--chunk` episodes per call.  Episodes are independent: with N ranks every rank runs its own 100
episodes per step (weak scaling) and the only collective is the NCCL sum of the confusion counters.

One JSON line on stdout (rank 0):
  value      episodes/s with the inputs already resident in HBM (device-timed, max over ranks)
  e2e        the same through the public module API from pinned HOST buffers, H2D + D2H in the
             timed region
  roofline   the dominant kernel: algorithmic DRAM bytes (or FLOPs) per launch / CUDA-event time
  e2e_driver the same metric through the drop-in driver (evaluate.test_few_shot over episode FILES:
             disk -> reader threads -> pinned staging -> H2D -> forward -> counters -> mIoU)
  extra      BASELINE.json configs[3] (ScanNet-shape 3-way, 40 % OOD shots) and configs[4] (the
             meta-training step, gradient all-reduce included at N > 1) measured in the same run
  cpu_baseline  the CPU oracle (restatement of the reference's path) on this box's host cores
`--impl reference` times that CPU path alone (the reference is Python: oracle/mpti_oracle.py is
its restatement; the reference tree itself cannot travel to the GPU box).
`--dump-outputs DIR` writes what the last timed step of the headline path returned (rank 0) as
DIR/logits.npy, loss.npy, pred.npy (float32): the inputs are seeded, so two builds of the project
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_WAY, K_SHOT, N_QUERY, N_PTS = 2, 5, 2, 2048
DATASET, NOISE = "s3dis", 0.0
METRIC = "MPTI episodes/s (2-way 5-shot, 2048 pts)"
UNIT = "episodes/s"
WORKLOADS = {
    # BASELINE.json configs[2] (the headline) and configs[4-1] (ScanNet-shape, 40 % OOD-noise shots)
    "s3dis_2way_5shot": dict(n_way=2, k_shot=5, dataset="s3dis", noise=0.0,
                             label="S3DIS-shape 2-way 5-shot MPTI eval, MDNS on, 100 sub-prototypes/"
                                   "way, k_connect 200 (BASELINE.json configs[2])"),
    "scannet_3way_5shot_ood": dict(n_way=3, k_shot=5, dataset="scannet", noise=0.4,
                                   label="ScanNet-shape 3-way 5-shot, 40 % OOD-noise shots, MDNS on "
                                         "(BASELINE.json configs[3])"),
}


def set_workload(name: str) -> str:
    global N_WAY, K_SHOT, N_QUERY, DATASET, NOISE, METRIC
    w = WORKLOADS[name]
    N_WAY, K_SHOT, DATASET, NOISE = w["n_way"], w["k_shot"], w["dataset"], w["noise"]
    N_QUERY = N_WAY
    METRIC = f"MPTI episodes/s ({N_WAY}-way {K_SHOT}-shot, 2048 pts)"
    return w["label"]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# synthetic episodes
# ------------------------------------------------------------------------------------------------
def build_host_batch(n_episodes: int, seed0: int):
    """Pinned host tensors laid out like the reference's collate output, batched:
    support (E, n_way, k_shot, N, 9) point-major, masks int32, query (E, n_q, N, 9), labels int64."""
    from r3dfsseg_b200.episodes import make_episode
    sx = torch.empty((n_episodes, N_WAY, K_SHOT, N_PTS, 9), dtype=torch.float32).pin_memory()
    sy = torch.empty((n_episodes, N_WAY, K_SHOT, N_PTS), dtype=torch.int32).pin_memory()
    qx = torch.empty((n_episodes, N_QUERY, N_PTS, 9), dtype=torch.float32).pin_memory()
    qy = torch.empty((n_episodes, N_QUERY, N_PTS), dtype=torch.int64).pin_memory()
    classes = np.zeros((n_episodes, N_WAY), dtype=np.int32)
    for i in range(n_episodes):
        ep = make_episode(seed0 + i, N_WAY, K_SHOT, dataset=DATASET, noise_ratio=NOISE)
        sx[i] = ep.support_x.transpose(2, 3)
        sy[i] = ep.support_y
        qx[i] = ep.query_x.transpose(1, 2)
        qy[i] = ep.query_y
        classes[i] = ep.sampled_classes
    return sx, sy, qx, qy, classes


DUMP_BYTES = 63 * 10**6  # array data; with the .npy headers the dump stays under 64 MB


def dump_outputs(out_dir: str, outs):
    """forward_episodes' outputs of every chunk of one step -> out_dir/{logits,loss,pred}.npy in
    float32 (pred holds class indices, exact in float32), episodes in input order.  Past DUMP_BYTES
    in all, only the first episodes are written."""
    arrays = {k: torch.cat([o[k] for o in outs]).float().cpu().numpy()
              for k in ("logits", "loss", "pred")}
    per_episode = sum(a[0].nbytes for a in arrays.values())
    keep = min(len(arrays["loss"]), DUMP_BYTES // per_episode)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[:keep])


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                 str(self.index), "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU path (oracle = restatement of the reference's implementation)
# ------------------------------------------------------------------------------------------------
def cpu_episodes_per_s(n_episodes: int, seed0: int, threads: int):
    from oracle import mpti_oracle as O
    from r3dfsseg_b200.episodes import make_episode
    torch.set_num_threads(threads)
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    eps = [make_episode(seed0 + i, N_WAY, K_SHOT, dataset=DATASET, noise_ratio=NOISE)
           for i in range(n_episodes)]
    t0 = time.perf_counter()
    with torch.no_grad():
        for ep in eps:
            # timing arm: FP32 Gram + topk stands in for faiss (the parity definition — FP64 distances
            # and a full stable argsort — would be an unfairly slow baseline)
            O.forward_episode(sd, ep.support_x, ep.support_y, ep.query_x, ep.query_y, eval_mdns=True,
                              timing_knn=True)
    dt = time.perf_counter() - t0
    return n_episodes / dt, dt


def run_reference_arm(args):
    """The reference's CPU implementation of the path (oracle port), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    per_step = args.ref_episodes_per_step
    for _ in range(args.warmup):
        cpu_episodes_per_s(per_step, 900, threads)
    t_tot, n_tot = 0.0, 0
    for s in range(args.steps):
        _, dt = cpu_episodes_per_s(per_step, 1000 + s * per_step, threads)
        t_tot += dt
        n_tot += per_step
    v = n_tot / t_tot
    sample = (f"{per_step} episode(s) per step x {args.steps} steps of the same {N_WAY}-way {K_SHOT}-shot "
              f"workload (MDNS on), torch CPU fp32, {threads} threads of ONE host (under torchrun "
              f"rank 0 alone runs this arm: at N > 1 it is still one host, not N)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload]["label"] + " - CPU oracle port of the "
                               "reference path", "episodes_per_step": per_step,
                   "n_points": N_PTS, "n_subprototypes": 100, "k_connect": 200},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# algorithmic work per stage and per call of `E` episodes (DESIGN.md "kernels" table)
# ------------------------------------------------------------------------------------------------
def node_slots() -> int:
    """prototype slots ((n_way+1) x 101, padded to 64) + query points (r3dfs_mpti_forward layout)"""
    return ((N_WAY + 1) * 101 + 63) // 64 * 64 + N_QUERY * N_PTS


def stage_work(E: int):
    B = E * (N_QUERY + N_WAY * K_SHOT)          # clouds
    M = B * N_PTS                               # points
    k = 20
    nn = node_slots()                           # node slots per graph
    n_sup = N_WAY * K_SHOT * N_PTS
    w = {}
    for i, C in enumerate((9, 64, 64)):
        w[f"knn{i}"] = dict(flops=2.0 * B * N_PTS * N_PTS * C + 3.0 * B * N_PTS * N_PTS,
                            bytes=4.0 * M * C + 4.0 * M * k, bound="tensor")
        w[f"pq{i}"] = dict(flops=2.0 * M * C * 128, bytes=4.0 * M * (C + 128), bound="tensor")
        w[f"edge{i}"] = dict(flops=2.0 * 64 * 64 * M * k, bytes=4.0 * M * (128 + 64) + 4.0 * M * k,
                             bound="tensor")
    w["mlp"] = dict(flops=2.0 * M * (192 * 512 + 512 * 256), bytes=4.0 * M * (192 + 256), bound="tensor")
    w["base"] = dict(flops=2.0 * M * (256 * 128 + 128 * 64), bytes=4.0 * M * (256 + 64), bound="tensor")
    w["qkv"] = dict(flops=2.0 * M * 256 * 192, bytes=4.0 * M * (256 + 192), bound="tensor")
    w["att"] = dict(flops=4.0 * B * N_PTS * N_PTS * 64, bytes=4.0 * M * (192 + 64), bound="tensor")
    # FPS: DRAM-level = two passes over the FP32 rows (distance to the first seed + min/max, then
    # quantisation) + ~3.5 % of the rows re-read per pick; on-chip = 100 sweeps of the byte rows
    w["fps"] = dict(flops=3.0 * 100 * E * n_sup * 192,
                    bytes=(2 + 0.035 * 100) * 4.0 * E * n_sup * 192,
                    onchip_bytes=100.0 * E * n_sup * 192, bound="hbm")
    w["proto"] = dict(flops=3.0 * 100 * E * n_sup * 192, bytes=2 * 4.0 * E * n_sup * 192, bound="hbm")
    w["mdns"] = dict(flops=2.0 * E * n_sup * 192, bytes=4.0 * E * n_sup * 192, bound="hbm")
    w["sets"] = dict(flops=0.0, bytes=2 * 4.0 * E * n_sup * 192, bound="hbm")
    w["dist"] = dict(flops=2.0 * E * nn * nn * 192, bytes=4.0 * E * nn * (192 + nn), bound="tensor")
    w["select"] = dict(flops=0.0, bytes=4.0 * E * nn * nn + 4.0 * E * nn * 200, bound="hbm")
    # edge similarities: compulsory = features once + lists in / similarities out; the gathered
    # neighbour rows (4*nn*200*192 B) come from L2
    w["sim"] = dict(flops=3.0 * E * nn * 200 * 192, bytes=4.0 * E * nn * (192 + 2 * 200),
                    l2_bytes=4.0 * E * nn * 200 * 192, bound="hbm")
    w["sym"] = dict(flops=0.0, bytes=6 * 8.0 * E * nn * 200, bound="hbm")
    w["cg"] = dict(flops=0.0, bytes=None, bound="hbm")  # filled from the measured iteration count
    w["input"] = dict(flops=0.0, bytes=2 * 4.0 * M * 9, bound="hbm")
    w["head"] = dict(flops=0.0, bytes=2 * 4.0 * E * N_QUERY * N_PTS * (N_WAY + 1), bound="hbm")
    return w


# ------------------------------------------------------------------------------------------------
# extra legs: the drop-in driver over episode files, BASELINE.json configs[3] and configs[4]
# ------------------------------------------------------------------------------------------------
def driver_leg(model, dev, dist, rank, world, host_batch, chunk, steps, test_classes):
    """MPTI episodes/s through evaluate.EpisodeEvaluator / test_few_shot's loop over an
    episode_io.EpisodeFolder: files on disk -> reader threads -> persistent pinned staging buffers ->
    H2D -> forward_episodes on several streams -> confusion counters (+ the NCCL sum at N > 1) ->
    mIoU.  Wall clock around the call, device synchronised on both sides, max over ranks."""
    import shutil
    import tempfile
    from r3dfsseg_b200 import episode_io as IO
    from r3dfsseg_b200.evaluate import EpisodeEvaluator
    h_sx, h_sy, h_qx, h_qy, classes = host_batch
    E = h_sx.shape[0]
    d = tempfile.mkdtemp(prefix="r3dfs_bench_eps_r%d_" % rank)
    try:
        for i in range(E):
            zs = np.zeros(tuple(h_sy[i].shape), np.int32)
            zq = np.zeros(tuple(h_qy[i].shape), np.int32)
            IO.write_episode(os.path.join(d, "%05d.r3ep" % i),
                             (h_sx[i].numpy(), h_sy[i].numpy(), h_qx[i].numpy(), h_qy[i].numpy(),
                              classes[i], zs, zq, h_sy[i].numpy()))
        folder = IO.EpisodeFolder(d)
        ev = EpisodeEvaluator(model, test_classes, batch=chunk, eval_mdns=True, n_inflight=4)
        res = ev.run(folder)  # warm-up: staging buffers, workspaces, page cache
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = ev.run(folder)  # every rank streams its own folder; counters are summed over ranks
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t[0])
        nbytes = sum(os.path.getsize(f) for f in folder.file_names)
        return {"value": world * E * steps / dt, "unit": UNIT,
                "path": "episode files (reference schema, %s) -> evaluate.EpisodeEvaluator.run: "
                        "%d reader threads, 4 batches of %d episodes in flight" % (
                            os.path.splitext(folder.file_names[0])[1], ev.n_readers, chunk),
                "file_bytes_per_step": int(nbytes), "mean_iou": res["mean_iou"],
                "timing": "wall clock, device synchronised on both sides, max over ranks"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def resident_leg(dev, dist, rank, world, workload, E_step, chunk, n_streams, steps, warmup):
    """Device-resident episodes/s of another workload (same timing rules as the main line)."""
    label = set_workload(workload)
    from r3dfsseg_b200 import _lib
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    model = MPTI_SelfAtten(default_args(N_WAY, K_SHOT))
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    h = build_host_batch(E_step, seed0=50_000 * (rank + 1))
    d_sx, d_sy, d_qx, d_qy = (t.to(dev) for t in h[:4])
    cfg = model._cfg(N_QUERY, mdns=True)
    need = _lib.lib().r3dfs_mpti_workspace(cfg, chunk)
    wss = [torch.empty(need, dtype=torch.uint8, device=dev) for _ in range(n_streams)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
    chunks = [(s, min(s + chunk, E_step)) for s in range(0, E_step, chunk)]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    acc = []

    def step():
        cur = torch.cuda.current_stream()
        for st in streams:
            st.wait_stream(cur)
        for ci, (a, b) in enumerate(chunks):
            with torch.cuda.stream(streams[ci % n_streams]):
                out = model.forward_episodes(d_sx[a:b].transpose(3, 4), d_sy[a:b],
                                             d_qx[a:b].transpose(2, 3), d_qy[a:b], eval=True,
                                             workspace=wss[ci % n_streams])
                acc.append(out["pred"])
        for st in streams:
            cur.wait_stream(st)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(steps)]
    for s_ in range(steps):
        flush.zero_()
        ev[s_][0].record()
        step()
        ev[s_][1].record()
    torch.cuda.synchronize()
    ms = float(sum(a.elapsed_time(b) for a, b in ev))
    if dist is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    pred = torch.cat([p.reshape(-1) for p in acc[-len(chunks):]]).cpu()
    acc_pts = float((pred == h[3].reshape(-1).to(torch.int32)).float().mean())
    return {"metric": METRIC, "value": world * E_step * steps / (ms * 1e-3), "unit": UNIT,
            "ms_per_step": ms / steps, "workload": label, "episodes_per_step_per_gpu": E_step,
            "episodes_per_call": chunk, "streams": n_streams, "point_accuracy_synthetic": acc_pts}


def train_leg(dev, dist, rank, world, steps, warmup):
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "bench_train", os.path.join(ROOT, "scripts", "bench_train.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    line = mod.measure(dev, dist, rank, world, steps, warmup, n_episodes=8, cpu_steps=0)
    keep = ("metric", "value", "unit", "ms_per_step", "phases_ms", "allreduce_us_1p5MB",
            "gpu_launches", "final_loss")
    out = {k: line[k] for k in keep}
    out["workload"] = line["config"]["workload"]
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--episodes", type=int, default=100, help="episodes per step per GPU")
    ap.add_argument("--chunk", type=int, default=25, help="episodes per C-ABI call")
    ap.add_argument("--streams", type=int, default=4,
                    help="CUDA streams the chunks of a step are spread over (independent episodes)")
    ap.add_argument("--cpu-episodes", type=int, default=5, help="cpu_baseline sample size")
    ap.add_argument("--ref-episodes-per-step", type=int, default=2)
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the configs[3] / configs[4] / driver legs (profiling runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="s3dis_2way_5shot", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's logits / loss / pred as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the b200 path")
    workload_label = set_workload(args.workload)
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: W >= 3

    if args.impl == "reference":
        run_reference_arm(args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL may print its version banner on stdout; keep stdout for the one JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    from r3dfsseg_b200 import _lib, ops
    from r3dfsseg_b200.episodes import default_args
    from r3dfsseg_b200.models import MPTI_SelfAtten

    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights_fixture.pt"))
    model = MPTI_SelfAtten(default_args(N_WAY, K_SHOT))
    model.load_state_dict(sd)
    model = model.to(dev).eval()

    E_step, chunk = args.episodes, min(args.chunk, args.episodes)
    h_sx, h_sy, h_qx, h_qy, classes = build_host_batch(E_step, seed0=10_000 * (rank + 1))
    test_classes = list(range(10 if DATASET == "scannet" else 6))
    slot_host = torch.tensor(classes + 1, dtype=torch.int32)  # test_classes.index(c) + 1
    d_sx, d_sy, d_qx, d_qy = (t.to(dev) for t in (h_sx, h_sy, h_qx, h_qy))
    d_slot = slot_host.to(dev)
    counters = torch.zeros((3, len(test_classes) + 1), dtype=torch.int64, device=dev)
    step_counters = torch.zeros_like(counters)
    cfg = model._cfg(N_QUERY, mdns=True)
    ws = torch.empty(_lib.lib().r3dfs_mpti_workspace(cfg, chunk), dtype=torch.uint8, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    chunks = [(s, min(s + chunk, E_step)) for s in range(0, E_step, chunk)]
    outs = [None] * len(chunks)  # what forward_episodes returned for each chunk of the last step
    n_stage = len(_lib.STAGES)

    def new_events():
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_stage)]
        for e in evs:
            e.record()  # materialise the cudaEvent_t handle
        return evs

    n_streams = max(1, min(args.streams, len(chunks)))
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]
    wss = [ws] + [torch.empty_like(ws) for _ in range(n_streams - 1)]

    def run_step_resident(stage_ev=None):
        """Chunks are independent episodes: they are spread round-robin over `n_streams` streams
        (each with its own workspace) so latency-bound kernels of one chunk overlap the other's.
        With stage events the chunks run serialised on the current stream (clean per-stage times)."""
        if stage_ev is not None or n_streams == 1:
            for ci, (a, b) in enumerate(chunks):
                out = model.forward_episodes(d_sx[a:b].transpose(3, 4), d_sy[a:b],
                                             d_qx[a:b].transpose(2, 3), d_qy[a:b], eval=True,
                                             workspace=ws,
                                             stage_events=None if stage_ev is None else stage_ev[ci])
                outs[ci] = out
                ops.confusion_accumulate(out["pred"], d_qy[a:b], d_slot[a:b], step_counters)
        else:
            cur = torch.cuda.current_stream()
            for s in streams:
                s.wait_stream(cur)
            for ci, (a, b) in enumerate(chunks):
                s = streams[ci % n_streams]
                with torch.cuda.stream(s):
                    out = model.forward_episodes(d_sx[a:b].transpose(3, 4), d_sy[a:b],
                                                 d_qx[a:b].transpose(2, 3), d_qy[a:b], eval=True,
                                                 workspace=wss[ci % n_streams])
                    outs[ci] = out
            for s in streams:
                cur.wait_stream(s)
            for ci, (a, b) in enumerate(chunks):
                ops.confusion_accumulate(outs[ci]["pred"], d_qy[a:b], d_slot[a:b], step_counters)
        if dist is not None:
            dist.all_reduce(step_counters, op=dist.ReduceOp.SUM)  # the path's only collective
        counters.add_(step_counters)
        step_counters.zero_()

    h_pred = torch.empty((E_step, N_QUERY, N_PTS), dtype=torch.int32).pin_memory()
    h_loss = torch.empty((E_step,), dtype=torch.float32).pin_memory()

    def run_step_e2e():
        cur = torch.cuda.current_stream()
        for s in streams:
            s.wait_stream(cur)
        for ci, (a, b) in enumerate(chunks):
            s = streams[ci % n_streams]
            with torch.cuda.stream(s):
                sx = h_sx[a:b].to(dev, non_blocking=True)
                sy = h_sy[a:b].to(dev, non_blocking=True)
                qx = h_qx[a:b].to(dev, non_blocking=True)
                qy = h_qy[a:b].to(dev, non_blocking=True)
                out = model.forward_episodes(sx.transpose(3, 4), sy, qx.transpose(2, 3), qy,
                                             eval=True, workspace=wss[ci % n_streams])
                h_pred[a:b].copy_(out["pred"], non_blocking=True)
                h_loss[a:b].copy_(out["loss"], non_blocking=True)
                for t_ in (sx, sy, qx, qy, out["pred"], out["loss"], out["logits"]):
                    t_.record_stream(s)
        for s in streams:
            cur.wait_stream(s)

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up ------------------------------------------------------------------------------
    for _ in range(args.warmup):
        run_step_resident()
    for _ in range(2):
        run_step_e2e()
    sync_all()

    # ---- timed: K steps, device-timed per step, L2 flushed between steps ------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    L = _lib.lib()
    step_events = [[new_events() for _ in chunks] for _ in range(args.steps)]
    t_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            for _ in range(args.steps)]
    sync_all()
    launches0 = L.r3dfs_launch_count()
    wall0 = time.perf_counter()
    for s in range(args.steps):
        flush.zero_()
        t_ev[s][0].record()
        run_step_resident()
        t_ev[s][1].record()
    sync_all()
    wall_resident = time.perf_counter() - wall0
    launches = L.r3dfs_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    # per-stage device times: the same K steps again, serialised on one stream with stage events
    for s in range(args.steps):
        flush.zero_()
        run_step_resident(step_events[s])
    sync_all()
    ms_steps = [a.elapsed_time(b) for a, b in t_ev]
    total_ms = float(sum(ms_steps))

    # ---- timed: e2e (pinned host -> device -> host) ----------------------------------------------
    e_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            for _ in range(args.steps)]
    sync_all()
    for s in range(args.steps):
        flush.zero_()
        e_ev[s][0].record()
        run_step_e2e()
        e_ev[s][1].record()
    sync_all()
    e2e_ms = float(sum(a.elapsed_time(b) for a, b in e_ev))
    clocks = sampler.stop()

    if dist is not None:
        t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms = float(t[0]), float(t[1])

    # ---- per-stage device times (rank 0), averaged per call ---------------------------------------
    stage_ms = {name: 0.0 for name in _lib.STAGES[1:]}
    n_calls = 0
    for s in range(args.steps):
        for evs in step_events[s]:
            n_calls += 1
            for i in range(1, n_stage):
                stage_ms[_lib.STAGES[i]] += evs[i - 1].elapsed_time(evs[i])
    stage_ms = {k: v / n_calls for k, v in stage_ms.items()}
    diag = model.forward_episodes(d_sx[:chunk].transpose(3, 4), d_sy[:chunk],
                                  d_qx[:chunk].transpose(2, 3), d_qy[:chunk], eval=True,
                                  workspace=ws, want_diag=True)["diag"]
    cg_iters = float(diag["cg_iters"].float().mean())
    torch.cuda.synchronize()

    peaks = load_peaks()
    work = stage_work(chunk)
    nn = node_slots()
    # CG: per iteration 6 B (u16 column + fp32 value) per stored non-zero of the merged symmetric
    # rows (<= 2*nn*200, mutual pairs stored once per row: ~0.66 of that) + the padded vectors.
    # The 25 matrices of a call (175 MB) do not stay in L2, so this is DRAM traffic (ncu: 9.8 GB).
    work["cg"]["bytes"] = chunk * cg_iters * (6.0 * 0.66 * 2 * nn * 200 + 7 * 4.0 * nn * 4)
    work["cg"]["compulsory_bytes"] = chunk * (6.0 * 0.66 * 2 * nn * 200 + 7 * 4.0 * nn * 4)
    # 3xTF32 ceiling: measured 2047 TF32 MAC/clk/SM (scripts/microbench/mma_rate.cu) x SMs x the SM
    # clock seen during this run / 3 products per reference-math product
    sm_clock_hz = 1e6 * (clocks.get("sm_mhz") or 1965.0)
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    tf32x3_tflops = 2.0 * 2047 * n_sm * sm_clock_hz / 3.0 / 1e12
    stages = {}
    for name, ms in stage_ms.items():
        wk = work.get(name)
        if wk is None or ms <= 0:
            continue
        ent = {"ms_per_call": round(ms, 4), "bound": wk["bound"]}
        if wk["bound"] == "tensor":
            ent["tflops"] = round(wk["flops"] / (ms * 1e-3) / 1e12, 3)
            ent["frac"] = round(ent["tflops"] / tf32x3_tflops, 5)
            ent["frac_of_bf16_peak"] = round(ent["tflops"] / peaks["bf16_tflops_sustained"], 5)
        else:
            ent["gbs"] = round(wk["bytes"] / (ms * 1e-3) / 1e9, 2)   # DRAM-level algorithmic bytes
            ent["frac"] = round(ent["gbs"] / peaks["hbm_gbs"], 5)
            for key, label in (("l2_bytes", "l2_gbs"), ("onchip_bytes", "onchip_gbs")):
                if key in wk:  # re-swept data that lives in L2 / shared memory: NOT a roofline fraction
                    ent[label] = round(wk[key] / (ms * 1e-3) / 1e9, 2)
        stages[name] = ent
    # dominant KERNEL = the kernel with the largest summed device time per call (several stages
    # are launches of the same kernel)
    kernel_of = {"knn0": "knn_tc3_kernel<4>", "knn1": "knn_tc3_kernel<16>",
                 "knn2": "knn_tc3_kernel<16>",
                 "edge0": "edge_tc_kernel", "edge1": "edge_tc_kernel", "edge2": "edge_tc_kernel",
                 "pq0": "linear_tc_kernel", "pq1": "linear_ts_kernel", "pq2": "linear_ts_kernel",
                 "mlp": "linear_ts_kernel", "base": "linear_ts_kernel", "qkv": "linear_ts_kernel",
                 "att": "attention_tc2_kernel", "fps": "fps_q8_kernel", "cg": "lp_cg_kernel",
                 "dist": "linear_ts_kernel<DIST>", "select": "knn_select_reg_kernel",
                 "proto": "assign_kernel+proto_mean_kernel",
                 "sym": "in_bits/in_rank/in_fill_rank/merge_rows kernels",
                 "sim": "edge_sim_kernel"}
    launches_of = {"mlp": 2, "base": 2}
    groups = {}
    for name, ent in stages.items():
        kname = kernel_of.get(name)
        if kname is None:
            continue
        gk = groups.setdefault(kname, dict(ms=0.0, flops=0.0, bytes=0.0, launches=0,
                                            bound=ent["bound"], stages=[]))
        gk["ms"] += ent["ms_per_call"]
        gk["flops"] += work[name]["flops"] or 0.0
        gk["bytes"] += work[name]["bytes"] or 0.0
        gk["launches"] += launches_of.get(name, 1)
        gk["stages"].append(name)
    top = max(groups, key=lambda k: groups[k]["ms"])
    gt = groups[top]
    step_ms = sum(stage_ms.values())
    if gt["bound"] == "tensor":
        ach = gt["flops"] / (gt["ms"] * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": round(ach, 3), "peak": round(tf32x3_tflops, 1),
                "unit": "TFLOP/s", "frac": round(ach / tf32x3_tflops, 5),
                "frac_of_bf16_peak": round(ach / peaks["bf16_tflops_sustained"], 5),
                "traffic": None,
                "note": "reference-math FLOPs vs the 3xTF32 ceiling (measured TF32 issue rate x SMs "
                        "x clock / 3)"}
    else:
        ach = gt["bytes"] / (gt["ms"] * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": round(ach, 2), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm_gbs"], 5), "traffic": None}
    # DRAM bytes per launch of that kernel from the committed ncu --set full capture (same workload)
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        ent = tr["kernels"].get(top.split("<")[0])
        if ent and tr["episodes_per_call"] == chunk and args.workload == "s3dis_2way_5shot":
            roof["traffic"] = ent["read"] + ent["write"]
            roof["traffic_source"] = "profiles/ncu_traffic.json (ncu dram__bytes_read+write per launch)"
            roof["algorithmic_bytes_per_launch"] = gt["bytes"] / gt["launches"]
    except (OSError, ValueError, KeyError):
        pass
    roof.update(kernel=top, stages=gt["stages"], peak_source=peaks["source"],
                launches_per_call=gt["launches"],
                ms_per_launch=round(gt["ms"] / gt["launches"], 4),
                share_of_step=round(gt["ms"] / step_ms, 4))

    n_total = world * E_step * args.steps
    value = n_total / (total_ms * 1e-3)
    e2e_value = n_total / (e2e_ms * 1e-3)
    h2d = int(sum(t.numel() * t.element_size() for t in (h_sx, h_sy, h_qx, h_qy)))
    d2h = int(h_pred.numel() * 4 + h_loss.numel() * 4)

    # ---- the other legs (all ranks take part) -----------------------------------------------------
    e2e_driver, extra = None, {}
    if not args.no_extra:
        del wss, ws, flush, d_sx, d_sy, d_qx, d_qy
        torch.cuda.empty_cache()
        e2e_driver = driver_leg(model, dev, dist, rank, world, (h_sx, h_sy, h_qx, h_qy, classes),
                                chunk, args.steps, test_classes)
        torch.cuda.empty_cache()
        main_workload = args.workload
        other = "scannet_3way_5shot_ood" if main_workload == "s3dis_2way_5shot" else "s3dis_2way_5shot"
        extra[other] = resident_leg(dev, dist, rank, world, other, E_step, chunk, n_streams,
                                    args.steps, args.warmup)
        set_workload(main_workload)
        torch.cuda.empty_cache()
        # (8+ warm-up steps: with 3 the 4-GPU run still had NCCL's lazy set-up of the two new
        # message sizes and the 3.4 GB workspace allocation inside the timed region — 26.3 ms per
        # step against 17.9 for scripts/bench_train.py alone)
        extra["train_step"] = train_leg(dev, dist, rank, world, args.steps, max(8, args.warmup))

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, dt = cpu_episodes_per_s(args.cpu_episodes, 10_000, threads)
        cpu_base = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": f"{args.cpu_episodes} episodes of the same workload (seeds 10000..), "
                              f"oracle/mpti_oracle.py (CPU restatement of the reference path), "
                              f"torch fp32, {threads} threads, {dt:.1f} s"}

    if rank == 0:
        cnt = counters.cpu().numpy().astype(np.float64)
        iou = cnt[2] / np.maximum(cnt[0] + cnt[1] - cnt[2], 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label,
                       "episodes_per_step_per_gpu": E_step, "episodes_per_call": chunk,
                       "n_points": N_PTS, "weights": "seeded fixture (tests/golden/weights_fixture.pt)",
                       "l2": "512 MiB flush write between timed steps", "sharding": "episodes",
                       "streams": n_streams},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "e2e_driver": e2e_driver,
            "extra": extra,
            "gpu_launches": int(launches),
            "roofline": roof,
            "cpu_baseline": cpu_base,
            "clocks": clocks,
            "stages": stages,
            "cg_iters_mean": cg_iters,
            "mean_iou_synthetic": float(np.mean(iou[1:])),
            "wall_s_timed_region": wall_resident,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
