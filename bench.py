#!/usr/bin/env python
"""Headline benchmark: spatial-feature-memory write+read throughput (frames/s) on B200.

Workload (BASELINE.json configs[1]): 64 synthetic MP3D-shaped episodes x 20 frames advanced in lock step on one
GPU, 480x640 RGB-D, per-pixel C=256 fp32 features (CHW, the reference's image_features layout), 500x500 grid of
0.2 m cells.  One *step* = one pass over the whole workload = 64 x 20 = 1280 frames; per frame-step the hot path
is  back-project+quantise -> read (normalise, fp16, gather, pool x3) -> write (count, scatter-mean, finalise).

  value        frames/s, inputs resident in HBM, CUDA events, max over ranks
  e2e          the same metric through the Python plugin API with HOST (pinned) inputs: H2D of depth, pose and
               features and D2H of the pooled levels inside the timed region
  roofline     dominant kernel (eod_write_mean): algorithmic bytes per launch / mean CUDA-event duration of that
               launch inside the timed region, vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline the oracle port of the same path (torch-CPU restatement of the reference ops) on the host cores
  value_with_fusion   the same timed loop with the tcgen05 projection + fusion of the three levels inside every frame-step
  write_alone  the dominant kernel timed back to back with nothing else on the GPU, right after the timed loop (same power
               state): splits the in-bench roofline loss into concurrency and clock
  roofline_1000  the same workload on the north-star 1000x1000 grid (0.2 m cells), timed the same way
  parity_check   after the timed region: the bench's own batch / inputs, a few frames of 2 episodes against the CPU oracle
                 (oracle/path_check.py) - the oracle is the checker here, never the thing measured
  extras       (not part of `value`) more stages of the path on the same batch: the tcgen05 projection + fusion of the
               three levels alone, and the object regime (detections as mask probabilities + boxes) through step_detections

`--impl reference` times that CPU implementation alone (the reference cannot run as committed: hard-coded
.cuda() and detectron2 imports), on a bounded sample of the same workload per step.

`--dump-outputs DIR` writes, after the timed steps, what the last of them handed its caller: the three pooled levels of its
last frame (level0..2, (E,C,h,w)) and the grid state (sums (E,cells,C), counts (E,cells)), each as DIR/<name>.npy in float32.
The inputs are seeded, so two builds run with the same arguments can be compared output for output; every step starts from
a reset grid, so the dumped arrays do not depend on --steps / --warmup either.  Counts repeat bit for bit; the write adds
fp32 features in a run-dependent order, so sums (and the fp16 levels read from them) may differ in the last bits.

Multi-GPU (torchrun, one process per GPU): episodes are sharded `episode % world == rank`, per-GPU work fixed
(64 episodes each, "weak"), no collective on the hot path; one all_reduce(MAX) for the time and one
all_reduce(SUM) for the frame counters after the loop.
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "memory write+read frames/sec (480x640, C=256)"
UNIT = "frames/s"
H, W, C = 480, 640, 256
MAP_W = MAP_H = 500
CELL = np.float32(0.02 * 10)
N_EPISODES, N_FRAMES = 64, 20
N_PIX = H * W


def _gen_episode(args):
    seed, n_frames, map_w, map_h, cell = args
    episodes = importlib.import_module("embodied-object-detection_b200.episodes")
    ep = episodes.make_episode(seed, n_frames, H, W, map_w, map_h, float(cell))
    return ep.depth, ep.xyzhe, ep.map_world_shift


def make_inputs(episode_ids, n_frames=N_FRAMES, map_w=MAP_W, map_h=MAP_H, cell=CELL):
    """Host-side synthetic episodes (seed 1234 + episode id), generated in parallel on the host cores."""
    jobs = [(1234 + int(e), n_frames, map_w, map_h, cell) for e in episode_ids]
    workers = max(1, min(len(jobs), (os.cpu_count() or 2) - 1, 32))
    if workers > 1:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(workers) as pool:
            out = pool.map(_gen_episode, jobs)
    else:
        out = [_gen_episode(j) for j in jobs]
    depth = np.stack([o[0] for o in out])            # (E, T, H, W)
    xyzhe = np.stack([o[1] for o in out])            # (E, T, 5)
    shift = np.stack([o[2] for o in out])            # (E, 3)
    return depth, xyzhe, shift


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(index: int):
    """Pin this rank's CPU threads - and with them the first-touch placement of its pinned staging buffers - to the NUMA node
    its GPU hangs off.  Unbound, the 8 ranks of a box stream most of their H2D traffic across the socket interconnect and the
    e2e arm is host-memory bound at less than half of 8 x PCIe.  Best effort: returns the node, or None when sysfs says nothing."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)], capture_output=True,
                             text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        dom, rest = bus.split(":", 1)
        node = int(open(f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(E: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one write-kernel launch, from the committed ncu pass
    (profiles/write_kernel_traffic.json, written by profiles/summarize.py); None if it was taken at another batch size."""
    p = os.path.join(ROOT, "profiles", "write_kernel_traffic.json")
    try:
        d = json.load(open(p))
        return float(d["traffic_bytes_per_launch"]) if int(d["episodes_per_launch"]) == E else None
    except Exception:
        return None


def pcie_info(gpu: int):
    """PCIe link of this rank's GPU (the e2e arm is bounded by it) and the box's topology matrix, for the record."""
    info = {}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(gpu), "--query-gpu=pci.bus_id,pcie.link.gen.current,pcie.link.width.current,pcie.link.gen.max",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=10).stdout.strip()
        info["link"] = q
        topo = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=10).stdout
        info["topo"] = [l[:200] for l in topo.splitlines() if l.startswith("GPU")][:9]
    except Exception as exc:
        info["error"] = repr(exc)[:100]
    return info


DUMP_SAMPLE = 1 << 21          # elements per dumped array at most: 5 arrays x 8 MB in float32


def dump_outputs(out_dir: str, arrays: dict, seed: int = 0) -> None:
    """Write each tensor as out_dir/<name>.npy in float32.  One larger than DUMP_SAMPLE elements is represented by its elements at
    DUMP_SAMPLE distinct flat positions (row-major over its logical shape, ascending) drawn by numpy's default_rng(seed): the
    positions depend on the shape alone, so they are the same in every run."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        n = t.numel()
        if n > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(seed).choice(n, DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def write_launch_bytes(E: int, touched_per_launch: float, c: int = C) -> float:
    """Algorithmic bytes of ONE eod_write_mean launch over E episodes (DESIGN.md 'Roofline accounting'):
    features read once + index plane + touched grid rows read-modify-written + per-cell sample counts."""
    return E * (N_PIX * c * 4 + N_PIX * 4) + touched_per_launch * (c * 4 * 2 + 4)


def frame_bytes(visible_per_frame: float, c: int = C) -> float:
    """Whole-path algorithmic bytes per frame (SURVEY 8d / BASELINE.md 5), M = V (every pixel sampled)."""
    v = visible_per_frame
    write = N_PIX * 4 + 64 + N_PIX * c * 4 + v * (c * 4 * 2 + 8)
    read = N_PIX * 4 + v * (c * 4 + 4) + 6300 * c * 2
    return write + read


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the path (reference ops restated on the CPU)
# ---------------------------------------------------------------------------------------------------------
def cpu_frames(depth, xyzhe, shift, n_frames, feats):
    """Run n_frames of ONE episode through the CPU port: C back-projection, torch read chain, sparse-equivalent
    (index_add_) write of the dense per-pixel features.  Returns seconds."""
    import oracle
    from oracle import reference_ops as R
    intr = R.intrinsics(W, H, math.radians(67.5))
    T = R.transform3d(torch.from_numpy(xyzhe)).numpy()
    sums = torch.zeros(MAP_W * MAP_H, C)
    counts = torch.zeros(MAP_W * MAP_H)
    observed = torch.ones(H, W, dtype=torch.bool)
    t0 = time.perf_counter()
    for t in range(n_frames):
        idx = oracle.backproject_quantize(depth[t], T[t], intr, np.zeros(3, np.float32), shift, CELL, MAP_W, MAP_H, 0, 0.5, want=("idx",))["idx"]
        proj = torch.from_numpy(idx).long()
        R.read_frame(sums, counts, proj)
        sums, counts = R.write_mean_frame(sums, counts, feats[t % len(feats)], observed, proj, stride=1)
    return time.perf_counter() - t0


def run_cpu_sample(n_frames: int):
    torch.set_num_threads(os.cpu_count() or 1)
    depth, xyzhe, shift = make_inputs([0], n_frames=max(n_frames, 2))
    g = torch.Generator().manual_seed(0)
    feats = [torch.randn(1, C, H, W, generator=g) for _ in range(2)]
    cpu_frames(depth[0], xyzhe[0], shift[0], 1, feats)          # warm-up
    sec = cpu_frames(depth[0], xyzhe[0], shift[0], n_frames, feats)
    return n_frames / sec, sec


def main_reference(args, rank, world):
    if rank != 0:
        return
    n_frames = 4
    torch.set_num_threads(os.cpu_count() or 1)
    depth, xyzhe, shift = make_inputs([0], n_frames=n_frames)
    g = torch.Generator().manual_seed(0)
    feats = [torch.randn(1, C, H, W, generator=g) for _ in range(2)]
    for _ in range(max(args.warmup, 1)):
        cpu_frames(depth[0], xyzhe[0], shift[0], 1, feats)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_frames(depth[0], xyzhe[0], shift[0], n_frames, feats)
    sec = time.perf_counter() - t0
    fps = args.steps * n_frames / sec
    sample = f"{n_frames} frames of episode 0 per step (of the 64x20-frame workload); sparse-equivalent index_add_ write"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world),
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(world):
    return {"workload": f"configs[1]: {N_EPISODES} episodes x {N_FRAMES} frames per GPU, 480x640 RGB-D, dense per-pixel C=256 fp32 "
                        f"features (CHW), 500x500 grid @0.2 m, write=per-cell mean (stride 1) + visibility counts, "
                        f"read=normalise+fp16+gather+pool to 60x80/30x40/15x20",
            "episodes_per_gpu": N_EPISODES, "frames_per_episode": N_FRAMES, "grid": [MAP_W, MAP_H], "channels": C,
            "parallelism": f"episode-sharded x{world}, no hot-path collective",
            "l2_policy": "inputs larger than L2 (20.1 GB of features per frame-step, two alternating slabs)"}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def timed_steps(batch, n_steps, one_step, barrier, sharding, dev):
    """K steps bracketed by barrier + synchronize, CUDA events on the caller's stream, max over ranks -> total ms."""
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(n_steps):
        one_step()
    ev1.record()
    barrier()
    return sharding.max_over_ranks(ev0.elapsed_time(ev1), dev)


def run_parity_check(batch, depth, pose, shifts, intr, cell, slabs, depth_h, T_h, shift_h, my_eps, n_frames=3, checked=(0, 37)):
    """Outside the timed region: the bench's own EpisodeBatch (E=64, pipeline=True) and its own resident inputs, n_frames
    frames, two episodes against the CPU oracle - synchronised pass (levels bit-exact on the downloaded state), then the same
    frames back to back as the timed loop enqueues them (final state of all 64 episodes must agree)."""
    from oracle import path_check
    host = {e: dict(depth=depth_h[e], T=T_h[e], shift=shift_h[e]) for e in checked}
    frames = [dict(depth=depth[t], pose=pose[t], feat=slabs[t & 1]) for t in range(n_frames)]
    t0 = time.perf_counter()
    res = path_check.check_dense_steps(batch, frames, shifts, intr, cell, host, synced=True)
    state = (batch.sums[list(checked)].clone(), batch.counts.clone())
    res2 = path_check.check_dense_steps(batch, frames, shifts, intr, cell, host, synced=False)
    all_counts_equal = bool(torch.equal(batch.counts, state[1]))
    scale = float(state[0].abs().max())
    sums_drift = float((batch.sums[list(checked)] - state[0]).abs().max()) / max(scale, 1e-30)
    out = {"checked_episodes": [int(my_eps[e]) for e in checked], "frames": n_frames, "grid": [batch.map_w, batch.map_h],
           "synced": {k: v for k, v in path_check.summary(res).items() if k not in ("episodes", "frames", "synced")},
           "back_to_back": {k: v for k, v in path_check.summary(res2).items() if k not in ("episodes", "frames", "synced")},
           "back_to_back_counts_equal_all_episodes": all_counts_equal, "back_to_back_sums_drift_over_scale": sums_drift,
           "tolerance": {"indices/counts/levels": "bit-exact", "sums": "max|a-b| <= 1e-5 * max|ref|"},
           "seconds": round(time.perf_counter() - t0, 2)}
    out["ok"] = bool(res["ok"] and res2["ok"] and all_counts_equal and sums_drift <= 1e-6)
    return out


def main_gpu(args, rank, local_rank, world):
    eod = importlib.import_module("embodied-object-detection_b200")
    sharding = eod.sharding
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    eod._lib.lib()                                                   # fail loudly when the extension is missing
    numa_node = None if args.no_numa else bind_to_gpu_numa_node(local_rank)

    E = N_EPISODES
    my_eps = [rank + world * i for i in range(E)]                    # weak scaling: 64 episodes per GPU
    depth_h, xyzhe_h, shift_h = make_inputs(my_eps)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    T = eod.transform3d(torch.from_numpy(xyzhe_h.reshape(-1, 5))).reshape(E, N_FRAMES, 4, 4)
    pose = T[:, :, :3, :].reshape(E, N_FRAMES, 12).permute(1, 0, 2).contiguous().to(dev)       # (T, E, 12)
    depth = torch.from_numpy(depth_h).permute(1, 0, 2, 3).contiguous().to(dev)                 # (T, E, H, W)
    shifts = torch.from_numpy(np.concatenate([np.zeros_like(shift_h), shift_h], 1)).to(dev)   # (E, 6)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    slabs = [torch.randn((E, C, H, W), device=dev, generator=gen) for _ in range(2)]          # 2 x 20.1 GB
    # inputs are resident and static for the whole run, which is what pipeline=True asks of the caller
    batch = eod.EpisodeBatch(E, MAP_W, MAP_H, C, H, W, dev, variant=args.write_variant, pipeline=not args.no_pipeline)
    last_levels = []                                                 # what step() returned for the last frame of the last step

    def one_step():
        batch.reset()
        for t in range(N_FRAMES):
            levels = batch.step(depth[t], pose[t], shifts, intr, float(CELL), slabs[t & 1])
        batch.join()                                                 # the timing events sit on the caller's stream
        last_levels[:] = levels

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()                                                  # samples cover warm-up + timed steps (all under load)
    for _ in range(args.warmup):
        one_step()
    barrier()
    launches0 = eod.ops.launch_count
    batch.profile(True)
    ms_total = timed_steps(batch, args.steps, one_step, barrier, sharding, dev)
    clocks = sampler.stop()
    launches = eod.ops.launch_count - launches0
    stage_ms = batch.stage_ms()
    batch.profile(False)
    visible_last_step = float(batch.counts.sum().item())            # +1 per visible cell per frame since the reset
    if args.dump_outputs and rank == 0:                              # before the extras below reuse the batch
        dump_outputs(args.dump_outputs, {**{f"level{k}": l for k, l in enumerate(last_levels)}, "sums": batch.sums, "counts": batch.counts})
    totals = sharding.gather_counters({"frames": float(args.steps * E * N_FRAMES), "visible": visible_last_step}, dev)

    ms_per_step = ms_total / args.steps
    value = totals["frames"] / (ms_total / 1e3)
    vis_per_frame = visible_last_step / (E * N_FRAMES)
    peak, peak_src = measured_peak_gbs()
    wbytes = write_launch_bytes(E, vis_per_frame * E)
    achieved = wbytes / (stage_ms["write"] * 1e-3) / 1e9 if stage_ms.get("write") else None
    path_gbs = frame_bytes(vis_per_frame) * (value / world) / 1e9

    # ---- the dominant kernel alone, back to back, in the power state the timed loop left behind ----
    write_alone = None
    if not args.no_extras:
        batch.join()
        batch.project(depth[0], pose[0], shifts, intr, float(CELL))
        batch._count(None)
        n_alone = 20
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        batch._write(slabs[1], None)
        a.record()
        for i in range(n_alone):
            batch._write(slabs[i & 1], None)
        b.record()
        torch.cuda.synchronize()
        batch._finalize()
        ms_alone = a.elapsed_time(b) / n_alone
        write_alone = {"launch_ms": ms_alone, "GBps": wbytes / ms_alone / 1e6, "frac": wbytes / ms_alone / 1e6 / peak, "launches": n_alone,
                       "note": "same kernel, same batch, nothing else resident: in-bench loss = overlap with read/count/expand/project of the "
                               "neighbouring frames + SM clock under the power cap"}
        batch.reset()

    # ---- the same loop with projection + fusion of the three levels in every frame-step (north-star subsystem 4) ----
    with_fusion = None
    if not args.no_extras:
        g = torch.Generator(device=dev).manual_seed(5 + rank)
        N_OUT = 256
        ws = [eod.ops.project_split_weights(torch.randn((N_OUT, C), device=dev, generator=g) / C ** 0.5) for _ in range(3)]
        bias = [torch.randn((N_OUT,), device=dev, generator=g) for _ in range(3)]
        res = [torch.randn((E, N_OUT, H >> s_, W >> s_), device=dev, generator=g) for s_ in (3, 4, 5)]   # the FPN's p3-p5 (timm.py:170-189)
        outs = [torch.empty_like(r) for r in res]

        def one_step_fused():
            batch.reset()
            for t in range(N_FRAMES):
                levels = batch.step(depth[t], pose[t], shifts, intr, float(CELL), slabs[t & 1])
                eod.ops.project_fuse_levels(levels, ws, bias, res, 5.0, 0, outs)
            batch.join()

        one_step_fused()
        ms_f = timed_steps(batch, args.steps, one_step_fused, barrier, sharding, dev)
        with_fusion = {"value": world * args.steps * E * N_FRAMES / (ms_f / 1e3), "unit": UNIT, "ms_per_step": ms_f / args.steps,
                       "stages": "back-project -> read -> project+fuse (tcgen05, MAP_FEAT_FUSION sum, weight 5) -> write, every frame-step",
                       "extra_bytes_per_frame": int(6300 * (C * 2 + 2 * N_OUT * 4))}
        del res, outs

    parity = None
    if rank == 0 and not args.no_parity:
        try:
            parity = run_parity_check(batch, depth, pose, shifts, intr, float(CELL), slabs, depth_h, T.numpy(), shift_h, my_eps)
        except Exception as exc:                                     # a failed check must be visible, never silently dropped
            parity = {"ok": False, "error": repr(exc)[:300]}

    extras = run_extras(eod, batch, dev, depth, pose, shifts, intr, slabs) if (rank == 0 and not args.no_extras) else None
    if world > 1:
        torch.distributed.barrier()
    # ---- e2e through the plugin API with host buffers (rank-local, then max over ranks) ----
    e2e = None if args.no_e2e else run_e2e(eod, batch, dev, depth_h, pose.cpu(), shifts, intr, args, world, sharding, slabs)
    e2e_variants = None
    if not args.no_e2e and not args.no_extras:
        try:
            e2e_variants = run_e2e_variants(eod, batch, dev, depth_h, pose.cpu(), shifts, intr, args, world, sharding, slabs)
        except Exception as exc:
            e2e_variants = {"error": repr(exc)[:300]}

    # ---- the north-star grid: 1000 x 1000 cells (0.2 m), same episodes, same timing method ----
    roofline_1000 = None
    if not args.no_extras:
        try:
            del batch
            torch.cuda.empty_cache()
            roofline_1000 = run_grid_1000(eod, dev, depth, pose, shift_h, intr, slabs, depth_h, T.numpy(), my_eps, args, barrier, sharding,
                                          world, rank, peak)
        except Exception as exc:
            roofline_1000 = {"error": repr(exc)[:300]}

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(world), "clocks": clocks, "gpu_launches": int(launches),
        "e2e": e2e, "e2e_variants": e2e_variants, "value_with_fusion": with_fusion, "write_alone": write_alone, "parity_check": parity,
        "roofline_1000": roofline_1000, "extras": extras, "host": {"numa_node": numa_node, "cpus": os.cpu_count(), "pcie": pcie_info(local_rank)},
        "roofline": {"bound": "hbm", "kernel": "write_mean_chw_tma_kernel<256>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "frac_of_nominal_8TBs": (achieved / 8000.0) if achieved else None,
                     "traffic": measured_traffic(E), "peak_source": peak_src, "bytes_per_launch": wbytes, "launch_ms": stage_ms.get("write"),
                     "stage_ms": stage_ms, "visible_cells_per_frame": vis_per_frame,
                     "whole_path": {"bytes_per_frame": frame_bytes(vis_per_frame), "achieved_gbs_per_gpu": path_gbs,
                                    "frac": path_gbs / peak}},
    }
    if rank == 0:
        if world == 1 and not args.no_cpu:
            fps, sec = run_cpu_sample(args.cpu_frames)
            out["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": f"{args.cpu_frames} frames of episode 0 ({sec:.1f} s): C back-projection + torch-CPU read chain "
                                             f"+ sparse-equivalent (index_add_) write; the literal one-hot matmul of the reference needs "
                                             f"{N_PIX * MAP_W * MAP_H / 1e9:.0f} GB at stride 1"}
        print(json.dumps(out))


def main_cfg5(args, rank, local_rank, world):
    """BASELINE configs[4]: 512 synthetic episodes x 100 frames, 512-d dense features, 1000x1000 grid, sharded by episode over
    the ranks (STRONG scaling: the job is fixed).  Each rank keeps --slots grids resident and streams its share of the
    episodes through them in waves (EpisodeRunner); no collective on the hot path, one all_reduce of counters at the end."""
    eod = importlib.import_module("embodied-object-detection_b200")
    sharding = eod.sharding
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    eod._lib.lib()
    n_ep, T_, Cc, mw, mh, R = args.cfg5_episodes, args.cfg5_frames, 512, 1000, 1000, args.slots
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    provider = eod.runner.PooledSyntheticProvider(n_ep, T_, Cc, R, dev, H, W, mw, mh, float(CELL), pool=64)
    runner = eod.EpisodeRunner(provider, mw, mh, Cc, R, height=H, width=W, device=dev, test_type="episodic", rank=rank, world=world,
                               intr=intr, cell=float(CELL))

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    runner.run(max_steps=max(3, args.warmup) * 4)                      # warm-up: a dozen frame-steps of the first wave
    barrier()
    runner.batch.profile(True)
    frames = steps_run = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        st = runner.run()
        frames += st["frames"]
        steps_run += st["steps"]
    ev1.record()
    barrier()
    clocks = sampler.stop()
    ms_total = sharding.max_over_ranks(ev0.elapsed_time(ev1), dev)
    stage_ms = runner.batch.stage_ms()
    runner.batch.profile(False)
    totals = sharding.gather_counters({"frames": float(frames), "steps": float(steps_run)}, dev)
    value = totals["frames"] / (ms_total / 1e3)
    # size-independent check at the full size: the first slot's first episode, replayed alone through a one-episode batch,
    # must land in the same state as inside the lock-step batch (counts exact, sums to reduction-order noise)
    check = None
    if rank == 0 and not args.no_parity:
        n_chk = 4
        runner.run(max_steps=n_chk)
        torch.cuda.synchronize()
        e0 = runner.schedule.streams[0][0]
        solo = eod.EpisodeBatch(1, mw, mh, Cc, H, W, dev)
        traj = e0 % provider.pool
        for t in range(n_chk):
            solo.step(provider.depth[traj, t][None], provider.pose[traj, t][None], provider.shifts[traj][None], intr, float(CELL),
                      provider.feat[(provider._k - n_chk + t) & 1][0:1].contiguous())
        torch.cuda.synchronize()
        scale = float(solo.sums.abs().max())
        check = {"frames": n_chk, "counts_equal": bool(torch.equal(solo.counts[0], runner.batch.counts[0])),
                 "sums_max_diff_over_scale": float((solo.sums[0] - runner.batch.sums[0]).abs().max()) / max(scale, 1e-30),
                 "norm16_equal_up_to_1ulp": bool(((solo.norm16[0].view(torch.int16).int() - runner.batch.norm16[0].view(torch.int16).int()).abs() <= 1).all())}
        check["ok"] = check["counts_equal"] and check["sums_max_diff_over_scale"] <= 1e-6
        del solo
    peak, peak_src = measured_peak_gbs()
    wbytes = write_launch_bytes(R, 0.0, Cc)
    achieved = wbytes / stage_ms["write"] / 1e6 if stage_ms.get("write") else None
    out = {"metric": "memory write+read frames/sec (480x640, C=512)", "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"configs[4]: {n_ep} episodes x {T_} frames, 480x640 RGB-D, dense per-pixel C=512 fp32 features (CHW), 1000x1000 grid "
                                  f"@0.2 m, sharded by episode over {world} GPU(s), {R} resident grids per GPU refilled in waves (EpisodeRunner, "
                                  f"TEST_TYPE episodic); 64 distinct ray-cast trajectories replayed by the {n_ep} episodes",
                      "episodes": n_ep, "frames_per_episode": T_, "grid": [mw, mh], "channels": Cc, "slots_per_gpu": R,
                      "parallelism": f"episode-sharded x{world}, no hot-path collective",
                      "l2_policy": f"inputs larger than L2 ({R * Cc * N_PIX * 4 / 1e9:.1f} GB of features per frame-step, two alternating slabs)"},
           "clocks": clocks, "frames": totals["frames"], "frame_steps_per_rank": int(totals["steps"] / world / max(1, args.steps)),
           "roofline": {"bound": "hbm", "kernel": "write_mean_chw_tma_kernel<512>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak if achieved else None, "peak_source": peak_src, "bytes_per_launch": wbytes,
                        "launch_ms": stage_ms.get("write"), "stage_ms": stage_ms, "note": "feature + index bytes of a full wave (touched grid rows not counted)"},
           "self_check": check}
    if rank == 0:
        print(json.dumps(out))


def run_grid_1000(eod, dev, depth, pose, shift_h, intr, slabs, depth_h, T_h, my_eps, args, barrier, sharding, world, rank, peak):
    """BASELINE north-star target: 480x640, C=256 on a 1000x1000 grid.  Same 64 episodes per GPU (the depth maps are replayed
    into the larger map: only map_world_shift changes), 0.2 m cells as everywhere in the reference's implicit memory
    (SMNet/build_memory_data.py:136), same pipelined loop, CUDA events, stage events for the write launch."""
    E, mw, mh = N_EPISODES, 1000, 1000
    shift_1k = shift_h.copy()
    shift_1k[:, 0] -= np.float32((mw - MAP_W) * float(CELL) / 2)
    shift_1k[:, 2] -= np.float32((mh - MAP_H) * float(CELL) / 2)
    shifts = torch.from_numpy(np.concatenate([np.zeros_like(shift_1k), shift_1k], 1)).to(dev)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, dev, pipeline=not args.no_pipeline)

    def one_step():
        batch.reset()
        for t in range(N_FRAMES):
            batch.step(depth[t], pose[t], shifts, intr, float(CELL), slabs[t & 1])
        batch.join()

    one_step()
    one_step()
    steps = max(2, min(args.steps, 5))
    batch.profile(True)
    ms = timed_steps(batch, steps, one_step, barrier, sharding, dev)
    stage_ms = batch.stage_ms()
    batch.profile(False)
    vis = float(batch.counts.sum().item()) / (E * N_FRAMES)
    wbytes = write_launch_bytes(E, vis * E)
    value = world * steps * E * N_FRAMES / (ms / 1e3)
    achieved = wbytes / stage_ms["write"] / 1e6
    out = {"grid": [mw, mh], "cell_m": float(CELL), "channels": C, "episodes_per_gpu": E, "value": value, "unit": UNIT, "steps": steps,
           "ms_per_step": ms / steps, "kernel": "write_mean_chw_tma_kernel<256>", "achieved": achieved, "peak": peak, "frac": achieved / peak,
           "bytes_per_launch": wbytes, "launch_ms": stage_ms["write"], "stage_ms": stage_ms, "visible_cells_per_frame": vis,
           "whole_path_frac": frame_bytes(vis) * (value / world) / 1e9 / peak,
           "resident_bytes": int(batch.sums.numel() * 4 + batch.norm16.numel() * 2 + batch.counts.numel() * 4)}
    if rank == 0 and not args.no_parity:
        try:
            out["parity_check"] = run_parity_check(batch, depth, pose, shifts, intr, float(CELL), slabs, depth_h, T_h, shift_1k, my_eps, n_frames=2)
        except Exception as exc:
            out["parity_check"] = {"ok": False, "error": repr(exc)[:300]}
    return out


def run_extras(eod, batch, dev, depth, pose, shifts, intr, slabs=None):
    """Two more stages of the same path, timed on the bench batch after the headline loop (CUDA events, resident inputs; not part
    of `value`): the tensor-core projection + fusion of the three read levels (SURVEY 8a A13) and the reference's live object
    regime (kept detections as 28x28 mask probabilities + boxes; mask pasting folded into the write).  Best effort."""
    out = {}
    try:
        E = batch.E
        ops = eod.ops
        g = torch.Generator(device=dev).manual_seed(5)
        levels = [l.permute(0, 3, 1, 2) for l in batch.levels]                        # the last frame's pooled levels, channels-last memory
        N = 256
        ws = [ops.project_split_weights(torch.randn((N, C), device=dev, generator=g) / C ** 0.5) for _ in range(3)]
        bias = [torch.randn((N,), device=dev, generator=g) for _ in range(3)]
        res = [torch.randn((E, N, l.shape[2], l.shape[3]), device=dev, generator=g) for l in levels]
        outs = [torch.empty_like(r) for r in res]
        for _ in range(3):
            ops.project_fuse_levels(levels, ws, bias, res, 5.0, 0, outs)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            ops.project_fuse_levels(levels, ws, bias, res, 5.0, 0, outs)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 10
        nbytes = sum(l.numel() * 2 for l in levels) + 2 * sum(r.numel() * 4 for r in res)
        out["project_fuse"] = {"ms_per_frame_step": ms, "GBps": nbytes / ms / 1e6, "kernel": "project_fuse_persistent_kernel (tcgen05)",
                               "shape": f"E={E}, K={C} -> N={N}, levels 60x80/30x40/15x20"}
        del res, outs
        rng = np.random.default_rng(0)
        Kmax = 16
        bf = np.zeros((E, Kmax, C), np.float32); pr = np.zeros((E, Kmax, 28, 28), np.float32); bx = np.zeros((E, Kmax, 4), np.float32)
        n = np.zeros(E, np.int32)
        for e in range(E):
            f, p_, b_ = eod.episodes.make_mask_head_detections(rng, H, W, C, (4, Kmax), 28)
            n[e] = f.shape[0]; bf[e, : n[e]], pr[e, : n[e]], bx[e, : n[e]] = f, p_, b_
        det = [torch.from_numpy(x).to(dev) for x in (bf, pr, bx, n)]
        batch.join()
        for t in range(3):
            batch.step_detections(depth[t], pose[t], shifts, intr, float(CELL), *det)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(N_FRAMES):
            batch.step_detections(depth[t], pose[t], shifts, intr, float(CELL), *det)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / N_FRAMES
        out["object_regime"] = {"ms_per_frame_step": ms, "frames_per_s": E / ms * 1e3,
                                "shape": f"E={E}, C={C}, <= {Kmax} detections per frame, 28x28 mask probabilities + boxes, every 8th observed pixel"}
        if slabs is not None:
            # the same dense frame loop with the features taken as channels-last fp32 (EOD_LAYOUT_HWC): the resident random slabs are
            # simply read as (E,H,W,C) - what a backbone running in torch.channels_last hands over; one step = N_FRAMES frame-steps
            layout0, pipe0 = batch.layout, batch.pipeline
            try:
                batch.join()
                batch.layout, batch.pipeline = eod._lib.LAYOUT_HWC, True
                hwc = [s_.view(E, H, W, C) for s_ in slabs]
                batch.reset()
                for t in range(3):
                    batch.step(depth[t], pose[t], shifts, intr, float(CELL), hwc[t & 1])
                batch.join()
                batch.profile(True)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for t in range(N_FRAMES):
                    batch.step(depth[t], pose[t], shifts, intr, float(CELL), hwc[t & 1])
                batch.join()
                b.record()
                torch.cuda.synchronize()
                st = batch.stage_ms()
                batch.profile(False)
                ms = a.elapsed_time(b) / N_FRAMES
                peak, _ = measured_peak_gbs()
                fb = E * (N_PIX * C * 4 + N_PIX * 4)
                out["dense_hwc_f32"] = {"ms_per_frame_step": ms, "frames_per_s": E / ms * 1e3, "write_launch_ms": st.get("write"),
                                        "write_GBps": fb / st["write"] / 1e6 if st.get("write") else None,
                                        "write_frac_of_peak": fb / st["write"] / 1e6 / peak if st.get("write") else None,
                                        "kernel": "write_mean_hwc_kernel<256, f32>", "note": "same loop as the headline, features read channels-last"}
            finally:
                batch.join()
                batch.layout, batch.pipeline = layout0, pipe0
                batch.reset()
    except Exception as exc:                                                          # never lose the headline line to an extra
        out["error"] = repr(exc)[:200]
    return out


def run_e2e(eod, batch, dev, depth_h, pose_h, shifts, intr, args, world, sharding, slabs):
    """frames/s through EpisodeBatch.step with HOST inputs: per frame-step, H2D of depth (E,H,W), pose (E,12) and
    features (E,C,H,W) from pinned memory on a copy stream (double-buffered against compute), and D2H of the three
    pooled fp16 levels.  The feature H2D (20.1 GB per frame-step) makes this PCIe-bound by construction."""
    E = batch.E
    batch.join()
    batch.pipeline = False                                           # host-fed inputs: every step is ordered on the caller's stream
    n_slots = 4                                                      # pinned staging: 4 episode-frames of features (1.26 GB)
    g = torch.Generator().manual_seed(7)
    pin_feat = torch.randn((n_slots, C, H, W), generator=g).pin_memory()
    pin_depth = torch.from_numpy(depth_h).permute(1, 0, 2, 3).contiguous().pin_memory()      # (T, E, H, W)
    pin_pose = pose_h.contiguous().pin_memory()
    dev_feat = slabs                                                 # reuse the two resident 20.1 GB slabs as H2D targets
    dev_depth = [torch.empty((E, H, W), device=dev) for _ in range(2)]
    dev_pose = [torch.empty((E, 12), device=dev) for _ in range(2)]
    host_levels = [torch.empty(l.shape, dtype=l.dtype).pin_memory() for l in batch.levels]
    copy_s = torch.cuda.Stream(device=dev)
    comp_s = torch.cuda.current_stream(dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    h2d = E * (C * H * W * 4 + H * W * 4 + 12 * 4)
    d2h = sum(l.numel() * 2 for l in batch.levels)
    frames_per_step = E * args.e2e_frames

    def upload(t, buf):
        with torch.cuda.stream(copy_s):
            copy_s.wait_event(freed[buf])
            for e in range(E):
                dev_feat[buf][e].copy_(pin_feat[(e + t) % n_slots], non_blocking=True)
            dev_depth[buf].copy_(pin_depth[t % N_FRAMES], non_blocking=True)
            dev_pose[buf].copy_(pin_pose[t % N_FRAMES], non_blocking=True)
            ready[buf].record(copy_s)

    def one_step():
        batch.reset()
        upload(0, 0)
        for t in range(args.e2e_frames):
            b = t & 1
            if t + 1 < args.e2e_frames:
                upload(t + 1, b ^ 1)
            comp_s.wait_event(ready[b])
            levels = batch.step(dev_depth[b], dev_pose[b], shifts, intr, float(CELL), dev_feat[b])
            for hl, l in zip(host_levels, batch.levels):
                hl.copy_(l, non_blocking=True)
            freed[b].record(comp_s)
        torch.cuda.synchronize()
        return float(host_levels[2].float().abs().sum())             # device->host result actually read on the host

    for f in freed:
        f.record(comp_s)
    one_step()                                                        # warm-up
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        one_step()
    sec = time.perf_counter() - t0
    sec = sharding.max_over_ranks(sec, dev)
    return {"value": world * frames_per_step * args.e2e_steps / sec, "unit": UNIT,
            "h2d_bytes_per_step": int(h2d * args.e2e_frames), "d2h_bytes_per_step": int(d2h * args.e2e_frames),
            "frames_per_step": frames_per_step, "steps": args.e2e_steps,
            "h2d_GBps_per_rank": h2d * args.e2e_frames * args.e2e_steps / sec / 1e9,
            "note": "bounded: e2e step = %d frame-steps of the 64-episode batch; PCIe-bound (features cross the bus, which the "
                    "reference never does: its features are produced on the device)" % args.e2e_frames}


def h2d_ceiling(dev, world, sharding, nbytes=1 << 30, reps=6):
    """What this rank's PCIe link + host memory deliver while EVERY rank copies at once: plain cudaMemcpyAsync of a pinned
    1 GiB buffer, all ranks started together.  The dense e2e arm cannot beat this number; it explains N-GPU e2e scaling."""
    pin = torch.empty((nbytes,), dtype=torch.uint8).pin_memory()
    dst = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    dst.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        dst.copy_(pin, non_blocking=True)
    torch.cuda.synchronize()
    sec = sharding.max_over_ranks(time.perf_counter() - t0, dev)
    return nbytes * reps / sec / 1e9


def run_e2e_variants(eod, batch, dev, depth_h, pose_h, shifts, intr, args, world, sharding, slabs):
    """Two more end-to-end arms through the public API with HOST inputs (wall clock, max over ranks), plus the H2D ceiling:
      dense_bf16_hwc  features uploaded as channels-last bf16 (EOD_LAYOUT_HWC_BF16: what a bf16 backbone emits, BASELINE
                      configs[3]); the arithmetic stays fp32 after an exact widening - half the bytes on the bus;
      object_regime   the reference's live regime through step_detections: per frame-step depth, pose, <=16 kept detections
                      ((K,C) features, 28x28 mask probabilities, boxes) go up, the coarsest pooled level comes back."""
    E = batch.E
    out = {"h2d_ceiling_GBps_per_rank_all_ranks_busy": h2d_ceiling(dev, world, sharding)}
    comp_s = torch.cuda.current_stream(dev)
    copy_s = torch.cuda.Stream(device=dev)
    n_fr = args.e2e_frames
    pin_depth = torch.from_numpy(depth_h).permute(1, 0, 2, 3).contiguous().pin_memory()      # (T, E, H, W)
    pin_pose = pose_h.contiguous().pin_memory()
    NB = 3                                               # input staging depth of the object-regime arms (the dense arms use two)
    dev_depth = [torch.empty((E, H, W), device=dev) for _ in range(2)]
    dev_pose = [torch.empty((E, 12), device=dev) for _ in range(NB)]
    ready = [torch.cuda.Event() for _ in range(NB)]
    freed = [torch.cuda.Event() for _ in range(NB)]

    def run(upload_extra, step_fn, d2h_fn, n_frames, depth_src=None, depth_dst=None):
        depth_src = pin_depth if depth_src is None else depth_src
        depth_dst = dev_depth if depth_dst is None else depth_dst

        nb = len(depth_dst)                              # 2: double buffered; 3: the upload of frame t+1 waits for frame t-2, not t-1
        fin = [None] * nb                                # finalize event of the last step that read buffer b (pipelined steps outlive the call)

        def upload(t, b):
            with torch.cuda.stream(copy_s):
                copy_s.wait_event(freed[b])
                if fin[b] is not None:
                    copy_s.wait_event(fin[b])
                depth_dst[b].copy_(depth_src[t % N_FRAMES], non_blocking=True)
                dev_pose[b].copy_(pin_pose[t % N_FRAMES], non_blocking=True)
                upload_extra(t, b)
                ready[b].record(copy_s)

        def one():
            batch.reset()
            upload(0, 0)
            for t in range(n_frames):
                b = t % nb
                if t + 1 < n_frames:
                    upload(t + 1, (t + 1) % nb)
                comp_s.wait_event(ready[b])
                step_fn(b)
                fin[b] = batch._e_fin
                d2h_fn()
                freed[b].record(comp_s)
            batch.join()
            torch.cuda.synchronize()

        for f in freed:
            f.record(comp_s)
        one()
        if world > 1:
            torch.distributed.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            one()
        return sharding.max_over_ranks(time.perf_counter() - t0, dev)

    batch.join()
    batch.pipeline = False
    # ---- dense, bf16 channels-last upload ----
    g = torch.Generator().manual_seed(11)
    n_slots = 4
    pin_feat = torch.randn((n_slots, H, W, C), generator=g).to(torch.bfloat16).pin_memory()
    dev_feat = [torch.empty((E, H, W, C), dtype=torch.bfloat16, device=dev) for _ in range(2)]
    host_levels = [torch.empty(l.shape, dtype=l.dtype).pin_memory() for l in batch.levels]
    layout0 = batch.layout
    batch.layout = eod._lib.LAYOUT_HWC_BF16

    def up_feat(t, b):
        for e in range(E):
            dev_feat[b][e].copy_(pin_feat[(e + t) % n_slots], non_blocking=True)

    def d2h_levels():
        for hl, l in zip(host_levels, batch.levels):
            hl.copy_(l, non_blocking=True)

    sec = run(up_feat, lambda b: batch.step(dev_depth[b], dev_pose[b], shifts, intr, float(CELL), dev_feat[b]), d2h_levels, n_fr)
    batch.layout = layout0
    h2d = E * (C * H * W * 2 + H * W * 4 + 48)
    out["dense_bf16_hwc"] = {"value": world * E * n_fr * args.e2e_steps / sec, "unit": UNIT, "h2d_bytes_per_step": int(h2d * n_fr),
                             "d2h_bytes_per_step": int(sum(l.numel() * 2 for l in batch.levels) * n_fr),
                             "h2d_GBps_per_rank": h2d * n_fr * args.e2e_steps / sec / 1e9}
    del dev_feat, pin_feat
    # ---- object regime ----
    rng = np.random.default_rng(3)
    Kmax, n_var = 16, 4
    bf = np.zeros((n_var, E, Kmax, C), np.float32); pr = np.zeros((n_var, E, Kmax, 28, 28), np.float32); bx = np.zeros((n_var, E, Kmax, 4), np.float32)
    n = np.zeros((n_var, E), np.int32)
    for v in range(n_var):
        for e in range(E):
            f, p_, b_ = eod.episodes.make_mask_head_detections(rng, H, W, C, (4, Kmax), 28)
            n[v, e] = f.shape[0]; bf[v, e, : n[v, e]], pr[v, e, : n[v, e]], bx[v, e, : n[v, e]] = f, p_, b_
    pin_det = [torch.from_numpy(x).pin_memory() for x in (bf, pr, bx, n)]
    dev_det = [[torch.empty(x.shape[1:], dtype=x.dtype, device=dev) for x in pin_det] for _ in range(NB)]
    host_l2 = torch.empty(batch.levels[2].shape, dtype=torch.float16).pin_memory()

    def up_det(t, b):
        for d, p_ in zip(dev_det[b], pin_det):
            d.copy_(p_[t % n_var], non_blocking=True)

    # D2H of the coarsest pooled level off the compute stream: a device-to-device copy into a double-buffered staging tensor (6 us) is
    # ordered behind the read; the copy to pinned host memory runs on its own stream, so the next frame-step's launches do not queue
    # behind 0.18 ms of PCIe (the inline copy serialised frame-steps: profiles/diag_e2e_obj.py)
    d2h_s = torch.cuda.Stream(device=dev)
    stage_l2 = [torch.empty_like(batch.levels[2]) for _ in range(2)]
    d2h_done = [torch.cuda.Event() for _ in range(2)]
    for ev_ in d2h_done:
        ev_.record(comp_s)
    d2h_k = [0]

    def d2h_l2():
        k = d2h_k[0] & 1
        d2h_k[0] += 1
        comp_s.wait_event(d2h_done[k])                     # the staging half is free again
        stage_l2[k].copy_(batch.levels[2])
        ready_ev = torch.cuda.Event()
        ready_ev.record(comp_s)
        with torch.cuda.stream(d2h_s):
            d2h_s.wait_event(ready_ev)
            host_l2.copy_(stage_l2[k], non_blocking=True)
            d2h_done[k].record(d2h_s)

    n_fr_obj = 5 * n_fr
    batch.pipeline = True          # the write side of frame t runs under the staging / geometry / paste of frame t+1; inputs are ordered on the
    dev_depth3 = dev_depth + [torch.empty((E, H, W), device=dev) for _ in range(NB - 2)]
    sec = run(up_det, lambda b: batch.step_detections(dev_depth3[b], dev_pose[b], shifts, intr, float(CELL), *dev_det[b], inputs_ready=False),   # caller's stream
              d2h_l2, n_fr_obj, None, dev_depth3)
    h2d = E * (H * W * 4 + 48) + sum(int(x[0].numel() * x.element_size()) for x in pin_det)
    out["object_regime"] = {"value": world * E * n_fr_obj * args.e2e_steps / sec, "unit": UNIT, "ms_per_frame_step": 1e3 * sec / (n_fr_obj * args.e2e_steps),
                            "h2d_bytes_per_step": int(h2d * n_fr_obj), "d2h_bytes_per_step": int(host_l2.numel() * 2 * n_fr_obj),
                            "shape": f"E={E}, C={C}, <= {Kmax} detections per frame; D2H = the coarsest pooled level (15x20) per frame-step"}
    # ---- object regime with the depth in the sensor's own format: uint16 millimetres (robot_demo.py:515), divided inside the kernel ----
    pin_depth16 = (torch.from_numpy(depth_h).permute(1, 0, 2, 3) * 1000.0).round().clamp_(0, 65535).to(torch.uint16).contiguous().pin_memory()
    dev_depth16 = [torch.empty((E, H, W), dtype=torch.uint16, device=dev) for _ in range(NB)]
    sec = run(up_det, lambda b: batch.step_detections(dev_depth16[b], dev_pose[b], shifts, intr, float(CELL), *dev_det[b], inputs_ready=False),
              d2h_l2, n_fr_obj, pin_depth16, dev_depth16)
    h2d = E * (H * W * 2 + 48) + sum(int(x[0].numel() * x.element_size()) for x in pin_det)
    out["object_regime_u16_depth"] = {"value": world * E * n_fr_obj * args.e2e_steps / sec, "unit": UNIT, "ms_per_frame_step": 1e3 * sec / (n_fr_obj * args.e2e_steps),
                                      "h2d_bytes_per_step": int(h2d * n_fr_obj), "d2h_bytes_per_step": int(host_l2.numel() * 2 * n_fr_obj),
                                      "shape": "as object_regime, depth uploaded as uint16 millimetres (eod_backproject_quantize_u16)"}
    # ---- the same with the frame-step captured into one CUDA graph (EpisodeBatch.capture_step_detections): one launch per frame-step
    # instead of ~12 launches on two streams; the uploaded buffers are copied device-to-device into the graph's static inputs ----
    try:
        graphed = batch.capture_step_detections(dev_depth16[0], dev_pose[0], shifts, intr, float(CELL), *dev_det[0])
        sec = run(up_det, lambda b: graphed(dev_depth16[b], dev_pose[b], shifts, *dev_det[b]),
                  d2h_l2, n_fr_obj, pin_depth16, dev_depth16)
        out["object_regime_u16_depth_graph"] = {"value": world * E * n_fr_obj * args.e2e_steps / sec, "unit": UNIT,
                                                "ms_per_frame_step": 1e3 * sec / (n_fr_obj * args.e2e_steps), "h2d_bytes_per_step": int(h2d * n_fr_obj),
                                                "d2h_bytes_per_step": int(host_l2.numel() * 2 * n_fr_obj),
                                                "shape": "as object_regime_u16_depth, one CUDA-graph launch per frame-step"}
        del graphed
    except Exception as exc:
        out["object_regime_u16_depth_graph"] = {"error": repr(exc)[:300]}
    batch.join()
    batch.pipeline = False
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline loop and of value_with_fusion; roofline_1000 "
                    "times max(2, min(steps, 5)) steps of its larger grid and reports that count as its own 'steps'")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-frames", type=int, default=8)
    ap.add_argument("--e2e-frames", type=int, default=4)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--write-variant", type=int, default=0, help="diagnostics: 0 auto, 1 LDG, 2 TMA, 3 TMA dry (no result)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run oracle check of the benchmarked path")
    ap.add_argument("--workload", default="cfg1", choices=["cfg1", "cfg5"], help="cfg1: BASELINE configs[1] (default, the driver's line); "
                    "cfg5: configs[4], 512 episodes x 100 frames, C=512, 1000x1000, strong scaling over --gpus")
    ap.add_argument("--slots", type=int, default=32, help="cfg5: resident grids per GPU")
    ap.add_argument("--cfg5-episodes", type=int, default=512)
    ap.add_argument("--cfg5-frames", type=int, default=100)
    ap.add_argument("--no-extras", action="store_true", help="skip the projection+fusion and object-regime stage timings")
    ap.add_argument("--no-numa", action="store_true", help="diagnostics: do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-pipeline", action="store_true", help="diagnostics: stream-ordered EpisodeBatch.step (no cross-frame overlap)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's pooled levels and grid state "
                    f"as DIR/<name>.npy (float32; arrays over {DUMP_SAMPLE} elements as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "cfg1"):
        ap.error("--dump-outputs applies to the default workload on the GPU (--impl b200 --workload cfg1)")
    rank, local_rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        return main_reference(args, rank, world)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "cfg5":
            main_cfg5(args, rank, local_rank, world)
        else:
            main_gpu(args, rank, local_rank, world)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
