"""Cost of the deterministic object write: EpisodeBatch.step_detections(pipeline=True) at the bench's object shape (E=64, 480x640,
500x500 grid, <= 16 kept detections, fp32 depth resident) with the default object write and with object_variant=WRITE_DET, at C=256
and C=512.  Alternating rounds timed with CUDA events (frame-step = one step_detections of all E episodes, steady state), then one
torch.profiler pass of the deterministic batch for the per-stage split: run pre-passes, main pass, segmented reduce.  The card's name,
power limit and SM clock are read in the same run.  Writes one JSON file (argv[1], default profiles/objects_det.json).
PROF_E / PROF_K / PROF_T / PROF_ROUNDS override batch, max detections, steps per round and rounds."""
import importlib
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
eod = importlib.import_module("embodied-object-detection_b200")
dev = torch.device("cuda:0")
H, W, MW, MH, CELL = 480, 640, 500, 500, 0.2
E = int(os.environ.get("PROF_E", 64))
KMAX = int(os.environ.get("PROF_K", 16))
T = int(os.environ.get("PROF_T", 20))
ROUNDS = int(os.environ.get("PROF_ROUNDS", 3))
OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "objects_det.json")

# kernels of the deterministic write by stage (write_mean.cu / write_objects.cu)
STAGES = {"prepass": ("det_tile_runs", "det_scan_tiles", "det_cell_runs", "det_scan_list"), "main": ("write_objects_det_kernel",),
          "reduce": ("det_claim", "det_reduce", "det_chunk", "det_final")}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power, sm, sm_max = [x.strip() for x in q[0].split(",")] if q else ("?", "?", "?", "?")
    return {"name": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}


def inputs():
    eps = [eod.episodes.make_episode(1234 + e, 4, H, W, MW, MH, CELL) for e in range(E)]
    Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, 4, 4, 4)
    pose = Tm[:, :, :3, :].reshape(E, 4, 12).permute(1, 0, 2).contiguous().to(dev)
    depth = torch.from_numpy(np.stack([ep.depth for ep in eps])).permute(1, 0, 2, 3).contiguous().to(dev)
    shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(dev)
    return depth, pose, shifts


def detections(rng, C):
    out = []
    for _ in range(2):
        bf, pr, bx = np.zeros((E, KMAX, C), np.float32), np.zeros((E, KMAX, 28, 28), np.float32), np.zeros((E, KMAX, 4), np.float32)
        n = np.zeros(E, np.int32)
        for e in range(E):
            f, p, b = eod.episodes.make_mask_head_detections(rng, H, W, C, (4, KMAX), 28)
            n[e] = f.shape[0]
            bf[e, :n[e]], pr[e, :n[e]], bx[e, :n[e]] = f, p, b
        out.append(tuple(torch.from_numpy(a).to(dev) for a in (bf, pr, bx, n)))
    return out


def steps(batch, geo, dets, intr, t0, n):
    depth, pose, shifts = geo
    for t in range(t0, t0 + n):
        bf, pr, bx, nn = dets[t & 1]
        batch.step_detections(depth[t % 4], pose[t % 4], shifts, intr, CELL, bf, pr, bx, nn)
    batch.join()


def measure(C, geo, intr) -> dict:
    dets = detections(np.random.default_rng(C), C)
    batches = {"default": eod.EpisodeBatch(E, MW, MH, C, H, W, dev, pipeline=True),
               "det": eod.EpisodeBatch(E, MW, MH, C, H, W, dev, pipeline=True, object_variant=eod._lib.WRITE_DET)}
    for b in batches.values():
        steps(b, geo, dets, intr, 0, 4)                                     # warm-up: workspaces, modules, allocator
    torch.cuda.synchronize()
    ms = {k: [] for k in batches}
    t = 4
    for _ in range(ROUNDS):
        for k, b in batches.items():
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            steps(b, geo, dets, intr, t, T)
            z.record()
            torch.cuda.synchronize()
            ms[k].append(a.elapsed_time(z) / T)
        t += T
    res = {"C": C, "frame_step_ms": {k: v for k, v in ms.items()},
           "frame_step_ms_median": {k: float(np.median(v)) for k, v in ms.items()}}
    res["det_over_default"] = res["frame_step_ms_median"]["det"] / res["frame_step_ms_median"]["default"]
    res["det_overflowed"] = batches["det"]._det_ws.overflowed()
    # per-stage split of the deterministic write (kernel time summed over the profiled steps, per frame-step)
    n_prof = 6
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        steps(batches["det"], geo, dets, intr, t, n_prof)
        torch.cuda.synchronize()
    stage_us = {k: 0.0 for k in STAGES}
    kernels = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        kernels[ev.key] = us / n_prof / 1e3
        for k, names in STAGES.items():
            if any(s in ev.key for s in names):
                stage_us[k] += us
    res["det_stage_ms"] = {k: v / n_prof / 1e3 for k, v in stage_us.items()}
    res["det_kernels_ms"] = dict(sorted(kernels.items(), key=lambda kv: -kv[1])[:16])
    del batches
    torch.cuda.empty_cache()
    return res


def main():
    info = {"card": card(), "E": E, "H": H, "W": W, "grid": [MW, MH], "k_max": KMAX, "steps_per_round": T, "rounds": ROUNDS,
            "pipeline": True, "depth": "fp32 resident"}
    geo = inputs()
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    info["results"] = [measure(C, geo, intr) for C in (256, 512)]
    info["card_after"] = card()
    os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
    with open(OUT, "w") as f:
        json.dump(info, f, indent=1)
    print(json.dumps(info, indent=1))


if __name__ == "__main__":
    main()
