"""Deterministic write (EOD_WRITE_DET) against the default write, by feature layout, and what it costs an EpisodeRunner run.

Part 1, the bench batch (E=64, 480x640, C=256, 500x500): fp32 CHW, fp32 channels-last and bf16 channels-last, each with the default
and the deterministic write.  The write launch alone (count and finalize outside the window; for WRITE_DET the window holds its nine
launches: pre-passes, main pass, segmented reduce), then whole frame-steps (EpisodeBatch.step, pipelined).  Every arm reads two
resident feature slabs used alternately (10-20 GB each, far beyond the 126 MB L2); the arms are interleaved over several rounds so that
they share the box's drift.

Part 2, one configs[4]-shaped EpisodeRunner run (PooledSyntheticProvider, R=32 resident 1000x1000x512 grids, ragged waves of
episodic episodes): default against WRITE_DET with the workspace at its default size (HW/4 runs per episode and frame), frames/s over
the whole run and whether the workspace overflowed.

CUDA events throughout.  The GPU name, its power limit and the median SM clock sampled during the run are recorded in the same
output."""
import importlib, json, math, os, subprocess, sys, threading
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
eod = importlib.import_module("embodied-object-detection_b200")
lib = eod._lib
dev = torch.device("cuda:0")
H, W, mw, mh, cell, C, E = 480, 640, 500, 500, 0.2, 256, 64
N = H * W
ROUNDS, ITERS, STEPS = 3, 6, 30
R5, C5, G5, EP5, T5 = 32, 512, 1000, 96, 100          # runner: slots, channels, grid side, episodes, frames per episode


def smi(query):
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={query}", "--format=csv,noheader,nounits"], capture_output=True,
                             text=True, timeout=10).stdout.strip()
        return [x.strip() for x in out.split(",")]
    except (OSError, subprocess.SubprocessError):
        return None


clocks, stop = [], threading.Event()


def sample_clock():
    while not stop.is_set():
        v = smi("clocks.sm")
        if v and v[0].replace(".", "").isdigit():
            clocks.append(float(v[0]))
        stop.wait(0.2)


sampler = threading.Thread(target=sample_clock, daemon=True)
sampler.start()

# ---- part 1: write launch and frame-step by layout ---------------------------------------------------------------------------
eps = [eod.episodes.make_episode(1234 + e, 2, H, W, mw, mh, cell) for e in range(E)]
Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, 2, 4, 4)
pose = Tm[:, :, :3, :].reshape(E, 2, 12).permute(1, 0, 2).contiguous().to(dev)
depth = torch.from_numpy(np.stack([ep.depth for ep in eps])).permute(1, 0, 2, 3).contiguous().to(dev)
shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(dev)
intr = eod.compute_intrinsics(W, H, math.radians(67.5))

g = torch.Generator(device=dev).manual_seed(7)
chw = [torch.randn((E, C, H, W), device=dev, generator=g) for _ in range(2)]
hwc = [c.permute(0, 2, 3, 1).contiguous() for c in chw]
hwc16 = [h.to(torch.bfloat16) for h in hwc]

# arm -> (layout, variant, slabs, bytes per feature element)
ARMS = {}
for name, layout, slabs, eb in (("chw_f32", lib.LAYOUT_CHW, chw, 4), ("hwc_f32", lib.LAYOUT_HWC, hwc, 4), ("hwc_bf16", lib.LAYOUT_HWC_BF16, hwc16, 2)):
    ARMS[name] = (layout, lib.WRITE_AUTO, slabs, eb)
    ARMS[name + "_det"] = (layout, lib.WRITE_DET, slabs, eb)

write_ms = {k: [] for k in ARMS}
batch = eod.EpisodeBatch(E, mw, mh, C, H, W, dev)
batch.project(depth[0], pose[0], shifts, intr, cell)
for r in range(ROUNDS):
    for name, (layout, variant, slabs, _) in ARMS.items():
        batch.layout, batch.variant = layout, variant
        for t in range(ITERS + 1):
            batch._count(None)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); batch._write(slabs[t & 1], None); b.record()
            batch._finalize()
            torch.cuda.synchronize()
            if t:                                                    # the first launch of an arm in a round is its warm-up
                write_ms[name].append(a.elapsed_time(b))
overflow_write = batch._det_ws.overflowed()
ws_bytes_bench = batch._det_ws.nbytes
del batch
torch.cuda.empty_cache()

step_ms = {k: [] for k in ARMS}
b2 = eod.EpisodeBatch(E, mw, mh, C, H, W, dev, pipeline=True)
for r in range(ROUNDS):
    for name, (layout, variant, slabs, _) in ARMS.items():
        b2.join(); torch.cuda.synchronize()
        b2.layout, b2.variant = layout, variant
        for t in range(3):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, slabs[t & 1])
        b2.join(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(STEPS):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, slabs[t & 1])
        b2.join(); b.record(); torch.cuda.synchronize()
        step_ms[name].append(a.elapsed_time(b) / STEPS)
overflow_step = b2._det_ws.overflowed()
EB = {name: arm[3] for name, arm in ARMS.items()}
del b2, ARMS, slabs, chw, hwc, hwc16, depth          # the runner below needs the memory
torch.cuda.empty_cache()

out = {"gpu": torch.cuda.get_device_name(0), "power_limit_W": (smi("power.limit") or [None])[0],
       "max_sm_clock_MHz": (smi("clocks.max.sm") or [None])[0], "E": E, "H": H, "W": W, "C": C, "grid": [mw, mh], "rounds": ROUNDS,
       "det_workspace_GB": ws_bytes_bench / 1e9, "det_overflowed": bool(overflow_write or overflow_step), "arms": {}}
for name, eb in EB.items():
    ms, sm = float(np.median(write_ms[name])), float(np.median(step_ms[name]))
    out["arms"][name] = {"write_ms": ms, "write_ms_min": float(min(write_ms[name])), "write_ms_max": float(max(write_ms[name])),
                         "feature_GBps": E * N * C * eb / ms / 1e6, "frame_step_ms": sm, "frame_step_ms_rounds": step_ms[name],
                         "frames_per_s": E / sm * 1e3}

# ---- part 2: configs[4]-shaped EpisodeRunner, default against WRITE_DET ------------------------------------------------------
intr5 = eod.compute_intrinsics(W, H, math.radians(67.5))
provider = eod.runner.PooledSyntheticProvider(EP5, T5, C5, R5, dev, H, W, G5, G5, cell, pool=64)
runs = {}
for name, variant in (("default", lib.WRITE_AUTO), ("det", lib.WRITE_DET)):
    runner = eod.EpisodeRunner(provider, G5, G5, C5, R5, height=H, width=W, device=dev, test_type="episodic", intr=intr5, cell=cell,
                               variant=variant)
    runner.run(max_steps=12)                                         # warm-up: the first wave's first frame-steps
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    st = runner.run()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    grid_bytes = runner.batch.sums.numel() * 4 + runner.batch.counts.numel() * 4 + runner.batch.norm16.numel() * 2
    runs[name] = {"frames": st["frames"], "frame_steps": st["steps"], "ms": ms, "frames_per_s": st["frames"] / ms * 1e3,
                  "grids_GB": grid_bytes / 1e9}
    if variant == lib.WRITE_DET:
        runs[name].update(det_overflowed=st["det_overflowed"], det_workspace_GB=runner.batch._det_ws.nbytes / 1e9)
    del runner
    torch.cuda.empty_cache()
stop.set()
sampler.join()
out["runner"] = {"slots": R5, "C": C5, "grid": [G5, G5], "episodes": EP5, "frames_per_episode": T5, "test_type": "episodic", **runs}
out["median_sm_clock_MHz"] = float(np.median(clocks)) if clocks else None
out["clock_samples"] = len(clocks)
print(json.dumps(out))
if len(sys.argv) > 1:                                                # optional: also write the record to a file
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as fh:
        json.dump(out, fh, indent=1)
