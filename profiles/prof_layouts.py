"""Dense write kernel by feature layout at the bench batch (E=64, 480x640, C=256, 500x500): fp32 CHW (TMA ring), bf16 / fp16 CHW
(the 16-bit TMA ring: what a bf16 / autocast backbone emits in NCHW), bf16 channels-last, the dry ring (variant 3: stream the tiles,
no arithmetic) of the fp32 and 16-bit units, and the two ways a bf16 NCHW producer could feed the write without a 16-bit CHW layout:
``.float()`` then the fp32 CHW write, or a permute to channels-last then the bf16 HWC write (the conversion is inside the timed
window).  Then whole frame-steps (EpisodeBatch.step, pipelined) for the same arms.  CUDA events; every arm reads two resident
feature slabs used alternately (>= 10 GB each, far beyond the 126 MB L2); the arms are interleaved over several rounds so that they
share the box's drift.  GB/s = E * (N*C*e + N*4) / ms with e = 2 bytes for every arm fed from bf16 / fp16 features (the bytes the
producer's tensor holds), 4 for fp32.  The GPU name, its power limit and the median SM clock sampled during the run are recorded in
the same output."""
import importlib, json, math, os, subprocess, sys, threading
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
eod = importlib.import_module("embodied-object-detection_b200")
lib = eod._lib
dev = torch.device("cuda:0")
H, W, mw, mh, cell, C, E = 480, 640, 500, 500, 0.2, 256, 64
N = H * W
ROUNDS, ITERS, STEPS = 3, 6, 30


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


eps = [eod.episodes.make_episode(1234 + e, 2, H, W, mw, mh, cell) for e in range(E)]
Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, 2, 4, 4)
pose = Tm[:, :, :3, :].reshape(E, 2, 12).permute(1, 0, 2).contiguous().to(dev)
depth = torch.from_numpy(np.stack([ep.depth for ep in eps])).permute(1, 0, 2, 3).contiguous().to(dev)
shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(dev)
intr = eod.compute_intrinsics(W, H, math.radians(67.5))

g = torch.Generator(device=dev).manual_seed(7)
f32 = [torch.randn((E, C, H, W), device=dev, generator=g) for _ in range(2)]          # fp32 CHW slabs (also the .float() targets)
bf16 = [f.to(torch.bfloat16) for f in f32]                                           # the bf16 NCHW producer's output
f16 = [f.to(torch.float16) for f in f32]
hwc = [torch.empty((E, H, W, C), dtype=torch.bfloat16, device=dev) for _ in range(2)]
for s in range(2):
    hwc[s].copy_(bf16[s].permute(0, 2, 3, 1))                                       # resident channels-last bf16 slabs


def to_float(t):           # workaround 1: widen the whole slab, then the fp32 CHW write
    f32[t & 1].copy_(bf16[t & 1])
    return f32[t & 1]


def to_hwc(t):             # workaround 2: permute to channels-last, then the bf16 HWC write
    hwc[t & 1].copy_(bf16[t & 1].permute(0, 2, 3, 1))
    return hwc[t & 1]


# arm -> (layout, variant, feature of step t, bytes per element of the producer's features)
ARMS = {
    "chw_f32": (lib.LAYOUT_CHW, lib.WRITE_AUTO, lambda t: f32[t & 1], 4),
    "chw_bf16": (lib.LAYOUT_CHW_BF16, lib.WRITE_AUTO, lambda t: bf16[t & 1], 2),
    "chw_f16": (lib.LAYOUT_CHW_F16, lib.WRITE_AUTO, lambda t: f16[t & 1], 2),
    "hwc_bf16": (lib.LAYOUT_HWC_BF16, lib.WRITE_AUTO, lambda t: hwc[t & 1], 2),
    "bf16_float_then_chw_f32": (lib.LAYOUT_CHW, lib.WRITE_AUTO, to_float, 2),
    "bf16_permute_then_hwc_bf16": (lib.LAYOUT_HWC_BF16, lib.WRITE_AUTO, to_hwc, 2),
    "chw_f32_dry": (lib.LAYOUT_CHW, lib.WRITE_TMA_DRY, lambda t: f32[t & 1], 4),
    "chw_bf16_dry": (lib.LAYOUT_CHW_BF16, lib.WRITE_TMA_DRY, lambda t: bf16[t & 1], 2),
}
STEP_ARMS = ["chw_f32", "chw_bf16", "chw_f16", "hwc_bf16", "bf16_float_then_chw_f32", "bf16_permute_then_hwc_bf16"]

sampler = threading.Thread(target=sample_clock, daemon=True)
sampler.start()
write_ms = {k: [] for k in ARMS}
batch = eod.EpisodeBatch(E, mw, mh, C, H, W, dev)
batch.project(depth[0], pose[0], shifts, intr, cell)
for r in range(ROUNDS):
    for name, (layout, variant, feat, _) in ARMS.items():
        batch.layout, batch.variant = layout, variant
        for t in range(ITERS + 1):
            batch._count(None)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); batch._write(feat(t), None); b.record()
            batch._finalize()
            torch.cuda.synchronize()
            if t:                                                    # the first launch of an arm in a round is its warm-up
                write_ms[name].append(a.elapsed_time(b))
del batch
torch.cuda.empty_cache()

step_ms = {k: [] for k in STEP_ARMS}
b2 = eod.EpisodeBatch(E, mw, mh, C, H, W, dev, pipeline=True)
for r in range(ROUNDS):
    for name in STEP_ARMS:
        layout, variant, feat, _ = ARMS[name]
        b2.layout = layout
        for t in range(3):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, feat(t))
        b2.join(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(STEPS):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, feat(t))
        b2.join(); b.record(); torch.cuda.synchronize()
        step_ms[name].append(a.elapsed_time(b) / STEPS)
stop.set()
sampler.join()

out = {"gpu": torch.cuda.get_device_name(0), "power_limit_W": (smi("power.limit") or [None])[0],
       "max_sm_clock_MHz": (smi("clocks.max.sm") or [None])[0], "median_sm_clock_MHz": float(np.median(clocks)) if clocks else None,
       "clock_samples": len(clocks), "E": E, "H": H, "W": W, "C": C, "grid": [mw, mh], "rounds": ROUNDS, "arms": {}}
for name, (_, _, _, eb) in ARMS.items():
    ms = float(np.median(write_ms[name]))
    arm = {"write_ms": ms, "write_ms_min": float(min(write_ms[name])), "write_ms_max": float(max(write_ms[name])),
           "GBps": E * (N * C * eb + N * 4) / ms / 1e6}
    if name in step_ms:
        sm = float(np.median(step_ms[name]))
        arm.update(frame_step_ms=sm, frame_step_ms_rounds=step_ms[name], frames_per_s=E / sm * 1e3)
    out["arms"][name] = arm
print(json.dumps(out))
if len(sys.argv) > 1:                                                # optional: also write the record to a file
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as fh:
        json.dump(out, fh, indent=1)
