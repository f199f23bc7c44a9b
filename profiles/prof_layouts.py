"""Dense write kernel by feature layout at the bench batch (E=64, 480x640, C=256, 500x500): fp32 CHW (TMA ring), fp32
channels-last, bf16 channels-last (a bf16 backbone's output: half the bytes of the dominant stream), and whole frame-steps
(EpisodeBatch.step, pipelined) for fp32 CHW vs bf16 HWC.  CUDA events."""
import importlib, json, math, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
eod = importlib.import_module("embodied-object-detection_b200")
ops = eod.ops
dev = torch.device("cuda:0")
H, W, mw, mh, cell, C, E = 480, 640, 500, 500, 0.2, 256, 64
eps = [eod.episodes.make_episode(1234 + e, 2, H, W, mw, mh, cell) for e in range(E)]
Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, 2, 4, 4)
pose = Tm[:, :, :3, :].reshape(E, 2, 12).permute(1, 0, 2).contiguous().to(dev)
depth = torch.from_numpy(np.stack([ep.depth for ep in eps])).permute(1, 0, 2, 3).contiguous().to(dev)
shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(dev)
intr = eod.compute_intrinsics(W, H, math.radians(67.5))
out = {}
for layout, name in ((eod._lib.LAYOUT_CHW, "chw_f32"), (eod._lib.LAYOUT_HWC, "hwc_f32"), (eod._lib.LAYOUT_HWC_BF16, "hwc_bf16")):
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, dev, layout=layout)
    feats = [torch.randn((E, C, H, W) if layout == 0 else (E, H, W, C), device=dev) for _ in range(2)]
    if layout == eod._lib.LAYOUT_HWC_BF16:
        feats = [f.to(torch.bfloat16) for f in feats]
    batch.project(depth[0], pose[0], shifts, intr, cell)
    ms = []
    for t in range(8):
        batch._count(None)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); batch._write(feats[t & 1], None); b.record()
        batch._finalize()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    ms = sorted(ms[2:])
    eb = feats[0].element_size()
    out[name] = {"write_ms": ms[len(ms) // 2], "GBps": E * (H * W * C * eb + H * W * 4) / ms[len(ms) // 2] / 1e6}
    if name != "hwc_f32":
        # whole frame-steps, pipelined like the bench
        b2 = eod.EpisodeBatch(E, mw, mh, C, H, W, dev, layout=layout, pipeline=True)
        for t in range(3):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, feats[t & 1])
        b2.join(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(20):
            b2.step(depth[t & 1], pose[t & 1], shifts, intr, cell, feats[t & 1])
        b2.join(); b.record(); torch.cuda.synchronize()
        out[name]["frame_step_ms"] = a.elapsed_time(b) / 20
        out[name]["frames_per_s"] = E / out[name]["frame_step_ms"] * 1e3
        del b2
    del batch, feats
    torch.cuda.empty_cache()
print(json.dumps(out))
