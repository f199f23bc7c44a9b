"""Write kernel alone (CHW TMA, E=64, C=256, 500x500) under the diagnostic knobs: ring depth (EOD_TMA_STAGES) and no reductions
(EOD_TMA_NO_RED, wrong results - profiling only).  One process per setting (the knobs are read once)."""
import importlib, json, math, os, subprocess, sys
if len(sys.argv) > 1:
    import numpy as np, torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    eod = importlib.import_module("embodied-object-detection_b200")
    dev = torch.device("cuda:0")
    H, W, mw, mh, cell, C, E = 480, 640, 500, 500, 0.2, 256, 64
    eps = [eod.episodes.make_episode(1234 + e, 2, H, W, mw, mh, cell) for e in range(E)]
    Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, 2, 4, 4)
    pose = Tm[:, 0, :3, :].reshape(E, 12).contiguous().to(dev)
    depth = torch.from_numpy(np.stack([ep.depth[0] for ep in eps])).to(dev)
    shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(dev)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, dev)
    feats = [torch.randn((E, C, H, W), device=dev) for _ in range(2)]
    batch.project(depth, pose, shifts, intr, cell)
    batch._count(None)
    for t in range(3):
        batch._write(feats[t & 1], None)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for t in range(20):
        batch._write(feats[t & 1], None)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 20
    print(json.dumps({"setting": sys.argv[1], "write_ms": ms, "GBps": E * (H * W * C * 4 + H * W * 4) / ms / 1e6}))
else:
    for name, env in (("default", {}), ("no_red", {"EOD_TMA_NO_RED": "1"}), ("stages5", {"EOD_TMA_STAGES": "5"}), ("stages4", {"EOD_TMA_STAGES": "4"}),
                      ("dry", None), ("default2", {})):
        e = dict(os.environ)
        if env is None:
            continue
        e.update(env)
        subprocess.run([sys.executable, __file__, name], env=e)
