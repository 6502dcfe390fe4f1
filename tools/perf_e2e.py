"""GPU-box helper: the e2e call (vq_forward_lighting_host, pinned host buffers) at 4K with the library's row chunking, next to
what the PCIe link does on plain copies of the same buffers."""
import os, sys, time, json
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import vqengine_b200 as vq
from vqengine_b200 import synth
import bench
ctx = vq.Context(0)
W, H = 3840, 2160
envk = bench.build_env_maps_gpu(ctx, vq, torch)
ctx.environment_prepare(envk["env"]) if hasattr(ctx, "environment_prepare") else None
planes = synth.gbuffer(W, H)
pf, pv = synth.scene_constants(W, H, envk["spec_mips"])
hpl = [torch.from_numpy(p).pin_memory() for p in planes]
hgb = vq.GBuffer(vq.image_of(hpl[0]), vq.image_of(hpl[1]), vq.image_of(hpl[2]), vq.null_image())
hout = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()
ctx.resize(W, H)
def timeit(fn, reps=6):
    fn(); fn(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps): fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps
dt = timeit(lambda: ctx.forward_lighting_host(pf, pv, hgb, envk["env"], hout))
res = {"e2e": {"ms": round(dt * 1e3, 3), "Mpixels_per_s": round(W * H / dt / 1e6, 1)}}
d = torch.empty((H, W, 4), dtype=torch.float32, device="cuda"); d2 = torch.empty_like(d)
nb = d.numel() * 4
s2 = torch.cuda.Stream()
t_up = timeit(lambda: d.copy_(hpl[0], non_blocking=True))
t_dn = timeit(lambda: hout.copy_(d, non_blocking=True))
def both():
    d.copy_(hpl[0], non_blocking=True)
    with torch.cuda.stream(s2): hout.copy_(d2, non_blocking=True)
t_b = timeit(both)
def three_up():
    for p in hpl: d.copy_(p, non_blocking=True)
t3 = timeit(three_up)
res["link"] = {"h2d_GBps": round(nb / t_up / 1e9, 1), "d2h_GBps": round(nb / t_dn / 1e9, 1), "both_each_GBps": round(nb / t_b / 1e9, 1),
               "h2d_3_planes_ms": round(t3 * 1e3, 3), "floor_ms": round(max(3 * nb / (nb / t_up), nb / (nb / t_dn)) * 1e3, 3)}
print(json.dumps(res, indent=1))
