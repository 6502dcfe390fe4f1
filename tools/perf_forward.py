"""GPU-box helper: time K1 at 4K (prepared environment), print us + GB/s. Parity is checked by the tests:
   python -m pytest tests/test_forward_gpu.py -q -m gpu -k "full_size or config3" """
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import vqengine_b200 as vq
from vqengine_b200 import synth
import bench
ctx = vq.Context(0)
envk = bench.build_env_maps_gpu(ctx, vq, torch)
W, H = 3840, 2160
planes = synth.gbuffer(W, H)
pf, pv = synth.scene_constants(W, H, envk["spec_mips"])
dpl = [torch.from_numpy(p).cuda() for p in planes]
gb = vq.GBuffer(vq.image_of(dpl[0]), vq.image_of(dpl[1]), vq.image_of(dpl[2]), vq.null_image())
out = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
ms = bench.time_gpu(torch, lambda: ctx.forward_lighting(pf, pv, gb, envk["env"], out), 30, warmup=5)
print(f"forward 4K prepared: {ms*1e3:.1f} us  {W*H/ms/1e3:.0f} Mpx/s  {64*W*H/ms/1e6:.0f} GB/s  nan={int(torch.isnan(out).sum())}")
ctx.environment_invalidate()
ms2 = bench.time_gpu(torch, lambda: ctx.forward_lighting(pf, pv, gb, envk["env"], out), 30, warmup=5)
print(f"forward 4K per-call padding: {ms2*1e3:.1f} us")
