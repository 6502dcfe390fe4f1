"""-m gpu: `bench.py --dump-outputs DIR` writes a fixed, seeded pixel sample of the frame its last timed step computed as .npy
files (float32 pixels, float64 indices, at most 64 MB together): the same bytes from run to run, and the lit frame itself (checked
against the oracle on the bench's own inputs). `--steps` sets the number of timed launches."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from gpu_util import assert_scaled, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 3840, 2160


def _bench_dump(d, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
                        "--no-extra", "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert j["steps"] == steps and j["gpu_launches"] == steps
    files = sorted(os.listdir(d))
    assert files == ["frame_sample.npy", "frame_sample_index.npy"]
    assert sum(os.path.getsize(d / f) for f in files) <= 64_000_000
    return np.load(d / "frame_sample.npy"), np.load(d / "frame_sample_index.npy")


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path, ctx, vq, orc):
    px, idx = _bench_dump(tmp_path / "a", 4)
    assert px.dtype == np.float32 and idx.dtype == np.float64 and px.shape == (len(idx), 4)
    assert idx[0] >= 0 and idx[-1] < W * H and (np.diff(idx) > 0).all() and (idx == np.round(idx)).all()
    px2, idx2 = _bench_dump(tmp_path / "b", 2)
    assert px.tobytes() == px2.tobytes() and idx.tobytes() == idx2.tobytes()

    # the sample is the lit frame of the bench's workload: the oracle on the same seeded inputs, on two row bands
    import bench
    import torch
    from vqengine_b200 import synth
    envk = bench.build_env_maps_gpu(ctx, vq, torch)
    planes = synth.gbuffer(W, H, seed=synth.SEED_BASE + 3)
    pf, pv = synth.scene_constants(W, H, envk["spec_mips"])
    env_np = {k: host(envk[k]) for k in ("diff", "spec", "lut")}
    ii = idx.astype(np.int64)
    for r0 in (7, 1500):
        ref = orc.forward_lighting(pf, pv, planes, env_np["diff"], envk["diff_res"], env_np["spec"], envk["spec_res"],
                                   envk["spec_mips"], env_np["lut"], r0, r0 + 12)
        sel = (ii >= r0 * W) & (ii < (r0 + 12) * W)
        assert sel.sum() > 1000
        assert_scaled(f"dumped rows {r0}", px[sel], ref.reshape(-1, 4)[ii[sel]])
    ctx.environment_invalidate()


def test_bench_dump_outputs_needs_the_gpu_path():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "unused"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
