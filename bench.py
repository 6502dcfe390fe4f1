#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 shading backend (contract: task brief + BASELINE.json).

A "step" is ONE forward-PBR lighting pass (K1) with 4 point lights, 1 directional light and IBL, inputs resident in HBM:
  N = 1   the 3840x2160 synthetic G-buffer of BASELINE.json's metric "Mpixels/s forward-PBR @4K";
  N > 1   BASELINE config 5's 7680x4320 frame, STRONG-scaled: rank r shades rows [r*4320/N, (r+1)*4320/N) and the kernel itself
          stores every pixel into the frame of every rank over NVLink and runs the cross-rank rendezvous (ONE kernel = shade +
          tile assembly + barrier), so `value` includes the gather the north star names; kernel-only is under "kernel_only".
  value      = Mpixels/s of the whole job (max over ranks of the device time)
  e2e        = the same pass through the blocking host-buffer C-ABI call (pinned host G-buffer in,
               host image out; H2D/D2H inside the timed region)
  roofline   = algorithmic 64 B/pixel / kernel time, against the measured HBM copy peak
  cpu_baseline = the scalar oracle (CPU port of the HLSL) on this box's host cores, bounded row sample
  extra      = per-kernel timings for the other SURVEY.md §8 rows (post chain @4K, IBL integrals)
`--impl reference` times the reference's shader text compiled for the CPU (oracle/_ref/libhlslref.so), or the CPU oracle when that
library is absent (the reference's D3D12/HLSL path itself cannot run here).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

W4K, H4K = 3840, 2160
W8K, H8K = 7680, 4320
BYTES_PER_PX = 64          # SURVEY.md §8(d): 3 x float4 in + 1 x float4 out
METRIC = "forward_pbr_4k_mpixels_per_s"
UNIT = "Mpixels/s"
WORKLOAD = "forward-PBR 3840x2160 G-buffer (3 float4 planes), 4 point + 1 directional + IBL (64^2 diffuse, 512^2 x9 specular, 1024^2 LUT)"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _forward_source_digest():
    import hashlib
    h = hashlib.sha256()
    for f in ("vq_forward.cu", "vq_common.cuh"):
        h.update(open(os.path.join(ROOT, "vqengine_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def forward_profile_facts():
    """dram bytes and warp-instructions per 4K launch of K1 from the committed ncu capture (profiles/forward_traffic.json). The file
    carries the digest of the kernel source it was captured from: a stale file (the kernel changed since) is refused, not quoted."""
    tp = os.path.join(ROOT, "profiles", "forward_traffic.json")
    try:
        j = json.load(open(tp))
    except Exception:
        return None, None, "profiles/forward_traffic.json absent"
    if j.get("source_digest") != _forward_source_digest():
        return None, None, f"profiles/forward_traffic.json is stale (captured from source {j.get('source_digest')}, tree is {_forward_source_digest()})"
    return j.get("dram_bytes_per_launch"), j.get("warp_instructions_per_launch"), j.get("capture", "profiles/")


def pin_to_gpu_numa_node(torch, local):
    """e2e copies cross PCIe from pinned host memory: keep this rank's threads (and so its first-touch pinned pages) on the NUMA
    node its GPU hangs off. Returns a short description for the JSON line."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        if bus is None:
            return "unpinned (no pci ids)"
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "unpinned (single node)"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"numa node {node} ({len(cpus)} cpus)"
        return f"unpinned (node {node} has no allowed cpus)"
    except Exception as ex:
        return f"unpinned ({type(ex).__name__})"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def build_env_maps_gpu(ctx, vq, torch, hdri_w=2048, hdri_h=1024, diff_res=64, spec_res=512, spec_mips=9, lut=1024):
    """IBL inputs of the forward pass, produced by OUR kernels from a synthetic HDRI (setup, untimed)."""
    from vqengine_b200 import synth
    levels = vq.mip_level_count(hdri_w, hdri_h)
    pyr_t = torch.zeros((vq.pyramid_texel_count(hdri_w, hdri_h, levels), 4), dtype=torch.float32, device="cuda")
    pyr_t[: hdri_w * hdri_h] = torch.from_numpy(synth.hdri(hdri_w, hdri_h)).cuda().reshape(-1, 4)
    pyr = vq.pyramid_of(pyr_t, hdri_w, hdri_h, levels)
    ctx.hdri_build_mips(pyr)
    diff = torch.zeros((6 * diff_res * diff_res, 4), dtype=torch.float32, device="cuda")
    ctx.diffuse_irradiance(pyr, vq.cubemap_of(diff, diff_res, 1), n_phi=64, n_theta=16, src_mip=3)
    # per-face Gaussian blur (EnvironmentMapRendering.cpp:279-373)
    faces = diff.view(6, diff_res, diff_res, 4)
    tmp = torch.empty_like(faces[0]); blurred = torch.empty_like(faces)
    for f in range(6):
        ctx.gaussian_blur(faces[f], tmp, False)
        ctx.gaussian_blur(tmp, blurred[f], True)
    spec = torch.zeros((vq.cubemap_texel_count(spec_res, spec_mips), 4), dtype=torch.float32, device="cuda")
    ctx.specular_prefilter(pyr, vq.cubemap_of(spec, spec_res, spec_mips), 512)
    lut_t = torch.zeros((lut, lut, 2), dtype=torch.float32, device="cuda")
    ctx.brdf_integration_lut(lut_t, 2048)
    torch.cuda.synchronize()
    keep = dict(pyr_t=pyr_t, pyr=pyr, diff=blurred.reshape(-1, 4).contiguous(), spec=spec, lut=lut_t,
                diff_res=diff_res, spec_res=spec_res, spec_mips=spec_mips, levels=levels, hdri_w=hdri_w, hdri_h=hdri_h)
    keep["env"] = vq.EnvironmentMaps(vq.cubemap_of(keep["diff"], diff_res, 1), vq.cubemap_of(spec, spec_res, spec_mips),
                                     vq.image_of(lut_t, 2))
    # the RENDER_TARGET -> SHADER_RESOURCE transition after prefiltering: bordered sampling copies, built once
    ctx.environment_prepare(keep["env"])
    torch.cuda.synchronize()
    return keep


DUMP_PIXELS = 1 << 21       # 2M pixels x float4 = 32 MB (+ 16 MB of indices): within 64 MB for the 4K and the 8K frame alike
DUMP_SEED = 0


def dump_sample_index(torch, frame):
    """The fixed sample of the frame (H x W x 4) that --dump-outputs writes: DUMP_PIXELS flat pixel indices y * W + x drawn
    without replacement from a generator seeded with DUMP_SEED, sorted, on the frame's device."""
    h, w, _ = frame.shape
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, size=min(DUMP_PIXELS, h * w), replace=False))
    return torch.from_numpy(idx).to(frame.device)


def write_dump(out_dir, idx, px):
    """frame_sample.npy: the RGBA of the sampled pixels (N x 4 float32); frame_sample_index.npy: their flat indices (float64, exact)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame_sample.npy"), px.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "frame_sample_index.npy"), idx.cpu().numpy().astype(np.float64))


def time_gpu(torch, fn, iters, warmup=3, min_warm_ms=30.0, min_timed_ms=20.0):
    """CUDA-event timing on the current stream. Warm-up runs at least `warmup` launches AND `min_warm_ms` of GPU work (the
    SM clock needs a few ms of load to leave its idle state after host-side input generation); the timed region is at
    least `iters` launches and about `min_timed_ms` long."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); n = 0
    while True:
        fn(); n += 1
        if n >= warmup:
            e1.record(); torch.cuda.synchronize()
            if e0.elapsed_time(e1) >= min_warm_ms or n >= 2000:
                break
    per = max(e0.elapsed_time(e1) / n, 1e-3)
    iters = max(iters, min(int(min_timed_ms / per), 2000))
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters   # ms


def extra_passes(ctx, vq, torch, envk, peak):
    """Per-kernel numbers for the other SURVEY.md §8 rows (single GPU; not part of `value`)."""
    from vqengine_b200 import synth
    out = {}
    w, h = W4K, H4K
    px = w * h
    img = torch.from_numpy(synth.hdr_image(w, h)).cuda()
    a, b, t, c = (torch.empty_like(img) for _ in range(4))
    e = torch.empty((2 * h, 2 * w, 4), dtype=torch.float32, device="cuda")
    r = torch.empty_like(e)
    (dx, dy), sc = vq.spd_setup(w, h)
    mips = [torch.empty((h >> l, w >> l, 4), dtype=torch.float32, device="cuda") for l in range(1, sc.mips + 1)]
    tm = synth.default_tonemapper()
    cas_c, easu_c, rcas_c = vq.cas_setup(0.8, w, h, w, h), vq.fsr_easu_con(w, h, w, h, 2 * w, 2 * h), vq.fsr_rcas_con(0.2)
    passes = [
        ("spd", lambda: ctx.spd_downsample(sc, img, mips), px * (16 + 16 / 3)),
        ("blur_x", lambda: ctx.gaussian_blur(img, a, False), px * 32),
        ("blur_y", lambda: ctx.gaussian_blur(a, b, True), px * 32),
        ("tonemap", lambda: ctx.tonemap(tm, b, t), px * 32),
        ("cas", lambda: ctx.cas(cas_c, t, c), px * 32),
        ("fsr_easu_2x", lambda: ctx.fsr_easu(easu_c, c, e), px * 16 + 4 * px * 16),
        ("fsr_rcas_8k", lambda: ctx.fsr_rcas(rcas_c, e, r), 4 * px * 32),
    ]
    chain_ms, chain_bytes = 0.0, 0.0
    for name, fn, nbytes in passes:
        ms = time_gpu(torch, fn, 10)
        gbs = nbytes / ms / 1e6
        out[name] = {"ms": round(ms, 4), "algorithmic_GBps": round(gbs, 1), "hbm_frac": round(gbs / peak, 3)}
        chain_ms += ms; chain_bytes += nbytes
    out["post_chain_4k"] = {"ms": round(chain_ms, 4), "input_Mpixels_per_s": round(px / chain_ms / 1e3, 1),
                            "algorithmic_GBps": round(chain_bytes / chain_ms / 1e6, 1),
                            "hbm_frac": round(chain_bytes / chain_ms / 1e6 / peak, 3)}
    del img, a, b, t, c, e, r, mips
    # IBL integrals (bound: SFU/FP32 + L1/L2, not HBM; texels/s and samples/s are the honest figures)
    pyr = envk["pyr"]
    res, nm = envk["spec_res"], envk["spec_mips"]
    spec = torch.empty_like(envk["spec"])
    ms = time_gpu(torch, lambda: ctx.specular_prefilter(pyr, vq.cubemap_of(spec, res, nm), 512), 3, warmup=1)
    texels = vq.cubemap_texel_count(res, nm)
    out["ibl_specular_prefilter"] = {"config": f"{envk['hdri_w']}x{envk['hdri_h']} HDRI -> {res}^2 x6 x{nm} mips, 512 samples",
                                     "ms": round(ms, 3), "texels_per_s": round(texels / ms * 1e3),
                                     "samples_per_s": round(texels * 512 / ms * 1e3)}
    diff = torch.empty((6 * 64 * 64, 4), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.diffuse_irradiance(pyr, vq.cubemap_of(diff, 64, 1), n_phi=64, n_theta=16, src_mip=3), 5, warmup=1)
    out["ibl_diffuse_irradiance"] = {"config": "2048x1024 HDRI -> 64^2 x6, 64x16 = 1024 samples (BASELINE config 2)",
                                     "ms": round(ms, 4), "texels_per_s": round(6 * 64 * 64 / ms * 1e3),
                                     "samples_per_s": round(6 * 64 * 64 * 1024 / ms * 1e3)}
    ms = time_gpu(torch, lambda: ctx.diffuse_irradiance(pyr, vq.cubemap_of(diff, 64, 1), step=0.01, src_mip=3), 1, warmup=1)
    out["ibl_diffuse_irradiance_reference_step"] = {"config": "step 0.010 -> 629x158 = 99382 samples/texel (engine default)",
                                                    "ms": round(ms, 3), "samples_per_s": round(6 * 64 * 64 * 99382 / ms * 1e3)}
    lut = torch.empty((1024, 1024, 2), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.brdf_integration_lut(lut, 2048), 2, warmup=1)
    out["brdf_lut"] = {"config": "1024^2, 2048 samples", "ms": round(ms, 3), "samples_per_s": round(1024 * 1024 * 2048 / ms * 1e3)}
    ms = time_gpu(torch, lambda: ctx.hdri_build_mips(pyr), 5, warmup=1)
    nb = envk["hdri_w"] * envk["hdri_h"] * (16 * 4 / 3 + 16 / 3)
    out["hdri_min_pyramid"] = {"ms": round(ms, 4), "algorithmic_GBps": round(nb / ms / 1e6, 1)}
    out.update(surface_producer_pass(ctx, vq, torch, peak))
    out.update(frame_format_passes(ctx, vq, torch, envk, peak))
    out.update(shadow_passes(ctx, vq, torch, envk, peak))
    return out


def frame_format_passes(ctx, vq, torch, envk, peak):
    """SURVEY 8(f).2/(f).3: .hdr decode / encode at BASELINE config 5's HDRI size, skydome + ApplyReflections at 4K"""
    import time
    from vqengine_b200 import synth
    out = {}
    hw, hh = 4096, 2048
    src = torch.from_numpy(synth.hdri(hw, hh)).cuda()
    data = ctx.hdr_save_host(src)                               # warm-up (allocations, worker threads, lazy module load)
    t0 = time.perf_counter(); data = ctx.hdr_save_host(src); t_save = time.perf_counter() - t0
    info, offs = vq.hdr_parse(data)
    n = len(data)
    dfile = torch.zeros(((n + 15) // 16 * 16 + 16,), dtype=torch.uint8, device="cuda")
    dfile[:n] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    doffs = torch.from_numpy(offs.view(np.int64)).cuda()
    img = torch.empty((hh, hw, 4), dtype=torch.float32, device="cuda")
    lum = torch.zeros((1,), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: vq._check(vq.lib.vq_hdr_decode(ctx._h, dfile.data_ptr(), n, C.byref(info), doffs.data_ptr(),
                                                                vq.image_of(img), lum.data_ptr(), vq._stream_ptr(None))), 10)
    nb = n + hw * hh * 16
    out["hdr_decode_4096x2048"] = {"config": f".hdr file {n / 1e6:.1f} MB (RLE, {n / hw / hh:.2f} B/texel) -> RGBA32F + max luminance, bit-exact vs stbi_loadf",
                                   "ms": round(ms, 4), "Mtexels_per_s": round(hw * hh / ms / 1e3, 1),
                                   "algorithmic_GBps": round(nb / ms / 1e6, 1), "hbm_frac": round(nb / ms / 1e6 / peak, 3)}
    ctx.hdr_load_host(data, img)                                # warm-up
    t0 = time.perf_counter(); ctx.hdr_load_host(data, img); t_load = time.perf_counter() - t0
    out["hdr_decode_4096x2048"]["e2e_host_file_to_device_image_ms"] = round(t_load * 1e3, 2)
    ms = time_gpu(torch, lambda: ctx.hdr_encode_rgbe(src), 10)
    nb = hw * hh * 20
    out["hdr_encode_rgbe_4096x2048"] = {"ms": round(ms, 4), "algorithmic_GBps": round(nb / ms / 1e6, 1), "hbm_frac": round(nb / ms / 1e6 / peak, 3),
                                        "e2e_device_image_to_host_file_ms": round(t_save * 1e3, 2)}
    half = torch.empty((hh // 2, hw // 2, 4), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.image_resize(src, half), 10)
    nb = hw * hh * 16 + (hw // 2) * hh * 32 + (hw // 2) * (hh // 2) * 16      # read in, write + read the intermediate, write out
    out["image_resize_4096x2048_to_2048x1024"] = {"config": "stbir_resize_float (Mitchell, separable, edge clamp), bit-exact; gather tables cached in the context, horizontal taps staged in shared memory",
                                                   "ms": round(ms, 4), "algorithmic_GBps": round(nb / ms / 1e6, 1), "hbm_frac": round(nb / ms / 1e6 / peak, 3)}
    w, h = W4K, H4K
    _, inv = synth.sky_view_proj(0.7, 0.1, 1.0, w / h)
    scene = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.skydome(inv.astype(np.float32).reshape(16), envk["pyr"], scene), 10)
    out["skydome_4k"] = {"config": "every pixel background (no mask), 2048x1024 HDRI level 0", "ms": round(ms, 4),
                         "algorithmic_GBps": round(w * h * 16 / ms / 1e6, 1), "hbm_frac": round(w * h * 16 / ms / 1e6 / peak, 3)}
    refl = torch.rand((h, w, 4), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.apply_reflections(scene, refl), 10)
    out["apply_reflections_4k"] = {"ms": round(ms, 4), "algorithmic_GBps": round(w * h * 48 / ms / 1e6, 1),
                                   "hbm_frac": round(w * h * 48 / ms / 1e6 / peak, 3)}
    return out


def surface_scene_gpu(ctx, vq, torch, w, h, n_materials=4, tex_res=1024):
    """SURVEY 8(f).1 workload: n materials x up to 6 RGBA8 maps of tex_res^2 (mip chains built on the GPU by
    vq_texture_build_mips) + the three interpolant planes and the SSAO plane of a w x h frame"""
    from vqengine_b200 import synth
    mats, texs = synth.materials(n_materials, tex_res, uniform=True)
    keep, mts, tex_bytes = [], [], 0
    for t in texs:
        mt = vq.MaterialTextures()
        for slot, lvl0 in t.items():
            if lvl0 is None:
                continue
            th, tw = lvl0.shape[:2]
            levels = vq.mip_level_count(tw, th)
            buf = torch.zeros(vq.pyramid_texel_count(tw, th, levels) * 4, dtype=torch.uint8, device="cuda")
            buf[: tw * th * 4] = torch.from_numpy(lvl0.reshape(-1)).cuda()
            desc = vq.texture_of(buf, tw, th, levels)
            ctx.texture_build_mips(desc)
            setattr(mt, slot, desc)
            keep.append(buf); tex_bytes += buf.numel()
        mts.append(mt)
    table = ctx.material_table(mats, mts)
    planes = [torch.from_numpy(p).cuda() for p in synth.surface_inputs(w, h, n_materials)]
    si = vq.SurfaceInputs(vq.image_of(planes[0]), vq.image_of(planes[1]), vq.image_of(planes[2]), vq.image_of(planes[3], 1))
    return {"table": table, "inputs": si, "keep": keep + planes, "texture_bytes": tex_bytes, "n_materials": n_materials,
            "tex_res": tex_res, "mats": mats, "mts": mts}


def surface_producer_pass(ctx, vq, torch, peak):
    w, h = W4K, H4K
    sc = surface_scene_gpu(ctx, vq, torch, w, h)
    g = [torch.empty((h, w, 4), dtype=torch.float32, device="cuda") for _ in range(4)]
    gb = vq.GBuffer(*(vq.image_of(t) for t in g))
    ms = time_gpu(torch, lambda: ctx.gbuffer_from_materials(sc["inputs"], sc["table"], 0.3, gb), 10)
    # the same frame with the texel records switched off (every Sample() = 8 x LDG.32 of its own map): what the records buy
    prev = os.environ.get("VQ_SURFACE_RECORDS")
    os.environ["VQ_SURFACE_RECORDS"] = "0"
    try:
        t2 = ctx.material_table(sc["mats"], sc["mts"])
    finally:
        if prev is None: os.environ.pop("VQ_SURFACE_RECORDS", None)
        else: os.environ["VQ_SURFACE_RECORDS"] = prev
    ms_maps = time_gpu(torch, lambda: ctx.gbuffer_from_materials(sc["inputs"], t2, 0.3, gb), 10)
    t2.close()
    nbytes = w * h * (48 + 4 + 64)          # 3 float4 interpolant planes + SSAO in, 4 float4 G-buffer planes out
    out = {"surface_producer_4k": {
        "config": f"{sc['n_materials']} materials (separate maps / ORM / constants / tiled non-pow2), {sc['tex_res']}^2 RGBA8 "
                  f"maps = {sc['texture_bytes'] / 1e6:.1f} MB (L2-resident side data; materials with same-size maps sampled from 16-byte texel records), SSAO + emissive planes",
        "ms": round(ms, 4), "ms_map_by_map": round(ms_maps, 4), "Mpixels_per_s": round(w * h / ms / 1e3, 1), "algorithmic_bytes_per_px": 116,
        "algorithmic_GBps": round(nbytes / ms / 1e6, 1), "hbm_frac": round(nbytes / ms / 1e6 / peak, 3)}}
    tw = 4096
    levels = vq.mip_level_count(tw, tw)
    buf = torch.randint(0, 256, (vq.pyramid_texel_count(tw, tw, levels) * 4,), dtype=torch.uint8, device="cuda")
    desc = vq.texture_of(buf, tw, tw, levels)
    ms = time_gpu(torch, lambda: ctx.texture_build_mips(desc), 10)
    nb = tw * tw * 4 * (4 / 3 + 1 / 3)      # every level read once (except the last), every level but 0 written once
    out["texture_box_mips_4096"] = {"ms": round(ms, 4), "algorithmic_GBps": round(nb / ms / 1e6, 1),
                                    "hbm_frac": round(nb / ms / 1e6 / peak, 3), "launches": (levels - 1 + 5) // 6}
    sc["table"].close()
    return out


def shadow_passes(ctx, vq, torch, envk, peak):
    """SURVEY 8(f).4: the forward pass with shadow maps bound (1 point caster with the 20-tap cube PCF, 1 spot caster and a shadowing
    directional light with the 5x5 PCF) against the same lights unshadowed, and the MIN depth pyramid of a 4K depth buffer."""
    import numpy as np
    from vqengine_b200 import synth
    w, h = W4K, H4K
    planes = synth.gbuffer(w, h, seed=synth.SEED_BASE + 3)
    pf, pv = synth.scene_constants(w, h, envk["spec_mips"], n_point=2, n_spot=1, casters=True)
    L = pf.Lights
    m = np.zeros(16, np.float32); m[0] = 1 / 25; m[5] = 1 / 25; m[14] = 0.5; m[15] = 1.0
    for sc in range(L.numSpotCasters):
        for k in range(16): L.shadowViews[sc].m[k] = float(m[k])
    for k in range(16): L.shadowViewDirectional.m[k] = float(m[k])
    L.directional.shadowing = 1
    res_pt, res_2d = 1024, 2048
    pf.f2SpotLightShadowMapDimensions.x = pf.f2SpotLightShadowMapDimensions.y = float(res_2d)
    pf.f2DirectionalLightShadowMapDimensions.x = pf.f2DirectionalLightShadowMapDimensions.y = float(res_2d)
    dpl = [torch.from_numpy(p).cuda() for p in planes[:3]]
    gb = vq.GBuffer(vq.image_of(dpl[0]), vq.image_of(dpl[1]), vq.image_of(dpl[2]), vq.null_image())
    out = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    cubes = torch.rand((max(L.numPointCasters, 1), 6, res_pt, res_pt), device="cuda", generator=g) * 1.2
    spots = torch.rand((max(L.numSpotCasters, 1), res_2d, res_2d), device="cuda", generator=g) * 0.4 + 0.3
    dmap = torch.rand((res_2d, res_2d), device="cuda", generator=g) * 0.4 + 0.3
    ms0 = time_gpu(torch, lambda: ctx.forward_lighting(pf, pv, gb, envk["env"], out), 10)
    ms1 = time_gpu(torch, lambda: ctx.forward_lighting_shadowed(pf, pv, gb, envk["env"], out, cubes, spots, dmap), 10)
    r = {"forward_4k_casters_shadowed": {
        "ms": round(ms1, 4), "ms_same_lights_unshadowed": round(ms0, 4),
        "casters": f"{L.numPointCasters} point (20-tap cube PCF, {res_pt}^2 faces) + {L.numSpotCasters} spot + directional (5x5 PCF, {res_2d}^2)",
        "Mpixels_per_s": round(w * h / ms1 / 1e3, 1), "structure": "shadow_pcf_kernel (shadowed-tap counts per caster, 5 bits each, 8 B/pixel) + forward_kernel<SHADOWED> (caster lights weighted by 1 - taps/N)",
        "bound": "PCF kernel: instruction issue on the ALU pipe (about 50 instructions per cube tap, 6 per planar tap; 70 taps per pixel)"}}
    depth = torch.rand((h, w), device="cuda", generator=g)
    n = vq.depth_pyramid_level_count(w, h)
    levels = torch.empty((vq.depth_pyramid_texel_count(w, h, n),), dtype=torch.float32, device="cuda")
    ms = time_gpu(torch, lambda: ctx.depth_min_pyramid(depth, levels), 10)
    nb = w * h * 4 * 2 + int(w * h * 4 * (1 / 3 + 2 / 3))     # copy (read + write) + every level written once, padded level read once
    r["depth_min_pyramid_4k"] = {"ms": round(ms, 4), "levels": n, "algorithmic_GBps": round(nb / ms / 1e6, 1), "hbm_frac": round(nb / ms / 1e6 / peak, 3)}
    return r


def ibl_rows_strong_scaling(ctx, vq, torch, dist, rank, world, envk, iters=20):
    """SURVEY 8(e) rows 3-4 (optional): the diffuse-irradiance cube (BASELINE config 2 grid; the engine's step 0.010 as well) and the
    BRDF LUT strong-scaled by contiguous row blocks — every C-ABI pass takes [row_begin,row_end) — with ONE NCCL all-gather of the rows
    inside the timed region (393 KB / 8 MB: nothing worth fusing)."""
    from vqengine_b200 import distributed as vd
    out = {}
    pyr = envk["pyr"]

    def timed(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    res = 64
    rows = 6 * res
    if rows % world == 0:
        cube = torch.zeros((rows * res, 4), dtype=torch.float32, device="cuda")
        rb, re = vd.equal_tiles(rows, world)[rank]
        mine = cube[rb * res:re * res]
        for name, kw, n in (("diffuse_irradiance_config2", dict(n_phi=64, n_theta=16, src_mip=3), iters), ("diffuse_irradiance_step_0.010", dict(step=0.01, src_mip=3), 3)):
            def step():
                ctx.diffuse_irradiance(pyr, vq.cubemap_of(cube, res, 1), row_begin=rb, row_end=re, **kw)
                dist.all_gather_into_tensor(cube, mine)
            out[name] = {"ms": round(timed(step, n), 4), "rows_per_rank": re - rb}
    lut = torch.zeros((1024, 1024, 2), dtype=torch.float32, device="cuda")
    if 1024 % world == 0:
        rb, re = vd.equal_tiles(1024, world)[rank]
        mine = lut[rb:re]

        def step():
            ctx.brdf_integration_lut(lut, 2048, rb, re)
            dist.all_gather_into_tensor(lut, mine)
        out["brdf_lut_1024"] = {"ms": round(timed(step, 5), 4), "rows_per_rank": re - rb}
    out["note"] = "row blocks per rank + one NCCL all-gather per step; 1-GPU times are in the N = 1 line's `extra`"
    return out


class PeerFlags:
    """world 32-bit flag words per rank in symmetric memory + the VqPeerSignal that points at them: the rendezvous a fused
    compute+gather kernel runs in its last CTA (include/vqcuda.h). `next()` advances the epoch for one more step."""

    def __init__(self, vq, torch, dist, rank, world):
        import torch.distributed._symmetric_memory as symm
        self.t = symm.empty((world,), dtype=torch.int32, device=torch.device("cuda", torch.cuda.current_device()))
        self.hdl = symm.rendezvous(self.t, dist.group.WORLD)
        self.t.zero_(); torch.cuda.synchronize(); dist.barrier()
        self.sig = vq.PeerSignal()
        order = [rank] + [(rank + k) % world for k in range(1, world)]
        for i, r in enumerate(order):
            self.sig.flags[i] = int(self.hdl.buffer_ptrs[r])
        self.sig.n_ranks, self.sig.my_index, self.sig.epoch = world, rank, 0
        self.order = order

    def next(self):
        self.sig.epoch += 1
        return self.sig


def ibl_specular_strong_scaling(ctx, vq, torch, dist, rank, world, hdri_w=4096, hdri_h=2048, res=512, mips=9, iters=20):
    """BASELINE config 5 (IBL half): 4096x2048 HDRI -> 512^2 x6 x9-mip specular prefilter, STRONG scaling. Rank r takes block r of
    every mip whose rows divide by the world size (equal cost and equal bytes), the 2x2 mip is computed by every rank.
      fused_p2p : ONE persistent kernel per rank and step (vq_specular_prefilter_ranges): all of the rank's blocks, every texel
                  stored into all ranks' cubemaps over NVLink while the SMs integrate, the cross-rank rendezvous run by the
                  kernel's last CTA — no per-mip launches, no host-issued barrier;
      nccl      : the same single launch into the local cubemap, then pack -> ONE all_gather_into_tensor -> unpack."""
    from vqengine_b200 import synth, distributed as vd
    levels = vq.mip_level_count(hdri_w, hdri_h)
    pyr_t = torch.zeros((vq.pyramid_texel_count(hdri_w, hdri_h, levels), 4), dtype=torch.float32, device="cuda")
    pyr_t[: hdri_w * hdri_h] = torch.from_numpy(synth.hdri(hdri_w, hdri_h)).cuda().reshape(-1, 4)
    pyr = vq.pyramid_of(pyr_t, hdri_w, hdri_h, levels)
    ctx.hdri_build_mips(pyr)
    n_tex = vq.cubemap_texel_count(res, mips)
    cube_t = torch.zeros((n_tex, 4), dtype=torch.float32, device="cuda")
    cube = vq.cubemap_of(cube_t, res, mips)
    plan = vd.InterleavedSpecularPlan(res, mips, world)
    my_rows = plan.row_ranges(rank)

    def compute():
        ctx.specular_prefilter_ranges(pyr, [cube], my_rows, 512)

    def step():
        compute()
        if dist is not None and world > 1:
            plan.gather(cube_t, rank)

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        if dist: dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / iters], dtype=torch.float64, device="cuda")
        if dist: dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    ms_compute = timed(compute)
    ms = timed(step) if (dist is not None and world > 1) else ms_compute
    fused = None
    if dist is not None and world > 1:
        try:
            import torch.distributed._symmetric_memory as symm
            sym_t = symm.empty((n_tex, 4), dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
            hdl = symm.rendezvous(sym_t, dist.group.WORLD)
            flags = PeerFlags(vq, torch, dist, rank, world)
            cubes = [vq.cubemap_of(hdl.get_buffer(r, (n_tex, 4), torch.float32), res, mips) for r in flags.order]

            def fused_step():
                ctx.specular_prefilter_ranges(pyr, cubes, my_rows, 512, signal=flags.next())

            step(); fused_step(); torch.cuda.synchronize(); dist.barrier()
            same = torch.tensor([1.0 if torch.equal(sym_t, cube_t) else 0.0], device="cuda")
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
            ms_f = timed(fused_step)
            fused = {"ms": round(ms_f, 4), "texels_per_s": round(n_tex / ms_f * 1e3), "equals_nccl_allgather": bool(same.item() == 1.0),
                     "launches_per_step": 1,
                     "how": "vq_specular_prefilter_ranges: one persistent kernel per rank (device work list over the rank's blocks of every mip), every texel stored into all ranks' cubemaps (symmetric-memory peer pointers, NVLink P2P), rendezvous through peer flag words in the kernel's last CTA"}
            del sym_t
        except Exception as ex:   # symmetric memory unavailable on this box: keep the NCCL numbers
            fused = {"error": repr(ex)[:300]}
    del pyr_t, cube_t
    return {"config": f"{hdri_w}x{hdri_h} HDRI -> {res}^2 x6 x{mips} mips, 512 samples; strong scaling over {world} GPU(s): every mip split into {world} equal row blocks (tiny mips replicated); {iters} timed iterations",
            "ms": round(ms, 4), "texels_per_s": round(n_tex / ms * 1e3), "ms_compute_only": round(ms_compute, 4),
            "rows_per_rank": sum(b - a for a, b in my_rows), "replicated_mips": [m for (m, _, _, _) in plan.replicated],
            "launches_per_step_compute": 1, "fused_p2p": fused}


# ------------------------------------------------------------------------------------------------
def cpu_reference_forward(planes, rows_target_s=12.0, env=None, threads=None):
    """cpu_baseline of the GPU arm: the scalar oracle over a bounded row sample of the 4K workload. Preferred form: one process per
    host core, run in a FRESH interpreter (`bench.py --impl cpu-port`: no fork of this process, which holds a CUDA context) —
    on the pool's boxes processes scale where the threads of one process do not. Fallback: std::thread row split in this process."""
    try:
        env_ = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-port", "--steps", "4", "--warmup", "1"],
                           capture_output=True, text=True, timeout=420, env=env_)
        j = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        px = j["rows"] * j["reps"] * W4K
        return {"value": round(j["value"], 4), "unit": UNIT, "cores": j.get("effective_cores", j["procs"]), "processes": j["procs"], "kind": "port",
                "sample": f"4 x {j['reps']} x ({j['rows']} of {H4K} rows x {W4K} px of the same 4K G-buffer) = {4 * px} px at {j['ms']:.1f} ms per pass, scalar C++ "
                          f"oracle, one forked process per host core ({j['one_process_mpx_s']} Mpixels/s per process)"}
    except Exception as ex:
        print(f"# multi-process cpu_baseline unavailable ({ex!r}); using threads", file=sys.stderr)
    return _cpu_reference_forward_threads(planes, rows_target_s, env, threads)


def _cpu_reference_forward_threads(planes, rows_target_s=12.0, env=None, threads=None):
    """The scalar oracle on `threads` host threads over a bounded row sample of the 4K workload."""
    import oracle_lib as orc
    from vqengine_b200 import synth
    threads = threads or orc.cpu_threads()
    probe_rows = 16
    pf, pv = synth.scene_constants(W4K, H4K, env["spec_mips"])
    args = (env["diff"], env["diff_res"], env["spec"], env["spec_res"], env["spec_mips"], env["lut"])
    t0 = time.perf_counter()
    orc.forward_lighting(pf, pv, planes, *args, 0, probe_rows, threads)
    rate = probe_rows * W4K / (time.perf_counter() - t0)
    rows = int(min(planes[0].shape[0], max(probe_rows, rows_target_s * rate / W4K)))
    # repeat the (bounded) sample until about rows_target_s of CPU work has been timed
    t0 = time.perf_counter(); reps = 0
    while True:
        orc.forward_lighting(pf, pv, planes, *args, 0, rows, threads)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= rows_target_s or reps >= 200:
            break
    return {"value": round(reps * rows * W4K / dt / 1e6, 4), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{reps} x ({rows} of {H4K} rows x {W4K} px of the same 4K G-buffer) = {reps * rows * W4K} px in {dt:.1f} s, scalar C++ oracle, std::thread row split"}


def cpu_reference_image_class(hw=4096, hh=2048):
    """cpu_baseline for the SURVEY 8(f).2 rows, kind "reference": the engine's OWN Image class (Libs/VQUtils/Source/Image.cpp
    compiled unmodified into oracle/_ref/libvqimageref.so) timed on this box's host cores, single-threaded as in the engine —
    Image::LoadFromFile (stbi_loadf + CalculateMaxLuminance), Image::CreateResizedImage (stbir_resize_float), Image::SaveToDisk
    (stbi_write_hdr) on the same 4096x2048 HDRI the GPU rows are measured on. Returns None when the library is not present."""
    import tempfile
    import oracle_lib as orc
    from vqengine_b200 import synth
    if orc.image_ref() is None:
        return None
    src = synth.hdri(hw, hh)
    with tempfile.TemporaryDirectory() as td:
        path_in, path_out = os.path.join(td, "in.hdr"), os.path.join(td, "out.hdr")
        open(path_in, "wb").write(orc.hdr_encode(src))
        t0 = time.perf_counter(); texels, lum = orc.ref_image_load(path_in); t_load = time.perf_counter() - t0
        if texels is None:
            return None
        t0 = time.perf_counter(); half = orc.ref_image_resize(texels, hw // 2, hh // 2); t_resize = time.perf_counter() - t0
        t0 = time.perf_counter(); ok = orc.ref_image_save(path_out, texels); t_save = time.perf_counter() - t0
        if not ok:
            return None
    return {"kind": "reference", "cores": 1, "unit": "ms",
            "sample": f"one {hw}x{hh} equirect HDRI through the reference's Image class (oracle/_ref/libvqimageref.so), file on tmpfs/disk cache",
            "image_load_from_file_ms": round(t_load * 1e3, 1), "image_create_resized_half_ms": round(t_resize * 1e3, 1),
            "image_save_to_disk_ms": round(t_save * 1e3, 1)}


def _nolib():
    """vqengine_b200's synthetic inputs + ctypes struct mirror WITHOUT libvqcuda.so: the CPU arms (`--impl reference`,
    `--impl cpu-port`) must not load the product. The two plain-data modules are imported under an alias package whose
    __init__ never runs."""
    import importlib
    import types
    name = "vqengine_b200_nolib"
    if name not in sys.modules:
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(ROOT, "vqengine_b200")]
        sys.modules[name] = pkg
    return importlib.import_module(name + ".synth")


_ENV_JOB = {}


def _env_rows_worker(job):
    import oracle_lib as orc
    kind, a, b, n = job
    j = _ENV_JOB
    if kind == "spec":
        return a, b, orc.specular_prefilter(j["pyr"], j["hw"], j["hh"], j["levels"], j["spec_res"], j["spec_mips"], n, a, b, 1)
    return a, b, orc.brdf_integration_lut(j["lut"], j["lut"], 2048, a, b, 1)[a:b]


def cpu_env(hdri_w=2048, hdri_h=1024, diff_res=64, spec_res=512, spec_mips=9, lut=1024):
    """The forward pass's IBL inputs for the CPU arms at the SAME sizes as the GPU arm's (64^2 diffuse, 512^2 x 9 specular, 1024^2
    LUT from the same seeded 2048x1024 HDRI), built by the ORACLE on the host cores (untimed set-up; one forked process per
    core, cached in the temp dir for the other CPU arm of the same box). Mip 0 of the specular cube (roughness 0: every one of the
    512 samples is the same direction) is built with one sample per texel — the same texels up to the rounding of the replayed
    sums — which keeps the set-up to tens of seconds."""
    import multiprocessing as mp
    import tempfile
    import numpy as np
    import oracle_lib as orc
    synth = _nolib()
    if os.environ.get("VQ_CPU_ENV_SMALL"):                    # the CPU test-suite's hook: same code path, toy sizes
        hdri_w, hdri_h, diff_res, spec_res, spec_mips, lut = 256, 128, 16, 64, 6, 64
    cache = os.path.join(tempfile.gettempdir(), f"vq_cpu_env_{hdri_w}x{hdri_h}_{diff_res}_{spec_res}x{spec_mips}_{lut}.npz")
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return dict(diff=z["diff"], diff_res=diff_res, spec=z["spec"], spec_res=spec_res, spec_mips=spec_mips, lut=z["lut"])
        except Exception:
            pass
    t0 = time.perf_counter()
    levels = orc.lib().orc_mip_level_count(hdri_w, hdri_h)
    pyr = orc.hdri_build_mips(synth.hdri(hdri_w, hdri_h), levels)
    diff = orc.diffuse_irradiance(pyr, hdri_w, hdri_h, levels, diff_res, n_phi=64, n_theta=16, src_mip=3)
    faces = diff.reshape(6, diff_res, diff_res, 4)
    diff = np.ascontiguousarray(np.stack([orc.gaussian_blur(orc.gaussian_blur(f, False), True) for f in faces]).reshape(-1, 4))
    _ENV_JOB.update(pyr=pyr, hw=hdri_w, hh=hdri_h, levels=levels, spec_res=spec_res, spec_mips=spec_mips, lut=lut)
    procs = orc.cpu_threads()
    rows0 = 6 * spec_res
    total_rows = int(orc.lib().orc_cubemap_row_count(spec_res, spec_mips))
    jobs = [("spec", a, min(a + 64, rows0), 1) for a in range(0, rows0, 64)]                       # mip 0, one sample
    jobs += [("spec", a, min(a + 8, total_rows), 512) for a in range(rows0, total_rows, 8)]         # mips 1.., 512 samples
    jobs += [("lut", a, min(a + 8, lut), 0) for a in range(0, lut, 8)]
    spec = np.zeros((int(orc.lib().orc_cubemap_texel_count(spec_res, spec_mips)), 4), np.float32)
    lut_img = np.zeros((lut, lut, 2), np.float32)
    row_tex = [0]
    for m in range(spec_mips):
        n = spec_res >> m
        row_tex += [row_tex[-1] + n * (k + 1) - n * k for k in range(6 * n)]
    with mp.get_context("fork").Pool(procs) as pool:
        for kind, a, b, r in pool.imap_unordered(_env_rows_worker_tagged, jobs, chunksize=1):
            if kind == "spec":
                spec[row_tex[a]:row_tex[b]] = r[row_tex[a]:row_tex[b]]
            else:
                lut_img[a:b] = r
    try:
        np.savez(cache, diff=diff, spec=spec, lut=lut_img)
    except Exception:
        pass
    print(f"# cpu_env: full-size IBL maps built by the oracle in {time.perf_counter() - t0:.1f} s on {procs} processes", file=sys.stderr)
    return dict(diff=diff, diff_res=diff_res, spec=spec, spec_res=spec_res, spec_mips=spec_mips, lut=lut_img)


def _env_rows_worker_tagged(job):
    a, b, r = _env_rows_worker(job)
    return job[0], a, b, r


_REF_JOB = {}


def _cpu_rows_worker(job):
    """forked worker: rows [rb,re) of the band, `reps` times over, through the reference's shader text compiled as C++ ('text') or the
    scalar port ('port')"""
    import oracle_lib as orc
    j = _REF_JOB
    rb, re, reps = job
    acc = 0.0
    for _ in range(reps):
        if j["kind"] == "text":
            orc.hlsl_forward_gbuffer(j["pf"], j["pv"], j["planes"], *j["env"], row_begin=rb, row_end=re, out=j["out"])
            acc += float(j["out"][rb:re, :, :3].sum())
        else:
            acc += float(orc.forward_lighting(j["pf"], j["pv"], j["planes"], *j["env"], rb, re, 1, out=j["out"])[rb:re, :, :3].sum())
    return acc


def _cpu_arm(kind, steps, warmup, planes, pf, pv, a, budget_s=60.0):
    """`kind` over a bounded band of the 4K G-buffer, one FORKED PROCESS per host core (the compiled shader's cbuffers are process
    globals; and processes were measured to scale where threads of one process did not). A step = the whole band `reps` times,
    every process shading its own rows, `reps` sized from a probe so that a step lasts about budget_s / (steps + warmup) seconds
    (long enough for the task hand-off not to matter). Returns dict(value Mpx/s, ms, rows, reps, procs, one_process_mpx_s)."""
    import multiprocessing as mp
    import numpy as np
    import oracle_lib as orc
    procs = orc.cpu_threads()
    band = planes[0].shape[0]
    budget_s = float(os.environ.get("VQ_CPU_ARM_BUDGET_S", budget_s))     # tests shorten it
    _REF_JOB.update(kind=kind, pf=pf, pv=pv, planes=planes, env=a, out=np.zeros((band, W4K, 4), np.float32))
    t0 = time.perf_counter()
    _cpu_rows_worker((0, 4, 1))
    one = 4 * W4K / (time.perf_counter() - t0)                           # px/s of one process
    n = min(procs, band)
    cuts = [(band * i // n, band * (i + 1) // n) for i in range(n)]
    with mp.get_context("fork").Pool(procs) as pool:
        def step(reps):
            return sum(pool.map(_cpu_rows_worker, [(rb, re, reps) for rb, re in cuts], chunksize=1))
        step(1)                                                           # first touch of every process's pages
        t0 = time.perf_counter(); step(1); dt = time.perf_counter() - t0
        rate = band * W4K / dt                                            # measured parallel rate (a box may grant fewer CPUs than it lists)
        reps = int(max(1, round(budget_s / (steps + warmup) * rate / (band * W4K))))
        for _ in range(warmup):
            step(reps)
        t0 = time.perf_counter()
        work = 0.0
        for _ in range(steps):
            work += step(reps)
        dt = (time.perf_counter() - t0) / steps
    assert work != 0.0
    value = band * reps * W4K / dt / 1e6
    # a box may grant far fewer CPUs than it lists (round 1: 20 vs 106 Mpixels/s on two "128-core" boxes): report what the
    # run actually got, in units of one process's rate
    return {"value": value, "ms": dt * 1e3, "rows": band, "reps": reps, "procs": procs,
            "one_process_mpx_s": round(one / 1e6, 3), "effective_cores": round(value / (one / 1e6), 1)}


def _cpu_workload():
    synth = _nolib()
    env = cpu_env()
    planes = synth.gbuffer(W4K, 512, seed=synth.SEED_BASE + 3)   # a 512-row band of the 4K G-buffer
    pf, pv = synth.scene_constants(W4K, H4K, env["spec_mips"])
    a = (env["diff"], env["diff_res"], env["spec"], env["spec_res"], env["spec_mips"], env["lut"])
    return planes, pf, pv, a


def run_cpu_port(args):
    """hidden helper (`--impl cpu-port`): the scalar port, one process per core, as one JSON line. The GPU arm runs this in a fresh
    interpreter for its cpu_baseline leg (no fork of a process that holds a CUDA context)."""
    planes, pf, pv, a = _cpu_workload()
    r = _cpu_arm("port", args.steps, args.warmup, planes, pf, pv, a, budget_s=15.0)
    print(json.dumps({"impl": "cpu-port", **{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()}}))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import oracle_lib as orc
    planes, pf, pv, a = _cpu_workload()
    port = text = None
    try:
        port = _cpu_arm("port", args.steps, args.warmup, planes, pf, pv, a, budget_s=10.0)
    except Exception as ex:
        print(f"# multi-process port unavailable ({ex!r})", file=sys.stderr)
    try:
        if orc.hlsl_ref() is not None:
            # agreement with the port on a few rows (PSMain renormalises the interpolated normal; the G-buffer pass takes it as is)
            chk = orc.hlsl_forward_gbuffer(pf, pv, planes, *a, row_begin=0, row_end=2)[:2]
            want = orc.forward_lighting(pf, pv, planes, *a, 0, 2, 1)[:2]
            rel = float(np.max(np.abs(chk - want) / np.maximum(1.0, np.abs(want))))
            text = _cpu_arm("text", args.steps, args.warmup, planes, pf, pv, a)
            text["max_scaled_delta_vs_port"] = rel
    except Exception as ex:                                        # library missing / fork unavailable: time the port instead
        print(f"# reference shader text arm unavailable ({ex!r}); timing the CPU port", file=sys.stderr)
    port_note = (f"the scalar C++ port of the same math on the same box: {port['value']:.2f} Mpixels/s ({port['procs']} processes, "
                 f"{port['one_process_mpx_s']} per process)") if port else "scalar port not timed"
    if text is not None:
        v, ms, kind, cores = text["value"], text["ms"], "reference", text["effective_cores"]
        sample = (f"each step = {text['reps']} x ({text['rows']} rows x {W4K} px of the 4K G-buffer) through the reference's own ForwardLighting.hlsl PSMain "
                  f"(+ Lighting/BRDF/ShadingMath.hlsl) compiled as C++ (oracle/_ref/libhlslref.so), {text['procs']} forked processes = {cores} effective cores "
                  f"({text['one_process_mpx_s']} Mpixels/s per process); texture fetches served by the oracle's samplers; max scaled "
                  f"|delta| vs the port {text['max_scaled_delta_vs_port']:.1e}; {port_note}")
        note = "the reference's D3D12/HLSL path needs Windows; this arm runs its shader text compiled for the CPU"
    else:
        threads = orc.cpu_threads()
        if port is None:                                           # last resort: threads of this process
            t0 = time.perf_counter(); orc.forward_lighting(pf, pv, planes, *a, 0, 16, threads)
            rate = 16 * W4K / (time.perf_counter() - t0)
            rows = int(min(512, max(16, 60.0 * rate / W4K / (args.steps + args.warmup))))
            for _ in range(args.warmup):
                orc.forward_lighting(pf, pv, planes, *a, 0, rows, threads)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                orc.forward_lighting(pf, pv, planes, *a, 0, rows, threads)
            dt = (time.perf_counter() - t0) / args.steps
            port = {"value": rows * W4K / dt / 1e6, "ms": dt * 1e3, "rows": rows, "procs": threads}
        v, ms, kind, cores = port["value"], port["ms"], "port", port.get("effective_cores", port["procs"])
        sample = f"each step = {port.get('reps', 1)} x ({port['rows']} rows x {W4K} px of the 4K G-buffer) through the scalar C++ oracle on {cores} host cores"
        note = "the reference's D3D12/HLSL path needs Windows; this arm is the CPU port (oracle) of the identical math"
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": WORKLOAD, "frame": f"{W4K}x{H4K}", "note": note,
                                 "sample": "a 512-row band of the 4K G-buffer per step (bounded CPU sample); IBL maps at the GPU arm's sizes"},
                      "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
                      "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0,
                      "product_library_loaded": any("libvqcuda" in l for l in open("/proc/self/maps")) if os.path.exists("/proc/self/maps") else None}))


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu-port"])
    ap.add_argument("--no-extra", action="store_true", help="skip the per-kernel extra section")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed seeded sample of the frame the last "
                    "step computed to DIR/*.npy (inputs are seeded: two builds can be compared output for output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's frame: it needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "cpu-port":
        return run_cpu_port(args)

    import numpy as np
    import torch
    import vqengine_b200 as vq
    from vqengine_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the product has no CPU path"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    peak, peak_src = hbm_peak()
    numa = pin_to_gpu_numa_node(torch, local)
    ctx = vq.Context(local)
    envk = build_env_maps_gpu(ctx, vq, torch)

    # ---- the workload: N = 1 the metric's 4K frame; N > 1 config 5's 8K frame cut into `world` row tiles (strong scaling) ----
    FW, FH = (W4K, H4K) if world == 1 else (W8K, H8K)
    rb, re = (FH * rank) // world, (FH * (rank + 1)) // world
    rows = re - rb
    planes = synth.gbuffer(FW, rows, seed=synth.SEED_BASE + 3 + rank)        # this rank's rows of the frame's G-buffer
    pf, pv = synth.scene_constants(FW, FH, envk["spec_mips"])
    dpl = [torch.from_numpy(p).cuda() for p in planes]
    gb = vq.GBuffer(vq.image_of(dpl[0]), vq.image_of(dpl[1]), vq.image_of(dpl[2]), vq.null_image())
    out = torch.zeros((rows, FW, 4), dtype=torch.float32, device="cuda")
    kernel_only = lambda: ctx.forward_lighting(pf, pv, gb, envk["env"], out)
    frame = full = flags = None
    fused_note = None
    if world > 1:
        import torch.distributed._symmetric_memory as symm
        frame = symm.empty((FH, FW, 4), dtype=torch.float32, device=torch.device("cuda", local))   # every rank holds the assembled frame
        hdl = symm.rendezvous(frame, dist.group.WORLD)
        frame.zero_(); torch.cuda.synchronize(); dist.barrier()
        flags = PeerFlags(vq, torch, dist, rank, world)
        # local frame first, then the peers in a rotated order so that the ranks do not all write to the same peer at once
        imgs = [vq.Image(int(hdl.buffer_ptrs[r]), FW, FH, FW * 16) for r in flags.order]
        step = lambda: ctx.forward_lighting_multi(pf, pv, gb, envk["env"], imgs, rb, signal=flags.next())
        fused_note = ("vq_forward_lighting_multi_signal: ONE kernel per rank shades its rows, stores every pixel into every rank's frame "
                      "(symmetric-memory peer pointers, NVLink P2P) and runs the cross-rank rendezvous in its last CTA")
    else:
        step = kernel_only

    def timed(fn, n):
        """n launches of fn between barriers; device time, max over ranks -> ms per launch"""
        torch.cuda.synchronize()
        if dist: dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if dist: dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist: dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    # what the caller of the timed step receives: the lit frame (at N > 1 the assembled frame every rank holds)
    dump_idx = dump_sample_index(torch, out if world == 1 else frame) if args.dump_outputs and rank == 0 else None
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local); sampler.start()
    time.sleep(0.15)
    lt0 = vq.launch_count()
    ms_step = timed(step, args.steps)
    timed_launches = vq.launch_count() - lt0
    # gathered on the stream right behind the last timed step, before the clock tail below overwrites `out`
    dump_px = (out if world == 1 else frame).reshape(-1, 4)[dump_idx] if dump_idx is not None else None
    # keep the GPU busy a little longer so that the clock sampler sees the load even for short runs
    t_end = time.time() + 0.4
    while time.time() < t_end:
        kernel_only()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if dump_px is not None:
        write_dump(args.dump_outputs, dump_idx, dump_px)
        del dump_px
    px_all = FW * FH
    value = px_all / ms_step / 1e3   # Mpixels/s
    ms_kernel = timed(kernel_only, args.steps) if world > 1 else ms_step

    # ---- e2e: the blocking host-buffer call on this rank's tile, pinned host memory, H2D + D2H inside the timed region ----
    hpl = [torch.from_numpy(p).pin_memory() for p in planes]
    hgb = vq.GBuffer(vq.image_of(hpl[0]), vq.image_of(hpl[1]), vq.image_of(hpl[2]), vq.null_image())
    hout = torch.zeros((rows, FW, 4), dtype=torch.float32).pin_memory()
    ctx.resize(FW, rows)
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        ctx.forward_lighting_host(pf, pv, hgb, envk["env"], hout)
    torch.cuda.synchronize()
    if dist: dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.forward_lighting_host(pf, pv, hgb, envk["env"], hout)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / e2e_steps
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if dist: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = px_all / float(t.item()) / 1e6
    kernel_only(); torch.cuda.synchronize()
    assert torch.equal(hout.cuda(), out), "host-buffer path and device path disagree"
    h2d, d2h = 3 * FW * rows * 16, FW * rows * 16
    # what the link itself does on this box with the same pinned buffers: plain copies of one plane, each direction alone and both
    # at once — the floor of the e2e step is max(h2d_bytes / h2d rate, d2h_bytes / d2h rate) with the two directions overlapped
    pcie = None
    try:
        dbuf = torch.empty_like(out)
        s2 = torch.cuda.Stream()
        def link(fn, reps=4):
            fn(); torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps): fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / reps
        nbytes = dbuf.numel() * 4
        t_up = link(lambda: dbuf.copy_(hpl[0], non_blocking=True))
        t_dn = link(lambda: hout.copy_(dbuf, non_blocking=True))
        dbuf2 = torch.empty_like(out)
        def both():
            dbuf.copy_(hpl[0], non_blocking=True)
            with torch.cuda.stream(s2): hout.copy_(dbuf2, non_blocking=True)
        t_both = link(both)
        up, dn = nbytes / t_up / 1e9, nbytes / t_dn / 1e9
        floor_s = max(h2d / (up * 1e9), d2h / (dn * 1e9))
        pcie = {"h2d_GBps": round(up, 1), "d2h_GBps": round(dn, 1), "both_directions_GBps_each": round(nbytes / t_both / 1e9, 1),
                "link_floor_ms_per_step": round(floor_s * 1e3, 3), "e2e_ms_per_step": round(float(t.item()) * 1e3, 3),
                "e2e_frac_of_link_floor": round(floor_s / float(t.item()), 3)}
        del dbuf, dbuf2
    except Exception as ex:          # a side measurement: never let it cost the bench line
        pcie = {"error": repr(ex)[:200]}

    # ---- multi-GPU: the NCCL baseline of the same step (kernel, then one all-gather of the tiles) and the identity check ----
    gather = None
    if dist:
        full = torch.empty((FH, FW, 4), dtype=torch.float32, device="cuda")
        nccl_step = lambda: (kernel_only(), dist.all_gather_into_tensor(full, out))
        for _ in range(2):
            nccl_step()
        ms_nccl = timed(nccl_step, max(5, args.steps // 2))
        step(); nccl_step(); torch.cuda.synchronize(); dist.barrier()
        same = torch.tensor([1.0 if torch.equal(frame, full) else 0.0], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        ingress = (world - 1) * (FH // world) * FW * 16
        gather = {"fused_p2p": {"ms_per_step": round(ms_step, 5), "value": round(value, 1), "equals_nccl_allgather": bool(same.item() == 1.0),
                                "nvlink_ingress_bytes_per_rank": ingress, "nvlink_ingress_GBps_per_rank": round(ingress / ms_step / 1e6, 1),
                                "nvlink_nominal_GBps_per_direction": 900, "how": fused_note},
                  "nccl_allgather": {"ms_per_step": round(ms_nccl, 5), "value": round(px_all / ms_nccl / 1e3, 1)},
                  "kernel_only": {"ms_per_step": round(ms_kernel, 5), "value": round(px_all / ms_kernel / 1e3, 1),
                                  "note": "the rank's rows shaded into a local tile, no assembly: what round 1 reported as `value`"}}
        del full, frame
        full = frame = None

    line = None
    if rank == 0:
        # the dominant kernel, timed alone on this rank's rows (at N = 1 that is the step itself)
        achieved = BYTES_PER_PX * FW * rows / (ms_kernel * 1e-3) / 1e9
        traffic, winst, cap = forward_profile_facts()
        issue = None
        if winst and clocks.get("sm_mhz"):
            # issue-slot roofline: warp-instructions per 4K launch (ncu) / (SMs x 4 schedulers x SM clock under load)
            sm_count = torch.cuda.get_device_properties(local).multi_processor_count
            floor_ms = winst / (sm_count * 4 * clocks["sm_mhz"] * 1e6) * 1e3
            ms_4k = ms_kernel * (W4K * H4K) / (FW * rows)
            issue = {"warp_instructions_per_4k_launch": winst, "issue_floor_ms_4k": round(floor_ms, 4),
                     "frac_of_issue_floor": round(floor_ms / ms_4k, 4), "note": "one instruction per scheduler and cycle; " + str(cap)}
        if world == 1:
            cfg = {"workload": WORKLOAD, "frame": f"{FW}x{FH}", "parallelism": "1 GPU"}
        else:
            cfg = {"workload": WORKLOAD.replace("3840x2160", "7680x4320"), "frame": f"{FW}x{FH}", "rows_per_gpu": rows,
                   "parallelism": f"row-tiles x{world} (strong scaling of BASELINE config 5's frame), fused peer-store assembly + in-kernel rendezvous inside `value`",
                   "nvlink": f"every rank receives (N-1)/N x 531 MB = {(world - 1) * (FH // world) * FW * 16 / 1e6:.0f} MB per step",
                   "n1_line": "at N = 1 bench.py shades the metric's 3840x2160 frame (same kernel, same Mpixels/s unit)"}
        cfg["l2_policy"] = "inputs + output per step exceed the 126 MB L2 (4K: 398 + 133 MB); no flush needed"
        cfg["host_numa"] = numa
        line = {"metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_step, 5), "higher_is_better": True,
                "scaling": "strong" if world > 1 else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "roofline": {"bound": "hbm", "kernel": "forward_kernel", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": cap, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": BYTES_PER_PX * FW * rows, "issue": issue},
                "e2e": {"value": round(e2e_val, 1), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "vq_forward_lighting_host (pinned host buffers, 8 row chunks pipelined over 3 streams)", "pcie": pcie},
                "gpu_launches": int(timed_launches), "clocks": clocks}
        if gather: line["allgather"] = gather
    ibl_strong = None
    if not args.no_extra:
        del hpl, hout
        hpl = hout = None
        ibl_strong = ibl_specular_strong_scaling(ctx, vq, torch, dist, rank, world)
    if rank == 0 and ibl_strong is not None:
        line["ibl_specular_prefilter_strong"] = ibl_strong
    if world > 1 and not args.no_extra:
        small = ibl_rows_strong_scaling(ctx, vq, torch, dist, rank, world, envk)
        if rank == 0:
            line["ibl_rows_strong"] = small
    if world == 1 and rank == 0:
        if not args.no_extra:
            line["extra"] = extra_passes(ctx, vq, torch, envk, peak)
            line["extra"]["note"] = "per-kernel figures for the other SURVEY.md section-8 rows; not part of `value`"
        if not args.no_cpu:
            line["cpu_baseline"] = cpu_reference_forward(planes, env=cpu_env())
            try:                     # the (f).2 rows have a compilable reference: time it beside the kernels
                ref_img = cpu_reference_image_class()
                if ref_img is not None:
                    line["cpu_baseline_image_class"] = ref_img
            except Exception as ex:  # never let the side measurement cost the bench line
                line["cpu_baseline_image_class"] = {"error": repr(ex)[:200]}
    if rank == 0:
        print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
