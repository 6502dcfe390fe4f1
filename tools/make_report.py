"""Builds profiles/README.md from the round-2 bench JSON lines kept under profiles/ (r02_bench_{1,2,4,8}gpu.json) next to the
round-1 lines (r01_bench_*.json) they are compared with. Round 1's own report is kept as profiles/r01_README.md."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = os.path.join(ROOT, "profiles")


def load(name):
    p = os.path.join(P, name)
    if not os.path.exists(p):
        return None
    for line in reversed(open(p).read().splitlines()):
        line = line.strip()
        if line.startswith("{"):
            try:
                return json.loads(line)
            except Exception:
                pass
    return None


b = {n: load(f"r02_bench_{n}gpu.json") for n in (1, 2, 4, 8)}
old = {n: load(f"r01_bench_{n}gpu.json") for n in (1, 2, 8)}
b1 = b[1]
peak = b1["roofline"]["peak"]
out = []
out.append("# profiles/ — round-2 measurements and ncu evidence (B200, sm_100a)\n")
out.append("All numbers are CUDA-event timings from `bench.py` on `gpurun` B200 boxes (no profiler attached); the ncu files are for per-kernel "
           f"shares, DRAM traffic and stall reasons only. Roofline denominator: **measured** HBM copy bandwidth {peak:.0f} GB/s "
           "(`MEASURED_PEAKS.json`, \"of measured\"). Round 1's report: `r01_README.md`.\n")

out.append("## Headline (BASELINE.json metric: forward-PBR @4K), 1 GPU\n")
r = b1["roofline"]
o1 = old[1]
out.append("| | round 1 | round 2 |")
out.append("|---|---|---|")
out.append(f"| K1 4K step | {o1['ms_per_step']:.4f} ms, {o1['value']:.0f} Mpixels/s | **{b1['ms_per_step']:.4f} ms, {b1['value']:.0f} Mpixels/s** |")
out.append(f"| fraction of the HBM roofline (64 B/px algorithmic, of measured) | {o1['roofline']['frac']:.3f} | **{r['frac']:.3f}** |")
if r.get("issue"):
    out.append(f"| warp-instructions per 4K launch (ncu) | 234.2 M (904 per 32 pixels) | {r['issue']['warp_instructions_per_4k_launch'] / 1e6:.1f} M "
               f"({r['issue']['warp_instructions_per_4k_launch'] / (3840 * 2160 / 32):.0f} per 32 pixels); issue floor {r['issue']['issue_floor_ms_4k']:.4f} ms, "
               f"the step runs at {r['issue']['frac_of_issue_floor']:.2f} of it |")
out.append(f"| DRAM traffic per launch (ncu) vs algorithmic | 649.0 MB vs 530.8 MB | {(r.get('traffic') or 0) / 1e6:.1f} MB vs {r['algorithmic_bytes_per_launch'] / 1e6:.1f} MB |")
out.append(f"| e2e (host buffers, PCIe inside the timed region) | {o1['e2e']['value']:.0f} Mpixels/s | {b1['e2e']['value']:.0f} Mpixels/s (PCIe-bound: {(b1['e2e']['h2d_bytes_per_step'] + b1['e2e']['d2h_bytes_per_step']) / 1e6:.0f} MB per frame) |")
cb = b1.get("cpu_baseline")
if cb:
    out.append(f"\nCPU baseline (scalar C++ oracle = CPU port of the HLSL, one process per host core, IBL maps at the GPU arm's sizes): "
               f"**{cb['value']:.1f} Mpixels/s on {cb.get('processes', '?')} processes = {cb['cores']} effective cores** — {cb['sample']}.")
    out.append(f"GPU/CPU = {b1['value'] / cb['value']:.0f}x (HBM-resident), {b1['e2e']['value'] / cb['value']:.0f}x end to end. "
               "(A large ratio says nothing about kernel quality; the roofline fraction does.)\n")
out.append(f"Clocks during the timed region: {b1.get('clocks')}; host threads pinned: {b1['config'].get('host_numa')}\n")

multi = [n for n in (2, 4, 8) if b[n]]
if multi:
    out.append("## Multi-GPU: BASELINE config 5's 7680x4320 frame, strong-scaled; `value` = ONE fused kernel per rank (shade + peer-store assembly + in-kernel rendezvous)\n")
    out.append("| N | value: fused step, Mpixels/s (ms) | kernel only (no assembly) | kernel + NCCL all-gather | NVLink ingress per rank | = NCCL result | e2e Mpixels/s |")
    out.append("|---|---|---|---|---|---|---|")
    for n in multi:
        x = b[n]; a = x["allgather"]; f = a["fused_p2p"]
        out.append(f"| {n} | **{x['value']:.0f}** ({x['ms_per_step']:.3f}) | {a['kernel_only']['value']:.0f} ({a['kernel_only']['ms_per_step']:.3f}) | "
                   f"{a['nccl_allgather']['value']:.0f} ({a['nccl_allgather']['ms_per_step']:.3f}) | {f['nvlink_ingress_bytes_per_rank'] / 1e6:.0f} MB at "
                   f"{f['nvlink_ingress_GBps_per_rank']:.0f} GB/s (900 nominal) | {f['equals_nccl_allgather']} | {x['e2e']['value']:.0f} |")
    out.append("\nOne GPU shades the 4K frame at "
               f"{b1['value']:.0f} Mpixels/s; the assembled-frame throughput is bounded by NVLink ingress from N = 4 on ((N-1)/N x 531 MB must arrive at every rank).\n")

out.append("## IBL specular prefilter, strong scaling (BASELINE config 5: 4096x2048 HDRI -> 512^2 x6 x9 mips, 512 samples; target >= 6x at 8 GPUs)\n")
out.append("| N | compute only, ms | + NCCL all-gather, ms | fused peer stores + in-kernel rendezvous (ONE kernel), ms | speed-up of the fused step vs 1 GPU | = NCCL result |")
out.append("|---|---|---|---|---|---|")
base = b1["ibl_specular_prefilter_strong"]["ms"]
out.append(f"| 1 | {base:.3f} | — | — | 1.00x | — |")
for n in multi:
    s = b[n].get("ibl_specular_prefilter_strong")
    if not s:
        continue
    f = s.get("fused_p2p") or {}
    fms = f.get("ms")
    out.append(f"| {n} | {s['ms_compute_only']:.3f} | {s['ms']:.3f} ({base / s['ms']:.2f}x) | " + (f"**{fms:.3f}**" if fms else f"{f}") + " | "
               + (f"**{base / fms:.2f}x**" if fms else "—") + f" | {f.get('equals_nccl_allgather')} |")
if old[8] and "ibl_specular_prefilter_strong" in old[8]:
    so = old[8]["ibl_specular_prefilter_strong"]
    out.append(f"\nRound 1 at 8 GPUs (one launch per mip, host barrier): {so['ms']:.3f} ms with NCCL; driver's SCALE_r01: 4.97x NCCL / 5.75x fused.")

ex = b1.get("extra", {})
oex = o1.get("extra", {})
out.append("\n## Per-kernel table (1 GPU, 3840x2160 unless stated)\n")
out.append("| pass | ms | algorithmic GB/s | frac of measured HBM peak | round 1 ms | note |")
out.append("|---|---|---|---|---|---|")
out.append(f"| K1 forward PBR (4 point + 1 dir + IBL) | {b1['ms_per_step']:.4f} | {r['achieved']:.0f} | {r['frac']:.3f} | {o1['ms_per_step']:.4f} | latency-bound on its gathers: "
           "issue 56 %, L1 data pipe 55 %, FMA 45 % (r02_forward_b_summary.txt) |")
names = [("spd", "K10 SPD (11 mips)"), ("blur_x", "K5 blur X"), ("blur_y", "K5 blur Y"), ("tonemap", "K6 tonemap sRGB"), ("cas", "K7 CAS"),
         ("fsr_easu_2x", "K8 EASU 4K->8K"), ("fsr_rcas_8k", "K9 RCAS @8K"), ("post_chain_4k", "post chain total (config 4)")]
notes = {"fsr_easu_2x": "2x2 output quad per thread, packed fp32x2 (r02_post_variants.txt)",
         "tonemap": "the 133 MB output is partly still in the 126 MB L2 when the kernel retires: ~0.75 of the real DRAM traffic rate (ncu r01_post_b)",
         "blur_y": "see tonemap", "cas": "see tonemap", "fsr_rcas_8k": "see tonemap"}
for k, label in names:
    if k in ex:
        e = ex[k]
        out.append(f"| {label} | {e['ms']:.4f} | {e['algorithmic_GBps']:.0f} | {e['hbm_frac']:.3f} | {oex.get(k, {}).get('ms', '—')} | {notes.get(k, '')} |")
for k, label in [("ibl_specular_prefilter", "K3 specular prefilter"), ("ibl_diffuse_irradiance", "K2 diffuse irradiance (config 2)"),
                 ("ibl_diffuse_irradiance_reference_step", "K2 diffuse, engine step 0.010"), ("brdf_lut", "K4 BRDF LUT"), ("hdri_min_pyramid", "K11 HDRI min pyramid")]:
    if k in ex:
        e = ex[k]
        rate = f"{e.get('texels_per_s', 0):.3e} texels/s, " if "texels_per_s" in e else ""
        rate += f"{e.get('samples_per_s', 0):.3e} samples/s" if "samples_per_s" in e else (f"{e.get('algorithmic_GBps')} GB/s" if "algorithmic_GBps" in e else "")
        out.append(f"| {label} | {e['ms']:.4f} | — | — | {oex.get(k, {}).get('ms', '—')} | {e.get('config', '')}; {rate} (SFU/FP32-bound, HBM % is low by construction) |")
out.append("\n## SURVEY 8(f) rows (1 GPU)\n")
out.append("| pass | ms | algorithmic GB/s | frac of measured HBM peak | note |")
out.append("|---|---|---|---|---|")
for k, label in [("surface_producer_4k", "(f).1 surface producer 4K"), ("texture_box_mips_4096", "(f).1 RGBA8 box mips 4096^2"),
                 ("hdr_decode_4096x2048", "(f).2 .hdr decode 4096x2048"), ("hdr_encode_rgbe_4096x2048", "(f).2 RGBE encode 4096x2048"),
                 ("image_resize_4096x2048_to_2048x1024", "(f).2 Mitchell downsize 4096x2048 -> 2048x1024"),
                 ("skydome_4k", "(f).3 skydome 4K"), ("apply_reflections_4k", "(f).3 ApplyReflections 4K"), ("depth_min_pyramid_4k", "(f).4 MIN depth pyramid 4K")]:
    if k in ex:
        e = ex[k]
        note = e.get("config", "")
        for kk in ("e2e_host_file_to_device_image_ms", "e2e_device_image_to_host_file_ms"):
            if kk in e:
                note += f"; {kk} = {e[kk]}"
        out.append(f"| {label} | {e['ms']:.4f} | {e['algorithmic_GBps']:.0f} | {e['hbm_frac']:.3f} | {note} |")
if "forward_4k_casters_shadowed" in ex:
    e = ex["forward_4k_casters_shadowed"]
    out.append(f"| (f).4 forward pass with shadow maps bound 4K | {e['ms']:.4f} | — | — | {e['casters']}; the same lights unshadowed: {e['ms_same_lights_unshadowed']} ms; "
               "two launches: the PCF kernel (every decision rounded as the oracle rounds it, tap counts per caster into 8 B/pixel) + the SHADOWED instantiation of K1, which weights the caster lights with them; round 2 began at 2.26 ms with a second full-BRDF pass (r02_shadow_variants.txt) |")
ric = b1.get("cpu_baseline_image_class")
if ric and "error" not in ric:
    out.append(f"\nReference CPU path for the (f).2 rows (the engine's own `Image` class compiled unmodified, 1 host core, same 4096x2048 HDRI): "
               f"`Image::LoadFromFile` {ric['image_load_from_file_ms']} ms, `Image::CreateResizedImage` to half size {ric['image_create_resized_half_ms']} ms, "
               f"`Image::SaveToDisk` {ric['image_save_to_disk_ms']} ms.")

out.append("\n## How these were produced\n")
out.append("All on `gpurun` B200 boxes from this tree (scripts under `tools/`):\n")
out.append("* `bash tools/gpu_final.sh` — `pytest -m gpu` (-> `r02_gpu_tests.txt`), smoke, `python bench.py` (-> `r02_bench_1gpu.json`), compute-sanitizer memcheck / racecheck "
           "over one small launch of every kernel (`tools/sanitize_small.py` -> `r02_sanitize_{memcheck,racecheck}.txt`), the ncu launch list of the bench command (-> `r02_launches_bench.csv`).")
out.append("* Parity tests of one pass family, its timings for the in-tree library and for builds with other tuning constants "
           "(-> `r02_{surface,shadow,frame}_variants.txt`), one full ncu capture (-> `r02_{surface_d,surface_e,shadow_b,shadow_c,frame_b}_summary.txt`; "
           "`tools/ncu_lines.py` attributes executed instructions and stall samples to source lines); `tools/perf_e2e.py` (-> `r02_e2e_link.txt`).")
out.append("* `bash tools/gpu_2gpu.sh N` under `gpurun --gpus N` — the driver's torchrun command for `bench.py --gpus N` (-> `r02_bench_{2,4,8}gpu.json`).")
out.append("* K1 at 4K, the forward parity tests, `ncu --set full --clock-control none --import-source on -k regex:forward_kernel` "
           "over `tools/perf_forward.py` (-> `r02_forward_{a,b}_summary.txt` via `tools/ncu_summary.py`, `forward_traffic.json` via `tools/make_forward_traffic.py`); "
           "A/B logs `r02_forward_variants_{a,b,c,d}.txt`.")
out.append("* K1 + 2x EASU A/B over builds with other tuning constants (-> `r02_post_variants.txt`); `tools/ubench_gather.cu` "
           "(-> `r02_ubench_gather.txt`): what a warp-wide gather costs in the L1 data pipe.")
out.append("* `python tests/diag_fullsize.py` (-> `r02_diag_fullsize.txt`): where the first full-size parity run disagreed with the oracle, and why (DESIGN.md §5).")
out.append("* `r02_shadow_first_run.txt`, `r02_shadow_a_summary.txt`: the first execution of the (f).4 kernels (15 parity tests, timings, memcheck, ncu).")
out.append("\n## Files\n")
for f in sorted(os.listdir(P)):
    if f != "README.md":
        out.append(f"* `{f}`")
open(os.path.join(P, "README.md"), "w").write("\n".join(out) + "\n")
print("wrote profiles/README.md")
