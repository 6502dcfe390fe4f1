"""CPU (-m "not gpu"): byte compatibility of include/vq_shader_data.h with the REFERENCE'S OWN shared CPU/GPU struct header.
Shaders/LightingConstantBufferData.h is compiled unmodified as its CPU side (VQ_CPU; <DirectXMath.h> is a stand-in with the
public XMFLOATn / XMMATRIX storage layouts, oracle/ref_shim/dxmath_shim) next to our header, and sizeof / offsetof of every
member the hot path reads are compared where VQ_REFERENCE names the engine's sources. Everywhere, our header is compared with
the reference's numbers stored in tests/golden/ref_golden.json (tests/golden/make_ref_golden.py)."""
import json
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("VQ_REFERENCE")

PAIRS = {   # reference struct -> (ours, members)
    "PointLight": ("VqPointLight", ["position", "range", "color", "brightness", "attenuation", "depthBias"]),
    "SpotLight": ("VqSpotLight", ["position", "outerConeAngle", "color", "brightness", "spotDir", "depthBias", "innerConeAngle", "range"]),
    "DirectionalLight": ("VqDirectionalLight", ["lightDirection", "brightness", "color", "depthBias", "shadowing", "enabled"]),
    "SceneLighting": ("VqSceneLighting", ["numPointLights", "numSpotLights", "numPointCasters", "numSpotCasters", "directional",
                                          "shadowViewDirectional", "point_lights", "point_casters", "spot_lights", "spot_casters", "shadowViews"]),
    "PerFrameData": ("VqPerFrameData", ["Lights", "f2PointLightShadowMapDimensions", "f2SpotLightShadowMapDimensions",
                                        "f2DirectionalLightShadowMapDimensions", "fAmbientLightingFactor", "fHDRIOffsetInRadians"]),
    "PerViewLightingData": ("VqPerViewLightingData", ["matView", "matViewToWorld", "matProjInverse", "WorldFrustumPlanes", "CameraPosition",
                                                      "MaxEnvMapLODLevels", "ScreenDimensions", "EnvironmentMapDiffuseOnlyIllumination"]),
    "MaterialData": ("VqMaterialData", ["diffuse", "alpha", "emissiveColor", "emissiveIntensity", "specular", "normalMapMipBias",
                                        "uvScaleOffset", "roughness", "metalness", "displacement", "textureConfig"]),
}


TEXCFG = [("VQ_TEXCFG_DIFFUSE", "HasDiffuseMap"), ("VQ_TEXCFG_NORMAL", "HasNormalMap"), ("VQ_TEXCFG_AO", "HasAmbientOcclusionMap"),
          ("VQ_TEXCFG_ALPHA_MASK", "HasAlphaMask"), ("VQ_TEXCFG_ROUGHNESS", "HasRoughnessMap"), ("VQ_TEXCFG_METALLIC", "HasMetallicMap"),
          ("VQ_TEXCFG_HEIGHT", "HasHeightMap"), ("VQ_TEXCFG_EMISSIVE", "HasEmissiveMap"), ("VQ_TEXCFG_ORM", "HasOcclusionRoughnessMetalnessMap")]
COUNTS = [("VQ_NUM_LIGHTS_POINT", "NUM_LIGHTS__POINT"), ("VQ_NUM_LIGHTS_SPOT", "NUM_LIGHTS__SPOT"),
          ("VQ_NUM_SHADOWING_LIGHTS_POINT", "NUM_SHADOWING_LIGHTS__POINT"), ("VQ_NUM_SHADOWING_LIGHTS_SPOT", "NUM_SHADOWING_LIGHTS__SPOT")]


def probe(tmp_path, reference=False):
    """sizeof / offsetof of every compared member, the texture-configuration bits and the array extents, read from our header
    or (reference=True) from the reference's, as {our name: value}"""
    lines = ['#include <cstddef>', '#include <cstdio>', f'#include "{"LightingConstantBufferData.h" if reference else "vq_shader_data.h"}"',
             'int main() { std::printf("{");']
    for rs, (ours, members) in PAIRS.items():
        t = f"VQ_SHADER_DATA::{rs}" if reference else ours
        lines.append(f'  std::printf("\\"{ours}\\": %zu, ", sizeof({t}));')
        lines += [f'  std::printf("\\"{ours}.{m}\\": %zu, ", offsetof({t}, {m}));' for m in members]
    for ours, fn in TEXCFG:   # the reference's decoder, as the bit mask it accepts
        v = " | ".join(f"(VQ_SHADER_DATA::{fn}(1u << {b}) ? {1 << b}u : 0u)" for b in range(9)) if reference else ours
        lines.append(f'  std::printf("\\"{ours}\\": %u, ", (unsigned)({v}));')
    for ours, theirs in COUNTS:
        lines.append(f'  std::printf("\\"{ours}\\": %d, ", (int)({theirs if reference else ours}));')
    lines += ['  std::printf("\\"end\\": 0}");', '  return 0; }']
    src = tmp_path / ("probe_ref.cpp" if reference else "probe.cpp")
    src.write_text("\n".join(lines))
    exe = str(src)[:-4]
    inc = ["-I", os.path.join(ROOT, "oracle", "ref_shim", "dxmath_shim"), "-I", os.path.join(REF, "Shaders")] if reference else []
    subprocess.check_call(["g++", "-std=c++17", "-w", str(src), *inc, "-I", os.path.join(ROOT, "include"), "-o", exe])
    d = json.loads(subprocess.run([exe], capture_output=True, text=True, timeout=60, check=True).stdout)
    del d["end"]
    return d


def test_layouts_match_the_stored_reference_numbers(tmp_path):
    if not shutil.which("g++"):
        pytest.skip("g++ not available")
    import ref_golden
    want = ref_golden.load()["struct_layout"]
    assert probe(tmp_path) == want
    assert want["VqPerFrameData"] == 7120


def test_layouts_match_the_reference_header(tmp_path):
    hdr = os.path.join(REF or "", "Shaders", "LightingConstantBufferData.h")
    if not REF or not os.path.exists(hdr) or not shutil.which("g++"):
        pytest.skip("reference header / g++ not available")
    lines = ['#include <cstddef>', '#include <cstdio>', '#include "LightingConstantBufferData.h"', '#include "vq_shader_data.h"',
             'int main() { int bad = 0;']
    for rs, (ours, members) in PAIRS.items():
        lines.append(f'  if (sizeof(VQ_SHADER_DATA::{rs}) != sizeof({ours})) {{ std::printf("sizeof {rs}: %zu vs %zu\\n", sizeof(VQ_SHADER_DATA::{rs}), sizeof({ours})); ++bad; }}')
        for m in members:
            lines.append(f'  if (offsetof(VQ_SHADER_DATA::{rs}, {m}) != offsetof({ours}, {m})) {{ std::printf("offsetof {rs}.{m}: %zu vs %zu\\n", '
                         f'offsetof(VQ_SHADER_DATA::{rs}, {m}), offsetof({ours}, {m})); ++bad; }}')
    # the texture-configuration bit field: our VQ_TEXCFG_* constants against the reference's own Has*Map() decoders, and the
    # array extents
    for ours, fn in [("VQ_TEXCFG_DIFFUSE", "HasDiffuseMap"), ("VQ_TEXCFG_NORMAL", "HasNormalMap"), ("VQ_TEXCFG_AO", "HasAmbientOcclusionMap"),
                     ("VQ_TEXCFG_ALPHA_MASK", "HasAlphaMask"), ("VQ_TEXCFG_ROUGHNESS", "HasRoughnessMap"), ("VQ_TEXCFG_METALLIC", "HasMetallicMap"),
                     ("VQ_TEXCFG_HEIGHT", "HasHeightMap"), ("VQ_TEXCFG_EMISSIVE", "HasEmissiveMap"), ("VQ_TEXCFG_ORM", "HasOcclusionRoughnessMetalnessMap")]:
        lines.append(f'  if (VQ_SHADER_DATA::{fn}({ours}) != 1 || VQ_SHADER_DATA::{fn}(0x1ff & ~{ours}) != 0) {{ std::printf("{ours} vs {fn}\\n"); ++bad; }}')
    for ours, theirs in [("VQ_NUM_LIGHTS_POINT", "NUM_LIGHTS__POINT"), ("VQ_NUM_LIGHTS_SPOT", "NUM_LIGHTS__SPOT"),
                         ("VQ_NUM_SHADOWING_LIGHTS_POINT", "NUM_SHADOWING_LIGHTS__POINT"), ("VQ_NUM_SHADOWING_LIGHTS_SPOT", "NUM_SHADOWING_LIGHTS__SPOT")]:
        lines.append(f'  if ({ours} != {theirs}) {{ std::printf("{ours} != {theirs}\\n"); ++bad; }}')
    lines += ['  std::printf("checked, %d mismatches, sizeof PerFrameData %zu\\n", bad, sizeof(VQ_SHADER_DATA::PerFrameData));', '  return bad; }']
    src = tmp_path / "layout.cpp"
    src.write_text("\n".join(lines))
    exe = str(tmp_path / "layout")
    subprocess.check_call(["g++", "-std=c++17", "-w", str(src), "-I", os.path.join(ROOT, "oracle", "ref_shim", "dxmath_shim"),
                           "-I", os.path.join(REF, "Shaders"), "-I", os.path.join(ROOT, "include"), "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    print(r.stdout)
    assert r.returncode == 0, r.stdout
    assert "0 mismatches" in r.stdout and "7120" in r.stdout
    import ref_golden
    assert probe(tmp_path, reference=True) == ref_golden.load()["struct_layout"]
