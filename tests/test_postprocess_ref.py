"""CPU (-m "not gpu"): the reference's OWN engine-side wrappers around the FidelityFX setup — FPostProcessParameters::
FFSR1_EASU::UpdateEASUConstantBlock, FFSR1_RCAS::UpdateRCASConstantBlock / GetLinearSharpness / SetLinearSharpness
(Source/Engine/PostProcess/PostProcess.cpp:37-99 compiled unmodified into oracle/_ref/libvqppref.so) — against the product's
host-side setup (vq_fsr_easu_con / vq_fsr_rcas_con) and the C++ host mirror (vq::FPostProcessParameters)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import ref_golden as rg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pp(orc):
    if orc.pp_ref() is None:
        pytest.skip("oracle/_ref/libvqppref.so not built (no /root/reference here)")
    return orc.pp_ref()


@pytest.mark.parametrize("args", rg.EASU)
def test_easu_constant_block(pp, vq, args):
    con = (C.c_uint * 16)()
    pp.vqpp_easu(con, *[C.c_uint(a) for a in args])
    assert list(con) == list(vq.fsr_easu_con(*[float(a) for a in args])) == rg.stored("easu", args)


@pytest.mark.parametrize("stops", [0.0, 0.2, 0.5, 1.0, 2.0, 0.01])
def test_rcas_constant_block_and_sharpness_conversion(pp, vq, stops):
    con = (C.c_uint * 4)()
    pp.vqpp_rcas(con, C.c_float(stops))
    assert list(con) == list(vq.fsr_rcas_con(stops)) == rg.stored("rcas", stops)
    lin = pp.vqpp_rcas_linear_from_stops(C.c_float(stops))
    assert lin == pytest.approx(0.5 ** stops, rel=1e-6)
    if stops > 0:
        assert pp.vqpp_rcas_stops_from_linear(C.c_float(lin)) == pytest.approx(stops, rel=1e-5, abs=1e-6)


def test_host_mirror_matches_reference_wrappers(pp, tmp_path):
    """vq::FPostProcessParameters (vqengine_b200/host) fills the same blocks and converts sharpness the same way"""
    host = os.path.join(ROOT, "vqengine_b200", "host")
    if not shutil.which("g++") or not os.path.exists(os.path.join(host, "libvqhost.so")):
        pytest.skip("g++ / libvqhost.so not available")
    src = tmp_path / "pp.cpp"
    src.write_text(r'''
#include "vq_renderer.hpp"
#include <cstdio>
int main() {
    vq::FPostProcessParameters p;
    p.FSR_EASUParams.UpdateEASUConstantBlock(1478, 831, 1920, 1080, 1920, 1080);
    for (unsigned w : p.FSR_EASUParams.EASUConstantBlock) std::printf("%08x ", w);
    std::printf("\n");
    p.FSR_RCASParams.RCASSharpnessStops = 0.37f; p.FSR_RCASParams.UpdateRCASConstantBlock();
    for (unsigned w : p.FSR_RCASParams.RCASConstantBlock) std::printf("%08x ", w);
    std::printf("\n%.9g\n", p.FSR_RCASParams.GetLinearSharpness());
    p.FSR_RCASParams.SetLinearSharpness(0.3f); std::printf("%.9g\n", p.FSR_RCASParams.RCASSharpnessStops);
    return 0;
}''')
    exe = str(tmp_path / "pp")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["g++", "-std=c++17", str(src), "-I", host, "-I", os.path.join(cuda, "include"), "-L", host, "-lvqhost",
                           "-L", os.path.join(ROOT, "vqengine_b200"), "-lvqcuda", "-L", os.path.join(cuda, "lib64"), "-lcudart",
                           f"-Wl,-rpath,{host}", f"-Wl,-rpath,{os.path.join(ROOT, 'vqengine_b200')}", f"-Wl,-rpath,{os.path.join(cuda, 'lib64')}",
                           "-o", exe])
    lines = subprocess.run([exe], capture_output=True, text=True, timeout=60).stdout.split("\n")
    easu = (C.c_uint * 16)(); pp.vqpp_easu(easu, *[C.c_uint(a) for a in (1478, 831, 1920, 1080, 1920, 1080)])
    rcas = (C.c_uint * 4)(); pp.vqpp_rcas(rcas, C.c_float(0.37))
    assert lines[0].split() == [f"{w:08x}" for w in easu]
    assert lines[1].split() == [f"{w:08x}" for w in rcas]
    assert float(lines[2]) == pytest.approx(pp.vqpp_rcas_linear_from_stops(C.c_float(0.37)), rel=1e-6)
    assert float(lines[3]) == pytest.approx(pp.vqpp_rcas_stops_from_linear(C.c_float(0.3)), rel=1e-5)


@pytest.mark.parametrize("kind,case", [("easu", a) for a in rg.EASU] + [("rcas", s) for s in rg.RCAS])
def test_constant_blocks_equal_the_stored_reference(vq, kind, case):
    """vq_fsr_easu_con / vq_fsr_rcas_con == the blocks UpdateEASUConstantBlock / UpdateRCASConstantBlock filled (stored in
    tests/golden/ref_golden.json)"""
    assert rg.port(kind, case) == rg.stored(kind, case)
