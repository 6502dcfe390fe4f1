"""CPU (-m "not gpu"): the reference's OWN VQ_DXGI_UTILS::MipImage — Source/Renderer/Resources/DXGIUtils.cpp compiled
unmodified and in place into oracle/_ref/libvqmipref.so (oracle/Makefile; <dxgiformat.h> and Engine/GPUMarker.h are generated
stand-ins) — against the oracle's restatements: the HDRI MIN pyramid (K11) and the RGBA8 box chain of material textures
((f).1), level by level over whole chains with even sizes (the reference indexes (x+1, y+1) unconditionally)."""
import numpy as np
import pytest

import ref_golden as rg


@pytest.fixture(scope="module")
def ref(orc):
    if orc.mip_ref() is None:
        pytest.skip("oracle/_ref/libvqmipref.so not built (no /root/reference here)")
    return orc


@pytest.mark.parametrize("w,h", rg.MIP_HDRI)
def test_hdri_min_pyramid_equals_reference_mip_image(ref, vq, w, h):
    """K11's oracle (MipImage_MinFilter applied down the pyramid, TextureManager.cpp:714-727) == the reference's MipImage
    applied level after level, bit for bit, for as long as both dimensions stay even"""
    from vqengine_b200 import synth
    img = synth.hdri(w, h)
    levels = vq.mip_level_count(w, h)
    pyr = ref.hdri_build_mips(img, levels)
    cur, lw, lh = img, w, h
    for l in range(1, levels):
        if lw % 2 or lh % 2:
            break
        cur = ref.ref_mip_image(cur)
        lw, lh = lw // 2, lh // 2
        off = vq.pyramid_offset(w, h, l)
        mine = pyr[off: off + lw * lh].reshape(lh, lw, 4)
        assert np.array_equal(mine.view(np.uint32), cur.view(np.uint32)), (l, lw, lh)
    assert l >= 2 or min(w, h) <= 2
    assert rg.reference("mip_hdri", (w, h)) == rg.stored("mip_hdri", (w, h))


@pytest.mark.parametrize("w,h", rg.MIP_RGBA8)
def test_rgba8_box_chain_equals_reference_mip_image(ref, vq, w, h):
    rng = np.random.default_rng(w * 7 + h)
    img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    levels = vq.mip_level_count(w, h)
    chain = ref.texture_mip_chain(img, levels)
    cur, lw, lh = img, w, h
    for l in range(1, levels):
        if lw % 2 or lh % 2:
            break
        cur = ref.ref_mip_image(cur)
        lw, lh = lw // 2, lh // 2
        off = vq.pyramid_offset(w, h, l) * 4
        mine = chain[off: off + lw * lh * 4].reshape(lh, lw, 4)
        assert np.array_equal(mine, cur), (l, lw, lh)
    assert rg.reference("mip_rgba8", (w, h)) == rg.stored("mip_rgba8", (w, h))


@pytest.mark.parametrize("kind,case", [("mip_hdri", c) for c in rg.MIP_HDRI] + [("mip_rgba8", c) for c in rg.MIP_RGBA8])
def test_mip_chains_equal_the_stored_reference(kind, case):
    """every even-sized level of the oracle's chains == the reference's MipImage output stored in tests/golden/ref_golden.json"""
    assert rg.port(kind, case) == rg.stored(kind, case)
