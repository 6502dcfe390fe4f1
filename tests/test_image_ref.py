"""CPU (-m "not gpu"): the reference's OWN Image class — Libs/VQUtils/Source/Image.cpp compiled unmodified and in place into
oracle/_ref/libvqimageref.so (oracle/Makefile; only the MSVC-only Log.h / utils.h are shadowed) — against the oracle:
Image::LoadFromFile (texels AND the MaxLuminance it stores), Image::CreateResizedImage, Image::SaveToDisk,
Image::CalculateMipLevelCount. This is the engine's code path end to end, one level above the stb pins."""
import os

import numpy as np
import pytest

import ref_golden as rg


@pytest.fixture(scope="module")
def ref(orc):
    if orc.image_ref() is None:
        pytest.skip("oracle/_ref/libvqimageref.so not built (no /root/reference here)")
    return orc


def _img(w, h, seed):
    rng = np.random.default_rng(seed)
    a = (rng.random((h, w, 4), dtype=np.float32) ** 2 * 7).astype(np.float32)
    a[:, : w // 3, :3] = np.float32(0.25)
    a[..., 3] = 1.0
    return a


@pytest.mark.parametrize("w,h", rg.IMG_LOAD)
def test_load_from_file_texels_and_max_luminance(ref, vq, tmp_path, w, h):
    orc = ref
    path = str(tmp_path / f"in_{w}x{h}.hdr")
    data = orc.hdr_encode(_img(w, h, w + h))
    open(path, "wb").write(data)
    texels, lum = orc.ref_image_load(path)                 # Image::LoadFromFile
    rc, mine, my_lum = orc.hdr_decode(data)
    assert rc == 0 and texels is not None
    assert np.array_equal(texels.view(np.uint32), mine.view(np.uint32))
    assert np.float32(lum) == np.float32(my_lum)           # Image::MaxLuminance == CalculateMaxLuminance restated
    assert rg.reference("image_load", (w, h)) == rg.stored("image_load", (w, h))
    info, _ = vq.hdr_parse(data)                           # the product's host parser sees the same image
    assert (info.width, info.height) == (w, h)


@pytest.mark.parametrize("w,h,ow,oh", rg.IMG_RESIZE)
def test_create_resized_image(ref, w, h, ow, oh):
    a = _img(w, h, w * 3 + h)
    assert np.array_equal(ref.ref_image_resize(a, ow, oh).view(np.uint32), ref.resize_downsample(a, ow, oh).view(np.uint32))
    assert rg.reference("image_resize", (w, h, ow, oh)) == rg.stored("image_resize", (w, h, ow, oh))


@pytest.mark.parametrize("w,h", rg.IMG_SAVE)
def test_save_to_disk_is_byte_identical(ref, vq, tmp_path, w, h):
    a = _img(w, h, 11 * w + h)
    path = str(tmp_path / "out.hdr")
    assert ref.ref_image_save(path, a)                     # Image::SaveToDisk
    data = open(path, "rb").read()
    assert data == ref.hdr_encode(a) and rg.sha(data) == rg.stored("image_save", (w, h))
    assert data == vq.hdr_pack_file(ref.linear_to_rgbe(a))  # the product's host packer on the oracle's RGBE texels


def test_calculate_mip_level_count(ref, vq):
    for w, h in rg.MIP_COUNT:
        want = ref.ref_mip_level_count(w, h)               # Image::CalculateMipLevelCount
        assert want == rg.stored("mip_count", (w, h))
        assert want == int(ref.lib().orc_mip_level_count(w, h)) == vq.mip_level_count(w, h), (w, h)


def test_engine_downsize_flow_4k_to_1k(ref, tmp_path):
    """CreateEnvironmentMapTextureFromHiResAndSaveToDisk (EnvironmentMap.cpp:142-209) through the reference's Image class:
    LoadFromFile -> CreateResizedImage -> SaveToDisk, against oracle decode -> resize -> encode: identical file"""
    from vqengine_b200 import synth
    src = synth.hdri(512, 256)
    hi = str(tmp_path / "hi.hdr"); lo = str(tmp_path / "lo.hdr")
    open(hi, "wb").write(ref.hdr_encode(src))
    texels, _ = ref.ref_image_load(hi)
    small = ref.ref_image_resize(texels, 128, 64)
    assert ref.ref_image_save(lo, small)
    rc, dec, _ = ref.hdr_decode(open(hi, "rb").read())
    assert open(lo, "rb").read() == ref.hdr_encode(ref.resize_downsample(dec, 128, 64))
    assert rg.sha(open(lo, "rb").read()) == rg.stored("downsize_flow", (512, 256))


@pytest.mark.parametrize("kind,case", [("image_load", c) for c in rg.IMG_LOAD] + [("image_resize", c) for c in rg.IMG_RESIZE]
                         + [("image_save", c) for c in rg.IMG_SAVE] + [("downsize_flow", (512, 256))])
def test_image_class_outputs_equal_the_stored_reference(kind, case):
    """LoadFromFile texels + MaxLuminance, CreateResizedImage, SaveToDisk bytes and the 4k->1k-style downsize flow of the
    reference's Image class (stored in tests/golden/ref_golden.json) == the oracle's decode / resize / encode"""
    assert rg.port(kind, case) == rg.stored(kind, case)


def test_calculate_mip_level_count_equals_the_stored_reference(orc, vq):
    for w, h in rg.MIP_COUNT:
        assert rg.stored("mip_count", (w, h)) == int(orc.lib().orc_mip_level_count(w, h)) == vq.mip_level_count(w, h), (w, h)
