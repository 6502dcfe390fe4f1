"""-m gpu parity: SURVEY §8(f).2 (.hdr decode / encode kernels, bit-exact) and §8(f).3 (skydome, ApplyReflections)
against the scalar oracle, through the C-ABI."""
import os

import numpy as np
import pytest
import torch

from gpu_util import dev, host, assert_abs, TOL
from test_frame_oracle import _crafted, _gold_file, _rand_image, GOLD, HEADER, HERE

pytestmark = pytest.mark.gpu


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _decode_both(ctx, orc, data):
    rc, ref, lum_ref = orc.hdr_decode(data)
    assert rc == 0
    out, lum = ctx.hdr_decode(data)
    got = host(out)
    assert got.shape == ref.shape
    assert np.array_equal(_bits(got), _bits(ref)), "decode is not bit-exact"
    assert _bits(host(lum))[0] == _bits(np.float32(lum_ref)), "max luminance differs"
    return got


@pytest.mark.parametrize("name", sorted(GOLD))
def test_decode_golden_files(ctx, orc, name):
    """files written by the reference's stbi_write_hdr, decoded bit-for-bit as its stbi_loadf does"""
    _decode_both(ctx, orc, _gold_file(name))


@pytest.mark.parametrize("w,h", [(8, 1), (9, 5), (64, 8), (127, 3), (129, 2), (1000, 4), (2048, 16), (7, 3), (1, 1), (5, 40)])
def test_decode_encoded_images(ctx, orc, w, h):
    _decode_both(ctx, orc, orc.hdr_encode(_rand_image(w, h, seed=w * 7 + h)))


@pytest.mark.parametrize("style", ["mixed", "runs_of_1", "zero_records"])
def test_decode_crafted_streams(ctx, orc, style):
    """runs of 1 double the stream (falls off the shared-memory staging path), zero-length records are no-ops"""
    data, _ = _crafted(700, 6, style, seed=17)
    _decode_both(ctx, orc, data)


def test_decode_flat_first_scanline_and_short_file(ctx, orc):
    rng = np.random.default_rng(4)
    px = rng.integers(1, 256, (3, 16, 4), dtype=np.uint8)
    px[0, 0] = (200, 100, 50, 130)
    full = HEADER + b"-Y 3 +X 16\n" + px.tobytes()
    _decode_both(ctx, orc, full)
    _decode_both(ctx, orc, full[:-37])          # flat data that ends early: missing bytes read as 0 (stbi__get8)


def test_load_host_blocking_call(ctx, orc):
    data = orc.hdr_encode(_rand_image(300, 20, seed=8))
    rc, ref, lum_ref = orc.hdr_decode(data)
    out = torch.zeros((20, 300, 4), dtype=torch.float32, device="cuda")
    lum = ctx.hdr_load_host(data, out)
    assert np.array_equal(_bits(host(out)), _bits(ref)) and np.float32(lum) == np.float32(lum_ref)


def test_decode_rejects_bad_input(ctx, vq):
    out = torch.zeros((4, 4, 4), dtype=torch.float32, device="cuda")
    with pytest.raises(vq.VqError):
        ctx.hdr_load_host(b"#?RADIANCF\nFORMAT=32-bit_rle_rgbe\n\n-Y 4 +X 4\n" + bytes(64), out)
    data = HEADER + b"-Y 4 +X 9\n" + bytes(200)
    with pytest.raises(vq.VqError):              # wrong output size
        ctx.hdr_load_host(data, out)


@pytest.mark.parametrize("w,h", [(8, 1), (64, 8), (300, 4), (7, 3), (1, 1), (1023, 5)])
def test_encode_rgbe_bit_exact(ctx, orc, w, h):
    a = _rand_image(w, h, seed=w + 3 * h)
    a[0, 0, :3] = 0.0
    if w > 2:
        a[0, 1, :3] = np.float32(5e-33)         # below the 1e-32 cut-off -> 0,0,0,0
        a[0, 2, :3] = (np.float32(1.1e-32), 0, 0)
    a[-1, -1, :3] = (3e30, 1e29, 7.0)
    got = host(ctx.hdr_encode_rgbe(dev(a)))
    assert np.array_equal(got, orc.linear_to_rgbe(a))


def test_save_host_is_byte_identical(ctx, orc):
    for w, h in [(64, 8), (7, 3), (300, 4)]:
        a = _rand_image(w, h, seed=w)
        data = ctx.hdr_save_host(dev(a))
        assert data == orc.hdr_encode(a)
        if orc.stb_ref() is not None:
            assert data == orc.hdr_encode(a, "ref")
    for name in GOLD:
        src = np.load(os.path.join(HERE, "golden", f"hdr_{name}_src.npy"))
        assert ctx.hdr_save_host(dev(src)) == _gold_file(name)


def test_round_trip_at_baseline_size(ctx, orc, vq):
    """BASELINE config 5's HDRI size (4096 x 2048), size-independent properties: decode(save(x)) is what RGBE can hold,
    a second save/decode changes nothing (idempotence), and decode(save(x)) <= x within 1/128 of the largest channel."""
    from vqengine_b200 import synth
    w, h = 4096, 2048
    x = dev(synth.hdri(w, h))
    f1 = ctx.hdr_save_host(x)
    d1, lum1 = ctx.hdr_decode(f1)
    f2 = ctx.hdr_save_host(d1)
    d2, lum2 = ctx.hdr_decode(f2)
    torch.cuda.synchronize()
    assert f1 == f2 and torch.equal(d1, d2) and torch.equal(lum1, lum2)
    assert bool((d1[..., :3] <= x[..., :3]).all())
    mx = x[..., :3].max(dim=2, keepdim=True).values
    assert bool(((x[..., :3] - d1[..., :3]) <= mx / 128.0 + 1e-30).all())
    lum = (0.2126 * d1[..., 0] + 0.7152 * d1[..., 1] + 0.0722 * d1[..., 2]).max()
    assert abs(float(lum) - float(lum1[0])) <= 1e-5 * float(lum)
    # one face-sized block against the oracle, bit for bit
    rc, ref, _ = orc.hdr_decode(f1)
    assert rc == 0 and np.array_equal(_bits(host(d1)), _bits(ref))


def _sky_setup(hw=256, hh=128, smooth=True):
    import oracle_lib as orc
    from vqengine_b200 import synth
    img = synth.smooth_hdri(hw, hh) if smooth else synth.hdri(hw, hh)
    levels = orc.lib().orc_mip_level_count(hw, hh)
    pyr = orc.hdri_build_mips(img, levels)
    return pyr, levels


@pytest.mark.parametrize("w,h,yaw,pitch,rows,masked", [
    pytest.param(96, 54, 0.0, 0.0, None, False, id="96-54-0.0-0.0"),
    pytest.param(257, 33, 1.3, -0.4, None, False, id="257-33-1.3--0.4"),
    pytest.param(64, 64, -2.6, 0.9, None, False, id="64-64--2.6-0.9"),
    pytest.param(1, 1, 0.5, 0.1, None, False, id="1-1-0.5-0.1"),
    # a thread shades rows y and y+1 of a column: odd row counts, a range starting on an odd row, a mask, one row
    pytest.param(257, 33, -0.9, 0.3, None, False, id="257-33-odd-rows"),
    pytest.param(160, 91, -0.9, 0.3, (7, 60), True, id="160-91-rows7-60-mask"),
    pytest.param(64, 1, -0.9, 0.3, None, False, id="64-1-one-row"),
    pytest.param(3840, 17, -0.9, 0.3, (2, 17), False, id="3840-17-rows2-17"),
])
def test_skydome_matches_oracle(ctx, vq, orc, w, h, yaw, pitch, rows, masked):
    """also: pixels outside the row range or under a surface in the mask keep their value, bit for bit"""
    from vqengine_b200 import synth
    hw, hh = 256, 128
    pyr, levels = _sky_setup(hw, hh)
    _, inv = synth.sky_view_proj(yaw, pitch, 1.1, w / h)
    inv32 = inv.astype(np.float32).reshape(16)
    rng = np.random.default_rng(3)
    base = rng.random((h, w, 4), dtype=np.float32)
    written = np.ones((h, w), dtype=bool)
    mask = None
    if masked:
        mask = rng.random((h, w, 4), dtype=np.float32) + 0.1
        written = rng.random((h, w)) < 0.5
        mask[written, :3] = 0.0
    r0, r1 = rows if rows else (0, h)
    written[:r0] = False; written[r1:] = False
    ref = orc.skydome(pyr, hw, hh, levels, inv32, base.copy(), normal_mask=mask, rows=rows)
    dpyr, dmask = dev(pyr), dev(mask) if masked else None    # held until the kernel has run: the descriptors do not own them
    out = dev(base)
    ctx.skydome(inv32, vq.pyramid_of(dpyr, hw, hh, levels), out, normal_mask=dmask, row_begin=r0, row_end=r1)
    got = host(out)
    assert np.array_equal(_bits(got[~written]), _bits(base[~written]))
    r = assert_abs(f"skydome{w}x{h}", got, ref)
    print(r)


def test_skydome_noisy_hdri_mask_and_rows(ctx, vq, orc):
    """the BASELINE-style HDRI (per-texel noise, peaks of 16): a single bilinear sample amplifies the 1e-7 difference
    between the kernel's polynomial atan and the oracle's libm atan2 by the texel-to-texel contrast, so the bound is
    1e-4 * max(1, local contrast) — asserted as: 99.9 % of texels within 1e-4, all within 2e-3. Also: mask, row range."""
    from vqengine_b200 import synth
    hw, hh, w, h = 512, 256, 160, 90
    pyr, levels = _sky_setup(hw, hh, smooth=False)
    _, inv = synth.sky_view_proj(0.7, 0.2, 1.2, w / h)
    inv32 = inv.astype(np.float32).reshape(16)
    rng = np.random.default_rng(1)
    mask = rng.random((h, w, 4), dtype=np.float32) + 0.1
    hole = rng.random((h, w)) < 0.4
    mask[hole, :3] = 0.0
    base = rng.random((h, w, 4), dtype=np.float32)
    ref = orc.skydome(pyr, hw, hh, levels, inv32, base.copy(), normal_mask=mask, rows=(10, 70))
    out = dev(base)
    ctx.skydome(inv32, vq.pyramid_of(dev(pyr), hw, hh, levels), out, normal_mask=dev(mask), row_begin=10, row_end=70)
    got = host(out)
    untouched = ~hole
    untouched[:10] = True; untouched[70:] = True
    assert np.array_equal(got[untouched], base[untouched])
    d = np.abs(got - ref)
    assert (d <= TOL).mean() >= 0.999 and d.max() <= 2e-3, (float((d <= TOL).mean()), float(d.max()))


@pytest.mark.parametrize("w,h,bv", [(64, 36, False), (257, 3, True), (1, 1, True), (480, 270, False)])
def test_apply_reflections_bit_exact(ctx, orc, w, h, bv):
    rng = np.random.default_rng(w + h)
    s = rng.random((h, w, 4), dtype=np.float32) * 8; r = rng.random((h, w, 4), dtype=np.float32)
    b = rng.random((h, w, 4), dtype=np.float32) if bv else None
    ref = orc.apply_reflections(s.copy(), r, b)
    ds = dev(s)
    ctx.apply_reflections(ds, dev(r), dev(b) if bv else None)
    assert np.array_equal(_bits(host(ds)), _bits(ref))


def test_frame_passes_on_pitched_images(ctx, vq, orc):
    """row pitch larger than the row (sub-rectangle of a wider allocation)"""
    rng = np.random.default_rng(3)
    w, h, wp = 50, 20, 64
    big_s = torch.from_numpy(rng.random((h, wp, 4), dtype=np.float32)).cuda()
    big_r = torch.from_numpy(rng.random((h, wp, 4), dtype=np.float32)).cuda()
    s0 = big_s.cpu().numpy().copy()
    ref = orc.apply_reflections(np.ascontiguousarray(s0[:, :w]), np.ascontiguousarray(big_r.cpu().numpy()[:, :w]))
    sv, rv = big_s[:, :w], big_r[:, :w]
    ctx.apply_reflections(sv, rv)
    got = host(big_s)
    assert np.array_equal(_bits(got[:, :w]), _bits(ref)) and np.array_equal(got[:, w:], s0[:, w:])
    a = _rand_image(w, h, seed=2)
    big = torch.zeros((h, wp, 4), dtype=torch.float32, device="cuda")
    big[:, :w] = dev(a)
    assert ctx.hdr_save_host(big[:, :w]) == orc.hdr_encode(a)


# ---- Image::CreateResizedImage (stbir_resize_float) ------------------------------------------------------------------
@pytest.mark.parametrize("w,h,ow,oh", [(64, 32, 32, 16), (100, 37, 41, 13), (33, 17, 33, 9), (16, 16, 16, 16), (128, 64, 16, 8),
                                       (50, 50, 49, 1), (257, 3, 100, 3), (9, 9, 1, 1), (1024, 512, 256, 128)])
def test_image_resize_bit_exact(ctx, orc, w, h, ow, oh):
    rng = np.random.default_rng(w * 5 + h)
    a = (rng.random((h, w, 4), dtype=np.float32) * 5).astype(np.float32)
    out = torch.zeros((oh, ow, 4), dtype=torch.float32, device="cuda")
    ctx.image_resize(dev(a), out)
    assert np.array_equal(_bits(host(out)), _bits(orc.resize_downsample(a, ow, oh)))


def test_image_resize_engine_sizes_and_errors(ctx, vq, orc):
    """the engine's case (EnvironmentMap.cpp:159-166): 2:1 equirect down by 2x / 4x; size-independent properties at
    4096x2048 -> 2048x1024 plus a bit-exact band against the oracle; upsizing is rejected"""
    from vqengine_b200 import synth
    w, h = 4096, 2048
    src = synth.hdri(w, h)
    d = dev(src)
    half = torch.zeros((h // 2, w // 2, 4), dtype=torch.float32, device="cuda")
    ctx.image_resize(d, half)
    quarter = torch.zeros((h // 4, w // 4, 4), dtype=torch.float32, device="cuda")
    ctx.image_resize(d, quarter)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(half).all()) and bool((half[..., 3] - 1.0).abs().max() <= 2e-6)     # alpha = 1 stays 1 (weights sum to 1)
    assert abs(float(half.mean()) - float(d.mean())) <= 1e-3 * float(d.mean())
    assert abs(float(quarter.mean()) - float(d.mean())) <= 1e-3 * float(d.mean())
    ref = orc.resize_downsample(src, w // 2, h // 2)
    assert np.array_equal(_bits(host(half)), _bits(ref))
    with pytest.raises(vq.VqError):
        ctx.image_resize(half, torch.zeros((h, w, 4), dtype=torch.float32, device="cuda"))
    # pitched source and destination
    big = torch.zeros((40, 96, 4), dtype=torch.float32, device="cuda"); a = _rand_image(80, 40, seed=4); big[:, :80] = dev(a)
    outb = torch.full((20, 64, 4), -3.0, dtype=torch.float32, device="cuda")
    ctx.image_resize(big[:, :80], outb[:, :40])
    got = host(outb)
    assert np.array_equal(_bits(got[:, :40]), _bits(orc.resize_downsample(a, 40, 20))) and (got[:, 40:] == -3.0).all()


def test_decode_very_wide_scanlines(ctx, orc):
    """the widest scanlines the format can run-length encode (width < 32768): 120 KB of expanded planes per block, the
    compressed bytes no longer fit next to them and are read from global memory (STAGED = false instantiation)"""
    _decode_both(ctx, orc, orc.hdr_encode(_rand_image(30000, 2, seed=12)))
    _decode_both(ctx, orc, orc.hdr_encode(_rand_image(32767, 1, seed=13)))
    a = _rand_image(32768, 1, seed=14)                 # one texel wider: stb writes (and reads) it flat
    data = orc.hdr_encode(a)
    assert len(data) > 32768 * 4
    _decode_both(ctx, orc, data)
    assert ctx.hdr_save_host(dev(a)) == data
