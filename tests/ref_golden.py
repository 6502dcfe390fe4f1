"""Stored outputs of the reference's own code (the oracle/_ref libraries built from the original engine's sources) on the cases of
tests/test_cubemap_ref.py, test_mip_ref.py, test_image_ref.py and test_postprocess_ref.py, so that those comparisons also run where
the original sources are absent. tests/golden/ref_golden.json holds them, written by tests/golden/make_ref_golden.py.

Each case has two computations: `reference(kind, key)` through the oracle/_ref library and `port(kind, key)` through the oracle or
the product. Where the library exists the live tests require both to equal the stored value; elsewhere the golden tests require
the port to. Large outputs are stored as the sha256 of their bytes."""
import hashlib
import json
import os
import tempfile

import numpy as np

import oracle_lib as orc

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.json")

CUBE_RES = [1, 2, 8, 64, 512]
MIP_HDRI = [(64, 32), (256, 128), (16, 16), (128, 2), (2048, 1024)]
MIP_RGBA8 = [(64, 64), (256, 32), (16, 2), (1024, 1024)]
IMG_LOAD = [(64, 8), (7, 3), (300, 5), (8, 1), (129, 2)]
IMG_RESIZE = [(64, 32, 32, 16), (100, 37, 41, 13), (128, 64, 16, 8), (33, 17, 33, 9)]
IMG_SAVE = [(64, 8), (7, 3), (300, 5)]
MIP_COUNT = [(2048, 1024), (4096, 2048), (4096, 4096), (512, 512), (1, 1), (3, 1000), (8192, 4096), (640, 360)]
EASU = [(1920, 1080, 1920, 1080, 3840, 2160), (1478, 831, 1920, 1080, 1920, 1080), (1280, 720, 1280, 720, 2560, 1440),
        (2227, 1253, 3840, 2160, 3840, 2160), (960, 540, 960, 540, 3840, 2160)]
RCAS = [0.0, 0.2, 0.5, 1.0, 2.0, 0.01, 0.37]


def load() -> dict:
    return json.load(open(PATH))


def sha(a) -> str:
    return hashlib.sha256(a if isinstance(a, bytes) else np.ascontiguousarray(a).tobytes()).hexdigest()


def key(*a) -> str:
    return "x".join(str(v) for v in a)


def image(w, h, seed):
    """the float RGBA test image of tests/test_image_ref.py"""
    rng = np.random.default_rng(seed)
    a = (rng.random((h, w, 4), dtype=np.float32) ** 2 * 7).astype(np.float32)
    a[:, : w // 3, :3] = np.float32(0.25)
    a[..., 3] = 1.0
    return a


def cube_points(res):
    return sorted({0, res - 1, res // 2, res // 3, (2 * res) // 3})


def rgba8(w, h):
    return np.random.default_rng(w * 7 + h).integers(0, 256, (h, w, 4), dtype=np.uint8)


def _mip_levels(img, take_level):
    """sha256 of every level after the first while both dimensions stay even (the reference indexes (x+1, y+1) unconditionally)"""
    h, w = img.shape[:2]
    out, lw, lh = [], w, h
    for l in range(1, int(orc.lib().orc_mip_level_count(w, h))):
        if lw % 2 or lh % 2:
            break
        lw, lh = lw // 2, lh // 2
        out.append(sha(take_level(l, lw, lh)))
    return out


def _ref_chain(img):
    cur = [img]
    def step(l, lw, lh):
        cur[0] = orc.ref_mip_image(cur[0])
        return cur[0]
    return step


def _file_bytes(write):
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "f.hdr")
        assert write(p)
        return open(p, "rb").read()


def port(kind, k):
    import vqengine_b200 as vq
    from vqengine_b200 import synth
    if kind == "cube_dirs":
        d = np.zeros(3, np.float32)
        out = []
        for face in range(6):
            for py in cube_points(k):
                for px in cube_points(k):
                    orc.lib().orc_cube_texel_direction(face, px, py, k, orc._p(d))
                    out.append([f"{int(v):08x}" for v in (d + np.float32(0)).view(np.uint32)])
        return out
    if kind == "mip_hdri":
        w, h = k
        pyr = orc.hdri_build_mips(synth.hdri(w, h), vq.mip_level_count(w, h))
        return _mip_levels(synth.hdri(w, h), lambda l, lw, lh: pyr[vq.pyramid_offset(w, h, l):][: lw * lh])
    if kind == "mip_rgba8":
        w, h = k
        chain = orc.texture_mip_chain(rgba8(w, h), vq.mip_level_count(w, h))
        return _mip_levels(rgba8(w, h), lambda l, lw, lh: chain[vq.pyramid_offset(w, h, l) * 4:][: lw * lh * 4])
    if kind == "image_load":
        w, h = k
        rc, texels, lum = orc.hdr_decode(orc.hdr_encode(image(w, h, w + h)))
        assert rc == 0
        return {"texels": sha(texels), "max_luminance": f"{int(np.float32(lum).view(np.uint32)):08x}"}
    if kind == "image_resize":
        w, h, ow, oh = k
        return sha(orc.resize_downsample(image(w, h, w * 3 + h), ow, oh))
    if kind == "image_save":
        w, h = k
        return sha(orc.hdr_encode(image(w, h, 11 * w + h)))
    if kind == "mip_count":
        return int(orc.lib().orc_mip_level_count(*k))
    if kind == "downsize_flow":
        rc, dec, _ = orc.hdr_decode(orc.hdr_encode(synth.hdri(512, 256)))
        return sha(orc.hdr_encode(orc.resize_downsample(dec, 128, 64)))
    if kind == "easu":
        return [int(v) for v in vq.fsr_easu_con(*[float(a) for a in k])]
    if kind == "rcas":
        return [int(v) for v in vq.fsr_rcas_con(k)]
    raise KeyError(kind)


def reference(kind, k):
    import ctypes as C
    from vqengine_b200 import synth
    if kind == "cube_dirs":
        lib = C.CDLL(os.path.join(orc.ORACLE_DIR, "_ref", "libvqcuberef.so"))
        d = np.zeros(3, np.float32)
        out = []
        for face in range(6):
            for py in cube_points(k):
                for px in cube_points(k):
                    lib.cuberef_texel_direction(face, px, py, k, orc._p(d))
                    out.append([f"{int(v):08x}" for v in (d + np.float32(0)).view(np.uint32)])
        return out
    if kind == "mip_hdri":
        img = synth.hdri(*k)
        return _mip_levels(img, _ref_chain(img))
    if kind == "mip_rgba8":
        img = rgba8(*k)
        return _mip_levels(img, _ref_chain(img))
    if kind == "image_load":
        w, h = k
        data = orc.hdr_encode(image(w, h, w + h))
        with tempfile.TemporaryDirectory() as td:
            p = os.path.join(td, "in.hdr")
            open(p, "wb").write(data)
            texels, lum = orc.ref_image_load(p)
        return {"texels": sha(texels), "max_luminance": f"{int(np.float32(lum).view(np.uint32)):08x}"}
    if kind == "image_resize":
        w, h, ow, oh = k
        return sha(orc.ref_image_resize(image(w, h, w * 3 + h), ow, oh))
    if kind == "image_save":
        w, h = k
        return sha(_file_bytes(lambda p: orc.ref_image_save(p, image(w, h, 11 * w + h))))
    if kind == "mip_count":
        return orc.ref_mip_level_count(*k)
    if kind == "downsize_flow":
        with tempfile.TemporaryDirectory() as td:
            hi = os.path.join(td, "hi.hdr")
            open(hi, "wb").write(orc.hdr_encode(synth.hdri(512, 256)))
            texels, _ = orc.ref_image_load(hi)
        return sha(_file_bytes(lambda p: orc.ref_image_save(p, orc.ref_image_resize(texels, 128, 64))))
    if kind == "easu":
        con = (C.c_uint * 16)()
        orc.pp_ref().vqpp_easu(con, *[C.c_uint(a) for a in k])
        return list(con)
    if kind == "rcas":
        con = (C.c_uint * 4)()
        orc.pp_ref().vqpp_rcas(con, C.c_float(k))
        return list(con)
    raise KeyError(kind)


def cases():
    """(kind, case, reference library needed) for every stored value"""
    yield from (("cube_dirs", r, "libvqcuberef.so") for r in CUBE_RES)
    yield from (("mip_hdri", c, "libvqmipref.so") for c in MIP_HDRI)
    yield from (("mip_rgba8", c, "libvqmipref.so") for c in MIP_RGBA8)
    yield from (("image_load", c, "libvqimageref.so") for c in IMG_LOAD)
    yield from (("image_resize", c, "libvqimageref.so") for c in IMG_RESIZE)
    yield from (("image_save", c, "libvqimageref.so") for c in IMG_SAVE)
    yield from (("mip_count", c, "libvqimageref.so") for c in MIP_COUNT)
    yield ("downsize_flow", (512, 256), "libvqimageref.so")
    yield from (("easu", c, "libvqppref.so") for c in EASU)
    yield from (("rcas", s, "libvqppref.so") for s in RCAS)


def stored(kind, k):
    return load()[kind][key(*k) if isinstance(k, tuple) else str(k)]
