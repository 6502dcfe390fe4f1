"""vqengine_b200 — B200 (sm_100a) headless shading backend for VQEngine's per-pixel passes.

The product is the C-ABI shared library ``libvqcuda.so`` (include/vqcuda.h), built in-tree from
``vqengine_b200/csrc`` by ``__graft_entry__.build()``. This Python package is only the thin ctypes
driver used by the tests and ``bench.py``: it mirrors the C structs, loads the library and turns
torch CUDA tensors into the ``{ptr, width, height, pitch}`` descriptors the ABI takes. torch is used
for device memory, streams and torch.distributed — plumbing, not compute.

There is NO CPU fallback: importing works without a GPU (so symbols/struct layouts can be checked),
but every device call fails with VQ_ERR_NO_DEVICE, and a missing library raises ImportError.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvqcuda.so")

from .shader_data import *          # noqa: F401,F403  (struct mirror + constants: plain data, no library)
from .shader_data import f32, i32, u32


# every symbol include/vqcuda.h declares (tests/test_abi.py checks the library exports all of them)
ABI_SYMBOLS = [
    "vq_ctx_create", "vq_ctx_destroy", "vq_ctx_resize", "vq_last_error", "vq_version", "vq_launch_count",
    "vq_forward_lighting", "vq_hdri_build_mips", "vq_diffuse_irradiance", "vq_specular_prefilter",
    "vq_brdf_integration_lut", "vq_gaussian_blur_x", "vq_gaussian_blur_y", "vq_tonemap", "vq_cas",
    "vq_fsr_easu", "vq_fsr_rcas", "vq_spd_downsample", "vq_fsr_easu_con", "vq_fsr_rcas_con", "vq_cas_setup",
    "vq_spd_setup", "vq_mip_level_count", "vq_cubemap_texel_count", "vq_cubemap_offset", "vq_cubemap_row_count",
    "vq_pyramid_texel_count", "vq_pyramid_offset", "vq_forward_lighting_host", "vq_environment_prepare",
    "vq_environment_invalidate", "vq_forward_lighting_multi",
    "vq_texture_build_mips", "vq_material_table_create", "vq_material_table_destroy", "vq_gbuffer_from_materials",
    "vq_hdr_parse", "vq_hdr_decode", "vq_hdr_load_host", "vq_hdr_encode_rgbe", "vq_hdr_pack_file", "vq_hdr_save_host",
    "vq_skydome", "vq_apply_reflections", "vq_specular_prefilter_multi", "vq_specular_prefilter_ranges", "vq_forward_lighting_multi_signal", "vq_image_resize", "vq_resize_axis_table",
    "vq_forward_lighting_shadowed", "vq_depth_pyramid_level_count", "vq_depth_pyramid_texel_count", "vq_depth_min_pyramid",
]


class VqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"vqcuda error {code}: {msg}")
        self.code = code


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    P = C.POINTER
    lib.vq_ctx_create.argtypes = [C.c_int, P(vp)]
    lib.vq_ctx_destroy.argtypes = [vp]
    lib.vq_ctx_resize.argtypes = [vp, C.c_int, C.c_int]
    lib.vq_last_error.restype = C.c_char_p
    lib.vq_version.restype = C.c_char_p
    lib.vq_launch_count.restype = C.c_uint64
    lib.vq_forward_lighting.argtypes = [vp, P(PerFrameData), P(PerViewLightingData), P(GBuffer), P(EnvironmentMaps),
                                        Image, C.c_int, C.c_int, vp]
    lib.vq_forward_lighting_multi.argtypes = [vp, P(PerFrameData), P(PerViewLightingData), P(GBuffer), P(EnvironmentMaps),
                                              P(Image), C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.vq_forward_lighting_multi_signal.argtypes = [vp, P(PerFrameData), P(PerViewLightingData), P(GBuffer), P(EnvironmentMaps),
                                                     P(Image), C.c_int, C.c_int, C.c_int, C.c_int, P(PeerSignal), vp]
    lib.vq_forward_lighting_host.argtypes = [vp, P(PerFrameData), P(PerViewLightingData), P(GBuffer),
                                             P(EnvironmentMaps), Image]
    lib.vq_environment_prepare.argtypes = [vp, P(EnvironmentMaps), vp]
    lib.vq_environment_invalidate.argtypes = [vp]
    lib.vq_hdri_build_mips.argtypes = [vp, Pyramid, vp]
    lib.vq_diffuse_irradiance.argtypes = [vp, P(DiffuseIrradianceParams), Pyramid, Cubemap, C.c_int, C.c_int, vp]
    lib.vq_specular_prefilter.argtypes = [vp, Pyramid, Cubemap, C.c_int, C.c_int, C.c_int, vp]
    lib.vq_specular_prefilter_multi.argtypes = [vp, Pyramid, P(Cubemap), C.c_int, C.c_int, C.c_int, C.c_int, vp]
    lib.vq_specular_prefilter_ranges.argtypes = [vp, Pyramid, P(Cubemap), C.c_int, C.c_int, P(C.c_int), C.c_int, P(PeerSignal), vp]
    lib.vq_brdf_integration_lut.argtypes = [vp, Image, C.c_int, C.c_int, C.c_int, vp]
    lib.vq_gaussian_blur_x.argtypes = [vp, P(BlurParams), Image, Image, vp]
    lib.vq_gaussian_blur_y.argtypes = [vp, P(BlurParams), Image, Image, vp]
    lib.vq_tonemap.argtypes = [vp, P(TonemapperParams), Image, Image, vp]
    lib.vq_cas.argtypes = [vp, P(u32), Image, Image, vp]
    lib.vq_fsr_easu.argtypes = [vp, P(u32), C.c_int, Image, Image, vp]
    lib.vq_fsr_rcas.argtypes = [vp, P(u32), Image, Image, vp]
    lib.vq_spd_downsample.argtypes = [vp, P(SpdConstants), Image, P(Image), vp]
    lib.vq_fsr_easu_con.argtypes = [P(u32), f32, f32, f32, f32, f32, f32]
    lib.vq_fsr_easu_con.restype = None
    lib.vq_fsr_rcas_con.argtypes = [P(u32), f32]
    lib.vq_fsr_rcas_con.restype = None
    lib.vq_cas_setup.argtypes = [P(u32), f32, f32, f32, f32, f32]
    lib.vq_cas_setup.restype = None
    lib.vq_spd_setup.argtypes = [P(u32), P(SpdConstants), P(u32), C.c_int]
    lib.vq_spd_setup.restype = None
    lib.vq_mip_level_count.argtypes = [C.c_uint64, C.c_uint64]
    lib.vq_cubemap_texel_count.argtypes = [C.c_int, C.c_int]
    lib.vq_cubemap_texel_count.restype = C.c_uint64
    lib.vq_cubemap_offset.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.vq_cubemap_offset.restype = C.c_uint64
    lib.vq_cubemap_row_count.argtypes = [C.c_int, C.c_int]
    lib.vq_pyramid_texel_count.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.vq_pyramid_texel_count.restype = C.c_uint64
    lib.vq_pyramid_offset.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.vq_pyramid_offset.restype = C.c_uint64
    lib.vq_texture_build_mips.argtypes = [vp, Texture2D, vp]
    lib.vq_material_table_create.argtypes = [vp, P(MaterialData), P(MaterialTextures), C.c_int, P(vp)]
    lib.vq_material_table_destroy.argtypes = [vp, vp]
    lib.vq_gbuffer_from_materials.argtypes = [vp, P(SurfaceInputs), vp, f32, C.c_int, P(GBuffer), C.c_int, C.c_int, vp]
    u64 = C.c_uint64
    lib.vq_hdr_parse.argtypes = [vp, u64, P(HdrInfo), P(u64)]
    lib.vq_hdr_decode.argtypes = [vp, vp, u64, P(HdrInfo), vp, Image, vp, vp]
    lib.vq_hdr_load_host.argtypes = [vp, vp, u64, Image, P(f32)]
    lib.vq_hdr_encode_rgbe.argtypes = [vp, Image, vp, vp]
    lib.vq_hdr_pack_file.argtypes = [vp, C.c_int, C.c_int, vp, u64, P(u64)]
    lib.vq_hdr_save_host.argtypes = [vp, Image, vp, u64, P(u64)]
    lib.vq_image_resize.argtypes = [vp, Image, Image, vp]
    lib.vq_resize_axis_table.argtypes = [C.c_int, C.c_int, P(C.c_int), P(C.c_int), P(f32), C.c_int, P(C.c_int)]
    lib.vq_skydome.argtypes = [vp, P(Matrix), Pyramid, P(Image), Image, C.c_int, C.c_int, vp]
    lib.vq_apply_reflections.argtypes = [vp, Image, Image, P(Image), vp]
    lib.vq_forward_lighting_shadowed.argtypes = [vp, P(PerFrameData), P(PerViewLightingData), P(GBuffer), P(EnvironmentMaps),
                                                 P(ShadowMaps), Image, C.c_int, C.c_int, vp]
    lib.vq_depth_pyramid_level_count.argtypes = [C.c_int, C.c_int]
    lib.vq_depth_pyramid_texel_count.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.vq_depth_pyramid_texel_count.restype = C.c_uint64
    lib.vq_depth_min_pyramid.argtypes = [vp, Image, vp, C.c_int, vp]
    return lib


lib = _load()


def _check(rc: int) -> None:
    if rc != VQ_OK:
        raise VqError(rc, (lib.vq_last_error() or b"").decode())


# ---- host-side helpers (no GPU needed) ---------------------------------------------------------
def fsr_easu_con(vp_w, vp_h, in_w, in_h, out_w, out_h):
    con = (u32 * 16)()
    lib.vq_fsr_easu_con(con, vp_w, vp_h, in_w, in_h, out_w, out_h)
    return con


def fsr_rcas_con(stops: float):
    con = (u32 * 4)()
    lib.vq_fsr_rcas_con(con, stops)
    return con


def cas_setup(sharpness, in_w, in_h, out_w, out_h):
    con = (u32 * 8)()
    lib.vq_cas_setup(con, sharpness, in_w, in_h, out_w, out_h)
    return con


def spd_setup(width: int, height: int, mips: int = -1, left: int = 0, top: int = 0):
    d = (u32 * 2)()
    c = SpdConstants()
    rect = (u32 * 4)(left, top, width, height)
    lib.vq_spd_setup(d, C.byref(c), rect, mips)
    return (d[0], d[1]), c


def mip_level_count(w: int, h: int) -> int:
    return lib.vq_mip_level_count(w, h)


def cubemap_texel_count(res: int, mips: int) -> int:
    return lib.vq_cubemap_texel_count(res, mips)


def cubemap_offset(res: int, mip: int, face: int) -> int:
    return lib.vq_cubemap_offset(res, mip, face)


def cubemap_row_count(res: int, mips: int) -> int:
    return lib.vq_cubemap_row_count(res, mips)


def pyramid_texel_count(w: int, h: int, levels: int) -> int:
    return lib.vq_pyramid_texel_count(w, h, levels)


def pyramid_offset(w: int, h: int, level: int) -> int:
    return lib.vq_pyramid_offset(w, h, level)


# ---- Radiance .hdr, host side (no GPU needed) ----------------------------------------------------
def hdr_parse(file_bytes: bytes):
    """-> (HdrInfo, channel_offsets numpy uint64 [4*height+1] or None for flat files). Raises VqError on a bad file."""
    import numpy as np
    buf = (C.c_uint8 * len(file_bytes)).from_buffer_copy(file_bytes)
    info = HdrInfo()
    _check(lib.vq_hdr_parse(buf, len(file_bytes), C.byref(info), None))
    if info.flat:
        return info, None
    offs = np.zeros(4 * info.height + 1, dtype=np.uint64)
    _check(lib.vq_hdr_parse(buf, len(file_bytes), C.byref(info), offs.ctypes.data_as(C.POINTER(C.c_uint64))))
    return info, (None if info.flat else offs)


def hdr_pack_file(rgbe) -> bytes:
    """[H, W, 4] uint8 RGBE texels -> the .hdr file image (host side of Image::SaveToDisk)."""
    import numpy as np
    a = np.ascontiguousarray(rgbe, dtype=np.uint8)
    h, w = a.shape[:2]
    n = C.c_uint64(0)
    _check(lib.vq_hdr_pack_file(a.ctypes.data, w, h, None, 0, C.byref(n)))
    out = np.empty(n.value, dtype=np.uint8)
    _check(lib.vq_hdr_pack_file(a.ctypes.data, w, h, out.ctypes.data, n.value, C.byref(n)))
    return out.tobytes()


def resize_axis_table(in_size: int, out_size: int):
    """-> (start int32 [out], count int32 [out], weights float32 [out, max_taps]) of one axis of vq_image_resize"""
    import numpy as np
    mt = C.c_int(0)
    _check(lib.vq_resize_axis_table(in_size, out_size, None, None, None, 0, C.byref(mt)))
    start = np.zeros(out_size, dtype=np.int32); count = np.zeros(out_size, dtype=np.int32)
    w = np.zeros((out_size, mt.value), dtype=np.float32)
    _check(lib.vq_resize_axis_table(in_size, out_size, start.ctypes.data_as(C.POINTER(C.c_int)), count.ctypes.data_as(C.POINTER(C.c_int)),
                                    w.ctypes.data_as(C.POINTER(f32)), mt.value, C.byref(mt)))
    return start, count, w


# ---- descriptors from torch tensors ------------------------------------------------------------
def depth_pyramid_level_count(w: int, h: int) -> int:
    return int(lib.vq_depth_pyramid_level_count(w, h))


def depth_pyramid_texel_count(w: int, h: int, levels: int) -> int:
    return int(lib.vq_depth_pyramid_texel_count(w, h, levels))


def image_of(t, channels: int = 4) -> Image:
    """[H, W, channels] float32 tensor (CUDA, or pinned/pageable host for the *_host calls)."""
    assert t.dim() == 3 and t.shape[2] == channels and t.dtype.is_floating_point and t.element_size() == 4
    assert t.stride(2) == 1 and t.stride(1) == channels, "rows must be dense"
    return Image(t.data_ptr(), t.shape[1], t.shape[0], t.stride(0) * 4)


def null_image() -> Image:
    return Image(None, 0, 0, 0)


def cubemap_of(t, res: int, mips: int) -> Cubemap:
    assert t.is_contiguous() and t.numel() == cubemap_texel_count(res, mips) * 4
    return Cubemap(t.data_ptr(), res, mips)


def pyramid_of(t, w: int, h: int, levels: int) -> Pyramid:
    assert t.is_contiguous() and t.numel() == pyramid_texel_count(w, h, levels) * 4
    return Pyramid(t.data_ptr(), w, h, levels)


def texture_of(t, w: int, h: int, levels: int) -> Texture2D:
    """uint8 tensor holding the packed RGBA8 mip chain of a w x h texture; None -> null SRV"""
    if t is None:
        return Texture2D(None, 0, 0, 0)
    assert t.is_contiguous() and t.element_size() == 1 and t.numel() == pyramid_texel_count(w, h, levels) * 4
    return Texture2D(t.data_ptr(), w, h, levels)


def _stream_ptr(stream) -> C.c_void_p:
    if stream is None:
        import torch
        stream = torch.cuda.current_stream()
    return C.c_void_p(stream.cuda_stream)


class Context:
    """Owns a VqContext (IRenderPass::Initialize / Destroy)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _check(lib.vq_ctx_create(device, C.byref(self._h)))
        self.device = device

    def close(self):
        if self._h:
            lib.vq_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def resize(self, w: int, h: int):
        _check(lib.vq_ctx_resize(self._h, w, h))

    # K1
    def forward_lighting(self, per_frame, per_view, gbuffer: GBuffer, env: EnvironmentMaps, out, row_begin=0,
                         row_end=None, stream=None):
        o = image_of(out)
        _check(lib.vq_forward_lighting(self._h, C.byref(per_frame), C.byref(per_view), C.byref(gbuffer), C.byref(env), o,
                                       row_begin, o.height if row_end is None else row_end, _stream_ptr(stream)))

    def forward_lighting_multi(self, per_frame, per_view, gbuffer: GBuffer, env: EnvironmentMaps, out_images, dst_row_offset,
                               row_begin=0, row_end=None, stream=None, signal: "PeerSignal" = None):
        """out_images: list of Image descriptors (local frame first, then the peers' mapped frames); signal: the in-kernel
        cross-rank rendezvous (vq_forward_lighting_multi_signal)"""
        arr = (Image * len(out_images))(*out_images)
        h = gbuffer.position_ao.height
        if signal is None:
            _check(lib.vq_forward_lighting_multi(self._h, C.byref(per_frame), C.byref(per_view), C.byref(gbuffer), C.byref(env), arr,
                                                 len(out_images), dst_row_offset, row_begin, h if row_end is None else row_end,
                                                 _stream_ptr(stream)))
        else:
            _check(lib.vq_forward_lighting_multi_signal(self._h, C.byref(per_frame), C.byref(per_view), C.byref(gbuffer), C.byref(env),
                                                        arr, len(out_images), dst_row_offset, row_begin,
                                                        h if row_end is None else row_end, C.byref(signal), _stream_ptr(stream)))

    # SURVEY 8(f).4: the pass with shadow maps bound, and the MIN depth pyramid
    def forward_lighting_shadowed(self, per_frame, per_view, gbuffer: GBuffer, env: EnvironmentMaps, out, point_cubes=None,
                                  spot_maps=None, directional_map=None, row_begin=0, row_end=None, stream=None):
        """point_cubes [casters,6,R,R], spot_maps [casters,H,W], directional_map [H,W]: contiguous float32 CUDA tensors or None"""
        sm = ShadowMaps()
        if point_cubes is not None:
            assert point_cubes.is_contiguous() and point_cubes.dim() == 4 and point_cubes.shape[1] == 6 and point_cubes.shape[2] == point_cubes.shape[3]
            sm.point_cubes, sm.point_res = point_cubes.data_ptr(), point_cubes.shape[2]
        if spot_maps is not None:
            assert spot_maps.is_contiguous() and spot_maps.dim() == 3
            sm.spot_maps, sm.spot_width, sm.spot_height = spot_maps.data_ptr(), spot_maps.shape[2], spot_maps.shape[1]
        if directional_map is not None:
            assert directional_map.is_contiguous() and directional_map.dim() == 2
            sm.directional_map, sm.directional_width, sm.directional_height = directional_map.data_ptr(), directional_map.shape[1], directional_map.shape[0]
        o = image_of(out)
        _check(lib.vq_forward_lighting_shadowed(self._h, C.byref(per_frame), C.byref(per_view), C.byref(gbuffer), C.byref(env),
                                                C.byref(sm), o, row_begin, o.height if row_end is None else row_end, _stream_ptr(stream)))

    def depth_min_pyramid(self, depth, levels_out, n_levels=None, stream=None):
        """depth: [H,W] float32 CUDA tensor (dense rows); levels_out: flat float32 CUDA tensor of depth_pyramid_texel_count floats"""
        assert depth.dim() == 2 and depth.stride(1) == 1 and depth.element_size() == 4
        h, w = depth.shape
        n = depth_pyramid_level_count(w, h) if n_levels is None else n_levels
        assert levels_out.is_contiguous() and levels_out.numel() >= depth_pyramid_texel_count(w, h, n)
        _check(lib.vq_depth_min_pyramid(self._h, Image(depth.data_ptr(), w, h, depth.stride(0) * 4), levels_out.data_ptr(), n,
                                        _stream_ptr(stream)))

    def forward_lighting_host(self, per_frame, per_view, host_gbuffer: GBuffer, env: EnvironmentMaps, host_out):
        _check(lib.vq_forward_lighting_host(self._h, C.byref(per_frame), C.byref(per_view), C.byref(host_gbuffer),
                                            C.byref(env), image_of(host_out)))

    def environment_prepare(self, env: EnvironmentMaps, stream=None):
        _check(lib.vq_environment_prepare(self._h, C.byref(env), _stream_ptr(stream)))

    def environment_invalidate(self):
        _check(lib.vq_environment_invalidate(self._h))

    # SURVEY 8(f).1: material textures -> G-buffer
    def texture_build_mips(self, tex: Texture2D, stream=None):
        _check(lib.vq_texture_build_mips(self._h, tex, _stream_ptr(stream)))

    def material_table(self, materials, textures) -> "MaterialTable":
        return MaterialTable(self, materials, textures)

    def gbuffer_from_materials(self, inputs: SurfaceInputs, table: "MaterialTable", ambient_factor: float, gbuffer: GBuffer,
                               alpha_mask: bool = False, row_begin=0, row_end=None, stream=None):
        h = inputs.position_u.height
        _check(lib.vq_gbuffer_from_materials(self._h, C.byref(inputs), table._h, ambient_factor, 1 if alpha_mask else 0,
                                             C.byref(gbuffer), row_begin, h if row_end is None else row_end,
                                             _stream_ptr(stream)))

    # SURVEY 8(f).2: Radiance .hdr
    def hdr_decode(self, file_bytes: bytes, stream=None):
        """file image (host bytes) -> ([H, W, 4] float32 CUDA tensor, 1-element max-luminance tensor); asynchronous."""
        import numpy as np
        import torch
        info, offs = hdr_parse(file_bytes)
        n = len(file_bytes)
        # uploads, the zero fill and the launch all go onto ONE stream (`stream`, default: torch's current one), so the
        # kernel is ordered after its inputs without an event
        s = stream if stream is not None else torch.cuda.current_stream()
        with torch.cuda.stream(s):
            dfile = torch.zeros(((n + 15) // 16 * 16 + 16,), dtype=torch.uint8, device=f"cuda:{self.device}")
            dfile[:n] = torch.frombuffer(bytearray(file_bytes), dtype=torch.uint8).to(dfile.device)
            doffs = torch.from_numpy(offs.view(np.int64)).to(dfile.device) if offs is not None else None
            out = torch.empty((info.height, info.width, 4), dtype=torch.float32, device=dfile.device)
            lum = torch.zeros((1,), dtype=torch.float32, device=dfile.device)
            _check(lib.vq_hdr_decode(self._h, dfile.data_ptr(), n, C.byref(info), doffs.data_ptr() if doffs is not None else None,
                                     image_of(out), lum.data_ptr(), _stream_ptr(s)))
        out._vq_keepalive = (dfile, doffs)
        return out, lum

    def hdr_load_host(self, file_bytes: bytes, out):
        """blocking vq_hdr_load_host; returns Image::MaxLuminance"""
        buf = (C.c_uint8 * len(file_bytes)).from_buffer_copy(file_bytes)
        lum = f32(0)
        _check(lib.vq_hdr_load_host(self._h, buf, len(file_bytes), image_of(out), C.byref(lum)))
        return lum.value

    def hdr_encode_rgbe(self, src, stream=None):
        """[H, W, 4] float32 CUDA tensor -> [H, W, 4] uint8 RGBE CUDA tensor"""
        import torch
        out = torch.empty(src.shape, dtype=torch.uint8, device=src.device)
        _check(lib.vq_hdr_encode_rgbe(self._h, image_of(src), out.data_ptr(), _stream_ptr(stream)))
        return out

    def hdr_save_host(self, src) -> bytes:
        """blocking vq_hdr_save_host: device image -> .hdr file image"""
        import numpy as np
        h, w = src.shape[:2]
        cap = 256 + w * h * 6 + h * 8
        out = np.empty(cap, dtype=np.uint8)
        n = C.c_uint64(0)
        _check(lib.vq_hdr_save_host(self._h, image_of(src), out.ctypes.data, cap, C.byref(n)))
        return out[:n.value].tobytes()

    def image_resize(self, src, dst, stream=None):
        """Image::CreateResizedImage (stbir_resize_float): dst is [H', W', 4] with H' <= H, W' <= W"""
        _check(lib.vq_image_resize(self._h, image_of(src), image_of(dst), _stream_ptr(stream)))

    # SURVEY 8(f).3: skydome + reflection composite
    def skydome(self, inv_view_proj, pyr: Pyramid, scene, normal_mask=None, row_begin=0, row_end=None, stream=None):
        m = Matrix((f32 * 16)(*[float(x) for x in inv_view_proj]))
        o = image_of(scene)
        mask = image_of(normal_mask) if normal_mask is not None else None
        _check(lib.vq_skydome(self._h, C.byref(m), pyr, C.byref(mask) if mask is not None else None, o, row_begin,
                              o.height if row_end is None else row_end, _stream_ptr(stream)))

    def apply_reflections(self, scene, reflection, bounding_volumes=None, stream=None):
        bv = image_of(bounding_volumes) if bounding_volumes is not None else None
        _check(lib.vq_apply_reflections(self._h, image_of(scene), image_of(reflection),
                                        C.byref(bv) if bv is not None else None, _stream_ptr(stream)))

    # K11 / K2 / K3 / K4
    def hdri_build_mips(self, pyr: Pyramid, stream=None):
        _check(lib.vq_hdri_build_mips(self._h, pyr, _stream_ptr(stream)))

    def diffuse_irradiance(self, pyr: Pyramid, cube: Cubemap, step=0.0, n_phi=64, n_theta=16, src_mip=3,
                           row_begin=0, row_end=None, stream=None):
        p = DiffuseIrradianceParams(step, n_phi, n_theta, src_mip)
        _check(lib.vq_diffuse_irradiance(self._h, C.byref(p), pyr, cube, row_begin,
                                         6 * cube.res if row_end is None else row_end, _stream_ptr(stream)))

    def specular_prefilter(self, pyr: Pyramid, cube: Cubemap, num_samples=512, row_begin=0, row_end=None, stream=None):
        _check(lib.vq_specular_prefilter(self._h, pyr, cube, num_samples, row_begin,
                                         cubemap_row_count(cube.res, cube.mips) if row_end is None else row_end,
                                         _stream_ptr(stream)))

    def specular_prefilter_multi(self, pyr: Pyramid, cubes, num_samples=512, row_begin=0, row_end=None, stream=None):
        """cubes: list of Cubemap descriptors of identical shape (local first, then the peers' mapped buffers)"""
        arr = (Cubemap * len(cubes))(*cubes)
        _check(lib.vq_specular_prefilter_multi(self._h, pyr, arr, len(cubes), num_samples, row_begin,
                                               cubemap_row_count(cubes[0].res, cubes[0].mips) if row_end is None else row_end,
                                               _stream_ptr(stream)))

    def specular_prefilter_ranges(self, pyr: Pyramid, cubes, row_ranges, num_samples=512, signal: "PeerSignal" = None, stream=None):
        """ONE persistent launch over several [begin,end) row ranges into all `cubes`, with the optional in-kernel rendezvous"""
        arr = (Cubemap * len(cubes))(*cubes)
        flat = [int(v) for ab in row_ranges for v in ab]
        rr = (C.c_int * len(flat))(*flat)
        _check(lib.vq_specular_prefilter_ranges(self._h, pyr, arr, len(cubes), num_samples, rr, len(row_ranges),
                                                C.byref(signal) if signal is not None else None, _stream_ptr(stream)))

    def brdf_integration_lut(self, out, num_samples=2048, row_begin=0, row_end=None, stream=None):
        o = image_of(out, 2)
        _check(lib.vq_brdf_integration_lut(self._h, o, num_samples, row_begin,
                                           o.height if row_end is None else row_end, _stream_ptr(stream)))

    # post chain
    def gaussian_blur(self, src, dst, vertical: bool, stream=None):
        p = BlurParams(src.shape[1], src.shape[0])
        fn = lib.vq_gaussian_blur_y if vertical else lib.vq_gaussian_blur_x
        _check(fn(self._h, C.byref(p), image_of(src), image_of(dst), _stream_ptr(stream)))

    def tonemap(self, params: TonemapperParams, src, dst, stream=None):
        _check(lib.vq_tonemap(self._h, C.byref(params), image_of(src), image_of(dst), _stream_ptr(stream)))

    def cas(self, con, src, dst, stream=None):
        _check(lib.vq_cas(self._h, con, image_of(src), image_of(dst), _stream_ptr(stream)))

    def fsr_easu(self, con, src, dst, address_mode=VQ_ADDRESS_WRAP, stream=None):
        _check(lib.vq_fsr_easu(self._h, con, address_mode, image_of(src), image_of(dst), _stream_ptr(stream)))

    def fsr_rcas(self, con, src, dst, stream=None):
        _check(lib.vq_fsr_rcas(self._h, con, image_of(src), image_of(dst), _stream_ptr(stream)))

    def spd_downsample(self, constants: SpdConstants, src, mips, stream=None):
        arr = (Image * len(mips))(*[image_of(m) for m in mips])
        _check(lib.vq_spd_downsample(self._h, C.byref(constants), image_of(src), arr, _stream_ptr(stream)))


class MaterialTable:
    """device-resident materials (vq_material_table_create); keeps the texel tensors' descriptors alive by reference"""

    def __init__(self, ctx: Context, materials, textures):
        n = len(materials)
        assert n == len(textures) and n >= 1
        self._ctx = ctx
        self._mats = (MaterialData * n)(*materials)
        self._tex = (MaterialTextures * n)(*textures)
        self._h = C.c_void_p()
        _check(lib.vq_material_table_create(ctx._h, self._mats, self._tex, n, C.byref(self._h)))

    def close(self):
        if self._h:
            lib.vq_material_table_destroy(self._ctx._h, self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def launch_count() -> int:
    return int(lib.vq_launch_count())
