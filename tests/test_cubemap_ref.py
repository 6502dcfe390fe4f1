"""CPU: the oracle's cube-face orientation (SURVEY A35) against the reference's own per-face view matrices —
Source/Renderer/Resources/CubemapUtility.cpp compiled UNMODIFIED in place (oracle/_ref/libvqcuberef.so; DirectXMath stand-in with
the library's documented XMMatrixLookAtLH). The engine renders every cubemap face with CalculateViewMatrix(face) times a 90-degree
projection (EnvironmentMapRendering.cpp:170-176); the look direction through a pixel centre follows from that matrix alone and
must equal oracle CubeTexelDirection — the table every IBL kernel and the forward pass's cube sampler are built on."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as orc
import ref_golden as rg

LIB = os.path.join(orc.ORACLE_DIR, "_ref", "libvqcuberef.so")
needs_ref = pytest.mark.skipif(not os.path.exists(LIB), reason="oracle/_ref/libvqcuberef.so not built (needs the engine sources at build time)")


@needs_ref
def test_face_view_matrices_are_the_d3d_cube_convention():
    ref = C.CDLL(LIB)
    want = {0: (1, 0, 0), 1: (-1, 0, 0), 2: (0, 1, 0), 3: (0, -1, 0), 4: (0, 0, 1), 5: (0, 0, -1)}   # RIGHT LEFT UP DOWN FRONT BACK
    for face, fwd in want.items():
        m = np.zeros(16, np.float32)
        ref.cuberef_view_matrix(face, orc._p(m))
        m = m.reshape(4, 4)
        assert np.array_equal(m[:3, 2], np.float32(fwd))             # third column of a look-at = the view direction
        assert np.allclose(m[:3, :3] @ m[:3, :3].T, np.eye(3)) and np.array_equal(m[3], np.float32([0, 0, 0, 1]))


@needs_ref
@pytest.mark.parametrize("res", rg.CUBE_RES)
def test_texel_directions_equal_the_reference_matrices(res):
    ref = C.CDLL(LIB)
    assert rg.reference("cube_dirs", res) == rg.stored("cube_dirs", res)
    o = orc.lib()
    a, b = np.zeros(3, np.float32), np.zeros(3, np.float32)
    pts = sorted({0, res - 1, res // 2, res // 3, (2 * res) // 3})
    for face in range(6):
        for py in pts:
            for px in pts:
                o.orc_cube_texel_direction(face, px, py, res, orc._p(a))
                ref.cuberef_texel_direction(face, px, py, res, orc._p(b))
                assert np.array_equal(a + np.float32(0), b + np.float32(0)), (face, px, py, a, b)     # +0: -0.0 == 0.0
                # and back: the direction selects the same face and pixel
                f, sx, sy = C.c_int(0), C.c_float(0), C.c_float(0)
                o.orc_direction_to_cube_face(orc._p(b), C.byref(f), C.byref(sx), C.byref(sy))
                assert f.value == face
                assert abs((sx.value * 0.5 + 0.5) * res - (px + 0.5)) < 1e-3 and abs((0.5 - sy.value * 0.5) * res - (py + 0.5)) < 1e-3


@pytest.mark.parametrize("res", rg.CUBE_RES)
def test_texel_directions_equal_the_stored_reference(res):
    """the oracle's texel directions == the reference's, as stored in tests/golden/ref_golden.json"""
    assert rg.port("cube_dirs", res) == rg.stored("cube_dirs", res)
