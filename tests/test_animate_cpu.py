"""CPU checks of animating the camera and the materials on the device (r1_scene_move_camera, r1_scene_set_materials; DESIGN.md
section 4.11).

r1_camera_constants is r1_scene_set_camera's arithmetic, so its constants equal set_camera + get_camera bit for bit: for the
built-in scenes' camera arguments, whose constants are pinned to the reference's recorded ones (tests/test_abi_cpu.py), and for
seeded random cameras.  Also: header, Python and library agree on the new names, and every refusal that needs no device comes back
before one is touched.  The device side is tested by tests/test_animate_gpu.py."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT

F = np.float32
ASPECT = F(1280) / F(720)                              # the reference's SCREEN_W / SCREEN_H (rayweek1.cpp:564)
# rays1_host.cpp's builders: lookfrom, lookat, vfov, aperture, focus_dist (vup = 0, 1, 0)
BUILTIN_CAMERAS = {
    "small": ((2, 1, 2), (0, 0, 0), 60, F(0.1), 5.0),
    "medium": ((0, 2, 3), (0, 0, 0), 60, F(0.1) * F(0.2), 3.0),
    "large": ((3, 8, 15), (0, 0, 0), 60, F(0.1), 10.0),
}


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def set_camera_constants(r1, lookfrom, lookat, vup, vfov, aspect, aperture, focus):
    """r1_scene_set_camera + r1_scene_get_camera on a scene of its own"""
    lib = r1.lib
    sc = lib.r1_scene_create(1)
    try:
        v = lambda x: np.array(x, F)  # noqa: E731
        assert lib.r1_scene_set_camera(sc, v(lookfrom), v(lookat), v(vup), vfov, aspect, aperture, focus) == 0
        out = np.zeros(22, F)
        assert lib.r1_scene_get_camera(sc, out) == 0
        return out
    finally:
        lib.r1_scene_destroy(sc)


@pytest.mark.parametrize("name", sorted(BUILTIN_CAMERAS))
def test_camera_constants_are_the_reference_constants(r1, golden_rays, name):
    lookfrom, lookat, vfov, aperture, focus = BUILTIN_CAMERAS[name]
    got = r1.camera_constants(lookfrom, lookat, (0, 1, 0), vfov, ASPECT, aperture, focus)
    assert got.dtype == F and got.shape == (22,)
    assert np.array_equal(bits(got), bits(golden_rays[name]["camera"]))
    assert np.array_equal(bits(got), bits(set_camera_constants(r1, lookfrom, lookat, (0, 1, 0), vfov, ASPECT, aperture, focus)))


def test_camera_constants_equal_set_camera_for_random_cameras(r1):
    rng = np.random.default_rng(2024)
    for k in range(300):
        lookfrom = rng.normal(scale=10.0 ** rng.uniform(-2, 4), size=3).astype(F)
        lookat = (lookfrom + rng.normal(scale=10.0 ** rng.uniform(-2, 3), size=3)).astype(F)
        vup = rng.normal(size=3).astype(F) if k % 3 else np.array([0, 1, 0], F)
        args = (lookfrom, lookat, vup, F(rng.uniform(5, 150)), F(rng.uniform(0.3, 3.0)), F(rng.uniform(0, 2) * (k % 4 != 0)),
                F(10.0 ** rng.uniform(-1, 3)))
        got = r1.camera_constants(*args)
        want = set_camera_constants(r1, *args)
        assert np.array_equal(bits(got), bits(want)), (k, args)


def test_header_python_and_library_agree_on_the_names(r1):
    header = open(os.path.join(ROOT, "include", "rays1_b200.h")).read()
    for fn in ("r1_camera_constants", "r1_scene_move_camera", "r1_scene_set_materials"):
        assert re.search(r"\bint %s\(" % fn, header) and fn in r1.EXPORTED
        assert getattr(r1.lib, fn).argtypes is not None
    assert "#define R1_ABI_VERSION 2" in header and r1.lib.r1_abi_version() == 2
    assert callable(r1.camera_constants) and callable(r1.Scene.move_camera) and callable(r1.Scene.set_materials)


def test_refusals_come_back_before_a_device_is_touched(r1):
    lib = r1.lib
    raw = C.CDLL(r1.LIB_PATH)                          # unchecked argument types, so that null pointers can be passed
    v3, out = (C.c_float * 3)(0, 0, 1), (C.c_float * 22)()
    f = C.c_float
    raw.r1_camera_constants.argtypes = [C.c_void_p] * 3 + [f] * 4 + [C.c_void_p]
    for args in ((None, v3, v3), (v3, None, v3), (v3, v3, None)):
        assert raw.r1_camera_constants(*args, 60, 1, 0, 1, out) == -1
    assert raw.r1_camera_constants(v3, v3, v3, 60, 1, 0, 1, None) == -1
    cam = np.zeros(22, F)
    assert lib.r1_scene_move_camera(None, -1, cam.ctypes.data) == -1
    ms = C.c_double(0)
    buf = (C.c_float * 12)()
    assert lib.r1_scene_set_materials(None, -1, 0, 1, buf, None, None, None, C.byref(ms)) == -1
    sc = lib.r1_scene_create(4)
    try:
        for j in range(3):
            assert lib.r1_scene_add_sphere(sc, j, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0) == j
        assert lib.r1_scene_move_camera(sc, -1, None) == -1 and b"null" in lib.r1_last_error()
        for first, n in ((0, 4), (3, 1), (2, 2), (1, 0xFFFFFFFF), (0xFFFFFFFF, 2)):
            for ptrs in ((buf, None, None), (None, buf, None), (None, None, buf), (buf, buf, buf)):
                assert lib.r1_scene_set_materials(sc, -1, first, n, *ptrs, None, C.byref(ms)) == -1, (first, n)
                assert lib.r1_scene_set_materials(sc, 0, first, n, *ptrs, None, None) == -1, (first, n)
            assert b"out of range" in lib.r1_last_error()
        for first in (0, 2):
            assert lib.r1_scene_set_materials(sc, -1, first, 1, None, None, None, None, C.byref(ms)) == -1
            assert b"no material field" in lib.r1_last_error()
        # valid arguments on a scene that is not committed: refused by the state check, never a crash
        assert lib.r1_scene_move_camera(sc, -1, cam.ctypes.data) == -2
        assert lib.r1_scene_move_camera(sc, 0, cam.ctypes.data) == -2
        for first, n, ptrs in ((0, 3, (buf, buf, buf)), (1, 2, (None, buf, None)), (3, 0, (None, None, None)), (0, 0, (buf, None, None))):
            assert lib.r1_scene_set_materials(sc, -1, first, n, *ptrs, None, C.byref(ms)) == -2
            assert lib.r1_scene_set_materials(sc, 0, first, n, *ptrs, None, None) == -2
            assert b"not committed" in lib.r1_last_error()
    finally:
        lib.r1_scene_destroy(sc)


def test_python_refuses_bad_arguments_without_a_device(r1):
    from test_scan_edges_gpu import RawScene
    with pytest.raises(ValueError, match="lookat"):
        r1.camera_constants((0, 0, 1), (0, 0), (0, 1, 0), 60, 1.5, 0, 1)
    with pytest.raises(ValueError, match="vup"):
        r1.camera_constants((0, 0, 1), (0, 0, 0), (0, 1, 0, 0), 60, 1.5, 0, 1)
    s = RawScene((0, 0, 1, 0, 0, 0, 40, 0, 10), [(0.0, 0.0, 0.0, 1.0, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0.0)], commit=False)
    try:
        for bad in (np.zeros(21, F), np.zeros((2, 11), F)):
            with pytest.raises(ValueError, match="22"):
                s.move_camera(bad)
        with pytest.raises(ValueError, match="at least one"):
            s.set_materials()
        with pytest.raises(ValueError, match="CUDA tensor"):
            s.set_materials(kind=np.zeros(1, np.int32))
        with pytest.raises(ValueError, match="CUDA tensor"):
            s.set_materials(param=[1.5])
        torch = pytest.importorskip("torch")
        for kw in ({"kind": torch.zeros(1, dtype=torch.int32)}, {"albedo": torch.zeros(1, 3)}, {"param": torch.zeros(1)}):
            with pytest.raises(ValueError, match="CUDA tensor"):
                s.set_materials(**kw)
    finally:
        s.close()
