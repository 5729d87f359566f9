"""A batch of views (r1_render_views, r1_render_views_device; DESIGN.md section 4.14) without a device: every refusal that needs no
device comes before any device is looked up, in the documented order, and the Python wrappers check the arrays they are given."""
import ctypes as C

import numpy as np
import pytest

F = np.float32


@pytest.fixture(scope="module")
def scene(r1):
    s = r1.create_scene("small", commit=False)
    yield s
    s.close()


def has_gpu(r1):
    try:
        return r1.device_count() > 0
    except r1.Rays1Error:
        return False


def params(r1, w=16, h=9, spp=1, variant=0, **kw):
    p = r1.RenderParams(w, h, spp, 50, variant, 0, 0, 1, 1, 0, 0, -1)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


CAMS = np.zeros((4, 22), F)
SEEDS = np.arange(4, dtype=np.uint32)
RGB = np.zeros(16, np.uint8)


def call(r1, s, p, n=2, cams=CAMS, seeds=SEEDS, out=RGB, device=False, rays=RGB):
    """rc of one call through the raw ABI; None stands for a null pointer, p = None for null params"""
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    pp = C.byref(p) if p is not None else None
    res = r1.Result()
    if device:
        return r1.lib.r1_render_views_device(s.handle, pp, n, ptr(cams), ptr(seeds), ptr(out), ptr(rays), None, C.byref(res))
    return r1.lib.r1_render_views(s.handle, pp, n, ptr(cams), ptr(seeds), ptr(out), None, C.byref(res))


@pytest.mark.parametrize("device", [False, True])
def test_arguments_are_refused_before_any_device(r1, scene, device):
    arg = -1
    assert call(r1, scene, params(r1), n=0, device=device) == arg
    assert call(r1, scene, params(r1), cams=None, device=device) == arg
    assert call(r1, scene, params(r1), out=None, device=device) == arg
    if device:
        assert call(r1, scene, params(r1), rays=None, device=True) == arg
    assert call(r1, scene, None, device=device) == arg
    for bad in (dict(width=0), dict(spp=0), dict(max_bounces=-1), dict(world=0), dict(rank=1)):
        assert call(r1, scene, params(r1, **bad), device=device) == arg, bad
    for variant in (1, 2, 3, 4, 5, 8, 10):
        assert call(r1, scene, params(r1, variant=variant), device=device) == arg, variant
        assert "variant" in r1.lib.r1_last_error().decode()
    assert call(r1, scene, params(r1, threads=1024), device=device) == arg
    assert call(r1, scene, params(r1, blocks_per_sm=1), device=device) == arg
    assert "default tuning" in r1.lib.r1_last_error().decode()
    # the argument checks come before the limits: n_views = 0 with a batch far too large is still R1_ERR_ARG
    assert call(r1, scene, params(r1, w=65536, h=32768), n=0, device=device) == arg


@pytest.mark.parametrize("device", [False, True])
def test_the_batch_pixel_bound(r1, scene, device):
    """K x local pixels must stay below 2^32 - 1 (0xffffffff marks an empty pool entry); refused before any device is looked up"""
    third = (2 ** 32 - 1) // 3                                                       # 3 x third = 2^32 - 1
    assert call(r1, scene, params(r1, w=third, h=1), n=3, device=device) == -4
    assert call(r1, scene, params(r1, w=65536, h=32768), n=2, device=device) == -4   # 2^32
    assert "too many pixels" in r1.lib.r1_last_error().decode()
    # the whole batch's samples: 2^31 pixels x 2^17 spp needs more than g / spp in 64 bits can take
    assert call(r1, scene, params(r1, w=32768, h=32768, spp=1 << 17), n=2, device=device) == -4
    assert "too many samples" in r1.lib.r1_last_error().decode()
    # just inside both bounds the call goes on to the device: none here (R1_ERR_CUDA), or with one the scene is not committed
    want = -2 if has_gpu(r1) else -3
    assert call(r1, scene, params(r1, w=(2 ** 32 - 2) // 2, h=1), n=2, device=device) == want
    assert call(r1, scene, params(r1, w=32768, h=32768, spp=1 << 16), n=1, device=device) == want


def test_no_cpu_fallback_without_a_gpu(r1, scene):
    if has_gpu(r1):
        pytest.skip("a GPU is present")
    cams = np.zeros((3, 22), F)
    with pytest.raises(r1.Rays1Error, match=r"\(-3\)"):
        scene.render_views(cams, width=16, height=9, spp=1)
    with pytest.raises(r1.Rays1Error, match=r"\(-3\)"):
        scene.render_views(cams, seeds=[1, 2, 0xFFFFFFFF], width=16, height=9, spp=1, sums=True)
    with pytest.raises(r1.Rays1Error, match=r"\(-3\)"):
        scene.render_views_device(cams, 1 << 20, 1 << 21, width=16, height=9, spp=1)
    for variant in (0, 6, 7, 9, 11):                                                 # every accepted variant reaches the device
        assert call(r1, scene, params(r1, variant=variant), n=3, seeds=None) == -3
    assert call(r1, scene, params(r1), n=3, seeds=None, device=True) == -3
    # ... and the Python wrappers refuse what the library refuses
    with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
        scene.render_views(np.zeros((0, 22), F), width=16, height=9, spp=1)
    with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
        scene.render_views(cams, width=16, height=9, spp=1, variant=r1.VARIANT_WAVEFRONT)


@pytest.mark.parametrize("device", [False, True])
def test_python_checks_cams_and_seeds(r1, scene, device):
    def run(cams, seeds=None):
        if device:
            return scene.render_views_device(cams, 1 << 20, 1 << 21, seeds=seeds, width=16, height=9, spp=1)
        return scene.render_views(cams, seeds=seeds, width=16, height=9, spp=1)

    with pytest.raises(ValueError, match="float32"):
        run(np.zeros((2, 22), np.float64))
    with pytest.raises(ValueError, match="float32"):
        run([[0.0] * 22])
    for shape in ((22,), (2, 21), (2, 23), (1, 2, 22)):
        with pytest.raises(ValueError, match=r"cams must hold 22 constants per view, shape \(K, 22\), not shape"):
            run(np.zeros(shape, F))
    cams = np.zeros((3, 22), F)
    with pytest.raises(ValueError, match="seeds must be integers"):
        run(cams, np.zeros(3, F))
    for seeds in (np.zeros(2, np.uint32), np.zeros(4, np.uint32), np.zeros((3, 1), np.uint32), 5):
        with pytest.raises(ValueError, match=r"seeds must hold one seed per view, shape \(3,\), not shape"):
            run(cams, seeds)
    for seeds in ([0, -1, 2], [0, 1, 2 ** 32]):
        with pytest.raises(ValueError, match=r"seeds must lie in 0 \.\. 2\^32 - 1"):
            run(cams, seeds)


def test_exported(r1):
    assert {"r1_render_views", "r1_render_views_device"} <= set(r1.EXPORTED)
    assert r1.lib.r1_abi_version() == 2
