"""Every hit kernel against the oracle from the world origin to the edge of the float range, on the GPU.

The ladder of tests/test_magnitudes_cpu.py (three base scenes moved by x -> s x + T up to |T| = 2^126) traced by every variant
with a per-ray kernel, bit for bit against the oracle's Hitable::hit: PACKED, SCALAR, COOP, DEFERRED, TENSOR, TENSOR_STREAM, and
BVH with the host tree, with the device builder's tree and with a level-0 tree refitted by r1_scene_move_spheres.  The device's
scan records must equal the restatement the CPU test filters with, the tensor filter probe must flag every sphere the exact test
could accept, and whole renders of every variant must equal the CPU restatement of the integrator at levels up to 2^120."""
import numpy as np
import pytest

import lbvh_restatement as lbvh
from test_magnitudes_cpu import BASES, LEVELS, base_spheres, move_cam22, moved, scan_records, transform, windows  # noqa: F401
from test_magnitudes_cpu import ladder  # noqa: F401  (module fixture)
from test_move_spheres_gpu import cuda, tree_bytes
from test_render_oracle_gpu import check, expected  # noqa: F401  (module fixture)
from test_scan_edges_gpu import RawScene, check_against_oracle, spec

pytestmark = pytest.mark.gpu

F = np.float32
RAY_VARIANTS = ("packed", "scalar", "coop", "deferred", "tensor", "tensor_stream")


def committed(r1, L):
    """a fresh commit of a ladder scene, its camera installed"""
    s = RawScene((0, 0, 1, 0, 0, 0, 40, 0, 10), L["spheres"], commit=False)
    s.set_camera_raw(L["cam22"], 0)
    return s


def device_buildable(spheres):
    """whether every sphere that can be hit has a finite radius_sq: the device builder and r1_scene_move_spheres refuse the rest
    (R1_ERR_ARG).  False where the ground sphere's radius, scaled, squares beyond float (scaled 66 and up, scale 2^60 and up)."""
    r = np.array([sp[3] for sp in spheres], F)
    with np.errstate(over="ignore"):
        return bool(np.isfinite((r * r)[r > 0]).all())


def scan_bytes(soa):
    """the scan block [n_pad float4 x 4 lanes] the restatement predicts, in the supergroup layout; the padding up to n_pad holds
    spheres that can never be hit (0, 0, 0, +inf)"""
    n = len(soa["cx"])
    n_pad = (n + 15) // 16 * 16
    lanes, kk = scan_records(soa)
    out = np.zeros((n_pad, 4), F)
    for i in range(n_pad):
        g, k = divmod(i, 4)
        f4 = (g >> 2) * 16 + (g & 3)
        rec = (lanes[i, 0], lanes[i, 1], lanes[i, 2], kk[i]) if i < n else (F(0), F(0), F(0), F(np.inf))
        for j, v in enumerate(rec):
            out[f4 + 4 * j, k] = v
    return out.view(np.uint8).reshape(-1)


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_trace_rays_match_the_oracle(r1, ladder, name, level):
    L = ladder[name, level]
    s = committed(r1, L)
    try:
        rec = s.device_records()
        want_scan = scan_bytes(L["soa"])
        assert np.array_equal(rec[:want_scan.size], want_scan), "%s %s: the scan records differ from r1_encode.h's" % (name, level)
        for w, want in L["hits"].items():
            check_against_oracle(r1, s, want, L["org"], L["d"], *w, RAY_VARIANTS + ("bvh",), "%s %s host tree" % (name, level))
        if not device_buildable(L["spheres"]):
            with pytest.raises(r1.Rays1Error):
                s.build_bvh(r1.BVH_BUILD_DEVICE)
            return
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(lbvh.build(L["soa"])), "%s %s: device tree" % (name, level)
        for w, want in L["hits"].items():
            check_against_oracle(r1, s, want, L["org"], L["d"], *w, ("bvh",), "%s %s device tree" % (name, level))
    finally:
        s.close()


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_moved_scenes_trace_like_the_oracle(r1, ladder, name, level):
    """commit at level 0, move every sphere (centre and radius) to the level, trace; then move back to the original bytes"""
    L0, L = ladder[name, "level0"], ladder[name, level]
    s = committed(r1, L0)
    try:
        orig = s.device_records()
        if not device_buildable(L["spheres"]):
            sp = L["spheres"]
            with pytest.raises(r1.Rays1Error):
                s.move_spheres(cuda(np.array([x[:3] for x in sp], F)), cuda(np.array([x[3] for x in sp], F)))
            assert np.array_equal(s.device_records(), orig), "%s %s: a refused move writes nothing" % (name, level)
            return
        for builder in (r1.BVH_BUILD_HOST, r1.BVH_BUILD_DEVICE):
            s.build_bvh(builder)
            sp = L["spheres"]
            s.move_spheres(cuda(np.array([x[:3] for x in sp], F)), cuda(np.array([x[3] for x in sp], F)))
            for w, want in L["hits"].items():
                check_against_oracle(r1, s, want, L["org"], L["d"], *w, ("packed", "tensor", "bvh"), "%s %s moved (%d)" % (name, level, builder))
            sp = L0["spheres"]
            s.move_spheres(cuda(np.array([x[:3] for x in sp], F)), cuda(np.array([x[3] for x in sp], F)))
            assert np.array_equal(s.device_records(), orig), "%s %s: moving back restores every byte" % (name, level)
    finally:
        s.close()


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_tensor_filter_probe_flags_every_candidate(r1, ladder, name, level):
    """every sphere whose discriminant the oracle accepts (it returns a hit there in some window) has e >= 0"""
    L = ladder[name, level]
    s = committed(r1, L)
    try:
        n = len(L["soa"]["cx"])
        e = s.filter_probe(L["org"], L["d"], n)
        for w, (idx, *_) in L["hits"].items():
            k = np.nonzero(idx >= 0)[0]
            ek = e[k, idx[k]]
            assert ((ek >= 0) & ~np.signbit(ek)).all(), "%s %s %s: %d hits unflagged" % (name, level, w, (~(ek >= 0)).sum())
        dead = np.ones(e.shape[1], bool)
        dead[:n] = L["soa"]["inv_radius"] == 0
        assert (e[:, dead] < 0).all()
    finally:
        s.close()


RENDER_LEVELS = tuple("scaled%d" % k for k in (30, 60, 64, 66, 90, 120)) + ("level0", "rigid20", "rigid40")
RENDER_VARIANTS = ("mega", "packed", "scalar", "coop", "deferred", "dual", "wavefront", "tensor", "tensor_stream", "bvh")


@pytest.mark.parametrize("level", RENDER_LEVELS)
def test_renders_match_the_integrator(r1, expected, monkeypatch, level):  # noqa: F811
    """n120 with the camera moved with the scene, 48x27x4 at 8 bounces, every variant and both BVH builders; a scene moved there
    from level 0 renders the same bytes.  From scaled 66 on, the ground's radius_sq overflows: the device builder and the move
    refuse it, and the other variants must still match the integrator."""
    cam, sph = spec("n120")
    s0 = RawScene(cam, sph, commit=False)
    cam22 = s0.camera()
    s0.close()
    sc, t = transform(level)
    msph, mcam = moved(sph, sc, t), move_cam22(cam22, sc, t)
    s = RawScene(cam, msph, commit=False)
    s.set_camera_raw(mcam, 0)
    try:
        ref = None
        for v in RENDER_VARIANTS:
            rgb, sums, res = check(r1, expected, monkeypatch, s, 48, 27, 4, mb=8, variant=r1.VARIANTS[v], what="n120 %s %s" % (level, v))
            ref = ref or (rgb, res.num_rays)
        if not device_buildable(msph):
            with pytest.raises(r1.Rays1Error):
                s.build_bvh(r1.BVH_BUILD_DEVICE)
            return
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        check(r1, expected, monkeypatch, s, 48, 27, 4, mb=8, variant=r1.VARIANT_MEGAKERNEL_BVH, what="n120 %s bvh device" % level)
        m = RawScene(cam, sph, commit=False)
        m.set_camera_raw(mcam, 0)
        try:
            m.move_spheres(cuda(np.array([x[:3] for x in msph], F)), cuda(np.array([x[3] for x in msph], F)))
            for v in ("packed", "tensor"):
                rgb, res = m.render(48, 27, 4, 8, variant=r1.VARIANTS[v])
                assert np.array_equal(rgb, ref[0]) and res.num_rays == ref[1], "n120 %s: moved scene, %s" % (level, v)
        finally:
            m.close()
    finally:
        forget(expected, s)
        s.close()


def forget(expected, s):  # noqa: F811
    """drop the oracle renders cached under this scene's handle: a later scene may be allocated at the same address"""
    so = expected.scenes.pop(s.handle, None)
    if so is not None:
        expected.oracle.scene_destroy(so)
    for key in [k for k in expected.renders if k[0] == s.handle]:
        del expected.renders[key]

