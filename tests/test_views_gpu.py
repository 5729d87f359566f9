"""A batch of views (r1_render_views, r1_render_views_device; DESIGN.md section 4.14) on the GPU.

View v of a batch must be byte for byte what move_camera(cams[v]) followed by render_sums(seed = seeds[v]) gives on the same device:
the same fixed-point sums, bytes and rank rows, and the batch's ray count is the sum of those renders' counts.  Checked for every
variant a batch takes on scenes from 5 to 10^5 spheres, at sizes where view boundaries fall inside a warp's 32 samples, against the
oracle directly, for rank shares, after the device's records changed, on torch streams, and for the device's camera, which a batch
leaves as it was."""
import numpy as np
import pytest

from test_animate_gpu import orbit
from test_gpu_parity import scenes  # noqa: F401  (module fixture: the four built-in scenes)
from test_move_spheres_gpu import Fresh, cam22, random_spheres
from test_render_oracle_gpu import Expected, assert_matches
from test_tensor_stream_gpu import big_scenes  # noqa: F401  (module fixture: grids of 5 048 and 8 016 spheres)

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
F = np.float32

SIZES = ((1, 1, 1), (7, 3, 5), (33, 7, 3), (96, 54, 8))
KS = (1, 3, 37)
MAX_K = max(KS)
SEEDS = np.array([0xFFFFFFFF] + [(v * 2654435761 + 12345) & 0xFFFFFFFF for v in range(1, MAX_K)], np.uint32)
PACKED, TENSOR, STREAM, BVH = 7, 6, 9, 11


@pytest.fixture(scope="module")
def extra(r1):
    """n769: 769 random spheres (the streamed filter's first size past the resident one); cloud: 10^5 spheres"""
    import make_scene
    cam, sph = make_scene.cloud_scene(100000, seed=5)
    cloud = [tuple(F(v) for v in sp[:4]) + (int(sp[4]),) + tuple(F(v) for v in sp[5:]) for sp in sph]
    out = {"n769": Fresh(r1, cam22(r1), random_spheres(r1, 769, 769)), "cloud": Fresh(r1, cam22(r1), cloud)}
    yield out
    for s in out.values():
        s.close()


def cams_of(r1, name, k=MAX_K):
    dist = {"small": 12.0, "medium": 14.0, "large": 16.0}.get(name, 45.0)
    return np.stack([orbit(r1, v, dist) for v in range(k)])


def singles(s, cams, seeds, w, h, spp, variant, **kw):
    """move_camera + render_sums per view; the device's camera is restored afterwards"""
    home = s.camera()
    out = []
    try:
        for cam, seed in zip(cams, seeds):
            s.move_camera(cam)
            out.append(s.render_sums(w, h, spp, variant=variant, seed=int(seed), **kw))
    finally:
        s.move_camera(home)
    return out


def first_pixel(a, b):
    lr, x = np.argwhere((a != b).reshape(a.shape[0], -1, 3).any(axis=2))[0]
    return int(x), int(lr)


def assert_views(rgb, sums, res, want, what):
    """sums, then bytes, then the total ray count; a failure names the view and the first differing pixel"""
    assert rgb.shape[0] == sums.shape[0] == len(want), what
    for v, (wr, ws, _) in enumerate(want):
        assert rgb[v].shape == wr.shape, "%s view %d: shape %s, single render %s" % (what, v, rgb[v].shape, wr.shape)
        if not np.array_equal(sums[v], ws):
            x, lr = first_pixel(sums[v], ws)
            raise AssertionError("%s view %d: sums differ first at (x %d, local row %d): batch %s, single %s"
                                 % (what, v, x, lr, sums[v][lr, x].tolist(), ws[lr, x].tolist()))
        if not np.array_equal(rgb[v], wr):
            x, lr = first_pixel(rgb[v], wr)
            raise AssertionError("%s view %d: bytes differ first at (x %d, local row %d)" % (what, v, x, lr))
    total = sum(r.num_rays for _, _, r in want)
    assert res.num_rays == total, "%s: %d rays, the single renders %d" % (what, res.num_rays, total)


# ---- 1. every view equals its single render ----------------------------------------------------------------------------------

# grid5048: beyond the 4096 spheres PACKED stages, so it runs the unstaged batch instance
CASES = [(n, v) for n in ("small", "medium", "large", "synth4096", "grid5048") for v in (0, PACKED)] + \
        [("large", TENSOR), ("n769", STREAM), ("n769", BVH), ("cloud", BVH)]


@pytest.mark.parametrize("name,variant", CASES, ids=["%s-%d" % c for c in CASES])
def test_each_view_equals_its_single_render(r1, scenes, extra, big_scenes, name, variant):  # noqa: F811
    s = scenes[name] if name in scenes else big_scenes[5048] if name == "grid5048" else extra[name]
    cams = cams_of(r1, name)
    for w, h, spp in SIZES:
        want = singles(s, cams, SEEDS, w, h, spp, variant)
        for k in KS:
            rgb, sums, res = s.render_views(cams[:k], SEEDS[:k], width=w, height=h, spp=spp, variant=variant, sums=True)
            assert_views(rgb, sums, res, want[:k], "%s variant %d %dx%dx%d K=%d" % (name, variant, w, h, spp, k))
            assert res.num_samples == k * w * h * spp and res.launches == 2
        if w * h > 1:   # the cameras are used: the views differ
            assert not np.array_equal(want[0][0], want[1][0])


def test_seeds_default_to_the_render_seed(r1, scenes):  # noqa: F811
    s = scenes["medium"]
    cams = cams_of(r1, "medium", 5)
    want = singles(s, cams, [77] * 5, 33, 7, 3, 0)
    rgb, sums, res = s.render_views(cams, width=33, height=7, spp=3, seed=77, sums=True)
    assert_views(rgb, sums, res, want, "seeds=None")
    rgb2, res2 = s.render_views(cams, width=33, height=7, spp=3, seed=77)
    assert np.array_equal(rgb, rgb2) and res2.num_rays == res.num_rays


# ---- 2. the oracle, directly ---------------------------------------------------------------------------------------------------

class ViewExpected(Expected):
    """the oracle's renders of a GPU scene seen through given camera constants"""

    def __init__(self, r1, oracle, cam):
        super().__init__(r1, oracle)
        self.cam = cam

    def scene(self, s):
        if s.handle not in self.scenes:
            so = self.oracle.scene_create_from_soa(s.soa())
            self.oracle.scene_set_camera(so, self.cam)
            self.scenes[s.handle] = so
        return self.scenes[s.handle]


def test_views_match_the_oracle(r1, oracle, scenes):  # noqa: F811
    s = scenes["medium"]
    w, h, spp = 33, 7, 3
    cams, seeds = cams_of(r1, "medium", 3), SEEDS[:3]
    rgb, sums, res = s.render_views(cams, seeds, width=w, height=h, spp=spp, sums=True)
    total = 0
    for v in range(3):
        e = ViewExpected(r1, oracle, cams[v])
        try:
            want_rays = e.render(s, w, h, spp, 50, int(seeds[v]), 0, 1, 1)[2]
            assert_matches(e, s, sums[v], rgb[v], want_rays, w, h, spp, seed=int(seeds[v]), what="view %d" % v)
            total += want_rays
        finally:
            e.close()
    assert res.num_rays == total


# ---- 3. rank shares --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("row_tile", [1, 2])
def test_rank_shares(r1, scenes, row_tile):  # noqa: F811
    s = scenes["large"]
    cams, seeds = cams_of(r1, "large", 3), SEEDS[:3]
    for (w, h, spp) in ((33, 7, 3), (9, 2, 2)):        # 9x2: rank 2 of 3 owns no rows
        for rank in range(3):
            kw = dict(rank=rank, world=3, row_tile=row_tile)
            want = singles(s, cams, seeds, w, h, spp, 0, **kw)
            rgb, sums, res = s.render_views(cams, seeds, width=w, height=h, spp=spp, sums=True, **kw)
            assert rgb.shape == (3, r1.local_rows(h, row_tile, rank, 3), w, 3)
            assert_views(rgb, sums, res, want, "rank %d/3 tile %d %dx%dx%d" % (rank, row_tile, w, h, spp))
    assert r1.local_rows(2, 1, 2, 3) == 0


# ---- 4. device state -------------------------------------------------------------------------------------------------------------

def test_batches_see_moved_spheres_and_new_materials(r1):
    spheres = random_spheres(r1, 769, 11)
    s = Fresh(r1, cam22(r1), spheres)
    try:
        rng = np.random.default_rng(3)
        n = 300
        centres = np.array([sp[:3] for sp in spheres[100:100 + n]], F) + rng.normal(0, 0.5, (n, 3)).astype(F)
        s.move_spheres(torch.from_numpy(centres).cuda())
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        kind = torch.from_numpy(rng.choice([0, 1, 2], 769).astype(np.int32)).cuda()
        albedo = torch.from_numpy(rng.uniform(0, 1, (769, 3)).astype(F)).cuda()
        s.set_materials(kind=kind, albedo=albedo)
        cams = cams_of(r1, "n769", 4)
        for variant in (0, PACKED, STREAM, BVH):
            want = singles(s, cams, SEEDS[:4], 33, 7, 3, variant)
            rgb, sums, res = s.render_views(cams, SEEDS[:4], width=33, height=7, spp=3, variant=variant, sums=True)
            assert_views(rgb, sums, res, want, "moved + recoloured, variant %d" % variant)
        fresh = Fresh(r1, cam22(r1), spheres)     # the batch rendered the device's records, not the host's
        try:
            assert not np.array_equal(fresh.render_views(cams, SEEDS[:4], width=33, height=7, spp=3)[0], rgb)
        finally:
            fresh.close()
    finally:
        s.close()


def test_a_batch_leaves_the_device_camera(r1, scenes):  # noqa: F811
    s = scenes["large"]
    home = s.camera()
    cams = cams_of(r1, "large", 3)
    before, rb = s.render(33, 7, 3)                          # the committed camera
    s.render_views(cams, width=33, height=7, spp=3)
    after, ra = s.render(33, 7, 3)
    assert np.array_equal(before, after) and rb.num_rays == ra.num_rays
    moved = orbit(r1, 9, 20.0)
    try:
        s.move_camera(moved)
        want, rw = s.render(33, 7, 3)
        s.render_views(cams, width=33, height=7, spp=3, variant=TENSOR)
        got, rg = s.render(33, 7, 3)
        assert np.array_equal(want, got) and rw.num_rays == rg.num_rays
        assert not np.array_equal(want, before)
    finally:
        s.move_camera(home)
    assert np.array_equal(s.camera(), home)


def test_a_bvh_batch_after_a_move_needs_a_tree(r1):
    spheres = random_spheres(r1, 200, 4)
    s = Fresh(r1, cam22(r1), spheres)
    try:
        s.move_spheres(torch.from_numpy(np.array([sp[:3] for sp in spheres[:10]], F) + 0.25).cuda())
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            s.render(16, 9, 1, variant=BVH)
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            s.render_views(cams_of(r1, "n200", 2), width=16, height=9, spp=1, variant=BVH)
        rgb, _ = s.render_views(cams_of(r1, "n200", 2), width=16, height=9, spp=1, variant=PACKED)   # no sticky error
        assert rgb.shape == (2, 9, 16, 3)
    finally:
        s.close()


# ---- 5. the device path --------------------------------------------------------------------------------------------------------

def device_views(s, st, cams, seeds, w, h, spp, **kw):
    k = len(cams)
    rgb = torch.zeros(k * w * h * 3, dtype=torch.uint8, device="cuda:0")
    rays = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    res = s.render_views_device(cams, rgb.data_ptr(), rays.data_ptr(), seeds=seeds, stream_ptr=st.cuda_stream, width=w, height=h, spp=spp, **kw)
    return rgb, rays, res


def test_device_batches_on_a_torch_stream(r1, scenes):  # noqa: F811
    s = scenes["large"]
    w, h, spp = 96, 54, 8
    cams = cams_of(r1, "large", 8)
    a_cams, b_cams = cams[:5], cams[5:]
    want_a = s.render_views(a_cams, SEEDS[:5], width=w, height=h, spp=spp)
    want_b = s.render_views(b_cams, SEEDS[5:8], width=w, height=h, spp=spp, variant=PACKED)
    st = torch.cuda.Stream(0)
    with torch.cuda.stream(st):
        torch.cuda._sleep(1_000_000_000)                                  # keeps both batches queued until both are enqueued
        a = device_views(s, st, a_cams, SEEDS[:5], w, h, spp)
        b = device_views(s, st, b_cams, SEEDS[5:8], w, h, spp, variant=PACKED)
    assert not st.query(), "the stream finished before the second batch was enqueued: the test proves nothing"
    res = s.render_wait()
    assert res.num_samples == 3 * w * h * spp and res.launches == 2 and res.kernel_ms > 0
    st.synchronize()
    for (rgb, rays, _), (want, wres) in ((a, want_a), (b, want_b)):
        assert np.array_equal(rgb.cpu().numpy().reshape(want.shape), want)
        assert int(rays.item()) == wres.num_rays


# ---- 6. one view with the scene's own camera -------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["small", "large", "synth4096"])
def test_one_view_is_a_render(r1, scenes, name):  # noqa: F811
    s = scenes[name]
    w, h, spp = 96, 54, 8
    want, wres = s.render(w, h, spp, seed=5)
    rgb, res = s.render_views(s.camera()[None], [5], width=w, height=h, spp=spp)
    assert np.array_equal(rgb[0], want) and res.num_rays == wres.num_rays
    assert res.num_samples == w * h * spp == wres.num_samples and res.launches == 2 and res.n_units == 0


# ---- 7. a batch of more than 2^31 pixels -----------------------------------------------------------------------------------------

def test_a_batch_past_2_31_pixels_resolves_every_pixel(r1, scenes):  # noqa: F811
    """resolve indexes pixels in 32 bits, so a batch above 2^31 pixels is resolved in two launches; both halves equal the single
    renders.  Needs ~80 GB of device memory (68.7 GB of accumulators); kept last in the file, since the accumulators stay allocated."""
    if torch.cuda.mem_get_info(0)[0] < 90e9:
        pytest.skip("needs 90 GB of free device memory")
    s = scenes["small"]
    w, h, kw = 32768, 32769, dict(spp=1, max_bounces=4)                  # 1 073 774 592 pixels a view; two views: 2^31 + 74 752
    npix = w * h
    cams, seeds = cams_of(r1, "small", 2), SEEDS[:2]
    out = torch.zeros(2 * npix * 3, dtype=torch.uint8, device="cuda:0")
    rays = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    s.render_views_device(cams, out.data_ptr(), rays.data_ptr(), seeds=seeds, width=w, height=h, **kw)
    res = s.render_wait()
    assert res.launches == 3 and res.num_samples == 2 * npix
    one = torch.zeros(npix * 3, dtype=torch.uint8, device="cuda:0")
    one_rays = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    home, total = s.camera(), 0
    try:
        for v in range(2):
            s.move_camera(cams[v])
            s.render_device(one.data_ptr(), one_rays.data_ptr(), width=w, height=h, seed=int(seeds[v]), **kw)
            s.render_wait()
            assert torch.equal(out[v * npix * 3:(v + 1) * npix * 3], one), "view %d differs from its single render" % v
            total += int(one_rays.item())
    finally:
        s.move_camera(home)
    assert int(rays.item()) == total
