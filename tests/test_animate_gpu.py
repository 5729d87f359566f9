"""Animating the camera and the materials on the device (r1_scene_move_camera, r1_scene_set_materials; DESIGN.md section 4.11) on
the GPU.

After set_materials a device holds exactly the shade records r1_scene_commit writes for a scene with the new materials (compared
byte for byte with a fresh scene of those values, committed from the host).  After move_camera and / or set_materials, renders of
every variant and the parity calls equal a fresh scene's; so does every frame of a loop that moves spheres, the camera and the
materials together, which no other path can do without a re-commit.  Also: a render already enqueued keeps its camera, a change on a
torch stream lands between two renders on it, the wavefront graph is rebuilt once per new camera, refusals leave every byte in
place, and the state rules."""
import numpy as np
import pytest

from test_bvh_gpu import RENDER_CASES
from test_move_spheres_gpu import ENCODE_SCENES, Fresh, cam22, centres_of, cuda, random_spheres, records_equal, spheres_of, with_values
from test_tensor_stream_gpu import assert_same

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
F = np.float32


# ---- scenes and values ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def base(r1):
    """name -> sphere list and camera of the module's scenes"""
    import make_scene
    out = {}
    for name in ("large", "synth4096"):
        s = r1.create_scene(name, commit=False)
        out[name] = (spheres_of(r1, s), s.camera())
        s.close()
    for n in (1, 17, 769, 5048):
        out["n%d" % n] = (random_spheres(r1, n, n), cam22(r1))
    cam, sph = make_scene.cloud_scene(100000, seed=5)
    out["cloud"] = ([tuple(F(v) for v in sp[:4]) + (int(sp[4]),) + tuple(F(v) for v in sp[5:]) for sp in sph], cam22(r1))
    return out


def can_hit(sp):
    """inv_radius != 0, as r1_scene_add_sphere derives it"""
    r = F(sp[3])
    return bool(r > 0 and F(1) / r != 0)


def with_materials(spheres, first, kind=None, albedo=None, param=None):
    """the sphere list with new fields for spheres first .. first + n - 1, Metal params clamped as the device (and add_sphere) store them"""
    out = list(spheres)
    n = len(next(a for a in (kind, albedo, param) if a is not None))
    for j in range(n):
        sp = list(out[first + j])
        if kind is not None:
            sp[4] = int(kind[j])
        if albedo is not None:
            sp[5:8] = [F(v) for v in albedo[j]]
        if param is not None:
            sp[8] = F(param[j])
        if sp[4] == 1:                                                   # R1_MAT_METAL
            sp[8] = sp[8] if sp[8] < 1 else F(1)
        out[first + j] = tuple(sp)
    return out


def set_materials(s, first=0, kind=None, albedo=None, param=None, **kw):
    t = lambda a, dt: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dt)).cuda(0)  # noqa: E731
    return s.set_materials(t(kind, np.int32), t(albedo, F), t(param, F), first=first, **kw)


def random_materials(rng, spheres, first, k):
    """kinds that keep every sphere that can be hit shaded (NONE only for the others), albedos, and params of every kind"""
    hit = np.array([can_hit(sp) for sp in spheres[first:first + k]], bool)
    kind = rng.choice([0, 1, 2], k).astype(np.int32)
    kind[~hit] = rng.choice([-1, 0, 1, 2], int((~hit).sum()))
    albedo = rng.uniform(0, 1, (k, 3)).astype(F)
    param = np.where(kind == 2, rng.choice([1.0, 1.33, 1.5, 2.4, 24.2], k), rng.uniform(0, 1.5, k)).astype(F)
    return kind, albedo, param


def orbit(r1, k, dist, height=0.5, target=(0, 0, 0), aperture=0.1):
    """the camera of frame k of an orbit around `target`"""
    a = 0.4 + 0.35 * k
    frm = np.array([dist * np.sin(a), dist * height, dist * np.cos(a)]) + target
    return r1.camera_constants(frm, target, (0, 1, 0), 60, F(16) / F(9), aperture, dist)


def orbit_of(r1, name, k):
    return orbit(r1, k, 16.0) if name == "large" else orbit(r1, k, 45.0)


FIELDS = ("kap", "k", "a", "p", "ka", "kp", "ap")                         # every combination of the given arrays


# ---- 1. encoding ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ENCODE_SCENES)
def test_new_materials_encode_like_a_commit(r1, base, name):
    spheres, cam = base[name]
    n = len(spheres)
    s = Fresh(r1, cam, spheres)
    try:
        orig = s.device_records()
        rng = np.random.default_rng(n + 1)
        cur = list(spheres)
        steps = [(0, n, f) for f in FIELDS] + [(n // 3, max(1, n // 4), "kap"), (n - 1, 1, "kp"), (n // 2, n - n // 2, "a"), (n // 2, 0, "kap")]
        for first, k, fields in steps:
            kind, albedo, param = random_materials(rng, cur, first, k)
            args = {"kind": kind if "k" in fields else None, "albedo": albedo if "a" in fields else None, "param": param if "p" in fields else None}
            ms = set_materials(s, first, **args)
            assert ms >= 0
            if k:
                cur = with_materials(cur, first, **args)
            records_equal(r1, s, cur, cam, "%s materials %d+%d %s" % (name, first, k, fields))
        # the original materials restore the original bytes
        set_materials(s, 0, kind=[sp[4] for sp in spheres], albedo=[sp[5:8] for sp in spheres], param=[sp[8] for sp in spheres])
        assert np.array_equal(s.device_records(), orig)
    finally:
        s.close()


def test_edge_values_encode_like_a_commit(r1):
    L, M, D, N = 0, 1, 2, -1
    spheres = [(F(3 * i), F(0), F(0), F(1), L, F(0.5), F(0.5), F(0.5), F(0)) for i in range(12)]
    spheres[3] = (F(9), F(0), F(0), F(0), N, F(0), F(0), F(0), F(0))            # never hit: radius 0
    spheres[4] = (F(12), F(0), F(0), F(-1), N, F(0), F(0), F(0), F(0))          # never hit: negative radius
    cam = cam22(r1)
    s = Fresh(r1, cam, spheres)
    try:
        nan = F(np.nan)
        kind = [M, M, D, L, L, D, D, L, M, M, L, D]
        albedo = [(-0.5, 0.2, 2.0), (1, 1, 1), (0, 0, 0), (0.1, 0.2, 0.3), (0.4, 0.5, 0.6), (1, 1, 1), (1, 1, 1), (-1, -2, -3),
                  (0.9, 0.1, 0.5), (0.3, 0.3, 0.3), (7, 8, 9), (1, 1, 1)]
        param = [1.7, nan, 1.0, 0, 0, 24.2, 1.5, -3.0, -0.5, 1.0, 0.25, 1.5]   # fuzz > 1, NaN fuzz, ior 1 / 24.2 / 1.5, fuzz < 0
        steps = [(0, {"kind": kind, "albedo": albedo, "param": param}),
                 # kind switches in each direction, kept params: METAL -> DIELECTRIC (kept fuzz 1), DIELECTRIC -> METAL with kept
                 # ior 1 and 24.2 (clamped to 1), DIELECTRIC -> LAMBERT, LAMBERT -> METAL (kept -3), NONE on spheres never hit
                 (0, {"kind": [D, M, M, N, N, M, L, M, M, M, L, D]}),
                 (5, {"param": [2.0, nan, 1.5, 0.5]}),                          # METAL 2 -> 1, LAMBERT NaN kept, METAL 1.5 -> 1
                 (3, {"kind": [L, D], "param": [0.0, 1.5]}),                      # spheres never hit take any kind
                 (9, {"albedo": [(-0.0, 0.0, np.inf)] * 3})]
        cur = list(spheres)
        for first, args in steps:
            set_materials(s, first, **args)
            cur = with_materials(cur, first, **args)
            records_equal(r1, s, cur, cam, "edge values at %d: %s" % (first, sorted(args)))
        assert cur[5][4] == M and cur[5][8] == 1 and np.isnan(cur[6][8]) and cur[0][4] == D and cur[0][8] == 1
        # radius +inf: inv_radius 0, never hit, so NONE is accepted here (r1_scene_add_sphere refuses it for radius > 0)
        inf_sphere = [(F(0), F(0), F(0), F(np.inf), L, F(0.5), F(0.5), F(0.5), F(0))] + spheres[1:]
        t = Fresh(r1, cam, inf_sphere)
        try:
            before = t.device_records()
            set_materials(t, 0, kind=[N])
            after = t.device_records()
            geo = 32 * 16 + 16                                                   # shade record [2 * 0 + 1]; n_pad = 16
            assert after[geo:geo + 16].view(np.int32)[1] == N and after[geo:geo + 4].view(F)[0] == 0
            after[geo + 4:geo + 8] = before[geo + 4:geo + 8]
            assert np.array_equal(after, before), "only the kind changes"
        finally:
            t.close()
    finally:
        s.close()


# ---- 2. renders ----------------------------------------------------------------------------------------------------------

def render_variants(r1, n):
    v = [r1.VARIANT_MEGAKERNEL, r1.VARIANT_MEGAKERNEL_PACKED, r1.VARIANT_MEGAKERNEL_SCALAR, r1.VARIANT_WAVEFRONT, r1.VARIANT_MEGAKERNEL_TENSOR_STREAM]
    if n <= 768:
        v.append(r1.VARIANT_MEGAKERNEL_TENSOR)
    return v


def same_render(r1, a, b, case, variant, what, sums=False):
    w, h, spp, rank, world = case
    x, rx = a.render(w, h, spp, rank=rank, world=world, variant=variant)
    y, ry = b.render(w, h, spp, rank=rank, world=world, variant=variant)
    assert np.array_equal(x, y) and rx.num_rays == ry.num_rays, (what, case, variant)
    if sums:
        _, sx, _ = a.render_sums(w, h, spp, rank=rank, world=world, variant=variant)
        _, sy, _ = b.render_sums(w, h, spp, rank=rank, world=world, variant=variant)
        assert np.array_equal(sx, sy), (what, case, variant, "sums")


@pytest.mark.parametrize("change", ("camera", "materials", "both"))
@pytest.mark.parametrize("name", ("large", "n769"))
def test_changed_scenes_render_like_fresh_ones(r1, base, name, change):
    spheres, cam = base[name]
    host_tree, dev_tree = Fresh(r1, cam, spheres), Fresh(r1, cam, spheres)
    try:
        host_tree.build_bvh(r1.BVH_BUILD_HOST)
        dev_tree.build_bvh(r1.BVH_BUILD_DEVICE)
        rng = np.random.default_rng(5)
        cur_cam, cur = cam, list(spheres)
        for frame in range(2):
            if change in ("camera", "both"):
                cur_cam = orbit_of(r1, name, frame)
                for s in (host_tree, dev_tree):
                    s.move_camera(cur_cam)
            if change in ("materials", "both"):
                kind, albedo, param = random_materials(rng, cur, 0, len(cur))
                for s in (host_tree, dev_tree):
                    set_materials(s, 0, kind, albedo, param)
                cur = with_materials(cur, 0, kind, albedo, param)
            f = Fresh(r1, cur_cam, cur)
            try:
                what = "%s %s frame %d" % (name, change, frame)
                for case in RENDER_CASES:
                    for v in render_variants(r1, len(spheres)):
                        same_render(r1, host_tree, f, case, v, what, sums=case is RENDER_CASES[0])
                    same_render(r1, host_tree, f, case, r1.VARIANT_MEGAKERNEL_BVH, what + ", host tree", sums=case is RENDER_CASES[0])
                    same_render(r1, dev_tree, f, case, r1.VARIANT_MEGAKERNEL_BVH, what + ", device tree")
                assert np.array_equal(host_tree.camera(), cam)                    # the host scene keeps its camera
            finally:
                f.close()
    finally:
        host_tree.close()
        dev_tree.close()


def test_parity_calls_see_the_new_camera_and_materials(r1, base):
    spheres, cam = base["large"]
    s = Fresh(r1, cam, spheres)
    try:
        rng = np.random.default_rng(9)
        kind, albedo, param = random_materials(rng, spheres, 0, len(spheres))
        new_cam = orbit_of(r1, "large", 3)
        s.move_camera(new_cam)
        set_materials(s, 0, kind, albedo, param)
        f = Fresh(r1, new_cam, with_materials(spheres, 0, kind, albedo, param))
        try:
            n = 4000
            su, tv, disk = rng.uniform(0, 1, n).astype(F), rng.uniform(0, 1, n).astype(F), rng.uniform(-0.7, 0.7, (n, 2)).astype(F)
            for a, b in zip(s.get_ray(su, tv, disk), f.get_ray(su, tv, disk)):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "get_ray"
            real = np.array([i for i, sp in enumerate(spheres) if can_hit(sp)])
            unit = lambda v: (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(F)  # noqa: E731
            d, nrm = unit(rng.normal(size=(n, 3))), unit(rng.normal(size=(n, 3)))
            p = rng.normal(scale=5, size=(n, 3)).astype(F)
            ball = (unit(rng.normal(size=(n, 3))) * rng.uniform(0, 1, (n, 1)) ** (1 / 3)).astype(F)
            idx, ru = rng.choice(real, n).astype(np.int32), rng.uniform(0, 1, n).astype(F)
            for a, b in zip(s.scatter(d, p, nrm, idx, ball, ru), f.scatter(d, p, nrm, idx, ball, ru)):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "scatter"
            m = 256
            xy = np.stack([rng.integers(0, 96, m), rng.integers(0, 54, m)], 1).astype(np.int32)
            st, st4 = rng.integers(1, 2 ** 32, m, dtype=np.uint64).astype(np.uint32), rng.integers(1, 2 ** 32, (m, 4), dtype=np.uint64).astype(np.uint32)
            (ca, ra), (cb, rb) = s.replay_pixels(xy, 96, 54, 2, st, st4), f.replay_pixels(xy, 96, 54, 2, st, st4)
            assert np.array_equal(ca.view(np.uint32), cb.view(np.uint32)) and np.array_equal(ra, rb), "replay_pixels"
            f0 = Fresh(r1, cam, spheres)
            try:
                assert not np.array_equal(ca, f0.replay_pixels(xy, 96, 54, 2, st, st4)[0]), "the change is visible"
            finally:
                f0.close()
            # r1_trace_rays reads neither: the same hits as before the change
            o = rng.normal(scale=8, size=(n, 3)).astype(F) + F([0, 2, 0])
            assert_same(s.trace_rays(o, d), f.trace_rays(o, d), "trace_rays")
        finally:
            f.close()
    finally:
        s.close()


# ---- 3. the whole frame loop ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ("large", "n5048"))
def test_frames_of_moved_spheres_camera_and_materials_equal_fresh_scenes(r1, base, name):
    """per frame: move_spheres (with refit) + move_camera + set_materials, then BVH and TENSOR_STREAM renders against a fresh scene"""
    spheres, cam = base[name]
    s = Fresh(r1, cam, spheres)
    try:
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        rng = np.random.default_rng(21)
        c0 = centres_of(spheres)
        vel = rng.normal(scale=0.25, size=c0.shape)
        cur = list(spheres)
        for frame in range(4):
            c = (c0 + frame * vel).astype(F)
            s.move_spheres(cuda(c))
            fc = orbit_of(r1, name, frame)
            s.move_camera(fc)
            first = frame * len(cur) // 8
            k = len(cur) - first
            kind, albedo, param = random_materials(rng, cur, first, k)
            set_materials(s, first, kind, albedo if frame % 2 == 0 else None, param)
            cur = with_materials(with_values(cur, 0, c), first, kind, albedo if frame % 2 == 0 else None, param)
            f = Fresh(r1, fc, cur)
            try:
                assert np.array_equal(s.device_records(), f.device_records()), "frame %d records" % frame
                for case in ((96, 54, 8, 0, 1), (96, 54, 8, 1, 3)):
                    for v in (r1.VARIANT_MEGAKERNEL_BVH, r1.VARIANT_MEGAKERNEL_TENSOR_STREAM):
                        same_render(r1, s, f, case, v, "%s frame %d" % (name, frame), sums=True)
            finally:
                f.close()
    finally:
        s.close()


# ---- 4. ordering ---------------------------------------------------------------------------------------------------------

def device_render(s, st, w, h, spp, **kw):
    rgb = torch.zeros(w * h * 3, dtype=torch.uint8, device="cuda:0")
    rays = torch.zeros(1, dtype=torch.int64, device="cuda:0")
    s.render_device(rgb.data_ptr(), rays.data_ptr(), st.cuda_stream, width=w, height=h, spp=spp, **kw)
    return rgb, rays


def same_as(pair, f, w, h, spp):
    want, res = f.render(w, h, spp)
    return np.array_equal(pair[0].cpu().numpy().reshape(want.shape), want) and int(pair[1].item()) == res.num_rays


def test_an_enqueued_render_keeps_its_camera(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        w, h, spp = 64, 36, 4
        st = torch.cuda.Stream(0)
        new_cam = orbit_of(r1, "n769", 1)
        with torch.cuda.stream(st):
            torch.cuda._sleep(1_000_000_000)                              # keeps the first render queued while the camera moves
            before = device_render(s, st, w, h, spp)
            s.move_camera(new_cam)
            after = device_render(s, st, w, h, spp)
        assert not st.query(), "the stream finished before the camera moved: the test proves nothing"
        st.synchronize()
        f0, f = Fresh(r1, cam, spheres), Fresh(r1, new_cam, spheres)
        try:
            assert same_as(before, f0, w, h, spp) and same_as(after, f, w, h, spp)
            assert not np.array_equal(before[0].cpu().numpy(), after[0].cpu().numpy())
        finally:
            f0.close()
            f.close()
    finally:
        s.close()


def test_materials_on_a_torch_stream_are_ordered_between_renders(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        w, h, spp = 64, 36, 4
        st = torch.cuda.Stream(0)
        kind, albedo, param = random_materials(np.random.default_rng(4), spheres, 0, len(spheres))
        with torch.cuda.stream(st):
            d_albedo = torch.zeros(len(spheres), 3, dtype=torch.float32, device="cuda:0")
            d_albedo.copy_(cuda(albedo))                                    # produced on the stream, consumed by the change after it
            before = device_render(s, st, w, h, spp)
            s.set_materials(torch.from_numpy(kind).cuda(0), d_albedo, cuda(param))
            after = device_render(s, st, w, h, spp)
        st.synchronize()
        f0, f = Fresh(r1, cam, spheres), Fresh(r1, cam, with_materials(spheres, 0, kind, albedo, param))
        try:
            assert same_as(before, f0, w, h, spp) and same_as(after, f, w, h, spp)
            assert not np.array_equal(before[0].cpu().numpy(), after[0].cpu().numpy())
        finally:
            f0.close()
            f.close()
    finally:
        s.close()


def test_a_new_camera_rebuilds_the_wavefront_graph_once(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        builds = lambda: r1.lib.r1_wavefront_graph_builds(0)  # noqa: E731
        wf = dict(variant=r1.VARIANT_WAVEFRONT)
        s.render(160, 90, 8, **wf)
        n0 = builds()
        s.render(160, 90, 8, **wf)
        assert builds() == n0, "same arguments: no rebuild"
        new_cam = orbit_of(r1, "n769", 2)
        s.move_camera(new_cam)
        a, ra = s.render(160, 90, 8, **wf)
        assert builds() == n0 + 1, "a new camera: rebuilt once"
        s.render(160, 90, 8, **wf)
        s.move_camera(new_cam.copy())
        s.render(160, 90, 8, **wf)
        assert builds() == n0 + 1, "an unchanged camera: no rebuild"
        kind, albedo, param = random_materials(np.random.default_rng(8), spheres, 0, len(spheres))
        set_materials(s, 0, kind, albedo, param)
        b, rb = s.render(160, 90, 8, **wf)
        assert builds() == n0 + 1, "new materials: the graph reads them from the same records"
        for img, res, sph in ((a, ra, spheres), (b, rb, with_materials(spheres, 0, kind, albedo, param))):
            f = Fresh(r1, new_cam, sph)
            try:
                want, rw = f.render(160, 90, 8, **wf)
                assert np.array_equal(img, want) and res.num_rays == rw.num_rays
            finally:
                f.close()
    finally:
        s.close()


# ---- 5. refusals and state -----------------------------------------------------------------------------------------------

def test_refusals_leave_every_byte_in_place(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        rec = s.device_records()
        n = len(spheres)
        real = [i for i, sp in enumerate(spheres) if can_hit(sp)]
        never = [i for i, sp in enumerate(spheres) if not can_hit(sp)]
        kind, albedo, param = random_materials(np.random.default_rng(3), spheres, 0, n)
        bad = []
        for v in (3, -2, 2 ** 31 - 1, -2 ** 31):
            k = kind.copy(); k[real[5]] = v; bad.append((k, "kind %d" % v))
        k = kind.copy(); k[never[0]] = 7; bad.append((k, "kind 7 on a sphere never hit"))
        k = kind.copy(); k[real[-1]] = r1.MAT_NONE; bad.append((k, "NONE on a sphere that can be hit"))
        for k, what in bad:
            with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
                set_materials(s, 0, k, albedo, param)
            assert np.array_equal(s.device_records(), rec), what
        for first, k in ((n - 5, 10), (n, 1)):
            with pytest.raises(r1.Rays1Error, match=r"\(-1\).*out of range"):
                set_materials(s, first, param=np.ones(k, F))
        assert np.array_equal(s.device_records(), rec)
        # the Python refusals of bad tensors
        good = cuda(albedo)
        for kw, match in (({"kind": torch.from_numpy(kind).cuda(0).long()}, "int32"), ({"albedo": good.double()}, "float32"),
                          ({"albedo": good.t()}, "contiguous|shape"), ({"albedo": good[:, :2].contiguous()}, "shape"),
                          ({"param": cuda(param).reshape(-1, 1)}, "shape"), ({"albedo": good, "param": cuda(param[:3])}, "shape"),
                          ({"kind": torch.from_numpy(kind).cuda(0), "albedo": good[:5]}, "shape"), ({"param": cuda(param).cpu()}, "CUDA")):
            with pytest.raises(ValueError, match=match):
                s.set_materials(**kw)
        if torch.cuda.device_count() > 1:
            with pytest.raises(ValueError, match="device"):
                s.set_materials(albedo=good, device=1)
            with pytest.raises(ValueError, match="device"):
                s.set_materials(albedo=good, param=cuda(param).cuda(1))
        assert np.array_equal(s.device_records(), rec)
    finally:
        s.close()


def test_state_rules(r1, base):
    spheres, cam = base["n17"]
    u = Fresh(r1, cam, spheres, commit=False)
    try:
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):                # not committed
            u.move_camera(cam)
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            set_materials(u, 0, param=np.ones(3, F))
    finally:
        u.close()
    s = Fresh(r1, cam, spheres)
    try:
        orig = s.device_records()
        host = (s.soa(), s.camera(), s.tensor_operand(), s.bvh())
        base_rgb, r0 = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        new_cam = orbit(r1, 1, 30.0)
        kind, albedo, param = random_materials(np.random.default_rng(6), spheres, 0, len(spheres))
        s.move_camera(new_cam)
        set_materials(s, 0, kind, albedo, param)
        # a material change keeps the geometry: a BVH render on a device without a tree uploads the host tree
        f = Fresh(r1, new_cam, with_materials(spheres, 0, kind, albedo, param))
        try:
            same_render(r1, s, f, (48, 27, 4, 0, 1), r1.VARIANT_MEGAKERNEL_BVH, "host tree uploaded after new materials")
            nodes, leaves, depth = s.bvh_on_device()
            assert (nodes.tobytes(), leaves.tobytes(), depth) == (host[3][0].tobytes(), host[3][1].tobytes(), host[3][2])
            s.build_bvh(r1.BVH_BUILD_HOST)                                  # still allowed: nothing moved
            changed = s.device_records()
            n_pad = (len(spheres) + 15) // 16 * 16                          # [scan | exact | shade | operand]: 16, 16, 32 bytes
            assert np.array_equal(changed[:32 * n_pad], orig[:32 * n_pad]), "scan and exact records are kept"
            assert np.array_equal(changed[64 * n_pad:], orig[64 * n_pad:]), "the tensor operand is kept"
            assert np.array_equal(changed, f.device_records())
        finally:
            f.close()
        # the host getters describe the committed scene
        got = (s.soa(), s.camera(), s.tensor_operand(), s.bvh())
        for k in host[0]:
            assert np.array_equal(got[0][k].view(np.uint8), host[0][k].view(np.uint8)), k
        assert np.array_equal(got[1], host[1]) and np.array_equal(got[2], host[2])
        assert got[3][0].tobytes() == host[3][0].tobytes()
        # spheres changed on the host after the commit
        r1._check(r1.lib.r1_scene_add_sphere(s.handle, 0, 0, 0, 1, r1.MAT_LAMBERT, 0.5, 0.5, 0.5, 0), "add")
        with pytest.raises(r1.Rays1Error, match=r"\(-2\).*commit it again"):
            s.move_camera(cam)
        with pytest.raises(r1.Rays1Error, match=r"\(-2\).*commit it again"):
            set_materials(s, 0, param=np.ones(3, F))
        # a re-commit restores the host's camera and materials
        t = Fresh(r1, cam, spheres)
        try:
            t.move_camera(new_cam)
            set_materials(t, 0, kind, albedo, param)
            r1._check(r1.lib.r1_scene_commit(t.handle, 0), "commit")
            assert np.array_equal(t.device_records(), orig)
            rgb, res = t.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_PACKED)
            assert np.array_equal(rgb, base_rgb) and res.num_rays == r0.num_rays
        finally:
            t.close()
    finally:
        s.close()


def test_changes_touch_only_their_device(r1, base):
    if r1.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        r1._check(r1.lib.r1_scene_commit(s.handle, 1), "commit")
        rec0 = s.device_records(0)
        rgb0, r0 = s.render(64, 36, 4, device=0)
        kind, albedo, param = random_materials(np.random.default_rng(12), spheres, 0, len(spheres))
        new_cam = orbit_of(r1, "n769", 4)
        s.move_camera(new_cam, device=1)
        dev1 = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda(1)  # noqa: E731
        s.set_materials(dev1(kind, np.int32), dev1(albedo, F), dev1(param, F))
        assert np.array_equal(s.device_records(0), rec0)
        rgb, res = s.render(64, 36, 4, device=0)
        assert np.array_equal(rgb, rgb0) and res.num_rays == r0.num_rays
        f = Fresh(r1, new_cam, with_materials(spheres, 0, kind, albedo, param))
        try:
            assert np.array_equal(s.device_records(1), f.device_records())
            want, rw = f.render(64, 36, 4)
            got, rg = s.render(64, 36, 4, device=1)
            assert np.array_equal(got, want) and rg.num_rays == rw.num_rays
        finally:
            f.close()
    finally:
        s.close()
