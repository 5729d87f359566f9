"""Moving spheres on the device (r1_scene_move_spheres, DESIGN.md section 4.10) on the GPU.

After a move, a device holds exactly the records r1_scene_commit writes for a scene with the moved values (compared byte for byte
with a fresh scene of those values, committed from the host), and its BVH, host-built or device-built, equals the refit's CPU
restatement (tests/refit_restatement.py).  Renders and traces of a moved scene equal the fresh scene's for every variant.  Also:
refusals leave every byte in place, the state rules after a move, streams, a second GPU and a 10^6-sphere cloud."""
import os
import sys

import numpy as np
import pytest

import lbvh_restatement as lbvh
import refit_restatement as refit
from conftest import ROOT
from test_bvh_cpu import check_structure
from test_bvh_gpu import RENDER_CASES
from test_scan_edges_gpu import FLT_MAX
from test_tensor_stream_gpu import assert_same

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene  # noqa: E402

torch = pytest.importorskip("torch")
F = np.float32


# ---- scenes --------------------------------------------------------------------------------------------------------------

class Fresh:
    """a scene from explicit spheres (cx, cy, cz, radius, kind, r, g, b, param) and 22 raw camera constants, committed to `device`
    through the raw ABI: no padding, so it has exactly these spheres"""

    def __init__(self, r1, cam22, spheres, device=0, commit=True):
        from test_scan_edges_gpu import RawScene
        self.s = RawScene((0, 0, 1, 0, 0, 0, 40, 0, 10), spheres, commit=False)
        self.s.set_camera_raw(cam22, device if commit else None)
        self.spheres = spheres

    def __getattr__(self, name):
        return getattr(self.s, name)


def spheres_of(r1, s):
    """the sphere list of a scene, radii recovered from radius_sq and inv_radius"""
    soa = s.soa()
    out = []
    for i in range(len(soa["cx"])):
        r2, inv = soa["radius_sq"][i], soa["inv_radius"][i]
        if inv == 0:
            r = F(0) if r2 == 0 else -np.sqrt(r2, dtype=F)
            cands = [r, np.nextafter(r, F(0)), np.nextafter(r, F(-np.inf))]
        else:
            r = F(1) / inv
            cands = [r, np.nextafter(r, F(0)), np.nextafter(r, F(np.inf)), np.sqrt(r2, dtype=F)]
        for c in cands:
            if F(c * c) == r2 and (F(1) / c if c > 0 else F(0)) == inv:
                break
        else:
            raise AssertionError("sphere %d: no radius gives radius_sq %r and inv_radius %r" % (i, r2, inv))
        kind = int(soa["kind"][i])
        out.append((soa["cx"][i], soa["cy"][i], soa["cz"][i], F(c), kind, *soa["albedo"][i], soa["param"][i]))
    return out


def with_values(spheres, first, centres, radii=None):
    out = list(spheres)
    for j in range(len(centres)):
        sp = list(out[first + j])
        sp[0:3] = [F(v) for v in centres[j]]
        if radii is not None:
            sp[3] = F(radii[j])
        out[first + j] = tuple(sp)
    return out


def random_spheres(r1, n, seed):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-3 * n ** (1 / 3) - 2, 3 * n ** (1 / 3) + 2, (n, 3)).astype(F)
    r = rng.uniform(0.2, 1.5, n).astype(F)
    kind = rng.choice([0, 1, 2], n, p=[0.6, 0.25, 0.15])
    out = []
    for i in range(n):
        par = F(1.5) if kind[i] == 2 else F(0.3) if kind[i] == 1 else F(0)
        out.append((c[i, 0], c[i, 1], c[i, 2], r[i], int(kind[i]), F(0.7), F(0.5), F(0.3), par))
    if n > 3:
        out[n // 2] = (F(0), F(-1000), F(0), F(0), r1.MAT_NONE, F(0), F(0), F(0), F(0))     # a sphere that can never be hit
    return out


CAM22 = None


def cam22(r1):
    global CAM22
    if CAM22 is None:
        s = r1.create_scene("medium", commit=False)
        CAM22 = s.camera()
        s.close()
    return CAM22


ENCODE_SCENES = ("large", "synth4096", "n1", "n17", "n769", "n5048", "cloud")


@pytest.fixture(scope="module")
def base(r1):
    """name -> sphere list and camera of the module's scenes"""
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


def centres_of(spheres):
    return np.array([sp[:3] for sp in spheres], F).reshape(-1, 3)


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, F)).cuda(0)


def records_equal(r1, moved, spheres, cam, what):
    f = Fresh(r1, cam, spheres)
    try:
        a, b = moved.device_records(), f.device_records()
        assert a.nbytes == b.nbytes, what
        if not np.array_equal(a, b):
            i = int(np.nonzero(a != b)[0][0])
            raise AssertionError("%s: device records differ from a fresh commit's at byte %d of %d" % (what, i, a.nbytes))
    finally:
        f.close()


# ---- 1. encoding ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ENCODE_SCENES)
def test_moved_records_equal_a_fresh_commit(r1, base, name):
    spheres, cam = base[name]
    n = len(spheres)
    s = Fresh(r1, cam, spheres)
    try:
        orig = s.device_records()
        rng = np.random.default_rng(n)
        c0 = centres_of(spheres)
        moves = [(0, n, True), (0, n, False), (n // 3, max(1, n // 4), True), (n - 1, 1, False), (n // 2, n - n // 2, True)]
        cur = list(spheres)
        for first, k, with_r in moves:
            c = (c0[first:first + k] + rng.normal(scale=0.5, size=(k, 3))).astype(F)
            radii = None
            if with_r:
                old = np.array([sp[3] for sp in cur[first:first + k]], F)
                radii = np.where(old > 0, old * rng.uniform(0.5, 1.5, k).astype(F), old).astype(F)
            ms = s.move_spheres(cuda(c), cuda(radii) if radii is not None else None, first=first)
            assert ms >= 0
            cur = with_values(cur, first, c, radii)
            records_equal(r1, s, cur, cam, "%s move %d+%d radii=%s" % (name, first, k, with_r))
        # moving back restores the original bytes
        s.move_spheres(cuda(c0), cuda(np.array([sp[3] for sp in spheres], F)))
        assert np.array_equal(s.device_records(), orig)
    finally:
        s.close()


def test_edge_values_encode_like_a_commit(r1, base):
    spheres, cam = base["n17"]
    s = Fresh(r1, cam, spheres)
    try:
        tiny = np.float32(1e-40)
        c = np.array([[0, -0.0, 0], [-0.0, -0.0, -0.0], [tiny, -tiny, 1e-45], [3e38, 3e38, 3e38], [-3e38, 1, 3e38], [1e19, -1e19, 1e19],
                      [1e-30, 2e-30, -3e-30], [5, 5, 5]], F)
        radii = np.array([1, 2, 1e-23, 1.8e19, 1e-3, 1e18, 1e-23, 1e-44], F)       # 1e-23: radius_sq underflows to 0; 1e-44: 1 / r is inf
        old = np.array([sp[3] for sp in spheres[:len(c)]], F)
        radii = np.where(old > 0, radii, old).astype(F)
        assert F(radii[2] * radii[2]) == 0 or old[2] <= 0
        s.move_spheres(cuda(c), cuda(radii))
        records_equal(r1, s, with_values(spheres, 0, c, radii), cam, "edge values")
        s.move_spheres(cuda(c[::-1].copy()), first=9)
        records_equal(r1, s, with_values(with_values(spheres, 0, c, radii), 9, c[::-1]), cam, "edge values, kept radii")
    finally:
        s.close()


# ---- 2. refit ------------------------------------------------------------------------------------------------------------

def tree_bytes(tree):
    return tree[0].tobytes(), tree[1].tobytes(), tree[2]


@pytest.mark.parametrize("builder", ("host", "device"))
@pytest.mark.parametrize("name", ("large", "n769", "n5048", "cloud"))
def test_refit_equals_the_restatement(r1, base, name, builder):
    spheres, cam = base[name]
    s = Fresh(r1, cam, spheres)
    try:
        s.build_bvh(r1.BVH_BUILD_HOST if builder == "host" else r1.BVH_BUILD_DEVICE)
        tree = s.bvh() if builder == "host" else lbvh.build(s.soa())
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(tree)
        c0 = centres_of(spheres)
        s.move_spheres(cuda(c0))                                          # unchanged positions: the identity
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(tree)
        rng = np.random.default_rng(7)
        span = float(np.abs(c0).max())
        for step, scale in enumerate((0.01, 0.2, 1.0)):                  # jitter, then motion that tangles the tree
            c = (c0 + rng.normal(scale=scale * span ** 0.5, size=c0.shape)).astype(F) if step < 2 else c0[rng.permutation(len(c0))]
            s.move_spheres(cuda(c))
            cur = with_values(spheres, 0, c)
            f = Fresh(r1, cam, cur)
            try:
                got = s.bvh_on_device()
                want = refit.refit(tree, refit.exact_of(f.soa()))
                assert tree_bytes(got) == tree_bytes(want), "%s %s step %d" % (name, builder, step)
                check_structure(f, *got)
                assert np.array_equal(s.device_records(), f.device_records())
            finally:
                f.close()
        s.build_bvh(r1.BVH_BUILD_DEVICE)                                   # a rebuild reads the moved records
        f = Fresh(r1, cam, cur, commit=False)
        try:
            assert tree_bytes(s.bvh_on_device()) == tree_bytes(lbvh.build(f.soa()))
        finally:
            f.close()
    finally:
        s.close()


# ---- 3. renders and traces -----------------------------------------------------------------------------------------------

def variants(r1, n):
    v = [r1.VARIANT_MEGAKERNEL, r1.VARIANT_MEGAKERNEL_PACKED, r1.VARIANT_MEGAKERNEL_SCALAR, r1.VARIANT_MEGAKERNEL_COOP,
         r1.VARIANT_MEGAKERNEL_DEFERRED, r1.VARIANT_MEGAKERNEL_DUAL, r1.VARIANT_WAVEFRONT, r1.VARIANT_MEGAKERNEL_TENSOR_STREAM]
    if n <= 768:
        v.append(r1.VARIANT_MEGAKERNEL_TENSOR)
    return v


def same_render(r1, a, b, case, variant, what):
    w, h, spp, rank, world = case
    x, rx = a.render(w, h, spp, rank=rank, world=world, variant=variant)
    y, ry = b.render(w, h, spp, rank=rank, world=world, variant=variant)
    assert np.array_equal(x, y) and rx.num_rays == ry.num_rays, (what, case, variant)


@pytest.mark.parametrize("name", ("large", "n769"))
def test_moved_scenes_render_like_fresh_ones(r1, oracle, base, name):
    spheres, cam = base[name]
    host_tree, dev_tree = Fresh(r1, cam, spheres), Fresh(r1, cam, spheres)
    try:
        host_tree.build_bvh(r1.BVH_BUILD_HOST)
        dev_tree.build_bvh(r1.BVH_BUILD_DEVICE)
        c0 = centres_of(spheres)
        rng = np.random.default_rng(11)
        vel = rng.normal(scale=0.3, size=c0.shape)
        for frame in range(3):
            c = (c0 + frame * vel).astype(F)
            for s in (host_tree, dev_tree):
                s.move_spheres(cuda(c))
            f = Fresh(r1, cam, with_values(spheres, 0, c))
            try:
                for case in RENDER_CASES:
                    for v in variants(r1, len(spheres)):
                        same_render(r1, host_tree, f, case, v, "%s frame %d" % (name, frame))
                    same_render(r1, host_tree, f, case, r1.VARIANT_MEGAKERNEL_BVH, "%s frame %d, refit host tree" % (name, frame))
                    same_render(r1, dev_tree, f, case, r1.VARIANT_MEGAKERNEL_BVH, "%s frame %d, refit device tree" % (name, frame))
                # rays against the oracle on the moved scene
                soa = f.soa()
                real = np.nonzero(soa["inv_radius"] > 0)[0]
                from test_scan_edges_gpu import aimed_rays
                o, d = aimed_rays(soa, rng.choice(real, 1500), rng, rng.choice([1.0, 20.0, 400.0], 1500))
                o, d = o.astype(F), d.astype(F)
                so = oracle.scene_create_from_soa(soa)
                try:
                    want = oracle.hit(so, o, d, 0.001, FLT_MAX)
                finally:
                    oracle.scene_destroy(so)
                for v in (r1.VARIANT_MEGAKERNEL_PACKED, r1.VARIANT_MEGAKERNEL_BVH):
                    assert_same(host_tree.trace_rays(o, d, 0.001, FLT_MAX, variant=v), want, "%s frame %d variant %d" % (name, frame, v))
                    assert_same(dev_tree.trace_rays(o, d, 0.001, FLT_MAX, variant=v), want, "%s frame %d variant %d" % (name, frame, v))
                dev_tree.build_bvh(r1.BVH_BUILD_DEVICE)                  # a rebuilt device tree renders alike too
                for case in RENDER_CASES:
                    same_render(r1, dev_tree, f, case, r1.VARIANT_MEGAKERNEL_BVH, "%s frame %d, rebuilt device tree" % (name, frame))
            finally:
                f.close()
    finally:
        host_tree.close()
        dev_tree.close()


# ---- 4. refusals and state -----------------------------------------------------------------------------------------------

def test_refusals_leave_every_byte_in_place(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        rec, tree = s.device_records(), tree_bytes(s.bvh_on_device())
        c = centres_of(spheres)
        real = [i for i, sp in enumerate(spheres) if sp[3] > 0]
        never = [i for i, sp in enumerate(spheres) if not sp[3] > 0]
        r = np.array([sp[3] for sp in spheres], F)
        bad = []
        r0 = r.copy(); r0[real[5]] = 0; bad.append((c, r0, "can no longer be hit"))
        rn = r.copy(); rn[never[0]] = 1; bad.append((c, rn, "could now be hit"))
        ri = r.copy(); ri[real[7]] = np.inf; bad.append((c, ri, "infinite radius"))
        rq = r.copy(); rq[real[8]] = 1e20; bad.append((c, rq, "radius_sq overflows"))
        cn = c.copy(); cn[real[9], 1] = np.nan; bad.append((cn, None, "NaN centre"))
        ci = c.copy(); ci[real[-1], 2] = -np.inf; bad.append((ci, r, "infinite centre"))
        for cc, rr, what in bad:
            with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
                s.move_spheres(cuda(cc), cuda(rr) if rr is not None else None)
            assert np.array_equal(s.device_records(), rec), what
            assert tree_bytes(s.bvh_on_device()) == tree, what
        with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
            s.move_spheres(cuda(c[:10]), first=len(c) - 5)
        cn = c.copy(); cn[never[0]] = np.nan                              # a sphere that can never be hit may take any value
        s.move_spheres(cuda(cn))
        records_equal(r1, s, with_values(spheres, 0, cn), cam, "NaN centre of a sphere that can never be hit")
    finally:
        s.close()


def test_state_rules(r1, base):
    spheres, cam = base["n17"]
    u = Fresh(r1, cam, spheres, commit=False)
    try:
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):                # not committed
            u.move_spheres(cuda(centres_of(spheres)))
    finally:
        u.close()
    s = Fresh(r1, cam, spheres)
    try:
        orig = s.device_records()
        c = centres_of(spheres) + F(0.25)
        s.move_spheres(cuda(c))
        with pytest.raises(r1.Rays1Error, match=r"\(-2\).*R1_BVH_BUILD_DEVICE"):
            s.render(32, 18, 2, variant=r1.VARIANT_MEGAKERNEL_BVH)
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            s.trace_rays(np.zeros((1, 3), F), np.array([[0, 0, -1]], F), variant=r1.VARIANT_MEGAKERNEL_BVH)
        with pytest.raises(r1.Rays1Error, match=r"\(-2\)"):
            s.build_bvh(r1.BVH_BUILD_HOST)
        assert np.array_equal(s.soa()["cx"], centres_of(spheres)[:, 0])  # the host scene keeps its values
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        f = Fresh(r1, cam, with_values(spheres, 0, c))
        try:
            same_render(r1, s, f, (48, 27, 4, 0, 1), r1.VARIANT_MEGAKERNEL_BVH, "after a device build")
        finally:
            f.close()
        r1._check(r1.lib.r1_scene_commit(s.handle, 0), "commit")          # a re-commit restores the host records and the host tree
        assert np.array_equal(s.device_records(), orig)
        base_rgb, r0 = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        rgb, res = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)
        assert np.array_equal(rgb, base_rgb) and res.num_rays == r0.num_rays
        assert tree_bytes(s.bvh_on_device()) == tree_bytes(s.bvh())
        s.build_bvh(r1.BVH_BUILD_HOST)
    finally:
        s.close()


def test_python_refuses_bad_tensors(r1, base):
    spheres, cam = base["n17"]
    s = Fresh(r1, cam, spheres)
    try:
        rec = s.device_records()
        c = cuda(centres_of(spheres))
        for bad, match in ((c.double(), "float32"), (c.t(), "contiguous|shape"), (c[:, :2].contiguous(), "shape"), (c.cpu(), "CUDA")):
            with pytest.raises(ValueError, match=match):
                s.move_spheres(bad)
        with pytest.raises(ValueError, match="shape"):
            s.move_spheres(c, radii=cuda(np.ones(3, F)))
        if torch.cuda.device_count() > 1:
            with pytest.raises(ValueError, match="device"):
                s.move_spheres(c, device=1)
        assert np.array_equal(s.device_records(), rec)
    finally:
        s.close()


# ---- 5. streams ----------------------------------------------------------------------------------------------------------

def test_a_move_on_a_torch_stream_is_ordered_between_renders(r1, base):
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        w, h, spp = 64, 36, 4
        st = torch.cuda.Stream(0)
        rgb = [torch.zeros(w * h * 3, dtype=torch.uint8, device="cuda:0") for _ in range(2)]
        rays = [torch.zeros(1, dtype=torch.int64, device="cuda:0") for _ in range(2)]
        c = centres_of(spheres) + np.float32(0.5)
        with torch.cuda.stream(st):
            d = cuda(np.zeros_like(c))
            d.copy_(cuda(c))                                              # produced on the stream, consumed by the move after it
            s.render_device(rgb[0].data_ptr(), rays[0].data_ptr(), st.cuda_stream, width=w, height=h, spp=spp)
            s.move_spheres(d)
            s.render_device(rgb[1].data_ptr(), rays[1].data_ptr(), st.cuda_stream, width=w, height=h, spp=spp)
        st.synchronize()
        f0, f = Fresh(r1, cam, spheres), Fresh(r1, cam, with_values(spheres, 0, c))
        try:
            before, _ = f0.render(w, h, spp)
            after, res = f.render(w, h, spp)
            assert np.array_equal(rgb[1].cpu().numpy().reshape(after.shape), after) and int(rays[1].item()) == res.num_rays
            assert np.array_equal(rgb[0].cpu().numpy().reshape(before.shape), before)
            assert not np.array_equal(before, after)
        finally:
            f0.close()
            f.close()
    finally:
        s.close()


# ---- 6. more GPUs --------------------------------------------------------------------------------------------------------

def test_a_move_touches_only_its_device(r1, base):
    if r1.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    spheres, cam = base["n769"]
    s = Fresh(r1, cam, spheres)
    try:
        r1._check(r1.lib.r1_scene_commit(s.handle, 1), "commit")
        rec0 = s.device_records(0)
        c = torch.from_numpy(centres_of(spheres) + F(1)).cuda(1)
        s.move_spheres(c)
        assert np.array_equal(s.device_records(0), rec0)
        f = Fresh(r1, cam, with_values(spheres, 0, c.cpu().numpy()))
        try:
            assert np.array_equal(s.device_records(1), f.device_records())
        finally:
            f.close()
    finally:
        s.close()


# ---- 7. scale ------------------------------------------------------------------------------------------------------------

def test_million_sphere_cloud_moved_and_refitted(r1, tmp_path):
    cam, sph = make_scene.cloud_scene(1000000)
    path = str(tmp_path / "cloud.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path)
    try:
        s.build_bvh(r1.BVH_BUILD_DEVICE)
        soa = s.soa()
        c0 = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1)
        rng = np.random.default_rng(2)
        c = (c0 + rng.normal(scale=0.5, size=c0.shape)).astype(F)
        c[-8:] = c0[-8:]                                                  # the ground and the padding stay
        ms = s.move_spheres(cuda(c))
        moved = [tuple(c[i]) + tuple(sp[3:]) for i, sp in enumerate(sph)]
        path2 = str(tmp_path / "cloud_moved.r1scene")
        r1.write_scene_file(path2, cam, moved)
        f = r1.create_scene_from_file(path2)
        try:
            assert np.array_equal(s.device_records(), f.device_records())
            a, ra = s.render(160, 90, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)
            b, rb = f.render(160, 90, 4, variant=r1.VARIANT_MEGAKERNEL_BVH)
            assert np.array_equal(a, b) and ra.num_rays == rb.num_rays
        finally:
            f.close()
        print("cloud 10^6: move + refit %.3f ms" % ms)
    finally:
        s.close()
