"""The filters at every magnitude of the float range, without a GPU.

Every other ray-level and render-level test places its scenes near the world origin.  The three filters in front of the exact test
rest on relative error bounds: the FFMA2 filter of the brute-force scans (margins 2^-17 of S = |o|^2 + |c|^2, DESIGN.md section
4.1), the split-TF32 tensor filter (2^-16 of |c|^2 and of |o|^2, section 4.0) and the BVH box test (2^-9 of distance + diagonal,
section 4.8).  Here the same scenes are moved through a ladder of magnitudes, x -> s x + T with T = 2^k (1, 0.75, -0.5):

    rigid    s = 1, k from 10 to 126: from k ~ 24 on the centres collapse onto the float grid (coincident spheres, ties at scale)
    scaled   s = 2^(k - 12): the layout stays resolvable at every level
    scale    T = 0, s from 2^-12 to 2^60: roots against t_min, and |c| beyond 2^64 with |c - o| small

Beyond |c| = 2^64, |c|^2 overflows float.  The filters' range is |c|^2 < 2^120 and |o|^2 < 2^120 (r1_encode.h kFarC2); outside it
their records make every sphere that can be hit a candidate, and the exact test decides.  Each filter is restated here in numpy
from the records the library writes (the tensor operand) or that r1_encode.h specifies (the scan lanes;
tests/test_magnitudes_gpu.py compares those with the device's records), and must flag every sphere the oracle's Hitable::hit
returns, at every level.  tests/test_magnitudes_gpu.py runs the kernels on the same fixtures."""
import numpy as np
import pytest

import lbvh_restatement as lbvh
import refit_restatement as refit
from conftest import rmse
from test_bvh_cpu import check_conservative, surface_rays, zero_component_rays
from test_scan_edges_gpu import FLT_MAX, T_BOUND, RawScene, aimed_rays, spec
from test_tensor_cpu import ray_rows

F = np.float32
T_DIR = np.array([1.0, 0.75, -0.5])
BASES = ("n120", "ties", "large")
RIGID = (10, 20, 30, 40, 50, 60, 62, 63, 63.5, 64, 65, 70, 100, 126)       # 63.5 stands for T = 1.5 * 2^63
SCALED = (10, 20, 30, 40, 50, 60, 62, 63, 63.5, 64, 65, 70)
SCALE = (-12, -6, 12, 30, 60, 62)
# above scaled 70 the layout's own distances (|c - o| ~ 2^(k - 7)) square beyond float: every exact test misses there, so the
# ladder of hits stops at 70; the renders of tests/test_magnitudes_gpu.py still go to scaled 120
LEVELS = ("level0",) + tuple("rigid%g" % k for k in RIGID) + tuple("scaled%g" % k for k in SCALED) + tuple("scale%d" % e for e in SCALE)
FAR_C2 = 2.0 ** 120                        # r1_encode.h kFarC2
FAR_KK = F(-2.0 ** 122)                    # r1_encode.h kFarKK


def transform(level):
    """(s, T) of a level name: level0, rigid<k>, scaled<k> or scale<e>; k = 63.5 means 1.5 * 2^63"""
    def offset(k):
        return T_DIR * (1.5 * 2.0 ** 63 if k == 63.5 else 2.0 ** k)
    if level == "level0":
        return 1.0, np.zeros(3)
    if level.startswith("rigid"):
        return 1.0, offset(float(level[5:]))
    if level.startswith("scaled"):
        k = float(level[6:])
        return 2.0 ** (int(k) - 12), offset(k)
    return 2.0 ** int(level[5:]), np.zeros(3)


def base_spheres(r1, name):
    """(camera args, sphere tuples) of a base scene: the sweep / tie specs of tests/test_scan_edges_gpu.py, or a built-in scene"""
    if name in ("n120", "ties"):
        return spec(name)
    s = r1.create_scene(name, commit=False)
    soa = s.soa()
    s.close()
    sph = []
    for i in range(len(soa["cx"])):
        inv = soa["inv_radius"][i]
        r0 = F(1) / inv if inv > 0 else -np.sqrt(soa["radius_sq"][i], dtype=F)
        r = next(c for c in (r0, np.nextafter(r0, F(0)), np.nextafter(r0, F(np.inf) if inv > 0 else F(-np.inf)))
                 if F(c * c) == soa["radius_sq"][i] and (F(1) / c if c > 0 else F(0)) == inv)
        sph.append((soa["cx"][i], soa["cy"][i], soa["cz"][i], r, int(soa["kind"][i]), *soa["albedo"][i], soa["param"][i]))
    return (0, 2, 20, 0, 0, 0, 40, 0.0, 20), sph


def moved(sph, s, t):
    """spheres at s x + T (float64, rounded once to float32), radii times s (exact: s is a power of two)"""
    out = []
    for sp in sph:
        c = (np.array(sp[:3], np.float64) * s + t).astype(F)
        out.append((*c, F(F(sp[3]) * F(s)), int(sp[4]), *sp[5:]))
    return out


def move_cam22(cam22, s, t):
    """the 22 raw camera constants under x -> s x + T: origin and lower-left corner mapped, horizontal, vertical and the lens
    radius scaled, u / v / w kept"""
    c = np.array(cam22, np.float64)
    out = c.copy()
    out[0:3] = c[0:3] * s + t
    out[3:6] = c[3:6] * s + t
    out[6:12] = c[6:12] * s
    out[21] = c[21] * s
    return out.astype(F)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def ladder_rays(soa, s, seed=21):
    """aimed rays (centres and +-2 % silhouettes from gaps {1, 20, 400} s), rays from surfaces, from inside spheres, axis-aligned
    rays with +-0 components, and rays from the world origin towards spheres.  Built in float64 at the level, rounded once."""
    rng = np.random.default_rng(seed)
    real = np.nonzero(soa["inv_radius"] > 0)[0]
    with np.errstate(invalid="ignore", divide="ignore"):
        o1, d1 = aimed_rays(soa, rng.choice(real, 900), rng, rng.choice([1.0, 20.0, 400.0], 900) * s)
    o2, d2 = surface_rays(soa, rng, 200)
    i = rng.choice(real, 200)
    ctr = np.stack([soa["cx"][i], soa["cy"][i], soa["cz"][i]], 1).astype(np.float64)
    o3 = ctr + rng.uniform(-0.3, 0.3, ctr.shape) / soa["inv_radius"][i, None]
    d3 = _unit(rng.normal(size=ctr.shape))
    o4, d4 = zero_component_rays(soa, rng, 200)
    j = rng.choice(real, 100)
    c = np.stack([soa["cx"][j], soa["cy"][j], soa["cz"][j]], 1).astype(np.float64)
    o5 = np.zeros_like(c)
    d5 = _unit(c + rng.uniform(-0.5, 0.5, c.shape) / soa["inv_radius"][j, None])
    org = np.concatenate([o1, o2, o3, o4, o5]).astype(F)
    raw = np.concatenate([d1, d2, d3, d4, d5]).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        d = _unit(raw).astype(F)
    d = np.where(d == 0, np.copysign(F(0), raw), d).astype(F)                  # keep the -0 components
    ok = np.isfinite(d).all(1) & np.isfinite(org).all(1)    # where the float grid swallows a gap, an aimed direction can vanish
    return np.ascontiguousarray(org[ok]), np.ascontiguousarray(d[ok])


def windows(s):
    return ((0.001, FLT_MAX), (T_BOUND, FLT_MAX), (float(F(0.5 * s)), float(F(40.0 * s))))


class Ladder:
    """scene (base, level) -> host scene, SoA, rays and the oracle's hits per window, built once per module"""

    def __init__(self, r1, oracle):
        self.r1, self.oracle, self.bases, self.cache = r1, oracle, {}, {}

    def base(self, name):
        if name not in self.bases:
            cam, sph = base_spheres(self.r1, name)
            s = RawScene(cam, sph, commit=False)
            self.bases[name] = (cam, sph, s.camera())
            s.close()
        return self.bases[name]

    def spheres(self, name, level):
        cam, sph, cam22 = self.base(name)
        s, t = transform(level)
        return moved(sph, s, t), move_cam22(cam22, s, t)

    def __getitem__(self, key):
        if key not in self.cache:
            name, level = key
            sph, cam22 = self.spheres(name, level)
            scene = RawScene(self.base(name)[0], sph, commit=False)
            scene.set_camera_raw(cam22)
            soa = scene.soa()
            s, _ = transform(level)
            org, d = ladder_rays(soa, s)
            so = self.oracle.scene_create_from_soa(soa)
            try:
                hits = {w: self.oracle.hit(so, org, d, *w) for w in windows(s)}
            finally:
                self.oracle.scene_destroy(so)
            self.cache[key] = dict(scene=scene, soa=soa, org=org, d=d, hits=hits, s=s, cam22=cam22, spheres=sph)
        return self.cache[key]

    def close(self):
        for v in self.cache.values():
            v["scene"].close()


@pytest.fixture(scope="module")
def ladder(r1, oracle):
    lad = Ladder(r1, oracle)
    yield lad
    lad.close()


# ---- the FFMA2 filter, restated ---------------------------------------------------------------------------------------------

def fma(a, b, c):
    """fmaf for float32 arrays: the product is exact in float64, the sum rounds once there and once more to float32 (the double
    rounding can differ from fmaf in the last bit; decisions that close to zero count as undecided)"""
    with np.errstate(over="ignore", invalid="ignore"):
        return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F)


def scan_records(soa):
    """the scan lanes -cx, -cy, -cz, kk of every sphere (r1_encode.h enc::scan_lanes)"""
    c = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1).astype(np.float64)
    real = soa["inv_radius"] != 0
    with np.errstate(over="ignore", invalid="ignore"):
        c2 = (c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]) + c[:, 2] * c[:, 2]
        kk = (c2 - soa["radius_sq"].astype(np.float64)) - c2 / 131072.0
        kf = kk.astype(F)
    kf = np.where(kf.astype(np.float64) > kk, np.nextafter(kf, F(-np.inf)), kf)
    kf = np.nextafter(kf, F(-np.inf))
    far = real & (c2 >= FAR_C2)
    keep = real & ~far
    n = np.where(keep[:, None], -c.astype(F), F(0)).astype(F)
    kf = np.where(far, FAR_KK, np.where(real, kf, F(np.inf))).astype(F)
    return n, kf


def dot3(a, b):
    """r1_device.cuh dot3: fma(a.z, b.z, fma(a.y, b.y, a.x * b.x))"""
    return fma(a[:, 2], b[:, 2], fma(a[:, 1], b[:, 1], (a[:, 0] * b[:, 0]).astype(F)))


def ray_consts(org, d):
    """r1_device.cuh ray_const: (o.d, |o|^2 (1 - 2^-17), 2o, d), or the constants that flag every sphere for |o|^2 >= 2^120"""
    with np.errstate(over="ignore", invalid="ignore"):
        oo = dot3(org, org)
        inr = oo < F(2.0 ** 120)
        od = np.where(inr, dot3(org, d), F(0)).astype(F)
        oo = np.where(inr, (oo * F(1.0 - 1.0 / 131072.0)).astype(F), F(-2.0 ** 126)).astype(F)
        o2 = np.where(inr[:, None], (org + org).astype(F), F(0)).astype(F)
        dd = np.where(inr[:, None], d, F(0)).astype(F)
    return od, oo, o2, dd


def packed_filter(soa, org, d):
    """e [rays, spheres] of filter_packed, and whether each decision is within a few ulps of zero"""
    n, kk = scan_records(soa)
    od, oo, o2, dd = ray_consts(org, d)
    R = lambda v: v[:, None]  # noqa: E731
    with np.errstate(over="ignore", invalid="ignore"):
        m = fma(n[None, :, 0], R(dd[:, 0]), fma(n[None, :, 1], R(dd[:, 1]), fma(n[None, :, 2], R(dd[:, 2]), R(od))))
        P = fma(n[None, :, 0], R(o2[:, 0]), fma(n[None, :, 1], R(o2[:, 1]), fma(n[None, :, 2], R(o2[:, 2]), kk[None, :])))
        Q = (P + R(oo)).astype(F)
        e = fma(m, m, -Q)
        scale = np.maximum(np.abs((m.astype(np.float64) ** 2)), np.abs(Q.astype(np.float64)))
        close = np.isfinite(scale) & (np.abs(e.astype(np.float64)) <= 4 * 2.0 ** -23 * scale)
    return e, close


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_packed_filter_flags_every_hit(ladder, name, level):
    L = ladder[name, level]
    e, close = packed_filter(L["soa"], L["org"], L["d"])
    for w, (idx, t, _, _) in L["hits"].items():
        k = np.nonzero(idx >= 0)[0]
        ek, ck = e[k, idx[k]], close[k, idx[k]]
        bad = (np.signbit(ek) | np.isnan(ek)) & ~ck               # a NaN's sign bit is not a decision this filter may rest on
        assert not bad.any(), "%s %s %s: the FFMA2 filter skips %d hits, e.g. ray %d sphere %d (e = %r)" % (
            name, level, w, bad.sum(), k[bad][0], idx[k[bad][0]], ek[bad][0])
    placeholder = L["soa"]["inv_radius"] == 0
    assert np.signbit(e[:, placeholder]).all(), "placeholders are never candidates"


# ---- the tensor filter, restated ----------------------------------------------------------------------------------------------

def tensor_rows(org, d):
    """tc::ray_row of live rays: test_tensor_cpu.ray_rows within the range, 0 x 9, -1, 2^121 outside it"""
    with np.errstate(over="ignore", invalid="ignore"):
        a = ray_rows(org, d)
        inr = dot3(org, org) < F(2.0 ** 120)
    flag = np.zeros(32, F)
    flag[[9, 20, 31]] = F(-1), F(0), F(-1)
    flag[10] = F(2.0 ** 121)
    return np.where(inr[:, None], a, flag[None, :]).astype(F)


def tensor_filter(scene, org, d):
    a = tensor_rows(org, d).astype(np.float64)
    op = scene.tensor_operand().astype(np.float64)
    b = np.concatenate([op[:, 0:11], op[:, 11:22], op[:, 22:32]], 1)
    with np.errstate(over="ignore", invalid="ignore"):
        return a @ b.T


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_tensor_filter_flags_every_hit(ladder, name, level):
    """the split operands as the library builds them (the sphere side) and as tc::ray_row builds them, products and sum in float64"""
    L = ladder[name, level]
    e = tensor_filter(L["scene"], L["org"], L["d"])
    n = len(L["soa"]["cx"])
    for w, (idx, t, _, _) in L["hits"].items():
        k = np.nonzero(idx >= 0)[0]
        ek = e[k, idx[k]]
        bad = ~(ek >= 0)
        assert not bad.any(), "%s %s %s: the tensor filter skips %d hits, e.g. ray %d sphere %d (e = %r)" % (
            name, level, w, bad.sum(), k[bad][0], idx[k[bad][0]], ek[bad][0])
    dead = np.ones(e.shape[1], bool)
    dead[:n] = L["soa"]["inv_radius"] == 0
    assert (e[:, dead] < 0).all(), "padding rows and placeholders are never candidates"


# ---- the BVH box test ------------------------------------------------------------------------------------------------------------

class Tree:
    """a scene view whose bvh() is a given tree (check_conservative reads soa() and bvh())"""

    def __init__(self, soa, tree):
        self._soa, self._tree = soa, tree

    def soa(self):
        return self._soa

    def bvh(self):
        return self._tree


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_box_test_passes_every_winner(oracle, ladder, name, level):
    """the host tree, the device builder's restated tree and a level-0 tree refitted to this level"""
    L = ladder[name, level]
    soa, org, d, ws = L["soa"], L["org"], L["d"], tuple(L["hits"])
    checked = check_conservative(L["scene"], oracle, org, d, ws, "%s %s host tree" % (name, level))
    assert checked > 0
    check_conservative(Tree(soa, lbvh.build(soa)), oracle, org, d, ws, "%s %s device builder" % (name, level))
    base = ladder[name, "level0"]
    tree = refit.refit(base["scene"].bvh(), refit.exact_of(soa))
    check_conservative(Tree(soa, tree), oracle, org, d, ws, "%s %s refit of level 0" % (name, level))


# ---- the fixture itself -----------------------------------------------------------------------------------------------------------

def test_ladder_covers_the_range():
    assert transform("rigid63.5")[1][0] == 1.5 * 2.0 ** 63
    s, t = transform("scaled64")
    assert s == 2.0 ** 52 and (t == T_DIR * 2.0 ** 64).all()
    s, t = transform("scale-12")
    assert s == 2.0 ** -12 and not t.any()
    assert all((T_DIR * 2.0 ** k).astype(F).astype(np.float64).tolist() == (T_DIR * 2.0 ** k).tolist() for k in RIGID if k != 63.5)


@pytest.mark.parametrize("level", LEVELS)
@pytest.mark.parametrize("name", BASES)
def test_every_level_has_hits(ladder, name, level):
    L = ladder[name, level]
    s = L["s"]
    for w, (idx, *_) in L["hits"].items():
        if w[0] == T_BOUND and s < 2.0 ** -6:
            continue                                             # 2^-24 is below 0.001 s: the other windows carry these levels
        assert (idx >= 0).sum() >= 300, (name, level, w, int((idx >= 0).sum()))
    c = np.stack([L["soa"]["cx"], L["soa"]["cy"], L["soa"]["cz"]], 1).astype(np.float64)
    if level in ("rigid64", "rigid65", "rigid70", "rigid100", "rigid126", "scaled64", "scaled65", "scaled70", "scale62"):
        idx = L["hits"][(0.001, FLT_MAX)][0]
        far = np.linalg.norm(c, axis=1) > 2.0 ** 64
        assert far[idx[idx >= 0]].sum() >= 100, "hits on spheres whose |c| exceeds 2^64"


@pytest.mark.parametrize("level,like", (("scaled30", "scaled20"), ("scaled50", "scaled20"), ("scaled60", "scaled20"), ("scaled63", "scaled20"),
                                        ("scale30", "scale12")))
def test_scaled_levels_render_alike(r1, oracle, ladder, level, like):
    """the oracle's renders of two levels of one layout: the same picture up to rounding.  (Level 0 itself differs: there t_min =
    0.001 is not negligible against the scene, so it keeps paths other levels lose to self-hits and the reverse.)"""
    name = "n120"
    imgs = []
    for lv in (like, level):
        sph, cam22 = ladder.spheres(name, lv)
        s = RawScene(spec(name)[0], sph, commit=False)
        so = oracle.scene_create_from_soa(s.soa())
        oracle.scene_set_camera(so, cam22)
        imgs.append(oracle.render_keyed(so, 64, 36, 16, 8, 0, 0, 1, 1)[1])
        oracle.scene_destroy(so)
        s.close()
    err = rmse(imgs[0], imgs[1])
    assert err < 6.0, (level, like, err)
    assert imgs[0].std() > 10
