"""Every scan against the oracle where scans branch: ragged sphere counts, candidate floods, ties, root boundaries.

The built-in scenes reach only some shapes of the scans' loops.  The per-lane scans (scalar, packed, deferred, dual, wavefront)
finish a scene with (n8 mod 32) / 4 = 0, 2, 4 or 6 groups one by one; the cooperative scan's last step holds (n_pad / 16) mod 8
supergroups (8 when 0); the tensor filter reads its last 128-sphere chunk in (n32 mod 128) / 32 pieces (4 when 0).  The scenes
below reach each of them:

    A  sweep: every multiple of 8 from 8 to 136 (all tails, all coop last steps, n32 = 32 .. 160), the counts 1, 5, 13, 31
       and 33 built unpadded through the raw ABI, and 200 / 488 / 760 / 1000 spheres.  A seeded cluster of mixed radii with a
       large ground sphere LAST, i.e. in the tail.
    B  floods: spheres of radius ~5 with centres inside a unit cube, so every ray's line flags nearly every sphere -- the
       cooperative queue (92 entries, drained above 60) and the deferred queue (188) fill and drain many times per scan.
    C  ties: exact duplicates (same centre and radius, another material) at index pairs that straddle a group of 4, the lanes
       of a cooperative supergroup, two supergroups, a 32-sphere chunk, a 128-sphere tensor chunk, and the first and last
       sphere; near-ties one ulp apart.  Hitable::hit keeps the lower index on a tie.
    D  root boundaries: t_max = t and one ulp above, t_min = t and one ulp below, for ordinary, on-surface, inside and tangent
       (discr = +0) rays, with t_min = 0.001 and with the smallest t_min r1_trace_rays takes (2^-24).
    E  renders of the scans with no ray kernel (dual, wavefront) and of every other variant and switch, byte for byte
       against PACKED on the A, B and C scenes.

Ray-level cases compare index, t, p and normal of every ray bit for bit with the oracle's Hitable::hit.
tests/test_scan_edges_cpu.py checks that these fixtures contain what this docstring claims."""
import numpy as np
import pytest

import rays1bench_b200 as r1mod
from test_gpu_parity import bits

pytestmark = pytest.mark.gpu

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)
T_BOUND = 2.0 ** -24                                 # the smallest t_min r1_trace_rays accepts
RAY_VARIANTS = ("scalar", "packed", "coop", "deferred", "tensor", "mega")
UNPADDED = (1, 5, 13, 31, 33)
SWEEP = tuple(range(8, 137, 8)) + UNPADDED + (200, 488, 760, 1000)
FLOODS = (96, 488, 760, 4096)
TIE_COUNT = 200
# exact duplicates (lower, higher): inside a group of 4; across groups 0 / 1 (coop lanes j = 0 / 1); lanes j = 1 / 3 of one
# supergroup; across supergroups 0 / 1; across the 32-sphere chunks; across tensor chunks 0 / 1; across the start of the
# per-lane tail (192); the first and the last sphere
TIE_PAIRS = ((1, 2), (3, 4), (6, 14), (15, 16), (31, 32), (127, 128), (191, 196), (0, 199))
# near-ties (lower, higher, the one whose root is one ulp nearer on the axis ray)
NEAR_PAIRS = ((40, 41, 40), (60, 100, 60), (70, 71, 71), (140, 150, 150))
FLOOD_RENDER_TENSOR = (488, 760)                     # tc3 flood renders kept to these (long candidate loops per chunk)


def lane_tail_groups(n):
    """groups the per-lane scans test one by one after their 32-sphere chunks"""
    return ((n + 7) // 8 * 8 % 32) // 4


def coop_last_steps(n):
    """supergroups in the cooperative scan's last step"""
    return (n + 15) // 16 % 8 or 8


def n32_of(n):
    return (n + 31) // 32 * 32


# ---- scene specs: (camera args, spheres) as r1.write_scene_file takes them ----------------------------------------------------

def _f(*v):
    return tuple(float(F32(x)) for x in v)


def _material(rng):
    k = rng.choice([r1mod.MAT_LAMBERT, r1mod.MAT_METAL, r1mod.MAT_DIELECTRIC], p=[0.6, 0.25, 0.15])
    r, g, b = rng.uniform(0.1, 0.9, 3)
    param = {r1mod.MAT_LAMBERT: 0.0, r1mod.MAT_METAL: rng.uniform(0.0, 0.5), r1mod.MAT_DIELECTRIC: 1.5}[int(k)]
    if k == r1mod.MAT_DIELECTRIC:
        r = g = b = 0.0
    return (int(k),) + _f(r, g, b, param)


def cluster_spec(n):
    """n - 1 spheres of radius 0.15 .. 1.2 in a box that grows with n, then the ground (radius 1000) as sphere n - 1"""
    rng = np.random.default_rng(4242 + n)
    side = 2.0 * max(1.0, (n - 1) ** (1.0 / 3.0))
    sph = []
    for _ in range(n - 1):
        x, z = rng.uniform(-side, side, 2)
        y = rng.uniform(0.2, side)
        r = np.exp(rng.uniform(np.log(0.15), np.log(1.2)))
        m = _material(rng)
        sph.append(_f(x, y, z, r) + m)
    sph.append(_f(0, -1000, 0, 1000) + (r1mod.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0))
    cam = _f(0, 1.2 * side + 1, 3.2 * side + 3, 0, 0.4 * side, 0, 50, 0.02, 10)
    return cam, sph


def flood_spec(n):
    """radius 5 +- 0.05, centres in the unit cube: every ray's line through the cluster flags nearly every sphere"""
    rng = np.random.default_rng(777 + n)
    sph = []
    for _ in range(n):
        c = rng.uniform(-0.5, 0.5, 3)
        k = int(rng.choice([r1mod.MAT_LAMBERT, r1mod.MAT_METAL]))
        sph.append(_f(*c, 5.0 + rng.uniform(-0.05, 0.05)) + (k,) + _f(*rng.uniform(0.1, 0.9, 3), rng.uniform(0, 0.3)))
    return _f(0, 8, 30, 0, 0, 0, 40, 0.02, 30), sph


def pair_centre(k):
    """centre of tie pair k: integers, radius 1, in a row along x (tangent and on-surface rays are exact there)"""
    return (4.0 * (k - 6), 2.0, 0.0)


def near_centres(k):
    """near-tie pair k: the same sphere at z = 6 and one ulp above; on the axis ray from z = 12 their roots are 5 and 5 - ulp"""
    x = 4.0 * (k - 6) + 2.0
    return (x, 2.0, 6.0), (x, 2.0, float(np.nextafter(F32(6), F32(np.inf))))


def tie_spec():
    """TIE_COUNT spheres: the TIE_PAIRS as exact duplicates (lower: red Lambertian, higher: green metal), the NEAR_PAIRS, and
    small filler spheres far below the row"""
    rng = np.random.default_rng(99)
    sph = [None] * TIE_COUNT
    red, green = (r1mod.MAT_LAMBERT,) + _f(0.9, 0.1, 0.1, 0), (r1mod.MAT_METAL,) + _f(0.1, 0.9, 0.1, 0.0)
    for k, (lo, hi) in enumerate(TIE_PAIRS):
        c = pair_centre(k)
        sph[lo] = _f(*c, 1.0) + red
        sph[hi] = _f(*c, 1.0) + green
    for k, (lo, hi, nearer) in enumerate(NEAR_PAIRS):
        up, down = near_centres(k)
        sph[nearer] = _f(*up, 1.0) + red
        sph[lo + hi - nearer] = _f(*down, 1.0) + green
    for i in range(TIE_COUNT):
        if sph[i] is None:
            x, z = rng.integers(-40, 41, 2)
            sph[i] = _f(x, -30, z, 0.25) + _material(rng)
    return _f(0, 14, 24, 0, 1, 0, 55, 0.0, 24), sph


def spec(name):
    if name == "ties":
        return tie_spec()
    if name.startswith("flood"):
        return flood_spec(int(name[5:]))
    return cluster_spec(int(name[1:]))


def count_of(name):
    return TIE_COUNT if name == "ties" else int(name[5:] if name.startswith("flood") else name[1:])


# ---- scenes --------------------------------------------------------------------------------------------------------------

class RawScene(r1mod.Scene):
    """A scene built through the raw ABI (r1_scene_create / add_sphere / set_camera / commit): no padding to 8, so the device
    sees exactly len(spheres) spheres.  `handle` is the r1_scene itself."""

    def __init__(self, cam, spheres, commit=True):
        lib = r1mod.lib
        super().__init__(lib.r1_scene_create(len(spheres)), "raw%d" % len(spheres))
        for c in spheres:
            r1mod._check(lib.r1_scene_add_sphere(self._ptr, *c[:4], int(c[4]), *c[5:]), "r1_scene_add_sphere")
        v = lambda *x: np.array(x, np.float32)  # noqa: E731
        r1mod._check(lib.r1_scene_set_camera(self._ptr, v(*cam[0:3]), v(*cam[3:6]), v(0, 1, 0), cam[6], 16.0 / 9.0, cam[7], cam[8]),
                     "r1_scene_set_camera")
        if commit:
            r1mod._check(lib.r1_scene_commit(self._ptr, 0), "r1_scene_commit")

    @property
    def handle(self):
        return self._ptr

    def close(self):
        if self._ptr:
            r1mod.lib.r1_scene_destroy(self._ptr)
            self._ptr = None


def make_scene(r1, name, directory, commit=True):
    """names: "n<count>" (A; unpadded through the raw ABI for the UNPADDED counts), "flood<count>" (B), "ties" (C)"""
    cam, sph = spec(name)
    if name.startswith("n") and count_of(name) in UNPADDED:
        return RawScene(cam, sph, commit)
    path = str(directory / ("%s.r1scene" % name))
    r1.write_scene_file(path, cam, sph)
    return r1.create_scene_from_file(path, commit=commit)


class SceneCache:
    def __init__(self, r1, directory, commit=True):
        self.r1, self.dir, self.commit, self.scenes = r1, directory, commit, {}

    def __getitem__(self, name):
        if name not in self.scenes:
            self.scenes[name] = make_scene(self.r1, name, self.dir, self.commit)
        return self.scenes[name]

    def close(self):
        for s in self.scenes.values():
            s.close()


@pytest.fixture(scope="module")
def edge_scenes(r1, tmp_path_factory):
    r1.configure(width=1280, height=720, spp=250, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    cache = SceneCache(r1, tmp_path_factory.mktemp("edges"))
    yield cache
    cache.close()


# ---- rays ----------------------------------------------------------------------------------------------------------------

def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def aimed_rays(soa, idx, rng, gaps):
    """rays at the centres (a third) and at +-2 % silhouettes of spheres `idx`, from `gaps` units outside them"""
    n = len(idx)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1).astype(np.float64)
    rad = 1.0 / soa["inv_radius"][idx].astype(np.float64)
    u = _unit(rng.normal(size=(n, 3)))
    u[:, 1] = np.abs(u[:, 1])
    o = ctr + u * (rad + gaps)[:, None]
    side = _unit(np.cross(u, rng.normal(size=(n, 3))))
    k = rng.uniform(0.98, 1.02, n) * (rng.uniform(size=n) > 1.0 / 3.0)
    d = _unit(ctr + side * (rad * k)[:, None] - o)
    return o, d


def sweep_rays(soa, seed=5):
    """A: 1 200 random rays around the cluster, 900 aimed at random spheres from 5 .. 20 000 units, 300 aimed at the spheres
    of the scan's last 32 (the tail groups; the ground among them) from 0.5 .. 3 units -- 2 400 rays, not a multiple of 128"""
    rng = np.random.default_rng(seed)
    n = len(soa["cx"])
    real = np.where(soa["inv_radius"] > 0)[0]
    box = max(2.0, 2.0 * (n - 1) ** (1.0 / 3.0))
    o1 = rng.uniform(-1.3 * box, 1.3 * box, (1200, 3)) + [0, box * 0.6, 0]
    d1 = _unit(rng.normal(size=(1200, 3)))
    o2, d2 = aimed_rays(soa, rng.choice(real, 900), rng, rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], 900))
    tail = real[real >= ((n + 7) // 8 * 8 - 1) // 32 * 32]
    o3, d3 = aimed_rays(soa, rng.choice(tail, 300), rng, rng.uniform(0.5, 3.0, 300))
    return np.concatenate([o1, o2, o3]).astype(F32), np.concatenate([d1, d2, d3]).astype(F32)


def flood_rays(n=1000, seed=11):
    """B: 600 rays from 12 .. 60 units outside the cluster through it, 400 from inside every sphere (only far roots)"""
    rng = np.random.default_rng(seed)
    u = _unit(rng.normal(size=(600, 3)))
    o1 = u * rng.uniform(12, 60, (600, 1))
    d1 = _unit(rng.uniform(-2, 2, (600, 3)) - o1)
    o2 = rng.uniform(-1.5, 1.5, (n - 600, 3))
    d2 = _unit(rng.normal(size=(n - 600, 3)))
    return np.concatenate([o1, o2]).astype(F32), np.concatenate([d1, d2]).astype(F32)


def tangent_rays():
    """rays tangent to the exact-duplicate pairs (integer centres, radius 1): o = c + (1, 0, -L), d = +z and the like;
    co = (-1, 0, L), nb = L, q = L^2 + 1, discr = fma(L, L, -q) + 1 = +0 exactly, root t = L for both duplicates"""
    org, d = [], []
    for k in range(len(TIE_PAIRS)):
        c = np.array(pair_centre(k))
        for L in (3.0, 5.0, 7.0):
            for off, dd in (((1, 0, -L), (0, 0, 1)), ((-1, 0, -L), (0, 0, 1)), ((0, 1, -L), (0, 0, 1)), ((0, 1, L), (0, 0, -1))):
                org.append(c + off)
                d.append(dd)
    return np.array(org, F32), np.array(d, F32)


def near_tie_rays():
    """the axis ray of each near-tie pair: from z = 12 along -z, roots 5 and 5 - ulp"""
    org = [near_centres(k)[0][:2] + (12.0,) for k in range(len(NEAR_PAIRS))]
    return np.array(org, F32), np.tile(np.array([0, 0, -1], F32), (len(org), 1))


def tie_rays(soa, seed=3):
    """C: per exact and near pair 160 rays aimed at it from 5 .. 200 units above the row, the tangent rays, the near-tie axis
    rays, each axis ray again from 1 .. 4 units further"""
    rng = np.random.default_rng(seed)
    idx = np.repeat([lo for lo, _ in TIE_PAIRS] + [lo for lo, _, _ in NEAR_PAIRS], 160)
    o1, d1 = aimed_rays(soa, idx, rng, rng.uniform(5.0, 200.0, len(idx)))
    o2, d2 = tangent_rays()
    o3, d3 = near_tie_rays()
    o4 = np.repeat(o3, 4, 0) + np.tile(np.array([[0, 0, 1], [0, 0, 2], [0, 0, 3], [0, 0, 4]], F32), (len(o3), 1))
    d4 = np.repeat(d3, 4, 0)
    return (np.concatenate([o1, o2, o3, o4]).astype(F32), np.concatenate([d1, d2, d3, d4]).astype(F32))


def scene_rays(name, soa):
    if name == "ties":
        return tie_rays(soa)
    if name.startswith("flood"):
        return flood_rays()
    return sweep_rays(soa)


# ---- D: root boundaries ---------------------------------------------------------------------------------------------------

BOUNDARY_SCENES = ("ties", "n120", "flood96")


def boundary_rays(name, soa, oracle_scene, oracle, t_min, n=16, seed=8):
    """rays of scene `name` that hit with this t_min: aimed rays, rays from hit points of the first pass (on a surface, up to
    rounding) in fresh directions, rays from inside spheres; in the tie scene also tangent rays and rays from points exactly
    on the pairs' surfaces.  Returns (org, dir, t) of at most n hits per kind."""
    rng = np.random.default_rng(seed)
    o, d = scene_rays(name, soa)
    pick = rng.choice(len(o), 400, replace=False)
    o, d = o[pick], d[pick]
    first = oracle.hit(oracle_scene, o, d, t_min)
    kinds = [(o, d)]
    hit = first[0] >= 0
    p = first[2][hit][:n]
    kinds.append((p, _unit(rng.normal(size=p.shape)).astype(F32)))
    real = np.where(soa["inv_radius"] > 0)[0]
    i = rng.choice(real, n)
    ctr = np.stack([soa["cx"][i], soa["cy"][i], soa["cz"][i]], 1)
    kinds.append(((ctr + rng.uniform(-0.1, 0.1, ctr.shape)).astype(F32), _unit(rng.normal(size=ctr.shape)).astype(F32)))
    if name == "ties":
        kinds.append(tangent_rays())
        c = np.array([pair_centre(k) for k in range(len(TIE_PAIRS))], F32)
        on = np.concatenate([c + [1, 0, 0], c + [0, 0, 1], c + [0, -1, 0]]).astype(F32)
        kinds.append((on, _unit(rng.normal(size=on.shape)).astype(F32)))
    out_o, out_d = [], []
    for ko, kd in kinds:
        ko, kd = np.ascontiguousarray(ko, F32), np.ascontiguousarray(kd, F32)
        h = oracle.hit(oracle_scene, ko, kd, t_min)[0] >= 0
        out_o.append(ko[h][:n])
        out_d.append(kd[h][:n])
    org, dd = np.concatenate(out_o), np.concatenate(out_d)
    return org, dd, oracle.hit(oracle_scene, org, dd, t_min)[1]


def boundary_queries(t_min, t):
    """(t_min, t_max) per ray: the hit at t must vanish with t_max = t and stay with one ulp more; with t_min = t the near root
    t is out (the far root or another sphere answers), with one ulp less it stays"""
    up, down = np.nextafter(F32(t), F32(np.inf)), np.nextafter(F32(t), F32(-np.inf))
    return ((t_min, float(t)), (t_min, float(up)), (float(t), FLT_MAX), (float(down), FLT_MAX))


# ---- checks ---------------------------------------------------------------------------------------------------------------

def variants_for(n):
    return [v for v in RAY_VARIANTS if v != "tensor" or n32_of(n) <= 768]


def check_against_oracle(r1, s, want, org, d, t_min, t_max, variants, what):
    for v in variants:
        got = s.trace_rays(org, d, t_min, t_max, variant=r1.VARIANTS[v])
        bad = np.where(got[0] != want[0])[0]
        assert len(bad) == 0, "%s, %s: %d rays differ, e.g. ray %d: index %d, oracle %d" % (what, v, len(bad), bad[0], got[0][bad[0]],
                                                                                           want[0][bad[0]])
        for name, a, b in zip(("t", "p", "normal"), got[1:], want[1:]):
            assert np.array_equal(bits(a), bits(b)), "%s, %s: %s differs" % (what, v, name)


def check_scene(r1, oracle, s, name, windows):
    soa = s.soa()
    org, d = scene_rays(name, soa)
    assert len(org) % 128 != 0
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in windows:
            want = oracle.hit(so, org, d, t_min, t_max)
            check_against_oracle(r1, s, want, org, d, t_min, t_max, variants_for(len(soa["cx"])), "%s [%g, %g]" % (name, t_min, t_max))
    finally:
        oracle.scene_destroy(so)


@pytest.mark.parametrize("n", SWEEP)
def test_sphere_count_sweep_matches_oracle(r1, oracle, edge_scenes, n):
    """A: every variant's hits bit for bit, whole range and a window, at every tail shape"""
    s = edge_scenes["n%d" % n]
    assert s.count() == (n if n in UNPADDED else (n + 7) // 8 * 8)
    check_scene(r1, oracle, s, "n%d" % n, ((0.001, FLT_MAX), (0.5, 40.0)))
    if n32_of(n) > 768:
        with pytest.raises(r1.Rays1Error, match=r"\(-4\).*768"):
            s.trace_rays([[0, 3, 20]], [[0, 0, -1]], variant=r1.VARIANT_MEGAKERNEL_TENSOR)


@pytest.mark.parametrize("n", FLOODS)
def test_candidate_floods_match_oracle(r1, oracle, edge_scenes, n):
    """B: a warp's 32 rays each flag (nearly) every sphere; from outside and from inside all spheres (far roots)"""
    check_scene(r1, oracle, edge_scenes["flood%d" % n], "flood%d" % n, ((0.001, FLT_MAX), (6.0, 40.0)))


def test_ties_go_to_the_lower_index(r1, oracle, edge_scenes):
    """C: exact duplicates at every straddle, tangent rays on them, near-ties one ulp apart -- whole range and from t_min = 2^-24"""
    check_scene(r1, oracle, edge_scenes["ties"], "ties", ((0.001, FLT_MAX), (T_BOUND, FLT_MAX), (4.0, 30.0)))


@pytest.mark.parametrize("name", BOUNDARY_SCENES)
@pytest.mark.parametrize("t_min", (0.001, T_BOUND), ids=("tmin_0.001", "tmin_2^-24"))
def test_root_boundaries_match_oracle(r1, oracle, edge_scenes, name, t_min):
    """D: per hit ray, t_max = t / t + ulp and t_min = t / t - ulp, every variant against the oracle"""
    s = edge_scenes[name]
    soa = s.soa()
    so = oracle.scene_create_from_soa(soa)
    try:
        org, d, t = boundary_rays(name, soa, so, oracle, t_min)
        assert len(org) >= 40
        variants = variants_for(len(soa["cx"]))
        for k in range(len(org)):
            for lo, hi in boundary_queries(t_min, t[k]):
                want = oracle.hit(so, org[k:k + 1], d[k:k + 1], lo, hi)
                check_against_oracle(r1, s, want, org[k:k + 1], d[k:k + 1], lo, hi, variants, "%s ray %d [%r, %r]" % (name, k, lo, hi))
    finally:
        oracle.scene_destroy(so)


def test_trace_rays_accepts_t_min_at_the_bound(r1, oracle, edge_scenes):
    """t_min = 2^-24 is accepted and answers like Hitable::hit on the two rays where a smaller t_min would not: a ray starting
    on its tangent point (nb = 0, discr = +0: a miss) and a ray from the centre of sphere 0 with sphere 2 ahead (the far root of
    sphere 0, t = 1); one ulp below the bound is refused"""
    sph = [_f(0, 0, 0, 1) + (r1mod.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0), _f(30, 0, 0, 1) + (r1mod.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0),
           _f(0, 0, 5, 1) + (r1mod.MAT_LAMBERT,) + _f(0.5, 0.5, 0.5, 0)]
    s = RawScene(_f(0, 0, 20, 0, 0, 0, 40, 0, 20), sph)
    try:
        org = np.array([[1, 0, 0], [0, 0, 0], [1, 0, -3]], F32)
        d = np.array([[0, 0, -1], [0, 0, 1], [0, 0, 1]], F32)
        so = oracle.scene_create_from_soa(s.soa())
        want = oracle.hit(so, org, d, T_BOUND)
        oracle.scene_destroy(so)
        assert list(want[0]) == [-1, 0, 0] and want[1][1] == 1 and want[1][2] == 3
        check_against_oracle(r1, s, want, org, d, T_BOUND, FLT_MAX, RAY_VARIANTS, "t_min = 2^-24")
        with pytest.raises(r1.Rays1Error, match=r"\(-1\).*2\^-24"):
            s.trace_rays(org, d, float(np.nextafter(F32(T_BOUND), F32(0))))
    finally:
        s.close()


# ---- E: renders --------------------------------------------------------------------------------------------------------------

RENDER_SCENES = tuple("n%d" % n for n in SWEEP) + tuple("flood%d" % n for n in FLOODS) + ("ties",)
RENDER_CASES = ((48, 27, 4, 0, 1), (7, 3, 5, 0, 1), (48, 27, 4, 1, 3))


def render_runs(r1, name):
    """(variant, threads, environment) of every render compared with PACKED"""
    V = r1
    runs = [(V.VARIANT_MEGAKERNEL_SCALAR, 0, {}), (V.VARIANT_MEGAKERNEL_COOP, 0, {}), (V.VARIANT_MEGAKERNEL_DEFERRED, 0, {}),
            (V.VARIANT_MEGAKERNEL_DUAL, 0, {}), (V.VARIANT_MEGAKERNEL_DUAL, 512, {}), (V.VARIANT_WAVEFRONT, 0, {})]
    n = count_of(name)
    if n32_of(n) <= 768 and (not name.startswith("flood") or n in FLOOD_RENDER_TENSOR):
        runs.append((V.VARIANT_MEGAKERNEL_TENSOR, 0, {}))
    for v in (V.VARIANT_MEGAKERNEL_PACKED, V.VARIANT_MEGAKERNEL_COOP, V.VARIANT_MEGAKERNEL_DEFERRED, V.VARIANT_MEGAKERNEL_DUAL):
        runs.append((v, 0, {"R1_FORCE_UNSTAGED": "1"}))
    return runs


@pytest.mark.parametrize("name", RENDER_SCENES)
def test_every_variant_renders_like_packed(r1, edge_scenes, monkeypatch, name):
    """E: scalar, coop, deferred, DUAL (768 and 512 threads), WAVEFRONT, TENSOR and R1_FORCE_UNSTAGED=1 renders
    byte-identical to PACKED with the same ray count, on a 48x27 frame, a 7x3 image and as rank 1 of 3"""
    s = edge_scenes[name]
    for w, h, spp, rank, world in RENDER_CASES:
        base, r0 = s.render(w, h, spp, rank=rank, world=world, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        if (w, h) == (48, 27) and world == 1:
            assert base.any()
        for v, threads, env in render_runs(r1, name):
            for k, val in env.items():
                monkeypatch.setenv(k, val)
            rgb, res = s.render(w, h, spp, rank=rank, world=world, variant=v, threads=threads)
            for k in env:
                monkeypatch.delenv(k)
            assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays, (name, (w, h, spp, rank, world), v, threads, env)


def test_deferred_renders_a_4096_sphere_scene(r1, edge_scenes):
    """With the sample pool, the deferred scan's per-warp queues and 4096 staged spheres need more than 227 KB of shared memory
    at 1024 threads: the default runs fewer threads and renders the same bytes as PACKED; 1024 threads asked for are refused
    with R1_ERR_LIMIT naming shared memory"""
    s = edge_scenes["flood4096"]
    base, r0 = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    rgb, res = s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_DEFERRED)
    assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
    with pytest.raises(r1.Rays1Error, match=r"\(-4\).*shared memory"):
        s.render(48, 27, 4, variant=r1.VARIANT_MEGAKERNEL_DEFERRED, threads=1024)
