"""CPU checks that the fixtures of tests/test_scan_edges_gpu.py contain what those tests rely on -- so that they cannot pass by
testing nothing -- and the t_min domain of r1_trace_rays, which is checked before any device is touched."""
import numpy as np
import pytest

from test_scan_edges_gpu import (BOUNDARY_SCENES, FLOODS, NEAR_PAIRS, SWEEP, T_BOUND, TIE_PAIRS, UNPADDED, boundary_queries,
                                 boundary_rays, coop_last_steps, flood_rays, lane_tail_groups, make_scene, n32_of, near_tie_rays,
                                 pair_centre, scene_rays, tangent_rays)

F32 = np.float32
FLT_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def host_scenes(r1, tmp_path_factory):
    """the GPU file's scenes, host side only"""
    d = tmp_path_factory.mktemp("edges_cpu")
    made = {}

    def get(name):
        if name not in made:
            made[name] = make_scene(r1, name, d, commit=False)
        return made[name]
    yield get
    for s in made.values():
        s.close()


def test_sweep_covers_every_scan_shape():
    assert {lane_tail_groups(n) for n in SWEEP} == {0, 2, 4, 6}
    for tail in (0, 2, 4, 6):   # every tail shape also at an unpadded or a multiple-of-8 count
        assert any(lane_tail_groups(n) == tail and n % 8 == 0 for n in SWEEP)
    assert {coop_last_steps(n) for n in SWEEP} == set(range(1, 9))
    assert {32, 64, 96, 128, 160} <= {n32_of(n) for n in SWEEP}
    assert any(n32_of(n) > 768 for n in SWEEP), "one count above the tensor filter's limit"


@pytest.mark.parametrize("n", SWEEP)
def test_sweep_scene_has_its_count_and_hits_in_the_tail(r1, oracle, host_scenes, n):
    """the scene has n spheres (unpadded counts stay unpadded), the last is the ground, and the rays hit every part of it:
    the spheres after the last full 32-sphere chunk (or the last chunk) a few hundred times"""
    s = host_scenes("n%d" % n)
    soa = s.soa()
    assert s.count() == n and (soa["inv_radius"] > 0).all()
    assert soa["radius_sq"][-1] == 1.0e6 and soa["cy"][-1] == -1000
    org, d = scene_rays("n%d" % n, soa)
    so = oracle.scene_create_from_soa(soa)
    idx = oracle.hit(so, org, d)[0]
    oracle.scene_destroy(so)
    tail = ((n + 7) // 8 * 8 - 1) // 32 * 32
    assert (idx >= tail).sum() >= 300
    if n >= 64:
        assert ((idx >= 0) & (idx < tail)).sum() >= 300
    assert (idx < 0).sum() >= 100


@pytest.mark.parametrize("n", FLOODS)
def test_floods_flag_nearly_every_sphere(r1, host_scenes, n):
    """float64 discr >= 0 for >= 90 % of the spheres on >= 90 % of the rays: every 32-sphere chunk of every warp puts far more
    than 60 entries (the cooperative queue's drain threshold) into the queues"""
    soa = host_scenes("flood%d" % n).soa()
    org, d = flood_rays()
    c = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1).astype(np.float64)
    co = c[None, :, :] - org.astype(np.float64)[:, None, :]
    nb = np.einsum("rsk,rk->rs", co, d.astype(np.float64))
    discr = nb * nb - (co * co).sum(-1) + soa["radius_sq"].astype(np.float64)[None, :]
    flagged = discr >= 0
    assert (flagged.mean(1) >= 0.9).mean() >= 0.9
    warps = flagged[: len(org) // 32 * 32, : n // 32 * 32].reshape(-1, 32, n // 32, 32).sum((1, 3))
    assert warps.min() > 60
    inside = (np.linalg.norm(co[600:], axis=-1) < np.sqrt(soa["radius_sq"])[None, :]).all(1)
    assert inside.all(), "the last 400 rays start inside every sphere"


def test_tie_scene_duplicates_and_near_ties(r1, oracle, host_scenes):
    """exact duplicates: bit-identical sphere records, materials differ, and the oracle returns the lower index for every ray
    that reaches the pair; near-ties: roots one ulp apart on the axis ray, the nearer sphere returned"""
    soa = host_scenes("ties").soa()
    geo = ("cx", "cy", "cz", "radius_sq", "inv_radius")
    for lo, hi in TIE_PAIRS:
        assert all(soa[k][lo].view(np.uint32) == soa[k][hi].view(np.uint32) for k in geo)
        assert soa["kind"][lo] != soa["kind"][hi]
    org, d = scene_rays("ties", soa)
    so = oracle.scene_create_from_soa(soa)
    idx = oracle.hit(so, org, d)[0]
    for lo, hi in TIE_PAIRS:
        assert (idx == lo).sum() >= 60 and (idx == hi).sum() == 0, (lo, hi)
    o, dd = near_tie_rays()
    near = oracle.hit(so, o, dd)
    oracle.scene_destroy(so)
    for k, (lo, hi, nearer) in enumerate(NEAR_PAIRS):
        roots = {}
        for i in (lo, hi):
            one = oracle.scene_create_from_soa({key: v[i:i + 1] for key, v in soa.items()})
            roots[i] = oracle.hit(one, o[k:k + 1], dd[k:k + 1])[1][0]
            oracle.scene_destroy(one)
        assert roots[nearer] == np.nextafter(roots[lo + hi - nearer], F32(-np.inf)), (lo, hi, roots)
        assert near[0][k] == nearer and near[1][k] == roots[nearer]


@pytest.mark.parametrize("name", BOUNDARY_SCENES)
@pytest.mark.parametrize("t_min", (0.001, T_BOUND), ids=("tmin_0.001", "tmin_2^-24"))
def test_boundary_queries_reach_both_outcomes(r1, oracle, host_scenes, name, t_min):
    """t_max = t excludes the hit and one ulp more includes it; t_min = t excludes the near root -- for some rays the same
    sphere's far root answers, for others another sphere or nothing (in the flood always another sphere: dozens of far roots
    lie just behind) -- and one ulp less keeps it"""
    soa = host_scenes(name).soa()
    so = oracle.scene_create_from_soa(soa)
    org, d, t = boundary_rays(name, soa, so, oracle, t_min)
    first = oracle.hit(so, org, d, t_min)
    assert len(org) >= 40 and (first[0] >= 0).all()
    same_far = other = 0
    for k in range(len(org)):
        res = [oracle.hit(so, org[k:k + 1], d[k:k + 1], lo, hi) for lo, hi in boundary_queries(t_min, t[k])]
        assert res[0][0][0] == -1, "t_max = t excludes the hit"
        assert res[1][0][0] == first[0][k] and res[1][1][0] == t[k], "t_max = t + ulp includes it"
        assert res[3][0][0] == first[0][k] and res[3][1][0] == t[k], "t_min = t - ulp includes it"
        assert res[2][0][0] == -1 or res[2][1][0] > t[k], "t_min = t excludes it"
        same_far += int(res[2][0][0] == first[0][k])
        other += int(res[2][0][0] != first[0][k])
    oracle.scene_destroy(so)
    assert (same_far >= 10 or name.startswith("flood")) and other >= 5, (same_far, other)


def test_tangent_rays_have_a_zero_discriminant(r1, oracle, host_scenes):
    """discr = fma(nb, nb, -q) + r^2 is +0 (sign bit clear: a candidate) in float32 for every tangent ray, and the oracle hits
    the pair's lower index at t = L, the tangent point"""
    soa = host_scenes("ties").soa()
    org, d = tangent_rays()
    per_pair = len(org) // len(TIE_PAIRS)
    f64 = np.float64
    for k, (lo, _) in enumerate(TIE_PAIRS):
        c = np.array([soa["cx"][lo], soa["cy"][lo], soa["cz"][lo]], F32)
        assert tuple(c) == pair_centre(k)
        for o, dd in zip(org[k * per_pair:(k + 1) * per_pair], d[k * per_pair:(k + 1) * per_pair]):
            co = (c - o).astype(F32)
            # every product and sum below is exact in float32 (small integers), so float64 arithmetic rounds like the fmas
            nb = F32(f64(co[2]) * dd[2] + F32(f64(co[1]) * dd[1] + F32(co[0] * dd[0])))
            q = F32(f64(co[2]) * co[2] + F32(f64(co[1]) * co[1] + F32(co[0] * co[0])))
            discr = F32(F32(f64(nb) * nb - f64(q)) + soa["radius_sq"][lo])
            assert discr == 0 and not np.signbit(discr)
    so = oracle.scene_create_from_soa(soa)
    res = oracle.hit(so, org, d)
    oracle.scene_destroy(so)
    want_idx = np.repeat([lo for lo, _ in TIE_PAIRS], per_pair)
    assert np.array_equal(res[0], want_idx)
    assert np.array_equal(res[1], np.abs(org[:, 2] - np.repeat([pair_centre(k)[2] for k in range(len(TIE_PAIRS))], per_pair)))


@pytest.mark.parametrize("t_min", (0.0, -1.0, float("nan"), 2.0 ** -25), ids=("0", "-1", "nan", "2^-25"))
def test_trace_rays_refuses_t_min_below_2_pow_minus_24(r1, t_min):
    """below 2^-24 the floored square root and the unsigned root keys can differ from Hitable::hit: refused with R1_ERR_ARG before
    the device is looked at (this scene is not even committed)"""
    s = r1.create_scene("small", commit=False)
    try:
        with pytest.raises(r1.Rays1Error, match=r"\(-1\).*2\^-24"):
            s.trace_rays([[0, 1, 3]], [[0, 0, -1]], t_min=t_min)
    finally:
        s.close()


def test_unpadded_scenes_stay_unpadded(r1, host_scenes):
    for n in UNPADDED:
        s = host_scenes("n%d" % n)
        assert s.count() == n and len(s.soa()["cx"]) == n
