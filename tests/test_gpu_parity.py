"""Parity of the CUDA path (through the C ABI) against the reference: golden vectors recorded from the reference's
compiled code, the oracle on fresh seeded inputs, and size-independent properties at the full BASELINE.json sizes.
Tolerances: hit index exact; t / p / normal / scatter direction within 1e-5 (north_star; in practice hit results are
bit-identical because the exact candidate path uses the reference's as-built arithmetic); rays per sample within 0.5 %;
per-channel image RMSE vs the reference's 16384-spp render <= 1/255."""
import os
import subprocess

import numpy as np
import pytest

from conftest import SCENES, rmse

pytestmark = pytest.mark.gpu

REL = 1e-5
ALL = SCENES + ("synth4096",)   # synth4096 = BASELINE.json config 5; its fixtures come from the MAX_SPHERES = 4096 build of the reference


def record(key, value):
    """measured maxima, kept next to the run (gpurun_out/parity_errors.json) so that they can be quoted in profiles/"""
    import json
    from conftest import ROOT
    path = os.path.join(ROOT, "gpurun_out", "parity_errors.json")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        data = json.load(open(path)) if os.path.exists(path) else {}
        data[key] = value
        json.dump(data, open(path, "w"), indent=1, sort_keys=True)
    except OSError:
        pass
    print("%s: %s" % (key, value))


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def scenes(r1):
    r1.configure(width=1280, height=720, spp=250, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=True)
    out = {name: r1.create_scene(name) for name in SCENES + ("synth4096",)}
    yield out
    for s in out.values():
        s.close()


# ---- hit() ----------------------------------------------------------------------------------------------------------

def refuses_tensor(r1, scene, org, d):
    """above 768 spheres the tensor-core filter has no operand: R1_ERR_LIMIT, never a silent fall-back to another scan"""
    with pytest.raises(r1.Rays1Error, match=r"\(-4\).*768"):
        scene.trace_rays(org, d, variant=r1.VARIANT_MEGAKERNEL_TENSOR)


# "mega" resolves as in r1_render: the tensor-core filter on the large scene, the packed scan elsewhere
@pytest.mark.parametrize("variant", ["mega", "coop", "scalar", "deferred", "tensor", "packed"])
@pytest.mark.parametrize("name", ALL)
def test_hit_matches_reference_golden(r1, scenes, golden_rays, name, variant):
    g = golden_rays[name]
    org = np.concatenate([g["seg_org"], g["edge_org"]])
    d = np.concatenate([g["seg_dir"], g["edge_dir"]])
    want_idx = np.concatenate([g["seg_index"], g["edge_index"]])
    want_t = np.concatenate([g["seg_t"], g["edge_t"]])
    want_p = np.concatenate([g["seg_p"], g["edge_p"]])
    want_n = np.concatenate([g["seg_normal"], g["edge_normal"]])
    if variant == "tensor" and name == "synth4096":
        return refuses_tensor(r1, scenes[name], org, d)
    idx, t, p, n = scenes[name].trace_rays(org, d, variant=r1.VARIANTS[variant])
    assert np.array_equal(idx, want_idx), "hit sphere index differs for %d rays" % int((idx != want_idx).sum())
    m = idx >= 0
    assert m.sum() > 1000
    assert np.abs(t[m] - want_t[m]).max() <= REL * np.abs(want_t[m]).max()
    assert (np.abs(t[m] - want_t[m]) <= REL * np.abs(want_t[m])).all()
    assert np.abs(p[m] - want_p[m]).max() <= REL * max(1.0, np.abs(want_p[m]).max())
    assert np.abs(n[m] - want_n[m]).max() <= REL
    # stronger than the contract: the exact path reproduces the reference's arithmetic bit for bit
    assert np.array_equal(bits(t[m]), bits(want_t[m]))
    assert np.array_equal(bits(n[m]), bits(want_n[m]))
    assert (t[~m] == 0).all()


@pytest.mark.parametrize("name", SCENES + ("synth4096",))
def test_hit_matches_oracle_on_fresh_rays(r1, scenes, oracle, name):
    """seeded random rays from points around the scene (inside spheres, on the ground, far away), incl. the 4096-sphere scene"""
    rng = np.random.default_rng(1234)
    n = 6000
    org = (rng.normal(size=(n, 3)) * [8, 2, 8] + [0, 2, 0]).astype(np.float32)
    org[: n // 4] = (rng.normal(size=(n // 4, 3)) * [12, 0.02, 7] + [0, 0.5, 0]).astype(np.float32)  # among the small spheres
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    so = oracle.scene_create(name)
    for t_min, t_max in ((0.001, float(np.finfo(np.float32).max)), (0.5, 6.0)):
        want = oracle.hit(so, org, d, t_min, t_max)
        got = scenes[name].trace_rays(org, d, t_min, t_max)
        assert np.array_equal(got[0], want[0])
        m = want[0] >= 0
        assert m.sum() > 500
        assert np.array_equal(bits(got[1][m]), bits(want[1][m]))
        assert np.array_equal(bits(got[2][m]), bits(want[2][m]))
        assert np.array_equal(bits(got[3][m]), bits(want[3][m]))
    oracle.scene_destroy(so)


@pytest.mark.parametrize("variant", ["mega", "coop", "scalar", "deferred", "tensor", "packed"])
@pytest.mark.parametrize("name", ("large", "synth4096"))
def test_filter_is_conservative_for_far_and_grazing_rays(r1, scenes, oracle, name, variant):
    """The 8-instruction filter works in the expanded form (cancellation at |o|^2 + |c|^2): rays from far away that graze
    a sphere within +-2 % of its radius are where a non-conservative filter would lose hits.  Bit-exact vs the oracle."""
    rng = np.random.default_rng(4321)
    soa = scenes[name].soa()
    real = np.where(soa["inv_radius"] > 0)[0]
    n = 6000
    idx = rng.choice(real, n)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1).astype(np.float64)
    rad = 1.0 / soa["inv_radius"][idx].astype(np.float64)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    u[:, 1] = np.abs(u[:, 1])                                   # stay above the ground plane
    dist = rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n)
    org = ctr + u * dist[:, None]
    side = np.cross(u, rng.normal(size=(n, 3))); side /= np.linalg.norm(side, axis=1, keepdims=True)
    target = ctr + side * (rad * rng.uniform(0.98, 1.02, n))[:, None]
    d = target - org; d /= np.linalg.norm(d, axis=1, keepdims=True)
    org, d = org.astype(np.float32), d.astype(np.float32)
    if variant == "tensor" and name == "synth4096":
        return refuses_tensor(r1, scenes[name], org, d)
    so = oracle.scene_create(name)
    want = oracle.hit(so, org, d)
    oracle.scene_destroy(so)
    got = scenes[name].trace_rays(org, d, variant=r1.VARIANTS[variant])
    assert np.array_equal(got[0], want[0]), "%d rays lost or gained a hit" % int((got[0] != want[0]).sum())
    m = want[0] >= 0
    assert m.sum() > 1500
    assert np.array_equal(bits(got[1][m]), bits(want[1][m]))
    assert np.array_equal(bits(got[3][m]), bits(want[3][m]))


def tensor_filter_rays(soa, n=4096, seed=99):
    """fresh rays around the scene + rays grazing spheres from 5 .. 300 units away"""
    rng = np.random.default_rng(seed)
    org = (rng.normal(size=(n, 3)) * [8, 2, 8] + [0, 2, 0])
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    idx = rng.choice(real, n)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1).astype(np.float64)
    rad = 1.0 / soa["inv_radius"][idx].astype(np.float64)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    o2 = ctr + u * rng.choice([5.0, 50.0, 300.0], n)[:, None]
    side = np.cross(u, rng.normal(size=(n, 3))); side /= np.linalg.norm(side, axis=1, keepdims=True)
    d2 = ctr + side * (rad * rng.uniform(0.98, 1.02, n))[:, None] - o2
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True)
    return np.concatenate([org, o2]).astype(np.float32), np.concatenate([d, d2]).astype(np.float32)


def tensor_filter_far_rays(soa, n=2048, seed=77):
    """tensor_filter_rays plus rays grazing spheres from 2 000 and 20 000 units away (where the FFMA2 filter is tested too):
    the filter's cancellation grows with |o|^2"""
    rng = np.random.default_rng(seed)
    org, d = tensor_filter_rays(soa, n, seed)
    real = np.where(soa["inv_radius"] > 0)[0]
    idx = rng.choice(real, n)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1).astype(np.float64)
    rad = 1.0 / soa["inv_radius"][idx].astype(np.float64)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    u[:, 1] = np.abs(u[:, 1])                                   # stay above the ground plane
    o3 = ctr + u * rng.choice([2000.0, 20000.0], n)[:, None]
    side = np.cross(u, rng.normal(size=(n, 3))); side /= np.linalg.norm(side, axis=1, keepdims=True)
    d3 = ctr + side * (rad * rng.uniform(0.98, 1.02, n))[:, None] - o3
    d3 /= np.linalg.norm(d3, axis=1, keepdims=True)
    return np.concatenate([org, o3.astype(np.float32)]), np.concatenate([d, d3.astype(np.float32)])


def tensor_filter_truth(soa, org, d, margin=2.0 ** -16):
    """float64 values of the filter polynomial and of Hitable::hit's discriminant for every (ray, sphere), from the float32 inputs"""
    o, dd = org.astype(np.float64), d.astype(np.float64)
    c = np.stack([soa["cx"], soa["cy"], soa["cz"]], 1).astype(np.float64)
    r2 = soa["radius_sq"].astype(np.float64)
    co = c[None, :, :] - o[:, None, :]
    nb = (co * dd[:, None, :]).sum(2)
    discr = nb * nb - ((co * co).sum(2) - r2[None, :])
    big_s = (c * c).sum(1)[None, :] + (o * o).sum(1)[:, None]
    return discr + margin * big_s, discr, big_s


@pytest.mark.parametrize("name", ("large", "medium", "small"))
def test_tensor_filter_is_conservative(r1, scenes, name):
    """R1_VARIANT_MEGAKERNEL_TENSOR evaluates the filter as a TF32 GEMM with split operands (r1_tensor.cuh).  Its values must stay
    within a fraction of the margin of the float64 polynomial, and every sphere whose discriminant the exact test could accept
    (true value above minus the exact path's own rounding bound) must be flagged."""
    soa = scenes[name].soa()
    n_sph = len(soa["cx"])
    org, d = tensor_filter_rays(soa)
    e = scenes[name].filter_probe(org, d, n_sph).astype(np.float64)
    want, discr, big_s = tensor_filter_truth(soa, org, d)
    real = soa["inv_radius"] > 0
    err = np.abs(e[:, :n_sph] - want)[:, real] / big_s[:, real]
    record("tensor_filter_rel_err_%s" % name, {"max": float(err.max()), "p99.9": float(np.quantile(err, 0.999)), "margin": 2.0 ** -16})
    assert err.max() < 0.1 * 2.0 ** -16, "tensor filter error %.3g of S eats the margin" % err.max()
    must = (discr >= -4.0e-6 * big_s) & real[None, :]            # the exact path's rounding bound is 3.1e-6 S (DESIGN.md section 4.1)
    assert must.sum() > 4000
    assert (e[:, :n_sph][must] >= 0).all() and not np.signbit(e[:, :n_sph][must]).any()
    assert (e[:, n_sph:] < 0).all() and (e[:, :n_sph][:, ~real] < 0).all(), "padding rows must never be flagged"
    flagged = (~np.signbit(e[:, :n_sph])) & real[None, :]
    record("tensor_filter_flag_ratio_%s" % name, float(flagged.sum() / max(1, ((discr >= 0) & real[None, :]).sum())))


def test_tensor_renders_the_same_bytes_at_every_group_count(r1, scenes):
    """same hits, same bytes: the tensor-core filter only decides which spheres get the exact test.  r1::megakernel_tc3 at the
    default and at every group count it builds (threads = 128 x groups), on four frames; rank shares; the shared-memory limit."""
    for name, (w, h, spp) in (("large", (200, 117, 40)), ("medium", (160, 90, 16)), ("small", (64, 36, 8)), ("large", (7, 3, 5))):
        base, r0 = scenes[name].render(w, h, spp, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        for groups in (None, 4, 5, 6, 7):                        # accumulator buffers pooled among the groups
            alt, ra = scenes[name].render(w, h, spp, variant=r1.VARIANT_MEGAKERNEL_TENSOR, threads=128 * groups if groups else 0)
            assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays, (name, "tc3", groups)
    for world in (2, 3):
        parts = [scenes["large"].render(200, 117, 40, rank=r, world=world, variant=r1.VARIANT_MEGAKERNEL_TENSOR)[0] for r in range(world)]
        whole, _ = scenes["large"].render(200, 117, 40, variant=r1.VARIANT_MEGAKERNEL_PACKED)
        rows = [r1.global_row(lr, r1.DEFAULT_ROW_TILE, r, world) for r in range(world) for lr in range(parts[r].shape[0])]
        assert np.array_equal(np.concatenate(parts)[np.argsort(rows)], whole)
    with pytest.raises(r1.Rays1Error):
        scenes["synth4096"].render(64, 36, 2, variant=r1.VARIANT_MEGAKERNEL_TENSOR)   # above the shared-memory limit of the B tile


def test_default_variant_picks_the_kernel_by_scene(r1, scenes):
    """R1_VARIANT_MEGAKERNEL: the tensor-core filter for scan-heavy scenes that fit its shared-memory operand, else the packed filter"""
    name = lambda scene, v=r1.VARIANT_MEGAKERNEL: r1.lib.r1_kernel_name(scenes[scene].handle, v).decode()  # noqa: E731
    assert name("large") == "megakernel_tc3" and name("medium") == "megakernel_pool" and name("small") == "megakernel_pool"
    assert name("synth4096") == "megakernel_pool"
    assert name("large", r1.VARIANT_MEGAKERNEL_PACKED) == "megakernel_pool" and name("large", r1.VARIANT_MEGAKERNEL_TENSOR) == "megakernel_tc3"


def test_trace_rays_refuses_variants_without_a_ray_kernel(r1, scenes):
    """wavefront and dual have no per-ray kernel: refused, not answered by another scan; so is an unknown variant"""
    for v in (r1.VARIANT_WAVEFRONT, r1.VARIANT_MEGAKERNEL_DUAL, 8, -1):
        with pytest.raises(r1.Rays1Error, match=r"\(-1\)"):
            scenes["large"].trace_rays([[0, 5, 20]], [[0, 0, -1]], variant=v)
    idx, _, _, _ = scenes["large"].trace_rays([[0, 3, 20]], [[0, 0, -1]], variant=r1.VARIANT_MEGAKERNEL_TENSOR)
    assert idx[0] >= 0


def test_hit_empty_and_single(r1, scenes):
    idx, t, p, n = scenes["small"].trace_rays(np.zeros((0, 3)), np.zeros((0, 3)))
    assert idx.shape == (0,)
    idx, t, p, n = scenes["small"].trace_rays([[0, 0, 5]], [[0, 0, -1]])
    assert idx[0] == 0 and t[0] == pytest.approx(5.5)


# ---- scatter() / camera -------------------------------------------------------------------------------------------------
# Tolerance: 1e-5 FLAT for every material, every ior (north_star).  Stronger, and asserted: the device follows the association
# of the reference's binary including its rsqrtss + Newton normalise (r1_device.cuh "scatter", "unit3"), so the scattered
# direction, the attenuation and the flag are BIT-IDENTICAL to the reference's on every recorded ray.

def per_material_max(err, kinds):
    return {("lambert", "metal", "dielectric")[k]: float(err[kinds == k].max()) for k in (0, 1, 2) if (kinds == k).any()}


@pytest.mark.parametrize("name", ALL)
def test_scatter_matches_reference_golden(r1, scenes, golden_rays, name):
    g = golden_rays[name]
    m = (g["seg_index"] >= 0) & (g["seg_depth"] < 50)
    ok, att, dout = scenes[name].scatter(g["seg_dir"][m], g["seg_p"][m], g["seg_normal"][m], g["seg_index"][m],
                                         g["seg_rand_sphere"][m], g["seg_rand_u"][m])
    assert np.array_equal(ok, g["seg_scat_ok"][m])
    assert np.array_equal(bits(att), bits(g["seg_atten"][m])) or np.abs(att - g["seg_atten"][m]).max() < 1e-7
    err = np.abs(dout - g["seg_scat_dir"][m]).max(axis=1)
    kinds = scenes[name].soa()["kind"][g["seg_index"][m]]
    record("scatter_golden_max_abs_err/%s" % name, per_material_max(err, kinds))
    assert (err <= REL).all(), "scatter direction off by %g" % err.max()
    assert np.array_equal(bits(dout), bits(g["seg_scat_dir"][m])) and np.array_equal(bits(att), bits(g["seg_atten"][m]))
    for k in (0, 1, 2):
        assert (kinds == k).sum() > 20, "material %d under-sampled" % k


@pytest.mark.parametrize("name", ("large", "synth4096"))
def test_dielectric_exit_rays_match_reference_golden(r1, scenes, golden_rays, name):
    """rays leaving the ior >= 5 dielectric spheres from inside (320 on the large scene, ior up to 24.2, rayweek1.cpp:692; 2704
    on synth4096): hit() bit-identical, Dielectric::scatter within 1e-5 flat -- both the refracting rays, where
    1 - k^2 (1 - dt^2) amplifies rounding by k^2 <= 585, and the totally reflected ones"""
    g = golden_rays[name]
    idx, t, p, n = scenes[name].trace_rays(g["diel_org"], g["diel_dir"])
    assert np.array_equal(idx, g["diel_index"]) and len(idx) >= 200
    assert np.array_equal(bits(t), bits(g["diel_t"])) and np.array_equal(bits(n), bits(g["diel_normal"])) and np.array_equal(bits(p), bits(g["diel_p"]))
    soa = scenes[name].soa()
    assert (soa["kind"][idx] == 2).all() and (soa["param"][idx] >= 5).all()
    ok, att, dout = scenes[name].scatter(g["diel_dir"], p, n, idx, g["diel_rand_sphere"], g["diel_rand_u"])
    assert ok.all() and (att == 1).all()
    err = np.abs(dout - g["diel_scat_dir"]).max(axis=1)
    refracted = (g["diel_scat_dir"] * g["diel_normal"]).sum(1) > 0
    assert refracted.sum() >= 150 and (~refracted).sum() >= 100
    record("scatter_dielectric_exit_max_abs_err/%s" % name, {"refracted": float(err[refracted].max()), "reflected": float(err[~refracted].max()),
                                                              "max_ior": float(soa["param"][idx].max()), "rays": int(len(idx))})
    assert (err <= REL).all(), err.max()
    assert np.array_equal(bits(dout), bits(g["diel_scat_dir"]))


@pytest.mark.parametrize("name", ALL)
def test_scatter_matches_oracle_on_fresh_inputs(r1, scenes, oracle, name):
    rng = np.random.default_rng(99)
    n = 4000
    soa = scenes[name].soa()
    real = np.where(soa["inv_radius"] > 0)[0]
    idx = rng.choice(real, n).astype(np.int32)
    diel = np.where((soa["kind"] == 2) & (soa["inv_radius"] > 0))[0]
    idx[: n // 4] = rng.choice(diel, n // 4)                       # a quarter of the inputs on dielectrics of every ior, half of them exiting
    nrm = rng.normal(size=(n, 3)); nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    din = rng.normal(size=(n, 3)); din = (din / np.linalg.norm(din, axis=1, keepdims=True)).astype(np.float32)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1)
    p = (ctr + nrm / soa["inv_radius"][idx][:, None]).astype(np.float32)
    rs = rng.uniform(-1, 1, size=(n * 3, 3)); rs = rs[(rs ** 2).sum(1) < 1][:n].astype(np.float32)
    ru = rng.uniform(0, 1, n).astype(np.float32)
    so = oracle.scene_create(name)
    want = oracle.scatter(so, din, p, nrm, idx, rs, ru)
    got = scenes[name].scatter(din, p, nrm, idx, rs, ru)
    oracle.scene_destroy(so)
    err = np.abs(got[2] - want[2]).max(axis=1)
    record("scatter_fresh_vs_oracle_max_abs_err/%s" % name, per_material_max(err, soa["kind"][idx]))
    assert (err <= REL).all(), err.max()
    # the same arithmetic on both sides: the same bits, including Metal's dot(dir, n) > 0 decision
    assert np.array_equal(got[0], want[0]) and np.array_equal(bits(got[1]), bits(want[1])) and np.array_equal(bits(got[2]), bits(want[2]))


@pytest.mark.parametrize("name", ALL)
def test_camera_rays_match_reference_golden(r1, scenes, golden_rays, name):
    g = golden_rays[name]
    m = g["seg_depth"] == 0
    org, d = scenes[name].get_ray(g["seg_cam_su"][m], g["seg_cam_tv"][m], g["seg_cam_disk"][m])
    assert np.abs(org - g["seg_org"][m]).max() <= REL * np.abs(g["seg_org"][m]).max()
    assert np.abs(d - g["seg_dir"][m]).max() <= REL
    # stronger: the binary's association, its normalise and its camera constants -> Camera::getRay is bit-identical
    assert np.array_equal(bits(scenes[name].camera()), bits(g["camera"]))
    assert np.array_equal(bits(org), bits(g["seg_org"][m])) and np.array_equal(bits(d), bits(g["seg_dir"][m]))
    # and r1_scene_set_camera_raw installs constants as given
    s = r1.create_scene(name)
    cam = g["camera"].copy(); cam[0] += 0.5
    s.set_camera_raw(cam, device=0)
    org2, _ = s.get_ray(g["seg_cam_su"][m][:8], g["seg_cam_tv"][m][:8], np.zeros((8, 2), np.float32))
    s.close()
    assert np.allclose(org2[:, 0], cam[0]) and not np.allclose(org2[:, 0], g["camera"][0])


# ---- RNG ------------------------------------------------------------------------------------------------------------------------

def test_rng_is_counter_based_and_uniform(r1):
    a = r1.rng_draws(123, 45, 0, 64)
    assert np.array_equal(a, r1.rng_draws(123, 45, 0, 64)), "same (pixel, sample, seed) -> same stream"
    assert np.array_equal(a[:16], r1.rng_draws(123, 45, 0, 16)), "draw k does not depend on how many draws follow"
    assert not np.array_equal(a, r1.rng_draws(124, 45, 0, 64))
    assert not np.array_equal(a, r1.rng_draws(123, 46, 0, 64))
    assert not np.array_equal(a, r1.rng_draws(123, 45, 1, 64))
    # first draws of 20000 consecutive (pixel, sample) keys: uniform in [0,1) at 24-bit resolution, uncorrelated
    firsts = np.array([r1.rng_draws(p, s, 0, 2) for p in range(200) for s in range(100)], np.uint32)
    u = (firsts >> 8).astype(np.float64) / 2 ** 24
    assert abs(u.mean() - 0.5) < 0.01 and abs(u.var() - 1 / 12) < 0.005
    hist, _ = np.histogram(u[:, 0], bins=64, range=(0, 1))
    chi2 = ((hist - hist.mean()) ** 2 / hist.mean()).sum()
    assert chi2 < 120, chi2  # 63 dof, p ~ 1e-5
    assert abs(np.corrcoef(u[:, 0], u[:, 1])[0, 1]) < 0.03
    assert abs(np.corrcoef(u[:-1, 0], u[1:, 0])[0, 1]) < 0.03


# ---- the trace loop: statistics against the reference ------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ALL)
def test_image_rmse_and_rays_per_sample_vs_reference(r1, scenes, golden_render, ref_stats, name):
    """matched high spp: reference 16384 spp (tests/golden) vs GPU 16384 spp at 320x180.  synth4096 (config 5) is compared with
    the reference built with MAX_SPHERES = 4096 (rayweek1.cpp:174), not with the oracle port."""
    g = golden_render[name]
    h, w = g["rgb"].shape[:2]
    spp = int(g["spp"])
    rgb, res = scenes[name].render(w, h, spp)
    e = rmse(rgb, g["rgb"])
    rps = res.num_rays / (w * h * spp)
    ref = ref_stats["default_workload"][name]["rays_per_sample"]
    ref_same = ref_stats["render"][name]["rays_per_sample"]        # the reference's own count for this very render
    record("render_320x180x%d/%s" % (spp, name), {"rmse_per_channel_255": e, "rays_per_sample": rps, "reference_rays_per_sample": ref_same,
                                                   "reference_rays_per_sample_1280x720": ref})
    assert e <= 1.0, "per-channel RMSE %.3f / 255 exceeds 1/255" % e
    assert abs(rps / ref - 1) < 0.005, (rps, ref)
    assert abs(rps / ref_same - 1) < 0.005, (rps, ref_same)
    assert res.num_samples == w * h * spp
    # no systematic bias per channel either
    bias = (rgb.astype(np.float64) - g["rgb"]).mean(axis=(0, 1))
    assert np.abs(bias).max() < 0.25, bias


@pytest.mark.parametrize("name", ALL)
def test_full_size_default_workload(r1, scenes, ref_stats, name):
    """BASELINE.json configs 1-3 and 5 at full size: 1280x720x250, depth 50."""
    rgb, res = scenes[name].render(1280, 720, 250)
    ref = ref_stats["default_workload"][name]
    rps = res.num_rays / (1280 * 720 * 250)
    record("rays_per_sample_1280x720x250/%s" % name, {"gpu": rps, "reference": ref["rays_per_sample"]})
    assert abs(rps / ref["rays_per_sample"] - 1) < 0.005
    assert rgb.shape == (720, 1280, 3) and res.num_samples == 1280 * 720 * 250
    # sky at the top of the picture (last rows: row 0 is the BOTTOM), gradient blue > red
    top = rgb[-20:].reshape(-1, 3).mean(0)
    assert top[2] > top[0] and top[2] > 200
    assert res.launches == 2 and res.kernel_ms > 0 and res.trace_ms <= res.kernel_ms


def test_config4_4k_sample_counts_need_64_bits(r1, ref_stats, capfd):
    """BASELINE.json config 4: large scene, 3840x2160, 1024 spp = 8 493 465 600 samples -- the count the reference itself
    gets wrong (int arithmetic, rayweek1.cpp:893).  (a) rays per sample at 4K within 0.5 % of the reference's figure for this
    scene (the camera keeps its 16:9 aspect, so the figure does not depend on the resolution); (b) one rank's share of the
    8-GPU partition at the full 1024 spp; (c) the whole image through benchmark(): total samples and rays beyond 2^32."""
    W, H, SPP = 3840, 2160, 1024
    r1.configure(width=W, height=H, spp=SPP, max_bounces=50, variant=0, n_gpus=1, seed=0, quiet=False)
    try:
        scene = r1.create_large_scene()
        ref = ref_stats["default_workload"]["large"]["rays_per_sample"]
        rgb, res = scene.render(W, H, 16)
        assert rgb.shape == (H, W, 3) and res.num_samples == W * H * 16
        assert abs(res.num_rays / (W * H * 16) / ref - 1) < 0.005
        part, rp = scene.render(W, H, SPP, rank=0, world=8)
        assert part.shape == (270, W, 3) and rp.num_samples == W * 270 * SPP == 1061683200
        assert abs(rp.num_rays / rp.num_samples / ref - 1) < 0.01          # an eighth of the rows (every 8th row)
        capfd.readouterr()
        pixels = np.zeros((H, W, 3), np.uint8)
        out = r1.benchmark(scene, pixels, False, "large")                  # the reference-facing call; ~4 s of GPU time
        lines = capfd.readouterr().out.splitlines()
        assert "total samples:  %d" % (W * H * SPP) in lines and W * H * SPP == 8493465600 > 2 ** 32
        assert "total rays:     %d" % out.num_rays in lines and out.num_rays > 2 ** 32
        assert abs(out.num_rays / (W * H * SPP) / ref - 1) < 0.005
        record("config4_3840x2160x1024", {"num_samples": W * H * SPP, "num_rays": int(out.num_rays), "rays_per_sample": out.num_rays / (W * H * SPP),
                                          "kernel_ms": out.kernel_ms})
        rows8 = [r1.global_row(lr, r1.DEFAULT_ROW_TILE, 0, 8) for lr in range(270)]
        assert np.array_equal(pixels[rows8], part), "the 8-GPU share is a subset of the single-GPU picture, byte for byte"
    finally:
        r1.configure(width=1280, height=720, spp=250, quiet=True)


@pytest.mark.parametrize("name", SCENES)
def test_wavefront_full_size_matches_megakernel(r1, scenes, name):
    """the wavefront variant (queues compacted with ballot + popc, CUDA-graph loop) renders the same bytes at full size"""
    a, ra = scenes[name].render(1280, 720, 32)
    b, rb = scenes[name].render(1280, 720, 32, variant=r1.VARIANT_WAVEFRONT)
    assert np.array_equal(a, b) and ra.num_rays == rb.num_rays
    part, rp = scenes[name].render(1280, 720, 32, variant=r1.VARIANT_WAVEFRONT, rank=1, world=4)
    rows = [r1.global_row(lr, r1.DEFAULT_ROW_TILE, 1, 4) for lr in range(part.shape[0])]
    assert np.array_equal(part, a[rows])


def test_wavefront_graph_is_cached_across_renders(r1, scenes):
    """the wavefront's CUDA-graph WHILE loop is instantiated once and re-launched while the render arguments stay the same"""
    s = scenes["medium"]
    a, ra = s.render(160, 90, 8, variant=r1.VARIANT_WAVEFRONT)
    n0 = r1.lib.r1_wavefront_graph_builds(0)
    for _ in range(3):
        b, rb = s.render(160, 90, 8, variant=r1.VARIANT_WAVEFRONT)
        assert np.array_equal(a, b) and ra.num_rays == rb.num_rays
    assert r1.lib.r1_wavefront_graph_builds(0) == n0, "same arguments: no rebuild"
    c, rc = s.render(160, 90, 9, variant=r1.VARIANT_WAVEFRONT)
    assert r1.lib.r1_wavefront_graph_builds(0) == n0 + 1, "another spp: rebuilt once"
    ref, rr = s.render(160, 90, 9)
    assert np.array_equal(c, ref) and rc.num_rays == rr.num_rays


# ---- determinism / partition invariance --------------------------------------------------------------------------------

def test_bitwise_invariance(r1, scenes):
    """same (w, h, spp, seed) -> same bytes for: repeat runs, the scalar scan, 2 / 3 / 8 interleaved ranks, other CTA counts"""
    s = scenes["large"]
    w, h, spp = 200, 117, 40
    base, r0 = s.render(w, h, spp)
    again, r1_ = s.render(w, h, spp)
    assert np.array_equal(base, again) and r0.num_rays == r1_.num_rays
    for v in (r1.VARIANT_MEGAKERNEL_SCALAR, r1.VARIANT_MEGAKERNEL_COOP, r1.VARIANT_MEGAKERNEL_DEFERRED, r1.VARIANT_MEGAKERNEL_DUAL,
              r1.VARIANT_MEGAKERNEL_PACKED, r1.VARIANT_MEGAKERNEL_TENSOR):
        alt, ra = s.render(w, h, spp, variant=v)
        assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays, v
    more, rm = s.render(w, h, spp, blocks_per_sm=2)
    assert np.array_equal(base, more) and rm.num_rays == r0.num_rays
    for threads in (512, 768):
        alt, ra = s.render(w, h, spp, threads=threads)
        assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays
    alt, ra = s.render(w, h, spp, threads=512, variant=r1.VARIANT_MEGAKERNEL_DUAL)
    assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays
    tiny, rt = s.render(7, 3, 5)                                  # fewer samples than one warp's 64 path slots
    tiny2, rt2 = s.render(7, 3, 5, variant=r1.VARIANT_MEGAKERNEL_DUAL)
    assert np.array_equal(tiny, tiny2) and rt.num_rays == rt2.num_rays
    wave, rw = s.render(w, h, spp, variant=r1.VARIANT_WAVEFRONT)
    assert np.array_equal(base, wave) and rw.num_rays == r0.num_rays
    assert rw.launches > 5
    for world in (2, 3, 8):
        parts, rays = [], 0
        for rank in range(world):
            rgb, res = s.render(w, h, spp, rank=rank, world=world)
            parts.append(rgb)
            rays += res.num_rays
        assert np.array_equal(r1.assemble_rows(parts, h), base), world
        assert rays == r0.num_rays
    parts = [s.render(w, h, spp, rank=rank, world=3, row_tile=8)[0] for rank in range(3)]   # 8-row tiles give the same picture
    assert np.array_equal(r1.assemble_rows(parts, h, 8), base)
    other, _ = s.render(w, h, spp, seed=1)
    assert not np.array_equal(base, other)
    assert rmse(base, other) < 12


def test_edge_sizes_and_depth_cap(r1, scenes):
    s = scenes["medium"]
    rgb, res = s.render(1, 1, 1)
    assert rgb.shape == (1, 1, 3) and 1 <= res.num_rays <= 51
    rgb, res = s.render(33, 7, 3)                      # ragged: width not a warp multiple, height < row tile
    assert res.num_samples == 33 * 7 * 3 and rgb.any()
    rgb, res = s.render(16, 9, 5, max_bounces=0)       # cap 0: exactly one ray per sample, hits are black
    assert res.num_rays == 16 * 9 * 5
    rgb1, res1 = s.render(64, 36, 16, max_bounces=1)
    rgb50, res50 = s.render(64, 36, 16, max_bounces=50)
    assert res1.num_rays < res50.num_rays <= 64 * 36 * 16 * 51
    rgb, res = s.render(40, 10, 2, rank=7, world=8, row_tile=8)    # a rank that owns no rows
    assert rgb.shape[0] == 0 and res.num_rays == 0
    rgb, res = s.render(640, 360, 1)
    assert res.num_samples == 640 * 360


def test_outputs_stay_inside_the_callers_buffers(r1, scenes):
    """(compute-sanitizer is closed on this GPU pool.)  Host side: r1_render / benchmark() write exactly rows * width * 3 bytes --
    guard bytes on both sides of the caller's buffer stay untouched, for ragged sizes and for a rank's share.  Device side: the
    device-buffer entry point leaves a guard band behind d_rgb and around d_num_rays alone."""
    import ctypes as C
    import torch
    s = scenes["medium"]
    for (w, h, spp, rank, world) in ((33, 7, 3, 0, 1), (129, 65, 2, 1, 3), (640, 360, 1, 0, 1)):
        rows = r1.local_rows(h, r1.DEFAULT_ROW_TILE, rank, world)
        n = rows * w * 3
        raw = np.full(n + 512, 0xA5, np.uint8)
        p = r1.RenderParams(w, h, spp, 50, 0, 0, rank, world, r1.DEFAULT_ROW_TILE, 0, 0, -1)
        res = r1.Result()
        r1._check(r1.lib.r1_render(s.handle, C.byref(p), raw[256:256 + n], C.byref(res)), "r1_render")
        assert (raw[:256] == 0xA5).all() and (raw[256 + n:] == 0xA5).all() and res.num_samples == rows * w * spp
        ref, _ = s.render(w, h, spp, rank=rank, world=world)
        assert np.array_equal(raw[256:256 + n].reshape(rows, w, 3), ref)
    w, h, spp = 200, 117, 4
    guard = 4096
    d_rgb = torch.full((h * w * 3 + guard,), 0x5A, dtype=torch.uint8, device="cuda:0")
    d_rays = torch.full((3,), -1, dtype=torch.int64, device="cuda:0")
    s.render_device(d_rgb.data_ptr(), d_rays[1:].data_ptr(), torch.cuda.current_stream().cuda_stream, width=w, height=h, spp=spp, device=0)
    torch.cuda.synchronize()
    assert bool((d_rgb[h * w * 3:] == 0x5A).all()) and int(d_rays[0]) == -1 and int(d_rays[2]) == -1 and int(d_rays[1]) > w * h * spp
    ref, rr = s.render(w, h, spp)
    assert np.array_equal(d_rgb[: h * w * 3].cpu().numpy().reshape(h, w, 3), ref) and int(d_rays[1]) == rr.num_rays


# ---- the reference's surface ------------------------------------------------------------------------------------------------

def test_benchmark_surface(r1, tmp_path, monkeypatch, capfd):
    monkeypatch.chdir(tmp_path)
    r1.configure(width=160, height=90, spp=32, quiet=False)
    try:
        scene = r1.create_small_scene()
        pixels = np.zeros((90, 160, 3), np.uint8)
        res = r1.benchmark(scene, pixels, True, "small")
        with pytest.raises(r1.Rays1Error):
            scene.handle  # consumed (delete scene, rayweek1.cpp:905)
        out = capfd.readouterr().out.splitlines()
        assert out[0] == "small"
        assert out[1].startswith("elapsed time:   ") and out[1].endswith("s")
        assert out[2] == "total samples:  %d" % (160 * 90 * 32)
        assert out[3] == "total rays:     %d" % res.num_rays
        assert out[4].startswith("mrays/s:        ")
        assert out[5].startswith("threads:        1/")
        assert out[6].startswith("tile size:      ")
        assert abs(res.num_rays / (160 * 90 * 32) / 1.798 - 1) < 0.02
        raw = open(tmp_path / "out_small.tga", "rb").read()
        assert len(raw) == 18 + 160 * 90 * 3 and raw[2] == 2 and raw[16] == 24
        body = np.frombuffer(raw[18:], np.uint8).reshape(90, 160, 3)
        assert np.array_equal(body, pixels), "pixels were swapped to BGR in place, like the reference"
        fresh, _ = r1.create_small_scene().render(160, 90, 32)
        assert np.array_equal(body[:, :, ::-1], fresh)
    finally:
        r1.configure(width=1280, height=720, spp=250, quiet=True)


def test_drop_in_executable(r1, tmp_path):
    out = subprocess.run([r1.EXE_PATH, "-n", "2", "-w", "--spp", "4"], cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.splitlines()
    assert [l for l in lines if l in ("small", "medium", "large")] == ["small", "small", "medium", "medium", "large", "large"]
    assert sum(l == "total samples:  %d" % (1280 * 720 * 4) for l in lines) == 6
    for name in ("small", "medium", "large"):
        txt = open(tmp_path / ("out_%s.txt" % name)).read()
        tok = txt.split("|")
        assert tok[0] == "b200" and tok[1].endswith("s") and int(tok[2]) > 1280 * 720 * 4 and tok[3].endswith(" mrays/s") and tok[4] == ""
        assert os.path.getsize(tmp_path / ("out_%s.tga" % name)) == 18 + 1280 * 720 * 3


def test_bench_steps_tool_runs_the_executable(r1, tmp_path):
    """tools/bench_steps.py --quick --num 2 --save: the reference's driver flow (compile, run with -n / -w, collect out_<scene>.txt)"""
    import sys
    from conftest import ROOT
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_steps.py"), "--latest", "--quick", "--num", "2", "--save", "--outdir",
                          str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.count("total samples:  %d" % (80 * 60 * 100)) == 6          # 3 scenes x 2 runs at the QUICKBENCH size (common.h:3-16)
    for name in ("small", "medium", "large"):
        assert open(tmp_path / ("out_%s.txt" % name)).read().startswith("b200|")
        assert os.path.getsize(tmp_path / ("out_%s.tga" % name)) == 18 + 80 * 60 * 3


def test_in_process_multi_gpu_matches_single_gpu(r1, tmp_path):
    """--gpus 2 in ONE process (NCCL gather + reduce, rays1_host.cpp:render_multi) renders the same bytes and ray count."""
    if r1.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    outs = {}
    for g in (1, 2):
        d = tmp_path / ("g%d" % g)
        d.mkdir()
        out = subprocess.run([r1.EXE_PATH, "-w", "--gpus", str(g), "--scene", "large", "--spp", "16", "--width", "640", "--height", "360"],
                             cwd=d, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr
        rays = [l for l in out.stdout.splitlines() if l.startswith("total rays:")][0]
        outs[g] = (open(d / "out_large.tga", "rb").read(), rays)
    assert outs[1] == outs[2]


def test_scene_file_renders_like_builtin_scene(r1, tmp_path):
    """--scene-file (SURVEY 8f rank 3) through the executable: same bytes as the built-in large scene."""
    import sys
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_scene
    cam, sph = make_scene.grid_scene(30, 16, 0, (3, 8, 15), 10.0)
    path = str(tmp_path / "large.r1scene")
    r1.write_scene_file(path, cam, sph)
    common = ["-w", "--spp", "8", "--width", "320", "--height", "180"]
    a = subprocess.run([r1.EXE_PATH, "--scene-file", path] + common, cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert a.returncode == 0, a.stderr
    file_tga = open(tmp_path / "out_large.tga", "rb").read()
    file_txt = open(tmp_path / "out_large.txt").read()
    os.remove(tmp_path / "out_large.tga")
    b = subprocess.run([r1.EXE_PATH, "--scene", "large"] + common, cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert b.returncode == 0, b.stderr
    assert open(tmp_path / "out_large.tga", "rb").read() == file_tga
    assert file_txt.split("|")[2] == open(tmp_path / "out_large.txt").read().split("|")[2]   # same ray count


def test_unstaged_global_memory_scan_matches_staged(r1, scenes, monkeypatch):
    """scenes above 4096 spheres scan from global memory instead of shared memory (template flag kStaged); forced here on
    the large scene so that the two paths can be compared byte for byte"""
    s = scenes["large"]
    base, r0 = s.render(160, 90, 24)
    monkeypatch.setenv("R1_FORCE_UNSTAGED", "1")
    for v in (r1.VARIANT_MEGAKERNEL, r1.VARIANT_MEGAKERNEL_COOP, r1.VARIANT_MEGAKERNEL_SCALAR, r1.VARIANT_MEGAKERNEL_DEFERRED, r1.VARIANT_MEGAKERNEL_DUAL):
        alt, ra = s.render(160, 90, 24, variant=v)
        assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays, v


def test_scene_above_staging_limit(r1, tmp_path):
    """5044 spheres (> 4096): the megakernel renders from global memory; the staged-only entry points say so"""
    import sys
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_scene
    cam, sph = make_scene.grid_scene(72, 70, 480, (7, 18, 34), 22.0)
    path = str(tmp_path / "big.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path)
    assert s.count() == 5048
    rgb, res = s.render(96, 54, 16)
    assert rgb.any() and 96 * 54 * 16 < res.num_rays < 96 * 54 * 16 * 6
    again, _ = s.render(96, 54, 16, world=2, rank=0)
    assert np.array_equal(again, rgb[[r1.global_row(lr, r1.DEFAULT_ROW_TILE, 0, 2) for lr in range(again.shape[0])]])
    with pytest.raises(r1.Rays1Error, match="stages at most"):
        s.render(96, 54, 16, variant=r1.VARIANT_WAVEFRONT)
    with pytest.raises(r1.Rays1Error, match="stages at most"):
        s.trace_rays([[0, 5, 20]], [[0, 0, -1]])
    s.close()


def test_tensor_variant_with_a_ragged_last_chunk(r1, tmp_path):
    """676 spheres = 5 accumulator chunks of 128 + one of 64 (and 36 of 704 rows padding): the default variant resolves to the
    tensor kernel and renders the same bytes as the FFMA2 kernel, whole and as rank 1 of 3"""
    import sys
    from conftest import ROOT
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_scene
    cam, sph = make_scene.grid_scene(28, 24, 480, (9, 6, 16), 14.0)
    path = str(tmp_path / "mid.r1scene")
    r1.write_scene_file(path, cam, sph)
    s = r1.create_scene_from_file(path)
    assert s.count() == 680 and r1.lib.r1_kernel_name(s.handle, r1.VARIANT_MEGAKERNEL).decode() == "megakernel_tc3"
    base, r0 = s.render(120, 68, 12, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    alt, ra = s.render(120, 68, 12)
    assert np.array_equal(base, alt) and ra.num_rays == r0.num_rays and base.any()
    part, _ = s.render(120, 68, 12, rank=1, world=3)
    assert np.array_equal(part, base[[r1.global_row(lr, r1.DEFAULT_ROW_TILE, 1, 3) for lr in range(part.shape[0])]])
    s.close()


@pytest.mark.parametrize("name", ALL)
def test_per_pixel_replay_matches_reference_color(r1, scenes, golden_rays, name):
    """SURVEY 8f rank 4: the GPU integrator (production scan / exact test / scatter / sky, the reference's generators replayed
    from recorded states) against the colour the reference's own color() returned for the same 4096 samples per scene.
    Path-level parity: RNG consumption order, depth logic, attenuation order, ray counting.  The result is BIT-IDENTICAL: every
    ray count and every float colour, on all four scenes."""
    from conftest import GOLDEN
    g = dict(np.load(os.path.join(GOLDEN, "replay_%s.npz" % name)))
    col, rays = scenes[name].replay_pixels(g["xy"], 1280, 720, 1, g["state"], g["state4"])
    record("replay_4096_samples/%s" % name, {"same_ray_count": float((rays == g["rays"]).mean()),
                                             "colour_bit_identical": float((bits(col) == bits(g["color"])).all(axis=1).mean())})
    assert np.array_equal(rays, g["rays"])
    assert np.array_equal(bits(col), bits(g["color"]))
    # depth cap honoured: with max_bounces = 3 no sample traces more than 4 rays
    col3, rays3 = scenes[name].replay_pixels(g["xy"][:512], 1280, 720, 1, g["state"][:512], g["state4"][:512], max_bounces=3)
    assert rays3.max() <= 4
