"""The tensor-core path (R1_VARIANT_MEGAKERNEL_TENSOR, r1::megakernel_tc3) at every scene size it accepts.

tc3 scans the scene's sphere operand in accumulator chunks of 128 spheres; the last chunk holds n32 - 128 (chunks - 1) columns
and is read in that many / 32 pieces.  The scenes below come from tools/make_scene.grid_scene, whose ground sphere and three big
spheres come last -- in the last chunk, where a mishandled ragged chunk would lose hits:

    grid   spheres  n32  chunks  last chunk
    16x15    248    256    2       128      below the default variant's 256-sphere threshold (n8 = 248)
    18x14    256    256    2       128      the threshold itself
    17x16    280    288    3        32      one piece after full chunks
    21x16    344    352    3        96      three pieces (the odd count of the two-loads-in-flight read)
    22x21    472    480    4        96
    24x22    536    544    5        32      7 ray groups barely fit shared memory (2 544 bytes left)
    28x24    680    704    6        64      6 ray groups barely fit (496 bytes left)
    28x27    760    768    6       128      the largest operand (96 KB)
    31x25    784    800    -        -       refused: the operand holds at most 768 spheres

Per scene: which kernel the default variant picks; hits of fresh, grazing and far rays through the tensor filter against the
oracle, bit for bit; the filter's values against the float64 polynomial; renders byte-identical to the packed FFMA2 kernel for
every ray-group count tc3 takes."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_gpu_parity import bits, record, tensor_filter_far_rays, tensor_filter_truth

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_scene  # noqa: E402

# (grid w, grid h): (spheres after the loader's padding to 8, n32)
GRIDS = {(16, 15): (248, 256), (18, 14): (256, 256), (17, 16): (280, 288), (21, 16): (344, 352), (22, 21): (472, 480),
         (24, 22): (536, 544), (28, 24): (680, 704), (28, 27): (760, 768), (31, 25): (784, 800)}
TENSOR = [g for g, (_, n32) in GRIDS.items() if n32 <= 768]
IDS = ["%dx%d" % g for g in GRIDS]
SMEM_LIMIT = 227 * 1024


def tc3_smem_bytes(groups, n32):
    """r1::tc3_smem_bytes, which launch_megakernel_tc3_t checks: the rsqrt table, control, B tile and exact spheres (144 bytes
    per sphere), and per ray group the A tile (16 KB) and four warp pools (4 x 1152 bytes)"""
    return (16 + 2048 * 2) + 256 + n32 * (128 + 16) + groups * (128 * 128 + 4 * 1152) + 256


def grid_scene(r1, directory, gw, gh, commit=True):
    """the grid scene of `tools/make_scene.py --grid gw gh` (the camera frames the grid), through a scene file"""
    scale = max(gw / 30.0, gh / 16.0)
    cam, sph = make_scene.grid_scene(gw, gh, 480, (3 * scale, 8 * scale, 15 * scale), 10.0 * scale)
    path = os.path.join(str(directory), "%dx%d.r1scene" % (gw, gh))
    r1.write_scene_file(path, cam, sph)
    return r1.create_scene_from_file(path, commit=commit)


@pytest.fixture(scope="module")
def sweep(r1, tmp_path_factory):
    d = tmp_path_factory.mktemp("sweep")
    out = {g: grid_scene(r1, d, *g) for g in GRIDS}
    yield out
    for s in out.values():
        s.close()


def n32_of(r1, scene):
    n32 = C.c_uint32(0)
    r1.lib.r1_tensor_operand(scene.handle, np.zeros(16, np.uint8), 16, C.byref(n32))   # sets n32 whatever the outcome
    return n32.value


@pytest.mark.parametrize("grid", list(GRIDS), ids=IDS)
def test_default_variant_by_sphere_count(r1, sweep, grid):
    s = sweep[grid]
    count, n32 = GRIDS[grid]
    assert s.count() == count and n32_of(r1, s) == n32
    want = "megakernel_tc3" if count >= 256 and n32 <= 768 else "megakernel_pool"
    assert r1.lib.r1_kernel_name(s.handle, r1.VARIANT_MEGAKERNEL).decode() == want


def sweep_rays(soa, gw, gh, n=4000, seed=2024):
    """rays from around the grid in every direction (half of them reach the ground sphere, the last real sphere), rays among the
    small spheres, and rays grazing random spheres from 5 .. 20 000 units away"""
    rng = np.random.default_rng(seed)
    org = rng.normal(size=(n, 3)) * [0.4 * gw, 2, 0.4 * gh] + [0, 2, 0]
    org[: n // 4] = rng.normal(size=(n // 4, 3)) * [0.4 * gw, 0.02, 0.4 * gh] + [0, 0.5, 0]
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    real = np.where(soa["inv_radius"] > 0)[0]
    idx = rng.choice(real, n)
    ctr = np.stack([soa["cx"][idx], soa["cy"][idx], soa["cz"][idx]], 1).astype(np.float64)
    rad = 1.0 / soa["inv_radius"][idx].astype(np.float64)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    u[:, 1] = np.abs(u[:, 1])
    o2 = ctr + u * rng.choice([5.0, 50.0, 300.0, 2000.0, 20000.0], n)[:, None]
    side = np.cross(u, rng.normal(size=(n, 3))); side /= np.linalg.norm(side, axis=1, keepdims=True)
    d2 = ctr + side * (rad * rng.uniform(0.98, 1.02, n))[:, None] - o2
    d2 /= np.linalg.norm(d2, axis=1, keepdims=True)
    return np.concatenate([org, o2]).astype(np.float32), np.concatenate([d, d2]).astype(np.float32)


@pytest.mark.parametrize("grid", TENSOR, ids=["%dx%d" % g for g in TENSOR])
def test_tensor_hits_match_oracle(r1, sweep, oracle, grid):
    """trace_rays through tc3's filter (its chunks, its ragged last chunk) and the exact test: the oracle's hit record bit for bit,
    whole range and a t window; a few hundred of the hits are spheres of the last chunk"""
    s = sweep[grid]
    soa = s.soa()
    n32 = n32_of(r1, s)
    last = 128 * ((n32 - 1) // 128)                              # first sphere of the last chunk
    org, d = sweep_rays(soa, *grid)
    so = oracle.scene_create_from_soa(soa)
    try:
        for t_min, t_max in ((0.001, float(np.finfo(np.float32).max)), (0.5, 6.0)):
            want = oracle.hit(so, org, d, t_min, t_max)
            got = s.trace_rays(org, d, t_min, t_max, variant=r1.VARIANT_MEGAKERNEL_TENSOR)
            assert np.array_equal(got[0], want[0]), "%d rays lost or gained a hit" % int((got[0] != want[0]).sum())
            m = want[0] >= 0
            assert m.sum() > 1000
            for a, b in zip(got[1:], want[1:]):
                assert np.array_equal(bits(a[m]), bits(b[m]))
            assert (got[1][~m] == 0).all()
        full = oracle.hit(so, org, d)[0]
    finally:
        oracle.scene_destroy(so)
    assert (full >= last).sum() >= 300, "too few hits in the last chunk to exercise it"
    assert (full[full >= 0] < last).sum() >= 300


@pytest.mark.parametrize("grid", TENSOR, ids=["%dx%d" % g for g in TENSOR])
def test_tensor_filter_is_conservative_on_the_sweep(r1, sweep, grid):
    """r1_filter_probe on the sweep scenes with rays grazing spheres from up to 20 000 units: values within a tenth of the
    margin of the float64 polynomial, every sphere the exact test could accept flagged, padding rows never"""
    s = sweep[grid]
    soa = s.soa()
    n_sph = len(soa["cx"])
    n = 1024
    org, d = tensor_filter_far_rays(soa, n=n)
    e = s.filter_probe(org, d, n_sph).astype(np.float64)
    assert e.shape[1] == GRIDS[grid][1]
    want, discr, big_s = tensor_filter_truth(soa, org, d)
    real = soa["inv_radius"] > 0
    err = np.abs(e[:, :n_sph] - want)[:, real] / big_s[:, real]
    far = err[2 * n:]                                            # the rays from 2 000 and 20 000 units
    record("tensor_filter_rel_err_sweep_n32_%d" % GRIDS[grid][1], {"max": float(err.max()), "far_max": float(far.max()),
                                                                     "p99.9": float(np.quantile(err, 0.999)), "margin": 2.0 ** -16})
    assert err.max() < 0.1 * 2.0 ** -16, "tensor filter error %.3g of S eats the margin" % err.max()
    must = (discr >= -4.0e-6 * big_s) & real[None, :]
    assert must[2 * n:].sum() > 1000
    assert (e[:, :n_sph][must] >= 0).all() and not np.signbit(e[:, :n_sph][must]).any()
    assert (e[:, n_sph:] < 0).all() and (e[:, :n_sph][:, ~real] < 0).all(), "padding rows must never be flagged"


def fits(groups, n32):
    return tc3_smem_bytes(groups, n32) <= SMEM_LIMIT


@pytest.mark.parametrize("grid", TENSOR, ids=["%dx%d" % g for g in TENSOR])
def test_tensor_group_counts_render_like_packed(r1, sweep, grid):
    """variant TENSOR (tc3) against PACKED, byte for byte and ray for ray, with 4 .. 7 ray groups per CTA (threads = 128 x groups),
    on a frame, on a 7x3 image (fewer samples than one group has lanes) and as rank 1 of 3.  A group count whose shared memory
    does not fit the scene is refused with R1_ERR_LIMIT -- exactly those -- and leaves nothing behind: the next render works."""
    s = sweep[grid]
    n32 = GRIDS[grid][1]
    cases = ((96, 54, 8, 0, 1), (7, 3, 5, 0, 1), (96, 54, 8, 1, 3))
    base = {c: s.render(c[0], c[1], c[2], rank=c[3], world=c[4], variant=r1.VARIANT_MEGAKERNEL_PACKED) for c in cases}
    assert base[cases[0]][0].any()
    for groups in (None, 4, 6, 7):
        threads = 128 * groups if groups else 0
        g = groups or 5
        for c in cases:
            if not fits(g, n32):
                with pytest.raises(r1.Rays1Error, match=r"\(-4\).*shared memory"):
                    s.render(c[0], c[1], c[2], rank=c[3], world=c[4], variant=r1.VARIANT_MEGAKERNEL_TENSOR, threads=threads)
                continue
            rgb, res = s.render(c[0], c[1], c[2], rank=c[3], world=c[4], variant=r1.VARIANT_MEGAKERNEL_TENSOR, threads=threads)
            assert np.array_equal(rgb, base[c][0]) and res.num_rays == base[c][1].num_rays, (grid, groups, c)
    rgb, res = s.render(96, 54, 8, variant=r1.VARIANT_MEGAKERNEL_TENSOR)   # after any refusal: no sticky error
    assert np.array_equal(rgb, base[cases[0]][0]) and res.num_rays == base[cases[0]][1].num_rays
    whole = base[cases[0]][0]
    part = base[cases[2]][0]
    assert np.array_equal(part, whole[[r1.global_row(lr, r1.DEFAULT_ROW_TILE, 1, 3) for lr in range(part.shape[0])]])


def test_above_768_spheres_tensor_is_refused_and_default_is_packed(r1, sweep):
    s = sweep[(31, 25)]
    with pytest.raises(r1.Rays1Error, match="768"):
        s.render(96, 54, 8, variant=r1.VARIANT_MEGAKERNEL_TENSOR)
    with pytest.raises(r1.Rays1Error, match=r"\(-4\).*768"):
        s.trace_rays([[0, 3, 20]], [[0, 0, -1]], variant=r1.VARIANT_MEGAKERNEL_TENSOR)
    base, r0 = s.render(96, 54, 8, variant=r1.VARIANT_MEGAKERNEL_PACKED)
    rgb, res = s.render(96, 54, 8)
    assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays and base.any()


def test_tensor_has_one_render_kernel_whatever_the_environment(r1, monkeypatch):
    """R1_TC1, R1_TC2, R1_TC_FLAGS and R1_TC3 are not tuning knobs of this library: with them set, TENSOR still names
    megakernel_tc3, and a render of the large scene is the same bytes and rays as without them."""
    s = r1.create_large_scene()
    try:
        base, r0 = s.render(7, 3, 5, variant=r1.VARIANT_MEGAKERNEL_TENSOR)
        for key, value in (("R1_TC1", "1"), ("R1_TC2", "4"), ("R1_TC_FLAGS", "2"), ("R1_TC3", "4")):
            monkeypatch.setenv(key, value)
        assert r1.lib.r1_kernel_name(s.handle, r1.VARIANT_MEGAKERNEL_TENSOR).decode() == "megakernel_tc3"
        rgb, res = s.render(7, 3, 5, variant=r1.VARIANT_MEGAKERNEL_TENSOR)
        assert np.array_equal(rgb, base) and res.num_rays == r0.num_rays
    finally:
        s.close()
