"""What the renderer converges to, and renders at the 2^20-spp limit.

1. r1_render_sums of one sphere under the sky against the float64 expectation of tests/estimator_reference.py, at 2^16 to 2^20
   spp on 20x12 frames: per channel an aggregate |z| <= 5 and a per-pixel chi^2 below its 1e-6 quantile, exact ray counts where
   they are deterministic and the dielectric's within |z| <= 5.  This is the one test of the random part of a render -- the
   generator, the direct samplers (disk radius sqrt(u), ball radius u^(1/3) through lg2 / ex2, z = 1 - rand02, azimuth
   rand02 pi) and which draws feed which sampler -- that does not restate those formulas.  Renders are pure functions of their
   inputs, so each outcome is fixed.
2. At spp = 2^20 (4096 samples per unit, 256 units per pixel, sums near 2^52) whole renders are compared bit for bit with
   orc_render_keyed fed r1_sample_points, for every variant and knob of test_render_oracle_gpu."""
import pytest

import estimator_reference as er
from test_gpu_parity import scenes  # noqa: F401  (module fixture: the four built-in scenes)
from test_render_oracle_gpu import RUNS, check, expected, global_rows, sample_keys  # noqa: F401  (expected: module fixture)
from test_scan_edges_gpu import RawScene, _f

pytestmark = pytest.mark.gpu

W, H = 20, 12
# case -> samples per pixel (2^16 .. 2^20)
SPP = {"sky_pinhole": 1 << 16, "sky_lens": 1 << 18, "lambert": 1 << 20, "mirror": 1 << 17, "fuzz": 1 << 18, "glass": 1 << 17,
       "ior24": 1 << 17, "ior24_mb1": 1 << 16, "ior24_mb2": 1 << 16, "ior24_mb3": 1 << 16}
LAMBERT_VARIANTS = ("packed", "tensor_stream", "bvh", "wavefront")


class Cases:
    """the committed scenes of estimator_reference.CASES and their models, made on first use"""

    def __init__(self):
        self.scenes, self.models = {}, {}

    def get(self, name):
        if name not in self.scenes:
            cam, spec, mb = er.CASES[name]
            s = RawScene(_f(*cam), [_f(*c[:4]) + (c[4],) + _f(*c[5:]) for c in spec])
            self.scenes[name] = s
            self.models[name] = er.expectation(s.camera(), s.soa(), W, H, mb)
        return self.scenes[name], self.models[name]

    def close(self):
        for s in self.scenes.values():
            s.close()


@pytest.fixture(scope="module")
def cases(r1):
    c = Cases()
    yield c
    c.close()


def converges(r1, cases, name, spp, variant=0):
    s, model = cases.get(name)
    _, sums, res = s.render_sums(W, H, spp, er.CASES[name][2], variant)
    what = "%s %dx%dx%d variant %d" % (name, W, H, spp, variant)
    st = er.converge_stats(model, sums, res.num_rays, spp, what, deterministic_rays=er.CASES[name][1][0][4] != er.MAT_DIELECTRIC)
    print("gpu %-12s spp 2^%d variant %2d %s" % (name, spp.bit_length() - 1, variant, st))


@pytest.mark.parametrize("name", sorted(er.CASES))
def test_render_converges_to_the_expectation(r1, cases, name):
    converges(r1, cases, name, SPP[name])


@pytest.mark.parametrize("variant", LAMBERT_VARIANTS)
def test_lambertian_converges_in_every_scan(r1, cases, variant):
    converges(r1, cases, "lambert", 1 << 17, r1.VARIANTS[variant])


# ---- bit for bit at the accumulator limit -------------------------------------------------------------------------------------

LIMIT = 1 << 20
LIMIT_RENDERS = ((2, 1, 1, 0, 1), (2, 1, 2, 0, 1), (2, 3, 2, 1, 3))     # w, h, max_bounces, rank, world


@pytest.fixture(scope="module")
def limit_scene(r1, expected, scenes):  # noqa: F811
    """the medium scene, with the oracle's renders at 2^20 spp put into `expected`'s cache: computed here in one piece, since at
    (2 + 4 max_bounces) 4 B per sample the points of one row pass the budget by which Expected splits whole images"""
    s = scenes["medium"]
    so = expected.scene(s)
    for w, h, mb, rank, world in LIMIT_RENDERS:
        ys = global_rows(expected.oracle, h, rank, world, 1)
        pts = r1.sample_points(*sample_keys(ys, w, LIMIT), 0, mb)
        assert pts.shape == (len(ys) * w * LIMIT, 2 + 4 * mb)
        expected.renders[(s.handle, w, h, LIMIT, mb, 0, rank, world, 1)] = expected.oracle.render_keyed(so, w, h, LIMIT, mb, 0, rank, world, 1, pts)
        del pts
    return s


@pytest.mark.parametrize("run", sorted(RUNS))
def test_renders_at_2_to_the_20_samples_per_pixel(r1, expected, limit_scene, monkeypatch, run):
    v, threads, bps, env = RUNS[run]
    for w, h, mb, rank, world in LIMIT_RENDERS:
        _, sums, _ = check(r1, expected, monkeypatch, limit_scene, w, h, LIMIT, mb=mb, rank=rank, world=world, variant=v, threads=threads,
                           blocks_per_sm=bps, env=env, what="medium at 2^20 spp %s" % run)
        assert sums.max() > 1 << 40, "the sums reach the range where 2^20 samples of 2^-24 units live"
