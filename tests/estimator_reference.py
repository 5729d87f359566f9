"""What a render converges to, in float64: per pixel E[radiance], E[radiance^2] and E[rays per sample] for scenes of ONE sphere
under the sky, integrated by tensor Gauss-Legendre quadrature.  tests/test_estimator_cpu.py compares it with the oracle's libm mode
and tests/test_estimator_gpu.py with r1_render_sums; both test the random part of a render -- the generator, the direct samplers
and which draws feed which sampler -- which the bit-for-bit tests inject and so never see.

The model reads the scene's own float32 camera constants (Scene.camera(), 22 values) and its SoA.  A sample's primary ray is
jittered uniformly over its pixel and leaves a uniform point of the lens disk (radius lens_radius).  The sky is c0 + c1 d_y per
channel (c0 = (1 + b) / 2, c1 = (b - 1) / 2, b = (0.5, 0.7, 1.0)).  The pixel is integrated with Gauss nodes in s and t, the lens
in polar form with Gauss nodes in the radius (density 2 rho) and the periodic trapezoid rule in the angle.  The sampling of the
scatter is integrated in closed form (Lambertian) or by a 2-D quadrature computed once (metal fuzz); a dielectric path is a
geometric chain, below.

Only pixels that lie wholly inside or wholly outside the silhouette (with a margin, see `classify`) have a smooth integrand; the
others get NaN and are not tested.

What the model ignores, each far below the resolution of the tests (a pixel mean to about 1e-4, an aggregate to about 1e-5):
  * the renderer's directions are normalised with a 12-bit table and one Newton step, a relative error <= 1.6e-7;
  * float32 hit points and normals (relative 1e-7), and the float32 camera arithmetic;
  * the SFU approximations of the samplers (sqrt, lg2 / ex2, sin / cos: about 1e-6 in where a point falls);
  * the 24-bit uniforms (a law on a grid of 2^-24 instead of the continuum) and the float rounding of the Fresnel probability;
  * the quantiser: each sample is rounded to 2^-24, an error <= 2^-25 per sample;
  * Lambertian scatters that graze a surface whose float hit point lies just inside it and hit it again (t > 0.001 needs
    cos < ~1e-4, probability ~1e-8 per sample); they change the radiance by < 1 for < 1e-8 of the samples."""
import numpy as np

SKY_B = np.array([0.5, 0.7, 1.0])
C0, C1 = (1 + SKY_B) / 2, (SKY_B - 1) / 2
KAPPA_LAMBERT = 0.8                      # E[unit(n + u)] = KAPPA n, u uniform in the unit ball
COS2_LAMBERT = 2.0 / 3.0                 # E[(unit(n + u) . n)^2]
FIXED = 2.0 ** -24                       # one unit of the renderer's fixed-point sums
MARGIN = 2e-3                            # relative clearance of a tested pixel from the silhouette
MAT_NONE, MAT_LAMBERT, MAT_METAL, MAT_DIELECTRIC = -1, 0, 1, 2

# ---- the scenes: (camera (from xyz, at xyz, vfov, aperture, focus) with vup (0, 1, 0) and aspect 16:9, spheres, max_bounces) ----
PLACEHOLDER = (999999999.0, 999999999.0, 999999999.0, 0.0, MAT_NONE, 0.0, 0.0, 0.0, 0.0)
# a unit sphere at the origin seen from 2.8 units above and in front of it: it covers the whole view (corner rays 16 degrees off
# axis, the silhouette at 20.9), so every pixel is inside and a frame's ray count is known; the visible normals reach n_y 0.2 .. 0.95
NEAR = (0.0, 1.6, 2.3, 0.0, 0.0, 0.0, 16.0, 0.1, 2.8)
CASES = {
    "sky_pinhole": ((0.0, 0.0, 0.0, 0.0, 0.8, -1.0, 90.0, 0.0, 1.0), [PLACEHOLDER], 50),        # tilted up: d_y from -0.1 to 0.95
    "sky_lens": ((0.0, 0.0, 0.0, 0.0, -0.7, -1.0, 70.0, 3.0, 1.5), [PLACEHOLDER], 50),          # lens radius 1.5 = focus distance
    "lambert": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_LAMBERT, 0.7, 0.5, 0.3, 0.0)], 50),
    "mirror": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_METAL, 0.9, 0.8, 0.7, 0.0)], 50),
    "fuzz": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_METAL, 0.9, 0.8, 0.7, 0.3)], 50),                 # r.n >= 0.6 > 0.3 on every pixel
    "glass": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_DIELECTRIC, 1.0, 1.0, 1.0, 1.5)], 50),
    "ior24": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_DIELECTRIC, 1.0, 1.0, 1.0, 24.2)], 50),
    "ior24_mb1": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_DIELECTRIC, 1.0, 1.0, 1.0, 24.2)], 1),
    "ior24_mb2": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_DIELECTRIC, 1.0, 1.0, 1.0, 24.2)], 2),
    "ior24_mb3": (NEAR, [(0.0, 0.0, 0.0, 1.0, MAT_DIELECTRIC, 1.0, 1.0, 1.0, 24.2)], 3),
}


def gauss01(n):
    x, w = np.polynomial.legendre.leggauss(n)
    return (x + 1) / 2, w / 2


def _dot(a, b):
    return (a * b).sum(axis=-1)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


class Camera:
    """the 22 float32 constants of r1_scene_get_camera, in float64: origin, llc, horizontal, vertical, u, v, w, lens_radius"""

    def __init__(self, cam22):
        c = np.asarray(cam22, np.float32).astype(np.float64)
        self.origin, self.llc, self.hor, self.ver, self.u, self.v = (c[3 * k: 3 * k + 3] for k in range(6))
        self.lens = c[21]

    def rays(self, s, t, dx, dy):
        """s, t (...), lens point dx, dy (...) -> origins and unit directions (..., 3)"""
        off = self.lens * (self.u * dx[..., None] + self.v * dy[..., None])
        d = self.llc + s[..., None] * self.hor + t[..., None] * self.ver - self.origin - off
        return self.origin + off, _unit(d)


def lens_nodes(lens, n_rad, n_ang, law="sqrt"):
    """points and weights of the unit disk for E over a uniform lens point; law "uniform" (radius u instead of sqrt(u)) is the
    density 1 over rho in [0, 1) and serves to predict what a wrong disk sampler would do"""
    if lens == 0:
        return np.zeros(1), np.zeros(1), np.ones(1)
    r, wr = gauss01(n_rad)
    wr = wr * (2 * r if law == "sqrt" else 1.0)
    a = 2 * np.pi * (np.arange(n_ang) + 0.5) / n_ang
    R, A = np.meshgrid(r, a, indexing="ij")
    W = np.repeat(wr[:, None], n_ang, axis=1) / n_ang
    return (R * np.cos(A)).ravel(), (R * np.sin(A)).ravel(), W.ravel()


def primary_rays(cam, w, h, n_pix=6, n_rad=6, n_ang=12, law="sqrt"):
    """per pixel (row y = 0 at the bottom, as the renderer's rows) the quadrature rays: org, dir [h, w, Q, 3], weights [Q].
    law "jitter" takes the lens point from the jitter's own uniforms (radius sqrt(u0), angle 2 pi u1), to predict what a
    sampler reading the lens disk from draws 0 and 1 would do"""
    X, Y = np.meshgrid(np.arange(w), np.arange(h))
    if law == "jitter":
        j, wj = gauss01(4 * n_pix)
        js, jt = (a.ravel() for a in np.meshgrid(np.arange(len(j)), np.arange(len(j)), indexing="ij"))
        s, t = (X[..., None] + j[js]) / w, (Y[..., None] + j[jt]) / h
        dx, dy = np.sqrt(j[js]) * np.cos(2 * np.pi * j[jt]), np.sqrt(j[js]) * np.sin(2 * np.pi * j[jt])
        o, d = cam.rays(s, t, np.broadcast_to(dx, s.shape), np.broadcast_to(dy, s.shape))
        return o, d, wj[js] * wj[jt]
    j, wj = gauss01(n_pix)
    dx, dy, wl = lens_nodes(cam.lens, n_rad, n_ang, law)
    js, jt, jl = np.meshgrid(np.arange(n_pix), np.arange(n_pix), np.arange(len(wl)), indexing="ij")
    js, jt, jl = js.ravel(), jt.ravel(), jl.ravel()
    weight = wj[js] * wj[jt] * wl[jl]
    s = (X[..., None] + j[js]) / w
    t = (Y[..., None] + j[jt]) / h
    o, d = cam.rays(s, t, np.broadcast_to(dx[jl], s.shape), np.broadcast_to(dy[jl], s.shape))
    return o, d, weight


def _impact(o, d, c, r):
    """distance of the sphere's centre from each ray's line over the radius, and the ray parameter of the closest approach"""
    oc = c - o
    tc = _dot(oc, d)
    q = np.linalg.norm(oc - tc[..., None] * d, axis=-1) / r
    return q, tc


def classify(cam, w, h, c, r):
    """-> inside, outside [h, w]: the pixel's every ray (any jitter, any lens point) hits the sphere / misses it.  Decided on a
    grid of 9 x 9 jitter points (edges included) and, with a lens, radii 0, 1/4 .. 1 at 32 angles.  q (impact over radius) is
    nearly linear across a pixel, so between grid points an eighth of the range apart it cannot leave the sampled range by a
    quarter of that range: a pixel counts as inside when max q + (max q - min q) / 4 < 1 - MARGIN, outside when
    min q - (max q - min q) / 4 > 1 + MARGIN"""
    g = np.linspace(0, 1, 9)
    if cam.lens > 0:
        rr, aa = np.meshgrid(np.linspace(0, 1, 5), 2 * np.pi * np.arange(32) / 32, indexing="ij")
        lx, ly = (rr * np.cos(aa)).ravel(), (rr * np.sin(aa)).ravel()
    else:
        lx = ly = np.zeros(1)
    gs, gt, gl = (a.ravel() for a in np.meshgrid(g, g, np.arange(len(lx)), indexing="ij"))
    X, Y = np.meshgrid(np.arange(w), np.arange(h))
    o, d = cam.rays((X[..., None] + gs) / w, (Y[..., None] + gt) / h, np.broadcast_to(lx[gl], X.shape + gs.shape),
                    np.broadcast_to(ly[gl], X.shape + gs.shape))
    q, tc = _impact(o, d, np.asarray(c, np.float64), r)
    spread = (q.max(axis=-1) - q.min(axis=-1)) / 4
    ahead = (tc > r).all(axis=-1)
    inside = ahead & (q.max(axis=-1) + spread < 1 - MARGIN)
    outside = (q.min(axis=-1) - spread > 1 + MARGIN) | (tc < -r).all(axis=-1)
    return inside, outside


def sky(d):
    """radiance of the sky seen along unit directions d [..., 3] -> [..., 3]"""
    return C0 + C1 * d[..., 1:2]


def sky_moments(d):
    L = sky(d)
    return L, L * L


def fuzz_moments(f, n=96):
    """kappa(f) = E[(r + f u) . r / |r + f u|] and lambda(f) = E[((r + f u) . r)^2 / |r + f u|^2] for a unit r and u uniform in the
    unit ball (density 3 rho^2 in the radius, cos uniform in [-1, 1]); 2-D Gauss-Legendre, smooth for f < 1"""
    rho, wr = gauss01(n)
    c, wc = gauss01(n)
    c = 2 * c - 1
    R, Cc = np.meshgrid(rho, c, indexing="ij")
    W = np.outer(wr * 3 * rho ** 2, wc)
    a = 1 + f * R * Cc
    n2 = 1 + 2 * f * R * Cc + (f * R) ** 2
    return float((W * a / np.sqrt(n2)).sum()), float((W * a * a / n2).sum())


def _hit_outside(o, d, c, r):
    oc = o - c
    b = _dot(oc, d)
    disc = b * b - (_dot(oc, oc) - r * r)
    if (disc <= 0).any():
        raise ValueError("a quadrature ray of a pixel classed inside misses the sphere")
    t = -b - np.sqrt(disc)
    p = o + t[..., None] * d
    return p, (p - c) / r


def _exit_point(o, d, c, r):
    oc = o - c
    b = _dot(oc, d)
    t = -b + np.sqrt(np.maximum(b * b - (_dot(oc, oc) - r * r), 0))
    p = o + t[..., None] * d
    return p, (p - c) / r


def _reflect(d, n):
    return d - 2 * _dot(d, n)[..., None] * n


def _fresnel(d, n, ior):
    """Dielectric::scatter's math (rayweek1.cpp:470-511) at a hit with outward normal n: -> (probability of reflection, the
    refracted unit direction).  From outside: ni_over_nt = 1 / ior, cosine = -d.n; from inside: the normal flipped, ni_over_nt
    = ior, cosine = ior d.n.  Refraction iff the discriminant 1 - k^2 (1 - dt^2) > 0; then Schlick with r0s = (1 - ior) /
    (1 + ior), r0 = r0s^2, prob = r0 + (1 - r0) (1 - cosine)^5; else prob = 1.  A path reflects when ru < prob, ru uniform in
    [0, 1): the probability is prob clipped to [0, 1]."""
    dn = _dot(d, n)
    out = dn > 0
    n1 = np.where(out[..., None], -n, n)
    k = np.where(out, ior, 1.0 / ior)
    cosine = np.where(out, ior * dn, -dn)
    dt = _dot(d, n1)
    disc = 1 - k * k * (1 - dt * dt)
    ok = disc > 0
    refr = k[..., None] * (d - dt[..., None] * n1) - n1 * np.sqrt(np.maximum(disc, 0))[..., None]
    r0s = (1 - ior) / (1 + ior)
    x = 1 - cosine
    prob = np.where(ok, r0s * r0s + (1 - r0s * r0s) * x ** 5, 1.0)
    return np.clip(prob, 0, 1), _unit(refr)


def _surface_moments(kind, albedo, param, mb, d, p, n, c, r):
    """per quadrature ray that hits the sphere at p (outward normal n): E[L], E[L^2] [..., 3], E[rays], E[rays^2]"""
    a = np.asarray(albedo, np.float64)
    one = np.ones(d.shape[:-1])
    if mb == 0:
        return np.zeros(d.shape), np.zeros(d.shape), one, one
    if kind == MAT_LAMBERT:
        ny = n[..., 1:2]
        wy2 = COS2_LAMBERT * ny * ny + (1 - COS2_LAMBERT) / 2 * (1 - ny * ny)
        m1 = a * (C0 + C1 * KAPPA_LAMBERT * ny)
        m2 = a * a * (C0 * C0 + 2 * C0 * C1 * KAPPA_LAMBERT * ny + C1 * C1 * wy2)
        return m1, m2, 2 * one, 4 * one
    if kind == MAT_METAL:
        rf = _reflect(d, n)
        if (_dot(rf, n) <= param * (1 + 1e-6)).any():
            raise ValueError("metal of fuzz %g: a reflection leaves at r.n <= fuzz, its scatter can fail" % param)
        kap, lam = fuzz_moments(param) if param > 0 else (1.0, 1.0)
        ry = rf[..., 1:2]
        wy2 = lam * ry * ry + (1 - lam) / 2 * (1 - ry * ry)
        m1 = a * (C0 + C1 * kap * ry)
        m2 = a * a * (C0 * C0 + 2 * C0 * C1 * kap * ry + C1 * C1 * wy2)
        return m1, m2, 2 * one, 4 * one
    if kind == MAT_DIELECTRIC:
        ior = float(param)
        R1, refr = _fresnel(d, n, ior)
        L1, L2 = sky_moments(_reflect(d, n))
        m1, m2 = R1[..., None] * L1, R1[..., None] * L2
        n1, n2 = 2 * R1, 4 * R1
        # the chain inside: the j-th internal hit (depth j) scatters while j < mb; every internal hit of a sphere has the
        # same angle, but the directions are followed hit by hit all the same
        live = 1 - R1
        q, dq = p, refr
        for j in range(1, mb):
            q, nn = _exit_point(q, dq, c, r)
            Ri, out = _fresnel(dq, nn, ior)
            L1, L2 = sky_moments(out)
            leave = live * (1 - Ri)
            m1, m2 = m1 + leave[..., None] * L1, m2 + leave[..., None] * L2
            n1, n2 = n1 + leave * (2 + j), n2 + leave * (2 + j) ** 2
            live = live * Ri
            dq = _unit(_reflect(dq, nn))
            if live.max() < 1e-17:        # what is left can change no mean by more than 1e-15
                break
        n1, n2 = n1 + live * (mb + 1), n2 + live * (mb + 1) ** 2     # black at the cap after mb + 1 rays
        return m1, m2, n1, n2
    raise ValueError("material %r" % kind)


def expectation(cam22, soa, w, h, max_bounces, n_pix=6, n_rad=6, n_ang=12, law="sqrt"):
    """-> dict of per-pixel arrays [h, w(, 3)]: mean, second (E[L^2]), rays, rays2 (E[rays^2]) per sample, inside, outside.
    Pixels that are neither wholly inside nor wholly outside the silhouette are NaN.  soa: one sphere (a real sphere, or the
    MAT_NONE placeholder for the sky alone)."""
    cam = Camera(cam22)
    kind = int(soa["kind"][0])
    assert len(soa["kind"]) == 1, "the model covers one sphere under the sky"
    o, d, wq = primary_rays(cam, w, h, n_pix, n_rad, n_ang, law)
    avg = lambda x: np.tensordot(x, wq, axes=([2], [0])) if x.ndim == 3 else np.einsum("yxqc,q->yxc", x, wq)  # noqa: E731
    m1, m2 = sky_moments(d)
    out = dict(mean=avg(m1), second=avg(m2), rays=np.ones((h, w)), rays2=np.ones((h, w)))
    if kind == MAT_NONE:
        out["inside"], out["outside"] = np.zeros((h, w), bool), np.ones((h, w), bool)
        return out
    c = np.array([soa["cx"][0], soa["cy"][0], soa["cz"][0]], np.float64)
    r = float(np.sqrt(np.float64(soa["radius_sq"][0])))
    inside, outside = classify(cam, w, h, c, r)
    out["inside"], out["outside"] = inside, outside
    if inside.any():
        p, n = _hit_outside(o[inside], d[inside], c, r)
        s1, s2, k1, k2 = _surface_moments(kind, soa["albedo"][0], float(soa["param"][0]), max_bounces, d[inside], p, n, c, r)
        for key, v in (("mean", s1), ("second", s2), ("rays", k1), ("rays2", k2)):
            out[key][inside] = np.tensordot(v, wq, axes=([1], [0]))
    mixed = ~(inside | outside)
    for key in ("mean", "second", "rays", "rays2"):
        out[key][mixed] = np.nan
    return out


# ---- comparison with a render's fixed-point sums ---------------------------------------------------------------------------------

DETERMINISTIC_VAR = 1e-14                # a channel whose per-sample variance is below this is a constant per pixel
DETERMINISTIC_TOL = 4 * FIXED            # ... and must then equal it to a few fixed-point units (quantiser, one ulp of the sky)
Z_MAX = 5.0                              # bound of an aggregate z


def compare(model, sums, spp, select):
    """per channel over the pixels `select`: the aggregate z (sum of errors over the square root of the summed variances of the
    means), the per-pixel chi^2 and its degrees of freedom, and the largest |error| of a deterministic channel (else 0)"""
    got = sums[select].astype(np.float64) * FIXED / spp
    want = model["mean"][select]
    var1 = np.maximum(model["second"][select] - want * want, 0)
    out = []
    for ch in range(3):
        err, v = got[:, ch] - want[:, ch], var1[:, ch]
        if v.max() < DETERMINISTIC_VAR:
            out.append(dict(det=True, max_err=float(np.abs(err).max()), z=0.0, chi2=0.0, dof=0))
            continue
        sd = np.sqrt(v / spp)
        out.append(dict(det=False, max_err=0.0, z=float(err.sum() / np.sqrt((sd * sd).sum())), chi2=float(((err / sd) ** 2).sum()),
                        dof=int(len(err))))
    return out


def ray_z(model, rays, spp, select):
    """z of a frame's ray count against the model (every pixel of the frame must be in `select`)"""
    mean, m2 = model["rays"][select], model["rays2"][select]
    return (rays - spp * mean.sum()) / np.sqrt(spp * np.maximum(m2 - mean * mean, 0).sum())


def converge_stats(model, sums, rays, spp, what, deterministic_rays):
    """checks a frame (every pixel must be classed inside or outside) against the model and returns its statistics:
    per-channel aggregate |z| <= Z_MAX, per-pixel chi^2 below its 1e-6 quantile, deterministic channels to DETERMINISTIC_TOL,
    and the ray count exact (deterministic_rays) or within Z_MAX of its expectation"""
    from scipy.stats import chi2
    select = model["inside"] | model["outside"]
    assert select.all(), "%s: %d pixels straddle the silhouette" % (what, (~select).sum())
    stats = compare(model, sums, spp, select)
    for ch, st in zip("rgb", stats):
        if st["det"]:
            assert st["max_err"] <= DETERMINISTIC_TOL, "%s %s: a constant channel is off by %.3g" % (what, ch, st["max_err"])
            continue
        assert abs(st["z"]) <= Z_MAX, "%s %s: aggregate z %.2f" % (what, ch, st["z"])
        limit = chi2.isf(1e-6, st["dof"])
        assert st["chi2"] <= limit, "%s %s: chi^2 %.1f over %d pixels (1e-6 quantile %.1f)" % (what, ch, st["chi2"], st["dof"], limit)
    n = select.size * spp
    if deterministic_rays:
        want = model["rays"].sum() * spp
        assert rays == round(want) and abs(want - round(want)) < 1e-6, "%s: %d rays, the model says exactly %.1f" % (what, rays, want)
        rz = 0.0
    else:
        rz = float(ray_z(model, rays, spp, select))
        assert abs(rz) <= Z_MAX, "%s: %d rays (%.6f per sample), model %.6f per sample, z %.2f" % (what, rays, rays / n,
                                                                                                   model["rays"].mean(), rz)
    return dict(z=[round(s["z"], 2) for s in stats], chi2_dof=[round(s["chi2"] / s["dof"], 3) if s["dof"] else None for s in stats],
                max_err_det=[s["max_err"] if s["det"] else None for s in stats], rays_per_sample=rays / n, ray_z=round(rz, 2))
