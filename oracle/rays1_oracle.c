/*
 * rays1_oracle.c -- CPU restatement of the Rays1 (`src/latest` == step13) trace loop.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product path (rays1bench_b200/, the C-ABI
 * library, the drop-in executable) may include, link, load or call this file.  Only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs use it,
 * and only as the checker / the CPU baseline.
 *
 * Parity status: PINNED.  Every function below is checked (tests/test_oracle_*.py) against
 *   (1) golden vectors recorded from the reference's own compiled code (oracle/ref_harness.cpp
 *       builds /root/reference/src/latest/{rayweek1,soa_sphere}.cpp where they lie and calls
 *       Hitable::hit, Material::scatter, Camera::getRay, render_tile; vectors committed under
 *       tests/golden/ by oracle/make_golden.py), and
 *   (2) the known answers quoted in SURVEY.md section 8a (xorshift, unit-sphere sample, camera).
 *
 * All citations are file:line relative to /root/reference/.
 * Plain C11, scalar; explicit fmaf() exactly where the reference writes fma()
 * (src/latest/rayweek1.cpp:196,199), no other contraction (build with -ffp-contract=off).
 */
#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#define ORC_API __attribute__((visibility("default")))

enum { ORC_MAT_NONE = -1, ORC_MAT_LAMBERT = 0, ORC_MAT_METAL = 1, ORC_MAT_DIELECTRIC = 2 };

/* ------------------------------------------------------------------ RNG (src/latest/mymath.h:17-73) */

/* mymath.h:17-25 -- xorshift32 with shifts 13 / 17 / 15 (sic). */
static inline uint32_t xorshift32(uint32_t *state)
{
    uint32_t x = *state;
    x ^= x << 13;
    x ^= x >> 17;
    x ^= x << 15;
    *state = x;
    return x;
}

/* mymath.h:27-30 */
static inline float myrand01(uint32_t *state)
{
    return (float)(xorshift32(state) & 0xFFFFFF) * (float)(1.0 / 16777216.0);
}

/* mymath.h:32-35 */
static inline float myrand02(uint32_t *state)
{
    return (float)(xorshift32(state) & 0xFFFFFF) / (float)(0xFFFFFF / 2 + 1);
}

/* mymath.h:41-56 -- four independent lanes, lane k = state4[k]. */
static inline void myrand01_x4(uint32_t state4[4], float out[4])
{
    for (int k = 0; k < 4; ++k)
        out[k] = (float)(int32_t)(xorshift32(&state4[k]) & 0xFFFFFF) * (float)(1.0 / (0xFFFFFF + 1));
}

/* mymath.h:58-73 */
static inline void myrand02_x4(uint32_t state4[4], float out[4])
{
    for (int k = 0; k < 4; ++k)
        out[k] = (float)(int32_t)(xorshift32(&state4[k]) & 0xFFFFFF) * (float)(1.0 / (0xFFFFFF / 2 + 1));
}

typedef struct { float x, y, z; } v3;

static inline v3 v3_make(float x, float y, float z) { v3 r = { x, y, z }; return r; }
static inline v3 v3_add(v3 a, v3 b) { return v3_make(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 v3_sub(v3 a, v3 b) { return v3_make(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 v3_mul(v3 a, v3 b) { return v3_make(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 v3_scale(v3 a, float s) { return v3_make(a.x * s, a.y * s, a.z * s); }
/* mymath.h:203-204 -- dot = sum(a*b) = (x + y) + z */
static inline float v3_dot(v3 a, v3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
/* mymath.h:206-208 -- unit_vector = v * (1 / length(v)).  Built with -ffast-math (bench.py:175) this is vrsqrtss + ONE Newton
 * step, in this order (disassembly of the Ray ctor inlined into scatter() / getRay()):
 *     y = rsqrtss(x) ; a = y * x ; a = fma(a, y, -3) ; b = y * -0.5 ; inv = a * b ; v * inv
 * RSQRTSS is a 2048-case table on Intel CPUs (rays1bench_b200/csrc/r1_rsqrt12_table.h, measured by tools/gen_rsqrt12_table.c),
 * restated here so that the oracle gives the same bits on any host.  The step's result is always slightly below 1/sqrt(x)
 * (-1.5 eps^2): directions come out up to 1.6e-7 SHORT of unit length, which is visible in the statistics of large scenes
 * (far hit points land inside their spheres and self-hit; DESIGN.md section 3).  g_as_built = 0 keeps the exact 1 / sqrtf. */
#include "../rays1bench_b200/csrc/r1_rsqrt12_table.h"
static const uint16_t k_rsqrt12[R1_RSQRT12_ENTRIES] = R1_RSQRT12_INIT;
static int g_as_built;
static inline float rsqrt12(float x)
{
    uint32_t xb, yb;
    memcpy(&xb, &x, 4);
    if (xb < 0x00800000u) return INFINITY;                                  /* zero / denormal (and negative: not used) */
    yb = r1_rsqrt12_bits(xb, k_rsqrt12);   /* the one definition the CUDA kernels use too */
    float y;
    memcpy(&y, &yb, 4);
    return y;
}
static inline float inv_length_as_built(float x)
{
    const float y = rsqrt12(x);
    const float a = fmaf(y * x, y, -3.0f), b = y * -0.5f;
    return a * b;
}
static inline v3 v3_unit(v3 v)
{
    const float x = v3_dot(v, v);
    return v3_scale(v, g_as_built ? inv_length_as_built(x) : 1.0f / sqrtf(x));
}
/* the CPU's own RSQRTSS, for the test that pins the table against real hardware (x86 only) */
#if defined(__SSE__)
#include <xmmintrin.h>
ORC_API float orc_hw_rsqrtss(float x) { return _mm_cvtss_f32(_mm_rsqrt_ss(_mm_set_ss(x))); }
#else
ORC_API float orc_hw_rsqrtss(float x) { return rsqrt12(x); }
#endif
ORC_API float orc_rsqrt12(float x) { return rsqrt12(x); }
/* mymath.h:188-195 */
static inline v3 v3_cross(v3 a, v3 b)
{
    return v3_make(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}

/* mymath.h:224-235 -- rejection sampling in the unit ball from the x4 stream: [0,2)-1 per lane. */
static inline v3 random_in_unit_sphere(uint32_t state4[4])
{
    float r[4];
    v3 p;
    do {
        myrand02_x4(state4, r);
        p = v3_make(r[0] - 1.0f, r[1] - 1.0f, r[2] - 1.0f);
    } while (v3_dot(p, p) >= 1.0f);
    return p;
}

/* rayweek1.cpp:353-362 -- rejection sampling in the unit disk from the scalar stream.
 * The reference draws both coordinates inside one constructor call; gcc evaluates the
 * arguments right to left, so the FIRST draw lands in y (checked against the harness). */
static inline void random_in_unit_disk(uint32_t *state, float *px, float *py)
{
    float x, y;
    do {
        y = myrand02(state) - 1.0f;
        x = myrand02(state) - 1.0f;
    } while ((x * x + y * y) + 0.0f >= 1.0f);
    *px = x;
    *py = y;
}

/* ------------------------------------------------------------------ scene storage */

/* soa_sphere.h:38-53 -- SoA sphere container; materials flattened to (kind, albedo, param). */
typedef struct orc_scene {
    uint32_t count, capacity;
    float *cx, *cy, *cz, *radius_sq, *inv_radius;
    int32_t *kind;      /* ORC_MAT_* ; -1 for the placeholder's nullptr material */
    float *albedo;      /* 3 per sphere */
    float *param;       /* Metal: fuzz (clamped to <= 1, rayweek1.cpp:424); Dielectric: ior */
    /* Camera (rayweek1.cpp:388-393) */
    v3 origin, llc, horizontal, vertical, u, v, w;
    float lens_radius;
} orc_scene;

static void scene_reserve(orc_scene *s, uint32_t cap)
{
    if (cap <= s->capacity) return;
    s->cx = realloc(s->cx, cap * sizeof(float));
    s->cy = realloc(s->cy, cap * sizeof(float));
    s->cz = realloc(s->cz, cap * sizeof(float));
    s->radius_sq = realloc(s->radius_sq, cap * sizeof(float));
    s->inv_radius = realloc(s->inv_radius, cap * sizeof(float));
    s->kind = realloc(s->kind, cap * sizeof(int32_t));
    s->albedo = realloc(s->albedo, 3 * cap * sizeof(float));
    s->param = realloc(s->param, cap * sizeof(float));
    s->capacity = cap;
}

/* soa_sphere.cpp:70-85 -- add(): radius_sq = r*r ; inv_radius = r > 0 ? 1/r : 0. */
static void scene_add(orc_scene *s, v3 c, float radius, int kind, v3 albedo, float param)
{
    if (s->count == s->capacity) scene_reserve(s, 2 * s->capacity + 16);
    uint32_t i = s->count++;
    s->cx[i] = c.x;
    s->cy[i] = c.y;
    s->cz[i] = c.z;
    s->radius_sq[i] = radius * radius;
    s->inv_radius[i] = radius > 0 ? (1.0f / radius) : 0;
    s->kind[i] = kind;
    s->albedo[3 * i + 0] = albedo.x;
    s->albedo[3 * i + 1] = albedo.y;
    s->albedo[3 * i + 2] = albedo.z;
    s->param[i] = param;
}

static void add_lambert(orc_scene *s, v3 c, float r, v3 a) { scene_add(s, c, r, ORC_MAT_LAMBERT, a, 0.0f); }
/* rayweek1.cpp:422-425 -- fuzz = f < 1 ? f : 1 */
static void add_metal(orc_scene *s, v3 c, float r, v3 a, float f) { scene_add(s, c, r, ORC_MAT_METAL, a, f < 1 ? f : 1); }
static void add_dielectric(orc_scene *s, v3 c, float r, float ior) { scene_add(s, c, r, ORC_MAT_DIELECTRIC, v3_make(1, 1, 1), ior); }

/* rayweek1.cpp:575-576, 647-648, 715-716 -- pad to a multiple of SIMD_WIDTH (8) with radius-0 spheres at 999999999. */
static void scene_pad(orc_scene *s, uint32_t multiple)
{
    while (s->count % multiple != 0)
        scene_add(s, v3_make(999999999.0f, 999999999.0f, 999999999.0f), 0.0f, ORC_MAT_NONE, v3_make(0, 0, 0), 0.0f);
}

/* rayweek1.cpp:366-379 -- Camera::init */
static void camera_init(orc_scene *s, v3 lookfrom, v3 lookat, v3 vup, float vfov, float aspect, float aperture, float focus_dist)
{
    /* The builders call Camera::init with constants, so gcc folds it at COMPILE time -- with the fast-math reassociations applied
     * first: `vfov * (float)M_PI / 180 / 2` becomes vfov * C with C = (float)M_PI * (1.0f / 360.0f), the functions (tanf, the
     * 1 / sqrtf of unit_vector) are then evaluated correctly rounded, everything else in source order.  Checked bit for bit against
     * the constants recorded from the reference's binary for all four scenes (tests/golden/rays_*.npz "camera").  With
     * g_as_built = 0: the source order, theta = vfov * pi / 180, tanf(theta / 2). */
    s->lens_radius = aperture / 2;
    float half_height;
    if (g_as_built) {
        const float c = (float)M_PI * (1.0f / 360.0f);
        half_height = (float)tan((double)(vfov * c));
    } else {
        float theta = vfov * (float)M_PI / 180;
        half_height = tanf(theta / 2);
    }
    float half_width = aspect * half_height;
    s->origin = lookfrom;
    {   /* unit_vector folded at compile time: the exact 1 / sqrt, not the run-time rsqrtss + Newton step */
        v3 a = v3_sub(lookfrom, lookat);
        s->w = v3_scale(a, 1.0f / sqrtf(v3_dot(a, a)));
        v3 b = v3_cross(vup, s->w);
        s->u = v3_scale(b, 1.0f / sqrtf(v3_dot(b, b)));
    }
    s->v = v3_cross(s->w, s->u);
    s->llc = v3_sub(v3_sub(v3_sub(s->origin, v3_scale(s->u, half_width * focus_dist)),
                           v3_scale(s->v, half_height * focus_dist)),
                    v3_scale(s->w, focus_dist));
    s->horizontal = v3_scale(s->u, 2 * half_width * focus_dist);
    s->vertical = v3_scale(s->v, 2 * half_height * focus_dist);
}

/* rayweek1.cpp:552-579 */
static void build_small(orc_scene *s, float aspect)
{
    camera_init(s, v3_make(2, 1, 2), v3_make(0, 0, 0), v3_make(0, 1, 0), 60, aspect, 0.1f, 5.0f);
    add_lambert(s, v3_make(0, 0, -1), 0.5f, v3_make(0.1f, 0.2f, 0.5f));
    add_lambert(s, v3_make(0, -100.5f, -1), 100.0f, v3_make(0.8f, 0.8f, 0));
    add_metal(s, v3_make(1, 0, -1), 0.5f, v3_make(0.8f, 0.6f, 0.2f), 0.3f);
    add_dielectric(s, v3_make(-1, 0, -1), 0.5f, 1.5f);
    add_dielectric(s, v3_make(-1, 0, -1), -0.45f, 1.5f);
    scene_pad(s, 8);
}

/* rayweek1.cpp:582-651 -- "the aras_p scene" */
static void build_medium(orc_scene *s, float aspect)
{
    camera_init(s, v3_make(0, 2, 3), v3_make(0, 0, 0), v3_make(0, 1, 0), 60, aspect, 0.1f * 0.2f, 3);
    add_lambert(s, v3_make(0, -100.5f, -1), 100, v3_make(0.8f, 0.8f, 0.8f));
    add_lambert(s, v3_make(2, 0, -1), 0.5f, v3_make(0.8f, 0.4f, 0.4f));
    add_lambert(s, v3_make(0, 0, -1), 0.5f, v3_make(0.4f, 0.8f, 0.4f));
    add_metal(s, v3_make(-2, 0, -1), 0.5f, v3_make(0.4f, 0.4f, 0.8f), 0);
    add_metal(s, v3_make(2, 0, 1), 0.5f, v3_make(0.4f, 0.8f, 0.4f), 0);
    add_metal(s, v3_make(0, 0, 1), 0.5f, v3_make(0.4f, 0.8f, 0.4f), 0.2f);
    add_metal(s, v3_make(-2, 0, 1), 0.5f, v3_make(0.4f, 0.8f, 0.4f), 0.6f);
    add_dielectric(s, v3_make(0.5f, 1, 0.5f), 0.5f, 1.5f);
    add_lambert(s, v3_make(-1.5f, 1.5f, 0.f), 0.3f, v3_make(0.8f, 0.6f, 0.2f));
    /* four rows of nine: z = -3 lambert greys, z = -4 metal greys, z = -5 metal hues, z = -6 lambert hues (last one metal) */
    static const float grey[9] = { 0.1f, 0.2f, 0.3f, 0.4f, 0.5f, 0.6f, 0.7f, 0.8f, 0.9f };
    static const float hue[9][3] = {
        { 0.8f, 0.1f, 0.1f }, { 0.8f, 0.5f, 0.1f }, { 0.8f, 0.8f, 0.1f }, { 0.4f, 0.8f, 0.1f }, { 0.1f, 0.8f, 0.1f },
        { 0.1f, 0.8f, 0.5f }, { 0.1f, 0.8f, 0.8f }, { 0.1f, 0.1f, 0.8f }, { 0.5f, 0.1f, 0.8f } };
    for (int k = 0; k < 9; ++k) add_lambert(s, v3_make((float)(4 - k), 0, -3), 0.5f, v3_make(grey[k], grey[k], grey[k]));
    for (int k = 0; k < 9; ++k) add_metal(s, v3_make((float)(4 - k), 0, -4), 0.5f, v3_make(grey[k], grey[k], grey[k]), 0);
    for (int k = 0; k < 9; ++k) add_metal(s, v3_make((float)(4 - k), 0, -5), 0.5f, v3_make(hue[k][0], hue[k][1], hue[k][2]), 0);
    for (int k = 0; k < 8; ++k) add_lambert(s, v3_make((float)(4 - k), 0, -6), 0.5f, v3_make(hue[k][0], hue[k][1], hue[k][2]));
    add_metal(s, v3_make(-4, 0, -6), 0.5f, v3_make(0.5f, 0.1f, 0.8f), 0);
    add_lambert(s, v3_make(1.5f, 1.5f, -2), 0.3f, v3_make(0.1f, 0.2f, 0.5f));
    scene_pad(s, 8);
}

/* rayweek1.cpp:654-719 (grid 30 x 16) generalised by (gw, gh, ior_mod) for the synthetic 4096-sphere
 * scene of SURVEY.md section 8d config 5 (grid 66 x 62, ior = 1.2 + 0.05*(i % 480)).  libc srand(111)/rand(). */
static void build_grid(orc_scene *s, float aspect, int gw, int gh, int ior_mod, v3 lookfrom, float focus)
{
    camera_init(s, lookfrom, v3_make(0, 0, 0), v3_make(0, 1, 0), 60, aspect, 0.1f, focus);
    int W = gw, H = gh;
    srand(111);
    for (int y = 0; y < H; ++y) {
        for (int x = 0; x < W; ++x) {
            v3 pos = v3_make((x - W / 2) * 1.1f, 0, (y - H / 2) * 1.1f);
            /* :679-681, :692, :696 as the fast-math build evaluates them (checked bit for bit against the recorded SoA):
             * x / 255.0f -> x * (1 / 255.0f);  1.2f + i * 0.05f -> fma;  0.01f + 0.5f * y / H -> fma(0.5f * y, 1 / H, 0.01f) */
            float r = g_as_built ? (rand() & 0xff) * (1.0f / 255.0f) : (rand() & 0xff) / 255.0f;
            float g = g_as_built ? (rand() & 0xff) * (1.0f / 255.0f) : (rand() & 0xff) / 255.0f;
            float b = g_as_built ? (rand() & 0xff) * (1.0f / 255.0f) : (rand() & 0xff) / 255.0f;
            int i = x + y * W;
            float radius = 0.45f;
            if (i % 20 == 0) {
                int k = ior_mod ? (i % ior_mod) : i;
                add_dielectric(s, pos, radius, g_as_built ? fmaf((float)k, 0.05f, 1.2f) : 1.2f + k * 0.05f);
            } else if (i % 10 == 0) {
                pos = v3_add(pos, v3_make(0, 0.1f, 0));
                add_metal(s, pos, radius, v3_make(r, g, b),
                          g_as_built ? fmaf(0.5f * y, 1.0f / (float)(H), 0.01f) : 0.01f + 0.5f * y / (float)(H));
            } else {
                add_lambert(s, pos, radius, v3_make(r, g, b));
            }
        }
    }
    add_lambert(s, v3_make(0, -1000.5f, 0), 1000, v3_make(0.5f, 0.5f, 0.5f));
    add_metal(s, v3_make(5, 3, 0), 2, v3_make(0.5f, 0.5f, 0.8f), 0.65f);
    add_dielectric(s, v3_make(0, 3, 0), 2, 1.5f);
    add_metal(s, v3_make(-5, 3, 0), 2, v3_make(0.8f, 0.2f, 0.2f), 0.05f);
    scene_pad(s, 8);
}

ORC_API orc_scene *orc_scene_create(const char *name, int image_w, int image_h)
{
    orc_scene *s = calloc(1, sizeof(*s));
    float aspect = (float)image_w / (float)image_h; /* rayweek1.cpp:564 */
    if (!strcmp(name, "small")) build_small(s, aspect);
    else if (!strcmp(name, "medium")) build_medium(s, aspect);
    else if (!strcmp(name, "large")) build_grid(s, aspect, 30, 16, 0, v3_make(3, 8, 15), 10.0f);
    else if (!strcmp(name, "synth4096")) build_grid(s, aspect, 66, 62, 480, v3_make(6, 16, 30), 20.0f);
    else { free(s); return NULL; }
    return s;
}

/* A scene from its SoA as given (e.g. r1_scene_get_soa of a scene file), placeholders included, no padding added; the camera
 * stays zero until orc_scene_set_camera.  For hit() on scenes the named builders do not make. */
ORC_API orc_scene *orc_scene_create_from_soa(int n, const float *cx, const float *cy, const float *cz, const float *radius_sq,
                                             const float *inv_radius, const int32_t *kind, const float *albedo, const float *param)
{
    if (n < 0) return NULL;
    orc_scene *s = calloc(1, sizeof(*s));
    scene_reserve(s, (uint32_t)n + 1);
    size_t b = (size_t)n * 4;
    memcpy(s->cx, cx, b); memcpy(s->cy, cy, b); memcpy(s->cz, cz, b);
    memcpy(s->radius_sq, radius_sq, b); memcpy(s->inv_radius, inv_radius, b);
    memcpy(s->kind, kind, b); memcpy(s->albedo, albedo, 3 * b); memcpy(s->param, param, b);
    s->count = (uint32_t)n;
    return s;
}

ORC_API void orc_scene_destroy(orc_scene *s)
{
    if (!s) return;
    free(s->cx); free(s->cy); free(s->cz); free(s->radius_sq); free(s->inv_radius);
    free(s->kind); free(s->albedo); free(s->param);
    free(s);
}

ORC_API uint32_t orc_scene_count(const orc_scene *s) { return s->count; }

ORC_API void orc_scene_get_soa(const orc_scene *s, float *cx, float *cy, float *cz, float *radius_sq, float *inv_radius,
                               int32_t *kind, float *albedo, float *param)
{
    size_t n = s->count;
    memcpy(cx, s->cx, n * 4); memcpy(cy, s->cy, n * 4); memcpy(cz, s->cz, n * 4);
    memcpy(radius_sq, s->radius_sq, n * 4); memcpy(inv_radius, s->inv_radius, n * 4);
    memcpy(kind, s->kind, n * 4); memcpy(albedo, s->albedo, 3 * n * 4); memcpy(param, s->param, n * 4);
}

/* out[22] = origin, llc, horizontal, vertical, u, v, w (3 each), lens_radius */
ORC_API void orc_scene_get_camera(const orc_scene *s, float *out)
{
    const v3 *src[7] = { &s->origin, &s->llc, &s->horizontal, &s->vertical, &s->u, &s->v, &s->w };
    for (int k = 0; k < 7; ++k) { out[3 * k] = src[k]->x; out[3 * k + 1] = src[k]->y; out[3 * k + 2] = src[k]->z; }
    out[21] = s->lens_radius;
}

/* Installs the 22 camera constants as given (order of orc_scene_get_camera).  The reference's Camera::init is folded at
 * compile time by gcc -ffast-math and differs from a run-time evaluation of rayweek1.cpp:366-379 by up to 4 ulp; fixtures
 * that need bit-identical primary rays (per-pixel replay) install the recorded constants. */
ORC_API void orc_scene_set_camera(orc_scene *s, const float *cam)
{
    v3 *dst[7] = { &s->origin, &s->llc, &s->horizontal, &s->vertical, &s->u, &s->v, &s->w };
    for (int k = 0; k < 7; ++k) *dst[k] = v3_make(cam[3 * k], cam[3 * k + 1], cam[3 * k + 2]);
    s->lens_radius = cam[21];
}

/* ------------------------------------------------------------------ hit (rayweek1.cpp:152-339) */

typedef struct { float t; v3 p, normal; int32_t index; } hit_rec;

/* 1: arithmetic association of the reference AS BUILT by bench.py:175 (gcc -ffast-math); 0: as written in the source. */

static int scene_hit(const orc_scene *s, v3 o, v3 d, float t_min, float t_max, hit_rec *rec)
{
    int hit_index = -1;
    float hit_t = 0.0f;
    /* Phase 1 and phase 2 of the reference are fused here: candidates are visited in ascending index order in
     * both (positive_idx[] is filled in index order, :209-224, and consumed in order, :284-314), so testing each
     * sphere as it is scanned gives the same (t_max, hit_index) sequence. */
    for (uint32_t i = 0; i < s->count; ++i) {
        /* :192-194 */
        const float cox = s->cx[i] - o.x, coy = s->cy[i] - o.y, coz = s->cz[i] - o.z;
        /* :196 */
        const float nb = fmaf(coz, d.z, fmaf(coy, d.y, cox * d.x));
        /* :199-200.  The source reads  c = |co|^2 - r^2 ; discr = nb*nb - c.  The reference is BUILT with
         * -ffast-math (bench.py:175), and gcc 13 reassociates that into  discr = fmsub(nb, nb, |co|^2) + r^2
         * (vfmsub132ps + vaddps in the disassembly of Hitable::hit).  The two differ by one rounding at
         * magnitude |co|^2 -- 0.06 absolute on the r = 1000 ground sphere -- so the oracle follows the binary
         * (g_as_built = 1, default) and keeps the source order selectable for the tolerance study in DESIGN.md. */
        const float q = fmaf(coz, coz, fmaf(coy, coy, cox * cox));
        const float discr = g_as_built ? (fmaf(nb, nb, -q) + s->radius_sq[i]) : (nb * nb - (q - s->radius_sq[i]));
        /* :204 -- candidate iff the SIGN BIT of discr is clear */
        if (signbit(discr)) continue;
        /* :288-292 -- placeholder or non-positive radius */
        if (s->inv_radius[i] == 0) continue;
        /* :294-313 */
        const float discr_sq = sqrtf(discr);
        float temp = nb - discr_sq;
        if (temp < t_max && temp > t_min) { t_max = temp; hit_t = temp; hit_index = (int)i; continue; }
        temp = nb + discr_sq;
        if (temp < t_max && temp > t_min) { t_max = temp; hit_t = temp; hit_index = (int)i; continue; }
    }
    /* :316-322 */
    if (hit_index != -1) {
        rec->t = hit_t;
        /* :319 point_at_parameter = o + t*d ; contracted to one fma per component in the fast-math build */
        rec->p = g_as_built ? v3_make(fmaf(hit_t, d.x, o.x), fmaf(hit_t, d.y, o.y), fmaf(hit_t, d.z, o.z))
                            : v3_add(o, v3_scale(d, hit_t));
        rec->normal = v3_scale(v3_sub(rec->p, v3_make(s->cx[hit_index], s->cy[hit_index], s->cz[hit_index])),
                               s->inv_radius[hit_index]);
        rec->index = hit_index;
    }
    return hit_index != -1;
}

/* Batch form of Hitable::hit for parity tests. dir must already be unit length (Ray ctor, :104-108). */
ORC_API void orc_hit(const orc_scene *s, int n, const float *org, const float *dir, float t_min, float t_max,
                     int32_t *index, float *t, float *p, float *normal)
{
    for (int k = 0; k < n; ++k) {
        hit_rec rec;
        memset(&rec, 0, sizeof(rec));
        int h = scene_hit(s, v3_make(org[3 * k], org[3 * k + 1], org[3 * k + 2]),
                          v3_make(dir[3 * k], dir[3 * k + 1], dir[3 * k + 2]), t_min, t_max, &rec);
        index[k] = h ? rec.index : -1;
        t[k] = h ? rec.t : 0.0f;
        p[3 * k] = rec.p.x; p[3 * k + 1] = rec.p.y; p[3 * k + 2] = rec.p.z;
        normal[3 * k] = rec.normal.x; normal[3 * k + 1] = rec.normal.y; normal[3 * k + 2] = rec.normal.z;
    }
}

/* ------------------------------------------------------------------ scatter (rayweek1.cpp:396-512) */

/* g_as_built (hit(), above) also selects the association the reference's BINARY uses in scatter().  Read from the
 * disassembly of oracle/_ref/libref_rays1.so (gcc 13.3, bench.py:175 flags; Lambertian/Metal/Dielectric::scatter):
 *   - every dot() is mul, mul, mul, add, add -- (x + y) + z, never contracted (mymath.h:203-204);
 *   - reflect (:414-417) is one fnmadd per component: v - (2 dn) n with 2 dn = dn + dn;
 *   - Metal's  reflected + fuzz * rs  (:430) is one fma per component;
 *   - refract (:439-452): w = fma(dt, dt, -1); m = (k k) w; taken iff m > -1; discriminant = m + 1;
 *     refracted = fnmadd(n', sqrt(discriminant), k * fnmadd(dt, n', uv));
 *   - schlick (:454-459): r0s = (1 - ior) / (ior + 1); powf(x, 5) expanded by -ffast-math into ((x x)(x x)) * ((1 - r0) x)
 *     with 1 - r0 = fnmadd(r0s, r0s, 1) and the sum as fma(r0s, r0s, .);
 *   - the Ray ctor's normalise (:104-108, mymath.h:206-208) is vrsqrtss + one Newton step (hardware-specific table, <= 2e-7
 *     from the exact value); restated here as 1 / sqrtf.
 * The source order (g_as_built = 0) differs from the binary by up to 7.6e-6 on the golden rays (k^2 = ior^2 up to 585
 * amplifies the rounding of 1 - dt^2); the as-built order by the normalise only (~2e-7). */
static int g_as_built = 1;
ORC_API void orc_set_as_built(int v) { g_as_built = v; }

/* :414-417 */
static inline v3 reflect(v3 v, v3 n)
{
    if (g_as_built) {
        const float dn = v3_dot(v, n), k = dn + dn;
        return v3_make(fmaf(-n.x, k, v.x), fmaf(-n.y, k, v.y), fmaf(-n.z, k, v.z));
    }
    return v3_sub(v, v3_scale(n, 2 * v3_dot(v, n)));
}

/* :439-452 */
static inline int refract(v3 uv, v3 n, float ni_over_nt, v3 *refracted)
{
    float dt = v3_dot(uv, n);
    float discriminant = 1.0f - ni_over_nt * ni_over_nt * (1 - dt * dt);
    if (discriminant > 0) {
        *refracted = v3_sub(v3_scale(v3_sub(uv, v3_scale(n, dt)), ni_over_nt), v3_scale(n, sqrtf(discriminant)));
        return 1;
    }
    return 0;
}

/* :454-459 */
static inline float schlick(float cosine, float ref_idx)
{
    float r0 = (1 - ref_idx) / (1 + ref_idx);
    r0 = r0 * r0;
    return r0 + (1 - r0) * powf((1 - cosine), 5);
}

/* One scatter event with the random inputs made explicit: `rs` is the unit-ball sample the reference would draw
 * from state4 (Lambertian :405, Metal :430 -- drawn even when fuzz == 0), `ru` the scalar uniform Dielectric draws
 * (:503).  Returns the reference's bool; *dir_out is the normalised scattered direction (Ray ctor). */
static int scatter_explicit(const orc_scene *s, int idx, v3 dir_in, v3 p, v3 normal, v3 rs, float ru, v3 *atten, v3 *dir_out)
{
    const float *al = &s->albedo[3 * idx];
    switch (s->kind[idx]) {
    case ORC_MAT_LAMBERT: { /* :403-409 */
        /* target = p + n + rs ; dir = unit(target - p).  Built with -ffast-math the reference cancels p and computes
         * unit(n + rs) (checked against the recorded scatter directions: 1.8e-7 vs 7.5e-6 for the source order). */
        if (g_as_built) {
            *dir_out = v3_unit(v3_add(normal, rs));
        } else {
            v3 target = v3_add(v3_add(p, normal), rs);
            *dir_out = v3_unit(v3_sub(target, p));
        }
        *atten = v3_make(al[0], al[1], al[2]);
        return 1;
    }
    case ORC_MAT_METAL: { /* :427-433 */
        v3 reflected = reflect(dir_in, normal);
        const float fuzz = s->param[idx];
        if (g_as_built) *dir_out = v3_unit(v3_make(fmaf(fuzz, rs.x, reflected.x), fmaf(fuzz, rs.y, reflected.y), fmaf(fuzz, rs.z, reflected.z)));
        else *dir_out = v3_unit(v3_add(reflected, v3_scale(rs, fuzz)));
        *atten = v3_make(al[0], al[1], al[2]);
        return v3_dot(*dir_out, normal) > 0;
    }
    case ORC_MAT_DIELECTRIC: { /* :470-511 */
        const float ref_idx = s->param[idx];
        *atten = v3_make(1, 1, 1);
        if (g_as_built) { /* the binary's association, see the notes above reflect() */
            const float dn = v3_dot(dir_in, normal);
            v3 n1;
            float k, cosine, dt;
            if (dn > 0) { n1 = v3_make(-normal.x, -normal.y, -normal.z); k = ref_idx; cosine = dn * ref_idx; dt = v3_dot(n1, dir_in); }
            else { n1 = normal; k = 1.0f / ref_idx; cosine = -dn; dt = dn; }
            const float m = (k * k) * fmaf(dt, dt, -1.0f);
            float prob = 1.0f;
            v3 refr = v3_make(0, 0, 0);
            if (m > -1.0f) {
                const float sq = sqrtf(m + 1.0f);
                const v3 a = v3_make(fmaf(-dt, n1.x, dir_in.x), fmaf(-dt, n1.y, dir_in.y), fmaf(-dt, n1.z, dir_in.z));
                refr = v3_make(fmaf(-n1.x, sq, k * a.x), fmaf(-n1.y, sq, k * a.y), fmaf(-n1.z, sq, k * a.z));
                const float r0s = (1.0f - ref_idx) / (ref_idx + 1.0f), x = 1.0f - cosine;
                prob = fmaf(r0s, r0s, ((x * x) * (x * x)) * (fmaf(-r0s, r0s, 1.0f) * x));
            }
            *dir_out = v3_unit(ru < prob ? reflect(dir_in, normal) : refr);
            return 1;
        }
        v3 outward_normal, refracted = v3_make(0, 0, 0);
        v3 reflected = reflect(dir_in, normal);
        float ni_over_nt, reflect_prob, cosine;
        if (v3_dot(dir_in, normal) > 0) {
            outward_normal = v3_make(-normal.x, -normal.y, -normal.z);
            ni_over_nt = ref_idx;
            cosine = ref_idx * v3_dot(dir_in, normal);
        } else {
            outward_normal = normal;
            ni_over_nt = 1.0f / ref_idx;
            cosine = -v3_dot(dir_in, normal);
        }
        if (refract(dir_in, outward_normal, ni_over_nt, &refracted)) reflect_prob = schlick(cosine, ref_idx);
        else reflect_prob = 1;
        if (ru < reflect_prob) *dir_out = v3_unit(reflected);
        else *dir_out = v3_unit(refracted);
        return 1;
    }
    default:
        return 0;
    }
}

ORC_API void orc_scatter(const orc_scene *s, int n, const float *dir_in, const float *p, const float *normal,
                         const int32_t *index, const float *rand_sphere, const float *rand_u, int32_t *ok,
                         float *atten, float *dir_out)
{
    for (int k = 0; k < n; ++k) {
        v3 a = v3_make(0, 0, 0), d = v3_make(0, 0, 0);
        ok[k] = scatter_explicit(s, index[k], v3_make(dir_in[3 * k], dir_in[3 * k + 1], dir_in[3 * k + 2]),
                                 v3_make(p[3 * k], p[3 * k + 1], p[3 * k + 2]),
                                 v3_make(normal[3 * k], normal[3 * k + 1], normal[3 * k + 2]),
                                 v3_make(rand_sphere[3 * k], rand_sphere[3 * k + 1], rand_sphere[3 * k + 2]), rand_u[k], &a, &d);
        atten[3 * k] = a.x; atten[3 * k + 1] = a.y; atten[3 * k + 2] = a.z;
        dir_out[3 * k] = d.x; dir_out[3 * k + 1] = d.y; dir_out[3 * k + 2] = d.z;
    }
}

/* ------------------------------------------------------------------ camera ray (rayweek1.cpp:381-386) */

static inline void camera_ray(const orc_scene *s, float su, float tv, float disk_x, float disk_y, v3 *org, v3 *dir)
{
    float rdx = s->lens_radius * disk_x, rdy = s->lens_radius * disk_y;
    if (g_as_built) {
        /* the binary: offset = fma(v, rd.y, u * rd.x) ; dir = ((llc - origin) + fma(t, vertical, s * horizontal)) - offset */
        v3 offset = v3_make(fmaf(s->v.x, rdy, s->u.x * rdx), fmaf(s->v.y, rdy, s->u.y * rdx), fmaf(s->v.z, rdy, s->u.z * rdx));
        *org = v3_add(s->origin, offset);
        v3 lo = v3_sub(s->llc, s->origin);
        v3 sv = v3_make(fmaf(tv, s->vertical.x, su * s->horizontal.x), fmaf(tv, s->vertical.y, su * s->horizontal.y),
                        fmaf(tv, s->vertical.z, su * s->horizontal.z));
        *dir = v3_unit(v3_sub(v3_add(lo, sv), offset));
        return;
    }
    v3 offset = v3_add(v3_scale(s->u, rdx), v3_scale(s->v, rdy));
    *org = v3_add(s->origin, offset);
    v3 d = v3_sub(v3_sub(v3_add(v3_add(s->llc, v3_scale(s->horizontal, su)), v3_scale(s->vertical, tv)), s->origin), offset);
    *dir = v3_unit(d);
}

ORC_API void orc_get_ray(const orc_scene *s, int n, const float *su, const float *tv, const float *disk, float *org, float *dir)
{
    for (int k = 0; k < n; ++k) {
        v3 o, d;
        camera_ray(s, su[k], tv[k], disk[2 * k], disk[2 * k + 1], &o, &d);
        org[3 * k] = o.x; org[3 * k + 1] = o.y; org[3 * k + 2] = o.z;
        dir[3 * k] = d.x; dir[3 * k + 1] = d.y; dir[3 * k + 2] = d.z;
    }
}

/* ------------------------------------------------------------------ integrator + tile loop */

typedef struct {
    const orc_scene *scene;
    uint8_t *image;         /* RGB8, row 0 = bottom of the picture (rayweek1.cpp:750, common.h:106) */
    int image_w, image_h, tile_w, tile_h, spp, max_bounces;
    uint32_t state;         /* rayweek1.cpp:90 */
    uint32_t state4[4];     /* rayweek1.cpp:91 */
    uint64_t num_rays;
} thread_data;

/* rayweek1.cpp:515-536, recursion unrolled into a loop; attenuations are multiplied innermost-first as the
 * recursion does (a0 * (a1 * (... * leaf))) by keeping them on a small stack. */
static v3 color(v3 o, v3 d, thread_data *td)
{
    v3 stack[64];
    int depth = 0;
    v3 leaf;
    for (;;) {
        ++td->num_rays; /* :517 */
        hit_rec rec;
        if (scene_hit(td->scene, o, d, 0.001f, FLT_MAX, &rec)) { /* :519 */
            v3 atten, nd;
            int ok = 0;
            if (depth < td->max_bounces) { /* :523 (short-circuit: no RNG draw past the cap) */
                v3 rs = v3_make(0, 0, 0);
                float ru = 0;
                int kind = td->scene->kind[rec.index];
                if (kind == ORC_MAT_LAMBERT || kind == ORC_MAT_METAL) rs = random_in_unit_sphere(td->state4);
                /* Dielectric draws its uniform AFTER computing reflect_prob (:503); order within one stream only */
                if (kind == ORC_MAT_DIELECTRIC) ru = myrand01(&td->state);
                ok = scatter_explicit(td->scene, rec.index, d, rec.p, rec.normal, rs, ru, &atten, &nd);
            }
            if (ok) {
                stack[depth++] = atten;
                o = rec.p;
                d = nd;
                continue;
            }
            leaf = v3_make(0, 0, 0); /* :527-528 */
            break;
        }
        /* :532-534 */
        float t = 0.5f * (d.y + 1.0f);
        if (g_as_built) {   /* the binary: it = 1 - t ; fma(t, (0.5, 0.7, 1.0), it) per component */
            const float it = 1.0f - t;
            leaf = v3_make(fmaf(t, 0.5f, it), fmaf(t, 0.7f, it), fmaf(t, 1.0f, it));
        } else {
            leaf = v3_add(v3_scale(v3_make(1.0f, 1.0f, 1.0f), 1 - t), v3_scale(v3_make(0.5f, 0.7f, 1.0f), t));
        }
        break;
    }
    while (depth > 0) leaf = v3_mul(stack[--depth], leaf);
    return leaf;
}

/* rayweek1.cpp:61-68 */
static int tiles_required(int tile_w, int width)
{
    int n = width / tile_w;
    if (n * tile_w < width) n++;
    return n;
}

/* rayweek1.cpp:722-782 */
static void render_tile(int tile_index, thread_data *td)
{
    int num_tiles_x = tiles_required(td->tile_w, td->image_w);
    int tile_x = tile_index % num_tiles_x, tile_y = tile_index / num_tiles_x;
    int y0 = tile_y * td->tile_h, y1 = y0 + td->tile_h;
    int x0 = tile_x * td->tile_w, x1 = x0 + td->tile_w;
    if (x1 > td->image_w) x1 = td->image_w;
    if (y1 > td->image_h) y1 = td->image_h;
    const float inv_w = 1.0f / td->image_w, inv_h = 1.0f / td->image_h;
    for (int y = y1 - 1; y >= y0; --y) {
        uint8_t *row = &td->image[(size_t)y * td->image_w * 3];
        for (int x = x0; x < x1; ++x) {
            v3 col = v3_make(0, 0, 0);
            for (int s = 0; s < td->spp; ++s) {
                float xi[4];
                myrand01_x4(td->state4, xi); /* :759 */
                float u = (xi[0] + (float)x) * inv_w, v = (xi[1] + (float)y) * inv_h;
                float dx, dy;
                random_in_unit_disk(&td->state, &dx, &dy); /* :760, :383 */
                v3 o, d;
                camera_ray(td->scene, u, v, dx, dy, &o, &d);
                col = v3_add(col, color(o, d, td)); /* :762 */
            }
            col = v3_scale(col, (float)(1.0f / td->spp)); /* :765 */
            col = v3_make(sqrtf(col.x), sqrtf(col.y), sqrtf(col.z)); /* :767 */
            row[3 * x + 0] = (uint8_t)(int)(col.x * 255.99f); /* :769-775 */
            row[3 * x + 1] = (uint8_t)(int)(col.y * 255.99f);
            row[3 * x + 2] = (uint8_t)(int)(col.z * 255.99f);
        }
    }
}

/* rayweek1.cpp:785-842 -- dynamic tile self-scheduling over std::thread; here pthreads + one atomic. */
typedef struct { thread_data td; int *next_tile; int num_tiles; } worker_arg;

static void *worker(void *p)
{
    worker_arg *a = p;
    int tile;
    while ((tile = __atomic_fetch_add(a->next_tile, 1, __ATOMIC_SEQ_CST)) < a->num_tiles) render_tile(tile, &a->td);
    return NULL;
}

/* benchmark() body (rayweek1.cpp:845-891) with runtime width/height/spp/threads.  threads <= 0 -> single-thread
 * branch with the MULTITHREADED==0 seeds (:880-881).  Returns total rays; *elapsed_s covers dispatch..join like :848,:891. */
ORC_API uint64_t orc_render(const orc_scene *s, uint8_t *rgb, int w, int h, int spp, int max_bounces, int threads, double *elapsed_s)
{
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    thread_data base;
    memset(&base, 0, sizeof(base));
    base.scene = s; base.image = rgb; base.image_w = w; base.image_h = h;
    base.tile_w = 32 < w ? 32 : w; base.tile_h = 32 < h ? 32 : h; /* :855-864 */
    base.spp = spp; base.max_bounces = max_bounces;
    int num_tiles = tiles_required(base.tile_w, w) * tiles_required(base.tile_h, h);
    uint64_t num_rays = 0;
    if (threads <= 0) {
        base.state = 10001;
        /* _mm_set_epi32(1001,1003,1005,1007): lane 0 = 1007 */
        base.state4[0] = 1007; base.state4[1] = 1005; base.state4[2] = 1003; base.state4[3] = 1001;
        for (int i = 0; i < num_tiles; ++i) render_tile(i, &base);
        num_rays = base.num_rays;
    } else {
        pthread_t *th = malloc(sizeof(pthread_t) * threads);
        worker_arg *args = malloc(sizeof(worker_arg) * threads);
        int next_tile = 0;
        for (int i = 0; i < threads; ++i) {
            args[i].td = base;
            args[i].td.state = 200u * i + 10001u; /* :801 */
            /* :802 _mm_set_epi32(200i+10001, +10003, +10005, +10007) -> lane 0 = 200i+10007 */
            args[i].td.state4[0] = 200u * i + 10007u; args[i].td.state4[1] = 200u * i + 10005u;
            args[i].td.state4[2] = 200u * i + 10003u; args[i].td.state4[3] = 200u * i + 10001u;
            args[i].next_tile = &next_tile; args[i].num_tiles = num_tiles;
            pthread_create(&th[i], NULL, worker, &args[i]);
        }
        for (int i = 0; i < threads; ++i) { pthread_join(th[i], NULL); num_rays += args[i].td.num_rays; }
        free(th); free(args);
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    if (elapsed_s) *elapsed_s = (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
    return num_rays;
}

/* Per-pixel replay (SURVEY.md 8f rank 4): the pixel loop of render_tile (:752-765) for ONE pixel from given generator
 * states -- jitter from the x4 stream, lens disk from the scalar stream, color() -- returning the float radiance sum over
 * spp samples and the rays traced.  Counterpart of ref_replay_pixels in oracle/ref_harness.cpp and of r1_replay_pixels. */
ORC_API void orc_replay_pixels(const orc_scene *s, int n, const int32_t *xy, int image_w, int image_h, int spp, int max_bounces,
                               const uint32_t *state_in, const uint32_t *state4_in, float *color_sum, uint32_t *rays_out)
{
    const float inv_w = 1.0f / image_w, inv_h = 1.0f / image_h;
    for (int k = 0; k < n; ++k) {
        thread_data td;
        memset(&td, 0, sizeof(td));
        td.scene = s; td.max_bounces = max_bounces;
        td.state = state_in[k];
        memcpy(td.state4, state4_in + 4 * k, 16);
        v3 col = v3_make(0, 0, 0);
        for (int smp = 0; smp < spp; ++smp) {
            float xi[4], dx, dy;
            myrand01_x4(td.state4, xi);
            float u = (xi[0] + (float)xy[2 * k]) * inv_w, v = (xi[1] + (float)xy[2 * k + 1]) * inv_h;
            random_in_unit_disk(&td.state, &dx, &dy);
            v3 o, d;
            camera_ray(s, u, v, dx, dy, &o, &d);
            col = v3_add(col, color(o, d, &td));
        }
        color_sum[3 * k] = col.x; color_sum[3 * k + 1] = col.y; color_sum[3 * k + 2] = col.z;
        rays_out[k] = (uint32_t)td.num_rays;
    }
}

/* Debug aid, counterpart of ref_trace_sample (oracle/ref_harness.cpp): one sample of one pixel, segment by segment. */
ORC_API int orc_trace_sample(const orc_scene *s, int x, int y, int image_w, int image_h, uint32_t state, const uint32_t *state4, int max_segments,
                             float *org, float *dir, int32_t *index, float *t, int32_t *scat_ok)
{
    thread_data td;
    memset(&td, 0, sizeof(td));
    td.scene = s; td.max_bounces = 50; td.state = state;
    memcpy(td.state4, state4, 16);
    float xi[4], dx, dy;
    myrand01_x4(td.state4, xi);
    float u = (xi[0] + (float)x) * (1.0f / image_w), v = (xi[1] + (float)y) * (1.0f / image_h);
    random_in_unit_disk(&td.state, &dx, &dy);
    v3 o, d;
    camera_ray(s, u, v, dx, dy, &o, &d);
    int n = 0;
    for (int depth = 0; n < max_segments; ++depth) {
        org[3 * n] = o.x; org[3 * n + 1] = o.y; org[3 * n + 2] = o.z; dir[3 * n] = d.x; dir[3 * n + 1] = d.y; dir[3 * n + 2] = d.z;
        hit_rec rec;
        int hit = scene_hit(s, o, d, 0.001f, FLT_MAX, &rec);
        index[n] = hit ? rec.index : -1; t[n] = hit ? rec.t : 0.0f; scat_ok[n] = 0;
        if (!hit || depth >= 50) { ++n; break; }
        v3 rs = v3_make(0, 0, 0), atten, nd;
        float ru = 0;
        int kind = s->kind[rec.index];
        if (kind == ORC_MAT_LAMBERT || kind == ORC_MAT_METAL) rs = random_in_unit_sphere(td.state4);
        if (kind == ORC_MAT_DIELECTRIC) ru = myrand01(&td.state);
        int ok = scatter_explicit(s, rec.index, d, rec.p, rec.normal, rs, ru, &atten, &nd);
        scat_ok[n] = ok; ++n;
        if (!ok) break;
        o = rec.p; d = nd;
    }
    return n;
}

/* ------------------------------------------------------------------ the device integrator (DESIGN.md section 3)
 * The GPU renderer does not run the reference's loop above: it keys a counter-based generator by (pixel, sample), multiplies the
 * throughput forward, and sums every sample into 64-bit fixed point.  Restated here from that formulation -- not from the
 * renderer's code -- so that a whole render can be compared bit for bit: sums, bytes and ray count.  The integer sums make the
 * result independent of the order samples finish in.  What a CPU cannot reproduce are the SFU approximations the renderer
 * samples the lens disk and the unit ball with; those come in as `points` (r1_sample_points), or, with points == NULL, are
 * evaluated in double precision with libm (statistically the same render, not the same bits). */

/* Stafford variant 13 */
static inline uint64_t keyed_mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
typedef struct { uint32_t k0, k1; } keyed_rng;
static inline uint64_t keyed_seed_mix(uint32_t seed) { return keyed_mix64(0x9E3779B97F4A7C15ull * ((uint64_t)seed + 1u)); }
static inline keyed_rng keyed_stream(uint32_t pixel, uint32_t sample, uint64_t seed_mix)
{
    const uint64_t z = keyed_mix64((((uint64_t)pixel << 32) | sample) ^ seed_mix);
    keyed_rng r = { (uint32_t)z, (uint32_t)(z >> 32) };
    return r;
}
static inline uint32_t keyed_draw(keyed_rng r, uint32_t i)
{
    uint32_t x = r.k0 + 0x9E3779B9u * i;
    x ^= x >> 16; x *= 0x21f0aaadu;
    x ^= r.k1;
    x ^= x >> 15; x *= 0x735a2d97u;
    x ^= x >> 15;
    return x;
}
static inline float keyed_rand01(keyed_rng r, uint32_t i) { return (float)(keyed_draw(r, i) >> 8) * 0x1p-24f; }
static inline float keyed_rand02(keyed_rng r, uint32_t i) { return (float)(keyed_draw(r, i) >> 8) * 0x1p-23f; }

ORC_API uint32_t orc_keyed_draw(uint32_t pixel, uint32_t sample, uint32_t seed, uint32_t i)
{
    return keyed_draw(keyed_stream(pixel, sample, keyed_seed_mix(seed)), i);
}

/* one sample's radiance -> 2^-24 fixed point as cvt.rni.sat.u32.f32 does it: round half to even, NaN and negatives 0,
 * values above 2^32 - 1 saturated */
static inline uint32_t quantise_radiance(float c)
{
    const float x = c * 16777216.0f;
    if (!(x > 0.0f)) return 0u;
    if (x >= 4294967295.0f) return 0xFFFFFFFFu;   /* the float nearest 2^32 - 1 is 2^32 */
    return (uint32_t)rintf(x);
}
/* a pixel's sum -> one byte: mean, gamma 2, (int)(c * 255.99f) (rayweek1.cpp:765-775 on the fixed-point sum) */
static inline uint8_t resolve_sum(uint64_t sum, float inv_spp)
{
    const float mean = ((float)sum * 0x1p-24f) * inv_spp;
    return (uint8_t)(int)(sqrtf(mean) * 255.99f);
}
ORC_API uint32_t orc_quantise_radiance(float c) { return quantise_radiance(c); }
ORC_API uint8_t orc_resolve(uint64_t sum, int spp) { return resolve_sum(sum, (float)(1.0f / spp)); }

/* the interleaved row-tile partition: tile k of row_tile rows belongs to rank k % world */
static inline int keyed_global_row(int lr, int row_tile, int rank, int world) { return ((lr / row_tile) * world + rank) * row_tile + lr % row_tile; }
ORC_API int orc_local_rows(int height, int row_tile, int rank, int world)
{
    if (row_tile <= 0) row_tile = 1;
    int rows = 0;
    while (keyed_global_row(rows, row_tile, rank, world) < height) ++rows;
    return rows;
}

/* the lens-disk point and the unit-ball samples in double precision: radius sqrt(u) / cbrt(u), azimuth a * pi */
static void disk_libm(keyed_rng r, float *px, float *py)
{
    const double rad = sqrt((double)keyed_rand01(r, 2)), a = (double)keyed_rand02(r, 3) * M_PI;
    *px = (float)(rad * cos(a));
    *py = (float)(rad * sin(a));
}
static v3 ball_libm(keyed_rng r, uint32_t i, float u)
{
    const float z = 1.0f - keyed_rand02(r, i + 1);
    const double a = (double)keyed_rand02(r, i + 2) * M_PI, rad = cbrt((double)u);
    const double rho = rad * sqrt(fmax(0.0, 1.0 - (double)z * z));
    return v3_make((float)(rho * cos(a)), (float)(rho * sin(a)), (float)(rad * z));
}

/* The rank's rows of a render (ascending global row, like r1_render): sums[local pixel][3], rgb[local pixel][3], *num_rays.
 * points: per local pixel, per sample 2 + 4 max_bounces floats as r1_sample_points writes them (disk x, y; then ru, ball x, y, z
 * per depth -- ru is drawn here, only the ball is taken from the table), or NULL.  Returns the number of local pixels. */
ORC_API int64_t orc_render_keyed(const orc_scene *s, int width, int height, int spp, int max_bounces, uint32_t seed, int rank, int world,
                                 int row_tile, const float *points, uint64_t *sums, uint8_t *rgb, uint64_t *num_rays)
{
    const int built = g_as_built;
    g_as_built = 1;                        /* the renderer's association throughout */
    if (row_tile <= 0) row_tile = 1;
    const int rows = orc_local_rows(height, row_tile, rank, world);
    const size_t per_sample = 2 + 4 * (size_t)max_bounces;
    const uint64_t seed_mix = keyed_seed_mix(seed);
    const float inv_w = 1.0f / width, inv_h = 1.0f / height, inv_spp = (float)(1.0f / spp);
    uint64_t rays = 0;
    for (int lr = 0; lr < rows; ++lr) {
        const int y = keyed_global_row(lr, row_tile, rank, world);
        for (int x = 0; x < width; ++x) {
            const size_t lp = (size_t)lr * width + x;
            uint64_t acc[3] = { 0, 0, 0 };
            for (int smp = 0; smp < spp; ++smp) {
                const keyed_rng key = keyed_stream((uint32_t)y * (uint32_t)width + (uint32_t)x, (uint32_t)smp, seed_mix);
                const float *pt = points ? points + (lp * (size_t)spp + (size_t)smp) * per_sample : NULL;
                /* primary ray: jitter from draws 0 and 1, lens disk from draws 2 and 3 */
                const float u = (keyed_rand01(key, 0) + (float)x) * inv_w, v = (keyed_rand01(key, 1) + (float)y) * inv_h;
                float px, py;
                if (pt) { px = pt[0]; py = pt[1]; }
                else disk_libm(key, &px, &py);
                v3 o, d;
                camera_ray(s, u, v, px, py, &o, &d);
                v3 thr = v3_make(1, 1, 1), contrib = v3_make(0, 0, 0);
                for (int depth = 0;; ) {
                    ++rays;
                    hit_rec rec;
                    if (!scene_hit(s, o, d, 0.001f, FLT_MAX, &rec)) {
                        const float t = 0.5f * (d.y + 1.0f), it = 1.0f - t;
                        contrib = v3_mul(thr, v3_make(fmaf(t, 0.5f, it), fmaf(t, 0.7f, it), fmaf(t, 1.0f, it)));
                        break;
                    }
                    if (depth >= max_bounces) break;                       /* black, no draw past the cap */
                    const uint32_t draw0 = 4u + 3u * (uint32_t)depth;
                    const float ru = keyed_rand01(key, draw0);
                    const v3 rs = pt ? v3_make(pt[2 + 4 * depth + 1], pt[2 + 4 * depth + 2], pt[2 + 4 * depth + 3]) : ball_libm(key, draw0, ru);
                    v3 atten, nd;
                    if (!scatter_explicit(s, rec.index, d, rec.p, rec.normal, rs, ru, &atten, &nd)) break;   /* black */
                    thr = v3_mul(thr, atten);
                    o = rec.p; d = nd; ++depth;
                }
                acc[0] += quantise_radiance(contrib.x);
                acc[1] += quantise_radiance(contrib.y);
                acc[2] += quantise_radiance(contrib.z);
            }
            for (int c = 0; c < 3; ++c) {
                if (sums) sums[3 * lp + c] = acc[c];
                if (rgb) rgb[3 * lp + c] = resolve_sum(acc[c], inv_spp);
            }
        }
    }
    g_as_built = built;
    if (num_rays) *num_rays = rays;
    return (int64_t)rows * width;
}

/* ------------------------------------------------------------------ RNG known-answer entry points */

ORC_API uint32_t orc_xorshift32(uint32_t *state) { return xorshift32(state); }
ORC_API float orc_myrand01(uint32_t *state) { return myrand01(state); }
ORC_API float orc_myrand02(uint32_t *state) { return myrand02(state); }
ORC_API void orc_myrand01_x4(uint32_t *state4, float *out) { myrand01_x4(state4, out); }
ORC_API void orc_random_in_unit_sphere(uint32_t *state4, float *out)
{
    v3 p = random_in_unit_sphere(state4);
    out[0] = p.x; out[1] = p.y; out[2] = p.z;
}
ORC_API void orc_random_in_unit_disk(uint32_t *state, float *out) { random_in_unit_disk(state, &out[0], &out[1]); }
