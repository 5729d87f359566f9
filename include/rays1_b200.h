/*
 * rays1_b200.h -- C ABI of the B200-native Rays1 trace loop (librays1_b200.so).
 *
 * The reference (montib/rays1bench) has no FFI layer: its boundary for this path is four free C++ functions in one
 * translation unit (create_small/medium/large_scene, benchmark) plus main().  BASELINE.json's north_star asks for the
 * scene builders to feed device buffers "through a thin C-ABI layer called from the C++ host code"; this header is
 * that layer.  Part 1 is the device-facing ABI the host code binds; part 2 is the reference-shaped host surface
 * exported with C linkage so that non-C++ callers (ctypes in tests/ and bench.py) can drive the same code the
 * drop-in executable runs.  Plain pointers and sizes only; every function that can fail returns 0 on success and a
 * negative code otherwise, with the message available from r1_last_error().  There is NO CPU fallback: every
 * compute entry point fails with R1_ERR_CUDA when no sm_100 device / driver is present.
 *
 * file:line citations are relative to /root/reference/.
 */
#ifndef RAYS1_B200_H
#define RAYS1_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R1_ABI_VERSION 2

enum {
    R1_OK = 0,
    R1_ERR_ARG = -1,    /* bad argument */
    R1_ERR_STATE = -2,  /* call order (e.g. render before commit) */
    R1_ERR_CUDA = -3,   /* CUDA runtime / driver error, or no device */
    R1_ERR_LIMIT = -4   /* scene larger than the on-chip staging limit */
};

/* Material tags: replace the reference's virtual Material hierarchy (src/latest/rayweek1.cpp:131-136, 396-512). */
enum { R1_MAT_NONE = -1, R1_MAT_LAMBERT = 0, R1_MAT_METAL = 1, R1_MAT_DIELECTRIC = 2 };

/* Kernel variants measured against each other (north_star (2)). */
enum {
    R1_VARIANT_MEGAKERNEL = 0, /* default: the fastest megakernel for the scene -- R1_VARIANT_MEGAKERNEL_TENSOR for scan-heavy scenes
                                  that fit its shared-memory operand (256 .. 768 spheres), R1_VARIANT_MEGAKERNEL_PACKED otherwise
                                  (and whenever blocks_per_sm / threads are given: they tune the packed kernel) */
    R1_VARIANT_WAVEFRONT = 1,  /* generate / intersect / shade kernels over compacted ray queues, CUDA-graph WHILE loop */
    R1_VARIANT_MEGAKERNEL_SCALAR = 2, /* A/B: megakernel with a per-lane scalar FFMA scan */
    R1_VARIANT_MEGAKERNEL_COOP = 3,   /* A/B: megakernel with the warp-cooperative scan (quads share sphere loads, candidates
                                         resolved through a per-warp shared-memory queue) */
    R1_VARIANT_MEGAKERNEL_DEFERRED = 4, /* A/B: per-lane packed scan, candidates deferred to a per-warp queue and resolved once per
                                         scan with every lane busy */
    R1_VARIANT_MEGAKERNEL_DUAL = 5,    /* A/B: two paths per lane share every sphere load (768 threads x 80 registers) */
    R1_VARIANT_MEGAKERNEL_TENSOR = 6,  /* persistent threads, per-lane path state machine, the filter as a split-TF32 GEMM on the tensor
                                         cores (tcgen05.mma, accumulators in TMEM), 128 rays x 64 spheres per instruction; scenes of up
                                         to 768 spheres */
    R1_VARIANT_MEGAKERNEL_PACKED = 7,  /* persistent threads, per-lane path state machine, per-lane packed f32x2 (FFMA2) filter */
    /* 8 stays unassigned: callers built against earlier versions of this header may rely on it being refused as an unknown
       variant (R1_ERR_ARG), and the ABI tests use it as their example of one. */
    R1_VARIANT_MEGAKERNEL_TENSOR_STREAM = 9, /* the filter of R1_VARIANT_MEGAKERNEL_TENSOR with the sphere operand streamed through a
                                               ring of 128-sphere chunks in shared memory, shared by the CTA's ray groups: scenes of
                                               any size; threads / 128 = ray groups (1 .. 4, default 4) */
    /* 10 stays unassigned as well (tests use it as an unknown variant). */
    R1_VARIANT_MEGAKERNEL_BVH = 11 /* persistent threads, per-lane path state machine, nearest hit by a per-lane stack traversal of a
                                      binned-SAH BVH2 (leaves of <= 4 spheres, boxes widened per ray so that no sphere the exact test
                                      accepts is skipped): scenes of any size, same bytes as every other variant.  The tree is built
                                      on the host and uploaded on the first BVH render or trace on a device: that call's
                                      elapsed_seconds includes it, its kernel_ms does not.  threads: 512, 768 or 1024 (default) */
};

typedef struct r1_scene r1_scene; /* opaque: host SoA + per-device buffers */

/* Replaces RESULT (src/common/common.h:36-45) with the extra fields the roofline needs. */
typedef struct r1_result {
    double elapsed_seconds; /* host steady_clock: call entry -> result bytes where the caller asked for them */
    double kernel_ms;       /* CUDA events around the trace kernel(s) + resolve on the launching stream */
    double trace_ms;        /* CUDA events around the dominant trace kernel alone */
    uint64_t num_rays;      /* the reference's counting rule: one per color() call (rayweek1.cpp:517) */
    uint64_t num_samples;   /* pixels rendered by this call x spp */
    uint32_t launches;      /* kernels launched by this call */
    uint32_t n_units;       /* (pixel, sample-chunk) work units handed out */
} r1_result;

typedef struct r1_render_params {
    int32_t width, height;   /* full image; SCREEN_W / SCREEN_H (common.h:19-20) */
    int32_t spp;             /* NUM_SAMPLES_PER_PIXEL (common.h:23-28) */
    int32_t max_bounces;     /* MAX_BOUNCES (common.h:18) */
    int32_t variant;         /* R1_VARIANT_* */
    uint32_t seed;           /* global seed of the counter-based RNG */
    int32_t rank, world;     /* this call renders the row tiles k with k % world == rank (world = 1: all rows) */
    int32_t row_tile;        /* rows per interleaved tile; <= 0 -> 1 (single rows balance the ranks best) */
    int32_t blocks_per_sm;   /* persistent CTAs per SM; <= 0 -> tuned default */
    int32_t threads;         /* threads per CTA: 512, 768 or 1024; <= 0 -> tuned default */
    int32_t device;          /* CUDA device to run on (must have been committed); < 0 -> device of the last commit */
} r1_render_params;

/* ---- part 1: device-facing ABI ------------------------------------------------------------------------------ */

int r1_abi_version(void);
const char *r1_last_error(void);
/* Number of CUDA devices visible, or a negative error. */
int r1_device_count(void);

/* Scene storage: replaces SphereSOA + Camera + Scene (soa_sphere.h:14-69, rayweek1.cpp:364-394, 539-549). */
r1_scene *r1_scene_create(uint32_t capacity_hint);
void r1_scene_destroy(r1_scene *scene);
/* Camera::init (rayweek1.cpp:366-379). */
int r1_scene_set_camera(r1_scene *scene, const float lookfrom[3], const float lookat[3], const float vup[3], float vfov_deg,
                        float aspect, float aperture, float focus_dist);
/* Installs the 22 camera constants directly, in the order r1_scene_get_camera returns them -- for callers that already hold
 * camera constants of their own (r1_scene_set_camera itself reproduces the reference's constants bit for bit: it evaluates
 * Camera::init the way gcc -ffast-math folds it for the reference's builders). */
int r1_scene_set_camera_raw(r1_scene *scene, const float cam[22]);
/* Host only (no device needed): the 22 constants r1_scene_set_camera installs for these arguments, in r1_scene_get_camera's order --
 * r1_scene_set_camera is this function followed by r1_scene_set_camera_raw.  For r1_scene_move_camera.  R1_ERR_ARG for a null
 * pointer. */
int r1_camera_constants(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov_deg, float aspect, float aperture,
                        float focus_dist, float out[22]);
/* SphereSOA::add (soa_sphere.cpp:70-85): stores radius*radius and radius > 0 ? 1/radius : 0.  Metal's `param` is the
 * fuzz (clamped to <= 1 as the Metal ctor does, rayweek1.cpp:424), Dielectric's the refraction index.  Returns the
 * sphere's index (>= 0) or a negative error. */
int r1_scene_add_sphere(r1_scene *scene, float cx, float cy, float cz, float radius, int mat_kind, float r, float g, float b,
                        float param);
/* Pads with the reference's placeholder (radius 0 at 999999999, material none) to a multiple of `multiple`
 * (rayweek1.cpp:575-576; SIMD_WIDTH = 8 there). */
int r1_scene_pad(r1_scene *scene, uint32_t multiple);
uint32_t r1_scene_count(const r1_scene *scene);
/* Host copies of the SoA arrays, `count` entries each (albedo: 3 per sphere) -- for bit-parity checks.  They describe the scene as
 * built on the host: r1_scene_move_spheres and r1_scene_set_materials change a device's records only. */
int r1_scene_get_soa(const r1_scene *scene, float *cx, float *cy, float *cz, float *radius_sq, float *inv_radius, int32_t *kind,
                     float *albedo, float *param);
/* out[22] = origin, lower-left corner, horizontal, vertical, u, v, w (3 each), lens radius (rayweek1.cpp:388-393).  The host's
 * camera: r1_scene_move_camera changes a device's camera only. */
int r1_scene_get_camera(const r1_scene *scene, float *out);
/* Uploads the scan / shading buffers to CUDA device `device` (replicated per device; may be called once per device). */
int r1_scene_commit(r1_scene *scene, int device);

/* The hot path: render_tile + color + hit + scatter for every pixel x sample of this rank's rows
 * (rayweek1.cpp:722-782, 515-536, 152-339, 396-512), RGB8 out, row 0 = BOTTOM of the picture (rayweek1.cpp:750).
 *
 * r1_render: host buffer.  rgb_host holds the rank's rows packed top-of-partition first in ascending global row order
 * (world = 1: the whole width*height*3 image); the device->host copy is inside elapsed_seconds. */
int r1_render(r1_scene *scene, const r1_render_params *params, uint8_t *rgb_host, r1_result *result);
/* r1_render_device: device buffers, asynchronous on `cuda_stream` (a cudaStream_t; NULL = default stream).
 * d_rgb: r1_local_pixels()*3 bytes; d_num_rays: one uint64, zeroed and then accumulated by the kernels.  The caller
 * owns both (e.g. torch CUDA tensors that a following NCCL gather / reduce reads).  result->num_rays is NOT filled. */
int r1_render_device(r1_scene *scene, const r1_render_params *params, void *d_rgb, void *d_num_rays, void *cuda_stream,
                     r1_result *result);
/* Blocks until the last r1_render_device of this scene on `device` (< 0: device of the last commit) has finished and
 * fills kernel_ms / trace_ms (CUDA events recorded on the launching stream), launches, n_units, num_samples. */
int r1_render_wait(r1_scene *scene, int device, r1_result *result);
/* A batch of views: K = n_views images of one scene state in one persistent launch and one resolve (two above 2^31 batch
 * pixels: the resolve's index is 32-bit, so it runs in pieces of at most 2^31 pixels).  View v is byte for byte what
 * r1_scene_move_camera(cams + 22 v) followed by r1_render_sums with params->seed = seeds[v] gives on that device: the same pixel
 * sums, bytes and rank rows; num_rays is the sum of those K renders' counts.  The batch renders the device's current records
 * (moved spheres, changed materials) and does NOT change the device's camera.
 * cams: n_views x 22 floats (r1_scene_get_camera's order; r1_camera_constants computes them).  seeds: n_views, or NULL for
 * params->seed in every view.  Both are HOST arrays, read before the call returns.
 * Outputs are view-major, each view laid out as r1_render lays out one image: rgb_host n_views x r1_local_pixels() x 3 bytes,
 * sums_host (NULL: not returned) n_views x r1_local_pixels() x 3 uint64 as r1_render_sums returns them.
 * Variants: R1_VARIANT_MEGAKERNEL (resolved as for r1_render), PACKED, TENSOR, TENSOR_STREAM and BVH (with a single render's tree
 * rules); the A/B variants, WAVEFRONT and tuning (threads or blocks_per_sm > 0) are refused with R1_ERR_ARG.  Before any device
 * is looked up: bad params, n_views == 0, a null cams or output pointer: R1_ERR_ARG; n_views x r1_local_pixels() >= 2^32 - 1, or
 * too many samples: R1_ERR_LIMIT.  result->n_units is 0 (the batch's kernels take samples, not units).
 * r1_render_views_device: d_rgb as rgb_host, d_num_rays one uint64; asynchronous on cuda_stream like r1_render_device (num_rays
 * not filled; r1_render_wait completes it).  The cameras are copied on the stream, so a batch already enqueued keeps its own. */
int r1_render_views(r1_scene *scene, const r1_render_params *params, uint32_t n_views, const float *cams, const uint32_t *seeds,
                    uint8_t *rgb_host, uint64_t *sums_host, r1_result *result);
int r1_render_views_device(r1_scene *scene, const r1_render_params *params, uint32_t n_views, const float *cams, const uint32_t *seeds,
                           void *d_rgb, void *d_num_rays, void *cuda_stream, r1_result *result);
/* Diagnostics: how many times the wavefront variant had to (re)build its CUDA-graph WHILE loop on `device` -- the
 * instantiated graph is cached and re-launched while the render arguments stay the same.  Negative on error. */
int r1_wavefront_graph_builds(int device);
/* Rows / pixels owned by `rank` under the interleaved row-tile partition, and the global row of local row `lr`. */
int64_t r1_local_rows(int height, int row_tile, int rank, int world);
int64_t r1_local_pixels(int width, int height, int row_tile, int rank, int world);
int r1_global_row(int local_row, int row_tile, int rank, int world);

/* Multi-GPU epilogue on the gathering device: `d_gathered` holds `world` slices of `stride` bytes, slice r = rank r's
 * packed local rows; writes the full width*height*3 image (row 0 = bottom) to d_out.  Asynchronous on cuda_stream. */
int r1_deinterleave_rows(int device, const void *d_gathered, uint64_t stride, void *d_out, int width, int height, int row_tile,
                         int world, void *cuda_stream);

/* Parity entry points (host buffers, n rays each, xyz interleaved) -- the device functions the kernels use. */
/* Hitable::hit (rayweek1.cpp:152-339); index = -1 on a miss.  dir must be unit length (Ray ctor, :104-108).  `variant` picks
 * the filter: R1_VARIANT_MEGAKERNEL resolves as in r1_render; SCALAR, COOP, DEFERRED and PACKED run that kernel's scan;
 * TENSOR runs the filter of megakernel_tc3 (128-sphere accumulator chunks, the short last chunk included) and returns
 * R1_ERR_LIMIT above 768 spheres; TENSOR_STREAM runs the streamed filter of megakernel_tcs and BVH the BVH traversal of
 * megakernel_bvh at any sphere count, while every other variant returns R1_ERR_LIMIT above 4096 (they stage the scene in shared memory); WAVEFRONT and DUAL have no per-ray
 * kernel and return R1_ERR_ARG.  t_min must be >= 2^-24
 * (renders use 0.001): below it the exact test's floored square root and the unsigned root keys of COOP and DEFERRED can differ
 * from Hitable::hit, so a smaller t_min or a NaN returns R1_ERR_ARG before any device is touched.  For every finite origin and
 * scene every variant returns Hitable::hit's records bit for bit: the expanded filters hold their error bounds for |c|^2 and |o|^2
 * below 2^120 and flag every sphere that can be hit beyond that (DESIGN.md section 4.1), so far scenes are slow, not wrong. */
int r1_trace_rays(r1_scene *scene, int n, const float *org, const float *dir, float t_min, float t_max, int variant,
                  int32_t *index, float *t, float *p, float *normal);
/* Name of the trace kernel `variant` resolves to for this scene with default tuning ("megakernel_tc3", "megakernel_tcs", "megakernel_bvh",
 * "megakernel_pool", ...);
 * static storage. */
const char *r1_kernel_name(r1_scene *scene, int variant);
/* Host only (no device needed): the sphere operand of the tensor-core filter for this scene -- n32 rows (sphere count padded to
 * 32) of 128 bytes: 32 TF32 words {hi x 11 | hi x 11 | lo x 10} of the 11 lifted features in the tcgen05 K-major no-swizzle
 * layout, byte offset of (row r, word k) = (r / 8) * 1024 + (k / 4) * 128 + (r % 8) * 16 + (k % 4) * 4.  out = NULL: only
 * *n32_out is set.  R1_ERR_LIMIT for empty scenes and above 768 spheres.  Built from the host scene: spheres moved on a device by
 * r1_scene_move_spheres are not seen here (r1_scene_export_device returns a device's operand). */
int r1_tensor_operand(const r1_scene *scene, void *out, uint64_t out_bytes, uint32_t *n32_out);
/* Host only (no device needed): the BVH of R1_VARIANT_MEGAKERNEL_BVH for this scene, built now if it is not cached yet (adding
 * spheres drops the cached tree).  nodes: n_nodes x 64 bytes {float lo0[3], hi0[3], lo1[3], hi1[3]; int32 child[2]; float diag[2]},
 * node 0 = root; child >= 0: inner node, child < 0: leaf with ~child = first record << 3 | count (1 .. 4), child = -1: none;
 * diag = bound on the box's diagonal.  leaves: n_leaf_records x 32 bytes {float cx, cy, cz, radius_sq (the scene's values); int32
 * sphere index; 3 x 0}, ascending index within a leaf.  Spheres with inv_radius == 0 are not in the tree.  depth = deepest inner
 * node (root = 1), at most 64.  A NULL buffer skips that copy (the counts are still returned).  Built from the host scene: spheres
 * moved on a device by r1_scene_move_spheres are not seen here (r1_bvh_export_device returns a device's tree). */
int r1_bvh_export(const r1_scene *scene, void *nodes, uint64_t nodes_bytes, void *leaves, uint64_t leaves_bytes, uint32_t *n_nodes,
                  uint32_t *n_leaf_records, uint32_t *depth);
/* Builders of r1_scene_build_bvh.  HOST: the tree r1_bvh_export returns (binned SAH, built on the host and cached in the scene).
 * DEVICE: a linear BVH (Morton codes, radix sort, Karras' radix tree, leaves of <= 4 spheres) built on the device from the
 * committed scene; a pure function of the scene, in r1_bvh_export's layout, depth at most 62 (DESIGN.md section 4.9). */
enum { R1_BVH_BUILD_HOST = 0, R1_BVH_BUILD_DEVICE = 1 };
/* Builds the BVH of R1_VARIANT_MEGAKERNEL_BVH for `device` now (< 0: device of the last commit) and makes it the tree that BVH
 * renders and traces there use, replacing any tree the device holds.  HOST: the host tree (cached in the scene) uploaded;
 * DEVICE: the linear BVH, built on the device from the committed scene.  Synchronous.  device_ms (optional): CUDA events around
 * the device work (the upload for HOST; every kernel and the sort for DEVICE).  R1_ERR_ARG for a null scene, an unknown builder
 * or (DEVICE) a sphere that can be hit with a non-finite centre or radius_sq; R1_ERR_STATE if the scene is not committed there or
 * its spheres changed since; R1_ERR_LIMIT from 2^28 spheres that can be hit.  A re-commit drops the device's tree: the next BVH
 * render or trace builds and uploads the host tree again. */
int r1_scene_build_bvh(r1_scene *scene, int device, int builder, double *device_ms);
/* The tree `device` (< 0: device of the last commit) holds, in r1_bvh_export's layout; R1_ERR_STATE if it holds none, R1_ERR_ARG
 * for a null scene or a buffer smaller than the tree.  A NULL buffer skips that copy (the counts are still returned). */
int r1_bvh_export_device(r1_scene *scene, int device, void *nodes, uint64_t nodes_bytes, void *leaves, uint64_t leaves_bytes,
                         uint32_t *n_nodes, uint32_t *n_leaf_records, uint32_t *depth);
/* Moves spheres first .. first + n - 1 of the scene committed on `device` (< 0: device of the last commit), for animated scenes.
 * d_centre: n x 3 floats (xyz interleaved).  d_radius: n floats, or NULL to keep the radii.  Both are DEVICE pointers on that device.
 * The device's records of those spheres become exactly what r1_scene_commit writes for a scene with these values (radius_sq =
 * radius * radius and inv_radius = radius > 0 ? 1 / radius : 0, as r1_scene_add_sphere derives them; materials are kept).
 * If the device holds a BVH, it is refitted in place (same topology, new boxes and leaf records; DESIGN.md section 4.10).
 * Runs on cuda_stream (NULL = legacy default stream) and returns when that work is done.
 * device_ms (optional): CUDA events around the device work.
 * Only that device changes.  The host scene keeps its values: r1_scene_get_soa, r1_tensor_operand and r1_bvh_export still describe
 * the committed scene, and a re-commit restores its records there and drops the device's tree.  After a move, a BVH render or trace
 * on a device without a tree is refused (R1_ERR_STATE) instead of uploading the host tree, and so is r1_scene_build_bvh with
 * R1_BVH_BUILD_HOST; R1_BVH_BUILD_DEVICE builds from the moved records.
 * R1_ERR_ARG: null scene; first + n > count (no wrap in uint32); n > 0 with a null d_centre; a sphere whose new radius changes
 *   whether it can be hit (inv_radius != 0 before and after); a sphere that can be hit with a non-finite centre or radius_sq
 *   (the rule of the device builder).  Nothing is written in any of these cases.
 * R1_ERR_STATE: not committed there, or the spheres changed on the host since the commit.
 * Any finite position traces and renders like the oracle: spheres with |c|^2 >= 2^120 are encoded as candidates of every ray
 * (DESIGN.md section 4.1). */
int r1_scene_move_spheres(r1_scene *scene, int device, uint32_t first, uint32_t n, const float *d_centre, const float *d_radius,
                          void *cuda_stream, double *device_ms);
/* Installs 22 camera constants (r1_scene_get_camera's order; r1_camera_constants computes them) for renders and parity calls on
 * `device` (< 0: device of the last commit), for animated scenes.  No upload: the constants reach a kernel by value when it is
 * launched, so a render already enqueued with r1_render_device keeps the camera it was launched with, and the next one uses the new
 * camera.  The wavefront variant's cached graph is rebuilt once for a new camera (r1_wavefront_graph_builds).  Values are not
 * checked, as r1_scene_set_camera_raw does not check them.
 * State rules (shared with r1_scene_set_materials; DESIGN.md section 4.11): only that device changes; the host scene keeps its
 * camera (r1_scene_get_camera) and a re-commit restores it there; renders of every variant, r1_get_ray, r1_scatter and
 * r1_replay_pixels on that device see the new constants; r1_trace_rays reads neither the camera nor the materials.
 * R1_ERR_ARG: null scene or cam.  R1_ERR_STATE: not committed there, or the spheres changed on the host since the commit. */
int r1_scene_move_camera(r1_scene *scene, int device, const float cam[22]);
/* Sets the materials of spheres first .. first + n - 1 of the scene committed on `device` (< 0: device of the last commit), for
 * animated scenes.  d_kind: n int32 (R1_MAT_*), d_albedo: n x 3 floats (rgb interleaved), d_param: n floats (Metal fuzz, Dielectric
 * ior), all DEVICE pointers on that device; any one may be NULL to keep that field.  The device's shade records of those spheres
 * become exactly what r1_scene_commit writes for a scene whose spheres were added with the resulting (kind, albedo, param): Metal's
 * param clamped to <= 1 as r1_scene_add_sphere does (a NaN fuzz becomes 1; a kept param is clamped when it meets a new Metal kind),
 * 1 / ior and the Schlick r0 of dielectrics in IEEE float (where an ior makes them NaN -- NaN or infinite ior -- the NaN's bits may
 * differ from the host's); inv_radius is kept.  Geometry and BVH are untouched: the scan, exact and
 * tensor-operand records stay, a tree the device holds stays valid, and a BVH render on a device without a tree still uploads the
 * host tree (unless spheres were moved there).
 * Runs on cuda_stream (NULL = legacy default stream) and returns when that work is done.  device_ms (optional): CUDA events around
 * the device work.
 * State rules: those of r1_scene_move_camera; r1_scene_get_soa still returns the host's materials and r1_scene_export_device the new
 * shade records.
 * R1_ERR_ARG: null scene; first + n > count (no wrap in uint32); n > 0 with all three pointers NULL; a kind outside -1 .. 2;
 *   R1_MAT_NONE for a sphere that can be hit (inv_radius != 0) -- the device form of r1_scene_add_sphere's "radius > 0 needs a
 *   material" rule, which differs from it only for radius +inf (inv_radius 0: never hit, so NONE is accepted here).  Nothing is
 *   written in any of these cases.
 * R1_ERR_STATE: not committed there, or the spheres changed on the host since the commit. */
int r1_scene_set_materials(r1_scene *scene, int device, uint32_t first, uint32_t n, const int32_t *d_kind, const float *d_albedo,
                           const float *d_param, void *cuda_stream, double *device_ms);
/* The device's scene records ([scan | exact | shade | tensor operand], the layout r1_scene_commit uploads), for parity checks:
 * *bytes = the layout's size.  out = NULL: only *bytes is set.  R1_ERR_ARG for a null scene or out_bytes < *bytes, R1_ERR_STATE if
 * the scene is not committed to `device` (< 0: device of the last commit). */
int r1_scene_export_device(r1_scene *scene, int device, void *out, uint64_t out_bytes, uint64_t *bytes);
/* Values of the tensor-core FILTER (R1_VARIANT_MEGAKERNEL_TENSOR) for n rays against every sphere: e[ray * n32 + sphere], n32 =
 * sphere count padded to 32; the filter flags a sphere iff the sign bit of e is clear, and must flag every sphere Hitable::hit's
 * discriminant test (rayweek1.cpp:192-204) accepts.  layout must be 0 (the renderer's operand layout); any other value returns
 * R1_ERR_ARG before any device is touched. */
int r1_filter_probe(r1_scene *scene, int n, const float *org, const float *dir, int layout, float *e);
/* Material::scatter (rayweek1.cpp:403-409, 427-433, 470-511) with the random inputs injected: rand_sphere is the
 * unit-ball sample, rand_u the [0,1) uniform. */
int r1_scatter(r1_scene *scene, int n, const float *dir_in, const float *p, const float *normal, const int32_t *index,
               const float *rand_sphere, const float *rand_u, int32_t *ok, float *atten, float *dir_out);
/* Camera::getRay (rayweek1.cpp:381-386) with the lens-disk sample injected (disk: 2 per ray). */
int r1_get_ray(r1_scene *scene, int n, const float *su, const float *tv, const float *disk, float *org, float *dir);
/* Replay (parity): the pixel loop of render_tile (rayweek1.cpp:752-765) for n pixels, one per thread, driven by the
 * REFERENCE's xorshift streams from the given states (state: scalar stream, state4: the four lanes of the x4 stream) with
 * its rejection loops, through the production scan / scatter code.  color_sum = float radiance summed over spp samples
 * (3 per pixel), num_rays = color() calls per pixel.  Compared with recorded runs of the reference's own color(). */
int r1_replay_pixels(r1_scene *scene, int n, const int32_t *xy, int width, int height, int spp, int max_bounces,
                     const uint32_t *state, const uint32_t *state4, float *color_sum, uint32_t *num_rays);
/* First `n` draws of the counter-based generator for (pixel, sample, seed): raw u32 -- for distribution tests. */
int r1_rng_draws(uint32_t pixel, uint32_t sample, uint32_t seed, int n, uint32_t *out);
/* The random points a render draws for n (global pixel y * width + x, sample) keys under the global `seed`, through the
 * renderer's own generator and samplers (SFU approximations included).  out: n x (2 + 4 * bounces) floats, per key the
 * lens-disk point (x, y), then for every depth d < bounces (ru, rs.x, rs.y, rs.z): ru = the [0,1) uniform of draw 4 + 3 d,
 * rs = the unit-ball sample of that bounce.  With these, a CPU restatement of the integrator reproduces a render bit for bit.
 * 0 <= bounces <= 1024. */
int r1_sample_points(int n, const uint32_t *pixel, const uint32_t *sample, uint32_t seed, int bounces, float *out);
/* r1_render, plus the rank's fixed-point pixel sums the bytes were resolved from: sums = r1_local_pixels() x 3 uint64
 * (r, g, b) in local pixel order, each the sum over the pixel's samples of round(radiance * 2^24), saturated to 32 bits. */
int r1_render_sums(r1_scene *scene, const r1_render_params *params, uint64_t *sums, uint8_t *rgb_host, r1_result *result);
/* FP32 FMA throughput microbenchmark on `device`: independent FFMA chains (packed = 0) or FFMA2 (packed = 1).
 * Returns TFLOP/s (FMA = 2) in *tflops.  *sm_mhz_est (optional) = clock64 ticks of one thread / elapsed time: a rough
 * cross-check only -- on the B200 boxes of this project clock64 did not tick at the SM clock (it read ~300 MHz while
 * nvidia-smi showed 1965 MHz under the same load), so bench.py reports the nvidia-smi clock instead. */
int r1_fma_peak(int device, int packed, double *tflops, double *sm_mhz_est);
/* TMEM read throughput microbenchmark: `warps` warps per SM (1 CTA per SM) each read 32 lanes x 32 columns per tcgen05.ld.
 * Returns bytes per second per SM -- the bound of the tensor-core filter (4 bytes per ray-sphere test leave TMEM). */
int r1_tmem_read_peak(int device, int warps, double *bytes_per_second_per_sm);

/* ---- part 2: the reference's host surface, C linkage ------------------------------------------------------------- */

/* Workload the reference fixes at compile time (common.h:3-31), runtime here. Any field <= 0 keeps its default:
 * 1280 x 720, 250 spp, 50 bounces, 1 GPU, megakernel. */
int r1_host_configure(int width, int height, int spp, int max_bounces, int variant, int n_gpus, uint32_t seed);
/* Non-zero: benchmark() does not print its report block (callers that print their own). */
int r1_host_set_quiet(int quiet);
/* create_small_scene / create_medium_scene / create_large_scene (rayweek1.cpp:552, 582, 654) and the synthetic
 * 4096-sphere stress scene (SURVEY.md 8d config 5) by name: "small" | "medium" | "large" | "synth4096".
 * commit != 0 also uploads the device buffers to GPUs 0 .. n_gpus-1 (what the C++ builders always do); commit == 0
 * builds the host SoA only.  Returns a Scene* (see rays1_host.h) or NULL (r1_last_error() says why). */
void *r1_host_create_scene(const char *name, int commit);
/* Scene from a text description (SURVEY.md 8f: scenes beyond the three hard-coded builders).  One statement per line:
 *   camera <from.xyz> <at.xyz> <vfov_deg> <aperture> <focus_dist>
 *   sphere <c.xyz> <radius> lambert <r> <g> <b> | metal <r> <g> <b> <fuzz> | dielectric <ior> | none
 * Padded to a multiple of 8 like the built-in scenes.  Returns a Scene* or NULL. */
void *r1_host_create_scene_from_file(const char *path, int commit);
/* The r1_scene inside a host Scene (borrowed). */
r1_scene *r1_host_scene_handle(void *scene);
/* benchmark(scene, pixels, write_tga, scene_name) (rayweek1.cpp:845-927): renders, prints the reference's report block,
 * deletes the scene (in every case, also on error), optionally writes out_<name>.tga (which swaps R/B in `pixels` in place,
 * common.h:108-114).  `pixels_bytes` is the size of the caller's buffer: R1_ERR_ARG if it is smaller than the configured
 * width * height * 3.  CUDA / NCCL failures come back as a negative code (the C++ benchmark() of rays1_host.h exits instead,
 * like the reference's surface without error paths would). */
int r1_host_benchmark(void *scene, uint8_t *pixels, uint64_t pixels_bytes, int write_tga, const char *scene_name, double *elapsed_seconds,
                      uint64_t *num_rays, double *kernel_ms);
void r1_host_destroy_scene(void *scene);
/* tga_write_rgb24 (common.h:86-122): 18-byte header, type 2, 24 bpp, bottom-left origin; swaps R and B in `pixels`.
 * R1_ERR_ARG if pixels_bytes < width * height * 3 or a dimension does not fit the 16-bit header fields. */
int r1_host_write_tga(const char *filename, int width, int height, uint8_t *pixels, uint64_t pixels_bytes);
/* log_results (common.h:47-77): out_<scene>.txt = "version|%.3fs|<rays>|%0.3f mrays/s|" averaged over the runs. */
int r1_host_log_results(const char *version, const char *scene, const double *elapsed_seconds, const uint64_t *num_rays,
                        int num_runs);

#ifdef __cplusplus
}
#endif
#endif /* RAYS1_B200_H */
