/*
 * ppg.h -- C ABI of the B200-native guided path tracer (libppg_b200.so).
 *
 * This is the drop-in boundary for ONE hot path of Tom94/practical-path-guiding:
 * the GuidedPathTracer integrator plugin
 *   (reference: mitsuba/src/integrators/path/guided_path.cpp, "GP" below).
 *
 * What Mitsuba binds for that plugin (and what each entry point here replaces):
 *   - extern "C" CreateInstance(const Properties&) / GetDescription()
 *       (GP:2422 via include/mitsuba/core/cobject.h:99-107, src/libcore/plugin.cpp:40-96)
 *       -> ppg_params_default / ppg_params_set / ppg_create / ppg_description
 *   - GuidedPathTracer::GuidedPathTracer(const Properties&)            GP:1014-1085
 *       + MonteCarloIntegrator(const Properties&)   src/librender/integrator.cpp:190-225
 *       -> ppg_params (same names, defaults and validation)
 *   - Integrator::render(Scene*, RenderQueue*, const RenderJob*, int,int,int) -> bool
 *       (include/mitsuba/render/integrator.h:74-75, impl GP:1516-1585)
 *       -> ppg_set_scene + ppg_render
 *   - Integrator::cancel()                      (integrator.h:77-84, impl GP:1643-1648)
 *       -> ppg_cancel
 *   - dumpSDTree                                                        GP:1191-1208
 *       -> ppg_dump_sdtree
 *
 * Plain C types only: pointers + sizes, no C++/torch types, no exceptions cross
 * this boundary. All functions return PPG_OK (0) or a negative ppg_status.
 * The library owns all device memory; the caller owns every host array it
 * passes in (they may be freed as soon as the call returns) and the output
 * buffers it passes to ppg_render.
 *
 * There is NO CPU fallback: if no CUDA device is usable, ppg_create fails with
 * PPG_ERR_NO_DEVICE.
 */
#ifndef PPG_H
#define PPG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPG_ABI_VERSION 2   /* 2: bitmap textures, bumpmap, environment map */

typedef enum ppg_status {
    PPG_OK = 0,
    PPG_ERR_INVALID_ARGUMENT = -1, /* bad enum string / out-of-range value: the reference Assert(false)s (GP:1023,1034,1045,1054,1065,1080) or Log(EError)s (integrator.cpp:220-224) */
    PPG_ERR_NO_DEVICE = -2,        /* no usable CUDA device (no CPU fallback exists) */
    PPG_ERR_CUDA = -3,             /* a CUDA call failed; see ppg_last_error */
    PPG_ERR_NO_SCENE = -4,         /* ppg_render before ppg_set_scene */
    PPG_ERR_CANCELLED = -5,        /* ppg_cancel was called; partial film is still written (render() returns false in the reference, GP:1270-1277) */
    PPG_ERR_UNSUPPORTED = -6,      /* feature outside the hot-path scope (e.g. participating media, README.md:5-7) */
    PPG_ERR_IO = -7,
    PPG_ERR_COMM = -8              /* the user-supplied collective callback failed */
} ppg_status;

/* ---- integrator parameters (GP:1014-1085 + integrator.cpp:190-225) ------------------- */

typedef enum ppg_nee { PPG_NEE_NEVER = 0, PPG_NEE_KICKSTART = 1, PPG_NEE_ALWAYS = 2 } ppg_nee;                          /* GP:2278-2282 */
typedef enum ppg_sample_combination { PPG_COMB_DISCARD = 0, PPG_COMB_AUTOMATIC = 1, PPG_COMB_INVERSEVAR = 2 } ppg_sample_combination; /* GP:135-139 */
typedef enum ppg_loss { PPG_LOSS_NONE = 0, PPG_LOSS_KL = 1, PPG_LOSS_VAR = 2 } ppg_loss;                                /* GP:141-145 */
typedef enum ppg_spatial_filter { PPG_SFILTER_NEAREST = 0, PPG_SFILTER_STOCHASTIC = 1, PPG_SFILTER_BOX = 2 } ppg_spatial_filter; /* GP:147-151 */
typedef enum ppg_directional_filter { PPG_DFILTER_NEAREST = 0, PPG_DFILTER_BOX = 1 } ppg_directional_filter;            /* GP:153-156 */
typedef enum ppg_budget_type { PPG_BUDGET_SPP = 0, PPG_BUDGET_SECONDS = 1 } ppg_budget_type;                             /* GP:2298-2301 */

typedef struct ppg_params {
    /* guided_path.cpp parameters; the field comment is the XML name, type and default */
    int32_t nee;                      /* string  "nee"                      = "never"     */
    int32_t sample_combination;       /* string  "sampleCombination"        = "automatic" */
    int32_t spatial_filter;           /* string  "spatialFilter"            = "nearest"   */
    int32_t directional_filter;       /* string  "directionalFilter"        = "nearest"   */
    int32_t bsdf_sampling_fraction_loss; /* string "bsdfSamplingFractionLoss" = "none"    */
    int32_t sd_tree_max_memory;       /* integer "sdTreeMaxMemory"          = -1 (MB)     */
    int32_t s_tree_threshold;         /* integer "sTreeThreshold"           = 12000       */
    float   d_tree_threshold;         /* float   "dTreeThreshold"           = 0.01        */
    float   bsdf_sampling_fraction;   /* float   "bsdfSamplingFraction"     = 0.5         */
    int32_t spp_per_pass;             /* integer "sppPerPass"               = 4           */
    int32_t budget_type;              /* string  "budgetType"               = "seconds"   */
    float   budget;                   /* float   "budget"                   = 300         */
    int32_t dump_sd_tree;             /* boolean "dumpSDTree"               = false       */
    /* MonteCarloIntegrator parameters (integrator.cpp:190-225) */
    int32_t max_depth;                /* integer "maxDepth"                 = -1          */
    int32_t rr_depth;                 /* integer "rrDepth"                  = 5           */
    int32_t strict_normals;           /* boolean "strictNormals"            = false       */
    int32_t hide_emitters;            /* boolean "hideEmitters"             = false       */
    /* not in the reference: the reference's sampler seed is ignored
     * (src/samplers/independent.cpp:55-59) and it is not reproducible; ours is
     * a counter-based generator keyed by (seed, pass, pixel, sample). */
    uint64_t seed;                    /* integer "seed"                     = 1234        */
} ppg_params;

/* Fill in the reference defaults. */
void ppg_params_default(ppg_params *p);

/* Set one parameter from its XML (name, value-as-string) pair, exactly like the
 * Properties lookups of the reference constructor: enum-valued strings are
 * validated (unknown value -> PPG_ERR_INVALID_ARGUMENT, the reference's
 * Assert(false)); booleans accept "true"/"false"; unknown names ->
 * PPG_ERR_INVALID_ARGUMENT. */
int ppg_params_set(ppg_params *p, const char *name, const char *value);

/* Range checks of integrator.cpp:220-224 (rrDepth > 0; maxDepth == -1 or > 0)
 * plus sppPerPass >= 1, budget > 0. */
int ppg_params_validate(const ppg_params *p);

/* ---- scene description: flat arrays of what the hot path touches -------------------- */

typedef enum ppg_bsdf_type {
    PPG_BSDF_DIFFUSE = 0,        /* src/bsdfs/diffuse.cpp:110-150 */
    PPG_BSDF_NULL_BLACK = 1,     /* shape with an emitter and no BSDF: black diffuse (src/librender/shape.cpp:48-72) */
    PPG_BSDF_DIELECTRIC = 2,     /* src/bsdfs/dielectric.cpp:228-392: delta reflection + refraction, fresnelDielectricExt (libcore/util.cpp:651-683) */
    PPG_BSDF_CONDUCTOR = 3,      /* src/bsdfs/conductor.cpp:223-286: delta reflection, fresnelConductorExact per channel (libcore/util.cpp:740-765) */
    PPG_BSDF_ROUGHCONDUCTOR = 4, /* src/bsdfs/roughconductor.cpp:257-416 with MicrofacetDistribution (src/bsdfs/microfacet.h): Beckmann or GGX,
                                    visible-normal sampling; glossy => guided */
    PPG_BSDF_ROUGHPLASTIC = 5,   /* src/bsdfs/roughplastic.cpp:326-507: rough dielectric coat over a diffuse base; the rough transmittance
                                    (src/bsdfs/rtrans.h) is passed as a per-material 100-entry table + scalars */
    PPG_BSDF_ROUGHDIELECTRIC = 6,/* src/bsdfs/roughdielectric.cpp:270-600: rough refractive interface (reflectance = specularReflectance,
                                    specular_transmittance, eta[0] = intIOR/extIOR, alpha, distribution); draws one extra path-sampler number */
    PPG_BSDF_PLASTIC = 7,        /* src/bsdfs/plastic.cpp:245-441: smooth dielectric coat (delta reflection) over a diffuse base; reflectance = diffuse,
                                    specular_reflectance, eta[0], fdr_int = fresnelDiffuseReflectance(1/eta), specular_sampling_weight,
                                    PPG_BSDF_FLAG_NONLINEAR.  Mixed delta + smooth: exercises GP:1672-1676 */
    PPG_BSDF_THINDIELECTRIC = 8  /* src/bsdfs/thindielectric.cpp:153-306: delta reflection + index-matched (ENull) transmission with the internal
                                    reflections folded in; reflectance = specularReflectance, specular_transmittance, eta[0].  Null transitions
                                    are looked through by the emitter lookup (GP:2184-2245) and by light sampling (scene.cpp:619-679) */
} ppg_bsdf_type;

typedef enum ppg_microfacet { PPG_MICROFACET_BECKMANN = 0, PPG_MICROFACET_GGX = 1 } ppg_microfacet;   /* microfacet.h:47-60 */

#define PPG_BSDF_FLAG_TWOSIDED 1u /* src/bsdfs/twosided.cpp:108-184 wrapping the model */
#define PPG_BSDF_FLAG_NONLINEAR 2u /* roughplastic "nonlinear" (roughplastic.cpp:366-369) */
#define PPG_BSDF_FLAG_MASK 4u     /* src/bsdfs/mask.cpp:113-220 wrapping the (possibly twosided) model: constant `opacity`; a smooth/null hybrid */
#define PPG_BSDF_FLAG_BUMPMAP 8u  /* src/bsdfs/bumpmap.cpp:161-238 wrapping everything above: the shading frame is perturbed by the gradient of the
                                     displacement texture `bump_texture` (Frame getFrame(its), :139-159) */
#define PPG_BSDF_TABLE_SIZE 100   /* theta samples of the rough-transmittance tables (the .dat files of data/microfacet) */

typedef struct ppg_bsdf {
    int32_t  type;            /* ppg_bsdf_type */
    uint32_t flags;
    float    reflectance[3];  /* diffuse / roughplastic: diffuse reflectance; dielectric / conductor: specularReflectance. Linear Rec.709 RGB (scenehandler.cpp:597-613) */
    float    specular_transmittance[3];  /* dielectric */
    float    eta[3];          /* dielectric: eta[0] = intIOR / extIOR; conductor: eta / extEta per channel */
    float    k[3];            /* conductor: k / extEta per channel */
    float    alpha;           /* rough models: isotropic roughness (clamped to >= 1e-4 like microfacet.h:63) */
    int32_t  distribution;    /* rough models: ppg_microfacet */
    float    specular_reflectance[3];   /* roughplastic */
    float    fdr_int;         /* roughplastic: 1 - internal diffuse rough transmittance (Fdr of roughplastic.cpp:364) */
    float    specular_sampling_weight;  /* roughplastic: sAvg / (dAvg + sAvg) (roughplastic.cpp:269-272) */
    int32_t  table;           /* roughplastic: index into ppg_scene_desc.bsdf_tables (external rough transmittance over cos(theta)^(1/4)) */
    float    opacity[3];      /* PPG_BSDF_FLAG_MASK: linear RGB opacity (mask.cpp:63-66) */
    uint32_t reflectance_texture;   /* 1 + index into ppg_scene_desc.textures of the bitmap that replaces `reflectance` (diffuse "reflectance",
                                       roughplastic / plastic "diffuseReflectance"); 0 = the constant above.  For roughplastic / plastic the
                                       caller sets specular_sampling_weight from the texture's average (roughplastic.cpp:269-272) */
    uint32_t bump_texture;          /* PPG_BSDF_FLAG_BUMPMAP: 1 + index of the displacement texture */
    uint32_t reserved;
} ppg_bsdf;                   /* 112 bytes */

/* Bitmap texture (src/textures/bitmap.cpp).  The integrator fetches BSDFs without ray differentials (GP:1934 its.getBSDF() ->
 * hasUVPartials stays false, render/skdtree.h:417), so every lookup is the bilinear one at MIP level 0 (bitmap.cpp:431-453,
 * render/mipmap.h:575-596) whatever `filterType` says; only level 0 is passed.  Texels are IEEE half floats like the reference's
 * storage (bitmap.cpp:178-183), linear RGB (3 channels) or luminance (1 channel), row-major, row 0 first as decoded from the file. */
typedef enum ppg_wrap { PPG_WRAP_REPEAT = 0, PPG_WRAP_CLAMP = 1, PPG_WRAP_MIRROR = 2 } ppg_wrap;   /* mipmap.h:503-563 */
typedef struct ppg_texture {
    uint32_t width, height;
    uint32_t channels;        /* 1 or 3 */
    uint32_t wrap_u, wrap_v;  /* ppg_wrap */
    float    uv_scale[2];     /* Texture2D: uv' = uv * scale + offset (librender/texture.cpp:81-121) */
    float    uv_offset[2];
    uint32_t reserved;
    uint64_t first_texel;     /* offset (in uint16 elements) of texel (0,0) in ppg_scene_desc.texels */
} ppg_texture;                /* 48 bytes */

/* Environment emitter (src/emitters/envmap.cpp; `sunsky` is baked into one on the host, src/emitters/sunsky.cpp:122-225):
 * lat-long RGB map in half precision, looked up bilinearly (u repeats, v clamps) with u = atan2(v.x, -v.z) / 2pi,
 * v = acos(v.y) / pi for v = world_to_env * d (envmap.cpp:380-410); evaluated when a ray leaves the scene (GP:1902-1914, 2228-2243). */
typedef struct ppg_envmap {
    uint32_t width, height;   /* 0 x 0: the scene has no environment emitter */
    const uint16_t *texels;   /* width * height * 3 half floats */
    float    scale;           /* envmap "scale" */
    float    world_to_env[9]; /* row-major linear part of the inverse emitter-to-world transform */
} ppg_envmap;

typedef struct ppg_shape {
    uint32_t first_triangle;  /* triangles of a shape are contiguous */
    uint32_t n_triangles;
    int32_t  bsdf;            /* index into bsdfs */
    int32_t  emitter;         /* index into area_radiance (RGB triples), or -1 */
    uint32_t has_normals;     /* 0: face normals (skdtree.h:386-388) */
    uint32_t has_uvs;
    uint32_t reserved[2];
} ppg_shape;                  /* 32 bytes */

/* Analytic sphere (src/shapes/sphere.cpp); its ppg_shape has n_triangles == 0.  The object-to-world transform is restricted to
 * translation + uniform scale (all the bundled scenes need), so local coordinates are p - center. */
typedef struct ppg_sphere {
    float   center[3];
    float   radius;
    int32_t shape;         /* index into ppg_scene_desc.shapes (BSDF / emitter of the sphere) */
    int32_t flip_normals;  /* "flipNormals": normals point inwards */
} ppg_sphere;

typedef struct ppg_camera {   /* src/sensors/perspective.cpp:120-298 + librender/sensor.cpp:239-300 */
    float to_world[16];       /* row-major 4x4 camera-to-world (lookAt: columns left, up, dir, origin) */
    float x_fov_deg;          /* horizontal field of view after fovAxis resolution */
    float near_clip, far_clip;
    int32_t film_width, film_height;   /* crop window == full film */
} ppg_camera;

typedef struct ppg_scene_desc {
    uint32_t n_vertices;
    uint32_t n_triangles;
    uint32_t n_shapes;
    uint32_t n_bsdfs;
    uint32_t n_emitters;
    const float    *positions;      /* 3*n_vertices, world space */
    const float    *normals;        /* 3*n_vertices (ignored for shapes with has_normals==0), may be NULL */
    const float    *uvs;            /* 2*n_vertices, may be NULL */
    const uint32_t *indices;        /* 3*n_triangles */
    const uint32_t *triangle_shape; /* n_triangles: owning shape */
    const ppg_shape *shapes;
    const ppg_bsdf  *bsdfs;
    const float    *area_radiance;  /* 3*n_emitters: area-light radiance RGB (src/emitters/area.cpp:104-109) */
    const float    *bsdf_tables;    /* n_bsdf_tables * PPG_BSDF_TABLE_SIZE floats, may be NULL */
    uint32_t        n_bsdf_tables;
    uint32_t        n_spheres;
    const ppg_sphere *spheres;      /* may be NULL */
    ppg_camera camera;
    float aabb_min[3], aabb_max[3]; /* Scene::getAABB(): kd-tree AABB + sensor + emitter AABBs (librender/scene.cpp:387-413) */
    /* ABI 2 */
    uint32_t n_textures;
    uint32_t reserved;
    const ppg_texture *textures;    /* may be NULL */
    const uint16_t *texels;         /* half floats of all textures */
    uint64_t n_texels;              /* length of texels (bounds check) */
    ppg_envmap envmap;
} ppg_scene_desc;

/* Flat scene files for C / C++ hosts (written by `python -m ppg_b200.convert scene.xml scene.ppgscene`): fills *desc with pointers into
 * memory owned by *file (free with ppg_scene_file_free after ppg_set_scene).  `integrator_props`, if not NULL, receives the XML's
 * integrator parameters as "name=value" lines (valid until the file is freed).  No CUDA device is needed. */
typedef struct ppg_scene_file ppg_scene_file;
int ppg_scene_file_load(const char *path, ppg_scene_desc *desc, ppg_scene_file **file, const char **integrator_props);
void ppg_scene_file_free(ppg_scene_file *file);

/* ---- per-iteration statistics (the reference's log lines, GP:1176-1186, 1323-1326) --- */

#define PPG_MAX_ITERATIONS 40
#define PPG_KERNEL_CLASSES 8
typedef enum ppg_kernel_class {
    PPG_K_BOUNCE = 0,   /* ray generation + intersect + shade + guide + compaction, one launch per path depth */
    PPG_K_COMMIT = 1,   /* vertex records -> building trees (splat) */
    PPG_K_FILM = 2,     /* film / variance / develop */
    PPG_K_REFINE = 3,   /* S-tree refine */
    PPG_K_RESET = 4,    /* D-tree reset (count, scan, fill) */
    PPG_K_BUILD = 5,    /* D-tree build */
    PPG_K_ADAM = 6,
    PPG_K_OTHER = 7
} ppg_kernel_class;

typedef struct ppg_iteration_stats {
    int32_t  iteration;            /* k */
    int32_t  passes;               /* passes rendered in this iteration incl. FINAL extension */
    int32_t  is_final;
    int32_t  total_passes;         /* m_passesRendered after the iteration */
    float    seconds;              /* render passes only (GP:1321) */
    float    variance;             /* "Var:" of GP:1325 */
    float    reset_seconds, build_seconds;
    /* "Distribution statistics" block of GP:1176-1186, gathered after build */
    int32_t  depth_min, depth_max;           float depth_avg;
    float    mean_radiance_min, mean_radiance_avg, mean_radiance_max;
    uint64_t nodes_min, nodes_max;           float nodes_avg;
    float    weight_min, weight_avg, weight_max;
    uint32_t s_tree_nodes, s_tree_leaves;
    double   s_tree_depth_avg;     /* d_S: mean S-tree descent depth over recorded vertices (0 if not measured) */
    uint64_t vertices;             /* ray casts (path vertices) traced in this iteration: the "samples" of Msamples/s */
    uint64_t paths;
    uint64_t recorded_vertices;    /* guiding records committed (== sum of stat. weights when all weights are 1) */
} ppg_iteration_stats;

typedef struct ppg_stats {
    int32_t  n_iterations;
    int32_t  total_passes;
    uint64_t total_paths;
    uint64_t total_vertices;       /* paths x bounces: sum of ray casts */
    double   render_seconds;       /* wall clock of ppg_render */
    double   device_seconds;       /* CUDA-event time of all kernels */
    double   final_variance;
    uint64_t kernel_launches;
    /* CUDA-event time per kernel class, measured on the launching stream (index: ppg_kernel_class) */
    double   kernel_ms[PPG_KERNEL_CLASSES];
    uint64_t kernel_count[PPG_KERNEL_CLASSES];
    double   render_device_ms;     /* CUDA-event time of the whole render on the library's stream (with ppg_nccl_init: including the final film allreduce) */
    uint64_t truncated_paths;      /* paths still alive at the 64-bounce cap of maxDepth = -1 (they keep the radiance gathered so far) */
    uint64_t dropped_records;      /* sampling-fraction records beyond the record buffer (0 in every configuration measured) */
    uint64_t sub_batches;          /* wavefronts the learning iterations were split into (sampling-fraction step-size control) */
    uint64_t invalid_rays;         /* rays with a non-finite origin or direction, treated as misses (the reference's kd-tree clips them away) */
    ppg_iteration_stats iterations[PPG_MAX_ITERATIONS];
} ppg_stats;

/* ---- lifecycle ---------------------------------------------------------------------- */

typedef struct ppg_integrator ppg_integrator;

/* "Guided path tracer" -- GetDescription() of MTS_EXPORT_PLUGIN (GP:2422). */
const char *ppg_description(void);
int ppg_abi_version(void);

/* CreateInstance(props): validates the parameters and binds CUDA device
 * `device` (-1: current device). */
int ppg_create(const ppg_params *params, int device, ppg_integrator **out);
void ppg_destroy(ppg_integrator *h);

/* Upload the scene (builds the BVH on the host, copies everything to HBM). */
int ppg_set_scene(ppg_integrator *h, const ppg_scene_desc *scene);

/* Tile sharding (SURVEY 8e): this process renders only its share of the 32x32
 * image blocks.  The blocks are dealt round-robin to the ranks along a
 * scattered order (block j*s mod B goes to rank j mod world_size, s = the
 * golden-ratio stride coprime to the block count B), so that every rank's
 * blocks cover the whole image and the shares differ by at most one block.
 * Default is rank 0 of 1. */
int ppg_set_shard(ppg_integrator *h, int rank, int world_size);

/* The one exchange step of the sharded path: after the passes of a training
 * iteration and before build/refine, the library calls
 *     cb(user, device_ptr, n_floats)
 * on a device buffer holding this rank's packed training statistics
 * [quadtree node sums | per-leaf statistical weights | per-leaf Adam batch
 * accumulators | variance numerator]; the callback must sum it in place over
 * all ranks (e.g. ncclAllReduce / torch.distributed.all_reduce) and return 0
 * once the result is visible in device memory. Also used to sum the film at
 * the end. Not set (default) -> single-rank, no exchange. */
typedef int (*ppg_allreduce_fn)(void *user, void *device_ptr, size_t n_floats);
int ppg_set_allreduce(ppg_integrator *h, ppg_allreduce_fn cb, void *user);

/* Multi-GPU without a host round trip: the library dlopen()s libnccl.so.2 and enqueues ncclAllReduce on its own stream.
 * One rank calls ppg_nccl_unique_id (ncclGetUniqueId, 128 bytes), the host distributes the bytes (MPI, a file, torch.distributed
 * ...), then every rank calls ppg_nccl_init, which creates the communicator (ncclCommInitRank) and implies
 * ppg_set_shard(rank, world_size).  Takes precedence over a ppg_set_allreduce callback.  PPG_ERR_COMM if NCCL is unavailable. */
#define PPG_NCCL_UNIQUE_ID_BYTES 128
int ppg_nccl_unique_id(void *id_out);
int ppg_nccl_init(ppg_integrator *h, const void *id, int rank, int world_size);

/* budgetType = seconds reads a monotonic clock (GP:1259-1262, 1434-1514).  A host may supply its own (seconds since ppg_render
 * started rendering; used by the tests to drive the time-based schedule deterministically).  NULL restores the steady clock. */
typedef double (*ppg_clock_fn)(void *user);
int ppg_set_clock(ppg_integrator *h, ppg_clock_fn fn, void *user);

/* Progressive film: the reference puts every finished image block into the film while rendering (renderproc.cpp:143-151), which
 * is what a GUI or a time-limited job reads.  When set, the callback receives the current weight-normalised RGB film (DEVICE pointer,
 * W*H*3 floats, this rank's pixels) after every performRenderPasses, i.e. after every iteration and after every batch of the
 * final iteration of a seconds budget (GP:1482-1501); it runs on the host thread that drives ppg_render. */
typedef void (*ppg_film_fn)(void *user, const float *rgb_dev, int width, int height, int passes_rendered);
int ppg_set_film_callback(ppg_integrator *h, ppg_film_fn fn, void *user);

/* Integrator::render(). Runs the whole iteration schedule (GP:1342-1514),
 * develops the film into rgb_out (W*H*3 floats, row-major, host memory;
 * weight-normalised like hdrfilm) and fills *stats (may be NULL).
 * One host thread drives it; returns PPG_ERR_CANCELLED if ppg_cancel hit. */
int ppg_render(ppg_integrator *h, float *rgb_out, ppg_stats *stats);

/* Same, but the film stays in HBM: *rgb_dev receives a device pointer to
 * W*H*3 floats owned by the library (valid until the next render/destroy). */
int ppg_render_device(ppg_integrator *h, float **rgb_dev, ppg_stats *stats);

/* Integrator::cancel(): thread-safe, asynchronous. */
int ppg_cancel(ppg_integrator *h);

/* dumpSDTree wire format (GP:1191-1208, 699-711, 945-951), current sampling trees. */
int ppg_dump_sdtree(ppg_integrator *h, const char *path);

/* scene->getDestinationFile(): with dumpSDTree=true every non-final iteration writes "<destination>-NN.sdt"
 * (NN = two-digit iteration index, GP:1191-1195, 1417-1419). NULL/"" disables the per-iteration dumps. */
int ppg_set_destination(ppg_integrator *h, const char *destination);

/* Copy the variance-estimate helper images (sum, sum of squares; W*H*4 floats
 * each: R,G,B,weight) of the last performRenderPasses to the host. Either may be NULL. */
int ppg_get_moment_images(ppg_integrator *h, float *sum_rgbw, float *sumsq_rgbw);

/* Copy `bytes` from device memory handed out by the library (ppg_render_device, the film callback) to the host: lets a C / C++ host without the CUDA
 * runtime (e.g. the Mitsuba plugin shim) read such buffers. */
int ppg_copy_from_device(void *host_dst, const void *device_src, size_t bytes);

const char *ppg_last_error(void);

/* ---- batch operators on SD-tree arrays (kernel-level entry points) ------------------- *
 * These run the SAME device functions the render kernels use on caller-supplied
 * flat tree arrays, so parity tests can compare them element-wise against the
 * oracle. All pointers are HOST pointers; copies happen inside.
 *
 * D-tree arrays: node i has sums[4*i..4*i+3] and children[4*i..4*i+3]
 * (uint16, 0 = leaf), the reference's QuadTreeNode (GP:158-371, 368-370).
 * tree_first_node[t] is the index of the root of tree t; tree_sum / tree_weight
 * are DTree::m_atomic (GP:538-557).                                                    */

/* DTreeWrapper::pdf (GP:623-625 -> 415-421, 232-245): n directions (xyz). */
int ppg_op_dtree_pdf(int device,
                     const float *sums, const uint16_t *children, size_t n_nodes,
                     const uint32_t *tree_first_node, const float *tree_sum, const float *tree_weight, size_t n_trees,
                     const uint32_t *query_tree, const float *query_dir, size_t n, float *pdf_out);

/* DTreeWrapper::sample (GP:619-621 -> 431-442, 257-301) with REPLAYED uniforms:
 * rnd holds rnd_stride floats per query, consumed in the reference's order (one per level, two at the leaf).
 * dir_out: 3 floats per query. */
int ppg_op_dtree_sample(int device,
                        const float *sums, const uint16_t *children, size_t n_nodes,
                        const uint32_t *tree_first_node, const float *tree_sum, const float *tree_weight, size_t n_trees,
                        const uint32_t *query_tree, const float *rnd, size_t rnd_stride, size_t n, float *dir_out);

/* DTreeWrapper::record (GP:575-584 -> 395-413, 303-338) for n records into the
 * building sums (in/out) and per-tree statistical weights (in/out); filter = ppg_directional_filter. */
int ppg_op_dtree_record(int device,
                        float *sums_inout, const uint16_t *children, size_t n_nodes,
                        const uint32_t *tree_first_node, float *tree_weight_inout, size_t n_trees,
                        const uint32_t *rec_tree, const float *rec_dir, const float *rec_radiance,
                        const float *rec_wo_pdf, const float *rec_weight, size_t n, int filter);

/* The sampling-fraction replay of a commit launch (adam_hist -> exclusive_scan -> adam_scatter -> adam_seq -> adam_progress, with the
 * launch shapes the renderer uses) on given records, for testing it against the reference's AdamOptimizer.
 * states: 6 floats per leaf (iter, m, v, variable, batchAcc, batchGrad), the start of the first batch.  Records as the commit kernel
 * appends them: rec_a 4 floats {bits(leaf), product, woPdf, bsdfPdf}, rec_b 2 floats {dTreePdf, weight}; counts[b * replicas + r]
 * records of batch b, replica r follow each other in that order.  Of a group of `total` records the first min(total, cap) are
 * replayed, as in a commit launch with a record list of capacity cap.  The batches run one after the other on the same counting
 * buffers.  replicas > 1 or merge != 0: every replica replays its records from the state at the start of the batch, then
 * adam_pack, a sum over the replicas in replica order (standing in for the allreduce) and adam_merge.  loss = PPG_LOSS_KL | VAR.
 * Outputs, per batch (any may be NULL): states_out 6 floats per leaf; replica_out 6 floats per leaf per replica before the merge;
 * theta_out the variable written into the leaf record; sorted_a_out / sorted_b_out the bucketed record lists (layout of rec_a /
 * rec_b, min(total, cap) entries per group); progress_out {sum steps * |f after - f before| * 2^20, sum steps}. */
int ppg_op_fraction_replay(int device, const float *states, size_t n_leaves, const float *rec_a, const float *rec_b, const size_t *counts,
                           int n_batches, int replicas, int merge, size_t cap, int loss, float *states_out, float *replica_out, float *theta_out,
                           float *sorted_a_out, float *sorted_b_out, unsigned long long *progress_out);

/* The acceleration structure ppg_set_scene builds over the scene's triangles (binned-SAH BVH; it takes the place of the reference's ShapeKDTree,
 * src/librender/skdtree.cpp), on the HOST alone -- no CUDA device needed: for tests of the builder and for timing it.  positions 3 floats per vertex,
 * indices 3 per triangle; threads <= 0: the library's default (the cores this process may use, at most 16; PPG_HOST_THREADS overrides).
 * nodes_out: 8 floats per node {min.xyz, bits(left), max.xyz, bits(count)} -- count == 0: inner node with children `left`, `left + 1`; otherwise a
 * leaf over order_out[left .. left + count) -- capacity in nodes (2 * n_triangles + 1 always suffices); order_out: n_triangles triangle indices.
 * The result does not depend on the thread count.  Any output pointer may be NULL. */
int ppg_op_bvh_build(const float *positions, const uint32_t *indices, size_t n_triangles, int threads,
                     float *nodes_out, size_t nodes_capacity, uint32_t *order_out, size_t *n_nodes_out, int *max_depth_out, double *ms_out);

/* Scene::sampleAttenuatedEmitterDirect (src/librender/scene.cpp:876-897 -> AreaLight / Sphere / EnvironmentMap::sampleDirect, then
 * Scene::evalTransmittance) at n reference points of the handle's scene, as the light-sampling block of Li calls it (GP:1964-1973):
 * ref, ref_n 3n floats (ref_n = 0: no front-side test, records.inl:160-164), sample 2n uniforms, max_interactions = maxDepth - depth - 1
 * (negative: unlimited).  d_out 3n, value_out 3n (radiance x transmittance / pdf), pdf_out n (0: the sample carries nothing), dist_out n.
 * Needs a scene that runs the full-feature kernels (any non-diffuse BSDF, sphere, texture or an environment emitter). */
int ppg_op_emitter_sample_direct(ppg_integrator *h, size_t n, const float *ref, const float *ref_n, const float *sample, int max_interactions,
                                 float *d_out, float *value_out, float *pdf_out, float *dist_out);

/* Scene::pdfEmitterDirect of the environment emitter (EnvironmentMap::pdfDirect, src/emitters/envmap.cpp:545-548, 603-633, times the
 * discrete emitter choice) for n world directions d (3n), and optionally its radiance there (evalEnvironment, :380-410; value_out 3n or NULL). */
int ppg_op_env_pdf(ppg_integrator *h, size_t n, const float *d, float *pdf_out, float *value_out);

/* STree::dTreeWrapper(p, size) (GP:897-905, 761-769): S-tree nodes as uint32
 * pairs (child0, child1); child0 == 0 marks a leaf. Outputs the leaf NODE index
 * and the voxel size (3 floats) per query point. */
int ppg_op_stree_lookup(int device,
                        const uint32_t *node_children, size_t n_nodes,
                        const float aabb_min[3], const float aabb_extent[3],
                        const float *points, size_t n, uint32_t *leaf_out, float *size_out);

#ifdef __cplusplus
}
#endif
#endif /* PPG_H */
