// ppg_host.cu -- host side of libppg_b200.so: the C ABI of include/ppg.h, the iteration schedule of the
// reference integrator (GP = mitsuba/src/integrators/path/guided_path.cpp), BVH construction and the
// launch sequence of the wavefront kernels.  C++ host, CUDA kernels, no torch, no CPU fallback.
#include "../../include/ppg.h"
#include "ppg_kernels.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <string>
#include <system_error>
#include <thread>
#include <vector>
#ifdef __linux__
#include <sched.h>
#endif

using namespace ppg;

// ------------------------------------------------------------------ errors
static thread_local std::string g_lastError;
static int fail(int code, const std::string &msg) { g_lastError = msg; return code; }
// "no exceptions cross this boundary" (ppg.h): the entry points that allocate host memory in proportion to their input run under this guard
template <class F> static int guarded(const char *what, F body) {
    try { return body(); }
    catch (const std::bad_alloc &) { return fail(PPG_ERR_INVALID_ARGUMENT, std::string(what) + ": out of host memory"); }
    catch (const std::exception &e) { return fail(PPG_ERR_INVALID_ARGUMENT, std::string(what) + ": " + e.what()); }
}
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            g_lastError = std::string(#call) + ": " + cudaGetErrorString(e_) + " (" + __FILE__ + ":" + std::to_string(__LINE__) + ")"; \
            return PPG_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

template <class T> struct DevBuf {
    T *p = nullptr; size_t n = 0;
    ~DevBuf() { release(); }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    cudaError_t alloc(size_t count) {
        if (count <= n && p) return cudaSuccess;
        release();
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    // grow preserving contents
    cudaError_t grow(size_t count, cudaStream_t s) {
        if (count <= n && p) return cudaSuccess;
        T *q = nullptr; cudaError_t e = cudaMalloc(&q, count * sizeof(T));
        if (e != cudaSuccess) return e;
        if (p && n) cudaMemcpyAsync(q, p, n * sizeof(T), cudaMemcpyDeviceToDevice, s);
        cudaStreamSynchronize(s);
        if (p) cudaFree(p);
        p = q; n = count; return cudaSuccess;
    }
};

// ------------------------------------------------------------------ parameters (GP:1014-1085, integrator.cpp:190-225)
extern "C" void ppg_params_default(ppg_params *p) {
    p->nee = PPG_NEE_NEVER; p->sample_combination = PPG_COMB_AUTOMATIC; p->spatial_filter = PPG_SFILTER_NEAREST;
    p->directional_filter = PPG_DFILTER_NEAREST; p->bsdf_sampling_fraction_loss = PPG_LOSS_NONE;
    p->sd_tree_max_memory = -1; p->s_tree_threshold = 12000; p->d_tree_threshold = 0.01f; p->bsdf_sampling_fraction = 0.5f;
    p->spp_per_pass = 4; p->budget_type = PPG_BUDGET_SECONDS; p->budget = 300.0f; p->dump_sd_tree = 0;
    p->max_depth = -1; p->rr_depth = 5; p->strict_normals = 0; p->hide_emitters = 0; p->seed = 1234;
}

static bool parse_enum(const char *v, const char *const *names, int n, int32_t *out) {
    for (int i = 0; i < n; ++i) if (!strcmp(v, names[i])) { *out = i; return true; }
    return false;
}
static bool parse_bool(const char *v, int32_t *out) {
    if (!strcmp(v, "true")) { *out = 1; return true; }
    if (!strcmp(v, "false")) { *out = 0; return true; }
    return false;
}
static bool parse_int(const char *v, long long *out) { char *e = nullptr; *out = strtoll(v, &e, 10); return e && *e == '\0' && e != v; }
static bool parse_float(const char *v, float *out) { char *e = nullptr; *out = strtof(v, &e); return e && *e == '\0' && e != v; }

extern "C" int ppg_params_set(ppg_params *p, const char *name, const char *value) {
    if (!p || !name || !value) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    static const char *const nee[] = {"never", "kickstart", "always"};
    static const char *const comb[] = {"discard", "automatic", "inversevar"};
    static const char *const sf[] = {"nearest", "stochastic", "box"};
    static const char *const df[] = {"nearest", "box"};
    static const char *const loss[] = {"none", "kl", "var"};
    static const char *const bt[] = {"spp", "seconds"};
    bool ok; long long iv;
    std::string n(name);
    if (n == "nee") ok = parse_enum(value, nee, 3, &p->nee);
    else if (n == "sampleCombination") ok = parse_enum(value, comb, 3, &p->sample_combination);
    else if (n == "spatialFilter") ok = parse_enum(value, sf, 3, &p->spatial_filter);
    else if (n == "directionalFilter") ok = parse_enum(value, df, 2, &p->directional_filter);
    else if (n == "bsdfSamplingFractionLoss") ok = parse_enum(value, loss, 3, &p->bsdf_sampling_fraction_loss);
    else if (n == "budgetType") ok = parse_enum(value, bt, 2, &p->budget_type);
    else if (n == "sdTreeMaxMemory") { ok = parse_int(value, &iv); if (ok) p->sd_tree_max_memory = (int32_t) iv; }
    else if (n == "sTreeThreshold") { ok = parse_int(value, &iv); if (ok) p->s_tree_threshold = (int32_t) iv; }
    else if (n == "sppPerPass") { ok = parse_int(value, &iv); if (ok) p->spp_per_pass = (int32_t) iv; }
    else if (n == "maxDepth") { ok = parse_int(value, &iv); if (ok) p->max_depth = (int32_t) iv; }
    else if (n == "rrDepth") { ok = parse_int(value, &iv); if (ok) p->rr_depth = (int32_t) iv; }
    else if (n == "seed") { ok = parse_int(value, &iv); if (ok) p->seed = (uint64_t) iv; }
    else if (n == "dTreeThreshold") ok = parse_float(value, &p->d_tree_threshold);
    else if (n == "bsdfSamplingFraction") ok = parse_float(value, &p->bsdf_sampling_fraction);
    else if (n == "budget") ok = parse_float(value, &p->budget);
    else if (n == "dumpSDTree") ok = parse_bool(value, &p->dump_sd_tree);
    else if (n == "strictNormals") ok = parse_bool(value, &p->strict_normals);
    else if (n == "hideEmitters") ok = parse_bool(value, &p->hide_emitters);
    else return fail(PPG_ERR_INVALID_ARGUMENT, "unknown integrator parameter '" + n + "'");
    if (!ok) return fail(PPG_ERR_INVALID_ARGUMENT, "invalid value '" + std::string(value) + "' for parameter '" + n + "'");
    return PPG_OK;
}

extern "C" int ppg_params_validate(const ppg_params *p) {
    if (!p) return fail(PPG_ERR_INVALID_ARGUMENT, "null params");
    auto in = [](int v, int lo, int hi) { return v >= lo && v <= hi; };
    if (!in(p->nee, 0, 2) || !in(p->sample_combination, 0, 2) || !in(p->spatial_filter, 0, 2) || !in(p->directional_filter, 0, 1) ||
        !in(p->bsdf_sampling_fraction_loss, 0, 2) || !in(p->budget_type, 0, 1))
        return fail(PPG_ERR_INVALID_ARGUMENT, "enum parameter out of range (the reference Assert(false)s, GP:1023-1080)");
    if (p->rr_depth <= 0) return fail(PPG_ERR_INVALID_ARGUMENT, "'rrDepth' must be set to a value greater than zero!");
    if (p->max_depth <= 0 && p->max_depth != -1) return fail(PPG_ERR_INVALID_ARGUMENT, "'maxDepth' must be set to -1 (infinite) or a value greater than zero!");
    if (p->spp_per_pass < 1) return fail(PPG_ERR_INVALID_ARGUMENT, "'sppPerPass' must be at least 1");
    if (!(p->budget > 0)) return fail(PPG_ERR_INVALID_ARGUMENT, "'budget' must be positive");
    if (!(p->bsdf_sampling_fraction >= 0.f && p->bsdf_sampling_fraction <= 1.f)) return fail(PPG_ERR_INVALID_ARGUMENT, "'bsdfSamplingFraction' must lie in [0,1]");
    return PPG_OK;
}

extern "C" const char *ppg_description(void) { return "Guided path tracer"; }
extern "C" int ppg_abi_version(void) { return PPG_ABI_VERSION; }
extern "C" const char *ppg_last_error(void) { return g_lastError.c_str(); }

// ------------------------------------------------------------------ flat scene files (python -m ppg_b200.convert)
struct ppg_scene_file { std::vector<std::vector<char>> blobs; std::string props; };
extern "C" int ppg_scene_file_load(const char *path, ppg_scene_desc *d, ppg_scene_file **file, const char **integrator_props) {
    if (!path || !d || !file) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    FILE *f = fopen(path, "rb");
    if (!f) return fail(PPG_ERR_IO, std::string("cannot open ") + path);
    char magic[8];
    if (fread(magic, 1, 8, f) != 8 || memcmp(magic, "PPGSCN02", 8) != 0) { fclose(f); return fail(PPG_ERR_IO, "not a PPGSCN02 scene file"); }
    long fileBytes = 0;                                   // no array can be larger than the file: a corrupt header must not turn into a huge allocation
    if (fseek(f, 0, SEEK_END) != 0 || (fileBytes = ftell(f)) < 8 || fseek(f, 8, SEEK_SET) != 0) { fclose(f); return fail(PPG_ERR_IO, "cannot size the scene file"); }
    ppg_scene_file *sf = new (std::nothrow) ppg_scene_file();
    if (!sf) { fclose(f); return fail(PPG_ERR_IO, "out of memory"); }
    memset(d, 0, sizeof(*d));
    struct Arr { const char *p; size_t bytes; uint64_t dims[4]; uint32_t ndim; };
    auto fail_io = [&](const char *m) { fclose(f); delete sf; return fail(PPG_ERR_IO, m); };
    static const size_t esz[6] = {4, 4, 4, 2, 1, 8};
    std::vector<std::pair<std::string, Arr>> arrs;
    for (;;) {
        uint32_t nl;
        if (fread(&nl, 4, 1, f) != 1) break;
        if (nl > 64) return fail_io("corrupt scene file (name)");
        std::string name(nl, 0); uint32_t hdr[2];
        if (fread(&name[0], 1, nl, f) != nl || fread(hdr, 4, 2, f) != 2 || hdr[0] > 5 || hdr[1] > 4) return fail_io("corrupt scene file (header)");
        Arr a; a.ndim = hdr[1]; size_t count = 1;
        for (uint32_t k = 0; k < a.ndim; ++k) {
            if (fread(&a.dims[k], 8, 1, f) != 1) return fail_io("corrupt scene file (dims)");
            if (a.dims[k] > (uint64_t) fileBytes || (a.dims[k] && count > (size_t) fileBytes / (size_t) a.dims[k])) return fail_io("corrupt scene file (array larger than the file)");
            count *= (size_t) a.dims[k];
        }
        a.bytes = count * esz[hdr[0]];
        if (a.bytes > (size_t) fileBytes) return fail_io("corrupt scene file (array larger than the file)");
        try { sf->blobs.emplace_back(a.bytes + 8); } catch (const std::bad_alloc &) { return fail_io("out of memory"); }
        if (a.bytes && fread(sf->blobs.back().data(), 1, a.bytes, f) != a.bytes) return fail_io("truncated scene file");
        a.p = sf->blobs.back().data();
        arrs.emplace_back(name, a);
    }
    fclose(f);
    auto get = [&](const char *n) -> const Arr * { for (auto &kv : arrs) if (kv.first == n) return &kv.second; return nullptr; };
    const Arr *P = get("positions"), *N = get("normals"), *UV = get("uvs"), *I = get("indices"), *TS = get("triangle_shape"), *SH = get("shapes"), *B = get("bsdfs"),
              *R = get("area_radiance"), *T = get("bsdf_tables"), *SP = get("spheres"), *CW = get("cam_to_world"), *CAM = get("cam"), *BB = get("aabb"),
              *TX = get("textures"), *TL = get("texels"), *ET = get("env_texels"), *EM = get("env_meta"), *IP = get("integrator");
    if (!P || !N || !UV || !I || !TS || !SH || !B || !R || !CW || !CAM || !BB || CW->bytes != 64 || CAM->bytes != 40 || BB->bytes != 24 || B->bytes % sizeof(ppg_bsdf) || SH->bytes % sizeof(ppg_shape))
        { delete sf; return fail(PPG_ERR_IO, "scene file lacks a required array"); }
    // per-vertex / per-triangle arrays must cover what the counts promise (ppg_set_scene indexes them without further checks)
    if (P->bytes % 12 || I->bytes % 12 || R->bytes % 12 || N->bytes != P->bytes || UV->bytes != P->bytes / 12 * 8 || TS->bytes != I->bytes / 12 * 4 ||
        (T && T->bytes % (4 * PPG_BSDF_TABLE_SIZE)) || (SP && SP->bytes % sizeof(ppg_sphere)) || (TX && TX->bytes % sizeof(ppg_texture)) ||
        (ET && ET->bytes && (ET->ndim != 3 || ET->dims[2] != 3 || ET->bytes != ET->dims[0] * ET->dims[1] * 6)))
        { delete sf; return fail(PPG_ERR_IO, "scene file: array sizes do not match each other"); }
    d->n_vertices = (uint32_t) (P->bytes / 12); d->n_triangles = (uint32_t) (I->bytes / 12); d->n_shapes = (uint32_t) (SH->bytes / sizeof(ppg_shape));
    d->n_bsdfs = (uint32_t) (B->bytes / sizeof(ppg_bsdf)); d->n_emitters = (uint32_t) (R->bytes / 12);
    d->positions = (const float *) P->p; d->normals = (const float *) N->p; d->uvs = (const float *) UV->p; d->indices = (const uint32_t *) I->p;
    d->triangle_shape = (const uint32_t *) TS->p; d->shapes = (const ppg_shape *) SH->p; d->bsdfs = (const ppg_bsdf *) B->p; d->area_radiance = (const float *) R->p;
    if (T && T->bytes) { d->bsdf_tables = (const float *) T->p; d->n_bsdf_tables = (uint32_t) (T->bytes / (4 * PPG_BSDF_TABLE_SIZE)); }
    if (SP && SP->bytes) { d->spheres = (const ppg_sphere *) SP->p; d->n_spheres = (uint32_t) (SP->bytes / sizeof(ppg_sphere)); }
    memcpy(d->camera.to_world, CW->p, 64);
    const double *cam = (const double *) CAM->p;
    d->camera.x_fov_deg = (float) cam[0]; d->camera.near_clip = (float) cam[1]; d->camera.far_clip = (float) cam[2]; d->camera.film_width = (int32_t) cam[3]; d->camera.film_height = (int32_t) cam[4];
    memcpy(d->aabb_min, BB->p, 12); memcpy(d->aabb_max, BB->p + 12, 12);
    if (TX && TX->bytes && TL) { d->textures = (const ppg_texture *) TX->p; d->n_textures = (uint32_t) (TX->bytes / sizeof(ppg_texture)); d->texels = (const uint16_t *) TL->p; d->n_texels = TL->bytes / 2; }
    if (ET && ET->bytes && EM && EM->bytes == 40 && ET->ndim == 3) {
        d->envmap.height = (uint32_t) ET->dims[0]; d->envmap.width = (uint32_t) ET->dims[1]; d->envmap.texels = (const uint16_t *) ET->p;
        const float *em = (const float *) EM->p; d->envmap.scale = em[0]; memcpy(d->envmap.world_to_env, em + 1, 36);
    }
    if (IP) sf->props.assign(IP->p, IP->bytes);
    if (integrator_props) *integrator_props = sf->props.c_str();
    *file = sf;
    return PPG_OK;
}
extern "C" void ppg_scene_file_free(ppg_scene_file *file) { delete file; }

// ------------------------------------------------------------------ host BVH (binned SAH) + Wald triangle constants
namespace {
struct H3 { float x, y, z; };
static inline float half_to_float(uint16_t h) {                                  // IEEE binary16 -> binary32 (host side of the texel tables)
    const uint32_t sgn = (uint32_t) (h >> 15) << 31, e = (h >> 10) & 31u, m = h & 1023u;
    uint32_t bits;
    if (e == 0) {
        if (m == 0) bits = sgn;
        else { int sh = 0; uint32_t mm = m; while (!(mm & 1024u)) { mm <<= 1; ++sh; } bits = sgn | ((uint32_t) (113 - sh) << 23) | ((mm & 1023u) << 13); }
    } else if (e == 31) bits = sgn | 0x7f800000u | (m << 13);
    else bits = sgn | ((e + 112u) << 23) | (m << 13);
    float f; memcpy(&f, &bits, 4); return f;
}
static inline H3 h3(float x, float y, float z) { return H3{x, y, z}; }
static inline H3 operator-(H3 a, H3 b) { return h3(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline H3 hcross(H3 a, H3 b) { return h3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
static inline float hdot(H3 a, H3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline float hcomp(H3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// restated from include/mitsuba/render/triaccel.h:60-93 (Wald's projection-plane precomputation)
static void wald_constants(H3 A, H3 B, H3 C, float out[9], int &k) {
    static const int mod3[4] = {1, 2, 0, 1};
    const H3 b = C - A, c = B - A, N = hcross(c, b);
    k = 0;
    for (int j = 0; j < 3; ++j) if (std::fabs(hcomp(N, j)) > std::fabs(hcomp(N, k))) k = j;
    const int u = mod3[k], v = mod3[k + 1];
    const float n_k = hcomp(N, k), denom = hcomp(b, u) * hcomp(c, v) - hcomp(b, v) * hcomp(c, u);
    if (denom == 0) { k = 3; for (int i = 0; i < 9; ++i) out[i] = 0; return; }
    out[0] = hcomp(N, u) / n_k; out[1] = hcomp(N, v) / n_k; out[2] = hdot(A, N) / n_k;   // n_u n_v n_d
    out[3] = hcomp(A, u); out[4] = hcomp(A, v);                                           // a_u a_v
    out[5] = hcomp(b, u) / denom; out[6] = -hcomp(b, v) / denom;                          // b_nu b_nv
    out[7] = hcomp(c, v) / denom; out[8] = -hcomp(c, u) / denom;                          // c_nu c_nv
}

static int bvh_env_int(const char *name, int dflt) { const char *v = getenv(name); return v && *v ? atoi(v) : dflt; }   // tuning experiments only

// Host-side parallelism of ppg_set_scene (per-triangle tables, BVH build, texel repacking): plain std::thread fork / join over index ranges.
// PPG_HOST_THREADS overrides the count (default: the cores this process may run on, at most 16).  Every parallel loop below computes
// exactly what its serial form computes (min / max / integer counts / independent elements), so the scene tables do not depend on the count.
static int host_threads() {
    static const int n = [] {
        int t = bvh_env_int("PPG_HOST_THREADS", 0);
        if (t <= 0) {
            t = (int) std::thread::hardware_concurrency();
#ifdef __linux__
            cpu_set_t set; CPU_ZERO(&set);
            if (sched_getaffinity(0, sizeof(set), &set) == 0) t = CPU_COUNT(&set);
#endif
            t = std::min(t, 16);
        }
        return std::max(t, 1);
    }();
    return n;
}
template <class F> static void parallel_for(size_t n, int threads, size_t minChunk, F fn) {   // fn(begin, end, chunk index)
    const int T = (int) std::max<size_t>(1, std::min<size_t>((size_t) threads, n / std::max<size_t>(minChunk, 1)));
    if (T <= 1) { fn((size_t) 0, n, 0); return; }
    std::vector<std::thread> pool; pool.reserve(T - 1);
    int started = 1;
    for (int k = 1; k < T; ++k) {
        try { pool.emplace_back([&, k] { fn(n * k / T, n * (k + 1) / T, k); }); ++started; }
        catch (const std::system_error &) { break; }                 // no more threads to be had: the remaining chunks run here
    }
    fn((size_t) 0, n / T, 0);
    for (int k = started; k < T; ++k) fn(n * k / T, n * (k + 1) / T, k);
    for (auto &th : pool) th.join();
}

struct HostBvh {
    std::vector<float> nodes;        // 8 floats per node
    std::vector<uint32_t> order;     // leaf order -> original triangle
    int maxDepth = 0;                // the device walk keeps one stack entry per level (PPG_BVH_STACK)
};
// Binned-SAH BVH (16 bins per axis, leaves of at most PPG_BVH_LEAF triangles, a traversal-cost term decides the last splits).
// The tree is a function of the triangle bounds alone: a node's split depends only on the triangles of its range, children work on disjoint
// ranges of `order`.  It is therefore built in any order -- big nodes one after the other with their O(n) loops spread over the threads, the
// subtrees below them concurrently -- into an arena, and numbered afterwards in the order a depth-first stack visits it (right child first),
// which is the numbering the device layout (siblings adjacent, `left` = index of the first child) has always had.
static void build_bvh(const std::vector<H3> &tminV, const std::vector<H3> &tmaxV, HostBvh &out, int threads) {
    const uint32_t nt = (uint32_t) tminV.size();
    out.order.resize(nt);
    std::vector<H3> cenV(nt);
    const H3 *const tmin = tminV.data(), *const tmax = tmaxV.data(); H3 *const cen = cenV.data();
    parallel_for(nt, threads, 1 << 15, [&](size_t b, size_t e, int) {
        for (size_t t = b; t < e; ++t) { out.order[t] = (uint32_t) t; cen[t] = h3(0.5f * (tmin[t].x + tmax[t].x), 0.5f * (tmin[t].y + tmax[t].y), 0.5f * (tmin[t].z + tmax[t].z)); }
    });
    const int maxLeaf = std::min(std::max(bvh_env_int("PPG_BVH_LEAF", 4), 1), 15);   // <= 15: the device stack packs the count in 4 bits
    const float Ct = (float) bvh_env_int("PPG_BVH_CT_X10", 10) * 0.1f;
    constexpr int NB = 16;
    struct Node { H3 mn, mx; uint32_t left, count; };                                 // count == 0: inner node, `left` = arena index of its first child
    struct Job { uint32_t node, first, count; int depth; };
    struct Bounds { H3 mn, mx, cmn, cmx; };
    struct Bins { H3 mn[3][NB], mx[3][NB]; uint32_t c[3][NB]; };
    const H3 big = h3(1e30f, 1e30f, 1e30f), small = h3(-1e30f, -1e30f, -1e30f);
    auto hmin = [](H3 a, H3 b) { return h3(std::min(a.x, b.x), std::min(a.y, b.y), std::min(a.z, b.z)); };
    auto hmax = [](H3 a, H3 b) { return h3(std::max(a.x, b.x), std::max(a.y, b.y), std::max(a.z, b.z)); };
    auto area = [](H3 mn, H3 mx) { const float dx = mx.x - mn.x, dy = mx.y - mn.y, dz = mx.z - mn.z; return 2.f * (dx * dy + dy * dz + dz * dx); };
    auto binOf = [&](uint32_t t, int ax, float lo, float hi) { int b = (int) (NB * (hcomp(cen[t], ax) - lo) / (hi - lo)); return std::min(std::max(b, 0), NB - 1); };

    std::vector<Node> arena(2 * (size_t) nt + 1);
    std::atomic<uint32_t> arenaUsed{1};
    std::atomic<int> deepest{0};
    const uint32_t *order = out.order.data();

    // one node: bounds, best binned split, partition of its range.  Returns true and the left count when the node was split.
    auto process = [&](const Job &j, int loopThreads, uint32_t &nlOut) -> bool {
        Bounds bd{big, small, big, small};
        if (loopThreads > 1) {
            std::vector<Bounds> part((size_t) loopThreads, Bounds{big, small, big, small});
            parallel_for(j.count, loopThreads, 1 << 14, [&](size_t b, size_t e, int k) {
                Bounds l{big, small, big, small};
                for (size_t i = j.first + b; i < j.first + e; ++i) { const uint32_t t = order[i]; l.mn = hmin(l.mn, tmin[t]); l.mx = hmax(l.mx, tmax[t]); l.cmn = hmin(l.cmn, cen[t]); l.cmx = hmax(l.cmx, cen[t]); }
                part[k] = l;
            });
            for (const Bounds &l : part) { bd.mn = hmin(bd.mn, l.mn); bd.mx = hmax(bd.mx, l.mx); bd.cmn = hmin(bd.cmn, l.cmn); bd.cmx = hmax(bd.cmx, l.cmx); }
        } else
            for (uint32_t i = j.first; i < j.first + j.count; ++i) { const uint32_t t = order[i]; bd.mn = hmin(bd.mn, tmin[t]); bd.mx = hmax(bd.mx, tmax[t]); bd.cmn = hmin(bd.cmn, cen[t]); bd.cmx = hmax(bd.cmx, cen[t]); }
        Node nd; nd.mn = bd.mn; nd.mx = bd.mx; nd.left = j.first; nd.count = j.count;
        arena[j.node] = nd;
        if (j.count <= 1) return false;
        // binned SAH over the three axes (one pass fills the bins of all axes with a centroid extent)
        bool axisOk[3]; float lo[3], hi[3];
        for (int ax = 0; ax < 3; ++ax) { lo[ax] = hcomp(bd.cmn, ax); hi[ax] = hcomp(bd.cmx, ax); axisOk[ax] = hi[ax] > lo[ax]; }
        auto clearBins = [&](Bins &B) { for (int ax = 0; ax < 3; ++ax) if (axisOk[ax]) for (int b = 0; b < NB; ++b) { B.mn[ax][b] = big; B.mx[ax][b] = small; B.c[ax][b] = 0; } };
        auto fillBins = [&](Bins &B, size_t b0, size_t e0) {
            for (size_t i = j.first + b0; i < j.first + e0; ++i) {
                const uint32_t t = order[i];
                for (int ax = 0; ax < 3; ++ax) {
                    if (!axisOk[ax]) continue;
                    const int b = binOf(t, ax, lo[ax], hi[ax]);
                    B.c[ax][b]++; B.mn[ax][b] = hmin(B.mn[ax][b], tmin[t]); B.mx[ax][b] = hmax(B.mx[ax][b], tmax[t]);
                }
            }
        };
        Bins bins; clearBins(bins);
        if (loopThreads > 1) {
            std::vector<Bins> part((size_t) loopThreads);
            for (Bins &B : part) clearBins(B);
            parallel_for(j.count, loopThreads, 1 << 14, [&](size_t b, size_t e, int k) { fillBins(part[k], b, e); });
            for (const Bins &B : part)
                for (int ax = 0; ax < 3; ++ax) if (axisOk[ax]) for (int b = 0; b < NB; ++b) { bins.c[ax][b] += B.c[ax][b]; bins.mn[ax][b] = hmin(bins.mn[ax][b], B.mn[ax][b]); bins.mx[ax][b] = hmax(bins.mx[ax][b], B.mx[ax][b]); }
        } else fillBins(bins, 0, j.count);
        float bestCost = std::numeric_limits<float>::infinity(); int bestAxis = -1, bestBin = -1;
        for (int ax = 0; ax < 3; ++ax) {
            if (!axisOk[ax]) continue;
            const H3 *bmn = bins.mn[ax], *bmx = bins.mx[ax]; const uint32_t *bc = bins.c[ax];
            float rightArea[NB]; uint32_t rightCount[NB];
            H3 rmn = big, rmx = small; uint32_t rc = 0;
            for (int b = NB - 1; b > 0; --b) { rmn = hmin(rmn, bmn[b]); rmx = hmax(rmx, bmx[b]); rc += bc[b]; rightArea[b] = rc ? area(rmn, rmx) : 0.f; rightCount[b] = rc; }
            H3 lmn = big, lmx = small; uint32_t lc = 0;
            for (int b = 0; b < NB - 1; ++b) {
                lmn = hmin(lmn, bmn[b]); lmx = hmax(lmx, bmx[b]); lc += bc[b];
                if (lc == 0 || rightCount[b + 1] == 0) continue;
                const float cost = area(lmn, lmx) * lc + rightArea[b + 1] * rightCount[b + 1];
                if (cost < bestCost) { bestCost = cost; bestAxis = ax; bestBin = b; }
            }
        }
        // SAH with a traversal term: splitting pays when Ct * A + A_L N_L + A_R N_R < A * N (intersection cost 1)
        const float leafCost = area(bd.mn, bd.mx) * ((float) j.count - Ct);
        if (bestAxis >= 0 && (j.count > (uint32_t) maxLeaf || bestCost < leafCost)) {
            uint32_t *first = out.order.data() + j.first;
            uint32_t *mid = std::partition(first, first + j.count, [&](uint32_t t) { return binOf(t, bestAxis, lo[bestAxis], hi[bestAxis]) <= bestBin; });
            const uint32_t nl = (uint32_t) (mid - first);
            if (nl > 0 && nl < j.count) { nlOut = nl; return true; }
        }
        if (j.count > (uint32_t) maxLeaf) { nlOut = j.count / 2; return true; }     // degenerate centroids: split in the middle
        return false;
    };
    auto split = [&](const Job &j, uint32_t nl, Job &l, Job &r) {
        const uint32_t c0 = arenaUsed.fetch_add(2u);
        arena[j.node].left = c0; arena[j.node].count = 0;
        l = Job{c0, j.first, nl, j.depth + 1}; r = Job{c0 + 1, j.first + nl, j.count - nl, j.depth + 1};
    };
    auto noteDepth = [&](int d) { int cur = deepest.load(std::memory_order_relaxed); while (d > cur && !deepest.compare_exchange_weak(cur, d, std::memory_order_relaxed)) {} };

    // phase 1: the big nodes, one at a time, loops spread over the threads; everything smaller is queued
    const uint32_t bigCount = threads > 1 ? std::max<uint32_t>(1u << 16, nt / (4u * (uint32_t) threads)) : 0xFFFFFFFFu;
    std::vector<Job> top, queued; top.push_back(Job{0, 0, nt, 0});
    if (threads <= 1) { queued.swap(top); }
    while (!top.empty()) {
        const Job j = top.back(); top.pop_back();
        if (j.count < bigCount) { queued.push_back(j); continue; }
        noteDepth(j.depth);
        uint32_t nl = 0;
        if (process(j, threads, nl)) { Job l, r; split(j, nl, l, r); top.push_back(l); top.push_back(r); }
    }
    // phase 2: the subtrees below, each by one thread, largest first
    std::sort(queued.begin(), queued.end(), [](const Job &a, const Job &b) { return a.count > b.count; });
    std::atomic<size_t> nextJob{0};
    auto worker = [&] {
        std::vector<Job> stack;
        for (;;) {
            const size_t q = nextJob.fetch_add(1);
            if (q >= queued.size()) break;
            stack.push_back(queued[q]);
            int localDeepest = 0;
            while (!stack.empty()) {
                const Job j = stack.back(); stack.pop_back();
                localDeepest = std::max(localDeepest, j.depth);
                uint32_t nl = 0;
                if (process(j, 1, nl)) { Job l, r; split(j, nl, l, r); stack.push_back(l); stack.push_back(r); }
            }
            noteDepth(localDeepest);
        }
    };
    {
        const int T = (int) std::min<size_t>((size_t) std::max(threads, 1), queued.size());
        std::vector<std::thread> pool;
        for (int k = 1; k < T; ++k) { try { pool.emplace_back(worker); } catch (const std::system_error &) { break; } }   // the queue is dynamic: fewer threads, same result
        worker();
        for (auto &th : pool) th.join();
    }
    out.maxDepth = deepest.load();
    // phase 3: number the nodes as the depth-first stack of a serial build allocates them: a split node takes the next two indices when it is
    // popped, its right child is popped before its left one
    const uint32_t nNodes = arenaUsed.load();
    out.nodes.resize((size_t) nNodes * 8);
    struct Visit { uint32_t finalIndex, arenaIndex; };
    std::vector<Visit> st; st.push_back(Visit{0, 0});
    uint32_t finalUsed = 1;
    while (!st.empty()) {
        const Visit v = st.back(); st.pop_back();
        const Node &nd = arena[v.arenaIndex];
        uint32_t left = nd.left;
        if (nd.count == 0) { left = finalUsed; finalUsed += 2; st.push_back(Visit{left, nd.left}); st.push_back(Visit{left + 1, nd.left + 1}); }
        float *f = &out.nodes[8 * (size_t) v.finalIndex];
        f[0] = nd.mn.x; f[1] = nd.mn.y; f[2] = nd.mn.z; memcpy(&f[3], &left, 4);
        f[4] = nd.mx.x; f[5] = nd.mx.y; f[6] = nd.mx.z; memcpy(&f[7], &nd.count, 4);
    }
}
static void triangle_bounds(const float *positions, const uint32_t *indices, uint32_t nt, std::vector<H3> &tmin, std::vector<H3> &tmax, int threads) {
    auto P = [&](uint32_t i) { return h3(positions[3 * i], positions[3 * i + 1], positions[3 * i + 2]); };
    parallel_for(nt, threads, 1 << 15, [&](size_t b0, size_t e0, int) {
        for (size_t t = b0; t < e0; ++t) {
            const H3 a = P(indices[3 * t]), b = P(indices[3 * t + 1]), c = P(indices[3 * t + 2]);
            tmin[t] = h3(std::min(a.x, std::min(b.x, c.x)), std::min(a.y, std::min(b.y, c.y)), std::min(a.z, std::min(b.z, c.z)));
            tmax[t] = h3(std::max(a.x, std::max(b.x, c.x)), std::max(a.y, std::max(b.y, c.y)), std::max(a.z, std::max(b.z, c.z)));
        }
    });
}
}  // namespace

// ------------------------------------------------------------------ the integrator object
struct ppg_integrator {
    ppg_params prm;
    int device = 0, numSMs = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t evA = nullptr, evB = nullptr;
    TreeStats *hTreeStats = nullptr; bool treeStatsPending[PPG_MAX_ITERATIONS] = {};       // pinned; see build_sd_tree
    cudaEvent_t evLive[2] = {nullptr, nullptr}; uint32_t *liveHost = nullptr;   // pinned read-backs of the live counts, looked at one check point late
    std::atomic<bool> cancelled{false};
    std::string destination;
    int rank = 0, world = 1;
    ppg_allreduce_fn allreduce = nullptr; void *allreduceUser = nullptr;
    void *ncclComm = nullptr;                              // ncclComm_t when ppg_nccl_init was called: collectives are enqueued on `stream`, no host sync
    bool multi() const { return world > 1 && (ncclComm || allreduce); }
    ppg_clock_fn clockFn = nullptr; void *clockUser = nullptr; ppg_film_fn filmFn = nullptr; void *filmUser = nullptr;
    float clock_s() const { return clockFn ? (float) clockFn(clockUser) : (float) std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - startTime).count() / 1000; }
    unsigned long long adamProgress[2] = {0, 0};          // [sum steps * |df| * 2^20, sum steps] of the last Adam replay
    uint64_t lastRecorded = 0;                             // guiding records of the last performRenderPasses (this rank): bounds the growth of the S-tree

    // scene
    bool haveScene = false;
    DevBuf<float4> dAccel, dGeom, dBvh, dBsdf, dRadiance, dGroups, dEmitterInfo, dEmitterGeom, dSpheres, dTexMeta; DevBuf<uint2> dTexels, dEnvTexels; DevBuf<float> dEmitterCdf, dEmitterTriCdf, dBsdfTables, dEnvCdfRows, dEnvCdfCols, dEnvRowWeights; DevBuf<EnvLight> dEnvLight; DevBuf<uint32_t> dEmitterFlags; DevBuf<int4> dMeta;
    SceneView sceneView; Camera cam; uint32_t sceneSmemBytes = 0;
    float aabbMin[3], aabbMax[3];
    int W = 0, H = 0;
    DevBuf<uint32_t> dPixelMap, dPixelMapPerm; uint32_t nLocalPixels = 0, minLocalPixels = 0, maxLocalPixels = 0;

    // film
    DevBuf<float4> dImage, dSqImage, dFilm; DevBuf<float> dRgb; DevBuf<double> dVar;
    std::vector<DevBuf<float4> *> images; std::vector<float> variances;

    // SD-tree
    uint32_t capNodes = 0; size_t capPool = 0;
    DevBuf<uint2> dSnodes; DevBuf<float4> dLeafA; DevBuf<float> dBweight, dSampSum, dSampWeight, dAdam, dAdamBefore /* 4 x capNodes: iter, batchAcc, batchGrad, theta before a replay */;
    DevBuf<uint32_t> dAdamCount, dAdamCursor, dAdamOffset; DevBuf<float4> dAdamRecA, dAdamSortA; DevBuf<float2> dAdamRecB, dAdamSortB; size_t adamCap = 0;
    DevBuf<int> dSampDepth, dBuildDepth; DevBuf<uint32_t> dSampCount, dBuildCount, dBuildBase, dScalars /* [0]=nNodes [1]=totalBuild */;
    DevBuf<uint32_t> dStable; DevBuf<TreeStats> dTreeStats;
    DevBuf<SampNode> dSamp; DevBuf<uint2> dBchildren; DevBuf<float> dTrain /* bsums | packed tail */;
    uint32_t hNodes = 1; uint32_t hTotalBuild = 1;
    float extent[3];

    // wavefront
    size_t pathCapacity = 0; int maxBounces = 0, nSlabs = 0; int recordMode = 0; int stateVecs = 5, slabSets = 1;
    DevBuf<float4> dStateA, dStateB, dSlabs, dLiFinal; DevBuf<uint32_t> dLive, dWork; DevBuf<unsigned long long> dCounters;
    DevBuf<float4> dHits; DevBuf<uint32_t> dTraceWork; int gridTrace = 0; uint32_t traceMinPaths = 0;   // separate nearest-hit pass (ppg_trace.cu), BVH scenes only
    DevBuf<uint32_t> dOrder, dBinCount; bool binMaterials = false;                                        // ... which also bins the paths by the BSDF class they hit
    int gridBounce = 0, gridCommit = 0;

    // per-kernel-class CUDA-event timing on the launching stream
    struct Timed { cudaEvent_t a, b; int cls; uint32_t launches; };
    std::vector<Timed> evPool; size_t evUsed = 0; cudaEvent_t evRender0 = nullptr, evRender1 = nullptr;
    bool kernelTiming = true;
    void tic(int cls) {
        if (!kernelTiming) return;
        if (evUsed == evPool.size()) { Timed t; cudaEventCreate(&t.a); cudaEventCreate(&t.b); t.cls = cls; t.launches = 1; evPool.push_back(t); }
        evPool[evUsed].cls = cls; evPool[evUsed].launches = 1; cudaEventRecord(evPool[evUsed].a, stream);
    }
    void toc(uint32_t nLaunches = 1) { if (!kernelTiming) return; evPool[evUsed].launches = nLaunches; cudaEventRecord(evPool[evUsed].b, stream); ++evUsed; }   // one bracket may hold several launches of a class
    void resolve_timers() {   // call after a stream synchronize
        for (size_t i = 0; i < evUsed; ++i) {
            float ms = 0; if (cudaEventElapsedTime(&ms, evPool[i].a, evPool[i].b) == cudaSuccess) { stats.kernel_ms[evPool[i].cls] += ms; stats.kernel_count[evPool[i].cls] += evPool[i].launches; }
        }
        evUsed = 0;
    }

    // run state (GP:2313-2323)
    bool isBuilt = false, isFinalIter = false, doNee = false; int iter = 0, passesRendered = 0; uint32_t nRealEmitters = 0; bool fullFeature = false;
    bool useNee() const { return prm.nee != PPG_NEE_NEVER && nRealEmitters > 0; }
    std::chrono::steady_clock::time_point startTime;
    ppg_stats stats; uint64_t launches = 0; double deviceMs = 0;

    ~ppg_integrator();
    void destroy_body() {
        for (auto *b : images) delete b;
        for (auto &t : evPool) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
        if (evRender0) cudaEventDestroy(evRender0);
        if (evRender1) cudaEventDestroy(evRender1);
        if (evA) cudaEventDestroy(evA);
        if (evB) cudaEventDestroy(evB);
        for (auto &e : evLive) if (e) cudaEventDestroy(e);
        if (liveHost) cudaFreeHost(liveHost);
        if (hTreeStats) cudaFreeHost(hTreeStats);
        if (stream) cudaStreamDestroy(stream);
    }
};

ppg_integrator::~ppg_integrator() { destroy_body(); }
static double elapsed_ms(std::chrono::steady_clock::time_point s) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - s).count(); }
static float elapsed_s(std::chrono::steady_clock::time_point s) {
    return (float) std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - s).count() / 1000;
}

extern "C" int ppg_create(const ppg_params *params, int device, ppg_integrator **out) {
    if (!params || !out) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    int rc = ppg_params_validate(params);
    if (rc != PPG_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(PPG_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) device = 0; }
    if (device >= ndev) return fail(PPG_ERR_NO_DEVICE, "CUDA device index out of range");
    CK(cudaSetDevice(device));
    ppg_integrator *h = new ppg_integrator();
    h->prm = *params; h->device = device;
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
    h->numSMs = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaEventCreate(&h->evA)); CK(cudaEventCreate(&h->evB)); CK(cudaEventCreate(&h->evRender0)); CK(cudaEventCreate(&h->evRender1));
    for (auto &e : h->evLive) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CK(cudaHostAlloc((void **) &h->liveHost, 128 * sizeof(uint32_t), cudaHostAllocDefault));
    CK(cudaHostAlloc((void **) &h->hTreeStats, PPG_MAX_ITERATIONS * sizeof(TreeStats), cudaHostAllocDefault));
    if (const char *e = getenv("PPG_KERNEL_TIMING")) h->kernelTiming = atoi(e) != 0;
    memset(&h->stats, 0, sizeof(h->stats));
    *out = h;
    return PPG_OK;
}
static void release_comm(ppg_integrator *h);
extern "C" void ppg_destroy(ppg_integrator *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    release_comm(h);
    delete h;
}
extern "C" int ppg_set_destination(ppg_integrator *h, const char *destination) {
    if (!h) return PPG_ERR_INVALID_ARGUMENT; h->destination = destination ? destination : ""; return PPG_OK;
}
extern "C" int ppg_cancel(ppg_integrator *h) { if (!h) return PPG_ERR_INVALID_ARGUMENT; h->cancelled.store(true); return PPG_OK; }
extern "C" int ppg_set_allreduce(ppg_integrator *h, ppg_allreduce_fn cb, void *user) {
    if (!h) return PPG_ERR_INVALID_ARGUMENT; h->allreduce = cb; h->allreduceUser = user; return PPG_OK;
}

static int env_int(const char *name, int dflt) { const char *v = getenv(name); return v && *v ? atoi(v) : dflt; }   // tuning experiments only

// ------------------------------------------------------------------ NCCL, resolved at run time (no link-time dependency: single-GPU hosts need no NCCL)
namespace {
struct NcclId { char internal[PPG_NCCL_UNIQUE_ID_BYTES]; };                // ncclUniqueId (nccl.h:37-38), passed by value
struct NcclApi {
    void *lib = nullptr;
    int (*getUniqueId)(NcclId *) = nullptr;
    int (*commInitRank)(void **, int, NcclId, int) = nullptr;
    int (*allReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*commDestroy)(void *) = nullptr;
    const char *(*getErrorString)(int) = nullptr;
};
static NcclApi *nccl_api() {
    static NcclApi api; static bool tried = false;
    if (!tried) {
        tried = true;
        // a process that already holds NCCL (e.g. PyTorch's bundled copy) gets that one: same soname
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) { api.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
        if (api.lib) {
            api.getUniqueId = (int (*)(NcclId *)) dlsym(api.lib, "ncclGetUniqueId");
            api.commInitRank = (int (*)(void **, int, NcclId, int)) dlsym(api.lib, "ncclCommInitRank");
            api.allReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t)) dlsym(api.lib, "ncclAllReduce");
            api.commDestroy = (int (*)(void *)) dlsym(api.lib, "ncclCommDestroy");
            api.getErrorString = (const char *(*)(int)) dlsym(api.lib, "ncclGetErrorString");
            if (!api.getUniqueId || !api.commInitRank || !api.allReduce) api.lib = nullptr;
        }
    }
    return api.lib ? &api : nullptr;
}
}  // namespace

static void release_comm(ppg_integrator *h) {
    if (h->ncclComm) { NcclApi *a = nccl_api(); if (a && a->commDestroy) a->commDestroy(h->ncclComm); h->ncclComm = nullptr; }
}
extern "C" int ppg_nccl_unique_id(void *id_out) {
    NcclApi *a = nccl_api();
    if (!a || !id_out) return fail(PPG_ERR_COMM, "libnccl.so.2 could not be loaded");
    NcclId id; const int rc = a->getUniqueId(&id);
    if (rc != 0) return fail(PPG_ERR_COMM, std::string("ncclGetUniqueId: ") + (a->getErrorString ? a->getErrorString(rc) : "error"));
    memcpy(id_out, &id, sizeof(id));
    return PPG_OK;
}
extern "C" int ppg_nccl_init(ppg_integrator *h, const void *id, int rank, int world_size) {
    if (!h || !id || world_size < 1 || rank < 0 || rank >= world_size) return fail(PPG_ERR_INVALID_ARGUMENT, "bad communicator arguments");
    NcclApi *a = nccl_api();
    if (!a) return fail(PPG_ERR_COMM, "libnccl.so.2 could not be loaded");
    CK(cudaSetDevice(h->device));
    release_comm(h);
    NcclId nid; memcpy(&nid, id, sizeof(nid));
    void *comm = nullptr;
    const int rc = a->commInitRank(&comm, world_size, nid, rank);
    if (rc != 0) return fail(PPG_ERR_COMM, std::string("ncclCommInitRank: ") + (a->getErrorString ? a->getErrorString(rc) : "error"));
    h->ncclComm = comm;
    return ppg_set_shard(h, rank, world_size);
}
extern "C" int ppg_set_clock(ppg_integrator *h, ppg_clock_fn fn, void *user) { if (!h) return PPG_ERR_INVALID_ARGUMENT; h->clockFn = fn; h->clockUser = user; return PPG_OK; }
extern "C" int ppg_set_film_callback(ppg_integrator *h, ppg_film_fn fn, void *user) { if (!h) return PPG_ERR_INVALID_ARGUMENT; h->filmFn = fn; h->filmUser = user; return PPG_OK; }

// sum `n` floats in place over all ranks.  NCCL: enqueued on the render stream, nothing waits on the host.  Callback: the stream is drained
// first and the callback returns once the result is visible in device memory.
static int allreduce_sum(ppg_integrator *h, float *dev, size_t n) {
    if (h->world <= 1) return PPG_OK;
    if (h->ncclComm) {
        const int rc = nccl_api()->allReduce(dev, dev, n, /* ncclFloat32 */ 7, /* ncclSum */ 0, h->ncclComm, h->stream);
        if (rc != 0) return fail(PPG_ERR_COMM, "ncclAllReduce failed");
        return PPG_OK;
    }
    if (!h->allreduce) return PPG_OK;
    CK(cudaStreamSynchronize(h->stream));
    if (h->allreduce(h->allreduceUser, dev, n) != 0) return fail(PPG_ERR_COMM, "allreduce callback failed");
    return PPG_OK;
}

static int build_pixel_map(ppg_integrator *h) {
    // 32x32 image blocks (scene.cpp:24), dealt to the ranks round-robin along a scattered order of the blocks (golden-ratio stride, coprime to
    // the block count): every rank's blocks are spread over the whole image whatever the image width (plain `block % world` gives each rank
    // whole COLUMNS of blocks when the blocks per row are a multiple of the world size, and the columns of an image do not cost the same).
    // A rank visits its blocks row-major; row-major inside a block.
    const int bs = 32, bx = (h->W + bs - 1) / bs, by = (h->H + bs - 1) / bs, nb = bx * by;
    std::vector<int> owner((size_t) nb, 0);
    if (h->world > 1) {
        auto gcd = [](uint64_t a, uint64_t b) { while (b) { const uint64_t t = a % b; a = b; b = t; } return a; };
        uint64_t stride = std::max<uint64_t>(1, (uint64_t) ((double) nb * 0.6180339887498949));
        while (gcd(stride, (uint64_t) nb) != 1) ++stride;
        for (uint64_t j = 0; j < (uint64_t) nb; ++j) owner[(j * stride) % nb] = (int) (j % h->world);
    }
    std::vector<uint32_t> map; map.reserve((size_t) h->W * h->H / h->world + 1024);
    for (int b = 0; b < nb; ++b) {
        if (owner[b] != h->rank) continue;
        const int x0 = (b % bx) * bs, y0 = (b / bx) * bs;
        if (env_int("PPG_PIXEL_ORDER", 0) == 1) {      // experiment: Morton order inside the block (results do not depend on the order)
            for (uint32_t m = 0; m < (uint32_t) (bs * bs); ++m) {
                uint32_t x = 0, y = 0;
                for (int bit = 0; bit < 5; ++bit) { x |= ((m >> (2 * bit)) & 1u) << bit; y |= ((m >> (2 * bit + 1)) & 1u) << bit; }
                if (x0 + (int) x < h->W && y0 + (int) y < h->H) map.push_back((uint32_t) (x0 + x) | ((uint32_t) (y0 + y) << 16));
            }
            continue;
        }
        for (int y = y0; y < std::min(y0 + bs, h->H); ++y)
            for (int x = x0; x < std::min(x0 + bs, h->W); ++x) map.push_back((uint32_t) x | ((uint32_t) y << 16));
    }
    h->nLocalPixels = (uint32_t) map.size();
    h->minLocalPixels = 0xffffffffu; h->maxLocalPixels = 0;   // smallest / largest share of any rank: decisions every rank must take alike
    for (int r = 0; r < h->world; ++r) {
        uint64_t c = 0;
        for (int b = 0; b < nb; ++b) { if (owner[b] != r) continue; const int x0 = (b % bx) * bs, y0 = (b / bx) * bs; c += (uint64_t) (std::min(x0 + bs, h->W) - x0) * (std::min(y0 + bs, h->H) - y0); }
        h->minLocalPixels = std::min<uint32_t>(h->minLocalPixels, (uint32_t) c); h->maxLocalPixels = std::max<uint32_t>(h->maxLocalPixels, (uint32_t) c);
    }
    CK(h->dPixelMap.alloc(std::max<size_t>(map.size(), 1)));
    if (!map.empty()) CK(cudaMemcpy(h->dPixelMap.p, map.data(), map.size() * 4, cudaMemcpyHostToDevice));
    // A second, scattered order of the same pixels (golden-ratio stride over runs of 8 pixels, coprime to the run count): any contiguous range of it is spread evenly over
    // the image.  The sub-batches of a learning iteration (perform_render_passes) take their pixels from it, so that every S-tree leaf receives its
    // share of every sub-batch -- like the reference, whose worker threads interleave image blocks while the sampling fractions adapt.
    std::vector<uint32_t> perm(map.size());
    if (!map.empty()) {
        const uint64_t n = map.size();
        auto gcd = [](uint64_t a, uint64_t b) { while (b) { const uint64_t t = a % b; a = b; b = t; } return a; };
        // ... in runs of 8 consecutive map entries (8 neighbouring pixels of one block row): a quarter of a warp starts coherent,
        // which the BVH walk of the first bounce -- the largest launch of a sub-batch -- feels; a slice of 10^4 paths still holds
        // > 10^3 runs spread over the whole image
        const uint64_t run = (uint64_t) std::max(env_int("PPG_PERM_RUN", 8), 1), nr = (n + run - 1) / run;
        uint64_t rs = std::max<uint64_t>(1, (uint64_t) ((double) nr * 0.6180339887498949));
        while (gcd(rs, nr) != 1) ++rs;
        uint64_t w = 0;
        for (uint64_t r = 0; r < nr; ++r) { const uint64_t src = (r * rs) % nr; for (uint64_t k = src * run; k < std::min(n, (src + 1) * run); ++k) perm[w++] = map[k]; }
    }
    CK(h->dPixelMapPerm.alloc(std::max<size_t>(perm.size(), 1)));
    if (!perm.empty()) CK(cudaMemcpy(h->dPixelMapPerm.p, perm.data(), perm.size() * 4, cudaMemcpyHostToDevice));
    return PPG_OK;
}

extern "C" int ppg_set_shard(ppg_integrator *h, int rank, int world_size) {
    if (!h || world_size < 1 || rank < 0 || rank >= world_size) return fail(PPG_ERR_INVALID_ARGUMENT, "bad shard");
    CK(cudaSetDevice(h->device));
    h->rank = rank; h->world = world_size;
    if (h->haveScene) return build_pixel_map(h);
    return PPG_OK;
}

static int ppg_set_scene_impl(ppg_integrator *h, const ppg_scene_desc *s);
extern "C" int ppg_set_scene(ppg_integrator *h, const ppg_scene_desc *s) { return guarded("ppg_set_scene", [&] { return ppg_set_scene_impl(h, s); }); }
static int ppg_set_scene_impl(ppg_integrator *h, const ppg_scene_desc *s) {
    if (!h || !s) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    if (!s->n_triangles || !s->positions || !s->indices || !s->triangle_shape || !s->shapes || !s->bsdfs)
        return fail(PPG_ERR_INVALID_ARGUMENT, "scene needs triangles, shapes and bsdfs");
    if ((s->n_emitters && !s->area_radiance) || (s->n_spheres && !s->spheres)) return fail(PPG_ERR_INVALID_ARGUMENT, "emitter / sphere count without its array");
    if (s->camera.film_width <= 0 || s->camera.film_height <= 0 || s->camera.film_width > 65535 || s->camera.film_height > 65535)
        return fail(PPG_ERR_INVALID_ARGUMENT, "film size out of range");
    CK(cudaSetDevice(h->device));
    const uint32_t nt = s->n_triangles;
    for (uint32_t t = 0; t < nt; ++t) {
        if (s->triangle_shape[t] >= s->n_shapes) return fail(PPG_ERR_INVALID_ARGUMENT, "triangle_shape out of range");
        for (int k = 0; k < 3; ++k) if (s->indices[3 * t + k] >= s->n_vertices) return fail(PPG_ERR_INVALID_ARGUMENT, "vertex index out of range");
    }
    for (uint32_t i = 0; i < s->n_shapes; ++i) {
        if (s->shapes[i].bsdf < 0 || (uint32_t) s->shapes[i].bsdf >= s->n_bsdfs) return fail(PPG_ERR_INVALID_ARGUMENT, "shape bsdf out of range");
        if (s->shapes[i].emitter >= (int) s->n_emitters) return fail(PPG_ERR_INVALID_ARGUMENT, "shape emitter out of range");
    }
    for (uint32_t i = 0; i < s->n_bsdfs; ++i) {
        const int t = s->bsdfs[i].type;
        if (t != PPG_BSDF_DIFFUSE && t != PPG_BSDF_NULL_BLACK && t != PPG_BSDF_DIELECTRIC && t != PPG_BSDF_CONDUCTOR && t != PPG_BSDF_ROUGHCONDUCTOR && t != PPG_BSDF_ROUGHPLASTIC && t != PPG_BSDF_ROUGHDIELECTRIC && t != PPG_BSDF_PLASTIC && t != PPG_BSDF_THINDIELECTRIC)
            return fail(PPG_ERR_UNSUPPORTED, "BSDF type outside the implemented hot-path scope");
        if ((s->bsdfs[i].flags & PPG_BSDF_FLAG_MASK) && t == PPG_BSDF_THINDIELECTRIC) return fail(PPG_ERR_UNSUPPORTED, "mask around another null-type BSDF");
        if (t == PPG_BSDF_ROUGHPLASTIC && (!s->bsdf_tables || s->bsdfs[i].table < 0 || (uint32_t) s->bsdfs[i].table >= s->n_bsdf_tables))
            return fail(PPG_ERR_INVALID_ARGUMENT, "roughplastic needs its rough-transmittance table (ppg_scene_desc.bsdf_tables)");
        if ((t == PPG_BSDF_DIELECTRIC || t == PPG_BSDF_ROUGHDIELECTRIC || t == PPG_BSDF_THINDIELECTRIC) && !(s->bsdfs[i].eta[0] > 0)) return fail(PPG_ERR_INVALID_ARGUMENT, "dielectric needs eta > 0");
        if ((t == PPG_BSDF_DIELECTRIC || t == PPG_BSDF_ROUGHDIELECTRIC || t == PPG_BSDF_THINDIELECTRIC) && (s->bsdfs[i].flags & PPG_BSDF_FLAG_TWOSIDED)) return fail(PPG_ERR_INVALID_ARGUMENT, "twosided cannot wrap a transmissive BSDF (twosided.cpp)");
        if (s->bsdfs[i].reflectance_texture > s->n_textures || s->bsdfs[i].bump_texture > s->n_textures) return fail(PPG_ERR_INVALID_ARGUMENT, "BSDF texture index out of range");
        if (s->bsdfs[i].reflectance_texture && t != PPG_BSDF_DIFFUSE && t != PPG_BSDF_ROUGHPLASTIC && t != PPG_BSDF_PLASTIC)
            return fail(PPG_ERR_UNSUPPORTED, "reflectance_texture: only the diffuse reflectance of diffuse / roughplastic / plastic can be textured");
        if ((s->bsdfs[i].flags & PPG_BSDF_FLAG_BUMPMAP) && !s->bsdfs[i].bump_texture) return fail(PPG_ERR_INVALID_ARGUMENT, "bumpmap: A displacement texture must be specified");
    }
    if (s->n_textures && (!s->textures || !s->texels)) return fail(PPG_ERR_INVALID_ARGUMENT, "textures without texel data");
    for (uint32_t i = 0; i < s->n_textures; ++i) {
        const ppg_texture &t = s->textures[i];
        if (!t.width || !t.height || (t.channels != 1 && t.channels != 3) || t.wrap_u > 2 || t.wrap_v > 2) return fail(PPG_ERR_INVALID_ARGUMENT, "texture: bad size, channel count or wrap mode");
        if (t.first_texel + (uint64_t) t.width * t.height * t.channels > s->n_texels) return fail(PPG_ERR_INVALID_ARGUMENT, "texture: texel range out of bounds");
    }
    for (uint32_t k = 0; k < s->n_spheres; ++k)       // spheres carry no texture coordinates here
        if (s->spheres[k].shape >= 0 && (uint32_t) s->spheres[k].shape < s->n_shapes) {
            const ppg_bsdf &b = s->bsdfs[s->shapes[s->spheres[k].shape].bsdf];
            if (b.reflectance_texture || (b.flags & PPG_BSDF_FLAG_BUMPMAP)) return fail(PPG_ERR_UNSUPPORTED, "textured / bump-mapped BSDF on an analytic sphere");
        }
    const bool haveEnv = s->envmap.width && s->envmap.height;
    if (haveEnv && !s->envmap.texels) return fail(PPG_ERR_INVALID_ARGUMENT, "envmap without texel data");
    auto P = [&](uint32_t i) { return h3(s->positions[3 * i], s->positions[3 * i + 1], s->positions[3 * i + 2]); };
    std::vector<H3> tmin(nt), tmax(nt);
    triangle_bounds(s->positions, s->indices, nt, tmin, tmax, host_threads());
    HostBvh bvh; build_bvh(tmin, tmax, bvh, host_threads());
    if (bvh.maxDepth >= PPG_BVH_STACK) return fail(PPG_ERR_UNSUPPORTED, "BVH deeper than the device traversal stack");
    // brute-force layout for tiny scenes: coplanar groups ordered by projection axis (see bvh_intersect)
    uint32_t kBegin[4] = {0, 0, 0, 0};
    std::vector<float> groups;
    if (nt <= PPG_BRUTE_FORCE_TRIS) {
        struct Tri { int k; float w[9]; uint32_t t; };
        std::vector<Tri> tris(nt);
        for (uint32_t t = 0; t < nt; ++t) { tris[t].t = t; wald_constants(P(s->indices[3 * t]), P(s->indices[3 * t + 1]), P(s->indices[3 * t + 2]), tris[t].w, tris[t].k); }
        static const int mod3[4] = {1, 2, 0, 1};
        std::vector<uint32_t> order; std::vector<char> used(nt, 0);
        for (int k = 0; k < 3; ++k) {
            kBegin[k] = (uint32_t) (groups.size() / 8);
            for (uint32_t a = 0; a < nt; ++a) {
                if (used[a] || tris[a].k != k) continue;
                // gather the triangles lying in (numerically) the same plane as `a`
                std::vector<uint32_t> members;
                for (uint32_t b = a; b < nt; ++b) {
                    if (used[b] || tris[b].k != k) continue;
                    const float *wa = tris[a].w, *wb = tris[b].w;
                    const float scale = 1.0f + std::fabs(wa[2]);
                    if (std::fabs(wa[0] - wb[0]) <= 1e-6f && std::fabs(wa[1] - wb[1]) <= 1e-6f && std::fabs(wa[2] - wb[2]) <= 1e-6f * scale) { members.push_back(b); used[b] = 1; }
                }
                float umin = 1e30f, vmin = 1e30f, umax = -1e30f, vmax = -1e30f;
                for (uint32_t b : members)
                    for (int c = 0; c < 3; ++c) {
                        const H3 v = P(s->indices[3 * b + c]);
                        umin = std::min(umin, hcomp(v, mod3[k])); umax = std::max(umax, hcomp(v, mod3[k]));
                        vmin = std::min(vmin, hcomp(v, mod3[k + 1])); vmax = std::max(vmax, hcomp(v, mod3[k + 1]));
                    }
                const float pad = 0.01f * std::max(umax - umin, vmax - vmin) + 1e-3f * (1.0f + std::max(std::max(std::fabs(umin), std::fabs(umax)), std::max(std::fabs(vmin), std::fabs(vmax))));
                const uint32_t fc = (uint32_t) order.size() | ((uint32_t) members.size() << 16);
                float g[8] = {tris[a].w[0], tris[a].w[1], tris[a].w[2], 0.f, umin - pad, vmin - pad, umax + pad, vmax + pad};
                memcpy(&g[3], &fc, 4);
                groups.insert(groups.end(), g, g + 8);
                for (uint32_t b : members) order.push_back(tris[b].t);
            }
        }
        kBegin[3] = (uint32_t) (groups.size() / 8);
        for (uint32_t t = 0; t < nt; ++t) if (tris[t].k == 3) order.push_back(t);
        if (groups.size() / 8 <= 32) bvh.order = order;       // the candidate mask of the lock-step test has 32 bits
        else { groups.clear(); kBegin[0] = kBegin[1] = kBegin[2] = kBegin[3] = 0; }
    }
    const bool bruteForce = !groups.empty();
    if (groups.empty()) groups.assign(8, 0.f);
    std::vector<float> accel(12 * (size_t) nt), geom(24 * (size_t) nt); std::vector<int32_t> meta(4 * (size_t) nt);
    parallel_for(nt, host_threads(), 1 << 14, [&](size_t slot0, size_t slot1, int) {
    for (uint32_t slot = (uint32_t) slot0; slot < (uint32_t) slot1; ++slot) {
        const uint32_t t = bvh.order[slot];
        const uint32_t i0 = s->indices[3 * t], i1 = s->indices[3 * t + 1], i2 = s->indices[3 * t + 2];
        float w[9]; int k; wald_constants(P(i0), P(i1), P(i2), w, k);
        float *a = &accel[12 * (size_t) slot];
        a[0] = w[0]; a[1] = w[1]; a[2] = w[2]; memcpy(&a[3], &k, 4);
        a[4] = w[3]; a[5] = w[4]; a[6] = w[5]; a[7] = w[6];
        a[8] = w[7]; a[9] = w[8]; memcpy(&a[10], &t, 4); memcpy(&a[11], &slot, 4);
        const uint32_t vi[3] = {i0, i1, i2};
        float *g = &geom[24 * (size_t) slot];
        for (int k2 = 0; k2 < 3; ++k2) {
            const float *p = &s->positions[3 * vi[k2]];
            const float nz[3] = {0, 0, 0}; const float *n = s->normals ? &s->normals[3 * vi[k2]] : nz;
            const float uz[2] = {0, 0}; const float *uv = s->uvs ? &s->uvs[2 * vi[k2]] : uz;
            g[4 * k2] = p[0]; g[4 * k2 + 1] = p[1]; g[4 * k2 + 2] = p[2]; g[4 * k2 + 3] = n[0];
            g[12 + 4 * k2] = n[1]; g[12 + 4 * k2 + 1] = n[2]; g[12 + 4 * k2 + 2] = uv[0]; g[12 + 4 * k2 + 3] = uv[1];
        }
        const ppg_shape &sh = s->shapes[s->triangle_shape[t]];
        meta[4 * (size_t) slot] = sh.bsdf; meta[4 * (size_t) slot + 1] = sh.emitter;
        meta[4 * (size_t) slot + 2] = ((sh.has_normals && s->normals) ? 1 : 0) | ((sh.has_uvs && s->uvs) ? 2 : 0); meta[4 * (size_t) slot + 3] = (int32_t) s->triangle_shape[t];
    }
    });
    h->fullFeature = false;
    for (uint32_t i = 0; i < s->n_bsdfs; ++i) if ((s->bsdfs[i].type != PPG_BSDF_DIFFUSE && s->bsdfs[i].type != PPG_BSDF_NULL_BLACK) || (s->bsdfs[i].flags & ~PPG_BSDF_FLAG_TWOSIDED)) h->fullFeature = true;   // any non-diffuse model or wrapper other than twosided
    if (s->n_spheres) h->fullFeature = true;                                            // ... or analytic spheres: the full-feature kernel variants
    if (s->n_textures || haveEnv) h->fullFeature = true;                                // ... or textures / an environment emitter
    std::vector<float> bsdf(4 * PPG_BSDF_F4 * (size_t) s->n_bsdfs, 0.f);
    for (uint32_t i = 0; i < s->n_bsdfs; ++i) {
        float *b = &bsdf[4 * PPG_BSDF_F4 * (size_t) i]; const ppg_bsdf &m = s->bsdfs[i];
        b[0] = m.reflectance[0]; b[1] = m.reflectance[1]; b[2] = m.reflectance[2];
        uint32_t type = (uint32_t) m.type;
        if (m.type == PPG_BSDF_NULL_BLACK) { b[0] = b[1] = b[2] = 0.f; type = PPG_BSDF_DIFFUSE; }
        const uint32_t tf = type | ((m.flags & 0xffffffu) << 8); memcpy(&b[3], &tf, 4);
        b[4] = m.specular_transmittance[0]; b[5] = m.specular_transmittance[1]; b[6] = m.specular_transmittance[2]; b[7] = m.eta[0];
        b[8] = m.eta[0]; b[9] = m.eta[1]; b[10] = m.eta[2]; b[11] = m.eta[0] != 0.f ? 1.0f / m.eta[0] : 0.f;
        b[12] = m.k[0]; b[13] = m.k[1]; b[14] = m.k[2];
        b[15] = std::max(m.alpha, 1e-4f) * (m.distribution == PPG_MICROFACET_BECKMANN ? -1.0f : 1.0f);   // microfacet.h:63 clamp; sign encodes the distribution
        b[16] = m.specular_reflectance[0]; b[17] = m.specular_reflectance[1]; b[18] = m.specular_reflectance[2]; b[19] = m.fdr_int;
        b[20] = m.specular_sampling_weight; const uint32_t tab = (uint32_t) std::max(m.table, 0); memcpy(&b[21], &tab, 4);
        memcpy(&b[22], &m.reflectance_texture, 4); memcpy(&b[23], &m.bump_texture, 4);
        b[24] = m.opacity[0]; b[25] = m.opacity[1]; b[26] = m.opacity[2];
        b[27] = m.opacity[0] * 0.212671f + m.opacity[1] * 0.715160f + m.opacity[2] * 0.072169f;                // getLuminance (spectrum.h:725-727)
    }
    std::vector<float> rad(4 * (size_t) std::max<uint32_t>(s->n_emitters, 1), 0.f);
    for (uint32_t i = 0; i < s->n_emitters; ++i) { rad[4 * i] = s->area_radiance[3 * i]; rad[4 * i + 1] = s->area_radiance[3 * i + 1]; rad[4 * i + 2] = s->area_radiance[3 * i + 2]; }
    const size_t nBvh = bvh.nodes.size() / 8;
    CK(h->dAccel.alloc(3 * (size_t) nt)); CK(h->dGeom.alloc(6 * (size_t) nt)); CK(h->dMeta.alloc(nt)); CK(h->dBvh.alloc(2 * nBvh));
    CK(h->dBsdf.alloc(PPG_BSDF_F4 * (size_t) s->n_bsdfs));
    CK(h->dBsdfTables.alloc(std::max<size_t>((size_t) s->n_bsdf_tables * PPG_BSDF_TABLE_SIZE, 1)));
    if (s->n_bsdf_tables) { CK(cudaMemcpy(h->dBsdfTables.p, s->bsdf_tables, (size_t) s->n_bsdf_tables * PPG_BSDF_TABLE_SIZE * 4, cudaMemcpyHostToDevice)); }
    CK(h->dRadiance.alloc(std::max<uint32_t>(s->n_emitters, 1)));
    CK(cudaMemcpy(h->dAccel.p, accel.data(), accel.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->dGeom.p, geom.data(), geom.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->dMeta.p, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->dBvh.p, bvh.nodes.data(), bvh.nodes.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->dBsdf.p, bsdf.data(), bsdf.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->dRadiance.p, rad.data(), rad.size() * 4, cudaMemcpyHostToDevice));
    SceneView &v = h->sceneView;
    v.accel = h->dAccel.p; v.geom = h->dGeom.p; v.meta = h->dMeta.p; v.bvh = h->dBvh.p; v.bsdf = h->dBsdf.p; v.bsdfTables = h->dBsdfTables.p; v.radiance = h->dRadiance.p;
    CK(h->dGroups.alloc(groups.size() / 4));
    CK(cudaMemcpy(h->dGroups.p, groups.data(), groups.size() * 4, cudaMemcpyHostToDevice));
    v.groups = h->dGroups.p; v.nGroups = bruteForce ? (uint32_t) (groups.size() / 8) : 0u;
    for (int k = 0; k < 4; ++k) v.kBegin[k] = kBegin[k];
    {   // emitter sampling tables for next event estimation (TriMesh::prepareSamplingTable trimesh.cpp:388-403; Scene::configure scene.cpp:357-381)
        const uint32_t ne = std::max<uint32_t>(s->n_emitters, 1);
        std::vector<float> ecdf(1, 0.f), tcdf, egeom; std::vector<float> einfo(4 * (size_t) ne, 0.f); std::vector<uint32_t> eflags(ne, 0u);
        for (uint32_t e = 0; e < s->n_emitters; ++e) {
            int shape = -1;
            for (uint32_t si = 0; si < s->n_shapes; ++si) if (s->shapes[si].emitter == (int) e) shape = (int) si;
            const uint32_t first = (uint32_t) (egeom.size() / 24), cdfOff = (uint32_t) tcdf.size();
            uint32_t ntri = 0; float invArea = 0.f;
            int sphere = -1;
            for (uint32_t k = 0; k < s->n_spheres; ++k) if (shape >= 0 && s->spheres[k].shape == shape) sphere = (int) k;
            if (sphere >= 0) {                                                                      // sphere.cpp:128: m_invSurfaceArea
                const uint32_t tag = PPG_SPHERE_BIT | (uint32_t) sphere; const float r = s->spheres[sphere].radius;
                invArea = 1 / (4 * 3.14159265358979323846f * r * r);
                memcpy(&einfo[4 * e], &tag, 4); memcpy(&einfo[4 * e + 1], &ntri, 4); einfo[4 * e + 2] = invArea; memcpy(&einfo[4 * e + 3], &cdfOff, 4);
                ecdf.push_back(ecdf.back() + 1.0f);
                continue;
            }
            if (shape >= 0) {
                const ppg_shape &sh = s->shapes[shape];
                if ((uint64_t) sh.first_triangle + sh.n_triangles > nt) return fail(PPG_ERR_INVALID_ARGUMENT, "shape triangle range out of bounds");
                ntri = sh.n_triangles; eflags[e] = (sh.has_normals && s->normals) ? 1u : 0u;
                std::vector<float> c(1, 0.f);
                for (uint32_t t = sh.first_triangle; t < sh.first_triangle + sh.n_triangles; ++t) {
                    const uint32_t vi[3] = {s->indices[3 * t], s->indices[3 * t + 1], s->indices[3 * t + 2]};
                    const H3 p0 = P(vi[0]), p1 = P(vi[1]), p2 = P(vi[2]);
                    const H3 cr = hcross(p1 - p0, p2 - p0);
                    c.push_back(c.back() + 0.5f * std::sqrt(hdot(cr, cr)));                       // Triangle::surfaceArea
                    float g[24];
                    for (int k2 = 0; k2 < 3; ++k2) {
                        const float *p = &s->positions[3 * vi[k2]];
                        const float nz[3] = {0, 0, 0}; const float *n = s->normals ? &s->normals[3 * vi[k2]] : nz;
                        g[4 * k2] = p[0]; g[4 * k2 + 1] = p[1]; g[4 * k2 + 2] = p[2]; g[4 * k2 + 3] = n[0];
                        g[12 + 4 * k2] = n[1]; g[12 + 4 * k2 + 1] = n[2]; g[12 + 4 * k2 + 2] = 0.f; g[12 + 4 * k2 + 3] = 0.f;
                    }
                    egeom.insert(egeom.end(), g, g + 24);
                }
                const float sum = c.back();                                                        // DiscreteDistribution::normalize
                if (sum > 0) { const float nrm = 1.0f / sum; for (size_t i = 1; i < c.size(); ++i) c[i] *= nrm; c.back() = 1.0f; invArea = 1.0f / sum; }
                tcdf.insert(tcdf.end(), c.begin(), c.end());
            }
            memcpy(&einfo[4 * e], &first, 4); memcpy(&einfo[4 * e + 1], &ntri, 4); einfo[4 * e + 2] = invArea; memcpy(&einfo[4 * e + 3], &cdfOff, 4);
            ecdf.push_back(ecdf.back() + 1.0f);                                                    // getSamplingWeight() == 1
        }
        v.envLight = 0xFFFFFFFFu;
        if (haveEnv) { v.envLight = s->n_emitters; ecdf.push_back(ecdf.back() + 1.0f); }          // the environment emitter: last entry of the light list
        v.nLights = (uint32_t) ecdf.size() - 1u;
        float norm = 0.f;
        if (ecdf.back() > 0) { norm = 1.0f / ecdf.back(); for (size_t i = 1; i < ecdf.size(); ++i) ecdf[i] *= norm; ecdf.back() = 1.0f; }
        if (ecdf.size() < 2) { ecdf.push_back(1.0f); v.nLights = 1u; }                             // no light at all: one empty entry (never sampled, useNee() is false)
        if (tcdf.empty()) tcdf.assign(2, 0.f);
        if (egeom.empty()) egeom.assign(24, 0.f);
        CK(h->dEmitterCdf.alloc(ecdf.size())); CK(h->dEmitterInfo.alloc(ne)); CK(h->dEmitterTriCdf.alloc(tcdf.size())); CK(h->dEmitterGeom.alloc(egeom.size() / 4)); CK(h->dEmitterFlags.alloc(ne));
        CK(cudaMemcpy(h->dEmitterCdf.p, ecdf.data(), ecdf.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->dEmitterInfo.p, einfo.data(), einfo.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->dEmitterTriCdf.p, tcdf.data(), tcdf.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->dEmitterGeom.p, egeom.data(), egeom.size() * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->dEmitterFlags.p, eflags.data(), eflags.size() * 4, cudaMemcpyHostToDevice));
        v.emitterCdf = h->dEmitterCdf.p; v.emitterInfo = h->dEmitterInfo.p; v.emitterTriCdf = h->dEmitterTriCdf.p; v.emitterGeom = h->dEmitterGeom.p; v.emitterFlags = h->dEmitterFlags.p;
        v.emitterNormalization = norm; h->nRealEmitters = s->n_emitters + (haveEnv ? 1u : 0u);
    }
    {   // analytic spheres
        std::vector<float> sph(8 * (size_t) std::max<uint32_t>(s->n_spheres, 1), 0.f);
        for (uint32_t k = 0; k < s->n_spheres; ++k) {
            const ppg_sphere &sp = s->spheres[k];
            if (sp.shape < 0 || (uint32_t) sp.shape >= s->n_shapes || !(sp.radius > 0)) return fail(PPG_ERR_INVALID_ARGUMENT, "sphere: bad shape index or radius");
            float *o = &sph[8 * (size_t) k];
            o[0] = sp.center[0]; o[1] = sp.center[1]; o[2] = sp.center[2]; o[3] = sp.radius;
            const int32_t bs = s->shapes[sp.shape].bsdf, em = s->shapes[sp.shape].emitter; const uint32_t fl = sp.flip_normals ? 1u : 0u;
            memcpy(&o[4], &bs, 4); memcpy(&o[5], &em, 4); memcpy(&o[6], &fl, 4);
        }
        CK(h->dSpheres.alloc(sph.size() / 4));
        CK(cudaMemcpy(h->dSpheres.p, sph.data(), sph.size() * 4, cudaMemcpyHostToDevice));
        v.spheres = h->dSpheres.p; v.nSpheres = s->n_spheres;
    }
    {   // bitmap textures and the environment map: half texels repacked to one uint2 {r | g << 16, b} per texel
        auto pack = [](const uint16_t *src, size_t nTexels, uint32_t channels, uint2 *dst) {
            parallel_for(nTexels, host_threads(), 1 << 18, [&](size_t i0, size_t i1, int) {
                for (size_t i = i0; i < i1; ++i) {
                    const uint16_t r = src[i * channels], g = channels == 3 ? src[i * channels + 1] : r, b = channels == 3 ? src[i * channels + 2] : r;
                    dst[i] = make_uint2((uint32_t) r | ((uint32_t) g << 16), (uint32_t) b);
                }
            });
        };
        size_t total = 0;
        for (uint32_t i = 0; i < s->n_textures; ++i) total += (size_t) s->textures[i].width * s->textures[i].height;
        if (total >= (1ull << 32)) return fail(PPG_ERR_UNSUPPORTED, "more than 2^32 texels");
        std::vector<uint2> tex(std::max<size_t>(total, 1)); std::vector<float> tmeta(8 * (size_t) std::max<uint32_t>(s->n_textures, 1), 0.f);
        size_t off = 0;
        for (uint32_t i = 0; i < s->n_textures; ++i) {
            const ppg_texture &t = s->textures[i];
            pack(s->texels + t.first_texel, (size_t) t.width * t.height, t.channels, tex.data() + off);
            float *m = &tmeta[8 * (size_t) i];
            const uint32_t wr = t.wrap_u | (t.wrap_v << 8), o32 = (uint32_t) off;
            memcpy(&m[0], &t.width, 4); memcpy(&m[1], &t.height, 4); memcpy(&m[2], &wr, 4); memcpy(&m[3], &o32, 4);
            m[4] = t.uv_scale[0]; m[5] = t.uv_scale[1]; m[6] = t.uv_offset[0]; m[7] = t.uv_offset[1];
            off += (size_t) t.width * t.height;
        }
        CK(h->dTexels.alloc(tex.size())); CK(h->dTexMeta.alloc(tmeta.size() / 4));
        CK(cudaMemcpy(h->dTexels.p, tex.data(), tex.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->dTexMeta.p, tmeta.data(), tmeta.size() * 4, cudaMemcpyHostToDevice));
        v.texMeta = h->dTexMeta.p; v.texels = h->dTexels.p; v.nTextures = s->n_textures;
        v.envW = v.envH = 0; v.envScale = 1.f; v.envTexels = nullptr;
        for (int i = 0; i < 9; ++i) v.worldToEnv[i] = (i % 4 == 0) ? 1.f : 0.f;
        if (haveEnv) {
            std::vector<uint2> env((size_t) s->envmap.width * s->envmap.height);
            pack(s->envmap.texels, env.size(), 3, env.data());
            CK(h->dEnvTexels.alloc(env.size()));
            CK(cudaMemcpy(h->dEnvTexels.p, env.data(), env.size() * sizeof(uint2), cudaMemcpyHostToDevice));
            v.envTexels = h->dEnvTexels.p; v.envW = s->envmap.width; v.envH = s->envmap.height; v.envScale = s->envmap.scale;
            for (int i = 0; i < 9; ++i) v.worldToEnv[i] = s->envmap.world_to_env[i];
        }
        // light sampling of the environment emitter: the tables of EnvironmentMap::configure (src/emitters/envmap.cpp:260-329), in the reference's float / double mix
        v.env = nullptr;
        if (haveEnv) {
            EnvLight el; memset(&el, 0, sizeof(el));
            const uint32_t Wd = s->envmap.width, Hd = s->envmap.height;
            const double kPi = 3.14159265358979323846;
            auto lum = [&](uint32_t x, uint32_t y) {                                               // Color3::getLuminance of texel (x, y)
                const uint16_t *px = s->envmap.texels + ((size_t) y * Wd + x) * 3;
                return half_to_float(px[0]) * 0.212671f + half_to_float(px[1]) * 0.715160f + half_to_float(px[2]) * 0.072169f;
            };
            std::vector<float> cols((size_t) (Wd + 1) * Hd, 0.f), rows((size_t) Hd + 1, 0.f), weights(Hd, 0.f);
            size_t colPos = 0, rowPos = 0; float rowSum = 0.0f;
            rows[rowPos++] = 0;
            for (uint32_t y = 0; y < Hd; ++y) {
                float colSum = 0;
                cols[colPos++] = 0;
                for (uint32_t x = 0; x < Wd; ++x) { colSum += lum(x, y); cols[colPos++] = colSum; }
                const float normalization = 1.0f / colSum;
                for (uint32_t x = 1; x < Wd; ++x) cols[colPos - x - 1] *= normalization;
                cols[colPos - 1] = 1.0f;
                const float weight = (float) std::sin((double) ((float) y + 0.5f) * kPi / (double) Hd);
                weights[y] = weight;
                rowSum += colSum * weight;
                rows[rowPos++] = rowSum;
            }
            if (rowSum == 0) return fail(PPG_ERR_INVALID_ARGUMENT, "The environment map is completely black -- this is not allowed.");
            if (!std::isfinite(rowSum)) return fail(PPG_ERR_INVALID_ARGUMENT, "The environment map contains an invalid floating point value (nan/inf) -- giving up.");
            const float normalization = 1.0f / rowSum;
            for (uint32_t y = 1; y < Hd; ++y) rows[rowPos - y - 1] *= normalization;
            rows[rowPos - 1] = 1.0f;
            el.normalization = (float) (1.0 / ((double) rowSum * (2 * kPi / (double) Wd) * (kPi / (double) Hd)));
            el.pixelX = (float) (2 * kPi / (double) Wd); el.pixelY = (float) (kPi / (double) Hd);
            float ctr[3], dd = 0.f;                                                                // AABB::getBSphere (libcore/aabb.cpp:44-47), radius x 1.5 (envmap.cpp:333)
            for (int i = 0; i < 3; ++i) { ctr[i] = (s->aabb_max[i] + s->aabb_min[i]) * 0.5f; el.center[i] = ctr[i]; }
            { const float ex = ctr[0] - s->aabb_max[0], ey = ctr[1] - s->aabb_max[1], ez = ctr[2] - s->aabb_max[2]; dd = std::sqrt(ex * ex + ey * ey + ez * ez); }
            el.radius = std::max(1e-4f, dd * 1.5f);
            const float *m = s->envmap.world_to_env;                                               // the emitter-to-world rotation back from its inverse
            const double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], hh = m[7], ii = m[8];
            const double det = a * (e * ii - f * hh) - b * (d * ii - f * g) + c * (d * hh - e * g);
            if (!(std::fabs(det) > 0)) return fail(PPG_ERR_INVALID_ARGUMENT, "envmap: singular world_to_env");
            const double id = 1.0 / det;
            const double inv[9] = {(e * ii - f * hh) * id, (c * hh - b * ii) * id, (b * f - c * e) * id, (f * g - d * ii) * id, (a * ii - c * g) * id, (c * d - a * f) * id,
                                   (d * hh - e * g) * id, (b * g - a * hh) * id, (a * e - b * d) * id};
            for (int k = 0; k < 9; ++k) el.toWorld[k] = (float) inv[k];
            CK(h->dEnvCdfRows.alloc(rows.size())); CK(h->dEnvCdfCols.alloc(cols.size())); CK(h->dEnvRowWeights.alloc(weights.size()));
            CK(cudaMemcpy(h->dEnvCdfRows.p, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->dEnvCdfCols.p, cols.data(), cols.size() * 4, cudaMemcpyHostToDevice));
            CK(cudaMemcpy(h->dEnvRowWeights.p, weights.data(), weights.size() * 4, cudaMemcpyHostToDevice));
            el.cdfRows = h->dEnvCdfRows.p; el.cdfCols = h->dEnvCdfCols.p; el.rowWeights = h->dEnvRowWeights.p;
            CK(h->dEnvLight.alloc(1));
            CK(cudaMemcpy(h->dEnvLight.p, &el, sizeof(el), cudaMemcpyHostToDevice));
            v.env = h->dEnvLight.p;
        }
    }
    v.nTris = nt; v.nBvhNodes = (uint32_t) nBvh; v.nBsdfs = s->n_bsdfs; v.nEmitters = std::max<uint32_t>(s->n_emitters, 1);
    const size_t sceneBytes = 16 * ((size_t) 3 * nt + 6 * nt + nt + 2 * nBvh + PPG_BSDF_F4 * s->n_bsdfs + v.nEmitters + 2 * std::max<uint32_t>(v.nGroups, 1));
    h->sceneSmemBytes = sceneBytes <= 48 * 1024 ? (uint32_t) sceneBytes : 0u;   // small scenes (CBOX: ~9 KB) live in shared memory
    // camera (src/sensors/perspective.cpp:120-298; lookAt columns: left, up, dir, origin -- transform.cpp:191-214)
    const float *m = s->camera.to_world;
    Camera &c = h->cam;
    c.left = make_float3(m[0], m[4], m[8]); c.up = make_float3(m[1], m[5], m[9]); c.dir = make_float3(m[2], m[6], m[10]); c.o = make_float3(m[3], m[7], m[11]);
    const float aspect = (float) s->camera.film_width / (float) s->camera.film_height;
    c.tanX = std::tan(0.5f * s->camera.x_fov_deg * (3.14159265358979323846f / 180.0f)); c.tanY = c.tanX / aspect;
    c.nearClip = s->camera.near_clip; c.farClip = s->camera.far_clip; c.W = s->camera.film_width; c.H = s->camera.film_height;
    h->W = c.W; h->H = c.H;
    for (int i = 0; i < 3; ++i) { h->aabbMin[i] = s->aabb_min[i]; h->aabbMax[i] = s->aabb_max[i]; }
    // STree::STree (GP:850-860): cubify from the min corner
    const float sx = h->aabbMax[0] - h->aabbMin[0], sy = h->aabbMax[1] - h->aabbMin[1], sz = h->aabbMax[2] - h->aabbMin[2];
    const float mxs = std::max(std::max(sx, sy), sz);
    for (int i = 0; i < 3; ++i) { const float mx = h->aabbMin[i] + mxs; h->extent[i] = mx - h->aabbMin[i]; }
    const size_t npx = (size_t) h->W * h->H;
    CK(h->dImage.alloc(npx)); CK(h->dSqImage.alloc(npx)); CK(h->dFilm.alloc(npx)); CK(h->dRgb.alloc(3 * npx)); CK(h->dVar.alloc(1));
    h->haveScene = true;
    return build_pixel_map(h);
}

// ------------------------------------------------------------------ SD-tree storage
static int ensure_tree_capacity(ppg_integrator *h, uint32_t nodes, size_t pool) {
    if (nodes > h->capNodes) {
        const uint32_t cap = std::max<uint32_t>(nodes, std::max<uint32_t>(2 * h->capNodes, 1u << 16));
        CK(h->dSnodes.grow(cap, h->stream)); CK(h->dLeafA.grow(cap, h->stream)); CK(h->dBweight.grow(cap, h->stream));
        CK(h->dSampSum.grow(cap, h->stream)); CK(h->dSampWeight.grow(cap, h->stream)); CK(h->dAdam.grow(6 * (size_t) cap, h->stream));
        CK(h->dAdamBefore.grow(4 * (size_t) cap, h->stream)); CK(h->dSampDepth.grow(cap, h->stream));
        {   // record-bucket bookkeeping must stay zero between commit launches: reallocate zeroed
            h->dAdamCount.release(); h->dAdamCursor.release(); h->dAdamOffset.release();
            CK(h->dAdamCount.alloc(cap)); CK(h->dAdamCursor.alloc(cap)); CK(h->dAdamOffset.alloc(cap));
            CK(cudaMemsetAsync(h->dAdamCount.p, 0, 4 * (size_t) cap, h->stream)); CK(cudaMemsetAsync(h->dAdamCursor.p, 0, 4 * (size_t) cap, h->stream));
        }
        CK(h->dBuildDepth.grow(cap, h->stream)); CK(h->dSampCount.grow(cap, h->stream)); CK(h->dBuildCount.grow(cap, h->stream));
        CK(h->dBuildBase.grow(cap, h->stream));
        h->capNodes = cap;
    }
    if (pool > h->capPool) {
        const size_t cap = std::max<size_t>(pool, std::max<size_t>(2 * h->capPool, (size_t) 1 << 20));
        CK(h->dSamp.grow(cap, h->stream)); CK(h->dBchildren.grow(cap, h->stream));
        h->capPool = cap;
    }
    // bsums (4 floats per pool node) followed by the packed exchange tail (building weights, or 6 Adam arrays; + scalars)
    CK(h->dTrain.grow(4 * h->capPool + 6 * (size_t) h->capNodes + 64, h->stream));
    return PPG_OK;
}

static MaintParams maint(ppg_integrator *h) {
    MaintParams M;
    M.snodes = h->dSnodes.p; M.leafA = h->dLeafA.p; M.bweight = h->dBweight.p; M.sampSum = h->dSampSum.p; M.sampWeight = h->dSampWeight.p;
    M.sampDepth = h->dSampDepth.p; M.sampCount = h->dSampCount.p; M.adam = h->dAdam.p; M.buildCount = h->dBuildCount.p; M.buildDepth = h->dBuildDepth.p;
    M.nNodes = h->dScalars.p; M.capNodes = h->capNodes; M.samp = h->dSamp.p; M.bchildren = h->dBchildren.p; M.bsums = reinterpret_cast<float4 *>(h->dTrain.p);
    return M;
}

// new STree (GP:1519): one leaf whose sampling tree is a single empty quadtree node
static int init_tree(ppg_integrator *h) {
    CK(h->dScalars.alloc(8)); CK(h->dTreeStats.alloc(1));
    CK(cudaMemsetAsync(h->dScalars.p, 0, 32, h->stream));
    // buffers persist across renders (cudaMalloc/cudaFree are synchronous and slow): only their contents are reset
    int rc = ensure_tree_capacity(h, std::max<uint32_t>(h->capNodes, 1u << 16), std::max<size_t>(h->capPool, (size_t) 1 << 20));
    if (rc) return rc;
    CK(cudaMemsetAsync(h->dSnodes.p, 0, sizeof(uint2) * h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dLeafA.p, 0, sizeof(float4) * h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dBweight.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dSampSum.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dSampWeight.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dAdam.p, 0, 24 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dAdamCount.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dAdamCursor.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dSampDepth.p, 0, 4 * (size_t) h->capNodes, h->stream));
    CK(cudaMemsetAsync(h->dSamp.p, 0, sizeof(SampNode), h->stream));          // one empty quadtree node at pool offset 0
    const uint32_t one[2] = {1u, 1u};
    CK(cudaMemcpyAsync(h->dScalars.p, one, 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->dSampCount.p, one, 4, cudaMemcpyHostToDevice, h->stream));
    h->hNodes = 1; h->hTotalBuild = 1;
    CK(cudaStreamSynchronize(h->stream));
    return PPG_OK;
}

static TreeView tree_view(ppg_integrator *h) {
    TreeView T;
    T.snodes = h->dSnodes.p; T.stable = h->dStable.p; T.leafA = h->dLeafA.p; T.samp = h->dSamp.p; T.bchildren = h->dBchildren.p;
    T.bsums = reinterpret_cast<float4 *>(h->dTrain.p); T.bweight = h->dBweight.p;
    T.aabbMin = make_float3(h->aabbMin[0], h->aabbMin[1], h->aabbMin[2]); T.extent = make_float3(h->extent[0], h->extent[1], h->extent[2]);
    return T;
}

// resetSDTree, GP:1108-1113
static int reset_sd_tree(ppg_integrator *h) {
    const double thr = std::sqrt(std::pow(2.0, h->iter) * h->prm.spp_per_pass / 4) * h->prm.s_tree_threshold;
    const float threshold = (float) (size_t) thr;                   // (size_t) cast then Float comparison, GP:1111 + 953-955
    // upper bound of the node count after refinement: every leaf can at most double per halving of its weight;
    // the total weight of the last iteration bounds the number of new leaves by 2*W/threshold
    bool memCapped = false;
    if (h->prm.sd_tree_max_memory >= 0) {   // GP:958-967 (footprint approximated by node counts: 2 trees x 24 B per node + per-tree overhead)
        const size_t fp = (size_t) h->hTotalBuild * 2 * 24 + (size_t) h->hNodes * 96;
        memCapped = fp / 1000000 >= (size_t) h->prm.sd_tree_max_memory;
    }
    if (!memCapped) {
        // capacity: the refinement creates at most 2 nodes per threshold worth of recorded weight.  The total weight of the iteration is at most
        // its number of guiding records (weights <= 1); with several ranks the reduced weights hold about world x this rank's records.
        const double totalW = 1.25 * (double) h->lastRecorded * h->world + 4096;
        const double est = h->hNodes + 4.0 * totalW / std::max(1.0f, threshold) + 1024;
        int rc = ensure_tree_capacity(h, (uint32_t) std::min<double>(est, 4.0e9), h->capPool);
        if (rc) return rc;
        MaintParams M = maint(h);
        h->tic(PPG_K_REFINE); stree_refine_kernel<<<1, 1024, 0, h->stream>>>(M, threshold, h->dScalars.p + 5); h->toc(); h->launches++;
    }
    MaintParams M = maint(h);
    const int blocks = h->numSMs * 4;
    h->tic(PPG_K_RESET);
    dtree_reset_kernel<false><<<blocks, 128, 0, h->stream>>>(M, nullptr, 20, h->prm.d_tree_threshold); h->launches++;
    exclusive_scan_kernel<<<1, 1024, 0, h->stream>>>(h->dBuildCount.p, h->dBuildBase.p, h->dScalars.p, h->dScalars.p + 1); h->launches++;
    h->toc();
    uint32_t sc[8];
    CK(cudaMemcpyAsync(sc, h->dScalars.p, 32, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (sc[5]) return fail(PPG_ERR_CUDA, "S-tree refinement ran out of node capacity");
    h->hNodes = sc[0]; h->hTotalBuild = sc[1];
    int rc = ensure_tree_capacity(h, h->hNodes, std::max<size_t>(h->hTotalBuild, 1));
    if (rc) return rc;
    M = maint(h);
    h->tic(PPG_K_RESET);
    dtree_reset_kernel<true><<<blocks, 128, 0, h->stream>>>(M, h->dBuildBase.p, 20, h->prm.d_tree_threshold); h->launches++;
    leaf_after_reset_kernel<<<blocks, 256, 0, h->stream>>>(M, h->dBuildBase.p); h->launches++;
    h->toc();
    // prefix table of the refined S-tree (stree_lookup): the first 3 * PPG_STREE_TABLE_BITS levels of every descent become one load
    CK(h->dStable.alloc((size_t) 1 << (3 * PPG_STREE_TABLE_BITS)));
    h->tic(PPG_K_REFINE); stree_table_kernel<<<h->numSMs * 8, 256, 0, h->stream>>>(h->dSnodes.p, h->dStable.p); h->toc(); h->launches++;
    CK(cudaGetLastError());
    return PPG_OK;      // no synchronize: the passes queue behind the reset
}

// the one exchange step (SURVEY 8e): sum the building statistics over all ranks
__global__ void pack_tail_kernel(float *tail, float *bweight, uint32_t n, int dir) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        if (dir == 0) tail[i] = bweight[i]; else bweight[i] = tail[i];
    }
}
static int exchange_training_statistics(ppg_integrator *h) {
    if (!h->multi()) return PPG_OK;
    float *tail = h->dTrain.p + 4 * (size_t) h->hTotalBuild;
    pack_tail_kernel<<<h->numSMs, 256, 0, h->stream>>>(tail, h->dBweight.p, h->hNodes, 0); h->launches++;
    int rc = allreduce_sum(h, h->dTrain.p, 4 * (size_t) h->hTotalBuild + (size_t) h->hNodes); if (rc) return rc;
    pack_tail_kernel<<<h->numSMs, 256, 0, h->stream>>>(tail, h->dBweight.p, h->hNodes, 1); h->launches++;
    return PPG_OK;
}
// a host scalar made identical on all ranks (rank 0's value wins): time-based decisions must not diverge
static int sync_scalar(ppg_integrator *h, float *v) {
    if (!h->multi()) return PPG_OK;
    float *slot = h->dTrain.p + h->dTrain.n - 16;
    const float mine = h->rank == 0 ? *v : 0.f;
    CK(cudaMemcpyAsync(slot, &mine, 4, cudaMemcpyHostToDevice, h->stream));
    int rc = allreduce_sum(h, slot, 1); if (rc) return rc;
    CK(cudaMemcpyAsync(v, slot, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PPG_OK;
}

// buildSDTree, GP:1115-1189
static int build_sd_tree(ppg_integrator *h, ppg_iteration_stats &st) {
    int rc = exchange_training_statistics(h);
    if (rc) return rc;
    MaintParams M = maint(h);
    h->tic(PPG_K_BUILD); dtree_build_kernel<<<h->numSMs * 4, 128, 0, h->stream>>>(M, h->dBuildBase.p); h->toc(); h->launches++;
    CK(cudaGetLastError());
    // "Distribution statistics" (GP:1121-1186): reduced on the device, 64 bytes come back
    CK(cudaMemsetAsync(h->dTreeStats.p, 0, sizeof(TreeStats), h->stream));
    tree_stats_kernel<<<1, 1024, 0, h->stream>>>(M, h->dTreeStats.p); h->launches++;
    // the statistics are only reported: they go to pinned memory and are folded into ppg_stats after the render's last synchronize
    const int slot = std::min(h->iter, PPG_MAX_ITERATIONS - 1);
    CK(cudaMemcpyAsync(h->hTreeStats + slot, h->dTreeStats.p, sizeof(TreeStats), cudaMemcpyDeviceToHost, h->stream));
    h->treeStatsPending[slot] = true;
    st.s_tree_nodes = h->hNodes;
    h->isBuilt = true;
    return PPG_OK;
}
static void finish_tree_stats(ppg_integrator *h) {      // after a stream synchronize
    for (int i = 0; i < PPG_MAX_ITERATIONS; ++i) {
        if (!h->treeStatsPending[i]) continue;
        h->treeStatsPending[i] = false;
        const TreeStats &ts = h->hTreeStats[i]; ppg_iteration_stats &st = h->stats.iterations[i];
        const int nPoints = (int) ts.leaves, nPointsNodes = (int) ts.leavesWithNodes;
        float avgDepth = (float) ts.depthSum, avgR = (float) ts.meanSum, avgN = (float) ts.nodesSum, avgW = (float) ts.weightSum;
        if (nPoints > 0) { avgDepth /= nPoints; avgR /= nPoints; if (nPointsNodes > 0) avgN /= nPointsNodes; avgW /= nPoints; }
        st.depth_min = nPoints ? ts.depthMin : std::numeric_limits<int>::max(); st.depth_max = ts.depthMax; st.depth_avg = avgDepth;
        st.mean_radiance_min = nPoints ? ts.meanMin : std::numeric_limits<float>::max(); st.mean_radiance_avg = avgR; st.mean_radiance_max = ts.meanMax;
        st.nodes_min = nPointsNodes ? ts.nodesMin : std::numeric_limits<size_t>::max(); st.nodes_max = ts.nodesMax; st.nodes_avg = avgN;
        st.weight_min = nPoints ? ts.weightMin : std::numeric_limits<float>::max(); st.weight_avg = avgW; st.weight_max = ts.weightMax;
        st.s_tree_leaves = ts.leaves;
    }
}

// ------------------------------------------------------------------ wavefront buffers
static int ensure_wavefront(ppg_integrator *h) {
    const size_t perPass = (size_t) h->maxLocalPixels * h->prm.spp_per_pass;       // the largest share of any rank: every rank splits an iteration into the same batches
    h->maxBounces = h->prm.max_depth > 0 ? h->prm.max_depth : 64;
    h->nSlabs = std::max(1, h->maxBounces - 1);
    const bool nee = h->useNee();
    const bool full = nee || h->prm.spatial_filter != PPG_SFILTER_NEAREST || h->prm.bsdf_sampling_fraction_loss != PPG_LOSS_NONE;
    h->recordMode = full ? 2 : 1;
    const int stateVecs = nee ? 7 : 5, slabSets = nee ? 2 : 1;
    const size_t perPath = 2 * 16 * (size_t) stateVecs + 16 + (size_t) h->nSlabs * (full ? 96 : 48) * slabSets;
    size_t cap = (size_t) 1 << 23;
    if (const char *e = getenv("PPG_PATH_CAPACITY")) cap = std::max<size_t>(strtoull(e, nullptr, 10), 1024);
    size_t budget = (size_t) 24 << 30;
    if (const char *e = getenv("PPG_WAVEFRONT_BYTES")) budget = strtoull(e, nullptr, 10);
    cap = std::min(cap, budget / perPath);
    cap = std::max(cap, perPass);                          // one pass must fit
    cap = (cap / std::max<size_t>(perPass, 1)) * std::max<size_t>(perPass, 1);   // whole passes only
    cap = std::max(cap, perPass);
    if (cap >= (1ull << 30)) return fail(PPG_ERR_INVALID_ARGUMENT, "pass too large for 30-bit path ids");
    if (cap != h->pathCapacity || stateVecs != h->stateVecs || slabSets != h->slabSets) {
        h->dStateA.release(); h->dStateB.release(); h->dSlabs.release(); h->dLiFinal.release();
        CK(h->dStateA.alloc(stateVecs * cap)); CK(h->dStateB.alloc(stateVecs * cap)); CK(h->dLiFinal.alloc(cap));
        CK(h->dSlabs.alloc((size_t) h->nSlabs * (full ? 6 : 3) * cap * slabSets));
        h->pathCapacity = cap; h->stateVecs = stateVecs; h->slabSets = slabSets;
    }
    CK(h->dLive.alloc(h->maxBounces + 2)); CK(h->dWork.alloc(h->maxBounces + 2)); CK(h->dCounters.alloc(8));
    if (h->prm.bsdf_sampling_fraction_loss != PPG_LOSS_NONE) {
        // sampling-fraction records: one per (recorded vertex, leaf) pair.  Sized once for the largest wavefront with 16 records per path (mean path
        // lengths of the bundled scenes: 4 - 9 vertices; the spatial box filter touches ~2 leaves per vertex); a record beyond it is dropped and
        // counted in ppg_stats.dropped_records.  Allocating per batch (cudaMalloc / cudaFree are synchronous) cost 11 ms per sub-batch.
        const size_t want = cap * 16 * (h->prm.spatial_filter == PPG_SFILTER_BOX ? 2 : 1);
        if (want > h->adamCap) {
            h->dAdamRecA.release(); h->dAdamRecB.release(); h->dAdamSortA.release(); h->dAdamSortB.release();
            CK(h->dAdamRecA.alloc(want)); CK(h->dAdamRecB.alloc(want)); CK(h->dAdamSortA.alloc(want)); CK(h->dAdamSortB.alloc(want));
            h->adamCap = want;
        }
    }
    // persistent grids: resident blocks per SM from the occupancy calculator
    int occ = 0;
    if (h->sceneSmemBytes) occ = h->fullFeature ? ppg_bounce_occupancy_11(h->sceneSmemBytes) : ppg_bounce_occupancy_10(h->sceneSmemBytes);
    else occ = h->fullFeature ? ppg_bounce_occupancy_01(0) : ppg_bounce_occupancy_00(0);
    CK(cudaGetLastError());
    // one block per resident slot; warps claim their work dynamically (bounce_kernel)
    h->gridBounce = h->numSMs * std::max(occ, 1) * std::max(env_int("PPG_GRID_MULT", 1), 1);
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, commit_kernel<1>, PPG_BLOCK, 0));
    h->gridCommit = h->numSMs * std::max(occ, 1);
    // Scenes walked through the BVH find their hits in a separate pass of persistent warps (ppg_trace.cu) whenever the wavefront is large enough
    // to pay for the second launch per depth; tiny learning sub-batches keep the fused kernel.  PPG_TRACE_MIN_PATHS=0 turns the pass off.
    h->gridTrace = 0;
    h->traceMinPaths = (uint32_t) std::max(env_int("PPG_TRACE_MIN_PATHS", 32768), 0);
    if (!h->sceneSmemBytes && h->sceneView.nGroups == 0u && h->sceneView.nTris != 0u && h->traceMinPaths != 0u) {
        CK(h->dHits.alloc(h->pathCapacity)); CK(h->dTraceWork.alloc(h->maxBounces + 2));
        h->binMaterials = h->fullFeature && env_int("PPG_BIN_MATERIALS", 1) != 0;       // one kind of BSDF only: nothing to sort
        if (h->binMaterials) { CK(h->dOrder.alloc((size_t) PPG_BINS * h->pathCapacity)); CK(h->dBinCount.alloc((size_t) PPG_BINS * (h->maxBounces + 2))); }
        h->gridTrace = h->numSMs * std::max(ppg_trace_occupancy(), 1);
        CK(cudaGetLastError());
    }
    return PPG_OK;
}

static PathState path_state(float4 *base, size_t cap, bool nee) {
    PathState s; s.s0 = base; s.s1 = base + cap; s.s2 = base + 2 * cap; s.s3 = base + 3 * cap; s.s4 = base + 4 * cap;
    s.s5 = nee ? base + 5 * cap : nullptr; s.s6 = nee ? base + 6 * cap : nullptr; return s;
}
static VertexSlab slab_at(ppg_integrator *h, int k, int set = 0) {
    const size_t cap = h->pathCapacity; const int per = h->recordMode == 2 ? 6 : 3;
    float4 *b = h->dSlabs.p + (size_t) set * h->nSlabs * per * cap;
    VertexSlab s;
    // field-major layout: field f of slab k at ((f * nSlabs) + k) * cap, so that slab k+1 of a field is +cap (commit's slabStride)
    s.v0 = b + ((size_t) 0 * h->nSlabs + k) * cap; s.v1 = b + ((size_t) 1 * h->nSlabs + k) * cap; s.v2 = b + ((size_t) 2 * h->nSlabs + k) * cap;
    if (per == 6) { s.v3 = b + ((size_t) 3 * h->nSlabs + k) * cap; s.v4 = b + ((size_t) 4 * h->nSlabs + k) * cap; s.v5 = b + ((size_t) 5 * h->nSlabs + k) * cap; }
    else { s.v3 = s.v4 = s.v5 = nullptr; }
    return s;
}

static void launch_bounce(ppg_integrator *h, const RenderParams &P, bool first, int record, int grid, bool nee) {
    // scene staged in shared memory or read from HBM; lean instantiations for diffuse-only triangle scenes
    const BounceLaunch L{h->stream, grid, record, nee ? 1 : 0, first ? 1 : 0};
    if (P.sceneSmemBytes) { if (h->fullFeature) ppg_launch_bounce_11(P, L); else ppg_launch_bounce_10(P, L); }
    else { if (h->fullFeature) ppg_launch_bounce_01(P, L); else ppg_launch_bounce_00(P, L); }
    h->launches++;
}

// one batch of `nPasses` passes as a single wavefront, over `pixelCount` of this rank's pixels taken from `pixelMap` (a range of the block-ordered
// map or of its scattered permutation).  A rank without pixels in the batch still takes part in the collective of the Adam replay.
static int render_batch(ppg_integrator *h, int nPasses, const uint32_t *pixelMap, uint32_t pixelCount) {
    const uint32_t nPaths = (uint32_t) ((size_t) nPasses * pixelCount * h->prm.spp_per_pass);
    const int record = h->isFinalIter ? 0 : h->recordMode;
    const bool nee = h->useNee();                      // the NEE kernels also carry the MIS state when doNee is off (kickstart after 128 spp)
    const int lossMode = (record && h->isBuilt) ? h->prm.bsdf_sampling_fraction_loss : PPG_LOSS_NONE;       // GP:2152
    const bool useAdam = lossMode != PPG_LOSS_NONE;
    const bool neeSlabs = nee && h->doNee && h->prm.nee != PPG_NEE_ALWAYS;
    if (useAdam) CK(cudaMemsetAsync(h->dScalars.p + 3, 0, 4, h->stream));      // record cursor (buffers: ensure_wavefront)
    if (nPaths) {
        CK(cudaMemsetAsync(h->dLive.p, 0, 4 * (size_t) (h->maxBounces + 2), h->stream));
        CK(cudaMemsetAsync(h->dWork.p, 0, 4 * (size_t) (h->maxBounces + 2), h->stream));
        CK(cudaMemcpyAsync(h->dLive.p, &nPaths, 4, cudaMemcpyHostToDevice, h->stream));
        RenderParams P;
        P.scene = h->sceneView; P.cam = h->cam; P.tree = tree_view(h);
        P.liFinal = h->dLiFinal.p; P.pixelMap = pixelMap; P.counters = h->dCounters.p;
        P.nPaths = nPaths; P.nLocalPixels = pixelCount; P.spp = (uint32_t) h->prm.spp_per_pass;
        P.passBase = (uint64_t) h->passesRendered; P.seed = h->prm.seed;
        P.maxDepth = h->prm.max_depth; P.rrDepth = h->prm.rr_depth; P.strictNormals = h->prm.strict_normals; P.hideEmitters = h->prm.hide_emitters;
        P.isBuilt = h->isBuilt ? 1 : 0; P.lossMode = h->prm.bsdf_sampling_fraction_loss; P.fixedFraction = h->prm.bsdf_sampling_fraction;
        P.sceneSmemBytes = h->sceneSmemBytes;
        P.neeMode = h->prm.nee; P.doNee = (nee && h->doNee) ? 1 : 0; P.training = record != 0 ? 1 : 0;
        PathState A = path_state(h->dStateA.p, h->pathCapacity, nee), B = path_state(h->dStateB.p, h->pathCapacity, nee);
        const int bb = h->sceneSmemBytes ? PPG_BOUNCE_BLOCK : PPG_BOUNCE_BLOCK_HBM;
        const int grid = std::min<int>(h->gridBounce, (int) ((nPaths + bb - 1) / bb));
        const bool useTrace = h->gridTrace > 0 && nPaths >= h->traceMinPaths;
        P.hits = useTrace ? h->dHits.p : nullptr; P.traceWork = nullptr;
        const bool bins = useTrace && h->binMaterials;
        P.order = bins ? h->dOrder.p : nullptr; P.binCount = nullptr; P.binStride = (uint32_t) h->pathCapacity;
        if (useTrace) CK(cudaMemsetAsync(h->dTraceWork.p, 0, 4 * (size_t) (h->maxBounces + 2), h->stream));
        if (bins) CK(cudaMemsetAsync(h->dBinCount.p, 0, 4 * (size_t) PPG_BINS * (h->maxBounces + 2), h->stream));
        int lastDepth = 0, pendingDepth = 0; uint32_t bracket = 0;
        for (int depth = 1; depth <= h->maxBounces; ++depth) {
            P.depth = depth; P.in = (depth & 1) ? B : A; P.out = (depth & 1) ? A : B;
            P.liveIn = h->dLive.p + (depth - 1); P.liveOut = h->dLive.p + depth; P.work = h->dWork.p + depth;
            const int k = std::min(depth - 1, h->nSlabs - 1);
            P.slab = slab_at(h, k);
            if (nee) { P.neeSlab = slab_at(h, k, 1); P.prevSlab = slab_at(h, std::max(k - 1, 0)); if (depth - 1 >= h->nSlabs) P.prevSlab = slab_at(h, h->nSlabs - 1); }
            const int rec = (depth - 1 < h->nSlabs) ? record : 0;
            if (h->cancelled.load()) { if (bracket) h->toc(bracket); return PPG_ERR_CANCELLED; }   // Integrator::cancel() (GP:1643-1648): the batch in flight is dropped
            if (!bracket) h->tic(PPG_K_BOUNCE);                                // one event pair around the consecutive bounce launches (2 records per launch were
            if (useTrace) {                                                    // nearest hits of this depth's rays, then the bounce kernel shades them
                P.traceWork = h->dTraceWork.p + depth;
                if (bins) P.binCount = h->dBinCount.p + (size_t) PPG_BINS * depth;
                ppg_launch_trace(P, h->stream, std::min<int>(h->gridTrace, (int) ((nPaths + 255) / 256)), depth == 1, h->sceneView.nSpheres != 0u); h->launches++;
            }
            launch_bounce(h, P, depth == 1, rec, grid, nee);                   // ~1.5 ms of host time per CBOX step: visible at 8 GPUs, where a step takes 38 ms)
            ++bracket;
            lastDepth = depth;
            // unbounded path length (maxDepth == -1 runs up to the 64-bounce cap): stop launching once the wavefront is empty.  The live count is
            // copied to pinned memory at every check point and LOOKED AT one check point later, after the next launches are queued: the host
            // never drains the stream (a blocking read-back cost ~25 us of idle GPU per check: 3-5 ms per CBOX step), and a dead wavefront costs
            // at most two check intervals of empty launches (~2 us each).
            const bool small = nPaths <= 65536u;          // small wavefronts are launch bound: look every 4 bounces from the start
            if ((h->prm.max_depth <= 0 || small) && depth < h->maxBounces && depth % 4 == 0 && (small || depth >= 8)) {
                CK(cudaMemcpyAsync(h->liveHost + depth, h->dLive.p + depth, 4, cudaMemcpyDeviceToHost, h->stream));
                CK(cudaEventRecord(h->evLive[(depth >> 2) & 1], h->stream));
                if (pendingDepth) {
                    CK(cudaEventSynchronize(h->evLive[(pendingDepth >> 2) & 1]));
                    if (h->liveHost[pendingDepth] == 0) break;
                }
                pendingDepth = depth;
            }
        }
        if (bracket) h->toc(bracket);
        {   // survivors of the bounce cap (maxDepth == -1 only) keep the radiance they have; they are counted (ppg_stats.truncated_paths)
            const PathState last = (lastDepth & 1) ? A : B;
            flush_kernel<<<std::max(grid / 4, 1), PPG_BLOCK, 0, h->stream>>>(last, h->dLive.p + lastDepth, h->dLiFinal.p, h->dCounters.p + 3); h->launches++;
        }
        if (record) {
            CommitParams C;
            C.tree = tree_view(h); C.slab0 = slab_at(h, 0); C.slabStride = h->pathCapacity; C.liveCounts = h->dLive.p; C.liFinal = h->dLiFinal.p;
            C.spatialFilter = h->prm.spatial_filter; C.directionalFilter = h->prm.directional_filter;
            C.lossMode = lossMode;
            C.statisticalWeight = (h->prm.nee == PPG_NEE_KICKSTART && h->doNee && nee) ? 0.5f : 1.0f;   // GP:2152
            C.seed = h->prm.seed; C.snodes = h->dSnodes.p; C.nSlabs = (uint32_t) std::min(h->nSlabs, lastDepth);
            C.nee0 = neeSlabs ? slab_at(h, 0, 1) : C.slab0;
            C.adamRecA = h->dAdamRecA.p; C.adamRecB = h->dAdamRecB.p; C.adamTotal = h->dScalars.p + 3; C.adamCap = (uint32_t) std::min<size_t>(h->adamCap, 0xFFFFFFFFu);
            C.dropped = h->dCounters.p + 4;
            dim3 g(std::min<int>(h->gridCommit, (int) ((nPaths + PPG_BLOCK - 1) / PPG_BLOCK)), C.nSlabs * (neeSlabs ? 2 : 1));
            h->tic(PPG_K_COMMIT);
            if (record == 1) commit_kernel<1><<<g, PPG_BLOCK, 0, h->stream>>>(C); else commit_kernel<2><<<g, PPG_BLOCK, 0, h->stream>>>(C);
            h->toc(); h->launches++;
        }
        h->tic(PPG_K_FILM);
        film_kernel<<<std::min<int>(h->numSMs * 8, (int) ((pixelCount + PPG_BLOCK - 1) / PPG_BLOCK)), PPG_BLOCK, 0, h->stream>>>(
            h->dLiFinal.p, pixelMap, pixelCount, (uint32_t) h->prm.spp_per_pass, (uint32_t) nPasses, h->W, h->dImage.p, h->dSqImage.p);
        h->toc(); h->launches++;
    }
    if (useAdam) {
        // replay the sampling-fraction records leaf by leaf (see adam_seq_kernel)
        MaintParams M = maint(h);
        const bool multi = h->multi();
        float *tail = h->dTrain.p + 4 * (size_t) h->hTotalBuild;       // [6 x nNodes] exchange area (the building weights are packed there only at iteration end)
        adam_pack_kernel<<<h->numSMs, 256, 0, h->stream>>>(M, tail, h->dAdamBefore.p, nullptr, 0); h->launches++;
        h->tic(PPG_K_OTHER);      // bucket the records by leaf (histogram, scan, scatter): "other"; the sequential replay itself: "adam"
        adam_hist_kernel<<<h->numSMs * 4, 256, 0, h->stream>>>(h->dAdamRecA.p, h->dScalars.p + 3, (uint32_t) h->adamCap, h->dAdamCount.p); h->launches++;
        exclusive_scan_kernel<<<1, 1024, 0, h->stream>>>(h->dAdamCount.p, h->dAdamOffset.p, h->dScalars.p, h->dScalars.p + 4); h->launches++;
        adam_scatter_kernel<<<h->numSMs * 4, 256, 0, h->stream>>>(h->dAdamRecA.p, h->dAdamRecB.p, h->dScalars.p + 3, (uint32_t) h->adamCap, h->dAdamOffset.p,
                                                                  h->dAdamCursor.p, h->dAdamSortA.p, h->dAdamSortB.p); h->launches++;
        h->toc();
        h->tic(PPG_K_ADAM);
        adam_seq_kernel<<<h->numSMs * 16, 128, 0, h->stream>>>(M, h->dAdamSortA.p, h->dAdamSortB.p, h->dAdamOffset.p, h->dAdamCount.p, h->dAdamCursor.p,
                                                              lossMode == PPG_LOSS_KL ? 1.0f : 2.0f); h->launches++;
        h->toc();
        if (multi) {
            // replicas replayed their own records from the common state: merge them (step counts and batch accumulators add up relative to
            // the common start, moments and the variable are averaged) so that all ranks continue identically
            adam_pack_kernel<<<h->numSMs, 256, 0, h->stream>>>(M, tail, h->dAdamBefore.p, nullptr, 1); h->launches++;
            int rc = allreduce_sum(h, tail, 6 * (size_t) h->hNodes); if (rc) return rc;
            adam_merge_kernel<<<h->numSMs, 256, 0, h->stream>>>(M, tail, h->dAdamBefore.p, 1.0f / (float) h->world, (float) (h->world - 1)); h->launches++;
        }
        // movement of the fractions in this replay (identical on all ranks after the merge): steers the size of the next sub-batch
        CK(cudaMemsetAsync(h->dCounters.p + 6, 0, 16, h->stream));
        adam_progress_kernel<<<h->numSMs, 256, 0, h->stream>>>(M, h->dAdamBefore.p, h->dCounters.p + 6); h->launches++;
        CK(cudaMemcpyAsync(h->adamProgress, h->dCounters.p + 6, 16, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaGetLastError());
    return PPG_OK;
}

// performRenderPasses, GP:1210-1329
static int perform_render_passes(ppg_integrator *h, float &variance, int numPasses, ppg_iteration_stats &st) {
    const size_t npx = (size_t) h->W * h->H;
    CK(cudaMemsetAsync(h->dImage.p, 0, sizeof(float4) * npx, h->stream));
    CK(cudaMemsetAsync(h->dSqImage.p, 0, sizeof(float4) * npx, h->stream));
    CK(cudaMemsetAsync(h->dCounters.p, 0, 64, h->stream));
    const auto t0 = std::chrono::steady_clock::now();
    CK(cudaEventRecord(h->evA, h->stream));
    const size_t perPass = (size_t) h->nLocalPixels * h->prm.spp_per_pass;
    const size_t perPassMax = (size_t) h->maxLocalPixels * h->prm.spp_per_pass;                 // rank independent
    const int maxBatch = (int) std::max<size_t>(1, perPassMax ? h->pathCapacity / perPassMax : 1);
    // Sampling-fraction learning (GP:672-697).  The reference takes an optimiser step after every ~2 records WHILE the passes run, so the
    // fractions that guide the paths follow the optimiser with a lag of a few paths.  A wavefront samples all its paths with the fractions
    // it starts with; the Adam replay after it (adam_seq_kernel) then takes every step the reference would.  To bound that staleness a
    // learning iteration is rendered as a sequence of sub-batches (first fractions of a pass in the scattered pixel order, later whole passes)
    // whose size follows a step-size control: see `target` below.  All quantities that shape the sequence are identical on every rank.
    const bool learning = h->isBuilt && !h->isFinalIter && h->prm.bsdf_sampling_fraction_loss != PPG_LOSS_NONE;
    // Step-size control: after every replay the device reports how far the fractions moved (steps-weighted mean |df|).  The next sub-batch is sized
    // so that the fractions move by about `target` during it: that movement IS the staleness of the fractions a wavefront samples with.
    // Measured on SPACESHIP 640x360 (recorded vertices of iterations 1-4 against the CPU restatement of the reference, which learns online like it; its
    // own run-to-run spread is ~0.5 %): target 0.005 -> +0.2 % (2200 sub-batches), 0.01 -> +0.4 % (1130), 0.02 -> +1.2 % (223), 0.04 -> +4 % (58).
    static const double target = std::max(env_int("PPG_LOSS_TARGET_X1000", 20), 1) * 1e-3;
    static const double growthMax = std::max(env_int("PPG_LOSS_GROWTH_MAX_PCT", 100), 1) * 0.01;
    static const double leafPaths = std::max(env_int("PPG_LOSS_LEAF_PATHS_X10", 40), 1) * 0.1;   // paths per S-tree leaf in the first sub-batch
    const double pathsPerPass = (double) npx * h->prm.spp_per_pass;                                  // whole image
    const double minFrac = std::min(1.0, std::max(256.0, leafPaths * 0.5 * (h->hNodes + 1)) / std::max(pathsPerPass, 1.0));
    double done = 0.0, frac = 0.0;          // passes rendered in this call (real number), fraction of the pass in progress
    double want = learning ? minFrac : (double) maxBatch, lastSize = 0.0;
    int local = 0; int rcode = PPG_OK;
    while (local < numPasses) {
        int rc = PPG_OK; int nb = 0;
        if (learning && lastSize > 0.0) {
            CK(cudaStreamSynchronize(h->stream));                       // the progress read-back of the batch just issued
            const double moved = h->adamProgress[1] ? (double) h->adamProgress[0] / 1048576.0 / (double) h->adamProgress[1] : 0.0;
            const double ratio = moved > 0.0 ? target / moved : 2.0;
            want = lastSize * std::min(2.0, std::max(0.5, ratio));
            want = std::max(minFrac, std::min(want, std::max(minFrac, growthMax * done)));
            ++h->stats.sub_batches;
            static const int trace2 = env_int("PPG_TRACE", 0);
            if (trace2 > 1) fprintf(stderr, "[ppg trace]   sub-batch %.5f passes moved %.4f next %.5f at %.2f ms\n", lastSize, moved, want, elapsed_ms(t0));
        }
        if (frac > 0.0 || want < 1.0) {
            // a slice [frac, f1) of one pass, in the scattered pixel order
            double f1 = std::min(1.0, frac + want);
            if (1.0 - f1 < 0.5 * want) f1 = 1.0;                       // no tiny remainder
            const uint32_t p0 = (uint32_t) std::llround(frac * h->nLocalPixels), p1 = f1 >= 1.0 ? h->nLocalPixels : (uint32_t) std::llround(f1 * h->nLocalPixels);
            rc = render_batch(h, 1, h->dPixelMapPerm.p + p0, p1 - p0);
            lastSize = f1 - frac; done += f1 - frac; frac = f1;
            if (frac >= 1.0) { frac = 0.0; nb = 1; }
        } else {
            nb = std::min(std::min(maxBatch, numPasses - local), std::max(1, (int) want));
            rc = render_batch(h, nb, h->dPixelMap.p, h->nLocalPixels);
            lastSize = nb; done += nb;
        }
        if (rc == PPG_ERR_CANCELLED) { rcode = rc; break; }
        if (rc) return rc;
        h->passesRendered += nb; local += nb;
        if (h->cancelled.load()) { rcode = PPG_ERR_CANCELLED; break; }
        if (nb == 0) continue;
        bool shouldAbort = false;
        if (h->prm.budget_type == PPG_BUDGET_SECONDS) {              // GP:1259-1262, checked per batch
            CK(cudaStreamSynchronize(h->stream));
            float el = h->clock_s();
            rc = sync_scalar(h, &el); if (rc) return rc;
            shouldAbort = (int) el > h->prm.budget;
        }
        if (shouldAbort) break;
    }
    add_image_kernel<<<h->numSMs * 4, 256, 0, h->stream>>>(h->dFilm.p, h->dImage.p, npx); h->launches++;   // film->put(block), renderproc.cpp:143-151
    if (h->prm.sample_combination == PPG_COMB_INVERSEVAR) {            // GP:1292-1296: keep the iteration's image (ring of the last four)
        if (h->images.size() < 4) { DevBuf<float4> *img = new DevBuf<float4>(); CK(img->alloc(npx)); h->images.push_back(img); }
        else std::rotate(h->images.begin(), h->images.begin() + 1, h->images.end());
        CK(cudaMemcpyAsync(h->images.back()->p, h->dImage.p, sizeof(float4) * npx, cudaMemcpyDeviceToDevice, h->stream));
    }
    // variance, GP:1298-1319: the numerator is reduced on the device (double), summed over ranks as a float, and read back together with the counters
    const int N = local * h->prm.spp_per_pass;
    CK(cudaMemsetAsync(h->dVar.p, 0, 8, h->stream));
    if (h->nLocalPixels)
        variance_kernel<<<std::min<int>(h->numSMs * 4, (int) ((h->nLocalPixels + PPG_BLOCK - 1) / PPG_BLOCK)), PPG_BLOCK, 0, h->stream>>>(
            h->dImage.p, h->dSqImage.p, h->dPixelMap.p, h->nLocalPixels, h->W, (float) N, h->dVar.p);
    h->launches++;
    float *slot = h->dTrain.p + h->dTrain.n - 16;
    double_to_float_kernel<<<1, 1, 0, h->stream>>>(h->dVar.p, slot); h->launches++;
    if (h->multi()) { int rc = allreduce_sum(h, slot, 1); if (rc) return rc; }
    float numF = 0; unsigned long long cnt[8];
    CK(cudaMemcpyAsync(&numF, slot, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(cnt, h->dCounters.p, 64, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(h->evB, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    float ms = 0; cudaEventElapsedTime(&ms, h->evA, h->evB); h->deviceMs += ms;
    h->resolve_timers();
    variance = (float) ((double) numF / ((double) h->W * h->H * (N - 1)));
    if (h->prm.sample_combination == PPG_COMB_INVERSEVAR) { h->variances.push_back(variance); if (h->variances.size() > 4) h->variances.erase(h->variances.begin()); }
    st.seconds += elapsed_s(t0); st.passes += local; st.variance = variance; st.total_passes = h->passesRendered;
    st.vertices += cnt[0]; st.paths += (uint64_t) local * perPass; st.recorded_vertices += cnt[1];
    if (cnt[1]) st.s_tree_depth_avg = (double) cnt[2] / (double) cnt[1];
    h->stats.total_vertices += cnt[0]; h->stats.total_paths += (uint64_t) local * perPass;
    h->stats.truncated_paths += cnt[3]; h->stats.dropped_records += cnt[4]; h->stats.invalid_rays += cnt[5];
    h->lastRecorded = cnt[1];
    static const int trace = env_int("PPG_TRACE", 0);
    if (trace)    // cumulative kernel times after every iteration's passes (stderr): where a render's time goes, iteration by iteration
        fprintf(stderr, "[ppg trace] iter %d final %d passes %d sub_batches %llu vertices %llu entered at %.1f ms wall %.1f ms | cumulative ms: bounce %.1f commit %.1f adam %.1f other %.1f film %.1f launches %llu\n",
                h->iter, (int) h->isFinalIter, local, (unsigned long long) h->stats.sub_batches, (unsigned long long) cnt[0], elapsed_ms(h->startTime) - elapsed_ms(t0), elapsed_ms(t0),
                h->stats.kernel_ms[PPG_K_BOUNCE], h->stats.kernel_ms[PPG_K_COMMIT], h->stats.kernel_ms[PPG_K_ADAM], h->stats.kernel_ms[PPG_K_OTHER], h->stats.kernel_ms[PPG_K_FILM],
                (unsigned long long) h->launches);
    return rcode;
}

static ppg_iteration_stats &iter_stats(ppg_integrator *h) {
    ppg_iteration_stats &st = h->stats.iterations[std::min(h->iter, PPG_MAX_ITERATIONS - 1)];
    memset(&st, 0, sizeof(st)); st.iteration = h->iter;
    return st;
}
// progressive film (renderproc.cpp:143-151 puts finished blocks into the film while rendering): hand the current film to the host's callback
static int flush_film(ppg_integrator *h) {
    if (!h->filmFn) return PPG_OK;
    const size_t npx = (size_t) h->W * h->H;
    develop_kernel<<<h->numSMs * 4, 256, 0, h->stream>>>(h->dFilm.p, h->dRgb.p, npx, 1.0f, 0); h->launches++;
    CK(cudaStreamSynchronize(h->stream));
    h->filmFn(h->filmUser, h->dRgb.p, h->W, h->H, h->passesRendered);
    return PPG_OK;
}
static int clear_film(ppg_integrator *h) { CK(cudaMemsetAsync(h->dFilm.p, 0, sizeof(float4) * (size_t) h->W * h->H, h->stream)); return PPG_OK; }

static int dump_iteration(ppg_integrator *h) {      // dumpSDTree: "<dest>-NN.sdt", GP:1191-1195
    if (h->destination.empty() || h->rank != 0) return PPG_OK;
    char ext[32]; snprintf(ext, sizeof(ext), "-%02d.sdt", h->iter);
    return ppg_dump_sdtree(h, (h->destination + ext).c_str());
}

// renderSPP, GP:1342-1426
static int render_spp(ppg_integrator *h) {
    const int nPasses = (int) std::ceil((size_t) h->prm.budget / (float) h->prm.spp_per_pass);
    float currentVarAtEnd = std::numeric_limits<float>::infinity();
    while (h->passesRendered < nPasses) {
        const int sppRendered = h->passesRendered * h->prm.spp_per_pass;
        h->doNee = h->prm.nee == PPG_NEE_NEVER ? false : (h->prm.nee == PPG_NEE_KICKSTART ? sppRendered < 128 : true);   // doNeeWithSpp, GP:1331-1340, 1362
        int remainingPasses = nPasses - h->passesRendered;
        int passesThisIteration = std::min(remainingPasses, 1 << std::min(h->iter, 30));
        if (remainingPasses - passesThisIteration < 2 * passesThisIteration) passesThisIteration = remainingPasses;
        h->isFinalIter = passesThisIteration >= remainingPasses;
        ppg_iteration_stats &st = iter_stats(h);
        int rc = clear_film(h); if (rc) return rc;
        auto t0 = std::chrono::steady_clock::now();
        rc = reset_sd_tree(h); if (rc) return rc;
        st.reset_seconds = elapsed_s(t0);                               // host time up to the node-count read-back inside the reset
        float variance = 0;
        rc = perform_render_passes(h, variance, passesThisIteration, st); if (rc) return rc;
        rc = flush_film(h); if (rc) return rc;
        const float lastVarAtEnd = currentVarAtEnd;
        currentVarAtEnd = passesThisIteration * variance / remainingPasses;
        remainingPasses -= passesThisIteration;
        if (h->prm.sample_combination == PPG_COMB_AUTOMATIC && remainingPasses > 0 &&
            (remainingPasses < passesThisIteration || (sppRendered > 256 && currentVarAtEnd > lastVarAtEnd))) {
            h->isFinalIter = true;
            rc = perform_render_passes(h, variance, remainingPasses, st); if (rc) return rc;
            rc = flush_film(h); if (rc) return rc;
        }
        st.is_final = h->isFinalIter;
        t0 = std::chrono::steady_clock::now();
        rc = build_sd_tree(h, st); if (rc) return rc;
        st.build_seconds = elapsed_s(t0);
        if (h->prm.dump_sd_tree && !h->isFinalIter) { rc = dump_iteration(h); if (rc) return rc; }     // GP:1417-1419
        ++h->iter; h->stats.n_iterations = std::min(h->iter, PPG_MAX_ITERATIONS);
    }
    return PPG_OK;
}

// renderTime, GP:1434-1514
static int render_time(ppg_integrator *h) {
    const float nSeconds = h->prm.budget;
    float currentVarAtEnd = std::numeric_limits<float>::infinity(), elapsedSeconds = 0;
    while (elapsedSeconds < nSeconds) {
        const int sppRendered = h->passesRendered * h->prm.spp_per_pass;
        h->doNee = h->prm.nee == PPG_NEE_NEVER ? false : (h->prm.nee == PPG_NEE_KICKSTART ? sppRendered < 128 : true);   // GP:1452
        float remainingTime = nSeconds - elapsedSeconds;
        const int passesThisIteration = 1 << std::min(h->iter, 30);
        ppg_iteration_stats &st = iter_stats(h);
        const auto startIter = std::chrono::steady_clock::now(); const float startIterClock = h->clock_s();
        int rc = clear_film(h); if (rc) return rc;
        rc = reset_sd_tree(h); if (rc) return rc;
        st.reset_seconds = elapsed_s(startIter);
        float variance = 0;
        rc = perform_render_passes(h, variance, passesThisIteration, st); if (rc) return rc;
        rc = flush_film(h); if (rc) return rc;
        float secondsIter = h->clock_s() - startIterClock;
        rc = sync_scalar(h, &secondsIter); if (rc) return rc;
        const float lastVarAtEnd = currentVarAtEnd;
        currentVarAtEnd = secondsIter * variance / remainingTime;
        remainingTime -= secondsIter;
        if (h->prm.sample_combination == PPG_COMB_AUTOMATIC && remainingTime > 0 &&
            (remainingTime < secondsIter || (sppRendered > 256 && currentVarAtEnd > lastVarAtEnd))) {
            h->isFinalIter = true;
            do {
                rc = perform_render_passes(h, variance, passesThisIteration, st); if (rc) return rc;
                rc = flush_film(h); if (rc) return rc;
                elapsedSeconds = h->clock_s();
                rc = sync_scalar(h, &elapsedSeconds); if (rc) return rc;
            } while (elapsedSeconds < nSeconds);
        }
        st.is_final = h->isFinalIter;
        const auto t0 = std::chrono::steady_clock::now();
        rc = build_sd_tree(h, st); if (rc) return rc;
        st.build_seconds = elapsed_s(t0);
        if (h->prm.dump_sd_tree && !h->isFinalIter) { rc = dump_iteration(h); if (rc) return rc; }     // GP:1504-1506
        ++h->iter; h->stats.n_iterations = std::min(h->iter, PPG_MAX_ITERATIONS);
        elapsedSeconds = h->clock_s();
        rc = sync_scalar(h, &elapsedSeconds); if (rc) return rc;
    }
    return PPG_OK;
}

// render, GP:1516-1585
static int ppg_render_device_impl(ppg_integrator *h, float **rgb_dev, ppg_stats *stats);
extern "C" int ppg_render_device(ppg_integrator *h, float **rgb_dev, ppg_stats *stats) { return guarded("ppg_render_device", [&] { return ppg_render_device_impl(h, rgb_dev, stats); }); }
static int ppg_render_device_impl(ppg_integrator *h, float **rgb_dev, ppg_stats *stats) {
    if (!h) return fail(PPG_ERR_INVALID_ARGUMENT, "null handle");
    if (!h->haveScene) return fail(PPG_ERR_NO_SCENE, "ppg_render called before ppg_set_scene");
    CK(cudaSetDevice(h->device));
    h->cancelled.store(false);
    const auto wall0 = std::chrono::steady_clock::now();
    memset(&h->stats, 0, sizeof(h->stats)); h->launches = 0; h->deviceMs = 0; h->evUsed = 0;
    memset(h->treeStatsPending, 0, sizeof(h->treeStatsPending));
    CK(cudaEventRecord(h->evRender0, h->stream));
    int rc = init_tree(h); if (rc) return rc;                                   // m_sdTree = new STree(scene->getAABB()), GP:1519
    rc = ensure_wavefront(h); if (rc) return rc;
    h->iter = 0; h->isFinalIter = false; h->isBuilt = false; h->passesRendered = 0;
    for (auto *b : h->images) delete b;
    h->images.clear(); h->variances.clear();
    rc = clear_film(h); if (rc) return rc;
    h->startTime = std::chrono::steady_clock::now();
    rc = h->prm.budget_type == PPG_BUDGET_SPP ? render_spp(h) : render_time(h);
    if (rc != PPG_OK && rc != PPG_ERR_CANCELLED) return rc;
    const size_t npx = (size_t) h->W * h->H;
    const int blocks = h->numSMs * 4;
    if (h->prm.sample_combination == PPG_COMB_INVERSEVAR && !h->images.empty()) {   // GP:1567-1582
        float totalWeight = 0;
        for (float v : h->variances) totalWeight += 1.0f / v;
        CK(cudaMemsetAsync(h->dRgb.p, 0, 12 * npx, h->stream));
        for (size_t i = 0; i < h->images.size(); ++i) {
            develop_kernel<<<blocks, 256, 0, h->stream>>>(h->images[i]->p, h->dRgb.p, npx, 1.0f / h->variances[i] / totalWeight, 1); h->launches++;
        }
    } else {
        develop_kernel<<<blocks, 256, 0, h->stream>>>(h->dFilm.p, h->dRgb.p, npx, 1.0f, 0); h->launches++;
    }
    if (h->ncclComm && h->world > 1) {     // disjoint tiles: summing the zero-padded frames assembles the film on every rank; on the render stream
        int rc2 = allreduce_sum(h, h->dRgb.p, 3 * npx); if (rc2) return rc2;
    }
    CK(cudaEventRecord(h->evRender1, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->resolve_timers(); finish_tree_stats(h);
    { float ms = 0; cudaEventElapsedTime(&ms, h->evRender0, h->evRender1); h->stats.render_device_ms = ms; }
    if (!h->ncclComm && h->multi()) {      // callback path: the collective runs outside the library's stream, after the timed region
        int rc2 = allreduce_sum(h, h->dRgb.p, 3 * npx); if (rc2) return rc2;
    }
    CK(cudaGetLastError());
    h->stats.total_passes = h->passesRendered;
    h->stats.render_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - wall0).count();
    h->stats.device_seconds = h->deviceMs / 1000.0;
    h->stats.final_variance = h->stats.n_iterations ? h->stats.iterations[h->stats.n_iterations - 1].variance : 0;
    h->stats.kernel_launches = h->launches;
    if (stats) *stats = h->stats;
    if (rgb_dev) *rgb_dev = h->dRgb.p;
    return rc;
}

extern "C" int ppg_render(ppg_integrator *h, float *rgb_out, ppg_stats *stats) {
    float *dev = nullptr;
    const int rc = ppg_render_device(h, &dev, stats);
    if (rc != PPG_OK && rc != PPG_ERR_CANCELLED) return rc;
    if (rgb_out) CK(cudaMemcpy(rgb_out, dev, 12 * (size_t) h->W * h->H, cudaMemcpyDeviceToHost));
    return rc;
}

extern "C" int ppg_copy_from_device(void *host_dst, const void *device_src, size_t bytes) {
    if (!host_dst || !device_src) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    CK(cudaMemcpy(host_dst, device_src, bytes, cudaMemcpyDeviceToHost));
    return PPG_OK;
}

extern "C" int ppg_get_moment_images(ppg_integrator *h, float *sum_rgbw, float *sumsq_rgbw) {
    if (!h || !h->haveScene) return fail(PPG_ERR_NO_SCENE, "no scene");
    CK(cudaSetDevice(h->device));
    const size_t npx = (size_t) h->W * h->H;
    if (sum_rgbw) CK(cudaMemcpy(sum_rgbw, h->dImage.p, 16 * npx, cudaMemcpyDeviceToHost));
    if (sumsq_rgbw) CK(cudaMemcpy(sumsq_rgbw, h->dSqImage.p, 16 * npx, cudaMemcpyDeviceToHost));
    return PPG_OK;
}

// dumpSDTree wire format (GP:1191-1208, 699-711, 945-951): 16 floats camera matrix, then for every leaf with
// sampling weight > 0, in forEachLeaf order (child 0 before child 1): pos, size, mean, u64 weight, u64 nNodes,
// nNodes x 4 x (f32 sum, u16 child)
static int ppg_dump_sdtree_impl(ppg_integrator *h, const char *path);
extern "C" int ppg_dump_sdtree(ppg_integrator *h, const char *path) { return guarded("ppg_dump_sdtree", [&] { return ppg_dump_sdtree_impl(h, path); }); }
static int ppg_dump_sdtree_impl(ppg_integrator *h, const char *path) {
    if (!h || !path) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    if (!h->haveScene || h->capNodes == 0) return fail(PPG_ERR_NO_SCENE, "no SD-tree yet");
    CK(cudaSetDevice(h->device));
    const uint32_t n = h->hNodes;
    std::vector<uint2> sn(n); std::vector<float4> la(n); std::vector<float> ssum(n), sw(n); std::vector<uint32_t> scnt(n);
    CK(cudaMemcpy(sn.data(), h->dSnodes.p, sizeof(uint2) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(la.data(), h->dLeafA.p, sizeof(float4) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ssum.data(), h->dSampSum.p, 4 * (size_t) n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(sw.data(), h->dSampWeight.p, 4 * (size_t) n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(scnt.data(), h->dSampCount.p, 4 * (size_t) n, cudaMemcpyDeviceToHost));
    std::vector<SampNode> pool(std::max<size_t>(h->hTotalBuild, 1));
    CK(cudaMemcpy(pool.data(), h->dSamp.p, sizeof(SampNode) * pool.size(), cudaMemcpyDeviceToHost));
    FILE *f = fopen(path, "wb");
    if (!f) return fail(PPG_ERR_IO, std::string("cannot open ") + path);
    float cm[16];
    const Camera &c = h->cam;   // camera-to-world matrix, row-major (GP:1197-1205)
    cm[0] = c.left.x; cm[1] = c.up.x; cm[2] = c.dir.x; cm[3] = c.o.x; cm[4] = c.left.y; cm[5] = c.up.y; cm[6] = c.dir.y; cm[7] = c.o.y;
    cm[8] = c.left.z; cm[9] = c.up.z; cm[10] = c.dir.z; cm[11] = c.o.z; cm[12] = 0; cm[13] = 0; cm[14] = 0; cm[15] = 1;
    fwrite(cm, 4, 16, f);
    struct E { uint32_t n; float p[3], s[3]; int axis; };
    std::vector<E> st; E root; root.n = 0; root.axis = 0;
    for (int i = 0; i < 3; ++i) { root.p[i] = h->aabbMin[i]; root.s[i] = h->extent[i]; }
    st.push_back(root);
    while (!st.empty()) {
        E e = st.back(); st.pop_back();
        if (sn[e.n].x == 0u) {
            if (!(sw[e.n] > 0)) continue;
            const float mean = (1 / (3.14159265358979323846f * 4 * sw[e.n])) * ssum[e.n];
            fwrite(e.p, 4, 3, f); fwrite(e.s, 4, 3, f); fwrite(&mean, 4, 1, f);
            const uint64_t w64 = (uint64_t) sw[e.n], nn = scnt[e.n];
            fwrite(&w64, 8, 1, f); fwrite(&nn, 8, 1, f);
            uint32_t base; memcpy(&base, &la[e.n].x, 4);
            if ((size_t) base + scnt[e.n] > pool.size()) { fclose(f); return fail(PPG_ERR_IO, "SD-tree is being rebuilt (render cancelled between reset and build): nothing consistent to dump"); }
            for (uint32_t k = 0; k < scnt[e.n]; ++k) {
                const SampNode &q = pool[base + k];
                const float s4[4] = {q.sums.x, q.sums.y, q.sums.z, q.sums.w};
                const uint16_t c4[4] = {(uint16_t) (q.children.x & 0xffff), (uint16_t) (q.children.x >> 16), (uint16_t) (q.children.y & 0xffff), (uint16_t) (q.children.y >> 16)};
                for (int j = 0; j < 4; ++j) { fwrite(&s4[j], 4, 1, f); fwrite(&c4[j], 2, 1, f); }
            }
        } else {
            E a = e, b = e;
            a.s[e.axis] = b.s[e.axis] = e.s[e.axis] / 2; b.p[e.axis] += b.s[e.axis];
            a.axis = b.axis = (e.axis + 1) % 3; a.n = sn[e.n].x; b.n = sn[e.n].y;
            st.push_back(b); st.push_back(a);
        }
    }
    fclose(f);
    return PPG_OK;
}

// ------------------------------------------------------------------ kernel-level entry points on caller-supplied tree arrays
namespace {
struct ReplayRng { const float *v; uint32_t n, i; __device__ float next1D() { return i < n ? v[i++] : 0.5f; } };

__global__ void op_pdf_kernel(const SampNode *pool, const uint32_t *first, const float *tsum, const float *tweight, const uint32_t *qt, const float *qd, size_t n, float *out) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const uint32_t t = qt[i];
        float mean = 0.f; if (tweight[t] != 0.f) mean = (1.f / (PPG_PI * 4.f * tweight[t])) * tsum[t];
        out[i] = dtree_pdf(pool + first[t], mean > 0.f, dir_to_canonical(f3(qd[3 * i], qd[3 * i + 1], qd[3 * i + 2])));
    }
}
__global__ void op_sample_kernel(const SampNode *pool, const uint32_t *first, const float *tsum, const float *tweight, const uint32_t *qt, const float *rnd, size_t stride, size_t n, float *out) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const uint32_t t = qt[i];
        float mean = 0.f; if (tweight[t] != 0.f) mean = (1.f / (PPG_PI * 4.f * tweight[t])) * tsum[t];
        ReplayRng r{rnd + stride * i, (uint32_t) stride, 0u};
        const float3 d = canonical_to_dir(dtree_sample(pool + first[t], mean > 0.f, r));
        out[3 * i] = d.x; out[3 * i + 1] = d.y; out[3 * i + 2] = d.z;
    }
}
__global__ void op_record_kernel(TreeView T, const uint32_t *rt, const float *rd, const float *rrad, const float *rpdf, const float *rw, size_t n, int filter) {
    const size_t nPad = (n + 31) / 32 * 32;
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < nPad; i += (size_t) gridDim.x * blockDim.x) {
        const bool ok = i < n;
        const uint32_t t = ok ? rt[i] : 0u; const float w = ok ? rw[i] : 0.f;
        const bool wOk = ok && isfinite(w) && w > 0.f;
        warp_aggregated_add(T.bweight, t, w, wOk);
        if (wOk) {
            const float4 la = T.leafA[t];
            dtree_record_irradiance(T.bchildren, T.bsums, __float_as_uint(la.y), dir_to_canonical(f3(rd[3 * i], rd[3 * i + 1], rd[3 * i + 2])), rrad[i] / rpdf[i], w, filter);
        }
    }
}
__global__ void op_lookup_kernel(const uint2 *snodes, const uint32_t *table, float3 mn, float3 ext, const float *pts, size_t n, uint32_t *leaf, float *size) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        int lv; const uint32_t l = stree_lookup(snodes, table, mn, ext, f3(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]), lv);
        leaf[i] = l;
        const float3 v = voxel_size(ext, lv);
        size[3 * i] = v.x; size[3 * i + 1] = v.y; size[3 * i + 2] = v.z;
    }
}
// Scene::sampleAttenuatedEmitterDirect at caller-supplied reference points, exactly as the bounce kernel's light-sampling block calls it
__global__ void op_emitter_sample_kernel(SceneView scene, const float *ref, const float *refN, const float *smp, int maxInteractions, size_t n,
                                         float *dOut, float *valueOut, float *pdfOut, float *distOut) {
    const SceneAccess<false> sc(scene);
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const float3 p = f3(ref[3 * i], ref[3 * i + 1], ref[3 * i + 2]), rn = f3(refN[3 * i], refN[3 * i + 1], refN[3 * i + 2]);
        DirectSample ds; ds.value = f3(0, 0, 0); ds.d = f3(0, 0, 0); ds.pdf = 0.f; float dist = 0.f;
        const bool ok = sample_emitter_direct<true>(sc, p, rn, smp[2 * i], smp[2 * i + 1], ds, dist);
        if (ok) ds.value = ds.value * eval_transmittance(sc, p, ds.d, dist, maxInteractions);
        else { ds.value = f3(0, 0, 0); ds.pdf = 0.f; dist = 0.f; }
        dOut[3 * i] = ds.d.x; dOut[3 * i + 1] = ds.d.y; dOut[3 * i + 2] = ds.d.z;
        valueOut[3 * i] = ds.value.x; valueOut[3 * i + 1] = ds.value.y; valueOut[3 * i + 2] = ds.value.z;
        pdfOut[i] = ds.pdf; distOut[i] = dist;
    }
}
__global__ void op_env_pdf_kernel(SceneView scene, const float *dir, size_t n, float *pdfOut, float *valueOut) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const float3 d = f3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        pdfOut[i] = pdf_emitter_direct<true>(scene, PPG_ENV_EMITTER, f3(0, 0, 0), f3(0, 0, 0), d, f3(0, 0, 0), 0.f);
        if (valueOut) { const float3 v = env_eval(scene, d); valueOut[3 * i] = v.x; valueOut[3 * i + 1] = v.y; valueOut[3 * i + 2] = v.z; }
    }
}
template <class T> struct Up {
    DevBuf<T> b;
    int up(const T *host, size_t n) { if (b.alloc(std::max<size_t>(n, 1)) != cudaSuccess) return 1; return n ? cudaMemcpy(b.p, host, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess : 0; }
};
static int op_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(PPG_ERR_NO_DEVICE, "no CUDA device available (no CPU fallback)"); }
    if (device < 0) device = 0;
    if (device >= ndev) return fail(PPG_ERR_NO_DEVICE, "device index out of range");
    CK(cudaSetDevice(device));
    return PPG_OK;
}
static std::vector<SampNode> to_pool(const float *sums, const uint16_t *children, size_t n) {
    std::vector<SampNode> pool(n);
    for (size_t i = 0; i < n; ++i) {
        pool[i].sums = make_float4(sums[4 * i], sums[4 * i + 1], sums[4 * i + 2], sums[4 * i + 3]);
        pool[i].children = make_uint2((uint32_t) children[4 * i] | ((uint32_t) children[4 * i + 1] << 16), (uint32_t) children[4 * i + 2] | ((uint32_t) children[4 * i + 3] << 16));
        pool[i].pad = make_uint2(0u, 0u);
    }
    return pool;
}
}  // namespace

extern "C" int ppg_op_dtree_pdf(int device, const float *sums, const uint16_t *children, size_t n_nodes, const uint32_t *tree_first_node,
                                const float *tree_sum, const float *tree_weight, size_t n_trees, const uint32_t *query_tree, const float *query_dir,
                                size_t n, float *pdf_out) {
    int rc = op_device(device); if (rc) return rc;
    std::vector<SampNode> pool = to_pool(sums, children, n_nodes);
    Up<SampNode> dp; Up<uint32_t> df, dq; Up<float> ds, dw, dd; DevBuf<float> out;
    if (dp.up(pool.data(), n_nodes) || df.up(tree_first_node, n_trees) || ds.up(tree_sum, n_trees) || dw.up(tree_weight, n_trees) || dq.up(query_tree, n) || dd.up(query_dir, 3 * n))
        return fail(PPG_ERR_CUDA, "upload failed");
    CK(out.alloc(std::max<size_t>(n, 1)));
    if (n) op_pdf_kernel<<<296, 256>>>(dp.b.p, df.b.p, ds.b.p, dw.b.p, dq.b.p, dd.b.p, n, out.p);
    CK(cudaGetLastError());
    CK(cudaMemcpy(pdf_out, out.p, 4 * n, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
extern "C" int ppg_op_dtree_sample(int device, const float *sums, const uint16_t *children, size_t n_nodes, const uint32_t *tree_first_node,
                                   const float *tree_sum, const float *tree_weight, size_t n_trees, const uint32_t *query_tree, const float *rnd,
                                   size_t rnd_stride, size_t n, float *dir_out) {
    int rc = op_device(device); if (rc) return rc;
    std::vector<SampNode> pool = to_pool(sums, children, n_nodes);
    Up<SampNode> dp; Up<uint32_t> df, dq; Up<float> ds, dw, dr; DevBuf<float> out;
    if (dp.up(pool.data(), n_nodes) || df.up(tree_first_node, n_trees) || ds.up(tree_sum, n_trees) || dw.up(tree_weight, n_trees) || dq.up(query_tree, n) || dr.up(rnd, rnd_stride * n))
        return fail(PPG_ERR_CUDA, "upload failed");
    CK(out.alloc(std::max<size_t>(3 * n, 1)));
    if (n) op_sample_kernel<<<296, 256>>>(dp.b.p, df.b.p, ds.b.p, dw.b.p, dq.b.p, dr.b.p, rnd_stride, n, out.p);
    CK(cudaGetLastError());
    CK(cudaMemcpy(dir_out, out.p, 12 * n, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
extern "C" int ppg_op_dtree_record(int device, float *sums_inout, const uint16_t *children, size_t n_nodes, const uint32_t *tree_first_node,
                                   float *tree_weight_inout, size_t n_trees, const uint32_t *rec_tree, const float *rec_dir, const float *rec_radiance,
                                   const float *rec_wo_pdf, const float *rec_weight, size_t n, int filter) {
    int rc = op_device(device); if (rc) return rc;
    std::vector<uint2> bch(n_nodes);
    for (size_t i = 0; i < n_nodes; ++i)
        bch[i] = make_uint2((uint32_t) children[4 * i] | ((uint32_t) children[4 * i + 1] << 16), (uint32_t) children[4 * i + 2] | ((uint32_t) children[4 * i + 3] << 16));
    std::vector<float4> la(n_trees);
    for (size_t t = 0; t < n_trees; ++t) { uint32_t b = tree_first_node[t]; float fb; memcpy(&fb, &b, 4); la[t] = make_float4(fb, fb, 0.f, 0.f); }
    Up<uint2> dch; Up<float4> dla; Up<float> dsums, dwt, dd, drad, dpdf, dw; Up<uint32_t> drt;
    if (dch.up(bch.data(), n_nodes) || dla.up(la.data(), n_trees) || dsums.up(sums_inout, 4 * n_nodes) || dwt.up(tree_weight_inout, n_trees) || drt.up(rec_tree, n) ||
        dd.up(rec_dir, 3 * n) || drad.up(rec_radiance, n) || dpdf.up(rec_wo_pdf, n) || dw.up(rec_weight, n))
        return fail(PPG_ERR_CUDA, "upload failed");
    TreeView T; memset(&T, 0, sizeof(T));
    T.leafA = dla.b.p; T.bchildren = dch.b.p; T.bsums = reinterpret_cast<float4 *>(dsums.b.p); T.bweight = dwt.b.p;
    if (n) op_record_kernel<<<296, 256>>>(T, drt.b.p, dd.b.p, drad.b.p, dpdf.b.p, dw.b.p, n, filter);
    CK(cudaGetLastError());
    CK(cudaMemcpy(sums_inout, dsums.b.p, 16 * n_nodes, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(tree_weight_inout, dwt.b.p, 4 * n_trees, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
__global__ void op_sum_kernel(float *acc, const float *x, size_t n) {
    for (size_t i = blockIdx.x * (size_t) blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) acc[i] += x[i];
}
// The sampling-fraction replay of render_batch on caller-given records: the same kernels, in the same order, with the same launch shapes.
extern "C" int ppg_op_fraction_replay(int device, const float *states, size_t n_leaves, const float *rec_a, const float *rec_b, const size_t *counts,
                                      int n_batches, int replicas, int merge, size_t cap, int loss, float *states_out, float *replica_out, float *theta_out,
                                      float *sorted_a_out, float *sorted_b_out, unsigned long long *progress_out) {
  return guarded("ppg_op_fraction_replay", [&]() -> int {
    if (!states || !counts || !n_leaves || n_leaves >= 0xFFFFFFFFull || n_batches < 1 || replicas < 1 || !cap || cap >= 0xFFFFFFFFull ||
        (loss != PPG_LOSS_KL && loss != PPG_LOSS_VAR))
        return fail(PPG_ERR_INVALID_ARGUMENT, "ppg_op_fraction_replay: bad arguments");
    const size_t R = (size_t) replicas, L = n_leaves;
    const bool doMerge = replicas > 1 || merge != 0;
    size_t nTotal = 0;
    for (size_t g = 0; g < (size_t) n_batches * R; ++g) nTotal += counts[g];
    if (nTotal && (!rec_a || !rec_b)) return fail(PPG_ERR_INVALID_ARGUMENT, "ppg_op_fraction_replay: null records");
    for (size_t i = 0; i < nTotal; ++i) { uint32_t leaf; memcpy(&leaf, rec_a + 4 * i, 4); if (leaf >= L) return fail(PPG_ERR_INVALID_ARGUMENT, "ppg_op_fraction_replay: leaf index out of range"); }
    int rc = op_device(device); if (rc) return rc;
    int dev = 0, numSMs = 0; CK(cudaGetDevice(&dev)); CK(cudaDeviceGetAttribute(&numSMs, cudaDevAttrMultiProcessorCount, dev));
    const uint32_t nNodes = (uint32_t) L;
    Up<float> dAdam; Up<uint32_t> dNodes;
    if (dAdam.up(states, 6 * L) || dNodes.up(&nNodes, 1)) return fail(PPG_ERR_CUDA, "upload failed");
    DevBuf<float4> dLeafA, dRecA, dSortA; DevBuf<float2> dRecB, dSortB; DevBuf<uint32_t> dCount, dCursor, dOffset, dScalars;
    DevBuf<float> dBefore, dStart, dOut6, dSum6; DevBuf<unsigned long long> dProgress;
    CK(dLeafA.alloc(L)); CK(dCount.alloc(L)); CK(dCursor.alloc(L)); CK(dOffset.alloc(L)); CK(dScalars.alloc(2)); CK(dBefore.alloc(4 * L)); CK(dProgress.alloc(2));
    CK(dRecA.alloc(cap)); CK(dRecB.alloc(cap)); CK(dSortA.alloc(cap)); CK(dSortB.alloc(cap));
    if (doMerge) { CK(dStart.alloc(6 * L)); CK(dOut6.alloc(6 * L)); CK(dSum6.alloc(6 * L)); }
    CK(cudaMemset(dLeafA.p, 0, 16 * L)); CK(cudaMemset(dCount.p, 0, 4 * L)); CK(cudaMemset(dCursor.p, 0, 4 * L));     // as ensure_tree leaves them
    MaintParams M; memset(&M, 0, sizeof(M));
    M.adam = dAdam.b.p; M.leafA = dLeafA.p; M.nNodes = dNodes.b.p; M.capNodes = nNodes;
    const float ratioPower = loss == PPG_LOSS_KL ? 1.0f : 2.0f;
    std::vector<float> la(4 * L);
    size_t first = 0;
    for (int b = 0; b < n_batches; ++b) {
        adam_pack_kernel<<<numSMs, 256>>>(M, nullptr, dBefore.p, nullptr, 0);
        if (doMerge) { CK(cudaMemcpy(dStart.p, dAdam.b.p, 24 * L, cudaMemcpyDeviceToDevice)); CK(cudaMemset(dSum6.p, 0, 24 * L)); }
        for (size_t r = 0; r < R; ++r) {
            const size_t total = counts[(size_t) b * R + r], kept = std::min(total, cap);
            if (r) CK(cudaMemcpy(dAdam.b.p, dStart.p, 24 * L, cudaMemcpyDeviceToDevice));
            // the commit launch: `total` records appended, the first `cap` of them stored
            if (kept) { CK(cudaMemcpy(dRecA.p, rec_a + 4 * first, 16 * kept, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dRecB.p, rec_b + 2 * first, 8 * kept, cudaMemcpyHostToDevice)); }
            const uint32_t total32 = (uint32_t) std::min<size_t>(total, 0xFFFFFFFFu);
            CK(cudaMemcpy(dScalars.p, &total32, 4, cudaMemcpyHostToDevice));
            adam_hist_kernel<<<numSMs * 4, 256>>>(dRecA.p, dScalars.p, (uint32_t) cap, dCount.p);
            exclusive_scan_kernel<<<1, 1024>>>(dCount.p, dOffset.p, dNodes.b.p, dScalars.p + 1);
            adam_scatter_kernel<<<numSMs * 4, 256>>>(dRecA.p, dRecB.p, dScalars.p, (uint32_t) cap, dOffset.p, dCursor.p, dSortA.p, dSortB.p);
            adam_seq_kernel<<<numSMs * 16, 128>>>(M, dSortA.p, dSortB.p, dOffset.p, dCount.p, dCursor.p, ratioPower);
            CK(cudaGetLastError());
            if (kept && sorted_a_out) CK(cudaMemcpy(sorted_a_out + 4 * first, dSortA.p, 16 * kept, cudaMemcpyDeviceToHost));
            if (kept && sorted_b_out) CK(cudaMemcpy(sorted_b_out + 2 * first, dSortB.p, 8 * kept, cudaMemcpyDeviceToHost));
            if (replica_out) CK(cudaMemcpy(replica_out + ((size_t) b * R + r) * 6 * L, dAdam.b.p, 24 * L, cudaMemcpyDeviceToHost));
            if (doMerge) {
                adam_pack_kernel<<<numSMs, 256>>>(M, dOut6.p, dBefore.p, nullptr, 1);
                op_sum_kernel<<<numSMs, 256>>>(dSum6.p, dOut6.p, 6 * L);          // the allreduce, summing the replicas in order
            }
            first += total;
        }
        if (doMerge) adam_merge_kernel<<<numSMs, 256>>>(M, dSum6.p, dBefore.p, 1.0f / (float) R, (float) (R - 1));
        CK(cudaMemset(dProgress.p, 0, 16));
        adam_progress_kernel<<<numSMs, 256>>>(M, dBefore.p, dProgress.p);
        CK(cudaGetLastError());
        if (progress_out) CK(cudaMemcpy(progress_out + 2 * b, dProgress.p, 16, cudaMemcpyDeviceToHost));
        if (states_out) CK(cudaMemcpy(states_out + (size_t) b * 6 * L, dAdam.b.p, 24 * L, cudaMemcpyDeviceToHost));
        if (theta_out) {
            CK(cudaMemcpy(la.data(), dLeafA.p, 16 * L, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < L; ++i) theta_out[(size_t) b * L + i] = la[4 * i + 2];
        }
    }
    return PPG_OK;
  });
}
// The acceleration structure ppg_set_scene builds, on the host alone (no CUDA device needed): for tests of the builder and for timing it.
extern "C" int ppg_op_bvh_build(const float *positions, const uint32_t *indices, size_t n_triangles, int threads, float *nodes_out, size_t nodes_capacity,
                                uint32_t *order_out, size_t *n_nodes_out, int *max_depth_out, double *ms_out) {
  return guarded("ppg_op_bvh_build", [&]() -> int {
    if (!positions || !indices || !n_triangles || n_triangles >= 0xFFFFFFFFull) return fail(PPG_ERR_INVALID_ARGUMENT, "ppg_op_bvh_build: empty or oversized input");
    const uint32_t nt = (uint32_t) n_triangles;
    const auto t0 = std::chrono::steady_clock::now();
    const int T = threads > 0 ? threads : host_threads();
    std::vector<H3> tmin(nt), tmax(nt);
    triangle_bounds(positions, indices, nt, tmin, tmax, T);
    HostBvh bvh; build_bvh(tmin, tmax, bvh, T);
    if (ms_out) *ms_out = elapsed_ms(t0);
    if (n_nodes_out) *n_nodes_out = bvh.nodes.size() / 8;
    if (max_depth_out) *max_depth_out = bvh.maxDepth;
    if (nodes_out) { if (nodes_capacity < bvh.nodes.size() / 8) return fail(PPG_ERR_INVALID_ARGUMENT, "ppg_op_bvh_build: nodes_out too small (2 * n_triangles + 1 always suffices)"); memcpy(nodes_out, bvh.nodes.data(), bvh.nodes.size() * 4); }
    if (order_out) memcpy(order_out, bvh.order.data(), (size_t) nt * 4);
    return PPG_OK;
  });
}
extern "C" int ppg_op_emitter_sample_direct(ppg_integrator *h, size_t n, const float *ref, const float *ref_n, const float *sample, int max_interactions,
                                            float *d_out, float *value_out, float *pdf_out, float *dist_out) {
    if (!h || !h->haveScene) return fail(PPG_ERR_NO_SCENE, "ppg_op_emitter_sample_direct needs a handle with a scene");
    if (!ref || !ref_n || !sample || !d_out || !value_out || !pdf_out || !dist_out) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    if (!h->fullFeature) return fail(PPG_ERR_UNSUPPORTED, "emitter-level ops run the full-feature code path (scene with spheres, textures, non-diffuse BSDFs or an environment emitter)");
    CK(cudaSetDevice(h->device));
    Up<float> dr, dn, ds; DevBuf<float> od, ov, op, ot;
    if (dr.up(ref, 3 * n) || dn.up(ref_n, 3 * n) || ds.up(sample, 2 * n)) return fail(PPG_ERR_CUDA, "upload failed");
    CK(od.alloc(std::max<size_t>(3 * n, 1))); CK(ov.alloc(std::max<size_t>(3 * n, 1))); CK(op.alloc(std::max<size_t>(n, 1))); CK(ot.alloc(std::max<size_t>(n, 1)));
    if (n) op_emitter_sample_kernel<<<296, 128>>>(h->sceneView, dr.b.p, dn.b.p, ds.b.p, max_interactions, n, od.p, ov.p, op.p, ot.p);
    CK(cudaGetLastError());
    CK(cudaMemcpy(d_out, od.p, 12 * n, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(value_out, ov.p, 12 * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(pdf_out, op.p, 4 * n, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(dist_out, ot.p, 4 * n, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
extern "C" int ppg_op_env_pdf(ppg_integrator *h, size_t n, const float *d, float *pdf_out, float *value_out) {
    if (!h || !h->haveScene) return fail(PPG_ERR_NO_SCENE, "ppg_op_env_pdf needs a handle with a scene");
    if (!h->sceneView.envW) return fail(PPG_ERR_NO_SCENE, "the scene has no environment emitter");
    if (!d || !pdf_out) return fail(PPG_ERR_INVALID_ARGUMENT, "null argument");
    CK(cudaSetDevice(h->device));
    Up<float> dd; DevBuf<float> op, ov;
    if (dd.up(d, 3 * n)) return fail(PPG_ERR_CUDA, "upload failed");
    CK(op.alloc(std::max<size_t>(n, 1))); CK(ov.alloc(std::max<size_t>(3 * n, 1)));
    if (n) op_env_pdf_kernel<<<296, 128>>>(h->sceneView, dd.b.p, n, op.p, value_out ? ov.p : nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(pdf_out, op.p, 4 * n, cudaMemcpyDeviceToHost));
    if (value_out) CK(cudaMemcpy(value_out, ov.p, 12 * n, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
extern "C" int ppg_op_stree_lookup(int device, const uint32_t *node_children, size_t n_nodes, const float aabb_min[3], const float aabb_extent[3],
                                   const float *points, size_t n, uint32_t *leaf_out, float *size_out) {
    int rc = op_device(device); if (rc) return rc;
    Up<uint2> dn; Up<float> dp; DevBuf<uint32_t> dl; DevBuf<float> dsz;
    if (dn.up(reinterpret_cast<const uint2 *>(node_children), n_nodes) || dp.up(points, 3 * n)) return fail(PPG_ERR_CUDA, "upload failed");
    CK(dl.alloc(std::max<size_t>(n, 1))); CK(dsz.alloc(std::max<size_t>(3 * n, 1)));
    DevBuf<uint32_t> dt; CK(dt.alloc((size_t) 1 << (3 * PPG_STREE_TABLE_BITS)));
    stree_table_kernel<<<296, 256>>>(dn.b.p, dt.p);     // the same prefix table the render kernels use
    if (n) op_lookup_kernel<<<296, 256>>>(dn.b.p, dt.p, make_float3(aabb_min[0], aabb_min[1], aabb_min[2]), make_float3(aabb_extent[0], aabb_extent[1], aabb_extent[2]), dp.b.p, n, dl.p, dsz.p);
    CK(cudaGetLastError());
    CK(cudaMemcpy(leaf_out, dl.p, 4 * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(size_out, dsz.p, 12 * n, cudaMemcpyDeviceToHost));
    return PPG_OK;
}
