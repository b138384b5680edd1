// TEST INFRASTRUCTURE -- C API of the CPU oracle (see ppg_oracle.h).
// Built twice by oracle/Makefile:
//   oracle/libppg_oracle.so           restated SD-tree (sdtree_port.h)              -- "port"
//   oracle/_ref/libppg_oracle_ref.so  reference SD-tree compiled verbatim (-DPPGO_BACKEND_REF,
//                                     guided_path.cpp:25-1008 piped in ahead of this file) -- "reference" trees
#ifdef PPGO_BACKEND_REF
#include "sdtree_ref/ref_backend.h"
typedef ppgo::RefBackend BackendT;
#else
#include "backend_port.h"
typedef ppgo::PortBackend BackendT;
#endif
#include "ppg_oracle.h"

#include <memory>

using namespace ppgo;

struct ppgo_handle {
    std::unique_ptr<Tracer<BackendT>> tracer;   // when a scene is given
    std::unique_ptr<BackendT> tree;             // tree-only handle
    std::vector<float> capLi; std::vector<int32_t> capDepth; float *userLi = nullptr; int32_t *userDepth = nullptr;
    BackendT &T() { return tracer ? tracer->tree : *tree; }
};

extern "C" {

int ppgo_is_reference_backend(void) {
#ifdef PPGO_BACKEND_REF
    return 1;
#else
    return 0;
#endif
}

ppgo_handle *ppgo_create(const ppg_params *p, const ppg_scene_desc *scene, const float *aabb_min, const float *aabb_max, int nthreads) {
    ppgo_handle *h = new ppgo_handle();
    if (nthreads <= 0) nthreads = omp_get_max_threads();
    if (scene) h->tracer.reset(new Tracer<BackendT>(*p, *scene, nthreads));
    else h->tree.reset(new BackendT(aabb_min, aabb_max));
    return h;
}
void ppgo_destroy(ppgo_handle *h) { delete h; }

int ppgo_set_capture(ppgo_handle *h, float *li, int32_t *depth) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    Tracer<BackendT> &t = *h->tracer;
    const size_t n = (size_t) t.W * t.H * t.prm.spp_per_pass;
    h->capLi.assign(3 * n, 0.f); h->capDepth.assign(n, 0);
    h->userLi = li; h->userDepth = depth;
    t.captureLi = &h->capLi; t.captureDepth = &h->capDepth;
    return PPG_OK;
}
static void flush_capture(ppgo_handle *h) {
    if (h->userLi) std::memcpy(h->userLi, h->capLi.data(), h->capLi.size() * sizeof(float));
    if (h->userDepth) std::memcpy(h->userDepth, h->capDepth.data(), h->capDepth.size() * sizeof(int32_t));
}

int ppgo_render(ppgo_handle *h, float *rgb_out, ppg_stats *stats) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    const bool ok = h->tracer->render(rgb_out);
    if (stats) *stats = h->tracer->stats;
    flush_capture(h);
    return ok ? PPG_OK : PPG_ERR_CANCELLED;
}

int ppgo_set_shard(ppgo_handle *h, int rank, int world_size) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    h->tracer->shardRank = rank; h->tracer->shardWorld = world_size; return PPG_OK;
}
int ppgo_set_allreduce(ppgo_handle *h, ppg_allreduce_fn cb, void *user) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    h->tracer->allreduce = cb; h->tracer->allreduceUser = user; return PPG_OK;
}

int ppgo_step_reset(ppgo_handle *h, int iter) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    Tracer<BackendT> &t = *h->tracer;
    if (iter == 0) { t.passesRendered = 0; t.startTime = std::chrono::steady_clock::now(); }
    t.iter = iter; std::fill(t.film.begin(), t.film.end(), 0.f);
    t.doNee = t.doNeeWithSpp(t.passesRendered * t.prm.spp_per_pass);
    t.resetSDTree();
    return PPG_OK;
}
int ppgo_step_passes(ppgo_handle *h, int n_passes, int is_final, float *variance_out) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    Tracer<BackendT> &t = *h->tracer;
    t.isFinalIter = is_final != 0;
    ppg_iteration_stats st; std::memset(&st, 0, sizeof(st));
    const ppg_budget_type keep = (ppg_budget_type) t.prm.budget_type; t.prm.budget_type = PPG_BUDGET_SPP;
    float var = 0; t.performRenderPasses(var, n_passes, st);
    t.prm.budget_type = keep;
    if (variance_out) *variance_out = var;
    flush_capture(h);
    return PPG_OK;
}
int ppgo_step_build(ppgo_handle *h, ppg_iteration_stats *st) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    ppg_iteration_stats tmp; std::memset(&tmp, 0, sizeof(tmp));
    h->tracer->buildSDTree(tmp);
    if (st) *st = tmp;
    return PPG_OK;
}
int ppgo_get_moment_images(ppgo_handle *h, float *sum_rgbw, float *sumsq_rgbw) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    if (sum_rgbw) std::memcpy(sum_rgbw, h->tracer->image.data(), h->tracer->image.size() * sizeof(float));
    if (sumsq_rgbw) std::memcpy(sumsq_rgbw, h->tracer->sqImage.data(), h->tracer->sqImage.size() * sizeof(float));
    return PPG_OK;
}

int ppgo_bsdf_eval_pdf(const ppg_bsdf *b, size_t n, const float *wi, const float *wo, float *eval_out, float *pdf_out, const float *tables) {
    for (size_t i = 0; i < n; ++i) {
        const F3 a = f3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]), c = f3(wo[3 * i], wo[3 * i + 1], wo[3 * i + 2]);
        const F3 e = bsdf_eval(*b, a, c, tables);
        eval_out[3 * i] = e.x; eval_out[3 * i + 1] = e.y; eval_out[3 * i + 2] = e.z; pdf_out[i] = bsdf_pdf(*b, a, c, tables);
    }
    return PPG_OK;
}
int ppgo_bsdf_sample(const ppg_bsdf *b, size_t n, const float *wi, const float *sample, float *wo_out, float *weight_out, float *pdf_out, uint8_t *delta_out, const float *tables) {
    for (size_t i = 0; i < n; ++i) {
        BsdfSample bs; bs.wo = f3(0, 0, 0); float pdf = 0;
        Pcg32 extra; extra.seed(splitmix64(i), i);                      // the model's own draws from the path sampler (roughdielectric)
        const F3 w = bsdf_sample(*b, f3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]), sample[2 * i], sample[2 * i + 1], bs, pdf, tables, &extra);
        wo_out[3 * i] = bs.wo.x; wo_out[3 * i + 1] = bs.wo.y; wo_out[3 * i + 2] = bs.wo.z;
        weight_out[3 * i] = w.x; weight_out[3 * i + 1] = w.y; weight_out[3 * i + 2] = w.z; pdf_out[i] = pdf; if (delta_out) delta_out[i] = bs.delta;
    }
    return PPG_OK;
}

// ---- the restated microfacet distribution (ppg_cpu_tracer.h: struct Microfacet, mts_erf / mts_erfinv), entry by entry like oracle/microfacet_ref/wrapper.h
int ppgo_mf_eval(int type, float alpha, size_t n, const float *m, float *out) {
    const Microfacet d(type, alpha);
    for (size_t i = 0; i < n; ++i) out[i] = d.eval(f3(m[3 * i], m[3 * i + 1], m[3 * i + 2]));
    return PPG_OK;
}
int ppgo_mf_smith_g1(int type, float alpha, size_t n, const float *v, const float *m, float *out) {
    const Microfacet d(type, alpha);
    for (size_t i = 0; i < n; ++i) out[i] = d.smithG1(f3(v[3 * i], v[3 * i + 1], v[3 * i + 2]), f3(m[3 * i], m[3 * i + 1], m[3 * i + 2]));
    return PPG_OK;
}
int ppgo_mf_pdf(int type, float alpha, size_t n, const float *wi, const float *m, float *out) {
    const Microfacet d(type, alpha);
    for (size_t i = 0; i < n; ++i) out[i] = d.pdfVisible(f3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]), f3(m[3 * i], m[3 * i + 1], m[3 * i + 2]));
    return PPG_OK;
}
int ppgo_mf_sample(int type, float alpha, size_t n, const float *wi, const float *sample, float *m_out, float *pdf_out) {
    const Microfacet d(type, alpha);
    for (size_t i = 0; i < n; ++i) {
        const F3 w = f3(wi[3 * i], wi[3 * i + 1], wi[3 * i + 2]);
        const F3 m = d.sampleVisible(w, sample[2 * i], sample[2 * i + 1]);
        m_out[3 * i] = m.x; m_out[3 * i + 1] = m.y; m_out[3 * i + 2] = m.z; pdf_out[i] = d.pdfVisible(w, m);
    }
    return PPG_OK;
}
// the restated helpers of src/libcore/util.cpp / warp.cpp
int ppgo_fresnel_dielectric_ext(size_t n, const float *cosThetaI, float eta, float *f_out, float *cos_t_out) {
    for (size_t i = 0; i < n; ++i) { float ct = 0; f_out[i] = fresnel_dielectric_ext(cosThetaI[i], ct, eta); cos_t_out[i] = ct; }
    return PPG_OK;
}
int ppgo_fresnel_conductor_exact(size_t n, const float *cosThetaI, const float eta[3], const float k[3], float *out) {
    for (size_t i = 0; i < n; ++i) for (int c = 0; c < 3; ++c) out[3 * i + c] = fresnel_conductor_exact(cosThetaI[i], eta[c], k[c]);
    return PPG_OK;
}
int ppgo_coordinate_system(size_t n, const float *a, float *b_out, float *c_out) {
    for (size_t i = 0; i < n; ++i) {
        F3 b, c; coordinate_system(f3(a[3 * i], a[3 * i + 1], a[3 * i + 2]), b, c);
        b_out[3 * i] = b.x; b_out[3 * i + 1] = b.y; b_out[3 * i + 2] = b.z; c_out[3 * i] = c.x; c_out[3 * i + 1] = c.y; c_out[3 * i + 2] = c.z;
    }
    return PPG_OK;
}
int ppgo_square_to_cosine_hemisphere(size_t n, const float *sample, float *out) {
    for (size_t i = 0; i < n; ++i) { const F3 v = square_to_cosine_hemisphere(sample[2 * i], sample[2 * i + 1]); out[3 * i] = v.x; out[3 * i + 1] = v.y; out[3 * i + 2] = v.z; }
    return PPG_OK;
}
int ppgo_triaccel(size_t n, const float *A, const float *B, const float *C, const float *o, const float *d, const float *mint, const float *maxt,
                  int *k_out, float *consts_out, unsigned char *hit_out, float *tuv_out) {
    for (size_t i = 0; i < n; ++i) {
        TriAccelP t; t.k = 0; t.n_u = t.n_v = t.n_d = t.a_u = t.a_v = t.b_nu = t.b_nv = t.c_nu = t.c_nv = 0;
        triaccel_load(t, f3(A[3 * i], A[3 * i + 1], A[3 * i + 2]), f3(B[3 * i], B[3 * i + 1], B[3 * i + 2]), f3(C[3 * i], C[3 * i + 1], C[3 * i + 2]));
        k_out[i] = t.k;
        const float c9[9] = {t.n_u, t.n_v, t.n_d, t.a_u, t.a_v, t.b_nu, t.b_nv, t.c_nu, t.c_nv};
        for (int j = 0; j < 9; ++j) consts_out[9 * i + j] = c9[j];
        float u = 0, v = 0, tt = 0;
        hit_out[i] = triaccel_intersect(t, f3(o[3 * i], o[3 * i + 1], o[3 * i + 2]), f3(d[3 * i], d[3 * i + 1], d[3 * i + 2]), mint[i], maxt[i], u, v, tt) ? 1 : 0;
        tuv_out[3 * i] = tt; tuv_out[3 * i + 1] = u; tuv_out[3 * i + 2] = v;
    }
    return PPG_OK;
}
// RoughTransmittance::eval with alpha and eta fixed (rtrans.h:183-193): |cos|^(1/4) -> evalCubicInterp1D over PPG_BSDF_TABLE_SIZE samples, then the clamp of :233
int ppgo_rough_transmittance(size_t n, const float *cosTheta, const float *values, float *out) {
    for (size_t i = 0; i < n; ++i) out[i] = rough_transmittance(values, cosTheta[i]);
    return PPG_OK;
}
// the discrete distributions of the light sampling as the tracer builds and uses them: cumulative weights normalised like DiscreteDistribution::normalize
// (Scene::buildEmitterSamplers), Scene::cdfSample, and the sample reuse of sample_emitter_direct
int ppgo_discrete(size_t n_entries, const float *weights, size_t n, const float *sample, float *pdf_out, float *sum_out, unsigned *index_out, float *reused_out) {
    std::vector<float> cdf(1, 0.0f);
    for (size_t i = 0; i < n_entries; ++i) cdf.push_back(cdf.back() + weights[i]);
    const float sum = cdf.back(); *sum_out = sum;
    if (sum > 0) { const float nrm = 1.0f / sum; for (size_t i = 1; i < cdf.size(); ++i) cdf[i] *= nrm; cdf.back() = 1.0f; }
    for (size_t i = 0; i < n_entries; ++i) pdf_out[i] = cdf[i + 1] - cdf[i];
    for (size_t i = 0; i < n; ++i) {
        const size_t k = Scene::cdfSample(cdf, sample[i]);
        index_out[i] = (unsigned) k; reused_out[i] = (sample[i] - cdf[k]) / (cdf[k + 1] - cdf[k]);
    }
    return PPG_OK;
}
int ppgo_mf_erf(size_t n, const float *x, float *erf_out, float *erfinv_out) {
    for (size_t i = 0; i < n; ++i) { erf_out[i] = mts_erf(x[i]); erfinv_out[i] = mts_erfinv(x[i]); }
    return PPG_OK;
}

// Scene::sampleAttenuatedEmitterDirect at n reference points (area, sphere and environment emitters); pdf 0 = the sample carries nothing
int ppgo_emitter_sample_direct(ppgo_handle *h, size_t n, const float *ref, const float *ref_n, const float *sample, int max_interactions,
                               float *d_out, float *value_out, float *pdf_out, float *dist_out) {
    if (!h->tracer) return PPG_ERR_NO_SCENE;
    const Scene &sc = h->tracer->sc;
    for (size_t i = 0; i < n; ++i) {
        DirectSample ds; ds.value = f3(0, 0, 0); ds.d = f3(0, 0, 0); ds.pdf = 0; ds.dist = 0;
        const bool ok = sample_emitter_direct(sc, f3(ref[3 * i], ref[3 * i + 1], ref[3 * i + 2]), f3(ref_n[3 * i], ref_n[3 * i + 1], ref_n[3 * i + 2]),
                                              sample[2 * i], sample[2 * i + 1], ds, max_interactions);
        if (!ok) { ds.value = f3(0, 0, 0); ds.pdf = 0; }
        d_out[3 * i] = ds.d.x; d_out[3 * i + 1] = ds.d.y; d_out[3 * i + 2] = ds.d.z;
        value_out[3 * i] = ds.value.x; value_out[3 * i + 1] = ds.value.y; value_out[3 * i + 2] = ds.value.z;
        pdf_out[i] = ds.pdf; dist_out[i] = ok ? ds.dist : 0.f;
    }
    return PPG_OK;
}
// Texture2D::eval / evalGradient of texture `tex` of the handle's scene at n texture coordinates (the per-vertex uv BEFORE the texture's own scale / offset):
// rgb_out 3n (BitmapTexture::eval -> evalBilinear level 0), grad_out 2n (the luminances of d/du, d/dv that BumpMap::getFrame uses)
int ppgo_texture_eval(ppgo_handle *h, uint32_t tex, size_t n, const float *uv, float *rgb_out, float *grad_out) {
    if (!h->tracer || tex >= h->tracer->sc.textures.size()) return PPG_ERR_INVALID_ARGUMENT;
    const Scene &sc = h->tracer->sc;
    for (size_t i = 0; i < n; ++i) {
        const F3 c = sc.evalTexture(tex, uv[2 * i], uv[2 * i + 1]);
        rgb_out[3 * i] = c.x; rgb_out[3 * i + 1] = c.y; rgb_out[3 * i + 2] = c.z;
        sc.evalTextureGradientLum(tex, uv[2 * i], uv[2 * i + 1], grad_out[2 * i], grad_out[2 * i + 1]);
    }
    return PPG_OK;
}
// Scene::pdfEmitterDirect of the environment emitter for n world directions, and its radiance there (evalEnvironment)
int ppgo_env_pdf(ppgo_handle *h, size_t n, const float *d, float *pdf_out, float *value_out) {
    if (!h->tracer || !h->tracer->sc.hasEnvironment()) return PPG_ERR_NO_SCENE;
    const Scene &sc = h->tracer->sc;
    for (size_t i = 0; i < n; ++i) {
        const F3 dw = f3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
        pdf_out[i] = pdf_emitter_direct(sc, kEnvEmitter, f3(0, 0, 0), f3(0, 0, 0), dw, f3(0, 0, 0), 0.f);
        if (value_out) { const F3 v = sc.evalEnvironment(dw); value_out[3 * i] = v.x; value_out[3 * i + 1] = v.y; value_out[3 * i + 2] = v.z; }
    }
    return PPG_OK;
}

// Vertex::commit for n path vertices (sequential): leaf = the S-tree leaf of `o`.  verbatim != 0 runs the reference's OWN struct Vertex (reference backend only),
// otherwise the restated commit_vertex of ppg_cpu_tracer.h.  arrays: o, d, throughput, bsdf_val, radiance, rnd: 3n; the pdfs, weight: n; is_delta: n (u8)
int ppgo_tree_commit(ppgo_handle *h, size_t n, const float *o, const float *d, const float *throughput, const float *bsdf_val, const float *radiance,
                     const float *wo_pdf, const float *bsdf_pdf, const float *dtree_pdf, const float *weight, const uint8_t *is_delta, const float *rnd,
                     int sfilter, int dfilter, int loss, int verbatim) {
    BackendT &T = h->T();
#ifndef PPGO_BACKEND_REF
    if (verbatim) return PPG_ERR_UNSUPPORTED;
#endif
    for (size_t i = 0; i < n; ++i) {
        float voxel[3]; BackendT::Leaf *leaf = T.lookup(o + 3 * i, voxel);
#ifdef PPGO_BACKEND_REF
        if (verbatim) {
            T.commitVerbatim(leaf, o + 3 * i, voxel, d + 3 * i, throughput + 3 * i, bsdf_val + 3 * i, radiance + 3 * i, wo_pdf[i], bsdf_pdf[i], dtree_pdf[i], is_delta[i] != 0,
                             weight[i], sfilter, dfilter, loss, rnd + 3 * i);
            continue;
        }
#endif
        CommitRec v;
        v.o = f3(o[3 * i], o[3 * i + 1], o[3 * i + 2]); v.d = f3(d[3 * i], d[3 * i + 1], d[3 * i + 2]); v.voxel = f3(voxel[0], voxel[1], voxel[2]);
        v.throughput = f3(throughput[3 * i], throughput[3 * i + 1], throughput[3 * i + 2]); v.bsdfVal = f3(bsdf_val[3 * i], bsdf_val[3 * i + 1], bsdf_val[3 * i + 2]);
        v.radiance = f3(radiance[3 * i], radiance[3 * i + 1], radiance[3 * i + 2]);
        v.woPdf = wo_pdf[i]; v.bsdfPdf = bsdf_pdf[i]; v.dTreePdf = dtree_pdf[i]; v.isDelta = is_delta[i] != 0;
        commit_vertex(T, leaf, v, weight[i], sfilter, dfilter, loss, rnd + 3 * i);
    }
    return PPG_OK;
}

// dumpSDTree: the .sdt file the reference itself writes for the tree in its current state (reference backend only: its own BlobWriter / dump code)
int ppgo_tree_dump(ppgo_handle *h, const char *path, const float *cam_to_world) {
#ifdef PPGO_BACKEND_REF
    return h->T().dump(path, cam_to_world) ? PPG_OK : PPG_ERR_IO;
#else
    (void) h; (void) path; (void) cam_to_world; return PPG_ERR_UNSUPPORTED;
#endif
}

int ppgo_tree_refine(ppgo_handle *h, uint64_t threshold, int max_mb) { h->T().refine((size_t) threshold, max_mb); return PPG_OK; }
int ppgo_tree_reset(ppgo_handle *h, int max_depth, float threshold) { h->T().resetAll(max_depth, threshold, 1); return PPG_OK; }
int ppgo_tree_build(ppgo_handle *h) { h->T().buildAll(1); return PPG_OK; }

int ppgo_tree_record(ppgo_handle *h, size_t n, const float *o, const float *d, const float *radiance, const float *product,
                     const float *wo_pdf, const float *bsdf_pdf, const float *dtree_pdf, const float *weight, const uint8_t *is_delta,
                     const float *rnd, int sfilter, int dfilter, int loss) {
    BackendT &T = h->T();
    static const float zero3[3] = {0.5f, 0.5f, 0.5f};
    for (size_t i = 0; i < n; ++i) {
        float voxel[3]; BackendT::Leaf *leaf = T.lookup(o + 3 * i, voxel);
        T.record(leaf, o + 3 * i, voxel, d + 3 * i, radiance[i], product ? product[i] : 0.f, wo_pdf[i], bsdf_pdf ? bsdf_pdf[i] : 0.f,
                 dtree_pdf ? dtree_pdf[i] : 0.f, weight ? weight[i] : 1.0f, is_delta ? is_delta[i] != 0 : false, sfilter, dfilter, loss,
                 rnd ? rnd + 3 * i : zero3);
    }
    return PPG_OK;
}
int ppgo_tree_lookup(ppgo_handle *h, size_t n, const float *p, uint32_t *leaf_out, float *size_out) {
    BackendT &T = h->T();
    for (size_t i = 0; i < n; ++i) {
        float voxel[3]; BackendT::Leaf *leaf = T.lookup(p + 3 * i, voxel);
        if (leaf_out) leaf_out[i] = (uint32_t) T.leafIndex(leaf);
        if (size_out) { size_out[3 * i] = voxel[0]; size_out[3 * i + 1] = voxel[1]; size_out[3 * i + 2] = voxel[2]; }
    }
    return PPG_OK;
}
int ppgo_tree_pdf(ppgo_handle *h, size_t n, const uint32_t *leaf, const float *dir, float *pdf_out) {
    BackendT &T = h->T();
    for (size_t i = 0; i < n; ++i) pdf_out[i] = T.pdf(T.leafAt(leaf[i]), dir + 3 * i);
    return PPG_OK;
}
int ppgo_tree_sample(ppgo_handle *h, size_t n, const uint32_t *leaf, const float *rnd, size_t rnd_stride, float *dir_out) {
    BackendT &T = h->T();
    for (size_t i = 0; i < n; ++i) T.sampleReplay(T.leafAt(leaf[i]), rnd + rnd_stride * i, rnd_stride, dir_out + 3 * i);
    return PPG_OK;
}
int ppgo_tree_fraction(ppgo_handle *h, size_t n, const uint32_t *leaf, float *frac_out) {
    BackendT &T = h->T();
    for (size_t i = 0; i < n; ++i) frac_out[i] = T.bsdfSamplingFraction(T.leafAt(leaf[i]));
    return PPG_OK;
}
// seed the sampling-fraction optimiser of S-tree node `node` (6 floats: iter, m, v, variable, batchAcc, batchGrad)
int ppgo_tree_set_adam(ppgo_handle *h, uint32_t node, const float state6[6]) {
    BackendT &T = h->T();
    if (node >= T.numNodes() || !T.isLeaf(node)) return PPG_ERR_INVALID_ARGUMENT;
    T.setAdamState(node, state6);
    return PPG_OK;
}
int ppgo_tree_counts(ppgo_handle *h, uint64_t counts[4]) {
    BackendT &T = h->T();
    counts[0] = T.numNodes(); counts[1] = counts[2] = counts[3] = 0;
    for (size_t i = 0; i < T.numNodes(); ++i) if (T.isLeaf(i)) { counts[1]++; counts[2] += T.treeSize(i, false); counts[3] += T.treeSize(i, true); }
    return PPG_OK;
}
int ppgo_tree_export(ppgo_handle *h, int which, uint32_t *s_children, int32_t *s_axis, uint8_t *s_is_leaf,
                     uint64_t *tree_first, uint32_t *tree_count, float *tree_sum, float *tree_weight, int32_t *tree_depth,
                     float *sums, uint16_t *children, float *adam, float *aabb_min_max) {
    BackendT &T = h->T();
    const bool building = which != 0;
    uint64_t off = 0;
    for (size_t i = 0; i < T.numNodes(); ++i) {
        const bool leaf = T.isLeaf(i);
        if (s_children) { s_children[2 * i] = leaf ? 0 : T.child(i, 0); s_children[2 * i + 1] = leaf ? 0 : T.child(i, 1); }
        if (s_axis) s_axis[i] = T.axis(i);
        if (s_is_leaf) s_is_leaf[i] = leaf;
        if (adam) T.adamState(i, adam + 6 * i);
        if (!leaf) {
            if (tree_first) tree_first[i] = off;
            if (tree_count) tree_count[i] = 0;
            if (tree_sum) tree_sum[i] = 0;
            if (tree_weight) tree_weight[i] = 0;
            if (tree_depth) tree_depth[i] = 0;
            continue;
        }
        const size_t n = T.treeSize(i, building);
        if (tree_first) tree_first[i] = off;
        if (tree_count) tree_count[i] = (uint32_t) n;
        if (tree_sum) tree_sum[i] = T.treeSum(i, building);
        if (tree_weight) tree_weight[i] = T.treeWeight(i, building);
        if (tree_depth) tree_depth[i] = T.treeDepth(i, building);
        if (sums || children) {
            for (size_t k = 0; k < n; ++k) {
                float s[4]; uint16_t c[4]; T.treeNode(i, building, k, s, c);
                if (sums) std::memcpy(sums + 4 * (off + k), s, sizeof(s));
                if (children) std::memcpy(children + 4 * (off + k), c, sizeof(c));
            }
        }
        off += n;
    }
    if (aabb_min_max) T.aabb(aabb_min_max, aabb_min_max + 3);
    return PPG_OK;
}

}  // extern "C"
