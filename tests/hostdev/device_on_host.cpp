// TEST INFRASTRUCTURE -- C entry points over the product's CUDA device functions compiled for the host (see cuda_host_shim.h); same shape as oracle/microfacet_ref/wrapper.h.
#include "cuda_host_shim.h"
#include "../../practical-path-guiding_b200/csrc/ppg_kernels.cuh"      // (includes ppg_device.cuh; the __global__ functions run here as plain loops of one thread)
#include "../../include/ppg.h"
#include <cstddef>
#include <vector>
using namespace ppg;
static inline float3 v3(const float *p, size_t i) { return make_float3(p[3 * i], p[3 * i + 1], p[3 * i + 2]); }
extern "C" {
int dev_mf_eval(int type, float alpha, size_t n, const float *m, float *out) { for (size_t i = 0; i < n; ++i) out[i] = mf_eval(type, alpha, v3(m, i)); return 0; }
int dev_mf_smith_g1(int type, float alpha, size_t n, const float *v, const float *m, float *out) { for (size_t i = 0; i < n; ++i) out[i] = mf_smithG1(type, alpha, v3(v, i), v3(m, i)); return 0; }
int dev_mf_pdf(int type, float alpha, size_t n, const float *wi, const float *m, float *out) { for (size_t i = 0; i < n; ++i) out[i] = mf_pdfVisible(type, alpha, v3(wi, i), v3(m, i)); return 0; }
int dev_mf_sample(int type, float alpha, size_t n, const float *wi, const float *sample, float *m_out, float *pdf_out) {
    for (size_t i = 0; i < n; ++i) {
        const float3 m = mf_sampleVisible(type, alpha, v3(wi, i), sample[2 * i], sample[2 * i + 1]);
        m_out[3 * i] = m.x; m_out[3 * i + 1] = m.y; m_out[3 * i + 2] = m.z; pdf_out[i] = mf_pdfVisible(type, alpha, v3(wi, i), m);
    }
    return 0;
}
int dev_erf(size_t n, const float *x, float *erf_out, float *erfinv_out) { for (size_t i = 0; i < n; ++i) { erf_out[i] = mts_erf(x[i]); erfinv_out[i] = mts_erfinv(x[i]); } return 0; }
int dev_fresnel_dielectric_ext(size_t n, const float *c, float eta, float *f_out, float *ct_out) { for (size_t i = 0; i < n; ++i) { float ct = 0; f_out[i] = fresnel_dielectric_ext(c[i], ct, eta); ct_out[i] = ct; } return 0; }
int dev_fresnel_conductor_exact(size_t n, const float *c, const float eta[3], const float k[3], float *out) {
    for (size_t i = 0; i < n; ++i) for (int ch = 0; ch < 3; ++ch) out[3 * i + ch] = fresnel_conductor_exact(c[i], eta[ch], k[ch]);
    return 0;
}
int dev_coordinate_system(size_t n, const float *a, float *b_out, float *c_out) {
    for (size_t i = 0; i < n; ++i) { float3 b, c; coordinate_system(v3(a, i), b, c); b_out[3 * i] = b.x; b_out[3 * i + 1] = b.y; b_out[3 * i + 2] = b.z; c_out[3 * i] = c.x; c_out[3 * i + 1] = c.y; c_out[3 * i + 2] = c.z; }
    return 0;
}
int dev_square_to_cosine_hemisphere(size_t n, const float *s, float *out) { for (size_t i = 0; i < n; ++i) { const float3 v = square_to_cosine_hemisphere(s[2 * i], s[2 * i + 1]); out[3 * i] = v.x; out[3 * i + 1] = v.y; out[3 * i + 2] = v.z; } return 0; }
// the kernels' triangle test on the accel rows ppg_set_scene packs: {n_u, n_v, n_d, bits(k)}, {a_u, a_v, b_nu, b_nv}, {c_nu, c_nv, -, -}
int dev_tri_intersect(size_t n, const int *k, const float *consts /* 9n, TriAccel order */, const float *o, const float *d, const float *mint, const float *maxt, unsigned char *hit_out, float *tuv_out) {
    for (size_t i = 0; i < n; ++i) {
        const float *c = consts + 9 * i;
        const float4 A = make_float4(c[0], c[1], c[2], __int_as_float(k[i])), B = make_float4(c[3], c[4], c[5], c[6]), C = make_float4(c[7], c[8], 0.f, 0.f);
        float u = 0, v = 0, t = 0;
        hit_out[i] = tri_intersect(A, B, C, v3(o, i), v3(d, i), mint[i], maxt[i], u, v, t) ? 1 : 0;
        tuv_out[3 * i] = t; tuv_out[3 * i + 1] = u; tuv_out[3 * i + 2] = v;
    }
    return 0;
}
// ---- whole BSDF models: the device Bsdf record as load_bsdf() rebuilds it from the 28 floats ppg_set_scene packs per material (ppg_host.cu: "bsdf" table)
static Bsdf make_bsdf(const ppg_bsdf &m, const float *tables) {
    Bsdf b; b.refl = make_float3(m.reflectance[0], m.reflectance[1], m.reflectance[2]);
    b.type = (uint32_t) m.type; b.flags = m.flags & 0xffffffu;
    if (m.type == PPG_BSDF_NULL_BLACK) { b.refl = make_float3(0, 0, 0); b.type = PPG_BSDF_T_DIFFUSE; }
    b.trans = b.etaRgb = b.k = b.specRefl = make_float3(0, 0, 0); b.eta = b.invEta = 1.f; b.alpha = 0.1f; b.distr = 1; b.fdrInt = b.ssw = 0.f; b.lut = nullptr;
    b.opacity = make_float3(1, 1, 1); b.maskProb = 1.f; b.reflTex = b.bumpTex = 0u;
    if (b.flags & PPG_BSDF_MASK) { b.opacity = make_float3(m.opacity[0], m.opacity[1], m.opacity[2]); b.maskProb = m.opacity[0] * 0.212671f + m.opacity[1] * 0.715160f + m.opacity[2] * 0.072169f; }
    if (b.type != PPG_BSDF_T_DIFFUSE) {
        b.trans = make_float3(m.specular_transmittance[0], m.specular_transmittance[1], m.specular_transmittance[2]); b.eta = m.eta[0];
        b.etaRgb = make_float3(m.eta[0], m.eta[1], m.eta[2]); b.invEta = m.eta[0] != 0.f ? 1.0f / m.eta[0] : 0.f; b.k = make_float3(m.k[0], m.k[1], m.k[2]);
        b.alpha = std::max(m.alpha, 1e-4f); b.distr = m.distribution == PPG_MICROFACET_BECKMANN ? 0 : 1;
        if (b.type == PPG_BSDF_T_ROUGHPLASTIC || b.type == PPG_BSDF_T_PLASTIC) {
            b.specRefl = make_float3(m.specular_reflectance[0], m.specular_reflectance[1], m.specular_reflectance[2]); b.fdrInt = m.fdr_int; b.ssw = m.specular_sampling_weight;
            b.lut = tables ? tables + (size_t) std::max(m.table, 0) * PPG_BSDF_LUT : nullptr;
        }
    }
    return b;
}
int dev_bsdf_eval_pdf(const ppg_bsdf *m, size_t n, const float *wi, const float *wo, float *eval_out, float *pdf_out, const float *tables) {
    const Bsdf b = make_bsdf(*m, tables);
    for (size_t i = 0; i < n; ++i) { const float3 e = bsdf_eval(b, v3(wi, i), v3(wo, i)); eval_out[3 * i] = e.x; eval_out[3 * i + 1] = e.y; eval_out[3 * i + 2] = e.z; pdf_out[i] = bsdf_pdf(b, v3(wi, i), v3(wo, i)); }
    return 0;
}
int dev_bsdf_sample(const ppg_bsdf *m, size_t n, const float *wi, const float *sample, float *wo_out, float *weight_out, float *pdf_out, unsigned char *delta_out, const float *tables) {
    const Bsdf b = make_bsdf(*m, tables);
    for (size_t i = 0; i < n; ++i) {
        float3 wo = make_float3(0, 0, 0); float eta = 1.f, pdf = 0.f; bool delta = false, isNull = false;
        Pcg32 extra; extra.seed(splitmix64(i), i);                      // like ppgo_bsdf_sample: the model's own draws from the path sampler (roughdielectric)
        const float3 w = bsdf_sample(b, v3(wi, i), sample[2 * i], sample[2 * i + 1], wo, eta, delta, pdf, extra, isNull);
        wo_out[3 * i] = wo.x; wo_out[3 * i + 1] = wo.y; wo_out[3 * i + 2] = wo.z; weight_out[3 * i] = w.x; weight_out[3 * i + 1] = w.y; weight_out[3 * i + 2] = w.z;
        pdf_out[i] = pdf; if (delta_out) delta_out[i] = delta ? 1 : 0;
    }
    return 0;
}
// bitmap textures: one ppg_texture packed the way ppg_set_scene packs it (uint2 {r | g << 16, b} per texel, two float4 of meta), then tex_eval / tex_gradient_lum
int dev_texture_eval(const ppg_texture *t, const uint16_t *texels /* the whole texel array of the scene */, size_t n, const float *uv, float *rgb_out, float *grad_out) {
    const size_t nTexels = (size_t) t->width * t->height;
    std::vector<uint2> tex(nTexels);
    const uint16_t *src = texels + t->first_texel;
    for (size_t i = 0; i < nTexels; ++i) {
        const uint16_t r = src[i * t->channels], g = t->channels == 3 ? src[i * t->channels + 1] : r, b = t->channels == 3 ? src[i * t->channels + 2] : r;
        tex[i] = make_uint2((uint32_t) r | ((uint32_t) g << 16), (uint32_t) b);
    }
    float4 meta[2];
    const uint32_t wr = t->wrap_u | (t->wrap_v << 8);
    meta[0] = make_float4(__uint_as_float(t->width), __uint_as_float(t->height), __uint_as_float(wr), __uint_as_float(0u));
    meta[1] = make_float4(t->uv_scale[0], t->uv_scale[1], t->uv_offset[0], t->uv_offset[1]);
    SceneView sc; memset(&sc, 0, sizeof(sc)); sc.texMeta = meta; sc.texels = tex.data(); sc.nTextures = 1;
    for (size_t i = 0; i < n; ++i) {
        const float2 q = make_float2(uv[2 * i], uv[2 * i + 1]);
        const float3 c = tex_eval(sc, 0u, q); const float2 g = tex_gradient_lum(sc, 0u, q);
        rgb_out[3 * i] = c.x; rgb_out[3 * i + 1] = c.y; rgb_out[3 * i + 2] = c.z; grad_out[2 * i] = g.x; grad_out[2 * i + 1] = g.y;
    }
    return 0;
}
// cdf_sample + the sample reuse of the device's sample_emitter_direct, on a normalised cdf (n_entries + 1 values) the host built
int dev_discrete(size_t n_entries, const float *cdf, size_t n, const float *sample, unsigned *index_out, float *reused_out) {
    for (size_t i = 0; i < n; ++i) {
        const uint32_t k = cdf_sample(cdf, (uint32_t) n_entries + 1u, sample[i]);
        const float c0 = cdf[k], c1 = cdf[k + 1];
        index_out[i] = k; reused_out[i] = (sample[i] - c0) / (c1 - c0);
    }
    return 0;
}
// ---- SD-tree: S-tree descent through the prefix table stree_table_kernel builds, D-tree pdf / sample on a sampling pool laid out like the device's (SampNode)
int dev_stree_lookup(const uint32_t *node_children /* 2 per node */, size_t n_nodes, const float aabb_min[3], const float extent[3], const float *points, size_t n, uint32_t *leaf_out, float *size_out) {
    std::vector<uint2> sn(n_nodes);
    for (size_t i = 0; i < n_nodes; ++i) sn[i] = make_uint2(node_children[2 * i], node_children[2 * i + 1]);
    std::vector<uint32_t> table((size_t) 1 << (3 * PPG_STREE_TABLE_BITS));
    stree_table_kernel(sn.data(), table.data());
    const float3 mn = make_float3(aabb_min[0], aabb_min[1], aabb_min[2]), ex = make_float3(extent[0], extent[1], extent[2]);
    for (size_t i = 0; i < n; ++i) {
        int lv = 0; leaf_out[i] = stree_lookup(sn.data(), table.data(), mn, ex, v3(points, i), lv);
        const float3 v = voxel_size(ex, lv); size_out[3 * i] = v.x; size_out[3 * i + 1] = v.y; size_out[3 * i + 2] = v.z;
    }
    return 0;
}
struct ReplayRng { const float *v; uint32_t n, i; float next1D() { return i < n ? v[i++] : 0.5f; } };
int dev_dtree(const float *sums, const uint16_t *children, size_t n_nodes, const uint32_t *tree_first, const float *tree_sum, const float *tree_weight,
              const uint32_t *query_tree, const float *query_dir, const float *rnd, size_t rnd_stride, size_t n, float *pdf_out, float *dir_out) {
    std::vector<SampNode> pool(n_nodes);
    for (size_t i = 0; i < n_nodes; ++i) {
        pool[i].sums = make_float4(sums[4 * i], sums[4 * i + 1], sums[4 * i + 2], sums[4 * i + 3]);
        pool[i].children = make_uint2((uint32_t) children[4 * i] | ((uint32_t) children[4 * i + 1] << 16), (uint32_t) children[4 * i + 2] | ((uint32_t) children[4 * i + 3] << 16));
        pool[i].pad = make_uint2(0u, 0u);
    }
    for (size_t i = 0; i < n; ++i) {
        const uint32_t t = query_tree[i];
        float mean = 0.f; if (tree_weight[t] != 0.f) mean = (1.f / (PPG_PI * 4.f * tree_weight[t])) * tree_sum[t];       // DTree::mean, GP:386-394
        pdf_out[i] = dtree_pdf(pool.data() + tree_first[t], mean > 0.f, dir_to_canonical(v3(query_dir, i)));
        ReplayRng r{rnd + rnd_stride * i, (uint32_t) rnd_stride, 0u};
        const float3 d = canonical_to_dir(dtree_sample(pool.data() + tree_first[t], mean > 0.f, r));
        dir_out[3 * i] = d.x; dir_out[3 * i + 1] = d.y; dir_out[3 * i + 2] = d.z;
    }
    return 0;
}
// the sampling-fraction replay of adam_seq_kernel (fraction_begin / fraction_k / fraction_link / fraction_end), walked sequentially over records in array
// order: each leaf replays its records in the order they appear.  states 6 floats per leaf (in/out); rec_a 4 floats {bits(leaf), product, woPdf, bsdfPdf},
// rec_b 2 floats {dTreePdf, weight} per record, as record_into_leaf appends them
int dev_fraction_replay(float *states, size_t n_leaves, const float *rec_a, const float *rec_b, size_t n, int loss) {
    const bool var = loss == PPG_LOSS_VAR;
    std::vector<FractionChain> chain(n_leaves); std::vector<char> live(n_leaves, 0);
    for (size_t i = 0; i < n; ++i) {
        const uint32_t leaf = __float_as_uint(rec_a[4 * i]);
        if (leaf >= n_leaves) return 1;
        if (!live[leaf]) { chain[leaf] = fraction_begin(states + 6 * (size_t) leaf); live[leaf] = 1; }
        const float product = rec_a[4 * i + 1], woPdf = rec_a[4 * i + 2], bsdfPdf = rec_a[4 * i + 3], dTreePdf = rec_b[2 * i], weight = rec_b[2 * i + 1];
        fraction_link(chain[leaf], fraction_k(product, woPdf, bsdfPdf, dTreePdf, var), bsdfPdf, dTreePdf, weight, var);
    }
    for (size_t l = 0; l < n_leaves; ++l) if (live[l]) fraction_end(chain[l], states + 6 * l);
    return 0;
}
int dev_rough_transmittance(size_t n, const float *c, const float *values, float *out) { for (size_t i = 0; i < n; ++i) out[i] = rough_transmittance(values, c[i]); return 0; }
}
