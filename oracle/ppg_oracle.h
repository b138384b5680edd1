/* TEST INFRASTRUCTURE -- C API of the CPU oracle (libppg_oracle.so / _ref/libppg_oracle_ref.so).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it. */
#ifndef PPG_ORACLE_H
#define PPG_ORACLE_H
#include "../include/ppg.h"
#ifdef __cplusplus
extern "C" {
#endif
typedef struct ppgo_handle ppgo_handle;

/* 1 if this library embeds the reference's verbatim SD-tree code, 0 for the restatement */
int ppgo_is_reference_backend(void);

/* full integrator (scene may be NULL for a tree-only handle; then aabb_min/max give the S-tree box) */
ppgo_handle *ppgo_create(const ppg_params *p, const ppg_scene_desc *scene, const float *aabb_min, const float *aabb_max, int nthreads);
void ppgo_destroy(ppgo_handle *h);
int ppgo_render(ppgo_handle *h, float *rgb_out, ppg_stats *stats);
/* tile sharding + exchange callback with the product's semantics (ppg_set_shard / ppg_set_allreduce); the buffer is a HOST pointer here */
int ppgo_set_shard(ppgo_handle *h, int rank, int world_size);
int ppgo_set_allreduce(ppgo_handle *h, ppg_allreduce_fn cb, void *user);
/* capture per-sample radiance of the LAST pass rendered: li (W*H*spp*3), depth (W*H*spp) -- set before ppgo_render */
int ppgo_set_capture(ppgo_handle *h, float *li, int32_t *depth);
/* step-wise driving (tests): iteration k reset, n passes, build */
int ppgo_step_reset(ppgo_handle *h, int iter);
int ppgo_step_passes(ppgo_handle *h, int n_passes, int is_final, float *variance_out);
int ppgo_step_build(ppgo_handle *h, ppg_iteration_stats *st);
int ppgo_get_moment_images(ppgo_handle *h, float *sum_rgbw, float *sumsq_rgbw);

/* ---- BSDF level (no handle): n queries on one material; wi/wo local frames (3n floats), sample = 2n uniforms.
 * eval_out 3n (f * cos), pdf_out n, and for sampling: wo_out 3n, weight_out 3n (f * cos / pdf), pdf_out n, delta_out n (u8) */
int ppgo_bsdf_eval_pdf(const ppg_bsdf *b, size_t n, const float *wi, const float *wo, float *eval_out, float *pdf_out, const float *tables /* may be NULL */);
int ppgo_bsdf_sample(const ppg_bsdf *b, size_t n, const float *wi, const float *sample, float *wo_out, float *weight_out, float *pdf_out, uint8_t *delta_out, const float *tables);

/* ---- microfacet level: the restated MicrofacetDistribution (type: ppg_microfacet; isotropic, visible-normal sampling) -- m, v, wi: 3n local directions */
int ppgo_mf_eval(int type, float alpha, size_t n, const float *m, float *out);
int ppgo_mf_smith_g1(int type, float alpha, size_t n, const float *v, const float *m, float *out);
int ppgo_mf_pdf(int type, float alpha, size_t n, const float *wi, const float *m, float *out);
int ppgo_mf_sample(int type, float alpha, size_t n, const float *wi, const float *sample, float *m_out, float *pdf_out);
int ppgo_mf_erf(size_t n, const float *x, float *erf_out, float *erfinv_out);
/* restated helpers: fresnelDielectricExt / fresnelConductorExact (per channel; out 3n) / coordinateSystem / warp::squareToCosineHemisphere */
int ppgo_fresnel_dielectric_ext(size_t n, const float *cosThetaI, float eta, float *f_out, float *cos_t_out);
int ppgo_fresnel_conductor_exact(size_t n, const float *cosThetaI, const float eta[3], const float k[3], float *out);
int ppgo_coordinate_system(size_t n, const float *a, float *b_out, float *c_out);
int ppgo_square_to_cosine_hemisphere(size_t n, const float *sample, float *out);
/* TriAccel::load + rayIntersect for n (triangle, ray) pairs: k, the nine constants, hit flag, (t, u, v) */
int ppgo_triaccel(size_t n, const float *A, const float *B, const float *C, const float *o, const float *d, const float *mint, const float *maxt,
                  int *k_out, float *consts_out, unsigned char *hit_out, float *tuv_out);
/* discrete distribution over n_entries weights as the light sampling builds and samples it: normalised entries, sum, and for n samples index + reused sample */
int ppgo_discrete(size_t n_entries, const float *weights, size_t n, const float *sample, float *pdf_out, float *sum_out, unsigned *index_out, float *reused_out);
int ppgo_rough_transmittance(size_t n, const float *cosTheta, const float *values /* PPG_BSDF_TABLE_SIZE */, float *out);

/* ---- emitter level (handle with a scene): Scene::sampleAttenuatedEmitterDirect at n reference points -- ref, ref_n 3n (ref_n 0 = two-sided),
 * sample 2n; d_out 3n, value_out 3n (radiance * transmittance / pdf), pdf_out n (0: nothing), dist_out n -- and the environment emitter's
 * light-sampling density (Scene::pdfEmitterDirect) / radiance for n world directions */
int ppgo_emitter_sample_direct(ppgo_handle *h, size_t n, const float *ref, const float *ref_n, const float *sample, int max_interactions,
                               float *d_out, float *value_out, float *pdf_out, float *dist_out);
int ppgo_env_pdf(ppgo_handle *h, size_t n, const float *d, float *pdf_out, float *value_out /* 3n or NULL */);
/* bitmap texture `tex` of the handle's scene at n uv pairs: bilinear value (3n) and the luminance gradient the bump map uses (2n) */
int ppgo_texture_eval(ppgo_handle *h, uint32_t tex, size_t n, const float *uv, float *rgb_out, float *grad_out);

/* ---- SD-tree level operations (work on the handle's tree) */
/* Vertex::commit (GP:1730-1768) for n vertices; verbatim != 0: the reference's own struct Vertex (reference backend only), else the restated commit_vertex */
int ppgo_tree_commit(ppgo_handle *h, size_t n, const float *o, const float *d, const float *throughput, const float *bsdf_val, const float *radiance,
                     const float *wo_pdf, const float *bsdf_pdf, const float *dtree_pdf, const float *weight, const uint8_t *is_delta, const float *rnd,
                     int sfilter, int dfilter, int loss, int verbatim);
/* dumpSDTree (GP:1191-1208) through the reference's own writer code; PPG_ERR_UNSUPPORTED on the restated backend */
int ppgo_tree_dump(ppgo_handle *h, const char *path, const float *cam_to_world /* 16, row major */);
int ppgo_tree_refine(ppgo_handle *h, uint64_t threshold, int max_mb);
int ppgo_tree_reset(ppgo_handle *h, int max_depth, float threshold);
int ppgo_tree_build(ppgo_handle *h);
/* Vertex::commit's record step for n records (sequential, deterministic order).
 * arrays: o,voxel,d: 3n; radiance,product,wo_pdf,bsdf_pdf,dtree_pdf,weight: n; is_delta: n (u8); rnd: 3n */
int ppgo_tree_record(ppgo_handle *h, size_t n, const float *o, const float *d, const float *radiance, const float *product,
                     const float *wo_pdf, const float *bsdf_pdf, const float *dtree_pdf, const float *weight, const uint8_t *is_delta,
                     const float *rnd, int sfilter, int dfilter, int loss);
/* lookup: leaf node index + voxel size */
int ppgo_tree_lookup(ppgo_handle *h, size_t n, const float *p, uint32_t *leaf_out, float *size_out);
int ppgo_tree_pdf(ppgo_handle *h, size_t n, const uint32_t *leaf, const float *dir, float *pdf_out);
int ppgo_tree_sample(ppgo_handle *h, size_t n, const uint32_t *leaf, const float *rnd, size_t rnd_stride, float *dir_out);
int ppgo_tree_fraction(ppgo_handle *h, size_t n, const uint32_t *leaf, float *frac_out);
/* counts[0]=S-tree nodes, [1]=leaves, [2]=total sampling quadtree nodes, [3]=total building quadtree nodes */
/* Seed the sampling-fraction optimiser (AdamOptimizer::State) of leaf `node`: iter, m, v, variable, batchAcc, batchGrad. */
int ppgo_tree_set_adam(ppgo_handle *h, uint32_t node, const float state6[6]);
int ppgo_tree_counts(ppgo_handle *h, uint64_t counts[4]);
/* export: s_children 2*N u32 (0,0 for leaves), s_axis N i32, s_is_leaf N u8;
 * per S-tree node i (valid for leaves): tree_first[which][i], tree_count, tree_sum, tree_weight, tree_depth;
 * quadtree nodes concatenated in S-tree node order: sums 4 floats, children 4 u16. which: 0 sampling, 1 building.
 * adam: 6 floats per S-tree node (iter, m, v, variable, batchAcc, batchGrad). Any pointer may be NULL. */
int ppgo_tree_export(ppgo_handle *h, int which, uint32_t *s_children, int32_t *s_axis, uint8_t *s_is_leaf,
                     uint64_t *tree_first, uint32_t *tree_count, float *tree_sum, float *tree_weight, int32_t *tree_depth,
                     float *sums, uint16_t *children, float *adam, float *aabb_min_max);
#ifdef __cplusplus
}
#endif
#endif
