// TEST INFRASTRUCTURE -- adapter: restated SD-tree (sdtree_port.h) behind the tracer's backend interface.
#pragma once
#include "sdtree_port.h"
#include "ppg_cpu_tracer.h"
#include "backend_common.h"

namespace ppgo {

struct PortRng {   // the Sampler interface the D-tree sampler needs (next2D draws x first)
    Pcg32 &r;
    float next1D() { return r.next1D(); }
    V2 next2D() { V2 p; p.x = r.next1D(); p.y = r.next1D(); return p; }
};
struct ReplayRng {  // replays a caller-provided list of uniforms (FakeSampler of test_chisquare.cpp:58-86)
    const float *v; size_t n, i = 0;
    float next1D() { return i < n ? v[i++] : 0.5f; }
    V2 next2D() { V2 p; p.x = next1D(); p.y = next1D(); return p; }
};

struct PortBackend {
    typedef SNode Leaf;
    STree t;
    PortBackend(const float mn[3], const float mx[3]) : t(V3{mn[0], mn[1], mn[2]}, V3{mx[0], mx[1], mx[2]}) {}

    Leaf *lookup(const float *p, float *voxel) {
        V3 size; const uint32_t n = t.lookup(V3{p[0], p[1], p[2]}, &size);
        voxel[0] = size.x; voxel[1] = size.y; voxel[2] = size.z;
        return &t.nodes[n];
    }
    float bsdfSamplingFraction(Leaf *l) const { return l->dTree.bsdfSamplingFraction(); }
    void sample(Leaf *l, Pcg32 &rng, float *dir) const { PortRng r{rng}; V3 d = l->dTree.sample(r); dir[0] = d.x; dir[1] = d.y; dir[2] = d.z; }
    void sampleReplay(Leaf *l, const float *rnd, size_t n, float *dir) const { ReplayRng r{rnd, n}; V3 d = l->dTree.sample(r); dir[0] = d.x; dir[1] = d.y; dir[2] = d.z; }
    float pdf(Leaf *l, const float *d) const { return l->dTree.pdf(V3{d[0], d[1], d[2]}); }

    // the spatial-filter switch of Vertex::commit, GP:1742-1767
    void record(Leaf *leaf, const float *o, const float *voxel, const float *d, float radiance, float product, float woPdf, float bsdfPdf,
                float dTreePdf, float weight, bool isDelta, int sfilter, int dfilter, int loss, const float *rnd) {
        DTreeRecord rec{V3{d[0], d[1], d[2]}, radiance, product, woPdf, bsdfPdf, dTreePdf, weight, isDelta};
        if (sfilter == PPG_SFILTER_NEAREST) leaf->dTree.record(rec, dfilter, loss);
        else if (sfilter == PPG_SFILTER_STOCHASTIC) {
            V3 off{voxel[0], voxel[1], voxel[2]};
            off.x *= rnd[0] - 0.5f; off.y *= rnd[1] - 0.5f; off.z *= rnd[2] - 0.5f;
            const V3 origin = t.clip(V3{o[0] + off.x, o[1] + off.y, o[2] + off.z});
            t.nodes[t.lookup(origin)].dTree.record(rec, dfilter, loss);
        } else t.recordBox(V3{o[0], o[1], o[2]}, V3{voxel[0], voxel[1], voxel[2]}, rec, dfilter, loss);
    }

    void refine(size_t thr, int maxMB) { t.refine(thr, maxMB); }
    void resetAll(int maxDepth, float thr, int nthreads) {   // GP:1112, 924-933
        const int n = (int) t.nodes.size();
#pragma omp parallel for num_threads(nthreads)
        for (int i = 0; i < n; ++i) if (t.nodes[i].isLeaf) t.nodes[i].dTree.reset(maxDepth, thr);
    }
    void buildAll(int nthreads) {                            // GP:1119
        const int n = (int) t.nodes.size();
#pragma omp parallel for num_threads(nthreads)
        for (int i = 0; i < n; ++i) if (t.nodes[i].isLeaf) t.nodes[i].dTree.build();
    }

    // ---- uniform accessors used by statistics/export (shared with the verbatim backend)
    Leaf *leafAt(size_t i) { return &t.nodes[i]; }
    size_t leafIndex(Leaf *l) const { return (size_t) (l - &t.nodes[0]); }
    size_t numNodes() const { return t.nodes.size(); }
    bool isLeaf(size_t i) const { return t.nodes[i].isLeaf; }
    int axis(size_t i) const { return t.nodes[i].axis; }
    uint32_t child(size_t i, int c) const { return t.nodes[i].children[c]; }
    struct TreeView { const void *nodes; size_t n; float sum, weight; int maxDepth; };
    size_t treeSize(size_t i, bool building) const { const DTree &d = building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling; return d.nodes.size(); }
    float treeSum(size_t i, bool building) const { return (building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling).sum; }
    float treeWeight(size_t i, bool building) const { return (building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling).weight; }
    int treeDepth(size_t i, bool building) const { return (building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling).maxDepth; }
    float treeMean(size_t i, bool building) const { return (building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling).mean(); }
    void treeNode(size_t i, bool building, size_t k, float *sums, uint16_t *children) const {
        const QNode &q = (building ? t.nodes[i].dTree.building : t.nodes[i].dTree.sampling).nodes[k];
        for (int j = 0; j < 4; ++j) { sums[j] = q.sum[j]; children[j] = q.child[j]; }
    }
    void adamState(size_t i, float *out6) const {
        const Adam &a = t.nodes[i].dTree.opt;
        out6[0] = (float) a.iter; out6[1] = a.m1; out6[2] = a.m2; out6[3] = a.variable; out6[4] = a.batchAcc; out6[5] = a.batchGrad;
    }
    void setAdamState(size_t i, const float *in6) {
        Adam &a = t.nodes[i].dTree.opt;
        a.iter = (int) in6[0]; a.m1 = in6[1]; a.m2 = in6[2]; a.variable = in6[3]; a.batchAcc = in6[4]; a.batchGrad = in6[5];
    }
    void aabb(float *mn, float *mx) const { mn[0] = t.amin.x; mn[1] = t.amin.y; mn[2] = t.amin.z; mx[0] = t.amax.x; mx[1] = t.amax.y; mx[2] = t.amax.z; }

    // flat [building sums (4 per quadtree node) | building weight] per leaf in node order (the exchange buffer of SURVEY 8e)
    size_t packSize() const { size_t n = 0; for (const auto &nd : t.nodes) if (nd.isLeaf) n += 4 * nd.dTree.building.nodes.size() + 1; return n; }
    void packBuilding(float *buf, bool unpack) {
        size_t o = 0;
        for (auto &nd : t.nodes) {
            if (!nd.isLeaf) continue;
            for (auto &q : nd.dTree.building.nodes) for (int j = 0; j < 4; ++j) { if (unpack) q.sum[j] = buf[o]; else buf[o] = q.sum[j]; ++o; }
            if (unpack) nd.dTree.building.weight = buf[o]; else buf[o] = nd.dTree.building.weight;
            ++o;
        }
    }
    void statistics(ppg_iteration_stats &st) const;
};

inline void PortBackend::statistics(ppg_iteration_stats &st) const { backend_statistics(*this, st); }

}  // namespace ppgo
