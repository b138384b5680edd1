// TEST INFRASTRUCTURE -- adapter: the reference's OWN SD-tree classes (compiled verbatim
// from /root/reference by oracle/Makefile; the extract is piped into the compiler and
// this header is appended after it) behind the tracer's backend interface.
// Expects: shim.h, then guided_path.cpp lines 25-1008 + closing '}', to precede it
// in the translation unit, with private members opened (-Dprivate=public after the std headers).
#pragma once
#include "../ppg_cpu_tracer.h"
#include "../backend_common.h"   // backend_statistics<>

namespace ppgo {

struct RefSampler : public mitsuba::Sampler {
    Pcg32 *r = nullptr; const float *v = nullptr; size_t n = 0, i = 0;
    mitsuba::Float next1D() override { if (r) return r->next1D(); return i < n ? v[i++] : 0.5f; }
    mitsuba::Point2 next2D() override { mitsuba::Point2 p; p.x = next1D(); p.y = next1D(); return p; }
};

struct RefBackend {
    typedef mitsuba::DTreeWrapper Leaf;
    mitsuba::STree *t;
    static mitsuba::AABB mk(const float mn[3], const float mx[3]) { mitsuba::AABB a; a.min = mitsuba::Point(mn[0], mn[1], mn[2]); a.max = mitsuba::Point(mx[0], mx[1], mx[2]); return a; }
    RefBackend(const float mn[3], const float mx[3]) : t(new mitsuba::STree(mk(mn, mx))) {}
    ~RefBackend() { delete t; }
    RefBackend(const RefBackend &) = delete;

    Leaf *lookup(const float *p, float *voxel) {
        mitsuba::Vector size; Leaf *l = t->dTreeWrapper(mitsuba::Point(p[0], p[1], p[2]), size);
        voxel[0] = size.x; voxel[1] = size.y; voxel[2] = size.z; return l;
    }
    float bsdfSamplingFraction(Leaf *l) const { return l->bsdfSamplingFraction(); }
    void sample(Leaf *l, Pcg32 &rng, float *dir) const { RefSampler s; s.r = &rng; mitsuba::Vector d = l->sample(&s); dir[0] = d.x; dir[1] = d.y; dir[2] = d.z; }
    void sampleReplay(Leaf *l, const float *rnd, size_t n, float *dir) const { RefSampler s; s.v = rnd; s.n = n; mitsuba::Vector d = l->sample(&s); dir[0] = d.x; dir[1] = d.y; dir[2] = d.z; }
    float pdf(Leaf *l, const float *d) const { return l->pdf(mitsuba::Vector(d[0], d[1], d[2])); }

    // the spatial-filter switch of Vertex::commit (GP:1742-1767 lies outside the verbatim extract, so it is restated here)
    void record(Leaf *leaf, const float *o, const float *voxel, const float *d, float radiance, float product, float woPdf, float bsdfPdf,
                float dTreePdf, float weight, bool isDelta, int sfilter, int dfilter, int loss, const float *rnd) {
        typedef mitsuba::Vector Vector; typedef mitsuba::Point Point;
        typedef mitsuba::EDirectionalFilter EDF; typedef mitsuba::EBsdfSamplingFractionLoss ELS;
        mitsuba::DTreeRecord rec{Vector(d[0], d[1], d[2]), radiance, product, woPdf, bsdfPdf, dTreePdf, weight, isDelta};
        const EDF df = dfilter == 0 ? EDF::ENearest : EDF::EBox;
        const ELS ls = loss == 0 ? ELS::ENone : (loss == 1 ? ELS::EKL : ELS::EVariance);
        if (sfilter == PPG_SFILTER_NEAREST) leaf->record(rec, df, ls);
        else if (sfilter == PPG_SFILTER_STOCHASTIC) {
            Vector offset(voxel[0], voxel[1], voxel[2]);
            offset.x *= rnd[0] - 0.5f; offset.y *= rnd[1] - 0.5f; offset.z *= rnd[2] - 0.5f;
            Point origin = t->aabb().clip(Point(o[0], o[1], o[2]) + offset);
            mitsuba::DTreeWrapper *splat = t->dTreeWrapper(origin);
            if (splat) splat->record(rec, df, ls);
        } else t->record(Point(o[0], o[1], o[2]), Vector(voxel[0], voxel[1], voxel[2]), rec, df, ls);
    }

    // Vertex::commit (GP:1730-1768) -- the reference's OWN code (struct Vertex is piped in verbatim after the SD-tree extract): validity test, radiance / throughput
    // per channel above Epsilon, product with the BSDF value, the record, and the spatial-filter switch with its three jitter numbers
    void commitVerbatim(Leaf *leaf, const float *o, const float *voxel, const float *d, const float *throughput, const float *bsdfVal, const float *radiance,
                        float woPdf, float bsdfPdf, float dTreePdf, bool isDelta, float weight, int sfilter, int dfilter, int loss, const float *rnd) {
        typedef mitsuba::EDirectionalFilter EDF; typedef mitsuba::EBsdfSamplingFractionLoss ELS; typedef mitsuba::ESpatialFilter ESF;
        mitsuba::Vertex v;
        v.dTree = leaf; v.dTreeVoxelSize = mitsuba::Vector(voxel[0], voxel[1], voxel[2]);
        v.ray = mitsuba::Ray(mitsuba::Point(o[0], o[1], o[2]), mitsuba::Vector(d[0], d[1], d[2]), 0);
        for (int c = 0; c < 3; ++c) { v.throughput[c] = throughput[c]; v.bsdfVal[c] = bsdfVal[c]; v.radiance[c] = radiance[c]; }
        v.woPdf = woPdf; v.bsdfPdf = bsdfPdf; v.dTreePdf = dTreePdf; v.isDelta = isDelta;
        RefSampler s; s.v = rnd; s.n = 3;
        v.commit(*t, weight, sfilter == PPG_SFILTER_NEAREST ? ESF::ENearest : (sfilter == PPG_SFILTER_STOCHASTIC ? ESF::EStochasticBox : ESF::EBox),
                 dfilter == 0 ? EDF::ENearest : EDF::EBox, loss == 0 ? ELS::ENone : (loss == 1 ? ELS::EKL : ELS::EVariance), &s);
    }
    // dumpSDTree (GP:1191-1208) with the reference's own writers: BlobWriter (GP:35-57), STree::dump (GP:945-951), DTreeWrapper / DTree::dump (GP:699-711)
    bool dump(const char *path, const float cam[16]) const {
        { mitsuba::BlobWriter blob(path); for (int i = 0; i < 16; ++i) blob << (float) cam[i]; t->dump(blob); }
        std::ifstream check(path, std::ios::binary); return check.good();
    }
    void refine(size_t thr, int maxMB) { t->refine(thr, maxMB); }
    void resetAll(int maxDepth, float thr, int nthreads) { omp_set_num_threads(nthreads); t->forEachDTreeWrapperParallel([=](mitsuba::DTreeWrapper *d) { d->reset(maxDepth, thr); }); }
    void buildAll(int nthreads) { omp_set_num_threads(nthreads); t->forEachDTreeWrapperParallel([](mitsuba::DTreeWrapper *d) { d->build(); }); }

    Leaf *leafAt(size_t i) { return &t->m_nodes[i].dTree; }
    size_t leafIndex(Leaf *l) const { for (size_t i = 0; i < t->m_nodes.size(); ++i) if (&t->m_nodes[i].dTree == l) return i; return (size_t) -1; }
    size_t numNodes() const { return t->m_nodes.size(); }
    bool isLeaf(size_t i) const { return t->m_nodes[i].isLeaf; }
    int axis(size_t i) const { return t->m_nodes[i].axis; }
    uint32_t child(size_t i, int c) const { return t->m_nodes[i].children[c]; }
    const mitsuba::DTree &dt(size_t i, bool building) const { return building ? t->m_nodes[i].dTree.building : t->m_nodes[i].dTree.sampling; }
    size_t treeSize(size_t i, bool b) const { return dt(i, b).numNodes(); }
    float treeSum(size_t i, bool b) const { return dt(i, b).m_atomic.sum; }
    float treeWeight(size_t i, bool b) const { return dt(i, b).statisticalWeight(); }
    int treeDepth(size_t i, bool b) const { return dt(i, b).depth(); }
    float treeMean(size_t i, bool b) const { return dt(i, b).mean(); }
    void treeNode(size_t i, bool b, size_t k, float *sums, uint16_t *children) const {
        const mitsuba::QuadTreeNode &q = dt(i, b).node(k);
        for (int j = 0; j < 4; ++j) { sums[j] = q.sum(j); children[j] = q.child(j); }
    }
    void adamState(size_t i, float *out6) const {
        const auto &s = t->m_nodes[i].dTree.bsdfSamplingFractionOptimizer.m_state;
        out6[0] = (float) s.iter; out6[1] = s.firstMoment; out6[2] = s.secondMoment; out6[3] = s.variable; out6[4] = s.batchAccumulation; out6[5] = s.batchGradient;
    }
    void setAdamState(size_t i, const float *in6) {
        auto &s = t->m_nodes[i].dTree.bsdfSamplingFractionOptimizer.m_state;
        s.iter = (int) in6[0]; s.firstMoment = in6[1]; s.secondMoment = in6[2]; s.variable = in6[3]; s.batchAccumulation = in6[4]; s.batchGradient = in6[5];
    }
    void aabb(float *mn, float *mx) const { const mitsuba::AABB &a = t->aabb(); for (int i = 0; i < 3; ++i) { mn[i] = a.min[i]; mx[i] = a.max[i]; } }
    size_t packSize() const { size_t n = 0; for (const auto &nd : t->m_nodes) if (nd.isLeaf) n += 4 * nd.dTree.building.numNodes() + 1; return n; }
    void packBuilding(float *buf, bool unpack) {
        size_t o = 0;
        for (auto &nd : t->m_nodes) {
            if (!nd.isLeaf) continue;
            for (auto &q : nd.dTree.building.m_nodes) for (int j = 0; j < 4; ++j) { if (unpack) q.setSum(j, buf[o]); else buf[o] = q.sum(j); ++o; }
            if (unpack) nd.dTree.building.setStatisticalWeight(buf[o]); else buf[o] = nd.dTree.building.statisticalWeight();
            ++o;
        }
    }
    void statistics(ppg_iteration_stats &st) const { backend_statistics(*this, st); }
};

}  // namespace ppgo
