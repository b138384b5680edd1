// ppg_kernels.cuh -- the non-bounce kernels of the wavefront pipeline (flush, commit, film, SD-tree maintenance, Adam replay).
// Included by ppg_host.cu only; the structures shared with the bounce kernel live in ppg_wavefront.cuh.
#pragma once
#include "ppg_wavefront.cuh"

namespace ppg {

// paths still alive after the last bounce (only possible with maxDepth == -1 and the bounce cap) keep their radiance; counted in *truncated
__global__ void __launch_bounds__(PPG_BLOCK) flush_kernel(PathState in, const uint32_t *liveIn, float4 *liFinal, unsigned long long *truncated) {
    const uint32_t nIn = *liveIn;
    if (blockIdx.x == 0 && threadIdx.x == 0 && nIn) atomicAdd(truncated, (unsigned long long) nIn);
    for (uint32_t i = blockIdx.x * PPG_BLOCK + threadIdx.x; i < nIn; i += gridDim.x * PPG_BLOCK) {
        const float4 c = in.s2[i], e = in.s3[i];
        liFinal[__float_as_uint(e.y)] = make_float4(c.z, c.w, e.x, 1.f);
    }
}

// ------------------------------------------------------------------ commit: vertices -> building trees
struct CommitParams {
    TreeView tree;
    VertexSlab slab0;              // slab of depth 1; slab k lives at +k*slabStride entries
    size_t slabStride;
    const uint32_t *liveCounts;    // liveCounts[k]: entries of slab k (the input live count of that bounce)
    const float4 *liFinal;
    int spatialFilter, directionalFilter, lossMode;   // lossMode already gated by isBuilt (GP:2152)
    float statisticalWeight;       // 1.0; 0.5 while nee=kickstart samples lights (GP:2152)
    VertexSlab nee0;               // NEE slabs (blockIdx.y >= nSlabs): fixed radiance, weight 0.5 (GP:2014)
    uint32_t nSlabs;
    uint64_t seed;
    const uint2 *snodes;
    // sampling-fraction learning: one record per (vertex, leaf) pair, consumed by adam_seq_kernel
    float4 *adamRecA;              // bits(leaf), product, woPdf, bsdfPdf
    float2 *adamRecB;              // dTreePdf, statistical weight
    uint32_t *adamTotal;           // device counter of appended records
    uint32_t adamCap;
    unsigned long long *dropped;   // records beyond adamCap (surfaced as ppg_stats.dropped_records)
};

// DTreeWrapper::record (GP:575-584) into the building tree of S-tree node `leaf`.
// weightDone: the statistical-weight add was already issued by the caller (warp-aggregated).
__device__ __forceinline__ void record_into_leaf(const CommitParams &C, uint32_t leaf, float3 d, float radiance, float product, float woPdf, float bsdfPdf,
                                                 float dTreePdf, float weight, bool isDelta, int directionalFilter, int lossMode, bool weightDone) {
    const TreeView &T = C.tree;
    const float4 la = __ldg(&T.leafA[leaf]);
    if (!isDelta) {
        const bool wOk = isfinite(weight) && weight > 0.f;                    // DTree::recordIrradiance, GP:395-413
        if (wOk) {
            if (!weightDone) red_add(&T.bweight[leaf], weight);
            dtree_record_irradiance(T.bchildren, T.bsums, __float_as_uint(la.y), dir_to_canonical(d), radiance / woPdf, weight, directionalFilter);
        }
    }
    if (lossMode != 0 && product > 0.f) {
        // optimizeBsdfSamplingFraction (GP:672-697) is order dependent: defer it to adam_seq_kernel, which replays the
        // records of each leaf sequentially.  Opportunistic warp aggregation of the list cursor (one atomic per warp).
        const unsigned m = __activemask();
        const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(C.adamTotal, (uint32_t) __popc(m));
        base = __shfl_sync(m, base, leader);
        const uint32_t idx = base + __popc(m & ((1u << lane) - 1u));
        if (idx < C.adamCap) {
            C.adamRecA[idx] = make_float4(__uint_as_float(leaf), product, woPdf, bsdfPdf);
            C.adamRecB[idx] = make_float2(dTreePdf, weight);
        } else atomicAdd(C.dropped, 1ull);
    }
}

template <int RECORD>
__global__ void __launch_bounds__(PPG_BLOCK) commit_kernel(const CommitParams P) {
    const bool neeSlab = blockIdx.y >= P.nSlabs;
    const uint32_t k = neeSlab ? blockIdx.y - P.nSlabs : blockIdx.y;
    const uint32_t n = P.liveCounts[k];
    const size_t so = (size_t) k * P.slabStride;
    VertexSlab S;      // select field by field (values), never by address: kernel parameters live in the param space
    S.v0 = neeSlab ? P.nee0.v0 : P.slab0.v0; S.v1 = neeSlab ? P.nee0.v1 : P.slab0.v1; S.v2 = neeSlab ? P.nee0.v2 : P.slab0.v2;
    S.v3 = neeSlab ? P.nee0.v3 : P.slab0.v3; S.v4 = neeSlab ? P.nee0.v4 : P.slab0.v4; S.v5 = neeSlab ? P.nee0.v5 : P.slab0.v5;
    const float vertexWeight = neeSlab ? 0.5f : P.statisticalWeight;
    for (uint32_t base = blockIdx.x * PPG_BLOCK; base < n; base += gridDim.x * PPG_BLOCK) {
        const uint32_t i = base + threadIdx.x;
        bool ok = i < n;
        float4 v0, v1, v2, v4 = make_float4(0, 0, 0, 0), v5 = make_float4(0, 0, 0, 0);
        uint32_t pid = PPG_INVALID;
        if (ok) { v2 = __ldcs(&S.v2[so + i]); pid = __float_as_uint(v2.w); ok = pid != PPG_INVALID; }
        float3 d = f3(0, 0, 1), radiance = f3(0, 0, 0), thr = f3(1, 1, 1), bsdfVal = f3(0, 0, 0); float woPdf = 0.f, bsdfPdf = 0.f, dTreePdf = 0.f;
        uint32_t leaf = 0; bool isDelta = false;
        if (ok) {
            v0 = __ldcs(&S.v0[so + i]); v1 = __ldcs(&S.v1[so + i]);
            isDelta = pid >> 31; const bool absolute = (pid >> 30) & 1u; pid &= 0x3fffffffu;
            const float4 lf = absolute ? make_float4(v2.x * 2.f, v2.y * 2.f, v2.z * 2.f, 0.f) : __ldg(&P.liFinal[pid]);
            d = f3(v0.x, v0.y, v0.z); woPdf = v0.w; thr = f3(v1.x, v1.y, v1.z); leaf = __float_as_uint(v1.w);
            radiance = f3(lf.x - v2.x, lf.y - v2.y, lf.z - v2.z);                  // everything recorded after the vertex was created
            if (RECORD == 2) {
                const float4 v3 = __ldcs(&S.v3[so + i]); bsdfVal = f3(v3.x, v3.y, v3.z); bsdfPdf = v3.w;
                v4 = __ldcs(&S.v4[so + i]); v5 = __ldcs(&S.v5[so + i]); dTreePdf = v4.w;
            }
            // Vertex::commit, GP:1730-1768
            if (!(woPdf > 0.f) || !is_valid(radiance) || !is_valid(bsdfVal)) ok = false;
        }
        float3 local = f3(0, 0, 0);
        if (ok) {
            if (thr.x * woPdf > PPG_EPSILON) local.x = radiance.x / thr.x;
            if (thr.y * woPdf > PPG_EPSILON) local.y = radiance.y / thr.y;
            if (thr.z * woPdf > PPG_EPSILON) local.z = radiance.z / thr.z;
        }
        const float3 prod = local * bsdfVal;
        const float avgLocal = (local.x + local.y + local.z) * (1.0f / 3.0f);       // Spectrum::average()
        const float avgProduct = (prod.x + prod.y + prod.z) * (1.0f / 3.0f);
        const bool nearest = RECORD == 1 || P.spatialFilter == 0;
        if (nearest) {
            // nearest: the vertex's own leaf.  The statistical-weight counter of a leaf is ONE address that every vertex
            // of that leaf hits (iteration 0: one address for the whole wavefront) -> one atomic per distinct leaf per warp.
            // All 32 lanes reach this call (the loop trip count is block-uniform).
            const float w = vertexWeight;
            warp_aggregated_add(P.tree.bweight, leaf, w, ok && !isDelta && isfinite(w) && w > 0.f);
            if (ok) record_into_leaf(P, leaf, d, avgLocal, avgProduct, woPdf, bsdfPdf, dTreePdf, w, isDelta, P.directionalFilter, P.lossMode, true);
        } else if (ok) {
            const float3 o = f3(v4.x, v4.y, v4.z);
            const uint32_t lo = __float_as_uint(v5.z);
            const float3 voxel = voxel_size(P.tree.extent, (int) (lo & 0xffu));
            if (P.spatialFilter == 1) {
                // stochastic box filter, GP:1746-1763: jitter the position inside the voxel-sized box, clip, re-lookup
                const uint64_t sampleIndex = ((uint64_t) __float_as_uint(v5.y) << 32) | __float_as_uint(v5.x);
                Pcg32 r; seed_vertex_rng(r, P.seed, sampleIndex, lo >> 8);
                float3 off = voxel;
                off.x *= r.next1D() - 0.5f; off.y *= r.next1D() - 0.5f; off.z *= r.next1D() - 0.5f;
                float3 q = o + off;
                const float3 mx = P.tree.aabbMin + P.tree.extent;
                q.x = fminf(fmaxf(q.x, P.tree.aabbMin.x), mx.x); q.y = fminf(fmaxf(q.y, P.tree.aabbMin.y), mx.y); q.z = fminf(fmaxf(q.z, P.tree.aabbMin.z), mx.z);
                int lv; const uint32_t splat = stree_lookup(P.snodes, P.tree.stable, P.tree.aabbMin, P.tree.extent, q, lv);
                record_into_leaf(P, splat, d, avgLocal, avgProduct, woPdf, bsdfPdf, dTreePdf, vertexWeight, isDelta, P.directionalFilter, P.lossMode, false);
            } else {
                // box filter, STree::record GP:935-943 + STreeNode::record GP:823-839: every leaf overlapping the voxel-sized box
                const float volume = voxel.x * voxel.y * voxel.z;
                const float w0 = vertexWeight / volume;
                const float3 min1 = o - voxel * 0.5f, max1 = o + voxel * 0.5f;
                struct E { uint32_t n; float3 mn, sz; int axis; };
                E st[64]; int sp = 0;
                st[sp++] = E{0u, P.tree.aabbMin, P.tree.extent, 0};
                while (sp) {
                    const E e = st[--sp];
                    const float lx = fmaxf(fminf(max1.x, e.mn.x + e.sz.x) - fmaxf(min1.x, e.mn.x), 0.f);
                    const float ly = fmaxf(fminf(max1.y, e.mn.y + e.sz.y) - fmaxf(min1.y, e.mn.y), 0.f);
                    const float lz = fmaxf(fminf(max1.z, e.mn.z + e.sz.z) - fmaxf(min1.z, e.mn.z), 0.f);
                    const float w = lx * ly * lz;
                    if (!(w > 0.f)) continue;
                    const uint2 c = __ldg(&P.snodes[e.n]);
                    if (c.x == 0u) {
                        record_into_leaf(P, e.n, d, avgLocal, avgProduct, woPdf, bsdfPdf, dTreePdf, w0 * w, isDelta, P.directionalFilter, P.lossMode, false);
                    } else if (sp + 2 <= 64) {
                        float3 sz = e.sz, mn1 = e.mn;
                        if (e.axis == 0) { sz.x /= 2.f; mn1.x += sz.x; } else if (e.axis == 1) { sz.y /= 2.f; mn1.y += sz.y; } else { sz.z /= 2.f; mn1.z += sz.z; }
                        const int na = (e.axis + 1) % 3;
                        st[sp++] = E{c.y, mn1, sz, na};
                        st[sp++] = E{c.x, e.mn, sz, na};
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------ film
// block->put(samplePos, spec) and squaredBlock->put(samplePos, spec*spec) (GP:1633-1634); invalid samples are
// dropped (imageblock.h:150-154).  Box filter: the sample lands in its own pixel with weight 1.
__global__ void __launch_bounds__(PPG_BLOCK) film_kernel(const float4 *liFinal, const uint32_t *pixelMap, uint32_t nLocalPixels, uint32_t spp,
                                                         uint32_t passesInBatch, int W, float4 *image, float4 *sqImage) {
    for (uint32_t lp = blockIdx.x * PPG_BLOCK + threadIdx.x; lp < nLocalPixels; lp += gridDim.x * PPG_BLOCK) {
        float4 a = make_float4(0, 0, 0, 0), q = make_float4(0, 0, 0, 0);
        for (uint32_t pb = 0; pb < passesInBatch; ++pb)
            for (uint32_t s = 0; s < spp; ++s) {
                const float4 L = liFinal[((size_t) pb * nLocalPixels + lp) * spp + s];
                if (!is_valid(f3(L.x, L.y, L.z))) continue;
                a.x += L.x; a.y += L.y; a.z += L.z; a.w += 1.f;
                q.x += L.x * L.x; q.y += L.y * L.y; q.z += L.z * L.z; q.w += 1.f;
            }
        const uint32_t xy = pixelMap[lp];
        const size_t px = (size_t) (xy >> 16) * W + (xy & 0xffffu);
        float4 A = image[px], Q = sqImage[px];
        A.x += a.x; A.y += a.y; A.z += a.z; A.w += a.w;
        Q.x += q.x; Q.y += q.y; Q.z += q.z; Q.w += q.w;
        image[px] = A; sqImage[px] = Q;
    }
}

// variance estimate with the getPixel() quirk (SURVEY A.6; GP:1300-1313): sum over this rank's pixels of
// min(lum(S2/W - (S1/W)^2/N), 1e4), accumulated in double
__global__ void __launch_bounds__(PPG_BLOCK) variance_kernel(const float4 *image, const float4 *sqImage, const uint32_t *pixelMap, uint32_t nLocalPixels,
                                                             int W, float N, double *out) {
    __shared__ double sh[PPG_BLOCK / 32];
    double acc = 0.0;
    for (uint32_t lp = blockIdx.x * PPG_BLOCK + threadIdx.x; lp < nLocalPixels; lp += gridDim.x * PPG_BLOCK) {
        const uint32_t xy = pixelMap[lp];
        const size_t px = (size_t) (xy >> 16) * W + (xy & 0xffffu);
        const float4 A = image[px], Q = sqImage[px];
        const float iw = A.w != 0.f ? 1.0f / A.w : 0.f, isw = Q.w != 0.f ? 1.0f / Q.w : 0.f;
        const float p0 = A.x * iw, p1 = A.y * iw, p2 = A.z * iw;
        const float l0 = Q.x * isw - p0 * p0 / N, l1 = Q.y * isw - p1 * p1 / N, l2 = Q.z * isw - p2 * p2 / N;
        const float lum = l0 * 0.212671f + l1 * 0.715160f + l2 * 0.072169f;
        acc += (double) fminf(lum, 10000.0f);
    }
    for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0; for (int w = 0; w < PPG_BLOCK / 32; ++w) t += sh[w];
        atomicAdd(out, t);
    }
}

__global__ void add_image_kernel(float4 *dst, const float4 *src, size_t n) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        float4 a = dst[i]; const float4 b = src[i];
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; dst[i] = a;
    }
}
// film develop: weight-normalised RGB (hdrfilm); accumulate != 0: out += scale * normalised (inverse-variance combination, GP:1567-1582)
__global__ void develop_kernel(const float4 *film, float *rgb, size_t n, float scale, int accumulate) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t) gridDim.x * blockDim.x) {
        const float4 a = film[i];
        const float iw = a.w != 0.f ? 1.0f / a.w : 0.f;
        if (accumulate) { rgb[3 * i] += a.x * iw * scale; rgb[3 * i + 1] += a.y * iw * scale; rgb[3 * i + 2] += a.z * iw * scale; }
        else { rgb[3 * i] = a.x * iw * scale; rgb[3 * i + 1] = a.y * iw * scale; rgb[3 * i + 2] = a.z * iw * scale; }
    }
}

// ------------------------------------------------------------------ SD-tree maintenance (device side)
struct MaintParams {
    uint2 *snodes;                // S-tree nodes
    float4 *leafA;                // per node leaf record
    float *bweight;               // per node building statistical weight
    float *sampSum, *sampWeight;  // per node: DTree::m_atomic of the sampling tree
    int *sampDepth;               // per node: m_maxDepth of the sampling tree
    uint32_t *sampCount;          // per node: node count of the sampling tree
    float *adam;                  // per node: 6 floats (iter, m, v, variable, batchAcc, batchGrad)
    uint32_t *buildCount;         // per node: node count of the building tree
    int *buildDepth;              // per node: m_maxDepth of the building tree
    uint32_t *nNodes;             // device scalar: current S-tree node count
    uint32_t capNodes;
    SampNode *samp; uint2 *bchildren; float4 *bsums;
};

// STree::refine (GP:957-998) as a single persistent block: rounds over the frontier of newly created nodes;
// a leaf splits while its building weight exceeds the threshold (GP:953-955), both children inherit the parent's
// leaf record (shared sampling tree, Adam state) with half the building weight (GP:876-895).  Children are allocated
// with a block prefix sum, so node numbering is deterministic (required for identical replicas across ranks).
__global__ void __launch_bounds__(1024) stree_refine_kernel(MaintParams M, float threshold, uint32_t *overflow) {
    __shared__ uint32_t sScan[1024];
    __shared__ uint32_t sBase, sBegin, sEnd, sAny;
    if (threadIdx.x == 0) { sBegin = 0; sEnd = *M.nNodes; }
    __syncthreads();
    for (;;) {
        const uint32_t begin = sBegin, end = sEnd;
        if (threadIdx.x == 0) { sBase = end; sAny = 0; }
        __syncthreads();
        for (uint32_t chunk = begin; chunk < end; chunk += 1024) {
            const uint32_t n = chunk + threadIdx.x;
            bool split = false;
            if (n < end) split = M.snodes[n].x == 0u && M.bweight[n] > threshold;
            // block exclusive scan of the split flags
            sScan[threadIdx.x] = split ? 1u : 0u;
            __syncthreads();
            for (int off = 1; off < 1024; off <<= 1) {
                uint32_t v = threadIdx.x >= off ? sScan[threadIdx.x - off] : 0u;
                __syncthreads();
                sScan[threadIdx.x] += v;
                __syncthreads();
            }
            const uint32_t incl = sScan[threadIdx.x], total = sScan[1023];
            const uint32_t base = sBase;
            if (split) {
                const uint32_t c0 = base + 2 * (incl - 1);
                if (c0 + 1 >= M.capNodes) *overflow = 1u;             // the host sizes the arrays from the recorded weight; never seen, but never silent
                else {
                    const float4 la = M.leafA[n];
                    const float half = M.bweight[n] / 2.f;
                    for (int c = 0; c < 2; ++c) {
                        const uint32_t ci = c0 + c;
                        M.snodes[ci] = make_uint2(0u, 0u);
                        M.leafA[ci] = la; M.bweight[ci] = half;
                        M.sampSum[ci] = M.sampSum[n]; M.sampWeight[ci] = M.sampWeight[n]; M.sampDepth[ci] = M.sampDepth[n]; M.sampCount[ci] = M.sampCount[n];
                        for (int j = 0; j < 6; ++j) M.adam[6 * ci + j] = M.adam[6 * n + j];
                    }
                    M.snodes[n] = make_uint2(c0, c0 + 1);
                    M.bweight[n] = 0.f;
                }
            }
            __syncthreads();
            if (threadIdx.x == 0) { sBase = min(base + 2 * total, M.capNodes & ~1u); if (total) sAny = 1; }
            __syncthreads();
        }
        if (threadIdx.x == 0) { sBegin = end; sEnd = sBase; }
        __syncthreads();
        if (!sAny || sBegin >= sEnd) break;
    }
    if (threadIdx.x == 0) *M.nNodes = sEnd;
}

// Prefix table of the S-tree (see stree_lookup): entry `key` = where the walk stands after following the 3*BITS
// interleaved digits of key (x digit first), or the leaf it ended in earlier.
__global__ void stree_table_kernel(const uint2 *snodes, uint32_t *table) {
    const uint32_t nKeys = 1u << (3 * PPG_STREE_TABLE_BITS);
    for (uint32_t key = blockIdx.x * blockDim.x + threadIdx.x; key < nKeys; key += gridDim.x * blockDim.x) {
        uint32_t n = 0, depth = 0, leaf = 0;
        for (int level = 0; level < 3 * PPG_STREE_TABLE_BITS; ++level) {
            const uint2 c = snodes[n];
            if (c.x == 0u) { leaf = 1; break; }
            const uint32_t bit = (key >> (3 * PPG_STREE_TABLE_BITS - 1 - level)) & 1u;
            n = bit ? c.y : c.x; ++depth;
        }
        if (!leaf && snodes[n].x == 0u) leaf = 1;
        table[key] = n | (depth << 24) | (leaf << 31);
    }
}

// DTree::reset (GP:456-514), one thread per S-tree leaf.  The new building topology is the refinement of the leaf's
// sampling tree: child i of a node at `depth` is subdivided iff depth < maxDepth and sum_i/total > threshold (for a
// brand-new subtree the provisional sums are parent_sum/4; if total == 0 the fraction is 0.25^depth).  The DFS uses
// the reference's stack discipline so that node numbering is identical to the reference's.
// FILL == false: count nodes only (-> buildCount, buildDepth).  FILL == true: write the topology at buildBase and zero sums.
template <bool FILL>
__global__ void __launch_bounds__(128) dtree_reset_kernel(MaintParams M, const uint32_t *buildBase, int newMaxDepth, float subdivisionThreshold) {
    const uint32_t nNodes = *M.nNodes;
    for (uint32_t leaf = blockIdx.x * blockDim.x + threadIdx.x; leaf < nNodes; leaf += gridDim.x * blockDim.x) {
        if (M.snodes[leaf].x != 0u) { if (!FILL) M.buildCount[leaf] = 0; continue; }
        const SampNode *prev = M.samp + __float_as_uint(M.leafA[leaf].x);
        const float total = M.sampSum[leaf];
        const uint32_t base = FILL ? buildBase[leaf] : 0u;
        struct S { uint16_t nodeIndex, otherNodeIndex; uint8_t otherIsPrev, depth; float quarter; };
        S stack[64]; int sp = 0;
        stack[sp++] = S{0, 0, 1, 1, 0.f};
        uint32_t count = 1; int maxDepth = 0;
        if (FILL) { M.bchildren[base] = make_uint2(0u, 0u); M.bsums[base] = make_float4(0, 0, 0, 0); }
        bool full = false;
        while (sp && !full) {
            const S s = stack[--sp];
            maxDepth = max(maxDepth, (int) s.depth);
            float4 osum; uint2 och = make_uint2(0u, 0u);
            if (s.otherIsPrev) { osum = prev[s.otherNodeIndex].sums; och = prev[s.otherNodeIndex].children; }
            else osum = make_float4(s.quarter, s.quarter, s.quarter, s.quarter);
            uint32_t childOut[4] = {0, 0, 0, 0};
            for (int i = 0; i < 4; ++i) {
                const float si = sum4(osum, i);
                const float fraction = total > 0.f ? (si / total) : ldexpf(1.0f, -2 * (int) s.depth);   // std::pow(0.25f, depth), exact
                if ((int) s.depth < newMaxDepth && fraction > subdivisionThreshold) {
                    const uint32_t oc = s.otherIsPrev ? child16(och, i) : 0u;
                    if (sp < 64) {
                        if (oc != 0u) stack[sp++] = S{(uint16_t) count, (uint16_t) oc, 1, (uint8_t) (s.depth + 1), 0.f};
                        else stack[sp++] = S{(uint16_t) count, (uint16_t) count, 0, (uint8_t) (s.depth + 1), si / 4.f};
                    }
                    childOut[i] = count;
                    if (FILL) { M.bchildren[base + count] = make_uint2(0u, 0u); M.bsums[base + count] = make_float4(0, 0, 0, 0); }
                    ++count;
                    if (count > 65535u) { full = true; break; }                      // GP:499-503
                }
            }
            if (FILL) M.bchildren[base + s.nodeIndex] = make_uint2(childOut[0] | (childOut[1] << 16), childOut[2] | (childOut[3] << 16));
        }
        if (!FILL) { M.buildCount[leaf] = count; M.buildDepth[leaf] = maxDepth; }
    }
}

// DTree::build (GP:520-533, 346-366) + "sampling = building" (GP:610-613), one thread per S-tree leaf.
// Children have larger indices than their parent (reset appends), so one reverse sweep equals the recursion.
__global__ void __launch_bounds__(128) dtree_build_kernel(MaintParams M, const uint32_t *buildBase) {
    const uint32_t nNodes = *M.nNodes;
    for (uint32_t leaf = blockIdx.x * blockDim.x + threadIdx.x; leaf < nNodes; leaf += gridDim.x * blockDim.x) {
        if (M.snodes[leaf].x != 0u) continue;
        const uint32_t base = buildBase[leaf], count = M.buildCount[leaf];
        for (uint32_t k = count; k-- > 0;) {
            float4 s = M.bsums[base + k];
            const uint2 ch = M.bchildren[base + k];
            float *sp = reinterpret_cast<float *>(&s);
            for (int i = 0; i < 4; ++i) {
                const uint32_t c = child16(ch, i);
                if (c == 0u) continue;
                const float4 cs = M.samp[base + c].sums;          // already built (c > k)
                float sum = 0.f; sum += cs.x; sum += cs.y; sum += cs.z; sum += cs.w;
                sp[i] = sum;
            }
            SampNode out; out.sums = s; out.children = ch; out.pad = make_uint2(0u, 0u);
            M.samp[base + k] = out;
        }
        const float4 r = M.samp[base].sums;
        float sum = 0.f; sum += r.x; sum += r.y; sum += r.z; sum += r.w;
        const float w = M.bweight[leaf];
        M.sampSum[leaf] = sum; M.sampWeight[leaf] = w; M.sampDepth[leaf] = M.buildDepth[leaf]; M.sampCount[leaf] = count;
        // DTree::mean() > 0 (GP:387-393)
        float mean = 0.f;
        if (w != 0.f) { const float factor = 1.f / (PPG_PI * 4.f * w); mean = factor * sum; }
        float4 la = M.leafA[leaf];
        la.x = __uint_as_float(base); la.y = __uint_as_float(base); la.w = __uint_as_float(mean > 0.f ? 1u : 0u);
        M.leafA[leaf] = la;
    }
}

// after reset: point every leaf at its new building tree and zero the building statistical weight (GP:457)
__global__ void leaf_after_reset_kernel(MaintParams M, const uint32_t *buildBase) {
    const uint32_t nNodes = *M.nNodes;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < nNodes; n += gridDim.x * blockDim.x) {
        float4 la = M.leafA[n]; la.y = __uint_as_float(buildBase[n]); M.leafA[n] = la;
        M.bweight[n] = 0.f;
    }
}

// exclusive prefix sum of counts[0..n) by a single block (n is at most a few 1e5..1e6 S-tree nodes, once per iteration)
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const uint32_t *counts, uint32_t *offsets, const uint32_t *nPtr, uint32_t *totalOut) {
    __shared__ uint32_t sScan[1024];
    __shared__ uint32_t sCarry;
    const uint32_t n = *nPtr;
    if (threadIdx.x == 0) sCarry = 0;
    __syncthreads();
    for (uint32_t chunk = 0; chunk < n; chunk += 1024) {
        const uint32_t i = chunk + threadIdx.x;
        const uint32_t v = i < n ? counts[i] : 0u;
        sScan[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            uint32_t t = threadIdx.x >= off ? sScan[threadIdx.x - off] : 0u;
            __syncthreads();
            sScan[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < n) offsets[i] = sCarry + sScan[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 0) sCarry += sScan[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) *totalOut = sCarry;
}

// ---- sampling-fraction learning (GP:69-133, 672-697) ----------------------------------------------------------------
// The reference runs optimizeBsdfSamplingFraction under a per-leaf spin lock: every record updates the leaf's batch
// accumulators at the CURRENT theta and takes an Adam step whenever the accumulated weight exceeds batchSize = 1.  That
// is inherently sequential per leaf but independent across leaves, so the records of one commit launch are bucketed by
// leaf (histogram -> scan -> scatter) and each leaf replays its bucket sequentially with the reference's exact arithmetic.
// (The order inside a bucket is arbitrary -- as it is between the reference's worker threads.)

// count records per leaf; lanes with the same leaf share one atomic
__global__ void __launch_bounds__(256) adam_hist_kernel(const float4 *recA, const uint32_t *total, uint32_t cap, uint32_t *count) {
    const uint32_t n = min(*total, cap);
    const uint32_t nPad = (n + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nPad; i += gridDim.x * blockDim.x) {
        const bool ok = i < n;
        const uint32_t leaf = ok ? __float_as_uint(recA[i].x) : 0u;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(m, leaf);
            if ((int) (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&count[leaf], (uint32_t) __popc(peers));
        }
    }
}
// move every record into its leaf's bucket
__global__ void __launch_bounds__(256) adam_scatter_kernel(const float4 *recA, const float2 *recB, const uint32_t *total, uint32_t cap, const uint32_t *offset,
                                                           uint32_t *cursor, float4 *outA, float2 *outB) {
    const uint32_t n = min(*total, cap);
    const uint32_t nPad = (n + 31u) & ~31u;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nPad; i += gridDim.x * blockDim.x) {
        const bool ok = i < n;
        float4 a = make_float4(0, 0, 0, 0); float2 b = make_float2(0, 0);
        if (ok) { a = recA[i]; b = recB[i]; }
        const uint32_t leaf = __float_as_uint(a.x);
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(m, leaf);
            const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
            uint32_t base = 0;
            if (lane == leader) base = atomicAdd(&cursor[leaf], (uint32_t) __popc(peers));
            base = __shfl_sync(peers, base, leader);
            const uint32_t pos = offset[leaf] + base + __popc(peers & ((1u << lane) - 1u));
            outA[pos] = a; outB[pos] = b;
        }
    }
}
// ---- the replay chain of one leaf, factored out of adam_seq_kernel so that the same source also runs host-compiled (tests/hostdev)
// AdamOptimizer::State (GP:116-124) plus what the chain keeps between steps.  beta^iter as running double-precision products (the reference
// evaluates std::pow(float, int) in double, GP:98-99; a pow() per step would sit on the sequential chain); the fraction f = logistic(variable)
// and f (1 - f) are re-evaluated after a step, not per record.
struct FractionChain {
    int iter; float m1, m2, variable, batchAcc, batchGrad;
    double b1pow, b2pow;
    float f, g, fdf;          // f, 1 - f, f (1 - f)
};
__device__ __forceinline__ void fraction_logistic(FractionChain &s) {
    s.f = __fdividef(1.f, 1.f + __expf(-s.variable)); s.g = 1.f - s.f; s.fdf = s.f * s.g;      // logistic (GP:64-66), fast intrinsics
}
// `st`: the 6 floats of MaintParams::adam (iter, m, v, variable, batchAcc, batchGrad)
__device__ __forceinline__ FractionChain fraction_begin(const float *st) {
    FractionChain s;
    s.iter = (int) st[0]; s.m1 = st[1]; s.m2 = st[2]; s.variable = st[3]; s.batchAcc = st[4]; s.batchGrad = st[5];
    s.b1pow = pow((double) 0.9f, (double) s.iter); s.b2pow = pow((double) 0.999f, (double) s.iter);
    fraction_logistic(s);
    return s;
}
__device__ __forceinline__ void fraction_end(const FractionChain &s, float *st) {
    st[0] = (float) s.iter; st[1] = s.m1; st[2] = s.m2; st[3] = s.variable; st[4] = s.batchAcc; st[5] = s.batchGrad;
}
// The chain's latency is what the replay costs (the hottest leaf of SPACESHIP 1080p holds > 10^6 records per iteration), so everything that does
// not depend on theta is taken off it: each record is reduced to {k, b, c, w} with
//     dL/df = -ratio / woPdf * (bsdfPdf - dTreePdf),  ratio = (product / mix)^p,  mix = f * b + (1 - f) * c,  b = bsdfPdf,  c = dTreePdf
//   KL (p = 1):  dL/df = -k / mix,      k = product * (bsdfPdf - dTreePdf) / woPdf
//   var (p = 2): dL/df = -k / mix^2,    k = product^2 * (bsdfPdf - dTreePdf) / woPdf
// and the chain keeps one fast division per record and {division, rsqrt, exp} per step.  The mixture is the reference's expression (GP:680), not
// c + f (b - c): where dTreePdf > 2^24 bsdfPdf the difference loses bsdfPdf, and at a saturated fraction (f rounds to 1 for theta >= 17) that
// mixture is exactly 0 -- an infinite dL/df times f (1 - f) = 0 made the moments NaN and pinned theta at -20 for good.
__device__ __forceinline__ float fraction_k(float product, float woPdf, float bsdfPdf, float dTreePdf, bool var) {
    return (var ? product * product : product) * (bsdfPdf - dTreePdf) / woPdf;
}
// AdamOptimizer::step (GP:97-109)
__device__ __forceinline__ void fraction_step(FractionChain &s) {
    const float grad = __fdividef(s.batchGrad, s.batchAcc);
    ++s.iter; s.b1pow *= (double) 0.9f; s.b2pow *= (double) 0.999f;
    const float lr = 0.01f * sqrtf(1.f - (float) s.b2pow) / (1.f - (float) s.b1pow);     // depends on the step count only: off the chain
    s.m1 = 0.9f * s.m1 + (1.f - 0.9f) * grad;
    s.m2 = 0.999f * s.m2 + (1.f - 0.999f) * grad * grad;
    s.variable -= __fdividef(lr * s.m1, sqrtf(s.m2) + 1e-08f);
    s.variable = fminf(fmaxf(s.variable, -20.0f), 20.0f);
    s.batchGrad = 0.f; s.batchAcc = 0.f;
    fraction_logistic(s);
}
// one record: the gradient at the current variable (optimizeBsdfSamplingFraction, GP:672-697), AdamOptimizer::append (GP:85-95) and the
// step once the accumulated weight exceeds batchSize = 1
__device__ __forceinline__ void fraction_link(FractionChain &s, float k, float b, float c, float w, bool var) {
    const float mix = s.f * b + s.g * c;
    const float dLoss_df = -__fdividef(k, var ? mix * mix : mix);
    const float g = fmaf(dLoss_df, s.fdf, 0.01f * s.variable);
    s.batchGrad = fmaf(g, w, s.batchGrad); s.batchAcc += w;
    if (s.batchAcc > 1.0f) fraction_step(s);                 // batchSize = 1, GP:89
}

// One WARP per leaf.  The chain over a leaf's records is sequential (theta changes every ~2 records), so its speed is the latency of one link.
// The 32 lanes fetch the next 32 records with coalesced loads while the chain runs; every lane then walks the chain redundantly on values handed
// around with shuffles (no divergence, no dependent global load in the chain).  The first version (one THREAD per leaf, a dependent 24-byte fetch
// per record) spent ~0.3 us per record: 310 of 1000 ms on SPACESHIP 640x360, where the hottest leaf of an iteration holds > 100 000 records.
// The optimiser is not bit-reproducible in the reference either (records arrive in thread order): approximate-division rounding is far below that.
__global__ void __launch_bounds__(128) adam_seq_kernel(MaintParams M, const float4 *recA, const float2 *recB, const uint32_t *offset, uint32_t *count,
                                                       uint32_t *cursor, float ratioPower) {
    const uint32_t nNodes = *M.nNodes;
    const uint32_t lane = threadIdx.x & 31u, warpsPerGrid = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t leaf = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; leaf < nNodes; leaf += warpsPerGrid) {
        const uint32_t n = count[leaf];
        __syncwarp();
        if (lane == 0) { count[leaf] = 0; cursor[leaf] = 0; }              // ready for the next commit launch
        if (n == 0) continue;
        float *st = M.adam + 6 * (size_t) leaf;
        FractionChain s = fraction_begin(st);
        const uint32_t o = offset[leaf];
        float4 na = make_float4(0, 0, 0, 0); float2 nb = make_float2(0, 0);
        if (lane < n) { na = __ldg(&recA[o + lane]); nb = __ldg(&recB[o + lane]); }
        const bool var = ratioPower == 2.f;
        for (uint32_t base = 0; base < n; base += 32u) {
            const float4 ca = na; const float2 cb = nb;
            const uint32_t nxt = base + 32u + lane;
            if (nxt < n) { na = __ldg(&recA[o + nxt]); nb = __ldg(&recB[o + nxt]); }      // in flight while this chunk's chain runs
            const float kl = fraction_k(ca.y, ca.z, ca.w, cb.x, var);      // this lane's record, off the chain
            const uint32_t m = min(32u, n - base);
            for (uint32_t j = 0; j < m; ++j) {
                const float k_ = __shfl_sync(0xffffffffu, kl, j), b_ = __shfl_sync(0xffffffffu, ca.w, j), c_ = __shfl_sync(0xffffffffu, cb.x, j), w_ = __shfl_sync(0xffffffffu, cb.y, j);
                fraction_link(s, k_, b_, c_, w_, var);
            }
        }
        if (lane == 0) {
            fraction_end(s, st);
            float4 la = M.leafA[leaf]; la.z = s.variable; M.leafA[leaf] = la;
        }
    }
}
// N > 1 ranks: every rank replays its own records from the common state; the replicas are then merged.  The exchange buffer holds the SUM over
// ranks of [iter - iterBefore | m1 | m2 | variable | batchAcc | batchGrad] (6 arrays of nNodes floats).  Step counts add up, moments and the
// variable are averaged, and the batch accumulators add up RELATIVE to the common start (each rank's value contains the carried-over part once).
__global__ void adam_pack_kernel(MaintParams M, float *out6, float *before3, const float *unused, int stage) {
    const uint32_t nNodes = *M.nNodes;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < nNodes; n += gridDim.x * blockDim.x) {
        const float *st = M.adam + 6 * (size_t) n;
        if (stage == 0) { before3[n] = st[0]; before3[(size_t) nNodes + n] = st[4]; before3[2 * (size_t) nNodes + n] = st[5]; before3[3 * (size_t) nNodes + n] = st[3]; continue; }   // before the replay
        out6[n] = st[0] - before3[n];
        out6[(size_t) nNodes + n] = st[1]; out6[2 * (size_t) nNodes + n] = st[2]; out6[3 * (size_t) nNodes + n] = st[3];
        out6[4 * (size_t) nNodes + n] = st[4]; out6[5 * (size_t) nNodes + n] = st[5];
    }
}
__global__ void adam_merge_kernel(MaintParams M, const float *sum6, const float *before3, float invWorld, float worldMinus1) {
    const uint32_t nNodes = *M.nNodes;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < nNodes; n += gridDim.x * blockDim.x) {
        float *st = M.adam + 6 * (size_t) n;
        st[0] = before3[n] + sum6[n];
        st[1] = sum6[(size_t) nNodes + n] * invWorld; st[2] = sum6[2 * (size_t) nNodes + n] * invWorld; st[3] = sum6[3 * (size_t) nNodes + n] * invWorld;
        const float acc = sum6[4 * (size_t) nNodes + n] - worldMinus1 * before3[(size_t) nNodes + n];
        const float grad = sum6[5 * (size_t) nNodes + n] - worldMinus1 * before3[2 * (size_t) nNodes + n];
        st[4] = acc > 0.f ? acc : 0.f; st[5] = acc > 0.f ? grad : 0.f;
        float4 la = M.leafA[n]; la.z = st[3]; M.leafA[n] = la;
    }
}
// "Distribution statistics" of buildSDTree (GP:1121-1186) over all leaves: one block, warp-shuffle + shared-memory reduction
struct TreeStats {
    uint32_t leaves, leavesWithNodes; int depthMin, depthMax; float meanMin, meanMax, weightMin, weightMax;
    unsigned long long nodesMin, nodesMax; double depthSum, meanSum, nodesSum, weightSum;
};
__global__ void __launch_bounds__(1024) tree_stats_kernel(MaintParams M, TreeStats *out) {
    const uint32_t nNodes = *M.nNodes;
    uint32_t leaves = 0, withNodes = 0; int dMin = 0x7fffffff, dMax = 0; float rMin = 3.4e38f, rMax = 0.f, wMin = 3.4e38f, wMax = 0.f;
    unsigned long long nMin = ~0ull, nMax = 0ull; double dSum = 0, rSum = 0, nSum = 0, wSum = 0;
    for (uint32_t i = threadIdx.x; i < nNodes; i += blockDim.x) {
        if (M.snodes[i].x != 0u) continue;
        ++leaves;
        const int depth = M.sampDepth[i]; dMin = min(dMin, depth); dMax = max(dMax, depth); dSum += depth;
        const float w = M.sampWeight[i];
        float mean = 0.f; if (w != 0.f) { const float factor = 1.f / (PPG_PI * 4.f * w); mean = factor * M.sampSum[i]; }       // DTree::mean(), GP:387-393
        rMin = fminf(rMin, mean); rMax = fmaxf(rMax, mean); rSum += mean;
        const uint32_t cnt = M.sampCount[i];
        if (cnt > 1u) { nMin = min(nMin, (unsigned long long) cnt); nMax = max(nMax, (unsigned long long) cnt); nSum += cnt; ++withNodes; }
        wMin = fminf(wMin, w); wMax = fmaxf(wMax, w); wSum += w;
    }
    __shared__ TreeStats sh[32];
    for (int off = 16; off; off >>= 1) {
        leaves += __shfl_xor_sync(0xffffffffu, leaves, off); withNodes += __shfl_xor_sync(0xffffffffu, withNodes, off);
        dMin = min(dMin, __shfl_xor_sync(0xffffffffu, dMin, off)); dMax = max(dMax, __shfl_xor_sync(0xffffffffu, dMax, off));
        rMin = fminf(rMin, __shfl_xor_sync(0xffffffffu, rMin, off)); rMax = fmaxf(rMax, __shfl_xor_sync(0xffffffffu, rMax, off));
        wMin = fminf(wMin, __shfl_xor_sync(0xffffffffu, wMin, off)); wMax = fmaxf(wMax, __shfl_xor_sync(0xffffffffu, wMax, off));
        nMin = min(nMin, __shfl_xor_sync(0xffffffffu, nMin, off)); nMax = max(nMax, __shfl_xor_sync(0xffffffffu, nMax, off));
        dSum += __shfl_xor_sync(0xffffffffu, dSum, off); rSum += __shfl_xor_sync(0xffffffffu, rSum, off);
        nSum += __shfl_xor_sync(0xffffffffu, nSum, off); wSum += __shfl_xor_sync(0xffffffffu, wSum, off);
    }
    if ((threadIdx.x & 31) == 0) {
        TreeStats t; t.leaves = leaves; t.leavesWithNodes = withNodes; t.depthMin = dMin; t.depthMax = dMax; t.meanMin = rMin; t.meanMax = rMax; t.weightMin = wMin; t.weightMax = wMax;
        t.nodesMin = nMin; t.nodesMax = nMax; t.depthSum = dSum; t.meanSum = rSum; t.nodesSum = nSum; t.weightSum = wSum;
        sh[threadIdx.x >> 5] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        TreeStats t = sh[0];
        for (int w = 1; w < (int) (blockDim.x >> 5); ++w) {
            const TreeStats &o = sh[w];
            t.leaves += o.leaves; t.leavesWithNodes += o.leavesWithNodes; t.depthMin = min(t.depthMin, o.depthMin); t.depthMax = max(t.depthMax, o.depthMax);
            t.meanMin = fminf(t.meanMin, o.meanMin); t.meanMax = fmaxf(t.meanMax, o.meanMax); t.weightMin = fminf(t.weightMin, o.weightMin); t.weightMax = fmaxf(t.weightMax, o.weightMax);
            t.nodesMin = min(t.nodesMin, o.nodesMin); t.nodesMax = max(t.nodesMax, o.nodesMax);
            t.depthSum += o.depthSum; t.meanSum += o.meanSum; t.nodesSum += o.nodesSum; t.weightSum += o.weightSum;
        }
        *out = t;
    }
}
// How far did the sampling fractions move in the replay that just ended?  Sum over leaves of steps * |f_after - f_before| and of steps, in fixed
// point (2^-20) so that the result does not depend on the summation order: every rank derives the size of its next sub-batch from it
// (perform_render_passes), and all ranks must decide alike.  `before4`: [iter | batchAcc | batchGrad | theta] saved by adam_pack_kernel stage 0.
__global__ void adam_progress_kernel(MaintParams M, const float *before4, unsigned long long *out2) {
    const uint32_t nNodes = *M.nNodes;
    unsigned long long moved = 0, steps = 0;
    for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < nNodes; n += gridDim.x * blockDim.x) {
        const float *st = M.adam + 6 * (size_t) n;
        const float ds = st[0] - before4[n];
        if (!(ds > 0.f)) continue;
        const float df = fabsf(logistic(st[3]) - logistic(before4[3 * (size_t) nNodes + n]));
        const unsigned long long s = (unsigned long long) ds;
        steps += s; moved += s * (unsigned long long) (df * 1048576.0f);
    }
    for (int off = 16; off; off >>= 1) { moved += __shfl_xor_sync(0xffffffffu, moved, off); steps += __shfl_xor_sync(0xffffffffu, steps, off); }
    if ((threadIdx.x & 31) == 0 && steps) { atomicAdd(&out2[0], moved); atomicAdd(&out2[1], steps); }
}
__global__ void double_to_float_kernel(const double *in, float *out) { *out = (float) *in; }

}  // namespace ppg
