// forest.cuh -- per-thread traversal of the packed forest (forest.cu), in the tail of feature_kernel
// (features.cu).  Semantics: cv::ml::RTrees::predict(.., PREDICT_SUM)
// (OpenCV DTreesImpl::predictTrees: left iff x[var] <= split.c, sum of leaf values) followed by the
// score line of KeypointLearningDetector::runForest (impl/KeypointLearning.hpp:281-287).
#pragma once
#include "kpl_internal.h"
#include "kpl_math.cuh"

namespace kpl {

#ifndef KPL_TREES_IN_FLIGHT
#define KPL_TREES_IN_FLIGHT 4
#endif
static constexpr int TREES_IN_FLIGHT = KPL_TREES_IN_FLIGHT;

// x[var * stride] is feature `var` of this thread's point (a shared-memory column: bank == lane for
// stride 32, so the data-dependent var never conflicts).  Four trees are walked concurrently so
// four independent block loads (L2 resident) are in flight per thread; nd[] counts 32-byte blocks.
//
// `fragile` reports whether any split DECIDED on the way (the nodes actually visited) had |x[var] - thr| <= 1e-5:
// a feature difference of the north star's tolerance against another implementation could send that walk the
// other way and move the score by 1/ntrees (BASELINE.md s5, call site hpp:281-287).
static constexpr float KPL_FRAGILE_EPS = 1e-5f;

template <bool FRAGILE>
__device__ __forceinline__ float forest_score(const float* x, int stride, const PackedNode* __restrict__ nodes,
                                              const int32_t* __restrict__ roots, int ntrees, bool& fragile)
{
    double sum = 0.0;
    bool frag = false;
    for (int t0 = 0; t0 < ntrees; t0 += TREES_IN_FLIGHT) {
        int nd[TREES_IN_FLIGHT];
        float val[TREES_IN_FLIGHT];
        bool live[TREES_IN_FLIGHT];
#pragma unroll
        for (int u = 0; u < TREES_IN_FLIGHT; ++u) {
            live[u] = (t0 + u) < ntrees;
            nd[u] = live[u] ? __ldg(roots + t0 + u) : 0;
            val[u] = 0.0f;
        }
        bool any = true;
        while (any) {
            any = false;
#pragma unroll
            for (int u = 0; u < TREES_IN_FLIGHT; ++u) {
                if (live[u]) {
                    // one 32-byte block: the node, its left child, its right child (pack_forest): two levels per sector
                    const uint4* blk = reinterpret_cast<const uint4*>(nodes) + 2 * (size_t)nd[u];
                    const uint4 pl = __ldg(blk);
                    const uint2 r = __ldg(reinterpret_cast<const uint2*>(blk + 1));
                    const uint32_t pvar = pl.y & 1023u;
                    if (pvar == KPL_LEAF_VAR) { val[u] = __uint_as_float(pl.x); live[u] = false; }
                    else {
                        // DTreesImpl::predictTrees: go left iff value <= split.c
                        const float xp = x[pvar * stride];
                        const bool left = xp <= __uint_as_float(pl.x);
                        if (FRAGILE) frag |= fabsf(__fsub_rn(xp, __uint_as_float(pl.x))) <= KPL_FRAGILE_EPS;
                        const uint32_t cthr = left ? pl.z : r.x, cpk = left ? pl.w : r.y;
                        const uint32_t cvar = cpk & 1023u;
                        if (cvar == KPL_LEAF_VAR) { val[u] = __uint_as_float(cthr); live[u] = false; }
                        else {
                            const float xc = x[cvar * stride];
                            if (FRAGILE) frag |= fabsf(__fsub_rn(xc, __uint_as_float(cthr))) <= KPL_FRAGILE_EPS;
                            nd[u] += (int)(cpk >> 10) + ((xc <= __uint_as_float(cthr)) ? 0 : 1);
                            any = true;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < TREES_IN_FLIGHT; ++u) sum += (double)val[u];   // exact: leaf values are small integers
    }
    fragile = frag;
    const float fsum = __double2float_rn(sum);                                           // predict() returns float
    return __fsub_rn(1.0f, __fdiv_rn(fsum, __fmul_rn((float)ntrees, 1.0f)));             // hpp:287
}

}  // namespace kpl
