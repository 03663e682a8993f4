// nms.cu -- threshold + radius non-maxima suppression over the same uniform grid, and the plain
// radius-search kernels used for neighbour-set parity and for the exact work counters.
// Replaces the NMS loop of KeypointLearningDetector::detectKeypoints
// (impl/KeypointLearning.hpp:202-256, draws-remove branch off as in TestDetector :128).
#include <algorithm>
#include "kpl_internal.h"
#include "kpl_math.cuh"

namespace kpl {

__device__ __forceinline__ void key_to_cell_n(uint32_t key, int dimx, int dimy, int& cx, int& cy, int& cz)
{
    uint32_t t = key / (uint32_t)dimx;
    cx = (int)(key - t * (uint32_t)dimx);
    cz = (int)(t / (uint32_t)dimy);
    cy = (int)(t - (uint32_t)cz * (uint32_t)dimy);
}

// keypoint iff score >= th (compared in double, hpp:207) and no point with d2 < r_nms^2 has a
// strictly larger score (hpp:219).  A pure local-maximum test: order independent.
__global__ void __launch_bounds__(128)
nms_kernel(const float4* __restrict__ s_pos, const float* __restrict__ s_score, const uint32_t* __restrict__ skey,
           const int32_t* __restrict__ cell_start, const uint8_t* __restrict__ s_role, int dimx, int dimy, int dimz,
           int n, float rn2, int reach, double th, uint8_t* __restrict__ flag, unsigned long long* __restrict__ counters)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool above = false, near = false;
    if (i < n) {
        const float4 p = __ldg(s_pos + i);
        const uint32_t orig = __float_as_uint(p.w);
        const float my = __ldg(s_score + i);
        const bool owned = !s_role || ((s_role[i] & 3) == 3);
        above = owned && isfinite(my) && !((double)my < th);
        near = owned && isfinite(my) && fabs((double)my - th) <= 1e-5;
        bool is_max = above;
        if (above) {
            int cx, cy, cz;
            key_to_cell_n(__ldg(skey + i), dimx, dimy, cx, cy, cz);
            const int z0 = max(cz - reach, 0), z1 = min(cz + reach, dimz - 1);
            const int y0 = max(cy - reach, 0), y1 = min(cy + reach, dimy - 1);
            const int x0 = max(cx - reach, 0), x1 = min(cx + reach, dimx - 1);
            for (int z = z0; z <= z1 && is_max; ++z)
                for (int y = y0; y <= y1 && is_max; ++y) {
                    const int64_t base = ((int64_t)z * dimy + y) * dimx;
                    const int s = __ldg(cell_start + base + x0), e = __ldg(cell_start + base + x1 + 1);
                    for (int j = s; j < e; ++j) {
                        const float4 c = __ldg(s_pos + j);
                        if (dist2(p.x, p.y, p.z, c.x, c.y, c.z) < rn2 && my < __ldg(s_score + j)) { is_max = false; break; }
                    }
                }
        }
        flag[orig] = is_max ? 1 : 0;
    }
    unsigned m = __ballot_sync(0xFFFFFFFFu, above);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(counters + 2, (unsigned long long)__popc(m));
    m = __ballot_sync(0xFFFFFFFFu, near);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(counters + 7, (unsigned long long)__popc(m));
}

cudaError_t launch_nms(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th, int64_t flag_off)
{
    const kpl_params& U = c->params;
    cudaError_t e;
    if ((e = ensure(c->flag, (size_t)(flag_off + n)))) return e;
    const double rn = (double)U.radius_nms;
    nms_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->s_pos.p, s_score, c->key_b.p, c->cell_start.p,
                                                                   use_role ? c->s_role.p : nullptr,
                                                                   c->grid.dim[0], c->grid.dim[1], c->grid.dim[2], (int)n,
                                                                   (float)(rn * rn), c->grid.reach_nms, th, c->flag.p + flag_off, c->counters.p);
    c->launches++;
    return cudaGetLastError();
}

// ---- draws-remove branch (impl/KeypointLearning.hpp:233-250, setNonMaximaDrawsRemove(true)) ------------
// The reference walks the points in index order with a skip list: a local maximum i that ties with
// neighbours ("draws": equal score, d2 < r_nms^2, j != i) is dropped if an earlier surviving maximum put it
// on the skip list; otherwise it survives only if at least one draw lies closer than
// non_maxima_draws_threshold_, and every such close draw goes on the skip list.  Equivalent order-free
// statement, which is what runs here:
//   cand(i)   = above threshold, no strictly greater neighbour, at least one CLOSE draw
//   active(i) = cand(i) and no j < i with cand(j), active(j), j a close draw of i
//   keypoint  = active(i);  local maxima without any draw are keypoints as in the plain branch; local
//               maxima whose draws are all farther than the threshold are dropped (as in the reference).
// active() is resolved in rounds: an undecided candidate becomes skipped as soon as a lower-index close
// draw is active, and active once all of them are decided; the lowest undecided index always resolves, so
// the loop ends, and decisions never change once made (stale reads only postpone a decision).
// state: 0 not a keypoint, 1 keypoint, 2 undecided candidate, 3 skipped candidate.
// With roles (a slab of a sharded cloud) only OWNED points are classified and decided: a halo point's own
// lower-index draws may lie beyond the halo, so its state is always its owner's decision, copied in by the
// caller between rounds.  "Lower index" is then the GLOBAL index: gidx maps a local original index to it
// (nullptr: the identity, a single cloud or a batch, whose views keep their own index order).
__device__ __forceinline__ float draw_distance(const float4& p, const float4& c)
{
    // (pointIn.getVector3fMap() - drawPoint.getVector3fMap()).norm(): Eigen reduction order a0 + (a1 + a2)
    const float dx = __fsub_rn(p.x, c.x), dy = __fsub_rn(p.y, c.y), dz = __fsub_rn(p.z, c.z);
    return __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fadd_rn(__fmul_rn(dy, dy), __fmul_rn(dz, dz))));
}

template <int PASS>   // 0: classify, 1: one resolution round
__global__ void __launch_bounds__(128)
nms_draws_kernel(const float4* __restrict__ s_pos, const float* __restrict__ s_score, const uint32_t* __restrict__ skey,
                 const int32_t* __restrict__ cell_start, const uint8_t* __restrict__ s_role, int dimx, int dimy, int dimz,
                 int n, float rn2, int reach, double th, float draws_thr, const int32_t* __restrict__ gidx,
                 uint8_t* __restrict__ s_state, unsigned long long* __restrict__ counters)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool above = false, near = false;
    if (i < n) {
        const float4 p = __ldg(s_pos + i);
        const uint32_t orig = __float_as_uint(p.w);
        const float my = __ldg(s_score + i);
        const bool owned = !s_role || ((s_role[i] & 3) == 3);
        if (PASS == 0) {
            above = owned && isfinite(my) && !((double)my < th);
            near = owned && isfinite(my) && fabs((double)my - th) <= 1e-5;
        }
        const bool work = PASS == 0 ? above : (owned && s_state[i] == 2);
        if (work) {
            int cx, cy, cz;
            key_to_cell_n(__ldg(skey + i), dimx, dimy, cx, cy, cz);
            const int z0 = max(cz - reach, 0), z1 = min(cz + reach, dimz - 1);
            const int y0 = max(cy - reach, 0), y1 = min(cy + reach, dimy - 1);
            const int x0 = max(cx - reach, 0), x1 = min(cx + reach, dimx - 1);
            bool is_max = true, has_draw = false, close_draw = false;   // PASS 0
            bool lower_active = false, lower_undecided = false;         // PASS 1
            const uint32_t my_order = PASS == 1 && gidx ? (uint32_t)__ldg(gidx + orig) : orig;
            for (int z = z0; z <= z1 && is_max; ++z)
                for (int y = y0; y <= y1 && is_max; ++y) {
                    const int64_t base = ((int64_t)z * dimy + y) * dimx;
                    const int s = __ldg(cell_start + base + x0), e = __ldg(cell_start + base + x1 + 1);
                    for (int j = s; j < e; ++j) {
                        const float4 c = __ldg(s_pos + j);
                        if (!(dist2(p.x, p.y, p.z, c.x, c.y, c.z) < rn2)) continue;
                        const float sj = __ldg(s_score + j);
                        if (PASS == 0) {
                            if (my < sj) { is_max = false; break; }
                            if (my == sj && j != i) {
                                has_draw = true;
                                if (draw_distance(p, c) < draws_thr) close_draw = true;
                            }
                        } else if (my == sj && (gidx ? (uint32_t)__ldg(gidx + __float_as_uint(c.w)) : __float_as_uint(c.w)) < my_order &&
                                   draw_distance(p, c) < draws_thr) {
                            // a lower-index close draw: active (1) skips this point, undecided (2) postpones it;
                            // a close draw that is a keypoint without draws cannot exist (it ties with this point)
                            const uint8_t st = s_state[j];
                            if (st == 1) lower_active = true;
                            else if (st == 2) lower_undecided = true;
                        }
                    }
                }
            if (PASS == 0) s_state[i] = !is_max ? 0 : (!has_draw ? 1 : (close_draw ? 2 : 0));
            else if (lower_active) s_state[i] = 3;
            else if (!lower_undecided) s_state[i] = 1;
            else atomicAdd(counters + 6, 1ull);       // still undecided: another round is needed
        } else if (PASS == 0) s_state[i] = 0;
    }
    if (PASS == 0) {
        unsigned m = __ballot_sync(0xFFFFFFFFu, above);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(counters + 2, (unsigned long long)__popc(m));
        m = __ballot_sync(0xFFFFFFFFu, near);
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(counters + 7, (unsigned long long)__popc(m));
    }
}

__global__ void __launch_bounds__(256) state_to_flag_kernel(const float4* __restrict__ s_pos, const uint8_t* __restrict__ s_role,
                                                            const uint8_t* __restrict__ s_state, int n, uint8_t* __restrict__ flag)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[__float_as_uint(__ldg(&s_pos[i].w))] = s_state[i] == 1 && (!s_role || (s_role[i] & 3) == 3) ? 1 : 0;
}

cudaError_t launch_nms_draws_classify(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th)
{
    const kpl_params& U = c->params;
    cudaError_t e;
    if ((e = ensure(c->flag, n)) || (e = ensure(c->s_state, n))) return e;
    const double rn = (double)U.radius_nms;
    nms_draws_kernel<0><<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->s_pos.p, s_score, c->key_b.p, c->cell_start.p,
                                                                              use_role ? c->s_role.p : nullptr, c->grid.dim[0], c->grid.dim[1],
                                                                              c->grid.dim[2], (int)n, (float)(rn * rn), c->grid.reach_nms,
                                                                              th, U.draws_threshold, nullptr, c->s_state.p, c->counters.p);
    c->launches++;
    return cudaGetLastError();
}

// one resolution round; counters[6] = candidates left undecided by it
cudaError_t launch_nms_draws_round(kpl_ctx* c, int64_t n, bool use_role, const int32_t* gidx, const float* s_score, double th)
{
    const kpl_params& U = c->params;
    cudaError_t e;
    if ((e = cudaMemsetAsync(c->counters.p + 6, 0, sizeof(unsigned long long), c->stream))) return e;
    const double rn = (double)U.radius_nms;
    nms_draws_kernel<1><<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->s_pos.p, s_score, c->key_b.p, c->cell_start.p,
                                                                              use_role ? c->s_role.p : nullptr, c->grid.dim[0], c->grid.dim[1],
                                                                              c->grid.dim[2], (int)n, (float)(rn * rn), c->grid.reach_nms,
                                                                              th, U.draws_threshold, gidx, c->s_state.p, c->counters.p);
    c->launches++;
    c->stats.nms_rounds++;
    return cudaGetLastError();
}

cudaError_t launch_nms_draws_flags(kpl_ctx* c, int64_t n, bool use_role, int64_t flag_off)
{
    cudaError_t e;
    if ((e = ensure(c->flag, (size_t)(flag_off + n)))) return e;
    state_to_flag_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->s_pos.p, use_role ? c->s_role.p : nullptr, c->s_state.p,
                                                                            (int)n, c->flag.p + flag_off);
    c->launches++;
    return cudaGetLastError();
}

// A whole cloud, or a batch of views: each view is a connected component of its own (§5.4 padding layers) that keeps its
// own index order inside the concatenation, so the rounds over the stacked grid resolve every view at once.
cudaError_t launch_nms_draws(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th, int64_t flag_off)
{
    cudaError_t e;
    if ((e = launch_nms_draws_classify(c, n, use_role, s_score, th))) return e;
    for (int round = 0; round < nms_round_cap(n); ++round) {
        if ((e = launch_nms_draws_round(c, n, use_role, nullptr, s_score, th))) return e;
        unsigned long long undecided = 0;
        if ((e = cudaMemcpyAsync(&undecided, c->counters.p + 6, sizeof undecided, cudaMemcpyDeviceToHost, c->stream))) return e;
        if ((e = cudaStreamSynchronize(c->stream))) return e;
        c->syncs++;
        if (undecided == 0) break;
    }
    return launch_nms_draws_flags(c, n, use_role, flag_off);
}

// setNonMaxima(false) (hpp:189-196): every scored point is a keypoint.
__global__ void __launch_bounds__(256) all_flags_kernel(const float* __restrict__ score, int64_t n, uint8_t* __restrict__ flag)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) flag[i] = isnan(score[i]) ? 0 : 1;
}
cudaError_t launch_all_flags(kpl_ctx* c, int64_t n, const float* score, int64_t flag_off)
{
    cudaError_t e;
    if ((e = ensure(c->flag, (size_t)(flag_off + n)))) return e;
    all_flags_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(score, n, c->flag.p + flag_off);
    c->launches++;
    return cudaGetLastError();
}

// ---- plain radius search (FLANN radiusSearch semantics: d2 < (float)(r*r), self included) -----
static constexpr unsigned long long HASH_MUL = 0x9E3779B97F4A7C15ull;

template <bool LISTS>
__global__ void __launch_bounds__(128)
radius_kernel(const float4* __restrict__ s_pos, const uint32_t* __restrict__ skey, const int32_t* __restrict__ cell_start,
              const int32_t* __restrict__ inv_or_queries, int dimx, int dimy, int dimz, int n, int64_t m, float r2, int reach,
              int32_t* __restrict__ counts, unsigned long long* __restrict__ hash,
              const int64_t* __restrict__ offsets, int32_t* __restrict__ indices)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= m) return;
    // LISTS: t indexes the query list, inv_or_queries[t] is the SORTED position of that query.
    const int i = LISTS ? inv_or_queries[t] : (int)t;
    const float4 p = __ldg(s_pos + i);
    int cx, cy, cz;
    key_to_cell_n(__ldg(skey + i), dimx, dimy, cx, cy, cz);
    const int z0 = max(cz - reach, 0), z1 = min(cz + reach, dimz - 1);
    const int y0 = max(cy - reach, 0), y1 = min(cy + reach, dimy - 1);
    const int x0 = max(cx - reach, 0), x1 = min(cx + reach, dimx - 1);
    int cnt = 0;
    unsigned long long h = 0;
    int64_t w = LISTS ? offsets[t] : 0;
    for (int z = z0; z <= z1; ++z)
        for (int y = y0; y <= y1; ++y) {
            const int64_t base = ((int64_t)z * dimy + y) * dimx;
            const int s = __ldg(cell_start + base + x0), e = __ldg(cell_start + base + x1 + 1);
            for (int j = s; j < e; ++j) {
                const float4 c = __ldg(s_pos + j);
                if (dist2(p.x, p.y, p.z, c.x, c.y, c.z) < r2) {
                    const uint32_t oj = __float_as_uint(c.w);
                    if (LISTS) indices[w++] = (int32_t)oj;
                    cnt++;
                    h += ((unsigned long long)oj + 1ull) * HASH_MUL;
                }
            }
        }
    if (!LISTS) {
        const uint32_t orig = __float_as_uint(p.w);
        if (counts) counts[orig] = cnt;
        if (hash) hash[orig] = h;
    }
}

// ---- nearest cloud point of arbitrary query points ------------------------------------------------------
// pcl::KdTreeFLANN::nearestKSearch(point, 1, ...) as TrainDetector uses it to snap its positive / negative
// samples onto cloud indices before computePointsForTrainingFeatures (src/main_train_detector.cpp:419-436).
// One thread per query: shells of cells around the query's (clamped) cell until the best squared distance is
// provably smaller than anything outside the scanned block; ties go to the lower index.
__global__ void __launch_bounds__(128)
nearest_kernel(const float4* __restrict__ s_pos, const int32_t* __restrict__ cell_start, GridDesc g, const float4* __restrict__ queries,
               int64_t m, int32_t* __restrict__ idx_out, float* __restrict__ d2_out)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= m) return;
    const float4 q = __ldg(queries + t);
    const float v[3] = {q.x, q.y, q.z};
    int c[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double f = floor(__ddiv_rn(__dsub_rn((double)v[a], g.org[a]), g.cell)) - (double)g.off[a];
        f = fmin(fmax(f, 0.0), (double)(g.dim[a] - 1));
        c[a] = isfinite(v[a]) ? (int)f : 0;
    }
    float best = CUDART_INF_F;
    uint32_t bidx = 0xFFFFFFFFu;
    auto scan = [&](int z, int y, int x0, int x1) {
        x0 = max(x0, 0); x1 = min(x1, g.dim[0] - 1);
        if (z < 0 || z >= g.dim[2] || y < 0 || y >= g.dim[1] || x0 > x1) return;
        const int64_t base = ((int64_t)z * g.dim[1] + y) * g.dim[0];
        const int s = __ldg(cell_start + base + x0), e = __ldg(cell_start + base + x1 + 1);
        for (int j = s; j < e; ++j) {
            const float4 p = __ldg(s_pos + j);
            const float d2 = dist2(q.x, q.y, q.z, p.x, p.y, p.z);
            const uint32_t oi = __float_as_uint(p.w);
            if (d2 < best || (d2 == best && oi < bidx)) { best = d2; bidx = oi; }
        }
    };
    const int maxdim = max(g.dim[0], max(g.dim[1], g.dim[2]));
    for (int R = 0; R <= maxdim; ++R) {
        for (int z = c[2] - R; z <= c[2] + R; ++z)
            for (int y = c[1] - R; y <= c[1] + R; ++y) {
                if (abs(z - c[2]) == R || abs(y - c[1]) == R) scan(z, y, c[0] - R, c[0] + R);      // a face row of the shell
                else { scan(z, y, c[0] - R, c[0] - R); if (R > 0) scan(z, y, c[0] + R, c[0] + R); }   // its two end cells
            }
        if (bidx != 0xFFFFFFFFu) {
            double guard = (double)R * g.cell;
            guard = guard * guard * (1.0 - 1e-6);
            if ((double)best < guard) break;
        }
    }
    idx_out[t] = (int32_t)bidx;
    if (d2_out) d2_out[t] = best;
}

cudaError_t launch_nearest(kpl_ctx* c, const float4* d_queries, int64_t m, int32_t* d_idx, float* d_d2)
{
    if (m == 0) return cudaSuccess;
    nearest_kernel<<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(c->s_pos.p, c->cell_start.p, c->grid, d_queries, m, d_idx, d_d2);
    c->launches++;
    return cudaGetLastError();
}

static int reach_for(const GridDesc& g, double radius)
{
    return (int)floor(radius * (1.0 + 4.76837158203125e-07) / g.cell) + 1;
}

cudaError_t launch_radius_stats(kpl_ctx* c, int64_t n, double radius, int32_t* d_counts, unsigned long long* d_hash)
{
    radius_kernel<false><<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(
        c->s_pos.p, c->key_b.p, c->cell_start.p, nullptr, c->grid.dim[0], c->grid.dim[1], c->grid.dim[2], (int)n, n,
        (float)(radius * radius), reach_for(c->grid, radius), d_counts, d_hash, nullptr, nullptr);
    c->launches++;
    return cudaGetLastError();
}

// d_queries holds SORTED positions of the m queries; d_offsets[m+1] their output offsets.
cudaError_t launch_radius_lists(kpl_ctx* c, int64_t n, double radius, const int32_t* d_queries, int64_t m,
                                const int64_t* d_offsets, int32_t* d_indices)
{
    if (m == 0) return cudaSuccess;
    radius_kernel<true><<<(unsigned)((m + 127) / 128), 128, 0, c->stream>>>(
        c->s_pos.p, c->key_b.p, c->cell_start.p, d_queries, c->grid.dim[0], c->grid.dim[1], c->grid.dim[2], (int)n, m,
        (float)(radius * radius), reach_for(c->grid, radius), nullptr, nullptr, d_offsets, d_indices);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace kpl
