// kpl_internal.h -- shared declarations of the CUDA implementation behind include/kpl.h.
// Built for sm_100a only, with -fmad=false: every float expression below is evaluated with
// separately rounded multiplies and adds, which is the arithmetic contract of the hot path
// (FLANN L2_Simple / Eigen / the reference's own helpers are FMA-free on the authors' platform).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/kpl.h"

namespace kpl {

// Canonical uniform grid.  cell = r_feat*(1+2^-20)/cells_per_radius; coordinates are computed in
// double so that two points closer than r_feat are never more than cells_per_radius cells apart.
// A batch of independent views (kpl_detect_batch) shares ONE grid: every view keeps the cells of its own
// canonical grid (origin = its bounding-box minimum) and the views are stacked along z with empty padding
// layers between them, so no kernel ever pairs points of two views and the (cell key, index) order inside a
// view is the one of its stand-alone run.
struct ViewDesc {
    double org[3];        // the view's own grid origin
    int32_t zoff, dimz;   // first stacked z layer / number of layers of the view
};
struct GridDesc {
    double org[3];
    double cell;
    int32_t dim[3];
    int32_t off[3];       // cell offset of a forced (slab) grid, 0 otherwise
    int32_t reach_feat;   // cells to search for radius_features
    int32_t reach_nms;    // cells to search for radius_nms
    int64_t ncells;
    // batch of views (nullptr / 0 for a single cloud)
    const ViewDesc* views;          // device, nviews entries
    const int32_t* layer_view;      // device, dim[2] entries: view of a stacked z layer, -1 = padding
    const int64_t* view_offsets;    // device, nviews + 1 entries: first point of each view
    int32_t nviews;
    // slab of a larger cloud: the x faces of the local grid that are NOT faces of the global grid.  A k-NN
    // search that would have to look beyond such a face cannot be exact (normals.cu)
    int32_t interior_lo, interior_hi;
    int32_t guard_cells;  // points in the outermost guard_cells columns next to an interior face are expected to be clipped
    int32_t forced;       // 1: a ForcedGrid, whose points no bounding-box pass has checked (grid.cu: cell_key_kernel flags them)
};

// A grid given by the caller (a slab of a larger cloud) instead of the canonical grid of the cloud's bounding box
struct ForcedGrid {
    double origin[3];                                // the GLOBAL origin: a point's cell is floor((v - origin) / cell) - offset
    int32_t dims[3], offset[3];
    int32_t interior_lo, interior_hi, guard_cells;   // as in GridDesc
};

// One forest node, 8 bytes: thr_or_value + packed(child_block_offset << 10 | var); var == 1023 => leaf.
// Nodes are grouped in 32-byte blocks {node, left child, right child, unused}: see pack_forest (forest.cu).
struct __align__(8) PackedNode {
    float thr;
    uint32_t packed;
};
static constexpr uint32_t KPL_LEAF_VAR = 1023u;

struct ForestInfo {
    int32_t ntrees = 0, nnodes = 0, var_count = 0, max_depth = 0;
    int32_t max_var = -1;                 // largest variable index any split reads (checked against annuli*bins per call)
};

// The loaded forests: forest 0 (kpl_load_forest / kpl_set_forest, which every entry point scores with) and the ones
// kpl_add_forest* appended, concatenated into one node array.  pack_forest's child offsets are relative, so a forest moves
// by shifting its roots by the blocks before it; desc[k] = (first root of forest k, its tree count).  Empty: no forest loaded.
struct ForestSet {
    std::vector<ForestInfo> info;
    std::vector<PackedNode> nodes;        // host copy of the concatenation
    std::vector<int32_t> roots;           // shifted roots, forest after forest
    std::vector<int2> desc;
    PackedNode* d_nodes = nullptr;
    int32_t* d_roots = nullptr;
    int2* d_desc = nullptr;
};

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
};

struct HostForestArrays {
    std::vector<int32_t> roots, var, left, right;
    std::vector<float> thr, value;
    int32_t var_count = 0;
};

// forest_yaml.cpp
int parse_forest_yaml(const char* path, HostForestArrays& out, std::string& err);

}  // namespace kpl

struct kpl_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    kpl_params params;
    kpl::ForestSet forests;
    kpl::GridDesc grid;
    kpl_timings timings;
    kpl_stats stats;
    std::string err;
    int launches = 0;

    // device buffers (grown on demand, never shrunk)
    kpl::DevBuf<float4> in_xyz, in_nrm;          // staged host input (host API only)
    kpl::DevBuf<uint8_t> in_role, s_role;
    kpl::DevBuf<uint32_t> key_a, key_b, idx_a, idx_b;
    kpl::DevBuf<uint8_t> cub_tmp;
    kpl::DevBuf<int32_t> cell_start;
    kpl::DevBuf<int32_t> row_warps_n, row_offset_n;   // normal kernels' work list: warps per cell row and their prefix sum
    int nwarps_norm = 0, nwarps_feat = 0;         // sizes of work_n / warp_starts for the grid in place
    kpl::DevBuf<int2> work_n;                     // (first sorted position, count <= 32) per warp of the normal kernels
    // feature kernel: queries (sorted positions) in Hilbert order of a sub-cell lattice, 32 consecutive ones per warp
    // (grid.cu: build_lists); warp w takes entries [warp_starts[w], warp_starts[w + 1]) of the order.  _all / _n: every
    // point (cooperative k-NN normals; the feature kernel too when no roles are given), _role: the points with a scoring role
    kpl::DevBuf<uint64_t> ckey_a, ckey_b;
    kpl::DevBuf<int32_t> qorder_a, qorder_all, warp_starts_n, qorder_role, warp_starts_role;
    const int32_t* qorder_f = nullptr;            // the feature kernel's list for the grid in place (one of the above)
    const int32_t* warp_starts_f = nullptr;
    kpl::DevBuf<uint32_t> warp_order;             // launch order of the warps, most expensive first (few-wave launches)
    bool have_warp_order = false;
    kpl::DevBuf<float4> s_pos, s_nrm;            // cell-sorted positions (w = original index bits) / normals
    kpl::DevBuf<float> feat;                     // n x F, sorted order
    kpl::DevBuf<float> s_score, score;           // sorted order / original order
    kpl::DevBuf<uint8_t> flag;                   // keypoint flag, original order
    kpl::DevBuf<uint8_t> fragile;                // near-split flag of the forest walk, original order (forest.cuh)
    // kpl_detect_forests / kpl_detect_batch_forests (and the organized batch's inner batch): scores, flags and fragile flags
    // hold K x n entries, forest-major.  range_off = the K*V + 1 boundaries {k*n + view_offsets[v]} of the (forest, view)
    // ranges of the keypoint list (host copy kept for the asynchronous upload); a single cloud is V = 1
    kpl::DevBuf<int64_t> range_off;
    std::vector<int64_t> range_off_h;
    kpl::DevBuf<kpl::ViewDesc> views;            // kpl_detect_batch: per-view grids
    kpl::DevBuf<int32_t> layer_view;
    kpl::DevBuf<int64_t> view_offsets;
    kpl::DevBuf<int32_t> qlist;                  // kpl_features with an index subset: sorted positions of the queries
    kpl::DevBuf<uint8_t> s_state;                // draws-remove NMS state, sorted order
    kpl::DevBuf<int32_t> kp_idx;
    kpl::DevBuf<float> scratch_f;                // fetch / reorder scratch
    kpl::DevBuf<int32_t> scratch_i;
    // kpl_detect_batch_organized: finite-pixel flags, compact index -> pixel index (frame f's pixel p is f*width*height + p),
    // the compacted positions / normals the detection runs on, the frames' first compacted points (+ their count), the
    // per-frame viewpoints, and the pixel-order scores / frame keypoint offsets of the host entry point
    kpl::DevBuf<uint8_t> org_flag;
    kpl::DevBuf<int32_t> org_pix;
    kpl::DevBuf<float4> org_xyz, org_nrm;
    kpl::DevBuf<int64_t> org_frame_off, org_kp_off;
    kpl::DevBuf<float> org_vp, org_score;
    // [0] feature pairs [1] candidate pairs [2] above th [3] n_kp [4] unscored [5] scored [6] scratch [7] near threshold
    // [8] fragile points [9] clipped k-NN searches (slab edge) [10] scratch [11..15] sizes of the query lists (grid.cu: build_lists)
    kpl::DevBuf<unsigned long long> counters;
    static constexpr int NCOUNTERS = 16;
    int syncs = 0;                               // cudaStreamSynchronize calls of the call in flight
    const float4* cur_xyz = nullptr;             // original-order inputs of the call in flight (device)
    const float4* cur_nrm = nullptr;
    float* d_bbox = nullptr;                     // 6 ordered-int encoded floats + flags
    int64_t last_n = 0;
    int last_F = 0;
    int last_nforests = 1;                       // forests scored by the last call (the fragile mask holds last_nforests x n bytes)
    bool last_has_normals = false, last_has_features = false, last_has_fragile = false;
    bool fast_math = false;                      // feature kernel variant chosen by the arithmetic self-test
    bool keep_intermediates = false;             // kpl_set_keep_intermediates: materialise feature rows in kpl_detect*
    cudaEvent_t ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

namespace kpl {

// ---- launch wrappers implemented in the .cu files; all enqueue on ctx->stream and return cudaError_t
cudaError_t launch_bbox(kpl_ctx* c, const float4* xyz, int64_t n, float* d_bbox /* 8 uint32 */);
cudaError_t build_grid(kpl_ctx* c, const float4* xyz, const float4* nrm_or_null, const uint8_t* role_or_null, int64_t n);
cudaError_t launch_normals_knn(kpl_ctx* c, int64_t n);
cudaError_t launch_normals_radius(kpl_ctx* c, int64_t n);
cudaError_t launch_flip_normals(kpl_ctx* c, int64_t n);
cudaError_t launch_check_normals(kpl_ctx* c, int64_t n, bool use_role);
bool normals_knn_uses_work_list(const kpl_params& P);
cudaError_t launch_bbox_init(kpl_ctx* c);
cudaError_t launch_gather_keypoints(kpl_ctx* c, const float4* d_xyz, const int32_t* d_kp_idx, int64_t nkp, float4* d_out);
// nframes frames of W x H pixels; d_viewpoints: NULL (params.viewpoint) or 3 device floats per frame
cudaError_t launch_normals_integral_image(kpl_ctx* c, const float4* d_xyz, int W, int H, int nframes, float smoothing_size,
                                          const float* d_viewpoints, float4* d_out);
// organized frames (n pixels each) -> finite pixels in ascending order (org_pix) and org_frame_off; d_scores (NULL or
// nforests x nframes * n floats, forest-major) is set to NaN
cudaError_t launch_organized_select(kpl_ctx* c, const float4* d_xyz, int64_t n, int nframes, int nforests, float* d_scores);
// the m selected pixels' positions and normals (per pixel) -> org_xyz / org_nrm
cudaError_t launch_organized_gather(kpl_ctx* c, const float4* d_xyz, const float4* d_nrm, int64_t m);
// after the detection of the m compacted points by nforests forests (forest-major K x m scores, keypoints ascending in
// [0, K*m)): scores to pixel order (forest k's at k * nframes * n), keypoints (in place) to frame-local pixel indices,
// (forest, frame) keypoint offsets (nforests * nframes + 1)
cudaError_t launch_organized_map_back(kpl_ctx* c, int64_t m, int64_t n, int nframes, int nforests, float* d_scores, int32_t* d_kp,
                                      int64_t* d_kp_off);
cudaError_t build_lists(kpl_ctx* c, int64_t n, int span_n, bool curve_normals, bool want_features, bool use_role, int64_t longest_first_below);
cudaError_t launch_count_occupied_cells(kpl_ctx* c, int64_t n, unsigned long long* d_out);
cudaError_t build_query_list(kpl_ctx* c, int64_t n, const int32_t* d_indices, int64_t m);
cudaError_t launch_scatter_rows(kpl_ctx* c, const float* d_rows, int64_t m, int width, float* d_out);
cudaError_t launch_view_ranges(kpl_ctx* c, int64_t n, int32_t* d_kp_idx, const int64_t* d_view_offsets, int nviews, int64_t* d_kp_offsets);
cudaError_t launch_bbox_views(kpl_ctx* c, const float4* xyz, int64_t n, const int64_t* d_view_offsets, int nviews, uint32_t* d_bbox);
// nforests: forests 0 .. nforests - 1 of c->forests are scored in the kernel's tail (0: features only, kpl_features).
// qlist != nullptr: features of the m_list listed sorted positions only (rows in list order, c->feat holds m_list x F).
cudaError_t launch_features(kpl_ctx* c, int64_t n, bool use_role, int nforests, bool store_rows, const int32_t* d_qlist = nullptr, int64_t m_list = 0);
// Threshold + NMS of one forest's n sorted scores s_score (th compared in double); the keypoint flags (original order) go to
// c->flag.p + flag_off.  kpl_detect* pass c->s_score.p, params.threshold and 0; kpl_detect_forests forest k's slice.
cudaError_t launch_nms(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th, int64_t flag_off);
cudaError_t launch_nms_draws(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th, int64_t flag_off);
// the pieces of launch_nms_draws, for a caller that exchanges halo states between rounds (shard.cu); gidx: global index of
// every local original index (nullptr: the identity)
cudaError_t launch_nms_draws_classify(kpl_ctx* c, int64_t n, bool use_role, const float* s_score, double th);
cudaError_t launch_nms_draws_round(kpl_ctx* c, int64_t n, bool use_role, const int32_t* gidx, const float* s_score, double th);
cudaError_t launch_nms_draws_flags(kpl_ctx* c, int64_t n, bool use_role, int64_t flag_off);
// setNonMaxima(false): every scored point of the n original-order scores is a keypoint
cudaError_t launch_all_flags(kpl_ctx* c, int64_t n, const float* score, int64_t flag_off);
// resolution rounds of a cloud of n points never exceed this cap (the lowest undecided index resolves in every round)
inline int nms_round_cap(int64_t n) { return (int)(n < (1 << 20) ? n : (1 << 20)); }
cudaError_t launch_compact(kpl_ctx* c, int64_t n, int32_t* d_kp_idx_out);

cudaError_t uniform_sample(kpl_ctx* c, const float4* xyz, int64_t n, float leaf, const float mn[3], const float mx[3],
                           int32_t* d_idx_out, std::string& err);
cudaError_t launch_nearest(kpl_ctx* c, const float4* d_queries, int64_t m, int32_t* d_idx, float* d_d2);
cudaError_t launch_radius_stats(kpl_ctx* c, int64_t n, double radius, int32_t* d_counts, unsigned long long* d_hash);
cudaError_t launch_radius_lists(kpl_ctx* c, int64_t n, double radius, const int32_t* d_queries, int64_t m,
                                const int64_t* d_offsets, int32_t* d_indices);
cudaError_t launch_unsort_rows(kpl_ctx* c, const float* d_sorted_rows, int64_t n, int width, float* d_out_orig_order);
cudaError_t launch_unsort_normals(kpl_ctx* c, int64_t n, float4* d_out_orig_order);

// canonical grid (capi.cu): the cell of kpl_params, the cells spanned by a bounding box [lo, hi], the cells a search
// of `radius` has to visit on each side.  The same expressions make a slab plan the grid of the unsharded run.
double canonical_cell(const kpl_params& P);
int32_t grid_dim(double lo, double hi, double cell);
int grid_reach(double radius, double cell);

// detection phases (capi.cu), shared with the slab-sharded driver (shard.cu); all but detect_reset return kpl_status
void detect_reset(kpl_ctx* ctx);
// nforests: the call scores forests 0 .. nforests - 1 (the *_forests entry points: all of them; every other entry point: 1).
// with_role: a caller-supplied role array (kpl_detect*), which rules out draws-remove NMS; the kpl_shard_* driver passes false
int detect_check(kpl_ctx* ctx, int64_t n, int nforests, bool with_role);
int detect_begin(kpl_ctx* ctx);
// forced == nullptr: the canonical grid of the cloud's bounding box; cell_override > 0 replaces the canonical cell
int prepare_grid(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, const uint8_t* d_role, int64_t n, const ForcedGrid* forced, double cell_override = 0.0);
// scores of forests 0 .. nforests - 1, forest-major
int detect_score_phase(kpl_ctx* ctx, bool normals_given, bool use_role, int64_t n, int nforests);
// threshold + NMS of each of the nforests forest-major score slices (thresholds: NULL = params.threshold, else one per
// forest), then one compaction of the nforests x n flags into an ascending list of indices in [0, nforests * n)
int detect_nms_phase(kpl_ctx* ctx, bool use_role, int64_t n, int nforests, const double* thresholds, int32_t* d_kp_out);
int detect_finish(kpl_ctx* ctx, int64_t n, int64_t* n_kp_out);

template <typename T>
cudaError_t ensure(DevBuf<T>& b, size_t n)
{
    if (n <= b.cap) return cudaSuccess;
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
    size_t want = n + n / 8 + 64;
    cudaError_t e = cudaMalloc((void**)&b.p, want * sizeof(T));
    if (e == cudaSuccess) b.cap = want;
    return e;
}

}  // namespace kpl
