// capi.cu -- the extern "C" surface declared in include/kpl.h and the stage orchestration.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include "kpl_internal.h"

namespace kpl {
int pack_forest(const HostForestArrays& in, std::vector<PackedNode>& nodes, std::vector<int32_t>& roots, int& max_depth, int& max_var, std::string& err);
}
using namespace kpl;

#define KPL_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            char b__[512];                                                                          \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            ctx->err = b__;                                                                         \
            return e__ == cudaErrorMemoryAllocation ? KPL_E_NOMEM : KPL_E_CUDA;                     \
        }                                                                                           \
    } while (0)

static int fail(kpl_ctx* ctx, int code, const std::string& msg)
{
    ctx->err = msg;
    return code;
}

static float dec_float(uint32_t u)
{
    uint32_t b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    float f;
    memcpy(&f, &b, 4);
    return f;
}

template <typename T>
static void release(DevBuf<T>& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

static void free_forest_set(ForestSet& S)
{
    if (S.d_nodes) cudaFree(S.d_nodes);
    if (S.d_roots) cudaFree(S.d_roots);
    if (S.d_desc) cudaFree(S.d_desc);
    S = ForestSet();
}

extern "C" {

const char* kpl_version(void) { return "kpl-b200 0.1 (sm_100a)"; }

int kpl_device_count(void)
{
    int count = 0, usable = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    for (int d = 0; d < count; ++d) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) usable++;
    }
    return usable;
}

int kpl_params_default(kpl_params* p)
{
    if (!p) return KPL_E_INVALID;
    memset(p, 0, sizeof *p);
    p->radius_features = 20.f;
    p->radius_nms = 4.f;
    p->threshold = (double)0.85f;
    p->n_annulus = 5;
    p->n_bins = 10;
    p->non_maxima = 1;
    p->draws_remove = 0;
    p->draws_threshold = 0.f;
    p->normals_mode = KPL_NORMALS_KNN;
    p->k_normals = 10;
    p->flip_normals = 0;
    p->cells_per_radius = 4;
    p->grid_forced = 0;
    p->slab_interior_lo = p->slab_interior_hi = 0;
    p->slab_guard_cells = 0;
    p->slab_owned_lo = p->slab_owned_hi = 0;
    p->uniform_sampling_centre = 0;
    p->eigen32_normalize = 0;
    p->report_fragile = 0;
    return KPL_OK;
}

int kpl_create(int device, kpl_ctx** out)
{
    if (!out) return KPL_E_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return KPL_E_CUDA;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return KPL_E_CUDA;
    if (prop.major != 10) return KPL_E_CUDA;   // sm_100a cubin only: no fallback path exists
    if (cudaSetDevice(device) != cudaSuccess) return KPL_E_CUDA;
    kpl_ctx* ctx = new (std::nothrow) kpl_ctx();
    if (!ctx) return KPL_E_NOMEM;
    ctx->device = device;
    kpl_params_default(&ctx->params);
    memset(&ctx->timings, 0, sizeof ctx->timings);
    memset(&ctx->stats, 0, sizeof ctx->stats);
    bool ok = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) == cudaSuccess;
    ctx->stream = ctx->own_stream;
    for (int i = 0; ok && i < 8; ++i) ok = cudaEventCreate(&ctx->ev[i]) == cudaSuccess;
    ok = ok && cudaMalloc((void**)&ctx->d_bbox, 8 * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && ensure(ctx->counters, kpl_ctx::NCOUNTERS) == cudaSuccess;
    if (!ok) { kpl_destroy(ctx); return KPL_E_CUDA; }
    *out = ctx;
    return KPL_OK;
}

void kpl_destroy(kpl_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    release(ctx->in_xyz); release(ctx->in_nrm); release(ctx->in_role); release(ctx->s_role);
    release(ctx->key_a); release(ctx->key_b); release(ctx->idx_a); release(ctx->idx_b); release(ctx->cub_tmp);
    release(ctx->row_warps_n); release(ctx->row_offset_n); release(ctx->fragile); release(ctx->views); release(ctx->layer_view);
    release(ctx->view_offsets); release(ctx->qlist);
    release(ctx->cell_start); release(ctx->work_n); release(ctx->ckey_a); release(ctx->ckey_b); release(ctx->qorder_a); release(ctx->qorder_all); release(ctx->warp_starts_n); release(ctx->qorder_role); release(ctx->warp_starts_role);
    release(ctx->warp_order); release(ctx->s_pos); release(ctx->s_nrm); release(ctx->feat);
    release(ctx->s_score); release(ctx->score); release(ctx->flag); release(ctx->s_state); release(ctx->kp_idx);
    release(ctx->scratch_f); release(ctx->scratch_i); release(ctx->counters);
    release(ctx->org_flag); release(ctx->org_pix); release(ctx->org_xyz); release(ctx->org_nrm); release(ctx->org_frame_off);
    release(ctx->kp_off); release(ctx->org_vp); release(ctx->org_score);
    if (ctx->d_bbox) cudaFree(ctx->d_bbox);
    free_forest_set(ctx->forests);
    release(ctx->range_off);
    for (int i = 0; i < 8; ++i) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* kpl_last_error(const kpl_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int kpl_set_stream(kpl_ctx* ctx, void* s)
{
    if (!ctx) return KPL_E_INVALID;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return KPL_OK;
}

int kpl_set_keep_intermediates(kpl_ctx* ctx, int on)
{
    if (!ctx) return KPL_E_INVALID;
    ctx->keep_intermediates = on != 0;
    return KPL_OK;
}

int kpl_set_params(kpl_ctx* ctx, const kpl_params* p)
{
    if (!ctx || !p) return KPL_E_INVALID;
    if (!(p->radius_features > 0.f) || !std::isfinite(p->radius_features)) return fail(ctx, KPL_E_INVALID, "radius_features must be > 0");
    if (p->radius_nms < 0.f || !std::isfinite(p->radius_nms)) return fail(ctx, KPL_E_INVALID, "radius_nms must be >= 0");
    if (p->n_annulus < 1 || p->n_bins < 1 || (int64_t)p->n_annulus * p->n_bins > 1022) return fail(ctx, KPL_E_INVALID, "annuli*bins must be in [1,1022]");
    if (p->normals_mode < 0 || p->normals_mode > 2) return fail(ctx, KPL_E_INVALID, "bad normals_mode");
    if (p->k_normals < 1 || p->k_normals > 64) return fail(ctx, KPL_E_INVALID, "k_normals must be in [1,64]");
    if (p->cells_per_radius < 1 || p->cells_per_radius > 16) return fail(ctx, KPL_E_INVALID, "cells_per_radius must be in [1,16]");
    ctx->params = *p;
    return KPL_OK;
}

int kpl_get_params(const kpl_ctx* ctx, kpl_params* p)
{
    if (!ctx || !p) return KPL_E_INVALID;
    *p = ctx->params;
    return KPL_OK;
}

// Uploads a forest set (host arrays complete) and replaces ctx->forests with it; on failure ctx->forests is left as it was.
static int upload_forest_set(kpl_ctx* ctx, ForestSet& S)
{
    S.d_nodes = nullptr; S.d_roots = nullptr; S.d_desc = nullptr;
    cudaError_t e = cudaMalloc((void**)&S.d_nodes, S.nodes.size() * sizeof(PackedNode));
    if (!e) e = cudaMalloc((void**)&S.d_roots, S.roots.size() * sizeof(int32_t));
    if (!e) e = cudaMalloc((void**)&S.d_desc, S.desc.size() * sizeof(int2));
    if (!e) e = cudaMemcpy(S.d_nodes, S.nodes.data(), S.nodes.size() * sizeof(PackedNode), cudaMemcpyHostToDevice);
    if (!e) e = cudaMemcpy(S.d_roots, S.roots.data(), S.roots.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (!e) e = cudaMemcpy(S.d_desc, S.desc.data(), S.desc.size() * sizeof(int2), cudaMemcpyHostToDevice);
    if (e) {
        cudaFree(S.d_nodes); cudaFree(S.d_roots); cudaFree(S.d_desc);
        return fail(ctx, e == cudaErrorMemoryAllocation ? KPL_E_NOMEM : KPL_E_CUDA, std::string("forest set upload: ") + cudaGetErrorString(e));
    }
    free_forest_set(ctx->forests);
    ctx->forests = std::move(S);
    return KPL_OK;
}

// Appends a packed forest to a copy of the set: its roots shifted by the blocks already there (child offsets are relative)
static void append_forest(ForestSet& S, const ForestInfo& info, const std::vector<PackedNode>& nodes, const std::vector<int32_t>& roots)
{
    const int32_t shift = (int32_t)(S.nodes.size() / 4);
    S.desc.push_back(make_int2((int)S.roots.size(), (int)roots.size()));
    for (int32_t r : roots) S.roots.push_back(r + shift);
    S.nodes.insert(S.nodes.end(), nodes.begin(), nodes.end());
    S.info.push_back(info);
}

static int pack_checked(kpl_ctx* ctx, const HostForestArrays& H, std::vector<PackedNode>& nodes, std::vector<int32_t>& roots, ForestInfo& info)
{
    int max_depth = 0, max_var = -1;
    std::string err;
    int rc = pack_forest(H, nodes, roots, max_depth, max_var, err);
    if (rc) return fail(ctx, rc, err);
    if (roots.empty()) return fail(ctx, KPL_E_FOREST, "forest has no trees");
    info.ntrees = (int32_t)roots.size(); info.nnodes = (int32_t)H.var.size(); info.var_count = H.var_count; info.max_depth = max_depth; info.max_var = max_var;
    info.digest = fnv1a64(roots.data(), roots.size() * sizeof(int32_t), fnv1a64(nodes.data(), nodes.size() * sizeof(PackedNode)));
    info.digest = fnv1a64(&H.var_count, sizeof H.var_count, info.digest);
    return KPL_OK;
}

// Installs forest 0 alone (replace) or appends a forest to the set.  A forest that does not pack leaves the set as it was.
static int install_forest(kpl_ctx* ctx, const HostForestArrays& H, bool replace)
{
    std::vector<PackedNode> nodes;
    std::vector<int32_t> roots;
    ForestInfo info;
    int rc = pack_checked(ctx, H, nodes, roots, info);
    if (rc) return rc;
    KPL_CUDA(cudaSetDevice(ctx->device));
    ForestSet S;
    if (replace) free_forest_set(ctx->forests);     // the old set goes first: a failed upload leaves no forest loaded
    else { S.info = ctx->forests.info; S.nodes = ctx->forests.nodes; S.roots = ctx->forests.roots; S.desc = ctx->forests.desc; }
    append_forest(S, info, nodes, roots);
    return upload_forest_set(ctx, S);
}

static int add_forest(kpl_ctx* ctx, const HostForestArrays& H, int32_t* index_out)
{
    if (ctx->forests.info.empty()) return fail(ctx, KPL_E_FOREST, "no forest 0 loaded: kpl_load_forest / kpl_set_forest come first");
    if ((int)ctx->forests.info.size() >= KPL_MAX_FORESTS) return fail(ctx, KPL_E_INVALID, "the forest set is full (KPL_MAX_FORESTS)");
    int rc = install_forest(ctx, H, false);
    if (rc) return rc;
    if (index_out) *index_out = (int32_t)ctx->forests.info.size() - 1;
    return KPL_OK;
}

int kpl_load_forest(kpl_ctx* ctx, const char* path)
{
    if (!ctx || !path) return KPL_E_INVALID;
    HostForestArrays H;
    std::string err;
    int rc = parse_forest_yaml(path, H, err);
    if (rc) return fail(ctx, rc, err);
    return install_forest(ctx, H, true);
}

static HostForestArrays forest_arrays(int32_t ntrees, int32_t nnodes, const int32_t* roots, const int32_t* var, const float* thr,
                                      const int32_t* left, const int32_t* right, const float* value, int32_t var_count)
{
    HostForestArrays H;
    H.roots.assign(roots, roots + ntrees); H.var.assign(var, var + nnodes); H.thr.assign(thr, thr + nnodes);
    H.left.assign(left, left + nnodes); H.right.assign(right, right + nnodes); H.value.assign(value, value + nnodes);
    H.var_count = var_count;
    return H;
}

int kpl_set_forest(kpl_ctx* ctx, int32_t ntrees, int32_t nnodes, const int32_t* roots, const int32_t* var, const float* thr,
                   const int32_t* left, const int32_t* right, const float* value, int32_t var_count)
{
    if (!ctx || ntrees < 1 || nnodes < 1 || !roots || !var || !thr || !left || !right || !value) return KPL_E_INVALID;
    return install_forest(ctx, forest_arrays(ntrees, nnodes, roots, var, thr, left, right, value, var_count), true);
}

int kpl_add_forest(kpl_ctx* ctx, const char* path, int32_t* index_out)
{
    if (!ctx || !path) return KPL_E_INVALID;
    HostForestArrays H;
    std::string err;
    int rc = parse_forest_yaml(path, H, err);
    if (rc) return fail(ctx, rc, err);
    return add_forest(ctx, H, index_out);
}

int kpl_add_forest_arrays(kpl_ctx* ctx, int32_t ntrees, int32_t nnodes, const int32_t* roots, const int32_t* var, const float* thr,
                          const int32_t* left, const int32_t* right, const float* value, int32_t var_count, int32_t* index_out)
{
    if (!ctx || ntrees < 1 || nnodes < 1 || !roots || !var || !thr || !left || !right || !value) return KPL_E_INVALID;
    return add_forest(ctx, forest_arrays(ntrees, nnodes, roots, var, thr, left, right, value, var_count), index_out);
}

int kpl_forest_count(const kpl_ctx* ctx, int32_t* count_out)
{
    if (!ctx || !count_out) return KPL_E_INVALID;
    *count_out = (int32_t)ctx->forests.info.size();
    return KPL_OK;
}

int kpl_forest_info(const kpl_ctx* ctx, int32_t* ntrees, int32_t* nnodes, int32_t* var_count, int32_t* max_depth)
{
    if (!ctx) return KPL_E_INVALID;
    const ForestInfo F = ctx->forests.info.empty() ? ForestInfo() : ctx->forests.info[0];
    if (ntrees) *ntrees = F.ntrees;
    if (nnodes) *nnodes = F.nnodes;
    if (var_count) *var_count = F.var_count;
    if (max_depth) *max_depth = F.max_depth;
    return KPL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// stage orchestration (device pointers in, device results out)
// ------------------------------------------------------------------------------------------------
static const double CELL_PAD = 1.0 + 9.5367431640625e-07;    // 1 + 2^-20: points closer than r never lie more than cells_per_radius cells apart
static const double REACH_PAD = 1.0 + 4.76837158203125e-07;   // 1 + 2^-21

double kpl::canonical_cell(const kpl_params& P) { return (double)P.radius_features * CELL_PAD / (double)P.cells_per_radius; }
int32_t kpl::grid_dim(double lo, double hi, double cell) { return (int32_t)std::min(2147483000.0, std::floor((hi - lo) / cell) + 1.0); }
int kpl::grid_reach(double radius, double cell) { return (int)std::floor(radius * REACH_PAD / cell) + 1; }

static void clear_batch(GridDesc& g)
{
    g.views = nullptr; g.layer_view = nullptr; g.view_offsets = nullptr; g.nviews = 0;
    g.interior_lo = g.interior_hi = 0; g.guard_cells = 0;
    g.forced = 0;
}

static int finish_grid(kpl_ctx* ctx, int64_t n)
{
    GridDesc& g = ctx->grid;
    const kpl_params& P = ctx->params;
    double ncells = 1.0;
    for (int a = 0; a < 3; ++a) {
        if (g.dim[a] < 1) return fail(ctx, KPL_E_GRID, "bad grid dimensions");
        ncells *= (double)g.dim[a];
    }
    if (ncells > 2147483646.0) return fail(ctx, KPL_E_GRID, "uniform grid would exceed 2^31-2 cells: cloud too sparse for radius_features/cells_per_radius");
    g.ncells = (int64_t)ncells;
    g.reach_feat = grid_reach(P.radius_features, g.cell);
    g.reach_nms = grid_reach(P.radius_nms, g.cell);
    ctx->stats.grid_cells = g.ncells;
    for (int a = 0; a < 3; ++a) { ctx->stats.grid_dims[a] = g.dim[a]; ctx->stats.grid_origin[a] = g.org[a]; }
    ctx->stats.grid_cell = g.cell;
    ctx->last_n = n;
    return KPL_OK;
}

// Grid of ONE cloud.  A forced grid (slab of a larger cloud) is known a priori: no bounding-box pass and no host
// synchronisation; a non-finite point or a point outside the forced grid is reported by the flags cell_key_kernel
// raises, which detect_finish() / check_forced_grid() read.  cell_override > 0 replaces the canonical cell size
// (kpl_normals sizes its k-NN grid from the data).
int kpl::prepare_grid(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, const uint8_t* d_role, int64_t n, const ForcedGrid* forced, double cell_override)
{
    GridDesc& g = ctx->grid;
    clear_batch(g);
    g.cell = cell_override > 0.0 ? cell_override : canonical_cell(ctx->params);
    if (forced) {
        KPL_CUDA(launch_bbox_init(ctx));
        for (int a = 0; a < 3; ++a) { g.org[a] = forced->origin[a]; g.dim[a] = forced->dims[a]; g.off[a] = forced->offset[a]; }
        g.interior_lo = forced->interior_lo; g.interior_hi = forced->interior_hi; g.guard_cells = forced->guard_cells;
        g.forced = 1;
    } else {
        KPL_CUDA(launch_bbox(ctx, d_xyz, n, ctx->d_bbox));
        uint32_t hb[8];
        KPL_CUDA(cudaMemcpyAsync(hb, ctx->d_bbox, sizeof hb, cudaMemcpyDeviceToHost, ctx->stream));
        KPL_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->syncs++;
        if (hb[6]) return fail(ctx, KPL_E_NONFINITE, "input cloud holds non-finite points");
        for (int a = 0; a < 3; ++a) {
            const double lo = (double)dec_float(hb[a]), hi = (double)dec_float(hb[3 + a]);
            g.off[a] = 0; g.org[a] = lo;
            g.dim[a] = grid_dim(lo, hi, g.cell);
        }
    }
    int rc = finish_grid(ctx, n);
    if (rc) return rc;
    ctx->cur_xyz = d_xyz;
    ctx->cur_nrm = d_nrm;
    KPL_CUDA(build_grid(ctx, d_xyz, d_nrm, d_role, n));
    return KPL_OK;
}

// Grid of a cloud passed to a public entry point: the one kpl_params force (setForcedGrid, a role slab through
// kpl_detect), else the canonical grid of its bounding box.
static int prepare_params_grid(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, const uint8_t* d_role, int64_t n)
{
    const kpl_params& P = ctx->params;
    if (!P.grid_forced) return prepare_grid(ctx, d_xyz, d_nrm, d_role, n, nullptr);
    ForcedGrid f;
    for (int a = 0; a < 3; ++a) { f.origin[a] = P.grid_origin[a]; f.dims[a] = P.grid_dims[a]; f.offset[a] = P.grid_offset[a]; }
    f.interior_lo = P.slab_interior_lo; f.interior_hi = P.slab_interior_hi; f.guard_cells = P.slab_guard_cells;
    return prepare_grid(ctx, d_xyz, d_nrm, d_role, n, &f);
}

// Grid of a batch of independent views (kpl_detect_batch): view v keeps the cells of its own canonical grid (origin =
// its bounding-box minimum) and occupies the z layers [zoff_v, zoff_v + dimz_v) of one stacked grid; `pad` empty
// layers separate two views, so no radius search of any kernel can pair points of different views, and the k-NN
// search is confined to the view's own layers (normals.cu: LocalGrid).  One host synchronisation for all boxes.
static int prepare_grid_batch(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, int64_t n, const int64_t* h_offsets, int nviews)
{
    const kpl_params& P = ctx->params;
    GridDesc& g = ctx->grid;
    clear_batch(g);
    g.cell = canonical_cell(P);
    KPL_CUDA(ensure(ctx->view_offsets, (size_t)nviews + 1));
    KPL_CUDA(ensure(ctx->views, (size_t)nviews));
    KPL_CUDA(ensure(ctx->scratch_i, (size_t)nviews * 8 + 16));
    KPL_CUDA(cudaMemcpyAsync(ctx->view_offsets.p, h_offsets, ((size_t)nviews + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    KPL_CUDA(launch_bbox_init(ctx));
    uint32_t* d_boxes = (uint32_t*)ctx->scratch_i.p;
    KPL_CUDA(launch_bbox_views(ctx, d_xyz, n, ctx->view_offsets.p, nviews, d_boxes));
    std::vector<uint32_t> hb((size_t)nviews * 8);
    KPL_CUDA(cudaMemcpyAsync(hb.data(), d_boxes, hb.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    const int pad = std::max(std::max(grid_reach(P.radius_features, g.cell), grid_reach(P.radius_nms, g.cell)), 1);
    std::vector<ViewDesc> hv((size_t)nviews);
    int64_t z = 0;
    int dimx = 1, dimy = 1;
    for (int v = 0; v < nviews; ++v) {
        const uint32_t* b = hb.data() + (size_t)v * 8;
        if (b[6]) return fail(ctx, KPL_E_NONFINITE, "a view of the batch holds non-finite points");
        int d[3];
        for (int a = 0; a < 3; ++a) {
            const double lo = (double)dec_float(b[a]), hi = (double)dec_float(b[3 + a]);
            hv[(size_t)v].org[a] = lo;
            d[a] = grid_dim(lo, hi, g.cell);
        }
        dimx = std::max(dimx, d[0]); dimy = std::max(dimy, d[1]);
        hv[(size_t)v].zoff = (int32_t)z; hv[(size_t)v].dimz = d[2];
        z += (int64_t)d[2] + pad;
        if (z > 2147483000ll) return fail(ctx, KPL_E_GRID, "the stacked grid of the batch exceeds 2^31 layers");
    }
    g.dim[0] = dimx; g.dim[1] = dimy; g.dim[2] = (int32_t)(z - pad);
    for (int a = 0; a < 3; ++a) { g.off[a] = 0; g.org[a] = hv[0].org[a]; }
    int rc = finish_grid(ctx, n);
    if (rc) return rc;
    std::vector<int32_t> layer((size_t)g.dim[2], -1);
    for (int v = 0; v < nviews; ++v)
        for (int l = 0; l < hv[(size_t)v].dimz; ++l) layer[(size_t)hv[(size_t)v].zoff + l] = v;
    KPL_CUDA(ensure(ctx->layer_view, layer.size()));
    KPL_CUDA(cudaMemcpyAsync(ctx->views.p, hv.data(), hv.size() * sizeof(ViewDesc), cudaMemcpyHostToDevice, ctx->stream));
    KPL_CUDA(cudaMemcpyAsync(ctx->layer_view.p, layer.data(), layer.size() * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));      // hv / layer are stack-lifetime host buffers
    ctx->syncs++;
    g.views = ctx->views.p; g.layer_view = ctx->layer_view.p; g.view_offsets = ctx->view_offsets.p; g.nviews = nviews;
    ctx->cur_xyz = d_xyz;
    ctx->cur_nrm = d_nrm;
    KPL_CUDA(build_grid(ctx, d_xyz, d_nrm, nullptr, n));
    return KPL_OK;
}

// Work list of the normal kernel and query order of the feature kernel for the grid in place.
static int prepare_lists(kpl_ctx* ctx, bool normals_given, bool want_features, bool use_role)
{
    const kpl_params& P = ctx->params;
    int span_n = -1;
    bool curve_normals = false;
    if (!normals_given) {
        if (P.normals_mode == KPL_NORMALS_KNN) curve_normals = normals_knn_uses_work_list(P);
        else if (P.normals_mode == KPL_NORMALS_RADIUS) span_n = P.cells_per_radius;
    }
    // A launch of few waves (a slab of a multi-GPU job, a single view) ends with a long idle tail unless the expensive
    // warps start first; a cloud whose sorted arrays exceed the L2 keeps the spatial order of its queries instead, so
    // that concurrently running warps keep sharing candidate rows (there the tail is a percent of the launch anyway).
    const int64_t slots = 148 * 28;
    const int64_t longest_first_below = ctx->last_n * 32 < (int64_t)120e6 ? 24 * slots : 0;
    KPL_CUDA(build_lists(ctx, ctx->last_n, span_n, curve_normals, want_features, use_role, longest_first_below));
    return KPL_OK;
}

static int prepare_normals(kpl_ctx* ctx, bool given, int64_t n)
{
    const kpl_params& P = ctx->params;
    if (!given) {
        if (P.normals_mode == KPL_NORMALS_KNN) KPL_CUDA(launch_normals_knn(ctx, n));
        else if (P.normals_mode == KPL_NORMALS_RADIUS) KPL_CUDA(launch_normals_radius(ctx, n));
        else return fail(ctx, KPL_E_SIZE_MISMATCH, "normals_mode is GIVEN but no normals were passed");
        if (P.flip_normals) KPL_CUDA(launch_flip_normals(ctx, n));
    }
    ctx->last_has_normals = true;
    return KPL_OK;
}

void kpl::detect_reset(kpl_ctx* ctx)
{
    (void)cudaGetLastError();      // a stale error of an earlier, unrelated runtime call must not be blamed on this call
    ctx->launches = 0;
    ctx->syncs = 0;
    ctx->err.clear();
    ctx->last_has_normals = ctx->last_has_features = ctx->last_has_fragile = false;
    ctx->last_nforests = 1;
    memset(&ctx->timings, 0, sizeof ctx->timings);
    memset(&ctx->stats, 0, sizeof ctx->stats);
    ctx->stats.n_views = 1;
}

namespace kpl {

int detect_check(kpl_ctx* ctx, int64_t n, int nforests, bool with_role)
{
    const kpl_params& P = ctx->params;
    const std::vector<ForestInfo>& info = ctx->forests.info;
    if (n < 0 || n > 2147483000ll) return fail(ctx, KPL_E_INVALID, "point count out of range");
    if (info.empty()) return fail(ctx, KPL_E_FOREST, "no forest loaded");
    // a caller that drives a slab by itself cannot see the neighbours' decisions, which its own depend on (the kpl_shard_*
    // entry points exchange them between the resolution rounds)
    if (P.draws_remove && P.non_maxima && with_role)
        return fail(ctx, KPL_E_UNSUPPORTED, "draws-remove NMS walks the whole cloud in index order (hpp:233-250): not available with a role array; use the kpl_shard_* entry points");
    const int F = P.n_annulus * P.n_bins;
    for (int k = 0; k < nforests; ++k) {
        char b[160];
        if (info[k].var_count > 0 && info[k].var_count != F) {
            snprintf(b, sizeof b, "annuli*bins does not match the var_count of forest %d", k);
            return fail(ctx, KPL_E_VARCOUNT, b);
        }
        // whatever var_count says, no split may read beyond the A*B floats of a feature row
        if (info[k].max_var >= F) {
            snprintf(b, sizeof b, "forest %d splits on a variable index >= annuli*bins", k);
            return fail(ctx, KPL_E_VARCOUNT, b);
        }
    }
    // scores, flags and fragile flags hold nforests x n entries, forest-major
    if ((int64_t)nforests * n > 2147483000ll) return fail(ctx, KPL_E_INVALID, "forest count x point count out of range");
    return KPL_OK;
}

// Phase A of a detection: grid (already built by the caller), normals, features + forest -> scores of every point
// whose role asks for one.  Events 1..4 bracket the stages.
int detect_score_phase(kpl_ctx* ctx, bool normals_given, bool use_role, int64_t n, int nforests)
{
    const kpl_params& P = ctx->params;
    const int F = P.n_annulus * P.n_bins;
    int rc = prepare_lists(ctx, normals_given, true, use_role);
    if (rc) return rc;
    KPL_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    rc = prepare_normals(ctx, normals_given, n);
    if (rc) return rc;
    KPL_CUDA(launch_check_normals(ctx, n, use_role));
    KPL_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    // the forests are evaluated in the tail of the feature kernel
    KPL_CUDA(launch_features(ctx, n, use_role, nforests, ctx->keep_intermediates));
    ctx->last_has_features = ctx->keep_intermediates; ctx->last_F = F;
    ctx->last_has_fragile = P.report_fragile != 0;
    KPL_CUDA(cudaEventRecord(ctx->ev[3], ctx->stream));
    KPL_CUDA(cudaEventRecord(ctx->ev[4], ctx->stream));     // forest_ms: the forests have no stage of their own
    return KPL_OK;
}

// Threshold + NMS of forest k's scores (slice k of the forest-major scores) into slice k of the keypoint flags.
static int nms_flags(kpl_ctx* ctx, bool use_role, int64_t n, int k, double th)
{
    const kpl_params& P = ctx->params;
    const int64_t off = (int64_t)k * n;
    if (P.non_maxima && P.draws_remove) KPL_CUDA(launch_nms_draws(ctx, n, use_role, ctx->s_score.p + off, th, off));
    else if (P.non_maxima) KPL_CUDA(launch_nms(ctx, n, use_role, ctx->s_score.p + off, th, off));
    else KPL_CUDA(launch_all_flags(ctx, n, ctx->score.p + off, off));
    return KPL_OK;
}

// Phase B: threshold + NMS of every forest's slice of the scores in place, then one compaction of the nforests x n flags:
// ascending keypoint indices in [0, nforests * n) into d_kp_out.
int detect_nms_phase(kpl_ctx* ctx, bool use_role, int64_t n, int nforests, const double* thresholds, int32_t* d_kp_out)
{
    KPL_CUDA(ensure(ctx->flag, (size_t)nforests * n));      // before slice 0: a later growth would drop the flags of earlier slices
    for (int k = 0; k < nforests; ++k) {
        int rc = nms_flags(ctx, use_role, n, k, thresholds ? thresholds[k] : ctx->params.threshold);
        if (rc) return rc;
    }
    KPL_CUDA(launch_compact(ctx, (int64_t)nforests * n, d_kp_out));
    return KPL_OK;
}

// End of a call: counters and grid flags to the host (the one unavoidable synchronisation), stats and timings.
int detect_finish(kpl_ctx* ctx, int64_t n, int64_t* n_kp_out)
{
    KPL_CUDA(cudaSetDevice(ctx->device));
    KPL_CUDA(cudaEventRecord(ctx->ev[5], ctx->stream));
    unsigned long long hc[kpl_ctx::NCOUNTERS];
    uint32_t hb[8];
    KPL_CUDA(cudaMemcpyAsync(hc, ctx->counters.p, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaMemcpyAsync(hb, ctx->d_bbox, sizeof hb, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    if (ctx->grid.forced && hb[7]) return fail(ctx, KPL_E_GRID, "a point lies outside the forced grid (or is not finite)");
    if (hc[9]) {
        char b[256];
        snprintf(b, sizeof b, "%llu k-NN normals that kept points depend on were clipped by a slab face: widen normal_support_cells", hc[9]);
        return fail(ctx, KPL_E_HALO, b);
    }
    const int32_t nkp = (int32_t)(hc[3] & 0xFFFFFFFFull);
    if (n_kp_out) *n_kp_out = nkp;
    kpl_timings& T = ctx->timings;
    cudaEventElapsedTime(&T.grid_ms, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&T.normals_ms, ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&T.features_ms, ctx->ev[2], ctx->ev[3]);
    cudaEventElapsedTime(&T.forest_ms, ctx->ev[3], ctx->ev[4]);
    cudaEventElapsedTime(&T.nms_ms, ctx->ev[4], ctx->ev[5]);
    cudaEventElapsedTime(&T.total_ms, ctx->ev[0], ctx->ev[5]);
    kpl_stats& S = ctx->stats;
    S.n_points = n;
    S.feature_pairs = (int64_t)hc[0]; S.candidate_pairs = (int64_t)hc[1]; S.n_above_threshold = (int64_t)hc[2];
    S.n_keypoints = nkp; S.kernel_launches = ctx->launches; S.n_scored = (int64_t)hc[5]; S.n_unscored = (int64_t)hc[4];
    S.fast_math = ctx->fast_math ? 1 : 0;
    S.n_near_threshold = (int64_t)hc[7]; S.n_fragile_points = (int64_t)hc[8];
    S.host_syncs = ctx->syncs;
    return KPL_OK;
}

int detect_begin(kpl_ctx* ctx)
{
    KPL_CUDA(cudaSetDevice(ctx->device));
    KPL_CUDA(cudaMemsetAsync(ctx->counters.p, 0, kpl_ctx::NCOUNTERS * sizeof(unsigned long long), ctx->stream));
    KPL_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    return KPL_OK;
}

}  // namespace kpl

// ------------------------------------------------------------------------------------------------
// kpl_detect*: one driver behind every entry point
// ------------------------------------------------------------------------------------------------

// Grid -> scores -> NMS, the body of every detection: the params grid of one cloud (h_view_off NULL; roles allowed) or the
// stacked grid of nviews views at host offsets h_view_off, then one feature pass whose tail walks K forests, each forest's
// threshold + NMS on its slice of the forest-major K x n scores, and one compaction into the ascending list d_kp.
static int detect_body(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, const uint8_t* d_role, int64_t n,
                       const int64_t* h_view_off, int nviews, int K, const double* thresholds, int32_t* d_kp)
{
    int rc = h_view_off ? prepare_grid_batch(ctx, d_xyz, d_nrm, n, h_view_off, nviews) : prepare_params_grid(ctx, d_xyz, d_nrm, d_role, n);
    if (rc) return rc;
    if ((rc = detect_score_phase(ctx, d_nrm != nullptr, d_role != nullptr, n, K))) return rc;
    return detect_nms_phase(ctx, d_role != nullptr, n, K, thresholds, d_kp);
}

// One cloud, or a batch of independent views in ONE pass (one stacked grid, one query order, one launch per stage -- a
// 200 k-point view alone is 1.5 waves of the feature kernel and a handful of host round trips).  d_scores: NULL or the
// K x n scores.  d_kp_off: NULL (kpl_detect*), or the K x nviews + 1 offsets of the (forest, view) ranges, which
// launch_view_ranges cuts from the one list (view-local indices).  No host round trip beyond those of the grid, the
// draws-remove rounds and detect_finish.
static int run_detect(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, const uint8_t* d_role, int64_t n,
                      const int64_t* h_view_off, int nviews, int K, const double* thresholds, float* d_scores, int32_t* d_kp,
                      int64_t* d_kp_off, int64_t* n_kp_out)
{
    ctx->stats.n_points = n; ctx->stats.n_views = nviews;
    ctx->last_nforests = K;
    if (n == 0) {       // no runtime call unless there are offsets to zero
        if (d_kp_off) {
            KPL_CUDA(cudaSetDevice(ctx->device));
            KPL_CUDA(cudaMemsetAsync(d_kp_off, 0, ((size_t)K * nviews + 1) * sizeof(int64_t), ctx->stream));
        }
        return KPL_OK;
    }
    int rc = detect_begin(ctx);
    if (rc) return rc;
    if ((rc = detect_body(ctx, d_xyz, d_nrm, d_role, n, h_view_off, nviews, K, thresholds, d_kp))) return rc;
    if (d_kp_off) {
        // the boundaries of the (forest, view) ranges: {k*n + h_view_off[v]} for k < K, v < nviews, then K*n.  One forest of
        // a batch splits at the view offsets the stacked grid holds on the device.  The host copy is a member: a pageable
        // source is staged by cudaMemcpyAsync before it returns, the member keeps it anyway.
        const int64_t* d_bounds = ctx->view_offsets.p;
        if (K > 1 || !h_view_off) {
            const size_t nb = (size_t)K * nviews + 1;
            ctx->range_off_h.resize(nb);
            for (int k = 0; k < K; ++k)
                for (int v = 0; v < nviews; ++v) ctx->range_off_h[(size_t)k * nviews + v] = (int64_t)k * n + (h_view_off ? h_view_off[v] : 0);
            ctx->range_off_h[nb - 1] = (int64_t)K * n;
            KPL_CUDA(ensure(ctx->range_off, nb));
            KPL_CUDA(cudaMemcpyAsync(ctx->range_off.p, ctx->range_off_h.data(), nb * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
            d_bounds = ctx->range_off.p;
        }
        KPL_CUDA(launch_view_ranges(ctx, (int64_t)K * n, d_kp, d_bounds, K * nviews, d_kp_off));
    }
    if (d_scores) KPL_CUDA(cudaMemcpyAsync(d_scores, ctx->score.p, (size_t)K * n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return detect_finish(ctx, n, n_kp_out);
}

// A batch of organized frames of one size: integral-image normals of every frame (or the caller's per-pixel normals),
// the finite pixels compacted in ascending pixel order, the compacted frames detected as the views of one batch, and the
// results mapped back to pixel order.  Each frame's view is the cloud the single-frame path (computeOrganized /
// KeypointLearningDetector::compute) detects after dropping its NaN points, in the same order, so its results are that
// path's.  One host round trip for the per-frame finite counts, which the batch needs as host view offsets; a frame
// without a finite point is left out of the batch (views must not be empty) and gets an empty keypoint range.  K forests
// (kpl_detect_batch_organized_forests) score the inner batch from one feature pass; the results stay forest-major through
// the map back: K x F x W*H scores, K x F + 1 keypoint offsets.
static int run_detect_organized_batch(kpl_ctx* ctx, const float4* d_xyz, const float4* d_nrm, int32_t W, int32_t H, int32_t F,
                                      float smoothing_size, const float* h_viewpoints, int K, const double* thresholds,
                                      float* d_scores, int32_t* d_kp, int64_t* d_kp_off, int64_t* n_kp_out)
{
    const int64_t n = (int64_t)W * H, total = n * F;
    ctx->stats.n_views = F;
    ctx->last_nforests = K;
    int rc = detect_begin(ctx);
    if (rc) return rc;
    if (!d_nrm) {
        const float* d_vp = nullptr;
        if (h_viewpoints) {
            KPL_CUDA(ensure(ctx->org_vp, (size_t)F * 3));
            KPL_CUDA(cudaMemcpyAsync(ctx->org_vp.p, h_viewpoints, (size_t)F * 3 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
            d_vp = ctx->org_vp.p;
        }
        KPL_CUDA(ensure(ctx->in_nrm, (size_t)total));        // per-pixel normals; the staging buffer is free without caller normals
        KPL_CUDA(launch_normals_integral_image(ctx, d_xyz, W, H, F, smoothing_size, d_vp, ctx->in_nrm.p));
        d_nrm = ctx->in_nrm.p;
    }
    KPL_CUDA(launch_organized_select(ctx, d_xyz, n, F, K, d_scores));
    KPL_CUDA(cudaEventRecord(ctx->ev[6], ctx->stream));
    std::vector<int64_t> frame_off((size_t)F + 1);
    KPL_CUDA(cudaMemcpyAsync(frame_off.data(), ctx->org_frame_off.p, frame_off.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    const int64_t m = frame_off[(size_t)F];
    std::vector<int64_t> view_off(1, 0);
    for (int32_t f = 0; f < F; ++f)
        if (frame_off[(size_t)f + 1] > frame_off[(size_t)f]) view_off.push_back(frame_off[(size_t)f + 1]);
    kpl_timings& T = ctx->timings;
    if (m == 0) {
        KPL_CUDA(cudaMemsetAsync(d_kp_off, 0, ((size_t)K * F + 1) * sizeof(int64_t), ctx->stream));
        cudaEventElapsedTime(&T.normals_ms, ctx->ev[0], ctx->ev[6]);
        T.total_ms = T.normals_ms;
        ctx->stats.n_points = 0; ctx->stats.kernel_launches = ctx->launches; ctx->stats.host_syncs = ctx->syncs;
        return KPL_OK;
    }
    KPL_CUDA(launch_organized_gather(ctx, d_xyz, d_nrm, m));
    if ((rc = detect_body(ctx, ctx->org_xyz.p, ctx->org_nrm.p, nullptr, m, view_off.data(), (int)view_off.size() - 1, K, thresholds, d_kp)))
        return rc;
    KPL_CUDA(launch_organized_map_back(ctx, m, n, F, K, d_scores, d_kp, d_kp_off));
    if ((rc = detect_finish(ctx, m, n_kp_out))) return rc;
    // the integral images and the compaction are part of the normals stage; the grid stage starts after them
    float prep = 0.f;
    cudaEventElapsedTime(&prep, ctx->ev[0], ctx->ev[6]);
    cudaEventElapsedTime(&T.grid_ms, ctx->ev[6], ctx->ev[1]);
    T.normals_ms += prep;
    return KPL_OK;
}

// host (possibly strided) -> device float4 staging
static int upload_vec3(kpl_ctx* ctx, DevBuf<float4>& dst, const float* src, int32_t stride, int64_t n)
{
    if (stride < 12 || (stride & 3)) return fail(ctx, KPL_E_INVALID, "stride must be a multiple of 4 and >= 12 bytes");
    KPL_CUDA(ensure(dst, (size_t)n));
    if (stride == 16) KPL_CUDA(cudaMemcpyAsync(dst.p, src, (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream));
    else KPL_CUDA(cudaMemcpy2DAsync(dst.p, 16, src, (size_t)stride, stride >= 16 ? 16 : 12, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    return KPL_OK;
}

static int upload_inputs(kpl_ctx* ctx, const float* xyz, int32_t xs, const float* normals, int32_t ns, const uint8_t* role, int64_t n)
{
    if (!xyz && n > 0) return fail(ctx, KPL_E_INVALID, "xyz is NULL");
    KPL_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return KPL_OK;
    int rc = upload_vec3(ctx, ctx->in_xyz, xyz, xs, n);
    if (rc) return rc;
    if (normals) { rc = upload_vec3(ctx, ctx->in_nrm, normals, ns, n); if (rc) return rc; }
    if (role) {
        KPL_CUDA(ensure(ctx->in_role, (size_t)n));
        KPL_CUDA(cudaMemcpyAsync(ctx->in_role.p, role, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    }
    return KPL_OK;
}

// Where a call's points come from: one cloud of n points on the params grid (kpl_detect*, kpl_detect_forests*), n_views
// views at host view_offsets (kpl_detect_batch*), or n_views organized frames of width x height pixels
// (kpl_detect_batch_organized*).
enum class Layout { Cloud, Views, Frames };

// One kpl_detect* call as its entry point passes it on: host arrays (xyz / normals at their strides) for the host entry
// points, float4 device arrays for the _device ones.
struct DetectCall {
    const void* xyz; int32_t xyz_stride; const void* normals; int32_t normals_stride;
    const uint8_t* role = nullptr;                  // a cloud only
    int64_t n = 0;                                  // a cloud's points; detect_prologue counts those of a batch
    Layout layout = Layout::Cloud;
    const int64_t* view_offsets = nullptr;          // views: n_views + 1 host offsets
    int32_t n_views = 1;                            // views or frames
    int32_t width = 0, height = 0; float smoothing = 0.f; const float* viewpoints = nullptr;      // frames
    bool all_forests = false;                       // the *_forests entry points score the whole set, the others forest 0
    int K = 1; const double* thresholds = nullptr;  // K: set by detect_prologue
    bool offsets = false;                           // the call returns the K x n_views + 1 keypoint offsets
    void *scores = nullptr, *kp = nullptr, *kp_offsets = nullptr; float* kp_xyzi = nullptr;

    DetectCall(const void* x, int32_t xs, const void* nrm, int32_t ns) : xyz(x), xyz_stride(xs), normals(nrm), normals_stride(ns) {}
    DetectCall& cloud(int64_t n_, const uint8_t* role_ = nullptr) { n = n_; role = role_; return *this; }
    DetectCall& views(const int64_t* off, int32_t nv) { layout = Layout::Views; view_offsets = off; n_views = nv; offsets = true; return *this; }
    DetectCall& frames(int32_t w, int32_t h, int32_t f, float s, const float* vp)
    {
        layout = Layout::Frames; width = w; height = h; n_views = f; smoothing = s; viewpoints = vp; offsets = true;
        return *this;
    }
    DetectCall& forests(const double* th) { all_forests = true; thresholds = th; offsets = true; return *this; }
    DetectCall& out(void* s, void* k, void* ko, float* xyzi = nullptr) { scores = s; kp = k; kp_offsets = ko; kp_xyzi = xyzi; return *this; }
};

// The start of every kpl_detect* entry point.  The reset comes first, so that a refused call leaves nothing of the
// previous one; then the refusals in the order kpl.h states: NULL arguments, layout, detect_check (with the forced grid a
// batch cannot use).  The strides of a host call are checked last, by its upload.
static int detect_prologue(kpl_ctx* ctx, DetectCall& c, int64_t* n_kp_out)
{
    if (!ctx) return KPL_E_INVALID;
    detect_reset(ctx);
    if (n_kp_out) *n_kp_out = 0;
    if (c.all_forests) c.K = (int)ctx->forests.info.size();
    const bool points = c.layout != Layout::Cloud || c.n > 0;       // a batch holds at least one point
    if ((points && !c.xyz) || ((points || c.offsets) && !c.kp) || (c.offsets && !c.kp_offsets))
        return fail(ctx, KPL_E_INVALID, "NULL input or output array");
    if (c.layout == Layout::Views) {
        const int64_t* off = c.view_offsets;
        if (c.n_views < 1 || !off) return fail(ctx, KPL_E_INVALID, "view_offsets / n_views missing");
        if (off[0] != 0) return fail(ctx, KPL_E_INVALID, "view_offsets[0] must be 0");
        for (int32_t v = 0; v < c.n_views; ++v)
            if (off[v + 1] <= off[v]) return fail(ctx, KPL_E_INVALID, "view_offsets must be strictly ascending (empty views are not allowed)");
        c.n = off[c.n_views];
    } else if (c.layout == Layout::Frames) {
        if (c.width < 1 || c.height < 1 || c.n_views < 1) return fail(ctx, KPL_E_INVALID, "width, height and n_frames must be >= 1");
        c.n = (int64_t)c.width * c.height * c.n_views;
        if (c.n > 2147483000ll) return fail(ctx, KPL_E_INVALID, "point count out of range");
        if (!(c.smoothing > 0.f) || !std::isfinite(c.smoothing)) return fail(ctx, KPL_E_INVALID, "normal smoothing size must be > 0");
    }
    int rc = detect_check(ctx, c.n, c.K, c.role != nullptr);
    if (rc) return rc;
    if (c.layout != Layout::Cloud && ctx->params.grid_forced) return fail(ctx, KPL_E_INVALID, "a forced grid cannot be combined with a batch");
    return KPL_OK;
}

// A call whose arrays are on the device, past its prologue.  The drivers set the device before their first runtime call.
static int run_call(kpl_ctx* ctx, const DetectCall& c, int64_t* n_kp_out)
{
    const float4 *xyz = (const float4*)c.xyz, *nrm = (const float4*)c.normals;
    float* scores = (float*)c.scores;
    int32_t* kp = (int32_t*)c.kp;
    int64_t* kp_off = (int64_t*)c.kp_offsets;
    if (c.layout == Layout::Frames)
        return run_detect_organized_batch(ctx, xyz, nrm, c.width, c.height, c.n_views, c.smoothing, c.viewpoints, c.K, c.thresholds, scores, kp,
                                          kp_off, n_kp_out);
    return run_detect(ctx, xyz, nrm, c.role, c.n, c.view_offsets, c.n_views, c.K, c.thresholds, scores, kp, kp_off, n_kp_out);
}

static int detect_device(kpl_ctx* ctx, DetectCall c, int64_t* n_kp_out)
{
    const int rc = detect_prologue(ctx, c, n_kp_out);
    return rc ? rc : run_call(ctx, c, n_kp_out);
}

// Host arrays in, host results out: the n points staged (every pixel of the frames), the driver, then the copies of the
// K x n scores (the pixel-order org_score of frames, ctx->score otherwise), the keypoints, kpl_detect_xyzi's keypoint
// cloud and the offsets, and one synchronisation.  A cloud without points and offsets has nothing to copy back.
static int detect_host(kpl_ctx* ctx, DetectCall c, int64_t* n_kp_out)
{
    int rc = detect_prologue(ctx, c, n_kp_out);
    if (rc || (rc = upload_inputs(ctx, (const float*)c.xyz, c.xyz_stride, (const float*)c.normals, c.normals_stride, c.role, c.n))) return rc;
    const int64_t n = c.n;
    const size_t noff = c.offsets ? (size_t)c.K * c.n_views + 1 : 0;
    if (n > 0) KPL_CUDA(ensure(ctx->kp_idx, (size_t)c.K * n));
    if (noff) KPL_CUDA(ensure(ctx->kp_off, noff));
    float* d_scores = nullptr;
    if (c.layout == Layout::Frames && c.scores) {
        KPL_CUDA(ensure(ctx->org_score, (size_t)c.K * n));
        d_scores = ctx->org_score.p;
    }
    DetectCall staged = c;
    staged.xyz = ctx->in_xyz.p; staged.normals = c.normals ? ctx->in_nrm.p : nullptr; staged.role = c.role ? ctx->in_role.p : nullptr;
    staged.out(d_scores, ctx->kp_idx.p, noff ? ctx->kp_off.p : nullptr);
    int64_t nkp = 0;
    if ((rc = run_call(ctx, staged, &nkp))) return rc;
    if (n == 0 && !noff) return KPL_OK;
    if (c.scores && n > 0)
        KPL_CUDA(cudaMemcpyAsync(c.scores, d_scores ? d_scores : ctx->score.p, (size_t)c.K * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (nkp > 0) KPL_CUDA(cudaMemcpyAsync(c.kp, ctx->kp_idx.p, (size_t)nkp * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (nkp > 0 && c.kp_xyzi) {
        // the keypoint cloud of hpp:246-253 (x, y, z of the input point, intensity = its response), gathered on the
        // device: a host-side gather of ~1e5 scattered rows out of a 160 MB array costs milliseconds of cache misses
        KPL_CUDA(ensure(ctx->scratch_f, (size_t)nkp * 4));
        KPL_CUDA(launch_gather_keypoints(ctx, ctx->in_xyz.p, ctx->kp_idx.p, nkp, (float4*)ctx->scratch_f.p));
        KPL_CUDA(cudaMemcpyAsync(c.kp_xyzi, ctx->scratch_f.p, (size_t)nkp * 16, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (noff) KPL_CUDA(cudaMemcpyAsync(c.kp_offsets, ctx->kp_off.p, noff * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++; ctx->stats.host_syncs = ctx->syncs; ctx->stats.kernel_launches = ctx->launches;
    if (n_kp_out) *n_kp_out = nkp;
    return KPL_OK;
}

extern "C" {

int kpl_detect_xyzi(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                    const uint8_t* role, int64_t n, float* scores_out, int32_t* kp_idx_out, float* kp_xyzi_out, int64_t* n_kp_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.cloud(n, role).out(scores_out, kp_idx_out, nullptr, kp_xyzi_out), n_kp_out);
}

int kpl_detect(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
               const uint8_t* role, int64_t n, float* scores_out, int32_t* kp_idx_out, int64_t* n_kp_out)
{
    return kpl_detect_xyzi(ctx, xyz, xyz_stride, normals, normals_stride, role, n, scores_out, kp_idx_out, nullptr, n_kp_out);
}

int kpl_detect_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const void* d_role, int64_t n,
                      void* d_scores, void* d_kp_idx, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.cloud(n, (const uint8_t*)d_role).out(d_scores, d_kp_idx, nullptr), n_kp_out);
}

int kpl_detect_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride, int64_t n,
                       const double* thresholds, float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.cloud(n).forests(thresholds).out(scores_out, kp_idx_out, kp_offsets_out), nullptr);
}

int kpl_detect_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int64_t n, const double* thresholds,
                              void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.cloud(n).forests(thresholds).out(d_scores, d_kp_idx, d_kp_offsets), n_kp_out);
}

int kpl_detect_batch(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                     const int64_t* view_offsets, int32_t n_views, float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.views(view_offsets, n_views).out(scores_out, kp_idx_out, kp_offsets_out), nullptr);
}

int kpl_detect_batch_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                             const int64_t* view_offsets, int32_t n_views, const double* thresholds, float* scores_out,
                             int32_t* kp_idx_out, int64_t* kp_offsets_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.views(view_offsets, n_views).forests(thresholds).out(scores_out, kp_idx_out, kp_offsets_out), nullptr);
}

int kpl_detect_batch_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const int64_t* view_offsets, int32_t n_views,
                            void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.views(view_offsets, n_views).out(d_scores, d_kp_idx, d_kp_offsets), n_kp_out);
}

int kpl_detect_batch_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, const int64_t* view_offsets, int32_t n_views,
                                    const double* thresholds, void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.views(view_offsets, n_views).forests(thresholds).out(d_scores, d_kp_idx, d_kp_offsets), n_kp_out);
}

int kpl_detect_batch_organized(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                               int32_t width, int32_t height, int32_t n_frames, float smoothing_size, const float* viewpoints,
                               float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.frames(width, height, n_frames, smoothing_size, viewpoints).out(scores_out, kp_idx_out, kp_offsets_out), nullptr);
}

int kpl_detect_batch_organized_forests(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                                       int32_t width, int32_t height, int32_t n_frames, float smoothing_size, const float* viewpoints,
                                       const double* thresholds, float* scores_out, int32_t* kp_idx_out, int64_t* kp_offsets_out)
{
    DetectCall c(xyz, xyz_stride, normals, normals_stride);
    return detect_host(ctx, c.frames(width, height, n_frames, smoothing_size, viewpoints).forests(thresholds).out(scores_out, kp_idx_out, kp_offsets_out), nullptr);
}

int kpl_detect_batch_organized_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int32_t width, int32_t height,
                                      int32_t n_frames, float smoothing_size, const float* viewpoints, void* d_scores, void* d_kp_idx,
                                      void* d_kp_offsets, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.frames(width, height, n_frames, smoothing_size, viewpoints).out(d_scores, d_kp_idx, d_kp_offsets), n_kp_out);
}

int kpl_detect_batch_organized_forests_device(kpl_ctx* ctx, const void* d_xyz4, const void* d_normals4, int32_t width, int32_t height,
                                              int32_t n_frames, float smoothing_size, const float* viewpoints, const double* thresholds,
                                              void* d_scores, void* d_kp_idx, void* d_kp_offsets, int64_t* n_kp_out)
{
    DetectCall c(d_xyz4, 16, d_normals4, 16);
    return detect_device(ctx, c.frames(width, height, n_frames, smoothing_size, viewpoints).forests(thresholds).out(d_scores, d_kp_idx, d_kp_offsets), n_kp_out);
}

// Forced grids skip the bounding-box round trip (prepare_grid): entry points other than kpl_detect* read the
// out-of-grid flag here.
static int check_forced_grid(kpl_ctx* ctx)
{
    if (!ctx->grid.forced) return KPL_OK;
    uint32_t hb[8];
    KPL_CUDA(cudaMemcpyAsync(hb, ctx->d_bbox, sizeof hb, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    if (hb[7]) return fail(ctx, KPL_E_GRID, "a point lies outside the forced grid (or is not finite)");
    return KPL_OK;
}

// The k-NN search is exact on any grid, so a stand-alone kpl_normals call (TestDetector runs the normal estimation
// before the detector exists, main_test_detector.cpp:162-169, and knows no radiusFeatures there) sizes its grid from
// the data: about KNN_TARGET points per occupied cell, whatever the unit of the cloud.
static const double KNN_TARGET = 14.0;

static int prepare_knn_grid(kpl_ctx* ctx, int64_t n)
{
    const kpl_params& P = ctx->params;
    if (P.grid_forced || P.normals_mode != KPL_NORMALS_KNN) return prepare_params_grid(ctx, ctx->in_xyz.p, nullptr, nullptr, n);
    // first guess from the bounding box as if the points filled it; surfaces and curves then show far more points per
    // occupied cell than wanted, and the cell is refined from the measured occupancy (occupancy ~ cell^2 on a surface)
    KPL_CUDA(launch_bbox(ctx, ctx->in_xyz.p, n, ctx->d_bbox));
    uint32_t hb[8];
    KPL_CUDA(cudaMemcpyAsync(hb, ctx->d_bbox, sizeof hb, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    if (hb[6]) return fail(ctx, KPL_E_NONFINITE, "input cloud holds non-finite points");
    double ext[3], vol = 1.0, longest = 0.0;
    for (int a = 0; a < 3; ++a) { ext[a] = (double)dec_float(hb[3 + a]) - (double)dec_float(hb[a]); longest = std::max(longest, ext[a]); }
    if (!(longest > 0.0)) longest = 1.0;                                   // all points coincide: any cell will do
    for (int a = 0; a < 3; ++a) vol *= std::max(ext[a], longest * 1e-3);
    const double k = (double)std::max(P.k_normals, 1);
    const double target = KNN_TARGET * k / 10.0;
    const double min_cell = std::cbrt(vol / 1.0e9) * 1.001 + longest * 1e-7;  // at most ~1e9 cells
    double cell = std::max(std::cbrt(vol * target / (double)n), min_cell);
    for (int pass = 0; pass < 3; ++pass) {
        int rc = prepare_grid(ctx, ctx->in_xyz.p, nullptr, nullptr, n, nullptr, cell);
        if (rc) return rc;
        if (pass == 2) break;
        KPL_CUDA(cudaMemsetAsync(ctx->counters.p + 10, 0, sizeof(unsigned long long), ctx->stream));
        KPL_CUDA(launch_count_occupied_cells(ctx, n, ctx->counters.p + 10));
        unsigned long long occupied = 0;
        KPL_CUDA(cudaMemcpyAsync(&occupied, ctx->counters.p + 10, sizeof occupied, cudaMemcpyDeviceToHost, ctx->stream));
        KPL_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->syncs++;
        const double occ = (double)n / (double)std::max<unsigned long long>(occupied, 1);
        if (occ <= 3.0 * target || cell <= min_cell) break;
        cell = std::max(cell * std::sqrt(target / occ), min_cell);
    }
    return KPL_OK;
}


int kpl_normals(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, float* normals_out)
{
    if (!ctx || (n > 0 && !normals_out)) return KPL_E_INVALID;
    detect_reset(ctx);
    if (n == 0) return KPL_OK;
    if (ctx->params.normals_mode == KPL_NORMALS_GIVEN) return fail(ctx, KPL_E_INVALID, "normals_mode must be KNN or RADIUS");
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    KPL_CUDA(cudaMemsetAsync(ctx->counters.p, 0, kpl_ctx::NCOUNTERS * sizeof(unsigned long long), ctx->stream));
    KPL_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
    if ((rc = prepare_knn_grid(ctx, n))) return rc;
    if ((rc = check_forced_grid(ctx))) return rc;
    if ((rc = prepare_lists(ctx, false, false, false))) return rc;
    KPL_CUDA(cudaEventRecord(ctx->ev[1], ctx->stream));
    if ((rc = prepare_normals(ctx, false, n))) return rc;
    KPL_CUDA(cudaEventRecord(ctx->ev[2], ctx->stream));
    KPL_CUDA(ensure(ctx->scratch_f, (size_t)n * 4));
    KPL_CUDA(launch_unsort_normals(ctx, n, (float4*)ctx->scratch_f.p));
    KPL_CUDA(cudaMemcpyAsync(normals_out, ctx->scratch_f.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    cudaEventElapsedTime(&ctx->timings.grid_ms, ctx->ev[0], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->timings.normals_ms, ctx->ev[1], ctx->ev[2]);
    ctx->timings.total_ms = ctx->timings.grid_ms + ctx->timings.normals_ms;
    ctx->stats.n_points = n; ctx->stats.kernel_launches = ctx->launches; ctx->stats.host_syncs = ctx->syncs;
    return KPL_OK;
}

// Organized clouds: pcl::IntegralImageNormalEstimation(SIMPLE_3D_GRADIENT, smoothing 5.0) (hpp:138-145), csrc/organized.cu.
int kpl_normals_organized(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int32_t width, int32_t height, float smoothing_size, float* normals_out)
{
    if (!ctx || width < 1 || height < 1 || !xyz || !normals_out) return KPL_E_INVALID;
    detect_reset(ctx);
    if (!(smoothing_size > 0.f) || !std::isfinite(smoothing_size)) return fail(ctx, KPL_E_INVALID, "normal smoothing size must be > 0");
    const int64_t n = (int64_t)width * height;
    if (n > 2147483000ll) return fail(ctx, KPL_E_INVALID, "point count out of range");
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    KPL_CUDA(ensure(ctx->in_nrm, (size_t)n));
    KPL_CUDA(launch_normals_integral_image(ctx, ctx->in_xyz.p, width, height, 1, smoothing_size, nullptr, ctx->in_nrm.p));
    KPL_CUDA(cudaMemcpyAsync(normals_out, ctx->in_nrm.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    ctx->stats.n_points = n; ctx->stats.kernel_launches = ctx->launches; ctx->stats.host_syncs = ctx->syncs;
    return KPL_OK;
}

// computePointsForTrainingFeatures (hpp:299-318).  With an index subset (TrainDetector's pattern: a few thousand
// samples of a large cloud, main_train_detector.cpp:419-439) only the listed queries are evaluated and only m x F
// floats are ever materialised.
int kpl_features(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, const float* normals, int32_t normals_stride,
                 int64_t n, const int32_t* indices, int64_t m, float* features_out)
{
    if (!ctx || m < 0 || (m > 0 && !features_out)) return KPL_E_INVALID;
    detect_reset(ctx);
    if (!indices && m != n) return fail(ctx, KPL_E_INVALID, "indices == NULL requires m == n");
    if (n == 0 || m == 0) return KPL_OK;
    if (m > 2147483000ll) return fail(ctx, KPL_E_INVALID, "too many feature indices");
    const int F = ctx->params.n_annulus * ctx->params.n_bins;
    if (indices)
        for (int64_t k = 0; k < m; ++k)
            if (indices[k] < 0 || indices[k] >= n) return fail(ctx, KPL_E_INVALID, "feature index out of range");
    int rc = upload_inputs(ctx, xyz, xyz_stride, normals, normals_stride, nullptr, n);
    if (rc) return rc;
    KPL_CUDA(cudaMemsetAsync(ctx->counters.p, 0, kpl_ctx::NCOUNTERS * sizeof(unsigned long long), ctx->stream));
    if ((rc = prepare_params_grid(ctx, ctx->in_xyz.p, normals ? ctx->in_nrm.p : nullptr, nullptr, n))) return rc;
    if ((rc = check_forced_grid(ctx))) return rc;
    if ((rc = prepare_lists(ctx, normals != nullptr, indices == nullptr, false))) return rc;
    if ((rc = prepare_normals(ctx, normals != nullptr, n))) return rc;
    const float* d_src = nullptr;
    if (indices) {
        KPL_CUDA(ensure(ctx->in_role, (size_t)m * sizeof(int32_t)));          // the role staging buffer is free here
        int32_t* d_idx = reinterpret_cast<int32_t*>(ctx->in_role.p);
        KPL_CUDA(cudaMemcpyAsync(d_idx, indices, (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        KPL_CUDA(build_query_list(ctx, n, d_idx, m));
        KPL_CUDA(launch_features(ctx, n, false, 0, true, ctx->qlist.p, m));
        KPL_CUDA(ensure(ctx->scratch_f, (size_t)m * F));
        KPL_CUDA(launch_scatter_rows(ctx, ctx->feat.p, m, F, ctx->scratch_f.p));
        d_src = ctx->scratch_f.p;
    } else {
        KPL_CUDA(launch_features(ctx, n, false, 0, true));
        ctx->last_has_features = true; ctx->last_F = F;
        KPL_CUDA(ensure(ctx->scratch_f, (size_t)n * F));
        KPL_CUDA(launch_unsort_rows(ctx, ctx->feat.p, n, F, ctx->scratch_f.p));
        d_src = ctx->scratch_f.p;
    }
    KPL_CUDA(cudaMemcpyAsync(features_out, d_src, (size_t)m * F * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long hc[kpl_ctx::NCOUNTERS];
    KPL_CUDA(cudaMemcpyAsync(hc, ctx->counters.p, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->syncs++;
    ctx->stats.fast_math = ctx->fast_math ? 1 : 0;
    ctx->stats.n_points = n; ctx->stats.n_scored = (int64_t)hc[5]; ctx->stats.feature_pairs = (int64_t)hc[0]; ctx->stats.candidate_pairs = (int64_t)hc[1];
    ctx->stats.kernel_launches = ctx->launches; ctx->stats.host_syncs = ctx->syncs;
    return KPL_OK;
}

int kpl_radius_stats(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, double radius, int32_t* counts_out, uint64_t* hash_out)
{
    if (!ctx || !(radius >= 0)) return KPL_E_INVALID;
    detect_reset(ctx);
    if (n == 0) return KPL_OK;
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    if ((rc = prepare_params_grid(ctx, ctx->in_xyz.p, nullptr, nullptr, n))) return rc;
    if ((rc = check_forced_grid(ctx))) return rc;
    KPL_CUDA(ensure(ctx->scratch_i, (size_t)n * 3 + 2));
    int32_t* d_counts = ctx->scratch_i.p;
    unsigned long long* d_hash = (unsigned long long*)(ctx->scratch_i.p + ((n + 1) & ~1ll));
    KPL_CUDA(launch_radius_stats(ctx, n, radius, d_counts, d_hash));
    if (counts_out) KPL_CUDA(cudaMemcpyAsync(counts_out, d_counts, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (hash_out) KPL_CUDA(cudaMemcpyAsync(hash_out, d_hash, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->stats.kernel_launches = ctx->launches;
    return KPL_OK;
}

int kpl_nearest(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, const float* queries, int32_t q_stride, int64_t m,
                int32_t* idx_out, float* d2_out)
{
    if (!ctx || m < 0 || (m > 0 && (!queries || !idx_out))) return KPL_E_INVALID;
    detect_reset(ctx);
    if (m == 0) return KPL_OK;
    if (n <= 0) return fail(ctx, KPL_E_INVALID, "the cloud is empty");
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    if ((rc = prepare_params_grid(ctx, ctx->in_xyz.p, nullptr, nullptr, n))) return rc;
    if ((rc = check_forced_grid(ctx))) return rc;
    if ((rc = upload_vec3(ctx, ctx->in_nrm, queries, q_stride, m))) return rc;          // the normals staging buffer is free here
    KPL_CUDA(ensure(ctx->scratch_i, (size_t)m + 2));
    KPL_CUDA(ensure(ctx->scratch_f, (size_t)m + 2));
    KPL_CUDA(launch_nearest(ctx, ctx->in_nrm.p, m, ctx->scratch_i.p, ctx->scratch_f.p));
    KPL_CUDA(cudaMemcpyAsync(idx_out, ctx->scratch_i.p, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (d2_out) KPL_CUDA(cudaMemcpyAsync(d2_out, ctx->scratch_f.p, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->stats.n_points = n; ctx->stats.kernel_launches = ctx->launches;
    return KPL_OK;
}

int kpl_radius_neighbors(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, double radius,
                         const int32_t* queries, int64_t m, int64_t* offsets_out, int32_t* indices_out)
{
    if (!ctx || !(radius >= 0) || m < 0 || !offsets_out || (m > 0 && !queries)) return KPL_E_INVALID;
    detect_reset(ctx);
    offsets_out[0] = 0;
    if (n == 0 || m == 0) { for (int64_t k = 0; k <= m; ++k) offsets_out[k] = 0; return KPL_OK; }
    for (int64_t k = 0; k < m; ++k) if (queries[k] < 0 || queries[k] >= n) return fail(ctx, KPL_E_INVALID, "query index out of range");
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    if ((rc = prepare_params_grid(ctx, ctx->in_xyz.p, nullptr, nullptr, n))) return rc;
    if ((rc = check_forced_grid(ctx))) return rc;
    KPL_CUDA(ensure(ctx->scratch_i, (size_t)n + 2));
    KPL_CUDA(launch_radius_stats(ctx, n, radius, ctx->scratch_i.p, nullptr));
    std::vector<int32_t> counts((size_t)n), sidx((size_t)n);
    KPL_CUDA(cudaMemcpyAsync(counts.data(), ctx->scratch_i.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaMemcpyAsync(sidx.data(), ctx->idx_b.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int64_t k = 0; k < m; ++k) offsets_out[k + 1] = offsets_out[k] + counts[(size_t)queries[k]];
    if (!indices_out) return KPL_OK;
    std::vector<int32_t> inv((size_t)n), qpos((size_t)m);
    for (int64_t i = 0; i < n; ++i) inv[(size_t)sidx[(size_t)i]] = (int32_t)i;
    for (int64_t k = 0; k < m; ++k) qpos[(size_t)k] = inv[(size_t)queries[k]];
    const int64_t total = offsets_out[m];
    int32_t *d_q = nullptr, *d_idx = nullptr;
    int64_t* d_off = nullptr;
    KPL_CUDA(cudaMalloc((void**)&d_q, (size_t)m * sizeof(int32_t)));
    KPL_CUDA(cudaMalloc((void**)&d_off, (size_t)(m + 1) * sizeof(int64_t)));
    KPL_CUDA(cudaMalloc((void**)&d_idx, (size_t)std::max<int64_t>(total, 1) * sizeof(int32_t)));
    cudaError_t e = cudaMemcpyAsync(d_q, qpos.data(), (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
    if (!e) e = cudaMemcpyAsync(d_off, offsets_out, (size_t)(m + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (!e) e = launch_radius_lists(ctx, n, radius, d_q, m, d_off, d_idx);
    if (!e && total > 0) e = cudaMemcpyAsync(indices_out, d_idx, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream);
    if (!e) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_q); cudaFree(d_off); cudaFree(d_idx);
    KPL_CUDA(e);
    for (int64_t k = 0; k < m; ++k) std::sort(indices_out + offsets_out[k], indices_out + offsets_out[k + 1]);
    ctx->stats.kernel_launches = ctx->launches;
    return KPL_OK;
}

int kpl_uniform_sample(kpl_ctx* ctx, const float* xyz, int32_t xyz_stride, int64_t n, float leaf, int32_t* idx_out, int64_t* m_out)
{
    if (!ctx || !m_out || (n > 0 && !idx_out)) return KPL_E_INVALID;
    detect_reset(ctx);
    *m_out = 0;
    if (!(leaf > 0.f) || !std::isfinite(leaf)) return fail(ctx, KPL_E_INVALID, "leaf must be > 0");
    if (n < 0 || n > 2147483000ll) return fail(ctx, KPL_E_INVALID, "point count out of range");
    if (n == 0) return KPL_OK;
    int rc = upload_inputs(ctx, xyz, xyz_stride, nullptr, 0, nullptr, n);
    if (rc) return rc;
    KPL_CUDA(launch_bbox(ctx, ctx->in_xyz.p, n, ctx->d_bbox));
    uint32_t hb[8];
    KPL_CUDA(cudaMemcpyAsync(hb, ctx->d_bbox, sizeof hb, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    if (hb[6]) return fail(ctx, KPL_E_NONFINITE, "input cloud holds non-finite points");
    float mn[3], mx[3];
    for (int a = 0; a < 3; ++a) { mn[a] = dec_float(hb[a]); mx[a] = dec_float(hb[3 + a]); }
    KPL_CUDA(ensure(ctx->kp_idx, (size_t)n));
    KPL_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 8 * sizeof(unsigned long long), ctx->stream));
    std::string err;
    cudaError_t e = uniform_sample(ctx, ctx->in_xyz.p, n, leaf, mn, mx, ctx->kp_idx.p, err);
    if (e == cudaErrorInvalidValue && !err.empty()) return fail(ctx, KPL_E_GRID, err);
    KPL_CUDA(e);
    unsigned long long hc[8];
    KPL_CUDA(cudaMemcpyAsync(hc, ctx->counters.p, sizeof hc, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    const int64_t m = (int64_t)(hc[3] & 0xFFFFFFFFull);
    if (m > 0) KPL_CUDA(cudaMemcpyAsync(idx_out, ctx->kp_idx.p, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    *m_out = m;
    ctx->stats.n_points = n; ctx->stats.kernel_launches = ctx->launches;
    return KPL_OK;
}

int kpl_fetch_u8(kpl_ctx* ctx, const char* what, uint8_t* out, int64_t capacity)
{
    if (!ctx || !what || !out) return KPL_E_INVALID;
    const int64_t n = ctx->last_n;
    if (n <= 0) return fail(ctx, KPL_E_INVALID, "nothing to fetch");
    if (strcmp(what, "fragile")) return fail(ctx, KPL_E_INVALID, "unknown fetch target");
    const int64_t bytes = n * ctx->last_nforests;         // forest-major after kpl_detect_forests
    if (capacity < bytes) return fail(ctx, KPL_E_INVALID, "fetch buffer too small");
    if (!ctx->last_has_fragile || ctx->fragile.cap < (size_t)bytes)
        return fail(ctx, KPL_E_INVALID, "the last call did not report fragile splits (kpl_params.report_fragile)");
    KPL_CUDA(cudaSetDevice(ctx->device));
    KPL_CUDA(cudaMemcpyAsync(out, ctx->fragile.p, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return KPL_OK;
}

int kpl_get_timings(const kpl_ctx* ctx, kpl_timings* t)
{
    if (!ctx || !t) return KPL_E_INVALID;
    *t = ctx->timings;
    return KPL_OK;
}

int kpl_get_stats(const kpl_ctx* ctx, kpl_stats* s)
{
    if (!ctx || !s) return KPL_E_INVALID;
    *s = ctx->stats;
    return KPL_OK;
}

int kpl_fetch(kpl_ctx* ctx, const char* what, float* out, int64_t capacity_floats)
{
    if (!ctx || !what || !out) return KPL_E_INVALID;
    const int64_t n = ctx->last_n;
    if (n <= 0) return fail(ctx, KPL_E_INVALID, "nothing to fetch");
    KPL_CUDA(cudaSetDevice(ctx->device));
    if (!strcmp(what, "normals")) {
        if (!ctx->last_has_normals) return fail(ctx, KPL_E_INVALID, "no normals from the last call");
        if (capacity_floats < n * 4) return fail(ctx, KPL_E_INVALID, "fetch buffer too small");
        KPL_CUDA(ensure(ctx->scratch_f, (size_t)n * 4));
        KPL_CUDA(launch_unsort_normals(ctx, n, (float4*)ctx->scratch_f.p));
        KPL_CUDA(cudaMemcpyAsync(out, ctx->scratch_f.p, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    } else if (!strcmp(what, "features")) {
        if (!ctx->last_has_features) return fail(ctx, KPL_E_INVALID, "no feature rows from the last call (kpl_detect keeps them only after kpl_set_keep_intermediates(ctx, 1))");
        const int F = ctx->last_F;
        if (capacity_floats < n * F) return fail(ctx, KPL_E_INVALID, "fetch buffer too small");
        KPL_CUDA(ensure(ctx->scratch_f, (size_t)n * F));
        KPL_CUDA(launch_unsort_rows(ctx, ctx->feat.p, n, F, ctx->scratch_f.p));
        KPL_CUDA(cudaMemcpyAsync(out, ctx->scratch_f.p, (size_t)n * F * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    } else return fail(ctx, KPL_E_INVALID, "unknown fetch target");
    KPL_CUDA(cudaStreamSynchronize(ctx->stream));
    return KPL_OK;
}

}  // extern "C"
