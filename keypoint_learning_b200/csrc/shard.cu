// shard.cu -- one large cloud over the GPUs of a node: x slabs of the canonical grid, halo strips and score
// strips exchanged with the two neighbours over NCCL (ncclSend / ncclRecv over NVLink), keypoints gathered on
// rank 0.  No counterpart in the reference, which drives ONE detector from one thread
// (src/main_test_detector.cpp:123-187); this is the layer a multi-GPU driver of that loop binds to (include/kpl.h).
//
// Why the result is bit-identical to the single-GPU run: slabs are cut at cell-column boundaries of the grid of the
// WHOLE cloud and every rank builds its grid with the global origin, so a point has the same cell -- and inside a
// cell the same rank among its cell mates, because strips are sent in ascending global index -- as in the
// unsharded run.  The canonical accumulation order of every histogram is therefore unchanged.
//
// NCCL is loaded at run time (dlopen "libnccl.so.2"): the library itself links only cudart, and a process that has
// torch's NCCL loaded shares it.
#include <dlfcn.h>
#include <nccl.h>
#include <cub/device/device_radix_sort.cuh>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include "kpl_internal.h"

using namespace kpl;

namespace {

// ---- NCCL entry points, resolved once --------------------------------------------------------------------
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
};

NcclApi* nccl_api(std::string* why = nullptr)
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            api.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) { api.err = std::string("libnccl.so.2 could not be loaded: ") + (dlerror() ? dlerror() : "?"); return; }
        bool ok = true;
        auto sym = [&](const char* n) { void* p = dlsym(api.handle, n); if (!p) { ok = false; api.err = std::string("NCCL symbol missing: ") + n; } return p; };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.Send = (decltype(api.Send))sym("ncclSend");
        api.Recv = (decltype(api.Recv))sym("ncclRecv");
        api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
        api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
        api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
        if (!ok) { dlclose(api.handle); api.handle = nullptr; }
    });
    if (!api.handle && why) *why = api.err;
    return api.handle ? &api : nullptr;
}

// ---- host geometry shared by the plan, the partition and set_slab -----------------------------------------
inline int64_t cell_coord(float v, double org, double cell) { return (int64_t)std::floor(((double)v - org) / cell); }

inline const float* point_at(const float* xyz, int32_t stride, int64_t i)
{
    return reinterpret_cast<const float*>(reinterpret_cast<const char*>(xyz) + (size_t)i * (size_t)stride);
}

}  // namespace

// One record per rank, all-gathered at the end of a detection so that every rank takes the same decision.
struct ShardRecord {
    unsigned long long n_kp;       // keypoints among the owned points
    unsigned long long clipped;    // k-NN searches clipped by a slab face (KPL_E_HALO)
    unsigned long long bad_grid;   // a point outside the forced grid / not finite
    unsigned long long reserved;
};

struct kpl_shard {
    kpl_ctx* ctx = nullptr;
    kpl_slab_plan plan;
    int rank = 0, world = 1;
    bool in_process = false;
    NcclApi* nccl = nullptr;
    ncclComm_t comm = nullptr;
    int64_t n_own = 0, n_l = 0, n_r = 0, n_loc = 0;     // owned / received left / received right / all local points
    int64_t send_l = 0, send_r = 0;                      // strip sizes sent to the left / right neighbour
    ForcedGrid grid{};                                   // local grid: columns [offset[0], offset[0] + dims[0]) of the global grid
    bool has_slab = false;
    bool has_nrm = false;                                // the caller's normals (kpl_shard_set_slab_normals) instead of estimated ones
    DevBuf<float4> loc_xyz;                              // [left halo | owned | right halo]
    DevBuf<float4> loc_nrm;                              // the caller's normals, same layout (has_nrm)
    DevBuf<uint8_t> role;
    DevBuf<int32_t> gidx;                                // global index of every owned point
    DevBuf<int32_t> loc_gidx;                            // global index of every local point, [left halo | owned | right halo]
    DevBuf<int32_t> sel_l, sel_r;                        // owned-local indices of the strips
    DevBuf<float4> sbuf_l, sbuf_r;                       // packed position strips
    DevBuf<float4> snb_l, snb_r;                         // packed normal strips (has_nrm)
    DevBuf<float> ssc_l, ssc_r;                          // packed score strips
    DevBuf<int32_t> sgi_l, sgi_r;                        // global indices of the strip points (sent once per resident slab)
    DevBuf<uint8_t> st_orig;                             // draws-remove NMS states in local original order (halo parts received)
    // packed state strips, two sets used in turn: an in-process peer copy of round k (on the receiver's stream) may still
    // read one while round k + 1 packs the other; the exchange of round k + 1 synchronises every stream before round k + 2
    DevBuf<uint8_t> sst_l[2], sst_r[2];
    int sst = 0;                                         // the set packed last
    DevBuf<unsigned long long> und_all;                  // undecided candidates of every rank after a round (NCCL)
    unsigned long long h_undecided = 0;                  // the same, this rank (in-process group)
    DevBuf<int32_t> kp_local, kp_global, kp_all, kp_sorted;
    DevBuf<uint8_t> sort_tmp;
    DevBuf<ShardRecord> rec, rec_all;
    DevBuf<unsigned long long> sizes, sizes_all;
    std::vector<ShardRecord> h_rec;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    float exchange_ms = 0.f, gather_ms = 0.f;
};

namespace {

#define KS_CUDA(call)                                                                               \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess) {                                                                   \
            char b__[512];                                                                          \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            s->ctx->err = b__;                                                                      \
            return e__ == cudaErrorMemoryAllocation ? KPL_E_NOMEM : KPL_E_CUDA;                     \
        }                                                                                           \
    } while (0)

#define KS_NCCL(call)                                                                               \
    do {                                                                                            \
        ncclResult_t r__ = (call);                                                                  \
        if (r__ != ncclSuccess) {                                                                   \
            char b__[512];                                                                          \
            snprintf(b__, sizeof b__, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, s->nccl->GetErrorString(r__)); \
            s->ctx->err = b__;                                                                      \
            return KPL_E_NCCL;                                                                      \
        }                                                                                           \
    } while (0)

int sfail(kpl_shard* s, int code, const std::string& msg)
{
    s->ctx->err = msg;
    return code;
}

template <typename T>
void srelease(DevBuf<T>& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

// ---- device kernels of the sharded step ----------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_strip_kernel(const float4* __restrict__ owned, const int32_t* __restrict__ sel, int64_t m,
                                                         float4* __restrict__ out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < m) out[k] = owned[sel[k]];
}
// both records of a strip point when the caller gave the normals: one launch per side, as without them
__global__ void __launch_bounds__(256) pack_strip_normals_kernel(const float4* __restrict__ owned, const float4* __restrict__ owned_nrm,
                                                                 const int32_t* __restrict__ sel, int64_t m, float4* __restrict__ out,
                                                                 float4* __restrict__ out_nrm)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < m) {
        const int32_t i = sel[k];
        out[k] = owned[i];
        out_nrm[k] = owned_nrm[i];
    }
}
__global__ void __launch_bounds__(256) pack_scores_kernel(const float* __restrict__ owned_scores, const int32_t* __restrict__ sel, int64_t m,
                                                          float* __restrict__ out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < m) out[k] = owned_scores[sel[k]];
}
__global__ void __launch_bounds__(256) pack_states_kernel(const uint8_t* __restrict__ owned_states, const int32_t* __restrict__ sel, int64_t m,
                                                          uint8_t* __restrict__ out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < m) out[k] = owned_states[sel[k]];
}
// draws-remove states of the owned points, cell-sorted -> local original order (the order the strips are selected in)
__global__ void __launch_bounds__(256) owned_states_kernel(const float4* __restrict__ s_pos, const uint8_t* __restrict__ s_role,
                                                           const uint8_t* __restrict__ s_state, int64_t n, uint8_t* __restrict__ st_orig)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n && s_role[i] == KPL_ROLE_OWNED) st_orig[__float_as_uint(s_pos[i].w)] = s_state[i];
}
// states of halo points (their owners' decisions) arrived in local original order, as the scores do
__global__ void __launch_bounds__(256) halo_states_kernel(const float4* __restrict__ s_pos, const uint8_t* __restrict__ s_role,
                                                          const uint8_t* __restrict__ st_orig, int64_t n, uint8_t* __restrict__ s_state)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n && s_role[i] == KPL_ROLE_HALO) s_state[i] = st_orig[__float_as_uint(s_pos[i].w)];
}
// scores of halo points arrived in original (local) order; NMS reads the cell-sorted copy
__global__ void __launch_bounds__(256) halo_scores_kernel(const float4* __restrict__ s_pos, const uint8_t* __restrict__ s_role,
                                                          const float* __restrict__ score, int64_t n, float* __restrict__ s_score)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n && s_role[i] == KPL_ROLE_HALO) s_score[i] = score[__float_as_uint(s_pos[i].w)];
}
__global__ void __launch_bounds__(256) to_global_kernel(const int32_t* __restrict__ kp_local, const unsigned long long* __restrict__ counters,
                                                        const int32_t* __restrict__ gidx, int64_t n_l, int64_t n, int32_t* __restrict__ kp_global)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t cnt = (int64_t)(counters[3] & 0xFFFFFFFFull);
    if (i < n && i < cnt) kp_global[i] = gidx[kp_local[i] - n_l];
}
__global__ void record_kernel(const unsigned long long* __restrict__ counters, const uint32_t* __restrict__ bbox, ShardRecord* __restrict__ rec)
{
    rec->n_kp = counters[3] & 0xFFFFFFFFull;
    rec->clipped = counters[9];
    rec->bad_grid = bbox[7];
    rec->reserved = 0;
}

// ---- transport -------------------------------------------------------------------------------------------------
// A call drives the ranks S[0..n): the one rank of an NCCL communicator, or every rank of an in-process group from
// one host thread.  Errors are reported on S[0]'s context.
int on_rank(kpl_shard** S, int r, int rc)
{
    if (rc && r) S[0]->ctx->err = S[r]->ctx->err;
    return rc;
}

// f on every rank of the call, in rank order, up to the first failure
template <typename F>
int each_rank(kpl_shard** S, int n, F f)
{
    for (int r = 0; r < n; ++r)
        if (int rc = f(S[r])) return on_rank(S, r, rc);
    return KPL_OK;
}

// what an exchange moves: positions (with the caller's normals, when given) and scores every detection, draws-remove
// states every resolution round, global indices once per resident slab
enum class Strip { positions, scores, states, gidx };

// the buffers of one exchange: the packed strips a rank sends, the ends of its local array that receive
struct Strips {
    const void *send_l, *send_r;
    void *recv_l, *recv_r;
    size_t item;
};

// the strip sets one exchange of `kind` moves (out[0..return value)): the normal strips travel with the positions
int strips(kpl_shard* t, Strip kind, Strips* out)
{
    const int64_t hi = t->n_l + t->n_own;
    switch (kind) {
    case Strip::scores: out[0] = {t->ssc_l.p, t->ssc_r.p, t->ctx->score.p, t->ctx->score.p + hi, sizeof(float)}; return 1;
    case Strip::states: out[0] = {t->sst_l[t->sst].p, t->sst_r[t->sst].p, t->st_orig.p, t->st_orig.p + hi, sizeof(uint8_t)}; return 1;
    case Strip::gidx: out[0] = {t->sgi_l.p, t->sgi_r.p, t->loc_gidx.p, t->loc_gidx.p + hi, sizeof(int32_t)}; return 1;
    default:
        out[0] = {t->sbuf_l.p, t->sbuf_r.p, t->loc_xyz.p, t->loc_xyz.p + hi, sizeof(float4)};
        if (!t->has_nrm) return 1;
        out[1] = {t->snb_l.p, t->snb_r.p, t->loc_nrm.p, t->loc_nrm.p + hi, sizeof(float4)};
        return 2;
    }
}

// Strips of one kind with both neighbours: a rank receives the right strip of its left neighbour and the left strip of
// its right neighbour.  NCCL: grouped ncclSend / ncclRecv on the context stream.  In-process group: every stream is
// synchronised, then peer copies.
int exchange(kpl_shard** S, int n, Strip kind)
{
    kpl_shard* s = S[0];
    Strips b[2], p[2];
    if (!s->in_process) {
        const int nb = strips(s, kind, b);
        cudaStream_t st = s->ctx->stream;
        KS_NCCL(s->nccl->GroupStart());
        for (int k = 0; k < nb; ++k) {
            if (s->rank > 0) {
                if (s->send_l) KS_NCCL(s->nccl->Send(b[k].send_l, (size_t)s->send_l * b[k].item, ncclChar, s->rank - 1, s->comm, st));
                if (s->n_l) KS_NCCL(s->nccl->Recv(b[k].recv_l, (size_t)s->n_l * b[k].item, ncclChar, s->rank - 1, s->comm, st));
            }
            if (s->rank < s->world - 1) {
                if (s->send_r) KS_NCCL(s->nccl->Send(b[k].send_r, (size_t)s->send_r * b[k].item, ncclChar, s->rank + 1, s->comm, st));
                if (s->n_r) KS_NCCL(s->nccl->Recv(b[k].recv_r, (size_t)s->n_r * b[k].item, ncclChar, s->rank + 1, s->comm, st));
            }
        }
        KS_NCCL(s->nccl->GroupEnd());
        return KPL_OK;
    }
    for (int r = 0; r < n; ++r) {
        kpl_ctx* c = S[r]->ctx;
        if (cudaSetDevice(c->device) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
            return sfail(s, KPL_E_CUDA, "kpl_shard_detect_group: stream synchronisation failed");
        c->syncs++;
    }
    for (int r = 0; r < n; ++r) {
        kpl_shard* t = S[r];
        const int nb = strips(t, kind, b);
        cudaError_t e = cudaSetDevice(t->ctx->device);
        if (!e && r > 0 && t->n_l) {
            strips(S[r - 1], kind, p);
            for (int k = 0; !e && k < nb; ++k)
                e = cudaMemcpyAsync(b[k].recv_l, p[k].send_r, (size_t)t->n_l * b[k].item, cudaMemcpyDefault, t->ctx->stream);
        }
        if (!e && r < n - 1 && t->n_r) {
            strips(S[r + 1], kind, p);
            for (int k = 0; !e && k < nb; ++k)
                e = cudaMemcpyAsync(b[k].recv_r, p[k].send_l, (size_t)t->n_r * b[k].item, cudaMemcpyDefault, t->ctx->stream);
        }
        if (e) return sfail(s, KPL_E_CUDA, std::string("peer copy: ") + cudaGetErrorString(e));
    }
    return KPL_OK;
}

// The keypoint lists of all ranks into rank 0's kp_all, in rank order: NCCL send / receive, or peer copies.
int gather_keypoints(kpl_shard** S, int n, const std::vector<int64_t>& counts)
{
    kpl_shard* s = S[0];
    cudaStream_t st = s->ctx->stream;
    if (s->in_process) {
        int64_t off = 0;
        for (int r = 0; r < n; ++r) {
            if (counts[(size_t)r]) KS_CUDA(cudaMemcpyAsync(s->kp_all.p + off, S[r]->kp_global.p, (size_t)counts[(size_t)r] * sizeof(int32_t), cudaMemcpyDefault, st));
            off += counts[(size_t)r];
        }
        return KPL_OK;
    }
    KS_NCCL(s->nccl->GroupStart());
    if (s->rank == 0) {
        int64_t off = counts[0];
        for (int p = 1; p < s->world; ++p) {
            if (counts[(size_t)p]) KS_NCCL(s->nccl->Recv(s->kp_all.p + off, (size_t)counts[(size_t)p], ncclInt32, p, s->comm, st));
            off += counts[(size_t)p];
        }
    } else if (counts[(size_t)s->rank]) {
        KS_NCCL(s->nccl->Send(s->kp_global.p, (size_t)counts[(size_t)s->rank], ncclInt32, 0, s->comm, st));
    }
    KS_NCCL(s->nccl->GroupEnd());
    if (s->rank == 0 && counts[0]) KS_CUDA(cudaMemcpyAsync(s->kp_all.p, s->kp_global.p, (size_t)counts[0] * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return KPL_OK;
}

// ---- the phases of one detection (everything is enqueued on the context stream) --------------------------------
// the per-call reset of the rank's context, then its position strips (and normal strips)
int phase_pack(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    detect_reset(c);
    KS_CUDA(cudaSetDevice(c->device));
    KS_CUDA(cudaEventRecord(s->ev[0], c->stream));
    const float4* owned = s->loc_xyz.p + s->n_l;
    const float4* owned_nrm = s->has_nrm ? s->loc_nrm.p + s->n_l : nullptr;
    const int64_t m[2] = {s->send_l, s->send_r};
    const int32_t* sel[2] = {s->sel_l.p, s->sel_r.p};
    float4* out[2] = {s->sbuf_l.p, s->sbuf_r.p};
    float4* out_nrm[2] = {s->snb_l.p, s->snb_r.p};
    for (int k = 0; k < 2; ++k) {
        if (!m[k]) continue;
        const unsigned blocks = (unsigned)((m[k] + 255) / 256);
        if (s->has_nrm) pack_strip_normals_kernel<<<blocks, 256, 0, c->stream>>>(owned, owned_nrm, sel[k], m[k], out[k], out_nrm[k]);
        else pack_strip_kernel<<<blocks, 256, 0, c->stream>>>(owned, sel[k], m[k], out[k]);
        KS_CUDA(cudaGetLastError());
    }
    return KPL_OK;
}

int phase_score(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    KS_CUDA(cudaSetDevice(c->device));
    KS_CUDA(cudaEventRecord(s->ev[1], c->stream));
    int rc = detect_begin(c);
    if (rc) return rc;
    c->launches += 2;
    if ((rc = prepare_grid(c, s->loc_xyz.p, s->has_nrm ? s->loc_nrm.p : nullptr, s->role.p, s->n_loc, &s->grid))) return rc;
    if ((rc = detect_score_phase(c, s->has_nrm, true, s->n_loc, 1))) return rc;
    KS_CUDA(cudaEventRecord(s->ev[2], c->stream));
    const float* owned_scores = c->score.p + s->n_l;
    if (s->send_l) pack_scores_kernel<<<(unsigned)((s->send_l + 255) / 256), 256, 0, c->stream>>>(owned_scores, s->sel_l.p, s->send_l, s->ssc_l.p);
    if (s->send_r) pack_scores_kernel<<<(unsigned)((s->send_r + 255) / 256), 256, 0, c->stream>>>(owned_scores, s->sel_r.p, s->send_r, s->ssc_r.p);
    KS_CUDA(cudaGetLastError());
    c->launches += 2;
    return KPL_OK;
}

bool draws_remove(const kpl_ctx* c) { return c->params.non_maxima && c->params.draws_remove; }

// the draws-remove states of the owned strip points, packed for the neighbours
int pack_states(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    if (s->send_l + s->send_r == 0) return KPL_OK;
    owned_states_kernel<<<(unsigned)((s->n_loc + 255) / 256), 256, 0, c->stream>>>(c->s_pos.p, c->s_role.p, c->s_state.p, s->n_loc, s->st_orig.p);
    const uint8_t* owned = s->st_orig.p + s->n_l;
    s->sst ^= 1;
    if (s->send_l) pack_states_kernel<<<(unsigned)((s->send_l + 255) / 256), 256, 0, c->stream>>>(owned, s->sel_l.p, s->send_l, s->sst_l[s->sst].p);
    if (s->send_r) pack_states_kernel<<<(unsigned)((s->send_r + 255) / 256), 256, 0, c->stream>>>(owned, s->sel_r.p, s->send_r, s->sst_r[s->sst].p);
    KS_CUDA(cudaGetLastError());
    c->launches += 1 + (s->send_l > 0) + (s->send_r > 0);
    return KPL_OK;
}

// keypoints (owned points only) to global indices, and the rank's record
int phase_records(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    to_global_kernel<<<(unsigned)((s->n_own + 255) / 256), 256, 0, c->stream>>>(s->kp_local.p, c->counters.p, s->gidx.p, s->n_l, s->n_own, s->kp_global.p);
    record_kernel<<<1, 1, 0, c->stream>>>(c->counters.p, (const uint32_t*)c->d_bbox, s->rec.p);
    KS_CUDA(cudaGetLastError());
    c->launches += 2;
    return KPL_OK;
}

// Threshold + NMS.  Draws-remove: only the classification here; the resolution rounds need the neighbours' decisions and
// run over all ranks (nms_draws_rounds), then phase_draws_keypoints.
int phase_nms(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    KS_CUDA(cudaSetDevice(c->device));             // an in-process group drives ranks on several devices from one thread
    KS_CUDA(cudaEventRecord(s->ev[3], c->stream));
    if (s->n_l + s->n_r > 0)
        halo_scores_kernel<<<(unsigned)((s->n_loc + 255) / 256), 256, 0, c->stream>>>(c->s_pos.p, c->s_role.p, c->score.p, s->n_loc, c->s_score.p);
    c->launches++;
    if (draws_remove(c)) {
        KS_CUDA(launch_nms_draws_classify(c, s->n_loc, true, c->s_score.p, c->params.threshold));
        return pack_states(s);
    }
    int rc = detect_nms_phase(c, true, s->n_loc, 1, nullptr, s->kp_local.p);
    return rc ? rc : phase_records(s);
}

// one draws-remove resolution round of the owned points, on the halo states the last exchange brought in
int phase_draws_round(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    KS_CUDA(cudaSetDevice(c->device));
    if (s->n_l + s->n_r > 0) {
        halo_states_kernel<<<(unsigned)((s->n_loc + 255) / 256), 256, 0, c->stream>>>(c->s_pos.p, c->s_role.p, s->st_orig.p, s->n_loc, c->s_state.p);
        KS_CUDA(cudaGetLastError());
        c->launches++;
    }
    KS_CUDA(launch_nms_draws_round(c, s->n_loc, true, s->loc_gidx.p, c->s_score.p, c->params.threshold));
    if (s->in_process)      // read by the host after the next exchange, which synchronises every stream of the group
        KS_CUDA(cudaMemcpyAsync(&s->h_undecided, c->counters.p + 6, sizeof s->h_undecided, cudaMemcpyDeviceToHost, c->stream));
    return pack_states(s);
}

// The draws-remove rounds over the slabs.  After the classification and after every round, the owned states of the
// strip points go to the neighbours, so that a halo point always holds its owner's decision (a stale one only postpones
// a decision).  Every rank stops on the same global count of undecided candidates, within the same cap: no rank is left
// waiting in a collective.  One host synchronisation per round.
int nms_draws_rounds(kpl_shard** S, int n)
{
    kpl_shard* s = S[0];
    kpl_ctx* c = s->ctx;
    if (!draws_remove(c)) return KPL_OK;
    int rc = exchange(S, n, Strip::states);
    for (int round = 0; !rc && round < nms_round_cap(s->plan.n_points); ++round) {
        if ((rc = each_rank(S, n, phase_draws_round)) || (rc = exchange(S, n, Strip::states))) return rc;
        unsigned long long undecided = 0;
        if (s->in_process) {
            for (int r = 0; r < n; ++r) undecided += S[r]->h_undecided;
        } else {
            std::vector<unsigned long long> all((size_t)s->world);
            KS_NCCL(s->nccl->AllGather(c->counters.p + 6, s->und_all.p, 1, ncclUint64, s->comm, c->stream));
            KS_CUDA(cudaMemcpyAsync(all.data(), s->und_all.p, all.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
            KS_CUDA(cudaStreamSynchronize(c->stream));
            c->syncs++;
            for (unsigned long long u : all) undecided += u;
        }
        if (undecided == 0) break;
    }
    return rc;
}

// draws-remove: flags of the decided owned points, compaction, records
int phase_draws_keypoints(kpl_shard* s)
{
    kpl_ctx* c = s->ctx;
    if (!draws_remove(c)) return KPL_OK;
    KS_CUDA(cudaSetDevice(c->device));
    KS_CUDA(launch_nms_draws_flags(c, s->n_loc, true, 0));
    KS_CUDA(launch_compact(c, s->n_loc, s->kp_local.p));
    return phase_records(s);
}

// after the records of all ranks reached the host: the same verdict on every rank
int verdict(kpl_shard* s, int64_t& total, std::vector<int64_t>& counts)
{
    total = 0;
    counts.assign((size_t)s->world, 0);
    unsigned long long clipped = 0, bad = 0;
    for (int r = 0; r < s->world; ++r) {
        counts[(size_t)r] = (int64_t)s->h_rec[(size_t)r].n_kp;
        total += counts[(size_t)r];
        clipped += s->h_rec[(size_t)r].clipped;
        bad += s->h_rec[(size_t)r].bad_grid;
    }
    if (bad) return sfail(s, KPL_E_GRID, "a point lies outside its slab grid (or is not finite)");
    if (clipped) {
        char b[256];
        snprintf(b, sizeof b, "%llu k-NN normals that kept points depend on were clipped by a slab face: widen normal_support_cells (now %d)",
                 clipped, s->plan.normal_support_cells);
        return sfail(s, KPL_E_HALO, b);
    }
    return KPL_OK;
}

int sort_keypoints(kpl_shard* s, int64_t total)
{
    kpl_ctx* c = s->ctx;
    if (total <= 0) return KPL_OK;
    int end_bit = 1;
    while (end_bit < 32 && (1ll << end_bit) < s->plan.n_points) end_bit++;
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const uint32_t*)s->kp_all.p, (uint32_t*)s->kp_sorted.p, (int)total, 0, end_bit, c->stream);
    KS_CUDA(ensure(s->sort_tmp, bytes));
    bytes = s->sort_tmp.cap;
    KS_CUDA(cub::DeviceRadixSort::SortKeys(s->sort_tmp.p, bytes, (const uint32_t*)s->kp_all.p, (uint32_t*)s->kp_sorted.p, (int)total, 0, end_bit, c->stream));
    c->launches += 1 + (end_bit + 7) / 8;
    return KPL_OK;
}

int check_ready(kpl_shard* s)
{
    if (!s || !s->ctx) return KPL_E_INVALID;
    if (!s->has_slab) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab was not called");
    // estimated radius-mode normals (hpp:130-137) need every neighbour within r_feat of a point whose normal matters: the
    // halo must then be two search reaches wide, which no device check can verify after the fact
    if (s->world > 1 && !s->has_nrm && s->ctx->params.normals_mode == KPL_NORMALS_RADIUS && s->plan.normal_support_cells < s->plan.reach_feat)
        return sfail(s, KPL_E_HALO, "radius-mode normals need normal_support_cells >= reach_feat (the whole r_feat ball of every halo point that matters)");
    return detect_check(s->ctx, s->n_loc, 1, false);
}

void finish_timings(kpl_shard* s, bool gathered)
{
    float a = 0.f, b = 0.f, g = 0.f;
    cudaEventElapsedTime(&a, s->ev[0], s->ev[1]);
    cudaEventElapsedTime(&b, s->ev[2], s->ev[3]);
    if (gathered) cudaEventElapsedTime(&g, s->ev[4], s->ev[5]);
    s->exchange_ms = a + b;
    s->gather_ms = g;
    (void)cudaGetLastError();
}

int copy_out(kpl_shard* s, float* scores_owned_out, int32_t* kp_global_out, int64_t kp_capacity, int64_t total)
{
    kpl_ctx* c = s->ctx;
    KS_CUDA(cudaSetDevice(c->device));
    if (scores_owned_out)
        KS_CUDA(cudaMemcpyAsync(scores_owned_out, c->score.p + s->n_l, (size_t)s->n_own * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (s->rank == 0 && kp_global_out && total > 0) {
        if (kp_capacity < total) return sfail(s, KPL_E_INVALID, "kp_global_out is too small");
        KS_CUDA(cudaMemcpyAsync(kp_global_out, s->kp_sorted.p, (size_t)total * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    }
    KS_CUDA(cudaStreamSynchronize(c->stream));
    c->syncs++;
    c->stats.host_syncs = c->syncs;
    c->stats.kernel_launches = c->launches;
    return KPL_OK;
}

// One sharded detection over the ranks S[0..n) of this call.  The verdict over the records of all ranks comes before a
// rank-local error of detect_finish, so that every rank returns the same status.
int detect_step(kpl_shard** S, int n, float* const* scores_owned_out, int32_t* kp_global_out, int64_t kp_capacity, int64_t* n_kp_out)
{
    kpl_shard* s = S[0];
    kpl_ctx* c = s->ctx;
    int rc;
    if ((rc = each_rank(S, n, check_ready)) || (rc = each_rank(S, n, phase_pack)) || (rc = exchange(S, n, Strip::positions)) ||
        (rc = each_rank(S, n, phase_score)) || (rc = exchange(S, n, Strip::scores)) || (rc = each_rank(S, n, phase_nms)) ||
        (rc = nms_draws_rounds(S, n)) || (rc = each_rank(S, n, phase_draws_keypoints)))
        return rc;
    // the records of all ranks to S[0]'s host: all-gathered, or one copy per in-process rank
    if (!s->in_process) {
        KS_NCCL(s->nccl->AllGather(s->rec.p, s->rec_all.p, sizeof(ShardRecord), ncclChar, s->comm, c->stream));
        KS_CUDA(cudaMemcpyAsync(s->h_rec.data(), s->rec_all.p, (size_t)s->world * sizeof(ShardRecord), cudaMemcpyDeviceToHost, c->stream));
    }
    int local_err = KPL_OK, err_rank = 0;
    for (int r = 0; r < n; ++r) {
        kpl_ctx* t = S[r]->ctx;
        if (s->in_process) {
            KS_CUDA(cudaSetDevice(t->device));
            KS_CUDA(cudaMemcpyAsync(&s->h_rec[(size_t)r], S[r]->rec.p, sizeof(ShardRecord), cudaMemcpyDeviceToHost, t->stream));
        }
        int64_t local_kp = 0;
        const int e = detect_finish(t, S[r]->n_loc, &local_kp);      // the synchronisation; also fills stats / timings of the rank
        if (e && !local_err && e != KPL_E_HALO && e != KPL_E_GRID) { local_err = e; err_rank = r; }
    }
    int64_t total = 0;
    std::vector<int64_t> counts;
    if ((rc = verdict(s, total, counts))) return rc;                   // identical on every rank: nobody is left waiting in a collective
    if (local_err) return on_rank(S, err_rank, local_err);
    if (n_kp_out) *n_kp_out = total;
    // keypoint lists to rank 0 (sizes are known everywhere now), then one sort into ascending global index
    KS_CUDA(cudaSetDevice(c->device));
    KS_CUDA(cudaEventRecord(s->ev[4], c->stream));
    if (s->rank == 0) { KS_CUDA(ensure(s->kp_all, (size_t)total + 1)); KS_CUDA(ensure(s->kp_sorted, (size_t)total + 1)); }
    if ((rc = gather_keypoints(S, n, counts))) return rc;
    if (s->rank == 0 && (rc = sort_keypoints(s, total))) return rc;
    KS_CUDA(cudaEventRecord(s->ev[5], c->stream));
    for (int r = 0; r < n; ++r) {
        rc = copy_out(S[r], scores_owned_out ? scores_owned_out[r] : nullptr, r == 0 ? kp_global_out : nullptr, kp_capacity, total);
        if (rc) return on_rank(S, r, rc);
        finish_timings(S[r], r == 0);
    }
    return KPL_OK;
}

}  // namespace

extern "C" {

// ---------------------------------------------------------------------------------------------------------------
// host-only planning
// ---------------------------------------------------------------------------------------------------------------
int kpl_slab_plan_make(const float* xyz, int32_t stride, int64_t n, const kpl_params* p, int32_t world, int32_t normal_support_cells,
                       kpl_slab_plan* out)
{
    if (!xyz || !p || !out || n < 1 || world < 1 || world > KPL_MAX_RANKS || normal_support_cells < 0) return KPL_E_INVALID;
    if (stride < 12 || (stride & 3) || !(p->radius_features > 0.f) || p->cells_per_radius < 1) return KPL_E_INVALID;
    memset(out, 0, sizeof *out);
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int64_t i = 0; i < n; ++i) {
        const float* v = point_at(xyz, stride, i);
        for (int a = 0; a < 3; ++a) {
            if (!std::isfinite(v[a])) return KPL_E_NONFINITE;
            lo[a] = std::min(lo[a], v[a]); hi[a] = std::max(hi[a], v[a]);
        }
    }
    // the canonical grid of the whole cloud: the plan IS the grid of the unsharded run
    const double cell = canonical_cell(*p);
    out->cell = cell; out->world = world; out->n_points = n;
    double ncells = 1.0;
    for (int a = 0; a < 3; ++a) {
        out->origin[a] = (double)lo[a];
        out->dims[a] = grid_dim(lo[a], hi[a], cell);
        ncells *= (double)out->dims[a];
    }
    if (ncells > 2147483646.0) return KPL_E_GRID;
    out->reach_feat = grid_reach(p->radius_features, cell);
    out->reach_nms = grid_reach(p->radius_nms, cell);
    out->normal_support_cells = normal_support_cells;
    out->halo = std::max(out->reach_feat + normal_support_cells, out->reach_nms);
    const int nx = out->dims[0], ny = out->dims[1], nz = out->dims[2];
    const int H = out->halo;
    if (world > 1 && (int64_t)nx < (int64_t)world * H) return KPL_E_INVALID;

    // ---- cost of every cell column: neighbour pairs of its points + points
    std::vector<double> col_pts((size_t)nx, 0.0), col_pairs((size_t)nx, 0.0);
    const bool model_pairs = ncells <= 48.0e6;
    if (model_pairs) {
        const size_t N = (size_t)ncells;
        std::vector<float> cnt(N, 0.f), box(N), tmp(N);
        for (int64_t i = 0; i < n; ++i) {
            const float* v = point_at(xyz, stride, i);
            const int64_t cx = cell_coord(v[0], out->origin[0], cell), cy = cell_coord(v[1], out->origin[1], cell), cz = cell_coord(v[2], out->origin[2], cell);
            cnt[((size_t)cz * ny + cy) * nx + cx] += 1.f;
        }
        // separable box sum over +-reach_feat cells (running window along each axis)
        const int R = out->reach_feat;
        auto pass = [&](const std::vector<float>& src, std::vector<float>& dst, size_t len, size_t step, size_t lines, auto line_base) {
            for (size_t l = 0; l < lines; ++l) {
                const size_t b = line_base(l);
                double acc = 0.0;
                for (size_t k = 0; k < std::min(len, (size_t)R + 1); ++k) acc += src[b + k * step];
                for (size_t k = 0; k < len; ++k) {
                    dst[b + k * step] = (float)acc;
                    if (k + R + 1 < len) acc += src[b + (k + R + 1) * step];
                    if (k >= (size_t)R) acc -= src[b + (k - R) * step];
                }
            }
        };
        pass(cnt, box, (size_t)nx, 1, (size_t)ny * nz, [&](size_t l) { return l * (size_t)nx; });
        pass(box, tmp, (size_t)ny, (size_t)nx, (size_t)nx * nz, [&](size_t l) { return (l / nx) * (size_t)nx * ny + (l % nx); });
        pass(tmp, box, (size_t)nz, (size_t)nx * ny, (size_t)nx * ny, [&](size_t l) { return l; });
        for (size_t k = 0; k < N; ++k)
            if (cnt[k] > 0.f) { col_pairs[k % (size_t)nx] += (double)cnt[k] * (double)box[k]; col_pts[k % (size_t)nx] += (double)cnt[k]; }
    } else {
        for (int64_t i = 0; i < n; ++i) col_pts[(size_t)cell_coord(point_at(xyz, stride, i)[0], out->origin[0], cell)] += 1.0;
        col_pairs = col_pts;
    }
    std::vector<double> cum_pairs((size_t)nx + 1, 0.0), cum_pts((size_t)nx + 1, 0.0);
    for (int x = 0; x < nx; ++x) { cum_pairs[(size_t)x + 1] = cum_pairs[(size_t)x] + col_pairs[(size_t)x]; cum_pts[(size_t)x + 1] = cum_pts[(size_t)x] + col_pts[(size_t)x]; }
    // per-point work of everything a rank holds (grid build, k-NN normals): ~7 % of scoring an average point
    const double per_point = 0.07 * cum_pairs[(size_t)nx] / std::max(1.0, cum_pts[(size_t)nx]);
    auto clampx = [&](int x) { return (size_t)std::min(std::max(x, 0), nx); };
    auto cost = [&](int c0, int c1) {
        return (cum_pairs[clampx(c1)] - cum_pairs[clampx(c0)]) + per_point * (cum_pts[clampx(c1 + H)] - cum_pts[clampx(c0 - H)]);
    };
    // smallest per-rank cost bound that `world` slabs of >= H columns can meet (bisection over a greedy sweep)
    auto greedy = [&](double limit, std::vector<int>& cuts) {
        cuts.assign(1, 0);
        int c0 = 0;
        for (int r = 0; r < world && c0 < nx; ++r) {
            const int left = world - 1 - r;                       // slabs still to place after this one
            int c1 = std::min(c0 + std::max(H, 1), nx);
            if (r == world - 1) c1 = nx;
            else {
                while (c1 < nx - left * H && cost(c0, c1 + 1) <= limit) ++c1;
                c1 = std::min(c1, nx - left * std::max(H, 1));
                c1 = std::max(c1, c0 + 1);
            }
            cuts.push_back(c1);
            c0 = c1;
        }
        if ((int)cuts.size() != world + 1 || cuts.back() != nx) return false;
        for (int r = 0; r < world; ++r) if (cost(cuts[(size_t)r], cuts[(size_t)r + 1]) > limit) return false;
        return true;
    };
    std::vector<int> cuts, best;
    double lo_t = 0.0, hi_t = cost(0, nx) * 1.0001 + 1.0;
    if (!greedy(hi_t, best)) return KPL_E_INVALID;
    for (int it = 0; it < 60; ++it) {
        const double mid = 0.5 * (lo_t + hi_t);
        if (greedy(mid, cuts)) { hi_t = mid; best = cuts; } else lo_t = mid;
    }
    for (int r = 0; r <= world; ++r) out->cuts[r] = best[(size_t)r];
    for (int r = 0; r < world; ++r) {
        out->cost[r] = cost(best[(size_t)r], best[(size_t)r + 1]);
        if (world > 1 && best[(size_t)r + 1] - best[(size_t)r] < H) return KPL_E_INVALID;
    }
    return KPL_OK;
}

int kpl_slab_partition(const kpl_slab_plan* plan, const float* xyz, int32_t stride, int64_t n, int32_t rank, int32_t* idx_out, int64_t* m_out)
{
    if (!plan || !xyz || !idx_out || !m_out || rank < 0 || rank >= plan->world || stride < 12 || (stride & 3)) return KPL_E_INVALID;
    const int64_t c0 = plan->cuts[rank], c1 = plan->cuts[rank + 1];
    int64_t m = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t cx = cell_coord(point_at(xyz, stride, i)[0], plan->origin[0], plan->cell);
        if (cx >= c0 && cx < c1) idx_out[m++] = (int32_t)i;
    }
    *m_out = m;
    return KPL_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// per-rank job
// ---------------------------------------------------------------------------------------------------------------
int kpl_nccl_unique_id(void* id128_out)
{
    if (!id128_out) return KPL_E_INVALID;
    NcclApi* api = nccl_api();
    if (!api) return KPL_E_NCCL;
    ncclUniqueId id;
    if (api->GetUniqueId(&id) != ncclSuccess) return KPL_E_NCCL;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128_out, &id, sizeof id);
    return KPL_OK;
}

int kpl_shard_create(kpl_ctx* ctx, const kpl_slab_plan* plan, int32_t rank, const void* nccl_id128, kpl_shard** out)
{
    if (!ctx || !plan || !out || rank < 0 || rank >= plan->world) return KPL_E_INVALID;
    *out = nullptr;
    kpl_shard* s = new (std::nothrow) kpl_shard();
    if (!s) return KPL_E_NOMEM;
    s->ctx = ctx; s->plan = *plan; s->rank = rank; s->world = plan->world;
    s->in_process = nccl_id128 == nullptr;
    s->h_rec.resize((size_t)s->world);
    bool ok = cudaSetDevice(ctx->device) == cudaSuccess;
    for (int i = 0; ok && i < 6; ++i) ok = cudaEventCreate(&s->ev[i]) == cudaSuccess;
    ok = ok && ensure(s->rec, 1) == cudaSuccess && ensure(s->rec_all, (size_t)s->world) == cudaSuccess &&
         ensure(s->sizes, 3) == cudaSuccess && ensure(s->sizes_all, 3 * (size_t)s->world) == cudaSuccess &&
         ensure(s->und_all, (size_t)s->world) == cudaSuccess;
    if (!ok) { ctx->err = "kpl_shard_create: CUDA resources"; kpl_shard_destroy(s); return KPL_E_CUDA; }
    if (!s->in_process) {
        std::string why;
        s->nccl = nccl_api(&why);
        if (!s->nccl) { ctx->err = "NCCL is not available: " + why; kpl_shard_destroy(s); return KPL_E_NCCL; }
        ncclUniqueId id;
        memcpy(&id, nccl_id128, sizeof id);
        ncclResult_t r = s->nccl->CommInitRank(&s->comm, s->world, id, rank);
        if (r != ncclSuccess) {
            ctx->err = std::string("ncclCommInitRank: ") + s->nccl->GetErrorString(r);
            s->comm = nullptr;
            kpl_shard_destroy(s);
            return KPL_E_NCCL;
        }
    }
    *out = s;
    return KPL_OK;
}

int kpl_shard_set_plan(kpl_shard* s, const kpl_slab_plan* plan)
{
    if (!s || !plan) return KPL_E_INVALID;
    if (plan->world != s->world) return sfail(s, KPL_E_INVALID, "kpl_shard_set_plan: the communicator was created for another world size");
    s->plan = *plan;
    s->has_slab = s->has_nrm = false;
    s->n_own = s->n_l = s->n_r = s->n_loc = s->send_l = s->send_r = 0;
    return KPL_OK;
}

void kpl_shard_destroy(kpl_shard* s)
{
    if (!s) return;
    if (s->ctx) { cudaSetDevice(s->ctx->device); cudaStreamSynchronize(s->ctx->stream); }
    if (s->comm && s->nccl) s->nccl->CommDestroy(s->comm);
    srelease(s->loc_xyz); srelease(s->role); srelease(s->gidx); srelease(s->loc_gidx); srelease(s->sel_l); srelease(s->sel_r);
    srelease(s->loc_nrm); srelease(s->snb_l); srelease(s->snb_r);
    srelease(s->sbuf_l); srelease(s->sbuf_r); srelease(s->ssc_l); srelease(s->ssc_r); srelease(s->sgi_l); srelease(s->sgi_r);
    srelease(s->st_orig); srelease(s->und_all);
    for (int k = 0; k < 2; ++k) { srelease(s->sst_l[k]); srelease(s->sst_r[k]); }
    srelease(s->kp_local); srelease(s->kp_global); srelease(s->kp_all); srelease(s->kp_sorted); srelease(s->sort_tmp);
    srelease(s->rec); srelease(s->rec_all); srelease(s->sizes); srelease(s->sizes_all);
    for (int i = 0; i < 6; ++i) if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    delete s;
}

// Strip selection on the host (the owned points are host data here anyway), uploads, and -- NCCL groups -- the
// exchange of the strip sizes.  In-process groups exchange their sizes in kpl_shard_detect_group.
static int set_slab_local(kpl_shard* s, const float* xyz, int32_t stride, const int32_t* gidx, int64_t n_own)
{
    kpl_ctx* c = s->ctx;
    if (!xyz || !gidx || n_own < 1) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab: empty slab");
    if (stride < 12 || (stride & 3)) return sfail(s, KPL_E_INVALID, "stride must be a multiple of 4 and >= 12 bytes");
    KS_CUDA(cudaSetDevice(c->device));
    const kpl_slab_plan& L = s->plan;
    const int c0 = L.cuts[s->rank], c1 = L.cuts[s->rank + 1], H = L.halo;
    std::vector<int32_t> sl, sr;
    for (int64_t i = 0; i < n_own; ++i) {
        const int64_t cx = cell_coord(point_at(xyz, stride, i)[0], L.origin[0], L.cell);
        if (cx < c0 || cx >= c1) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab: a point does not belong to this rank's columns");
        if (i > 0 && gidx[i] <= gidx[i - 1]) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab: global indices must be strictly ascending");
        if (s->rank > 0 && cx < c0 + H) sl.push_back((int32_t)i);
        if (s->rank < s->world - 1 && cx >= c1 - H) sr.push_back((int32_t)i);
    }
    s->n_own = n_own; s->send_l = (int64_t)sl.size(); s->send_r = (int64_t)sr.size();
    // the local grid: this rank's columns and the halo columns beyond its interior faces
    const int x0 = s->rank > 0 ? std::max(c0 - H, 0) : 0, x1 = s->rank < s->world - 1 ? std::min(c1 + H, L.dims[0]) : L.dims[0];
    ForcedGrid& g = s->grid;
    for (int a = 0; a < 3; ++a) { g.origin[a] = L.origin[a]; g.dims[a] = L.dims[a]; g.offset[a] = 0; }
    g.dims[0] = x1 - x0; g.offset[0] = x0;
    g.interior_lo = s->rank > 0; g.interior_hi = s->rank < s->world - 1; g.guard_cells = L.normal_support_cells;
    KS_CUDA(ensure(s->gidx, (size_t)n_own));
    KS_CUDA(ensure(s->sel_l, sl.size() + 1)); KS_CUDA(ensure(s->sel_r, sr.size() + 1));
    KS_CUDA(ensure(s->sbuf_l, sl.size() + 1)); KS_CUDA(ensure(s->sbuf_r, sr.size() + 1));
    if (s->has_nrm) { KS_CUDA(ensure(s->snb_l, sl.size() + 1)); KS_CUDA(ensure(s->snb_r, sr.size() + 1)); }
    KS_CUDA(ensure(s->ssc_l, sl.size() + 1)); KS_CUDA(ensure(s->ssc_r, sr.size() + 1));
    for (int k = 0; k < 2; ++k) { KS_CUDA(ensure(s->sst_l[k], sl.size() + 1)); KS_CUDA(ensure(s->sst_r[k], sr.size() + 1)); }
    KS_CUDA(ensure(s->sgi_l, sl.size() + 1)); KS_CUDA(ensure(s->sgi_r, sr.size() + 1));
    std::vector<int32_t> gl(sl.size()), gr(sr.size());
    for (size_t k = 0; k < sl.size(); ++k) gl[k] = gidx[sl[k]];
    for (size_t k = 0; k < sr.size(); ++k) gr[k] = gidx[sr[k]];
    KS_CUDA(ensure(s->kp_local, (size_t)n_own + 1)); KS_CUDA(ensure(s->kp_global, (size_t)n_own + 1));
    KS_CUDA(cudaMemcpyAsync(s->gidx.p, gidx, (size_t)n_own * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    if (!sl.empty()) KS_CUDA(cudaMemcpyAsync(s->sel_l.p, sl.data(), sl.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    if (!sr.empty()) KS_CUDA(cudaMemcpyAsync(s->sel_r.p, sr.data(), sr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    if (!gl.empty()) KS_CUDA(cudaMemcpyAsync(s->sgi_l.p, gl.data(), gl.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    if (!gr.empty()) KS_CUDA(cudaMemcpyAsync(s->sgi_r.p, gr.data(), gr.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    KS_CUDA(cudaStreamSynchronize(c->stream));          // sl / sr / gidx / gl / gr are host buffers of this call
    return KPL_OK;
}

// An in-process rank's owned records, which kpl_shard_set_slab staged at the start of `buf`, move to their place.
static cudaError_t place_owned(kpl_shard* s, DevBuf<float4>& buf)
{
    DevBuf<float4> staged;
    if (s->in_process) std::swap(staged, buf);
    cudaError_t e = ensure(buf, (size_t)s->n_loc);
    if (!e && staged.p) e = cudaMemcpyAsync(buf.p + s->n_l, staged.p, (size_t)s->n_own * sizeof(float4), cudaMemcpyDeviceToDevice, s->ctx->stream);
    if (!e && staged.p) e = cudaStreamSynchronize(s->ctx->stream);
    srelease(staged);
    return e;
}

// [left halo | owned | right halo] once the strip sizes n_l / n_r are known: the local cloud buffer (and the normal
// buffer) and the roles.
static int set_slab_layout(kpl_shard* s, int64_t n_l, int64_t n_r)
{
    kpl_ctx* c = s->ctx;
    s->n_l = n_l; s->n_r = n_r; s->n_loc = n_l + s->n_own + n_r;
    if (s->n_loc > 2147483000ll) return sfail(s, KPL_E_INVALID, "slab too large");
    KS_CUDA(cudaSetDevice(c->device));
    KS_CUDA(place_owned(s, s->loc_xyz));
    if (s->has_nrm) KS_CUDA(place_owned(s, s->loc_nrm));
    KS_CUDA(ensure(s->role, (size_t)s->n_loc));
    KS_CUDA(cudaMemsetAsync(s->role.p, KPL_ROLE_HALO, (size_t)s->n_loc, c->stream));
    KS_CUDA(cudaMemsetAsync(s->role.p + n_l, KPL_ROLE_OWNED, (size_t)s->n_own, c->stream));
    // global indices: the owned part here, the halo parts by the gidx exchange that follows the layout of every rank
    KS_CUDA(ensure(s->loc_gidx, (size_t)s->n_loc));
    KS_CUDA(cudaMemcpyAsync(s->loc_gidx.p + n_l, s->gidx.p, (size_t)s->n_own * sizeof(int32_t), cudaMemcpyDeviceToDevice, c->stream));
    KS_CUDA(ensure(s->st_orig, (size_t)s->n_loc));
    s->has_slab = true;
    return KPL_OK;
}

static bool bad_stride(int32_t stride) { return stride < 12 || (stride & 3); }

// host (possibly strided) -> device float4 records, as the single-GPU upload stages them (capi.cu: upload_vec3)
static cudaError_t upload_records(float4* dst, const float* src, int32_t stride, int64_t n, cudaStream_t st)
{
    if (stride == 16) return cudaMemcpyAsync(dst, src, (size_t)n * 16, cudaMemcpyHostToDevice, st);
    return cudaMemcpy2DAsync(dst, 16, src, (size_t)stride, stride >= 16 ? 16 : 12, (size_t)n, cudaMemcpyHostToDevice, st);
}

// kpl_shard_set_slab with or without the caller's normals (nrm == nullptr: estimated on the device)
static int set_slab(kpl_shard* s, const float* xyz, int32_t stride, const float* nrm, int32_t nrm_stride, const int32_t* gidx, int64_t n_own)
{
    s->has_slab = false;
    s->has_nrm = nrm != nullptr;
    int rc = set_slab_local(s, xyz, stride, gidx, n_own);
    if (rc) return rc;
    kpl_ctx* c = s->ctx;
    if (s->in_process) {
        // the group driver takes n_l / n_r from the peers; the layout follows there (kpl_shard_detect_group)
        s->n_l = s->n_r = -1;
        KS_CUDA(ensure(s->loc_xyz, (size_t)n_own));
        if (stride == 16) KS_CUDA(cudaMemcpy(s->loc_xyz.p, xyz, (size_t)n_own * 16, cudaMemcpyHostToDevice));
        else KS_CUDA(cudaMemcpy2D(s->loc_xyz.p, 16, xyz, (size_t)stride, 12, (size_t)n_own, cudaMemcpyHostToDevice));
        if (s->has_nrm) {
            KS_CUDA(ensure(s->loc_nrm, (size_t)n_own));
            KS_CUDA(upload_records(s->loc_nrm.p, nrm, nrm_stride, n_own, c->stream));
            KS_CUDA(cudaStreamSynchronize(c->stream));
        }
        return KPL_OK;
    }
    // the strip sizes and whether this rank's normals travel with its positions: every rank must choose alike, or the
    // strip exchanges would not match
    unsigned long long mine[3] = {(unsigned long long)s->send_l, (unsigned long long)s->send_r, (unsigned long long)s->has_nrm};
    KS_CUDA(cudaMemcpyAsync(s->sizes.p, mine, sizeof mine, cudaMemcpyHostToDevice, c->stream));
    KS_NCCL(s->nccl->AllGather(s->sizes.p, s->sizes_all.p, 3, ncclUint64, s->comm, c->stream));
    std::vector<unsigned long long> all(3 * (size_t)s->world);
    KS_CUDA(cudaMemcpyAsync(all.data(), s->sizes_all.p, all.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    KS_CUDA(cudaStreamSynchronize(c->stream));
    for (int r = 0; r < s->world; ++r)
        if (all[3 * (size_t)r + 2] != mine[2])
            return sfail(s, KPL_E_INVALID, "every rank must call kpl_shard_set_slab_normals, or every rank kpl_shard_set_slab");
    rc = set_slab_layout(s, s->rank > 0 ? (int64_t)all[3 * (size_t)(s->rank - 1) + 1] : 0,     // the left neighbour's RIGHT strip
                         s->rank < s->world - 1 ? (int64_t)all[3 * (size_t)(s->rank + 1)] : 0); // the right neighbour's LEFT strip
    if (!rc) rc = exchange(&s, 1, Strip::gidx);
    if (!rc) rc = kpl_shard_upload(s, xyz, stride);
    return rc || !s->has_nrm ? rc : kpl_shard_upload_normals(s, nrm, nrm_stride);
}

int kpl_shard_set_slab(kpl_shard* s, const float* xyz, int32_t stride, const int32_t* gidx, int64_t n_own)
{
    if (!s) return KPL_E_INVALID;
    return set_slab(s, xyz, stride, nullptr, 0, gidx, n_own);
}

int kpl_shard_set_slab_normals(kpl_shard* s, const float* xyz, int32_t stride, const float* normals, int32_t normals_stride,
                               const int32_t* gidx, int64_t n_own)
{
    if (!s) return KPL_E_INVALID;
    s->has_slab = s->has_nrm = false;
    if (!normals) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab_normals: normals_owned is NULL");
    if (bad_stride(normals_stride)) return sfail(s, KPL_E_INVALID, "normals_stride must be a multiple of 4 and >= 12 bytes");
    return set_slab(s, xyz, stride, normals, normals_stride, gidx, n_own);
}

int kpl_shard_upload(kpl_shard* s, const float* xyz, int32_t stride)
{
    if (!s || !xyz) return KPL_E_INVALID;
    if (!s->has_slab) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab was not called");
    if (stride < 12 || (stride & 3)) return sfail(s, KPL_E_INVALID, "stride must be a multiple of 4 and >= 12 bytes");
    kpl_ctx* c = s->ctx;
    KS_CUDA(cudaSetDevice(c->device));
    float4* dst = s->loc_xyz.p + s->n_l;
    if (stride == 16) KS_CUDA(cudaMemcpyAsync(dst, xyz, (size_t)s->n_own * 16, cudaMemcpyHostToDevice, c->stream));
    else KS_CUDA(cudaMemcpy2DAsync(dst, 16, xyz, (size_t)stride, 12, (size_t)s->n_own, cudaMemcpyHostToDevice, c->stream));
    return KPL_OK;
}

int kpl_shard_upload_normals(kpl_shard* s, const float* normals, int32_t normals_stride)
{
    if (!s || !normals) return KPL_E_INVALID;
    if (!s->has_nrm) return sfail(s, KPL_E_INVALID, "kpl_shard_upload_normals: the slab was not set with normals (kpl_shard_set_slab_normals)");
    if (!s->has_slab) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab_normals was not called");
    if (bad_stride(normals_stride)) return sfail(s, KPL_E_INVALID, "normals_stride must be a multiple of 4 and >= 12 bytes");
    KS_CUDA(cudaSetDevice(s->ctx->device));
    KS_CUDA(upload_records(s->loc_nrm.p + s->n_l, normals, normals_stride, s->n_own, s->ctx->stream));
    return KPL_OK;
}

int kpl_shard_detect(kpl_shard* s, float* scores_owned_out, int32_t* kp_global_out, int64_t kp_capacity, int64_t* n_kp_out)
{
    if (!s) return KPL_E_INVALID;
    if (n_kp_out) *n_kp_out = 0;
    if (s->in_process) return sfail(s, KPL_E_INVALID, "ranks of an in-process group are driven by kpl_shard_detect_group");
    return detect_step(&s, 1, &scores_owned_out, kp_global_out, kp_capacity, n_kp_out);
}

// All ranks of an in-process group from one host thread: the same phases, strips moved by peer copies.  The streams
// of the ranks are synchronised between phases (this is the path for hosts without NCCL and for single-GPU tests,
// not the fast path).
int kpl_shard_detect_group(kpl_shard** S, int32_t world, float** scores_owned_out, int32_t* kp_global_out, int64_t kp_capacity,
                           int64_t* n_kp_out)
{
    if (!S || world < 1 || !S[0]) return KPL_E_INVALID;
    if (n_kp_out) *n_kp_out = 0;
    kpl_shard* s = S[0];                       // errors are reported on rank 0's context
    for (int r = 0; r < world; ++r)
        if (!S[r] || !S[r]->in_process || S[r]->world != world || S[r]->rank != r) return sfail(s, KPL_E_INVALID, "kpl_shard_detect_group: not the ranks 0..world-1 of one in-process group");
    for (int r = 1; r < world; ++r)           // the strip exchanges only match when every rank's normals travel, or none
        if (S[r]->has_nrm != s->has_nrm)
            return sfail(s, KPL_E_INVALID, "every rank must call kpl_shard_set_slab_normals, or every rank kpl_shard_set_slab");
    // first call after set_slab: the strip sizes come from the peers, then the global indices of the halo points
    bool laid_out = false;
    for (int r = 0; r < world; ++r) {
        kpl_shard* t = S[r];
        if (t->has_slab) continue;
        if (t->n_own < 1) return sfail(s, KPL_E_INVALID, "kpl_shard_set_slab was not called on every rank");
        const int rc = set_slab_layout(t, r > 0 ? S[r - 1]->send_r : 0, r < world - 1 ? S[r + 1]->send_l : 0);
        if (rc) return on_rank(S, r, rc);
        laid_out = true;
    }
    if (laid_out) {
        const int rc = exchange(S, world, Strip::gidx);
        if (rc) return rc;
    }
    return detect_step(S, world, scores_owned_out, kp_global_out, kp_capacity, n_kp_out);
}

int kpl_shard_get_info(const kpl_shard* s, kpl_shard_info* out)
{
    if (!s || !out) return KPL_E_INVALID;
    memset(out, 0, sizeof *out);
    out->n_owned = s->n_own; out->n_left = std::max<int64_t>(s->n_l, 0); out->n_right = std::max<int64_t>(s->n_r, 0);
    out->send_left = s->send_l; out->send_right = s->send_r;
    out->halo_bytes = (s->send_l + s->send_r) * (int64_t)(sizeof(float4) + sizeof(float) + (s->has_nrm ? sizeof(float4) : 0));
    out->local_dims[0] = s->grid.dims[0]; out->local_dims[1] = s->plan.dims[1]; out->local_dims[2] = s->plan.dims[2];
    out->local_offset[0] = s->grid.offset[0];
    out->rank = s->rank; out->world = s->world;
    out->exchange_ms = s->exchange_ms; out->gather_ms = s->gather_ms;
    return KPL_OK;
}

const void* kpl_shard_device_scores(const kpl_shard* s)
{
    return (s && s->has_slab && s->ctx->score.p) ? (const void*)(s->ctx->score.p + s->n_l) : nullptr;
}

}  // extern "C"
