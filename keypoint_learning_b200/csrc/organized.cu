// organized.cu -- normals of an ORGANIZED cloud: pcl::IntegralImageNormalEstimation with SIMPLE_3D_GRADIENT and
// setNormalSmoothingSize(5.0), the branch KeypointLearningDetector::initCompute takes when no normals were set and the
// surface is organized (impl/KeypointLearning.hpp:138-145).
//
// [3P-recalled] PCL 1.8.0 features/impl/integral_image_normal.hpp (computeFeature: depth-change map, two-pass distance
// map; computeFeatureFull with BORDER_POLICY_IGNORE and no depth-dependent smoothing; computePointNormal) and
// features/impl/integral_image2D.hpp (IntegralImage2D<float,3>: sums in double, non-finite elements skipped).  The
// estimator is PCL code that is absent from this build, so this is a restatement from the pinned version; the tests hold
// it bit for bit to an independent CPU restatement of the same PCL sources (tests/test_gpu_parity.py).
//
// The two distance-map passes and the integral image are recurrences with a fixed evaluation order; they are evaluated
// as WAVEFRONTS by one thread block per frame (every element with the same number of the recurrence's longest dependency
// chain is independent), which reproduces the sequential results bit for bit -- including PCL's reads of the neighbouring
// row at the first / last column.  Every kernel takes a batch of frames of one size, stored frame after frame; a single
// organized cloud is the batch of one frame.
//
// The second half of the file turns a batch of organized frames into the concatenated views of kpl_detect_batch: the
// finite pixels of every frame, compacted in ascending pixel order, and back (kpl_detect_batch_organized, capi.cu).
#include <algorithm>
#include <cmath>
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include "kpl_internal.h"
#include "kpl_math.cuh"

namespace kpl {

__global__ void __launch_bounds__(256) ii_change_kernel(const float4* __restrict__ xyz, int W, int H, int nframes, float factor, unsigned char* __restrict__ change)
{
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t per_frame = (int64_t)(W - 1) * (H - 1);
    if (t >= per_frame * nframes) return;
    const int64_t f = t / per_frame, tf = t - f * per_frame;
    const int ri = (int)(tf / (W - 1)), ci = (int)(tf - (int64_t)ri * (W - 1));
    const int64_t index = f * W * H + (int64_t)ri * W + ci;
    const float depth = __ldg(&xyz[index].z), depthR = __ldg(&xyz[index + 1].z), depthD = __ldg(&xyz[index + W].z);
    const float lim = __fmul_rn(__fmul_rn(factor, __fadd_rn(fabsf(depth), 1.0f)), 2.0f);
    // only zeros are ever written: the order of the writes does not matter
    if (fabsf(__fsub_rn(depth, depthR)) > lim || !isfinite(depth) || !isfinite(depthR)) { change[index] = 0; change[index + 1] = 0; }
    if (fabsf(__fsub_rn(depth, depthD)) > lim || !isfinite(depth) || !isfinite(depthD)) { change[index] = 0; change[index + W] = 0; }
}

__global__ void __launch_bounds__(256) ii_dist_init_kernel(const unsigned char* __restrict__ change, int64_t n, float far_value, float* __restrict__ dist)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) dist[i] = change[i] == 0 ? 0.0f : far_value;
}

// Both passes of the distance map, one block per frame.  Forward: element (ri, ci), ri >= 1, ci >= 1, reads
// (ri-1, ci-1..ci+1) and (ri, ci-1): all of them carry a smaller 2*ri + ci.  Backward: the mirror image.
__global__ void __launch_bounds__(1024) ii_distance_kernel(float* __restrict__ dist, int W, int H)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    dist += (int64_t)blockIdx.x * W * H;
    for (int t = 3; t <= 2 * (H - 1) + (W - 1); ++t) {
        const int rlo = max(1, (t - (W - 1) + 1) / 2), rhi = min(H - 1, (t - 1) / 2);
        for (int ri = rlo + tid; ri <= rhi; ri += nt) {
            const int ci = t - 2 * ri;
            const float* prev = dist + (int64_t)(ri - 1) * W;
            float* cur = dist + (int64_t)ri * W;
            const float upLeft = __fadd_rn(prev[ci - 1], 1.4f), up = __fadd_rn(prev[ci], 1.0f), upRight = __fadd_rn(prev[ci + 1], 1.4f);
            const float left = __fadd_rn(cur[ci - 1], 1.0f);
            const float m = fminf(fminf(upLeft, up), fminf(left, upRight));
            if (m < cur[ci]) cur[ci] = m;
        }
        __syncthreads();
    }
    for (int t = 0; t <= 2 * (H - 2) + (W - 2); ++t) {
        // mirrored coordinates r' = H-2-ri, c' = W-2-ci, wavefront 2*r' + c'
        const int rlo = max(0, (t - (W - 2) + 1) / 2), rhi = min(H - 2, t / 2);
        for (int rp = rlo + tid; rp <= rhi; rp += nt) {
            const int cp = t - 2 * rp;
            const int ri = H - 2 - rp, ci = W - 2 - cp;
            const float* next = dist + (int64_t)(ri + 1) * W;
            float* cur = dist + (int64_t)ri * W;
            // ci == 0 reads next[-1], the last element of the current row, as PCL does
            const float lowerLeft = __fadd_rn(next[ci - 1], 1.4f), lower = __fadd_rn(next[ci], 1.0f), lowerRight = __fadd_rn(next[ci + 1], 1.4f);
            const float right = __fadd_rn(cur[ci + 1], 1.0f);
            const float m = fminf(fminf(lowerLeft, lower), fminf(right, lowerRight));
            if (m < cur[ci]) cur[ci] = m;
        }
        __syncthreads();
    }
}

// IntegralImage2D<float,3>::computeIntegralImages, first order: I[r+1][c+1] = ((I[r][c+1] + I[r+1][c]) - I[r][c]) + v in
// double, v skipped when the element's float sum is not finite.  Wavefront over r + c, one block per frame.  I: per
// frame (H+1) x (W+1) x 3.
__global__ void __launch_bounds__(1024) ii_integral_kernel(const float4* __restrict__ xyz, int W, int H, double* __restrict__ I)
{
    const int tid = threadIdx.x, nt = blockDim.x;
    const int S = W + 1;
    xyz += (int64_t)blockIdx.x * W * H;
    I += (int64_t)blockIdx.x * S * (H + 1) * 3;
    for (int64_t i = tid; i < (int64_t)S * 3; i += nt) I[i] = 0.0;                               // row 0
    for (int r = tid; r <= H; r += nt) { double* p = I + (int64_t)r * S * 3; p[0] = p[1] = p[2] = 0.0; }   // column 0
    __syncthreads();
    for (int t = 0; t <= (H - 1) + (W - 1); ++t) {
        const int rlo = max(0, t - (W - 1)), rhi = min(H - 1, t);
        for (int r = rlo + tid; r <= rhi; r += nt) {
            const int c = t - r;
            const float4 e = __ldg(xyz + (int64_t)r * W + c);
            const bool fin = isfinite(__fadd_rn(e.x, __fadd_rn(e.y, e.z)));
            const float ev[3] = {e.x, e.y, e.z};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                double v = __dsub_rn(__dadd_rn(I[((int64_t)r * S + (c + 1)) * 3 + a], I[((int64_t)(r + 1) * S + c) * 3 + a]), I[((int64_t)r * S + c) * 3 + a]);
                if (fin) v = __dadd_rn(v, (double)ev[a]);
                I[((int64_t)(r + 1) * S + (c + 1)) * 3 + a] = v;
            }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ double ii_sum(const double* __restrict__ I, int S, int sx, int sy, int w, int h, int a)
{
    // getFirstOrderSum: (lower_right + upper_left - upper_right - lower_left), left to right
    return __dsub_rn(__dsub_rn(__dadd_rn(I[((int64_t)(sy + h) * S + sx + w) * 3 + a], I[((int64_t)sy * S + sx) * 3 + a]),
                               I[((int64_t)sy * S + sx + w) * 3 + a]),
                     I[((int64_t)(sy + h) * S + sx) * 3 + a]);
}

// vps: NULL (every frame is seen from (vpx, vpy, vpz)) or 3 floats per frame
__global__ void __launch_bounds__(256) ii_normals_kernel(const float4* __restrict__ xyz, const float* __restrict__ dist, const double* __restrict__ I,
                                                         int W, int H, int nframes, float smoothing_size, float vpx, float vpy, float vpz,
                                                         const float* __restrict__ vps, float4* __restrict__ out)
{
    const int64_t index = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t n = (int64_t)W * H;
    if (index >= n * nframes) return;
    const float nanf_ = CUDART_NAN_F;
    float4 res = make_float4(nanf_, nanf_, nanf_, nanf_);
    const int64_t f = index / n, pix = index - f * n;
    const int ri = (int)(pix / W), ci = (int)(pix - (int64_t)ri * W);
    const int border = (int)smoothing_size;
    const float4 p = __ldg(xyz + index);
    if (ri >= border && ri < H - border && ci >= border && ci < W - border && isfinite(p.z)) {
        const float smoothing = fminf(dist[index], smoothing_size);
        I += f * (W + 1) * (H + 1) * 3;
        if (vps) { vpx = __ldg(vps + 3 * f); vpy = __ldg(vps + 3 * f + 1); vpz = __ldg(vps + 3 * f + 2); }
        if (smoothing > 2.0f) {
            const int rw = (int)smoothing, rh = rw, rw2 = rw / 2, rh2 = rh / 2, S = W + 1;
            double gx[3], gy[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                gx[a] = __dsub_rn(ii_sum(I, S, ci + rw2, ri - rh2, 1, rh, a), ii_sum(I, S, ci - rw2, ri - rh2, 1, rh, a));
                gy[a] = __dsub_rn(ii_sum(I, S, ci - rw2, ri + rh2, rw, 1, a), ii_sum(I, S, ci - rw2, ri - rh2, rw, 1, a));
            }
            // gradient_y.cross(gradient_x)
            const double nx_ = __dsub_rn(__dmul_rn(gy[1], gx[2]), __dmul_rn(gy[2], gx[1]));
            const double ny_ = __dsub_rn(__dmul_rn(gy[2], gx[0]), __dmul_rn(gy[0], gx[2]));
            const double nz_ = __dsub_rn(__dmul_rn(gy[0], gx[1]), __dmul_rn(gy[1], gx[0]));
            const double len = __dadd_rn(__dmul_rn(nx_, nx_), __dadd_rn(__dmul_rn(ny_, ny_), __dmul_rn(nz_, nz_)));
            if (len != 0.0) {
                const double s = __dsqrt_rn(len);
                float nx = __double2float_rn(__ddiv_rn(nx_, s)), ny = __double2float_rn(__ddiv_rn(ny_, s)), nz = __double2float_rn(__ddiv_rn(nz_, s));
                // flipNormalTowardsViewpoint
                const float vx = __fsub_rn(vpx, p.x), vy = __fsub_rn(vpy, p.y), vz = __fsub_rn(vpz, p.z);
                const float cos_theta = __fadd_rn(__fadd_rn(__fmul_rn(vx, nx), __fmul_rn(vy, ny)), __fmul_rn(vz, nz));
                if (cos_theta < 0.0f) { nx = -nx; ny = -ny; nz = -nz; }
                res = make_float4(nx, ny, nz, nanf_);           // curvature = bad_point for this method
            }
        }
    }
    out[index] = res;
}

// Integral images of the frames that share one chunk of scratch ((W+1)(H+1)*24 B per frame, 7.4 MB at 640 x 480); a
// larger batch runs in chunks, back to back on the stream.  A chunk holds at least one frame.
static const size_t II_CHUNK_BYTES = (size_t)256 << 20;

// d_xyz: nframes x width*height float4 (row-major, frame after frame, NaN = no measurement) -> d_out: (nx, ny, nz,
// curvature) per pixel.  d_viewpoints: NULL (the params' viewpoint) or 3 floats per frame, on the device.  The change
// map, the distance map and the integral images live in borrowed buffers (s_state, s_score, scratch_f): nothing reads
// them after the call.
cudaError_t launch_normals_integral_image(kpl_ctx* c, const float4* d_xyz, int W, int H, int nframes, float smoothing_size,
                                          const float* d_viewpoints, float4* d_out)
{
    const int64_t n = (int64_t)W * H, total = n * nframes;
    const size_t frame_doubles = (size_t)(W + 1) * (H + 1) * 3;
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)nframes, II_CHUNK_BYTES / (frame_doubles * sizeof(double))));
    cudaError_t e;
    DevBuf<uint8_t>& change = c->s_state;
    if ((e = ensure(change, (size_t)total)) || (e = ensure(c->s_score, (size_t)total)) ||
        (e = ensure(c->scratch_f, (size_t)chunk * frame_doubles * 2 + 16)))
        return e;
    float* dist = c->s_score.p;
    double* I = reinterpret_cast<double*>(c->scratch_f.p);
    const float factor = 20.0f * 0.001f;                       // max_depth_change_factor_ (constructor default; the reference never sets it)
    if ((e = cudaMemsetAsync(change.p, 255, (size_t)total, c->stream))) return e;
    if (W > 1 && H > 1) {
        const int64_t m = (int64_t)(W - 1) * (H - 1) * nframes;
        ii_change_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(d_xyz, W, H, nframes, factor, change.p);
    }
    ii_dist_init_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(change.p, total, (float)(W + H), dist);
    ii_distance_kernel<<<nframes, 1024, 0, c->stream>>>(dist, W, H);
    c->launches += 3;
    const kpl_params& P = c->params;
    for (int f0 = 0; f0 < nframes; f0 += chunk) {
        const int nf = std::min(chunk, nframes - f0);
        const int64_t first = (int64_t)f0 * n, m = (int64_t)nf * n;
        ii_integral_kernel<<<nf, 1024, 0, c->stream>>>(d_xyz + first, W, H, I);
        ii_normals_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(d_xyz + first, dist + first, I, W, H, nf, smoothing_size,
                                                                             P.viewpoint[0], P.viewpoint[1], P.viewpoint[2],
                                                                             d_viewpoints ? d_viewpoints + 3 * (int64_t)f0 : nullptr, d_out + first);
        c->launches += 2;
    }
    return cudaGetLastError();
}

// ---- batches of organized frames: finite pixels -> the concatenated views of a batch, and back --------------------
// Finite flag of every pixel (x, y and z finite: pcl::isFinite, the rule of bbox_kernel); the pixel-order scores of all
// nforests slices start as NaN (the value a point the detection never saw gets, as std::nanf("") in the C++ facade and
// np.nan in capi.py).
__global__ void __launch_bounds__(256) org_finite_kernel(const float4* __restrict__ xyz, int64_t total, int nforests, uint8_t* __restrict__ flag,
                                                         float* __restrict__ scores)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float4 p = __ldg(xyz + i);
    flag[i] = isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    if (scores)
        for (int k = 0; k < nforests; ++k) scores[k * total + i] = __int_as_float(0x7FC00000);
}

// frame_off[f] = first compacted point of frame f = lower bound of f * n in the ascending pixel list; frame_off[nframes]
// is the number of finite pixels.  frame_off[nframes + 1] holds the selected count on entry.
__global__ void __launch_bounds__(256) org_frame_offsets_kernel(const int32_t* __restrict__ pix, int64_t n, int nframes, int64_t* __restrict__ frame_off)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f > nframes) return;
    const int64_t bound = (int64_t)f * n;
    int64_t lo = 0, hi = frame_off[nframes + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)pix[mid] < bound) lo = mid + 1; else hi = mid;
    }
    frame_off[f] = lo;
}

__global__ void __launch_bounds__(256) org_gather_kernel(const float4* __restrict__ xyz, const float4* __restrict__ nrm, const int32_t* __restrict__ pix,
                                                         int64_t m, float4* __restrict__ xyz_c, float4* __restrict__ nrm_c)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int32_t p = pix[k];
    xyz_c[k] = __ldg(xyz + p);
    nrm_c[k] = __ldg(nrm + p);
}

// kp_off[j] = first keypoint of (forest j / nframes, frame j % nframes): the keypoints are ascending indices into the
// forest-major K x m compacted points, forest k's frame f starts at k*m + frame_off[f] (m = frame_off[nframes]), and
// j = K * nframes gives K*m, the end of the list
__global__ void __launch_bounds__(256) org_kp_offsets_kernel(const int32_t* __restrict__ kp, const int32_t* __restrict__ d_nkp,
                                                             const int64_t* __restrict__ frame_off, int nframes, int nforests,
                                                             int64_t* __restrict__ kp_off)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > nforests * nframes) return;
    const int k = j / nframes;
    const int64_t bound = k * frame_off[nframes] + frame_off[j - k * nframes];
    int lo = 0, hi = *d_nkp;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int64_t)kp[mid] < bound) lo = mid + 1; else hi = mid;
    }
    kp_off[j] = lo;
}

// forest-major compacted scores (K x m) -> pixel order (forest k's at k * total, total = nframes * n pixels); keypoints:
// index c into the K x m compacted points -> frame-local pixel index of point c - (c / m) * m, in place
__global__ void __launch_bounds__(256) org_map_back_kernel(const int32_t* __restrict__ pix, int64_t m, int64_t n, int64_t total, int64_t km,
                                                           const float* __restrict__ score_c, float* __restrict__ scores,
                                                           int32_t* __restrict__ kp, const int32_t* __restrict__ d_nkp)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= km) return;
    if (scores) {
        const int64_t k = i / m;
        scores[k * total + pix[i - k * m]] = score_c[i];
    }
    if (i < *d_nkp) {
        const int64_t c = kp[i];
        const int64_t p = pix[c - c / m * m];
        kp[i] = (int32_t)(p - p / n * n);
    }
}

cudaError_t launch_organized_select(kpl_ctx* c, const float4* d_xyz, int64_t n, int nframes, int nforests, float* d_scores)
{
    const int64_t total = n * nframes;
    cudaError_t e;
    if ((e = ensure(c->org_flag, (size_t)total)) || (e = ensure(c->org_pix, (size_t)total)) || (e = ensure(c->org_frame_off, (size_t)nframes + 2)))
        return e;
    org_finite_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(d_xyz, total, nforests, c->org_flag.p, d_scores);
    thrust::counting_iterator<int32_t> it(0);
    int64_t* d_m = c->org_frame_off.p + nframes + 1;
    size_t bytes = 0;
    cub::DeviceSelect::Flagged(nullptr, bytes, it, c->org_flag.p, c->org_pix.p, d_m, (int)total, c->stream);
    if ((e = ensure(c->cub_tmp, bytes))) return e;
    bytes = c->cub_tmp.cap;
    if ((e = cub::DeviceSelect::Flagged(c->cub_tmp.p, bytes, it, c->org_flag.p, c->org_pix.p, d_m, (int)total, c->stream))) return e;
    org_frame_offsets_kernel<<<(nframes + 1 + 255) / 256, 256, 0, c->stream>>>(c->org_pix.p, n, nframes, c->org_frame_off.p);
    c->launches += 4;
    return cudaGetLastError();
}

cudaError_t launch_organized_gather(kpl_ctx* c, const float4* d_xyz, const float4* d_nrm, int64_t m)
{
    cudaError_t e;
    if ((e = ensure(c->org_xyz, (size_t)m)) || (e = ensure(c->org_nrm, (size_t)m))) return e;
    org_gather_kernel<<<(unsigned)((m + 255) / 256), 256, 0, c->stream>>>(d_xyz, d_nrm, c->org_pix.p, m, c->org_xyz.p, c->org_nrm.p);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_organized_map_back(kpl_ctx* c, int64_t m, int64_t n, int nframes, int nforests, float* d_scores, int32_t* d_kp,
                                      int64_t* d_kp_off)
{
    const int32_t* d_nkp = (const int32_t*)(c->counters.p + 3);
    const int64_t km = m * nforests;
    org_kp_offsets_kernel<<<(nforests * nframes + 1 + 255) / 256, 256, 0, c->stream>>>(d_kp, d_nkp, c->org_frame_off.p, nframes, nforests, d_kp_off);
    org_map_back_kernel<<<(unsigned)((km + 255) / 256), 256, 0, c->stream>>>(c->org_pix.p, m, n, n * nframes, km, c->score.p, d_scores, d_kp, d_nkp);
    c->launches += 2;
    return cudaGetLastError();
}

}  // namespace kpl
