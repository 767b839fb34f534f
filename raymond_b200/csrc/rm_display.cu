// rm_display.cu — the display transform that follows the path in the reference's one working front-end
// (cli_old/src/main.rs:157-181), as a GPU epilogue of the accumulator, the host PNG writer (:194-197), and the
// feature-guided denoiser of rm_renderer_read_denoised and rm_render_tiled_denoised (no counterpart in the reference).
//
//   tone_mapped = 1 - exp(p * -1.0 * exposure);  tone_mapped = tone_mapped.powf(1.0 / gamma);
//   (tone_mapped * 255.0).cast::<u8>()  -> Some(v): the pixel;  None (any channel NaN or outside (-1, 256)): the
//   pixel keeps its initial (0, 0, 0)
// p = tile.data / tile.sample_count (src/trace.rs:95).  exp / pow are CUDA's f64 libm here and glibc's in the
// reference: a last-ulp difference can move a value across an integer boundary only when it lies within ~1e-13
// of it, so the 8-bit images agree except for isolated pixels, by one level (tests state the tolerance).

#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "rm_internal.hpp"

namespace rm {

__global__ void __launch_bounds__(256) k_tonemap(const double* __restrict__ sums, size_t n_pixels, double divisor, double exposure, double inv_gamma,
                                                  unsigned char* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pixels; i += (size_t)gridDim.x * blockDim.x) {
        unsigned char px[3];
        bool ok = true;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const double p = sums[i * 3 + c] / divisor;
            double t = 1.0 - exp(p * -1.0 * exposure);
            t = pow(t, inv_gamma);
            const double v = t * 255.0;
            // NumCast f64 -> u8: Some(trunc) iff -1 < v < 256
            if (!(v > -1.0 && v < 256.0)) ok = false;
            px[c] = (unsigned char)(int)v;
        }
        out[i * 3 + 0] = ok ? px[0] : 0;
        out[i * 3 + 1] = ok ? px[1] : 0;
        out[i * 3 + 2] = ok ? px[2] : 0;
    }
}

int tonemap_device(const double* sums_device, size_t n_pixels, double divisor, double exposure, double gamma, unsigned char* out_device, void* stream) {
    if (n_pixels == 0) return RM_OK;
    const unsigned blocks = (unsigned)std::min<size_t>((n_pixels + 255) / 256, 148 * 16);
    k_tonemap<<<blocks, 256, 0, (cudaStream_t)stream>>>(sums_device, n_pixels, divisor, exposure, 1.0 / gamma, out_device);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("k_tonemap: ") + cudaGetErrorString(e));
    return RM_OK;
}

// ---- the edge-avoiding a-trous denoiser of rm_renderer_read_denoised and rm_render_tiled_denoised (include/raymond.h gives the
// filter).  Each pixel is one float4 of (mean colour, variance) that the iterations update, and two of guides that stay: (albedo,
// depth) and (normal, 0).  One device filters the whole frame (k_denoise_pack, k_atrous); the shares of a task filter a slice of
// rows each (k_denoise_reduce, k_atrous_slice) with the same per-pixel functions, so a pixel's result depends only on its inputs.

int resolve_denoise_settings(const rm_denoise_settings* settings, rm_denoise_settings* out, const char* who) {
    rm_denoise_settings s{1, 0, 1e4, 0.1, 0.3, 1.0};       // the defaults stated in include/raymond.h
    if (settings) s = *settings;
    // the filter uses each sigma as an f32, and the squares of sigma_normal and sigma_albedo: all of them must be normal f32 values
    // (a square that underflows to 0 or a sigma that overflows to inf would make the centre tap's weight NaN)
    const auto usable = [](double x, bool squared) {
        const float f = (float)x, g = squared ? f * f : f;
        return std::isfinite(x) && x > 0.0 && std::isfinite(g) && g >= FLT_MIN;
    };
    if (s.iterations < 1 || s.iterations > 10 || !usable(s.sigma_color, false) || !usable(s.sigma_normal, true) || !usable(s.sigma_albedo, true) ||
        !usable(s.sigma_depth, false))
        return fail(RM_ERR_INVALID_ARGUMENT, std::string(who) + ": iterations outside 1..10 or a sigma outside the f32 range the filter needs");
    *out = s;
    return RM_OK;
}

__device__ __forceinline__ bool finite4(float4 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z) && isfinite(a.w); }
__device__ __forceinline__ bool finite3(float4 a) { return isfinite(a.x) && isfinite(a.y) && isfinite(a.z); }

// One pixel's means after n samples from its sums (S, Q and albedo / normal per channel, depth), formed in f64 exactly as
// include/raymond.h defines m and se2, then rounded to f32 once.
__device__ __forceinline__ void pack_pixel(const double* S, const double* Q, const double* alb, const double* nrm, double depth, double n,
                                           float4* cv, float4* az, float4* nm) {
    float m[3];
    double se2 = 0.0;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const double s = S[c], q = Q[c];
        const double mean = s / n;
        const double d = q - s * mean;
        se2 += (d < 0.0 ? 0.0 : d) / (n - 1.0) / n;
        m[c] = (float)mean;
    }
    *cv = make_float4(m[0], m[1], m[2], (float)se2);
    *az = make_float4((float)(alb[0] / n), (float)(alb[1] / n), (float)(alb[2] / n), (float)(depth / n));
    *nm = make_float4((float)(nrm[0] / n), (float)(nrm[1] / n), (float)(nrm[2] / n), 0.0f);
}

__global__ void __launch_bounds__(256) k_denoise_pack(const double* __restrict__ sums, const double* __restrict__ moments, const double* __restrict__ aov,
                                                      size_t n_pixels, double n, float4* __restrict__ cv, float4* __restrict__ az, float4* __restrict__ nm) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pixels) pack_pixel(sums + i * 3, moments + i * 3, aov + i * 3, aov + (n_pixels + i) * 3, aov[6 * n_pixels + i], n, cv + i, az + i, nm + i);
}

// Share `share`'s rows: S, Q and the 7 feature planes of every pixel summed over all shares' whole-frame sums, read in place in
// share order (the association of k_reduce_slice), then packed into the share's own rows.
__global__ void __launch_bounds__(256) k_denoise_reduce(const __grid_constant__ DenoiseSlices d, int share, size_t W, size_t H, double n) {
    const size_t y0 = slice_begin(H, share, d.count), rows = slice_begin(H, share + 1, d.count) - y0;
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n_pixels = W * H;
    if (k >= rows * W) return;
    const size_t i = y0 * W + k;
    double S[3], Q[3], alb[3], nrm[3], depth = d.aov[0][6 * n_pixels + i];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        S[c] = d.sums[0][i * 3 + c];
        Q[c] = d.moments[0][i * 3 + c];
        alb[c] = d.aov[0][i * 3 + c];
        nrm[c] = d.aov[0][(n_pixels + i) * 3 + c];
    }
    for (int j = 1; j < d.count; j++) {
#pragma unroll
        for (int c = 0; c < 3; c++) {
            S[c] += d.sums[j][i * 3 + c];
            Q[c] += d.moments[j][i * 3 + c];
            alb[c] += d.aov[j][i * 3 + c];
            nrm[c] += d.aov[j][(n_pixels + i) * 3 + c];
        }
        depth += d.aov[j][6 * n_pixels + i];
    }
    float4* const packed = (float4*)d.packed[share];
    pack_pixel(S, Q, alb, nrm, depth, n, packed + k, packed + 2 * rows * W + k, packed + 3 * rows * W + k);
}

// Row qy of the three planes a pass reads (index x of each pointer = pixel (x, qy)).
struct TapRow { const float4 *cv, *az, *nm; };

// One pixel of one iteration at tap distance `step`: 5x5 taps, dy outer and dx inner, both ascending, so the sums have one order.
// `rows(qy)` finds the row wherever it is held.
template <class Rows>
__device__ __forceinline__ float4 atrous_pixel(const Rows& rows, int x, int y, int W, int H, int step, float sigma_c, float sigma_n2, float sigma_a2,
                                               float sigma_z) {
    const TapRow rp = rows(y);
    const float4 cp = rp.cv[x], ap = rp.az[x], np = rp.nm[x];
    if (!(finite4(cp) && finite4(ap) && finite3(np))) return cp;
    const float kern[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
    // the denominators depend on p only: each division becomes a product with the f32 reciprocal, formed once per pixel
    const float rc = 1.0f / (sigma_c * sqrtf(cp.w) + 1e-6f), rn = 1.0f / sigma_n2, ra = 1.0f / sigma_a2;
    const float rz = 1.0f / (sigma_z * (float)step * ap.w + 1e-6f);
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; dy++) {
        const int qy = y + dy * step;
        if (qy < 0 || qy >= H) continue;
        const TapRow row = rows(qy);
#pragma unroll
        for (int dx = -2; dx <= 2; dx++) {
            const int qx = x + dx * step;
            if (qx < 0 || qx >= W) continue;
            const float4 cq = row.cv[qx], aq = row.az[qx], nq = row.nm[qx];
            if (!(finite4(cq) && finite4(aq) && finite3(nq))) continue;
            const float cr = cp.x - cq.x, cg = cp.y - cq.y, cb = cp.z - cq.z;
            const float nx = np.x - nq.x, ny = np.y - nq.y, nz = np.z - nq.z;
            const float ax = ap.x - aq.x, ay = ap.y - aq.y, azz = ap.z - aq.z;
            const float e = sqrtf(cr * cr + cg * cg + cb * cb) * rc + (nx * nx + ny * ny + nz * nz) * rn + (ax * ax + ay * ay + azz * azz) * ra +
                            fabsf(ap.w - aq.w) * rz;
            const float w = kern[dx + 2] * kern[dy + 2] * expf(-e);
            sw += w;
            sr += w * cq.x; sg += w * cq.y; sb += w * cq.z;
            sv += w * w * cq.w;
        }
    }
    return make_float4(sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}

// A pass's result: the next pass's input, or (last pass, `out` non-NULL) the f64 colour in the mapped host frame.
__device__ __forceinline__ void put_pixel(float4 c, float4* cv_out, double* out, size_t p) {
    if (out) { out[p * 3 + 0] = c.x; out[p * 3 + 1] = c.y; out[p * 3 + 2] = c.z; }
    else *cv_out = c;
}

struct FrameRows {      // the whole frame in one buffer per plane
    const float4 *cv, *az, *nm;
    int W;
    __device__ TapRow operator()(int qy) const { const size_t o = (size_t)qy * W; return {cv + o, az + o, nm + o}; }
};

__global__ void __launch_bounds__(256) k_atrous(const float4* __restrict__ cv_in, const float4* __restrict__ az, const float4* __restrict__ nm,
                                                float4* __restrict__ cv_out, double* __restrict__ out, int W, int H, int step, float sigma_c,
                                                float sigma_n2, float sigma_a2, float sigma_z) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || y >= H) return;
    const size_t p = (size_t)y * W + x;
    put_pixel(atrous_pixel(FrameRows{cv_in, az, nm, W}, x, y, W, H, step, sigma_c, sigma_n2, sigma_a2, sigma_z), cv_out + p, out, p);
}

struct SliceRows {      // row qy from the packed rows of the share that owns it (colour plane `plane` of the ping-pong pair)
    const DenoiseSlices* d;
    size_t W, H;
    unsigned plane;
    __device__ TapRow operator()(int qy) const {
        const size_t j = ((size_t)(qy + 1) * d->count - 1) / H;      // the last share whose first row is <= qy
        const size_t y0 = slice_begin(H, j, d->count), plane_px = (slice_begin(H, j + 1, d->count) - y0) * W;
        const float4* row = (const float4*)d->packed[j] + ((size_t)qy - y0) * W;
        return {row + plane * plane_px, row + 2 * plane_px, row + 3 * plane_px};
    }
};

// Pass `pass` of share `share`'s rows: colour plane pass & 1 in, (pass + 1) & 1 out; taps beyond the slice (up to 2 * 2^pass rows)
// are read from the shares that own them.
__global__ void __launch_bounds__(256) k_atrous_slice(const __grid_constant__ DenoiseSlices d, int share, double* __restrict__ out, int W, int H,
                                                      unsigned pass, float sigma_c, float sigma_n2, float sigma_a2, float sigma_z) {
    const size_t y0 = slice_begin(H, share, d.count), rows = slice_begin(H, share + 1, d.count) - y0;
    const int x = blockIdx.x * blockDim.x + threadIdx.x, yl = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= W || (size_t)yl >= rows) return;
    const int y = (int)y0 + yl;
    const float4 c = atrous_pixel(SliceRows{&d, (size_t)W, (size_t)H, pass & 1u}, x, y, W, H, 1 << pass, sigma_c, sigma_n2, sigma_a2, sigma_z);
    put_pixel(c, (float4*)d.packed[share] + ((pass + 1) & 1u) * rows * W + (size_t)yl * W + x, out, (size_t)y * W + x);
}

int denoise_to_host(const double* sums, const double* moments, const double* aov, size_t W, size_t H, double n, const rm_denoise_settings& s,
                    rm_vec3* out_mapped, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    const size_t np = W * H;
    float4* buf = nullptr;      // cv ping, cv pong, albedo + depth, normal
    cudaError_t e = (cudaError_t)dev_alloc((void**)&buf, std::max<size_t>(np, 1) * 4 * sizeof(float4));
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("denoiser buffers: ") + cudaGetErrorString(e));
    float4* const cv[2] = {buf, buf + np};
    k_denoise_pack<<<(unsigned)((np + 255) / 256), 256, 0, stream>>>(sums, moments, aov, np, n, cv[0], buf + 2 * np, buf + 3 * np);
    const dim3 tb(16, 16), grid((unsigned)((W + 15) / 16), (unsigned)((H + 15) / 16));
    const float sn = (float)s.sigma_normal, sa = (float)s.sigma_albedo;
    for (uint32_t i = 0; i < s.iterations; i++)
        k_atrous<<<grid, tb, 0, stream>>>(cv[i & 1], buf + 2 * np, buf + 3 * np, cv[(i + 1) & 1], i + 1 == s.iterations ? (double*)out_mapped : nullptr,
                                          (int)W, (int)H, 1 << i, (float)s.sigma_color, sn * sn, sa * sa, (float)s.sigma_depth);
    e = cudaGetLastError();
    const cudaError_t done = cudaStreamSynchronize(stream);      // before the buffers go back to the pool
    if (e == cudaSuccess) e = done;
    dev_release(buf);
    if (e != cudaSuccess) return fail(RM_ERR_CUDA, std::string("denoiser: ") + cudaGetErrorString(e));
    return RM_OK;
}

int denoise_reduce_slice(const DenoiseSlices& d, int share, size_t W, size_t H, double n, void* stream) {
    const size_t px = (slice_begin(H, share + 1, d.count) - slice_begin(H, share, d.count)) * W;
    if (px == 0) return 0;
    k_denoise_reduce<<<(unsigned)((px + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, share, W, H, n);
    return (int)cudaGetLastError();
}

int denoise_pass_slice(const DenoiseSlices& d, int share, size_t W, size_t H, uint32_t pass, const rm_denoise_settings& s, rm_vec3* out_mapped,
                       void* stream) {
    const size_t rows = slice_begin(H, share + 1, d.count) - slice_begin(H, share, d.count);
    if (rows == 0) return 0;
    const float sn = (float)s.sigma_normal, sa = (float)s.sigma_albedo;
    const dim3 tb(16, 16), grid((unsigned)((W + 15) / 16), (unsigned)((rows + 15) / 16));
    k_atrous_slice<<<grid, tb, 0, (cudaStream_t)stream>>>(d, share, (double*)out_mapped, (int)W, (int)H, pass, (float)s.sigma_color, sn * sn, sa * sa,
                                                          (float)s.sigma_depth);
    return (int)cudaGetLastError();
}

}  // namespace rm

using namespace rm;

extern "C" {

int rm_tonemap_rgb8(const rm_vec3* frame, size_t pixels, double exposure, double gamma, int device, uint8_t* out) {
    if ((!frame || !out) && pixels) return fail(RM_ERR_INVALID_ARGUMENT, "rm_tonemap_rgb8: null argument");
    if (pixels == 0) return RM_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return fail(RM_ERR_CUDA, "no usable CUDA device " + std::to_string(device) + "; this library has no CPU path");
    }
    cudaSetDevice(device);
    void *d_in = nullptr, *d_out = nullptr;
    int e = dev_alloc(&d_in, pixels * sizeof(rm_vec3));
    if (e == 0) e = dev_alloc(&d_out, pixels * 3);
    int st = RM_OK;
    if (e != 0) st = fail(RM_ERR_CUDA, std::string("device allocation: ") + cudaGetErrorString((cudaError_t)e));
    if (st == RM_OK && cudaMemcpy(d_in, frame, pixels * sizeof(rm_vec3), cudaMemcpyHostToDevice) != cudaSuccess) st = fail(RM_ERR_CUDA, "H2D of the frame failed");
    if (st == RM_OK) st = tonemap_device((const double*)d_in, pixels, 1.0, exposure, gamma, (unsigned char*)d_out, nullptr);
    if (st == RM_OK && cudaMemcpy(out, d_out, pixels * 3, cudaMemcpyDeviceToHost) != cudaSuccess) st = fail(RM_ERR_CUDA, "D2H of the 8-bit image failed");
    cudaDeviceSynchronize();
    dev_release(d_in);
    dev_release(d_out);
    return st;
}

}  // extern "C"
