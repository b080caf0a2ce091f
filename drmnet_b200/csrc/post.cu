// "Next" rows either side of the render (SURVEY 8f N1, N2), sm_100a.  Small HBM-bound elementwise / gather kernels.
//
//  * drm_refmap_postprocess: the two steps DRMNet.get_input applies to every rendered stack right after the render
//    loop -- scale so the geometric mean of the luminance of LrK over L > 0 equals `target` (reference
//    models/drmnet.py:610-617) and the dataset transform log10(x + 0.1) + 1 (dataset/basedataset.py:52-53) -- fused into
//    one kernel: one CTA per sample reduces log-luminance in a fixed order (deterministic), then streams the stacks.
//  * drm_mirmap2envmap: mirror refmap -> lat-long envmap warp of utils/transform.py:106-144 (used by DRMNet.r0toenvmap,
//    models/drmnet.py:931-941), with the division by basis_r0 (:939) fused in.
#include <math.h>

#include "common.cuh"

namespace drm {

static constexpr int POST_THREADS = 256;

__device__ __forceinline__ float block_sum(float v, float* sh) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    if (lane == 0) sh[w] = v;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < POST_THREADS / 32; ++i) t += sh[i];  // same order in every thread
    __syncthreads();
    return t;
}

// in/out: [G, N, 3, res, res]; sample n = blockIdx.x
__global__ void __launch_bounds__(POST_THREADS) refmap_postprocess_kernel(const float* __restrict__ in, int G, int N,
                                                                          int res, float target, int transform,
                                                                          float* __restrict__ scale_out,
                                                                          float* __restrict__ out) {
    __shared__ float sh[POST_THREADS / 32];
    const int n = blockIdx.x;
    const int P = res * res;
    float scale = 1.f;
    if (target > 0.f) {
        const float* r = in + (size_t)n * 3 * P;  // stack 0 = LrK
        float s = 0.f, c = 0.f;
        for (int p = threadIdx.x; p < P; p += POST_THREADS) {
            const float L = 0.212671f * r[p] + 0.715160f * r[P + p] + 0.072169f * r[2 * P + p];
            if (L > 0.f) {
                s += logf(fmaxf(L, 1e-5f));
                c += 1.f;
            }
        }
        s = block_sum(s, sh);
        c = block_sum(c, sh);
        scale = target / expf(s / c);  // c == 0 -> NaN, as the reference's 0/0
    }
    if (scale_out && threadIdx.x == 0) scale_out[n] = scale;
    for (int gidx = 0; gidx < G; ++gidx) {
        const size_t base = ((size_t)gidx * N + n) * 3 * P;
        for (int e = threadIdx.x; e < 3 * P; e += POST_THREADS) {
            float v = in[base + e] * scale;
            if (transform == 1) v = log10f(v + 0.1f) + 1.f;
            out[base + e] = v;
        }
    }
}

// mirmap [B, C, H, W] (optionally divided by basis [C, H, W]) -> envmap [B, C, OH, OW]; view = (0,0,1), top = +Y,
// zenith = +Y, left edge = -Z, azimuth reversed: the defaults r0toenvmap uses
__global__ void mirmap2envmap_kernel(const float* __restrict__ mir, const float* __restrict__ basis, int B, int C, int H,
                                     int W, int OH, int OW, float* __restrict__ out) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= OH * OW) return;
    const int oi = o / OW, oj = o - oi * OW;
    const float theta = ((float)oi + 0.5f) * (float)(M_PI / OH);
    const float phi = -(((float)oj + 0.5f) * (float)(2.0 * M_PI / OW));  // reverse_azimuth
    // thetaphi2xyz(normal=[0,1,0], tangent=[0,0,-1]): binormal = [-1,0,0]
    const float st = sinf(theta), ct = cosf(theta), sp = sinf(phi), cp = cosf(phi);
    float x = -(st * sp), y = ct, z = -(st * cp);
    z += 1.f;  // + view
    const float nrm = fmaxf(sqrtf(x * x + y * y + z * z), 1e-12f);
    x /= nrm; y /= nrm; z /= nrm;
    // xyz2thetaphi(normal=top=[0,1,0], tangent=view=[0,0,1]): binormal = [1,0,0]
    const float th = acosf(y), ph = atan2f(x, z);
    const float u = ph * (float)(2.0 / M_PI), v = th * (float)(2.0 / M_PI) - 1.f;
    // grid_sample(bilinear, padding_mode=border, align_corners=False)
    float ix = ((u + 1.f) * W - 1.f) * 0.5f, iy = ((v + 1.f) * H - 1.f) * 0.5f;
    ix = fminf(fmaxf(ix, 0.f), (float)(W - 1));
    iy = fminf(fmaxf(iy, 0.f), (float)(H - 1));
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const int x0 = (int)fx0, y0 = (int)fy0, x1 = x0 + 1, y1 = y0 + 1;
    const float wx1 = ix - fx0, wy1 = iy - fy0, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
    for (int b = 0; b < B; ++b)
        for (int c = 0; c < C; ++c) {
            const float* m = mir + ((size_t)b * C + c) * H * W;
            const float* bs = basis ? basis + (size_t)c * H * W : nullptr;
            auto at = [&](int yy, int xx) {
                if (yy >= H || xx >= W) return 0.f;
                const float val = m[yy * W + xx];
                return bs ? val / bs[yy * W + xx] : val;
            };
            const float val = at(y0, x0) * (wx0 * wy0) + at(y0, x1) * (wx1 * wy0) + at(y1, x0) * (wx0 * wy1) +
                              at(y1, x1) * (wx1 * wy1);
            out[(((size_t)b * C + c) * OH + oi) * OW + oj] = val;
        }
}

// N3: shade pixels by a bilinear refmap lookup at the (theta, phi) of their normals -- the arithmetic of
// refmap2refimg_torch (utils/transform.py:170-198: xyz2thetaphi(normal,[0,1,0],[-1,0,0]) -> uv = (phi, theta) * 2/pi - 1
// -> grid_sample bilinear / border / align_corners=False).  One pixel of image b (refmap b of [B, C, H, W]): store(c, v)
// receives channel c.  Both lookup kernels inline it, so they shade a normal bit for bit alike.
template <typename Store>
__device__ __forceinline__ void refmap_lookup_pixel(const float* __restrict__ refmap, int b, int C, int H, int W, float x,
                                                    float y, float z, Store store) {
    const float th = acosf(y), ph = atan2f(z, -x + 0.f);
    const float u = ph * (float)(2.0 / M_PI) - 1.f, v = th * (float)(2.0 / M_PI) - 1.f;
    float ix = ((u + 1.f) * W - 1.f) * 0.5f, iy = ((v + 1.f) * H - 1.f) * 0.5f;
    ix = fminf(fmaxf(ix, 0.f), (float)(W - 1));
    iy = fminf(fmaxf(iy, 0.f), (float)(H - 1));
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const int x0 = (int)fx0, y0 = (int)fy0, x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
    const float wx1 = ix - fx0, wy1 = iy - fy0, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
    for (int c = 0; c < C; ++c) {
        const float* m = refmap + ((size_t)b * C + c) * H * W;
        store(c, m[y0 * W + x0] * (wx0 * wy0) + m[y0 * W + x1] * (wx1 * wy0) + m[y1 * W + x0] * (wx0 * wy1) +
                     m[y1 * W + x1] * (wx1 * wy1));
    }
}

// compacted normal lists [total_n, 3] -> colors [total_n, C], image b owning rows offsets[b] .. offsets[b+1]-1
__global__ void refmap_lookup_kernel(const float* __restrict__ refmap, const float* __restrict__ normals,
                                     const int64_t* __restrict__ offsets, int64_t total_n, int B, int C, int H, int W,
                                     float* __restrict__ colors) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= total_n) return;
    int lo = 0, hi = B;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (offsets[mid] <= p) lo = mid; else hi = mid;
    }
    refmap_lookup_pixel(refmap, lo, C, H, W, normals[3 * p], normals[3 * p + 1], normals[3 * p + 2],
                        [&](int c, float v) { colors[p * C + c] = v; });
}

// (b, y, x, channel) element strides of a dense image, each >= 0
struct ImageStrides {
    int64_t s[4];
};

// dense normal maps under a mask -> dense images: pixel (b, y, x) of B images of HW = H * W pixels.  blockIdx.y walks the
// images (grid-stride, gridDim.y <= 65535); a pixel whose mask byte is 0 gets zeros and its normal is not read.
__global__ void refmap_lookup_dense_kernel(const float* __restrict__ refmap, int Hr, int Wr,
                                           const float* __restrict__ normals, ImageStrides ns,
                                           const uint8_t* __restrict__ mask, int B, int HW, int W, int C,
                                           float* __restrict__ out, ImageStrides os) {
    const int64_t qq = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (qq >= HW) return;
    const int q = (int)qq, py = q / W, px = q - py * W;
    for (int b = blockIdx.y; b < B; b += gridDim.y) {
        float* o = out + b * os.s[0] + py * os.s[1] + px * os.s[2];
        if (mask && !mask[(size_t)b * HW + q]) {
            for (int c = 0; c < C; ++c) o[c * os.s[3]] = 0.f;
            continue;
        }
        const float* n = normals + b * ns.s[0] + py * ns.s[1] + px * ns.s[2];
        refmap_lookup_pixel(refmap, b, C, Hr, Wr, n[0], n[ns.s[3]], n[2 * ns.s[3]],
                            [&](int c, float v) { o[c * os.s[3]] = v; });
    }
}

__device__ __forceinline__ float block_max(float v, float* sh) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int d = 16; d; d >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, d));
    if (lane == 0) sh[w] = v;
    __syncthreads();
    float t = sh[0];
    for (int i = 1; i < POST_THREADS / 32; ++i) t = fmaxf(t, sh[i]);
    __syncthreads();
    return t;
}

// N4: ObsNet's conditioning transform chain `0p1tom1p1_normalizedLogarithmic_lowerbound<lb>` with dynamic_normalize
// (dataset/basedataset.py:56-76 applied right to left; models/obsnet.py:224,370): y = clip(x, lb);
// max = amax(y * mask), min = amin(y * mask + (1 - mask) * max) per sample; out = 2 (log10 y - log10 min)/(log10 max - log10 min) - 1.
__global__ void __launch_bounds__(POST_THREADS) normalized_log_kernel(const float* __restrict__ x,
                                                                      const float* __restrict__ mask, int C, int P,
                                                                      float lowerbound, float* __restrict__ out,
                                                                      float* __restrict__ log10min_out,
                                                                      float* __restrict__ log10max_out) {
    __shared__ float sh[POST_THREADS / 32];
    const int n = blockIdx.x;
    const float* xs = x + (size_t)n * C * P;
    const float* ms = mask + (size_t)n * P;
    float mx = -INFINITY;
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS) mx = fmaxf(mx, fmaxf(xs[e], lowerbound) * ms[e % P]);
    mx = block_max(mx, sh);
    float mn = -INFINITY;  // max of the negated values = -min
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS) {
        const float m = ms[e % P];
        mn = fmaxf(mn, -(fmaxf(xs[e], lowerbound) * m + (1.f - m) * mx));
    }
    mn = -block_max(mn, sh);
    const float lmax = log10f(mx), lmin = log10f(mn);
    if (threadIdx.x == 0) {
        if (log10min_out) log10min_out[n] = lmin;
        if (log10max_out) log10max_out[n] = lmax;
    }
    const float inv = 1.f / (lmax - lmin);
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS)
        out[(size_t)n * C * P + e] = (log10f(fmaxf(xs[e], lowerbound)) - lmin) * inv * 2.f - 1.f;
}

// N4 remainder: ObsNet's conditioning (models/obsnet.py:672-691, training path :368-371).  One CTA per sample:
// the dynamic normalisation of the raw refmap under its mask (above), then
//   cond = t(raw) * mask;  cond = sigma * n1 + cond (noisy_observe > 0);  cond += (1 - mask) * n2 (padding "noise")
// in that order, with the noise tensors drawn by the caller (torch.randn_like in the reference).
__global__ void __launch_bounds__(POST_THREADS) obsnet_condition_kernel(const float* __restrict__ x, const float* __restrict__ mask,
                                                                        int C, int P, float lowerbound, float sigma,
                                                                        const float* __restrict__ n1, const float* __restrict__ n2,
                                                                        float* __restrict__ cond, float* __restrict__ log10min_out,
                                                                        float* __restrict__ log10max_out) {
    __shared__ float sh[POST_THREADS / 32];
    const int n = blockIdx.x;
    const size_t base = (size_t)n * C * P;
    const float* xs = x + base;
    const float* ms = mask + (size_t)n * P;
    float mx = -INFINITY;
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS) mx = fmaxf(mx, fmaxf(xs[e], lowerbound) * ms[e % P]);
    mx = block_max(mx, sh);
    float mn = -INFINITY;
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS) {
        const float m = ms[e % P];
        mn = fmaxf(mn, -(fmaxf(xs[e], lowerbound) * m + (1.f - m) * mx));
    }
    mn = -block_max(mn, sh);
    const float lmax = log10f(mx), lmin = log10f(mn);
    if (threadIdx.x == 0) {
        if (log10min_out) log10min_out[n] = lmin;
        if (log10max_out) log10max_out[n] = lmax;
    }
    const float inv = 1.f / (lmax - lmin);
    for (int e = threadIdx.x; e < C * P; e += POST_THREADS) {
        const float m = ms[e % P];
        float c = ((log10f(fmaxf(xs[e], lowerbound)) - lmin) * inv * 2.f - 1.f) * m;
        if (n1) c = sigma * n1[base + e] + c;
        if (n2) c += (1.f - m) * n2[base + e];
        cond[base + e] = c;
    }
}

// the same transform with parameters fixed by an earlier dynamic call (dynamic_normalize=False, dataset/basedataset.py:68-72)
// and its inverse, BaseDataset.rescale (:98-110): x -> (x + 1) / 2 -> 10 ^ min(x (max - min) + min, clamp)
__global__ void normalized_log_apply_kernel(const float* __restrict__ x, const float* __restrict__ lmin,
                                            const float* __restrict__ lmax, int64_t per_sample, int64_t total,
                                            float lowerbound, int inverse, float clamp_before_exp, float* __restrict__ out) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int n = (int)(e / per_sample);
    const float a = lmin[n], b = lmax[n];
    if (!inverse) {
        out[e] = (log10f(fmaxf(x[e], lowerbound)) - a) / (b - a) * 2.f - 1.f;
    } else {
        float y = (x[e] + 1.f) / 2.f * (b - a) + a;
        if (clamp_before_exp != 0.f) y = fminf(y, clamp_before_exp);
        out[e] = powf(10.f, y);
    }
}

}  // namespace drm

using namespace drm;

extern "C" int drm_obsnet_condition(const float* raw_refmap, const float* raw_refmask, int B, int C, int H, int W,
                                    float lowerbound, float noisy_observe, const float* observe_noise,
                                    const float* padding_noise, float* cond, float* log10min_out, float* log10max_out,
                                    void* cuda_stream) {
    DRM_REQUIRE(raw_refmap && raw_refmask && cond, "obsnet_condition: null pointer");
    DRM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "obsnet_condition: sizes must be positive");
    DRM_REQUIRE(!(noisy_observe > 0.f) || observe_noise, "obsnet_condition: noisy_observe > 0 needs observe_noise");
    obsnet_condition_kernel<<<B, POST_THREADS, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        raw_refmap, raw_refmask, C, H * W, lowerbound, noisy_observe, noisy_observe > 0.f ? observe_noise : nullptr,
        padding_noise, cond, log10min_out, log10max_out);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_normalized_log_apply(const float* x, const float* log10min, const float* log10max, int B, int C, int H,
                                        int W, float lowerbound, int inverse, float clamp_before_exp, float* out,
                                        void* cuda_stream) {
    DRM_REQUIRE(x && log10min && log10max && out, "normalized_log_apply: null pointer");
    DRM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "normalized_log_apply: sizes must be positive");
    const int64_t per = (int64_t)C * H * W, total = per * B;
    normalized_log_apply_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        x, log10min, log10max, per, total, lowerbound, inverse, clamp_before_exp, out);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_refmap_lookup(const float* refmap, const float* normals, const int64_t* offsets, int64_t total_n,
                                 int B, int C, int H, int W, float* colors, void* cuda_stream) {
    DRM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && total_n >= 0, "refmap_lookup: sizes must be positive");
    DRM_REQUIRE(refmap && offsets && (total_n == 0 || (normals && colors)), "refmap_lookup: null pointer");
    if (total_n == 0) return DRM_OK;
    refmap_lookup_kernel<<<(unsigned)((total_n + 255) / 256), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(
        refmap, normals, offsets, total_n, B, C, H, W, colors);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_refmap_lookup_dense(const float* refmap, int Hr, int Wr, const float* normals,
                                       const int64_t normals_strides[4], const uint8_t* mask, int B, int H, int W, int C,
                                       float* out, const int64_t out_strides[4], void* cuda_stream) {
    DRM_REQUIRE(refmap && normals && normals_strides && out && out_strides,
                "refmap_lookup_dense: null pointer (refmap %p, normals %p, normals_strides %p, out %p, out_strides %p)",
                (const void*)refmap, (const void*)normals, (const void*)normals_strides, (void*)out,
                (const void*)out_strides);
    DRM_REQUIRE(B > 0 && H > 0 && W > 0 && Hr > 0 && Wr > 0,
                "refmap_lookup_dense: B=%d H=%d W=%d Hr=%d Wr=%d must be positive", B, H, W, Hr, Wr);
    DRM_REQUIRE(C >= 1 && C <= 4, "refmap_lookup_dense: C=%d not in 1..4", C);
    DRM_REQUIRE((int64_t)H * W < (1ll << 31), "refmap_lookup_dense: H*W = %lld pixels per image, below 2^31 required",
                (long long)H * W);
    ImageStrides ns, os;
    for (int k = 0; k < 4; ++k) {
        DRM_REQUIRE(normals_strides[k] >= 0, "refmap_lookup_dense: normals_strides[%d] = %lld is negative", k,
                    (long long)normals_strides[k]);
        DRM_REQUIRE(out_strides[k] >= 0, "refmap_lookup_dense: out_strides[%d] = %lld is negative", k,
                    (long long)out_strides[k]);
        ns.s[k] = normals_strides[k];
        os.s[k] = out_strides[k];
    }
    const int HW = H * W;
    const dim3 grid((unsigned)(((int64_t)HW + 255) / 256), (unsigned)(B < 65535 ? B : 65535));
    refmap_lookup_dense_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(refmap, Hr, Wr, normals, ns, mask,
                                                                                        B, HW, W, C, out, os);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_normalized_log(const float* x, const float* mask, int B, int C, int H, int W, float lowerbound,
                                  float* out, float* log10min_out, float* log10max_out, void* cuda_stream) {
    DRM_REQUIRE(x && mask && out, "normalized_log: null pointer");
    DRM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "normalized_log: sizes must be positive");
    normalized_log_kernel<<<B, POST_THREADS, 0, static_cast<cudaStream_t>(cuda_stream)>>>(x, mask, C, H * W, lowerbound, out,
                                                                                         log10min_out, log10max_out);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_refmap_postprocess(const float* in, int G, int N, int res, float target, int transform,
                                      float* scale_out, float* out, void* cuda_stream) {
    DRM_REQUIRE(in && out, "postprocess: null pointer");
    DRM_REQUIRE(G > 0 && N > 0 && res > 0, "postprocess: G=%d N=%d res=%d must be positive", G, N, res);
    DRM_REQUIRE(transform == 0 || transform == 1, "postprocess: transform %d (0 = none, 1 = log10(x + 0.1) + 1)", transform);
    refmap_postprocess_kernel<<<N, POST_THREADS, 0, static_cast<cudaStream_t>(cuda_stream)>>>(in, G, N, res, target,
                                                                                                transform, scale_out, out);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}

extern "C" int drm_mirmap2envmap(const float* mirmap, const float* basis, int B, int C, int H, int W, int OH, int OW,
                                 float* out, void* cuda_stream) {
    DRM_REQUIRE(mirmap && out, "mirmap2envmap: null pointer");
    DRM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && OH > 0 && OW > 0, "mirmap2envmap: sizes must be positive");
    const int total = OH * OW;
    mirmap2envmap_kernel<<<(total + 255) / 256, 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(mirmap, basis, B, C, H, W,
                                                                                                   OH, OW, out);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(1);
    return DRM_OK;
}
