// K1 (round 2): reflectance-map forward render as a dual-tree gather over a per-render moment pyramid (sm_100a).
//
// Replaces MitsubaRefMapRenderer.rendering (reference utils/mitsuba3_utils.py:411-430 -> :365-409 -> :217-246) and the
// per-render loops around it (models/drmnet.py:561-569, :680-691).  The defining sum (DESIGN.md 3)
//
//   out[k,i,j,c] = sum_{a,b<S} w_a w_b  sum_texels f_c(d_t; v_k, n(theta_i,a, phi_j,b); z_k) E[t,c] dOmega_t
//
// has 16384 S^2 x 2e6 terms per refmap.  Round 1 evaluated ~7e5 (sub-normal, texel) pairs per cell on three map levels;
// here the work per cell is ~1e4 pairs, independent of the map size up to a logarithm:
//
//   * SOURCE SIDE.  Per render a pyramid over the texels (cells of 2^l x 2^l texels, l = 1..L) stores, per cell, the
//     moments of the Fresnel-weighted energy in HALF-VECTOR space: mean mu (inside the unit ball), covariance Sigma,
//     RGB energy w, and the first-moment residuals of the R and B channels about the common mean.  2 - 2 n.h is linear
//     in h, so the mean of the GGX argument over a cell is exact and the lobe is expanded to second order in that one
//     scalar: a cell of half-vector radius r is accurate where r <= kappa sqrt(alpha^2 + delta^2) (delta = distance of
//     the normal from the cell) with kappa ~ 0.1 instead of the ~0.02 a centroid-only cell needs -- 25x fewer cells.
//     Rough lobes add the second-order terms of the shadowing factor G1(n.d) and a clamp of n.d at the horizon applied
//     to the cell's own distribution of n.d.  The diffuse lobe uses the same records in direction space.
//   * PIXEL SIDE.  Footprint lattices (1,2,4,8,16 Gauss-Legendre nodes per axis) are passes: pass p works on blocks of
//     4 x 8 nodes of the 2^p lattice (one warp; 32 cells at p = 0, an eighth of a cell at p = 4), accepts the cells of
//     the pyramid that are far enough for that lattice and hands the rest, unrefined, to its four child blocks of the
//     next pass through a list in global memory.  Every block walks its part of the tree with a private stack, so every
//     (node, texel) pair is counted exactly once by construction; pass 0 nodes carry the covariance of the refmap cell,
//     which makes the 1x1 lattice fourth-order accurate in (cell / lobe width).
//
// The inner loops are bound by the FP32 / MUFU pipes (DESIGN.md 5): the envmap is read once by the pyramid build and
// stays in L2 for the traversal.
#include <cuda_fp16.h>
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace drm {

static constexpr int TREE_THREADS = 256;
static constexpr int TREE_WARPS = 8;
static constexpr int REC4 = 5;         // float4 per pyramid record in global memory
static constexpr int SREC4 = 7;        // float4 per staged record of the diffuse pass
static constexpr int PAIR4 = 13;       // float4 per staged PAIR of records of the specular passes (26 fields x 2)
static constexpr int MAX_PYR = 14;
static constexpr int STACK_CAP = 1024; // entries per warp
static constexpr int BUF1 = 32;        // staged pyramid records per warp
static constexpr int BUF0 = 32;        // staged texel records per warp
static constexpr int TREE_MAX_P = 4;   // lattices 1,2,4,8,16
static constexpr int CHUNK = 128;      // ints per chunk of a hand-over list (2 header + 126 entries)
static constexpr int TREE_CHUNK = 64;  // renders per launch sequence: bounds the workspace for large batches

struct PyrGeom {
    int L, base;                 // top level; first stored level (1 for the specular pyramid; the diffuse one starts where
                                 // its cells reach ~0.03 rad)
    int H[MAX_PYR], W[MAX_PYR];
    long off[MAX_PYR];           // record offset of level l inside one pyramid
    long cells;                  // records per pyramid
};

struct TreeConst {  // per render
    float vhat[3], left[3], upp[3];
    float m, rough, alpha2, inv_a2m1, one_m_a2, eta;
    float base[3], cdiff[3];
    float thr[TREE_MAX_P + 1];  // half-vector-space distance beyond which lattice 2^p resolves the cell average
    int env, has_spec, has_diff, full2;
    int pk, pad[3];  // log2 of the render's footprint S
};

struct TreeArgs {
    const float* env;
    const TreeConst* rc;
    const float *sin_t, *cos_t, *sin_p, *cos_p;
    const float4* pyr_s;   // [N][geom_s.cells][REC4]
    const float4* pyr_d;   // [B][geom_d.cells][REC4]
    float* out;
    int* status;           // [0]: list / stack overflow flag
    const int* env_used;   // [B] envmaps whose diffuse pyramid this call reads
    const int* act;        // [TREE_MAX_P + 1][TREE_CHUNK] renders active in pass p, and their number
    const int* nact;
    // hand-over lists: chains of CHUNK-int chunks ([0] next chunk or -1, [1] entries, [2..] entries) in a pool per pass
    const int* pool_in;    // chunks written by the previous pass
    const int* heads_in;   // [N][blocks of the previous pass] first chunk or -1
    int* pool_out;         // this pass's pool, heads and allocation counter
    int* heads_out;
    int* pool_ctr;
    int* item_ctr;         // work counter of this pass's persistent CTAs
    int pool_cap;          // chunks in pool_out
    PyrGeom gs, gd;
    int B, He, We, N, res, pk, channel_first, pixcov;
    float cell, domega_k, kappa, rcap, rcap_simple, hz, hz_in, hz_nv, hz_fin, kappa_d, hz_d, hand, limb_nv, limb_boost, limb_x, limb_hand, limb_ramp, limb_sub, limb_cells;
    float glx[TREE_MAX_P + 1][16], glw[TREE_MAX_P + 1][16];  // Gauss-Legendre lattices 1, 2, 4, 8, 16
    int stats;                   // debug: count visits / accepted records per pass into status[16..]
    int diff_cov;                // diffuse pass: 1x1 lattice with the cell covariance (else the render's own lattice)
};

__device__ __forceinline__ float fresnel_dielectric_t(float cos_i, float eta) {
    const float eta_ti = fast_rcp(eta);
    const float ct2 = 1.f - eta_ti * eta_ti * (1.f - cos_i * cos_i);
    if (ct2 <= 0.f) return 1.f;
    const float ct = fast_sqrt(ct2);
    const float a_s = (cos_i - eta * ct) * fast_rcp(cos_i + eta * ct);
    const float a_p = (ct - eta * cos_i) * fast_rcp(ct + eta * cos_i);
    return 0.5f * (a_s * a_s + a_p * a_p);
}

__global__ void tree_tables_kernel(float* sin_t, float* cos_t, float* sin_p, float* cos_p, int He, int We) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < He) {
        const double t = (i + 0.5) * (M_PI / He);
        sin_t[i] = (float)sin(t);
        cos_t[i] = (float)cos(t);
    }
    if (i < We) {
        const double p = (i + 0.5) * (2.0 * M_PI / We);
        sin_p[i] = (float)sin(p);
        cos_p[i] = (float)cos(p);
    }
}

// clip z to [0,1] (mitsuba3_utils.py:239,242), BSDF constants, camera frame of look_at(v, 0, +Y) (:235-236), lattice thresholds
__global__ void tree_setup_kernel(const float* __restrict__ z6, const float* __restrict__ view3,
                                  const uint8_t* __restrict__ flip, const int32_t* __restrict__ env_index, int N, int B,
                                  float alpha_min, float cell, float level_scale, float level_scale0,
                                  float alpha_full2, int pixcov, float flat_scale, int S_uniform, const int32_t* __restrict__ S_per_render,
                                  TreeConst* __restrict__ rc, int* __restrict__ status) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    TreeConst c;
    float z[6];
    for (int i = 0; i < 6; ++i) z[i] = fminf(fmaxf(z6[6 * k + i], 0.f), 1.f);
    c.m = z[0];
    c.base[0] = z[1]; c.base[1] = z[2]; c.base[2] = z[3];
    c.rough = z[4];
    const float alpha = fmaxf(z[4] * z[4], alpha_min);
    c.alpha2 = alpha * alpha;
    c.inv_a2m1 = 1.f / c.alpha2 - 1.f;
    c.one_m_a2 = 1.f - c.alpha2;
    c.eta = 2.f / (1.f - sqrtf(0.08f * z[5])) - 1.f;
    {
        // Gauss-Legendre error of an S-point rule on a (alpha^2 + d^2)^-2 tail, weighted by the tail mass (DESIGN.md 5)
        const float ca = cell * alpha;
        c.thr[0] = 21.0f * sqrtf(ca);
        c.thr[1] = 7.5f * powf(cell, 2.f / 3.f) * powf(alpha, 1.f / 3.f);
        c.thr[2] = 2.4f * powf(cell, 0.8f) * powf(alpha, 0.2f);
        c.thr[3] = 1.2f * powf(cell, 8.f / 9.f) * powf(alpha, 1.f / 9.f);
        c.thr[4] = 0.f;
        for (int i = 0; i < TREE_MAX_P; ++i) c.thr[i] = (i == 0 ? level_scale0 : level_scale) * fmaxf(c.thr[i], 6.f * alpha);
        // ... which assumes that a band's share of the pixel is the tail mass.  A lattice is also accurate wherever the
        // lobe is flat across the cell: the 2^p-point rule (the 1x1 node with the cell covariance is fourth order like
        // the 2x2 rule) errs by ~ (cell / sqrt(alpha^2 + d^2))^(2^(p+1)), below 1e-4 beyond c_p cells.  The smaller of
        // the two distances serves: wide lobes leave the fine lattices early, sharp ones keep the calibrated rule.
        const float cp[TREE_MAX_P] = {pixcov ? 5.5f : 1e3f, 4.f, 2.6f, 1.7f};
        for (int i = 0; i < TREE_MAX_P; ++i) {
            const float flat = sqrtf(fmaxf(cp[i] * cp[i] * cell * cell * flat_scale * flat_scale - c.alpha2, 0.f));
            c.thr[i] = fminf(c.thr[i], flat);
        }
    }
    for (int i = 0; i < 3; ++i) c.cdiff[i] = (1.f - c.m) * c.base[i] * (float)M_1_PI;
    c.has_diff = c.cdiff[0] > 0.f || c.cdiff[1] > 0.f || c.cdiff[2] > 0.f;
    // F = (1-m) F_dielectric + m (c + (1-c) schlick) vanishes only for a non-metal with specular = 0 (eta = 1)
    c.has_spec = !(c.m == 0.f && z[5] == 0.f);
    float vx = view3[3 * k], vy = view3[3 * k + 1], vz = view3[3 * k + 2];
    const float inv = rsqrtf(vx * vx + vy * vy + vz * vz);
    vx *= inv; vy *= inv; vz *= inv;
    c.vhat[0] = vx; c.vhat[1] = vy; c.vhat[2] = vz;
    const float fx = -vx, fy = -vy, fz = -vz;  // forward
    float lx = fz, ly = 0.f, lz = -fx;         // up x forward, up = (0,1,0)
    const float linv = rsqrtf(lx * lx + lz * lz);
    lx *= linv; lz *= linv;
    c.upp[0] = fy * lz - fz * ly;  // forward x left
    c.upp[1] = fz * lx - fx * lz;
    c.upp[2] = fx * ly - fy * lx;
    const float sgn = (flip && flip[k]) ? -1.f : 1.f;
    c.left[0] = sgn * lx; c.left[1] = sgn * ly; c.left[2] = sgn * lz;
    const int e = env_index ? env_index[k] : k;
    if (e < 0 || e >= B) atomicOr(status, 2);  // reported by drm_render_status; the render uses a clamped index
    c.env = min(max(e, 0), B - 1);
    c.full2 = alpha >= alpha_full2;
    {
        // footprint: given per render, given for the call, or chosen from the ratio of cell width to lobe half-width
        // (the rule of renderer.auto_footprint: the cell average of the lobe resolved to ~2e-4)
        int S = S_per_render ? S_per_render[k] : S_uniform;
        if (S <= 0) {
            const float ratio = cell / alpha;
            S = ratio < 0.1f ? 1 : ratio < 0.6f ? 2 : ratio < 2.f ? 4 : ratio < 4.f ? 8 : 16;
        }
        int pk = 0;
        while ((1 << pk) < S && pk < TREE_MAX_P) ++pk;
        if ((1 << pk) != S) atomicOr(status, 8);  // not one of 1, 2, 4, 8, 16: rounded up, reported
        c.pk = pk;
        c.pad[0] = c.pad[1] = c.pad[2] = 0;
    }
    rc[k] = c;
}

// ---------------------------------------------------------------------------------------------------------------------
// Pyramid build.  A record holds the moments of a set of unit vectors x_t (half vectors for the specular pyramid,
// directions for the diffuse one) with RGB weights w_t,c, omega_t = sum_c w_t,c:
//   mu = sum omega x / sum omega,  Sigma = sum omega (x - mu)(x - mu)^T / sum omega,  w_c = sum_t w_t,c,
//   m_c = sum_t w_t,c (x_t - mu)  for c = R, B  (G follows: the three residuals sum to zero),
//   rh  = max_t |x_t - mu|  (chord).
// Sums are accumulated about a reference point inside the cell: Sigma ~ 1e-6 would drown in the rounding of mu mu^T.
// ---------------------------------------------------------------------------------------------------------------------
struct Mom {
    float ref[3], om, s1[3], s2[6], w[3], cR[3], cB[3];
    bool any;
    __device__ __forceinline__ void init() {
        om = 0.f; any = false;
        for (int i = 0; i < 3; ++i) { ref[i] = 0.f; s1[i] = 0.f; w[i] = 0.f; cR[i] = 0.f; cB[i] = 0.f; }
        for (int i = 0; i < 6; ++i) s2[i] = 0.f;
    }
    // a point mass (texel)
    __device__ __forceinline__ void add_point(const float* x, const float* wc) {
        const float o = wc[0] + wc[1] + wc[2];
        if (!(o > 0.f)) return;
        if (!any) { any = true; ref[0] = x[0]; ref[1] = x[1]; ref[2] = x[2]; }
        const float dx = x[0] - ref[0], dy = x[1] - ref[1], dz = x[2] - ref[2];
        om += o;
        s1[0] += o * dx; s1[1] += o * dy; s1[2] += o * dz;
        s2[0] += o * dx * dx; s2[1] += o * dy * dy; s2[2] += o * dz * dz;
        s2[3] += o * dx * dy; s2[4] += o * dx * dz; s2[5] += o * dy * dz;
        w[0] += wc[0]; w[1] += wc[1]; w[2] += wc[2];
        cR[0] += wc[0] * dx; cR[1] += wc[0] * dy; cR[2] += wc[0] * dz;
        cB[0] += wc[2] * dx; cB[1] += wc[2] * dy; cB[2] += wc[2] * dz;
    }
    // a child record
    __device__ __forceinline__ void add_record(const float4* r) {
        const float4 g0 = r[0], g1 = r[1], g2 = r[2], g3 = r[3], g4 = r[4];
        const float o = g2.z + g2.w + g3.x;
        if (!(o > 0.f)) return;
        if (!any) { any = true; ref[0] = g0.x; ref[1] = g0.y; ref[2] = g0.z; }
        const float dx = g0.x - ref[0], dy = g0.y - ref[1], dz = g0.z - ref[2];
        om += o;
        s1[0] += o * dx; s1[1] += o * dy; s1[2] += o * dz;
        s2[0] += o * (g1.x + dx * dx); s2[1] += o * (g1.y + dy * dy); s2[2] += o * (g1.z + dz * dz);
        s2[3] += o * (g1.w + dx * dy); s2[4] += o * (g2.x + dx * dz); s2[5] += o * (g2.y + dy * dz);
        w[0] += g2.z; w[1] += g2.w; w[2] += g3.x;
        cR[0] += g3.y + g2.z * dx; cR[1] += g3.z + g2.z * dy; cR[2] += g3.w + g2.z * dz;
        cB[0] += g4.x + g3.x * dx; cB[1] += g4.y + g3.x * dy; cB[2] += g4.z + g3.x * dz;
    }
    // mu etc.; rh is set by the caller (it needs the members again)
    __device__ __forceinline__ void finish(float4* r, float rh, float* mu_out) const {
        if (!any) {
            for (int i = 0; i < REC4; ++i) r[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            mu_out[0] = mu_out[1] = mu_out[2] = 0.f;
            return;
        }
        const float io = 1.f / om;
        const float ax = s1[0] * io, ay = s1[1] * io, az = s1[2] * io;
        mu_out[0] = ref[0] + ax; mu_out[1] = ref[1] + ay; mu_out[2] = ref[2] + az;
        r[0] = make_float4(mu_out[0], mu_out[1], mu_out[2], rh);
        r[1] = make_float4(fmaxf(s2[0] * io - ax * ax, 0.f), fmaxf(s2[1] * io - ay * ay, 0.f), fmaxf(s2[2] * io - az * az, 0.f),
                           s2[3] * io - ax * ay);
        r[2] = make_float4(s2[4] * io - ax * az, s2[5] * io - ay * az, w[0], w[1]);
        r[3] = make_float4(w[2], cR[0] - w[0] * ax, cR[1] - w[0] * ay, cR[2] - w[0] * az);
        r[4] = make_float4(cB[0] - w[2] * ax, cB[1] - w[2] * ay, cB[2] - w[2] * az, 0.f);
    }
};

// Envmap texels are fp32 or fp16 (T = float or __half), 3 scalars a texel, converted where they are loaded.  fp16 -> fp32
// is exact, so an fp16 envmap renders bit for bit like its fp32 upcast.  TreeArgs::env points to either; the kernels
// that read texels cast it to T.
__device__ __forceinline__ float texel_f(float x) { return x; }
__device__ __forceinline__ float texel_f(__half x) { return __half2float(x); }

// texel (r, c) of render rc / envmap e: half vector, v.h, Fresnel-weighted energy
template <typename T>
__device__ __forceinline__ void texel_spec(const TreeArgs& g, const TreeConst& rc, const T* __restrict__ env_b, int r,
                                           int c, float* h, float& vh, float* w) {
    const float st = g.sin_t[r], ct = g.cos_t[r], sp = g.sin_p[c], cp = g.cos_p[c];
    const float dx = st * sp, dy = ct, dz = -st * cp;
    const float dom = g.domega_k * st;
    const T* e = env_b + ((size_t)r * g.We + c) * 3;
    // |v + d|^2 from its components: 2 + 2 v.d cancels at grazing reflection (d ~ -v), which the limb cells see
    const float sx = rc.vhat[0] + dx, sy = rc.vhat[1] + dy, sz = rc.vhat[2] + dz;
    const float len2 = fmaxf(sx * sx + sy * sy + sz * sz, 1e-12f);
    const float inv_len = rsqrtf(len2);
    vh = 0.5f * len2 * inv_len;
    h[0] = sx * inv_len; h[1] = sy * inv_len; h[2] = sz * inv_len;
    const float Fd = fresnel_dielectric_t(vh, rc.eta);
    const float mm = fminf(fmaxf(1.f - vh, 0.f), 1.f);
    const float sw = (mm * mm) * (mm * mm) * mm;
    const float a = (1.f - rc.m) * Fd + rc.m * sw, b = rc.m * (1.f - sw);  // F_c = a + b base_c
    w[0] = texel_f(e[0]) * dom * (a + b * rc.base[0]);
    w[1] = texel_f(e[1]) * dom * (a + b * rc.base[1]);
    w[2] = texel_f(e[2]) * dom * (a + b * rc.base[2]);
}

template <typename T>
__device__ __forceinline__ void texel_diff(const TreeArgs& g, const T* __restrict__ env_b, int r, int c, float* d,
                                           float* w) {
    const float st = g.sin_t[r], ct = g.cos_t[r], sp = g.sin_p[c], cp = g.cos_p[c];
    d[0] = st * sp; d[1] = ct; d[2] = -st * cp;
    const float dom = g.domega_k * st;
    const T* e = env_b + ((size_t)r * g.We + c) * 3;
    w[0] = texel_f(e[0]) * dom; w[1] = texel_f(e[1]) * dom; w[2] = texel_f(e[2]) * dom;
}

// level `lev` of a pyramid straight from the texels (lev = 1 for the specular pyramid of render blockIdx.y, the base
// level of the diffuse pyramid of envmap blockIdx.y)
__global__ void tree_mark_used_kernel(const TreeConst* __restrict__ rc, int N, int* __restrict__ used) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < N && rc[k].has_diff) used[rc[k].env] = 1;
}

// drm_env_pyramid_build: mark the listed slots of a bank (ids == NULL: every slot); ids outside [0, B) are skipped
__global__ void env_mark_slots_kernel(const int32_t* __restrict__ ids, int n, int B, int* __restrict__ used) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (!ids) {
        if (i < B) used[i] = 1;
    } else if (i < n) {
        const int e = ids[i];
        if (e >= 0 && e < B) used[e] = 1;
    }
}

// per lattice pass p: the renders of this chunk whose own lattice is at least 2^p (one thread: a chunk has <= 64 renders)
__global__ void tree_active_kernel(const TreeConst* __restrict__ rc, int n, int* __restrict__ act, int* __restrict__ nact) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    for (int p = 0; p <= TREE_MAX_P; ++p) {
        int c = 0;
        for (int k = 0; k < n; ++k)
            if (rc[k].pk >= p) act[p * TREE_CHUNK + c++] = k;
        nact[p] = c;
    }
}

template <bool SPEC, typename T>
__device__ __forceinline__ void pyr_from_texels(const TreeArgs& g, int lev, float4* __restrict__ pyr) {
    const PyrGeom& G = SPEC ? g.gs : g.gd;
    const int Hl = G.H[lev], Wl = G.W[lev];
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= Hl * Wl) return;
    const int k = blockIdx.y;
    if (!SPEC && !g.env_used[k]) return;  // no render of this call reads this envmap's diffuse pyramid
    const int R = cell / Wl, C = cell - R * Wl;
    const int e = 1 << lev;
    const TreeConst* rcp = SPEC ? &g.rc[k] : nullptr;
    const T* env_b = reinterpret_cast<const T*>(g.env) + (size_t)(SPEC ? rcp->env : k) * g.He * g.We * 3;
    float4* rec = pyr + ((size_t)k * G.cells + G.off[lev] + cell) * REC4;
    if (SPEC && !rcp->has_spec) {
        for (int i = 0; i < REC4; ++i) rec[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    Mom M;
    M.init();
    const int r1 = min((R + 1) * e, g.He), c1 = min((C + 1) * e, g.We);
    for (int r = R * e; r < r1; ++r)
        for (int c = C * e; c < c1; ++c) {
            float x[3], w[3], vh;
            if (SPEC) texel_spec(g, *rcp, env_b, r, c, x, vh, w);
            else texel_diff(g, env_b, r, c, x, w);
            M.add_point(x, w);
        }
    float4 out[REC4];
    float mu[3];
    M.finish(out, 0.f, mu);
    float rh = 0.f;
    if (M.any) {
        for (int r = R * e; r < r1; ++r)
            for (int c = C * e; c < c1; ++c) {
                float x[3], w[3], vh;
                if (SPEC) texel_spec(g, *rcp, env_b, r, c, x, vh, w);
                else texel_diff(g, env_b, r, c, x, w);
                if (w[0] + w[1] + w[2] > 0.f) {
                    const float dx = x[0] - mu[0], dy = x[1] - mu[1], dz = x[2] - mu[2];
                    rh = fmaxf(rh, dx * dx + dy * dy + dz * dz);
                }
            }
        out[0].w = sqrtf(rh) * 1.0001f + 1e-7f;
    }
    for (int i = 0; i < REC4; ++i) rec[i] = out[i];
}

template <bool SPEC>
__global__ void pyr_from_texels_kernel(const TreeArgs g, int lev, float4* __restrict__ pyr) {
    pyr_from_texels<SPEC, float>(g, lev, pyr);
}
template <bool SPEC>
__global__ void pyr_from_texels_kernel_h(const TreeArgs g, int lev, float4* __restrict__ pyr) {
    pyr_from_texels<SPEC, __half>(g, lev, pyr);
}

// level lev from level lev - 1 of every pyramid (blockIdx.y = pyramid)
__global__ void pyr_merge_kernel(PyrGeom G, int lev, float4* __restrict__ pyr, const int* __restrict__ used) {
    const int Hl = G.H[lev], Wl = G.W[lev], Hc = G.H[lev - 1], Wc = G.W[lev - 1];
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    if (cell >= Hl * Wl) return;
    if (used && !used[blockIdx.y]) return;
    const int R = cell / Wl, C = cell - R * Wl;
    float4* base = pyr + (size_t)blockIdx.y * G.cells * REC4;
    const float4* child = base + G.off[lev - 1] * REC4;
    Mom M;
    M.init();
    for (int dr = 0; dr < 2; ++dr)
        for (int dc = 0; dc < 2; ++dc) {
            const int r = 2 * R + dr, c = 2 * C + dc;
            if (r < Hc && c < Wc) M.add_record(child + ((size_t)r * Wc + c) * REC4);
        }
    float4 out[REC4];
    float mu[3];
    M.finish(out, 0.f, mu);
    if (M.any) {
        float rh = 0.f;
        for (int dr = 0; dr < 2; ++dr)
            for (int dc = 0; dc < 2; ++dc) {
                const int r = 2 * R + dr, c = 2 * C + dc;
                if (r >= Hc || c >= Wc) continue;
                const float4* ch = child + ((size_t)r * Wc + c) * REC4;
                const float4 g0 = ch[0], g2 = ch[2], g3 = ch[3];
                if (!(g2.z + g2.w + g3.x > 0.f)) continue;
                const float dx = g0.x - mu[0], dy = g0.y - mu[1], dz = g0.z - mu[2];
                rh = fmaxf(rh, sqrtf(dx * dx + dy * dy + dz * dz) + g0.w);
            }
        out[0].w = rh * 1.0001f + 1e-7f;
    }
    float4* rec = base + (G.off[lev] + cell) * REC4;
    for (int i = 0; i < REC4; ++i) rec[i] = out[i];
}

// ---------------------------------------------------------------------------------------------------------------------
// Traversal
// ---------------------------------------------------------------------------------------------------------------------
// The view-side factor G1(n.v) / (4 n.v) (with D's normalisation) varies on the scale alpha at the limb however far the
// texel is.  A node of a lattice coarser than the render's own stands for the m x m nodes of that lattice in its
// sub-region: it carries their weighted mean of the factor and moves by the shift of the weighted centroid, which
// cancels the first-order cross term with the texel-dependent part (round 1, DESIGN.md 5.2).
__device__ __forceinline__ float view_term_t(const TreeConst& rc, float lz) {
    const float g1 = lz + sqrtf(lz * lz * rc.one_m_a2 + rc.alpha2);
    return lz > 0.f ? 1.f / (3.14159265358979f * rc.alpha2 * g1) : 0.f;
}

struct NodeT {
    float nx, ny, nz, nv, mult, wq, Fi;
    float q0, q1, q2, q3, q4, q5;  // n_x^2, n_y^2, n_z^2, 2 n_x n_y, 2 n_x n_z, 2 n_y n_z
    float P0, P1, P2, P3, P4, P5;  // covariance of the normal over the refmap cell (pass 0 of a render with S > 1)
    bool active;
};

__device__ __forceinline__ void make_node(const TreeArgs& g, const TreeConst& rc, int p, bool pixcov, int I, int J, bool spec,
                                          NodeT& nd) {
    const int pk = rc.pk, Sk = 1 << p, S = 1 << pk;
    const float* __restrict__ glx = g.glx[p];
    const float* __restrict__ glw = g.glw[p];
    const float* __restrict__ fx = g.glx[pk];
    const float* __restrict__ fw = g.glw[pk];
    const int NG = g.res << p;
    nd.active = I < NG && J < NG;
    const int i = I >> p, a = I & (Sk - 1), j = J >> p, b = J & (Sk - 1);
    float sa = 0.f, sb = 0.f, meanv = -1.f;
    if (spec && p < pk && nd.active) {
        const int m = S / Sk;
        float num = 0.f, den = 0.f, va = 0.f, vb = 0.f, ua = 0.f, ub = 0.f;
        for (int ia = 0; ia < m; ++ia) {
            const float xa = fx[a * m + ia], wa = fw[a * m + ia];
            const float st = sinf(((float)i + 0.5f + 0.5f * xa) * g.cell);
            for (int ib = 0; ib < m; ++ib) {
                const float xb = fx[b * m + ib];
                const float sp = sinf(((float)j + 0.5f + 0.5f * xb) * g.cell);
                const float w = wa * fw[b * m + ib];
                const float wv = w * view_term_t(rc, st * sp);
                num += wv; den += w;
                va += wv * xa; vb += wv * xb;
                ua += w * xa; ub += w * xb;
            }
        }
        if (num > 0.f) { meanv = num / den; sa = va / num - ua / den; sb = vb / num - ub / den; }
        else meanv = 0.f;
    }
    const float th = ((float)i + 0.5f + 0.5f * (glx[a] + sa)) * g.cell;
    const float ph = ((float)j + 0.5f + 0.5f * (glx[b] + sb)) * g.cell;
    float st, ct, sp, cp;
    sincosf(th, &st, &ct);
    sincosf(ph, &sp, &cp);
    const float lx = st * cp, lz = st * sp;
    nd.nx = lx * rc.left[0] + ct * rc.upp[0] + lz * rc.vhat[0];
    nd.ny = lx * rc.left[1] + ct * rc.upp[1] + lz * rc.vhat[1];
    nd.nz = lx * rc.left[2] + ct * rc.upp[2] + lz * rc.vhat[2];
    nd.nv = lz;  // n . v exactly, the frame is orthonormal
    nd.wq = nd.active ? glw[a] * glw[b] : 0.f;
    nd.mult = nd.wq * (meanv >= 0.f ? meanv : view_term_t(rc, lz));
    const float mm = fminf(fmaxf(1.f - lz, 0.f), 1.f);
    nd.Fi = (mm * mm) * (mm * mm) * mm;
    nd.q0 = nd.nx * nd.nx; nd.q1 = nd.ny * nd.ny; nd.q2 = nd.nz * nd.nz;
    nd.q3 = 2.f * nd.nx * nd.ny; nd.q4 = 2.f * nd.nx * nd.nz; nd.q5 = 2.f * nd.ny * nd.nz;
    nd.P0 = nd.P1 = nd.P2 = nd.P3 = nd.P4 = nd.P5 = 0.f;
    if (pixcov) {
        // uniform box in (theta, phi) of width cell: covariance (cell^2 / 12)(e_t e_t^T + e_p e_p^T), e = dn/dtheta, dn/dphi
        const float var = g.cell * g.cell * (1.f / 12.f);
        const float lxt = ct * cp, lzt = ct * sp, lxp = -st * sp, lzp = st * cp;
        float et[3], ep[3];
        for (int c = 0; c < 3; ++c) {
            et[c] = lxt * rc.left[c] - st * rc.upp[c] + lzt * rc.vhat[c];
            ep[c] = lxp * rc.left[c] + lzp * rc.vhat[c];
        }
        nd.P0 = var * (et[0] * et[0] + ep[0] * ep[0]);
        nd.P1 = var * (et[1] * et[1] + ep[1] * ep[1]);
        nd.P2 = var * (et[2] * et[2] + ep[2] * ep[2]);
        nd.P3 = 2.f * var * (et[0] * et[1] + ep[0] * ep[1]);
        nd.P4 = 2.f * var * (et[0] * et[2] + ep[0] * ep[2]);
        nd.P5 = 2.f * var * (et[1] * et[2] + ep[1] * ep[2]);
    }
}

__device__ __forceinline__ float warp_sum(float v) {
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
    for (int d = 16; d > 0; d >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}
__device__ __forceinline__ float chord_angle(float c2) { return 2.f * asinf(fminf(1.f, 0.5f * sqrtf(c2))); }
// The traversal decides with cheap approximations of the same angles: a decision only selects the level a part of the map
// is read at (every block still walks the whole map exactly once), so ~1e-4 rad of slack is harmless.
// angle of a squared chord c2 in [0,4]: acos(1 - c2/2) by Abramowitz-Stegun 4.4.45 (|error| < 7e-5 rad)
__device__ __forceinline__ float fast_chord_angle(float c2) {
    const float x = 1.f - 0.5f * c2, ax = fabsf(x);
    const float s = fast_sqrt(x >= 0.f ? 0.5f * c2 : fmaxf(2.f - 0.5f * c2, 0.f));  // sqrt(1 - |x|) without cancellation
    const float pol = 1.5707288f + ax * (-0.2121144f + ax * (0.0742610f - 0.0187293f * ax));
    const float a = s * pol;
    return x >= 0.f ? a : 3.14159265f - a;
}
// angle of a small chord c (a cell radius): 2 asin(c/2) by its series below 0.5, a generous bound above
__device__ __forceinline__ float fast_radius_angle(float c) {
    const float c2 = c * c;
    return c < 0.5f ? c * (1.f + c2 * (1.f / 24.f + c2 * (3.f / 640.f))) + 1e-5f : 1.6f * c;
}

// cone (axis, half angle) of the warp's active nodes, widened by the sub-cells the nodes stand for
__device__ __forceinline__ bool warp_cone(const TreeArgs& g, int p, const NodeT& nd, float& ax, float& ay, float& az, float& beta) {
    const float wa = nd.active ? 1.f : 0.f;
    ax = warp_sum(wa * nd.nx); ay = warp_sum(wa * nd.ny); az = warp_sum(wa * nd.nz);
    const float cnt = warp_sum(wa);
    if (cnt == 0.f) return false;
    const float inv = rsqrtf(fmaxf(ax * ax + ay * ay + az * az, 1e-30f));
    ax *= inv; ay *= inv; az *= inv;
    const float dx = nd.nx - ax, dy = nd.ny - ay, dz = nd.nz - az;
    // rounded term by term: with p known at compile time (p = 0) the compiler would otherwise fuse 0.75 cell + max into
    // one FMA and move cone decisions by an ulp against the same cone at a run-time p
    beta = __fadd_rn(warp_max(nd.active ? chord_angle(dx * dx + dy * dy + dz * dz) : 0.f),
                     __fmul_rn(0.75f, g.cell) / (float)(1 << p));
    return true;
}

enum : int { ACT_DROP = 0, ACT_ACCEPT = 1, ACT_REFINE = 2, ACT_HAND = 3 };

// packed fp32 pairs (FFMA2 / FADD2 / FMUL2 on sm_100a): the evaluation loops handle two pyramid records per iteration
typedef float2 f2;
__device__ __forceinline__ f2 F2(float a) { return make_float2(a, a); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ f2 max2(f2 a, float s) { return make_float2(fmaxf(a.x, s), fmaxf(a.y, s)); }
__device__ __forceinline__ f2 rcp2(f2 a) { return make_float2(fast_rcp(a.x), fast_rcp(a.y)); }
__device__ __forceinline__ f2 rsqrt2(f2 a) { return make_float2(fast_rsqrt(a.x), fast_rsqrt(a.y)); }
__device__ __forceinline__ f2 sqrt2(f2 a) { return make_float2(fast_sqrt(a.x), fast_sqrt(a.y)); }
__device__ __forceinline__ f2 lo(float4 v) { return make_float2(v.x, v.y); }
__device__ __forceinline__ f2 hi(float4 v) { return make_float2(v.z, v.w); }

// add the per-node sums to the cells of the CTA's 16 x 16 node tile, in fixed order (deterministic)
__device__ __forceinline__ void tile_writeback(const TreeArgs& g, int p, float* red, int k, int ti, int tj, float a0, float a1,
                                               float a2, bool overwrite) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ln = ((warp >> 1) * 4 + (lane >> 3)) * 16 + (warp & 1) * 8 + (lane & 7);  // node (row, col) inside the tile
    red[ln * 3 + 0] = a0; red[ln * 3 + 1] = a1; red[ln * 3 + 2] = a2;
    __syncthreads();
    const int Sk = 1 << p, cpt = 16 >> p;  // cells per tile edge
    if (cpt < 1) return;
    const int ncell = cpt * cpt;
    for (int o = tid; o < ncell * 3; o += TREE_THREADS) {
        const int cl = o / 3, c = o - cl * 3;
        const int ci = cl / cpt, cj = cl - ci * cpt;
        const int i = ti * cpt + ci, j = tj * cpt + cj;
        if (i >= g.res || j >= g.res) continue;
        float v = 0.f;
        for (int a = 0; a < Sk; ++a)
            for (int b = 0; b < Sk; ++b) v += red[((ci * Sk + a) * 16 + cj * Sk + b) * 3 + c];
        const size_t pix = (size_t)i * g.res + j;
        const size_t idx = g.channel_first ? ((size_t)k * 3 + c) * g.res * g.res + pix : ((size_t)k * g.res * g.res + pix) * 3 + c;
        g.out[idx] = overwrite ? v : g.out[idx] + v;
    }
}

// t-th tile of a tiles_x x tiles_x tile grid in the order the passes hand them out: the perimeter first (top row, bottom
// row, left column, right column), then the interior row by row.  The perimeter tiles hold the rim of the refmap (n.v -> 0
// on all four edges), whose blocks run several times longer than the others: started first, they no longer form the
// tail of the pass.
__device__ __forceinline__ void tile_of(int t, int tiles_x, int& ti, int& tj) {
    const int m = tiles_x - 1;
    if (tiles_x <= 2) { ti = t / tiles_x; tj = t - ti * tiles_x; }
    else if (t < tiles_x) { ti = 0; tj = t; }
    else if (t < 2 * tiles_x) { ti = m; tj = t - tiles_x; }
    else if (t < 2 * tiles_x + (m - 1)) { ti = 1 + t - 2 * tiles_x; tj = 0; }
    else if (t < 4 * m) { ti = 1 + t - 2 * tiles_x - (m - 1); tj = m; }
    else { const int q = t - 4 * m; ti = 1 + q / (m - 1); tj = 1 + q - (ti - 1) * (m - 1); }
}

// Resident CTAs per SM (`__launch_bounds__` minimum) of each specular instance and of the diffuse pass, measured on a
// B200 with the bench batch.  At 3 a thread has 80 registers.  The specular instances fit them without spilling because
// the item's render record and the warp's cone and thresholds live in shared memory (rc, WarpUni) and the evaluation
// loops load each staged float4 where they use it; 3 x (67 584 dynamic + 1 520 static) bytes of shared memory fit an
// SM.  Every pass is faster at 3 than at 2 (render step 178 -> 168 ms).  The diffuse pass: 80 registers, 12 bytes of
// spill, 16.2 -> 13.8 ms a step.  tests/test_kernel_resources.py holds the specular instances to these budgets.
static constexpr int SPEC_MINB[TREE_MAX_P + 1] = {3, 3, 3, 3, 3}, DIFF_MINB = 3;

// collect_stats: per pass p, status[50 + p] += cycles (in units of 1024) the warps spent in the barriers of the item loop,
// waiting for the slowest warp of their tile, and status[56 + p] += their cycles in the kernel.  Outside the 40 words
// drm_render_status copies: scripts/tree_stats.py reads them from the workspace.
static constexpr int STAT_TILE_WAIT = 50, STAT_WARP_CYCLES = 56;

// What a block's traversal decides with that is the same in every lane of its warp: its cone and the thresholds of this
// pass.  It lives in a per-warp shared slot and is read where it is used, so that it does not hold registers through
// the evaluation loops.
struct WarpUni {
    float ax, ay, az, beta;
    float thr_p, hand_p, hz_p, xthr, rcap, kappa2;
    int limb;
};

// ---- specular lobe, pass P (one instance per lattice 2^P) -------------------------------------------------------------
// The bodies of the texel-reading kernels are device templates on T under fp32 and fp16 __global__ wrappers.  They take
// threadIdx.x from the wrapper, where its range is known from the launch bounds, and this one takes TreeArgs by value:
// either way the fp32 kernels compile to other (equivalent) code than when they held the body themselves.
template <int P, typename T>
__device__ __forceinline__ void tree_spec_pass(const TreeArgs g, int tid) {
    extern __shared__ __align__(16) unsigned char tree_smem[];
    const int lane = tid & 31, warp = tid >> 5;
    int* stack = reinterpret_cast<int*>(tree_smem) + warp * STACK_CAP;
    float* buf1 = reinterpret_cast<float*>(tree_smem + TREE_WARPS * STACK_CAP * 4) + warp * (BUF1 / 2 * PAIR4 * 4);
    float4* buf0 = reinterpret_cast<float4*>(tree_smem + TREE_WARPS * STACK_CAP * 4 + TREE_WARPS * (BUF1 / 2) * PAIR4 * 16) + warp * (BUF0 * 2);
    float* red = reinterpret_cast<float*>(tree_smem);  // reused after the traversal: [256][3]

    constexpr int p = P;
    const int NG = g.res << p;
    const int tiles_x = (NG + 15) / 16;
    const int n_items = g.nact[p] * tiles_x * tiles_x;
    // barriers of the item loop; under collect_stats they also count the cycles the warp waits in them
    const bool stats = g.stats;
    long long t_warp = stats ? clock64() : 0, t_wait = 0;
    auto tile_sync = [&]() {
        const long long t = stats ? clock64() : 0;
        __syncthreads();
        if (stats) t_wait += clock64() - t;
    };
    // persistent CTAs: items = (active render, tile of 16 x 16 lattice nodes), tile-major so that the renders interleave,
    // handed out by a counter in the order of tile_of (the rim tiles take several times longer than the others)
    // the item's render record is read from shared memory where it is used: one copy per CTA instead of 34 registers
    __shared__ int next_item, next_k;
    __shared__ TreeConst rc;
    __shared__ WarpUni wu_s[TREE_WARPS];
    WarpUni& wu = wu_s[warp];
    while (true) {
    if (warp == 0) {
        int it = 0;
        if (lane == 0) it = atomicAdd(g.item_ctr, 1);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it < n_items) {
            const int kk = g.act[p * TREE_CHUNK + it % g.nact[p]];
            const int* src = reinterpret_cast<const int*>(g.rc + kk);
            int* dst = reinterpret_cast<int*>(&rc);
            for (int i = lane; i < (int)(sizeof(TreeConst) / 4); i += 32) dst[i] = src[i];
            if (lane == 0) next_k = kk;
        }
        if (lane == 0) next_item = it;
    }
    tile_sync();
    const int item = next_item;
    if (item >= n_items) break;
    const int k = next_k;
    const int tile = item / g.nact[p];
    const int pk = rc.pk;
    int ti, tj;
    tile_of(tile, tiles_x, ti, tj);
    const int I0 = ti * 16 + (warp >> 1) * 4, J0 = tj * 16 + (warp & 1) * 8;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    const bool pixcov = g.pixcov && p == 0 && pk > 0;  // the 1x1 node of a finer footprint carries the cell's covariance

    NodeT nd;
    make_node(g, rc, p, pixcov, I0 + (lane >> 3), J0 + (lane & 7), true, nd);
    float ax, ay, az, beta;
    const bool live = rc.has_spec && warp_cone(g, p, nd, ax, ay, az, beta);

    if (live) {
        const float4* pyr = g.pyr_s + (size_t)k * g.gs.cells * REC4;
        const T* env_b = reinterpret_cast<const T*>(g.env) + (size_t)rc.env * g.He * g.We * 3;
        // input: the top level of the pyramid (pass 0) or the parent block's hand-over list
        const int nbJ = (NG + 7) / 8;
        const int bI = I0 >> 2, bJ = J0 >> 3;
        const int* in_list = nullptr;  // entries of the current chunk
        int in_n, in_pos = 0, in_next = -1;
        if constexpr (p == 0) {
            in_n = g.gs.H[g.gs.L] * g.gs.W[g.gs.L];
        } else {
            const int nbJp = ((g.res << (p - 1)) + 7) / 8;
            const int nbIp = ((g.res << (p - 1)) + 3) / 4;
            const size_t pb = (size_t)k * nbIp * nbJp + (size_t)(bI >> 1) * nbJp + (bJ >> 1);
            in_next = g.heads_in[pb];
            in_n = 0;
        }
        int out_n = 0, out_cur = -1, out_fill = 0, out_head = -1;
        int sp = 0, n1 = 0, n0 = 0, sp_max = 0;
        int st_visits = 0, st_acc0 = 0, st_acc1 = 0, st_iters = 0;
        // at the limb (n.v -> 0) the lobe sits on the horizon of the normal and the cell average converges later
        const float nv_min = -warp_max(nd.active ? -nd.nv : -1.f);
        // ... and n.d = 2 (v.h)(n.h) - n.v moves by the cell's own spread of n.v, so where n.v comes within a few alpha of
        // zero the view factor and the shadowing ramp G1(n.d) vary across the cell however far the half vector is: blocks
        // that touch this rim (the outermost cells of the refmap for a sharp lobe) accept nothing that comes near on the
        // coarse lattices: it all goes down to the render's own lattice.
        // (a lattice whose sub-cells are narrower than limb_sub * alpha resolves that ramp: no rim rule on it)
        const float subw = g.cell / (float)(1 << p);
        const bool limb = nv_min < fmaxf(g.limb_nv, fminf(g.limb_x * sqrtf(rc.alpha2), g.limb_cells * g.cell)) &&
                          subw * subw > g.limb_sub * g.limb_sub * rc.alpha2;
        const float thr_p = rc.thr[p] * (limb ? g.limb_boost : 1.f);
        const float hand_p = limb ? g.limb_hand : g.hand;
        // the horizon ramp matters most where the lobe itself sits on it: n.v within a few lobe widths of zero
        const float hz_p = (limb || nv_min < g.hz_nv * sqrtf(rc.alpha2)) ? (p == pk && rc.full2 ? g.hz_fin : g.hz) : g.hz_in;
        const float xthr = g.limb_ramp * sqrtf(rc.alpha2);
        const float kappa2 = g.kappa * g.kappa;
        // wide cells need the second-order terms of G1(n.d) whatever the lobe: without them the cap is half as large
        const float rcap = rc.full2 ? g.rcap : g.rcap_simple;
        if (lane == 0) wu = WarpUni{ax, ay, az, beta, thr_p, hand_p, hz_p, xthr, rcap, kappa2, limb};
        __syncwarp();

        // Staged pairs: field f of records 2j, 2j+1 sits at buf1[(j * 26 + f) * 2 + {0,1}].  Fields: 0-2 mu, 3 tr Sigma,
        // 4-6 Sigma_xx,yy,zz, 7-9 2 Sigma_xy,xz,yz, 10 2 v.mu / |mu|^2, 11-13 w RGB, 14-16 m_R, 17-19 m_B,
        // 20 v.mu, 21 v Sigma v, 22-24 Sigma v (rough lobes only).
        const f2 NX = F2(nd.nx), NY = F2(nd.ny), NZ = F2(nd.nz), NV = F2(-nd.nv);
        const f2 Q0 = F2(nd.q0), Q1 = F2(nd.q1), Q2 = F2(nd.q2), Q3 = F2(0.5f * nd.q3), Q4 = F2(0.5f * nd.q4), Q5 = F2(0.5f * nd.q5);
        const f2 TRP = F2(nd.P0 + nd.P1 + nd.P2);
        auto eval1 = [&]() {
            const f2 CI = F2(rc.inv_a2m1), OMA = F2(rc.one_m_a2), A2 = F2(rc.alpha2);
            if (n1 & 1) {  // pad the last pair with a record of zero weight
                float* s = buf1 + ((n1 >> 1) * 26) * 2 + 1;
                if (lane < 26) s[lane * 2] = lane == 3 ? 1.f : 0.f;
                __syncwarp();
            }
            const int np = (n1 + 1) >> 1;
            f2 cR = F2(0.f), cG = F2(0.f), cB = F2(0.f);
            const float4* b4 = reinterpret_cast<const float4*>(buf1);
            if (!rc.full2) {
                for (int j = 0; j < np; ++j) {
                    const float4* s = b4 + j * PAIR4;
                    const float4 v0 = s[0], v1 = s[1];
                    const f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                    f2 u = fma2(ez, ez, fma2(ey, ey, fma2(ex, ex, hi(v1))));
                    f2 nmu = fma2(u, F2(-0.5f), F2(1.f));
                    if (pixcov) {  // the normal's spread over the cell also moves the mean of 2 - 2 n.h: + tr P (n.h)
                        u = fma2(TRP, nmu, u);
                        nmu = fma2(u, F2(-0.5f), F2(1.f));
                    }
                    const float4 v2 = s[2], v3 = s[3], v4 = s[4];
                    f2 nSn = mul2(Q0, lo(v2));
                    nSn = fma2(Q1, hi(v2), nSn); nSn = fma2(Q2, lo(v3), nSn);
                    nSn = fma2(Q3, hi(v3), nSn); nSn = fma2(Q4, lo(v4), nSn); nSn = fma2(Q5, hi(v4), nSn);
                    if (pixcov) {
                        const f2 mx = lo(v0), my = hi(v0), mz = lo(v1);
                        f2 pp = mul2(mul2(mx, mx), F2(nd.P0));
                        pp = fma2(mul2(my, my), F2(nd.P1), pp); pp = fma2(mul2(mz, mz), F2(nd.P2), pp);
                        pp = fma2(mul2(mx, my), F2(nd.P3), pp); pp = fma2(mul2(mx, mz), F2(nd.P4), pp);
                        pp = fma2(mul2(my, mz), F2(nd.P5), pp);
                        nSn = add2(nSn, pp);
                    }
                    const float4 v5 = s[5];
                    const f2 xm = max2(fma2(lo(v5), nmu, NV), 0.f);
                    const f2 sin2 = mul2(u, fma2(u, F2(-0.25f), F2(1.f)));
                    const f2 rq = rcp2(fma2(sin2, CI, F2(1.f)));
                    const f2 arg = fma2(mul2(xm, xm), OMA, A2);
                    const f2 sq = mul2(arg, rsqrt2(arg));
                    const f2 gg = mul2(xm, rcp2(add2(xm, sq)));
                    const f2 a = mul2(mul2(nmu, CI), rq);
                    const f2 Dg = mul2(mul2(rq, rq), gg);
                    const f2 t = fma2(mul2(a, F2(6.f)), a, mul2(rq, CI));
                    const f2 K = mul2(Dg, fma2(mul2(nSn, t), F2(2.f), F2(1.f)));
                    const f2 cn = mul2(mul2(Dg, a), F2(4.f));
                    const float4 v7 = s[7], v8 = s[8], v9 = s[9];
                    const f2 nmR = fma2(NZ, lo(v8), fma2(NY, hi(v7), mul2(NX, lo(v7))));
                    const f2 nmB = fma2(NZ, hi(v9), fma2(NY, lo(v9), mul2(NX, hi(v8))));
                    cR = fma2(cn, nmR, fma2(K, hi(v5), cR));
                    const float4 v6 = s[6];
                    cG = fma2(K, lo(v6), cG);
                    cG = fma2(cn, make_float2(-nmR.x - nmB.x, -nmR.y - nmB.y), cG);
                    cB = fma2(cn, nmB, fma2(K, hi(v6), cB));
                }
            } else {
                for (int j = 0; j < np; ++j) {
                    const float4* s = b4 + j * PAIR4;
                    const float4 v0 = s[0], v1 = s[1];
                    const f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                    f2 u = fma2(ez, ez, fma2(ey, ey, fma2(ex, ex, hi(v1))));
                    f2 nmu = fma2(u, F2(-0.5f), F2(1.f));
                    if (pixcov) {  // the normal's spread over the cell also moves the mean of 2 - 2 n.h: + tr P (n.h)
                        u = fma2(TRP, nmu, u);
                        nmu = fma2(u, F2(-0.5f), F2(1.f));
                    }
                    const float4 v2 = s[2], v3 = s[3], v4 = s[4];
                    f2 nSn = mul2(Q0, lo(v2));
                    nSn = fma2(Q1, hi(v2), nSn); nSn = fma2(Q2, lo(v3), nSn);
                    nSn = fma2(Q3, hi(v3), nSn); nSn = fma2(Q4, lo(v4), nSn); nSn = fma2(Q5, hi(v4), nSn);
                    f2 pS = nSn;
                    if (pixcov) {
                        const f2 mx = lo(v0), my = hi(v0), mz = lo(v1);
                        f2 pp = mul2(mul2(mx, mx), F2(nd.P0));
                        pp = fma2(mul2(my, my), F2(nd.P1), pp); pp = fma2(mul2(mz, mz), F2(nd.P2), pp);
                        pp = fma2(mul2(mx, my), F2(nd.P3), pp); pp = fma2(mul2(mx, mz), F2(nd.P4), pp);
                        pp = fma2(mul2(my, mz), F2(nd.P5), pp);
                        pS = add2(nSn, pp);
                    }
                    const float4 v10 = s[10], v11 = s[11], v12 = s[12];
                    const f2 vmu = lo(v10), vSv = hi(v10);
                    const f2 nSv = fma2(NZ, lo(v12), fma2(NY, hi(v11), mul2(NX, lo(v11))));
                    // mean and variance of n.d over the cell; the clamp at the horizon acts on that distribution
                    f2 x = fma2(mul2(vmu, F2(2.f)), nmu, fma2(nSv, F2(2.f), NV));
                    const f2 tnv = mul2(nmu, vmu);
                    f2 varx = mul2(mul2(nmu, nmu), vSv);
                    varx = fma2(mul2(tnv, F2(2.f)), nSv, varx);
                    varx = fma2(mul2(vmu, vmu), nSn, varx);
                    varx = mul2(max2(varx, 0.f), F2(4.f));
                    const f2 w = sqrt2(mul2(varx, F2(3.f)));
                    const bool st0 = x.x < w.x, st1 = x.y < w.y;
                    const f2 xe = max2(add2(x, w), 0.f);
                    const f2 xs2 = mul2(mul2(xe, xe), rcp2(max2(mul2(w, F2(4.f)), 1e-30f)));
                    x.x = st0 ? xs2.x : x.x;
                    x.y = st1 ? xs2.y : x.y;
                    const f2 xm = max2(x, 0.f);
                    const f2 sin2 = mul2(u, fma2(u, F2(-0.25f), F2(1.f)));
                    const f2 rq = rcp2(fma2(sin2, CI, F2(1.f)));
                    const f2 D = mul2(rq, rq);
                    const f2 arg = fma2(mul2(xm, xm), OMA, A2);
                    const f2 rsq = rsqrt2(arg);
                    const f2 sq = mul2(arg, rsq);
                    const f2 rxs = rcp2(add2(xm, sq));
                    const f2 gg = mul2(xm, rxs);
                    const f2 a = mul2(mul2(nmu, CI), rq);
                    const f2 Dg = mul2(D, gg);
                    const f2 t = fma2(mul2(a, F2(6.f)), a, mul2(rq, CI));
                    f2 K = mul2(Dg, fma2(mul2(pS, t), F2(2.f), F2(1.f)));
                    const f2 gx = mul2(mul2(A2, rsq), mul2(rxs, rxs));
                    const f2 spx = mul2(mul2(xm, OMA), rsq);
                    const f2 gxx = mul2(gx, fma2(spx, rsq, mul2(mul2(add2(spx, F2(1.f)), F2(2.f)), rxs)));  // = -g_xx
                    const f2 T2 = mul2(mul2(mul2(D, a), mul2(gx, F2(8.f))), fma2(nmu, nSv, mul2(vmu, nSn)));
                    f2 T3 = mul2(mul2(D, gxx), mul2(varx, F2(-0.5f)));
                    T3.x = st0 ? 0.f : T3.x;
                    T3.y = st1 ? 0.f : T3.y;
                    K = add2(K, add2(T2, T3));
                    const f2 cn = mul2(mul2(Dg, a), F2(4.f));
                    const float4 v5 = s[5], v7 = s[7], v8 = s[8], v9 = s[9];
                    const f2 nmR = fma2(NZ, lo(v8), fma2(NY, hi(v7), mul2(NX, lo(v7))));
                    const f2 nmB = fma2(NZ, hi(v9), fma2(NY, lo(v9), mul2(NX, hi(v8))));
                    cR = fma2(cn, nmR, fma2(K, hi(v5), cR));
                    const float4 v6 = s[6];
                    cG = fma2(K, lo(v6), cG);
                    cG = fma2(cn, make_float2(-nmR.x - nmB.x, -nmR.y - nmB.y), cG);
                    cB = fma2(cn, nmB, fma2(K, hi(v6), cB));
                }
            }
            a0 += nd.mult * (cR.x + cR.y);
            a1 += nd.mult * (cG.x + cG.y);
            a2 += nd.mult * (cB.x + cB.y);
            n1 = 0;
        };
        // Staged texels, two per iteration like the records: texels 2j, 2j+1 sit at buf0[4 j .. 4 j + 3] as
        // (hx0,hx1,hy0,hy1) (hz0,hz1,2vh0,2vh1) (wR0,wR1,wG0,wG1) (wB0,wB1,-,-).
        const f2 NVp = F2(nd.nv);
        auto eval0 = [&]() {
            const f2 CI = F2(rc.inv_a2m1), OMA = F2(rc.one_m_a2), A2 = F2(rc.alpha2);
            if (n0 & 1) {  // pad the last pair with a texel of zero weight
                float* s = reinterpret_cast<float*>(buf0 + (n0 >> 1) * 4) + 1;
                if (lane < 7) s[lane * 2] = lane < 3 ? (lane == 0 ? nd.nx : lane == 1 ? nd.ny : nd.nz) : 0.f;
                __syncwarp();
            }
            const int np = (n0 + 1) >> 1;
            f2 bR = F2(0.f), bG = F2(0.f), bB = F2(0.f);
#pragma unroll 2
            for (int j = 0; j < np; ++j) {
                const float4 v0 = buf0[4 * j], v1 = buf0[4 * j + 1], v2 = buf0[4 * j + 2], v3 = buf0[4 * j + 3];
                const f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                const f2 u2 = fma2(ez, ez, fma2(ey, ey, mul2(ex, ex)));  // 2 (1 - n.h), no cancellation
                const f2 nh = fma2(u2, F2(-0.5f), F2(1.f));
                const f2 xc = max2(sub2(mul2(hi(v1), nh), NVp), 0.f);   // n.d = |v+d| n.h - n.v
                const f2 sin2 = mul2(u2, fma2(u2, F2(-0.25f), F2(1.f)));
                const f2 q = fma2(sin2, CI, F2(1.f));
                const f2 sq = sqrt2(fma2(mul2(xc, xc), OMA, A2));
                const f2 ws = mul2(xc, rcp2(mul2(mul2(q, q), add2(xc, sq))));
                bR = fma2(ws, lo(v2), bR); bG = fma2(ws, hi(v2), bG); bB = fma2(ws, lo(v3), bB);
            }
            a0 += nd.mult * (bR.x + bR.y); a1 += nd.mult * (bG.x + bG.y); a2 += nd.mult * (bB.x + bB.y);
            n0 = 0;
        };

        bool done = false;
        while (true) {
            unsigned ent = 0;
            int ntake;
            if (sp > 0) {
                ntake = min(32, sp);
                if (lane < ntake) ent = (unsigned)stack[sp - 1 - lane];
                sp -= ntake;
            } else {
                if (p > 0 && in_pos >= in_n && in_next >= 0) {  // next chunk of the parent's list
                    const int* ch = g.pool_in + (size_t)in_next * CHUNK;
                    in_next = ch[0];
                    in_n = ch[1];
                    in_list = ch + 2;
                    in_pos = 0;
                }
                if (in_pos < in_n) {
                    ntake = min(32, in_n - in_pos);
                    if (lane < ntake) ent = p == 0 ? (((unsigned)g.gs.L << 28) | (unsigned)(in_pos + lane)) : (unsigned)in_list[in_pos + lane];
                    in_pos += ntake;
                } else {
                    ntake = 0;
                    done = true;  // one more turn of the loop flushes the staged records
                }
            }
            const bool has = lane < ntake;
            st_visits += ntake; st_iters += 1;
            __syncwarp();
            // ---- decide ----
            int act = ACT_DROP;
            const int lev = (int)(ent >> 28), id = (int)(ent & 0x0fffffffu);
            float h[3], vh = 0.f, w3[3];
            if (has) {
                float mx, my, mz, rha, wsum, vmu, im;
                if (lev > 0) {
                    // the verdict needs the mean, radius and energy; staging reads the rest of the record again
                    const float4* rp = pyr + (g.gs.off[lev] + id) * REC4;
                    const float4 r0 = rp[0], r2 = rp[2], r3 = rp[3];
                    mx = r0.x; my = r0.y; mz = r0.z;
                    wsum = r2.z + r2.w + r3.x;
                    const float m2 = fmaxf(mx * mx + my * my + mz * mz, 1e-30f);
                    im = fast_rsqrt(m2);
                    rha = fast_radius_angle(r0.w + fmaxf(1.f - m2 * im, 0.f));
                    vmu = rc.vhat[0] * mx + rc.vhat[1] * my + rc.vhat[2] * mz;
                } else {
                    const int r = id / g.We, c = id - r * g.We;
                    texel_spec(g, rc, env_b, r, c, h, vh, w3);
                    mx = h[0]; my = h[1]; mz = h[2];
                    wsum = w3[0] + w3[1] + w3[2];
                    im = 1.f; rha = 0.f; vmu = vh;
                }
                if (wsum > 0.f) {
                    const float ax = wu.ax, ay = wu.ay, az = wu.az, beta = wu.beta;
                    const float hx = mx * im - ax, hy = my * im - ay, hz = mz * im - az;
                    const float ang = fast_chord_angle(hx * hx + hy * hy + hz * hz);
                    const float dmin = fmaxf(ang - beta - rha, 0.f);
                    // direction of the cell d = 2 (v.h) h - v and its angular radius <= 2 rha: visibility, horizon
                    const float t2 = 2.f * vmu * im * im;
                    const float adc = ax * (t2 * mx - rc.vhat[0]) + ay * (t2 * my - rc.vhat[1]) + az * (t2 * mz - rc.vhat[2]);
                    const float spread = beta + 2.f * rha + 1e-3f;
                    const float ss = __sinf(fminf(spread, 1.5607f));
                    if (spread < 1.5607f && adc <= -ss) act = ACT_DROP;
                    // near for this lattice: small cells go to the child blocks, large ones are refined here so that
                    // their far parts stay on this lattice
                    else if (p < pk && dmin < wu.thr_p) act = (lev == 0 || rha <= wu.hand_p * wu.thr_p) ? ACT_HAND : ACT_REFINE;
                    // rim blocks: what lies within the shadowing ramp of their horizon goes down as well, in pieces of
                    // at most 0.05 rad
                    else if (p < pk && wu.limb && spread < 1.5607f &&
                             adc * __cosf(spread) - sqrtf(fmaxf(1.f - adc * adc, 0.f)) * ss < wu.xthr)
                        act = (lev == 0 || rha <= 0.05f) ? ACT_HAND : ACT_REFINE;
                    else if (lev > 0 && (rha > wu.rcap || rha * rha > wu.kappa2 * (rc.alpha2 + dmin * dmin) ||
                                         (2.f * rha > wu.hz_p && fabsf(adc) < ss))) act = ACT_REFINE;
                    else act = ACT_ACCEPT;
                }
            }
            // ---- hand over to the child blocks of the next pass ----
            {
                const unsigned mh = __ballot_sync(0xffffffffu, act == ACT_HAND);
                if (mh) {
                    const int cnt = __popc(mh);
                    if (out_cur < 0 || out_fill + cnt > CHUNK - 2) {  // close the current chunk, take a new one from the pool
                        int nc = 0;
                        if (lane == 0) nc = atomicAdd(g.pool_ctr, 1);
                        nc = __shfl_sync(0xffffffffu, nc, 0);
                        if (nc >= g.pool_cap) {
                            if (lane == 0) atomicOr(g.status, 1);  // pool exhausted: the result is incomplete
                            nc = -1;
                        }
                        if (lane == 0) {
                            if (out_cur >= 0) {
                                g.pool_out[(size_t)out_cur * CHUNK] = nc;
                                g.pool_out[(size_t)out_cur * CHUNK + 1] = out_fill;
                            }
                        }
                        if (out_cur < 0) out_head = nc;
                        out_cur = nc;
                        out_fill = 0;
                    }
                    if (act == ACT_HAND && out_cur >= 0)
                        g.pool_out[(size_t)out_cur * CHUNK + 2 + out_fill + __popc(mh & ((1u << lane) - 1u))] = (int)ent;
                    if (out_cur >= 0) out_fill += cnt;
                    out_n += cnt;
                }
            }
            // ---- refine: children onto the stack ----
            {
                int nch = 0, cr = 0, cc = 0, Wc = 0;
                if (act == ACT_REFINE) {
                    const int Wl = g.gs.W[lev];
                    const int r = id / Wl, c = id - r * Wl;
                    Wc = lev == 1 ? g.We : g.gs.W[lev - 1];
                    const int Hc = lev == 1 ? g.He : g.gs.H[lev - 1];
                    cr = 2 * r; cc = 2 * c;
                    nch = (cr + 1 < Hc ? 2 : 1) * (cc + 1 < Wc ? 2 : 1);
                }
                int inc = nch;
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += t;
                }
                const int total = __shfl_sync(0xffffffffu, inc, 31);
                if (total) {
                    if (sp + total > STACK_CAP) {
                        atomicOr(g.status, 4);  // traversal stack full
                    } else if (nch) {
                        int pos = sp + inc - nch;
                        const int two_c = (nch == 4) || (nch == 2 && cc + 1 < Wc);
                        const int two_r = (nch == 4) || (nch == 2 && !two_c);
                        const int tag = (int)((unsigned)(lev - 1) << 28);
                        stack[pos++] = tag | (cr * Wc + cc);
                        if (two_c) stack[pos++] = tag | (cr * Wc + cc + 1);
                        if (two_r) stack[pos++] = tag | ((cr + 1) * Wc + cc);
                        if (two_r && two_c) stack[pos++] = tag | ((cr + 1) * Wc + cc + 1);
                    }
                    if (sp + total <= STACK_CAP) sp += total;
                    sp_max = max(sp_max, sp);
                }
            }
            // ---- accept: stage the record for the evaluation ----
            {
                const unsigned m1 = __ballot_sync(0xffffffffu, act == ACT_ACCEPT && lev > 0);
                const unsigned m0 = __ballot_sync(0xffffffffu, act == ACT_ACCEPT && lev == 0);
                if (done || n1 + __popc(m1) > BUF1) { __syncwarp(); eval1(); __syncwarp(); }
                if (done || n0 + __popc(m0) > BUF0) { __syncwarp(); eval0(); __syncwarp(); }
                if (done) break;
                if (act == ACT_ACCEPT) {
                    if (lev > 0) {
                        const int slot = n1 + __popc(m1 & ((1u << lane) - 1u));
                        float* s = buf1 + ((slot >> 1) * 26) * 2 + (slot & 1);
                        const float4* rp = pyr + (g.gs.off[lev] + id) * REC4;
                        const float4 r0 = rp[0], r1 = rp[1], r2 = rp[2], r3 = rp[3], r4 = rp[4];
                        const float Sxx = r1.x, Syy = r1.y, Szz = r1.z, Sxy = r1.w, Sxz = r2.x, Syz = r2.y;
                        const float vx = rc.vhat[0], vy = rc.vhat[1], vz = rc.vhat[2];
                        const float vmu = vx * r0.x + vy * r0.y + vz * r0.z;
                        const float trS = Sxx + Syy + Szz;
                        const float svx = Sxx * vx + Sxy * vy + Sxz * vz, svy = Sxy * vx + Syy * vy + Syz * vz,
                                    svz = Sxz * vx + Syz * vy + Szz * vz;
                        s[0] = r0.x; s[2] = r0.y; s[4] = r0.z; s[6] = trS;
                        s[8] = Sxx; s[10] = Syy; s[12] = Szz; s[14] = 2.f * Sxy; s[16] = 2.f * Sxz; s[18] = 2.f * Syz;
                        s[20] = 2.f * vmu / fmaxf(1.f - trS, 1e-12f);
                        s[22] = r2.z; s[24] = r2.w; s[26] = r3.x;
                        s[28] = r3.y; s[30] = r3.z; s[32] = r3.w;
                        s[34] = r4.x; s[36] = r4.y; s[38] = r4.z;
                        s[40] = vmu; s[42] = vx * svx + vy * svy + vz * svz;
                        s[44] = svx; s[46] = svy; s[48] = svz; s[50] = 0.f;
                    } else {
                        const int slot = n0 + __popc(m0 & ((1u << lane) - 1u));
                        float* s = reinterpret_cast<float*>(buf0 + (slot >> 1) * 4) + (slot & 1);
                        s[0] = h[0]; s[2] = h[1]; s[4] = h[2]; s[6] = 2.f * vh;
                        s[8] = w3[0]; s[10] = w3[1]; s[12] = w3[2];
                    }
                }
                n1 += __popc(m1);
                n0 += __popc(m0);
                st_acc1 += __popc(m1); st_acc0 += __popc(m0);
            }
            __syncwarp();
        }
        if (p < pk && lane == 0) {
            const int nbI = (NG + 3) / 4;
            if (out_cur >= 0) {
                g.pool_out[(size_t)out_cur * CHUNK] = -1;
                g.pool_out[(size_t)out_cur * CHUNK + 1] = out_fill;
            }
            g.heads_out[(size_t)k * nbI * nbJ + (size_t)bI * nbJ + bJ] = out_head;
        }
        if (lane == 0 && g.stats) {
            atomicAdd(g.status + 16 + 4 * p, st_visits); atomicAdd(g.status + 17 + 4 * p, st_iters);
            atomicAdd(g.status + 18 + 4 * p, st_acc0); atomicAdd(g.status + 19 + 4 * p, st_acc1);
        }
        if (lane == 0) {  // high-water marks (drm_render_status)
            if (sp_max > g.status[1]) atomicMax(g.status + 1, sp_max);
            if (out_n > g.status[2 + p]) atomicMax(g.status + 2 + p, out_n);
        }
    } else if (p < pk && lane == 0) {
        const int nbJ = (NG + 7) / 8, nbI = (NG + 3) / 4;
        const int bI = I0 >> 2, bJ = J0 >> 3;
        if (bI < nbI && bJ < nbJ) g.heads_out[(size_t)k * nbI * nbJ + (size_t)bI * nbJ + bJ] = -1;
    }
    tile_sync();  // stacks and buffers are dead: the reduction reuses the memory
    tile_writeback(g, p, red, k, ti, tj, a0, a1, a2, false);
    tile_sync();  // ... and the next item's traversal reuses it again
    }
    if (stats && lane == 0) {
        atomicAdd(g.status + STAT_TILE_WAIT + p, (int)(t_wait >> 10));
        atomicAdd(g.status + STAT_WARP_CYCLES + p, (int)((clock64() - t_warp) >> 10));
    }
}

template <int P>
__global__ void __launch_bounds__(TREE_THREADS, SPEC_MINB[P]) tree_spec_pass_kernel(const TreeArgs g) {
    tree_spec_pass<P, float>(g, threadIdx.x);
}
template <int P>
__global__ void __launch_bounds__(TREE_THREADS, SPEC_MINB[P]) tree_spec_pass_kernel_h(const TreeArgs g) {
    tree_spec_pass<P, __half>(g, threadIdx.x);
}

// ---- specular lobe, pass P: the default instances ------------------------------------------------------------------
// tree_spec_pass with evaluation loops that issue fewer packed FP32 instructions (eval0, eval1; DESIGN.md 5).
// Traversal, decisions and staging are those of tree_spec_pass apart from constant factors folded into staged fields
// (-v.h per texel; 2 m_c, 2 v.mu, 4 v Sigma v, 4 Sigma v per record); the sums are the same, re-rounded.
// tree_spec_pass stays as it is, selected by DrmRenderOptions::spec_kernels = 1.

template <int P, typename T>
__device__ __forceinline__ void tree_spec_pass2(const TreeArgs g, int tid) {
    extern __shared__ __align__(16) unsigned char tree_smem[];
    const int lane = tid & 31, warp = tid >> 5;
    int* stack = reinterpret_cast<int*>(tree_smem) + warp * STACK_CAP;
    float* buf1 = reinterpret_cast<float*>(tree_smem + TREE_WARPS * STACK_CAP * 4) + warp * (BUF1 / 2 * PAIR4 * 4);
    float4* buf0 = reinterpret_cast<float4*>(tree_smem + TREE_WARPS * STACK_CAP * 4 + TREE_WARPS * (BUF1 / 2) * PAIR4 * 16) + warp * (BUF0 * 2);
    float* red = reinterpret_cast<float*>(tree_smem);  // reused after the traversal: [256][3]

    constexpr int p = P;
    const int NG = g.res << p;
    const int tiles_x = (NG + 15) / 16;
    const int n_items = g.nact[p] * tiles_x * tiles_x;
    // barriers of the item loop; under collect_stats they also count the cycles the warp waits in them
    const bool stats = g.stats;
    long long t_warp = stats ? clock64() : 0, t_wait = 0;
    auto tile_sync = [&]() {
        const long long t = stats ? clock64() : 0;
        __syncthreads();
        if (stats) t_wait += clock64() - t;
    };
    // persistent CTAs: items = (active render, tile of 16 x 16 lattice nodes), tile-major so that the renders interleave,
    // handed out by a counter in the order of tile_of (the rim tiles take several times longer than the others)
    // the item's render record is read from shared memory where it is used: one copy per CTA instead of 34 registers
    __shared__ int next_item, next_k;
    __shared__ TreeConst rc;
    __shared__ WarpUni wu_s[TREE_WARPS];
    __shared__ int wst_s[TREE_WARPS][6];
    WarpUni& wu = wu_s[warp];
    while (true) {
    if (warp == 0) {
        int it = 0;
        if (lane == 0) it = atomicAdd(g.item_ctr, 1);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it < n_items) {
            const int kk = g.act[p * TREE_CHUNK + it % g.nact[p]];
            const int* src = reinterpret_cast<const int*>(g.rc + kk);
            int* dst = reinterpret_cast<int*>(&rc);
            for (int i = lane; i < (int)(sizeof(TreeConst) / 4); i += 32) dst[i] = src[i];
            if (lane == 0) next_k = kk;
        }
        if (lane == 0) next_item = it;
    }
    tile_sync();
    const int item = next_item;
    if (item >= n_items) break;
    const int k = next_k;
    const int tile = item / g.nact[p];
    const int pk = rc.pk;
    int ti, tj;
    tile_of(tile, tiles_x, ti, tj);
    const int I0 = ti * 16 + (warp >> 1) * 4, J0 = tj * 16 + (warp & 1) * 8;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    const bool pixcov = g.pixcov && p == 0 && pk > 0;  // the 1x1 node of a finer footprint carries the cell's covariance

    NodeT nd;
    make_node(g, rc, p, pixcov, I0 + (lane >> 3), J0 + (lane & 7), true, nd);
    float ax, ay, az, beta;
    const bool live = rc.has_spec && warp_cone(g, p, nd, ax, ay, az, beta);

    if (live) {
        const float4* pyr = g.pyr_s + (size_t)k * g.gs.cells * REC4;
        const T* env_b = reinterpret_cast<const T*>(g.env) + (size_t)rc.env * g.He * g.We * 3;
        // input: the top level of the pyramid (pass 0) or the parent block's hand-over list
        const int nbJ = (NG + 7) / 8;
        const int bI = I0 >> 2, bJ = J0 >> 3;
        const int* in_list = nullptr;  // entries of the current chunk
        int in_n, in_pos = 0, in_next = -1;
        if constexpr (p == 0) {
            in_n = g.gs.H[g.gs.L] * g.gs.W[g.gs.L];
        } else {
            const int nbJp = ((g.res << (p - 1)) + 7) / 8;
            const int nbIp = ((g.res << (p - 1)) + 3) / 4;
            const size_t pb = (size_t)k * nbIp * nbJp + (size_t)(bI >> 1) * nbJp + (bJ >> 1);
            in_next = g.heads_in[pb];
            in_n = 0;
        }
        int out_cur = -1, out_fill = 0, out_head = -1;
        int sp = 0, n1 = 0, n0 = 0;
        // collect_stats counters [0..3] and the high-water marks of the stack [4] and of the hand-over list [5] in the
        // warp's shared slot, not in registers through the traversal (lane 0 keeps them)
        int* st = wst_s[warp];
        if (lane == 0) st[0] = st[1] = st[2] = st[3] = st[4] = st[5] = 0;
        // at the limb (n.v -> 0) the lobe sits on the horizon of the normal and the cell average converges later
        const float nv_min = -warp_max(nd.active ? -nd.nv : -1.f);
        // ... and n.d = 2 (v.h)(n.h) - n.v moves by the cell's own spread of n.v, so where n.v comes within a few alpha of
        // zero the view factor and the shadowing ramp G1(n.d) vary across the cell however far the half vector is: blocks
        // that touch this rim (the outermost cells of the refmap for a sharp lobe) accept nothing that comes near on the
        // coarse lattices: it all goes down to the render's own lattice.
        // (a lattice whose sub-cells are narrower than limb_sub * alpha resolves that ramp: no rim rule on it)
        const float subw = g.cell / (float)(1 << p);
        const bool limb = nv_min < fmaxf(g.limb_nv, fminf(g.limb_x * sqrtf(rc.alpha2), g.limb_cells * g.cell)) &&
                          subw * subw > g.limb_sub * g.limb_sub * rc.alpha2;
        const float thr_p = rc.thr[p] * (limb ? g.limb_boost : 1.f);
        const float hand_p = limb ? g.limb_hand : g.hand;
        // the horizon ramp matters most where the lobe itself sits on it: n.v within a few lobe widths of zero
        const float hz_p = (limb || nv_min < g.hz_nv * sqrtf(rc.alpha2)) ? (p == pk && rc.full2 ? g.hz_fin : g.hz) : g.hz_in;
        const float xthr = g.limb_ramp * sqrtf(rc.alpha2);
        const float kappa2 = g.kappa * g.kappa;
        // wide cells need the second-order terms of G1(n.d) whatever the lobe: without them the cap is half as large
        const float rcap = rc.full2 ? g.rcap : g.rcap_simple;
        if (lane == 0) wu = WarpUni{ax, ay, az, beta, thr_p, hand_p, hz_p, xthr, rcap, kappa2, limb};
        __syncwarp();

        // Staged pairs as in tree_spec_pass, except fields 14-19: 2 m_R, 2 m_B; 20: 2 v.mu; 21: 4 v Sigma v;
        // 22-24: 4 Sigma v.
        const f2 NX = F2(nd.nx), NY = F2(nd.ny), NZ = F2(nd.nz), NV = F2(-nd.nv);
        const f2 Q0 = F2(nd.q0), Q1 = F2(nd.q1), Q2 = F2(nd.q2), Q3 = F2(0.5f * nd.q3), Q4 = F2(0.5f * nd.q4), Q5 = F2(0.5f * nd.q5);
        const f2 TRP = F2(nd.P0 + nd.P1 + nd.P2);
        // The loops below evaluate the sums of tree_spec_pass in the same order.  Their cost is the FP32 pipe, where a
        // packed FFMA2 / FMUL2 / FADD2 takes the cycles of two scalar instructions, so they save packed instructions
        // and leave the clamps to FMNMX (integer/ALU pipe) and reciprocals and square roots to MUFU:
        //  * q = 1 + CI sin^2 = 1 + CI u (1 - u/4) as fma(u, fma(u, -CI/4, CI), 1);
        //  * sq as one sqrt, not arg * rsqrt(arg); the sharp lobe's D G1-ratio as rq^2 xm / (xm + sq);
        //  * constant factors 2 and 4 folded into staged fields and into 2 a, 2 CI.
        // The results differ from tree_spec_pass by rounding only.
        auto eval1 = [&]() {
            const float ci = rc.inv_a2m1;
            const f2 CI = F2(ci), CQ = F2(-0.25f * ci), CI2 = F2(2.f * ci), OMA = F2(rc.one_m_a2), A2 = F2(rc.alpha2);
            if (n1 & 1) {  // pad the last pair with a record of zero weight
                float* s = buf1 + ((n1 >> 1) * 26) * 2 + 1;
                if (lane < 26) s[lane * 2] = lane == 3 ? 1.f : 0.f;
                __syncwarp();
            }
            const int np = (n1 + 1) >> 1;
            f2 cR = F2(0.f), cG = F2(0.f), cB = F2(0.f);
            const float4* b4 = reinterpret_cast<const float4*>(buf1);
            if (!rc.full2) {
                for (int j = 0; j < np; ++j) {
                    const float4* s = b4 + j * PAIR4;
                    const float4 v0 = s[0], v1 = s[1];
                    const f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                    f2 u = fma2(ez, ez, fma2(ey, ey, fma2(ex, ex, hi(v1))));
                    f2 nmu = fma2(u, F2(-0.5f), F2(1.f));
                    if (pixcov) {  // the normal's spread over the cell also moves the mean of 2 - 2 n.h: + tr P (n.h)
                        u = fma2(TRP, nmu, u);
                        nmu = fma2(u, F2(-0.5f), F2(1.f));
                    }
                    const float4 v2 = s[2], v3 = s[3], v4 = s[4];
                    f2 nSn = mul2(Q0, lo(v2));
                    nSn = fma2(Q1, hi(v2), nSn); nSn = fma2(Q2, lo(v3), nSn);
                    nSn = fma2(Q3, hi(v3), nSn); nSn = fma2(Q4, lo(v4), nSn); nSn = fma2(Q5, hi(v4), nSn);
                    if (pixcov) {
                        const f2 mx = lo(v0), my = hi(v0), mz = lo(v1);
                        f2 pp = mul2(mul2(mx, mx), F2(nd.P0));
                        pp = fma2(mul2(my, my), F2(nd.P1), pp); pp = fma2(mul2(mz, mz), F2(nd.P2), pp);
                        pp = fma2(mul2(mx, my), F2(nd.P3), pp); pp = fma2(mul2(mx, mz), F2(nd.P4), pp);
                        pp = fma2(mul2(my, mz), F2(nd.P5), pp);
                        nSn = add2(nSn, pp);
                    }
                    const float4 v5 = s[5];
                    f2 x = fma2(lo(v5), nmu, NV);
                    x = max2(x, 0.f);
                    const f2 q = fma2(u, fma2(u, CQ, CI), F2(1.f));
                    const f2 xs = add2(x, sqrt2(fma2(mul2(x, x), OMA, A2)));
                    const f2 rq = rcp2(q);
                    const f2 Dg = mul2(mul2(rq, rq), mul2(x, rcp2(xs)));
                    const f2 ciq = mul2(rq, CI2);
                    const f2 a = mul2(nmu, ciq);                              // 2 a
                    const f2 K = mul2(Dg, fma2(nSn, fma2(mul2(a, a), F2(3.f), ciq), F2(1.f)));  // Dg (1 + 2 nSn t)
                    const f2 cn = mul2(Dg, a);
                    const float4 v6 = s[6], v7 = s[7], v8 = s[8], v9 = s[9];
                    const f2 nmR = fma2(NZ, lo(v8), fma2(NY, hi(v7), mul2(NX, lo(v7))));
                    const f2 nmB = fma2(NZ, hi(v9), fma2(NY, lo(v9), mul2(NX, hi(v8))));
                    cR = fma2(cn, nmR, fma2(K, hi(v5), cR));
                    cG = fma2(cn, make_float2(-nmR.x - nmB.x, -nmR.y - nmB.y), fma2(K, lo(v6), cG));
                    cB = fma2(cn, nmB, fma2(K, hi(v6), cB));
                }
            } else {
                for (int j = 0; j < np; ++j) {
                    const float4* s = b4 + j * PAIR4;
                    const float4 v0 = s[0], v1 = s[1];
                    const f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                    f2 u = fma2(ez, ez, fma2(ey, ey, fma2(ex, ex, hi(v1))));
                    f2 nmu = fma2(u, F2(-0.5f), F2(1.f));
                    if (pixcov) {  // the normal's spread over the cell also moves the mean of 2 - 2 n.h: + tr P (n.h)
                        u = fma2(TRP, nmu, u);
                        nmu = fma2(u, F2(-0.5f), F2(1.f));
                    }
                    const float4 v2 = s[2], v3 = s[3], v4 = s[4];
                    f2 nSn = mul2(Q0, lo(v2));
                    nSn = fma2(Q1, hi(v2), nSn); nSn = fma2(Q2, lo(v3), nSn);
                    nSn = fma2(Q3, hi(v3), nSn); nSn = fma2(Q4, lo(v4), nSn); nSn = fma2(Q5, hi(v4), nSn);
                    f2 pS = nSn;
                    if (pixcov) {
                        const f2 mx = lo(v0), my = hi(v0), mz = lo(v1);
                        f2 pp = mul2(mul2(mx, mx), F2(nd.P0));
                        pp = fma2(mul2(my, my), F2(nd.P1), pp); pp = fma2(mul2(mz, mz), F2(nd.P2), pp);
                        pp = fma2(mul2(mx, my), F2(nd.P3), pp); pp = fma2(mul2(mx, mz), F2(nd.P4), pp);
                        pp = fma2(mul2(my, mz), F2(nd.P5), pp);
                        pS = add2(nSn, pp);
                    }
                    const float4 v10 = s[10], v11 = s[11], v12 = s[12];
                    const f2 vmu = lo(v10), vSv = hi(v10);                   // 2 v.mu, 4 v Sigma v
                    const f2 nSv = fma2(NZ, lo(v12), fma2(NY, hi(v11), mul2(NX, lo(v11))));  // 4 n Sigma v
                    // mean and variance of n.d over the cell; the clamp at the horizon acts on that distribution
                    f2 x = fma2(vmu, nmu, fma2(nSv, F2(0.5f), NV));
                    const f2 vn = mul2(vmu, nSn);
                    f2 varx = mul2(mul2(nmu, nmu), vSv);
                    varx = fma2(mul2(nmu, vmu), nSv, varx);
                    varx = max2(fma2(vmu, vn, varx), 0.f);                   // 4 var(n.d)
                    const f2 w = sqrt2(mul2(varx, F2(3.f)));
                    const bool st0 = x.x < w.x, st1 = x.y < w.y;
                    const f2 xe = max2(add2(x, w), 0.f);
                    const f2 xs2 = mul2(mul2(xe, xe), rcp2(max2(mul2(w, F2(4.f)), 1e-30f)));
                    x.x = st0 ? xs2.x : x.x;
                    x.y = st1 ? xs2.y : x.y;
                    const f2 xm = max2(x, 0.f);
                    const f2 q = fma2(u, fma2(u, CQ, CI), F2(1.f));
                    const f2 rq = rcp2(q);
                    const f2 D = mul2(rq, rq);
                    const f2 arg = fma2(mul2(xm, xm), OMA, A2);
                    const f2 rsq = rsqrt2(arg);
                    const f2 sq = mul2(arg, rsq);
                    const f2 rxs = rcp2(add2(xm, sq));
                    const f2 ciq = mul2(rq, CI2);                             // 2 CI rq
                    const f2 a = mul2(nmu, ciq);                              // 2 a
                    const f2 Dg = mul2(D, mul2(xm, rxs));
                    f2 K = mul2(Dg, fma2(pS, fma2(mul2(a, a), F2(3.f), ciq), F2(1.f)));
                    const f2 gx = mul2(mul2(A2, rsq), mul2(rxs, rxs));
                    const f2 spx = mul2(mul2(xm, OMA), rsq);
                    const f2 gxx = mul2(gx, fma2(spx, rsq, mul2(mul2(add2(spx, F2(1.f)), F2(2.f)), rxs)));  // = -g_xx
                    const f2 T2 = mul2(mul2(mul2(D, a), gx), fma2(vn, F2(2.f), mul2(nmu, nSv)));
                    f2 T3 = mul2(mul2(D, gxx), mul2(varx, F2(-0.5f)));
                    T3.x = st0 ? 0.f : T3.x;
                    T3.y = st1 ? 0.f : T3.y;
                    K = add2(K, add2(T2, T3));
                    const f2 cn = mul2(Dg, a);
                    const float4 v5 = s[5], v6 = s[6], v7 = s[7], v8 = s[8], v9 = s[9];
                    const f2 nmR = fma2(NZ, lo(v8), fma2(NY, hi(v7), mul2(NX, lo(v7))));
                    const f2 nmB = fma2(NZ, hi(v9), fma2(NY, lo(v9), mul2(NX, hi(v8))));
                    cR = fma2(cn, nmR, fma2(K, hi(v5), cR));
                    cG = fma2(cn, make_float2(-nmR.x - nmB.x, -nmR.y - nmB.y), fma2(K, lo(v6), cG));
                    cB = fma2(cn, nmB, fma2(K, hi(v6), cB));
                }
            }
            a0 += nd.mult * (cR.x + cR.y);
            a1 += nd.mult * (cG.x + cG.y);
            a2 += nd.mult * (cB.x + cB.y);
            n1 = 0;
        };
        // Staged texels, two per float4 pair like the records: texels 2j, 2j+1 sit at buf0[4 j .. 4 j + 3] as
        // (hx0,hx1,hy0,hy1) (hz0,hz1,2vh0,2vh1) (wR0,wR1,wG0,wG1) (wB0,wB1,-vh0,-vh1); -v.h turns n.d into one FMA.
        // The loop takes four texels (two pairs A, B) an iteration.
        const f2 NVp = F2(nd.nv);
        auto eval0 = [&]() {
            const float ci = rc.inv_a2m1;
            const f2 CI = F2(ci), CQ = F2(-0.25f * ci), OMA = F2(rc.one_m_a2), A2 = F2(rc.alpha2);
            if (n0 & 3) {  // pad to whole quads with texels of zero weight at the node itself
                const int slot = n0 + (lane >> 3), f = lane & 7;
                if (slot < ((n0 + 3) & ~3)) {
                    float* s = reinterpret_cast<float*>(buf0 + (slot >> 1) * 4) + (slot & 1);
                    s[f * 2] = f == 0 ? nd.nx : f == 1 ? nd.ny : f == 2 ? nd.nz : 0.f;
                }
                __syncwarp();
            }
            const int nq = (n0 + 3) >> 2;
            f2 bR = F2(0.f), bG = F2(0.f), bB = F2(0.f);
            for (int j = 0; j < nq; ++j) {
                const float4* s = buf0 + 8 * j;
                const float4 v0 = s[0], v1 = s[1], v3 = s[3];
                f2 ex = sub2(NX, lo(v0)), ey = sub2(NY, hi(v0)), ez = sub2(NZ, lo(v1));
                const f2 uA = fma2(ez, ez, fma2(ey, ey, mul2(ex, ex)));   // 2 (1 - n.h), no cancellation
                f2 xA = sub2(fma2(uA, hi(v3), hi(v1)), NVp);               // n.d = |v+d| (1 - u/2) - n.v
                xA = max2(xA, 0.f);
                const f2 qA = fma2(uA, fma2(uA, CQ, CI), F2(1.f));
                const f2 dA = mul2(mul2(qA, qA), add2(xA, sqrt2(fma2(mul2(xA, xA), OMA, A2))));
                const float4 w0 = s[4], w1 = s[5], w3 = s[7];
                ex = sub2(NX, lo(w0)); ey = sub2(NY, hi(w0)); ez = sub2(NZ, lo(w1));
                const f2 uB = fma2(ez, ez, fma2(ey, ey, mul2(ex, ex)));
                f2 xB = sub2(fma2(uB, hi(w3), hi(w1)), NVp);
                xB = max2(xB, 0.f);
                const f2 qB = fma2(uB, fma2(uB, CQ, CI), F2(1.f));
                const f2 dB = mul2(mul2(qB, qB), add2(xB, sqrt2(fma2(mul2(xB, xB), OMA, A2))));
                const f2 wsA = mul2(xA, rcp2(dA)), wsB = mul2(xB, rcp2(dB));
                const float4 v2 = s[2], w2 = s[6];
                bR = fma2(wsA, lo(v2), bR); bG = fma2(wsA, hi(v2), bG); bB = fma2(wsA, lo(v3), bB);
                bR = fma2(wsB, lo(w2), bR); bG = fma2(wsB, hi(w2), bG); bB = fma2(wsB, lo(w3), bB);
            }
            a0 += nd.mult * (bR.x + bR.y); a1 += nd.mult * (bG.x + bG.y); a2 += nd.mult * (bB.x + bB.y);
            n0 = 0;
        };

        bool done = false;
        while (true) {
            unsigned ent = 0;
            int ntake;
            if (sp > 0) {
                ntake = min(32, sp);
                if (lane < ntake) ent = (unsigned)stack[sp - 1 - lane];
                sp -= ntake;
            } else {
                if (p > 0 && in_pos >= in_n && in_next >= 0) {  // next chunk of the parent's list
                    const int* ch = g.pool_in + (size_t)in_next * CHUNK;
                    in_next = ch[0];
                    in_n = ch[1];
                    in_list = ch + 2;
                    in_pos = 0;
                }
                if (in_pos < in_n) {
                    ntake = min(32, in_n - in_pos);
                    if (lane < ntake) ent = p == 0 ? (((unsigned)g.gs.L << 28) | (unsigned)(in_pos + lane)) : (unsigned)in_list[in_pos + lane];
                    in_pos += ntake;
                } else {
                    ntake = 0;
                    done = true;  // one more turn of the loop flushes the staged records
                }
            }
            const bool has = lane < ntake;
            if (stats && lane == 0) { st[0] += ntake; st[1] += 1; }
            __syncwarp();
            // ---- decide ----
            int act = ACT_DROP;
            const int lev = (int)(ent >> 28), id = (int)(ent & 0x0fffffffu);
            float h[3], vh = 0.f, w3[3];
            if (has) {
                float mx, my, mz, rha, wsum, vmu, im;
                if (lev > 0) {
                    // the verdict needs the mean, radius and energy; staging reads the rest of the record again
                    const float4* rp = pyr + (g.gs.off[lev] + id) * REC4;
                    const float4 r0 = rp[0], r2 = rp[2], r3 = rp[3];
                    mx = r0.x; my = r0.y; mz = r0.z;
                    wsum = r2.z + r2.w + r3.x;
                    const float m2 = fmaxf(mx * mx + my * my + mz * mz, 1e-30f);
                    im = fast_rsqrt(m2);
                    rha = fast_radius_angle(r0.w + fmaxf(1.f - m2 * im, 0.f));
                    vmu = rc.vhat[0] * mx + rc.vhat[1] * my + rc.vhat[2] * mz;
                } else {
                    const int r = id / g.We, c = id - r * g.We;
                    texel_spec(g, rc, env_b, r, c, h, vh, w3);
                    mx = h[0]; my = h[1]; mz = h[2];
                    wsum = w3[0] + w3[1] + w3[2];
                    im = 1.f; rha = 0.f; vmu = vh;
                }
                if (wsum > 0.f) {
                    const float ax = wu.ax, ay = wu.ay, az = wu.az, beta = wu.beta;
                    const float hx = mx * im - ax, hy = my * im - ay, hz = mz * im - az;
                    const float ang = fast_chord_angle(hx * hx + hy * hy + hz * hz);
                    const float dmin = fmaxf(ang - beta - rha, 0.f);
                    // direction of the cell d = 2 (v.h) h - v and its angular radius <= 2 rha: visibility, horizon
                    const float t2 = 2.f * vmu * im * im;
                    const float adc = ax * (t2 * mx - rc.vhat[0]) + ay * (t2 * my - rc.vhat[1]) + az * (t2 * mz - rc.vhat[2]);
                    const float spread = beta + 2.f * rha + 1e-3f;
                    const float ss = __sinf(fminf(spread, 1.5607f));
                    if (spread < 1.5607f && adc <= -ss) act = ACT_DROP;
                    // near for this lattice: small cells go to the child blocks, large ones are refined here so that
                    // their far parts stay on this lattice
                    else if (p < pk && dmin < wu.thr_p) act = (lev == 0 || rha <= wu.hand_p * wu.thr_p) ? ACT_HAND : ACT_REFINE;
                    // rim blocks: what lies within the shadowing ramp of their horizon goes down as well, in pieces of
                    // at most 0.05 rad
                    else if (p < pk && wu.limb && spread < 1.5607f &&
                             adc * __cosf(spread) - sqrtf(fmaxf(1.f - adc * adc, 0.f)) * ss < wu.xthr)
                        act = (lev == 0 || rha <= 0.05f) ? ACT_HAND : ACT_REFINE;
                    else if (lev > 0 && (rha > wu.rcap || rha * rha > wu.kappa2 * (rc.alpha2 + dmin * dmin) ||
                                         (2.f * rha > wu.hz_p && fabsf(adc) < ss))) act = ACT_REFINE;
                    else act = ACT_ACCEPT;
                }
            }
            // ---- hand over to the child blocks of the next pass ----
            {
                const unsigned mh = __ballot_sync(0xffffffffu, act == ACT_HAND);
                if (mh) {
                    const int cnt = __popc(mh);
                    if (out_cur < 0 || out_fill + cnt > CHUNK - 2) {  // close the current chunk, take a new one from the pool
                        int nc = 0;
                        if (lane == 0) nc = atomicAdd(g.pool_ctr, 1);
                        nc = __shfl_sync(0xffffffffu, nc, 0);
                        if (nc >= g.pool_cap) {
                            if (lane == 0) atomicOr(g.status, 1);  // pool exhausted: the result is incomplete
                            nc = -1;
                        }
                        if (lane == 0) {
                            if (out_cur >= 0) {
                                g.pool_out[(size_t)out_cur * CHUNK] = nc;
                                g.pool_out[(size_t)out_cur * CHUNK + 1] = out_fill;
                            }
                        }
                        if (out_cur < 0) out_head = nc;
                        out_cur = nc;
                        out_fill = 0;
                    }
                    if (act == ACT_HAND && out_cur >= 0)
                        g.pool_out[(size_t)out_cur * CHUNK + 2 + out_fill + __popc(mh & ((1u << lane) - 1u))] = (int)ent;
                    if (out_cur >= 0) out_fill += cnt;
                    if (lane == 0) st[5] += cnt;
                }
            }
            // ---- refine: children onto the stack ----
            {
                int nch = 0, cr = 0, cc = 0, Wc = 0;
                if (act == ACT_REFINE) {
                    const int Wl = g.gs.W[lev];
                    const int r = id / Wl, c = id - r * Wl;
                    Wc = lev == 1 ? g.We : g.gs.W[lev - 1];
                    const int Hc = lev == 1 ? g.He : g.gs.H[lev - 1];
                    cr = 2 * r; cc = 2 * c;
                    nch = (cr + 1 < Hc ? 2 : 1) * (cc + 1 < Wc ? 2 : 1);
                }
                int inc = nch;
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += t;
                }
                const int total = __shfl_sync(0xffffffffu, inc, 31);
                if (total) {
                    if (sp + total > STACK_CAP) {
                        atomicOr(g.status, 4);  // traversal stack full
                    } else if (nch) {
                        int pos = sp + inc - nch;
                        const int two_c = (nch == 4) || (nch == 2 && cc + 1 < Wc);
                        const int two_r = (nch == 4) || (nch == 2 && !two_c);
                        const int tag = (int)((unsigned)(lev - 1) << 28);
                        stack[pos++] = tag | (cr * Wc + cc);
                        if (two_c) stack[pos++] = tag | (cr * Wc + cc + 1);
                        if (two_r) stack[pos++] = tag | ((cr + 1) * Wc + cc);
                        if (two_r && two_c) stack[pos++] = tag | ((cr + 1) * Wc + cc + 1);
                    }
                    if (sp + total <= STACK_CAP) sp += total;
                    if (lane == 0) st[4] = max(st[4], sp);
                }
            }
            // ---- accept: stage the record for the evaluation ----
            {
                const unsigned m1 = __ballot_sync(0xffffffffu, act == ACT_ACCEPT && lev > 0);
                const unsigned m0 = __ballot_sync(0xffffffffu, act == ACT_ACCEPT && lev == 0);
                if (done || n1 + __popc(m1) > BUF1) { __syncwarp(); eval1(); __syncwarp(); }
                if (done || n0 + __popc(m0) > BUF0) { __syncwarp(); eval0(); __syncwarp(); }
                if (done) break;
                if (act == ACT_ACCEPT) {
                    if (lev > 0) {
                        const int slot = n1 + __popc(m1 & ((1u << lane) - 1u));
                        float* s = buf1 + ((slot >> 1) * 26) * 2 + (slot & 1);
                        const float4* rp = pyr + (g.gs.off[lev] + id) * REC4;
                        const float4 r0 = rp[0], r1 = rp[1], r2 = rp[2], r3 = rp[3], r4 = rp[4];
                        const float Sxx = r1.x, Syy = r1.y, Szz = r1.z, Sxy = r1.w, Sxz = r2.x, Syz = r2.y;
                        const float vx = rc.vhat[0], vy = rc.vhat[1], vz = rc.vhat[2];
                        const float vmu = vx * r0.x + vy * r0.y + vz * r0.z;
                        const float trS = Sxx + Syy + Szz;
                        const float svx = Sxx * vx + Sxy * vy + Sxz * vz, svy = Sxy * vx + Syy * vy + Syz * vz,
                                    svz = Sxz * vx + Syz * vy + Szz * vz;
                        s[0] = r0.x; s[2] = r0.y; s[4] = r0.z; s[6] = trS;
                        s[8] = Sxx; s[10] = Syy; s[12] = Szz; s[14] = 2.f * Sxy; s[16] = 2.f * Sxz; s[18] = 2.f * Syz;
                        s[20] = 2.f * vmu / fmaxf(1.f - trS, 1e-12f);
                        s[22] = r2.z; s[24] = r2.w; s[26] = r3.x;
                        s[28] = 2.f * r3.y; s[30] = 2.f * r3.z; s[32] = 2.f * r3.w;
                        s[34] = 2.f * r4.x; s[36] = 2.f * r4.y; s[38] = 2.f * r4.z;
                        s[40] = 2.f * vmu; s[42] = 4.f * (vx * svx + vy * svy + vz * svz);
                        s[44] = 4.f * svx; s[46] = 4.f * svy; s[48] = 4.f * svz; s[50] = 0.f;
                    } else {
                        const int slot = n0 + __popc(m0 & ((1u << lane) - 1u));
                        float* s = reinterpret_cast<float*>(buf0 + (slot >> 1) * 4) + (slot & 1);
                        s[0] = h[0]; s[2] = h[1]; s[4] = h[2]; s[6] = 2.f * vh;
                        s[8] = w3[0]; s[10] = w3[1]; s[12] = w3[2]; s[14] = -vh;
                    }
                }
                n1 += __popc(m1);
                n0 += __popc(m0);
                if (stats && lane == 0) { st[2] += __popc(m0); st[3] += __popc(m1); }
            }
            __syncwarp();
        }
        if (p < pk && lane == 0) {
            const int nbI = (NG + 3) / 4;
            if (out_cur >= 0) {
                g.pool_out[(size_t)out_cur * CHUNK] = -1;
                g.pool_out[(size_t)out_cur * CHUNK + 1] = out_fill;
            }
            g.heads_out[(size_t)k * nbI * nbJ + (size_t)bI * nbJ + bJ] = out_head;
        }
        if (lane == 0 && g.stats) {
            atomicAdd(g.status + 16 + 4 * p, st[0]); atomicAdd(g.status + 17 + 4 * p, st[1]);
            atomicAdd(g.status + 18 + 4 * p, st[2]); atomicAdd(g.status + 19 + 4 * p, st[3]);
        }
        if (lane == 0) {  // high-water marks (drm_render_status)
            if (st[4] > g.status[1]) atomicMax(g.status + 1, st[4]);
            if (st[5] > g.status[2 + p]) atomicMax(g.status + 2 + p, st[5]);
        }
    } else if (p < pk && lane == 0) {
        const int nbJ = (NG + 7) / 8, nbI = (NG + 3) / 4;
        const int bI = I0 >> 2, bJ = J0 >> 3;
        if (bI < nbI && bJ < nbJ) g.heads_out[(size_t)k * nbI * nbJ + (size_t)bI * nbJ + bJ] = -1;
    }
    tile_sync();  // stacks and buffers are dead: the reduction reuses the memory
    tile_writeback(g, p, red, k, ti, tj, a0, a1, a2, false);
    tile_sync();  // ... and the next item's traversal reuses it again
    }
    if (stats && lane == 0) {
        atomicAdd(g.status + STAT_TILE_WAIT + p, (int)(t_wait >> 10));
        atomicAdd(g.status + STAT_WARP_CYCLES + p, (int)((clock64() - t_warp) >> 10));
    }
}

template <int P>
__global__ void __launch_bounds__(TREE_THREADS, SPEC_MINB[P]) tree_spec_pass2_kernel(const TreeArgs g) {
    tree_spec_pass2<P, float>(g, threadIdx.x);
}
template <int P>
__global__ void __launch_bounds__(TREE_THREADS, SPEC_MINB[P]) tree_spec_pass2_kernel_h(const TreeArgs g) {
    tree_spec_pass2<P, __half>(g, threadIdx.x);
}

// ---- diffuse lobe: one pass, writes `out`.  1x1 lattice whose node carries the covariance of the refmap cell (fourth
// order in the cell size: cells up to 0.03 rad), or the render's own lattice for coarser refmaps ------------------------
template <typename T>
__device__ __forceinline__ void tree_diff(const TreeArgs& g, int tid) {
    extern __shared__ __align__(16) unsigned char tree_smem[];
    const int lane = tid & 31, warp = tid >> 5;
    int* stack = reinterpret_cast<int*>(tree_smem) + warp * STACK_CAP;
    float4* buf1 = reinterpret_cast<float4*>(tree_smem + TREE_WARPS * STACK_CAP * 4) + warp * (BUF1 * SREC4);
    float* red = reinterpret_cast<float*>(tree_smem);

    const int k = blockIdx.y;
    const TreeConst rc = g.rc[k];
    const int p = g.diff_cov ? 0 : rc.pk;  // the grid is sized for the finest lattice of the call
    const bool pixcov = g.diff_cov && rc.pk > 0;
    const int tiles_x = ((g.res << p) + 15) / 16;
    if ((int)blockIdx.x >= tiles_x * tiles_x) return;
    const int ti = blockIdx.x / tiles_x, tj = blockIdx.x - ti * tiles_x;
    const int I0 = ti * 16 + (warp >> 1) * 4, J0 = tj * 16 + (warp & 1) * 8;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    NodeT nd;
    make_node(g, rc, p, pixcov, I0 + (lane >> 3), J0 + (lane & 7), false, nd);
    float ax, ay, az, beta;
    const bool live = rc.has_diff && warp_cone(g, p, nd, ax, ay, az, beta);
    if (live) {
        const float4* pyr = g.pyr_d + (size_t)rc.env * g.gd.cells * REC4;
        const T* env_b = reinterpret_cast<const T*>(g.env) + (size_t)rc.env * g.He * g.We * 3;
        const int in_n = g.gd.H[g.gd.L] * g.gd.W[g.gd.L];
        int in_pos = 0, sp = 0, n1 = 0;
        const float vx = rc.vhat[0], vy = rc.vhat[1], vz = rc.vhat[2];
        const float Fi = nd.Fi, r = rc.rough;
        // K = x [ A + B y + Fo (C + D y + E y^2) ],  x = n.d, y = 1 + v.d, Fo = (1-x)^5  (DESIGN.md 5)
        const float A = 1.f - 0.5f * Fi, Bc = r * Fi, Cc = -0.5f * (1.f - 0.5f * Fi), Dc = r * (1.f - Fi), Ec = r * r * Fi;
        auto eval = [&]() {
            for (int i = 0; i < n1; ++i) {
                const float4* s = buf1 + i * SREC4;
                const float4 s0 = s[0], s1 = s[1], s2 = s[2], s3 = s[3], s4 = s[4], s5 = s[5], s6 = s[6];
                float x = nd.nx * s0.x + nd.ny * s0.y + nd.nz * s0.z;
                float nSn = nd.q0 * s1.x + nd.q1 * s1.y + nd.q2 * s1.z + nd.q3 * s2.x + nd.q4 * s2.y + nd.q5 * s2.z;
                if (pixcov)
                    nSn += s0.x * s0.x * nd.P0 + s0.y * s0.y * nd.P1 + s0.z * s0.z * nd.P2 + s0.x * s0.y * nd.P3 +
                           s0.x * s0.z * nd.P4 + s0.y * s0.z * nd.P5;
                const float w = fast_sqrt(3.f * fmaxf(nSn, 0.f));
                const bool straddle = x < w;
                const float xe = fmaxf(x + w, 0.f);
                x = straddle ? (w > 0.f ? xe * xe * fast_rcp(4.f * w) : 0.f) : x;
                x = fmaxf(x, 0.f);
                const float y = s0.w;
                const float mm = fmaxf(1.f - x, 0.f);
                const float m2 = mm * mm, m4 = m2 * m2, Fo = m4 * mm;
                const float gq = Cc + y * (Dc + Ec * y);
                const float lin = A + Bc * y + Fo * gq;
                const float gy = Dc + 2.f * Ec * y;
                const float Fo1 = -5.f * m4, Fo2 = 20.f * m2 * mm;
                const float Kx = lin + x * Fo1 * gq;
                const float Ky = x * (Bc + Fo * gy);
                const float Kxx = straddle ? 0.f : (2.f * Fo1 + x * Fo2) * gq;
                const float Kxy = Bc + Fo * gy + x * Fo1 * gy;
                const float Kyy = x * Fo * 2.f * Ec;
                const float nSv = nd.nx * s4.x + nd.ny * s4.y + nd.nz * s4.z;
                const float K = x * lin + 0.5f * (Kxx * nSn + 2.f * Kxy * nSv + Kyy * s2.w);
                const float nmR = nd.nx * s5.x + nd.ny * s5.y + nd.nz * s5.z, nmB = nd.nx * s6.x + nd.ny * s6.y + nd.nz * s6.z;
                const float gR = Kx * nmR + Ky * s5.w, gB = Kx * nmB + Ky * s6.w;
                const float vis = x > 0.f ? 1.f : 0.f;
                a0 += vis * (K * s3.x + gR);
                a1 += vis * (K * s3.y - (gR + gB));
                a2 += vis * (K * s3.z + gB);
            }
            n1 = 0;
        };
        while (true) {
            unsigned ent = 0;
            int ntake;
            if (sp > 0) {
                ntake = min(32, sp);
                if (lane < ntake) ent = (unsigned)stack[sp - 1 - lane];
                sp -= ntake;
            } else if (in_pos < in_n) {
                ntake = min(32, in_n - in_pos);
                if (lane < ntake) ent = ((unsigned)g.gd.L << 28) | (unsigned)(in_pos + lane);
                in_pos += ntake;
            } else {
                break;
            }
            const bool has = lane < ntake;
            __syncwarp();
            int act = ACT_DROP;
            const int lev = (int)(ent >> 28), id = (int)(ent & 0x0fffffffu);
            float4 r0 = make_float4(0.f, 0.f, 0.f, 0.f), r1 = r0, r2 = r0, r3 = r0, r4 = r0;
            if (has) {
                if (lev > 0) {
                    const float4* rp = pyr + (g.gd.off[lev] + id) * REC4;
                    r0 = rp[0]; r1 = rp[1]; r2 = rp[2]; r3 = rp[3]; r4 = rp[4];
                } else {
                    float d[3], w3[3];
                    const int rr = id / g.We, cc = id - rr * g.We;
                    texel_diff(g, env_b, rr, cc, d, w3);
                    r0 = make_float4(d[0], d[1], d[2], 0.f);
                    r2.z = w3[0]; r2.w = w3[1]; r3.x = w3[2];
                }
                const float wsum = r2.z + r2.w + r3.x;
                if (wsum > 0.f) {
                    const float m2 = r0.x * r0.x + r0.y * r0.y + r0.z * r0.z;
                    const float sm = sqrtf(m2);
                    const float rda = chord_angle((r0.w + (1.f - sm)) * (r0.w + (1.f - sm)));
                    const float adc = (ax * r0.x + ay * r0.y + az * r0.z) / fmaxf(sm, 1e-20f);
                    const float spread = beta + rda + 1e-3f;
                    const float ss = sinf(fminf(spread, 1.5607f));
                    if (spread < 1.5607f && adc <= -ss) act = ACT_DROP;
                    else if (lev > g.gd.base && (rda > g.kappa_d || (rda > g.hz_d && fabsf(adc) < ss))) act = ACT_REFINE;
                    else act = ACT_ACCEPT;
                }
            }
            {
                int nch = 0, cr = 0, cc = 0, Wc = 0;
                if (act == ACT_REFINE) {
                    const int Wl = g.gd.W[lev];
                    const int rr = id / Wl, c = id - rr * Wl;
                    Wc = lev == 1 ? g.We : g.gd.W[lev - 1];
                    const int Hc = lev == 1 ? g.He : g.gd.H[lev - 1];
                    cr = 2 * rr; cc = 2 * c;
                    nch = (cr + 1 < Hc ? 2 : 1) * (cc + 1 < Wc ? 2 : 1);
                }
                int inc = nch;
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += t;
                }
                const int total = __shfl_sync(0xffffffffu, inc, 31);
                if (total) {
                    if (sp + total > STACK_CAP) {
                        atomicOr(g.status, 1);
                    } else if (nch) {
                        int pos = sp + inc - nch;
                        const int two_c = (nch == 4) || (nch == 2 && cc + 1 < Wc);
                        const int two_r = (nch == 4) || (nch == 2 && !two_c);
                        const int tag = (int)((unsigned)(lev - 1) << 28);
                        stack[pos++] = tag | (cr * Wc + cc);
                        if (two_c) stack[pos++] = tag | (cr * Wc + cc + 1);
                        if (two_r) stack[pos++] = tag | ((cr + 1) * Wc + cc);
                        if (two_r && two_c) stack[pos++] = tag | ((cr + 1) * Wc + cc + 1);
                    }
                    if (sp + total <= STACK_CAP) sp += total;
                }
            }
            {
                const unsigned m1 = __ballot_sync(0xffffffffu, act == ACT_ACCEPT);
                if (n1 + __popc(m1) > BUF1) { __syncwarp(); eval(); __syncwarp(); }
                if (act == ACT_ACCEPT) {
                    float4* s = buf1 + (n1 + __popc(m1 & ((1u << lane) - 1u))) * SREC4;
                    const float Sxx = r1.x, Syy = r1.y, Szz = r1.z, Sxy = r1.w, Sxz = r2.x, Syz = r2.y;
                    const float svx = Sxx * vx + Sxy * vy + Sxz * vz, svy = Sxy * vx + Syy * vy + Syz * vz,
                                svz = Sxz * vx + Syz * vy + Szz * vz;
                    s[0] = make_float4(r0.x, r0.y, r0.z, 1.f + vx * r0.x + vy * r0.y + vz * r0.z);
                    s[1] = make_float4(Sxx, Syy, Szz, 0.f);
                    s[2] = make_float4(Sxy, Sxz, Syz, vx * svx + vy * svy + vz * svz);
                    s[3] = make_float4(r2.z, r2.w, r3.x, 0.f);
                    s[4] = make_float4(svx, svy, svz, 0.f);
                    s[5] = make_float4(r3.y, r3.z, r3.w, vx * r3.y + vy * r3.z + vz * r3.w);
                    s[6] = make_float4(r4.x, r4.y, r4.z, vx * r4.x + vy * r4.y + vz * r4.z);
                }
                n1 += __popc(m1);
            }
            __syncwarp();
        }
        __syncwarp();
        eval();
        const float wn = nd.nv > 0.f ? nd.wq : 0.f;
        a0 *= wn * rc.cdiff[0]; a1 *= wn * rc.cdiff[1]; a2 *= wn * rc.cdiff[2];
    }
    __syncthreads();
    tile_writeback(g, p, red, k, ti, tj, a0, a1, a2, true);
}

__global__ void __launch_bounds__(TREE_THREADS, DIFF_MINB) tree_diff_kernel(const TreeArgs g) {
    tree_diff<float>(g, threadIdx.x);
}
__global__ void __launch_bounds__(TREE_THREADS, DIFF_MINB) tree_diff_kernel_h(const TreeArgs g) {
    tree_diff<__half>(g, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
static void make_geom(PyrGeom& G, int He, int We, int want_base) {
    memset(&G, 0, sizeof(G));
    G.H[0] = He; G.W[0] = We;
    int l = 0;
    while ((long)G.H[l] * G.W[l] > 256 && l + 1 < MAX_PYR) {
        G.H[l + 1] = (G.H[l] + 1) / 2;
        G.W[l + 1] = (G.W[l] + 1) / 2;
        ++l;
    }
    G.L = l;
    G.base = want_base < l ? want_base : l;
    long off = 0;
    for (int i = 1; i <= l; ++i) {
        G.off[i] = off;
        if (i >= G.base) off += (long)G.H[i] * G.W[i];
        else G.off[i] = -1;
    }
    G.cells = off > 0 ? off : 1;
}

static void gauss_legendre_t(int S, float* x, float* w) {
    for (int i = 0; i < S; ++i) {
        double z = cos(M_PI * (i + 0.75) / (S + 0.5)), pp = 1.0;
        for (int it = 0; it < 100; ++it) {
            double p1 = 1.0, p2 = 0.0;
            for (int j = 0; j < S; ++j) {
                const double p3 = p2;
                p2 = p1;
                p1 = ((2.0 * j + 1.0) * z * p2 - j * p3) / (j + 1.0);
            }
            pp = S * (z * p1 - p2) / (z * z - 1.0);
            const double dz = p1 / pp;
            z -= dz;
            if (fabs(dz) < 1e-15) break;
        }
        x[S - 1 - i] = (float)z;
        w[S - 1 - i] = (float)(1.0 / ((1.0 - z * z) * pp * pp));  // = w_i / 2: the weights sum to 1
    }
}

struct TreeLayout {
    PyrGeom gs, gd;
    int pk;
    size_t nblocks[TREE_MAX_P];
    int pool_cap[2];
    int* status;
    int* env_used;
    int* act;
    int* nact;
    TreeConst* rc;
    float *sin_t, *cos_t, *sin_p, *cos_p;
    float4 *pyr_s, *pyr_d;
    int* pool[2];
    int* heads[2];
};

static int log2_exact(int S) {
    for (int p = 0; p <= TREE_MAX_P; ++p)
        if ((1 << p) == S) return p;
    return -1;
}

// the diffuse pyramid of an He x We envmap: the lobe reads no cell wider than ~0.03 rad, so the stored levels start at
// level 3 at 1000 rows, level 1 at 250 rows
static void make_diffuse_geom(PyrGeom& G, int He, int We) {
    int dbase = 0;
    while ((2 << dbase) * M_PI / He <= 0.03) ++dbase;
    make_geom(G, He, We, dbase);
}

// S: 1, 2, 4, 8, 16 = that footprint for every render; 0 = per render (given, or chosen on the device): sized for 16.
// prepared: the diffuse pyramids come from the caller (drm_render_refmaps_prepared), so neither they nor the mask of
// the envmaps in use take workspace.
static size_t tree_layout(TreeLayout& L, void* ws, int N, int B, int He, int We, int res, int S, bool prepared = false) {
    make_geom(L.gs, He, We, 1);
    make_diffuse_geom(L.gd, He, We);
    L.pk = S > 0 ? log2_exact(S) : TREE_MAX_P;
    const int NC = N < TREE_CHUNK ? N : TREE_CHUNK;
    Carver c(ws);
    L.status = c.take<int>(64);
    L.rc = c.take<TreeConst>(N);
    L.env_used = prepared ? nullptr : c.take<int>(B);
    L.act = c.take<int>((TREE_MAX_P + 1) * TREE_CHUNK);
    L.nact = c.take<int>(16);
    L.sin_t = c.take<float>(He);
    L.cos_t = c.take<float>(He);
    L.sin_p = c.take<float>(We);
    L.cos_p = c.take<float>(We);
    L.pyr_s = c.take<float4>((size_t)NC * L.gs.cells * REC4);
    L.pyr_d = prepared ? nullptr : c.take<float4>((size_t)B * L.gd.cells * REC4);
    // hand-over lists: pass p writes nblocks[p] chains that pass p + 1 reads; two pools alternate, sized for the average
    // list (the longest ones, at the limb, reach ~3000 entries) with a factor 3 of slack
    size_t need[2] = {1, 1}, needh[2] = {1, 1};
    for (int p = 0; p < L.pk; ++p) {
        const size_t NG = (size_t)res << p;
        L.nblocks[p] = ((NG + 3) / 4) * ((NG + 7) / 8);
        // measured chunks per block (worst render of the test set): pass 0: 44 (a wide lobe forced onto a fine lattice
        // hands most of the map down), 1: 8, 2: 3.7, 3: 1.3; the longest single list was 26 chunks
        static const size_t budget[TREE_MAX_P] = {64, 24, 10, 6};
        const size_t per_block = budget[p];
        const size_t n = (size_t)NC * L.nblocks[p] * per_block + 64;
        if (n > need[p & 1]) need[p & 1] = n;
        if ((size_t)NC * L.nblocks[p] > needh[p & 1]) needh[p & 1] = (size_t)NC * L.nblocks[p];
    }
    for (int i = 0; i < 2; ++i) {
        L.pool_cap[i] = (int)(need[i] < 0x7fffffff / CHUNK ? need[i] : 0x7fffffff / CHUNK);
        L.pool[i] = c.take<int>((size_t)L.pool_cap[i] * CHUNK);
        L.heads[i] = c.take<int>(needh[i]);
    }
    return c.used();
}

// Buffer of drm_env_pyramid_build: the diffuse pyramids [B][gd.cells][REC4] at offset 0 (where the render reads them),
// then the build's scratch: the direction tables of the texel rows and columns and the mask of the slots to build.
struct EnvPyrLayout {
    PyrGeom gd;
    float4* pyr;
    float *sin_t, *cos_t, *sin_p, *cos_p;
    int* used;
};

static size_t env_pyr_layout(EnvPyrLayout& L, void* buf, int B, int He, int We) {
    make_diffuse_geom(L.gd, He, We);
    Carver c(buf);
    L.pyr = c.take<float4>((size_t)B * L.gd.cells * REC4);
    L.sin_t = c.take<float>(He);
    L.cos_t = c.take<float>(He);
    L.sin_p = c.take<float>(We);
    L.cos_p = c.take<float>(We);
    L.used = c.take<int>(B);
    return c.used();
}

static bool env_sizes_ok(int B, int He, int We) {
    return B > 0 && B <= 65535 && He > 0 && We > 0 && (long)He * We < (1L << 28);
}

static constexpr size_t TREE_SMEM = (size_t)TREE_WARPS * STACK_CAP * 4 + (size_t)TREE_WARPS * (BUF1 / 2) * PAIR4 * 16 +
                                    (size_t)TREE_WARPS * BUF0 * 2 * 16;
static_assert(BUF1 * SREC4 <= (BUF1 / 2) * PAIR4 + 8 * BUF0, "the diffuse pass stages its records in the same region");

static constexpr int MAX_DEVICES = 64;

// The kernels that read envmap texels, per texel type: fp32 (the kernels above) or fp16 (their _h twins).
template <typename T> struct TexelKernels;
template <> struct TexelKernels<float> {
    template <int P> static constexpr void (*spec)(TreeArgs) = tree_spec_pass_kernel<P>;
    template <int P> static constexpr void (*spec2)(TreeArgs) = tree_spec_pass2_kernel<P>;
    static constexpr void (*diff)(TreeArgs) = tree_diff_kernel;
    template <bool SPEC> static constexpr void (*pyr)(TreeArgs, int, float4*) = pyr_from_texels_kernel<SPEC>;
};
template <> struct TexelKernels<__half> {
    template <int P> static constexpr void (*spec)(TreeArgs) = tree_spec_pass_kernel_h<P>;
    template <int P> static constexpr void (*spec2)(TreeArgs) = tree_spec_pass2_kernel_h<P>;
    static constexpr void (*diff)(TreeArgs) = tree_diff_kernel_h;
    template <bool SPEC> static constexpr void (*pyr)(TreeArgs, int, float4*) = pyr_from_texels_kernel_h<SPEC>;
};

// the diffuse pyramids of the envmaps with g.env_used set (blockIdx.y = envmap; the others exit at once).  g needs env,
// the direction tables, gd, He, We and domega_k.  Returns the kernels launched.
template <typename T>
static int launch_diffuse_pyramids(const TreeArgs& g, int B, float4* pyr, cudaStream_t st) {
    if (g.gd.L < 1) return 0;
    const int tb = 128;
    const int first = g.gd.base > 0 ? g.gd.base : 1;  // base 0: texels are read directly, level 1 is the first stored
    const int nb = g.gd.H[first] * g.gd.W[first];
    int launches = 0;
    TexelKernels<T>::template pyr<false><<<dim3((nb + tb - 1) / tb, B), tb, 0, st>>>(g, first, pyr);
    ++launches;
    for (int l = first + 1; l <= g.gd.L; ++l) {
        const int nl = g.gd.H[l] * g.gd.W[l];
        pyr_merge_kernel<<<dim3((nl + tb - 1) / tb, B), tb, 0, st>>>(g.gd, l, pyr, g.env_used);
        ++launches;
    }
    return launches;
}

// Pass P on a persistent grid of (SMs x resident CTAs of this instance), at most one CTA per item.  The grid size is
// queried once per device and instance (fp32 and fp16, default and pinned instances have their own slots).
template <int P, typename T, bool PINNED>
static cudaError_t launch_spec_pass(const TreeArgs& a, long items, cudaStream_t st) {
    static int resident[MAX_DEVICES];
    void (*kernel)(TreeArgs) = PINNED ? TexelKernels<T>::template spec<P> : TexelKernels<T>::template spec2<P>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_SMEM);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    int dev = 0;
    if (e == cudaSuccess) e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int per_sm = 0, sms = 0;
    int* slot = dev < MAX_DEVICES ? &resident[dev] : &per_sm;
    if (*slot == 0) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TREE_THREADS, TREE_SMEM);
        if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        *slot = max(per_sm, 1) * sms;
    }
    const int grid = (int)(items < *slot ? items : *slot);
    kernel<<<grid, TREE_THREADS, TREE_SMEM, st>>>(a);
    return cudaGetLastError();
}

}  // namespace drm

using namespace drm;

extern "C" size_t drm_render_workspace_bytes(int N, int B, int He, int We, int res, int S) {
    if (N <= 0 || B <= 0 || He <= 0 || We <= 0 || res <= 0 || (S != 0 && log2_exact(S) < 0)) return 0;
    if ((long)He * We >= (1L << 28)) return 0;
    TreeLayout L;
    return tree_layout(L, nullptr, N, B, He, We, res, S);
}

extern "C" size_t drm_render_prepared_workspace_bytes(int N, int B, int He, int We, int res, int S) {
    if (N <= 0 || B <= 0 || He <= 0 || We <= 0 || res <= 0 || (S != 0 && log2_exact(S) < 0)) return 0;
    if ((long)He * We >= (1L << 28)) return 0;
    TreeLayout L;
    return tree_layout(L, nullptr, N, B, He, We, res, S, true);
}

extern "C" size_t drm_env_pyramid_bytes(int B, int He, int We) {
    if (!env_sizes_ok(B, He, We)) return 0;
    EnvPyrLayout P;
    return env_pyr_layout(P, nullptr, B, He, We);
}

template <typename T>
static int env_pyramid_build(const T* env, int B, int He, int We, const int32_t* ids, int n_ids, void* pyramids,
                             size_t pyramid_bytes, cudaStream_t st) {
    EnvPyrLayout P;
    const size_t need = env_pyr_layout(P, pyramids, B, He, We);
    DRM_REQUIRE(pyramid_bytes >= need, "env_pyramid_build: pyramid buffer of %zu bytes needed for B=%d He=%d We=%d, %zu given",
                need, B, He, We, pyramid_bytes);
    if (ids && n_ids == 0) return DRM_OK;
    TreeArgs g;
    memset(&g, 0, sizeof(g));
    g.env = reinterpret_cast<const float*>(env); g.sin_t = P.sin_t; g.cos_t = P.cos_t; g.sin_p = P.sin_p; g.cos_p = P.cos_p;
    g.env_used = P.used; g.gd = P.gd;
    g.B = B; g.He = He; g.We = We;
    g.domega_k = (float)((2.0 * M_PI / We) * (M_PI / He));
    const int tb = 128;
    tree_tables_kernel<<<(max(He, We) + tb - 1) / tb, tb, 0, st>>>(P.sin_t, P.cos_t, P.sin_p, P.cos_p, He, We);
    if (ids) DRM_CHECK_CUDA(cudaMemsetAsync(P.used, 0, sizeof(int) * B, st));
    const int nmark = ids ? n_ids : B;
    env_mark_slots_kernel<<<(nmark + tb - 1) / tb, tb, 0, st>>>(ids, n_ids, B, P.used);
    count_launches(2 + launch_diffuse_pyramids<T>(g, B, P.pyr, st));
    DRM_CHECK_CUDA(cudaGetLastError());
    return DRM_OK;
}

extern "C" int drm_env_pyramid_build(const void* env, int env_half, int B, int He, int We, const int32_t* ids, int n_ids,
                                     void* pyramids, size_t pyramid_bytes, void* cuda_stream) {
    DRM_REQUIRE(env && pyramids, "env_pyramid_build: null pointer");
    DRM_REQUIRE(env_sizes_ok(B, He, We), "env_pyramid_build: B=%d He=%d We=%d: sizes must be positive, B <= 65535 and "
                "He * We < 2^28", B, He, We);
    DRM_REQUIRE(!ids || n_ids >= 0, "env_pyramid_build: n_ids=%d must not be negative", n_ids);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    if (env_half)
        return env_pyramid_build(static_cast<const __half*>(env), B, He, We, ids, n_ids, pyramids, pyramid_bytes, st);
    return env_pyramid_build(static_cast<const float*>(env), B, He, We, ids, n_ids, pyramids, pyramid_bytes, st);
}

extern "C" int drm_render_status(const void* workspace, int* status_host, void* cuda_stream) {
    DRM_REQUIRE(workspace && status_host, "render_status: null pointer");
    DRM_CHECK_CUDA(cudaMemcpyAsync(status_host, workspace, 40 * sizeof(int), cudaMemcpyDeviceToHost,
                                   static_cast<cudaStream_t>(cuda_stream)));
    return DRM_OK;
}

// drm_render_refmaps_opts (T = float) and drm_render_refmaps_half (T = __half): only the kernels that read texels differ.
// prepared (drm_render_refmaps_prepared): the diffuse pyramids of the B envmaps are `pyramids`, built by
// drm_env_pyramid_build; the call neither marks nor builds any.
template <typename T>
static int render_refmaps(const T* env, int B, int He, int We, const int32_t* env_index, const float* z6,
                          const float* view3, const uint8_t* flip, int N, int res, int S, float alpha_min,
                          int channel_first, float* out, void* workspace, size_t workspace_bytes, void* cuda_stream,
                          const DrmRenderOptions* opts, bool prepared = false, const void* pyramids = nullptr,
                          size_t pyramid_bytes = 0) {
    DRM_REQUIRE(env && z6 && view3 && out, "render: null pointer");
    DRM_REQUIRE(!prepared || pyramids, "render: null pointer (pyramids)");
    DRM_REQUIRE(N > 0 && B > 0 && He > 0 && We > 0 && res > 0, "render: N=%d B=%d He=%d We=%d res=%d must be positive", N, B, He, We, res);
    DRM_REQUIRE(S == 0 || log2_exact(S) >= 0, "render: footprint_S=%d must be 0 (per render) or 1, 2, 4, 8, 16", S);
    DRM_REQUIRE(res <= 4096, "render: res=%d too large", res);
    DRM_REQUIRE(B <= 65535, "render: at most 65535 envmaps per call (B=%d)", B);
    DRM_REQUIRE((long)He * We < (1L << 28), "render: envmap of %d x %d texels is too large", He, We);
    if (prepared) {
        EnvPyrLayout P;
        const size_t pneed = env_pyr_layout(P, nullptr, B, He, We);
        DRM_REQUIRE(pyramid_bytes >= pneed, "render: pyramid buffer of %zu bytes needed for B=%d He=%d We=%d, %zu given",
                    pneed, B, He, We, pyramid_bytes);
    }
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    DrmRenderOptions o;
    drm_render_default_options(&o);
    if (opts) o = *opts;
    const int32_t* S_per_render = o.footprint_per_render;
    const int S_layout = S_per_render ? 0 : S;
    TreeLayout L;
    const size_t need = tree_layout(L, workspace, N, B, He, We, res, S_layout, prepared);
    if (prepared) L.pyr_d = static_cast<float4*>(const_cast<void*>(pyramids));
    if (!workspace || workspace_bytes < need) {
        set_error("render: workspace of %zu bytes needed, %zu given", need, workspace_bytes);
        return DRM_EWORKSPACE;
    }
    if (!(alpha_min > 0.f)) alpha_min = fmaxf(1e-3f, (float)(1.25 * M_PI / He));
    DRM_REQUIRE(o.spec_kernels == 0 || o.spec_kernels == 1, "render: spec_kernels=%d must be 0 or 1", o.spec_kernels);
    const bool pinned = o.spec_kernels == 1;

    TreeArgs g;
    memset(&g, 0, sizeof(g));
    g.env = reinterpret_cast<const float*>(env); g.sin_t = L.sin_t; g.cos_t = L.cos_t; g.sin_p = L.sin_p; g.cos_p = L.cos_p;
    g.pyr_s = L.pyr_s; g.pyr_d = L.pyr_d; g.status = L.status; g.env_used = L.env_used; g.act = L.act; g.nact = L.nact;
    g.gs = L.gs; g.gd = L.gd;
    g.B = B; g.He = He; g.We = We; g.res = res; g.pk = L.pk; g.channel_first = channel_first;
    g.cell = (float)(M_PI / res);
    g.domega_k = (float)((2.0 * M_PI / We) * (M_PI / He));
    g.kappa = o.kappa; g.rcap = o.rcap; g.rcap_simple = o.rcap_simple; g.hz = o.horizon; g.hz_in = fmaxf(o.horizon, o.horizon_inner * fminf(1.f, powf((float)(M_PI / 128.0) / g.cell, 0.25f))); g.hz_nv = o.horizon_inner_nv; g.hz_fin = fmaxf(o.horizon, o.horizon_finest * fminf(1.f, powf((float)(M_PI / 128.0) / g.cell, 0.25f))); g.kappa_d = o.kappa_diffuse; g.hz_d = o.horizon_diffuse; g.hand = o.hand_over; g.limb_nv = o.limb_nv; g.limb_boost = o.limb_boost; g.limb_x = o.limb_x; g.limb_hand = o.limb_hand; g.limb_ramp = o.limb_ramp; g.limb_sub = o.limb_sub; g.limb_cells = o.limb_cells;
    for (int p = 0; p <= TREE_MAX_P; ++p) gauss_legendre_t(1 << p, g.glx[p], g.glw[p]);
    // the diffuse lobe: 1x1 lattice whose node carries the cell's covariance, or the render's own lattice when the cells
    // are too wide for that (coarse refmaps) or the covariance is switched off
    g.diff_cov = (o.pixel_covariance && g.cell <= 0.03f) ? 1 : 0;  // error ~ cell^4: 2e-5 at res 128, 4e-4 at res 64
    g.stats = o.collect_stats;

    const int tb = 128;
    DRM_CHECK_CUDA(cudaMemsetAsync(L.status, 0, 64 * sizeof(int), st));
    tree_tables_kernel<<<(max(He, We) + tb - 1) / tb, tb, 0, st>>>(L.sin_t, L.cos_t, L.sin_p, L.cos_p, He, We);
    // thresholds of the footprint lattices: calibrated at res 128 (round 1); coarser refmaps have cells much wider than
    // the lobe and the kink of G1(n.d) at the limb binds, so the thresholds grow with the cell size
    const float grow = (float)fmin(10.0, pow(fmax(1.0, (M_PI / res) / (M_PI / 128.0)), 1.5));
    tree_setup_kernel<<<(N + tb - 1) / tb, tb, 0, st>>>(z6, view3, flip, env_index, N, B, alpha_min, g.cell,
                                                       o.level_scale * grow, (o.pixel_covariance ? o.level_scale0 : o.level_scale) * grow,
                                                       o.full_second_order ? o.alpha_full2 : 1e30f, o.pixel_covariance, o.flat_scale,
                                                       S, S_per_render, L.rc, L.status);
    count_launches(2);
    // ---- diffuse pyramids of the envmaps in use (view independent: shared by every render of an envmap) --------------
    if (!prepared) {
        DRM_CHECK_CUDA(cudaMemsetAsync(L.env_used, 0, sizeof(int) * B, st));
        tree_mark_used_kernel<<<(N + tb - 1) / tb, tb, 0, st>>>(L.rc, N, L.env_used);
        count_launches(1 + launch_diffuse_pyramids<T>(g, B, L.pyr_d, st));
    }
    DRM_CHECK_CUDA(cudaFuncSetAttribute(TexelKernels<T>::diff, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TREE_SMEM));
    DRM_CHECK_CUDA(cudaFuncSetAttribute(TexelKernels<T>::diff, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // ---- renders, TREE_CHUNK at a time: specular pyramids, diffuse lobe (writes out), specular passes (add) ------------
    const size_t per_render_out = (size_t)res * res * 3;
    for (int k0 = 0; k0 < N; k0 += TREE_CHUNK) {
        const int n = N - k0 < TREE_CHUNK ? N - k0 : TREE_CHUNK;
        TreeArgs a = g;
        a.rc = L.rc + k0;
        a.N = n;
        a.out = out + (size_t)k0 * per_render_out;
        tree_active_kernel<<<1, 32, 0, st>>>(a.rc, n, L.act, L.nact);
        count_launches(1);
        if (L.gs.L >= 1) {
            const int n1 = L.gs.H[1] * L.gs.W[1];
            TexelKernels<T>::template pyr<true><<<dim3((n1 + tb - 1) / tb, n), tb, 0, st>>>(a, 1, L.pyr_s);
            count_launches(1);
            for (int l = 2; l <= L.gs.L; ++l) {
                const int nl = L.gs.H[l] * L.gs.W[l];
                pyr_merge_kernel<<<dim3((nl + tb - 1) / tb, n), tb, 0, st>>>(L.gs, l, L.pyr_s, nullptr);
                count_launches(1);
            }
        }
        {
            const int pd = a.diff_cov ? 0 : L.pk;  // grid for the finest lattice a render of this call may have
            const int NGd = res << pd;
            const int tiles = ((NGd + 15) / 16) * ((NGd + 15) / 16);
            TexelKernels<T>::diff<<<dim3(tiles, n), TREE_THREADS, TREE_SMEM, st>>>(a);
            count_launches(1);
        }
        for (int p = 0; p <= L.pk; ++p) {
            a.pixcov = (o.pixel_covariance && p == 0) ? 1 : 0;
            a.pool_in = nullptr; a.heads_in = nullptr; a.pool_out = nullptr; a.heads_out = nullptr; a.pool_ctr = nullptr;
            if (p > 0) { a.pool_in = L.pool[(p - 1) & 1]; a.heads_in = L.heads[(p - 1) & 1]; }
            if (p < L.pk) {
                a.pool_out = L.pool[p & 1]; a.heads_out = L.heads[p & 1]; a.pool_cap = L.pool_cap[p & 1];
                a.pool_ctr = L.status + 8 + p;
                DRM_CHECK_CUDA(cudaMemsetAsync(a.pool_ctr, 0, sizeof(int), st));
            }
            const int NG = res << p;
            const long items = (long)((NG + 15) / 16) * ((NG + 15) / 16) * n;  // upper bound: the active renders are fewer
            a.item_ctr = L.status + 44 + p;
            DRM_CHECK_CUDA(cudaMemsetAsync(a.item_ctr, 0, sizeof(int), st));
            if (pinned) {
                switch (p) {
                    case 0: DRM_CHECK_CUDA((launch_spec_pass<0, T, true>(a, items, st))); break;
                    case 1: DRM_CHECK_CUDA((launch_spec_pass<1, T, true>(a, items, st))); break;
                    case 2: DRM_CHECK_CUDA((launch_spec_pass<2, T, true>(a, items, st))); break;
                    case 3: DRM_CHECK_CUDA((launch_spec_pass<3, T, true>(a, items, st))); break;
                    default: DRM_CHECK_CUDA((launch_spec_pass<4, T, true>(a, items, st))); break;
                }
            } else {
                switch (p) {
                    case 0: DRM_CHECK_CUDA((launch_spec_pass<0, T, false>(a, items, st))); break;
                    case 1: DRM_CHECK_CUDA((launch_spec_pass<1, T, false>(a, items, st))); break;
                    case 2: DRM_CHECK_CUDA((launch_spec_pass<2, T, false>(a, items, st))); break;
                    case 3: DRM_CHECK_CUDA((launch_spec_pass<3, T, false>(a, items, st))); break;
                    default: DRM_CHECK_CUDA((launch_spec_pass<4, T, false>(a, items, st))); break;
                }
            }
            count_launches(1);
        }
    }
    DRM_CHECK_CUDA(cudaGetLastError());
    return DRM_OK;
}

extern "C" int drm_render_refmaps_opts(const float* env, int B, int He, int We, const int32_t* env_index, const float* z6,
                                       const float* view3, const uint8_t* flip, int N, int res, int S, float alpha_min,
                                       int channel_first, float* out, void* workspace, size_t workspace_bytes,
                                       void* cuda_stream, const DrmRenderOptions* opts) {
    return render_refmaps(env, B, He, We, env_index, z6, view3, flip, N, res, S, alpha_min, channel_first, out, workspace,
                          workspace_bytes, cuda_stream, opts);
}

extern "C" int drm_render_refmaps_half(const void* env, int B, int He, int We, const int32_t* env_index, const float* z6,
                                       const float* view3, const uint8_t* flip, int N, int res, int S, float alpha_min,
                                       int channel_first, float* out, void* workspace, size_t workspace_bytes,
                                       void* cuda_stream, const DrmRenderOptions* opts) {
    return render_refmaps(static_cast<const __half*>(env), B, He, We, env_index, z6, view3, flip, N, res, S, alpha_min,
                          channel_first, out, workspace, workspace_bytes, cuda_stream, opts);
}

extern "C" int drm_render_refmaps_prepared(const void* env, int env_half, const void* pyramids, size_t pyramid_bytes,
                                           int B, int He, int We, const int32_t* env_index, const float* z6,
                                           const float* view3, const uint8_t* flip, int N, int res, int S,
                                           float alpha_min, int channel_first, float* out, void* workspace,
                                           size_t workspace_bytes, void* cuda_stream, const DrmRenderOptions* opts) {
    if (env_half)
        return render_refmaps(static_cast<const __half*>(env), B, He, We, env_index, z6, view3, flip, N, res, S,
                              alpha_min, channel_first, out, workspace, workspace_bytes, cuda_stream, opts, true,
                              pyramids, pyramid_bytes);
    return render_refmaps(static_cast<const float*>(env), B, He, We, env_index, z6, view3, flip, N, res, S, alpha_min,
                          channel_first, out, workspace, workspace_bytes, cuda_stream, opts, true, pyramids,
                          pyramid_bytes);
}

extern "C" int drm_render_refmaps(const float* env, int B, int He, int We, const int32_t* env_index, const float* z6,
                                  const float* view3, const uint8_t* flip, int N, int res, int S, float alpha_min,
                                  int channel_first, float* out, void* workspace, size_t workspace_bytes,
                                  void* cuda_stream) {
    return drm_render_refmaps_opts(env, B, He, We, env_index, z6, view3, flip, N, res, S, alpha_min, channel_first, out,
                                   workspace, workspace_bytes, cuda_stream, nullptr);
}

extern "C" void drm_render_default_options(DrmRenderOptions* o) {
    if (!o) return;
    o->kappa = 0.1f;
    o->rcap = 0.06f;
    o->rcap_simple = 0.035f;
    o->horizon = 0.03f;
    o->kappa_diffuse = 0.1f;
    o->horizon_diffuse = 0.03f;
    o->level_scale = 0.6f;
    o->level_scale0 = 0.6f;
    o->pixel_covariance = 1;
    o->full_second_order = 1;
    o->alpha_full2 = 0.1f;
    o->hand_over = 0.5f;
    o->limb_nv = 0.0f;
    o->limb_boost = 2.f;
    o->limb_x = 4.f;
    o->flat_scale = 2.0f;
    o->footprint_per_render = nullptr;
    o->collect_stats = 0;
    o->horizon_inner = 0.06f;
    o->horizon_inner_nv = 4.f;
    o->horizon_finest = 0.0375f;
    o->limb_sub = 0.f;
    o->limb_cells = 1.3f;
    o->limb_hand = 32.f;
    o->limb_ramp = 0.f;
    o->spec_kernels = 0;
}
