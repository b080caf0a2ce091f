// K2: image -> refmap scatter as a deterministic sort-by-bin segmented select (sm_100a).
//
// Replaces refmap_mask_make (reference utils/img2refmap.py:6-37) and the xyz2thetaphi call inside it
// (utils/transform.py:84-89).  The reference tests every (cell, pixel) pair (O(res^2 n), [512,n,2] temporaries);
// here each pixel generates only the cells whose fp32 window predicate it can satisfy, the (cell, pixel) pairs are
// counting-sorted by cell and the lower median under the total order (channel-sum, pixel index) is selected per cell.
// Integer atomics only place pairs inside a cell's segment; the selection is order-independent, so every output is
// bit-exact and run-to-run deterministic.
//
//   pass 0  i2r_hist_pass     normals + colours read once: angles, window, sum key; the histogram atomic's return value
//                             is the pixel's rank inside its first cell -> (cell, key, rank) per pixel, 12 B
//   scan    i2r_scan_kernel   one kernel, two-level exclusive scan of the cell counts
//   pass 1  i2r_scatter_pass  pure placement pairs[offset(cell) + rank] = (tag | pixel, key): no atomics, no search
//                             (pixels with several cells -- windows wider than a cell -- recompute their window here)
//   select  i2r_select_small  64 cells per CTA staged in shared memory, element-parallel rank counting
//           i2r_select_big    warp per cell: cells above 1024 members, NaN-angle members, mean mode
//
// The passes that read pixels are templates on a pixel accessor: RowPixels reads the compacted rows of drm_img2refmap,
// ImagePixels reads dense images under a mask in place (the *_dense instances, drm_img2refmap_dense).
//
// HBM-bound integer/compare work by its bytes (24 B per pixel in, 13 B per cell out), no tensor cores; what limits the
// kernels today is instruction issue (acosf/atan2f and the window tests in pass 0, the rank counting in the select) and
// the L2 transaction rate of the 8-byte scattered stores in pass 1 -- see DESIGN.md.
#include <math.h>

#include "common.cuh"

namespace drm {

static constexpr uint32_t KEY_NAN = 0xFFFFFFFFu;  // sentinel: colour sum is NaN (ignored by nanmedian, :30-31)
static constexpr uint32_t CELL_NONE = 0x7FFFFFFFu, CELL_MULTI = 0x80000000u;

struct I2RArgs {
    const float* colors;
    const float* geom;  // normals [n,3] or thetaphi [n,2]
    const int64_t* offsets;
    int64_t total_n;
    int B, C, res, res2;
    int is_thetaphi;
    float thr, stepf, inv_step;
    int R;  // candidate radius in cells
    int min_points, reduce_mode;
    int64_t pair_capacity;
    // workspace
    int32_t* cnt_first;   // [M+1] pairs (cell, pixel) where the cell is the pixel's first one: their rank inside the
                          //       cell's segment is the value the histogram atomic returned
    int32_t* cnt_other;   // [M+1] the other pairs of pixels that fall into several cells (thr > step/2, or exact ties)
    int32_t* cursor;      // [M]   placement counter of those other pairs (pass 1)
    int32_t* nan_count;   // [B]
    int32_t* nan_list;    // [total_n]  (image b owns the slice starting at offsets[b])
    int32_t* bin_offset;  // [M+1] exclusive scan of cnt_first + cnt_other inside each tile of SCAN_TILE cells
    int32_t* block_sums;  // [tiles] exclusive scan of the tile totals (seg_offset() adds the two)
    int32_t* scan_ticket; // [1] counts finished scan tiles: the last one scans the tile totals
    uint2* pairs;         // (cell tag << 26 | global pixel index, key): one 64-bit load gives (key << 32) | tag | pixel,
                          // whose order inside a cell is the total order (key, pixel); tag = cell % SEL_CELLS
    uint32_t* cell0;      // [total_n] first cell of each pixel (CELL_NONE if none), bit 31 set if it has more cells
    uint32_t* key0;       // [total_n] sum key of the pixel
    int32_t* rank0;       // [total_n] rank of the pixel inside its first cell
    int32_t* block_image; // [ceil(total_n / 256)] image of the first pixel of each 256-pixel block
    int32_t* nankey_flag; // [B] set when some pixel of the image has a NaN colour sum
    int32_t* big_list;    // [M] cells left to the warp-per-cell select (large, NaN-angle members, mean mode)
    int32_t* big_count;   // [1]
    int32_t* status;      // bit 0: pair buffer overflow
    // outputs
    float* refmap;
    uint8_t* refmask;
    int32_t* counts;
    int32_t* sel_index;
};

static constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 8, SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// first pair of cell g: the scan leaves tile-local prefixes in bin_offset and the tiles' own prefixes in block_sums
__device__ __forceinline__ int seg_offset(const I2RArgs& a, int g) {
    return a.bin_offset[g] + a.block_sums[g / SCAN_TILE];
}

// theta = acos(n . [0,1,0]), phi = atan2(n . [0,0,1], n . [-1,0,0]) with the dot products evaluated literally
// (utils/transform.py:87-88 with normal=[0,1,0], tangent=[-1,0,0], binormal=cross=[0,0,1]); IEEE acosf/atan2f.
__device__ __forceinline__ void normal_to_thetaphi(float x, float y, float z, float& th, float& ph) {
    float ny = __fadd_rn(__fadd_rn(__fmul_rn(x, 0.f), __fmul_rn(y, 1.f)), __fmul_rn(z, 0.f));
    float nt = __fadd_rn(__fadd_rn(__fmul_rn(x, -1.f), __fmul_rn(y, 0.f)), __fmul_rn(z, 0.f));
    float nb = __fadd_rn(__fadd_rn(__fmul_rn(x, 0.f), __fmul_rn(y, 0.f)), __fmul_rn(z, 1.f));
    th = acosf(ny);
    ph = atan2f(nb, nt);
}

__global__ void normals_to_thetaphi_kernel(const float* __restrict__ normals, int64_t n, float* __restrict__ out) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n) return;
    float th, ph;
    normal_to_thetaphi(normals[3 * p], normals[3 * p + 1], normals[3 * p + 2], th, ph);
    out[2 * p] = th;
    out[2 * p + 1] = ph;
}

__device__ __forceinline__ int image_of(const int64_t* __restrict__ offsets, int B, int64_t p) {
    int lo = 0, hi = B;  // find b with offsets[b] <= p < offsets[b+1]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (offsets[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// image of the first pixel of every 256-pixel block (one binary search per block, done once; the passes then walk
// forward from it, usually zero steps)
__global__ void i2r_block_image_kernel(const int64_t* __restrict__ offsets, int B, int64_t nblk, int32_t* __restrict__ out) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < nblk) out[k] = image_of(offsets, B, k * 256);
}

// monotone uint key of the fp32 channel sum; -0.0 and +0.0 share a key (torch compares them equal)
__device__ __forceinline__ uint32_t sum_key(const float* __restrict__ c, int C) {
    float s;  // ((c0 + c1) + c2), colors.sum(-1) at img2refmap.py:30
    if (C == 3) {
        s = __fadd_rn(__fadd_rn(c[0], c[1]), c[2]);
    } else {
        s = c[0];
        for (int k = 1; k < C; ++k) s = __fadd_rn(s, c[k]);
    }
    if (isnan(s)) return KEY_NAN;
    s = __fadd_rn(s, 0.0f);  // -0.0 -> +0.0
    uint32_t b = __float_as_uint(s);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// sum_key of the channels c[0], c[cs], ..., c[(C-1)*cs]: the same sum in the same order
__device__ __forceinline__ uint32_t sum_key_strided(const float* __restrict__ c, int64_t cs, int C) {
    float s = c[0];
    for (int k = 1; k < C; ++k) s = __fadd_rn(s, c[k * cs]);
    if (isnan(s)) return KEY_NAN;
    s = __fadd_rn(s, 0.0f);
    uint32_t b = __float_as_uint(s);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// The cells of one axis whose window holds the angle x: centres are (arange + 0.5) * (pi / res) (img2refmap.py:16) and
// the fp32 predicate |centre - x| <= thr (:27) alone decides membership.  The rounded difference is monotone in the
// cell index, so the members are one run [lo, hi]: the candidates (+-1 cell for rounding) are trimmed from both ends.
__device__ __forceinline__ bool axis_cells(const I2RArgs& a, float x, int& lo, int& hi) {
    // floor() and the int conversion in one saturating instruction: +-inf and huge angles give an empty range
    lo = max(__float2int_rd((x - a.thr) * a.inv_step - 0.5f), 0);
    hi = min(__float2int_rd((x + a.thr) * a.inv_step - 0.5f), a.res - 2) + 1;
    const float thr = a.thr, step = a.stepf;
    if (hi - lo <= 2) {
        // up to three candidates (any window narrower than a cell): tested side by side, no loop
        const float f = (float)lo;  // (float)(lo + k) + 0.5f == f + (k + 0.5f) exactly
        const bool p0 = hi >= lo && fabsf(__fsub_rn(__fmul_rn(f + 0.5f, step), x)) <= thr;
        const bool p1 = hi > lo && fabsf(__fsub_rn(__fmul_rn(f + 1.5f, step), x)) <= thr;
        const bool p2 = hi > lo + 1 && fabsf(__fsub_rn(__fmul_rn(f + 2.5f, step), x)) <= thr;
        hi = p2 ? lo + 2 : p1 ? lo + 1 : lo;
        lo = p0 ? lo : p1 ? lo + 1 : lo + 2;
        return p0 || p1 || p2;
    }
    while (lo <= hi && fabsf(__fsub_rn(__fmul_rn((float)lo + 0.5f, step), x)) > thr) ++lo;
    while (hi > lo && fabsf(__fsub_rn(__fmul_rn((float)hi + 0.5f, step), x)) > thr) --hi;
    return lo <= hi;
}

__device__ __forceinline__ void load_angles(const I2RArgs& a, int64_t p, float& th, float& ph) {
    if (a.is_thetaphi) {
        const float2 v = reinterpret_cast<const float2*>(a.geom)[p];
        th = v.x;
        ph = v.y;
    } else {
        normal_to_thetaphi(a.geom[3 * p], a.geom[3 * p + 1], a.geom[3 * p + 2], th, ph);
    }
}

static constexpr int SEL_CELLS = 64;  // cells per CTA of the select kernel: a pair carries its cell id modulo this
static constexpr int PIX_BITS = 26;   // ... above the pixel index, so one call takes up to 2^26 pixels
static constexpr uint32_t PIX_MASK = (1u << PIX_BITS) - 1u;

// ---- pixel accessors: how the passes reach pixel p's colour, geometry and image.  The pass bodies below are templates
// on them; the compacted instances are the kernels of drm_img2refmap, the dense ones (*_dense) those of
// drm_img2refmap_dense.
//
// RowPixels: compacted rows -- colors [n, C], normals [n, 3] or thetaphi [n, 2]; image b owns rows offsets[b] ..
// offsets[b+1]-1 (pass 0 walks forward from block_image, the others search offsets).
struct RowPixels {
    __device__ __forceinline__ bool selected(const I2RArgs&, int64_t) const { return true; }
    __device__ __forceinline__ void load_geom(const I2RArgs& a, int64_t p, float g[3]) const {
        if (a.is_thetaphi) {
            const float2 v = reinterpret_cast<const float2*>(a.geom)[p];
            g[0] = v.x; g[1] = v.y; g[2] = 0.f;
        } else {
            g[0] = a.geom[3 * p]; g[1] = a.geom[3 * p + 1]; g[2] = a.geom[3 * p + 2];
        }
    }
    __device__ __forceinline__ void load_rgb(const I2RArgs& a, int64_t p, float c[3]) const {
        c[0] = a.colors[3 * p]; c[1] = a.colors[3 * p + 1]; c[2] = a.colors[3 * p + 2];
    }
    __device__ __forceinline__ void angles(const I2RArgs& a, int64_t p, float& th, float& ph) const { load_angles(a, p, th, ph); }
    __device__ __forceinline__ uint32_t key(const float* colors, int C, int64_t p) const { return sum_key(colors + p * C, C); }
    __device__ __forceinline__ float color(const float* colors, int C, int64_t p, int c) const { return colors[p * C + c]; }
    __device__ __forceinline__ int image_in_block(const I2RArgs& a, unsigned blk, int64_t p) const {
        int b = a.block_image[blk];
        while (b + 1 < a.B && a.offsets[b + 1] <= p) ++b;
        return b;
    }
    __device__ __forceinline__ int image(const I2RArgs& a, int64_t p) const { return image_of(a.offsets, a.B, p); }
    __device__ __forceinline__ int64_t base(const I2RArgs& a, int b) const { return a.offsets[b]; }
};

// ImagePixels: dense images -- pixel p = (b * H + y) * W + x of B images of H x W, colour channel c at
// colors[b*cs[0] + y*cs[1] + x*cs[2] + c*cs[3]] and normal component k likewise through ns (element strides, so any
// [B,H,W,C] or [B,C,H,W] view), included when mask[p] != 0 (mask [B,H,W] contiguous, NULL = every pixel).  The image
// of p is p / (H*W) and its first pixel b*H*W, so nan_list and sel_index hold the dense image-local index y*W + x.
// B*H*W <= 2^26, so pixel ids and the divisions are 32-bit.
struct ImagePixels {
    const uint8_t* mask;
    int64_t cs[4], ns[4];
    uint32_t HW, W;
    __device__ __forceinline__ int64_t at(const int64_t* s, int64_t p) const {
        const uint32_t q = (uint32_t)p, b = q / HW, r = q - b * HW, y = r / W, x = r - y * W;
        return (int64_t)b * s[0] + (int64_t)y * s[1] + (int64_t)x * s[2];
    }
    __device__ __forceinline__ bool selected(const I2RArgs&, int64_t p) const { return !mask || mask[p]; }
    __device__ __forceinline__ void load_geom(const I2RArgs& a, int64_t p, float g[3]) const {
        const float* n = a.geom + at(ns, p);
        g[0] = n[0]; g[1] = n[ns[3]]; g[2] = n[2 * ns[3]];
    }
    __device__ __forceinline__ void load_rgb(const I2RArgs& a, int64_t p, float c[3]) const {
        const float* v = a.colors + at(cs, p);
        c[0] = v[0]; c[1] = v[cs[3]]; c[2] = v[2 * cs[3]];
    }
    __device__ __forceinline__ void angles(const I2RArgs& a, int64_t p, float& th, float& ph) const {
        float g[3];
        load_geom(a, p, g);
        normal_to_thetaphi(g[0], g[1], g[2], th, ph);
    }
    __device__ __forceinline__ uint32_t key(const float* colors, int C, int64_t p) const {
        return sum_key_strided(colors + at(cs, p), cs[3], C);
    }
    __device__ __forceinline__ float color(const float* colors, int, int64_t p, int c) const {
        return colors[at(cs, p) + c * cs[3]];
    }
    __device__ __forceinline__ int image_in_block(const I2RArgs&, unsigned, int64_t p) const { return (int)((uint32_t)p / HW); }
    __device__ __forceinline__ int image(const I2RArgs&, int64_t p) const { return (int)((uint32_t)p / HW); }
    __device__ __forceinline__ int64_t base(const I2RArgs&, int b) const { return (int64_t)b * HW; }
};

// PASS 0: angles, window, sum key, histogram of the cells.  Each pixel keeps (first cell, key, rank inside that cell) so
// that pass 1 places it without touching its normal or colour again.  A thread takes HIST_PX pixels (256 apart): all
// their loads are issued first, and the rank that the histogram atomic returns is only consumed by the stores at the
// end, so the latency of one pixel's atomic hides behind the arithmetic of the next.  A pixel outside the mask keeps
// CELL_NONE and is not seen again.
static constexpr int HIST_PX = 2;
template <class P>
__device__ __forceinline__ void hist_pass_body(const I2RArgs& a, const P& px, unsigned tid) {
    int64_t p[HIST_PX];
    bool in[HIST_PX], sel[HIST_PX];
    float g[HIST_PX][3], col[HIST_PX][3];
#pragma unroll
    for (int u = 0; u < HIST_PX; ++u) {
        p[u] = ((int64_t)blockIdx.x * HIST_PX + u) * 256 + tid;
        in[u] = p[u] < a.total_n;
        const int64_t pc = in[u] ? p[u] : a.total_n - 1;
        sel[u] = px.selected(a, pc);
        px.load_geom(a, pc, g[u]);
        if (a.C == 3) px.load_rgb(a, pc, col[u]);
    }
    uint32_t cell0[HIST_PX], key[HIST_PX];
    int rank[HIST_PX];
#pragma unroll
    for (int u = 0; u < HIST_PX; ++u) {
        cell0[u] = CELL_NONE;
        rank[u] = 0;
        if (!in[u]) continue;
        if (!sel[u]) {
            key[u] = 0u;
            continue;
        }
        float th, ph;
        if (a.is_thetaphi) { th = g[u][0]; ph = g[u][1]; }
        else normal_to_thetaphi(g[u][0], g[u][1], g[u][2], th, ph);
        key[u] = a.C == 3 ? sum_key(col[u], 3) : px.key(a.colors, a.C, p[u]);
        const int b = px.image_in_block(a, blockIdx.x * HIST_PX + u, p[u]);
        if (key[u] == KEY_NAN) a.nankey_flag[b] = 1;
        if (isnan(th) || isnan(ph)) {
            // 'NaN > thr' is False (img2refmap.py:27): the pixel is a member of every cell of its image
            const int64_t base = px.base(a, b);
            const int slot = atomicAdd(&a.nan_count[b], 1);
            a.nan_list[base + slot] = (int32_t)(p[u] - base);
            continue;
        }
        int i0, i1, j0, j1;
        if (!(axis_cells(a, th, i0, i1) && axis_cells(a, ph, j0, j1))) continue;
        const int img0 = b * a.res2;
        const int first = img0 + i0 * a.res + j0;
        const bool multi = i1 > i0 || j1 > j0;
        rank[u] = atomicAdd(&a.cnt_first[first], 1);
        cell0[u] = (uint32_t)first | (multi ? CELL_MULTI : 0u);
        if (multi)
            for (int i = i0; i <= i1; ++i)
                for (int j = (i == i0 ? j0 + 1 : j0); j <= j1; ++j) atomicAdd(&a.cnt_other[img0 + i * a.res + j], 1);
    }
#pragma unroll
    for (int u = 0; u < HIST_PX; ++u) {
        if (!in[u]) continue;
        a.cell0[p[u]] = cell0[u];
        a.key0[p[u]] = key[u];
        a.rank0[p[u]] = rank[u];
    }
}

__global__ void __launch_bounds__(256) i2r_hist_pass(I2RArgs a) { hist_pass_body(a, RowPixels{}, threadIdx.x); }
__global__ void __launch_bounds__(256) i2r_hist_pass_dense(I2RArgs a, ImagePixels px) { hist_pass_body(a, px, threadIdx.x); }

__device__ __forceinline__ void place_pair(const I2RArgs& a, int64_t slot, int cell, uint32_t p, uint32_t key) {
    if (slot < a.pair_capacity) a.pairs[slot] = make_uint2(p | ((uint32_t)(cell % SEL_CELLS) << PIX_BITS), key);
    else atomicOr(a.status, 1);
}

// PASS 1: place (pixel, key) in the cell segments.  Four pixels per thread: the three record streams are read with
// 16-byte loads and the four segment-offset gathers are in flight together (the pass is latency-bound otherwise).
static constexpr int SCATTER_PX = 4;
template <class P>
__device__ __forceinline__ void scatter_pass_body(const I2RArgs& a, const P& px) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;  // quad of pixels
    const int64_t p0 = q * SCATTER_PX;
    if (p0 >= a.total_n) return;
    uint32_t c0[SCATTER_PX], key[SCATTER_PX];
    int rank[SCATTER_PX], off[SCATTER_PX];
    if (p0 + SCATTER_PX <= a.total_n) {
        const uint4 c = reinterpret_cast<const uint4*>(a.cell0)[q], k = reinterpret_cast<const uint4*>(a.key0)[q];
        const int4 r = reinterpret_cast<const int4*>(a.rank0)[q];
        c0[0] = c.x; c0[1] = c.y; c0[2] = c.z; c0[3] = c.w;
        key[0] = k.x; key[1] = k.y; key[2] = k.z; key[3] = k.w;
        rank[0] = r.x; rank[1] = r.y; rank[2] = r.z; rank[3] = r.w;
    } else {
#pragma unroll
        for (int u = 0; u < SCATTER_PX; ++u) {
            const bool in = p0 + u < a.total_n;
            c0[u] = in ? a.cell0[p0 + u] : CELL_NONE;
            key[u] = in ? a.key0[p0 + u] : 0u;
            rank[u] = in ? a.rank0[p0 + u] : 0;
        }
    }
#pragma unroll
    for (int u = 0; u < SCATTER_PX; ++u) off[u] = c0[u] != CELL_NONE ? seg_offset(a, (int)(c0[u] & ~CELL_MULTI)) : 0;
#pragma unroll
    for (int u = 0; u < SCATTER_PX; ++u)
        if (c0[u] != CELL_NONE) place_pair(a, (int64_t)off[u] + rank[u], (int)(c0[u] & ~CELL_MULTI), (uint32_t)(p0 + u), key[u]);
    bool any_multi = false;
#pragma unroll
    for (int u = 0; u < SCATTER_PX; ++u) any_multi |= c0[u] != CELL_NONE && (c0[u] & CELL_MULTI);
    if (!any_multi) return;
#pragma unroll
    for (int u = 0; u < SCATTER_PX; ++u) {
        if (c0[u] == CELL_NONE || !(c0[u] & CELL_MULTI)) continue;
        // the pixel's other cells: the same window arithmetic as pass 0; they fill the segment behind the first-cell pairs
        const int64_t p = p0 + u;
        const int b = px.image(a, p);
        float th, ph;
        px.angles(a, p, th, ph);
        int i0, i1, j0, j1;
        if (!(axis_cells(a, th, i0, i1) && axis_cells(a, ph, j0, j1))) continue;
        const int img0 = b * a.res2;
        for (int i = i0; i <= i1; ++i)
            for (int j = (i == i0 ? j0 + 1 : j0); j <= j1; ++j) {
                const int g = img0 + i * a.res + j;
                place_pair(a, (int64_t)seg_offset(a, g) + a.cnt_first[g] + atomicAdd(&a.cursor[g], 1), g, (uint32_t)p, key[u]);
            }
    }
}

__global__ void __launch_bounds__(256) i2r_scatter_pass(I2RArgs a) { scatter_pass_body(a, RowPixels{}); }
__global__ void __launch_bounds__(256) i2r_scatter_pass_dense(I2RArgs a, ImagePixels px) { scatter_pass_body(a, px); }

// ---- exclusive scan of cnt_first + cnt_other: ONE kernel.  Every CTA scans its tile of SCAN_TILE cells; the CTA that
// finishes last (a ticket counter) scans the tile totals.  The consumers add the two levels (seg_offset).
__device__ __forceinline__ int block_exclusive_scan(int v, int& total) {
    __shared__ int warp_sums[SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    if (w == 0) {
        int s = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0;
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += t;
        }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = s;
    }
    __syncthreads();
    const int wprefix = w ? warp_sums[w - 1] : 0;
    total = warp_sums[SCAN_THREADS / 32 - 1];
    __syncthreads();
    return wprefix + inc - v;
}

__global__ void __launch_bounds__(SCAN_THREADS) i2r_scan_kernel(const int32_t* __restrict__ in, const int32_t* __restrict__ in2,
                                                                int32_t* __restrict__ out, int32_t* block_sums,
                                                                int32_t* ticket, int64_t M) {
    __shared__ bool last;
    const int64_t start = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS], s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        v[k] = (start + k < M) ? in[start + k] + in2[start + k] : 0;
        s += v[k];
    }
    int total;
    int ex = block_exclusive_scan(s, total);
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        if (start + k < M) out[start + k] = ex;
        ex += v[k];
    }
    if (threadIdx.x == 0) {
        block_sums[blockIdx.x] = total;
        __threadfence();
        last = atomicAdd(ticket, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int nblocks = (int)gridDim.x;
    int carry = 0;
    for (int s0 = 0; s0 < nblocks; s0 += SCAN_THREADS) {
        const int i = s0 + threadIdx.x;
        const int t = i < nblocks ? __ldcg(&block_sums[i]) : 0;
        int tot;
        const int e = block_exclusive_scan(t, tot);
        if (i < nblocks) block_sums[i] = carry + e;
        carry += tot;
    }
}

// ---- selection of the lower median under the total order (sum key, pixel index) ----------------------------------
template <class P>
struct CellView {
    const uint2* seg;
    int nreg;
    const int32_t* nan_list;  // image-local indices
    int nnan;
    int64_t base;             // first pixel of the image
    const float* colors;      // global
    int C;
    P px;
    __device__ __forceinline__ uint64_t get(int e) const {  // (key << 32) | global pixel index
        if (e < nreg) {
            uint2 pr = seg[e];
            return ((uint64_t)pr.y << 32) | (pr.x & PIX_MASK);
        }
        const int64_t idx = base + nan_list[e - nreg];
        return ((uint64_t)px.key(colors, C, idx) << 32) | (uint32_t)idx;
    }
};

template <class P>
__device__ __forceinline__ void write_cell(const I2RArgs& a, const P& px, int64_t gbin, int64_t base, bool filled, int cnt,
                                           int64_t winner) {
    for (int c = 0; c < a.C; ++c) a.refmap[gbin * a.C + c] = filled ? px.color(a.colors, a.C, winner, c) : 0.f;
    a.refmask[gbin] = filled ? 1 : 0;
    if (a.counts) a.counts[gbin] = cnt;
    if (a.sel_index) a.sel_index[gbin] = filled ? (int32_t)(winner - base) : -1;
}

// Median mode, cells without NaN-angle members.  A CTA owns SEL_CELLS consecutive cells, i.e. one contiguous run of
// pairs: the run (and each pair's cell tag, left by pass 1) is staged in shared memory with coalesced loads, then the
// work is ELEMENT-parallel -- every staged pair counts the members of its own cell that are smaller (members are
// distinct 64-bit values) and the one whose rank is the lower-median rank names the winner.  All lanes stay busy
// whatever the cell sizes are; a warp's lanes belong to two or three neighbouring cells, so they read the same few
// shared-memory words (broadcast).  The cells' outputs are then written by one thread per cell, coalesced.
// When the 64 cells hold more pairs than the staging buffer they are taken in several batches.  Cells with more than
// SEL_MAXN members, cells with NaN-angle members and the mean mode are queued for the warp-per-cell kernel.
static constexpr int SEL_THREADS = 256, SEL_CAP = 3072, SEL_MAXN = 1024;

// rank + (v < mine) for 64-bit values: v < mine exactly when mine + ~v (= mine - v - 1 mod 2^64) carries out, so the
// comparison is one add-with-carry chain and its carry is added to the rank -- no predicates, no selects
// (the staging buffer holds ~v)
__device__ __forceinline__ uint32_t add_if_less(uint32_t rank, uint64_t not_v, uint32_t mlo, uint32_t mhi) {
    [[maybe_unused]] uint32_t t;
    asm("{\n\t"
        "add.cc.u32 %1, %4, %2;\n\t"
        "addc.cc.u32 %1, %5, %3;\n\t"
        "addc.u32 %0, %0, 0;\n\t"
        "}"
        : "+r"(rank), "=&r"(t)
        : "r"((uint32_t)not_v), "r"((uint32_t)(not_v >> 32)), "r"(mlo), "r"(mhi));
    return rank;
}
static constexpr int CELL_EMPTY = -1, CELL_QUEUED = -2;
template <class P>
__device__ __forceinline__ void select_small_body(const I2RArgs& a, const P& px, int64_t M) {
    __shared__ uint64_t buf[SEL_CAP];  // the staged pairs, complemented (see add_if_less)
    __shared__ int s_off[SEL_CELLS + 1];
    __shared__ int s_k[SEL_CELLS];         // median rank of the cell, or CELL_EMPTY / CELL_QUEUED
    __shared__ uint32_t s_win[SEL_CELLS];  // the winner's global pixel index
    const int tid = threadIdx.x;
    const int64_t g0 = blockIdx.x * (int64_t)SEL_CELLS;
    const int ncell = (int)min((int64_t)SEL_CELLS, M - g0);
    if (tid <= ncell) s_off[tid] = seg_offset(a, (int)(g0 + tid));
    __syncthreads();
    int b = 0, cnt = 0;
    if (tid < ncell) {
        b = (int)(g0 + tid) / a.res2;  // M < 2^31
        const int nreg = s_off[tid + 1] - s_off[tid], nnan = a.nan_count[b];
        cnt = nreg + nnan;  // (~angle_mask).sum(-1), img2refmap.py:28
        int k;
        if (cnt == 0 || cnt < a.min_points) k = CELL_EMPTY;
        else if (nnan > 0 || nreg > SEL_MAXN || a.reduce_mode != 0) k = CELL_QUEUED;
        else k = (nreg - 1) >> 1;  // lower median, torch.nanmedian (:31); corrected below if some keys are NaN
        s_k[tid] = k;
    }
    // the cells are taken in batches whose pairs fit the staging buffer: all of them at once unless they are large
    for (int c0 = 0; c0 < ncell;) {
        int c1 = ncell;
        if (s_off[ncell] - s_off[c0] > SEL_CAP) {
            c1 = c0 + 1;  // a cell beyond SEL_MAXN <= SEL_CAP is queued: staging a part of it is harmless
            while (c1 < ncell && s_off[c1 + 1] - s_off[c0] <= SEL_CAP) ++c1;
        }
        const int run0 = s_off[c0];
        const int staged = min(s_off[c1] - run0, SEL_CAP);
        __syncthreads();  // s_k written; the previous batch is done with buf
        {
            const uint64_t* __restrict__ src = reinterpret_cast<const uint64_t*>(a.pairs) + run0;
            for (int e = tid; e < staged; e += SEL_THREADS) buf[e] = ~src[e];
        }
        __syncthreads();
        if (tid >= c0 && tid < c1 && s_k[tid] >= 0 && a.nankey_flag[b]) {
            // NaN keys are the largest values, so rank (nvalid - 1) / 2 of the whole segment is the lower median of the
            // valid members
            const int off = s_off[tid] - run0, nreg = s_off[tid + 1] - s_off[tid];
            int nvalid = 0;
            for (int e = 0; e < nreg; ++e) nvalid += (uint32_t)(~buf[off + e] >> 32) != KEY_NAN;
            s_k[tid] = nvalid ? (nvalid - 1) >> 1 : CELL_EMPTY;
        }
        __syncthreads();
        for (int e = tid; e < staged; e += SEL_THREADS) {
            const uint64_t mine = ~buf[e];
            const int c = ((uint32_t)mine >> PIX_BITS);
            const int k = s_k[c];
            if (k < 0) continue;
            const int n = s_off[c + 1] - s_off[c];
            const uint64_t* __restrict__ seg = buf + (s_off[c] - run0);
            const uint32_t mlo = (uint32_t)mine, mhi = (uint32_t)(mine >> 32);
            uint32_t rank = 0;
            int f = 0;
#pragma unroll 1
            for (; f + 4 <= n; f += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) rank = add_if_less(rank, seg[f + u], mlo, mhi);
            }
#pragma unroll 1
            for (; f < n; ++f) rank = add_if_less(rank, seg[f], mlo, mhi);
            if ((int)rank == k) s_win[c] = mlo & PIX_MASK;
        }
        c0 = c1;
    }
    __syncthreads();
    if (tid < ncell) {
        const int k = s_k[tid];
        if (k == CELL_QUEUED) a.big_list[atomicAdd(a.big_count, 1)] = (int32_t)(g0 + tid);
        else write_cell(a, px, g0 + tid, px.base(a, b), k >= 0, cnt, k >= 0 ? (int64_t)s_win[tid] : 0);
    }
}

__global__ void __launch_bounds__(SEL_THREADS) i2r_select_small(I2RArgs a, int64_t M) { select_small_body(a, RowPixels{}, M); }
__global__ void __launch_bounds__(SEL_THREADS) i2r_select_small_dense(I2RArgs a, ImagePixels px, int64_t M) {
    select_small_body(a, px, M);
}

// one warp per queued cell
template <class P>
__device__ __forceinline__ void select_big_body(const I2RArgs& a, const P& px) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nbig = *a.big_count;
    for (int64_t q = warp0; q < nbig; q += nwarps) {
        const int64_t gbin = a.big_list[q];
        const int b = (int)(gbin / a.res2);
        const int64_t base = px.base(a, b);
        CellView<P> cv;
        cv.nreg = seg_offset(a, (int)gbin + 1) - seg_offset(a, (int)gbin);
        cv.seg = a.pairs + seg_offset(a, (int)gbin);
        cv.nnan = a.nan_count[b];
        cv.nan_list = a.nan_list + base;
        cv.base = base;
        cv.colors = a.colors;
        cv.C = a.C;
        cv.px = px;
        const int cnt = cv.nreg + cv.nnan;

        int64_t winner = -1;
        float mean_c = 0.f;
        bool filled = false;
        // valid = members whose sum is not NaN
        int nvalid = 0;
        for (int e0 = 0; e0 < cnt; e0 += 32) {
            int e = e0 + lane;
            bool v = e < cnt && (uint32_t)(cv.get(e) >> 32) != KEY_NAN;
            nvalid += __popc(__ballot_sync(0xffffffffu, v));
        }
        if (nvalid > 0) {
            filled = true;
            if (a.reduce_mode == 0) {
                const int k = (nvalid - 1) >> 1;  // lower median, torch.nanmedian (:31)
                for (int e0 = 0; e0 < cnt && winner < 0; e0 += 32) {
                    const int e = e0 + lane;
                    const uint64_t mine = e < cnt ? cv.get(e) : ~0ull;
                    int rank = 0;
                    for (int f = 0; f < cnt; ++f) rank += cv.get(f) < mine;
                    unsigned hit = __ballot_sync(0xffffffffu, e < cnt && rank == k);
                    if (hit) winner = (int64_t)(uint32_t)__shfl_sync(0xffffffffu, mine, __ffs(hit) - 1);
                }
            } else {
                // mean: fp32 sum over valid members in ascending pixel order; lane c owns channel c
                int64_t prev = -1;
                float acc = 0.f;
                for (int r = 0; r < nvalid; ++r) {
                    long long best = 0x7fffffffffffffffll;
                    for (int e0 = 0; e0 < cnt; e0 += 32) {
                        int e = e0 + lane;
                        if (e < cnt) {
                            uint64_t el = cv.get(e);
                            long long idx = (long long)(uint32_t)el;
                            if ((uint32_t)(el >> 32) != KEY_NAN && idx > prev) best = min(best, idx);
                        }
                    }
                    for (int d = 16; d; d >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, d));
                    if (lane < a.C) acc = __fadd_rn(acc, px.color(cv.colors, a.C, best, lane));
                    prev = best;
                }
                mean_c = __fdiv_rn(acc, (float)nvalid);
            }
        }
        if (lane < a.C) {
            float v = 0.f;
            if (filled) v = a.reduce_mode == 0 ? px.color(cv.colors, a.C, winner, lane) : mean_c;
            a.refmap[gbin * a.C + lane] = v;
        }
        if (lane == 0) {
            a.refmask[gbin] = filled ? 1 : 0;
            if (a.counts) a.counts[gbin] = cnt;
            if (a.sel_index) a.sel_index[gbin] = (filled && a.reduce_mode == 0) ? (int32_t)(winner - base) : -1;
        }
    }
}

__global__ void __launch_bounds__(256) i2r_select_big(I2RArgs a) { select_big_body(a, RowPixels{}); }
__global__ void __launch_bounds__(256) i2r_select_big_dense(I2RArgs a, ImagePixels px) { select_big_body(a, px); }

static int64_t pairs_per_pixel_bound(int res, float thr) {
    const double step = M_PI / res;
    int64_t per_axis = (int64_t)floor(2.0 * (double)thr / step + 1e-3) + 1;
    if (per_axis > res) per_axis = res;
    if (per_axis < 1) per_axis = 1;
    return per_axis * per_axis;
}

static size_t i2r_carve(I2RArgs& a, void* ws, int64_t total_n, int B, int res, float thr) {
    const int64_t M = (int64_t)B * res * res;
    const int64_t nblocks = (M + 1 + SCAN_TILE - 1) / SCAN_TILE;
    const size_t npx = (size_t)(total_n > 0 ? total_n : 1);
    Carver c(ws);
    a.cnt_first = c.take<int32_t>(M + 1);  // the zeroed block: carved first and contiguous, one memset
    a.cnt_other = c.take<int32_t>(M + 1);
    a.cursor = c.take<int32_t>(M);
    a.nan_count = c.take<int32_t>(B);
    a.nankey_flag = c.take<int32_t>(B);
    a.big_count = c.take<int32_t>(1);
    a.status = c.take<int32_t>(1);
    a.scan_ticket = c.take<int32_t>(1);
    a.bin_offset = c.take<int32_t>(M + 1);
    a.nan_list = c.take<int32_t>(npx);
    a.cell0 = c.take<uint32_t>(npx);
    a.key0 = c.take<uint32_t>(npx);
    a.rank0 = c.take<int32_t>(npx);
    a.big_list = c.take<int32_t>(M);
    a.block_sums = c.take<int32_t>(nblocks + 1);
    a.pair_capacity = total_n * pairs_per_pixel_bound(res, thr);
    a.pairs = c.take<uint2>(a.pair_capacity > 0 ? a.pair_capacity : 1);
    a.block_image = c.take<int32_t>((npx + 255) / 256 + HIST_PX);
    return c.used();
}

// the sizes, window constants and outputs that both entries set alike
static void i2r_set(I2RArgs& a, int B, int C, int res, float thr, int min_points, int reduce_mode, float* refmap,
                    uint8_t* refmask, int32_t* counts, int32_t* sel_index) {
    a.B = B; a.C = C; a.res = res; a.res2 = res * res;
    a.thr = thr;
    a.stepf = (float)(M_PI / res);  // python float pi/res rounded to fp32 once (img2refmap.py:16)
    a.inv_step = (float)(res / M_PI);
    a.R = (int)ceil((double)thr / (M_PI / res)) + 1;
    if (a.R > res) a.R = res;
    a.min_points = min_points; a.reduce_mode = reduce_mode;
    a.refmap = refmap; a.refmask = refmask; a.counts = counts; a.sel_index = sel_index;
}

// cnt_first, cnt_other, cursor, nan_count, big_count, status are carved first and contiguous (each 256-aligned)
static cudaError_t i2r_clear(const I2RArgs& a, cudaStream_t st) {
    return cudaMemsetAsync(a.cnt_first, 0, (size_t)((char*)a.bin_offset - (char*)a.cnt_first), st);
}

}  // namespace drm

using namespace drm;

extern "C" size_t drm_img2refmap_workspace_bytes(int64_t total_n, int B, int res, float thr) {
    if (total_n < 0 || B <= 0 || res <= 0 || !(thr >= 0.f)) return 0;
    I2RArgs a{};
    return i2r_carve(a, nullptr, total_n, B, res, thr);
}

extern "C" int drm_img2refmap(const float* colors, const float* geom, int input_is_thetaphi, const int64_t* offsets,
                              int64_t total_n, int B, int C, int res, float thr, int min_points, int reduce_mode,
                              float* refmap, uint8_t* refmask, int32_t* counts, int32_t* sel_index, void* workspace,
                              size_t workspace_bytes, void* cuda_stream) {
    DRM_REQUIRE(B > 0 && res > 0 && total_n >= 0, "img2refmap: B=%d res=%d total_n=%lld must be positive", B, res, (long long)total_n);
    DRM_REQUIRE(C >= 1 && C <= 4, "img2refmap: C=%d not in 1..4", C);
    DRM_REQUIRE(thr >= 0.f, "img2refmap: angle threshold must be a non-negative number");
    DRM_REQUIRE(reduce_mode == 0 || reduce_mode == 1, "img2refmap: reduce_mode %d (0 = median, 1 = mean)", reduce_mode);
    DRM_REQUIRE(offsets && refmap && refmask && (total_n == 0 || (colors && geom)), "img2refmap: null pointer");
    const int64_t M = (int64_t)B * res * res;
    DRM_REQUIRE(total_n <= (1ll << PIX_BITS), "img2refmap: %lld pixels in one call, at most 2^26 (split the batch)", (long long)total_n);
    DRM_REQUIRE(M < (1ll << 31), "img2refmap: B*res*res = %lld exceeds int32 cells", (long long)M);
    const int64_t per_px = pairs_per_pixel_bound(res, thr);
    if (total_n * per_px >= (1ll << 31)) {
        set_error("img2refmap: up to %lld (cell,pixel) pairs exceed the int32 segment offsets", (long long)(total_n * per_px));
        return DRM_EUNSUPPORTED;
    }
    I2RArgs a{};
    const size_t need = i2r_carve(a, workspace, total_n, B, res, thr);
    if (!workspace || workspace_bytes < need) {
        set_error("img2refmap: workspace of %zu bytes needed, %zu given", need, workspace_bytes);
        return DRM_EWORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    a.colors = colors; a.geom = geom; a.offsets = offsets; a.total_n = total_n; a.is_thetaphi = input_is_thetaphi;
    i2r_set(a, B, C, res, thr, min_points, reduce_mode, refmap, refmask, counts, sel_index);
    DRM_CHECK_CUDA(i2r_clear(a, st));
    const int64_t nblocks = (M + 1 + SCAN_TILE - 1) / SCAN_TILE;
    if (total_n > 0) {
        const int64_t nblk = (total_n + 255) / 256;
        i2r_block_image_kernel<<<(unsigned)((nblk + 255) / 256), 256, 0, st>>>(offsets, B, nblk, a.block_image);
        i2r_hist_pass<<<(unsigned)((nblk + HIST_PX - 1) / HIST_PX), 256, 0, st>>>(a);
    }
    i2r_scan_kernel<<<(unsigned)nblocks, SCAN_THREADS, 0, st>>>(a.cnt_first, a.cnt_other, a.bin_offset, a.block_sums,
                                                                a.scan_ticket, M + 1);
    if (total_n > 0) {
        const int64_t nquad = (total_n + SCATTER_PX - 1) / SCATTER_PX;
        i2r_scatter_pass<<<(unsigned)((nquad + 255) / 256), 256, 0, st>>>(a);
    }
    i2r_select_small<<<(unsigned)((M + SEL_CELLS - 1) / SEL_CELLS), SEL_THREADS, 0, st>>>(a, M);
    i2r_select_big<<<148 * 4, 256, 0, st>>>(a);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(total_n > 0 ? 6 : 3);
    return DRM_OK;
}

// The dense entry runs the passes over all B*H*W pixels, so its workspace is that of drm_img2refmap at total_n = B*H*W
// (and drm_img2refmap_status reads it with that total_n).
extern "C" size_t drm_img2refmap_dense_workspace_bytes(int B, int H, int W, int res, float thr) {
    if (B <= 0 || H <= 0 || W <= 0 || (int64_t)B * H * W > (1ll << PIX_BITS)) return 0;
    return drm_img2refmap_workspace_bytes((int64_t)B * H * W, B, res, thr);
}

extern "C" int drm_img2refmap_dense(const float* colors, const int64_t colors_strides[4], const float* normals,
                                    const int64_t normals_strides[4], const uint8_t* mask, int B, int H, int W, int C,
                                    int res, float thr, int min_points, int reduce_mode, float* refmap, uint8_t* refmask,
                                    int32_t* counts, int32_t* sel_index, void* workspace, size_t workspace_bytes,
                                    void* cuda_stream) {
    DRM_REQUIRE(colors && colors_strides && normals && normals_strides && refmap && refmask,
                "img2refmap_dense: null pointer (colors %p, colors_strides %p, normals %p, normals_strides %p, refmap %p, "
                "refmask %p)", (const void*)colors, (const void*)colors_strides, (const void*)normals,
                (const void*)normals_strides, (void*)refmap, (void*)refmask);
    DRM_REQUIRE(B > 0 && H > 0 && W > 0 && res > 0, "img2refmap_dense: B=%d H=%d W=%d res=%d must be positive", B, H, W, res);
    DRM_REQUIRE(C >= 1 && C <= 4, "img2refmap_dense: C=%d not in 1..4", C);
    DRM_REQUIRE(thr >= 0.f, "img2refmap_dense: angle threshold %g must be a non-negative number", (double)thr);
    DRM_REQUIRE(reduce_mode == 0 || reduce_mode == 1, "img2refmap_dense: reduce_mode %d (0 = median, 1 = mean)", reduce_mode);
    for (int k = 0; k < 4; ++k) {
        DRM_REQUIRE(colors_strides[k] >= 0, "img2refmap_dense: colors_strides[%d] = %lld is negative", k,
                    (long long)colors_strides[k]);
        DRM_REQUIRE(normals_strides[k] >= 0, "img2refmap_dense: normals_strides[%d] = %lld is negative", k,
                    (long long)normals_strides[k]);
    }
    const int64_t total_n = (int64_t)B * H * W, M = (int64_t)B * res * res;
    DRM_REQUIRE(total_n <= (1ll << PIX_BITS), "img2refmap_dense: B*H*W = %lld pixels in one call, at most 2^26 (split the "
                "batch)", (long long)total_n);
    DRM_REQUIRE(M < (1ll << 31), "img2refmap_dense: B*res*res = %lld exceeds int32 cells", (long long)M);
    const int64_t per_px = pairs_per_pixel_bound(res, thr);
    if (total_n * per_px >= (1ll << 31)) {
        set_error("img2refmap_dense: up to %lld (cell,pixel) pairs exceed the int32 segment offsets", (long long)(total_n * per_px));
        return DRM_EUNSUPPORTED;
    }
    I2RArgs a{};
    const size_t need = i2r_carve(a, workspace, total_n, B, res, thr);
    if (!workspace || workspace_bytes < need) {
        set_error("img2refmap_dense: workspace of %zu bytes needed, %zu given", need, workspace_bytes);
        return DRM_EWORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    a.colors = colors; a.geom = normals; a.offsets = nullptr; a.total_n = total_n; a.is_thetaphi = 0;
    i2r_set(a, B, C, res, thr, min_points, reduce_mode, refmap, refmask, counts, sel_index);
    ImagePixels px;
    px.mask = mask;
    for (int k = 0; k < 4; ++k) {
        px.cs[k] = colors_strides[k];
        px.ns[k] = normals_strides[k];
    }
    px.HW = (uint32_t)(H * W);
    px.W = (uint32_t)W;
    DRM_CHECK_CUDA(i2r_clear(a, st));
    const int64_t nblk = (total_n + 255) / 256, nquad = (total_n + SCATTER_PX - 1) / SCATTER_PX;
    i2r_hist_pass_dense<<<(unsigned)((nblk + HIST_PX - 1) / HIST_PX), 256, 0, st>>>(a, px);
    i2r_scan_kernel<<<(unsigned)((M + 1 + SCAN_TILE - 1) / SCAN_TILE), SCAN_THREADS, 0, st>>>(
        a.cnt_first, a.cnt_other, a.bin_offset, a.block_sums, a.scan_ticket, M + 1);
    i2r_scatter_pass_dense<<<(unsigned)((nquad + 255) / 256), 256, 0, st>>>(a, px);
    i2r_select_small_dense<<<(unsigned)((M + SEL_CELLS - 1) / SEL_CELLS), SEL_THREADS, 0, st>>>(a, px, M);
    i2r_select_big_dense<<<148 * 4, 256, 0, st>>>(a, px);
    DRM_CHECK_CUDA(cudaGetLastError());
    count_launches(5);
    return DRM_OK;
}

extern "C" int drm_img2refmap_status(const void* workspace, int64_t total_n, int B, int res, float thr, int32_t* status,
                                     void* cuda_stream) {
    DRM_REQUIRE(workspace && status && B > 0 && res > 0 && total_n >= 0 && thr >= 0.f, "img2refmap_status: bad arguments");
    I2RArgs a{};
    i2r_carve(a, const_cast<void*>(workspace), total_n, B, res, thr);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    DRM_CHECK_CUDA(cudaMemcpyAsync(&status[0], a.status, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    DRM_CHECK_CUDA(cudaMemcpyAsync(&status[1], a.big_count, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    DRM_CHECK_CUDA(cudaStreamSynchronize(st));
    return DRM_OK;
}

extern "C" int drm_normals_to_thetaphi(const float* normals, int64_t n, float* thetaphi, void* cuda_stream) {
    DRM_REQUIRE(n >= 0 && (n == 0 || (normals && thetaphi)), "normals_to_thetaphi: bad arguments");
    if (n == 0) return DRM_OK;
    normals_to_thetaphi_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(normals, n, thetaphi);
    DRM_CHECK_CUDA(cudaGetLastError());
    return DRM_OK;
}
