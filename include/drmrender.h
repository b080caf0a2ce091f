/*
 * drmrender.h -- C ABI of libdrmrender.so: B200 (sm_100a) implementation of DRMNet's data-parallel rendering hot path.
 *
 * This is the drop-in boundary.  Every entry point is `extern "C"`, takes plain device pointers and sizes, never
 * throws or aborts across the ABI, never calls cudaDeviceSynchronize, enqueues all work on the stream it is given and
 * returns 0 on success or a negative DRM_E* code (message via drm_last_error(), thread-local).
 * The caller owns every buffer including the workspace (query the size first); the library keeps no pointer after
 * the call returns.  There is no CPU fallback: without a CUDA device every compute entry returns DRM_ECUDA.
 *
 * Reference interfaces replaced (paths relative to the DRMNet repository):
 *   drm_render_refmaps      <- MitsubaRefMapRenderer.rendering()         utils/mitsuba3_utils.py:411-430 (-> :365-409, :217-246)
 *                              and the per-render Python loops that call it  models/drmnet.py:561-569, :680-691
 *   drm_img2refmap          <- refmap_mask_make()                        utils/img2refmap.py:6-37
 *                              (+ xyz2thetaphi as called there             utils/transform.py:55-89)
 *   drm_refmap_postprocess  <- luminance normalisation + log transform   models/drmnet.py:610-620, dataset/basedataset.py:52-53
 *   drm_mirmap2envmap       <- mirmap2envmap() inside DRMNet.r0toenvmap   utils/transform.py:106-144, models/drmnet.py:931-941
 */
#ifndef DRMRENDER_H
#define DRMRENDER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRM_VERSION 200 /* major*10000 + minor*100 + patch */

enum {
    DRM_OK = 0,
    DRM_EINVAL = -1, /* bad argument (null pointer, non-positive size, unsupported value) */
    DRM_EWORKSPACE = -2, /* workspace missing or too small */
    DRM_ECUDA = -3, /* CUDA runtime / driver error, or no device */
    DRM_EUNSUPPORTED = -4 /* valid request this build cannot serve */
};

int drm_version(void);
const char* drm_last_error(void);
/* process-wide count of kernels this library has launched so far (bench.py reports the per-step difference) */
int64_t drm_launch_count(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Reflectance-map forward render (SURVEY 8a R1-R5, R7).
 *
 *   env        [B, He, We, 3] fp32 RGB lat-long radiance, row 0 = zenith (+Y), u = atan2(x,-z)/2pi (device)
 *   env_index  [N] int32: which envmap render k uses (device)
 *   z6         [N, 6] fp32: metallic, base R, base G, base B, roughness, specular -- clipped to [0,1] by the kernel
 *              (utils/mitsuba3_utils.py:237-242); unnamed parameters carry the scene defaults 0,0,0,0,0,1 (:348-361)
 *   view3      [N, 3] fp32 camera position (any positive length; the sensor looks at the origin, up = +Y, :235-236)
 *   flip       [N] uint8 (may be NULL = no flip): mirrors the refmap columns (:38-40)
 *   footprint_S  S x S Gauss-Legendre sub-normals per refmap cell (box pixel filter, :116-117): 1, 2, 4, 8 or 16 for
 *              every render, or 0: per render -- DrmRenderOptions::footprint_per_render, else chosen on the device from
 *              the render's roughness (cell width / lobe half-width: the rule of renderer.auto_footprint).  Renders
 *              with different footprints run in the same launches
 *   alpha_min  lower clamp of the GGX alpha = roughness^2; <= 0 selects max(1e-3, 1.25*pi/He)
 *   channel_first  0: out [N, res, res, 3];  1: out [N, 3, res, res]   (:196-198)
 *   out        fp32 (device)
 * ------------------------------------------------------------------------------------------------------------- */
size_t drm_render_workspace_bytes(int N, int B, int He, int We, int res, int footprint_S);

int drm_render_refmaps(const float* env, int B, int He, int We,
                       const int32_t* env_index, const float* z6, const float* view3, const uint8_t* flip,
                       int N, int res, int footprint_S, float alpha_min, int channel_first,
                       float* out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Accuracy / cost constants of the hierarchical evaluation (DESIGN.md 5).  The defaults hold the result within 1e-4
 * (relative L2) of the full sum; they are arguments, not process environment: the library reads no environment variable. */
typedef struct DrmRenderOptions {
    float kappa;            /* a pyramid cell of half-vector radius r serves a block of normals at distance d when
                               r <= kappa * sqrt(alpha^2 + d^2) ... */
    float rcap;             /* ... and r <= rcap (radians) for renders evaluated with the full second-order terms, */
    float rcap_simple;      /* r <= rcap_simple for the others (alpha < alpha_full2) */
    float horizon;          /* cells wider than this (radians) are refined where they straddle the horizon n.d = 0 */
    float kappa_diffuse;    /* diffuse lobe: largest cell radius (radians) */
    float horizon_diffuse;  /* diffuse lobe: the same horizon rule */
    float level_scale;      /* scale of the distances beyond which a coarser footprint lattice is used (passes >= 1) */
    float level_scale0;     /* the same for the 1x1 lattice when it carries the cell covariance */
    int pixel_covariance;   /* pass 0 nodes carry the covariance of the refmap cell (fourth-order 1x1 lattice) */
    int full_second_order;  /* second-order terms of G1(n.d) and the horizon clamp per cell (needed by rough lobes) ... */
    float alpha_full2;      /* ... for renders with alpha >= this */
    float hand_over;        /* a cell too near for a pass's lattice goes to the next pass once its radius is below
                               hand_over * (that lattice's distance); larger cells are refined first */
    float limb_nv;          /* blocks of normals with min n.v below max(limb_nv, min(limb_x * alpha, limb_cells cells)) ... */
    float limb_boost;       /* ... use lattice distances scaled by this (the cell average converges later at the limb) ... */
    float limb_x;           /* ... (the rim of the refmap) ... */
    float limb_cells;       /* ... see limb_nv ... */
    float limb_sub;         /* ... on the lattices whose sub-cells are wider than limb_sub * alpha ... */
    float limb_hand;        /* hand_over of the rim blocks (default 32: near cells up to 32 lattice distances wide go down
                               whole; unbounded costs 5 % more on a 16x16-footprint render for the same errors, 16 is 3 %
                               cheaper with errors up 5 %, 8 leaves 1 % in single rim cells, 1 leaves 6e-3) */
    float limb_ramp;        /* rim blocks also hand down what lies within limb_ramp * alpha of their horizon n.d = 0
                               (default 0: off; with a finite limb_hand this is cheaper and accurate to ~3e-3 locally) */
    float flat_scale;       /* scale of the distances (in cells) beyond which a lattice is accurate because the lobe is
                               flat across the cell */
    const int32_t* footprint_per_render;  /* device, [N]: footprint S of each render (1, 2, 4, 8, 16; <= 0: chosen from
                               its roughness); NULL: footprint_S applies to every render */
    int collect_stats;      /* debug: count, per lattice pass, the pyramid cells visited and accepted (status words 16..35) */
    float horizon_inner;    /* the horizon width for blocks of normals whose n.v stays above horizon_inner_nv * alpha (and
                               outside the rim zone): the lobe does not sit on the horizon there; scaled by
                               (cell_128 / cell)^(1/4) for refmaps coarser than 128^2 and never below `horizon` */
    float horizon_inner_nv;
    float horizon_finest;   /* the horizon width near the limb on the render's own lattice (its nodes are the exact normals)
                               for the lobes that carry the per-cell horizon clamp (alpha >= alpha_full2); same scaling
                               with the cell size */
    int spec_kernels;       /* 0 (default): the specular lattice passes with the shorter evaluation loops; 1: the earlier
                               pass kernels (tree_spec_pass_kernel<P>), whose results differ by rounding only */
} DrmRenderOptions;

void drm_render_default_options(DrmRenderOptions* opts);

/* drm_render_refmaps with explicit options (opts == NULL: the defaults). */
int drm_render_refmaps_opts(const float* env, int B, int He, int We,
                            const int32_t* env_index, const float* z6, const float* view3, const uint8_t* flip,
                            int N, int res, int footprint_S, float alpha_min, int channel_first,
                            float* out, void* workspace, size_t workspace_bytes, void* cuda_stream,
                            const DrmRenderOptions* opts);

/* drm_render_refmaps_opts on an fp16 envmap: env is __half [B, He, We, 3] (IEEE binary16, device), read in place and
 * converted to fp32 texel by texel.  The conversion is exact, so the result is bit for bit that of
 * drm_render_refmaps_opts on the same map upcast to fp32, at half the envmap bytes.  Same arguments, validation,
 * workspace (drm_render_workspace_bytes), status words (drm_render_status) and options.  fp16 ends at 65504: radiance
 * above it (a sun) is +inf in the map and renders as inf or NaN, so convert with a clamp (torch: env.clamp(max=65504).half()). */
int drm_render_refmaps_half(const void* env, int B, int He, int We,
                            const int32_t* env_index, const float* z6, const float* view3, const uint8_t* flip,
                            int N, int res, int footprint_S, float alpha_min, int channel_first,
                            float* out, void* workspace, size_t workspace_bytes, void* cuda_stream,
                            const DrmRenderOptions* opts);

/* Envmap banks: the diffuse pyramid of an envmap depends on its texels alone (not on the view, the BRDF or the refmap),
 * so a caller that renders the same maps many times builds it once and renders by index.
 *
 * drm_env_pyramid_bytes: size of the buffer that holds the diffuse pyramids of B envmaps of He x We texels.  It starts
 *   with the pyramids, [B][cells][5] float4 records (cells depends on He and We), and ends with the build's scratch
 *   (direction tables and a mask of B ints).  0 for unsupported sizes (B > 65535, He * We >= 2^28).
 * drm_env_pyramid_build: builds the pyramids of the listed slots of env [B, He, We, 3] (fp32, or __half when env_half
 *   is nonzero) into `pyramids`.  ids [n_ids] int32 (device) lists the slots to build; ids outside [0, B) are skipped;
 *   NULL builds every slot.  The other slots keep their records.  A pyramid is valid only for the texels, He and We it
 *   was built from: rebuild a slot after its texels change.  Builds and renders that share a buffer must be ordered
 *   (one stream, or events).
 * drm_render_prepared_workspace_bytes / drm_render_refmaps_prepared: drm_render_refmaps_opts (drm_render_refmaps_half
 *   when env_half is nonzero) reading the diffuse pyramids from `pyramids` instead of building those of the envmaps in
 *   use in the workspace, so the workspace does not grow with B.  Bit for bit the result of drm_render_refmaps_opts on
 *   the same maps; same validation, status words (drm_render_status) and options.
 * Both entries check null pointers and sizes, and refuse a pyramid buffer smaller than drm_env_pyramid_bytes
 * (DRM_EINVAL, with the size needed in drm_last_error), before any CUDA call. */
size_t drm_env_pyramid_bytes(int B, int He, int We);

int drm_env_pyramid_build(const void* env, int env_half, int B, int He, int We, const int32_t* ids, int n_ids,
                          void* pyramids, size_t pyramid_bytes, void* cuda_stream);

size_t drm_render_prepared_workspace_bytes(int N, int B, int He, int We, int res, int footprint_S);

int drm_render_refmaps_prepared(const void* env, int env_half, const void* pyramids, size_t pyramid_bytes,
                                int B, int He, int We,
                                const int32_t* env_index, const float* z6, const float* view3, const uint8_t* flip,
                                int N, int res, int footprint_S, float alpha_min, int channel_first,
                                float* out, void* workspace, size_t workspace_bytes, void* cuda_stream,
                                const DrmRenderOptions* opts);

/* Copies the 40 status words of a finished (or enqueued: the copy is stream-ordered) render to status_host[40]:
 * [0] flags, 0 = clean: bit 0 = the pool of hand-over lists ran out (result incomplete), bit 1 = an env_index was out of
 * range, bit 2 = a traversal stack overflowed (result incomplete); [1] deepest traversal stack; [2..6] longest hand-over
 * list written by passes 0..4; [8..11] chunks of 128 ints the passes 0..3 took from their pools; with
 * DrmRenderOptions::collect_stats, [16 + 4p ..]: cells visited, traversal iterations, texels accepted, pyramid cells
 * accepted by pass p (summed over its blocks of 32 lattice nodes; they wrap for large batches). */
int drm_render_status(const void* workspace, int* status_host, void* cuda_stream);

/* Single-level evaluation of the same sum: every (sub-normal, texel) pair, S x S lattice, texels streamed by TMA
 * (round-1 kernel).  ~1e4 times more work than drm_render_refmaps; the validation path for whole images at sizes the
 * fp64 oracle cannot reach, footprint_S in 1..16 (any integer). */
size_t drm_render_flat_workspace_bytes(int N, int B, int He, int We, int res, int footprint_S);

int drm_render_refmaps_flat(const float* env, int B, int He, int We,
                            const int32_t* env_index, const float* z6, const float* view3, const uint8_t* flip,
                            int N, int res, int footprint_S, float alpha_min, int channel_first,
                            float* out, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Image -> refmap scatter (SURVEY 8a S1-S3), batched over B images through `offsets`.
 *
 *   colors     [total_n, C] fp32, C in 1..4 (device)
 *   normals_or_thetaphi  [total_n, 3] fp32 normals, or [total_n, 2] fp32 (theta, phi) when input_is_thetaphi != 0
 *   offsets    [B + 1] int64, image b owns rows offsets[b] .. offsets[b+1]-1 (device)
 *   thr        window half-width in radians (compared in fp32, utils/img2refmap.py:26-27)
 *   min_points cells with fewer members are empty (:28)
 *   reduce_mode 0 = lower median by channel sum (the reference, :30-34), 1 = mean in ascending pixel order (additive)
 *   refmap     [B, res, res, C] fp32, zeros where empty;  refmask [B, res, res] uint8 (0/1)
 *   counts     [B, res, res] int32 members per cell (may be NULL);  sel_index [B, res, res] int32 image-local index
 *              of the selected pixel, -1 where empty or in mean mode (may be NULL)
 * One call takes at most 2^26 pixels (total_n) -- a (cell, pixel) pair keeps its cell tag above a 26-bit pixel index;
 * larger batches are split by the caller (drmnet_b200/img2refmap.py does).
 *
 * drm_img2refmap_status: after a call on the same workspace and arguments, status[0] = flags (bit 0: the pair buffer
 *   overflowed -- cannot happen while workspace_bytes is the value drm_img2refmap_workspace_bytes returns; the outputs
 *   are not to be used if it is set), status[1] = cells that took the warp-per-cell path.  Synchronises the stream.
 *
 * drm_img2refmap_dense: the same scatter of B dense images of H x W pixels under a mask, read in place -- no compaction,
 *   no host read.  Bit for bit the outputs of drm_img2refmap on the compacted pixels (the masked pixels of each image in
 *   row-major order, offsets = running sums of the mask), except sel_index:
 *   colors     fp32, channel c of pixel (b, y, x) at colors[b*s[0] + y*s[1] + x*s[2] + c*s[3]], s = colors_strides
 *              (elements, each >= 0: [B,H,W,C] and [B,C,H,W] views alike), C in 1..4 (device)
 *   normals    fp32, component k of the normal likewise through normals_strides (device)
 *   mask       [B, H, W] uint8, contiguous, nonzero = the pixel takes part (device); NULL = every pixel
 *   sel_index  [B, res, res] int32 dense image-local index y*W + x of the selected pixel, -1 where empty or in mean mode
 *   The other arguments and outputs are those of drm_img2refmap.  One call takes at most 2^26 pixels counted densely
 *   (B*H*W, masked or not).  Null pointers, non-positive sizes, C outside 1..4, a negative stride and B*H*W > 2^26 are
 *   refused (DRM_EINVAL), and a workspace below drm_img2refmap_dense_workspace_bytes (DRM_EWORKSPACE), before any CUDA
 *   call; drm_last_error names the value.  The workspace is that of drm_img2refmap at total_n = B*H*W, so
 *   drm_img2refmap_status(workspace, B*H*W, B, res, thr, ...) reads its status words.
 *   drm_img2refmap_dense_workspace_bytes returns 0 for sizes the entry refuses.
 * ------------------------------------------------------------------------------------------------------------- */
size_t drm_img2refmap_workspace_bytes(int64_t total_n, int B, int res, float thr);

int drm_img2refmap(const float* colors, const float* normals_or_thetaphi, int input_is_thetaphi,
                   const int64_t* offsets, int64_t total_n, int B, int C, int res, float thr, int min_points,
                   int reduce_mode, float* refmap, uint8_t* refmask, int32_t* counts, int32_t* sel_index,
                   void* workspace, size_t workspace_bytes, void* cuda_stream);

int drm_img2refmap_status(const void* workspace, int64_t total_n, int B, int res, float thr, int32_t* status /* [2] */,
                          void* cuda_stream);

size_t drm_img2refmap_dense_workspace_bytes(int B, int H, int W, int res, float thr);

int drm_img2refmap_dense(const float* colors, const int64_t colors_strides[4], /* b, y, x, c in elements */
                         const float* normals, const int64_t normals_strides[4],
                         const uint8_t* mask /* [B,H,W] contiguous 0/1, NULL = every pixel */,
                         int B, int H, int W, int C, int res, float thr, int min_points, int reduce_mode,
                         float* refmap, uint8_t* refmask, int32_t* counts, int32_t* sel_index,
                         void* workspace, size_t workspace_bytes, void* cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Callers either side of the render (SURVEY 8f N1, N2).
 *
 * drm_refmap_postprocess: in/out [G, N, 3, res, res] fp32 (stack 0 = LrK).  target > 0: every stack of sample n is
 *   multiplied by target / geometric-mean luminance of LrK[n] over L > 0 (models/drmnet.py:610-617; 0.12 in the shipped
 *   configs), scale_out [N] receives the factor (may be NULL).  transform 1 applies log10(x + 0.1) + 1
 *   (dataset/basedataset.py:52-53), 0 none.  in may equal out.
 * drm_mirmap2envmap: mirror refmap [B, C, H, W] -> lat-long envmap [B, C, OH, OW] with the defaults of
 *   utils/transform.py:106-144 (view (0,0,1), bilinear, border); basis [C, H, W] (may be NULL) divides the refmap first
 *   (DRMNet.r0toenvmap, models/drmnet.py:939-940).
 * ------------------------------------------------------------------------------------------------------------- */
int drm_refmap_postprocess(const float* in, int G, int N, int res, float target, int transform,
                           float* scale_out, float* out, void* cuda_stream);

int drm_mirmap2envmap(const float* mirmap, const float* basis, int B, int C, int H, int W, int OH, int OW,
                      float* out, void* cuda_stream);

/* N3: colors[p, :] = bilinear lookup of refmap[b] (refmap [B, C, H, W]) at the (theta, phi) of normals[p] for the pixels
 * p of image b (offsets [B+1] int64) -- refmap2refimg_torch (utils/transform.py:170-198) for arbitrary normal lists.
 * Dense normal maps go to drm_refmap_lookup_dense without compaction. */
int drm_refmap_lookup(const float* refmap, const float* normals, const int64_t* offsets, int64_t total_n,
                      int B, int C, int H, int W, float* colors, void* cuda_stream);

/* N3 on dense normal maps, read in place -- no compaction, no host read: every pixel (b, y, x) of B images of H x W
 * pixels whose mask byte is nonzero is shaded with the arithmetic of drm_refmap_lookup (bit for bit the colours it gives
 * for the compacted pixels), every other pixel is set to 0 in every channel.
 *   refmap   [B, C, Hr, Wr] fp32, contiguous (device)
 *   normals  fp32, component k of the normal of pixel (b, y, x) at normals[b*s[0] + y*s[1] + x*s[2] + k*s[3]],
 *            s = normals_strides (elements, each >= 0: [B,H,W,3] and [B,3,H,W] views alike) (device)
 *   mask     [B, H, W] uint8, contiguous, nonzero = shade the pixel (device); NULL = every pixel
 *   out      fp32, channel c of pixel (b, y, x) at out[b*o[0] + y*o[1] + x*o[2] + c*o[3]], o = out_strides (each >= 0),
 *            C in 1..4 (device)
 * Null pointers, non-positive sizes, C outside 1..4, H*W >= 2^31 and a negative stride are refused (DRM_EINVAL) before
 * any CUDA call; drm_last_error names the value. */
int drm_refmap_lookup_dense(const float* refmap, int Hr, int Wr, const float* normals,
                            const int64_t normals_strides[4], /* b, y, x, k in elements */
                            const uint8_t* mask, int B, int H, int W, int C, float* out,
                            const int64_t out_strides[4] /* b, y, x, c in elements */, void* cuda_stream);

/* N4: ObsNet conditioning transform `0p1tom1p1_normalizedLogarithmic_lowerbound<lb>` with dynamic normalisation under a
 * mask (dataset/basedataset.py:56-76, models/obsnet.py:224,370): x [B, C, H, W], mask [B, H, W] float 0/1;
 * log10min_out / log10max_out [B] receive the per-sample parameters (may be NULL). */
int drm_normalized_log(const float* x, const float* mask, int B, int C, int H, int W, float lowerbound,
                       float* out, float* log10min_out, float* log10max_out, void* cuda_stream);

/* N4: ObsNet conditioning (models/obsnet.py:672-691; the training path :368-371 is the noise-free case): the transform
 * above of raw_refmap [B, C, H, W] under raw_refmask [B, H, W] (float 0/1), then, in the reference's order,
 *   cond = t(raw) * mask;  cond = noisy_observe * observe_noise + cond (if noisy_observe > 0);
 *   cond += (1 - mask) * padding_noise (padding_mode "noise"; NULL = "zeros").
 * The noise tensors [B, C, H, W] are drawn by the caller (torch.randn_like in the reference). */
int drm_obsnet_condition(const float* raw_refmap, const float* raw_refmask, int B, int C, int H, int W,
                         float lowerbound, float noisy_observe, const float* observe_noise, const float* padding_noise,
                         float* cond, float* log10min_out, float* log10max_out, void* cuda_stream);

/* N4: the same transform with the parameters of an earlier dynamic call (dynamic_normalize=False,
 * dataset/basedataset.py:68-72; LrK at models/obsnet.py:371), inverse = 0; or BaseDataset.rescale (:98-110), inverse = 1:
 * 10 ^ min((x + 1) / 2 * (max - min) + min, clamp_before_exp) (clamp_before_exp 0 = no clamp). */
int drm_normalized_log_apply(const float* x, const float* log10min, const float* log10max, int B, int C, int H, int W,
                             float lowerbound, int inverse, float clamp_before_exp, float* out, void* cuda_stream);

/* angles only: [n,3] normals -> [n,2] (theta, phi), the arithmetic of utils/transform.py:84-89 at img2refmap.py:20 */
int drm_normals_to_thetaphi(const float* normals, int64_t n, float* thetaphi, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* DRMRENDER_H */
