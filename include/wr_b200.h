/*
 * wr_b200.h -- C ABI of libwr_b200.so: the B200 (sm_100a) geometry path of WorldRenderer.
 *
 * Every entry point takes plain device pointers, sizes and a cudaStream_t passed as void*.
 * All buffers are owned by the caller; the context owns only scratch (snapped vertices, the
 * packed depth/id buffer, triangle queues).  Calls are asynchronous with respect to the host and
 * ordered on `stream`; nothing in here synchronises the device except scratch growth.
 * Return value: WR_OK (0) or a negative wr_status; wr_status_string() names it.
 *
 * What each entry point replaces in the reference (paths relative to
 * mvadapter/utils/mesh_utils/ of Tengpaz/WorldRenderer):
 *
 *   wr_ctx_create / wr_ctx_destroy   dr.RasterizeCudaContext / RasterizeGLContext   render.py:31-37
 *   wr_rasterize                     dr.rasterize      render.py:39-62  (call sites render.py:241, uv.py:40)
 *   wr_interpolate                   dr.interpolate    render.py:64-81  (render.py:244,261,275,281; uv.py:43)
 *   wr_texture                       dr.texture        render.py:83-120 (render.py:267)
 *   wr_vertex_normals                TexturedMesh._compute_vertex_normal            mesh.py:85-119
 *   wr_vertex_tangents               TexturedMesh._compute_tangent                  mesh.py:121-167
 *   wr_tangent_space_normals         view normal maps -> UV tangent space, the inline block of
 *                                    mvadapter/test/utils/pipeline_texture.py:358-396
 *   wr_render                        render() fused: clip transform utils.py:127-129, rasterize,
 *                                    interpolate pos/normal/uv, view depth utils.py:132-139,
 *                                    background fill + depth normalisers render.py:164-217,247-258,
 *                                    texture fetch render.py:260-269, normal normalise render.py:275-277
 *   wr_view_prep                     uv_render_geometry view side: camera-space normal + aoi_cos
 *                                    uv.py:108-119, Sobel + max-pool depth gradient uv.py:122-141
 *   wr_view_prep_sets                (new) the fused bake's view prep for up to four image sets of one rig
 *   wr_uv_unproject                  texel side of uv_render_geometry uv.py:87-90,143-169,
 *                                    uv_render_attr uv.py:193-222, SimpleUVValidityStrategy
 *                                    uv.py:248-298, ExponentialBlend uv.py:317-348, the view sum of
 *                                    uv_blend uv.py:411,421-423
 *   wr_uv_reduce_finalize_p2p        (new) the bake's exchange step fused with finalisation over NVLink peer memory
 *   wr_grid_sample                   F.grid_sample as used by uv_render_attr uv.py:200-218 (operator form)
 *   wr_uv_finalize                   hard stitch with the existing texture uv.py:452-455 (after the
 *                                    optional multi-GPU all-reduce of the accumulators)
 *   wr_view_scores                   SmartPainter's view scoring loop smart_paint.py:118-158
 *   wr_poisson_blend                 PoissonBlendingSolver.__call__ blend.py:214-324 (Jacobi kernel blend.py:60-100)
 *   wr_poisson_band_step             (new) wr_poisson_blend split into row bands across the GPUs of a multi-GPU bake
 *   wr_uv_padding / wr_inpaint_u8    uv_padding uv.py:373-382 -> inpaint_cvc cv_ops.py:11-35 (cvcuda.inpaint)
 *   wr_uv_padding_sets               (new) wr_uv_padding of up to four 3-channel atlases against one mask
 *
 * The raster contract (snap, fill rule, depth key, tie break) is DESIGN.md section 3.
 */
#ifndef WR_B200_H
#define WR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wr_ctx wr_ctx;

typedef enum wr_status {
    WR_OK = 0,
    WR_ERR_INVALID_ARGUMENT = -1,
    WR_ERR_OUT_OF_MEMORY = -2,
    WR_ERR_CUDA = -3,
    WR_ERR_NO_DEVICE = -4,
    WR_ERR_UNSUPPORTED = -5
} wr_status;

const char *wr_status_string(int status);
/* last CUDA error text recorded by this context (empty string if none) */
const char *wr_ctx_last_error(const wr_ctx *ctx);
/* Version of this header's ABI (struct layouts included).  wr_version() returns the value the LIBRARY was built with:
 * a caller compiled against another header must not go on (its argument structs have a different layout). */
#define WR_B200_ABI_VERSION 105
int wr_version(void);

/* One context per (device, stream in flight).  Not thread-safe, like the reference's contexts. */
int wr_ctx_create(int device, wr_ctx **out);
/* Waits for the device to finish the work in flight (kernels of the context's last calls may still read its scratch),
 * then frees the scratch. */
void wr_ctx_destroy(wr_ctx *ctx);
/* bytes of device scratch currently held */
uint64_t wr_ctx_scratch_bytes(const wr_ctx *ctx);

/*
 * Measurement aid (no reference counterpart): with profiling enabled every entry point records a
 * CUDA event on its launch stream before each of its kernels.  wr_ctx_profile_read waits for the last
 * call's final event and returns the number of stages of that call, writing their durations (ms).
 */
int wr_ctx_profile(wr_ctx *ctx, int enable);
int wr_ctx_profile_read(wr_ctx *ctx, float *stage_ms, int capacity);
const char *wr_ctx_profile_stage_name(const wr_ctx *ctx, int i);

/*
 * dr.rasterize.  pos: [B,V,4] f32 clip space when pos_batched != 0 (instanced mode), else [V,4]
 * shared by all B views.  tri: [F,3] i32.  tri_ranges: NULL, or HOST int32 [B,2] (start, count)
 * into tri (range mode; ids stay indices into tri).  rast: [B,H,W,4] f32 = (u, v, z/w, id+1),
 * zeros on background (may be NULL).  tri_id: [B,H,W] i32, -1 on background (may be NULL).
 */
int wr_rasterize(wr_ctx *ctx, const float *pos, int B, int V, int pos_batched, const int32_t *tri, int F,
                 const int32_t *tri_ranges, int H, int W, float *rast, int32_t *tri_id, void *stream);

/* dr.interpolate.  attr: [attr_B,V,A] f32 with attr_B in {1,B}; out: [B,H,W,A]. */
int wr_interpolate(wr_ctx *ctx, const float *attr, int attr_B, int V, int A, const float *rast, int B, int H,
                   int W, const int32_t *tri, int F, float *out, void *stream);

/* dr.texture, 2-D, no mip maps.  filter: 0 nearest, 1 linear.  boundary: 0 wrap, 1 clamp, 2 zero. */
int wr_texture(wr_ctx *ctx, const float *tex, int tex_B, int TH, int TW, int C, const float *uv, int B, int H,
               int W, int filter, int boundary, float *out, void *stream);

/* mesh.py:85-119.  v_nrm: [V,3] out.  The face normals are summed exactly (64-bit fixed point in the context
 * scratch), so the result does not depend on the order of the atomics: identical on every run, rank and GPU. */
int wr_vertex_normals(wr_ctx *ctx, const float *v_pos, int V, const int32_t *tri, int F, float *v_nrm,
                      void *stream);

/* mesh.py:121-167.  tri / tri_tex: [F,3] position and UV faces; v_nrm: [V,3] in; v_tang: [V,3] out.  The per-vertex
 * sum runs through float atomics (sum order varies); a vertex without a face gets NaN, as in the reference. */
int wr_vertex_tangents(wr_ctx *ctx, const float *v_pos, int V, const int32_t *tri, const float *v_tex, int Vt,
                       const int32_t *tri_tex, int F, const float *v_nrm, float *v_tang, void *stream);

/* pipeline_texture.py:358-396.  normal, tangent: [B,H,W,3] rendered maps (render(..., render_tangent=True));
 * image: [B,H,W,3] the views' normal images in [0,1]; view_axis: [B,3] the geometry tangent axis of each view;
 * out: [B,H,W,3] tangent-space normal colours in [0,1]. */
int wr_tangent_space_normals(wr_ctx *ctx, const float *normal, const float *tangent, const float *image,
                             const float *view_axis, int B, int H, int W, float *out, void *stream);

/* depth normalisers of render.py:164-217 */
enum { WR_DEPTH_NONE = 0, WR_DEPTH_CONTROLNET = 1, WR_DEPTH_ZERO123PP = 2, WR_DEPTH_SIMPLE = 3 };

/* element type of wr_render's position, depth, normal, tangent and attribute maps */
enum { WR_DTYPE_F32 = 0, WR_DTYPE_F16 = 1, WR_DTYPE_BF16 = 2 };

typedef struct wr_render_args {
    /* mesh */
    const float *v_pos;       /* [V,3] */
    const int32_t *tri;       /* [F,3] indices into v_pos */
    int V, F;
    const float *v_nrm;       /* [Vn,3] or NULL (no normal map) */
    const int32_t *tri_nrm;   /* [F,3] indices into v_nrm (the stitched faces, render.py:275); NULL = tri */
    int Vn;
    const float *v_tang;      /* [Vn,3] or NULL (no tangent map); indexed by tri_nrm like v_nrm (render.py:281) */
    const float *v_tex;       /* [Vt,2] or NULL (no attr map) */
    const int32_t *tri_tex;   /* [F,3] */
    int Vt;
    const float *texture;     /* [TH,TW,TC] */
    int TH, TW, TC;
    int tex_filter;           /* 0 nearest, 1 linear */
    /* cameras */
    const float *mvp;         /* [B,4,4] row major, 16-byte aligned */
    const float *w2c;         /* [B,4,4] */
    int B, H, W;
    /* depth */
    int depth_mode;           /* WR_DEPTH_* */
    float depth_p0, depth_p1; /* controlnet: far_clip, near_clip - far_clip; simple: scale, offset */
    int depth_clamp;          /* simple: clamp to [0,1] */
    float depth_bg;           /* value written where the mask is false (ignored for WR_DEPTH_NONE) */
    float normal_bg[3];
    float tangent_bg[3];
    float attr_bg;
    /* outputs, each may be NULL; out_pos / out_depth / out_normal / out_tangent / out_attr hold elements of out_dtype
       (declared float: cast a half buffer's pointer) */
    uint8_t *out_mask;        /* [B,H,W] 0/1 */
    float *out_pos;           /* [B,H,W,3] */
    float *out_depth;         /* [B,H,W] */
    float *out_normal;        /* [B,H,W,3] */
    float *out_tangent;       /* [B,H,W,3] normalised interpolated tangents (render.py:280-284) */
    float *out_geo;           /* [B,H,W,4] bake view map (pos.xyz, aoi_cos), aoi_cos as in uv.py:108-119; needs v_nrm, w2c */
    float *out_attr;          /* [B,H,W,TC] */
    int32_t *out_tri_id;      /* [B,H,W] */
    float *out_rast;          /* [B,H,W,4] nvdiffrast layout */
    /* cudaEvent_t or NULL: recorded on the stream once the raster passes are launched, before the shading pass.  A
       caller that renders groups of views on several streams (graph.RenderGraph(view_lanes, stagger)) makes group
       k + 1 wait for it, so that its issue-bound raster passes run next to the store-bound shading pass of group k. */
    void *raster_done_event;
    /* Element type of out_pos / out_depth / out_normal / out_tangent / out_attr; out_geo, out_rast and out_tri_id are
       unaffected.  Values are computed in float32 as for WR_DTYPE_F32 and rounded to nearest even on the store, so a
       16-bit map equals the float32 map converted (NaN payloads aside).  Any other value: WR_ERR_INVALID_ARGUMENT. */
    int out_dtype;            /* WR_DTYPE_F32 = 0 (default), WR_DTYPE_F16, WR_DTYPE_BF16 */
} wr_render_args;

int wr_render(wr_ctx *ctx, const wr_render_args *args, void *stream);

/*
 * View side of the bake.  normal [B,H,W,3], mask [B,H,W] u8, depth [B,H,W] (view depth, background
 * already 1e2 -- uv.py:101-103), position [B,H,W,3], w2c [B,4,4], images [B,H,W,3] or NULL,
 * view_masks [B,H,W] f32 or NULL.  dilation: max-pool kernel size (0 = no depth gradient).
 * Outputs (any may be NULL): aoi_cos [B,H,W]; depth_grad [B,H,W] (odd dilation only);
 * geo_map [B,H,W,4] = (pos.xyz, aoi_cos); attr_map [B,H,W,4] = (rgb, depth_grad);
 * the two packed maps are what wr_uv_unproject gathers from (two 16-byte taps per sample).
 */
int wr_view_prep(wr_ctx *ctx, const float *normal, const uint8_t *mask, const float *depth,
                 const float *position, const float *w2c, const float *images, int B, int H, int W,
                 int dilation, float *aoi_cos, float *depth_grad, float *geo_map, float *attr_map,
                 void *stream);

/*
 * Bake of several image sets of one camera rig in one pass (CameraProjection.project_sets): every set shares the
 * geometry, the validity and the weights, only the colours differ.
 */
#define WR_MAX_BAKE_SETS 4

/*
 * View prep of the fused bake for K image sets (1 <= K <= WR_MAX_BAKE_SETS); the geometry map comes from wr_render's
 * out_geo.  images: HOST array of K device pointers, each [B,H,W,3] f32 (read in place, not copied).
 * attr_map [B,H,W,K,4]: set 0 is (rgb_0, depth_grad) as in wr_view_prep, set k >= 1 is (rgb_k, 0); K = 1 is exactly
 * wr_view_prep's attr_map.  depth_grad [B,H,W] may be NULL.  The same kernel as wr_view_prep.
 */
int wr_view_prep_sets(wr_ctx *ctx, const float *depth, const float *const *images, int K, int B, int H, int W,
                      int dilation, float *depth_grad, float *attr_map, void *stream);

typedef struct wr_unproject_args {
    const float *uv_pos;      /* [Hu,Wu,3] */
    const uint8_t *uv_mask;   /* [Hu,Wu] */
    int Hu, Wu;
    const float *mvp;         /* [Nv,4,4] */
    int Nv, H, W;             /* views and their resolution */
    const float *geo_map;     /* [Nv,H,W,4] from wr_view_prep */
    const float *attr_map;    /* [Nv,H,W,4] (rgb, depth_grad), or [Nv,H,W,attr_sets,4] from wr_view_prep_sets;
                                 NULL => geometry only */
    const float *view_masks;  /* [Nv,H,W] f32 or NULL */
    /* SimpleUVValidityStrategy */
    float pos_error_eps, aoi_cos_thresh, mask_thresh, depth_grad_thresh;
    int use_depth_grad;       /* 0 => depth_grad_thresh ignored (None) */
    int first_view_dominate;
    /* ExponentialBlend (linear normalisation) */
    float alpha;
    const float *view_weight; /* DEVICE [Nv] or NULL */
    /* fused outputs */
    float *accum;             /* [Hu,Wu,5] = (sum w r, sum w g, sum w b, sum w, sum valid); accumulate != 0 adds */
    int accumulate;
    /* optional per-view materialisation (the reference's intermediate tensors), each may be NULL */
    float *uv_pos_ndc;        /* [Nv,Hu,Wu,2] */
    float *uv_pos_proj;       /* [Nv,Hu,Wu,3] */
    float *uv_pos_error;      /* [Nv,Hu,Wu] */
    float *uv_aoi_cos;        /* [Nv,Hu,Wu] */
    float *uv_depth_grad;     /* [Nv,Hu,Wu] */
    float *uv_attr_proj;      /* [Nv,Hu,Wu,3] */
    float *uv_mask_proj;      /* [Nv,Hu,Wu] */
    uint8_t *uv_valid;        /* [Nv,Hu,Wu] */
    float *uv_weight;         /* [Nv,Hu,Wu] normalised blend weight (single-rank meaning only) */
    /* fused finalisation (single GPU): when out_attr != NULL the kernel also stitches, see wr_uv_finalize */
    const float *old_attr;    /* [Hu,Wu,3] existing texture */
    float *out_attr;          /* [Hu,Wu,3] */
    uint8_t *out_valid_any;   /* [Hu,Wu] */
    /* Texel range [tex_lo, tex_hi) of the flattened atlas this call covers; tex_hi == 0 means all of it.  A multi-GPU
       bake unprojects its atlas chunk by chunk so that the exchange of a finished chunk runs under the next one. */
    long long tex_lo, tex_hi;
    /* Image sets in attr_map (0 or 1: one; at most WR_MAX_BAKE_SETS).  Set 0 is stitched through old_attr / out_attr
       above, set k >= 1 through old_attr_more[k - 1] (may be NULL) / out_attr_more[k - 1].  Every set gets the
       validity and weights of set 0 and its own colour sums, in the order of a one-set call: set k's atlas equals a
       one-set call on set k's images bit for bit.  attr_sets > 1 needs out_attr and out_valid_any and supports
       neither accum nor the per-view tensors other than uv_aoi_cos / uv_depth_grad (WR_ERR_UNSUPPORTED). */
    int attr_sets;
    const float *old_attr_more[WR_MAX_BAKE_SETS - 1];
    float *out_attr_more[WR_MAX_BAKE_SETS - 1];
} wr_unproject_args;

int wr_uv_unproject(wr_ctx *ctx, const wr_unproject_args *args, void *stream);

/* out = valid_any ? accum.rgb / max(accum.w, 1e-5) : old ; valid_any = accum.valid > 0 */
int wr_uv_finalize(wr_ctx *ctx, const float *accum, const float *old_attr, int Hu, int Wu, float *out_attr,
                   uint8_t *out_valid_any, void *stream);

/*
 * Multi-GPU bake (no reference counterpart; the reference is single-GPU): fused reduce-scatter + finalise +
 * all-gather of the accumulators through peer-mapped device memory (NVLink / NVSwitch).  accum[r],
 * out_attr[r], out_valid[r] are THIS process's mappings of rank r's buffers ([Hu,Wu,5] f32, [Hu,Wu,3] f32,
 * [Hu,Wu] u8; 16-byte aligned).  The caller must make sure every rank has finished writing its accumulators
 * before the call (device-side barrier) and must not read its atlas before a second barrier after it.
 * Result: identical on every rank; equals wr_uv_finalize of the rank-ordered sum.  Hu*Wu must be a multiple of 4.
 */
#define WR_MAX_P2P_RANKS 16
typedef struct wr_p2p_reduce_args {
    const float *accum[WR_MAX_P2P_RANKS];
    float *out_attr[WR_MAX_P2P_RANKS];
    uint8_t *out_valid[WR_MAX_P2P_RANKS];
    const float *old_attr;    /* local [Hu,Wu,3] or NULL (same texture on every rank) */
    int world, rank, Hu, Wu;
    /* Optional NVSwitch multicast mappings of the same three buffers (all NULL = peer pointers above are used):
       the sum is then computed in the switch (multimem.ld_reduce) and the result broadcast by one store
       (multimem.st).  The in-switch summation order is the hardware's. */
    const float *mc_accum;
    float *mc_attr;
    uint8_t *mc_valid;
    /* Upper bound on the thread blocks of the exchange kernel (0 = 8 per SM, the fastest when it runs alone).  The
       kernel is bound by NVLink, not by the SMs: a pipelined bake (parallel.BakePipeline) runs it with one or two
       blocks per SM so that the next bake's view passes keep the rest of the GPU. */
    int max_blocks;
    /* Texel range [tex_lo, tex_hi) to exchange (each rank owns 1/N of it); tex_hi == 0 means the whole atlas.
       tex_lo must be a multiple of 1024. */
    long long tex_lo, tex_hi;
} wr_p2p_reduce_args;
int wr_uv_reduce_finalize_p2p(wr_ctx *ctx, const wr_p2p_reduce_args *args, void *stream);

/*
 * F.grid_sample(mode="bilinear", padding_mode="zeros", align_corners=False) on channels-last maps
 * (uv.py:143-169, 200-218): map [B,H,W,C], ndc [B,Hs,Ws,2] -> out [B,Hs,Ws,C].
 */
int wr_grid_sample(wr_ctx *ctx, const float *map, int B, int H, int W, int C, const float *ndc, int Hs, int Ws,
                   float *out, void *stream);

/*
 * PoissonBlendingSolver.__call__ (blend.py:214-324).  src (guidance), tgt: [H,W,C] f32, C <= 4; mask: [H,W] u8,
 * non-zero = solve region (the caller applies the > 0.5 threshold of blend.py:229-232; the image border is
 * removed here, blend.py:233-236).  grad_mode: 0 "src", 1 "max", 2 "avg" (blend.py:243-281).  Exactly
 * num_iters Jacobi sweeps x <- (sum of the 4 neighbours + b) / 4 (blend.py:69).  out: [H,W,C] = tgt outside
 * the region, clamp(x, 0, 1) inside (blend.py:317-321); out may alias tgt only if tgt is not needed afterwards
 * (inplace=True) -- it is read by the first and written by the last kernel only.
 */
int wr_poisson_blend(wr_ctx *ctx, const float *src, const uint8_t *mask, const float *tgt, int H, int W, int C,
                     int num_iters, int grad_mode, float *out, void *stream);

/*
 * wr_poisson_blend split across `world` ranks by row bands (no reference counterpart).  The solve's 112 x 48 output
 * tiles are dealt out by tile rows: rank r owns tile rows shard_bounds(ceil(H / 48), world)[r] (parallel.py), so the
 * first ceil(H / 48) % world bands are one tile row taller and, with fewer tile rows than ranks, the last ranks own
 * none.  Every rank holds the whole src / mask / tgt.  Each point gets the float operations of wr_poisson_blend in
 * the same order: every rank's output equals wr_poisson_blend's, bit for bit.
 *
 * wr_poisson_band_layout reports the sizes of this rank's planes (0 for an empty band), the number of sweep launches
 * S = ceil(num_iters / 8) and the image rows [row_lo, row_hi) the rank finishes.  Any output pointer may be NULL.
 *
 * wr_poisson_band_step launches one step of the solve on `stream`:
 *   step 0           setup of the local planes (no peer access);
 *   step 1 .. S      8 Jacobi sweeps of the band (fewer in the last one); from step 2 on, first the 8 halo rows
 *                    above and below the band are pulled from the neighbouring ranks' iterate plane written by
 *                    their previous step (16-byte peer loads);
 *   step S + 1       finish: the band's rows of the result are stored into every rank's output (peer stores).
 * The caller puts a device-side barrier across the ranks after every step from 1 to S + 1, and after step 0 when
 * S == 0: a step may only read what the neighbours wrote before the last barrier, and a rank may read its output
 * after the barrier behind step S + 1.  No kernel waits on another rank.  A rank whose band is empty launches
 * nothing but must still join every barrier.
 */
typedef struct wr_poisson_band_args {
    const float *src;               /* [H,W,C] guidance, local */
    const uint8_t *mask;            /* [H,W] solve region, non-zero = inside (as in wr_poisson_blend), local */
    const float *tgt;               /* [H,W,C], local */
    int H, W, C;                    /* C <= 4 */
    int num_iters, grad_mode;       /* as in wr_poisson_blend */
    int world, rank;                /* world <= WR_MAX_P2P_RANKS */
    float *xa[WR_MAX_P2P_RANKS];    /* this process's mappings of rank r's two iterate planes (plane_bytes each, */
    float *xb[WR_MAX_P2P_RANKS];    /* 16-byte aligned); only the own rank's and the neighbours' are read */
    float *out[WR_MAX_P2P_RANKS];   /* rank r's output [H,W,C] */
    float *b;                       /* local right-hand side plane (plane_bytes, 16-byte aligned) */
    uint8_t *m;                     /* local region plane (mask_bytes, 4-byte aligned) */
    int step;                       /* 0 .. S + 1 */
} wr_poisson_band_args;
int wr_poisson_band_layout(int H, int W, int C, int world, int rank, int num_iters, uint64_t *plane_bytes,
                           uint64_t *mask_bytes, int *steps, int *row_lo, int *row_hi);
int wr_poisson_band_step(wr_ctx *ctx, const wr_poisson_band_args *args, void *stream);

/*
 * Seam fill standing in for cvcuda.inpaint(image, mask, radius) (cv_ops.py:32; third-party operator, absent):
 * pixels with mask != 0 are replaced by an inverse-square-distance average of the known pixels within `radius`
 * of their nearest known pixel (DESIGN.md section 4b); known pixels are copied.  img, out: [H,W,C] u8, C <= 4.
 */
int wr_inpaint_u8(wr_ctx *ctx, const uint8_t *img, const uint8_t *mask, int H, int W, int C, int radius,
                  uint8_t *out, void *stream);
/*
 * uv_padding (uv.py:373-382) in one call: attr [H,W,C] f32 is clamped to [0,1] and quantised as (x * 255)
 * truncated to u8 (cv_ops.py:23-24), texels with inside_mask == 0 are filled as in wr_inpaint_u8, and the result is
 * returned as u8 / 255 (cv_ops.py:35) -- known texels come back quantised, like in the reference.
 */
int wr_uv_padding(wr_ctx *ctx, const float *attr, const uint8_t *inside_mask, int H, int W, int C, int radius,
                  float *out, void *stream);
/*
 * wr_uv_padding of K atlases against one mask (1 <= K <= WR_MAX_BAKE_SETS): attr, out are HOST arrays of K device
 * pointers to [H,W,3] f32.  One jump flood serves all K; out[k] equals wr_uv_padding(attr[k], C = 3) bit for bit.
 */
int wr_uv_padding_sets(wr_ctx *ctx, const float *const *attr, const uint8_t *inside_mask, int H, int W, int K,
                       int radius, float *const *out, void *stream);

/*
 * View scoring of SmartPainter (smart_paint.py:118-158).  attr: [B,H,W,C] f32 (channel 0 = the rendered score map),
 * geo: [B,H,W,4] f32 from wr_render's out_geo (w = angle-of-incidence cosine, smart_paint.py:118-137).  Per view:
 * count = #{attr < lo and aoi > aoi_min}, fsum = sum over {attr > lo and aoi > aoi_min} of max(aoi - attr - margin, 0)
 * (the reference uses lo 1e-3, aoi_min 0.1, margin 0.3 and score = (count + fsum) / (H W)).  count: [B] i32,
 * fsum: [B] f32 (fixed summation order, deterministic).
 */
int wr_view_scores(wr_ctx *ctx, const float *attr, int C, const float *geo, int B, int H, int W, float lo,
                   float aoi_min, float margin, int32_t *count, float *fsum, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WR_B200_H */
