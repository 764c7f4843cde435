// Texture unprojection (UV bake).  Reference: uv.py:72-184 (uv_render_geometry), uv.py:193-222
// (uv_render_attr), uv.py:248-348 (validity + exponential blend), uv.py:385-468 (uv_blend, non-Poisson
// branch), driven by projection.py:54-204.  The reference materialises ~10 [Nv,Huv,Wuv,*] tensors; here
// one kernel walks the views per texel and keeps everything in registers.
//
//   k_view_prep        per view pixel (32x8 tiles, shared memory): camera-space normal -> aoi_cos, zero-padded
//                      Sobel magnitude, separable d x d max-pool; packs two float4 maps
//                      geo = (pos.xyz, aoi_cos), attr = (rgb, depth_grad) so that a bilinear sample is
//                      4 taps x 2 x 16-byte loads instead of 4 taps x (12 + 4 + 4 + 12) bytes
//   k_uv_unproject     per texel: project into every view, gather, validity, weight, accumulate
//   k_uv_finalize      stitch with the existing texture (after the optional all-reduce)
#include <cuda.h>           // CUtensorMap and its enums only: the encoder is fetched through cudaGetDriverEntryPoint (no -lcuda)
#include <cudaTypedefs.h>   // PFN_cuTensorMapEncodeTiled

#include "common.cuh"

namespace {

// ---- TMA: the depth tile of k_view_prep (32 x 32 outputs + halo) is ONE cp.async.bulk.tensor load whose out-of-
// bounds elements arrive as zeros -- which is exactly conv2d's zero padding, so the tile needs no bounds test.
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the async proxy (TMA) must see the initialised barrier
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned phase)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)), "r"(phase)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *map, int c0, int c1, int c2, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_addr(dst)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_addr(bar))
                 : "memory");
}

// View side of the bake in one pass.  A 32x32 output tile per 256-thread block; the depth tile (halo pad+1, zeros
// outside the image = conv2d zero padding), the Sobel magnitude (halo pad, -inf outside the image =
// max_pool2d padding) and the row maxima live in shared memory, so a pixel costs ~3 global loads instead
// of the 9 + d*d of the two-kernel form (measured 102 us -> see profiles/README.md on config C).
constexpr int kPrepTW = 32, kPrepTH = 32;  // output tile per block
constexpr int kPrepBH = 8;                 // block = 32 x 8 threads, four output rows per thread

// Maximum of n values STRIDE apart (one direction of the separable max-pool).  The reference's default window
// (depth_grad_dilation = 5, projection.py:77) is unrolled: five loads and two three-input maxima instead of a counted
// loop of load / max / increment / compare / branch -- a sixth of this issue-bound kernel's instructions.  The maximum
// does not depend on the order (the values are >= 0 or -inf, never -0; fmaxf drops a NaN whichever way round).
template <int STRIDE>
__device__ __forceinline__ float window_max(const float *p, int n)
{
    if (n == 5)
        return fmaxf(fmaxf(fmaxf(p[0], p[STRIDE]), p[2 * STRIDE]), fmaxf(p[3 * STRIDE], p[4 * STRIDE]));
    float m = p[0];
    for (int k = 1; k < n; ++k) m = fmaxf(m, p[k * STRIDE]);
    return m;
}

__global__ void __launch_bounds__(kPrepTW * kPrepBH) k_view_prep(const float *normal, const uint8_t *mask,
                                                                const float *depth, const float *position,
                                                                const float *w2c, const float *images, int H, int W,
                                                                int dilation, float *aoi_out, float *depth_grad,
                                                                float *geo_map, float *attr_map,
                                                                const __grid_constant__ CUtensorMap depth_map, int use_tma)
{
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long s_bar;
    wr_pdl_wait();   // dependent launch behind the shading kernel of the view pass (or whatever precedes it)
    wr_pdl_trigger();
    const int pad = dilation / 2;              // max-pool halo
    const int hd = pad + 1;                    // depth halo (Sobel needs one more ring)
    const int dh = kPrepTH + 2 * hd;
    // The TMA box starts at a column that is a multiple of 4 (the innermost coordinate of a bulk tensor load must be
    // 16-byte aligned -- measured: x = -3 or 61 is an illegal instruction, -4 works; rows are free) and is a whole
    // number of 16-byte units wide: `lead` columns left of the tile instead of hd, row pitch dw.
    const int lead = use_tma ? ((hd + 3) & ~3) : hd;
    const int dw = use_tma ? ((lead + kPrepTW + hd + 3) & ~3) : kPrepTW + 2 * hd;
    const int gw = kPrepTW + 2 * pad, gh = kPrepTH + 2 * pad;
    float *s_box = smem;                       // [dh][dw] as loaded
    float *s_d = s_box + (lead - hd);          // logical tile: column 0 = image column x0 - hd
    float *s_g = s_box + dh * dw;              // [gh][gw]
    float *s_r = s_g + gh * gw;                // [gh][kPrepTW] row maxima
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * kPrepTW, y0 = blockIdx.y * kPrepTH;
    if (dilation > 0) {
        const float *dv = depth + (size_t)b * H * W;
        // The tiles are 32 + 2 * halo columns wide.  Rows go by threadIdx.y and the first 32 columns by threadIdx.x
        // (no integer division); the few halo columns beyond 32 are walked as one flat list by the whole block, so
        // that no pass runs with only a handful of lanes.
        const int tid = threadIdx.y * kPrepTW + threadIdx.x;
        if (use_tma) {
            // one bulk tensor load of the [dh][dw] box at (x0 - hd, y0 - hd, b); elements outside the image are
            // zero-filled by the hardware
            if (tid == 0) mbar_init(&s_bar, 1);
            __syncthreads();
            if (tid == 0) {
                mbar_expect_tx(&s_bar, (unsigned)(dh * dw * sizeof(float)));
                tma_load_3d(s_box, &depth_map, x0 - lead, y0 - hd, b, &s_bar);
            }
            mbar_wait(&s_bar, 0);
        } else {
            auto load_depth = [&](int ry, int rx) {
                const int yy = y0 - hd + ry, xx = x0 - hd + rx;
                s_d[ry * dw + rx] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(dv + (size_t)yy * W + xx) : 0.0f;
            };
            for (int ry = threadIdx.y; ry < dh; ry += kPrepBH) load_depth(ry, threadIdx.x);
            {
                const int extra = dw - kPrepTW;
                for (int e = tid; e < extra * dh; e += kPrepTW * kPrepBH) load_depth(e / extra, kPrepTW + e % extra);
            }
            __syncthreads();
        }
        auto sobel = [&](int gy_, int gx_) {
            const int yy = y0 - pad + gy_, xx = x0 - pad + gx_;
            float g = -INFINITY;
            if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
                const float *c = s_d + (gy_ + 1) * dw + (gx_ + 1);  // centre of the 3x3 window in the depth tile
                const float s00 = c[-dw - 1], s01 = c[-dw], s02 = c[-dw + 1];
                const float s10 = c[-1], s12 = c[1];
                const float s20 = c[dw - 1], s21 = c[dw], s22 = c[dw + 1];
                const float gx = ((((s00 - s02) + 2.0f * s10) - 2.0f * s12) + s20) - s22;
                const float gy = ((((s00 + 2.0f * s01) + s02) - s20) - 2.0f * s21) - s22;
                g = wr_sqrt_z(gx * gx + gy * gy);   // flat depth: gradient exactly 0
            }
            s_g[gy_ * gw + gx_] = g;
        };
        for (int gy_ = threadIdx.y; gy_ < gh; gy_ += kPrepBH) sobel(gy_, threadIdx.x);
        {
            const int extra = gw - kPrepTW;
            for (int e = tid; e < extra * gh; e += kPrepTW * kPrepBH) sobel(e / extra, kPrepTW + e % extra);
        }
        __syncthreads();
        for (int ry = threadIdx.y; ry < gh; ry += kPrepBH) {  // row maxima: one output column per thread
            const float *row = s_g + ry * gw + threadIdx.x;
            s_r[ry * kPrepTW + threadIdx.x] = window_max<1>(row, dilation);
        }
        __syncthreads();
    }
    const int c = x0 + threadIdx.x;
    if (c >= W) return;
#pragma unroll
    for (int j = 0; j < kPrepTH / kPrepBH; ++j) {
        const int ty = threadIdx.y + j * kPrepBH;  // row inside the tile
        const int r = y0 + ty;
        if (r >= H) break;
        const size_t o = ((size_t)b * H + r) * W + c;
        float dg = 0.0f;
        if (dilation > 0) {
            const float *col = s_r + ty * kPrepTW + threadIdx.x;
            dg = window_max<kPrepTW>(col, dilation);
            if (depth_grad) depth_grad[o] = dg;
        }
        if (attr_map) {
            float ir = 0.f, ig = 0.f, ib = 0.f;
            if (images) { const float *im = images + 3 * o; ir = __ldg(im); ig = __ldg(im + 1); ib = __ldg(im + 2); }
            reinterpret_cast<float4 *>(attr_map)[o] = make_float4(ir, ig, ib, dg);
        }
        if (!normal) continue;  // geometry half already produced by wr_render (out_geo)
        const float *n = normal + 3 * o;
        const float nx = __ldg(n), ny = __ldg(n + 1), nz = __ldg(n + 2);
        float aoi;
        if (__ldg(mask + o)) {
            const float *R = w2c + 16 * b;
            const float x = (R[0] * nx + R[1] * ny) + R[2] * nz;
            const float y = (R[4] * nx + R[5] * ny) + R[6] * nz;
            const float z = (R[8] * nx + R[9] * ny) + R[10] * nz;
            const float ln = sqrtf((x * x + y * y) + z * z);
            aoi = z / fmaxf(ln, 1e-12f);
        } else {
            aoi = nz;  // uv.py:112: background keeps the render's normal (normal_background)
        }
        aoi = fminf(fmaxf(aoi, 0.0f), 1.0f);
        if (aoi_out) aoi_out[o] = aoi;
        if (geo_map) {
            const float *p = position + 3 * o;
            reinterpret_cast<float4 *>(geo_map)[o] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), aoi);
        }
    }
}

// F.grid_sample(mode="bilinear", padding_mode="zeros", align_corners=False) tap set (uv.py:143-169)
struct Bilinear {
    int x0, y0;
    float w00, w10, w01, w11;
    bool ok;
};

__device__ __forceinline__ Bilinear make_bilinear(float gx, float gy, int W, int H)
{
    Bilinear t;
    const float ix = ((gx + 1.0f) * (float)W - 1.0f) / 2.0f;
    const float iy = ((gy + 1.0f) * (float)H - 1.0f) / 2.0f;
    t.ok = isfinite(ix) && isfinite(iy);
    const float x0f = floorf(ix), y0f = floorf(iy);
    const float tx = ix - x0f, ty = iy - y0f;
    t.x0 = t.ok ? (int)fminf(fmaxf(x0f, -1e9f), 1e9f) : -2;
    t.y0 = t.ok ? (int)fminf(fmaxf(y0f, -1e9f), 1e9f) : -2;
    t.w00 = (1.0f - tx) * (1.0f - ty);
    t.w10 = tx * (1.0f - ty);
    t.w01 = (1.0f - tx) * ty;
    t.w11 = tx * ty;
    return t;
}

__device__ __forceinline__ void tap4(float4 &acc, const float4 v, float w)
{
    acc.x = acc.x + v.x * w; acc.y = acc.y + v.y * w; acc.z = acc.z + v.z * w; acc.w = acc.w + v.w * w;
}

// Taps are added in the order (0,0), (1,0), (0,1), (1,1); a tap outside the map adds nothing (zero padding).
__device__ __forceinline__ float4 sample4(const float4 *map, const Bilinear &t, int W, int H)
{
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!t.ok) return acc;
    if (t.x0 >= 0 && t.y0 >= 0 && t.x0 + 1 < W && t.y0 + 1 < H) {  // interior: one base offset, no per-tap tests
        const float4 *p = map + ((unsigned)t.y0 * (unsigned)W + (unsigned)t.x0);
        const float4 v00 = __ldg(p), v10 = __ldg(p + 1), v01 = __ldg(p + W), v11 = __ldg(p + W + 1);
        tap4(acc, v00, t.w00); tap4(acc, v10, t.w10); tap4(acc, v01, t.w01); tap4(acc, v11, t.w11);
        return acc;
    }
    const int xs[4] = { t.x0, t.x0 + 1, t.x0, t.x0 + 1 };
    const int ys[4] = { t.y0, t.y0, t.y0 + 1, t.y0 + 1 };
    const float ws[4] = { t.w00, t.w10, t.w01, t.w11 };
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (xs[k] >= 0 && xs[k] < W && ys[k] >= 0 && ys[k] < H) tap4(acc, __ldg(map + (size_t)ys[k] * W + xs[k]), ws[k]);
    return acc;
}

__device__ __forceinline__ float sample1(const float *map, const Bilinear &t, int W, int H)
{
    float acc = 0.f;
    if (!t.ok) return acc;
    const int xs[4] = { t.x0, t.x0 + 1, t.x0, t.x0 + 1 };
    const int ys[4] = { t.y0, t.y0, t.y0 + 1, t.y0 + 1 };
    const float ws[4] = { t.w00, t.w10, t.w01, t.w11 };
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (xs[k] >= 0 && xs[k] < W && ys[k] >= 0 && ys[k] < H) acc = acc + __ldg(map + (size_t)ys[k] * W + xs[k]) * ws[k];
    return acc;
}

// w^e of the exponential blend (uv.py:328-340).  pow(0, e) is 0 for e > 0 (the common case of an invalid view), and
// the exponents in use are small integers (alpha 3 or 6 with unit view weights): those are plain products, within
// an ulp or two of powf (the weights are compared at 1e-5); anything else goes through powf.
__device__ __forceinline__ float blend_pow(float w, float e)
{
    if (w == 0.0f && e > 0.0f) return 0.0f;
    if (e == 3.0f) return (w * w) * w;
    if (e == 6.0f) { const float c = (w * w) * w; return c * c; }
    if (e == 1.0f) return w;
    if (e == 2.0f) return w * w;
    return powf(w, e);
}

// MATERIALISE: 0 = blend only; 1 = any of the reference's per-view tensors; 2 = only uv_aoi_cos / uv_depth_grad, which
// is what CameraProjection(return_dict=True) asks for (no view-mask tap for invalid texel-views, no pointer tests
// for the other seven tensors).
template <int MATERIALISE>
__global__ void __launch_bounds__(256) k_uv_unproject(wr_unproject_args A)
{
    constexpr bool materialise = MATERIALISE != 0;
    constexpr bool light = MATERIALISE == 2;
    extern __shared__ float s_cam[];  // [Nv,16] mvp, then [Nv] exponent
    wr_pdl_wait();   // dependent launch behind k_view_prep
    wr_pdl_trigger();
    for (int i = threadIdx.x; i < A.Nv * 16; i += blockDim.x) s_cam[i] = A.mvp[i];
    float *s_expo = s_cam + A.Nv * 16;
    for (int i = threadIdx.x; i < A.Nv; i += blockDim.x)
        s_expo[i] = A.view_weight ? A.alpha / A.view_weight[i] : A.alpha;
    // bit v: row 3 of view v's matrix is exactly (0 0 0 1) -- an orthographic view (views beyond 32: general path)
    __shared__ unsigned s_unit_rows;
    if (threadIdx.x < 32) {
        bool unit = false;
        if ((int)threadIdx.x < A.Nv) {
            const float *m = A.mvp + 16 * threadIdx.x + 12;
            unit = m[0] == 0.0f && m[1] == 0.0f && m[2] == 0.0f && m[3] == 1.0f;
        }
        const unsigned bits = __ballot_sync(0xFFFFFFFFu, unit);
        if (threadIdx.x == 0) s_unit_rows = bits;
    }
    __syncthreads();
    unsigned unit_rows = s_unit_rows;

    const long long ntex = (long long)A.Hu * A.Wu;
    const long long o = A.tex_lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= (A.tex_hi ? A.tex_hi : ntex)) return;
    const bool inside = A.uv_mask[o] != 0;
    float sr = 0.f, sg = 0.f, sb = 0.f, sw = 0.f;
    int nvalid = 0;

    if (inside || materialise) {
        const float *up = A.uv_pos + 3 * o;
        const float ux = up[0], uy = up[1], uz = up[2];
        const long long npix = (long long)A.H * A.W;
        bool valid0 = false;
        // a finite texel under a (0 0 0 1) row has w = ((0 x + 0 y) + 0 z) + 1 = 1 exactly (a non-finite one: NaN)
        if (!(isfinite(ux) && isfinite(uy) && isfinite(uz))) unit_rows = 0u;
        for (int v = 0; v < A.Nv; ++v) {
            const float *m = s_cam + 16 * v;
            const float cx = ((m[0] * ux + m[1] * uy) + m[2] * uz) + m[3];
            const float cy = ((m[4] * ux + m[5] * uy) + m[6] * uz) + m[7];
            // uv.py:90, no w > 0 guard.  x / 1 == x exactly: an orthographic view skips the w row and the two IEEE
            // divisions behind a branch that is uniform in practice (a select would still execute them, and a texel
            // outside the charts -- clip x exactly 0 -- sends the whole warp through the division's slow path)
            float gx = cx, gy = cy;
            if (!(v < 32 && ((unit_rows >> v) & 1u))) {
                const float cw = ((m[12] * ux + m[13] * uy) + m[14] * uz) + m[15];
                gx = cx / cw;
                gy = cy / cw;
            }
            const Bilinear t = make_bilinear(gx, gy, A.W, A.H);
            const float4 geo = sample4(reinterpret_cast<const float4 *>(A.geo_map) + v * npix, t, A.W, A.H);
            const float dx = geo.x - ux, dy = geo.y - uy, dz = geo.z - uz;
            const float err = wr_sqrt_z((dx * dx + dy * dy) + dz * dz);
            bool valid = (err < A.pos_error_eps) && (geo.w > A.aoi_cos_thresh) && inside;
            // the colour / depth-gradient taps only matter for a texel that passed the geometry test
            float4 att = make_float4(0.f, 0.f, 0.f, 0.f);
            if (A.attr_map && (valid || materialise))
                att = sample4(reinterpret_cast<const float4 *>(A.attr_map) + v * npix, t, A.W, A.H);
            if (A.use_depth_grad) valid = valid && (att.w < A.depth_grad_thresh);
            float mp = 0.f;
            if (A.view_masks && (valid || (materialise && !light))) {
                mp = sample1(A.view_masks + v * npix, t, A.W, A.H);
                valid = valid && (mp > A.mask_thresh);
            }
            if (A.first_view_dominate) {
                if (v == 0) valid0 = valid;
                else valid = valid && !valid0;
            }
            float wgt = geo.w * (valid ? 1.0f : 0.0f);
            // pow(0, e) is 0 for e > 0 (the common case of an invalid view): skip the call
            wgt = blend_pow(wgt, s_expo[v]);
            sw = sw + wgt;
            sr = sr + att.x * wgt; sg = sg + att.y * wgt; sb = sb + att.z * wgt;
            nvalid += valid ? 1 : 0;
            if (light) {
                const size_t ov = (size_t)v * ntex + o;
                if (A.uv_aoi_cos) A.uv_aoi_cos[ov] = geo.w;
                if (A.uv_depth_grad) A.uv_depth_grad[ov] = att.w;
            } else if (materialise) {
                const size_t ov = (size_t)v * ntex + o;
                if (A.uv_pos_ndc) { A.uv_pos_ndc[2 * ov] = gx; A.uv_pos_ndc[2 * ov + 1] = gy; }
                if (A.uv_pos_proj) { A.uv_pos_proj[3 * ov] = geo.x; A.uv_pos_proj[3 * ov + 1] = geo.y; A.uv_pos_proj[3 * ov + 2] = geo.z; }
                if (A.uv_pos_error) A.uv_pos_error[ov] = err;
                if (A.uv_aoi_cos) A.uv_aoi_cos[ov] = geo.w;
                if (A.uv_depth_grad) A.uv_depth_grad[ov] = att.w;
                if (A.uv_attr_proj) { A.uv_attr_proj[3 * ov] = att.x; A.uv_attr_proj[3 * ov + 1] = att.y; A.uv_attr_proj[3 * ov + 2] = att.z; }
                if (A.uv_mask_proj) A.uv_mask_proj[ov] = mp;
                if (A.uv_valid) A.uv_valid[ov] = valid ? 1 : 0;
                if (A.uv_weight) A.uv_weight[ov] = wgt;
            }
        }
        if (materialise && !light && A.uv_weight) {  // ExponentialBlend "linear": w / clamp(sum w, 1e-5), clamp [0,1]
            const float den = fmaxf(sw, 1e-5f);
            for (int v = 0; v < A.Nv; ++v) {
                const size_t ov = (size_t)v * ntex + o;
                A.uv_weight[ov] = fminf(fmaxf(A.uv_weight[ov] / den, 0.0f), 1.0f);
            }
        }
    }

    if (A.accum) {
        float *a = A.accum + 5 * o;
        if (A.accumulate) { a[0] += sr; a[1] += sg; a[2] += sb; a[3] += sw; a[4] += (float)nvalid; }
        else { a[0] = sr; a[1] = sg; a[2] = sb; a[3] = sw; a[4] = (float)nvalid; }
    }
    if (A.out_attr || A.out_valid_any) {
        const float den = fmaxf(sw, 1e-5f);
        const float va = nvalid > 0 ? 1.0f : 0.0f;
        if (A.out_valid_any) A.out_valid_any[o] = nvalid > 0 ? 1 : 0;
        if (A.out_attr) {
            float o0 = 0.f, o1 = 0.f, o2 = 0.f;
            if (A.old_attr) { o0 = A.old_attr[3 * o]; o1 = A.old_attr[3 * o + 1]; o2 = A.old_attr[3 * o + 2]; }
            // den >= 1e-5 > 0; a texel without a valid view has sums of exactly 0
            A.out_attr[3 * o] = wr_div_zpos(sr, den) * va + o0 * (1.0f - va);
            A.out_attr[3 * o + 1] = wr_div_zpos(sg, den) * va + o1 * (1.0f - va);
            A.out_attr[3 * o + 2] = wr_div_zpos(sb, den) * va + o2 * (1.0f - va);
        }
    }
}

__global__ void __launch_bounds__(256) k_uv_finalize(const float *accum, const float *old_attr, long long ntex,
                                                     float *out_attr, uint8_t *out_valid_any)
{
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= ntex) return;
    const float *a = accum + 5 * o;
    const float den = fmaxf(a[3], 1e-5f);
    const bool any = a[4] > 0.5f;
    const float va = any ? 1.0f : 0.0f;
    if (out_valid_any) out_valid_any[o] = any ? 1 : 0;
    if (out_attr) {
        float o0 = 0.f, o1 = 0.f, o2 = 0.f;
        if (old_attr) { o0 = old_attr[3 * o]; o1 = old_attr[3 * o + 1]; o2 = old_attr[3 * o + 2]; }
        out_attr[3 * o] = wr_div_zpos(a[0], den) * va + o0 * (1.0f - va);
        out_attr[3 * o + 1] = wr_div_zpos(a[1], den) * va + o1 * (1.0f - va);
        out_attr[3 * o + 2] = wr_div_zpos(a[2], den) * va + o2 * (1.0f - va);
    }
}


// Generic F.grid_sample(bilinear, zeros, align_corners=False) for channels-last maps (uv.py:200-218).
__global__ void __launch_bounds__(256) k_grid_sample(const float *map, int H, int W, int C, const float *ndc,
                                                     long long nsamp_view, long long nsamp_total, float *out)
{
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= nsamp_total) return;
    const int b = (int)(o / nsamp_view);
    const float2 g = __ldg(reinterpret_cast<const float2 *>(ndc) + o);
    const Bilinear t = make_bilinear(g.x, g.y, W, H);
    const float *mv = map + (size_t)b * H * W * C;
    float *dst = out + o * C;
    const int xs[4] = { t.x0, t.x0 + 1, t.x0, t.x0 + 1 };
    const int ys[4] = { t.y0, t.y0, t.y0 + 1, t.y0 + 1 };
    const float ws[4] = { t.w00, t.w10, t.w01, t.w11 };
    for (int ch = 0; ch < C; ++ch) {
        float acc = 0.f;
        if (t.ok) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (xs[k] >= 0 && xs[k] < W && ys[k] >= 0 && ys[k] < H)
                    acc = acc + __ldg(mv + ((size_t)ys[k] * W + xs[k]) * C + ch) * ws[k];
        }
        dst[ch] = acc;
    }
}


// Fused reduce-scatter + finalise + all-gather of the bake accumulators over NVLink peer memory (multi-GPU
// bake, DESIGN.md section 8).  Every rank owns a contiguous range of 1024-texel blocks.  For its blocks it
//   1. sums the [.,5] accumulators of ALL ranks with coalesced 16-byte loads straight from peer memory (each
//      texel is summed by exactly one rank, in an order fixed by that rank),
//   2. finalises in shared memory / registers (divide, valid-any, stitch with the old texture), and
//   3. stores the finished texels into EVERY rank's atlas and mask (peer stores).
// One kernel replaces NCCL all-reduce (2 x 20 B per texel over the wire) + finalize; wire traffic per texel
// is 20 B in (reduce-scatter) + 13 B out (all-gather of the result).
constexpr int kP2PTexelsPerBlock = 1024;  // 256 threads x 4 texels

// NR: upper bound on the ranks of this instantiation (2, 4, 8, 16): the NR loads of a chunk are in flight together,
// so the register footprint follows the world size (128 registers at NR = 16 -- two resident blocks would own the
// whole register file of an SM, which matters when the exchange runs under another bake's view passes).
template <int NR>
__global__ void __launch_bounds__(256) k_uv_reduce_finalize_p2p(wr_p2p_reduce_args A, long long ntex, long long blk_lo,
                                                                long long blk_hi)
{
    __shared__ float4 s_sum[kP2PTexelsPerBlock * 5 / 4];  // 1280 float4 = 20 KB
    for (long long blk = blk_lo + blockIdx.x; blk < blk_hi; blk += gridDim.x) {
        const long long t0 = A.tex_lo + blk * kP2PTexelsPerBlock;
        const long long nt = min((long long)kP2PTexelsPerBlock, ntex - t0);  // multiple of 4 (ntex: end of the range)
        const int nchunks = (int)(nt * 5 / 4);
        // per chunk: one 16-byte load from every rank in flight together, starting at the next rank so that the
        // ranks do not all pull from rank 0 at the same moment.  The summation order (rank+1, rank+2, ...) is a
        // fixed function of the owner of the texel, and only the owner computes it: results are reproducible
        // and identical on every rank.
        for (int j = threadIdx.x; j < nchunks; j += blockDim.x) {
            float4 v[NR];
#pragma unroll
            for (int i = 0; i < NR; ++i) {
                if (i < A.world) {
                    int r = A.rank + 1 + i;
                    if (r >= A.world) r -= A.world;
                    v[i] = *(reinterpret_cast<const float4 *>(A.accum[r] + 5 * t0) + j);
                }
            }
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int i = 0; i < NR; ++i)
                if (i < A.world) { acc.x += v[i].x; acc.y += v[i].y; acc.z += v[i].z; acc.w += v[i].w; }
            s_sum[j] = acc;
        }
        __syncthreads();
        const int q = threadIdx.x;  // texels 4q .. 4q+3 of the block
        if (4 * q < nt) {
            const float *sf = reinterpret_cast<const float *>(s_sum) + 20 * q;
            float res[12];
            uchar4 anyv;
            uint8_t *ap = reinterpret_cast<uint8_t *>(&anyv);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float *a = sf + 5 * k;
                const float den = fmaxf(a[3], 1e-5f);
                const bool any = a[4] > 0.5f;
                const float va = any ? 1.0f : 0.0f;
                float o0 = 0.f, o1 = 0.f, o2 = 0.f;
                if (A.old_attr) {
                    const float *op = A.old_attr + 3 * (t0 + 4 * q + k);
                    o0 = op[0]; o1 = op[1]; o2 = op[2];
                }
                res[3 * k] = wr_div_zpos(a[0], den) * va + o0 * (1.0f - va);
                res[3 * k + 1] = wr_div_zpos(a[1], den) * va + o1 * (1.0f - va);
                res[3 * k + 2] = wr_div_zpos(a[2], den) * va + o2 * (1.0f - va);
                ap[k] = any ? 1 : 0;
            }
            const long long t = t0 + 4 * q;
            for (int r = 0; r < A.world; ++r) {
                float4 *d = reinterpret_cast<float4 *>(A.out_attr[r] + 3 * t);
                d[0] = make_float4(res[0], res[1], res[2], res[3]);
                d[1] = make_float4(res[4], res[5], res[6], res[7]);
                d[2] = make_float4(res[8], res[9], res[10], res[11]);
                *reinterpret_cast<uchar4 *>(A.out_valid[r] + t) = anyv;
            }
        }
        __syncthreads();
    }
}


// Same exchange through the NVSwitch multicast window (NVLS): multimem.ld_reduce returns the sum of all ranks'
// accumulators computed IN the switch (each rank pulls 20 B per owned texel instead of 20 B x world), and
// multimem.st writes the finished texels to every rank with one store (13 B out per owned texel instead of
// 13 B x world).
__device__ __forceinline__ float4 multimem_ld_reduce_add_f32x4(const float *mc_addr)
{
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(mc_addr)
                 : "memory");
    return v;
}
__device__ __forceinline__ void multimem_st_f32x4(float *mc_addr, float4 v)
{
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ void multimem_st_f32(float *mc_addr, float v)
{
    asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(mc_addr), "f"(v) : "memory");
}

// T threads per block, 4 T texels per block iteration.  T = 64 with one block per SM (4 K registers and 5 KB of
// shared memory per SM) is what runs: the exchange is bound by the NVSwitch round trips, not by the SMs, and a small
// footprint matters when it runs under another bake's view passes, whose kernels need the whole register file for
// their own occupancy.
template <int T>
__global__ void __launch_bounds__(T) k_uv_reduce_finalize_mc(wr_p2p_reduce_args A, long long ntex, long long blk_lo,
                                                             long long blk_hi)
{
    constexpr int kTexels = 4 * T;
    __shared__ float4 s_sum[kTexels * 5 / 4];
    for (long long blk = blk_lo + blockIdx.x; blk < blk_hi; blk += gridDim.x) {
        const long long t0 = A.tex_lo + blk * kTexels;
        const long long nt = min((long long)kTexels, ntex - t0);   // ntex: end of the range
        const int nchunks = (int)(nt * 5 / 4);
        {   // all five 16-byte reductions of a thread are issued before the first result is consumed
            float4 v[5];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const int j = threadIdx.x + k * T;
                if (j < nchunks) v[k] = multimem_ld_reduce_add_f32x4(A.mc_accum + 5 * t0 + 4 * (long long)j);
            }
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const int j = threadIdx.x + k * T;
                if (j < nchunks) s_sum[j] = v[k];
            }
        }
        __syncthreads();
        const int q = threadIdx.x;
        if (4 * q < nt) {
            const float *sf = reinterpret_cast<const float *>(s_sum) + 20 * q;
            float res[12];
            uint32_t anyw = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float *a = sf + 5 * k;
                const float den = fmaxf(a[3], 1e-5f);
                const bool any = a[4] > 0.5f;
                const float va = any ? 1.0f : 0.0f;
                float o0 = 0.f, o1 = 0.f, o2 = 0.f;
                if (A.old_attr) {
                    const float *op = A.old_attr + 3 * (t0 + 4 * q + k);
                    o0 = op[0]; o1 = op[1]; o2 = op[2];
                }
                res[3 * k] = wr_div_zpos(a[0], den) * va + o0 * (1.0f - va);
                res[3 * k + 1] = wr_div_zpos(a[1], den) * va + o1 * (1.0f - va);
                res[3 * k + 2] = wr_div_zpos(a[2], den) * va + o2 * (1.0f - va);
                anyw |= (any ? 1u : 0u) << (8 * k);
            }
            const long long t = t0 + 4 * q;
            float *d = A.mc_attr + 3 * t;
            multimem_st_f32x4(d, make_float4(res[0], res[1], res[2], res[3]));
            multimem_st_f32x4(d + 4, make_float4(res[4], res[5], res[6], res[7]));
            multimem_st_f32x4(d + 8, make_float4(res[8], res[9], res[10], res[11]));
            multimem_st_f32(reinterpret_cast<float *>(A.mc_valid + t), __uint_as_float(anyw));  // 4 mask bytes, bits preserved
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" int wr_grid_sample(wr_ctx *ctx, const float *map, int B, int H, int W, int C, const float *ndc, int Hs,
                              int Ws, float *out, void *stream_)
{
    if (!ctx || B < 0 || H <= 0 || W <= 0 || C <= 0 || Hs <= 0 || Ws <= 0) return WR_ERR_INVALID_ARGUMENT;
    if (B == 0) return WR_OK;
    if (!map || !ndc || !out) return WR_ERR_INVALID_ARGUMENT;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const long long nv = (long long)Hs * Ws, total = nv * B;
    k_grid_sample<<<wr_div_up(total, 256), 256, 0, stream>>>(map, H, W, C, ndc, nv, total, out);
    WR_CHECK_LAUNCH(ctx, "k_grid_sample");
    return WR_OK;
}

extern "C" int wr_view_prep(wr_ctx *ctx, const float *normal, const uint8_t *mask, const float *depth,
                            const float *position, const float *w2c, const float *images, int B, int H, int W,
                            int dilation, float *aoi_cos, float *depth_grad, float *geo_map, float *attr_map,
                            void *stream_)
{
    if (!ctx || B < 0 || H <= 0 || W <= 0 || dilation < 0) return WR_ERR_INVALID_ARGUMENT;
    if (dilation > 0 && (dilation & 1) == 0) return WR_ERR_UNSUPPORTED;  // even max-pool changes the map size
    if (B == 0) return WR_OK;
    if (normal) {
        if (!mask || !w2c || (geo_map && !position)) return WR_ERR_INVALID_ARGUMENT;
    } else if (aoi_cos || geo_map) {
        return WR_ERR_INVALID_ARGUMENT;
    }
    if (dilation > 0 && !depth) return WR_ERR_INVALID_ARGUMENT;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const int pad = dilation / 2, hd = pad + 1;
    // TMA needs 16-byte aligned rows (W % 4 == 0) and base; otherwise the block loads its tile by hand
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof(tmap));
    const int lead = (hd + 3) & ~3;
    const int boxw = (lead + kPrepTW + hd + 3) & ~3, boxh = kPrepTH + 2 * hd;
    int use_tma = 0;
    if (dilation > 0 && (W & 3) == 0 && (reinterpret_cast<uintptr_t>(depth) & 15u) == 0 && boxw <= 256 && boxh <= 256) {
        static PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
        static bool looked_up = false;
        if (!looked_up) {
            void *fn = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
                q == cudaDriverEntryPointSuccess)
                encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
            else
                cudaGetLastError();
            looked_up = true;
        }
        if (encode) {
            const cuuint64_t gdim[3] = { (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B };
            const cuuint64_t gstride[2] = { (cuuint64_t)W * 4, (cuuint64_t)W * H * 4 };
            const cuuint32_t box[3] = { (cuuint32_t)boxw, (cuuint32_t)boxh, 1 };
            const cuuint32_t estride[3] = { 1, 1, 1 };
            const CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(depth), gdim, gstride, box,
                                      estride, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                      CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            use_tma = r == CUDA_SUCCESS ? 1 : 0;
        }
    }
    const size_t smem = sizeof(float) * ((size_t)boxh * (use_tma ? boxw : kPrepTW + 2 * hd) +
                                         (size_t)(kPrepTH + 2 * pad) * (kPrepTW + 2 * pad) +
                                         (size_t)(kPrepTH + 2 * pad) * kPrepTW);
    if (smem > 48 * 1024) return WR_ERR_UNSUPPORTED;  // dilation > ~29
    const dim3 grid(wr_div_up(W, kPrepTW), wr_div_up(H, kPrepTH), B);
    wr_stage_begin(ctx);
    wr_stage(ctx, stream, "k_view_prep");
    wr_launch_s(k_view_prep, grid, dim3(kPrepTW, kPrepBH), dilation > 0 ? smem : 0, stream, !ctx->profiling, normal, mask,
                depth, position, w2c, images, H, W, dilation, aoi_cos, depth_grad, geo_map, attr_map, tmap, use_tma);
    WR_CHECK_LAUNCH(ctx, "k_view_prep");
    wr_stage(ctx, stream, "end");
    return WR_OK;
}

extern "C" int wr_uv_unproject(wr_ctx *ctx, const wr_unproject_args *args, void *stream_)
{
    if (!ctx || !args) return WR_ERR_INVALID_ARGUMENT;
    const wr_unproject_args &A = *args;
    if (A.Hu <= 0 || A.Wu <= 0 || A.Nv < 0 || A.H <= 0 || A.W <= 0) return WR_ERR_INVALID_ARGUMENT;
    if (!A.uv_pos || !A.uv_mask || (A.Nv > 0 && (!A.mvp || !A.geo_map))) return WR_ERR_INVALID_ARGUMENT;
    if (A.use_depth_grad && !A.attr_map) return WR_ERR_INVALID_ARGUMENT;
    const size_t smem = (size_t)A.Nv * 17 * sizeof(float);
    if (smem > 48 * 1024) return WR_ERR_UNSUPPORTED;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const int materialise = (A.uv_pos_ndc || A.uv_pos_proj || A.uv_pos_error || A.uv_aoi_cos || A.uv_depth_grad ||
                             A.uv_attr_proj || A.uv_mask_proj || A.uv_valid || A.uv_weight) ? 1 : 0;
    const long long ntex = (long long)A.Hu * A.Wu;
    wr_stage_begin(ctx);
    wr_stage(ctx, stream, "k_uv_unproject");
    const bool heavy = A.uv_pos_ndc || A.uv_pos_proj || A.uv_pos_error || A.uv_attr_proj || A.uv_mask_proj || A.uv_valid ||
                       A.uv_weight;
    if (A.tex_lo < 0 || A.tex_hi < 0 || A.tex_hi > ntex || (A.tex_hi && A.tex_lo >= A.tex_hi)) return WR_ERR_INVALID_ARGUMENT;
    const dim3 grid(wr_div_up((A.tex_hi ? A.tex_hi : ntex) - A.tex_lo, 256)), block(256);
    if (heavy) wr_launch_s(k_uv_unproject<1>, grid, block, smem, stream, !ctx->profiling, A);
    else if (materialise) wr_launch_s(k_uv_unproject<2>, grid, block, smem, stream, !ctx->profiling, A);
    else wr_launch_s(k_uv_unproject<0>, grid, block, smem, stream, !ctx->profiling, A);
    WR_CHECK_LAUNCH(ctx, "k_uv_unproject");
    wr_stage(ctx, stream, "end");
    return WR_OK;
}

extern "C" int wr_uv_finalize(wr_ctx *ctx, const float *accum, const float *old_attr, int Hu, int Wu, float *out_attr,
                              uint8_t *out_valid_any, void *stream_)
{
    if (!ctx || !accum || Hu <= 0 || Wu <= 0) return WR_ERR_INVALID_ARGUMENT;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const long long ntex = (long long)Hu * Wu;
    k_uv_finalize<<<wr_div_up(ntex, 256), 256, 0, stream>>>(accum, old_attr, ntex, out_attr, out_valid_any);
    WR_CHECK_LAUNCH(ctx, "k_uv_finalize");
    return WR_OK;
}

extern "C" int wr_uv_reduce_finalize_p2p(wr_ctx *ctx, const wr_p2p_reduce_args *args, void *stream_)
{
    if (!ctx || !args) return WR_ERR_INVALID_ARGUMENT;
    const wr_p2p_reduce_args &A = *args;
    if (A.world < 1 || A.world > WR_MAX_P2P_RANKS || A.rank < 0 || A.rank >= A.world || A.Hu <= 0 || A.Wu <= 0)
        return WR_ERR_INVALID_ARGUMENT;
    const long long natlas = (long long)A.Hu * A.Wu;
    if (natlas % 4 != 0) return WR_ERR_UNSUPPORTED;
    if (A.tex_lo < 0 || A.tex_hi < 0 || A.tex_hi > natlas || (A.tex_lo & 1023) || (A.tex_hi & 3) ||
        (A.tex_hi && A.tex_lo >= A.tex_hi))
        return WR_ERR_INVALID_ARGUMENT;
    const long long ntex = A.tex_hi ? A.tex_hi : natlas;   // end of the exchanged range (the kernels' `ntex`)
    const bool multicast = A.mc_accum && A.mc_attr && A.mc_valid;
    for (int r = 0; r < A.world && !multicast; ++r) {
        if (!A.accum[r] || !A.out_attr[r] || !A.out_valid[r]) return WR_ERR_INVALID_ARGUMENT;
        if ((reinterpret_cast<uintptr_t>(A.accum[r]) | reinterpret_cast<uintptr_t>(A.out_attr[r])) & 15u) return WR_ERR_INVALID_ARGUMENT;
        if (reinterpret_cast<uintptr_t>(A.out_valid[r]) & 3u) return WR_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    // The multicast exchange always runs the light instantiation (64 threads, 256 texels per iteration, one block per
    // SM): measured on 8 x B200 at 4096^2 it is as fast alone as 256-thread blocks (0.585 vs 0.596 ms) and costs the
    // view passes of a concurrent bake 0.16 ms instead of 0.42 ms (tools/bake_pipeline_probe.py).
    const bool light = multicast;
    const long long tpb = light ? 256 : kP2PTexelsPerBlock;
    const long long nblk = (ntex - A.tex_lo + tpb - 1) / tpb;   // blocks of the range, counted from tex_lo
    const long long blk_lo = nblk * A.rank / A.world, blk_hi = nblk * (A.rank + 1) / A.world;
    if (blk_hi > blk_lo) {
        // peer loads want many blocks in flight (8 per SM: 0.52 ms against 0.82 ms with one, 2 x B200, 4096^2); the
        // multicast kernel is fastest with ONE per SM (0.595 against 0.635 ms with eight, 8 x B200)
        int grid = (int)min(blk_hi - blk_lo, (long long)ctx->sm_count * (multicast ? 1 : 8));
        if (A.max_blocks > 0) grid = min(grid, A.max_blocks);
        wr_stage_begin(ctx);
        if (multicast) {
            wr_stage(ctx, stream, "k_uv_reduce_finalize_mc");
            if (light) k_uv_reduce_finalize_mc<64><<<grid, 64, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            else k_uv_reduce_finalize_mc<256><<<grid, 256, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            WR_CHECK_LAUNCH(ctx, "k_uv_reduce_finalize_mc");
        } else {
            wr_stage(ctx, stream, "k_uv_reduce_finalize_p2p");
            if (A.world <= 2) k_uv_reduce_finalize_p2p<2><<<grid, 256, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            else if (A.world <= 4) k_uv_reduce_finalize_p2p<4><<<grid, 256, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            else if (A.world <= 8) k_uv_reduce_finalize_p2p<8><<<grid, 256, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            else k_uv_reduce_finalize_p2p<WR_MAX_P2P_RANKS><<<grid, 256, 0, stream>>>(A, ntex, blk_lo, blk_hi);
            WR_CHECK_LAUNCH(ctx, "k_uv_reduce_finalize_p2p");
        }
        wr_stage(ctx, stream, "end");
    }
    return WR_OK;
}
