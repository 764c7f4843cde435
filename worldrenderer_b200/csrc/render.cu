// Fused render() shading pass (reference render.py:220-286 + utils.py:127-139).
//
// Input: the packed (depth_key << 32 | triangle id) buffer left by the raster stages.  Output: mask,
// world position, view depth (raw or SimpleNormalization), normal, optionally triangle id, the
// nvdiffrast-layout rast tensor and the textured attribute map -- everything render() returns, written
// once.  Operation order of every expression: DESIGN.md 3.4-3.6 / 4 (same as oracle/).
//
//   k_shade           one 4-row column strip per thread, 128 threads, 64 registers, no shared memory and no
//                     block barrier.  The four triangle ids of a strip (low words of the packed entries) are
//                     requested first; a warp whose strips are all background (78% of the warps of config B)
//                     writes its constant rows with 16-byte stores; covered pixels gather indices, then the
//                     vertices (16-byte records from the vertex pass for coarse meshes, PACKED), and derive
//                     everything render() returns.  The per-view depth range is reduced per warp and
//                     published with an atomic only when it improves an L1-cached read of the current range.
//                     Measured alternatives that LOST on config B (profiles/README.md): transposing the
//                     3-channel stores through shared memory (+7%), four pixels per thread with 16-byte
//                     accesses (+22%), a shared-memory prologue with a block barrier (+5%), prefetching the
//                     gathers of the next row (+17%), 48 registers / 10 blocks per SM (+4%, spills).
//   k_depth_finalize  second depth pass for normalisers that need the per-view min / max (covered pixels only:
//                     the constant background value is written by k_shade).
//
// Output element type (wr_render_args.out_dtype): float, __half or __nv_bfloat16 behind the position, depth, normal,
// tangent and attribute maps.  Every value is computed in float32 exactly as for float output and rounded to nearest
// even on the store only, so a half map equals the float map cast by torch.  A two-pass depth normaliser in half
// precision keeps the raw float32 view depth in scratch for k_depth_finalize, which writes the half map.
//
// The shading kernel resets every packed entry it consumes to WR_EMPTY_PIXEL, which leaves the
// buffer clean for the next call (no clear pass).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "texture.cuh"

namespace {

struct ShadeParams {
    wr_render_args a;
    unsigned long long *packed;  // [B,H,W]
    uint8_t *mask;               // [B,H,W] coverage: the caller's out_mask or scratch
    uint32_t *range;             // [B,4] zero-initialised: [0] = max of ~ordered(d) over all pixels (i.e. the
                                 // minimum), [1] = max of ordered(d) over covered pixels (0 = none)
    const float4 *pos4;          // [V]  (x, y, z, 0) written by the vertex pass
    const float4 *nrm4;          // [Vn] (x, y, z, 0) or nullptr
    int wide_ok;                 // W % 4 == 0 and 16-byte aligned pos / normal maps: background rows may use 16-byte stores
    int bg_final;                // two-pass depth whose background value is a constant (controlnet, zero123++):
                                 // written here, k_depth_finalize then only touches covered pixels
    float *depth_raw;            // [B,H,W] two-pass view depth read by k_depth_finalize: out_depth for float output,
                                 // scratch otherwise
};

// store conversion of the output maps: round to nearest even, as torch's casts
template <typename T> __device__ __forceinline__ T to_out(float x);
template <> __device__ __forceinline__ float to_out<float>(float x) { return x; }
template <> __device__ __forceinline__ __half to_out<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 to_out<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// two 16-bit elements in one 32-bit word, `lo` at the lower address
template <typename T> __device__ __forceinline__ uint32_t pack2(T lo, T hi)
{
    uint16_t a, b;
    memcpy(&a, &lo, 2);
    memcpy(&b, &hi, 2);
    return (uint32_t)a | ((uint32_t)b << 16);
}

struct PixelGeo {
    float px, py, pz;   // world position (zeros on background)
    float nx, ny, nz;   // normalised normal (background value on background)
    float tx, ty, tz;   // normalised tangent (generic instantiation only)
    float u, v, w;      // clamped barycentrics, w = (1 - u) - v
    float zw;           // clamped z/w (only when requested)
};

__device__ __forceinline__ float warp_min(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}

__device__ __forceinline__ float apply_simple(float d, float scale, float offset, int clamp)
{
    d = d * scale + offset;
    if (clamp) d = fminf(fmaxf(d, 0.0f), 1.0f);
    return d;
}

// Everything render() derives for a covered pixel (c, r) won by triangle `id`.  m = mvp of the view.
// The three world positions and normals of a triangle: one 16-byte gather each from the records the vertex
// pass left in scratch (L2-resident).
struct V3 {
    float x, y, z;
};
__device__ __forceinline__ V3 ld3(const float4 *p)
{
    const float4 t = __ldg(p);
    V3 r; r.x = t.x; r.y = t.y; r.z = t.z;
    return r;
}
__device__ __forceinline__ V3 ld3s(const float *p)
{
    V3 r; r.x = __ldg(p); r.y = __ldg(p + 1); r.z = __ldg(p + 2);
    return r;
}

struct TriVerts {
    V3 q0, q1, q2, n0, n1, n2;
};
struct TriIdx {
    int i0, i1, i2;
};

__device__ __forceinline__ TriIdx load_tri_idx(const wr_render_args &A, int id)
{
    TriIdx t;
    t.i0 = __ldg(A.tri + 3 * (size_t)id); t.i1 = __ldg(A.tri + 3 * (size_t)id + 1); t.i2 = __ldg(A.tri + 3 * (size_t)id + 2);
    return t;
}

// the normal gathers depend on the indices only: they are issued with the position gathers so that both round
// trips overlap
template <bool PACKED>
__device__ __forceinline__ TriVerts gather_tri(const wr_render_args &A, const float4 *pos4, const float4 *nrm4, int id,
                                               const TriIdx &t, bool want_normal)
{
    TriVerts v;
    constexpr bool packed = PACKED;  // the vertex pass wrote 16-byte records (wr_render decides per call)
    if (packed) {
        v.q0 = ld3(pos4 + t.i0); v.q1 = ld3(pos4 + t.i1); v.q2 = ld3(pos4 + t.i2);
    } else {
        v.q0 = ld3s(A.v_pos + 3 * (size_t)t.i0); v.q1 = ld3s(A.v_pos + 3 * (size_t)t.i1);
        v.q2 = ld3s(A.v_pos + 3 * (size_t)t.i2);
    }
    v.n0.x = v.n0.y = v.n0.z = 0.f;
    v.n1 = v.n0; v.n2 = v.n0;
    if (want_normal) {
        int j0 = t.i0, j1 = t.i1, j2 = t.i2;
        if (A.tri_nrm) {
            j0 = __ldg(A.tri_nrm + 3 * (size_t)id); j1 = __ldg(A.tri_nrm + 3 * (size_t)id + 1);
            j2 = __ldg(A.tri_nrm + 3 * (size_t)id + 2);
        }
        if ((unsigned)j0 < (unsigned)A.Vn && (unsigned)j1 < (unsigned)A.Vn && (unsigned)j2 < (unsigned)A.Vn) {
            if (packed) {
                v.n0 = ld3(nrm4 + j0); v.n1 = ld3(nrm4 + j1); v.n2 = ld3(nrm4 + j2);
            } else {
                v.n0 = ld3s(A.v_nrm + 3 * (size_t)j0); v.n1 = ld3s(A.v_nrm + 3 * (size_t)j1);
                v.n2 = ld3s(A.v_nrm + 3 * (size_t)j2);
            }
        }
    }
    return v;
}

// Everything render() derives for a covered pixel (c, r) won by triangle `id`.  m = mvp of the view.
__device__ __forceinline__ void shade_covered(const wr_render_args &A, const TriVerts &tv, const TriIdx &ti,
                                              const float *m, int id, int c, int r, bool want_normal, bool want_zw,
                                              bool want_tangent, PixelGeo &g)
{
    const int W = A.W, H = A.H;
    const int i0 = ti.i0, i1 = ti.i1, i2 = ti.i2;
    const float x0 = tv.q0.x, y0 = tv.q0.y, z0 = tv.q0.z;
    const float x1 = tv.q1.x, y1 = tv.q1.y, z1 = tv.q1.z;
    const float x2 = tv.q2.x, y2 = tv.q2.y, z2 = tv.q2.z;
    const float n0x = tv.n0.x, n0y = tv.n0.y, n0z = tv.n0.z;
    const float n1x = tv.n1.x, n1y = tv.n1.y, n1z = tv.n1.z;
    const float n2x = tv.n2.x, n2y = tv.n2.y, n2z = tv.n2.z;
    // clip-space vertices, utils.py:127-129 in the contract's operation order
    const float c0x = ((m[0] * x0 + m[1] * y0) + m[2] * z0) + m[3];
    const float c0y = ((m[4] * x0 + m[5] * y0) + m[6] * z0) + m[7];
    const float c0w = ((m[12] * x0 + m[13] * y0) + m[14] * z0) + m[15];
    const float c1x = ((m[0] * x1 + m[1] * y1) + m[2] * z1) + m[3];
    const float c1y = ((m[4] * x1 + m[5] * y1) + m[6] * z1) + m[7];
    const float c1w = ((m[12] * x1 + m[13] * y1) + m[14] * z1) + m[15];
    const float c2x = ((m[0] * x2 + m[1] * y2) + m[2] * z2) + m[3];
    const float c2y = ((m[4] * x2 + m[5] * y2) + m[6] * z2) + m[7];
    const float c2w = ((m[12] * x2 + m[13] * y2) + m[14] * z2) + m[15];
    const float fx = (float)(2 * c + 1 - W) / (float)W;
    const float fy = (float)(2 * r + 1 - H) / (float)H;
    const float p0x = c0x - fx * c0w, p0y = c0y - fy * c0w;
    const float p1x = c1x - fx * c1w, p1y = c1y - fy * c1w;
    const float p2x = c2x - fx * c2w, p2y = c2y - fy * c2w;
    const float a0 = p1x * p2y - p1y * p2x;
    const float a1 = p2x * p0y - p2y * p0x;
    const float a2 = p0x * p1y - p0y * p1x;
    const float iw = 1.0f / ((a0 + a1) + a2);
    const float b0 = a0 * iw, b1 = a1 * iw;
    const float u = (b0 >= 0.0f) ? (b0 > 1.0f ? 1.0f : b0) : 0.0f;
    const float v = (b1 >= 0.0f) ? (b1 > 1.0f ? 1.0f : b1) : 0.0f;
    const float w = (1.0f - u) - v;
    g.u = u; g.v = v; g.w = w;
    if (want_zw) {
        const float c0z = ((m[8] * x0 + m[9] * y0) + m[10] * z0) + m[11];
        const float c1z = ((m[8] * x1 + m[9] * y1) + m[10] * z1) + m[11];
        const float c2z = ((m[8] * x2 + m[9] * y2) + m[10] * z2) + m[11];
        const float zc = ((c0z * a0) + (c1z * a1)) + (c2z * a2);
        const float wc = ((c0w * a0) + (c1w * a1)) + (c2w * a2);
        const float zw = zc / wc;
        g.zw = (zw >= -1.0f) ? (zw > 1.0f ? 1.0f : zw) : -1.0f;
    }
    g.px = ((x0 * u) + (x1 * v)) + (x2 * w);
    g.py = ((y0 * u) + (y1 * v)) + (y2 * w);
    g.pz = ((z0 * u) + (z1 * v)) + (z2 * w);
    if (want_normal) {
        const float ix = ((n0x * u) + (n1x * v)) + (n2x * w);
        const float iy = ((n0y * u) + (n1y * v)) + (n2y * w);
        const float iz = ((n0z * u) + (n1z * v)) + (n2z * w);
        const float ln = sqrtf((ix * ix + iy * iy) + iz * iz);
        const float dn = fmaxf(ln, 1e-12f);
        g.nx = ix / dn; g.ny = iy / dn; g.nz = iz / dn;
    }
    if (want_tangent) {  // render.py:280-284: same faces as the normals (stitched_t_pos_idx)
        int j0 = i0, j1 = i1, j2 = i2;
        if (A.tri_nrm) {
            j0 = __ldg(A.tri_nrm + 3 * (size_t)id); j1 = __ldg(A.tri_nrm + 3 * (size_t)id + 1);
            j2 = __ldg(A.tri_nrm + 3 * (size_t)id + 2);
        }
        float ix = 0.f, iy = 0.f, iz = 0.f;
        if ((unsigned)j0 < (unsigned)A.Vn && (unsigned)j1 < (unsigned)A.Vn && (unsigned)j2 < (unsigned)A.Vn) {
            const float *t0 = A.v_tang + 3 * (size_t)j0, *t1 = A.v_tang + 3 * (size_t)j1, *t2 = A.v_tang + 3 * (size_t)j2;
            ix = ((__ldg(t0) * u) + (__ldg(t1) * v)) + (__ldg(t2) * w);
            iy = ((__ldg(t0 + 1) * u) + (__ldg(t1 + 1) * v)) + (__ldg(t2 + 1) * w);
            iz = ((__ldg(t0 + 2) * u) + (__ldg(t1 + 2) * v)) + (__ldg(t2 + 2) * w);
        }
        const float ln = sqrtf((ix * ix + iy * iy) + iz * iz);
        const float dn = fmaxf(ln, 1e-12f);
        g.tx = ix / dn; g.ty = iy / dn; g.tz = iz / dn;
    }
}

constexpr int kShadeRows = 4;       // rows per thread: that many independent id loads in flight before any use
constexpr int kShadeThreads = 128;
constexpr int kShadeMinBlocks = 8;  // 64 registers: measured 47.3 us vs 49.6 us unconstrained on config B

// Output sets with their own instantiation (no per-pixel pointer tests, ~30% fewer issued instructions on
// config B); every other combination runs the generic instantiation (OUTS < 0, runtime tests).
constexpr int kOutNormal = 1, kOutDepth = 2, kOutTwoPass = 4, kOutGeo = 8;
constexpr int kOutsRenderDefault = kOutNormal | kOutDepth | kOutTwoPass;  // mask + pos + normal + min/max depth
constexpr int kOutsSimpleDepth = kOutNormal | kOutDepth;                  // mask + pos + normal + simple depth
constexpr int kOutsBakeView = kOutGeo | kOutDepth;                        // mask + (pos, aoi_cos) + simple depth

// One column strip of kShadeRows pixels per thread.  grid = (ceil(W/128), ceil(H/kShadeRows), B), 128 threads.
// T: element type of the position, depth, normal, tangent and attribute maps.
template <int OUTS, bool PACKED, typename T>
__global__ void __launch_bounds__(kShadeThreads, kShadeMinBlocks) k_shade(ShadeParams P)
{
    const wr_render_args &A = P.a;
    constexpr bool kGeneric = OUTS < 0;
    constexpr bool kF32 = sizeof(T) == 4;
    T *const out_pos = reinterpret_cast<T *>(A.out_pos);
    T *const out_depth = reinterpret_cast<T *>(A.out_depth);
    T *const out_normal = reinterpret_cast<T *>(A.out_normal);
    T *const out_tangent = reinterpret_cast<T *>(A.out_tangent);
    T *const out_attr = reinterpret_cast<T *>(A.out_attr);
    const bool has_mask = kGeneric ? (P.mask != nullptr) : true;
    const bool has_geo = kGeneric ? (A.out_geo != nullptr) : ((OUTS & kOutGeo) != 0);
    const bool has_pos = kGeneric ? (A.out_pos != nullptr) : !has_geo;
    const bool has_normal = kGeneric ? (A.out_normal != nullptr) : ((OUTS & kOutNormal) != 0);
    const bool need_normal = has_normal || has_geo;
    const bool has_depth = kGeneric ? (A.out_depth != nullptr) : ((OUTS & kOutDepth) != 0);
    const bool two_pass = kGeneric ? (has_depth && A.depth_mode != WR_DEPTH_SIMPLE) : ((OUTS & kOutTwoPass) != 0);
    const bool has_id = kGeneric && A.out_tri_id != nullptr;
    const bool has_rast = kGeneric && A.out_rast != nullptr;
    const bool has_attr = kGeneric && A.out_attr != nullptr;
    const bool has_tangent = kGeneric && A.out_tangent != nullptr;

    wr_pdl_wait();
    wr_pdl_trigger();
    // Blocks map to strips in index order; permuting them so that background and covered blocks are resident
    // together made no difference (profiles/README.md).
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r0 = blockIdx.y * kShadeRows;
    const int b = blockIdx.z;
    const int W = A.W, H = A.H;
    const bool live = c < W;

    const size_t o0 = ((size_t)b * H + r0) * W + (live ? c : 0);
    const int nrows = live ? min(kShadeRows, H - r0) : 0;
    // Only the low word (triangle id; 0xFFFFFFFF = empty) of each packed entry is needed: four 4-byte loads in
    // flight per thread, issued before anything else so that the block prologue below overlaps their latency.
    const uint32_t *pk32 = reinterpret_cast<const uint32_t *>(P.packed);
    uint32_t idw[kShadeRows];
#pragma unroll
    for (int k = 0; k < kShadeRows; ++k) idw[k] = (k < nrows) ? pk32[2 * (o0 + (size_t)k * W)] : 0xFFFFFFFFu;

    // No shared memory and no block barrier: the view's matrices are read where they are used (one address for
    // the whole warp, served by L1), and the depth range is published per warp behind a cached read of the
    // current range -- a stale value only costs a redundant atomic, the range grows monotonically.
    const float *m = A.mvp + 16 * b;
    float wz0 = 0.f, wz1 = 0.f, wz2 = 0.f, wz3 = 0.f;
    if (has_depth) {
        const float *m2 = A.w2c + 16 * b + 8;
        wz0 = __ldg(m2); wz1 = __ldg(m2 + 1); wz2 = __ldg(m2 + 2); wz3 = __ldg(m2 + 3);
    }
    const float nbx = A.normal_bg[0], nby = A.normal_bg[1], nbz = A.normal_bg[2];
    float rot[9];
    if (has_geo) {
#pragma unroll
        for (int j = 0; j < 9; ++j) rot[j] = __ldg(A.w2c + 16 * b + 4 * (j / 3) + (j % 3));  // R = w2c[:3,:3]
    }
    float lo = INFINITY, hi = -INFINITY;
    const bool bg_final = two_pass && P.bg_final;

    // Strip without a covered pixel in the whole warp (78% of the warps of config B): every lane writes the same
    // constants, so position and normal rows go out as 24 full 16-byte stores each instead of 2 x 3 strided
    // 4-byte stores per lane.  Only the specialised instantiations take it (their output set is known).
    if (!kGeneric && !has_geo && P.wide_ok) {
        bool any = false;
#pragma unroll
        for (int k = 0; k < kShadeRows; ++k) any |= idw[k] != 0xFFFFFFFFu;
        const unsigned lane = threadIdx.x & 31;
        const int cw = c - (int)lane;  // first column of the warp
        if (__ballot_sync(0xFFFFFFFFu, any) == 0 && cw + 32 <= W) {
            const float d_bg = -(((wz0 * 0.0f + wz1 * 0.0f) + wz2 * 0.0f) + wz3);  // view depth of a background pixel (p = 0)
            float4 n4;  // elements 4*lane .. 4*lane+3 of the repeating (nbx, nby, nbz) row
            {
                const int e = (4 * (int)lane) % 3;
                const float t0 = e == 0 ? nbx : (e == 1 ? nby : nbz);
                const float t1 = e == 0 ? nby : (e == 1 ? nbz : nbx);
                const float t2 = e == 0 ? nbz : (e == 1 ? nbx : nby);
                n4 = make_float4(t0, t1, t2, t0);
            }
            if constexpr (kF32) {
                for (int k = 0; k < nrows; ++k) {
                    const size_t o = o0 + (size_t)k * W;
                    const size_t row4 = (3 * (o - lane)) >> 2;  // float4 index of the warp's row segment
                    if (lane < 24) {
                        reinterpret_cast<float4 *>(A.out_pos)[row4 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (has_normal) reinterpret_cast<float4 *>(A.out_normal)[row4 + lane] = n4;
                    }
                    P.mask[o] = 0;
                    if (has_depth) A.out_depth[o] = two_pass ? (bg_final ? A.depth_bg : d_bg) : A.depth_bg;
                }
            } else {
                // 16-bit maps: a row segment of 96 elements is 12 x 16 bytes, elements 8*lane .. 8*lane+7 per lane
                // (W % 8 == 0, see wide_ok); n4 holds the triple rotated for element 4*lane, this one for 8*lane
                const int e = (8 * (int)lane) % 3;
                const T h0 = to_out<T>(e == 0 ? nbx : (e == 1 ? nby : nbz));
                const T h1 = to_out<T>(e == 0 ? nby : (e == 1 ? nbz : nbx));
                const T h2 = to_out<T>(e == 0 ? nbz : (e == 1 ? nbx : nby));
                const uint4 n8 = make_uint4(pack2(h0, h1), pack2(h2, h0), pack2(h1, h2), pack2(h0, h1));
                const T dbg = to_out<T>(A.depth_bg);
#pragma unroll 1  // unrolled, it pushes the specialised 16-bit instantiations past 64 registers (spills)
                for (int k = 0; k < nrows; ++k) {
                    const size_t o = o0 + (size_t)k * W;
                    const size_t row8 = (3 * (o - lane)) >> 3;  // 16-byte index of the warp's row segment
                    if (lane < 12) {
                        reinterpret_cast<uint4 *>(out_pos)[row8 + lane] = make_uint4(0u, 0u, 0u, 0u);
                        if (has_normal) reinterpret_cast<uint4 *>(out_normal)[row8 + lane] = n8;
                    }
                    P.mask[o] = 0;
                    if (has_depth) {
                        if (two_pass && !bg_final) P.depth_raw[o] = d_bg;
                        else out_depth[o] = dbg;
                    }
                }
            }
            if (two_pass) lo = d_bg;
            goto publish;
        }
    }

    // Covered pixels need two dependent gathers (id -> vertex indices -> vertex records), row after row.  Issuing
    // the index loads of all rows together, or requesting the records of row k+1 before row k is shaded, was
    // measured: 45.7 / 52.9 us against 45.1 us for this plain loop (profiles/README.md) -- other warps hide the
    // round trips better than the extra registers do.
#pragma unroll 1
    for (int k = 0; k < nrows; ++k) {
        const int r = r0 + k;
        const size_t o = o0 + (size_t)k * W;
        const uint32_t idk = idw[0];
#pragma unroll
        for (int j = 0; j + 1 < kShadeRows; ++j) idw[j] = idw[j + 1];  // register rotation: no indexed local array
        idw[kShadeRows - 1] = 0xFFFFFFFFu;
        const bool covered = idk != 0xFFFFFFFFu;
        int id = -1;
        PixelGeo g;
        g.px = g.py = g.pz = 0.f;
        g.nx = nbx; g.ny = nby; g.nz = nbz;
        g.tx = A.tangent_bg[0]; g.ty = A.tangent_bg[1]; g.tz = A.tangent_bg[2];
        g.u = g.v = g.w = 0.f; g.zw = 0.f;
        if (covered) {
            P.packed[o] = WR_EMPTY_PIXEL;  // self-cleaning
            id = (int)idk;
            const TriIdx tik = load_tri_idx(A, id);
            const TriVerts tvk = gather_tri<PACKED>(A, P.pos4, P.nrm4, id, tik, need_normal);
            shade_covered(A, tvk, tik, m, id, c, r, need_normal, has_rast, has_tangent, g);
        }
        if (has_mask) P.mask[o] = covered ? 1 : 0;
        if (has_geo) {
            // uv.py:108-119: camera-space normal, re-normalised, z clamped to [0,1]; background keeps the
            // (un-rotated) background normal
            float aoi = g.nz;
            if (covered) {
                const float x = (rot[0] * g.nx + rot[1] * g.ny) + rot[2] * g.nz;
                const float y = (rot[3] * g.nx + rot[4] * g.ny) + rot[5] * g.nz;
                const float z = (rot[6] * g.nx + rot[7] * g.ny) + rot[8] * g.nz;
                const float ln = sqrtf((x * x + y * y) + z * z);
                aoi = z / fmaxf(ln, 1e-12f);
            }
            aoi = fminf(fmaxf(aoi, 0.0f), 1.0f);
            reinterpret_cast<float4 *>(A.out_geo)[o] = make_float4(g.px, g.py, g.pz, aoi);
        }
        if (has_pos) { T *d = out_pos + 3 * o; d[0] = to_out<T>(g.px); d[1] = to_out<T>(g.py); d[2] = to_out<T>(g.pz); }
        if (has_normal) { T *d = out_normal + 3 * o; d[0] = to_out<T>(g.nx); d[1] = to_out<T>(g.ny); d[2] = to_out<T>(g.nz); }
        if (has_tangent) { T *d = out_tangent + 3 * o; d[0] = to_out<T>(g.tx); d[1] = to_out<T>(g.ty); d[2] = to_out<T>(g.tz); }
        if (has_id) A.out_tri_id[o] = id;
        if (has_rast)
            reinterpret_cast<float4 *>(A.out_rast)[o] =
                covered ? make_float4(g.u, g.v, g.zw, (float)(id + 1)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (has_attr) {
            T *d = out_attr + (size_t)A.TC * o;
            if (covered) {
                const int t0 = __ldg(A.tri_tex + 3 * (size_t)id), t1 = __ldg(A.tri_tex + 3 * (size_t)id + 1),
                          t2 = __ldg(A.tri_tex + 3 * (size_t)id + 2);
                float tu = 0.f, tv = 0.f;
                if ((unsigned)t0 < (unsigned)A.Vt && (unsigned)t1 < (unsigned)A.Vt && (unsigned)t2 < (unsigned)A.Vt) {
                    const float *e0 = A.v_tex + 2 * (size_t)t0, *e1 = A.v_tex + 2 * (size_t)t1, *e2 = A.v_tex + 2 * (size_t)t2;
                    tu = ((__ldg(e0) * g.u) + (__ldg(e1) * g.v)) + (__ldg(e2) * g.w);
                    tv = ((__ldg(e0 + 1) * g.u) + (__ldg(e1 + 1) * g.v)) + (__ldg(e2 + 1) * g.w);
                }
                for (int c0 = 0; c0 < A.TC; c0 += 4) {
                    float acc[4];
                    sample_texture<4>(A.texture + c0, A.TH, A.TW, A.TC, min(4, A.TC - c0), tu, tv, A.tex_filter, 0, acc);
                    for (int j = 0; j < 4 && c0 + j < A.TC; ++j) d[c0 + j] = to_out<T>(acc[j]);
                }
            } else {
                const T bg = to_out<T>(A.attr_bg);
                for (int j = 0; j < A.TC; ++j) d[j] = bg;
            }
        }
        if (has_depth) {
            // view depth = -(w2c * (p,1)).z (render.py:248-249, utils.py:132-139); background uses p = 0
            const float zv = ((wz0 * g.px + wz1 * g.py) + wz2 * g.pz) + wz3;
            const float d = -zv;
            if (!two_pass) {
                out_depth[o] = to_out<T>(covered ? apply_simple(d, A.depth_p0, A.depth_p1, A.depth_clamp) : A.depth_bg);
            } else {
                if constexpr (kF32) A.out_depth[o] = (bg_final && !covered) ? A.depth_bg : d;
                else if (bg_final && !covered) out_depth[o] = to_out<T>(A.depth_bg);  // k_depth_finalize skips it
                else P.depth_raw[o] = d;
                lo = fminf(lo, d);
                if (covered) hi = fmaxf(hi, d);
            }
        }
    }

publish:
    if (two_pass) {
        // per-view (min over all pixels, max over covered pixels): warp shuffle -> shared atomics -> the
        // last warp of the block issues at most one global atomic pair
        lo = warp_min(lo);
        hi = warp_max(hi);
        if ((threadIdx.x & 31) == 0) {
            const uint32_t seen_lo = __ldg(P.range + 4 * b), seen_hi = __ldg(P.range + 4 * b + 1);
            if (lo < INFINITY && ~wr_float_ordered(lo) > seen_lo) atomicMax(P.range + 4 * b, ~wr_float_ordered(lo));
            if (hi > -INFINITY && wr_float_ordered(hi) > seen_hi) atomicMax(P.range + 4 * b + 1, wr_float_ordered(hi));
        }
    }
}

// Second depth pass (render.py:250-257): background <- per-view min, then the normaliser.  Four pixels per
// thread.  When the shading kernel already wrote the constant background value (bg_final) a group without a
// covered pixel is skipped after its 4-byte mask load -- on config B that is three quarters of the groups.
__device__ __forceinline__ float finalize_one(float d, bool covered, float lo, float den, int mode, float p0, float p1,
                                              float bg)
{
    float x = covered ? d : lo;
    if (mode == WR_DEPTH_CONTROLNET || mode == WR_DEPTH_ZERO123PP) {
        float n = (x - lo) / den;
        n = fminf(fmaxf(n, 0.0f), 1.0f);
        if (mode == WR_DEPTH_CONTROLNET) {
            n = 1.0f - n;
            n = n * p1 + p0;
        }
        x = covered ? n : bg;
    }
    return x;
}

// Reads the float32 view depth `raw` and writes `depth` (the same buffer for float output).
template <typename T>
__global__ void __launch_bounds__(256) k_depth_finalize(const float *raw, T *depth, const uint8_t *mask,
                                                        const uint32_t *range, long long npix_view, int mode, float p0,
                                                        float p1, float bg, int vec, int bg_final)
{
    wr_pdl_wait();
    const int b = blockIdx.y;
    T *dv = depth + (size_t)b * npix_view;
    const float *rv;
    if constexpr (sizeof(T) == 4) rv = dv;  // in place, as one pointer: the float kernel keeps its code
    else rv = raw + (size_t)b * npix_view;
    const uint8_t *mv = mask + (size_t)b * npix_view;
    const long long gi = (long long)blockIdx.x * 256 + threadIdx.x;  // group of 4 pixels
    if (vec) {
        if (gi >= (npix_view >> 2)) return;
        const uchar4 m = reinterpret_cast<const uchar4 *>(mv)[gi];
        if (bg_final && !(m.x | m.y | m.z | m.w)) return;
        const float4 d = reinterpret_cast<const float4 *>(rv)[gi];
        const float lo = wr_ordered_float(~range[4 * b]);
        const uint32_t hik = range[4 * b + 1];
        const float hi = hik == 0u ? lo : wr_ordered_float(hik);  // no covered pixel: filled image is constant lo
        const float den = (hi - lo) + 1e-5f;
        float4 o;
        o.x = finalize_one(d.x, m.x, lo, den, mode, p0, p1, bg);
        o.y = finalize_one(d.y, m.y, lo, den, mode, p0, p1, bg);
        o.z = finalize_one(d.z, m.z, lo, den, mode, p0, p1, bg);
        o.w = finalize_one(d.w, m.w, lo, den, mode, p0, p1, bg);
        if constexpr (sizeof(T) == 4)
            reinterpret_cast<float4 *>(dv)[gi] = o;
        else  // one 8-byte store
            reinterpret_cast<uint2 *>(dv)[gi] = make_uint2(pack2(to_out<T>(o.x), to_out<T>(o.y)),
                                                           pack2(to_out<T>(o.z), to_out<T>(o.w)));
    } else {
        const float lo = wr_ordered_float(~range[4 * b]);
        const uint32_t hik = range[4 * b + 1];
        const float hi = hik == 0u ? lo : wr_ordered_float(hik);
        const float den = (hi - lo) + 1e-5f;
        for (int j = 0; j < 4; ++j) {
            const long long i = gi * 4 + j;
            if (i < npix_view) dv[i] = to_out<T>(finalize_one(rv[i], mv[i] != 0, lo, den, mode, p0, p1, bg));
        }
    }
}

// One instantiation per output set (see kOuts*), vertex source and output element type.
template <typename T>
void launch_shade(const ShadeParams &P, bool use_pack, bool plain, bool two_pass, bool bake, dim3 grid, dim3 block,
                  cudaStream_t stream, bool pdl)
{
    if (use_pack) {
        if (plain && two_pass) wr_launch(k_shade<kOutsRenderDefault, true, T>, grid, block, stream, pdl, P);
        else if (plain) wr_launch(k_shade<kOutsSimpleDepth, true, T>, grid, block, stream, pdl, P);
        else if (bake) wr_launch(k_shade<kOutsBakeView, true, T>, grid, block, stream, pdl, P);
        else wr_launch(k_shade<-1, true, T>, grid, block, stream, pdl, P);
    } else {
        if (plain && two_pass) wr_launch(k_shade<kOutsRenderDefault, false, T>, grid, block, stream, pdl, P);
        else if (plain) wr_launch(k_shade<kOutsSimpleDepth, false, T>, grid, block, stream, pdl, P);
        else if (bake) wr_launch(k_shade<kOutsBakeView, false, T>, grid, block, stream, pdl, P);
        else wr_launch(k_shade<-1, false, T>, grid, block, stream, pdl, P);
    }
}

template <typename T>
void launch_finalize(const wr_render_args &A, const ShadeParams &P, cudaStream_t stream, bool pdl)
{
    const long long npv = (long long)A.H * A.W;
    T *const depth = reinterpret_cast<T *>(A.out_depth);
    const int vec = (npv & 3) == 0 && (reinterpret_cast<uintptr_t>(P.depth_raw) & 15u) == 0 &&
                    (reinterpret_cast<uintptr_t>(depth) & (4 * sizeof(T) - 1)) == 0 &&
                    (reinterpret_cast<uintptr_t>(P.mask) & 3u) == 0;
    wr_launch(k_depth_finalize<T>, dim3(wr_div_up(wr_div_up(npv, 4), 256), A.B), dim3(256), stream, pdl,
              (const float *)P.depth_raw, depth, (const uint8_t *)P.mask, (const uint32_t *)P.range, npv, A.depth_mode,
              A.depth_p0, A.depth_p1, A.depth_bg, vec, P.bg_final);
}

}  // namespace

extern "C" int wr_render(wr_ctx *ctx, const wr_render_args *args, void *stream_)
{
    if (!ctx || !args) return WR_ERR_INVALID_ARGUMENT;
    const wr_render_args &A = *args;
    if (A.B < 0 || A.V < 0 || A.F < 0 || A.H <= 0 || A.W <= 0 || A.H > 8192 || A.W > 8192) return WR_ERR_INVALID_ARGUMENT;
    if (A.out_dtype < WR_DTYPE_F32 || A.out_dtype > WR_DTYPE_BF16) return WR_ERR_INVALID_ARGUMENT;
    if (A.F >= (1 << 30)) return WR_ERR_UNSUPPORTED;
    if (A.out_rast && A.F > (1 << 24)) return WR_ERR_UNSUPPORTED;  // (float)(id + 1) is exact up to 2^24 faces
    if (A.B == 0) return WR_OK;
    if (!A.mvp || (A.V > 0 && !A.v_pos) || (A.F > 0 && !A.tri)) return WR_ERR_INVALID_ARGUMENT;
    if (reinterpret_cast<uintptr_t>(A.mvp) & 15u) return WR_ERR_INVALID_ARGUMENT;  // read as float4 rows
    if (A.out_depth && !A.w2c) return WR_ERR_INVALID_ARGUMENT;
    if (A.out_normal && !A.v_nrm) return WR_ERR_INVALID_ARGUMENT;
    if (A.out_geo && (!A.v_nrm || !A.w2c)) return WR_ERR_INVALID_ARGUMENT;
    if (A.out_tangent && !A.v_tang) return WR_ERR_INVALID_ARGUMENT;
    if (A.out_attr && (!A.v_tex || !A.tri_tex || !A.texture || A.TH <= 0 || A.TW <= 0 || A.TC <= 0)) return WR_ERR_INVALID_ARGUMENT;
    if (A.depth_mode < WR_DEPTH_NONE || A.depth_mode > WR_DEPTH_SIMPLE) return WR_ERR_INVALID_ARGUMENT;
    if (A.tex_filter < 0 || A.tex_filter > 1) return WR_ERR_UNSUPPORTED;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");

    VtxSrc src;
    src.pos = A.v_pos; src.mvp = A.mvp; src.V = A.V; src.batched = 0;
    RasterResult res;
    const bool two_pass = A.out_depth && A.depth_mode != WR_DEPTH_SIMPLE;
    const size_t npix = (size_t)A.B * A.H * A.W;
    void *extra = nullptr;
    wr_stage_begin(ctx);
    const size_t mask_bytes = (two_pass && !A.out_mask) ? wr_align256(npix) : 0;
    const size_t esize = A.out_dtype == WR_DTYPE_F32 ? 4 : 2;
    // float32 view depth of a two-pass normaliser with 16-bit output, behind the mask in the extra scratch
    const size_t raw_bytes = (two_pass && esize != 4) ? wr_align256(npix * 4) : 0;
    const bool want_nrm = A.v_nrm && (A.out_normal || A.out_geo);
    VertexPack pack;
    pack.v_nrm = want_nrm ? A.v_nrm : nullptr;
    pack.Vn = A.Vn;
    pack.offset = mask_bytes + raw_bytes;
    // 16-byte vertex records pay off when many pixels gather from few vertices (config A: 45.4 vs 47.4 us in
    // k_shade); for a mesh of sub-pixel triangles writing them costs more than they save (config B: +3.3 us)
    const bool use_pack = (long long)A.B * A.H * A.W >= 32ll * ((long long)A.V + (want_nrm ? A.Vn : 0));
    pack.pos4 = nullptr;
    pack.nrm4 = nullptr;
    int rc = wr_run_raster(ctx, src, A.B, A.tri, A.F, nullptr, A.H, A.W,
                           mask_bytes + raw_bytes + (use_pack ? wr_vertex_pack_bytes(A.V, A.Vn, want_nrm) : 0), &res, &extra,
                           stream, use_pack ? &pack : nullptr);
    if (rc != WR_OK) return rc;
    if (A.raster_done_event) {
        e = cudaEventRecord(static_cast<cudaEvent_t>(A.raster_done_event), stream);
        if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaEventRecord(raster_done_event)");
    }

    ShadeParams P;
    P.a = A;
    P.packed = res.packed;
    P.mask = A.out_mask ? A.out_mask : (two_pass ? static_cast<uint8_t *>(extra) : nullptr);
    P.range = reinterpret_cast<uint32_t *>(res.view_stats);
    P.pos4 = pack.pos4;
    P.nrm4 = pack.nrm4;
    // a warp's background row segment (32 pixels x 3 elements) starts on a 16-byte boundary: W % 4 == 0 for float,
    // W % 8 == 0 for 16-bit maps
    P.wide_ok = (A.W % (int)(16 / esize)) == 0 && (reinterpret_cast<uintptr_t>(A.out_pos) & 15u) == 0 &&
                (reinterpret_cast<uintptr_t>(A.out_normal) & 15u) == 0;
    P.bg_final = two_pass && (A.depth_mode == WR_DEPTH_CONTROLNET || A.depth_mode == WR_DEPTH_ZERO123PP);
    P.depth_raw = raw_bytes ? reinterpret_cast<float *>(static_cast<char *>(extra) + mask_bytes) : A.out_depth;
    wr_stage(ctx, stream, "k_shade");
    {
        const dim3 grid(wr_div_up(A.W, kShadeThreads), wr_div_up(A.H, kShadeRows), A.B);
        const bool extras = A.out_tri_id || A.out_rast || A.out_attr || A.out_tangent;
        const bool plain = P.mask && A.out_pos && A.out_normal && A.out_depth && !A.out_geo && !extras;
        const bool bake = P.mask && A.out_geo && A.out_depth && !two_pass && !A.out_pos && !A.out_normal && !extras;
        // dependent launch only when the raster stages were launched (the chain's first kernel is a plain launch)
        const bool pdl = !ctx->profiling && A.F > 0 && A.V > 0;
        const dim3 block(kShadeThreads);
        if (A.out_dtype == WR_DTYPE_F16) launch_shade<__half>(P, use_pack, plain, two_pass, bake, grid, block, stream, pdl);
        else if (A.out_dtype == WR_DTYPE_BF16) launch_shade<__nv_bfloat16>(P, use_pack, plain, two_pass, bake, grid, block, stream, pdl);
        else launch_shade<float>(P, use_pack, plain, two_pass, bake, grid, block, stream, pdl);
    }
    WR_CHECK_LAUNCH(ctx, "k_shade");
    wr_raster_consumed(ctx, &res);
    if (two_pass) {
        wr_stage(ctx, stream, "k_depth_finalize");
        if (A.out_dtype == WR_DTYPE_F16) launch_finalize<__half>(A, P, stream, !ctx->profiling);
        else if (A.out_dtype == WR_DTYPE_BF16) launch_finalize<__nv_bfloat16>(A, P, stream, !ctx->profiling);
        else launch_finalize<float>(A, P, stream, !ctx->profiling);
        WR_CHECK_LAUNCH(ctx, "k_depth_finalize");
    }
    wr_stage(ctx, stream, "end");
    return WR_OK;
}
