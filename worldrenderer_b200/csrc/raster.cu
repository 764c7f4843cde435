// Coverage + visibility for dr.rasterize (reference call sites render.py:241, uv.py:40) on sm_100a.
//
// Pipeline, all on one stream, no host round trip:
//   k_snap_vertices   one thread per (view, vertex): clip transform (fused render only), perspective
//                     divide, snap to 1/16 px, outcodes                       -> SnapVert[B,V] (16 B)
//   k_setup_triangles one thread per (view, triangle): cull, classify by screen extent.
//                     * small triangles (the 1M-face case: mostly sub-pixel) are rasterised in the
//                       same thread with exact int32 edge functions and resolved with one 64-bit
//                       atomicMin per covered sample (depth_key << 32 | id) into an L2-resident buffer
//                     * medium / large / to-be-clipped triangles are appended to per-view queues with
//                       one warp-aggregated atomic per warp
//   k_raster_queues   one warp per queued triangle (medium) or 64 warps striding over 16x16-pixel
//                     blocks with a conservative block reject (large): 8x4-pixel footprints, one sample
//                     per lane, warp ballot to skip empty footprints, int64 edge functions
//   k_resolve_rast    one thread per pixel: winning id -> (u, v, z/w, id+1) from the unsnapped vertices
//
// Contract: DESIGN.md section 3.  CPU statement of the same contract: oracle/wr_oracle.c.
#include "common.cuh"

namespace {

constexpr int kSmallMaxPix = 64;       // largest pixel bbox rasterised inside the setup thread
constexpr int kSmallMaxExtent = 1024;  // snapped extent below which int32 edge functions are exact
constexpr int kMediumMaxPix = 2048;    // largest pixel bbox handled by a single warp (<= 64 footprints + partials)
constexpr int kLargeStripes = 64;      // warps sharing one large triangle
constexpr int kLargeBlockLog2 = 4;     // large triangles are walked in 16x16-pixel blocks (conservative reject per block)

struct RasterParams {
    const SnapVert *sv;            // [B,V]
    const int32_t *tri;            // [F,3] (already offset in range mode)
    int F, V, tri_base;            // tri_base: id of tri[0] (range mode)
    int W, H;
    unsigned long long *depth;     // [B,H,W]
    uint32_t *queue;               // [B,Fq]
    int Fq;                        // queue stride (total triangle count)
    int *counters;                 // [B,4]: 0 medium queue length, 1 large queue length, 2 pixel-bbox area of the
                                   // representable large triangles in units of 1024 pixels (one 32 x 32 tile)
};

__device__ __forceinline__ int floor_div16(int a) { return a >> 4; }
__device__ __forceinline__ int ceil_div16(int a) { return -((-a) >> 4); }
__device__ __forceinline__ bool top_left(int dx, int dy) { return dy < 0 || (dy == 0 && dx > 0); }

// DESIGN.md 3.2b for one clip-space vertex: perspective divide, snap to 1/16 px, outcodes.
// w == 1 exactly (orthographic rows 0 0 0 1): rw == 1 and (a * 1) == a, so the divide and the three
// multiplications are skipped without changing a bit.
__device__ __forceinline__ SnapVert snap_one(const float4 c, int W, int H)
{
    SnapVert s;
    s.x = 0; s.y = 0; s.zw = 0.0f;
    uint32_t flags = 0;
    if (isfinite(c.x) && isfinite(c.y) && isfinite(c.z) && isfinite(c.w)) flags |= WR_SV_FINITE;
    uint32_t oc = 0;
    oc |= (c.x < -c.w) ? 1u : 0u;
    oc |= (c.x > c.w) ? 2u : 0u;
    oc |= (c.y < -c.w) ? 4u : 0u;
    oc |= (c.y > c.w) ? 8u : 0u;
    oc |= (c.z < -c.w) ? 16u : 0u;
    oc |= (c.z > c.w) ? 32u : 0u;
    flags |= oc << WR_SV_OC_SHIFT;
    if (c.w > 0.0f) {
        const bool unit_w = c.w == 1.0f;
        const float rw = unit_w ? 1.0f : 1.0f / c.w;
        const float fx = unit_w ? (c.x * (float)(8 * W)) : (c.x * (float)(8 * W)) * rw;
        const float fy = unit_w ? (c.y * (float)(8 * H)) : (c.y * (float)(8 * H)) * rw;
        if (fabsf(fx) <= WR_COORD_LIMIT && fabsf(fy) <= WR_COORD_LIMIT) {
            s.x = __float2int_rn(fx) + (8 * W - 8);   // relative to the sample of pixel (0, 0): see SnapVert
            s.y = __float2int_rn(fy) + (8 * H - 8);
            s.zw = c.z * rw;
            flags |= WR_SV_OK;
        }
    }
    s.flags = flags;
    return s;
}

// Both snap kernels also clear the per-view counter / depth-range block (consumed by the kernels launched after
// them on the same stream), which saves a separate memset launch.
__global__ void __launch_bounds__(256) k_snap_vertices(VtxSrc src, int view0, int W, int H, SnapVert *sv, int *stats,
                                                       int nstats)
{
    if (blockIdx.x == 0 && blockIdx.y == 0)
        for (int i = threadIdx.x; i < nstats; i += blockDim.x) stats[i] = 0;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y + view0;
    if (v >= src.V) return;
    const SnapVert s = snap_one(wr_load_clip(src, b, v), W, H);
    reinterpret_cast<int4 *>(sv)[(size_t)b * src.V + v] = *reinterpret_cast<const int4 *>(&s);
}

__device__ __forceinline__ SnapVert load_sv(const SnapVert *sv, size_t i)
{
    int4 r = __ldg(reinterpret_cast<const int4 *>(sv) + i);
    return *reinterpret_cast<SnapVert *>(&r);
}
// per-view base + 32-bit vertex index: one IMAD.WIDE.U32 per gather instead of 64-bit multiply-add chains
__device__ __forceinline__ SnapVert load_sv32(const SnapVert *view_base, unsigned i)
{
    int4 r = __ldg(reinterpret_cast<const int4 *>(view_base) + i);
    return *reinterpret_cast<SnapVert *>(&r);
}

__device__ __forceinline__ void resolve_sample(unsigned long long *dst, float zw, uint32_t id)
{
    const unsigned long long packed = ((unsigned long long)wr_depth_key(zw) << 32) | id;
    // (An early depth test -- read, compare, then atomicMin only if it can win -- was measured SLOWER on every
    // config: +28% setup on config B, +95% on config A; the dependent read costs more than the atomics it saves.)
    atomicMin(dst, packed);
}

// Small triangle (pixel bbox <= kSmallMaxPix, snapped extent < kSmallMaxExtent): exact int32 edge
// functions, one 64-bit atomicMin per covered sample.  DESIGN.md 3.3.
// The rows r0, r0 + rstep, ... <= r1 are walked (rstep > 1: several lanes share one triangle, k_setup_triangles).
__device__ __forceinline__ void raster_small(int x0, int y0, int x1, int y1, int x2, int y2, float z0, float z1,
                                             float z2, uint32_t id, int c0, int c1, int r0, int r1, int rstep, int W,
                                             int H, unsigned long long *depth_view, int area2)
{
    // area2 = (x1 - x0) * (y2 - y0) - (y1 - y0) * (x2 - x0), computed by the caller (|extent| < 2^10: fits int32)
    if (area2 < 0) {
        int ti; float tf;
        ti = x1; x1 = x2; x2 = ti;
        ti = y1; y1 = y2; y2 = ti;
        tf = z1; z1 = z2; z2 = tf;
        area2 = -area2;
    }
    const int dx0 = x2 - x1, dy0 = y2 - y1;  // edge opposite vertex 0
    const int dx1 = x0 - x2, dy1 = y0 - y2;
    const int dx2 = x1 - x0, dy2 = y1 - y0;
    const int bias0 = top_left(dx0, dy0) ? 0 : 1;
    const int bias1 = top_left(dx1, dy1) ? 0 : 1;
    const int bias2 = top_left(dx2, dy2) ? 0 : 1;
    const float inv_area = wr_rcp_int(area2);
    const int px0 = 16 * c0, py0 = 16 * r0;  // snapped coordinates are relative to the sample of pixel (0, 0)
    int e0r = dx0 * (py0 - y1) - dy0 * (px0 - x1);
    int e1r = dx1 * (py0 - y2) - dy1 * (px0 - x2);
    int e2r = dx2 * (py0 - y0) - dy2 * (px0 - x0);
    unsigned row = (unsigned)r0 * (unsigned)W;  // pixel offsets fit 32 bits (H, W <= 8192)
#pragma unroll 1
    for (int r = r0; r <= r1; r += rstep) {
        int e0 = e0r, e1 = e1r, e2 = e2r;
#pragma unroll 1
        for (int cc = c0; cc <= c1; ++cc) {
            if (e0 >= bias0 && e1 >= bias1 && e2 >= bias2) {
                const float b0 = __int2float_rn(e0) * inv_area;
                const float b1 = __int2float_rn(e1) * inv_area;
                const float b2 = (1.0f - b0) - b1;
                float zw = ((z0 * b0) + (z1 * b1)) + (z2 * b2);
                zw = zw + 0.0f;
                if (zw >= -1.0f && zw <= 1.0f) resolve_sample(depth_view + (row + (unsigned)cc), zw, id);
            }
            e0 -= 16 * dy0; e1 -= 16 * dy1; e2 -= 16 * dy2;
        }
        e0r += 16 * rstep * dx0; e1r += 16 * rstep * dx1; e2r += 16 * rstep * dx2;
        row += (unsigned)(rstep * W);
    }
}

// (A variant that compacted the block's live triangles through shared memory before the raster loop was
// measured 29% SLOWER on config B -- 73.7 vs 57.3 us -- the kernel is bound by its dependent gathers,
// not by divergence; see profiles/README.md.)
//
// LPT lanes per triangle.  1 for meshes of (sub-)pixel triangles.  For coarser meshes (a 50k-face object at 768^2
// has ~6x6-pixel bounding boxes) one thread per triangle means a few hundred thousand threads that each walk up to
// 64 samples serially -- less than two waves of the machine -- so 4 adjacent lanes share a triangle and take every
// fourth row of its bounding box; the bound for in-thread rasterisation grows to 4 x kSmallMaxPix samples, which
// also keeps such triangles out of the warp-per-triangle queue.  All LPT lanes read the same indices and snapped
// vertices (same sectors), lane 0 of the group does the queue append.
// Classification of one (view, triangle) from its three snapped vertices (DESIGN.md 3.1-3.3): culled, rasterised
// right here (small), or to be queued (push = 1 medium, 2 large / to be clipped; entry = queue word).
template <int LPT>
__device__ __forceinline__ void setup_one(const RasterParams &P, const SnapVert &a, const SnapVert &c, const SnapVert &d,
                                          int t, int sub, unsigned long long *depth_view, int &push, uint32_t &entry, int b)
{
    const int W = P.W, H = P.H;
    const uint32_t f_and = a.flags & c.flags & d.flags;
    // one test for the common case: all three vertices finite and snapped, no frustum plane has all three
    // outside; everything else (culled, or to be clipped by the queue pass) takes the cold branch
    constexpr uint32_t kFastMask = WR_SV_FINITE | WR_SV_OK | (63u << WR_SV_OC_SHIFT);
    if ((f_and & kFastMask) != (WR_SV_FINITE | WR_SV_OK)) {
        if ((f_and & WR_SV_FINITE) && ((f_and >> WR_SV_OC_SHIFT) & 63u) == 0 && sub == 0) {
            push = 2;
            entry = (uint32_t)(t + P.tri_base) | WR_QUEUE_SLOW;
        }
        return;
    }
    const int x0 = a.x, y0 = a.y, x1 = c.x, y1 = c.y, x2 = d.x, y2 = d.y;
    const float z0 = a.zw, z1 = c.zw, z2 = d.zw;
    const int xmin = min(x0, min(x1, x2)), xmax = max(x0, max(x1, x2));
    const int ymin = min(y0, min(y1, y2)), ymax = max(y0, max(y1, y2));
    // pixel (c, r) samples (16 c, 16 r); ceil(a / 16) == (a + 15) >> 4 with an arithmetic shift
    const int c0 = max((xmin + 15) >> 4, 0), c1 = min(xmax >> 4, W - 1);
    const int r0 = max((ymin + 15) >> 4, 0), r1 = min(ymax >> 4, H - 1);
    if (c0 > c1 || r0 > r1) return;
    const int npix = (c1 - c0 + 1) * (r1 - r0 + 1);  // <= 8192^2: fits int32
    if (xmax - xmin < kSmallMaxExtent && ymax - ymin < kSmallMaxExtent) {
        // extent below 2^10 sub-pixel units: the doubled area fits int32 exactly
        const int area2 = (x1 - x0) * (y2 - y0) - (y1 - y0) * (x2 - x0);
        if (area2 != 0) {
            if (npix <= kSmallMaxPix * LPT) {
                if (r0 + sub <= r1)
                    raster_small(x0, y0, x1, y1, x2, y2, z0, z1, z2, (uint32_t)(t + P.tri_base), c0, c1, r0 + sub, r1,
                                 LPT, W, H, depth_view, area2);
            } else if (sub == 0) {  // cannot happen for 64-px extents; kept for other thresholds
                push = (npix <= kMediumMaxPix) ? 1 : 2;
                entry = (uint32_t)(t + P.tri_base);
                if (push == 2) atomicAdd(P.counters + 4 * b + 2, npix >> 10);
            }
        }
    } else if (sub == 0) {
        const long long area2 = (long long)(x1 - x0) * (y2 - y0) - (long long)(y1 - y0) * (x2 - x0);
        if (area2 != 0) {
            push = (npix <= kMediumMaxPix) ? 1 : 2;
            entry = (uint32_t)(t + P.tri_base);
            if (push == 2) atomicAdd(P.counters + 4 * b + 2, npix >> 10);
        }
    }
}

template <int LPT>
__global__ void __launch_bounds__(256) k_setup_triangles(RasterParams P, int view0)
{
    wr_pdl_wait();
    wr_pdl_trigger();
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int t = gt / LPT;
    const int sub = gt % LPT;
    const int b = blockIdx.y + view0;
    const unsigned lane = threadIdx.x & 31;
    int push = 0;  // 0 none, 1 medium, 2 large
    uint32_t entry = 0;
    unsigned long long *depth_view = P.depth + (size_t)b * P.H * P.W;
    const unsigned vb = (unsigned)b * (unsigned)P.V;  // B * V < 2^31 (checked by the launcher): 32-bit record index

    if (t < P.F) {
        const int i0 = __ldg(P.tri + 3 * (size_t)t), i1 = __ldg(P.tri + 3 * (size_t)t + 1),
                  i2 = __ldg(P.tri + 3 * (size_t)t + 2);
        if ((unsigned)i0 < (unsigned)P.V && (unsigned)i1 < (unsigned)P.V && (unsigned)i2 < (unsigned)P.V) {
            const SnapVert a = load_sv32(P.sv, vb + (unsigned)i0), c = load_sv32(P.sv, vb + (unsigned)i1),
                           d = load_sv32(P.sv, vb + (unsigned)i2);
            setup_one<LPT>(P, a, c, d, t, sub, depth_view, push, entry, b);
        }
    }
    // warp-aggregated queue append: medium from the front, large / slow from the back
    if (__ballot_sync(0xFFFFFFFFu, push != 0) == 0) return;
#pragma unroll
    for (int q = 1; q <= 2; ++q) {
        const unsigned m = __ballot_sync(0xFFFFFFFFu, push == q);
        if (m == 0) continue;
        const int leader = __ffs(m) - 1;
        int base = 0;
        if ((int)lane == leader) base = atomicAdd(P.counters + 4 * b + (q - 1), __popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (push == q) {
            const int slot = base + __popc(m & ((1u << lane) - 1u));
            uint32_t *qv = P.queue + (size_t)b * P.Fq;
            if (q == 1) qv[slot] = entry;
            else qv[P.Fq - 1 - slot] = entry;
        }
    }
}

// All views of a vertex in one thread: the position is read once, B independent snap chains.
__global__ void __launch_bounds__(256) k_snap_vertices_allviews(VtxSrc src, int B, int W, int H, SnapVert *sv,
                                                                int *stats, int nstats, VertexPack pack)
{
    wr_pdl_trigger();
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < nstats; i += blockDim.x) stats[i] = 0;
    // the B view matrices are staged in shared memory once per block (16-byte broadcast reads instead of 16
    // global loads per view and thread); views beyond the staging capacity read global memory
    constexpr int kStageViews = 32;
    __shared__ float4 s_mvp[kStageViews * 4];
    for (int i = threadIdx.x; i < min(B, kStageViews) * 4; i += blockDim.x)
        s_mvp[i] = __ldg(reinterpret_cast<const float4 *>(src.mvp) + i);
    __syncthreads();
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (pack.nrm4 && v < pack.Vn) {
        const float *n = pack.v_nrm + 3 * (size_t)v;
        pack.nrm4[v] = make_float4(__ldg(n), __ldg(n + 1), __ldg(n + 2), 0.0f);
    }
    if (v >= src.V) return;
    const float *p = src.pos + 3 * (size_t)v;
    const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
    if (pack.pos4) pack.pos4[v] = make_float4(x, y, z, 0.0f);
    for (int b = 0; b < B; ++b) {
        float4 r0, r1, r2, r3;
        if (b < kStageViews) {
            r0 = s_mvp[4 * b]; r1 = s_mvp[4 * b + 1]; r2 = s_mvp[4 * b + 2]; r3 = s_mvp[4 * b + 3];
        } else {
            const float4 *m4 = reinterpret_cast<const float4 *>(src.mvp) + 4 * b;
            r0 = __ldg(m4); r1 = __ldg(m4 + 1); r2 = __ldg(m4 + 2); r3 = __ldg(m4 + 3);
        }
        float4 c;
        c.x = ((r0.x * x + r0.y * y) + r0.z * z) + r0.w;
        c.y = ((r1.x * x + r1.y * y) + r1.z * z) + r1.w;
        c.z = ((r2.x * x + r2.y * y) + r2.z * z) + r2.w;
        c.w = ((r3.x * x + r3.y * y) + r3.z * z) + r3.w;
        const SnapVert s = snap_one(c, W, H);
        reinterpret_cast<int4 *>(sv)[(size_t)b * src.V + v] = *reinterpret_cast<const int4 *>(&s);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Multi-view fast path of the fused render (meshes of small triangles, viewports up to 2048^2).
//
// The vertex pass leaves two words per (vertex, view), all views of a vertex side by side:
//     rec[b * V + v] = (x_u | y_u << 16, z/w)          8 bytes, fetched with one load
// x_u, y_u are the snapped coordinates of DESIGN.md 3.2 relative to an origin that is a whole number of pixels,
// biased by +32768 so that both halves are unsigned: pixel (c, r) samples x_u = 16 (c + lo_c), y_u = 16 (r + lo_r)
// with lo_c = 2048 - W/2, lo_r = 2048 - H/2, i.e. the viewport centre sits in the middle of the 16-bit range and
// +-1875 pixels around it are representable.  A vertex that is not finite, has w <= 0, lies outside the near / far
// planes or outside that range gets the SENTINEL xy = 0; a triangle with such a vertex takes the cold path, which
// recomputes the full 16-byte snapped vertices from the source and runs setup_one (the contract's one and only
// statement of culling / clipping) -- so the compact records can never change a result.
//
// k_setup_mv: one thread per (view, triangle).  One 8-byte load per vertex fetches xy and z/w; packed 16-bit
// min3 / max3 and a handful of SIMD-in-a-word operations decide whether the bounding box holds a sample at all --
// half of the (view, triangle) pairs of a dense mesh end there (~16 instructions instead of ~80 in the per-view
// kernel).  A triangle that spans less than two pixels (at most 2 x 2 samples) is tested sample by sample with
// three cross products of PERTURBED coordinates that carry the top-left rule (mv_fast), slivers of up to four
// samples with the plain cross products and an explicit tie-break (mv_single); everything else walks its box like
// raster_small or goes to the queues.
constexpr float kRecLimit = 30000.0f;  // |snapped coordinate| (centred) that still gets a record
constexpr unsigned kGuard = 0x10001000u;

struct MvParams {
    const uint2 *rec;              // [B][V] (xy, z/w bits)
    const int32_t *tri;            // [F,3]
    int F, V, B, Bq;
    int W, H;
    unsigned HW;                   // H * W (<= 2048^2 on this path): a view's offset into `depth` is one wide multiply
    unsigned lo_px, hi_px;         // packed (row << 16 | col) first / last pixel of the viewport in biased pixel units
    unsigned long long *depth;     // [B,H,W]
    uint32_t *queue;               // [B,Fq]
    int Fq;
    int *counters;                 // [B,4]
};

__device__ __forceinline__ void snap_rec(const float4 c, int W, int H, int addx, int addy, unsigned &xy, float &zw)
{
    // same expressions as snap_one; a record is written only when snap_one would flag the vertex OK | FINITE with
    // no near / far outcode AND the coordinates fit 16 bits
    xy = 0u; zw = 0.0f;
    if (c.w > 0.0f && c.w <= 3.402823466e38f && c.z >= -c.w && c.z <= c.w) {
        const bool unit_w = c.w == 1.0f;
        const float rw = unit_w ? 1.0f : 1.0f / c.w;
        const float fx = unit_w ? (c.x * (float)(8 * W)) : (c.x * (float)(8 * W)) * rw;
        const float fy = unit_w ? (c.y * (float)(8 * H)) : (c.y * (float)(8 * H)) * rw;
        if (fabsf(fx) <= kRecLimit && fabsf(fy) <= kRecLimit) {   // false for NaN / inf
            const int xi = __float2int_rn(fx) + addx, yi = __float2int_rn(fy) + addy;  // in [2760, 62776]
            xy = (unsigned)xi | ((unsigned)yi << 16);
            zw = c.z * rw;
        }
    }
}

__global__ void __launch_bounds__(256) k_snap_mv(VtxSrc src, int B, int W, int H, int addx, int addy, uint2 *rec,
                                                 int *stats, int nstats, VertexPack pack)
{
    wr_pdl_trigger();
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < nstats; i += blockDim.x) stats[i] = 0;
    // The views go through shared memory in groups of 32: the inner loop reads its matrix rows from there and its
    // orthographic flag from one bit mask (a per-iteration choice between a staged and a global row was compiled
    // into both loads and a select, a fifth of this issue-bound kernel's instructions).
    constexpr int kStageViews = 32;
    __shared__ float4 s_mvp[kStageViews * 4];
    __shared__ unsigned s_unit;
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (pack.nrm4 && v < pack.Vn) {
        const float *n = pack.v_nrm + 3 * (size_t)v;
        pack.nrm4[v] = make_float4(__ldg(n), __ldg(n + 1), __ldg(n + 2), 0.0f);
    }
    const bool live = v < src.V;
    float x = 0.f, y = 0.f, z = 0.f;
    if (live) {
        const float *p = src.pos + 3 * (size_t)v;
        x = __ldg(p); y = __ldg(p + 1); z = __ldg(p + 2);
        if (pack.pos4) pack.pos4[v] = make_float4(x, y, z, 0.0f);
    }
    const bool finite_pos = isfinite(x) && isfinite(y) && isfinite(z);
    uint2 *out = rec + (live ? v : 0);
    for (int b0 = 0; b0 < B; b0 += kStageViews) {
        const int nb = min(B - b0, kStageViews);
        if (b0) __syncthreads();   // the previous group's rows are no longer read
        for (int i = threadIdx.x; i < nb * 4; i += blockDim.x)
            s_mvp[i] = __ldg(reinterpret_cast<const float4 *>(src.mvp) + 4 * b0 + i);
        if (threadIdx.x < 32) {   // bit b: row 3 of view b0 + b is exactly (0 0 0 1)
            bool unit = false;
            if ((int)threadIdx.x < nb) {
                const float4 r3 = __ldg(reinterpret_cast<const float4 *>(src.mvp) + 4 * (b0 + threadIdx.x) + 3);
                unit = r3.x == 0.0f && r3.y == 0.0f && r3.z == 0.0f && r3.w == 1.0f;
            }
            const unsigned bits = __ballot_sync(0xFFFFFFFFu, unit);
            if (threadIdx.x == 0) s_unit = bits;
        }
        __syncthreads();
        if (!live) continue;
        const unsigned unit_bits = s_unit;
#pragma unroll 2
        for (int b = 0; b < nb; ++b) {
            const float4 r0 = s_mvp[4 * b], r1 = s_mvp[4 * b + 1], r2 = s_mvp[4 * b + 2];
            float4 c;
            c.x = ((r0.x * x + r0.y * y) + r0.z * z) + r0.w;
            c.y = ((r1.x * x + r1.y * y) + r1.z * z) + r1.w;
            c.z = ((r2.x * x + r2.y * y) + r2.z * z) + r2.w;
            unsigned rxy = 0u;
            float rzw = 0.0f;
            if ((unit_bits >> b) & 1u) {
                // Orthographic view (uniform branch).  For a finite vertex the contract's w = ((0 x + 0 y) + 0 z) + 1
                // is exactly 1, so snap_rec's unit-w expressions apply as they are; for a non-finite one 0 * inf = NaN
                // fails its w > 0 test -- the explicit finiteness test (once per vertex) stands in for that.
                if (finite_pos && c.z >= -1.0f && c.z <= 1.0f) {
                    const float fx = c.x * (float)(8 * W), fy = c.y * (float)(8 * H);
                    if (fabsf(fx) <= kRecLimit && fabsf(fy) <= kRecLimit) {
                        rxy = (unsigned)(__float2int_rn(fx) + addx) | ((unsigned)(__float2int_rn(fy) + addy) << 16);
                        rzw = c.z;
                    }
                }
            } else {
                const float4 r3 = s_mvp[4 * b + 3];
                c.w = ((r3.x * x + r3.y * y) + r3.z * z) + r3.w;
                snap_rec(c, W, H, addx, addy, rxy, rzw);
            }
            *out = make_uint2(rxy, __float_as_uint(rzw));
            out += src.V;
        }
    }
}

// Bounding box of a (view, triangle) in biased pixel units, packed (row << 16 | col), clamped to the viewport.
// t = (last | guard) - first keeps a guard bit per half exactly when last >= first in that half:
// (t & kGuard) == kGuard  <=>  the box holds a sample;  t == kGuard  <=>  exactly one.
__device__ __forceinline__ unsigned mv_box(unsigned a, unsigned c, unsigned d, unsigned lo_px, unsigned hi_px,
                                           unsigned &first)
{
    const unsigned mn = __vimin3_u16x2(a, c, d), mx = __vimax3_u16x2(a, c, d);
    first = __vmaxu2(((mn + 0x000F000Fu) >> 4) & 0x0FFF0FFFu, lo_px);
    const unsigned last = __vminu2((mx >> 4) & 0x0FFF0FFFu, hi_px);
    return (last | kGuard) - first;
}

// Sample exactly on an edge or a vertex (m == 0): the top-left rule of DESIGN.md 3.3 on the orientation-normalised
// edges.  a_i, b_i: vertex i relative to the sample; F_i: orientation-normalised edge functions.
__device__ __forceinline__ bool mv_tie_break(int a0, int b0, int a1, int b1, int a2, int b2, int F0, int F1, int F2,
                                          bool flip)
{
    int dx0 = a2 - a1, dy0 = b2 - b1, dx1 = a0 - a2, dy1 = b0 - b2, dx2 = a1 - a0, dy2 = b1 - b0;
    if (flip) { dx0 = -dx0; dy0 = -dy0; dx1 = -dx1; dy1 = -dy1; dx2 = -dx2; dy2 = -dy2; }
    return (F0 > 0 || top_left(dx0, dy0)) && (F1 > 0 || top_left(dx1, dy1)) && (F2 > 0 || top_left(dx2, dy2));
}

// One work item whose box holds exactly the sample of pixel (c, r) (viewport coordinates).  Exact integer
// arithmetic: with a_i = x_i - px, b_i = y_i - py the edge function of edge (v1 -> v2) at the sample is the cross
// product a1 b2 - a2 b1 (same integer as dx0 (py - y1) - dy0 (px - x1)), and the three add up to the doubled
// area.  A box with one sample is less than two pixels wide, so everything fits int32 with room to spare.
// Depth: the expressions of raster_small; for a clockwise triangle raster_small swaps vertices 1 and 2, which
// negates the edge functions and lets edges 1 and 2 trade places -- reproduced here by the sign of 1 / area and
// the selects on `flip` (float negation is exact, and the final + 0.0f removes the sign of a zero).
__device__ __forceinline__ void mv_single(const MvParams &P, unsigned xy0, unsigned xy1, unsigned xy2, float z0,
                                          float z1, float z2, int b, int c, int r, uint32_t id)
{
    const int px = (c + (int)(P.lo_px & 0xFFFFu)) << 4, py = (r + (int)(P.lo_px >> 16)) << 4;
    const int a0 = (int)(xy0 & 0xFFFFu) - px, b0 = (int)(xy0 >> 16) - py;
    const int a1 = (int)(xy1 & 0xFFFFu) - px, b1 = (int)(xy1 >> 16) - py;
    const int a2 = (int)(xy2 & 0xFFFFu) - px, b2 = (int)(xy2 >> 16) - py;
    const int E0 = a1 * b2 - a2 * b1, E1 = a2 * b0 - a0 * b2, E2 = a0 * b1 - a1 * b0;
    const int area2 = E0 + E1 + E2;
    if (area2 == 0) return;
    const bool flip = area2 < 0;
    const int F0 = flip ? -E0 : E0, F1 = flip ? -E1 : E1, F2 = flip ? -E2 : E2;
    const int m = __vimin3_s32(F0, F1, F2);
    if (m < 0) return;
    if (m == 0 && !mv_tie_break(a0, b0, a1, b1, a2, b2, F0, F1, F2, flip)) return;
    const float inv_area = wr_rcp_int(area2);   // signed: float(E) * inv_area == float(F) * (1 / |area|)
    const float w0 = __int2float_rn(E0) * inv_area;
    const float w1 = __int2float_rn(flip ? E2 : E1) * inv_area;
    const float w2 = (1.0f - w0) - w1;
    float zw = ((z0 * w0) + ((flip ? z2 : z1) * w1)) + ((flip ? z1 : z2) * w2);
    zw = zw + 0.0f;
    if (zw >= -1.0f && zw <= 1.0f)
        resolve_sample(P.depth + ((size_t)b * P.H * P.W + (unsigned)(r * P.W + c)), zw, id);
}

// Sample (pc, pr) (biased pixel coordinates) of a triangle that spans less than two pixels in x and in y, so that
// the vertices relative to the sample satisfy |a_i|, |b_i| <= 31.  Coverage including the top-left rule comes from
// ONE set of cross products: with a_i' = 1024 a_i - 32, b_i' = 1024 b_i - 1 (the sample moved by (1/32, 1/1024) of
// a sub-pixel unit towards +x, +y)
//     E0' = a1' b2' - a2' b1' = 2^20 E0 + 1024 (dx0 - 32 dy0),      (dx0, dy0) = v2 - v1, |dx0 - 32 dy0| <= 1023,
// so E0' has the sign of E0 when E0 != 0 and otherwise the sign of (dx0 - 32 dy0), which is positive exactly for
// a left edge (dy0 < 0) or a top edge (dy0 == 0, dx0 > 0) of a counter-clockwise triangle; for a clockwise one
// every sign flips, E' included.  Hence: covered <=> E0', E1', E2' all > 0 or all < 0 (their sum is 2^20 * area2,
// so a zero-area triangle can never pass).  |a_i'|, |b_i'| < 2^15: the products fit int32.  Equivalent to the
// orientation-normalised `e >= bias` test of raster_small bit for bit; the depth expressions are mv_single's.
__device__ __forceinline__ void mv_fast(const MvParams &P, unsigned xy0, unsigned xy1, unsigned xy2, float z0, float z1,
                                        float z2, unsigned long long *depth_view, unsigned pxy, uint32_t id)
{
    const int pc = (int)(pxy & 0xFFFFu), pr = (int)(pxy >> 16);
    const int cx = (pc << 14) + 32, cy = (pr << 14) + 1;   // 1024 * 16 * pixel + offset
    const int x0 = (int)(xy0 & 0xFFFFu), y0 = (int)(xy0 >> 16);
    const int x1 = (int)(xy1 & 0xFFFFu), y1 = (int)(xy1 >> 16);
    const int x2 = (int)(xy2 & 0xFFFFu), y2 = (int)(xy2 >> 16);
    const int a0 = x0 * 1024 - cx, b0 = y0 * 1024 - cy;
    const int a1 = x1 * 1024 - cx, b1 = y1 * 1024 - cy;
    const int a2 = x2 * 1024 - cx, b2 = y2 * 1024 - cy;
    const int Q0 = a1 * b2 - a2 * b1, Q1 = a2 * b0 - a0 * b2, Q2 = a0 * b1 - a1 * b0;
    const int lo = __vimin3_s32(Q0, Q1, Q2), hi = __vimax3_s32(Q0, Q1, Q2);
    if (lo <= 0 && hi >= 0) return;
    // covered: the exact edge functions for the depth (E_i = (Q_i - 1024 (dx_i - 32 dy_i)) / 2^20)
    const int px = pc << 4, py = pr << 4;
    const int u0 = x0 - px, v0 = y0 - py, u1 = x1 - px, v1 = y1 - py, u2 = x2 - px, v2 = y2 - py;
    const int E0 = u1 * v2 - u2 * v1, E1 = u2 * v0 - u0 * v2, E2 = u0 * v1 - u1 * v0;
    const int area2 = E0 + E1 + E2;
    const bool flip = lo < 0;
    const float inv_area = wr_rcp_int(area2);   // signed: float(E) * inv_area == float(F) * (1 / |area|)
    const float w0 = __int2float_rn(E0) * inv_area;
    const float w1 = __int2float_rn(flip ? E2 : E1) * inv_area;
    const float w2 = (1.0f - w0) - w1;
    float zw = ((z0 * w0) + ((flip ? z2 : z1) * w1)) + ((flip ? z1 : z2) * w2);
    zw = zw + 0.0f;
    if (zw >= -1.0f && zw <= 1.0f) {
        const unsigned rel = pxy - P.lo_px;  // no borrow: the sample lies in the viewport
        resolve_sample(depth_view + ((rel >> 16) * (unsigned)P.W + (rel & 0xFFFFu)), zw, id);
    }
}

// One work item whose box holds several samples: classify by size, rasterise a small triangle here (the loop of
// raster_small with the orientation handled by negating the edge vectors), or report it for the queues.
__device__ __forceinline__ void mv_multi(const MvParams &P, unsigned xy0, unsigned xy1, unsigned xy2, float z0,
                                         float z1, float z2, int b, uint32_t id, int &push)
{
    // signed coordinates relative to the sample of viewport pixel (0, 0)
    const int ox = (int)(P.lo_px & 0xFFFFu) << 4, oy = (int)(P.lo_px >> 16) << 4;
    const int x0 = (int)(xy0 & 0xFFFFu) - ox, y0 = (int)(xy0 >> 16) - oy;
    const int x1 = (int)(xy1 & 0xFFFFu) - ox, y1 = (int)(xy1 >> 16) - oy;
    const int x2 = (int)(xy2 & 0xFFFFu) - ox, y2 = (int)(xy2 >> 16) - oy;
    const int xmin = min(x0, min(x1, x2)), xmax = max(x0, max(x1, x2));
    const int ymin = min(y0, min(y1, y2)), ymax = max(y0, max(y1, y2));
    const int c0 = max((xmin + 15) >> 4, 0), c1 = min(xmax >> 4, P.W - 1);
    const int r0 = max((ymin + 15) >> 4, 0), r1 = min(ymax >> 4, P.H - 1);
    if (c0 > c1 || r0 > r1) return;
    const int npix = (c1 - c0 + 1) * (r1 - r0 + 1);
    int dx0 = x2 - x1, dy0 = y2 - y1;  // edge opposite vertex 0
    int dx1 = x0 - x2, dy1 = y0 - y2;
    int dx2 = x1 - x0, dy2 = y1 - y0;
    if (!(xmax - xmin < kSmallMaxExtent && ymax - ymin < kSmallMaxExtent && npix <= kSmallMaxPix)) {
        const long long a2 = (long long)dx2 * (y2 - y0) - (long long)dy2 * (x2 - x0);
        if (a2 != 0) {
            push = (npix <= kMediumMaxPix) ? 1 : 2;
            if (push == 2) atomicAdd(P.counters + 4 * b + 2, npix >> 10);
        }
        return;
    }
    int area2 = dx2 * (y2 - y0) - dy2 * (x2 - x0);  // extent below 2^10: exact in int32
    if (area2 == 0) return;
    const bool flip = area2 < 0;
    if (flip) {
        dx0 = -dx0; dy0 = -dy0; dx1 = -dx1; dy1 = -dy1; dx2 = -dx2; dy2 = -dy2;
        area2 = -area2;
    }
    const int bias0 = top_left(dx0, dy0) ? 0 : 1;
    const int bias1 = top_left(dx1, dy1) ? 0 : 1;
    const int bias2 = top_left(dx2, dy2) ? 0 : 1;
    const float za = flip ? z2 : z1, zb = flip ? z1 : z2;
    const float inv_area = wr_rcp_int(area2);
    const int px0 = 16 * c0, py0 = 16 * r0;
    int e0r = dx0 * (py0 - y1) - dy0 * (px0 - x1);
    int e1r = dx1 * (py0 - y2) - dy1 * (px0 - x2);
    int e2r = dx2 * (py0 - y0) - dy2 * (px0 - x0);
    unsigned long long *dv = P.depth + (size_t)b * P.H * P.W;
    unsigned row = (unsigned)(r0 * P.W);
#pragma unroll 1
    for (int r = r0; r <= r1; ++r) {
        int e0 = e0r, e1 = e1r, e2 = e2r;
#pragma unroll 1
        for (int cc = c0; cc <= c1; ++cc) {
            if (e0 >= bias0 && e1 >= bias1 && e2 >= bias2) {
                const float w0 = __int2float_rn(e0) * inv_area;
                const float w1 = __int2float_rn(flip ? e2 : e1) * inv_area;
                const float w2 = (1.0f - w0) - w1;
                float zw = ((z0 * w0) + (za * w1)) + (zb * w2);
                zw = zw + 0.0f;
                if (zw >= -1.0f && zw <= 1.0f) resolve_sample(dv + (row + (unsigned)cc), zw, id);
            }
            e0 -= 16 * dy0; e1 -= 16 * dy1; e2 -= 16 * dy2;
        }
        e0r += 16 * dx0; e1r += 16 * dx1; e2r += 16 * dx2;
        row += (unsigned)P.W;
    }
}

// Queue append of a lane with push != 0.  Pushes are rare on this path (a fine mesh queues a triangle only when its
// box holds more than 64 samples), so the common case must cost nothing: no warp-wide vote -- the lanes that do get
// here aggregate among themselves (whoever is active shares one atomic per queue).
__device__ __forceinline__ void mv_push(const MvParams &P, int push, int b, uint32_t entry)
{
    if (push == 0) return;
    const unsigned lane = threadIdx.x & 31;
    const unsigned m = __match_any_sync(__activemask(), (unsigned)push);   // same view for the whole block
    const int leader = __ffs(m) - 1;
    int base = 0;
    if ((int)lane == leader) base = atomicAdd(P.counters + 4 * b + (push - 1), __popc(m));
    base = __shfl_sync(m, base, leader);
    const int slot = base + __popc(m & ((1u << lane) - 1u));
    uint32_t *qv = P.queue + (size_t)b * P.Fq;
    if (push == 1) qv[slot] = entry;
    else qv[P.Fq - 1 - slot] = entry;
}

// cold (view, triangle) pair: the contract's own classification from the full snapped vertices
__device__ __forceinline__ void mv_cold(const RasterParams &Pold, const VtxSrc &src, int b, int i0, int i1, int i2, int t,
                                     unsigned long long *depth_view, int &push, uint32_t &entry)
{
    const SnapVert a = snap_one(wr_load_clip(src, b, i0), Pold.W, Pold.H);
    const SnapVert c = snap_one(wr_load_clip(src, b, i1), Pold.W, Pold.H);
    const SnapVert d = snap_one(wr_load_clip(src, b, i2), Pold.W, Pold.H);
    setup_one<1>(Pold, a, c, d, t, 0, depth_view, push, entry, b);
}

// One thread per (view, triangle), blockIdx.y = view: the parallelism of k_setup_triangles with the compact records.
__global__ void __launch_bounds__(256, 8) k_setup_mv(MvParams P, RasterParams Pold, VtxSrc src)
{
    wr_pdl_wait();
    wr_pdl_trigger();
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    int push = 0;
    uint32_t entry = (uint32_t)t;
    if (t < P.F) {
        const int i0 = __ldg(P.tri + 3 * (size_t)t), i1 = __ldg(P.tri + 3 * (size_t)t + 1), i2 = __ldg(P.tri + 3 * (size_t)t + 2);
        if (__vimax3_u32((unsigned)i0, (unsigned)i1, (unsigned)i2) < (unsigned)P.V) {
            // B * V < 2^31 (checked by the launcher): 32-bit record indices
            const unsigned vb = (unsigned)b * (unsigned)P.V;
            const uint2 ra = __ldg(P.rec + (vb + (unsigned)i0)), rc = __ldg(P.rec + (vb + (unsigned)i1)),
                        rd = __ldg(P.rec + (vb + (unsigned)i2));
            const unsigned a = ra.x, c = rc.x, d = rd.x;
            unsigned first;
            const unsigned tt = mv_box(a, c, d, P.lo_px, P.hi_px, first);
            // a vertex without a record has xy == 0 (a record's halves are >= 2760)
            if (__vimin3_u32(a, c, d) == 0u) {
                mv_cold(Pold, src, b, i0, i1, i2, t, P.depth + (size_t)b * P.H * P.W, push, entry);
            } else if ((tt & kGuard) == kGuard) {
                const float z0 = __uint_as_float(ra.y), z1 = __uint_as_float(rc.y), z2 = __uint_as_float(rd.y);
                unsigned long long *depth_view = P.depth + (unsigned long long)(unsigned)b * P.HW;
                const unsigned mn = __vimin3_u16x2(a, c, d), mx = __vimax3_u16x2(a, c, d);
                if (((mx - mn) & 0xFFE0FFE0u) == 0u) {
                    // spans less than two pixels: 1, 2 or 2 x 2 samples
                    mv_fast(P, a, c, d, z0, z1, z2, depth_view, first, (uint32_t)t);
                    if (tt != kGuard) {
                        // second column (bit 0), second row (bit 1), both (bit 2)
                        const unsigned ex = tt & 1u, ey = (tt >> 16) & 1u;
                        unsigned pending = ex | (ey << 1) | ((ex & ey) << 2);
#pragma unroll 1
                        while (pending) {
                            const unsigned j = __ffs(pending) - 1u;
                            pending &= pending - 1u;
                            mv_fast(P, a, c, d, z0, z1, z2, depth_view, first + (j == 0u ? 1u : (j == 1u ? 0x10000u : 0x10001u)),
                                    (uint32_t)t);
                        }
                    }
                } else {
                    const unsigned rel = first - P.lo_px;  // no borrow: first >= lo_px in both halves
                    const int c0 = (int)(rel & 0xFFFFu), r0 = (int)(rel >> 16);
                    const int nx = (int)(tt & 0xFFFu), ny = (int)((tt >> 16) & 0xFFFu);  // box = (nx + 1) x (ny + 1) samples
                    if ((nx + 1) * (ny + 1) <= 4 && ((mx - mn) & 0xFF80FF80u) == 0u) {
                        // a sliver of up to four samples that spans less than eight pixels (exact in int32)
#pragma unroll 1
                        for (int r = r0; r <= r0 + ny; ++r)
#pragma unroll 1
                            for (int cc = c0; cc <= c0 + nx; ++cc) mv_single(P, a, c, d, z0, z1, z2, b, cc, r, (uint32_t)t);
                    } else {
                        mv_multi(P, a, c, d, z0, z1, z2, b, (uint32_t)t, push);
                    }
                }
            }
        }
    }
    mv_push(P, push, b, entry);
}

// One warp rasterises one snapped triangle (or the stripe-th share of its 16x16 blocks).
// E is the integer type of the edge functions: int when the snapped extent is below 2^14 (products < 2^29),
// long long otherwise (coordinates up to 2^22).  Both are exact, so the choice cannot change a result.
template <typename E> __device__ __forceinline__ float edge_to_float(E e);
template <> __device__ __forceinline__ float edge_to_float<int>(int e) { return __int2float_rn(e); }
template <> __device__ __forceinline__ float edge_to_float<long long>(long long e) { return __ll2float_rn(e); }

template <bool LARGE, typename E>
__device__ void warp_raster_impl(int x0, int y0, int x1, int y1, int x2, int y2, float z0, float z1, float z2,
                                 uint32_t id, int W, int H, unsigned long long *depth_view, int stripe, unsigned lane)
{
    long long area2 = (long long)(x1 - x0) * (y2 - y0) - (long long)(y1 - y0) * (x2 - x0);
    if (area2 == 0) return;
    if (area2 < 0) {
        int ti; float tf;
        ti = x1; x1 = x2; x2 = ti;
        ti = y1; y1 = y2; y2 = ti;
        tf = z1; z1 = z2; z2 = tf;
        area2 = -area2;
    }
    const int xmin = min(x0, min(x1, x2)), xmax = max(x0, max(x1, x2));
    const int ymin = min(y0, min(y1, y2)), ymax = max(y0, max(y1, y2));
    const int c0 = max(ceil_div16(xmin), 0), c1 = min(floor_div16(xmax), W - 1);
    const int r0 = max(ceil_div16(ymin), 0), r1 = min(floor_div16(ymax), H - 1);
    if (c0 > c1 || r0 > r1) return;
    const int dx0 = x2 - x1, dy0 = y2 - y1;
    const int dx1 = x0 - x2, dy1 = y0 - y2;
    const int dx2 = x1 - x0, dy2 = y1 - y0;
    const E bias0 = top_left(dx0, dy0) ? 0 : 1;
    const E bias1 = top_left(dx1, dy1) ? 0 : 1;
    const E bias2 = top_left(dx2, dy2) ? 0 : 1;
    const float inv_area = 1.0f / __ll2float_rn(area2);
    const int lx = lane & 7, ly = lane >> 3;

    // Walks the 8x4-pixel footprints of the pixel rectangle [cl,ch] x [rl,rh].  The three edge functions are
    // evaluated once per footprint row for this lane's pixel and then advanced by a constant per 8-pixel step
    // (exact integer arithmetic either way).
    const E sx0 = -(E)dy0 * 128, sx1 = -(E)dy1 * 128, sx2 = -(E)dy2 * 128;  // +8 pixels in x = +128 sub-pixel units
    auto scan = [&](int cl, int ch, int rl, int rh) {
        for (int fy = rl & ~3; fy <= rh; fy += 4) {
            const int rr = fy + ly;
            const bool row_in = rr >= rl && rr <= rh;
            const int py = 16 * rr;
            int cc = (cl & ~7) + lx;
            const int px = 16 * cc;
            E e0 = (E)dx0 * (py - y1) - (E)dy0 * (px - x1);
            E e1 = (E)dx1 * (py - y2) - (E)dy1 * (px - x2);
            E e2 = (E)dx2 * (py - y0) - (E)dy2 * (px - x0);
            unsigned long long *row = depth_view + (size_t)rr * W;
            for (int fx = cl & ~7; fx <= ch; fx += 8, cc += 8, e0 += sx0, e1 += sx1, e2 += sx2) {
                const bool cov = row_in && cc >= cl && cc <= ch && e0 >= bias0 && e1 >= bias1 && e2 >= bias2;
                if (__ballot_sync(0xFFFFFFFFu, cov) == 0) continue;
                if (cov) {
                    const float b0 = edge_to_float<E>(e0) * inv_area;
                    const float b1 = edge_to_float<E>(e1) * inv_area;
                    const float b2 = (1.0f - b0) - b1;
                    float zw = ((z0 * b0) + (z1 * b1)) + (z2 * b2);
                    zw = zw + 0.0f;
                    if (zw >= -1.0f && zw <= 1.0f) resolve_sample(row + cc, zw, id);
                }
            }
        }
    };

    if (!LARGE) {
        scan(c0, c1, r0, r1);
    } else {
        constexpr int kB = 1 << kLargeBlockLog2;
        const int bx0 = c0 >> kLargeBlockLog2, bx1 = c1 >> kLargeBlockLog2, by0 = r0 >> kLargeBlockLog2,
                  by1 = r1 >> kLargeBlockLog2;
        const int nbx = bx1 - bx0 + 1;
        const long long nblocks = (long long)nbx * (by1 - by0 + 1);
        for (long long j = stripe; j < nblocks; j += kLargeStripes) {
            const int bx = bx0 + (int)(j % nbx), by = by0 + (int)(j / nbx);
            const int cl = max(c0, bx * kB), ch = min(c1, bx * kB + kB - 1);
            const int rl = max(r0, by * kB), rh = min(r1, by * kB + kB - 1);
            // conservative reject: evaluate every edge at the block corner where it is largest
            const int pxl = 16 * cl, pxh = 16 * ch, pyl = 16 * rl, pyh = 16 * rh;
            const E m0 = (E)dx0 * ((dx0 >= 0 ? pyh : pyl) - y1) - (E)dy0 * ((dy0 >= 0 ? pxl : pxh) - x1);
            const E m1 = (E)dx1 * ((dx1 >= 0 ? pyh : pyl) - y2) - (E)dy1 * ((dy1 >= 0 ? pxl : pxh) - x2);
            const E m2 = (E)dx2 * ((dx2 >= 0 ? pyh : pyl) - y0) - (E)dy2 * ((dy2 >= 0 ? pxl : pxh) - x0);
            if (m0 < bias0 || m1 < bias1 || m2 < bias2) continue;
            scan(cl, ch, rl, rh);
        }
    }
}

template <bool LARGE>
__device__ __forceinline__ void warp_raster(int x0, int y0, int x1, int y1, int x2, int y2, float z0, float z1, float z2,
                                            uint32_t id, int W, int H, unsigned long long *depth_view, int stripe,
                                            unsigned lane)
{
    const int ext_x = max(x0, max(x1, x2)) - min(x0, min(x1, x2));
    const int ext_y = max(y0, max(y1, y2)) - min(y0, min(y1, y2));
    // int32 is exact while every product stays below 2^29: extent < 2^14 (1024 px) plus the 8x4 footprint overhang
    if (ext_x < 16384 && ext_y < 16384)
        warp_raster_impl<LARGE, int>(x0, y0, x1, y1, x2, y2, z0, z1, z2, id, W, H, depth_view, stripe, lane);
    else
        warp_raster_impl<LARGE, long long>(x0, y0, x1, y1, x2, y2, z0, z1, z2, id, W, H, depth_view, stripe, lane);
}

__device__ __forceinline__ float plane_dist(int k, const float4 &p)
{
    switch (k) {
    case 0: return p.z + p.w;
    case 1: return p.w - p.z;
    case 2: return p.x + WR_GUARD_BAND * p.w;
    case 3: return WR_GUARD_BAND * p.w - p.x;
    case 4: return p.y + WR_GUARD_BAND * p.w;
    default: return WR_GUARD_BAND * p.w - p.y;
    }
}

__device__ __forceinline__ float lerp1(float a, float b, float t) { return (b - a) * t + a; }

// Sutherland-Hodgman against near, far and the four guard-band planes, fixed order (DESIGN.md 3.2c).
// Executed by one lane; poly / tmp live in shared memory.
__device__ int clip_polygon(float4 *poly, float4 *tmp, int n)
{
    float d[12];
    for (int k = 0; k < 6; ++k) {
        for (int i = 0; i < n; ++i) d[i] = plane_dist(k, poly[i]);
        int m = 0;
        for (int i = 0; i < n; ++i) {
            const int j = (i + 1 == n) ? 0 : i + 1;
            const bool in_i = d[i] >= 0.0f, in_j = d[j] >= 0.0f;
            if (in_i) tmp[m++] = poly[i];
            if (in_i != in_j) {
                const float t = d[i] / (d[i] - d[j]);
                float4 q;
                q.x = lerp1(poly[i].x, poly[j].x, t);
                q.y = lerp1(poly[i].y, poly[j].y, t);
                q.z = lerp1(poly[i].z, poly[j].z, t);
                q.w = lerp1(poly[i].w, poly[j].w, t);
                tmp[m++] = q;
            }
        }
        n = m;
        if (n < 3) return 0;
        for (int i = 0; i < n; ++i) poly[i] = tmp[i];
    }
    return n;
}

struct WarpClipScratch {
    float4 poly[12];
    float4 tmp[12];
    int X[12], Y[12];
    float zw[12];
    int n;
};

template <bool LARGE>
__device__ __forceinline__ void raster_queue(const RasterParams &P, const VtxSrc &src, int b, WarpClipScratch *clip_smem,
                                             bool slow_only = false)
{
    const unsigned lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long warps_total = (long long)gridDim.x * 8;
    const long long gw = (long long)blockIdx.x * 8 + warp;
    const int count = P.counters[4 * b + (LARGE ? 1 : 0)];
    const uint32_t *qv = P.queue + (size_t)b * P.Fq;
    unsigned long long *depth_view = P.depth + (size_t)b * P.H * P.W;
    const long long items = LARGE ? (long long)count * kLargeStripes : (long long)count;

#pragma unroll 1
    for (long long wi = gw; wi < items; wi += warps_total) {
        const int qi = LARGE ? (int)(wi / kLargeStripes) : (int)wi;
        const int stripe = LARGE ? (int)(wi % kLargeStripes) : 0;
        const uint32_t entry = LARGE ? qv[P.Fq - 1 - qi] : qv[qi];
        const uint32_t id = entry & ~WR_QUEUE_SLOW;
        const int t = (int)id - P.tri_base;
        const int i0 = __ldg(P.tri + 3 * (size_t)t), i1 = __ldg(P.tri + 3 * (size_t)t + 1),
                  i2 = __ldg(P.tri + 3 * (size_t)t + 2);
        if (!(entry & WR_QUEUE_SLOW)) {
            if (slow_only) continue;  // the tile pass owns the representable large triangles of this view
            SnapVert a, c, d;
            if (P.sv) {
                const size_t vb = (size_t)b * P.V;
                a = load_sv(P.sv, vb + i0); c = load_sv(P.sv, vb + i1); d = load_sv(P.sv, vb + i2);
            } else {  // multi-view fast path: no 16-byte snapped vertices in scratch, recompute (same expressions)
                a = snap_one(wr_load_clip(src, b, i0), P.W, P.H);
                c = snap_one(wr_load_clip(src, b, i1), P.W, P.H);
                d = snap_one(wr_load_clip(src, b, i2), P.W, P.H);
            }
            warp_raster<LARGE>(a.x, a.y, c.x, c.y, d.x, d.y, a.zw, c.zw, d.zw, id, P.W, P.H, depth_view, stripe, lane);
        } else if (LARGE) {
            WarpClipScratch &S = clip_smem[warp];
            __syncwarp();
            if (lane == 0) {
                S.poly[0] = wr_load_clip(src, b, i0);
                S.poly[1] = wr_load_clip(src, b, i1);
                S.poly[2] = wr_load_clip(src, b, i2);
                int n = clip_polygon(S.poly, S.tmp, 3);
                for (int i = 0; i < n; ++i) {
                    const float4 p = S.poly[i];
                    bool ok = false;
                    if (p.w > 0.0f) {
                        const float rw = 1.0f / p.w;
                        const float fx = (p.x * (float)(8 * P.W)) * rw;
                        const float fy = (p.y * (float)(8 * P.H)) * rw;
                        if (fabsf(fx) <= WR_COORD_LIMIT && fabsf(fy) <= WR_COORD_LIMIT) {
                            S.X[i] = __float2int_rn(fx) + (8 * P.W - 8);
                            S.Y[i] = __float2int_rn(fy) + (8 * P.H - 8);
                            S.zw[i] = p.z * rw;
                            ok = true;
                        }
                    }
                    if (!ok) { n = 0; break; }  // unrepresentable vertex: drop the whole polygon
                }
                S.n = n;
            }
            __syncwarp();
            const int n = S.n;
            for (int i = 1; i + 1 < n; ++i)  // fan (0, i, i+1); sub-triangles keep the parent id
                warp_raster<LARGE>(S.X[0], S.Y[0], S.X[i], S.Y[i], S.X[i + 1], S.Y[i + 1], S.zw[0], S.zw[i],
                                   S.zw[i + 1], id, P.W, P.H, depth_view, stripe, lane);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Tile pass for LARGE triangles (pixel bbox above kMediumMaxPix): binning + fine raster with the triangle lists of
// a band of tiles staged in shared memory and the depth / id resolve in registers.
//
// A warp per triangle (the medium class) issues one global atomicMin per covered sample; for a triangle of a
// million samples that is a million L2 atomics from 64 warps, with ~75 instructions per 8 x 4 footprint.  Here a
// block OWNS a band of kTileBand 32 x 32-pixel tiles; inside a tile every thread keeps four pixels (a column strip
// of four rows) of packed (depth key << 32 | id) values in registers.  The large queue of the view is walked in
// batches of 256 triangles; per band and batch:
//   stage   thread k fetches triangle k of the batch -- snapped vertices, orientation, 1 / area, z/w, the three
//           edge functions at the band's first sample with their per-column / per-row steps -- into shared memory;
//   bin     the same thread tests its triangle against the band's tiles: bounding box, then every edge at the tile
//           corner where it is largest (the coarse reject); a warp ballot per tile turns the verdicts into the
//           tile's triangle list, a 256-bit mask in shared memory;
//   fine    tile after tile, all 256 threads walk the set bits of the tile's mask (broadcast reads) and test their
//           four samples against each listed triangle: one addition and one comparison per edge and row, in int32
//           when the triangle's extent keeps every value below 2^30 and in int64 otherwise (exact either way); a
//           covered sample updates the thread's register copy;
//   resolve every pixel that was hit does ONE atomicMin on the global buffer (it may already hold a nearer small
//           triangle).
// Two block barriers per band and batch.  Same integers, same float expressions as warp_raster_impl, and a
// minimum is order independent, so results are identical bit for bit.  Triangles that need geometric clipping
// (WR_QUEUE_SLOW) stay with the stripe pass; views with more than kTileMaxQueue large triangles too (every band
// scans the whole queue, which stops paying off).
constexpr int kTile = 32;
constexpr int kTileBand = 8;
constexpr int kTileMaxQueue = 2048;
constexpr int kTileMinAvgTiles = 128;   // average pixel-bbox area of a large triangle, in tiles, from which the tile pass is used

struct TileTri {         // one staged triangle, orientation normalised
    long long e[3];      // edge functions at the sample of the band's first pixel
    int sx[3], sy[3];    // step per column / per row
    float inv_area, z[3];
    uint32_t id;
    uint32_t flags;      // bits 0-2: edge k excludes samples exactly on it; bit 3: int32 is exact around the band
};

struct TileScratch {
    TileTri tri[256];
    unsigned mask[kTileBand][8];   // tile, warp: which of the warp's 32 staged triangles are on the tile's list
};

template <typename E>
__device__ __forceinline__ void tile_fine(const TileTri &T, int col, int ly, unsigned long long (&best)[4])
{
    E e0 = (E)T.e[0] + (E)T.sx[0] * col + (E)T.sy[0] * ly;
    E e1 = (E)T.e[1] + (E)T.sx[1] * col + (E)T.sy[1] * ly;
    E e2 = (E)T.e[2] + (E)T.sx[2] * col + (E)T.sy[2] * ly;
    const E b0 = T.flags & 1u, b1 = (T.flags >> 1) & 1u, b2 = (T.flags >> 2) & 1u;
    const float inv_area = T.inv_area, z0 = T.z[0], z1 = T.z[1], z2 = T.z[2];
    const uint32_t id = T.id;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (e0 >= b0 && e1 >= b1 && e2 >= b2) {
            const float w0 = edge_to_float<E>(e0) * inv_area;
            const float w1 = edge_to_float<E>(e1) * inv_area;
            const float w2 = (1.0f - w0) - w1;
            float zw = ((z0 * w0) + (z1 * w1)) + (z2 * w2);
            zw = zw + 0.0f;
            if (zw >= -1.0f && zw <= 1.0f) {
                const unsigned long long packed = ((unsigned long long)wr_depth_key(zw) << 32) | id;
                best[j] = packed < best[j] ? packed : best[j];
            }
        }
        e0 += (E)T.sy[0]; e1 += (E)T.sy[1]; e2 += (E)T.sy[2];
    }
}

__device__ __forceinline__ void raster_tiles(const RasterParams &P, const VtxSrc &src, int b, int nlarge, TileScratch &S)
{
    const int W = P.W, H = P.H;
    const int tiles_x = (W + kTile - 1) / kTile, tiles_y = (H + kTile - 1) / kTile;
    const int bands_x = (tiles_x + kTileBand - 1) / kTileBand;
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lx = (int)lane, ly = (int)warp * 4;   // this thread's column and first row inside a tile
    const uint32_t *qv = P.queue + (size_t)b * P.Fq;
    unsigned long long *depth_view = P.depth + (size_t)b * H * W;
#pragma unroll 1
    for (int band = blockIdx.x; band < bands_x * tiles_y; band += gridDim.x) {
        const int tx0 = (band % bands_x) * kTileBand, ty = band / bands_x;
        const int ntx = min(kTileBand, tiles_x - tx0);
        const int r0 = ty * kTile, r1 = min(r0 + kTile, H) - 1;
        const int bc0 = tx0 * kTile, bc1 = min(bc0 + ntx * kTile, W) - 1;   // pixel columns of the band
#pragma unroll 1
        for (int base = 0; base < nlarge; base += 256) {
            // ---- stage + bin: triangle base + tid, once per band
            unsigned hit = 0;   // bit t: on the list of tile t of the band
            const int qi = base + (int)tid;
            if (qi < nlarge) {
                const uint32_t entry = qv[P.Fq - 1 - qi];
                if (!(entry & WR_QUEUE_SLOW)) {
                    const int t = (int)entry - P.tri_base;
                    const int i0 = __ldg(P.tri + 3 * (size_t)t), i1 = __ldg(P.tri + 3 * (size_t)t + 1),
                              i2 = __ldg(P.tri + 3 * (size_t)t + 2);
                    SnapVert a, c, d;
                    if (P.sv) {
                        const size_t vb = (size_t)b * P.V;
                        a = load_sv(P.sv, vb + i0); c = load_sv(P.sv, vb + i1); d = load_sv(P.sv, vb + i2);
                    } else {
                        a = snap_one(wr_load_clip(src, b, i0), W, H);
                        c = snap_one(wr_load_clip(src, b, i1), W, H);
                        d = snap_one(wr_load_clip(src, b, i2), W, H);
                    }
                    int x0 = a.x, y0 = a.y, x1 = c.x, y1 = c.y, x2 = d.x, y2 = d.y;
                    float z0 = a.zw, z1 = c.zw, z2 = d.zw;
                    long long area2 = (long long)(x1 - x0) * (y2 - y0) - (long long)(y1 - y0) * (x2 - x0);
                    if (area2 < 0) {
                        int ti; float tf;
                        ti = x1; x1 = x2; x2 = ti;
                        ti = y1; y1 = y2; y2 = ti;
                        tf = z1; z1 = z2; z2 = tf;
                        area2 = -area2;
                    }
                    const int xmin = min(x0, min(x1, x2)), xmax = max(x0, max(x1, x2));
                    const int ymin = min(y0, min(y1, y2)), ymax = max(y0, max(y1, y2));
                    const int cl = max(ceil_div16(xmin), bc0), ch = min(floor_div16(xmax), bc1);
                    const int rl = max(ceil_div16(ymin), r0), rh = min(floor_div16(ymax), r1);
                    if (area2 != 0 && cl <= ch && rl <= rh) {
                        const int vx[3] = { x0, x1, x2 }, vy[3] = { y0, y1, y2 };
                        const int pyl = 16 * rl, pyh = 16 * rh;
                        TileTri T;
                        // int32 is exact while every value stays below 2^31: extent < 2^14 plus the band (2^12 + 2^9)
                        T.flags = (xmax - xmin < 16384 && ymax - ymin < 16384) ? 8u : 0u;
                        hit = ((1u << (ch / kTile - tx0 + 1)) - 1u) & ~((1u << (cl / kTile - tx0)) - 1u);  // bbox columns
#pragma unroll
                        for (int k = 0; k < 3; ++k) {
                            const int k1 = (k + 1) % 3, k2 = (k + 2) % 3;   // edge k runs from vertex k1 to vertex k2
                            const int dx = vx[k2] - vx[k1], dy = vy[k2] - vy[k1];
                            const long long bias = top_left(dx, dy) ? 0 : 1;
                            T.flags |= (uint32_t)bias << k;
                            T.e[k] = (long long)dx * (16 * r0 - vy[k1]) - (long long)dy * (16 * bc0 - vx[k1]);
                            T.sx[k] = -16 * dy;
                            T.sy[k] = 16 * dx;
                            // coarse reject per tile: the edge at the corner of the clipped box where it is largest
                            const long long my = (long long)dx * ((dx >= 0 ? pyh : pyl) - vy[k1]);
                            for (int tt = 0; tt < ntx; ++tt) {
                                if (!(hit >> tt & 1u)) continue;
                                const int tcl = max(cl, bc0 + tt * kTile), tch = min(ch, bc0 + tt * kTile + kTile - 1);
                                const long long m = my - (long long)dy * ((dy >= 0 ? 16 * tcl : 16 * tch) - vx[k1]);
                                if (m < bias) hit &= ~(1u << tt);
                            }
                        }
                        if (hit) {
                            T.inv_area = 1.0f / __ll2float_rn(area2);
                            T.z[0] = z0; T.z[1] = z1; T.z[2] = z2;
                            T.id = entry;
                            S.tri[tid] = T;
                        }
                    }
                }
            }
            unsigned any = 0;
#pragma unroll
            for (int tt = 0; tt < kTileBand; ++tt) {
                const unsigned m = __ballot_sync(0xFFFFFFFFu, (hit >> tt) & 1u);
                if (lane == 0) S.mask[tt][warp] = m;
                any |= m;
            }
            if (__syncthreads_or(any != 0) == 0) continue;   // nothing of this batch touches the band
            // ---- fine + resolve, tile after tile
#pragma unroll 1
            for (int tt = 0; tt < ntx; ++tt) {
                unsigned long long best[4] = { WR_EMPTY_PIXEL, WR_EMPTY_PIXEL, WR_EMPTY_PIXEL, WR_EMPTY_PIXEL };
                const int col = tt * kTile + lx;   // column relative to the band
                bool touched = false;
#pragma unroll 1
                for (int w = 0; w < 8; ++w) {
                    unsigned bits = S.mask[tt][w];
                    touched |= bits != 0;
                    while (bits) {
                        const TileTri &Ts = S.tri[32 * w + __ffs(bits) - 1];
                        bits &= bits - 1u;
                        if (Ts.flags & 8u) tile_fine<int>(Ts, col, ly, best);
                        else tile_fine<long long>(Ts, col, ly, best);
                    }
                }
                const int cx = bc0 + col;
                if (touched && cx <= bc1) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int ry = r0 + ly + j;
                        if (ry <= r1 && best[j] != WR_EMPTY_PIXEL) atomicMin(depth_view + ((size_t)ry * W + cx), best[j]);
                    }
                }
            }
            __syncthreads();   // the lists have been consumed: the next batch may overwrite them
        }
    }
}

// Medium queue (one warp per triangle) then large / clipped queue (64 warps per triangle) in one launch.
__global__ void __launch_bounds__(256, 3) k_raster_queues(RasterParams P, VtxSrc src, int view0)
{
    __shared__ WarpClipScratch clip_smem[8];
    __shared__ TileScratch tile_smem;
    wr_pdl_wait();
    wr_pdl_trigger();
    const int b = blockIdx.y + view0;
    raster_queue<false>(P, src, b, clip_smem);
    // Large triangles: the tile pass when the view queued few enough of them and they are large against a tile
    // (measured, tools/exp_big.py: from ~128 tiles of pixel bounding box per triangle on average); below that the
    // stripe pass' parallelism wins.
    const int nlarge = P.counters[4 * b + 1];
    const bool tiles = nlarge > 0 && nlarge <= kTileMaxQueue &&
                       (long long)P.counters[4 * b + 2] >= (long long)kTileMinAvgTiles * nlarge;
    raster_queue<true>(P, src, b, clip_smem, tiles);
    if (tiles) raster_tiles(P, src, b, nlarge, tile_smem);
}

// (u, v, z/w) of the winning triangle at a pixel centre from the unsnapped clip-space vertices
// (DESIGN.md 3.4).  Shared with the fused render kernel through common include below.
__global__ void __launch_bounds__(256) k_resolve_rast(unsigned long long *packed, VtxSrc src, const int32_t *tri,
                                                      int H, int W, float *rast, int32_t *tri_id)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    const int b = blockIdx.z;
    if (c >= W) return;
    const size_t o = ((size_t)b * H + r) * W + c;
    const unsigned long long pk = packed[o];
    float4 out = make_float4(0.f, 0.f, 0.f, 0.f);
    int id = -1;
    if (pk != WR_EMPTY_PIXEL) {
        packed[o] = WR_EMPTY_PIXEL;  // self-cleaning: the next call skips the clear
        id = (int)(uint32_t)(pk & 0xFFFFFFFFull);
        const int i0 = __ldg(tri + 3 * (size_t)id), i1 = __ldg(tri + 3 * (size_t)id + 1), i2 = __ldg(tri + 3 * (size_t)id + 2);
        const float4 p0 = wr_load_clip(src, b, i0), p1 = wr_load_clip(src, b, i1), p2 = wr_load_clip(src, b, i2);
        const float fx = (float)(2 * c + 1 - W) / (float)W;
        const float fy = (float)(2 * r + 1 - H) / (float)H;
        const float p0x = p0.x - fx * p0.w, p0y = p0.y - fy * p0.w;
        const float p1x = p1.x - fx * p1.w, p1y = p1.y - fy * p1.w;
        const float p2x = p2.x - fx * p2.w, p2y = p2.y - fy * p2.w;
        const float a0 = p1x * p2y - p1y * p2x;
        const float a1 = p2x * p0y - p2y * p0x;
        const float a2 = p0x * p1y - p0y * p1x;
        const float iw = 1.0f / ((a0 + a1) + a2);
        const float b0 = a0 * iw, b1 = a1 * iw;
        const float z = ((p0.z * a0) + (p1.z * a1)) + (p2.z * a2);
        const float w = ((p0.w * a0) + (p1.w * a1)) + (p2.w * a2);
        const float zw = z / w;
        out.x = (b0 >= 0.0f) ? (b0 > 1.0f ? 1.0f : b0) : 0.0f;
        out.y = (b1 >= 0.0f) ? (b1 > 1.0f ? 1.0f : b1) : 0.0f;
        out.z = (zw >= -1.0f) ? (zw > 1.0f ? 1.0f : zw) : -1.0f;
        out.w = (float)(id + 1);
    }
    if (rast) reinterpret_cast<float4 *>(rast)[o] = out;
    if (tri_id) tri_id[o] = id;
}

}  // namespace

// Runs snap -> setup -> queue rasterisation into the context scratch.  `extra_bytes` of additional
// scratch are reserved behind the raster buffers and returned through `extra`.
int wr_run_raster(wr_ctx *ctx, const VtxSrc &src, int B, const int32_t *tri, int F, const int32_t *tri_ranges,
                  int H, int W, size_t extra_bytes, RasterResult *res, void **extra, cudaStream_t stream,
                  VertexPack *pack)
{
    const int V = src.V;
    // Multi-view fast path (k_snap_mv / k_setup_mv): fused render of a mesh whose triangles are small for this
    // viewport.  Coarse meshes keep the per-view kernels with several lanes per triangle.
    const bool use_mv = src.mvp && !tri_ranges && W <= 2048 && H <= 2048 && F > 0 && V > 0 &&
                        (long long)F * 4 > (long long)H * W && (long long)V * B < (1ll << 31);
    const size_t sv_bytes = use_mv ? wr_align256((size_t)V * B * sizeof(int2))
                                   : wr_align256((size_t)B * (size_t)(V > 0 ? V : 1) * sizeof(SnapVert));
    const size_t depth_bytes = wr_align256((size_t)B * H * W * sizeof(unsigned long long));
    const size_t queue_bytes = wr_align256((size_t)B * (size_t)(F > 0 ? F : 1) * sizeof(uint32_t));
    const size_t stats_bytes = wr_align256((size_t)B * 8 * sizeof(int));
    const size_t total = sv_bytes + depth_bytes + queue_bytes + stats_bytes + wr_align256(extra_bytes);
    int rc = wr_scratch_reserve(ctx, total, stream);
    if (rc != WR_OK) return rc;
    char *base = static_cast<char *>(ctx->scratch);
    // the packed buffer sits at offset 0 so that its "known clean" prefix survives calls of any shape
    unsigned long long *depth = reinterpret_cast<unsigned long long *>(base);
    SnapVert *sv = reinterpret_cast<SnapVert *>(base + depth_bytes);
    uint32_t *queue = reinterpret_cast<uint32_t *>(base + sv_bytes + depth_bytes);
    int *stats = reinterpret_cast<int *>(base + sv_bytes + depth_bytes + queue_bytes);  // [B,4] counters + [B,4] user
    char *extra_base = base + sv_bytes + depth_bytes + queue_bytes + stats_bytes;
    if (extra) *extra = extra_base;
    VertexPack vp;
    vp.v_nrm = nullptr; vp.Vn = 0; vp.offset = 0; vp.pos4 = nullptr; vp.nrm4 = nullptr;
    if (pack) {
        pack->pos4 = reinterpret_cast<float4 *>(extra_base + pack->offset);
        pack->nrm4 = pack->v_nrm ? reinterpret_cast<float4 *>(extra_base + pack->offset + wr_align256((size_t)(V > 0 ? V : 1) * 16))
                                 : nullptr;
        vp = *pack;
    }

    wr_stage(ctx, stream, "clear");
    const size_t packed_bytes = (size_t)B * H * W * sizeof(unsigned long long);
    cudaError_t e;
    if (ctx->clean_bytes < packed_bytes) {
        e = cudaMemsetAsync(depth, 0xFF, packed_bytes, stream);
        if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "memset depth");
    }
    ctx->clean_bytes = 0;  // dirty until the consuming kernel has been launched
    const bool have_work = F > 0 && V > 0 && B > 0;
    if (!have_work) {  // no snap kernel will run: clear the counter block here
        e = cudaMemsetAsync(stats, 0, (size_t)B * 8 * sizeof(int), stream);
        if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "memset counters");
    }
    res->packed = depth;
    res->packed_bytes = packed_bytes;
    res->view_stats = stats + 4 * B;

    if (have_work) {
        RasterParams P;
        if ((long long)B * V >= (1ll << 31)) return WR_ERR_UNSUPPORTED;  // 32-bit snapped-vertex record index
        P.sv = sv; P.tri = tri; P.F = F; P.V = V; P.tri_base = 0; P.W = W; P.H = H;
        P.depth = depth; P.queue = queue; P.Fq = F; P.counters = stats;
        // Persistent queue pass.  A mesh of (sub-)pixel triangles rarely queues anything, and then only a few
        // triangles (a ground plane under a dense object): a quarter of the grid is plenty for those and an empty
        // pass drains 1.5 us sooner on config B.
        const int qgrid = ((long long)F * 4 > (long long)H * W) ? (ctx->sm_count + 1) / 2 : ctx->sm_count * 2;
        wr_stage(ctx, stream, "k_snap_vertices");
        if (use_mv) {
            MvParams M;
            uint2 *rec = reinterpret_cast<uint2 *>(sv);
            M.rec = rec; M.tri = tri; M.F = F; M.V = V; M.B = B; M.Bq = B;
            M.W = W; M.H = H; M.HW = (unsigned)H * (unsigned)W;
            const int lo_c = 2048 - W / 2, lo_r = 2048 - H / 2;
            M.lo_px = (unsigned)lo_c | ((unsigned)lo_r << 16);
            M.hi_px = (unsigned)(lo_c + W - 1) | ((unsigned)(lo_r + H - 1) << 16);
            M.depth = depth; M.queue = queue; M.Fq = F; M.counters = stats;
            P.sv = nullptr;  // the queue pass recomputes the few snapped vertices it needs
            // stored = snapped (centred) + 8 W - 8 (relative to the sample of pixel 0) + 16 lo_c (bias)
            k_snap_mv<<<wr_div_up(vp.nrm4 && vp.Vn > V ? vp.Vn : V, 256), 256, 0, stream>>>(
                src, B, W, H, 8 * W - 8 + 16 * lo_c, 8 * H - 8 + 16 * lo_r, rec, stats, B * 8, vp);
            WR_CHECK_LAUNCH(ctx, "k_snap_mv");
            wr_stage(ctx, stream, "k_setup_triangles");
            const bool pdl = !ctx->profiling;
            wr_launch(k_setup_mv, dim3(wr_div_up(F, 256), B), dim3(256), stream, pdl, M, P, src);
            WR_CHECK_LAUNCH(ctx, "k_setup_mv");
            wr_stage(ctx, stream, "k_raster_queues");
            wr_launch(k_raster_queues, dim3(qgrid, B), dim3(256), stream, pdl, P, src, 0);
            WR_CHECK_LAUNCH(ctx, "k_raster_queues");
            return WR_OK;
        }
        if (src.mvp)
            k_snap_vertices_allviews<<<wr_div_up(vp.nrm4 && vp.Vn > V ? vp.Vn : V, 256), 256, 0, stream>>>(
                src, B, W, H, sv, stats, B * 8, vp);
        else
            k_snap_vertices<<<dim3(wr_div_up(V, 256), B), 256, 0, stream>>>(src, 0, W, H, sv, stats, B * 8);
        WR_CHECK_LAUNCH(ctx, "k_snap_vertices");
        if (!tri_ranges) {
            wr_stage(ctx, stream, "k_setup_triangles");
            const bool pdl = !ctx->profiling && src.mvp != nullptr;  // the chain starts at k_snap_vertices_allviews
            // coarse mesh for this viewport (expected bounding box of a triangle above ~8 samples): several lanes per
            // triangle.  2 / 4 / 8 lanes measured 38.4 / 36.7 / 41.0 us on config A (profiles/README.md).
            constexpr int kCoarseLanes = 4;
            const bool lpt4 = (long long)F * 4 <= (long long)H * W;
            if (lpt4)
                wr_launch(k_setup_triangles<kCoarseLanes>, dim3(wr_div_up((long long)F * kCoarseLanes, 256), B), dim3(256),
                          stream, pdl, P, 0);
            else
                wr_launch(k_setup_triangles<1>, dim3(wr_div_up(F, 256), B), dim3(256), stream, pdl, P, 0);
            WR_CHECK_LAUNCH(ctx, "k_setup_triangles");
            wr_stage(ctx, stream, "k_raster_queues");
            wr_launch(k_raster_queues, dim3(qgrid, B), dim3(256), stream, pdl, P, src, 0);
            WR_CHECK_LAUNCH(ctx, "k_raster_queues");
        } else {
            for (int b = 0; b < B; ++b) {
                const int start = tri_ranges[2 * b], count = tri_ranges[2 * b + 1];
                if (start < 0 || count < 0 || (long long)start + count > F) return WR_ERR_INVALID_ARGUMENT;
                if (count == 0) continue;
                RasterParams Q = P;
                Q.tri = tri + 3 * (size_t)start; Q.F = count; Q.tri_base = start;
                k_setup_triangles<1><<<dim3(wr_div_up(count, 256), 1), 256, 0, stream>>>(Q, b);
                WR_CHECK_LAUNCH(ctx, "k_setup_triangles(range)");
                k_raster_queues<<<dim3(qgrid, 1), 256, 0, stream>>>(Q, src, b);
                WR_CHECK_LAUNCH(ctx, "k_raster_queues(range)");
            }
        }
    }
    return WR_OK;
}

extern "C" int wr_rasterize(wr_ctx *ctx, const float *pos, int B, int V, int pos_batched, const int32_t *tri, int F,
                            const int32_t *tri_ranges, int H, int W, float *rast, int32_t *tri_id, void *stream_)
{
    if (!ctx || B < 0 || V < 0 || F < 0 || H <= 0 || W <= 0 || H > 8192 || W > 8192) return WR_ERR_INVALID_ARGUMENT;
    if (F >= (1 << 30)) return WR_ERR_UNSUPPORTED;
    // the rast tensor carries the id as (float)(id + 1): exact up to 2^24 faces only (the triangle-id output has no
    // such limit)
    if (rast && F > (1 << 24)) return WR_ERR_UNSUPPORTED;
    if ((V > 0 && !pos) || (F > 0 && !tri)) return WR_ERR_INVALID_ARGUMENT;
    if (B == 0) return WR_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    VtxSrc src;
    src.pos = pos; src.mvp = nullptr; src.V = V; src.batched = pos_batched ? 1 : 0;
    RasterResult res;
    wr_stage_begin(ctx);
    int rc = wr_run_raster(ctx, src, B, tri, F, tri_ranges, H, W, 0, &res, nullptr, stream);
    if (rc != WR_OK) return rc;
    if (rast || tri_id) {
        wr_stage(ctx, stream, "k_resolve_rast");
        k_resolve_rast<<<dim3(wr_div_up(W, 256), H, B), 256, 0, stream>>>(res.packed, src, tri, H, W, rast, tri_id);
        WR_CHECK_LAUNCH(ctx, "k_resolve_rast");
        wr_raster_consumed(ctx, &res);
    }
    wr_stage(ctx, stream, "end");
    return WR_OK;
}
