// Atlas post-processing behind uv_blend (reference uv.py:426-461) on sm_100a:
//
//   wr_poisson_blend   PoissonBlendingSolver.__call__ blend.py:214-324.  The reference builds gathered index
//                      lists (A [N,4] int64) and launches one Jacobi kernel per sweep with a
//                      cudaDeviceSynchronize after each (blend.py:60-100).  Here the solve region stays a 2-D
//                      image: planar, zero-padded scratch planes, and a temporally blocked stencil kernel
//                      that runs 8 sweeps per launch out of registers (4x8 points per thread; up / down
//                      neighbours through two shared-memory rows per warp, left / right by warp shuffle).
//   wr_inpaint         uv_padding -> inpaint_cvc uv.py:373-382, cv_ops.py:11-35: quantisation contract of the
//                      reference, fill by jump flooding + inverse-square-distance average (the cvcuda operator
//                      is third-party and absent; see oracle/wr_oracle_blend.c for the statement of the fill).
//                      wr_uv_padding_sets fills up to four 3-channel atlases from one jump flood.
//
// CPU statement of both: oracle/wr_oracle_blend.c (bit-identical results; the library is compiled with
// -fmad=false and IEEE division).
#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// Poisson blending
// ------------------------------------------------------------------------------------------------
constexpr int kPbHalo = 8;                      // sweeps per launch = halo width of a region
constexpr int kPbRegW = 128, kPbRegH = 64;      // region held by one block (32 x 64 / kPbRows threads)
constexpr int kPbOutW = kPbRegW - 2 * kPbHalo;  // 112
constexpr int kPbOutH = kPbRegH - 2 * kPbHalo;  // 48
constexpr int kPbRows = 8;                      // region rows per thread (4 columns wide)

struct PbPlanes {
    int H, W, C;
    int Hp, Wp;        // padded plane: kPbHalo zero rows / columns in front, rounded up to whole tiles behind
    int r0;            // image row of plane row kPbHalo (0, or the first row of a band)
    float *xa, *xb;    // [C,Hp,Wp] iterate (0 outside the solve region), ping-pong
    float *b;          // [C,Hp,Wp] right-hand side
    uint8_t *m;        // [Hp,Wp] solve region (image border removed, blend.py:233-236)
};

__device__ __forceinline__ float pb_px(const float *img, int H, int W, int C, int r, int c, int ch)
{
    if (r < 0 || r >= H || c < 0 || c >= W) return 0.0f;  // F.conv2d zero padding
    return __ldg(img + ((size_t)r * W + c) * C + ch);
}
__device__ __forceinline__ bool pb_in(const uint8_t *mask, int H, int W, int r, int c)
{
    return r > 0 && r < H - 1 && c > 0 && c < W - 1 && __ldg(mask + (size_t)r * W + c) != 0;
}

// One thread per padded-plane pixel: region mask, right-hand side (laplacian of the guidance + the fixed
// boundary neighbours, blend.py:243-299) and the initial iterate, all channels.
__global__ void __launch_bounds__(256) k_pb_setup(const float *src, const uint8_t *mask, const float *tgt, PbPlanes P,
                                                  int grad_mode)
{
    const int pc = blockIdx.x * blockDim.x + threadIdx.x;
    const int pr = blockIdx.y;
    if (pc >= P.Wp) return;
    const int r = pr + P.r0 - kPbHalo, c = pc - kPbHalo;
    const size_t po = (size_t)pr * P.Wp + pc;
    const size_t plane = (size_t)P.Hp * P.Wp;
    const bool inside = r >= 0 && r < P.H && c >= 0 && c < P.W;
    const bool m = inside && pb_in(mask, P.H, P.W, r, c);
    P.m[po] = m ? 1 : 0;
    const int dr[4] = {-1, 1, 0, 0}, dc[4] = {0, 0, -1, 1};  // up, down, left, right (blend.py:289-297)
    bool nm[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) nm[k] = inside && pb_in(mask, P.H, P.W, r + dr[k], c + dc[k]);
    for (int ch = 0; ch < P.C; ++ch) {
        float bval = 0.0f, x0 = 0.0f;
        if (m) {
            const float tc = pb_px(tgt, P.H, P.W, P.C, r, c, ch);
            float tn[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) tn[k] = pb_px(tgt, P.H, P.W, P.C, r + dr[k], c + dc[k], ch);
            const float sc = pb_px(src, P.H, P.W, P.C, r, c, ch);
            float lap;
            if (grad_mode == 0) {
                lap = 4.0f * sc;
#pragma unroll
                for (int k = 0; k < 4; ++k) lap = lap - pb_px(src, P.H, P.W, P.C, r + dr[k], c + dc[k], ch);
            } else {
                lap = 0.0f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float ds = sc - pb_px(src, P.H, P.W, P.C, r + dr[k], c + dc[k], ch);
                    const float dt = tc - tn[k];
                    const float pick = (grad_mode == 1) ? (fabsf(ds) > fabsf(dt) ? ds : dt) : (ds + dt) * 0.5f;
                    lap = (k == 0) ? pick : lap + pick;
                }
            }
            float fq = 0.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float v = nm[k] ? 0.0f : tn[k];
                fq = (k == 0) ? v : fq + v;
            }
            bval = lap + fq;
            x0 = tc;
        }
        P.b[ch * plane + po] = bval;
        P.xa[ch * plane + po] = x0;
        P.xb[ch * plane + po] = x0;
    }
}

// `sweeps` (<= kPbHalo) Jacobi sweeps of one 128x64 region of one channel plane; the inner 112x48 points are
// exact after them (every sweep invalidates one more ring of the region) and are written to xout.
// R = rows of the region per thread (4 columns wide): 4 -> 512 threads, 8 -> 256 threads with twice the
// independent work per thread and half the barriers, shuffles and shared-memory rows per point.
template <int R>
__global__ void __launch_bounds__(32 * (kPbRegH / R), 2) k_pb_jacobi(const float *__restrict__ xin, float *__restrict__ xout,
                                                                     const float *__restrict__ bpl,
                                                                     const uint8_t *__restrict__ mpl, int Hp, int Wp,
                                                                     int sweeps)
{
    constexpr int kBands = kPbRegH / R;           // warps per block
    __shared__ float4 s_top[2][kBands][32];       // first row of every warp's R-row band, per parity
    __shared__ float4 s_bot[2][kBands][32];       // last row
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const size_t plane = (size_t)Hp * Wp;
    const size_t chan = (size_t)blockIdx.z * plane;
    const int pr0 = blockIdx.y * kPbOutH + R * ty;  // padded-plane coordinates of this thread's R x 4 patch
    const int pc0 = blockIdx.x * kPbOutW + 4 * tx;
    // patch lies in the region's output tile (the halo is a whole number of patches in both directions)
    const bool owner = tx >= 2 && tx < 30 && ty >= kPbHalo / R && ty < (kPbRegH - kPbHalo) / R;
    static_assert(kPbHalo % R == 0 && kPbRegH % R == 0 && R * 4 <= 32, "patch rows must tile the halo");

    // The region mask and the right-hand side were written by k_pb_setup, before the previous sweep launch: in a
    // dependent launch they may be requested ahead of the wait, and the iterate right behind it, so that all three
    // round trips of a block overlap (and overlap the tail of the previous launch).
    wr_pdl_trigger();
    uchar4 mm[R];
    float4 x[R], b[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
        mm[i] = __ldg(reinterpret_cast<const uchar4 *>(mpl + (size_t)(pr0 + i) * Wp + pc0));
        b[i] = __ldg(reinterpret_cast<const float4 *>(bpl + chan + (size_t)(pr0 + i) * Wp + pc0));
    }
    wr_pdl_wait();
#pragma unroll
    for (int i = 0; i < R; ++i) x[i] = *reinterpret_cast<const float4 *>(xin + chan + (size_t)(pr0 + i) * Wp + pc0);
    unsigned mbits = 0;
#pragma unroll
    for (int i = 0; i < R; ++i)
        mbits |= ((mm[i].x ? 1u : 0u) | (mm[i].y ? 2u : 0u) | (mm[i].z ? 4u : 0u) | (mm[i].w ? 8u : 0u)) << (4 * i);
    // nothing to solve in the output tile: both ping-pong planes already hold the same values there
    if (__syncthreads_or(owner && mbits != 0) == 0) return;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    // Most warps lie entirely inside or entirely outside the solve region: the per-point mask selects (three
    // instructions each) are only executed by the warps that straddle its outline, and warps outside do nothing
    // but keep their (zero) rows published.  The branch is warp-uniform; every warp still reaches the barrier.
    constexpr unsigned kAll = R * 4 == 32 ? 0xFFFFFFFFu : ((1u << (R * 4)) - 1u);
    const bool w_full = __all_sync(0xFFFFFFFFu, mbits == kAll);
    const bool w_empty = __all_sync(0xFFFFFFFFu, mbits == 0u);
#pragma unroll 1
    for (int s = 0; s < sweeps; ++s) {
        const int par = s & 1;
        s_top[par][ty][tx] = x[0];
        s_bot[par][ty][tx] = x[R - 1];
        __syncthreads();
        if (w_empty) continue;
        const float4 up = ty > 0 ? s_bot[par][ty - 1][tx] : zero4;
        const float4 dn = ty < kBands - 1 ? s_top[par][ty + 1][tx] : zero4;
        float4 above = up;
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const float4 cur = x[i];
            const float4 below = (i < R - 1) ? x[i + 1] : dn;
            float lf = __shfl_up_sync(0xFFFFFFFFu, cur.w, 1);
            float rt = __shfl_down_sync(0xFFFFFFFFu, cur.x, 1);
            if (tx == 0) lf = 0.0f;
            if (tx == 31) rt = 0.0f;
            float4 n;
            n.x = ((((above.x + below.x) + lf) + cur.y) + b[i].x) * 0.25f;  // blend.py:69, left to right
            n.y = ((((above.y + below.y) + cur.x) + cur.z) + b[i].y) * 0.25f;
            n.z = ((((above.z + below.z) + cur.y) + cur.w) + b[i].z) * 0.25f;
            n.w = ((((above.w + below.w) + cur.z) + rt) + b[i].w) * 0.25f;
            if (w_full) {
                x[i] = n;
            } else {
                const unsigned mb = mbits >> (4 * i);
                x[i].x = (mb & 1u) ? n.x : 0.0f;
                x[i].y = (mb & 2u) ? n.y : 0.0f;
                x[i].z = (mb & 4u) ? n.z : 0.0f;
                x[i].w = (mb & 8u) ? n.w : 0.0f;
            }
            above = cur;
        }
    }
    if (owner) {
#pragma unroll
        for (int i = 0; i < R; ++i)
            *reinterpret_cast<float4 *>(xout + chan + (size_t)(pr0 + i) * Wp + pc0) = x[i];
    }
}

// Output atlases of k_pb_finish: one, or every rank's (peer stores: the finish of a band solve is its all-gather)
struct PbOut {
    float *p[WR_MAX_P2P_RANKS];
    int n;
};

// out = tgt outside the region, clamp(X, 0, 1) inside (blend.py:317-321); one thread per pixel of plane row
// blockIdx.y + kPbHalo, image row blockIdx.y + P.r0
__global__ void __launch_bounds__(256) k_pb_finish(const float *tgt, PbPlanes P, const float *x, PbOut out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y + P.r0;
    if (c >= P.W) return;
    const size_t po = (size_t)(blockIdx.y + kPbHalo) * P.Wp + (c + kPbHalo);
    const size_t plane = (size_t)P.Hp * P.Wp;
    const bool m = P.m[po] != 0;
    const size_t o = ((size_t)r * P.W + c) * P.C;
    for (int ch = 0; ch < P.C; ++ch) {
        float v;
        if (m) {
            v = x[ch * plane + po];
            v = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
        } else {
            v = __ldg(tgt + o + ch);
        }
        for (int k = 0; k < out.n; ++k) out.p[k][o + ch] = v;
    }
}

// The 2 * kPbHalo halo rows of a band's iterate plane x (kPbHalo above its first tile row, kPbHalo below its last),
// all channels, pulled with 16-byte loads from the same plane of the neighbouring bands: the last kPbHalo rows the
// band above owns and the first kPbHalo rows the band below owns.  up / dn are NULL at the edges of the image (the
// rows there are zero padding, written once by k_pb_setup).  Runs between two sweep launches, after a barrier
// behind the neighbours' previous launch.
__global__ void __launch_bounds__(256) k_pb_halo(float *x, int Hp, int Wp, const float *up, int up_Hp, const float *dn,
                                                 int dn_Hp)
{
    wr_pdl_trigger();  // the sweep launch behind may load its region mask and right-hand side meanwhile
    const int q = blockIdx.x * blockDim.x + threadIdx.x;  // float4 of the row
    const int i = blockIdx.y;                             // halo row, 0 .. 2 * kPbHalo - 1
    const bool top = i < kPbHalo;
    const float *nb = top ? up : dn;
    if (4 * q >= Wp || !nb) return;
    const int sr = top ? up_Hp - 2 * kPbHalo + i : i;     // row in the neighbour's plane
    const int dr = top ? i : Hp - 2 * kPbHalo + i;        // row in this band's plane
    const size_t nplane = (size_t)(top ? up_Hp : dn_Hp) * Wp;
    const size_t plane = (size_t)Hp * Wp;
    const float4 v = *(reinterpret_cast<const float4 *>(nb + blockIdx.z * nplane + (size_t)sr * Wp) + q);
    *(reinterpret_cast<float4 *>(x + blockIdx.z * plane + (size_t)dr * Wp) + q) = v;
}

// Tile rows [t0, t1) of the band of `rank`: shard_bounds(tiles_y, world)[rank] of parallel.py (the first
// tiles_y % world bands one tile row taller).  Non-empty bands are ranks 0 .. min(tiles_y, world) - 1.
void pb_band(int tiles_y, int world, int rank, int *t0, int *t1)
{
    const int base = tiles_y / world, extra = tiles_y % world;
    *t0 = rank * base + (rank < extra ? rank : extra);
    *t1 = *t0 + base + (rank < extra ? 1 : 0);
}

// ------------------------------------------------------------------------------------------------
// Seam inpainting
// ------------------------------------------------------------------------------------------------
constexpr int kSeedNone = -1;  // seeds are packed (row << 16 | column): same order as row * W + column

__device__ __forceinline__ int seed_dist2(int r, int c, int s)
{
    const int dy = r - (s >> 16), dx = c - (s & 0xFFFF);
    return dy * dy + dx * dx;
}

__global__ void __launch_bounds__(256) k_jfa_init(const uint8_t *mask, int H, int W, int invert, int *seed)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (c >= W) return;
    const size_t p = (size_t)r * W + c;
    const bool fill = (mask[p] != 0) != (invert != 0);
    seed[p] = fill ? kSeedNone : ((r << 16) | c);
}

__global__ void __launch_bounds__(256) k_jfa_pass(const int *__restrict__ sin, int *__restrict__ sout, int H, int W,
                                                  int step)
{
    wr_pdl_wait();   // every pass reads the seeds of the previous one
    wr_pdl_trigger();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (c >= W) return;
    int best = sin[(size_t)r * W + c];
    int bd = best == kSeedNone ? 0 : seed_dist2(r, c, best);
#pragma unroll
    for (int j = -1; j <= 1; ++j) {
        const int rr = r + j * step;
        if (rr < 0 || rr >= H) continue;
#pragma unroll
        for (int k = -1; k <= 1; ++k) {
            const int cc = c + k * step;
            if (cc < 0 || cc >= W) continue;
            const int s = __ldg(sin + (size_t)rr * W + cc);
            if (s == kSeedNone) continue;
            const int d = seed_dist2(r, c, s);
            if (best == kSeedNone || d < bd || (d == bd && s < best)) { best = s; bd = d; }
        }
    }
    sout[(size_t)r * W + c] = best;
}

template <typename T> struct Quant;
template <> struct Quant<uint8_t> {
    static __device__ __forceinline__ float load(const uint8_t *p) { return (float)__ldg(p); }
    static __device__ __forceinline__ void store(uint8_t *p, float q) { *p = (uint8_t)q; }
};
template <> struct Quant<float> {  // cv_ops.py:23-24 on the way in (after uv.py:381's clamp), :35 on the way out
    static __device__ __forceinline__ float load(const float *p)
    {
        float v = __ldg(p);
        v = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
        return (float)(int)(v * 255.0f);
    }
    static __device__ __forceinline__ void store(float *p, float q) { *p = q / 255.0f; }
};

template <typename T>
__global__ void __launch_bounds__(256) k_inpaint_fill(const T *img, const uint8_t *mask, int invert, const int *seed,
                                                      int H, int W, int C, int radius, T *out)
{
    wr_pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (c >= W) return;
    const size_t p = (size_t)r * W + c;
    const bool fill = (mask[p] != 0) != (invert != 0);
    const int q = seed[p];
    if (!fill || q == kSeedNone) {
        for (int ch = 0; ch < C; ++ch) Quant<T>::store(out + p * C + ch, Quant<T>::load(img + p * C + ch));
        return;
    }
    const int qr = q >> 16, qc = q & 0xFFFF;
    const float num = (float)(1 + seed_dist2(r, c, q));
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, ws = 0.0f;
    for (int tr = max(qr - radius, 0); tr <= min(qr + radius, H - 1); ++tr)
        for (int tc = max(qc - radius, 0); tc <= min(qc + radius, W - 1); ++tc) {
            if ((tr - qr) * (tr - qr) + (tc - qc) * (tc - qc) > radius * radius) continue;
            const size_t t = (size_t)tr * W + tc;
            if ((__ldg(mask + t) != 0) != (invert != 0)) continue;
            const int dy = r - tr, dx = c - tc;
            const float w = num / (float)(1 + dy * dy + dx * dx);
            for (int ch = 0; ch < C; ++ch) acc[ch] = acc[ch] + w * Quant<T>::load(img + t * C + ch);
            ws = ws + w;
        }
    for (int ch = 0; ch < C; ++ch) {
        float v = rintf(acc[ch] / ws);
        v = v > 255.0f ? 255.0f : v;
        Quant<T>::store(out + p * C + ch, v);
    }
}

// k_inpaint_fill<float> with C = 3 for up to WR_MAX_BAKE_SETS images against one mask and one seed map: every known
// neighbour is visited and weighted once for all K images.  Each channel gets the float operations of k_inpaint_fill
// in the same order, so out[k] is what k_inpaint_fill writes for in[k].
struct PadSets {
    const float *in[WR_MAX_BAKE_SETS];
    float *out[WR_MAX_BAKE_SETS];
};

template <int K>
__global__ void __launch_bounds__(256) k_inpaint_fill_sets(PadSets S, const uint8_t *inside, const int *seed, int H,
                                                           int W, int radius)
{
    wr_pdl_wait();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = blockIdx.y;
    if (c >= W) return;
    const size_t p = (size_t)r * W + c;
    const int q = seed[p];
    if (inside[p] != 0 || q == kSeedNone) {
#pragma unroll
        for (int k = 0; k < K; ++k)
            for (int ch = 0; ch < 3; ++ch) Quant<float>::store(S.out[k] + p * 3 + ch, Quant<float>::load(S.in[k] + p * 3 + ch));
        return;
    }
    const int qr = q >> 16, qc = q & 0xFFFF;
    const float num = (float)(1 + seed_dist2(r, c, q));
    float acc[K][3], ws = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k][0] = acc[k][1] = acc[k][2] = 0.f;
    for (int tr = max(qr - radius, 0); tr <= min(qr + radius, H - 1); ++tr)
        for (int tc = max(qc - radius, 0); tc <= min(qc + radius, W - 1); ++tc) {
            if ((tr - qr) * (tr - qr) + (tc - qc) * (tc - qc) > radius * radius) continue;
            const size_t t = (size_t)tr * W + tc;
            if (__ldg(inside + t) == 0) continue;
            const int dy = r - tr, dx = c - tc;
            const float w = num / (float)(1 + dy * dy + dx * dx);
#pragma unroll
            for (int k = 0; k < K; ++k)
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) acc[k][ch] = acc[k][ch] + w * Quant<float>::load(S.in[k] + t * 3 + ch);
            ws = ws + w;
        }
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            float v = rintf(acc[k][ch] / ws);
            v = v > 255.0f ? 255.0f : v;
            Quant<float>::store(S.out[k] + p * 3 + ch, v);
        }
}

// scratch behind the packed raster buffer's clean prefix, so a bake between two renders does not cost a clear
char *blend_scratch(wr_ctx *ctx, size_t bytes, cudaStream_t stream, int *rc)
{
    const size_t keep = wr_align256(ctx->clean_bytes);
    *rc = wr_scratch_reserve(ctx, keep + bytes, stream);
    if (*rc != WR_OK) return nullptr;
    return static_cast<char *>(ctx->scratch) + wr_align256(ctx->clean_bytes);  // clean_bytes is 0 after a regrow
}

// Jump flood of the known pixels of `mask` into the context scratch (opens the call's profiling stages); *seed: the
// seed map the fill reads.
int run_jfa(wr_ctx *ctx, const uint8_t *mask, int mask_is_inside, int H, int W, cudaStream_t stream, const int **seed)
{
    const size_t n = (size_t)H * W;
    int rc;
    char *base = blend_scratch(ctx, 2 * wr_align256(n * sizeof(int)), stream, &rc);
    if (!base) return rc;
    int *sa = reinterpret_cast<int *>(base), *sb = reinterpret_cast<int *>(base + wr_align256(n * sizeof(int)));
    const dim3 grid(wr_div_up(W, 256), H);
    wr_stage_begin(ctx);
    wr_stage(ctx, stream, "k_jfa_init");
    k_jfa_init<<<grid, 256, 0, stream>>>(mask, H, W, mask_is_inside, sa);
    WR_CHECK_LAUNCH(ctx, "k_jfa_init");
    int top = 1;
    while (top < (H > W ? H : W)) top <<= 1;
    wr_stage(ctx, stream, "k_jfa_pass");
    for (int step = top >> 1;; step >>= 1) {
        const int s = step >= 1 ? step : 1;  // the sequence ends with a second pass of step 1
        wr_launch(k_jfa_pass, grid, dim3(256), stream, true, (const int *)sa, sb, H, W, s);
        WR_CHECK_LAUNCH(ctx, "k_jfa_pass");
        int *t = sa; sa = sb; sb = t;
        if (step < 1) break;
    }
    *seed = sa;
    return WR_OK;
}

template <typename T>
int run_inpaint(wr_ctx *ctx, const T *img, const uint8_t *mask, int mask_is_inside, int H, int W, int C, int radius,
                T *out, cudaStream_t stream)
{
    if (!ctx || !img || !mask || !out || H <= 0 || W <= 0 || C <= 0 || C > 4 || radius < 0 || radius > 64)
        return WR_ERR_INVALID_ARGUMENT;
    if (H > 16384 || W > 16384) return WR_ERR_UNSUPPORTED;
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const int *seed = nullptr;
    const int rc = run_jfa(ctx, mask, mask_is_inside, H, W, stream, &seed);
    if (rc != WR_OK) return rc;
    const dim3 grid(wr_div_up(W, 256), H);
    wr_stage(ctx, stream, "k_inpaint_fill");
    wr_launch(k_inpaint_fill<T>, grid, dim3(256), stream, !ctx->profiling, img, mask, mask_is_inside, seed, H, W, C, radius,
              out);
    WR_CHECK_LAUNCH(ctx, "k_inpaint_fill");
    wr_stage(ctx, stream, "end");
    return WR_OK;
}

}  // namespace

extern "C" int wr_poisson_blend(wr_ctx *ctx, const float *src, const uint8_t *mask, const float *tgt, int H, int W,
                                int C, int num_iters, int grad_mode, float *out, void *stream_)
{
    if (!ctx || !src || !mask || !tgt || !out || H <= 0 || W <= 0 || C <= 0 || C > 4 || num_iters < 0 ||
        grad_mode < 0 || grad_mode > 2)
        return WR_ERR_INVALID_ARGUMENT;
    if (H > 16384 || W > 16384) return WR_ERR_UNSUPPORTED;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    PbPlanes P;
    P.H = H; P.W = W; P.C = C; P.r0 = 0;
    const int tiles_x = wr_div_up(W, kPbOutW), tiles_y = wr_div_up(H, kPbOutH);
    P.Wp = tiles_x * kPbOutW + 2 * kPbHalo;
    P.Hp = tiles_y * kPbOutH + 2 * kPbHalo;
    const size_t plane_bytes = wr_align256((size_t)P.Hp * P.Wp * sizeof(float) * C);
    const size_t mask_bytes = wr_align256((size_t)P.Hp * P.Wp);
    int rc;
    char *base = blend_scratch(ctx, 3 * plane_bytes + mask_bytes, stream, &rc);
    if (!base) return rc;
    P.xa = reinterpret_cast<float *>(base);
    P.xb = reinterpret_cast<float *>(base + plane_bytes);
    P.b = reinterpret_cast<float *>(base + 2 * plane_bytes);
    P.m = reinterpret_cast<uint8_t *>(base + 3 * plane_bytes);

    wr_stage_begin(ctx);
    wr_stage(ctx, stream, "k_pb_setup");
    k_pb_setup<<<dim3(wr_div_up(P.Wp, 256), P.Hp), 256, 0, stream>>>(src, mask, tgt, P, grad_mode);
    WR_CHECK_LAUNCH(ctx, "k_pb_setup");
    wr_stage(ctx, stream, "k_pb_jacobi");
    float *xin = P.xa, *xout = P.xb;
    for (int done = 0; done < num_iters; done += kPbHalo) {
        const int sweeps = num_iters - done < kPbHalo ? num_iters - done : kPbHalo;
        // every launch after the first is a dependent launch of its predecessor (the first follows k_pb_setup, whose
        // outputs it reads before its wait, so it is serialised normally)
        wr_launch(k_pb_jacobi<kPbRows>, dim3(tiles_x, tiles_y, C), dim3(32 * (kPbRegH / kPbRows)), stream, done > 0,
                  (const float *)xin, xout, (const float *)P.b, (const uint8_t *)P.m, P.Hp, P.Wp, sweeps);
        WR_CHECK_LAUNCH(ctx, "k_pb_jacobi");
        float *t = xin; xin = xout; xout = t;
    }
    wr_stage(ctx, stream, "k_pb_finish");
    PbOut po = {};
    po.p[0] = out;
    po.n = 1;
    k_pb_finish<<<dim3(wr_div_up(W, 256), H), 256, 0, stream>>>(tgt, P, xin, po);
    WR_CHECK_LAUNCH(ctx, "k_pb_finish");
    wr_stage(ctx, stream, "end");
    return WR_OK;
}

extern "C" int wr_poisson_band_layout(int H, int W, int C, int world, int rank, int num_iters, uint64_t *plane_bytes,
                                      uint64_t *mask_bytes, int *steps, int *row_lo, int *row_hi)
{
    if (H <= 0 || W <= 0 || C <= 0 || C > 4 || world < 1 || world > WR_MAX_P2P_RANKS || rank < 0 || rank >= world ||
        num_iters < 0)
        return WR_ERR_INVALID_ARGUMENT;
    if (H > 16384 || W > 16384) return WR_ERR_UNSUPPORTED;
    int t0, t1;
    pb_band(wr_div_up(H, kPbOutH), world, rank, &t0, &t1);
    const uint64_t Hb = t1 > t0 ? (uint64_t)(t1 - t0) * kPbOutH + 2 * kPbHalo : 0;
    const uint64_t Wp = (uint64_t)wr_div_up(W, kPbOutW) * kPbOutW + 2 * kPbHalo;
    if (plane_bytes) *plane_bytes = Hb * Wp * sizeof(float) * C;
    if (mask_bytes) *mask_bytes = Hb * Wp;
    if (steps) *steps = wr_div_up(num_iters, kPbHalo);
    if (row_lo) *row_lo = t0 * kPbOutH < H ? t0 * kPbOutH : H;
    if (row_hi) *row_hi = t1 * kPbOutH < H ? t1 * kPbOutH : H;
    return WR_OK;
}

extern "C" int wr_poisson_band_step(wr_ctx *ctx, const wr_poisson_band_args *args, void *stream_)
{
    if (!ctx || !args) return WR_ERR_INVALID_ARGUMENT;
    const wr_poisson_band_args &A = *args;
    if (A.H <= 0 || A.W <= 0 || A.C <= 0 || A.C > 4 || A.num_iters < 0 || A.grad_mode < 0 || A.grad_mode > 2 ||
        A.world < 1 || A.world > WR_MAX_P2P_RANKS || A.rank < 0 || A.rank >= A.world)
        return WR_ERR_INVALID_ARGUMENT;
    if (A.H > 16384 || A.W > 16384) return WR_ERR_UNSUPPORTED;
    const int S = wr_div_up(A.num_iters, kPbHalo);
    if (A.step < 0 || A.step > S + 1) return WR_ERR_INVALID_ARGUMENT;
    const int tiles_x = wr_div_up(A.W, kPbOutW), tiles_y = wr_div_up(A.H, kPbOutH);
    int t0, t1;
    pb_band(tiles_y, A.world, A.rank, &t0, &t1);
    if (t1 == t0) return WR_OK;  // no tile row here: this rank only takes part in the barriers
    // neighbouring bands (empty bands are the last ranks, so they are rank -1 / +1)
    const int up = t0 > 0 ? A.rank - 1 : -1, dn = t1 < tiles_y ? A.rank + 1 : -1;
    auto misaligned = [](const void *p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) != 0; };
    if (!A.src || !A.mask || !A.tgt || !A.b || !A.m || misaligned(A.b, 16) || misaligned(A.m, 4))
        return WR_ERR_INVALID_ARGUMENT;
    for (int r : {A.rank, up, dn}) {
        if (r < 0) continue;
        if (!A.xa[r] || !A.xb[r] || misaligned(A.xa[r], 16) || misaligned(A.xb[r], 16)) return WR_ERR_INVALID_ARGUMENT;
    }
    for (int r = 0; r < A.world; ++r)
        if (!A.out[r]) return WR_ERR_INVALID_ARGUMENT;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");

    // the band's planes: its tile rows plus kPbHalo rows on either side, the layout of wr_poisson_blend's planes
    auto band_rows = [&](int r) {
        int a, b;
        pb_band(tiles_y, A.world, r, &a, &b);
        return (b - a) * kPbOutH + 2 * kPbHalo;
    };
    PbPlanes P;
    P.H = A.H; P.W = A.W; P.C = A.C;
    P.Wp = tiles_x * kPbOutW + 2 * kPbHalo;
    P.Hp = band_rows(A.rank);
    P.r0 = t0 * kPbOutH;
    P.xa = A.xa[A.rank]; P.xb = A.xb[A.rank]; P.b = A.b; P.m = A.m;
    // launch j (1 .. S) reads plane (j - 1) % 2 and writes plane j % 2 (xa = 0), as in wr_poisson_blend
    float *const planes[2] = {P.xa, P.xb};

    wr_stage_begin(ctx);
    if (A.step == 0) {
        wr_stage(ctx, stream, "k_pb_setup");
        k_pb_setup<<<dim3(wr_div_up(P.Wp, 256), P.Hp), 256, 0, stream>>>(A.src, A.mask, A.tgt, P, A.grad_mode);
        WR_CHECK_LAUNCH(ctx, "k_pb_setup");
    } else if (A.step <= S) {
        const int par = (A.step - 1) & 1;
        // launch 1 reads the iterate k_pb_setup wrote on every rank alike: its halo rows are already right
        const bool halo = A.step > 1 && (up >= 0 || dn >= 0);
        if (halo) {
            const float *const *nb = par ? A.xb : A.xa;
            wr_stage(ctx, stream, "k_pb_halo");
            k_pb_halo<<<dim3(wr_div_up(P.Wp / 4, 256), 2 * kPbHalo, P.C), 256, 0, stream>>>(
                planes[par], P.Hp, P.Wp, up >= 0 ? nb[up] : nullptr, up >= 0 ? band_rows(up) : 0,
                dn >= 0 ? nb[dn] : nullptr, dn >= 0 ? band_rows(dn) : 0);
            WR_CHECK_LAUNCH(ctx, "k_pb_halo");
        }
        const int done = (A.step - 1) * kPbHalo;
        const int sweeps = A.num_iters - done < kPbHalo ? A.num_iters - done : kPbHalo;
        wr_stage(ctx, stream, "k_pb_jacobi");
        wr_launch(k_pb_jacobi<kPbRows>, dim3(tiles_x, t1 - t0, P.C), dim3(32 * (kPbRegH / kPbRows)), stream,
                  halo && !ctx->profiling, (const float *)planes[par], planes[par ^ 1], (const float *)P.b,
                  (const uint8_t *)P.m, P.Hp, P.Wp, sweeps);
        WR_CHECK_LAUNCH(ctx, "k_pb_jacobi");
    } else {
        PbOut po = {};
        for (int r = 0; r < A.world; ++r) po.p[r] = A.out[r];
        po.n = A.world;
        const int rows = (t1 * kPbOutH < A.H ? t1 * kPbOutH : A.H) - P.r0;
        wr_stage(ctx, stream, "k_pb_finish");
        k_pb_finish<<<dim3(wr_div_up(A.W, 256), rows), 256, 0, stream>>>(A.tgt, P, planes[S & 1], po);
        WR_CHECK_LAUNCH(ctx, "k_pb_finish");
    }
    wr_stage(ctx, stream, "end");
    return WR_OK;
}

extern "C" int wr_inpaint_u8(wr_ctx *ctx, const uint8_t *img, const uint8_t *mask, int H, int W, int C, int radius,
                             uint8_t *out, void *stream)
{
    return run_inpaint<uint8_t>(ctx, img, mask, 0, H, W, C, radius, out, static_cast<cudaStream_t>(stream));
}

extern "C" int wr_uv_padding(wr_ctx *ctx, const float *attr, const uint8_t *inside_mask, int H, int W, int C,
                             int radius, float *out, void *stream)
{
    return run_inpaint<float>(ctx, attr, inside_mask, 1, H, W, C, radius, out, static_cast<cudaStream_t>(stream));
}

extern "C" int wr_uv_padding_sets(wr_ctx *ctx, const float *const *attr, const uint8_t *inside_mask, int H, int W, int K,
                                  int radius, float *const *out, void *stream_)
{
    if (!ctx || !attr || !out || !inside_mask || H <= 0 || W <= 0 || K < 1 || K > WR_MAX_BAKE_SETS || radius < 0 ||
        radius > 64)
        return WR_ERR_INVALID_ARGUMENT;
    PadSets S = {};
    for (int k = 0; k < K; ++k) {
        if (!attr[k] || !out[k]) return WR_ERR_INVALID_ARGUMENT;
        S.in[k] = attr[k];
        S.out[k] = out[k];
    }
    if (H > 16384 || W > 16384) return WR_ERR_UNSUPPORTED;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaSetDevice");
    const int *seed = nullptr;
    const int rc = run_jfa(ctx, inside_mask, 1, H, W, stream, &seed);
    if (rc != WR_OK) return rc;
    const dim3 grid(wr_div_up(W, 256), H);
    wr_stage(ctx, stream, "k_inpaint_fill_sets");
    auto launch = [&](auto kernel) {
        wr_launch(kernel, grid, dim3(256), stream, !ctx->profiling, S, inside_mask, seed, H, W, radius);
    };
    switch (K) {
    case 1: launch(k_inpaint_fill_sets<1>); break;
    case 2: launch(k_inpaint_fill_sets<2>); break;
    case 3: launch(k_inpaint_fill_sets<3>); break;
    default: launch(k_inpaint_fill_sets<4>); break;
    }
    WR_CHECK_LAUNCH(ctx, "k_inpaint_fill_sets");
    wr_stage(ctx, stream, "end");
    return WR_OK;
}
