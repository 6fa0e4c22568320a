// raster.cu -- forward rasteriser: one warp per CTA, two neighbouring 16x8 screen tiles per warp, a 2x2 pixel
// quad per lane, z-buffer in registers.
//
// Replaces the GL draw loop + upload_background/download_pixels of the reference
// (csrc/rasterise_egl.cpp:349-396, csrc/rasterise_egl.cu:10-38,65-91): the background is read
// and the output written directly in the [B,H,W,C] tensors, top row first.
//
// A pair of tiles with nothing binned to either is copied in one go, both tiles' loads in flight (such a tile is pure
// latency: count -> background -> store).  Otherwise, per tile, the tile's bin (KIND_SMALL faces, int32 arithmetic
// only; its place is a function of the tile index, so count and references arrive in one hop), the image's overflow
// list if the bin was full, and the image's large list (KIND_LARGE: int64 tile-origin move; KIND_HARD: homogeneous
// fp64) are consumed in chunks of 32:
//   lane phase  : one face per lane -- load its 64-B coverage record, move the three edge functions
//                 to the tile origin, reject faces whose edge functions are negative on the whole
//                 tile, bound the face's nearest depth key over the tile, park survivors in shared
//                 memory;
//   warp phase  : survivors are taken nearest-first (REDUX.MIN over the bounds) and broadcast to all
//                 lanes, each lane testing its four pixels (S5, S7); the loop stops as soon as the
//                 nearest remaining bound is farther than every pixel already covered.
// The visible face of a pixel is min (depth key, face index) -- order independent, so neither the list
// order nor the early exit can change the result.
// Shape choices (one warp per CTA, pairs, the form of the warp-phase loop) are measured: DESIGN.md section 4.
#include "common.cuh"

namespace dirt {

#ifndef DIRT_RASTER_WARPS
#define DIRT_RASTER_WARPS 1   // one warp per CTA, 32 CTAs per SM: measured best (profiles/r01_sweep_warps2.txt) -- tiles retire
#endif                        // independently and the shared-memory slot addresses are compile-time constants
constexpr int WARPS_PER_BLOCK = DIRT_RASTER_WARPS;
#ifndef DIRT_RASTER_TILES
#define DIRT_RASTER_TILES 2   // tiles (neighbours in x) per warp: measured 0.167 -> 0.152 ms at cfg3 (empty pairs are copied together)
#endif
constexpr int TILES_PER_WARP = DIRT_RASTER_TILES;
#ifndef DIRT_RASTER_PREFETCH_BG
#define DIRT_RASTER_PREFETCH_BG 0
#endif
#ifndef DIRT_RASTER_MIN_BLOCKS
#define DIRT_RASTER_MIN_BLOCKS 32   // x 32 threads: <= 64 registers, measured best (profiles/r01_sweep_bounds.txt, _warps2.txt)
#endif

struct __align__(16) Slot {
    int32_t A0, B0, A1, B1;
    int32_t A2, B2, Q0, Q1;
    int32_t Q2;
    float zA, zB, zC;
    int32_t face, kind, pad0, pad1;
};
static_assert(sizeof(Slot) == 64, "Slot must be 64 bytes");

// best (depth key, face) of the lane's four pixels, packed key<<32 | face so one unsigned compare orders both
struct Quad {
    unsigned long long best[4];   // [0]=(row0,col0) [1]=(row0,col1) [2]=(row1,col0) [3]=(row1,col1)
};

__device__ __forceinline__ unsigned long long pack(uint32_t key, int32_t face)
{
    return ((unsigned long long)key << 32) | (uint32_t)face;
}

__device__ __forceinline__ int32_t clamp_q(int64_t q)
{
    const int64_t lim = (int64_t)1 << 30;
    return (int32_t)(q > lim ? lim : (q < -lim ? -lim : q));
}

// hard faces (H1-H3): homogeneous double-precision evaluation at this lane's four pixels.
// Returns the depth keys (0xFFFFFFFF where the pixel is not covered).
__device__ __noinline__ uint4 hard_face_keys(const float* __restrict__ verts, const TriInterp* __restrict__ itp_b,
                                             int face, int H, int W, int col0, int row0)
{
    const int4 ids = __ldg(reinterpret_cast<const int4*>(itp_b + face) + 2);   // {sC, v0, v1, v2}
    float p[3][4];
    const int vid[3] = {ids.y, ids.z, ids.w};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(verts) + vid[k]);
        p[k][0] = v.x; p[k][1] = v.y; p[k][2] = v.z; p[k][3] = v.w;
    }
    double gq[3][3], gs[3], gz[3];
    uint32_t keys[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
    // the same IEEE divisions the host does for Dims::ps (kept local: this path is rare and the hot loop's register
    // allocation is sensitive to the signature of its caller)
    PixelScale ps;
    ps.two_over_W = __ddiv_rn(2.0, (double)W); ps.two_over_H = __ddiv_rn(2.0, (double)H);
    ps.inv_W = __ddiv_rn(1.0, (double)W); ps.inv_H = __ddiv_rn(1.0, (double)H);
    if (exact::planes_double(p, ps, gq, gs, gz)) {
#pragma unroll
        for (int pix = 0; pix < 4; ++pix) {
            const int row = row0 + (pix >> 1), col = col0 + (pix & 1);
            bool in = true;
            double qv[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double v = exact::plane_double(gq[k], col, row);
                qv[k] = v;
                const bool own = gq[k][0] > 0.0 || (gq[k][0] == 0.0 && gq[k][1] > 0.0);
                if (!(v > 0.0 || (v == 0.0 && own))) in = false;
            }
            const double sum = __dadd_rn(__dadd_rn(qv[0], qv[1]), qv[2]);
            in = in && (sum > 0.0);
            const float z = (float)exact::plane_double(gz, col, row);
            if (in) keys[pix] = exact::depth_key(z);
        }
    }
    return make_uint4(keys[0], keys[1], keys[2], keys[3]);
}

// Consume one face list for this warp's tile.  SMALL: the list holds KIND_SMALL faces only.  FILTER: the list holds
// (tile, face) pairs of the whole image (the overflow list) and only those of tile `want_tile` count.
template <bool SMALL, bool FILTER>
__device__ __forceinline__ void consume_list(const int* __restrict__ list, int count, int want_tile, const TriCov* __restrict__ cov_b,
                                             const TriInterp* __restrict__ itp_b, const float* __restrict__ verts,
                                             Slot* slots, int lane, int tcol0, int trow0, int H, int W, Quad& quad,
                                             uint32_t& tile_max)
{
    int col0 = tcol0 + (lane & 7) * 2, row0 = trow0 + (lane >> 3) * 2;   // this lane's quad: (row0..row0+1) x (col0..col0+1)
    const float tc0 = (float)tcol0, tc1 = (float)(tcol0 + TILE_W - 1), tr0 = (float)trow0, tr1 = (float)(trow0 + TILE_H - 1);

    for (int base = 0; base < count; base += 32) {
        const int i = base + lane;
        int f = -1;
        if (i < count) {
            if (FILTER) {
                const int2 e = __ldg(reinterpret_cast<const int2*>(list) + i);
                f = (e.x == want_tile) ? e.y : -1;
            } else {
                f = __ldg(&list[i]);
            }
        }
        if (FILTER && !__any_sync(0xffffffffu, f >= 0)) continue;
        uint32_t order = 0xFFFFFFFFu;   // (nearest possible depth key << 5) | lane; 0xFFFFFFFF: not a candidate
        if (f >= 0) {
            const TriCov c = load_cov(cov_b + f);
            Slot s;
            s.face = f; s.kind = (int32_t)c.s.kind; s.pad0 = s.pad1 = 0;
            s.A0 = c.A0; s.B0 = c.B0; s.A1 = c.A1; s.B1 = c.B1; s.A2 = c.A2; s.B2 = c.B2;
            bool alive = false;
            float zA, zB, zC;
            if (SMALL || c.s.kind == KIND_SMALL) {
                const int oc = tcol0 - c.s.cref, orow = trow0 - c.s.rref;
                s.Q0 = c.s.q0r + c.A0 * oc + c.B0 * orow;
                s.Q1 = c.s.q1r + c.A1 * oc + c.B1 * orow;
                s.Q2 = c.s.q2r + c.A2 * oc + c.B2 * orow;
                zA = c.s.zA; zB = c.s.zB; zC = c.s.zC;
                // the largest value each edge function takes on the tile's pixel centres
                const int m0 = s.Q0 + max(0, (TILE_W - 1) * c.A0) + max(0, (TILE_H - 1) * c.B0);
                const int m1 = s.Q1 + max(0, (TILE_W - 1) * c.A1) + max(0, (TILE_H - 1) * c.B1);
                const int m2 = s.Q2 + max(0, (TILE_W - 1) * c.A2) + max(0, (TILE_H - 1) * c.B2);
                alive = (m0 | m1 | m2) >= 0;
            } else if (c.s.kind == KIND_LARGE) {
                const int64_t Q0 = c.l.q0 + (int64_t)c.A0 * tcol0 + (int64_t)c.B0 * trow0;
                const int64_t Q1 = c.l.q1 + (int64_t)c.A1 * tcol0 + (int64_t)c.B1 * trow0;
                const int64_t Q2 = c.l.q2 + (int64_t)c.A2 * tcol0 + (int64_t)c.B2 * trow0;
                const int64_t m0 = Q0 + max(0, (TILE_W - 1) * c.A0) + max(0, (TILE_H - 1) * c.B0);
                const int64_t m1 = Q1 + max(0, (TILE_W - 1) * c.A1) + max(0, (TILE_H - 1) * c.B1);
                const int64_t m2 = Q2 + max(0, (TILE_W - 1) * c.A2) + max(0, (TILE_H - 1) * c.B2);
                alive = (m0 >= 0) && (m1 >= 0) && (m2 >= 0);
                // clamping keeps every sign: |A*dx + B*dy| < 2^29 inside a tile
                s.Q0 = clamp_q(Q0); s.Q1 = clamp_q(Q1); s.Q2 = clamp_q(Q2);
                zA = c.l.zA; zB = c.l.zB; zC = c.l.zC;
            } else {   // KIND_HARD
                alive = c.s.kind == KIND_HARD;
                s.Q0 = s.Q1 = s.Q2 = 0;
                zA = zB = zC = 0.f;
            }
            s.zA = zA; s.zB = zB; s.zC = zC;
            if (alive) {
                uint32_t kmin = 0;
                if (c.s.kind != KIND_HARD) {
                    // the rounded depth is monotone in col and in row, so its minimum over the tile is at a corner
                    const float z00 = exact::depth_normal(zA, zB, zC, tc0, tr0), z01 = exact::depth_normal(zA, zB, zC, tc1, tr0);
                    const float z10 = exact::depth_normal(zA, zB, zC, tc0, tr1), z11 = exact::depth_normal(zA, zB, zC, tc1, tr1);
                    const float zmin = fminf(fminf(z00, z01), fminf(z10, z11));
                    kmin = (zmin >= 0.f) ? min(exact::depth_key(zmin), KEY_EMPTY) : 0u;   // NaN -> 0 (conservative)
                }
                order = (kmin << 5) | (uint32_t)lane;
                uint4* dst = reinterpret_cast<uint4*>(&slots[lane]);
                const uint4* src = reinterpret_cast<const uint4*>(&s);
                dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
            }
        }
        __syncwarp();
        while (true) {
            const uint32_t nearest = __reduce_min_sync(0xffffffffu, order);
            // strict: a face whose nearest key ties the farthest covered pixel could still win on face index
            if (nearest == 0xFFFFFFFFu || (nearest >> 5) > tile_max) break;
            order = (order == nearest) ? 0xFFFFFFFFu : order;   // orders are unique (the lane index sits in the low bits)
            const Slot s = slots[nearest & 31];
            // Keep just (col0,row0) live across iterations and derive the other per-lane constants here: under the
            // 64-register cap the compiler otherwise spills them or rebuilds them from %tid/%ctaid every iteration.
            asm volatile("" : "+r"(col0), "+r"(row0));
            const int dx = col0 - tcol0, dy = row0 - trow0;
            const float c0f = (float)col0, c1f = (float)(col0 + 1), r0f = (float)row0, r1f = (float)(row0 + 1);
            uint32_t k00, k01, k10, k11;
            if (SMALL || s.kind != (int32_t)KIND_HARD) {
                const int32_t a0 = s.Q0 + s.A0 * dx + s.B0 * dy, a1 = s.Q1 + s.A1 * dx + s.B1 * dy, a2 = s.Q2 + s.A2 * dx + s.B2 * dy;
                const int32_t b0 = a0 + s.B0, b1 = a1 + s.B1, b2 = a2 + s.B2;
                // all-ones where any edge function is negative (pixel outside): OR-ing it in turns the key into "no fragment"
                const uint32_t out00 = (uint32_t)((a0 | a1 | a2) >> 31);
                const uint32_t out01 = (uint32_t)(((a0 + s.A0) | (a1 + s.A1) | (a2 + s.A2)) >> 31);
                const uint32_t out10 = (uint32_t)((b0 | b1 | b2) >> 31);
                const uint32_t out11 = (uint32_t)(((b0 + s.A0) | (b1 + s.A1) | (b2 + s.A2)) >> 31);
                const float zr0 = __fmaf_rn(s.zB, r0f, s.zC), zr1 = __fmaf_rn(s.zB, r1f, s.zC);
                k00 = exact::depth_key(__fmaf_rn(s.zA, c0f, zr0)) | out00;
                k01 = exact::depth_key(__fmaf_rn(s.zA, c1f, zr0)) | out01;
                k10 = exact::depth_key(__fmaf_rn(s.zA, c0f, zr1)) | out10;
                k11 = exact::depth_key(__fmaf_rn(s.zA, c1f, zr1)) | out11;
            } else {
                const uint4 k = hard_face_keys(verts, itp_b, s.face, H, W, col0, row0);
                k00 = k.x; k01 = k.y; k10 = k.z; k11 = k.w;
            }
            const unsigned long long p00 = pack(k00, s.face), p01 = pack(k01, s.face);
            const unsigned long long p10 = pack(k10, s.face), p11 = pack(k11, s.face);
            if (p00 < quad.best[0]) quad.best[0] = p00;
            if (p01 < quad.best[1]) quad.best[1] = p01;
            if (p10 < quad.best[2]) quad.best[2] = p10;
            if (p11 < quad.best[3]) quad.best[3] = p11;
            const uint32_t far = max(max((uint32_t)(quad.best[0] >> 32), (uint32_t)(quad.best[1] >> 32)),
                                     max((uint32_t)(quad.best[2] >> 32), (uint32_t)(quad.best[3] >> 32)));
            tile_max = __reduce_max_sync(0xffffffffu, far);
        }
        __syncwarp();
    }
}

template <int CT>
__device__ __forceinline__ void shade_pixel(const TriInterp& ti, int col, int row, const float* __restrict__ cols,
                                            float* __restrict__ out, int C)
{
    // perspective-correct interpolation c2 + b0*(c0-c2) + b1*(c1-c2): exact for equal vertex colours
    // (tests/square_test.py).  Values only, no decision depends on them.
    const float dc = (float)(col - ti.cref), dr = (float)(row - ti.rref);
    const float S = fmaf(ti.sA, dc, fmaf(ti.sB, dr, ti.sC));
    const float cw = __fdividef(1.0f, S);
    const float b0 = fmaf(ti.q0A, dc, fmaf(ti.q0B, dr, ti.q0C)) * cw;
    const float b1 = fmaf(ti.q1A, dc, fmaf(ti.q1B, dr, ti.q1C)) * cw;
    if (CT == 4) {
        const float4 c0 = __ldg(reinterpret_cast<const float4*>(cols) + ti.v0);
        const float4 c1 = __ldg(reinterpret_cast<const float4*>(cols) + ti.v1);
        const float4 c2 = __ldg(reinterpret_cast<const float4*>(cols) + ti.v2);
        float4 o;
        o.x = fmaf(b0, c0.x - c2.x, fmaf(b1, c1.x - c2.x, c2.x));
        o.y = fmaf(b0, c0.y - c2.y, fmaf(b1, c1.y - c2.y, c2.y));
        o.z = fmaf(b0, c0.z - c2.z, fmaf(b1, c1.z - c2.z, c2.z));
        o.w = fmaf(b0, c0.w - c2.w, fmaf(b1, c1.w - c2.w, c2.w));
        *reinterpret_cast<float4*>(out) = o;
    } else {
        const float* c0 = cols + (size_t)ti.v0 * C;
        const float* c1 = cols + (size_t)ti.v1 * C;
        const float* c2 = cols + (size_t)ti.v2 * C;
        for (int ch = 0; ch < C; ++ch) {
            const float a2 = __ldg(&c2[ch]);
            out[ch] = fmaf(b0, __ldg(&c0[ch]) - a2, fmaf(b1, __ldg(&c1[ch]) - a2, a2));
        }
    }
}

// The same from the face's shading record (C <= 4): value_c = N_c(p) / S(p), the quotient refined once so that equal vertex
// colours give exactly that colour (tests/square_test.py) -- no barycentrics, no vertex-colour gathers.
template <int CT>
__device__ __forceinline__ void shade_pixel_record(const TriShade* __restrict__ rec, int col, int row, float* __restrict__ out, int C)
{
    const float4* r = reinterpret_cast<const float4*>(rec);
    const float4 v0 = __ldg(r), v1 = __ldg(r + 1), v2 = __ldg(r + 2), v3 = __ldg(r + 3);
    const uint32_t ref = __float_as_uint(v0.w);
    const float dc = (float)(col - (int)(ref & 0xffffu)), dr = (float)(row - (int)(ref >> 16));
    const float S = fmaf(v0.x, dc, fmaf(v0.y, dr, v0.z));
    const float rs = __fdividef(1.0f, S);
    auto quotient = [&](float A, float B, float Cc) -> float {
        const float n = fmaf(A, dc, fmaf(B, dr, Cc));
        const float q = n * rs;
        return fmaf(fmaf(-q, S, n), rs, q);
    };
    const float o0 = quotient(v1.x, v1.y, v1.z), o1 = quotient(v1.w, v2.x, v2.y), o2 = quotient(v2.z, v2.w, v3.x), o3 = quotient(v3.y, v3.z, v3.w);
    if (CT == 4) {
        *reinterpret_cast<float4*>(out) = make_float4(o0, o1, o2, o3);
    } else {
        out[0] = o0;
        if (C > 1) out[1] = o1;
        if (C > 2) out[2] = o2;
        if (C > 3) out[3] = o3;
    }
}

// MODE 0: colour forward (pixels [+ face ids]); MODE 1: visibility (face ids and/or G-buffer)
template <int MODE, int CT, bool REC>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32, DIRT_RASTER_MIN_BLOCKS) raster_kernel(
    const float* __restrict__ vertices, const float* __restrict__ background,
    const float* __restrict__ vertex_colors, float* __restrict__ pixels, int32_t* __restrict__ face_ids_out,
    float* __restrict__ gbuffer_out, Workspace ws, Dims d)
{
    __shared__ Slot slots_all[WARPS_PER_BLOCK][32];
    // grid: x = groups of WARPS_PER_BLOCK * TILES_PER_WARP tiles along a tile row, y = tile row, z = image
    const int lane = threadIdx.x & 31;
    const int warp = (WARPS_PER_BLOCK == 1) ? 0 : (int)__reduce_min_sync(0xffffffffu, threadIdx.x >> 5);   // known to be warp-uniform
    const int txb = (blockIdx.x * WARPS_PER_BLOCK + warp) * TILES_PER_WARP, ty = blockIdx.y;
    if (txb >= d.tiles_x) return;
    const int trow0 = ty * TILE_H;
    for (int b = blockIdx.z; b < d.B; b += gridDim.z) {   // gridDim.z == B unless B exceeds the grid limit

    const TriCov* cov_b = ws.cov + (size_t)b * d.F;
    const TriInterp* itp_b = ws.itp + (size_t)b * d.F;
    const float* verts = vertices + (size_t)b * d.V * 4;

#if DIRT_RASTER_TILES == 2
    // Two neighbouring tiles with nothing binned to either (most of a frame): one pass with both tiles' loads in
    // flight -- an empty tile is pure latency (range -> background -> store), so this doubles the bytes per resident warp.
    if (MODE == 0 && (CT == 4 || CT == 3) && txb + 1 < d.tiles_x && (txb + 2) * TILE_W <= d.W && trow0 + TILE_H <= d.H) {
        const int* cp = ws.tile_count + (size_t)b * d.tiles + ty * d.tiles_x + txb;
        const int cnt_a = cp[0], cnt_b = cp[1];
        if (cnt_a == 0 && cnt_b == 0 && ws.large_count[b] == 0) {
            const int col0 = txb * TILE_W + (lane & 7) * 2, row0 = trow0 + (lane >> 3) * 2;
            const size_t l00 = (size_t)row0 * d.W + col0;   // pixel (row0, col0) inside the image
            const size_t p00 = (size_t)b * d.H * d.W + l00;  // ... and in the batch
            const size_t bg00 = (size_t)b * d.bg_stride + l00;   // ... and in the background
            if (CT == 4) {
                const float4* src = reinterpret_cast<const float4*>(background) + bg00;
                float4* dst = reinterpret_cast<float4*>(pixels);
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = __ldg(src + (size_t)((i >> 1) & 1) * d.W + (i & 1) + (i >> 2) * TILE_W);
#pragma unroll
                for (int i = 0; i < 8; ++i) dst[p00 + (size_t)((i >> 1) & 1) * d.W + (i & 1) + (i >> 2) * TILE_W] = v[i];
            } else {
                // CT == 3: the two pixels of a quad row are 24 contiguous, 8-byte aligned bytes (checked at launch)
                const float2* src = reinterpret_cast<const float2*>(background + bg00 * 3);
                float2* dst = reinterpret_cast<float2*>(pixels);
                float2 v[12];
#pragma unroll
                for (int i = 0; i < 4; ++i) {   // i: bit 0 = row of the quad, bit 1 = tile of the pair
                    const size_t q = ((size_t)(i & 1) * d.W + (i >> 1) * TILE_W) * 3 / 2;
                    v[3 * i] = __ldg(src + q); v[3 * i + 1] = __ldg(src + q + 1); v[3 * i + 2] = __ldg(src + q + 2);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const size_t q = (p00 + (size_t)(i & 1) * d.W + (i >> 1) * TILE_W) * 3 / 2;
                    dst[q] = v[3 * i]; dst[q + 1] = v[3 * i + 1]; dst[q + 2] = v[3 * i + 2];
                }
            }
            if (face_ids_out) {
#pragma unroll
                for (int i = 0; i < 8; ++i) face_ids_out[p00 + (size_t)((i >> 1) & 1) * d.W + (i & 1) + (i >> 2) * TILE_W] = -1;
            }
            continue;
        }
    }
#endif
    for (int sub = 0; sub < TILES_PER_WARP; ++sub) {
    const int tx = txb + sub;
    if (tx >= d.tiles_x) break;
    const int t = ty * d.tiles_x + tx;
    const int tcol0 = tx * TILE_W;

#if DIRT_RASTER_PREFETCH_BG
    // Pull this tile's background lines towards L2 while the tile's list range is still on its way: tiles that show
    // no face (most of a frame) otherwise wait for the range and only then start the DRAM read of the background.
    if (MODE == 0 && CT == 4 && lane < 16) {
        const int r = trow0 + (lane >> 1), c = tcol0 + (lane & 1) * 8;
        if (r < d.H && c < d.W)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(background + ((size_t)b * d.bg_stride + (size_t)r * d.W + c) * 4));
    }
#endif
    const int nbin = ws.tile_count[(size_t)b * d.tiles + t];
    const int nlarge = ws.large_count[b];
    const int col0 = tcol0 + (lane & 7) * 2, row0 = trow0 + (lane >> 3) * 2;
    const size_t p00 = ((size_t)b * d.H + row0) * d.W + col0;   // pixel (row0, col0); the quad is p00 + {0, 1, W, W+1}
    const bool whole = tcol0 + TILE_W <= d.W && trow0 + TILE_H <= d.H;   // warp-uniform: no per-pixel bounds checks
    const int C = (CT > 0) ? CT : d.C;

    // ---- nothing binned to this tile: the background passes through ----------------------------------------
    if (nbin == 0 && nlarge == 0) {
        // pixel (row0, col0) of the background: p00 less the images a shared background does not have (a 32 x 32 -> 64-bit
        // product: this form keeps the kernel's register allocation as it was without shared backgrounds)
        const size_t l00 = p00 - (size_t)(unsigned)b * (unsigned)(d.H * d.W - d.bg_stride);
        if (MODE == 0 && CT == 3 && whole) {
            const float2* src = reinterpret_cast<const float2*>(background + l00 * 3);
            float2* dst = reinterpret_cast<float2*>(pixels);
            float2 v[6];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const size_t q = (size_t)i * d.W * 3 / 2;   // W is even
                v[3 * i] = __ldg(src + q); v[3 * i + 1] = __ldg(src + q + 1); v[3 * i + 2] = __ldg(src + q + 2);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const size_t q = (p00 + (size_t)i * d.W) * 3 / 2;
                dst[q] = v[3 * i]; dst[q + 1] = v[3 * i + 1]; dst[q + 2] = v[3 * i + 2];
                if (face_ids_out) { face_ids_out[p00 + (size_t)i * d.W] = -1; face_ids_out[p00 + (size_t)i * d.W + 1] = -1; }
            }
            continue;
        }
#pragma unroll
        for (int pix = 0; pix < 4; ++pix) {
            if (!whole && (row0 + (pix >> 1) >= d.H || col0 + (pix & 1) >= d.W)) continue;
            const size_t o = (size_t)(pix >> 1) * d.W + (pix & 1), p = p00 + o;
            if (face_ids_out) face_ids_out[p] = -1;
            if (MODE == 1) {
                if (gbuffer_out) reinterpret_cast<float4*>(gbuffer_out)[p] = make_float4(-1.f, -1.f, -1.f, __int_as_float(0x7f800000));
            } else if (CT == 4) {
                reinterpret_cast<float4*>(pixels)[p] = __ldg(reinterpret_cast<const float4*>(background) + l00 + o);
            } else {
                for (int ch = 0; ch < C; ++ch) pixels[p * C + ch] = __ldg(&background[(l00 + o) * C + ch]);
            }
        }
        continue;
    }

    Quad quad;
#pragma unroll
    for (int i = 0; i < 4; ++i) quad.best[i] = pack(KEY_EMPTY, 0);
    uint32_t tile_max = KEY_EMPTY;
    if (nbin > 0)
        consume_list<true, false>(ws.bins + ((size_t)b * d.tiles + t) * BIN_CAP, min(nbin, BIN_CAP), 0, cov_b, itp_b, verts,
                                  slots_all[warp], lane, tcol0, trow0, d.H, d.W, quad, tile_max);
    if (nbin > BIN_CAP) {   // the bin was full: this tile's share of its row's overflow list
        const size_t orow = (size_t)b * d.tiles_y + ty;
        consume_list<true, true>(reinterpret_cast<const int*>(ws.ovf + orow * OVF_ROW_CAP), min(ws.ovf_count[orow], OVF_ROW_CAP), t,
                                 cov_b, itp_b, verts, slots_all[warp], lane, tcol0, trow0, d.H, d.W, quad, tile_max);
    }
    if (nlarge > 0)
        consume_list<false, false>(ws.large_list + (size_t)b * d.F, nlarge, 0, cov_b, itp_b, verts, slots_all[warp], lane, tcol0,
                                   trow0, d.H, d.W, quad, tile_max);

    // tile coverage flags for the backward pass: a tile that shows any face marks itself and its 8 neighbours
    // (the backward pass reaches one pixel beyond its own tile)
    {
        const bool any_cov = __any_sync(0xffffffffu, ((uint32_t)(quad.best[0] >> 32) < KEY_EMPTY) | ((uint32_t)(quad.best[1] >> 32) < KEY_EMPTY) |
                                                     ((uint32_t)(quad.best[2] >> 32) < KEY_EMPTY) | ((uint32_t)(quad.best[3] >> 32) < KEY_EMPTY));
        if (any_cov && lane < 9) {
            const int nx = tx + (lane % 3) - 1, ny = ty + (lane / 3) - 1;
            if (nx >= 0 && nx < d.tiles_x && ny >= 0 && ny < d.tiles_y) ws.tile_flags[(size_t)b * d.tiles + ny * d.tiles_x + nx] = 1;
        }
    }

    const float* cols = vertex_colors + (size_t)b * d.col_stride * C;
    int prev_face = -1;
    TriInterp ti;
#pragma unroll
    for (int pix = 0; pix < 4; ++pix) {
        const int row = row0 + (pix >> 1), col = col0 + (pix & 1);
        if (!whole && (row >= d.H || col >= d.W)) continue;
        const bool covered = (uint32_t)(quad.best[pix] >> 32) < KEY_EMPTY;
        const int face = covered ? (int)(uint32_t)quad.best[pix] : -1;
        const size_t p = p00 + (size_t)(pix >> 1) * d.W + (pix & 1);
        if (face_ids_out) face_ids_out[p] = face;
        if (MODE == 1) {
            if (gbuffer_out) {
                float4 g = make_float4(-1.f, -1.f, -1.f, __int_as_float(0x7f800000));
                if (face >= 0) g = exact::gbuffer_at(load_interp(itp_b + face), col, row);
                reinterpret_cast<float4*>(gbuffer_out)[p] = g;
            }
        } else if (face < 0) {
            const float* bg = background + (p - (size_t)b * (d.H * d.W - d.bg_stride)) * C;   // as l00 above
            if (CT == 4) {
                reinterpret_cast<float4*>(pixels)[p] = __ldg(reinterpret_cast<const float4*>(bg));
            } else {
                for (int ch = 0; ch < C; ++ch) pixels[p * C + ch] = __ldg(&bg[ch]);
            }
        } else if (REC) {
            shade_pixel_record<CT>(ws.shade + (size_t)b * d.F + face, col, row, pixels + p * C, C);
        } else {
            if (face != prev_face) { ti = load_interp(itp_b + face); prev_face = face; }
            shade_pixel<CT>(ti, col, row, cols, pixels + p * C, C);
        }
    }
    }   // sub
    }   // b
}

cudaError_t launch_raster_forward(const float* vertices, const float* background, const float* vertex_colors, float* pixels,
                                  int32_t* face_ids_out, const Workspace& ws, const Dims& d, cudaStream_t stream,
                                  int* launches)
{
    if ((long long)d.B * d.tiles == 0) return cudaSuccess;
    const dim3 grid((unsigned)((d.tiles_x + WARPS_PER_BLOCK * TILES_PER_WARP - 1) / (WARPS_PER_BLOCK * TILES_PER_WARP)), (unsigned)d.tiles_y, (unsigned)min(d.B, 65535));
    ScopedKernelTimer timer(1, stream);
    const bool vec4 = d.C == 4 && ((uintptr_t)background % 16 == 0) && ((uintptr_t)pixels % 16 == 0) &&
                      ((uintptr_t)vertex_colors % 16 == 0);
    // C == 3 with an even width: every quad row (two pixels) is 24 contiguous, 8-byte aligned bytes
    const bool vec3 = d.C == 3 && d.W % 2 == 0 && ((uintptr_t)background % 8 == 0) && ((uintptr_t)pixels % 8 == 0);
    const bool rec = shade_records_ok(d);   // the setup pass of this call wrote the shading records (C <= 4)
    if (vec4 && rec)
        raster_kernel<0, 4, true><<<grid, WARPS_PER_BLOCK * 32, 0, stream>>>(vertices, background, vertex_colors, pixels,
                                                                             face_ids_out, nullptr, ws, d);
    else if (vec3 && rec)
        raster_kernel<0, 3, true><<<grid, WARPS_PER_BLOCK * 32, 0, stream>>>(vertices, background, vertex_colors, pixels,
                                                                             face_ids_out, nullptr, ws, d);
    else if (rec)
        raster_kernel<0, 0, true><<<grid, WARPS_PER_BLOCK * 32, 0, stream>>>(vertices, background, vertex_colors, pixels,
                                                                             face_ids_out, nullptr, ws, d);
    else   // more than four channels (or a frame beyond the records' 16-bit reference pixel): barycentrics + colour gathers
        raster_kernel<0, 0, false><<<grid, WARPS_PER_BLOCK * 32, 0, stream>>>(vertices, background, vertex_colors, pixels,
                                                                              face_ids_out, nullptr, ws, d);
    ++*launches;
    return cudaGetLastError();
}

cudaError_t launch_raster_visibility(const float* vertices, int32_t* face_ids, float* gbuffer, const Workspace& ws, const Dims& d,
                                     cudaStream_t stream, int* launches)
{
    if ((long long)d.B * d.tiles == 0) return cudaSuccess;
    const dim3 grid((unsigned)((d.tiles_x + WARPS_PER_BLOCK * TILES_PER_WARP - 1) / (WARPS_PER_BLOCK * TILES_PER_WARP)), (unsigned)d.tiles_y, (unsigned)min(d.B, 65535));
    raster_kernel<1, 0, false><<<grid, WARPS_PER_BLOCK * 32, 0, stream>>>(vertices, nullptr, nullptr, nullptr, face_ids, gbuffer, ws, d);
    ++*launches;
    return cudaGetLastError();
}

}  // namespace dirt
