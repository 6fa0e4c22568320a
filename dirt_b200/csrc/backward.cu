// backward.cu -- the RasteriseGrad pass: restates assemble_grads (csrc/rasterise_grad_egl.cu:93-236) on top of the
// face-id visibility buffer.
//
// Per pixel: Scharr filter of `pixels` per channel group (frame-edge clamp), colour-gradient splat with the undilated
// barycentrics, background gradient, occluder-edge dilation from the +-1 neighbour along the dominant-gradient axis
// (dithered by (x+y)%2), position-gradient splat.  Decision quantities (Scharr sums, their L1 norms, clip_w) follow the
// fixed fp32 operation order of DESIGN.md so that every discrete choice matches the oracle and the reference's own
// compiled kernel (oracle/_ref); accumulated values are ordinary fp32.
//
// One launch handles one channel group of width 3 or 1 on its slice [c0, c0+C) of the cs channels, or -- C = 4 -- the
// fused pair {3,1} of a 4-channel tensor.  Any channel count / grouping is a sequence of such launches (what the reference
// does at the Python level, dirt/rasterise_ops.py:86-108, without slicing or copying).
//
// Shape: one warp per 8x8 tile, two vertically adjacent pixels per lane, everything the tile needs staged in the warp's
// own slice of shared memory so that no phase waits on a chain of dependent global loads:
//  (0) 16x8 coverage flags written by the forward pass short-cut tiles that no face can reach (grad_background =
//      grad_pixels, nothing else).
//  (1) The tile's 10x12 halo of `face_ids` and of `pixels` arrive by TMA (cp.async.bulk.tensor, one elected lane, one
//      mbarrier each) -- or, for tiles touching the frame border and for tensors TMA cannot describe, by per-lane
//      cp.async with at()'s clamping.
//  (2) FACE TABLE: the distinct faces among the tile's 64 pixels and its 32-pixel ring get a slot each (warp match +
//      a small open-addressing hash in shared memory); their interpolation planes and vertex positions (TriInterp +
//      TriXY, 96 B) are copied into the table with cp.async while the Scharr sums are computed.
//  (3) G-BUFFER TILE: every lane evaluates (barycentrics, clip_w) of its two pixels and of one ring pixel from the table
//      and parks them in shared memory; the dilation of assemble_grads (:155-194) then only reads neighbouring entries.
//  (4) Every per-pixel term of assemble_grads is a product  scalar * barycentric  destined for vertex k of one face:
//      C colour scalars (grad_pixels) keyed by the pixel's own face, three position scalars (a, b, c = dL/d clip x, y, w
//      of the fragment) keyed by the possibly dilated face.  The warp loops over the occupied slots and reduces the
//      3*(C+3) sums of each face over its 32 lanes with a transposed butterfly (every lane ends up owning one finished
//      sum): ONE warp-wide RED per (face, tile) instead of the reference's atomicAdd per pixel per term
//      (csrc/rasterise_grad_egl.cu:139,227-229).  Faces with only a few records in the tile skip the butterfly
//      (vector REDs).
//  A tile with more distinct faces than the table holds takes the reference-shaped path (one atomic per term).
#include "common.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>
#include <type_traits>

namespace dirt {

#ifndef DIRT_BWD_WARPS
#define DIRT_BWD_WARPS 4
#endif
#ifndef DIRT_ABLATE
#define DIRT_ABLATE 0   // timing experiments only: 1 = no per-face reduction, 2 = no Scharr/dilation, 3 = both
#endif
#ifndef DIRT_BWD_SMALL_FACE
#define DIRT_BWD_SMALL_FACE 20  // faces owning at most this many records in a tile are added directly (0: always reduce);
                                // 12 / 20 / 32: 389.5 / 385.5 / 429 us at cfg3 (profiles/r02_kbench_tma_variants.txt, _ablation_notma.txt)
#endif
#ifndef DIRT_BWD_MIN_BLOCKS
#define DIRT_BWD_MIN_BLOCKS 8   // x 4 warps: <= 64 registers
#endif
#ifndef DIRT_BWD_SLOTS_C4
#define DIRT_BWD_SLOTS_C4 24    // face-table slots per tile (shared memory per warp: see BwdSmem)
#endif
#ifndef DIRT_BWD_SLOTS_C3
#define DIRT_BWD_SLOTS_C3 32
#endif
#ifndef DIRT_BWD_TMA
#define DIRT_BWD_TMA 1
#endif
// One image per warp.  A warp walking 2 / 4 / 8 consecutive images at its tile position with the next image's halos requested
// (TMA) under the current one measured 410 / 408 / 415 us against 363 us at cfg3 (profiles/r02_kbench_pipeline.txt): fewer,
// longer CTAs lose more than the prefetch wins.
constexpr int TILE = 8;               // backward tile edge: one warp per 8x8 tile, two pixels per lane
constexpr int HALO_ROWS = TILE + 2;   // 10
constexpr int HALO_COLS = TILE + 4;   // 12: col-1 .. col+10 (one pixel around for the Scharr taps, two more to the right
                                      // for the flat-order reads of 1-wide groups; also makes every TMA box row a multiple of 16 B)
constexpr int GB_COLS = TILE + 2;     // 10: the G-buffer tile has no use for the two extra columns
// A TMA box must start on a 16-byte boundary of the innermost dimension (measured: anything else is an illegal-instruction
// fault, profiles/r02_tma_probe2.txt).  The halo starts one pixel left of a tile whose first column is a multiple of 8, so
// the staged tiles of 4-byte pixels (face ids, 1- and 3-channel groups) are 16 pixels wide, starting FOUR pixels left of
// the tile (halo column hc sits at tile column hc + 3); 16-byte pixels (C = 4) keep the 12-pixel row starting at the halo.
constexpr int IDS_COLS = 16, IDS_COL0 = 3;
template <int C> struct PxTile {
    static constexpr int COLS = (C == 4) ? HALO_COLS : 16;   // pixels per staged row
    static constexpr int COL0 = (C == 4) ? 0 : 3;            // tile column of halo column 0
};

struct V3 { float x, y, z; };

// at(): nearest frame pixel for out-of-range taps; three components of the channel group starting at
// c0 (width n).  For n == 1 the reference reads "channels" 1 and 2 of a contiguous [B,H,W,1] tensor,
// i.e. the next two pixels in flat order (0 past the end of the tensor).
struct Frame { int B, H, W; };
__device__ __forceinline__ V3 group_at(const float* __restrict__ pixels, int b, int r, int c, const Frame d, int cs, int c0, int n)
{
    r = max(0, min(d.H - 1, r));
    c = max(0, min(d.W - 1, c));
    const size_t lin = ((size_t)b * d.H + r) * d.W + c;
    V3 v;
    if (n == 3) {
        const float* p = pixels + lin * cs + c0;
        v.x = __ldg(p); v.y = __ldg(p + 1); v.z = __ldg(p + 2);
    } else {
        const size_t total = (size_t)d.B * d.H * d.W;
        v.x = __ldg(pixels + lin * cs + c0);
        v.y = (lin + 1 < total) ? __ldg(pixels + (lin + 1) * cs + c0) : 0.f;
        v.z = (lin + 2 < total) ? __ldg(pixels + (lin + 2) * cs + c0) : 0.f;
    }
    return v;
}

// (a + b - c - d) * 3/32 + (e - f) * 10/32 in the order of operations of the reference's compiled kernel
// (csrc/rasterise_grad_egl.cu:126-127 as nvcc contracts it: FMUL (e-f)*10/32, then FFMA (a+b-c-d)*3/32 + that;
// profiles/r02_ref_assemble_grads_scharr_sass.txt)
__device__ __forceinline__ float scharr_comp(float a, float b, float c, float dd, float e, float f)
{
    const float X = __fsub_rn(__fsub_rn(__fadd_rn(a, b), c), dd);
    const float Y = __fsub_rn(e, f);
    return __fmaf_rn(X, 0.09375f, __fmul_rn(Y, 0.3125f));
}

__device__ __forceinline__ float l1(const float s[3])
{
    return __fadd_rn(__fadd_rn(fabsf(s[0]), fabsf(s[1])), fabsf(s[2]));
}

// ---- asynchronous copies ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_4(void* smem, const void* gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// generic-proxy accesses to shared memory (ours) before async-proxy ones (the next TMA write into the same buffer)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// TMA: one 3-D box [1][HALO_ROWS][box] of a [B][H][W * elems] tensor into shared memory; x (in elements) must be a multiple of 4
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}

// 16-byte vector reduction to global memory (sm_90+): four fp32 adds in one RED
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---- the warp's slice of shared memory ----------------------------------------------------------------------------
struct __align__(16) SlotRec {   // one face of the tile: interpolation planes + vertex ids + vertex positions
    TriInterp itp;               // 64 B
    TriXY xy;                    // 32 B
};
static_assert(sizeof(SlotRec) == 96, "SlotRec must be 96 bytes");

template <int C, int NSLOT>
struct BwdSmem {
    static constexpr int PX_BYTES = HALO_ROWS * PxTile<C>::COLS * C * 4;
    static constexpr int IDS_BYTES = HALO_ROWS * IDS_COLS * 4;
    static constexpr int GBUF_BYTES = HALO_ROWS * GB_COLS * 16;
    static constexpr int PX_OFF = 0;
    static constexpr int IDS_OFF = (PX_BYTES + 127) / 128 * 128;
    static constexpr int GBUF_OFF = IDS_OFF + (IDS_BYTES + 127) / 128 * 128;
    static constexpr int TABLE_OFF = GBUF_OFF + GBUF_BYTES;
    static constexpr int KEYS_OFF = TABLE_OFF + NSLOT * (int)sizeof(SlotRec);
    static constexpr int BAR_OFF = (KEYS_OFF + NSLOT * 4 + 7) / 8 * 8;
    static constexpr int BYTES = (BAR_OFF + 16 + 127) / 128 * 128;
};

// ---- Scharr sums from the staged tile -------------------------------------------------------------------------------
// Scharr sums of a single group (width N0) from the staged tile.  lr/lc: row / column of the pixel inside the staged tile.
template <int C, int N0>
__device__ __forceinline__ void scharr_smem(const float* __restrict__ tile, int lr, int lc, float (&sx)[3], float (&sy)[3])
{
    // comp k of the tap at (lr+dr, lc+dc): channel k (N0 == 3) or channel 0 of the pixel k places to the right (N0 == 1)
    constexpr int PITCH = PxTile<C>::COLS;
    auto T = [&](int dr, int dc, int k) -> float {
        return (N0 == 3) ? tile[((lr + dr) * PITCH + lc + dc) * C + k] : tile[((lr + dr) * PITCH + lc + dc + k) * C];
    };
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        // at(ox,oy) is image (row - oy, col + ox)
        const float a_mm = T(+1, -1, k), a_mp = T(-1, -1, k), a_pm = T(+1, +1, k), a_pp = T(-1, +1, k);
        const float a_m0 = T(0, -1, k), a_p0 = T(0, +1, k), a_0m = T(+1, 0, k), a_0p = T(-1, 0, k);
        sx[k] = scharr_comp(a_mm, a_mp, a_pm, a_pp, a_m0, a_p0);
        sy[k] = scharr_comp(a_mm, a_pm, a_mp, a_pp, a_0m, a_0p);
    }
}

// C == 4, groups {3,1}: both groups from 15 vector taps (rows lr-1..lr+1, columns lc-1..lc+3).
// Group {0,1,2} uses .xyz of columns lc-1..lc+1; group {3} uses .w, comp k being the pixel k places to the right.
__device__ __forceinline__ void scharr_smem_c4(const float* __restrict__ tile, int lr, int lc, float (&sx)[3], float (&sy)[3],
                                               float (&sx1)[3], float (&sy1)[3])
{
    const float4* t4 = reinterpret_cast<const float4*>(tile) + (lr * HALO_COLS + lc);
    float4 up[5], mid[5], dn[5];   // image rows lr-1 (at oy=+1), lr, lr+1 (at oy=-1); columns lc-1 .. lc+3
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        up[j] = t4[-HALO_COLS + j - 1];
        mid[j] = t4[j - 1];
        dn[j] = t4[HALO_COLS + j - 1];
    }
    // at(ox,oy) is image (row - oy, col + ox):  a_mm = dn[0], a_mp = up[0], a_pm = dn[2], a_pp = up[2], a_m0 = mid[0],
    // a_p0 = mid[2], a_0m = dn[1], a_0p = up[1]
    sx[0] = scharr_comp(dn[0].x, up[0].x, dn[2].x, up[2].x, mid[0].x, mid[2].x);
    sx[1] = scharr_comp(dn[0].y, up[0].y, dn[2].y, up[2].y, mid[0].y, mid[2].y);
    sx[2] = scharr_comp(dn[0].z, up[0].z, dn[2].z, up[2].z, mid[0].z, mid[2].z);
    sy[0] = scharr_comp(dn[0].x, dn[2].x, up[0].x, up[2].x, dn[1].x, up[1].x);
    sy[1] = scharr_comp(dn[0].y, dn[2].y, up[0].y, up[2].y, dn[1].y, up[1].y);
    sy[2] = scharr_comp(dn[0].z, dn[2].z, up[0].z, up[2].z, dn[1].z, up[1].z);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        sx1[k] = scharr_comp(dn[k].w, up[k].w, dn[k + 2].w, up[k + 2].w, mid[k].w, mid[k + 2].w);
        sy1[k] = scharr_comp(dn[k].w, dn[k + 2].w, up[k].w, up[k + 2].w, dn[k + 1].w, up[k + 1].w);
    }
}

// global-memory taps (tiles at the right frame edge, where the flat-order reads of a 1-wide group wrap into the next
// row): three components of group [c0, c0+N0) at the clamped pixel
template <int N0>
__device__ __forceinline__ void scharr_global(const float* __restrict__ pixels, int b, int row, int col, const Frame d, int cs,
                                              int c0, float (&sx)[3], float (&sy)[3])
{
    const V3 a_mm = group_at(pixels, b, row + 1, col - 1, d, cs, c0, N0), a_mp = group_at(pixels, b, row - 1, col - 1, d, cs, c0, N0);
    const V3 a_pm = group_at(pixels, b, row + 1, col + 1, d, cs, c0, N0), a_pp = group_at(pixels, b, row - 1, col + 1, d, cs, c0, N0);
    const V3 a_m0 = group_at(pixels, b, row, col - 1, d, cs, c0, N0), a_p0 = group_at(pixels, b, row, col + 1, d, cs, c0, N0);
    const V3 a_0m = group_at(pixels, b, row + 1, col, d, cs, c0, N0), a_0p = group_at(pixels, b, row - 1, col, d, cs, c0, N0);
    sx[0] = scharr_comp(a_mm.x, a_mp.x, a_pm.x, a_pp.x, a_m0.x, a_p0.x);
    sx[1] = scharr_comp(a_mm.y, a_mp.y, a_pm.y, a_pp.y, a_m0.y, a_p0.y);
    sx[2] = scharr_comp(a_mm.z, a_mp.z, a_pm.z, a_pp.z, a_m0.z, a_p0.z);
    sy[0] = scharr_comp(a_mm.x, a_pm.x, a_mp.x, a_pp.x, a_0m.x, a_0p.x);
    sy[1] = scharr_comp(a_mm.y, a_pm.y, a_mp.y, a_pp.y, a_0m.y, a_0p.y);
    sy[2] = scharr_comp(a_mm.z, a_pm.z, a_mp.z, a_pp.z, a_0m.z, a_0p.z);
}

// the rare tiles that need it (right frame edge) call it out of line: it is ~1000 instructions when inlined four times
template <int N0>
__device__ __noinline__ void scharr_global_call(const float* __restrict__ pixels, int b, int row, int col, int B, int H, int W, int cs,
                                                int c0, float* sxy)
{
    float sx[3], sy[3];
    scharr_global<N0>(pixels, b, row, col, Frame{B, H, W}, cs, c0, sx, sy);
#pragma unroll
    for (int k = 0; k < 3; ++k) { sxy[k] = sx[k]; sxy[3 + k] = sy[k]; }
}

// preferred neighbour offset of the dilation (csrc/rasterise_grad_egl.cu:185-190), as a step in the G-buffer tile:
// buffer offset (dx,dy) is image (col + dx, row - dy), i.e. +1 / -1 along a row, -GB_COLS / +GB_COLS across rows
__device__ __forceinline__ int dilation_step(const float (&sx)[3], const float (&sy)[3], int col, int row)
{
    int step = (l1(sx) > l1(sy)) ? 1 : -GB_COLS;
    if ((col + row) & 1) step = -step;
    return step;
}

// ---- per-face reduction -------------------------------------------------------------------------------------------
// Transposed butterfly over the lanes that differ in bits `bit`, bit/2, ..., 1: at every step a lane keeps half of its
// sums and hands the other half to its partner.  After STEPS steps each lane is left with OUT = ceil(N / 2^STEPS) sums.
template <int N, int STEPS>
struct TransposedReduce {
    static constexpr int H = (N + 1) / 2;
    static constexpr int OUT = TransposedReduce<H, STEPS - 1>::OUT;
    static __device__ __forceinline__ void run(float (&v)[N], int lane, int bit, float (&out)[OUT])
    {
        float w[H];
        const bool up = (lane & bit) != 0;
#pragma unroll
        for (int i = 0; i < H; ++i) {
            const float hi = (H + i < N) ? v[H + i] : 0.f;
            const float send = up ? v[i] : hi;
            const float keep = up ? hi : v[i];
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
        }
        TransposedReduce<H, STEPS - 1>::run(w, lane, bit >> 1, out);
    }
    // global index of out[0] on this lane: out[i] is sum base+i (entries beyond the valid range are padding)
    static __host__ __device__ constexpr int base(int lane, int bit)
    {
        return ((lane & bit) ? H : 0) + TransposedReduce<H, STEPS - 1>::base(lane, bit >> 1);
    }
    // is out[i] a real sum?  (checks the padding introduced at every level)
    static __host__ __device__ constexpr bool valid(int lane, int bit, int i)
    {
        return TransposedReduce<H, STEPS - 1>::valid(lane, bit >> 1, i) &&
               (((lane & bit) ? H : 0) + TransposedReduce<H, STEPS - 1>::base(lane, bit >> 1) + i < N);
    }
};
template <int N>
struct TransposedReduce<N, 0> {
    static constexpr int OUT = N;
    static __device__ __forceinline__ void run(float (&v)[N], int, int, float (&out)[N])
    {
#pragma unroll
        for (int i = 0; i < N; ++i) out[i] = v[i];
    }
    static __host__ __device__ constexpr int base(int, int) { return 0; }
    static __host__ __device__ constexpr bool valid(int, int, int i) { return i < N; }
};

// Which finished sum a lane owns after the butterfly, as a destination: bits 0-1 = vertex k of the face, bits 2-3 =
// component inside the vertex's row, bit 4 = row of grad_vertices (else grad_vertex_colors); -1 = none.  A table
// because the compiler, short of registers, otherwise recomputes the index arithmetic (~40 instructions)
// for every face of every tile.
template <int C>
struct OwnerTable {
    int meta[32];
};
template <int C>
constexpr OwnerTable<C> make_owner_table()
{
    // layout after the first (operand-level) butterfly step, see the per-face reduction: NS sums of vertex 0 (lanes
    // 0-15) or vertex 1 (lanes 16-31), then the lower / upper half of the NS sums of vertex 2
    constexpr int NS = C + 3, H2 = (NS + 1) / 2;
    using Red = TransposedReduce<NS + H2, 4>;
    OwnerTable<C> t{};
    for (int lane = 0; lane < 32; ++lane) {
        int m = -1;
        if (Red::valid(lane, 8, 0)) {
            const int q = Red::base(lane, 8);
            const bool up = (lane & 16) != 0;
            const int k = q < NS ? (up ? 1 : 0) : 2;
            const int j = q < NS ? q : (q - NS) + (up ? H2 : 0);
            if (j < NS) {
                const bool pos = j >= C;
                const int comp = pos ? (j - C == 2 ? 3 : j - C) : j;   // a, b, c go to x, y, w of the vertex row
                m = k | (comp << 2) | (pos ? 16 : 0);
            }
        }
        t.meta[lane] = m;
    }
    return t;
}
// global (not __constant__) memory: every lane reads its own entry, which the constant cache would serialise 32-fold
__device__ const OwnerTable<1> g_owner1 = make_owner_table<1>();
__device__ const OwnerTable<3> g_owner3 = make_owner_table<3>();
__device__ const OwnerTable<4> g_owner4 = make_owner_table<4>();
template <int C>
__device__ __forceinline__ int owner_meta(int lane)
{
    return __ldg(C == 1 ? &g_owner1.meta[lane] : C == 3 ? &g_owner3.meta[lane] : &g_owner4.meta[lane]);
}

// ---- reference-shaped path for one tile (face table overflow): one atomic per term ---------------------------------
template <int C>
__device__ __noinline__ void tile_generic(const float* __restrict__ vertices, const float* __restrict__ pixels,
                                          const float* __restrict__ grad_pixels, const int32_t* __restrict__ face_ids,
                                          float* __restrict__ gverts, float* __restrict__ gcols,   // rows of this image (or the shared rows); gcols at the group's first channel
                                          const TriInterp* __restrict__ itp_b, const Frame d, int V, int b, int col, int row0, int cs, int c0,
                                          int gstride, bool want_pos, bool want_col)
{
    constexpr int N0 = (C == 1) ? 1 : 3;
    constexpr int NG = (C == 4) ? 2 : 1;
    if (col >= d.W) return;
    const float* verts = vertices + (size_t)b * V * 4;
    const int32_t* ids = face_ids + (size_t)b * d.H * d.W;
    const float inf = __int_as_float(0x7f800000);
    for (int pix = 0; pix < 2; ++pix) {
        const int row = row0 + pix;
        if (row >= d.H) break;
        const size_t p = ((size_t)b * d.H + row) * d.W + col;
        const int f_own = ids[row * d.W + col];
        TriInterp t_own;
        float4 g_own = make_float4(-1.f, -1.f, -1.f, inf);
        if (f_own >= 0) {
            t_own = load_interp(itp_b + f_own);
            g_own = exact::gbuffer_at(t_own, col, row);
            const int vid[3] = {t_own.v0, t_own.v1, t_own.v2};
            const float bary[3] = {g_own.x, g_own.y, g_own.z};
            for (int ch = 0; want_col && ch < C; ++ch) {
                const float gp = __ldg(&grad_pixels[p * cs + c0 + ch]);
#pragma unroll
                for (int k = 0; k < 3; ++k) atomicAdd(&gcols[(size_t)vid[k] * gstride + ch], gp * bary[k]);
            }
        }
        const bool interior = col > 0 && row > 0 && col < d.W - 1 && row < d.H - 1;
        for (int gi = 0; want_pos && gi < NG; ++gi) {
            const int g0 = c0 + (gi ? 3 : 0), n = gi ? 1 : N0;
            float sx[3], sy[3];
            if (n == 3) scharr_global<3>(pixels, b, row, col, d, cs, g0, sx, sy);
            else scharr_global<1>(pixels, b, row, col, d, cs, g0, sx, sy);
            int f = f_own;
            float4 g = g_own;
            TriInterp tf = t_own;
            if (interior) {
                int dx = (l1(sx) > l1(sy)) ? 1 : 0, dy = 1 - dx;  // buffer (y-up) orientation
                if ((col + row) & 1) { dx = -dx; dy = -dy; }
                for (int attempt = 0; attempt < 2; ++attempt) {
                    const int nc = col + dx, nr = row - dy;
                    const int fn = ids[nr * d.W + nc];
                    if (fn >= 0) {
                        const TriInterp tn = load_interp(itp_b + fn);
                        const bool differs = (f_own < 0) || tn.v0 != t_own.v0 || tn.v1 != t_own.v1 || tn.v2 != t_own.v2;
                        const float4 gn = exact::gbuffer_at(tn, nc, nr);
                        if (differs && g_own.w > gn.w) {
                            g = gn; f = fn; tf = tn;
                            break;
                        }
                    }
                    dx = -dx; dy = -dy;
                }
            }
            if (f >= 0) {
                float dLdx = 0.f, dLdy = 0.f;
                for (int ch = 0; ch < n; ++ch) {
                    const float gp = __ldg(&grad_pixels[p * cs + g0 + ch]);
                    dLdx += gp * sx[ch];
                    dLdy += gp * sy[ch];
                }
                const int vid[3] = {tf.v0, tf.v1, tf.v2};
                const float bary[3] = {g.x, g.y, g.z};
                float clip_x = 0.f, clip_y = 0.f;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float2 xy = __ldg(reinterpret_cast<const float2*>(verts + (size_t)vid[k] * 4));
                    clip_x += bary[k] * xy.x;
                    clip_y += bary[k] * xy.y;
                }
                const float inv_w = 1.f / g.w;
                const float dxv_dxc = 0.5f * (float)d.W * inv_w, dyv_dyc = 0.5f * (float)d.H * inv_w;
                const float dxv_dwc = -dxv_dxc * clip_x * inv_w, dyv_dwc = -dyv_dyc * clip_y * inv_w;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float ax = dLdx * bary[k], ay = dLdy * bary[k];
                    atomicAdd(&gverts[(size_t)vid[k] * 4 + 0], ax * dxv_dxc);
                    atomicAdd(&gverts[(size_t)vid[k] * 4 + 1], ay * dyv_dyc);
                    atomicAdd(&gverts[(size_t)vid[k] * 4 + 3], ax * dxv_dwc + ay * dyv_dwc);
                }
            }
        }
    }
}

// G-buffer entry of a face at a pixel, from the tile's face table
__device__ __forceinline__ float4 table_gbuffer(const SlotRec* __restrict__ table, int slot, int col, int row)
{
    const float4* r = reinterpret_cast<const float4*>(table + slot);
    const float4 v0 = r[0], v1 = r[1], v2 = r[2];
    const int4 v3 = reinterpret_cast<const int4*>(r)[3];
    TriInterp t;
    t.q0A = v0.x; t.q0B = v0.y; t.q0C = v0.z; t.q1A = v0.w;
    t.q1B = v1.x; t.q1C = v1.y; t.sA = v1.z; t.sB = v1.w;
    t.sC = v2.x; t.cref = v3.x; t.rref = v3.y;
    return exact::gbuffer_at(t, col, row);
}

struct PixelTerms {      // everything one pixel contributes
    int key_col;         // slot of the own face (-1: uncovered)
    int key_pos;         // slot of the face receiving the position gradient (-1: none)
    // barycentrics (c: undilated, for the colour terms; p: of the fragment receiving the position gradient), arranged for
    // the first butterfly step: A = the vertex whose sums this lane keeps (vertex 0 on lanes 0-15, vertex 1 on lanes
    // 16-31), B = the one it hands to its partner, 2 = vertex 2
    float cA, cB, c2;
    float pA, pB, p2;
};

template <int C, int NSLOT, int NW, bool USE_TMA>
__global__ void __launch_bounds__(NW * 32, DIRT_BWD_MIN_BLOCKS * DIRT_BWD_WARPS / NW) backward_tile_kernel(
    const __grid_constant__ CUtensorMap px_map, const __grid_constant__ CUtensorMap ids_map,
    const float* __restrict__ vertices, const float* __restrict__ pixels, const float* __restrict__ grad_pixels,
    const int32_t* __restrict__ face_ids, float* __restrict__ grad_background, float* __restrict__ grad_vertices,
    float* __restrict__ grad_vertex_colors, Workspace ws, Dims d, const unsigned char* __restrict__ tile_flags,
    int cs, int c0,   // cs: channels per pixel in the tensors, c0: first channel of the group this launch handles (width C)
    int gstride,      // floats per vertex row of grad_vertex_colors as this launch sees it (cs, or 4 for the padded rows of C = 3)
    int flags,        // BWD_SHARED_GEOMETRY: vertex gradients accumulated over the batch ([V,.]); BWD_SKIP_POSITION / _COLOUR;
                      // SHARED_COLOURS: grad_vertex_colors accumulated over the batch; SHARED_BACKGROUND: no grad_background here
    unsigned long long expect_tag,   // != 0: the caller promised that the workspace holds the setup records with this tag
    int b_base)                      // first image of this launch (the grid's z extent holds at most 65535 images)
{
    using SM = BwdSmem<C, NSLOT>;
    constexpr int NS = C + 3;                  // scalars per pixel: C colour + (a,b,c)
    constexpr int N0 = (C == 1) ? 1 : 3;       // width of the first group
    constexpr bool TWO_GROUPS = (C == 4);      // {3,1}
    constexpr int REACH = (C == 3) ? 1 : 3;    // columns to the right of the pixel that its taps read

    extern __shared__ __align__(128) unsigned char smem_raw[];

    // grid: x = groups of NW tiles along a tile row, y = tile row, z = image
    // The warp index goes through a warp reduction so that the compiler KNOWS it (and the tile coordinates, the TMA /
    // border / right-edge predicates derived from it) to be warp-uniform: branches on them stay convergent and the
    // shuffles of the reduction need no re-convergence barriers.
    const int lane = threadIdx.x & 31;
    const int warp = (int)__reduce_min_sync(0xffffffffu, threadIdx.x >> 5);
    const int tx = blockIdx.x * NW + warp, ty = blockIdx.y, b = b_base + (int)blockIdx.z;
    if (tx >= d.btiles_x) return;
    const int H = d.H, W = d.W;
    const int trow0 = ty * TILE, tcol0 = tx * TILE;
    const int lcol = lane & 7, lrow0 = (lane >> 3) * 2;
    const int row0 = trow0 + lrow0, col = tcol0 + lcol;
    const bool want_pos = !(flags & BWD_SKIP_POSITION), want_col = !(flags & BWD_SKIP_COLOUR);
    const bool write_gb = want_col && !(flags & SHARED_BACKGROUND);   // the per-image grad_background

    if (expect_tag != 0 && (blockIdx.x | blockIdx.y | (unsigned)b | threadIdx.x) == 0 && ws.header->tag != expect_tag) {
        // the workspace was not filled by a forward / visibility call on these (vertices, faces, sizes): flag it
        // (dirt_workspace_status) and poison the result instead of returning plausible numbers
        ws.header->error = 1;
        if (d.V > 0) grad_vertices[0] = __int_as_float(0x7fc00000);
    }

    // ---- what every tile needs: the forward pass's coverage flag of its 16x8 tile and grad_pixels of this lane's pixels.
    // Nearly half of a frame's tiles end right here, so nothing else is set up before the flag is known.
    bool flagged;
    {
        bool f = false;
        if (lane == 0) f = tile_flags == nullptr || tile_flags[(size_t)b * d.tiles + ty * d.tiles_x + (tx >> 1)] != 0;
        flagged = (__ballot_sync(0xffffffffu, f) & 1u) != 0u;   // through a vote: known to be warp-uniform
    }
    if (!flagged && !write_gb) return;   // no face can reach the tile and no grad_background to write: grad_pixels is not read
    const size_t img = (size_t)b * H * W;
    const size_t p0 = img + (size_t)row0 * W + col;   // pixel 0 of this lane (pixel 1: + W)
    const bool in0 = col < W && row0 < H, in1 = col < W && row0 + 1 < H;
    float gp[2][C];
#pragma unroll
    for (int pix = 0; pix < 2; ++pix) {
#pragma unroll
        for (int ch = 0; ch < C; ++ch) gp[pix][ch] = 0.f;
        if (!(pix ? in1 : in0)) continue;
        const size_t p = p0 + (size_t)pix * W;
        if (C == 4) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(grad_pixels) + p);
            gp[pix][0] = v.x; gp[pix][1 % C] = v.y; gp[pix][2 % C] = v.z; gp[pix][3 % C] = v.w;
        } else {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) gp[pix][ch] = __ldg(grad_pixels + p * cs + c0 + ch);
        }
    }
    auto store_gb = [&](int pix, bool uncovered) {
        // grad_background: grad_pixels where uncovered, 0 elsewhere (:143-148, memset :247)
        const size_t p = p0 + (size_t)pix * W;
        if (C == 4) {
            reinterpret_cast<float4*>(grad_background)[p] =
                uncovered ? make_float4(gp[pix][0], gp[pix][1 % C], gp[pix][2 % C], gp[pix][3 % C]) : make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
#pragma unroll
            for (int ch = 0; ch < C; ++ch) grad_background[p * cs + c0 + ch] = uncovered ? gp[pix][ch] : 0.f;
        }
    };
    if (!flagged) {
        // the forward pass flagged every 16x8 tile that shows a face or touches one that does: nothing can reach this one
        if (in0) store_gb(0, true);
        if (in1) store_gb(1, true);
        return;
    }

    // ---- a tile a face may reach: its slice of shared memory, the ring cell of this lane, the staging mode
    unsigned char* const sm = smem_raw + warp * SM::BYTES;
    float* const tile = reinterpret_cast<float*>(sm + SM::PX_OFF);
    int* const ids_tile = reinterpret_cast<int*>(sm + SM::IDS_OFF);
    float4* const gbuf = reinterpret_cast<float4*>(sm + SM::GBUF_OFF);
    SlotRec* const table = reinterpret_cast<SlotRec*>(sm + SM::TABLE_OFF);
    int* const keys = reinterpret_cast<int*>(sm + SM::KEYS_OFF);
    uint64_t* const bars = reinterpret_cast<uint64_t*>(sm + SM::BAR_OFF);   // [0]: face ids, [1]: pixels
    // this lane's cells: its two pixels and one cell of the 32-cell ring around the tile (corners are never read)
    const int g0 = (lrow0 + 1) * GB_COLS + lcol + 1;                  // G-buffer tile index of pixel 0 (pixel 1: + GB_COLS)
    const int ring_r = lane < 8 ? 0 : lane < 16 ? TILE + 1 : lane - (lane < 24 ? 15 : 23);
    const int ring_c = lane < 8 ? lane + 1 : lane < 16 ? lane - 7 : lane < 24 ? 0 : TILE + 1;
    // whole halo (12 columns: the flat-order reads reach two past the 10) inside the frame: no clamping, every pixel is
    // interior.  (What a 16-wide TMA box holds beyond the halo may be out of bounds: zero-filled, never read.)
    const bool inner = tcol0 >= 1 && trow0 >= 1 && tcol0 + HALO_COLS - 2 <= W - 1 && trow0 + TILE <= H - 1;
    const bool use_tma = USE_TMA && inner;   // warp-uniform
    const bool per_item = !(flags & BWD_SHARED_GEOMETRY);
    const TriInterp* itp_b = ws.itp + (size_t)b * d.F;
    const TriXY* xy_b = ws.xy + (size_t)b * d.F;
    float* gverts = grad_vertices + (size_t)(per_item ? b : 0) * d.V * 4;
    float* gcols = grad_vertex_colors + (size_t)(per_item && !(flags & SHARED_COLOURS) ? b : 0) * d.V * gstride + c0;

    // ---- (1) stage the halo of face ids and pixels: TMA (one elected lane, one mbarrier each) or per-lane cp.async
    if (use_tma) {
        if (lane == 0) {
            mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            fence_proxy_async();
            mbar_expect_tx(&bars[0], SM::IDS_BYTES);
            tma_load_3d(ids_tile, &ids_map, tcol0 - 1 - IDS_COL0, trow0 - 1, b, &bars[0]);
            if (want_pos) {
                mbar_expect_tx(&bars[1], SM::PX_BYTES);
                tma_load_3d(tile, &px_map, (tcol0 - 1 - PxTile<C>::COL0) * C, trow0 - 1, b, &bars[1]);
            }
        }
        __syncwarp();   // the barriers exist before any lane waits on them
    } else {
        for (int e = lane; e < HALO_ROWS * HALO_COLS; e += 32) {
            const int hr = e / HALO_COLS, hc = e - hr * HALO_COLS;
            const int r = trow0 - 1 + hr, c = tcol0 - 1 + hc;
            int* const id_dst = ids_tile + hr * IDS_COLS + hc + IDS_COL0;
            if (r >= 0 && r < H && c >= 0 && c < W) cp_async_4(id_dst, face_ids + img + (size_t)r * W + c);
            else *id_dst = -1;
            if (!want_pos) continue;
            const int rc = max(0, min(H - 1, r)), cc = max(0, min(W - 1, c));
            const float* src = pixels + (img + (size_t)rc * W + cc) * cs + c0;
            float* const px_dst = tile + (hr * PxTile<C>::COLS + hc + PxTile<C>::COL0) * C;
            if (C == 4) cp_async_16(px_dst, src);
            else {
#pragma unroll
                for (int ch = 0; ch < C; ++ch) cp_async_4(px_dst + ch, src + ch);
            }
        }
        cp_async_commit();
    }
    if (lane < NSLOT) keys[lane] = -1;

    // ---- (2) face ids -> slots of the tile's face table ---------------------------------------------------------------
    if (use_tma) mbar_wait(&bars[0], 0);
    else cp_async_wait_all();
    __syncwarp();
    const int i0 = (lrow0 + 1) * IDS_COLS + lcol + 1 + IDS_COL0;
    const int id0 = ids_tile[i0], id1 = ids_tile[i0 + IDS_COLS], idr = ids_tile[ring_r * IDS_COLS + ring_c + IDS_COL0];
    if (write_gb && in0) store_gb(0, id0 < 0);
    if (write_gb && in1) store_gb(1, id1 < 0);
    // neighbours in the visibility buffer
    const int up0 = ids_tile[i0 - IDS_COLS], l0 = ids_tile[i0 - 1], r0 = ids_tile[i0 + 1];
    const int l1 = ids_tile[i0 + IDS_COLS - 1], r1 = ids_tile[i0 + IDS_COLS + 1], dn1 = ids_tile[i0 + 2 * IDS_COLS];
    if (!__any_sync(0xffffffffu, (id0 & id1 & idr) >= 0)) {
        // no face in the tile or its ring (the pixel halo must still land before the warp gives up its shared memory)
        if (use_tma && want_pos) mbar_wait(&bars[1], 0);
        return;
    }
    // per pixel: covered, or (interior pixels only) a covered 4-neighbour that could dilate into it
    bool near0, near1, interior0 = true, interior1 = true;
    {
        if (!inner) {
            interior0 = col > 0 && row0 > 0 && col < W - 1 && row0 < H - 1;
            interior1 = col > 0 && row0 + 1 < H - 1 && col < W - 1;
        }
        near0 = id0 >= 0 || (want_pos && interior0 && (up0 & l0 & r0 & id1) >= 0);   // any of the four non-negative
        near1 = id1 >= 0 || (want_pos && interior1 && (id0 & l1 & r1 & dn1) >= 0);
        if (!in0) near0 = false;
        if (!in1) near1 = false;
    }
    // slots: one leader per distinct id (warp match) inserts it into the open-addressing hash `keys`
    bool overflow = false;
    auto slot_of = [&](int id) -> int {
        const unsigned peers = __match_any_sync(0xffffffffu, id);
        const int leader = __ffs(peers) - 1;
        int slot = -1;
        if (id >= 0 && lane == leader) {
            int h = (NSLOT == 32) ? (int)(((unsigned)id * 2654435761u) >> 27) : (int)__umulhi((unsigned)id * 2654435761u, (unsigned)NSLOT);
#pragma unroll 1
            for (int probe = 0; probe < NSLOT; ++probe) {
                const int old = atomicCAS(&keys[h], -1, id);
                if (old == -1 || old == id) { slot = h; break; }
                h = (h + 1 == NSLOT) ? 0 : h + 1;
            }
            if (slot < 0) overflow = true;
        }
        return __shfl_sync(0xffffffffu, slot, leader);
    };
    const int slot0 = slot_of(id0);
    const int s1 = slot_of(id1);
    const int slotr = slot_of(idr);
    __syncwarp();
    if (__any_sync(0xffffffffu, overflow)) {
        // more distinct faces than slots: the reference-shaped path for this tile
        if (use_tma && want_pos) mbar_wait(&bars[1], 0);
        tile_generic<C>(vertices, pixels, grad_pixels, face_ids, gverts, gcols, itp_b, Frame{d.B, H, W}, d.V, b, col, row0, cs, c0, gstride, want_pos, want_col);
        return;
    }
    // fill the table: the lane whose index is an occupied slot copies that face's 96 bytes
    {
        const int k = lane < NSLOT ? keys[lane] : -1;
        if (k >= 0) {
            const uint4* src = reinterpret_cast<const uint4*>(itp_b + k);
            uint4* dst = reinterpret_cast<uint4*>(table + lane);
#pragma unroll
            for (int i = 0; i < 4; ++i) cp_async_16(dst + i, src + i);
            const uint4* srcx = reinterpret_cast<const uint4*>(xy_b + k);
            cp_async_16(dst + 4, srcx);
            cp_async_16(dst + 5, srcx + 1);
        }
        cp_async_commit();
    }

    // ---- (3) G-buffer tile: this lane's two pixels and its ring cell ---------------------------------------------------
    cp_async_wait_all();
    if (use_tma && want_pos) mbar_wait(&bars[1], 0);
    __syncwarp();   // table and pixel halo complete
    const float inf = __int_as_float(0x7f800000);
    float4 own[2];
    own[0] = make_float4(-1.f, -1.f, -1.f, inf);
    own[1] = own[0];
    if (slot0 >= 0) own[0] = table_gbuffer(table, slot0, col, row0);
    if (s1 >= 0) own[1] = table_gbuffer(table, s1, col, row0 + 1);
    gbuf[g0] = make_float4(own[0].x, own[0].y, own[0].w, __int_as_float(slot0));
    gbuf[g0 + GB_COLS] = make_float4(own[1].x, own[1].y, own[1].w, __int_as_float(s1));
    {
        float4 gr = make_float4(-1.f, -1.f, inf, __int_as_float(-1));
        if (want_pos && slotr >= 0) {
            const float4 t = table_gbuffer(table, slotr, tcol0 - 1 + ring_c, trow0 - 1 + ring_r);
            gr = make_float4(t.x, t.y, t.w, __int_as_float(slotr));
        }
        gbuf[ring_r * GB_COLS + ring_c] = gr;
    }
    __syncwarp();

    // ---- dilation and per-pixel terms ---------------------------------------------------------------------------------------
    const float halfW = 0.5f * (float)W, halfH = 0.5f * (float)H;
    const bool staged_taps = (tcol0 + TILE - 1 + REACH) <= W - 1;   // warp-uniform (see scharr_global)
    const bool upper = (lane & 16) != 0;   // which half of the warp: decides the arrangement of the weights in PixelTerms
    PixelTerms term[2];
    float sc[2][NS];    // scalars: [0,C) grad_pixels, C..C+2 = a,b,c
#pragma unroll
    for (int pix = 0; pix < 2; ++pix) {
        PixelTerms& T = term[pix];
        T.key_col = T.key_pos = -1;
        T.cA = T.cB = T.c2 = T.pA = T.pB = T.p2 = 0.f;
#pragma unroll
        for (int i = 0; i < NS; ++i) sc[pix][i] = (i < C) ? gp[pix][i % C] : 0.f;
        if (!(pix ? near1 : near0)) continue;
        const float4 me = own[pix];
        const int my_slot = pix ? s1 : slot0;
        const int g = g0 + pix * GB_COLS;
        const int row = row0 + pix;
        const bool interior = pix ? interior1 : interior0;
        if (want_col && my_slot >= 0) { T.key_col = my_slot; T.cA = upper ? me.y : me.x; T.cB = upper ? me.x : me.y; T.c2 = me.z; }
        if (!want_pos) continue;
#if DIRT_ABLATE >= 2
        T.key_pos = my_slot; T.pA = T.cA; T.pB = T.cB; T.p2 = T.c2;
        sc[pix][C] = gp[pix][0]; sc[pix][C + 1] = gp[pix][0]; sc[pix][C + 2] = gp[pix][0];
        continue;
#endif
        // Scharr sums -> gradient scalars and dilation steps of the group(s)
        float sx[3], sy[3], sx1[3], sy1[3];
        if (staged_taps) {
            if (C == 4) scharr_smem_c4(tile, lrow0 + pix + 1, lcol + 1, sx, sy, sx1, sy1);
            else scharr_smem<C, N0>(tile, lrow0 + pix + 1, lcol + 1 + PxTile<C>::COL0, sx, sy);
        } else {
            float t[6];
            scharr_global_call<N0>(pixels, b, row, col, d.B, H, W, cs, c0, t);
#pragma unroll
            for (int k = 0; k < 3; ++k) { sx[k] = t[k]; sy[k] = t[3 + k]; }
            if (TWO_GROUPS) {
                scharr_global_call<1>(pixels, b, row, col, d.B, H, W, cs, c0 + 3, t);
#pragma unroll
                for (int k = 0; k < 3; ++k) { sx1[k] = t[k]; sy1[k] = t[3 + k]; }
            }
        }
        float dLdx = 0.f, dLdy = 0.f, gx1 = 0.f, gy1 = 0.f;
#pragma unroll
        for (int ch = 0; ch < N0; ++ch) { dLdx += gp[pix][ch] * sx[ch]; dLdy += gp[pix][ch] * sy[ch]; }
        const int step0 = interior ? dilation_step(sx, sy, col, row) : 0;
        int step1 = 0;
        if (TWO_GROUPS) {
            gx1 = gp[pix][3 % C] * sx1[0]; gy1 = gp[pix][3 % C] * sy1[0];
            step1 = interior ? dilation_step(sx1, sy1, col, row) : 0;
        }

        // dilation (:155-194): the neighbour at +step, else the one at -step, replaces this pixel's fragment if it is
        // covered, is a different triangle (vertex triple) and is nearer.  Returns the G-buffer cell the fragment comes from.
        auto dilate = [&](int step) -> int {
            if (step == 0) return g;
#pragma unroll
            for (int attempt = 0; attempt < 2; ++attempt) {
                const int cell = attempt ? g - step : g + step;
                const float4 e = gbuf[cell];
                const int ns = __float_as_int(e.w);
                if (ns >= 0 && ns != my_slot && me.w > e.z) {
                    bool differs = my_slot < 0;
                    if (!differs) {
                        const int4 a = reinterpret_cast<const int4*>(table + ns)[2], bb = reinterpret_cast<const int4*>(table + my_slot)[2];
                        differs = a.y != bb.y || a.z != bb.z || a.w != bb.w;   // {sC, v0, v1, v2}
                    }
                    if (differs) return cell;
                }
            }
            return g;
        };
        auto position_terms = [&](const float4 fr, int slot, float gx, float gy, float& a, float& bb, float& cc) {
            // a = dL/dx_clip, b = dL/dy_clip, c = dL/dw_clip of the fragment (:196-232); fr = (b0, b1, b2, clip_w)
            const float4 q0 = reinterpret_cast<const float4*>(table + slot)[4];   // x0 y0 x1 y1
            const float2 q1 = reinterpret_cast<const float2*>(table + slot)[10];  // x2 y2
            const float clip_x = fr.x * q0.x + fr.y * q0.z + fr.z * q1.x;
            const float clip_y = fr.x * q0.y + fr.y * q0.w + fr.z * q1.y;
            const float inv_w = __fdividef(1.0f, fr.w);
            a = gx * halfW * inv_w;
            bb = gy * halfH * inv_w;
            cc = -(a * clip_x + bb * clip_y) * inv_w;
        };
        auto fragment_of = [&](int cell, int& slot) -> float4 {
            if (cell == g) { slot = my_slot; return me; }
            const float4 e = gbuf[cell];
            slot = __float_as_int(e.w);
            return make_float4(e.x, e.y, __fsub_rn(__fsub_rn(1.0f, e.x), e.y), e.z);
        };

        const int cell0 = dilate(step0);
        float gx = dLdx, gy = dLdy;
        if (TWO_GROUPS) {
            // the second group dilates to the same fragment whenever it prefers the same neighbour (the usual case):
            // the outcome of a dilation depends on the step and on the visibility buffer only
            const int cell1 = (step1 == step0) ? cell0 : dilate(step1);
            if (cell1 == cell0) {
                gx += gx1; gy += gy1;
            } else {
                // the two groups dilated differently (rare): this group's terms go out one by one
                int slot_b;
                const float4 fr = fragment_of(cell1, slot_b);
                if (slot_b >= 0) {
                    float a1, b1, c1;
                    position_terms(fr, slot_b, gx1, gy1, a1, b1, c1);
                    const int4 q = reinterpret_cast<const int4*>(table + slot_b)[2];   // {sC, v0, v1, v2}
                    const int vid[3] = {q.y, q.z, q.w};
                    const float bary[3] = {fr.x, fr.y, fr.z};
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        atomicAdd(&gverts[(size_t)vid[k] * 4 + 0], a1 * bary[k]);
                        atomicAdd(&gverts[(size_t)vid[k] * 4 + 1], b1 * bary[k]);
                        atomicAdd(&gverts[(size_t)vid[k] * 4 + 3], c1 * bary[k]);
                    }
                }
            }
        }
        int slot_a;
        const float4 fr = fragment_of(cell0, slot_a);
        if (slot_a >= 0) {
            T.key_pos = slot_a;
            T.pA = upper ? fr.y : fr.x; T.pB = upper ? fr.x : fr.y; T.p2 = fr.z;
            position_terms(fr, slot_a, gx, gy, sc[pix][C], sc[pix][C + 1], sc[pix][C + 2]);
        }
    }

    // ---- (4) per-face reduction -----------------------------------------------------------------------------------------
    // One iteration per occupied slot: the 3*(C+3) sums of the face are reduced over the 32 lanes with a transposed
    // butterfly (each lane ends up owning one finished sum) and leave the SM as ONE warp-wide RED.  Faces that own only a
    // few records in this tile skip the butterfly: their records are added directly, all such faces of the tile together,
    // in one pass of vector REDs at the end.
#if DIRT_ABLATE != 1
    {
        const int owner = owner_meta<C>(lane);
        // destination of this lane's finished sum: component (owner >> 2) & 3 of row `vid` of grad_vertices / grad_vertex_colors
        float* const owner_row = ((owner & 16) ? gverts : gcols) + ((owner >> 2) & 3);
        const int owner_stride = (owner & 16) ? 4 : (C == 4 ? 4 : gstride);
        const int kc0 = term[0].key_col, kc1 = term[1].key_col, kp0 = term[0].key_pos, kp1 = term[1].key_pos;
        unsigned direct = 0;   // bit 0/1: colour record of pixel 0/1, bit 2/3: position record of pixel 0/1
        // slots that own at least one record of this tile (faces of the ring that nothing dilates from own none)
        unsigned occupied = __reduce_or_sync(0xffffffffu, (kc0 >= 0 ? 1u << kc0 : 0u) | (kc1 >= 0 ? 1u << kc1 : 0u) |
                                                              (kp0 >= 0 ? 1u << kp0 : 0u) | (kp1 >= 0 ? 1u << kp1 : 0u));
        while (occupied) {
            const int s = __ffs(occupied) - 1;
            occupied &= occupied - 1;
            const bool mc0 = kc0 == s, mc1 = kc1 == s, mp0 = kp0 == s, mp1 = kp1 == s;
#if DIRT_BWD_SMALL_FACE > 0
            const unsigned records = __reduce_add_sync(0xffffffffu, (unsigned)mc0 + (unsigned)mc1 + (unsigned)mp0 + (unsigned)mp1);
            if (records <= DIRT_BWD_SMALL_FACE) {
                direct |= (mc0 ? 1u : 0u) | (mc1 ? 2u : 0u) | (mp0 ? 4u : 0u) | (mp1 ? 8u : 0u);
                continue;
            }
#endif
            // First butterfly step at operand level: this lane keeps the NS sums of vertex A and hands those of vertex B
            // to lane^16 (the weights were arranged per half-warp when they were stored), and the halves swap one half
            // each of the NS sums of vertex 2.  The remaining steps are the generic transposed butterfly.
            constexpr int H2 = (NS + 1) / 2;
            float keep[NS], send[NS], third[NS];
#pragma unroll
            for (int pix = 0; pix < 2; ++pix) {
                const PixelTerms& T = term[pix];
                const bool mc = pix ? mc1 : mc0, mp = pix ? mp1 : mp0;
                const float wcA = mc ? T.cA : 0.f, wcB = mc ? T.cB : 0.f, wc2 = mc ? T.c2 : 0.f;
                const float wpA = mp ? T.pA : 0.f, wpB = mp ? T.pB : 0.f, wp2 = mp ? T.p2 : 0.f;
#pragma unroll
                for (int j = 0; j < NS; ++j) {
                    const float a = (j < C) ? wcA : wpA, bb = (j < C) ? wcB : wpB, cc = (j < C) ? wc2 : wp2;
                    keep[j] = (pix == 0) ? a * sc[pix][j] : fmaf(a, sc[pix][j], keep[j]);
                    send[j] = (pix == 0) ? bb * sc[pix][j] : fmaf(bb, sc[pix][j], send[j]);
                    third[j] = (pix == 0) ? cc * sc[pix][j] : fmaf(cc, sc[pix][j], third[j]);
                }
            }
            float v[NS + H2];
#pragma unroll
            for (int j = 0; j < NS; ++j) v[j] = keep[j] + __shfl_xor_sync(0xffffffffu, send[j], 16);
#pragma unroll
            for (int i = 0; i < H2; ++i) {
                const float hi = (H2 + i < NS) ? third[H2 + i] : 0.f;
                const float snd = upper ? third[i] : hi, kp = upper ? hi : third[i];
                v[NS + i] = kp + __shfl_xor_sync(0xffffffffu, snd, 16);
            }
            float total[1];
            TransposedReduce<NS + H2, 4>::run(v, lane, 8, total);
            if (owner >= 0) {
                const int4 q = reinterpret_cast<const int4*>(table + s)[2];   // {sC, v0, v1, v2}
                const int vid = (owner & 1) ? q.z : ((owner & 2) ? q.w : q.y);
                atomicAdd(owner_row + (size_t)vid * owner_stride, total[0]);
            }
        }
#if DIRT_BWD_SMALL_FACE > 0
        if (__any_sync(0xffffffffu, direct != 0u)) {
#pragma unroll
            for (int rec = 0; rec < 4; ++rec) {
                if (!(direct & (1u << rec))) continue;
                const int pix = rec & 1;
                const PixelTerms& T = term[pix];
                const bool colour = rec < 2;
                const int s = colour ? T.key_col : T.key_pos;
                const int4 q = reinterpret_cast<const int4*>(table + s)[2];
                const int vid[3] = {q.y, q.z, q.w};
                const float wA = colour ? T.cA : T.pA, wB = colour ? T.cB : T.pB;
                const float w[3] = {upper ? wB : wA, upper ? wA : wB, colour ? T.c2 : T.p2};
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    if (colour) {
                        if (C == 4) red_add_v4(gcols + (size_t)vid[k] * 4, w[k] * sc[pix][0], w[k] * sc[pix][1 % NS], w[k] * sc[pix][2 % NS], w[k] * sc[pix][3 % NS]);
                        else if (C == 3 && cs == 3 && gstride == 4) red_add_v4(gcols + (size_t)vid[k] * 4, w[k] * sc[pix][0], w[k] * sc[pix][1 % NS], w[k] * sc[pix][2 % NS], 0.f);
                        else {
#pragma unroll
                            for (int j = 0; j < C; ++j) atomicAdd(gcols + (size_t)vid[k] * gstride + j, w[k] * sc[pix][j]);
                        }
                    } else {
                        red_add_v4(gverts + (size_t)vid[k] * 4, w[k] * sc[pix][C], w[k] * sc[pix][C + 1], 0.f, w[k] * sc[pix][C + 2]);
                    }
                }
            }
        }
#endif
    }
#endif
}

// grad_vertex_colors of a 3-channel launch is accumulated in 16-byte rows (one vector RED per vertex instead of three
// scalar ones) and brought to its [.,3] layout afterwards
__global__ void __launch_bounds__(256) unpad_rows_kernel(const float* __restrict__ in, float* __restrict__ out, long long rows)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // one output element
    if (i >= rows * 3) return;
    const long long r = i / 3;
    out[i] = in[r * 4 + (i - r * 3)];
}

// grad_background of a background the batch shares: grad_bg[h,w,c] = sum_b [face_ids[b,h,w] < 0] * grad_pixels[b,h,w,c], the
// batch sum of what the tile kernel writes per image (store_gb; assemble_grads :143-148).  One thread per pixel (VEC4: C = 4,
// one 16-byte load per image) or per element; the sum runs in fp32 in increasing b without atomics, so the result is
// deterministic and equal, bit for bit, to a sequential fp32 loop over the per-image gradients.  UNROLL images' loads are
// issued before any of them is added.
__device__ __forceinline__ void add_to(float& a, float v) { a += v; }
__device__ __forceinline__ void add_to(float4& a, float4 v) { a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w; }

template <bool VEC4>
__global__ void __launch_bounds__(256) background_grad_kernel(const float* __restrict__ grad_pixels, const int32_t* __restrict__ face_ids,
                                                             float* __restrict__ grad_background, int B, long long HW, int C)
{
    using T = typename std::conditional<VEC4, float4, float>::type;
    constexpr int UNROLL = 8;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // pixel (VEC4) or element of [H,W,C]
    const long long img = VEC4 ? HW : HW * C;                              // T elements per image
    if (i >= img) return;
    const long long pix = VEC4 ? i : i / C;
    const T* gp = reinterpret_cast<const T*>(grad_pixels) + i;
    T acc{};
    for (int b0 = 0; b0 < B; b0 += UNROLL) {
        int id[UNROLL];
        T v[UNROLL];
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            id[k] = 0;
            v[k] = T{};
            if (b0 + k < B) { id[k] = __ldg(face_ids + (b0 + k) * HW + pix); v[k] = __ldg(gp + (b0 + k) * img); }
        }
#pragma unroll
        for (int k = 0; k < UNROLL; ++k)
            if (id[k] < 0) add_to(acc, v[k]);   // covered pixels (and images past the batch) add nothing
    }
    reinterpret_cast<T*>(grad_background)[i] = acc;
}

// ---- host side --------------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled tensor_map_encoder()
{
    static PFN_cuTensorMapEncodeTiled fn = []() -> PFN_cuTensorMapEncodeTiled {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            return nullptr;
        return reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    }();
    return fn;
}

// [B][H][W*elems] tensor of 4-byte elements, box [1][HALO_ROWS][box_pixels*elems]
static bool make_tile_map(CUtensorMap* map, const void* base, CUtensorMapDataType type, int B, int H, int W, int elems, int box_pixels)
{
    PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W * elems, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)W * elems * 4, (cuuint64_t)H * W * elems * 4};
    const cuuint32_t box[3] = {(cuuint32_t)(box_pixels * elems), (cuuint32_t)HALO_ROWS, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return enc(map, type, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int C, int NSLOT, bool USE_TMA>
static cudaError_t launch_tile_kernel(const CUtensorMap& px_map, const CUtensorMap& ids_map, const float* vertices,
                                      const float* pixels, const float* grad_pixels, const int32_t* face_ids,
                                      float* grad_background, float* grad_vertices, float* grad_vertex_colors,
                                      const Workspace& ws, const Dims& d, const unsigned char* tflags, int cs, int c0,
                                      int gstride, int flags, unsigned long long expect_tag, cudaStream_t stream)
{
    constexpr int NW = DIRT_BWD_WARPS;
    auto kernel = backward_tile_kernel<C, NSLOT, NW, USE_TMA>;
    constexpr int smem = BwdSmem<C, NSLOT>::BYTES * NW;
    static bool configured = false;   // per instantiation
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    for (int b_base = 0; b_base < d.B; b_base += 65535) {   // z: image
        const dim3 grid((unsigned)((d.btiles_x + NW - 1) / NW), (unsigned)d.btiles_y, (unsigned)min(d.B - b_base, 65535));
        kernel<<<grid, NW * 32, smem, stream>>>(px_map, ids_map, vertices, pixels, grad_pixels, face_ids, grad_background,
                                                grad_vertices, grad_vertex_colors, ws, d, tflags, cs, c0, gstride, flags, expect_tag, b_base);
    }
    return cudaGetLastError();
}

cudaError_t launch_backward(const float* vertices, const float* pixels, const float* grad_pixels,
                            const int32_t* face_ids, float* grad_background, float* grad_vertices,
                            float* grad_vertex_colors, const Workspace& ws, const Dims& d, const GroupSpec& groups,
                            bool tile_flags_valid, int flags, unsigned long long expect_tag, cudaStream_t stream, int* launches)
{
    cudaError_t e;
    const size_t vrows = (size_t)((flags & BWD_SHARED_GEOMETRY) ? 1 : d.B) * d.V;                      // rows of grad_vertices
    const size_t crows = (size_t)((flags & (BWD_SHARED_GEOMETRY | SHARED_COLOURS)) ? 1 : d.B) * d.V;  // rows of grad_vertex_colors
    // C = 3 as one group: colour gradients go to padded rows in the workspace (see unpad_rows_kernel)
    const bool padded = d.C == 3 && groups.n == 1 && ws.gc_pad != nullptr && crows > 0;
    float* const gc_out = grad_vertex_colors;
    if (padded) grad_vertex_colors = ws.gc_pad;
    const int gstride = padded ? 4 : d.C;
    if (grad_vertex_colors == grad_vertices + vrows * 4) {
        // the two gradients are the halves of one flat buffer (what a multi-GPU job exchanges): one memset node
        if ((e = cudaMemsetAsync(grad_vertices, 0, sizeof(float) * (vrows * 4 + crows * gstride), stream)) != cudaSuccess) return e;
    } else {
        if ((e = cudaMemsetAsync(grad_vertices, 0, sizeof(float) * vrows * 4, stream)) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(grad_vertex_colors, 0, sizeof(float) * crows * gstride, stream)) != cudaSuccess) return e;
    }
    const auto finish = [&]() -> cudaError_t {
        if (!padded) return cudaSuccess;
        const long long n = (long long)crows * 3;
        unpad_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grad_vertex_colors, gc_out, (long long)crows);
        ++*launches;
        return cudaGetLastError();
    };
    if ((flags & SHARED_BACKGROUND) && !(flags & BWD_SKIP_COLOUR) && grad_background && d.B > 0) {
        // the batch-summed gradient of a shared background: one launch per call, whatever the channel grouping
        ScopedKernelTimer timer(3, stream);
        const long long HW = (long long)d.H * d.W;
        const bool vec4 = d.C == 4 && (((uintptr_t)grad_pixels | (uintptr_t)grad_background) % 16 == 0);
        const long long n = vec4 ? HW : HW * d.C;
        if (vec4) background_grad_kernel<true><<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grad_pixels, face_ids, grad_background, d.B, HW, d.C);
        else background_grad_kernel<false><<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grad_pixels, face_ids, grad_background, d.B, HW, d.C);
        ++*launches;
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    const long long total_tiles = (long long)d.B * d.btiles;
    if (total_tiles == 0) return finish();
    ScopedKernelTimer timer(2, stream);
    // C == 4 with the default grouping {3,1} and 16-byte aligned tensors: one fused launch.  Everything else: one launch
    // per channel group (width 3 or 1) on its slice of the channels -- what the reference does at the Python level
    // (dirt/rasterise_ops.py:86-108), except that nothing is sliced or copied and grad_vertices accumulates in place.
    const bool fused4 = d.C == 4 && groups.n == 2 && groups.width[0] == 3 && groups.width[1] == 1 &&
                        (((uintptr_t)pixels | (uintptr_t)grad_pixels | (uintptr_t)grad_background | (uintptr_t)grad_vertex_colors) % 16 == 0);
    const unsigned char* tflags = tile_flags_valid ? ws.tile_flags : nullptr;
    // TMA staging needs tensors it can describe: the group is the whole pixel (cs == C), rows are multiples of 16 bytes
    // and the bases 16-byte aligned; everything else is staged with per-lane cp.async
    CUtensorMap px_map, ids_map;
    memset(&px_map, 0, sizeof(px_map));
    memset(&ids_map, 0, sizeof(ids_map));
    if (!(flags & BWD_SKIP_POSITION) && !pixels) return cudaErrorInvalidValue;
    bool tma = DIRT_BWD_TMA && pixels && (d.C == 1 || d.C == 3 || fused4) && groups.n == (fused4 ? 2 : 1) && d.W % 4 == 0 &&
               ((uintptr_t)pixels % 16 == 0) && ((uintptr_t)face_ids % 16 == 0);
    if (tma)
        tma = make_tile_map(&px_map, pixels, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d.B, d.H, d.W, d.C, d.C == 4 ? PxTile<4>::COLS : PxTile<3>::COLS) &&
              make_tile_map(&ids_map, face_ids, CU_TENSOR_MAP_DATA_TYPE_INT32, d.B, d.H, d.W, 1, IDS_COLS);
#define DIRT_LAUNCH(CC, NSLOT, c0)                                                                                             \
    (tma ? launch_tile_kernel<CC, NSLOT, true>(px_map, ids_map, vertices, pixels, grad_pixels, face_ids, grad_background,       \
                                               grad_vertices, grad_vertex_colors, ws, d, tflags, d.C, c0, gstride, flags, expect_tag, stream)      \
         : launch_tile_kernel<CC, NSLOT, false>(px_map, ids_map, vertices, pixels, grad_pixels, face_ids, grad_background,      \
                                                grad_vertices, grad_vertex_colors, ws, d, tflags, d.C, c0, gstride, flags, expect_tag, stream))
    if (fused4) {
        ++*launches;
        const cudaError_t le = DIRT_LAUNCH(4, DIRT_BWD_SLOTS_C4, 0);
        return le != cudaSuccess ? le : finish();
    }
    int c0 = 0;
    for (int g = 0; g < groups.n; ++g) {
        const cudaError_t le = groups.width[g] == 3 ? DIRT_LAUNCH(3, DIRT_BWD_SLOTS_C3, c0) : DIRT_LAUNCH(1, DIRT_BWD_SLOTS_C3, c0);
        c0 += groups.width[g];
        ++*launches;
        if (le != cudaSuccess) return le;
    }
#undef DIRT_LAUNCH
    return finish();
}

}  // namespace dirt
