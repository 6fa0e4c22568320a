// setup.cu -- triangle setup and per-tile binning.
//
// Replaces, for the sm_100a path, what the reference delegates to the OpenGL vertex pipeline
// (clip -> NDC -> viewport; csrc/rasterise_egl.cpp:362-380) and the vertex expansion kernel
// upload_vertices (csrc/rasterise_grad_egl.cu:12-34).
//
//   setup_kernel : one thread per (image, face): S1-S6 of the visibility specification ->
//                  TriCov + TriInterp + TriXY records, and -- in the same pass -- binning: the face is appended to the
//                  fixed-capacity bin of every tile its bounding box touches (faces spanning <= SMALL_TILE_LIMIT
//                  tiles; position = atomicAdd on the tile's count, overflow -> the image's overflow list) or to
//                  the per-image large list.  The order inside a bin is irrelevant: visibility is the minimum of
//                  (depth key, face index).  No scan, no second pass.
#include "common.cuh"

namespace dirt {

constexpr float GUARD_BAND = 8388608.0f;  // 2^23 sub-pixel units = 32768 px

// 128 threads x 8 blocks per SM (<= 64 registers): measured best, profiles/r01_sweep_setup.txt
#ifndef DIRT_SETUP_THREADS
#define DIRT_SETUP_THREADS 128
#endif
#ifndef DIRT_SETUP_MIN_BLOCKS
#define DIRT_SETUP_MIN_BLOCKS 8
#endif
template <bool BIN>
__global__ void __launch_bounds__(DIRT_SETUP_THREADS, DIRT_SETUP_MIN_BLOCKS) setup_kernel(const float* __restrict__ vertices,
                                                    const int32_t* __restrict__ faces, const float* __restrict__ vertex_colors,
                                                    Workspace ws, Dims d)
{
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)d.B * d.F;
    if (gid == 0) ws.header->tag = workspace_tag(vertices, faces, d.B, d.H, d.W, d.V, d.F, d.face_stride == 0);
    if (gid >= total) return;
    const int b = (int)(gid / d.F);
    const int f = (int)(gid - (long long)b * d.F);
    const float* verts = vertices + (size_t)b * d.V * 4;

    // A face that cannot produce a fragment leaves a defined record (kind = culled, edge functions negative) and is not
    // binned.  Every rejection below ends here, so the path of a face that survives has no merges with default values.
    const auto cull = [&]() {
        uint4* c = reinterpret_cast<uint4*>(ws.cov + gid);
        c[0] = make_uint4(0u, 0u, 0u, 0u);                            // A0 B0 A1 B1
        c[1] = make_uint4(0u, 0u, 0u, 0u);                            // A2 B2 zA zB
        c[2] = make_uint4(~0u, ~0u, ~0u, ~0u);                        // q0 = q1 = -1
        c[3] = make_uint4(~0u, ~0u, 0u, KIND_CULLED);                 // q2 = -1, zC, kind
        uint4* i = reinterpret_cast<uint4*>(ws.itp + gid);
        i[0] = make_uint4(0u, 0u, 0u, 0u);
        i[1] = make_uint4(0u, 0u, 0u, 0u);
        i[2] = make_uint4(__float_as_uint(1.0f), 0u, 0u, 0u);         // sC = 1, v0..v2 = 0
        i[3] = make_uint4(0u, 0u, 0u, 0u);
        uint4* x = reinterpret_cast<uint4*>(ws.xy + gid);
        x[0] = make_uint4(0u, 0u, 0u, 0u);
        x[1] = make_uint4(0u, 0u, 0u, 0u);
    };

    int32_t vid[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) vid[k] = __ldg(&faces[((size_t)b * d.face_stride + f) * 3 + k]);
    if ((unsigned)vid[0] >= (unsigned)d.V || (unsigned)vid[1] >= (unsigned)d.V || (unsigned)vid[2] >= (unsigned)d.V) { cull(); return; }

    float p[3][4];
    bool finite = true;
    int n_behind = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(verts) + vid[k]);
        p[k][0] = v.x; p[k][1] = v.y; p[k][2] = v.z; p[k][3] = v.w;
        finite = finite && isfinite(v.x) && isfinite(v.y) && isfinite(v.z) && isfinite(v.w);
        if (!(v.w > 0.0f)) ++n_behind;
    }
    if (!finite || n_behind == 3) { cull(); return; }

    // S1-S3: window coordinates snapped to 1/256 px; a vertex behind the eye or outside the guard band makes the face "hard"
    bool hard = n_behind > 0;
    int32_t xi[3] = {0, 0, 0}, yi[3] = {0, 0, 0};
    if (!hard) {
        const float halfW = 0.5f * (float)d.W, halfH = 0.5f * (float)d.H;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float xn = __fdiv_rn(p[k][0], p[k][3]);
            const float yn = __fdiv_rn(p[k][1], p[k][3]);
            const float X = __fmul_rn(__fadd_rn(xn, 1.0f), halfW);
            const float Y = __fmul_rn(__fsub_rn(1.0f, yn), halfH);
            const float fx = __fmul_rn(X, 256.0f), fy = __fmul_rn(Y, 256.0f);
            if (!(fabsf(fx) <= GUARD_BAND) || !(fabsf(fy) <= GUARD_BAND)) hard = true;
            else { xi[k] = __float2int_rn(fx); yi[k] = __float2int_rn(fy); }
        }
    }

    // S6: interpolation and depth planes
    double gq[3][3], gs[3], gz[3];
    if (!exact::planes_double(p, d.ps, gq, gs, gz)) { cull(); return; }

    // S4-S5: edge functions and the pixel bounding box of a normal face; a hard face may touch any pixel
    int32_t A[3] = {0, 0, 0}, Bc[3] = {0, 0, 0};
    int64_t q_abs[3] = {-1, -1, -1};
    int cmin = 0, cmax = d.W - 1, rmin = 0, rmax = d.H - 1;
    if (!hard) {
        const int64_t ax = xi[0], ay = yi[0], bx = xi[1], by = yi[1], cx = xi[2], cy = yi[2];
        const int64_t area2 = (bx - ax) * (cy - ay) - (cx - ax) * (by - ay);
        if (area2 == 0) { cull(); return; }
        int32_t px[3] = {xi[0], xi[1], xi[2]}, py[3] = {yi[0], yi[1], yi[2]};
        if (area2 < 0) {
            int32_t t = px[1]; px[1] = px[2]; px[2] = t;
            t = py[1]; py[1] = py[2]; py[2] = t;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int a = (k + 1) % 3, bb = (k + 2) % 3;
            const int64_t Ak = (int64_t)py[a] - py[bb];
            const int64_t Bk = (int64_t)px[bb] - px[a];
            const int64_t Ck = -(Ak * px[a] + Bk * py[a]);
            const bool tl = (Ak > 0) || (Ak == 0 && Bk > 0);
            const int64_t Cpp = 128 * (Ak + Bk) + Ck - (tl ? 0 : 1);
            A[k] = (int32_t)Ak; Bc[k] = (int32_t)Bk; q_abs[k] = Cpp >> 8;
        }
        const int32_t xmin = min(px[0], min(px[1], px[2])), xmax = max(px[0], max(px[1], px[2]));
        const int32_t ymin = min(py[0], min(py[1], py[2])), ymax = max(py[0], max(py[1], py[2]));
        cmin = max((xmin + 127) >> 8, 0); cmax = min((xmax - 128) >> 8, d.W - 1);
        rmin = max((ymin + 127) >> 8, 0); rmax = min((ymax - 128) >> 8, d.H - 1);
        if (cmin > cmax || rmin > rmax) { cull(); return; }
    }

    // interpolation record: planes relative to the bbox corner of a normal face (absolute for a hard one)
    const int cref = hard ? 0 : cmin, rref = hard ? 0 : rmin;
    {
        const double cr = (double)cref, rr = (double)rref;
        TriInterp itp;
        itp.q0A = (float)gq[0][0]; itp.q0B = (float)gq[0][1];
        itp.q0C = (float)__dadd_rn(__dadd_rn(__dmul_rn(gq[0][0], cr), __dmul_rn(gq[0][1], rr)), gq[0][2]);
        itp.q1A = (float)gq[1][0]; itp.q1B = (float)gq[1][1];
        itp.q1C = (float)__dadd_rn(__dadd_rn(__dmul_rn(gq[1][0], cr), __dmul_rn(gq[1][1], rr)), gq[1][2]);
        itp.sA = (float)gs[0]; itp.sB = (float)gs[1];
        itp.sC = (float)__dadd_rn(__dadd_rn(__dmul_rn(gs[0], cr), __dmul_rn(gs[1], rr)), gs[2]);
        itp.v0 = vid[0]; itp.v1 = vid[1]; itp.v2 = vid[2];
        itp.cref = cref; itp.rref = rref;
        itp.pad0 = itp.pad1 = 0;
        union { TriInterp t; uint4 u[4]; } i; i.t = itp;
        uint4* dsti = reinterpret_cast<uint4*>(ws.itp + gid);
        dsti[0] = i.u[0]; dsti[1] = i.u[1]; dsti[2] = i.u[2]; dsti[3] = i.u[3];
        float4* dstx = reinterpret_cast<float4*>(ws.xy + gid);
        dstx[0] = make_float4(p[0][0], p[0][1], p[1][0], p[1][1]);
        dstx[1] = make_float4(p[2][0], p[2][1], 0.f, 0.f);
        // shading record: planes of N_c = q0*(c0 - c2) + q1*(c1 - c2) + S*c2 (q2 = S - q0 - q1), values only
        if (BIN && vertex_colors != nullptr) {
            const float* cols = vertex_colors + (size_t)b * d.col_stride * d.C;
            float4 out[4];
            out[0] = make_float4(itp.sA, itp.sB, itp.sC, __uint_as_float((uint32_t)cref | ((uint32_t)rref << 16)));
            float n[12];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                double c0 = 0.0, c1 = 0.0, c2 = 0.0;
                if (c < d.C) {
                    c0 = (double)__ldg(cols + (size_t)vid[0] * d.C + c);
                    c1 = (double)__ldg(cols + (size_t)vid[1] * d.C + c);
                    c2 = (double)__ldg(cols + (size_t)vid[2] * d.C + c);
                }
                const double d0 = c0 - c2, d1 = c1 - c2;
                const double nA = gq[0][0] * d0 + gq[1][0] * d1 + gs[0] * c2;
                const double nB = gq[0][1] * d0 + gq[1][1] * d1 + gs[1] * c2;
                const double nC = gq[0][2] * d0 + gq[1][2] * d1 + gs[2] * c2;
                n[3 * c] = (float)nA; n[3 * c + 1] = (float)nB; n[3 * c + 2] = (float)((nA * cr + nB * rr) + nC);
            }
            out[1] = make_float4(n[0], n[1], n[2], n[3]);
            out[2] = make_float4(n[4], n[5], n[6], n[7]);
            out[3] = make_float4(n[8], n[9], n[10], n[11]);
            float4* dsts = reinterpret_cast<float4*>(ws.shade + gid);
            dsts[0] = out[0]; dsts[1] = out[1]; dsts[2] = out[2]; dsts[3] = out[3];
        }
    }

    // tile bounding box and the layout of the coverage record.
    // "small" faces are binned per tile and rasterised entirely in int32: that needs a bounded tile count AND bounded
    // edge coefficients (a huge, mostly off-screen face can have a small clamped bbox): |A|,|B| < 2^18, |q_rel| < 2^29
    // keep q_rel + A*dcol + B*drow (|dcol|,|drow| < 2^9 inside the binned tiles) below 2^31.
    const int tx0 = cmin >> TILE_W_SHIFT, tx1 = cmax >> TILE_W_SHIFT;
    const int ty0 = rmin >> TILE_H_SHIFT, ty1 = rmax >> TILE_H_SHIFT;
    const int64_t q0r = q_abs[0] + (int64_t)A[0] * cmin + (int64_t)Bc[0] * rmin;
    const int64_t q1r = q_abs[1] + (int64_t)A[1] * cmin + (int64_t)Bc[1] * rmin;
    const int64_t q2r = q_abs[2] + (int64_t)A[2] * cmin + (int64_t)Bc[2] * rmin;
    const int32_t cmax_abs = max(max(max(abs(A[0]), abs(Bc[0])), max(abs(A[1]), abs(Bc[1]))), max(abs(A[2]), abs(Bc[2])));
    const int64_t qlim = (int64_t)1 << 29;
    const bool small = !hard && (tx1 - tx0 + 1) * (ty1 - ty0 + 1) <= SMALL_TILE_LIMIT && cmax_abs < (1 << 18) &&
                       q0r > -qlim && q0r < qlim && q1r > -qlim && q1r < qlim && q2r > -qlim && q2r < qlim;
    {
        TriCov cov;
        cov.A0 = A[0]; cov.B0 = Bc[0]; cov.A1 = A[1]; cov.B1 = Bc[1]; cov.A2 = A[2]; cov.B2 = Bc[2];
        const float zA = (float)gz[0], zB = (float)gz[1], zC = (float)gz[2];
        if (small) {
            cov.s.kind = KIND_SMALL;
            cov.s.q0r = (int32_t)q0r; cov.s.q1r = (int32_t)q1r; cov.s.q2r = (int32_t)q2r;
            cov.s.zA = zA; cov.s.zB = zB; cov.s.zC = zC;
            cov.s.cref = cmin; cov.s.rref = rmin; cov.s.pad = 0;
        } else {
            cov.l.kind = hard ? KIND_HARD : KIND_LARGE;
            cov.l.q0 = q_abs[0]; cov.l.q1 = q_abs[1]; cov.l.q2 = q_abs[2];
            cov.l.zA = zA; cov.l.zB = zB; cov.l.zC = zC;
        }
        union { TriCov t; uint4 u[4]; } c; c.t = cov;
        uint4* dst = reinterpret_cast<uint4*>(ws.cov + gid);
        dst[0] = c.u[0]; dst[1] = c.u[1]; dst[2] = c.u[2]; dst[3] = c.u[3];
    }
    if (!BIN) return;

    const auto to_large_list = [&]() {
        const int pos = atomicAdd(&ws.large_count[b], 1);
        ws.large_list[(size_t)b * d.F + pos] = f;
    };
    if (small) {
        int* counts = ws.tile_count + (size_t)b * d.tiles;
        const auto place = [&](int t, int pos) {
            if (pos < BIN_CAP) {
                ws.bins[((size_t)b * d.tiles + t) * BIN_CAP + pos] = f;
            } else {
                // the tile's bin is full: the overflow list of its row of tiles, and if that is full as well the large list
                // (a face that sits in both a bin and the large list is tested twice, which cannot change a minimum)
                const size_t row = (size_t)b * d.tiles_y + t / d.tiles_x;
                const int q = atomicAdd(&ws.ovf_count[row], 1);
                if (q < OVF_ROW_CAP) ws.ovf[row * OVF_ROW_CAP + q] = make_int2(t, f);
                else {
                    // one byte per face, claimed with an atomic OR on the word holding it
                    unsigned int* word = reinterpret_cast<unsigned int*>(ws.face_in_large) + (gid >> 2);
                    const unsigned int bit = 1u << (8 * (unsigned)(gid & 3));
                    if ((atomicOr(word, bit) & bit) == 0u) to_large_list();
                }
            }
        };
        if (tx1 - tx0 <= 1 && ty1 - ty0 <= 1) {
            // at most 2x2 tiles (nearly every face of a fine mesh): the position-returning atomics go out together, so the
            // thread waits for one round trip instead of up to four in a row
            const int t00 = ty0 * d.tiles_x + tx0, t01 = ty0 * d.tiles_x + tx1, t10 = ty1 * d.tiles_x + tx0, t11 = ty1 * d.tiles_x + tx1;
            const bool two_x = tx1 > tx0, two_y = ty1 > ty0;
            const int p00 = atomicAdd(&counts[t00], 1);
            const int p01 = two_x ? atomicAdd(&counts[t01], 1) : 0;
            const int p10 = two_y ? atomicAdd(&counts[t10], 1) : 0;
            const int p11 = (two_x && two_y) ? atomicAdd(&counts[t11], 1) : 0;
            place(t00, p00);
            if (two_x) place(t01, p01);
            if (two_y) place(t10, p10);
            if (two_x && two_y) place(t11, p11);
        } else {
            for (int ty = ty0; ty <= ty1; ++ty)
                for (int tx = tx0; tx <= tx1; ++tx) {
                    const int t = ty * d.tiles_x + tx;
                    place(t, atomicAdd(&counts[t], 1));
                }
        }
    } else {
        to_large_list();
    }
}

cudaError_t launch_setup_and_bin(const float* vertices, const int32_t* faces, const float* vertex_colors, const Workspace& ws,
                                 const Dims& d, cudaStream_t stream, int* launches)
{
    if (!shade_records_ok(d)) vertex_colors = nullptr;
    const long long total = (long long)d.B * d.F;
    cudaError_t e;
    if ((e = cudaMemsetAsync(ws.tile_count, 0, ws.zero_bytes, stream)) != cudaSuccess) return e;
    if (total > 0) {
        setup_kernel<true><<<(unsigned)((total + DIRT_SETUP_THREADS - 1) / DIRT_SETUP_THREADS), DIRT_SETUP_THREADS, 0, stream>>>(vertices, faces, vertex_colors, ws, d);
        ++*launches;
    }
    return cudaGetLastError();
}

cudaError_t launch_setup_only(const float* vertices, const int32_t* faces, const Workspace& ws, const Dims& d,
                              cudaStream_t stream, int* launches)
{
    const long long total = (long long)d.B * d.F;
    cudaError_t e;
    if ((e = cudaMemsetAsync(ws.header, 0, sizeof(Header), stream)) != cudaSuccess) return e;
    if (total > 0) {
        setup_kernel<false><<<(unsigned)((total + DIRT_SETUP_THREADS - 1) / DIRT_SETUP_THREADS), DIRT_SETUP_THREADS, 0, stream>>>(vertices, faces, nullptr, ws, d);
        ++*launches;
    }
    return cudaGetLastError();
}

}  // namespace dirt
