// api.cu -- the C ABI of libdirt_b200.so (include/dirt_b200.h): argument validation, workspace
// carving and kernel sequencing.  No device allocation, no host synchronisation, no global state
// other than a thread-local launch counter.
#include "../../include/dirt_b200.h"
#include "common.cuh"

using namespace dirt;

static_assert(BWD_SHARED_GEOMETRY == DIRT_BWD_SHARED_GEOMETRY && BWD_SKIP_POSITION == DIRT_BWD_SKIP_POSITION &&
              BWD_SKIP_COLOUR == DIRT_BWD_SKIP_COLOUR && SHARED_BACKGROUND == DIRT_SHARED_BACKGROUND &&
              SHARED_COLOURS == DIRT_SHARED_COLOURS && SHARED_FACES == DIRT_SHARED_FACES,
              "flag values of common.cuh and dirt_b200.h differ");

static constexpr int SHARING_BITS = DIRT_SHARED_BACKGROUND | DIRT_SHARED_COLOURS | DIRT_SHARED_FACES;

static thread_local int t_last_launches = 0;

extern "C" const char* dirt_error_string(int code)
{
    switch (code) {
        case DIRT_OK: return "ok";
        case DIRT_ERR_BAD_SHAPE:
            return "bad shape: need B >= 0, H > 0, W > 0, C > 0, V >= 0, F >= 0 (and sizes within int32 range)";
        case DIRT_ERR_NULL_POINTER: return "a required pointer is NULL";
        case DIRT_ERR_WORKSPACE_TOO_SMALL: return "workspace smaller than dirt_workspace_bytes()";
        case DIRT_ERR_BAD_CHANNEL_GROUPS: return "channel groups must each be 1 or 3 wide and sum to C";
        case DIRT_ERR_TOO_MANY_VERTICES: return "RasteriseGrad supports a maximum of 16777216 vertices";
        case DIRT_ERR_CUDA: return "a CUDA call or kernel launch failed";
        case DIRT_ERR_MISALIGNED: return "pointer not sufficiently aligned (workspace 256 B, vertices 16 B, others 4 B)";
        case DIRT_ERR_STALE_WORKSPACE:
            return "workspace_holds_setup was set, but the workspace does not hold the setup records of these (vertices, faces, sizes)";
        default: return "unknown error code";
    }
}

extern "C" int dirt_abi_version(void) { return 4; }

namespace dirt {
KernelTimer& kernel_timer()
{
    static thread_local KernelTimer t;
    return t;
}
}  // namespace dirt

extern "C" int dirt_kernel_timer_enable(int which)
{
    KernelTimer& t = kernel_timer();
    if (which < 0 || which > 3) return DIRT_ERR_BAD_SHAPE;
    if (which != 0 && !t.start) {
        if (cudaEventCreate(&t.start) != cudaSuccess || cudaEventCreate(&t.stop) != cudaSuccess) {
            t.start = t.stop = nullptr;
            return DIRT_ERR_CUDA;
        }
    }
    t.which = which;
    t.recorded = false;
    return DIRT_OK;
}

extern "C" float dirt_kernel_timer_elapsed_ms(void)
{
    KernelTimer& t = kernel_timer();
    if (!t.recorded) return -1.f;
    float ms = -1.f;
    if (cudaEventSynchronize(t.stop) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, t.start, t.stop) != cudaSuccess) return -1.f;
    return ms;
}

extern "C" int dirt_last_launch_count(void) { return t_last_launches; }

static bool shape_ok(int B, int H, int W, int C, int V, int F)
{
    if (B < 0 || H <= 0 || W <= 0 || C <= 0 || V < 0 || F < 0) return false;
    if (C / 3 + C % 3 > MAX_GROUPS) return false;             // the greedy split of C (groups of 3, then of 1) must fit GroupSpec
    if ((long long)H * W > (1ll << 30)) return false;         // row*W+col stays in int32
    if ((long long)W > (1 << 18) || (long long)H > (1 << 18)) return false;
    if ((long long)B * F > (1ll << 31) - 1) return false;
    if ((long long)B * ((W + TILE_W - 1) / TILE_W) * ((H + TILE_H - 1) / TILE_H) > (1ll << 31) - 1) return false;   // tile indices are int32
    return true;
}

extern "C" size_t dirt_workspace_bytes(int B, int H, int W, int C, int V, int F)
{
    if (!shape_ok(B, H, W, C > 0 ? C : 1, V, F)) return 0;
    Workspace ws = carve_workspace(nullptr, B, H, W, C, V, F);
    return ws.bytes + 256;
}

static int make_groups(int C, const int* channel_groups, int n_groups, GroupSpec* g)
{
    g->n = 0;
    if (channel_groups && n_groups > 0) {
        if (n_groups > MAX_GROUPS) return DIRT_ERR_BAD_CHANNEL_GROUPS;
        int sum = 0;
        for (int i = 0; i < n_groups; ++i) {
            if (channel_groups[i] != 1 && channel_groups[i] != 3) return DIRT_ERR_BAD_CHANNEL_GROUPS;
            g->width[i] = (unsigned char)channel_groups[i];
            sum += channel_groups[i];
        }
        if (sum != C) return DIRT_ERR_BAD_CHANNEL_GROUPS;
        g->n = n_groups;
        return DIRT_OK;
    }
    // the reference's own greedy split (dirt/rasterise_ops.py:80-108)
    if (C == 1 || C == 3) { g->width[0] = (unsigned char)C; g->n = 1; return DIRT_OK; }
    int begin = 0;
    while (begin < C) {
        const int w = (begin + 3 <= C) ? 3 : 1;
        if (g->n >= MAX_GROUPS) return DIRT_ERR_BAD_CHANNEL_GROUPS;
        g->width[g->n++] = (unsigned char)w;
        begin += w;
    }
    return DIRT_OK;
}

extern "C" size_t dirt_workspace_bytes_min(int B, int H, int W, int C, int V, int F)
{
    if (!shape_ok(B, H, W, C > 0 ? C : 1, V, F)) return 0;
    Workspace ws = carve_workspace(nullptr, B, H, W, C, V, F);
    return ws.bytes_without_face_ids + 256;
}

// needs_face_id_scratch: only a backward call without face ids derives them into the workspace's last block
static int check_workspace(void* workspace, size_t workspace_bytes, int B, int H, int W, int C, int V, int F,
                           bool needs_face_id_scratch = false)
{
    if (!workspace) return DIRT_ERR_NULL_POINTER;
    if ((uintptr_t)workspace % 256 != 0) return DIRT_ERR_MISALIGNED;
    const size_t need = needs_face_id_scratch ? dirt_workspace_bytes(B, H, W, C, V, F) : dirt_workspace_bytes_min(B, H, W, C, V, F);
    if (workspace_bytes < need) return DIRT_ERR_WORKSPACE_TOO_SMALL;
    return DIRT_OK;
}

#define CUDA_TRY(expr)                                   \
    do {                                                 \
        cudaError_t e__ = (expr);                        \
        if (e__ != cudaSuccess) { t_last_launches = launches; return DIRT_ERR_CUDA; } \
    } while (0)

extern "C" int dirt_rasterise_forward_ex(const float* background, const float* vertices, const float* vertex_colors,
                                         const int32_t* faces, float* pixels, int32_t* face_ids_out, int B, int H, int W,
                                         int C, int V, int F, void* workspace, size_t workspace_bytes, void* cuda_stream, int flags)
{
    int launches = 0;
    t_last_launches = 0;
    if (!shape_ok(B, H, W, C, V, F)) return DIRT_ERR_BAD_SHAPE;
    if (flags & ~SHARING_BITS) return DIRT_ERR_BAD_SHAPE;
    if (B == 0) return DIRT_OK;
    if (!background || !pixels) return DIRT_ERR_NULL_POINTER;
    if ((V > 0 && (!vertices || !vertex_colors)) || (F > 0 && !faces)) return DIRT_ERR_NULL_POINTER;
    if ((uintptr_t)vertices % 16 != 0) return DIRT_ERR_MISALIGNED;
    if ((uintptr_t)background % 4 || (uintptr_t)pixels % 4 || (uintptr_t)vertex_colors % 4 || (uintptr_t)faces % 4 ||
        (uintptr_t)face_ids_out % 4)
        return DIRT_ERR_MISALIGNED;
    int rc = check_workspace(workspace, workspace_bytes, B, H, W, C, V, F);
    if (rc != DIRT_OK) return rc;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const Workspace ws = carve_workspace(workspace, B, H, W, C, V, F);
    const Dims d = make_dims(B, H, W, C, V, F, flags);
    CUDA_TRY(launch_setup_and_bin(vertices, faces, vertex_colors, ws, d, stream, &launches));
    CUDA_TRY(launch_raster_forward(vertices, background, vertex_colors, pixels, face_ids_out, ws, d, stream, &launches));
    t_last_launches = launches;
    return DIRT_OK;
}

extern "C" int dirt_rasterise_forward(const float* background, const float* vertices, const float* vertex_colors,
                                      const int32_t* faces, float* pixels, int32_t* face_ids_out, int B, int H, int W,
                                      int C, int V, int F, void* workspace, size_t workspace_bytes, void* cuda_stream)
{
    return dirt_rasterise_forward_ex(background, vertices, vertex_colors, faces, pixels, face_ids_out, B, H, W, C, V, F,
                                     workspace, workspace_bytes, cuda_stream, 0);
}

extern "C" int dirt_rasterise_visibility(const float* vertices, const int32_t* faces, int32_t* face_ids, float* gbuffer,
                                         int B, int H, int W, int V, int F, void* workspace, size_t workspace_bytes,
                                         void* cuda_stream)
{
    int launches = 0;
    t_last_launches = 0;
    if (!shape_ok(B, H, W, 1, V, F)) return DIRT_ERR_BAD_SHAPE;
    if (B == 0) return DIRT_OK;
    if ((V > 0 && !vertices) || (F > 0 && !faces)) return DIRT_ERR_NULL_POINTER;
    if ((uintptr_t)vertices % 16 != 0 || (uintptr_t)gbuffer % 16 != 0 || (uintptr_t)face_ids % 4 != 0)
        return DIRT_ERR_MISALIGNED;
    int rc = check_workspace(workspace, workspace_bytes, B, H, W, 1, V, F);
    if (rc != DIRT_OK) return rc;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const Workspace ws = carve_workspace(workspace, B, H, W, 1, V, F);
    const Dims d = make_dims(B, H, W, 1, V, F);
    CUDA_TRY(launch_setup_and_bin(vertices, faces, nullptr, ws, d, stream, &launches));
    CUDA_TRY(launch_raster_visibility(vertices, face_ids, gbuffer, ws, d, stream, &launches));
    t_last_launches = launches;
    return DIRT_OK;
}

static int backward_impl(const float* vertices, const int32_t* faces, const float* pixels, const float* grad_pixels,
                         const int32_t* face_ids, float* grad_background, float* grad_vertices, float* grad_vertex_colors,
                         int B, int H, int W, int C, int V, int F, const int* channel_groups, int n_groups,
                         int workspace_holds_setup, int flags, void* workspace, size_t workspace_bytes, void* cuda_stream)
{
    int launches = 0;
    t_last_launches = 0;
    if (!shape_ok(B, H, W, C, V, F)) return DIRT_ERR_BAD_SHAPE;
    if (V > (1 << 24)) return DIRT_ERR_TOO_MANY_VERTICES;
    if (flags & ~(DIRT_BWD_SHARED_GEOMETRY | DIRT_BWD_SKIP_POSITION | DIRT_BWD_SKIP_COLOUR | SHARING_BITS)) return DIRT_ERR_BAD_SHAPE;
    GroupSpec groups;
    int rc = make_groups(C, channel_groups, n_groups, &groups);
    if (rc != DIRT_OK) return rc;
    if (B == 0) return DIRT_OK;
    if (!grad_pixels) return DIRT_ERR_NULL_POINTER;
    if (!(flags & DIRT_BWD_SKIP_POSITION) && !pixels) return DIRT_ERR_NULL_POINTER;
    // a shared background's gradient may be NULL: not wanted
    if (!(flags & (DIRT_BWD_SKIP_COLOUR | DIRT_SHARED_BACKGROUND)) && !grad_background) return DIRT_ERR_NULL_POINTER;
    if ((V > 0 && (!vertices || !grad_vertices || !grad_vertex_colors)) || (F > 0 && !faces)) return DIRT_ERR_NULL_POINTER;
    if ((uintptr_t)vertices % 16 != 0 || (uintptr_t)grad_vertices % 16 != 0) return DIRT_ERR_MISALIGNED;
    if ((uintptr_t)pixels % 4 || (uintptr_t)grad_pixels % 4 || (uintptr_t)grad_background % 4 ||
        (uintptr_t)grad_vertex_colors % 4 || (uintptr_t)faces % 4 || (uintptr_t)face_ids % 4)
        return DIRT_ERR_MISALIGNED;
    rc = check_workspace(workspace, workspace_bytes, B, H, W, C, V, F, face_ids == nullptr);
    if (rc != DIRT_OK) return rc;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const Workspace ws = carve_workspace(workspace, B, H, W, C, V, F);
    const Dims d = make_dims(B, H, W, C, V, F, flags & SHARING_BITS);
    const int32_t* ids = face_ids;
    // the tile coverage flags in the workspace describe `ids` when the raster kernel that produced them ran on this workspace
    const bool flags_valid = !ids || workspace_holds_setup;
    unsigned long long expect_tag = 0;
    if (!ids) {
        // no cached visibility: re-derive it exactly as the forward pass does
        CUDA_TRY(launch_setup_and_bin(vertices, faces, nullptr, ws, d, stream, &launches));
        CUDA_TRY(launch_raster_visibility(vertices, ws.face_ids, nullptr, ws, d, stream, &launches));
        ids = ws.face_ids;
    } else if (!workspace_holds_setup) {
        CUDA_TRY(launch_setup_only(vertices, faces, ws, d, stream, &launches));
    } else {
        // a promise: checked on the device against the tag the setup pass left in the workspace
        expect_tag = workspace_tag(vertices, faces, B, H, W, V, F, d.face_stride == 0);
    }
    CUDA_TRY(launch_backward(vertices, pixels, grad_pixels, ids, grad_background, grad_vertices, grad_vertex_colors, ws, d,
                             groups, flags_valid, flags, expect_tag, stream, &launches));
    t_last_launches = launches;
    return DIRT_OK;
}

extern "C" int dirt_rasterise_backward(const float* vertices, const int32_t* faces, const float* pixels,
                                       const float* grad_pixels, const int32_t* face_ids, float* grad_background,
                                       float* grad_vertices, float* grad_vertex_colors, int B, int H, int W, int C, int V,
                                       int F, const int* channel_groups, int n_groups, int workspace_holds_setup,
                                       void* workspace, size_t workspace_bytes, void* cuda_stream)
{
    return backward_impl(vertices, faces, pixels, grad_pixels, face_ids, grad_background, grad_vertices, grad_vertex_colors, B, H,
                         W, C, V, F, channel_groups, n_groups, workspace_holds_setup, 0, workspace, workspace_bytes, cuda_stream);
}

extern "C" int dirt_rasterise_backward_ex(const float* vertices, const int32_t* faces, const float* pixels,
                                          const float* grad_pixels, const int32_t* face_ids, float* grad_background,
                                          float* grad_vertices, float* grad_vertex_colors, int B, int H, int W, int C, int V,
                                          int F, const int* channel_groups, int n_groups, int workspace_holds_setup, int flags,
                                          void* workspace, size_t workspace_bytes, void* cuda_stream)
{
    return backward_impl(vertices, faces, pixels, grad_pixels, face_ids, grad_background, grad_vertices, grad_vertex_colors, B, H,
                         W, C, V, F, channel_groups, n_groups, workspace_holds_setup, flags, workspace, workspace_bytes, cuda_stream);
}

extern "C" int dirt_workspace_status(const void* workspace, size_t workspace_bytes, int B, int H, int W, int C, int V, int F,
                                     void* cuda_stream)
{
    if (!shape_ok(B, H, W, C, V, F)) return DIRT_ERR_BAD_SHAPE;
    if (B == 0) return DIRT_OK;
    int rc = check_workspace(const_cast<void*>(workspace), workspace_bytes, B, H, W, C, V, F);
    if (rc != DIRT_OK) return rc;
    const Workspace ws = carve_workspace(const_cast<void*>(workspace), B, H, W, C, V, F);
    Header h;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (cudaMemcpyAsync(&h, ws.header, sizeof(h), cudaMemcpyDeviceToHost, stream) != cudaSuccess) return DIRT_ERR_CUDA;
    if (cudaStreamSynchronize(stream) != cudaSuccess) return DIRT_ERR_CUDA;
    return h.error ? DIRT_ERR_STALE_WORKSPACE : DIRT_OK;
}
