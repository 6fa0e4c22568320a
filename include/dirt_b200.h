/*
 * dirt_b200.h -- C ABI of libdirt_b200.so, the sm_100a replacement for the
 * `Rasterise` / `RasteriseGrad` custom ops of pmh47/dirt.
 *
 * Every entry point takes plain device pointers and sizes (no torch / TF types),
 * enqueues all its work on the CUDA stream it is given, never synchronises the
 * host, never allocates device memory and keeps no global state.  The caller
 * owns every buffer, including the workspace.
 *
 * Reference interfaces replaced (paths relative to the reference checkout):
 *   dirt_rasterise_forward   <- REGISTER_OP("Rasterise") + RasteriseOpGpu::Compute
 *                               csrc/rasterise_egl.cpp:32-51, 276-408
 *   dirt_rasterise_backward  <- REGISTER_OP("RasteriseGrad") + RasteriseGradOpGpu::Compute
 *                               csrc/rasterise_grad_egl.cpp:33-53, 324-485 and the kernel
 *                               assemble_grads, csrc/rasterise_grad_egl.cu:93-236
 *   dirt_rasterise_visibility<- the backward G-buffer (barycentrics, clip-w, indices) that
 *                               the reference renders with GL, csrc/shaders.cpp:45-79,
 *                               csrc/rasterise_grad_egl.cpp:432-456 (debug / parity tests)
 *   height/width/channels    <- the HWC op attributes, csrc/hwc.h:7-30
 *
 * Layouts (all row-major, channels last, row 0 = top of the image = clip-space y=+1,
 * csrc/rasterise_egl.cu:23,80):
 *   background, pixels, grad_pixels, grad_background : float32 [B, H, W, C]
 *   vertices, grad_vertices                          : float32 [B, V, 4]   (clip space x,y,z,w)
 *   vertex_colors, grad_vertex_colors                : float32 [B, V, C]
 *   faces                                            : int32   [B, F, 3]
 *   face_ids                                         : int32   [B, H, W]   (-1 = background)
 * except for an input the whole batch shares (DIRT_SHARED_* below), which has no batch dimension.
 *   gbuffer                                          : float32 [B, H, W, 4] (bary0, bary1, bary2, clip_w;
 *                                                      (-1,-1,-1,+inf) where uncovered)
 */
#ifndef DIRT_B200_H
#define DIRT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Error codes: 0 on success, negative on failure.  Nothing aborts the process
 * (the reference LOG(FATAL)s on every CUDA/GL error, csrc/rasterise_egl.cpp:82-86). */
enum {
    DIRT_OK = 0,
    DIRT_ERR_BAD_SHAPE = -1,        /* B,H,W,C,V,F out of range (csrc/hwc.h:27-28; rasterise_egl.cpp:301-316) */
    DIRT_ERR_NULL_POINTER = -2,
    DIRT_ERR_WORKSPACE_TOO_SMALL = -3,
    DIRT_ERR_BAD_CHANNEL_GROUPS = -4, /* groups must be 1 or 3 wide and sum to C (rasterise_ops.py:80-108) */
    DIRT_ERR_TOO_MANY_VERTICES = -5,  /* V > 2^24, csrc/rasterise_grad_egl.cpp:399-405 */
    DIRT_ERR_CUDA = -6,               /* a CUDA runtime call or kernel launch failed */
    DIRT_ERR_MISALIGNED = -7,         /* a pointer is not aligned as required (workspace: 256 B, tensors: 4 B) */
    DIRT_ERR_STALE_WORKSPACE = -8     /* dirt_workspace_status: a backward call was promised setup records that were not there */
};

/* Human-readable text for an error code (static storage, never NULL). */
const char* dirt_error_string(int code);

/* Library / ABI version, bumped whenever a signature changes. */
int dirt_abi_version(void);

/* Bytes of device workspace that forward / backward / visibility need for these sizes.
 * Deterministic function of the sizes only (no data dependence, no host sync):
 * triangle records + bounded per-tile reference lists + per-tile counters. */
size_t dirt_workspace_bytes(int B, int H, int W, int C, int V, int F);

/* The same without the B*H*W*4-byte block that only a backward call WITHOUT face ids uses (it derives them there):
 * enough for forward, visibility, and every backward call that is handed the forward's face ids. */
size_t dirt_workspace_bytes_min(int B, int H, int W, int C, int V, int F);

/* Forward: pixels = rasterise(background, vertices, vertex_colors, faces).
 * Handles any C >= 1 in one pass (the reference runs one op per channel group of 3 or 1,
 * rasterise_ops.py:86-108; the forward result does not depend on the grouping).
 * face_ids_out may be NULL; when given it receives the per-pixel visible face index,
 * which dirt_rasterise_backward accepts back to skip re-deriving visibility. */
int dirt_rasterise_forward(const float* background, const float* vertices,
                           const float* vertex_colors, const int32_t* faces,
                           float* pixels, int32_t* face_ids_out,
                           int B, int H, int W, int C, int V, int F,
                           void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Inputs the whole batch shares (one mesh in B poses): a shared tensor has no batch dimension.  The values do not collide
 * with the DIRT_BWD_* bits, so one flags word serves a forward and its backward call.
 *  DIRT_SHARED_BACKGROUND  background is [H,W,C]; in a backward call grad_background is [H,W,C], the sum over the batch of
 *                          the per-image gradients, or NULL when it is not wanted (then nothing is computed for it).
 *  DIRT_SHARED_COLOURS     vertex_colors is [V,C]; in a backward call grad_vertex_colors is [V,C], summed over the batch
 *                          (grad_vertices stays [B,V,4] unless DIRT_BWD_SHARED_GEOMETRY is also set).
 *  DIRT_SHARED_FACES       faces is [F,3].  The setup records stay per image (the vertices are), and the workspace tag
 *                          includes the face layout, so a workspace_holds_setup promise across layouts is caught. */
enum {
    DIRT_SHARED_BACKGROUND = 8,
    DIRT_SHARED_COLOURS = 16,
    DIRT_SHARED_FACES = 32
};

/* dirt_rasterise_forward with a flags word (flags = 0 is dirt_rasterise_forward itself); only the DIRT_SHARED_* bits are
 * accepted. */
int dirt_rasterise_forward_ex(const float* background, const float* vertices,
                              const float* vertex_colors, const int32_t* faces,
                              float* pixels, int32_t* face_ids_out,
                              int B, int H, int W, int C, int V, int F,
                              void* workspace, size_t workspace_bytes, void* cuda_stream, int flags);

/* Backward: the RasteriseGrad op.  `pixels` is an input (deferred shading passes shaded
 * pixels, rasterise_ops.py:206-210).  channel_groups (host pointer) lists the widths of the
 * reference's channel groups, e.g. {3,1} for C=4; each group takes its own Scharr / dilation
 * decision and grad_vertices is summed over groups (rasterise_ops.py:163).  NULL/0 means the
 * reference's own greedy split of C.
 * face_ids may be NULL: visibility is then re-derived from (vertices, faces) inside the call.
 * workspace_holds_setup != 0 promises that `workspace` is the buffer a preceding dirt_rasterise_forward /
 * dirt_rasterise_visibility call on the SAME (vertices, faces, H, W) filled and that nothing has written to it
 * since: the per-face setup records are then reused instead of recomputed (only meaningful with face_ids).
 * The promise is checked on the device: the setup pass leaves a tag (hash of the vertices / faces pointers and the
 * sizes) in the workspace; a backward call that finds another tag sets an error flag in the workspace (reported by
 * dirt_workspace_status) and writes NaN into grad_vertices[0] instead of returning plausible numbers.  What the tag
 * cannot see is an in-place change of the vertex VALUES between the two calls; the Python layer covers that with
 * the tensors' version counters.
 * grad_vertices / grad_vertex_colors are zeroed by the library before accumulation;
 * grad_background is written exactly once per pixel. */
int dirt_rasterise_backward(const float* vertices, const int32_t* faces,
                            const float* pixels, const float* grad_pixels,
                            const int32_t* face_ids,
                            float* grad_background, float* grad_vertices, float* grad_vertex_colors,
                            int B, int H, int W, int C, int V, int F,
                            const int* channel_groups, int n_groups, int workspace_holds_setup,
                            void* workspace, size_t workspace_bytes, void* cuda_stream);

/* dirt_rasterise_backward with options (flags = 0 is dirt_rasterise_backward itself):
 *  DIRT_BWD_SHARED_GEOMETRY  the vertex gradients are ACCUMULATED OVER THE BATCH: grad_vertices is [V,4] and
 *      grad_vertex_colors [V,C], sum_b of the per-item results -- the gradient of geometry / colours that are parameters
 *      shared by the batch (SURVEY 8e; the reference leaves that sum to TensorFlow's broadcast gradient).  Saves the
 *      [B,V,.] buffers, their memsets and the reduction pass; it is the buffer a multi-GPU job all-reduces.
 *  DIRT_BWD_SKIP_POSITION    grad_vertices is not computed (left zero): no Scharr filter, no dilation, `pixels` is not read.
 *  DIRT_BWD_SKIP_COLOUR      grad_vertex_colors is not computed (left zero) and grad_background is not written.
 *  The two SKIP flags serve deferred shading, whose gradient is two RasteriseGrad calls of which only one output each
 *  is used (dirt/rasterise_ops.py:206-237: vertices from the shaded pixels, attributes / background from the G-buffer).
 *  The DIRT_SHARED_* bits of dirt_rasterise_forward_ex are accepted as well. */
enum {
    DIRT_BWD_SHARED_GEOMETRY = 1,
    DIRT_BWD_SKIP_POSITION = 2,
    DIRT_BWD_SKIP_COLOUR = 4
};
int dirt_rasterise_backward_ex(const float* vertices, const int32_t* faces,
                               const float* pixels, const float* grad_pixels,
                               const int32_t* face_ids,
                               float* grad_background, float* grad_vertices, float* grad_vertex_colors,
                               int B, int H, int W, int C, int V, int F,
                               const int* channel_groups, int n_groups, int workspace_holds_setup, int flags,
                               void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Waits for the stream and reports whether a backward call found the workspace not to hold the setup records it was
 * promised (DIRT_ERR_STALE_WORKSPACE), else DIRT_OK.  The only entry point that synchronises the host. */
int dirt_workspace_status(const void* workspace, size_t workspace_bytes,
                          int B, int H, int W, int C, int V, int F, void* cuda_stream);

/* Debug / parity: the visibility G-buffer alone (either output may be NULL). */
int dirt_rasterise_visibility(const float* vertices, const int32_t* faces,
                              int32_t* face_ids, float* gbuffer,
                              int B, int H, int W, int V, int F,
                              void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Multi-GPU (one process per GPU, one node): sum over the ranks of the batch-shared vertex gradient -- the [V,4 | V,C] buffer
 * a DIRT_BWD_SHARED_GEOMETRY call fills -- over peer memory, as ONE kernel of `world` CTAs per rank and step: every rank
 * pushes its buffer into its slot of every peer's exchange area (stores through the NVLink peer mapping), releases a flag
 * there, waits for the `world` flags of its own area and adds its slots in rank order into `out` (bit-identical on all
 * ranks).  The reference has no counterpart (no multi-GPU path: tests/multi_gpu_test.py); TensorFlow users would all-reduce
 * the op's gradient outside it.
 *   dirt_peer_exchange_bytes  size of one rank's exchange area for buffers of `count` floats (two step parities x world slots).
 *   peer_slots[p] / peer_flags[p]  HOST arrays of `world` DEVICE pointers: rank p's exchange area / its flag words
 *                                  (2*world uint32, zero before the first call) as mapped into THIS process (own rank
 *                                  included).  The mapping itself (cudaIpc / VMM handles) is the caller's plumbing.
 *   sequence  1, 2, 3, ... : the same value on every rank for the same step; consecutive calls on one stream.
 *   local != out, both 16-byte aligned, count a multiple of 4.  Only enqueues work on cuda_stream. */
size_t dirt_peer_exchange_bytes(int world, long long count);
int dirt_peer_exchange(const float* local, float* out, void* const* peer_slots, void* const* peer_flags,
                       int world, int rank, long long count, unsigned int sequence, void* cuda_stream);

/* Number of kernels the last call on this thread launched (bench.py's gpu_launches). */
int dirt_last_launch_count(void);

/* Profiling hooks (replace the reference's compile-time TIME_SECTIONS stamps,
 * csrc/rasterise_egl.cpp:284-286,398-405): bracket ONE kernel of subsequent calls on this thread with
 * CUDA events recorded on the call's own stream.  which: 0 = off, 1 = forward raster kernel,
 * 2 = backward (assemble-grads) kernel.  dirt_kernel_timer_elapsed_ms() waits for the last bracketed
 * launch and returns its duration in milliseconds (negative if nothing was timed).  which = 3: the kernel that sums a
 * shared background's gradient over the batch (DIRT_SHARED_BACKGROUND). */
int dirt_kernel_timer_enable(int which);
float dirt_kernel_timer_elapsed_ms(void);

#ifdef __cplusplus
}
#endif
#endif /* DIRT_B200_H */
