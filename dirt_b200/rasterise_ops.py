"""`rasterise` / `rasterise_batch` and their deferred-shading variants on the B200-native library.

Host-side mirror of the reference's dirt/rasterise_ops.py: same function names, argument order,
defaults and error behaviour, with `torch.Tensor` in place of `tf.Tensor` and a
`torch.autograd.Function` in place of `@ops.RegisterGradient('Rasterise')` (rasterise_ops.py:111-129).

Differences that a caller can observe:
* any channel count is rendered in ONE fused pass; the reference's greedy 3/1 channel grouping
  (rasterise_ops.py:86-108) only survives as the `channel_groups` argument of the backward kernel,
  where it changes the result (each group takes its own filter / dilation decision);
* tensors must live on a CUDA device (the reference registers a GPU kernel only,
  csrc/rasterise_egl.cpp:410); there is no CPU fallback.
"""
import ctypes

import torch

from . import _lib


def default_channel_groups(channels):
    """The reference's split of `channels` into op calls: one group if channels is 1 or 3, else greedily
    groups of 3 while at least 3 remain, then groups of 1 (dirt/rasterise_ops.py:80-108)."""
    if channels <= 0:
        raise ValueError('channels must be positive')
    if channels == 1 or channels == 3:
        return [channels]
    groups, begin = [], 0
    while begin < channels:
        width = 3 if begin + 3 <= channels else 1
        groups.append(width)
        begin += width
    return groups


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _workspace(B, H, W, C, V, F, device, face_id_scratch=False):
    """A workspace for one call -> (tensor, its size).  Without `face_id_scratch` it is the smaller size that serves every
    call whose caller holds the face ids (dirt_workspace_bytes_min: no B*H*W*4-byte block for deriving them), which is every
    call this module makes except a backward call without `face_ids`."""
    size = _lib.lib().dirt_workspace_bytes if face_id_scratch else _lib.lib().dirt_workspace_bytes_min
    # the allocation also covers a 3-channel call on the same geometry (its workspace carries padded gradient rows behind
    # the blocks that are laid out independently of C): deferred shading hands the G-buffer pass's workspace to the backward
    # call on the shaded, usually 3-channel, image
    alloc = max(int(size(B, H, W, C, V, F)), int(size(B, H, W, 3, V, F)), 256)
    return torch.empty(alloc, dtype=torch.uint8, device=device), alloc


def _require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError(
                'dirt_b200: rasterise needs CUDA tensors (the Rasterise op has no CPU kernel); got a tensor on %s'
                % t.device)


def _check_shapes(op, background, vertices, vertex_colors, faces, height, width, channels):
    # same conditions and wording as csrc/rasterise_egl.cpp:301-316
    if background.dim() != 4 or background.shape[1] != height or background.shape[2] != width or \
            background.shape[3] != channels:
        raise ValueError('%s expects background_tensor to be 4D, and bgcolor.shape == [None, height, width, channels]' % op)
    if vertices.dim() != 3 or vertices.shape[2] != 4:
        raise ValueError('%s expects vertices to be 3D, and vertices.shape[2] == 4' % op)
    if vertex_colors.dim() != 3 or vertex_colors.shape[1] != vertices.shape[1] or vertex_colors.shape[2] != channels:
        raise ValueError('%s expects vertex_colors to be 3D, and vertex_colors.shape == [None, vertices.shape[1], channels]' % op)
    if faces.dim() != 3 or faces.shape[2] != 3:
        raise ValueError('%s expects faces to be 3D, and faces.shape[2] == 3' % op)
    B = vertices.shape[0]
    if background.shape[0] != B or vertex_colors.shape[0] != B or faces.shape[0] != B:
        raise ValueError('%s expects all arguments to have same leading (batch) dimension' % op)


def rasterise_forward_raw(background, vertices, vertex_colors, faces, want_face_ids=True, return_workspace=False, shared=0):
    """One call of dirt_rasterise_forward_ex on contiguous CUDA tensors. Returns (pixels, face_ids or None)
    [, workspace tensor holding the per-face setup records, reusable by rasterise_backward_raw].
    `shared`: _lib.SHARED_* bits; a shared background / vertex_colors / faces has no batch dimension."""
    B, V, F = vertices.shape[0], vertices.shape[1], faces.shape[-2]
    H, W, C = background.shape[-3:]
    pixels = torch.empty((B, H, W, C), dtype=background.dtype, device=background.device)
    face_ids = torch.empty((B, H, W), dtype=torch.int32, device=background.device) if want_face_ids else None
    ws, nbytes = _workspace(B, H, W, C, V, F, background.device)
    with torch.cuda.device(background.device):
        rc = _lib.lib().dirt_rasterise_forward_ex(_ptr(background), _ptr(vertices), _ptr(vertex_colors), _ptr(faces),
                                                  _ptr(pixels), _ptr(face_ids), B, H, W, C, V, F, _ptr(ws), nbytes,
                                                  _stream_ptr(background.device), shared)
    _lib.check(rc, 'Rasterise')
    if return_workspace:
        ws._dirt_setup_of = _geometry_identity(vertices, faces, H, W)
        return pixels, face_ids, ws
    return pixels, face_ids


def _geometry_identity(vertices, faces, H, W):
    """What the setup records in a workspace were computed from: the tensors' storage AND their version counters
    (an in-place update of the vertices makes the records stale; the C ABI's own tag cannot see that)."""
    return (vertices.data_ptr(), vertices._version, tuple(vertices.shape), faces.data_ptr(), faces._version, tuple(faces.shape), H, W)


def rasterise_backward_raw(vertices, faces, pixels, grad_pixels, face_ids=None, channel_groups=None, setup_workspace=None,
                           shared_geometry=False, want_position=True, want_colour=True, shared=0, want_background=True):
    """One call of dirt_rasterise_backward (the RasteriseGrad op, csrc/rasterise_grad_egl.cpp:33-53).
    `setup_workspace`: the workspace tensor of the forward call on the same (vertices, faces); its setup records are
    reused only if it still describes exactly these tensors (storage, version counters, sizes), otherwise they are
    recomputed.  `shared_geometry`: accumulate the vertex gradients over the batch (DIRT_BWD_SHARED_GEOMETRY):
    grad_vertices [V,4] and grad_vertex_colors [V,C] instead of [B,V,.].  want_position / want_colour = False skip
    the position terms (grad_vertices comes back zero) / the colour terms (grad_vertex_colors zero, grad_background None).
    `shared`: the _lib.SHARED_* bits of the forward call.  A shared background's gradient is [H,W,C], summed over the batch,
    and is computed only when `want_background`; shared colours get a [V,C] gradient, summed over the batch; shared faces
    are [F,3].
    Returns (grad_background, grad_vertices, grad_vertex_colors)."""
    B, H, W, C = pixels.shape
    V, F = vertices.shape[1], faces.shape[-2]
    faces_rank = 2 if shared & _lib.SHARED_FACES else 3
    # wording of csrc/rasterise_grad_egl.cpp:349-377
    if vertices.dim() != 3 or vertices.shape[2] != 4:
        raise ValueError('RasteriseGrad expects vertices to be 3D, and vertices.shape[2] == 4')
    if faces.dim() != faces_rank or faces.shape[-1] != 3:
        raise ValueError('RasteriseGrad expects faces to be %dD, and faces.shape[%d] == 3' % (faces_rank, faces_rank - 1))
    if grad_pixels.shape != pixels.shape:
        raise ValueError('RasteriseGrad expects grad_pixels to be 4D, and grad_pixels.shape == [None, height, width, channels]')
    if (faces_rank == 3 and faces.shape[0] != B) or vertices.shape[0] != B:
        raise ValueError('RasteriseGrad expects all arguments to have same leading (batch) dimension')
    device = pixels.device
    if shared & _lib.SHARED_BACKGROUND:
        grad_background = torch.empty((H, W, C), dtype=torch.float32, device=device) if want_colour and want_background else None
    else:
        grad_background = torch.empty_like(pixels) if want_colour else None
    lead = () if shared_geometry else (B,)
    grad_vertices = torch.empty(lead + (V, 4), dtype=torch.float32, device=device)
    colour_lead = () if shared & _lib.SHARED_COLOURS else lead
    grad_vertex_colors = torch.empty(colour_lead + (V, C), dtype=torch.float32, device=device)
    if channel_groups is None:
        groups_ptr, n_groups = None, 0
    else:
        groups_arr = (ctypes.c_int * len(channel_groups))(*[int(g) for g in channel_groups])
        groups_ptr, n_groups = groups_arr, len(channel_groups)
    need = int(_lib.lib().dirt_workspace_bytes_min(B, H, W, C, V, F))
    reuse = int(setup_workspace is not None and face_ids is not None and setup_workspace.numel() >= need and
                getattr(setup_workspace, '_dirt_setup_of', None) == _geometry_identity(vertices, faces, H, W))
    ws = setup_workspace if reuse else _workspace(B, H, W, C, V, F, device, face_id_scratch=face_ids is None)[0]
    nbytes = int(ws.numel())
    flags = ((_lib.BWD_SHARED_GEOMETRY if shared_geometry else 0) | (0 if want_position else _lib.BWD_SKIP_POSITION) |
             (0 if want_colour else _lib.BWD_SKIP_COLOUR) | shared)
    with torch.cuda.device(device):
        rc = _lib.lib().dirt_rasterise_backward_ex(
            _ptr(vertices), _ptr(faces), _ptr(pixels), _ptr(grad_pixels), _ptr(face_ids),
            _ptr(grad_background), _ptr(grad_vertices), _ptr(grad_vertex_colors),
            B, H, W, C, V, F, groups_ptr, n_groups, reuse, flags, _ptr(ws), nbytes, _stream_ptr(device))
    _lib.check(rc, 'RasteriseGrad')
    return grad_background, grad_vertices, grad_vertex_colors


def workspace_status(workspace, B, H, W, C, V, F):
    """dirt_workspace_status: waits for the stream; raises if a backward call was handed a workspace that did not hold
    the setup records it was promised (csrc/api.cu)."""
    nbytes = int(workspace.numel())
    with torch.cuda.device(workspace.device):
        rc = _lib.lib().dirt_workspace_status(_ptr(workspace), nbytes, B, H, W, C, V, F, _stream_ptr(workspace.device))
    _lib.check(rc, 'RasteriseGrad')


def rasterise_visibility_raw(vertices, faces, height, width, want_gbuffer=True):
    """dirt_rasterise_visibility: (face_ids int32 [B,H,W], gbuffer float32 [B,H,W,4] or None)."""
    B, V, F = vertices.shape[0], vertices.shape[1], faces.shape[1]
    device = vertices.device
    face_ids = torch.empty((B, height, width), dtype=torch.int32, device=device)
    gbuffer = torch.empty((B, height, width, 4), dtype=torch.float32, device=device) if want_gbuffer else None
    ws, nbytes = _workspace(B, height, width, 1, V, F, device)
    with torch.cuda.device(device):
        rc = _lib.lib().dirt_rasterise_visibility(_ptr(vertices), _ptr(faces), _ptr(face_ids), _ptr(gbuffer), B, height,
                                                  width, V, F, _ptr(ws), nbytes, _stream_ptr(device))
    _lib.check(rc, 'RasteriseVisibility')
    return face_ids, gbuffer


class _Rasterise(torch.autograd.Function):
    """The Rasterise op with its registered gradient (dirt/rasterise_ops.py:111-129).  `shared`: _lib.SHARED_* bits of the
    inputs the whole batch shares (0: every input per image)."""

    @staticmethod
    def forward(ctx, background, vertices, vertex_colors, faces, channel_groups, shared=0):
        pixels, face_ids, ws = rasterise_forward_raw(background, vertices, vertex_colors, faces, want_face_ids=True,
                                                     return_workspace=True, shared=shared)
        ctx.save_for_backward(vertices, faces, pixels, face_ids)
        ctx.setup_workspace = ws   # per-face setup records of this (vertices, faces): backward reuses them
        ctx.channel_groups = channel_groups
        ctx.shared = shared
        ctx.mark_non_differentiable(face_ids)
        return pixels, face_ids

    @staticmethod
    def backward(ctx, grad_pixels, _grad_face_ids):
        want_background, want_vertices, want_colours = ctx.needs_input_grad[:3]
        if not (want_background or want_vertices or want_colours):
            return None, None, None, None, None, None
        vertices, faces, pixels, face_ids = ctx.saved_tensors
        grad_pixels = grad_pixels.contiguous().to(torch.float32)
        # a shared background that needs no gradient gets none: no per-image gradient is written and nothing is summed
        grad_background, grad_vertices, grad_vertex_colors = rasterise_backward_raw(
            vertices, faces, pixels, grad_pixels, face_ids, ctx.channel_groups, ctx.setup_workspace,
            want_position=want_vertices, want_colour=want_background or want_colours, shared=ctx.shared,
            want_background=want_background)
        return (grad_background if want_background else None, grad_vertices if want_vertices else None,
                grad_vertex_colors if want_colours else None, None, None, None)  # None: wrt faces


def _as_f32(x, device=None):
    t = torch.as_tensor(x, dtype=torch.float32) if not isinstance(x, torch.Tensor) else x.to(torch.float32)
    if device is not None and t.device != device:
        t = t.to(device)
    return t


def _as_i32(x, device=None):
    t = torch.as_tensor(x, dtype=torch.int32) if not isinstance(x, torch.Tensor) else x.to(torch.int32)
    if device is not None and t.device != device:
        t = t.to(device)
    return t


def _pick_device(*xs):
    # the device of the first CUDA tensor; host inputs (lists, numpy, CPU tensors) go to the current CUDA device,
    # as TensorFlow would place the GPU-only op there.  None (-> an error downstream) when there is no GPU.
    for x in xs:
        if isinstance(x, torch.Tensor) and x.is_cuda:
            return x.device
    if torch.cuda.is_available():
        return torch.device('cuda', torch.cuda.current_device())
    return None


def rasterise(background, vertices, vertex_colors, faces, height=None, width=None, channels=None, name=None):
    """Rasterises the given `vertices` and `faces` over `background` (dirt/rasterise_ops.py:13-48).

    Args:
        background: float32 tensor [height, width, channels], the image to render over
        vertices: float32 tensor [vertex count, 4] of clip-space vertex positions
        vertex_colors: float32 tensor [vertex count, channels]; interpolated perspective-correctly
        faces: int32 tensor [face count, 3] of vertex indices
        height, width, channels: optional ints; default to the shape of `background`
        name: accepted for signature compatibility, ignored

    Returns:
        float32 tensor [height, width, channels]
    """
    device = _pick_device(background, vertices, vertex_colors, faces)
    background = _as_f32(background, device)
    vertices = _as_f32(vertices, device)
    vertex_colors = _as_f32(vertex_colors, device)
    faces = _as_i32(faces, device)
    return rasterise_batch(background[None], vertices[None], vertex_colors[None], faces[None], height, width, channels, name)[0]


def rasterise_batch(background, vertices, vertex_colors, faces, height=None, width=None, channels=None, name=None):
    """Rasterises a batch of meshes with the same numbers of vertices and faces (dirt/rasterise_ops.py:51-108).

    As `rasterise`, with a leading batch dimension on every argument.
    """
    device = _pick_device(background, vertices, vertex_colors, faces)
    background = _as_f32(background, device)
    vertices = _as_f32(vertices, device)
    vertex_colors = _as_f32(vertex_colors, device)
    faces = _as_i32(faces, device)
    if background.dim() != 4:
        raise ValueError('Rasterise expects background_tensor to be 4D, and bgcolor.shape == [None, height, width, channels]')
    if height is None:
        height = int(background.shape[1])
    if width is None:
        width = int(background.shape[2])
    if channels is None:
        channels = int(background.shape[3])
    if not (channels > 0):
        raise ValueError('channels must be positive')  # `assert channels > 0`, rasterise_ops.py:87
    if not (width > 0 and height > 0):
        raise ValueError('width and height must be positive')  # csrc/hwc.h:28
    _check_shapes('Rasterise', background, vertices, vertex_colors, faces, height, width, channels)
    _require_cuda(background, vertices, vertex_colors, faces)
    groups = default_channel_groups(channels)
    pixels, _ = _Rasterise.apply(background.contiguous(), vertices.contiguous(), vertex_colors.contiguous(),
                                 faces.contiguous(), groups)
    return pixels


def rasterise_batch_shared(background, vertices, vertex_colors, faces, height=None, width=None, channels=None, name=None):
    """`rasterise_batch` for one mesh in B poses: only `vertices` [B,V,4] must carry the batch dimension.

    `background` is [B,H,W,C] or [H,W,C], `vertex_colors` [B,V,C] or [V,C], `faces` [B,F,3] or [F,3]: the rank of each
    decides whether it is per image or shared by the whole batch.  The pixels equal `rasterise_batch` called with the
    shared arguments expanded to B, without B copies of them; the gradient of a shared argument has that argument's own
    shape and is the sum of the per-image gradients over the batch (a shared background's gradient is only computed when
    the background requires grad).
    """
    device = _pick_device(background, vertices, vertex_colors, faces)
    background = _as_f32(background, device)
    vertices = _as_f32(vertices, device)
    vertex_colors = _as_f32(vertex_colors, device)
    faces = _as_i32(faces, device)
    if vertices.dim() != 3 or vertices.shape[2] != 4:
        raise ValueError('Rasterise expects vertices to be 3D, and vertices.shape[2] == 4')
    if background.dim() not in (3, 4):
        raise ValueError('Rasterise expects background_tensor to be 4D, and bgcolor.shape == [None, height, width, channels]')
    B = int(vertices.shape[0])
    shared = ((_lib.SHARED_BACKGROUND if background.dim() == 3 else 0) | (_lib.SHARED_COLOURS if vertex_colors.dim() == 2 else 0) |
              (_lib.SHARED_FACES if faces.dim() == 2 else 0))
    if height is None:
        height = int(background.shape[-3])
    if width is None:
        width = int(background.shape[-2])
    if channels is None:
        channels = int(background.shape[-1])
    if not (channels > 0):
        raise ValueError('channels must be positive')
    if not (width > 0 and height > 0):
        raise ValueError('width and height must be positive')
    # the checks (and messages) of rasterise_batch on batch-dimensioned views of the shared arguments (no copies)
    batched = lambda t, bit: t.expand((B,) + tuple(t.shape)) if shared & bit else t
    _check_shapes('Rasterise', batched(background, _lib.SHARED_BACKGROUND), vertices, batched(vertex_colors, _lib.SHARED_COLOURS),
                  batched(faces, _lib.SHARED_FACES), height, width, channels)
    _require_cuda(background, vertices, vertex_colors, faces)
    groups = default_channel_groups(channels)
    pixels, _ = _Rasterise.apply(background.contiguous(), vertices.contiguous(), vertex_colors.contiguous(), faces.contiguous(),
                                 groups, shared)
    return pixels


def _rasterise_grad_multichannel(vertices, faces, pixels, d_loss_by_pixels, single_or_batch, face_ids=None,
                                 setup_workspace=None, want_position=True, want_colour=True):
    """dirt/rasterise_ops.py:132-177: RasteriseGrad over the greedy channel groups of `pixels`, summing
    grad_vertices over groups and concatenating the others -- here one fused backward call (no slicing, no copies).
    Deferred shading uses only one half of each of its two calls (:206-237): want_position / want_colour = False
    skip the other half inside the kernel."""
    assert single_or_batch in ['single', 'batch']
    if single_or_batch == 'single':
        vertices, faces, pixels, d_loss_by_pixels = vertices[None], faces[None], pixels[None], d_loss_by_pixels[None]
        if face_ids is not None:
            face_ids = face_ids[None]
    assert pixels.dim() == 4
    groups = default_channel_groups(int(pixels.shape[3]))
    grad_background, grad_vertices, grad_vertex_colors = rasterise_backward_raw(
        vertices.contiguous(), faces.contiguous(), pixels.contiguous().to(torch.float32),
        d_loss_by_pixels.contiguous().to(torch.float32), face_ids, groups, setup_workspace,
        want_position=want_position, want_colour=want_colour)
    if single_or_batch == 'single':
        return {'grad_vertices': grad_vertices[0], 'grad_vertex_colors': grad_vertex_colors[0],
                'grad_background': None if grad_background is None else grad_background[0]}
    return {'grad_vertices': grad_vertices, 'grad_vertex_colors': grad_vertex_colors, 'grad_background': grad_background}


class _SetupHolder(object):
    """Carries the forward call's workspace (per-face setup records, tile coverage flags) from the G-buffer node to the
    vertex-gradient node of one deferred call without making it an autograd input."""

    def __init__(self, workspace):
        self.workspace = workspace


class _RasteriseAttributes(torch.autograd.Function):
    """G-buffer pass of deferred shading: gradients flow to attributes and background only
    (the second RasteriseGrad call of dirt/rasterise_ops.py:233-237)."""

    @staticmethod
    def forward(ctx, background, vertices, attributes, faces, holder):
        gbuffer, face_ids, ws = rasterise_forward_raw(background, vertices, attributes, faces, want_face_ids=True,
                                                      return_workspace=True)
        holder.workspace = ws
        ctx.holder = holder
        ctx.save_for_backward(vertices, faces, gbuffer, face_ids)
        ctx.mark_non_differentiable(face_ids)
        return gbuffer, face_ids

    @staticmethod
    def backward(ctx, d_loss_by_gbuffer, _unused):
        if not (ctx.needs_input_grad[0] or ctx.needs_input_grad[2]):
            return None, None, None, None, None
        vertices, faces, gbuffer, face_ids = ctx.saved_tensors
        # the vertex gradient of THIS call (filtering the G-buffer) is the one the reference discards (:233-237)
        grads = _rasterise_grad_multichannel(vertices, faces, gbuffer, d_loss_by_gbuffer, 'batch', face_ids,
                                             ctx.holder.workspace, want_position=False)
        return grads['grad_background'], None, grads['grad_vertex_colors'], None, None


class _InjectVertexGradient(torch.autograd.Function):
    """Identity on the shaded pixels whose backward adds the vertex gradient obtained by filtering the
    SHADED image (the first RasteriseGrad call of dirt/rasterise_ops.py:206-210)."""

    @staticmethod
    def forward(ctx, pixels, vertices, faces, face_ids, holder):
        ctx.holder = holder
        ctx.save_for_backward(pixels.detach(), vertices, faces, face_ids)
        return pixels.view_as(pixels)

    @staticmethod
    def backward(ctx, d_loss_by_pixels):
        if not ctx.needs_input_grad[1]:
            return d_loss_by_pixels, None, None, None, None
        pixels, vertices, faces, face_ids = ctx.saved_tensors
        d_loss_by_vertices = _rasterise_grad_multichannel(vertices, faces, pixels, d_loss_by_pixels, 'batch', face_ids,
                                                          ctx.holder.workspace, want_colour=False)['grad_vertices']
        return d_loss_by_pixels, d_loss_by_vertices, None, None, None


def _rasterise_deferred_internal(background, vertices, attributes, faces, shader_fn, shader_additional_inputs, single_or_batch, name):
    # dirt/rasterise_ops.py:180-257.  The reference wraps everything in one tf.custom_gradient; here the same
    # three gradient paths are expressed as two autograd nodes around an ordinary call of shader_fn, so tensors
    # and parameters that shader_fn uses receive their gradients from plain autograd.
    assert single_or_batch in ['single', 'batch']
    device = _pick_device(background, vertices, attributes, faces)
    background = _as_f32(background, device)
    vertices = _as_f32(vertices, device)
    attributes = _as_f32(attributes, device)
    faces = _as_i32(faces, device)
    if single_or_batch == 'single':
        background, vertices, attributes, faces = background[None], vertices[None], attributes[None], faces[None]
    if background.dim() != 4:
        raise ValueError('Rasterise expects background_tensor to be 4D, and bgcolor.shape == [None, height, width, channels]')
    _check_shapes('Rasterise', background, vertices, attributes, faces, int(background.shape[1]), int(background.shape[2]),
                  int(background.shape[3]))
    _require_cuda(background, vertices, attributes, faces)
    background, vertices, attributes, faces = background.contiguous(), vertices.contiguous(), attributes.contiguous(), faces.contiguous()
    holder = _SetupHolder(None)
    gbuffer, face_ids = _RasteriseAttributes.apply(background, vertices, attributes, faces, holder)
    if single_or_batch == 'single':
        pixels = shader_fn(gbuffer[0], *shader_additional_inputs)[None]
    else:
        pixels = shader_fn(gbuffer, *shader_additional_inputs)
    if pixels.dim() != 4 or pixels.shape[:3] != gbuffer.shape[:3]:
        raise ValueError('shader_fn must return pixels of shape [height, width, channels] per image')
    pixels = _InjectVertexGradient.apply(pixels.to(torch.float32), vertices, faces, face_ids, holder)
    return pixels[0] if single_or_batch == 'single' else pixels


def rasterise_deferred(background_attributes, vertices, vertex_attributes, faces, shader_fn, shader_additional_inputs=[], name=None):
    """Rasterises a G-buffer of vertex attributes and shades it with `shader_fn` (dirt/rasterise_ops.py:260-310).

    Equivalent to `shader_fn(rasterise(background_attributes, vertices, vertex_attributes, faces), *shader_additional_inputs)`
    in the forward direction; the gradient w.r.t. `vertices` is computed from the SHADED pixels, the gradients
    w.r.t. attributes / background from the G-buffer through `shader_fn`.
    """
    return _rasterise_deferred_internal(background_attributes, vertices, vertex_attributes, faces, shader_fn,
                                        list(shader_additional_inputs), 'single', name)


def rasterise_batch_deferred(background_attributes, vertices, vertex_attributes, faces, shader_fn, shader_additional_inputs=[], name=None):
    """Batched `rasterise_deferred` (dirt/rasterise_ops.py:313-333)."""
    return _rasterise_deferred_internal(background_attributes, vertices, vertex_attributes, faces, shader_fn,
                                        list(shader_additional_inputs), 'batch', name)
