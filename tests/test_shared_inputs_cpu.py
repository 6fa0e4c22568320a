"""CPU: argument validation of rasterise_batch_shared and of the C ABI's sharing bits (no kernel is launched)."""
import ctypes

import pytest
import torch


def test_rasterise_batch_shared_validates_arguments():
    import dirt_b200 as dirt
    B, H, W, C, V, F = 2, 8, 8, 3, 5, 4
    verts = torch.zeros(B, V, 4)
    bg, bg1 = torch.zeros(B, H, W, C), torch.zeros(H, W, C)
    cols, cols1 = torch.zeros(B, V, C), torch.zeros(V, C)
    faces, faces1 = torch.zeros(B, F, 3, dtype=torch.int32), torch.zeros(F, 3, dtype=torch.int32)
    # ranks
    with pytest.raises(ValueError, match='vertices to be 3D'):
        dirt.rasterise_batch_shared(bg1, torch.zeros(V, 4), cols1, faces1)
    with pytest.raises(ValueError, match='background_tensor to be 4D'):
        dirt.rasterise_batch_shared(torch.zeros(H, W), verts, cols1, faces1)
    with pytest.raises(ValueError, match='background_tensor to be 4D'):
        dirt.rasterise_batch_shared(torch.zeros(1, B, H, W, C), verts, cols1, faces1)
    with pytest.raises(ValueError, match='vertex_colors to be 3D'):
        dirt.rasterise_batch_shared(bg1, verts, torch.zeros(V), faces1)
    with pytest.raises(ValueError, match='faces to be 3D'):
        dirt.rasterise_batch_shared(bg1, verts, cols1, torch.zeros(F, dtype=torch.int32))
    # shapes inside a rank
    with pytest.raises(ValueError, match='vertex_colors to be 3D'):
        dirt.rasterise_batch_shared(bg1, verts, torch.zeros(V + 1, C), faces1)
    with pytest.raises(ValueError, match='vertex_colors to be 3D'):
        dirt.rasterise_batch_shared(bg1, verts, torch.zeros(V, C + 1), faces1)
    with pytest.raises(ValueError, match='faces to be 3D'):
        dirt.rasterise_batch_shared(bg1, verts, cols1, torch.zeros(F, 4, dtype=torch.int32))
    with pytest.raises(ValueError, match='background_tensor to be 4D'):
        dirt.rasterise_batch_shared(bg1, verts, cols1, faces1, height=H + 1)
    # a batched argument whose leading dimension is not B
    for args in ((bg[:1], verts, cols1, faces1), (bg1, verts, cols[:1], faces1), (bg1, verts, cols1, faces[:1]),
                 (torch.zeros(B + 1, H, W, C), verts, cols, faces)):
        with pytest.raises(ValueError, match='same leading'):
            dirt.rasterise_batch_shared(*args)
    # rasterise_batch keeps the reference's contract: a 3-D background is an error there
    with pytest.raises(ValueError, match='background_tensor to be 4D'):
        dirt.rasterise_batch(bg1, verts, cols, faces)
    if not torch.cuda.is_available():
        # valid arguments reach the device check: there is no CPU kernel
        for args in ((bg1, verts, cols1, faces1), (bg, verts, cols1, faces), (bg1, verts, cols, faces1)):
            with pytest.raises(RuntimeError, match='CUDA'):
                dirt.rasterise_batch_shared(*args)


def test_forward_ex_accepts_only_the_sharing_bits():
    from dirt_b200 import _lib
    L = _lib.lib()
    null = ctypes.c_void_p(0)
    p = lambda a: ctypes.c_void_p(a)
    ws = L.dirt_workspace_bytes_min(2, 8, 8, 4, 4, 2)

    def fwd(flags, B=2, bg=p(4096), verts=p(4096), ws_ptr=p(4096), nbytes=ws):
        return L.dirt_rasterise_forward_ex(bg, verts, p(4096), p(4096), p(4096), null, B, 8, 8, 4, 4, 2, ws_ptr, nbytes, null, flags)

    for bad in (_lib.BWD_SHARED_GEOMETRY, _lib.BWD_SKIP_POSITION, _lib.BWD_SKIP_COLOUR, 64, 8 | 64, 1 << 20):
        assert fwd(bad) == _lib.ERR_BAD_SHAPE, bad
        assert fwd(bad, B=0) == _lib.ERR_BAD_SHAPE, bad
    for ok in (0, 8, 16, 32, 8 | 16 | 32):
        assert fwd(ok, B=0) == 0, ok   # an empty batch is a no-op
        # the pointer checks still run (and fail before anything is launched)
        assert fwd(ok, bg=null) == _lib.ERR_NULL_POINTER
        assert fwd(ok, verts=p(4100)) == _lib.ERR_MISALIGNED
        assert fwd(ok, ws_ptr=p(4096 + 128)) == _lib.ERR_MISALIGNED
        assert fwd(ok, nbytes=ws - 1) == _lib.ERR_WORKSPACE_TOO_SMALL
    # the plain entry point is forward_ex(..., 0)
    assert L.dirt_rasterise_forward(null, null, null, null, null, null, 1, 8, 8, 3, 4, 2, null, 0, null) == _lib.ERR_NULL_POINTER
    assert L.dirt_rasterise_forward_ex(null, null, null, null, null, null, 1, 8, 8, 3, 4, 2, null, 0, null, 0) == _lib.ERR_NULL_POINTER


def test_backward_ex_accepts_the_sharing_bits():
    from dirt_b200 import _lib
    L = _lib.lib()
    null = ctypes.c_void_p(0)
    p = lambda a: ctypes.c_void_p(a)
    small = L.dirt_workspace_bytes_min(1, 8, 8, 3, 4, 2)

    def bwd(flags, grad_background=p(4096), nbytes=small - 1):
        # a too small workspace is the first thing a well-formed call is refused for (nothing is dereferenced)
        return L.dirt_rasterise_backward_ex(p(4096), p(4096), p(4096), p(4096), p(4096), grad_background, p(4096), p(4096),
                                            1, 8, 8, 3, 4, 2, None, 0, 0, flags, p(4096), nbytes, null)

    for ok in (8, 16, 32, 8 | 16 | 32, 8 | _lib.BWD_SHARED_GEOMETRY):
        assert bwd(ok) == _lib.ERR_WORKSPACE_TOO_SMALL, ok
    for bad in (64, 64 | 8, 128):
        assert bwd(bad) == _lib.ERR_BAD_SHAPE, bad
    # grad_background may be NULL for a shared background (not wanted), not for a per-image one
    assert bwd(_lib.SHARED_BACKGROUND, grad_background=null) == _lib.ERR_WORKSPACE_TOO_SMALL
    assert bwd(0, grad_background=null) == _lib.ERR_NULL_POINTER
    assert bwd(_lib.SHARED_COLOURS | _lib.SHARED_FACES, grad_background=null) == _lib.ERR_NULL_POINTER


def test_kernel_timer_names_the_background_gradient_kernel():
    from dirt_b200 import _lib
    L = _lib.lib()
    assert L.dirt_kernel_timer_enable(4) == _lib.ERR_BAD_SHAPE
    if not torch.cuda.is_available():
        return   # enabling a timer creates CUDA events
    assert L.dirt_kernel_timer_enable(3) == 0
    assert L.dirt_kernel_timer_enable(0) == 0
