"""ctypes wrapper around oracle/_ref/libdirt_ref_grad.so: the REFERENCE'S OWN gradient kernel.

TEST INFRASTRUCTURE ONLY.  oracle/Makefile (target `ref`) compiles /root/reference/csrc/rasterise_grad_egl.cu
UNMODIFIED, against the stand-in TensorFlow headers in oracle/ref_shim/, into oracle/_ref/ (git-ignored; it travels
to the GPU box with the snapshot).  It needs a GPU to run: `assemble_grads` is CUDA.  What it pins: every gradient
value and every dilation decision of csrc/rasterise_grad_egl.cu:93-236, given a G-buffer.  The G-buffer itself (what
the OpenGL driver renders in the reference) is an input -- tests feed it the CPU oracle's.

Only tests/, tests/golden/make_ref_golden.py and __graft_entry__.build() may use this module.
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, '_ref', 'libdirt_ref_grad.so')
REFERENCE_SOURCE = '/root/reference/csrc/rasterise_grad_egl.cu'
_lib = None


def can_build():
    return os.path.exists(REFERENCE_SOURCE)


def build(force=False):
    """make -C oracle ref (only where /root/reference exists, i.e. in the build container)."""
    if not can_build():
        raise RuntimeError('the reference checkout is not present; oracle/_ref can only be built in the build container')
    if force and os.path.exists(_SO):
        os.remove(_SO)
    proc = subprocess.run(['make', '-C', _HERE, 'ref'], capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError('building oracle/_ref failed:\n' + proc.stdout + proc.stderr)
    return _SO


def available():
    return os.path.exists(_SO)


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError('%s is missing (build it with `make -C oracle ref` where /root/reference exists)' % _SO)
        _lib = ctypes.CDLL(_SO)
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def fingerprint(*arrays):
    """sha256 over the dtype, shape and bytes of each array.  Golden data records with it, bit for bit, inputs and outputs
    of a reference-kernel run that are too large to store (tests/golden/ref_live_scenes.npz)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(('%s%s' % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def vertex_ids_image(faces, face_ids):
    """[B,H,W,3] int32: the three vertex indices of each pixel's visible face, -1 where uncovered
    (what the reference's backward fragment shader writes, csrc/shaders.cpp:62-76)."""
    faces = np.asarray(faces, np.int32)
    face_ids = np.asarray(face_ids, np.int32)
    out = np.full(face_ids.shape + (3,), -1, np.int32)
    for b in range(face_ids.shape[0]):
        covered = face_ids[b] >= 0
        out[b][covered] = faces[b][face_ids[b][covered]]
    return out


def assemble_grads(gbuffer, vertex_ids, pixels, grad_pixels, vertices, with_debug=False):
    """ONE native RasteriseGrad call (C = 1 or 3) of the reference kernel.
    -> grad_background [B,H,W,C], grad_vertices [B,V,4], grad_vertex_colors [B,V,C] (, debug_thingy [B,H,W,3])."""
    gbuffer, pixels, grad_pixels, vertices = _f32(gbuffer), _f32(pixels), _f32(grad_pixels), _f32(vertices)
    vertex_ids = np.ascontiguousarray(vertex_ids, np.int32)
    B, H, W, C = pixels.shape
    V = vertices.shape[1]
    assert C in (1, 3) and gbuffer.shape == (B, H, W, 4) and vertex_ids.shape == (B, H, W, 3)
    assert grad_pixels.shape == pixels.shape and vertices.shape == (B, V, 4)
    gv = np.empty((B, V, 4), np.float32)
    gc = np.empty((B, V, C), np.float32)
    gb = np.empty((B, H, W, C), np.float32)
    dbg = np.empty((B, H, W, 3), np.float32) if with_debug else None
    rc = lib().dirt_ref_assemble_grads(_ptr(gbuffer), _ptr(vertex_ids), _ptr(pixels), _ptr(grad_pixels), _ptr(vertices),
                                       _ptr(gv), _ptr(gc), _ptr(gb), _ptr(dbg) if with_debug else None,
                                       B, H, W, C, V)
    if rc != 0:
        raise RuntimeError('dirt_ref_assemble_grads failed: %d' % rc)
    return (gb, gv, gc, dbg) if with_debug else (gb, gv, gc)


def backward(vertices, faces, pixels, grad_pixels, gbuffer, face_ids, channel_groups=None):
    """The Python-level gradient of the reference for any channel count: one native call per channel group on a
    contiguous slice, grad_vertices summed over groups, the others concatenated
    (dirt/rasterise_ops.py:86-108,111-129; the explicit form is _rasterise_grad_multichannel, :132-177)."""
    from . import oracle
    pixels, grad_pixels = _f32(pixels), _f32(grad_pixels)
    C = pixels.shape[-1]
    groups = list(channel_groups) if channel_groups is not None else oracle.default_groups(C)
    assert sum(groups) == C
    vids = vertex_ids_image(faces, face_ids)
    gbs, gcs, gv_total, begin = [], [], None, 0
    for width in groups:
        sl = slice(begin, begin + width)
        gb, gv, gc = assemble_grads(gbuffer, vids, np.ascontiguousarray(pixels[..., sl]),
                                    np.ascontiguousarray(grad_pixels[..., sl]), vertices)
        gbs.append(gb)
        gcs.append(gc)
        gv_total = gv if gv_total is None else gv_total + gv
        begin += width
    return np.concatenate(gbs, axis=-1), gv_total, np.concatenate(gcs, axis=-1)


def upload_vertices(vertices, faces):
    """The reference's vertex expansion kernel (csrc/rasterise_grad_egl.cu:12-34): structured array [B, 3F]."""
    vertices = _f32(vertices)
    faces = np.ascontiguousarray(faces, np.int32)
    B, V, _ = vertices.shape
    F = faces.shape[1]
    dt = np.dtype([('position', np.float32, 4), ('barycentric', np.float32, 2), ('indices', np.int32, 3)])
    assert dt.itemsize == lib().dirt_ref_sizeof_vertex()
    out = np.empty((B, 3 * F), dt)
    rc = lib().dirt_ref_upload_vertices(_ptr(vertices), _ptr(faces), _ptr(out), B, V, F)
    if rc != 0:
        raise RuntimeError('dirt_ref_upload_vertices failed: %d' % rc)
    return out
