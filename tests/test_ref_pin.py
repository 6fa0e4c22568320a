"""Gradient parity pinned to the reference's own kernel.

tests/golden/ref_*.npz hold outputs of the reference's csrc/rasterise_grad_egl.cu compiled UNMODIFIED
(oracle/_ref, run on a B200 by tests/golden/make_ref_golden.py).  Here:
  * CPU: the oracle's backward pass reproduces them (same G-buffer, same pixels, same grad_pixels);
  * GPU: the CUDA path reproduces them through the C ABI; on the larger LIVE_SCENES, whose recorded runs keep the
    vertex gradients and fingerprints of the rest, the oracle and the CUDA path are checked against both.
Bars: grad_background exact (one writer per pixel); sums of atomics within 1e-4 relative for the CUDA path
(BASELINE.json north_star) and 2e-5 for the oracle, whose only difference from the reference is the order of the
fp32 additions (sequential on the CPU, atomic on the GPU).
"""
import glob
import json
import os

import numpy as np
import pytest

from conftest import rel_close
from dirt_b200 import scenes

GOLDEN = os.path.join(os.path.dirname(__file__), 'golden')
FIXTURES = sorted(glob.glob(os.path.join(GOLDEN, 'ref_grad_*.npz')))


def _name(path):
    return os.path.basename(path)[len('ref_grad_'):-len('.npz')]


def test_fixtures_present():
    if not FIXTURES:
        pytest.skip('tests/golden/ref_grad_*.npz not generated yet: run tests/golden/make_ref_golden.py on a GPU box')
    assert len(FIXTURES) >= 6, 'some of tests/golden/ref_grad_*.npz are missing (tests/golden/make_ref_golden.py)'


@pytest.mark.parametrize('path', FIXTURES, ids=_name)
def test_oracle_matches_reference_kernel(oracle, path):
    d = np.load(path)
    groups = [int(g) for g in d['channel_groups']]
    H, W = d['pixels'].shape[1:3]
    # the fixture's G-buffer is the oracle's own: make sure it still is, bit for bit
    ids, gbuffer = oracle.visibility(d['vertices'], d['faces'], H, W)
    np.testing.assert_array_equal(ids, d['face_ids'])
    np.testing.assert_array_equal(gbuffer, d['gbuffer'])
    gb, gv, gc = oracle.backward(d['vertices'], d['faces'], d['pixels'], d['grad_pixels'], groups)
    np.testing.assert_array_equal(gb, d['ref_grad_background'])
    for name, got, want in (('grad_vertices', gv, d['ref_grad_vertices']), ('grad_vertex_colors', gc, d['ref_grad_vertex_colors'])):
        ok, ratio = rel_close(got, want, rel=2e-5, name='oracle %s vs reference kernel' % name)
        assert ok, '%s: oracle %s off by %.2fx the tolerance from the reference kernel' % (_name(path), name, ratio)
    assert (d['ref_grad_vertices'][..., 2] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize('path', FIXTURES, ids=_name)
def test_cuda_matches_reference_kernel(cuda_lib, path):
    import torch
    from dirt_b200 import rasterise_ops as ops
    d = np.load(path)
    groups = [int(g) for g in d['channel_groups']]
    t = {k: torch.from_numpy(d[k]).cuda() for k in ('vertices', 'faces', 'pixels', 'grad_pixels', 'background', 'vertex_colors')}
    pixels_g, ids_g = ops.rasterise_forward_raw(t['background'], t['vertices'], t['vertex_colors'], t['faces'])
    np.testing.assert_array_equal(ids_g.cpu().numpy(), d['face_ids'])
    for ids_arg in (ids_g, None):
        gb, gv, gc = ops.rasterise_backward_raw(t['vertices'], t['faces'], t['pixels'], t['grad_pixels'], ids_arg, groups)
        np.testing.assert_array_equal(gb.cpu().numpy(), d['ref_grad_background'])
        for name, got, want in (('grad_vertices', gv, d['ref_grad_vertices']), ('grad_vertex_colors', gc, d['ref_grad_vertex_colors'])):
            ok, ratio = rel_close(got.cpu().numpy(), want, name='CUDA %s vs reference kernel' % name)
            assert ok, '%s: CUDA %s off by %.2fx the tolerance from the reference kernel' % (_name(path), name, ratio)


LIVE_SCENES = [
    ('cylinder_scene', dict(batch=2, seed=3), None),
    ('bent_square_scene', dict(channels=7), None),
    ('bent_square_scene', dict(channels=2, width=37, height=29), None),
    ('cube_scene', dict(width=160, height=120), None),
    ('config2', dict(), None),
    ('config3', dict(batch=3, width=160, height=128, level=3, background='uniform'), None),
    ('config5', dict(batch=1, width=256, height=256, n_long=96, n_lat=48), None),
    ('random_soup', dict(batch=2, width=61, height=45, n_faces=70, channels=4, seed=2), [1, 3]),
    ('random_soup', dict(batch=3, width=33, height=47, n_faces=50, channels=1, seed=8), None),
]


def live_spec(gen, kwargs, groups):
    """How tests/golden/ref_live_scenes.npz names the scene of a recorded run."""
    return json.dumps([gen, kwargs, groups], sort_keys=True)


def live_inputs(oracle, gen, kwargs):
    """The inputs of the reference kernel, the oracle and the CUDA path for one LIVE_SCENES entry:
    scene, face ids, G-buffer, pixels (the oracle's) and grad_pixels (seed 7)."""
    s = getattr(scenes, gen)(**kwargs)
    H, W = s['background'].shape[1:3]
    ids, gbuffer = oracle.visibility(s['vertices'], s['faces'], H, W)
    pixels = oracle.forward(**s)
    gp = np.random.default_rng(7).standard_normal(pixels.shape).astype(np.float32)
    return s, ids, gbuffer, pixels, gp


@pytest.mark.gpu
@pytest.mark.parametrize('gen,kwargs,groups', LIVE_SCENES, ids=lambda v: v if isinstance(v, str) else None)
def test_live_reference_kernel(cuda_lib, oracle, gen, kwargs, groups):
    """The reference kernel, the oracle and the CUDA path on the same inputs.  The reference kernel's run on each scene is
    recorded in tests/golden/ref_live_scenes.npz (tests/golden/make_ref_golden.py): its vertex gradients, and fingerprints
    of its inputs and of its grad_background, which must match bit for bit."""
    import torch
    from oracle.ref import fingerprint
    from dirt_b200 import rasterise_ops as ops
    golden = np.load(os.path.join(GOLDEN, 'ref_live_scenes.npz'))
    spec = live_spec(gen, kwargs, groups)
    run = next((k[:-len('_spec')] for k in golden.files if k.endswith('_spec') and str(golden[k]) == spec), None)
    assert run is not None, 'tests/golden/ref_live_scenes.npz has no reference run of %s' % spec
    s, ids, gbuffer, pixels, gp = live_inputs(oracle, gen, kwargs)
    assert fingerprint(s['vertices'], s['faces'], pixels, gp, ids, gbuffer) == str(golden[run + '_inputs']), \
        '%s: the inputs differ from those the reference kernel was run on' % spec
    gb_r = str(golden[run + '_ref_grad_background'])
    gv_r, gc_r = golden[run + '_ref_grad_vertices'], golden[run + '_ref_grad_vertex_colors']
    gb_o, gv_o, gc_o = oracle.backward(s['vertices'], s['faces'], pixels, gp, groups)
    assert fingerprint(gb_o) == gb_r, '%s: oracle grad_background differs from the reference kernel' % gen
    assert rel_close(gv_o, gv_r, rel=2e-5)[0] and rel_close(gc_o, gc_r, rel=2e-5)[0]
    t = {k: torch.from_numpy(v).cuda() for k, v in s.items()}
    gb_g, gv_g, gc_g = ops.rasterise_backward_raw(t['vertices'], t['faces'], torch.from_numpy(pixels).cuda(),
                                                  torch.from_numpy(gp).cuda(), torch.from_numpy(ids).cuda(), groups)
    assert fingerprint(gb_g.cpu().numpy()) == gb_r, '%s: CUDA grad_background differs from the reference kernel' % gen
    for name, got, want in (('grad_vertices', gv_g, gv_r), ('grad_vertex_colors', gc_g, gc_r)):
        ok, ratio = rel_close(got.cpu().numpy(), want, name='CUDA %s vs reference kernel' % name)
        assert ok, '%s: CUDA %s off by %.2fx the tolerance from the reference kernel' % (gen, name, ratio)


def test_reference_vertex_expansion():
    """upload_vertices (csrc/rasterise_grad_egl.cu:12-34) as the reference kernel ran it on a two-image cylinder scene
    (tests/golden/ref_upload_vertices.npz): position gather, barycentric corners, index triple."""
    d = np.load(os.path.join(GOLDEN, 'ref_upload_vertices.npz'))
    vertices, faces = d['vertices'], d['faces']
    B, F = faces.shape[:2]
    for b in range(B):
        np.testing.assert_array_equal(d['position'][b], vertices[b][faces[b].reshape(-1)])
        np.testing.assert_array_equal(d['indices'][b], np.repeat(faces[b], 3, axis=0))
        np.testing.assert_array_equal(d['barycentric'][b], np.tile(np.array([[1, 0], [0, 1], [0, 0]], np.float32), (F, 1)))
