"""GPU: rasterise_batch_shared (one background / face list / vertex-colour set for the whole batch) against rasterise_batch on
the same arguments expanded to the batch.  Forward: bit-equal pixels and face ids.  Backward: a shared background's gradient
bit-equal to the sequential fp32 sum of the per-image ones; shared colour gradients and per-image vertex gradients within
rel_close."""
import ctypes
import itertools

import numpy as np
import pytest

from conftest import rel_close
from dirt_b200 import scenes

pytestmark = pytest.mark.gpu

BG, COLS, FACES = 8, 16, 32
SUBSETS = [sum(c) for n in (1, 2, 3) for c in itertools.combinations((BG, COLS, FACES), n)]


def _soup(channels, batch=3):
    s = scenes.random_soup(batch=batch, width=64, height=48, n_faces=80, channels=channels, seed=channels)
    s['faces'] = np.repeat(s['faces'][:1], batch, axis=0)   # one face list for the batch
    return s


SCENES = {
    'cfg3_small': lambda: scenes.config3(batch=3, width=96, height=64, level=2, background='uniform'),   # C = 4: {3,1} fused
    'cfg4_small': lambda: scenes.config4(batch=3, width=96, height=64, level=2),                         # C = 3: [3] padded
    'soup_c1': lambda: _soup(1),                                                                           # [1]
    'soup_c5': lambda: _soup(5),                                                                           # [3,1,1], non-record path
    'soup_c7': lambda: _soup(7),                                                                           # [3,3,1]
    'b1': lambda: scenes.config3(batch=1, width=64, height=48, level=2, background='uniform'),
}


def _inputs(s, mask):
    """(expanded per-image inputs, shared inputs): item 0's background / colours / faces stand for the batch where shared."""
    import torch
    t = {k: torch.from_numpy(v).cuda() for k, v in s.items()}
    B = t['vertices'].shape[0]
    shared = {'background': t['background'][0].clone() if mask & BG else t['background'],
              'vertex_colors': t['vertex_colors'][0].clone() if mask & COLS else t['vertex_colors'],
              'faces': t['faces'][0].clone() if mask & FACES else t['faces'],
              'vertices': t['vertices']}
    expanded = {k: (v.expand((B,) + tuple(v.shape)).contiguous() if v.dim() < t[k].dim() else v.clone()) for k, v in shared.items()}
    return expanded, shared


def _sequential_sum(per_image):
    import torch
    acc = torch.zeros_like(per_image[0])
    for b in range(per_image.shape[0]):
        acc = acc + per_image[b]
    return acc


def _compare(s, mask, bg_grad=True, seed=0, label=''):
    import torch
    import dirt_b200 as dirt
    from dirt_b200 import rasterise_ops as ops
    ex, sh = _inputs(s, mask)
    # forward: pixels and face ids bit-equal
    px_e, ids_e = ops.rasterise_forward_raw(ex['background'], ex['vertices'], ex['vertex_colors'], ex['faces'])
    px_s, ids_s = ops.rasterise_forward_raw(sh['background'], sh['vertices'], sh['vertex_colors'], sh['faces'], shared=mask)
    assert torch.equal(ids_s, ids_e), label + ': face ids differ'
    assert torch.equal(px_s, px_e), label + ': pixels differ'
    # backward through autograd
    leaves = []
    for d in (ex, sh):
        d['vertices'] = d['vertices'].clone().requires_grad_(True)
        d['vertex_colors'] = d['vertex_colors'].clone().requires_grad_(True)
        d['background'] = d['background'].clone().requires_grad_(bg_grad)
    gp = torch.from_numpy(np.random.default_rng(seed).standard_normal(tuple(px_e.shape)).astype(np.float32)).cuda()
    out_e = dirt.rasterise_batch(ex['background'], ex['vertices'], ex['vertex_colors'], ex['faces'])
    out_s = dirt.rasterise_batch_shared(sh['background'], sh['vertices'], sh['vertex_colors'], sh['faces'])
    assert torch.equal(out_s, out_e), label + ': public-API pixels differ'
    (out_e * gp).sum().backward()
    (out_s * gp).sum().backward()
    if not bg_grad:
        assert sh['background'].grad is None
    elif mask & BG:
        assert sh['background'].grad.shape == sh['background'].shape
        assert torch.equal(sh['background'].grad, _sequential_sum(ex['background'].grad)), label + ': grad_background differs'
    else:
        assert torch.equal(sh['background'].grad, ex['background'].grad), label + ': grad_background differs'
    gc_e = ex['vertex_colors'].grad.double().cpu().numpy()
    if mask & COLS:
        assert sh['vertex_colors'].grad.shape == sh['vertex_colors'].shape
        gc_e = gc_e.sum(axis=0)
    ok, ratio = rel_close(sh['vertex_colors'].grad.cpu().numpy(), gc_e, name='shared grad_vertex_colors')
    assert ok, '%s: grad_vertex_colors off by %.2fx the tolerance' % (label, ratio)
    ok, ratio = rel_close(sh['vertices'].grad.cpu().numpy(), ex['vertices'].grad.cpu().numpy(), name='shared grad_vertices')
    assert ok, '%s: grad_vertices off by %.2fx the tolerance' % (label, ratio)


@pytest.mark.parametrize('name', sorted(SCENES))
@pytest.mark.parametrize('mask', SUBSETS)
def test_shared_inputs_match_the_expanded_batch(cuda_lib, name, mask):
    _compare(SCENES[name](), mask, label='%s mask %d' % (name, mask))


@pytest.mark.parametrize('name', ['cfg3_small', 'soup_c7'])
def test_shared_background_without_grad(cuda_lib, name):
    _compare(SCENES[name](), BG | FACES, bg_grad=False, label=name)


@pytest.mark.parametrize('name', ['cfg3_small', 'cfg4_small', 'soup_c1', 'soup_c7'])
def test_background_reduction_is_one_launch_per_call(cuda_lib, name):
    # the per-channel-group tile launches write no background gradient; one extra kernel sums it when it is wanted
    import torch
    from dirt_b200 import rasterise_ops as ops, _lib
    L = _lib.lib()
    s = SCENES[name]()
    ex, sh = _inputs(s, BG | FACES)
    px, ids, ws = ops.rasterise_forward_raw(sh['background'], sh['vertices'], sh['vertex_colors'], sh['faces'], True, True,
                                            shared=BG | FACES)
    gp = torch.randn_like(px)
    counts = {}
    for key, shared, want_bg in (('per_image', 0, True), ('shared', BG | FACES, True), ('shared_no_bg', BG | FACES, False)):
        faces = sh['faces'] if shared else ex['faces']
        gb, gv, gc = ops.rasterise_backward_raw(sh['vertices'], faces, px, gp, ids, None, None, shared=shared,
                                                want_background=want_bg)
        counts[key] = L.dirt_last_launch_count()
        if key == 'shared':
            assert gb.shape == px.shape[1:]
            per_image = ops.rasterise_backward_raw(sh['vertices'], ex['faces'], px, gp, ids)[0]
            assert torch.equal(gb, _sequential_sum(per_image))
        if key == 'shared_no_bg':
            assert gb is None
    assert counts['shared'] == counts['per_image'] + 1, counts
    assert counts['shared_no_bg'] == counts['per_image'], counts


def test_stale_workspace_across_face_layouts(cuda_lib):
    # a workspace filled with per-image faces does not hold the setup records of a shared-faces call, even when the face
    # list starts at the same address: the tag includes the layout
    import torch
    from dirt_b200 import rasterise_ops as ops, _lib
    L = _lib.lib()
    s = scenes.config3(batch=2, width=96, height=64, level=2, background='uniform')
    t = {k: torch.from_numpy(v).cuda() for k, v in s.items()}
    faces1 = t['faces'][0]   # same storage and address as the batched face list
    B, H, W, C = t['background'].shape
    V, F = t['vertices'].shape[1], t['faces'].shape[1]
    pixels, ids, ws_item = ops.rasterise_forward_raw(t['background'], t['vertices'], t['vertex_colors'], t['faces'], True, True)
    _, _, ws_shared = ops.rasterise_forward_raw(t['background'], t['vertices'], t['vertex_colors'], faces1, True, True,
                                                shared=FACES)
    gp = torch.randn_like(pixels)
    gb = torch.empty_like(pixels); gv = torch.empty((B, V, 4), device='cuda'); gc = torch.empty((B, V, C), device='cuda')
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for ws, stale in ((ws_item, True), (ws_shared, False)):
        rc = L.dirt_rasterise_backward_ex(p(t['vertices']), p(faces1), p(pixels), p(gp), p(ids), p(gb), p(gv), p(gc),
                                          B, H, W, C, V, F, None, 0, 1, FACES, p(ws), int(ws.numel()), stream)
        assert rc == 0
        if stale:
            with pytest.raises(RuntimeError):
                ops.workspace_status(ws, B, H, W, C, V, F)
            torch.cuda.synchronize()
            assert bool(torch.isnan(gv.flatten()[0]))
        else:
            ops.workspace_status(ws, B, H, W, C, V, F)
            assert bool(torch.isfinite(gv).all())


@pytest.mark.parametrize('name', ['cfg3', 'cfg4'])
def test_full_size_shared_inputs(cuda_lib, name):
    s = scenes.config3() if name == 'cfg3' else scenes.config4()
    _compare(s, BG | FACES, bg_grad=True, label=name)
    _compare(s, BG | FACES, bg_grad=False, label=name + ' no background gradient')
    _compare(s, BG | COLS | FACES, bg_grad=True, label=name + ' all shared')
