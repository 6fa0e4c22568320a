"""Generates tests/golden/ref_*.npz: outputs of the REFERENCE'S OWN gradient kernel.

    python tests/golden/make_ref_golden.py --out DIR      (needs a GPU and oracle/_ref: assemble_grads is CUDA)
    cp DIR/*.npz tests/golden/

oracle/_ref/libdirt_ref_grad.so is the reference's csrc/rasterise_grad_egl.cu compiled unmodified (oracle/Makefile,
target `ref`).  For each scene below this script takes the CPU oracle's visibility G-buffer (the part of the
reference that lives in the OpenGL driver) and the oracle's forward pixels, draws grad_pixels from a seeded
generator, and runs the reference kernel once per channel group, exactly as dirt/rasterise_ops.py:86-129 calls the
RasteriseGrad op.  Inputs and reference outputs go into one compressed .npz per scene, so the tests need neither
the reference nor a GPU to check the oracle, and no reference to check the CUDA path.

ref_live_scenes.npz holds the runs of tests/test_ref_pin.py's LIVE_SCENES, whose images are too large to store: the
vertex gradients themselves, and fingerprints (oracle.ref.fingerprint) of the inputs and of grad_background, which the
test regenerates and compares bit for bit.  ref_upload_vertices.npz holds the reference's vertex expansion of one scene.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from dirt_b200 import scenes  # noqa: E402  (scene generators only: numpy, no CUDA)
from oracle import oracle, ref  # noqa: E402
sys.path.insert(0, os.path.join(ROOT, 'tests'))
from test_ref_pin import LIVE_SCENES, live_inputs, live_spec  # noqa: E402

# name -> (generator, kwargs, channel groups or None for the reference's greedy split, grad_pixels seed)
SCENES = {
    'cylinder_48x36': ('cylinder_scene', dict(), None, 11),                                   # tests/rasterise_tests.py:52-89
    'bent_square_c3': ('bent_square_scene', dict(channels=3), None, 12),                      # tests/deferred_grad_test.py:19-55
    'bent_square_c1': ('bent_square_scene', dict(channels=1), None, 13),                      # 1-channel flat-order reads (A.4.1)
    'cfg3_small_c4': ('config3', dict(batch=2, width=96, height=80, level=2, background='uniform'), [3, 1], 14),
    'soup_c3': ('random_soup', dict(batch=2, width=61, height=45, n_faces=70, channels=3, seed=5), None, 15),
    'soup_behind_c1': ('random_soup', dict(batch=1, width=64, height=48, n_faces=40, channels=1, seed=11, behind_camera=True), None, 16),
}


def make(name):
    gen, kwargs, groups, seed = SCENES[name]
    s = getattr(scenes, gen)(**kwargs)
    B, H, W, C = s['background'].shape
    ids, gbuffer = oracle.visibility(s['vertices'], s['faces'], H, W)
    pixels = oracle.forward(**s)
    grad_pixels = np.random.default_rng(seed).standard_normal(pixels.shape).astype(np.float32)
    gb, gv, gc = ref.backward(s['vertices'], s['faces'], pixels, grad_pixels, gbuffer, ids, groups)
    used_groups = np.array(groups if groups is not None else oracle.default_groups(C), np.int32)
    return dict(vertices=s['vertices'], faces=s['faces'], vertex_colors=s['vertex_colors'], background=s['background'],
                pixels=pixels, grad_pixels=grad_pixels, face_ids=ids, gbuffer=gbuffer, channel_groups=used_groups,
                ref_grad_background=gb, ref_grad_vertices=gv, ref_grad_vertex_colors=gc)


def make_live():
    data = {}
    for i, (gen, kwargs, groups) in enumerate(LIVE_SCENES):
        s, ids, gbuffer, pixels, gp = live_inputs(oracle, gen, kwargs)
        gb, gv, gc = ref.backward(s['vertices'], s['faces'], pixels, gp, gbuffer, ids, groups)
        data.update({'live%d_spec' % i: np.array(live_spec(gen, kwargs, groups)),
                     'live%d_inputs' % i: np.array(ref.fingerprint(s['vertices'], s['faces'], pixels, gp, ids, gbuffer)),
                     'live%d_ref_grad_background' % i: np.array(ref.fingerprint(gb)),
                     'live%d_ref_grad_vertices' % i: gv, 'live%d_ref_grad_vertex_colors' % i: gc})
    return data


def make_upload_vertices():
    s = scenes.cylinder_scene(batch=2, seed=1)
    out = ref.upload_vertices(s['vertices'], s['faces'])
    return dict(vertices=s['vertices'], faces=s['faces'], position=out['position'], barycentric=out['barycentric'],
                indices=out['indices'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'tests', 'golden'))
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    oracle.build()
    for name in SCENES:
        data = make(name)
        path = os.path.join(args.out, 'ref_grad_%s.npz' % name)
        np.savez_compressed(path, **data)
        print('%s: %d covered pixels, |grad_vertices|max = %.4g, %d bytes' % (
            name, int((data['face_ids'] >= 0).sum()), float(np.abs(data['ref_grad_vertices']).max()), os.path.getsize(path)))
    for name, data in (('ref_live_scenes', make_live()), ('ref_upload_vertices', make_upload_vertices())):
        path = os.path.join(args.out, name + '.npz')
        np.savez_compressed(path, **data)
        print('%s: %d bytes' % (name, os.path.getsize(path)))


if __name__ == '__main__':
    main()
