"""Shared inputs at full size: what one background and one face list for the whole batch cost, against per-image copies.

Workloads cfg3 and cfg4 (bench.py's scenes, zero backgrounds), through the C ABI, each step = forward + backward with the
forward's face ids and setup records, vertex gradients accumulated over the batch (as bench.py), replayed as a CUDA graph and
timed with CUDA events.  Arms, run alternately in every round:
  a  per-image background [B,H,W,C] and faces [B,F,3] (today's inputs), grad_background [B,H,W,C] written
  b  shared background [H,W,C] and faces [F,3], no background gradient (a constant background: the common case)
  c  as b, plus the shared background's gradient [H,W,C] (background_grad_kernel)
Per arm: step ms (median over rounds, and the spread), forward / backward / background-gradient kernel ms
(dirt_kernel_timer_*, eager calls), algorithmic bytes from the shapes (the byte model of DESIGN.md section 4) and
torch.cuda.max_memory_allocated of the arm's buffers.  Then one public-API training step: rasterise_batch on expanded
inputs against rasterise_batch_shared (vertices and vertex colours require grad, the background does not).

    python profiles/shared_inputs.py [--steps 50] [--rounds 7] > profiles/r03_shared_inputs.txt
"""
import argparse
import ctypes
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BG, COLS, FACES, SHARED_GEOMETRY = 8, 16, 32, 1
ARMS = {'a': 'per-image background + faces, grad_background [B,H,W,C]',
        'b': 'shared background + faces, no background gradient',
        'c': 'shared background + faces + grad_background [H,W,C]'}


def algorithmic_bytes(arm, B, H, W, C, V, F):
    """(forward, backward) bytes the arm must move at least: bench.py's per-image model, with a shared input read once."""
    px = H * W * C * 4
    fwd = B * px + B * (V * 16 + V * C * 4)                 # pixels written, vertices and colours read
    fwd += (px + F * 12) if arm != 'a' else B * (px + F * 12)  # background, faces
    bwd = 2 * B * px + B * (V * 16 + V * 16 + V * C * 4)   # grad_pixels + pixels read, vertices read, vertex gradients
    bwd += F * 12 if arm != 'a' else B * F * 12
    if arm == 'a':
        bwd += B * px                                       # grad_background written per image
    if arm == 'c':
        bwd += B * H * W * 4 + B * px + px                  # background_grad_kernel: face ids + grad_pixels read, [H,W,C] written
    return fwd, bwd


class Arm:
    def __init__(self, torch, L, scene, arm, device):
        self.torch, self.L = torch, L
        t = {k: torch.from_numpy(v).to(device) for k, v in scene.items()}
        B, H, W, C = t['background'].shape
        V, F = t['vertices'].shape[1], t['faces'].shape[1]
        self.dims = (B, H, W, C, V, F)
        self.shared = 0 if arm == 'a' else BG | FACES
        self.background = t['background'] if arm == 'a' else t['background'][0].clone()
        self.faces = t['faces'] if arm == 'a' else t['faces'][0].clone()
        self.vertices, self.vertex_colors = t['vertices'], t['vertex_colors']
        self.pixels = torch.empty((B, H, W, C), device=device)
        self.face_ids = torch.empty((B, H, W), dtype=torch.int32, device=device)
        self.grad_pixels = torch.from_numpy(np.random.default_rng(2).standard_normal((B, H, W, C)).astype(np.float32)).to(device)
        self.grad_background = {'a': lambda: torch.empty((B, H, W, C), device=device), 'b': lambda: None,
                                'c': lambda: torch.empty((H, W, C), device=device)}[arm]()
        self.gv = torch.empty((V, 4), device=device)
        self.gc = torch.empty((V, C), device=device)
        self.ws_bytes = int(L.dirt_workspace_bytes(B, H, W, C, V, F))
        self.workspace = torch.empty(self.ws_bytes, dtype=torch.uint8, device=device)
        self.graph = None

    def _p(self, x):
        return ctypes.c_void_p(0 if x is None else x.data_ptr())

    def step(self):
        from dirt_b200 import _lib
        B, H, W, C, V, F = self.dims
        stream = ctypes.c_void_p(self.torch.cuda.current_stream().cuda_stream)
        p = self._p
        _lib.check(self.L.dirt_rasterise_forward_ex(p(self.background), p(self.vertices), p(self.vertex_colors), p(self.faces),
                                                    p(self.pixels), p(self.face_ids), B, H, W, C, V, F, p(self.workspace),
                                                    self.ws_bytes, stream, self.shared), 'Rasterise')
        _lib.check(self.L.dirt_rasterise_backward_ex(p(self.vertices), p(self.faces), p(self.pixels), p(self.grad_pixels),
                                                     p(self.face_ids), p(self.grad_background), p(self.gv), p(self.gc),
                                                     B, H, W, C, V, F, None, 0, 1, SHARED_GEOMETRY | self.shared,
                                                     p(self.workspace), self.ws_bytes, stream), 'RasteriseGrad')

    def capture(self):
        torch = self.torch
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            self.step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.step()

    def time_steps(self, n):
        torch = self.torch
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(n):
            self.graph.replay()
        stop.record()
        stop.synchronize()
        return start.elapsed_time(stop) / n

    def time_kernel(self, which, n):
        total, got = 0.0, 0
        self.L.dirt_kernel_timer_enable(which)
        for _ in range(n):
            self.L.dirt_kernel_timer_enable(which)   # clears the previous record
            self.step()
            ms = float(self.L.dirt_kernel_timer_elapsed_ms())
            if ms >= 0:
                total, got = total + ms, got + 1
        self.L.dirt_kernel_timer_enable(0)
        return total / got if got else None


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else 'nvidia-smi gave no output'
    except Exception as e:   # reported, not fatal
        return 'nvidia-smi unavailable (%s)' % e


def public_api_step(torch, scene, device, steps):
    """rasterise_batch on expanded inputs vs rasterise_batch_shared: one training step = forward, loss, backward."""
    import dirt_b200 as dirt
    t = {k: torch.from_numpy(v).to(device) for k, v in scene.items()}
    B = t['vertices'].shape[0]
    bg, faces = t['background'][0].clone(), t['faces'][0].clone()
    verts = t['vertices'].clone().requires_grad_(True)
    cols = t['vertex_colors'][0].clone().requires_grad_(True)
    gp = torch.from_numpy(np.random.default_rng(3).standard_normal(tuple(t['background'].shape)).astype(np.float32)).to(device)
    calls = {
        'rasterise_batch (expanded)': lambda: dirt.rasterise_batch(bg.expand((B,) + tuple(bg.shape)), verts,
                                                                   cols.expand((B,) + tuple(cols.shape)),
                                                                   faces.expand((B,) + tuple(faces.shape))),
        'rasterise_batch_shared': lambda: dirt.rasterise_batch_shared(bg, verts, cols, faces),
    }
    results = {}
    for rnd in range(3):
        for name, fn in calls.items():
            def step():
                verts.grad = None
                cols.grad = None
                (fn() * gp).sum().backward()
            step()
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            for _ in range(steps):
                step()
            stop.record()
            stop.synchronize()
            r = results.setdefault(name, {'ms': [], 'peak_mb': 0.0})
            r['ms'].append(start.elapsed_time(stop) / steps)
            r['peak_mb'] = max(r['peak_mb'], (torch.cuda.max_memory_allocated() - base) / 1e6)
    return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--rounds', type=int, default=7)
    ap.add_argument('--workloads', default='cfg3,cfg4')
    args = ap.parse_args()
    import torch
    from dirt_b200 import _lib, scenes
    if not torch.cuda.is_available():
        raise RuntimeError('profiles/shared_inputs.py measures on a CUDA device; there is nothing to measure without one')
    device = torch.device('cuda', 0)
    L = _lib.lib()
    print('card: %s | %s' % (torch.cuda.get_device_name(device), card()))
    print('torch %s, CUDA %s; %d steps per timed window, %d rounds, arms alternate inside each round' %
          (torch.__version__, torch.version.cuda, args.steps, args.rounds))
    for name in args.workloads.split(','):
        scene = scenes.config3() if name == 'cfg3' else scenes.config4()
        B, H, W, C = scene['background'].shape
        V, F = scene['vertices'].shape[1], scene['faces'].shape[1]
        print('\n== %s: B=%d %dx%d C=%d V=%d F=%d (zero background)' % (name, B, W, H, C, V, F))
        arms, mem = {}, {}
        for a in ARMS:
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            arms[a] = Arm(torch, L, scene, a, device)
            arms[a].step()
            torch.cuda.synchronize()
            mem[a] = (torch.cuda.max_memory_allocated() - base) / 1e6
            arms[a].capture()
        for a in arms:
            arms[a].time_steps(5)
        ms = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a in arms:
                ms[a].append(arms[a].time_steps(args.steps))
        kern = {a: (arms[a].time_kernel(1, 20), arms[a].time_kernel(2, 20), arms[a].time_kernel(3, 20) if a == 'c' else None)
                for a in arms}
        print('%-4s %-58s %9s %17s %8s %8s %8s %9s %9s %9s' % ('arm', 'inputs', 'step ms', 'spread (min-max)', 'fwd ms',
                                                              'bwd ms', 'bg ms', 'fwd MB', 'bwd MB', 'alloc MB'))
        for a in arms:
            f, b = algorithmic_bytes(a, B, H, W, C, V, F)
            kf, kb, kg = kern[a]
            print('%-4s %-58s %9.4f %8.4f-%-8.4f %8.4f %8.4f %8s %9.1f %9.1f %9.1f' % (
                a, ARMS[a], float(np.median(ms[a])), min(ms[a]), max(ms[a]), kf, kb, '%.4f' % kg if kg is not None else '-',
                f / 1e6, b / 1e6, mem[a]))
        del arms
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        res = public_api_step(torch, scene, device, max(5, args.steps // 5))
        print('public API, one training step (forward + loss + backward; vertices and [V,C] colours require grad, background does not):')
        for k, r in res.items():
            print('  %-30s %8.4f ms (min %.4f, max %.4f over %d rounds)   peak allocated %8.1f MB' %
                  (k, float(np.median(r['ms'])), min(r['ms']), max(r['ms']), len(r['ms']), r['peak_mb']))


if __name__ == '__main__':
    main()
