#!/usr/bin/env python
"""bench.py -- fwd+bwd Mpixels/s of the rasterise hot path on BASELINE.json's workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg4|cfg5|cfg2|cube]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward + one backward pass of the hot path over one batch of synthetic scenes
(BASELINE cfg3 by default: batch 64 per GPU, 512x512, 4-channel G-buffer, 5120-triangle icosphere with a
pose per item), called through the C ABI of libdirt_b200.so with every buffer already resident in HBM,
with the vertex gradients accumulated over the batch inside the backward kernel (DIRT_BWD_SHARED_GEOMETRY: one
[V, 4+C] buffer) and -- when N > 1 -- ONE sum of that buffer over the ranks per step: the library's peer-memory kernel
(dirt_peer_exchange; --collective nccl / the automatic fallback: NCCL's all-reduce), issued on a side stream so that it
overlaps the next step's forward pass (the batch shards over GPUs with no other exchange: weak scaling, 64 images per GPU).
The timed region is bracketed by barrier + synchronize on both sides; the start events are additionally aligned on the
device (a one-element all-reduce enqueued before them), and `multi_gpu` in the JSON line lists every rank's time with and
without the exchange.

One JSON line on rank 0:  value = B_total*H*W / step time (CUDA events, max over ranks);  e2e = the same
call with HOST (pinned) buffers, host<->device copies inside the timed region;  roofline = the dominant
kernel against the measured HBM copy peak;  cpu_baseline = the CPU oracle on a bounded sample.
--impl reference times the CPU port of the reference path (oracle/), the only runnable reference here.
--dump-outputs DIR writes the outputs of the last timed step as .npy files (dump_outputs); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.  The bench writes nothing into the tree.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only: no __pycache__ is written next to the sources
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'fwd+bwd Mpixels/sec'
UNIT = 'Mpixels/s'

WORKLOADS = {
    # name: (generator, kwargs, description)
    'cfg3': ('config3', dict(batch=64, width=512, height=512), 'BASELINE cfg3: batch=64/GPU, 512x512, 4-channel G-buffer, icosphere-4 (V=2562, F=5120), per-item pose'),
    'cfg4': ('config4', dict(batch=32, width=512, height=512), 'BASELINE cfg4 shard: batch=32/GPU, 512x512, 3-channel, icosphere-4'),
    'cfg5': ('config5', dict(batch=64, width=1024, height=1024), 'BASELINE cfg5: batch=64/GPU, 1024x1024, 3-channel, UV sphere (V=24866, F=49728)'),
    'cfg2': ('config2', dict(), 'BASELINE cfg2: batch=1, 256x256, 3-channel, icosphere-3'),
    'cube': ('cube_batch', dict(batch=64, width=640, height=480), 'samples/simple.py cube, batch=64/GPU, 640x480, 3-channel, 12 triangles (large-face path)'),
}


def algorithmic_bytes(B, H, W, C, V, F):
    """SURVEY 8(d): per image fwd = 2*H*W*C*4 + V*16 + V*C*4 + F*12; bwd = 3*H*W*C*4 + V*16 + F*12 + V*16 + V*C*4."""
    fwd = B * (2 * H * W * C * 4 + V * 16 + V * C * 4 + F * 12)
    bwd = B * (3 * H * W * C * 4 + V * 16 + F * 12 + V * 16 + V * C * 4)
    return fwd, bwd


def measured_peak_gbs():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs, burst copy)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md: 6.65 TB/s)'


def host_record():
    """Who ran the CPU legs (BASELINE.md section 4 asks for it next to every CPU number)."""
    model = None
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.lower().startswith('model name'):
                    model = line.split(':', 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count()
    import socket
    return {'hostname': socket.gethostname(), 'cpu_model': model, 'nproc': os.cpu_count(), 'usable_threads': usable}


def bind_to_gpu_numa_node(index):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned buffer is allocated: Linux
    places pages on the node of the thread that first touches them, and a pinned buffer on the far socket costs the
    H2D / D2H copies about half their rate once several ranks copy at once (SCALE_r01: 40 -> 20 GB/s per GPU at N=8).
    Returns what was done, for the JSON line."""
    info = {'node': None, 'cpus': None}

    def parse_cpulist(text):
        cpus = set()
        for part in text.strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return cpus

    try:
        cpus, node = None, None
        # the driver's own view first: the "CPU Affinity" / "NUMA Affinity" columns of `nvidia-smi topo -m`
        topo = subprocess.run(['nvidia-smi', 'topo', '-m'], capture_output=True, text=True, timeout=30).stdout
        import re
        lines = [re.sub(r'\x1b\[[0-9;]*m', '', l) for l in topo.splitlines()]
        header = next((l for l in lines if 'CPU Affinity' in l), None)
        row = next((l for l in lines if l.startswith('GPU%d\t' % index) or l.startswith('GPU%d ' % index)), None)
        if header and row:
            hcols = [c.strip() for c in header.split('\t')]
            rcols = [c.strip() for c in row.split('\t')]
            ci = hcols.index('CPU Affinity')   # the header line starts with an empty cell above the row labels
            if ci < len(rcols) and rcols[ci]:
                cpus = parse_cpulist(rcols[ci])
                ni = ci + 1
                node = int(rcols[ni]) if ni < len(rcols) and rcols[ni].isdigit() else None
        if not cpus:   # sysfs: PCI device -> NUMA node -> cpulist
            bdf = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=pci.bus_id', '--format=csv,noheader'],
                                 capture_output=True, text=True, timeout=20).stdout.strip().lower()
            if bdf.count(':') == 2 and len(bdf.split(':')[0]) == 8:
                bdf = bdf[4:]   # sysfs uses a 4-digit PCI domain
            with open('/sys/bus/pci/devices/%s/numa_node' % bdf) as f:
                node = int(f.read().strip())
            if node < 0:
                return info
            with open('/sys/devices/system/node/node%d/cpulist' % node) as f:
                cpus = parse_cpulist(f.read())
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info = {'node': node, 'cpus': len(cpus)}
    except Exception as exc:   # no sysfs / nvidia-smi: run unbound
        info['error'] = repr(exc)
    return info


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.samples = []
        self.proc = None

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append(line.strip())
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, smax, reasons = [], [], set()
        for line in self.samples:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), parts[2:6]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(smax)), 'reasons': sorted(reasons), 'samples': len(sm)}


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------

class PreparedStep:
    """Preallocated buffers + the two C-ABI calls of one step (forward, backward with cached visibility)."""

    def __init__(self, scene, device, grad_seed=2):
        import torch
        from dirt_b200 import _lib
        self.torch = torch
        self.lib = _lib.lib()
        self._check = _lib.check
        self.device = device
        self.host = scene
        B, H, W, C = scene['background'].shape
        V, F = scene['vertices'].shape[1], scene['faces'].shape[1]
        self.dims = (B, H, W, C, V, F)
        self.grad_pixels_host = np.random.default_rng(grad_seed).standard_normal((B, H, W, C)).astype(np.float32)
        dev = {k: torch.from_numpy(v).to(device) for k, v in scene.items()}
        self.background, self.vertices = dev['background'], dev['vertices']
        self.vertex_colors, self.faces = dev['vertex_colors'], dev['faces']
        self.grad_pixels = torch.from_numpy(self.grad_pixels_host).to(device)
        self.pixels = torch.empty_like(self.background)
        self.face_ids = torch.empty((B, H, W), dtype=torch.int32, device=device)
        self.grad_background = torch.empty_like(self.background)
        # gradient of the batch-shared geometry: [V,4] | [V,C] in ONE flat buffer (what the all-reduce moves); two of
        # them alternate so that the all-reduce of step k overlaps the kernels of step k+1
        self.flat_len = 4 * ((V * (4 + C) + 3) // 4)   # whole 16-byte words (the peer exchange moves float4s)
        self.shared_flat = [torch.zeros(self.flat_len, dtype=torch.float32, device=device) for _ in range(2)]
        self.shared_gv = [f[:V * 4].view(V, 4) for f in self.shared_flat]
        self.shared_gc = [f[V * 4:V * (4 + C)].view(V, C) for f in self.shared_flat]
        self.ws_bytes = int(self.lib.dirt_workspace_bytes(B, H, W, C, V, F))
        self.workspace = torch.empty(self.ws_bytes, dtype=torch.uint8, device=device)
        self.launches_per_step = 0
        self.graphs = None
        self.parity = 0
        self.comm_stream = torch.cuda.Stream(device, priority=-1)   # its few CTAs go ahead of the queued tiles
        self.comm_done = [None, None]
        self.peer = None          # dirt_b200.distributed.PeerExchange when the ranks can map each other's memory
        self.reduced_flat = None  # its output: the gradient summed over ranks, one buffer per step parity
        self.collective = 'none (N=1)'

    def setup_exchange(self, world, mode):
        """The sum over ranks of shared_flat: the library's peer-memory kernel, or NCCL's all-reduce (in place) if the peer
        mapping is unavailable / not wanted.  Collective: every rank calls it."""
        torch = self.torch
        V, C = self.dims[4], self.dims[3]
        width = 4 + C
        if world > 1 and mode != 'nccl':
            try:
                from dirt_b200.distributed import PeerExchange
                import torch.distributed as dist
                failure = None
                try:
                    self.peer = PeerExchange(self.flat_len, self.device)
                except Exception as e:
                    failure = e
                ok = torch.tensor([0.0 if failure is not None else 1.0], device=self.device)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # one rank without the mapping: nobody uses it
                if float(ok.item()) < 1.0:
                    self.peer = None
                    raise failure if failure is not None else RuntimeError('another rank could not map peer memory')
                self.reduced_flat = [torch.zeros_like(f) for f in self.shared_flat]
                self.collective = ('dirt_peer_exchange: [V,%d] fp32 gradient of the batch-shared geometry pushed into every peer\'s '
                                   'memory and summed in rank order, one kernel of %d CTAs per rank and step on a side stream, '
                                   'overlapping the next step' % (width, world))
                return
            except Exception as e:   # said out loud, and in the JSON line
                if mode == 'peer':
                    raise
                sys.stderr.write('bench: peer exchange unavailable (%s: %s); using the NCCL all-reduce\n' % (type(e).__name__, e))
                self.peer = None
        if world > 1:
            self.collective = ('nccl all_reduce([V,%d] fp32 gradient of the batch-shared geometry) once per step on a side stream, '
                               'overlapping the next step' % width)

    def _p(self, t):
        return ctypes.c_void_p(t.data_ptr())

    def forward(self):
        B, H, W, C, V, F = self.dims
        stream = ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)
        rc = self.lib.dirt_rasterise_forward(self._p(self.background), self._p(self.vertices), self._p(self.vertex_colors),
                                             self._p(self.faces), self._p(self.pixels), self._p(self.face_ids), B, H, W, C, V, F,
                                             self._p(self.workspace), self.ws_bytes, stream)
        self._check(rc, 'Rasterise')
        return self.lib.dirt_last_launch_count()

    def backward(self, which=0):
        B, H, W, C, V, F = self.dims
        stream = ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)
        # vertex gradients accumulated over the batch inside the kernel (flags = DIRT_BWD_SHARED_GEOMETRY)
        rc = self.lib.dirt_rasterise_backward_ex(self._p(self.vertices), self._p(self.faces), self._p(self.pixels),
                                                 self._p(self.grad_pixels), self._p(self.face_ids), self._p(self.grad_background),
                                                 self._p(self.shared_gv[which]), self._p(self.shared_gc[which]), B, H, W, C, V, F,
                                                 None, 0, 1, 1, self._p(self.workspace), self.ws_bytes, stream)
        self._check(rc, 'RasteriseGrad')
        return self.lib.dirt_last_launch_count()

    def local_step(self, which=0):
        """forward + backward, the gradient of the batch-shared geometry landing in shared_flat[which] (no collective)."""
        n = self.forward()
        n += self.backward(which)
        self.launches_per_step = n
        return n

    def capture(self):
        """Record local_step() into CUDA graphs, one per gradient buffer (every C-ABI call only enqueues work on the given stream)."""
        torch = self.torch
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self.local_step(0)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        self.graphs = []
        for which in (0, 1):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.local_step(which)
            self.graphs.append(g)

    def step(self, world):
        """One step.  With N > 1 the all-reduce of this step's [V, 4+C] buffer runs on a side stream, overlapping the next
        step's kernels (which write the OTHER buffer); the step after that waits for it before reusing the buffer."""
        torch = self.torch
        which = self.parity
        self.parity ^= 1
        cur = torch.cuda.current_stream(self.device)
        if world > 1 and self.comm_done[which] is not None:
            cur.wait_event(self.comm_done[which])   # the all-reduce that last read this buffer
        if self.graphs is not None:
            self.graphs[which].replay()
            n = self.launches_per_step
        else:
            n = self.local_step(which)
        if world > 1:   # the one exchange of the path: all-reduce of the [V, 4+C] shared-geometry gradient
            import torch.distributed as dist
            ready = torch.cuda.Event()
            ready.record(cur)
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(ready)
                if self.peer is not None:
                    self.peer.exchange(self.shared_flat[which], self.reduced_flat[which], self.comm_stream)
                else:
                    dist.all_reduce(self.shared_flat[which], op=dist.ReduceOp.SUM)
                done = torch.cuda.Event()
                done.record(self.comm_stream)
            self.comm_done[which] = done
        return n

    def drain(self):
        """Make the current stream wait for every outstanding all-reduce (end of a timed region)."""
        cur = self.torch.cuda.current_stream(self.device)
        for ev in self.comm_done:
            if ev is not None:
                cur.wait_event(ev)


class HostStep:
    """The same two calls with HOST buffers through the package's host entry point (dirt_b200.host.HostRasteriser):
    pinned inputs -> device, forward + backward, outputs -> pinned host, pipelined over batch chunks."""

    def __init__(self, prepared, chunks=4):
        from dirt_b200.host import HostRasteriser
        torch = prepared.torch
        self.p = prepared
        B, H, W, C, V, F = prepared.dims
        self.runner = HostRasteriser(B, H, W, C, V, F, device=prepared.device, chunks=chunks)
        pin = lambda a: torch.from_numpy(a).pin_memory()
        s = prepared.host
        self.h_in = dict(background=pin(s['background']), vertices=pin(s['vertices']), vertex_colors=pin(s['vertex_colors']),
                         faces=pin(s['faces']), grad_pixels=pin(prepared.grad_pixels_host))
        self.h2d = self.runner.h2d_bytes
        self.d2h = self.runner.d2h_bytes

    def step(self):
        return self.runner.step(**self.h_in)

    def copies_only(self):
        """The transfers of one step with no kernels: all inputs host->device on one stream while all outputs go
        device->host on another (PCIe is full duplex) -- the floor under the end-to-end time of this box."""
        torch, r = self.p.torch, self.runner
        cur = torch.cuda.current_stream(r.device)
        r.s_in.wait_stream(cur); r.s_out.wait_stream(cur)
        with torch.cuda.stream(r.s_in):
            for k, t in self.h_in.items():
                r.d[k].copy_(t, non_blocking=True)
        with torch.cuda.stream(r.s_out):
            for k, t in r.h_out.items():
                t.copy_(r.d[k], non_blocking=True)
        cur.wait_stream(r.s_in); cur.wait_stream(r.s_out)


def check_against_oracle(prep, scene, images=1):
    """Outside the timed region: the buffers the timed steps left behind against the CPU oracle (first `images` images)
    and, for the batch-accumulated vertex gradients, against the per-item call summed over the batch."""
    import torch
    from oracle import oracle
    from dirt_b200 import rasterise_ops as ops
    oracle.build()
    B, H, W, C, V, F = prep.dims
    n = min(images, B)
    prep.local_step(0)
    torch.cuda.synchronize(prep.device)
    sub = {k: np.ascontiguousarray(v[:n]) for k, v in scene.items()}
    pixels_o, ids_o = oracle.forward(**sub, return_face_ids=True)
    gp = prep.grad_pixels_host[:n]
    # RasteriseGrad is a function of (vertices, faces, pixels, grad_pixels): the oracle gets the SAME pixels the CUDA call
    # gets (the benched forward's output, itself compared with the oracle's below).  Feeding each side its own pixels
    # compares two different inputs wherever the Scharr norms tie -- flat-shaded faces (the cube) tie at most silhouette
    # pixels, and the last bit of a pixel value then picks the dilation direction.
    gb_o, gv_o, gc_o = oracle.backward(sub['vertices'], sub['faces'], np.ascontiguousarray(prep.pixels[:n].cpu().numpy()), gp)

    def worst(a, b):
        a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
        allowed = 1e-4 * np.maximum(np.maximum(np.abs(a), np.abs(b)), 1e-2 * np.abs(b).max())
        return float((np.abs(a - b) / allowed).max())

    res = {'images': n}
    res['face_ids_equal'] = bool((prep.face_ids[:n].cpu().numpy() == ids_o).all())
    res['pixels_err_over_tol'] = worst(prep.pixels[:n].cpu().numpy(), pixels_o)
    res['grad_background_equal'] = bool((prep.grad_background[:n].cpu().numpy() == gb_o).all())
    # per-item gradients of the same batch through the same library (the timed step accumulates them over the batch)
    gb, gv, gc = ops.rasterise_backward_raw(prep.vertices, prep.faces, prep.pixels, prep.grad_pixels, prep.face_ids)
    res['grad_vertices_err_over_tol'] = worst(gv[:n].cpu().numpy(), gv_o)
    res['grad_vertex_colors_err_over_tol'] = worst(gc[:n].cpu().numpy(), gc_o)
    res['shared_grad_vertices_err_over_tol'] = worst(prep.shared_gv[0].cpu().numpy(), gv.double().sum(0).cpu().numpy())
    res['shared_grad_vertex_colors_err_over_tol'] = worst(prep.shared_gc[0].cpu().numpy(), gc.double().sum(0).cpu().numpy())
    res['ok'] = bool(res['face_ids_equal'] and res['grad_background_equal'] and
                     all(v <= 1.0 for k, v in res.items() if k.endswith('_over_tol')))
    return res


DUMP_BYTES = 64 << 20


def dump_outputs(prep, which, out_dir, seed=0):
    """Writes what a caller of the timed path receives from its last step (gradient buffer `which`) as out_dir/<name>.npy:
    the batch-accumulated grad_vertices [V,4] and grad_vertex_colors [V,C] (summed over the ranks when N > 1), and
    pixels [n,C], face_ids [n] and grad_background [n,C] at the n pixels listed in pixel_index [n] (flat index b*H*W + y*W + x).
    n is every pixel of the batch, or a fixed sample drawn with `seed` when that would exceed DUMP_BYTES in all, so two builds
    run with the same arguments can be compared file for file."""
    torch = prep.torch
    B, H, W, C, V, F = prep.dims
    flat = prep.reduced_flat[which] if prep.peer is not None else prep.shared_flat[which]
    out = {'grad_vertices': flat[:V * 4].view(V, 4).cpu().numpy(),
           'grad_vertex_colors': flat[V * 4:V * (4 + C)].view(V, C).cpu().numpy()}
    n_pix = B * H * W
    per_pixel = 4 * (2 * C + 1) + 8   # pixels and grad_background (C float32 each), the face id (float32), the index (float64)
    n = min(n_pix, (DUMP_BYTES - 4096 - sum(a.nbytes for a in out.values())) // per_pixel)   # 4096: the six .npy headers
    index = np.arange(n_pix) if n == n_pix else np.sort(np.random.default_rng(seed).choice(n_pix, size=n, replace=False))
    idx = torch.from_numpy(index).to(prep.device)
    out['pixel_index'] = index.astype(np.float64)
    out['pixels'] = prep.pixels.view(n_pix, C)[idx].cpu().numpy()
    out['face_ids'] = prep.face_ids.view(n_pix)[idx].float().cpu().numpy()   # exact: face ids stay below 2^24
    out['grad_background'] = prep.grad_background.view(n_pix, C)[idx].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def numpy_baselines(scene, grad_pixels, threads, one_process_images=2, budget_s=20.0):
    """The reference-style numpy path (oracle/numpy_raster.py: coverage on a meshgrid of pixel centres, as
    tests/square_test.py:11-17 does for its square) fwd+bwd: (i) one process, (ii) a multiprocessing pool over the
    images on every host thread.  Bounded samples of the same workload (BASELINE.md section 4)."""
    from oracle import numpy_raster as npr
    B, H, W = scene['background'].shape[:3]
    out = {}
    n1 = min(one_process_images, B)
    sub = {k: v[:n1] for k, v in scene.items()}
    t0 = time.perf_counter()
    npr.forward_backward_batch(sub, grad_pixels[:n1], processes=1)
    dt1 = time.perf_counter() - t0
    out['numpy_1_process'] = {'value': n1 * H * W / dt1 / 1e6, 'unit': UNIT, 'cores': 1,
                              'sample': '%d images, %.1f s' % (n1, dt1)}
    # pool: as many images as one round of all workers renders within the budget
    procs = max(1, threads)
    nmp = max(1, min(B, int(procs * max(1.0, budget_s / max(dt1 / n1, 1e-3) / 4.0))))
    sub = {k: v[:nmp] for k, v in scene.items()}
    t0 = time.perf_counter()
    npr.forward_backward_batch(sub, grad_pixels[:nmp], processes=min(procs, nmp))
    dtm = time.perf_counter() - t0
    out['numpy_multiprocessing'] = {'value': nmp * H * W / dtm / 1e6, 'unit': UNIT, 'cores': min(procs, nmp),
                                    'sample': '%d images over %d processes, %.1f s (pool start-up included)' % (nmp, min(procs, nmp), dtm)}
    return out


def cpu_baseline(scene, grad_pixels, sample_images, threads=None, min_seconds=10.0):
    """fwd+bwd of the CPU oracle (a port of the reference path) on `sample_images` images of the workload,
    repeated until at least `min_seconds` of wall time have been spent (first pass untimed: page faults)."""
    from oracle import oracle
    if not threads:
        try:
            threads = len(os.sched_getaffinity(0))
        except AttributeError:
            threads = os.cpu_count() or 1
    n = min(sample_images, scene['background'].shape[0])
    threads = max(1, threads)   # the oracle splits the work over images and, with fewer images than threads, bands of rows
    oracle.set_threads(threads)
    sub = {k: np.ascontiguousarray(v[:n]) for k, v in scene.items()}
    gp = np.ascontiguousarray(grad_pixels[:n])

    def one_pass():
        pixels = oracle.forward(**sub)
        oracle.backward(sub['vertices'], sub['faces'], pixels, gp)

    one_pass()
    t0 = time.perf_counter()
    reps = 0
    while True:
        one_pass()
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds or reps >= 200:
            break
    H, W = scene['background'].shape[1:3]
    return reps * n * H * W / dt / 1e6, n, reps, dt, oracle.threads()


def run_ours(args):
    import torch
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device (there is no CPU fallback for the product path)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {'node': None, 'cpus': None}
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device, timeout=datetime.timedelta(seconds=120))
    from dirt_b200 import build as lib_build, scenes
    if rank == 0 and lib_build.is_stale():   # the bench times the library build() made; it never compiles into the tree
        sys.stderr.write('bench: %s is missing or older than its sources: run build() first\n' % lib_build.SO_PATH)
    if world > 1:
        dist.barrier()

    gen, kwargs, desc = WORKLOADS[args.workload]
    kwargs = dict(kwargs)
    if args.batch:
        kwargs['batch'] = args.batch
    if 'seed' not in kwargs and args.workload != 'cfg2':
        kwargs['seed'] = 1 + rank  # every rank renders different poses
    scene = getattr(scenes, gen)(**kwargs)
    if args.background == 'uniform':   # BASELINE's workloads use a zero background; this variant rules out any zero-data effect
        scene['background'] = np.random.default_rng(100 + rank).uniform(size=scene['background'].shape).astype(np.float32)
    prep = PreparedStep(scene, device)
    B, H, W, C, V, F = prep.dims

    def sync_all():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(device)

    prep.local_step()
    if not args.no_graph:
        prep.capture()
    prep.setup_exchange(world, args.collective)
    for _ in range(max(args.warmup, 3)):
        prep.step(world)
    prep.drain()
    sync_all()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    token = torch.zeros(1, device=device)

    def align_streams():
        # The host leaves dist.barrier() up to ~1 ms apart across 8 ranks (measured: profiles/r02e_scale_n8_diagnostics.txt);
        # a rank that starts early then waits, inside its timed region, for the late starter's first exchange.  A tiny
        # all-reduce ENQUEUED on the stream (no host wait) completes on all ranks together: the start events that follow
        # it in stream order are recorded within microseconds of each other, whatever the hosts do.
        if world > 1:
            dist.all_reduce(token)

    sync_all()
    align_streams()
    start.record()
    launches = 0
    for _ in range(args.steps):
        launches += prep.step(world)
    prep.drain()   # the last steps' all-reduces finish inside the timed region
    stop.record()
    sync_all()
    elapsed_ms = start.elapsed_time(stop)
    if args.dump_outputs and rank == 0:   # before anything below overwrites the buffers of the last timed step
        dump_outputs(prep, prep.parity ^ 1, args.dump_outputs)
    # keep the GPU busy a little longer so the clock sampler sees the loaded state even for short runs
    if sampler:   # rank 0 only: no collectives in here
        t_end = time.time() + 0.6
        while time.time() < t_end:
            prep.forward()
            prep.backward()
        torch.cuda.synchronize(device)
    clocks = sampler.finish() if sampler else None
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=device)
    multi = None
    if world > 1:
        # what limits the N-GPU step: every rank's own time for the timed region, and the same K steps with the
        # all-reduce left out (all ranks still running at once), each as the list over ranks
        local_start, local_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        align_streams()
        local_start.record()
        for _ in range(args.steps):
            prep.step(1)
        local_stop.record()
        sync_all()
        mine = torch.tensor([elapsed_ms / args.steps, local_start.elapsed_time(local_stop) / args.steps], dtype=torch.float64, device=device)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        multi = {'per_rank_ms_per_step': [round(float(e[0]), 5) for e in every],
                 'per_rank_ms_per_step_without_all_reduce': [round(float(e[1]), 5) for e in every]}
        if prep.peer is not None:
            # the peer-memory sum against NCCL's all-reduce of the same local buffers (outside the timed region)
            prep.parity = 0
            prep.step(world)
            prep.drain()
            torch.cuda.synchronize(device)
            want = prep.shared_flat[0].clone()
            dist.all_reduce(want, op=dist.ReduceOp.SUM)
            got = prep.reduced_flat[0]
            scale = float(want.abs().max().item()) + 1e-30
            err = float((got - want).abs().max().item()) / scale
            same = got.clone()
            dist.broadcast(same, src=0)
            multi['peer_exchange_check'] = {'max_err_over_max_abs_vs_nccl': err, 'ok': bool(err < 1e-5),
                                            'bit_identical_to_rank0': bool(torch.equal(same, got))}
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * B * H * W / (ms_per_step * 1e-3) / 1e6

    # per-phase and per-kernel timings (separate loops, same buffers; inputs exceed L2 so no flush is needed)
    def time_phase(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(device)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(device)
        return e0.elapsed_time(e1) / n

    n_phase = max(3, min(args.steps, 20))
    fwd_ms = time_phase(prep.forward, n_phase)
    bwd_ms = time_phase(prep.backward, n_phase)

    def time_kernel(which, fn, n):
        prep.lib.dirt_kernel_timer_enable(which)
        total = 0.0
        for _ in range(n):
            fn()
            total += float(prep.lib.dirt_kernel_timer_elapsed_ms())
        prep.lib.dirt_kernel_timer_enable(0)
        return total / n

    k_fwd_ms = time_kernel(1, prep.forward, n_phase)
    k_bwd_ms = time_kernel(2, prep.backward, n_phase)

    # end to end with host buffers
    e2e = None
    if not args.no_e2e:
        host = HostStep(prep, chunks=args.e2e_chunks)
        for _ in range(2):
            host.step()
        sync_all()
        n_e2e = max(2, min(args.steps, 5))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_e2e):
            host.step()
        e1.record()
        sync_all()
        te = torch.tensor([e0.elapsed_time(e1) / n_e2e], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_ms = float(te.item())
        # the transfers alone (same buffers, no kernels): what the PCIe link of this box allows
        host.copies_only()
        sync_all()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(n_e2e):
            host.copies_only()
        c1.record()
        sync_all()
        copy_ms = c0.elapsed_time(c1) / n_e2e
        e2e = {'value': world * B * H * W / (e2e_ms * 1e-3) / 1e6, 'unit': UNIT, 'ms_per_step': e2e_ms,
               'h2d_bytes_per_step': int(host.h2d), 'd2h_bytes_per_step': int(host.d2h),
               'transfers_only_ms': copy_ms, 'chunks': int(host.runner.chunks)}
        del host

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    os.sched_setaffinity(0, full_affinity)   # the CPU legs below (oracle) use every host thread again
    checked = None
    if args.check:   # default on; outside the timed region; never lets a checker problem take the bench line down
        try:
            checked = check_against_oracle(prep, scene)
        except Exception as e:
            checked = {'ok': False, 'error': '%s: %s' % (type(e).__name__, e)}

    peak, peak_src = measured_peak_gbs()
    fwd_bytes, bwd_bytes = algorithmic_bytes(B, H, W, C, V, F)
    if k_bwd_ms >= k_fwd_ms:
        dom, dom_ms, dom_bytes = 'backward_kernel', k_bwd_ms, bwd_bytes
    else:
        dom, dom_ms, dom_bytes = 'raster_kernel(forward)', k_fwd_ms, fwd_bytes
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:   # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            tr = json.load(f).get(args.workload, {}).get('backward' if dom == 'backward_kernel' else 'forward')
        if tr:
            traffic, traffic_src = tr['dram_bytes'], tr['source']
            cap = tr.get('images')   # the capture ran a smaller batch than this launch: per-launch traffic scales with it
            if cap and cap != B:
                traffic = int(traffic * B / cap)
                traffic_src += ' (captured at %d images per launch, scaled x%g to this launch of %d)' % (cap, B / cap, B)
    except Exception:
        pass
    roofline = {'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src, 'algorithmic_bytes_per_launch': int(dom_bytes),
                'kernel_ms': dom_ms,
                'forward_kernel': {'ms': k_fwd_ms, 'algorithmic_bytes': int(fwd_bytes), 'gbs': fwd_bytes / (k_fwd_ms * 1e-3) / 1e9},
                'backward_kernel': {'ms': k_bwd_ms, 'algorithmic_bytes': int(bwd_bytes), 'gbs': bwd_bytes / (k_bwd_ms * 1e-3) / 1e9},
                'step': {'ms': ms_per_step, 'algorithmic_bytes': int(fwd_bytes + bwd_bytes),
                         'gbs': (fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9,
                         'frac': (fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9 / peak}}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        mpix, n_img, reps, dt, threads = cpu_baseline(scene, prep.grad_pixels_host, args.cpu_sample)
        cpu = {'value': mpix, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'host': host_record(),
               'sample': 'oracle/dirt_oracle.c (OpenMP over images x row bands) fwd+bwd on the first %d images of the workload, '
                         '%d passes in %.1f s' % (n_img, reps, dt)}
        if not args.no_numpy_baseline:
            cpu['variants'] = numpy_baselines(scene, prep.grad_pixels_host, threads)
            cpu['variants']['c_openmp'] = {'value': mpix, 'unit': UNIT, 'cores': threads}

    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': desc, 'name': args.workload, 'batch_per_gpu': B, 'global_batch': B * world, 'height': H, 'width': W,
                   'channels': C, 'vertices': V, 'faces': F, 'parallelism': 'batch-sharded x%d' % world,
                   'collective': prep.collective,
                   'vertex_gradients': 'accumulated over the batch in the backward kernel (DIRT_BWD_SHARED_GEOMETRY)',
                   'background': args.background,
                   'l2': 'inputs larger than L2 (%.0f MB touched per step)' % ((fwd_bytes + bwd_bytes) / 1e6)},
        'phases_ms': {'forward_call': fwd_ms, 'backward_call': bwd_ms},
        'gpu_launches': int(launches), 'gpu_launches_per_step': int(prep.launches_per_step), 'cuda_graph': prep.graphs is not None,
        'clocks': clocks, 'roofline': roofline, 'numa': numa,
    }
    if multi:
        out['multi_gpu'] = multi
    if checked is not None:
        out['checked'] = checked['ok']
        out['check'] = checked
    if e2e:
        out['e2e'] = e2e
    if cpu:
        out['cpu_baseline'] = cpu
    emit(out)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
# reference arm: the CPU port of the reference path (the reference's GL/TF op cannot run in this image)
# ---------------------------------------------------------------------------------------------------------

def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if rank != 0:
        return
    from dirt_b200 import scenes
    from oracle import oracle
    oracle.build()
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 for its workers)
    try:
        host_threads = len(os.sched_getaffinity(0))
    except AttributeError:
        host_threads = os.cpu_count() or 1
    gen, kwargs, desc = WORKLOADS[args.workload]
    kwargs = dict(kwargs)
    sample = min(args.cpu_sample, kwargs.get('batch', 1))
    oracle.set_threads(max(1, host_threads))   # work items are images x row bands: every host thread gets work
    kwargs['batch'] = sample if 'batch' in kwargs else None
    if kwargs.get('batch') is None:
        kwargs.pop('batch', None)
    if args.workload != 'cfg2':
        kwargs['seed'] = 1
    scene = getattr(scenes, gen)(**kwargs)
    B, H, W, C = scene['background'].shape
    V, F = scene['vertices'].shape[1], scene['faces'].shape[1]
    gp = np.random.default_rng(2).standard_normal((B, H, W, C)).astype(np.float32)

    def step():
        pixels = oracle.forward(**scene)
        oracle.backward(scene['vertices'], scene['faces'], pixels, gp)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = B * H * W / dt / 1e6
    threads = oracle.threads()
    out = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': desc, 'name': args.workload, 'sample_images_per_step': B, 'height': H, 'width': W, 'channels': C,
                   'vertices': V, 'faces': F,
                   'note': 'the reference OpenGL/TensorFlow op cannot run in this image; this is the CPU port of its path '
                           '(oracle/dirt_oracle.c, OpenMP over images x row bands, all host threads) on a bounded sample of the same workload'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'host': host_record(),
                         'sample': '%d images of the workload per step, %d steps' % (B, args.steps),
                         'variants': None if args.no_numpy_baseline else numpy_baselines(scene, gp, host_threads)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(out)


_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner under
    torchrun), so file descriptor 1 is pointed at stderr for the duration of the run and the line goes to the saved one."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + '\n').encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, line)
    else:
        os.write(_JSON_FD, line)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg3', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='override the per-GPU batch (debugging)')
    ap.add_argument('--cpu-sample', type=int, default=64, help='images the CPU baseline renders per pass')
    ap.add_argument('--background', default='zeros', choices=['zeros', 'uniform'], help='background values (BASELINE: zeros)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--collective', choices=['auto', 'peer', 'nccl'], default='auto',
                    help='N>1: sum of the shared-geometry gradient over ranks by the library\'s peer-memory kernel (peer), by NCCL '
                         '(nccl), or the first that is available (auto)')
    ap.add_argument('--no-graph', action='store_true', help='launch every step call by call instead of replaying a CUDA graph')
    ap.add_argument('--e2e-chunks', type=int, default=12, help='batch chunks of the host copy/compute pipeline')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-numpy-baseline', action='store_true', help='skip the numpy variants of the CPU baseline')
    ap.add_argument('--check', dest='check', action='store_true', default=True,
                    help='after timing, validate the benched buffers against the CPU oracle ("checked": true); on by default')
    ap.add_argument('--no-check', dest='check', action='store_false', help='skip that validation')
    ap.add_argument('--no-numa-bind', action='store_true', help='do not pin the process to the NUMA node of its GPU')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last one computed to DIR/<name>.npy '
                                                           '(float32/float64, at most 64 MB: a fixed sample of the pixels)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
