#!/usr/bin/env python
"""Benchmark of the message-passing hot path (graph construction + MOTMPNet core forward).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # + the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic frame windows of
BASELINE.json configs[1] shape (15 frames x 150 detections, k=50, 12 message-passing steps):
ReID-distance KNN graph build + edge features, node/edge encoders, 12 fused MP steps with the
edge classifier.  Each GPU holds `--graphs` windows (weak scaling; windows are independent, no
collective).  Metric: edge-updates/s = 12 * directed edges processed / time.

Inputs are larger than L2 (node features x are [N,2048,8,4] fp32 = 590 MB per window).
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if __name__ == '__main__':
    # a benchmark run writes nothing into the source tree it runs from, bytecode caches of the modules it imports
    # included, so that a shared or read-only checkout stays exactly as the build left it
    sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from mpntrackseg_b200 import synth  # noqa: E402
from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params  # noqa: E402

METRIC = 'edge-updates/s'
UNIT = 'edge-updates/s'
NUM_STEPS_MP = 12
NUM_CLASS_STEPS = 11
DUMP_BYTES = 64_000_000


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--graphs', type=int, default=16, help='frame windows per GPU per step')
    ap.add_argument('--frames', type=int, default=15)
    ap.add_argument('--dets', type=int, default=150)
    ap.add_argument('--k', type=int, default=50)
    ap.add_argument('--pooled', action='store_true', help='node features already pooled [N,2048]')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--job-graphs', type=int, default=0,
                    help='configs[2]: a fixed job of this many windows split over the GPUs (strong scaling): every rank takes '
                         'job/world windows per step (overrides --graphs); use with --pooled (512 raw windows are 302 GB)')
    ap.add_argument('--mode', default='infer', choices=['infer', 'train'],
                    help="'train': BASELINE configs[3] -- KITTI-shaped training step (fwd+bwd, 12 MP steps, 11 classified) "
                         'with one NCCL all-reduce of the flat gradient bucket + Adam; extra to the headline contract')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned (edge_index, edge_attr, '
                         f'logits, pair_ptr) as DIR/<name>.npy, at most {DUMP_BYTES // 10**6} MB in all (rank 0 only)')
    a = ap.parse_args(argv)
    if a.steps < 1 or a.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if a.dump_outputs and (a.impl != 'b200' or a.mode != 'infer'):
        ap.error('--dump-outputs records the b200 inference step only')
    return a


def workload_name(a):
    feats = 'x[N,2048]' if a.pooled else 'x[N,2048,8,4]'
    if a.job_graphs:
        return (f'configs[2]: job of {a.job_graphs} independent windows T={a.frames} D={a.dets} k={a.k}, {NUM_STEPS_MP} MP steps, '
                f'{feats}, full forward incl. ReID-distance KNN build; sharded over the GPUs')
    return (f'configs[1]: MOTS20-scale windows T={a.frames} D={a.dets} k={a.k}, {NUM_STEPS_MP} MP steps, '
            f'{feats}, full forward incl. ReID-distance KNN build; {a.graphs} windows per GPU per step')


def config_dict(a, world):
    """The `config` object of the JSON line; identical in both arms (--impl b200 / reference)."""
    return {'workload': workload_name(a),
            'parallelism': f'independent windows sharded over {world} GPU(s), no collective',
            'l2_policy': 'inputs larger than L2 (node features 590 MB per window)' if not a.pooled
            else 'pooled inputs (18 MB per window); MP state is L2-resident by nature'}


def pin_to_gpu_numa(gpu_index):
    """Bind this rank to the CPUs NVML reports as local to its GPU BEFORE any page-locked buffer is allocated,
    so that the host side of every H2D copy reads node-local memory."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1 and 64 * i + b < ncpu}
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def make_windows(a, rank, world):
    """This rank's slice of the job's world*graphs windows (weak scaling: --graphs per GPU)."""
    from mpntrackseg_b200.sharding import shard_range
    lo, hi = shard_range(a.graphs * world, rank, world)
    wins = []
    cache = {}
    for g in range(lo, hi):
        seed = g % 128 if a.job_graphs else g          # a 512-window job reuses 128 distinct windows (host generation time)
        if seed not in cache:
            # (the k-boundary gap the parity fixtures enforce cannot be reached for very dense windows; timing does not need it)
            cache[seed] = synth.make_window(T=a.frames, D=a.dets, k=a.k, seed=seed, node_feats='pooled', node_dim=8,
                                            min_gap=1e-5 if a.dets <= 200 else 0)
        wins.append(cache[seed])
    return wins


def job_inputs(a, rank, world, dev):
    """This rank's windows, their node offsets ``node_ptr`` and inputs: the detection table ``cols``, its page-locked
    copy ``host`` and device copy ``devin``, both with one node-feature tensor per window (seeded by the rank)."""
    wins = make_windows(a, rank, world)
    gen = torch.Generator(device=dev).manual_seed(rank)
    node_ptr = [0]
    for w in wins:
        node_ptr.append(node_ptr[-1] + w.N)
    # the job's detection table: one set of columns for all windows (the way the reference holds a
    # sequence's graph_df) + one node-feature tensor per window
    cols = {k: torch.cat([torch.from_numpy(synth.det_columns(w)[k]) for w in wins])
            for k in ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')}
    for g in range(len(wins)):                      # one table for the job: window g owns its own frame numbers
        cols['frame'][node_ptr[g]:node_ptr[g + 1]] += g * (a.frames + 1)
    cols['reid'] = torch.cat([w.reid for w in wins])
    host = {k: v.pin_memory() for k, v in cols.items()}
    devin = {k: v.to(dev) for k, v in host.items()}
    host['x'], devin['x'] = [], []
    for w in wins:
        shape = (w.N, 2048) if a.pooled else (w.N, 2048, 8, 4)
        x = torch.randn(shape, generator=gen, device=dev).abs_()
        devin['x'].append(x)
        host['x'].append(x.cpu().pin_memory())
    return wins, node_ptr, cols, host, devin


def model_and_params():
    mp = default_graph_model_params(NUM_STEPS_MP, NUM_CLASS_STEPS)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    return mp, P


def dump_outputs(out_dir, batch, out, budget=DUMP_BYTES):
    """Write one step's results as ``out_dir/<name>.npy``: the graph batch's ``edge_index`` [2,E], ``edge_attr``
    [E,F] and ``pair_ptr``, and the classifier ``logits`` [num_class_steps,E].  Indices are stored as float64
    (exact), the rest as the float32 it was computed in.  When the files would exceed ``budget`` bytes, every
    per-edge array keeps the same seeded sample of edges; ``edge_sample.npy`` holds the sorted edge ids kept."""
    edge_index = batch.edge_index.cpu().numpy().astype(np.float64)
    edge_attr = batch.edge_attr.cpu().numpy()
    logits = out.logits.cpu().numpy()
    pair_ptr = np.asarray(batch.pair_ptr, dtype=np.float64)
    num_edges = edge_index.shape[1]
    per_edge = edge_index.itemsize * 2 + edge_attr.itemsize * edge_attr.shape[1] + logits.itemsize * logits.shape[0] + 8
    headers = 5 * 1024                  # 1 KB per file for its .npy header (128 bytes for these shapes)
    keep = min(num_edges, max(0, (budget - headers - pair_ptr.nbytes) // per_edge))
    sample = np.arange(num_edges) if keep == num_edges else \
        np.sort(np.random.default_rng(0).choice(num_edges, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(edge_index=edge_index[:, sample], edge_attr=edge_attr[sample], logits=logits[:, sample],
                  pair_ptr=pair_ptr, edge_sample=sample.astype(np.float64))
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), np.ascontiguousarray(arr))


# ------------------------------------------------------------------ reference arm (CPU)
def oracle_step(win, x, ds, mp, P):
    """The reference algorithm for one window on the host: graph build + core forward."""
    from oracle import graph_ref, mpn_ref
    g = graph_ref.build_graph(win.frame, win.reid, synth.det_columns(win), win.fps, ds)
    with torch.no_grad():
        out = mpn_ref.mpn_forward(P, mp, x, g['edge_index'], g['edge_attr'])
    return g['edge_index'].shape[1], out['classified_edges'][-1]


def cpu_sample(a, steps, warmup):
    """Time the oracle (kind 'port': CPU-PyTorch restatement of the reference, which is itself
    CPU PyTorch) on one window per step with all host threads."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ds = default_dataset_params(top_k_nns=a.k, frames_per_graph=a.frames)
    mp, P = model_and_params()
    win = synth.make_window(T=a.frames, D=a.dets, k=a.k, seed=0, node_feats='pooled', node_dim=8,
                            min_gap=1e-5 if a.dets <= 200 else 0)
    gen = torch.Generator().manual_seed(0)
    shape = (win.N, 2048) if a.pooled else (win.N, 2048, 8, 4)
    x = torch.randn(shape, generator=gen).abs_()
    for _ in range(warmup):
        oracle_step(win, x, ds, mp, P)
    t0 = time.perf_counter()
    edges = 0
    for _ in range(steps):
        e, _ = oracle_step(win, x, ds, mp, P)
        edges += e
    dt = time.perf_counter() - t0
    return dict(value=NUM_STEPS_MP * edges / dt, unit=UNIT, cores=cores, kind='port',
                sample=f'{steps} x 1 window (N={win.N}, E={edges // max(steps, 1)}) of the same workload, '
                       f'oracle graph build + core forward, {dt / max(steps, 1) * 1e3:.0f} ms/window'), dt / max(steps, 1)


def run_reference(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    base, ms = cpu_sample(a, a.steps, a.warmup)
    line = dict(impl='reference', metric=METRIC, value=base['value'], unit=UNIT, n_gpus=a.gpus, steps=a.steps,
                warmup=a.warmup, ms_per_step=ms * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic', config=config_dict(a, a.gpus),
                cpu_baseline=base,
                e2e=dict(value=base['value'], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                graphs_per_s=1.0 / ms)
    print(json.dumps(line))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from a background thread DURING the timed
    region (an `nvidia-smi -lms` subprocess was found to slow the timed loop down through driver locks)."""

    def __init__(self, gpu_index, period=0.02):
        import threading
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), 0, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            return
        self.period = period
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        names = {'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown,
                 'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        if not self.ok:
            return None
        self._stop.set()
        self.t.join(timeout=2)
        if not self.samples:
            return None
        sm = sorted(self.samples)
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons), samples=len(sm))


# ------------------------------------------------------------------ this repo's arm
def run_b200(a):
    import torch.distributed as dist
    from mpntrackseg_b200 import _cabi
    from mpntrackseg_b200.models.mpn import MOTMPNet

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    pin_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _cabi.lib()

    ds = default_dataset_params(top_k_nns=a.k, frames_per_graph=a.frames)
    mp, P = model_and_params()
    model = MOTMPNet(mp).to(dev).eval()
    model.load_state_dict(P, strict=False)      # core weights; the mask branch keeps its init

    wins, node_ptr, cols, host, devin = job_inputs(a, rank, world, dev)
    fps = wins[0].fps
    h2d_bytes = sum(t.numel() * t.element_size() for k, t in host.items() if k != 'x') + \
        sum(t.numel() * t.element_size() for t in host['x'])

    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import build_graph_batch

    def step(inputs):
        """One pass of the hot path over the GPU's windows: batched KNN graph build + edge features,
        node / edge encoders, 12 MP steps + classifier (block-diagonal batch)."""
        batch = build_graph_batch(inputs, node_ptr, ds, fps, device=dev)
        with torch.no_grad():
            out = model.forward_batch(batch)
        return batch, out

    copy_stream = torch.cuda.Stream(device=dev)

    def step_e2e_raw():
        """Raw-map arm (second number): the reference's stored [N,2048,8,4] node-core maps go host -> device every
        step (9.5 GB per 16 windows) and are pooled on the GPU; PCIe-bound by construction."""
        main = torch.cuda.current_stream()
        events = []
        with torch.cuda.stream(copy_stream):
            inputs = {k: v.to(dev, non_blocking=True) for k, v in host.items() if k != 'x'}
            small = torch.cuda.Event()
            small.record(copy_stream)
            inputs['x'] = []
            for hx in host['x']:
                inputs['x'].append(hx.to(dev, non_blocking=True))
                ev = torch.cuda.Event()
                ev.record(copy_stream)
                events.append(ev)
        main.wait_event(small)
        for v in inputs.values():
            if torch.is_tensor(v):
                v.record_stream(main)
        batch = build_graph_batch(inputs, node_ptr, ds, fps, device=dev)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        pooled = torch.empty((batch.num_nodes, 2048), dtype=torch.float32, device=dev)
        with torch.no_grad():
            for i, (x, ev) in enumerate(zip(inputs['x'], events)):
                main.wait_event(ev)                                   # this window's node features have landed
                x.record_stream(main)
                ops.avgpool(x if x.dim() > 2 else x[:, :, None, None], out=pooled[node_ptr[i]:node_ptr[i + 1]])
            batch.xs = model.encode_pooled(pooled, status=flags)      # one encoder launch for all windows
            out = model.forward_batch(batch, encoded=True)
        res = out.logits[-1].cpu()                                    # D2H of the result (last step's logits)
        assert not flags.any().item(), 'fp16 overflow in the encoder (would need the fp32 rerun)'
        return batch, res

    # ---- end-to-end arm through the embedding store (SURVEY.md f3): the job's windows are written once to a
    #      per-frame store (ReID [n,1+256] and the pooled node-core variant [n,1+2048] of EmbeddingStore.pool) and
    #      packed into page-locked memory (SequenceEmbeddings).  Every timed step copies the detection table, the
    #      ReID vectors and the pooled node-core vectors host -> device, builds the graphs, runs the forward and reads
    #      the last step's logits back; the copy of step i+1 overlaps the compute of step i (two device buffer sets).
    import shutil
    import tempfile
    import pandas as pd
    from mpntrackseg_b200.data.embedding_store import EmbeddingStore, SequenceEmbeddings
    tmp = tempfile.mkdtemp(prefix=f'mpn_store_r{rank}_', dir='/dev/shm' if os.path.isdir('/dev/shm') else None)
    seq_info = {'seq_path': tmp, 'det_file_name': 'synthetic_det', 'fps': fps}
    dsx = dict(ds, reid_embeddings_dir='reid', node_core_embeddings_dir='node_core', node_ext_embeddings_dir=None)
    store = EmbeddingStore(seq_info)
    n_tot = node_ptr[-1]
    table = {k: cols[k].numpy().copy() for k in ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')}
    table['detection_id'] = np.arange(n_tot, dtype=np.int64)
    det_df = pd.DataFrame(table)
    store.write('reid', table['frame'], table['detection_id'], cols['reid'])
    # the pooled store (what EmbeddingStore.pool writes from the reference's [n,1+2048,8,4] files; here the maps are
    # already on the device, so they are pooled there by the same kernel and only the pooled frames are written)
    pooled_rows = torch.cat([x if x.dim() == 2 else ops.avgpool(x) for x in devin['x']]).cpu()
    store.write('node_core_pooled', table['frame'], table['detection_id'], pooled_rows)
    del pooled_rows
    seq = SequenceEmbeddings(det_df, seq_info, dsx, pooled=True, pin_memory=True)
    shutil.rmtree(tmp, ignore_errors=True)
    host_tab = {k: torch.from_numpy(table[k]).pin_memory() for k in ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')}
    e2e_host = dict(host_tab, reid=seq.reid, x=seq.node_core)
    e2e_h2d = sum(t.numel() * t.element_size() for t in e2e_host.values())
    bufsets = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in e2e_host.items()} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]
    out_host = [None, None]

    def e2e_upload(i):
        b = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(free[b])                           # the compute that last read this buffer set is done
            for k, v in e2e_host.items():
                bufsets[b][k].copy_(v, non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_pipeline(steps):
        main = torch.cuda.current_stream()
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        for b in range(2):
            free[b].record(main)
        e2e_upload(0)
        for i in range(steps):
            b = i & 1
            if i + 1 < steps:
                e2e_upload(i + 1)
            main.wait_event(ready[b])
            inputs = bufsets[b]
            batch = build_graph_batch(inputs, node_ptr, ds, fps, device=dev)
            with torch.no_grad():
                batch.xs = model.encode_pooled(inputs['x'], status=flags)
                out = model.forward_batch(batch, encoded=True)
            free[b].record(main)
            last = out.logits[-1]
            if out_host[b] is None or out_host[b].shape != last.shape:
                out_host[b] = torch.empty(last.shape, dtype=last.dtype).pin_memory()
            out_host[b].copy_(last, non_blocking=True)                 # D2H of the step's result
        torch.cuda.synchronize()
        assert not flags.any().item(), 'fp16 overflow in the encoder (would need the fp32 rerun)'
        return out_host[(steps - 1) & 1]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # every loop keeps its last step's result alive, so the timed loop runs with the memory pool the warmup left
    for _ in range(a.warmup):
        last = step(devin)
    torch.cuda.synchronize()

    # ---- timed region: device-resident inputs (Python's cyclic GC is paused: a gen-2 collection inside
    #      a 7 ms step shows up as a 20-40 ms outlier)
    import gc
    gc.collect()
    gc.disable()
    sampler = ClockSampler(local) if rank == 0 and not os.environ.get('MPN_BENCH_NO_SAMPLER') else None
    lib.mpn_profile_begin()
    launches0 = lib.mpn_launch_count()
    sync_all()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.steps):
        last = step(devin)
    ev1.record()
    sync_all()
    ms = ev0.elapsed_time(ev1)
    edges = last[0].num_edges
    nodes = last[0].num_nodes
    launches = lib.mpn_launch_count() - launches0
    import ctypes as C
    prof_ms = (C.c_double * 2)()
    prof_n = (C.c_longlong * 2)()
    lib.mpn_profile_end(prof_ms, prof_n)
    clocks = sampler.stop() if sampler else None

    # ---- end to end: pinned host buffers in, logits out, copies inside the timed region
    e2e_pipeline(max(2, a.warmup))
    sync_all()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    res = e2e_pipeline(a.steps)
    t1.record()
    sync_all()
    ms_e2e = t0.elapsed_time(t1)
    d2h = res.numel() * res.element_size()
    # parity of the store arm with the device-resident arm on the same windows (same kernels, same inputs)
    with torch.no_grad():
        ref_last = step(devin)[1].logits[-1].cpu()
    e2e_max_diff = float((res - ref_last).abs().max())
    # bit-identical on the tensor-core path; if the forward fell back to the fp32 kernels (state beyond the scaled fp16
    # range) the device arm also re-encodes the nodes in fp32 while this arm keeps its tensor-core encoding: rounding level
    assert e2e_max_diff <= 1e-5 * max(1.0, float(ref_last.abs().max())), \
        f'store arm and device-resident arm disagree by {e2e_max_diff}'

    # ---- second number: raw [N,2048,8,4] maps from pinned memory every step (the round-1 e2e definition)
    raw_steps = min(a.steps, 5)
    ms_raw = None
    if not a.pooled:
        for _ in range(2):
            step_e2e_raw()
        sync_all()
        t0.record()
        for _ in range(raw_steps):
            step_e2e_raw()
        t1.record()
        sync_all()
        ms_raw = t0.elapsed_time(t1)
    gc.enable()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, *last)

    from mpntrackseg_b200.sharding import reduce_step_stats
    ms, (all_edges, all_nodes, h2d_total, d2h_total, h2d_raw_total) = reduce_step_stats(
        ms, [edges, nodes, e2e_h2d, d2h, h2d_bytes], device=dev)
    ms_e2e, _ = reduce_step_stats(ms_e2e, [0], device=dev)
    if ms_raw is not None:
        ms_raw, _ = reduce_step_stats(ms_raw, [0], device=dev)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except OSError:
            pass
        peak = float(peaks.get('hbm_gbs', 6650.0))
        edge_launches = max(int(prof_n[0]), 1)
        # algorithmic bytes of one mp_edge_kernel launch (DESIGN.md section 4):
        # per directed edge 200 B (e_init 64 + e 64 + e' 64 + row/col idx 8) + 4 B logit on classified
        # steps; per node x_init + x_lat read once = 256 B.
        cls_frac = NUM_CLASS_STEPS / NUM_STEPS_MP
        bytes_per_launch = edges * (200 + 4 * cls_frac) + nodes * 256
        avg_ms = float(prof_ms[0]) / edge_launches
        achieved = bytes_per_launch / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        # DRAM traffic of the dominant kernel: only a capture of THIS workload size counts (ncu --set full of the same
        # command, summarised in profiles/); otherwise null
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'r02_mp_edge_traffic.json')))
            if os.environ.get('MPN_ENGINE', 'auto') != 'fp32' and int(tr['edges']) == int(edges):
                traffic = float(tr['dram_bytes_per_launch'])
        except (OSError, KeyError, ValueError):
            pass
        kernel = 'mp_edge_tc3_kernel' if os.environ.get('MPN_ENGINE', 'auto') != 'fp32' else 'mp_edge_kernel'
        per_s = lambda t_ms, n_steps: NUM_STEPS_MP * all_edges * n_steps / (t_ms * 1e-3)
        line = dict(
            metric=METRIC, value=per_s(ms, a.steps), unit=UNIT, n_gpus=world,
            steps=a.steps, warmup=a.warmup, ms_per_step=ms / a.steps, higher_is_better=True,
            scaling='strong' if a.job_graphs else 'weak',
            vs_baseline=None, dtype='f32', data='synthetic', config=config_dict(a, world),
            edges_per_gpu=edges, nodes_per_gpu=nodes,
            graphs_per_s=a.graphs * world * a.steps / (ms * 1e-3),
            e2e=dict(value=per_s(ms_e2e, a.steps), unit=UNIT,
                     h2d_bytes_per_step=int(h2d_total), d2h_bytes_per_step=int(d2h_total),
                     graphs_per_s=a.graphs * world * a.steps / (ms_e2e * 1e-3), ms_per_step=ms_e2e / a.steps,
                     source='pooled embedding store (EmbeddingStore.pool -> SequenceEmbeddings, page-locked): detection '
                            'table + ReID [N,256] + node-core [N,2048] host->device every step, last-step logits read '
                            'back; step i+1 uploads while step i computes',
                     max_abs_diff_vs_device_arm=e2e_max_diff),
            gpu_launches=int(launches),
            roofline=dict(bound='hbm', kernel=kernel, achieved=achieved, peak=peak, unit='GB/s',
                          frac=achieved / peak if peak else None, traffic=traffic, algorithmic_bytes=bytes_per_launch,
                          peak_source='MEASURED_PEAKS.json hbm_gbs' if peaks else 'fallback 6650 GB/s',
                          avg_launch_ms=avg_ms, launches=edge_launches,
                          node_kernel_avg_launch_ms=float(prof_ms[1]) / max(int(prof_n[1]), 1),
                          mp_phase_edge_updates_per_s=edges * edge_launches / (float(prof_ms[0] + prof_ms[1]) * 1e-3)
                          if prof_ms[0] > 0 else None),
            clocks=clocks)
        if ms_raw is not None:
            line['e2e_raw_maps'] = dict(value=per_s(ms_raw, raw_steps), unit=UNIT, h2d_bytes_per_step=int(h2d_raw_total),
                                        steps=raw_steps, ms_per_step=ms_raw / raw_steps,
                                        source='reference layout [N,2048,8,4] maps host->device every step, pooled on the GPU')
        if not a.no_cpu_baseline and world == 1:
            base, _ = cpu_sample(a, steps=3, warmup=1)
            line['cpu_baseline'] = base
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------ training config (BASELINE configs[3])
def run_train(a):
    import torch.distributed as dist
    from mpntrackseg_b200 import _cabi
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    from mpntrackseg_b200.models.mpn import MOTMPNet
    from mpntrackseg_b200.sharding import reduce_step_stats
    from mpntrackseg_b200.training import CoreTrainer
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (('RANK', 0), ('WORLD_SIZE', 1), ('LOCAL_RANK', 0)))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    ds = default_dataset_params(top_k_nns=100, frames_per_graph=20)
    mp = default_graph_model_params(NUM_STEPS_MP, NUM_CLASS_STEPS)
    P = synth.make_params(mp, seed=6, gain=0.95, core_only=True)
    model = MOTMPNet(mp).to(dev)
    model.load_state_dict(P, strict=False)
    tr = CoreTrainer(model)
    w = synth.make_window(T=20, D=8, k=100, seed=100 + rank)
    g = MOTGraph.from_tensors(synth.det_columns(w), w.reid, w.x.to(dev), None, {'fps': w.fps}, ds).construct_graph_object()
    ident = w.ident.to(dev)
    labels = (ident[g.edge_index[0]] == ident[g.edge_index[1]]).float()
    lib = _cabi.lib()

    def timed(fn, steps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return e0.elapsed_time(e1), out

    # eager: every kernel launched from Python (the step is launch-bound); graphed: the same step captured once as a
    # CUDA graph (kernels + NCCL all-reduce + Adam) and replayed -- the headline number of this mode
    for _ in range(a.warmup):
        tr.train_step(g, labels)
    l0 = lib.mpn_launch_count()
    tr.train_step(g, labels)
    launches_per_step = int(lib.mpn_launch_count() - l0)
    ms_eager, _ = timed(lambda: tr.train_step(g, labels), max(3, min(a.steps, 10)))
    ms_eager /= max(3, min(a.steps, 10))
    for _ in range(a.warmup):
        tr.graphed_step(g, labels)
    ms, loss = timed(lambda: tr.graphed_step(g, labels), a.steps)
    ms, (edges,) = reduce_step_stats(ms, [g.edge_index.shape[1]], device=dev)
    ms_eager, _ = reduce_step_stats(ms_eager, [0], device=dev)
    if rank == 0:
        line = dict(metric='edge-updates/s (training step: fwd+bwd+all-reduce+Adam)', value=NUM_STEPS_MP * edges * a.steps / (ms * 1e-3),
                    unit=UNIT, n_gpus=world, steps=a.steps, warmup=a.warmup, ms_per_step=ms / a.steps, higher_is_better=True,
                    scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                    config={'workload': 'configs[3]: KITTI-shaped window T=20 D=8 k=100 per GPU, 12 MP steps, 11 classified, '
                                        'weighted BCE, one summed all-reduce of the 1.19 MB gradient bucket, Adam; the step '
                                        'is one CUDA-graph replay',
                            'parallelism': f'data parallel over {world} GPU(s), one NCCL all-reduce per step'},
                    edges_per_gpu=int(g.edge_index.shape[1]), nodes_per_gpu=int(w.N),
                    gpu_launches=launches_per_step * a.steps, kernels_per_step=launches_per_step,
                    eager_ms_per_step=ms_eager, loss=float(loss))
        if not a.no_cpu_baseline and world == 1:
            from oracle import graph_ref, mpn_ref
            torch.set_num_threads(os.cpu_count() or 1)
            rg = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds)
            lab = (w.ident[rg['edge_index'][0]] == w.ident[rg['edge_index'][1]]).float()
            Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
            def cpu_step():
                out = mpn_ref.mpn_forward(Pg, mp, w.x, rg['edge_index'], rg['edge_attr'])
                mpn_ref.weighted_bce_loss(out['classified_edges'], lab).backward()
            cpu_step()
            t0 = time.perf_counter()
            for _ in range(3):
                cpu_step()
            dt = (time.perf_counter() - t0) / 3
            line['cpu_baseline'] = dict(value=NUM_STEPS_MP * rg['edge_index'].shape[1] / dt, unit=UNIT, cores=os.cpu_count(), kind='port',
                                        sample=f'3 x fwd+bwd (autograd) of the same window on the oracle, {dt * 1e3:.0f} ms each')
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    args = parse()
    if args.job_graphs:
        _world = int(os.environ.get('WORLD_SIZE', '1'))
        assert args.job_graphs % _world == 0, '--job-graphs must be a multiple of the number of GPUs'
        args.graphs = args.job_graphs // _world
    if args.mode == 'train' and args.impl != 'reference':
        run_train(args)
    elif args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)
