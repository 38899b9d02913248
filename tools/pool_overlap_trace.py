"""Per-stream kernel timeline of the bench step (bench.py's inputs: 16 configs[1] windows, x [N,2048,8,4]) under
torch.profiler: which kernels of the other streams run while the node-feature pool runs on its side stream.

    python tools/pool_overlap_trace.py OUT_DIR [--steps 3]

Writes OUT_DIR/pool_overlap.pt.trace.json (chrome trace), OUT_DIR/pool_overlap_timeline.csv (every kernel: step,
stream, start and end in us from the step's first kernel, name) and prints, per step, the pool's span, the kernels of
the other streams that ran inside it and the time the other streams had no kernel inside it (host syncs, launch gaps).
Tracing slows the host: take step times from bench.py, not from this run."""
import argparse
import csv
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

import bench  # noqa: E402
from mpntrackseg_b200.data.mot_graph import build_graph_batch  # noqa: E402
from mpntrackseg_b200.models.mpn import MOTMPNet  # noqa: E402
from mpntrackseg_b200.config import default_dataset_params  # noqa: E402

POOL = 'avgpool_kernel'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('out_dir')
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    a = bench.parse([])
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    ds = default_dataset_params(top_k_nns=a.k, frames_per_graph=a.frames)
    mp, P = bench.model_and_params()
    model = MOTMPNet(mp).to(dev).eval()
    model.load_state_dict(P, strict=False)
    wins, node_ptr, _, _, devin = bench.job_inputs(a, 0, 1, dev)

    def step():
        batch = build_graph_batch(devin, node_ptr, ds, wins[0].fps, device=dev)
        with torch.no_grad():
            return model.forward_batch(batch)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                            torch.profiler.ProfilerActivity.CUDA]) as prof:
        for i in range(args.steps):
            with torch.profiler.record_function(f'step{i}'):
                step()
            torch.cuda.synchronize()
    trace = os.path.join(args.out_dir, 'pool_overlap.pt.trace.json')
    prof.export_chrome_trace(trace)

    ev = json.load(open(trace))['traceEvents']
    kernels = sorted((e for e in ev if e.get('cat') == 'kernel'), key=lambda e: e['ts'])
    steps = sorted((e for e in ev if e.get('cat') == 'gpu_user_annotation' and e['name'].startswith('step')),
                   key=lambda e: e['ts'])
    if not steps and kernels:                   # no step annotations on the device timeline: one span for the run
        steps = [{'ts': kernels[0]['ts'], 'dur': kernels[-1]['ts'] + kernels[-1]['dur'] - kernels[0]['ts'] + 1}]
    rows = []
    for si, s in enumerate(steps):
        ks = [k for k in kernels if s['ts'] <= k['ts'] < s['ts'] + s['dur']]
        if not ks:
            continue
        t0 = ks[0]['ts']
        for k in ks:
            rows.append((si, k['args'].get('stream'), k['ts'] - t0, k['ts'] + k['dur'] - t0, k['name']))
    with open(os.path.join(args.out_dir, 'pool_overlap_timeline.csv'), 'w', newline='') as f:
        w = csv.writer(f)
        w.writerow(['step', 'stream', 'start_us', 'end_us', 'kernel'])
        w.writerows((r[0], r[1], f'{r[2]:.1f}', f'{r[3]:.1f}', r[4]) for r in rows)

    for si in sorted({r[0] for r in rows}):
        ks = [r for r in rows if r[0] == si]
        pool = [r for r in ks if POOL in r[4]]
        if not pool:
            print(f'step {si}: no {POOL} launch')
            continue
        p0, p1, ps = pool[0][2], pool[0][3], pool[0][1]
        end = max(r[3] for r in ks)
        inside, busy = {}, []
        for r in ks:
            if r[1] == ps:
                continue
            o0, o1 = max(r[2], p0), min(r[3], p1)
            if o1 > o0:
                short = r[4].split('(')[0].split('<')[0].split('::')[-1]
                inside[short] = inside.get(short, 0.0) + (o1 - o0)
                busy.append((o0, o1))
        covered, cur = 0.0, p0
        for b0, b1 in sorted(busy):
            b0 = max(b0, cur)
            if b1 > b0:
                covered += b1 - b0
                cur = b1
        print(f'step {si}: step {end:.0f} us of kernels; pool on stream {ps} from {p0:.0f} to {p1:.0f} us ({p1 - p0:.0f} us); '
              f'other streams ran kernels for {covered:.0f} us of it and had none for {p1 - p0 - covered:.0f} us')
        for name, t in sorted(inside.items(), key=lambda kv: -kv[1]):
            print(f'    {t:8.1f} us  {name}')
        after = [r for r in ks if r[1] != ps and r[2] >= p1]
        if after:
            print(f'    first kernel after the pool: {after[0][4][:60]} at {after[0][2]:.0f} us')


if __name__ == '__main__':
    main()
