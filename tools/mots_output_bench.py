"""Times the MOTS output stage (paste, one owner per pixel, RLE strings) on the GPU against the host path the reference
runs (tracker/mpn_tracker.py:267-298): torchvision's paste in fp32 per detection, a per-frame argmax and a vectorised
numpy RLE.  Synthetic MOTS20-shaped sequence: 1920 x 1080, 20 pedestrian-shaped boxes per frame, smooth 56 x 56 masks.

The GPU time (CUDA events, after a warm-up, median of --repeats) covers ops.mots_rle and the device-to-host copy of the
strings.  The host path runs on the first --cpu-frames frames (about a second per frame), the GPU is timed on the same
frames and on the whole sequence.  Both must give the same strings, except in frames where a pixel's probability lies
within 1e-6 of the threshold; there the pixel sets must agree outside that band.

    python tools/mots_output_bench.py [--frames 600] [--cpu-frames 100] [--repeats 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mpntrackseg_b200 import synth  # noqa: E402
from mpntrackseg_b200.utils.mots import encode_mots_masks  # noqa: E402
from oracle import mots_ref  # noqa: E402

BAND = 1e-6


def cpu_path(masks, boxes, frame, shape, threshold=0.5):
    """(strings, bands) of the host path: fp32 paste per detection, per-frame argmax, numpy RLE."""
    from torchvision.models.detection.roi_heads import paste_masks_in_image
    strings, bands = [None] * frame.numel(), {}
    for f in torch.unique(frame).tolist():
        idx = torch.nonzero(frame == f).view(-1)
        p = paste_masks_in_image(masks[idx], boxes[idx], shape)[:, 0]
        near = ((p - threshold).abs() <= BAND).any(0)
        if bool(near.any()):
            bands[f] = near.numpy()
        p = torch.nan_to_num(p, nan=float('-inf'))
        win = torch.argmax(p, dim=0)
        for a, i in enumerate(idx.tolist()):
            m = ((win == a) & (p[a] > threshold)).numpy()
            if m.any():
                strings[i] = mots_ref.rle_to_string(mots_ref.rle_counts(m))
    return strings, bands


def gpu_ms(masks, boxes, frame, shape, repeats):
    args = (masks.cuda(), boxes.cuda(), frame.cuda(), shape)
    out = encode_mots_masks(*args)                       # warm-up
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        encode_mots_masks(*args)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times)), out


def decode(s, h, w):
    return np.zeros((h, w), bool) if s is None else mots_ref.rle_decode(mots_ref.rle_from_string(s), h, w)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=600)
    ap.add_argument('--cpu-frames', type=int, default=100)
    ap.add_argument('--repeats', type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    h, w = 1080, 1920
    masks, boxes, frame = synth.make_mots_sequence(frames=args.frames)
    n_cpu = int((frame <= args.cpu_frames).sum())
    sub = (masks[:n_cpu], boxes[:n_cpu], frame[:n_cpu])

    gpu_all, strings_all = gpu_ms(masks, boxes, frame, (h, w), args.repeats)
    gpu_sub, strings_sub = gpu_ms(*sub, (h, w), args.repeats)
    assert strings_sub == strings_all[:n_cpu]
    t0 = time.perf_counter()
    ref, bands = cpu_path(*sub, (h, w))
    cpu_s = time.perf_counter() - t0

    same = sum(a == b for a, b in zip(strings_sub, ref))
    for i in range(n_cpu):
        f = int(frame[i])
        if strings_sub[i] != ref[i]:
            assert f in bands, f'node {i}: strings differ in frame {f}, which has no pixel near the threshold'
            keep = ~bands[f]
            assert np.array_equal(decode(strings_sub[i], h, w)[keep], decode(ref[i], h, w)[keep]), f'node {i}'
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    print(json.dumps({
        'gpu': torch.cuda.get_device_name(), 'power_limit': power,
        'frames': args.frames, 'detections': int(frame.numel()), 'image': [h, w],
        'gpu_ms_all_frames': round(gpu_all, 3),
        'cpu_frames': args.cpu_frames, 'gpu_ms_cpu_frames': round(gpu_sub, 3), 'cpu_ms_cpu_frames': round(cpu_s * 1e3, 1),
        'speedup_cpu_frames': round(cpu_s * 1e3 / gpu_sub, 1),
        'strings_identical': same, 'strings_compared': n_cpu, 'frames_with_pixels_near_threshold': len(bands),
        'nonempty_masks': sum(s is not None for s in strings_all), 'chars': sum(len(s) for s in strings_all if s),
    }))


if __name__ == '__main__':
    main()
