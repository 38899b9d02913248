"""Seeded synthetic frame-window inputs and weights (there are no datasets or checkpoints
on the box). Shapes follow what the reference's offline preprocessing stores per
detection (reference: data/seq_processing/seq_processor.py:445-446,545-548):
ReID ``[N,256]``, node-core ``[N,2048,8,4]``, node-ext ``[N,256,14,14]``; nodes are
ordered by (frame, detection id) as ``MOTGraph._construct_graph_df`` orders them
(reference: data/mot_graph.py:145).

Everything here is host-side input generation; no arithmetic of the hot path lives here.
"""
import math
from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import torch

from .config import param_shapes


def make_window(T=15, D=30, k=50, seed=0, sigma=0.5, fps=30.0, reid_dim=256,
                node_feats='pooled', with_ext=False, min_gap=1e-5, first_frame=1,
                node_dim=2048):
    """One frame-window: ``D`` persistent identities seen in each of ``T`` frames.

    node_feats: 'pooled' -> x is [N,node_dim,1,1] (the avg-pool of the reference is then
    the identity, reference: models/mpn.py:351-352); 'full' -> x is [N,node_dim,8,4].
    The ReID embeddings are re-drawn for nodes whose k-th / (k+1)-th neighbour distance
    gap is below ``min_gap`` (relative) so that the top-k sets do not hinge on the last
    ulp of a distance (SURVEY.md H1).
    """
    g = torch.Generator().manual_seed(int(seed))
    N = T * D
    frame = torch.arange(first_frame, first_frame + T, dtype=torch.int64).repeat_interleave(D)
    ident = torch.arange(D, dtype=torch.int64).repeat(T)
    centroid = torch.randn(D, reid_dim, generator=g)
    reid = centroid[ident] + sigma * torch.randn(N, reid_dim, generator=g)
    reid = _enforce_knn_gap(reid, frame, k, min_gap, centroid, ident, sigma, g)

    # boxes: identity-specific size and start position, small per-frame drift
    h0 = 60.0 + 200.0 * torch.rand(D, generator=g, dtype=torch.float64)
    x0 = 1920.0 * torch.rand(D, generator=g, dtype=torch.float64)
    y0 = 400.0 + 600.0 * torch.rand(D, generator=g, dtype=torch.float64)
    vx = 4.0 * torch.randn(D, generator=g, dtype=torch.float64)
    vy = 1.0 * torch.randn(D, generator=g, dtype=torch.float64)
    t = (frame - first_frame).to(torch.float64)
    bb_height = h0[ident] * (1.0 + 0.02 * torch.randn(N, generator=g, dtype=torch.float64)).clamp(0.8, 1.2)
    bb_width = 0.4 * bb_height * (1.0 + 0.02 * torch.randn(N, generator=g, dtype=torch.float64)).clamp(0.8, 1.2)
    feet_x = x0[ident] + vx[ident] * t + torch.randn(N, generator=g, dtype=torch.float64)
    feet_y = y0[ident] + vy[ident] * t + torch.randn(N, generator=g, dtype=torch.float64)

    if node_feats == 'pooled':
        x = torch.randn(N, node_dim, 1, 1, generator=g).abs_()
    elif node_feats == 'full':
        x = torch.randn(N, node_dim, 8, 4, generator=g).abs_()
    else:
        raise ValueError(node_feats)
    x_ext = torch.randn(N, 256, 14, 14, generator=g) if with_ext else None

    return SimpleNamespace(
        T=T, D=D, k=k, N=N, fps=float(fps), seed=seed,
        frame=frame, detection_id=torch.arange(N, dtype=torch.int64), ident=ident,
        bb_height=bb_height.numpy(), bb_width=bb_width.numpy(),
        feet_x=feet_x.numpy(), feet_y=feet_y.numpy(),
        reid=reid.contiguous(), x=x, x_ext=x_ext)


def det_columns(win):
    """The detection-table columns ``compute_edge_feats_dict`` reads
    (reference: utils/graph.py:107-113), as a plain dict of float64 numpy arrays."""
    return {'frame': win.frame.numpy().astype(np.float64), 'bb_height': win.bb_height,
            'bb_width': win.bb_width, 'feet_x': win.feet_x, 'feet_y': win.feet_y}


def _knn_boundary_gaps(reid, frame, k):
    d = torch.cdist(reid.double(), reid.double())
    d[frame[:, None] == frame[None, :]] = float('inf')
    kk = min(k + 1, d.shape[1])
    vals = torch.topk(d, kk, dim=1, largest=False).values
    if kk <= k:
        return torch.full((d.shape[0],), float('inf'), dtype=torch.float64)
    a, b = vals[:, k - 1], vals[:, k]
    gap = (b - a) / a.clamp(min=1e-30)
    gap[~torch.isfinite(b)] = float('inf')
    return gap


def _enforce_knn_gap(reid, frame, k, min_gap, centroid, ident, sigma, g, max_rounds=20):
    if min_gap <= 0 or k is None:
        return reid
    for _ in range(max_rounds):
        bad = torch.nonzero(_knn_boundary_gaps(reid, frame, k) < min_gap).view(-1)
        if bad.numel() == 0:
            return reid
        reid = reid.clone()
        reid[bad] = centroid[ident[bad]] + sigma * torch.randn(bad.numel(), reid.shape[1], generator=g)
    raise RuntimeError('could not separate the k-th/(k+1)-th neighbour distances')


def make_params(model_params, seed=0, gain=1.0, core_only=False, dtype=torch.float32):
    """Deterministic weights with the reference's ``state_dict`` names and shapes.
    U(-b, b)*gain with b = 1/sqrt(fan_in), i.e. the bound torch's default Linear/Conv
    initialisation uses; the LayerNorm starts at (1, 0)."""
    g = torch.Generator().manual_seed(int(seed))
    out = OrderedDict()
    shapes = param_shapes(model_params, core_only=core_only)
    for name, shape in shapes.items():
        if name.endswith('num_batches_tracked'):
            out[name] = torch.tensor(100, dtype=torch.int64)
            continue
        if name.endswith('running_var') or (name.endswith('weight') and len(shape) == 1 and 'layer_norm' not in name):
            out[name] = (0.5 + torch.rand(shape, generator=g, dtype=torch.float64)).to(dtype)      # BatchNorm scale / variance
            continue
        if name.endswith('running_mean') or (name.endswith('bias') and name[:-4] + 'running_var' in shapes):
            out[name] = (0.2 * torch.randn(shape, generator=g, dtype=torch.float64)).to(dtype)
            continue
        if 'layer_norm' in name:
            out[name] = torch.ones(shape, dtype=dtype) if name.endswith('weight') else torch.zeros(shape, dtype=dtype)
            continue
        if name.endswith('weight'):
            fan_in = int(np.prod(shape[1:]))
            wname = name
        else:
            wshape = shapes[name[:-4] + 'weight']
            fan_in = int(np.prod(wshape[1:]))
        b = 1.0 / math.sqrt(fan_in)
        scale = gain if name.endswith('weight') else 1.0
        out[name] = ((torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * b * scale).to(dtype)
    return out


def make_mots_sequence(frames=600, per_frame=20, height=1080, width=1920, mask_size=56, seed=0):
    """A MOTS-shaped sequence for the mask output stage: ``per_frame`` pedestrian-shaped boxes (height 60-400 px,
    width 0.35-0.5 of it, some partly outside the image) in each of ``frames`` frames, and smooth 56 x 56 masks (a
    logistic ellipse per node).  Returns (masks [N,1,M,M] fp32, boxes [N,4] float64 (x1, y1, x2, y2), frame [N] int64)."""
    g = torch.Generator().manual_seed(int(seed))
    n = frames * per_frame
    frame = torch.arange(1, frames + 1, dtype=torch.int64).repeat_interleave(per_frame)
    bh = 60.0 + 340.0 * torch.rand(n, generator=g, dtype=torch.float64)
    bw = bh * (0.35 + 0.15 * torch.rand(n, generator=g, dtype=torch.float64))
    x1 = width * torch.rand(n, generator=g, dtype=torch.float64) - 0.5 * bw
    y1 = (height - 0.8 * bh) * torch.rand(n, generator=g, dtype=torch.float64) - 0.1 * bh
    boxes = torch.stack((x1, y1, x1 + bw, y1 + bh), dim=1)
    u = (torch.arange(mask_size, dtype=torch.float32) + 0.5) / mask_size
    cu, cv = 0.5 + 0.1 * torch.randn(2, n, 1, 1, generator=g)
    su, sv = 0.25 + 0.15 * torch.rand(2, n, 1, 1, generator=g)
    sharp = 3.0 + 6.0 * torch.rand(n, 1, 1, generator=g)
    r2 = ((u.view(1, 1, -1) - cu) / su) ** 2 + ((u.view(1, -1, 1) - cv) / sv) ** 2
    masks = torch.sigmoid(sharp * (1.0 - r2)).unsqueeze(1).contiguous()
    return masks, boxes, frame
