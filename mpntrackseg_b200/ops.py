"""Tensor-level wrappers over the C ABI (include/mpntrack_b200.h).

Each function validates device / dtype / contiguity, allocates outputs with torch (device
memory + stream plumbing only) and enqueues the library's kernels on torch's current
stream.  CPU tensors are rejected: there is no CPU fallback.
"""
import ctypes as C
import os
import warnings
from dataclasses import dataclass

import torch

from . import _cabi
from ._cabi import CoreWeights, EdgeLayout, check, lib, ptr, stream_ptr


def _req(t, dtype, name):
    if not torch.is_tensor(t):
        raise TypeError(f'{name}: expected a torch tensor, got {type(t).__name__}')
    if not t.is_cuda:
        raise RuntimeError(f'{name}: must be a CUDA tensor (no CPU fallback)')
    if t.dtype != dtype:
        raise TypeError(f'{name}: expected {dtype}, got {t.dtype}')
    if t.device.index != torch.cuda.current_device():
        # kernels are enqueued on the CURRENT device's stream (stream_ptr()); a tensor of another GPU would be dereferenced there
        raise RuntimeError(f'{name}: tensor lives on {t.device} but the current device is cuda:{torch.cuda.current_device()}; '
                           f'call under torch.cuda.device({t.device.index})')
    return t if t.is_contiguous() else t.contiguous()


def _ld(t):
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError('expected a 2-D tensor with unit column stride')
    return t.stride(0)


def _bytes(n, device):
    return torch.empty(max(int(n), 1), dtype=torch.uint8, device=device)


# ------------------------------------------------------------------ graph construction
def time_valid_pairs(frame_num, max_frame_dist=-1, node_graph_ptr=None):
    """[2, E_c] int64 candidate pairs (i<j), sorted by (i, j).  utils/graph.py:6-37"""
    f = _req(frame_num, torch.int64, 'frame_num')
    n = f.numel()
    gp = None if node_graph_ptr is None else _req(node_graph_ptr, torch.int64, 'node_graph_ptr')
    g = 0 if gp is None else gp.numel() - 1
    row_start = torch.empty(n + 1, dtype=torch.int64, device=f.device)
    total = C.c_int64(0)
    check(lib().mpn_time_valid_pairs_count(ptr(f), n, ptr(gp), g, int(max_frame_dist), ptr(row_start),
                                           C.byref(total), stream_ptr()), 'time_valid_pairs_count')
    pairs = torch.empty((2, total.value), dtype=torch.int64, device=f.device)
    if total.value == 0:                 # one detection, or all detections in one frame: no candidate pair
        return pairs
    check(lib().mpn_time_valid_pairs_fill(ptr(f), n, ptr(gp), g, int(max_frame_dist), ptr(row_start),
                                          ptr(pairs[0]), ptr(pairs[1]), stream_ptr()), 'time_valid_pairs_fill')
    return pairs


def pair_reid_dist(reid, pairs):
    """[E] fp32 ||a-b+1e-6||_2.  data/mot_graph.py:211,299-303"""
    reid = _req(reid, torch.float32, 'reid')
    pairs = _req(pairs, torch.int64, 'pairs')
    e = pairs.shape[1]
    out = torch.empty(e, dtype=torch.float32, device=reid.device)
    check(lib().mpn_pair_reid_dist(ptr(reid), reid.shape[0], reid.shape[1], ptr(pairs[0]), ptr(pairs[1]),
                                   e, ptr(out), stream_ptr()), 'pair_reid_dist')
    return out


def knn_mask(pwise_dist, edge_ixs, num_nodes, top_k, reciprocal, symmetric_edges):
    """bool [E'] keep mask.  utils/graph.py:40-87"""
    d = _req(pwise_dist.view(-1), torch.float32, 'pwise_dist')
    ei = _req(edge_ixs, torch.int64, 'edge_ixs')
    e = ei.shape[1]
    if d.numel() != e:
        raise ValueError(f'pwise_dist has {d.numel()} entries for {e} edges')
    ws = _bytes(lib().mpn_knn_mask_workspace(int(num_nodes)), d.device)
    keep = torch.empty(e, dtype=torch.uint8, device=d.device)
    check(lib().mpn_knn_mask(ptr(d), ptr(ei[0]), ptr(ei[1]), e, int(num_nodes), int(top_k), int(bool(reciprocal)),
                             int(bool(symmetric_edges)), ptr(ws), ptr(keep), stream_ptr()), 'knn_mask')
    return keep.view(torch.bool)


def assign_edge_labels(edge_index, node_ids, mode='closest'):
    """Float labels [E] of the network-flow formulation.  data/mot_graph.py:223-262"""
    if mode not in ('all', 'closest'):
        raise ValueError(f"true_edge_labels must be 'all' or 'closest', got {mode!r}")
    ei = _req(edge_index, torch.int64, 'edge_index')
    ids = _req(node_ids, torch.int64, 'node_ids')
    e, n = ei.shape[1], ids.numel()
    ws = torch.empty(max(2 * n, 1), dtype=torch.int32, device=ei.device)
    labels = torch.empty(e, dtype=torch.float32, device=ei.device)
    check(lib().mpn_assign_edge_labels(ptr(ei[0]), ptr(ei[1]), e, ptr(ids), n, 1 if mode == 'closest' else 0, ptr(ws),
                                       ptr(labels), stream_ptr()), 'assign_edge_labels')
    return labels


def compact_pairs(pairs, keep, dist=None):
    """pairs[:, keep] (and dist[keep]) in order.  data/mot_graph.py:219"""
    pairs = _req(pairs, torch.int64, 'pairs')
    k8 = _req(keep.view(torch.uint8) if keep.dtype == torch.bool else keep, torch.uint8, 'keep')
    e = pairs.shape[1]
    scan = torch.empty(e + 1, dtype=torch.int64, device=pairs.device)
    out = torch.empty_like(pairs)
    od = torch.empty_like(dist) if dist is not None else None
    kept = C.c_int64(0)
    check(lib().mpn_compact_pairs(ptr(pairs[0]), ptr(pairs[1]), ptr(dist), ptr(k8), e, ptr(scan), ptr(out[0]),
                                  ptr(out[1]), ptr(od), C.byref(kept), stream_ptr()), 'compact_pairs')
    k = kept.value
    # out rows are contiguous slabs of length e; re-pack to [2, k]
    res = torch.stack((out[0, :k], out[1, :k]))
    return (res, od[:k]) if dist is not None else res


def edge_feats_assemble(pairs, frame_f32, bb_height, bb_width, feet_x, feet_y, fps, reid_dist):
    """(edge_attr [2P, 5|6] fp32, edge_index [2, 2P] int64).
    utils/graph.py:90-124 + data/mot_graph.py:292-312"""
    pairs = _req(pairs, torch.int64, 'pairs')
    p = pairs.shape[1]
    cols = [_req(t, torch.float32, n) for t, n in ((frame_f32, 'frame'), (bb_height, 'bb_height'),
                                                    (bb_width, 'bb_width'), (feet_x, 'feet_x'), (feet_y, 'feet_y'))]
    ad = 6 if reid_dist is not None else 5
    rd = None if reid_dist is None else _req(reid_dist.view(-1), torch.float32, 'reid_dist')
    attr = torch.empty((2 * p, ad), dtype=torch.float32, device=pairs.device)
    eidx = torch.empty((2, 2 * p), dtype=torch.int64, device=pairs.device)
    check(lib().mpn_edge_feats_assemble(ptr(pairs[0]), ptr(pairs[1]), p, *[ptr(c) for c in cols], float(fps),
                                        ptr(rd), ad, ptr(attr), ptr(eidx), stream_ptr()), 'edge_feats_assemble')
    return attr, eidx


# [build code, rows repaired exactly] of the last knn_graph_pairs call.  Build code: 0 exact fp32, 1 dense Gram + row
# select, 2 thresholded candidate lists (nonzero = tensor cores).
LAST_KNN_STATS = [0, 0]


def knn_graph_pairs(frame_num, node_graph_ptr_host, reid, top_k, reciprocal, max_frame_dist=-1, engine=None):
    """Batched edge construction: (pairs [2,P] int64 batch-global ids sorted by (row,col), dist [P],
    graph_pair_ptr list[G+1]).  node_graph_ptr_host: python list / CPU tensor of G+1 node offsets.
    data/mot_graph.py:195-221 for every window of the batch in one pass."""
    f = _req(frame_num, torch.int64, 'frame_num')
    reid = _req(reid, torch.float32, 'reid')
    hp = [int(v) for v in node_graph_ptr_host]
    g = len(hp) - 1
    n = hp[-1]
    if f.numel() != n or reid.shape[0] != n:
        raise ValueError('frame_num / reid do not match node_graph_ptr')
    k = -1 if top_k is None else int(top_k)
    sizes = [hp[i + 1] - hp[i] for i in range(g)]
    cap = sum(s * min(k, s) if k >= 0 else s * (s - 1) // 2 for s in sizes)
    cap = max(cap, 1)
    dev = f.device
    h_ptr = (C.c_int64 * (g + 1))(*hp)
    d_ptr = torch.tensor(hp, dtype=torch.int64, device=dev)
    ws = _bytes(lib().mpn_knn_graph_workspace(n, sum(s * s for s in sizes), g), dev)
    pairs = torch.empty((2, cap), dtype=torch.int64, device=dev)
    dist = torch.empty(cap, dtype=torch.float32, device=dev)
    gpp = torch.empty(g + 1, dtype=torch.int64, device=dev)
    h_gpp = (C.c_int64 * (g + 1))()
    h_stats = (C.c_int64 * 2)()
    use_tc = int((engine or default_engine()) != 'fp32')
    check(lib().mpn_knn_graph_pairs(ptr(f), ptr(d_ptr), h_ptr, g, ptr(reid), reid.shape[1], k, int(bool(reciprocal)),
                                    int(max_frame_dist), use_tc, ptr(ws), cap, ptr(pairs[0]), ptr(pairs[1]), ptr(dist),
                                    ptr(gpp), h_gpp, h_stats, stream_ptr()), 'knn_graph_pairs')
    LAST_KNN_STATS[:] = list(h_stats)
    hg = list(h_gpp)
    p = hg[-1]
    return torch.stack((pairs[0, :p], pairs[1, :p])) if p != cap else pairs, dist[:p], hg


# ------------------------------------------------------------------ layout
@dataclass
class Layout:
    num_nodes: int
    num_edges: int
    num_out: int
    slot_row: torch.Tensor
    slot_col: torch.Tensor
    slot_edge: torch.Tensor
    out_ptr: torch.Tensor
    in_ptr: torch.Tensor

    def c_struct(self):
        return EdgeLayout(self.num_nodes, self.num_edges, self.num_out, self.slot_row.data_ptr(),
                          self.slot_col.data_ptr(), self.slot_edge.data_ptr(), self.out_ptr.data_ptr(),
                          self.in_ptr.data_ptr())


def edge_layout(edge_index, num_nodes):
    """Slot layout (flow_out group then flow_in group, row-sorted, stable)."""
    ei = _req(edge_index, torch.int64, 'edge_index')
    if ei.dim() != 2 or ei.shape[0] != 2:
        raise ValueError(f'edge_index must be [2, E], got {tuple(ei.shape)}')
    e, n, dev = ei.shape[1], int(num_nodes), ei.device
    ws = _bytes(lib().mpn_edge_layout_workspace(e, n), dev)
    i32 = dict(dtype=torch.int32, device=dev)
    srow, scol, sedge = (torch.empty(max(e, 1), **i32) for _ in range(3))
    optr, iptr = torch.empty(n + 1, **i32), torch.empty(n + 1, **i32)
    num_out = C.c_int64(0)
    check(lib().mpn_edge_layout_build(ptr(ei), e, n, ptr(ws), ptr(srow), ptr(scol), ptr(sedge), ptr(optr),
                                      ptr(iptr), C.byref(num_out), stream_ptr()), 'edge_layout_build')
    return Layout(n, e, num_out.value, srow, scol, sedge, optr, iptr)


# ------------------------------------------------------------------ encoders
def avgpool(x, out=None):
    """[N, C, H, W] -> [N, C] (optionally into a preallocated contiguous ``out``).  models/mpn.py:351-352"""
    x = _req(x, torch.float32, 'x')
    n, c = x.shape[0], x.shape[1]
    hw = 1
    for s in x.shape[2:]:
        hw *= s
    if hw == 1:
        if out is None:
            return x.reshape(n, c)
        out.copy_(x.reshape(n, c))
        return out
    return avgpool_windows([x], out)


def avgpool_windows(xs, out=None):
    """Every window's maps [N_i, C, H, W] -> one [sum N_i, C] buffer, window i in rows sum(N_<i):sum(N_<=i), in one
    launch (per 64 windows).  Each row is what ``avgpool`` gives for it, bit for bit."""
    xs = [_req(x, torch.float32, 'x') for x in xs]
    if not xs:
        raise ValueError('avgpool_windows: no windows')
    c, spatial = xs[0].shape[1], xs[0].shape[2:]
    if any(x.dim() < 3 or x.shape[1] != c or x.shape[2:] != spatial for x in xs):
        raise ValueError('avgpool_windows: every window must be [N_i, C, H, W] with the same C, H, W')
    hw = 1
    for s in spatial:
        hw *= s
    n_tot = sum(x.shape[0] for x in xs)
    if out is None:
        out = torch.empty((n_tot, c), dtype=torch.float32, device=xs[0].device)
    elif not (out.is_contiguous() and tuple(out.shape) == (n_tot, c) and out.dtype == torch.float32):
        raise ValueError('avgpool: out must be a contiguous fp32 [N, C] tensor')
    if hw == 1:
        torch.cat([x.reshape(x.shape[0], c) for x in xs], out=out)
        return out
    g = len(xs)
    check(lib().mpn_avgpool((C.c_void_p * g)(*[x.data_ptr() for x in xs]), (C.c_int64 * g)(*[x.shape[0] for x in xs]),
                            g, c, hw, ptr(out), stream_ptr()), 'avgpool')
    return out


def linear(inp, weight, bias, relu):
    """act(inp @ weight.T + bias).  models/mlp.py:12-23"""
    inp = _req(inp, torch.float32, 'input')
    w = _req(weight, torch.float32, 'weight')
    b = None if bias is None else _req(bias, torch.float32, 'bias')
    m, k = inp.shape
    o = w.shape[0]
    if w.shape[1] != k:
        raise ValueError(f'linear: input has {k} columns, weight expects {w.shape[1]}')
    out = torch.empty((m, o), dtype=torch.float32, device=inp.device)
    check(lib().mpn_linear(ptr(inp), m, k, ptr(w), ptr(b), o, int(bool(relu)), ptr(out), stream_ptr()), 'linear')
    return out


def node_encoder(x, weights, biases, engine=None, status=None):
    """encoder.node_model on pooled features x [N, K].  The shipped K -> 128 -> 32 stack runs as one
    tcgen05 kernel (engine 'tc' / 'auto'; every operand row split at its own power-of-two scale, so the error is
    relative at any magnitude); other widths, x off 16-byte alignment, engine 'fp32' and non-finite features or
    weights use the fp32 Linear kernel chain.  models/mpn.py:355
    status: optional int32[1] device tensor; if given the non-finite flag is left there for the caller to
    check (no host sync here) and no fallback is attempted."""
    engine = engine or default_engine()
    x = _req(x, torch.float32, 'x')
    ws_ = [_req(w, torch.float32, 'weight') for w in weights]
    bs_ = [_req(b, torch.float32, 'bias') for b in biases]
    n, k0 = x.shape

    def tc(st):
        out = torch.empty((n, 32), dtype=torch.float32, device=x.device)
        ws = _bytes(lib().mpn_node_encoder_tc_workspace(k0), x.device)
        check(lib().mpn_node_encoder_tc(ptr(x), n, k0, ptr(ws_[0]), ptr(bs_[0]), 128, ptr(ws_[1]), ptr(bs_[1]), 32,
                                        ptr(ws), ptr(out), ptr(st), stream_ptr()), 'node_encoder_tc')
        return out

    def fp32():
        h = x
        for w, b in zip(ws_, bs_):
            h = linear(h, w, b, relu=w.shape[0] != 1)
        return h

    fits = (len(ws_) == 2 and ws_[0].shape[0] == 128 and ws_[1].shape[0] == 32 and k0 % 64 == 0 and k0 >= 64
            and x.data_ptr() % 16 == 0)
    if not fits or n == 0:
        return fp32()
    return tc_or_fp32(engine, tc, fp32, 'node_encoder_tc: non-finite node features or encoder weights; use engine="fp32"',
                      'mpntrackseg_b200: non-finite node features or encoder weights, rerunning the encoder on the fp32 kernels',
                      status=status)


def gather_rows(inp, idx):
    inp = _req(inp, torch.float32, 'input')
    idx = _req(idx, torch.int32, 'idx')
    rows, width = idx.numel(), inp.shape[1]
    out = torch.empty((rows, width), dtype=torch.float32, device=inp.device)
    check(lib().mpn_gather_rows(ptr(inp), ptr(idx), rows, width, ptr(out), stream_ptr()), 'gather_rows')
    return out


def segment_sum(inp, in_off, width, seg_ptr, perm, out, col_off, accumulate=False, mode='sum', argmax=None):
    """out[:, col_off:col_off+width] (+)= the sum / mean / max of each segment; ``argmax`` (int32 [nodes, width], max only)
    receives the input row of each maximum (-1 for an empty segment)."""
    check(lib().mpn_segment_reduce(ptr(inp), _ld(inp), in_off, width, ptr(seg_ptr), ptr(perm), out.shape[0],
                                   int(accumulate), ptr(out), _ld(out), col_off, NODE_AGG[mode], ptr(argmax),
                                   stream_ptr()), 'segment_sum')


def edge_encoder(edge_attr, layout, weights, biases):
    """e_init in slot order.  models/mpn.py:355 (encoder.edge_model)"""
    attr = _req(edge_attr, torch.float32, 'edge_attr')
    ws = [_req(w, torch.float32, 'weight') for w in weights]
    bs = [_req(b, torch.float32, 'bias') for b in biases]
    dims = [ws[0].shape[1]] + [w.shape[0] for w in ws]
    e = layout.num_edges
    if attr.shape != (e, dims[0]):
        raise ValueError(f'edge_attr must be [{e}, {dims[0]}], got {tuple(attr.shape)}')
    if dims == [6, 18, 18, 16]:
        out = torch.empty((e, dims[-1]), dtype=torch.float32, device=attr.device)
        cdims = (C.c_int32 * len(dims))(*dims)
        cw = (C.c_void_p * len(ws))(*[w.data_ptr() for w in ws])
        cb = (C.c_void_p * len(bs))(*[b.data_ptr() for b in bs])
        check(lib().mpn_edge_encoder(ptr(attr), ptr(layout.slot_edge), e, cdims, len(ws), cw, cb, ptr(out),
                                     stream_ptr()), 'edge_encoder')
        return out
    h = gather_rows(attr, layout.slot_edge[:e]) if e else attr.new_empty((0, dims[0]))
    for w, b in zip(ws, bs):
        h = linear(h, w, b, relu=w.shape[0] != 1)
    return h


# ------------------------------------------------------------------ message passing
NODE_AGG = {'sum': 0, 'mean': 1, 'max': 2}


def core_weights(named, node_agg='sum'):
    """Build the mpn_core_weights struct from a dict of CUDA fp32 tensors keyed by the struct's
    field names; returns (struct, keepalive list).  node_agg: 'sum' | 'mean' | 'max' (models/mpn.py:263-273)."""
    if node_agg not in NODE_AGG:
        raise ValueError(f"node_agg_fn can only be 'max', 'mean' or 'sum', got {node_agg!r}")
    keep = {k: _req(v, torch.float32, k) for k, v in named.items()}
    dn = keep['node_w'].shape[0]
    de = keep['edge_w1'].shape[0]
    cw = CoreWeights()
    cw.dn, cw.de = dn, de
    cw.edge_h, cw.flow_h, cw.cls_h = keep['edge_w0'].shape[0], keep['fin_w0'].shape[0], keep['cls_w0'].shape[0]
    expect = {'edge_w0': (cw.edge_h, 4 * dn + 2 * de), 'edge_w1': (de, cw.edge_h),
              'fin_w0': (cw.flow_h, 2 * dn + de), 'fin_w1': (dn, cw.flow_h),
              'fout_w0': (cw.flow_h, 2 * dn + de), 'fout_w1': (dn, cw.flow_h),
              'node_w': (dn, 2 * dn), 'cls_w0': (cw.cls_h, de), 'cls_w1': (1, cw.cls_h)}
    for k, shp in expect.items():
        if tuple(keep[k].shape) != shp:
            raise ValueError(f'{k}: expected shape {shp}, got {tuple(keep[k].shape)}')
    for name, _ in CoreWeights._fields_[5:-1]:
        setattr(cw, name, keep[name].data_ptr())
    cw.node_agg = NODE_AGG[node_agg]
    return cw, list(keep.values())


ENGINES = ('auto', 'tc', 'fp32')


def default_engine():
    eng = os.environ.get('MPN_ENGINE', 'auto')
    if eng not in ENGINES:
        raise ValueError(f'MPN_ENGINE must be one of {ENGINES}, got {eng!r}')
    return eng


def tc_or_fp32(engine, tc, fp32, overflow, rerun, status=None):
    """The one tensor-core / fp32 policy.  ``tc(status)`` enqueues the tensor-core work, which sets a word of the zeroed
    int32 device tensor ``status`` (two words: one per kernel family for a caller that runs both) when a value left the
    fp16 range; ``fp32()`` computes on the fp32 kernels.  engine 'fp32' runs ``fp32()``.  Otherwise a caller's
    ``status`` is only handed to ``tc`` (the caller reads it: no host sync, no fallback here); without one, the status
    is read once: all 0 returns the tensor-core result, else engine 'tc' raises OverflowError(overflow) and 'auto'
    warns ``rerun`` and returns ``fp32()``."""
    if engine not in ENGINES:
        raise ValueError(f'engine must be one of {ENGINES}, got {engine!r}')
    if engine == 'fp32':
        return fp32()
    if status is not None:
        return tc(status)
    status = torch.zeros(2, dtype=torch.int32, device='cuda')
    out = tc(status)
    if status.view(torch.int64).item() == 0:                      # both words in the one host sync
        return out
    if engine == 'tc':
        raise OverflowError(overflow)
    warnings.warn(rerun)
    return fp32()


LAST_TC_SCHEDULE = {}     # filled by mp_forward(..., debug=True): {'sched': [...], 'amax': [...], 'xmax': [...]} by step


def mp_forward(cw, layout, x_init, e_init, num_steps, first_class_step, want_state=False, engine=None,
               status=None, debug=False):
    """Run the step loop.  Returns logits [S, E] (original edge order) and, if asked, the final
    node / edge latent states (edge state in slot order).  models/mpn.py:364-389

    engine: 'tc' = tcgen05 tensor-core kernels (fp16 hi/lo split operands in a per-step power-of-two
    scale, fp32 accumulate), 'fp32' = fp32 SIMT kernels, 'auto' (default) = 'tc', rerun on 'fp32' if an
    activation still left the fp16 range (one-step growth beyond the 1024x headroom of the scale) or a step's scale
    passed 2^17, beyond which rows of order 1 -- a quiet window batched with a loud one -- lose the parity bar.  status: optional int32[1] device tensor: the overflow flag is left there for the
    caller (no host sync, no fallback here)."""
    engine = engine or default_engine()
    x_init = _req(x_init, torch.float32, 'x_init')
    e_init = _req(e_init, torch.float32, 'e_init')
    n, e, dev = layout.num_nodes, layout.num_edges, x_init.device
    n_cls = 1 if num_steps == 0 else max(num_steps - first_class_step + 1, 0)
    n_cls = min(n_cls, max(num_steps, 1))
    first = max(first_class_step, 1)
    logits = torch.empty((n_cls, e), dtype=torch.float32, device=dev)
    x_out = torch.empty((n, cw.dn), dtype=torch.float32, device=dev) if want_state else None
    e_out = torch.empty((e, cw.de), dtype=torch.float32, device=dev) if want_state else None
    g = layout.c_struct()
    result = (logits, x_out, e_out) if want_state else logits

    def tc(st):
        ws = _bytes(lib().mpn_mp_tc_workspace(n, e), dev)
        check(lib().mpn_mp_forward_tc(C.byref(cw), C.byref(g), ptr(x_init), ptr(e_init), int(num_steps), int(first),
                                      ptr(ws), ptr(logits), ptr(x_out), ptr(e_out), ptr(st), stream_ptr()),
              'mp_forward_tc')
        if debug:
            hs, ha, hx = (C.c_int32 * (num_steps + 2))(), (C.c_float * (num_steps + 2))(), (C.c_float * (num_steps + 2))()
            check(lib().mpn_mp_tc_read_schedule(ptr(ws), n, e, int(num_steps), hs, ha, hx, stream_ptr()), 'mp_tc_read_schedule')
            LAST_TC_SCHEDULE.update(sched=list(hs), amax=list(ha), xmax=list(hx))
        return result

    def fp32():
        ws = _bytes(lib().mpn_mp_workspace(n, e), dev)
        check(lib().mpn_mp_forward(C.byref(cw), C.byref(g), ptr(x_init), ptr(e_init), int(num_steps), int(first),
                                   ptr(ws), ptr(logits), ptr(x_out), ptr(e_out), stream_ptr()), 'mp_forward')
        return result

    if num_steps < 1 or n == 0:
        return fp32()
    return tc_or_fp32(engine, tc, fp32, 'mp_forward_tc: an activation left the fp16 range, or the step scale passed the '
                      'split operands\' resolution; use engine="fp32"',
                      'mpntrackseg_b200: activation outside the fp16 range (or step scale beyond the split operands\' '
                      'resolution), rerunning the message-passing steps on the fp32 kernels', status=status)


def attn_aggregate(z, layout, logits):
    """(flow_in, flow_out) of the attentive aggregation, each shaped like ``z`` [N, C, H, W].
    models/mpn.py:117-134"""
    z = _req(z, torch.float32, 'z')
    lg = _req(logits.reshape(-1), torch.float32, 'logits')
    n = z.shape[0]
    feat = z[0].numel() if n else 0
    fin, fout = torch.empty_like(z), torch.empty_like(z)
    g = layout.c_struct()
    check(lib().mpn_attn_aggregate(ptr(z), n, feat, C.byref(g), ptr(lg), ptr(fin), ptr(fout), stream_ptr()),
          'attn_aggregate')
    return fin, fout


def attn_aggregate_backward(z, layout, logits, g_in, g_out, perm_c, ptr_c):
    """(d_z like z, d_logits [E] in the caller's edge order) of ``attn_aggregate`` for the output gradients
    g_in / g_out; perm_c / ptr_c: the slots sorted by column and their row pointer (int32)."""
    z = _req(z, torch.float32, 'z')
    lg = _req(logits.reshape(-1), torch.float32, 'logits')
    gi, go = _req(g_in, torch.float32, 'g_in'), _req(g_out, torch.float32, 'g_out')
    pc, qc = _req(perm_c, torch.int32, 'perm_c'), _req(ptr_c, torch.int32, 'ptr_c')
    n = z.shape[0]
    feat = z[0].numel() if n else 0
    dz = torch.empty_like(z)
    dl = torch.zeros_like(lg)
    wslot = torch.empty(max(layout.num_edges, 1), dtype=torch.float32, device=z.device)
    g = layout.c_struct()
    check(lib().mpn_attn_aggregate_backward(ptr(z), n, feat, C.byref(g), ptr(lg), ptr(gi), ptr(go), ptr(pc), ptr(qc), ptr(wslot),
                                            ptr(dz), ptr(dl), stream_ptr()), 'attn_aggregate_backward')
    return dz, dl


def weighted_bce(logits, labels, weight=1.0, want_grad=False):
    """Tracking loss over the classified steps: (loss scalar tensor, pos_weight tensor[, d loss / d logits]).
    logits: [S, E] tensor or the list ``outputs['classified_edges']``.  pl_module/pl_module.py:88-105"""
    if isinstance(logits, (list, tuple)):
        logits = torch.stack([t.reshape(-1) for t in logits])
    lg = _req(logits, torch.float32, 'logits')
    lb = _req(labels.reshape(-1), torch.float32, 'edge_labels')
    s, e = lg.shape
    if lb.numel() != e:
        raise ValueError(f'{lb.numel()} labels for {e} edges')
    dev = lg.device
    ws = _bytes(lib().mpn_weighted_bce_workspace(), dev)
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    pw = torch.zeros(1, dtype=torch.float32, device=dev)
    grad = torch.empty_like(lg) if want_grad else None
    check(lib().mpn_weighted_bce(ptr(lg), ptr(lb), s, e, float(weight), ptr(ws), ptr(loss), ptr(pw), ptr(grad),
                                 stream_ptr()), 'weighted_bce')
    return (loss, pw, grad) if want_grad else (loss, pw)


# ------------------------------------------------------------------ rounding / identities (SURVEY.md f2)
def _rate(counts):
    """1 - violated / constraints in float32, as the reference's tensor arithmetic (evaluation.py:404-409)."""
    viol = torch.tensor(float(counts[0] + counts[1]), dtype=torch.float32)
    return float((1 - viol / int(counts[2])).item()) if counts[2] else float('nan')


def constr_satisfaction(edge_index, edges_out, num_nodes, undirected_edges=True):
    """(rate, flow_in [N], flow_out [N]) of BINARISED edge values.  utils/evaluation.py:370-414"""
    ei = _req(edge_index, torch.int64, 'edge_index')
    v = _req(edges_out.reshape(-1), torch.float32, 'edges_out')
    e, n = ei.shape[1], int(num_nodes)
    ws = _bytes(lib().mpn_rounding_workspace(n), ei.device)
    fin = torch.empty(n, dtype=torch.float32, device=ei.device)
    fout = torch.empty(n, dtype=torch.float32, device=ei.device)
    counts = (C.c_int64 * 3)()
    check(lib().mpn_constr_satisfaction(ptr(ei[0]), ptr(ei[1]), ptr(v), e, n, int(bool(undirected_edges)), ptr(ws), ptr(fin),
                                        ptr(fout), counts, stream_ptr()), 'constr_satisfaction')
    return _rate(counts), fin, fout


def greedy_project(edge_index, edge_preds, num_nodes):
    """(round_preds [E] float 0/1, constraint satisfaction rate of the plain > 0.5 rounding).  tracker/projectors.py:11-67"""
    ei = _req(edge_index, torch.int64, 'edge_index')
    p = _req(edge_preds.reshape(-1), torch.float32, 'edge_preds')
    e, n = ei.shape[1], int(num_nodes)
    ws = _bytes(lib().mpn_rounding_workspace(n), ei.device)
    out = torch.empty(e, dtype=torch.float32, device=ei.device)
    counts = (C.c_int64 * 3)()
    check(lib().mpn_greedy_project(ptr(ei[0]), ptr(ei[1]), ptr(p), e, n, ptr(ws), ptr(out), counts, stream_ptr()), 'greedy_project')
    return out, _rate(counts)


def connected_components(edge_index, edge_vals, num_nodes):
    """(labels [N] int64, number of components) over the edges with value 1.  tracker/mpn_tracker.py:231-248"""
    ei = _req(edge_index, torch.int64, 'edge_index')
    v = _req(edge_vals.reshape(-1), torch.float32, 'edge_vals')
    e, n = ei.shape[1], int(num_nodes)
    ws = _bytes(lib().mpn_connected_components_workspace(n), ei.device)
    labels = torch.empty(n, dtype=torch.int64, device=ei.device)
    ncomp = C.c_int64(0)
    check(lib().mpn_connected_components(ptr(ei[0]), ptr(ei[1]), ptr(v), e, n, ptr(ws), ptr(labels), C.byref(ncomp), stream_ptr()),
          'connected_components')
    return labels, ncomp.value


# ------------------------------------------------------------------ MOTS output (tracker/mpn_tracker.py:267-298,398-417)
def paste_boxes(boxes, mask_size, padding=1):
    """[N, 4] int64 boxes of torchvision's ``expand_boxes(boxes, (M + 2 padding) / M).to(torch.int64)``
    (roi_heads.py), computed with the same torch ops in the boxes' own dtype, so that the truncation toward zero sees
    the same values."""
    scale = float(mask_size + 2 * padding) / mask_size
    w_half = (boxes[:, 2] - boxes[:, 0]) * 0.5
    h_half = (boxes[:, 3] - boxes[:, 1]) * 0.5
    x_c = (boxes[:, 2] + boxes[:, 0]) * 0.5
    y_c = (boxes[:, 3] + boxes[:, 1]) * 0.5
    w_half = w_half * scale
    h_half = h_half * scale
    return torch.stack((x_c - w_half, y_c - h_half, x_c + w_half, y_c + h_half), dim=1).to(torch.int64).contiguous()


def _mots_inputs(masks, boxes, img_shape, padding):
    if not torch.is_tensor(masks) or masks.dim() not in (3, 4) or (masks.dim() == 4 and masks.shape[1] != 1):
        raise ValueError(f'masks must be [N, 1, M, M] or [N, M, M], got {tuple(getattr(masks, "shape", ()))}')
    m = _req(masks.reshape(masks.shape[0], masks.shape[-2], masks.shape[-1]), torch.float32, 'masks')
    n, mh, mw = m.shape
    if mh != mw or mh == 0:
        raise ValueError(f'masks must be square and non-empty, got {mh} x {mw}')
    if not torch.is_tensor(boxes) or boxes.dtype not in (torch.float32, torch.float64):
        raise TypeError('boxes: expected a float32 or float64 tensor')
    b = _req(boxes, boxes.dtype, 'boxes')
    if tuple(b.shape) != (n, 4):
        raise ValueError(f'boxes must be [{n}, 4], got {tuple(b.shape)}')
    h, w = int(img_shape[0]), int(img_shape[1])
    if h < 1 or w < 1 or h * w >= 2 ** 31:
        raise ValueError(f'image {h} x {w} must have 1 .. 2^31 - 1 pixels')
    if padding < 0:
        raise ValueError(f'padding must be >= 0, got {padding}')
    return m, paste_boxes(b, mh, padding), n, mh, h, w


def paste_masks_in_image(masks, boxes, img_shape, padding=1):
    """[N, 1, H, W] fp32: torchvision's ``paste_masks_in_image`` (roi_heads.py) on the device.  masks [N, 1, M, M] fp32,
    boxes [N, 4] (x1, y1, x2, y2) float32 / float64, img_shape (H, W).  A box with no pixel inside the image gives an
    all-zero mask.  reference: tracker/mpn_tracker.py:267-298"""
    m, ib, n, ms, h, w = _mots_inputs(masks, boxes, img_shape, padding)
    out = torch.empty((n, 1, h, w), dtype=torch.float32, device=m.device)
    check(lib().mpn_paste_masks(ptr(m), n, ms, int(padding), ptr(ib), h, w, ptr(out), stream_ptr()), 'paste_masks')
    return out


def mots_rle(masks, boxes, frame, img_shape, threshold=0.5):
    """Run-length encoding of every node's pasted mask after the one-owner-per-pixel rule of its frame:
    ``(area [N] int64, chars uint8, char_ptr [N+1] int64)``; node i's RLE string (pycocotools' ``rleToString`` format)
    is ``chars[char_ptr[i]:char_ptr[i+1]]``, empty when its mask is.  masks [N, 1, M, M] or [N, M, M] fp32
    probabilities, boxes [N, 4] (x1, y1, x2, y2) float32 / float64, frame [N] int64 non-decreasing, img_shape (H, W).
    A pixel belongs to the node of its frame with the largest pasted probability (ties: lower index; NaN: -inf), and
    to its mask where that probability is > threshold.  One host sync (the totals).  See DESIGN.md, MOTS output."""
    padding = 1
    m, ib, n, ms, h, w = _mots_inputs(masks, boxes, img_shape, padding)
    f = _req(frame.reshape(-1), torch.int64, 'frame')
    if f.numel() != n:
        raise ValueError(f'frame has {f.numel()} entries for {n} masks')
    dev = m.device
    ws = _bytes(lib().mpn_mots_rle_workspace(n), dev)
    area = torch.empty(n, dtype=torch.int64, device=dev)
    cnt_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    char_ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    totals = (C.c_int64 * 2)()
    check(lib().mpn_mots_rle_count(ptr(m), n, ms, int(padding), ptr(ib), ptr(f), h, w, float(threshold), ptr(ws), ptr(area),
                                   ptr(cnt_ptr), ptr(char_ptr), totals, stream_ptr()), 'mots_rle_count')
    counts = torch.empty(max(totals[0], 1), dtype=torch.int32, device=dev)
    chars = torch.empty(max(totals[1], 1), dtype=torch.uint8, device=dev)
    check(lib().mpn_mots_rle_fill(ptr(m), n, ms, int(padding), ptr(ib), ptr(f), h, w, float(threshold), ptr(cnt_ptr),
                                  ptr(char_ptr), ptr(counts), ptr(chars), stream_ptr()), 'mots_rle_fill')
    return area, chars[:totals[1]], char_ptr
