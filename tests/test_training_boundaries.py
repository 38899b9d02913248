"""GPU tests of the training path against fp64, per element or per row, at the logits, shapes and scales where the
training kernels go wrong.  Each test asserts the regime or boundary it names.

* ``ops.weighted_bce`` (csrc/loss.cu) against ``bce_ref``: logits from 0 to +-inf for hard and soft labels, every
  positive fraction, edge counts past the 1,024-block cap of both partial kernels.  Gradient per element
  |d| <= 16u |ref| + 2^-120 w / E, loss |d| <= 16u loss (u = 2^-24); pos_weight exact; weight x 2^p bit for bit.
* ``CoreTrainer.loss_and_grads`` per row against fp64 autograd of the oracle: a row (one output unit of a weight or
  bias) may be off by 4x the CPU fp32 oracle's own error in that row plus 1e-5 of the row's fp64 maximum.  The bar is
  shown to reject a detached flow_in step and the loss gradient of confident negatives rounded to 0.  Exact
  transport: weight, layer-balance and input-scale transforms move the gradients by their powers of two, bit for bit.
* ``mpn_segment_reduce`` mean / max and ``mpn_segment_grad``, ``mpn_batchnorm_*`` and ``mpn_dropout_*`` directly.
"""
import importlib.util
import math
import os

import numpy as np
import pytest
import torch

import test_training_options as tto
from test_training_options import bn_fed_biases, load, make_data, make_model, oracle_loss_and_grads

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
LB = 256                    # csrc/loss.cu: threads per block of the partial kernels
BLOCK_CAP = 1024            # csrc/loss.cu: blocks of each partial kernel (grid-stride beyond)
BN_SLICE_ROWS, BN_SLICES = 256, 128     # csrc/train_ops.cu bn_slices: one row slice per 256 rows, at most 128


def dev():
    return torch.device('cuda:0')


def lib():
    from mpntrackseg_b200._cabi import lib as _lib
    return _lib()


def check(rc, what):
    from mpntrackseg_b200._cabi import check as _check
    _check(rc, what)


def ptr(t):
    from mpntrackseg_b200._cabi import ptr as _ptr
    return _ptr(t)


def sptr():
    from mpntrackseg_b200._cabi import stream_ptr
    return stream_ptr()


# ------------------------------------------------------------------ fp64 reference of the loss
def sp64(x):
    return torch.logaddexp(torch.zeros_like(x), x)


def pos_weight32(labels):
    """float32((E - pos) / pos), 0 without positives (the sum and the quotient in double, as csrc/loss.cu)."""
    e, pos = labels.numel(), float(labels.double().sum())
    return float(np.float32((e - pos) / pos)) if pos > 0 else 0.0


def bce_ref(logits, labels, weight, pw=None):
    """fp64 weighted BCE of [S, E] logits: (loss, grad [S, E], the two gradient terms' magnitude [S, E], pw).
    loss = w sum_s mean_e [(1 - y) sp(x) + pw y sp(-x)], grad = w / E ((1 - y) s(x) - pw y s(-x)); a side whose label
    weight is 0 contributes exactly 0, even where its softplus is infinite."""
    x = logits.double()
    y = labels.double().reshape(1, -1).expand_as(x)
    pw = pos_weight32(labels) if pw is None else pw
    wn, wp = 1.0 - y, pw * y
    zero = torch.zeros_like(x)
    term = torch.where(wn != 0, wn * sp64(x), zero) + torch.where(wp != 0, wp * sp64(-x), zero)
    e = x.shape[1]
    loss = weight * float(term.sum()) / e
    a, b = weight / e * wn * torch.sigmoid(x), weight / e * wp * torch.sigmoid(-x)
    return loss, a - b, a.abs() + b.abs(), pw


LOGITS = [0.0] + [s * v for v in (2.0 ** -20, 1, 8, 10, 12, 16, 17, 20, 40, 88, 89, 1e4, float('inf')) for s in (1, -1)]


def label_pattern(kind, e):
    i = torch.arange(e)
    blk = i // len(LOGITS)
    if kind == 'none':
        return torch.zeros(e)
    if kind == 'one':
        return (i == e // 2).float()
    if kind == 'half':
        return (blk % 2).float()
    if kind == 'all':
        return torch.ones(e)
    return torch.tensor([0.0, 0.3, 1.0])[blk % 3]           # 'soft'


def bce_inputs(kind, e, steps):
    lg = torch.tensor(LOGITS, dtype=torch.float32)
    idx = (torch.arange(e).view(1, -1) + 7 * torch.arange(steps).view(-1, 1)) % len(LOGITS)
    return lg[idx].contiguous(), label_pattern(kind, e)


def bce_errors(logits, labels, weight):
    loss, pw, grad = (t.cpu() for t in ops().weighted_bce(logits.to(dev()), labels.to(dev()), weight=weight,
                                                          want_grad=True))
    ref_loss, ref_g, mag, ref_pw = bce_ref(logits, labels, weight)
    e = logits.shape[1]
    bar = 16 * U * mag + 2.0 ** -120 * weight / e
    bad = ((grad.double() - ref_g).abs() > bar) | ~torch.isfinite(grad)
    return loss, pw, grad, ref_loss, ref_g, ref_pw, bad


def ops():
    from mpntrackseg_b200 import ops as _ops
    return _ops


@pytest.mark.parametrize('steps', [1, 12])
@pytest.mark.parametrize('e', [1, 255, 256, 257, 262145])
@pytest.mark.parametrize('kind', ['none', 'one', 'half', 'all', 'soft'])
def test_weighted_bce_per_element_against_fp64(kind, e, steps):
    logits, labels = bce_inputs(kind, e, steps)
    if e == 262145:                                     # both partial kernels stride past their block cap
        assert -(-e // LB) > BLOCK_CAP and -(-steps * e // LB) > BLOCK_CAP
    w = 0.7
    loss, pw, grad, ref_loss, ref_g, ref_pw, bad = bce_errors(logits, labels, w)
    assert float(pw) == ref_pw, (float(pw), ref_pw)
    if kind in ('none', 'all'):
        assert ref_pw == 0.0
    worst = float(((grad.double() - ref_g).abs() / ref_g.abs().clamp(min=1e-300)).max())
    where = [(float(logits.view(-1)[i]), float(labels[i % e])) for i in bad.view(-1).nonzero().view(-1)[:6].tolist()]
    assert not bad.any(), f'{int(bad.sum())} gradients off, worst relative {worst:.3g}, e.g. (logit, label) {where}'
    assert math.isfinite(float(loss)) == math.isfinite(ref_loss), (float(loss), ref_loss)
    if math.isfinite(ref_loss):
        assert abs(float(loss) - ref_loss) <= 16 * U * ref_loss, (float(loss), ref_loss)


@pytest.mark.parametrize('label', [0.0, 1.0, 0.3])
def test_weighted_bce_confident_logits_per_label(label):
    """One edge per logit of LOGITS with the given label (and one positive edge that fixes pw = E - 1)."""
    lg = torch.tensor(LOGITS + [0.5], dtype=torch.float32).view(1, -1)
    labels = torch.full((lg.shape[1],), label)
    labels[-1] = 1.0
    loss, pw, grad, ref_loss, ref_g, _, bad = bce_errors(lg, labels, 1.0)
    rel = ((grad.double() - ref_g).abs() / ref_g.abs().clamp(min=1e-300)).view(-1)
    report = {x: f'{float(r):.2g}' for x, r, b in zip(LOGITS, rel.tolist(), bad.view(-1).tolist()) if b}
    assert not bad.any(), f'label {label}: relative gradient errors by logit {report}'
    if label == 0.0:                                  # the confident negatives have a gradient of e^x, not 0
        assert (grad.view(-1)[[LOGITS.index(-20.0), LOGITS.index(-40.0)]] > 0).all()
    assert math.isfinite(float(loss)) == math.isfinite(ref_loss)
    if math.isfinite(ref_loss):
        assert abs(float(loss) - ref_loss) <= 16 * U * ref_loss, (float(loss), ref_loss)


def test_weighted_bce_weight_scales_bit_for_bit():
    g = torch.Generator().manual_seed(11)
    e = 70001
    logits = (torch.randn(3, e, generator=g) * 6).float()
    labels = (torch.rand(e, generator=g) < 0.2).float()
    base_loss, _, base_g = ops().weighted_bce(logits.to(dev()), labels.to(dev()), weight=0.7, want_grad=True)
    assert (base_g != 0).all() and base_g.abs().min() > 2.0 ** -100
    for p in range(-20, 21):
        loss, _, grad = ops().weighted_bce(logits.to(dev()), labels.to(dev()), weight=0.7 * 2.0 ** p, want_grad=True)
        assert torch.equal(loss, base_loss * 2.0 ** p), p
        assert torch.equal(grad, base_g * 2.0 ** p), p


@pytest.mark.parametrize('kind', ['none', 'one', 'half'])
def test_weighted_bce_nan_logit_gives_nan_loss(kind):
    logits, labels = bce_inputs(kind, 257, 2)
    logits = logits.clamp(-30, 30)
    for at in (0, 128, 256):                           # a label-0 edge and, with positives, a label-1 edge
        x = logits.clone()
        x[1, at] = float('nan')
        loss, _ = ops().weighted_bce(x.to(dev()), labels.to(dev()))
        assert math.isnan(float(loss)), (kind, at, float(labels[at]))


# ------------------------------------------------------------------ whole-network gradients per row
def oracle_grads(d, dtype, weight=1.0, p=0.0, masks=None, detach_in_step=None, zero_below=None):
    """Gradients of the core parameters by autograd of the oracle's training forward, with the loss gradient of
    ``bce_ref`` fed to the logits.  ``detach_in_step`` cuts the gradient path of that step's flow_in messages;
    ``zero_below`` zeroes the loss gradient of label-0 logits below it (both deliberate defects)."""
    params, bufs = tto.split_state(d['P'])
    Pg = {k: v.detach().to(dtype, copy=True).requires_grad_(True) for k, v in params.items()}
    bufs = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in bufs.items()}
    calls = []
    real = tto.aggregate

    def agg(msg, index, n, how):
        calls.append(1)
        if detach_in_step is not None and len(calls) == 2 * detach_in_step:       # out, in, out, in, ...
            msg = msg.detach()
        return real(msg, index, n, how)
    tto.aggregate = agg
    try:
        out = tto.train_forward(Pg, d['mp'], d['x'].to(dtype), d['ei'], d['ea'].to(dtype), bufs, p, masks)
    finally:
        tto.aggregate = real
    lg = torch.stack([o.view(-1) for o in out])
    loss, g_lg, _, _ = bce_ref(lg.detach(), d['labels'], weight)
    if zero_below is not None:
        g_lg = torch.where((d['labels'].view(1, -1) == 0) & (lg.detach() < zero_below), 0.0, g_lg)
    torch.autograd.backward(lg, g_lg.to(dtype))
    return loss, {k: v.grad for k, v in Pg.items() if v.grad is not None}, lg.detach()


def row_bar_failures(got, ref64, ref32, bn_fed=(), slack=4.0, true64=None):
    """Names of the tensors with a row off the per-row bar: |got - ref64|_row <= slack |ref32 - true64|_row
    + 1e-5 max_row |ref64| (BatchNorm-fed biases: the absolute rule of test_training_options).  ``true64`` (default
    ``ref64``) is the unaltered fp64 reference that sets the CPU oracle's own error.  A bias counts as one row: its
    entries are single sums over the edges, where one CPU sample of the rounding error can be arbitrarily lucky."""
    true64 = ref64 if true64 is None else true64
    bad = {}
    for k, r in ref64.items():
        g = got[k].detach().double().cpu()
        if k in bn_fed:
            if float((g - r).abs().max()) > 1e-6 * float(ref64[k[:-4] + 'weight'].abs().max()):
                bad[k] = 'bn-fed bias'
            continue
        rows = r.shape[0] if r.dim() > 1 else 1        # a bias is one row: each entry is a single sum over the
        eg = (g - r).abs().reshape(rows, -1).amax(1)
        ec = (ref32[k].double() - true64[k]).abs().reshape(rows, -1).amax(1)
        scale = r.abs().reshape(rows, -1).amax(1)
        over = eg > slack * ec + 1e-5 * scale
        if over.any():
            i = int(((eg - slack * ec) / scale.clamp(min=1e-300)).argmax())
            bad[k] = f'{int(over.sum())} rows, worst row {i}: {float(eg[i]):.3g} vs cpu {float(ec[i]):.3g} of {float(scale[i]):.3g}'
    return bad


def gpu_grads(d, weight=1.0, seed=None):
    from mpntrackseg_b200.training import CoreTrainer
    tr = CoreTrainer(make_model(d['mp'], d['P']), seed=seed)
    data = make_data(d['x'], d['ei'], d['ea'])
    loss = tr.loss_and_grads(data, d['labels'].to(dev()), tracking_weight=weight)
    return tr, float(loss), {k: v.clone() for k, v in tr.g.items()}


def assert_loss_on_own_logits(tr, d, loss, weight=1.0):
    """The loss bar 16u loss, against the fp64 loss of the logits the trainer computed (no dropout or BatchNorm:
    a second forward gives the same logits)."""
    lg, ctx = tr.forward_core(make_data(d['x'], d['ei'], d['ea']))
    lab = d['labels'][ctx['sedge'].long().cpu()]
    ref = bce_ref(lg.cpu(), lab, weight)[0]
    assert abs(loss - ref) <= 16 * U * ref, (loss, ref)


ROW_CASES = [('tiny_nonrecip', None), ('tiny_mean', None), ('tiny_max', None)]


@pytest.mark.parametrize('name,agg', ROW_CASES)
def test_training_gradients_per_row_against_fp64(name, agg):
    d = load(name, agg=agg)
    if bool((d['labels'] == d['labels'][0]).all()):   # tiny_mean / tiny_max: every edge a true link, pw = 0 and a zero
        g = torch.Generator().manual_seed(5)          # loss gradient; a seeded 30 % of true links instead
        d['labels'] = (torch.rand(d['labels'].shape, generator=g) < 0.3).float()
    tr, loss, got = gpu_grads(d, 0.8)
    ref_loss, ref64, lg = oracle_grads(d, torch.float64, 0.8)
    _, ref32, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'], 0.8)
    assert set(ref64) == set(got) and all(bool((g != 0).any()) for g in ref64.values())
    assert_loss_on_own_logits(tr, d, loss, 0.8)
    assert abs(loss - ref_loss) <= tto.LOSS_TOL * ref_loss
    bad = row_bar_failures(got, ref64, ref32, bn_fed_biases(d['P']))
    assert not bad, bad
    # the bar sees a detached flow_in step (step 2 of 3 has flow_in messages in these graphs)
    _, alt, _ = oracle_grads(d, torch.float64, 0.8, detach_in_step=2)
    assert row_bar_failures(got, alt, ref32, true64=ref64), 'a detached flow_in step passed the per-row bar'


def test_training_gradients_per_row_with_dropout():
    d = load('tiny_nonrecip', p=0.3)
    from mpntrackseg_b200.training import CoreTrainer
    tr = CoreTrainer(make_model(d['mp'], d['P']), seed=1234)
    data = make_data(d['x'], d['ei'], d['ea'])
    loss, ctx = tto.step_with_masks(tr, data, d['labels'])
    masks = tto.slot_masks(ctx, d['ei'])
    assert ctx['masks'] and any(not bool(m.all()) for m in ctx['masks'].values())
    ref_loss, ref64, _ = oracle_grads(d, torch.float64, 1.0, p=0.3, masks=masks)
    _, ref32, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'], 1.0, p=0.3,
                                           masks=masks)
    bad = row_bar_failures(tr.g, ref64, ref32)
    assert not bad, bad
    assert abs(float(loss) - ref_loss) <= tto.LOSS_TOL * ref_loss


CLS_OUT_BIAS = 'classifier.edge_model.fc_layers.2.bias'


@pytest.mark.parametrize('bias', [-8.0, -12.0, -17.0, -24.0])
@pytest.mark.parametrize('agg', ['sum', 'max'])
def test_training_gradients_of_a_confident_all_negative_window(bias, agg):
    """No true link in the window (pw = 0) and a classifier that rejects every edge: the loss gradient of each logit
    is w / E e^x, which fp32 1 - s(-x) rounds to 0 below x = -17."""
    d = load('tiny_nonrecip', agg=agg)
    d['labels'] = torch.zeros_like(d['labels'])
    d['P'] = dict(d['P'])
    d['P'][CLS_OUT_BIAS] = torch.full_like(d['P'][CLS_OUT_BIAS], bias)
    tr, loss, got = gpu_grads(d)
    ref_loss, ref64, lg = oracle_grads(d, torch.float64)
    _, ref32, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'])
    below = float((lg < -17).double().mean())
    if bias == -17.0:
        assert below >= 0.04, below
    if bias == -24.0:
        assert below >= 0.9, below
    if below == 1.0:                                  # every gradient of the parent's formula is exactly 0
        assert all(bool((g != 0).any()) for g in ref64.values())
    assert_loss_on_own_logits(tr, d, loss)
    bad = row_bar_failures(got, ref64, ref32)
    assert not bad, bad
    if below > 0:                                     # the bar sees the loss gradient of x < -17 rounded to 0
        _, alt, _ = oracle_grads(d, torch.float64, zero_below=-17.0)
        assert row_bar_failures(got, alt, ref32, true64=ref64), 'zeroed confident gradients passed the per-row bar'


# ------------------------------------------------------------------ exact transport
def scaled(d, factors):
    d = dict(d)
    d['P'] = dict(d['P'])
    for k, f in factors.items():
        d['P'][k] = d['P'][k] * f
    return d


def assert_transported(base, got, factors, what):
    for k, g in base.items():
        f = factors.get(k, 1.0)
        assert torch.equal(got[k], g * f), (what, k, f)


def test_tracking_weight_scales_gradients_bit_for_bit():
    d = load('tiny_nonrecip')
    _, loss, base = gpu_grads(d, 0.8)
    assert all(bool((g != 0).any()) for g in base.values())
    for p in (-20, -3, 5, 20):
        _, l2, got = gpu_grads(d, 0.8 * 2.0 ** p)
        assert l2 == loss * 2.0 ** p
        assert_transported(base, got, {k: 2.0 ** p for k in base}, f'weight 2^{p}')


MLPS = ['MPNet.edge_model.edge_model', 'MPNet.node_model.flow_out_model', 'MPNet.node_model.flow_in_model',
        'classifier.edge_model']


@pytest.mark.parametrize('a', [-12, -8, 8, 12])
@pytest.mark.parametrize('mlp', MLPS, ids=['edge', 'flow_out', 'flow_in', 'classifier'])
def test_mlp_layer_balance_transports_exactly(mlp, a):
    d = load('tiny_nonrecip')
    _, _, base = gpu_grads(d)
    tr, _, _ = gpu_grads(d)
    base_lg, _ = tr.forward_core(make_data(d['x'], d['ei'], d['ea']))
    w0, b0, w1 = f'{mlp}.fc_layers.0.weight', f'{mlp}.fc_layers.0.bias', f'{mlp}.fc_layers.2.weight'
    ds = scaled(d, {w0: 2.0 ** a, b0: 2.0 ** a, w1: 2.0 ** -a})
    tr2, _, got = gpu_grads(ds)
    lg, _ = tr2.forward_core(make_data(d['x'], d['ei'], d['ea']))
    assert torch.equal(lg, base_lg)
    assert_transported(base, got, {w0: 2.0 ** -a, b0: 2.0 ** -a, w1: 2.0 ** a}, f'{mlp} 2^{a}')


@pytest.mark.parametrize('p', [-16, 12])
def test_node_feature_scale_transports_exactly(p):
    d = load('tiny_nonrecip')
    _, _, base = gpu_grads(d)
    w0 = 'encoder.node_model.fc_layers.0.weight'
    ds = scaled(d, {w0: 2.0 ** -p})
    ds['x'] = d['x'] * 2.0 ** p
    _, _, got = gpu_grads(ds)
    assert_transported(base, got, {w0: 2.0 ** p}, f'x 2^{p}')


@pytest.mark.parametrize('a', [-8, 12])
@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_flow_output_scale_transports_exactly(agg, a):
    d = load('tiny_nonrecip', agg=agg)
    _, _, base = gpu_grads(d)
    flows = [f'MPNet.node_model.flow_{s}_model.fc_layers.2.{t}' for s in ('in', 'out') for t in ('weight', 'bias')]
    node_w = 'MPNet.node_model.node_model.0.weight'
    ds = scaled(d, {**{k: 2.0 ** a for k in flows}, node_w: 2.0 ** -a})
    _, _, got = gpu_grads(ds)
    assert_transported(base, got, {**{k: 2.0 ** -a for k in flows}, node_w: 2.0 ** a}, f'flow {agg} 2^{a}')


# ------------------------------------------------------------------ segment mean / max and their gradients
def scatter_stub():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'torch_scatter_stub', 'torch_scatter',
                        '__init__.py')
    spec = importlib.util.spec_from_file_location('_scatter_stub', path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


SEG_LENS = [0, 1, 2, 1025, 30000, 3, 0, 2, 5]


def segment_case(width, seed, ties=False):
    """Rows of a [slots, ld] input and the node segments of SEG_LENS (one segment per special column pattern)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.tensor(SEG_LENS)
    seg_ptr = torch.zeros(len(SEG_LENS) + 1, dtype=torch.int32)
    seg_ptr[1:] = torch.cumsum(lens, 0).to(torch.int32)
    slots, ld, in_off = int(lens.sum()), width + 5, 3
    v = torch.randn(slots, ld, generator=g)
    if ties:
        v = torch.randint(-3, 3, (slots, ld), generator=g).float()
    # node 5 (3 slots): every value 0 (dead ReLUs); node 7 (2 slots): -0.0 then +0.0; node 8 (5 slots): all -inf
    s5, s7, s8 = int(seg_ptr[5]), int(seg_ptr[7]), int(seg_ptr[8])
    v[s5:s5 + 3] = 0.0
    v[s7] = -0.0
    v[s7 + 1] = 0.0
    v[s8:s8 + 5] = float('-inf')
    return v, seg_ptr, in_off


def run_segment(v, seg_ptr, perm, in_off, width, mode, accumulate, prev):
    from mpntrackseg_b200.ops import segment_sum
    nodes = seg_ptr.numel() - 1
    col_off = 2
    out = torch.full((nodes, width + 4), 7.0, device=dev())
    out[:, col_off:col_off + width] = prev.to(dev())
    arg = torch.full((nodes, width), -7, dtype=torch.int32, device=dev()) if mode == 'max' else None
    segment_sum(v.to(dev()), in_off, width, seg_ptr.to(dev()), None if perm is None else perm.to(dev()), out, col_off,
                accumulate=accumulate, mode=mode, argmax=arg)
    out = out.cpu()
    assert (out[:, :col_off] == 7).all() and (out[:, col_off + width:] == 7).all()
    return out[:, col_off:col_off + width], (arg.cpu() if arg is not None else None)


@pytest.mark.parametrize('width', [1, 32, 33])
@pytest.mark.parametrize('permuted', [False, True])
@pytest.mark.parametrize('accumulate', [False, True])
def test_segment_mean_against_fp64(width, permuted, accumulate):
    v, seg_ptr, in_off = segment_case(width, 5)
    v = torch.where(torch.isfinite(v), v, torch.zeros_like(v))
    slots = v.shape[0]
    perm = torch.randperm(slots, generator=torch.Generator().manual_seed(6)).to(torch.int32) if permuted else None
    prev = torch.randn(seg_ptr.numel() - 1, width) if accumulate else torch.zeros(seg_ptr.numel() - 1, width)
    got, _ = run_segment(v, seg_ptr, perm, in_off, width, 'mean', accumulate, prev)
    rows = (perm.long() if permuted else torch.arange(slots))
    x = v[rows][:, in_off:in_off + width].double()
    for node in range(seg_ptr.numel() - 1):
        q0, q1 = int(seg_ptr[node]), int(seg_ptr[node + 1])
        cnt = q1 - q0
        ref = (x[q0:q1].sum(0) / cnt if cnt else torch.zeros(width, dtype=torch.float64)) + prev[node].double()
        bar = (1e-5 * x[q0:q1].abs().sum(0) / max(cnt, 1)) + U * prev[node].double().abs()
        err = (got[node].double() - ref).abs()
        assert (err <= bar).all(), (node, cnt, float((err / bar.clamp(min=1e-300)).max()))
        if cnt == 0:
            assert torch.equal(got[node], prev[node])


@pytest.mark.parametrize('width', [1, 32, 33])
@pytest.mark.parametrize('permuted', [False, True])
@pytest.mark.parametrize('ties', [False, True])
def test_segment_max_and_argmax_bit_exact(width, permuted, ties):
    v, seg_ptr, in_off = segment_case(width, 7, ties)
    slots = v.shape[0]
    perm = torch.randperm(slots, generator=torch.Generator().manual_seed(8)).to(torch.int32) if permuted else None
    if perm is not None:                  # keep the special patterns inside their segments under the permutation
        v = v.clone()
        v[perm.long()] = v.clone()
    nodes = seg_ptr.numel() - 1
    for accumulate in (False, True):
        prev = torch.randn(nodes, width) if accumulate else torch.zeros(nodes, width)
        got, arg = run_segment(v, seg_ptr, perm, in_off, width, 'max', accumulate, prev)
        rows = perm.long() if permuted else torch.arange(slots)
        x = v[rows][:, in_off:in_off + width]                                  # slot order
        index = torch.repeat_interleave(torch.arange(nodes), seg_ptr[1:] - seg_ptr[:-1])
        _, pos = scatter_stub().scatter_max(x, index, dim_size=nodes)
        empty = pos == slots
        ref_arg = torch.where(empty, -1, rows[pos.clamp(max=slots - 1)])
        ref_val = torch.where(empty, 0.0, x.gather(0, pos.clamp(max=slots - 1)))
        assert torch.equal(arg.long(), ref_arg), 'argmax'
        ref = ref_val + prev if accumulate else ref_val
        assert torch.equal(got.view(torch.int32), ref.view(torch.int32)), 'max values (bits)'
    if ties:                                                 # the 1,025-slot segment holds its maximum more than once
        seg = x[int(seg_ptr[3]):int(seg_ptr[4])]
        assert int((seg == seg.max(0).values).sum(0).min()) > 1
    assert (arg[7] == rows[int(seg_ptr[7])]).all()           # -0.0 then +0.0: the first slot, and its -0.0
    assert (arg[8] == rows[int(seg_ptr[8])]).all()           # all -inf: the first slot
    assert (arg[0] == -1).all() and (arg[6] == -1).all()     # empty segments


@pytest.mark.parametrize('width', [1, 32, 33])
def test_segment_grad_of_a_flow_in_slot_range(width):
    """Slots [0, q0) form the flow_out groups, [q0, q1) the flow_in groups (q0 > 0): max sends g to the argmax slot
    exactly, mean divides it by the segment size."""
    from mpntrackseg_b200.ops import segment_sum
    from mpntrackseg_b200.training import segment_grad
    g_ = torch.Generator().manual_seed(9)
    nodes = 6
    out_len, in_len = torch.tensor([2, 0, 3, 1, 1025, 0]), torch.tensor([1, 30000, 0, 2, 3, 1])
    q0 = int(out_len.sum())
    out_ptr = torch.zeros(nodes + 1, dtype=torch.int32)
    out_ptr[1:] = torch.cumsum(out_len, 0)
    in_ptr = torch.zeros(nodes + 1, dtype=torch.int32)
    in_ptr[0] = q0
    in_ptr[1:] = q0 + torch.cumsum(in_len, 0)
    q1 = int(in_ptr[-1])
    row = torch.cat((torch.repeat_interleave(torch.arange(nodes), out_len),
                     torch.repeat_interleave(torch.arange(nodes), in_len))).to(torch.int32)
    msg = torch.randint(-2, 3, (q1, width), generator=g_).float()                 # ties inside segments
    gf = torch.randn(nodes, 2 * width + 3, generator=g_)                           # g: a strided column slice
    arg = torch.empty((nodes, width), dtype=torch.int32, device=dev())
    f = torch.empty((nodes, width), device=dev())
    segment_sum(msg.to(dev()), 0, width, in_ptr.to(dev()), None, f, 0, mode='max', argmax=arg)
    gdev = gf.to(dev())[:, 3:3 + width]
    for mode in ('max', 'mean'):
        out = torch.full((q1, width), 5.0, device=dev())
        segment_grad(gdev, row.to(dev()), in_ptr.to(dev()), arg, q0, q1, mode, out)
        out = out.cpu()
        assert (out[:q0] == 5).all()
        g = gf[:, 3:3 + width]
        r = row[q0:q1].long()
        if mode == 'max':
            q = torch.arange(q0, q1).view(-1, 1)
            ref = torch.where(arg.cpu()[r].long() == q, g[r], torch.zeros(()))
            assert torch.equal(out[q0:], ref)
            assert int((out[q0:] != 0).sum()) == int((in_len > 0).sum()) * width
        else:
            cnt = (in_len[r]).double().view(-1, 1)
            ref = g[r].double() / cnt
            assert ((out[q0:].double() - ref).abs() <= U * ref.abs()).all()


# ------------------------------------------------------------------ BatchNorm1d forward / backward
EPS = 1e-5


def bn_columns(m, n, seed):
    """z [m, n] whose columns cycle through the regimes: (|mu| / sigma, sigma) in {0, 1e2, 1e4} x {2^-20, 1, 2^20},
    constant columns, gamma = 0, and columns whose BN + ReLU output is all 0; returns z, gamma, beta, names."""
    g = torch.Generator().manual_seed(seed)
    kinds = [(r, s) for r in (0.0, 1e2, 1e4) for s in (2.0 ** -20, 1.0, 2.0 ** 20)] + ['const', 'gamma0', 'dead']
    z = torch.empty(m, n, dtype=torch.float64)
    gamma = (torch.rand(n, generator=g, dtype=torch.float64) + 0.5)
    beta = torch.randn(n, generator=g, dtype=torch.float64) * 0.3
    names = []
    for c in range(n):
        k = kinds[c % len(kinds)]
        names.append(k)
        base = torch.randn(m, generator=g, dtype=torch.float64)
        if k == 'const':
            z[:, c] = 0.1
        elif k in ('gamma0', 'dead'):
            z[:, c] = 3.0 + 2.0 * base
            if k == 'gamma0':
                gamma[c] = 0.0
            else:
                beta[c] = -1e3
        else:
            r, s = k
            z[:, c] = s * (r + base) * (-1.0 if c % 2 else 1.0)
    return z.float(), gamma.float(), beta.float(), names


def bn_forward(z, gamma, beta, momentum=0.1, rm=None, rv=None, nbt=None, ldy_pad=0, p=0.0):
    """mpn_batchnorm_forward on a strided z (and y); returns y, stats and the running buffers."""
    m, n = z.shape
    zs = torch.empty((m, n + 3), device=dev())[:, 1:1 + n]
    zs.copy_(z)
    y = torch.empty((m, n + ldy_pad), device=dev())[:, :n]
    stats = torch.empty((4, n), device=dev())
    rm = torch.zeros(n, device=dev()) if rm is None else rm
    rv = torch.ones(n, device=dev()) if rv is None else rv
    nbt = torch.zeros(1, dtype=torch.int64, device=dev()) if nbt is None else nbt
    gd, bd = gamma.to(dev()), beta.to(dev())                      # held until the kernels have run
    check(lib().mpn_batchnorm_forward(ptr(zs), zs.stride(0), m, n, ptr(gd), ptr(bd), EPS,
                                      momentum, ptr(rm), ptr(rv), ptr(nbt), ptr(stats), 0.0, 0, None, 0, ptr(y),
                                      y.stride(0), None, sptr()), 'batchnorm')
    return zs, y, stats, rm, rv, nbt


def bn_ref(z, gamma, beta, drop_rows=None, biased_running=False, no_eps=False):
    z = z.double()
    if drop_rows is not None:
        keep = torch.ones(z.shape[0], dtype=torch.bool)
        keep[drop_rows] = False
        zz = z[keep]
    else:
        zz = z
    mu = zz.mean(0)
    var = ((zz - mu) ** 2).mean(0)
    invstd = 1.0 / torch.sqrt(var + (0.0 if no_eps else EPS))
    y = torch.relu(gamma.double() * (z - mu) * invstd + beta.double())
    m = zz.shape[0]
    unb = var if biased_running else var * m / (m - 1)
    return y, mu, var, invstd, unb


def y_bar(gamma, mu, invstd, y_ref):
    return 2.0 ** -17 * gamma.double().abs() * (1 + mu.abs() * invstd) + 4 * U * y_ref.abs()


def y_ok(y, ref, gamma):
    yr, mu, _, invstd, _ = ref
    return bool(((y.double() - yr).abs() <= y_bar(gamma, mu, invstd, yr)).all())


BN_M = [2, 3, 255, 256, 257, 32768, 32769, 10 ** 6]


@pytest.mark.parametrize('m', BN_M)
def test_batchnorm_forward_against_fp64(m):
    ns = [33] if m == 10 ** 6 else [1, 16, 31, 32, 33, 80]
    for n in ns:
        z, gamma, beta, names = bn_columns(m, n, seed=m + n)
        zs, y, stats, rm, rv, nbt = bn_forward(z, gamma, beta, ldy_pad=5)
        y = y.cpu()
        ref = bn_ref(z, gamma, beta)
        yr, mu, var, invstd, unb = ref
        err = (y.double() - yr).abs() / y_bar(gamma, mu, invstd, yr).clamp(min=1e-300)
        assert y_ok(y, ref, gamma), (m, n, names[int(err.amax(0).argmax())], float(err.max()))
        for c, k in enumerate(names):
            if k == 'dead':
                assert (y[:, c] == 0).all()
            if k == 'gamma0':
                assert (y[:, c] == torch.relu(beta[c])).all()
        assert int(nbt) == 1
        # running statistics (momentum 0.1 from 0 / 1) with the unbiased variance
        assert ((rm.cpu().double() - 0.1 * mu).abs() <= 0.1 * 2.0 ** -17 * (mu.abs() + var.sqrt()) + 1e-30).all()
        rv_bar = 2.0 ** -17 * (0.9 + 0.1 * unb) + 0.2 * 2.0 ** -34 * mu * mu * m / (m - 1)   # + (error of mean)^2
        assert ((rv.cpu().double() - (0.9 + 0.1 * unb)).abs() <= rv_bar).all()
        if m > BN_SLICE_ROWS and n == 33:             # the bars see one dropped row slice, a biased var, no eps
            slices = min(-(-m // BN_SLICE_ROWS), BN_SLICES)
            rps = -(-m // slices)
            assert not y_ok(y, bn_ref(z, gamma, beta, drop_rows=slice(rps, 2 * rps)), gamma)
            assert not y_ok(y, bn_ref(z, gamma, beta, no_eps=True), gamma)
            unb_b = bn_ref(z, gamma, beta, biased_running=True)[4]
            if m < 10 ** 5:                           # beyond, m / (m - 1) is under the running_var bar
                assert not ((rv.cpu().double() - (0.9 + 0.1 * unb_b)).abs() <= rv_bar).all()


@pytest.mark.parametrize('momentum', [0.1, 0.5])
def test_batchnorm_running_statistics_over_calls(momentum):
    """Five calls of m = 257, 2, 0, 32,769, 3 through training._Linear against nn.BatchNorm1d in fp64."""
    from mpntrackseg_b200.training import _Linear
    n, k = 33, 20
    g = torch.Generator().manual_seed(21)
    w, b = torch.randn(n, k, generator=g) * 0.3, torch.randn(n, generator=g)
    mod = torch.nn.BatchNorm1d(n, momentum=momentum).to(dev())
    ref = torch.nn.BatchNorm1d(n, momentum=momentum).double()
    with torch.no_grad():
        mod.weight.uniform_(0.5, 1.5)
        mod.bias.uniform_(-0.5, 0.5)
        ref.weight.copy_(mod.weight.double())
        ref.bias.copy_(mod.bias.double())
    ref.train()
    gw, gb = torch.zeros(n, k, device=dev()), torch.zeros(n, device=dev())
    bn = dict(mod=mod, gamma=mod.weight.data, beta=mod.bias.data, ggamma=torch.zeros(n, device=dev()),
              gbeta=torch.zeros(n, device=dev()))
    lin = _Linear(w.to(dev()), b.to(dev()), True, gw, gb, bn=bn)
    for m in (257, 2, 0, 32769, 3):
        x = torch.randn(m, k, generator=g) * 4 + 1
        y, (z, _) = lin.fwd(x.to(dev()))
        with torch.no_grad():
            yr = torch.relu(ref(z.cpu().double()))
        assert int(mod.num_batches_tracked) == int(ref.num_batches_tracked), m
        sd = (ref.running_var.abs().sqrt() + ref.running_mean.abs())
        assert ((mod.running_mean.cpu().double() - ref.running_mean).abs() <= 2.0 ** -17 * sd).all(), m
        assert ((mod.running_var.cpu().double() - ref.running_var).abs() <= 2.0 ** -17 * ref.running_var).all(), m
        if m:
            mu = z.cpu().double().mean(0)
            invstd = 1 / torch.sqrt(z.cpu().double().var(0, unbiased=False) + EPS)
            assert ((y.cpu().double() - yr).abs() <= y_bar(mod.weight.detach().cpu(), mu, invstd, yr)).all(), m


def bn_backward_ref(z, g, y, gamma, gscale):
    z, g, y = z.double(), g.double(), y.double()
    m = z.shape[0]
    mu = z.mean(0)
    invstd = 1 / torch.sqrt(((z - mu) ** 2).mean(0) + EPS)
    xhat = (z - mu) * invstd
    gp = torch.where(y > 0, g * gscale, 0.0)
    a, bb = gp.mean(0), (gp * xhat).mean(0)
    gz = gamma.double() * invstd * (gp - a - xhat * bb)
    c = 1 + mu.abs() * invstd                                       # cancellation factor of z - mean
    bar = 2.0 ** -17 * gamma.double().abs() * invstd * c * (gp.abs() + (1 + xhat.abs()) * (gp.abs().mean(0) + (gp * xhat).abs().mean(0)))
    return gz, bar, gp.sum(0), (gp * xhat).sum(0), gp.abs().sum(0), (c * gp.abs() * (1 + xhat.abs())).sum(0)


@pytest.mark.parametrize('m', [2, 3, 257, 32769, 10 ** 6])
@pytest.mark.parametrize('p', [0.0, 0.3])
def test_batchnorm_backward_against_fp64(m, p):
    n = 33
    z, gamma, beta, names = bn_columns(m, n, seed=100 + m)
    zs, y, stats, _, _, _ = bn_forward(z, gamma, beta)
    g = torch.randn(m, n, generator=torch.Generator().manual_seed(m))
    gs = torch.empty((m, n + 2), device=dev())[:, 2:]
    gs.copy_(g)
    gscale = 1.0 / (1.0 - p)
    ggamma0, gbeta0 = torch.randn(n), torch.randn(n)
    ggamma, gbeta = ggamma0.to(dev()), gbeta0.to(dev())
    gz = torch.empty((m, n + 1), device=dev())[:, :n]
    gd = gamma.to(dev())
    check(lib().mpn_batchnorm_backward(ptr(zs), zs.stride(0), ptr(gs), gs.stride(0), ptr(y), y.stride(0), m, n,
                                       ptr(gd), ptr(stats), gscale, ptr(ggamma), ptr(gbeta), ptr(gz),
                                       gz.stride(0), sptr()), 'batchnorm_backward')
    gz, y = gz.cpu(), y.cpu()
    ref, bar, sb, sg, sabs, sgx = bn_backward_ref(z, g, y, gamma, float(np.float32(gscale)))
    err = (gz.double() - ref).abs()
    assert (err <= bar + 4 * U * ref.abs()).all(), (m, names[int((err / bar.clamp(min=1e-300)).amax(0).argmax())])
    for c, k in enumerate(names):
        if k in ('dead', 'gamma0'):
            assert (gz[:, c] == 0).all(), k
    gbar = 2.0 ** -17 * sabs + U * gbeta0.double().abs()
    assert ((gbeta.cpu().double() - (gbeta0.double() + sb)).abs() <= gbar).all()
    assert ((ggamma.cpu().double() - (ggamma0.double() + sg)).abs() <= 2.0 ** -17 * sgx + U * ggamma0.double().abs()).all()


# ------------------------------------------------------------------ dropout
def dropout_mask(m, n, p, seed=5, counter=0, call=0, ldy_pad=0):
    y = torch.ones((m, n + ldy_pad), device=dev())[:, :n]
    cnt = torch.tensor([counter], dtype=torch.int64, device=dev())
    mask = torch.empty((m, n), dtype=torch.uint8, device=dev())
    check(lib().mpn_dropout_forward(ptr(y), y.stride(0), m, n, p, seed, ptr(cnt), call, ptr(mask), sptr()), 'dropout')
    return mask, y


P_DROP = [0.1, 0.5, 0.9, 1 - 2.0 ** -10]


@pytest.mark.parametrize('p', P_DROP)
def test_dropout_fraction_is_the_24_bit_threshold(p):
    m, n = 78125, 128                                     # 10^7 elements
    mask, _ = dropout_mask(m, n, p)
    N = m * n
    q = math.ceil(float(np.float32(p)) * 2 ** 24) / 2 ** 24
    frac = 1 - float(mask.double().mean())
    assert abs(frac - q) <= 5 * math.sqrt(q * (1 - q) / N), (p, frac, q)


def corr(a, b):
    a, b = a.double().view(-1), b.double().view(-1)
    a, b = a - a.mean(), b - b.mean()
    return float((a * b).sum() / torch.sqrt((a * a).sum() * (b * b).sum()))


def test_dropout_masks_are_uncorrelated():
    m, n = 10 ** 6, 16
    base, _ = dropout_mask(m, n, 0.5)
    flat = base.view(-1, 4)                                # the four elements of one Philox draw
    N = flat.shape[0]
    for i in range(4):
        for j in range(i + 1, 4):
            assert abs(corr(flat[:, i], flat[:, j])) <= 5 / math.sqrt(N), (i, j)
    nxt_call, _ = dropout_mask(m, n, 0.5, call=1)
    nxt_fwd, _ = dropout_mask(m, n, 0.5, counter=1)
    for other in (nxt_call, nxt_fwd):
        assert abs(corr(base, other)) <= 5 / math.sqrt(base.numel())


@pytest.mark.parametrize('p', [0.3, 1 - 2.0 ** -10])
def test_dropout_forward_and_backward_bit_exact(p):
    m, n = 4099, 33
    g = torch.Generator().manual_seed(17)
    relu = torch.relu(torch.randn(m, n, generator=g))
    ys = torch.empty((m, n + 7), device=dev())[:, 2:2 + n]
    ys.copy_(relu)
    yc = relu.to(dev()).contiguous()
    cnt = torch.tensor([3], dtype=torch.int64, device=dev())
    masks = []
    for y in (ys, yc):
        mask = torch.empty((m, n), dtype=torch.uint8, device=dev())
        check(lib().mpn_dropout_forward(ptr(y), y.stride(0), m, n, p, 77, ptr(cnt), 2, ptr(mask), sptr()), 'dropout')
        masks.append(mask.cpu())
    assert torch.equal(masks[0], masks[1])                       # strided y: the mask of the contiguous y
    assert torch.equal(ys.cpu(), yc.cpu())
    keep = masks[0].bool()
    assert keep.any() and not keep.all()
    one_minus_p = torch.tensor(1.0, dtype=torch.float32) - torch.tensor(p, dtype=torch.float32)
    ref = torch.where(keep, relu / one_minus_p, torch.zeros(()))
    assert torch.equal(yc.cpu(), ref)
    gy = torch.randn(m, n, generator=g)
    scale = 1.0 / (1.0 - p)
    out = torch.empty((m, n + 3), device=dev())[:, :n]
    gys = torch.empty((m, n + 1), device=dev())[:, 1:]
    gys.copy_(gy)
    check(lib().mpn_dropout_backward(ptr(gys), gys.stride(0), ptr(ys), ys.stride(0), m, n, scale, ptr(out),
                                     out.stride(0), sptr()), 'dropout_backward')
    ref_g = torch.where(yc.cpu() > 0, gy * torch.tensor(scale, dtype=torch.float32), torch.zeros(()))
    assert torch.equal(out.cpu(), ref_g)
