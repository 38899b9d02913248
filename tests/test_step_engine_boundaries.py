"""GPU tests of the message-passing step engines across input scale, layer balance and non-finite values, against
the oracle evaluated in fp64.

The other suites judge states with 1e-3 * max(1, row max) and logits with 1e-3 * max(1, |logit|): below 1 those bars
are absolute, so they cannot see an engine lose relative accuracy on small inputs.  Here the parameters are
transformed without changing the function the network computes (it is positively homogeneous between its biases),
the result is transported back and judged with the same bars against one fp64 oracle run per (graph, aggregation):

A. x0, e0 and every bias of the step loop and the classifier x 2^p: the exact answer is 2^p x the answer at p = 0;
B. one layer's weights and bias x 2^a, the next layer's weights x 2^-a: the same function;
C. a NaN or +-inf in one row of x0 / e0, one weight, each bias;
D. all-zero inputs, every hidden ReLU dead, and a circulant graph whose interior rows must agree bit for bit;
E. the S_RESOLVED boundary of the step scale;
F. loops of one and two steps.

'tc' either meets the bar or is flagged, and a flag needs a cause the test names from the code's own rules (the
schedule read back with debug=True, the small-input rule, the weight-packing rule): status bit 2 when a step runs at
s_t > S_RESOLVED or the constant x_init / e_init rows sit below the resolution floor, bit 1 when a weight has no
finite fp16 image in its slab, a bias or any input is not finite.  A flagged forward raises under 'tc'; 'auto' warns
and returns the 'fp32' result bit for bit.
"""
import math
import warnings

import numpy as np
import pytest
import torch

from mpntrackseg_b200 import ops, synth
from test_cuda_parity import assert_logits_close, dev, make_model
from test_kernel_boundaries import (S_RESOLVED, TC_TILE, _batch, _mixed_batch, assert_rows_close, model_params,
                                    oracle_steps, sms)

pytestmark = pytest.mark.gpu

STEPS, FIRST = 12, 2
INIT_SHIFT = 8              # csrc/mp_step_tc.cu: x_init / e_init are stored x 2^-8, their weight slabs carry 2^(8 - s_t)
FP16_LIMIT = 65000.0        # csrc/mp_step_tc.cu: the range check of the split operands and of the weight image
INIT_FLOOR = 2.0 ** (S_RESOLVED - 34)   # smallest stored max |x_init|, |e_init| the constant rows resolve (DESIGN §4)

EW = 'MPNet.edge_model.edge_model.fc_layers'
FI = 'MPNet.node_model.flow_in_model.fc_layers'
FO = 'MPNet.node_model.flow_out_model.fc_layers'
NM = 'MPNet.node_model.node_model.0'
CL = 'classifier.edge_model.fc_layers'
STEP_BIASES = [f'{EW}.0.bias', f'{EW}.2.bias', f'{FI}.0.bias', f'{FI}.2.bias', f'{FO}.0.bias', f'{FO}.2.bias',
               f'{NM}.bias', f'{CL}.0.bias', f'{CL}.2.bias']


# ------------------------------------------------------------------ the weight-packing rule of pack_weights_kernel
def _slab_factors():
    """{parameter: [(column slice, factor)]}: the power of two each packed weight carries in its fp16 slab (the
    constant-row slabs 2^INIT_SHIFT at s_t = 0), None for weights used in fp32 only (finiteness is all they need)."""
    c = 2.0 ** INIT_SHIFT
    return {f'{EW}.0.weight': [(slice(0, 32), None), (slice(32, 64), 1.0), (slice(64, 96), c), (slice(96, 128), 1.0),
                               (slice(128, 144), c), (slice(144, 160), 1.0)],
            f'{EW}.2.weight': [(slice(None), 1.0)],
            f'{FI}.0.weight': [(slice(0, 32), c), (slice(32, 80), 1.0)], f'{FI}.2.weight': [(slice(None), 1.0)],
            f'{FO}.0.weight': [(slice(0, 32), c), (slice(32, 80), 1.0)], f'{FO}.2.weight': [(slice(None), 1.0)],
            f'{NM}.weight': [(slice(None), 1.0)], f'{CL}.0.weight': [(slice(None), 1.0)],
            f'{CL}.2.weight': [(slice(None), None)]}


def packing_flag(P):
    """True when pack_weights_kernel must set status bit 1: a weight whose fp16 image times its slab factor is not
    below 65,000, or a non-finite weight or bias."""
    for name, parts in _slab_factors().items():
        w = P[name].double()
        for cols, f in parts:
            v = w[:, cols]
            if not torch.isfinite(v).all() or (f is not None and float(v.abs().max()) * f >= FP16_LIMIT):
                return True
    return any(not torch.isfinite(P[b]).all() for b in STEP_BIASES)


def small_input_flag(x0, e0):
    """True when the largest stored constant row |x_init|, |e_init| x 2^-INIT_SHIFT lies below the floor (status bit 2)."""
    m = max(float(x0.abs().max()), float(e0.abs().max())) * 2.0 ** -INIT_SHIFT
    return 0.0 < m < INIT_FLOOR


# ------------------------------------------------------------------ running the engines
class Graph:
    """One edge layout reused for every forward on the graph; edge tensors in the caller's order."""

    def __init__(self, ei, n):
        self.ei, self.n = ei, n
        self.lay = ops.edge_layout(ei.to(dev()), n)
        self.sedge = self.lay.slot_edge[:self.lay.num_edges].long()

    def run(self, model, x0, e0, engine, steps=STEPS, first=FIRST):
        """(logits [S, E], node state, edge state, status) with status = the tensor-core status word ('tc': no
        raise; None for the other engines)."""
        cw, keep = model.core_weights()
        st = torch.zeros(1, dtype=torch.int32, device=dev()) if engine == 'tc' else None
        with torch.no_grad():
            lg, xs, es = ops.mp_forward(cw, self.lay, x0.to(dev()), e0.to(dev())[self.sedge].contiguous(), steps, first,
                                        want_state=True, engine=engine, status=st, debug=engine == 'tc')
        e_state = torch.empty_like(es)
        e_state[self.sedge] = es
        del keep
        return lg.cpu(), xs.cpu(), e_state.cpu(), None if st is None else int(st.item())

    def raising(self, model, x0, e0, steps=STEPS, first=FIRST):
        """'tc' raises OverflowError; 'auto' warns and returns 'fp32' bit for bit; returns the 'fp32' result."""
        with pytest.raises(OverflowError):
            self.forward(model, x0, e0, 'tc', steps, first)
        ref = self.forward(model, x0, e0, 'fp32', steps, first)
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter('always')
            got = self.forward(model, x0, e0, 'auto', steps, first)
        assert any('fp16 range' in str(w.message) for w in caught), 'auto reruns on fp32 with a warning'
        assert all(bits_equal(a, b) for a, b in zip(got, ref)), "'auto' differs from 'fp32'"
        return ref

    def forward(self, model, x0, e0, engine, steps=STEPS, first=FIRST):
        cw, keep = model.core_weights()
        with torch.no_grad():
            lg, xs, es = ops.mp_forward(cw, self.lay, x0.to(dev()), e0.to(dev())[self.sedge].contiguous(), steps, first,
                                        want_state=True, engine=engine)
        e_state = torch.empty_like(es)
        e_state[self.sedge] = es
        del keep
        return lg.cpu(), xs.cpu(), e_state.cpu()


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def max_sched(steps=STEPS):
    return max(ops.LAST_TC_SCHEDULE['sched'][1:steps + 1])


def check(ref, got, what, scale=1.0):
    """got / scale against the fp64 reference with the suite's bars."""
    lg, xs, es = got[:3]
    assert_logits_close(lg.double().numpy() / scale, ref[0].numpy(), what)
    assert_rows_close(xs.double() / scale, ref[1], what + ' node state')
    assert_rows_close(es.double() / scale, ref[2], what + ' edge state')


def worst(ref, got, scale=1.0):
    """Largest error over the three outputs, in units of the bar (> 1: fails)."""
    out = []
    for i, (g, r) in enumerate(zip(got[:3], ref)):
        g = g.double().reshape(r.shape[0], -1) / scale
        r = r.double().reshape(r.shape[0], -1)
        bar = 1e-3 * (r.abs().clamp(min=1.0) if i == 0 else r.abs().amax(dim=1, keepdim=True).clamp(min=1.0))
        out.append(float(((g - r).abs() / bar).nan_to_num(float('inf')).max()))
    return max(out)


# ------------------------------------------------------------------ the main graph and its oracles (one per aggregation)
_CACHE = {}


def main_case(agg):
    if 'base' not in _CACHE:
        mp, P, blocks = _mixed_batch()
        ei, n, x0, e0 = _batch(blocks, [1.0] * 4)
        _CACHE['base'] = (P, blocks, Graph(ei, n), x0, e0)
    P, blocks, g, x0, e0 = _CACHE['base']
    mp = model_params(STEPS, agg)
    if agg not in _CACHE:
        _CACHE[agg] = oracle_steps(P, mp, g.ei, x0, e0)
    return mp, P, g, x0, e0, _CACHE[agg]


def scaled(P, factors):
    """A copy of P with the named tensors (or column ranges) multiplied by powers of two."""
    Q = {k: v.clone() for k, v in P.items()}
    for name, cols, f in factors:
        if cols is None:
            Q[name] *= f
        else:
            Q[name][:, cols] *= f
    return Q


# ================================================================== A. input scale
P_SCALES = [-24, -20, -16, -12, -8, -4, 0, 4, 8, 12]


@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_input_scale_transports_to_the_unscaled_oracle(agg):
    mp, P, g, x0, e0, ref = main_case(agg)
    model = make_model(mp, P)
    base32 = g.forward(model, x0, e0, 'fp32')
    for p in P_SCALES:
        f = 2.0 ** p
        Pp = scaled(P, [(b, None, f) for b in STEP_BIASES])
        model.load_state_dict(Pp, strict=False)
        xp, ep = x0 * f, e0 * f
        what = f'{agg} x 2^{p}'
        got32 = g.forward(model, xp, ep, 'fp32')
        assert all(bits_equal(a, b * f) for a, b in zip(got32, base32)), f'{what}: fp32 is not 2^p x its p = 0 result'
        got = g.run(model, xp, ep, 'tc')
        st, sched = got[3], max_sched()
        if st == 0:
            check(ref, got, f'{what} tc', scale=f)
            continue
        assert p != 0, f'{what}: the unscaled forward is flagged ({st})'
        if st & 2:
            assert sched > S_RESOLVED or small_input_flag(xp, ep), f'{what}: bit 2 without a cause, max s_t = {sched}'
        if st & 1:
            assert packing_flag(Pp), f'{what}: bit 1 without a weight outside its slab range'
        g.raising(model, xp, ep)


# ================================================================== B. layer balance
BALANCE_PAIRS = {
    'edge': ([(f'{EW}.0.weight', None), (f'{EW}.0.bias', None)], [(f'{EW}.2.weight', None)]),
    'flow_in': ([(f'{FI}.0.weight', None), (f'{FI}.0.bias', None)], [(f'{FI}.2.weight', None)]),
    'flow_out': ([(f'{FO}.0.weight', None), (f'{FO}.0.bias', None)], [(f'{FO}.2.weight', None)]),
    'classifier': ([(f'{CL}.0.weight', None), (f'{CL}.0.bias', None)], [(f'{CL}.2.weight', None)]),
    # both flow MLPs' outputs -> the node Linear's flow_in (0:32) and flow_out (32:64) columns; crosses FLOW_SHIFT
    'flow_to_node': ([(f'{FI}.2.weight', None), (f'{FI}.2.bias', None), (f'{FO}.2.weight', None),
                      (f'{FO}.2.bias', None)], [(f'{NM}.weight', slice(0, 64))]),
}
BALANCE_CASES = [(pair, 'sum') for pair in BALANCE_PAIRS] + [('flow_to_node', 'max')]


@pytest.mark.parametrize('pair,agg', BALANCE_CASES)
def test_layer_balance_keeps_the_function(pair, agg):
    mp, P, g, x0, e0, ref = main_case(agg)
    model = make_model(mp, P)
    base32 = g.forward(model, x0, e0, 'fp32')
    up, down = BALANCE_PAIRS[pair]
    for a in (-12, -8, 8, 12):
        f = 2.0 ** a
        Q = scaled(P, [(k, c, f) for k, c in up] + [(k, c, 1.0 / f) for k, c in down])
        model.load_state_dict(Q, strict=False)
        what = f'{pair} {agg} a={a}'
        # every product of the pair is exact in fp32, so the fp32 engine does not move at all
        assert all(bits_equal(x, y) for x, y in zip(g.forward(model, x0, e0, 'fp32'), base32)), f'{what}: fp32 moved'
        expect = packing_flag(Q)
        got = g.run(model, x0, e0, 'tc')
        if expect:
            assert got[3] & 1, f'{what}: a weight outside its slab range and no status bit 1'
            g.raising(model, x0, e0)
        else:
            assert got[3] == 0, f'{what}: flagged ({got[3]}, max s_t = {max_sched()}) with every weight in range'
            check(ref, got, f'{what} tc')


def test_packing_rule_sees_only_the_slab_factor():
    """The rule the tests above assume: 2^INIT_SHIFT for the constant-row slabs only, every block of edge_w0."""
    _, P, _, _, _, _ = main_case('sum')
    assert not packing_flag(P)
    assert packing_flag(scaled(P, [(f'{EW}.0.weight', slice(64, 96), 2.0 ** 12)]))     # 0.1 x 2^12 x 2^8 > 65,000
    assert not packing_flag(scaled(P, [(f'{EW}.0.weight', slice(96, 128), 2.0 ** 12)]))
    assert not packing_flag(scaled(P, [(f'{EW}.2.weight', None, 2.0 ** 12)]))
    assert packing_flag(scaled(P, [(f'{EW}.0.weight', slice(32, 64), 2.0 ** 20)]))


# ================================================================== C. non-finite values
def _neighbourhoods(ei, n, nodes, edges, steps):
    """Per step t = 1..steps: (nodes, edges) a bad value in the given node rows of x0 / edge rows of e0 can reach."""
    src, dst = ei
    bad_n = torch.zeros(n, dtype=torch.bool)
    bad_n[nodes] = True
    bad_e = torch.zeros(ei.shape[1], dtype=torch.bool)
    out = []
    for _ in range(steps):
        bad_e = bad_e | bad_n[src] | bad_n[dst]
        bad_e[edges] = True                                                   # e_init is reattached every step
        nb = bad_n.clone()
        nb[src[bad_e]] = True
        bad_n = nb
        out.append((bad_n.clone(), bad_e.clone()))
    return out


NONFINITE = [float('nan'), float('inf'), -float('inf')]
WEIGHT_SPOTS = [(f'{EW}.0.weight', (7, c)) for c in (5, 40, 70, 100, 130, 150)] + [
    (f'{EW}.2.weight', (3, 11)), (f'{FI}.0.weight', (9, 20)), (f'{FI}.2.weight', (4, 50)), (f'{FO}.0.weight', (2, 70)),
    (f'{FO}.2.weight', (31, 0)), (f'{NM}.weight', (6, 33)), (f'{CL}.0.weight', (5, 15)), (f'{CL}.2.weight', (0, 7))]


def test_nonfinite_input_rows_stay_in_their_neighbourhood():
    mp, P, g, x0, e0, ref = main_case('sum')
    model = make_model(mp, P)
    r, q = 17, int((g.ei[0] == 4000).nonzero()[0])                          # a node of window 0, an edge of window 2
    for kind, row in (('x0', r), ('e0', q)):
        reach = _neighbourhoods(g.ei, g.n, [r] if kind == 'x0' else [], [q] if kind == 'e0' else [], STEPS)
        last_n, last_e = reach[-1]
        assert (~last_n).sum() > g.n // 2, 'the bad value must leave most of the batch untouched'
        for v in NONFINITE:
            xb, eb = x0.clone(), e0.clone()
            (xb if kind == 'x0' else eb)[row, 3] = v
            what = f'{kind}[{row}] = {v}'
            got = g.raising(model, xb, eb)
            for i, t in enumerate(range(FIRST, STEPS + 1)):
                keep = ~reach[t - 1][1]
                assert_logits_close(got[0][i][keep].numpy(), ref[0][i][keep].numpy(), f'{what} step {t}')
            assert_rows_close(got[1][~last_n], ref[1][~last_n], f'{what} node state')
            assert_rows_close(got[2][~last_e], ref[2][~last_e], f'{what} edge state')


@pytest.mark.parametrize('spot', range(len(WEIGHT_SPOTS) + len(STEP_BIASES)))
def test_nonfinite_weight_or_bias_is_flagged(spot):
    mp, P, g, x0, e0, _ = main_case('sum')
    if spot < len(WEIGHT_SPOTS):
        name, idx = WEIGHT_SPOTS[spot]
    else:
        name, idx = STEP_BIASES[spot - len(WEIGHT_SPOTS)], (0,)
    model = make_model(mp, P)
    for v in NONFINITE:
        Q = {k: t.clone() for k, t in P.items()}
        Q[name][idx] = v
        assert packing_flag(Q)
        model.load_state_dict(Q, strict=False)
        got = g.run(model, x0, e0, 'tc')
        assert got[3] & 1, f'{name}{list(idx)} = {v}: no status bit 1'
        g.raising(model, x0, e0)


# ================================================================== D. degenerate and invariant states
@pytest.mark.parametrize('agg', ['sum', 'max'])
def test_zero_inputs(agg):
    mp, P, g, x0, e0, _ = main_case(agg)
    z0, ze = torch.zeros_like(x0), torch.zeros_like(e0)
    ref = oracle_steps(P, mp, g.ei, z0, ze)
    model = make_model(mp, P)
    got = g.run(model, z0, ze, 'tc')
    assert got[3] == 0, f'zero inputs flagged ({got[3]})'
    check(ref, got, f'zero {agg} tc')
    check(ref, g.forward(model, z0, ze, 'fp32'), f'zero {agg} fp32')


def test_dead_hidden_layers_give_the_later_biases():
    """Every layer-0 bias at -100: each hidden ReLU is dead, the logits are exactly the classifier's output bias and
    the edge state is ReLU of the edge MLP's output bias."""
    mp, P, g, x0, e0, _ = main_case('mean')
    Q = {k: v.clone() for k, v in P.items()}
    for name in (f'{EW}.0.bias', f'{FI}.0.bias', f'{FO}.0.bias', f'{CL}.0.bias'):
        Q[name].fill_(-100.0)
    ref = oracle_steps(Q, mp, g.ei, x0, e0)
    b_cls = float(Q[f'{CL}.2.bias'][0])
    assert bool((ref[0] == b_cls).all()), 'the oracle case must have every classifier ReLU dead'
    assert bool((ref[2] == Q[f'{EW}.2.bias'].double().clamp(min=0)).all()), 'every edge-MLP ReLU must be dead'
    model = make_model(mp, Q)
    for engine in ('tc', 'fp32'):
        got = g.run(model, x0, e0, engine)
        if engine == 'tc':
            assert got[3] == 0
        assert bool((got[0] == torch.tensor(b_cls, dtype=torch.float32)).all()), f'{engine}: logits != b_cls'
        check(ref, got, f'dead ReLUs {engine}')


def _circulant(n):
    """Node i links to i +- 1 and i +- 2 (mod n), listed offset by offset so that every row sees its slots in the
    same order."""
    i = torch.arange(n)
    return torch.cat([torch.stack((i, (i + d) % n)) for d in (1, 2, -1, -2)], dim=1)


@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_circulant_interior_rows_are_bit_identical(agg):
    """Equal x0 on every node, equal e0 on every edge: rows farther than 2 * steps + 2 from the wrap compute the same
    thing, so any lane-, tile-, granule- or swizzle-dependent error shows up as a difference of bits."""
    n = 3 * sms() * TC_TILE + 77
    assert n > 2 * sms() * TC_TILE and n % TC_TILE != 0
    ei = _circulant(n)
    g = Graph(ei, n)
    mp = model_params(STEPS, agg)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    model = make_model(mp, P)
    gen = torch.Generator().manual_seed(5)
    x0 = (torch.rand(1, 32, generator=gen) * 2).expand(n, 32).contiguous()
    e0 = (torch.rand(1, 16, generator=gen) * 2).expand(ei.shape[1], 16).contiguous()
    margin = 2 * STEPS + 2
    inner = torch.arange(margin, n - margin)
    for engine in ('tc', 'fp32'):
        lg, xs, es, st = g.run(model, x0, e0, engine)
        if engine == 'tc':
            assert st == 0, f'{agg}: flagged ({st})'
        assert torch.isfinite(xs).all() and xs[inner].abs().max() > 0
        assert (xs[inner] == xs[inner[0]]).all(), f'{agg} {engine}: interior node rows differ'
        es = es.view(4, n, 16)
        lg = lg.view(lg.shape[0], 4, n)
        for d in range(4):
            assert (es[d, inner] == es[d, inner[0]]).all(), f'{agg} {engine}: interior edge rows differ (offset {d})'
            assert (lg[:, d, inner] == lg[:, d, inner[0], None]).all(), f'{agg} {engine}: interior logits differ'


# ================================================================== E. the S_RESOLVED boundary
def test_step_scale_resolution_boundary():
    """The loud window's x0 x 2^k for the k at which the schedule peaks at exactly S_RESOLVED: not flagged, the quiet
    windows meet the bar; at the next k the schedule passes S_RESOLVED and the forward is flagged."""
    mp, P, blocks = _mixed_batch()
    model = make_model(mp, P)
    peaks = {}
    k = 0
    while True:
        ei, n, x0, e0 = _batch(blocks, [1.0, 2.0 ** k, 1.0, 1.0])
        g = Graph(ei, n)
        got = g.run(model, x0, e0, 'tc')
        peaks[k] = (max_sched(), got[3], g, x0, e0, got)
        if peaks[k][0] > S_RESOLVED:
            break
        k += 1
        assert k < 16, peaks
    assert peaks[k - 1][0] == S_RESOLVED and peaks[k][0] > S_RESOLVED, {j: v[0] for j, v in peaks.items()}
    assert peaks[k][1] & 2, 'a step above S_RESOLVED must set status bit 2'
    s, st, g, x0, e0, got = peaks[k - 1]
    assert st == 0, f'flagged at max s_t = {S_RESOLVED}'
    eo, no = 0, 0
    for i, b in enumerate(blocks):
        ne, nn = b[0].shape[1], b[1].shape[0]
        if i != 1:
            ref = oracle_steps(P, mp, b[0], b[1], b[2])
            check(ref, (got[0][:, eo:eo + ne], got[1][no:no + nn], got[2][eo:eo + ne]), f'quiet window {i} at s = {s}')
        eo, no = eo + ne, no + nn


# ================================================================== F. short loops
@pytest.mark.parametrize('steps,first', [(1, 1), (2, 1), (2, 2)])
@pytest.mark.parametrize('agg', ['sum', 'max'])
def test_short_loops(steps, first, agg):
    _, P, g, x0, e0, _ = main_case(agg)
    mp = model_params(steps, agg)
    mp['num_class_steps'] = steps - first + 1
    ref = oracle_steps(P, mp, g.ei, x0, e0)
    assert ref[0].shape[0] == steps - first + 1
    model = make_model(mp, P)
    for engine in ('tc', 'fp32'):
        got = g.run(model, x0, e0, engine, steps=steps, first=first)
        assert got[3] in (None, 0)
        check(ref, got, f'{steps} steps from {first} {agg} {engine}')
