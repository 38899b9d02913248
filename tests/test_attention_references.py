"""CPU checks of the fp64 restatement of the attention backward in test_attention_boundaries: its logit gradient
against fp64 autograd of the oracle's segment softmax, and its zeros and NaN."""
import math

import torch

from oracle import mpn_ref
from test_attention_boundaries import softmax_backward_ref, softmax_parts


def autograd_ref(l, seg, nseg, dw):
    """d <dw, w> / d l by fp64 autograd of mpn_ref.segment_softmax (through its segment max)."""
    lt = l.clone().requires_grad_(True)
    w = mpn_ref.segment_softmax(lt.view(-1, 1), seg).view(-1)
    (w * dw).sum().backward()
    return lt.grad


def segments_case(lead, seed, sizes=(1, 2, 3, 6, 40, 257)):
    """One segment per size; the first slot of each leads the others (uniform in [-1, 1]) by ``lead``."""
    g = torch.Generator().manual_seed(seed)
    seg = torch.cat([torch.full((s,), i) for i, s in enumerate(sizes)])
    l = torch.rand(seg.shape[0], generator=g, dtype=torch.float64) * 2 - 1
    starts = torch.cumsum(torch.tensor((0,) + sizes[:-1]), 0)
    l[starts] = 1.0 + lead
    perm = torch.randperm(seg.shape[0], generator=g)                     # segments interleaved in edge order
    dw = torch.randn(seg.shape[0], generator=g, dtype=torch.float64) * 10
    return l[perm], seg[perm], len(sizes), dw[perm]


def test_restatement_is_the_oracle_gradient_up_to_a_lead_of_20():
    """Per element, within 1e-12 of the scale at which fp64 autograd itself rounds: w_q (|dw_q| + sum_p w_p |dw_p|)."""
    for lead in (0.0, 2.0, 4.0, 8.0, 12.0, 17.0, 20.0):
        for seed in range(3):
            l, seg, nseg, dw = segments_case(lead, seed)
            ref = autograd_ref(l, seg, nseg, dw)
            got = softmax_backward_ref(l, seg, nseg, dw)
            w = softmax_parts(l, seg, nseg)[0]
            scale = w * (dw.abs() + mpn_ref.segment_add(w * dw.abs(), seg, nseg)[seg])
            err = (got - ref).abs() / scale
            assert float(err.max()) <= 1e-12, (lead, seed, float(err.max()))


def test_restatement_keeps_the_dominant_gradient_at_a_lead_of_45():
    """The dominant slot's gradient, about e^-45 of the others' scale, against 60-digit arithmetic of the oracle's
    function (the closed form, minus w_phi S at the argmax: the path through the segment max) on a 3-slot segment."""
    import mpmath
    mpmath.mp.dps = 60
    l = torch.tensor([45.0, 0.25, -0.5], dtype=torch.float64)
    dw = torch.tensor([1.5, -2.0, 0.75], dtype=torch.float64)
    seg = torch.zeros(3, dtype=torch.long)
    got = softmax_backward_ref(l, seg, 1, dw)
    ex = [mpmath.e ** (mpmath.mpf(float(x)) - 45) for x in l]
    den = sum(ex) + mpmath.mpf(1e-12)
    w = [x / den for x in ex]
    S = sum(a * float(b) for a, b in zip(w, dw))
    # exact gradient of exp(l - max) / (sum + eps) with the max path: the closed form, minus w_phi S at the argmax
    exact = [w[q] * (float(dw[q]) - S) for q in range(3)]
    exact[0] -= mpmath.mpf(1e-12) / den * S
    for q in range(3):
        assert abs(float(got[q]) - float(exact[q])) <= 1e-14 * abs(float(exact[q])), (q, float(got[q]), float(exact[q]))


def test_restatement_of_a_one_slot_segment_is_exactly_zero():
    for x, d in ((0.0, 3.0), (-7.5, -1e30), (88.0, 1e-30), (1e4, 2.5)):
        l, dw = torch.tensor([x], dtype=torch.float64), torch.tensor([d], dtype=torch.float64)
        seg = torch.zeros(1, dtype=torch.long)
        assert float(softmax_backward_ref(l, seg, 1, dw)[0]) == 0.0
        assert float(autograd_ref(l, seg, 1, dw)[0]) == 0.0


def test_restatement_has_nan_where_the_oracle_has_nan():
    """-inf logits (weight 0, gradient 0), an all -inf segment, +inf and NaN logits, and a non-finite dw of a weight-0
    slot: NaN at the same places as fp64 autograd of the oracle, equal values elsewhere up to rounding."""
    inf, nan = float('inf'), float('nan')
    cases = [
        ([0.5, -inf, 1.0, -inf], [1.0, 2.0, -3.0, 4.0]),
        ([-inf, -inf, -inf], [1.0, 2.0, 3.0]),
        ([0.5, inf, 1.0], [1.0, 2.0, 3.0]),
        ([0.5, nan, 1.0], [1.0, 2.0, 3.0]),
        ([0.5, -inf, 1.0], [1.0, inf, 3.0]),
        ([0.5, -inf, 1.0], [1.0, nan, 3.0]),
    ]
    for lv, dv in cases:
        # the case segment, then a finite one that must stay finite
        l = torch.tensor(lv + [0.25, 2.0], dtype=torch.float64)
        dw = torch.tensor(dv + [1.0, -1.0], dtype=torch.float64)
        seg = torch.tensor([0] * len(lv) + [1, 1])
        got, ref = softmax_backward_ref(l, seg, 2, dw), autograd_ref(l, seg, 2, dw)
        assert torch.equal(torch.isnan(got), torch.isnan(ref)), (lv, dv, got, ref)
        fin = ~torch.isnan(ref)
        assert bool(torch.isfinite(got[-2:]).all())
        assert float((got[fin] - ref[fin]).abs().max()) <= 1e-14, (lv, dv, got, ref)
        minus = torch.tensor(lv + [0.0, 0.0]) == -inf
        if bool(torch.isfinite(torch.tensor(dv)).all()) and not all(math.isinf(x) and x < 0 for x in lv):
            assert bool((got[minus] == 0).all())
