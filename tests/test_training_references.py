"""CPU checks of the fp64 references of test_training_boundaries: the weighted-BCE reference against torch's
BCE-with-logits in fp64 and its confident terms."""
import math

import numpy as np
import torch

from test_training_boundaries import bce_ref


def test_bce_reference_is_torch_bce_with_logits_in_fp64():
    """The reference equals F.binary_cross_entropy_with_logits(pos_weight=...) and its autograd in fp64 where that is
    accurate (|x| <= 16), for every positive fraction and a soft label."""
    import torch.nn.functional as F
    from oracle import mpn_ref
    g = torch.Generator().manual_seed(3)
    for labels in (torch.zeros(300), (torch.arange(300) == 7).float(), (torch.arange(300) % 2).float(),
                   torch.ones(300), torch.tensor([0.0, 0.3, 1.0]).repeat(100)):
        x = ((torch.rand(3, 300, generator=g) * 32 - 16)).double().requires_grad_(True)
        pos = labels.sum()
        pw = ((labels.shape[0] - pos) / pos) if pos else torch.zeros(1)
        loss = sum(0.7 * F.binary_cross_entropy_with_logits(x[s], labels.double(), pos_weight=pw.double())
                   for s in range(3))
        loss.backward()
        ref_loss, ref_g, _, rpw = bce_ref(x.detach(), labels, 0.7)
        assert rpw == float(np.float32(float(pw)))
        assert abs(float(loss) - ref_loss) <= 1e-12 * ref_loss
        assert float((x.grad - ref_g).abs().max()) <= 1e-12 * float(ref_g.abs().max())
        pos64 = float(labels.double().sum())           # the oracle on fp64 labels: pos_weight not rounded to fp32
        ref64 = bce_ref(x.detach(), labels, 0.7, pw=(300 - pos64) / pos64 if pos64 else 0.0)[0]
        assert abs(float(mpn_ref.weighted_bce_loss([x[s].detach() for s in range(3)], labels.double(), 0.7)) - ref64) \
            <= 1e-12 * ref64


def test_bce_reference_keeps_confident_terms():
    """Where fp32 1 - s(-x) rounds to 0 (x < -17) the reference keeps s(x) ~ e^x, and a zero-weight side of an
    infinite logit adds 0."""
    x = torch.tensor([[-20.0, -89.0, float('-inf'), float('inf')]])
    loss, grad, _, _ = bce_ref(x, torch.zeros(4), 1.0)
    assert abs(float(grad[0, 0]) - 1 / (1 + math.exp(20)) / 4) <= 1e-15 * math.exp(-20)
    assert float(grad[0, 1]) > 0 and float(grad[0, 2]) == 0 and float(grad[0, 3]) == 0.25
    assert math.isinf(loss)
    loss, _, _, _ = bce_ref(x[:, :3], torch.zeros(3), 1.0)
    assert 0 < loss < 1e-8
