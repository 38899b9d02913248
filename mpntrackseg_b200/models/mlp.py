"""``MLP`` with the reference's constructor and ``state_dict`` layout, evaluated by the
library's Linear(+ReLU) kernel.  reference: models/mlp.py:4-28"""
import torch
from torch import nn

from .. import ops


class MLP(nn.Module):
    """Linear [-> BatchNorm1d] -> ReLU [-> Dropout] per entry of ``fc_dims``; a layer of width 1 gets none of the
    three (reference: models/mlp.py:12-23).  Parameters and buffers live in ``fc_layers`` at the same Sequential
    slots as the reference, so its checkpoints load unchanged.

    Evaluation mode (what the tracker runs): BatchNorm1d is the affine map of its running statistics and is folded
    into the preceding Linear (W' = s W, b' = s (b - mean) + beta with s = gamma / sqrt(var + eps)); Dropout is the
    identity.  The fused kernels therefore see plain Linear + ReLU layers (``effective_linears``).  Training mode
    with BatchNorm (batch statistics) or Dropout (random masks) is trained as part of ``MOTMPNet`` (training.py's
    CoreTrainer); a standalone call of an ``MLP``, ``EdgeModel`` or ``TimeAwareNodeModel`` in that mode raises."""

    def __init__(self, input_dim, fc_dims, dropout_p=0.4, use_batchnorm=False):
        super().__init__()
        assert isinstance(fc_dims, (list, tuple)), \
            'fc_dims must be either a list or a tuple, but got {}'.format(type(fc_dims))
        self.dropout_p = dropout_p
        self.use_batchnorm = bool(use_batchnorm)
        layers = []
        for dim in fc_dims:
            layers.append(nn.Linear(input_dim, dim))
            if use_batchnorm and dim != 1:
                layers.append(nn.BatchNorm1d(dim))
            if dim != 1:
                layers.append(nn.ReLU(inplace=True))
            if dropout_p != 0 and dim != 1:
                layers.append(nn.Dropout(p=dropout_p))
            input_dim = dim
        self.fc_layers = nn.Sequential(*layers)

    def linears(self):
        return [m for m in self.fc_layers if isinstance(m, nn.Linear)]

    def _check_mode(self):
        if self.training and (self.use_batchnorm or self.dropout_p != 0):
            raise NotImplementedError('BatchNorm / Dropout in training mode run only inside a MOTMPNet training forward '
                                      '(model.train()(data), CoreTrainer); call eval() for a standalone MLP / EdgeModel / '
                                      'TimeAwareNodeModel')

    def effective_linears(self):
        """[(weight, bias)] of the Linear layers as the kernels evaluate them (BatchNorm folded in)."""
        self._check_mode()
        mods = list(self.fc_layers)
        out = []
        for i, m in enumerate(mods):
            if not isinstance(m, nn.Linear):
                continue
            w, b = m.weight, m.bias
            if i + 1 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm1d):
                bn = mods[i + 1]
                s = bn.weight / torch.sqrt(bn.running_var + bn.eps)
                w, b = w * s[:, None], (b - bn.running_mean) * s + bn.bias
            out.append((w, b))
        return out

    def forward(self, input):
        h = input
        for w, b in self.effective_linears():
            h = ops.linear(h, w, b, relu=w.shape[0] != 1)
        return h
