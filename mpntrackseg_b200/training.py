"""Training step of the core network on the GPU: forward with stored activations, weighted-BCE
loss over the classified steps, hand-written backward, gradient all-reduce and Adam.

reference: pl_module/pl_module.py:88-135 (_compute_loss, _train_val_step), scripts/train.py:65-77
(Adam lr 1e-3 / weight_decay 1e-4, accumulate_grad_batches 8 -- here 8 ranks with one graph each and
one summed all-reduce of a single flat gradient bucket), models/mpn.py:349-381 for the forward.

The arithmetic runs in the deterministic fp32 kernels of csrc/train_ops.cu (mpn_gemm, mpn_colsum,
mpn_gather_cols, mpn_segment_reduce, mpn_segment_grad, mpn_batchnorm_*, mpn_dropout_*, mpn_adam_step) and
csrc/loss.cu; torch only owns the buffers, does index bookkeeping (argsort of the column indices, the dropout
forward counter) and trivial elementwise adds of gradient buffers.  The model options of the reference MLPs are
trained as the reference trains them: node_agg_fn sum / mean / max (max sends the gradient to one argmax, the lowest
caller edge id among ties, like torch_scatter's scatter_max), BatchNorm1d with batch statistics over the rows of each
call (running statistics updated in the module's buffers) and Dropout with Philox masks.
Scope: the tracking loss of the core network (encoders, MPNet, classifier).  The mask branch / mask loss
are not trained here.
"""
import ctypes as C
from collections import OrderedDict

import torch

from . import ops
from ._cabi import check, lib, ptr, stream_ptr


# ------------------------------------------------------------------ thin wrappers
def _ld(t):
    if t.dim() != 2 or t.stride(1) != 1:
        raise ValueError('expected a 2-D tensor with unit column stride')
    return t.stride(0)


def gemm(a, b, ta=False, tb=False, bias=None, relu=False, mask=None, out=None, accumulate=False):
    """out = act(op(a) @ op(b) + bias) (+ out).  mask: a is multiplied by (mask > 0) elementwise."""
    m = a.shape[1] if ta else a.shape[0]
    k = a.shape[0] if ta else a.shape[1]
    n = b.shape[0] if tb else b.shape[1]
    kb = b.shape[1] if tb else b.shape[0]
    if k != kb:
        raise ValueError(f'gemm: inner sizes differ ({k} vs {kb})')
    if out is None:
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    check(lib().mpn_gemm(ptr(a), _ld(a), int(ta), ptr(mask), _ld(mask) if mask is not None else 0, ptr(b), _ld(b), int(tb),
                         ptr(bias), int(relu), int(accumulate), ptr(out), _ld(out), m, n, k, stream_ptr()), 'gemm')
    return out


def colsum(a, mask=None, out=None, accumulate=False):
    m, n = a.shape
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=a.device)
    check(lib().mpn_colsum(ptr(a), _ld(a), ptr(mask), _ld(mask) if mask is not None else 0, m, n, int(accumulate),
                           ptr(out), stream_ptr()), 'colsum')
    return out


def gather_cols(src, idx, out, col_off):
    rows = out.shape[0]
    check(lib().mpn_gather_cols(ptr(src), _ld(src), src.shape[1], ptr(idx), rows, ptr(out), _ld(out), col_off,
                                stream_ptr()), 'gather_cols')


AGG_MODES = {'sum': 0, 'mean': 1, 'max': 2}


def segment_sum(inp, in_off, width, seg_ptr, perm, out, col_off, accumulate=False, mode='sum', argmax=None):
    """out[:, col_off:col_off+width] (+)= the sum / mean / max of each segment; ``argmax`` (int32 [nodes, width], max only)
    receives the input row of each maximum (-1 for an empty segment)."""
    check(lib().mpn_segment_reduce(ptr(inp), _ld(inp), in_off, width, ptr(seg_ptr), ptr(perm), out.shape[0],
                                   int(accumulate), ptr(out), _ld(out), col_off, AGG_MODES[mode], ptr(argmax),
                                   stream_ptr()), 'segment_sum')


def segment_grad(g, row, seg_ptr, argmax, q0, q1, mode, out):
    """out[q] for the slots q in [q0, q1): the gradient of a mean / max ``segment_sum`` (without perm) from ``g``."""
    check(lib().mpn_segment_grad(ptr(g), _ld(g), ptr(row), ptr(seg_ptr), ptr(argmax), q0, q1, out.shape[1],
                                 AGG_MODES[mode], ptr(out), _ld(out), stream_ptr()), 'segment_grad')


class _Dropout:
    """Mask source of one training forward: call k of the forward numbered ``counter`` (a device int64) draws its mask
    from Philox4x32 keyed by ``seed``.  ``masks`` (tests only) collects each call's uint8 mask under its layer key."""

    def __init__(self, seed, counter, keep_masks=False):
        self.seed, self.counter, self.calls = seed, counter, 0
        self.masks = {} if keep_masks else None

    def next(self, key, shape, device):
        self.calls += 1
        if self.masks is None:
            return self.calls - 1, None
        m = self.masks[key] = torch.empty(shape, dtype=torch.uint8, device=device)
        return self.calls - 1, m


class _Linear:
    """y = act(x W^T + b) with its backward (ReLU folded in through the output mask).  With ``bn`` (the BatchNorm1d
    module and its parameter / gradient views) y = ReLU(BN(x W^T + b)) on batch statistics; with ``p`` > 0 the ReLU
    output is followed by inverted dropout.  ``fwd`` returns (y, state); ``bwd`` takes that state back."""

    def __init__(self, w, b, relu, gw, gb, bn=None, p=0.0, key=None):
        self.w, self.b, self.relu, self.gw, self.gb = w, b, relu, gw, gb
        self.bn, self.p, self.key = bn, float(p), key

    def fwd(self, x, drop=None, out=None, tag=''):
        if self.bn is None:
            y = gemm(x, self.w, tb=True, bias=self.b, relu=self.relu, out=out)
            if self.p:
                call, mask = drop.next(self.key + tag, y.shape, y.device)
                check(lib().mpn_dropout_forward(ptr(y), _ld(y), y.shape[0], y.shape[1], self.p, drop.seed,
                                                ptr(drop.counter), call, ptr(mask), stream_ptr()), 'dropout')
            return y, None
        mod, gamma, beta = self.bn['mod'], self.bn['gamma'], self.bn['beta']
        z = gemm(x, self.w, tb=True, bias=self.b)
        if out is None:
            out = torch.empty_like(z)
        stats = torch.empty((4, z.shape[1]), dtype=torch.float32, device=z.device)
        call, mask = drop.next(self.key + tag, z.shape, z.device) if self.p else (0, None)
        check(lib().mpn_batchnorm_forward(ptr(z), _ld(z), z.shape[0], z.shape[1], ptr(gamma), ptr(beta), float(mod.eps),
                                          float(mod.momentum), ptr(mod.running_mean), ptr(mod.running_var),
                                          ptr(mod.num_batches_tracked), ptr(stats), self.p,
                                          drop.seed if self.p else 0, ptr(drop.counter) if self.p else None, call,
                                          ptr(out), _ld(out), ptr(mask), stream_ptr()), 'batchnorm')
        return out, (z, stats)

    def bwd(self, x, y, gy, state=None, need_gx=True, out=None, accumulate=False):
        scale = 1.0 / (1.0 - self.p)
        if self.bn is not None:                      # gradient w.r.t. the Linear output z: no mask left to apply
            z, stats = state
            gz, mask = torch.empty_like(z), None
            check(lib().mpn_batchnorm_backward(ptr(z), _ld(z), ptr(gy), _ld(gy), ptr(y), _ld(y), z.shape[0], z.shape[1],
                                               ptr(self.bn['gamma']), ptr(stats), scale, ptr(self.bn['ggamma']),
                                               ptr(self.bn['gbeta']), ptr(gz), _ld(gz), stream_ptr()), 'batchnorm_backward')
        elif self.p:
            gz, mask = torch.empty_like(y), None
            check(lib().mpn_dropout_backward(ptr(gy), _ld(gy), ptr(y), _ld(y), y.shape[0], y.shape[1], scale, ptr(gz),
                                             _ld(gz), stream_ptr()), 'dropout_backward')
        else:
            gz, mask = gy, (y if self.relu else None)
        gemm(gz, x, ta=True, mask=mask, out=self.gw, accumulate=True)         # gW += (gy*[y>0])^T x
        colsum(gz, mask=mask, out=self.gb, accumulate=True)
        return gemm(gz, self.w, mask=mask, out=out, accumulate=accumulate) if need_gx else None   # gx = (gy*[y>0]) W


CORE_PREFIXES = ('encoder.', 'classifier.', 'MPNet.')


class _CoreLogits(torch.autograd.Function):
    """forward_core / backward_core as one autograd node over the core parameters.  With ``all_steps`` the output holds
    the logits of EVERY message-passing step (the attention branch reads them all, models/mpn.py:377)."""

    @staticmethod
    def forward(ctx, trainer, data, all_steps, *params):
        lg_slot, c = trainer.forward_core(data, all_steps=all_steps)
        ctx.trainer, ctx.c = trainer, c
        trainer.last_ctx = c
        out = torch.empty_like(lg_slot)
        out[:, c['sedge'].long()] = lg_slot                            # slot order -> the caller's edge order
        return out

    @staticmethod
    def backward(ctx, g_out):
        tr, c = ctx.trainer, ctx.c
        tr.grad.zero_()
        tr.backward_core(c, g_out[:, c['sedge'].long()].contiguous())
        return (None, None, None) + tuple(g.clone() for g in tr.g.values())


class AttnAggregate(torch.autograd.Function):
    """``ops.attn_aggregate`` with its hand-written backward (d z and d logits), so that the segmentation loss reaches
    the node feature maps AND, through the attention weights, the tracking network (models/mpn.py:117-137)."""

    @staticmethod
    def forward(ctx, z, logits, layout, perm_c, ptr_c):
        z = z.contiguous()
        flow_in, flow_out = ops.attn_aggregate(z, layout, logits)
        ctx.save_for_backward(z, logits, perm_c, ptr_c)
        ctx.layout = layout
        return flow_in, flow_out

    @staticmethod
    def backward(ctx, g_in, g_out):
        z, logits, perm_c, ptr_c = ctx.saved_tensors
        dz, dl = ops.attn_aggregate_backward(z, ctx.layout, logits, g_in.contiguous(), g_out.contiguous(), perm_c, ptr_c)
        return dz, dl.view_as(logits), None, None, None


class CoreTrainer:
    """Owns a flat parameter / gradient / Adam-state bucket for the core network of a ``MOTMPNet``."""

    def __init__(self, model, lr=1e-3, weight_decay=1e-4, betas=(0.9, 0.999), eps=1e-8, seed=None):
        """``seed`` keys the dropout masks (default ``torch.initial_seed()``); with the device-side forward counter it
        fixes every mask, so two trainers with the same seed draw the same masks forward for forward."""
        self.model = model
        from .models.mpn import _agg_name
        self.agg = _agg_name(model.MPNet.node_model.node_agg_fn)
        if self.agg not in AGG_MODES:
            raise NotImplementedError(f'node_agg_fn {self.agg!r}: the training kernels aggregate by sum / mean / max')
        for name, mod in model.named_modules():
            if name.startswith(CORE_PREFIXES) and isinstance(mod, torch.nn.BatchNorm1d) and mod.momentum is None:
                raise NotImplementedError(f'{name}: BatchNorm1d with momentum=None (cumulative average) is not built '
                                          'into the training kernels')
        self.named = OrderedDict((n, p) for n, p in model.named_parameters() if n.startswith(CORE_PREFIXES))
        dev = next(iter(self.named.values())).device
        total = sum(p.numel() for p in self.named.values())
        self.flat = torch.empty(total, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.g = OrderedDict()
        off = 0
        for n, p in self.named.items():                      # parameters become views of the flat bucket
            k = p.numel()
            self.flat[off:off + k].copy_(p.detach().reshape(-1))
            p.data = self.flat[off:off + k].view_as(p)
            self.g[n] = self.grad[off:off + k].view_as(p)
            off += k
        self.lr, self.weight_decay, self.betas, self.eps = lr, weight_decay, betas, eps
        self.t_dev = torch.zeros(1, dtype=torch.int64, device=dev)        # Adam step number, kept on the device
        self.seed = torch.initial_seed() if seed is None else int(seed)
        self.fwd_dev = torch.zeros(1, dtype=torch.int64, device=dev)      # training forwards so far (dropout counter)
        self._prep_cache, self._graphed = {}, {}
        object.__setattr__(model, '_core_trainer', self)       # one flat bucket per model: MOTMPNet.forward reuses it under autograd

    # ---------------------------------------------------------------- helpers
    def _lin(self, prefix, slot, relu, bn=None, p=0.0):
        w, b = self.named[f'{prefix}.{slot}.weight'], self.named[f'{prefix}.{slot}.bias']
        return _Linear(w.data, b.data, relu, self.g[f'{prefix}.{slot}.weight'], self.g[f'{prefix}.{slot}.bias'].view(-1),
                       bn=bn, p=p, key=f'{prefix}.{slot}')

    def _mlp(self, prefix):
        """The Linear layers of the MLP at ``prefix`` (models/mlp.py), each with the BatchNorm1d that follows it and the
        dropout probability of its ReLU output."""
        mlp = self.model.get_submodule(prefix)
        layers = list(mlp.fc_layers)
        slots = sorted({int(n[len(prefix) + 1:].split('.')[1]) for n in self.named
                        if n.startswith(prefix + '.fc_layers.') and self.named[n].dim() == 2})
        out = []
        for s in slots:
            relu = self.named[f'{prefix}.fc_layers.{s}.weight'].shape[0] != 1
            bn = None
            if s + 1 < len(layers) and isinstance(layers[s + 1], torch.nn.BatchNorm1d):
                k = f'{prefix}.fc_layers.{s + 1}'
                bn = dict(mod=layers[s + 1], gamma=self.named[k + '.weight'].data, beta=self.named[k + '.bias'].data,
                          ggamma=self.g[k + '.weight'], gbeta=self.g[k + '.bias'])
            out.append(self._lin(prefix + '.fc_layers', s, relu, bn=bn, p=mlp.dropout_p if relu else 0.0))
        return out

    def _forward_state(self):
        """Device state a training forward changes besides activations: BatchNorm running statistics and counters and the
        dropout forward counter."""
        bufs = [self.fwd_dev]
        for name, mod in self.model.named_modules():
            if name.startswith(CORE_PREFIXES) and isinstance(mod, torch.nn.BatchNorm1d):
                bufs += [mod.running_mean, mod.running_var, mod.num_batches_tracked]
        return bufs

    # ---------------------------------------------------------------- forward + backward
    def loss_and_grads(self, data, edge_labels, tracking_weight=1.0, zero_grad=True, prep=None):
        """Forward (models/mpn.py:349-381), loss (pl_module.py:88-105) and backward of the core network for
        one graph (or block-diagonal batch).  Gradients are ACCUMULATED into ``self.g`` (zeroed first
        unless zero_grad=False).  Returns the loss as a 1-element device tensor."""
        if zero_grad:
            self.grad.zero_()
        lg_all, ctx = self.forward_core(data, prep)
        # loss (slot order on both sides) and its gradient w.r.t. the logits
        labels = edge_labels.to(lg_all.device, torch.float32).reshape(-1)[ctx['sedge'].long()].contiguous()
        loss, _, g_logits = ops.weighted_bce(lg_all, labels, weight=tracking_weight, want_grad=True)
        self.backward_core(ctx, g_logits)
        return loss

    def prepare(self, data):
        """Index bookkeeping of one graph (slot layout, column-sorted permutation): built once per sample -- the host
        synchronisations of the step live here, the step itself has none."""
        n = int(data.x.shape[0])
        lay = ops.edge_layout(data.edge_index, n)
        e = lay.num_edges
        srow, scol, sedge = lay.slot_row[:e], lay.slot_col[:e], lay.slot_edge[:e]
        order = torch.argsort(scol, stable=True)                         # slots grouped by column
        perm_c = order.to(torch.int32)
        ptr_c = torch.zeros(n + 1, dtype=torch.int32, device=scol.device)
        ptr_c[1:] = torch.cumsum(torch.bincount(scol.long(), minlength=n), 0).to(torch.int32)
        return dict(lay=lay, n=n, e=e, srow=srow, scol=scol, sedge=sedge, perm_c=perm_c, ptr_c=ptr_c)

    def forward_core(self, data, prep=None, all_steps=False, keep_masks=False):
        """Forward with stored activations.  Returns (logits [num_class_steps, E] in SLOT order, ctx); ``ctx['sedge']``
        maps a slot to the caller's edge id.  BatchNorm layers normalise with the statistics of this call's rows and move
        their running statistics; dropout draws the masks of the next forward number.  ``keep_masks`` (tests) stores
        every dropout mask, in slot order, in ``ctx['masks']`` under '<Linear name>@<step>[.out|.in]'."""
        m = self.model
        x = data.x
        pooled = ops.avgpool(x) if x.dim() > 2 else x.contiguous()
        prep = prep or self.prepare(data)
        lay, n, e = prep['lay'], prep['n'], prep['e']
        srow, scol, sedge, perm_c, ptr_c = prep['srow'], prep['scol'], prep['sedge'], prep['perm_c'], prep['ptr_c']
        dev = pooled.device
        steps, first_cls = m.num_enc_steps, max(m.num_enc_steps - m.num_class_steps + 1, 1)
        n_out = lay.num_out

        enc_n, enc_e = self._mlp('encoder.node_model'), self._mlp('encoder.edge_model')
        edge_mlp = self._mlp('MPNet.edge_model.edge_model')
        flow = {'out': self._mlp('MPNet.node_model.flow_out_model'), 'in': self._mlp('MPNet.node_model.flow_in_model')}
        node_lin = self._lin('MPNet.node_model.node_model', 0, True)
        cls = self._mlp('classifier.edge_model')
        for what, mlp_ in (('edge model', edge_mlp), ('flow_out model', flow['out']), ('flow_in model', flow['in']), ('classifier', cls)):
            if len(mlp_) != 2:
                raise NotImplementedError(f'the training kernels expect two-layer MLPs; the {what} has {len(mlp_)} layers')
        dn, de = node_lin.w.shape[0], edge_mlp[-1].w.shape[0]
        fh = flow['out'][0].w.shape[0]
        if steps == 0:
            raise NotImplementedError('training with num_enc_steps == 0')
        drop = _Dropout(self.seed, self.fwd_dev, keep_masks)
        if any(l.p for l in enc_n + enc_e + edge_mlp + flow['out'] + flow['in'] + cls):
            self.fwd_dev.add_(1)

        # ---- encoders (activations kept)
        acts_n, st_n = [pooled], []
        for l in enc_n:
            y, st = l.fwd(acts_n[-1], drop)
            acts_n.append(y); st_n.append(st)
        x0 = acts_n[-1]
        acts_e, st_e = [ops.gather_rows(data.edge_attr.contiguous(), sedge) if e else data.edge_attr.new_empty((0, 6))], []
        for l in enc_e:
            y, st = l.fwd(acts_e[-1], drop)
            acts_e.append(y); st_e.append(st)
        e0 = acts_e[-1]

        # ---- message-passing steps
        xs, es, saved, logits, logit_steps = x0, e0, [], [], []
        ranges = (('out', 0, n_out, dn), ('in', n_out, e, 0))            # (name, slot range, column offset in [flow_in|flow_out])
        for step in range(1, steps + 1):
            a = torch.empty((e, 4 * dn + 2 * de), dtype=torch.float32, device=dev)
            gather_cols(x0, srow, a, 0); gather_cols(xs, srow, a, dn)
            gather_cols(x0, scol, a, 2 * dn); gather_cols(xs, scol, a, 3 * dn)
            gather_cols(e0, None, a, 4 * dn); gather_cols(es, None, a, 4 * dn + de)
            tag = f'@{step}'
            h, st_h = edge_mlp[0].fwd(a, drop, tag=tag)
            e2, st_e2 = edge_mlp[1].fwd(h, drop, tag=tag)
            c1, st_c1 = cls[0].fwd(e2, drop, tag=tag)
            lg, _ = cls[1].fwd(c1)
            b = torch.empty((e, 2 * dn + de), dtype=torch.float32, device=dev)
            gather_cols(a[:, 2 * dn:4 * dn], None, b, 0); gather_cols(e2, None, b, 2 * dn)
            g_ = torch.empty((e, fh), dtype=torch.float32, device=dev)
            msg = torch.empty((e, dn), dtype=torch.float32, device=dev)
            f = torch.empty((n, 2 * dn), dtype=torch.float32, device=dev)
            argmax = torch.empty((2, n, dn), dtype=torch.int32, device=dev) if self.agg == 'max' else None
            st_flow = {}
            for name, s0, s1, coff in ranges:
                # BatchNorm takes the statistics of this direction's rows and counts the call even when it has none
                if s1 > s0 or flow[name][0].bn is not None:
                    _, st0 = flow[name][0].fwd(b[s0:s1], drop, out=g_[s0:s1], tag=f'{tag}.{name}')
                    _, st1 = flow[name][1].fwd(g_[s0:s1], drop, out=msg[s0:s1], tag=f'{tag}.{name}')
                    st_flow[name] = (st0, st1)
                segment_sum(msg, 0, dn, lay.out_ptr if name == 'out' else lay.in_ptr, None, f, coff, mode=self.agg,
                            argmax=None if argmax is None else argmax[coff // dn])
            xs_new, _ = node_lin.fwd(f)
            saved.append(dict(a=a, h=h, e2=e2, c1=c1, b=b, g_=g_, msg=msg, f=f, xs_new=xs_new, argmax=argmax,
                              st=(st_h, st_e2, st_c1), st_flow=st_flow))
            if all_steps or step >= first_cls:
                logits.append(lg.view(-1))
                logit_steps.append(step)
            xs, es = xs_new, e2

        ctx = dict(lay=lay, sedge=sedge, srow=srow, scol=scol, perm_c=perm_c, ptr_c=ptr_c, n=n, e=e, n_out=n_out,
                   steps=steps, first_cls=first_cls, saved=saved, acts_n=acts_n, acts_e=acts_e, st_n=st_n, st_e=st_e,
                   dn=dn, de=de, logit_steps=logit_steps, masks=drop.masks)
        return torch.stack(logits), ctx

    def backward_core(self, ctx, g_logits):
        """Hand-written backward from d loss / d logits ([num_class_steps, E], slot order); parameter gradients are
        ACCUMULATED into ``self.g``."""
        lay, srow, perm_c, ptr_c = ctx['lay'], ctx['srow'], ctx['perm_c'], ctx['ptr_c']
        n, e, n_out, steps, first_cls, saved = ctx['n'], ctx['e'], ctx['n_out'], ctx['steps'], ctx['first_cls'], ctx['saved']
        acts_n, acts_e, dn, de = ctx['acts_n'], ctx['acts_e'], ctx['dn'], ctx['de']
        dev = g_logits.device
        enc_n, enc_e = self._mlp('encoder.node_model'), self._mlp('encoder.edge_model')
        edge_mlp = self._mlp('MPNet.edge_model.edge_model')
        flow = {'out': self._mlp('MPNet.node_model.flow_out_model'), 'in': self._mlp('MPNet.node_model.flow_in_model')}
        node_lin = self._lin('MPNet.node_model.node_model', 0, True)
        cls = self._mlp('classifier.edge_model')
        ranges = (('out', 0, n_out, dn), ('in', n_out, e, 0))
        g_logits = g_logits.contiguous()
        row_of = {step: i for i, step in enumerate(ctx['logit_steps'])}   # row of g_logits that belongs to a step

        # ---- backward through the steps
        gxs = torch.zeros((n, dn), dtype=torch.float32, device=dev)
        ge2_next = torch.zeros((e, de), dtype=torch.float32, device=dev)
        gx0 = torch.zeros((n, dn), dtype=torch.float32, device=dev)
        ge0 = torch.zeros((e, de), dtype=torch.float32, device=dev)
        for step in range(steps, 0, -1):
            sv = saved[step - 1]
            a, h, e2, c1, b, g_, msg, f, xs_new = (sv[k] for k in ('a', 'h', 'e2', 'c1', 'b', 'g_', 'msg', 'f', 'xs_new'))
            st_h, st_e2, st_c1 = sv['st']
            gf = node_lin.bwd(f, xs_new, gxs)                                           # [n, 2dn]
            gmsg = torch.empty((e, dn), dtype=torch.float32, device=dev)
            gb = torch.empty((e, 2 * dn + de), dtype=torch.float32, device=dev)
            for name, s0, s1, coff in ranges:
                if s1 <= s0:
                    continue
                if self.agg == 'sum':                                                   # d flow[row] -> each message
                    gather_cols(gf[:, coff:coff + dn], srow[s0:s1], gmsg[s0:s1], 0)
                else:
                    segment_grad(gf[:, coff:coff + dn], srow, lay.out_ptr if name == 'out' else lay.in_ptr,
                                 None if sv['argmax'] is None else sv['argmax'][coff // dn], s0, s1, self.agg, gmsg)
                l0, l1 = flow[name]
                st0, st1 = sv['st_flow'][name]
                gg = l1.bwd(g_[s0:s1], msg[s0:s1], gmsg[s0:s1], st1)
                l0.bwd(b[s0:s1], g_[s0:s1], gg, st0, out=gb[s0:s1])
            ge2 = ge2_next + gb[:, 2 * dn:]                                             # e' feeds the flow MLPs and step+1
            if step in row_of:
                gl = g_logits[row_of[step]].view(-1, 1)
                gc1 = cls[1].bwd(c1, None, gl)
                cls[0].bwd(e2, c1, gc1, st_c1, out=ge2, accumulate=True)
            gh = edge_mlp[1].bwd(h, e2, ge2, st_e2)
            ga = edge_mlp[0].bwd(a, h, gh, st_h)                                        # [e, 4dn+2de]
            gxs_new = torch.empty((n, dn), dtype=torch.float32, device=dev)
            for part, dst in ((0, gx0), (dn, gxs_new)):                                 # x_init part / x_latent part
                acc = dst is gx0
                segment_sum(ga, part, dn, lay.out_ptr, None, dst, 0, accumulate=acc)                 # x[row], flow_out group
                segment_sum(ga, part, dn, lay.in_ptr, None, dst, 0, accumulate=True)                 # x[row], flow_in group
                segment_sum(ga, 2 * dn + part, dn, ptr_c, perm_c, dst, 0, accumulate=True)           # x[col] of the edge MLP
                segment_sum(gb, part, dn, ptr_c, perm_c, dst, 0, accumulate=True)                    # x[col] of the flow MLPs
            ge0 += ga[:, 4 * dn:4 * dn + de]
            ge2_next = ga[:, 4 * dn + de:].contiguous()
            gxs = gxs_new
        gx0 += gxs                                                       # before step 1 the latent states are the
        ge0 += ge2_next                                                  # initial encodings (models/mpn.py:358-359)

        # ---- encoders
        g_act = gx0
        for i in range(len(enc_n) - 1, -1, -1):
            g_act = enc_n[i].bwd(acts_n[i], acts_n[i + 1], g_act, ctx['st_n'][i], need_gx=i > 0)
        g_act = ge0
        for i in range(len(enc_e) - 1, -1, -1):
            g_act = enc_e[i].bwd(acts_e[i], acts_e[i + 1], g_act, ctx['st_e'][i], need_gx=i > 0)

    # ---------------------------------------------------------------- autograd bridge
    def autograd_logits(self, data, all_steps=False):
        """Logits [num_class_steps, E] (or [num_enc_steps, E] with ``all_steps``) in the CALLER'S edge order, attached to
        the autograd graph of the core parameters: ``loss.backward()`` (pl_module.py:126-135) runs ``backward_core`` and
        fills ``p.grad``."""
        return _CoreLogits.apply(self, data, all_steps, *self.named.values())

    # ---------------------------------------------------------------- optimizer
    def all_reduce_grads(self, group=None):
        """One summed all-reduce of the single flat gradient bucket (1.19 MB); NCCL on GPUs."""
        from .sharding import all_reduce_sum_
        return all_reduce_sum_(self.grad, group)

    @property
    def t(self):
        return int(self.t_dev.item())

    def adam_step(self, grad_scale=1.0):
        check(lib().mpn_adam_step_dev(ptr(self.flat), ptr(self.grad), ptr(self.exp_avg), ptr(self.exp_avg_sq), self.flat.numel(),
                                      float(self.lr), float(self.betas[0]), float(self.betas[1]), float(self.eps),
                                      float(self.weight_decay), ptr(self.t_dev), float(grad_scale), stream_ptr()), 'adam_step')

    def train_step(self, data, edge_labels, tracking_weight=1.0, group=None, prep=None):
        """loss.backward() + gradient all-reduce (mean over ranks) + Adam, as Lightning drives it
        (pl_module.py:137-141, scripts/train.py:76 with the 8 accumulated batches spread over 8 ranks)."""
        loss = self.loss_and_grads(data, edge_labels, tracking_weight, prep=prep)
        world = self.all_reduce_grads(group)
        self.adam_step(grad_scale=1.0 / world)
        return loss

    def graphed_step(self, data, edge_labels, tracking_weight=1.0, group=None):
        """The same training step with its compute part (forward with activations, loss, backward: ~900 small kernels)
        captured ONCE as a CUDA graph for this sample and replayed on every call with the same ``data`` object; the NCCL
        all-reduce of the gradient bucket and the Adam step (two kernels, step counter on the device) follow on the same
        stream outside the graph.  Parameters and gradients live in fixed device buffers, so replays continue the
        optimisation exactly like ``train_step``; ``data.x`` / ``edge_attr`` / ``edge_labels`` are read from their
        current storage at replay time (update them in place to feed new values on the same graph structure)."""
        key = id(data)
        gs = self._graphed.get(key)
        if gs is None:
            gs = self._graphed[key] = _GraphedStep(self, data, edge_labels, tracking_weight)
        loss = gs.replay()
        world = self.all_reduce_grads(group)
        self.adam_step(grad_scale=1.0 / world)
        return loss


class _GraphedStep(object):
    """CUDA graph of ``CoreTrainer.loss_and_grads`` for one sample (no collective inside the capture)."""

    def __init__(self, trainer, data, edge_labels, tracking_weight):
        tr = self.trainer = trainer
        self.data, self.labels = data, edge_labels.to(data.edge_index.device, torch.float32).contiguous()
        self.prep = tr.prepare(data)
        state = [t.clone() for t in tr._forward_state()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                                   # warm-up off the capture (allocator, lazy inits)
            for _ in range(2):
                tr.loss_and_grads(data, self.labels, tracking_weight, prep=self.prep)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for t, s in zip(tr._forward_state(), state):                    # the warm-up forwards do not count as steps
            t.copy_(s)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = tr.loss_and_grads(data, self.labels, tracking_weight, prep=self.prep)

    def replay(self):
        self.graph.replay()
        return self.loss
