"""Drop-in ``MOTMPNet`` / ``MetaLayer`` with the reference's constructors, parameter names
and ``forward`` signatures, evaluated by the sm_100a kernels of libmpntrack_b200.so.

reference: src/mot_neural_solver/models/mpn.py (MetaLayer :11-57, EdgeModel :59-69,
TimeAwareNodeModel :71-99, MLPGraphIndependent :139-178, MOTMPNet :209-394).

The modules own ``nn.Parameter``s exactly where the reference does (so ``state_dict`` keys
match and its checkpoints load), and hand raw device pointers to the C ABI.  There is no
CPU path: CPU tensors raise.
"""
import torch
from torch import nn

from .. import ops
from ..config import core_dims
from .cnn import CNN, MaskRCNNPredictor
from .mlp import MLP


def _core_weight_tensors(edge_mlp, flow_in, flow_out, node_lin, cls_mlp):
    (e0w, e0b), (e1w, e1b) = edge_mlp.effective_linears()
    (i0w, i0b), (i1w, i1b) = flow_in.effective_linears()
    (o0w, o0b), (o1w, o1b) = flow_out.effective_linears()
    (c0w, c0b), (c1w, c1b) = cls_mlp.effective_linears()
    return {'edge_w0': e0w, 'edge_b0': e0b, 'edge_w1': e1w, 'edge_b1': e1b,
            'fin_w0': i0w, 'fin_b0': i0b, 'fin_w1': i1w, 'fin_b1': i1b,
            'fout_w0': o0w, 'fout_b0': o0b, 'fout_w1': o1w, 'fout_b1': o1b,
            'node_w': node_lin.weight, 'node_b': node_lin.bias,
            'cls_w0': c0w, 'cls_b0': c0b, 'cls_w1': c1w, 'cls_b1': c1b}


def _agg_name(node_agg_fn):
    """'sum' | 'mean' | 'max' from the model's ``node_agg_fn`` (the reference stores a lambda around the torch_scatter
    function; here the config string is kept and the kernels switch on it).  reference: models/mpn.py:263-273"""
    if node_agg_fn is None:
        return 'sum'
    if isinstance(node_agg_fn, str):
        return node_agg_fn.lower()
    raise NotImplementedError('node_agg_fn must be one of the strings the reference accepts (sum / mean / max)')


def _layout(edge_index, x, edge_attr):
    """Slot layout of ``edge_index`` over the rows of ``x``; its build rejects self-loops and node ids outside [0, N)
    (ValueError) before anything gathers by them."""
    layout = ops.edge_layout(edge_index, x.shape[0])
    if edge_attr.shape[0] != layout.num_edges:
        raise ValueError(f'edge_attr has {edge_attr.shape[0]} rows for {layout.num_edges} edges')
    return layout


class EdgeModel(nn.Module):
    """Edge update e' = MLP(cat[x[row], x[col], e]).  reference: models/mpn.py:59-69
    ``forward(node_feats [N,64], edge_index [2,E], edge_attr [E,32]) -> [E,16]`` in the caller's edge order."""

    def __init__(self, edge_model):
        super().__init__()
        self.edge_model = edge_model

    def forward(self, node_feats, edge_index, edge_attr):
        lins = self.edge_model.linears()
        de = lins[-1].out_features
        dn = (lins[0].in_features - 2 * de) // 4
        if node_feats.shape[1] != 2 * dn or edge_attr.shape[1] != 2 * de:
            raise NotImplementedError('the edge model is built for reattach_initial_nodes/edges = True '
                                      f'(x [N,{2 * dn}], edge_attr [E,{2 * de}])')
        layout = _layout(edge_index, node_feats, edge_attr)
        e, slot_edge = layout.num_edges, layout.slot_edge[:layout.num_edges]
        h = torch.cat((ops.gather_rows(node_feats, layout.slot_row[:e]), ops.gather_rows(node_feats, layout.slot_col[:e]),
                       ops.gather_rows(edge_attr, slot_edge)), dim=1)
        e_new = self.edge_model(h)
        out = torch.empty_like(e_new)
        out[slot_edge.long()] = e_new                            # back to the caller's edge order
        return out


class TimeAwareNodeModel(nn.Module):
    """Time-aware node update.  reference: models/mpn.py:71-99
    ``forward(x [N,64], edge_index [2,E], edge_attr [E,16]) -> [N,32]`` where ``edge_attr`` holds the already
    updated edge features (models/mpn.py:52).  ``node_agg_fn`` is the reference's name for the aggregation
    ('sum' | 'mean' | 'max' or its lambda).  The messages of the flow_out group (row < col) and of the flow_in group are
    computed in slot order, where each node's edges of one group are contiguous, and reduced per node in that order."""

    def __init__(self, flow_in_model, flow_out_model, node_model, node_agg_fn):
        super().__init__()
        self.flow_in_model = flow_in_model
        self.flow_out_model = flow_out_model
        self.node_model = node_model
        self.node_agg_fn = node_agg_fn

    def forward(self, x, edge_index, edge_attr):
        lins = self.flow_in_model.linears()
        lin0, dn = lins[0], lins[-1].out_features
        if lin0.in_features != 2 * dn + edge_attr.shape[1]:
            raise NotImplementedError(f'TimeAwareNodeModel expects x [N,{2 * dn}] and '
                                      f'edge_attr [E,{lin0.in_features - 2 * dn}]')
        if x.shape[1] != 2 * dn:
            raise NotImplementedError(f'TimeAwareNodeModel expects x [N,{2 * dn}] (reattach_initial_nodes = True)')
        agg = _agg_name(self.node_agg_fn)
        if agg not in ops.NODE_AGG:
            raise ValueError(f"node_agg_fn can only be 'max', 'mean' or 'sum', got {agg!r}")
        layout = _layout(edge_index, x, edge_attr)
        e, n_out = layout.num_edges, layout.num_out
        h = torch.cat((ops.gather_rows(x, layout.slot_col[:e]), ops.gather_rows(edge_attr, layout.slot_edge[:e])), dim=1)
        msg = torch.cat((self.flow_out_model(h[:n_out]), self.flow_in_model(h[n_out:])))
        flow = torch.empty((x.shape[0], 2 * dn), dtype=torch.float32, device=x.device)
        ops.segment_sum(msg, 0, dn, layout.in_ptr, None, flow, 0, mode=agg)      # cat(flow_in, flow_out), models/mpn.py:97
        ops.segment_sum(msg, 0, dn, layout.out_ptr, None, flow, dn, mode=agg)
        lin = self.node_model[0]
        return ops.linear(flow, lin.weight, lin.bias, relu=True)


class MetaLayer(nn.Module):
    """One message-passing step ``forward(x, edge_index, edge_attr) -> (x', edge_attr')``: the edge model, then the
    node model on the updated edge features, x = [x_init | x_latent], edge_attr = [e_init | e_latent] in the caller's
    edge order.  reference: models/mpn.py:11-57"""

    def __init__(self, edge_model=None, node_model=None):
        super().__init__()
        self.edge_model = edge_model
        self.node_model = node_model

    def _weights(self, classifier):
        em, nm = self.edge_model, self.node_model
        if em is None or nm is None:
            raise NotImplementedError('the fused step needs both an EdgeModel and a TimeAwareNodeModel')
        named = _core_weight_tensors(em.edge_model, nm.flow_in_model, nm.flow_out_model,
                                     nm.node_model[0], classifier)
        return ops.core_weights(named, node_agg=_agg_name(nm.node_agg_fn))

    def forward(self, x, edge_index, edge_attr):
        if self.edge_model is not None:
            edge_attr = self.edge_model(x, edge_index, edge_attr)
        if self.node_model is not None:
            x = self.node_model(x, edge_index, edge_attr)
        return x, edge_attr

    def __repr__(self):
        return '{}(edge_model={}, node_model={})'.format(self.__class__.__name__, self.edge_model, self.node_model)


class TimeAwareAttentionModel(nn.Module):
    """Attentive aggregation of the node feature maps followed by the 3x3 conv stack.
    ``forward(x, edge_index, edge_attr, cls_net)`` keeps the reference's signature; the fused path calls
    ``aggregate`` with a precomputed slot layout and the step's logits.  reference: models/mpn.py:102-137"""

    def __init__(self, node_model, flow_in_attention_model=None, flow_out_attention_model=None):
        super().__init__()
        self.node_model = node_model        # the two attention MLPs are built and dropped by the reference (:106-109)

    def aggregate(self, x, layout, logits, train_ctx=None):
        if train_ctx is not None:
            from ..training import AttnAggregate
            flow_in, flow_out = AttnAggregate.apply(x, logits, layout, train_ctx['perm_c'], train_ctx['ptr_c'])
        else:
            flow_in, flow_out = ops.attn_aggregate(x, layout, logits)
        return self.node_model(torch.cat((x, flow_in, flow_out), dim=1))

    def forward(self, x, edge_index, edge_attr, cls_net):
        dec_edge_feats, _ = cls_net(edge_attr)
        layout = ops.edge_layout(edge_index, x.shape[0])
        return self.aggregate(x.contiguous(), layout, dec_edge_feats.reshape(-1)), dec_edge_feats


class MaskModel(nn.Module):
    """Mask head on cat[feature_encoder(x_ext), node embedding].  reference: models/mpn.py:180-206"""

    def __init__(self, mask_model_params):
        super().__init__()
        self.feature_encoder = CNN(**mask_model_params['feature_encoder_feats_dict'])
        self.layer_norm = nn.LayerNorm([64, 14, 14])
        self.mask_head = CNN(**mask_model_params['mask_head_feats_dict'])
        self.mask_predictor = MaskRCNNPredictor(**mask_model_params['mask_predictor_feats_dict'])

    def forward(self, feature_embeds, node_embeds):
        h = torch.cat((self.feature_encoder(feature_embeds), node_embeds), dim=1)
        return self.mask_predictor(self.mask_head(self.layer_norm(h)))


class MLPGraphIndependent(nn.Module):
    """Independent node / edge MLPs (encoder, classifier).  reference: models/mpn.py:139-178"""

    def __init__(self, edge_in_dim=None, node_in_dim=None, edge_out_dim=None, node_out_dim=None,
                 node_dims=None, edge_dims=None, dropout_p=None, use_batchnorm=None):
        super().__init__()
        if node_in_dim is not None:
            self.node_model = MLP(input_dim=node_in_dim, fc_dims=list(node_dims) + [node_out_dim],
                                  dropout_p=dropout_p, use_batchnorm=use_batchnorm)
        else:
            self.node_model = None
        if edge_in_dim is not None:
            self.edge_model = MLP(input_dim=edge_in_dim, fc_dims=list(edge_dims) + [edge_out_dim],
                                  dropout_p=dropout_p, use_batchnorm=use_batchnorm)
        else:
            self.edge_model = None

    def forward(self, edge_feats=None, nodes_feats=None):
        out_node = self.node_model(nodes_feats) if self.node_model is not None else nodes_feats
        out_edge = self.edge_model(edge_feats) if self.edge_model is not None else edge_feats
        return out_edge, out_node


class BatchOutput(object):
    """Result of ``MOTMPNet.forward_batch``."""

    def __init__(self, logits, batch, spans):
        self.logits, self.batch, self.spans = logits, batch, spans

    def __len__(self):
        return self.batch.num_graphs if self.batch is not None else len(self.spans)

    def graph_logits(self, g):
        """[num_class_steps, E_g] logits of window ``g`` in the reference's per-window edge order."""
        if self.batch is None:
            a, b = self.spans[g]
            return self.logits[:, a:b]
        pp = self.batch.pair_ptr
        a, b, p = pp[g], pp[g + 1], pp[-1]
        return torch.cat((self.logits[:, a:b], self.logits[:, p + a:p + b]), dim=1)

    def graph_output(self, g):
        lg = self.graph_logits(g)
        return {'classified_edges': [lg[i].reshape(-1, 1) for i in range(lg.shape[0])], 'mask_predictions': []}

    def __getitem__(self, g):
        return self.graph_output(g)


class MOTMPNet(nn.Module):
    """Encoder -> ``num_enc_steps`` shared-weight message-passing steps -> edge classifier.

    ``forward(data)`` takes any object with ``x [N,2048,8,4]`` (or pooled ``[N,2048]`` /
    ``[N,2048,1,1]``), ``edge_index [2,E] int64``, ``edge_attr [E,6]`` (and ``x_ext`` for the
    mask branch) and returns ``{'classified_edges': [Tensor[E,1]]*num_class_steps,
    'mask_predictions': [...]}`` like the reference.  reference: models/mpn.py:209-394
    """

    def __init__(self, model_params, bb_encoder=None):
        super().__init__()
        self.node_cnn = bb_encoder
        self.model_params = model_params
        enc = model_params['encoder_feats_dict']
        self.encoder = MLPGraphIndependent(**enc)
        self.classifier = MLPGraphIndependent(**model_params['classifier_feats_dict'])
        # mask branch (cuDNN convolutions + the attentive-aggregation kernel); same module names and
        # registration order as the reference so that its checkpoints load with strict=True
        self.has_mask_branch = 'node_ext_encoder_feats_dict' in model_params
        if self.has_mask_branch:
            self.node_ext_encoder = CNN(**model_params['node_ext_encoder_feats_dict'])
            self.mask_predictor = MaskModel(model_params['mask_model_feats_dict'])
        self.MPNet = self._build_core_MPNet(model_params=model_params, encoder_feats_dict=enc)
        if self.has_mask_branch:
            self.MPAttentionNet = self._build_attention_MPNet(model_params=model_params)
        self.num_enc_steps = model_params['num_enc_steps']
        self.num_class_steps = model_params['num_class_steps']
        # 'auto' | 'tc' | 'fp32' (None = $MPN_ENGINE or 'auto'), see ops.mp_forward
        self.engine = None

    def _build_core_MPNet(self, model_params, encoder_feats_dict):
        """reference: models/mpn.py:250-317"""
        agg = model_params['node_agg_fn']
        assert agg.lower() in ('mean', 'max', 'sum'), "node_agg_fn can only be 'max', 'mean' or 'sum'."
        self.reattach_initial_nodes = model_params['reattach_initial_nodes']
        self.reattach_initial_edges = model_params['reattach_initial_edges']
        if not (self.reattach_initial_nodes and self.reattach_initial_edges):
            raise NotImplementedError('the fused kernel is built for reattach_initial_nodes/edges = True')
        self.edge_factor, self.node_factor = 2, 2
        d = core_dims(model_params)
        em, nm = model_params['edge_model_feats_dict'], model_params['node_model_feats_dict']
        edge_model = MLP(input_dim=d['edge_mlp_in'], fc_dims=em['dims'], dropout_p=em['dropout_p'],
                         use_batchnorm=em['use_batchnorm'])
        flow_in_model = MLP(input_dim=d['flow_mlp_in'], fc_dims=nm['dims'], dropout_p=nm['dropout_p'],
                            use_batchnorm=nm['use_batchnorm'])
        flow_out_model = MLP(input_dim=d['flow_mlp_in'], fc_dims=nm['dims'], dropout_p=nm['dropout_p'],
                             use_batchnorm=nm['use_batchnorm'])
        node_model = nn.Sequential(nn.Linear(2 * d['dn'], d['dn']), nn.ReLU(inplace=True))
        return MetaLayer(edge_model=EdgeModel(edge_model=edge_model),
                         node_model=TimeAwareNodeModel(flow_in_model=flow_in_model, flow_out_model=flow_out_model,
                                                       node_model=node_model, node_agg_fn=agg))

    def _build_attention_MPNet(self, model_params):
        """reference: models/mpn.py:319-331 (the two attention MLPs it constructs are never used)"""
        nx = model_params['node_ext_model_feats_dict']
        in_dim = 3 * model_params['node_ext_encoder_feats_dict']['dims'][-1] * self.node_factor
        return TimeAwareAttentionModel(node_model=CNN(input_dim=in_dim, **nx))

    # ------------------------------------------------------------------ forward
    def core_weights(self):
        return self.MPNet._weights(self.classifier.edge_model)

    def encode_nodes(self, x, status=None):
        """Global average pool + node MLP.  reference: models/mpn.py:351-355
        status: optional int32[1] device tensor receiving the fp16-overflow flag of the tensor-core
        encoder instead of a host sync + fallback here."""
        return self.encode_nodes_list([x], status=status)

    def encode_pooled(self, pooled, engine=None, status=None):
        """Node MLP on already pooled features [N, C] (one launch for any number of windows)."""
        lins = self.encoder.node_model.effective_linears()
        return ops.node_encoder(pooled, [w for w, _ in lins], [b for _, b in lins],
                                engine=engine or self.engine, status=status)

    def encode_nodes_list(self, xs, engine=None, status=None):
        """Node encoder over several windows' features in ONE kernel launch: every window is pooled into
        its slice of a [N_total, C] buffer, then the whole buffer goes through the MLP."""
        engine = engine or self.engine
        if len(xs) == 1 and xs[0].dim() == 2:
            pooled = xs[0]
        else:
            n_tot = sum(int(x.shape[0]) for x in xs)
            pooled = torch.empty((n_tot, xs[0].shape[1]), dtype=torch.float32, device=xs[0].device)
            off = 0
            for x in xs:
                ops.avgpool(x if x.dim() > 2 else x[:, :, None, None], out=pooled[off:off + x.shape[0]])
                off += x.shape[0]
        lins = self.encoder.node_model.effective_linears()
        return ops.node_encoder(pooled, [w for w, _ in lins], [b for _, b in lins], engine=engine, status=status)

    def encode_edges(self, edge_attr, layout):
        lins = self.encoder.edge_model.effective_linears()
        return ops.edge_encoder(edge_attr, layout, [w for w, _ in lins], [b for _, b in lins])

    def forward_batch(self, graphs, encoded=False):
        """Extension (not in the reference): evaluate several independent window graphs as one
        block-diagonal batch (what torch_geometric's DataLoader does with batch_size > 1): nodes are
        encoded per window, and one message-passing run covers all of them.  ``graphs`` is a
        ``data.mot_graph.GraphBatch`` (built in one pass by ``build_window_graphs``) or a list of
        ``Graph`` objects.  Returns a ``BatchOutput``: ``.logits`` [num_class_steps, E_total] in the
        batch's edge order and ``.graph_output(g)`` = the reference-style dict of window ``g``."""
        from ..data.mot_graph import GraphBatch
        if isinstance(graphs, GraphBatch):
            batch = graphs
            xs = list(batch.xs) if isinstance(batch.xs, (list, tuple)) else [batch.xs]
            edge_index, edge_attr, n = batch.edge_index, batch.edge_attr, batch.num_nodes
            spans = None
            pooled = None if encoded else batch.pooled_xs()
        else:
            xs, eis, eas, spans, off, eo = [], [], [], [], 0, 0
            for g in graphs:
                xs.append(g.x)
                eis.append(g.edge_index + off)
                eas.append(g.edge_attr)
                spans.append((eo, eo + g.edge_index.shape[1]))
                off += g.x.shape[0]
                eo += g.edge_index.shape[1]
            edge_index, edge_attr, n, batch, pooled = torch.cat(eis, dim=1), torch.cat(eas), off, None, None
        layout = ops.edge_layout(edge_index, n)
        first_class_step = self.num_enc_steps - self.num_class_steps + 1
        logits = self._core(xs, edge_attr, layout, first_class_step, encoded=encoded, pooled=pooled)[0]
        return BatchOutput(logits, batch, spans)

    def forward(self, data, return_state=False):
        x, edge_index, edge_attr = data.x, data.edge_index, data.edge_attr
        x_ext = getattr(data, 'x_ext', None) if self.has_mask_branch else None
        if self.training and ((torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()))
                              or self._core_has_train_only_layers()):
            # training (pl_module.py:122-135): model.train() + autograd on.  The core network runs through the
            # deterministic fp32 training kernels with a hand-written backward; loss.backward() fills p.grad of the
            # encoder / MPNet / classifier weights.  A training-mode call under no_grad takes this path too when the
            # core has BatchNorm or Dropout: batch statistics, running-statistic updates and fresh dropout masks, as
            # torch runs such a module, without a backward.  Evaluation-mode calls (model.eval(), with or without
            # no_grad) always take the inference kernels below.
            if return_state:
                raise NotImplementedError('return_state is an inference-only option')
            tr = self.core_trainer()
            first_class_step = max(self.num_enc_steps - self.num_class_steps + 1, 1)
            logits = tr.autograd_logits(data, all_steps=x_ext is not None)
            skip = first_class_step - 1 if x_ext is not None else 0
            out = {'classified_edges': [logits[i].view(-1, 1) for i in range(skip, logits.shape[0])], 'mask_predictions': []}
            if x_ext is not None:
                out['mask_predictions'] = self._mask_branch_train(x_ext, logits, tr, first_class_step)
            return out
        layout = ops.edge_layout(edge_index, x.shape[0])
        first_class_step = self.num_enc_steps - self.num_class_steps + 1
        # the attention branch needs the logits of EVERY step (models/mpn.py:377), the output only the last ones
        first_needed = 1 if x_ext is not None else first_class_step
        res = self._core([x], edge_attr, layout, first_needed, want_state=return_state)
        logits = res[0]
        skip = max(first_class_step, 1) - max(first_needed, 1) if self.num_enc_steps > 0 else 0
        out = {'classified_edges': [logits[i].view(-1, 1) for i in range(skip, logits.shape[0])],
               'mask_predictions': []}
        if x_ext is not None:
            out['mask_predictions'] = self._mask_branch(x_ext, layout, logits, first_class_step)
        if return_state:
            out['node_state'], out['edge_state_slots'], out['layout'] = res[1], res[2], layout
        return out

    def _core_has_train_only_layers(self):
        """True when a core MLP has BatchNorm1d or Dropout, whose training-mode forward the inference kernels lack."""
        return any(isinstance(m, MLP) and (m.use_batchnorm or m.dropout_p != 0)
                   for m in (self.encoder.node_model, self.encoder.edge_model, self.MPNet.edge_model.edge_model,
                             self.MPNet.node_model.flow_in_model, self.MPNet.node_model.flow_out_model,
                             self.classifier.edge_model))

    def core_trainer(self):
        """The ``training.CoreTrainer`` bound to this model (built on first use: it re-homes the core parameters
        into one flat bucket, so it is created explicitly or by the first training-mode forward, never by an
        evaluation call)."""
        tr = getattr(self, '_core_trainer', None)
        if tr is None:
            from ..training import CoreTrainer
            tr = CoreTrainer(self)
        return tr

    def _mask_branch_train(self, x_ext, logits, tr, first_class_step):
        """Mask predictions in training mode (pl_module.py:107-118 adds their BCE on the matched detections to the
        loss).  The convolution stacks are torch modules; the attentive aggregation is ``training.AttnAggregate`` with
        hand-written backward kernels, so the segmentation loss reaches every mask-branch parameter and, through the
        attention weights (softmax of every step's logits), the tracking network -- as in the reference."""
        c = tr.last_ctx
        return self._mask_branch(x_ext, c['lay'], logits, first_class_step, train_ctx=c)

    def _core(self, xs, edge_attr, layout, first_needed, want_state=False, encoded=False, pooled=None):
        """Encoders + step loop.  The tensor-core kernels report fp16-range overflow through one status word per
        kernel family (mpn_mp_forward_tc clears its own at the start), read once at the end (a single host sync); 'auto'
        then reruns on the fp32 kernels (``ops.tc_or_fp32``).
        pooled: (the pooled [N, C] node features of ``xs``, event that marks them ready) when the pool already runs
        on another stream; the edge encoder, which does not need them, is enqueued before the wait."""
        engine = self.engine or ops.default_engine()
        cw, keep = self.core_weights()

        def run(eng, status=None):
            e0 = self.encode_edges(edge_attr, layout)
            if encoded:
                x0 = xs[0] if len(xs) == 1 else torch.cat(xs)
            elif pooled is not None:
                torch.cuda.current_stream().wait_event(pooled[1])
                x0 = self.encode_pooled(pooled[0], engine=eng, status=None if status is None else status[0:1])
            else:
                x0 = self.encode_nodes_list(xs, engine=eng, status=None if status is None else status[0:1])
            res = ops.mp_forward(cw, layout, x0, e0, self.num_enc_steps, first_needed, want_state=want_state,
                                 engine=eng, status=None if status is None else status[1:2])
            return res if want_state else (res,)

        res = ops.tc_or_fp32(engine, lambda status: run(engine, status), lambda: run('fp32'),
                             'a value left the fp16 range on the tensor-core path, or the step scale passed the '
                             'split operands\' resolution; use engine="fp32"',
                             'mpntrackseg_b200: value outside the fp16 range (or step scale beyond the split operands\' '
                             'resolution), rerunning the forward on the fp32 kernels')
        del keep
        return res

    def _mask_branch(self, x_ext, layout, logits, first_class_step, train_ctx=None):
        """Attentive node-feature-map updates + mask head per classified step.
        reference: models/mpn.py:356,360,369-385 (and :387-392 for num_enc_steps == 0)"""
        z0 = self.node_ext_encoder(x_ext)
        z, masks = z0, []
        for step in range(1, self.num_enc_steps + 1):
            zc = torch.cat((z0, z), dim=1).contiguous()                # reattach the initial encoding (:373)
            z = self.MPAttentionNet.aggregate(zc, layout, logits[step - 1], train_ctx=train_ctx)
            if step >= first_class_step:
                masks.append(self.mask_predictor(x_ext, z))
        if self.num_enc_steps == 0:
            masks.append(self.mask_predictor(x_ext, z))
        return masks
