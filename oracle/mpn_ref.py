"""Oracle (test infrastructure): the MOTMPNet forward pass, loss and tracker glue on CPU.

Functional restatement over a ``state_dict``-style mapping ``P`` (name -> tensor) of
models/mpn.py:33-394, models/mlp.py:4-28, models/cnn.py:4-84, pl_module.py:88-120 and
mpn_tracker.py:122-135 of the reference, plus the two torch-scatter 2.0.4 primitives used
there.  See ``oracle/__init__.py`` for who may import this.
"""
import torch
import torch.nn.functional as F


# ---------------------------------------------------------------- torch-scatter 2.0.4
def segment_add(src, index, num_segments):
    """``scatter_add(src, index, dim=0, dim_size=num_segments)``: zero-filled index-add;
    on CPU the additions happen in ascending source order."""
    out = src.new_zeros((num_segments,) + tuple(src.shape[1:]))
    return out.index_add_(0, index, src)


def segment_softmax(src, index, eps=1e-12):
    """``torch_scatter.composite.scatter_softmax(src, index, dim=0)``:
    exp(src - max_of_segment) / (sum_of_segment + eps).  Segments = int(index.max()) + 1."""
    if src.numel() == 0:
        return src.clone()
    n = int(index.max()) + 1
    idx = index.view(-1, *([1] * (src.dim() - 1))).expand_as(src)
    seg_max = src.new_full((n,) + tuple(src.shape[1:]), float('-inf'))
    seg_max = seg_max.scatter_reduce(0, idx, src, 'amax', include_self=True)
    ex = (src - seg_max.gather(0, idx)).exp()
    seg_sum = segment_add(ex, index, n)
    return ex / (seg_sum.gather(0, idx) + eps)


# ---------------------------------------------------------------- building blocks
def _linear_slots(P, prefix):
    slots = sorted({int(k[len(prefix) + 1:].split('.')[1]) for k in P
                    if k.startswith(prefix + '.fc_layers.') and k.endswith('.weight')})
    return slots


def mlp(P, prefix, h):
    """Linear [-> BatchNorm1d (evaluation mode: running statistics)] -> ReLU per layer; a layer whose width is 1 is a
    bare Linear; Dropout is the identity in evaluation mode.  reference: models/mlp.py:12-23"""
    for s in _linear_slots(P, prefix):
        w, b = P[f'{prefix}.fc_layers.{s}.weight'], P[f'{prefix}.fc_layers.{s}.bias']
        if w.dim() != 2:
            continue                                   # a BatchNorm1d weight vector, handled with its Linear
        h = F.linear(h, w, b)
        bn = f'{prefix}.fc_layers.{s + 1}'
        if w.shape[0] != 1 and f'{bn}.running_mean' in P:
            h = F.batch_norm(h, P[f'{bn}.running_mean'], P[f'{bn}.running_var'], P[f'{bn}.weight'], P[f'{bn}.bias'],
                             training=False, eps=1e-5)
        if w.shape[0] != 1:
            h = F.relu(h)
    return h


def cnn(P, prefix, h, paddings, strides=None):
    """Conv2d -> ReLU after EVERY conv (the ``dims[i] != 0`` test is always true).
    reference: models/cnn.py:25-41"""
    n = len(paddings)
    for i in range(n):
        h = F.conv2d(h, P[f'{prefix}.layers.{2 * i}.weight'], P[f'{prefix}.layers.{2 * i}.bias'],
                     stride=1 if strides is None else strides[i], padding=paddings[i])
        h = F.relu(h)
    return h


def mask_rcnn_predictor(P, prefix, h, cfg):
    """(Transposed) convs with ReLU between, none after the last.
    reference: models/cnn.py:70-82"""
    n = len(cfg['dims'])
    for i in range(n):
        w, b = P[f'{prefix}.layers.{2 * i}.weight'], P[f'{prefix}.layers.{2 * i}.bias']
        if cfg['transposed'][i]:
            h = F.conv_transpose2d(h, w, b, stride=cfg['strides'][i], padding=cfg['paddings'][i])
        else:
            h = F.conv2d(h, w, b, stride=cfg['strides'][i], padding=cfg['paddings'][i])
        if i < n - 1:
            h = F.relu(h)
    return h


def edge_update(P, x, edge_index, e):
    """e' = MLP(cat[x[row], x[col], e]).  reference: models/mpn.py:67-69"""
    src, dst = edge_index[0], edge_index[1]
    return mlp(P, 'MPNet.edge_model.edge_model', torch.cat((x[src], x[dst], e), dim=1))


def node_update(P, x, edge_index, e, agg='sum'):
    """Time-aware node update: messages MLP(cat[x[col], e]) of edges with row<col are
    aggregated on ``row`` as flow_out, those with row>col as flow_in;
    x' = ReLU(Linear(cat[flow_in, flow_out])).  reference: models/mpn.py:83-99"""
    src, dst = edge_index[0], edge_index[1]
    n = x.shape[0]
    flows = {}
    for name, sel in (('flow_out', src < dst), ('flow_in', src > dst)):
        msg = mlp(P, f'MPNet.node_model.{name}_model', torch.cat((x[dst[sel]], e[sel]), dim=1))
        flows[name] = _aggregate(msg, src[sel], n, agg)
    both = torch.cat((flows['flow_in'], flows['flow_out']), dim=1)
    return F.relu(F.linear(both, P['MPNet.node_model.node_model.0.weight'],
                           P['MPNet.node_model.node_model.0.bias']))


def _aggregate(msg, index, n, agg):
    """reference: models/mpn.py:263-273"""
    if agg == 'sum':
        return segment_add(msg, index, n)
    idx = index.view(-1, 1).expand_as(msg)
    if agg == 'mean':
        cnt = segment_add(torch.ones_like(msg), index, n).clamp(min=1)
        return segment_add(msg, index, n) / cnt
    if agg == 'max':
        out = msg.new_zeros((n, msg.shape[1]))
        return out.scatter_reduce(0, idx, msg, 'amax', include_self=False)
    raise ValueError(agg)


def classify(P, e):
    """Edge logit, no final activation.  reference: models/mpn.py:114, models/mlp.py:14-21"""
    return mlp(P, 'classifier.edge_model', e)


def attention_update(P, model_params, x_ext, edge_index, logits):
    """Softmax of the edge logits over each node's future (row<col) resp. past (row>col)
    neighbours, weighted sum of the neighbours' x_ext maps, then the 3x3 conv stack on
    cat[x_ext, flow_in, flow_out].  reference: models/mpn.py:117-137"""
    src, dst = edge_index[0], edge_index[1]
    n = x_ext.shape[0]
    flows = {}
    for name, sel in (('flow_out', src < dst), ('flow_in', src > dst)):
        w = segment_softmax(logits[sel], src[sel])
        flows[name] = segment_add(x_ext[dst[sel]] * w[:, :, None, None], src[sel], n)
    cat = torch.cat((x_ext, flows['flow_in'], flows['flow_out']), dim=1)
    return cnn(P, 'MPAttentionNet.node_model', cat,
               model_params['node_ext_model_feats_dict']['paddings'])


def mask_model(P, model_params, feats, node_embeds):
    """reference: models/mpn.py:200-206"""
    mm = model_params['mask_model_feats_dict']
    f = cnn(P, 'mask_predictor.feature_encoder', feats,
            mm['feature_encoder_feats_dict']['paddings'])
    h = torch.cat((f, node_embeds), dim=1)
    h = F.layer_norm(h, (64, 14, 14), P['mask_predictor.layer_norm.weight'],
                     P['mask_predictor.layer_norm.bias'])
    h = cnn(P, 'mask_predictor.mask_head', h, mm['mask_head_feats_dict']['paddings'])
    return mask_rcnn_predictor(P, 'mask_predictor.mask_predictor', h,
                               mm['mask_predictor_feats_dict'])


# ---------------------------------------------------------------- the model
def encode(P, x, edge_attr):
    """Global average pool + node MLP; edge MLP.  reference: models/mpn.py:351-355"""
    pooled = x.mean(dim=(2, 3)) if x.dim() == 4 else x
    return mlp(P, 'encoder.node_model', pooled), mlp(P, 'encoder.edge_model', edge_attr)


def mpn_forward(P, model_params, x, edge_index, edge_attr, x_ext=None, return_state=False):
    """MOTMPNet.forward.  With ``x_ext=None`` only the core path (the one the edge
    logits depend on) is evaluated and 'mask_predictions' stays empty.
    reference: models/mpn.py:333-394"""
    x0, e0 = encode(P, x, edge_attr)
    return mp_steps(P, model_params, x0, e0, edge_index, x_ext=x_ext, return_state=return_state)


def mp_steps(P, model_params, x0, e0, edge_index, x_ext=None, return_state=False):
    """The step loop of ``mpn_forward`` from the encoded node / edge states ``x0`` [N, dn], ``e0`` [E, de]
    (edges in the caller's order).  reference: models/mpn.py:356-394"""
    steps = model_params['num_enc_steps']
    first_cls = steps - model_params['num_class_steps'] + 1
    agg = model_params['node_agg_fn']
    xs, es = x0, e0
    ext = x_ext is not None
    if ext:
        z0 = cnn(P, 'node_ext_encoder', x_ext, model_params['node_ext_encoder_feats_dict']['paddings'])
        zs = z0
    out = {'classified_edges': [], 'mask_predictions': []}
    for step in range(1, steps + 1):
        if model_params['reattach_initial_edges']:
            es = torch.cat((e0, es), dim=1)
        if model_params['reattach_initial_nodes']:
            xs = torch.cat((x0, xs), dim=1)
            if ext:
                zs = torch.cat((z0, zs), dim=1)
        e_new = edge_update(P, xs, edge_index, es)
        xs = node_update(P, xs, edge_index, e_new, agg)
        es = e_new
        logits = classify(P, es)
        if ext:
            zs = attention_update(P, model_params, zs, edge_index, logits)
        if step >= first_cls:
            out['classified_edges'].append(logits)
            if ext:
                out['mask_predictions'].append(mask_model(P, model_params, x_ext, zs))
    if steps == 0:
        out['classified_edges'].append(classify(P, es))
        if ext:
            out['mask_predictions'].append(mask_model(P, model_params, x_ext, zs))
    if return_state:
        out['node_state'], out['edge_state'] = xs, es
    return out


# ---------------------------------------------------------------- callers' glue
def weighted_bce_loss(classified_edges, edge_labels, tracking_weight=1.0):
    """Sum over classified steps of BCE-with-logits, positives weighted by #neg/#pos.
    reference: pl_module/pl_module.py:88-105"""
    pos = edge_labels.sum()
    if pos:
        pos_weight = (edge_labels.shape[0] - pos) / pos
    else:
        pos_weight = torch.zeros(1)
    loss = 0
    for logits in classified_edges:
        loss = loss + tracking_weight * F.binary_cross_entropy_with_logits(
            logits.view(-1), edge_labels.view(-1), pos_weight=pos_weight)
    return loss


def window_edge_preds(classified_edges, keep_mask):
    """sigmoid of the last step's logits scattered back to the unpruned edge list.
    reference: tracker/mpn_tracker.py:128-135"""
    p = torch.sigmoid(classified_edges[-1].view(-1))
    full = torch.zeros(keep_mask.shape[0])
    full[keep_mask] = p
    return full
