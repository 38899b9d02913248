"""Training of the core network with the reference MLPs' options: node_agg_fn mean / max, BatchNorm1d (batch
statistics) and Dropout, against torch autograd through a training-mode restatement of the oracle's forward.

The restatement (``train_forward`` below) is the oracle's ``mpn_forward`` with the training-mode semantics of
models/mlp.py (``F.batch_norm(training=True)`` on given running buffers, dropout with given masks) and a max aggregation
whose gradient goes to one argmax, the lowest caller edge id among ties (torch_scatter's CPU ``scatter_max``).  The CPU
tests pin it to ``nn.Sequential(Linear, BatchNorm1d, ReLU)`` in train() mode and, with the options off, to
``oracle.mpn_ref.mpn_forward`` bit for bit."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from cases import load_case
from oracle import mpn_ref

CORE = ('encoder.', 'classifier.', 'MPNet.')
LOSS_TOL, GRAD_TOL = 2e-4, 2e-3
# launches of one eager CoreTrainer.train_step on tiny_nonrecip with the shipped options (sum, no BatchNorm, no
# Dropout), as counted by mpn_launch_count at the commit before these options were trainable
SHIPPED_TRAIN_STEP_LAUNCHES = 228


# ------------------------------------------------------------------ training-mode restatement of the oracle
def _slots(P, prefix):
    return [s for s in mpn_ref._linear_slots(P, prefix) if P[f'{prefix}.fc_layers.{s}.weight'].dim() == 2]


def train_mlp(P, prefix, h, bufs, p=0.0, masks=None, tag=''):
    """models/mlp.py in train() mode: Linear [-> BatchNorm1d on the batch, updating ``bufs``] -> ReLU [-> dropout with
    the mask ``masks(name)`` of Linear ``name``, scaled by 1 / (1 - p)]; a layer of width 1 is a bare Linear."""
    for s in _slots(P, prefix):
        w, b = P[f'{prefix}.fc_layers.{s}.weight'], P[f'{prefix}.fc_layers.{s}.bias']
        h = F.linear(h, w, b)
        if w.shape[0] == 1:
            continue
        bn = f'{prefix}.fc_layers.{s + 1}'
        if f'{bn}.running_mean' in bufs:
            h = F.batch_norm(h, bufs[f'{bn}.running_mean'], bufs[f'{bn}.running_var'], P[f'{bn}.weight'], P[f'{bn}.bias'],
                             training=True, momentum=0.1, eps=1e-5)
            bufs[f'{bn}.num_batches_tracked'] += 1
        h = F.relu(h)
        if p:
            h = h * masks(f'{prefix}.fc_layers.{s}{tag}').to(h.dtype) / (1 - p)
    return h


def max_argmax(msg, index, n):
    """scatter_max values (0 for an empty segment) with the gradient to the lowest-index argmax of each segment."""
    out = msg.new_zeros((n, msg.shape[1]))
    if msg.shape[0] == 0:
        return out
    idx = index.view(-1, 1).expand_as(msg)
    val = out.scatter_reduce(0, idx, msg.detach(), 'amax', include_self=False)
    e = msg.shape[0]
    cand = torch.where(msg.detach() == val[index], torch.arange(e).view(-1, 1).expand_as(msg), e)
    arg = torch.full((n, msg.shape[1]), e, dtype=torch.int64).scatter_reduce(0, idx, cand, 'amin', include_self=True)
    return torch.where(arg < e, msg.gather(0, arg.clamp(max=e - 1)), out)


def aggregate(msg, index, n, agg):
    return max_argmax(msg, index, n) if agg == 'max' else mpn_ref._aggregate(msg, index, n, agg)


def train_forward(P, mp, x, ei, ea, bufs, p=0.0, masks=None):
    """models/mpn.py:349-381 in train() mode; returns the classified steps' logits."""
    src, dst = ei[0], ei[1]
    n, agg = x.shape[0], mp['node_agg_fn']
    x = x.mean(dim=(2, 3)) if x.dim() == 4 else x
    x0 = train_mlp(P, 'encoder.node_model', x, bufs, p, masks)
    e0 = train_mlp(P, 'encoder.edge_model', ea, bufs, p, masks)
    steps, first = mp['num_enc_steps'], mp['num_enc_steps'] - mp['num_class_steps'] + 1
    xs, es, out = x0, e0, []
    for step in range(1, steps + 1):
        xs, es = torch.cat((x0, xs), 1), torch.cat((e0, es), 1)
        e_new = train_mlp(P, 'MPNet.edge_model.edge_model', torch.cat((xs[src], xs[dst], es), 1), bufs, p, masks, f'@{step}')
        flows = {}
        for name, sel in (('out', src < dst), ('in', src > dst)):
            msg = train_mlp(P, f'MPNet.node_model.flow_{name}_model', torch.cat((xs[dst[sel]], e_new[sel]), 1), bufs, p,
                            masks, f'@{step}.{name}')
            flows[name] = aggregate(msg, src[sel], n, agg)
        xs = F.relu(F.linear(torch.cat((flows['in'], flows['out']), 1), P['MPNet.node_model.node_model.0.weight'],
                             P['MPNet.node_model.node_model.0.bias']))
        es = e_new
        lg = train_mlp(P, 'classifier.edge_model', es, bufs, p, masks, f'@{step}')
        if step >= first:
            out.append(lg)
    return out


def slot_masks(ctx, ei):
    """The trainer's dropout masks (slot order) as a lookup in the caller's order of each call's rows."""
    sedge, n_out = ctx['sedge'].long().cpu(), ctx['n_out']
    src, dst = ei[0], ei[1]

    def get(key):
        m = ctx['masks'][key].cpu()
        if key.startswith('encoder.node_model'):
            return m
        full = torch.zeros((ei.shape[1], m.shape[1]), dtype=m.dtype)
        if key.endswith('.out'):
            full[sedge[:n_out]] = m
            return full[src < dst]
        if key.endswith('.in'):
            full[sedge[n_out:]] = m
            return full[src > dst]
        full[sedge] = m
        return full
    return get


def split_state(P):
    params = {k: v for k, v in P.items() if v.is_floating_point() and not k.endswith(('running_mean', 'running_var'))}
    bufs = {k: v.clone() for k, v in P.items() if k.endswith(('running_mean', 'running_var', 'num_batches_tracked'))}
    return params, bufs


def oracle_loss_and_grads(P, mp, x, ei, ea, labels, weight=1.0, p=0.0, masks=None, dtype=torch.float32):
    params, bufs = split_state(P)
    Pg = {k: v.detach().to(dtype, copy=True).requires_grad_(True) for k, v in params.items()}
    bufs = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in bufs.items()}
    out = train_forward(Pg, mp, x.to(dtype), ei, ea.to(dtype), bufs, p, masks)
    loss = mpn_ref.weighted_bce_loss(out, labels.to(dtype), tracking_weight=weight)
    loss.backward()
    return float(loss.detach()), {k: v.grad for k, v in Pg.items() if v.grad is not None}, bufs, [o.detach() for o in out]


# ------------------------------------------------------------------ CPU checks of the restatement
def test_train_mlp_matches_torch_modules_in_train_mode():
    torch.manual_seed(5)
    seq = torch.nn.Sequential(torch.nn.Linear(7, 12), torch.nn.BatchNorm1d(12), torch.nn.ReLU(),
                              torch.nn.Linear(12, 5), torch.nn.BatchNorm1d(5), torch.nn.ReLU(), torch.nn.Linear(5, 1))
    with torch.no_grad():
        for m in seq:
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5); m.bias.uniform_(-0.3, 0.3)
                m.running_mean.uniform_(-0.2, 0.2); m.running_var.uniform_(0.5, 1.5)
    P = {f'm.fc_layers.{k}': v.detach().clone() for k, v in seq.state_dict().items()}
    params, bufs = split_state(P)
    seq.train()
    for rows in (2, 9, 33):
        x = torch.randn(rows, 7)
        ref = seq(x)
        got = train_mlp(params, 'm', x, bufs)
        torch.testing.assert_close(got, ref, rtol=0, atol=0)
    for k, v in seq.state_dict().items():
        if 'running' in k or 'num_batches' in k:
            assert torch.equal(bufs[f'm.fc_layers.{k}'], v), k


@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_train_forward_without_options_is_the_oracle_forward(agg):
    c = load_case('tiny_nonrecip')
    win, gold, mp = c['win'], c['gold'], copy.deepcopy(c['mp'])
    mp['node_agg_fn'] = agg
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    ea = torch.from_numpy(gold['edge_attr'])
    ref = mpn_ref.mpn_forward(c['P'], mp, win.x, ei, ea)['classified_edges']
    got = train_forward(c['P'], mp, win.x, ei, ea, {})
    assert len(got) == len(ref) and all(torch.equal(a, b) for a, b in zip(got, ref))


def test_max_argmax_gradient_goes_to_the_lowest_index_among_ties():
    msg = torch.tensor([[1.0, 2.0], [3.0, 2.0], [3.0, 0.5], [0.1, 0.2]], requires_grad=True)
    out = max_argmax(msg, torch.tensor([0, 0, 0, 2]), 4)
    assert torch.equal(out.detach(), torch.tensor([[3.0, 2.0], [0, 0], [0.1, 0.2], [0, 0]]))
    out.sum().backward()
    assert torch.equal(msg.grad, torch.tensor([[0.0, 1.0], [1.0, 0.0], [0.0, 0.0], [1.0, 1.0]]))


# ------------------------------------------------------------------ GPU
def dev():
    return torch.device('cuda:0')


class Data:
    pass


def make_data(x, ei, ea):
    d = Data()
    d.x, d.edge_index, d.edge_attr, d.x_ext = x.to(dev()), ei.to(dev()), ea.to(dev()), None
    return d


def make_model(mp, P):
    from mpntrackseg_b200.models.mpn import MOTMPNet
    model = MOTMPNet(mp).to(dev()).eval()
    model.engine = 'fp32'
    model.load_state_dict(P, strict=False)
    return model


def relayout(P, mp):
    """The core tensors of ``P`` under the state_dict names of ``mp``: adding or removing Dropout shifts the Sequential
    slots of the Linear and BatchNorm layers, not the order or shapes of their tensors."""
    from mpntrackseg_b200.config import param_shapes
    names, src = param_shapes(mp, core_only=True), [k for k in P if k.startswith(CORE)]
    assert len(names) == len(src) and all(tuple(P[k].shape) == tuple(s) for k, s in zip(src, names.values()))
    return {n: P[k] for n, k in zip(names, src)}


def load(name, agg=None, batchnorm=None, p=None):
    """A golden case's graph, weights and labels, with model options overridden (weights of a BatchNorm model come
    from the tiny_bn recipe: synth.make_params with the case's seed)."""
    from mpntrackseg_b200 import synth
    c = load_case(name)
    mp = copy.deepcopy(c['mp'])
    if agg is not None:
        mp['node_agg_fn'] = agg
    for k in ('encoder_feats_dict', 'edge_model_feats_dict', 'node_model_feats_dict', 'classifier_feats_dict'):
        if batchnorm is not None:
            mp[k]['use_batchnorm'] = batchnorm
        if p is not None:
            mp[k]['dropout_p'] = p
    if batchnorm and not c['mp']['encoder_feats_dict']['use_batchnorm']:
        P = synth.make_params(mp, seed=c['case']['wseed'], gain=c['case']['gain'])
    else:
        P = relayout(c['P'], mp)
    ei = torch.from_numpy(c['gold']['edge_index'].astype(np.int64))
    ea = torch.from_numpy(c['gold']['edge_attr'])
    labels = (c['win'].ident[ei[0]] == c['win'].ident[ei[1]]).float()
    return dict(mp=mp, P=P, x=c['win'].x, ei=ei, ea=ea, labels=labels)


def bn_fed_biases(P):
    """Biases of the Linear layers that feed a BatchNorm1d: their exact gradient is 0."""
    return {f'{base}.{int(s) - 1}.bias' for base, s, last in (k.rsplit('.', 2) for k in P) if last == 'running_mean'}


def assert_grads(got, ref, what='', bn_fed=()):
    """Each gradient within GRAD_TOL of its own max; a bias in ``bn_fed`` is rounding noise on both sides and is judged
    absolutely, against 1e-6 of the layer's weight-gradient max."""
    for k, g in ref.items():
        err = float((got[k].detach().cpu().to(g.dtype) - g).abs().max())
        if k in bn_fed:
            assert err <= 1e-6 * float(ref[k[:-4] + 'weight'].abs().max()), (what, k, err)
            continue
        scale = float(g.abs().max()) + 1e-30
        assert err / scale <= GRAD_TOL, (what, k, err / scale)


def assert_logits_bar(got, ref, what=''):
    for a, b in zip(got, ref):
        a, b = a.detach().cpu().double().view(-1), b.detach().cpu().double().view(-1)
        assert float((a - b).abs().max()) <= 1e-3 * max(1.0, float(b.abs().max())), what


AGG_CASES = [('tiny_mean', None), ('tiny_max', None), ('kitti_shape', 'mean'), ('kitti_shape', 'max')]


@pytest.mark.gpu
@pytest.mark.parametrize('name,agg', AGG_CASES)
def test_mean_max_training_matches_oracle_autograd(name, agg):
    from mpntrackseg_b200.training import CoreTrainer
    d = load(name, agg=agg)
    ref_loss, ref_g, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'], 0.8)
    data = make_data(d['x'], d['ei'], d['ea'])
    tr = CoreTrainer(make_model(d['mp'], d['P']))
    loss = tr.loss_and_grads(data, d['labels'].to(dev()), tracking_weight=0.8)
    assert abs(float(loss) - ref_loss) <= LOSS_TOL * max(1.0, abs(ref_loss))
    assert set(tr.g) == set(ref_g)
    assert_grads(tr.g, ref_g, name)
    g1 = tr.grad.clone()
    tr.loss_and_grads(data, d['labels'].to(dev()), tracking_weight=0.8)
    assert torch.equal(g1, tr.grad)

    # the reference's training call: model.train()(data), a torch loss, loss.backward()
    model = make_model(d['mp'], d['P'])
    with torch.no_grad():
        inf = model(data)['classified_edges']
    out = model.train()(data)
    assert_logits_bar(out['classified_edges'], inf, name)
    loss = mpn_ref.weighted_bce_loss(out['classified_edges'], d['labels'].to(dev()))
    ref_loss1, ref_g1, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'])
    assert abs(float(loss) - ref_loss1) <= LOSS_TOL * max(1.0, abs(ref_loss1))
    loss.backward()
    named = dict(model.named_parameters())
    assert_grads({k: named[k].grad for k in ref_g1}, ref_g1, name + ' autograd')


@pytest.mark.gpu
def test_max_ties_send_the_gradient_to_the_lowest_caller_edge():
    """Duplicated edges carry identical messages at every step, so their flow_out / flow_in groups hold exact ties."""
    from mpntrackseg_b200.training import CoreTrainer
    d = load('tiny_max')
    ei, ea = d['ei'], d['ea']
    g = torch.Generator().manual_seed(31)
    dup = torch.randperm(ei.shape[1], generator=g)[:ei.shape[1] // 3]
    ei, ea = torch.cat((ei, ei[:, dup]), 1), torch.cat((ea, ea[dup]), 0)
    labels = torch.cat((d['labels'], d['labels'][dup]))
    ref_loss, ref_g, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], ei, ea, labels, dtype=torch.float64)
    data = make_data(d['x'], ei, ea)
    tr = CoreTrainer(make_model(d['mp'], d['P']))
    loss = tr.loss_and_grads(data, labels.to(dev()))
    assert abs(float(loss) - ref_loss) <= LOSS_TOL * max(1.0, abs(ref_loss))
    assert_grads(tr.g, ref_g, 'ties')
    # the argmax of every segment is a slot of the lowest caller edge among equal messages: no duplicate's slot wins
    _, ctx = tr.forward_core(data)
    slot_of = torch.empty(ei.shape[1], dtype=torch.int64)
    slot_of[ctx['sedge'].long().cpu()] = torch.arange(ei.shape[1])
    dup_slots = slot_of[ei.shape[1] - dup.numel():]
    ties = 0
    for sv in ctx['saved']:
        arg = sv['argmax'].cpu().long()
        assert not torch.isin(arg, dup_slots).any()
        ties += int(torch.isin(arg, slot_of[dup]).sum())
    assert ties > 0, 'no tied maximum was exercised'


def hub_graph(deg, leaves, seed):
    """Hub rows with ``deg`` neighbours below and above them (flow_out and flow_in groups of ``deg`` slots), leaves on
    both sides, and an isolated node.  Low leaves only have row<col edges: they have no incoming (flow_in) group."""
    g = torch.Generator().manual_seed(seed)
    L, hubs = leaves, len(deg)
    pairs = []
    for i, d in enumerate(deg):
        h = L + i
        lo = torch.randperm(L, generator=g)[:d]
        hi = L + hubs + torch.randperm(L, generator=g)[:d]
        nb = torch.cat((lo, hi))
        pairs.append(torch.stack((torch.full_like(nb, h), nb)))
    p = torch.cat(pairs, 1)
    ei = torch.cat((p, p.flip(0)), 1)
    return ei, 2 * L + hubs + 1


@pytest.mark.gpu
@pytest.mark.parametrize('agg', ['mean', 'max'])
def test_mean_max_training_on_a_hub_graph(agg):
    from mpntrackseg_b200 import synth
    from mpntrackseg_b200.config import default_graph_model_params
    from mpntrackseg_b200.training import CoreTrainer
    ei, n = hub_graph([1, 17, 129, 1025, 1100], leaves=1200, seed=41)
    fin = torch.bincount(ei[0][ei[0] > ei[1]], minlength=n)
    assert int(torch.bincount(ei[0][ei[0] < ei[1]], minlength=n).max()) > 1024 and int(fin.max()) > 1024
    assert (fin == 0).sum() > 1 and int(torch.bincount(ei[0], minlength=n)[-1]) == 0
    mp = default_graph_model_params(3, 2)
    mp['node_agg_fn'] = agg
    P = synth.make_params(mp, seed=42, gain=1.0, core_only=True)
    g = torch.Generator().manual_seed(43)
    x, ea = torch.rand(n, 2048, generator=g), torch.rand(ei.shape[1], 6, generator=g)
    labels = (torch.rand(ei.shape[1], generator=g) < 0.3).float()
    ref_loss, ref_g, _, _ = oracle_loss_and_grads(P, mp, x, ei, ea, labels, 0.8, dtype=torch.float64)
    tr = CoreTrainer(make_model(mp, P))
    data = make_data(x, ei, ea)
    loss = tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert abs(float(loss) - ref_loss) <= LOSS_TOL * max(1.0, abs(ref_loss))
    assert_grads(tr.g, ref_g, f'hub {agg}')
    g1 = tr.grad.clone()
    tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert torch.equal(g1, tr.grad)


def bn_buffers(model):
    return {k: v.detach().cpu().clone() for k, v in model.state_dict().items()
            if k.startswith(CORE) and k.endswith(('running_mean', 'running_var', 'num_batches_tracked'))}


@pytest.mark.gpu
def test_batchnorm_training_matches_oracle_autograd_and_buffers():
    from mpntrackseg_b200.training import CoreTrainer
    d = load('tiny_bn', p=0)
    ref_loss, ref_g, ref_bufs, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'], 0.8)
    assert any('fc_layers.1.weight' in k for k in ref_g)                 # BatchNorm gamma / beta are trained
    model = make_model(d['mp'], d['P'])
    tr = CoreTrainer(model)
    data = make_data(d['x'], d['ei'], d['ea'])
    loss = tr.loss_and_grads(data, d['labels'].to(dev()), tracking_weight=0.8)
    assert abs(float(loss) - ref_loss) <= LOSS_TOL * max(1.0, abs(ref_loss))
    assert set(tr.g) == set(ref_g)
    assert_grads(tr.g, ref_g, 'bn', bn_fed_biases(d['P']))
    got = bn_buffers(model)
    assert set(got) == set(ref_bufs)
    for k, v in ref_bufs.items():
        if k.endswith('num_batches_tracked'):
            assert int(got[k]) == int(v), k
        else:
            assert float((got[k] - v).abs().max()) <= 1e-5 * max(1.0, float(v.abs().max())), k
    steps = d['mp']['num_enc_steps']
    assert int(got['MPNet.edge_model.edge_model.fc_layers.1.num_batches_tracked']) == 100 + steps

    # a training-mode forward under no_grad: batch statistics (the logits of any training forward without dropout),
    # the running statistics move, no backward
    before = bn_buffers(model)
    with torch.no_grad():
        out = model.train()(data)['classified_edges']
    lg, ctx = tr.forward_core(data)
    after = bn_buffers(model)
    assert int(after['classifier.edge_model.fc_layers.1.num_batches_tracked']) == \
        int(before['classifier.edge_model.fc_layers.1.num_batches_tracked']) + 2 * steps
    assert torch.equal(torch.stack([o.view(-1) for o in out])[:, ctx['sedge'].long()], lg)

    # three Adam steps, then evaluation mode folds the trained statistics into the inference kernels
    model = make_model(d['mp'], d['P'])
    tr = CoreTrainer(model)
    for _ in range(3):
        tr.train_step(data, d['labels'].to(dev()))
    torch.cuda.synchronize()
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items() if k.startswith(CORE)}
    with torch.no_grad():
        got = model.eval()(data)['classified_edges']
        ref = mpn_ref.mpn_forward(sd, d['mp'], d['x'], d['ei'], d['ea'])['classified_edges']
    assert_logits_bar(got, ref, 'bn eval after training')


@pytest.mark.gpu
def test_batchnorm_empty_and_single_row_calls():
    from mpntrackseg_b200.training import CoreTrainer
    d = load('tiny_bn', p=0)
    ei = d['ei']
    keep = ei[0] < ei[1]                                           # every edge row<col: flow_in gets 0 rows
    ei, ea, labels = ei[:, keep], d['ea'][keep], d['labels'][keep]
    model = make_model(d['mp'], d['P'])
    tr = CoreTrainer(model)
    before = bn_buffers(model)
    data = make_data(d['x'], ei, ea)
    tr.loss_and_grads(data, labels.to(dev()))
    after = bn_buffers(model)
    steps = d['mp']['num_enc_steps']
    for k in before:
        if 'flow_in_model' in k:
            if k.endswith('num_batches_tracked'):
                assert int(after[k]) == int(before[k]) + steps, k
            else:
                assert torch.equal(after[k], before[k]), k
        elif 'flow_out_model' in k and k.endswith('running_mean'):
            assert not torch.equal(after[k], before[k]), k
    _, ref_g, ref_bufs, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], ei, ea, labels)
    assert_grads(tr.g, ref_g, 'flow_in empty', bn_fed_biases(d['P']))
    for k, v in ref_bufs.items():
        assert float((after[k].double() - v.double()).abs().max()) <= 1e-5 * max(1.0, float(v.abs().max())), k

    one = make_data(d['x'][:2], torch.tensor([[0], [1]]), d['ea'][:1])   # the edge encoder sees 1 row
    with pytest.raises(ValueError, match='Expected more than 1 value per channel'):
        tr.loss_and_grads(one, torch.ones(1, device=dev()))


def step_with_masks(tr, data, labels):
    """One training forward with its dropout masks kept, the loss and the backward (gradients in ``tr.g``)."""
    from mpntrackseg_b200 import ops
    tr.grad.zero_()
    lg, ctx = tr.forward_core(data, keep_masks=True)
    lab = labels.to(dev())[ctx['sedge'].long()].contiguous()
    loss, _, gl = ops.weighted_bce(lg, lab, weight=1.0, want_grad=True)
    tr.backward_core(ctx, gl)
    return loss, ctx


@pytest.mark.gpu
@pytest.mark.parametrize('name,p', [('tiny_bn', None), ('kitti_shape', 0.3)], ids=['tiny_bn', 'kitti_shape_no_bn'])
def test_dropout_training(name, p):
    from mpntrackseg_b200.training import CoreTrainer
    d = load(name, p=p)
    p = d['mp']['edge_model_feats_dict']['dropout_p']
    assert p == 0.3
    data = make_data(d['x'], d['ei'], d['ea'])
    tr = CoreTrainer(make_model(d['mp'], d['P']), seed=1234)
    tr.forward_core(data)                                           # forward 1
    loss, ctx = step_with_masks(tr, data, d['labels'])              # forward 2
    masks = ctx['masks']
    assert len(masks) == 2 + 3 + 7 * d['mp']['num_enc_steps']      # encoders, then edge / flow_out / flow_in / classifier
    for k, m in masks.items():
        if m.numel():
            frac = 1 - float(m.float().mean())
            assert abs(frac - p) <= 5 * (p * (1 - p) / m.numel()) ** 0.5, (k, frac, m.numel())
    ref_loss, ref_g, _, _ = oracle_loss_and_grads(d['P'], d['mp'], d['x'], d['ei'], d['ea'], d['labels'], p=p,
                                                  masks=slot_masks(ctx, d['ei']))
    assert abs(float(loss) - ref_loss) <= LOSS_TOL * max(1.0, abs(ref_loss))
    assert_grads(tr.g, ref_g, f'dropout {name}', bn_fed_biases(d['P']))
    # the same seed and forward counter give the same masks and gradients; the next forward draws new masks
    tr2 = CoreTrainer(make_model(d['mp'], d['P']), seed=1234)
    tr2.forward_core(data)
    loss2, ctx2 = step_with_masks(tr2, data, d['labels'])
    assert torch.equal(tr2.grad, tr.grad) and float(loss2) == float(loss)
    assert all(torch.equal(ctx2['masks'][k], m) for k, m in masks.items())
    _, ctx3 = tr2.forward_core(data, keep_masks=True)
    assert all(not torch.equal(ctx3['masks'][k], m) for k, m in masks.items() if m.numel() > 64)


@pytest.mark.gpu
def test_dropout_p_to_zero_is_the_no_dropout_result():
    from mpntrackseg_b200.training import CoreTrainer
    grads = []
    for p in (2.0 ** -30, 0.0):
        d = load('tiny_bn', p=p)
        tr = CoreTrainer(make_model(d['mp'], d['P']), seed=7)
        data = make_data(d['x'], d['ei'], d['ea'])
        tr.loss_and_grads(data, d['labels'].to(dev()))
        lg, ctx = tr.forward_core(data, keep_masks=True)
        if p:
            assert ctx['masks'] and all(bool(m.all()) for m in ctx['masks'].values())
        grads.append((tr.grad.clone(), lg))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


GRAPH_OPTIONS = [dict(agg='mean'), dict(agg='max'), dict(batchnorm=True, p=0), dict(batchnorm=True, p=0.3)]


@pytest.mark.gpu
@pytest.mark.parametrize('opt', GRAPH_OPTIONS, ids=['mean', 'max', 'bn', 'bn_dropout'])
def test_graphed_steps_equal_eager_steps(opt):
    from mpntrackseg_b200.training import CoreTrainer
    d = load('tiny_nonrecip', **opt)
    data = make_data(d['x'], d['ei'], d['ea'])
    labels = d['labels'].to(dev())
    trs = [CoreTrainer(make_model(d['mp'], d['P']).train(), seed=99) for _ in range(2)]
    for _ in range(3):
        trs[0].train_step(data, labels)
        trs[1].graphed_step(data, labels)
    torch.cuda.synchronize()
    a, b = trs
    for x, y in ((a.flat, b.flat), (a.exp_avg, b.exp_avg), (a.exp_avg_sq, b.exp_avg_sq), (a.t_dev, b.t_dev)):
        assert torch.equal(x, y)
    for x, y in zip(a._forward_state(), b._forward_state()):
        assert torch.equal(x, y)
    if opt.get('p'):
        assert int(a.fwd_dev) == 3
        _, ca = a.forward_core(data, keep_masks=True)
        _, cb = b.forward_core(data, keep_masks=True)
        assert all(torch.equal(ca['masks'][k], cb['masks'][k]) for k in ca['masks'])


@pytest.mark.gpu
def test_shipped_options_keep_the_training_step_launches():
    from mpntrackseg_b200 import _cabi
    from mpntrackseg_b200.training import CoreTrainer
    d = load('tiny_nonrecip')
    tr = CoreTrainer(make_model(d['mp'], d['P']))
    data = make_data(d['x'], d['ei'], d['ea'])
    labels = d['labels'].to(dev())
    tr.train_step(data, labels)
    lib = _cabi.lib()
    l0 = lib.mpn_launch_count()
    tr.train_step(data, labels)
    assert int(lib.mpn_launch_count() - l0) == SHIPPED_TRAIN_STEP_LAUNCHES
