"""GPU tests of the kernels past their tile, degree and batch boundaries, against the oracle evaluated in fp64.

The parity suite feeds the kernels KNN windows: per-direction degrees of the order of k, at most 36,000 nodes,
windows of similar magnitude in one batch.  The cases here are built to cross the boundaries those graphs never
reach, and every test asserts that its case really crosses the boundary it names:

* more than one 128-node tile per CTA group in the persistent node kernels (N > 2 * SMs * 128);
* hub rows whose segments span many 16-slot granules and 128-slot tiles, at every alignment, lopsided and one-sided
  direction splits, duplicate edges;
* block-diagonal batches whose windows differ by orders of magnitude (one per-step scale for all of them);
* training hub rows with more than ATT_MAX_DEG = 1,024 slots (the attention kernels past it: test_attention_boundaries);
* the split-K paths of the training GEMM, and long segments of the training reductions;
* connected components and greedy rounding on graphs larger than one CTA.

Bars: logits as in the parity suite (``assert_logits_close``); node / edge states per row,
|d| <= 1e-3 * max(1, max_j |ref[r, j]|) -- a global scale would be set by the hub alone.
"""
import warnings

import numpy as np
import pytest
import torch

from mpntrackseg_b200 import ops, synth
from mpntrackseg_b200.config import default_graph_model_params
from oracle import mpn_ref, rounding_ref
from test_cuda_parity import assert_logits_close, dev, make_model

pytestmark = pytest.mark.gpu

STATE_TOL = 1e-3
ATT_MAX_DEG = 1024          # csrc/attention.cu: slots per node and direction cached in shared memory per pass
TC_TILE = 128               # nodes per tile of node_tc2_kernel / node_encoder_tc_kernel
S_RESOLVED = 17             # csrc/mp_step_tc.cu: a step above this scale no longer resolves rows of order 1 (status bit 2)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def persistent_sizes():
    """Node counts that give every CTA of the persistent node-side kernels two or three tiles per group."""
    t = 2 * sms() * TC_TILE
    return (t + 1, 3 * sms() * TC_TILE + 77)


def assert_rows_close(got, ref, what, tol=STATE_TOL):
    """Per-row bar: |got - ref| <= tol * max(1, max_j |ref[r, j]|)."""
    got = torch.as_tensor(got).double().cpu().reshape(ref.shape[0], -1)
    ref = torch.as_tensor(ref).double().cpu().reshape(ref.shape[0], -1)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    scale = ref.abs().amax(dim=1, keepdim=True).clamp(min=1.0) if ref.shape[1] else ref.new_ones((ref.shape[0], 1))
    err = (got - ref).abs() / scale
    bad = err > tol
    assert torch.isfinite(got).all(), f'{what}: non-finite values'
    assert not bad.any(), f'{what}: {int(bad.any(dim=1).sum())} rows off, worst {float(err.max()):.3e} at row {int(err.amax(dim=1).argmax())}'


def p64(P):
    return {k: v.double() for k, v in P.items()}


def model_params(steps, agg='sum'):
    mp = default_graph_model_params(steps, steps - 1)
    mp['node_agg_fn'] = agg
    return mp


# ------------------------------------------------------------------ graph generators
def sparse_graph(n, seed, per_node=2, isolated_frac=0.05):
    """Random undirected graph: about 2 * per_node directed edges per node, a few isolated nodes."""
    g = torch.Generator().manual_seed(seed)
    live = torch.nonzero(torch.rand(n, generator=g) >= isolated_frac).view(-1)
    m = per_node * n
    a = live[torch.randint(live.numel(), (m,), generator=g)]
    b = live[torch.randint(live.numel(), (m,), generator=g)]
    keep = a != b
    pairs = torch.stack((a[keep], b[keep]))
    return torch.cat((pairs, pairs.flip(0)), dim=1)


HUB_DEGREES = (1, 15, 16, 17, 31, 32, 33, 47, 48, 49, 127, 128, 129, 383, 384, 385, 1023, 1024, 1025, 4097)


def hub_graph(degrees, offset=0, leaves=None, seed=0, duplicates=0):
    """Undirected hub graph.  Nodes: [0, L) low leaves, then one hub per degree on consecutive rows, then L high
    leaves.  Hub h of degree d has d neighbours among the low leaves and d among the high ones, so its flow_in and its
    flow_out segment both hold d slots.  ``offset`` filler pairs among the low leaves come first in both slot groups and
    shift where every hub segment starts relative to the 16-slot granule and the 128-slot tile.  A run of degree-1 /
    2 / 3 rows follows the hubs, so that one granule holds the tail of one row, whole rows and the head of the next.
    ``duplicates`` hub edges are listed twice."""
    g = torch.Generator().manual_seed(seed)
    degrees = list(degrees) + [1, 2, 3, 1, 1, 2]
    L = leaves or max(max(degrees) + 16, 2 * offset + 64)
    H = len(degrees)
    n = 2 * L + H
    pairs = []
    if offset:
        a = torch.randperm(L, generator=g)[:offset]
        b = torch.randperm(L, generator=g)[:offset]
        b = torch.where(a == b, (b + 1) % L, b)
        pairs.append(torch.stack((a, b)))
    for i, d in enumerate(degrees):
        h = L + i
        lo = torch.randperm(L, generator=g)[:d]
        hi = L + H + torch.randperm(L, generator=g)[:d]
        nb = torch.cat((lo, hi))
        pairs.append(torch.stack((torch.full_like(nb, h), nb)))
    pairs = torch.cat(pairs, dim=1)
    if duplicates:
        pick = torch.randint(pairs.shape[1], (duplicates,), generator=g)
        pairs = torch.cat((pairs, pairs[:, pick]), dim=1)
    ei = torch.cat((pairs, pairs.flip(0)), dim=1)
    return ei[:, torch.randperm(ei.shape[1], generator=g)], n


def max_direction_degree(ei, n):
    out = torch.bincount(ei[0][ei[0] < ei[1]], minlength=n)
    inn = torch.bincount(ei[0][ei[0] > ei[1]], minlength=n)
    return int(torch.maximum(out, inn).max())


def directed_graph(n, m, seed, sign):
    """Only row < col (sign = +1) or only row > col (sign = -1) edges; no pair repeated reversed."""
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(n, (m,), generator=g)
    b = torch.randint(n, (m,), generator=g)
    keep = a != b
    lo, hi = torch.minimum(a, b)[keep], torch.maximum(a, b)[keep]
    return torch.stack((lo, hi)) if sign > 0 else torch.stack((hi, lo))


def lopsided_graph(seed):
    """About 100k flow_out slots (a 20k-slot hub among them) and a single flow_in slot."""
    n = 30000
    out = directed_graph(n, 80000, seed, +1)
    hub = torch.stack((torch.zeros(20000, dtype=torch.int64), torch.arange(1, 20001)))
    one_in = torch.tensor([[n - 1], [5]])
    return torch.cat((out, hub, one_in), dim=1), n


# ------------------------------------------------------------------ step loop on given encoded states
def encoded_states(n, e, seed, x_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 32, generator=g) * 2 * x_scale, torch.rand(e, 16, generator=g) * 2


def run_steps(model, ei, n, x0, e0, steps, engine, debug=False):
    """ops.mp_forward on the caller's edge order: (logits [S, E], node state, edge state in the caller's order)."""
    lay = ops.edge_layout(ei.to(dev()), n)
    e = lay.num_edges
    sedge = lay.slot_edge[:e].long()
    cw, keep = model.core_weights()
    with torch.no_grad():
        lg, xs, es = ops.mp_forward(cw, lay, x0.to(dev()), e0.to(dev())[sedge].contiguous(), steps, 2, want_state=True,
                                    engine=engine, debug=debug)
    e_state = torch.empty_like(es)
    e_state[sedge] = es
    del keep
    return lg.cpu(), xs.cpu(), e_state.cpu()


def oracle_steps(P, mp, ei, x0, e0):
    with torch.no_grad():
        ref = mpn_ref.mp_steps(p64(P), mp, x0.double(), e0.double(), ei, return_state=True)
    return torch.stack([t.view(-1) for t in ref['classified_edges']]), ref['node_state'], ref['edge_state']


def check_against(ref, got, what):
    lg, xs, es = got
    assert_logits_close(lg.numpy(), ref[0].numpy(), what)
    assert_rows_close(xs, ref[1], what + ' node state')
    assert_rows_close(es, ref[2], what + ' edge state')


# ================================================================== 1. persistent loops
@pytest.mark.parametrize('which', [0, 1])
@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_step_loop_beyond_one_tile_per_node_kernel_group(agg, which):
    """More than one 128-node tile per CTA group in node_tc2_kernel: the second and third tile reuse the barrier
    parities and TMEM of the first.  Both engines against the fp64 oracle, 3 steps."""
    n = persistent_sizes()[which]
    assert n > 2 * sms() * TC_TILE and n % TC_TILE != 0
    mp = model_params(3, agg)
    P = synth.make_params(mp, seed=11, gain=1.25, core_only=True)
    ei = sparse_graph(n, seed=which)
    assert int(torch.bincount(ei[0], minlength=n).eq(0).sum()) > 0, 'the case must hold isolated nodes'
    x0, e0 = encoded_states(n, ei.shape[1], seed=3 + which)
    ref = oracle_steps(P, mp, ei, x0, e0)
    for engine in ('tc', 'fp32'):
        check_against(ref, run_steps(make_model(mp, P, engine), ei, n, x0, e0, 3, engine), f'{agg} n={n} {engine}')


# ================================================================== 2. high degrees and segment alignment
def _hub_contract(mp, P, ei, n, what, must_not_raise):
    """'tc' meets the bar or raises OverflowError (must_not_raise: it meets the bar); 'fp32' and 'auto' meet it;
    two runs are bit-identical."""
    x0, e0 = encoded_states(n, ei.shape[1], seed=17)
    ref = oracle_steps(P, mp, ei, x0, e0)
    model = make_model(mp, P)
    for engine in ('fp32', 'auto'):
        check_against(ref, run_steps(model, ei, n, x0, e0, 3, engine), f'{what} {engine}')
    try:
        got = run_steps(model, ei, n, x0, e0, 3, 'tc')
    except OverflowError:
        assert not must_not_raise, f'{what}: tc raised'
        return None
    check_against(ref, got, f'{what} tc')
    again = run_steps(model, ei, n, x0, e0, 3, 'tc')
    assert all(torch.equal(a, b) for a, b in zip(got, again)), f'{what}: two runs differ'
    return got


@pytest.mark.parametrize('offset', [0, 1, 15, 127])
@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
def test_hub_segments_at_every_granule_and_tile_alignment(agg, offset):
    ei, n = hub_graph(HUB_DEGREES, offset=offset, seed=offset, duplicates=50)
    assert max_direction_degree(ei, n) > ATT_MAX_DEG
    mp = model_params(3, agg)
    P = synth.make_params(mp, seed=5, gain=1.25, core_only=True)
    _hub_contract(mp, P, ei, n, f'hubs {agg} o={offset}', must_not_raise=agg != 'sum')
    if agg == 'sum':                                       # moderate degrees: sum aggregation stays on the tensor cores
        small, n2 = hub_graph([d for d in HUB_DEGREES if d <= 64], offset=offset, seed=offset)
        assert 48 < max_direction_degree(small, n2) <= 64
        _hub_contract(mp, P, small, n2, f'hubs<=64 sum o={offset}', must_not_raise=True)


@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
@pytest.mark.parametrize('kind', ['out_only', 'in_only', 'lopsided'])
def test_one_sided_and_lopsided_direction_splits(kind, agg):
    if kind == 'lopsided':
        ei, n = lopsided_graph(seed=2)
        assert int((ei[0] > ei[1]).sum()) == 1 and int((ei[0] < ei[1]).sum()) >= 95000
    else:
        n = 20000
        ei = directed_graph(n, 60000, seed=3, sign=+1 if kind == 'out_only' else -1)
    mp = model_params(3, agg)
    P = synth.make_params(mp, seed=6, gain=1.25, core_only=True)
    _hub_contract(mp, P, ei, n, f'{kind} {agg}', must_not_raise=agg != 'sum' or kind != 'lopsided')


@pytest.mark.parametrize('engine', ['tc', 'fp32'])
def test_hub_forward_is_deterministic_and_order_invariant(engine):
    """A permutation that keeps every row's relative edge order permutes the logits bit for bit; a random
    permutation still meets the bar."""
    ei, n = hub_graph(HUB_DEGREES[:-1], offset=15, seed=4, duplicates=20)
    mp = model_params(3, 'mean')
    P = synth.make_params(mp, seed=7, gain=1.25, core_only=True)
    model = make_model(mp, P)
    x0, e0 = encoded_states(n, ei.shape[1], seed=8)
    base = run_steps(model, ei, n, x0, e0, 3, engine)
    g = torch.Generator().manual_seed(9)
    row_key = torch.randperm(n, generator=g)[ei[0]]
    keep_rows = torch.argsort(row_key, stable=True)                         # rows shuffled, each row's order kept
    rand = torch.randperm(ei.shape[1], generator=g)
    for perm, exact in ((keep_rows, True), (rand, False)):
        lg, xs, es = run_steps(model, ei[:, perm], n, x0, e0[perm], 3, engine)
        if exact:
            assert torch.equal(lg, base[0][:, perm]) and torch.equal(xs, base[1]) and torch.equal(es, base[2][perm])
        else:
            assert_logits_close(lg.numpy(), base[0][:, perm].numpy(), f'random permutation {engine}')
            assert_rows_close(xs, base[1], 'random permutation node state')


def test_edge_and_node_model_operators_on_hub_graphs():
    """EdgeModel / TimeAwareNodeModel / MetaLayer as standalone operators (fp32 kernels) on the hub graph."""
    ei, n = hub_graph(HUB_DEGREES, offset=1, seed=12, duplicates=10)
    assert max_direction_degree(ei, n) > ATT_MAX_DEG
    for agg in ('sum', 'mean', 'max'):
        mp = model_params(3, agg)
        P = synth.make_params(mp, seed=13, gain=1.25, core_only=True)
        model = make_model(mp, P)
        g = torch.Generator().manual_seed(14)
        x = torch.rand(n, 64, generator=g) * 2
        ea = torch.rand(ei.shape[1], 32, generator=g) * 2
        with torch.no_grad():
            e_ref = mpn_ref.edge_update(p64(P), x.double(), ei, ea.double())
            x_ref = mpn_ref.node_update(p64(P), x.double(), ei, e_ref, agg)
            e_new = model.MPNet.edge_model(x.to(dev()), ei.to(dev()), ea.to(dev()))
            x_new = model.MPNet.node_model(x.to(dev()), ei.to(dev()), e_ref.float().to(dev()))
            x_step, e_step = model.MPNet(x.to(dev()), ei.to(dev()), ea.to(dev()))
        assert_rows_close(e_new, e_ref, f'edge_model {agg}')
        assert_rows_close(x_new, x_ref, f'node_model {agg}')
        assert_rows_close(e_step, e_ref, f'MetaLayer edge {agg}')
        assert_rows_close(x_step, x_ref, f'MetaLayer node {agg}')
    # an id >= N, a negative id, a self-loop or an edge_attr of another length raises before anything gathers by them
    xd, ead, ed = x.to(dev()), ea.to(dev()), e_ref.float().to(dev())
    for col in (n, -1, int(ei[0, 0])):
        bad = ei.clone()
        bad[1, 0] = col
        bad = bad.to(dev())
        for call in (lambda: model.MPNet.edge_model(xd, bad, ead), lambda: model.MPNet(xd, bad, ead),
                     lambda: model.MPNet.node_model(xd, bad, ed)):
            with torch.no_grad(), pytest.raises(ValueError, match='self-loops or out of range'):
                call()
    ei_d = ei.to(dev())
    for call in (lambda: model.MPNet.edge_model(xd, ei_d, ead[1:]), lambda: model.MPNet(xd, ei_d, ead[1:]),
                 lambda: model.MPNet.node_model(xd, ei_d, ed[1:])):
        with torch.no_grad(), pytest.raises(ValueError, match='rows for'):
            call()
    torch.cuda.synchronize()


# ================================================================== 3. mixed-magnitude batches
def _mixed_batch(seed=0):
    """Four small KNN windows as one block-diagonal batch, encoded by the oracle; window 1 is the loud one."""
    from oracle import graph_ref
    from mpntrackseg_b200.config import default_dataset_params
    mp = default_graph_model_params(12, 11)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    blocks = []
    for i in range(4):
        w = synth.make_window(T=15, D=100, k=50, seed=200 + seed + i, node_feats='pooled')
        gr = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds)
        with torch.no_grad():
            x0, e0 = mpn_ref.encode(P, w.x, gr['edge_attr'])
        blocks.append((gr['edge_index'], x0, e0))
    return mp, P, blocks


def _batch(blocks, factors):
    eis, xs, es, off = [], [], [], 0
    for (ei, x0, e0), f in zip(blocks, factors):
        eis.append(ei + off)
        xs.append(x0 * f)
        es.append(e0)
        off += x0.shape[0]
    return torch.cat(eis, dim=1), off, torch.cat(xs), torch.cat(es)


def test_windows_of_very_different_magnitude_share_one_batch():
    """One per-step scale serves the whole batch.  A quiet window batched with a loud one (its encoded x0 x 2^k, k as
    large as the fp16 image of the first step's x_lat allows) must still meet the bar against the oracle run on that
    window alone -- or the forward is flagged: engine='tc' raises and 'auto' reruns on the fp32 kernels."""
    mp, P, blocks = _mixed_batch()
    k = int(np.floor(np.log2(60000.0 / float(blocks[1][1].abs().max()))))
    factors = [1.0, 2.0 ** k, 1.0, 1.0]
    ei, n, x0, e0 = _batch(blocks, factors)
    assert float(x0.abs().max()) < 65504.0
    refs = [oracle_steps(P, mp, b[0], b[1] * f, b[2]) for b, f in zip(blocks, factors)]
    model = make_model(mp, P)

    def check(got, what, loud=None):
        lg, xs, es = got
        eo, no = 0, 0
        for i, (b, ref) in enumerate(zip(blocks, refs)):
            ne, nn = b[0].shape[1], b[1].shape[0]
            part = (lg[:, eo:eo + ne], xs[no:no + nn], es[eo:eo + ne])
            if i == loud:          # states ~1e9 whose logits cancel: beyond fp32 arithmetic, whichever kernels run it
                assert all(torch.isfinite(t).all() for t in part), f'{what} window {i}'
            else:
                check_against(ref, part, f'{what} window {i}')
            eo, no = eo + ne, no + nn

    flagged = False
    try:
        got = run_steps(model, ei, n, x0, e0, 12, 'tc', debug=True)
    except OverflowError:
        flagged = True
    # the loud window doubles its state about once per step: from the fp16 limit of x0 the schedule climbs to s_t = 22
    assert max(ops.LAST_TC_SCHEDULE['sched'][1:13]) > S_RESOLVED, ops.LAST_TC_SCHEDULE['sched']
    if not flagged:
        check(got, 'tc', loud=1)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter('always')
        check(run_steps(model, ei, n, x0, e0, 12, 'auto'), 'auto', loud=1)
    assert flagged == any('fp16 range' in str(w.message) for w in caught), 'auto reruns on fp32 exactly when tc is flagged'
    # the same windows at their own magnitude stay on the tensor cores and meet the bar
    refs = [oracle_steps(P, mp, *b) for b in blocks]
    ei, n, x0, e0 = _batch(blocks, [1.0] * 4)
    check(run_steps(model, ei, n, x0, e0, 12, 'tc', debug=True), 'tc unscaled')
    assert 0 < max(ops.LAST_TC_SCHEDULE['sched'][1:13]) <= S_RESOLVED


# ================================================================== 5. training
def test_training_gradients_on_a_hub_graph():
    """CoreTrainer on hub rows up to 1,025 slots per direction, sum aggregation, 3 steps: gradients against fp64
    autograd through the oracle within 2e-3 of each tensor's maximum, bit-identical on a rerun."""
    from mpntrackseg_b200.training import CoreTrainer
    ei, n = hub_graph([1, 15, 17, 33, 129, 385, 1023, 1025], offset=15, seed=21, leaves=1100)
    assert max_direction_degree(ei, n) > ATT_MAX_DEG
    mp = model_params(3, 'sum')
    P = synth.make_params(mp, seed=22, gain=1.0, core_only=True)
    g = torch.Generator().manual_seed(23)
    x = torch.rand(n, 2048, generator=g)
    ea = torch.rand(ei.shape[1], 6, generator=g)
    labels = (torch.rand(ei.shape[1], generator=g) < 0.3).float()
    Pg = {k: v.double().requires_grad_(True) for k, v in P.items()}
    out = mpn_ref.mpn_forward(Pg, mp, x.double(), ei, ea.double())
    ref_loss = mpn_ref.weighted_bce_loss(out['classified_edges'], labels.double(), tracking_weight=0.8)
    ref_loss.backward()
    model = make_model(mp, P, 'fp32')
    tr = CoreTrainer(model)

    class _D:
        pass
    data = _D()
    data.x, data.edge_index, data.edge_attr = x.to(dev()), ei.to(dev()), ea.to(dev())
    loss = tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert abs(float(loss) - float(ref_loss)) <= 2e-4 * max(1.0, abs(float(ref_loss)))
    for k, p in Pg.items():
        scale = float(p.grad.abs().max()) + 1e-30
        err = float((tr.g[k].cpu().double() - p.grad).abs().max()) / scale
        assert err <= 2e-3, (k, err)
    g1 = tr.grad.clone()
    tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert torch.equal(g1, tr.grad)


GEMM_TOL = 1e-5             # of (|A| |B|)_ij (+ |bias| + |C|): fp32 accumulation sits orders of magnitude below


def _splitk_cap_k():
    """Smallest K at which mpn_gemm's split count reaches its cap of 256 for a single output tile."""
    return 256 * 512 + 16 * 7 + 1


def _gemm_bar(A, B, bias, c0):
    bar = A.abs() @ B.abs()
    if bias is not None:
        bar = bar + bias.abs()
    if c0 is not None:
        bar = bar + c0.abs()
    return GEMM_TOL * bar + 1e-30


def _gemm_case(m, n, k, ta, tb, opt, g, positive=False):
    """Operands as column slices of wider buffers (leading dimension != width)."""
    rnd = (lambda *s: torch.rand(*s, generator=g)) if positive else (lambda *s: torch.randn(*s, generator=g))
    A = rnd(m, k).double()
    B = rnd(k, n).double()
    a_buf = rnd(*((k, m + 5) if ta else (m, k + 5)))
    b_buf = rnd(*((n, k + 3) if tb else (k, n + 3)))
    a_buf[:, 2:2 + (m if ta else k)] = (A.t() if ta else A).float()
    b_buf[:, 1:1 + (k if tb else n)] = (B.t() if tb else B).float()
    a_dev = a_buf.to(dev())[:, 2:2 + (m if ta else k)]
    b_dev = b_buf.to(dev())[:, 1:1 + (k if tb else n)]
    mask = None
    if 'mask' in opt:
        mk = rnd(*((k, m) if ta else (m, k)))
        mask = mk.to(dev())
        A = A * ((mk.t() if ta else mk) > 0).double()
    bias = rnd(n).double() if 'bias' in opt else None
    c0 = rnd(m, n).double() if 'accumulate' in opt else None
    return A.float().double(), B.float().double(), a_dev, b_dev, mask, bias, c0


def _gemm_ref(A, B, bias, relu, c0):
    ref = A @ B
    if bias is not None:
        ref = ref + bias
    if c0 is not None:
        ref = ref + c0
    return ref.clamp(min=0) if relu else ref


def test_training_gemm_against_fp64_across_split_k_edges():
    from mpntrackseg_b200 import training
    g = torch.Generator().manual_seed(31)
    cap_k = _splitk_cap_k()
    ks = [0, 1, 2047, 2048, 2049, 2048 + 16 * 5 + 1, cap_k]
    opts = [(), ('mask',), ('bias', 'relu'), ('accumulate',), ('mask', 'bias', 'relu', 'accumulate')]
    shapes = [(1, 1), (63, 65), (64, 64), (65, 63), (1, 64), (65, 1)]
    i = 0
    for k in ks:
        for m, n in (shapes if k != cap_k else [(1, 1), (65, 63)]):
            for ta in (False, True):
                for tb in (False, True):
                    opt = opts[i % len(opts)]
                    i += 1
                    A, B, a, b, mask, bias, c0 = _gemm_case(m, n, k, ta, tb, opt, g)
                    out = c0.float().to(dev()) if c0 is not None else None
                    got = training.gemm(a, b, ta=ta, tb=tb, bias=None if bias is None else bias.float().to(dev()),
                                        relu='relu' in opt, mask=mask, out=out, accumulate=c0 is not None)
                    ref = _gemm_ref(A, B, bias, 'relu' in opt, c0)
                    err = (got.cpu().double() - ref).abs() / _gemm_bar(A, B, bias, c0)
                    assert float(err.max()) <= 1.0, (m, n, k, ta, tb, opt, float(err.max()))
    # the cap is really reached: 4 * SMs / 1 tile and ceil(K / 512) both exceed 256
    assert 4 * sms() > 256 and -(-cap_k // 512) > 256


def test_gemm_bar_rejects_a_dropped_k_slice():
    """The bar above is tight enough to see one missing 16-wide K step at every contraction length tested."""
    from mpntrackseg_b200 import training
    g = torch.Generator().manual_seed(32)
    for k in (16, 2047, 2049, 2048 + 16 * 5 + 1, _splitk_cap_k()):
        A, B, a, b, _, _, _ = _gemm_case(3, 2, k, False, True, (), g, positive=True)
        got = training.gemm(a, b, tb=True).cpu().double()
        bar = _gemm_bar(A, B, None, None)
        assert float(((got - A @ B).abs() / bar).max()) <= 1.0
        s = (k // 2) // 16 * 16
        dropped = A @ B - A[:, s:s + 16] @ B[s:s + 16]
        assert float(((got - dropped).abs() / bar).min()) > 1.0, k


def test_colsum_segment_sum_and_gather_cols_against_fp64():
    from mpntrackseg_b200 import training
    g = torch.Generator().manual_seed(33)
    for m in (0, 1, 255, 257, 40000):
        for n in (1, 63, 64, 65):
            buf = torch.randn(m, n + 7, generator=g)
            mk = torch.randn(m, n, generator=g)
            a = buf[:, 3:3 + n]
            for use_mask, acc in ((False, False), (True, True)):
                out0 = torch.randn(n, generator=g)
                out = out0.clone().to(dev())
                training.colsum(buf.to(dev())[:, 3:3 + n], mask=mk.to(dev()) if use_mask else None, out=out, accumulate=acc)
                av = a.double() * ((mk > 0).double() if use_mask else 1.0)
                ref = av.sum(0) + (out0.double() if acc else 0.0)
                bar = GEMM_TOL * (av.abs().sum(0) + (out0.abs().double() if acc else 0.0)) + 1e-30
                assert float(((out.cpu().double() - ref).abs() / bar).max()) <= 1.0, (m, n, use_mask, acc)
    # long permuted segments: one node owns 30,000 slots, others 0 / 1 / 1,025
    lens = torch.tensor([0, 1, 30000, 1025, 0, 7])
    e = int(lens.sum())
    ptr = torch.zeros(lens.numel() + 1, dtype=torch.int32)
    ptr[1:] = torch.cumsum(lens, 0).to(torch.int32)
    perm = torch.randperm(e, generator=g).to(torch.int32)
    inp = torch.randn(e, 40, generator=g)
    for acc in (False, True):
        out0 = torch.randn(lens.numel(), 50, generator=g)
        out = out0.clone().to(dev())
        ops.segment_sum(inp.to(dev()), 4, 33, ptr.to(dev()), perm.to(dev()), out, 9, accumulate=acc)
        ref = out0.double().clone()
        seg = torch.repeat_interleave(torch.arange(lens.numel()), lens)
        vals = inp.double()[perm.long(), 4:37]
        summed = torch.zeros(lens.numel(), 33, dtype=torch.float64).index_add_(0, seg, vals)
        ref[:, 9:42] = summed + (ref[:, 9:42] if acc else 0.0)
        absr = torch.zeros_like(summed).index_add_(0, seg, vals.abs())
        bar = GEMM_TOL * (absr + (out0.double()[:, 9:42].abs() if acc else 0.0)) + 1e-30
        got = out.cpu().double()
        assert float(((got[:, 9:42] - ref[:, 9:42]).abs() / bar).max()) <= 1.0
        assert torch.equal(got[:, :9], out0.double()[:, :9]) and torch.equal(got[:, 42:], out0.double()[:, 42:])
    idx = torch.randint(500, (7000,), generator=g).to(torch.int32)
    src = torch.randn(500, 37, generator=g)
    out = torch.zeros(7000, 45).to(dev())
    training.gather_cols(src.to(dev()), idx.to(dev()), out, 5)
    assert torch.equal(out.cpu()[:, 5:42], src[idx.long()]) and not out.cpu()[:, :5].any() and not out.cpu()[:, 42:].any()


# ================================================================== 6. rounding beyond one CTA
def _scipy_components(ei, vals, n):
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    m = vals == 1
    a = ei[:, m]
    return connected_components(csr_matrix((np.ones(a.shape[1], dtype=int), (a[0], a[1])), shape=(n, n)),
                                directed=False, return_labels=True)


def test_connected_components_of_long_identity_chains_stars_and_forests():
    """Tens of thousands of nodes, more than one CTA of 1,024 threads: identity chains 400 frames long (sequence
    order: node = frame * tracks + track), fed forward, reversed and shuffled; a star; a random forest."""
    g = torch.Generator().manual_seed(41)
    tracks, frames = 60, 400
    node = torch.arange(frames * tracks).view(frames, tracks)
    chain = torch.stack((node[:-1].reshape(-1), node[1:].reshape(-1)))
    n_chain = frames * tracks
    star_c = n_chain
    star = torch.stack((torch.full((3000,), star_c), torch.arange(star_c + 1, star_c + 3001)))
    f0 = star_c + 3001
    nf = 8000
    parents = torch.randint(0, nf, (nf,), generator=g) % torch.arange(nf).clamp(min=1)   # parent < child for child >= 1
    forest = torch.stack((f0 + parents[1:], f0 + torch.arange(1, nf)))
    forest = forest[:, torch.rand(nf - 1, generator=g) < 0.9]
    n = f0 + nf + 100                                                             # trailing isolated nodes
    ei = torch.cat((chain, star, forest), dim=1)
    assert n > 20000 and ei.shape[1] > 1024
    vals = torch.ones(ei.shape[1])
    vals[torch.rand(ei.shape[1], generator=g) < 0.02] = 0.0                      # some edges switched off
    ref_n, ref_l = _scipy_components(ei.numpy(), vals.numpy(), n)
    for order in ('forward', 'reversed', 'random'):
        perm = {'forward': torch.arange(ei.shape[1]), 'reversed': torch.arange(ei.shape[1]).flip(0),
                'random': torch.randperm(ei.shape[1], generator=g)}[order]
        e = ei[:, perm]
        if order == 'random':
            e = torch.where(torch.rand(e.shape[1], generator=g) < 0.5, e, e.flip(0))   # either endpoint first
        labels, ncomp = ops.connected_components(e.to(dev()), vals[perm].to(dev()), n)
        assert ncomp == ref_n, order
        assert np.array_equal(labels.cpu().numpy(), ref_l), order


def test_greedy_projection_on_a_hub_with_exact_ties():
    """A hub with thousands of active edges in both directions, predictions with many exact ties: rounding and
    constraint statistics bit-exact against the oracle."""
    g = torch.Generator().manual_seed(42)
    n = 12000
    hub = 6000
    out_nb = hub + 1 + torch.randperm(n - hub - 1, generator=g)[:3000]
    in_nb = torch.randperm(hub, generator=g)[:2500]
    rest = directed_graph(n, 20000, seed=43, sign=+1)
    ei = torch.cat((torch.stack((torch.full_like(out_nb, hub), out_nb)), torch.stack((in_nb, torch.full_like(in_nb, hub))),
                    rest), dim=1)
    ei = torch.unique(ei, dim=1)
    ei = ei[:, torch.randperm(ei.shape[1], generator=g)]
    preds = torch.tensor([0.2, 0.6, 0.75, 0.9])[torch.randint(4, (ei.shape[1],), generator=g)]
    assert int(((ei[0] == hub) & (preds > 0.5)).sum()) > 1024 and int(((ei[1] == hub) & (preds > 0.5)).sum()) > 1024
    ref_r, ref_rate = rounding_ref.greedy_project(ei.numpy(), preds.numpy(), n)
    got_r, rate = ops.greedy_project(ei.to(dev()), preds.to(dev()), n)
    assert np.array_equal(got_r.cpu().numpy(), ref_r) and rate == ref_rate
    for undirected in (False, True):
        e2 = torch.cat((ei, ei.flip(0)), dim=1) if undirected else ei
        v2 = torch.from_numpy(ref_r).repeat(2 if undirected else 1)
        r_rate, r_in, r_out = rounding_ref.constr_satisfaction_rate(e2.numpy(), n, v2.numpy(), undirected_edges=undirected)
        c_rate, c_in, c_out = ops.constr_satisfaction(e2.to(dev()), v2.to(dev()), n, undirected_edges=undirected)
        assert c_rate == r_rate and np.array_equal(c_in.cpu().numpy(), r_in) and np.array_equal(c_out.cpu().numpy(), r_out)
