"""The node-feature pool that build_graph_batch starts on a side stream and forward_batch joins: the same logits, bit
for bit, as pooling and encoding the maps in order on one stream; the one-launch pool of many windows equals the
per-window pool."""
import gc

import pytest
import torch

from mpntrackseg_b200 import ops, synth
from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params

pytestmark = pytest.mark.gpu


def dev():
    return torch.device('cuda:0')


def make_model():
    from mpntrackseg_b200.models.mpn import MOTMPNet
    mp = default_graph_model_params(5, 4)
    model = MOTMPNet(mp).to(dev()).eval()
    model.load_state_dict(synth.make_params(mp, seed=4, gain=2.0, core_only=True), strict=False)
    return model


DS = default_dataset_params(top_k_nns=6, frames_per_graph=7)


def windows(shapes, seed=0):
    """Detection tables of synthetic windows with [n, 2048, 8, 4] maps on the GPU; (T, D) per window."""
    out = []
    for i, (t, d) in enumerate(shapes):
        w = synth.make_window(T=t, D=d, k=6, seed=seed + i, node_feats='full')
        out.append(dict(synth.det_columns(w), reid=w.reid, x=w.x.to(dev())))
    return out


def reference_logits(model, wins):
    """Pool every window with ops.avgpool, encode once, forward the encoded batch: the path without a side stream."""
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    batch = build_window_graphs([dict(w, x=w['x'].clone()) for w in wins], DS, fps=30.0)
    with torch.no_grad():
        batch.xs = model.encode_pooled(torch.cat([ops.avgpool(w['x']) for w in wins]))
        return model.forward_batch(batch, encoded=True).logits


RAGGED = {1: [(5, 7)], 16: [(3 + i % 5, 4 + (7 * i) % 9) for i in range(15)] + [(1, 1)]}


@pytest.mark.parametrize('count', sorted(RAGGED))
def test_side_stream_pool_matches_the_in_order_path(count):
    """1 and 16 windows of ragged sizes, the last of the 16 a window of one node."""
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    model = make_model()
    wins = windows(RAGGED[count], seed=10 * count)
    batch = build_window_graphs(wins, DS, fps=30.0)
    assert batch.pooled_xs() is not None
    with torch.no_grad():
        got = model.forward_batch(batch).logits
    assert torch.equal(got, reference_logits(model, wins))


def test_maps_dropped_by_the_caller_after_the_build():
    from mpntrackseg_b200.data.mot_graph import build_graph_batch
    model = make_model()
    wins = windows(RAGGED[16], seed=3)
    exp = reference_logits(model, wins)
    node_ptr = [0]
    for w in wins:
        node_ptr.append(node_ptr[-1] + w['x'].shape[0])
    table = {k: torch.cat([torch.as_tensor(w[k]) for w in wins]).to(dev()) for k in
             ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y', 'reid')}
    table['x'] = [w['x'].clone() for w in wins]
    batch = build_graph_batch(table, node_ptr, DS, fps=30.0, device=dev())
    del table, wins
    gc.collect()
    junk = [torch.full((n, 2048, 8, 4), float('nan'), device=dev()) for n in (8, 30, 60)]     # reuse freed memory
    with torch.no_grad():
        got = model.forward_batch(batch).logits
    del junk
    assert torch.equal(got, exp)


def test_replaced_xs_ignores_the_stale_pool():
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    model = make_model()
    wins = windows(RAGGED[16], seed=5)
    other = [torch.rand_like(w['x']) for w in wins]
    batch = build_window_graphs(wins, DS, fps=30.0)
    batch.xs = other
    assert batch.pooled_xs() is None
    with torch.no_grad():
        got = model.forward_batch(batch).logits
    assert torch.equal(got, reference_logits(model, [dict(w, x=o) for w, o in zip(wins, other)]))


def test_pooled_features_take_the_in_order_path():
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    model = make_model()
    wins = windows(RAGGED[16][:4], seed=7)
    batch = build_window_graphs([dict(w, x=ops.avgpool(w['x'])) for w in wins], DS, fps=30.0)
    assert batch._pool is None
    with torch.no_grad():
        got = model.forward_batch(batch).logits
    assert torch.equal(got, reference_logits(model, wins))


def test_host_maps_start_no_pool():
    from mpntrackseg_b200.data.mot_graph import build_graph_batch
    wins = windows(RAGGED[16][:2], seed=8)
    table = {k: torch.cat([torch.as_tensor(w[k]) for w in wins]).to(dev()) for k in
             ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y', 'reid')}
    table['x'] = [w['x'].cpu() for w in wins]
    n = [w['x'].shape[0] for w in wins]
    assert build_graph_batch(table, [0, n[0], n[0] + n[1]], DS, fps=30.0, device=dev())._pool is None


@pytest.mark.parametrize('hw', (1, 4, 32))
def test_one_launch_pool_equals_the_per_window_pool(hw):
    """Ragged windows, one of no rows, more windows than one launch's table holds, and an unaligned view (the scalar
    kernel) among them."""
    g = torch.Generator(device=dev()).manual_seed(hw)
    c = 24
    sizes = [(7 * i) % 23 for i in range(70)] + [300]
    sizes[3] = 5
    xs = [torch.randn((n, c, hw, 1), generator=g, device=dev()) for n in sizes]
    buf = torch.randn(5 * c * hw + 1, generator=g, device=dev())
    xs[3] = buf[1:].view(5, c, hw, 1)
    assert hw == 1 or xs[3].data_ptr() % 16 != 0
    got = ops.avgpool_windows(xs)
    exp = torch.cat([ops.avgpool(x) for x in xs])
    assert torch.equal(got, exp)
    big = torch.full((sum(sizes) + 4, c), float('nan'), device=dev())
    ops.avgpool_windows(xs, out=big[2:-2])
    assert torch.equal(big[2:-2], exp) and big[:2].isnan().all() and big[-2:].isnan().all()
