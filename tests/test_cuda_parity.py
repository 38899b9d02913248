"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden
outputs of the reference.  Integer / index results must be bit-exact; edge logits within
the tolerance BASELINE.json states (1e-3 absolute on probabilities, decisions identical
outside +-1e-3 of 0.5; on raw logits 1e-3 * max(1, |logit|), SURVEY.md H2)."""
import numpy as np
import pytest
import torch

from cases import CASES, load_big_case, load_case
from mpntrackseg_b200 import synth
from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
from oracle import graph_ref, mpn_ref

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3


def dev():
    return torch.device('cuda:0')


def assert_logits_close(got, exp, what=''):
    got, exp = np.asarray(got, dtype=np.float64), np.asarray(exp, dtype=np.float64)
    assert got.shape == exp.shape, (got.shape, exp.shape)
    tol = 1e-3 * np.maximum(1.0, np.abs(exp))
    bad = np.abs(got - exp) > tol
    assert not bad.any(), f'{what}: {bad.sum()} logits off, max err {np.abs(got - exp).max():.3e}'
    pg, pe = 1 / (1 + np.exp(-got)), 1 / (1 + np.exp(-exp))
    assert np.abs(pg - pe).max() <= PROB_TOL, f'{what}: max |dp| {np.abs(pg - pe).max():.3e}'
    decisive = np.abs(pe - 0.5) > PROB_TOL
    assert ((pg > 0.5) == (pe > 0.5))[decisive].all(), f'{what}: binarised decisions differ'


ENGINES = ('tc', 'fp32')


def make_model(mp, P, engine=None):
    from mpntrackseg_b200.models.mpn import MOTMPNet
    model = MOTMPNet(mp).to(dev()).eval()
    model.engine = engine
    model.load_state_dict(P, strict=len(P) == len(model.state_dict()))   # core-only dicts leave the mask branch as is
    return model


class Data:
    pass


# ------------------------------------------------------------------ graph construction
@pytest.mark.parametrize('name', list(CASES))
def test_drop_in_graph_utils_match_oracle(name):
    from mpntrackseg_b200.utils.graph import compute_edge_feats_dict, get_knn_mask, get_time_valid_conn_ixs
    c = load_case(name)
    win, ds = c['win'], c['ds']
    mfd = c['max_frame_dist']
    pairs = get_time_valid_conn_ixs(win.frame, mfd, use_cuda=True)
    ref_pairs = graph_ref.time_valid_pairs(win.frame, mfd)
    assert pairs.device.type == 'cpu' and pairs.dtype == torch.int64
    assert torch.equal(pairs, ref_pairs)
    ref_d = graph_ref.pair_reid_dist(win.reid, ref_pairs)
    for recip in (True, False):
        keep = get_knn_mask(ref_d, ref_pairs, win.N, ds['top_k_nns'], use_cuda=True, reciprocal_k_nns=recip,
                            symmetric_edges=False)
        ref_keep = graph_ref.knn_keep_mask(ref_d, ref_pairs, win.N, ds['top_k_nns'], recip, symmetric_edges=False)
        assert keep.dtype == torch.bool and torch.equal(keep.cpu(), ref_keep)
    feats = compute_edge_feats_dict(ref_pairs, synth.det_columns(win), win.fps, use_cuda=True)
    ref_f = graph_ref.edge_geometry(ref_pairs, synth.det_columns(win), win.fps)
    assert set(feats) == set(ref_f)
    for k in ref_f:
        np.testing.assert_allclose(feats[k].cpu().numpy(), ref_f[k].numpy(), rtol=2e-6, atol=2e-7, err_msg=k)
    # differences and quotients are IEEE-exact; only logf may differ in the last ulp
    for k in ('secs_time_dists', 'norm_feet_x_dists', 'norm_feet_y_dists'):
        assert torch.equal(feats[k].cpu(), ref_f[k]), k


@pytest.mark.parametrize('name', list(CASES))
def test_motgraph_matches_reference_golden(name):
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    c = load_case(name)
    win, gold = c['win'], c['gold']
    g = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, c['ds'],
                 inference_mode=False, max_frame_dist=c['max_frame_dist']).construct_graph_object()
    assert g.edge_index.dtype == torch.int64 and g.edge_index.is_cuda
    assert np.array_equal(g.edge_index.cpu().numpy(), gold['edge_index'].astype(np.int64)), 'KNN edge set'
    np.testing.assert_allclose(g.edge_attr.cpu().numpy(), gold['edge_attr'], rtol=2e-6, atol=1e-6)
    assert g.num_nodes == win.N and g.num_edges == gold['edge_index'].shape[1]


def test_pair_dist_close_to_torch_formula():
    from mpntrackseg_b200 import ops
    win = synth.make_window(T=6, D=20, k=10, seed=9)
    pairs = graph_ref.time_valid_pairs(win.frame)
    d = ops.pair_reid_dist(win.reid.to(dev()), pairs.to(dev())).cpu()
    ref = graph_ref.pair_reid_dist(win.reid, pairs)
    np.testing.assert_allclose(d.numpy(), ref.numpy(), rtol=3e-6)


def test_knn_mask_symmetric_edges_and_ties():
    """Inference-time call (both directions listed, symmetric_edges=True) incl. k >= degree,
    exact ties (stable by index) and a batch of windows via node_graph_ptr."""
    from mpntrackseg_b200 import ops
    c = load_case('tracker_window')
    gold, ds = c['gold'], c['ds']
    win = c['win']
    ei = torch.from_numpy(gold['full_edge_index'].astype(np.int64))
    d = torch.from_numpy(gold['full_dists'])
    for k in (1, 3, 7, 40, 10 ** 6):
        for recip in (True, False):
            keep = ops.knn_mask(d.to(dev()), ei.to(dev()), win.N, k, recip, True).cpu()
            ref = graph_ref.knn_keep_mask(d, ei, win.N, k, recip, True)
            assert torch.equal(keep, ref), (k, recip)
    # quantised distances -> many exact ties at the k boundary
    dq = (d * 2).round() / 2
    for k in (2, 5):
        keep = ops.knn_mask(dq.to(dev()), ei.to(dev()), win.N, k, True, True).cpu()
        assert torch.equal(keep, graph_ref.knn_keep_mask(dq, ei, win.N, k, True, True)), k


def test_time_valid_pairs_batched_windows():
    from mpntrackseg_b200 import ops
    frames = [torch.arange(1, 5).repeat_interleave(3), torch.arange(10, 13).repeat_interleave(4),
              torch.tensor([7, 7, 8])]
    ptr = torch.tensor([0, 12, 24, 27])
    got = ops.time_valid_pairs(torch.cat(frames).to(dev()), 2, ptr.to(dev())).cpu()
    exp = torch.cat([graph_ref.time_valid_pairs(f, 2) + int(o) for f, o in zip(frames, ptr[:-1])], dim=1)
    assert torch.equal(got, exp)


def test_tracker_window_prune_and_predict():
    """mpn_tracker.py:107-135 glue on the CUDA path against the reference's golden output."""
    from mpntrackseg_b200.data.mot_graph import Graph, MOTGraph
    from mpntrackseg_b200.utils.graph import get_knn_mask
    c = load_case('tracker_window')
    win, gold, ds = c['win'], c['gold'], c['ds']
    full = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, ds, inference_mode=True,
                    max_frame_dist=ds['frames_per_graph'] - 1).construct_graph_object()
    assert np.array_equal(full.edge_index.cpu().numpy(), gold['full_edge_index'].astype(np.int64))
    np.testing.assert_allclose(full.reid_emb_dists.cpu().numpy(), gold['full_dists'], rtol=3e-6)
    start, end = (int(v) for v in gold['window'])
    frame = win.frame.to(dev())
    nodes_mask = (start <= frame) & (frame <= end)
    edges_mask = nodes_mask[full.edge_index[0]] & nodes_mask[full.edge_index[1]]
    first = int(torch.nonzero(nodes_mask)[0])
    sub = Graph(x=full.x[nodes_mask], x_ext=None, edge_attr=full.edge_attr[edges_mask],
                reid_emb_dists=full.reid_emb_dists[edges_mask],
                edge_index=full.edge_index.T[edges_mask].T - first)
    knn_mask = get_knn_mask(pwise_dist=sub.reid_emb_dists, edge_ixs=sub.edge_index, num_nodes=sub.num_nodes,
                            top_k_nns=ds['top_k_nns'], use_cuda=True, reciprocal_k_nns=ds['reciprocal_k_nns'],
                            symmetric_edges=True)
    assert np.array_equal(knn_mask.cpu().numpy(), gold['keep'])
    sub.edge_index = sub.edge_index.T[knn_mask].T
    sub.edge_attr = sub.edge_attr[knn_mask]
    model = make_model(c['mp'], c['P'])
    with torch.no_grad():
        out = model(sub)
    pruned = torch.sigmoid(out['classified_edges'][-1].view(-1))
    preds = torch.zeros(knn_mask.shape[0]).to(pruned.device)
    preds[knn_mask] = pruned
    assert float((preds.cpu() - torch.from_numpy(gold['edge_preds'])).abs().max()) <= PROB_TOL


def test_assign_edge_labels_against_golden():
    """MOTGraph.assign_edge_labels (data/mot_graph.py:223-262) on the GPU, both modes, bit-exact."""
    import os
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import Graph, MOTGraph
    gold = dict(np.load(os.path.join(os.path.dirname(__file__), 'golden', 'edge_labels.npz')))
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    ids = torch.from_numpy(gold['ids']).to(dev())
    for mode in ('all', 'closest'):
        got = ops.assign_edge_labels(ei, ids, mode)
        assert np.array_equal(got.cpu().numpy(), gold[f'labels_{mode}'])
    # through the reference-shaped entry point, shuffled edge order
    perm = torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(1)).to(dev())
    c = load_case('config1')
    cols = dict(synth.det_columns(c['win']), id=gold['ids'])
    mg = MOTGraph.from_tensors(cols, c['win'].reid, c['win'].x, None, {'fps': c['win'].fps}, dict(c['ds'], true_edge_labels='closest'))
    mg.graph_obj = Graph(x=c['win'].x, edge_index=ei[:, perm].contiguous())
    assert np.array_equal(mg.assign_edge_labels().cpu().numpy(), gold['labels_closest'][perm.cpu().numpy()])
    with pytest.raises(ValueError):
        ops.assign_edge_labels(ei, ids, 'nearest')


class _FullGraph(object):
    pass


def _sequence_full_graph(c, with_tables=True):
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    win, ds = c['win'], c['ds']
    mg = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, ds, inference_mode=True,
                  max_frame_dist=ds['frames_per_graph'] - 1)
    mg.construct_graph_object()
    if with_tables:                                            # the MOTGraph itself: detection table + embeddings available
        full = mg
    else:
        full = _FullGraph()
        full.graph_obj, full.graph_df = mg.graph_obj, {'frame': synth.det_columns(win)['frame']}
    full.frames = sorted(set(win.frame.tolist()))
    full.frames_per_graph = ds['frames_per_graph']
    return full


@pytest.mark.parametrize('inactive', [False, True])
@pytest.mark.parametrize('schedule', ['batched_rebuild', 'batched', 'window_by_window'])
def test_tracker_sequence_sliding_windows(inactive, schedule):
    """MPNTracker._evaluate_graph_in_batches (mpn_tracker.py:143-210) -- batched B200 schedule and the
    reference's window-by-window schedule -- against the reference's golden sequence output."""
    import os
    from mpntrackseg_b200.tracker import MPNTracker
    c = load_case('tracker_window')
    seq = dict(np.load(os.path.join(os.path.dirname(__file__), 'golden', 'tracker_sequence.npz')))
    tag = 'inactive' if inactive else 'knn'
    tracker = MPNTracker(dataset=None, graph_model=make_model(c['mp'], c['P']), use_gt=False,
                         eval_params={'set_pruned_edges_to_inactive': inactive}, dataset_params=c['ds'], window_batch=2)
    tracker.full_graph = _sequence_full_graph(c, with_tables=schedule == 'batched_rebuild')
    go = tracker.full_graph.graph_obj
    assert tracker._has_tables() == (schedule == 'batched_rebuild')
    if schedule == 'batched_rebuild':
        assert tracker._structured(go)
        tracker._evaluate_batched_rebuild()
    elif schedule == 'batched':
        tracker._evaluate_batched()
    else:
        tracker._evaluate_window_by_window(None)
    directed = go.edge_preds.cpu().numpy()
    assert np.abs(directed - seq[f'directed_preds_{tag}']).max() <= PROB_TOL
    from mpntrackseg_b200.utils.graph import to_lightweight_graph, to_undirected_graph
    to_undirected_graph(tracker.full_graph, attrs_to_update=('edge_preds', 'edge_labels'))
    assert np.array_equal(go.edge_index.cpu().numpy(), seq[f'undirected_edge_index_{tag}'].astype(np.int64))
    und = go.edge_preds.cpu().numpy()
    assert np.abs(und - seq[f'undirected_preds_{tag}']).max() <= PROB_TOL
    to_lightweight_graph(tracker.full_graph)
    assert not hasattr(go, 'x') and go.num_nodes == c['win'].N
    # identical decisions outside +-1e-3 of the 0.5 threshold
    ref_p = seq[f'undirected_preds_{tag}']
    sure = np.abs(ref_p - 0.5) > PROB_TOL
    kept = np.zeros(ref_p.shape[0], dtype=bool)
    und_ei = seq[f'undirected_edge_index_{tag}'].astype(np.int64)
    n = c['win'].N
    pos = {int(a) * n + int(b): i for i, (a, b) in enumerate(und_ei.T)}
    for a, b in go.edge_index.cpu().numpy().T:
        kept[pos[int(a) * n + int(b)]] = True
    assert np.array_equal(kept[sure], (ref_p >= 0.5)[sure])


def test_tracker_full_entry_point_and_general_undirected_merge():
    """_evaluate_graph_in_batches end to end, and to_undirected_graph on a shuffled (unstructured) edge list."""
    import os
    from mpntrackseg_b200.data.mot_graph import Graph
    from mpntrackseg_b200.tracker import MPNTracker
    from mpntrackseg_b200.utils.graph import to_undirected_graph
    c = load_case('tracker_window')
    seq = dict(np.load(os.path.join(os.path.dirname(__file__), 'golden', 'tracker_sequence.npz')))
    tracker = MPNTracker(graph_model=make_model(c['mp'], c['P']), eval_params={'set_pruned_edges_to_inactive': False},
                         dataset_params=c['ds'])
    tracker.full_graph = _sequence_full_graph(c)
    tracker._evaluate_graph_in_batches()
    go = tracker.full_graph.graph_obj
    assert go.edge_index.shape[1] == go.edge_preds.shape[0] and bool((go.edge_preds >= 0.5).all())
    assert abs(go.edge_index.shape[1] - seq['light_edge_index_knn'].shape[1]) <= 2
    # general path: shuffled directed edges
    ei = torch.from_numpy(np.concatenate((seq['undirected_edge_index_knn'], seq['undirected_edge_index_knn'][::-1]), axis=1)
                          .astype(np.int64))
    p = torch.from_numpy(seq['directed_preds_knn'])
    perm = torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(3))
    full = _FullGraph()
    full.graph_obj = Graph(x=torch.zeros(c['win'].N, 1), edge_index=ei[:, perm].to(dev()), edge_preds=p[perm].to(dev()))
    to_undirected_graph(full)
    assert np.array_equal(full.graph_obj.edge_index.cpu().numpy(), seq['undirected_edge_index_knn'].astype(np.int64))
    np.testing.assert_allclose(full.graph_obj.edge_preds.cpu().numpy(), seq['undirected_preds_knn'], rtol=1e-6, atol=1e-7)


# ------------------------------------------------------------------ layout
def test_edge_layout_invariants():
    from mpntrackseg_b200 import ops
    c = load_case('config1')
    ei = torch.from_numpy(c['gold']['edge_index'].astype(np.int64))
    n, e = c['win'].N, ei.shape[1]
    # shuffle the edge order: the layout must not rely on the reference's canonical order
    perm = torch.randperm(e, generator=torch.Generator().manual_seed(0))
    for edge_index in (ei, ei[:, perm]):
        lay = ops.edge_layout(edge_index.to(dev()), n)
        srow, scol, sedge = (t.cpu().long()[:e] for t in (lay.slot_row, lay.slot_col, lay.slot_edge))
        assert lay.num_out == int((edge_index[0] < edge_index[1]).sum())
        assert torch.equal(torch.sort(sedge).values, torch.arange(e))                 # a permutation
        assert torch.equal(edge_index[0][sedge], srow) and torch.equal(edge_index[1][sedge], scol)
        assert (srow[:lay.num_out] < scol[:lay.num_out]).all() and (srow[lay.num_out:] > scol[lay.num_out:]).all()
        for a, b in ((0, lay.num_out), (lay.num_out, e)):
            seg = srow[a:b]
            assert (seg[1:] >= seg[:-1]).all()
            same = seg[1:] == seg[:-1]
            assert (sedge[a:b][1:][same] > sedge[a:b][:-1][same]).all()               # stable inside a row
        optr, iptr = lay.out_ptr.cpu().long(), lay.in_ptr.cpu().long()
        assert optr[0] == 0 and optr[-1] == lay.num_out and iptr[0] == lay.num_out and iptr[-1] == e
        deg_out = torch.bincount(edge_index[0][edge_index[0] < edge_index[1]], minlength=n)
        deg_in = torch.bincount(edge_index[0][edge_index[0] > edge_index[1]], minlength=n)
        assert torch.equal(optr[1:] - optr[:-1], deg_out) and torch.equal(iptr[1:] - iptr[:-1], deg_in)


def test_edge_layout_rejects_self_loops():
    from mpntrackseg_b200 import ops
    ei = torch.tensor([[0, 1, 2], [1, 1, 0]], device=dev())
    with pytest.raises(ValueError, match='self-loops'):
        ops.edge_layout(ei, 3)


# ------------------------------------------------------------------ model
@pytest.mark.parametrize('engine', ENGINES)
@pytest.mark.parametrize('name', list(CASES))
def test_forward_matches_reference_golden(name, engine):
    c = load_case(name)
    win, gold = c['win'], c['gold']
    model = make_model(c['mp'], c['P'], engine)
    data = Data()
    data.x = win.x.to(dev())
    data.edge_index = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    data.edge_attr = torch.from_numpy(gold['edge_attr']).to(dev())
    with torch.no_grad():
        out = model(data, return_state=True)
    assert len(out['classified_edges']) == gold['logits'].shape[0]
    assert all(tuple(t.shape) == (gold['edge_index'].shape[1], 1) for t in out['classified_edges'])
    logits = torch.stack([t.view(-1) for t in out['classified_edges']]).cpu().numpy()
    assert_logits_close(logits, gold['logits'], name)
    scale = max(1.0, float(np.abs(gold['node_state']).max()))
    np.testing.assert_allclose(out['node_state'].cpu().numpy(), gold['node_state'], atol=2e-4 * scale, rtol=1e-3)
    lay = out['layout']
    e_state = torch.empty_like(out['edge_state_slots'])
    e_state[lay.slot_edge[:lay.num_edges].long()] = out['edge_state_slots']
    scale = max(1.0, float(np.abs(gold['edge_state']).max()))
    np.testing.assert_allclose(e_state.cpu().numpy(), gold['edge_state'], atol=2e-4 * scale, rtol=1e-3)


@pytest.mark.parametrize('engine', ENGINES)
def test_forward_is_deterministic_and_order_invariant(engine):
    """No float atomics: two runs are bit-identical; permuting the caller's edge order
    permutes the logits and nothing else."""
    c = load_case('config1')
    win, gold = c['win'], c['gold']
    model = make_model(c['mp'], c['P'], engine)
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    ea = torch.from_numpy(gold['edge_attr']).to(dev())
    data = Data()
    data.x, data.edge_index, data.edge_attr = win.x.to(dev()), ei, ea
    with torch.no_grad():
        a = model(data)['classified_edges'][-1]
        b = model(data)['classified_edges'][-1]
    assert torch.equal(a, b)
    e = ei.shape[1]
    half = e // 2
    # swap the two halves: still (row<col) group + (row>col) group, each internally stable
    perm = torch.cat((torch.arange(half, e), torch.arange(0, half))).to(dev())
    data.edge_index, data.edge_attr = ei[:, perm], ea[perm]
    with torch.no_grad():
        p = model(data)['classified_edges'][-1]
    assert torch.equal(p, a[perm])


def test_metalayer_single_step_matches_oracle():
    c = load_case('kitti_shape')
    win, gold, P = c['win'], c['gold'], c['P']
    model = make_model(c['mp'], P)
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    g = torch.Generator().manual_seed(5)
    x = torch.randn(win.N, 64, generator=g).abs()
    ea = torch.randn(ei.shape[1], 32, generator=g).abs()
    with torch.no_grad():
        e_ref = mpn_ref.edge_update(P, x, ei, ea)
        x_ref = mpn_ref.node_update(P, x, ei, e_ref)
        x_new, e_new = model.MPNet(x.to(dev()), ei.to(dev()), ea.to(dev()))
    np.testing.assert_allclose(e_new.cpu().numpy(), e_ref.numpy(), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(x_new.cpu().numpy(), x_ref.numpy(), rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize('engine', ENGINES)
def test_isolated_nodes_and_empty_graph(engine):
    """Nodes without in- or out-edges aggregate to zero (scatter_add zero fill); E = 0 works."""
    mp = default_graph_model_params(3, 2)
    P = synth.make_params(mp, seed=2, gain=1.5, core_only=True)
    model = make_model(mp, P, engine)
    g = torch.Generator().manual_seed(1)
    n = 9
    x = torch.randn(n, 2048, generator=g).abs()
    pairs = torch.tensor([[0, 0, 2], [2, 5, 5]])                       # nodes 1,3,4,6,7,8 isolated
    ei = torch.cat((pairs, pairs.flip(0)), dim=1)
    ea = torch.randn(3, 6, generator=g).repeat(2, 1)
    for edge_index, edge_attr in ((ei, ea), (ei[:, :0], ea[:0])):
        data = Data()
        data.x, data.edge_index, data.edge_attr = x.to(dev()), edge_index.to(dev()), edge_attr.to(dev())
        with torch.no_grad():
            out = model(data, return_state=True)
            ref = mpn_ref.mpn_forward(P, mp, x, edge_index, edge_attr, return_state=True)
        assert len(out['classified_edges']) == 2
        for a, b in zip(out['classified_edges'], ref['classified_edges']):
            assert tuple(a.shape) == tuple(b.shape)
            if b.numel():
                assert_logits_close(a.cpu().numpy(), b.numpy(), 'isolated')
        np.testing.assert_allclose(out['node_state'].cpu().numpy(), ref['node_state'].numpy(), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize('engine', ENGINES)
def test_config2_scale_against_oracle(engine):
    """MOTS20-scale window (BASELINE config 2: 15 frames x 150 detections, k=50): full hot
    path on the GPU (graph build + forward) against the oracle on the same inputs."""
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    win = synth.make_window(T=15, D=150, k=50, seed=4, node_feats='pooled')
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    mp = default_graph_model_params(12, 11)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    ref_g = graph_ref.build_graph(win.frame, win.reid, synth.det_columns(win), win.fps, ds)
    with torch.no_grad():
        ref = mpn_ref.mpn_forward(P, mp, win.x, ref_g['edge_index'], ref_g['edge_attr'])
    g = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, ds).construct_graph_object()
    assert torch.equal(g.edge_index.cpu(), ref_g['edge_index'])
    model = make_model(mp, P, engine)
    with torch.no_grad():
        out = model(g)
    got = torch.stack([t.view(-1) for t in out['classified_edges']]).cpu().numpy()
    exp = torch.stack([t.view(-1) for t in ref['classified_edges']]).numpy()
    assert_logits_close(got, exp, 'config2')


def test_encoders_against_torch():
    from mpntrackseg_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn(37, 2048, 8, 4, generator=g)
    np.testing.assert_allclose(ops.avgpool(x.to(dev())).cpu().numpy(), x.mean(dim=(2, 3)).numpy(), rtol=1e-5, atol=1e-6)
    x2 = torch.randn(5, 7, 3, 3, generator=g)                          # odd spatial size -> scalar path
    np.testing.assert_allclose(ops.avgpool(x2.to(dev())).cpu().numpy(), x2.mean(dim=(2, 3)).numpy(), rtol=1e-5, atol=1e-6)
    a, w, b = torch.randn(130, 2048, generator=g), torch.randn(128, 2048, generator=g) / 45, torch.randn(128, generator=g)
    ref = torch.relu(torch.nn.functional.linear(a, w, b))
    np.testing.assert_allclose(ops.linear(a.to(dev()), w.to(dev()), b.to(dev()), True).cpu().numpy(), ref.numpy(),
                               rtol=1e-4, atol=1e-4)
    a, w = torch.randn(3, 5, generator=g), torch.randn(1, 5, generator=g)
    np.testing.assert_allclose(ops.linear(a.to(dev()), w.to(dev()), None, False).cpu().numpy(),
                               torch.nn.functional.linear(a, w).numpy(), rtol=1e-5, atol=1e-6)


def _core_states(model, data):
    with torch.no_grad():
        out = model(data, return_state=True)
    return torch.stack([t.view(-1) for t in out['classified_edges']]).cpu().numpy(), out['node_state'].cpu()


def test_tc_engine_scales_activations_beyond_the_fp16_range():
    """Node states 10x beyond the fp16 maximum (65,504) stay on the tensor-core path: every step runs in its own
    power-of-two scale (mp_step_tc.cu "range bookkeeping"), and the logits still meet the 1e-3 bar against the
    oracle.  The encoders' last layers are multiplied by 32: the ReLU network is positively homogeneous up to its
    biases, so every activation grows 10-30x while the conditioning of the 12-step recurrence stays what it is for
    the benchmark weights (gain 1.25)."""
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    win = synth.make_window(T=15, D=150, k=50, seed=80, node_feats='pooled')     # the seed that overflowed in round 1
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    mp = default_graph_model_params(12, 11)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    for k in ('encoder.node_model.fc_layers.2', 'encoder.edge_model.fc_layers.4'):
        P[k + '.weight'] = P[k + '.weight'] * 32.0
        P[k + '.bias'] = P[k + '.bias'] * 32.0
    ref_g = graph_ref.build_graph(win.frame, win.reid, synth.det_columns(win), win.fps, ds)
    # At these magnitudes the fp32 oracle itself sits 6.5e-4 (relative) from the exact result, so two fp32-grade
    # evaluations can differ by more than the 1e-3 bar; the oracle is evaluated in fp64 here (same formulas, same
    # fp32 weights and inputs), which leaves the bar to the CUDA path alone (it lands at ~7e-4).
    with torch.no_grad():
        ref = mpn_ref.mpn_forward({k: v.double() for k, v in P.items()}, mp, win.x.double(), ref_g['edge_index'],
                                  ref_g['edge_attr'].double(), return_state=True)
    assert float(ref['node_state'].max()) > 10 * 65504.0, 'the case must exceed the fp16 range by 10x'
    g = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, ds).construct_graph_object()
    assert torch.equal(g.edge_index.cpu(), ref_g['edge_index'])
    model = make_model(mp, P, 'tc')
    got, x_state = _core_states(model, g)
    exp = torch.stack([t.view(-1) for t in ref['classified_edges']]).numpy()
    assert_logits_close(got, exp, 'scaled tc')
    np.testing.assert_allclose(x_state.numpy(), ref['node_state'].numpy(), rtol=2e-3, atol=1e-2)
    # the schedule really left s = 0, and is monotone here (the state only grows)
    lay = ops.edge_layout(g.edge_index, win.N)
    cw, keep = model.core_weights()
    with torch.no_grad():
        x0 = model.encode_nodes(g.x)
        e0 = model.encode_edges(g.edge_attr, lay)
        ops.mp_forward(cw, lay, x0, e0, 12, 2, engine='tc', debug=True)
    sched = ops.LAST_TC_SCHEDULE['sched'][1:13]
    assert sched[0] == 0 and max(sched) >= 4 and sched == sorted(sched), sched
    assert max(ops.LAST_TC_SCHEDULE['xmax'][1:14]) > 10 * 65504.0


def test_bench_workload_stays_on_the_tensor_core_path():
    """bench.py's windows (seeds 0..127 = what 8 ranks x 16 windows evaluate) with bench.py's weights run through
    engine='tc' without the fp16-range status (round 1 fell back to the fp32 kernels on seed 80: node state
    7.5e4 after 12 steps); all 16 windows of the batch that starts at seed 80 are checked against the fp64 oracle, each
    having run under the per-step scale its batch chose."""
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    mp = default_graph_model_params(12, 11)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    model = make_model(mp, P, 'tc')
    for lo in range(0, 128, 16):
        wins = [synth.make_window(T=15, D=150, k=50, seed=s, node_feats='pooled', node_dim=8, min_gap=0) for s in range(lo, lo + 16)]
        gen = torch.Generator(device=dev()).manual_seed(lo // 16)
        tabs = []
        for w in wins:
            t = {k: torch.from_numpy(v) for k, v in synth.det_columns(w).items()}
            t['reid'] = w.reid
            t['x'] = torch.randn((w.N, 2048), generator=gen, device=dev()).abs_()
            tabs.append(t)
        batch = build_window_graphs(tabs, ds, wins[0].fps, device=dev())
        with torch.no_grad():
            out = model.forward_batch(batch)                             # engine='tc' raises OverflowError on status != 0
        assert torch.isfinite(out.logits).all()
        if lo == 80:
            # every window of the batch ran under the batch's per-step scale, chosen for the largest of them
            P64 = {k: v.double() for k, v in P.items()}
            for i, w in enumerate(wins):
                ref_g = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds)
                with torch.no_grad():
                    ref = mpn_ref.mpn_forward(P64, mp, tabs[i]['x'].cpu().double(), ref_g['edge_index'],
                                              ref_g['edge_attr'].double(), return_state=True)
                if i == 0:
                    assert float(ref['node_state'].max()) > 65504.0
                got = out.graph_logits(i).cpu().numpy()
                exp = torch.stack([t.view(-1) for t in ref['classified_edges']]).numpy()
                assert_logits_close(got, exp, f'bench seed {80 + i}')


def test_tc_engine_reports_fp16_overflow_and_auto_falls_back():
    """A one-step jump beyond the 1024x headroom of the per-step scale (node Linear x 3e4), or a weight that has no
    finite fp16 image (x 1e6): engine='tc' raises, 'auto' reruns on the fp32 kernels."""
    c = load_case('kitti_shape')
    win, gold = c['win'], c['gold']
    mp = dict(c['mp'], num_enc_steps=3, num_class_steps=2)
    data = Data()
    data.x = win.x.to(dev())
    data.edge_index = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    data.edge_attr = torch.from_numpy(gold['edge_attr']).to(dev())
    for factor in (3.0e4, 1.0e6):
        P = {k: (v * factor if k.startswith('MPNet.node_model.node_model.0') else v) for k, v in c['P'].items()}
        with torch.no_grad():
            ref = make_model(mp, P, 'fp32')(data)['classified_edges'][-1]
            assert torch.isfinite(ref).all()
            with pytest.raises(OverflowError):
                make_model(mp, P, 'tc')(data)
            with pytest.warns(UserWarning, match='fp16 range'):
                auto = make_model(mp, P, 'auto')(data)['classified_edges'][-1]
        # 'auto' keeps the tensor-core node encoder (no overflow there), so compare to tolerance, not bitwise
        np.testing.assert_allclose(auto.cpu().numpy(), ref.cpu().numpy(), rtol=1e-3, atol=1e-3 * float(ref.abs().max()))


def test_edge_and_node_model_forward_match_oracle():
    """EdgeModel.forward / TimeAwareNodeModel.forward as standalone operators (models/mpn.py:67-69, 83-99)."""
    c = load_case('kitti_shape')
    win, gold, P = c['win'], c['gold'], c['P']
    model = make_model(c['mp'], P)
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    perm = torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(1))
    ei = ei[:, perm]                                                     # any edge order
    g = torch.Generator().manual_seed(6)
    x = torch.randn(win.N, 64, generator=g).abs()
    ea = torch.randn(ei.shape[1], 32, generator=g).abs()
    with torch.no_grad():
        e_ref = mpn_ref.edge_update(P, x, ei, ea)
        x_ref = mpn_ref.node_update(P, x, ei, e_ref)
        e_new = model.MPNet.edge_model(x.to(dev()), ei.to(dev()), ea.to(dev()))
        x_new = model.MPNet.node_model(x.to(dev()), ei.to(dev()), e_ref.to(dev()))
    assert tuple(e_new.shape) == tuple(e_ref.shape) and tuple(x_new.shape) == tuple(x_ref.shape)
    np.testing.assert_allclose(e_new.cpu().numpy(), e_ref.numpy(), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(x_new.cpu().numpy(), x_ref.numpy(), rtol=1e-4, atol=1e-3)


def test_single_frame_and_single_node_windows_build_empty_graphs():
    """A window with one detection, or with all detections in one frame, has no time-valid pair: the reference
    returns an empty edge set (utils/graph.py:6-37)."""
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    from mpntrackseg_b200.utils.graph import get_time_valid_conn_ixs
    ds = default_dataset_params(top_k_nns=5, frames_per_graph=15)
    for frames in ([3], [7, 7, 7, 7]):
        f = torch.tensor(frames, dtype=torch.int64)
        pairs = get_time_valid_conn_ixs(f, 'max', use_cuda=True)
        assert tuple(pairs.shape) == (2, 0) and torch.equal(pairs, graph_ref.time_valid_pairs(f, 'max'))
        n = len(frames)
        cols = {'frame': np.asarray(frames, dtype=np.float64), 'bb_height': np.full(n, 100.0), 'bb_width': np.full(n, 40.0),
                'feet_x': np.arange(n, dtype=np.float64), 'feet_y': np.zeros(n)}
        g = MOTGraph.from_tensors(cols, torch.randn(n, 256), torch.randn(n, 2048, 1, 1).to(dev()), None, {'fps': 30.0}, ds).construct_graph_object()
        assert tuple(g.edge_index.shape) == (2, 0) and g.edge_attr.shape[0] == 0


def test_batched_graph_build_and_forward_match_per_window_path():
    """build_window_graphs + forward_batch (one pass, batch-global ids) == per-window MOTGraph + forward,
    and both match the oracle's edge sets."""
    from mpntrackseg_b200.data.mot_graph import MOTGraph, build_window_graphs
    shapes = [(6, 9, 5), (5, 12, 7), (7, 6, 40), (4, 8, 3)]
    wins = [synth.make_window(T=t, D=d, k=k, seed=30 + i) for i, (t, d, k) in enumerate(shapes)]
    mp = default_graph_model_params(5, 4)
    P = synth.make_params(mp, seed=4, gain=2.0, core_only=True)
    model = make_model(mp, P, 'tc')
    for recip, mfd in ((True, 'max'), (False, 2)):
        ds = default_dataset_params(top_k_nns=6, frames_per_graph=7, reciprocal_k_nns=recip)
        inputs = [dict(synth.det_columns(w), reid=w.reid, x=w.x) for w in wins]
        batch = build_window_graphs(inputs, ds, fps=30.0, max_frame_dist=mfd)
        assert batch.num_graphs == len(wins)
        with torch.no_grad():
            out = model.forward_batch(batch)
        for g, w in enumerate(wins):
            ref_g = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds, max_frame_dist=mfd)
            gg = batch.graph(g)
            assert torch.equal(gg.edge_index.cpu(), ref_g['edge_index']), (g, recip)
            np.testing.assert_allclose(gg.edge_attr.cpu().numpy(), ref_g['edge_attr'].numpy(), rtol=3e-6, atol=1e-6)
            single = MOTGraph.from_tensors(synth.det_columns(w), w.reid, w.x, None, {'fps': 30.0}, ds,
                              max_frame_dist=mfd).construct_graph_object()
            assert torch.equal(single.edge_index, gg.edge_index)
            with torch.no_grad():
                ref = mpn_ref.mpn_forward(P, mp, w.x, ref_g['edge_index'], ref_g['edge_attr'])
            got = out.graph_logits(g).cpu().numpy()
            exp = torch.stack([t.view(-1) for t in ref['classified_edges']]).numpy()
            assert_logits_close(got, exp, f'batch graph {g}')
            assert len(out[g]['classified_edges']) == 4


def test_batched_builder_inference_mode_keeps_all_time_valid_pairs():
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    w = synth.make_window(T=6, D=7, k=5, seed=77)
    ds = default_dataset_params(top_k_nns=5, frames_per_graph=4)
    batch = build_window_graphs([dict(synth.det_columns(w), reid=w.reid, x=w.x)], ds, fps=30.0, inference_mode=True,
                                max_frame_dist=3)
    ref = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds, inference_mode=True, max_frame_dist=3)
    assert torch.equal(batch.edge_index.cpu(), ref['edge_index'])
    np.testing.assert_allclose(batch.reid_emb_dists.cpu().numpy(), ref['reid_emb_dists'].numpy(), rtol=3e-6)


@pytest.mark.parametrize('name', ['tiny_full', 'config1'])
def test_full_forward_with_mask_branch_matches_reference_golden(name):
    """MOTMPNet.forward(data) with x_ext: attentive aggregation kernel + cuDNN convs against the
    reference's own full forward (mask_predictions of the classified steps)."""
    c = load_case(name)
    win, gold = c['win'], c['gold']
    model = make_model(c['mp'], c['P'], 'tc')
    data = Data()
    data.x, data.x_ext = win.x.to(dev()), win.x_ext.to(dev())
    data.edge_index = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    data.edge_attr = torch.from_numpy(gold['edge_attr']).to(dev())
    with torch.backends.cudnn.flags(allow_tf32=False), torch.no_grad():
        out = model(data)
    logits = torch.stack([t.view(-1) for t in out['classified_edges']]).cpu().numpy()
    assert_logits_close(logits, gold['logits'], name)
    assert len(out['mask_predictions']) == c['mp']['num_class_steps']
    m = out['mask_predictions'][-1]
    assert tuple(m.shape) == (win.N, 1, 56, 56)
    np.testing.assert_allclose(m[:, 0, ::7, ::7].cpu().numpy(), gold['mask_last_sample'], rtol=2e-3, atol=2e-3)
    means = np.array([float(t.double().mean()) for t in out['mask_predictions']])
    np.testing.assert_allclose(means, gold['mask_step_means'], rtol=2e-3, atol=1e-4)


def test_attn_aggregate_against_oracle_softmax():
    from mpntrackseg_b200 import ops
    c = load_case('tiny_nonrecip')
    ei = torch.from_numpy(c['gold']['edge_index'].astype(np.int64))
    n = c['win'].N
    g = torch.Generator().manual_seed(8)
    z = torch.randn(n, 6, 5, 5, generator=g)
    logits = torch.randn(ei.shape[1], 1, generator=g) * 3
    lay = ops.edge_layout(ei.to(dev()), n)
    fin, fout = ops.attn_aggregate(z.to(dev()), lay, logits.to(dev()))
    src, dst = ei
    for name, sel, got in (('out', src < dst, fout), ('in', src > dst, fin)):
        w = mpn_ref.segment_softmax(logits[sel], src[sel])
        ref = mpn_ref.segment_add(z[dst[sel]] * w[:, :, None, None], src[sel], n)
        np.testing.assert_allclose(got.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-6, err_msg=name)


def test_node_encoder_tc_against_fp32():
    """Also beyond one 128-node tile per CTA (n > 2 * SMs * 128: the mbarrier parities and the TMA weight stream carry
    over to the next tile), with an odd number of 64-wide K chunks (k0 = 192)."""
    from mpntrackseg_b200 import ops
    g = torch.Generator().manual_seed(12)
    t = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 128
    cases = [(n, 2048) for n in (1, 127, 300, 2250)] + [(t + 1, 64), (t + 1, 192), (t + 1, 2048), (5 * t // 2 + 3, 64),
                                                        (5 * t // 2 + 3, 192)]
    for n, k0 in cases:
        x = torch.randn(n, k0, generator=g).abs()
        w0, b0 = torch.randn(128, k0, generator=g) / (k0 ** 0.5), torch.randn(128, generator=g) * 0.1
        w1, b1 = torch.randn(32, 128, generator=g) / 11, torch.randn(32, generator=g) * 0.1
        ref = torch.relu(torch.nn.functional.linear(torch.relu(torch.nn.functional.linear(x.double(), w0.double(), b0.double())),
                                                    w1.double(), b1.double())).float()
        args = (x.to(dev()), [w0.to(dev()), w1.to(dev())], [b0.to(dev()), b1.to(dev())])
        got_tc = ops.node_encoder(*args, engine='tc').cpu()
        got_32 = ops.node_encoder(*args, engine='fp32').cpu()
        scale = float(ref.abs().max())
        assert float((got_32 - ref).abs().max()) <= 2e-5 * scale
        assert float((got_tc - ref).abs().max()) <= 2e-5 * scale, (n, k0)
    assert max(n for n, _ in cases) > 2 * t


def test_weighted_bce_loss_and_gradient_against_oracle():
    """pl_module.py:88-105 on the GPU (loss value and d loss / d logits) against torch autograd on CPU."""
    from mpntrackseg_b200 import ops
    g = torch.Generator().manual_seed(21)
    for e, pos_frac in ((1000, 0.1), (37, 0.0), (5000, 0.5)):
        logits = (torch.randn(3, e, generator=g) * 3).requires_grad_(True)
        labels = (torch.rand(e, generator=g) < pos_frac).float()
        ref = mpn_ref.weighted_bce_loss([logits[i].view(-1, 1) for i in range(3)], labels, tracking_weight=0.7)
        ref.backward()
        loss, pw, grad = ops.weighted_bce(logits.detach().to(dev()), labels.to(dev()), weight=0.7, want_grad=True)
        assert abs(float(loss) - float(ref)) <= 1e-5 * max(1.0, abs(float(ref)))
        pos = float(labels.sum())
        assert abs(float(pw) - ((e - pos) / pos if pos else 0.0)) <= 1e-4 * max(1.0, e)
        np.testing.assert_allclose(grad.cpu().numpy(), logits.grad.numpy(), rtol=2e-4, atol=1e-8)


def test_tensor_core_gram_knn_equals_exact_path_and_repairs_near_ties():
    """KNN edge set from the tcgen05 Gram distances == exact fp32 path == oracle, including windows whose
    embeddings produce exact ties / sub-band gaps at the k boundary (those rows must take the exact repair)."""
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    ds = default_dataset_params(top_k_nns=9, frames_per_graph=8)
    wins = [synth.make_window(T=8, D=20, k=9, seed=50 + i) for i in range(3)]
    # window 1: duplicated embeddings (exact distance ties); window 2: tiny perturbations (gaps below the band)
    g = torch.Generator().manual_seed(3)
    wins[1].reid = wins[1].reid[torch.arange(wins[1].N) % 40].contiguous()
    base = wins[2].reid[torch.arange(wins[2].N) % 40]
    wins[2].reid = (base + 1e-7 * torch.randn(base.shape, generator=g)).contiguous()
    inputs = [dict(synth.det_columns(w), reid=w.reid, x=w.x) for w in wins]
    tc = build_window_graphs(inputs, ds, fps=30.0, engine='tc')
    stats = list(ops.LAST_KNN_STATS)
    ex = build_window_graphs(inputs, ds, fps=30.0, engine='fp32')
    assert stats[0] == 1 and stats[1] > 0, stats            # tensor-core path ran and repaired some rows
    assert ops.LAST_KNN_STATS[0] == 0
    assert tc.pair_ptr == ex.pair_ptr
    assert torch.equal(tc.edge_index, ex.edge_index)
    np.testing.assert_allclose(tc.edge_attr.cpu().numpy(), ex.edge_attr.cpu().numpy(), rtol=3e-6, atol=1e-6)
    ref = graph_ref.build_graph(wins[0].frame, wins[0].reid, synth.det_columns(wins[0]), 30.0, ds)
    assert torch.equal(tc.graph(0).edge_index.cpu(), ref['edge_index'])


@pytest.mark.parametrize('recip', [True, False])
def test_knn_graph_pairs_ragged_windows_match_oracle(recip):
    """Batched builder on ragged windows (1 node, one frame only, sizes around the 32-bit word and 128-row tile
    boundaries, k above and below the row length) against the oracle, window by window, for both engines.  One
    window has duplicated embeddings: its distances come in exactly tied groups that sit one ulp apart, where the
    order depends on the summation order of the distance itself -- there the two engines must agree with each other
    (the tensor-core path has to repair those rows with the exact kernel's arithmetic)."""
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    shapes = [(1, 1), (1, 6), (2, 1), (3, 11), (5, 13), (9, 15), (4, 65), (7, 37)]      # (T, D): N = 1, 6, 2, 33, 65, 135, 260, 259
    wins = [synth.make_window(T=t, D=d, k=3, seed=70 + i) for i, (t, d) in enumerate(shapes)]
    tied = 5
    wins[tied].reid = wins[tied].reid[torch.arange(wins[tied].N) % 20].contiguous()
    inputs = [dict(synth.det_columns(w), reid=w.reid, x=w.x) for w in wins]
    for k in (1, 4, 40, 300):
        ds = default_dataset_params(top_k_nns=k, frames_per_graph=9, reciprocal_k_nns=recip)
        tc = build_window_graphs(inputs, ds, fps=30.0, engine='tc')
        ex = build_window_graphs(inputs, ds, fps=30.0, engine='fp32')
        assert tc.pair_ptr == ex.pair_ptr and torch.equal(tc.edge_index, ex.edge_index), (recip, k)
        for g, w in enumerate(wins):
            if g == tied:
                continue
            ref = graph_ref.build_graph(w.frame, w.reid, synth.det_columns(w), w.fps, ds)
            got = tc.graph(g)
            assert torch.equal(got.edge_index.cpu(), ref['edge_index']), (recip, k, g, w.N)
            np.testing.assert_allclose(got.edge_attr.cpu().numpy(), ref['edge_attr'].numpy(), rtol=3e-6, atol=1e-6)


def test_tensor_core_gram_config2_window_no_repairs_needed():
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    w = synth.make_window(T=15, D=150, k=50, seed=4)
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    inp = [dict(synth.det_columns(w), reid=w.reid, x=w.x)]
    tc = build_window_graphs(inp, ds, fps=30.0, engine='tc')
    repaired = ops.LAST_KNN_STATS[1]
    ex = build_window_graphs(inp, ds, fps=30.0, engine='fp32')
    assert torch.equal(tc.edge_index, ex.edge_index)
    assert repaired <= w.N // 20, repaired                  # well-separated data: (almost) nothing to repair


def _oracle_loss_and_grads(P, mp, x, ei, ea, labels, weight):
    Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    out = mpn_ref.mpn_forward(Pg, mp, x, ei, ea)
    loss = mpn_ref.weighted_bce_loss(out['classified_edges'], labels, tracking_weight=weight)
    loss.backward()
    return float(loss), {k: v.grad for k, v in Pg.items() if v.grad is not None}


@pytest.mark.parametrize('name', ['tiny_nonrecip', 'kitti_shape'])
def test_training_backward_matches_autograd_of_the_oracle(name):
    """Hand-written backward (csrc/train_ops.cu, training.py) of the core network + weighted BCE against
    torch autograd through the CPU oracle on the same graph, weights and labels."""
    from mpntrackseg_b200.training import CoreTrainer
    c = load_case(name)
    win, gold, mp = c['win'], c['gold'], c['mp']
    P = {k: v for k, v in c['P'].items() if k.startswith(('encoder.', 'classifier.', 'MPNet.'))}
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    ea = torch.from_numpy(gold['edge_attr'])
    labels = (win.ident[ei[0]] == win.ident[ei[1]]).float()
    assert 0 < labels.sum() < labels.numel()
    ref_loss, ref_g = _oracle_loss_and_grads(P, mp, win.x, ei, ea, labels, 0.8)
    model = make_model(mp, c['P'], 'fp32')
    tr = CoreTrainer(model)
    data = Data()
    data.x, data.edge_index, data.edge_attr = win.x.to(dev()), ei.to(dev()), ea.to(dev())
    loss = tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert abs(float(loss) - ref_loss) <= 2e-4 * max(1.0, abs(ref_loss))
    assert set(tr.g) == set(ref_g)
    for k, g in ref_g.items():
        got = tr.g[k].cpu()
        scale = float(g.abs().max()) + 1e-12
        err = float((got - g).abs().max()) / scale
        assert err <= 2e-3, (k, err, scale)
    # two identical passes -> bit-identical gradients (deterministic reductions)
    g1 = tr.grad.clone()
    tr.loss_and_grads(data, labels.to(dev()), tracking_weight=0.8)
    assert torch.equal(g1, tr.grad)


def test_motmpnet_forward_under_autograd_fills_parameter_gradients():
    """The reference's training call (pl_module.py:122-135): model(data) with autograd on, a torch loss on
    the returned logits, loss.backward().  p.grad of the core weights must match autograd through the oracle; a torch
    optimizer step must move the weights the kernels read."""
    c = load_case('tiny_nonrecip')
    win, gold, mp = c['win'], c['gold'], c['mp']
    P = {k: v for k, v in c['P'].items() if k.startswith(('encoder.', 'classifier.', 'MPNet.'))}
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    ea = torch.from_numpy(gold['edge_attr'])
    labels = (win.ident[ei[0]] == win.ident[ei[1]]).float()
    ref_loss, ref_g = _oracle_loss_and_grads(P, mp, win.x, ei, ea, labels, 1.0)
    model = make_model(mp, c['P'], 'fp32').train()
    data = Data()
    data.x, data.edge_index, data.edge_attr, data.x_ext = win.x.to(dev()), ei.to(dev()), ea.to(dev()), None
    opt = torch.optim.Adam([p for n, p in model.named_parameters() if n in P], lr=1e-3)
    out = model(data)
    assert len(out['classified_edges']) == mp['num_class_steps'] and out['classified_edges'][-1].shape == (ei.shape[1], 1)
    with torch.no_grad():
        ref_logits = model.eval()(data)['classified_edges']
    model.train()
    for a, b in zip(out['classified_edges'], ref_logits):           # same logits as the inference kernels, caller's edge order
        assert float((a.detach() - b).abs().max()) <= 1e-3 * max(1.0, float(b.abs().max()))
    loss = mpn_ref.weighted_bce_loss(out['classified_edges'], labels.to(dev()))
    assert abs(float(loss) - ref_loss) <= 2e-4 * max(1.0, abs(ref_loss))
    loss.backward()
    named = dict(model.named_parameters())
    for k, g in ref_g.items():
        got = named[k].grad.cpu()
        scale = float(g.abs().max()) + 1e-12
        assert float((got - g).abs().max()) / scale <= 2e-3, k
    before = named['classifier.edge_model.fc_layers.2.bias'].detach().clone()
    opt.step()
    assert not torch.equal(before, named['classifier.edge_model.fc_layers.2.bias'].detach())
    with torch.no_grad():
        moved = model.eval()(data)['classified_edges'][-1]
    assert float((moved - ref_logits[-1]).abs().max()) > 0        # the kernels read the updated weights


def test_training_through_the_mask_branch_matches_autograd_of_the_oracle():
    """The reference's full training loss (pl_module.py:88-120: weighted tracking BCE + segmentation BCE on the matched
    detections, every classified step) on the full model: model.train()(data) with x_ext, torch loss, loss.backward().
    Gradients of ALL parameters (mask branch through cuDNN + the attention backward kernels, tracking network through the
    attention weights and the logits) against autograd through the oracle."""
    import torch.nn.functional as F
    # the convolutions of the mask branch are cuDNN: full fp32 for a gradient comparison with the CPU oracle (torch's
    # default lets cuDNN use TF32, whose 10-bit products show up as several percent on these small, cancelling gradients)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        _mask_branch_training_check(F)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32


def _mask_branch_training_check(F):
    c = load_case('tiny_full')
    win, gold, mp, P = c['win'], c['gold'], c['mp'], c['P']
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    ea = torch.from_numpy(gold['edge_attr'])
    labels = (win.ident[ei[0]] == win.ident[ei[1]]).float()
    g = torch.Generator().manual_seed(17)
    gt_masks = (torch.rand(win.N, 1, 56, 56, generator=g) > 0.5).float()
    ixs = torch.arange(0, win.N, 3)
    w_track, w_seg = 0.8, 0.6

    def full_loss(out, lab, gtm):
        pos = lab.sum()
        pw = (lab.shape[0] - pos) / pos
        loss = 0
        for lg, mk in zip(out['classified_edges'], out['mask_predictions']):
            loss = loss + w_track * F.binary_cross_entropy_with_logits(lg.view(-1), lab, pos_weight=pw)
            loss = loss + w_seg * F.binary_cross_entropy_with_logits(mk[ixs.to(mk.device)], gtm[ixs.to(gtm.device)])
        return loss

    Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    ref_out = mpn_ref.mpn_forward(Pg, mp, win.x, ei, ea, x_ext=win.x_ext)
    assert tuple(ref_out['mask_predictions'][-1].shape) == tuple(gt_masks.shape)
    ref_loss = full_loss(ref_out, labels, gt_masks)
    ref_loss.backward()
    model = make_model(mp, P, 'fp32').train()
    data = Data()
    data.x, data.edge_index, data.edge_attr, data.x_ext = win.x.to(dev()), ei.to(dev()), ea.to(dev()), win.x_ext.to(dev())
    out = model(data)
    assert len(out['classified_edges']) == mp['num_class_steps'] == len(out['mask_predictions'])
    loss = full_loss(out, labels.to(dev()), gt_masks.to(dev()))
    assert abs(float(loss) - float(ref_loss)) <= 5e-4 * max(1.0, abs(float(ref_loss)))
    loss.backward()
    named = dict(model.named_parameters())
    checked, worst = 0, {}
    for k, p in Pg.items():
        if p.grad is None:
            continue
        got = named[k].grad
        assert got is not None, k
        scale = float(p.grad.abs().max()) + 1e-12
        worst[k] = float((got.cpu() - p.grad).abs().max()) / scale
        checked += 1
    core = ('encoder.', 'classifier.', 'MPNet.')
    # hand-written kernels (tracking network): 3e-3 of each tensor's largest entry, as in the tracking-only test; the
    # mask branch is cuDNN arithmetic (algorithm choice, e.g. Winograd for the 3x3 stacks, is the library's): 2e-2
    bad = {k: round(v, 5) for k, v in worst.items() if v > (3e-3 if k.startswith(core) else 2e-2)}
    assert not bad, f'gradient mismatches: {bad}; worst overall {sorted(worst.items(), key=lambda kv: -kv[1])[:6]}'
    assert checked >= 40 and any(k.startswith('MPAttentionNet') for k in Pg) and Pg['MPNet.node_model.node_model.0.weight'].grad is not None
    print('worst relative gradient errors:', sorted(((round(v, 5), k) for k, v in worst.items()), reverse=True)[:8])


def test_adam_step_matches_torch_adam():
    from mpntrackseg_b200.training import CoreTrainer
    c = load_case('tiny_nonrecip')
    win, gold, mp = c['win'], c['gold'], c['mp']
    ei = torch.from_numpy(gold['edge_index'].astype(np.int64))
    ea = torch.from_numpy(gold['edge_attr'])
    labels = (win.ident[ei[0]] == win.ident[ei[1]]).float()
    model = make_model(mp, c['P'], 'fp32')
    tr = CoreTrainer(model, lr=1e-3, weight_decay=1e-4)
    data = Data()
    data.x, data.edge_index, data.edge_attr = win.x.to(dev()), ei.to(dev()), ea.to(dev())
    ref_p = [p.detach().clone().requires_grad_(True) for p in tr.named.values()]
    opt = torch.optim.Adam(ref_p, lr=1e-3, weight_decay=1e-4)
    for _ in range(3):
        tr.loss_and_grads(data, labels.to(dev()))
        for rp, g in zip(ref_p, tr.g.values()):
            rp.grad = g.detach().clone()
        opt.step()
        tr.adam_step()
    for rp, p in zip(ref_p, tr.named.values()):
        np.testing.assert_allclose(p.detach().cpu().numpy(), rp.detach().cpu().numpy(), rtol=1e-5, atol=1e-7)


def test_embedding_store_pool_and_motgraph_from_store(tmp_path):
    """f3: a store in the reference's layout -> pooled variant -> MOTGraph(seq_det_df, start_frame, end_frame, ...)
    builds the same graph / logits as the tensor-taking form; SequenceEmbeddings slices are the window's rows."""
    import pandas as pd
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.embedding_store import EmbeddingStore, SequenceEmbeddings
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    win = synth.make_window(T=8, D=9, k=6, seed=41, node_feats='full')
    cols = synth.det_columns(win)
    df = pd.DataFrame(dict(cols, frame=win.frame.numpy(), detection_id=np.arange(win.N), bb_left=np.zeros(win.N)))
    seq_info = {'seq_path': str(tmp_path), 'det_file_name': 'det', 'fps': win.fps}
    ds = dict(default_dataset_params(top_k_nns=6, frames_per_graph=5), reid_embeddings_dir='reid',
              node_core_embeddings_dir='core', node_ext_embeddings_dir=None)
    store = EmbeddingStore(seq_info)
    store.write('reid', win.frame, df.detection_id.values, win.reid)
    store.write('core', win.frame, df.detection_id.values, win.x)
    store.pool('core', 'core_pooled', device=dev())
    pooled_ref = ops.avgpool(win.x.to(dev())).cpu()
    got = torch.cat([store.read_frame('core_pooled', f) for f in store.frames('core_pooled')])
    assert torch.equal(got[:, 0], torch.arange(win.N, dtype=torch.float32)) and torch.equal(got[:, 1:], pooled_ref)
    np.testing.assert_allclose(got[:, 1:].numpy(), win.x.mean(dim=(2, 3)).numpy(), rtol=1e-5, atol=1e-6)

    seq = SequenceEmbeddings(df, seq_info, ds, pooled=True)
    a, b = seq.rows(3, 7)
    assert (a, b) == (2 * win.D, 7 * win.D) and seq.node_core.is_pinned()
    reid_w, core_w = seq.window(3, 7, device=dev())
    torch.cuda.synchronize()
    assert torch.equal(reid_w.cpu(), win.reid[a:b]) and torch.equal(core_w.cpu(), pooled_ref[a:b])

    mp = default_graph_model_params(4, 3)
    P = synth.make_params(mp, seed=3, gain=2.0, core_only=True)
    model = make_model(mp, P)
    sel = slice(a, b)
    tab = {k: v[sel] for k, v in cols.items()}
    g_ref = MOTGraph.from_tensors(tab, win.reid[sel], win.x[sel].to(dev()), None, seq_info, ds).construct_graph_object()
    for pooled_flag, exact in ((False, True), (True, True)):
        mg = MOTGraph(seq_det_df=df, start_frame=3, end_frame=7, step_size=1, seq_info_dict=seq_info,
                      dataset_params=dict(ds, node_core_pooled=pooled_flag))
        g = mg.construct_graph_object()
        assert torch.equal(g.edge_index, g_ref.edge_index) and torch.equal(g.edge_attr, g_ref.edge_attr)
        with torch.no_grad():
            a_, b_ = model(g)['classified_edges'][-1], model(g_ref)['classified_edges'][-1]
        assert torch.equal(a_, b_) if exact else torch.allclose(a_, b_)


@pytest.mark.parametrize('engine', ENGINES)
def test_config5_dense_crowd_window_matches_reference_golden(engine):
    """BASELINE.json configs[4] (15 frames x 300 detections, k = 100; N = 4,500, E = 179 k, node state 4.8e4): graph
    build bit-exact, logits within the bar, against outputs of the reference itself (tests/golden/config5.npz)."""
    from mpntrackseg_b200.data.mot_graph import MOTGraph, build_window_graphs
    c = load_big_case('config5')
    win, ds, gold = c['win'], c['ds'], c['gold']
    g = MOTGraph.from_tensors(synth.det_columns(win), win.reid, win.x, None, {'fps': win.fps}, ds).construct_graph_object()
    assert np.array_equal(g.edge_index.cpu().numpy(), gold['edge_index'].astype(np.int64))
    np.testing.assert_allclose(g.edge_attr[::16].cpu().numpy(), gold['edge_attr_sample'], rtol=2e-6, atol=2e-7)
    tab = {k: torch.from_numpy(v) for k, v in synth.det_columns(win).items()}
    tab.update(reid=win.reid, x=win.x.to(dev()))
    batch = build_window_graphs([tab], ds, win.fps, device=dev(), engine=engine)         # the batched (Gram) builder
    assert torch.equal(batch.edge_index, g.edge_index)
    model = make_model(c['mp'], c['P'], engine)
    with torch.no_grad():
        out = model(g)
    lg = [t.view(-1).cpu().numpy() for t in out['classified_edges']]
    assert_logits_close(lg[-1], gold['logits_last'], 'config5 last step')
    assert_logits_close(lg[0], gold['logits_first'], 'config5 first classified step')
    np.testing.assert_allclose(np.array([float(np.mean(v.astype(np.float64))) for v in lg]), gold['logits_step_means'],
                               rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize('k', [25, 50, 100, 128])
def test_thresholded_and_dense_knn_builds_keep_the_same_pairs(k, monkeypatch):
    """The two tensor-core graph builds (thresholded candidate lists: default up to k = 64, forced up to k = 128 with
    MPN_KNN_THRESHOLDED; dense blocks + row select: MPN_KNN_DENSE) and the exact fp32 build return identical pairs on
    the configs[4] window (N = 4,500) next to a configs[1]-sized one."""
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    c = load_big_case('config5')
    win = c['win']
    ds = dict(c['ds'], top_k_nns=k)
    tab = {kk: torch.from_numpy(v) for kk, v in synth.det_columns(win).items()}
    tab.update(reid=win.reid, x=win.x.to(dev()))
    w2 = synth.make_window(T=15, D=150, k=k, seed=11, node_feats='pooled', node_dim=win.x.shape[1], min_gap=2e-6)
    tab2 = {kk: torch.from_numpy(v) for kk, v in synth.det_columns(w2).items()}
    tab2.update(reid=w2.reid, x=w2.x.to(dev()))
    got = {}
    for name, env in (('thresholded', 'MPN_KNN_THRESHOLDED'), ('dense', 'MPN_KNN_DENSE')):
        monkeypatch.setenv(env, '1')
        got[name] = build_window_graphs([tab, tab2], ds, win.fps, device=dev(), engine='tc')
        monkeypatch.delenv(env)
    exact = build_window_graphs([tab, tab2], ds, win.fps, device=dev(), engine='fp32')
    for name, b in got.items():
        assert b.pair_ptr == exact.pair_ptr, (name, k)
        assert torch.equal(b.edge_index, exact.edge_index), (name, k)
        np.testing.assert_allclose(b.edge_attr.cpu().numpy(), exact.edge_attr.cpu().numpy(), rtol=3e-6, atol=1e-6)
    assert torch.equal(got['thresholded'].edge_attr, got['dense'].edge_attr), k


@pytest.mark.parametrize('engine', ENGINES)
def test_window_beyond_5120_nodes_takes_the_streamed_row_select(engine):
    """A window of 5,400 detections is above the limit (5,120) of the register-held row select: row_select_kernel
    re-reads its rows (csrc/knn_graph.cu) and must produce the reference's kept pairs (tests/golden/big_window.npz),
    alone and next to a small window in the same batch; on the tensor cores through the dense Gram build (code 1)."""
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import build_window_graphs
    c = load_big_case('big_window')
    win, ds, gold = c['win'], c['ds'], c['gold']
    tab = {k: torch.from_numpy(v) for k, v in synth.det_columns(win).items()}
    tab.update(reid=win.reid, x=win.x.to(dev()))
    small = synth.make_window(T=6, D=9, k=20, seed=3, node_feats='pooled', node_dim=8)
    stab = {k: torch.from_numpy(v) for k, v in synth.det_columns(small).items()}
    stab.update(reid=small.reid, x=small.x.to(dev()))
    ref_small = graph_ref.build_graph(small.frame, small.reid, synth.det_columns(small), small.fps, ds)
    for tabs in ([tab], [stab, tab]):
        batch = build_window_graphs(tabs, ds, win.fps, device=dev(), engine=engine)
        if engine == 'tc':
            assert ops.LAST_KNN_STATS[0] == 1, ops.LAST_KNN_STATS
        gi = len(tabs) - 1
        g = batch.graph(gi)
        p = g.edge_index.shape[1] // 2
        assert np.array_equal(g.edge_index[:, :p].cpu().numpy(), gold['pairs'].astype(np.int64))
        np.testing.assert_allclose(g.edge_attr[:p:8, 5].cpu().numpy(), gold['reid_dist_sample'], rtol=2e-6)
        if gi:
            assert torch.equal(batch.graph(0).edge_index.cpu(), ref_small['edge_index'])


# ------------------------------------------------------------------ rounding + identity assignment (SURVEY.md f2)
@pytest.mark.parametrize('tag', ['a', 'b'])
def test_rounding_and_identities_match_the_reference(tag):
    """Greedy projection, constraint statistics and connected components against outputs of the reference's own
    GreedyProjector / compute_constr_satisfaction_rate and scipy's connected_components (tests/golden/rounding.npz):
    integer work, so everything is bit-exact."""
    import os
    from types import SimpleNamespace
    from mpntrackseg_b200 import ops
    from mpntrackseg_b200.data.mot_graph import Graph
    from mpntrackseg_b200.tracker.mpn_tracker import MPNTracker
    from mpntrackseg_b200.utils.evaluation import compute_constr_satisfaction_rate
    gold = dict(np.load(os.path.join(os.path.dirname(__file__), 'golden', 'rounding.npz')))
    n = int(gold[f'n_{tag}'])
    ei = torch.from_numpy(gold[f'edge_index_{tag}'].astype(np.int64)).to(dev())
    preds = torch.from_numpy(gold[f'preds_{tag}']).to(dev())
    go = Graph(x=torch.zeros(n, 1, device=dev()), edge_index=ei, edge_preds=preds.clone())
    # statistics of the plain rounding on the both-directions edge list (undirected_edges=True)
    r0 = (preds > 0.5).float()
    both = Graph(x=go.x, edge_index=torch.cat((ei, ei.flip(0)), dim=1))
    rate_u, fin, fout = compute_constr_satisfaction_rate(both, torch.cat((r0, r0)), undirected_edges=True, return_flow_vals=True)
    assert rate_u == float(gold[f'rate_undirected_{tag}'])
    assert np.array_equal(fin.cpu().numpy(), gold[f'flow_in_{tag}']) and np.array_equal(fout.cpu().numpy(), gold[f'flow_out_{tag}'])
    with pytest.raises(ValueError):
        compute_constr_satisfaction_rate(go, preds, undirected_edges=False)             # not binarised
    # the tracker's two steps
    tr = MPNTracker(eval_params={'rounding_method': 'greedy'})
    tr.full_graph = SimpleNamespace(graph_obj=go)
    tr._project_graph_model_output()
    assert tr.full_graph.constr_satisf_rate == float(gold[f'rate_{tag}'])
    assert np.array_equal(go.edge_preds.cpu().numpy(), gold[f'round_{tag}'])
    rate_after, fin, fout = compute_constr_satisfaction_rate(go, go.edge_preds, undirected_edges=False, return_flow_vals=True)
    assert rate_after == 1.0 and float(fin.max()) <= 1 and float(fout.max()) <= 1
    labels = tr._assign_ped_ids()
    assert np.array_equal(labels.cpu().numpy(), gold[f'labels_{tag}'])
    # components of an arbitrary (not path-shaped) edge set, shuffled edge order
    perm = torch.randperm(ei.shape[1], generator=torch.Generator().manual_seed(3)).to(dev())
    lab2, ncomp = ops.connected_components(ei[:, perm], r0[perm], n)
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    m = r0.cpu().numpy() == 1
    ref_n, ref_l = connected_components(csr_matrix((np.ones(int(m.sum()), dtype=int), tuple(ei.cpu().numpy()[:, m])), shape=(n, n)),
                                        directed=False, return_labels=True)
    assert ncomp == ref_n and np.array_equal(lab2.cpu().numpy(), ref_l)


def test_graphed_training_step_continues_like_the_eager_one():
    """CoreTrainer.graphed_step (the whole step as one CUDA-graph replay, Adam step counter on the device) produces
    the same parameters as the eager train_step after the same number of steps."""
    from mpntrackseg_b200.training import CoreTrainer
    c = load_case('tiny_nonrecip')
    win, gold = c['win'], c['gold']
    data = Data()
    data.x = win.x.to(dev())
    data.edge_index = torch.from_numpy(gold['edge_index'].astype(np.int64)).to(dev())
    data.edge_attr = torch.from_numpy(gold['edge_attr']).to(dev())
    labels = (win.ident[gold['edge_index'][0]] == win.ident[gold['edge_index'][1]]).float().to(dev())
    trainers = []
    for _ in range(2):
        model = make_model(c['mp'], c['P'])
        model.train()
        trainers.append(CoreTrainer(model))
    losses = [[], []]
    for _ in range(4):
        losses[0].append(float(trainers[0].train_step(data, labels)))
        losses[1].append(float(trainers[1].graphed_step(data, labels)))
    torch.cuda.synchronize()
    assert trainers[0].t == trainers[1].t == 4
    np.testing.assert_allclose(losses[1], losses[0], rtol=1e-6)
    assert losses[0][-1] < losses[0][0]
    assert torch.equal(trainers[0].flat, trainers[1].flat)


# ------------------------------------------------------------------ property tests (hypothesis)
def _hyp():
    hyp = pytest.importorskip('hypothesis')
    return hyp, hyp.strategies


def test_property_knn_mask_equals_oracle_on_random_windows():
    """get_knn_mask on random small windows (random sizes, k, reciprocity, duplicated embeddings -> exact ties):
    the CUDA mask equals the oracle's bit for bit."""
    hyp, st = _hyp()
    from mpntrackseg_b200.utils.graph import get_knn_mask

    @hyp.settings(max_examples=25, deadline=None, derandomize=True)
    @hyp.given(t=st.integers(2, 6), d=st.integers(1, 9), k=st.integers(1, 12), recip=st.booleans(), sym=st.booleans(),
               dup=st.booleans(), seed=st.integers(0, 10_000))
    def run(t, d, k, recip, sym, dup, seed):
        g = torch.Generator().manual_seed(seed)
        n = t * d
        frame = torch.arange(t).repeat_interleave(d)
        reid = torch.randn(n, 32, generator=g)
        if dup and n > 3:
            reid[n // 2] = reid[0]                                                   # exact ties at some k boundary
            reid[n - 1] = reid[1]
        pairs = graph_ref.time_valid_pairs(frame, 'max')
        if pairs.shape[1] == 0:
            return
        dist = graph_ref.pair_reid_dist(reid, pairs)
        if sym:
            pairs, dist = torch.cat((pairs, pairs.flip(0)), dim=1), torch.cat((dist, dist))
        ref = graph_ref.knn_keep_mask(dist, pairs, n, k, recip, symmetric_edges=sym)
        got = get_knn_mask(dist, pairs, n, k, use_cuda=True, reciprocal_k_nns=recip, symmetric_edges=sym)
        assert torch.equal(got.cpu(), ref)

    run()


def test_property_greedy_projection_and_components_on_random_graphs():
    """Random prediction graphs: the projection is feasible (every flow <= 1), only switches edges off, keeps every
    edge of a node that was feasible to begin with unless its other endpoint forced it off, is deterministic; the
    component labels equal scipy's for any edge order."""
    hyp, st = _hyp()
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    from mpntrackseg_b200 import ops

    @hyp.settings(max_examples=25, deadline=None, derandomize=True)
    @hyp.given(n=st.integers(2, 60), dens=st.floats(0.02, 0.6), seed=st.integers(0, 10_000))
    def run(n, dens, seed):
        g = torch.Generator().manual_seed(seed)
        ii, jj = torch.triu_indices(n, n, offset=1)
        keep = torch.rand(ii.numel(), generator=g) < dens
        if int(keep.sum()) == 0:
            return
        ei = torch.stack((ii[keep], jj[keep])).to(dev())
        preds = (torch.rand(ei.shape[1], generator=g).round(decimals=1)).to(dev())        # many exact ties
        r1, rate = ops.greedy_project(ei, preds, n)
        r2, _ = ops.greedy_project(ei, preds, n)
        assert torch.equal(r1, r2)
        assert bool(((r1 == 0) | (preds > 0.5)).all())                                   # nothing is switched on
        _, fin, fout = ops.constr_satisfaction(ei, r1, n, undirected_edges=False)
        assert float(fin.max()) <= 1 and float(fout.max()) <= 1
        r0 = (preds > 0.5).float()
        rate0, fin0, fout0 = ops.constr_satisfaction(ei, r0, n, undirected_edges=False)
        assert rate == rate0
        untouched = (fout0[ei[0]] <= 1) & (fin0[ei[1]] <= 1)                              # both constraints fine initially
        assert torch.equal(r1[untouched], r0[untouched])
        perm = torch.randperm(ei.shape[1], generator=g).to(dev())
        labels, ncomp = ops.connected_components(ei[:, perm], r1[perm], n)
        m = r1.cpu().numpy() == 1
        ref_n, ref_l = connected_components(csr_matrix((np.ones(int(m.sum()), dtype=int), tuple(ei.cpu().numpy()[:, m])), shape=(n, n)),
                                            directed=False, return_labels=True)
        assert ncomp == ref_n and np.array_equal(labels.cpu().numpy(), ref_l)

    run()
