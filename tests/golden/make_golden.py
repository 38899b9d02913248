"""Generate tests/golden/*.npz by running the UNMODIFIED reference on seeded inputs.

Run in the build container only (needs /root/reference; the GPU box does not have it):

    python tests/golden/make_golden.py

The reference modules ``mot_neural_solver.models.mpn`` and ``mot_neural_solver.utils.graph``
are imported from /root/reference/src with the pure-torch ``torch_scatter`` stand-in of
``tests/golden/torch_scatter_stub`` (the only import they miss in this image).  Inputs and
weights come from ``mpntrackseg_b200.synth`` (seeded), so the fixtures hold outputs only,
plus an input checksum that the tests re-verify.  ``data/mot_graph.py`` and
``tracker/mpn_tracker.py`` cannot be imported here (torch_geometric / pycocotools are
absent); their <=35 lines of glue around the imported functions are applied inline below,
line-cited.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, 'torch_scatter_stub'))
sys.path.insert(0, '/root/reference/src')

import pandas as pd  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from mot_neural_solver.models.mpn import MOTMPNet as RefMOTMPNet  # noqa: E402
from mot_neural_solver.utils.graph import (  # noqa: E402
    compute_edge_feats_dict, get_knn_mask, get_time_valid_conn_ixs, to_lightweight_graph, to_undirected_graph)

from mpntrackseg_b200 import synth  # noqa: E402
from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params  # noqa: E402

from cases import BIG_CASES, CASES, COMPACT, TRACKER_CASE, case_model_params, checksum, save_compact  # noqa: E402


def det_df(win):
    return pd.DataFrame(synth.det_columns(win))


def ref_build_graph(win, ds, inference_mode, max_frame_dist):
    """Inline of MOTGraph._get_edge_ixs + construct_graph_object around the imported
    reference functions (reference: data/mot_graph.py:206-219, 292-312)."""
    df = det_df(win)
    edge_ixs = get_time_valid_conn_ixs(frame_num=win.frame, max_frame_dist=max_frame_dist,
                                       use_cuda=False)
    n_cand = edge_ixs.shape[1]
    if not inference_mode and ds['top_k_nns'] is not None:
        d = F.pairwise_distance(win.reid[edge_ixs[0]], win.reid[edge_ixs[1]])
        keep = get_knn_mask(pwise_dist=d, edge_ixs=edge_ixs, num_nodes=win.N,
                            top_k_nns=ds['top_k_nns'], reciprocal_k_nns=ds['reciprocal_k_nns'],
                            symmetric_edges=False, use_cuda=False)
        edge_ixs = edge_ixs.T[keep].T
    fd = compute_edge_feats_dict(edge_ixs=edge_ixs, det_df=df, fps=win.fps, use_cuda=False)
    feats = torch.stack([fd[n] for n in ds['edge_feats_to_use'] if n in fd]).T
    emb = []
    for i in range(0, edge_ixs[0].shape[0], 50000):
        emb.append(F.pairwise_distance(win.reid[edge_ixs[0][i:i + 50000]],
                                       win.reid[edge_ixs[1][i:i + 50000]]).view(-1, 1))
    emb = torch.cat(emb, dim=0)
    if 'emb_dist' in ds['edge_feats_to_use']:
        feats = torch.cat((feats, emb), dim=1)
    edge_attr = torch.cat((feats, feats), dim=0)
    edge_index = torch.cat((edge_ixs, torch.stack((edge_ixs[1], edge_ixs[0]))), dim=1)
    dists = torch.cat((emb, emb)).view(-1) if inference_mode else None
    return n_cand, edge_index, edge_attr, dists


def centred_params(mp, wseed, gain, ref_model, data):
    """Weights from synth.make_params, classifier bias shifted so that the last step's
    logits have median 0 (SURVEY.md H3: default-init logits never cross 0)."""
    P = synth.make_params(mp, seed=wseed, gain=gain)
    ref_model.load_state_dict(P, strict=True)
    with torch.no_grad():
        last = core_forward(ref_model, data)['classified_edges'][-1]
    shift = float(last.median())
    key = [k for k in P if k.startswith('classifier.edge_model') and k.endswith('bias')][-1]
    P[key] = P[key] - shift
    ref_model.load_state_dict(P, strict=True)
    return P, shift


def core_forward(model, data):
    """The reference forward restricted to the modules the edge logits depend on: the
    same sub-module calls, in the same order, as MOTMPNet.forward
    (reference: models/mpn.py:351-381 minus the x_ext / mask lines 356,373,377(ext),384-385)."""
    x = model.global_avgpool(data.x).view(data.x.size(0), -1)
    e_lat, x_lat = model.encoder(data.edge_attr, x)
    e0, x0 = e_lat, x_lat
    first = model.num_enc_steps - model.num_class_steps + 1
    out = {'classified_edges': []}
    for step in range(1, model.num_enc_steps + 1):
        e_lat = torch.cat((e0, e_lat), dim=1)
        x_lat = torch.cat((x0, x_lat), dim=1)
        x_lat, e_lat = model.MPNet(x_lat, data.edge_index, e_lat)
        dec, _ = model.classifier(e_lat)
        if step >= first:
            out['classified_edges'].append(dec)
    if model.num_enc_steps == 0:
        dec, _ = model.classifier(e_lat)
        out['classified_edges'].append(dec)
    out['node_state'], out['edge_state'] = x_lat, e_lat
    return out


class Data:
    pass


def run_case(name, c):
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    mp = case_model_params(c)
    mfd = c.get('max_frame_dist', 'max')
    n_cand, edge_index, edge_attr, _ = ref_build_graph(win, ds, False, mfd)
    data = Data()
    data.x, data.edge_index, data.edge_attr = win.x, edge_index, edge_attr
    data.x_ext = win.x_ext
    torch.manual_seed(0)
    model = RefMOTMPNet(mp).eval()
    P, shift = centred_params(mp, c['wseed'], c['gain'], model, data)
    with torch.no_grad():
        core = core_forward(model, data)
        logits = torch.stack([t.view(-1) for t in core['classified_edges']])
        out = dict(
            n_candidates=np.int64(n_cand),
            edge_index=edge_index.numpy().astype(np.int32),
            edge_attr=edge_attr.numpy(),
            logits=logits.numpy(),
            node_state=core['node_state'].numpy(), edge_state=core['edge_state'].numpy(),
            bias_shift=np.float64(shift),
            input_checksum=checksum(win.frame, win.reid, win.x, win.bb_height, win.feet_x),
            param_checksum=checksum(*P.values()))
        if c.get('full'):
            full = model(data)                                   # the reference's own forward
            fl = torch.stack([t.view(-1) for t in full['classified_edges']])
            assert torch.equal(fl, logits), 'core sub-module loop != MOTMPNet.forward logits'
            m = full['mask_predictions'][-1]
            out['mask_last_sample'] = m[:, 0, ::7, ::7].numpy()
            out['mask_step_means'] = np.array([float(t.double().mean()) for t in full['mask_predictions']])
    stats = dict(N=win.N, E=edge_index.shape[1], cand=n_cand,
                 logit_std=float(logits[-1].std()) if logits.numel() else 0.0,
                 frac_pos=float((logits[-1] > 0).float().mean()) if logits.numel() else 0.0)
    print(name, stats)
    (save_compact if name in COMPACT else np.savez_compressed)(os.path.join(HERE, f'{name}.npz'), **out)


def run_tracker_case():
    """Whole-sequence graph without KNN, then one sliding window pruned and evaluated the
    way MPNTracker does (reference: tracker/mpn_tracker.py:80-84,167-179,107-135)."""
    c = TRACKER_CASE
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    mp = default_graph_model_params(*c['steps'])
    fpg = ds['frames_per_graph']
    max_frame_dist = 1 * (fpg - 1)                                       # mpn_tracker.py:80-81
    n_cand, edge_index, edge_attr, dists = ref_build_graph(win, ds, True, max_frame_dist)
    frames = torch.unique(win.frame)
    start, end = int(frames[2]), int(frames[2 + fpg - 1])
    nodes_mask = (start <= win.frame) & (win.frame <= end)               # mpn_tracker.py:171
    edges_mask = nodes_mask[edge_index[0]] & nodes_mask[edge_index[1]]   # mpn_tracker.py:172-173
    first = int(torch.nonzero(nodes_mask)[0])
    sub_ei = edge_index.T[edges_mask].T - first                          # mpn_tracker.py:179
    sub_attr, sub_d = edge_attr[edges_mask], dists[edges_mask]
    n_sub = int(nodes_mask.sum())
    keep = get_knn_mask(pwise_dist=sub_d, edge_ixs=sub_ei, num_nodes=n_sub, top_k_nns=ds['top_k_nns'],
                        use_cuda=False, reciprocal_k_nns=ds['reciprocal_k_nns'], symmetric_edges=True)
    data = Data()
    data.x, data.x_ext = win.x[nodes_mask], None
    data.edge_index, data.edge_attr = sub_ei.T[keep].T, sub_attr[keep]
    model = RefMOTMPNet(mp).eval()
    P, shift = centred_params(mp, c['wseed'], c['gain'], model, data)
    with torch.no_grad():
        core = core_forward(model, data)
    pruned = torch.sigmoid(core['classified_edges'][-1].view(-1))        # mpn_tracker.py:129
    preds = torch.zeros(keep.shape[0])
    preds[keep] = pruned                                                 # mpn_tracker.py:133-134
    print('tracker_window', dict(N=win.N, E_full=edge_index.shape[1], n_sub=n_sub,
                                 E_sub=int(edges_mask.sum()), kept=int(keep.sum()),
                                 logit_std=float(core['classified_edges'][-1].std())))
    np.savez_compressed(
        os.path.join(HERE, 'tracker_window.npz'),
        n_candidates=np.int64(n_cand), full_edge_index=edge_index.numpy().astype(np.int32),
        full_edge_attr=edge_attr.numpy(), full_dists=dists.numpy(),
        window=np.array([start, end]), keep=keep.numpy(), edge_preds=preds.numpy(),
        bias_shift=np.float64(shift),
        input_checksum=checksum(win.frame, win.reid, win.x, win.bb_height, win.feet_x),
        param_checksum=checksum(*P.values()))


def run_edge_labels_case():
    """Edge labels ('closest' and 'all') of the config1 training graph, computed the way
    MOTGraph.assign_edge_labels does (reference: data/mot_graph.py:228-259) with the torch_scatter stand-in's
    scatter_min; every 7th detection is turned into a false positive (id -1)."""
    from torch_scatter import scatter_min
    c = CASES['config1']
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    _, edge_index, _, _ = ref_build_graph(win, ds, False, c.get('max_frame_dist', 'max'))
    ids = win.ident.clone().long()
    ids[::7] = -1
    per_edge_ids = torch.stack([ids[edge_index[0]], ids[edge_index[1]]])                      # :230
    same_id = (per_edge_ids[0] == per_edge_ids[1]) & (per_edge_ids[0] != -1)                  # :231
    out = {}
    lab_all = torch.zeros_like(same_id, dtype=torch.float)
    lab_all[same_id] = 1                                                                      # :235
    out['labels_all'] = lab_all.numpy()
    labels = torch.zeros_like(same_id, dtype=torch.float)
    same_ids_ixs = torch.where(same_id)
    se = edge_index.T[same_id].T
    time_dists = torch.abs(se[0] - se[1])                                                     # :240
    active = torch.zeros(se.shape[1], dtype=torch.bool)
    for mask in (se[0] < se[1], se[0] > se[1]):                                               # :243, :252
        arg = scatter_min(time_dists[mask], se[0][mask], dim=0, dim_size=win.N)[1]            # :244-245, :253-254
        orig = torch.cat((se[1][mask], torch.as_tensor([-1])))                                # :246-247
        active |= orig[arg][se[0]] == se[1]                                                   # :248-249
    labels[same_ids_ixs[0][active]] = 1                                                       # :258-259
    out['labels_closest'] = labels.numpy()
    print('edge_labels', dict(E=edge_index.shape[1], same_id=int(same_id.sum()), closest=int(labels.sum())))
    np.savez_compressed(os.path.join(HERE, 'edge_labels.npz'), **out, edge_index=edge_index.numpy().astype(np.int32),
                        ids=ids.numpy())


class _GraphObj:
    """The attribute bag the reference's to_undirected_graph / to_lightweight_graph work on."""

    def device(self):
        return torch.device('cpu')


class _MotGraph:
    pass


def run_tracker_sequence_case():
    """All sliding windows of the TRACKER_CASE sequence, averaged per edge, then merged to an undirected
    graph and pruned at 0.5 -- the loop of MPNTracker._evaluate_graph_in_batches
    (reference: tracker/mpn_tracker.py:153-207) inlined around the imported reference functions, with the
    weights of the tracker_window fixture.  Stored for both settings of set_pruned_edges_to_inactive."""
    c = TRACKER_CASE
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    mp = default_graph_model_params(*c['steps'])
    fpg = ds['frames_per_graph']
    n_cand, edge_index, edge_attr, dists = ref_build_graph(win, ds, True, 1 * (fpg - 1))
    gold_w = dict(np.load(os.path.join(HERE, 'tracker_window.npz')))
    P = synth.make_params(mp, seed=c['wseed'], gain=c['gain'])
    key = [k for k in P if k.startswith('classifier.edge_model') and k.endswith('bias')][-1]
    P[key] = P[key] - float(gold_w['bias_shift'])
    assert checksum(*P.values()) == str(gold_w['param_checksum'])
    model = RefMOTMPNet(mp).eval()
    model.load_state_dict(P, strict=True)
    all_frames = np.array(sorted(set(win.frame.tolist())))
    frame_num_per_node = win.frame
    node_names = torch.arange(win.N)
    out = {}
    for inactive in (False, True):
        overall = torch.zeros(edge_index.shape[1])
        num = overall.clone()
        for start_frame, end_frame in zip(all_frames, all_frames[fpg - 1:]):                  # :167
            nodes_mask = (start_frame <= frame_num_per_node) & (frame_num_per_node <= end_frame)
            edges_mask = nodes_mask[edge_index[0]] & nodes_mask[edge_index[1]]
            sub_ei = edge_index.T[edges_mask].T - node_names[nodes_mask][0]
            sub_attr, sub_d = edge_attr[edges_mask], dists[edges_mask]
            knn_mask = get_knn_mask(pwise_dist=sub_d, edge_ixs=sub_ei, num_nodes=int(nodes_mask.sum()),
                                    top_k_nns=ds['top_k_nns'], use_cuda=False,
                                    reciprocal_k_nns=ds['reciprocal_k_nns'], symmetric_edges=True)   # :107-110
            data = Data()
            data.x, data.x_ext = win.x[nodes_mask], None
            data.edge_index, data.edge_attr = sub_ei.T[knn_mask].T, sub_attr[knn_mask]
            with torch.no_grad():
                core = core_forward(model, data)
            pruned = torch.sigmoid(core['classified_edges'][-1].view(-1))                     # :129
            edge_preds = torch.zeros(knn_mask.shape[0])
            edge_preds[knn_mask] = pruned                                                     # :133-134
            pred_mask = torch.ones_like(knn_mask) if inactive else knn_mask                   # :137-141
            overall[edges_mask] += edge_preds                                                 # :195
            num[torch.where(edges_mask)[0][pred_mask]] += 1                                   # :197
        final = overall / num                                                                 # :203
        final[torch.isnan(final)] = 0
        g = _MotGraph()
        g.graph_obj = _GraphObj()
        g.graph_obj.edge_index, g.graph_obj.edge_preds, g.graph_obj.num_nodes = edge_index.clone(), final.clone(), win.N
        to_undirected_graph(g, attrs_to_update=('edge_preds', 'edge_labels'))                 # :206
        und_ei, und_p = g.graph_obj.edge_index.clone(), g.graph_obj.edge_preds.clone()
        to_lightweight_graph(g)                                                               # :207
        tag = 'inactive' if inactive else 'knn'
        out[f'directed_preds_{tag}'] = final.numpy()
        out[f'undirected_edge_index_{tag}'] = und_ei.numpy().astype(np.int32)
        out[f'undirected_preds_{tag}'] = und_p.numpy()
        out[f'light_edge_index_{tag}'] = g.graph_obj.edge_index.numpy().astype(np.int32)
        out[f'light_preds_{tag}'] = g.graph_obj.edge_preds.numpy()
        print('tracker_sequence', tag, dict(windows=len(all_frames) - fpg + 1, E_full=edge_index.shape[1],
                                            undirected=und_ei.shape[1], kept=int(g.graph_obj.edge_index.shape[1]),
                                            never_predicted=int((num == 0).sum())))
    np.savez_compressed(os.path.join(HERE, 'tracker_sequence.npz'), **out,
                        input_checksum=gold_w['input_checksum'], param_checksum=gold_w['param_checksum'])


def ref_build_graph_chunked(win, ds):
    """ref_build_graph for windows whose 9-14 M candidate pairs do not fit an un-chunked gather: the pair distances are
    evaluated in chunks of 50 000 (the reference's own inference-mode loop, data/mot_graph.py:299-303; a pair's distance
    does not depend on its chunk)."""
    edge_ixs = get_time_valid_conn_ixs(frame_num=win.frame, max_frame_dist='max', use_cuda=False)
    n_cand = edge_ixs.shape[1]
    d = torch.cat([F.pairwise_distance(win.reid[edge_ixs[0][i:i + 50000]], win.reid[edge_ixs[1][i:i + 50000]])
                   for i in range(0, n_cand, 50000)])
    keep = get_knn_mask(pwise_dist=d, edge_ixs=edge_ixs, num_nodes=win.N, top_k_nns=ds['top_k_nns'],
                        reciprocal_k_nns=ds['reciprocal_k_nns'], symmetric_edges=False, use_cuda=False)
    edge_ixs, d = edge_ixs.T[keep].T, d[keep]
    fd = compute_edge_feats_dict(edge_ixs=edge_ixs, det_df=det_df(win), fps=win.fps, use_cuda=False)
    feats = torch.stack([fd[n] for n in ds['edge_feats_to_use'] if n in fd]).T
    feats = torch.cat((feats, d.view(-1, 1)), dim=1)
    return n_cand, torch.cat((edge_ixs, torch.stack((edge_ixs[1], edge_ixs[0]))), dim=1), torch.cat((feats, feats), dim=0)


def run_config5_case():
    """BASELINE.json configs[4]: dense crowd window, 15 frames x 300 detections, k = 100 (N = 4,500, E ~ 195 k).  The
    fixture keeps the edge list, a strided sample of the edge features and the logits of the last step (+ per-step
    means), not all 11 x E logits."""
    c = BIG_CASES['config5']
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    mp = default_graph_model_params(*c['steps'])
    n_cand, edge_index, edge_attr = ref_build_graph_chunked(win, ds)
    data = Data()
    data.x, data.edge_index, data.edge_attr, data.x_ext = win.x, edge_index, edge_attr, None
    model = RefMOTMPNet(mp).eval()
    P, shift = centred_params(mp, c['wseed'], c['gain'], model, data)
    with torch.no_grad():
        core = core_forward(model, data)
    logits = torch.stack([t.view(-1) for t in core['classified_edges']])
    print('config5', dict(N=win.N, E=edge_index.shape[1], cand=n_cand, logit_std=float(logits[-1].std()),
                          frac_pos=float((logits[-1] > 0).float().mean()), node_max=float(core['node_state'].max())))
    save_compact(os.path.join(HERE, 'config5.npz'), n_candidates=np.int64(n_cand),
                 edge_index=edge_index.numpy().astype(np.int32), edge_attr_sample=edge_attr[::16].numpy(),
                 logits_last=logits[-1].numpy(), logits_first=logits[0].numpy(),
                 logits_step_means=logits.double().mean(dim=1).numpy(), bias_shift=np.float64(shift),
                 input_checksum=checksum(win.frame, win.reid, win.x, win.bb_height, win.feet_x),
                 param_checksum=checksum(*P.values()))


def run_big_window_case():
    """A window of 5,400 detections (> 5,120: the batched builder's streamed row select): kept pairs only."""
    c = BIG_CASES['big_window']
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    n_cand, edge_index, edge_attr = ref_build_graph_chunked(win, ds)
    p = edge_index.shape[1] // 2
    print('big_window', dict(N=win.N, pairs=p, cand=n_cand))
    np.savez_compressed(os.path.join(HERE, 'big_window.npz'), n_candidates=np.int64(n_cand),
                        pairs=edge_index[:, :p].numpy().astype(np.int32), reid_dist_sample=edge_attr[:p:8, 5].numpy(),
                        input_checksum=checksum(win.frame, win.reid, win.bb_height, win.feet_x))


def _reference_function(path, name, glob):
    """Compile ONE function of a reference module that cannot be imported here (its module imports packages that
    are absent) straight from the reference's source file; nothing is copied into the repo."""
    import ast
    src = open(path).read()
    fn = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == name)
    code = compile(ast.Module(body=[fn], type_ignores=[]), path, 'exec')
    exec(code, glob)
    return glob[name]


def _reference_class(path, name, glob):
    import ast
    src = open(path).read()
    cls = next(n for n in ast.parse(src).body if isinstance(n, ast.ClassDef) and n.name == name)
    exec(compile(ast.Module(body=[cls], type_ignores=[]), path, 'exec'), glob)
    return glob[name]


def run_rounding_case():
    """Rounding + identity assignment (SURVEY.md f2) by the reference's own code on seeded sequence graphs:
    compute_constr_satisfaction_rate (utils/evaluation.py:370-414) and GreedyProjector (tracker/projectors.py:11-67)
    are compiled from their files (the modules import motmetrics / pulp, absent here) with the torch_scatter stand-in;
    the identities come from scipy's connected_components as in tracker/mpn_tracker.py:231-248."""
    from types import SimpleNamespace
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components
    from torch_scatter import scatter_add
    csr = _reference_function('/root/reference/src/mot_neural_solver/utils/evaluation.py', 'compute_constr_satisfaction_rate',
                              {'torch': torch, 'scatter_add': scatter_add})
    Greedy = _reference_class('/root/reference/src/mot_neural_solver/tracker/projectors.py', 'GreedyProjector',
                              {'torch': torch, 'scatter_add': scatter_add, 'compute_constr_satisfaction_rate': csr})
    out = {}
    for tag, (T, D, seed, p_link, p_noise) in {'a': (12, 9, 51, 0.9, 0.12), 'b': (30, 25, 52, 0.8, 0.05)}.items():
        g = torch.Generator().manual_seed(seed)
        n = T * D
        frame = torch.arange(T).repeat_interleave(D)
        ident = torch.arange(D).repeat(T)
        ii, jj = torch.triu_indices(n, n, offset=1)
        ok = (frame[jj] > frame[ii]) & (frame[jj] - frame[ii] <= 3)
        ii, jj = ii[ok], jj[ok]
        same = (ident[ii] == ident[jj]) & (frame[jj] - frame[ii] == 1)
        u = torch.rand(ii.numel(), generator=g)
        preds = torch.where(same, 0.55 + 0.45 * torch.rand(ii.numel(), generator=g), 0.5 * torch.rand(ii.numel(), generator=g))
        preds = torch.where(same & (u > p_link), 0.3 * torch.rand(ii.numel(), generator=g), preds)          # missed links
        preds = torch.where(~same & (u < p_noise), 0.5 + 0.5 * torch.rand(ii.numel(), generator=g), preds)  # spurious links
        preds[::7] = preds[::7].round(decimals=1)                                                             # exact ties
        keep = preds > 0.05                                                                                  # a pruned edge list
        edge_index, preds = torch.stack((ii[keep], jj[keep])), preds[keep].float()
        graph_obj = SimpleNamespace(edge_index=edge_index, edge_preds=preds.clone(), num_nodes=n)
        rounded0 = (preds > 0.5).float()
        rate_u, fin_u, fout_u = csr(graph_obj=SimpleNamespace(edge_index=torch.cat((edge_index, edge_index.flip(0)), dim=1),
                                                              num_nodes=n),
                                    edges_out=torch.cat((rounded0, rounded0)), undirected_edges=True, return_flow_vals=True)
        proj = Greedy(SimpleNamespace(graph_obj=graph_obj))
        proj.project()
        final = graph_obj.edge_preds
        mask = (final == 1).numpy()
        nz = edge_index.numpy()[:, mask]
        ncomp, labels = connected_components(csgraph=csr_matrix((final.numpy()[mask].astype(int), (tuple(nz))), shape=(n, n)),
                                             directed=False, return_labels=True)
        print('rounding', tag, dict(N=n, E=edge_index.shape[1], on=int(rounded0.sum()), kept=int(final.sum()),
                                    rate=proj.constr_satisf_rate, comps=ncomp))
        out.update({f'edge_index_{tag}': edge_index.numpy().astype(np.int32), f'preds_{tag}': preds.numpy(),
                    f'round_{tag}': final.numpy(), f'rate_{tag}': np.float64(proj.constr_satisf_rate),
                    f'rate_undirected_{tag}': np.float64(rate_u), f'flow_in_{tag}': fin_u.numpy(), f'flow_out_{tag}': fout_u.numpy(),
                    f'labels_{tag}': labels.astype(np.int64), f'ncomp_{tag}': np.int64(ncomp), f'n_{tag}': np.int64(n)})
    np.savez_compressed(os.path.join(HERE, 'rounding.npz'), **out)


def run_embedding_store_case():
    """Per-frame embedding files in the layout the reference's preprocessing writes, read back by the reference's
    own ``load_precomputed_embeddings`` (utils/rgb.py:150-188; utils/rgb.py itself needs skimage / pycocotools, so
    the function is compiled from the file).  Store layout restated from seq_processor.py:445-446,462-472."""
    import os.path as osp
    import tempfile
    loader = _reference_function('/root/reference/src/mot_neural_solver/utils/rgb.py', 'load_precomputed_embeddings',
                                 {'osp': osp, 'np': np, 'torch': torch})
    g = torch.Generator().manual_seed(31)
    frames = np.array([4, 4, 4, 5, 5, 7, 7, 7, 7], dtype=np.int64)
    det_ids = np.array([10, 11, 12, 13, 14, 15, 16, 17, 18], dtype=np.int64)
    reid = torch.randn(9, 8, generator=g)
    core = torch.randn(9, 6, 8, 4, generator=g)
    tmp = tempfile.mkdtemp()
    seq_info = {'seq_path': tmp, 'det_file_name': 'det'}
    reid_t = torch.cat((torch.from_numpy(det_ids).view(-1, 1).float(), reid), dim=1)                       # :446
    core_t = torch.cat((torch.from_numpy(det_ids).view(-1, 1, 1, 1).float().expand(-1, -1, 8, 4), core), dim=1)   # :445
    for name, t in (('reid', reid_t), ('core', core_t)):
        d = osp.join(tmp, 'processed_data', 'embeddings', 'det', name)
        os.makedirs(d)
        for f in np.unique(frames):                                                                        # :462-472
            torch.save(t[torch.from_numpy(frames == f)], osp.join(d, f'{f}.pt'))
    keep = np.array([0, 2, 3, 5, 6, 8])                       # the window's table: frames 4, 5, 7 with some detections filtered
    df = pd.DataFrame({'frame': frames[keep], 'detection_id': det_ids[keep]})
    out_reid = loader(det_df=df, seq_info_dict=seq_info, embeddings_dir=osp.join('embeddings', 'det', 'reid'), use_cuda=False)
    out_core = loader(det_df=df, seq_info_dict=seq_info, embeddings_dir=osp.join('embeddings', 'det', 'core'), use_cuda=False,
                      embedding_dim='3D')
    sub = df[df.frame != 5]
    out_sub = loader(det_df=sub, seq_info_dict=seq_info, embeddings_dir=osp.join('embeddings', 'det', 'reid'), use_cuda=False)
    np.savez_compressed(os.path.join(HERE, 'embedding_store.npz'), frames=frames, det_ids=det_ids, reid=reid.numpy(),
                        core=core.numpy(), keep=keep, out_reid=out_reid.numpy(), out_core=out_core.numpy(),
                        out_sub=out_sub.numpy(), file_reid_5=torch.load(osp.join(tmp, 'processed_data', 'embeddings', 'det', 'reid', '5.pt')).numpy(),
                        file_core_7=torch.load(osp.join(tmp, 'processed_data', 'embeddings', 'det', 'core', '7.pt')).numpy())
    print('embedding_store', tuple(out_reid.shape), tuple(out_core.shape), tuple(out_sub.shape))


if __name__ == '__main__':
    torch.set_num_threads(os.cpu_count() or 1)
    only = sys.argv[1:]
    for name, case in CASES.items():
        if not only or name in only:
            run_case(name, case)
    if not only or 'tracker_window' in only:
        run_tracker_case()
    if not only or 'tracker_sequence' in only:
        run_tracker_sequence_case()
    if not only or 'edge_labels' in only:
        run_edge_labels_case()
    if not only or 'embedding_store' in only:
        run_embedding_store_case()
    if not only or 'rounding' in only:
        run_rounding_case()
    if 'config5' in only:                       # minutes of CPU time each: only on request
        run_config5_case()
    if 'big_window' in only:
        run_big_window_case()
