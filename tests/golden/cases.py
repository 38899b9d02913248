"""Golden-case definitions shared by make_golden.py (writer, needs the reference) and the
tests (readers, need only the committed .npz files).  Inputs and weights are regenerated
from seeds through mpntrackseg_b200.synth; fixtures hold the reference's outputs."""
import hashlib
import os
import zipfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

# fixtures that would be larger than 1 MB as plain .npz files; make_golden.py writes them with save_compact
COMPACT = ('config1', 'kitti_shape', 'config5')
# graph arrays of a compact fixture are stored as digests: the oracle rebuilds them bit for bit from the seeded inputs
GRAPH_KEYS = ('edge_index', 'edge_attr', 'edge_attr_sample')
_GRAPHS = {}

CASES = {
    # name: window kwargs, dataset kwargs, model steps, weight seed/gain, extras
    'tiny_full': dict(win=dict(T=5, D=8, k=6, seed=11, node_feats='full', with_ext=True),
                      ds=dict(top_k_nns=6, frames_per_graph=5), steps=(4, 3), wseed=3, gain=2.45,
                      full=True),
    'tiny_nonrecip': dict(win=dict(T=6, D=7, k=5, seed=12, node_feats='pooled'),
                          ds=dict(top_k_nns=5, frames_per_graph=6, reciprocal_k_nns=False),
                          steps=(3, 3), wseed=4, gain=2.4, max_frame_dist=3),
    'config1': dict(win=dict(T=15, D=30, k=50, seed=1, node_feats='pooled', with_ext=True),
                    ds=dict(top_k_nns=50, frames_per_graph=15), steps=(12, 11), wseed=5, gain=1.37,
                    full=True),
    'kitti_shape': dict(win=dict(T=20, D=8, k=100, seed=2, node_feats='pooled'),
                        ds=dict(top_k_nns=100, frames_per_graph=20), steps=(12, 11), wseed=6,
                        gain=0.95),
    # non-default model options (models/mpn.py:263-273 node_agg_fn; models/mlp.py:14-21 BatchNorm1d / Dropout, eval mode)
    'tiny_mean': dict(win=dict(T=6, D=7, k=5, seed=14, node_feats='pooled'), ds=dict(top_k_nns=5, frames_per_graph=6),
                      steps=(4, 3), wseed=9, gain=2.6, model=dict(node_agg_fn='mean')),
    'tiny_max': dict(win=dict(T=6, D=7, k=5, seed=15, node_feats='pooled'), ds=dict(top_k_nns=5, frames_per_graph=6),
                     steps=(4, 3), wseed=10, gain=2.6, model=dict(node_agg_fn='max')),
    'tiny_bn': dict(win=dict(T=6, D=7, k=5, seed=16, node_feats='pooled'), ds=dict(top_k_nns=5, frames_per_graph=6),
                    steps=(4, 3), wseed=11, gain=2.0, model=dict(batchnorm=True, dropout_p=0.3)),
    'steps0': dict(win=dict(T=4, D=6, k=4, seed=13, node_feats='pooled'),
                   ds=dict(top_k_nns=4, frames_per_graph=4), steps=(0, 0), wseed=7, gain=1.0),
}

# large cases, fixtures hold a reduced set of outputs (see make_golden.run_config5_case / run_big_window_case)
BIG_CASES = {
    'config5': dict(win=dict(T=15, D=300, k=100, seed=5, node_feats='pooled', node_dim=2048, min_gap=2e-6), ds=dict(top_k_nns=100, frames_per_graph=15),
                    steps=(12, 11), wseed=12, gain=1.15),
    'big_window': dict(win=dict(T=15, D=360, k=20, seed=6, node_feats='pooled', node_dim=8, min_gap=2e-6), ds=dict(top_k_nns=20, frames_per_graph=15)),
}

TRACKER_CASE = dict(win=dict(T=9, D=9, k=7, seed=21, node_feats='pooled'),
                    ds=dict(top_k_nns=7, frames_per_graph=5), steps=(4, 3), wseed=8, gain=2.2)


def case_model_params(c):
    """graph_model_params of a case: the shipped widths with the case's step counts and option overrides."""
    from mpntrackseg_b200.config import default_graph_model_params
    mp = default_graph_model_params(*c['steps'])
    over = c.get('model', {})
    if 'node_agg_fn' in over:
        mp['node_agg_fn'] = over['node_agg_fn']
    for k in ('encoder_feats_dict', 'edge_model_feats_dict', 'node_model_feats_dict', 'classifier_feats_dict'):
        if over.get('batchnorm'):
            mp[k]['use_batchnorm'] = True
        if 'dropout_p' in over:
            mp[k]['dropout_p'] = over['dropout_p']
    return mp


def checksum(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(np.ascontiguousarray(t.detach().cpu().numpy() if torch.is_tensor(t) else t).tobytes())
    return h.hexdigest()


def save_compact(path, **arrays):
    """``np.savez_compressed`` for the COMPACT fixtures, without dropping anything.  A graph array (GRAPH_KEYS) is
    stored as the SHA-256 of the reference's array (``<key>__sha256``); the loaders rebuild it with the oracle and
    require the same digest.  A float32 array is stored as its four byte planes (``<key>__planes``, uint8
    [4, *shape]), which LZMA compresses much better than interleaved bytes."""
    with zipfile.ZipFile(path, 'w', zipfile.ZIP_LZMA) as zf:
        for key, a in arrays.items():
            a = np.asarray(a)
            if key in GRAPH_KEYS:
                key, a = f'{key}__sha256', np.array(checksum(a))
            elif a.dtype == np.float32 and a.ndim:
                key, a = f'{key}__planes', np.moveaxis(np.ascontiguousarray(a)[..., None].view(np.uint8), -1, 0)
            with zf.open(f'{key}.npy', 'w') as f:
                np.lib.format.write_array(f, a)


def _load_gold(name):
    """The arrays of ``<name>.npz``, float32 byte planes (see save_compact) joined back."""
    gold = {}
    with np.load(os.path.join(HERE, f'{name}.npz')) as z:
        for key in z.files:
            if key.endswith('__planes'):
                gold[key[:-8]] = np.ascontiguousarray(np.moveaxis(z[key], 0, -1)).view(np.float32)[..., 0]
            else:
                gold[key] = z[key]
    return gold


def _rebuild_graph(name, gold, win, ds, max_frame_dist):
    """Replace the ``<key>__sha256`` entries of a compact fixture by the oracle's graph arrays, which must have the
    reference's digests (the oracle builds the graph with the reference's own torch ops, bit for bit)."""
    for key in [k for k in gold if k.endswith('__sha256')]:
        if name not in _GRAPHS:
            from mpntrackseg_b200 import synth
            from oracle import graph_ref
            g = graph_ref.build_graph(win.frame, win.reid, synth.det_columns(win), win.fps, ds, inference_mode=False,
                                      max_frame_dist=max_frame_dist)
            ea = g['edge_attr'].numpy()
            # dtypes and the feature sample stride as make_golden.py stores them
            _GRAPHS[name] = dict(edge_index=g['edge_index'].numpy().astype(np.int32), edge_attr=ea,
                                 edge_attr_sample=ea[::16])
        arr = _GRAPHS[name][key[:-8]].copy()
        assert checksum(arr) == str(gold.pop(key)), f"{name}: the oracle's {key[:-8]} differs from the reference's"
        gold[key[:-8]] = arr


def load_case(name):
    """Rebuild the seeded inputs / weights of a golden case and load its reference outputs."""
    from mpntrackseg_b200 import synth
    from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
    c = TRACKER_CASE if name == 'tracker_window' else CASES[name]
    gold = _load_gold(name)
    win = synth.make_window(**c['win'])
    assert checksum(win.frame, win.reid, win.x, win.bb_height, win.feet_x) == str(gold['input_checksum']), \
        'seeded inputs differ from the ones the fixture was generated with'
    ds = default_dataset_params(**c['ds'])
    _rebuild_graph(name, gold, win, ds, c.get('max_frame_dist', 'max'))
    mp = case_model_params(c)
    P = synth.make_params(mp, seed=c['wseed'], gain=c['gain'])
    key = [k for k in P if k.startswith('classifier.edge_model') and k.endswith('bias')][-1]
    P[key] = P[key] - float(gold['bias_shift'])
    assert checksum(*P.values()) == str(gold['param_checksum'])
    return dict(case=c, win=win, ds=ds, mp=mp, P=P, gold=gold,
                max_frame_dist=c.get('max_frame_dist', 'max'))


def load_big_case(name):
    """Seeded inputs (and weights) of a BIG_CASES entry + its reduced reference outputs."""
    from mpntrackseg_b200 import synth
    from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
    c = BIG_CASES[name]
    gold = _load_gold(name)
    win = synth.make_window(**c['win'])
    ds = default_dataset_params(**c['ds'])
    out = dict(case=c, win=win, ds=ds, gold=gold)
    if 'steps' in c:
        assert checksum(win.frame, win.reid, win.x, win.bb_height, win.feet_x) == str(gold['input_checksum'])
        _rebuild_graph(name, gold, win, ds, 'max')
        mp = default_graph_model_params(*c['steps'])
        P = synth.make_params(mp, seed=c['wseed'], gain=c['gain'])
        key = [k for k in P if k.startswith('classifier.edge_model') and k.endswith('bias')][-1]
        P[key] = P[key] - float(gold['bias_shift'])
        assert checksum(*P.values()) == str(gold['param_checksum'])
        out.update(mp=mp, P=P)
    else:
        assert checksum(win.frame, win.reid, win.bb_height, win.feet_x) == str(gold['input_checksum'])
    return out
