"""``Graph`` attribute bag and ``MOTGraph`` edge construction / assembly on the GPU.
reference: src/mot_neural_solver/data/mot_graph.py (Graph :21-83, _get_edge_ixs :195-221,
construct_graph_object :283-316).

The reference's ``Graph`` derives from torch_geometric's ``Data``; only the attribute-bag
behaviour and ``num_nodes`` / ``num_edges`` are used on the hot path, so this one is a plain
object.  ``MOTGraph`` here takes the detection table and the already-loaded appearance
tensors (disk IO of the per-frame ``.pt`` files is outside the hot path).
"""
import numpy as np
import torch

from .. import ops

_DATA_ATTRS = ('x', 'x_ext', 'edge_attr', 'edge_index', 'mask_attr', 'node_names', 'edge_labels',
               'edge_preds', 'reid_emb_dists')


class Graph(object):
    """reference: data/mot_graph.py:21-83"""

    def __init__(self, **kwargs):
        for k, v in kwargs.items():
            setattr(self, k, v)

    @property
    def num_nodes(self):
        if getattr(self, '_num_nodes', None) is not None:        # pinned by to_lightweight_graph before x is dropped
            return self._num_nodes
        return self.x.size(0)

    @num_nodes.setter
    def num_nodes(self, n):
        self._num_nodes = int(n)

    @property
    def num_edges(self):
        return self.edge_index.size(1)

    def _change_attrs_types(self, attr_change_fn):
        for name in _DATA_ATTRS:
            val = getattr(self, name, None)
            if val is not None:
                setattr(self, name, attr_change_fn(val))

    def tensor(self):
        self._change_attrs_types(torch.tensor)
        return self

    def float(self):
        self._change_attrs_types(lambda t: t.float())
        return self

    def numpy(self):
        self._change_attrs_types(lambda t: t if isinstance(t, np.ndarray) else t.detach().cpu().numpy())
        return self

    def cpu(self):
        self._change_attrs_types(lambda t: t.cpu())
        return self

    def cuda(self):
        self._change_attrs_types(lambda t: t.cuda())
        return self

    def to(self, device):
        self._change_attrs_types(lambda t: t.to(device))     # in place, returns None (mot_graph.py:76-77)

    def device(self):
        if isinstance(getattr(self, 'edge_index', None), torch.Tensor):
            return self.edge_index.device
        return torch.device('cpu')


def _col(table, name, dev):
    v = table[name]
    if torch.is_tensor(v):
        return v.to(dev)
    v = v.values if hasattr(v, 'values') else v
    return torch.as_tensor(np.asarray(v)).to(dev)


class MOTGraph(object):
    """Edge construction + Graph assembly for one frame window.

    ``MOTGraph(seq_det_df, start_frame, end_frame, ensure_end_is_in, step_size, seq_info_dict, dataset_params,
    inference_mode, max_frame_dist)`` is the reference's constructor (data/mot_graph.py:94-106): the window's rows are
    selected from the sequence table (``_construct_graph_df``, :108-147) and the appearance tensors are loaded from
    the per-frame embedding store (``_load_appearance_data``, :153-193) when the graph is built.
    ``MOTGraph.from_tensors(graph_df, reid, node_core, node_ext, ...)`` takes an already selected table (DataFrame
    or dict of arrays with columns frame, bb_height, bb_width, feet_x, feet_y, rows sorted by (frame, detection id))
    and already loaded tensors ``reid [N,256]``, ``node_core [N,2048,8,4]`` (or pooled), ``node_ext [N,256,14,14]``.
    """

    def __init__(self, seq_det_df=None, start_frame=None, end_frame=None, ensure_end_is_in=False, step_size=None,
                 seq_info_dict=None, dataset_params=None, inference_mode=False, max_frame_dist=None):
        self.dataset_params = dataset_params
        self.step_size = step_size
        self.seq_info_dict = seq_info_dict or {}
        self.inference_mode = inference_mode
        self.max_frame_dist = max_frame_dist if max_frame_dist is not None or dataset_params is None \
            else dataset_params['max_frame_dist']
        self.device = torch.device('cuda')
        self.reid_embeddings = self.node_core_feats = self.node_ext_feats = None
        self.graph_obj = None
        if seq_det_df is not None:
            self.graph_df, self.frames = self._construct_graph_df(seq_det_df=seq_det_df.copy(), start_frame=start_frame,
                                                                  end_frame=end_frame, ensure_end_is_in=ensure_end_is_in)

    @classmethod
    def from_tensors(cls, graph_df, reid_embeddings, node_core_feats, node_ext_feats=None, seq_info_dict=None,
                     dataset_params=None, inference_mode=False, max_frame_dist=None):
        self = cls(seq_info_dict=seq_info_dict, dataset_params=dataset_params, inference_mode=inference_mode,
                   max_frame_dist=max_frame_dist)
        self.graph_df = graph_df
        self.reid_embeddings = reid_embeddings.to(self.device, torch.float32)
        self.node_core_feats = node_core_feats
        self.node_ext_feats = node_ext_feats
        return self

    def _construct_graph_df(self, seq_det_df, start_frame, end_frame=None, ensure_end_is_in=False):
        """Frames of the window and its rows of the sequence table, sorted by (frame, detection_id).
        reference: data/mot_graph.py:108-147"""
        if end_frame is not None:
            valid_frames = np.arange(start_frame, end_frame + 1, self.step_size)
            if ensure_end_is_in and (end_frame not in valid_frames):
                valid_frames = valid_frames.tolist() + [end_frame]
        else:
            valid_frames = np.arange(start_frame, seq_det_df.frame.max(), self.step_size)
            if self.dataset_params['frames_per_graph'] != 'max':
                valid_frames = valid_frames[:self.dataset_params['frames_per_graph']]
            if self.dataset_params['max_detects'] is not None:
                scene_df_ = seq_det_df[seq_det_df.frame.isin(valid_frames)].copy()
                frames_cumsum = scene_df_.groupby('frame')['bb_left'].count().cumsum()
                valid_frames = frames_cumsum[frames_cumsum <= self.dataset_params['max_detects']].index
        graph_df = seq_det_df[seq_det_df.frame.isin(valid_frames)].copy()
        graph_df = graph_df.sort_values(by=['frame', 'detection_id']).reset_index(drop=True)
        return graph_df, sorted(graph_df.frame.unique())

    def _load_appearance_data(self):
        """(reid, node_core, node_ext) of the window's detections from the embedding store; with
        ``dataset_params['node_core_pooled'] = True`` the pooled ``[N,2048]`` variant written by
        ``EmbeddingStore.pool`` is read instead of the ``[N,2048,8,4]`` maps.  reference: data/mot_graph.py:153-193"""
        import os.path as osp
        from .embedding_store import load_precomputed_embeddings
        dp = self.dataset_params
        emb_dir = osp.join('embeddings', self.seq_info_dict['det_file_name'])
        load = lambda d, dim: load_precomputed_embeddings(det_df=self.graph_df, seq_info_dict=self.seq_info_dict,
                                                          embeddings_dir=osp.join(emb_dir, d), use_cuda=True,
                                                          embedding_dim=dim, pin_memory=True)
        reid = load(dp['reid_embeddings_dir'], '1D')
        if dp['reid_embeddings_dir'] == dp['node_core_embeddings_dir']:
            core = reid.clone()
        elif dp.get('node_core_pooled', False):
            core = load(dp['node_core_embeddings_dir'] + '_pooled', '1D')
        else:
            core = load(dp['node_core_embeddings_dir'], '3D')
        ext = load(dp['node_ext_embeddings_dir'], '3D') if dp.get('node_ext_embeddings_dir') else None
        return reid, core, ext

    def _get_edge_ixs(self, reid_embeddings):
        """Time-valid pairs, pruned to reciprocal top-k ReID neighbours in training mode.
        Returns (pairs [2,P] int64 on the GPU, reid distance per pair or None).
        reference: data/mot_graph.py:195-221"""
        frame = _col(self.graph_df, 'frame', self.device).to(torch.int64)
        mfd = self.max_frame_dist
        pairs = ops.time_valid_pairs(frame, -1 if mfd == 'max' else int(mfd))
        dist = None
        k = self.dataset_params['top_k_nns']
        if not self.inference_mode and k is not None:
            dist = ops.pair_reid_dist(reid_embeddings, pairs)
            keep = ops.knn_mask(dist, pairs, frame.numel(), k, self.dataset_params['reciprocal_k_nns'],
                                symmetric_edges=False)
            pairs, dist = ops.compact_pairs(pairs, keep, dist)
        return pairs, dist

    def construct_graph_object(self):
        """reference: data/mot_graph.py:283-316"""
        dev = self.device
        if self.reid_embeddings is None:
            self.reid_embeddings, self.node_core_feats, self.node_ext_feats = self._load_appearance_data()
        pairs, dist = self._get_edge_ixs(self.reid_embeddings)
        if dist is None:
            dist = ops.pair_reid_dist(self.reid_embeddings, pairs)
        use = self.dataset_params['edge_feats_to_use']
        cols = {n: _col(self.graph_df, n, dev).float() for n in ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')}
        with_dist = 'emb_dist' in use
        attr, edge_index = ops.edge_feats_assemble(pairs, cols['frame'], cols['bb_height'], cols['bb_width'],
                                                   cols['feet_x'], cols['feet_y'], self.seq_info_dict['fps'],
                                                   dist if with_dist else None)
        order = ('secs_time_dists', 'norm_feet_x_dists', 'norm_feet_y_dists', 'bb_height_dists',
                 'bb_width_dists', 'emb_dist')
        wanted = [order.index(n) for n in use if n in order and (n != 'emb_dist')]
        if with_dist:
            wanted.append(5)                                   # emb_dist is appended last (mot_graph.py:306-307)
        if wanted != list(range(attr.shape[1])):
            attr = attr[:, wanted].contiguous()
        self.graph_obj = Graph(x=self.node_core_feats, x_ext=self.node_ext_feats, edge_attr=attr,
                               edge_index=edge_index)
        if self.inference_mode:
            self.graph_obj.reid_emb_dists = torch.cat((dist, dist))
        self.graph_obj.to(dev)
        return self.graph_obj


    def assign_edge_labels(self):
        """graph_obj.edge_labels [E] float per dataset_params['true_edge_labels'] ('closest' | 'all') from the
        ``id`` column of the detection table.  reference: data/mot_graph.py:223-262"""
        mode = self.dataset_params.get('true_edge_labels', 'closest')
        ids = _col(self.graph_df, 'id', self.device).to(torch.int64)
        self.graph_obj.edge_labels = ops.assign_edge_labels(self.graph_obj.edge_index, ids, mode)
        return self.graph_obj.edge_labels


class GraphBatch(object):
    """Block-diagonal batch of independent window graphs built in one pass (extension; the
    reference builds one window per ``MOTGraph``).  Node / edge ids are batch-global:
    ``edge_index = [all (i<j) pairs of all windows | the same pairs reversed]``; window ``g`` owns
    nodes ``node_ptr[g]:node_ptr[g+1]`` and pairs ``pair_ptr[g]:pair_ptr[g+1]`` of each half."""

    def __init__(self, xs, node_ptr, edge_index, edge_attr, pair_ptr, reid_emb_dists=None):
        self.xs, self.node_ptr, self.pair_ptr = xs, list(node_ptr), list(pair_ptr)
        self.edge_index, self.edge_attr, self.reid_emb_dists = edge_index, edge_attr, reid_emb_dists
        self._pool = None           # (xs it was pooled from, [N, C] pooled buffer, event of the side stream)

    def pooled_xs(self):
        """(pooled [N, C] buffer, event that marks it ready) of the node-feature pool ``build_graph_batch`` started on a
        side stream, or None when there is none or ``xs`` has been replaced since.  Wait on the event before reading."""
        if self._pool is None or self._pool[0] is not self.xs:
            return None
        return self._pool[1], self._pool[2]

    @property
    def num_graphs(self):
        return len(self.node_ptr) - 1

    @property
    def num_nodes(self):
        return self.node_ptr[-1]

    @property
    def num_edges(self):
        return self.edge_index.size(1)

    def graph(self, g):
        """Window ``g`` as a reference-style ``Graph`` (local node ids, reference edge order)."""
        a, b, p = self.pair_ptr[g], self.pair_ptr[g + 1], self.pair_ptr[-1]
        ei = torch.cat((self.edge_index[:, a:b], self.edge_index[:, p + a:p + b]), dim=1) - self.node_ptr[g]
        ea = torch.cat((self.edge_attr[a:b], self.edge_attr[p + a:p + b]), dim=0)
        x = self.xs[g] if isinstance(self.xs, (list, tuple)) else self.xs[self.node_ptr[g]:self.node_ptr[g + 1]]
        return Graph(x=x, x_ext=None, edge_attr=ea, edge_index=ei)


def build_window_graphs(windows, dataset_params, fps, inference_mode=False, max_frame_dist=None, device=None,
                        engine=None):
    """Edge construction + assembly (``MOTGraph._get_edge_ixs`` + ``construct_graph_object``,
    reference: data/mot_graph.py:195-221, 283-316) for a list of windows at once, on the GPU, with one
    host synchronisation.  Each window is a mapping with ``frame, bb_height, bb_width, feet_x, feet_y``
    (arrays / tensors, rows sorted by (frame, detection id)), ``reid`` [n,256] and ``x`` (node features)."""
    dev = device or torch.device('cuda')
    node_ptr = [0]
    for w in windows:
        node_ptr.append(node_ptr[-1] + int(w['reid'].shape[0]))
    table = {name: torch.cat([_col(w, name, dev).view(-1) for w in windows])
             for name in ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')}
    table['reid'] = torch.cat([w['reid'].to(dev, torch.float32) for w in windows])
    table['x'] = [w['x'] if w['x'].is_cuda else w['x'].to(dev) for w in windows]
    return build_graph_batch(table, node_ptr, dataset_params, fps, inference_mode, max_frame_dist, dev, engine)


def build_graph_batch(table, node_ptr, dataset_params, fps, inference_mode=False, max_frame_dist=None, device=None,
                      engine=None):
    """Same as ``build_window_graphs`` for a detection table that is already ONE set of columns (the way
    the reference holds a sequence's ``graph_df``): ``table`` maps ``frame, bb_height, bb_width, feet_x,
    feet_y`` to [N_total] tensors, ``reid`` to [N_total,256] and ``x`` to the node features (one tensor
    or a list with one tensor per window); window g owns rows ``node_ptr[g]:node_ptr[g+1]``.

    When ``x`` holds CUDA fp32 feature maps ([n, C, H, W], the same C, H, W for every window), their average pool
    is enqueued first, on a side stream, and the graph build runs on a stream of higher priority, so that the pool
    fills the GPU around the build's kernels and host synchronisations; ``MOTMPNet.forward_batch`` waits for the
    pool before the node encoder.  ``table['x']`` is therefore read at once: it
    must be ready on the current stream when this is called, as any argument of a kernel on that stream."""
    dev = device or torch.device('cuda')
    pool = _start_pool(table['x'])
    if pool is None:
        return _build(table, node_ptr, dataset_params, fps, inference_mode, max_frame_dist, dev, engine)
    # the build runs on a stream of higher priority than the pool's: the pool is cut into short blocks, so a build
    # kernel gets its SMs as soon as the pool blocks on them end, and the pool fills the GPU while the host waits
    cur = torch.cuda.current_stream()
    build = _stream('build', priority=-1)
    build.wait_stream(cur)
    with torch.cuda.stream(build):
        batch = _build(table, node_ptr, dataset_params, fps, inference_mode, max_frame_dist, dev, engine)
    cur.wait_stream(build)
    for t in (batch.edge_index, batch.edge_attr, batch.reid_emb_dists):
        if t is not None:
            t.record_stream(cur)
    batch._pool = (table['x'],) + pool
    return batch


def _build(table, node_ptr, dataset_params, fps, inference_mode, max_frame_dist, dev, engine):
    col = lambda name, dt: table[name].to(dev, dt).view(-1)
    frame = col('frame', torch.int64)
    reid = table['reid'].to(dev, torch.float32)
    mfd = dataset_params['max_frame_dist'] if max_frame_dist is None else max_frame_dist
    k = None if inference_mode else dataset_params['top_k_nns']
    pairs, dist, pair_ptr = ops.knn_graph_pairs(frame, node_ptr, reid, k, dataset_params['reciprocal_k_nns'],
                                                -1 if mfd == 'max' else int(mfd), engine=engine)
    use = dataset_params['edge_feats_to_use']
    with_dist = 'emb_dist' in use
    attr, edge_index = ops.edge_feats_assemble(pairs, frame.float(), col('bb_height', torch.float32),
                                               col('bb_width', torch.float32), col('feet_x', torch.float32),
                                               col('feet_y', torch.float32), fps, dist if with_dist else None)
    order = ('secs_time_dists', 'norm_feet_x_dists', 'norm_feet_y_dists', 'bb_height_dists', 'bb_width_dists')
    wanted = [order.index(n) for n in use if n in order] + ([5] if with_dist else [])
    if wanted != list(range(attr.shape[1])):
        attr = attr[:, wanted].contiguous()
    return GraphBatch(table['x'], node_ptr, edge_index, attr, pair_ptr,
                      torch.cat((dist, dist)) if inference_mode else None)


_STREAMS = {}


def _stream(name, priority=0):
    """One cached stream per (purpose, device) of the current device."""
    key = (name, torch.cuda.current_device())
    if key not in _STREAMS:
        _STREAMS[key] = torch.cuda.Stream(priority=priority)
    return _STREAMS[key]


def _start_pool(x):
    """Enqueue the pool of the node-feature maps ``x`` (a tensor or a list of per-window tensors) on a side stream of
    the current device: (pooled [N, C] buffer, event recorded after it), or None for inputs that are not CUDA fp32
    maps of one shape per node (pooled features, CPU tensors, no windows), which the node encoder pools itself."""
    xs = list(x) if isinstance(x, (list, tuple)) else [x]
    if not xs or not all(torch.is_tensor(t) and t.is_cuda and t.dtype == torch.float32 and t.dim() >= 3 and
                         t.shape[1:] == xs[0].shape[1:] and t.device.index == torch.cuda.current_device() for t in xs):
        return None
    cur = torch.cuda.current_stream()
    side = _stream('pool')
    pooled = torch.empty((sum(t.shape[0] for t in xs), xs[0].shape[1]), dtype=torch.float32, device=cur.device)
    side.wait_stream(cur)                       # the maps are ready on the current stream, and the buffer is allocated
    for t in xs:                                # neither is reused before the side stream is done with it, even if the
        t.record_stream(side)                   # caller drops its maps right after build_graph_batch
    pooled.record_stream(side)
    with torch.cuda.stream(side):
        ops.avgpool_windows(xs, out=pooled)
        done = torch.cuda.Event()
        done.record(side)
    return pooled, done
