"""Sliding-window evaluation of a whole sequence graph (SURVEY.md section 8 row f1).

``MPNTracker`` keeps the reference's names and contracts for the part of the tracker that drives the
hot path -- ``_predict_edges_and_masks`` (one window: KNN prune -> network -> sigmoid -> scatter back) and
``_evaluate_graph_in_batches`` (all overlapping windows of a sequence, per-edge averaging, directed ->
undirected merge, pruning at 0.5).  reference: tracker/mpn_tracker.py:96-210, utils/graph.py:165-207.
Dataset loading is outside this path; rounding, id assignment (:212-260) and the MOTS result (:267-298, :398-417) run on
the device after it.

B200 design of ``_evaluate_graph_in_batches`` (same results, different schedule):
  * every node of the sequence is encoded ONCE (avg-pool + 2048->128->32 on tcgen05) instead of once per
    window it appears in (``frames_per_graph`` times in the reference) -- the encoder is per node, so the
    values are the same;
  * when the sequence graph carries its detection table and ReID embeddings (a ``MOTGraph``), the windows of a
    batch are pruned TOGETHER: their node rows are replicated into one table and the batched builder
    (``build_graph_batch``: time-valid pairs + distances + KNN + edge features in one pass, one host sync) rebuilds
    each window's pruned graph -- the same candidate pairs, distances and features the sequence graph holds;
    the kept pairs are mapped back to sequence edge ids with a binary search over the sorted pair list.
    Otherwise a window's candidate edges are found from a row pointer over the (i < j)-sorted pair list and pruned
    window by window with ``get_knn_mask``;
  * windows are evaluated in block-diagonal batches (``MOTMPNet.forward_batch``), predictions are accumulated
    on the device.
The mask branch (``x_ext`` present and the model has the attention / mask modules) is evaluated window by
window through ``_predict_edges_and_masks`` exactly as the reference does.
"""
import numpy as np
import torch

from ..data.mot_graph import Graph
from ..utils.graph import get_knn_mask, to_lightweight_graph, to_undirected_graph


class MPNTracker(object):
    """reference: tracker/mpn_tracker.py:26-56"""

    def __init__(self, dataset=None, graph_model=None, use_gt=False, eval_params=None, dataset_params=None,
                 logger=None, window_batch=16):
        self.dataset = dataset
        self.use_gt = use_gt
        self.logger = logger
        self.eval_params = eval_params
        self.dataset_params = dataset_params
        self.graph_model = graph_model
        self.window_batch = int(window_batch)
        self.full_graph = None
        if self.graph_model is not None:
            self.graph_model.eval()

    # ------------------------------------------------------------------ one window, reference schedule
    def _predict_edges_and_masks(self, subgraph, pred_oracle_mode=None):
        """reference: tracker/mpn_tracker.py:96-141"""
        knn_mask = get_knn_mask(pwise_dist=subgraph.reid_emb_dists, edge_ixs=subgraph.edge_index,
                                num_nodes=subgraph.num_nodes, top_k_nns=self.dataset_params['top_k_nns'],
                                use_cuda=True, reciprocal_k_nns=self.dataset_params['reciprocal_k_nns'],
                                symmetric_edges=True)
        subgraph.edge_index = subgraph.edge_index.T[knn_mask].T.contiguous()
        subgraph.edge_attr = subgraph.edge_attr[knn_mask]
        if hasattr(subgraph, 'edge_labels'):
            subgraph.edge_labels = subgraph.edge_labels[knn_mask]
        node_preds = None
        if self.use_gt:
            pruned_edge_preds = subgraph.edge_labels
            node_preds = getattr(subgraph, 'mask_labels', None)
        else:
            with torch.no_grad():
                output = self.graph_model(subgraph)
            masks = output.get('mask_predictions') or []
            if pred_oracle_mode == 'gt_edge':
                pruned_edge_preds = subgraph.edge_labels
            else:
                pruned_edge_preds = torch.sigmoid(output['classified_edges'][-1].view(-1))
            if pred_oracle_mode == 'gt_mask':
                node_preds = subgraph.mask_labels
            elif masks:
                node_preds = torch.sigmoid(masks[-1])
        edge_preds = torch.zeros(knn_mask.shape[0], device=pruned_edge_preds.device)
        edge_preds[knn_mask] = pruned_edge_preds.float()
        if self.eval_params['set_pruned_edges_to_inactive']:
            return edge_preds, torch.ones_like(knn_mask), node_preds
        return edge_preds, knn_mask, node_preds

    # ------------------------------------------------------------------ whole sequence
    def _windows(self):
        all_frames = np.array(self.full_graph.frames)
        fpg = self.full_graph.frames_per_graph
        return list(zip(all_frames, all_frames[fpg - 1:]))               # mpn_tracker.py:167

    def _frame_per_node(self, dev):
        df = self.full_graph.graph_df
        f = df['frame']
        f = f.values if hasattr(f, 'values') else f
        return torch.as_tensor(np.asarray(f)).to(dev, torch.int64).view(-1)

    def _evaluate_graph_in_batches(self, pred_oracle_mode=None):
        """reference: tracker/mpn_tracker.py:143-210"""
        go = self.full_graph.graph_obj
        x_ext = getattr(go, 'x_ext', None)
        needs_masks = x_ext is not None and getattr(self.graph_model, 'has_mask_branch', False)
        if self.use_gt or pred_oracle_mode is not None or needs_masks or not self._structured(go):
            self._evaluate_window_by_window(pred_oracle_mode)
        elif self._has_tables():
            self._evaluate_batched_rebuild()
        else:
            self._evaluate_batched()
        to_undirected_graph(self.full_graph, attrs_to_update=('edge_preds', 'edge_labels'))
        to_lightweight_graph(self.full_graph)

    @staticmethod
    def _structured(go):
        """[pairs i < j sorted by (i, j) | the same pairs flipped]: what MOTGraph.construct_graph_object builds."""
        ei = go.edge_index
        e = ei.shape[1]
        if e == 0 or e % 2:
            return False
        h = e // 2
        if not bool((ei[0, :h] < ei[1, :h]).all()) or not torch.equal(ei[:, h:], ei[:, :h].flip(0)):
            return False
        key = ei[0, :h] * (int(ei.max()) + 1) + ei[1, :h]
        if not bool((key[1:] > key[:-1]).all()):
            return False
        # every node's later partners are a contiguous index range (all time-valid pairs, nodes sorted by frame)
        same_row = ei[0, 1:h] == ei[0, :h - 1]
        return bool((ei[1, 1:h][same_row] == ei[1, :h - 1][same_row] + 1).all())

    def _evaluate_window_by_window(self, pred_oracle_mode):
        """The reference's schedule, on the device (used for the mask branch and the debugging modes)."""
        go = self.full_graph.graph_obj
        dev = go.edge_index.device
        frame = self._frame_per_node(dev)
        total = torch.zeros(go.num_edges, device=dev)
        count = torch.zeros(go.num_edges, device=dev)
        node_total, node_count = None, torch.zeros(go.num_nodes, device=dev)
        for start_frame, end_frame in self._windows():
            nodes_mask = (int(start_frame) <= frame) & (frame <= int(end_frame))
            edges_mask = nodes_mask[go.edge_index[0]] & nodes_mask[go.edge_index[1]]
            first = int(torch.nonzero(nodes_mask)[0])
            sub = Graph(x=go.x[nodes_mask], x_ext=None if getattr(go, 'x_ext', None) is None else go.x_ext[nodes_mask],
                        edge_attr=go.edge_attr[edges_mask], reid_emb_dists=go.reid_emb_dists[edges_mask],
                        edge_index=(go.edge_index.T[edges_mask].T - first).contiguous())
            for name in ('edge_labels',):
                if hasattr(go, name):
                    setattr(sub, name, getattr(go, name)[edges_mask])
            for name in ('mask_labels', 'mask_gt_ixs'):
                if hasattr(go, name):
                    setattr(sub, name, getattr(go, name)[nodes_mask])
            edge_preds, pred_mask, node_preds = self._predict_edges_and_masks(sub, pred_oracle_mode)
            total[edges_mask] += edge_preds
            count[torch.where(edges_mask)[0][pred_mask]] += 1
            if node_preds is not None:
                if node_total is None:
                    node_total = torch.zeros((go.num_nodes,) + tuple(node_preds.shape[1:]), device=dev)
                node_total[nodes_mask] += node_preds
                node_count[nodes_mask] += 1
        final = total / count
        final[torch.isnan(final)] = 0
        go.edge_preds = final
        if node_total is not None:
            go.node_preds = node_total / node_count.view(-1, 1, 1, 1)

    _TABLE_COLS = ('frame', 'bb_height', 'bb_width', 'feet_x', 'feet_y')

    def _has_tables(self):
        mg = self.full_graph
        df = getattr(mg, 'graph_df', None)
        try:
            cols_ok = df is not None and all(c in df for c in self._TABLE_COLS)
        except TypeError:
            cols_ok = False
        return (cols_ok and getattr(mg, 'reid_embeddings', None) is not None and
                'fps' in (getattr(mg, 'seq_info_dict', None) or {}) and getattr(mg, 'max_frame_dist', None) is not None)

    def _window_node_ranges(self, frame):
        windows = self._windows()
        starts = torch.tensor([int(w[0]) for w in windows], device=frame.device)
        ends = torch.tensor([int(w[1]) for w in windows], device=frame.device)
        return (torch.searchsorted(frame, starts, right=False).tolist(),
                torch.searchsorted(frame, ends, right=True).tolist())

    def _evaluate_batched_rebuild(self):
        """Batched schedule for a sequence graph that still has its detection table and embeddings."""
        from ..data.mot_graph import build_graph_batch
        mg = self.full_graph
        go, model, ds = mg.graph_obj, self.graph_model, self.dataset_params
        dev = go.edge_index.device
        frame = self._frame_per_node(dev)
        assert bool((frame[1:] >= frame[:-1]).all()), 'nodes must be sorted by frame (mot_graph.py:145)'
        n, half = go.num_nodes, go.num_edges // 2
        keys = go.edge_index[0, :half] * n + go.edge_index[1, :half]                  # ascending (checked by _structured)
        df = mg.graph_df
        col = lambda c: torch.as_tensor(np.asarray(df[c].values if hasattr(df[c], 'values') else df[c])).to(dev)
        cols = {c: col(c) for c in self._TABLE_COLS}
        reid = mg.reid_embeddings.to(dev, torch.float32)
        with torch.no_grad():
            x_enc = model.encode_nodes(go.x)                                          # every node once
        total = torch.zeros(2 * half, device=dev)
        count = torch.zeros(2 * half, device=dev)
        all_inactive = bool(self.eval_params['set_pruned_edges_to_inactive'])
        n0s, n1s = self._window_node_ranges(frame)
        for b0 in range(0, len(n0s), self.window_batch):
            rng = list(zip(n0s[b0:b0 + self.window_batch], n1s[b0:b0 + self.window_batch]))
            idx = torch.cat([torch.arange(a, b, device=dev) for a, b in rng])         # sequence node id of every batch row
            node_ptr = [0]
            for a, b in rng:
                node_ptr.append(node_ptr[-1] + (b - a))
            table = {c: v[idx] for c, v in cols.items()}
            table['reid'], table['x'] = reid[idx], x_enc[idx]
            batch = build_graph_batch(table, node_ptr, ds, mg.seq_info_dict['fps'], inference_mode=False,
                                      max_frame_dist=mg.max_frame_dist, device=dev)
            pairs = batch.pair_ptr[-1]
            if pairs == 0:
                continue
            with torch.no_grad():
                out = model.forward_batch(batch, encoded=True)
            probs = torch.sigmoid(out.logits[-1]).float()
            gi, gj = idx[batch.edge_index[0, :pairs]], idx[batch.edge_index[1, :pairs]]
            ids = torch.searchsorted(keys, gi * n + gj)                                # exact hits: same candidate pairs
            total.index_add_(0, ids, probs[:pairs])
            total.index_add_(0, ids + half, probs[pairs:])
            if not all_inactive:
                one = torch.ones(pairs, device=dev)
                count.index_add_(0, ids, one)
                count.index_add_(0, ids + half, one)
        if all_inactive:
            # every window that contains both endpoints predicts the edge (pruned ones as 0): windows t with
            # t <= f_i and f_j <= t + fpg - 1, f = frame position in the sequence's frame list
            all_frames = torch.as_tensor(np.array(mg.frames)).to(dev, frame.dtype)
            fpos = torch.searchsorted(all_frames, frame)
            fi, fj = fpos[go.edge_index[0, :half]], fpos[go.edge_index[1, :half]]
            fpg, nwin = mg.frames_per_graph, len(n0s)
            c = (torch.minimum(fi, torch.full_like(fi, nwin - 1)) - (fj - fpg + 1).clamp(min=0) + 1).clamp(min=0).float()
            count = torch.cat((c, c))
        final = total / count
        final[torch.isnan(final)] = 0
        go.edge_preds = final

    def _evaluate_batched(self):
        go = self.full_graph.graph_obj
        model = self.graph_model
        dev = go.edge_index.device
        ds = self.dataset_params
        frame = self._frame_per_node(dev)
        assert bool((frame[1:] >= frame[:-1]).all()), 'nodes must be sorted by frame (mot_graph.py:145)'
        n, half = go.num_nodes, go.num_edges // 2
        pi, pj = go.edge_index[0, :half], go.edge_index[1, :half]
        # CSR over the (i, j)-sorted pair list; within a row the j's ascend, so "j < n1" is a prefix of the row
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        rowlen = torch.bincount(pi, minlength=n)
        rowptr[1:] = torch.cumsum(rowlen, 0)
        jfirst = torch.full((n,), n, dtype=torch.int64, device=dev)      # first partner of every row (n = none)
        has = rowlen > 0
        jfirst[has] = pj[rowptr[:-1][has]]
        with torch.no_grad():
            x_enc = model.encode_nodes(go.x)                             # every node once
        total = torch.zeros(2 * half, device=dev)
        count = torch.zeros(2 * half, device=dev)
        all_inactive = bool(self.eval_params['set_pruned_edges_to_inactive'])
        n0s, n1s = self._window_node_ranges(frame)
        for b0 in range(0, len(n0s), self.window_batch):
            graphs, ids_kept = [], []
            for n0, n1 in zip(n0s[b0:b0 + self.window_batch], n1s[b0:b0 + self.window_batch]):
                # pairs of row i start at rowptr[i] with j = jfirst[i], jfirst[i] + 1, ... : keep those with j < n1
                cnt = torch.minimum(rowlen[n0:n1], (n1 - jfirst[n0:n1]).clamp(min=0))
                m = int(cnt.sum())
                ids = torch.repeat_interleave(rowptr[n0:n1] - torch.cumsum(cnt, 0) + cnt, cnt) + torch.arange(m, device=dev)
                sub_ei = torch.stack((torch.cat((pi[ids], pj[ids])), torch.cat((pj[ids], pi[ids])))) - n0
                both = torch.cat((ids, ids + half))
                keep = get_knn_mask(pwise_dist=go.reid_emb_dists[both], edge_ixs=sub_ei, num_nodes=n1 - n0,
                                    top_k_nns=ds['top_k_nns'], use_cuda=True,
                                    reciprocal_k_nns=ds['reciprocal_k_nns'], symmetric_edges=True)
                kept = both[keep]
                graphs.append(Graph(x=x_enc[n0:n1], x_ext=None, edge_attr=go.edge_attr[kept],
                                    edge_index=sub_ei[:, keep].contiguous()))
                ids_kept.append(kept)
                if all_inactive:
                    count[both] += 1
            with torch.no_grad():
                out = model.forward_batch(graphs, encoded=True)
            probs = torch.sigmoid(out.logits[-1])
            flat = torch.cat(ids_kept)
            total.index_add_(0, flat, probs.float())
            if not all_inactive:
                count.index_add_(0, flat, torch.ones_like(probs, dtype=torch.float32))
        final = total / count
        final[torch.isnan(final)] = 0
        go.edge_preds = final

    # ------------------------------------------------------------------ rounding + identities (SURVEY.md f2)
    def _project_graph_model_output(self):
        """Rounds the edge predictions of the (undirected, pruned) sequence graph into a feasible flow on the GPU.
        reference: tracker/mpn_tracker.py:212-229 -- except that the graph stays on the device (the reference turns
        it into numpy here); ``constr_satisf_rate`` is set on ``full_graph`` as there."""
        from .projectors import ExactProjector, GreedyProjector
        method = self.eval_params['rounding_method']
        if method == 'greedy':
            projector = GreedyProjector(self.full_graph)
        elif method == 'exact':
            projector = ExactProjector(self.full_graph, solver_backend=self.eval_params.get('solver_backend', 'pulp'))
        else:
            raise RuntimeError("Rounding type for projector not understood")
        projector.project()
        self.full_graph.constr_satisf_rate = projector.constr_satisf_rate

    def _assign_ped_ids(self):
        """One identity per connected component of the active edges (tracker/mpn_tracker.py:231-248; the reference
        calls scipy's connected_components on the host).  Returns the [N] int64 labels on the device; when the sequence
        graph carries a ``graph_df`` they are also stored as its ``ped_id`` column (one device -> host copy)."""
        from .. import ops
        go = self.full_graph.graph_obj
        labels, _ = ops.connected_components(go.edge_index, (go.edge_preds == 1).float(), go.num_nodes)
        self.ped_ids = labels
        df = getattr(self.full_graph, 'graph_df', None)
        if df is not None and hasattr(df, 'copy') and not isinstance(df, dict):
            assert len(labels) == df.shape[0], "Ped Ids Label format is wrong"
            self.final_projected_output = df.copy()
            self.final_projected_output['ped_id'] = labels.cpu().numpy()
        return labels

    # ------------------------------------------------------------------ MOTS result
    def save_mots_results(self, path, class_id=2, threshold=0.5):
        """Writes the tracker's MOTS result: one line ``"<frame> <id> <class_id> <H> <W> <rle>"`` per node with a
        non-empty mask, sorted by frame, then node index (reference: tracker/mpn_tracker.py:267-298, :398-417).  Each
        node's averaged mask ``graph_obj.node_preds`` is pasted into its box (``graph_df`` columns bb_left, bb_top,
        bb_width, bb_height, frame) of the ``seq_info_dict`` frame_height x frame_width image; within a frame every pixel
        goes to the node with the largest probability, and to its mask where that is > threshold.  id = the node's
        ``_assign_ped_ids`` label.  Runs after ``_assign_ped_ids``.  Returns (lines written, nodes whose mask is
        empty and were skipped)."""
        from ..utils.mots import encode_mots_masks, write_mots_txt
        mg = self.full_graph
        go = mg.graph_obj
        node_preds = getattr(go, 'node_preds', None)
        if node_preds is None:
            raise RuntimeError('save_mots_results: the sequence graph has no node_preds (evaluate it with the mask '
                               'branch: node features x_ext and a model with the mask modules)')
        labels = getattr(self, 'ped_ids', None)
        if labels is None:
            raise RuntimeError('save_mots_results: call _assign_ped_ids first')
        dev = node_preds.device
        df = mg.graph_df
        col = lambda c: np.asarray(df[c].values if hasattr(df[c], 'values') else df[c])
        left, top = col('bb_left').astype(np.float64), col('bb_top').astype(np.float64)
        boxes = np.stack((left, top, left + col('bb_width').astype(np.float64), top + col('bb_height').astype(np.float64)), 1)
        frame = col('frame').astype(np.int64)
        h, w = int(mg.seq_info_dict['frame_height']), int(mg.seq_info_dict['frame_width'])
        strings = encode_mots_masks(node_preds.float(), torch.from_numpy(boxes).to(dev), torch.from_numpy(frame).to(dev),
                                    (h, w), threshold)
        written = write_mots_txt(path, frame, labels.cpu().numpy(), class_id, h, w, strings)
        return written, len(strings) - written
