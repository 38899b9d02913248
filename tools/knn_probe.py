"""Development probe: batched KNN graph build (16 bench windows) -- stats and time of the thresholded vs dense path.
Run as: python tools/knn_probe.py ; MPN_KNN_DENSE=1 python tools/knn_probe.py"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mpntrackseg_b200 import ops, synth

dev = torch.device('cuda:0')
G, T, D, K = int(os.environ.get('G', 16)), 15, int(os.environ.get('D', 150)), int(os.environ.get('K', 50))
wins = [synth.make_window(T=T, D=D, k=K, seed=s, node_feats='pooled', node_dim=8, min_gap=0) for s in range(G)]
frame = torch.cat([w.frame for w in wins]).to(dev)
reid = torch.cat([w.reid for w in wins]).to(dev)
ptr = [0]
for w in wins:
    ptr.append(ptr[-1] + w.N)
for it in range(3):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pairs, dist, gpp = ops.knn_graph_pairs(frame, ptr, reid, K, True, -1, engine='tc')
    e1.record()
    torch.cuda.synchronize()
    print('dense' if os.environ.get('MPN_KNN_DENSE') else 'thresholded', 'iter', it, 'ms', round(e0.elapsed_time(e1), 3),
          'pairs', pairs.shape[1], 'stats [build code (0 exact, 1 dense, 2 thresholded, 3 general), repaired rows]', ops.LAST_KNN_STATS)
