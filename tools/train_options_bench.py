"""Cost of the trainable model options: the configs[3] graphed training step (KITTI-shaped window T=20 D=8 k=100,
12 message-passing steps, 11 classified, as ``bench.py --mode train`` runs it on one GPU) with node_agg_fn sum (the
shipped config), mean and max, BatchNorm1d, and BatchNorm1d + Dropout 0.3.  Prints one JSON line per option with ms
per step, launches per step (mpn_launch_count of one eager step) and the card's name and power limit.

    python tools/train_options_bench.py --steps 50 --warmup 5
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPTIONS = {'sum': {}, 'mean': dict(agg='mean'), 'max': dict(agg='max'), 'batchnorm': dict(bn=True),
           'batchnorm_dropout0.3': dict(bn=True, p=0.3)}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def run(name, opt, steps, warmup):
    import torch
    from mpntrackseg_b200 import _cabi, synth
    from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    from mpntrackseg_b200.models.mpn import MOTMPNet
    from mpntrackseg_b200.training import CoreTrainer
    dev = torch.device('cuda:0')
    ds = default_dataset_params(top_k_nns=100, frames_per_graph=20)
    mp = default_graph_model_params(12, 11)
    mp['node_agg_fn'] = opt.get('agg', 'sum')
    for k in ('encoder_feats_dict', 'edge_model_feats_dict', 'node_model_feats_dict', 'classifier_feats_dict'):
        mp[k]['use_batchnorm'] = opt.get('bn', False)
        mp[k]['dropout_p'] = opt.get('p', 0)
    P = synth.make_params(mp, seed=6, gain=0.95, core_only=True)
    model = MOTMPNet(mp).to(dev)
    model.load_state_dict(P, strict=False)
    tr = CoreTrainer(model)
    w = synth.make_window(T=20, D=8, k=100, seed=100)
    g = MOTGraph.from_tensors(synth.det_columns(w), w.reid, w.x.to(dev), None, {'fps': w.fps}, ds).construct_graph_object()
    ident = w.ident.to(dev)
    labels = (ident[g.edge_index[0]] == ident[g.edge_index[1]]).float()
    lib = _cabi.lib()
    tr.train_step(g, labels)
    l0 = lib.mpn_launch_count()
    tr.train_step(g, labels)
    launches = int(lib.mpn_launch_count() - l0)
    for _ in range(warmup):
        tr.graphed_step(g, labels)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = tr.graphed_step(g, labels)
    e1.record()
    torch.cuda.synchronize()
    return dict(option=name, ms_per_step=e0.elapsed_time(e1) / steps, launches_per_step=launches, steps=steps,
                warmup=warmup, edges=int(g.edge_index.shape[1]), nodes=int(w.N), loss=float(loss), gpu=card())


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--options', nargs='*', default=list(OPTIONS), choices=list(OPTIONS))
    a = ap.parse_args()
    for name in a.options:
        print(json.dumps(run(name, OPTIONS[name], a.steps, a.warmup)), flush=True)


if __name__ == '__main__':
    main()
