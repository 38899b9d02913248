"""bench.py --dump-outputs: what the last timed step returned, as .npy files within a size budget."""
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _step_result(num_edges=5000, num_nodes=900, steps=11, seed=0):
    g = torch.Generator().manual_seed(seed)
    batch = SimpleNamespace(edge_index=torch.randint(0, num_nodes, (2, num_edges), generator=g),
                            edge_attr=torch.randn(num_edges, 6, generator=g), pair_ptr=[0, 1000, 2500])
    return batch, SimpleNamespace(logits=torch.randn(steps, num_edges, generator=g))


@pytest.mark.parametrize('budget', [bench.DUMP_BYTES, 100_000])
def test_dump_keeps_one_seeded_edge_sample_within_the_budget(tmp_path, budget):
    batch, out = _step_result()
    bench.dump_outputs(str(tmp_path / 'a'), batch, out, budget=budget)
    bench.dump_outputs(str(tmp_path / 'b'), batch, out, budget=budget)
    names = ('edge_index', 'edge_attr', 'logits', 'pair_ptr', 'edge_sample')
    got = {n: np.load(tmp_path / 'a' / f'{n}.npy') for n in names}
    assert sorted(os.listdir(tmp_path / 'a')) == sorted(f'{n}.npy' for n in names)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= budget
    for n in names:
        assert np.array_equal(got[n], np.load(tmp_path / 'b' / f'{n}.npy'))     # same sample every time

    sample = got['edge_sample'].astype(np.int64)
    assert np.all(np.diff(sample) > 0)
    if budget == bench.DUMP_BYTES:
        assert np.array_equal(sample, np.arange(5000))
    else:
        assert 0 < len(sample) < 5000
    assert np.array_equal(got['edge_index'], batch.edge_index.numpy()[:, sample].astype(np.float64))
    assert np.array_equal(got['edge_attr'], batch.edge_attr.numpy()[sample])
    assert np.array_equal(got['logits'], out.logits.numpy()[:, sample])
    assert np.array_equal(got['pair_ptr'], [0, 1000, 2500])


@pytest.mark.gpu
def test_bench_dump_is_the_step_on_the_seeded_inputs(tmp_path):
    """The dump equals, edge for edge, one hot-path step run here on the inputs bench.py builds from the same
    arguments (the forward is deterministic, so the comparison is exact)."""
    from mpntrackseg_b200.config import default_dataset_params
    from mpntrackseg_b200.data.mot_graph import build_graph_batch
    from mpntrackseg_b200.models.mpn import MOTMPNet
    args = ['--gpus', '1', '--steps', '2', '--warmup', '1', '--graphs', '2', '--frames', '4', '--dets', '12', '--k', '6',
            '--pooled', '--no-cpu-baseline', '--dump-outputs', str(tmp_path / 'dump')]
    subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, check=True, cwd=str(tmp_path))
    got = {f[:-4]: np.load(tmp_path / 'dump' / f) for f in os.listdir(tmp_path / 'dump')}
    assert sorted(got) == ['edge_attr', 'edge_index', 'edge_sample', 'logits', 'pair_ptr']
    assert got['edge_index'].dtype == got['edge_sample'].dtype == got['pair_ptr'].dtype == np.float64
    assert got['edge_attr'].dtype == got['logits'].dtype == np.float32

    a = bench.parse(args)
    dev = torch.device('cuda', 0)
    wins, node_ptr, _, _, devin = bench.job_inputs(a, 0, 1, dev)
    mp, P = bench.model_and_params()
    model = MOTMPNet(mp).to(dev).eval()
    model.load_state_dict(P, strict=False)
    batch = build_graph_batch(devin, node_ptr, default_dataset_params(top_k_nns=a.k, frames_per_graph=a.frames),
                              wins[0].fps, device=dev)
    with torch.no_grad():
        logits = model.forward_batch(batch).logits.cpu().numpy()
    assert np.array_equal(got['edge_sample'], np.arange(batch.num_edges))        # small enough to be written whole
    assert 0 <= got['edge_index'].min() and got['edge_index'].max() < node_ptr[-1]
    assert np.array_equal(got['edge_index'], batch.edge_index.cpu().numpy())
    assert np.array_equal(got['edge_attr'], batch.edge_attr.cpu().numpy())
    assert np.array_equal(got['pair_ptr'], batch.pair_ptr)
    assert logits.shape == (bench.NUM_CLASS_STEPS, batch.num_edges)
    assert np.array_equal(got['logits'], logits)
