"""GPU tests of the kernels between the detection table and the first message-passing step, against fp64.

Covered: the node encoder (tensor-core kernel and fp32 Linear chain), the average pool, the fused edge encoder and
its generic fallback, the edge features, the per-pair ReID distance and the exclusive scan behind ``compact_pairs``
and ``time_valid_pairs``.  The cases cross the boundaries the parity suite's windows never reach: operand scales
from 2^-24 to 2^12, rows of very different magnitude in one launch, degenerate and non-finite rows, every launch
gate, grid strides, unaligned views, and scans of more than 1,024 chunks.  Each test asserts that its case reaches
the path or boundary it names; grid caps are computed from the device's SM count.  The reference is always fp64.
"""
import math
import warnings

import pytest
import torch

from mpntrackseg_b200 import ops, synth
from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
from oracle import graph_ref, mpn_ref
from test_cuda_parity import assert_logits_close, dev, make_model
from test_kernel_boundaries import TC_TILE, persistent_sizes, sms

pytestmark = pytest.mark.gpu

ENGINES = ('tc', 'fp32')
U = 2.0 ** -24                   # unit roundoff of fp32


def pow2(t, p):
    """t * 2^p, exact (no result here is subnormal)."""
    return t * (2.0 ** p)


def uniform(shape, bound, g):
    return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1).mul_(bound).float()


# ------------------------------------------------------------------ node encoder
ENC_TOL = 2e-5
SCALES = (-24, -20, -16, -12, -8, -4, 0, 4, 8, 12)
SENTINEL = 7                     # mpn_node_encoder_tc clears the status word first: 0 afterwards proves it ran


def enc_params(k0, seed):
    """Weights and biases of the shipped K -> 128 -> 32 stack at torch's default Linear scale (|W0| <= 1/sqrt(K),
    |W1| <= 1/sqrt(128))."""
    g = torch.Generator().manual_seed(seed)
    w0, b0 = uniform((128, k0), k0 ** -0.5, g), uniform((128,), k0 ** -0.5, g)
    w1, b1 = uniform((32, 128), 128 ** -0.5, g), uniform((32,), 128 ** -0.5, g)
    return [w0, w1], [b0, b1]


def enc_input(n, k0, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, k0, generator=g).abs_()


def ramp_rows(x):
    """Rows whose 64-wide chunk c is x 2^c: the kernel's running row shift is passed every 4 chunks, and the row's
    accumulator is rescaled each time."""
    return x * 2.0 ** (torch.arange(x.shape[1]) // 64).float()


def enc_ref(x, ws, bs):
    """(ReLU output, layer-2 output before its ReLU), both fp64."""
    h = torch.relu(x.double() @ ws[0].double().T + bs[0].double())
    z = h @ ws[1].double().T + bs[1].double()
    return torch.relu(z), z


def encode(x, ws, bs, engine):
    """ops.node_encoder with cuda copies of the arguments; x may already be on the device (views)."""
    with torch.no_grad():
        return ops.node_encoder(x.to(dev()), [w.to(dev()) for w in ws], [b.to(dev()) for b in bs], engine=engine).cpu()


def encode_tc(x, ws, bs):
    """The tensor-core kernel without fallback: the status word must be cleared by it and stay clear."""
    st = torch.full((1,), SENTINEL, dtype=torch.int32, device=dev())
    with torch.no_grad():
        out = ops.node_encoder(x.to(dev()), [w.to(dev()) for w in ws], [b.to(dev()) for b in bs], engine='tc', status=st)
    assert int(st.item()) == 0, f'the tensor-core encoder did not run clean (status {int(st.item())})'
    return out.cpu()


def run_encoder(x, ws, bs, engine):
    return encode_tc(x, ws, bs) if engine == 'tc' else encode(x, ws, bs, 'fp32')


def assert_enc_close(got, x, ws, bs, what, tol=ENC_TOL):
    """Per row: |got - ref| <= 2e-5 * max_j |z_rj|, z the fp64 layer-2 output before its ReLU."""
    ref, z = enc_ref(x, ws, bs)
    got = got.double()
    assert torch.isfinite(got).all(), f'{what}: non-finite output'
    scale = z.abs().amax(dim=1, keepdim=True)
    err = (got - ref).abs()
    bad = err > tol * scale
    rel = (err / scale.clamp(min=1e-300)).amax(dim=1)
    assert not bad.any(), f'{what}: {int(bad.any(dim=1).sum())} of {x.shape[0]} rows off, worst {float(rel.max()):.3e} (bar {tol})'


@pytest.mark.parametrize('p', SCALES)
@pytest.mark.parametrize('engine', ENGINES)
def test_node_encoder_input_scale(engine, p):
    """x * 2^p with both biases * 2^p: the exact output is 2^p times the unscaled one, and the bar is relative."""
    ws, bs = enc_params(2048, seed=1)
    x = pow2(enc_input(300, 2048, seed=2), p)
    bs = [pow2(b, p) for b in bs]
    assert_enc_close(run_encoder(x, ws, bs, engine), x, ws, bs, f'{engine} x * 2^{p}')


@pytest.mark.parametrize('q', (-8, -4, 0, 4))
@pytest.mark.parametrize('layer', (0, 1))
@pytest.mark.parametrize('engine', ENGINES)
def test_node_encoder_weight_scale(engine, layer, q):
    """W0 * 2^q (with b0, b1 * 2^q) or W1 * 2^q (with b1 * 2^q)."""
    ws, bs = enc_params(2048, seed=3)
    ws[layer] = pow2(ws[layer], q)
    bs = [pow2(b, q) if i >= layer else b for i, b in enumerate(bs)]
    x = enc_input(300, 2048, seed=4)
    assert_enc_close(run_encoder(x, ws, bs, engine), x, ws, bs, f'{engine} W{layer} * 2^{q}')


@pytest.mark.parametrize('engine', ENGINES)
def test_node_encoder_is_scale_equivariant(engine):
    """out(x 2^p, b 2^p) == 2^p out(x, b) bit for bit: every scaling inside both engines is a power of two."""
    ws, bs = enc_params(2048, seed=5)
    x = enc_input(260, 2048, seed=6)
    x[:20] = ramp_rows(x[:20])
    base = run_encoder(x, ws, bs, engine)
    assert float(base.abs().max()) > 0
    for p in SCALES:
        got = run_encoder(pow2(x, p), ws, [pow2(b, p) for b in bs], engine)
        assert torch.equal(got, pow2(base, p)), f'{engine}: output at 2^{p} is not 2^{p} times the unscaled one'


@pytest.mark.parametrize('engine', ENGINES)
def test_node_encoder_rows_of_different_magnitude_in_one_launch(engine):
    """Rows at 2^-16 interleaved with rows at 2^0, as two windows pooled into one buffer by encode_nodes_list.  The
    biases are zero, so the quiet rows' outputs are of their own order and checked at their own scale."""
    ws, bs = enc_params(2048, seed=7)
    bs = [torch.zeros_like(b) for b in bs]
    x = enc_input(512, 2048, seed=8)
    quiet = torch.arange(512) % 2 == 1
    x[quiet] = pow2(x[quiet], -16)
    got = run_encoder(x, ws, bs, engine)
    assert_enc_close(got[quiet], x[quiet], ws, bs, f'{engine} quiet rows')
    assert_enc_close(got[~quiet], x[~quiet], ws, bs, f'{engine} loud rows')


@pytest.mark.parametrize('engine', ENGINES)
def test_node_encoder_degenerate_rows(engine):
    """All-zero rows, rows with one nonzero entry, rows whose largest |x| is 6.5e4 and 1e6 (beyond the fp16 range
    unscaled), rows growing 2^31-fold along K and rows jumping 1e3-fold halfway: the tensor-core kernel keeps them
    without a status bit."""
    ws, bs = enc_params(2048, seed=9)
    x = enc_input(200, 2048, seed=10)
    x[0:10] = 0
    x[10:20] = 0
    x[torch.arange(10, 20), torch.arange(10, 20) * 97] = torch.linspace(1e-3, 50.0, 10)
    x[20:30] *= 6.5e4 / x[20:30].amax(dim=1, keepdim=True)
    x[30:40] *= 1e6 / x[30:40].amax(dim=1, keepdim=True)
    assert float(x[30:40].max()) > 65504
    x[40:50] = ramp_rows(x[40:50])
    x[50:60, 1000:] *= 1e3
    got = run_encoder(x, ws, bs, engine)
    assert_enc_close(got, x, ws, bs, f'{engine} degenerate rows')


@pytest.mark.parametrize('bad', ('nan row', 'inf row', 'nan weight'))
def test_node_encoder_non_finite_input_sets_the_status(bad):
    """A NaN / inf row or a NaN weight: 'tc' raises OverflowError, 'auto' warns and returns the fp32 chain's
    result, and with status= the flag is left for the caller."""
    ws, bs = enc_params(2048, seed=11)
    x = enc_input(150, 2048, seed=12)
    if bad == 'nan row':
        x[37, 5] = float('nan')
    elif bad == 'inf row':
        x[140, 2000] = float('inf')
    else:
        ws[0][3, 17] = float('nan')
    with pytest.raises(OverflowError):
        encode(x, ws, bs, 'tc')
    with pytest.warns(UserWarning, match='fp32 kernels'):
        auto = encode(x, ws, bs, 'auto')
    ref = encode(x, ws, bs, 'fp32')
    assert torch.equal(auto.isnan(), ref.isnan()) and torch.equal(torch.nan_to_num(auto), torch.nan_to_num(ref))
    st = torch.zeros(1, dtype=torch.int32, device=dev())
    with torch.no_grad():
        ops.node_encoder(x.to(dev()), [w.to(dev()) for w in ws], [b.to(dev()) for b in bs], engine='tc', status=st)
    assert int(st.item()) & 1


@pytest.mark.parametrize('k0', (64, 128, 192, 2048, 4096))
def test_node_encoder_widths_on_the_tensor_cores(k0):
    """Beyond the shipped K = 2048 the bar grows with K: the fp32 accumulator of the MMAs truncates once per MMA, so
    its error grows with the number of K steps (2.7e-5 measured at K = 4096 on a B200, scaled or not)."""
    ws, bs = enc_params(k0, seed=13)
    x = pow2(enc_input(300, k0, seed=14), -12)
    bs = [pow2(b, -12) for b in bs]
    assert_enc_close(encode_tc(x, ws, bs), x, ws, bs, f'k0 {k0}', tol=ENC_TOL * max(1, k0 / 2048))


@pytest.mark.parametrize('case', ('k0=100', 'odd offset'))
def test_node_encoder_gates_to_the_fp32_chain(case):
    """k0 not a multiple of 64, or x off 16-byte alignment: even engine='tc' runs the fp32 chain (the tensor-core
    launcher, which clears the status word, is never called), bit for bit engine='fp32'."""
    k0 = 100 if case == 'k0=100' else 2048
    ws, bs = enc_params(k0, seed=15)
    x = enc_input(200, k0, seed=16)
    xd = x.to(dev())
    if case == 'odd offset':
        buf = torch.empty(x.numel() + 1, device=dev())
        xd = buf[1:].view(x.shape)
        xd.copy_(x)
        assert xd.is_contiguous() and xd.data_ptr() % 16 != 0
    st = torch.full((1,), SENTINEL, dtype=torch.int32, device=dev())
    with torch.no_grad():
        got = ops.node_encoder(xd, [w.to(dev()) for w in ws], [b.to(dev()) for b in bs], engine='tc', status=st).cpu()
    assert int(st.item()) == SENTINEL, 'the tensor-core launcher ran'
    assert torch.equal(got, encode(x, ws, bs, 'fp32'))
    assert_enc_close(got, x, ws, bs, case)


@pytest.mark.parametrize('which', ('1', '129', 'persistent'))
def test_node_encoder_row_counts_at_small_scale(which):
    """One row, a partial second tile, and more than one tile per CTA group (the mbarrier parities and the weight
    stream carry over), at x * 2^-16."""
    n = persistent_sizes()[0] if which == 'persistent' else int(which)
    if which == 'persistent':
        assert n > 2 * sms() * TC_TILE
    ws, bs = enc_params(2048, seed=17)
    x = pow2(enc_input(n, 2048, seed=18), -16)
    bs = [pow2(b, -16) for b in bs]
    assert_enc_close(encode_tc(x, ws, bs), x, ws, bs, f'n {n}')


@pytest.mark.parametrize('engine', ('tc', 'auto'))
def test_forward_with_tiny_node_features_matches_the_oracle(engine):
    """A window whose node features are * 2^-16 and whose node-encoder layer-0 weights are * 2^16: x_init is the same
    in exact arithmetic, but the encoder sees tiny inputs.  Logits against the oracle in fp64; 'auto' must stay
    on the tensor cores (no fallback warning)."""
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    win = synth.make_window(T=15, D=150, k=50, seed=4, node_feats='pooled')
    ds = default_dataset_params(top_k_nns=50, frames_per_graph=15)
    mp = default_graph_model_params(12, 11)
    P = synth.make_params(mp, seed=9, gain=1.25, core_only=True)
    key = 'encoder.node_model.fc_layers.0.weight'
    assert tuple(P[key].shape) == (128, 2048)
    P[key] = pow2(P[key], 16)
    x = pow2(win.x, -16)
    ref_g = graph_ref.build_graph(win.frame, win.reid, synth.det_columns(win), win.fps, ds)
    with torch.no_grad():
        ref = mpn_ref.mpn_forward({k: v.double() for k, v in P.items()}, mp, x.double(), ref_g['edge_index'],
                                  ref_g['edge_attr'].double())
    g = MOTGraph.from_tensors(synth.det_columns(win), win.reid, x, None, {'fps': win.fps}, ds).construct_graph_object()
    assert torch.equal(g.edge_index.cpu(), ref_g['edge_index'])
    model = make_model(mp, P, engine)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter('always')
        with torch.no_grad():
            out = model(g)
    assert not [w for w in caught if 'fp32 kernels' in str(w.message)], 'the forward left the tensor cores'

    got = torch.stack([t.view(-1) for t in out['classified_edges']]).cpu().numpy()
    exp = torch.stack([t.view(-1) for t in ref['classified_edges']]).numpy()
    assert_logits_close(got, exp, f'tiny node features, {engine}')


# ------------------------------------------------------------------ average pool
POOL_HW = (2, 4, 6, 8, 12, 16, 32, 64, 128, 256)
POOL_THREADS, POOL_UNROLL = 256, 4          # csrc/encoder.cu: avgpool_vec_kernel block size and loads in flight


def pool_group(hw):
    """GROUP of avgpool_vec_kernel for this hw, or None for the scalar kernel."""
    vec = hw // 4
    return vec if hw % 4 == 0 and 1 <= vec <= 32 and vec & (vec - 1) == 0 else None


def pool_rows(hw):
    """A row count past one UNROLL * stride sweep of the capped grid, not a multiple of ROWS_PER_WARP."""
    group = pool_group(hw)
    if group is None:
        cap = 8 * sms() * POOL_THREADS            # one row per thread, grid capped at 8 blocks per SM
        return cap + 37, cap
    rows_per_warp = 32 // group
    sweep = POOL_UNROLL * 16 * sms() * (POOL_THREADS // 32) * rows_per_warp     # grid capped at 16 blocks per SM
    return sweep + 3 * rows_per_warp + (rows_per_warp > 1), sweep


def pool_bar(x, hw, vector):
    """Per row: (ceil(log2 hw) + 2) u mean|x| for the vector kernel's tree, hw u mean|x| for the scalar loop."""
    f = (math.ceil(math.log2(hw)) + 2) if vector else hw
    return f * U * x.double().abs().mean(dim=-1)


def check_pool(x, got, hw, vector, what):
    rows = x.reshape(-1, hw)
    ref = rows.double().mean(dim=-1)
    err = (got.reshape(-1).double().cpu() - ref).abs()
    bar = pool_bar(rows, hw, vector)
    bad = err > bar
    assert not bad.any(), f'{what}: {int(bad.sum())} rows off, worst {float((err / bar.clamp(min=1e-300)).max()):.2f} x the bar'


@pytest.mark.parametrize('data', ('randn', 'offset 1e4'))
@pytest.mark.parametrize('hw', POOL_HW)
def test_avgpool_against_fp64(hw, data):
    """Every GROUP of the vector kernel and the scalar kernel (hw 2, 6, 12 and 256); row counts past one sweep of the
    capped grid and not a multiple of ROWS_PER_WARP; rows of 1e4 + N(0,1), where the sum cancels nothing but
    rounds at 1e4."""
    rows, sweep = pool_rows(hw)
    assert rows > sweep
    group = pool_group(hw)
    if group is not None:
        assert rows % (32 // group) != 0 or group == 32
    g = torch.Generator().manual_seed(hw)
    x = torch.randn(rows, 1, hw, 1, generator=g)
    if data != 'randn':
        x += 1e4
    got = ops.avgpool(x.to(dev()))
    check_pool(x, got, hw, group is not None, f'hw {hw} {data}')
    small = x[:37]
    check_pool(small, ops.avgpool(small.to(dev())), hw, group is not None, f'hw {hw} {data}, 37 rows')


def test_avgpool_unaligned_input_takes_the_scalar_kernel():
    g = torch.Generator().manual_seed(20)
    x = torch.randn(300, 7, 4, 4, generator=g) + 1e4
    buf = torch.empty(x.numel() + 1, device=dev())
    xd = buf[1:].view(x.shape)
    xd.copy_(x)
    assert xd.is_contiguous() and xd.data_ptr() % 16 != 0
    check_pool(x, ops.avgpool(xd), 16, False, 'odd offset')


def test_avgpool_into_a_slice_of_a_larger_buffer():
    g = torch.Generator().manual_seed(21)
    x = torch.randn(50, 64, 8, 4, generator=g)
    big = torch.full((70, 64), float('nan'), device=dev())
    out = big[7:57]
    assert out.is_contiguous()
    res = ops.avgpool(x.to(dev()), out=out)
    assert res.data_ptr() == out.data_ptr()
    check_pool(x, out, 32, True, 'out= slice')
    assert big[:7].isnan().all() and big[57:].isnan().all(), 'the pool wrote outside its slice'


def test_avgpool_hw_one_and_no_rows():
    g = torch.Generator().manual_seed(22)
    x = torch.randn(9, 5, 1, 1, generator=g)
    assert torch.equal(ops.avgpool(x.to(dev())).cpu(), x.reshape(9, 5))
    out = torch.empty(9, 5, device=dev())
    ops.avgpool(x.to(dev()), out=out)
    assert torch.equal(out.cpu(), x.reshape(9, 5))
    empty = ops.avgpool(torch.empty(0, 5, 8, 4, device=dev()))
    assert tuple(empty.shape) == (0, 5)


# ------------------------------------------------------------------ edge encoder
EDGE_TOL = 1e-5


def edge_params(dims, seed):
    g = torch.Generator().manual_seed(seed)
    ws = [uniform((o, i), i ** -0.5, g) for i, o in zip(dims[:-1], dims[1:])]
    bs = [uniform((o,), i ** -0.5, g) for i, o in zip(dims[:-1], dims[1:])]
    return ws, bs


def mlp64(x, ws, bs):
    """(fp64 output, fp64 magnitude |W|...|x| + |b| of the last layer: the scale of its rounding errors)."""
    h, m = x.double(), x.double().abs()
    for w, b in zip(ws, bs):
        w, b = w.double(), b.double()
        h = torch.relu(h @ w.T + b)
        m = m @ w.abs().T + b.abs()
    return h, m


def random_edges(n, e, seed):
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(n, (e,), generator=g)
    b = (a + 1 + torch.randint(n - 1, (e,), generator=g)) % n
    return torch.stack((a, b))


def run_edge_encoder(attr, ei, n, ws, bs):
    lay = ops.edge_layout(ei.to(dev()), n)
    assert lay.num_edges == ei.shape[1]
    with torch.no_grad():
        out = ops.edge_encoder(attr.to(dev()), lay, [w.to(dev()) for w in ws], [b.to(dev()) for b in bs])
    return out.cpu(), lay.slot_edge[:lay.num_edges].long().cpu()


def check_edge(attr, ei, n, ws, bs, what):
    """In slot order, per row |got - ref| <= 1e-5 * max_j (|W| ... |x| + |b|)_j."""
    got, slot_edge = run_edge_encoder(attr, ei, n, ws, bs)
    ref, mag = mlp64(attr, ws, bs)
    ref, mag = ref[slot_edge], mag[slot_edge]
    assert got.shape == ref.shape
    err = (got.double() - ref).abs()
    scale = mag.amax(dim=1, keepdim=True)
    bad = err > EDGE_TOL * scale
    assert not bad.any(), f'{what}: {int(bad.any(dim=1).sum())} rows off, worst {float((err / scale).max()):.3e}'
    return got, slot_edge


@pytest.mark.parametrize('case', ('one edge', 'grid stride'))
def test_edge_encoder_edge_counts(case):
    """E = 1, and E beyond the capped grid (4 * SMs blocks of 256 threads): the grid-stride loop."""
    ws, bs = edge_params((6, 18, 18, 16), seed=30)
    if case == 'one edge':
        ei, n = torch.tensor([[0], [1]]), 2
    else:
        cap = 4 * sms() * 256
        n, e = 50000, 2 * cap + 3
        ei = random_edges(n, e, seed=31)
        assert ei.shape[1] > cap
    g = torch.Generator().manual_seed(32)
    attr = torch.randn(ei.shape[1], 6, generator=g) * 3
    check_edge(attr, ei, n, ws, bs, case)


def test_edge_encoder_large_features_and_dead_rows():
    """Features up to +-1e4, and rows whose every ReLU is dead: with W0[:, 0] > 0.1 and b1 < 0, a row with
    feature 0 at -1e4 has h1 = h2 = 0 and must give exactly ReLU(b2)."""
    ws, bs = edge_params((6, 18, 18, 16), seed=33)
    ws[0][:, 0] = ws[0][:, 0].abs() + 0.1
    bs[1] = -bs[1].abs() - 1e-3
    n, e = 3000, 20000
    ei = random_edges(n, e, seed=34)
    g = torch.Generator().manual_seed(35)
    attr = (torch.rand(e, 6, generator=g) * 2 - 1) * torch.tensor([1.0, 10.0, 1e2, 1e3, 1e4, 1.0])
    dead = torch.arange(e) % 5 == 0
    attr[dead] = torch.rand(int(dead.sum()), 6, generator=g) * 2 - 1
    attr[dead, 0] = -1e4
    got, slot_edge = check_edge(attr, ei, n, ws, bs, 'large features')
    dead_slots = dead[slot_edge]
    assert int(dead_slots.sum()) > 0
    assert torch.equal(got[dead_slots], torch.relu(bs[2]).expand(int(dead_slots.sum()), 16))


def test_edge_encoder_no_edges():
    ws, bs = edge_params((6, 18, 18, 16), seed=36)
    lay = ops.edge_layout(torch.empty(2, 0, dtype=torch.int64, device=dev()), 3)
    out = ops.edge_encoder(torch.empty(0, 6, device=dev()), lay, [w.to(dev()) for w in ws], [b.to(dev()) for b in bs])
    assert tuple(out.shape) == (0, 16)


def test_edge_encoder_other_widths_take_gather_and_linear():
    """6-32-16 is not the fused kernel's shape: gather_rows + linear_kernel, whose k (6, 32) and o (32, 16) are not
    multiples of the 16-deep K slab or the 64-wide tile, over more than one 64-row tile."""
    ws, bs = edge_params((6, 32, 16), seed=37)
    n, e = 400, 1000
    ei = random_edges(n, e, seed=38)
    g = torch.Generator().manual_seed(39)
    attr = (torch.rand(e, 6, generator=g) * 2 - 1) * 1e3
    check_edge(attr, ei, n, ws, bs, '6-32-16')


# ------------------------------------------------------------------ edge features
LOG_COLS = (3, 4)


def det_table(n, seed, frame_max, aspect=False, equal_h=False):
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.rand(*s, generator=g, dtype=torch.float64)    # noqa: E731
    frame = torch.sort(torch.randint(0, frame_max + 1, (n,), generator=g)).values.double()
    h = 20.0 + 400.0 * rnd(n)
    w = 0.4 * h * (0.5 + rnd(n))
    if aspect:
        w[::2] = h[::2] * 1e3
        h[1::2] = w[1::2] * 1e3
    if equal_h:
        h[:] = 137.25
    fx = (rnd(n) * 2 - 1) * 3000.0
    fy = (rnd(n) * 2 - 1) * 2000.0
    return {'frame': frame.numpy(), 'bb_height': h.numpy(), 'bb_width': w.numpy(), 'feet_x': fx.numpy(), 'feet_y': fy.numpy()}


def check_edge_feats(pairs, cols, fps, with_rd):
    p = pairs.shape[1]
    t = {k: torch.from_numpy(v).float().to(dev()) for k, v in cols.items()}
    rd = torch.rand(p, generator=torch.Generator().manual_seed(p)) * 10 if with_rd else None
    attr, eidx = ops.edge_feats_assemble(pairs.to(dev()), t['frame'], t['bb_height'], t['bb_width'], t['feet_x'],
                                         t['feet_y'], fps, None if rd is None else rd.to(dev()))
    attr, eidx = attr.cpu(), eidx.cpu()
    assert attr.shape == (2 * p, 6 if with_rd else 5)
    assert torch.equal(eidx, torch.cat((pairs, pairs.flip(0)), dim=1))
    assert torch.equal(attr[:p], attr[p:])
    ref = graph_ref.edge_geometry(pairs, cols, fps)
    names = ('secs_time_dists', 'norm_feet_x_dists', 'norm_feet_y_dists', 'bb_height_dists', 'bb_width_dists')
    for c, name in enumerate(names):
        if c in LOG_COLS:
            err = (attr[:p, c].double() - ref[name].double()).abs()
            assert (err <= 2e-6 * ref[name].double().abs()).all(), f'{name}: worst {float(err.max()):.3e}'
        else:
            assert torch.equal(attr[:p, c], ref[name]), name
    if with_rd:
        assert torch.equal(attr[:p, 5], rd)
    return attr[:p]


@pytest.mark.parametrize('fps', (30.0, 29.97, 7.5))
def test_edge_feats_frames_fps_and_signs(fps):
    """Frame numbers up to 10^6, fps 30 / 29.97 / 7.5, negative feet coordinates, attr_dim 5 and 6."""
    cols = det_table(600, seed=40, frame_max=10 ** 6)
    assert cols['frame'].max() > 9e5 and (cols['feet_x'] < 0).any()
    pairs = graph_ref.time_valid_pairs(torch.from_numpy(cols['frame']).long())
    for with_rd in (False, True):
        check_edge_feats(pairs, cols, fps, with_rd)


def test_edge_feats_equal_heights_and_extreme_aspect_ratios():
    cols = det_table(300, seed=41, frame_max=50, equal_h=True)
    pairs = graph_ref.time_valid_pairs(torch.from_numpy(cols['frame']).long())
    attr = check_edge_feats(pairs, cols, 30.0, False)
    assert torch.equal(attr[:, 3], torch.zeros(pairs.shape[1])), 'log ratio of equal heights must be exactly 0'
    cols = det_table(300, seed=42, frame_max=50, aspect=True)
    pairs = graph_ref.time_valid_pairs(torch.from_numpy(cols['frame']).long())
    attr = check_edge_feats(pairs, cols, 30.0, True)
    assert float(attr[:, 4].abs().max()) > 6.0                            # |log(1e3 ratios)|


def test_edge_feats_single_pair():
    cols = det_table(2, seed=43, frame_max=3)
    cols['frame'][:] = (4.0, 1.0e6)
    pairs = torch.tensor([[0], [1]])
    for with_rd in (False, True):
        check_edge_feats(pairs, cols, 29.97, with_rd)


# ------------------------------------------------------------------ pair distance
DIST_DIMS = (1, 3, 4, 5, 31, 32, 33, 100, 128, 256, 2048)
EPS = 1e-6


def dist_bar(reid, pairs, dim):
    """(fp64 reference, per-pair bar).  The bar is (dim/32 + 6) 2^-23 relative to ||a - b + eps||; where a - b cancels
    eps the rounding of a - b (relative to |a - b|) governs, so the scale there is ||(|a - b| + eps)||^2 / ref."""
    ref, mag = [], []
    for s in range(0, pairs.shape[1], 2048):
        d = reid[pairs[0, s:s + 2048]].double() - reid[pairs[1, s:s + 2048]].double()
        ref.append((d + EPS).norm(dim=1))
        mag.append((d.abs() + EPS).norm(dim=1))
    ref, mag = torch.cat(ref), torch.cat(mag)
    return ref, (dim / 32 + 6) * 2.0 ** -23 * mag * mag / ref


def dist_case(dim, scale, seed, n_base=180):
    """n_base random embeddings and 20 near copies (identical, or off by 1e-8 relative) of the first 20; every
    pair i < j."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(n_base, dim, generator=g)
    near = base[:20].clone()
    near[10:] += 1e-8 * torch.randn(10, dim, generator=g)
    reid = pow2(torch.cat((base, near)), scale)
    n = reid.shape[0]
    i, j = torch.triu_indices(n, n, offset=1)
    return reid.contiguous(), torch.stack((i, j))


@pytest.mark.parametrize('dim', DIST_DIMS)
def test_pair_dist_against_fp64(dim):
    """Embedding scales 2^-20 ... 2^13 and near-identical pairs, with more pairs than the capped grid has warps."""
    warps = 16 * sms() * 8                        # grid capped at 16 blocks of 8 warps per SM, one warp per pair
    n_base = max(180, int(math.sqrt(2 * warps)) - 18)
    for scale in (-20, -10, 0, 13):
        reid, pairs = dist_case(dim, scale, seed=dim, n_base=n_base)
        assert pairs.shape[1] > warps
        got = ops.pair_reid_dist(reid.to(dev()), pairs.to(dev())).cpu().double()
        ref, bar = dist_bar(reid, pairs, dim)
        err = (got - ref).abs()
        assert (err <= bar).all(), f'dim {dim} scale 2^{scale}: worst {float((err / bar).max()):.2f} x the bar'
        assert (pairs[1] >= n_base).any()


@pytest.mark.parametrize('dim', (128, 256))
def test_pair_dist_unaligned_embeddings_equal_the_aligned_copy(dim):
    """A contiguous view at an odd element offset (4-byte aligned only) gives the same bits as the aligned copy."""
    reid, pairs = dist_case(dim, 0, seed=50 + dim)
    buf = torch.empty(reid.numel() + 1, device=dev())
    view = buf[1:].view(reid.shape)
    view.copy_(reid)
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    aligned = ops.pair_reid_dist(reid.to(dev()), pairs.to(dev()))
    assert torch.equal(ops.pair_reid_dist(view, pairs.to(dev())), aligned)


# ------------------------------------------------------------------ scans
SCAN_CHUNK, SCAN_TOTALS_BLOCK = 2048, 1024      # csrc/common.cu: values per scan chunk, threads scanning the chunk totals
BIG_SCAN = SCAN_CHUNK * SCAN_TOTALS_BLOCK


@pytest.mark.parametrize('mask', ('random', 'zeros', 'ones'))
@pytest.mark.parametrize('n', (2047, 2048, 2049, BIG_SCAN, BIG_SCAN + 1))
def test_compact_pairs_equals_boolean_indexing(n, mask):
    g = torch.Generator().manual_seed(n)
    pairs = torch.stack((torch.arange(n), torch.randint(1 << 40, (n,), generator=g)))
    dist = torch.randn(n, generator=g)
    keep = {'random': torch.rand(n, generator=g) < 0.3, 'zeros': torch.zeros(n, dtype=torch.bool),
            'ones': torch.ones(n, dtype=torch.bool)}[mask]
    got, gd = ops.compact_pairs(pairs.to(dev()), keep.to(dev()), dist.to(dev()))
    assert torch.equal(got.cpu(), pairs[:, keep]) and torch.equal(gd.cpu(), dist[keep])
    assert torch.equal(ops.compact_pairs(pairs.to(dev()), keep.to(dev())).cpu(), pairs[:, keep])
    if n > BIG_SCAN:
        assert math.ceil(n / SCAN_CHUNK) > SCAN_TOTALS_BLOCK


WINDOW_FRAMES = torch.tensor([[0, 0, 1, 1], [0, 1, 1, 1], [0, 0, 0, 1], [1, 0, 1, 0], [5, 2, 2, 5]])


def test_time_valid_pairs_over_many_small_windows():
    """More than 2,048 * 1,024 nodes in windows of 4 nodes in 2 frames (patterns above): about one pair per node.
    Each window must give graph_ref.time_valid_pairs of its 4 frames, offset by its first node."""
    w = BIG_SCAN // 4 + 3
    n = 4 * w
    assert math.ceil(n / SCAN_CHUNK) > SCAN_TOTALS_BLOCK
    g = torch.Generator().manual_seed(60)
    pat = torch.randint(WINDOW_FRAMES.shape[0], (w,), generator=g)
    frame = (WINDOW_FRAMES[pat] + 10 * torch.arange(w)[:, None]).reshape(-1)
    ptr = torch.arange(0, n + 1, 4)
    got = ops.time_valid_pairs(frame.to(dev()), -1, ptr.to(dev())).cpu()
    # graph_ref per pattern (it depends on the frame differences only), laid out window by window
    refs = [graph_ref.time_valid_pairs(f) for f in WINDOW_FRAMES]
    counts = torch.tensor([r.shape[1] for r in refs])
    table = torch.zeros(len(refs), 2, int(counts.max()), dtype=torch.int64)
    for k, r in enumerate(refs):
        table[k, :, :r.shape[1]] = r
    per = counts[pat]
    win = torch.repeat_interleave(torch.arange(w), per)
    local = torch.arange(int(per.sum())) - torch.repeat_interleave(torch.cumsum(per, 0) - per, per)
    exp = table[pat[win], :, local].T + 4 * win
    assert got.shape == exp.shape and torch.equal(got, exp)
