"""GPU tests of the attentive aggregation (csrc/attention.cu: ``ops.attn_aggregate``, ``ops.attn_aggregate_backward``)
per element against an fp64 restatement, at the softmax sharpness, degrees, map sizes and non-finite logits where the
kernels go wrong.  Each test asserts that its case reaches the regime it names.

The restatement (``attn_ref``) evaluates the oracle's functions (``mpn_ref.segment_softmax`` / ``segment_add``) in fp64
on the kernels' fp32 inputs.  Its logit gradient is

    d_q = w_q (dw_q - S)                                                      for q != q*
    d_q* = w_q* sum_{p != q*} w_p (dw_q* - dw_p) - w_phi sum_{p != q*} w_p dw_p

with dw_q = <G[row], z[col_q]>, S = sum_p w_p dw_p, w_phi = 1e-12 / (s + 1e-12) and q* the slot of the segment's
largest logit (the lowest edge id among ties).  This is the gradient of the oracle, including its path through the
segment max, written so that nothing cancels when w_q* -> 1.
test_attention_references.py pins it to that autograd on the CPU.

Bars, per element, with A_q = sum_i |G_i z[col_q, i]|:

* flows: |d| <= tol sum_q w_q |z[col_q, i]|;
* d_z: |d| <= tol sum_q w_q |G[row_q]|, the same sums with absolute values;
* d_logits: |d| <= tol w_q (|sum_{p != q} w_p (dw_q - dw_p)| + sum_{p != q} w_p (A_q + A_p) + w_phi (|dw_q| + A_q)):
  the conditioning of the function in its inputs, with the absolute value taken of the sum rather than of each term
  (which can only tighten it).  For q* the w_phi term is w_phi sum_{p != q*} w_p (|dw_p| + A_p), the conditioning of
  its own w_phi term: w_phi |dw_q*| would exceed the whole gradient beyond a lead of about 30;
* each bar has an absolute floor at the scale 2^-126 tol, for weights and products in the subnormal range.

tol = (BASE_ULPS + L) u (u = 2^-24), where L is the length of the longest chain of sequential fp32 additions behind the
element (the a-priori bound of a recursive sum grows with it): the weights' softmax sum, ceil(deg / 256) per thread,
for every output; plus the segment's degree for the flows (one thread adds the slots in order), the column's slot
count for d_z, and feat / 32 + 5 for d_logits (the per-lane dot products and their tree).  BASE_ULPS covers expf,
the trees of the sums, the division and the products.  The worst measured ratio to the bar is printed per case.

Logits lie on a 2^-10 grid below 2^13, so that l - max is exact in fp32 and the only roundings of the forward are
expf, the sums and the division.
"""
import math

import numpy as np
import pytest
import torch

from mpntrackseg_b200 import ops
from oracle import mpn_ref
from test_cuda_parity import dev
from test_kernel_boundaries import hub_graph

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BASE_ULPS = 32
TINY = 2.0 ** -126
ATT_MAX_DEG = 1024          # csrc/attention.cu: slots per node and direction cached in shared memory per pass
GRID = 2.0 ** -10


# ------------------------------------------------------------------ fp64 restatement
def segments(ei, n):
    """Segment of each edge: 2 row + 1 for the flow_out group (row < col), 2 row for flow_in."""
    return 2 * ei[0] + (ei[0] < ei[1]).long(), 2 * n


def seg_sum(v, seg, nseg):
    return mpn_ref.segment_add(v, seg, nseg)


def softmax_parts(l64, seg, nseg):
    """(w, w_phi per edge, q* per segment (-1: none), segment max) of exp(l - max) / (sum + 1e-12)."""
    m = l64.new_full((nseg,), float('-inf')).scatter_reduce(0, seg, l64, 'amax', include_self=True)
    ex = (l64 - m[seg]).exp()
    den = seg_sum(ex, seg, nseg) + 1e-12
    w, wphi = ex / den[seg], 1e-12 / den[seg]
    e = l64.shape[0]
    cand = torch.where(l64 == m[seg], torch.arange(e), e)
    qs = torch.full((nseg,), e, dtype=torch.long).scatter_reduce(0, seg, cand, 'amin', include_self=True)
    return w, wphi, torch.where(qs < e, qs, -1), m


def softmax_backward_ref(l64, seg, nseg, dw):
    """d loss / d logits of the segment softmax for the weight gradients ``dw`` (the formula of the module docstring)."""
    w, wphi, qs, _ = softmax_parts(l64, seg, nseg)
    e = l64.shape[0]
    S = seg_sum(w * dw, seg, nseg)
    d = w * (dw - S[seg])
    has = qs[seg] >= 0
    q_of = torch.where(has, qs[seg], 0)
    other = has & (torch.arange(e) != q_of)                  # p != q* of its segment
    zero = torch.zeros_like(dw)
    direct = seg_sum(torch.where(other, w * (dw[q_of] - dw), zero), seg, nseg)
    rest = seg_sum(torch.where(other, w * dw, zero), seg, nseg)
    star = qs[qs >= 0]
    sseg = seg[star]
    d[star] = w[star] * direct[sseg] - wphi[star] * rest[sseg]
    return d


def dots(G, z, rows, cols, chunk=1 << 24):
    """(dw_q = <G[rows_q], z[cols_q]>, A_q = sum_i |G[rows_q, i] z[cols_q, i]|) in fp64, in chunks of edges."""
    e, feat = rows.shape[0], G.shape[1]
    dw, A = torch.empty(e, dtype=torch.float64), torch.empty(e, dtype=torch.float64)
    step = max(1, chunk // max(feat, 1))
    for a in range(0, e, step):
        p = G[rows[a:a + step]].double() * z[cols[a:a + step]].double()
        dw[a:a + step], A[a:a + step] = p.sum(1), p.abs().sum(1)
    return dw, A


def attn_ref(ei, n, z, logits, g_in, g_out):
    """fp64 outputs of the aggregation and its backward with their per-element bars (flattened maps)."""
    src, dst = ei[0], ei[1]
    z2, gi, go = z.reshape(n, -1), g_in.reshape(n, -1), g_out.reshape(n, -1)
    feat = z2.shape[1]
    seg, nseg = segments(ei, n)
    l64 = logits.reshape(-1).double()
    w, wphi, qs, _ = softmax_parts(l64, seg, nseg)
    out = src < dst
    r = {}
    z64 = z2.double()
    deg_seg = seg_sum(torch.ones_like(l64), seg, nseg)
    tol_w = U * (BASE_ULPS + torch.ceil(deg_seg / 256))          # per segment
    for name, sel, d in (('out', out, 1), ('in', ~out, 0)):
        zc, ws = z64[dst[sel]], w[sel].view(-1, 1)
        tol = (tol_w[2 * torch.arange(n) + d] + U * deg_seg[2 * torch.arange(n) + d]).view(-1, 1)
        r['flow_' + name] = seg_sum(zc * ws, src[sel], n)
        r['flow_' + name + '_bar'] = tol * (seg_sum(zc.abs() * ws, src[sel], n) +
                                            TINY * (seg_sum(zc.abs(), src[sel], n) + seg_sum(torch.ones_like(ws), src[sel], n)))
    # d_z[c] = sum over the edges with col = c of w G_dir[row]
    Gsel = torch.where(out.view(-1, 1), go[src].double(), gi[src].double()) if ei.shape[1] else gi[:0].double()
    ws = w.view(-1, 1)
    cdeg = seg_sum(torch.ones_like(l64), dst, n)
    tol = (U * (BASE_ULPS + torch.ceil(deg_seg.max() / 256) + cdeg)).view(-1, 1) if ei.shape[1] else U
    r['dz'] = seg_sum(Gsel * ws, dst, n)
    r['dz_bar'] = tol * (seg_sum(Gsel.abs() * ws, dst, n) + TINY * (seg_sum(Gsel.abs(), dst, n) + cdeg.view(-1, 1)))
    del Gsel
    G_edge_rows = src + n * out.long()                       # rows of cat(g_in, g_out)
    dw, A = dots(torch.cat((gi, go)), z2, G_edge_rows, dst)
    r['dl'] = softmax_backward_ref(l64, seg, nseg, dw)
    # bar.  sum_{p != q} of w_p, w_p A_p, w_p (dw_q - dw_p): as totals minus the own term where w_q <= 1/2 or so, summed
    # over the other slots directly for q* (where the totals minus w_q* would cancel)
    W, S, WA = seg_sum(w, seg, nseg)[seg], seg_sum(w * dw, seg, nseg)[seg], seg_sum(w * A, seg, nseg)[seg]
    star = qs[qs >= 0]
    is_star = torch.zeros_like(w, dtype=torch.bool)
    is_star[star] = True
    other = (qs[seg] >= 0) & ~is_star
    zero = torch.zeros_like(w)
    q_of = torch.where(qs[seg] >= 0, qs[seg], 0)
    W_ex = torch.where(is_star, seg_sum(torch.where(other, w, zero), seg, nseg)[seg], W - w)
    WA_ex = torch.where(is_star, seg_sum(torch.where(other, w * A, zero), seg, nseg)[seg], WA - w * A)
    diff = torch.where(is_star, seg_sum(torch.where(other, w * (dw[q_of] - dw), zero), seg, nseg)[seg],
                       dw * (W - w) - (S - w * dw))
    phi = torch.where(is_star, seg_sum(torch.where(other, w * (dw.abs() + A), zero), seg, nseg)[seg], dw.abs() + A)
    cond = diff.abs() + W_ex * A + WA_ex + wphi * phi
    deg = deg_seg[seg]
    tol = tol_w[seg] + U * (math.ceil(feat / 32) + 5)
    r['dl_bar'] = tol * (w * cond + TINY * (1 + deg * A + seg_sum(A, seg, nseg)[seg]))
    r.update(w=w, wphi=wphi, qs=qs, seg=seg, nseg=nseg, dw=dw, A=A, feat=feat)
    return r


# ------------------------------------------------------------------ GPU side
def col_perm(lay, n):
    """The slots sorted by column and their row pointer, as CoreTrainer.prepare builds them."""
    scol = lay.slot_col[:lay.num_edges]
    perm_c = torch.argsort(scol, stable=True).to(torch.int32)
    ptr_c = torch.zeros(n + 1, dtype=torch.int32, device=dev())
    ptr_c[1:] = torch.cumsum(torch.bincount(scol.long(), minlength=n), 0).to(torch.int32)
    return perm_c, ptr_c


def run_gpu(ei, n, z, logits, g_in, g_out):
    lay = ops.edge_layout(ei.to(dev()), n)
    perm_c, ptr_c = col_perm(lay, n)
    zd, ld = z.to(dev()), logits.to(dev())
    fin, fout = ops.attn_aggregate(zd, lay, ld)
    dz, dl = ops.attn_aggregate_backward(zd, lay, ld, g_in.to(dev()), g_out.to(dev()), perm_c, ptr_c)
    torch.cuda.synchronize()
    return {'flow_in': fin.cpu(), 'flow_out': fout.cpu(), 'dz': dz.cpu(), 'dl': dl.cpu()}


def ratio(got, ref, bar):
    """Per element |got - ref| / bar; NaN must sit where the reference has NaN, infinities must be equal."""
    got, ref, bar = got.reshape(-1).double(), ref.reshape(-1).double(), bar.reshape(-1)
    nan_g, nan_r = torch.isnan(got), torch.isnan(ref)
    assert torch.equal(nan_g, nan_r), f'NaN at {int((nan_g & ~nan_r).sum())} extra / {int((nan_r & ~nan_g).sum())} missing places'
    inf_r = torch.isinf(ref)
    assert torch.equal(got[inf_r], ref[inf_r]), 'infinities differ'
    fin = ~nan_r & ~inf_r
    diff = (got[fin] - ref[fin]).abs()
    return torch.where(diff == 0, torch.zeros_like(diff), diff / bar[fin])       # a zero bar asks for equality


def assert_close(got, r, what):
    """Every output within its bar; returns the worst ratio of each."""
    worst = {}
    for k in ('flow_in', 'flow_out', 'dz', 'dl'):
        q = ratio(got[k], r[k], r[k + '_bar'])
        worst[k] = float(q.max()) if q.numel() else 0.0
    print(what, {k: f'{v:.3g}' for k, v in worst.items()})
    bad = {k: v for k, v in worst.items() if v > 1}
    assert not bad, (what, bad)
    return worst


def old_formula(r):
    """d_logits = w (dw - S) with w, dw rounded to fp32 and S summed in fp32: the backward before the dominant slot got
    its own sum (the test's emulation, with exact dot products)."""
    w32, dw32 = r['w'].float(), r['dw'].float()
    S32 = seg_sum(w32 * dw32, r['seg'], r['nseg'])
    return (w32 * (dw32 - S32[r['seg']])).double()


# ------------------------------------------------------------------ cases
def grid_logits(e, g, lo=-1.0, hi=1.0):
    return torch.round((torch.rand(e, generator=g, dtype=torch.float64) * (hi - lo) + lo) / GRID) * GRID


def pick_per_segment(seg, nseg, g, k=1):
    """k distinct random edges of each segment (fewer where the segment is smaller), as a list of index tensors."""
    key = torch.rand(seg.shape[0], generator=g, dtype=torch.float64)
    order = torch.argsort(seg * 2.0 + key)                 # by segment, random within
    s = seg[order]
    start = torch.zeros(nseg + 1, dtype=torch.long)
    start[1:] = torch.cumsum(torch.bincount(s, minlength=nseg), 0)
    rank = torch.arange(seg.shape[0]) - start[s]
    return [order[rank == i] for i in range(k)]


def sharp_logits(ei, n, lead, seed):
    """Base logits uniform on [-1, 1]; one edge per segment 1 + lead (number), or: 'tie' two edges at 4,
    'ulp' one at 4 and one at the next fp32 below 4."""
    g = torch.Generator().manual_seed(seed)
    seg, nseg = segments(ei, n)
    l = grid_logits(ei.shape[1], g)
    first, second = pick_per_segment(seg, nseg, g, 2)
    if lead == 'tie':
        l[first], l[second] = 4.0, 4.0
    elif lead == 'ulp':
        l[first], l[second] = 4.0, float(np.nextafter(np.float32(4.0), np.float32(0)))
    else:
        l[first] = 1.0 + lead
    return l.float(), first, second


def maps(n, shape, seed, magnitude=False):
    """Seeded maps [n, *shape]: normal, or |v| in [0.5, 2) with a random sign (no product of two of them underflows)."""
    g = torch.Generator().manual_seed(seed)
    if not magnitude:
        return torch.randn((n,) + tuple(shape), generator=g)
    v = torch.rand((n,) + tuple(shape), generator=g) * 1.5 + 0.5
    return torch.where(torch.rand((n,) + tuple(shape), generator=g) < 0.5, -v, v)


DEGREES = [1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2049, 4097]


def degree_graph():
    """Hub rows with every degree of DEGREES in both directions (plus a run of 1 / 2 / 3-slot rows), duplicate
    leaf edges, one-sided leaves and isolated nodes."""
    ei, n = hub_graph(DEGREES, offset=7, leaves=4200, seed=11)
    filler = torch.nonzero((ei[0] < 4200) & (ei[1] < 4200)).view(-1)[:6]   # leaf-leaf pairs listed twice
    ei = torch.cat((ei, ei[:, filler]), dim=1)
    out, inn = ei[0] < ei[1], ei[0] > ei[1]
    do, di = torch.bincount(ei[0][out], minlength=n), torch.bincount(ei[0][inn], minlength=n)
    for d in DEGREES:
        assert bool(((do == d) | (di == d)).any()), d
    assert int(torch.maximum(do, di).max()) > 4 * ATT_MAX_DEG
    assert int(torch.bincount(ei[1], minlength=n).max()) > ATT_MAX_DEG          # d_z columns past one pass too
    assert bool(((do == 0) & (di == 0)).any()), 'an isolated node'
    assert bool(((do > 0) & (di == 0)).any()) and bool(((di > 0) & (do == 0)).any()), 'one-sided nodes'
    key = ei[0] * n + ei[1]
    assert torch.unique(key).numel() < key.numel(), 'duplicate edges'
    return ei, n


_DEG_GRAPH = {}


def deg_graph():
    if not _DEG_GRAPH:
        _DEG_GRAPH['g'] = degree_graph()
    return _DEG_GRAPH['g']


LEADS = [0, 2, 8, 12, 17, 25, 40, 88, 1e4, 'tie', 'ulp']


@pytest.mark.parametrize('lead', LEADS, ids=[str(v) for v in LEADS])
def test_attention_per_element_across_softmax_sharpness_and_degree(lead):
    """Every degree of DEGREES (to 4,097 slots per direction: four passes of ATT_MAX_DEG) at one sharpness: the top
    logit of each segment leads the rest by ``lead``, or exact / one-ulp ties at the top.  The old backward
    (w (dw - S) in fp32) is shown to fail the same bar from a lead of 12 (a lead of 1e4 leaves it exact)."""
    ei, n = deg_graph()
    feat = 33
    z = maps(n, (feat, 1, 1), seed=1)
    g_in, g_out = maps(n, (feat, 1, 1), seed=2), maps(n, (feat, 1, 1), seed=3)
    logits, first, second = sharp_logits(ei, n, lead, seed=4)
    r = attn_ref(ei, n, z, logits, g_in, g_out)
    seg, nseg = r['seg'], r['nseg']
    deg = seg_sum(torch.ones(ei.shape[1], dtype=torch.float64), seg, nseg)
    multi = deg[seg[first]] >= 2
    top = logits.double()[first][multi]
    l64 = logits.double()
    rest = l64.clone()
    rest[first] = float('-inf')
    second_max = rest.new_full((nseg,), float('-inf')).scatter_reduce(0, seg, rest, 'amax', include_self=True)
    gap = top - second_max[seg[first][multi]]
    if isinstance(lead, str):
        assert bool((gap <= 2.0 ** -21).all()) and bool((gap >= 0).all())
        assert (float(gap.max()) == 0) == (lead == 'tie')
        assert bool((r['w'][first][multi] <= 0.5 + 1e-6).all())
    else:
        assert float(gap.min()) >= lead and float(gap.max()) <= lead + 2
        if lead > 0:
            assert bool((r['qs'][seg[first]] == first).all())      # the lead edge is each segment's q*
        if lead >= 12:                                             # the regime where w_q* -> 1 cancels
            assert float((1 - r['w'][first][multi]).max()) <= max(4200 * math.exp(-lead), 2e-12)
    got = run_gpu(ei, n, z, logits, g_in, g_out)
    assert_close(got, r, f'lead {lead}')
    if not isinstance(lead, str) and 12 <= lead <= 88:
        q = ratio(old_formula(r), r['dl'], r['dl_bar'])
        assert float(q.max()) > 1, f'the fp32 form w (dw - S) passed the bar at lead {lead}: {float(q.max()):.3g}'


MAP_SHAPES = [(1, 1, 1), (31, 1, 1), (33, 1, 1), (257, 1, 1), (64, 14, 14), (3, 5, 7)]


@pytest.mark.parametrize('shape', MAP_SHAPES, ids=['x'.join(map(str, s)) for s in MAP_SHAPES])
def test_attention_per_element_across_map_size(shape):
    """feat = 1, 31, 33, 257, the shipped 64x14x14 = 12,544 floats and a non-square 3x5x7 map, on hub rows past one
    pass of ATT_MAX_DEG, with each segment's lead drawn from {0, 8, 17, 40}."""
    feat = int(np.prod(shape))
    if feat > 1000:                                         # the fp64 reference holds E x feat products
        ei, n = hub_graph([1, 2, 33, 257], offset=3, leaves=300, seed=5)
    else:
        ei, n = hub_graph([1, 2, 33, 257, 1025], offset=3, leaves=1100, seed=5)
    z = maps(n, shape, seed=6)
    g_in, g_out = maps(n, shape, seed=7), maps(n, shape, seed=8)
    g = torch.Generator().manual_seed(9)
    seg, nseg = segments(ei, n)
    l = grid_logits(ei.shape[1], g)
    (first,) = pick_per_segment(seg, nseg, g, 1)
    leads = torch.tensor([0.0, 8.0, 17.0, 40.0])[torch.randint(4, (first.numel(),), generator=g)]
    l[first] = 1.0 + leads.double()
    logits = l.float()
    r = attn_ref(ei, n, z, logits, g_in, g_out)
    assert r['feat'] == feat
    got = run_gpu(ei, n, z, logits, g_in, g_out)
    assert tuple(got['flow_in'].shape) == tuple(z.shape) and tuple(got['dz'].shape) == tuple(z.shape)
    assert_close(got, r, f'map {shape}')


def test_attention_empty_and_one_slot_segments():
    """Degree 0 (zero flows and d_z, no d_logits written) and 1-slot segments (w = 1, d_logit exactly 0, the flow is
    the neighbour's map)."""
    ei = torch.tensor([[0, 1, 2, 3, 3, 4], [1, 0, 3, 2, 4, 3]])
    n = 7                                                   # nodes 5, 6 have no edges
    z = maps(n, (5, 2, 3), seed=10)
    g_in, g_out = maps(n, (5, 2, 3), seed=11), maps(n, (5, 2, 3), seed=12)
    logits = torch.tensor([0.5, -3.0, 7.0, 2.0, -1.0, 88.0])
    r = attn_ref(ei, n, z, logits, g_in, g_out)
    got = run_gpu(ei, n, z, logits, g_in, g_out)
    assert_close(got, r, 'degree 0 / 1')
    assert bool((got['flow_in'][5:] == 0).all()) and bool((got['flow_out'][5:] == 0).all()) and bool((got['dz'][5:] == 0).all())
    one = torch.tensor([0, 1, 2, 5])                        # edges alone in their segment
    assert bool((r['dl'][one] == 0).all()) and bool((got['dl'][one] == 0).all())
    assert torch.equal(got['flow_out'][0], z[1]) and torch.equal(got['flow_in'][1], z[0])


# ------------------------------------------------------------------ bit-exact invariances
def inv_case(seed):
    ei, n = hub_graph([1, 2, 33, 1025], offset=5, leaves=1100, seed=seed)
    shape = (6, 3, 2)
    z, g_in, g_out = (maps(n, shape, seed=seed + k, magnitude=True) for k in (1, 2, 3))
    g = torch.Generator().manual_seed(seed + 4)
    seg, nseg = segments(ei, n)
    l = grid_logits(ei.shape[1], g, -4.0, 4.0)
    (first,) = pick_per_segment(seg, nseg, g, 1)
    l[first] = 5.0                                          # leads up to 9: weights stay far above the subnormals
    return ei, n, z, l.float(), g_in, g_out


@pytest.mark.parametrize('p', [-64, -24, 24, 64])
def test_attention_scale_transport_is_exact(p):
    """z x 2^p gives flows and d_logits x 2^p and the same d_z; G x 2^p gives d_z and d_logits x 2^p: bit for bit."""
    ei, n, z, logits, g_in, g_out = inv_case(20)
    base = run_gpu(ei, n, z, logits, g_in, g_out)
    f = 2.0 ** p
    zs = run_gpu(ei, n, z * f, logits, g_in, g_out)
    gs = run_gpu(ei, n, z, logits, g_in * f, g_out * f)
    for k in ('flow_in', 'flow_out', 'dl'):
        assert torch.equal(zs[k], base[k] * f), ('z', k)
    assert torch.equal(zs['dz'], base['dz'])
    for k in ('dz', 'dl'):
        assert torch.equal(gs[k], base[k] * f), ('G', k)
    assert torch.equal(gs['flow_in'], base['flow_in']) and torch.equal(gs['flow_out'], base['flow_out'])
    for t in (base, zs, gs):                                # the transport is exact, not flushed
        assert all(bool(torch.isfinite(t[k]).all()) for k in t)
        assert float(t['dl'].abs()[t['dl'] != 0].min()) >= TINY and float(t['flow_in'].abs().max()) > 0


@pytest.mark.parametrize('c', [-1536.0, -37.25, 1.0 / 1024, 4096.0])
def test_attention_logit_shift_changes_nothing(c):
    """Adding an exactly representable constant to every logit leaves every output bit-identical."""
    ei, n, z, logits, g_in, g_out = inv_case(30)
    shifted = logits + c
    assert torch.equal(shifted.double(), logits.double() + c)             # exact in fp32
    base, got = run_gpu(ei, n, z, logits, g_in, g_out), run_gpu(ei, n, z, shifted, g_in, g_out)
    for k in base:
        assert torch.equal(got[k], base[k]), k


# ------------------------------------------------------------------ non-finite values
def test_attention_non_finite_logits_and_maps():
    """-inf on some logits (weight 0, gradient exactly 0), a segment whose logits are all -inf, +inf and NaN logits
    (NaN over their segment), inf and NaN in the maps of neighbours whose every edge has weight 0 (0 x inf: NaN over
    the segments that list them): NaN exactly where the restatement has it, the bars elsewhere."""
    ei, n = hub_graph([1, 2, 33, 257, 1025], offset=3, leaves=1100, seed=40)
    shape = (7, 2, 2)
    z = maps(n, shape, seed=41)
    g_in, g_out = maps(n, shape, seed=42), maps(n, shape, seed=43)
    g = torch.Generator().manual_seed(44)
    seg, nseg = segments(ei, n)
    l = grid_logits(ei.shape[1], g, -3.0, 3.0)
    deg = torch.bincount(seg, minlength=nseg)
    big = [int(s) for s in torch.nonzero(deg >= 30).view(-1)]          # hub segments
    assert len(big) >= 6
    first, second, third = pick_per_segment(seg, nseg, g, 3)
    pick = {s: (int(first[seg[first] == s]), int(second[seg[second] == s]), int(third[seg[third] == s])) for s in big}
    minus_inf = [pick[s][k] for s in big[:3] for k in (1, 2)]
    l[minus_inf] = float('-inf')
    small = second[(deg[seg[second]] >= 3) & (deg[seg[second]] < 30)]  # leaf rows with three or more slots
    l[small] = float('-inf')
    l[seg == big[3]] = float('-inf')
    l[pick[big[4]][0]] = float('inf')
    l[pick[big[5]][0]] = float('nan')
    # an inf map entry in a neighbour of big[0], a NaN one in a neighbour of big[1]; every edge to them gets weight 0
    zc = z.clone()
    c_inf, c_nan = int(ei[1][pick[big[0]][1]]), int(ei[1][pick[big[1]][1]])
    zc[c_inf].view(-1)[3] = float('inf')
    zc[c_nan].view(-1)[5] = float('nan')
    l[(ei[1] == c_inf) | (ei[1] == c_nan)] = float('-inf')
    logits = l.float()
    r = attn_ref(ei, n, zc, logits, g_in, g_out)
    got = run_gpu(ei, n, zc, logits, g_in, g_out)
    assert_close(got, r, 'non-finite')
    # the regimes: weight-0 edges with gradient exactly 0 where the segment stays finite, NaN segments
    wzero = (logits == float('-inf')) & (r['w'] == 0) & torch.isfinite(r['dl'])
    assert int(wzero.sum()) >= 10
    assert bool((got['dl'][wzero] == 0).all()) and bool((r['dl'][wzero] == 0).all())
    for s in (big[3], big[4], big[5], big[0], big[1]):
        assert bool(torch.isnan(r['dl'][seg == s]).all()), s
    flow = lambda s: (got['flow_out'] if s % 2 else got['flow_in'])[s // 2].reshape(-1)   # noqa: E731
    assert bool(torch.isnan(flow(big[3])).all())
    assert bool(torch.isnan(flow(big[0])[3])) and bool(torch.isnan(flow(big[1])[5]))
    assert int(torch.isnan(flow(big[0])).sum()) <= 2                   # only the positions of the inf / NaN entries


# ------------------------------------------------------------------ mask-branch gradient through every step
STEP_CASES = [(1, 1), (4, 1), (4, 3), (4, 4)]


def mask_branch_case(steps, class_steps, agg):
    import copy
    import test_training_options as tto
    d = tto.load('tiny_nonrecip', agg=agg)
    mp = copy.deepcopy(d['mp'])
    mp['num_enc_steps'], mp['num_class_steps'] = steps, class_steps
    P = dict(d['P'])
    for k in ('classifier.edge_model.fc_layers.2.weight', 'classifier.edge_model.fc_layers.2.bias'):
        P[k] = P[k] * 0.25                                  # moderate logits: |l| <= 8 over four steps
    n, e = d['x'].shape[0], d['ei'].shape[1]
    g = torch.Generator().manual_seed(100 + steps * 10 + class_steps)
    shape = (4, 3, 3)
    zs = [torch.randn((n,) + shape, generator=g) for _ in range(steps)]
    Gs = [(torch.randn((n,) + shape, generator=g), torch.randn((n,) + shape, generator=g)) for _ in range(steps)]
    hs = [torch.randn(e, generator=g) for _ in range(steps)]
    return d, mp, P, zs, Gs, hs


def mask_branch_loss(logits, aggregate, zs, Gs, hs, first_cls):
    """sum over steps of <G_in, flow_in> + <G_out, flow_out>, plus <h, logits> of the classified steps only: earlier
    steps reach the core network through the attention alone."""
    loss = 0
    for s, lg in enumerate(logits):
        fin, fout = aggregate(zs[s], lg)
        loss = loss + (fin * Gs[s][0]).sum() + (fout * Gs[s][1]).sum()
        if s + 1 >= first_cls:
            loss = loss + (lg.reshape(-1) * hs[s]).sum()
    return loss


def oracle_mask_branch_grads(d, mp, P, zs, Gs, hs, dtype):
    import test_training_options as tto
    params, bufs = tto.split_state(P)
    Pg = {k: v.detach().to(dtype, copy=True).requires_grad_(True) for k, v in params.items()}
    mp_all = dict(mp, num_class_steps=mp['num_enc_steps'])   # every step's logits; they do not depend on this count
    out = tto.train_forward(Pg, mp_all, d['x'].to(dtype), d['ei'], d['ea'].to(dtype), bufs)
    src, dst = d['ei']
    n = d['x'].shape[0]

    def aggregate(z, lg):
        flows = {}
        for name, sel in (('out', src < dst), ('in', src > dst)):
            w = mpn_ref.segment_softmax(lg.view(-1, 1)[sel], src[sel])
            flows[name] = mpn_ref.segment_add(z.to(dtype)[dst[sel]] * w[:, :, None, None], src[sel], n)
        return flows['in'], flows['out']

    first_cls = mp['num_enc_steps'] - mp['num_class_steps'] + 1
    loss = mask_branch_loss(out, aggregate, zs, [(a.to(dtype), b.to(dtype)) for a, b in Gs], [h.to(dtype) for h in hs],
                            first_cls)
    loss.backward()
    return {k: v.grad for k, v in Pg.items() if v.grad is not None}


@pytest.mark.parametrize('agg', ['sum', 'mean', 'max'])
@pytest.mark.parametrize('steps,class_steps', STEP_CASES, ids=[f'{a}-{b}' for a, b in STEP_CASES])
def test_mask_branch_gradient_through_every_step(steps, class_steps, agg):
    """CoreTrainer.autograd_logits(all_steps=True) followed by AttnAggregate on a seeded map per step: the core
    parameters' gradients per row against fp64 autograd of the oracle's per-step logits (row_bar_failures)."""
    import test_training_options as tto
    from test_training_boundaries import row_bar_failures
    from mpntrackseg_b200.training import AttnAggregate, CoreTrainer
    d, mp, P, zs, Gs, hs = mask_branch_case(steps, class_steps, agg)
    tr = CoreTrainer(tto.make_model(mp, P))
    data = tto.make_data(d['x'], d['ei'], d['ea'])
    lg_all = tr.autograd_logits(data, all_steps=True)
    c = tr.last_ctx
    assert tuple(lg_all.shape) == (steps, d['ei'].shape[1]) and c['logit_steps'] == list(range(1, steps + 1))
    assert float(lg_all.detach().abs().max()) <= 16
    seen = []

    def aggregate(z, lg):
        zd = z.to(dev()).requires_grad_(True)
        ld = lg.view(-1, 1)
        ld.retain_grad()
        seen.append((zd, ld))
        return AttnAggregate.apply(zd, ld, c['lay'], c['perm_c'], c['ptr_c'])

    first_cls = steps - class_steps + 1
    loss = mask_branch_loss(list(lg_all), aggregate, zs, [(a.to(dev()), b.to(dev())) for a, b in Gs],
                            [h.to(dev()) for h in hs], first_cls)
    loss.backward()
    for zd, ld in seen:
        assert zd.grad is not None and tuple(zd.grad.shape) == tuple(zd.shape)
        assert ld.grad is not None and tuple(ld.grad.shape) == tuple(ld.shape)
    got = {k: p.grad for k, p in tr.model.named_parameters() if k in tr.named and p.grad is not None}
    ref64 = oracle_mask_branch_grads(d, mp, P, zs, Gs, hs, torch.float64)
    ref32 = oracle_mask_branch_grads(d, mp, P, zs, Gs, hs, torch.float32)
    # with one step the node model feeds no logit: the oracle has no gradient for it, the trainer an exact zero
    assert set(ref64) <= set(got), set(ref64) - set(got)
    assert all(bool((got[k] == 0).all()) for k in set(got) - set(ref64)), sorted(set(got) - set(ref64))
    assert steps == 1 or set(ref64) == set(got)
    bad = row_bar_failures(got, ref64, ref32)
    assert not bad, bad
