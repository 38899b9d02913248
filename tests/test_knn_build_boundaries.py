"""GPU tests of the batched KNN graph build (csrc/knn_graph.cu, csrc/knn_graph_tc.cu) across embedding scale,
dimension, build gates and degenerate windows, against the exact fp32 build and an fp64 oracle.

The build has three routes; ``ops.LAST_KNN_STATS[0]`` reports which one ran:
0 exact fp32 (``engine='fp32'``, a gate that rules the tensor cores out, or the whole-call exact rerun),
1 dense Gram blocks + row select (its keys in registers up to SEL_MAX_N = 5,120 nodes, re-read from the row above),
2 thresholded candidate lists (every window >= TG_MIN_TILES * 128 = 1,024 nodes, at most SEL_MAX_N, k <= 64, or
  k <= CAND_CAP / 4 = 128 with MPN_KNN_THRESHOLDED).
Each tensor-core route pre-ranks with approximate Gram distances and recomputes exactly every row whose k-th and
(k+1)-th distances fall inside an error band, so its kept edge set must equal the exact build's.  Every test asserts
that its case reached the route, gate, fallback or rerun it names.

Bars:
* the tensor-core build's pairs and per-window pair offsets are identical to ``engine='fp32'`` on the same inputs;
* its distances match fp32 with rtol 3e-6 and an absolute tolerance of 1e-6 * the largest embedding norm;
* against the fp64 oracle (the reference's ||a - b + 1e-6||, in fp64), every pair whose two rows have a k-th / (k+1)-th
  relative gap above 1e-5 is kept iff the oracle keeps it; windows whose distances tie exactly by construction are
  compared with the oracle's index-ordered ranking on every row.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from mpntrackseg_b200 import ops, synth
from oracle import graph_ref

EXACT, DENSE, THRESHOLDED = 0, 1, 2
EPS = 1e-6                  # the reference's F.pairwise_distance eps
GAP = 1e-5                  # fp64 relative k-th / (k+1)-th gap above which a row's top-k set is decided
K = 50
TS = 128                    # csrc/knn_graph_tc.cu: rows per Gram tile
TG_MIN_N = 8 * TS           # TG_MIN_TILES * TS: smallest window of the thresholded build
SEL_MAX_N = 20 * 256        # csrc/knn_graph.cu: largest window whose row select keeps its keys in registers
CAND_CAP = 512              # candidate list slots per row
TG_DEFAULT_MAX_K = 64
MAX_WINDOWS = 65535         # gridDim.y of bit_transpose_kernel / dist_blocks_kernel
SCALES = [2.0 ** e for e in range(-20, 14)]


def dev():
    return torch.device('cuda', torch.cuda.current_device())


# ------------------------------------------------------------------ inputs
def bench_window(seed=4, T=15, D=150, dim=256):
    """A bench-shaped window (T frames x D identities, N = T * D) with the synthetic ReID embeddings, no min_gap:
    the k-th / (k+1)-th gaps are whatever the draw gives."""
    w = synth.make_window(T=T, D=D, k=K, seed=seed, reid_dim=dim, node_dim=1, min_gap=0)
    return w.reid, w.frame


def batch(windows):
    """[(reid, frame), ...] -> (reid, frame, node_graph_ptr) of one block-diagonal batch."""
    ptr = [0]
    for r, _ in windows:
        ptr.append(ptr[-1] + r.shape[0])
    reid = torch.cat([r for r, _ in windows])
    frame = torch.cat([f for _, f in windows])
    return reid.contiguous(), frame, ptr


def sized_window(n, seed, dim=256, frames=15):
    """n nodes spread over `frames` frames (as evenly as n allows), synthetic embeddings."""
    per = -(-n // frames)
    reid, _ = bench_window(seed=seed, T=frames, D=per, dim=dim)
    frame = torch.arange(1, frames + 1).repeat_interleave(per)
    return reid[:n].contiguous(), frame[:n].contiguous()


# ------------------------------------------------------------------ builds
def run(reid, frame, ptr, k, recip, engine, mfd=-1):
    """One knn_graph_pairs call: (pairs [2,P] cpu, dist [P] cpu, pair_ptr, [build code, repaired rows])."""
    r = reid if reid.is_cuda else reid.to(dev())
    pairs, dist, gpp = ops.knn_graph_pairs(frame.to(dev()), ptr, r, k, recip, mfd, engine=engine)
    return pairs.cpu(), dist.cpu(), gpp, list(ops.LAST_KNN_STATS)


def against_exact(reid, frame, ptr, k, recip, code, mfd=-1):
    """The tensor-core build (asserted to be build `code`) equals the exact fp32 build; returns its output and stats."""
    got = run(reid, frame, ptr, k, recip, 'tc', mfd)
    ex = run(reid, frame, ptr, k, recip, 'fp32', mfd)
    assert got[3][0] == code, f'build {got[3][0]} ran, expected {code} (stats {got[3]})'
    assert ex[3][0] == EXACT, ex[3]
    diff = mismatch(got, ex)
    assert not diff, f'build {code}, k={k}, reciprocal={recip}: {diff}'
    return got


def mismatch(got, ex):
    """'' if the two builds keep the same pairs with the same per-window offsets, else what differs."""
    if got[2] != ex[2]:
        bad = [g for g in range(len(ex[2]) - 1) if got[2][g + 1] - got[2][g] != ex[2][g + 1] - ex[2][g]]
        return f'pair_ptr differs in {len(bad)} windows (first {bad[:5]})'
    if not torch.equal(got[0], ex[0]):
        n = int(torch.cat((got[0], ex[0]), 1).max()) + 1
        a, b = set((got[0][0] * n + got[0][1]).tolist()), set((ex[0][0] * n + ex[0][1]).tolist())
        return f'{len(a - b)} pairs kept only by the tensor-core build, {len(b - a)} only by the exact one (of {len(b)})'
    return ''


def assert_dist_close(got, ex, reid):
    atol = 1e-6 * float(reid.double().norm(dim=1).max())
    np.testing.assert_allclose(got[1].numpy(), ex[1].numpy(), rtol=3e-6, atol=atol)


# ------------------------------------------------------------------ fp64 oracle
def d64(a, frame, mfd=-1):
    """fp64 ||a_lo - a_hi + eps|| over all pairs of one window (lo / hi = smaller / larger node index, as the reference
    evaluates its (i < j) pairs), +inf where the pair is not time-valid.  Expanded as
    ||a||^2 + ||b||^2 - 2 a.b + 2 eps (sum a - sum b) + dim eps^2 (fp64 error ~1e-16 of ||a||^2 + ||b||^2)."""
    a = a.double()
    n2, s1 = (a * a).sum(1), a.sum(1)
    idx = torch.arange(a.shape[0], device=a.device)
    ds = torch.where(idx[:, None] < idx[None, :], s1[:, None] - s1[None, :], s1[None, :] - s1[:, None])
    d2 = n2[:, None] + n2[None, :] - 2.0 * (a @ a.T) + 2.0 * EPS * ds + a.shape[1] * EPS * EPS
    gap = (frame[:, None] - frame[None, :]).abs().to(a.device)
    ok = (gap > 0) & ((gap <= mfd) if mfd >= 0 else True)
    return torch.where(ok, d2.clamp(min=0).sqrt(), torch.full_like(d2, math.inf)), ok


def oracle_keep(d, ok, k, recip):
    """Kept (i < j) pairs of one window from an fp64 distance matrix (ranks: ascending distance, ties by index, as the
    reference's stable argsort) and the rows whose top-k set is decided by more than the relative gap GAP."""
    n = d.shape[0]
    vals, order = torch.sort(d, dim=1, stable=True)
    rank = torch.empty_like(order)
    rank.scatter_(1, order, torch.arange(n, device=d.device).expand(n, n).contiguous())
    near = rank < k
    keep = (near & near.T) if recip else (near | near.T)
    keep = torch.triu(keep & ok, diagonal=1)
    if k >= n:
        certain = torch.ones(n, dtype=torch.bool, device=d.device)
    else:
        vk, vk1 = vals[:, k - 1], vals[:, k]
        certain = ~torch.isfinite(vk1) | ((vk1 - vk) > GAP * vk1)
    return keep, certain


def pair_matrix(pairs, n0, n, device):
    m = torch.zeros(n, n, dtype=torch.bool, device=device)
    p = pairs.to(device)
    sel = (p[0] >= n0) & (p[0] < n0 + n)
    m[p[0, sel] - n0, p[1, sel] - n0] = True
    return m


def oracle_wrong_rows(got, reid, frame, ptr, k, recip, mfd=-1):
    """Rows that take part in a pair the device keeps and the fp64 oracle does not, or the other way round, among
    the pairs whose two rows are decided."""
    wrong = 0
    for g in range(len(ptr) - 1):
        n0, n = ptr[g], ptr[g + 1] - ptr[g]
        if n == 0:
            continue
        d, ok = d64(reid[n0:n0 + n].to(dev()), frame[n0:n0 + n].to(dev()), mfd)
        keep, certain = oracle_keep(d, ok, k, recip)
        bad = (pair_matrix(got[0], n0, n, dev()) != keep) & certain[:, None] & certain[None, :]
        wrong += int((bad.any(0) | bad.any(1)).sum())
    return wrong


def index_order_keep(frame, ptr, k, recip, mfd=-1):
    """Kept pairs when every distance of a window ties (identical embeddings): each row's top k are its first k
    time-valid partners in index order (the reference's stable sort)."""
    rows, cols = [], []
    for g in range(len(ptr) - 1):
        n0, n = ptr[g], ptr[g + 1] - ptr[g]
        f = frame[n0:n0 + n].to(dev())
        gap = (f[:, None] - f[None, :]).abs()
        ok = (gap > 0) & ((gap <= mfd) if mfd >= 0 else True)
        near = ok & (ok.cumsum(1) <= k)
        keep = torch.triu(((near & near.T) if recip else (near | near.T)) & ok, diagonal=1)
        i, j = torch.nonzero(keep, as_tuple=True)
        rows.append(i.cpu() + n0)
        cols.append(j.cpu() + n0)
    return torch.stack((torch.cat(rows), torch.cat(cols)))


def test_fp64_oracle_matches_graph_ref_on_double_inputs():
    """The expanded fp64 distance of d64 is the reference's pair distance (graph_ref.pair_reid_dist on double
    inputs, eps included) at the scales the sweep covers."""
    reid, frame = bench_window(seed=6, T=4, D=30, dim=256)
    pairs = graph_ref.time_valid_pairs(frame)
    for a in (reid, F.normalize(reid, dim=1)):
        for s in (2.0 ** -20, 1.0, 2.0 ** 13):
            x = (a * s).double()
            ref = graph_ref.pair_reid_dist(x, pairs)
            d, ok = d64(x, frame)
            assert torch.equal(ok[pairs[0], pairs[1]], torch.ones(pairs.shape[1], dtype=torch.bool))
            got = d[pairs[0], pairs[1]]
            assert float(((got - ref).abs() / ref).max()) < 1e-9, s


# ------------------------------------------------------------------ A. embedding magnitude
def sweep(reid, frame, ptr, scales, builds, monkeypatch):
    """Per scale and build: 'ok', or the wrong-row counts against fp32 and the fp64 oracle."""
    report, failed = [], False
    for s in scales:
        x = (reid * s).contiguous()
        xd = x.to(dev())
        norm = float(x.double().norm(dim=1).max())
        for name, env, code in builds:
            if env:
                monkeypatch.setenv(env, '1')
            for recip in (True, False):
                got = run(xd, frame, ptr, K, recip, 'tc')
                ex = run(xd, frame, ptr, K, recip, 'fp32')
                diff = mismatch(got, ex)
                wrong = oracle_wrong_rows(got, x, frame, ptr, K, recip)
                line = f'{name} scale 2^{int(math.log2(s))} |a|max {norm:.3g} recip={recip}: build {got[3][0]}, ' \
                       f'{got[3][1]} rows repaired'
                bad = got[3][0] != code or diff or wrong
                if not bad:
                    try:
                        assert_dist_close(got, ex, x)
                    except AssertionError as e:
                        diff = 'distances: ' + str(e).splitlines()[-1]
                        bad = True
                if bad:
                    failed = True
                    ex_wrong = oracle_wrong_rows(ex, x, frame, ptr, K, recip)
                    line += f' -- vs fp32: {diff or "same"}; wrong rows vs fp64: {wrong} (fp32 build: {ex_wrong})'
                report.append(line)
            if env:
                monkeypatch.delenv(env)
    return report, failed


@pytest.mark.gpu
@pytest.mark.parametrize('norm', ['raw', 'l2'])
def test_embedding_scale_thresholded_and_dense(norm, monkeypatch):
    """Power-of-two scales 2^-20 ... 2^13 of a bench-shaped window, raw and L2-normalised, through the thresholded
    build (default gate, k = 50) and the dense build (MPN_KNN_DENSE)."""
    reid, frame = bench_window()
    if norm == 'l2':
        reid = F.normalize(reid, dim=1)
    reid, frame, ptr = batch([(reid, frame)])
    report, failed = sweep(reid, frame, ptr, SCALES, [('thresholded', None, THRESHOLDED), ('dense', 'MPN_KNN_DENSE', DENSE)],
                           monkeypatch)
    assert not failed, '\n'.join(report)


@pytest.mark.gpu
@pytest.mark.parametrize('norm', ['raw', 'l2'])
def test_embedding_scale_streamed_row_select(norm, monkeypatch):
    """A window of 5,200 nodes (above SEL_MAX_N): Gram blocks + the streamed row select, at a few scales."""
    reid, frame = bench_window(seed=12, T=26, D=200)
    assert reid.shape[0] > SEL_MAX_N
    if norm == 'l2':
        reid = F.normalize(reid, dim=1)
    reid, frame, ptr = batch([(reid, frame)])
    report, failed = sweep(reid, frame, ptr, [2.0 ** -20, 2.0 ** -13, 2.0 ** -8, 1.0, 2.0 ** 13],
                           [('dense', None, DENSE)], monkeypatch)
    assert not failed, '\n'.join(report)


@pytest.mark.gpu
@pytest.mark.parametrize('amax, code', [(64000.0, THRESHOLDED), (66000.0, EXACT)])
def test_largest_value_at_the_overflow_guard(amax, code):
    """Largest |v| = 64,000 still runs on the tensor cores; 66,000 trips the < 65,000 guard of pack_reid_kernel and
    the whole call reruns exactly (build code 0)."""
    reid, frame = bench_window(seed=5)
    reid = (reid / reid.abs().max() * amax).contiguous()
    assert float(reid.abs().max()) == amax
    _, _, ptr = batch([(reid, frame)])
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, code)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


# ------------------------------------------------------------------ B. dimension and alignment gates
@pytest.mark.gpu
@pytest.mark.parametrize('dim, code', [(64, THRESHOLDED), (128, THRESHOLDED), (320, THRESHOLDED), (512, THRESHOLDED),
                                       (32, EXACT), (100, EXACT), (576, EXACT)])
def test_dimension_gate(dim, code):
    """Multiples of 64 up to the workspace's 512 run on the tensor cores (64 = one K chunk); other dims and dims above
    512 run exact and still match."""
    reid, frame = bench_window(seed=7, dim=dim)
    _, _, ptr = batch([(reid, frame)])
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, code)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
def test_unaligned_embeddings_run_exact():
    """A reid view whose data pointer is 4 bytes past a 16-byte boundary (storage offset 1) runs exact."""
    reid, frame = bench_window(seed=8)
    n, dim = reid.shape
    flat = torch.zeros(n * dim + 1, device=dev())
    view = flat[1:].view(n, dim)
    view.copy_(reid.to(dev()))
    assert view.is_contiguous() and view.data_ptr() % 16 != 0
    _, _, ptr = batch([(reid, frame)])
    for recip in (True, False):
        got = against_exact(view, frame, ptr, K, recip, EXACT)
        assert torch.equal(got[0], run(reid.to(dev()), frame, ptr, K, recip, 'tc')[0])
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


# ------------------------------------------------------------------ C. build selection
@pytest.mark.gpu
@pytest.mark.parametrize('n, code', [(TG_MIN_N - 1, DENSE), (TG_MIN_N, THRESHOLDED), (TG_MIN_N + 1, THRESHOLDED),
                                     (SEL_MAX_N, THRESHOLDED), (SEL_MAX_N + 1, DENSE)])
def test_window_size_gates(n, code):
    reid, frame = sized_window(n, seed=n)
    _, _, ptr = batch([(reid, frame)])
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, code)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('k, forced, code', [(TG_DEFAULT_MAX_K, False, THRESHOLDED), (TG_DEFAULT_MAX_K + 1, False, DENSE),
                                             (CAND_CAP // 4, True, THRESHOLDED), (CAND_CAP // 4 + 1, True, DENSE)])
def test_k_gates(k, forced, code, monkeypatch):
    """k <= 64 by default, k <= CAND_CAP / 4 = 128 with MPN_KNN_THRESHOLDED; above it the dense build runs."""
    if forced:
        monkeypatch.setenv('MPN_KNN_THRESHOLDED', '1')
    reid, frame = bench_window(seed=9)
    _, _, ptr = batch([(reid, frame)])
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, k, recip, code)
        assert oracle_wrong_rows(got, reid, frame, ptr, k, recip) == 0


@pytest.mark.gpu
def test_one_small_window_sends_the_batch_dense():
    """One 1,023-node window among three of >= 1,024: the whole batch takes the dense build."""
    wins = [sized_window(n, seed=20 + i) for i, n in enumerate((TG_MIN_N, TG_MIN_N - 1, 1500, 2250))]
    reid, frame, ptr = batch(wins)
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, DENSE)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
def test_partial_last_tiles_on_the_thresholded_build():
    """Windows whose size is not a multiple of 128 (partial last tile, li clamped to n - 1 in the Gram epilogue)."""
    sizes = (TG_MIN_N + 1, 9 * TS - 1, 10 * TS + 3, 2250)
    assert all(n % TS for n in sizes)
    reid, frame, ptr = batch([sized_window(n, seed=30 + i) for i, n in enumerate(sizes)])
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, THRESHOLDED)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


# ------------------------------------------------------------------ D. degenerate windows on the thresholded build
@pytest.mark.gpu
@pytest.mark.parametrize('sizes, code', [((TG_MIN_N,), THRESHOLDED), ((5400, K - 20), DENSE)])
@pytest.mark.parametrize('recip', [True, False])
def test_all_identical_embeddings(recip, sizes, code):
    """Every distance of a window ties and every row with more than k nodes in its window is flagged.  One 1,024-node
    window: every candidate list overflows CAND_CAP; the result is the reference's index-ordered top-k (graph_ref on
    the same inputs).  A 5,400-node window next to one smaller than k: the row select that re-reads rows above
    SEL_MAX_N resolves the ties straddling k by index."""
    wins = []
    for i, n in enumerate(sizes):
        r, f = sized_window(n, seed=40 + i)
        wins.append((r[:1].expand_as(r).contiguous(), f))
    reid, frame, ptr = batch(wins)
    got = against_exact(reid, frame, ptr, K, recip, code)
    assert got[3][1] == sum(n for n in sizes if n > K), got[3]
    assert torch.equal(got[0], index_order_keep(frame, ptr, K, recip))
    if len(sizes) == 1:
        pairs = graph_ref.time_valid_pairs(frame)
        d = graph_ref.pair_reid_dist(reid.double(), pairs)
        assert float(d.max()) == float(d.min())
        keep = graph_ref.knn_keep_mask(d, pairs, reid.shape[0], K, recip, symmetric_edges=False)
        assert torch.equal(got[0], pairs[:, keep])


@pytest.mark.gpu
@pytest.mark.parametrize('recip', [True, False])
def test_duplicated_identities(recip):
    """Each embedding appears six times in a bench-shaped window: groups of exactly tied distances straddle the k
    boundary and go through cand_select_kernel's tie resolution by index."""
    reid, frame = bench_window(seed=41)
    reid = reid[torch.arange(reid.shape[0]) % 375].contiguous()
    _, _, ptr = batch([(reid, frame)])
    d, ok = d64(reid.to(dev()), frame.to(dev()))
    vals = torch.sort(d, dim=1).values
    tied = (vals[:, K] - vals[:, K - 1]) <= 1e-12 * vals[:, K]     # duplicates of one embedding at the boundary
    assert int(tied.sum()) > 0
    got = against_exact(reid, frame, ptr, K, recip, THRESHOLDED)
    assert got[3][1] > 0, got[3]
    assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('recip', [True, False])
def test_large_common_offset(recip):
    """v = 1000 + 0.01 * noise: ||a||^2 + ||b||^2 - 2 a.b cancels catastrophically; the band must flag the rows."""
    reid, frame = bench_window(seed=42)
    reid = (1000.0 + 0.01 * reid).contiguous()
    _, _, ptr = batch([(reid, frame)])
    got = against_exact(reid, frame, ptr, K, recip, THRESHOLDED)
    assert got[3][1] > 0, got[3]
    assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


def sample_thresholds_infinite(frame, n, k, mfd=-1):
    """Rows of one window whose row_threshold_kernel tau is +inf: fewer than 8 time-valid entries among the two sample
    column tiles (nt/4, 3nt/4), or rank r = ceil(2.5 k nv / n) + 6 above their count nv."""
    nt = -(-n // TS)
    cols = torch.cat([torch.arange(t * TS, min(t * TS + TS, n)) for t in (nt // 4, (3 * nt) // 4)])
    gap = (frame[:, None] - frame[cols][None, :]).abs()
    ok = (gap > 0) & ((gap <= mfd) if mfd >= 0 else True)
    ok &= torch.arange(n)[:, None] != cols[None, :]
    nv = ok.sum(1)
    r = (5 * k * nv + 2 * n - 1) // (2 * n) + 6
    return (nv < 8) | (r > nv)


@pytest.mark.gpu
@pytest.mark.parametrize('recip', [True, False])
def test_almost_all_detections_in_one_frame(recip):
    """1,000 detections in frame 1 and one in each of 24 other frames: the frame-1 rows see too few valid sample
    entries (tau = +inf, the list overflows) and fewer than k valid partners."""
    reid, _ = sized_window(TG_MIN_N, seed=43)
    frame = torch.cat((torch.ones(1000, dtype=torch.int64), torch.arange(2, 26)))
    _, _, ptr = batch([(reid, frame)])
    inf_rows = int(sample_thresholds_infinite(frame, frame.numel(), K).sum())
    assert inf_rows >= 1000, inf_rows
    got = against_exact(reid, frame, ptr, K, recip, THRESHOLDED)
    assert got[3][1] >= inf_rows, got[3]
    assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('mfd', [1, 2])
def test_small_max_frame_dist(mfd):
    """Most candidates are not time-valid: rows with a finite tau still end with fewer than k valid candidates
    (nvalid < k), so more rows are flagged than those whose tau is +inf."""
    reid, frame = bench_window(seed=44)
    _, _, ptr = batch([(reid, frame)])
    inf_rows = int(sample_thresholds_infinite(frame, frame.numel(), K, mfd).sum())
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, THRESHOLDED, mfd=mfd)
        assert got[3][1] > inf_rows, (got[3], inf_rows)
        assert oracle_wrong_rows(got, reid, frame, ptr, K, recip, mfd=mfd) == 0


@pytest.mark.gpu
def test_more_flagged_rows_than_scratch_slots_reruns_exact():
    """One 5,120-node and four 1,024-node windows of identical embeddings: 9,216 flagged rows, but the exact repair
    has sum(n^2) / max(n) = 5,939 scratch rows, so the whole call reruns exact (build code 0)."""
    sizes = (SEL_MAX_N,) + (TG_MIN_N,) * 4
    wins = []
    for i, n in enumerate(sizes):
        r, f = sized_window(n, seed=50 + i)
        wins.append((r[:1].expand_as(r).contiguous(), f))
    reid, frame, ptr = batch(wins)
    scratch_rows = sum(n * n for n in sizes) // max(sizes)
    assert sum(sizes) > scratch_rows
    for recip in (True, False):
        got = against_exact(reid, frame, ptr, K, recip, EXACT)
        assert torch.equal(got[0], index_order_keep(frame, ptr, K, recip))
    # the large window alone: all of its rows flagged, as many as it has scratch rows, no rerun
    reid, frame, ptr = batch(wins[:1])
    got = against_exact(reid, frame, ptr, K, True, THRESHOLDED)
    assert got[3][1] == SEL_MAX_N, got[3]
    assert torch.equal(got[0], index_order_keep(frame, ptr, K, True))


# ------------------------------------------------------------------ E. batch structure
@pytest.mark.gpu
@pytest.mark.parametrize('recip', [True, False])
def test_empty_windows_on_the_dense_build(recip):
    """Windows of 0 nodes first, between and last: TileCursor, the window binary searches and window_max_kernel."""
    sizes = (0, 300, 0, 0, 260, 0, 500, 0)
    wins = [sized_window(n, seed=60 + i) if n else (torch.zeros(0, 256), torch.zeros(0, dtype=torch.int64))
            for i, n in enumerate(sizes)]
    reid, frame, ptr = batch(wins)
    got = against_exact(reid, frame, ptr, K, recip, DENSE)
    assert [got[2][g + 1] - got[2][g] for g in range(len(sizes)) if sizes[g] == 0] == [0] * sizes.count(0)
    assert oracle_wrong_rows(got, reid, frame, ptr, K, recip) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('engine', ['tc', 'fp32'])
def test_window_count_limit(engine):
    """65,535 two-node windows, each spanning two frames, keep exactly their one pair; 65,536 are rejected."""
    g = MAX_WINDOWS
    reid = torch.randn(2 * g, 64, generator=torch.Generator().manual_seed(70))
    frame = torch.tensor([1, 2]).repeat(g)
    ptr = list(range(0, 2 * g + 1, 2))
    pairs, dist, gpp, stats = run(reid, frame, ptr, K, True, engine)
    assert stats[0] == (DENSE if engine == 'tc' else EXACT), stats
    assert gpp == list(range(g + 1))
    assert torch.equal(pairs, torch.stack((torch.arange(0, 2 * g, 2), torch.arange(1, 2 * g, 2))))
    ref = graph_ref.pair_reid_dist(reid, pairs)
    np.testing.assert_allclose(dist.numpy(), ref.numpy(), rtol=3e-6, atol=1e-6 * float(reid.norm(dim=1).max()))
    more = torch.randn(2 * (g + 1), 64)
    with pytest.raises(ValueError, match='knn_graph_pairs'):
        run(more, torch.tensor([1, 2]).repeat(g + 1), list(range(0, 2 * g + 3, 2)), K, True, engine)
    torch.cuda.empty_cache()
