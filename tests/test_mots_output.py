"""GPU checks of the MOTS output stage (csrc/mots_output.cu through ops / utils.mots / MPNTracker) against the CPU
restatement oracle/mots_ref.py.

Pasted probabilities: |dp| <= 1e-6 per pixel against torchvision's paste on float64 masks.  RLE: areas and strings
identical in every frame where no pixel has an oracle probability within 1e-6 of the threshold; in the other frames
both strings are decoded and the pixel sets compared outside that band."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from mpntrackseg_b200 import ops, synth
from mpntrackseg_b200.utils.mots import encode_mots_masks, write_mots_txt
from oracle import mots_ref

pytestmark = pytest.mark.gpu

BAND = 1e-6


def dev():
    return torch.device('cuda:0')


def gpu_rle(masks, boxes, frame, shape, threshold=0.5):
    area, chars, char_ptr = ops.mots_rle(masks.to(dev()), boxes.to(dev()), frame.to(dev()), shape, threshold)
    data = chars.cpu().numpy().tobytes()
    ptr = char_ptr.cpu().tolist()
    strings = [data[a:b].decode('ascii') if b > a else None for a, b in zip(ptr[:-1], ptr[1:])]
    return area.cpu().tolist(), strings


def decode(s, h, w):
    if s is None:
        return np.zeros((h, w), dtype=bool)
    c = mots_ref.rle_from_string(s)
    assert sum(c) == h * w and all(v >= 0 for v in c)
    return mots_ref.rle_decode(c, h, w)


def check_against_oracle(masks, boxes, frame, shape, threshold=0.5, nodes=None):
    """Returns (areas, strings) of the GPU after checking them against the oracle (for the given node subset)."""
    h, w = shape
    area, strings = gpu_rle(masks, boxes, frame, shape, threshold)
    sel = torch.arange(masks.shape[0]) if nodes is None else torch.as_tensor(nodes)
    ref, bands = mots_ref.mots_strings(masks[sel], boxes[sel], frame[sel], shape, threshold, BAND)
    for a, i in enumerate(sel.tolist()):
        got = decode(strings[i], h, w)
        assert area[i] == int(got.sum()), i
        f = int(frame[i])
        if f not in bands:
            assert strings[i] == ref[a], f'node {i} (frame {f}): {strings[i]!r} != {ref[a]!r}'
        else:
            keep = ~bands[f].numpy()
            assert np.array_equal(got[keep], decode(ref[a], h, w)[keep]), f'node {i} (frame {f}) outside the band'
    return area, strings


# ------------------------------------------------------------------ dense paste
def _expanded(x0, y0, x1, y1, m=28, padding=1):
    """A float box whose torchvision expansion is (x0, y0, x1, y1) up to rounding."""
    s = (m + 2 * padding) / m
    cx, cy, hw, hh = (x0 + x1) / 2, (y0 + y1) / 2, (x1 - x0) / 2 / s, (y1 - y0) / 2 / s
    return [cx - hw, cy - hh, cx + hw, cy + hh]


def _paste_boxes(h, w):
    return torch.tensor([
        [0.37 * w, 0.21 * h, 0.71 * w + 0.3, 0.83 * h + 0.6],            # fractional, inside
        _expanded(-0.7, -1.2, 0.6 * w + 2.3, 0.5 * h + 1.7),              # expanded corners at -0.7 / -1.2: truncate to 0 / -1
        [-0.4 * w, 0.1 * h, 0.3 * w, 0.6 * h],                           # partly outside the left edge
        [0.6 * w, 0.2 * h, 1.4 * w, 0.7 * h],                            # right edge
        [0.2 * w, -0.5 * h, 0.5 * w, 0.4 * h],                           # top edge
        [0.3 * w, 0.6 * h, 0.9 * w, 1.5 * h],                            # bottom edge
        [w + 10.0, h + 5.0, w + 60.0, h + 90.0],                         # entirely outside: empty
        [-80.0, -90.0, -20.0, -10.0],                                    # entirely outside, negative side
        [0.5 * w + 3.0, 0.5 * h, 0.5 * w - 4.0, 0.5 * h + 6.0],          # x2 < x1: w clamped to 1
        [0.5 * w, 0.4 * h, 0.5 * w + 0.2, 0.4 * h + 0.1],                # 1-pixel box
        [-0.3 * w - 7.0, -0.2 * h - 3.0, 1.3 * w + 5.0, 1.25 * h + 9.0],  # larger than the image
    ], dtype=torch.float64)


@pytest.mark.parametrize('shape', [(1, 1), (1, 173), (151, 1), (1080, 1920)])
@pytest.mark.parametrize('m,padding', [(28, 1), (56, 1), (28, 0), (28, 2)])
def test_dense_paste_against_torchvision(shape, m, padding):
    h, w = shape
    g = torch.Generator().manual_seed(m * 7 + padding + h)
    boxes = _paste_boxes(h, w)
    masks = torch.rand(boxes.shape[0], 1, m, m, generator=g)
    ib = ops.paste_boxes(boxes.to(dev()), m, padding).cpu()
    assert torch.equal(ib, mots_ref.integer_boxes(boxes, m, padding))
    if (m, padding) == (28, 1):
        assert ib[1, 0] == 0 and ib[1, 1] == -1                           # truncation toward zero, not floor
    got = ops.paste_masks_in_image(masks.to(dev()), boxes.to(dev()), shape, padding=padding)
    assert got.shape == (boxes.shape[0], 1, h, w) and got.dtype == torch.float32
    ref = mots_ref.paste(masks, boxes, shape, padding=padding)
    err = (got[:, 0].cpu().double() - ref).abs().max().item()
    assert err <= 1e-6, err
    assert not bool(got[6:8].any())                                      # boxes outside the image


def test_dense_paste_fp32_boxes_follow_their_own_rounding():
    g = torch.Generator().manual_seed(5)
    boxes = (torch.rand(40, 4, generator=g, dtype=torch.float64) * 190).sort(dim=1).values.float()     # x1 <= y1 <= x2 <= y2
    masks = torch.rand(40, 1, 28, 28, generator=g)
    got = ops.paste_masks_in_image(masks.to(dev()), boxes.to(dev()), (200, 310))
    from torchvision.models.detection.roi_heads import paste_masks_in_image
    ref = paste_masks_in_image(masks.double(), boxes, (200, 310))           # expansion in float32, paste in float64
    assert (got.cpu().double() - ref).abs().max().item() <= 1e-6


# ------------------------------------------------------------------ RLE
def _scale_one_box(x0, y0, p):
    """A float box whose integer box is exactly (x0, y0, x0 + p - 1, y0 + p - 1) for a (p - 2)^2 mask with padding 1:
    the resize is then the identity and the pasted image is the padded mask itself."""
    s = p / (p - 2)
    half = (p - 1) / 2 / s
    cx, cy = x0 + (p - 1) / 2 + 0.2, y0 + (p - 1) / 2 + 0.2
    return [cx - half, cy - half, cx + half, cy + half]


def test_rle_first_count_zero_and_last_pixel():
    h, w = 37, 23
    masks = torch.full((2, 1, 28, 28), 0.95)
    boxes = torch.tensor([[-3.0, -2.0, 8.0, 10.0], [15.0, 25.0, 30.0, 45.0]], dtype=torch.float64)
    frame = torch.tensor([1, 2])
    _, strings = check_against_oracle(masks, boxes, frame, (h, w))
    c0, c1 = mots_ref.rle_from_string(strings[0]), mots_ref.rle_from_string(strings[1])
    assert c0[0] == 0                                                    # touches pixel (0, 0)
    assert decode(strings[1], h, w)[-1, -1] and len(c1) % 2 == 0         # ends on the last pixel: no trailing zeros


def test_rle_full_height_columns_merge_and_full_image():
    h, w = 40, 30
    masks = torch.full((3, 1, 28, 28), 0.9)
    boxes = torch.tensor([[5.0, -10.0, 12.0, 50.0],                     # full-height columns: one run
                          [-10.0, -10.0, 40.0, 50.0],                   # the full image
                          [0.0, 3.0, 29.0, 20.0]], dtype=torch.float64)
    frame = torch.tensor([1, 2, 3])
    _, strings = check_against_oracle(masks, boxes, frame, (h, w))
    c = mots_ref.rle_from_string(strings[0])
    assert len(c) == 3 and c[1] % h == 0 and c[1] > h                   # several columns, one run
    assert mots_ref.rle_from_string(strings[1]) == [0, h * w]


def test_rle_checkerboard_has_the_most_runs():
    h, w, m = 70, 50, 28
    p = m + 2
    cb = ((torch.arange(m).view(-1, 1) + torch.arange(m).view(1, -1)) % 2).float() * 0.8 + 0.1
    masks = torch.stack((cb, 1 - cb)).unsqueeze(1)
    boxes = torch.tensor([_scale_one_box(3, 5, p), _scale_one_box(12, 30, p)], dtype=torch.float64)
    frame = torch.tensor([1, 2])
    assert ops.paste_boxes(boxes.to(dev()), m).cpu().tolist() == [[3, 5, 3 + p - 1, 5 + p - 1], [12, 30, 12 + p - 1, 30 + p - 1]]
    _, strings = check_against_oracle(masks, boxes, frame, (h, w))
    for s in strings:
        assert len(mots_ref.rle_from_string(s)) == 2 * (m * m // 2) + 1  # every set pixel is a run of its own


def test_rle_exact_half_is_not_set():
    h, w, m = 60, 60, 28
    p = m + 2
    g = torch.Generator().manual_seed(2)
    up = float(np.nextafter(np.float32(0.5), np.float32(1)))
    vals = torch.tensor([0.5, up, 0.25, 0.75])
    masks = vals[torch.randint(0, 4, (2, 1, m, m), generator=g)]
    boxes = torch.tensor([_scale_one_box(4, 7, p), _scale_one_box(20, 25, p)], dtype=torch.float64)
    frame = torch.tensor([1, 2])
    area, strings = gpu_rle(masks, boxes, frame, (h, w))
    for i, (x0, y0) in enumerate(((4, 7), (20, 25))):
        want = np.zeros((h, w), dtype=bool)
        want[y0 + 1:y0 + 1 + m, x0 + 1:x0 + 1 + m] = (masks[i, 0] > 0.5).numpy()
        assert np.array_equal(decode(strings[i], h, w), want) and area[i] == int(want.sum())
    ref, _ = mots_ref.mots_strings(masks, boxes, frame, (h, w))
    assert strings == ref


def test_rle_nan_mask_erases_nothing():
    h, w = 80, 90
    g = torch.Generator().manual_seed(3)
    masks = torch.rand(3, 1, 28, 28, generator=g) * 0.5 + 0.4
    masks[0] = float('nan')                                              # all NaN
    masks[2, 0, 5:9, 10:20] = float('nan')                               # a NaN patch
    boxes = torch.tensor([[10.0, 10.0, 60.0, 70.0], [20.0, 15.0, 70.0, 75.0], [5.0, 20.0, 50.0, 78.0]], dtype=torch.float64)
    frame = torch.tensor([4, 4, 4])
    area, strings = check_against_oracle(masks, boxes, frame, (h, w))
    assert area[0] == 0 and strings[0] is None and area[1] > 0 and area[2] > 0


# ------------------------------------------------------------------ ownership
def test_identical_detections_lower_index_wins():
    g = torch.Generator().manual_seed(4)
    mk = torch.rand(1, 1, 28, 28, generator=g)
    masks = mk.repeat(3, 1, 1, 1)
    boxes = torch.tensor([[10.0, 12.0, 50.0, 70.0]] * 3, dtype=torch.float64)
    area, strings = check_against_oracle(masks, boxes, torch.tensor([2, 2, 2]), (90, 80))
    assert area[0] > 0 and area[1:] == [0, 0] and strings[1:] == [None, None]


def test_nested_boxes_and_a_chain_of_three():
    g = torch.Generator().manual_seed(6)
    masks = torch.rand(5, 1, 56, 56, generator=g)
    boxes = torch.tensor([[10.0, 10.0, 90.0, 110.0], [30.0, 40.0, 60.0, 80.0],                 # nested (frame 1)
                          [5.0, 5.0, 45.0, 60.0], [30.0, 20.0, 75.0, 80.0], [60.0, 40.0, 99.0, 100.0]],  # chain (frame 2)
                         dtype=torch.float64)
    check_against_oracle(masks, boxes, torch.tensor([1, 1, 2, 2, 2]), (120, 100))


def test_sixty_four_mutually_overlapping_detections():
    g = torch.Generator().manual_seed(7)
    n = 64
    c = torch.tensor([200.0, 150.0]) + 10 * torch.randn(n, 2, generator=g, dtype=torch.float64)
    half = torch.stack((30 + 20 * torch.rand(n, generator=g, dtype=torch.float64),
                        60 + 30 * torch.rand(n, generator=g, dtype=torch.float64)), 1)
    boxes = torch.cat((c - half, c + half), 1)
    masks = torch.rand(n, 1, 28, 28, generator=g)
    area, _ = check_against_oracle(masks, boxes, torch.full((n,), 9), (300, 400))
    assert sum(a > 0 for a in area) > 32


def test_identical_boxes_in_different_frames_do_not_interact():
    masks = torch.full((3, 1, 28, 28), 0.8)
    boxes = torch.tensor([[10.0, 12.0, 50.0, 70.0]] * 3, dtype=torch.float64)
    area, strings = check_against_oracle(masks, boxes, torch.tensor([1, 2, 3]), (90, 80))
    assert area[0] > 0 and area == [area[0]] * 3 and strings == [strings[0]] * 3


def test_mask_emptied_by_its_neighbours_is_skipped(tmp_path):
    masks = torch.stack((torch.full((1, 28, 28), 0.9), torch.full((1, 28, 28), 0.7), torch.full((1, 28, 28), 0.95)))
    boxes = torch.tensor([[0.0, 0.0, 60.0, 60.0], [10.0, 10.0, 30.0, 30.0], [5.0, 40.0, 20.0, 58.0]], dtype=torch.float64)
    frame = torch.tensor([1, 1, 1])
    area, strings = check_against_oracle(masks, boxes, frame, (64, 64))
    assert area[1] == 0 and strings[1] is None and area[0] > 0 and area[2] > 0
    path = tmp_path / 'out.txt'
    assert write_mots_txt(str(path), frame.numpy(), [4, 5, 6], 2, 64, 64, strings) == 2
    assert [ln.split()[1] for ln in path.read_text().splitlines()] == ['4', '6']


# ------------------------------------------------------------------ scale, edges, determinism
def test_synthetic_sequence_against_the_oracle():
    """The 600-frame 1080 x 1920 sequence of 20 detections per frame in one call; the oracle (about a second per frame
    on the CPU) checks every 20th frame."""
    masks, boxes, frame = synth.make_mots_sequence()
    nodes = torch.nonzero(frame % 20 == 1).view(-1)
    area, strings = check_against_oracle(masks, boxes, frame, (1080, 1920), nodes=nodes)
    assert sum(s is not None for s in strings) > 0.8 * len(strings)
    again = encode_mots_masks(masks.to(dev()), boxes.to(dev()), frame.to(dev()), (1080, 1920))
    assert again == strings


def test_two_runs_give_identical_bytes():
    masks, boxes, frame = synth.make_mots_sequence(frames=50, seed=3)
    args = (masks.to(dev()), boxes.to(dev()), frame.to(dev()), (1080, 1920))
    a1, c1, p1 = ops.mots_rle(*args)
    a2, c2, p2 = ops.mots_rle(*args)
    assert torch.equal(a1, a2) and torch.equal(c1, c2) and torch.equal(p1, p2)


def test_empty_and_rejected_inputs():
    area, chars, ptr = ops.mots_rle(torch.zeros(0, 1, 56, 56, device=dev()), torch.zeros(0, 4, dtype=torch.float64, device=dev()),
                                    torch.zeros(0, dtype=torch.int64, device=dev()), (1080, 1920))
    assert area.numel() == 0 and chars.numel() == 0 and ptr.tolist() == [0]
    assert encode_mots_masks(torch.zeros(0, 56, 56, device=dev()), torch.zeros(0, 4, device=dev()),
                             torch.zeros(0, dtype=torch.int64, device=dev()), (4, 4)) == []
    m = torch.rand(2, 1, 28, 28, device=dev())
    b = torch.tensor([[1.0, 1.0, 5.0, 5.0]] * 2, dtype=torch.float64, device=dev())
    f = torch.tensor([1, 1], device=dev())
    with pytest.raises(ValueError, match='2\\^31'):
        ops.mots_rle(m, b, f, (2 ** 15, 2 ** 16))
    with pytest.raises(ValueError, match='2\\^31'):
        ops.paste_masks_in_image(m, b, (2 ** 16, 2 ** 15))
    lib = ops.lib()
    h_tot = (C.c_int64 * 2)()
    rc = lib.mpn_mots_rle_count(ops.ptr(m), 2, 28, 1, ops.ptr(b), ops.ptr(f), 2 ** 15, 2 ** 16, 0.5, ops.ptr(m), ops.ptr(f),
                                ops.ptr(f), ops.ptr(f), h_tot, ops.stream_ptr())
    assert rc == -1 and b'2^31' in lib.mpn_last_error()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ops.mots_rle(m.cpu(), b, f, (8, 8))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ops.paste_masks_in_image(m, b.cpu(), (8, 8))
    with pytest.raises(ValueError, match='non-decreasing'):
        ops.mots_rle(m, b, torch.tensor([2, 1], device=dev()), (8, 8))
    with pytest.raises(ValueError, match='square'):
        ops.mots_rle(torch.rand(2, 28, 27, device=dev()), b, f, (8, 8))
    with pytest.raises(TypeError):
        ops.mots_rle(m.double(), b, f, (8, 8))


# ------------------------------------------------------------------ end to end
def test_tracker_writes_the_oracle_result(tmp_path):
    from mpntrackseg_b200.config import default_dataset_params, default_graph_model_params
    from mpntrackseg_b200.data.mot_graph import MOTGraph
    from mpntrackseg_b200.models.mpn import MOTMPNet
    from mpntrackseg_b200.tracker import MPNTracker
    win = synth.make_window(T=6, D=5, k=4, seed=31, node_feats='pooled', with_ext=True)
    ds = default_dataset_params(top_k_nns=4, frames_per_graph=3)
    mp = default_graph_model_params(4, 3)
    model = MOTMPNet(mp).to(dev()).eval()
    model.load_state_dict(synth.make_params(mp, seed=5, gain=2.0))
    cols = synth.det_columns(win)
    cols['bb_left'] = win.feet_x - win.bb_width / 2
    cols['bb_top'] = win.feet_y - win.bb_height
    h, w = 1080, 1920
    mg = MOTGraph.from_tensors(cols, win.reid, win.x.to(dev()), win.x_ext.to(dev()),
                               {'fps': win.fps, 'frame_height': h, 'frame_width': w}, ds, inference_mode=True,
                               max_frame_dist=ds['frames_per_graph'] - 1)
    mg.construct_graph_object()
    mg.frames = sorted(set(win.frame.tolist()))
    mg.frames_per_graph = ds['frames_per_graph']
    tracker = MPNTracker(graph_model=model, eval_params={'set_pruned_edges_to_inactive': False, 'rounding_method': 'greedy'},
                         dataset_params=ds)
    tracker.full_graph = mg
    with pytest.raises(RuntimeError, match='node_preds'):
        tracker.save_mots_results(str(tmp_path / 'none.txt'))
    tracker._evaluate_graph_in_batches()
    tracker._project_graph_model_output()
    labels = tracker._assign_ped_ids()
    path = tmp_path / 'seq.txt'
    written, skipped = tracker.save_mots_results(str(path))
    node_preds = mg.graph_obj.node_preds.cpu()
    assert node_preds.shape == (win.N, 1, 56, 56)
    boxes = torch.from_numpy(np.stack((cols['bb_left'], cols['bb_top'], cols['bb_left'] + cols['bb_width'],
                                       cols['bb_top'] + cols['bb_height']), 1))
    ref, bands = mots_ref.mots_strings(node_preds, boxes, win.frame, (h, w))
    lines = path.read_text().splitlines()
    want = mots_ref.mots_lines(win.frame.tolist(), labels.cpu().tolist(), 2, h, w, ref)
    assert written == len(lines) and written + skipped == win.N and written > 0
    assert all(ln.split()[2:5] == ['2', '1080', '1920'] for ln in lines)
    if not bands:
        assert lines == want
    else:                                  # frames with a pixel near the threshold: same pixels outside that band
        by_frame = lambda ls: {f: [ln for ln in ls if int(ln.split()[0]) == f] for f in set(win.frame.tolist())}
        got_f, want_f = by_frame(lines), by_frame(want)
        for f in got_f:
            if f not in bands:
                assert got_f[f] == want_f[f], f
                continue
            assert len(got_f[f]) == len(want_f[f]), f
            keep = ~bands[f].numpy()
            for a, b in zip(got_f[f], want_f[f]):
                assert a.split()[:5] == b.split()[:5]
                assert np.array_equal(decode(a.split()[5], h, w)[keep], decode(b.split()[5], h, w)[keep])
    assert math.isfinite(float(node_preds.sum()))
