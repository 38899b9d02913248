"""CPU checks of the MOTS output restatement (oracle/mots_ref.py): the paste against torchvision, the RLE against the
worked examples of pycocotools' format, the string round trip, and the result file's line format and order."""
import numpy as np
import pytest
import torch
from torchvision.models.detection.roi_heads import paste_masks_in_image

from oracle import mots_ref


@pytest.mark.parametrize('m,padding', [(28, 1), (56, 1), (28, 0), (28, 2)])
def test_paste_equals_torchvision_bit_for_bit(m, padding):
    g = torch.Generator().manual_seed(m + padding)
    h, w = 97, 131
    masks = torch.rand(9, 1, m, m, generator=g, dtype=torch.float64)
    boxes = torch.tensor([[20.3, 15.7, 60.9, 80.2],            # inside
                          [-12.4, 30.0, 25.5, 70.1],           # partly outside the left edge
                          [100.2, 10.0, 150.8, 40.0],          # right edge
                          [40.0, -20.6, 70.3, 12.9],           # top edge
                          [10.0, 70.2, 50.0, 120.7],           # bottom edge
                          [-30.0, -40.0, 170.5, 140.0],        # larger than the image
                          [5.0, 5.0, 5.4, 5.2],                # 1-pixel box
                          [0.3, 0.2, 1.1, 0.9],                # expanded corners truncate toward zero
                          [60.5, 50.5, 61.0, 51.0]], dtype=torch.float64)
    ref = paste_masks_in_image(masks, boxes, (h, w), padding=padding)[:, 0]
    got = mots_ref.paste(masks, boxes, (h, w), padding=padding)
    assert torch.equal(got, ref)


def test_integer_boxes_truncate_toward_zero():
    b = mots_ref.integer_boxes(torch.tensor([[-0.5, -1.0, 3.0, 2.0]], dtype=torch.float64), 28, 1)
    # w_half = 3.5 * 0.5 * 30/28 = 1.875, x_c = 1.25: x0 = -0.625 -> 0; h_half = 1.607..., y_c = 0.5: y0 = -1.107 -> -1
    assert b.tolist() == [[0, -1, 3, 2]]


def test_rle_worked_examples():
    m = np.zeros((4, 3), bool)
    m[1:3, 1] = True
    m[0, 2] = True
    assert mots_ref.rle_counts(m) == [5, 2, 1, 1, 3]
    assert mots_ref.rle_to_string([5, 2, 1, 1, 3]) == '521O2'
    h, w = 1080, 1920
    m = np.zeros((h, w), bool)
    m[100:400, 500:620] = True
    c = mots_ref.rle_counts(m)
    assert c[:4] == [540100, 300, 780, 300] and len(c) == 241
    assert mots_ref.rle_to_string(c).startswith('T^_`0\\9\\h000')
    assert mots_ref.rle_to_string(mots_ref.rle_counts(np.zeros((h, w), bool))) == 'PPYo1'
    assert mots_ref.rle_to_string(mots_ref.rle_counts(np.ones((h, w), bool))) == '0PPYo1'


def test_rle_decode_inverts_counts():
    rng = np.random.default_rng(4)
    for shape in ((1, 1), (1, 17), (13, 1), (31, 29)):
        m = rng.random(shape) < 0.4
        assert np.array_equal(mots_ref.rle_decode(mots_ref.rle_counts(m), *shape), m)


def test_rle_string_round_trip():
    rng = np.random.default_rng(7)
    for _ in range(50):
        m = rng.random((rng.integers(1, 40), rng.integers(1, 40))) < rng.random()
        c = mots_ref.rle_counts(m)
        assert mots_ref.rle_from_string(mots_ref.rle_to_string(c)) == c
    big = [2 ** 20 + 3, 2 ** 21, 5, 2 ** 30 + 7, 1, 2 ** 31 - 2]               # counts above 2^20
    neg = [100, 90000, 3, 5, 80000, 1, 70000, 2]                             # negative deltas cnt[i] - cnt[i-2]
    for c in (big, neg, [0], [0, 5], [7]):
        assert mots_ref.rle_from_string(mots_ref.rle_to_string(c)) == c


def test_owner_rule_ties_nan_and_threshold():
    p = torch.tensor([[[0.7, 0.5, float('nan')]], [[0.7, 0.4, 0.6]], [[0.9, 0.6, 0.2]]], dtype=torch.float64)
    own = mots_ref.owner_masks(p, torch.tensor([1, 1, 2]))
    assert own[0, 0].tolist() == [True, False, False]       # tie -> lower index; 0.5 is not > 0.5
    assert own[1, 0].tolist() == [False, False, True]       # the NaN erases nothing
    assert own[2, 0].tolist() == [True, True, False]        # another frame does not interact


def test_write_mots_txt_format_and_order(tmp_path):
    from mpntrackseg_b200.utils.mots import write_mots_txt
    frames = [3, 1, 3, 1, 2]
    ids = [7, 4, 0, 9, 4]
    strings = ['a1', None, 'c3', 'd4', 'e5']
    path = tmp_path / 'seq.txt'
    assert write_mots_txt(str(path), frames, ids, 2, 1080, 1920, strings) == 4
    assert path.read_text().splitlines() == ['1 9 2 1080 1920 d4', '2 4 2 1080 1920 e5', '3 7 2 1080 1920 a1',
                                             '3 0 2 1080 1920 c3']
    assert mots_ref.mots_lines(frames, ids, 2, 1080, 1920, strings) == path.read_text().splitlines()
