"""CPU restatement of the tracker's MOTS output stage.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE, under the same rules as the rest of ``oracle/``: only ``tests/`` and the
CPU arm of ``tools/mots_output_bench.py`` import it, as the checker.  ``tests/test_mots_references.py`` pins it to
torchvision's paste and to the worked examples of pycocotools' RLE format.

reference: tracker/mpn_tracker.py:267-298 (torchvision ``paste_masks_in_image``, ``ensure_unique_masks``, pycocotools
RLE) and :398-417 (the result file).  pycocotools is not vendored; ``rle_counts`` / ``rle_to_string`` /
``rle_from_string`` restate ``rleEncode`` / ``rleToString`` / ``rleFrString`` of its ``maskApi.c``.  The overlap rule and
the line format are this project's (DESIGN.md, MOTS output):
  1. integer box: torchvision's ``expand_boxes`` with scale (M + 2 pad) / M in the boxes' dtype, ``.to(int64)``;
  2. p_i(y, x): torchvision's ``paste_mask_in_image`` of the zero-padded mask, here on float64;
  3. within a frame a pixel belongs to the node with the largest p_i (ties: lower index, NaN as -inf), and to its mask
     where p_i > threshold;
  4. pycocotools RLE of the column-major H x W mask;
  5. ``"<frame> <id> <class_id> <H> <W> <rle>"`` per node with a non-empty mask, sorted by frame, then node index.
"""
import numpy as np
import torch
import torch.nn.functional as F
from torchvision.models.detection.roi_heads import paste_mask_in_image


def integer_boxes(boxes, mask_size, padding=1):
    """[N, 4] int64: torchvision's ``expand_boxes`` (roi_heads.py) + ``.to(torch.int64)``."""
    scale = float(mask_size + 2 * padding) / mask_size
    w_half = (boxes[:, 2] - boxes[:, 0]) * 0.5
    h_half = (boxes[:, 3] - boxes[:, 1]) * 0.5
    x_c = (boxes[:, 2] + boxes[:, 0]) * 0.5
    y_c = (boxes[:, 3] + boxes[:, 1]) * 0.5
    w_half *= scale
    h_half *= scale
    out = torch.zeros_like(boxes)
    out[:, 0], out[:, 2] = x_c - w_half, x_c + w_half
    out[:, 1], out[:, 3] = y_c - h_half, y_c + h_half
    return out.to(torch.int64)


def _inside(b, h, w):
    return max(int(b[0]), 0) < min(int(b[2]) + 1, w) and max(int(b[1]), 0) < min(int(b[3]) + 1, h)


def paste(masks, boxes, img_shape, padding=1):
    """[N, H, W] float64 p_i(y, x): torchvision's ``paste_mask_in_image`` on float64 masks with the integer boxes of
    step 1.  A box with no pixel inside the image gives zeros (torchvision's slicing would raise or wrap there)."""
    m = masks.reshape(masks.shape[0], masks.shape[-2], masks.shape[-1]).double()
    ib = integer_boxes(boxes, m.shape[-1], padding)
    h, w = int(img_shape[0]), int(img_shape[1])
    out = torch.zeros((m.shape[0], h, w), dtype=torch.float64)
    padded = F.pad(m, (padding,) * 4)
    for i in range(m.shape[0]):
        if _inside(ib[i], h, w):
            out[i] = paste_mask_in_image(padded[i], ib[i], h, w)
    return out


def owner_masks(probs, frame, threshold=0.5):
    """[N, H, W] bool: pixel (y, x) of node i's mask iff i has the largest probability of its frame there (NaN as
    -inf, ties to the lower index) and that probability is > threshold."""
    p = torch.nan_to_num(probs, nan=float('-inf'))
    frame = torch.as_tensor(frame)
    out = torch.zeros(p.shape, dtype=torch.bool)
    for f in torch.unique(frame).tolist():
        idx = torch.nonzero(frame == f).view(-1)
        win = torch.argmax(p[idx], dim=0)               # first maximum = lower node index
        for a, i in enumerate(idx.tolist()):
            out[i] = (win == a) & (p[i] > threshold)
    return out


def rle_counts(mask):
    """pycocotools ``rleEncode`` of one H x W mask in column-major order: run lengths starting with the zeros."""
    flat = np.asarray(mask, dtype=np.uint8).flatten(order='F')
    if flat.size == 0:
        return [0]
    change = np.flatnonzero(flat[1:] != flat[:-1]) + 1
    edges = np.concatenate(([0], change, [flat.size]))
    counts = np.diff(edges).tolist()
    return ([0] + counts) if flat[0] else counts


def rle_to_string(counts):
    """pycocotools ``rleToString``."""
    s = []
    for i, x in enumerate(counts):
        x = int(x)
        if i > 2:
            x -= int(counts[i - 2])
        more = True
        while more:
            c = x & 0x1f
            x >>= 5
            more = (x != -1) if (c & 0x10) else (x != 0)
            if more:
                c |= 0x20
            s.append(chr(c + 48))
    return ''.join(s)


def rle_from_string(s):
    """pycocotools ``rleFrString``: the counts of a string."""
    counts, p = [], 0
    while p < len(s):
        x = k = 0
        more = True
        while more:
            c = ord(s[p]) - 48
            x |= (c & 0x1f) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(counts) > 2:
            x += counts[-2]
        counts.append(x)
    return counts


def rle_decode(counts, h, w):
    """H x W bool mask of column-major counts."""
    flat = np.zeros(h * w, dtype=bool)
    pos, val = 0, False
    for c in counts:
        if val:
            flat[pos:pos + c] = True
        pos += c
        val = not val
    return flat.reshape((w, h)).T


def mots_strings(masks, boxes, frame, img_shape, threshold=0.5, band=1e-6):
    """(strings, bands): the RLE string of every node's mask (None when it is empty), frame by frame; bands maps each
    frame that has a pixel whose probability (of any of its nodes) lies within ``band`` of the threshold to the [H, W]
    bool mask of those pixels."""
    frame = torch.as_tensor(frame).view(-1)
    strings, bands = [None] * frame.numel(), {}
    for f in torch.unique(frame).tolist():
        idx = torch.nonzero(frame == f).view(-1)
        probs = paste(masks[idx], boxes[idx], img_shape)
        near = ((probs - threshold).abs() <= band).any(0)
        if bool(near.any()):
            bands[int(f)] = near
        for i, o in zip(idx.tolist(), owner_masks(probs, torch.zeros(idx.numel(), dtype=torch.int64), threshold)):
            if bool(o.any()):
                strings[i] = rle_to_string(rle_counts(o.numpy()))
    return strings, bands


def mots_lines(frames, ids, class_id, h, w, strings):
    """Lines of the result file: one per non-empty mask, sorted by frame, then node index."""
    order = sorted((int(f), i) for i, f in enumerate(frames) if strings[i] is not None)
    return [f'{f} {int(ids[i])} {int(class_id)} {int(h)} {int(w)} {strings[i]}' for f, i in order]
