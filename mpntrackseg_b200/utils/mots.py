"""MOTS result of the tracker: each node's mask as an RLE string, and the result file.
reference: utils/mots.py (mask helpers) and tracker/mpn_tracker.py:267-298, :398-417.

The paste, the one-owner-per-pixel rule and the run-length encoding run on the GPU (``ops.mots_rle``); only the
characters of the strings come back to the host.  The contract is stated in DESIGN.md (MOTS output).
"""
import numpy as np

from .. import ops

# MOTS20 and KITTI-MOTS class id of pedestrians
PEDESTRIAN_CLASS_ID = 2


def encode_mots_masks(masks, boxes, frame, img_shape, threshold=0.5):
    """RLE strings (pycocotools' ``rleToString`` format, column-major H x W) of every node's mask after the
    one-owner-per-pixel rule of its frame: a list of N ``str``, ``None`` where the mask is empty.
    masks [N, 1, M, M] or [N, M, M] fp32 probabilities, boxes [N, 4] (x1, y1, x2, y2), frame [N] int64 non-decreasing,
    img_shape (H, W); all on the current CUDA device."""
    _, chars, char_ptr = ops.mots_rle(masks, boxes, frame, img_shape, threshold)
    data = chars.cpu().numpy().tobytes()
    ptr = char_ptr.cpu().tolist()
    return [data[a:b].decode('ascii') if b > a else None for a, b in zip(ptr[:-1], ptr[1:])]


def write_mots_txt(path, frames, ids, class_id, height, width, strings):
    """Writes ``"<frame> <id> <class_id> <H> <W> <rle>"`` for every node whose string is not None, sorted by frame,
    then by node index.  Returns the number of lines written."""
    frames = np.asarray(frames, dtype=np.int64).reshape(-1)
    ids = np.asarray(ids, dtype=np.int64).reshape(-1)
    if not (len(frames) == len(ids) == len(strings)):
        raise ValueError(f'{len(frames)} frames, {len(ids)} ids and {len(strings)} strings')
    order = np.argsort(frames, kind='stable')
    lines = [f'{frames[i]} {ids[i]} {int(class_id)} {int(height)} {int(width)} {strings[i]}\n'
             for i in order if strings[i] is not None]
    with open(path, 'w') as fh:
        fh.writelines(lines)
    return len(lines)
