"""``Segmentation`` chunk and its ``evaluate`` (reference chunk/segmentation.py:18-67 -> lib/gala/evaluate.py).

``evaluate`` scores a segmentation against a ground truth with the reference's five numbers -- Rand index, adjusted Rand
index, variation of information, Fowlkes-Mallows index, edit distance -- quirks included (see
oracle/evaluation_oracle.py).  Both volumes are uploaded and the contingency table is built and reduced on the GPU
(``DeviceChunk.evaluate``); there is no CPU fallback.  The reference's ``remap``, ``mask_fragments`` and ``mask_except`` are
not part of this class.
"""
from __future__ import annotations

import numpy as np

from .base import Chunk

SCORE_KEYS = ("rand_index", "adjusted_rand_index", "variation_of_information", "fowlkes_mallows_index", "edit_distance")


def scores_from_sums(sums) -> dict:
    """The reference's result dict from the device's integer sums (a ``_native.ContingencySums``), in gala's order of float64
    operations (evaluate.py:1183-1300 for Rand / adjusted Rand / Fowlkes-Mallows).  VI = (sum a' log2 a' + sum b' log2 b'
    - 2 sum n log2 n) / N' over the table without label 0, which equals gala's H(Y|X) + H(X|Y); the three sums arrive in
    exact fixed point, so the difference is taken exactly and rounded once.  The edit distance is
    (#{pairs without label 0 above size_threshold} - #{non-zero seg ids}, 0.0), as the reference's (evaluate.py:194-209)
    computes it."""
    def fixed(v):
        return int(v[0]) | (int(v[1]) << 64)

    with np.errstate(divide="ignore", invalid="ignore"):
        n, sum1, sum2, sum3 = (np.float64(v) for v in (sums.voxels, sums.sum_sq_pairs, sums.sum_sq_seg, sums.sum_sq_gt))
        a = (sum1 - n) / 2.0
        b = (sum2 - sum1) / 2
        c = (sum3 - sum1) / 2
        d = (sum1 + n ** 2 - sum2 - sum3) / 2
        ri = (a + d) / (a + b + c + d)
        nk = a + b + c + d
        ari = (nk * (a + d) - ((a + b) * (a + c) + (c + d) * (b + d))) / (nk ** 2 - ((a + b) * (a + c) + (c + d) * (b + d)))
        fm = a / (np.sqrt((a + b) * (a + c)))
        vi_fixed = fixed(sums.xlogx_seg) + fixed(sums.xlogx_gt) - 2 * fixed(sums.xlogx_pairs)
        vi = np.float64(vi_fixed / 2 ** 62) / np.float64(sums.nonzero_voxels)
    edit = (np.float64(int(sums.pairs_over_threshold) - int(sums.seg_labels)), np.float64(0.0))
    return dict(zip(SCORE_KEYS, (ri, ari, vi, fm, edit)))


def format_scores(scores: dict) -> str:
    """The five lines the reference's ``Segmentation.evaluate`` prints (chunk/segmentation.py:56-60), in its order."""
    return (f"rand index: {scores['rand_index']: .3f}\n"
            f"adjusted rand index: {scores['adjusted_rand_index']: .3f}\n"
            f"variation of information: {scores['variation_of_information']: .3f}\n"
            f"edit distance: {scores['edit_distance']}\n"
            f"Fowlkes Mallows Index: {scores['fowlkes_mallows_index']: .3f}\n")


def label_array(array, what: str) -> np.ndarray:
    """A host label volume as uint32 or uint64 for the device: signed ids are read as unsigned of the same width and uint8 /
    uint16 (and bool) are widened -- bijections that keep 0, which leave every score unchanged."""
    array = np.asarray(array)
    if array.dtype != bool and not np.issubdtype(array.dtype, np.integer):
        raise TypeError(f"{what} must be an integer label volume, not {array.dtype}")
    if array.dtype.itemsize < 4:
        array = array.astype(np.int32 if array.dtype.kind == "i" else np.uint32)
    return np.ascontiguousarray(array).view(np.uint64 if array.dtype.itemsize == 8 else np.uint32)


class Segmentation(Chunk):
    """A chunk of segmentation volume: a 3-D integer array."""

    def __init__(self, array, **kwargs):
        arr = array.array if isinstance(array, Chunk) else array
        if not isinstance(arr, np.ndarray) or arr.ndim != 3:
            raise ValueError("a Segmentation is a 3-D (z, y, x) array")
        if not np.issubdtype(arr.dtype, np.integer):
            raise TypeError(f"a Segmentation holds integer ids, not {arr.dtype}")
        super().__init__(array, **kwargs)

    @classmethod
    def from_chunk(cls, chunk: Chunk) -> "Segmentation":
        if not isinstance(chunk, Chunk):
            raise TypeError("from_chunk takes a Chunk")
        return cls(chunk.array, voxel_offset=chunk.voxel_offset, voxel_size=chunk.voxel_size)

    def evaluate(self, groundtruth, size_threshold: float = 1000) -> dict:
        """Scores of this segmentation against ``groundtruth`` (a Chunk or an ndarray of the same shape), like the
        reference's: a dict with ``rand_index``, ``adjusted_rand_index``, ``variation_of_information``,
        ``fowlkes_mallows_index`` and ``edit_distance`` (false merges, false splits), whose five lines are also printed.
        ``size_threshold``: pairs of at most this many voxels are left out of the edit distance."""
        from .device import DeviceChunk
        gt = groundtruth.array if isinstance(groundtruth, Chunk) else np.asarray(groundtruth)
        if gt.shape != self.array.shape:
            raise ValueError(f"the ground truth has shape {gt.shape}, the segmentation {self.array.shape}")
        seg, gt = label_array(self.array, "the segmentation"), label_array(gt, "the ground truth")
        seg = DeviceChunk.from_labels(seg)
        truth = DeviceChunk.from_labels(gt, device=seg.tensor.device)
        scores = seg.evaluate(truth, size_threshold=size_threshold)
        print(format_scores(scores), end="")
        return scores
