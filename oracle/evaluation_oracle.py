"""CPU oracle of `evaluate-segmentation`: the reference's scores restated in numpy (reference chunk/segmentation.py:33-67,
lib/gala/evaluate.py), checked against the real reference's outputs in tests/golden/evaluate_pins.json.

The reference builds ``contingency_table`` (evaluate.py:212-250) as a scipy ``coo_matrix`` of shape (max seg id + 1,
max gt id + 1); here the table is the list of the label pairs that occur, ``np.unique`` of the stacked pairs -- the same
entries without the empty rows and columns, which none of the five scores reads.  Every score is computed from a handful
of sums over that list, in gala's order of float64 operations:

* Rand, adjusted Rand, Fowlkes-Mallows (evaluate.py:1183-1300): the table WITHOUT ignored labels (``norm=False``, label 0
  counts); n, sum1 = sum n_ij^2, sum2 = sum a_i^2, sum3 = sum b_j^2 -> a, b, c, d -> the three formulas.
* variation of information (evaluate.py:623-691, 1049-1101): label 0 ignored on both sides, log2, H(Y|X) + H(X|Y), which
  over the table with those voxels dropped equals (sum a' log a' + sum b' log b' - 2 sum n log n) / N' (a', b' the marginals
  of that reduced table, N' its total); NaN when N' = 0, like gala's 0/0.
* edit distance (evaluate.py:155-209): label 0 ignored, entries <= size_threshold zeroed.  false_merges = #{entries left}
  - #{distinct non-zero seg ids} (the rows of the relabelled table, empty ones included; it can be negative);
  false_splits is always 0.0 because ``(r.sum(axis=0) - 1)[1:]`` slices the one row of a 1 x n ``np.matrix`` away.
"""
from __future__ import annotations

import numpy as np

SCORE_KEYS = ("rand_index", "adjusted_rand_index", "variation_of_information", "fowlkes_mallows_index", "edit_distance")


def contingency_pairs(seg, gt):
    """-> (seg_ids, gt_ids, counts) uint64, one entry per label pair that occurs, sorted by (seg id, gt id)."""
    s = np.asarray(seg).astype(np.uint64).ravel()
    g = np.asarray(gt).astype(np.uint64).ravel()
    if s.shape != g.shape:
        raise ValueError("seg and gt must have the same shape")
    pairs, counts = np.unique(np.stack([s, g], axis=1), axis=0, return_counts=True)
    return pairs[:, 0].copy(), pairs[:, 1].copy(), counts.astype(np.uint64)


def _xlogx_sum(v) -> float:
    v = np.asarray(v, np.float64)
    v = v[v > 1]
    return float(np.sum(v * np.log2(v)))


def sums(seg, gt, size_threshold=1000):
    """The sums the scores are made of (the fields of cfb_contingency_sums; the x log2 x sums as floats)."""
    s, g, c = contingency_pairs(seg, gt)
    ci = [int(v) for v in c]
    _, a = _group(s, c)
    _, b = _group(g, c)
    nz = (s != 0) & (g != 0)
    _, a_nz = _group(s[nz], c[nz])
    _, b_nz = _group(g[nz], c[nz])
    return dict(voxels=int(np.asarray(seg).size), entries=int(c.size), sum_sq_pairs=sum(x * x for x in ci),
                sum_sq_seg=sum(int(x) ** 2 for x in a), sum_sq_gt=sum(int(x) ** 2 for x in b), nonzero_voxels=int(c[nz].sum()),
                seg_labels=int(np.count_nonzero(np.unique(s) != 0)),
                pairs_over_threshold=int(np.count_nonzero(c[nz].astype(np.float64) > size_threshold)),
                xlogx_pairs=_xlogx_sum(c[nz]), xlogx_seg=_xlogx_sum(a_nz), xlogx_gt=_xlogx_sum(b_nz))


def _group(ids, counts):
    """-> (distinct ids, summed counts)"""
    if ids.size == 0:
        return ids, np.zeros(0, np.uint64)
    u, inv = np.unique(ids, return_inverse=True)
    out = np.zeros(u.size, np.uint64)
    np.add.at(out, inv.ravel(), counts.astype(np.uint64))
    return u, out


def rand_values(n, sum1, sum2, sum3):
    """evaluate.py:1183-1221 on the four sums (float64)."""
    n, sum1, sum2, sum3 = (np.float64(v) for v in (n, sum1, sum2, sum3))
    a = (sum1 - n) / 2.0
    b = (sum2 - sum1) / 2
    c = (sum3 - sum1) / 2
    d = (sum1 + n ** 2 - sum2 - sum3) / 2
    return a, b, c, d


def scores_from_sums(voxels, sum_sq_pairs, sum_sq_seg, sum_sq_gt, nonzero_voxels, seg_labels, pairs_over_threshold,
                     xlogx_pairs, xlogx_seg, xlogx_gt):
    """The reference's result dict from the sums; the x log2 x sums may be floats or exact fractions (anything that
    subtracts exactly and converts with float())."""
    with np.errstate(divide="ignore", invalid="ignore"):
        a, b, c, d = rand_values(voxels, sum_sq_pairs, sum_sq_seg, sum_sq_gt)
        ri = (a + d) / (a + b + c + d)                                             # evaluate.py:1224-1244
        nk = a + b + c + d
        ari = (nk * (a + d) - ((a + b) * (a + c) + (c + d) * (b + d))) / (      # evaluate.py:1247-1270
            nk ** 2 - ((a + b) * (a + c) + (c + d) * (b + d)))
        fm = a / (np.sqrt((a + b) * (a + c)))                                      # evaluate.py:1273-1296
        vi = np.float64(float(xlogx_seg + xlogx_gt - 2 * xlogx_pairs)) / np.float64(nonzero_voxels)
    edit = (np.float64(int(pairs_over_threshold) - int(seg_labels)), np.float64(0.0))
    return dict(zip(SCORE_KEYS, (ri, ari, vi, fm, edit)))


def evaluate(seg, gt, size_threshold=1000):
    """Segmentation(seg).evaluate(gt, size_threshold) of the reference, without its printout."""
    s = sums(seg, gt, size_threshold)
    return scores_from_sums(s["voxels"], s["sum_sq_pairs"], s["sum_sq_seg"], s["sum_sq_gt"], s["nonzero_voxels"], s["seg_labels"],
                            s["pairs_over_threshold"], s["xlogx_pairs"], s["xlogx_seg"], s["xlogx_gt"])


def format_scores(scores) -> str:
    """The five lines Segmentation.evaluate prints (chunk/segmentation.py:56-60), in its order."""
    return (f"rand index: {scores['rand_index']: .3f}\n"
            f"adjusted rand index: {scores['adjusted_rand_index']: .3f}\n"
            f"variation of information: {scores['variation_of_information']: .3f}\n"
            f"edit distance: {scores['edit_distance']}\n"
            f"Fowlkes Mallows Index: {scores['fowlkes_mallows_index']: .3f}\n")
