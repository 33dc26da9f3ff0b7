"""CPU oracle for the operators either side of `inference` (SURVEY.md section 8 f3) -- TEST INFRASTRUCTURE.

Plain numpy restatements, each citing the reference file:line it follows, of
  * ``Image.normalize_contrast``   chunk/image/base.py:30-132  (upstream: uint8 LUT per section)
  * ``Chunk.maskout``              chunk/base.py:811-829       (up/downstream: multiply by a coarser mask)
  * ``Chunk.crop_margin``          chunk/base.py:691-726       (downstream)
  * ``AffinityMap.quantize``       chunk/affinity_map/base.py:33-57 (downstream: affinity -> uint8 image)

Pinning, bit-exact: ``tests/test_operators_oracle.py`` compares these functions with outputs of the REAL reference
classes, ``tests/golden/operators.npz`` (``tests/golden/make_golden_operators.py``) and, on fresh random inputs,
``tests/golden/reference_pins.*`` (``tests/golden/make_golden_reference.py``).

Reference quirks restated literally (the product mirrors them and DESIGN.md lists them):
  * ``normalize_contrast(per_section=True)``: the whole-array branch is the ``else`` clause of the ``for`` loop over
    sections (image/base.py:113-132), so it ALSO runs after the per-section pass; with ``per_section=False`` nothing runs.
  * the histogram is ``np.bincount(..., minlength=255)`` (image/base.py:106): 255 bins unless the value 255 occurs, and
    bin 0 (pure black) is zeroed before the cdf (image/base.py:38).
Never imported by the product path.
"""
from __future__ import annotations

import numpy as np


# ---- clamping values (reference chunk/image/base.py:30-62) -----------------------------------
def find_section_clamping_values(hist: np.ndarray, lower_clip_fraction: float, upper_clip_fraction: float):
    filtered = np.array(hist, dtype=np.int64)
    filtered[0] = 0  # pure black carries no information (:38)
    cdf = np.cumsum(filtered).astype(np.uint64)  # the reference accumulates in uint64 in a python loop (:40-43)
    total = int(cdf[-1])
    if total == 0:
        return 0, 0
    lower = 0
    for i, val in enumerate(cdf):  # (:50-54)
        if float(val) / float(total) > lower_clip_fraction:
            break
        lower = i
    upper = 0
    for i, val in enumerate(cdf):  # (:56-60)
        if float(val) / float(total) > 1 - upper_clip_fraction:
            break
        upper = i
    return lower, upper


# ---- lookup table (reference chunk/image/base.py:64-91) --------------------------------------
def hist_to_lookup_table(hist, lower_clip_fraction, upper_clip_fraction, minval=1, maxval=255):
    lower, upper = find_section_clamping_values(hist, lower_clip_fraction, upper_clip_fraction)
    if lower == upper:
        return None  # "no need to perform any transform" (:78-81)
    lut = np.arange(0, 256, dtype=np.float32)
    lut = (lut - float(lower)) * (maxval / (float(upper) - float(lower)))  # float32 array x python scalar (:85-86)
    np.clip(lut, minval, maxval, out=lut)
    lut = np.round(lut)  # half to even
    return lut.astype(np.uint8)


def _normalize_array(array, lower_clip_fraction, upper_clip_fraction, minval, maxval):  # (:101-111)
    hist = np.bincount(array.flatten(), minlength=255)
    lut = hist_to_lookup_table(hist, lower_clip_fraction, upper_clip_fraction, minval=minval, maxval=maxval)
    if lut is not None:
        array = lut[array]
    return array


# ---- Image.normalize_contrast (reference chunk/image/base.py:93-132) -------------------------
def normalize_contrast(image: np.ndarray, lower_clip_fraction=0.01, upper_clip_fraction=0.01, minval=1, maxval=255,
                       per_section=True) -> np.ndarray:
    """image: (z, y, x) uint8.  Returns the array the reference leaves in ``Image.array``."""
    assert image.dtype == np.uint8 and image.ndim == 3
    out = image.copy()
    if per_section:
        for z in range(out.shape[0]):  # (:114-123)
            out[z] = _normalize_array(out[z], lower_clip_fraction, upper_clip_fraction, minval, maxval)
        # for-else: the loop never breaks, so the whole-array pass runs as well (:124-131)
        out = _normalize_array(out, lower_clip_fraction, upper_clip_fraction, minval, maxval)
    return out


# ---- Chunk.maskout (reference chunk/base.py:811-829): self = mask, argument = the chunk that is modified ---------
def maskout(mask: np.ndarray, mask_voxel_size, chunk: np.ndarray, chunk_voxel_size) -> np.ndarray:
    mvs, cvs = tuple(mask_voxel_size), tuple(chunk_voxel_size)
    assert all(m >= c for m, c in zip(mvs, cvs))          # (:816)
    assert all(m % c == 0 for m, c in zip(mvs, cvs))      # (:819)
    factor = tuple(m // c for m, c in zip(mvs, cvs))
    out = chunk.copy()
    for offset in np.ndindex(factor):                     # (:822-828)
        out[..., offset[0]::factor[0], offset[1]::factor[1], offset[2]::factor[2]] *= mask
    return out


# ---- Chunk.crop_margin (reference chunk/base.py:691-726) --------------------------------------
def crop_margin(array: np.ndarray, voxel_offset, margin_size):
    sz, sy, sx = array.shape[-3:]
    m = tuple(margin_size)
    if len(m) == 3:
        new = array[..., m[0]:sz - m[0], m[1]:sy - m[1], m[2]:sx - m[2]]
    elif len(m) == 6:  # -z,-y,-x,+z,+y,+x
        new = array[..., m[0]:sz - m[3], m[1]:sy - m[4], m[2]:sx - m[5]]
    else:
        raise ValueError('only support 3 or 6 elements.')
    offset = tuple(o + mm for o, mm in zip(voxel_offset, m))  # zip stops after the three lower margins (:721-722)
    return new, offset


# ---- AffinityMap.quantize (reference chunk/affinity_map/base.py:33-57) ------------------------
def quantize(aff: np.ndarray, mode: str = 'xy') -> np.ndarray:
    if mode == 'z':
        image = aff[-1, :, :, :]
    elif mode == 'xy':
        image = (aff[0, ...] + aff[1, ...]) / 2.
    else:
        raise ValueError(f'only support xy and z mode, but got {mode}')
    return (image * 255.).astype(np.uint8)
