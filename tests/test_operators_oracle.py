"""Pins oracle/operators_oracle.py (SURVEY.md section 8 f3) to golden vectors made by the REAL reference
(tests/golden/make_golden_operators.py) and to what the reference classes computed on fresh random inputs
(tests/golden/make_golden_reference.py)."""
import os

import numpy as np
import pytest

from oracle import operators_oracle as OP

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "operators.npz")


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(GOLDEN))


NC_CASES = {"nc_default": dict(), "nc_custom": dict(lower_clip_fraction=0.05, upper_clip_fraction=0.02, minval=0, maxval=200),
            "nc_zero_clip": dict(lower_clip_fraction=0.0, upper_clip_fraction=0.0), "nc_not_per_section": dict(per_section=False)}


@pytest.mark.parametrize("tag", sorted(NC_CASES))
def test_normalize_contrast_golden(gold, tag):
    out = OP.normalize_contrast(gold["image"], **NC_CASES[tag])
    assert out.dtype == np.uint8
    np.testing.assert_array_equal(out, gold[tag])


def test_normalize_contrast_quirks(gold):
    # per_section=False is a no-op in the reference (the whole-array branch is the for loop's else clause)
    np.testing.assert_array_equal(gold["nc_not_per_section"], gold["image"])
    # black and constant sections are left alone by the per-section pass, but the trailing whole-array pass still applies
    assert (gold["nc_default"] != gold["image"]).any()


def test_quantize_maskout_crop_golden(gold):
    np.testing.assert_array_equal(OP.quantize(gold["aff"], "xy"), gold["quant_xy"])
    np.testing.assert_array_equal(OP.quantize(gold["aff"], "z"), gold["quant_z"])
    with pytest.raises(ValueError):
        OP.quantize(gold["aff"], "yz")
    np.testing.assert_array_equal(OP.maskout(gold["mask"], (2, 4, 4), gold["aff"], (1, 1, 1)), gold["maskout_aff"])
    np.testing.assert_array_equal(OP.maskout(gold["mask"], (8, 16, 16), gold["image2"], (4, 4, 4)), gold["maskout_img"])
    a3, o3 = OP.crop_margin(gold["aff"], (5, 6, 7), (1, 2, 3))
    a6, o6 = OP.crop_margin(gold["aff"], (5, 6, 7), (1, 0, 3, 2, 4, 0))
    np.testing.assert_array_equal(a3, gold["crop3"]); assert tuple(o3) == tuple(gold["crop3_offset"])
    np.testing.assert_array_equal(a6, gold["crop6"]); assert tuple(o6) == tuple(gold["crop6_offset"])
    with pytest.raises(ValueError):
        OP.crop_margin(gold["aff"], (0, 0, 0), (1, 2))


def real_reference_case(seed):
    rng = np.random.default_rng(seed)
    z, y, x = 5, 33, 47
    img = (rng.random((z, y, x)) ** (1 + seed) * rng.integers(60, 256)).astype(np.uint8)
    img[seed % z] //= 8
    lo, hi = [(0.01, 0.01), (0.1, 0.0), (0.0, 0.2)][seed]
    aff = rng.random((3, 4, 12, 10), dtype=np.float32)
    mask = rng.integers(0, 2, size=(2, 3, 5), dtype=np.uint8)
    return img, (lo, hi, 1 + seed, 255 - 10 * seed, True), aff, mask


MARGINS = ((1, 2, 3), (0, 1, 2, 1, 0, 3))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_against_real_reference(pins, seed):
    """normalize-contrast, quantize, maskout and crop-margin on fresh random inputs: oracle == the reference's Image /
    AffinityMap / Chunk methods, bit for bit (recorded by tests/golden/make_golden_reference.py)."""
    img, nc_args, aff, mask = real_reference_case(seed)
    pins.exact(f"operators/{seed}/normalize_contrast", OP.normalize_contrast(img, *nc_args))
    for mode in ("xy", "z"):
        pins.exact(f"operators/{seed}/quantize_{mode}", OP.quantize(aff, mode))
    pins.exact(f"operators/{seed}/maskout", OP.maskout(mask, (8, 16, 8), aff, (4, 4, 4)))
    for k, margin in enumerate(MARGINS):
        a, o = OP.crop_margin(aff, (3, 2, 1), margin)
        pins.exact(f"operators/{seed}/crop_margin/{k}", a)
        pins.value(f"operators/{seed}/crop_margin/{k}/offset", tuple(o))


def normalize_contrast_cases():
    """Random shapes, clip fractions and output ranges, including degenerate histograms (empty, single value, value 255
    present / absent)."""
    rng = np.random.default_rng(85)
    for k in range(60):
        z, y, x = int(rng.integers(1, 5)), int(rng.integers(1, 25)), int(rng.integers(1, 25))
        lo = float(rng.choice([0.0, 0.01, 0.1, 0.5, 0.9, 1.0]))
        hi = float(rng.choice([0.0, 0.01, 0.1, 0.5, 1.0]))
        mn, mx = int(rng.integers(0, 41)), int(rng.integers(41, 256))
        kind = ("uniform", "dark", "top", "const", "zero")[k % 5]
        if kind == "uniform":
            img = rng.integers(0, 256, (z, y, x), dtype=np.uint8)
        elif kind == "dark":
            img = rng.integers(0, 12, (z, y, x), dtype=np.uint8)
        elif kind == "top":
            img = rng.integers(250, 256, (z, y, x), dtype=np.uint8)
        elif kind == "const":
            img = np.full((z, y, x), rng.integers(0, 256), np.uint8)
        else:
            img = np.zeros((z, y, x), np.uint8)
        yield img, (lo, hi, mn, mx, True)


def test_normalize_contrast_property_against_real_reference(pins):
    """60 seeded random cases (normalize_contrast_cases): oracle == real reference, bit for bit."""
    for i, (img, args) in enumerate(normalize_contrast_cases()):
        pins.exact(f"normalize_contrast_random/{i}", OP.normalize_contrast(img, *args))
