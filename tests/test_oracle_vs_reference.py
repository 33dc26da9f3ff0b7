"""Pins the oracle and the product's host code to the REAL reference classes: each test builds seeded inputs, computes
this project's side and compares it with what the reference computed on the same inputs (recorded under tests/golden/
by tests/golden/make_golden_reference.py, which imports the `*_cases` generators below).
Ports of the reference's own hot-path tests, tests/flow/divid_conquer/test_inferencer.py."""
import numpy as np
import pytest
import torch

from oracle import inferencer_oracle as O

# Identity-backend and host-glue arithmetic is elementwise numpy and reproduces the reference bit for bit anywhere.  The
# network cases run torch-CPU convolutions, whose fp32 sums another CPU or torch build may order differently.
NET_ATOL_SAME_TORCH, NET_ATOL_OTHER_TORCH = 1e-6, 1e-4


@pytest.fixture(scope="module")
def net_atol(pins):
    return NET_ATOL_SAME_TORCH if torch.__version__ == pins.get("_torch") else NET_ATOL_OTHER_TORCH


def non_aligned_case():  # reference test_inferencer.py:141-169 (smaller in z)
    img = np.random.default_rng(1).integers(1, 255, size=(28 + 4 + 6, 192 + 64 + 7, 192 * 2 + 64 + 9), dtype=np.uint8)
    return img, dict(input_patch_size=(32, 256, 256), output_patch_overlap=(4, 64, 64), num_output_channels=2)


def test_non_aligned_input_chunk(pins):
    img, kw = non_aligned_case()
    o, _ = O.infer_chunk(img, framework="identity", **kw)
    pins.exact("non_aligned/out", o)
    np.testing.assert_allclose(img.astype(np.float32) / 255, o[0], rtol=1e-5, atol=1e-5)


ALIGNED_KW = dict(input_patch_size=(10, 128, 128), output_patch_overlap=(2, 32, 32), num_output_channels=3)


def aligned_image():
    """Chunk.create(size=(18, 224, 224), dtype='uint8') -- the 'sin' pattern, equal to the reference's (pinned below)."""
    from chunkflow_b200 import Chunk
    return Chunk.create(size=(18, 224, 224), dtype="uint8").array


def test_aligned_input_size_and_offset(pins):  # reference test_inferencer.py:34-58
    image = aligned_image()
    pins.exact("aligned/in", image)
    o, off = O.infer_chunk(image, (5, 6, 7), framework="identity", mask_output_chunk=False, **ALIGNED_KW)
    assert off == (7, 38, 39)
    pins.value("aligned/offset", off)
    pins.exact("aligned/out", o)


def test_test_time_augmentation(pins):  # reference test_inferencer.py:6-32
    o, _ = O.infer_chunk(aligned_image(), framework="identity", mask_output_chunk=False, augment=True, **ALIGNED_KW)
    pins.close("tta_identity/out", o, atol=1e-7)


NET_KW = dict(input_patch_size=(8, 32, 32), output_patch_overlap=(2, 8, 8), num_output_channels=3)


def network_image():
    return np.random.default_rng(2).integers(0, 256, size=(10, 36, 44), dtype=np.uint8)


def test_network_path_bit_exact(pins, unet_model, net_atol):
    o, _ = O.infer_chunk(network_image(), framework="pytorch", model=unet_model, **NET_KW)
    pins.close("network/out", o, atol=net_atol)


PATCH_MASK_GEOMETRIES = [((10, 128, 128), (2, 32, 32)), ((8, 32, 32), (2, 8, 8))]


def test_myelin_and_patch_mask(pins):
    for ps, ov in PATCH_MASK_GEOMETRIES:
        pins.exact(f"patch_mask/{ps}/{ov}", O.make_patch_mask(ps, ov))


CROPPED_KW = dict(input_patch_size=(10, 40, 40), output_patch_size=(8, 32, 32), output_patch_overlap=(2, 8, 8))


def cropped_image():
    return np.random.default_rng(13).integers(1, 256, size=(2 * 6 + 4, 2 * 24 + 16, 2 * 24 + 16), dtype=np.uint8)


def test_cropped_output_patch_and_crop_margin(pins):
    """SURVEY section 8 f2: output patch smaller than the input patch, explicit crop margin through `patch_num`, a global
    voxel offset, no chunk-wise mask.  (The reference's own test of this configuration is skipped upstream as 'known bug',
    test_inferencer.py:98-139; with mask_output_chunk=True the reference itself produces NaN / asserts.)  The GPU path is
    compared with the oracle on exactly this configuration in tests/test_gpu_parity.py."""
    o, off = O.infer_chunk(cropped_image(), (123, 345, 567), num_output_channels=1, framework="identity",
                           mask_output_chunk=False, **CROPPED_KW)
    pins.value("cropped/offset", off)
    pins.exact("cropped/out", o)


def network_tta_image():
    return np.random.default_rng(3).integers(0, 256, size=(10, 36, 36), dtype=np.uint8)


def test_network_test_time_augmentation_literal(pins, unet_model, net_atol):
    """--augment with a REAL network through the reference: its flips act on the channel / batch axes (transform.py:30-52);
    the oracle's literal mode (what the device path is tested against) reproduces the reference."""
    o, _ = O.infer_chunk(network_tta_image(), framework="pytorch", model=unet_model, augment=True, **NET_KW)
    pins.close("network_tta/out", o, atol=max(net_atol, 1e-7))
    # ... and equals 1/4 (n(x) + rev_c n(x) + T n(T x) + rev_c T n(T x)): symmetric under channel reversal
    np.testing.assert_allclose(o[0], o[2], rtol=0, atol=1e-6)   # up to the order of the 8-term fp32 sum


def patch_mask_random_cases():
    rng = np.random.default_rng(2026)
    for _ in range(60):
        ps = tuple(int(v) for v in rng.integers(2, 40, 3))
        ov = tuple(int(rng.integers(0, p // 2 + 1)) for p in ps)
        yield ps, ov


def test_patch_mask_random_geometries_reference_native_oracle(pins):
    """PatchMask of the REAL reference (patch/patch_mask.py:6-68) == the native library's host code (`cfb_make_patch_mask`)
    == the oracle, bit for bit, on 60 random patch sizes / overlaps (rows a3 / a4)."""
    from chunkflow_b200 import _native
    for i, (ps, ov) in enumerate(patch_mask_random_cases()):
        pins.exact(f"patch_mask_random/{i}", _native.make_patch_mask(ps, ov))
        pins.exact(f"patch_mask_random/{i}", O.make_patch_mask(ps, ov))


def identity_random_cases():
    rng = np.random.default_rng(7)
    for _ in range(12):
        ps = tuple(int(v) for v in rng.integers(4, 13, 3))
        ov = tuple(int(rng.integers(1, p // 2 + 1)) for p in ps)
        size = tuple(int(p + rng.integers(0, 2 * p)) for p in ps)
        img = rng.integers(1, 255, size=size, dtype=np.uint8)
        off = tuple(int(v) for v in rng.integers(-5, 6, 3))
        kw = dict(input_patch_size=ps, output_patch_overlap=ov, num_output_channels=int(rng.integers(1, 4)))
        yield img, off, kw, int(rng.integers(1, 4))


def test_identity_random_geometries_oracle_equals_reference(pins):
    """Whole-operator arithmetic (patch grid with clamped last patches, blend order, chunk mask, normalise) on random small
    chunk / patch / overlap combinations, identity backend: oracle == real reference, bit for bit (rows a1, a2, a5-a7, a11-a13)."""
    for i, (img, off, kw, _batch) in enumerate(identity_random_cases()):
        o, o_off = O.infer_chunk(img, voxel_offset=off, framework="identity", **kw)
        pins.exact(f"identity_random/{i}/out", o)
        pins.value(f"identity_random/{i}/offset", o_off)


def cropped_random_cases():
    rng = np.random.default_rng(31)
    for _ in range(8):
        crop = tuple(int(v) for v in rng.integers(0, 4, 3))
        out_ps = tuple(int(v) for v in rng.integers(4, 11, 3))
        in_ps = tuple(o + 2 * c for o, c in zip(out_ps, crop))
        ov = tuple(int(rng.integers(1, o // 2 + 1)) for o in out_ps)
        num = tuple(int(v) for v in rng.integers(1, 4, 3))
        in_ov = tuple(2 * c + o for c, o in zip(crop, ov))
        size = tuple((p - io) * n + io for p, io, n in zip(in_ps, in_ov, num))       # reference inferencer.py:131-135
        img = rng.integers(1, 256, size=size, dtype=np.uint8)
        off = tuple(int(v) for v in rng.integers(-50, 50, 3))
        kw = dict(input_patch_size=in_ps, output_patch_size=out_ps, output_patch_overlap=ov)
        yield img, off, kw, num, int(rng.integers(1, 3)), int(rng.integers(1, 4))


def test_cropped_output_random_aligned_geometries(pins):
    """Row f2 on random configurations: output patch smaller than the input patch (crop margin per patch), aligned chunk
    built from `patch_num`, no chunk-wise mask, random voxel offset: oracle == real reference, bit for bit."""
    for i, (img, off, kw, _num, c, _batch) in enumerate(cropped_random_cases()):
        o, o_off = O.infer_chunk(img, off, num_output_channels=c, framework="identity", mask_output_chunk=False, **kw)
        pins.value(f"cropped_random/{i}/offset", o_off)
        pins.exact(f"cropped_random/{i}/out", o)


def myelin_random_cases():
    rng = np.random.default_rng(41)
    for k in range(6):
        ps = tuple(int(v) for v in rng.integers(4, 11, 3))
        ov = tuple(int(rng.integers(1, p // 2 + 1)) for p in ps)
        size = tuple(int(p + rng.integers(0, 2 * p)) for p in ps)
        if k % 2:
            img = rng.random(size, dtype=np.float32)
        else:
            img = rng.integers(1, 255, size=size, dtype=np.uint8)
        thr = float(rng.uniform(0.2, 0.8))
        yield img, dict(input_patch_size=ps, output_patch_overlap=ov, num_output_channels=4, mask_myelin_threshold=thr)


def test_myelin_threshold_and_float_input_random(pins):
    """`--mask-myelin-threshold` (inferencer.py:468-477 -> Chunk.mask_using_last_channel, chunk/base.py:685-689) and a float32
    input chunk (no /255), identity backend with 4 output channels, random geometry: oracle == real reference, bit for bit."""
    for i, (img, kw) in enumerate(myelin_random_cases()):
        o, _ = O.infer_chunk(img, framework="identity", **kw)
        assert o.shape == (3,) + img.shape
        pins.exact(f"myelin_random/{i}/out", o)


def chunk_create_cases():
    rng = np.random.default_rng(5)
    for k in range(10):
        size = tuple(int(v) for v in rng.integers(1, 40, 3))
        if k % 3 == 2:
            size = (int(rng.integers(1, 4)),) + size
        for dtype in ("uint8", "float32"):
            for pattern in ("sin", "zero"):
                off = tuple(int(v) for v in rng.integers(-9, 9, 3))
                yield dict(size=size, dtype=np.dtype(dtype), pattern=pattern, voxel_offset=off, voxel_size=(4, 4, 40))


def test_chunk_create_sin_and_zero_match_the_reference(pins):
    """`create-chunk` inputs (chunk/base.py:139-199): pattern 'sin' / 'zero', uint8 and float32, 3-D and 4-D sizes: the product's
    Chunk.create == the real reference's, bit for bit (row a17; 'random' deviates by design: the reference relabels with cc3d)."""
    from chunkflow_b200 import Chunk
    for i, kw in enumerate(chunk_create_cases()):
        got = Chunk.create(**kw)
        pins.exact(f"chunk_create/{i}/array", got.array)
        pins.value(f"chunk_create/{i}/offset_size", [tuple(got.voxel_offset), tuple(got.voxel_size)])


def chunk_glue_cases():
    rng = np.random.default_rng(17)
    for _ in range(25):
        c = int(rng.integers(1, 4))
        size = tuple(int(v) for v in rng.integers(6, 20, 3))
        off = tuple(int(v) for v in rng.integers(-20, 20, 3))
        base = rng.random((c,) + size, dtype=np.float32)
        # cutout of a random inner box, global coordinates
        lo = tuple(int(rng.integers(0, s - 2)) for s in size)
        hi = tuple(int(rng.integers(l + 1, s + 1)) for l, s in zip(lo, size))
        sl = tuple(slice(o + l, o + h) for o, l, h in zip(off, lo, hi))
        # a patch that sticks out of the buffer on some sides
        psz = tuple(int(v) for v in rng.integers(3, 10, 3))
        poff = tuple(int(o + rng.integers(-p + 1, s)) for o, p, s in zip(off, psz, size))
        patch = rng.random((c,) + psz, dtype=np.float32)
        margin = tuple(int(rng.integers(0, (s - 1) // 2)) for s in size)
        thr = float(rng.uniform(0.2, 0.8)) if c > 1 else None
        yield base, off, sl, patch, poff, margin, thr


def test_chunk_glue_cutout_blend_crop_match_the_reference(pins):
    """Row a16: the product's host `Chunk` (cutout in global slices, blend with clipping at the buffer border, crop_margin,
    mask_using_last_channel) against the real reference's `Chunk` on random boxes (chunk/base.py:685-726,761-807)."""
    from chunkflow_b200 import Chunk
    for i, (base, off, sl, patch, poff, margin, thr) in enumerate(chunk_glue_cases()):
        ours = Chunk(base.copy(), voxel_offset=off)
        a = ours.cutout(sl)
        pins.exact(f"chunk_glue/{i}/cutout", a.array)
        pins.value(f"chunk_glue/{i}/cutout_offset", tuple(a.voxel_offset))
        ours.blend(Chunk(patch.copy(), voxel_offset=poff))
        pins.exact(f"chunk_glue/{i}/blend", ours.array)
        a = ours.crop_margin(margin)
        pins.exact(f"chunk_glue/{i}/crop", a.array)
        pins.value(f"chunk_glue/{i}/crop_offset", tuple(a.voxel_offset))
        if thr is not None:
            a = Chunk(base.copy(), voxel_offset=off).mask_using_last_channel(thr)
            pins.exact(f"chunk_glue/{i}/myelin", a.array)
            pins.value(f"chunk_glue/{i}/myelin_offset", tuple(a.voxel_offset))


def transform_cases():
    rng = np.random.default_rng(3)
    for _ in range(6):
        b, c, z, n = (int(v) for v in (rng.integers(1, 4), rng.integers(1, 4), rng.integers(1, 5), rng.integers(2, 9)))
        x = rng.random((b, c, z, n, n), dtype=np.float32)
        outs = [rng.random(x.shape, dtype=np.float32) for _ in range(8)]   # y == x: every transform keeps the shape
        yield x, outs


def test_transform_sequences_literal_mode_matches_the_reference(pins):
    """Row a15, host plug-in path: the product's TransformSequences('reference') == the real reference's
    (flow/divid_conquer/transform.py:114-156) on random 5-D buffers -- every one of the 8 forward copies and 8 backward results."""
    from chunkflow_b200.flow.divid_conquer.transform import TransformSequences
    ours = TransformSequences('reference')
    for i, (x, outs) in enumerate(transform_cases()):
        fo = ours.forward(x)
        assert len(fo) == 8
        for k, p in enumerate(fo):
            pins.exact(f"transform/{i}/forward/{k}", p)
        for k, p in enumerate(ours.backward([o.copy() for o in outs])):
            pins.exact(f"transform/{i}/backward/{k}", p)


# A `-f universal` plugin file (the contract of the reference's examples/inference/universal_identity.py): the input patch,
# as float32, times the output patch mask.
IDENTITY_PLUGIN = """import numpy as np


class PatchInferencer:
    def __init__(self, model_weight_file, output_patch_mask):
        self.output_patch_mask = output_patch_mask

    @property
    def compute_device(self):
        return "cpu"

    def __call__(self, input_patch):
        return input_patch.astype(np.float32) * self.output_patch_mask
"""
PLUGIN_ATTRIBUTES = ("input_patch_size", "output_patch_size", "output_patch_overlap", "num_output_channels", "crop_margin",
                     "input_patch_overlap", "input_patch_stride", "output_patch_stride")


def plugin_cases():
    rng = np.random.default_rng(23)
    for _ in range(5):
        out_ps = tuple(int(v) for v in rng.integers(4, 12, 3))
        crop = tuple(int(v) for v in rng.integers(0, 3, 3))
        in_ps = tuple(o + 2 * c for o, c in zip(out_ps, crop))
        ov = tuple(int(rng.integers(1, o // 2 + 1)) for o in out_ps)
        kw = dict(input_patch_size=in_ps, output_patch_size=out_ps, output_patch_overlap=ov, num_output_channels=1)
        # the plugin multiplies by the OUTPUT patch mask: feed it a patch of the output size, like the reference's own test does
        patch = rng.random((2, 1) + out_ps, dtype=np.float32)
        big = rng.random((1, 3) + in_ps, dtype=np.float32)
        yield kw, patch, big


def test_plugin_surface_matches_the_reference(pins, tmp_path):
    """Rows a8 / a10 / B3: the plugin base class carries the attributes the reference's Inferencer reads, with the same values,
    and `Universal` drives a plugin file of the reference's example contract to the same per-patch result as the reference's
    Universal."""
    from chunkflow_b200.flow.divid_conquer.patch.universal import Universal
    plugin = tmp_path / "universal_identity.py"
    plugin.write_text(IDENTITY_PLUGIN)
    for i, (kw, patch, big) in enumerate(plugin_cases()):
        ours = Universal(str(plugin), None, **kw)
        pins.value(f"plugin/{i}/attributes", [tuple(np.atleast_1d(getattr(ours, n))) for n in PLUGIN_ATTRIBUTES])
        pins.exact(f"plugin/{i}/mask", np.asarray(ours.output_patch_mask_numpy))
        pins.exact(f"plugin/{i}/call", ours(patch.copy()))
        pins.exact(f"plugin/{i}/crop", ours._crop_output_patch(big))


CLI_COMMANDS = ("inference", "create-chunk", "connected-components", "normalize-contrast", "crop-margin", "quantize")


def test_cli_inference_options_match_the_reference_source(pins):
    """Boundary B1: every option of the reference's `inference` command (flow/flow.py:1850-1893, read as text by the
    golden generator: importing that module needs cloud packages) exists here with the same flags, the same default and
    the same `required` -- plus the extra `b200` framework choice.  Also the flag names of the neighbouring commands."""
    from chunkflow_b200.flow import cli

    def ours(command):
        table = {}
        for p in command.params:
            for o in p.opts + p.secondary_opts:
                table[o] = p
        return table

    mine = ours(cli.inference)
    ref_opts = pins.get("cli/inference")
    assert len(ref_opts) == 19
    for flags, default, required in ref_opts:
        for f in flags:
            for part in f.split("/"):
                assert part in mine, part
        p = mine[flags[0].split("/")[0]]
        got = p.default
        if isinstance(default, list):      # a tuple default (JSON keeps it as a list)
            default, got = tuple(default), tuple(got)
        assert got == default or (default is None and got in (None, ())), (flags, default, p.default)
        assert bool(p.required) == required, flags
    assert set(mine["--framework"].type.choices) == {"universal", "identity", "pytorch", "b200"}
    for command, obj in (("create-chunk", cli.create_chunk), ("connected-components", cli.connected_components),
                         ("normalize-contrast", cli.normalize_contrast), ("crop-margin", cli.crop_margin), ("quantize", cli.quantize)):
        have = ours(obj)
        for flags, _, _ in pins.get(f"cli/{command}"):
            for f in flags:
                if f == "--crop-bbox/--no-crop-bbox":   # crop-margin's bounding-box bookkeeping belongs to the storage operators
                    continue
                for part in f.split("/"):
                    assert part in have, (command, part)


def test_inferencer_constructor_signature_matches_the_reference(pins):
    """Boundary B2: the constructor keywords of the reference's Inferencer (inferencer.py:36-54), in order, with the same
    defaults; the product appends `device` and `precision`.  Both have compute_device, __enter__, __exit__ and __call__."""
    import inspect
    from chunkflow_b200 import Inferencer as Ours
    from reference_pins import REQUIRED, plain
    theirs = pins.get("inferencer/signature")
    mine = plain([[n, REQUIRED if p.default is inspect.Parameter.empty else p.default]
                  for n, p in inspect.signature(Ours.__init__).parameters.items()])
    assert [n for n, _ in mine[:len(theirs)]] == [n for n, _ in theirs]
    for (n, d_mine), (_, d_ref) in zip(mine, theirs):
        assert d_mine == d_ref, (n, d_mine, d_ref)
    assert [n for n, _ in mine[len(theirs):]] == ["device", "precision"]
    for name in ("compute_device", "__enter__", "__exit__", "__call__"):
        assert hasattr(Ours, name)
    assert pins.get("inferencer/attributes") == ["compute_device", "__enter__", "__exit__", "__call__"]
