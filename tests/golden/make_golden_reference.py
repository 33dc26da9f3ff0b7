"""Record what the REAL reference computes on the inputs of the pinning tests (test_oracle_vs_reference.py, the reference
cases of test_operators_oracle.py and the agglomerate plugin signature) into tests/golden/reference_pins.{json,npz}.
Needs the reference tree (see oracle/reference_harness.py for where it is looked for and the I/O modules it stubs):

    python tests/golden/make_golden_reference.py

Each block below is the reference's side of one test; the inputs come from the test module's `*_case(s)` generators.
"""
import ast
import inspect
import io
import os
import re
import sys
import tempfile
import warnings
from contextlib import redirect_stderr, redirect_stdout

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import reference_harness as H  # noqa: E402
from reference_pins import REQUIRED, Pins  # noqa: E402
import test_operators_oracle as TO  # noqa: E402
import test_oracle_vs_reference as T  # noqa: E402
from conftest import MODEL_FILE  # noqa: E402


def quiet():
    return redirect_stdout(io.StringIO())


def signature_table(params):
    return [[name, REQUIRED if default is inspect.Parameter.empty else default] for name, default in params]


def inferencer_pins(pins, Inferencer, Chunk, PatchMask):
    def run(chunk, offset=(0, 0, 0), **kw):
        with quiet():
            with Inferencer(kw.pop("model", None), None, kw.pop("input_patch_size"), **kw) as inf:
                return inf(Chunk(chunk, voxel_offset=offset))

    img, kw = T.non_aligned_case()
    pins.exact("non_aligned/out", run(img, batch_size=5, framework="identity", mask_output_chunk=True, **kw).array)

    with quiet():
        image = Chunk.create(size=(18, 224, 224), dtype="uint8").array
    pins.exact("aligned/in", image)
    r = run(image, offset=(5, 6, 7), input_size=(18, 224, 224), mask_output_chunk=False, framework="identity",
            dtype="float32", **T.ALIGNED_KW)
    pins.value("aligned/offset", tuple(r.voxel_offset))
    pins.exact("aligned/out", r.array)
    r = run(image, input_size=(18, 224, 224), mask_output_chunk=False, framework="identity", augment=True, dtype="float32",
            **T.ALIGNED_KW)
    pins.close("tta_identity/out", r.array)

    r = run(T.network_image(), model=MODEL_FILE, batch_size=1, framework="pytorch", mask_output_chunk=True, **T.NET_KW)
    pins.close("network/out", r.array)
    r = run(T.network_tta_image(), model=MODEL_FILE, batch_size=1, framework="pytorch", mask_output_chunk=True, augment=True,
            **T.NET_KW)
    pins.close("network_tta/out", r.array)

    for ps, ov in T.PATCH_MASK_GEOMETRIES:
        pins.exact(f"patch_mask/{ps}/{ov}", np.asarray(PatchMask(ps, ov)))
    for i, (ps, ov) in enumerate(T.patch_mask_random_cases()):
        pins.exact(f"patch_mask_random/{i}", np.asarray(PatchMask(ps, ov)))

    r = run(T.cropped_image(), offset=(123, 345, 567), num_output_channels=1, framework="identity", batch_size=5,
            mask_output_chunk=False, patch_num=(2, 2, 2), **T.CROPPED_KW)
    pins.value("cropped/offset", tuple(r.voxel_offset))
    pins.exact("cropped/out", r.array)

    for i, (img, off, kw, batch) in enumerate(T.identity_random_cases()):
        r = run(img, offset=off, batch_size=batch, framework="identity", mask_output_chunk=True, **kw)
        pins.exact(f"identity_random/{i}/out", r.array)
        pins.value(f"identity_random/{i}/offset", tuple(r.voxel_offset))
    for i, (img, off, kw, num, c, batch) in enumerate(T.cropped_random_cases()):
        r = run(img, offset=off, num_output_channels=c, framework="identity", batch_size=batch, mask_output_chunk=False,
                patch_num=num, **kw)
        pins.value(f"cropped_random/{i}/offset", tuple(r.voxel_offset))
        pins.exact(f"cropped_random/{i}/out", r.array)
    for i, (img, kw) in enumerate(T.myelin_random_cases()):
        r = run(img, framework="identity", mask_output_chunk=True, batch_size=2, **kw)
        pins.exact(f"myelin_random/{i}/out", r.array)

    sig = [(n, p.default) for n, p in inspect.signature(Inferencer.__init__).parameters.items()]
    pins.value("inferencer/signature", signature_table(sig))
    pins.value("inferencer/attributes", [n for n in ("compute_device", "__enter__", "__exit__", "__call__") if hasattr(Inferencer, n)])


def chunk_pins(pins, Chunk):
    for i, kw in enumerate(T.chunk_create_cases()):
        with quiet():
            want = Chunk.create(**kw)
        pins.exact(f"chunk_create/{i}/array", want.array)
        pins.value(f"chunk_create/{i}/offset_size", [tuple(want.voxel_offset), tuple(want.voxel_size)])
    for i, (base, off, sl, patch, poff, margin, thr) in enumerate(T.chunk_glue_cases()):
        theirs = Chunk(base.copy(), voxel_offset=off)
        b = theirs.cutout(sl)
        pins.exact(f"chunk_glue/{i}/cutout", b.array)
        pins.value(f"chunk_glue/{i}/cutout_offset", tuple(b.voxel_offset))
        theirs.blend(Chunk(patch.copy(), voxel_offset=poff))
        pins.exact(f"chunk_glue/{i}/blend", theirs.array)
        b = theirs.crop_margin(margin)
        pins.exact(f"chunk_glue/{i}/crop", b.array)
        pins.value(f"chunk_glue/{i}/crop_offset", tuple(b.voxel_offset))
        if thr is not None:
            b = Chunk(base.copy(), voxel_offset=off).mask_using_last_channel(threshold=thr)
            pins.exact(f"chunk_glue/{i}/myelin", b.array)
            pins.value(f"chunk_glue/{i}/myelin_offset", tuple(b.voxel_offset))


def plugin_pins(pins):
    from chunkflow.flow.divid_conquer.patch.universal import Universal
    from chunkflow.flow.divid_conquer.transform import TransformSequences
    theirs = TransformSequences()
    for i, (x, outs) in enumerate(T.transform_cases()):
        for k, p in enumerate(theirs.forward(x)):
            pins.exact(f"transform/{i}/forward/{k}", p)
        for k, p in enumerate(theirs.backward([o.copy() for o in outs])):
            pins.exact(f"transform/{i}/backward/{k}", p)
    with tempfile.TemporaryDirectory() as tmp:
        plugin = os.path.join(tmp, "universal_identity.py")
        with open(plugin, "w") as f:
            f.write(T.IDENTITY_PLUGIN)
        for i, (kw, patch, big) in enumerate(T.plugin_cases()):
            u = Universal(plugin, None, **kw)
            pins.value(f"plugin/{i}/attributes", [tuple(np.atleast_1d(getattr(u, n))) for n in T.PLUGIN_ATTRIBUTES])
            pins.exact(f"plugin/{i}/mask", np.asarray(u.output_patch_mask_numpy))
            pins.exact(f"plugin/{i}/call", u(patch.copy()))
            pins.exact(f"plugin/{i}/crop", u._crop_output_patch(big))


def cli_pins(pins):
    """The options of the reference's click commands, read from flow/flow.py as text (importing it needs cloud packages):
    per option [flags, literal default or None, required]."""
    with open(os.path.join(H.REFERENCE_ROOT, "chunkflow", "flow", "flow.py")) as f:
        src = f.read()
    for command in T.CLI_COMMANDS:
        seg = src[src.index(f"@main.command('{command}')"):]
        seg = seg[:seg.index("\ndef ")]
        opts = []
        for m in re.finditer(r"@click\.option\((.*?)\)\s*(?=@click\.option|@operator|@generator|@main|$)", seg, re.S):
            body = m.group(1)
            flags = re.findall(r"'(-{1,2}[A-Za-z][\w/-]*)'", body.split("help=")[0])
            default = re.search(r"default=(\([^)]*\)|[^,\s)]+)", body)
            try:
                value = ast.literal_eval(default.group(1)) if default else None
            except (ValueError, SyntaxError):
                value = None     # an expression such as Cartesian(...): only `inference`'s defaults are compared, all literals
            opts.append([flags, value, "required=True" in body])
        pins.value(f"cli/{command}", opts)


def operator_pins(pins, Chunk):
    from chunkflow.chunk.affinity_map import AffinityMap
    from chunkflow.chunk.image.base import Image
    for seed in (0, 1, 2):
        img, nc_args, aff, mask = TO.real_reference_case(seed)
        im = Image(img.copy())
        with quiet(), redirect_stderr(io.StringIO()):
            im.normalize_contrast(*nc_args)
        pins.exact(f"operators/{seed}/normalize_contrast", np.asarray(im.array))
        for mode in ("xy", "z"):
            pins.exact(f"operators/{seed}/quantize_{mode}", np.asarray(AffinityMap(aff.copy()).quantize(mode).array))
        c = Chunk(aff.copy(), voxel_size=(4, 4, 4))
        Chunk(mask, voxel_size=(8, 16, 8)).maskout(c)
        pins.exact(f"operators/{seed}/maskout", np.asarray(c.array))
        for k, margin in enumerate(TO.MARGINS):
            r = Chunk(aff.copy(), voxel_offset=(3, 2, 1)).crop_margin(margin)
            pins.exact(f"operators/{seed}/crop_margin/{k}", np.asarray(r.array))
            pins.value(f"operators/{seed}/crop_margin/{k}/offset", tuple(r.voxel_offset))
    for i, (img, args) in enumerate(TO.normalize_contrast_cases()):
        im = Image(img.copy())
        with quiet(), redirect_stderr(io.StringIO()):
            im.normalize_contrast(*args)
        pins.exact(f"normalize_contrast_random/{i}", np.asarray(im.array))


def agglomerate_pins(pins):
    with open(os.path.join(H.REFERENCE_ROOT, "chunkflow", "plugins", "agglomerate.py")) as f:
        tree = ast.parse(f.read())     # importing the plugin needs waterz
    fn = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "execute")
    names = [a.arg for a in fn.args.args]
    defaults = [ast.literal_eval(d) for d in fn.args.defaults]
    params = zip(names, [inspect.Parameter.empty] * (len(names) - len(defaults)) + defaults)
    pins.value("agglomerate/execute_signature", signature_table(params))


def main():
    import torch
    torch.cuda.is_available = lambda: False  # the reference moves to CUDA whenever it can (pytorch.py:41-46)
    Inferencer, Chunk, PatchMask = H.import_reference()
    warnings.simplefilter("ignore")
    pins = Pins(record=True)
    inferencer_pins(pins, Inferencer, Chunk, PatchMask)
    chunk_pins(pins, Chunk)
    plugin_pins(pins)
    cli_pins(pins)
    operator_pins(pins, Chunk)
    agglomerate_pins(pins)
    pins.save(torch=torch.__version__, numpy=np.__version__)
    print("reference outputs recorded:", len(pins.meta), "entries")


if __name__ == "__main__":
    main()
