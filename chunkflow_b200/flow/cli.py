"""``chunkflow``-style command line for the inference hot path.

Chained multi-command group with lazily pulled operator generators, like the reference
(chunkflow/lib/flow.py:44-105).  The two commands on the hot path, plus the operators either side of it on the GPU
(`normalize-contrast`, `crop-margin`, `quantize`; `to-device` / `to-host` keep the chunk in GPU memory in between):

    python -m chunkflow_b200.flow.cli create-chunk --size 64 256 256 \
        inference --input-patch-size 20 256 256 --output-patch-overlap 4 64 64 \
                  --num-output-channels 3 --framework b200 --batch-size 12 --mask-output-chunk

``inference`` keeps every flag of the reference operator (chunkflow/flow/flow.py:1853-1893) and adds
the ``b200`` framework choice; ``-f pytorch`` is accepted for the canonical model file.
"""
from functools import update_wrapper
from time import time

import click
import numpy as np

from chunkflow_b200.chunk import Chunk

state = {"dry_run": False, "verbose": 1}


def default_none(ctx, _, value):
    """click turns a missing nargs=3 option into an empty tuple; the operators expect None."""
    return None if value is None or len(value) == 0 else value


@click.group(chain=True)
@click.option("--mip", type=click.INT, default=0, help="default mip level of chunks.")
@click.option("--dry-run/--real-run", default=False, help="dry run or real run.")
@click.option("--verbose/--quiet", default=True, help="print informations or not.")
def main(mip, dry_run, verbose):
    """Compose operators and create your own pipeline (inference hot path only)."""
    state["mip"] = mip
    state["dry_run"] = dry_run
    state["verbose"] = verbose


@main.result_callback()
def process_commands(operators, mip, dry_run, verbose):
    stream = [{"log": {"timer": {}}}]
    for op in operators:
        stream = op(stream)
    tasks = []
    for task in stream:   # pull-driven execution
        tasks.append(task)
    return tasks


def operator(func):
    """Wrap a command so that it returns a closure over the task stream (reference lib/flow.py:82-93)."""
    def new_func(*args, **kwargs):
        def op(stream):
            return func(stream, *args, **kwargs)
        return op
    return update_wrapper(new_func, func)


@main.command("create-chunk")
@click.option("--name", type=str, default="create-chunk", help="name of operator")
@click.option("--size", "-s", type=click.INT, nargs=3, default=(64, 64, 64), help="the size of created chunk")
@click.option("--dtype", "-d", type=click.Choice(["uint8", "float32", "float64"]), default="uint8",
              help="the data type of chunk (the reference's integer label types need cc3d and are not part of this path)")
@click.option("--pattern", "-p", type=click.Choice(["sin", "random", "zero"]), default="sin")
@click.option("--voxel-offset", "-t", type=click.INT, nargs=3, default=(0, 0, 0), help="offset in voxel number.")
@click.option("--voxel-size", "-e", type=click.INT, nargs=3, default=(1, 1, 1), help="voxel size in nm")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="name of created chunk")
@operator
def create_chunk(tasks, name, size, dtype, pattern, voxel_offset, voxel_size, output_chunk_name):
    """Create a fake chunk for easy test (reference flow/flow.py:652-678)."""
    for task in tasks:
        task[output_chunk_name] = Chunk.create(size=size, dtype=np.dtype(dtype), pattern=pattern,
                                               voxel_offset=voxel_offset, voxel_size=voxel_size)
        yield task


@main.command("inference")
@click.option("--name", type=str, default="inference", help="name of this operator")
@click.option("--convnet-model", "-m", type=str, default=None, help="convnet model path or type.")
@click.option("--convnet-weight-path", "-w", type=str, default=None, help="convnet weight path")
@click.option("--input-patch-size", "-s", type=click.INT, nargs=3, required=True, help="input patch size")
@click.option("--output-patch-size", "-z", type=click.INT, nargs=3, default=None, callback=default_none,
              help="output patch size")
@click.option("--output-patch-overlap", "-v", type=click.INT, nargs=3, default=(4, 64, 64), help="patch overlap")
@click.option("--output-crop-margin", type=click.INT, nargs=3, default=None, callback=default_none,
              help="margin size of output chunk cropping.")
@click.option("--patch-num", "-n", default=None, callback=default_none, type=click.INT, nargs=3,
              help="patch number in z,y,x.")
@click.option("--num-input-channels", type=click.INT, default=1, help="number of input channels")
@click.option("--num-output-channels", "-c", type=click.INT, default=3, help="number of output channels")
@click.option("--dtype", "-d", type=click.Choice(["float32", "float16"]), default="float32",
              help="float32: fp16 hi/lo split tensor-core arithmetic with fp32 accumulation (1e-3 parity mode); "
                   "float16: single-pass fp16 tensor cores. The result is float32 either way.")
@click.option("--framework", "-f", type=click.Choice(["universal", "identity", "pytorch", "b200"]), default="universal",
              help="inference framework")
@click.option("--batch-size", "-b", type=click.INT, default=1, help="mini batch size of input patch.")
@click.option("--bump", type=click.Choice(["wu", "zung"]), default="wu", help="bump function type (only support wu now!).")
@click.option("--mask-output-chunk/--no-mask-output-chunk", default=False,
              help="mask output chunk will make the whole chunk like one output patch. "
                   "This will also work with non-aligned chunk size.")
@click.option("--mask-myelin-threshold", "-y", default=None, type=click.FLOAT,
              help="mask myelin if netoutput have myelin channel.")
@click.option("--augment/--no-augment", default=False,
              help="transform the input patch and transform back the output patch")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@operator
def inference(tasks, name, convnet_model, convnet_weight_path, input_patch_size, output_patch_size,
              output_patch_overlap, output_crop_margin, patch_num, num_input_channels, num_output_channels, dtype,
              framework, batch_size, bump, mask_output_chunk, mask_myelin_threshold, augment, input_chunk_name,
              output_chunk_name):
    """Perform convolutional network inference for chunks (reference flow/flow.py:1894-1933)."""
    from chunkflow_b200.flow.divid_conquer.inferencer import Inferencer
    with Inferencer(
            convnet_model, convnet_weight_path,
            input_patch_size=input_patch_size, output_patch_size=output_patch_size,
            num_input_channels=num_input_channels, num_output_channels=num_output_channels,
            output_patch_overlap=output_patch_overlap, output_crop_margin=output_crop_margin,
            patch_num=patch_num, framework=framework, dtype=dtype, batch_size=batch_size, bump=bump,
            augment=augment, mask_output_chunk=mask_output_chunk, mask_myelin_threshold=mask_myelin_threshold,
            dry_run=state["dry_run"]) as inferencer:
        for task in tasks:
            if task is not None:
                if "log" not in task:
                    task["log"] = {"timer": {}}
                start = time()
                chunk_in = task[input_chunk_name]
                if isinstance(chunk_in, Chunk) or inferencer.patch_inferencer is not None or state["dry_run"]:
                    task[output_chunk_name] = inferencer(_to_host(chunk_in))
                else:  # a DeviceChunk (see `to-device`): the result stays in GPU memory too
                    task[output_chunk_name] = inferencer.infer_device(chunk_in)
                task["log"]["timer"][name] = time() - start
                task["log"]["compute_device"] = inferencer.compute_device
                if state["verbose"]:
                    out = task[output_chunk_name]
                    print(f"{name}: {out.shape} in {task['log']['timer'][name]:.3f} s on "
                          f"{task['log']['compute_device']} ({np.prod(out.shape[-3:]) / task['log']['timer'][name] / 1e6:.1f} Mvoxels/s)")
            yield task


# ---------------------------------------------------------------------------------------------
# operators either side of `inference`, on the GPU (SURVEY.md section 8 f3).  A task's chunk is either a host
# `Chunk` (moved to the GPU for the kernel and back, like `inference` does) or -- after `to-device` -- a `DeviceChunk`
# that stays in GPU memory from operator to operator until `to-host`.
# ---------------------------------------------------------------------------------------------
def _to_host(chunk):
    return chunk if isinstance(chunk, Chunk) else chunk.to_chunk()


def _on_device(chunk, device):
    """(DeviceChunk, was_host)"""
    from chunkflow_b200.chunk.device import DeviceChunk
    if isinstance(chunk, DeviceChunk):
        return chunk, False
    return DeviceChunk.from_chunk(chunk, device=device), True


@main.command("to-device")
@click.option("--device", type=str, default="cuda:0", help="GPU that will hold the chunk between operators.")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@operator
def to_device(tasks, device, input_chunk_name, output_chunk_name):
    """(extension) Move the chunk to GPU memory; the following operators run on it there."""
    for task in tasks:
        if task is not None:
            task[output_chunk_name] = _on_device(task[input_chunk_name], device)[0]
        yield task


@main.command("to-host")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@operator
def to_host(tasks, input_chunk_name, output_chunk_name):
    """(extension) Bring a GPU-resident chunk back to host memory."""
    for task in tasks:
        if task is not None:
            task[output_chunk_name] = _to_host(task[input_chunk_name])
        yield task


@main.command("normalize-contrast")
@click.option("--name", type=str, default="normalize-contrast-nkem", help="name of operator.")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@click.option("--lower-clip-fraction", "-l", type=click.FLOAT, default=0.01, help="lower intensity fraction to clip out.")
@click.option("--upper-clip-fraction", "-u", type=click.FLOAT, default=0.01, help="upper intensity fraction to clip out.")
@click.option("--minval", type=click.INT, default=1, help="the minimum intensity of transformed chunk.")
@click.option("--maxval", type=click.INT, default=255, help="the maximum intensity of transformed chunk.")
@click.option("--per-section/--whole", default=True, help="per section normalization or normalize the whole chunk.")
@operator
def normalize_contrast(tasks, name, input_chunk_name, output_chunk_name, lower_clip_fraction, upper_clip_fraction, minval,
                       maxval, per_section):
    """Normalize the section contrast (reference flow/flow.py:1672-1711, chunk/image/base.py:93-132)."""
    import torch
    from chunkflow_b200.chunk.device import DeviceChunk
    for task in tasks:
        if task is not None:
            start = time()
            dev, was_host = _on_device(task[input_chunk_name], "cuda:0")
            if not was_host:  # the reference works on a clone (flow.py:1699)
                dev = DeviceChunk(dev.tensor.clone(), voxel_offset=dev.voxel_offset, voxel_size=dev.voxel_size)
            dev.normalize_contrast(lower_clip_fraction=lower_clip_fraction, upper_clip_fraction=upper_clip_fraction,
                                   minval=minval, maxval=maxval, per_section=per_section)
            torch.cuda.synchronize(dev.tensor.device)
            task[output_chunk_name] = dev.to_chunk() if was_host else dev
            task["log"]["timer"][name] = time() - start
        yield task


@main.command("crop-margin")
@click.option("--name", type=str, default="crop-margin", help="name of this operator")
@click.option("--margin-size", "-m", type=click.INT, nargs=6, default=None, callback=default_none,
              help="crop the chunk margin: -z -y -x +z +y +x.")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name.")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name.")
@operator
def crop_margin(tasks, name, margin_size, input_chunk_name, output_chunk_name):
    """Crop the margin of chunk (reference flow/flow.py:2053-2084; the bounding-box form needs a task bbox and is not
    part of this path)."""
    import torch
    if not margin_size:
        raise click.UsageError("crop-margin: --margin-size is required here (no task bounding boxes on this path)")
    for task in tasks:
        if task is not None:
            start = time()
            dev, was_host = _on_device(task[input_chunk_name], "cuda:0")
            out = dev.crop_margin(margin_size)
            torch.cuda.synchronize(out.tensor.device)
            task[output_chunk_name] = out.to_chunk() if was_host else out
            task["log"]["timer"][name] = time() - start
        yield task


@main.command("quantize")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@click.option("--mode", type=click.Choice(["xy", "z"]), default="xy", help="xy: average of xy channel; z: only the z channel")
@operator
def quantize(tasks, input_chunk_name, output_chunk_name, mode):
    """Transform an affinity map to a uint8 image (reference flow/flow.py:2250-2273, chunk/affinity_map/base.py:33-57)."""
    import torch
    for task in tasks:
        if task is not None:
            dev, was_host = _on_device(task[input_chunk_name], "cuda:0")
            out = dev.quantize(mode=mode)
            torch.cuda.synchronize(out.tensor.device)
            task[output_chunk_name] = out.to_chunk() if was_host else out
        yield task


@main.command("connected-components")
@click.option("--name", type=str, default="connected-components", help="threshold a map and get the targets.")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name")
@click.option("--threshold", "-t", type=click.FLOAT, default=None, help="threshold to cut the map.")
@click.option("--connectivity", "-c", type=click.Choice(["6", "18", "26"]), default="6",
              help="number of neighboring voxels used. Default is 6.")
@operator
def connected_components(tasks, name, input_chunk_name, output_chunk_name, threshold, connectivity):
    """Threshold the probability map to get a segmentation (reference flow/flow.py:1803-1830, chunk/base.py:128-137)."""
    import torch
    connectivity = int(connectivity)
    for task in tasks:
        if task is not None:
            start = time()
            dev, was_host = _on_device(task[input_chunk_name], "cuda:0")
            out = dev.connected_component(threshold=threshold, connectivity=connectivity)
            torch.cuda.synchronize(out.tensor.device)
            task[output_chunk_name] = out.to_chunk() if was_host else out
            task["log"]["timer"][name] = time() - start
        yield task


@main.command("agglomerate")
@click.option("--name", type=str, default="agglomerate", help="name of this operator")
@click.option("--input-chunk-name", "-i", type=str, default="chunk", help="input chunk name (the affinity map)")
@click.option("--output-chunk-name", "-o", type=str, default="chunk", help="output chunk name (the segmentation)")
@click.option("--threshold", "-t", type=click.FLOAT, default=0.7, help="merge until the score 1 - mean affinity reaches this.")
@click.option("--aff-threshold-low", type=click.FLOAT, default=0.001, help="watershed: affinities up to this are no edges.")
@click.option("--aff-threshold-high", type=click.FLOAT, default=0.9999, help="watershed: affinities from this on always connect.")
@click.option("--flip-channel/--no-flip-channel", default=True,
              help="the channels are stored x, y, z (chunkflow) and read in reverse (waterz wants z, y, x).")
@operator
def agglomerate(tasks, name, input_chunk_name, output_chunk_name, threshold, aff_threshold_low, aff_threshold_high, flip_channel):
    """Watershed + mean-affinity agglomeration of an affinity map (the reference runs this as `plugin -f agglomerate`:
    plugins/agglomerate.py:8-48 -> waterz.agglomerate; README.md:39)."""
    import torch
    for task in tasks:
        if task is not None:
            start = time()
            dev, was_host = _on_device(task[input_chunk_name], "cuda:0")
            out = dev.agglomerate(threshold=threshold, aff_threshold_low=aff_threshold_low, aff_threshold_high=aff_threshold_high,
                                  flip_channel=flip_channel)
            torch.cuda.synchronize(out.tensor.device)
            task[output_chunk_name] = out.to_chunk() if was_host else out
            task["log"]["timer"][name] = time() - start
        yield task


@main.command("load-npy")
@click.option("--file-name", "-f", type=click.Path(exists=True, file_okay=True, dir_okay=False, readable=True, resolve_path=True),
              required=True, help="file name path")
@click.option("--voxel-offset", "-t", type=int, nargs=3, default=(0, 0, 0), help="voxel offset")
@click.option("--voxel-size", "-s", type=click.FLOAT, nargs=3, default=(1, 1, 1), help="voxel size")
@click.option("--output-name", "-o", type=str, default="chunk", help="output name in the task dictionary.")
@operator
def load_npy(tasks, file_name, voxel_offset, voxel_size, output_name):
    """Load a chunk from a .npy file (reference flow/flow.py:1321-1341), e.g. a ground truth for `evaluate-segmentation`."""
    for task in tasks:
        if task is not None:
            if not file_name.endswith(".npy"):
                raise click.BadParameter(f"{file_name} is not a .npy file", param_hint="--file-name")
            task[output_name] = Chunk(np.load(file_name), voxel_offset=voxel_offset, voxel_size=voxel_size)
        yield task


@main.command("evaluate-segmentation")
@click.option("--segmentation-chunk-name", "-s", type=str, default="chunk", help="chunk name of segmentation")
@click.option("--groundtruth-chunk-name", "-g", type=str, default="groundtruth")
@click.option("--output", "-o", type=str, default="seg_score", help="segmentation evaluation result name.")
@operator
def evaluate_segmentation(tasks, segmentation_chunk_name, groundtruth_chunk_name, output):
    """Score a segmentation against a ground truth: Rand index, adjusted Rand index, variation of information,
    Fowlkes-Mallows index, edit distance (reference flow/flow.py:1519-1542, chunk/segmentation.py:33-67).  Either chunk may
    be on the host or, after `to-device`, on the GPU; the contingency table is built on the GPU either way."""
    from chunkflow_b200.chunk.device import DeviceChunk
    from chunkflow_b200.chunk.segmentation import Segmentation, format_scores
    for task in tasks:
        if task is not None:
            seg, gt = task[segmentation_chunk_name], task[groundtruth_chunk_name]
            if isinstance(seg, Chunk) and isinstance(gt, Chunk):
                task[output] = Segmentation(seg.array, voxel_offset=seg.voxel_offset).evaluate(gt)
            else:
                dev = seg if isinstance(seg, DeviceChunk) else gt
                seg, gt = (c if isinstance(c, DeviceChunk) else _device_labels(c, dev.tensor.device) for c in (seg, gt))
                task[output] = seg.evaluate(gt)
                print(format_scores(task[output]), end="")
        yield task


def _device_labels(chunk, device):
    from chunkflow_b200.chunk.device import DeviceChunk
    from chunkflow_b200.chunk.segmentation import label_array
    return DeviceChunk.from_labels(label_array(chunk.array, "a label chunk"), device=device)


if __name__ == "__main__":
    main()
