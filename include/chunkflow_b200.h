/*
 * chunkflow_b200 -- C-ABI of the B200-native `inference` hot path.
 *
 * Drop-in boundary for chunkflow's overlap-tile convnet inference.  The reference is
 * pure Python; each entry point names the reference interface it replaces
 * (paths relative to the reference tree, v1.1.7):
 *
 *   cfb_create / cfb_destroy      Inferencer.__init__ / __exit__
 *                                 chunkflow/flow/divid_conquer/inferencer.py:36-171,177-181
 *   cfb_set_weight / cfb_commit_weights
 *                                 PyTorch.__init__ weight loading
 *                                 chunkflow/flow/divid_conquer/patch/pytorch.py:48-63
 *   cfb_patch_mask                PatchMask / make_patch_mask
 *                                 chunkflow/flow/divid_conquer/patch/patch_mask.py:6-48
 *   cfb_patch_grid                Inferencer._construct_patch_slices_list   inferencer.py:255-292
 *   cfb_output_shape              Inferencer._update_parameters_for_input_chunk   inferencer.py:183-204
 *   cfb_infer_chunk_device/_host  Inferencer.__call__   inferencer.py:360-479
 *                                 (Chunk.cutout chunk/base.py:761-781, Chunk.blend chunk/base.py:792-807,
 *                                  PyTorch.__call__ patch/pytorch.py:98-119)
 *   cfb_patch_forward_host        PatchInferencer.__call__ plugin level
 *                                 patch/pytorch.py:98-119, patch/universal.py:60-69, patch/identity.py:30-51
 *   cfb_device_name               Inferencer.compute_device   inferencer.py:173-175
 *   cfb_watershed_device, cfb_region_graph_*, cfb_agglomerate_edges_host, cfb_relabel_device
 *                                 plugins/agglomerate.py:8-48 (execute -> waterz.agglomerate)
 *
 * Plain pointers and sizes only -- no torch types.  Device pointers are raw CUDA device
 * addresses (e.g. torch.Tensor.data_ptr()) owned by the caller.  All functions return
 * CFB_OK (0) or a negative error code; cfb_last_error() returns the message of the last
 * failure on the calling thread.  There is NO CPU fallback: without a CUDA device every
 * compute entry point fails with CFB_ERR_CUDA.
 */
#ifndef CHUNKFLOW_B200_H_
#define CHUNKFLOW_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFB_OK 0
#define CFB_ERR_INVALID_ARGUMENT (-1)
#define CFB_ERR_CUDA (-2)
#define CFB_ERR_WEIGHTS (-3)
#define CFB_ERR_OUTPUT_RANGE (-4) /* some output >= 1.0001 (reference inferencer.py:465-466) */
#define CFB_ERR_UNSUPPORTED (-5)
#define CFB_ERR_CAPACITY (-6) /* a caller-sized table is too small: call again with a larger one */

/* framework: which patch backend runs on the device */
#define CFB_FRAMEWORK_UNET3L 0   /* fixed 3-level 3D U-Net (chunkflow_b200/convnet/unet3l.py) */
#define CFB_FRAMEWORK_IDENTITY 1 /* reference patch/identity.py: output = input patch */

/* precision of the convolution stack */
#define CFB_PRECISION_F32_SIMT 0   /* fp32 FFMA direct convolution (exact-order-free fp32) */
#define CFB_PRECISION_F16X3_UMMA 1 /* tcgen05 fp16 hi/lo split, fp32 accumulate (~fp32 accuracy) */
#define CFB_PRECISION_F16_UMMA 2   /* tcgen05 single-pass fp16, fp32 accumulate (reference --dtype float16) */
#define CFB_PRECISION_F16F8_UMMA 3 /* tcgen05 fp16 main product + ONE e4m3 (K = 32) product carrying both correction terms,
                                      fp32 accumulate: two tensor-core products per multiply instead of f16x3's three
                                      (csrc/act_format.cuh) */

/* test-time augmentation (`--augment`, reference inferencer.py:422-431 + transform.py).
 * REFERENCE reproduces the reference's arithmetic literally: its FlipLR / FlipUD call np.fliplr / np.flipud on
 * arr[..., z, :, :] of the 5-D (B, C, z, y, x) buffers, i.e. they reverse the CHANNEL and BATCH axes
 * (transform.py:30-52), so the average over its 8 sequences is
 *   1/4 * (n(x) + rev_c n(x) + T n(T x) + rev_c T n(T x)),   T = transpose y<->x, rev_c = output channels reversed.
 * SPATIAL is the evidently intended augmentation: the 8 combinations of {transpose} x {flip x} x {flip y}, each
 * undone on the output, averaged (an explicit opt-in; it does NOT reproduce the reference's numbers). */
#define CFB_AUGMENT_NONE 0
#define CFB_AUGMENT_REFERENCE 1
#define CFB_AUGMENT_SPATIAL 2

/* dtype of the input chunk */
#define CFB_DTYPE_U8 0
#define CFB_DTYPE_F32 1
#define CFB_DTYPE_U32 2 /* connected components on an integer segmentation */
#define CFB_DTYPE_U64 3 /* label volumes of evaluate-segmentation */

typedef struct cfb_engine* cfb_handle;

typedef struct cfb_params {
  int32_t struct_size;             /* = sizeof(cfb_params), for ABI checks */
  int32_t device;                  /* CUDA device ordinal */
  int32_t framework;               /* CFB_FRAMEWORK_* */
  int32_t precision;               /* CFB_PRECISION_* */
  int32_t input_patch_size[3];     /* z, y, x */
  int32_t output_patch_size[3];    /* z, y, x (<= input; crop margin = (in-out)/2) */
  int32_t output_patch_overlap[3]; /* z, y, x */
  int32_t output_crop_margin[3];   /* z, y, x: margin of the output chunk that is dropped */
  int32_t num_input_channels;      /* must be 1 */
  int32_t num_output_channels;     /* channels returned (network may produce more; first N kept) */
  int32_t batch_size;              /* patches in flight per launch (scheduling hint) */
  int32_t mask_output_chunk;       /* 1: normalise by the accumulated weight volume */
  int32_t augment;                 /* CFB_AUGMENT_*: test-time augmentation (reference transform.py:114-156) */
  int32_t has_myelin_threshold;    /* 1: drop last channel, zero where it is >= threshold */
  float mask_myelin_threshold;
  int32_t check_output_range;      /* 1: fail with CFB_ERR_OUTPUT_RANGE like the reference assert */
} cfb_params;

const char* cfb_last_error(void);
int cfb_version(void);
/* Number of CUDA devices visible (0 if none / no driver). Never fails. */
int cfb_device_count(void);

/* Free / total bytes of device memory (used to size the number of patches in flight). */
int cfb_device_memory(int32_t device, int64_t* free_bytes, int64_t* total_bytes);

int cfb_create(const cfb_params* params, cfb_handle* out);
int cfb_destroy(cfb_handle h);
/* Name of the CUDA device the engine runs on (valid until cfb_destroy). */
const char* cfb_device_name(cfb_handle h);

/* Weights: fp32 host arrays in PyTorch state_dict layout, keyed by state_dict name
 * ("enc0.0.weight", "enc0.0.bias", ... "head.bias"). commit packs them for the kernels. */
int cfb_set_weight(cfb_handle h, const char* name, const float* host_data, int64_t numel);
int cfb_commit_weights(cfb_handle h);

/* Device-free: fp32 patch mask for (patch z,y,x ; overlap z,y,x) into host memory
 * (prod(patch) floats).  Replaces make_patch_mask, patch/patch_mask.py:15-48. */
int cfb_make_patch_mask(const int32_t patch_size[3], const int32_t overlap[3], float* host_out);

/* Copies the fp32 patch mask (prod(output_patch_size) floats) to host memory. */
int cfb_patch_mask(cfb_handle h, float* host_out);

/* Patch grid for a chunk of the given size: writes the number of patches and, if
 * starts_zyx != NULL, up to `capacity` chunk-local input start triples (z,y,x per patch,
 * z-major then y then x, last patch per axis clamped). */
int cfb_patch_grid(cfb_handle h, int64_t cz, int64_t cy, int64_t cx,
                   int64_t* num_patches, int32_t* starts_zyx, int64_t capacity);

/* Output chunk shape (C, z, y, x) for an input chunk (z, y, x). */
int cfb_output_shape(cfb_handle h, int64_t cz, int64_t cy, int64_t cx, int64_t out_czyx[4]);

/* Whole-chunk inference, input and output resident in device memory.
 * d_in : (cz,cy,cx) uint8 or float32, contiguous; d_out: (C,oz,oy,ox) float32.
 * `stream` is a cudaStream_t (NULL = default stream).  Asynchronous unless
 * check_output_range is set (the range check synchronises the stream). */
int cfb_infer_chunk_device(cfb_handle h, const void* d_in, int32_t in_dtype,
                           int64_t cz, int64_t cy, int64_t cx, float* d_out, void* stream);

/* Same, host buffers: H2D copy of the chunk, inference, D2H copy of the result. */
int cfb_infer_chunk_host(cfb_handle h, const void* h_in, int32_t in_dtype,
                         int64_t cz, int64_t cy, int64_t cx, float* h_out);

/* One oversized chunk split across GPUs (BASELINE config #5; the reference has no counterpart, its unit of
 * parallelism is one process per GPU on independent chunks, distributed/kubernetes/deploy.yml:37):
 *   cfb_infer_slab_device     processes only the patches whose z-row index is in [zrow_begin, zrow_end) and leaves
 *                             d_out as the UN-normalised partial sum; d_weight (oz,oy,ox), if not NULL, receives this
 *                             slab's partial weight sum.
 *   cfb_slab_nonzero          the any-nonzero flag of the input of the last slab / chunk call (all ranks OR it to
 *                             reproduce the reference's all-zero shortcut, inferencer.py:387-393); synchronises.
 *   cfb_halo_add_device       d_dst[i] += d_src[i]: the owner of a plane adds the partial sums received from the
 *                             other ranks whose slabs overlap it (NCCL send/recv of the planes, then this kernel).
 *   cfb_weight_volume_device  planes [z_begin, z_end) of the weight volume (sum of the bump masks of ALL patches of
 *                             a (cz,cy,cx) chunk, reference inferencer.py:294-333; 1/W if `invert`): pure geometry,
 *                             so the owner computes it locally -- no weight halo is exchanged.
 *   cfb_normalize_device      d_out *= 1/d_weight (or *= d_weight if weight_is_inverse; NULL = no weight), the
 *                             reference's `< 1.0001` assertion (CFB_ERR_OUTPUT_RANGE, when check_output_range is set),
 *                             myelin masking; all_zero_input != 0 forces the result to zero. */
int cfb_infer_slab_device(cfb_handle h, const void* d_in, int32_t in_dtype,
                          int64_t cz, int64_t cy, int64_t cx,
                          int64_t zrow_begin, int64_t zrow_end,
                          float* d_out, float* d_weight, void* stream);
int cfb_slab_nonzero(cfb_handle h, int32_t* nonzero, void* stream);
int cfb_halo_add_device(float* d_dst, const float* d_src, int64_t count, void* stream);
int cfb_weight_volume_device(cfb_handle h, int64_t cz, int64_t cy, int64_t cx, int64_t z_begin, int64_t z_end,
                             int32_t invert, float* d_weight, void* stream);
int cfb_normalize_device(cfb_handle h, float* d_out, const float* d_weight, int32_t weight_is_inverse,
                         int64_t channels, int64_t oz, int64_t oy, int64_t ox, int32_t all_zero_input, void* stream);

/* PatchInferencer plugin level: `batch` input patches (batch,1,pz,py,px) float32 in
 * [0,1] on the host -> (batch,C,oz,oy,ox) float32 on the host, already cropped and
 * multiplied by the patch mask (reference patch/pytorch.py:112-113). */
int cfb_patch_forward_host(cfb_handle h, const float* h_patches, int32_t batch, float* h_out);

/* Plugin level for user-supplied patch backends (`-f universal`, framework='prebuilt';
 * reference patch/universal.py:43-69, inferencer.py:209-211,404-455).  The user's callable
 * maps host patches to host outputs that are ALREADY cropped and bump-masked; extract,
 * blend and normalise still run on the device:
 *   begin   : upload the chunk, build the patch grid, zero the accumulators
 *   extract : patches [first, first+nb) -> (nb,1,pz,py,px) float32 on the host
 *   blend   : (nb,C,oz,oy,ox) float32 masked outputs from the host -> accumulate
 *   end     : normalise (+ range check, myelin) and copy (C,oz,oy,ox) to the host */
int cfb_plugin_begin(cfb_handle h, const void* h_in, int32_t in_dtype, int64_t cz, int64_t cy, int64_t cx);
int cfb_plugin_extract(cfb_handle h, int64_t first, int32_t nb, float* h_patches);
int cfb_plugin_blend(cfb_handle h, int64_t first, int32_t nb, const float* h_masked_outputs);
int cfb_plugin_end(cfb_handle h, float* h_out);

/* Timing of the last cfb_infer_chunk_* call, CUDA events on the work stream (ms):
 * [0] total device time, [1] convnet kernels, [2] blend+normalise, [3] h2d, [4] d2h.
 * Kernel launches of the last call are returned through *launches. */
int cfb_last_timing(cfb_handle h, float ms[5], int64_t* launches);

/* Per-layer profiling (tracing aid; reference keeps only wall-clock per operator,
 * flow/flow.py:1926-1932).  When enabled every network kernel launch of the following
 * inference calls is bracketed by CUDA events on the work stream.  cfb_layer_timing
 * synchronises and reports, for up to `capacity` kernel classes: a name (<=31 chars),
 * total milliseconds and launch count accumulated since profiling was enabled. */
int cfb_set_profiling(cfb_handle h, int32_t enabled);
int cfb_layer_timing(cfb_handle h, int32_t capacity, int32_t* count, char (*names)[32], float* ms,
                     int64_t* launches);

/* Test hook: raw network output (before crop/mask) of one host patch, (Cnet,pz,py,px). */
int cfb_debug_net_forward_host(cfb_handle h, const float* h_patch, float* h_out);
/* Test hook: one 3x3x3 convolution layer run through the engine's precision path.
 * in (cin,z,y,x) fp32 host, weight (cout,cin,3,3,3), bias (cout) -> out (cout,z,y,x). */
int cfb_debug_conv3_host(cfb_handle h, const float* h_in, int32_t cin, int32_t z, int32_t y, int32_t x,
                         const float* h_weight, const float* h_bias, int32_t cout, int32_t relu,
                         float* h_out);

/* ---------------------------------------------------------------------------------------------
 * Operators either side of `inference`, on device memory (SURVEY.md section 8 f3): the chunk can stay in HBM
 * between operators.  Stand-alone entry points (no handle); every pointer is a device pointer on the current
 * device; work is enqueued on `stream` (a cudaStream_t, may be NULL).  Results are bit-identical to the reference's
 * numpy code.  Python mirror: chunkflow_b200/chunk/device.py (DeviceChunk).
 * ------------------------------------------------------------------------------------------- */
#define CFB_QUANTIZE_XY 0
#define CFB_QUANTIZE_Z 1

/* In-place Image.normalize_contrast (reference chunk/image/base.py:30-132) of a (z,y,x) uint8 image: per-section
 * 256-bin histogram (bin 0 ignored, 255 bins unless the value 255 occurs) -> clamping values at the clip fractions ->
 * float32 lookup table clipped to [minval,maxval], rounded half to even -> applied; then, as in the reference (the
 * whole-array branch is the `else` of its `for` loop), once more with the histogram of the WHOLE normalised array.
 * per_section == 0 does nothing, exactly like the reference.  0 <= minval <= maxval <= 255. */
int cfb_normalize_contrast_device(void* d_image, int64_t z, int64_t y, int64_t x, double lower_clip_fraction,
                                  double upper_clip_fraction, int32_t minval, int32_t maxval, int32_t per_section,
                                  void* stream);

/* In-place Chunk.maskout (reference chunk/base.py:811-829): chunk[c,z,y,x] *= mask[z/fz, y/fy, x/fx], the mask being
 * (z/fz, y/fy, x/fx) voxels at an integer multiple (fz,fy,fx) of the chunk's voxel size.  dtype pairs as numpy allows
 * them in place: (U8 chunk, U8/bool mask), (F32 chunk, U8/bool mask), (F32 chunk, F32 mask). */
int cfb_maskout_device(void* d_chunk, int32_t chunk_dtype, int64_t channels, int64_t z, int64_t y, int64_t x,
                       const void* d_mask, int32_t mask_dtype, int64_t fz, int64_t fy, int64_t fx, void* stream);

/* Chunk.crop_margin (reference chunk/base.py:691-726): d_dst (channels, z-m0-m3, y-m1-m4, x-m2-m5) receives
 * src[..., m0:z-m3, m1:y-m4, m2:x-m5]; margin = {-z,-y,-x,+z,+y,+x} (the 3-element form is m3..5 = m0..2). */
int cfb_crop_margin_device(const void* d_src, int32_t dtype, int64_t channels, int64_t z, int64_t y, int64_t x,
                           const int64_t margin[6], void* d_dst, void* stream);

/* AffinityMap.quantize (reference chunk/affinity_map/base.py:33-57): (channels,z,y,x) float32 -> (z,y,x) uint8,
 * CFB_QUANTIZE_XY: uint8(((a[0] + a[1]) / 2) * 255), CFB_QUANTIZE_Z: uint8(a[channels-1] * 255); float32
 * arithmetic, C truncation. */
int cfb_quantize_device(const float* d_affinity, int64_t channels, int64_t z, int64_t y, int64_t x, int32_t mode,
                        uint8_t* d_out, void* stream);

/* `connected-components` (SURVEY.md section 8 f4): Chunk.connected_component (reference chunk/base.py:128-137) =
 * [Chunk.threshold: array > threshold (:728-737)] + cc3d.connected_components(seg, connectivity).  d_in: (z,y,x) uint8 / uint32
 * labels (0 = background; equal non-zero values connect) or float32 (thresholded first); connectivity 6 / 18 / 26;
 * d_labels: (z,y,x) uint32, components numbered 1..N in the order of their first voxel in a raster scan (x fastest), like cc3d.
 * d_workspace: cfb_connected_components_workspace(z,y,x) bytes of device memory.  num_labels (host, may be NULL; when given the
 * stream is synchronised) receives N. */
int cfb_connected_components_device(const void* d_in, int32_t in_dtype, int64_t z, int64_t y, int64_t x, float threshold,
                                    int32_t connectivity, uint32_t* d_labels, void* d_workspace, uint32_t* num_labels,
                                    void* stream);
int64_t cfb_connected_components_workspace(int64_t z, int64_t y, int64_t x);

/* `agglomerate` (SURVEY.md section 8 f4): the reference's plugin (chunkflow/plugins/agglomerate.py:8-48) hands the affinity
 * map to waterz.agglomerate(affs, [threshold], fragments=, aff_threshold_low=, aff_threshold_high=,
 * scoring_function='OneMinus<MeanAffinity<RegionGraphType, ScoreValue>>') -- watershed fragments, region graph,
 * hierarchical merging.  waterz is a third-party package that is not vendored in the reference tree; its published algorithm
 * is restated in oracle/agglomeration_oracle.py ("parity unpinned").  Four steps, the voxel passes on the device:
 *
 * d_affs: (3, z, y, x) float32.  flip_channel != 0: the channels are in chunkflow's order x, y, z (the plugin's
 * `flip_channel`, agglomerate.py:26-29: waterz wants z, y, x) and are read in reverse instead of being copied.
 *
 * cfb_watershed_device: steepest-ascent watershed (waterz backend/watershed.hpp; Zlateski & Seung, arXiv:1505.00249) ->
 * d_fragments (z,y,x) uint32, basins numbered 1..N in raster order of their first voxel, 0 = voxels whose strongest edge does
 * not exceed aff_threshold_low.  Plateau interiors drain towards the neighbour one breadth-first step closer to a plateau
 * corner (order independent; the sequential code's queue order is not reproduced, see the oracle).  d_workspace:
 * cfb_watershed_workspace(z,y,x) bytes.  num_fragments (host, may be NULL; the stream is synchronised either way). */
int64_t cfb_watershed_workspace(int64_t z, int64_t y, int64_t x);
int cfb_watershed_device(const float* d_affs, int32_t flip_channel, int64_t z, int64_t y, int64_t x, float aff_threshold_low,
                         float aff_threshold_high, uint32_t* d_fragments, void* d_workspace, uint32_t* num_fragments,
                         void* stream);

/* Region graph (waterz backend/region_graph.hpp with the MeanAffinity statistics): for every pair of touching fragments
 * (6-neighbourhood, ids != 0) the SUM of the affinities on the faces between them, in 2^-30 fixed point (each affinity clamped
 * to [0,1], NaN = 0, rounded to nearest even: the sum does not depend on the order of the atomics), and their COUNT.  Built in
 * an open-addressing table of `table_slots` (a power of two) slots inside d_workspace (cfb_region_graph_workspace(table_slots)
 * bytes); returns CFB_ERR_CAPACITY when the table is too full -- call again with more slots.  *num_edges = pairs found.
 * cfb_region_graph_read copies the edges to the host, sorted by (u, v), u < v. */
int64_t cfb_region_graph_workspace(int64_t table_slots);
int cfb_region_graph_device(const float* d_affs, int32_t flip_channel, const uint32_t* d_fragments, int64_t z, int64_t y, int64_t x,
                            void* d_workspace, int64_t table_slots, int64_t* num_edges, void* stream);
int cfb_region_graph_read(void* d_workspace, int64_t table_slots, int64_t num_edges, uint32_t* h_u, uint32_t* h_v,
                          uint64_t* h_sum_fixed, uint32_t* h_count, void* stream);

/* The merge loop (waterz backend/IterativeRegionMerging.hpp, scoring function OneMinus<MeanAffinity>), on the HOST like
 * waterz's own: repeatedly merge the edge with the smallest score 1 - sum / (count * 2^30) (ties: the edge holding the smallest
 * original (u, v) pair first) until the smallest score reaches `threshold`; a merged cluster is known by its smallest id,
 * edges to a common neighbour pool their statistics.  root_of[i], i < num_nodes (= largest fragment id + 1), receives the id node i ends up with
 * (root_of[0] == 0).  No GPU involved. */
int cfb_agglomerate_edges_host(int64_t num_nodes, int64_t num_edges, const uint32_t* u, const uint32_t* v,
                               const uint64_t* sum_fixed, const uint32_t* count, float threshold, uint32_t* root_of);

/* d_out[i] = d_map[d_labels[i]] (labels >= map_size pass through): applies root_of to the fragments. */
int cfb_relabel_device(const uint32_t* d_labels, int64_t n, const uint32_t* d_map, int64_t map_size, uint32_t* d_out,
                       void* stream);

/* `evaluate-segmentation` (reference flow/flow.py:1519-1542 -> chunk/segmentation.py:33-67 -> lib/gala/evaluate.py).
 *
 * cfb_contingency_device: one pass over d_seg and d_gt (n voxels each, CFB_DTYPE_U32 or CFB_DTYPE_U64, 16-byte aligned; every
 * id is a label, 0 and 2^64 - 1 included) builds the contingency table -- the number of voxels of every (seg id, gt id) pair
 * that occurs -- with exact 64-bit counts in an open-addressing table of `table_slots` (a power of two) slots inside
 * d_workspace (cfb_contingency_workspace(table_slots) bytes).  *num_entries = pairs found.  Returns CFB_ERR_CAPACITY when the
 * pairs fill more than half the slots: call again with a larger table.  Synchronises the stream.
 *
 * cfb_contingency_scores: reduces the table (the workspace of a successful cfb_contingency_device) to the exact integer sums
 * below, in the same number whatever the order of the device's atomics.  Synchronises the stream.
 *
 * cfb_contingency_read: copies the table to the host, sorted by (seg id, gt id). */
typedef struct cfb_contingency_sums {
  uint64_t voxels;               /* n */
  uint64_t entries;              /* pairs (s, g) in the table */
  uint64_t sum_sq_pairs;         /* sum of n_sg^2 over the table */
  uint64_t sum_sq_seg;           /* sum of a_s^2, a_s = sum_g n_sg (label 0 included) */
  uint64_t sum_sq_gt;            /* sum of b_g^2, b_g = sum_s n_sg */
  uint64_t nonzero_voxels;       /* voxels with s != 0 and g != 0 */
  uint64_t seg_labels;           /* distinct s != 0 */
  uint64_t pairs_over_threshold; /* pairs with s != 0, g != 0 and n_sg > size_threshold */
  /* sums of x log2 x in 128-bit fixed point with 62 fractional bits, {low word, high word}; each term is a double,
   * converted exactly; terms with label 0 on either side left out:
   * over n_sg (s != 0, g != 0); over a'_s = sum_{g != 0} n_sg (s != 0); over b'_g = sum_{s != 0} n_sg (g != 0) */
  uint64_t xlogx_pairs[2];
  uint64_t xlogx_seg[2];
  uint64_t xlogx_gt[2];
} cfb_contingency_sums;

int64_t cfb_contingency_workspace(int64_t table_slots);
int cfb_contingency_device(const void* d_seg, int32_t seg_dtype, const void* d_gt, int32_t gt_dtype, int64_t n, void* d_workspace,
                           int64_t table_slots, int64_t* num_entries, void* stream);
int cfb_contingency_scores(void* d_workspace, int64_t table_slots, int64_t n, int64_t num_entries, double size_threshold,
                           cfb_contingency_sums* out, void* stream);
int cfb_contingency_read(void* d_workspace, int64_t table_slots, int64_t num_entries, uint64_t* h_seg, uint64_t* h_gt,
                         uint64_t* h_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CHUNKFLOW_B200_H_ */
