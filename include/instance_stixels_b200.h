/*
 * instance_stixels_b200 -- C ABI of the Blackwell-native stixel hot path.
 *
 * This is the drop-in boundary for ONE path of tudelft-iv/instance_stixels:
 *   column join -> per-column cost tables -> ground/object/sky DP ->
 *   backtracking/emission -> instance grouping,
 * i.e. everything `Stixels::Compute` + its setters/getters do in the
 * reference (InstanceStixels/src/Stixels.cu:43-776).  Plain pointers and
 * sizes only; no C++/torch types.  Every entry point cites the reference
 * interface it replaces (paths relative to the reference repository root).
 *
 * The C++ class `Stixels` in include/InstanceStixels/Stixels.hpp has the
 * reference's public signatures and forwards to these functions, so
 * apps/run_cityscapes.cu and apps/stixels_wrapper.cu compile against it
 * unchanged (see INTEGRATION.md).
 *
 * All functions return ISX_OK (0) or a negative isx_status; the text of the
 * last failure is available through isx_last_error().  There is no CPU
 * fallback: without a CUDA device every compute entry point fails with
 * ISX_ERR_CUDA.
 */
#ifndef INSTANCE_STIXELS_B200_H_
#define INSTANCE_STIXELS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ISX_ABI_VERSION 2

typedef enum isx_status {
  ISX_OK = 0,
  ISX_ERR_INVALID_ARGUMENT = -1, /* reference: throws std::invalid_argument (Stixels.cu:292-313) */
  ISX_ERR_NOT_INITIALIZED = -2,
  ISX_ERR_CUDA = -3,             /* reference: CUDA_CHECK_RETURN -> exit(1) (util.h:27-42) */
  ISX_ERR_CAPACITY = -4,         /* batch larger than isx_initialize(max_batch), column with >= 200 stixels */
  ISX_ERR_UNSUPPORTED = -5
} isx_status;

/* Geometric stixel types, InstanceStixels/include/InstanceStixels/types.h:22-24 */
#define ISX_GROUND 0
#define ISX_OBJECT 1
#define ISX_SKY 2

/* configuration.h:29-34 */
#define ISX_MAX_STIXELS_PER_COLUMN 200
#define ISX_DOWNSAMPLE_FACTOR 8
#define ISX_INSTANCE_CLASSES 8      /* Cityscapes trainIds 11..18 (Stixels.cu:47) */
#define ISX_FIRST_INSTANCE_CLASS 11 /* StixelsKernels.cu:926 */
/* Tallest frame isx_initialize accepts.  The reference stops at 1024 rows (one
 * thread per row in one block); its tile DP does not need that, and up to 2047
 * rows the reference's padded sizes (rows_power2 = 2048,
 * rows_power2_segmentation = 256) and so the segmentation layout stay the same.
 * Taller frames are refused with ISX_ERR_UNSUPPORTED. */
#define ISX_MAX_ROWS 2047

/* Same members, defaults and "-1 == unset" sentinels as `StixelConfig`
 * (types.h:30-141).  isx_config_init() writes the reference's defaults. */
typedef struct isx_config {
  float rows, cols; /* floats in the reference too (types.h:33-34) */
  int32_t max_dis;
  float invalid_disparity;
  float eps;
  int32_t min_pts;
  int32_t size_filter;
  int32_t n_semantic_classes;
  int32_t n_offset_channels;
  float prior_weight, segmentation_weight, instance_weight, disparity_weight;
  int32_t pairwise; /* convenience storage only, like types.h:57-60 */
  int32_t column_step;
  float focal, baseline, camera_center_x, camera_center_y;
  float sigma_disparity_object, sigma_disparity_ground, sigma_sky;
  float pout, pout_sky, pord, pgrav, pblg;
  float pground_given_nexist, pobject_given_nexist, psky_given_nexist;
  float pnexist_dis, pground, pobject, psky;
  int32_t width_margin;
  float sigma_camera_tilt, sigma_camera_height;
  int32_t median_join;
  float epsilon, range_objects_z;
  float road_vdisparity_threshold;
} isx_config;

/* Bit-identical to `Section` (types.h:186-194): 8 x 4 bytes. */
typedef struct isx_section {
  int32_t type; /* ISX_GROUND/OBJECT/SKY; -1 terminates a column */
  int32_t vB, vT;
  float disparity;
  int32_t semantic_class;
  float cost;
  float instance_meanx;
  float instance_meany;
} isx_section;

/* The scalar members of `StixelsData` (types.h:196-205). */
typedef struct isx_frame_meta {
  int32_t rows, cols, realcols, max_sections, max_dis, column_step;
  int32_t semantic_classes;
  float alpha_ground;
  int32_t vhor; /* flipped: rows - vhor_in - 1 (Stixels.cu:377,627) */
} isx_frame_meta;

/* Arguments of Stixels::SetRoadParameters (Stixels.cu:375-381), per frame. */
typedef struct isx_road {
  int32_t vhor; /* horizon image row, top-left origin */
  float camera_tilt, camera_height, alpha_ground;
} isx_road;

/* One entry of the map Stixels::GetInstanceStixels returns
 * (Stixels.cu:744-776): key (column, index-from-top), value DBSCAN label
 * (-1 = noise; labels are per semantic class like the reference's). */
typedef struct isx_instance {
  int32_t column;
  int32_t index;
  int32_t label;
  int32_t semantic_class;
} isx_instance;

/* Where one frame of a batch lies in the packed result arrays (isx_wait_batch_packed): the used Sections of its
 * columns back to back (column 0 first, inside a column top to bottom like the reference's array, no
 * terminators), and its instance records.  `error` holds the per-frame error bits (1: a column reached
 * MAX_STIXELS_PER_COLUMN, 2: instance offsets out of range); `overflow` != 0 means the frame did not fit the
 * packed arrays (bit 0: sections, bit 1: instance records) and must be read with isx_fetch_batch_results. */
typedef struct isx_packed_frame {
  int32_t section_offset, section_count;
  int32_t instance_offset, instance_count;
  int32_t error, overflow;
  int32_t reserved[2];
} isx_packed_frame;

typedef struct isx_context *isx_handle;

/* ------------------------------------------------------------------ */
/* Library                                                            */
int isx_abi_version(void);
/* Number of CUDA kernels this library has launched in this process (the
 * bench reports it as gpu_launches). */
uint64_t isx_kernel_launch_count(void);
const char *isx_last_error(isx_handle h); /* h may be NULL: last global error */

/* ------------------------------------------------------------------ */
/* Object lifetime and configuration                                  */

/* StixelConfig default member initialisers (types.h:30-141). */
void isx_config_init(isx_config *cfg);
/* Stixels::Stixels() (Stixels.cu:33); `device` = CUDA ordinal. */
int isx_create(isx_handle *out, int device);
/* Stixels::~Stixels(); also performs Finish() if still initialised. */
int isx_destroy(isx_handle h);
/* Stixels::SetConfig (Stixels.cu:292-338): ISX_ERR_INVALID_ARGUMENT where
 * the reference throws. */
int isx_set_config(isx_handle h, const isx_config *cfg);
/* The fine-grained setters the reference keeps public (Stixels.hpp:58-88). */
int isx_set_disparity_parameters(isx_handle h, int rows, int cols, int max_dis, float invalid_disparity,
                                 float sigma_disparity_object, float sigma_disparity_ground,
                                 float sigma_sky); /* Stixels.cu:425-437 */
int isx_set_segmentation_parameters(isx_handle h, int classes, int instance_channels); /* :402-406 */
int isx_set_clustering_parameters(isx_handle h, float eps, int min_pts, int size_filter); /* :395-400 */
int isx_set_weight_parameters(isx_handle h, float prior_weight, float disparity_weight,
                              float segmentation_weight, float instance_weight); /* :408-423 */
int isx_set_probabilities(isx_handle h, float pout, float pout_sky, float pground_given_nexist,
                          float pobject_given_nexist, float psky_given_nexist, float pnexist_dis,
                          float pground, float pobject, float psky, float pord, float pgrav,
                          float pblg); /* :361-373 */
int isx_set_camera_parameters(isx_handle h, float focal, float baseline, float sigma_camera_tilt,
                              float sigma_camera_height, float camera_center_x,
                              float camera_center_y); /* :383-393 */
int isx_set_model_parameters(isx_handle h, int column_step, int median_join, float epsilon,
                             float range_objects_z, int width_margin); /* :439-446 */
/* Stixels::Initialize (Stixels.cu:43-248): allocations + LUT precompute.
 * `max_batch` >= 1 is the number of frames one batched call may carry (the
 * reference has no batching; its Initialize is max_batch == 1).  Frames of
 * more than ISX_MAX_ROWS rows are refused with ISX_ERR_UNSUPPORTED. */
int isx_initialize(isx_handle h, int max_batch);
/* Stixels::Finish (Stixels.cu:250-283). */
int isx_finish(isx_handle h);
/* Stixels::IsInitialized (Stixels.hpp:96). */
int isx_is_initialized(isx_handle h);
/* Stixels::GetRealCols / GetMaxSections (Stixels.cu:778-784). */
int isx_real_cols(isx_handle h);
int isx_max_sections(isx_handle h);
/* Length (in int32) of one frame's segmentation tensor
 * [realcols][classes+offsets][rows_power2_segmentation] (Stixels.cu:136-139). */
size_t isx_segmentation_elems(isx_handle h);

/* ------------------------------------------------------------------ */
/* Single-frame path: the reference's call sequence                   */
/* (apps/run_cityscapes.cu:346,383-387,406-411,430-431)               */

/* Stixels::SetDisparityImage (Stixels.cu:348-355): host [rows][cols] fp32. */
int isx_set_disparity_image(isx_handle h, const float *host, size_t n);
/* Stixels::GetInputDisparityImageOnDevice (Stixels.cu:357-359). */
float *isx_input_disparity_device(isx_handle h);
/* Stixels::SetSegmentation (Stixels.cu:340-346): host int32
 * [realcols][21][rows_power2_segmentation]. */
int isx_set_segmentation(isx_handle h, const int32_t *host, size_t n);
/* Stixels::SetRoadParameters (Stixels.cu:375-381). */
int isx_set_road_parameters(isx_handle h, int vhor, float camera_tilt, float camera_height,
                            float alpha_ground);
/* Stixels::Compute (Stixels.cu:449-637).  `sections` receives
 * realcols*max_sections entries, `meta` the StixelsData scalars.
 * `d_segmentation_local` is the optional borrowed DEVICE tensor of the ROS
 * path (apps/stixels_wrapper.cu:208-209); unlike the reference it is NOT
 * modified.  Instance grouping (ClusterInstances, :639-681) runs inside. */
int isx_compute(isx_handle h, int pairwise, isx_section *sections, isx_frame_meta *meta,
                const int32_t *d_segmentation_local);
/* Stixels::ClusterInstances (Stixels.cu:639-681).  Grouping already ran in
 * isx_compute; kept because the reference exposes it publicly. Idempotent. */
int isx_cluster_instances(isx_handle h);
/* The grouping step on its own: what Stixels::ClusterInstances asks of the cuML fork per class,
 * `ML::dbscanFit(handle, X, n, 2, eps, min_pts, labels, 0, false, core_candidates)` (Stixels.cu:660-666).
 * `xy` = n x 2 instance-centre votes, `core_candidates` = the size-filter mask, `labels` out
 * (-1 = noise, clusters numbered by their lowest-index core point).  Host buffers, runs on `device`. */
int isx_dbscan_fit_host(int device, const float *xy, int n, float eps, int min_pts,
                        const unsigned char *core_candidates, int *labels);
/* Stixels::GetInstanceStixels (Stixels.cu:744-776).  Writes up to `capacity`
 * entries, ordered by (semantic class, column, index); *n = total count. */
int isx_get_instance_stixels(isx_handle h, isx_instance *out, int capacity, int *n);

/* ------------------------------------------------------------------ */
/* Batched paths (no reference counterpart: the reference processes one
 * frame per Compute call).  Frames are independent.                   */

/* Host buffers in, host buffers out; H2D/D2H copies are inside the call,
 * pipelined over CUDA streams.  `disparity` = [n][rows][cols],
 * `segmentation` = [n][isx_segmentation_elems], `roads` = [n].
 * `sections` = [n][realcols][max_sections]; `instances` receives frame after
 * frame at most `instances_capacity` entries in total, `instance_offsets`
 * = [n+1] prefix of per-frame counts.  instances/instance_offsets may be NULL. */
int isx_compute_batch_host(isx_handle h, int pairwise, int n, const float *disparity,
                           const int32_t *segmentation, const isx_road *roads, isx_section *sections,
                           isx_instance *instances, int instances_capacity, int32_t *instance_offsets);

/* Inputs already resident in device memory (the bench's `value` leg): runs
 * the kernels on the handle's stream and leaves results on the device.
 * Layouts as above. Returns after enqueueing; isx_synchronize() waits. */
int isx_compute_batch_device(isx_handle h, int pairwise, int n, const float *d_disparity,
                             const int32_t *d_segmentation, const isx_road *roads);
int isx_synchronize(isx_handle h);
/* Asynchronous form of isx_compute_batch_host for a streaming caller: isx_submit_batch_host enqueues the
 * copies and kernels of one batch (same arguments, same layouts) and returns once they are queued;
 * isx_wait_batch_host waits for the OLDEST batch in flight, after which that batch's `sections` buffer is
 * complete, and delivers its packed instance records.  At most three batches may be in flight per handle
 * (submit, submit, submit, wait, submit, wait, ...): with two, the head and tail of one batch hide behind the
 * kernels of the other; with three, the input copies of a batch are also queued before the batch two ahead of it
 * has delivered its results, so the copy engine never waits for the host thread.  `disparity`, `segmentation` and `sections` must stay valid (and should be pinned) until the
 * batch has been waited for.  The synchronous entry points refuse to run while batches are in flight. */
int isx_submit_batch_host(isx_handle h, int pairwise, int n, const float *disparity, const int32_t *segmentation,
                          const isx_road *roads, isx_section *sections);
int isx_wait_batch_host(isx_handle h, isx_instance *instances, int instances_capacity, int32_t *instance_offsets);
/* The result arrays of a batch in flight (device arrays + the pinned host arrays the device packs into) are
 * allocated when a submit first needs them -- tens of milliseconds inside the caller's stream.  A caller that knows
 * how many batches it keeps in flight (1 .. 3) reserves them up front. */
int isx_reserve_in_flight(isx_handle h, int batches);
/* Zero-copy form of isx_wait_batch_host: waits for the oldest batch in flight and hands out the packed results
 * where the device wrote them (pinned host memory owned by the handle): `*sections` / `*instances` are the packed
 * arrays, `*counts` = [n][realcols] stixels per column, `*frames` = [n] descriptors (offsets into the packed
 * arrays), `*n` = frames of the batch.  The `sections` buffer given to isx_submit_batch_host (may be NULL for
 * callers that only use this form) is not written.  The pointers stay valid until the second isx_submit_batch_host
 * after this call.  Any pointer argument may be NULL. */
int isx_wait_batch_packed(isx_handle h, const isx_section **sections, const int32_t **counts,
                          const isx_instance **instances, const isx_packed_frame **frames, int *n);
/* Narrow host inputs, extensions beside the float API for callers whose data is narrower at its source (over the
 * host link the input bytes are what limits a batch): `disparity` = uint16 [n][rows][cols], pixel value =
 * u16 * disparity_scale (a 16-bit disparity PNG with scale 1/256 is what apps/run_cityscapes.cu:141-147 turns
 * into floats on the host); `segmentation` = int16 [n][realcols][channels][ceil(rows/8)], the same values as
 * the int32 tensor without the zero padding to rows_power2_segmentation (isx_narrow_segmentation_elems() per
 * frame).  Widened on the device; results are bit-identical to the float entry points called with the widened
 * arrays.  rows*cols must be a multiple of 8.  Otherwise like isx_compute_batch_host / isx_submit_batch_host. */
size_t isx_narrow_segmentation_elems(isx_handle h);
int isx_compute_batch_host_u16(isx_handle h, int pairwise, int n, const uint16_t *disparity, float disparity_scale,
                               const int16_t *segmentation, const isx_road *roads, isx_section *sections,
                               isx_instance *instances, int instances_capacity, int32_t *instance_offsets);
int isx_submit_batch_host_u16(isx_handle h, int pairwise, int n, const uint16_t *disparity, float disparity_scale,
                              const int16_t *segmentation, const isx_road *roads, isx_section *sections);
/* Copy results of the last device batch to host buffers (same layouts as
 * isx_compute_batch_host). */
int isx_fetch_batch_results(isx_handle h, int n, isx_section *sections, isx_instance *instances,
                            int instances_capacity, int32_t *instance_offsets);
/* cudaStream_t of the handle as an integer (for CUDA-event timing by the
 * caller on the stream the kernels are launched on). */
uint64_t isx_stream(isx_handle h);
/* Orders every result of the batches enqueued so far (backtracking and instance grouping run on a second
 * stream) before whatever the caller enqueues next on isx_stream().  isx_synchronize, isx_fetch_batch_results
 * and isx_rasterize_batch_device do this themselves; a caller that records its own events or launches its own
 * consumers on isx_stream() after isx_compute_batch_device calls it first.  Asynchronous. */
int isx_flush(isx_handle h);

/* Pinned host memory for callers without the CUDA headers (the batched entry points copy from / into the
 * caller's buffers asynchronously: pageable memory works but is staged by the driver at a fraction of the link
 * rate).  Portable across devices and mapped, so a Section array allocated here is filled by the device directly. */
void *isx_host_alloc(size_t bytes);
void isx_host_free(void *p);

/* ------------------------------------------------------------------ */
/* Frame pool (SURVEY.md 8e): one context and one host worker thread per GPU inside ONE process; a call shards
 * its frames into contiguous blocks, frame f -> worker f * G / n, and every worker streams its block from the front
 * through isx_submit_batch_host / isx_wait_batch_host in sub-batches of `max_batch` frames (three in flight); a
 * worker that has used up its block takes sub-batches from the back of the fullest other block, so that a GPU behind
 * a slower host link does not set the time of the call.  No collective: frames are independent, results land in the
 * caller's arrays in frame order whoever computed them.  `devices` may name a GPU more than once (several workers
 * on one GPU).  The reference has no counterpart (one frame per Compute). */
typedef struct isx_pool *isx_pool_handle;
int isx_pool_create(isx_pool_handle *out, const int *devices, int n_devices, const isx_config *cfg, int max_batch);
int isx_pool_destroy(isx_pool_handle p);
int isx_pool_size(isx_pool_handle p);          /* number of workers */
int isx_pool_real_cols(isx_pool_handle p);
size_t isx_pool_segmentation_elems(isx_pool_handle p);
/* Same arguments and layouts as isx_compute_batch_host, any n >= 1.  Blocks until all frames are done. */
int isx_pool_compute_host(isx_pool_handle p, int pairwise, int n, const float *disparity,
                          const int32_t *segmentation, const isx_road *roads, isx_section *sections,
                          isx_instance *instances, int instances_capacity, int32_t *instance_offsets);
const char *isx_pool_last_error(isx_pool_handle p);
/* Frames every worker processed in the last isx_pool_compute_host call (its own block -/+ what was taken over);
 * returns the number of entries written. */
int isx_pool_frames_by_worker(isx_pool_handle p, int *frames, int capacity);

/* ------------------------------------------------------------------ */
/* Introspection for parity tests / profiling (device -> host copies of
 * the intermediates of the LAST batch, frame `frame`).                */
typedef enum isx_tensor {
  ISX_T_JOINED_DISPARITY = 0, /* float [realcols][rows], bottom-up (StixelsKernels.cu:980-1095) */
  ISX_T_OBJECT_LUT = 1,       /* float [realcols][max_dis][rows+1] (StixelsKernels.cu:959-978) */
  ISX_T_DISPARITY_PS = 2,     /* float [realcols][rows+1] Blelloch-order prefix (StixelsKernels.h:73-103) */
  ISX_T_VALID_PS = 3,         /* float [realcols][rows+1] */
  ISX_T_GROUND_PS = 4,        /* float [realcols][rows+1] */
  ISX_T_SKY_PS = 5,           /* float [realcols][rows+1] */
  ISX_T_COST_TABLE = 6,       /* float [realcols][rows][3] final DP costs (cost_table, StixelsKernels.cu:339) */
  ISX_T_INDEX_TABLE = 7,      /* int32 [realcols][rows][3] = vB*3+prev_type like index_table (:340) */
  ISX_T_GROUND_TABLES = 8,    /* float [3][rows]: ground_function | normalization_ground | inv_sigma2_ground (Stixels.cu:790-817) */
  ISX_T_OBJ_COST_LUT = 9,     /* float [max_dis][max_dis] (Stixels.cu:122-129) */
  ISX_T_OBJECT_DISPARITY_RANGE = 10 /* float [max_dis] (Stixels.cu:111-115) */
} isx_tensor;
/* Per-stage device time, measured with CUDA events on the handle's stream
 * around the launches of every enqueued chunk while profiling is enabled.
 * Stages: 0 column join | 1 frame tables (pairwise) | 2 column tables + object
 * LUT | 3 DP | 4 backtracking + candidate collection | 5 grouping + packing.
 * isx_get_stage_times synchronises, accumulates into ms[0..n_stages) /
 * chunks[] (number of timed launches per stage) and optionally resets. */
int isx_set_profiling(isx_handle h, int enable);
int isx_get_stage_times(isx_handle h, double *ms, long *chunks, int n_stages, int reset);
/* Developer trace of the host-batch pipeline while profiling is enabled: per chunk 10 time stamps in ms relative to
 * the first (input copy begin | end; join | frame tables | column tables | DP begin | DP end; emission begin |
 * grouping begin | emission end).  Returns the number of chunks written (or a negative status); call it before
 * isx_get_stage_times, which consumes the same events. */
int isx_get_chunk_trace(isx_handle h, double *ms, int max_chunks);
/* Frames per kernel launch of the last batch (batches are cut into chunks: 32 frames in unary mode, 64 in pairwise
 * mode, ISX_CHUNK overrides). */
/* DP work since isx_initialize in units of 32 x 32 cells: `total` = every (tile, chunk) pair of every column,
 * `evaluated` = those the kernels actually walked (the unary DP prunes chunks that provably cannot win). */
int isx_get_dp_units(isx_handle h, unsigned long long *evaluated, unsigned long long *total);
int isx_chunk_frames(isx_handle h);
/* instance records per frame the packed result arrays hold (isx_submit_batch_host copies that many per frame) */
int isx_instance_capacity(isx_handle h);
size_t isx_tensor_elems(isx_handle h, int tensor);
int isx_read_tensor(isx_handle h, int tensor, int frame, void *host, size_t bytes);


/* ------------------------------------------------------------------------
 * Segmentation ingest (SURVEY.md 8f rank 2).  The reference bakes the layout transform between the
 * CNN and the stixel path into its ONNX export: `FlipAndPad` (tools/CNN_training/models/
 * wrappers.py:35-61: permute(0,3,1,2), rows flipped, zero-padded to rows_power2_segmentation, x *= 8,
 * x.int()), whose output TRTOnnxCNN::inferOnDevice (InstanceStixels/src/TRTOnnxCNN.cpp:134-165) hands
 * to Compute as d_segmentation_local.  These two entry points run that transform on the handle's
 * stream, so any CNN runtime can feed the path with its plain [channels][rows/8][cols/8] float output
 * (19 x -log softmax, y offset, x offset; rows top-down).  With column_step 4 every CNN column feeds
 * two stixel columns (SURVEY.md 8c O3).
 * ------------------------------------------------------------------------ */
/* single frame: fills the tensor SetSegmentation would upload (ordered before the next isx_compute) */
int isx_set_segmentation_from_cnn_device(isx_handle h, const float *d_cnn, int cnn_rows, int cnn_cols);
/* n frames [n][channels][cnn_rows][cnn_cols] -> d_segmentation [n][realcols][channels][rows_power2_segmentation],
 * the layout isx_compute_batch_device takes; asynchronous on isx_stream() */
int isx_flip_and_pad_batch_device(isx_handle h, int n, const float *d_cnn, int cnn_rows, int cnn_cols,
                                  int32_t *d_segmentation);

/* ------------------------------------------------------------------------
 * Result images (SURVEY.md 8f rank 3): the stixels of frames [first, first + n) of the last batch (or of the last
 * isx_compute: first = 0, n = 1) drawn as the reference's evaluation tooling draws them
 * (tools/visualization/clustering_visualization.py: draw_stixels :397-409, draw_instance_masks :118-142) -- every
 * stixel fills the inclusive rectangle x in [c*w, c*w+w-1], y in [rows-1-vT, rows-1-vB]:
 *   d_label_ids    uint8 [n][rows][cols]  Cityscapes label id of the class (trainId2label[class].id)
 *   d_instance_ids int32 [n][rows][cols]  class*1000 + label for instance stixels with 0 <= label < 1000, else 0
 *   d_disparity    float [n][rows][cols]  stixel disparity
 * Any of the three may be NULL.  Device buffers, asynchronous on isx_stream().
 * ------------------------------------------------------------------------ */
int isx_rasterize_batch_device(isx_handle h, int first, int n, uint8_t *d_label_ids, int32_t *d_instance_ids,
                               float *d_disparity);

/* ------------------------------------------------------------------------
 * Device results: the stixels of frames [first, first + n) of the last batch (or of the last isx_compute: first = 0,
 * n = 1) in the caller's DEVICE buffers, for consumers on the GPU (a tracker, a BEV grid, a second network).
 * Frame-ordered CSR: the used Sections of frame f (0 = `first`) at [frame_offsets[f], frame_offsets[f+1]), column 0
 * first, each column top to bottom (the order of isx_wait_batch_packed and of Stixels::Get3DVertices); column c of
 * frame f starts at column_offsets[f*realcols + c], column_offsets[n*realcols] = frame_offsets[n].  Per stixel:
 *   labels[i]     the DBSCAN label of the stixels GetInstanceStixels lists (-1 = noise), -2 for every other stixel
 *   vertices[i]   [4][3] what Stixels::Get3DVertices computes for the stixel, bit for bit (needs camera_center_x/y)
 * frame_errors[f] = the frame's error bits (1: a column reached MAX_STIXELS_PER_COLUMN, 2: instance offsets out of
 * range).  `capacity` counts stixels (entries of sections / labels / vertices): a frame's stixels are written only if
 * frame_offsets[f+1] <= capacity, nothing past it; offsets and errors are always complete.  No atomics: the same
 * bytes on every call.  Asynchronous on isx_stream().
 * ------------------------------------------------------------------------ */
typedef struct isx_device_results { /* device pointers; NULL = not written (frame_offsets is required) */
  isx_section *sections;            /* [capacity], 16-byte aligned */
  int32_t *frame_offsets;           /* [n+1] */
  int32_t *column_offsets;          /* [n*realcols+1] */
  int32_t *labels;                  /* [capacity] */
  float *vertices;                  /* [capacity][4][3] */
  int32_t *frame_errors;            /* [n] */
  int32_t capacity, reserved;
} isx_device_results;               /* 56 bytes */
int isx_export_batch_device(isx_handle h, int first, int n, const isx_device_results *out);

/* ------------------------------------------------------------------------
 * Road estimation (SURVEY.md 8f rank 1): the step in front of the stixel path.
 * Replaces `class RoadEstimation` (InstanceStixels/include/InstanceStixels/RoadEstimation.h:31-93,
 * src/RoadEstimation.cu:24-193, src/RoadEstimationKernels.cu:25-60) including its one third-party
 * step, cv::HoughLines(vDisp, lines, 1.0, CV_PI/180, 25) (RoadEstimation.cu:152), which runs on
 * the device here: v-disparity histogram -> maximum -> binary image -> standard Hough accumulator
 * -> local maxima.  Only the candidate lines (a few hundred (index, votes) pairs) travel to the
 * host, where they are ordered like OpenCV orders them and the first line with a pitch inside
 * +-50 degrees yields the camera properties with the reference's own sinf/cosf/atanf
 * (RoadEstimation.cu:155-193).
 * ------------------------------------------------------------------------ */
typedef struct isx_road_estimator *isx_road_handle;

/* What RoadEstimation::Compute leaves in its getters (RoadEstimation.h:46-50). */
typedef struct isx_road_estimate {
  int32_t ok;            /* return value of RoadEstimation::Compute */
  int32_t horizon_point; /* GetHorizonPoint(): (int)ceil(rho / sin(theta)), image row from the top */
  float pitch;           /* GetPitch() */
  float camera_height;   /* GetCameraHeight() */
  float slope;           /* GetSlope() -> alpha_ground of SetRoadParameters (apps/run_cityscapes.cu:396-407) */
  float rho, theta;      /* the Hough line behind it */
} isx_road_estimate;

int isx_road_create(isx_road_handle *out, int device);
void isx_road_destroy(isx_road_handle h);
/* RoadEstimation::Initialize (RoadEstimation.cu:32-84); max_batch sizes the batched entry point. */
int isx_road_initialize(isx_road_handle h, float camera_center_y, float baseline, float focal, int rows, int cols,
                        int max_dis, float road_vdisparity_threshold, int max_batch);
int isx_road_finish(isx_road_handle h);        /* RoadEstimation::Finish (:86-94) */
int isx_road_is_initialized(isx_road_handle h);
/* RoadEstimation::Compute(const std::vector<pixel_t>&) (:96-105): host image [rows][cols]. */
int isx_road_compute_host(isx_road_handle h, const float *disparity, size_t n_pixels, isx_road_estimate *out);
/* RoadEstimation::Compute(pixel_t* d_im) (:107-137): device image, e.g. Stixels::GetInputDisparityImageOnDevice(). */
int isx_road_compute_device(isx_road_handle h, const float *d_disparity, isx_road_estimate *out);
/* Extension: n frames [n][rows][cols] resident on the device, one estimate per frame. */
int isx_road_compute_batch_device(isx_road_handle h, int n, const float *d_disparity, isx_road_estimate *out);

/* Like isx_compute_batch_device, but each frame's road parameters are estimated on the device from its own
 * disparity image, with `road` (RoadEstimation::Compute(pixel_t*) per frame), in stream order on isx_stream().
 * A frame whose estimation fails (ok == 0) uses the last accepted estimate in frame order, as the getters of
 * RoadEstimation keep it (RoadEstimation.cu:123-133).  Before any estimate has been accepted, it uses `fallback`.
 * fallback != NULL: reset that state to *fallback.  NULL: continue from the state the previous call on `road` left
 * (only this entry point reads or writes that state).
 * d_estimates [n] (optional, device): what isx_road_compute_batch_device would return for each frame.
 * d_roads [n] (optional, device): the road each frame was computed with.  Returns after enqueueing: the caller's
 * thread never waits, and every accessor of the last batch (isx_export_batch_device, isx_fetch_batch_results,
 * isx_rasterize_batch_device, isx_flush, isx_synchronize) works as after isx_compute_batch_device.
 * The line is selected on the device as the argmax of (votes, -accumulator index) over the local maxima above the
 * vote threshold whose pitch is in range -- the line the host walk of isx_road_compute_* accepts -- so the
 * estimates are bit-identical to isx_road_compute_batch_device; unlike that walk it has no cap on the number of
 * candidate lines (isx_road_compute_* return ISX_ERR_CAPACITY beyond 65536).  The ground tables of the frames are
 * computed on the host in stream order (a host function per chunk, cached per road).
 * `road` must be initialised on h's device with h's rows, cols and max_dis, and n must not exceed either handle's
 * max_batch; refusals (ISX_ERR_INVALID_ARGUMENT, ISX_ERR_CAPACITY for sizes) enqueue nothing.  The first call on a
 * road handle builds its table of per-cell estimates on the host (numangle x numrho cells) and must pass a
 * `fallback`.  `road` must not be used from another thread during the call. */
int isx_compute_batch_device_road(isx_handle h, isx_road_handle road, int pairwise, int n,
                                  const float *d_disparity, const int32_t *d_segmentation,
                                  const isx_road *fallback, isx_road_estimate *d_estimates, isx_road *d_roads);
const char *isx_road_last_error(isx_road_handle h);
/* Intermediates of the last call, frame `frame` of it (tests): 0 = v-disparity int32 [rows][max_dis],
 * 1 = binary image uint8 [rows][max_dis], 2 = Hough accumulator int32 [numangle+2][numrho+2]. */
size_t isx_road_tensor_bytes(isx_road_handle h, int tensor);
int isx_road_read_tensor(isx_road_handle h, int tensor, int frame, void *host, size_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* INSTANCE_STIXELS_B200_H_ */
