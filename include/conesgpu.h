/*
 * conesgpu.h — C ABI of libconesgpu.so, the B200 (sm_100a) implementation of the
 * cones_perception point-cloud hot path.
 *
 * The reference (dmn-sjk/cones_perception) has no plugin/FFI interface; its seam is the
 * body of two ROS subscriber callbacks.  Each entry point below names the reference
 * lines it replaces (paths relative to the upstream repository):
 *
 *   cp_ground_remove   GroundRemover::cloud_handler body   src/ground_removal.cpp:54-79
 *   cp_detect          ConeDetector::cloud_handler          src/cone_detection.cpp:151-167
 *                      + the centroid mean loop             src/cone_detection.cpp:261-273
 *                      (filter_points_position :189-204, downsample :240-249,
 *                       euclidan_cluster :206-220, perception_handling::euclidan_dist
 *                       src/perception_handling/utils.cpp:32-34)
 *   cp_batch_*         the same path over many independent frames per launch
 *                      (BASELINE.json configs 3-5)
 *   cp_batch_ground_remove  GroundRemover::cloud_handler for every frame of a batch:
 *                      one groundless_cloud message per frame, on the device or the host
 *
 * Plain C types only: no exceptions, no C++ or torch types cross this boundary.
 * A handle is used by one thread at a time (the reference nodes are single-threaded
 * ros::spin(), src/cone_detection.cpp:127, src/ground_removal.cpp:47).
 * There is no CPU fallback: every compute entry point fails with CP_E_CUDA when no
 * sm_100-class device is usable.
 */
#ifndef CONESGPU_H
#define CONESGPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct cp_handle cp_handle;

typedef enum cp_status {
  CP_OK = 0,
  CP_E_PARAM = 1,    /* NULL pointer, non-finite or out-of-range parameter           */
  CP_E_BADFIELD = 2, /* x/y/z field missing, big-endian data, point_step too small   */
  CP_E_CAPACITY = 3, /* more points / survivors / voxels / clusters than the handle or
                        the caller's output buffer can hold — never silently truncated */
  CP_E_CUDA = 4,     /* CUDA runtime error; see cp_last_error()                      */
  CP_E_NOMEM = 5,
  CP_E_STATE = 6     /* call order violated (e.g. results read before a batch ran)   */
} cp_status;

/* sensor_msgs/PointCloud2 with the fields already resolved to byte offsets, the way
 * pcl::fromROSMsg resolves them (src/cone_detection.cpp:151,153; ground_removal.cpp:54).
 * off_intensity < 0: field absent => intensity = 0 (ground_removal node behaviour).
 * The cone_detection node fakes a missing field at offset 0 (src/cone_detection.cpp:
 * 142-151): its shell passes off_intensity = 0 in that case. */
typedef struct cp_cloud_view {
  const uint8_t* data;
  uint32_t width, height, point_step, row_step;
  int32_t off_x, off_y, off_z, off_intensity;
  uint8_t is_bigendian, is_dense;
} cp_cloud_view;

/* GroundRemover members, src/ground_removal.cpp:18-19 (names as in
 * config/ground_removal_params.yaml).  num_of_sectors only sizes the reference's table;
 * the sector angle is fixed at (360/16 = 22 deg) by the member initialiser (:20). */
typedef struct cp_ground_params {
  int32_t num_of_sectors;
  float default_lowest_point;
} cp_ground_params;

/* Optional second ground model (the reference has none: PARITY UNPINNED): a seeded RANSAC plane per frame, for
 * scans from a pitching or rolling sensor, where the sector model's "z < lowest z of the sector + 0.1" keeps the far
 * ground.  Selected per handle with cp_set_ground_plane; the sector model stays the default.  Frame f has N_f points.
 *   Draw:     hypothesis h takes the frame-local indices idx_j = (u32)((((splitmix64(seed + 3h + j)) >> 32) * N_f) >> 32),
 *             j = 0, 1, 2 (splitmix64: the standard finaliser, golden-ratio increment added first).  The draw depends
 *             on (seed, h, N_f) alone, never on the frame's place in the batch.  N_f < 3: no hypotheses.
 *   Plane:    in double, no contraction: u = p1 - p0, v = p2 - p0, n = u x v, L = |n|.  Invalid if a sample point is
 *             not finite, L is 0 or not finite, or nz/L < cos(max_tilt) after flipping n to nz >= 0.  Otherwise
 *             n /= L, d = -(nx p0x + ny p0y + nz p0z); a, b, c, d rounded to float.  cos(max_tilt) in double.
 *   Distance: s = fmaf(c, z, fmaf(b, y, fmaf(a, x, d))) in fp32.
 *   Score:    finite points with fabsf(s) <= inlier_distance.  Best: the highest count, ties to the lowest h.
 *   Verdict:  keep iff the point is finite and s >= ground_height; no valid plane: keep every finite point.
 * The ground node's message keeps its format (survivors in input order, then N_f - G_f padding points). */
typedef struct cp_plane_params {
  uint64_t seed;
  uint32_t n_hypotheses;   /* 1 .. 256 */
  float inlier_distance;   /* scoring: |s| <= inlier_distance; finite, > 0 */
  float ground_height;     /* verdict: keep iff s >= ground_height; finite */
  float max_tilt_deg;      /* (0, 90]: a plane whose normal is further than this from +z is invalid */
} cp_plane_params;

/* ConeDetector members, src/cone_detection.cpp:22-43, same types and (typo'd) names as
 * config/cones_detection_params_*.yaml. */
typedef struct cp_detect_params {
  double distance_treshold_max, distance_treshold_min, level_threshold, angle_threshold;
  double voxel_filter_leaf_size_x, voxel_filter_leaf_size_y, voxel_filter_leaf_size_z;
  int32_t min_cluster_size, max_cluster_size;
  float cone_width, cone_height; /* CONE_WIDTH 0.228f, CONE_HEIGHT 0.325f (:22-23) */
} cp_detect_params;

/* one detected cone candidate before the host-side extension / temporal gate
 * (src/cone_detection.cpp:276-340 stays in the node shell) */
typedef struct cp_cluster {
  float x, y;         /* mean of member voxel centroids (fp32, ascending voxel index) */
  uint32_t size;      /* member voxels                                               */
  uint32_t min_index; /* smallest member voxel index: canonical cluster label        */
} cp_cluster;

typedef struct cp_frame_counters {
  uint32_t n_points;      /* N  input points                           */
  uint32_t n_ground_kept; /* G  after ground removal (= N when off)    */
  uint32_t n_cropped;     /* C  after the distance/angle/level crop    */
  uint32_t n_voxels;      /* V  occupied voxels                        */
  uint32_t n_components;  /*    connected components before the filter */
  uint32_t n_clusters;    /* K  components with min <= size <= max     */
  uint32_t key_bits;      /*    significant bits of this frame's voxel key */
  uint32_t passthrough;   /*    1 if VoxelGrid's int32 overflow guard fired */
} cp_frame_counters;

typedef struct cp_config {
  int32_t device;          /* CUDA device ordinal                                   */
  uint64_t max_points;     /* total points per call/batch                           */
  uint32_t max_frames;     /* frames per batch                                      */
  uint32_t max_point_step; /* bytes per point of host clouds to stage (>= 16)       */
  uint64_t max_survivors;  /* points after the crop, whole batch (0 = max_points)   */
  uint64_t max_voxels;     /* voxels, whole batch (0 = max_survivors)               */
} cp_config;

const char* cp_strerror(cp_status s);
const char* cp_last_error(const cp_handle* h); /* detail of the last failure, never NULL */
uint32_t cp_abi_version(void);
const char* cp_create_error(void);            /* detail of the last failed cp_create */

cp_status cp_create(cp_handle** out, const cp_config* cfg);
void cp_destroy(cp_handle* h);

/* Page-locked host memory for message buffers (north_star: "PointCloud2 staged to device through pinned
 * cudaMemcpyAsync"): a cloud that already lives in such a buffer is DMA'd straight from it, with no
 * pass through the library's staging ring.  write_combined != 0 asks for cudaHostAllocWriteCombined
 * (fast for the CPU to fill sequentially and for the GPU to read, very slow for the CPU to read back).
 * The pages are placed by the calling thread's NUMA policy: bind the thread next to the GPU first
 * (cones_perception_b200/placement.py).  No handle is needed; device selects the context. */
cp_status cp_pinned_alloc(int32_t device, size_t bytes, int32_t write_combined, void** out);
void cp_pinned_free(void* p);

/* --- node-equivalent single-frame calls (host buffers in, host buffers out) -------- */

/* src/ground_removal.cpp:54-79.  out_xyzi32 receives width*height points in the PCL
 * PointXYZI layout toROSMsg emits (:86): x@0 y@4 z@8 1.0f@12 intensity@16, 32 B/point,
 * survivors first (input order) then zero points.  low17 (optional) receives the 17
 * per-sector minima.  Only the survivors are copied back from the device; the padding points
 * (value-initialised PointXYZI: 1.0f at offset 12) are written into out_xyzi32 by the host while
 * the GPU works, so the whole buffer is overwritten by the call. */
cp_status cp_ground_remove(cp_handle* h, const cp_cloud_view* in, const cp_ground_params* g,
                           void* out_xyzi32, uint32_t* n_kept, float* low17);

/* src/cone_detection.cpp:151-167 + :261-273.  ground may be NULL (ground_removal:=false)
 * or non-NULL to fuse the ground_removal node in front (ground_removal:=true).
 * Clusters are returned in canonical order: size descending, then min_index ascending. */
cp_status cp_detect(cp_handle* h, const cp_cloud_view* in, const cp_detect_params* d,
                    const cp_ground_params* ground, cp_cluster* out, uint32_t cap,
                    uint32_t* n_clusters, cp_frame_counters* counters);

/* --- batches of independent frames ------------------------------------------------- */

/* Describe a batch whose points are already in device memory (HBM-resident input).
 * d_points: n_frames frames back to back, frame f holding frame_points[f] points of
 * point_step bytes each with the given field offsets; the pointer must stay valid until
 * the batch has run. */
cp_status cp_batch_set_device_input(cp_handle* h, const void* d_points, uint32_t n_frames,
                                    const uint32_t* frame_points, uint32_t point_step,
                                    int32_t off_x, int32_t off_y, int32_t off_z,
                                    int32_t off_intensity);

/* Stage a batch from host memory (cudaMemcpyAsync on the handle's stream).
 * Lifetime of the source buffers:
 *   - pageable memory (a ROS message's std::vector): fully consumed when the call returns — it
 *     is packed through the library's pinned ring;
 *   - page-locked memory (cudaHostAlloc / cudaHostRegister), contiguous rows: the DMA reads the
 *     caller's buffer directly and is still in flight when the call returns.  The buffer must
 *     stay valid and unmodified until cp_sync / cp_batch_results (or cp_detect*) of this batch
 *     has returned. */
cp_status cp_batch_set_host_input(cp_handle* h, const cp_cloud_view* frames, uint32_t n_frames);

/* src/ground_removal.cpp:54-79 for every frame of the staged batch (cp_batch_set_device_input /
 * cp_batch_set_host_input; stage host clouds without an intensity field with off_intensity < 0, as
 * cp_ground_remove does).  Frame f's message is out_xyzi32[32*P_f .. 32*(P_f + N_f)), P_f = sum of N_g
 * for g < f, N_f = width*height of frame f: exactly the bytes cp_ground_remove writes for that frame alone
 * (survivors in input order, then N_f - G_f PCL padding points).  out_xyzi32 NULL: device output only
 * (cp_batch_ground_device_output), cap_points is then not read.  n_kept[n_frames] (G_f) and
 * low17[17*n_frames] (each frame's sector minima) are optional.
 * Only the survivors are copied back; the host writes the padding into out_xyzi32 while the GPU works.
 * Returns after the device work is complete, so another handle can read the device output at once (the
 * two-node chain: cp_batch_set_device_input(d_out, ..., point_step 32, offsets 0/4/8/16)).
 * Ends the run: cp_batch_results, cp_batch_cone_colors and cp_batch_track return CP_E_STATE until the next
 * cp_batch_run.  The input stays staged, and a following cp_batch_run on it returns what it would have.
 * CP_E_PARAM: NULL g.  CP_E_STATE: nothing staged.  CP_E_CAPACITY: cap_points < sum of N_f.
 * CP_E_NOMEM: the max_points x 32 B device buffer of the messages cannot be allocated. */
cp_status cp_batch_ground_remove(cp_handle* h, const cp_ground_params* g, void* out_xyzi32, uint64_t cap_points,
                                 uint32_t* n_kept, float* low17);
/* The complete messages of the last cp_batch_ground_remove on the device (sum N_f points x 32 B, padding
 * included).  Valid until the next cp_ground_remove / cp_batch_ground_remove on this handle.
 * CP_E_PARAM: NULL argument.  CP_E_STATE: no cp_batch_ground_remove since the last staging or run. */
cp_status cp_batch_ground_device_output(cp_handle* h, const void** d_out_xyzi32, uint64_t* n_points);

/* Select the ground model of this handle.  p NULL: the sector model of the reference (the default).  p non-NULL: the
 * plane model (cp_plane_params) for every later cp_ground_remove, cp_batch_ground_remove, cp_detect, cp_batch_run
 * and cp_detect_batch with non-NULL ground params, whose num_of_sectors and default_lowest_point are then ignored.
 * A run with the plane model is the two-node chain on the device: the plane ground node's messages, then the detector
 * without ground removal on them, so its crop taps (CP_TAP_CROP_INDEX ...) index the messages, not the input; the
 * counters' n_ground_kept is G_f.  Under the plane model: a non-NULL low17 returns CP_E_PARAM, CP_TAP_SECTOR_LOW
 * returns CP_E_STATE, and so do the colour calls with CP_COLOR_CLOUD_GROUNDLESS and a NULL cloud, cp_batch_cone_colors
 * and cp_batch_track in colour mode under CP_COLOR_CLOUD_GROUNDLESS (STAGED crops work as before).
 * CP_E_PARAM: n_hypotheses outside 1..256, inlier_distance not finite and > 0, ground_height not finite, max_tilt_deg
 * outside (0, 90]. */
cp_status cp_set_ground_plane(cp_handle* h, const cp_plane_params* p);
/* The plane each frame chose in the last run or ground call made with the plane model (calls cp_sync first):
 * planes[n_frames][4] (a, b, c, d), inliers[n_frames] (its score), hypothesis[n_frames] (-1: no valid plane, then the
 * plane is NaN and the inliers 0).  Any pointer may be NULL.  CP_E_STATE: the last run or ground call did not use
 * the plane model.  CP_E_CAPACITY: cap_frames < n_frames. */
cp_status cp_ground_planes(cp_handle* h, float* planes, uint32_t* inliers, int32_t* hypothesis, uint32_t cap_frames);

/* Enqueue the whole pipeline for the current batch on the handle's stream (async). */
cp_status cp_batch_run(cp_handle* h, const cp_detect_params* d, const cp_ground_params* ground);

/* Wait for the stream; surfaces device-side capacity errors. */
cp_status cp_sync(cp_handle* h);

/* After cp_sync: per-frame counters (n_frames entries) and clusters.  cluster_offsets has
 * n_frames+1 entries; frame f's clusters are out[cluster_offsets[f] .. cluster_offsets[f+1]). */
cp_status cp_batch_results(cp_handle* h, cp_frame_counters* counters, uint32_t* cluster_offsets,
                           cp_cluster* out, uint64_t cap, uint64_t* n_total);

/* One call = stage (H2D) + run + results (D2H) for host-resident frames. */
cp_status cp_detect_batch(cp_handle* h, const cp_cloud_view* frames, uint32_t n_frames,
                          const cp_detect_params* d, const cp_ground_params* ground,
                          cp_frame_counters* counters, uint32_t* cluster_offsets, cp_cluster* out,
                          uint64_t cap, uint64_t* n_total);

/* Device time of the last cp_batch_run (CUDA events on the handle's stream), ms.  A one-frame batch that took the
 * single-launch path is not bracketed by events (each record costs about a microsecond of a ~50 us call):
 * CP_E_STATE; cp_set_stage_timing(h, 1) routes such a frame through the multi-launch path, which is timed. */
cp_status cp_last_run_ms(cp_handle* h, float* ms);
/* Per-kernel device times of the two streaming passes (CUDA events on the handle's stream
 * around each launch).  Off by default; bench.py switches it on for the roofline pass. */
typedef enum cp_stage {
  CP_STAGE_SECTOR_MIN = 0,        /* ground_sector_min_kernel (two-kernel front end)   */
  CP_STAGE_MASK_CROP_COMPACT = 1, /* keep_mask_kernel (only when pass 2 runs as its own kernel) */
  CP_STAGE_FRONT_FUSED = 2,       /* front_fused_kernel: both passes, pass 2 from L2   */
  CP_STAGE_FRONT_CLUSTER = 3,     /* front_cluster_kernel: one HBM pass, 16-CTA clusters */
  CP_STAGE_FRAME_BACKEND = 4      /* frame_backend_kernel: pass 2 (keep bits) + VoxelGrid + clustering +
                                     centroids, one CTA per frame                         */
} cp_stage;
cp_status cp_set_stage_timing(cp_handle* h, int on);
cp_status cp_stage_ms(cp_handle* h, cp_stage stage, float* ms);
/* Device timestamps of the last run (stage timing on), in ms after the start of `base`'s last run (NULL: this
 * handle's own): [0] run start, [1]/[2] pass 1 start/end, [3]/[4] pass 2 start/end, [5] run end.  With two
 * handles alternating this shows how consecutive batches overlap (tools/timeline_probe.py). */
/* The exact-path atan2f (the reference's libm atan2f, restated) on n pairs: parity test hook. */
cp_status cp_debug_atan2f(cp_handle* h, const float* y, const float* x, uint32_t n, float* out);
cp_status cp_debug_timeline(cp_handle* h, const cp_handle* base, float out_ms[6]);
/* Device pointers of the last run's results (valid until the next run on this handle):
 * packed cp_cluster records, n_frames+1 cluster offsets, and the total cluster count.
 * Lets a multi-GPU caller hand the cone lists to NCCL without a host round trip: offsets and
 * records are one allocation, d_clusters == d_cluster_offsets + round_up(n_frames_max + 1, 4)
 * 32-bit words (n_frames_max = cp_config.max_frames), so one collective can move both. */
cp_status cp_device_results(cp_handle* h, const void** d_clusters, const uint32_t** d_cluster_offsets,
                            const uint32_t** d_n_clusters);
/* --- multi-GPU result path over peer memory (NVLink 5 / NVSwitch) --------------------------
 * Frames are sharded across GPUs with no data-path collective; the only exchange is the result:
 * every rank's packed cone list is gathered on one rank.  Instead of a separate collective, each
 * cp_batch_run ends with a publish kernel that stores the rank's result block
 * [cluster offsets | cp_cluster records] into the gathering rank's buffer through a CUDA-IPC peer
 * mapping and then raises a per-rank sequence flag there.  Double-buffered by run parity.
 *   rank 0:  cp_gather_create(h, world, slot_words, handle)   -> broadcast the 64-byte handle
 *   others:  cp_gather_open(h, handle, rank, world, slot_words)
 *   then cp_batch_run as usual on every rank; run number = cp_gather_seq(h)
 *   rank 0:  cp_gather_wait(h, seq, timeout_ms); cp_gather_read(h, seq, out, cap)
 * slot_words (multiple of 4) >= round_up(max_frames + 1, 4) + 4 * (cone capacity per rank); every
 * handle of the gather must be created with the same cp_config.max_frames (a slot is laid out like
 * the handle's own result block).  A rank that finds more cones than its slot holds is never
 * truncated silently: its own cp_sync and the gathering rank's cp_gather_wait return CP_E_CAPACITY. */
cp_status cp_gather_create(cp_handle* h, uint32_t world, uint32_t slot_words, uint8_t handle_out[64]);
cp_status cp_gather_open(cp_handle* h, const uint8_t handle[64], uint32_t rank, uint32_t world,
                         uint32_t slot_words);
uint32_t cp_gather_seq(const cp_handle* h);
cp_status cp_gather_wait(cp_handle* h, uint32_t seq, uint32_t timeout_ms);
cp_status cp_gather_read(cp_handle* h, uint32_t seq, void* out_host, uint64_t cap_bytes);
/* 32-point rows (512 B in the compact layout) that pass 2 actually read in the last synchronised run;
 * rows lying entirely below every sector's ground threshold are skipped without being loaded. */
uint64_t cp_last_rows_loaded(const cp_handle* h);
/* Clustering work of the last synchronised run, whole batch (SURVEY.md §5 "pairs tested"): candidate voxel pairs
 * the union kernels looked at, and how many of those had their squared distance evaluated against r2 (the rest
 * left early because both voxels already hung under the same root).  The reference's kd-tree visits
 * O(V * k log k) instead (src/cone_detection.cpp:206-220). */
void cp_last_pairs(const cp_handle* h, uint64_t* visited, uint64_t* tested);
/* Kernel launches enqueued by the last cp_batch_run / cp_detect / cp_ground_remove / cp_batch_ground_remove /
 * cp_batch_cone_colors (the latter counts its own launches only; it does not grow with the number of frames or
 * clusters, and neither does cp_batch_ground_remove's). */
uint32_t cp_last_launch_count(const cp_handle* h);
/* The handle's stream as a cudaStream_t, for callers that time with their own events. */
void* cp_stream(cp_handle* h);

/* --- colour path (SURVEY.md §8 f3): crops, range images and the classifier network ---
 * Only needed with classify_colors:=true. */
typedef struct cp_cone_center {
  float x, y; /* the centroid AFTER the radial extension (src/cone_detection.cpp:276-278), as passed at :309 */
} cp_cone_center;
#define CP_CONE_IMG_ROWS 15 /* scripts/color_classifier_server.py:27-30 */
#define CP_CONE_IMG_COLS 12
enum {
  CP_CONE_EMPTY = 1,         /* no point in the box: the service skips the cone (color_classifier_server.py:83-84) */
  CP_CONE_BAD_INDEX = 2,     /* numpy would raise IndexError (elevation above +15 deg, non-finite coordinates) */
  CP_CONE_BAD_INTENSITY = 4, /* interp1d would raise ValueError (intensity outside [0, 255] or NaN) */
  CP_CONE_AMBIGUOUS = 8      /* a pixel coordinate lies within 1e-9 of a rounding boundary: image not guaranteed */
};
/* Replaces ConeDetector::get_reconstructed_cone (src/cone_detection.cpp:222-238) for n_centers cones in one
 * pass: the points of the raw cloud with |x-cx| <= CONE_WIDTH/1.5 and |y-cy| <= CONE_WIDTH/1.5 (the reference's
 * double-precision comparisons, both ends inclusive), in cloud order.
 *   cloud: the raw cloud, or NULL to use frame `frame` of the input already on the device (the cloud the last
 *          cp_detect / cp_batch_set_*_input call of this handle staged) — no second host-to-device copy.  With
 *          cp_set_color_cloud(h, CP_COLOR_CLOUD_GROUNDLESS) and a last run that fused ground removal, NULL crops
 *          that frame's ground-node message instead (see cp_set_color_cloud).
 *   crop_offsets[n_centers+1]: cone c owns crop_xyzi[4*crop_offsets[c] .. 4*crop_offsets[c+1]).
 *   crop_xyzi: x, y, z, intensity per point (cap_points points); NULL to get the offsets only.
 * CP_E_CAPACITY if the crops hold more than cap_points points (crop_offsets is still complete). */
cp_status cp_cone_crops(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                        uint32_t n_centers, float cone_width, uint32_t* crop_offsets, float* crop_xyzi,
                        uint32_t cap_points);
/* cp_cone_crops followed on the device by ColorClassifier.to_image (scripts/color_classifier_server.py:
 * 130-156): images[n_centers][15][12] uint8 (the classifier's input before the float cast at :108),
 * counts[n_centers] = points per crop, flags[n_centers] = CP_CONE_* bits (image all zero unless flags is 0 or
 * CP_CONE_AMBIGUOUS).  counts / flags may be NULL.  180 bytes per cone travel back instead of the crops. */
cp_status cp_cone_images(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                         uint32_t n_centers, float cone_width, uint8_t* images, uint32_t* counts, uint32_t* flags);
/* to_image alone, on host crops in the cp_cone_crops format (what handle_classify_color receives, :78-90). */
cp_status cp_rasterize_crops(cp_handle* h, const float* crop_xyzi, const uint32_t* crop_offsets, uint32_t n_crops,
                             uint8_t* images, uint32_t* flags);

/* The classifier network of scripts/color_classifier_server.py (models/dam_net/dam_net.tflite, evaluated there
 * by tf.lite.Interpreter, :66-71 and :108-120): conv 3x3 (1 -> c1, ReLU), max-pool 2x2, conv 3x3 (c1 -> c2, ReLU),
 * max-pool 2x2, per-channel scale + shift (the folded batch normalisation), dense (2*c2 -> n_classes), softmax.
 * Tensors in the flatbuffer's own layouts.  PARITY UNPINNED: TensorFlow-Lite cannot be installed next to this
 * library's tests; the implementation is held to a numpy restatement of TFLite's reference kernels and to the
 * human labels of the reference's 577 recorded crops (tests/test_dam_net.py). */
typedef struct cp_color_net {
  uint32_t c1, c2, n_classes; /* dam_net: 16, 32, 3 */
  const float* conv1_w;       /* [c1][3][3][1]   (OHWI) */
  const float* conv1_b;       /* [c1] */
  const float* conv2_w;       /* [c2][3][3][c1] */
  const float* conv2_b;       /* [c2] */
  const float* bn_scale;      /* [c2]  the MUL constant */
  const float* bn_shift;      /* [c2]  the ADD constant */
  const float* dense_w;       /* [n_classes][2 * c2], features in NHWC order */
  const float* dense_b;       /* [n_classes] */
  float threshold;            /* 0.8: below it the colour is 0 = unknown (color_classifier_server.py:116-120) */
} cp_color_net;
cp_status cp_color_net_load(cp_handle* h, const cp_color_net* net);
/* The same from the bytes of the .tflite file the reference's launch parameter ~model_path names.  Any graph other
 * than the architecture above is refused with CP_E_PARAM (cp_last_error says why). */
cp_status cp_color_net_load_tflite(cp_handle* h, const void* data, size_t bytes, float threshold);
/* handle_classify_color (scripts/color_classifier_server.py:78-126) for n_centers cones, entirely on the device:
 * box gather -> to_image -> network.  colors[c]: 0 unknown, 1 yellow, 2 blue, 3 orange, 255 = no answer for this
 * cone (flags[c] has CP_CONE_EMPTY: the service skips it; CP_CONE_BAD_*: the service call would raise).
 * probs (optional) [n_centers][n_classes] softmax outputs; flags (optional) CP_CONE_* bits. */
#define CP_CONE_LOW_CONFIDENCE 16 /* the largest probability lies within 2e-6 of the threshold */
cp_status cp_cone_colors(cp_handle* h, const cp_cloud_view* cloud, uint32_t frame, const cp_cone_center* centers,
                         uint32_t n_centers, float cone_width, uint8_t* colors, float* probs, uint32_t* flags);
/* After a batch run (cp_batch_run, cp_detect_batch or cp_detect): handle_classify_color
 * (scripts/color_classifier_server.py:78-126) for EVERY cluster record of the run, entirely on the device.
 * Cluster k (the k-th record cp_batch_results returns, frame-major, canonical order) is classified at its
 * centroid moved radially by extension_length (src/cone_detection.cpp:276-278, restated exactly), using the
 * raw cloud of its own frame from the run's staged input (or, with CP_COLOR_CLOUD_GROUNDLESS after a run with
 * ground removal, that frame's ground-node message: cp_set_color_cloud).  One pass over the batch finds every crop.
 *   colors[k]: 0 unknown, 1 yellow, 2 blue, 3 orange, 255 no answer (as cp_cone_colors)
 *   probs  (optional) [K][n_classes], flags (optional) CP_CONE_* bits, counts (optional) crop points per cluster.
 * The output is per cluster: the service's response rules (a shorter response when a crop is empty, a failed
 * call when a crop is bad) depend on which cones a node sends, and `flags` holds what is needed to apply them.
 * extension_length is the node parameter cone_position_extension_length (default 0.05).
 * Calls cp_sync first (the final records can come from the back-half retry) and leaves the run's results
 * (cp_batch_results, cp_device_results, the gather slot) untouched.  Device input must stay valid until this
 * call returns.  CP_E_PARAM: non-finite extension_length, cone_width not positive and finite, NULL colors with
 * clusters present.  CP_E_STATE: no run, input re-staged since the run, or no colour net loaded.
 * CP_E_CAPACITY: cap < number of clusters. */
cp_status cp_batch_cone_colors(cp_handle* h, float cone_width, double extension_length, uint8_t* colors,
                               float* probs, uint32_t* flags, uint32_t* counts, uint64_t cap);
/* Which cloud colour crops of the staged input are cut from: cp_cone_crops / cp_cone_images / cp_cone_colors with
 * cloud NULL, cp_batch_cone_colors and cp_batch_track in colour mode.  An explicit cloud argument is used as given.
 *   CP_COLOR_CLOUD_STAGED (the default): the staged cloud itself.
 *   CP_COLOR_CLOUD_GROUNDLESS: when the last run fused ground removal (cp_detect, cp_batch_run or cp_detect_batch
 *     with non-NULL ground), frame f is cropped from the message the ground node publishes for it
 *     (src/ground_removal.cpp:54-79): the points its filter keeps, in input order, then N_f - G_f points (0, 0, 0,
 *     intensity 0).  That is what cp_batch_ground_remove writes for the frame, so the crops, images and colours equal
 *     those of the reference's two-node launch (ground_removal:=true), where the detector crops from the
 *     groundless_cloud message.  Intensities are what the staged view reads: stage clouds without an intensity
 *     field with off_intensity < 0, as the ground node reads them.  After a run without ground removal the output
 *     is the same as with CP_COLOR_CLOUD_STAGED.
 * CP_E_PARAM: any other value.  The colour calls then return CP_E_STATE with CP_COLOR_CLOUD_GROUNDLESS and cloud
 * NULL when no run has been made on the staged input (the sector minima would belong to another input). */
enum { CP_COLOR_CLOUD_STAGED = 0, CP_COLOR_CLOUD_GROUNDLESS = 1 };
cp_status cp_set_color_cloud(cp_handle* h, int32_t cloud);
/* --- what the cone-detection node publishes, over frame sequences (src/cone_detection.cpp:276-340) ---------------
 * After a run (cp_batch_run, cp_detect_batch or cp_detect): the radial extension, the temporal gate / points buffer,
 * the colour carry-over from the previous frame's colour clouds, the colour service's response rules and the four
 * published clouds, for every frame of the run, on the device.
 *   seq_offsets[n_seqs + 1]: the run's frames as contiguous sequences, each a series of consecutive messages to one
 *     node (NULL with n_seqs = 1: the whole run is one sequence).  Sequence s continues the handle's state slot s
 *     (s < cp_config.max_frames): the last frame that slot saw, its extended cones and the colour cloud each was
 *     published in.  A fresh slot (or one cleared by cp_track_reset) is a node that has just started: its first frame
 *     publishes nothing.  An empty sequence leaves its slot unchanged.
 *   out: the published cones, frame-major, then by cloud 0..3 (unknown, yellow, blue, orange); within a cloud the
 *     node's push_back order (cones with a carried colour in record order, then the cones that needed a colour).
 *   cloud_offsets[4 * n_frames + 1]: cloud c of frame f is out[cloud_offsets[4 f + c] .. cloud_offsets[4 f + c + 1]).
 * Colour mode (classify_colors != 0) classifies every record on the device (the chain of cp_batch_cone_colors, on the
 * cloud cp_set_color_cloud selects; needs a loaded net) and applies the service's response rules to each frame's need list: a bad crop (CP_CONE_BAD_*) leaves
 * every needed cone unknown; otherwise the answers of the non-empty crops fill the need list from the front.
 * Calls cp_sync first and leaves the run's results untouched.  No slot changes on any error.
 * CP_E_PARAM: non-finite threshold or extension length, cone_width not positive and finite in colour mode, n_seqs
 * 0 or > max_frames, seq_offsets not a non-decreasing partition of [0, n_frames], NULL cloud_offsets / n_out, NULL
 * out with cones to publish.  CP_E_STATE: no run (or input staged since), no colour net in colour mode, or the run
 * was already tracked.  CP_E_CAPACITY: cap < *n_out (set); cap = number of clusters always suffices. */
typedef struct cp_track_params {
  int32_t classify_colors;               /* node parameter classify_colors                      */
  int32_t use_points_buffer;             /* node parameter use_points_buffer                    */
  double cones_matching_dist_theshold;   /* 0.5 (reference spelling)                            */
  double cone_position_extension_length; /* 0.05                                                */
  float cone_width;                      /* CONE_WIDTH, box of the colour crops (colour mode only) */
} cp_track_params;
typedef struct cp_tracked_cone {
  float x, y;       /* the extended centroid as published (z = 0)                          */
  uint32_t cluster; /* index of its record in the run (cp_batch_results order)             */
  uint32_t color;   /* 0 unknown, 1 yellow, 2 blue, 3 orange: the cloud it is published in  */
} cp_tracked_cone;
cp_status cp_batch_track(cp_handle* h, const cp_track_params* t, const uint32_t* seq_offsets, uint32_t n_seqs,
                         cp_tracked_cone* out, uint32_t* cloud_offsets, uint64_t cap, uint64_t* n_out);
/* Clears every state slot (each behaves like a node that has just started). */
cp_status cp_track_reset(cp_handle* h);
/* Test hook, like cp_debug_sort: the kernels of cp_batch_track on caller-supplied records (record_offsets[n_frames+1],
 * frame-major) and per-record service answers (colors as cp_batch_cone_colors returns them, CP_CONE_* flags; read in
 * colour mode only).  Uses and advances the same state slots; needs no run. */
cp_status cp_debug_track(cp_handle* h, const cp_track_params* t, const cp_cluster* records,
                         const uint32_t* record_offsets, uint32_t n_frames, const uint8_t* colors,
                         const uint32_t* flags, const uint32_t* seq_offsets, uint32_t n_seqs,
                         cp_tracked_cone* out, uint32_t* cloud_offsets, uint64_t cap, uint64_t* n_out);

/* The network alone on host images [n][15][12] uint8 (parity tests; logits optional, before the softmax). */
cp_status cp_classify_images(cp_handle* h, const uint8_t* images, uint32_t n_images, uint8_t* colors, float* probs,
                             float* logits);

/* --- stage taps for parity tests (valid after cp_sync, whole batch, frame-major) ----
 * Every tap copies device state of the last run to host memory.  count = entries written. */
typedef enum cp_tap {
  CP_TAP_SECTOR_LOW = 0,   /* float   [n_frames*17]  per-sector minima                    */
  CP_TAP_CROP_INDEX = 1,   /* uint32  [C_total]  frame-local input index of each survivor */
  CP_TAP_CROP_POINTS = 2,  /* float4  [C_total]  surviving points x,y,z,intensity         */
  CP_TAP_CROP_OFFSETS = 3, /* uint32  [n_frames+1]                                        */
  CP_TAP_VOXEL_KEYS = 4,   /* uint32  [C_total]  sorted PCL voxel idx, with multiplicity  */
  CP_TAP_VOXEL_ORDER = 5,  /* uint32  [C_total]  survivor position of each sorted record  */
  CP_TAP_VOXEL_CLOUD = 6,  /* float4  [V_total]  voxel centroids x,y,z,intensity          */
  CP_TAP_VOXEL_OFFSETS = 7,/* uint32  [n_frames+1]                                        */
  CP_TAP_LABELS = 8,       /* int32   [V_total]  frame-local min voxel index of component */
  /* plane model (cp_set_ground_plane), last run or ground call with it; H = n_hypotheses */
  CP_TAP_PLANE_HYPOTHESES = 9, /* float4 [n_frames*H]  a, b, c, d of every hypothesis, NaN when invalid */
  CP_TAP_PLANE_COUNTS = 10     /* uint32 [n_frames*H]  inliers of every hypothesis                     */
} cp_tap;
cp_status cp_debug_tap(cp_handle* h, cp_tap which, void* out, uint64_t cap_bytes, uint64_t* count);

/* Stand-alone exercise of the radix sort used inside the pipeline (tests only):
 * sorts n (key, value) pairs on the device by the low `bits` bits of the key, stably. */
cp_status cp_debug_sort(cp_handle* h, uint64_t* keys, uint32_t* vals, uint32_t n, uint32_t bits);

#ifdef __cplusplus
}
#endif
#endif
