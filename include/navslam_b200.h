/*
 * navslam_b200.h -- C ABI of libnavslam_b200.so, the sm_100a CUDA implementation of
 * NAV-SLAM's data-parallel front end (reference: wuHakureReimu/NAV-SLAM).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  The
 * image shape is a run-time argument here; the reference bakes MAX_ROWS/MAX_COLS into
 * its signatures (utils/pointcloud.h:9-10), so the symbols the reference's main.c binds
 * (init_slam, slam_localization, slam_mapping, convertToPointCloud, buildKDTree, ...) are
 * exported with byte-identical signatures by the per-shape shim built from
 * nav-slam_b200/shim/navslam_shim.c on top of this library (see include/navslam_ref_abi.h
 * and INTEGRATION.md).
 *
 * Conventions
 *   - every function returning int returns 0 on success, non-zero on failure;
 *     nav_last_error() then describes the failure (thread-local).  There is no CPU
 *     fallback anywhere: without a CUDA device nav_create()/nav_kdtree_build() fail.
 *   - "host" arguments are ordinary host pointers (pageable or pinned; pinned memory,
 *     e.g. from nav_host_alloc, is DMA'd directly, pageable memory is staged).
 *     "dev" arguments are device pointers on the context's device.
 *   - points are the reference's `Point` (3 x double, 24 B, utils/pointcloud.h:39-44),
 *     clouds are row-major [rows][cols] arrays of points WITHOUT the 8-byte PointCloud
 *     header (pass &cloud->ToF_position[0][0]).
 *   - labels are the reference's `int feature[rows][cols]` (src/slam.c:11): 1 = edge.
 *   - nearest-neighbour answers are exact: idx = the LOWEST index among the points that
 *     attain the minimum of dsq = (dx*dx + dy*dy) + dz*dz evaluated in binary64 without
 *     FMA (the reference's arithmetic, utils/kdtree.c:14-17), dist = sqrt(dsq).  The
 *     reference returns the first such point its DFS visits (utils/kdtree.c:117); the two
 *     differ only when two distinct points are at exactly the same distance.
 */
#ifndef NAVSLAM_B200_H
#define NAVSLAM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { double x, y, z; } nav_point;                          /* Point,  utils/pointcloud.h:39-44 */
typedef struct { double x, y, z, roll, pitch, yaw; } nav_pos;          /* Pos (mm, degrees), utils/pointcloud.h:32-35 */
typedef struct { nav_point ori, nearest; double distance; } nav_corr;  /* NeighborResult, utils/kdtree.h:14-18 */

typedef struct nav_ctx nav_ctx;       /* one image shape on one device */
typedef struct nav_kdtree nav_kdtree; /* device-resident flat kd-tree  */

/* ---- library ------------------------------------------------------------------- */
const char *nav_version(void);
const char *nav_last_error(void);
int nav_device_count(void);          /* 0 when no CUDA device is usable */
void *nav_host_alloc(size_t bytes);  /* pinned host memory (cudaHostAlloc) */
void nav_host_free(void *p);
/* page-lock / release memory the caller already owns (cudaHostRegister): pinned buffers are DMA'd directly */
int nav_host_register(void *p, size_t bytes);
int nav_host_unregister(void *p);

/* ---- context ------------------------------------------------------------------- */
/* n_seq = number of independent sequences processed side by side (1..NAV_MAX_SEQ);
 * every cloud/label/global argument of the frame calls below then holds n_seq images
 * back to back.  Returns NULL on failure (no device, shape unsupported). */
#define NAV_MAX_SEQ 16
nav_ctx *nav_create(int rows, int cols, int device, int n_seq);
void nav_destroy(nav_ctx *ctx);
int nav_rows(const nav_ctx *ctx);
int nav_cols(const nav_ctx *ctx);
/* use_own != 0: back to the context's own non-blocking stream; otherwise run on the caller's
 * cudaStream_t (0 = the legacy default stream) */
int nav_set_stream(nav_ctx *ctx, void *cuda_stream, int use_own);
int nav_synchronize(nav_ctx *ctx);
/* number of kernels this library has launched on behalf of ctx since creation */
uint64_t nav_launch_count(const nav_ctx *ctx);

/* ---- function-level mirrors, HOST buffers (one image each) ------------------------ */
/* replaces convertToPointCloud, utils/pointcloud.c:8 (utils/pointcloud.h:55) */
int nav_convert_to_pointcloud(nav_ctx *ctx, const int *distances, nav_point *cloud_out);
/* replaces extract_feature, src/slam.c:11: sets feature[i]=1 where curvature > 0.1, never writes 0 */
int nav_extract_feature(nav_ctx *ctx, const nav_point *cloud, int *feature);
/* the curvature extract_feature thresholds (binary64, reference association order); 0 on the
 * two border columns each side.  The reference does not return it; exposed for parity tests. */
int nav_curvature(nav_ctx *ctx, const nav_point *cloud, double *curvature_out);
/* replaces flattenPoints, src/slam.c:64: stable compaction of one row where row_feature == 1 */
int nav_flatten_points(nav_ctx *ctx, const nav_point *row_points, const int *row_feature,
                       nav_point *flattened_out, size_t *num_points_out);
/* the per-point rigid transform of src/slam.c:145-160,402-416: out = pos.xyz + R(pos.rpy deg) * p */
int nav_transform_cloud(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos, nav_point *global_out);

/* ---- kd-tree, replaces utils/kdtree.h:21-27 ---------------------------------------- */
/* Build from n host points (the caller's array is NOT permuted; idx refers to it). */
nav_kdtree *nav_kdtree_build(int device, const nav_point *points, size_t n);
/* the *_dev entry points run on the given cudaStream_t (0 = legacy default stream) and do not synchronise */
nav_kdtree *nav_kdtree_build_dev(int device, const void *dev_points, size_t n, void *cuda_stream);
/* Split rule of the build.  CYCLIC: axis = depth % 3 as utils/kdtree.c:72 -- with distinct coordinates
 * the exported tree is the reference's tree node for node.  WIDEST (what the two builders above use):
 * every node splits the axis of largest extent of its points; same answers from every query (the search
 * is exact either way), 4x faster searches on maps made of surfaces (profiles/README.md).
 * points_on_device = 0: host points, own stream, synchronised; 1: device points on cuda_stream. */
#define NAV_KD_SPLIT_CYCLIC 0
#define NAV_KD_SPLIT_WIDEST 1
nav_kdtree *nav_kdtree_build_ex(int device, const void *points, size_t n, int points_on_device,
                                void *cuda_stream, int split_rule);
void nav_kdtree_free(nav_kdtree *tree);
size_t nav_kdtree_size(const nav_kdtree *tree);
/* batched exact 1-NN.  idx[i] = -1 and dist[i] = +inf for an empty tree.  nearest_out may be NULL. */
int nav_kdtree_nn_batch(nav_kdtree *tree, const nav_point *queries, size_t nq,
                        int32_t *idx_out, double *dist_out, nav_point *nearest_out);
int nav_kdtree_nn_batch_dev(nav_kdtree *tree, const void *dev_queries, size_t nq,
                            void *dev_idx_out, void *dev_dist_out, void *cuda_stream);

/* ---- config 5b over peer memory ------------------------------------------------------------------
 * Queries sharded across the GPUs of one node against a replicated tree (BASELINE config 5): every rank's search
 * kernel stores its shard's answers directly into the result buffers of all ranks (CUDA IPC mappings, NVLink
 * stores) -- the all-gather is the kernel's epilogue, no collective follows.  One process per GPU:
 *   p = nav_peer_create(device, nq_total, my_handle);            exchange the 64-byte handles (any transport)
 *   nav_peer_connect(p, world, rank, all_handles);
 *   nav_kdtree_nn_allgather_dev(tree, p, my_queries, q_lo, n_mine, &idx, &dist, stream);   per frame
 * idx / dist (device pointers into this rank's buffer) hold the answers of ALL queries once the stream has
 * passed the call; they stay valid until the call after the next one.  world <= 8. */
typedef struct nav_peer nav_peer;
/* contiguous shard [lo, hi) of rank `rank` of n items (the first n % world ranks hold one more), and its inverse */
void nav_shard_range(int64_t n, int world, int rank, int64_t *lo, int64_t *hi);
int nav_shard_owner(int64_t n, int world, int64_t i);
nav_peer *nav_peer_create(int device, size_t nq_total, unsigned char handle_out[64]);
int nav_peer_connect(nav_peer *p, int world, int rank, const unsigned char *handles /* world x 64 bytes */);
int nav_kdtree_nn_allgather_dev(nav_kdtree *tree, nav_peer *p, const void *dev_queries, size_t q_lo, size_t nq_shard,
                                void **idx_full, void **dist_full, void *cuda_stream);
/* The MAP sharded instead of the queries (a map that is rebuilt every frame costs each of N ranks the build of
 * 1/N of it): `tree` holds this rank's part of the points, idx_offset the index of its first point in the whole
 * map; dev_queries are ALL nq queries (the same on every rank).  Partial answers go to the rank that owns the
 * query, the owners take the minimum (squared distance, index) -- the pair a search of the whole map keeps -- and
 * deliver it to every rank: two rounds over peer memory.  Same results as one tree over all points. */
int nav_kdtree_nn_sharded_map_dev(nav_kdtree *tree, nav_peer *p, const void *dev_queries, size_t nq, int64_t idx_offset,
                                  void **idx_full, void **dist_full, void *cuda_stream);
int nav_peer_check(nav_peer *p);   /* after a synchronisation: did every rank deliver every call? */
void nav_peer_destroy(nav_peer *p);
/* exact brute force on the same contract.  use_tensor_cores == 0: plain binary64 scan.
 * use_tensor_cores != 0: tcgen05 candidate tiles (bf16 hi/mid/lo splits, fp32 accumulate in TMEM) flag
 * every 32-point group that can contain the nearest neighbour, then an exact binary64 re-rank of the
 * flagged groups; same answers for any input.  Inputs whose centred coordinates could overflow the fp32
 * operands are answered by the binary64 re-rank of every group.  Measured on B200 it beats the fp64
 * scan from ~4 K points but never the kd-tree (profiles/README.md), so nothing selects it automatically. */
int nav_bruteforce_nn_batch_dev(int device, const void *dev_points, size_t n, const void *dev_queries,
                                size_t nq, void *dev_idx_out, void *dev_dist_out,
                                int use_tensor_cores, void *cuda_stream);
/* copy the flat node array out for inspection: nodes_out[n] points in storage (in-order) layout,
 * orig_idx_out[n] their indices in the build input, axis_out[n] (may be NULL) their split axes */
int nav_kdtree_export(nav_kdtree *tree, nav_point *nodes_out, int32_t *orig_idx_out, int32_t *axis_out);
uint64_t nav_kdtree_launch_count(const nav_kdtree *tree);

/* ---- SLAM step, HOST buffers; replaces headers/slam.h:22-28 -------------------------- */
/* init_slam (src/slam.c:134): global_out = pose(cloud); builds the per-row map of frame 0. */
int nav_slam_init(nav_ctx *ctx, const nav_pos *pos, const nav_point *cloud, nav_point *global_out);
/* the matching half of slam_localization (src/slam.c:180-284): labels, query transform, per-row
 * exact NN against the previous frame's labelled points, per-row dedupe.  corr_out receives up to
 * corr_cap entries in the reference's order; *n_corr_out the number found. */
int nav_slam_match(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos_predict,
                   const nav_pos *pos_last, nav_corr *corr_out, size_t corr_cap, size_t *n_corr_out);
/* whole slam_localization (src/slam.c:178-390): nav_slam_match + the reference's 200-iteration
 * translation-only Adam fit on the host.  verbose != 0 prints the reference's per-iteration lines. */
int nav_slam_localization(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos_predict,
                          const nav_pos *pos_last, nav_pos *pos_out, double *error_out, int verbose);
/* The same step with the fit driven by five sufficient statistics reduced on the device (N, sum r,
 * sum |r|^2 with r = ori - nearest; SURVEY 8f #2): nothing but 40 bytes comes back and each of the 200
 * iterations is O(1).  Sums are formed in a different order than the reference's sequential loop, so
 * the pose agrees with nav_slam_localization to rounding (about 1e-9 relative), not bit for bit.  The sums
 * are formed in a fixed order (deterministic).  cloud may be a frame queued by nav_slam_prefetch, or NULL
 * for the oldest prefetched frame. */
int nav_slam_localization_fast(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos_predict,
                               const nav_pos *pos_last, nav_pos *pos_out, double *error_out, size_t *n_corr_out);
/* the five totals {N, sum rx, sum ry, sum rz, sum |r|^2} the last nav_slam_localization_fast call, or the last
 * frame of nav_slam_run, was fitted from (r = ori - nearest of each dedupe winner).  Fails if no such fit has
 * completed on this context. */
int nav_slam_fit_stats(nav_ctx *ctx, double out[5]);
/* slam_mapping (src/slam.c:393): global_out = pose(cloud), per-row map for the next frame.
 * cloud == NULL reuses the cloud (and labels) of the preceding nav_slam_match/localization call; with
 * global_out == NULL as well the call only queues the map kernel and does not synchronise. */
int nav_slam_mapping(nav_ctx *ctx, const nav_pos *pos, const nav_point *cloud, nav_point *global_out);
/* one front-end frame with raw per-pixel outputs (SURVEY 8d "one frame of work"): labels, queries,
 * NN vs the previous frame, then mapping with pos_final.  nn_idx = flat pixel (row*cols+col) of the
 * match in the previous frame, -1 if unlabelled or the row's map is empty; nn_dist = -1 if
 * unlabelled, +inf if the map is empty.  A labelled point whose dsq to every map point of its row is
 * +inf or NaN (a diverged pose) gets the outcome of an empty row: nn_idx = -1, nn_dist = +inf, and the
 * closed loop makes no correspondence for it.  Any output pointer may be NULL. */
int nav_frontend_frame(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos_predict,
                       const nav_pos *pos_last, const nav_pos *pos_final, int *feature_out,
                       int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out);

/* nav_frontend_frame for L5-type input (SURVEY 8f #3): takes the depth matrix of
 * utils/pointcloud.h:13-17 (int mm, rows x cols) instead of the cloud; convertToPointCloud
 * (utils/pointcloud.c:8) runs on the device in front of the frame kernel, so 4 B/pixel cross PCIe
 * instead of 24.  cloud_out (optional) receives the converted lidar-frame cloud. */
int nav_frontend_frame_depth(nav_ctx *ctx, const int *distances, const nav_pos *pos_predict,
                             const nav_pos *pos_last, const nav_pos *pos_final, nav_point *cloud_out,
                             int *feature_out, int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out);

/* Pipelined variant of nav_frontend_frame for streams of frames: returns immediately; the upload of
 * this frame, the kernels of the previous one and the downloads of the one before overlap on three
 * CUDA streams.  All host pointers must be pinned (nav_host_alloc / cudaHostRegister).  The outputs
 * of a frame are complete after nav_frontend_wait(), or once two further frames have been queued
 * (use distinct output buffers for consecutive frames).  If the four output buffers are adjacent in
 * host memory in the order feature | nn_idx | nn_dist | global they are filled by a single copy. */
int nav_frontend_frame_async(nav_ctx *ctx, const nav_point *cloud, const nav_pos *pos_predict,
                             const nav_pos *pos_last, const nav_pos *pos_final, int *feature_out,
                             int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out);
int nav_frontend_wait(nav_ctx *ctx);

/* General form of the pipelined call.  Exactly one of cloud / distances is the input: `distances` is the L5
 * depth matrix of utils/pointcloud.h:13-17 (int mm, rows x cols, n_seq == 1), converted on the device
 * (utils/pointcloud.c:8) -- 4 B/pixel cross PCIe instead of 24.  Every output is optional.  mask_out returns
 * the labels as bit masks, uint32 [n_seq][rows][ceil(cols/16)], bit i (i < 16) of word b = label of column
 * 16*b + i: 32 KB instead of the 512 KB of feature_out at 64x2048.  cloud_out (depth input only) receives
 * the converted lidar-frame cloud.  Adjacent host buffers feature_out | nn_idx_out | nn_dist_out (or
 * nn_idx_out | nn_dist_out when feature_out is NULL) are filled by a single copy. */
typedef struct {
    const nav_point *cloud;
    const int *distances;
    nav_point *cloud_out;
    int *feature_out;
    uint32_t *mask_out;
    int32_t *nn_idx_out;
    double *nn_dist_out;
    nav_point *global_out;
} nav_frame_io;
int nav_frontend_submit(nav_ctx *ctx, const nav_frame_io *io, const nav_pos *pos_predict,
                        const nav_pos *pos_last, const nav_pos *pos_final);
/* nav_frontend_frame_depth, pipelined (src/main.c:194-197,308: depth -> xyz -> SLAM step per frame) */
int nav_frontend_frame_depth_async(nav_ctx *ctx, const int *distances, const nav_pos *pos_predict,
                                   const nav_pos *pos_last, const nav_pos *pos_final, nav_point *cloud_out,
                                   int *feature_out, int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out);

/* Closed loop with pose feedback (src/main.c:300-318): localization(t) needs pose(t-1) and mapping(t) needs
 * pose(t), but the upload of frame t+1 and its labels (src/slam.c:11, pose independent) need neither.
 * nav_slam_prefetch queues both on a copy stream and returns at once; a later
 * nav_slam_localization_fast(ctx, cloud, ...) with the same `cloud` pointer (or NULL = the oldest prefetched
 * frame) finds the frame resident and labelled and only runs match + dedupe + statistics (2.5 KB come back).
 * nav_slam_mapping(ctx, pos, NULL, NULL) then maps that frame without synchronising.  There are three prefetch
 * slots, and the frame a localization call consumed keeps its slot until nav_slam_mapping has queued its
 * map: up to three frames may wait ahead of the next localization call, two while a consumed frame still
 * waits for its mapping (a prefetch into that slot is refused).  The host buffer must be pinned and stay
 * untouched until the localization call that consumes it returns.
 *     nav_slam_prefetch(ctx, frame[1]);
 *     for (t = 1; t < n; ++t) {
 *         if (t + 1 < n) nav_slam_prefetch(ctx, frame[t + 1]);
 *         nav_slam_localization_fast(ctx, frame[t], &predict, &last, &pose, &err, NULL);
 *         nav_slam_mapping(ctx, &pose, NULL, NULL);
 *     }
 * Poses are identical to the same calls without prefetch. */
int nav_slam_prefetch(nav_ctx *ctx, const nav_point *cloud);
/* the same for L5 input: uploads the depth matrix and converts it on the device; consume it with
 * nav_slam_localization_fast(ctx, NULL, ...) */
int nav_slam_prefetch_depth(nav_ctx *ctx, const int *distances);
/* The loop above as one call (src/main.c:300-318 with the EKF's prediction supplied by the caller): for
 * t = 0 .. n_frames-1: pred = predict(user, t, &last) -- or last + deltas[t] when predict is NULL --,
 * poses_out[t] = nav_slam_localization_fast(frames[t], pred, last), nav_slam_mapping(poses_out[t]),
 * last = poses_out[t]; `last` starts as *pos_start (the pose nav_slam_init mapped frame -1 with).
 * frames[t]: pinned nav_point[rows*cols] clouds, or pinned int[rows*cols] depth matrices when depth_input != 0.
 * error_out / n_corr_out: optional per-frame RMS residual and correspondence count.  Same poses as the
 * separate calls. */
typedef void (*nav_predict_fn)(void *user, int t, const nav_pos *last, nav_pos *pred_out);
int nav_slam_run(nav_ctx *ctx, const void *const *frames, int n_frames, int depth_input, nav_predict_fn predict,
                 void *user, const nav_pos *deltas, const nav_pos *pos_start, nav_pos *poses_out, double *error_out,
                 size_t *n_corr_out);

/* ---- data formats either side of the path (host code; SURVEY 8f #3, #4) ----------------- */
/* replaces L9_LidarProcessData (src/main.c:77-128): parses "frame,row,col,x,y,z,conf" records after one
 * header line into frames_out[max_frames][rows][cols] (use nav_host_alloc memory to make the frames a
 * DMA source); a change of the frame number starts the next frame; records outside the image are
 * skipped.  Pixels that no record names keep whatever frames_out held (the reference leaves its stack
 * array uninitialised there).  Same values as fscanf("%lf") bit for bit. */
int nav_l9_csv_read(const char *path, int rows, int cols, size_t max_frames, nav_point *frames_out,
                    int *timestamps_out, size_t *n_frames_out);
/* replaces LidarProcessData (src/main.c:12-75): `parsed_data.json`, a top-level array whose elements are
 * objects {"time_main": integer, "distance": [integers, row-major], ...}.  Every array element is one
 * frame; integer distances with index < rows*cols are stored, everything else of distances_out keeps
 * its previous content (the reference leaves its stack array uninitialised there).  The document must
 * be valid JSON, otherwise nothing is read (as with jansson's json_loadf). */
int nav_l5_json_read(const char *path, int rows, int cols, size_t max_frames, int *distances_out,
                     int *timestamps_out, size_t *n_frames_out);
/* replaces IMUProcessData (src/main.c:130-178): "params": [roll, pitch, yaw, x, y, z] of every object of
 * the same file into params_out[frame][6]; like json_real_value(), an element written as an integer
 * reads as 0.0.  Only objects count as frames. */
int nav_imu_json_read(const char *path, size_t max_frames, double *params_out, int *timestamps_out,
                      size_t *n_frames_out);
/* the header line of point_cloud_data.csv (src/main.c:243) */
const char *nav_csv_header(void);
/* replaces the per-frame fprintf loop of src/main.c:320-352 (L5) / :433-464 (L9): rows*cols lines
 * "%zu,%d,%d,%.2f,%.2f,%.2f,%d" + 18 pose columns "%.2f", byte-identical to glibc's printf.
 * distances / imu / ekf_pos may be NULL (printed as 0 / 0.00).  Returns the bytes written, 0 if cap is
 * too small (340 B per line always suffices for finite data below 1e300). */
size_t nav_csv_format_frame(char *buf, size_t cap, unsigned long long timestamp, int rows, int cols,
                            const nav_point *global_cloud, const int *distances, const double imu[6],
                            const nav_pos *lidar_pos, const nav_pos *ekf_pos);

/* The same text produced on the GPU (three small kernels: line lengths, prefix sum, format into shared
 * memory + coalesced store).  global_cloud == NULL formats the context's resident global cloud of the
 * frame mapped last (no upload at all); distances == NULL prints 0.  buf should be pinned memory
 * (nav_host_alloc).  Frames holding inf / nan / |v| >= 2^57 are formatted by nav_csv_format_frame on
 * the host instead -- identical bytes either way.  Returns 0 and *n_bytes_out, 1 on failure. */
int nav_csv_format_frame_gpu(nav_ctx *ctx, unsigned long long timestamp, const nav_point *global_cloud,
                             const int *distances, const double imu[6], const nav_pos *lidar_pos,
                             const nav_pos *ekf_pos, char *buf, size_t cap, size_t *n_bytes_out);
/* Device-resident variant: d_global_cloud (NULL = resident cloud), d_distances (NULL = 0) and d_text are
 * device pointers; cap >= rows*cols*(124 + length of the 18 pose columns) (rows*cols*604 always
 * suffices).  Synchronises the context's stream to report *n_bytes_out.  Returns 2 when the frame
 * needs the host formatter (see above); d_text is then undefined. */
int nav_csv_format_frame_dev(nav_ctx *ctx, unsigned long long timestamp, const nav_point *d_global_cloud,
                             const int *d_distances, const double imu[6], const nav_pos *lidar_pos,
                             const nav_pos *ekf_pos, char *d_text, size_t cap, size_t *n_bytes_out);

/* ---- device-resident entry points (inputs already in HBM) ------------------------------ */
/* labels for n_images images [n_images][rows][cols] in one launch (pose independent) */
int nav_extract_feature_batch_dev(nav_ctx *ctx, const void *dev_clouds, size_t n_images,
                                  void *dev_labels_out);
/* nav_frontend_frame on device data: dev_cloud holds n_seq images; poses are n_seq-long host arrays;
 * results stay in the context (nav_frame_results_dev) */
int nav_frontend_frame_dev(nav_ctx *ctx, const void *dev_cloud, const nav_pos *pos_predict,
                           const nav_pos *pos_last, const nav_pos *pos_final);
int nav_slam_init_dev(nav_ctx *ctx, const void *dev_cloud, const nav_pos *pos);
/* replay of a recorded sequence with known poses: n_frames consecutive frames (each n_seq images) at
 * dev_frames, pose arrays of n_frames*n_seq entries; equivalent to n_frames nav_frontend_frame_dev
 * calls (frame f is matched against frame f-1), issued from one host call */
int nav_frontend_sequence_dev(nav_ctx *ctx, const void *dev_frames, size_t n_frames, const nav_pos *pos_predict,
                              const nav_pos *pos_last, const nav_pos *pos_final);
typedef struct {
    void *labels;   /* int32  [n_seq][rows][cols] */
    void *nn_idx;   /* int32  [n_seq][rows][cols] */
    void *nn_dist;  /* double [n_seq][rows][cols] */
    void *global;   /* point  [n_seq][rows][cols] */
    void *map_mask; /* uint32 [n_seq][rows][ceil(cols/16)] edge-point bit masks of the frame just mapped */
} nav_frame_results;
int nav_frame_results_dev(nav_ctx *ctx, nav_frame_results *out);

/* copy out the map the context holds for one (sequence,row): the labelled global points of the
 * frame mapped last, compacted in column order (= the flattenedPoints array of src/slam.c:170-171),
 * and the column each came from.  pts_out needs room for cols points; col_out may be NULL. */
int nav_row_map_export(nav_ctx *ctx, int seq, int row, nav_point *pts_out, int32_t *col_out, size_t *n_out);

/* how many labels the fp32 filter of the curvature stencil could not decide and re-evaluated with
 * the reference's exact binary64 arithmetic since the context was created (statistics only) */
uint64_t nav_exact_fallback_count(nav_ctx *ctx);

/* per-kernel device time accumulated with CUDA events on the context's stream (enable first) */
int nav_profile_enable(nav_ctx *ctx, int on);
/* name = "labels" | "match" | "map"; returns accumulated ms and launches since the last reset */
int nav_profile_read(nav_ctx *ctx, const char *name, double *ms_out, uint64_t *launches_out, int reset);

#ifdef __cplusplus
}
#endif
#endif
