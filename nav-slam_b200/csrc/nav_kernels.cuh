// nav_kernels.cuh -- launch wrappers shared between the .cu files of libnavslam_b200.
#pragma once
#include "nav_common.cuh"

namespace nav {

// ---- stencil.cu
void launch_labels(const double *cloud, int *labels, double *curv_or_null, long long n_rows, int cols,
                   int sm_count, unsigned *n_exact, cudaStream_t stream);
// depth matrices of n_img images [n_img][rows][cols] -> xyz clouds (a2)
void launch_convert(const int *dist, const double *tan_col, const double *tan_row, double *out, int rows,
                    int cols, int n_img, int sm_count, cudaStream_t stream);
// int32 [n_points][3] (whole millimetres) -> double [n_points][3], exact
void launch_widen_mm(const int *in, double *out, long long n_points, int sm_count, cudaStream_t stream);
void launch_transform(const double *in, double *out, long long n, const PoseXf &pose, int sm_count,
                      cudaStream_t stream);

// ---- rowmap.cu : the per-row "tree" of the SLAM step
// Device-resident state of one context: the mapped (global-frame) cloud of the previous frame, left
// in image order, plus per 16-column block a label mask and a bounding box of its labelled points,
// and per 256-column block a super box.
struct RowMap {
    double *pts;      // [n_seq*rows][cols][3]   global cloud of the frame mapped last
    unsigned *mask;   // [n_seq*rows][n_chunks]  bit i = column 16*b+i is an edge point
    float4 *box;      // [n_seq*rows][n_chunks][2]   {lo.xyz,-}, {hi.xyz,-} rounded outward (+inf/-inf when empty)
    float4 *sbox;     // [n_seq*rows][n_super][2]
    int n_chunks, n_super;
};

struct MatchOut {
    int *nn_idx;          // [n_seq*rows][cols]
    double *nn_dist;      // [n_seq*rows][cols]
    nav_corr *corr_rows;  // [n_seq*rows][cols]  per-row deduped correspondences
    int *corr_row_count;  // [n_seq*rows]
};

// where k_dedupe_rows posts the fit statistics of a whole frame for the host to poll (closed loop):
// host[0..4] = {N, sum rx, sum ry, sum rz, sum |r|^2}, host[5] = seq (written last, as a 64-bit word)
struct FitMailbox {
    double *host;       // host-mapped pinned memory, 6 doubles
    unsigned *ticket;   // device counter of finished row CTAs (zero between launches)
    unsigned long long seq;
};

// a whole sequence of frames with known poses in one launch (one thread-block cluster per image row walks
// through the frames); map0 is searched by frame 0, frame f builds the map for frame f+1 in the other buffer.
// d_pose_loc / d_pose_fin: device arrays [n_frames][n_seq].  Needs row_cluster_supported(cols).
// seq_out (optional): per-frame outputs -- slot f of every non-null ring receives frame f (nav_sequence_out), and
// part != null adds the statistics dedupe, CTA partials [n_frames][n_seq*rows*tiles][5] for launch_seq_fit_totals.
// kind (NAV_RUN_INPUT_*): frames of xyz doubles, frame_stride in doubles; or depth matrices / integer-mm clouds
// (int32, 1 or 3 per pixel), frame_stride in int32, converted inside the kernel (depth with the context's tan tables).
int frame_seq_inline_frames();  // sequences up to this length (one sequence) carry their poses as kernel parameters
// the context's tan tables of a2 (device memory: tan of every column, of every image row), for depth frames
struct TanTables {
    const double *col, *row;
};
struct SeqOut {
    unsigned *mask;   // [n_frames][n_seq*rows][n_chunks]
    int *nn_idx;      // [n_frames][n_seq*rows][cols]
    double *nn_dist;  // [n_frames][n_seq*rows][cols]
    double *part;     // [n_frames][n_seq*rows*tiles][5]
};
int launch_frame_seq(int kind, const void *frames, long long frame_stride, int n_frames, int *labels, const RowMap &map0,
                     const RowMap &map1, const MatchOut &out, const PoseXf *d_pose_loc, const PoseXf *d_pose_fin,
                     int n_seq, int rows, int cols, unsigned *n_exact, cudaStream_t stream, const PoseXf *h_pose_loc,
                     const PoseXf *h_pose_fin, const SeqOut *seq_out, bool *bulk_out,  // *bulk_out: staged by bulk copies
                     const TanTables &tan);
// fit totals stats[f][s][0..4] of the partials part[f][s][n_part][5], in the closed loop's summation order:
// row_partials = false for tile partials (k_frame_seq, k_dedupe_stats), true for row totals (k_dedupe_rows)
void launch_seq_fit_totals(const double *part, bool row_partials, int n_part, int n_frames, int n_seq, double *stats,
                           cudaStream_t stream);

size_t dedupe_smem_bytes(int cols);
int configure_row_kernels(int cols);  // opt in to large dynamic shared memory; 0 on success

void launch_frame_map(const double *cloud, const int *labels, const RowMap &map, const PoseBatch &poses,
                      int n_seq, int rows, int cols, cudaStream_t stream);
// The queries of a frame search whose smallest rounded distance sqrt(dsq) is reached by at least two map points
// of the row (the reference tie rule resolves them on the host): one record per query, appended in any order.
struct TieRec {
    long long px;  // flat pixel (sequence * rows + row) * cols + column
    double q[3];   // the query exactly as the search used it
};
struct TieList {
    TieRec *rec;      // capacity: one record per pixel of the context
    unsigned *count;  // zeroed before the launch
};

// map_next/final_poses non-null: the kernel also builds the next map (frame transformed with its final
// pose) into *map_next, which must be a different buffer than `map`.  ties non-null (fused labels only): the
// search also lists its tied queries there.
void launch_frame_match(const double *cloud, int *labels, bool fused_labels, const RowMap &map,
                        const MatchOut &out, const PoseBatch &poses, int n_seq, int rows, int cols,
                        unsigned *n_exact, cudaStream_t stream, const RowMap *map_next = nullptr,
                        const PoseBatch *final_poses = nullptr, bool pdl = false, const TieList *ties = nullptr);
// nn_idx[fix[i].x] = fix[i].y for i < n (the host's answers for tied queries)
void launch_apply_tie_fix(const int2 *fix, int n, int *nn_idx, cudaStream_t stream);
// row_stats (optional): [n_seq*rows][5] per-row {n, sum r (3), sum |r|^2} of the deduped correspondences;
// write_corr = false skips the correspondence entries themselves
void launch_dedupe(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                   const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream,
                   double *row_stats = nullptr, bool write_corr = true, const FitMailbox *mail = nullptr);
// whether the tiles of a row fit one thread-block cluster, as launch_frame_seq, launch_dedupe_stats and
// launch_loop_step need (rows up to 2048 columns)
bool row_cluster_supported(int cols);
// statistics-only dedupe spread over the tiles of a row (thread-block cluster per row); part: [n_seq*rows*tiles][5]
int launch_dedupe_stats(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                        const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream, double *part,
                        const FitMailbox &mail);
// the closed-loop step in one launch: (do_map) map of the previous frame from prev_cloud / prev_labels /
// prev_poses, match of this frame against it, statistics dedupe, mailbox post.  Needs row_cluster_supported(cols).
int launch_loop_step(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                     const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream,
                     const double *prev_cloud, const int *prev_labels, const PoseBatch &prev_poses, bool do_map,
                     double *part, const FitMailbox &mail);

// The closed loop on device-resident frames (nav_slam_run_dev): the same k_loop_step, its poses read from a device
// record per sequence that the previous launch's fit wrote.  What the host knows up front, per frame and sequence:
struct LoopTab {
    double Rq[9];   // rotation of the prediction (query pose)
    double Rm[9];   // rotation of the fitted pose (map pose)
    double rpy[3];  // roll, pitch, yaw of the fitted pose: last + (pred - last), the fit never moves them
    double d[3];    // deltas[t].xyz: pred.xyz = last.xyz + d
};
// the device pose record of one sequence: this frame's query pose (R from the table, t = pred.xyz, shift =
// pred.xyz - last.xyz, as make_pose forms it) and the previous frame's map pose (t = last.xyz, shift 0)
struct LoopRec {
    PoseXf loc, map;
};
struct DevLoop {
    int t, n_frames, n_seq;
    int do_match;              // 0: the launch after the last frame, which only maps it
    int *labels_out;           // this frame's labels (the next launch maps the frame with them)
    const LoopRec *rec_in;     // [n_seq] poses of frame t
    LoopRec *rec_out;          // [n_seq] poses of frame t+1, written by the fit (a different buffer)
    const LoopTab *tab;        // [n_frames][n_seq]
    unsigned *ticket;          // [n_seq] finished CTAs of each sequence (zero between launches)
    unsigned *n_exact;
    nav_pos *poses;            // [n_frames][n_seq]
    double *error;             // [n_frames][n_seq] or null
    double *fit_stats;         // [n_frames][n_seq][5] or null
};
// launch t of the device loop: cloud = frame t, prev_cloud / prev_labels = frame t-1 (do_map); part: the CTA partials
// [n_seq*rows*tiles][5].  Needs row_cluster_supported(cols) and the fit tables (upload_fit_tables).
// kind (NAV_RUN_INPUT_*): cloud / prev_cloud are xyz doubles, or depth / integer-mm int32 converted in the kernel.
int launch_loop_step_dev(int kind, const DevLoop &dl, const void *cloud, const void *prev_cloud, const int *prev_labels,
                         bool do_map, const RowMap &map, const MatchOut &out, int n_seq, int rows, int cols,
                         double *part, cudaStream_t stream, const TanTables &tan);
// the fit's bias tables (1 - beta^t, formed on the host) into the device's constant memory, queued on `stream`
int upload_fit_tables(const double *c1, const double *c2, cudaStream_t stream);
// fit_translation on the device, one thread per stat vector (nav_debug_fit_from_stats_dev)
void launch_fit_debug(const double *stats, const nav_pos *pred, const nav_pos *last, size_t n, nav_pos *pose_out,
                      double *err_out, cudaStream_t stream);
void launch_gather_corr(const nav_corr *corr_rows, const int *corr_row_count, nav_corr *corr_out,
                        int *corr_total, int n_seq, int rows, int cols, cudaStream_t stream);
void launch_flatten_row(const double *row_pts, const int *row_feature, const unsigned *row_mask, double *out,
                        int *col_out, int *count, int cols, cudaStream_t stream);

// ---- csvfmt.cu : CSV rows of one frame formatted on the device (src/main.c:320-352)
struct CsvJob {
    const double *cloud;  // [n][3] global cloud
    const int *dist;      // [n] or null (prints 0)
    unsigned long long ts;
    long long n;
    int cols, ts_len, tail_len;
    char tail[480];  // ",%.2f" x 18 + "\n", the same on every line (formatted on the host)
};
size_t csv_scratch_bytes(long long n);
// writes the text to d_text (needs n * (124 + tail_len) bytes); d_scratch[0..8) = total bytes,
// d_scratch[8..12) = 1 if some value needs the host formatter (inf, nan, |v| >= 2^57)
int launch_csv_format(const CsvJob &job, char *d_text, void *d_scratch, cudaStream_t stream);
// io.cu: the 18 pose columns of a line

}  // namespace nav
