/*
 * navslam_oracle.c -- CPU ORACLE, TEST INFRASTRUCTURE ONLY (see navslam_oracle.h).
 *
 * Restates, with runtime shapes and flat arrays, what the reference computes on
 * the front-end path.  Build with: gcc -std=gnu11 -O2 -ffp-contract=off (the
 * reference's CMakeLists.txt:5,9 flags; baseline x86-64 has no FMA contraction,
 * -ffp-contract=off makes that explicit).  All arithmetic is IEEE binary64 in
 * the reference's association order, so results are bit-identical to the
 * reference's on the same libm.
 */
#include "navslam_oracle.h"

#include <stdio.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ a2 -- */
/* utils/pointcloud.c:8-48.  45 x 45 degree field of view; angle of column i is
 * (-22.5 + i*45/(C-1)) deg converted as deg*M_PI/180; x = d, y = -d*tan(theta),
 * z = -d*tan(phi); d <= 0 -> (0,0,0). */
void nso_convert_to_pointcloud(int rows, int cols, const int *dist, nso_point *out) {
    const double fov = 45.0;
    const double col_step = fov / (cols - 1);
    const double row_step = fov / (rows - 1);
    for (int r = 0; r < rows; ++r) {
        for (int c = 0; c < cols; ++c) {
            nso_point *o = &out[(size_t)r * cols + c];
            double d = dist[(size_t)r * cols + c];
            if (d <= 0) {
                o->x = o->y = o->z = 0.0;
                continue;
            }
            double theta = -fov / 2.0 + c * col_step;
            double phi = -fov / 2.0 + r * row_step;
            theta = theta * M_PI / 180.0;
            phi = phi * M_PI / 180.0;
            o->x = d;
            o->y = -d * tan(theta);
            o->z = -d * tan(phi);
        }
    }
}

/* ------------------------------------------------------------------ a3 -- */
/* src/slam.c:28-33: Euclidean distance with the association (dx*dx + dy*dy) + dz*dz */
static inline double pt_dist(const nso_point *a, const nso_point *b) {
    double dx = a->x - b->x, dy = a->y - b->y, dz = a->z - b->z;
    return sqrt(dx * dx + dy * dy + dz * dz);
}

/* src/slam.c:18-55 for one interior point: neighbours at -2,-1,+1,+2 in the same row. */
static double curvature_at(const nso_point *row, int j) {
    static const int taps[4] = {-2, -1, 1, 2};
    double d[4];
    double sum = 0.0;
    for (int t = 0; t < 4; ++t) {
        d[t] = pt_dist(&row[j], &row[j + taps[t]]);
        sum += d[t];
    }
    double avg = sum / 4;
    if (!(avg > 0)) return 0.0;
    double var = 0.0;
    for (int t = 0; t < 4; ++t) var += (d[t] - avg) * (d[t] - avg);
    return var / 4 / (avg * avg + 1e-6f); /* float literal promoted, src/slam.c:54 */
}

void nso_curvature(int rows, int cols, const nso_point *cloud, double *curv) {
    for (int r = 0; r < rows; ++r) {
        const nso_point *row = cloud + (size_t)r * cols;
        for (int c = 0; c < cols; ++c)
            curv[(size_t)r * cols + c] = (c >= 2 && c < cols - 2) ? curvature_at(row, c) : 0.0;
    }
}

/* src/slam.c:15-16,57-58: columns [2, C-3], label 1 iff curvature > 0.1, never writes 0 */
void nso_extract_feature(int rows, int cols, const nso_point *cloud, int *feature) {
    for (int r = 0; r < rows; ++r) {
        const nso_point *row = cloud + (size_t)r * cols;
        for (int c = 2; c < cols - 2; ++c)
            if (curvature_at(row, c) > 0.1) feature[(size_t)r * cols + c] = 1;
    }
}

/* ------------------------------------------------------------------ a4 -- */
size_t nso_flatten(int cols, const nso_point *row, const int *row_feature, nso_point *out) {
    size_t n = 0;
    for (int c = 0; c < cols; ++c)
        if (row_feature[c] == 1) out[n++] = row[c];
    return n;
}

/* ------------------------------------------------------------------ a7 -- */
/* src/slam.c:95-115: R = Rz(yaw) * Ry(pitch) * Rx(roll) */
void nso_rotation(double roll, double pitch, double yaw, double R[9]) {
    double cr = cos(roll), sr = sin(roll);
    double cp = cos(pitch), sp = sin(pitch);
    double cy = cos(yaw), sy = sin(yaw);
    R[0] = cy * cp;
    R[1] = cy * sp * sr - sy * cr;
    R[2] = cy * sp * cr + sy * sr;
    R[3] = sy * cp;
    R[4] = sy * sp * sr + cy * cr;
    R[5] = sy * sp * cr - cy * sr;
    R[6] = -sp;
    R[7] = cp * sr;
    R[8] = cp * cr;
}

void nso_deg_rotation(const nso_pos *pos, double R[9]) {
    /* src/slam.c:8: DEG2RAD(x) = x * M_PI / 180.0 */
    nso_rotation(pos->roll * M_PI / 180.0, pos->pitch * M_PI / 180.0, pos->yaw * M_PI / 180.0, R);
}

/* src/slam.c:147-158: out = t + ((R0*x + R1*y) + R2*z) per component */
void nso_transform(size_t n, const nso_point *in, const double R[9], const double t[3], nso_point *out) {
    for (size_t i = 0; i < n; ++i) {
        double x = in[i].x, y = in[i].y, z = in[i].z;
        double rx = R[0] * x + R[1] * y + R[2] * z;
        double ry = R[3] * x + R[4] * y + R[5] * z;
        double rz = R[6] * x + R[7] * y + R[8] * z;
        out[i].x = t[0] + rx;
        out[i].y = t[1] + ry;
        out[i].z = t[2] + rz;
    }
}

/* src/slam.c:118-131 */
void nso_shift(size_t n, const nso_point *in, const double d[3], nso_point *out) {
    for (size_t i = 0; i < n; ++i) {
        out[i].x = in[i].x - d[0];
        out[i].y = in[i].y - d[1];
        out[i].z = in[i].z - d[2];
    }
}

/* --------------------------------------------------------------- a5/a6 -- */
struct nso_node {
    nso_point p;
    nso_node *lo, *hi;
};

static inline double axis_key(const nso_point *p, int axis) {
    return axis == 0 ? p->x : (axis == 1 ? p->y : p->z);
}

static inline void pt_swap(nso_point *a, nso_point *b) {
    nso_point t = *a;
    *a = *b;
    *b = t;
}

/* utils/kdtree.c:20-62 as a loop: Lomuto partition, pivot = last element, keys with
 * (key - pivot) <= 0 are packed to the front in order, then the pivot is dropped in. */
static void lomuto_select(nso_point *p, size_t first, size_t last, size_t nth, int axis) {
    while (first < last) {
        double pivot = axis_key(&p[last], axis);
        size_t store = first;
        for (size_t j = first; j < last; ++j) {
            double cmp = axis_key(&p[j], axis) - pivot;
            if (cmp <= 0) {
                pt_swap(&p[store], &p[j]);
                ++store;
            }
        }
        pt_swap(&p[store], &p[last]);
        if (store == nth) return;
        if (store < nth)
            first = store + 1;
        else
            last = store - 1;
    }
}

/* utils/kdtree.c:65-82: axis = depth % 3, median = n/2, children on [0,m) and [m+1,n) */
nso_node *nso_tree_build(nso_point *pts, size_t n, int depth) {
    if (n == 0) return NULL;
    size_t m = n / 2;
    lomuto_select(pts, 0, n - 1, m, depth % 3);
    nso_node *node = (nso_node *)malloc(sizeof(nso_node));
    node->p = pts[m];
    node->lo = nso_tree_build(pts, m, depth + 1);
    node->hi = nso_tree_build(pts + m + 1, n - m - 1, depth + 1);
    return node;
}

void nso_tree_free(nso_node *root) {
    if (!root) return;
    nso_tree_free(root->lo);
    nso_tree_free(root->hi);
    free(root);
}

/* utils/kdtree.c:110-152: strict '<' update, near child first, far child iff |delta| < best.
 * The reference's euclideanDistance uses pow(d,2), which gcc -O2 folds to d*d; the sum is
 * (dx*dx + dy*dy) + dz*dz with root - target as the operand order (sign is squared away). */
void nso_tree_nn(const nso_node *root, const nso_point *q, nso_point *best, double *best_dist, int depth) {
    if (!root) return;
    double d = pt_dist(&root->p, q);
    if (d < *best_dist) {
        *best_dist = d;
        *best = root->p;
    }
    int axis = depth % 3;
    double delta = axis_key(q, axis) - axis_key(&root->p, axis);
    const nso_node *near_side = delta < 0 ? root->lo : root->hi;
    const nso_node *far_side = delta < 0 ? root->hi : root->lo;
    nso_tree_nn(near_side, q, best, best_dist, depth + 1);
    if (fabs(delta) < *best_dist) nso_tree_nn(far_side, q, best, best_dist, depth + 1);
}

static size_t preorder_rec(const nso_node *n, int depth, nso_point *out, int *depth_out, size_t pos, size_t cap) {
    if (!n || pos >= cap) return pos;
    out[pos] = n->p;
    depth_out[pos] = depth;
    pos = preorder_rec(n->lo, depth + 1, out, depth_out, pos + 1, cap);
    return preorder_rec(n->hi, depth + 1, out, depth_out, pos, cap);
}
size_t nso_tree_preorder(const nso_node *root, nso_point *out, int *depth_out, size_t cap) {
    return preorder_rec(root, 0, out, depth_out, 0, cap);
}

/* canonical exact NN: argmin of dsq, lowest index on equal dsq */
static inline double pt_dsq(const nso_point *a, const nso_point *b) {
    double dx = a->x - b->x, dy = a->y - b->y, dz = a->z - b->z;
    return dx * dx + dy * dy + dz * dz;
}

void nso_nn_brute(const nso_point *pts, size_t n, const nso_point *q, size_t nq, int32_t *idx, double *dist) {
    for (size_t i = 0; i < nq; ++i) {
        double best = INFINITY;
        int32_t bi = -1;
        for (size_t j = 0; j < n; ++j) {
            double d = pt_dsq(&pts[j], &q[i]);
            if (d < best) {
                best = d;
                bi = (int32_t)j;
            }
        }
        idx[i] = bi;
        dist[i] = bi < 0 ? INFINITY : sqrt(best);
    }
}

void nso_nn_tie_count(const nso_point *pts, size_t n, const nso_point *q, size_t nq, int32_t *count) {
    for (size_t i = 0; i < nq; ++i) {
        double best = INFINITY;
        for (size_t j = 0; j < n; ++j) {
            double d = pt_dist(&pts[j], &q[i]);
            if (d < best) best = d;
        }
        int32_t c = 0;
        for (size_t j = 0; j < n; ++j)
            if (pt_dist(&pts[j], &q[i]) == best) ++c;
        count[i] = c;
    }
}

/* ------------------------------------------------------ whole SLAM step -- */
struct nso_slam {
    int rows, cols, tie_mode;
    int frame_count;
    double error;
    nso_node **trees;   /* tie_mode 0: per-row reference-shaped trees                 */
    nso_point *map_pts; /* both modes: previous frame's labelled global points per row */
    int32_t *map_col;   /*   ... and the column each came from                        */
    size_t *map_n;
    /* scratch */
    int *feature;
    nso_point *global_tmp, *query_tmp;
};

nso_slam *nso_slam_create(int rows, int cols, int tie_mode) {
    nso_slam *s = (nso_slam *)calloc(1, sizeof(nso_slam));
    size_t n = (size_t)rows * cols;
    s->rows = rows;
    s->cols = cols;
    s->tie_mode = tie_mode;
    s->trees = (nso_node **)calloc(rows, sizeof(nso_node *));
    s->map_pts = (nso_point *)malloc(n * sizeof(nso_point));
    s->map_col = (int32_t *)malloc(n * sizeof(int32_t));
    s->map_n = (size_t *)calloc(rows, sizeof(size_t));
    s->feature = (int *)malloc(n * sizeof(int));
    s->global_tmp = (nso_point *)malloc(n * sizeof(nso_point));
    s->query_tmp = (nso_point *)malloc(n * sizeof(nso_point));
    return s;
}

static void drop_trees(nso_slam *s) {
    for (int r = 0; r < s->rows; ++r) {
        nso_tree_free(s->trees[r]);
        s->trees[r] = NULL;
    }
}

void nso_slam_destroy(nso_slam *s) {
    if (!s) return;
    drop_trees(s);
    free(s->trees);
    free(s->map_pts);
    free(s->map_col);
    free(s->map_n);
    free(s->feature);
    free(s->global_tmp);
    free(s->query_tmp);
    free(s);
}

double nso_slam_error(const nso_slam *s) { return s->error; }
int nso_slam_frame_count(const nso_slam *s) { return s->frame_count; }

/* shared body of init_slam (src/slam.c:134-175) and slam_mapping (src/slam.c:393-431) */
static void map_frame(nso_slam *s, const nso_pos *pos, const nso_point *cloud, nso_point *global_out) {
    size_t n = (size_t)s->rows * s->cols;
    double R[9];
    nso_deg_rotation(pos, R);
    double t[3] = {pos->x, pos->y, pos->z};
    nso_point *g = global_out ? global_out : s->global_tmp;
    nso_transform(n, cloud, R, t, g);
    memset(s->feature, 0, n * sizeof(int));
    nso_extract_feature(s->rows, s->cols, cloud, s->feature);
    drop_trees(s); /* the reference leaks the old trees (src/slam.c:422-427) */
    nso_point *scratch = (nso_point *)malloc((size_t)s->cols * sizeof(nso_point));
    for (int r = 0; r < s->rows; ++r) {
        size_t base = (size_t)r * s->cols, k = 0;
        for (int c = 0; c < s->cols; ++c) {
            if (s->feature[base + c] == 1) {
                s->map_pts[base + k] = g[base + c];
                s->map_col[base + k] = c;
                ++k;
            }
        }
        s->map_n[r] = k;
        if (s->tie_mode == 0) {
            memcpy(scratch, s->map_pts + base, k * sizeof(nso_point));
            s->trees[r] = nso_tree_build(scratch, k, 0); /* works on a copy, like flattenedPoints */
        }
    }
    free(scratch);
    s->frame_count++;
}

void nso_slam_init(nso_slam *s, const nso_pos *pos, const nso_point *cloud, nso_point *global_out) {
    s->frame_count = 0;
    s->error = 0.0;
    map_frame(s, pos, cloud, global_out);
}

void nso_slam_map(nso_slam *s, const nso_pos *pos, const nso_point *cloud, nso_point *global_out) {
    map_frame(s, pos, cloud, global_out);
}

/* one query against row r's map.  Returns the column of the match in the previous frame
 * (-1 if the row's map is empty: the reference reads an uninitialised Point there,
 * utils/kdtree.c:112 + src/slam.c:242 -- undefined, so no correspondence is produced).
 * A query whose dsq to every map point of the row is +inf or NaN has no nearest point either:
 * -1 with *dist = +inf, as for an empty row. */
static int32_t row_query(const nso_slam *s, int r, const nso_point *q, nso_point *nearest, double *dist) {
    size_t base = (size_t)r * s->cols, n = s->map_n[r];
    if (n == 0) return -1;
    if (s->tie_mode == 0) {
        double best = INFINITY;
        nso_tree_nn(s->trees[r], q, nearest, &best, 0);
        *dist = best;
        if (!(best < INFINITY)) return -1;
        for (size_t j = 0; j < n; ++j) {
            const nso_point *p = &s->map_pts[base + j];
            if (p->x == nearest->x && p->y == nearest->y && p->z == nearest->z) return s->map_col[base + j];
        }
        return -1;
    }
    int32_t bi;
    nso_nn_brute(s->map_pts + base, n, q, 1, &bi, dist);
    if (bi < 0) return -1;
    *nearest = s->map_pts[base + bi];
    return s->map_col[base + bi];
}

/* query cloud of src/slam.c:180-210: T = pos_predict + R*p, Q = T - (pos_predict - pos_last) */
static void make_queries(nso_slam *s, const nso_point *cloud, const nso_pos *pp, const nso_pos *pl,
                         double transform[6], nso_point *T, nso_point *Q) {
    size_t n = (size_t)s->rows * s->cols;
    double R[9];
    nso_deg_rotation(pp, R);
    transform[0] = pp->x - pl->x;
    transform[1] = pp->y - pl->y;
    transform[2] = pp->z - pl->z;
    transform[3] = pp->roll - pl->roll;
    transform[4] = pp->pitch - pl->pitch;
    transform[5] = pp->yaw - pl->yaw;
    double t[3] = {pp->x, pp->y, pp->z};
    nso_transform(n, cloud, R, t, T);
    nso_shift(n, T, transform, Q);
}

size_t nso_slam_localize(nso_slam *s, const nso_point *cloud, const nso_pos *pos_predict,
                         const nso_pos *pos_last, nso_pos *pos_out, nso_corr *corr_out,
                         size_t corr_cap, int *iterations_out) {
    size_t n = (size_t)s->rows * s->cols;
    double transform[6];
    memset(s->feature, 0, n * sizeof(int));
    nso_extract_feature(s->rows, s->cols, cloud, s->feature);
    make_queries(s, cloud, pos_predict, pos_last, transform, s->global_tmp, s->query_tmp);

    /* correspondences with the per-row dedupe of src/slam.c:247-283: one entry per distinct
     * matched point (exact xyz equality), the closer query replaces (strict >), order of
     * first appearance is kept */
    nso_corr *res = (nso_corr *)malloc(n * sizeof(nso_corr));
    size_t count = 0;
    for (int r = 0; r < s->rows; ++r) {
        size_t row_start = count;
        for (int c = 0; c < s->cols; ++c) {
            size_t p = (size_t)r * s->cols + c;
            if (s->feature[p] != 1) continue;
            nso_point nearest;
            double dist;
            if (row_query(s, r, &s->query_tmp[p], &nearest, &dist) < 0) continue;
            size_t hit = count;
            for (size_t i = row_start; i < count; ++i) {
                if (res[i].nearest.x == nearest.x && res[i].nearest.y == nearest.y &&
                    res[i].nearest.z == nearest.z) {
                    hit = i;
                    break;
                }
            }
            if (hit == count) {
                res[count].ori = s->global_tmp[p];
                res[count].nearest = nearest;
                res[count].distance = dist;
                ++count;
            } else if (res[hit].distance > dist) {
                res[hit].ori = s->global_tmp[p];
                res[hit].nearest = nearest;
                res[hit].distance = dist;
            }
        }
    }

    /* translation-only Adam fit, src/slam.c:218-379 (the ErrDistance loop :301-308 is a dead
     * store and is not restated) */
    const double lr = 0.1, tol = 1e-6, b1 = 0.9, b2 = 0.999, eps = 1e-8;
    double m[3] = {0, 0, 0}, v[3] = {0, 0, 0};
    double prev_err = 0, total = 0;
    int valid = 0, iters = 0;
    for (int iter = 0; iter < 200; ++iter) {
        double g[3] = {0.0, 0.0, 0.0};
        total = 0;
        valid = 0;
        for (size_t i = 0; i < count; ++i) {
            double dx = (res[i].ori.x - transform[0]) - res[i].nearest.x;
            double dy = (res[i].ori.y - transform[1]) - res[i].nearest.y;
            double dz = (res[i].ori.z - transform[2]) - res[i].nearest.z;
            total += dx * dx + dy * dy + dz * dz;
            g[0] -= dx;
            g[1] -= dy;
            g[2] -= dz;
            ++valid;
        }
        iters = iter + 1;
        if (fabs(total - prev_err) < tol) break;
        prev_err = total;
        if (valid > 0) {
            g[0] /= valid;
            g[1] /= valid;
            g[2] /= valid;
        }
        int t = iter + 1;
        for (int j = 0; j < 3; ++j) {
            m[j] = b1 * m[j] + (1 - b1) * g[j];
            v[j] = b2 * v[j] + (1 - b2) * g[j] * g[j];
            double mh = m[j] / (1 - pow(b1, t));
            double vh = v[j] / (1 - pow(b2, t));
            transform[j] -= lr * mh / (sqrt(vh) + eps);
        }
    }
    s->error = valid > 0 ? sqrt(total / valid) : 0.0;
    pos_out->x = pos_last->x + transform[0];
    pos_out->y = pos_last->y + transform[1];
    pos_out->z = pos_last->z + transform[2];
    pos_out->roll = pos_last->roll + transform[3];
    pos_out->pitch = pos_last->pitch + transform[4];
    pos_out->yaw = pos_last->yaw + transform[5];
    if (iterations_out) *iterations_out = iters;
    if (corr_out) memcpy(corr_out, res, (count < corr_cap ? count : corr_cap) * sizeof(nso_corr));
    free(res);
    return count;
}

void nso_frontend_frame(nso_slam *s, const nso_point *cloud, const nso_pos *pos_predict,
                        const nso_pos *pos_last, const nso_pos *pos_final,
                        int *feature_out, int32_t *nn_idx, double *nn_dist, nso_point *global_out) {
    size_t n = (size_t)s->rows * s->cols;
    double transform[6];
    memset(s->feature, 0, n * sizeof(int));
    nso_extract_feature(s->rows, s->cols, cloud, s->feature);
    make_queries(s, cloud, pos_predict, pos_last, transform, s->global_tmp, s->query_tmp);
    for (int r = 0; r < s->rows; ++r) {
        for (int c = 0; c < s->cols; ++c) {
            size_t p = (size_t)r * s->cols + c;
            if (s->feature[p] != 1) {
                nn_idx[p] = -1;
                nn_dist[p] = -1.0;
                continue;
            }
            nso_point nearest;
            double dist = INFINITY;
            int32_t col = row_query(s, r, &s->query_tmp[p], &nearest, &dist);
            nn_idx[p] = col < 0 ? -1 : (int32_t)((size_t)r * s->cols + col);
            nn_dist[p] = dist;
        }
    }
    if (feature_out) memcpy(feature_out, s->feature, n * sizeof(int));
    map_frame(s, pos_final, cloud, global_out);
}

/* ---------------------------------------------------------------- caller-side data formats ---- */
/* src/main.c:77-128 */
int nso_l9_csv_read(const char *path, int rows, int cols, size_t max_frames, nso_point *frames,
                    int32_t *timestamps, size_t *n_frames) {
    FILE *fp = fopen(path, "r");
    *n_frames = 0;
    if (!fp) return 1;
    char header[256];
    if (!fgets(header, sizeof(header), fp)) { /* main.c:87-91 */
        fclose(fp);
        return 0;
    }
    int frame, row, col, conf, current = -1;
    double x, y, z;
    size_t count = 0;
    while (fscanf(fp, "%d,%d,%d,%lf,%lf,%lf,%d", &frame, &row, &col, &x, &y, &z, &conf) == 7) { /* main.c:99 */
        /* main.c:100 accepts col == MAX_COLS (one past the row); that write is out of bounds, so the
         * restatement skips it like every other out-of-range record */
        if (row < 0 || row >= rows || col < 0 || col >= cols) continue;
        if (frame != current) { /* main.c:105-112 */
            if (current != -1) count++;
            if (count >= max_frames) {
                fclose(fp);
                *n_frames = max_frames;
                return 2;
            }
            current = frame;
            if (timestamps) timestamps[count] = frame;
        }
        nso_point *d = &frames[count * (size_t)rows * cols + (size_t)row * cols + col];
        d->x = x; /* main.c:115-117 */
        d->y = y;
        d->z = z;
    }
    *n_frames = current != -1 ? count + 1 : 0; /* main.c:121-125 */
    fclose(fp);
    return 0;
}

/* src/main.c:320-352 (the L5 handler passes doubles to every %.2f) */
size_t nso_csv_format_frame(char *buf, size_t cap, unsigned long long timestamp, int rows, int cols,
                            const nso_point *g, const int32_t *distances, const double *imu6,
                            const nso_pos *lp, const nso_pos *ep) {
    static const double zero6[6] = {0, 0, 0, 0, 0, 0};
    const double *im = imu6 ? imu6 : zero6;
    const nso_pos zp = {0, 0, 0, 0, 0, 0};
    if (!ep) ep = &zp;
    size_t off = 0;
    for (int row = 0; row < rows; ++row)
        for (int col = 0; col < cols; ++col) {
            const nso_point *p = &g[(size_t)row * cols + col];
            int n = snprintf(buf + off, cap - off,
                             "%zu,%d,%d,%.2f,%.2f,%.2f,%d,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,%.2f,"
                             "%.2f,%.2f,%.2f,%.2f,%.2f,%.2f\n",
                             (size_t)timestamp, row, col, p->x, p->y, p->z,
                             distances ? (int)distances[(size_t)row * cols + col] : 0, im[0], im[1], im[2], im[3],
                             im[4], im[5], lp->x, lp->y, lp->z, lp->roll, lp->pitch, lp->yaw, ep->x, ep->y, ep->z,
                             ep->roll, ep->pitch, ep->yaw);
            if (n < 0 || (size_t)n >= cap - off) return 0;
            off += (size_t)n;
        }
    return off;
}
