/*
 * navslam_shim.c -- per-shape drop-in for the reference's slam.c + kdtree.c + pointcloud.c.
 *
 * Compiled once per image shape (-DMAX_ROWS=R -DMAX_COLS=C) into
 * libnavslam_shim_<R>x<C>.so, it exports the reference's own symbols with byte-identical
 * signatures (include/navslam_ref_abi.h) and forwards every data-parallel body to
 * libnavslam_b200.so (CUDA, sm_100a).  What stays on the host is what the reference's design
 * keeps scalar: the rotation matrix, the pose difference and the Adam translation fit (inside
 * nav_slam_localization).  There is no CPU fallback: a CUDA failure prints the library's error
 * and aborts, because the reference's signatures have no error channel (SURVEY section 5).
 *
 * KDNode* values handed out here are opaque handles (tagged structs), never dereferenced by the
 * reference's main.c.
 */
#include "navslam_ref_abi.h"

#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "navslam_b200.h"

#define TAG_ROW 0x4e41565f524f5721ull  /* "NAV_ROW!" */
#define TAG_TREE 0x4e41565f54524545ull /* "NAV_TREE" */

typedef struct {
    uint64_t tag;
    nav_ctx *ctx;
    nav_kdtree *tree;  /* TAG_TREE */
    int row;           /* TAG_ROW  */
    int depth0;
    Point *host_copy;  /* points in build order, for printKDTree */
    size_t n;
} shim_handle;

#define MAX_ATTRS 16
static struct {
    SLAM_attr *attr;
    nav_ctx *ctx;
    shim_handle rows[MAX_ROWS];
    Point *last_cloud; /* identity of the frame last uploaded by slam_localization */
    int last_ts;
} g_slots[MAX_ATTRS];
static nav_ctx *g_default_ctx;

/* The reference's callers keep their clouds in ordinary (pageable) memory -- one PointCloud on the stack of
 * the L5 handler (src/main.c:250), ten in the L9 handler (src/main.c:363), the SLAM_attr with its hundred
 * global clouds (src/main.c:252,381).  Copying 3 MB frames through a bounce buffer costs more than the GPU
 * work, so with NAVSLAM_PIN=1 the shim page-locks those buffers where they lie the first time it sees them;
 * a failed registration just leaves the buffer on the staged path.  Opt-in, because the reference's
 * interface has no teardown call: a registration is keyed by address, so it is only safe for buffers that
 * live as long as the program does (which is how main.c holds them) -- a caller that frees a cloud and
 * gets the same address back from malloc would DMA into the pages of the old mapping. */
#define MAX_PINNED 16
static const void *g_pinned[MAX_PINNED];
static unsigned g_pin_next;

static int pin_enabled(void) {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("NAVSLAM_PIN");
        v = e && e[0] == '1';
    }
    return v;
}

static void pin_buffer(const void *p, size_t bytes) {
    if (!pin_enabled() || bytes < (1u << 16)) return; /* small frames are not worth a registration */
    for (int i = 0; i < MAX_PINNED; ++i)
        if (g_pinned[i] == p) return;
    unsigned slot = g_pin_next++ % MAX_PINNED;
    if (g_pinned[slot]) nav_host_unregister((void *)g_pinned[slot]);
    g_pinned[slot] = nav_host_register((void *)p, bytes) == 0 ? p : NULL;
}

static void unpin_buffer(const void *p) {
    for (int i = 0; i < MAX_PINNED; ++i)
        if (g_pinned[i] == p && p) {
            nav_host_unregister((void *)p);
            g_pinned[i] = NULL;
        }
}

static void die(const char *what) {
    fprintf(stderr, "navslam_shim(%dx%d): %s: %s\n", MAX_ROWS, MAX_COLS, what, nav_last_error());
    abort();
}

/* NAVSLAM_TIES=reference: every context the shim creates resolves exact distance ties as the reference does (the
 * first tied point its per-row tree search reaches, NAV_TIE_REFERENCE) instead of by lowest index, so that
 * integer-valued data gives the reference's correspondences, poses and CSV bit for bit.  Opt-in: it costs a host
 * round trip per slam_localization, and the default output stays as it was. */
static int ties_reference(void) {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("NAVSLAM_TIES");
        v = e && strcmp(e, "reference") == 0;
    }
    return v;
}

static nav_ctx *new_ctx(void) {
    nav_ctx *c = nav_create(MAX_ROWS, MAX_COLS, 0, 1);
    if (!c) die("nav_create");
    if (ties_reference() && nav_set_tie_rule(c, NAV_TIE_REFERENCE)) die("NAVSLAM_TIES=reference");
    return c;
}

static nav_ctx *default_ctx(void) {
    if (!g_default_ctx) g_default_ctx = new_ctx();
    return g_default_ctx;
}

static void release_all(void);

static int slot_of(SLAM_attr *attr, int create) {
    int free_slot = -1;
    for (int i = 0; i < MAX_ATTRS; ++i) {
        if (g_slots[i].attr == attr) return i;
        if (!g_slots[i].attr && free_slot < 0) free_slot = i;
    }
    if (!create) return -1;
    if (free_slot < 0) {
        fprintf(stderr, "navslam_shim: more than %d SLAM_attr objects in use\n", MAX_ATTRS);
        abort();
    }
    g_slots[free_slot].attr = attr;
    g_slots[free_slot].ctx = new_ctx();
    static int at_exit_registered;
    if (!at_exit_registered) { /* after the first CUDA call, so that it runs before the runtime's own teardown */
        at_exit_registered = 1;
        atexit(release_all);
    }
    for (int r = 0; r < MAX_ROWS; ++r) {
        shim_handle *h = &g_slots[free_slot].rows[r];
        memset(h, 0, sizeof(*h));
        h->tag = TAG_ROW;
        h->ctx = g_slots[free_slot].ctx;
        h->row = r;
    }
    return free_slot;
}

struct nav_ctx *navslam_context_of(SLAM_attr *attr) {
    int s = slot_of(attr, 0);
    return s < 0 ? NULL : g_slots[s].ctx;
}

/* The reference never frees its row trees (src/slam.c:167-172 leaks them) and has no teardown call, so a
 * slot -- a nav_ctx with a few hundred MB of device buffers at 64x2048 -- would otherwise live for ever.
 * navslam_release() gives a SLAM_attr's slot back (init_slam on the same address re-uses its slot anyway);
 * whatever is still held at exit is destroyed by the atexit handler. */
void navslam_release(SLAM_attr *attr) {
    int s = slot_of(attr, 0);
    if (s < 0) return;
    unpin_buffer(attr);
    nav_destroy(g_slots[s].ctx);
    memset(&g_slots[s], 0, sizeof(g_slots[s]));
}

static void release_all(void) {
    for (int i = 0; i < MAX_ATTRS; ++i)
        if (g_slots[i].attr) navslam_release(g_slots[i].attr);
    for (int i = 0; i < MAX_PINNED; ++i)
        if (g_pinned[i]) unpin_buffer(g_pinned[i]);
    if (g_default_ctx) nav_destroy(g_default_ctx);
    g_default_ctx = NULL;
}

static void publish_rows(int s) {
    for (int r = 0; r < MAX_ROWS; ++r) g_slots[s].attr->kdtree_lastframe[r] = (KDNode *)&g_slots[s].rows[r];
}

/* layout probes for tests/test_abi.py (compared with the reference's own compiled sizeof/offsetof) */
int navslam_abi_rows(void) { return MAX_ROWS; }
int navslam_abi_cols(void) { return MAX_COLS; }
size_t navslam_abi_sizeof_pointcloud(void) { return sizeof(PointCloud); }
size_t navslam_abi_sizeof_slam_attr(void) { return sizeof(SLAM_attr); }
size_t navslam_abi_sizeof_kdnode(void) { return sizeof(KDNode); }
size_t navslam_abi_sizeof_neighbor_result(void) { return sizeof(NeighborResult); }
size_t navslam_abi_offsetof_frame_count(void) { return offsetof(SLAM_attr, frameCount); }
size_t navslam_abi_offsetof_trees(void) { return offsetof(SLAM_attr, kdtree_lastframe); }
size_t navslam_abi_offsetof_error(void) { return offsetof(SLAM_attr, error); }

/* ---------------------------------------------------------------- slam.h ---------------- */
/* headers/slam.h:22, src/slam.c:134-175 */
void init_slam(SLAM_attr *attr, Pos pos, PointCloud *lidarPointCloud) {
    int s = slot_of(attr, 1);
    pin_buffer(attr, sizeof(SLAM_attr));
    pin_buffer(lidarPointCloud, sizeof(PointCloud));
    attr->frameCount = 0;
    attr->error = 0.0;
    attr->globalPointCloud[0].ToF_timestamps = lidarPointCloud->ToF_timestamps;
    if (nav_slam_init(g_slots[s].ctx, (const nav_pos *)&pos, (const nav_point *)&lidarPointCloud->ToF_position[0][0],
                      (nav_point *)&attr->globalPointCloud[0].ToF_position[0][0]))
        die("init_slam");
    publish_rows(s);
    g_slots[s].last_cloud = NULL;
    attr->frameCount++;
}

/* headers/slam.h:25, src/slam.c:178-390.  Prints the reference's per-iteration lines. */
Pos slam_localization(SLAM_attr *attr, PointCloud *lidarPointCloud, Pos pos_predict, Pos pos_last) {
    int s = slot_of(attr, 0);
    if (s < 0) {
        fprintf(stderr, "navslam_shim: slam_localization before init_slam\n");
        abort();
    }
    Pos out;
    double err = 0.0;
    pin_buffer(lidarPointCloud, sizeof(PointCloud));
    /* default: the reference's sequential Adam loop on the host (bit-identical poses and the same
     * per-iteration stdout).  NAVSLAM_ADAM=stats: fit from five device-reduced sums (no 3.5 MB
     * correspondence download, no 200 x N host loop; poses equal to ~1e-9 relative, no per-iteration
     * lines). */
    static int fast = -1;
    if (fast < 0) {
        const char *e = getenv("NAVSLAM_ADAM");
        fast = e && strcmp(e, "stats") == 0;
    }
    if (fast && ties_reference()) {
        fprintf(stderr, "navslam_shim(%dx%d): NAVSLAM_ADAM=stats cannot be combined with NAVSLAM_TIES=reference: the "
                        "fit from device-reduced sums deduplicates on the device, the reference tie rule needs the "
                        "host round trip of the default fit\n", MAX_ROWS, MAX_COLS);
        abort();
    }
    if (fast) {
        if (nav_slam_localization_fast(g_slots[s].ctx, (const nav_point *)&lidarPointCloud->ToF_position[0][0],
                                       (const nav_pos *)&pos_predict, (const nav_pos *)&pos_last, (nav_pos *)&out,
                                       &err, NULL))
            die("slam_localization");
    } else if (nav_slam_localization(g_slots[s].ctx, (const nav_point *)&lidarPointCloud->ToF_position[0][0],
                                     (const nav_pos *)&pos_predict, (const nav_pos *)&pos_last, (nav_pos *)&out, &err,
                                     1))
        die("slam_localization");
    attr->error = err;
    g_slots[s].last_cloud = &lidarPointCloud->ToF_position[0][0];
    g_slots[s].last_ts = lidarPointCloud->ToF_timestamps;
    return out;
}

/* headers/slam.h:28, src/slam.c:393-431 */
void slam_mapping(SLAM_attr *attr, Pos pos, PointCloud *lidarPointCloud) {
    int s = slot_of(attr, 0);
    if (s < 0) {
        fprintf(stderr, "navslam_shim: slam_mapping before init_slam\n");
        abort();
    }
    if (attr->frameCount < 0 || attr->frameCount >= 100) {
        /* the reference writes past globalPointCloud[100] here (SURVEY D6); refuse instead */
        fprintf(stderr, "navslam_shim: slam_mapping with frameCount=%d outside globalPointCloud[100]\n",
                attr->frameCount);
        abort();
    }
    attr->globalPointCloud[attr->frameCount].ToF_timestamps = lidarPointCloud->ToF_timestamps;
    /* Strict drop-in: the cloud is uploaded and labelled again, exactly as the reference
     * re-runs extract_feature (src/slam.c:420).  NAVSLAM_TRUST_FRAME=1 lets the shim reuse the
     * device-resident cloud + labels when the same buffer was just localised. */
    const nav_point *cloud = (const nav_point *)&lidarPointCloud->ToF_position[0][0];
    pin_buffer(lidarPointCloud, sizeof(PointCloud));
    static int trust = -1;
    if (trust < 0) {
        const char *e = getenv("NAVSLAM_TRUST_FRAME");
        trust = e && e[0] == '1';
    }
    if (trust && g_slots[s].last_cloud == &lidarPointCloud->ToF_position[0][0] &&
        g_slots[s].last_ts == lidarPointCloud->ToF_timestamps)
        cloud = NULL;
    if (nav_slam_mapping(g_slots[s].ctx, (const nav_pos *)&pos, cloud,
                         (nav_point *)&attr->globalPointCloud[attr->frameCount].ToF_position[0][0]))
        die("slam_mapping");
    g_slots[s].last_cloud = NULL;
    publish_rows(s);
    attr->frameCount++;
}

/* ---------------------------------------------------------------- pointcloud.h ---------- */
/* utils/pointcloud.h:55, utils/pointcloud.c:8-48 */
void convertToPointCloud(int distances[MAX_ROWS][MAX_COLS], Point pointCloud[MAX_ROWS][MAX_COLS]) {
    if (nav_convert_to_pointcloud(default_ctx(), &distances[0][0], (nav_point *)&pointCloud[0][0]))
        die("convertToPointCloud");
}

/* utils/pointcloud.h:57, utils/pointcloud.c:50-58 (the index printed is i*MAX_ROWS+j there) */
void printPointCloud(PointCloud pointcloud) {
    for (int i = 0; i < MAX_ROWS; i++)
        for (int j = 0; j < MAX_COLS; j++) {
            Point p = pointcloud.ToF_position[i][j];
            printf("point %d: (%f, %f, %f) \n", i * MAX_ROWS + j, p.x, p.y, p.z);
        }
}

/* ---------------------------------------------------------------- slam.c externals ------ */
void extract_feature(PointCloud *lidarPointCloud, int feature[MAX_ROWS][MAX_COLS]) {
    if (nav_extract_feature(default_ctx(), (const nav_point *)&lidarPointCloud->ToF_position[0][0], &feature[0][0]))
        die("extract_feature");
}

void flattenPoints(Point rowPoints[MAX_COLS], int rowFeature[MAX_COLS], Point flattenedPoints[MAX_COLS],
                   size_t *numPoints) {
    if (nav_flatten_points(default_ctx(), (const nav_point *)rowPoints, rowFeature, (nav_point *)flattenedPoints,
                           numPoints))
        die("flattenPoints");
}

void compute_posdiff(Pos *pos_now, Pos *pos_last, double pos_diff[6]) {
    pos_diff[0] = pos_now->x - pos_last->x;
    pos_diff[1] = pos_now->y - pos_last->y;
    pos_diff[2] = pos_now->z - pos_last->z;
    pos_diff[3] = pos_now->roll - pos_last->roll;
    pos_diff[4] = pos_now->pitch - pos_last->pitch;
    pos_diff[5] = pos_now->yaw - pos_last->yaw;
}

void getRotationMatrix(double roll, double pitch, double yaw, double R[3][3]) {
    const double cr = cos(roll), sr = sin(roll), cp = cos(pitch), sp = sin(pitch), cy = cos(yaw), sy = sin(yaw);
    R[0][0] = cy * cp;
    R[0][1] = cy * sp * sr - sy * cr;
    R[0][2] = cy * sp * cr + sy * sr;
    R[1][0] = sy * cp;
    R[1][1] = sy * sp * sr + cy * cr;
    R[1][2] = sy * sp * cr - cy * sr;
    R[2][0] = -sp;
    R[2][1] = cp * sr;
    R[2][2] = cp * cr;
}

/* src/slam.c:118-131 (un-headered helper of the reference; the frame kernel does this per query) */
void mapCoordinatesToLastFrame(PointCloud *globalPointCloudData, double transform[3], PointCloud *positionInLastFrame) {
    for (int row = 0; row < MAX_ROWS; ++row)
        for (int col = 0; col < MAX_COLS; ++col) {
            const Point *g = &globalPointCloudData->ToF_position[row][col];
            Point *o = &positionInLastFrame->ToF_position[row][col];
            o->x = g->x - transform[0];
            o->y = g->y - transform[1];
            o->z = g->z - transform[2];
        }
}

int getAxis(int depth) { return depth % 3; }

double euclideanDistance(Point p1, Point p2) {
    const double dx = p1.x - p2.x, dy = p1.y - p2.y, dz = p1.z - p2.z;
    return sqrt(dx * dx + dy * dy + dz * dz);
}

/* ---------------------------------------------------------------- kdtree.h -------------- */
/* utils/kdtree.h:21.  Unlike the reference the caller's array is left in its original order
 * (indices returned by navslam_nn_batch refer to it).  depth selects the root axis (depth % 3). */
KDNode *buildKDTree(Point *points, size_t numPoints, int depth) {
    if (numPoints == 0) return NULL; /* utils/kdtree.c:67 */
    if (depth % 3 != 0) {
        fprintf(stderr, "navslam_shim: buildKDTree with depth %% 3 != 0 is not supported\n");
        abort();
    }
    shim_handle *h = (shim_handle *)calloc(1, sizeof(shim_handle));
    h->tag = TAG_TREE;
    h->depth0 = depth;
    h->n = numPoints;
    h->tree = nav_kdtree_build(0, (const nav_point *)points, numPoints);
    if (!h->tree) die("buildKDTree");
    h->host_copy = (Point *)malloc(numPoints * sizeof(Point));
    memcpy(h->host_copy, points, numPoints * sizeof(Point));
    return (KDNode *)h;
}

void freeKDTree(KDNode *root) {
    shim_handle *h = (shim_handle *)root;
    if (!h || h->tag != TAG_TREE) return; /* row handles belong to their SLAM_attr slot */
    nav_kdtree_free(h->tree);
    free(h->host_copy);
    h->tag = 0;
    free(h);
}

struct nav_kdtree *navslam_tree_of(KDNode *root) {
    shim_handle *h = (shim_handle *)root;
    return h && h->tag == TAG_TREE ? h->tree : NULL;
}

int navslam_nn_batch(KDNode *root, const Point *targets, size_t n, int *index_out, double *dist_out,
                     Point *nearest_out) {
    shim_handle *h = (shim_handle *)root;
    if (!h) {
        for (size_t i = 0; i < n; ++i) {
            index_out[i] = -1;
            dist_out[i] = INFINITY;
        }
        return 0;
    }
    if (h->tag != TAG_TREE) {
        fprintf(stderr, "navslam_shim: navslam_nn_batch needs a handle from buildKDTree\n");
        abort();
    }
    if (nav_kdtree_nn_batch(h->tree, (const nav_point *)targets, n, index_out, dist_out, (nav_point *)nearest_out))
        die("navslam_nn_batch");
    return 0;
}

/* utils/kdtree.h:27, utils/kdtree.c:110-152: one query per call (kept for ABI completeness; the
 * SLAM step never goes through it).  Outputs change only if a point closer than *bestDist exists. */
void nearestNeighborSearch(KDNode *root, Point *target, Point *result, double *bestDist, int depth) {
    (void)depth;
    if (!root) return; /* utils/kdtree.c:112 */
    int idx = -1;
    double dist = INFINITY;
    Point near;
    navslam_nn_batch(root, target, 1, &idx, &dist, &near);
    if (idx >= 0 && dist < *bestDist) {
        *bestDist = dist;
        *result = near;
    }
}

/* ---- printKDTree (utils/kdtree.h:30, utils/kdtree.c:94-107): debug dump in the reference's
 * pre-order.  The device structures are flat, so the pointer tree the reference would have
 * built (median split, Lomuto quick-select with the last element as pivot, utils/kdtree.c:20-82)
 * is re-created on the host from the same points purely for printing. */
static void select_nth(Point *p, size_t first, size_t last, size_t nth, int axis) {
    while (first < last) {
        const Point pv = p[last];
        size_t store = first;
        for (size_t j = first; j < last; ++j) {
            const double cmp = axis == 0 ? p[j].x - pv.x : (axis == 1 ? p[j].y - pv.y : p[j].z - pv.z);
            if (cmp <= 0) {
                Point t = p[store];
                p[store] = p[j];
                p[j] = t;
                ++store;
            }
        }
        Point t = p[store];
        p[store] = p[last];
        p[last] = t;
        if (store == nth) return;
        if (store < nth)
            first = store + 1;
        else
            last = store - 1;
    }
}

/* utils/kdtree.c:20-62 has external linkage in the reference: same in-place partial ordering */
void nth_element(Point *points, size_t first, size_t last, size_t nth, int axis) {
    select_nth(points, first, last, nth, axis);
}

static void print_subtree(Point *p, size_t n, int build_depth, int print_depth) {
    if (n == 0) return;
    const size_t m = n / 2;
    select_nth(p, 0, n - 1, m, build_depth % 3);
    printf("深度 %d: Point(x=%.2f, y=%.2f, z=%.2f)\n", print_depth, p[m].x, p[m].y, p[m].z);
    print_subtree(p, m, build_depth + 1, print_depth + 1);
    print_subtree(p + m + 1, n - m - 1, build_depth + 1, print_depth + 1);
}

void printKDTree(KDNode *root, int depth) {
    shim_handle *h = (shim_handle *)root;
    if (!h) return;
    Point *work = NULL;
    size_t n = 0;
    if (h->tag == TAG_TREE) {
        n = h->n;
        work = (Point *)malloc(n * sizeof(Point));
        memcpy(work, h->host_copy, n * sizeof(Point));
    } else if (h->tag == TAG_ROW) {
        /* the row's map = labelled global points of the last mapped frame, in column order:
         * exactly the flattenedPoints array the reference hands to buildKDTree (src/slam.c:170-171) */
        work = (Point *)malloc((size_t)MAX_COLS * sizeof(Point));
        if (nav_row_map_export(h->ctx, 0, h->row, (nav_point *)work, NULL, &n)) die("printKDTree");
        if (!work) return;
    } else {
        return;
    }
    print_subtree(work, n, 0, depth);
    free(work);
}
