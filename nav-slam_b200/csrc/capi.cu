// capi.cu -- the C ABI of libnavslam_b200.so (include/navslam_b200.h): contexts, host<->device
// staging, and the host-side scalar pieces the reference keeps on the CPU (rotation matrix from
// libm sin/cos, tan tables, the translation-only Adam fit of src/slam.c:218-379).
#include <assert.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <time.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <utility>
#include <vector>

#include "nav_kdtree.cuh"
#include "csv_fixed2.cuh"
#include "nav_kernels.cuh"

using namespace nav;

// ------------------------------------------------------------------ errors ------------------
static thread_local char g_err[512] = "";

static int fail(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

// error channel for the other translation units of the library (io.cu)
int nav_io_fail(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define CUP(call)                                                                             \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return nullptr;                                                                   \
        }                                                                                     \
    } while (0)

extern "C" const char *nav_version(void) { return "navslam_b200 0.2 (sm_100a)"; }
extern "C" const char *nav_last_error(void) { return g_err; }

extern "C" int nav_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// pointers this thread has already seen to be pinned (Stager::is_pinned); nav_host_free / nav_host_unregister
// forget theirs
static const void **pinned_seen() {
    static thread_local const void *seen[16] = {};
    return seen;
}
static void pinned_forget(const void *p) {
    const void **seen = pinned_seen();
    for (int i = 0; i < 16; ++i)
        if (seen[i] && seen[i] >= p) seen[i] = nullptr;  // conservatively: everything at or above the base address
}

extern "C" void *nav_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        fail("cudaHostAlloc(%zu) failed", bytes);
        return nullptr;
    }
    return p;
}
extern "C" void nav_host_free(void *p) {
    if (!p) return;
    pinned_forget(p);
    cudaFreeHost(p);
}
// page-lock memory the caller already owns (cudaHostRegister), so that the host-buffer calls DMA it
// directly instead of staging it through a bounce buffer
extern "C" int nav_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return fail("nav_host_register: null argument");
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail("nav_host_register(%p, %zu): %s", p, bytes, cudaGetErrorString(e));
    }
    return 0;
}
extern "C" int nav_host_unregister(void *p) {
    if (!p) return 0;
    pinned_forget(p);
    if (cudaHostUnregister(p) != cudaSuccess) {
        cudaGetLastError();
        return fail("nav_host_unregister(%p) failed", p);
    }
    return 0;
}

// ------------------------------------------------------------------ staging -----------------
struct PendingOut {
    void *dst;
    const void *src;
    size_t bytes;
};

struct Stager {
    unsigned char *buf = nullptr;
    size_t cap = 0, used = 0;
    std::vector<PendingOut> pending;

    // cudaPointerGetAttributes costs about a microsecond; the pipelined entry points are called with the
    // same few buffers frame after frame, so pointers already seen to be pinned are remembered
    // (a buffer that stops being pinned would merely be copied through the driver's own staging)
    static bool is_pinned(const void *p) {
        const void **seen = pinned_seen();
        static thread_local unsigned next = 0;
        for (int i = 0; i < 16; ++i)
            if (seen[i] == p) return true;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        if (at.type != cudaMemoryTypeHost) return false;
        seen[next++ & 15u] = p;
        return true;
    }
    // staging space lives for one API call; growing needs the stream idle
    unsigned char *take(size_t bytes, cudaStream_t stream) {
        bytes = (bytes + 255) & ~(size_t)255;
        if (used + bytes > cap) {
            if (used != 0) return nullptr;  // caller reserves up front
            cudaStreamSynchronize(stream);
            if (buf) cudaFreeHost(buf);
            buf = nullptr;
            cap = 0;
            if (cudaHostAlloc((void **)&buf, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
            cap = bytes;
        }
        unsigned char *p = buf + used;
        used += bytes;
        return p;
    }
    int reserve(size_t bytes, cudaStream_t stream) {
        if (used != 0 || !pending.empty()) {  // a previous call bailed out half way
            cudaStreamSynchronize(stream);
            used = 0;
            pending.clear();
        }
        if (bytes <= cap) return 0;
        unsigned char *p = take(bytes, stream);
        used = 0;
        return p ? 0 : 1;
    }
    int h2d(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
        if (bytes == 0) return 0;
        const void *from = src;
        if (!is_pinned(src)) {
            unsigned char *s = take(bytes, stream);
            if (!s) return 1;
            memcpy(s, src, bytes);
            from = s;
        }
        return cudaMemcpyAsync(dst, from, bytes, cudaMemcpyHostToDevice, stream) != cudaSuccess;
    }
    int d2h(void *dst, const void *src, size_t bytes, cudaStream_t stream) {
        if (bytes == 0) return 0;
        void *to = dst;
        if (!is_pinned(dst)) {
            unsigned char *s = take(bytes, stream);
            if (!s) return 1;
            pending.push_back({dst, s, bytes});
            to = s;
        }
        return cudaMemcpyAsync(to, src, bytes, cudaMemcpyDeviceToHost, stream) != cudaSuccess;
    }
    int finish(cudaStream_t stream) {
        cudaError_t e = cudaStreamSynchronize(stream);
        for (auto &p : pending) memcpy(p.dst, p.src, p.bytes);
        pending.clear();
        used = 0;
        return e != cudaSuccess;
    }
    void release() {
        if (buf) cudaFreeHost(buf);
        buf = nullptr;
        cap = used = 0;
    }
};

// ------------------------------------------------------------------ context -----------------
struct ProfSlot {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
    size_t used = 0;
    double ms = 0;
    uint64_t launches = 0;
};

struct nav_ctx {
    int rows = 0, cols = 0, n_seq = 1, device = 0, sm_count = 148;
    size_t npx = 0, ntot = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    double *d_cloud = nullptr, *d_global = nullptr, *d_curv = nullptr, *d_nn_dist = nullptr;
    unsigned *d_n_exact = nullptr;  // labels the fp32 filter could not decide (exact re-evaluations)
    int *d_labels = nullptr, *d_nn_idx = nullptr;
    RowMap map = {};      // the map the next match searches (frame mapped last)
    RowMap map_alt = {};  // second buffer: the fused frame kernel builds the next map here, then they swap
    nav_corr *d_corr_rows = nullptr, *d_corr = nullptr;
    int *d_corr_row_count = nullptr, *d_corr_total = nullptr;
    // the raw frames of the blocking calls, before they become xyz (raw_buf): [0] depth (allocated by nav_create,
    // one image), [1] integer mm.  Each async slot and prefetch slot holds its own pair.
    int *raw[2] = {nullptr, nullptr};
    double *d_tan_col = nullptr, *d_tan_row = nullptr;
    double *d_flat = nullptr;
    int *d_flat_count = nullptr;
    int *h_small = nullptr;  // pinned scratch for counts
    char *d_csv = nullptr;   // device text of one frame's CSV rows (lazy)
    void *d_csv_scratch = nullptr;
    size_t csv_cap = 0;
    Stager stage;
    bool have_map = false, cloud_resident = false;
    uint64_t launches = 0;
    // pipelined host path (nav_frontend_submit / nav_frontend_frame_async): copy-in / copy-out streams and
    // as many slots as there are map buffers -- the download of frame t reads the map built by frame t
    // (global cloud, label masks) straight out of its ping-pong buffer, which frame t+2 overwrites; frame
    // t+2 uses the same slot and waits for that download.
    static constexpr int kSlots = 2;
    struct AsyncSlot {
        double *d_cloud = nullptr, *d_nn_dist = nullptr;
        int *d_labels = nullptr, *d_nn_idx = nullptr;
        int *raw[2] = {nullptr, nullptr};
        cudaEvent_t in_done = nullptr, compute_done = nullptr, out_done = nullptr;
    } slots[kSlots];
    cudaStream_t s_in = nullptr, s_out = nullptr;
    uint64_t async_frames = 0;
    bool async_synced = true;  // the context's own result buffers hold the last pipelined frame
    // closed-loop prefetch (nav_slam_prefetch): the next frame is uploaded and labelled on the copy-in
    // stream while the current one is matched and fitted
    struct PreSlot {
        double *d_cloud = nullptr;
        int *d_labels = nullptr;
        int *raw[2] = {nullptr, nullptr};
        cudaEvent_t ready = nullptr, released = nullptr;
        const void *host_src = nullptr;  // identity of the prefetched frame
        bool pending = false;
        bool release_recorded = false;   // `released` already marks the end of the slot's last reader
    } pre[3];
    int pre_next = 0;
    PreSlot *cur_pre = nullptr;  // the prefetched slot the last localization call consumed
    // the frame the last localization call worked on (mapping with cloud == NULL maps this one)
    const double *cur_cloud = nullptr;
    int *cur_labels = nullptr;
    double *d_row_stats = nullptr;  // [n_seq*rows][5] per-row sufficient statistics of the translation fit
    double *d_tile_stats = nullptr; // [n_seq*rows*tiles][5] per-tile partial sums (k_dedupe_stats)
    // closed loop: the dedupe kernel posts the frame's five totals + a sequence number here (host-mapped,
    // polled by nav_slam_localization_fast instead of a copy + stream synchronisation)
    double *h_fit = nullptr;
    unsigned *d_fit_ticket = nullptr;
    unsigned long long fit_seq = 0;
    // poses of a sequence launch (nav_frontend_sequence_dev): device array + a ring of pinned staging buffers
    static constexpr int kPoseRing = 4;
    struct PoseRing {
        void *host = nullptr;
        size_t cap = 0;
        cudaEvent_t done = nullptr;
    } pose_ring[kPoseRing];
    int pose_ring_next = 0;
    void *d_pose = nullptr;
    size_t d_pose_cap = 0;
    int seq_path = -1;  // how the last sequence replay ran (nav_debug_sequence_path)
    // per-frame partials of the fit statistics of nav_frontend_sequence_out_dev (grows like d_pose)
    double *d_seq_part = nullptr;
    size_t d_seq_part_cap = 0;
    // the device closed loop (nav_slam_run_dev): pose records [2][n_seq] around the host tables [n_frames][n_seq]
    // (grows like d_pose), per-sequence tickets, and the second slot of the label ring (the first is d_labels)
    void *d_loop = nullptr;
    size_t d_loop_cap = 0;
    unsigned *d_loop_ticket = nullptr;
    int *d_labels_alt = nullptr;
    // depth / integer-mm frames of a per-frame replay, converted to xyz: two frame slots, so that a conversion never
    // overwrites the frame a kernel still in flight reads (lazy)
    double *d_conv = nullptr;
    bool fit_tables_queued = false;  // the fit's bias tables were uploaded on the context's stream (nav_set_stream
                                     // synchronises the old stream, so a later stream finds them in place)
    // NAV_RUN_TRACE=1: nav_slam_run prints where the host side of the closed loop spends its time
    // [prefetch call, launches of match + dedupe, wait for the statistics, fit, mapping call]
    bool trace = false;
    double trace_us[5] = {0, 0, 0, 0, 0};
    bool prof = false;
    ProfSlot prof_labels, prof_match, prof_map;
    // tie rule (nav_set_tie_rule).  NAV_TIE_REFERENCE: the match kernel lists its tied queries here (one record per
    // pixel at most), and the blocking calls re-answer them on the host with the reference's own search
    int tie_rule = NAV_TIE_LOWEST_INDEX;
    TieRec *d_tie_rec = nullptr;
    unsigned *d_tie_count = nullptr;
    int2 *d_tie_fix = nullptr;  // (pixel, nn_idx) answers of the host, one per record
    uint64_t tie_resolved = 0;
    double tie_ms[3] = {0, 0, 0};  // profiler (c->prof): host ms of the copies, the searches, the upload
    uint64_t tie_calls = 0;
};

static void rotation_from_pos(const nav_pos *pos, double R[9]) {
    // DEG2RAD(x) = x * M_PI / 180.0 (src/slam.c:8), then src/slam.c:95-115 with the host libm
    const double roll = pos->roll * M_PI / 180.0, pitch = pos->pitch * M_PI / 180.0,
                 yaw = pos->yaw * M_PI / 180.0;
    const double cr = cos(roll), sr = sin(roll), cp = cos(pitch), sp = sin(pitch), cy = cos(yaw),
                 sy = sin(yaw);
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

static PoseXf make_pose(const nav_pos *pos, const nav_pos *last) {
    PoseXf q;
    rotation_from_pos(pos, q.R);
    q.t[0] = pos->x;
    q.t[1] = pos->y;
    q.t[2] = pos->z;
    // transform[0..2] = pos_predict - pos_last (src/slam.c:84-88)
    q.shift[0] = last ? pos->x - last->x : 0.0;
    q.shift[1] = last ? pos->y - last->y : 0.0;
    q.shift[2] = last ? pos->z - last->z : 0.0;
    return q;
}

struct ProfScope {
    nav_ctx *c;
    ProfSlot *s;
    size_t slot = 0;
    ProfScope(nav_ctx *ctx, ProfSlot *ps) : c(ctx), s(ps) {
        if (!c->prof) return;
        if (s->used == s->ev.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            s->ev.push_back({a, b});
        }
        slot = s->used++;
        cudaEventRecord(s->ev[slot].first, c->stream);
    }
    ~ProfScope() {
        if (!c->prof) return;
        cudaEventRecord(s->ev[slot].second, c->stream);
    }
};

static void prof_collect(nav_ctx *c, ProfSlot *s) {
    if (s->used == 0) return;
    cudaStreamSynchronize(c->stream);
    for (size_t i = 0; i < s->used; ++i) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, s->ev[i].first, s->ev[i].second) == cudaSuccess) s->ms += ms;
        s->launches++;
    }
    s->used = 0;
}

extern "C" void nav_destroy(nav_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    void *ptrs[] = {c->d_cloud, c->d_global, c->d_curv, c->d_nn_dist, c->d_labels, c->d_nn_idx, c->map.pts,
                    c->map.mask, c->d_n_exact, c->map.box, c->map.sbox, c->map_alt.pts, c->map_alt.mask,
                    c->map_alt.box, c->map_alt.sbox, c->d_corr_rows, c->d_corr,
                    c->d_corr_row_count, c->d_corr_total, c->raw[0], c->raw[1], c->d_tan_col, c->d_tan_row, c->d_flat,
                    c->d_flat_count, c->d_tie_rec, c->d_tie_count, c->d_tie_fix};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    if (c->h_small) cudaFreeHost(c->h_small);
    if (c->d_csv) cudaFree(c->d_csv);
    if (c->d_csv_scratch) cudaFree(c->d_csv_scratch);
    for (auto &sl : c->slots) {
        for (void *p : {(void *)sl.d_cloud, (void *)sl.d_labels, (void *)sl.raw[0], (void *)sl.raw[1]})  // the other outputs live inside d_labels
            if (p) cudaFree(p);
        for (cudaEvent_t e : {sl.in_done, sl.compute_done, sl.out_done})
            if (e) cudaEventDestroy(e);
    }
    for (auto &ps : c->pre) {
        for (void *p : {(void *)ps.d_cloud, (void *)ps.d_labels, (void *)ps.raw[0], (void *)ps.raw[1]})
            if (p) cudaFree(p);
        for (cudaEvent_t e : {ps.ready, ps.released})
            if (e) cudaEventDestroy(e);
    }
    if (c->d_row_stats) cudaFree(c->d_row_stats);
    if (c->d_tile_stats) cudaFree(c->d_tile_stats);
    if (c->h_fit) cudaFreeHost(c->h_fit);
    for (auto &pr : c->pose_ring) {
        if (pr.host) cudaFreeHost(pr.host);
        if (pr.done) cudaEventDestroy(pr.done);
    }
    if (c->d_pose) cudaFree(c->d_pose);
    if (c->d_seq_part) cudaFree(c->d_seq_part);
    for (void *p : {c->d_loop, (void *)c->d_loop_ticket, (void *)c->d_labels_alt, (void *)c->d_conv})
        if (p) cudaFree(p);
    if (c->d_fit_ticket) cudaFree(c->d_fit_ticket);
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    c->stage.release();
    for (ProfSlot *s : {&c->prof_labels, &c->prof_match, &c->prof_map})
        for (auto &e : s->ev) {
            cudaEventDestroy(e.first);
            cudaEventDestroy(e.second);
        }
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

extern "C" nav_ctx *nav_create(int rows, int cols, int device, int n_seq) {
    if (rows < 1 || cols < 1 || n_seq < 1 || n_seq > NAV_MAX_SEQ) {
        fail("nav_create: bad shape %dx%d n_seq=%d (n_seq must be 1..%d)", rows, cols, n_seq, NAV_MAX_SEQ);
        return nullptr;
    }
    int ndev = nav_device_count();
    if (ndev == 0) {
        fail("nav_create: no CUDA device visible -- libnavslam_b200 has no CPU fallback");
        return nullptr;
    }
    if (device < 0 || device >= ndev) {
        fail("nav_create: device %d out of range (0..%d)", device, ndev - 1);
        return nullptr;
    }
    CUP(cudaSetDevice(device));
    nav_ctx *c = new nav_ctx();
    c->rows = rows;
    c->cols = cols;
    c->n_seq = n_seq;
    c->device = device;
    c->npx = (size_t)rows * cols;
    c->ntot = c->npx * n_seq;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    int max_smem = 0;
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (dedupe_smem_bytes(cols) > (size_t)max_smem) {
        fail("nav_create: %d columns need %zu B of shared memory per row CTA, device allows %d", cols,
             dedupe_smem_bytes(cols), max_smem);
        delete c;
        return nullptr;
    }
#define ALLOC(ptr, bytes)                                                             \
    if (cudaMalloc((void **)&(ptr), (bytes)) != cudaSuccess) {                        \
        fail("nav_create: cudaMalloc(%zu) failed for " #ptr, (size_t)(bytes));        \
        nav_destroy(c);                                                               \
        return nullptr;                                                               \
    }
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        fail("nav_create: cudaStreamCreate failed");
        delete c;
        return nullptr;
    }
    c->stream = c->own_stream;
    const size_t nt = c->ntot, nr = (size_t)n_seq * rows;
    c->map.n_chunks = div_up(cols, kChunk);
    c->map.n_super = div_up(c->map.n_chunks, kChunksPerSuper);
    ALLOC(c->d_cloud, nt * 24);
    ALLOC(c->d_labels, nt * 4);
    ALLOC(c->d_nn_idx, nt * 4);
    ALLOC(c->d_nn_dist, nt * 8);
    ALLOC(c->map.pts, nt * 24);
    ALLOC(c->map.mask, nr * c->map.n_chunks * 4);
    ALLOC(c->d_n_exact, 4);
    ALLOC(c->d_row_stats, nr * 5 * 8);
    ALLOC(c->d_tile_stats, nr * (size_t)div_up(cols, 256) * 5 * 8);
    ALLOC(c->map.box, nr * c->map.n_chunks * 32);
    ALLOC(c->map.sbox, nr * c->map.n_super * 32);
    c->map_alt.n_chunks = c->map.n_chunks;
    c->map_alt.n_super = c->map.n_super;
    ALLOC(c->map_alt.pts, nt * 24);
    ALLOC(c->map_alt.mask, nr * c->map.n_chunks * 4);
    ALLOC(c->map_alt.box, nr * c->map.n_chunks * 32);
    ALLOC(c->map_alt.sbox, nr * c->map.n_super * 32);
    ALLOC(c->d_corr_rows, nt * sizeof(nav_corr));
    ALLOC(c->d_corr, nt * sizeof(nav_corr));
    ALLOC(c->d_corr_row_count, nr * 4);
    ALLOC(c->d_corr_total, (size_t)n_seq * 4);
    ALLOC(c->raw[0], c->npx * 4);
    ALLOC(c->d_tan_col, (size_t)cols * 8);
    ALLOC(c->d_tan_row, (size_t)rows * 8);
    ALLOC(c->d_flat, (size_t)cols * 24 * 2 + (size_t)cols * 8);
    ALLOC(c->d_flat_count, 4);
    ALLOC(c->d_fit_ticket, 4);
#undef ALLOC
    cudaMemsetAsync(c->map.mask, 0, nr * c->map.n_chunks * 4, c->stream);
    cudaMemsetAsync(c->d_n_exact, 0, 4, c->stream);
    cudaMemsetAsync(c->d_fit_ticket, 0, 4, c->stream);
    if (cudaHostAlloc((void **)&c->h_small, 4096, cudaHostAllocDefault) != cudaSuccess ||
        cudaHostAlloc((void **)&c->h_fit, 64, cudaHostAllocMapped) != cudaSuccess) {
        fail("nav_create: pinned scratch allocation failed");
        nav_destroy(c);
        return nullptr;
    }
    // the mailbox flag (h_fit[5]) must not hold a sequence number the host will wait for before any post
    memset(c->h_fit, 0, 64);
    // tan tables of utils/pointcloud.c:10-41, evaluated with the host libm exactly as the reference
    {
        std::vector<double> tc(cols), tr(rows);
        const double fov = 45.0;
        const double col_step = fov / (cols - 1), row_step = fov / (rows - 1);
        for (int i = 0; i < cols; ++i) {
            double theta = -fov / 2.0 + i * col_step;
            theta = theta * M_PI / 180.0;
            tc[i] = tan(theta);
        }
        for (int j = 0; j < rows; ++j) {
            double phi = -fov / 2.0 + j * row_step;
            phi = phi * M_PI / 180.0;
            tr[j] = tan(phi);
        }
        cudaMemcpy(c->d_tan_col, tc.data(), (size_t)cols * 8, cudaMemcpyHostToDevice);
        cudaMemcpy(c->d_tan_row, tr.data(), (size_t)rows * 8, cudaMemcpyHostToDevice);
    }
    if (configure_row_kernels(cols) != 0) {
        fail("nav_create: cannot opt in to %zu B dynamic shared memory", dedupe_smem_bytes(cols));
        nav_destroy(c);
        return nullptr;
    }
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) {
        fail("nav_create: device initialisation failed: %s", cudaGetErrorString(cudaGetLastError()));
        nav_destroy(c);
        return nullptr;
    }
    return c;
}

extern "C" int nav_rows(const nav_ctx *c) { return c ? c->rows : 0; }
extern "C" int nav_cols(const nav_ctx *c) { return c ? c->cols : 0; }
extern "C" uint64_t nav_launch_count(const nav_ctx *c) { return c ? c->launches : 0; }

extern "C" int nav_set_stream(nav_ctx *c, void *s, int use_own) {
    if (!c) return fail("nav_set_stream: null context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    c->stream = use_own ? c->own_stream : (cudaStream_t)s;  // s == 0 is the legacy default stream
    return 0;
}

extern "C" int nav_synchronize(nav_ctx *c) {
    if (!c) return fail("nav_synchronize: null context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int nav_profile_enable(nav_ctx *c, int on) {
    if (!c) return fail("nav_profile_enable: null context");
    c->prof = on != 0;
    return 0;
}

extern "C" int nav_profile_read(nav_ctx *c, const char *name, double *ms, uint64_t *launches, int reset) {
    if (!c || !name) return fail("nav_profile_read: null argument");
    const char *tie_names[3] = {"tie_copies", "tie_search", "tie_upload"};
    for (int i = 0; i < 3; ++i)
        if (!strcmp(name, tie_names[i])) {
            if (ms) *ms = c->tie_ms[i];
            if (launches) *launches = c->tie_calls;
            if (reset) {
                c->tie_ms[i] = 0;
                if (i == 2) c->tie_calls = 0;
            }
            return 0;
        }
    ProfSlot *s = !strcmp(name, "labels") ? &c->prof_labels
                  : !strcmp(name, "match") ? &c->prof_match
                  : !strcmp(name, "map")   ? &c->prof_map
                                           : nullptr;
    if (!s) return fail("nav_profile_read: unknown kernel '%s'", name);
    prof_collect(c, s);
    if (ms) *ms = s->ms;
    if (launches) *launches = s->launches;
    if (reset) {
        s->ms = 0;
        s->launches = 0;
    }
    return 0;
}

#define CTX_ENTER(c, name)                                  \
    if (!(c)) return fail(name ": null context");           \
    CU(cudaSetDevice((c)->device));

static int finish_call(nav_ctx *c, const char *name) {
    if (c->stage.finish(c->stream)) {
        cudaError_t e = cudaGetLastError();
        return fail("%s: device execution failed: %s", name, cudaGetErrorString(e));
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("%s: %s", name, cudaGetErrorString(e));
    return 0;
}

// device-side building blocks (no sync) -------------------------------------------------------
static void run_labels(nav_ctx *c, const double *d_cloud, int *d_labels, double *d_curv, size_t n_images) {
    ProfScope ps(c, &c->prof_labels);
    launch_labels(d_cloud, d_labels, d_curv, (long long)n_images * c->rows, c->cols, c->sm_count, c->d_n_exact,
                  c->stream);
    c->launches++;
}

// a synchronous entry point that touches the maps must not overtake the downloads of pipelined frames
// still reading them (nav_frontend_submit): order the context's stream behind those copies
static void order_after_async(nav_ctx *c) {
    if (!c->async_frames || c->async_synced) return;
    for (auto &sl : c->slots)
        if (sl.out_done) cudaStreamWaitEvent(c->stream, sl.out_done, 0);
}

// transform + label masks + boxes of the frame whose labels are in d_labels (a7 + a4/a5)
static void run_map(nav_ctx *c, const double *d_cloud, const int *d_labels, const PoseBatch &poses) {
    order_after_async(c);
    ProfScope ps(c, &c->prof_map);
    launch_frame_map(d_cloud, d_labels, c->map, poses, c->n_seq, c->rows, c->cols, c->stream);
    c->launches++;
    c->have_map = true;
}

// ---- the reference tie rule (NAV_TIE_REFERENCE) ------------------------------------------------------------------
// The device search keeps the lowest column among equal dsq.  The reference keeps the first point of the smallest
// rounded distance sqrt(dsq) that the depth-first search of its per-row tree reaches.  The two differ only where two
// map points of the row share that smallest rounded distance; the match kernel's kRefTies variant lists exactly those
// queries, and resolve_ties re-answers them here with the reference's own tree and search, built per call for the
// rows the list names (no tree outlives the call, so no map update can leave a stale one behind).
// Host code compiled with -ffp-contract=off, like adam_fit: every operation rounds as the reference's does.
static double ref_key(const nav_point &p, int axis) { return axis == 0 ? p.x : (axis == 1 ? p.y : p.z); }

// utils/kdtree.c:20-62: Lomuto partition with the last element as pivot, (key - pivot) <= 0 to the front
static void ref_select(nav_point *p, size_t first, size_t last, size_t nth, int axis) {
    while (first < last) {
        const double pivot = ref_key(p[last], axis);
        size_t store = first;
        for (size_t j = first; j < last; ++j) {
            const double cmp = ref_key(p[j], axis) - pivot;
            if (cmp <= 0) {
                std::swap(p[store], p[j]);
                ++store;
            }
        }
        std::swap(p[store], p[last]);
        if (store == nth) return;
        if (store < nth)
            first = store + 1;
        else
            last = store - 1;
    }
}

// utils/kdtree.c:65-82 in place: the node of p[0..n) is p[n/2] (axis depth % 3), its children are p[0..m) and
// p[m+1..n) -- the pointer tree of the reference, laid out as the array it was selected in
static void ref_build(nav_point *p, size_t n, int depth) {
    if (n == 0) return;
    const size_t m = n / 2;
    ref_select(p, 0, n - 1, m, depth % 3);
    ref_build(p, m, depth + 1);
    ref_build(p + m + 1, n - m - 1, depth + 1);
}

// utils/kdtree.c:110-152: dist = sqrt((dx*dx + dy*dy) + dz*dz) with root - target, update on strict '<', near side
// first, far side iff fabs(delta) < best
static void ref_nn(const nav_point *p, size_t n, int depth, const nav_point &q, nav_point &best, double &best_dist) {
    if (n == 0) return;
    const size_t m = n / 2;
    const nav_point &r = p[m];
    const double dx = r.x - q.x, dy = r.y - q.y, dz = r.z - q.z;
    const double d = sqrt(dx * dx + dy * dy + dz * dz);
    if (d < best_dist) {
        best_dist = d;
        best = r;
    }
    const int axis = depth % 3;
    const double delta = ref_key(q, axis) - ref_key(r, axis);
    const nav_point *lo = p, *hi = p + m + 1;
    const size_t n_lo = m, n_hi = n - m - 1;
    if (delta < 0) {
        ref_nn(lo, n_lo, depth + 1, q, best, best_dist);
        if (fabs(delta) < best_dist) ref_nn(hi, n_hi, depth + 1, q, best, best_dist);
    } else {
        ref_nn(hi, n_hi, depth + 1, q, best, best_dist);
        if (fabs(delta) < best_dist) ref_nn(lo, n_lo, depth + 1, q, best, best_dist);
    }
}

// After a match launched with the tie list: re-answers the listed queries against `map` (the map that launch searched)
// and rewrites their entries of d_nn_idx on the context's stream.  nn_dist needs no change: the reference's minimum is
// the device's.  Synchronises the stream once (twice when something is listed).
static double now_us();
static int resolve_ties(nav_ctx *c, const RowMap &map, int *d_nn_idx, const char *name) {
    CU(cudaMemcpyAsync(c->h_small, c->d_tie_count, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const size_t n = (size_t)(unsigned)c->h_small[0];
    if (n == 0) return 0;
    if (n > c->ntot) return fail("%s: tie list overflow (%zu records for %zu pixels)", name, n, c->ntot);
    double t[4] = {c->prof ? now_us() : 0.0, 0.0, 0.0, 0.0};
    const size_t cols = (size_t)c->cols, n_chunks = (size_t)map.n_chunks;
    std::vector<TieRec> rec(n);
    CU(cudaMemcpyAsync(rec.data(), c->d_tie_rec, n * sizeof(TieRec), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    // the searched rows the list names, in order; records grouped by row (stable: the list order is the device's)
    std::stable_sort(rec.begin(), rec.end(), [&](const TieRec &a, const TieRec &b) {
        return a.px / (long long)cols < b.px / (long long)cols;
    });
    std::vector<long long> rids;
    for (const TieRec &r : rec)
        if (rids.empty() || rids.back() != r.px / (long long)cols) rids.push_back(r.px / (long long)cols);
    std::vector<nav_point> row_pts(rids.size() * cols);
    std::vector<unsigned> row_mask(rids.size() * n_chunks);
    for (size_t i = 0; i < rids.size(); ++i) {
        CU(cudaMemcpyAsync(&row_pts[i * cols], map.pts + rids[i] * cols * 3, cols * 24, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(&row_mask[i * n_chunks], map.mask + rids[i] * n_chunks, n_chunks * 4, cudaMemcpyDeviceToHost,
                           c->stream));
    }
    CU(cudaStreamSynchronize(c->stream));
    if (c->prof) t[1] = now_us();
    std::vector<int2> fix(n);
    std::vector<nav_point> flat(cols), tree(cols);
    std::vector<int> flat_col(cols);
    size_t k = 0;
    for (size_t i = 0; i < rids.size(); ++i) {
        // flattenedPoints (src/slam.c:170-171): the row's labelled map points in column order, as k_flatten_row
        // compacts them for nav_row_map_export
        size_t m = 0;
        for (size_t col = 0; col < cols; ++col)
            if ((row_mask[i * n_chunks + col / kChunk] >> (col % kChunk)) & 1u) {
                flat[m] = row_pts[i * cols + col];
                flat_col[m++] = (int)col;
            }
        std::copy(flat.begin(), flat.begin() + m, tree.begin());  // the reference builds on a copy of the row
        ref_build(tree.data(), m, 0);
        const int row = (int)(rids[i] % c->rows);
        for (; k < n && rec[k].px / (long long)cols == rids[i]; ++k) {
            const nav_point q = {rec[k].q[0], rec[k].q[1], rec[k].q[2]};
            nav_point near = {0.0, 0.0, 0.0};
            double best = INFINITY;
            ref_nn(tree.data(), m, 0, q, near, best);
            // the new match: the lowest column whose map point is the returned xyz (as the oracle's row_query)
            int col = -1;
            for (size_t j = 0; j < m && col < 0; ++j)
                if (flat[j].x == near.x && flat[j].y == near.y && flat[j].z == near.z) col = flat_col[j];
            if (!(best < INFINITY) || col < 0)
                return fail("%s: a tied query of row %lld found no map point in the reference search", name, rids[i]);
#ifndef NDEBUG
            // the reference's minimum is the device's sqrt(best), the smallest rounded distance of the row
            double brute = INFINITY;
            for (size_t j = 0; j < m; ++j) {
                const double dx = flat[j].x - q.x, dy = flat[j].y - q.y, dz = flat[j].z - q.z;
                brute = fmin(brute, sqrt(dx * dx + dy * dy + dz * dz));
            }
            assert(best == brute);
#endif
            fix[k] = make_int2((int)(rec[k].px), row * c->cols + col);
        }
    }
    c->tie_resolved += n;
    if (c->prof) t[2] = now_us();
    // a pageable source: the copy has left `fix` when the call returns
    CU(cudaMemcpyAsync(c->d_tie_fix, fix.data(), n * sizeof(int2), cudaMemcpyHostToDevice, c->stream));
    launch_apply_tie_fix(c->d_tie_fix, (int)n, d_nn_idx, c->stream);
    c->launches++;
    if (c->prof) {
        t[3] = now_us();
        for (int i = 0; i < 3; ++i) c->tie_ms[i] += (t[i + 1] - t[i]) * 1e-3;
        c->tie_calls++;
    }
    return 0;
}

static int refuse_ref_ties(const char *name) {
    return fail("%s: not available under the reference tie rule (NAV_TIE_REFERENCE): this call runs without a host "
                "round trip, and the rule resolves ties on the host; use the blocking calls, or the lowest-index rule",
                name);
}
#define REFUSE_UNDER_REF_TIES(c, name) \
    if ((c) && (c)->tie_rule == NAV_TIE_REFERENCE) return refuse_ref_ties(name);

// one match launch against c->map: labels (a3: fused into the match kernel, or already in d_labels) + queries (a7) +
// exact per-row NN (a6).  fin != null: the next map from the final poses (a7, a4/a5) into c->map_alt, after which the
// two maps change places.  ref_ties (the calling API's name; fused labels only): the reference tie rule -- the tied
// queries are re-answered on the host against the map that was searched (a blocking step).
static int run_frame_match(nav_ctx *c, const double *d_cloud, int *d_labels, bool fused_labels, const MatchOut &out,
                           const PoseBatch &poses, const PoseBatch *fin, bool pdl, const char *ref_ties) {
    const TieList ties = {c->d_tie_rec, c->d_tie_count};
    if (ref_ties) CU(cudaMemsetAsync(c->d_tie_count, 0, 4, c->stream));
    {
        ProfScope ps(c, &c->prof_match);
        launch_frame_match(d_cloud, d_labels, fused_labels, c->map, out, poses, c->n_seq, c->rows, c->cols,
                           c->d_n_exact, c->stream, fin ? &c->map_alt : nullptr, fin, pdl, ref_ties ? &ties : nullptr);
    }
    c->launches++;
    if (fin) std::swap(c->map, c->map_alt);  // the search read the map that is map_alt now
    return ref_ties ? resolve_ties(c, fin ? c->map_alt : c->map, out.nn_idx, ref_ties) : 0;
}

// the match (run_frame_match), then the per-row dedupe (a8) producing the correspondence list and/or the per-row fit
// statistics; under the reference tie rule the dedupe reads the host's answers
enum { kDedupeNone = 0, kDedupeCorr = 1, kDedupeStats = 2 };
static int run_match(nav_ctx *c, const double *d_cloud, int *d_labels, bool fused_labels, const PoseBatch &poses,
                     int dedupe, const FitMailbox *mail = nullptr, const char *ref_ties = nullptr) {
    order_after_async(c);
    MatchOut out = {c->d_nn_idx, c->d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
    if (run_frame_match(c, d_cloud, d_labels, fused_labels, out, poses, nullptr, false, ref_ties)) return 1;
    if (dedupe & kDedupeCorr) {
        launch_dedupe(d_cloud, d_labels, c->map, out, poses, c->n_seq, c->rows, c->cols, c->stream,
                      (dedupe & kDedupeStats) ? c->d_row_stats : nullptr, true);
        launch_gather_corr(c->d_corr_rows, c->d_corr_row_count, c->d_corr, c->d_corr_total, c->n_seq, c->rows,
                           c->cols, c->stream);
        c->launches += 2;
    } else if (dedupe & kDedupeStats) {
        if (mail && c->n_seq == 1 && row_cluster_supported(c->cols))
            launch_dedupe_stats(d_cloud, d_labels, c->map, out, poses, c->n_seq, c->rows, c->cols, c->stream,
                                c->d_tile_stats, *mail);
        else
            launch_dedupe(d_cloud, d_labels, c->map, out, poses, c->n_seq, c->rows, c->cols, c->stream, c->d_row_stats,
                          false, mail);
        c->launches += 1;
    }
    return 0;
}

static PoseBatch pose_batch(const nav_ctx *c, const nav_pos *pos, const nav_pos *last);

// the whole front-end frame in ONE launch: labels (a3) + queries (a7) + exact per-row NN against the
// current map (a6) + the next map from the final pose (a7, a4/a5) into the other map buffer
// ref_ties: the reference tie rule (blocking; see run_match)
static int run_frame_fused(nav_ctx *c, const double *d_cloud, int *d_labels, int *d_nn_idx, double *d_nn_dist,
                           const nav_pos *pos_predict, const nav_pos *pos_last, const nav_pos *pos_final,
                           bool pdl = false, const char *ref_ties = nullptr) {
    const MatchOut out = {d_nn_idx, d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
    const PoseBatch loc = pose_batch(c, pos_predict, pos_last), fin = pose_batch(c, pos_final, nullptr);
    return run_frame_match(c, d_cloud, d_labels, true, out, loc, &fin, pdl && !c->prof, ref_ties);
}

static PoseBatch pose_batch(const nav_ctx *c, const nav_pos *pos, const nav_pos *last) {
    PoseBatch b;
    memset(&b, 0, sizeof(b));
    for (int s = 0; s < c->n_seq; ++s) b.p[s] = make_pose(&pos[s], last ? &last[s] : nullptr);
    return b;
}

// ------------------------------------------------------------------ frame formats -----------
// A frame (n_seq images) comes as xyz doubles (NAV_RUN_INPUT_XYZ, 24 B/point), a depth matrix (NAV_RUN_INPUT_DEPTH,
// int32, 4 B/pixel) or integer-mm xyz (NAV_RUN_INPUT_MM, int32 x 3, 12 B/point).  The int32 formats cross PCIe raw and
// become xyz on the device (to_xyz), or are read raw by the sequence and device-loop kernels.

// bytes of one element (a double of xyz, an int32 otherwise) and of one frame of `kind`
static size_t elem_bytes(int kind) { return kind == NAV_RUN_INPUT_XYZ ? sizeof(double) : sizeof(int); }
static size_t frame_bytes(const nav_ctx *c, int kind) {
    return c->ntot * elem_bytes(kind) * (kind == NAV_RUN_INPUT_DEPTH ? 1 : 3);
}

// frame f of a device-resident recording (frames back to back)
static const void *frame_at(const nav_ctx *c, const void *frames, int kind, size_t f) {
    return (const unsigned char *)frames + f * frame_bytes(c, kind);
}

// The frame formats of the device-resident calls: a kind other than the three, or a frame pointer off its element's
// alignment (8 bytes for xyz doubles, 4 for int32), is refused before anything is queued.
static int check_frame_input(const char *name, const void *frames, int kind) {
    if (kind != NAV_RUN_INPUT_XYZ && kind != NAV_RUN_INPUT_DEPTH && kind != NAV_RUN_INPUT_MM)
        return fail("%s: input_kind %d is none of NAV_RUN_INPUT_XYZ (0), NAV_RUN_INPUT_DEPTH (1), NAV_RUN_INPUT_MM (2)",
                    name, kind);
    const unsigned align = (unsigned)elem_bytes(kind);
    if (((uintptr_t)frames & (align - 1u)) != 0)
        return fail("%s: the frame pointer %p is not %u-byte aligned", name, frames, align);
    return 0;
}

// where a raw frame of `kind` is uploaded: slot [0] (depth) or [1] (integer mm) of its holder's pair, allocated at
// frame_bytes on first use.  NULL, with the error set, if that allocation fails.
static int *raw_buf(const nav_ctx *c, int *(&raw)[2], int kind) {
    int *&p = raw[kind == NAV_RUN_INPUT_MM];
    if (!p) CUP(cudaMalloc((void **)&p, frame_bytes(c, kind)));
    return p;
}

// n_img images of depth or integer-mm xyz at `raw` -> xyz doubles, on `stream`: k_convert (a2) or k_widen_mm, the
// arithmetic the in-kernel conversion of k_frame_seq / k_loop_step shares.  The caller orders `stream`.
static void to_xyz(nav_ctx *c, int kind, const int *raw, double *xyz, int n_img, cudaStream_t stream) {
    if (kind == NAV_RUN_INPUT_DEPTH)
        launch_convert(raw, c->d_tan_col, c->d_tan_row, xyz, c->rows, c->cols, n_img, c->sm_count, stream);
    else
        launch_widen_mm(raw, xyz, (long long)(n_img * c->npx), c->sm_count, stream);
    c->launches++;
}

// ------------------------------------------------------------------ function level ----------
extern "C" int nav_convert_to_pointcloud(nav_ctx *c, const int *distances, nav_point *cloud_out) {
    CTX_ENTER(c, "nav_convert_to_pointcloud");
    if (!distances || !cloud_out) return fail("nav_convert_to_pointcloud: null argument");
    if (c->stage.reserve(c->npx * 28 + 512, c->stream)) return fail("nav_convert_to_pointcloud: staging");
    if (c->stage.h2d(c->raw[0], distances, c->npx * 4, c->stream)) return fail("nav_convert_to_pointcloud: H2D");
    to_xyz(c, NAV_RUN_INPUT_DEPTH, c->raw[0], c->d_cloud, 1, c->stream);  // one image, whatever n_seq
    c->cloud_resident = false;
    if (c->stage.d2h(cloud_out, c->d_cloud, c->npx * 24, c->stream)) return fail("nav_convert_to_pointcloud: D2H");
    return finish_call(c, "nav_convert_to_pointcloud");
}

extern "C" int nav_extract_feature(nav_ctx *c, const nav_point *cloud, int *feature) {
    CTX_ENTER(c, "nav_extract_feature");
    if (!cloud || !feature) return fail("nav_extract_feature: null argument");
    if (c->stage.reserve(c->npx * 28 + 512, c->stream)) return fail("nav_extract_feature: staging");
    if (c->stage.h2d(c->d_cloud, cloud, c->npx * 24, c->stream)) return fail("nav_extract_feature: H2D");
    c->cloud_resident = false;
    run_labels(c, c->d_cloud, c->d_labels, nullptr, 1);
    int *lab = (int *)c->stage.take(c->npx * 4, c->stream);
    if (!lab) return fail("nav_extract_feature: staging");
    CU(cudaMemcpyAsync(lab, c->d_labels, c->npx * 4, cudaMemcpyDeviceToHost, c->stream));
    if (finish_call(c, "nav_extract_feature")) return 1;
    // the reference only ever stores 1s (src/slam.c:58); whatever the caller had elsewhere stays
    for (size_t i = 0; i < c->npx; ++i)
        if (lab[i]) feature[i] = 1;
    return 0;
}

extern "C" int nav_curvature(nav_ctx *c, const nav_point *cloud, double *curv_out) {
    CTX_ENTER(c, "nav_curvature");
    if (!cloud || !curv_out) return fail("nav_curvature: null argument");
    if (!c->d_curv) CU(cudaMalloc((void **)&c->d_curv, c->npx * 8));
    if (c->stage.reserve(c->npx * 32 + 512, c->stream)) return fail("nav_curvature: staging");
    if (c->stage.h2d(c->d_cloud, cloud, c->npx * 24, c->stream)) return fail("nav_curvature: H2D");
    c->cloud_resident = false;
    run_labels(c, c->d_cloud, c->d_labels, c->d_curv, 1);
    if (c->stage.d2h(curv_out, c->d_curv, c->npx * 8, c->stream)) return fail("nav_curvature: D2H");
    return finish_call(c, "nav_curvature");
}

extern "C" int nav_flatten_points(nav_ctx *c, const nav_point *row_points, const int *row_feature,
                                  nav_point *flattened_out, size_t *num_points_out) {
    CTX_ENTER(c, "nav_flatten_points");
    if (!row_points || !row_feature || !flattened_out || !num_points_out)
        return fail("nav_flatten_points: null argument");
    const size_t cols = c->cols;
    double *d_in = c->d_flat, *d_out = c->d_flat + cols * 3;
    int *d_feat = (int *)(c->d_flat + cols * 6);  // followed by cols ints of column scratch
    if (c->stage.reserve(cols * 56 + 1024, c->stream)) return fail("nav_flatten_points: staging");
    if (c->stage.h2d(d_in, row_points, cols * 24, c->stream)) return fail("nav_flatten_points: H2D");
    if (c->stage.h2d(d_feat, row_feature, cols * 4, c->stream)) return fail("nav_flatten_points: H2D");
    launch_flatten_row(d_in, d_feat, nullptr, d_out, nullptr, c->d_flat_count, c->cols, c->stream);
    c->launches++;
    CU(cudaMemcpyAsync(c->h_small, c->d_flat_count, 4, cudaMemcpyDeviceToHost, c->stream));
    unsigned char *tmp = c->stage.take(cols * 24, c->stream);
    if (!tmp) return fail("nav_flatten_points: staging");
    CU(cudaMemcpyAsync(tmp, d_out, cols * 24, cudaMemcpyDeviceToHost, c->stream));
    if (finish_call(c, "nav_flatten_points")) return 1;
    const size_t n = (size_t)c->h_small[0];
    memcpy(flattened_out, tmp, n * 24);  // like the reference, entries past n are left untouched
    *num_points_out = n;
    return 0;
}

extern "C" int nav_transform_cloud(nav_ctx *c, const nav_point *cloud, const nav_pos *pos, nav_point *global_out) {
    CTX_ENTER(c, "nav_transform_cloud");
    if (!cloud || !pos || !global_out) return fail("nav_transform_cloud: null argument");
    if (!c->d_global) CU(cudaMalloc((void **)&c->d_global, c->npx * 24));
    if (c->stage.reserve(c->npx * 48 + 512, c->stream)) return fail("nav_transform_cloud: staging");
    if (c->stage.h2d(c->d_cloud, cloud, c->npx * 24, c->stream)) return fail("nav_transform_cloud: H2D");
    c->cloud_resident = false;
    launch_transform(c->d_cloud, c->d_global, (long long)c->npx, make_pose(pos, nullptr), c->sm_count, c->stream);
    c->launches++;
    if (c->stage.d2h(global_out, c->d_global, c->npx * 24, c->stream)) return fail("nav_transform_cloud: D2H");
    return finish_call(c, "nav_transform_cloud");
}

// ------------------------------------------------------------------ SLAM step ----------------
// the frame nav_slam_mapping(pos, NULL, ...) maps from now on: the one in the context's own buffers, or (pre != null)
// the prefetched frame of slot `pre`, which is then no longer waiting
static void set_current_frame(nav_ctx *c, nav_ctx::PreSlot *pre = nullptr) {
    if (pre) pre->pending = false;
    c->cur_pre = pre;
    c->cur_cloud = pre ? pre->d_cloud : c->d_cloud;
    c->cur_labels = pre ? pre->d_labels : c->d_labels;
    c->cloud_resident = true;
}

static int upload_cloud(nav_ctx *c, const nav_point *cloud, const char *name) {
    if (c->stage.h2d(c->d_cloud, cloud, c->ntot * 24, c->stream)) return fail("%s: H2D of the cloud failed", name);
    return 0;
}

extern "C" int nav_slam_init(nav_ctx *c, const nav_pos *pos, const nav_point *cloud, nav_point *global_out) {
    CTX_ENTER(c, "nav_slam_init");
    if (!pos || !cloud) return fail("nav_slam_init: null argument");
    if (c->stage.reserve(c->ntot * 48 + 1024, c->stream)) return fail("nav_slam_init: staging");
    for (auto &ps : c->pre) ps.pending = false;  // a new sequence starts: frames prefetched for the old one are dropped
    if (upload_cloud(c, cloud, "nav_slam_init")) return 1;
    run_labels(c, c->d_cloud, c->d_labels, nullptr, c->n_seq);
    run_map(c, c->d_cloud, c->d_labels, pose_batch(c, pos, nullptr));
    set_current_frame(c);
    if (global_out && c->stage.d2h(global_out, c->map.pts, c->ntot * 24, c->stream))
        return fail("nav_slam_init: D2H");
    return finish_call(c, "nav_slam_init");
}

// nav_slam_init_dev (xyz) and nav_slam_init_dev_ex; `name` is the entry point the caller used
static int slam_init_dev(nav_ctx *c, const char *name, const void *dev_frame, int kind, const nav_pos *pos) {
    if (!pos || !dev_frame) return fail("%s: null argument", name);
    if (check_frame_input(name, dev_frame, kind)) return 1;
    for (auto &ps : c->pre) ps.pending = false;
    const double *cloud = (const double *)dev_frame;
    if (kind != NAV_RUN_INPUT_XYZ) {  // converted into the context's cloud buffer, then labelled and mapped as xyz
        order_after_async(c);
        to_xyz(c, kind, (const int *)dev_frame, c->d_cloud, c->n_seq, c->stream);
        cloud = c->d_cloud;
    }
    run_labels(c, cloud, c->d_labels, nullptr, c->n_seq);
    run_map(c, cloud, c->d_labels, pose_batch(c, pos, nullptr));
    c->cloud_resident = false;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int nav_slam_init_dev(nav_ctx *c, const void *dev_cloud, const nav_pos *pos) {
    CTX_ENTER(c, "nav_slam_init_dev");
    return slam_init_dev(c, "nav_slam_init_dev", dev_cloud, NAV_RUN_INPUT_XYZ, pos);
}

extern "C" int nav_slam_init_dev_ex(nav_ctx *c, const void *dev_frame, int input_kind, const nav_pos *pos) {
    CTX_ENTER(c, "nav_slam_init_dev_ex");
    return slam_init_dev(c, "nav_slam_init_dev_ex", dev_frame, input_kind, pos);
}

extern "C" int nav_slam_match(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict,
                              const nav_pos *pos_last, nav_corr *corr_out, size_t corr_cap, size_t *n_corr_out) {
    CTX_ENTER(c, "nav_slam_match");
    if (!cloud || !pos_predict || !pos_last || !n_corr_out) return fail("nav_slam_match: null argument");
    if (c->n_seq != 1) return fail("nav_slam_match: host correspondence lists need n_seq == 1");
    if (!c->have_map) return fail("nav_slam_match: call nav_slam_init first");
    if (c->stage.reserve(c->ntot * 24 + c->ntot * sizeof(nav_corr) + 1024, c->stream))
        return fail("nav_slam_match: staging");
    if (upload_cloud(c, cloud, "nav_slam_match")) return 1;
    if (run_match(c, c->d_cloud, c->d_labels, true, pose_batch(c, pos_predict, pos_last), kDedupeCorr, nullptr,
                  c->tie_rule == NAV_TIE_REFERENCE ? "nav_slam_match" : nullptr))
        return 1;
    set_current_frame(c);
    CU(cudaMemcpyAsync(c->h_small, c->d_corr_total, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const size_t n = (size_t)c->h_small[0];
    *n_corr_out = n;
    const size_t take = n < corr_cap ? n : corr_cap;
    if (corr_out && take && c->stage.d2h(corr_out, c->d_corr, take * sizeof(nav_corr), c->stream))
        return fail("nav_slam_match: D2H");
    return finish_call(c, "nav_slam_match");
}

// the reference's translation-only Adam fit, src/slam.c:218-379, on the deduped correspondences.
// Sequential binary64 sums in list order: bit-identical to the reference by construction.
static void adam_fit(const nav_corr *res, size_t count, double transform[6], double *error_out, int verbose) {
    const double lr = 0.1, tol = 1e-6, b1 = 0.9, b2 = 0.999, eps = 1e-8;
    double m[3] = {0, 0, 0}, v[3] = {0, 0, 0};
    double prev = 0, total = 0;
    int valid = 0;
    for (int iter = 0; iter < 200; ++iter) {
        double g[3] = {0.0, 0.0, 0.0};
        total = 0;
        valid = 0;
        for (size_t i = 0; i < count; ++i) {
            const double dx = (res[i].ori.x - transform[0]) - res[i].nearest.x;
            const double dy = (res[i].ori.y - transform[1]) - res[i].nearest.y;
            const double dz = (res[i].ori.z - transform[2]) - res[i].nearest.z;
            total += dx * dx + dy * dy + dz * dz;
            g[0] -= dx;
            g[1] -= dy;
            g[2] -= dz;
            ++valid;
        }
        if (fabs(total - prev) < tol) {
            if (verbose) printf("收敛，停止迭代！\n");
            break;
        }
        prev = total;
        if (valid > 0) {
            g[0] /= valid;
            g[1] /= valid;
            g[2] /= valid;
        }
        const int t = iter + 1;
        for (int j = 0; j < 3; ++j) {
            m[j] = b1 * m[j] + (1 - b1) * g[j];
            v[j] = b2 * v[j] + (1 - b2) * g[j] * g[j];
            const double mh = m[j] / (1 - pow(b1, t));
            const double vh = v[j] / (1 - pow(b2, t));
            transform[j] -= lr * mh / (sqrt(vh) + eps);
        }
        if (verbose) printf("Iteration %d, Total Error: %.6f\n", iter, total);
    }
    *error_out = valid > 0 ? sqrt(total / valid) : 0.0;
}

extern "C" int nav_slam_localization(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict,
                                     const nav_pos *pos_last, nav_pos *pos_out, double *error_out, int verbose) {
    CTX_ENTER(c, "nav_slam_localization");
    if (!pos_out) return fail("nav_slam_localization: null argument");
    static thread_local std::vector<nav_corr> corr;
    corr.resize(c->npx);
    size_t n = 0;
    if (nav_slam_match(c, cloud, pos_predict, pos_last, corr.data(), corr.size(), &n)) return 1;
    double transform[6] = {pos_predict->x - pos_last->x,       pos_predict->y - pos_last->y,
                           pos_predict->z - pos_last->z,       pos_predict->roll - pos_last->roll,
                           pos_predict->pitch - pos_last->pitch, pos_predict->yaw - pos_last->yaw};
    double err = 0.0;
    adam_fit(corr.data(), n, transform, &err, verbose);
    if (error_out) *error_out = err;
    pos_out->x = pos_last->x + transform[0];
    pos_out->y = pos_last->y + transform[1];
    pos_out->z = pos_last->z + transform[2];
    pos_out->roll = pos_last->roll + transform[3];
    pos_out->pitch = pos_last->pitch + transform[4];
    pos_out->yaw = pos_last->yaw + transform[5];
    return 0;
}

// ---- closed loop with prefetch -------------------------------------------------------------------------
// The reference's loop is serial in the pose (src/main.c:300-318: localization(t) needs pose(t-1), mapping(t)
// needs pose(t)), but uploading frame t+1 and labelling it (a3 is pose independent) need neither.
// nav_slam_prefetch queues both on the copy-in stream, so they run under frame t's match, download and
// host fit; nav_slam_localization_fast then finds the frame resident and labelled.

static int pre_setup(nav_ctx *c) {
    if (c->pre[0].d_cloud) return 0;
    if (!c->s_in) CU(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
    for (auto &ps : c->pre) {
        CU(cudaMalloc((void **)&ps.d_cloud, c->ntot * 24));
        CU(cudaMalloc((void **)&ps.d_labels, c->ntot * 4));
        CU(cudaEventCreateWithFlags(&ps.ready, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ps.released, cudaEventDisableTiming));
    }
    return 0;
}

// src: a host frame of `kind` (NAV_RUN_INPUT_*; depth needs n_seq == 1)
static int prefetch_common(nav_ctx *c, const char *name, int kind, const void *src) {
    if (!src) return fail("%s: null argument", name);
    if (kind == NAV_RUN_INPUT_DEPTH && c->n_seq != 1) return fail("%s: depth input needs n_seq == 1", name);
    if (!Stager::is_pinned(src)) return fail("%s: the host buffer must be pinned (nav_host_alloc / cudaHostRegister)", name);
    if (pre_setup(c)) return 1;
    nav_ctx::PreSlot &ps = c->pre[c->pre_next];
    if (ps.pending) return fail("%s: three prefetched frames are already waiting for nav_slam_localization_fast", name);
    // the frame the last localization call matched stays in its slot until its map kernel is queued:
    // nav_slam_mapping(pos, NULL, ...) maps it from there
    const bool holds_resident = c->cloud_resident && c->cur_cloud == ps.d_cloud;
    if (holds_resident && !ps.release_recorded)
        return fail("%s: the slot still holds the frame matched last; call nav_slam_mapping before prefetching "
                    "another frame", name);
    if (holds_resident) c->cloud_resident = false;  // overwritten below: nothing is left for mapping(NULL)
    // otherwise the slot's last reader is already queued on the context's stream: the match of a frame that
    // was not mapped from the slot, or the map kernel after which nav_slam_mapping / nav_slam_run recorded
    // `released` (right behind that kernel, so that a prefetch issued later does not wait for more)
    if (!ps.release_recorded) CU(cudaEventRecord(ps.released, c->stream));
    ps.release_recorded = false;
    CU(cudaStreamWaitEvent(c->s_in, ps.released, 0));
    int *raw = nullptr;
    if (kind != NAV_RUN_INPUT_XYZ && !(raw = raw_buf(c, ps.raw, kind))) return 1;
    CU(cudaMemcpyAsync(raw ? (void *)raw : ps.d_cloud, src, frame_bytes(c, kind), cudaMemcpyHostToDevice, c->s_in));
    if (raw) to_xyz(c, kind, raw, ps.d_cloud, c->n_seq, c->s_in);
    launch_labels(ps.d_cloud, ps.d_labels, nullptr, (long long)c->n_seq * c->rows, c->cols, c->sm_count, c->d_n_exact,
                  c->s_in);
    c->launches++;
    CU(cudaEventRecord(ps.ready, c->s_in));
    ps.host_src = src;
    ps.pending = true;
    c->pre_next = (c->pre_next + 1) % 3;
    return 0;
}

extern "C" int nav_slam_prefetch(nav_ctx *c, const nav_point *cloud) {
    CTX_ENTER(c, "nav_slam_prefetch");
    return prefetch_common(c, "nav_slam_prefetch", NAV_RUN_INPUT_XYZ, cloud);
}

extern "C" int nav_slam_prefetch_depth(nav_ctx *c, const int *distances) {
    CTX_ENTER(c, "nav_slam_prefetch_depth");
    return prefetch_common(c, "nav_slam_prefetch_depth", NAV_RUN_INPUT_DEPTH, distances);
}

extern "C" int nav_slam_prefetch_mm(nav_ctx *c, const int32_t *cloud_mm) {
    CTX_ENTER(c, "nav_slam_prefetch_mm");
    return prefetch_common(c, "nav_slam_prefetch_mm", NAV_RUN_INPUT_MM, cloud_mm);
}

// slam_localization with the fit driven by five sufficient statistics reduced on the device
// (SURVEY 8f #2): no correspondence list crosses PCIe and the 200 iterations are O(1) each.
// Same update rule as src/slam.c:341-370; sums are formed in a different order than the
// reference's sequential loop, so poses agree to rounding (about 1e-9 relative), not bit for bit.
//
// The totals come back through host-mapped memory: the dedupe kernel's last CTA writes them followed by
// the call's sequence number (FitMailbox), and the host polls that word -- no copy is queued and the
// stream is not synchronised, which is worth several microseconds of a 60-90 us closed-loop step.
static double now_us() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

static int wait_fit_mail(nav_ctx *c, const char *name) {
    volatile unsigned long long *flag = (volatile unsigned long long *)(c->h_fit + 5);
    for (unsigned spins = 0; *flag != c->fit_seq; ++spins) {
        if ((spins & 0x3ffu) == 0x3ffu) {  // every ~1000 polls: has the stream died or drained without posting?
            const cudaError_t q = cudaStreamQuery(c->stream);
            if (q != cudaErrorNotReady) {
                if (q == cudaSuccess && *flag == c->fit_seq) break;
                cudaGetLastError();
                return fail("%s: device execution failed: %s", name,
                            q == cudaSuccess ? "statistics were not posted" : cudaGetErrorString(q));
            }
        }
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    c->stage.used = 0;  // the upload (if it was staged) has been consumed by the kernels that posted
    return 0;
}

// the bias corrections 1 - beta^t of the fit, tables computed once with the same pow() calls the loop used to make;
// the device loop (nav_slam_run_dev) gets a copy of these very values
static void fit_bias_tables(const double **c1, const double **c2) {
    static double c1_tab[kFitIters], c2_tab[kFitIters];
    static bool have_tab = false;
    if (!have_tab) {
        for (int i = 0; i < kFitIters; ++i) {
            c1_tab[i] = 1 - pow(0.9, i + 1);
            c2_tab[i] = 1 - pow(0.999, i + 1);
        }
        __atomic_thread_fence(__ATOMIC_RELEASE);
        have_tab = true;
    }
    *c1 = c1_tab;
    *c2 = c2_tab;
}

// the O(1)-per-iteration Adam loop on the five totals (fit_translation, also exported as nav_slam_fit_from_stats)
static void fit_from_stats(const double st[5], const nav_pos *pos_predict, const nav_pos *pos_last, nav_pos *pos_out,
                           double *error_out, size_t *n_corr_out) {
    const double *c1, *c2;
    fit_bias_tables(&c1, &c2);
    double t[6] = {pos_predict->x - pos_last->x,       pos_predict->y - pos_last->y,
                   pos_predict->z - pos_last->z,       pos_predict->roll - pos_last->roll,
                   pos_predict->pitch - pos_last->pitch, pos_predict->yaw - pos_last->yaw};
    const double err = fit_translation(st, t, c1, c2);
    if (error_out) *error_out = err;
    if (n_corr_out) *n_corr_out = (size_t)st[0];
    pos_out->x = pos_last->x + t[0];
    pos_out->y = pos_last->y + t[1];
    pos_out->z = pos_last->z + t[2];
    pos_out->roll = pos_last->roll + t[3];
    pos_out->pitch = pos_last->pitch + t[4];
    pos_out->yaw = pos_last->yaw + t[5];
}

// the prefetched frame uploaded from `cloud`, or (cloud == NULL) the oldest one waiting
static nav_ctx::PreSlot *find_prefetched(nav_ctx *c, const void *cloud) {
    for (int k = 0; k < 3; ++k) {
        nav_ctx::PreSlot &cand = c->pre[(c->pre_next + k) % 3];  // pre_next is the slot written longest ago
        if (cand.pending && (!cloud || cand.host_src == cloud)) return &cand;
    }
    return nullptr;
}

// first half: queue match + dedupe/statistics of the frame (prefetched or uploaded here); nothing is waited for
static int loc_fast_launch(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict, const nav_pos *pos_last) {
    if (!pos_predict || !pos_last) return fail("nav_slam_localization_fast: null argument");
    if (c->n_seq != 1) return fail("nav_slam_localization_fast: needs n_seq == 1");
    if (!c->have_map) return fail("nav_slam_localization_fast: call nav_slam_init first");
    // a prefetched frame?  (cloud == NULL: the oldest one waiting; otherwise the one uploaded from `cloud`)
    nav_ctx::PreSlot *ps = find_prefetched(c, cloud);
    if (!ps && !cloud) return fail("nav_slam_localization_fast: cloud == NULL but no frame has been prefetched");
    const double t0 = c->trace ? now_us() : 0.0;
    const PoseBatch poses = pose_batch(c, pos_predict, pos_last);
    const FitMailbox mail = {c->h_fit, c->d_fit_ticket, ++c->fit_seq};
    if (ps) {
        CU(cudaStreamWaitEvent(c->stream, ps->ready, 0));
        if (run_match(c, ps->d_cloud, ps->d_labels, false, poses, kDedupeStats, &mail)) return 1;
    } else {
        if (c->stage.reserve(c->ntot * 24 + 1024, c->stream)) return fail("nav_slam_localization_fast: staging");
        if (upload_cloud(c, cloud, "nav_slam_localization_fast")) return 1;
        if (run_match(c, c->d_cloud, c->d_labels, true, poses, kDedupeStats, &mail)) return 1;
    }
    set_current_frame(c, ps);
    CU(cudaGetLastError());
    if (c->trace) c->trace_us[1] += now_us() - t0;
    return 0;
}

// second half: wait for the statistics and fit
static int loc_fast_finish(nav_ctx *c, const nav_pos *pos_predict, const nav_pos *pos_last, nav_pos *pos_out,
                           double *error_out, size_t *n_corr_out) {
    if (!pos_out) return fail("nav_slam_localization_fast: null argument");
    const double t1 = c->trace ? now_us() : 0.0;
    if (wait_fit_mail(c, "nav_slam_localization_fast")) return 1;
    const double t2 = c->trace ? now_us() : 0.0;
    fit_from_stats(c->h_fit, pos_predict, pos_last, pos_out, error_out, n_corr_out);
    if (c->trace) {
        c->trace_us[2] += t2 - t1;
        c->trace_us[3] += now_us() - t2;
    }
    return 0;
}

extern "C" int nav_slam_localization_fast(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict,
                                          const nav_pos *pos_last, nav_pos *pos_out, double *error_out,
                                          size_t *n_corr_out) {
    CTX_ENTER(c, "nav_slam_localization_fast");
    REFUSE_UNDER_REF_TIES(c, "nav_slam_localization_fast");
    if (!pos_out) return fail("nav_slam_localization_fast: null argument");
    if (loc_fast_launch(c, cloud, pos_predict, pos_last)) return 1;
    return loc_fast_finish(c, pos_predict, pos_last, pos_out, error_out, n_corr_out);
}

extern "C" int nav_slam_fit_from_stats(const double stats[5], const nav_pos *pos_predict, const nav_pos *pos_last,
                                       nav_pos *pos_out, double *error_out) {
    if (!stats || !pos_predict || !pos_last || !pos_out) return fail("nav_slam_fit_from_stats: null argument");
    fit_from_stats(stats, pos_predict, pos_last, pos_out, error_out, nullptr);
    return 0;
}

extern "C" int nav_slam_fit_stats(nav_ctx *c, double out[5]) {
    CTX_ENTER(c, "nav_slam_fit_stats");
    if (!out) return fail("nav_slam_fit_stats: null argument");
    if (c->fit_seq == 0) return fail("nav_slam_fit_stats: no closed-loop fit has run on this context");
    // the localization call that launched the fit waited for this post before it returned (wait_fit_mail);
    // a different number means that call failed
    if (*(volatile unsigned long long *)(c->h_fit + 5) != c->fit_seq)
        return fail("nav_slam_fit_stats: the last closed-loop fit did not complete");
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    memcpy(out, c->h_fit, 5 * sizeof(double));
    return 0;
}

// The closed loop of a whole sequence in one call: the loop of src/main.c:300-318 with the EKF prediction
// supplied by the caller -- a callback, or an array of dead-reckoning increments (pred = last + delta[t]).
// Frame t+1 is prefetched (upload + labels on the copy-in stream) while frame t is matched and fitted.
extern "C" int nav_slam_run(nav_ctx *c, const void *const *frames, int n_frames, int input_kind,
                            nav_predict_fn predict, void *user, const nav_pos *deltas, const nav_pos *pos_start,
                            nav_pos *poses_out, double *error_out, size_t *n_corr_out) {
    CTX_ENTER(c, "nav_slam_run");
    REFUSE_UNDER_REF_TIES(c, "nav_slam_run");
    if (!frames || n_frames < 0 || !pos_start || !poses_out || (!predict && !deltas))
        return fail("nav_slam_run: null argument");
    if (c->n_seq != 1) return fail("nav_slam_run: needs n_seq == 1");
    if (!c->have_map) return fail("nav_slam_run: call nav_slam_init first");
    nav_pos last = *pos_start;
    // every non-zero value other than NAV_RUN_INPUT_MM means depth matrices
    const int kind = input_kind == NAV_RUN_INPUT_XYZ || input_kind == NAV_RUN_INPUT_MM ? input_kind : NAV_RUN_INPUT_DEPTH;
    auto prefetch = [&](int t) { return prefetch_common(c, "nav_slam_run", kind, frames[t]); };
    // a frame that is not a cloud is found as the oldest prefetched one, never uploaded as a cloud
    auto cloud_of = [&](int t) { return kind == NAV_RUN_INPUT_XYZ ? (const nav_point *)frames[t] : nullptr; };
    for (auto &ps : c->pre) ps.pending = false;
    // the loop maps its own frames: a frame an earlier localization call left unmapped in a prefetch slot is
    // given up, so that the slot can be refilled
    if (n_frames > 0) c->cloud_resident = false;
    // one launch per frame (k_loop_step) where a row fits one thread-block cluster; wider rows keep the three launches
    // per frame (match, statistics dedupe, map) of the separate calls
    const bool fused = row_cluster_supported(c->cols);
    nav_ctx::PreSlot *deferred = nullptr;  // fused: the frame whose map the next launch builds first
    static const bool want_trace = getenv("NAV_RUN_TRACE") != nullptr;
    c->trace = want_trace;
    for (double &v : c->trace_us) v = 0.0;
    if (n_frames > 0 && prefetch(0)) return 1;
    for (int t = 0; t < n_frames; ++t) {
        nav_pos pred;
        if (predict) {
            predict(user, t, &last, &pred);
        } else {
            pred.x = last.x + deltas[t].x;
            pred.y = last.y + deltas[t].y;
            pred.z = last.z + deltas[t].z;
            pred.roll = last.roll + deltas[t].roll;
            pred.pitch = last.pitch + deltas[t].pitch;
            pred.yaw = last.yaw + deltas[t].yaw;
        }
        double err = 0.0;
        size_t nc = 0;
        // queue match + statistics of frame t, THEN the upload + labels of frame t+1 (their API calls cost
        // host time that is otherwise spent polling), then wait for the statistics and fit
        if (fused) {
            // one launch: map of frame t-1 from its fitted pose (deferred from the previous iteration), match of
            // frame t, statistics dedupe, mailbox post (k_loop_step)
            const double t0 = c->trace ? now_us() : 0.0;
            nav_ctx::PreSlot *ps = find_prefetched(c, cloud_of(t));
            if (!ps) return fail("nav_slam_run: frame %d was not prefetched", t);
            order_after_async(c);
            const PoseBatch poses = pose_batch(c, &pred, &last);
            const PoseBatch prev_poses = pose_batch(c, &last, nullptr);
            const FitMailbox mail = {c->h_fit, c->d_fit_ticket, ++c->fit_seq};
            const MatchOut out = {c->d_nn_idx, c->d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
            CU(cudaStreamWaitEvent(c->stream, ps->ready, 0));
            CU((cudaError_t)launch_loop_step(ps->d_cloud, ps->d_labels, c->map, out, poses, 1, c->rows, c->cols, c->stream,
                                             deferred ? deferred->d_cloud : nullptr, deferred ? deferred->d_labels : nullptr,
                                             prev_poses, deferred != nullptr, c->d_tile_stats, mail));
            c->launches++;
            if (deferred) {  // this launch was the last reader of the previous frame's slot
                CU(cudaEventRecord(deferred->released, c->stream));
                deferred->release_recorded = true;
            }
            set_current_frame(c, ps);
            deferred = ps;
            if (c->trace) c->trace_us[1] += now_us() - t0;
        } else if (loc_fast_launch(c, cloud_of(t), &pred, &last)) {
            return 1;
        }
        const double tp = c->trace ? now_us() : 0.0;
        if (t + 1 < n_frames && prefetch(t + 1)) return 1;
        if (c->trace) c->trace_us[0] += now_us() - tp;
        if (loc_fast_finish(c, &pred, &last, &poses_out[t], &err, &nc)) return 1;
        if (error_out) error_out[t] = err;
        if (n_corr_out) n_corr_out[t] = nc;
        const double tm = c->trace ? now_us() : 0.0;
        if (!fused || t + 1 == n_frames) {  // fused: only the last frame is mapped by a launch of its own
            if (nav_slam_mapping(c, &poses_out[t], nullptr, nullptr)) return 1;
        }
        if (c->trace) c->trace_us[4] += now_us() - tm;
        last = poses_out[t];
    }
    if (c->trace && n_frames > 0) {
        fprintf(stderr, "nav_slam_run trace, us per frame over %d frames: prefetch call %.2f, match+dedupe launches %.2f, "
                        "wait for statistics %.2f, fit %.2f, mapping call %.2f\n", n_frames, c->trace_us[0] / n_frames,
                c->trace_us[1] / n_frames, c->trace_us[2] / n_frames, c->trace_us[3] / n_frames, c->trace_us[4] / n_frames);
        c->trace = false;
    }
    return 0;
}

static bool on_ctx_device(const nav_ctx *c, const void *p);

// The closed loop of nav_slam_run on frames resident in HBM, with no host in the loop: launch t (k_loop_step<true>)
// maps frame t-1 from its fitted pose, matches frame t from its predicted pose -- both read from the device pose
// record -- and the last CTA of each sequence fits the pose and writes the record of frame t+1; one more launch maps
// the last frame.  Only the translation depends on the fit, so every rotation (and the fitted roll / pitch / yaw)
// is formed here up front with the host libm, exactly as make_pose forms it in nav_slam_run.
// Depth and integer-mm frames are read raw by the same kernel (k_loop_step<true, kind>), converted where the tile is
// staged and where the previous frame is mapped: still n_frames + 1 launches.  `name`: the entry point the caller used.
static int slam_run_dev(nav_ctx *c, const char *name, const void *dev_frames, int kind, int n_frames,
                        const nav_pos *deltas, const nav_pos *pos_start, const nav_run_dev_out *out) {
    REFUSE_UNDER_REF_TIES(c, name);
    if (!dev_frames || !deltas || !pos_start || !out || !out->poses)
        return fail("%s: null argument (dev_frames, deltas, pos_start, out and out->poses are required)", name);
    if (check_frame_input(name, dev_frames, kind)) return 1;
    if (n_frames < 0) return fail("%s: n_frames = %d is negative", name, n_frames);
    if (!row_cluster_supported(c->cols))
        return fail("%s: rows of %d columns are wider than one thread-block cluster (2048 columns at most)", name,
                    c->cols);
    if (!c->have_map) return fail("%s: call nav_slam_init or nav_slam_init_dev first", name);
    const std::pair<const void *, const char *> fields[] = {
        {dev_frames, "dev_frames"}, {out->poses, "out->poses"}, {out->error, "out->error"}, {out->fit_stats, "out->fit_stats"}};
    for (const auto &fd : fields)
        if (fd.first && !on_ctx_device(c, fd.first))
            return fail("%s: %s is not device or managed memory on device %d", name, fd.second, c->device);
    if (n_frames == 0) return 0;
    const int ns = c->n_seq;
    const size_t n_tab = (size_t)n_frames * ns;
    const size_t rec_bytes = (size_t)ns * sizeof(LoopRec), bytes = rec_bytes + n_tab * sizeof(LoopTab);
    // one-time set-up and growth of the scratch (these may synchronise)
    if (!c->fit_tables_queued) {
        const double *c1, *c2;
        fit_bias_tables(&c1, &c2);
        CU((cudaError_t)upload_fit_tables(c1, c2, c->stream));
        c->fit_tables_queued = true;
    }
    if (!c->d_loop_ticket) {
        CU(cudaMalloc((void **)&c->d_loop_ticket, NAV_MAX_SEQ * sizeof(unsigned)));
        CU(cudaMemsetAsync(c->d_loop_ticket, 0, NAV_MAX_SEQ * sizeof(unsigned), c->stream));
    }
    if (!c->d_labels_alt) CU(cudaMalloc((void **)&c->d_labels_alt, c->ntot * 4));
    if (c->d_loop_cap < bytes + rec_bytes) {
        CU(cudaStreamSynchronize(c->stream));
        if (c->d_loop) cudaFree(c->d_loop);
        c->d_loop = nullptr;
        c->d_loop_cap = 0;
        CU(cudaMalloc(&c->d_loop, bytes + rec_bytes));
        c->d_loop_cap = bytes + rec_bytes;
    }
    nav_ctx::PoseRing &pr = c->pose_ring[c->pose_ring_next];
    c->pose_ring_next = (c->pose_ring_next + 1) % nav_ctx::kPoseRing;
    if (pr.done) CU(cudaEventSynchronize(pr.done));  // the staging buffer's previous upload (several calls ago)
    if (pr.cap < bytes) {
        if (pr.host) cudaFreeHost(pr.host);
        pr.host = nullptr;
        pr.cap = 0;
        CU(cudaHostAlloc((void **)&pr.host, bytes, cudaHostAllocDefault));
        pr.cap = bytes;
    }
    if (!pr.done) CU(cudaEventCreateWithFlags(&pr.done, cudaEventDisableTiming));
    // staging: the records of frame 0, then the tables; on the device the records of frame 1 follow the tables
    LoopRec *rec0 = (LoopRec *)pr.host;
    LoopTab *tab = (LoopTab *)((unsigned char *)pr.host + rec_bytes);
    for (int s = 0; s < ns; ++s) {
        const nav_pos &st = pos_start[s], &d = deltas[s];
        const nav_pos pred = {st.x + d.x, st.y + d.y, st.z + d.z, st.roll + d.roll, st.pitch + d.pitch, st.yaw + d.yaw};
        rec0[s].loc = make_pose(&pred, &st);
        rec0[s].map = make_pose(&st, nullptr);
        nav_pos last = st;
        for (int t = 0; t < n_frames; ++t) {
            const nav_pos &dt = deltas[(size_t)t * ns + s];
            nav_pos p = last, f = last;  // prediction and fitted pose; only roll / pitch / yaw are used here
            p.roll = last.roll + dt.roll;
            p.pitch = last.pitch + dt.pitch;
            p.yaw = last.yaw + dt.yaw;
            f.roll = last.roll + (p.roll - last.roll);  // fit_from_stats: pos_last + (pos_predict - pos_last)
            f.pitch = last.pitch + (p.pitch - last.pitch);
            f.yaw = last.yaw + (p.yaw - last.yaw);
            LoopTab &tb = tab[(size_t)t * ns + s];
            rotation_from_pos(&p, tb.Rq);
            rotation_from_pos(&f, tb.Rm);
            tb.rpy[0] = f.roll;
            tb.rpy[1] = f.pitch;
            tb.rpy[2] = f.yaw;
            tb.d[0] = dt.x;
            tb.d[1] = dt.y;
            tb.d[2] = dt.z;
            last = f;
        }
    }
    unsigned char *dl_base = (unsigned char *)c->d_loop;
    LoopRec *d_rec[2] = {(LoopRec *)dl_base, (LoopRec *)(dl_base + bytes)};
    const LoopTab *d_tab = (const LoopTab *)(dl_base + rec_bytes);
    order_after_async(c);
    CU(cudaMemcpyAsync(c->d_loop, pr.host, bytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaEventRecord(pr.done, c->stream));
    // the label ring: frame t's labels go where the launch of frame t+1 maps them from; the last frame's land in
    // d_labels, as nav_frame_results_dev reports them
    auto labels_of = [&](int t) { return ((n_frames - 1 - t) & 1) ? c->d_labels_alt : c->d_labels; };
    auto frame = [&](int t) { return frame_at(c, dev_frames, kind, (size_t)t); };
    const MatchOut mo = {c->d_nn_idx, c->d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
    const TanTables tan = {c->d_tan_col, c->d_tan_row};
    for (int t = 0; t <= n_frames; ++t) {  // t == n_frames: the last frame's map
        const bool match = t < n_frames;
        const DevLoop dl = {t, n_frames, ns, match ? 1 : 0, match ? labels_of(t) : nullptr, d_rec[t & 1],
                            d_rec[(t + 1) & 1], d_tab, c->d_loop_ticket, c->d_n_exact, (nav_pos *)out->poses,
                            out->error, out->fit_stats};
        CU((cudaError_t)launch_loop_step_dev(kind, dl, match ? frame(t) : nullptr, t > 0 ? frame(t - 1) : nullptr,
                                             t > 0 ? labels_of(t - 1) : nullptr, t > 0, c->map, mo, ns, c->rows, c->cols,
                                             c->d_tile_stats, c->stream, tan));
        c->launches++;
    }
    c->cloud_resident = false;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int nav_slam_run_dev(nav_ctx *c, const void *dev_frames, int n_frames, const nav_pos *deltas,
                                const nav_pos *pos_start, const nav_run_dev_out *out) {
    CTX_ENTER(c, "nav_slam_run_dev");
    return slam_run_dev(c, "nav_slam_run_dev", dev_frames, NAV_RUN_INPUT_XYZ, n_frames, deltas, pos_start, out);
}

extern "C" int nav_slam_run_dev_ex(nav_ctx *c, const void *dev_frames, int input_kind, int n_frames,
                                   const nav_pos *deltas, const nav_pos *pos_start, const nav_run_dev_out *out) {
    CTX_ENTER(c, "nav_slam_run_dev_ex");
    return slam_run_dev(c, "nav_slam_run_dev_ex", dev_frames, input_kind, n_frames, deltas, pos_start, out);
}

// test seam: how the last nav_frontend_sequence_dev / nav_frontend_sequence_out_dev of the context ran -- 0: one
// launch per frame, 1: one k_frame_seq launch staging with cp.async, 2: one k_frame_seq launch staging with bulk
// copies; -1 before the first replay
extern "C" int nav_debug_sequence_path(const nav_ctx *c) { return c ? c->seq_path : -1; }

// test seam: the device fit (fit_translation with the uploaded tables) on n stat vectors, one thread each
extern "C" int nav_debug_fit_from_stats_dev(const double *dev_stats, const nav_pos *dev_pred, const nav_pos *dev_last,
                                            size_t n, nav_pos *dev_pose_out, double *dev_err_out, void *stream) {
    if (!dev_stats || !dev_pred || !dev_last || !dev_pose_out) return fail("nav_debug_fit_from_stats_dev: null argument");
    const double *c1, *c2;
    fit_bias_tables(&c1, &c2);
    CU((cudaError_t)upload_fit_tables(c1, c2, (cudaStream_t)stream));
    launch_fit_debug(dev_stats, dev_pred, dev_last, n, dev_pose_out, dev_err_out, (cudaStream_t)stream);
    CU(cudaGetLastError());
    return 0;
}

extern "C" int nav_slam_mapping(nav_ctx *c, const nav_pos *pos, const nav_point *cloud, nav_point *global_out) {
    CTX_ENTER(c, "nav_slam_mapping");
    if (!pos) return fail("nav_slam_mapping: null argument");
    if (c->stage.reserve(c->ntot * 48 + 1024, c->stream)) return fail("nav_slam_mapping: staging");
    if (cloud) {
        if (upload_cloud(c, cloud, "nav_slam_mapping")) return 1;
        run_labels(c, c->d_cloud, c->d_labels, nullptr, c->n_seq);
        set_current_frame(c);
    } else if (!c->cloud_resident || !c->cur_cloud) {
        return fail("nav_slam_mapping: cloud == NULL but no cloud is resident from a preceding match");
    }
    run_map(c, c->cur_cloud, c->cur_labels, pose_batch(c, pos, nullptr));
    if (c->cur_pre && c->cur_cloud == c->cur_pre->d_cloud) {
        // the map kernel just queued is the last reader of the frame's prefetch slot: the slot is free behind it
        CU(cudaEventRecord(c->cur_pre->released, c->stream));
        c->cur_pre->release_recorded = true;
    }
    if (!cloud && !global_out) {  // nothing to wait for: the map kernel is queued, errors surface at the next call
        CU(cudaGetLastError());
        return 0;
    }
    if (global_out && c->stage.d2h(global_out, c->map.pts, c->ntot * 24, c->stream))
        return fail("nav_slam_mapping: D2H");
    return finish_call(c, "nav_slam_mapping");
}

// the blocking front-end frame from a host frame of `kind` (NAV_RUN_INPUT_*).  A depth matrix (4 B/pixel instead of
// the 24 B/pixel cloud; L5 ingest fused with the frame, SURVEY 8f #3, device part) or integer-mm xyz (12 B/point) is
// uploaded, made xyz on the device and fed straight to the frame kernel; the converted lidar-frame cloud is returned
// only if the caller asks for it (cloud_out)
static int frontend_frame(nav_ctx *c, const char *name, int kind, const void *src, const nav_pos *pos_predict,
                          const nav_pos *pos_last, const nav_pos *pos_final, nav_point *cloud_out, int *feature_out,
                          int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out) {
    if (!src || !pos_predict || !pos_last || !pos_final) return fail("%s: null argument", name);
    if (kind == NAV_RUN_INPUT_DEPTH && c->n_seq != 1) return fail("%s: needs n_seq == 1", name);
    if (!c->have_map) return fail("%s: call nav_slam_init first", name);
    const size_t raw_bytes = kind == NAV_RUN_INPUT_XYZ ? 0 : frame_bytes(c, kind);
    if (c->stage.reserve(raw_bytes + c->ntot * (24 + 24 + 4 + 4 + 8) + 4096, c->stream)) return fail("%s: staging", name);
    if (kind == NAV_RUN_INPUT_XYZ) {
        if (upload_cloud(c, (const nav_point *)src, name)) return 1;
    } else {
        int *raw = raw_buf(c, c->raw, kind);
        if (!raw) return 1;
        if (c->stage.h2d(raw, src, raw_bytes, c->stream)) return fail("%s: H2D", name);
        to_xyz(c, kind, raw, c->d_cloud, c->n_seq, c->stream);
    }
    order_after_async(c);
    if (run_frame_fused(c, c->d_cloud, c->d_labels, c->d_nn_idx, c->d_nn_dist, pos_predict, pos_last, pos_final, false,
                        c->tie_rule == NAV_TIE_REFERENCE ? name : nullptr))
        return 1;
    set_current_frame(c);
    if (cloud_out && c->stage.d2h(cloud_out, c->d_cloud, c->ntot * 24, c->stream)) return fail("%s: D2H", name);
    if (feature_out && c->stage.d2h(feature_out, c->d_labels, c->ntot * 4, c->stream)) return fail("%s: D2H", name);
    if (nn_idx_out && c->stage.d2h(nn_idx_out, c->d_nn_idx, c->ntot * 4, c->stream)) return fail("%s: D2H", name);
    if (nn_dist_out && c->stage.d2h(nn_dist_out, c->d_nn_dist, c->ntot * 8, c->stream)) return fail("%s: D2H", name);
    if (global_out && c->stage.d2h(global_out, c->map.pts, c->ntot * 24, c->stream)) return fail("%s: D2H", name);
    return finish_call(c, name);
}

extern "C" int nav_frontend_frame(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict,
                                  const nav_pos *pos_last, const nav_pos *pos_final, int *feature_out,
                                  int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out) {
    CTX_ENTER(c, "nav_frontend_frame");
    return frontend_frame(c, "nav_frontend_frame", NAV_RUN_INPUT_XYZ, cloud, pos_predict, pos_last, pos_final, nullptr,
                          feature_out, nn_idx_out, nn_dist_out, global_out);
}

extern "C" int nav_frontend_frame_mm(nav_ctx *c, const int32_t *cloud_mm, const nav_pos *pos_predict,
                                     const nav_pos *pos_last, const nav_pos *pos_final, int *feature_out,
                                     int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out) {
    CTX_ENTER(c, "nav_frontend_frame_mm");
    return frontend_frame(c, "nav_frontend_frame_mm", NAV_RUN_INPUT_MM, cloud_mm, pos_predict, pos_last, pos_final,
                          nullptr, feature_out, nn_idx_out, nn_dist_out, global_out);
}

extern "C" int nav_frontend_frame_depth(nav_ctx *c, const int *distances, const nav_pos *pos_predict,
                                        const nav_pos *pos_last, const nav_pos *pos_final, nav_point *cloud_out,
                                        int *feature_out, int32_t *nn_idx_out, double *nn_dist_out,
                                        nav_point *global_out) {
    CTX_ENTER(c, "nav_frontend_frame_depth");
    return frontend_frame(c, "nav_frontend_frame_depth", NAV_RUN_INPUT_DEPTH, distances, pos_predict, pos_last,
                          pos_final, cloud_out, feature_out, nn_idx_out, nn_dist_out, global_out);
}

// ------------------------------------------------------------------ CSV rows on the device ---
// SURVEY 8f #4: the text of src/main.c:320-352 for one frame, produced where the global cloud lives.
namespace nav {
size_t csv_pose_columns(char *out, const double imu[6], const nav_pos *lidar_pos, const nav_pos *ekf_pos);  // io.cu
}

static int csv_job(nav_ctx *c, const char *name, unsigned long long timestamp, const double *d_cloud,
                   const int *d_dist, const double imu[6], const nav_pos *lp, const nav_pos *ep, CsvJob &job) {
    char tail[18 * 340 + 4];
    const size_t tail_len = csv_pose_columns(tail, imu, lp, ep);
    if (tail_len > (size_t)kCsvTailMax) return -1;  // a pose column beyond 2^57 or not finite: host formatter
    job.cloud = d_cloud;
    job.dist = d_dist;
    job.ts = timestamp;
    job.n = (long long)c->npx;
    job.cols = c->cols;
    job.ts_len = dec_len(timestamp);
    job.tail_len = (int)tail_len;
    memcpy(job.tail, tail, tail_len);
    if (!c->d_csv_scratch) {
        if (cudaMalloc(&c->d_csv_scratch, csv_scratch_bytes((long long)c->npx)) != cudaSuccess)
            return fail("%s: out of device memory", name);
    }
    return 0;
}

// Device-resident variant: d_global_cloud (NULL = the context's global cloud of the frame mapped last,
// i.e. what nav_slam_mapping / nav_frontend_frame just produced) and d_distances (NULL = 0) are device
// pointers, d_text receives the text; needs cap >= rows*cols*(124 + 18*23 + 1) unless the poses are
// short.  *n_bytes_out is valid on return (the call synchronises the context's stream).  Returns 2
// (and writes nothing useful) when some value needs the host formatter (inf, nan, |v| >= 2^57).
extern "C" int nav_csv_format_frame_dev(nav_ctx *c, unsigned long long timestamp, const nav_point *d_global_cloud,
                                        const int *d_distances, const double imu[6], const nav_pos *lidar_pos,
                                        const nav_pos *ekf_pos, char *d_text, size_t cap, size_t *n_bytes_out) {
    CTX_ENTER(c, "nav_csv_format_frame_dev");
    if (!lidar_pos || !d_text || !n_bytes_out) return fail("nav_csv_format_frame_dev: null argument");
    if (c->n_seq != 1) return fail("nav_csv_format_frame_dev: needs n_seq == 1");
    if (!d_global_cloud && !c->have_map) return fail("nav_csv_format_frame_dev: no frame has been mapped yet");
    CsvJob job;
    const int rc = csv_job(c, "nav_csv_format_frame_dev", timestamp,
                           d_global_cloud ? (const double *)d_global_cloud : c->map.pts, d_distances, imu, lidar_pos,
                           ekf_pos, job);
    if (rc > 0) return rc;
    if (rc < 0) return 2;
    if (cap < c->npx * (size_t)(kCsvHeadMax + job.tail_len)) return fail("nav_csv_format_frame_dev: d_text too small");
    if (launch_csv_format(job, d_text, c->d_csv_scratch, c->stream)) return fail("nav_csv_format_frame_dev: launch failed");
    c->launches += 3;
    CU(cudaMemcpyAsync(c->h_small, c->d_csv_scratch, 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *n_bytes_out = (size_t) * (unsigned long long *)c->h_small;
    return ((unsigned *)c->h_small)[2] ? 2 : 0;
}

// Host-facing variant: the text lands in buf (pinned memory avoids a staging copy).  global_cloud
// NULL = format the context's resident global cloud without any upload; distances NULL = 0.
// Frames with values outside the device formatter's range are formatted by nav_csv_format_frame on
// the host (same bytes).  Returns 0 and *n_bytes_out, or 1 (cap too small, CUDA failure).
extern "C" int nav_csv_format_frame_gpu(nav_ctx *c, unsigned long long timestamp, const nav_point *global_cloud,
                                        const int *distances, const double imu[6], const nav_pos *lidar_pos,
                                        const nav_pos *ekf_pos, char *buf, size_t cap, size_t *n_bytes_out) {
    CTX_ENTER(c, "nav_csv_format_frame_gpu");
    if (!lidar_pos || !buf || !n_bytes_out) return fail("nav_csv_format_frame_gpu: null argument");
    if (c->n_seq != 1) return fail("nav_csv_format_frame_gpu: needs n_seq == 1");
    if (!global_cloud && !c->have_map) return fail("nav_csv_format_frame_gpu: no frame has been mapped yet");
    *n_bytes_out = 0;
    if (c->stage.reserve(c->npx * 28 + 4096, c->stream)) return fail("nav_csv_format_frame_gpu: staging");
    const double *d_cloud = c->map.pts;
    if (global_cloud) {
        if (!c->d_global) CU(cudaMalloc((void **)&c->d_global, c->npx * 24));
        if (c->stage.h2d(c->d_global, global_cloud, c->npx * 24, c->stream)) return fail("nav_csv_format_frame_gpu: H2D");
        d_cloud = c->d_global;
    }
    if (distances && c->stage.h2d(c->raw[0], distances, c->npx * 4, c->stream)) return fail("nav_csv_format_frame_gpu: H2D");
    CsvJob job;
    int rc = csv_job(c, "nav_csv_format_frame_gpu", timestamp, d_cloud, distances ? c->raw[0] : nullptr, imu, lidar_pos,
                     ekf_pos, job);
    if (rc > 0) return rc;
    bool host_format = rc < 0;
    if (!host_format) {
        const size_t need = c->npx * (size_t)(kCsvHeadMax + job.tail_len);
        if (need > c->csv_cap) {
            CU(cudaStreamSynchronize(c->stream));
            if (c->d_csv) cudaFree(c->d_csv);
            c->d_csv = nullptr;
            c->csv_cap = 0;
            if (cudaMalloc((void **)&c->d_csv, need) != cudaSuccess) return fail("nav_csv_format_frame_gpu: out of device memory");
            c->csv_cap = need;
        }
        if (launch_csv_format(job, c->d_csv, c->d_csv_scratch, c->stream)) return fail("nav_csv_format_frame_gpu: launch failed");
        c->launches += 3;
        CU(cudaMemcpyAsync(c->h_small, c->d_csv_scratch, 16, cudaMemcpyDeviceToHost, c->stream));
        if (finish_call(c, "nav_csv_format_frame_gpu")) return 1;
        const size_t total = (size_t) * (unsigned long long *)c->h_small;
        host_format = ((unsigned *)c->h_small)[2] != 0;
        if (!host_format) {
            if (total > cap) return fail("nav_csv_format_frame_gpu: buf too small (%zu bytes needed)", total);
            if (Stager::is_pinned(buf)) {
                CU(cudaMemcpyAsync(buf, c->d_csv, total, cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
            } else {
                if (c->stage.reserve(total + 256, c->stream)) return fail("nav_csv_format_frame_gpu: staging");
                if (c->stage.d2h(buf, c->d_csv, total, c->stream)) return fail("nav_csv_format_frame_gpu: D2H");
                if (finish_call(c, "nav_csv_format_frame_gpu")) return 1;
            }
            *n_bytes_out = total;
            return 0;
        }
    } else if (finish_call(c, "nav_csv_format_frame_gpu")) {
        return 1;
    }
    // rare: inf / nan / |v| >= 2^57 somewhere in the frame -> the host writer prints the same bytes
    std::vector<nav_point> tmp;
    const nav_point *src = global_cloud;
    if (!src) {
        tmp.resize(c->npx);
        CU(cudaMemcpy(tmp.data(), c->map.pts, c->npx * 24, cudaMemcpyDeviceToHost));
        src = tmp.data();
    }
    const size_t n = nav_csv_format_frame(buf, cap, timestamp, c->rows, c->cols, src, distances, imu, lidar_pos, ekf_pos);
    if (n == 0) return fail("nav_csv_format_frame_gpu: buf too small");
    *n_bytes_out = n;
    return 0;
}

// ------------------------------------------------------------------ pipelined host path ------
// Same work as nav_frontend_frame, but nothing blocks: frame t's upload (copy-in stream), frame
// t-1's kernels (context stream) and frame t-2's downloads (copy-out stream) overlap, with two
// device slots for the per-frame buffers.  All host pointers must be pinned.  Outputs of frame t
// are valid after nav_frontend_wait() (or after two further submissions).
static int async_setup(nav_ctx *c) {
    if (c->slots[0].d_cloud) return 0;
    // the closed-loop prefetch (pre_setup) may have created the copy-in stream already
    if (!c->s_in) CU(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
    if (!c->s_out) CU(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
    for (auto &sl : c->slots) {
        CU(cudaMalloc((void **)&sl.d_cloud, c->ntot * 24));
        // labels, NN index and NN distance of a slot are one allocation [labels | nn_idx | nn_dist], so
        // that a caller whose host buffers are laid out the same way gets them with a single copy
        CU(cudaMalloc((void **)&sl.d_labels, c->ntot * 16));
        sl.d_nn_idx = sl.d_labels + c->ntot;
        sl.d_nn_dist = (double *)(sl.d_nn_idx + c->ntot);
        CU(cudaEventCreateWithFlags(&sl.in_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&sl.compute_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&sl.out_done, cudaEventDisableTiming));
    }
    return 0;
}

// nav_frontend_submit (cloud_mm == null: the input is io->cloud or io->distances) and nav_frontend_submit_mm (the input
// is cloud_mm, io carries outputs only)
static int frontend_submit(nav_ctx *c, const char *name, const int32_t *cloud_mm, const nav_frame_io *io,
                           const nav_pos *pos_predict, const nav_pos *pos_last, const nav_pos *pos_final) {
    if (!c) return fail("%s: null context", name);
    CU(cudaSetDevice(c->device));
    REFUSE_UNDER_REF_TIES(c, name);
    if (!io || !pos_predict || !pos_last || !pos_final) return fail("%s: null argument", name);
    if (cloud_mm) {
        if (io->cloud || io->distances || io->cloud_out)
            return fail("%s: the frame is cloud_mm; io->cloud, io->distances and io->cloud_out must be NULL", name);
    } else {
        if (!io->cloud == !io->distances) return fail("%s: give exactly one of cloud and distances", name);
        if (io->distances && c->n_seq != 1) return fail("%s: depth input needs n_seq == 1", name);
        if (io->cloud_out && !io->distances) return fail("%s: cloud_out is the converted depth matrix; there is none", name);
    }
    const int kind = cloud_mm ? NAV_RUN_INPUT_MM : io->distances ? NAV_RUN_INPUT_DEPTH : NAV_RUN_INPUT_XYZ;
    const void *src = cloud_mm ? (const void *)cloud_mm : io->distances ? (const void *)io->distances : io->cloud;
    if (!c->have_map) return fail("%s: call nav_slam_init first", name);
    if (async_setup(c)) return 1;
    const void *hp[] = {src, io->cloud_out, io->feature_out, io->mask_out, io->nn_idx_out, io->nn_dist_out,
                        io->global_out};
    for (const void *p : hp)
        if (p && !Stager::is_pinned(p))
            return fail("%s: host buffers must be pinned (nav_host_alloc / cudaHostRegister)", name);
    static_assert(nav_ctx::kSlots == 2, "slots pair up with the two map buffers (see nav_ctx)");
    nav_ctx::AsyncSlot &sl = c->slots[c->async_frames % nav_ctx::kSlots];
    const bool reused = c->async_frames >= (uint64_t)nav_ctx::kSlots;
    // copy-in: the slot's cloud was last read by the kernels of frame t-2
    if (reused) CU(cudaStreamWaitEvent(c->s_in, sl.compute_done, 0));
    int *raw = nullptr;
    if (kind != NAV_RUN_INPUT_XYZ && !(raw = raw_buf(c, sl.raw, kind))) return 1;
    CU(cudaMemcpyAsync(raw ? (void *)raw : sl.d_cloud, src, frame_bytes(c, kind), cudaMemcpyHostToDevice, c->s_in));
    CU(cudaEventRecord(sl.in_done, c->s_in));
    // kernels: need the upload, and the slot's output buffers released by the downloads of frame t-2
    CU(cudaStreamWaitEvent(c->stream, sl.in_done, 0));
    if (reused) CU(cudaStreamWaitEvent(c->stream, sl.out_done, 0));
    if (raw) to_xyz(c, kind, raw, sl.d_cloud, c->n_seq, c->stream);  // 4 or 12 B/point crossed PCIe instead of 24
    if (run_frame_fused(c, sl.d_cloud, sl.d_labels, sl.d_nn_idx, sl.d_nn_dist, pos_predict, pos_last, pos_final)) return 1;
    CU(cudaEventRecord(sl.compute_done, c->stream));
    c->cloud_resident = false;
    c->async_synced = false;
    // copy-out.  The mapped cloud and the label masks are persistent state (the next frame searches them):
    // they are read straight out of the map buffer this frame built, which stays untouched until the
    // frame after next -- and that frame waits for this slot's downloads (out_done) first.
    CU(cudaStreamWaitEvent(c->s_out, sl.compute_done, 0));
    int *f = io->feature_out;
    int32_t *ni = io->nn_idx_out;
    double *nd = io->nn_dist_out;
    if (f && ni == f + c->ntot && (void *)nd == (void *)(ni + c->ntot)) {  // labels | idx | dist adjacent: one copy
        CU(cudaMemcpyAsync(f, sl.d_labels, c->ntot * 16, cudaMemcpyDeviceToHost, c->s_out));
    } else if (!f && ni && (void *)nd == (void *)(ni + c->ntot)) {          // idx | dist adjacent
        CU(cudaMemcpyAsync(ni, sl.d_nn_idx, c->ntot * 12, cudaMemcpyDeviceToHost, c->s_out));
    } else {
        if (f) CU(cudaMemcpyAsync(f, sl.d_labels, c->ntot * 4, cudaMemcpyDeviceToHost, c->s_out));
        if (ni) CU(cudaMemcpyAsync(ni, sl.d_nn_idx, c->ntot * 4, cudaMemcpyDeviceToHost, c->s_out));
        if (nd) CU(cudaMemcpyAsync(nd, sl.d_nn_dist, c->ntot * 8, cudaMemcpyDeviceToHost, c->s_out));
    }
    if (io->mask_out)
        CU(cudaMemcpyAsync(io->mask_out, c->map.mask, (size_t)c->n_seq * c->rows * c->map.n_chunks * 4,
                           cudaMemcpyDeviceToHost, c->s_out));
    if (io->global_out) CU(cudaMemcpyAsync(io->global_out, c->map.pts, c->ntot * 24, cudaMemcpyDeviceToHost, c->s_out));
    if (io->cloud_out) CU(cudaMemcpyAsync(io->cloud_out, sl.d_cloud, c->ntot * 24, cudaMemcpyDeviceToHost, c->s_out));
    CU(cudaEventRecord(sl.out_done, c->s_out));
    c->async_frames++;
    return 0;
}

extern "C" int nav_frontend_submit(nav_ctx *c, const nav_frame_io *io, const nav_pos *pos_predict,
                                   const nav_pos *pos_last, const nav_pos *pos_final) {
    return frontend_submit(c, "nav_frontend_submit", nullptr, io, pos_predict, pos_last, pos_final);
}

extern "C" int nav_frontend_submit_mm(nav_ctx *c, const int32_t *cloud_mm, const nav_frame_io *io,
                                      const nav_pos *pos_predict, const nav_pos *pos_last, const nav_pos *pos_final) {
    if (!cloud_mm) return fail("nav_frontend_submit_mm: null argument");
    return frontend_submit(c, "nav_frontend_submit_mm", cloud_mm, io, pos_predict, pos_last, pos_final);
}

extern "C" int nav_frontend_frame_async(nav_ctx *c, const nav_point *cloud, const nav_pos *pos_predict,
                                        const nav_pos *pos_last, const nav_pos *pos_final, int *feature_out,
                                        int32_t *nn_idx_out, double *nn_dist_out, nav_point *global_out) {
    REFUSE_UNDER_REF_TIES(c, "nav_frontend_frame_async");
    if (!cloud) return fail("nav_frontend_frame_async: null argument");
    nav_frame_io io = {};
    io.cloud = cloud;
    io.feature_out = feature_out;
    io.nn_idx_out = nn_idx_out;
    io.nn_dist_out = nn_dist_out;
    io.global_out = global_out;
    return nav_frontend_submit(c, &io, pos_predict, pos_last, pos_final);
}

extern "C" int nav_frontend_frame_depth_async(nav_ctx *c, const int *distances, const nav_pos *pos_predict,
                                              const nav_pos *pos_last, const nav_pos *pos_final, nav_point *cloud_out,
                                              int *feature_out, int32_t *nn_idx_out, double *nn_dist_out,
                                              nav_point *global_out) {
    REFUSE_UNDER_REF_TIES(c, "nav_frontend_frame_depth_async");
    if (!distances) return fail("nav_frontend_frame_depth_async: null argument");
    nav_frame_io io = {};
    io.distances = distances;
    io.cloud_out = cloud_out;
    io.feature_out = feature_out;
    io.nn_idx_out = nn_idx_out;
    io.nn_dist_out = nn_dist_out;
    io.global_out = global_out;
    return nav_frontend_submit(c, &io, pos_predict, pos_last, pos_final);
}

extern "C" int nav_frontend_wait(nav_ctx *c) {
    CTX_ENTER(c, "nav_frontend_wait");
    CU(cudaStreamSynchronize(c->stream));
    if (c->s_out) CU(cudaStreamSynchronize(c->s_out));
    if (c->s_in) CU(cudaStreamSynchronize(c->s_in));
    // the synchronous entry points and nav_frame_results_dev read labels / nn_idx / nn_dist from the
    // context's own buffers: bring all three up to date with the last pipelined frame
    if (c->async_frames && !c->async_synced) {
        nav_ctx::AsyncSlot &sl = c->slots[(c->async_frames - 1) % nav_ctx::kSlots];
        CU(cudaMemcpyAsync(c->d_labels, sl.d_labels, c->ntot * 4, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(c->d_nn_idx, sl.d_nn_idx, c->ntot * 4, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(c->d_nn_dist, sl.d_nn_dist, c->ntot * 8, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->async_synced = true;
    }
    return 0;
}

// ------------------------------------------------------------------ device resident ----------
extern "C" int nav_extract_feature_batch_dev(nav_ctx *c, const void *dev_clouds, size_t n_images, void *dev_labels) {
    CTX_ENTER(c, "nav_extract_feature_batch_dev");
    if (!dev_clouds || !dev_labels) return fail("nav_extract_feature_batch_dev: null argument");
    run_labels(c, (const double *)dev_clouds, (int *)dev_labels, nullptr, n_images);
    CU(cudaGetLastError());
    return 0;
}

extern "C" int nav_frontend_frame_dev(nav_ctx *c, const void *dev_cloud, const nav_pos *pos_predict,
                                      const nav_pos *pos_last, const nav_pos *pos_final) {
    CTX_ENTER(c, "nav_frontend_frame_dev");
    REFUSE_UNDER_REF_TIES(c, "nav_frontend_frame_dev");
    if (!dev_cloud || !pos_predict || !pos_last || !pos_final) return fail("nav_frontend_frame_dev: null argument");
    if (!c->have_map) return fail("nav_frontend_frame_dev: call nav_slam_init_dev first");
    order_after_async(c);
    if (run_frame_fused(c, (const double *)dev_cloud, c->d_labels, c->d_nn_idx, c->d_nn_dist, pos_predict, pos_last,
                        pos_final))
        return 1;
    c->cloud_resident = false;
    CU(cudaGetLastError());
    return 0;
}

// device (or managed) memory of the context's device?
static bool on_ctx_device(const nav_ctx *c, const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();  // not a sticky error: clear it
        return false;
    }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == c->device;
}

// nav_frontend_sequence_dev, and with per-frame outputs (so != null) nav_frontend_sequence_out_dev; their _ex forms
// with a frame kind (NAV_RUN_INPUT_*).  `name`: the entry point the caller used.
static int frontend_sequence(nav_ctx *c, const char *name, const void *dev_frames, int kind, size_t n_frames,
                             const nav_pos *pos_predict, const nav_pos *pos_last, const nav_pos *pos_final,
                             const nav_sequence_out *so) {
    REFUSE_UNDER_REF_TIES(c, name);
    if (!dev_frames || !pos_predict || !pos_last || !pos_final) return fail("%s: null argument", name);
    if (check_frame_input(name, dev_frames, kind)) return 1;
    if (!c->have_map) return fail("%s: call nav_slam_init_dev first", name);
    if (so) {
        const std::pair<const void *, const char *> fields[] = {
            {so->label_mask, "label_mask"}, {so->nn_idx, "nn_idx"}, {so->nn_dist, "nn_dist"}, {so->fit_stats, "fit_stats"}};
        for (const auto &fd : fields)
            if (fd.first && !on_ctx_device(c, fd.first))
                return fail("%s: out->%s is not device or managed memory on device %d", name, fd.second, c->device);
        if (!so->label_mask && !so->nn_idx && !so->nn_dist && !so->fit_stats) so = nullptr;
    }
    const bool raw = kind != NAV_RUN_INPUT_XYZ;
    const long long stride = (long long)(frame_bytes(c, kind) / elem_bytes(kind));  // in elements, for k_frame_seq
    order_after_async(c);
    // One launch for the whole sequence (k_frame_seq: a thread-block cluster per image row walks through the
    // frames with a cluster barrier per frame) when a row's tiles fit a cluster; NAV_SEQ_LAUNCHES=1 keeps one
    // launch per frame.  The per-kernel profiler wants separate launches too.
    // Measured (profiles/README.md): the same 14.4-14.5 us per 64x2048 frame as separate launches for one
    // sequence -- the chain of one row is what takes that long -- with one launch instead of n_frames for the
    // host to issue; several sequences side by side (n_seq > 1) fill the machine better as separate launches.
    static const bool per_frame = getenv("NAV_SEQ_LAUNCHES") != nullptr;
    const bool fused =
        !per_frame && !c->prof && c->n_seq == 1 && n_frames > 1 && row_cluster_supported(c->cols) && n_frames <= 0x7fffffff;
    // fit statistics: CTA partials per frame in scratch -- one per (row, tile) from k_frame_seq or k_dedupe_stats
    // (rows up to 2048 columns), one per row from k_dedupe_rows (wider rows) -- then one totals launch
    const size_t nr = (size_t)c->n_seq * c->rows;
    const bool tile_parts = row_cluster_supported(c->cols);
    const size_t part_frame = tile_parts ? nr * div_up(c->cols, 256) : nr;  // partials per frame
    double *part = nullptr;
    if (so && so->fit_stats && n_frames > 0) {
        const size_t bytes = n_frames * part_frame * 5 * sizeof(double);
        if (c->d_seq_part_cap < bytes) {
            CU(cudaStreamSynchronize(c->stream));
            if (c->d_seq_part) cudaFree(c->d_seq_part);
            c->d_seq_part = nullptr;
            c->d_seq_part_cap = 0;
            CU(cudaMalloc((void **)&c->d_seq_part, bytes));
            c->d_seq_part_cap = bytes;
        }
        part = c->d_seq_part;
    }
    const SeqOut seq_out = {so ? (unsigned *)so->label_mask : nullptr, so ? (int *)so->nn_idx : nullptr,
                            so ? (double *)so->nn_dist : nullptr, part};
    const TanTables tan = {c->d_tan_col, c->d_tan_row};
    // the per-frame path converts depth / integer-mm frames into two context-owned frame slots first
    if (!fused && raw && n_frames > 0 && !c->d_conv) CU(cudaMalloc((void **)&c->d_conv, c->ntot * 24 * 2));
    c->seq_path = 0;
    if (fused) {
        bool bulk = false;
        const size_t n_pose = n_frames * (size_t)c->n_seq, bytes = n_pose * 2 * sizeof(PoseXf);
        const MatchOut out = {c->d_nn_idx, c->d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
        if ((int)n_frames <= frame_seq_inline_frames()) {  // short sequence: poses as kernel parameters
            PoseXf loc[64], fin[64];
            static_assert(sizeof(loc) / sizeof(loc[0]) >= 64, "");
            if (frame_seq_inline_frames() > 64) return fail("%s: inline pose capacity", name);
            for (size_t i = 0; i < n_pose; ++i) {
                loc[i] = make_pose(&pos_predict[i], &pos_last[i]);
                fin[i] = make_pose(&pos_final[i], nullptr);
            }
            CU((cudaError_t)launch_frame_seq(kind, dev_frames, stride, (int)n_frames, c->d_labels, c->map, c->map_alt, out,
                                             nullptr, nullptr, c->n_seq, c->rows, c->cols, c->d_n_exact, c->stream, loc, fin,
                                             so ? &seq_out : nullptr, &bulk, tan));
        } else {
            nav_ctx::PoseRing &pr = c->pose_ring[c->pose_ring_next];
            c->pose_ring_next = (c->pose_ring_next + 1) % nav_ctx::kPoseRing;
            if (pr.done) CU(cudaEventSynchronize(pr.done));  // the staging buffer's previous upload (several sequences ago)
            if (pr.cap < bytes) {
                if (pr.host) cudaFreeHost(pr.host);
                pr.host = nullptr;
                pr.cap = 0;
                CU(cudaHostAlloc((void **)&pr.host, bytes, cudaHostAllocDefault));
                pr.cap = bytes;
            }
            if (!pr.done) CU(cudaEventCreateWithFlags(&pr.done, cudaEventDisableTiming));
            if (c->d_pose_cap < bytes) {
                CU(cudaStreamSynchronize(c->stream));
                if (c->d_pose) cudaFree(c->d_pose);
                c->d_pose = nullptr;
                c->d_pose_cap = 0;
                CU(cudaMalloc((void **)&c->d_pose, bytes));
                c->d_pose_cap = bytes;
            }
            PoseXf *loc = (PoseXf *)pr.host, *fin = loc + n_pose;
            for (size_t i = 0; i < n_pose; ++i) {
                loc[i] = make_pose(&pos_predict[i], &pos_last[i]);
                fin[i] = make_pose(&pos_final[i], nullptr);
            }
            CU(cudaMemcpyAsync(c->d_pose, pr.host, bytes, cudaMemcpyHostToDevice, c->stream));
            CU(cudaEventRecord(pr.done, c->stream));
            CU((cudaError_t)launch_frame_seq(kind, dev_frames, stride, (int)n_frames, c->d_labels, c->map, c->map_alt, out,
                                             (const PoseXf *)c->d_pose, (const PoseXf *)c->d_pose + n_pose, c->n_seq, c->rows,
                                             c->cols, c->d_n_exact, c->stream, nullptr, nullptr, so ? &seq_out : nullptr, &bulk,
                                             tan));
        }
        c->seq_path = bulk ? 2 : 1;
        c->launches++;
        if (n_frames & 1) std::swap(c->map, c->map_alt);
    } else {
        const size_t n_chunks = (size_t)c->map.n_chunks;
        for (size_t f = 0; f < n_frames; ++f) {
            const void *frame = frame_at(c, dev_frames, kind, f);
            const double *cl = (const double *)frame;
            if (raw) {  // frame f into slot f % 2: the kernels of frame f-1 read the other slot
                cl = c->d_conv + (f & 1) * c->ntot * 3;
                to_xyz(c, kind, (const int *)frame, (double *)cl, c->n_seq, c->stream);
            }
            const size_t o = f * (size_t)c->n_seq;
            // consecutive launches overlap (programmatic dependent launch): frame f+1 computes its labels
            // while frame f finishes its searches.  With per-frame outputs the copies and the dedupe of frame f
            // come between them, and the launches are ordinary; so they are with a conversion between them, whose
            // output the frame kernel reads in front of its dependency wait.
            if (run_frame_fused(c, cl, c->d_labels, c->d_nn_idx, c->d_nn_dist, pos_predict + o, pos_last + o, pos_final + o,
                                /*pdl=*/!so && !raw))
                return 1;
            if (!so) continue;
            // frame f's results while the context holds them: the map just built carries its label masks, and
            // the map it searched (now map_alt) is intact until the next frame's kernel
            if (seq_out.nn_idx)
                CU(cudaMemcpyAsync(seq_out.nn_idx + f * c->ntot, c->d_nn_idx, c->ntot * 4, cudaMemcpyDeviceToDevice, c->stream));
            if (seq_out.nn_dist)
                CU(cudaMemcpyAsync(seq_out.nn_dist + f * c->ntot, c->d_nn_dist, c->ntot * 8, cudaMemcpyDeviceToDevice,
                                   c->stream));
            if (seq_out.mask)
                CU(cudaMemcpyAsync(seq_out.mask + f * nr * n_chunks, c->map.mask, nr * n_chunks * 4, cudaMemcpyDeviceToDevice,
                                   c->stream));
            if (part) {
                const MatchOut out = {c->d_nn_idx, c->d_nn_dist, c->d_corr_rows, c->d_corr_row_count};
                const PoseBatch loc = pose_batch(c, pos_predict + o, pos_last + o);
                double *pf = part + f * part_frame * 5;
                if (tile_parts) {
                    const FitMailbox no_mail = {nullptr, nullptr, 0ull};
                    CU((cudaError_t)launch_dedupe_stats(cl, c->d_labels, c->map_alt, out, loc, c->n_seq, c->rows, c->cols,
                                                        c->stream, pf, no_mail));
                } else {
                    launch_dedupe(cl, c->d_labels, c->map_alt, out, loc, c->n_seq, c->rows, c->cols, c->stream, pf, false);
                }
                c->launches++;
            }
        }
    }
    if (part) {
        launch_seq_fit_totals(part, !tile_parts, (int)(part_frame / c->n_seq), (int)n_frames, c->n_seq,
                              (double *)so->fit_stats, c->stream);
        c->launches++;
    }
    c->cloud_resident = false;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int nav_frontend_sequence_dev(nav_ctx *c, const void *dev_frames, size_t n_frames,
                                         const nav_pos *pos_predict, const nav_pos *pos_last,
                                         const nav_pos *pos_final) {
    CTX_ENTER(c, "nav_frontend_sequence_dev");
    return frontend_sequence(c, "nav_frontend_sequence_dev", dev_frames, NAV_RUN_INPUT_XYZ, n_frames, pos_predict,
                             pos_last, pos_final, nullptr);
}

extern "C" int nav_frontend_sequence_out_dev(nav_ctx *c, const void *dev_frames, size_t n_frames,
                                             const nav_pos *pos_predict, const nav_pos *pos_last,
                                             const nav_pos *pos_final, const nav_sequence_out *out) {
    CTX_ENTER(c, "nav_frontend_sequence_out_dev");
    return frontend_sequence(c, "nav_frontend_sequence_out_dev", dev_frames, NAV_RUN_INPUT_XYZ, n_frames, pos_predict,
                             pos_last, pos_final, out);
}

extern "C" int nav_frontend_sequence_dev_ex(nav_ctx *c, const void *dev_frames, int input_kind, size_t n_frames,
                                            const nav_pos *pos_predict, const nav_pos *pos_last,
                                            const nav_pos *pos_final, const nav_sequence_out *out) {
    CTX_ENTER(c, "nav_frontend_sequence_dev_ex");
    return frontend_sequence(c, "nav_frontend_sequence_dev_ex", dev_frames, input_kind, n_frames, pos_predict, pos_last,
                             pos_final, out);
}

extern "C" int nav_frame_results_dev(nav_ctx *c, nav_frame_results *out) {
    if (!c || !out) return fail("nav_frame_results_dev: null argument");
    out->labels = c->d_labels;
    out->nn_idx = c->d_nn_idx;
    out->nn_dist = c->d_nn_dist;
    out->global = c->map.pts;
    out->map_mask = c->map.mask;
    return 0;
}

extern "C" int nav_row_map_export(nav_ctx *c, int seq, int row, nav_point *pts_out, int32_t *col_out, size_t *n_out) {
    CTX_ENTER(c, "nav_row_map_export");
    if (!pts_out || !n_out) return fail("nav_row_map_export: null argument");
    if (seq < 0 || seq >= c->n_seq || row < 0 || row >= c->rows) return fail("nav_row_map_export: bad row");
    *n_out = 0;
    if (!c->have_map) return 0;
    const size_t rid = (size_t)seq * c->rows + row, cols = c->cols;
    double *d_out = c->d_flat + cols * 3;
    int *d_col = (int *)(c->d_flat + cols * 6) + cols;
    launch_flatten_row(c->map.pts + rid * cols * 3, nullptr, c->map.mask + rid * c->map.n_chunks, d_out, d_col,
                       c->d_flat_count, c->cols, c->stream);
    c->launches++;
    CU(cudaStreamSynchronize(c->stream));
    int n = 0;
    CU(cudaMemcpy(&n, c->d_flat_count, 4, cudaMemcpyDeviceToHost));
    if (n > 0) {
        CU(cudaMemcpy(pts_out, d_out, (size_t)n * 24, cudaMemcpyDeviceToHost));
        if (col_out) CU(cudaMemcpy(col_out, d_col, (size_t)n * 4, cudaMemcpyDeviceToHost));
    }
    *n_out = (size_t)n;
    return 0;
}

extern "C" int nav_set_tie_rule(nav_ctx *c, int rule) {
    CTX_ENTER(c, "nav_set_tie_rule");
    if (rule != NAV_TIE_LOWEST_INDEX && rule != NAV_TIE_REFERENCE)
        return fail("nav_set_tie_rule: unknown tie rule %d (NAV_TIE_LOWEST_INDEX = 0, NAV_TIE_REFERENCE = 1)", rule);
    if (rule == NAV_TIE_REFERENCE && !c->d_tie_rec) {  // one record per pixel: the list cannot overflow
        TieRec *rec = nullptr;
        unsigned *count = nullptr;
        int2 *fix = nullptr;
        if (cudaMalloc((void **)&rec, c->ntot * sizeof(TieRec)) != cudaSuccess ||
            cudaMalloc((void **)&count, 4) != cudaSuccess || cudaMalloc((void **)&fix, c->ntot * sizeof(int2)) != cudaSuccess) {
            cudaGetLastError();
            for (void *p : {(void *)rec, (void *)count, (void *)fix})
                if (p) cudaFree(p);
            return fail("nav_set_tie_rule: cudaMalloc of the tie list (%zu records) failed", c->ntot);
        }
        c->d_tie_rec = rec;
        c->d_tie_count = count;
        c->d_tie_fix = fix;
    }
    c->tie_rule = rule;
    return 0;
}

extern "C" int nav_tie_rule(const nav_ctx *c) { return c ? c->tie_rule : NAV_TIE_LOWEST_INDEX; }

extern "C" uint64_t nav_tie_resolve_count(const nav_ctx *c) { return c ? c->tie_resolved : 0; }

extern "C" uint64_t nav_exact_fallback_count(nav_ctx *c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    unsigned v = 0;
    cudaStreamSynchronize(c->stream);
    cudaMemcpy(&v, c->d_n_exact, 4, cudaMemcpyDeviceToHost);
    return v;
}

// ------------------------------------------------------------------ kd-tree ------------------
struct nav_kdtree {
    int device = 0, sm_count = 148;
    size_t n = 0;
    KdNode *d_nodes = nullptr;
    double *d_pts = nullptr;  // build input order, for nearest_out
    double *d_bbox = nullptr; // lo.xyz, hi.xyz of the points (query ordering)
    cudaStream_t stream = nullptr;
    cudaStream_t user_stream = nullptr;  // caller's stream of the most recent *_dev call
    bool on_user_stream = false;         // ... whose work may still be in flight
    uint64_t launches = 0;
    // query scratch
    double *d_q = nullptr, *d_dist = nullptr;
    int *d_idx = nullptr;
    size_t q_cap = 0;
};

extern "C" void nav_kdtree_free(nav_kdtree *t) {
    if (!t) return;
    cudaSetDevice(t->device);
    if (t->on_user_stream) cudaStreamSynchronize(t->user_stream);
    if (t->stream) cudaStreamSynchronize(t->stream);
    // nodes / points / box come from the stream-ordered pool (no device-wide synchronisation, no
    // page mapping per build); the query scratch of the host path is plain cudaMalloc memory
    for (void *p : {(void *)t->d_nodes, (void *)t->d_pts, (void *)t->d_bbox})
        if (p) cudaFreeAsync(p, t->stream);
    for (void *p : {(void *)t->d_q, (void *)t->d_dist, (void *)t->d_idx})
        if (p) cudaFree(p);
    if (t->stream) {
        cudaStreamSynchronize(t->stream);
        cudaStreamDestroy(t->stream);
    }
    delete t;
}

static nav_kdtree *kd_new(int device, size_t n, bool on_user_stream, cudaStream_t user_stream) {
    int ndev = nav_device_count();
    if (ndev == 0) {
        fail("nav_kdtree_build: no CUDA device visible -- libnavslam_b200 has no CPU fallback");
        return nullptr;
    }
    if (device < 0 || device >= ndev) {
        fail("nav_kdtree_build: device %d out of range", device);
        return nullptr;
    }
    if (n > (size_t)0x7fffffff) {
        fail("nav_kdtree_build: %zu points exceed the 2^31-1 limit of int32 indices", n);
        return nullptr;
    }
    CUP(cudaSetDevice(device));
    nav_kdtree *t = new nav_kdtree();
    t->device = device;
    t->n = n;
    cudaDeviceGetAttribute(&t->sm_count, cudaDevAttrMultiProcessorCount, device);
    t->on_user_stream = on_user_stream;
    t->user_stream = user_stream;
    bool ok = cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking) == cudaSuccess;
    const cudaStream_t as = on_user_stream ? user_stream : t->stream;  // the stream the build runs on
    // tree storage and the build's workspace come from the library's own stream-ordered pool
    // (kd_pool_alloc): no device-wide synchronisation, no page mapping per build, and the device's
    // default pool is left as the application configured it
    ok = ok && kd_pool_alloc((void **)&t->d_bbox, 64, device, as) == cudaSuccess;  // 48 B box + 8 B work-queue counter
    if (ok && n)
        ok = kd_pool_alloc((void **)&t->d_nodes, n * sizeof(KdNode), device, as) == cudaSuccess &&
             kd_pool_alloc((void **)&t->d_pts, n * 24, device, as) == cudaSuccess;
    if (!ok) {
        cudaGetLastError();
        fail("nav_kdtree_build: device allocation for %zu points failed", n);
        nav_kdtree_free(t);
        return nullptr;
    }
    return t;
}

static int default_split_rule() {
    // NAV_KD_SPLIT=cyclic|widest overrides the rule of nav_kdtree_build / nav_kdtree_build_dev (read once)
    static const char *e = getenv("NAV_KD_SPLIT");
    if (e && !strcmp(e, "cyclic")) return kSplitCyclic;
    return kSplitWidest;
}

extern "C" nav_kdtree *nav_kdtree_build_ex(int device, const void *points, size_t n, int points_on_device,
                                           void *cuda_stream, int split_rule) {
    const char *name = points_on_device ? "nav_kdtree_build_dev" : "nav_kdtree_build";
    if (n && !points) {
        fail("%s: null points", name);
        return nullptr;
    }
    if (split_rule != kSplitCyclic && split_rule != kSplitWidest) {
        fail("%s: unknown split rule %d", name, split_rule);
        return nullptr;
    }
    nav_kdtree *t = kd_new(device, n, points_on_device != 0, (cudaStream_t)cuda_stream);
    if (!t) return nullptr;
    // device input: the caller's stream (0 = legacy default stream), no synchronisation;
    // host input: the tree's own stream, synchronised before returning
    cudaStream_t s = points_on_device ? (cudaStream_t)cuda_stream : t->stream;
    cudaError_t e = cudaSuccess;
    if (n) {
        e = cudaMemcpyAsync(t->d_pts, points, n * 24,
                            points_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess)
            e = kd_build(t->d_pts, n, t->d_nodes, t->d_bbox, t->sm_count, s, &t->launches, split_rule);
        if (e == cudaSuccess && !points_on_device) e = cudaStreamSynchronize(s);
    }
    if (e != cudaSuccess) {
        fail("%s: %s", name, cudaGetErrorString(e));
        nav_kdtree_free(t);
        return nullptr;
    }
    return t;
}

extern "C" nav_kdtree *nav_kdtree_build_dev(int device, const void *dev_points, size_t n, void *cuda_stream) {
    return nav_kdtree_build_ex(device, dev_points, n, 1, cuda_stream, default_split_rule());
}

extern "C" nav_kdtree *nav_kdtree_build(int device, const nav_point *points, size_t n) {
    return nav_kdtree_build_ex(device, points, n, 0, nullptr, default_split_rule());
}

extern "C" size_t nav_kdtree_size(const nav_kdtree *t) { return t ? t->n : 0; }
extern "C" uint64_t nav_kdtree_launch_count(const nav_kdtree *t) { return t ? t->launches : 0; }

__global__ void k_gather_nearest(const double *__restrict__ pts, const int *__restrict__ idx, long long nq,
                                 double *__restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nq;
         i += (long long)gridDim.x * blockDim.x) {
        const int j = idx[i];
        if (j >= 0) {
            out[i * 3] = pts[(long long)j * 3];
            out[i * 3 + 1] = pts[(long long)j * 3 + 1];
            out[i * 3 + 2] = pts[(long long)j * 3 + 2];
        }
    }
}

extern "C" int nav_kdtree_nn_batch_dev(nav_kdtree *t, const void *dev_queries, size_t nq, void *dev_idx,
                                       void *dev_dist, void *cuda_stream) {
    if (!t) return fail("nav_kdtree_nn_batch_dev: null tree");
    if (nq && (!dev_queries || !dev_idx || !dev_dist)) return fail("nav_kdtree_nn_batch_dev: null argument");
    CU(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;  // 0 = legacy default stream
    if (t->on_user_stream && t->user_stream != s) CU(cudaStreamSynchronize(t->user_stream));  // build / last search
    t->user_stream = s;
    t->on_user_stream = true;
    CU(kd_nn(t->d_nodes, t->n, t->d_bbox, (const double *)dev_queries, nq, (int *)dev_idx, (double *)dev_dist,
             t->sm_count, s, &t->launches, (unsigned long long *)(t->d_bbox + 6)));
    return 0;
}

// the shard arithmetic the peer-memory kernels use (host copies, for the tests: it must agree with
// nav-slam_b200/sharding.py shard_bounds on every rank)
extern "C" void nav_shard_range(int64_t n, int world, int rank, int64_t *lo, int64_t *hi) {
    long long a = 0, b = 0;
    shard_range((long long)n, world, rank, a, b);
    if (lo) *lo = a;
    if (hi) *hi = b;
}
extern "C" int nav_shard_owner(int64_t n, int world, int64_t i) { return shard_owner((long long)n, world, (long long)i); }

// ------------------------------------------------------------------ peer-memory exchange -----
// Config 5b (queries sharded across the GPUs of a node against a replicated tree): instead of a collective
// behind the search, every rank's search kernel writes its shard's answers straight into the result buffers of
// ALL ranks (CUDA IPC mappings of each other's memory, NVLink / NVSwitch stores) and posts a flag; a one-warp
// kernel on each rank waits for the eight flags.  Buffers are double-buffered by call parity: a rank can be at
// most one call ahead of the slowest one, because it needs everybody's flag of call k before it starts k + 1.
struct nav_peer {
    int device = 0, world = 1, rank = 0;
    size_t nq_cap = 0, half = 0;
    unsigned char *own = nullptr;
    unsigned char *peer[kMaxPeers] = {};
    bool opened[kMaxPeers] = {};
    unsigned long long seq = 0;
};

// one half (call parity) of a rank's buffer: final dist | final idx | partial dsq | partial idx | flags A | flags B
struct PeerLayout {
    size_t dist, idx, pdsq, pidx, flags_a, flags_b, half;
};
static PeerLayout peer_layout(size_t nq_cap) {
    const size_t part = nq_cap + 2 * kMaxPeers;  // world shards of ceil(nq / world) entries, rounded up to even
    PeerLayout l;
    l.dist = 0;
    l.idx = l.dist + nq_cap * 8;
    l.pdsq = l.idx + nq_cap * 4;
    l.pidx = l.pdsq + part * 8;
    l.flags_a = l.pidx + part * 4;
    l.flags_b = l.flags_a + kMaxPeers * 8;
    l.half = l.flags_b + kMaxPeers * 8;
    return l;
}
static size_t peer_half_bytes(size_t nq_cap) { return peer_layout(nq_cap).half; }

extern "C" void nav_peer_destroy(nav_peer *p) {
    if (!p) return;
    cudaSetDevice(p->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < kMaxPeers; ++r)
        if (p->opened[r]) cudaIpcCloseMemHandle(p->peer[r]);
    if (p->own) cudaFree(p->own);
    delete p;
}

extern "C" nav_peer *nav_peer_create(int device, size_t nq_cap, unsigned char handle_out[64]) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the handle is exchanged as 64 bytes");
    if (!handle_out || nq_cap == 0) {
        fail("nav_peer_create: null argument");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        fail("nav_peer_create: cudaSetDevice(%d) failed", device);
        return nullptr;
    }
    nav_peer *p = new nav_peer();
    p->device = device;
    p->nq_cap = (nq_cap + 1) & ~(size_t)1;
    p->half = peer_half_bytes(p->nq_cap);
    const size_t bytes = 2 * p->half + 64;
    cudaIpcMemHandle_t h;
    if (cudaMalloc((void **)&p->own, bytes) != cudaSuccess || cudaMemset(p->own, 0, bytes) != cudaSuccess ||
        cudaIpcGetMemHandle(&h, p->own) != cudaSuccess) {
        fail("nav_peer_create: %s", cudaGetErrorString(cudaGetLastError()));
        nav_peer_destroy(p);
        return nullptr;
    }
    memcpy(handle_out, &h, 64);
    return p;
}

// handles: world x 64 bytes, in rank order (this rank's own entry is ignored)
extern "C" int nav_peer_connect(nav_peer *p, int world, int rank, const unsigned char *handles) {
    if (!p || !handles) return fail("nav_peer_connect: null argument");
    if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return fail("nav_peer_connect: bad world %d / rank %d", world, rank);
    CU(cudaSetDevice(p->device));
    p->world = world;
    p->rank = rank;
    for (int r = 0; r < world; ++r) {
        if (r == rank) {
            p->peer[r] = p->own;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + (size_t)r * 64, 64);
        void *ptr = nullptr;
        const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail("nav_peer_connect: cannot map the buffer of rank %d: %s", r, cudaGetErrorString(e));
        }
        p->peer[r] = (unsigned char *)ptr;
        p->opened[r] = true;
    }
    return 0;
}

// Answers this rank's shard (nq_shard queries at dev_queries, queries q_lo .. q_lo + nq_shard - 1 of the whole
// set) and delivers it to every rank; when the stream reaches the end of this call the full (idx, dist) arrays
// of ALL ranks' shards are complete in this rank's buffer: *idx_full / *dist_full point at them (valid until
// the call after the next one).
extern "C" int nav_kdtree_nn_allgather_dev(nav_kdtree *t, nav_peer *p, const void *dev_queries, size_t q_lo,
                                           size_t nq_shard, void **idx_full, void **dist_full, void *cuda_stream) {
    if (!t || !p || !idx_full || !dist_full) return fail("nav_kdtree_nn_allgather_dev: null argument");
    if (nq_shard && !dev_queries) return fail("nav_kdtree_nn_allgather_dev: null queries");
    if (q_lo + nq_shard > p->nq_cap) return fail("nav_kdtree_nn_allgather_dev: shard exceeds the buffer (%zu)", p->nq_cap);
    if (t->device != p->device) return fail("nav_kdtree_nn_allgather_dev: tree and buffer live on different devices");
    CU(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    if (t->on_user_stream && t->user_stream != s) CU(cudaStreamSynchronize(t->user_stream));
    t->user_stream = s;
    t->on_user_stream = true;
    const unsigned long long seq = ++p->seq;
    const size_t off = (seq & 1ull) * p->half;
    const PeerLayout l = peer_layout(p->nq_cap);
    KdFanOut fan = {};
    for (int r = 0; r < p->world; ++r) {
        unsigned char *b = p->peer[r] + off;
        fan.dist[r] = (double *)(b + l.dist);
        fan.idx[r] = (int *)(b + l.idx);
        fan.flags[r] = (unsigned long long *)(b + l.flags_a);
    }
    fan.ticket = (unsigned *)(p->own + 2 * p->half);
    fan.q_lo = (long long)q_lo;
    fan.seq = seq;
    fan.world = p->world;
    fan.rank = p->rank;
    CU(kd_nn_fanout(t->d_nodes, t->n, (const double *)dev_queries, nq_shard, fan, s, &t->launches));
    CU(peer_wait((const unsigned long long *)(p->own + off + l.flags_a), p->world, seq,
                 (unsigned *)(p->own + 2 * p->half + 4), s));
    t->launches++;
    *dist_full = p->own + off + l.dist;
    *idx_full = p->own + off + l.idx;
    return 0;
}

// The MAP sharded instead of the queries: `t` holds this rank's part of the map points (idx_offset = index of its
// first point in the whole map).  Every rank searches its part for ALL nq queries (the same array on every rank)
// and sends each partial answer -- squared distance and global index -- to the rank that owns the query; the owners
// take the minimum (distance, index), which is the pair a search of the whole map keeps, and deliver it to every
// rank.  Two exchange rounds over peer memory, no collective; the build of a 10 M-point map costs each of eight
// ranks the build of 1.25 M points.
extern "C" int nav_kdtree_nn_sharded_map_dev(nav_kdtree *t, nav_peer *p, const void *dev_queries, size_t nq,
                                             int64_t idx_offset, void **idx_full, void **dist_full, void *cuda_stream) {
    if (!t || !p || !idx_full || !dist_full) return fail("nav_kdtree_nn_sharded_map_dev: null argument");
    if (nq && !dev_queries) return fail("nav_kdtree_nn_sharded_map_dev: null queries");
    if (nq > p->nq_cap) return fail("nav_kdtree_nn_sharded_map_dev: %zu queries exceed the buffer (%zu)", nq, p->nq_cap);
    if (idx_offset < 0 || idx_offset + (int64_t)t->n > 0x7fffffffLL) return fail("nav_kdtree_nn_sharded_map_dev: index range");
    if (t->device != p->device) return fail("nav_kdtree_nn_sharded_map_dev: tree and buffer live on different devices");
    CU(cudaSetDevice(t->device));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    if (t->on_user_stream && t->user_stream != s) CU(cudaStreamSynchronize(t->user_stream));
    t->user_stream = s;
    t->on_user_stream = true;
    const PeerLayout l = peer_layout(p->nq_cap);
    unsigned *err = (unsigned *)(p->own + 2 * p->half + 4);
    KdFanOut fan = {};
    fan.ticket = (unsigned *)(p->own + 2 * p->half);
    fan.world = p->world;
    fan.rank = p->rank;
    fan.nq_total = (long long)nq;
    fan.shard_cap = (int)(((nq + p->world - 1) / p->world + 1) & ~(size_t)1);
    fan.idx_offset = (int)idx_offset;
    long long lo, hi;
    shard_range((long long)nq, p->world, p->rank, lo, hi);
    fan.q_lo = lo;
    // round 1: partial answers to the owners of the queries
    unsigned long long seq = ++p->seq;
    size_t off = (seq & 1ull) * p->half;
    for (int r = 0; r < p->world; ++r) {
        unsigned char *b = p->peer[r] + off;
        fan.pdsq[r] = (double *)(b + l.pdsq);
        fan.pidx[r] = (int *)(b + l.pidx);
        fan.dist[r] = (double *)(b + l.dist);
        fan.idx[r] = (int *)(b + l.idx);
        fan.flags[r] = (unsigned long long *)(b + l.flags_a);
    }
    fan.seq = seq;
    CU(kd_nn_partial(t->d_nodes, t->n, (const double *)dev_queries, nq, fan, s, &t->launches));
    CU(peer_wait((const unsigned long long *)(p->own + off + l.flags_a), p->world, seq, err, s));
    // round 2: merge this rank's query shard and deliver it to everybody (same half, second set of flags)
    for (int r = 0; r < p->world; ++r) fan.flags[r] = (unsigned long long *)(p->peer[r] + off + l.flags_b);
    CU(peer_merge(fan, s));
    CU(peer_wait((const unsigned long long *)(p->own + off + l.flags_b), p->world, seq, err, s));
    t->launches += 3;
    *dist_full = p->own + off + l.dist;
    *idx_full = p->own + off + l.idx;
    return 0;
}

// after a synchronisation: 0 if every wait so far saw all ranks arrive, else an error naming the first missing rank
extern "C" int nav_peer_check(nav_peer *p) {
    if (!p) return fail("nav_peer_check: null argument");
    CU(cudaSetDevice(p->device));
    unsigned err = 0;
    CU(cudaMemcpy(&err, p->own + 2 * p->half + 4, 4, cudaMemcpyDeviceToHost));
    if (err) return fail("nav_peer: rank %u did not deliver within 30 s", err - 1u);
    return 0;
}

extern "C" int nav_kdtree_nn_batch(nav_kdtree *t, const nav_point *queries, size_t nq, int32_t *idx_out,
                                   double *dist_out, nav_point *nearest_out) {
    if (!t) return fail("nav_kdtree_nn_batch: null tree");
    if (nq == 0) return 0;
    if (!queries || !idx_out || !dist_out) return fail("nav_kdtree_nn_batch: null argument");
    CU(cudaSetDevice(t->device));
    if (t->on_user_stream) {  // a device-side build or search on the caller's stream may still be running
        CU(cudaStreamSynchronize(t->user_stream));
        t->on_user_stream = false;
    }
    if (nq > t->q_cap) {
        for (void *p : {(void *)t->d_q, (void *)t->d_dist, (void *)t->d_idx})
            if (p) cudaFree(p);
        t->d_q = t->d_dist = nullptr;
        t->d_idx = nullptr;
        t->q_cap = 0;
        CU(cudaMalloc((void **)&t->d_q, nq * 24 * 2));  // queries + gathered nearest points
        CU(cudaMalloc((void **)&t->d_dist, nq * 8));
        CU(cudaMalloc((void **)&t->d_idx, nq * 4));
        t->q_cap = nq;
    }
    CU(cudaMemcpyAsync(t->d_q, queries, nq * 24, cudaMemcpyHostToDevice, t->stream));
    CU(kd_nn(t->d_nodes, t->n, t->d_bbox, t->d_q, nq, t->d_idx, t->d_dist, t->sm_count, t->stream, &t->launches,
             (unsigned long long *)(t->d_bbox + 6)));
    CU(cudaMemcpyAsync(idx_out, t->d_idx, nq * 4, cudaMemcpyDeviceToHost, t->stream));
    CU(cudaMemcpyAsync(dist_out, t->d_dist, nq * 8, cudaMemcpyDeviceToHost, t->stream));
    if (nearest_out && t->n) {
        double *d_near = t->d_q + nq * 3;
        k_gather_nearest<<<(unsigned)((nq + 255) / 256), 256, 0, t->stream>>>(t->d_pts, t->d_idx, (long long)nq, d_near);
        t->launches++;
        CU(cudaMemcpyAsync(nearest_out, d_near, nq * 24, cudaMemcpyDeviceToHost, t->stream));
    }
    CU(cudaStreamSynchronize(t->stream));
    return 0;
}

extern "C" int nav_kdtree_export(nav_kdtree *t, nav_point *nodes_out, int32_t *orig_idx_out, int32_t *axis_out) {
    if (!t || !nodes_out || !orig_idx_out) return fail("nav_kdtree_export: null argument");
    CU(cudaSetDevice(t->device));
    if (t->on_user_stream) CU(cudaStreamSynchronize(t->user_stream));
    CU(cudaStreamSynchronize(t->stream));
    std::vector<KdNode> h(t->n);
    CU(cudaMemcpy(h.data(), t->d_nodes, t->n * sizeof(KdNode), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < t->n; ++i) {
        nodes_out[i].x = h[i].x;
        nodes_out[i].y = h[i].y;
        nodes_out[i].z = h[i].z;
        orig_idx_out[i] = h[i].idx;
        if (axis_out) axis_out[i] = h[i].axis;
    }
    return 0;
}

extern "C" int nav_bruteforce_nn_batch_dev(int device, const void *dev_points, size_t n, const void *dev_queries,
                                           size_t nq, void *dev_idx, void *dev_dist, int use_tensor_cores,
                                           void *cuda_stream) {
    if (nav_device_count() == 0) return fail("nav_bruteforce_nn_batch_dev: no CUDA device");
    if (nq && (!dev_queries || !dev_idx || !dev_dist || (n && !dev_points)))
        return fail("nav_bruteforce_nn_batch_dev: null argument");
    CU(cudaSetDevice(device));
    if (use_tensor_cores) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        static const bool want_stats = getenv("NAV_TC_STATS") != nullptr;  // prints the re-rank volume (forces a sync)
        unsigned long long evals = 0;
        CU(bf_nn_tc((const double *)dev_points, n, (const double *)dev_queries, nq, (int *)dev_idx, (double *)dev_dist,
                    sms, (cudaStream_t)cuda_stream, want_stats ? &evals : nullptr));
        if (want_stats)
            fprintf(stderr, "nav_bruteforce_nn_batch_dev[tensor cores]: n=%zu nq=%zu exact re-rank evaluations=%llu (%.1f per query)\n",
                    n, nq, evals, nq ? (double)evals / (double)nq : 0.0);
        return 0;
    }
    CU(bf_nn((const double *)dev_points, n, (const double *)dev_queries, nq, (int *)dev_idx, (double *)dev_dist,
             (cudaStream_t)cuda_stream));
    return 0;
}
