// stencil.cu -- range-image kernels: curvature / edge labels (a3), depth->xyz (a2), rigid
// transform (a7).  Reference arithmetic: src/slam.c:11-61, utils/pointcloud.c:8-48,
// src/slam.c:145-160.
//
// Curvature stencil layout.  An image row is an AoS run of C points (24 B each).  One CTA owns a
// tile of kTile consecutive columns of one row: it stages the tile plus a 2-point halo on each
// side in shared memory with coalesced 8-byte loads, computes for every staged point the two
// *forward* distances f1(j)=|p_j - p_{j+1}| and f2(j)=|p_j - p_{j+2}| once (the backward taps of
// the reference are the same numbers: p_j - p_{j-1} = -(p_{j-1} - p_j) exactly, and the sign is
// squared away), shares them through shared memory, and then evaluates
//     S = ((d-2 + d-1) + d+1) + d+2, avg = S/4, V = sum (d-avg)^2 in tap order,
//     curv = (V/4) / (avg*avg + (double)1e-6f), label = curv > 0.1
// exactly as src/slam.c:37-58 does.  That halves the fp64 square roots (2 per point, not 4; the
// reference evaluates 8).  Algorithmic traffic: 24 B read + 4 B written per point (SURVEY 8d).
#include <stdlib.h>

#include "nav_bulk.cuh"
#include "nav_kernels.cuh"
#include "stencil_tile.cuh"

namespace nav {

// labels for n_rows image rows (any number of images back to back): persistent grid-stride loop
// over (row, 256-column tile) pairs, fp32-filtered evaluation with exact fallback (stencil_tile.cuh)
__global__ void __launch_bounds__(kTile)
k_labels(const double *__restrict__ cloud, int *__restrict__ labels, long long n_rows, int cols,
         int tiles_per_row, unsigned *__restrict__ n_exact) {
    __shared__ StencilSmem s;
    const long long n_tiles = n_rows * tiles_per_row;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long row = tile / tiles_per_row;
        const int c0 = (int)(tile % tiles_per_row) * kTile;
        tile_stage(s, cloud + row * (long long)cols * 3, c0, cols);
        __syncthreads();
        const int label = tile_labels_filtered(s, c0, cols, n_exact);
        const int col = c0 + threadIdx.x;
        if (col < cols) labels[row * (long long)cols + col] = label;
    }
}

// ---- the same stencil as a 1-D stream fed by the TMA engine ----------------------------------------
// Batched labelling is a pure HBM stream (28 B/point).  Images are stored back to back, so the whole
// batch is treated as ONE run of n_pts points: a tile is 240 consecutive points (+2 halo points each
// side), wherever row boundaries fall -- the stencil is only *evaluated* for columns [2, cols-3],
// whose taps never leave their row, and border columns get label 0.
//   * loads: cp.async.bulk (TMA, 1-D) of the 5 856-byte tile into a 4-stage shared-memory ring; one
//     elected thread issues the copy for tile k+3 while the CTA works on tile k.  Every tile starts
//     at a multiple of 48 bytes, so the 16-byte alignment rule holds for the start of any tile; the
//     size rule (a multiple of 16 bytes) fails only for the last tile of an odd-sized batch, whose
//     final 8 bytes are stored by the producer thread itself.
//   * full/empty mbarriers instead of __syncthreads: warps never wait for each other, only for data.
//   * each warp owns 30 output points: its 32 lanes compute the forward distances of 32 consecutive
//     points (fp64 differences -> fp32) and exchange them with two shuffles; lanes 2..31 then decide
//     their label (fp32 filter, exact binary64 fallback, stencil_tile.cuh).  No shared-memory round
//     trip for the distances, 94 % lane efficiency.
#ifndef NAV_STENCIL_STAGES
#define NAV_STENCIL_STAGES 4
#endif
constexpr int kStages = NAV_STENCIL_STAGES;
constexpr int kWarpOut = 30;                 // output points per warp per tile
constexpr int kWarps = kTile / 32;           // 8 warps
constexpr int kTileOut = kWarps * kWarpOut;  // 240 output points per tile
constexpr int kTileIn = kTileOut + 2 * kHalo;
constexpr int kTileInBytes = kTileIn * 24;
static_assert(kTileInBytes % 16 == 0 && (kTileOut * 24) % 16 == 0, "bulk copies move multiples of 16 bytes");

// Measured on the 1000-image batch (share of the measured HBM peak): 6 CTAs/SM (40 registers, spills)
// 66.8 %, 5 CTAs/SM (48 registers) 72.5 %, 4 CTAs/SM (54 registers) 73.8 %; the same ring with the
// arithmetic removed reaches 94 %, so the kernel is bound by instruction issue, not by bytes in flight.
#ifndef NAV_STENCIL_MIN_CTAS
#define NAV_STENCIL_MIN_CTAS 4
#endif
__global__ void __launch_bounds__(kTile, NAV_STENCIL_MIN_CTAS)
k_labels_tma(const double *__restrict__ cloud, int *__restrict__ labels, unsigned n_pts, unsigned cols,
             unsigned n_tiles, unsigned *__restrict__ n_exact) {
    __shared__ __align__(128) double s_pts[kStages][kTileIn * 3];
    __shared__ __align__(8) unsigned long long s_full[kStages], s_empty[kStages];
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kStages; ++i) {
            mbar_init(&s_full[i], 1);
            mbar_init(&s_empty[i], kWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // producer (thread 0): fetch this CTA's next tile into the next ring slot
    unsigned p_tile = blockIdx.x, p_stage = 0, p_round = 0;
    auto issue = [&]() {
        if (p_tile < n_tiles) {
            if (p_round > 0) mbar_wait(&s_empty[p_stage], (p_round - 1) & 1u);  // all warps released the slot
            const long long g0 = (long long)p_tile * kTileOut - kHalo;  // first staged point
            const long long lo = g0 < 0 ? 0 : g0;
            const long long hi = g0 + kTileIn > (long long)n_pts ? (long long)n_pts : g0 + kTileIn;
            const unsigned bytes = (unsigned)(hi - lo) * 24u;
            // bulk copies move multiples of 16 bytes.  Every tile starts at a multiple of 48 bytes and holds
            // an even number of points, except the last tile of a batch with an odd number of points: its
            // size is 8 mod 16.  The trailing double (z of the very last point, a tap of column cols-3) is
            // then stored by hand; this thread's arrive below publishes it together with the copy.
            const unsigned bulk = bytes & ~15u;
            double *dst = &s_pts[p_stage][(int)(lo - g0) * 3];
            if (bulk != bytes) dst[bulk / 8] = __ldg(cloud + lo * 3 + bulk / 8);
            mbar_expect_tx(&s_full[p_stage], bulk);
            bulk_g2s(dst, cloud + lo * 3, bulk, &s_full[p_stage]);
        }
        p_tile += gridDim.x;
        if (++p_stage == kStages) {
            p_stage = 0;
            ++p_round;
        }
    };
    if (threadIdx.x == 0)
        for (int k = 0; k < kStages - 1; ++k) issue();

    // this lane's point: global index and column, advanced incrementally from tile to tile (32-bit:
    // launch_labels only takes this kernel for batches of fewer than 2^31 points)
    const unsigned li = warp * kWarpOut + lane;  // local index in the staged tile
    const unsigned step = gridDim.x * (unsigned)kTileOut;
    const unsigned step_col = step % cols;
    unsigned g = blockIdx.x * (unsigned)kTileOut + li - kHalo;  // wraps to 0xfffffffe/f for the very first lanes
    unsigned col = (g + cols) % cols;                          // (those are never evaluated: lane < 2)
    const bool out_lane = lane >= 2;

    // ring state as plain registers -- slot pointer, barrier addresses -- advanced and wrapped by hand, so
    // that the loop does not re-derive shared-memory addresses from the slot number in every iteration
    const double *pts = s_pts[0];
    unsigned full_addr = smem_u32(&s_full[0]), empty_addr = smem_u32(&s_empty[0]);
    const unsigned full_end = full_addr + 8u * kStages;
    unsigned parity = 0;
    for (unsigned tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        if (threadIdx.x == 0) issue();
        mbar_wait_addr(full_addr, parity);
        // (slots outside the batch buffer, first/last tile only, hold stale data; they feed border
        //  columns exclusively, which are never evaluated)
#ifdef NAV_STENCIL_NOCOMPUTE  // experiment: the memory path alone (one shared-memory read per lane, label 0)
        if (out_lane && g < n_pts) labels[g] = pts[li * 3] == 12345.678 ? 1 : 0;
#else
        const float f1 = tile_dist32(pts, li, li + 1), f2 = tile_dist32(pts, li, li + 2);
        const float dm2 = __shfl_up_sync(0xffffffffu, f2, 2), dm1 = __shfl_up_sync(0xffffffffu, f1, 1);
        if (out_lane && g < n_pts) {
            int label = 0;
            if (col >= kHalo && col < cols - kHalo) label = label_from_taps32(dm2, dm1, f1, f2, pts, li, n_exact);
            labels[g] = label;
        }
#endif
        __syncwarp();
        if (lane == 0) mbar_arrive_addr(empty_addr);
        g += step;
        col += step_col;
        if (col >= cols) col -= cols;
        pts += kTileIn * 3;
        full_addr += 8u;
        empty_addr += 8u;
        if (full_addr == full_end) {
            pts = s_pts[0];
            full_addr -= 8u * kStages;
            empty_addr -= 8u * kStages;
            parity ^= 1u;
        }
    }
}

// exact binary64 curvature (test hook of the C ABI) and the labels derived from it
__global__ void __launch_bounds__(kTile)
k_curvature(const double *__restrict__ cloud, int *__restrict__ labels, double *__restrict__ curv_out,
            long long n_rows, int cols, int tiles_per_row) {
    __shared__ StencilSmem s;
    const long long n_tiles = n_rows * tiles_per_row;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long row = tile / tiles_per_row;
        const int c0 = (int)(tile % tiles_per_row) * kTile;
        tile_stage(s, cloud + row * (long long)cols * 3, c0, cols);
        __syncthreads();
        const double curv = tile_curvature_exact(s, c0, cols);
        const int col = c0 + threadIdx.x;
        if (col < cols) {
            const long long o = row * (long long)cols + col;
            labels[o] = curv > 0.1 ? 1 : 0;
            curv_out[o] = curv;
        }
    }
}

void launch_labels(const double *cloud, int *labels, double *curv_or_null, long long n_rows, int cols,
                   int sm_count, unsigned *n_exact, cudaStream_t stream) {
    if (n_rows <= 0 || cols <= 0) return;
    const int tiles_per_row = div_up(cols, kTile);
    const long long n_tiles = n_rows * tiles_per_row;
    long long grid = (long long)sm_count * 8;
    if (grid > n_tiles) grid = n_tiles;
    const long long n_pts = n_rows * (long long)cols;
    const long long n_tiles_1d = (n_pts + kTileOut - 1) / kTileOut;
    const bool tma_ok = cols >= 5 && (((uintptr_t)cloud) % 16 == 0) && n_tiles_1d >= 4LL * sm_count &&
                        n_pts < (1LL << 31);
    if (tma_ok && !curv_or_null) {  // persistent: exactly one resident wave
        static int per_sm = 0;
        if (!per_sm && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_labels_tma, kTile, 0) != cudaSuccess)
            per_sm = 4;
        grid = (long long)sm_count * (per_sm > 0 ? per_sm : 4);
    }
    if (curv_or_null)
        k_curvature<<<(unsigned)grid, kTile, 0, stream>>>(cloud, labels, curv_or_null, n_rows, cols, tiles_per_row);
    else if (tma_ok)
        k_labels_tma<<<(unsigned)(grid < n_tiles_1d ? grid : n_tiles_1d), kTile, 0, stream>>>(
            cloud, labels, (unsigned)n_pts, (unsigned)cols, (unsigned)n_tiles_1d, n_exact);
    else
        k_labels<<<(unsigned)grid, kTile, 0, stream>>>(cloud, labels, n_rows, cols, tiles_per_row, n_exact);
}

// ---------------------------------------------------------------- a2 ------------------------
// utils/pointcloud.c:18-47.  tan(theta_col) / tan(phi_row) come from the host's libm (the
// reference's own tan), uploaded once per context; y = (-d) * tan is one rounded multiply (depth_point).
// n_img images of `rows` rows back to back: tan_row is indexed by the row within its image.
__global__ void k_convert(const int *__restrict__ dist, const double *__restrict__ tan_col,
                          const double *__restrict__ tan_row, double *__restrict__ out, int rows, int cols, int n_img) {
    const long long n = (long long)n_img * rows * cols;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)((i / cols) % rows), c = (int)(i % cols);
        const P3 p = depth_point(dist[i], tan_col[c], tan_row[r]);
        out[i * 3 + 0] = p.x;
        out[i * 3 + 1] = p.y;
        out[i * 3 + 2] = p.z;
    }
}

void launch_convert(const int *dist, const double *tan_col, const double *tan_row, double *out, int rows,
                    int cols, int n_img, int sm_count, cudaStream_t stream) {
    const long long n = (long long)n_img * rows * cols;
    if (n <= 0) return;
    long long grid = (n + 255) / 256;
    if (grid > sm_count * 8LL) grid = sm_count * 8LL;
    k_convert<<<(unsigned)grid, 256, 0, stream>>>(dist, tan_col, tan_row, out, rows, cols, n_img);
}

// ---------------------------------------------------------------- integer-mm xyz -----------
// L9 clouds in whole millimetres cross PCIe as int32 [n][3] (12 B/point instead of 24) and are widened here.  Every
// int32 is exact in binary64, so the cloud equals the one the host would have uploaded as doubles, bit for bit.
// The 3n values are one flat run: a 16-byte load of four ints and two 16-byte stores of four doubles per step for the
// first n4 groups of four, the rest one at a time.  n4 = 0 unless both buffers are 16-byte aligned (a frame of a
// device-resident recording may start on any 4-byte boundary).
__global__ void k_widen_mm(const int *__restrict__ in, double *__restrict__ out, long long n_vals, long long n4) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int4 *in4 = reinterpret_cast<const int4 *>(in);
    double2 *out2 = reinterpret_cast<double2 *>(out);
    for (long long i = t; i < n4; i += stride) {
        const int4 v = __ldg(in4 + i);
        out2[2 * i] = make_double2(mm_coord(v.x), mm_coord(v.y));
        out2[2 * i + 1] = make_double2(mm_coord(v.z), mm_coord(v.w));
    }
    for (long long i = 4 * n4 + t; i < n_vals; i += stride) out[i] = mm_coord(in[i]);
}

void launch_widen_mm(const int *in, double *out, long long n_points, int sm_count, cudaStream_t stream) {
    const long long n_vals = n_points * 3;
    if (n_vals <= 0) return;
    const bool vec = (((uintptr_t)in | (uintptr_t)out) & 15u) == 0;
    long long grid = (vec ? n_vals / 4 : n_vals) / 256 + 1;
    if (grid > sm_count * 8LL) grid = sm_count * 8LL;
    k_widen_mm<<<(unsigned)grid, 256, 0, stream>>>(in, out, n_vals, vec ? n_vals >> 2 : 0);
}

// ---------------------------------------------------------------- a7 ------------------------
__global__ void k_transform(const double *__restrict__ in, double *__restrict__ out, long long n, PoseXf pose) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        P3 p = {in[i * 3], in[i * 3 + 1], in[i * 3 + 2]};
        P3 g = xf_point(pose, p);
        out[i * 3] = g.x;
        out[i * 3 + 1] = g.y;
        out[i * 3 + 2] = g.z;
    }
}

void launch_transform(const double *in, double *out, long long n, const PoseXf &pose, int sm_count,
                      cudaStream_t stream) {
    if (n <= 0) return;
    long long grid = (n + 255) / 256;
    if (grid > sm_count * 8LL) grid = sm_count * 8LL;
    k_transform<<<(unsigned)grid, 256, 0, stream>>>(in, out, n, pose);
}

}  // namespace nav
