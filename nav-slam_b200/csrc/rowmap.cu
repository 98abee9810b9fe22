// rowmap.cu -- the per-row map ("kdtree_lastframe[row]", headers/slam.h:14) of the SLAM step and
// the per-row exact nearest-neighbour match against it.
//
// What the reference does (src/slam.c:167-172, 236-284, 422-427; utils/kdtree.c): for every image
// row it compacts the previous frame's edge points (global frame) into an array (flattenPoints),
// builds a pointer kd-tree over those <= MAX_COLS points, and answers one exact 1-NN query per
// labelled point of the current frame against the tree of the *same row*; results are then
// de-duplicated per row.
//
// What this file does instead (same answers, B200-shaped).  A lidar ring is a polyline: points of
// neighbouring columns are neighbours in space.  So the "tree" of a row is simply the mapped
// global cloud of that row, left in place, plus
//     * a 16-bit label mask per block of 16 columns (which of the 16 points are map points),
//     * the bounding box of the labelled points of every 16-column block (leaf box),
//     * the bounding box of every 256-column block (super box).
// Everything is local to a (row, 256-column tile), so both kernels run one independent CTA per
// tile -- 512 CTAs for a 64x2048 image -- with no cross-CTA prefix sums and no compaction (a4) on
// the matching path at all.  Correctness never depends on the polyline assumption: a query visits
// every block whose box lower bound is <= its current best, and the lower bound is a true lower
// bound of the rounded distance the reference computes (nav_common.cuh).
//
//   k_frame_map   : rigid transform of the tile (a7) -> global cloud, label masks, leaf/super boxes
//   k_frame_match : curvature/labels of the tile (a3, fp32-filtered + exact fallback), then one
//                   thread per labelled column: query transform (a7) and exact search (a5/a6),
//                   seeded with the leaf block of its own column.  Ties -> lowest column.
//   k_dedupe_rows : per-row dedupe of src/slam.c:247-283 (a8) with shared-memory atomics
//   k_export_row / k_flatten_row : stable row compaction (a4) for the API and the shim
#include <limits.h>
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>
#include <utility>

#include "nav_bulk.cuh"
#include "nav_kernels.cuh"
#include "stencil_tile.cuh"

namespace nav {

constexpr unsigned kFull = 0xffffffffu;
#ifndef NAV_MATCH_MIN_CTAS
#define NAV_MATCH_MIN_CTAS 4  // 64 registers/thread: keeps the fp32 query bracket live instead of re-converting it
                              // (measured, frames/s single / 8 sequences: 3 CTAs 53.5 K / 56.2 K, 4 CTAs 58.3 K / 62.5 K, 5 CTAs 48.8 K / 63.7 K)
#endif
static_assert(kTile == kChunk * kChunksPerSuper, "one CTA tile = one super block of 16 leaf blocks");

__device__ __forceinline__ P3 load_p3(const double *__restrict__ p) {
    P3 v = {p[0], p[1], p[2]};
    return v;
}
__device__ __forceinline__ P3 ldg_p3(const double *__restrict__ p) {
    P3 v = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
    return v;
}
__device__ __forceinline__ void store_p3(double *__restrict__ p, const P3 &v) {
    p[0] = v.x;
    p[1] = v.y;
    p[2] = v.z;
}

// min / max over the 16 lanes of a half warp with one redux.sync each: floats compare like their
// order-preserving integer images (non-negative floats as they are, negative ones with the magnitude
// bits flipped), so an integer min / max over the half warp is the float min / max
__device__ __forceinline__ int float_order_key(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float float_from_order_key(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }
__device__ __forceinline__ float half_min(float v, unsigned half_mask) {
    return float_from_order_key(__reduce_min_sync(half_mask, float_order_key(v)));
}
__device__ __forceinline__ float half_max(float v, unsigned half_mask) {
    return float_from_order_key(__reduce_max_sync(half_mask, float_order_key(v)));
}

// ---------------------------------------------------------------------------------------------
// One (row, 256-column tile) of the map: transform the thread's own column, write the global
// cloud, the 16-bit label masks, the leaf boxes and the tile's super box.  Called by all kTile
// threads of the CTA (contains one __syncthreads).  mask_out (optional): a second copy of the label masks,
// laid out as map.mask ([n_seq*rows][n_chunks]).
__device__ __forceinline__ void map_tile(bool lab, bool valid, const P3 &p, const PoseXf &pose, const RowMap &map,
                                         int rid, int tile, int c, long long base, float4 *s_lo, float4 *s_hi,
                                         unsigned *__restrict__ mask_out = nullptr) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, half = lane >> 4, l16 = lane & 15;
    P3 g = {0, 0, 0};
    if (valid) {
        g = xf_point(pose, p);
        store_p3(map.pts + (base + c) * 3, g);
    }
    const unsigned ballot = __ballot_sync(kFull, lab);
    const unsigned mask16 = (ballot >> (half * 16)) & 0xffffu;
    // boxes are stored in fp32 rounded outward (see box_lower_bound32); rounding is monotone, so the
    // min of the rounded-down coordinates is the rounded-down min (same for max / rounded up)
    const unsigned half_mask = 0xffffu << (half * 16);
    const float inf = __int_as_float(0x7f800000);
    const float4 flo = make_float4(half_min(lab ? __double2float_rd(g.x) : inf, half_mask),
                                   half_min(lab ? __double2float_rd(g.y) : inf, half_mask),
                                   half_min(lab ? __double2float_rd(g.z) : inf, half_mask), 0.f);
    const float4 fhi = make_float4(half_max(lab ? __double2float_ru(g.x) : -inf, half_mask),
                                   half_max(lab ? __double2float_ru(g.y) : -inf, half_mask),
                                   half_max(lab ? __double2float_ru(g.z) : -inf, half_mask), 0.f);
    const int leaf_in_tile = warp * 2 + half;
    const int leaf = tile * kChunksPerSuper + leaf_in_tile;
    if (l16 == 0) {
        s_lo[leaf_in_tile] = flo;
        s_hi[leaf_in_tile] = fhi;
        if (leaf < map.n_chunks) {
            map.mask[(long long)rid * map.n_chunks + leaf] = mask16;
            if (mask_out) mask_out[(long long)rid * map.n_chunks + leaf] = mask16;
            float4 *b = map.box + ((long long)rid * map.n_chunks + leaf) * 2;
            b[0] = flo;
            b[1] = fhi;
        }
    }
    __syncthreads();
    if (warp == 0) {
        float4 a = s_lo[l16], b = s_hi[l16];
#pragma unroll
        for (int d = 8; d >= 1; d >>= 1) {
            a.x = fminf(a.x, __shfl_xor_sync(kFull, a.x, d, 16));
            a.y = fminf(a.y, __shfl_xor_sync(kFull, a.y, d, 16));
            a.z = fminf(a.z, __shfl_xor_sync(kFull, a.z, d, 16));
            b.x = fmaxf(b.x, __shfl_xor_sync(kFull, b.x, d, 16));
            b.y = fmaxf(b.y, __shfl_xor_sync(kFull, b.y, d, 16));
            b.z = fmaxf(b.z, __shfl_xor_sync(kFull, b.z, d, 16));
        }
        if (lane == 0) {
            float4 *o = map.sbox + ((long long)rid * map.n_super + tile) * 2;
            o[0] = a;
            o[1] = b;
        }
    }
}

// grid = n_rows * tiles_per_row CTAs of kTile threads; thread = one column
__global__ void __launch_bounds__(kTile)
k_frame_map(const double *__restrict__ cloud, const int *__restrict__ labels, RowMap map,
            const __grid_constant__ PoseBatch poses, int rows, int cols, int tiles_per_row) {
    __shared__ float4 s_lo[kChunksPerSuper], s_hi[kChunksPerSuper];
    const int rid = blockIdx.x / tiles_per_row;  // sequence * rows + row
    const int tile = blockIdx.x % tiles_per_row;
    const long long base = (long long)rid * cols;
    const int c = tile * kTile + threadIdx.x;
    const bool valid = c < cols;
    bool lab = false;
    P3 p = {0, 0, 0};
    if (valid) {
        lab = labels[base + c] == 1;
        p = ldg_p3(cloud + (base + c) * 3);
    }
    map_tile(lab, valid, p, poses.p[rid / rows], map, rid, tile, c, base, s_lo, s_hi);
}

// exclusive prefix of `pred` over the block (thread order), plus the block total
__device__ __forceinline__ int block_excl_count(bool pred, int *s_warp, int &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_warps = blockDim.x >> 5;
    const unsigned m = __ballot_sync(kFull, pred);
    const int in_warp = __popc(m & ((1u << lane) - 1u));
    __syncthreads();  // protects s_warp reuse across rounds
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
        int v = lane < n_warps ? s_warp[lane] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += t;
        }
        s_warp[32 + lane] = incl - v;
        if (lane == 31) s_warp[64] = incl;
    }
    __syncthreads();
    total = s_warp[64];
    return s_warp[32 + warp] + in_warp;
}

// block_excl_count with one barrier instead of three: every thread adds up the warp counts itself.  s_warp is
// written without a barrier in front, so two uses must be separated by a barrier of the caller's (match_tile is
// called once per kernel, or once per frame of k_frame_seq with the frame's other barriers in between).
__device__ __forceinline__ int block_excl_count_once(bool pred, int *s_warp, int &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(kFull, pred);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < kTile / 32; ++w) {
        const int v = s_warp[w];
        before += w < warp ? v : 0;
        all += v;
    }
    total = all;
    return before + __popc(m & ((1u << lane) - 1u));
}

// scan the labelled points of one 16-column block of the map row.  `pts` points at column col0 of
// the block (shared-memory copy for the CTA's own neighbourhood, global memory otherwise).  Four
// candidates are loaded before any arithmetic so that their load latencies overlap; a short last
// group repeats its final candidate, which the lexicographic compare ignores.
// kRefTies: best2 also tracks the second smallest dsq over the scanned columns (each column counts once, so two
// columns with the same xyz both count; the repeated padding candidate does not).
template <bool kRefTies = false>
__device__ __forceinline__ void scan_leaf(const double *pts, unsigned mask, int col0, const P3 &q, double &best,
                                          int &bcol, double &best2) {
    while (mask) {
        int b[4];
        bool real[4];  // kRefTies: false for the padding repeats of a short last group
        b[0] = __ffs(mask) - 1;
        real[0] = true;
        mask &= mask - 1;
#pragma unroll
        for (int i = 1; i < 4; ++i) {
            real[i] = mask != 0;
            b[i] = mask ? __ffs(mask) - 1 : b[i - 1];
            mask &= mask - 1;  // 0 & anything stays 0
        }
        double x[4], y[4], z[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double *p = pts + b[i] * 3;
            x[i] = p[0];
            y[i] = p[1];
            z[i] = p[2];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            // operand order of euclideanDistance(root->point, *target), utils/kdtree.c:116
            const double d = dsq3(dsub(x[i], q.x), dsub(y[i], q.y), dsub(z[i], q.z));
            const int col = col0 + b[i];
            if (d < best || (d == best && col < bcol)) {
                if (kRefTies) best2 = best;
                best = d;
                bcol = col;
            } else if (kRefTies && real[i]) {
                best2 = fmin(best2, d);
            }
        }
    }
}

__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void cp_async_wait_group() {
    asm volatile("cp.async.wait_group %0;" ::"n"(kPending) : "memory");
}

// tile_stage (stencil_tile.cuh) with asynchronous copies: columns [c0-2, c0+kTile+2) of one row into pts
__device__ __forceinline__ void tile_stage_async(double *pts, const double *__restrict__ row_ptr, int c0, int cols) {
    const int first = c0 - kHalo;
    for (int i = threadIdx.x; i < kTilePts * 3; i += kTile) {
        const int col = first + i / 3;
        if (col >= 0 && col < cols)
            cp_async8(&pts[i], row_ptr + (long long)first * 3 + i);
        else
            pts[i] = 0.0;
    }
}

// the CTA's neighbourhood of the row map, prefetched into shared memory while the labels are
// computed: its own 256 columns plus one 16-column leaf on each side (almost every query finds its
// neighbour there), and the super boxes of the whole row
constexpr int kNbLeaves = kChunksPerSuper + 2;
constexpr int kMaxSuperSmem = 64;  // rows wider than 64*256 columns read the super boxes from global memory
constexpr int kMaxRowLeafSmem = 128;  // leaf boxes of the whole row (rows up to 2048 columns); wider rows use global memory
struct MapSmem {
    double pts[kNbLeaves * kChunk * 3];
    float4 box[kNbLeaves * 2];
    float4 sbox[kMaxSuperSmem * 2];
    float4 rbox[kMaxRowLeafSmem * 2];
    // mask[j]: leaf leaf0 + j.  k_frame_seq's bulk copy moves the row's mask words in whole 16-byte groups, from
    // the group that holds leaf0 (= 16 * tile - 1, i.e. 3 mod 4): up to three words in front, three behind.
    unsigned mask_lead[3];
    unsigned mask[kNbLeaves + 3];
};
static_assert(offsetof(MapSmem, mask) % 16 == 12 && sizeof(MapSmem) % 16 == 0, "mask word leaf0 + 1 on a 16-byte boundary");

// one row of the map as the search sees it
struct RowView {
    const double *pts;
    const unsigned *mask;
    const float4 *box;
    const float4 *sbox;
    int n_leaf, n_sup, leaf0;  // leaf0: first leaf of the CTA's shared-memory neighbourhood (may be -1)
};

// row rid (first pixel base = rid * cols) of `map`, as seen by the CTA of 256-column tile `tile`
__device__ __forceinline__ RowView row_view(const RowMap &map, int rid, long long base, int tile) {
    return {map.pts + base * 3, map.mask + (long long)rid * map.n_chunks, map.box + (long long)rid * map.n_chunks * 2,
            map.sbox + (long long)rid * map.n_super * 2, map.n_chunks, map.n_super, tile * kChunksPerSuper - 1};
}

// map data outside the shared-memory neighbourhood: through the read-only path when the map was written by
// an earlier launch, with ordinary (coherent) loads when this launch wrote it (k_loop_step)
template <bool kCoherent, typename T>
__device__ __forceinline__ T ld_map(const T *p) {
    if (kCoherent) return *p;
    return __ldg(p);
}

// asynchronous prefetch (cp.async) of a CTA's neighbourhood of the row map into shared memory (MapSmem);
// complete after cp_async_wait_all + a barrier.  Called by all kTile threads.
template <bool kCoherent>
__device__ __forceinline__ void prefetch_neighbourhood(MapSmem &sm, const RowView &rv, int cols) {
    const int leaf0 = rv.leaf0, n_leaf = rv.n_leaf, n_sup = rv.n_sup;
    const int col_lo = leaf0 * kChunk;
    for (int i = threadIdx.x; i < kNbLeaves * kChunk * 3; i += kTile) {
        const int col = col_lo + i / 3;
        if (col >= 0 && col < cols) cp_async8(&sm.pts[i], rv.pts + (long long)col_lo * 3 + i);
    }
    if (threadIdx.x < kNbLeaves * 2) {
        const int lf = leaf0 + (int)threadIdx.x / 2;
        if (lf >= 0 && lf < n_leaf) cp_async16(&sm.box[threadIdx.x], rv.box + (long long)leaf0 * 2 + threadIdx.x);
    } else if (threadIdx.x >= 64 && threadIdx.x < 64 + kNbLeaves) {
        const int j = threadIdx.x - 64, lf = leaf0 + j;
        sm.mask[j] = (lf >= 0 && lf < n_leaf) ? ld_map<kCoherent>(rv.mask + lf) : 0u;
    } else if (threadIdx.x >= 128 && (int)threadIdx.x < 128 + 2 * min(n_sup, kMaxSuperSmem)) {
        cp_async16(&sm.sbox[threadIdx.x - 128], rv.sbox + (threadIdx.x - 128));
    }
    // every leaf box of the row: a query near the edge of its tile (or far from its neighbour) tests
    // the leaves of other super blocks too, and sixteen dependent global loads made those warps the tail
    if (n_leaf <= kMaxRowLeafSmem && (int)threadIdx.x < 2 * n_leaf) cp_async16(&sm.rbox[threadIdx.x], rv.box + threadIdx.x);
}

// ---- bulk staging (k_frame_seq<kBulk = true>): one thread issues one cp.async.bulk per contiguous range and
// every consumer waits on the range's mbarrier.  Taken when the rules of the copies hold for every range
// (frame_seq_bulk_ok): an even number of columns (a row, and every span of it starting at an even column, is then
// 16-byte aligned and a multiple of 48 bytes long), a mask row of a multiple of four words, 16-byte aligned base
// pointers, and a row whose leaf boxes fit sm.rbox.

// columns [max(c0-2, 0), min(c0+kTile+2, cols)) of one row (row_ptr = its column 0) into pts, laid out as
// tile_stage_async does; the slots of columns outside the row are not written (k_frame_seq zeroes them once)
__device__ __forceinline__ void tile_stage_bulk(double *pts, const double *row_ptr, int c0, int cols,
                                                unsigned long long *bar) {
    const int first = c0 - kHalo, lo = max(first, 0), hi = min(first + kTilePts, cols);
    const unsigned bytes = (unsigned)(hi - lo) * 24u;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(pts + (lo - first) * 3, row_ptr + (long long)lo * 3, bytes, bar);
}

// ---- raw tiles of depth (kE = 1) and integer-mm (kE = 3) frames: kE int32 per column, columns [c0-4, c0+kTile+4)
// of the row.  The span is rounded out to whole groups of four columns, so that for rows of a multiple of four
// columns it starts on a 16-byte boundary and is a multiple of 16 bytes long (16 B per 4 depth values, 48 B per 4 mm
// points).  Element li of the RawTile view (column c0 - kHalo + li) is element li + kRawLead - kHalo of the buffer.
constexpr int kRawLead = 4;
constexpr int kRawPts = kTile + 2 * kRawLead;  // 264 staged columns
template <int kKind>
constexpr int kRawElems = kKind == kKindMm ? 3 : 1;  // int32 per point

// the 4-byte cp.async form (any 4-byte aligned row): slots of columns outside the row are zeroed
template <int kE>
__device__ __forceinline__ void raw_stage_async(int *raw, const int *__restrict__ row_ptr, int c0, int cols) {
    const int first = c0 - kRawLead;
    for (int i = threadIdx.x; i < kRawPts * kE; i += kTile) {
        const int col = first + i / kE;
        if (col >= 0 && col < cols)
            cp_async4(&raw[i], row_ptr + (long long)first * kE + i);
        else
            raw[i] = 0;
    }
}
// the bulk form (rows of a multiple of four columns, 16-byte aligned): one copy of the columns inside the row; the
// other slots are not written (k_frame_seq zeroes them once)
template <int kE>
__device__ __forceinline__ void raw_stage_bulk(int *raw, const int *row_ptr, int c0, int cols, unsigned long long *bar) {
    const int first = c0 - kRawLead, lo = max(first, 0), hi = min(first + kRawPts, cols);
    const unsigned bytes = (unsigned)(hi - lo) * 4u * kE;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(raw + (lo - first) * kE, row_ptr + (long long)lo * kE, bytes, bar);
}
// the tans of the staged columns (depth only; zero outside the row), read once per launch: they do not change from
// frame to frame.  Complete after the caller's next CTA barrier.
__device__ __forceinline__ void stage_tan_cols(double *s_tan, const double *__restrict__ tan_col, int c0, int cols) {
    for (int i = threadIdx.x; i < kRawPts; i += kTile) {
        const int col = c0 - kRawLead + i;
        s_tan[i] = col >= 0 && col < cols ? tan_col[col] : 0.0;
    }
}
// the RawTile view of a raw buffer
template <int kKind>
__device__ __forceinline__ RawTile<kKind> raw_view(const int *raw, const double *s_tan, double tan_r) {
    if constexpr (kKind == kKindDepth)
        return RawTile<kKindDepth>{raw + (kRawLead - kHalo), s_tan + (kRawLead - kHalo), tan_r};
    else
        return RawTile<kKindMm>{raw + (kRawLead - kHalo) * 3};
}

// the neighbourhood of prefetch_neighbourhood, clamped to the row: the points of its leaves, the leaf boxes of
// the row (rbox), the super boxes and the mask words.  sm.box is not staged: search_row reads it only for rows
// wider than kMaxRowLeafSmem leaves.  The mask words go in whole 16-byte groups of the row (MapSmem); words of
// leaves outside the row are never written (k_frame_seq zeroes them once).
__device__ __forceinline__ void stage_neighbourhood_bulk(MapSmem &sm, const RowView &rv, int cols,
                                                         unsigned long long *bar) {
    const int leaf0 = rv.leaf0, lf_lo = max(leaf0, 0), lf_hi = min(leaf0 + kNbLeaves, rv.n_leaf);
    const int col_lo = lf_lo * kChunk, col_hi = min(lf_hi * kChunk, cols);
    const int w_lo = lf_lo & ~3, w_hi = min((lf_hi + 3) & ~3, rv.n_leaf);
    const unsigned pts_b = (unsigned)(col_hi - col_lo) * 24u, row_b = (unsigned)rv.n_leaf * 32u,
                   sup_b = (unsigned)rv.n_sup * 32u, mask_b = (unsigned)(w_hi - w_lo) * 4u;
    mbar_expect_tx(bar, pts_b + row_b + sup_b + mask_b);
    bulk_g2s(sm.pts + (lf_lo - leaf0) * kChunk * 3, rv.pts + (long long)col_lo * 3, pts_b, bar);
    bulk_g2s(sm.rbox, rv.box, row_b, bar);
    bulk_g2s(sm.sbox, rv.sbox, sup_b, bar);
    bulk_g2s(sm.mask + (w_lo - leaf0), rv.mask + w_lo, mask_b, bar);
}

// exact nearest labelled map point of the row for query q of column qc: seed leaf, its neighbours, then the
// box hierarchy.  best = smallest dsq (INFINITY if the row map is empty), bcol = its column (lowest on ties).
// kRefTies: *best2_out = the second smallest dsq over the scanned columns (scan_leaf).  The pruning needs no change
// for it to see every column whose rounded distance sqrt(dsq) equals sqrt(best): two doubles with the same correctly
// rounded square root differ by a factor of at most (1 + 2^-51), so such a column has dsq <= (1 + 2^-51) * best, and
// no float lies strictly between best_up = float_round_up(best) and that dsq.  A leaf's fp32 lower bound is a float
// <= the dsq of each of its points (box_lower_bound32), hence <= best_up, and the leaf is scanned.  best_up only
// decreases towards its final value, so this holds for every test made along the way: the warp-cooperative cull
// (wbest >= the lane's best_up, and the warp's bound is below the lane's), the per-lane super-box path of rows wider
// than 2048 columns and the neighbour leaves alike; while best_up is +inf nothing is pruned.
template <bool kCoherent, bool kRefTies = false>
__device__ __forceinline__ void search_row(const MapSmem &sm, const RowView &rv, int qc, const P3 &q, double &best,
                                           int &bcol, unsigned wmask, double *best2_out = nullptr) {
    const double *m_pts = rv.pts;
    const unsigned *m_mask = rv.mask;
    const float4 *m_box = rv.box, *m_sbox = rv.sbox;
    const int n_leaf = rv.n_leaf, n_sup = rv.n_sup, leaf0 = rv.leaf0;
    const Q32 q32 = make_q32(q);
    const bool sup_in_smem = n_sup <= kMaxSuperSmem, row_in_smem = n_leaf <= kMaxRowLeafSmem;

    best = INFINITY;
    float best_up = INFINITY;  // float(best) rounded up
    bcol = -1;
    double &b2 = kRefTies ? *best2_out : best;  // kRefTies only (scan_leaf<false> never touches it)
    if (kRefTies) b2 = INFINITY;
    const int seed = qc / kChunk;
    scan_leaf<kRefTies>(sm.pts + (seed - leaf0) * kChunk * 3, sm.mask[seed - leaf0], seed * kChunk, q, best, bcol, b2);
    best_up = __double2float_ru(best);
    // The leaves next to the seed come first, addressed RELATIVE to the seed: the lanes of a warp hold
    // queries of neighbouring columns with different seeds, and stepping through "seed-1, seed+1, ..."
    // together lets every lane scan its own neighbour in the same loop iteration.  (Walking absolute
    // leaf indices instead made the warp execute the union of all lanes' neighbour scans.)
    // Measured (64x2048, frames/s single sequence / 8 sequences per launch): kNear 2: 55.3 K / 55.9 K,
    // kNear 1: 57.8 K / 61.3 K, kNear 0: 49.5 K / 61.0 K -- one neighbour each side gives the mask tests below
    // a tight bound; a second one is rarely needed and costs two more box tests per query.
#ifndef NAV_MATCH_KNEAR
#define NAV_MATCH_KNEAR 1
#endif
    constexpr int kNear = NAV_MATCH_KNEAR;
#pragma unroll
    for (int d = 1; d <= kNear; ++d) {
#pragma unroll
        for (int sgn = -1; sgn <= 1; sgn += 2) {
            const int lf = seed + sgn * d, j = lf - leaf0;
            if (lf < 0 || lf >= n_leaf) continue;
            const bool near_leaf = j >= 0 && j < kNbLeaves;
            const float4 blo = row_in_smem ? sm.rbox[lf * 2] : (near_leaf ? sm.box[j * 2] : ld_map<kCoherent>(m_box + lf * 2));
            const float4 bhi = row_in_smem ? sm.rbox[lf * 2 + 1] : (near_leaf ? sm.box[j * 2 + 1] : ld_map<kCoherent>(m_box + lf * 2 + 1));
            if (box_lower_bound32(blo, bhi, q32) > best_up) continue;
            if (near_leaf)
                scan_leaf<kRefTies>(sm.pts + j * kChunk * 3, sm.mask[j], lf * kChunk, q, best, bcol, b2);
            else
                scan_leaf<kRefTies>(m_pts + (long long)lf * kChunk * 3, ld_map<kCoherent>(m_mask + lf), lf * kChunk, q, best, bcol, b2);
            best_up = __double2float_ru(best);
        }
    }
    // Everything else through the boxes (exactness does not depend on the order of visits).
    // Rows whose leaf boxes are all in shared memory (<= 2048 columns): WARP-COOPERATIVE culling.  The 32 lanes
    // hold queries of neighbouring columns, so their candidate sets are nearly the same; instead of every lane
    // testing 8 super boxes and 16-48 leaf boxes, the warp tests every leaf box of the row ONCE -- lane l takes
    // leaves l, l+32, ... -- against the bounding box of the warp's 32 queries and the loosest of their bounds.
    // That test is a lower bound of every lane's own test (gaps to a bigger box are smaller, rounding down is
    // monotone), so the surviving leaves are a superset of what any lane needs.  Each lane then tests only the
    // survivors against its own query (a warp-uniform loop over a handful of leaves) and scans the ones that pass.
    if (row_in_smem && wmask == kFull) {
        const unsigned lane = threadIdx.x & 31u;
        float wdn[3], wup[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            wdn[d] = float_from_order_key(__reduce_min_sync(kFull, float_order_key(q32.dn[d])));
            wup[d] = float_from_order_key(__reduce_max_sync(kFull, float_order_key(q32.up[d])));
        }
        // best_up >= 0 (or +inf): such floats order like their bit patterns
        const float wbest = __int_as_float(__reduce_max_sync(kFull, __float_as_int(best_up)));
        Q32 wq;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            wq.dn[d] = wdn[d];
            wq.up[d] = wup[d];
        }
        constexpr int kWords = kMaxRowLeafSmem / 32;
        unsigned surv[kWords];
#pragma unroll
        for (int k = 0; k < kWords; ++k) {
            const int lf = k * 32 + (int)lane;
            bool keep = false;
            if (lf < n_leaf) keep = !(box_lower_bound32(sm.rbox[lf * 2], sm.rbox[lf * 2 + 1], wq) > wbest);
            surv[k] = __ballot_sync(kFull, keep);
        }
        // the leaves visited above are done
#pragma unroll
        for (int k = 0; k < kWords; ++k) {
            unsigned own = 0;
            for (unsigned w = surv[k]; w; w &= w - 1) {  // warp-uniform loop
                const int b = __ffs(w) - 1, lf = k * 32 + b;
                const bool pass = !(box_lower_bound32(sm.rbox[lf * 2], sm.rbox[lf * 2 + 1], q32) > best_up);
                own |= (unsigned)pass << b;
            }
#pragma unroll
            for (int d = -kNear; d <= kNear; ++d) {
                const int j = seed + d - k * 32;
                if (j >= 0 && j < 32) own &= ~(1u << j);
            }
            while (own) {
                const int lf = k * 32 + __ffs(own) - 1, j = lf - leaf0;
                own &= own - 1;
                if (box_lower_bound32(sm.rbox[lf * 2], sm.rbox[lf * 2 + 1], q32) > best_up) continue;
                if (j >= 0 && j < kNbLeaves)
                    scan_leaf<kRefTies>(sm.pts + j * kChunk * 3, sm.mask[j], lf * kChunk, q, best, bcol, b2);
                else
                    scan_leaf<kRefTies>(m_pts + (long long)lf * kChunk * 3, ld_map<kCoherent>(m_mask + lf), lf * kChunk, q, best, bcol, b2);
                best_up = __double2float_ru(best);
            }
        }
        return;  // b2 lives in *best2_out
    }
    for (int sc = 0; sc < n_sup; ++sc) {
        const float4 slo = sup_in_smem ? sm.sbox[sc * 2] : ld_map<kCoherent>(m_sbox + sc * 2);
        const float4 shi = sup_in_smem ? sm.sbox[sc * 2 + 1] : ld_map<kCoherent>(m_sbox + sc * 2 + 1);
        if (box_lower_bound32(slo, shi, q32) > best_up) continue;
        const int l1 = min(n_leaf, (sc + 1) * kChunksPerSuper);
        if (row_in_smem) {
            // all leaf boxes of the row sit in shared memory: the sixteen lower bounds of a super block are
            // evaluated as independent chains, four at a time, into a bit mask -- instead of sixteen
            // dependent test-and-branch rounds -- and only the leaves that pass are visited (and re-tested
            // against the then-current best)
            const int l0 = sc * kChunksPerSuper;
            unsigned pass = 0;
#pragma unroll
            for (int g = 0; g < kChunksPerSuper; g += 4) {
                float lb[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int lf = min(l0 + g + i, n_leaf - 1);
                    lb[i] = box_lower_bound32(sm.rbox[lf * 2], sm.rbox[lf * 2 + 1], q32);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) pass |= (unsigned)!(lb[i] > best_up) << (g + i);
            }
            // drop the leaves visited above and those beyond the end of the row
            for (int d = -kNear; d <= kNear; ++d) {
                const int j = seed + d - l0;
                if (j >= 0 && j < kChunksPerSuper) pass &= ~(1u << j);
            }
            if (l1 - l0 < kChunksPerSuper) pass &= (1u << (l1 - l0)) - 1u;
            while (pass) {
                const int lf = l0 + __ffs(pass) - 1, j = lf - leaf0;
                pass &= pass - 1;
                if (box_lower_bound32(sm.rbox[lf * 2], sm.rbox[lf * 2 + 1], q32) > best_up) continue;
                if (j >= 0 && j < kNbLeaves)
                    scan_leaf<kRefTies>(sm.pts + j * kChunk * 3, sm.mask[j], lf * kChunk, q, best, bcol, b2);
                else
                    scan_leaf<kRefTies>(m_pts + (long long)lf * kChunk * 3, ld_map<kCoherent>(m_mask + lf), lf * kChunk, q, best, bcol, b2);
                best_up = __double2float_ru(best);
            }
            continue;
        }
        for (int lf = sc * kChunksPerSuper; lf < l1; ++lf) {
            if (lf >= seed - kNear && lf <= seed + kNear) continue;  // already visited
            const int j = lf - leaf0;
            const bool near_leaf = j >= 0 && j < kNbLeaves;
            const float4 blo = near_leaf ? sm.box[j * 2] : ld_map<kCoherent>(m_box + lf * 2);
            const float4 bhi = near_leaf ? sm.box[j * 2 + 1] : ld_map<kCoherent>(m_box + lf * 2 + 1);
            if (box_lower_bound32(blo, bhi, q32) > best_up) continue;
            if (near_leaf)
                scan_leaf<kRefTies>(sm.pts + j * kChunk * 3, sm.mask[j], lf * kChunk, q, best, bcol, b2);
            else
                scan_leaf<kRefTies>(m_pts + (long long)lf * kChunk * 3, ld_map<kCoherent>(m_mask + lf), lf * kChunk, q, best, bcol, b2);
            best_up = __double2float_ru(best);
        }
    }
}

// what the query of a thread found (the statistics dedupe of k_loop_step and k_frame_seq<kOut> starts from it)
struct TileQuery {
    int qc;                    // the query's column; -1 for a thread without a query
    int key;                   // the column of its nearest map point; -1 for none (empty map row)
    unsigned long long dbits;  // the bits of its nn_dist as stored (INFINITY when key is -1)
    P3 ori;                    // the query point in the global frame, xf_point(pose, p), before the shift
};

// The match of one (row, 256-column tile) once its labels are known and the cp.async group of the map neighbourhood
// has been waited for: nn_idx / nn_dist = -1 / -1.0 for the unlabelled columns; the labelled columns are compacted so
// that the search runs on densely populated warps; each query -- point_at(t) of its column-in-tile t, transformed
// with the pose pose_at() returns -- is searched in the row (search_row) and its nn_idx / nn_dist stored.  The pose
// is taken where it is used: a reference passed in from the caller kept its parameter offset in a per-thread
// register, and the pose reads of k_frame_match<fused labels, fused map> became per-thread constant loads (measured
// 2.7 % slower per-frame launches on a B200).  Called by all kTile threads
// (contains barriers).  Whole warps without a query skip the search; in the last warp with queries the spare lanes
// repeat its last query, so that the warp-cooperative part of the search always runs with 32 lanes (they store
// nothing).  kRefTies: every query whose smallest rounded distance is reached by at least two map points of the row
// is also appended to `ties`.
template <bool kCoherent, bool kRefTies, typename PointAt, typename PoseAt>
__device__ __forceinline__ TileQuery match_tile(const MapSmem &sm, const RowView &rv, int *s_warp, int *s_qcol,
                                                int label, PointAt point_at, PoseAt pose_at, const MatchOut &out,
                                                long long base, int row, int cols, int c0, const TieList &ties) {
    const int c = c0 + threadIdx.x;
    if (c < cols && label != 1) {
        out.nn_idx[base + c] = -1;
        out.nn_dist[base + c] = -1.0;
    }
    int nq;
    const int slot = block_excl_count_once(label == 1, s_warp, nq);  // its barrier also publishes a cp.async prefetch
    if (label == 1) s_qcol[slot] = threadIdx.x;
    __syncthreads();
    TileQuery m = {-1, -1, 0ull, {0, 0, 0}};
    if ((int)(threadIdx.x & ~31u) < nq) {
        const bool has_query = (int)threadIdx.x < nq;
        const int t = s_qcol[min((int)threadIdx.x, nq - 1)];  // column-in-tile handled by this thread
        const int qc = c0 + t;
        const PoseXf &pose = pose_at();
        const P3 ori = xf_point(pose, point_at(t));
        const P3 q = shift_point(pose, ori);
        double best, best2;
        int bcol;
        search_row<kCoherent, kRefTies>(sm, rv, qc, q, best, bcol, kFull, kRefTies ? &best2 : nullptr);
        if (kRefTies) {
            // tied: at least two map columns at the smallest rounded distance (exact duplicates included: they
            // resolve to the same answer).  The spare lanes repeat a query and append nothing; one atomic per warp.
            const bool tied = has_query && bcol >= 0 && __dsqrt_rn(best2) == __dsqrt_rn(best);
            const unsigned tm = __ballot_sync(kFull, tied);
            if (tm) {
                const unsigned lane = threadIdx.x & 31u;
                unsigned first = 0;
                if (lane == 0) first = atomicAdd(ties.count, (unsigned)__popc(tm));
                first = __shfl_sync(kFull, first, 0);
                if (tied) {
                    TieRec *r = ties.rec + first + __popc(tm & ((1u << lane) - 1u));
                    r->px = base + qc;
                    r->q[0] = q.x;
                    r->q[1] = q.y;
                    r->q[2] = q.z;
                }
            }
        }
        if (has_query) {
            const double dist = bcol >= 0 ? __dsqrt_rn(best) : INFINITY;
            out.nn_idx[base + qc] = bcol >= 0 ? row * cols + bcol : -1;
            out.nn_dist[base + qc] = dist;
            m.qc = qc;
            m.key = bcol;
            m.dbits = (unsigned long long)__double_as_longlong(dist);
            m.ori = ori;
        }
    }
    return m;
}

// grid as k_frame_map.  kFusedLabels: compute the labels of the tile here (and store them);
// otherwise read them from `labels`.  kFuseMap: also build the NEXT map (this frame transformed with
// its final pose) into map_next -- a second buffer, because neighbouring CTAs are still searching the
// current one -- which makes the whole front-end frame a single launch.
// kRefTies: the reference tie rule's variant -- every query whose smallest rounded distance is reached by at least
// two map points of the row is appended to `ties` (the host re-answers it with the reference's own search).
template <bool kFusedLabels, bool kFuseMap, bool kRefTies = false>
__global__ void __launch_bounds__(kTile, NAV_MATCH_MIN_CTAS)
k_frame_match(const double *__restrict__ cloud, int *__restrict__ labels, RowMap map, MatchOut out,
              const __grid_constant__ PoseBatch poses, int rows, int cols, int tiles_per_row,
              unsigned *__restrict__ n_exact, RowMap map_next, const __grid_constant__ PoseBatch final_poses,
              int pdl, TieList ties) {
    __shared__ StencilSmem s;
    // grid = (tiles per row, rows, sequences): no integer divisions to find the tile
    const int tile = blockIdx.x, row = blockIdx.y, seq = blockIdx.z;
    const int rid = seq * rows + row;
    const long long base = (long long)rid * cols;
    const int c0 = tile * kTile;
    const int c = c0 + threadIdx.x;

    __shared__ int s_warp[65];
    __shared__ int s_qcol[kTile];
    __shared__ MapSmem sm;
    const RowView rv = row_view(map, rid, base, tile);
    // asynchronous prefetch (cp.async) of the neighbourhood; consumed after the compaction
    auto prefetch_map = [&]() { prefetch_neighbourhood<false>(sm, rv, cols); };
    // Programmatic dependent launch (pdl != 0, kernel launched with the stream-serialisation attribute):
    // the next frame's launch may start while this one still runs.  Everything in front of
    // griddepcontrol.wait touches only this frame's own cloud (and shared memory); the previous frame's
    // map and every global store come after it, when the previous grid has completed and flushed.
    if (pdl) asm volatile("griddepcontrol.launch_dependents;");
    if (!pdl) prefetch_map();
    int label = 0;
    if (kFusedLabels) {
        tile_stage(s, cloud + base * 3, c0, cols);
        __syncthreads();
        label = tile_labels_filtered(s, c0, cols, n_exact);
    }
    if (pdl) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        prefetch_map();
    }
    if (kFusedLabels) {
        if (c < cols) labels[base + c] = label;
    } else {
        label = c < cols ? labels[base + c] : 0;
    }
    // the lidar-frame point of column-in-tile t
    auto point_at = [&](int t) {
        if (kFusedLabels) {
            const double *sp = s.pts + (t + kHalo) * 3;
            return P3{sp[0], sp[1], sp[2]};
        }
        return ldg_p3(cloud + (base + (c0 + t)) * 3);
    };
    if (kFuseMap) {  // a7 + a4/a5 for the next frame's search, into the other map buffer
        __shared__ float4 s_lo[kChunksPerSuper], s_hi[kChunksPerSuper];
        const P3 own = c < cols ? point_at(threadIdx.x) : P3{0, 0, 0};
        map_tile(label == 1, c < cols, own, final_poses.p[seq], map_next, rid, tile, c, base, s_lo, s_hi);
    }
    cp_async_wait_all();
    match_tile<false, kRefTies>(sm, rv, s_warp, s_qcol, label, point_at, [&]() -> const PoseXf & { return poses.p[seq]; }, out, base, row, cols, c0, ties);
}

__device__ __forceinline__ void cluster_arrive_all() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_all() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}

void launch_frame_map(const double *cloud, const int *labels, const RowMap &map, const PoseBatch &poses,
                      int n_seq, int rows, int cols, cudaStream_t stream) {
    const int tiles = div_up(cols, kTile);
    k_frame_map<<<n_seq * rows * tiles, kTile, 0, stream>>>(cloud, labels, map, poses, rows, cols, tiles);
}

template <bool kFusedLabels, bool kFuseMap, bool kRefTies = false>
static void launch_match_variant(int grid, cudaStream_t stream, bool pdl, const double *cloud, int *labels,
                                 const RowMap &map, const MatchOut &out, const PoseBatch &poses, int rows, int cols,
                                 int tiles, unsigned *n_exact, const RowMap &map_next, const PoseBatch &final_poses,
                                 const TieList &ties = TieList{nullptr, nullptr}) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)tiles, (unsigned)rows, (unsigned)(grid / (tiles * rows)));
    cfg.blockDim = dim3(kTile);
    cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, k_frame_match<kFusedLabels, kFuseMap, kRefTies>, cloud, labels, map, out, poses, rows, cols,
                       tiles, n_exact, map_next, final_poses, pdl ? 1 : 0, ties);
}

// pdl: launch with programmatic stream serialisation, so that consecutive frame launches on one stream
// overlap (the next frame's stencil phase runs under this frame's tail).  Safe next to any other work
// on the stream: only k_frame_match itself releases its dependents early, and only this kernel's
// cloud-reading phase runs in front of the dependency wait.
void launch_frame_match(const double *cloud, int *labels, bool fused_labels, const RowMap &map,
                        const MatchOut &out, const PoseBatch &poses, int n_seq, int rows, int cols,
                        unsigned *n_exact, cudaStream_t stream, const RowMap *map_next,
                        const PoseBatch *final_poses, bool pdl, const TieList *ties) {
    const int tiles = div_up(cols, kTile);
    const int grid = n_seq * rows * tiles;
    // programmatic serialisation only on ordinary streams (not the legacy / per-thread default streams)
    pdl = pdl && stream != nullptr && stream != cudaStreamLegacy && stream != cudaStreamPerThread;
    if (ties) {  // the reference tie rule: the two forms of the blocking calls (labels fused, map fused or not)
        if (map_next && final_poses)
            launch_match_variant<true, true, true>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                                   n_exact, *map_next, *final_poses, *ties);
        else
            launch_match_variant<true, false, true>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                                    n_exact, map, poses, *ties);
        return;
    }
    if (map_next && final_poses) {
        if (fused_labels)
            launch_match_variant<true, true>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                             n_exact, *map_next, *final_poses);
        else
            launch_match_variant<false, true>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                              n_exact, *map_next, *final_poses);
    } else {
        if (fused_labels)
            launch_match_variant<true, false>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                              n_exact, map, poses);
        else
            launch_match_variant<false, false>(grid, stream, pdl, cloud, labels, map, out, poses, rows, cols, tiles,
                                               n_exact, map, poses);
    }
}

constexpr int kRowThreads = 512;

// The fixed summation order of the fit totals: adds the five partial sums of `n_part` CTAs or rows
// (part[i*5 + k]) thread-strided with independent loads, then a shuffle tree, then warp by warp, and writes
// them to dst[0..4].  Called by all T = blockDim.x threads.  Every kernel that reports totals of the same
// partials uses this, so they are the same bits whichever kernel formed them.
template <int T>
__device__ __forceinline__ void sum_fit_partials(const double *__restrict__ part, int n_part, double (*s_tot)[5],
                                                 double *dst) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double t[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < n_part; i += T) {
        double v[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) v[k] = __ldcg(part + (long long)i * 5 + k);
#pragma unroll
        for (int k = 0; k < 5; ++k) t[k] = dadd(t[k], v[k]);
    }
#pragma unroll
    for (int k = 0; k < 5; ++k)
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) t[k] = dadd(t[k], __shfl_xor_sync(kFull, t[k], d));
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 5; ++k) s_tot[warp][k] = t[k];
    __syncthreads();
    if (threadIdx.x < 5) {
        double a = 0.0;
        for (int w = 0; w < T / 32; ++w) a = dadd(a, s_tot[w][threadIdx.x]);
        dst[threadIdx.x] = a;
    }
}

// Called by every thread of the CTA that finished last: adds the partials of all `n_part` CTAs
// (sum_fit_partials) and posts the totals followed by the sequence number to the host mailbox.  T = blockDim.x.
template <int T>
__device__ __forceinline__ void post_fit_totals(const double *__restrict__ part, int n_part, const FitMailbox &mail,
                                                double (*s_tot)[5]) {
    sum_fit_partials<T>(part, n_part, s_tot, mail.host);
    __syncthreads();
    if (threadIdx.x == 0) {
        // cumulative, by the thread that writes the flag: the five totals (ordered before it by the barrier)
        // reach the host before the sequence number does
        __threadfence_system();
        *mail.ticket = 0u;
        *(volatile unsigned long long *)(mail.host + 5) = mail.seq;
    }
}

// per-row dedupe, src/slam.c:247-283: one entry per matched map point; the query with the smallest
// distance wins (earliest column on equal distance, strict '>' at slam.c:264); entries in order of
// the first query that matched the point.  One CTA per (sequence,row); dynamic smem = 16 B * cols.
// row_stats != null: additionally reduce the sufficient statistics of the translation fit over the row's
// entries (SURVEY 8f #2; r = ori - nearest): row_stats[rid][0..4] = {n, sum rx, sum ry, sum rz, sum |r|^2},
// summed in a fixed order (thread-strided, then a shuffle tree, then warp by warp) -- deterministic, and
// the host adds the rows in order.  write_corr == 0 skips the 56-byte entries (the statistics are all
// the caller wants).
__global__ void __launch_bounds__(kRowThreads)
k_dedupe_rows(const double *__restrict__ cloud, const int *__restrict__ labels, RowMap map, MatchOut out,
              const __grid_constant__ PoseBatch poses, int rows, int cols, double *__restrict__ row_stats,
              int write_corr, FitMailbox mail) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    __shared__ int s_warp[65];
    __shared__ double s_red[kRowThreads / 32][4];
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    unsigned long long *s_best = (unsigned long long *)s_raw;
    int *s_first = (int *)(s_best + cols);
    int *s_win = s_first + cols;
    const int rid = blockIdx.x;
    const int seq = rid / rows, row = rid % rows;
    const long long base = (long long)rid * cols;
    const PoseXf &pose = poses.p[seq];
    for (int j = threadIdx.x; j < cols; j += kRowThreads) {
        s_best[j] = ~0ull;
        s_first[j] = INT_MAX;
        s_win[j] = INT_MAX;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cols; c += kRowThreads) {
        const int idx = out.nn_idx[base + c];
        if (labels[base + c] != 1 || idx < 0) continue;
        const int key = idx - row * cols;
        atomicMin(&s_best[key], (unsigned long long)__double_as_longlong(out.nn_dist[base + c]));
        atomicMin(&s_first[key], c);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cols; c += kRowThreads) {
        const int idx = out.nn_idx[base + c];
        if (labels[base + c] != 1 || idx < 0) continue;
        const int key = idx - row * cols;
        if ((unsigned long long)__double_as_longlong(out.nn_dist[base + c]) == s_best[key]) atomicMin(&s_win[key], c);
    }
    __syncthreads();
    int n_out = 0;
    nav_corr *rows_out = out.corr_rows + base;
    for (int c0 = 0; c0 < cols; c0 += kRowThreads) {
        const int c = c0 + threadIdx.x;
        int key = -1;
        bool is_first = false;
        if (c < cols && labels[base + c] == 1) {
            const int idx = out.nn_idx[base + c];
            if (idx >= 0) {
                key = idx - row * cols;
                is_first = s_first[key] == c;
            }
        }
        int total;
        const int pos = n_out + block_excl_count(is_first, s_warp, total);
        if (is_first) {
            const P3 ori = xf_point(pose, load_p3(cloud + (base + s_win[key]) * 3));
            const double *np = map.pts + (base + key) * 3;
            nav_corr e;
            e.ori.x = ori.x;
            e.ori.y = ori.y;
            e.ori.z = ori.z;
            e.nearest.x = np[0];
            e.nearest.y = np[1];
            e.nearest.z = np[2];
            e.distance = __longlong_as_double((long long)s_best[key]);
            if (write_corr) rows_out[pos] = e;
            if (row_stats) {
                const double rx = dsub(ori.x, np[0]), ry = dsub(ori.y, np[1]), rz = dsub(ori.z, np[2]);
                acc[0] = dadd(acc[0], rx);
                acc[1] = dadd(acc[1], ry);
                acc[2] = dadd(acc[2], rz);
                acc[3] = dadd(acc[3], dsq3(rx, ry, rz));
            }
        }
        n_out += total;
    }
    if (threadIdx.x == 0) out.corr_row_count[rid] = n_out;
    if (row_stats) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) acc[k] = dadd(acc[k], __shfl_xor_sync(kFull, acc[k], d));
        if (lane == 0)
#pragma unroll
            for (int k = 0; k < 4; ++k) s_red[warp][k] = acc[k];
        __syncthreads();
        if (threadIdx.x < 4) {
            double t = 0.0;
            for (int w = 0; w < kRowThreads / 32; ++w) t = dadd(t, s_red[w][threadIdx.x]);
            row_stats[(long long)rid * 5 + 1 + threadIdx.x] = t;
        }
        if (threadIdx.x == 0) row_stats[(long long)rid * 5] = (double)n_out;
        // mail.host != null (one sequence): the CTA that finishes last adds the rows in row order -- the same
        // sequential sums the host used to form from the downloaded rows, so the same bits -- and posts the five
        // totals followed by the call's sequence number into host-mapped memory: the host polls that word
        // instead of queueing a copy and synchronising the stream
        if (mail.host) {
            __shared__ bool s_last;
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) s_last = atomicAdd(mail.ticket, 1u) == gridDim.x - 1;
            __syncthreads();
            if (s_last) {
                __threadfence();
                __shared__ double s_tot[kRowThreads / 32][5];
                post_fit_totals<kRowThreads>(row_stats, (int)gridDim.x, mail, s_tot);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// The same dedupe when only the fit statistics are wanted (closed loop, nav_slam_localization_fast): the
// order of the entries does not matter, so a row is spread over its tiles -- one CTA per (row, 256-column
// tile), the CTAs of a row forming a thread-block CLUSTER.  Every CTA owns the "best distance" and
// "winning column" slots of the 256 map columns of its tile in its shared memory; queries post to the
// owner's slots through distributed shared memory (a query's neighbour is almost always in its own or the
// next tile), with cluster barriers between the three phases of src/slam.c:247-283: smallest distance per
// matched map point, earliest column among those, and the winners' residuals.  512 CTAs instead of 64, one
// column per thread: 23 us -> a few us per 64x2048 frame.
// Partial sums: per CTA in a fixed order (shuffle tree, then warp by warp); the CTA that finishes last adds
// the partials of the whole frame in a fixed order and posts the totals to the host mailbox.
// Phases 1-3 of the cluster dedupe.  Called by ALL threads of every CTA of the row's cluster (four cluster
// barriers inside).  key = matched map column of this thread's query (or -1), dbits = bits of its distance,
// c = the query's column.  Returns whether this query is the one kept for its map point.
// The slots are reached with shared::cluster addresses, and the smallest distance is posted with a 64-bit
// compare-and-swap loop.  The hardware has no 64-bit atomic min on shared memory: for atomicMin(u64) on a generic
// address the compiler falls back, for shared addresses, to an LDS + ATOMS compare-and-swap loop, and ATOMS
// only reaches the issuing CTA's own shared memory.  Posts to another CTA of the cluster through a `mapa.u64`
// pointer were lost that way, and rows whose matches crossed tiles kept wrong (and run-to-run varying) dedupe
// winners.  64-bit compare-and-swap and 32-bit min on distributed shared memory are single ATOM instructions.
__device__ __forceinline__ unsigned cluster_slot(const void *local, unsigned rank) {
    unsigned r;
    asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"((unsigned)__cvta_generic_to_shared(local)), "r"(rank));
    return r;
}

__device__ __forceinline__ bool cluster_dedupe_winner(unsigned long long *s_best, int *s_win, int key,
                                                      unsigned long long dbits, int c) {
    s_best[threadIdx.x] = ~0ull;
    s_win[threadIdx.x] = INT_MAX;
    unsigned r_best = 0, r_win = 0;
    if (key >= 0) {  // the slots of map column `key` live in the CTA of its tile (rank = tile index in the cluster)
        const unsigned owner = (unsigned)(key / kTile);
        r_best = cluster_slot(s_best + key % kTile, owner);
        r_win = cluster_slot(s_win + key % kTile, owner);
    }
    cluster_sync_all();  // every CTA of the row has initialised its slots
    if (key >= 0) {
        unsigned long long cur;
        asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(cur) : "r"(r_best) : "memory");
        while (dbits < cur) {
            unsigned long long seen;
            asm volatile("atom.shared::cluster.cas.b64 %0, [%1], %2, %3;"
                         : "=l"(seen) : "r"(r_best), "l"(cur), "l"(dbits) : "memory");
            if (seen == cur) break;
            cur = seen;
        }
    }
    cluster_sync_all();
    if (key >= 0) {
        unsigned long long best;
        asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(best) : "r"(r_best) : "memory");
        if (best == dbits) asm volatile("red.shared::cluster.min.s32 [%0], %1;" ::"r"(r_win), "r"(c) : "memory");
    }
    cluster_sync_all();
    int win = -1;
    if (key >= 0) asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(win) : "r"(r_win) : "memory");
    cluster_sync_all();  // nobody leaves (or reuses its slots) while a neighbour may still read them
    return key >= 0 && win == c;
}

struct StatsSmem {
    double red[kTile / 32][4];
    int cnt[kTile / 32];
    double tot[kTile / 32][5];
    bool last;
};

// CTA partial of the fit statistics (r = residual of a winner, zero otherwise) -> part[blockIdx.x][5]; the CTA
// that finishes last adds the partials of the whole frame and posts them.  Called by all kTile threads.
__device__ __forceinline__ void block_post_stats(StatsSmem &ss, bool winner, double rx, double ry, double rz,
                                                 double *__restrict__ part, const FitMailbox &mail) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc[4] = {rx, ry, rz, winner ? dsq3(rx, ry, rz) : 0.0};
    const int n_w = __popc(__ballot_sync(kFull, winner));
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) acc[k] = dadd(acc[k], __shfl_xor_sync(kFull, acc[k], d));
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) ss.red[warp][k] = acc[k];
        ss.cnt[warp] = n_w;
    }
    __syncthreads();
    double *mine = part + (long long)blockIdx.x * 5;
    if (threadIdx.x < 4) {
        double t = 0.0;
        for (int w = 0; w < kTile / 32; ++w) t = dadd(t, ss.red[w][threadIdx.x]);
        mine[1 + threadIdx.x] = t;
    } else if (threadIdx.x == 4) {
        int n = 0;
        for (int w = 0; w < kTile / 32; ++w) n += ss.cnt[w];
        mine[0] = (double)n;
    }
    if (!mail.host) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();  // cumulative: publishes the five stores above (ordered before it by the barrier)
        ss.last = atomicAdd(mail.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!ss.last) return;
    __threadfence();
    post_fit_totals<kTile>(part, (int)gridDim.x, mail, ss.tot);
}

// The statistics dedupe of a tile's search results (k_loop_step, k_frame_seq<kOut>): the winners of the cluster
// dedupe, their residuals ori - nearest back into COLUMN order (thread = column, as in k_dedupe_stats) so that the
// partial sums are formed in the same order and the totals are the same bits whichever kernel produced them, then
// block_post_stats.  ori_at(t): the winner's ori, t = its column in the tile.  Called by all kTile threads of every
// CTA of the row's cluster once the search is over; its point buffer sm.pts and the query list s_qcol are reused
// (the cluster barriers are CTA barriers too).
template <typename OriAt>
__device__ __forceinline__ void tile_fit_stats(const TileQuery &m, OriAt ori_at, const double *__restrict__ map_pts,
                                               long long base, int c0, MapSmem &sm, int *s_qcol,
                                               unsigned long long *s_best, int *s_win, StatsSmem &ss,
                                               double *__restrict__ part, const FitMailbox &mail) {
    const bool winner = cluster_dedupe_winner(s_best, s_win, m.key, m.dbits, m.qc);
    double *s_r = sm.pts;
    int *s_flag = s_qcol;
    s_flag[threadIdx.x] = 0;
    __syncthreads();
    if (winner) {
        const int t = m.qc - c0;
        const P3 ori = ori_at(t);
        const double *np = map_pts + (base + m.key) * 3;
        s_r[t * 3] = dsub(ori.x, np[0]);
        s_r[t * 3 + 1] = dsub(ori.y, np[1]);
        s_r[t * 3 + 2] = dsub(ori.z, np[2]);
        s_flag[t] = 1;
    }
    __syncthreads();
    const bool mine = s_flag[threadIdx.x] != 0;
    const double rx = mine ? s_r[threadIdx.x * 3] : 0.0, ry = mine ? s_r[threadIdx.x * 3 + 1] : 0.0,
                 rz = mine ? s_r[threadIdx.x * 3 + 2] : 0.0;
    block_post_stats(ss, mine, rx, ry, rz, part, mail);
}

__global__ void __launch_bounds__(kTile)
k_dedupe_stats(const double *__restrict__ cloud, const int *__restrict__ labels, RowMap map, MatchOut out,
               const __grid_constant__ PoseBatch poses, int rows, int cols, int tiles_per_row,
               double *__restrict__ part, FitMailbox mail) {
    __shared__ unsigned long long s_best[kTile];
    __shared__ int s_win[kTile];
    __shared__ StatsSmem ss;
    const int rid = blockIdx.x / tiles_per_row, tile = blockIdx.x % tiles_per_row;
    const int seq = rid / rows, row = rid % rows;
    const long long base = (long long)rid * cols;
    const int c = tile * kTile + threadIdx.x;
    int key = -1;
    unsigned long long dbits = 0;
    if (c < cols && labels[base + c] == 1) {
        const int idx = out.nn_idx[base + c];
        if (idx >= 0) {
            key = idx - row * cols;
            dbits = (unsigned long long)__double_as_longlong(out.nn_dist[base + c]);
        }
    }
    const bool winner = cluster_dedupe_winner(s_best, s_win, key, dbits, c);
    double rx = 0.0, ry = 0.0, rz = 0.0;
    if (winner) {
        const P3 ori = xf_point(poses.p[seq], load_p3(cloud + (base + c) * 3));
        const double *np = map.pts + (base + key) * 3;
        rx = dsub(ori.x, np[0]);
        ry = dsub(ori.y, np[1]);
        rz = dsub(ori.z, np[2]);
    }
    block_post_stats(ss, winner, rx, ry, rz, part, mail);
}

// ---------------------------------------------------------------------------------------------
// One launch per frame of the closed loop (nav_slam_run), one thread-block cluster per image row:
//   1. (do_map) the map of the PREVIOUS frame from its fitted pose (what k_frame_map does), in place --
//      a row's map is written and searched by the same cluster, a cluster barrier in between;
//   2. the match of this frame (labels already computed by the prefetch) exactly as k_frame_match;
//   3. the statistics dedupe of k_dedupe_stats on the results still in registers, and the mailbox post.
// The serial chain of a frame is then: fit -> this launch -> the host sees the totals.
//
// The pose source is a compile-time choice.  kDevLoop = false (nav_slam_run): the poses of this frame and of the
// previous one are kernel parameters (LoopPoses<false>), the labels were computed by the prefetch, and the last CTA
// posts the totals to the host mailbox.  kDevLoop = true (nav_slam_run_dev, frames resident in HBM): the poses are the
// device record of the sequence (LoopRec), which the previous launch's fit wrote; the tile's labels are computed here
// from the staged tile, as k_frame_seq does, and stored for the next launch's map; the tickets count per sequence, and
// the last CTA of a sequence adds that sequence's partials, runs the fit (fit_translation) and writes the frame's
// pose, error and totals and the next frame's record.  With do_match = 0 the launch only maps the previous frame.
#ifdef NAV_SEQ_TIMING
// developer instrumentation (profiles/prof_slam_run_dev.py): thread 0 of the last CTA of every sequence stamps
// %globaltimer before the partials are added, before the fit and after the outputs are written
__device__ unsigned long long *g_loop_stamps;  // [frames][n_seq][4]
extern "C" int nav_debug_set_loop_stamps(void *dev_ptr) {
    return (int)cudaMemcpyToSymbol(g_loop_stamps, &dev_ptr, sizeof(void *));
}
#define NAV_LOOP_STAMP(k)                                                                                         \
    do {                                                                                                          \
        if (threadIdx.x == 0 && g_loop_stamps) {                                                                  \
            unsigned long long t_;                                                                                \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                               \
            g_loop_stamps[((long long)ps.t * ps.n_seq + seq) * 4 + (k)] = t_;                                     \
        }                                                                                                         \
    } while (0)
#else
#define NAV_LOOP_STAMP(k)
#endif

// the fit's bias corrections 1 - beta1^t, 1 - beta2^t (upload_fit_tables: the host's pow() values)
__constant__ double c_fit_bias[2][kFitIters];

template <bool kDevLoop>
struct LoopPoses {
    PoseBatch cur, prev;  // this frame's query poses, the previous frame's map poses
};
template <>
struct LoopPoses<true> : DevLoop {};

// the fit tail of the device loop, by thread 0 of the last CTA of sequence `seq` once st = its totals:
// outputs of frame dl.t and the pose record of frame dl.t + 1
__device__ __forceinline__ void loop_fit_tail(const DevLoop &dl, int seq, const LoopRec &rec, const double *st) {
    const long long fs = (long long)dl.t * dl.n_seq + seq;
    const LoopTab &tb = dl.tab[fs];
    double tr[3] = {rec.loc.shift[0], rec.loc.shift[1], rec.loc.shift[2]};  // pred - last, as make_pose forms it
    double s[5];
#pragma unroll
    for (int k = 0; k < 5; ++k) s[k] = st[k];
    const double err = fit_translation(s, tr, c_fit_bias[0], c_fit_bias[1]);
    const double *last = rec.map.t;
    nav_pos p;
    p.x = last[0] + tr[0];
    p.y = last[1] + tr[1];
    p.z = last[2] + tr[2];
    p.roll = tb.rpy[0];
    p.pitch = tb.rpy[1];
    p.yaw = tb.rpy[2];
    dl.poses[fs] = p;
    if (dl.error) dl.error[fs] = err;
    if (dl.fit_stats)
#pragma unroll
        for (int k = 0; k < 5; ++k) dl.fit_stats[fs * 5 + k] = s[k];
    LoopRec &nx = dl.rec_out[seq];
    const double pt[3] = {p.x, p.y, p.z};
#pragma unroll
    for (int k = 0; k < 9; ++k) nx.map.R[k] = tb.Rm[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        nx.map.t[k] = pt[k];
        nx.map.shift[k] = 0.0;
    }
    if (dl.t + 1 < dl.n_frames) {  // pred = last + deltas[t+1] (nav_slam_run's prediction), shift = pred - last
        const LoopTab &tn = dl.tab[fs + dl.n_seq];
#pragma unroll
        for (int k = 0; k < 9; ++k) nx.loc.R[k] = tn.Rq[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            nx.loc.t[k] = pt[k] + tn.d[k];
            nx.loc.shift[k] = nx.loc.t[k] - pt[k];
        }
    }
}

// kKind (kDevLoop only, NAV_RUN_INPUT_*): depth and integer-mm frames are read raw, as k_frame_seq reads them -- this
// frame's tile staged with 4-byte cp.async and converted on read, the previous frame's column converted as it is
// loaded for its map; cloud / prev_cloud then point at int32.
template <bool kDevLoop, int kKind = kKindXyz>
__global__ void __launch_bounds__(kTile, NAV_MATCH_MIN_CTAS)
k_loop_step(const double *__restrict__ cloud, const int *__restrict__ labels, RowMap map, MatchOut out,
            const __grid_constant__ LoopPoses<kDevLoop> ps, int rows, int cols, int tiles_per_row,
            const double *__restrict__ prev_cloud, const int *__restrict__ prev_labels, int do_map,
            double *__restrict__ part, FitMailbox mail, TanTables tan) {
    static_assert(kDevLoop || kKind == kKindXyz, "the host loop converts its frames in the prefetch");
    constexpr bool kRaw = kKind != kKindXyz;
    constexpr int kE = kRawElems<kKind>;
    __shared__ __align__(16) int s_raw[kRawPts * kE];  // kRaw: this frame's tile, raw
    __shared__ double s_tan[kRawPts];                  // depth: the tans of the staged columns
    __shared__ int s_warp[65];
    __shared__ int s_qcol[kTile];
    __shared__ MapSmem sm;
    __shared__ unsigned long long s_best[kTile];
    __shared__ int s_win[kTile];
    __shared__ StatsSmem ss;
    // kDevLoop only: the sequence's pose record, the staged tile of this frame and the label filter's taps
    __shared__ LoopRec s_rec;
    __shared__ __align__(16) double s_pts[kTilePts * 3];
    __shared__ float s_f1[kTile + kHalo], s_f2[kTile + kHalo];
    __shared__ double s_st[5];
    const int rid = blockIdx.x / tiles_per_row;
    const int tile = blockIdx.x % tiles_per_row;
    const int seq = rid / rows, row = rid % rows;
    const long long base = (long long)rid * cols;
    const int c0 = tile * kTile;
    const int c = c0 + threadIdx.x;
    int label = 0;
    double tan_r = 0.0;
    if constexpr (kKind == kKindDepth) {
        stage_tan_cols(s_tan, tan.col, c0, cols);  // published by the barrier below
        tan_r = tan.row[row];
    }
    if constexpr (kDevLoop) {
        if (ps.do_match) {
            if constexpr (kRaw)
                raw_stage_async<kE>(s_raw, (const int *)cloud + base * kE, c0, cols);
            else
                tile_stage_async(s_pts, cloud + base * 3, c0, cols);
            cp_async_commit();
        }
        constexpr int kRecWords = (int)(sizeof(LoopRec) / sizeof(double));
        static_assert(kRecWords <= kTile, "one word of the record per thread");
        if ((int)threadIdx.x < kRecWords) ((double *)&s_rec)[threadIdx.x] = ((const double *)(ps.rec_in + seq))[threadIdx.x];
        __syncthreads();
    } else {
        label = c < cols ? labels[base + c] : 0;
    }
    if (do_map) {
        __shared__ float4 s_lo[kChunksPerSuper], s_hi[kChunksPerSuper];
        bool lab = false;
        P3 p = {0, 0, 0};
        if (c < cols) {
            lab = prev_labels[base + c] == 1;
            if constexpr (kKind == kKindDepth)
                p = depth_point(((const int *)prev_cloud)[base + c], s_tan[threadIdx.x + kRawLead], tan_r);
            else if constexpr (kKind == kKindMm)
                p = RawTile<kKindMm>{(const int *)prev_cloud + (base + c) * 3}.at(0);
            else
                p = load_p3(prev_cloud + (base + c) * 3);
        }
        if constexpr (kDevLoop)
            map_tile(lab, c < cols, p, s_rec.map, map, rid, tile, c, base, s_lo, s_hi);
        else
            map_tile(lab, c < cols, p, ps.prev.p[seq], map, rid, tile, c, base, s_lo, s_hi);
        if constexpr (kDevLoop) {
            if (!ps.do_match) return;  // the last frame's map: nothing reads it in this launch
        }
        // release / acquire: the row's new map is visible to all CTAs of its cluster.  The device loop computes the
        // tile's labels between the arrive and the wait (they need nothing from the other tiles).
        cluster_arrive_all();
    }
    if constexpr (kDevLoop) {
        cp_async_wait_all();
        __syncthreads();
        if constexpr (kRaw)
            label = tile_labels_filtered(raw_view<kKind>(s_raw, s_tan, tan_r), s_f1, s_f2, c0, cols, ps.n_exact);
        else
            label = tile_labels_filtered(s_pts, s_f1, s_f2, c0, cols, ps.n_exact);
        if (c < cols) ps.labels_out[base + c] = label;
    }
    if (do_map) cluster_wait_all();
    const RowView rv = row_view(map, rid, base, tile);
    prefetch_neighbourhood<true>(sm, rv, cols);
    cp_async_wait_all();
    auto point_at = [&](int t) {  // the lidar-frame point of column-in-tile t
        if constexpr (kRaw) {
            return raw_view<kKind>(s_raw, s_tan, tan_r).at(t + kHalo);
        } else if constexpr (kDevLoop) {
            const double *sp = s_pts + (t + kHalo) * 3;
            return P3{sp[0], sp[1], sp[2]};
        } else {
            return load_p3(cloud + (base + (c0 + t)) * 3);
        }
    };
    const TileQuery m = match_tile<true, false>(sm, rv, s_warp, s_qcol, label, point_at,
                                                [&]() -> const PoseXf & {
                                                    if constexpr (kDevLoop)
                                                        return s_rec.loc;
                                                    else
                                                        return ps.cur.p[seq];
                                                },
                                                out, base, row, cols, c0, TieList{nullptr, nullptr});
    tile_fit_stats(m, [&](int) { return m.ori; }, map.pts, base, c0, sm, s_qcol, s_best, s_win, ss, part, mail);
    if constexpr (kDevLoop) {
        // the per-sequence ticket (block_post_stats without a mailbox has written this CTA's partial)
        const unsigned n_cta = (unsigned)(rows * tiles_per_row);
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();  // cumulative: publishes the partial (ordered before it by the barrier)
            ss.last = atomicAdd(ps.ticket + seq, 1u) == n_cta - 1;
        }
        __syncthreads();
        if (!ss.last) return;
        __threadfence();
        NAV_LOOP_STAMP(0);
        // the sequence's rows*tiles partials in the order k_seq_fit_totals and the mailbox post use
        sum_fit_partials<kTile>(part + (long long)seq * n_cta * 5, (int)n_cta, ss.tot, s_st);
        __syncthreads();
        if (threadIdx.x == 0) {
            NAV_LOOP_STAMP(1);
            loop_fit_tail(ps, seq, s_rec, s_st);
            ps.ticket[seq] = 0u;
            NAV_LOOP_STAMP(2);
        }
    }
}

bool row_cluster_supported(int cols) { return div_up(cols, kTile) <= 8; }  // portable cluster size

// a launch of kTile-thread CTAs in which the `tiles` CTAs of an image row form one thread-block cluster
template <typename... Params, typename... Args>
static int launch_row_clusters(void (*kernel)(Params...), dim3 grid, int tiles, cudaStream_t stream, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(kTile);
    cfg.stream = stream;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = (unsigned)tiles;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    return (int)cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// f(std::integral_constant<int, K>) for the frame kind K == kind (NAV_RUN_INPUT_*), and f(std::bool_constant<b>):
// a run-time choice turned into the template argument of a kernel
template <typename F>
static int with_kind(int kind, F &&f) {
    if (kind == kKindDepth) return f(std::integral_constant<int, kKindDepth>{});
    if (kind == kKindMm) return f(std::integral_constant<int, kKindMm>{});
    return f(std::integral_constant<int, kKindXyz>{});
}
template <typename F>
static int with_flag(bool b, F &&f) {
    return b ? f(std::true_type{}) : f(std::false_type{});
}

int launch_dedupe_stats(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                        const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream, double *part,
                        const FitMailbox &mail) {
    const int tiles = div_up(cols, kTile);
    return launch_row_clusters(k_dedupe_stats, dim3((unsigned)(n_seq * rows * tiles)), tiles, stream, cloud, labels, map,
                               out, poses, rows, cols, tiles, part, mail);
}

int launch_loop_step(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                     const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream,
                     const double *prev_cloud, const int *prev_labels, const PoseBatch &prev_poses, bool do_map,
                     double *part, const FitMailbox &mail) {
    const int tiles = div_up(cols, kTile);
    LoopPoses<false> ps;
    ps.cur = poses;
    ps.prev = prev_poses;
    const TanTables no_tan = {nullptr, nullptr};
    return launch_row_clusters(k_loop_step<false>, dim3((unsigned)(n_seq * rows * tiles)), tiles, stream, cloud, labels,
                               map, out, ps, rows, cols, tiles, prev_cloud, prev_labels, do_map ? 1 : 0, part, mail,
                               no_tan);
}

int launch_loop_step_dev(int kind, const DevLoop &dl, const void *cloud, const void *prev_cloud, const int *prev_labels,
                         bool do_map, const RowMap &map, const MatchOut &out, int n_seq, int rows, int cols,
                         double *part, cudaStream_t stream, const TanTables &tan) {
    const int tiles = div_up(cols, kTile);
    LoopPoses<true> ps;
    static_cast<DevLoop &>(ps) = dl;
    const FitMailbox no_mail = {nullptr, nullptr, 0ull};
    return with_kind(kind, [&](auto k) {
        return launch_row_clusters(k_loop_step<true, k>, dim3((unsigned)(n_seq * rows * tiles)), tiles, stream,
                                   (const double *)cloud, (const int *)nullptr, map, out, ps, rows, cols, tiles,
                                   (const double *)prev_cloud, prev_labels, do_map ? 1 : 0, part, no_mail, tan);
    });
}

// queued on `stream`, in front of the kernels that read the tables; c1 / c2 must stay valid (the host's static tables).
// A second upload by another context rewrites the same values, so it never changes what a running kernel reads.
int upload_fit_tables(const double *c1, const double *c2, cudaStream_t stream) {
    const size_t bytes = kFitIters * sizeof(double);
    cudaError_t e = cudaMemcpyToSymbolAsync(c_fit_bias, c1, bytes, 0, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(c_fit_bias, c2, bytes, bytes, cudaMemcpyHostToDevice, stream);
    return (int)e;
}

// fit_translation on n stat vectors, one thread each: the pose last + (pred - last) with the fitted translation, as
// nav_slam_fit_from_stats forms it
__global__ void k_fit_debug(const double *__restrict__ stats, const nav_pos *__restrict__ pred,
                            const nav_pos *__restrict__ last, size_t n, nav_pos *__restrict__ pose_out,
                            double *__restrict__ err_out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const nav_pos a = pred[i], b = last[i];
    double st[5];
    for (int k = 0; k < 5; ++k) st[k] = stats[i * 5 + k];
    double t[6] = {a.x - b.x, a.y - b.y, a.z - b.z, a.roll - b.roll, a.pitch - b.pitch, a.yaw - b.yaw};
    const double err = fit_translation(st, t, c_fit_bias[0], c_fit_bias[1]);
    nav_pos p;
    p.x = b.x + t[0];
    p.y = b.y + t[1];
    p.z = b.z + t[2];
    p.roll = b.roll + t[3];
    p.pitch = b.pitch + t[4];
    p.yaw = b.yaw + t[5];
    pose_out[i] = p;
    if (err_out) err_out[i] = err;
}

void launch_fit_debug(const double *stats, const nav_pos *pred, const nav_pos *last, size_t n, nav_pos *pose_out,
                      double *err_out, cudaStream_t stream) {
    if (n == 0) return;
    k_fit_debug<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(stats, pred, last, n, pose_out, err_out);
}

// ---------------------------------------------------------------------------------------------
// A whole SEQUENCE of frames with known poses in ONE launch (nav_frontend_sequence_dev).  Frame t+1 of an image
// row only depends on the map the eight tiles of the SAME row built from frame t, so the CTAs of a row form a
// thread-block cluster that walks through the frames on its own, with a cluster barrier per frame where
// separate launches had a grid-wide dependency: no launch latency between frames, and rows that are ahead are
// not held back by rows that are behind.  Per frame the body is that of k_frame_match<fused labels, fused map>:
// labels (a3), query transform (a7), exact search of the row map of the previous frame (a6), the next map from
// the frame's final pose into the other map buffer (a7, a4/a5).  labels / nn_idx / nn_dist hold the results of
// the last frame, as after the same number of separate launches.
// kOut (nav_frontend_sequence_out_dev): every frame also stores its label masks, nn_idx and nn_dist into slot f of
// the caller's rings (SeqOut), and -- when o.part is set -- runs the statistics dedupe of k_loop_step on the search
// results still in registers, writing the CTA partials of frame f to o.part (k_seq_fit_totals adds them up).  The
// four cluster barriers of the dedupe sit between the frame's cluster wait and its arrive, so arrive and wait
// still alternate; the dedupe reads the map the frame searched, which frame f+1 overwrites only after its
// cluster wait, i.e. after every CTA of the row has finished its dedupe.
#ifdef NAV_SEQ_TIMING
// developer instrumentation (profiles/prof_seq_phases.py; build rowmap.cu with -DNAV_SEQ_TIMING): thread 0 of every
// CTA stamps %globaltimer at seven points of every frame of k_frame_seq
__device__ unsigned long long *g_seq_stamps;   // [frames][ctas][8]
#define NAV_STAMP(k)                                                                                              \
    do {                                                                                                          \
        if (threadIdx.x == 0 && g_seq_stamps) {                                                                   \
            unsigned long long t_;                                                                                \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                               \
            const int cta_ = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;                      \
            g_seq_stamps[((long long)f * gridDim.x * gridDim.y * gridDim.z + cta_) * 8 + (k)] = t_;               \
        }                                                                                                         \
    } while (0)
extern "C" int nav_debug_set_seq_stamps(void *dev_ptr) {
    return (int)cudaMemcpyToSymbol(g_seq_stamps, &dev_ptr, sizeof(void *));
}
#else
#define NAV_STAMP(k)
#endif

constexpr int kSeqInlineFrames = 64;
struct SeqArgs {
    const double *frames;     // [n_frames][n_seq*rows][cols][3]
    long long frame_stride;   // doubles between consecutive frames
    int n_frames, n_seq;
    const PoseXf *pose_loc;   // [n_frames][n_seq] predicted pose + shift (queries)
    const PoseXf *pose_fin;   // [n_frames][n_seq] final pose (map)
};
// poses of a short sequence travel as kernel parameters (CUDA 12.1+: up to 32 764 bytes): no upload to queue
// in front of the launch, no staging buffer to guard
struct SeqInlinePoses {
    PoseXf loc[kSeqInlineFrames], fin[kSeqInlineFrames];
};
static_assert(sizeof(SeqInlinePoses) + 256 < 32764, "inline poses must fit the kernel parameter space");

// kBulk (frame_seq_bulk_ok): the frame's tile and the map neighbourhood arrive by bulk copies, one thread issues
// them and every thread waits on an mbarrier -- s_bar[slot] for the tile in that slot, s_bar[2] for the
// neighbourhood.  Otherwise every thread issues its share of 8- and 16-byte cp.async and waits for its own groups,
// and a CTA barrier publishes them.
// kKind (NAV_RUN_INPUT_*): xyz frames are staged as doubles; depth and integer-mm frames are staged raw, 4 or 12 B per
// point, into s_raw and converted where they are read (RawTile: depth_point / mm_coord, the arithmetic of k_convert and
// k_widen_mm) -- no conversion pass, so no CTA barrier is added per frame.  a.frames / a.frame_stride then count int32.
template <bool kInline, bool kOut, bool kBulk, int kKind = kKindXyz>
__global__ void __launch_bounds__(kTile, NAV_MATCH_MIN_CTAS)
k_frame_seq(SeqArgs a, int *__restrict__ labels, RowMap map0, RowMap map1, MatchOut out, int rows, int cols,
            unsigned *__restrict__ n_exact, const __grid_constant__ SeqInlinePoses ip, SeqOut o, TanTables tan) {
    constexpr bool kRaw = kKind != kKindXyz;
    constexpr int kE = kRawElems<kKind>;
    __shared__ __align__(16) double s_pts[2][kTilePts * 3];  // the tile of this frame / of the next one (in flight)
    __shared__ __align__(16) int s_raw[2][kRawPts * kE];     // kRaw: the same, raw
    __shared__ double s_tan[kRawPts];                        // depth: the tans of the staged columns
    __shared__ float s_f1[kTile + kHalo], s_f2[kTile + kHalo];
    __shared__ int s_warp[65];
    __shared__ int s_qcol[kTile];
    __shared__ MapSmem sm;
    __shared__ float4 s_lo[kChunksPerSuper], s_hi[kChunksPerSuper];
    const int tile = blockIdx.x, row = blockIdx.y, seq = blockIdx.z;
    const int rid = seq * rows + row;
    const long long base = (long long)rid * cols;
    const int c0 = tile * kTile;
    const int c = c0 + threadIdx.x;
    // ring slots: per frame n_seq*rows rows of cols pixels / n_chunks mask words / `tiles` CTA partials
    const long long px_frame = (long long)a.n_seq * rows * cols, cta_frame = (long long)a.n_seq * rows * gridDim.x;
    __shared__ __align__(8) unsigned long long s_bar[3];
    // kRaw: the frames as int32, the tile of slot `slot` as points, and where frame f's row starts
    const int *raw_frames = (const int *)a.frames;
    double tan_r = 0.0;
    if constexpr (kKind == kKindDepth) {
        stage_tan_cols(s_tan, tan.col, c0, cols);  // published by the barrier in front of the first labels
        tan_r = tan.row[row];
    }
    auto raw_tile = [&](auto slot) { return raw_view<kKind>(s_raw[slot], s_tan, tan_r); };  // kRaw only
    auto raw_row = [&](int f) { return raw_frames + (long long)f * a.frame_stride + base * kE; };
    if constexpr (kBulk) {
        // the copies only ever write the slots of columns inside the row and the mask words of leaves inside it;
        // the rest reads as zero, as the cp.async path leaves it
        if constexpr (kRaw) {
            for (int i = threadIdx.x; i < kRawPts * kE; i += kTile) {
                const int col = c0 - kRawLead + i / kE;
                if (col < 0 || col >= cols) s_raw[0][i] = s_raw[1][i] = 0;
            }
        } else {
            for (int i = threadIdx.x; i < kTilePts * 3; i += kTile) {
                const int col = c0 - kHalo + i / 3;
                if (col < 0 || col >= cols) s_pts[0][i] = s_pts[1][i] = 0.0;
            }
        }
        if (threadIdx.x < 3) sm.mask_lead[threadIdx.x] = 0u;
        if (threadIdx.x < kNbLeaves + 3) sm.mask[threadIdx.x] = 0u;
        if (threadIdx.x == 0) {
            for (int i = 0; i < 3; ++i) mbar_init(&s_bar[i], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the zeros above before the copies
            if constexpr (kRaw)
                raw_stage_bulk<kE>(s_raw[0], raw_row(0), c0, cols, &s_bar[0]);
            else
                tile_stage_bulk(s_pts[0], a.frames + base * 3, c0, cols, &s_bar[0]);
        }
    } else {
        if constexpr (kRaw)
            raw_stage_async<kE>(s_raw[0], raw_row(0), c0, cols);
        else
            tile_stage_async(s_pts[0], a.frames + base * 3, c0, cols);
        cp_async_commit();
    }
    for (int f = 0; f < a.n_frames; ++f) {
        NAV_STAMP(0);
        const double *pts = s_pts[f & 1];
        const RowMap &map = (f & 1) ? map1 : map0;
        const RowMap &map_next = (f & 1) ? map0 : map1;
        const RowView rv = row_view(map, rid, base, tile);
        // this frame's tile has landed
        if constexpr (kBulk) {
            mbar_wait(&s_bar[f & 1], (unsigned)(f >> 1) & 1u);  // phase f / 2 of its slot's barrier
        } else {
            cp_async_wait_group<0>();
            __syncthreads();
        }
        NAV_STAMP(1);
        // the labels need nothing from the row's other tiles: they are computed BEFORE waiting for the cluster
        // (the barrier was only signalled at the end of the previous frame), which turns the wait for the row's
        // slowest tile into useful time
        int label;
        if constexpr (kRaw)
            label = tile_labels_filtered(raw_tile(f & 1), s_f1, s_f2, c0, cols, n_exact);
        else
            label = tile_labels_filtered(pts, s_f1, s_f2, c0, cols, n_exact);
        // the next frame's tile starts its way from HBM now and has the whole search to arrive.  Its slot was last
        // read in frame f-1; the barrier that ends the labels is behind those reads (cp.async path: the cluster wait).
        // Nothing but generic reads touched the slot since its last copy, so the refill needs no proxy fence.
        if constexpr (kBulk) {
            if (threadIdx.x == 0 && f + 1 < a.n_frames) {
                if constexpr (kRaw)
                    raw_stage_bulk<kE>(s_raw[(f + 1) & 1], raw_row(f + 1), c0, cols, &s_bar[(f + 1) & 1]);
                else
                    tile_stage_bulk(s_pts[(f + 1) & 1], a.frames + (long long)(f + 1) * a.frame_stride + base * 3, c0,
                                    cols, &s_bar[(f + 1) & 1]);
            }
        }
        NAV_STAMP(2);
        if (f > 0) cluster_wait_all();  // the row's map of the previous frame is complete (also a CTA barrier)
        NAV_STAMP(3);
        if constexpr (kBulk) {
            if (threadIdx.x == 0) {
                // The row's map was written by the CTAs of the cluster with generic stores, ordered before this
                // thread by the release / acquire of the cluster barrier; the async proxy of the copies below is
                // ordered behind it by this thread's proxy fence, which is enough as the copies are issued by this
                // thread after the fence.  (Frame 0 reads a map of an earlier launch.)  The same for shared memory:
                // the generic reads and writes of sm (search, statistics dedupe) precede the CTA barrier above, the
                // async writes of the copies follow the fence.
                asm volatile("fence.proxy.async.global;" ::: "memory");
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                stage_neighbourhood_bulk(sm, rv, cols, &s_bar[2]);
            }
        } else {
            prefetch_neighbourhood<true>(sm, rv, cols);
            cp_async_commit();
            if (f + 1 < a.n_frames) {
                if constexpr (kRaw)
                    raw_stage_async<kE>(s_raw[(f + 1) & 1], raw_row(f + 1), c0, cols);
                else
                    tile_stage_async(s_pts[(f + 1) & 1], a.frames + (long long)(f + 1) * a.frame_stride + base * 3, c0,
                                     cols);
            }
            cp_async_commit();
        }
        if (c < cols) {
            labels[base + c] = label;
            if (kOut && label != 1) {
                if (o.nn_idx) o.nn_idx[f * px_frame + base + c] = -1;
                if (o.nn_dist) o.nn_dist[f * px_frame + base + c] = -1.0;
            }
        }
        const PoseXf &pose = kInline ? ip.loc[f] : a.pose_loc[(long long)f * a.n_seq + seq];
        auto point_at = [&](int t) {  // the lidar-frame point of column-in-tile t
            if constexpr (kRaw) {
                return raw_tile(f & 1).at(t + kHalo);
            } else {
                const double *sp = pts + (t + kHalo) * 3;
                return P3{sp[0], sp[1], sp[2]};
            }
        };
        {
            const P3 own = c < cols ? point_at(threadIdx.x) : P3{0, 0, 0};
            unsigned *mask_out = nullptr;
            if (kOut && o.mask) mask_out = o.mask + f * (long long)a.n_seq * rows * map_next.n_chunks;
            map_tile(label == 1, c < cols, own, kInline ? ip.fin[f] : a.pose_fin[(long long)f * a.n_seq + seq], map_next, rid,
                     tile, c, base, s_lo, s_hi, mask_out);
        }
        NAV_STAMP(4);
        // the neighbourhood of the map; the next tile may still be in flight
        if constexpr (kBulk)
            mbar_wait(&s_bar[2], (unsigned)f & 1u);
        else
            cp_async_wait_group<1>();
        NAV_STAMP(5);
        const TileQuery m = match_tile<true, false>(sm, rv, s_warp, s_qcol, label, point_at, [&]() -> const PoseXf & { return pose; }, out, base, row, cols,
                                                    c0, TieList{nullptr, nullptr});
        if (kOut && m.qc >= 0) {
            if (o.nn_idx) o.nn_idx[f * px_frame + base + m.qc] = m.key >= 0 ? row * cols + m.key : -1;
            if (o.nn_dist) o.nn_dist[f * px_frame + base + m.qc] = __longlong_as_double((long long)m.dbits);
        }
        if (kOut && o.part) {  // uniform over the grid: every CTA of the cluster takes it
            __shared__ unsigned long long s_best[kTile];
            __shared__ int s_win[kTile];
            __shared__ StatsSmem ss;
            // part + (rid * tiles + tile) * 5: the CTA order of k_dedupe_stats.  The winner's ori is transformed
            // again from the tile, the same bits as during the search.
            const FitMailbox no_mail = {nullptr, nullptr, 0ull};
            tile_fit_stats(m, [&](int t) { return xf_point(pose, point_at(t)); }, map.pts, base, c0, sm, s_qcol, s_best,
                           s_win, ss, o.part + (f * cta_frame + (long long)rid * gridDim.x) * 5, no_mail);
        }
        // this CTA's part of the row's next map is written and it no longer reads the current one: signal the
        // cluster (release) and go on; the matching wait sits in front of the next frame's map prefetch
        NAV_STAMP(6);
        cluster_arrive_all();
    }
    cluster_wait_all();  // every arrive has its wait
}

int frame_seq_inline_frames() { return kSeqInlineFrames; }

// Whether k_frame_seq can stage with bulk copies (kBulk): every range it copies must start on a 16-byte boundary and
// be a multiple of 16 bytes long.  xyz: rows of an even number of columns up to 2048 whose mask rows are a multiple of
// four words -- 64x2048 and every width that is a multiple of 64 -- take the bulk path; odd widths (e.g. 257) and
// even ones with a ragged mask row (e.g. 1800: 113 words) keep the cp.async path.  Depth and integer-mm frames (raw
// spans of whole groups of four columns): rows of a multiple of four columns, frames and frame stride on 16 bytes, and
// the same mask-row and map conditions; any other shape stages with 4-byte cp.async.
static bool frame_seq_bulk_ok(int kind, const void *frames, long long frame_stride, const RowMap &m0, const RowMap &m1,
                              int cols) {
    auto al16 = [](const void *p) { return ((uintptr_t)p & 15u) == 0; };
    auto map_ok = [&](const RowMap &m) { return al16(m.pts) && al16(m.mask) && al16(m.box) && al16(m.sbox); };
    const bool maps = cols <= kMaxRowLeafSmem * kChunk && div_up(cols, kChunk) % 4 == 0 && al16(frames) && map_ok(m0) &&
                      map_ok(m1);
    if (kind == kKindXyz) return cols % 2 == 0 && frame_stride % 2 == 0 && maps;
    return cols % 4 == 0 && frame_stride % 4 == 0 && maps;
}

// h_pose_loc / h_pose_fin != null (n_seq == 1, n_frames <= frame_seq_inline_frames()): the poses are passed as
// kernel parameters and the device arrays are not read.  seq_out != null: the output mode of k_frame_seq.
int launch_frame_seq(int kind, const void *frames, long long frame_stride, int n_frames, int *labels, const RowMap &map0,
                     const RowMap &map1, const MatchOut &out, const PoseXf *d_pose_loc, const PoseXf *d_pose_fin,
                     int n_seq, int rows, int cols, unsigned *n_exact, cudaStream_t stream, const PoseXf *h_pose_loc,
                     const PoseXf *h_pose_fin, const SeqOut *seq_out, bool *bulk_out, const TanTables &tan) {
    const bool bulk = frame_seq_bulk_ok(kind, frames, frame_stride, map0, map1, cols);
    if (bulk_out) *bulk_out = bulk;
    const int tiles = div_up(cols, kTile);
    const SeqArgs a = {(const double *)frames, frame_stride, n_frames, n_seq, d_pose_loc, d_pose_fin};
    const bool inl = h_pose_loc && h_pose_fin && n_seq == 1 && n_frames <= kSeqInlineFrames;
    const dim3 grid((unsigned)tiles, (unsigned)rows, (unsigned)n_seq);
    const SeqOut no_out = {nullptr, nullptr, nullptr, nullptr};
    static const SeqInlinePoses none = {};
    SeqInlinePoses ip;  // the launch copies its parameters at the call
    if (inl) {
        for (int f = 0; f < n_frames; ++f) {
            ip.loc[f] = h_pose_loc[f];
            ip.fin[f] = h_pose_fin[f];
        }
        for (int f = n_frames; f < kSeqInlineFrames; ++f) ip.loc[f] = ip.fin[f] = h_pose_loc[0];
    }
    return with_kind(kind, [&](auto k) {
        return with_flag(bulk, [&](auto b) {
            return with_flag(inl, [&](auto i) {
                return with_flag(seq_out != nullptr, [&](auto o) {
                    return launch_row_clusters(k_frame_seq<i, o, b, k>, grid, tiles, stream, a, labels, map0, map1, out,
                                               rows, cols, n_exact, inl ? ip : none, seq_out ? *seq_out : no_out, tan);
                });
            });
        });
    });
}

// Fit totals of frame blockIdx.x, sequence blockIdx.y: part = [n_frames][n_seq][n_part][5] partials, stats =
// [n_frames][n_seq][5].  T = kTile adds the tile partials of k_frame_seq / k_dedupe_stats, T = kRowThreads the row
// totals of k_dedupe_rows -- each in the order the closed loop's post uses for them (sum_fit_partials<T>).
template <int T>
__global__ void __launch_bounds__(T) k_seq_fit_totals(const double *__restrict__ part, int n_part, double *stats) {
    __shared__ double s_tot[T / 32][5];
    const long long fs = (long long)blockIdx.x * gridDim.y + blockIdx.y;
    sum_fit_partials<T>(part + fs * n_part * 5, n_part, s_tot, stats + fs * 5);
}

void launch_seq_fit_totals(const double *part, bool row_partials, int n_part, int n_frames, int n_seq, double *stats,
                           cudaStream_t stream) {
    const dim3 grid((unsigned)n_frames, (unsigned)n_seq);
    if (row_partials)
        k_seq_fit_totals<kRowThreads><<<grid, kRowThreads, 0, stream>>>(part, n_part, stats);
    else
        k_seq_fit_totals<kTile><<<grid, kTile, 0, stream>>>(part, n_part, stats);
}

size_t dedupe_smem_bytes(int cols) { return (size_t)cols * 16; }

int configure_row_kernels(int cols) {
    static int configured[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    const int need = (int)dedupe_smem_bytes(cols);
    if (need <= 48 * 1024 || (dev >= 0 && dev < 64 && configured[dev] >= need)) return 0;
    cudaError_t e = cudaFuncSetAttribute(k_dedupe_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, need);
    if (e == cudaSuccess && dev >= 0 && dev < 64) configured[dev] = need;
    return (int)e;
}

void launch_dedupe(const double *cloud, const int *labels, const RowMap &map, const MatchOut &out,
                   const PoseBatch &poses, int n_seq, int rows, int cols, cudaStream_t stream, double *row_stats,
                   bool write_corr, const FitMailbox *mail) {
    FitMailbox mb = {nullptr, nullptr, 0ull};
    if (mail && row_stats && n_seq == 1) mb = *mail;
    k_dedupe_rows<<<n_seq * rows, kRowThreads, dedupe_smem_bytes(cols), stream>>>(
        cloud, labels, map, out, poses, rows, cols, row_stats, write_corr ? 1 : 0, mb);
}

// rows of one sequence back to back: corr_out[seq][offset(row) + i]
__global__ void k_gather_corr(const nav_corr *__restrict__ corr_rows, const int *__restrict__ row_count,
                              nav_corr *__restrict__ corr_out, int *__restrict__ corr_total, int rows, int cols) {
    __shared__ int s_off;
    const int rid = blockIdx.x;
    const int seq = rid / rows, row = rid % rows;
    if (threadIdx.x == 0) {
        int off = 0;
        for (int r = 0; r < row; ++r) off += row_count[seq * rows + r];
        s_off = off;
        if (row == rows - 1) corr_total[seq] = off + row_count[rid];
    }
    __syncthreads();
    const int n = row_count[rid];
    const double *src = (const double *)(corr_rows + (long long)rid * cols);
    double *dst = (double *)(corr_out + (long long)seq * rows * cols + s_off);
    for (int i = threadIdx.x; i < n * 7; i += blockDim.x) dst[i] = src[i];
}

__global__ void k_apply_tie_fix(const int2 *__restrict__ fix, int n, int *__restrict__ nn_idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) nn_idx[fix[i].x] = fix[i].y;
}

void launch_apply_tie_fix(const int2 *fix, int n, int *nn_idx, cudaStream_t stream) {
    k_apply_tie_fix<<<div_up(n, 256), 256, 0, stream>>>(fix, n, nn_idx);
}

void launch_gather_corr(const nav_corr *corr_rows, const int *corr_row_count, nav_corr *corr_out,
                        int *corr_total, int n_seq, int rows, int cols, cudaStream_t stream) {
    k_gather_corr<<<n_seq * rows, 256, 0, stream>>>(corr_rows, corr_row_count, corr_out, corr_total, rows, cols);
}

// ---------------------------------------------------------------------------------------------
// flattenPoints (src/slam.c:64-72): stable compaction of one row where feature == 1 (function-level
// mirror), or where the map's label mask is set (k_export_row: the flattenedPoints array the
// reference would hand to buildKDTree, src/slam.c:170-171)
__global__ void __launch_bounds__(kRowThreads)
k_flatten_row(const double *__restrict__ row_pts, const int *__restrict__ row_feature,
              const unsigned *__restrict__ row_mask, double *__restrict__ out, int *__restrict__ col_out,
              int *__restrict__ count, int cols) {
    __shared__ int s_warp[65];
    int carry = 0;
    for (int c0 = 0; c0 < cols; c0 += kRowThreads) {
        const int c = c0 + threadIdx.x;
        bool lab = false;
        if (c < cols) lab = row_feature ? row_feature[c] == 1 : ((row_mask[c / kChunk] >> (c % kChunk)) & 1u) != 0;
        int total;
        const int pos = carry + block_excl_count(lab, s_warp, total);
        if (lab) {
            store_p3(out + (long long)pos * 3, load_p3(row_pts + (long long)c * 3));
            if (col_out) col_out[pos] = c;
        }
        carry += total;
    }
    if (threadIdx.x == 0) *count = carry;
}

void launch_flatten_row(const double *row_pts, const int *row_feature, const unsigned *row_mask, double *out,
                        int *col_out, int *count, int cols, cudaStream_t stream) {
    k_flatten_row<<<1, kRowThreads, 0, stream>>>(row_pts, row_feature, row_mask, out, col_out, count, cols);
}

}  // namespace nav
