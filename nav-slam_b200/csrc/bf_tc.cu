// bf_tc.cu -- brute-force nearest neighbour with tensor-core candidate tiles and an exact re-rank
// (north_star item 4: "||q||^2 + ||p||^2 - 2 q.p" for small maps).
//
// The reference has no counterpart; the contract is the one of utils/kdtree.c:110-152 as restated in
// include/navslam_b200.h: exact 1-NN on dsq = (dx*dx + dy*dy) + dz*dz, lowest index on ties.
//
// Maximising  s(q,p) = q'.p' - |p'|^2/2  (coordinates relative to the centre c of the map's bounding
// box) is minimising |q - p|^2.  s is a K = 32 inner product that the 5th-generation tensor cores
// evaluate for a 128-query x 256-point tile per instruction pair:
//   * every centred coordinate is split into three bf16 terms x = h + m + l (24 significant bits);
//     the nine cross products of a coordinate pair fill 9 K-slots, 27 for x,y,z; three more slots
//     carry -|p'|^2/2 (split the same way) against 1.0; two slots are zero.  bf16 x bf16 products are
//     exact in fp32, so the only error is the fp32 accumulation inside the MMA, bounded by
//     E = 2^-16 * (3 Qmax Pmax + 1.5 Pmax^2)  (about 4x the 17-term truncation bound per K=16 MMA).
//   * operands are pre-tiled in global memory in the canonical no-swizzle K-major UMMA layout
//     [k-chunk of 8][row group][8 rows][16 B], so one cp.async.bulk brings a tile into shared memory
//     ready for tcgen05.mma; accumulators live in TMEM (2 x 256 columns, double buffered).
//   * warp roles: warp 4 = bulk-copy producer, warp 5 = MMA issuer (one elected lane each),
//     warps 0-3 = epilogue (tcgen05.ld of their 32 TMEM lanes, max over each 32-column group).
//   * pass 1 leaves the per-query maximum of the computed s; pass 2 recomputes the tiles and flags
//     every 32-point group whose maximum is within 2E of it: the true nearest neighbour (and every
//     point tied with it) is in a flagged group.  k_tc_rerank evaluates the flagged groups with the
//     reference's binary64 arithmetic in ascending index order.
// The answer is therefore exact for any input; only the run time depends on how many groups survive
// (dense maps far from their centre flag many).  profiles/README.md records where this beats the tree.
#include <cuda_bf16.h>
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include "nav_kdtree.cuh"

namespace nav {

constexpr int kTcM = 128;        // queries per tile (UMMA M)
constexpr int kTcN = 256;        // points per tile (UMMA N)
constexpr int kTcK = 32;         // two K=16 MMAs
constexpr int kTcGroup = 32;     // points per candidate group (= one tcgen05.ld.x32)
constexpr int kTcStages = 4;
constexpr int kTcABytes = kTcM * kTcK * 2;  // 8 KB
constexpr int kTcBBytes = kTcN * kTcK * 2;  // 16 KB
constexpr int kTcThreads = 192;

// ---- order-preserving keys for fp64 atomics -------------------------------------------------------
__device__ __forceinline__ unsigned long long okey(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double okey_inv(unsigned long long k) {
    unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

// stats[0..2] = min xyz keys, [3..5] = max xyz keys of the points, [6] = max |q - c| coordinate key
__global__ void k_tc_bbox(const double *__restrict__ pts, long long n, unsigned long long *__restrict__ stats) {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double v = pts[i * 3 + a];
            lo[a] = fmin(lo[a], v);
            hi[a] = fmax(hi[a], v);
        }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], d));
            hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], d));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&stats[a], okey(lo[a]));
            atomicMax(&stats[3 + a], okey(hi[a]));
        }
    }
}

__device__ __forceinline__ void centre_of(const unsigned long long *stats, double c[3], double &pmax) {
    pmax = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double lo = okey_inv(stats[a]), hi = okey_inv(stats[3 + a]);
        c[a] = 0.5 * (lo + hi);
        pmax = fmax(pmax, fmax(fabs(hi - c[a]), fabs(lo - c[a])));
    }
}

__device__ __forceinline__ void split3(double x, __nv_bfloat16 out[3]) {
    out[0] = __float2bfloat16_rn((float)x);
    const double r1 = x - (double)__bfloat162float(out[0]);
    out[1] = __float2bfloat16_rn((float)r1);
    const double r2 = r1 - (double)__bfloat162float(out[1]);
    out[2] = __float2bfloat16_rn((float)r2);
}

// element (row r, k) of a tile with R rows in the canonical K-major no-swizzle layout
__device__ __forceinline__ size_t canon_off(int r, int k, int R) {
    return ((size_t)(k >> 3) * (R >> 3) + (r >> 3)) * 64 + (size_t)(r & 7) * 8 + (k & 7);  // in bf16 elements
}

// B operand: one thread per point (padding rows of the last tile included)
__global__ void k_tc_prep_points(const double *__restrict__ pts, long long n, long long n_pad,
                                 const unsigned long long *__restrict__ stats, __nv_bfloat16 *__restrict__ bop) {
    double c[3], pmax;
    centre_of(stats, c, pmax);
    for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < n_pad; j += (long long)gridDim.x * blockDim.x) {
        __nv_bfloat16 row[kTcK];
#pragma unroll
        for (int k = 0; k < kTcK; ++k) row[k] = __float2bfloat16_rn(0.f);
        if (j < n) {
            double w = 0.0;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double x = pts[j * 3 + a] - c[a];
                w += x * x;
                __nv_bfloat16 s[3];
                split3(x, s);
#pragma unroll
                for (int qa = 0; qa < 3; ++qa)
#pragma unroll
                    for (int pb = 0; pb < 3; ++pb) row[9 * a + 3 * qa + pb] = s[pb];
            }
            __nv_bfloat16 ws[3];
            split3(-0.5 * w, ws);
            row[27] = ws[0];
            row[28] = ws[1];
            row[29] = ws[2];
        } else {
            row[27] = __float2bfloat16_rn(-3.0e38f);  // padding can never be a maximum
        }
        __nv_bfloat16 *tile = bop + (j / kTcN) * (size_t)(kTcN * kTcK);
        const int r = (int)(j % kTcN);
#pragma unroll
        for (int k = 0; k < kTcK; ++k) tile[canon_off(r, k, kTcN)] = row[k];
    }
}

// A operand; also accumulates the largest |q - c| coordinate into stats[6]
__global__ void k_tc_prep_queries(const double *__restrict__ q, long long nq, long long nq_pad,
                                  unsigned long long *__restrict__ stats, __nv_bfloat16 *__restrict__ aop) {
    double c[3], pmax;
    centre_of(stats, c, pmax);
    double qmax = 0.0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nq_pad; i += (long long)gridDim.x * blockDim.x) {
        __nv_bfloat16 row[kTcK];
#pragma unroll
        for (int k = 0; k < kTcK; ++k) row[k] = __float2bfloat16_rn(0.f);
        if (i < nq) {
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const double x = q[i * 3 + a] - c[a];
                qmax = fmax(qmax, fabs(x));
                __nv_bfloat16 s[3];
                split3(x, s);
#pragma unroll
                for (int qa = 0; qa < 3; ++qa)
#pragma unroll
                    for (int pb = 0; pb < 3; ++pb) row[9 * a + 3 * qa + pb] = s[qa];
            }
            row[27] = row[28] = row[29] = __float2bfloat16_rn(1.f);
        }
        __nv_bfloat16 *tile = aop + (i / kTcM) * (size_t)(kTcM * kTcK);
        const int r = (int)(i % kTcM);
#pragma unroll
        for (int k = 0; k < kTcK; ++k) tile[canon_off(r, k, kTcM)] = row[k];
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) qmax = fmax(qmax, __shfl_xor_sync(0xffffffffu, qmax, d));
    if ((threadIdx.x & 31) == 0 && qmax > 0.0) atomicMax(&stats[6], okey(qmax));
}

// ---- PTX helpers ------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned tc_smem(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_bar_init(unsigned long long *b, unsigned n) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem(b)), "r"(n));
}
__device__ __forceinline__ void tc_bar_expect(unsigned long long *b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_bar_arrive(unsigned long long *b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem(b)) : "memory");
}
__device__ __forceinline__ void tc_bar_wait(unsigned long long *b, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "TCW_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra TCD_%=;\n\t"
        "bra TCW_%=;\n\t"
        "TCD_%=:\n\t}" ::"r"(tc_smem(b)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tc_bulk(void *dst, const void *src, unsigned bytes, unsigned long long *b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     tc_smem(dst)),
                 "l"(src), "r"(bytes), "r"(tc_smem(b))
                 : "memory");
}
// K-major, no swizzle: start address, leading (k-chunk) and stride (8-row group) byte offsets in 16-byte
// units, descriptor version 1 (Blackwell)
__device__ __forceinline__ unsigned long long tc_desc(unsigned smem_addr, unsigned lbo_bytes, unsigned sbo_bytes) {
    return (unsigned long long)((smem_addr & 0x3ffffu) >> 4) | ((unsigned long long)(lbo_bytes >> 4) << 16) |
           ((unsigned long long)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, fp32 accumulate, M = 128, N = 256, K = 16
__device__ __forceinline__ void tc_mma(unsigned tmem_d, unsigned long long da, unsigned long long db, unsigned idesc,
                                       unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit(unsigned long long *b) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(b))
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// max over 32 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ float tc_group_max(unsigned taddr) {
    unsigned v[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    float m = __uint_as_float(v[0]);
#pragma unroll
    for (int i = 1; i < 32; ++i) m = fmaxf(m, __uint_as_float(v[i]));
    return m;
}

// kPass 1: rowmax[q] = max over all points of the computed s.  kPass 2: group_mask[t][q] bit g set iff
// the maximum of group g of tile t is >= rowmax[q] - 2E.
template <int kPass>
__global__ void __launch_bounds__(kTcThreads, 1)
k_tc_tiles(const __nv_bfloat16 *__restrict__ aop, const __nv_bfloat16 *__restrict__ bop, int n_tiles, long long nq_pad,
           const unsigned long long *__restrict__ stats, float *__restrict__ rowmax,
           unsigned char *__restrict__ group_mask) {
    extern __shared__ __align__(1024) unsigned char tc_dyn[];
    __shared__ __align__(8) unsigned long long bar_a, bar_full[kTcStages], bar_empty[kTcStages], bar_tfull[2],
        bar_tempty[2];
    __shared__ unsigned tmem_slot;
    unsigned char *sm_a = tc_dyn;
    unsigned char *sm_b = tc_dyn + kTcABytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long qtile = blockIdx.x;

    if (threadIdx.x == 0) {
        tc_bar_init(&bar_a, 1);
        for (int i = 0; i < kTcStages; ++i) {
            tc_bar_init(&bar_full[i], 1);
            tc_bar_init(&bar_empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            tc_bar_init(&bar_tfull[i], 1);
            tc_bar_init(&bar_tempty[i], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_slot;

    if (warp == 4) {
        if (lane == 0) {  // ---- producer: bulk copies of pre-tiled operands
            tc_bar_expect(&bar_a, kTcABytes);
            tc_bulk(sm_a, (const unsigned char *)aop + qtile * (size_t)kTcABytes, kTcABytes, &bar_a);
            for (int t = 0; t < n_tiles; ++t) {
                const int s = t % kTcStages;
                if (t >= kTcStages) tc_bar_wait(&bar_empty[s], (unsigned)((t / kTcStages - 1) & 1));
                tc_bar_expect(&bar_full[s], kTcBBytes);
                tc_bulk(sm_b + (size_t)s * kTcBBytes, (const unsigned char *)bop + (size_t)t * kTcBBytes, kTcBBytes,
                        &bar_full[s]);
            }
        }
    } else if (warp == 5) {
        if (lane == 0) {  // ---- MMA issuer
            // idesc: D=f32 (bit 4), A=B=bf16 (bits 7, 10), K-major both, N>>3 at bit 17, M>>4 at bit 24
            const unsigned idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(kTcN >> 3) << 17) |
                                   ((unsigned)(kTcM >> 4) << 24);
            tc_bar_wait(&bar_a, 0);
            for (int t = 0; t < n_tiles; ++t) {
                const int s = t % kTcStages, a = t & 1;
                if (t >= 2) tc_bar_wait(&bar_tempty[a], (unsigned)((t / 2 - 1) & 1));
                tc_bar_wait(&bar_full[s], (unsigned)((t / kTcStages) & 1));
                tc_fence_after();
                const unsigned a_addr = tc_smem(sm_a), b_addr = tc_smem(sm_b + (size_t)s * kTcBBytes);
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    // one MMA consumes two 16-byte k-chunks: chunk stride = (rows/8)*128 B, row-group stride = 128 B
                    const unsigned long long da = tc_desc(a_addr + k * 2 * (kTcM / 8) * 128, (kTcM / 8) * 128, 128);
                    const unsigned long long db = tc_desc(b_addr + k * 2 * (kTcN / 8) * 128, (kTcN / 8) * 128, 128);
                    tc_mma(tmem_base + (unsigned)a * kTcN, da, db, idesc, (unsigned)k);
                }
                tc_commit(&bar_empty[s]);  // shared-memory slot reusable once these MMAs have read it
                tc_commit(&bar_tfull[a]);  // accumulator a complete
            }
        }
    } else {  // ---- epilogue: warp w owns TMEM lanes 32w .. 32w+31 = query rows of the tile
        const long long q = qtile * kTcM + warp * 32 + lane;
        double c[3], pmax;
        centre_of(stats, c, pmax);
        const double qmax = stats[6] ? okey_inv(stats[6]) : 0.0;
        const float two_e = (float)(2.0 * ldexp(3.0 * qmax * pmax + 1.5 * pmax * pmax, -16)) * 1.0001f + 1e-30f;
        float run = -INFINITY;
        const float thr = kPass == 2 ? rowmax[q] - two_e : 0.f;
        const unsigned lane_base = tmem_base + ((unsigned)(warp * 32) << 16);
        for (int t = 0; t < n_tiles; ++t) {
            const int a = t & 1;
            tc_bar_wait(&bar_tfull[a], (unsigned)((t / 2) & 1));
            tc_fence_after();
            unsigned bits = 0;
#pragma unroll 1
            for (int g = 0; g < kTcN / kTcGroup; ++g) {
                const float m = tc_group_max(lane_base + (unsigned)(a * kTcN + g * kTcGroup));
                if (kPass == 1)
                    run = fmaxf(run, m);
                else if (m >= thr)
                    bits |= 1u << g;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) tc_bar_arrive(&bar_tempty[a]);
            if (kPass == 2) group_mask[(size_t)t * nq_pad + q] = (unsigned char)bits;
        }
        if (kPass == 1) rowmax[q] = run;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// exact re-rank: one warp per query.  Lanes first fetch the flag bytes of 32 tiles at a time, then the
// warp walks the flagged groups: lane l evaluates point l of the group (one coalesced 768-byte read)
// with the reference's binary64 arithmetic, and a lexicographic (dsq, index) min-reduction keeps the
// lowest index among equal dsq.
__global__ void __launch_bounds__(256)
k_tc_rerank(const double *__restrict__ pts, long long n, const double *__restrict__ queries, long long nq,
            long long nq_pad, int n_tiles, const unsigned char *__restrict__ group_mask,
            const unsigned long long *__restrict__ stats, int *__restrict__ idx_out, double *__restrict__ dist_out,
            unsigned long long *__restrict__ n_evals) {
    const long long qi = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (qi >= nq) return;
    const double qx = queries[qi * 3], qy = queries[qi * 3 + 1], qz = queries[qi * 3 + 2];
    double best = INFINITY;
    int bidx = INT_MAX;
    unsigned evals = 0;
    // The bf16 operands of the tiles are bounded by Qmax, Pmax and 1.5 Pmax^2, every fp32 product and partial sum
    // by 3 Qmax Pmax + 1.5 Pmax^2 (times a factor near 1).  Beyond 2^90 -- or with an infinite centre -- some of
    // them may have overflowed to inf / NaN and the flags mean nothing: then every group is re-ranked.
    double c[3], pmax;
    centre_of(stats, c, pmax);
    const double qmax = stats[6] ? okey_inv(stats[6]) : 0.0;
    const double bound = fmax(fmax(qmax, pmax), 3.0 * qmax * pmax + 1.5 * pmax * pmax);
    const bool scan_all = !(bound < 0x1p90) || !(fabs(c[0]) + fabs(c[1]) + fabs(c[2]) < INFINITY);
    for (int t0 = 0; t0 < n_tiles; t0 += 32) {
        const int tl = t0 + lane;
        unsigned mine = 0;
        if (tl < n_tiles) mine = scan_all ? 0xffu : group_mask[(size_t)tl * nq_pad + qi];
        unsigned any = __ballot_sync(0xffffffffu, mine != 0);
        while (any) {
            const int src = __ffs(any) - 1;
            any &= any - 1;
            unsigned m = __shfl_sync(0xffffffffu, mine, src);
            while (m) {
                const int g = __ffs(m) - 1;
                m &= m - 1;
                const long long j = (long long)(t0 + src) * kTcN + g * kTcGroup + lane;
                if (j < n) {
                    const double d = dsq3(dsub(pts[j * 3], qx), dsub(pts[j * 3 + 1], qy), dsub(pts[j * 3 + 2], qz));
                    if (d < best || (d == best && (int)j < bidx)) {
                        best = d;
                        bidx = (int)j;
                    }
                }
                evals += 1;
            }
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, d);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, d);
        if (ob < best || (ob == best && oi < bidx)) {
            best = ob;
            bidx = oi;
        }
    }
    if (lane == 0) {
        // no point at a finite dsq (every dsq +inf or NaN): no answer, as in k_bf_nn
        const bool found = best < INFINITY;
        idx_out[qi] = found ? bidx : -1;
        dist_out[qi] = found ? __dsqrt_rn(best) : INFINITY;
        if (n_evals) atomicAdd(n_evals, (unsigned long long)evals * kTcGroup);
    }
}

__global__ void k_tc_init_stats(unsigned long long *stats) {
    if (threadIdx.x < 3) stats[threadIdx.x] = ~0ull;
    if (threadIdx.x >= 3 && threadIdx.x < 9) stats[threadIdx.x] = 0ull;
}

#define TC_CHECK(call)               \
    do {                             \
        cudaError_t e_ = (call);     \
        if (e_ != cudaSuccess) {     \
            status = e_;             \
            goto done;               \
        }                            \
    } while (0)

cudaError_t bf_nn_tc(const double *d_pts, size_t n, const double *d_queries, size_t nq, int *d_idx, double *d_dist,
                     int sm_count, cudaStream_t stream, unsigned long long *h_evals_out) {
    if (nq == 0) return cudaSuccess;
    if (n == 0) return bf_nn(d_pts, n, d_queries, nq, d_idx, d_dist, stream);
    cudaError_t status = cudaSuccess;
    const long long n_tiles = ((long long)n + kTcN - 1) / kTcN, n_pad = n_tiles * kTcN;
    const long long q_tiles = ((long long)nq + kTcM - 1) / kTcM, nq_pad = q_tiles * kTcM;
    unsigned long long *stats = nullptr;
    __nv_bfloat16 *aop = nullptr, *bop = nullptr;
    float *rowmax = nullptr;
    unsigned char *mask = nullptr;
    // 8 KB A + 4 x 16 KB B, padded to 120 KB so that only one CTA (which owns all 512 TMEM columns) fits per SM
    const size_t dyn = 120 * 1024;
    static_assert(kTcABytes + kTcStages * kTcBBytes <= 120 * 1024, "operand ring exceeds the dynamic smem request");
    static bool configured = false;
    int device = 0;
    if (n_tiles > 0x7fffffffLL || q_tiles > 0x7fffffffLL) return cudaErrorInvalidValue;
    if (!configured) {
        TC_CHECK(cudaFuncSetAttribute(k_tc_tiles<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        TC_CHECK(cudaFuncSetAttribute(k_tc_tiles<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
        configured = true;
    }
    TC_CHECK(cudaGetDevice(&device));
    // workspace from the library's own stream-ordered pool (kd_pool_alloc, kdbuild.cu)
    TC_CHECK(kd_pool_alloc((void **)&stats, 9 * sizeof(unsigned long long), device, stream));
    TC_CHECK(kd_pool_alloc((void **)&aop, (size_t)nq_pad * kTcK * 2, device, stream));
    TC_CHECK(kd_pool_alloc((void **)&bop, (size_t)n_pad * kTcK * 2, device, stream));
    TC_CHECK(kd_pool_alloc((void **)&rowmax, (size_t)nq_pad * 4, device, stream));
    TC_CHECK(kd_pool_alloc((void **)&mask, (size_t)n_tiles * nq_pad, device, stream));
    {
        const int g1 = (int)((n + 255) / 256 < (size_t)sm_count * 8 ? (n + 255) / 256 : (size_t)sm_count * 8);
        const int g2 = (int)((n_pad + 127) / 128 < (long long)sm_count * 16 ? (n_pad + 127) / 128 : (long long)sm_count * 16);
        const int g3 = (int)((nq_pad + 127) / 128 < (long long)sm_count * 16 ? (nq_pad + 127) / 128 : (long long)sm_count * 16);
        k_tc_init_stats<<<1, 32, 0, stream>>>(stats);
        k_tc_bbox<<<g1, 256, 0, stream>>>(d_pts, (long long)n, stats);
        k_tc_prep_points<<<g2, 128, 0, stream>>>(d_pts, (long long)n, n_pad, stats, bop);
        k_tc_prep_queries<<<g3, 128, 0, stream>>>(d_queries, (long long)nq, nq_pad, stats, aop);
        k_tc_tiles<1><<<(unsigned)q_tiles, kTcThreads, dyn, stream>>>(aop, bop, (int)n_tiles, nq_pad, stats, rowmax, mask);
        k_tc_tiles<2><<<(unsigned)q_tiles, kTcThreads, dyn, stream>>>(aop, bop, (int)n_tiles, nq_pad, stats, rowmax, mask);
        k_tc_rerank<<<(unsigned)((nq * 32 + 255) / 256), 256, 0, stream>>>(d_pts, (long long)n, d_queries, (long long)nq, nq_pad,
                                                                      (int)n_tiles, mask, stats, d_idx, d_dist, stats + 8);
    }
    TC_CHECK(cudaGetLastError());
    if (h_evals_out) {
        TC_CHECK(cudaMemcpyAsync(h_evals_out, stats + 8, 8, cudaMemcpyDeviceToHost, stream));
        TC_CHECK(cudaStreamSynchronize(stream));
    }
done:
    cudaFreeAsync(stats, stream);
    cudaFreeAsync(aop, stream);
    cudaFreeAsync(bop, stream);
    cudaFreeAsync(rowmax, stream);
    cudaFreeAsync(mask, stream);
    return status;
}

}  // namespace nav
