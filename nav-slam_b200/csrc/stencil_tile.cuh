// stencil_tile.cuh -- the curvature / edge-label stencil on one shared-memory tile (a3).
//
// Reference arithmetic (src/slam.c:18-58), all binary64:
//     d_k = sqrt((dx*dx + dy*dy) + dz*dz)  for the same-row neighbours k = -2,-1,+1,+2
//     S = ((d-2 + d-1) + d+1) + d+2 ; avg = S/4 ; if avg > 0: V = sum_k (d_k-avg)^2 (tap order)
//     curv = (V/4) / (avg*avg + (double)1e-6f) ; label = curv > 0.1
//
// Two evaluators over a tile of kTile columns + 2 halo points each side staged in shared memory:
//
//  * tile_curvature_exact(): the reference's arithmetic operation for operation (separately rounded
//    __d*_rn, never fused), with the two forward distances |p_j - p_{j+1}|, |p_j - p_{j+2}| computed
//    once per point and shared -- the backward taps are the same numbers because IEEE subtraction
//    is antisymmetric and the sign is squared away.  Bit-identical curvature.
//
//  * tile_labels_filtered(): the label only needs the SIGN of (curv - 0.1).  Coordinate
//    differences are still taken in binary64 (the survey measured that rounding the *inputs* to
//    fp32 flips labels, SURVEY D5), then everything runs in fp32 together with a rigorous bound
//    `err` on |c32 - curv| (derivation below).  A point is decided in fp32 only when c32 is
//    farther than err from the threshold; otherwise (about 1 point in 10^4 on lidar data, and any
//    NaN/inf/denormal case) that lane re-evaluates the exact binary64 expression.  The labels are
//    therefore bit-identical to the reference's while the fp64 pipe does 12 operations per point
//    instead of ~80, which is what lets the batched stencil run at HBM speed.
//
//    Error bound (u = 2^-24; every fp32 op below is a correctly rounded add/mul/fma except
//    sqrt.approx (<= 2^-22 relative) and rcp.approx (<= 2^-23)):
//      diff32 = diff64 (1+u)                        -> dsq32 = dsq (1+5u)   (two squares, 3 roundings)
//      d32 = d (1+g), g <= 2.5u + 4u                -> take g = 8u
//      avg32: three adds of non-negative terms      -> |avg32-avg| <= 12u avg
//      e32_k = fl(d32_k - avg32), d_k <= 4 avg      -> |e32_k-e_k| <= 50u avg =: h
//      V32 (fma chain of non-negative terms)        -> |V32-V| <= 2 h A + 4 h^2 + 4.1u V,  A >= sum|e_k|
//      den32 = fma(avg32,avg32,1e-6f)               -> |den32-den| <= 26u den
//      c32 = 0.25 * V32 * rcp(den32)                -> |c32-curv| <= 25u avg A/den + 40u curv + 1e-11
//    The kernel uses 64u (avg32 A32 / den32) + 64u c32 + 1e-9, i.e. more than twice that.
//    Range: overflow (|diff| > 1.8e19) gives inf, then avg = inf, e = inf - inf = NaN and the point
//    goes to the exact path, as does any NaN input.  Underflow (a squared difference below
//    FLT_MIN, flushed by sqrt.approx.ftz) costs an ABSOLUTE error below 2e-19 in that distance;
//    an absolute error eps in one d_k moves c by at most 2*3avg*eps/den <= 3000 eps (den >= 2e-3 avg),
//    i.e. < 1e-15, far inside the 1e-9 slack.  avg32 == 0 means all four distances are below 1.1e-19,
//    for which the reference's curvature is < 1e-30: label 0.
#pragma once
#include "nav_common.cuh"

namespace nav {

constexpr int kTile = 256;  // columns per CTA tile (= 16 leaf blocks = 1 super block of the row map)
constexpr int kHalo = 2;

constexpr int kTilePts = kTile + 2 * kHalo;  // staged points per tile

struct StencilSmem {
    double pts[kTilePts * 3];
    union {
        struct {
            double f1[kTile + kHalo];
            double f2[kTile + kHalo];
        } ex;
        struct {
            float f1[kTile + kHalo];
            float f2[kTile + kHalo];
        } fl;
    };
};

// stage columns [c0-2, c0+kTile+2) of one row; slots outside the row are zero and only feed the
// border columns, which the reference never evaluates (src/slam.c:16)
__device__ __forceinline__ void tile_stage(StencilSmem &s, const double *__restrict__ row_ptr, int c0, int cols) {
    const int first = c0 - kHalo;
    for (int i = threadIdx.x; i < (kTile + 2 * kHalo) * 3; i += kTile) {
        const int col = first + i / 3;
        double v = 0.0;
        if (col >= 0 && col < cols) v = __ldg(row_ptr + (long long)first * 3 + i);
        s.pts[i] = v;
    }
}

// ---- the narrow frame formats (NAV_RUN_INPUT_DEPTH / _MM), converted point by point where they are read.  One
// definition for the conversion kernels (k_convert, k_widen_mm) and for the kernels that stage raw tiles, so the
// bits cannot drift between them.
constexpr int kKindXyz = NAV_RUN_INPUT_XYZ, kKindDepth = NAV_RUN_INPUT_DEPTH, kKindMm = NAV_RUN_INPUT_MM;

// a2 of one pixel, utils/pointcloud.c:18-47: tan(theta_col) / tan(phi_row) are the host libm's values, y = (-d) * tan
// is one rounded multiply; d <= 0 is no return, (0, 0, 0)
__device__ __forceinline__ P3 depth_point(int dist, double tan_c, double tan_r) {
    const double d = (double)dist;
    P3 p = {0.0, 0.0, 0.0};
    if (!(d <= 0.0)) {
        p.x = d;
        p.y = dmul(-d, tan_c);
        p.z = dmul(-d, tan_r);
    }
    return p;
}
// whole millimetres: every int32 is exact in binary64
__device__ __forceinline__ double mm_coord(int v) { return (double)v; }

// A tile of a depth or integer-mm row staged raw in shared memory: element li is column c0 - kHalo + li, as in the
// xyz tile.  Columns outside the row hold zeros, which both conversions turn into (0, 0, 0), the xyz tile's padding.
template <int kKind>
struct RawTile;
template <>
struct RawTile<kKindDepth> {
    const int *d;         // depth of element li at d[li]
    const double *tan_c;  // tan of its column at tan_c[li]
    double tan_r;         // tan of the image row
    __device__ __forceinline__ P3 at(int li) const { return depth_point(d[li], tan_c[li], tan_r); }
};
template <>
struct RawTile<kKindMm> {
    const int *v;  // x, y, z of element li at v[3 li ..]
    __device__ __forceinline__ P3 at(int li) const {
        const int *p = v + li * 3;
        return P3{mm_coord(p[0]), mm_coord(p[1]), mm_coord(p[2])};
    }
};

__device__ __forceinline__ double curvature_from_taps(double dm2, double dm1, double dp1, double dp2) {
    const double sum = dadd(dadd(dadd(dm2, dm1), dp1), dp2);
    const double avg = dmul(sum, 0.25);  // sum / 4: exact scaling
    double curv = 0.0;
    if (avg > 0.0) {
        double e = dsub(dm2, avg);
        double var = dmul(e, e);
        e = dsub(dm1, avg);
        var = dadd(var, dmul(e, e));
        e = dsub(dp1, avg);
        var = dadd(var, dmul(e, e));
        e = dsub(dp2, avg);
        var = dadd(var, dmul(e, e));
        curv = __ddiv_rn(dmul(var, 0.25), dadd(dmul(avg, avg), (double)1e-6f));
    }
    return curv;
}

// exact distance between staged points a and b (local indices)
__device__ __forceinline__ double tile_dist(const double *pts, int a, int b) {
    const double *p = pts + a * 3, *q = pts + b * 3;
    return __dsqrt_rn(dsq3(dsub(p[0], q[0]), dsub(p[1], q[1]), dsub(p[2], q[2])));
}

template <int kKind>
__device__ __forceinline__ double tile_dist(const RawTile<kKind> &t, int a, int b) {
    const P3 p = t.at(a), q = t.at(b);
    return __dsqrt_rn(dsq3(dsub(p.x, q.x), dsub(p.y, q.y), dsub(p.z, q.z)));
}

// exact curvature of the thread's own column; needs tile_stage + __syncthreads before.
// Contains two __syncthreads: call from all kTile threads.
__device__ __forceinline__ double tile_curvature_exact(StencilSmem &s, int c0, int cols) {
    for (int i = threadIdx.x; i < kTile + kHalo; i += kTile) {
        s.ex.f1[i] = tile_dist(s.pts, i, i + 1);
        s.ex.f2[i] = tile_dist(s.pts, i, i + 2);
    }
    __syncthreads();
    const int col = c0 + threadIdx.x, li = threadIdx.x + kHalo;
    double curv = 0.0;
    if (col >= kHalo && col < cols - kHalo)
        curv = curvature_from_taps(s.ex.f2[li - 2], s.ex.f1[li - 1], s.ex.f1[li], s.ex.f2[li]);
    __syncthreads();
    return curv;
}

__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// fp32 forward distance: differences in binary64, everything after in fp32
__device__ __forceinline__ float tile_dist32(const double *pts, int a, int b) {
    const double *p = pts + a * 3, *q = pts + b * 3;
    const float dx = (float)dsub(p[0], q[0]), dy = (float)dsub(p[1], q[1]), dz = (float)dsub(p[2], q[2]);
    return sqrt_approx(__fmaf_rn(dx, dx, __fmaf_rn(dy, dy, dz * dz)));
}

template <int kKind>
__device__ __forceinline__ float tile_dist32(const RawTile<kKind> &t, int a, int b) {
    const P3 p = t.at(a), q = t.at(b);
    const float dx = (float)dsub(p.x, q.x), dy = (float)dsub(p.y, q.y), dz = (float)dsub(p.z, q.z);
    return sqrt_approx(__fmaf_rn(dx, dx, __fmaf_rn(dy, dy, dz * dz)));
}

// the reference's exact binary64 label of staged point li (rare path: kept out of line so that its
// sqrt/div sequences do not inflate the register budget of the streaming kernels)
static __device__ __noinline__ int label_exact_at(const double *pts, int li) {
    const double curv = curvature_from_taps(tile_dist(pts, li, li - 2), tile_dist(pts, li, li - 1),
                                            tile_dist(pts, li, li + 1), tile_dist(pts, li, li + 2));
    return curv > 0.1 ? 1 : 0;
}
template <int kKind>
static __device__ __noinline__ int label_exact_at(RawTile<kKind> t, int li) {
    const double curv = curvature_from_taps(tile_dist(t, li, li - 2), tile_dist(t, li, li - 1), tile_dist(t, li, li + 1),
                                            tile_dist(t, li, li + 2));
    return curv > 0.1 ? 1 : 0;
}

// decide one label from the four fp32 tap distances, falling back to the reference's binary64
// expression (evaluated from the staged points around local index li) when fp32 cannot decide.
// Pts: the staged xyz tile (const double *) or a RawTile
template <typename Pts>
__device__ __forceinline__ int label_from_taps32(float dm2, float dm1, float dp1, float dp2, Pts pts, int li,
                                                 unsigned *n_exact) {
    const float avg = 0.25f * (((dm2 + dm1) + dp1) + dp2);
    const float e0 = dm2 - avg, e1 = dm1 - avg, e2 = dp1 - avg, e3 = dp2 - avg;
    const float var = __fmaf_rn(e3, e3, __fmaf_rn(e2, e2, __fmaf_rn(e1, e1, e0 * e0)));
    const float a_sum = (fabsf(e0) + fabsf(e1)) + (fabsf(e2) + fabsf(e3)) + 3.1e-5f * avg;  // A >= sum|e_k|
    const float rden = rcp_approx(__fmaf_rn(avg, avg, 1e-6f));
    const float c32 = 0.25f * var * rden;
    const float u64 = 64.f * 5.9604645e-8f;
    const float err = __fmaf_rn(u64, avg * a_sum * rden, __fmaf_rn(u64, c32, 1e-9f));
    if (avg == 0.f) return 0;
    if (c32 - err > 0.1000001f) return 1;
    if (c32 + err < 0.0999999f) return 0;
    // too close to call in fp32 (or NaN/inf): the reference's own arithmetic
    if (n_exact) atomicAdd(n_exact, 1u);
    return label_exact_at(pts, li);
}

// label (0/1) of the thread's own column; needs tile_stage + __syncthreads before.
// Contains two __syncthreads: call from all kTile threads.  *n_exact counts exact re-evaluations.
template <typename Pts>
__device__ __forceinline__ int tile_labels_filtered(Pts pts, float *f1, float *f2, int c0, int cols,
                                                    unsigned *n_exact) {
    for (int i = threadIdx.x; i < kTile + kHalo; i += kTile) {
        f1[i] = tile_dist32(pts, i, i + 1);
        f2[i] = tile_dist32(pts, i, i + 2);
    }
    __syncthreads();
    const int col = c0 + threadIdx.x, li = threadIdx.x + kHalo;
    int label = 0;
    if (col >= kHalo && col < cols - kHalo)
        label = label_from_taps32(f2[li - 2], f1[li - 1], f1[li], f2[li], pts, li, n_exact);
    __syncthreads();
    return label;
}
__device__ __forceinline__ int tile_labels_filtered(StencilSmem &s, int c0, int cols, unsigned *n_exact) {
    return tile_labels_filtered((const double *)s.pts, s.fl.f1, s.fl.f2, c0, cols, n_exact);
}

}  // namespace nav
