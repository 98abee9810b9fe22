// nav_common.cuh -- shared device helpers for libnavslam_b200 (sm_100a).
//
// Bit-exactness contract: the reference (wuHakureReimu/NAV-SLAM) is binary64 C compiled for
// baseline x86-64, i.e. every +,-,*,/ and sqrt is a separately rounded IEEE operation in source
// association order (no FMA contraction).  All arithmetic that decides an output goes through the
// __d*_rn intrinsics below, which nvcc never fuses, so labels, distances and transformed points
// are bit-identical to the reference's.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/navslam_b200.h"

namespace nav {

struct P3 {
    double x, y, z;
};

// T = t + R*p  (src/slam.c:147-158), Q = T - shift (src/slam.c:126-128)
struct PoseXf {
    double R[9];
    double t[3];
    double shift[3];
};
struct PoseBatch {
    PoseXf p[NAV_MAX_SEQ];
};

__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

// (dx*dx + dy*dy) + dz*dz, the association of src/slam.c:32 and utils/kdtree.c:16
__device__ __forceinline__ double dsq3(double dx, double dy, double dz) {
    return dadd(dadd(dmul(dx, dx), dmul(dy, dy)), dmul(dz, dz));
}
__device__ __forceinline__ double dsq_pts(const P3 &a, const P3 &b) {
    return dsq3(dsub(a.x, b.x), dsub(a.y, b.y), dsub(a.z, b.z));
}

// rotated = (R0*x + R1*y) + R2*z ; out = t + rotated   (src/slam.c:151-158)
__device__ __forceinline__ P3 xf_point(const PoseXf &q, const P3 &p) {
    P3 o;
    o.x = dadd(q.t[0], dadd(dadd(dmul(q.R[0], p.x), dmul(q.R[1], p.y)), dmul(q.R[2], p.z)));
    o.y = dadd(q.t[1], dadd(dadd(dmul(q.R[3], p.x), dmul(q.R[4], p.y)), dmul(q.R[5], p.z)));
    o.z = dadd(q.t[2], dadd(dadd(dmul(q.R[6], p.x), dmul(q.R[7], p.y)), dmul(q.R[8], p.z)));
    return o;
}
__device__ __forceinline__ P3 shift_point(const PoseXf &q, const P3 &g) {
    P3 o;
    o.x = dsub(g.x, q.shift[0]);
    o.y = dsub(g.y, q.shift[1]);
    o.z = dsub(g.z, q.shift[2]);
    return o;
}

// Lower bound of the *computed* dsq between q and any point inside the box [lo,hi]: rounding is
// monotone, so evaluating the clamped per-axis gaps with the same rounded operations in the same
// association order can never exceed the dsq3() of a point in the box.
__device__ __forceinline__ double box_lower_bound(const double *__restrict__ box, const P3 &q) {
    double ex = fmax(0.0, fmax(dsub(box[0], q.x), dsub(q.x, box[3])));
    double ey = fmax(0.0, fmax(dsub(box[1], q.y), dsub(q.y, box[4])));
    double ez = fmax(0.0, fmax(dsub(box[2], q.z), dsub(q.z, box[5])));
    return dsq3(ex, ey, ez);
}

// The same bound with fp32 boxes: the box is stored rounded OUTWARD (lo down, hi up), the query is
// bracketed by q_dn <= q <= q_up, and every operation rounds down, so
//   ex <= the real per-axis gap <= |RN64(p - q)| for every point p of the box,
// hence s = RD(ex^2+ey^2+ez^2) <= the real sum <= dsq3(...)/(1 - 2^-51); the final factor (1 - 2^-20)
// makes the result STRICTLY smaller than any dsq the reference arithmetic can produce for that box.
// Pruning "lb32 > float_round_up(best)" therefore never discards a candidate with dsq <= best.
struct Q32 {
    float dn[3], up[3];
};
__device__ __forceinline__ Q32 make_q32(const P3 &q) {
    Q32 r;
    r.dn[0] = __double2float_rd(q.x);
    r.dn[1] = __double2float_rd(q.y);
    r.dn[2] = __double2float_rd(q.z);
    r.up[0] = __double2float_ru(q.x);
    r.up[1] = __double2float_ru(q.y);
    r.up[2] = __double2float_ru(q.z);
    return r;
}
__device__ __forceinline__ float box_lower_bound32(const float4 lo, const float4 hi, const Q32 &q) {
    const float ex = fmaxf(0.f, fmaxf(__fsub_rd(lo.x, q.up[0]), __fsub_rd(q.dn[0], hi.x)));
    const float ey = fmaxf(0.f, fmaxf(__fsub_rd(lo.y, q.up[1]), __fsub_rd(q.dn[1], hi.y)));
    const float ez = fmaxf(0.f, fmaxf(__fsub_rd(lo.z, q.up[2]), __fsub_rd(q.dn[2], hi.z)));
    const float s = __fmaf_rd(ez, ez, __fmaf_rd(ey, ey, __fmul_rd(ex, ex)));
    return __fmul_rd(s, 0.99999905f);
}

// The closed loop's translation fit (src/slam.c:341-370 on five sufficient statistics): 200 Adam iterations on
// st = {N, sum rx, sum ry, sum rz, sum |r|^2}, starting from t[0..2] = pred - last; t is updated in place and the
// RMS residual returned.  c1[i] / c2[i] = 1 - beta1^(i+1) / 1 - beta2^(i+1), tables the host forms once with its
// pow() (the only libm call of the loop).  One source for the host (nav_slam_fit_from_stats, the host closed loop)
// and the device (nav_slam_run_dev): the rest is + - * /, sqrt, fabs and fmax, device code is built with
// -fmad=false and host code with -ffp-contract=off, so both sides give the same bits.
constexpr int kFitIters = 200;
__host__ __device__ inline double fit_translation(const double st[5], double t[3], const double *c1, const double *c2) {
    const double lr = 0.1, tol = 1e-6, b1 = 0.9, b2 = 0.999, eps = 1e-8;
    const double N = st[0], S[3] = {st[1], st[2], st[3]}, Q = st[4];
    double m[3] = {0, 0, 0}, v[3] = {0, 0, 0}, prev = 0, total = 0;
    for (int iter = 0; iter < kFitIters; ++iter) {
        total = Q - 2.0 * (t[0] * S[0] + t[1] * S[1] + t[2] * S[2]) + N * (t[0] * t[0] + t[1] * t[1] + t[2] * t[2]);
        if (N == 0) total = 0;
        if (fabs(total - prev) < tol) break;
        prev = total;
        const double k1 = c1[iter], k2 = c2[iter];
        for (int j = 0; j < 3; ++j) {
            const double g = N > 0 ? -(S[j] - N * t[j]) / N : 0.0;
            m[j] = b1 * m[j] + (1 - b1) * g;
            v[j] = b2 * v[j] + (1 - b2) * g * g;
            const double mh = m[j] / k1, vh = v[j] / k2;
            t[j] -= lr * mh / (sqrt(vh) + eps);
        }
    }
    return N > 0 ? sqrt(fmax(total, 0.0) / N) : 0.0;
}

constexpr int kChunk = 16;       // map points per leaf box
constexpr int kChunksPerSuper = 16;

__host__ __device__ inline int div_up(int a, int b) { return (a + b - 1) / b; }

}  // namespace nav
