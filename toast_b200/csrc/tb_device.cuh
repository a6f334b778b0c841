// tb_device.cuh -- device-side building blocks shared by the operator kernels (tb_ops.cu)
// and the fused destriper passes (tb_solver.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "tb_math.cuh"

namespace tbd {

constexpr int kThreads = 256;          // threads per CTA
#ifndef TB_PER_THREAD
#define TB_PER_THREAD 4
#endif
constexpr int kPerThread = TB_PER_THREAD; // samples per thread per tile
constexpr int kTile = kThreads * kPerThread; // samples per tile (flattened interval space)

// The reference loops `for view: for isamp in [first, last)`.  We flatten that iteration
// space: flat index t in [0, total) <-> (view, sample) with prefix[v] <= t < prefix[v+1],
// sample = first[v] + (t - prefix[v]).  Overlapping intervals are visited twice exactly like
// the reference; samples outside every interval are never touched.
struct Views {
    const int64_t *first;  // [n_view]
    const int64_t *prefix; // [n_view + 1]
    int n_view;
    int64_t total;
};

__device__ __forceinline__ int find_view(const Views &v, int64_t t) {
    int lo = 0, hi = v.n_view;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (__ldg(v.prefix + mid) <= t) {
            lo = mid;
        } else {
            hi = mid;
        }
    }
    return lo;
}

// A thread visits increasing flat indices, and a tile rarely straddles an interval: locate the
// view once per tile (one binary search) and then only step forward, instead of a 7-deep chain
// of dependent loads per sample (ground scans have ~100 intervals per observation).
struct ViewCursor {
    int view;
    int64_t beg, end, first; // prefix[view], prefix[view + 1], first[view]
};
__device__ __forceinline__ ViewCursor view_cursor(const Views &v, int64_t t) {
    ViewCursor c;
    if (t >= v.total) t = v.total - 1;
    c.view = (v.n_view > 1 && t > 0) ? find_view(v, t) : 0;
    c.beg = __ldg(v.prefix + c.view);
    c.end = __ldg(v.prefix + c.view + 1);
    c.first = __ldg(v.first + c.view);
    return c;
}
__device__ __forceinline__ void view_seek(const Views &v, ViewCursor &c, int64_t t) {
    while (t >= c.end) { // t < total is the caller's responsibility
        ++c.view;
        c.beg = c.end;
        c.end = __ldg(v.prefix + c.view + 1);
        c.first = __ldg(v.first + c.view);
    }
}

// Tile decomposition with TIME-MAJOR CTA order: consecutive CTAs work on the same time window
// of consecutive detectors, so the pixels they scatter to / gather from are neighbours on the
// sky and the zmap / map tiles stay resident in the 126 MB L2.
struct TileId {
    int64_t t0; // first flat index of the tile
    int det;
};
__device__ __forceinline__ TileId tile_of_block(int64_t block, int64_t n_det) {
    TileId r;
    int64_t tile = block / n_det;
    r.det = (int)(block - tile * n_det);
    r.t0 = tile * (int64_t)kTile;
    return r;
}

// floor(n / d) for 0 <= n < 2^51 via one multiply (inv = 1.0 / d): (n + 0.5) / d is at least
// 0.5/d away from an integer while the rounding error is ~ 2^-52 n/d.
__device__ __forceinline__ int64_t fast_div(int64_t n, double inv_d) {
    return (int64_t)(((double)n + 0.5) * inv_d);
}

// streaming 8-byte loads that do not pollute L1 (each datum is used once)
__device__ __forceinline__ double ld_stream(const double *p) { return __ldcs(p); }
__device__ __forceinline__ int64_t ld_stream(const int64_t *p) {
    return (int64_t)__ldcs((const long long *)p);
}
__device__ __forceinline__ uint8_t ld_stream(const uint8_t *p) {
    return (uint8_t)__ldcs((const unsigned char *)p);
}
__device__ __forceinline__ void st_stream(double *p, double v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(int64_t *p, int64_t v) { __stcs((long long *)p, (long long)v); }

__device__ __forceinline__ tbm::Quat ld_quat(const double *p) {
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
    double2 a = __ldg(p2);
    double2 b = __ldg(p2 + 1);
    return tbm::Quat{a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ tbm::Quat ld_quat_stream(const double *p) {
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
    double2 a = __ldcs(p2);
    double2 b = __ldcs(p2 + 1);
    return tbm::Quat{a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void st_quat_stream(double *p, const tbm::Quat &q) {
    double2 *p2 = reinterpret_cast<double2 *>(p);
    __stcs(p2, make_double2(q.x, q.y));
    __stcs(p2 + 1, make_double2(q.z, q.w));
}

// ---- warp-level segmented sums --------------------------------------------------------------
// Lanes hold consecutive samples; equal keys come in runs (a detector dwells on a pixel / a
// baseline step for several samples).  Sum each run inside the warp and let the run's LAST
// lane issue the atomic, which divides the atomic traffic by the mean run length.
struct Runs {
    int dist;     // distance of this lane from the head lane of its run
    bool is_tail; // this lane is the last of its run
};

// CAP (power of two <= 32) bounds the run length: runs are additionally cut at lane multiples
// of CAP so that log2(CAP) shuffle steps suffice.  Shuffles share the LSU/shared-memory data
// pipe with the loads, so for short natural runs (a few samples per pixel) a small CAP is
// cheaper than the extra atomics it causes.
template <int CAP = 32>
__device__ __forceinline__ Runs find_runs(int64_t key, int lane) {
    int64_t prev = __shfl_up_sync(0xffffffffu, key, 1);
    bool head = (lane == 0) || (prev != key) || ((CAP < 32) && ((lane & (CAP - 1)) == 0));
    unsigned heads = __ballot_sync(0xffffffffu, head);
    unsigned upto = heads & (0xffffffffu >> (31 - lane));
    int head_lane = 31 - __clz(upto);
    Runs r;
    r.dist = lane - head_lane;
    unsigned tails = (heads >> 1) | 0x80000000u;
    r.is_tail = (tails >> lane) & 1u;
    return r;
}

// the same for 32-bit keys (one shuffle instead of two)
template <int CAP = 32>
__device__ __forceinline__ Runs find_runs32(int32_t key, int lane) {
    int32_t prev = __shfl_up_sync(0xffffffffu, key, 1);
    bool head = (lane == 0) || (prev != key) || ((CAP < 32) && ((lane & (CAP - 1)) == 0));
    unsigned heads = __ballot_sync(0xffffffffu, head);
    unsigned upto = heads & (0xffffffffu >> (31 - lane));
    int head_lane = 31 - __clz(upto);
    Runs r;
    r.dist = lane - head_lane;
    unsigned tails = (heads >> 1) | 0x80000000u;
    r.is_tail = (tails >> lane) & 1u;
    return r;
}

template <int CAP = 32>
__device__ __forceinline__ double seg_sum(double v, const Runs &r) {
#pragma unroll
    for (int off = 1; off < CAP; off <<= 1) {
        double u = __shfl_up_sync(0xffffffffu, v, off);
        if (r.dist >= off) v += u;
    }
    return v;
}

// ---- on-the-fly pointing ---------------------------------------------------------------------
// boresight (x) detector quaternion with flagged samples -> identity boresight
// (ops_pointing_detector.cpp:33-68)
__device__ __forceinline__ tbm::Quat detector_quat(const double *boresight, int64_t s, bool flagged,
                                                   const tbm::Quat &fp) {
    tbm::Quat b = flagged ? tbm::Quat{0.0, 0.0, 0.0, 1.0} : ld_quat(boresight + 4 * s);
    return tbm::qmul(b, fp);
}

// ---- PCG amplitude arithmetic ----------------------------------------------------------------
// Shared by the separate kernels (k_pcg_direction, k_bx_prescale) and the fused one
// (k_pcg_direction_prescale), which must leave the same bits.
// next search direction: proposal *= beta; proposal += precond
__device__ __forceinline__ double pcg_direction(double d, double beta, double s) {
    return d * beta + s;
}
// one detector's entry of the prescaled amplitudes: {a w, w}, zeros for a flagged baseline
__device__ __forceinline__ double2 bx_scaled(bool good, double a, double w) {
    return make_double2(good ? a * w : 0.0, good ? w : 0.0);
}

} // namespace tbd
