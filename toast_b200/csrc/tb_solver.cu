// tb_solver.cu -- the per-PCG-iteration destriper passes, fused.
//
// One SolverLHS.apply of the reference (ops/mapmaker_solve.py:342-506) runs, per observation,
//   TemplateMatrix.add_to_signal -> [PixelsHealpix, StokesWeights] -> BuildNoiseWeighted
//   ... zmap sync, covariance_apply ...
//   add_to_signal -> [pixels, weights] -> ScanMap(subtract) -> NoiseWeight -> project_signal
// as 7-9 separate kernels around a `det_temp` timestream that is zeroed and refilled twice.
// Here each half is ONE kernel and det_temp lives in a register:
//   pass 1 (k_bin)      zmap[pix] += (F a)[s] * w_det * weights[s]
//   pass 2 (k_project)  out[amp(s)] += w_det * ((F a)[s] - sum_k weights[s,k] * map[pix,k])
// With stored pointing a pass streams 33 B per det-sample (pixel 8 + weights 24 + flag 1); with
// REGEN the pointing is recomputed from the boresight in registers and only the flag byte is read.
#include <type_traits>

#include "tb_device.cuh"
#include "tb_pixelise.cuh"
#include "tb_runtime.cuh"

using namespace tbd;

#include "tb_obs.cuh"

namespace {

struct ObsDev {
    Views V;
    int64_t n_det, n_samp;
    const int64_t *amp_view_off, *amp_offsets, *g2l;
    const double *fp, *cal, *eta, *gamma, *det_scale;
    double inv_step, inv_nps;
    int64_t n_pix_submap;
    tbm::PixCtx ctx; // HEALPix observations
    tbw::Wcs wcs;    // WCS observations
    double U_sign;
    const double *boresight;
    const uint8_t *shared_flags;
    uint8_t shared_mask;
    const uint8_t *solver_flags;
    uint8_t solver_mask;
    const int64_t *pixels;
    const double *weights;
    const double *hwp;
    const int32_t *lpix;
    const double2 *wqu;
    const int2 *lpp;
    const double2 *pair_rot;
    const int4 *xrec;
    const double2 *xqu;
    const int4 *xblocks;
    int x_paired;
};

__device__ unsigned long long g_exact_count_solver = 0ull;

#ifndef TB_BIN_RUN_CAP
#define TB_BIN_RUN_CAP 8
#endif
constexpr int kBinRunCap = TB_BIN_RUN_CAP; // see find_runs<CAP>

// pixel + weights of one sample, either streamed from HBM or regenerated from the boresight with
// the pixelisation policy PIX (tb_pixelise.cuh: the device function tb_pointing_fused[_wcs] runs).
// NNZ = 1: the intensity weight alone (stored [n_det, n_samp], or cal[det] as
// ops_stokes_weights.cpp's I mode sets it); w1 = w2 = 0.
template <bool REGEN, class PIX, int NNZ>
__device__ __forceinline__ void sample_pointing(const ObsDev &o, int det, int64_t s, bool need,
                                                int64_t &pix, double &w0, double &w1, double &w2,
                                                int &n_exact) {
    if (!REGEN) {
        int64_t i = (int64_t)det * o.n_samp + s;
        pix = ld_stream(o.pixels + i);
        if constexpr (NNZ == 1) {
            w0 = ld_stream(o.weights + i);
            w1 = w2 = 0.0;
        } else {
            const double *w = o.weights + 3 * i;
            w0 = ld_stream(w);
            w1 = ld_stream(w + 1);
            w2 = ld_stream(w + 2);
        }
    } else {
        pix = -1;
        w0 = w1 = w2 = 0.0;
        bool bad = o.shared_flags ? ((__ldg(o.shared_flags + s) & o.shared_mask) != 0) : false;
        if (bad || !need) return;
        tbm::Quat f = ld_quat(o.fp + 4 * det);
        tbm::Quat q = tbm::qmul(ld_quat(o.boresight + 4 * s), f);
        if constexpr (std::is_same_v<typename PIX::Geom, tbw::Wcs>) {
            pix = PIX::pixel(o.wcs, q, n_exact);
        } else {
            pix = PIX::pixel(o.ctx, q, n_exact);
        }
        if constexpr (NNZ == 1) {
            w0 = __ldg(o.cal + det);
            return;
        }
        double cal = __ldg(o.cal + det), eta = __ldg(o.eta + det);
        if (o.hwp) {
            tbm::stokes_iqu<true>(q, cal, eta, o.U_sign, __ldg(o.gamma + det), __ldg(o.hwp + s), w0,
                                  w1, w2);
        } else {
            tbm::stokes_iqu<false>(q, cal, eta, o.U_sign, 0.0, 0.0, w0, w1, w2);
        }
    }
}

#define TBS_TILE_LOOP(o)                                                                   \
    TileId _tile = tile_of_block(blockIdx.x, (o).n_det);                                   \
    const int det = _tile.det;                                                             \
    const int lane = threadIdx.x & 31;                                                     \
    ViewCursor _vc = view_cursor((o).V, _tile.t0 + threadIdx.x);                           \
    _Pragma("unroll") for (int _k = 0; _k < kPerThread; ++_k)

#define TBS_COORDS(o)                                                                      \
    int64_t _t = _tile.t0 + (int64_t)_k * kThreads + threadIdx.x;                          \
    bool valid = _t < (o).V.total;                                                         \
    int view = 0;                                                                          \
    int64_t off = 0, s = 0;                                                                \
    if (valid) {                                                                           \
        view_seek((o).V, _vc, _t);                                                         \
        view = _vc.view;                                                                   \
        off = _t - _vc.beg;                                                                \
        s = _vc.first + off;                                                               \
    }

// ---- pass 1: template -> timestream -> noise-weighted map -------------------------------------
// FROM_SIGNAL: bin a stored timestream instead of the template amplitudes (RHS / final BinMap).
// NNZ: map values per pixel, 3 (I, Q, U) or 1 (intensity).
#ifndef TB_REGEN_CTAS
#define TB_REGEN_CTAS 4
#endif
template <bool REGEN, class PIX, bool FROM_SIGNAL, int NNZ>
__global__ void __launch_bounds__(kThreads, REGEN ? TB_REGEN_CTAS : 6)
k_bin(ObsDev o, const double *__restrict__ amps, const uint8_t *__restrict__ aflags,
      const double *__restrict__ signal, double *__restrict__ zmap) {
    int n_exact = 0;
    TBS_TILE_LOOP(o) {
        TBS_COORDS(o)
        int64_t key = -1;
        double z0 = 0.0, z1 = 0.0, z2 = 0.0;
        if (valid) {
            int64_t i = (int64_t)det * o.n_samp + s;
            bool ok = o.solver_flags ? ((ld_stream(o.solver_flags + i) & o.solver_mask) == 0) : true;
            double tod = 0.0;
            if (FROM_SIGNAL) {
                if (ok) tod = ld_stream(signal + i);
            } else {
                int64_t amp = __ldg(o.amp_offsets + det) + __ldg(o.amp_view_off + view) +
                              fast_div(off, o.inv_step);
                if (__ldg(aflags + amp) == 0) tod = __ldg(amps + amp);
            }
            int64_t pix;
            double w0, w1, w2;
            sample_pointing<REGEN, PIX, NNZ>(o, det, s, ok, pix, w0, w1, w2, n_exact);
            if (ok && pix >= 0) {
                int64_t gsm = fast_div(pix, o.inv_nps);
                key = __ldg(o.g2l + gsm) * o.n_pix_submap + (pix - gsm * o.n_pix_submap);
                double sd = tod * __ldg(o.det_scale + det);
                z0 = sd * w0;
                z1 = sd * w1;
                z2 = sd * w2;
            }
        }
        Runs r = find_runs<kBinRunCap>(key, lane);
        z0 = seg_sum<kBinRunCap>(z0, r);
        if constexpr (NNZ == 3) {
            z1 = seg_sum<kBinRunCap>(z1, r);
            z2 = seg_sum<kBinRunCap>(z2, r);
        }
        if (r.is_tail && key >= 0) {
            double *z = zmap + key * NNZ;
            atomicAdd(z, z0);
            if constexpr (NNZ == 3) {
                atomicAdd(z + 1, z1);
                atomicAdd(z + 2, z2);
            }
        }
    }
    if (REGEN && n_exact) atomicAdd(&g_exact_count_solver, (unsigned long long)n_exact);
}

// ---- pass 2: (template - scanned map) -> noise weight -> template projection ------------------
template <bool REGEN, class PIX, bool FROM_SIGNAL, int NNZ>
__global__ void __launch_bounds__(kThreads, REGEN ? TB_REGEN_CTAS : 6)
k_project(ObsDev o, const double *__restrict__ amps, const uint8_t *__restrict__ aflags,
          const double *__restrict__ signal, const double *__restrict__ binned,
          double *__restrict__ amps_out) {
    int n_exact = 0;
    TBS_TILE_LOOP(o) {
        TBS_COORDS(o)
        int64_t key = -1;
        double v = 0.0;
        if (valid) {
            int64_t i = (int64_t)det * o.n_samp + s;
            int64_t amp = __ldg(o.amp_offsets + det) + __ldg(o.amp_view_off + view) +
                          fast_div(off, o.inv_step);
            bool amp_ok = __ldg(aflags + amp) == 0;
            bool ok = o.solver_flags ? ((ld_stream(o.solver_flags + i) & o.solver_mask) == 0) : true;
            if (amp_ok) key = amp;
            // flagged samples contribute exactly 0 (template_offset.cpp:312-321), so nothing
            // else needs to be read for them
            bool need = amp_ok && ok;
            double tod = 0.0;
            if (FROM_SIGNAL) {
                if (need) tod = ld_stream(signal + i);
            } else {
                if (amp_ok) tod = __ldg(amps + amp);
            }
            int64_t pix;
            double w0, w1, w2;
            sample_pointing<REGEN, PIX, NNZ>(o, det, s, need, pix, w0, w1, w2, n_exact);
            if (need) {
                if (pix >= 0) {
                    int64_t gsm = fast_div(pix, o.inv_nps);
                    const double *m = binned + NNZ * (__ldg(o.g2l + gsm) * o.n_pix_submap +
                                                      (pix - gsm * o.n_pix_submap));
                    double sc = 0.0; // ops_scan_map.cpp:59-64
                    sc += w0 * __ldg(m);
                    if constexpr (NNZ == 3) {
                        sc += w1 * __ldg(m + 1);
                        sc += w2 * __ldg(m + 2);
                    }
                    tod -= sc;
                }
                v = tod * __ldg(o.det_scale + det);
            }
        }
        Runs r = find_runs(key, lane);
        v = seg_sum(v, r);
        if (r.is_tail && key >= 0) atomicAdd(amps_out + key, v);
    }
    if (REGEN && n_exact) atomicAdd(&g_exact_count_solver, (unsigned long long)n_exact);
}

// =================================================================================================
// Compact solver pointing.
//
// The pointing is static across PCG iterations, so the solver keeps a derived copy that is
// cheaper to stream than the operator-facing (int64 pixel, 3 x f64 weight, u8 flag) = 33 B:
//   lpix  int32   local pixel index into the map (global2local and the flag test folded in):
//                 >= 0 good sample; -1 flagged (contributes nothing); -2 unflagged but off the
//                 map (pass 2 keeps the template value, nothing is scanned)
//   wqu   double2 the Q and U weights, bit-identical copies; the I weight is the per-detector
//                 constant cal[det] (ops_stokes_weights.cpp:99,130), verified while packing
// = 20 B per det-sample, and both arrays are read with perfectly coalesced LDG.32 / LDG.128
// (5 L1 wavefronts per warp instead of ~22 for the 24-byte-stride weight rows).
// =================================================================================================
__device__ unsigned int g_pack_mismatch = 0u;

// NNZ = 1: intensity weights [n_det, n_samp]; only lpix is written (the 4-byte form)
template <int NNZ>
__global__ void __launch_bounds__(kThreads)
k_pack_pointing(ObsDev o, int32_t *__restrict__ lpix, double2 *__restrict__ wqu) {
    const int64_t total = o.n_det * o.n_samp;
    unsigned bad = 0;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * kThreads) {
        int det = (int)(i / o.n_samp);
        int64_t pix = ld_stream(o.pixels + i);
        double w0, w1 = 0.0, w2 = 0.0;
        if constexpr (NNZ == 1) {
            w0 = ld_stream(o.weights + i);
        } else {
            const double *w = o.weights + 3 * i;
            w0 = ld_stream(w);
            w1 = ld_stream(w + 1);
            w2 = ld_stream(w + 2);
        }
        bool ok = o.solver_flags ? ((ld_stream(o.solver_flags + i) & o.solver_mask) == 0) : true;
        int32_t lp = -1;
        if (ok) {
            lp = -2;
            if (pix >= 0) {
                int64_t gsm = fast_div(pix, o.inv_nps);
                int64_t lsm = __ldg(o.g2l + gsm);
                if (lsm >= 0) {
                    lp = (int32_t)(lsm * o.n_pix_submap + (pix - gsm * o.n_pix_submap));
                    if (w0 != __ldg(o.cal + det)) bad = 1;
                }
            }
        }
        lpix[i] = lp;
        if constexpr (NNZ == 3) wqu[i] = make_double2(w1, w2);
    }
    if (bad) atomicOr(&g_pack_mismatch, 1u);
}

// =================================================================================================
// Detector-pair LHS passes.
//
// Focalplanes hold polarisation pairs: detectors 2p and 2p+1 share a line of sight, so at every
// sample they fall in the same pixel.  One thread therefore handles sample s of BOTH rows of a
// pair: when the two local pixels coincide their noise-weighted contributions are added in
// registers and ONE run / RED triple (pass 1) or ONE map gather (pass 2) serves both detectors,
// which halves the scattered map traffic that limits these passes.  Nothing is assumed: rows
// whose pixels differ (unpaired layouts, pixel-boundary rounding) take a second reduction stream
// that costs nothing when no lane of the warp needs it.
// =================================================================================================
#ifndef TB_PAIR_CTAS
#define TB_PAIR_CTAS 8
#endif
template <bool PASS2>
__global__ void __launch_bounds__(kThreads, TB_PAIR_CTAS)
k_lhs_pair(ObsDev o, int64_t n_pair, const double *__restrict__ amps,
           const uint8_t *__restrict__ aflags, const double *__restrict__ binned,
           double *__restrict__ out) {
    TileId _tile = tile_of_block(blockIdx.x, n_pair);
    const int d0 = 2 * _tile.det;
    const bool has1 = (d0 + 1) < o.n_det;
    const int d1 = has1 ? d0 + 1 : d0;
    const int lane = threadIdx.x & 31;
    const double scale0 = __ldg(o.det_scale + d0), scale1 = __ldg(o.det_scale + d1);
    const double c0 = __ldg(o.cal + d0), c1 = __ldg(o.cal + d1);
    const int64_t ao0 = __ldg(o.amp_offsets + d0), ao1 = __ldg(o.amp_offsets + d1);
    ViewCursor vc = view_cursor(o.V, _tile.t0 + threadIdx.x);
#pragma unroll 2
    for (int k = 0; k < kPerThread; ++k) {
        int64_t t = _tile.t0 + (int64_t)k * kThreads + threadIdx.x;
        int64_t keyA = -1, keyB = -1;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0;
        if (t < o.V.total) {
            view_seek(o.V, vc, t);
            const int view = vc.view;
            int64_t off = t - vc.beg;
            int64_t i0 = (int64_t)d0 * o.n_samp + vc.first + off;
            int64_t i1 = i0 + o.n_samp;
            int32_t lp0 = __ldcs(o.lpix + i0);
            double2 wq0 = __ldcs(o.wqu + i0);
            int32_t lp1 = -1;
            double2 wq1 = make_double2(0.0, 0.0);
            if (has1) {
                lp1 = __ldcs(o.lpix + i1);
                wq1 = __ldcs(o.wqu + i1);
            }
            int64_t rel = __ldg(o.amp_view_off + view) + fast_div(off, o.inv_step);
            int64_t amp0 = ao0 + rel, amp1 = ao1 + rel;
            bool ok0 = __ldg(aflags + amp0) == 0;
            bool ok1 = has1 && (__ldg(aflags + amp1) == 0);
            double tod0 = ok0 ? __ldg(amps + amp0) : 0.0;
            double tod1 = ok1 ? __ldg(amps + amp1) : 0.0;
            if (!PASS2) {
                double sd0 = tod0 * scale0, sd1 = tod1 * scale1;
                if (lp0 >= 0) {
                    keyA = lp0;
                    a0 = sd0 * c0;
                    a1 = sd0 * wq0.x;
                    a2 = sd0 * wq0.y;
                }
                if (lp1 >= 0) {
                    if (lp1 == lp0) {
                        a0 += sd1 * c1;
                        a1 += sd1 * wq1.x;
                        a2 += sd1 * wq1.y;
                    } else {
                        keyB = lp1;
                        b0 = sd1 * c1;
                        b1 = sd1 * wq1.x;
                        b2 = sd1 * wq1.y;
                    }
                }
            } else {
                if (ok0) keyA = amp0;
                if (ok1) keyB = amp1;
                bool need0 = ok0 && lp0 != -1, need1 = ok1 && lp1 != -1;
                double m0 = 0.0, m1 = 0.0, m2 = 0.0;
                bool have = false;
                if (need0 && lp0 >= 0) {
                    const double *m = binned + 3 * (int64_t)lp0;
                    m0 = __ldg(m);
                    m1 = __ldg(m + 1);
                    m2 = __ldg(m + 2);
                    have = true;
                    double sc = 0.0; // ops_scan_map.cpp:59-64
                    sc += c0 * m0;
                    sc += wq0.x * m1;
                    sc += wq0.y * m2;
                    tod0 -= sc;
                }
                if (need1 && lp1 >= 0) {
                    if (!(have && lp1 == lp0)) {
                        const double *m = binned + 3 * (int64_t)lp1;
                        m0 = __ldg(m);
                        m1 = __ldg(m + 1);
                        m2 = __ldg(m + 2);
                    }
                    double sc = 0.0;
                    sc += c1 * m0;
                    sc += wq1.x * m1;
                    sc += wq1.y * m2;
                    tod1 -= sc;
                }
                if (need0) a0 = tod0 * scale0;
                if (need1) b0 = tod1 * scale1;
            }
        }
        if (!PASS2) {
            Runs r = find_runs<kBinRunCap>(keyA, lane);
            a0 = seg_sum<kBinRunCap>(a0, r);
            a1 = seg_sum<kBinRunCap>(a1, r);
            a2 = seg_sum<kBinRunCap>(a2, r);
            if (r.is_tail && keyA >= 0) {
                double *z = out + keyA * 3;
                atomicAdd(z, a0);
                atomicAdd(z + 1, a1);
                atomicAdd(z + 2, a2);
            }
            if (__any_sync(0xffffffffu, keyB >= 0)) {
                Runs rb = find_runs<kBinRunCap>(keyB, lane);
                b0 = seg_sum<kBinRunCap>(b0, rb);
                b1 = seg_sum<kBinRunCap>(b1, rb);
                b2 = seg_sum<kBinRunCap>(b2, rb);
                if (rb.is_tail && keyB >= 0) {
                    double *z = out + keyB * 3;
                    atomicAdd(z, b0);
                    atomicAdd(z + 1, b1);
                    atomicAdd(z + 2, b2);
                }
            }
        } else {
            Runs r = find_runs(keyA, lane);
            a0 = seg_sum(a0, r);
            if (r.is_tail && keyA >= 0) atomicAdd(out + keyA, a0);
            if (has1) {
                Runs rb = find_runs(keyB, lane);
                b0 = seg_sum(b0, rb);
                if (rb.is_tail && keyB >= 0) atomicAdd(out + keyB, b0);
            }
        }
    }
}

int g_use_pair = 1; // tb_set_option("pair", 0/1)

// =================================================================================================
// Detector pairs with SHARED weights (12 B per det-sample).
//
// The (Q,U) weights of the two detectors of a polarisation pair are not independent: both are
// eta*cal*(cos, sin) of an angle that differs by a constant (2 x the polariser offset, +4 x the
// gamma offset with a HWP), i.e. (q1,u1) = [[A,-B],[B,A]] (q0,u0) with a per-pair constant
// (A, B) -- (-1, 0) for the usual orthogonal pair.  tb_obs_pack_pointing fits (A, B) from one
// sample and VERIFIES the relation on every in-interval sample of the pair to 1e-13 relative
// (three orders inside the 1e-10 parity bar); only then are these kernels used.  A pair-sample is
// then one 8-byte record (both local pixels) + one 16-byte record (q0,u0): 24 B / 2 det-samples.
// =================================================================================================
__device__ unsigned int g_pair_mismatch = 0u;

__global__ void k_pair_fit(ObsDev o, int64_t n_pair, int64_t s_fit, double2 *__restrict__ rot) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pair) return;
    int64_t d0 = 2 * p, d1 = d0 + 1;
    double A = 0.0, B = 0.0;
    if (d1 < o.n_det) {
        double2 a = o.wqu[d0 * o.n_samp + s_fit], b = o.wqu[d1 * o.n_samp + s_fit];
        double n2 = a.x * a.x + a.y * a.y;
        if (n2 > 0.0) {
            A = (b.x * a.x + b.y * a.y) / n2;
            B = (b.y * a.x - b.x * a.y) / n2;
            // orthogonal / parallel pairs: snap to the exact rotation
            if (fabs(A - rint(A)) < 1e-14 && fabs(B - rint(B)) < 1e-14) {
                A = rint(A);
                B = rint(B);
            }
        }
    }
    rot[p] = make_double2(A, B);
}

__global__ void __launch_bounds__(kThreads)
k_pack_pairs(ObsDev o, int64_t n_pair, const double2 *__restrict__ rot, int2 *__restrict__ lpp) {
    const int64_t total = n_pair * o.V.total;
    unsigned bad = 0;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * kThreads) {
        int64_t p = i / o.V.total;
        int64_t t = i - p * o.V.total;
        int view = o.V.n_view > 1 ? find_view(o.V, t) : 0;
        int64_t s = __ldg(o.V.first + view) + (t - __ldg(o.V.prefix + view));
        int64_t d0 = 2 * p, d1 = d0 + 1;
        int64_t i0 = d0 * o.n_samp + s;
        int2 lp = make_int2(__ldcs(o.lpix + i0), -1);
        if (d1 < o.n_det) {
            int64_t i1 = i0 + o.n_samp;
            lp.y = __ldcs(o.lpix + i1);
            double2 a = __ldcs(o.wqu + i0), b = __ldcs(o.wqu + i1), r = __ldg(rot + p);
            double ex = b.x - (r.x * a.x - r.y * a.y);
            double ey = b.y - (r.y * a.x + r.x * a.y);
            double n2 = b.x * b.x + b.y * b.y;
            if (!(ex * ex + ey * ey <= 1e-26 * n2)) bad = 1;
        }
        lpp[p * o.n_samp + s] = lp;
    }
    if (bad) atomicOr(&g_pair_mismatch, 1u);
}

#ifndef TB_PAIRW_CTAS
#define TB_PAIRW_CTAS 8
#endif
template <bool PASS2>
__global__ void __launch_bounds__(kThreads, TB_PAIRW_CTAS)
k_lhs_pairw(ObsDev o, int64_t n_pair, const double *__restrict__ amps,
            const uint8_t *__restrict__ aflags, const double *__restrict__ binned,
            double *__restrict__ out) {
    TileId _tile = tile_of_block(blockIdx.x, n_pair);
    const int d0 = 2 * _tile.det;
    const bool has1 = (d0 + 1) < o.n_det;
    const int d1 = has1 ? d0 + 1 : d0;
    const int lane = threadIdx.x & 31;
    const double scale0 = __ldg(o.det_scale + d0), scale1 = __ldg(o.det_scale + d1);
    const double c0 = __ldg(o.cal + d0), c1 = __ldg(o.cal + d1);
    const double2 rot = __ldg(o.pair_rot + _tile.det);
    const int64_t ao0 = __ldg(o.amp_offsets + d0), ao1 = __ldg(o.amp_offsets + d1);
    ViewCursor vc = view_cursor(o.V, _tile.t0 + threadIdx.x);
#pragma unroll 2
    for (int k = 0; k < kPerThread; ++k) {
        int64_t t = _tile.t0 + (int64_t)k * kThreads + threadIdx.x;
        int64_t keyA = -1, keyB = -1;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0;
        if (t < o.V.total) {
            view_seek(o.V, vc, t);
            const int view = vc.view;
            int64_t off = t - vc.beg;
            int64_t ip = (int64_t)_tile.det * o.n_samp + vc.first + off;
            int64_t i0 = ip + (int64_t)_tile.det * o.n_samp; // row 2p of the per-detector array
            int2 lp = __ldcs(o.lpp + ip);
            double2 wq0 = __ldcs(o.wqu + i0);
            const int32_t lp0 = lp.x, lp1 = lp.y;
            double2 wq1 = make_double2(rot.x * wq0.x - rot.y * wq0.y, rot.y * wq0.x + rot.x * wq0.y);
            int64_t rel = __ldg(o.amp_view_off + view) + fast_div(off, o.inv_step);
            int64_t amp0 = ao0 + rel, amp1 = ao1 + rel;
            bool ok0 = __ldg(aflags + amp0) == 0;
            bool ok1 = has1 && (__ldg(aflags + amp1) == 0);
            double tod0 = ok0 ? __ldg(amps + amp0) : 0.0;
            double tod1 = ok1 ? __ldg(amps + amp1) : 0.0;
            if (!PASS2) {
                double sd0 = tod0 * scale0, sd1 = tod1 * scale1;
                if (lp0 >= 0) {
                    keyA = lp0;
                    a0 = sd0 * c0;
                    a1 = sd0 * wq0.x;
                    a2 = sd0 * wq0.y;
                }
                if (lp1 >= 0) {
                    if (lp1 == lp0) {
                        a0 += sd1 * c1;
                        a1 += sd1 * wq1.x;
                        a2 += sd1 * wq1.y;
                    } else {
                        keyB = lp1;
                        b0 = sd1 * c1;
                        b1 = sd1 * wq1.x;
                        b2 = sd1 * wq1.y;
                    }
                }
            } else {
                if (ok0) keyA = amp0;
                if (ok1) keyB = amp1;
                bool need0 = ok0 && lp0 != -1, need1 = ok1 && lp1 != -1;
                double m0 = 0.0, m1 = 0.0, m2 = 0.0;
                bool have = false;
                if (need0 && lp0 >= 0) {
                    const double *m = binned + 3 * (int64_t)lp0;
                    m0 = __ldg(m);
                    m1 = __ldg(m + 1);
                    m2 = __ldg(m + 2);
                    have = true;
                    double sc = 0.0; // ops_scan_map.cpp:59-64
                    sc += c0 * m0;
                    sc += wq0.x * m1;
                    sc += wq0.y * m2;
                    tod0 -= sc;
                }
                if (need1 && lp1 >= 0) {
                    if (!(have && lp1 == lp0)) {
                        const double *m = binned + 3 * (int64_t)lp1;
                        m0 = __ldg(m);
                        m1 = __ldg(m + 1);
                        m2 = __ldg(m + 2);
                    }
                    double sc = 0.0;
                    sc += c1 * m0;
                    sc += wq1.x * m1;
                    sc += wq1.y * m2;
                    tod1 -= sc;
                }
                if (need0) a0 = tod0 * scale0;
                if (need1) b0 = tod1 * scale1;
            }
        }
        if (!PASS2) {
            Runs r = find_runs<kBinRunCap>(keyA, lane);
            a0 = seg_sum<kBinRunCap>(a0, r);
            a1 = seg_sum<kBinRunCap>(a1, r);
            a2 = seg_sum<kBinRunCap>(a2, r);
            if (r.is_tail && keyA >= 0) {
                double *z = out + keyA * 3;
                atomicAdd(z, a0);
                atomicAdd(z + 1, a1);
                atomicAdd(z + 2, a2);
            }
            if (__any_sync(0xffffffffu, keyB >= 0)) {
                Runs rb = find_runs<kBinRunCap>(keyB, lane);
                b0 = seg_sum<kBinRunCap>(b0, rb);
                b1 = seg_sum<kBinRunCap>(b1, rb);
                b2 = seg_sum<kBinRunCap>(b2, rb);
                if (rb.is_tail && keyB >= 0) {
                    double *z = out + keyB * 3;
                    atomicAdd(z, b0);
                    atomicAdd(z + 1, b1);
                    atomicAdd(z + 2, b2);
                }
            }
        } else {
            Runs r = find_runs(keyA, lane);
            a0 = seg_sum(a0, r);
            if (r.is_tail && keyA >= 0) atomicAdd(out + keyA, a0);
            if (has1) {
                Runs rb = find_runs(keyB, lane);
                b0 = seg_sum(b0, rb);
                if (rb.is_tail && keyB >= 0) atomicAdd(out + keyB, b0);
            }
        }
    }
}

int g_use_pairw = 1; // tb_set_option("pairw", 0/1)

// =================================================================================================
// Crossing list.
//
// While a detector crosses one pixel its samples share the pixel AND (almost always) the baseline
// amplitude, so their contributions differ only through the (Q,U) weights -- and those enter both
// passes LINEARLY:
//   pass 1  zmap[pix] += sum_s  a w_d (cal, q_s, u_s)        = a w_d (n cal, Q, U)
//   pass 2  out[amp]  += sum_s  w_d (a - (cal, q_s, u_s).m)  = w_d (n a - (n cal, Q, U).m)
// with n the number of samples of the run and (Q, U) = sum_s (q_s, u_s).  The pointing is static
// across PCG iterations, so tb_obs_pack_pointing collapses every run of consecutive samples
// with the same (pixel of detector 0, pixel of detector 1, baseline) into ONE 32-byte record
// {lp0, lp1, n, amp_rel | Q, U}; runs are cut at 32-sample boundaries so that a warp builds its
// records alone.  Both LHS passes then stream records instead of samples: 32 B per crossing of a
// detector PAIR -- 6.7 B / det-sample at the 2.4 samples per crossing of the nside-2048
// satellite scan, < 2 B / det-sample for ground scans -- with no segmented reduction left in
// pass 1 (adjacent records hit different pixels) and one map gather per crossing in pass 2.
// Flags are part of the run state (a flagged sample has lp = -1), runs with both detectors
// flagged are dropped.  Sums are re-associated: 1e-16 relative, inside the 1e-10 parity bar.
// =================================================================================================
constexpr int kXPer = 4;
constexpr int kXTile = kThreads * kXPer; // records per CTA

struct XState {
    int32_t lp0, lp1, amp_rel;
    double2 wq;
};

// state of flat sample t of row `row` (a detector pair when paired, else one detector);
// NNZ = 1 reads no (Q, U) weights
template <int NNZ>
__device__ __forceinline__ XState x_state(const ObsDev &o, int paired, int64_t row, int64_t t) {
    XState st;
    st.lp0 = st.lp1 = -1;
    st.amp_rel = -1;
    st.wq = make_double2(0.0, 0.0);
    if (t >= o.V.total) return st;
    int view = o.V.n_view > 1 ? find_view(o.V, t) : 0;
    int64_t off = t - __ldg(o.V.prefix + view);
    int64_t s = __ldg(o.V.first + view) + off;
    int64_t d0 = paired ? 2 * row : row;
    int64_t i0 = d0 * o.n_samp + s;
    st.lp0 = __ldcs(o.lpix + i0);
    if constexpr (NNZ == 3) st.wq = __ldcs(o.wqu + i0);
    if (paired && d0 + 1 < o.n_det) st.lp1 = __ldcs(o.lpix + i0 + o.n_samp);
    st.amp_rel = (int32_t)(__ldg(o.amp_view_off + view) + fast_div(off, o.inv_step));
    return st;
}

// FILL = false: counts[chunk] = records of the chunk; FILL = true: write them at base[chunk].
// NNZ = 1: intensity records (xrec only, no xqu).  Its counting pass on paired rows also adds
// the records whose two detectors fall in different pixels (each takes two entries of the
// block-ordered list) to counts[n_chunks], read as an unsigned counter.
template <bool FILL, int NNZ>
__global__ void __launch_bounds__(kThreads)
k_xbuild(ObsDev o, int paired, int64_t n_rows, int64_t chunks_per_row, int32_t *__restrict__ counts,
         const int64_t *__restrict__ base, int4 *__restrict__ xrec, double2 *__restrict__ xqu) {
    const int lane = threadIdx.x & 31;
    const int64_t n_chunks = n_rows * chunks_per_row;
    const int64_t warp0 = ((int64_t)blockIdx.x * kThreads + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * kThreads) >> 5;
    for (int64_t c = warp0; c < n_chunks; c += n_warps) {
        int64_t row = c / chunks_per_row;
        int64_t t = (c - row * chunks_per_row) * 32 + lane;
        XState st = x_state<NNZ>(o, paired, row, t);
        int32_t p0 = __shfl_up_sync(0xffffffffu, st.lp0, 1);
        int32_t p1 = __shfl_up_sync(0xffffffffu, st.lp1, 1);
        int32_t pa = __shfl_up_sync(0xffffffffu, st.amp_rel, 1);
        bool head = (lane == 0) || p0 != st.lp0 || p1 != st.lp1 || pa != st.amp_rel;
        bool keep = !(st.lp0 == -1 && st.lp1 == -1);
        unsigned heads = __ballot_sync(0xffffffffu, head);
        unsigned kept_heads = __ballot_sync(0xffffffffu, head && keep);
        if (!FILL) {
            if (lane == 0) counts[c] = __popc(kept_heads);
            if constexpr (NNZ == 1) {
                if (paired) {
                    const unsigned split = __ballot_sync(
                        0xffffffffu, head && st.lp0 >= 0 && st.lp1 >= 0 && st.lp0 != st.lp1);
                    if (lane == 0 && split)
                        atomicAdd(reinterpret_cast<unsigned int *>(counts + n_chunks),
                                  (unsigned int)__popc(split));
                }
            }
            continue;
        }
        unsigned upto = heads & (0xffffffffu >> (31 - lane));
        int head_lane = 31 - __clz(upto);
        Runs r;
        r.dist = lane - head_lane;
        r.is_tail = (((heads >> 1) | 0x80000000u) >> lane) & 1u;
        double Q = 0.0, U = 0.0;
        if constexpr (NNZ == 3) {
            Q = seg_sum(st.wq.x, r);
            U = seg_sum(st.wq.y, r);
        }
        if (r.is_tail && keep) {
            int64_t idx = base[c] + __popc(kept_heads & ((1u << head_lane) - 1u));
            xrec[idx] = make_int4(st.lp0, st.lp1, (r.dist + 1) | ((int)row << 8), st.amp_rel);
            if constexpr (NNZ == 3) xqu[idx] = make_double2(Q, U);
        }
    }
}

int g_use_x = 1; // tb_set_option("crossings", 0/1)

#ifndef TB_X_CTAS
#define TB_X_CTAS 8
#endif
template <bool PASS2>
__global__ void __launch_bounds__(kThreads, TB_X_CTAS)
k_lhs_x(ObsDev o, const double *__restrict__ amps, const uint8_t *__restrict__ aflags,
        const double *__restrict__ binned, double *__restrict__ out) {
    const int4 blk = __ldg(o.xblocks + blockIdx.x);
    const int row = blk.x;
    const int d0 = o.x_paired ? 2 * row : row;
    const bool has1 = o.x_paired && (d0 + 1) < o.n_det;
    const int d1 = has1 ? d0 + 1 : d0;
    const int lane = threadIdx.x & 31;
    const double scale0 = __ldg(o.det_scale + d0), scale1 = __ldg(o.det_scale + d1);
    const double c0 = __ldg(o.cal + d0), c1 = __ldg(o.cal + d1);
    double2 rot = make_double2(0.0, 0.0);
    if (has1) rot = __ldg(o.pair_rot + row);
    const int64_t ao0 = __ldg(o.amp_offsets + d0), ao1 = __ldg(o.amp_offsets + d1);
#pragma unroll 2
    for (int k = 0; k < kXPer; ++k) {
        const int i = blk.y + k * kThreads + threadIdx.x;
        int32_t lp0 = -1, lp1 = -1, arel = -1;
        bool ok0 = false, ok1 = false;
        double a0 = 0.0, a1 = 0.0, a2 = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0;
        if (i < blk.z) {
            const int4 r = __ldcs(o.xrec + i);
            const double2 qu = __ldcs(o.xqu + i);
            lp0 = r.x;
            lp1 = r.y;
            arel = r.w;
            const double n = (double)(r.z & 0xFF); // (row index in the upper bits)
            const int64_t amp0 = ao0 + arel, amp1 = ao1 + arel;
            ok0 = __ldg(aflags + amp0) == 0;
            ok1 = has1 && (__ldg(aflags + amp1) == 0);
            const double tod0 = ok0 ? __ldg(amps + amp0) : 0.0;
            const double tod1 = ok1 ? __ldg(amps + amp1) : 0.0;
            const double2 qu1 = make_double2(rot.x * qu.x - rot.y * qu.y, rot.y * qu.x + rot.x * qu.y);
            if (!PASS2) {
                const double sd0 = tod0 * scale0, sd1 = tod1 * scale1;
                if (lp0 >= 0) {
                    a0 = sd0 * (c0 * n);
                    a1 = sd0 * qu.x;
                    a2 = sd0 * qu.y;
                }
                if (lp1 >= 0) {
                    if (lp1 == lp0) {
                        a0 += sd1 * (c1 * n);
                        a1 += sd1 * qu1.x;
                        a2 += sd1 * qu1.y;
                        lp1 = -1;
                    } else {
                        b0 = sd1 * (c1 * n);
                        b1 = sd1 * qu1.x;
                        b2 = sd1 * qu1.y;
                    }
                }
            } else {
                const bool need0 = ok0 && lp0 != -1, need1 = ok1 && lp1 != -1;
                double m0 = 0.0, m1 = 0.0, m2 = 0.0;
                bool have = false;
                double v0 = n * tod0, v1 = n * tod1;
                if (need0 && lp0 >= 0) {
                    const double *m = binned + 3 * (int64_t)lp0;
                    m0 = __ldg(m);
                    m1 = __ldg(m + 1);
                    m2 = __ldg(m + 2);
                    have = true;
                    double sc = 0.0;
                    sc += (c0 * n) * m0;
                    sc += qu.x * m1;
                    sc += qu.y * m2;
                    v0 -= sc;
                }
                if (need1 && lp1 >= 0) {
                    if (!(have && lp1 == lp0)) {
                        const double *m = binned + 3 * (int64_t)lp1;
                        m0 = __ldg(m);
                        m1 = __ldg(m + 1);
                        m2 = __ldg(m + 2);
                    }
                    double sc = 0.0;
                    sc += (c1 * n) * m0;
                    sc += qu1.x * m1;
                    sc += qu1.y * m2;
                    v1 -= sc;
                }
                if (need0) a0 = v0 * scale0;
                if (need1) b0 = v1 * scale1;
            }
        }
        if (!PASS2) {
            if (lp0 >= 0) {
                double *z = out + (int64_t)lp0 * 3;
                atomicAdd(z, a0);
                atomicAdd(z + 1, a1);
                atomicAdd(z + 2, a2);
            }
            if (lp1 >= 0) { // only when the two detectors of the pair fall in different pixels
                double *z = out + (int64_t)lp1 * 3;
                atomicAdd(z, b0);
                atomicAdd(z + 1, b1);
                atomicAdd(z + 2, b2);
            }
        } else {
            // adjacent records share the baseline: one segmented sum per detector, one RED per run
            Runs r = find_runs((int64_t)arel, lane);
            a0 = seg_sum(a0, r);
            if (has1) b0 = seg_sum(b0, r);
            if (r.is_tail && arel >= 0) {
                if (ok0) atomicAdd(out + ao0 + arel, a0);
                if (ok1) atomicAdd(out + ao1 + arel, b0);
            }
        }
    }
}

ObsDev make_dev(const tb_obs *obs, int regen) {
    const tb_obs_desc &d = obs->d;
    ObsDev o;
    o.V = obs->V;
    o.n_det = d.n_det;
    o.n_samp = d.n_samp;
    o.amp_view_off = obs->amp_view_off;
    o.amp_offsets = obs->amp_offsets;
    o.g2l = obs->g2l;
    o.fp = obs->fp;
    o.cal = obs->cal;
    o.eta = obs->eta;
    o.gamma = obs->gamma;
    o.det_scale = obs->det_scale;
    o.inv_step = 1.0 / (double)d.step_length;
    o.inv_nps = 1.0 / (double)d.n_pix_submap;
    o.n_pix_submap = d.n_pix_submap;
    if (obs->is_wcs) {
        o.ctx = tbm::PixCtx{};
        o.wcs = obs->wcs;
    } else {
        o.ctx = tbm::make_pix_ctx(d.nside, 1.0);
        o.wcs = tbw::Wcs{};
    }
    o.U_sign = d.IAU ? -1.0 : 1.0;
    o.boresight = d.boresight;
    o.shared_flags = d.shared_flags;
    o.shared_mask = d.shared_flag_mask;
    o.solver_flags = d.solver_flags;
    o.solver_mask = d.solver_flag_mask;
    o.pixels = d.pixels;
    o.weights = d.weights;
    o.hwp = d.hwp;
    o.lpix = obs->lpix;
    o.wqu = obs->wqu;
    o.lpp = obs->lpp;
    o.pair_rot = obs->pair_rot;
    o.xrec = obs->xrec;
    o.xqu = obs->xqu;
    o.xblocks = obs->xblocks;
    o.x_paired = obs->x_paired;
    if (regen) {
        TB_REQUIRE(d.boresight != nullptr && d.focalplane != nullptr,
                   "regen needs boresight and focalplane");
    } else {
        TB_REQUIRE(d.pixels != nullptr && d.weights != nullptr,
                   "stored-pointing pass needs pixels and weights");
    }
    return o;
}

inline int64_t obs_blocks(const tb_obs *obs) {
    int64_t tiles = (obs->V.total + kTile - 1) / kTile;
    return tiles * obs->d.n_det;
}

#define TBS_LAUNCH(kernel, nb, stream, ...)                                                \
    do {                                                                                   \
        if ((nb) > 0) {                                                                    \
            TB_REQUIRE((nb) < 2147483647LL, "grid too large");                             \
            kernel<<<(unsigned)(nb), kThreads, 0, (cudaStream_t)(stream)>>>(__VA_ARGS__);  \
            TB_CUDA(cudaGetLastError());                                                   \
            tbr::count_launch();                                                           \
        }                                                                                  \
    } while (0)

// the per-sample pass 1 (k_bin) with stored or regenerated pointing
template <bool FROM_SIGNAL, int NNZ>
void launch_bin_samples(const tb_obs *obs, const ObsDev &o, const double *amps,
                        const uint8_t *aflags, const double *signal, double *zmap, int regen,
                        void *stream) {
    int64_t nb = obs_blocks(obs);
    if (!regen) {
        auto k = k_bin<false, tbp::PixHealpix<true>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, zmap);
    } else if (obs->is_wcs) {
        auto k = k_bin<true, tbp::PixWcs, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, zmap);
    } else if (obs->d.nest) {
        auto k = k_bin<true, tbp::PixHealpix<true>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, zmap);
    } else {
        auto k = k_bin<true, tbp::PixHealpix<false>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, zmap);
    }
}

// the per-sample pass 2 (k_project) with stored or regenerated pointing
template <bool FROM_SIGNAL, int NNZ>
void launch_project_samples(const tb_obs *obs, const ObsDev &o, const double *amps,
                            const uint8_t *aflags, const double *signal, const double *binned,
                            double *out, int regen, void *stream) {
    int64_t nb = obs_blocks(obs);
    if (!regen) {
        auto k = k_project<false, tbp::PixHealpix<true>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, binned, out);
    } else if (obs->is_wcs) {
        auto k = k_project<true, tbp::PixWcs, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, binned, out);
    } else if (obs->d.nest) {
        auto k = k_project<true, tbp::PixHealpix<true>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, binned, out);
    } else {
        auto k = k_project<true, tbp::PixHealpix<false>, FROM_SIGNAL, NNZ>;
        TBS_LAUNCH(k, nb, stream, o, amps, aflags, signal, binned, out);
    }
}

// Intensity observations always take the per-sample kernels here: the crossing-list and
// detector-pair kernels are IQU-only.
template <bool FROM_SIGNAL>
void launch_bin(const tb_obs *obs, const double *amps, const uint8_t *aflags, const double *signal,
                double *zmap, int regen, void *stream) {
    ObsDev o = make_dev(obs, regen);
    if (obs->nnz == 1) {
        launch_bin_samples<FROM_SIGNAL, 1>(obs, o, amps, aflags, signal, zmap, regen, stream);
    } else if (!regen && !FROM_SIGNAL && g_use_x && o.xrec != nullptr) {
        auto k = k_lhs_x<false>;
        TBS_LAUNCH(k, obs->n_xblocks, stream, o, amps, aflags, nullptr, zmap);
    } else if (!regen && !FROM_SIGNAL && g_use_pair && o.lpix != nullptr) {
        int64_t n_pair = (o.n_det + 1) / 2;
        int64_t nbp = ((o.V.total + kTile - 1) / kTile) * n_pair;
        if (g_use_pairw && o.lpp != nullptr) {
            auto k = k_lhs_pairw<false>;
            TBS_LAUNCH(k, nbp, stream, o, n_pair, amps, aflags, nullptr, zmap);
        } else {
            auto k = k_lhs_pair<false>;
            TBS_LAUNCH(k, nbp, stream, o, n_pair, amps, aflags, nullptr, zmap);
        }
    } else {
        launch_bin_samples<FROM_SIGNAL, 3>(obs, o, amps, aflags, signal, zmap, regen, stream);
    }
}

template <bool FROM_SIGNAL>
void launch_project(const tb_obs *obs, const double *amps, const uint8_t *aflags,
                    const double *signal, const double *binned, double *out, int regen,
                    void *stream) {
    ObsDev o = make_dev(obs, regen);
    if (obs->nnz == 1) {
        launch_project_samples<FROM_SIGNAL, 1>(obs, o, amps, aflags, signal, binned, out, regen,
                                               stream);
    } else if (!regen && !FROM_SIGNAL && g_use_x && o.xrec != nullptr) {
        auto k = k_lhs_x<true>;
        TBS_LAUNCH(k, obs->n_xblocks, stream, o, amps, aflags, binned, out);
    } else if (!regen && !FROM_SIGNAL && g_use_pair && o.lpix != nullptr) {
        int64_t n_pair = (o.n_det + 1) / 2;
        int64_t nbp = ((o.V.total + kTile - 1) / kTile) * n_pair;
        if (g_use_pairw && o.lpp != nullptr) {
            auto k = k_lhs_pairw<true>;
            TBS_LAUNCH(k, nbp, stream, o, n_pair, amps, aflags, binned, out);
        } else {
            auto k = k_lhs_pair<true>;
            TBS_LAUNCH(k, nbp, stream, o, n_pair, amps, aflags, binned, out);
        }
    } else {
        launch_project_samples<FROM_SIGNAL, 3>(obs, o, amps, aflags, signal, binned, out, regen,
                                               stream);
    }
}

// ---- amplitude-vector kernels ------------------------------------------------------------------
constexpr int kRedBlocks = 592; // 4 x 148 SMs
struct RedScratch {
    double *partials = nullptr; // [2 * kRedBlocks]
    unsigned int *counter = nullptr;
};
RedScratch g_red[64];

RedScratch &red_scratch() {
    int dev = 0;
    TB_CUDA(cudaGetDevice(&dev));
    RedScratch &r = g_red[dev & 63];
    if (r.partials == nullptr) {
        TB_CUDA(cudaMalloc(&r.partials, sizeof(double) * 2 * kRedBlocks));
        TB_CUDA(cudaMalloc(&r.counter, sizeof(unsigned int)));
        TB_CUDA(cudaMemset(r.counter, 0, sizeof(unsigned int)));
    }
    return r;
}

__device__ __forceinline__ double block_sum(double v, double *sh) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0) {
        for (int w = 0; w < kThreads / 32; ++w) t += sh[w];
    }
    return t; // valid in thread 0
}

// Deterministic grid reduction: each CTA writes its partial(s); the last CTA to finish adds them
// in index order.  NRED = 1 or 2 results.
template <int NRED>
__device__ __forceinline__ void grid_finish(double p0, double p1, double *partials,
                                            unsigned int *counter, double *out) {
    __shared__ bool last;
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = p0;
        if (NRED == 2) partials[kRedBlocks + blockIdx.x] = p1;
        __threadfence();
        unsigned int done = atomicAdd(counter, 1u);
        last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (last && threadIdx.x < 32) {
        __threadfence();
        for (int r = 0; r < NRED; ++r) {
            double acc = 0.0;
            // fixed order: lane-strided partial sums, then a fixed shuffle tree
            for (unsigned int b = threadIdx.x; b < gridDim.x; b += 32)
                acc += ((volatile double *)partials)[r * kRedBlocks + b];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
            if (threadIdx.x == 0) out[r] = acc;
        }
        if (threadIdx.x == 0) *counter = 0u;
    }
}

__global__ void __launch_bounds__(kThreads)
k_amp_dot(const double *__restrict__ a, const double *__restrict__ b,
          const uint8_t *__restrict__ flags, int64_t n, double *partials, unsigned int *counter,
          double *out) {
    __shared__ double sh[kThreads / 32];
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        if (flags == nullptr || flags[i] == 0) acc += a[i] * b[i];
    }
    double t = block_sum(acc, sh);
    grid_finish<1>(t, 0.0, partials, counter, out);
}

__global__ void __launch_bounds__(kThreads)
k_pcg_update(const double *__restrict__ delta, const double *__restrict__ dq,
             double *__restrict__ x, double *__restrict__ r, const double *__restrict__ d,
             const double *__restrict__ q, double *__restrict__ s,
             const double *__restrict__ var, const uint8_t *__restrict__ flags, int64_t n,
             double *partials, unsigned int *counter, double *sums) {
    __shared__ double sh[kThreads / 32];
    const double alpha = delta[0] / dq[0];
    double rr = 0.0, sr = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        // mapmaker_solve.py:681-694: temp = d * alpha; x += temp; temp = q * alpha; r -= temp
        double xi = x[i] + d[i] * alpha;
        double ri = r[i] - q[i] * alpha;
        x[i] = xi;
        r[i] = ri;
        bool good = flags[i] == 0;
        double si = good ? ri * var[i] : 0.0;
        s[i] = si;
        if (good) {
            rr += ri * ri;
            sr += si * ri;
        }
    }
    double t0 = block_sum(rr, sh);
    double t1 = block_sum(sr, sh);
    grid_finish<2>(t0, t1, partials, counter, sums);
}

__global__ void __launch_bounds__(kThreads)
k_pcg_direction(const double *__restrict__ dnew, const double *__restrict__ dold,
                double *__restrict__ d, const double *__restrict__ s, int64_t n) {
    const double beta = dnew[0] / dold[0];
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        d[i] = d[i] * beta + s[i]; // proposal *= beta; proposal += precond
    }
}

inline int red_grid(int64_t n) {
    int64_t b = (n + kThreads - 1) / kThreads;
    if (b < 1) b = 1;
    if (b > kRedBlocks) b = kRedBlocks;
    return (int)b;
}

// the body of tb_obs_create / tb_obs_create_wcs / tb_obs_create_intensity; `wcs` NULL: a HEALPix
// observation
tb_obs *obs_create(const tb_obs_desc *desc, const tb_wcs_desc *wcs, int nnz) {
    try {
        tbr::require_device();
        TB_REQUIRE(desc != nullptr, "NULL descriptor");
        const tb_obs_desc &d = *desc;
        TB_REQUIRE(d.n_det > 0 && d.n_samp > 0 && d.n_view >= 0, "bad observation shape");
        TB_REQUIRE(d.step_length > 0, "step_length must be positive");
        tbw::Wcs w{};
        if (wcs) {
            w = tbp::wcs_from_desc(wcs);
            TB_REQUIRE(d.n_pix_submap > 0 && d.n_submap * d.n_pix_submap >= w.n_pix,
                       "the submaps do not cover the projection");
        } else {
            TB_REQUIRE(d.nside > 0 && (d.nside & (d.nside - 1)) == 0 && d.nside <= (1 << 24),
                       "nside must be a power of two <= 2^24");
        }
        TB_REQUIRE(d.global2local && d.det_scale && d.amp_offsets && d.n_amp_views && d.intervals,
                   "missing descriptor arrays");
        tb_obs *o = new tb_obs();
        o->d = d;
        o->is_wcs = wcs != nullptr;
        o->wcs = w;
        o->nnz = nnz;
        // pack: int64 [first(nv), prefix(nv+1), amp_view_off(nv), amp_offsets(nd), g2l(ns)]
        //       double [fp(4nd), cal, eta, gamma, det_scale]
        int64_t nv = d.n_view, nd = d.n_det, ns = d.n_submap;
        std::vector<int64_t> ib(3 * nv + 1 + nd + ns);
        int64_t total = 0, acc = 0;
        for (int64_t v = 0; v < nv; ++v) {
            int64_t a = d.intervals[v].first, b = d.intervals[v].last;
            TB_REQUIRE(a >= 0 && b <= d.n_samp, "interval outside [0, n_samp)");
            ib[v] = a;
            ib[nv + v] = total;
            if (b > a) total += b - a;
            ib[2 * nv + 1 + v] = acc;
            acc += d.n_amp_views[v];
        }
        ib[2 * nv] = total;
        for (int64_t i = 0; i < nd; ++i) ib[3 * nv + 1 + i] = d.amp_offsets[i];
        int64_t n_local = 0;
        for (int64_t i = 0; i < ns; ++i) {
            ib[3 * nv + 1 + nd + i] = d.global2local[i];
            if (d.global2local[i] + 1 > n_local) n_local = d.global2local[i] + 1;
        }
        o->n_local_pix = n_local * (int64_t)d.n_pix_submap;
        std::vector<double> db(8 * nd, 0.0);
        for (int64_t i = 0; i < nd; ++i) {
            if (d.focalplane)
                for (int k = 0; k < 4; ++k) db[4 * i + k] = d.focalplane[4 * i + k];
            double eps = d.epsilon ? d.epsilon[i] : 0.0;
            db[4 * nd + i] = d.cal ? d.cal[i] : 1.0;
            db[5 * nd + i] = (1.0 - eps) / (1.0 + eps);
            db[6 * nd + i] = d.gamma ? d.gamma[i] : 0.0;
            db[7 * nd + i] = d.det_scale[i];
        }
        // keep the double block 32-byte aligned: fp quaternions are read as double2
        while ((ib.size() * sizeof(int64_t)) % 32 != 0) ib.push_back(0);
        size_t ibytes = ib.size() * sizeof(int64_t), dbytes = db.size() * sizeof(double);
        TB_CUDA(cudaMalloc(&o->blob, ibytes + dbytes));
        TB_CUDA(cudaMemcpy(o->blob, ib.data(), ibytes, cudaMemcpyHostToDevice));
        TB_CUDA(cudaMemcpy((char *)o->blob + ibytes, db.data(), dbytes, cudaMemcpyHostToDevice));
        const int64_t *di = (const int64_t *)o->blob;
        const double *dd = (const double *)((char *)o->blob + ibytes);
        o->V.first = di;
        o->V.prefix = di + nv;
        o->V.n_view = (int)nv;
        o->V.total = total;
        o->amp_view_off = di + 2 * nv + 1;
        o->amp_offsets = di + 3 * nv + 1;
        o->g2l = di + 3 * nv + 1 + nd;
        o->fp = dd;
        o->cal = dd + 4 * nd;
        o->eta = dd + 5 * nd;
        o->gamma = dd + 6 * nd;
        o->det_scale = dd + 7 * nd;
        o->n_amp_det = acc;
        // the host arrays of the descriptor are not retained
        o->d.intervals = nullptr;
        o->d.epsilon = o->d.gamma = o->d.cal = o->d.det_scale = nullptr;
        o->d.amp_offsets = o->d.n_amp_views = o->d.global2local = nullptr;
        return o;
    } catch (const tbr::Error &e) {
        tbr::set_error(e.code, e.msg);
        return nullptr;
    }
}

} // namespace

extern "C" {

tb_obs *tb_obs_create(const tb_obs_desc *desc) { return obs_create(desc, nullptr, 3); }

tb_obs *tb_obs_create_wcs(const tb_obs_desc *desc, const tb_wcs_desc *wcs) {
    if (wcs == nullptr) {
        tbr::set_error(TB_ERR_ARG, "NULL projection");
        return nullptr;
    }
    return obs_create(desc, wcs, 3);
}

tb_obs *tb_obs_create_intensity(const tb_obs_desc *desc, const tb_wcs_desc *wcs) {
    return obs_create(desc, wcs, 1);
}

int tb_obs_nnz(const tb_obs *obs) { return obs ? obs->nnz : 0; }

void tb_obs_destroy(tb_obs *obs) {
    if (obs == nullptr) return;
    if (obs->blob) cudaFree(obs->blob);
    if (obs->lpix) cudaFree(obs->lpix);
    if (obs->wqu) cudaFree(obs->wqu);
    if (obs->lpp) cudaFree(obs->lpp);
    if (obs->pair_rot) cudaFree(obs->pair_rot);
    if (obs->xrec) cudaFree(obs->xrec);
    if (obs->xqu) cudaFree(obs->xqu);
    if (obs->xblocks) cudaFree(obs->xblocks);
    if (obs->stable) cudaFree(obs->stable);
    tb_free_blocked(obs);
    delete obs;
}

} // extern "C"

// Per-row constants {cal0, cal1, A, B} of the crossing list (rows = detector pairs when paired),
// and whether they are the same for every row (then they travel as kernel arguments).  Read by
// the block-ordered passes.
void tb_build_row_table(tb_obs *obs) {
    const int64_t n_rows = obs->n_xrows, n_det = obs->d.n_det;
    if (obs->stable) cudaFree(obs->stable);
    obs->stable = nullptr;
    std::vector<double> cal(n_det);
    TB_CUDA(cudaMemcpy(cal.data(), obs->cal, sizeof(double) * n_det, cudaMemcpyDeviceToHost));
    std::vector<double2> rot;
    if (obs->x_paired) {
        rot.assign(n_rows, make_double2(0.0, 0.0)); // (intensity rows: no weight rotation)
        if (obs->pair_rot)
            TB_CUDA(cudaMemcpy(rot.data(), obs->pair_rot, sizeof(double2) * n_rows,
                               cudaMemcpyDeviceToHost));
    }
    std::vector<double4> tab(n_rows);
    bool uniform = true;
    for (int64_t r = 0; r < n_rows; ++r) {
        int64_t d0 = obs->x_paired ? 2 * r : r, d1 = d0 + 1;
        bool has1 = obs->x_paired && d1 < n_det;
        // a missing partner never contributes (n1 = 0): give it the constants of row 0 so that
        // an odd detector count does not break uniformity
        tab[r] = make_double4(cal[d0], has1 ? cal[d1] : (r > 0 ? tab[0].y : cal[d0]),
                              has1 ? rot[r].x : (r > 0 ? tab[0].z : 0.0),
                              has1 ? rot[r].y : (r > 0 ? tab[0].w : 0.0));
        if (tab[r].x != tab[0].x || tab[r].y != tab[0].y || tab[r].z != tab[0].z ||
            tab[r].w != tab[0].w)
            uniform = false;
    }
    TB_CUDA(cudaMalloc(&obs->stable, sizeof(double4) * n_rows));
    TB_CUDA(cudaMemcpy(obs->stable, tab.data(), sizeof(double4) * n_rows, cudaMemcpyHostToDevice));
    obs->s_uniform = uniform ? 1 : 0;
    obs->s_const[0] = tab[0].x;
    obs->s_const[1] = tab[0].y;
    obs->s_const[2] = tab[0].z;
    obs->s_const[3] = tab[0].w;
}

// Records per 32-sample chunk of the crossing list in one row layout (the counting pass of
// k_xbuild); for paired intensity rows also the records whose detectors fall in different pixels.
static std::vector<int32_t> count_crossings(tb_obs *obs, int paired, int64_t n_rows, int64_t cpr,
                                            int64_t *n_split, cudaStream_t st) {
    const int64_t n_chunks = n_rows * cpr;
    ObsDev o = make_dev(obs, 0);
    int32_t *counts = nullptr;
    TB_CUDA(cudaMalloc(&counts, sizeof(int32_t) * (n_chunks + 1)));
    int grid = tbr::sm_count() * 8;
    if (obs->nnz == 1) {
        TB_CUDA(cudaMemsetAsync(counts + n_chunks, 0, sizeof(int32_t), st));
        k_xbuild<false, 1><<<grid, kThreads, 0, st>>>(o, paired, n_rows, cpr, counts, nullptr,
                                                      nullptr, nullptr);
    } else {
        k_xbuild<false, 3><<<grid, kThreads, 0, st>>>(o, paired, n_rows, cpr, counts, nullptr,
                                                      nullptr, nullptr);
    }
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    std::vector<int32_t> hc(n_chunks + 1, 0);
    TB_CUDA(cudaMemcpyAsync(hc.data(), counts,
                            sizeof(int32_t) * (obs->nnz == 1 ? n_chunks + 1 : n_chunks),
                            cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    cudaFree(counts);
    if (n_split) *n_split = (int64_t)(uint32_t)hc[n_chunks];
    hc.pop_back();
    return hc;
}

// Collapse the packed pointing into the crossing list (k_lhs_x) when that is the smaller stream.
// Intensity observations always get it (the block-ordered list is built from it), in the row
// layout that gives the block-ordered list fewer entries: detector pairs share a record while
// both detectors stay in one pixel, but a record whose detectors fall in different pixels takes
// two entries, so pairs whose partners point apart are better kept as one row per detector.
static void build_crossings(tb_obs *obs, cudaStream_t st) {
    if (obs->xrec) cudaFree(obs->xrec);
    if (obs->xqu) cudaFree(obs->xqu);
    if (obs->xblocks) cudaFree(obs->xblocks);
    obs->xrec = nullptr;
    obs->xqu = nullptr;
    obs->xblocks = nullptr;
    obs->n_xrec = obs->n_xblocks = obs->n_xrows = 0;
    if (obs->stable) cudaFree(obs->stable);
    obs->stable = nullptr;
    tb_free_blocked(obs);
    if (obs->lpix == nullptr || obs->V.total <= 0) return;
    const bool intensity = obs->nnz == 1;
    const int64_t n_det = obs->d.n_det;
    const int64_t cpr = (obs->V.total + 31) / 32;
    int paired = obs->lpp != nullptr ? 1 : 0;
    std::vector<int32_t> hc;
    if (intensity) {
        paired = 0;
        hc = count_crossings(obs, 0, n_det, cpr, nullptr, st);
        if (n_det >= 2) {
            int64_t split = 0, records_p = 0, entries_u = 0;
            std::vector<int32_t> hp = count_crossings(obs, 1, (n_det + 1) / 2, cpr, &split, st);
            for (int32_t c : hc) entries_u += c;
            for (int32_t c : hp) records_p += c;
            // (the 32-bit split counter is exact whenever the paired list can be built at all)
            if (records_p < 2147483647LL && records_p + split < entries_u) {
                paired = 1;
                hc.swap(hp);
            }
        }
    }
    const int64_t n_rows = paired ? (n_det + 1) / 2 : n_det;
    const int64_t n_chunks = n_rows * cpr;
    if (!intensity) hc = count_crossings(obs, paired, n_rows, cpr, nullptr, st);
    ObsDev o = make_dev(obs, 0);
    int grid = tbr::sm_count() * 8;
    std::vector<int64_t> hb(n_chunks);
    std::vector<int64_t> row_ptr(n_rows + 1);
    int64_t total = 0;
    for (int64_t r = 0; r < n_rows; ++r) {
        row_ptr[r] = total;
        for (int64_t c = r * cpr; c < (r + 1) * cpr; ++c) {
            hb[c] = total;
            total += hc[c];
        }
    }
    row_ptr[n_rows] = total;
    // worth it only when the records are a smaller stream than the per-sample form (intensity:
    // a 16-byte record replaces at least one 17-byte stored sample)
    const double per_sample = (paired ? 12.0 : 20.0) * (double)obs->V.total * (double)n_det;
    if (total == 0 || total >= 2147483647LL) return;
    if (!intensity && 32.0 * (double)total > 0.8 * per_sample) return;
    int64_t *base = nullptr;
    TB_CUDA(cudaMalloc(&base, sizeof(int64_t) * n_chunks));
    TB_CUDA(cudaMemcpyAsync(base, hb.data(), sizeof(int64_t) * n_chunks, cudaMemcpyHostToDevice,
                            st));
    TB_CUDA(cudaMalloc(&obs->xrec, sizeof(int4) * total));
    if (intensity) {
        k_xbuild<true, 1><<<grid, kThreads, 0, st>>>(o, paired, n_rows, cpr, nullptr, base,
                                                     obs->xrec, nullptr);
    } else {
        TB_CUDA(cudaMalloc(&obs->xqu, sizeof(double2) * total));
        k_xbuild<true, 3><<<grid, kThreads, 0, st>>>(o, paired, n_rows, cpr, nullptr, base,
                                                     obs->xrec, obs->xqu);
    }
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    // CTA table, TIME-major like tile_of_block: tile k of every row, then tile k + 1, ... so that
    // resident CTAs work on the same time window (= the same sky region) of all rows
    std::vector<int4> blocks;
    int64_t max_tiles = 0;
    for (int64_t r = 0; r < n_rows; ++r) {
        int64_t nt = (row_ptr[r + 1] - row_ptr[r] + kXTile - 1) / kXTile;
        if (nt > max_tiles) max_tiles = nt;
    }
    for (int64_t k = 0; k < max_tiles; ++k) {
        for (int64_t r = 0; r < n_rows; ++r) {
            int64_t b = row_ptr[r] + k * kXTile;
            if (b >= row_ptr[r + 1]) continue;
            int64_t e = b + kXTile < row_ptr[r + 1] ? b + kXTile : row_ptr[r + 1];
            blocks.push_back(make_int4((int)r, (int)b, (int)e, 0));
        }
    }
    TB_CUDA(cudaMalloc(&obs->xblocks, sizeof(int4) * blocks.size()));
    TB_CUDA(cudaMemcpyAsync(obs->xblocks, blocks.data(), sizeof(int4) * blocks.size(),
                            cudaMemcpyHostToDevice, st));
    TB_CUDA(cudaStreamSynchronize(st));
    cudaFree(base);
    obs->n_xrec = total;
    obs->n_xblocks = (int64_t)blocks.size();
    obs->n_xrows = n_rows;
    obs->x_paired = paired;
    tb_build_row_table(obs);
    tb_build_blocked(obs, st);
}

extern "C" {

int tb_obs_pack_pointing(tb_obs *obs, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs != nullptr, "NULL observation");
    TB_REQUIRE(obs->d.pixels && obs->d.weights, "packing needs stored pixels and weights");
    int64_t total = obs->d.n_det * obs->d.n_samp;
    TB_REQUIRE((int64_t)obs->d.n_pix_submap * obs->d.n_submap < 2147483647LL,
               "map too large for 32-bit local pixel indices");
    if (obs->lpix == nullptr) {
        TB_CUDA(cudaMalloc(&obs->lpix, sizeof(int32_t) * total));
        if (obs->nnz == 3) TB_CUDA(cudaMalloc(&obs->wqu, sizeof(double2) * total));
    }
    ObsDev o = make_dev(obs, 0);
    unsigned zero = 0;
    TB_CUDA(cudaMemcpyToSymbolAsync(g_pack_mismatch, &zero, sizeof(zero), 0,
                                    cudaMemcpyHostToDevice, (cudaStream_t)stream));
    int grid = tbr::sm_count() * 8;
    if (obs->nnz == 1)
        k_pack_pointing<1><<<grid, kThreads, 0, (cudaStream_t)stream>>>(o, obs->lpix, nullptr);
    else
        k_pack_pointing<3><<<grid, kThreads, 0, (cudaStream_t)stream>>>(o, obs->lpix, obs->wqu);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    unsigned bad = 0;
    TB_CUDA(cudaMemcpyFromSymbolAsync(&bad, g_pack_mismatch, sizeof(bad), 0,
                                      cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    TB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (obs->lpp) cudaFree(obs->lpp);
    if (obs->pair_rot) cudaFree(obs->pair_rot);
    obs->lpp = nullptr;
    obs->pair_rot = nullptr;
    if (bad) {
        // the I weight is not the per-detector constant: keep the general kernels
        cudaFree(obs->lpix);
        cudaFree(obs->wqu);
        obs->lpix = nullptr;
        obs->wqu = nullptr;
    } else if (obs->V.total > 0 && obs->nnz == 1) {
        // intensity: no weights to relate within a pair, the crossing list picks its rows
        build_crossings(obs, (cudaStream_t)stream);
    } else if (obs->V.total > 0) {
        // pair form: fit the per-pair weight rotation on the first in-interval sample, then
        // verify it on every sample while writing the paired pixel records
        int64_t n_pair = (obs->d.n_det + 1) / 2;
        std::vector<int64_t> hv(obs->V.n_view * 2 + 1);
        TB_CUDA(cudaMemcpy(hv.data(), obs->V.first, sizeof(int64_t) * hv.size(),
                           cudaMemcpyDeviceToHost)); // first[nv], prefix[nv+1] are contiguous
        int64_t s_fit = 0;
        for (int v = 0; v < obs->V.n_view; ++v) {
            if (hv[obs->V.n_view + v + 1] > hv[obs->V.n_view + v]) {
                s_fit = hv[v];
                break;
            }
        }
        TB_CUDA(cudaMalloc(&obs->lpp, sizeof(int2) * n_pair * obs->d.n_samp));
        TB_CUDA(cudaMalloc(&obs->pair_rot, sizeof(double2) * n_pair));
        TB_CUDA(cudaMemsetAsync(obs->lpp, 0xFF, sizeof(int2) * n_pair * obs->d.n_samp,
                                (cudaStream_t)stream));
        TB_CUDA(cudaMemcpyToSymbolAsync(g_pair_mismatch, &zero, sizeof(zero), 0,
                                        cudaMemcpyHostToDevice, (cudaStream_t)stream));
        o = make_dev(obs, 0);
        k_pair_fit<<<(unsigned)((n_pair + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
            o, n_pair, s_fit, obs->pair_rot);
        TB_CUDA(cudaGetLastError());
        tbr::count_launch();
        k_pack_pairs<<<grid, kThreads, 0, (cudaStream_t)stream>>>(o, n_pair, obs->pair_rot,
                                                                  obs->lpp);
        TB_CUDA(cudaGetLastError());
        tbr::count_launch();
        unsigned pbad = 0;
        TB_CUDA(cudaMemcpyFromSymbolAsync(&pbad, g_pair_mismatch, sizeof(pbad), 0,
                                          cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        TB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
        if (pbad) { // weights of the pair are not related by a fixed rotation: k_lhs_pair
            cudaFree(obs->lpp);
            cudaFree(obs->pair_rot);
            obs->lpp = nullptr;
            obs->pair_rot = nullptr;
        }
        build_crossings(obs, (cudaStream_t)stream);
    }
    TB_API_END
}

int tb_obs_crossing_stats(const tb_obs *obs, int64_t *n_records, int64_t *n_rows, int *paired) {
    TB_API_BEGIN
    TB_REQUIRE(obs != nullptr, "NULL observation");
    if (n_records) *n_records = obs->xrec ? obs->n_xrec : 0;
    if (n_rows) *n_rows = obs->xrec ? obs->n_xrows : 0;
    if (paired) *paired = obs->xrec ? obs->x_paired : 0;
    TB_API_END
}

int tb_obs_has_compact_pointing(const tb_obs *obs) { return (obs && obs->lpix) ? 1 : 0; }
int tb_obs_has_pair_weights(const tb_obs *obs) { return (obs && obs->lpp) ? 1 : 0; }

extern int tb_peer_ctas_per_sm; // tb_peer.cu
extern int tb_prior_chunk;      // tb_prior.cu

int tb_get_option(const char *name) {
    if (name == nullptr) return -1;
    std::string n(name);
    if (n == "pair") return g_use_pair;
    if (n == "pairw") return g_use_pairw;
    if (n == "crossings") return g_use_x;
    if (n == "peer_ctas") return tb_peer_ctas_per_sm;
    if (n == "blocked") return g_use_bx;
    if (n == "prior_chunk") return tb_prior_chunk;
    return -1;
}

int tb_set_option(const char *name, int value) {
    TB_API_BEGIN
    TB_REQUIRE(name != nullptr, "NULL option name");
    if (std::string(name) == "pair") {
        g_use_pair = value;
    } else if (std::string(name) == "pairw") {
        g_use_pairw = value;
    } else if (std::string(name) == "crossings") {
        g_use_x = value;
    } else if (std::string(name) == "blocked") {
        g_use_bx = value;
    } else if (std::string(name) == "prior_chunk") {
        TB_REQUIRE(value >= 0, "prior_chunk must be >= 0");
        tb_prior_chunk = value;
    } else if (std::string(name) == "peer_ctas") {
        TB_REQUIRE(value >= 1 && value <= 16, "peer_ctas must be in [1, 16]");
        tb_peer_ctas_per_sm = value;
    } else {
        throw tbr::Error{TB_ERR_ARG, std::string("unknown option: ") + name};
    }
    TB_API_END
}

int tb_lhs_pass1(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                 double *zmap, int regen, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && amplitudes && amp_flags && zmap, "NULL argument");
    launch_bin<false>(obs, amplitudes, amp_flags, nullptr, zmap, regen, stream);
    TB_API_END
}

int tb_lhs_pass2(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                 const double *binned, double *amplitudes_out, int regen, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && amplitudes && amp_flags && binned && amplitudes_out, "NULL argument");
    launch_project<false>(obs, amplitudes, amp_flags, nullptr, binned, amplitudes_out, regen,
                          stream);
    TB_API_END
}

int tb_obs_sorted_passes(const tb_obs *) { return 0; }

int tb_obs_set_pixel_chunks(tb_obs *obs, int64_t n_chunks, const int64_t *pixel_bounds) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && pixel_bounds && n_chunks >= 1 && n_chunks <= 4096, "bad chunk arguments");
    TB_REQUIRE(obs->brec != nullptr, "the observation has no block-ordered crossing list");
    for (int64_t c = 0; c < n_chunks; ++c)
        TB_REQUIRE(pixel_bounds[c] <= pixel_bounds[c + 1], "pixel bounds must be non-decreasing");
    tb_blocked_set_chunks(obs, n_chunks, pixel_bounds);
    TB_API_END
}

int tb_rhs_project(const tb_obs *obs, const double *signal, const uint8_t *amp_flags,
                   const double *binned, double *amplitudes_out, int regen, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && signal && amp_flags && binned && amplitudes_out, "NULL argument");
    launch_project<true>(obs, nullptr, amp_flags, signal, binned, amplitudes_out, regen, stream);
    TB_API_END
}

int tb_bin_signal(const tb_obs *obs, const double *signal, double *zmap, int regen,
                  void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && signal && zmap, "NULL argument");
    launch_bin<true>(obs, nullptr, nullptr, signal, zmap, regen, stream);
    TB_API_END
}

int tb_amp_dot(const double *a, const double *b, const uint8_t *flags, int64_t n, double *out,
               void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    RedScratch &r = red_scratch();
    k_amp_dot<<<red_grid(n), kThreads, 0, (cudaStream_t)stream>>>(a, b, flags, n, r.partials,
                                                                   r.counter, out);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    TB_API_END
}

int tb_pcg_update(const double *delta, const double *dq, double *x, double *r, const double *d,
                  const double *q, double *s, const double *offset_var, const uint8_t *flags,
                  int64_t n, double *sums, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    RedScratch &rs = red_scratch();
    k_pcg_update<<<red_grid(n), kThreads, 0, (cudaStream_t)stream>>>(
        delta, dq, x, r, d, q, s, offset_var, flags, n, rs.partials, rs.counter, sums);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    TB_API_END
}

int tb_pcg_direction(const double *delta_new, const double *delta_old, double *d, const double *s,
                     int64_t n, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    k_pcg_direction<<<red_grid(n), kThreads, 0, (cudaStream_t)stream>>>(delta_new, delta_old, d, s,
                                                                         n);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
    TB_API_END
}

} // extern "C"
