// tb_ops.cu -- one CUDA kernel per TOAST hot-path operator kernel, behind the C ABI of
// include/toast_b200.h.  Each entry point replaces the `_libtoast` function cited in the
// header; semantics (index arrays, optional flags, intervals, in-place accumulation) follow the
// reference's CPU branch, the launch geometry is B200-first:
//   * the (view, sample) loops are flattened so every thread has work,
//   * CTAs are ordered time-major / detector-minor (see tb_device.cuh) so scattered map
//     traffic stays in L2,
//   * once-used timestream data is read/written with streaming (evict-first) accesses.
#include "tb_device.cuh"
#include "tb_pixelise.cuh"
#include "tb_runtime.cuh"

using namespace tbd;

namespace {

__device__ unsigned long long g_exact_count = 0ull;
double g_guard_scale = 1.0;

// ---- host helpers ------------------------------------------------------------------------------

Views make_views(tbr::Resolver &R, const tb_interval *iv, int64_t n_view, int64_t n_samp) {
    TB_REQUIRE(n_view >= 0, "negative number of intervals");
    TB_REQUIRE(n_view == 0 || iv != nullptr, "intervals pointer is NULL");
    std::vector<int64_t> buf(2 * n_view + 1);
    int64_t total = 0;
    for (int64_t v = 0; v < n_view; ++v) {
        int64_t a = iv[v].first, b = iv[v].last;
        TB_REQUIRE(a >= 0 && b <= n_samp, "interval outside [0, n_samp)");
        buf[v] = a;
        buf[n_view + v] = total;
        if (b > a) total += b - a;
    }
    buf[2 * n_view] = total;
    const int64_t *d = R.small(buf.data(), buf.size());
    Views V;
    V.first = d;
    V.prefix = d + n_view;
    V.n_view = (int)n_view;
    V.total = total;
    return V;
}

inline int64_t n_blocks(const Views &V, int64_t n_det) {
    int64_t tiles = (V.total + kTile - 1) / kTile;
    return tiles * n_det;
}

void check_index(const int32_t *idx, int64_t n_det, int64_t n_buf, const char *what) {
    TB_REQUIRE(idx != nullptr, std::string(what) + " index array is NULL");
    for (int64_t i = 0; i < n_det; ++i) {
        TB_REQUIRE(idx[i] >= 0 && idx[i] < n_buf, std::string(what) + " index out of range");
    }
}

#define TB_LAUNCH(kernel, blocks, R, ...)                                                   \
    do {                                                                                    \
        int64_t _nb = (blocks);                                                             \
        if (_nb > 0) {                                                                      \
            TB_REQUIRE(_nb < 2147483647LL, "grid too large");                               \
            kernel<<<(unsigned)_nb, kThreads, 0, (R).stream()>>>(__VA_ARGS__);              \
            TB_CUDA(cudaGetLastError());                                                    \
            tbr::count_launch();                                                            \
        }                                                                                   \
    } while (0)

// Iterate the kPerThread samples of this thread's tile; BODY sees `det`, `s` (sample), `view`
// and `off` (= s - first[view]).  All lanes of a warp run the same trip count (needed by the
// kernels that shuffle); `valid` is false for the padding past the end.
#define TB_FOR_TILE_SAMPLES(V, n_det)                                                       \
    TileId _tile = tile_of_block(blockIdx.x, (n_det));                                      \
    const int det = _tile.det;                                                              \
    ViewCursor _vc = view_cursor((V), _tile.t0 + threadIdx.x);                              \
    _Pragma("unroll") for (int _k = 0; _k < kPerThread; ++_k)

#define TB_SAMPLE_COORDS(V)                                                                 \
    int64_t _t = _tile.t0 + (int64_t)_k * kThreads + threadIdx.x;                           \
    bool valid = _t < (V).total;                                                            \
    int view = 0;                                                                           \
    int64_t off = 0, s = 0;                                                                 \
    if (valid) {                                                                            \
        view_seek((V), _vc, _t);                                                            \
        view = _vc.view;                                                                    \
        off = _t - _vc.beg;                                                                 \
        s = _vc.first + off;                                                                \
    }

// ================================================================================================
// a1 pointing_detector
// ================================================================================================
__global__ void __launch_bounds__(kThreads)
k_pointing_detector(Views V, int64_t n_det, int64_t n_samp, const double *__restrict__ fp,
                    const double *__restrict__ boresight, const int32_t *__restrict__ qidx,
                    double *__restrict__ quats, const uint8_t *__restrict__ flags, uint8_t mask) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        tbm::Quat f = ld_quat(fp + 4 * det);
        bool bad = flags ? ((__ldg(flags + s) & mask) != 0) : false;
        tbm::Quat q = detector_quat(boresight, s, bad, f);
        st_quat_stream(quats + ((int64_t)__ldg(qidx + det) * n_samp + s) * 4, q);
    }
}

// ================================================================================================
// a2 pixels_healpix
// ================================================================================================
// occupancy targets measured on B200 (profiles/r1_kernels_c2.json): these kernels are fp64 /
// integer ALU bound and a few spills cost less than fewer resident warps
#ifndef TB_POINT_CTAS
#define TB_POINT_CTAS 4
#endif
template <bool NEST>
__global__ void __launch_bounds__(kThreads, 6)
k_pixels_healpix(Views V, int64_t n_det, int64_t n_samp, tbm::PixCtx ctx,
                 const int32_t *__restrict__ qidx, const double *__restrict__ quats,
                 const uint8_t *__restrict__ flags, uint8_t mask,
                 const int32_t *__restrict__ pidx, int64_t *__restrict__ pixels,
                 uint8_t *__restrict__ hsub, double inv_nps) {
    int n_exact = 0;
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        tbm::Quat q = ld_quat_stream(quats + ((int64_t)__ldg(qidx + det) * n_samp + s) * 4);
        double dx, dy, dz;
        tbm::rot_zaxis(q, dx, dy, dz);
        int ex = 0;
        int64_t p = tbm::vec2pix<NEST>(ctx, dx, dy, dz, &ex);
        n_exact += ex;
        if (flags && ((__ldg(flags + s) & mask) != 0)) {
            p = -1;
        } else {
            int64_t sm = fast_div(p, inv_nps);
            if (hsub[sm] == 0) hsub[sm] = 1;
        }
        st_stream(pixels + (int64_t)__ldg(pidx + det) * n_samp + s, p);
    }
    if (n_exact) atomicAdd(&g_exact_count, (unsigned long long)n_exact);
}

// ================================================================================================
// f4 pixels_wcs: detector quaternions -> pixel numbers of a flat projection (tb_wcs.cuh)
// ================================================================================================
__global__ void __launch_bounds__(kThreads, 4)
k_pixels_wcs(Views V, int64_t n_det, int64_t n_samp, tbw::Wcs w, const int32_t *__restrict__ qidx,
             const double *__restrict__ quats, const uint8_t *__restrict__ flags, uint8_t mask,
             const int32_t *__restrict__ pidx, int64_t *__restrict__ pixels,
             uint8_t *__restrict__ hsub, double inv_nps) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        tbm::Quat q = ld_quat_stream(quats + ((int64_t)__ldg(qidx + det) * n_samp + s) * 4);
        int64_t p = tbw::quat_to_wcs_pixel(w, q);
        if (flags && ((__ldg(flags + s) & mask) != 0)) p = -1;
        if (p >= 0 && hsub != nullptr) {
            int64_t sm = fast_div(p, inv_nps);
            if (hsub[sm] == 0) hsub[sm] = 1;
        }
        st_stream(pixels + (int64_t)__ldg(pidx + det) * n_samp + s, p);
    }
}

// ================================================================================================
// a3 stokes_weights_IQU / stokes_weights_I
// ================================================================================================
template <bool HWP>
__global__ void __launch_bounds__(kThreads)
k_stokes_iqu(Views V, int64_t n_det, int64_t n_samp, const int32_t *__restrict__ qidx,
             const double *__restrict__ quats, const int32_t *__restrict__ widx,
             double *__restrict__ weights, const double *__restrict__ hwp,
             const double *__restrict__ epsilon, const double *__restrict__ gamma,
             const double *__restrict__ cal, double U_sign) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        double eps = __ldg(epsilon + det);
        double eta = (1.0 - eps) / (1.0 + eps);
        double c = __ldg(cal + det);
        double g = __ldg(gamma + det);
        tbm::Quat q = ld_quat_stream(quats + ((int64_t)__ldg(qidx + det) * n_samp + s) * 4);
        double w0, w1, w2;
        tbm::stokes_iqu<HWP>(q, c, eta, U_sign, g, HWP ? __ldg(hwp + s) : 0.0, w0, w1, w2);
        double *w = weights + ((int64_t)__ldg(widx + det) * n_samp + s) * 3;
        st_stream(w, w0);
        st_stream(w + 1, w1);
        st_stream(w + 2, w2);
    }
}

__global__ void __launch_bounds__(kThreads)
k_stokes_i(Views V, int64_t n_det, int64_t n_samp, const int32_t *__restrict__ widx,
           double *__restrict__ weights, const double *__restrict__ cal) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        st_stream(weights + (int64_t)__ldg(widx + det) * n_samp + s, __ldg(cal + det));
    }
}

// ================================================================================================
// a1+a2+a3 fused: boresight -> quats / pixels / weights in one pass
// ================================================================================================
struct FusedOut {
    const int32_t *qidx;
    double *quats;
    const int32_t *pidx;
    int64_t *pixels;
    const int32_t *widx;
    double *weights;
    uint8_t *hsub;
};

// PIX: the pixelisation policy of tb_pixelise.cuh (HEALPix NEST / RING, or WCS)
template <class PIX, bool HWP>
__global__ void __launch_bounds__(kThreads, TB_POINT_CTAS)
k_pointing_fused(Views V, int64_t n_det, int64_t n_samp, typename PIX::Geom geom,
                 const double *__restrict__ fp, const double *__restrict__ boresight,
                 const uint8_t *__restrict__ flags, uint8_t mask, FusedOut o,
                 const double *__restrict__ hwp, const double *__restrict__ epsilon,
                 const double *__restrict__ gamma, const double *__restrict__ cal, double U_sign,
                 double inv_nps) {
    int n_exact = 0;
    int64_t last_sm = -1;
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        tbm::Quat f = ld_quat(fp + 4 * det);
        bool bad = flags ? ((__ldg(flags + s) & mask) != 0) : false;
        tbm::Quat q = detector_quat(boresight, s, bad, f);
        if (o.quats) st_quat_stream(o.quats + ((int64_t)__ldg(o.qidx + det) * n_samp + s) * 4, q);
        if (o.pixels) {
            int64_t p = PIX::pixel(geom, q, n_exact);
            if (bad) {
                p = -1;
            } else if (o.hsub && (!PIX::kMayMiss || p >= 0)) {
                // the thread's samples mostly stay in one submap: look at the mask only when
                // the submap changes
                const int64_t sm = PIX::submap(geom, p, inv_nps);
                if (sm != last_sm) {
                    if (o.hsub[sm] == 0) o.hsub[sm] = 1;
                    last_sm = sm;
                }
            }
            st_stream(o.pixels + (int64_t)__ldg(o.pidx + det) * n_samp + s, p);
        }
        if (o.weights) {
            double eps = __ldg(epsilon + det);
            double eta = (1.0 - eps) / (1.0 + eps);
            double w0, w1, w2;
            tbm::stokes_iqu<HWP>(q, __ldg(cal + det), eta, U_sign, __ldg(gamma + det),
                                 HWP ? __ldg(hwp + s) : 0.0, w0, w1, w2);
            double *w = o.weights + ((int64_t)__ldg(o.widx + det) * n_samp + s) * 3;
            st_stream(w, w0);
            st_stream(w + 1, w1);
            st_stream(w + 2, w2);
        }
    }
    if (n_exact) atomicAdd(&g_exact_count, (unsigned long long)n_exact);
}

// ================================================================================================
// a4 noise_weight
// ================================================================================================
__global__ void __launch_bounds__(kThreads)
k_noise_weight(Views V, int64_t n_det, int64_t n_samp, double *__restrict__ data,
               const int32_t *__restrict__ didx, const double *__restrict__ wt) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        double *p = data + (int64_t)__ldg(didx + det) * n_samp + s;
        st_stream(p, ld_stream(p) * __ldg(wt + det));
    }
}

// ================================================================================================
// a5 build_noise_weighted: scatter-add with warp-aggregated runs
// ================================================================================================
template <int NNZ> // 1, 3, or 0 = runtime nnz (no aggregation)
__global__ void __launch_bounds__(kThreads)
k_build_noise_weighted(Views V, int64_t n_det, int64_t n_samp, int64_t nnz_rt,
                       const int64_t *__restrict__ g2l, double *__restrict__ zmap,
                       int64_t n_pix_submap, double inv_nps, const int32_t *__restrict__ pidx,
                       const int64_t *__restrict__ pixels, const int32_t *__restrict__ widx,
                       const double *__restrict__ weights, const int32_t *__restrict__ didx,
                       const double *__restrict__ data, const int32_t *__restrict__ fidx,
                       const uint8_t *__restrict__ dflags, const double *__restrict__ scale,
                       uint8_t dmask, const uint8_t *__restrict__ sflags, uint8_t smask) {
    const int lane = threadIdx.x & 31;
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        int64_t key = -1; // local pixel offset into zmap (in pixels), -1 = nothing to add
        double z0 = 0.0, z1 = 0.0, z2 = 0.0;
        if (valid) {
            int64_t p = ld_stream(pixels + (int64_t)__ldg(pidx + det) * n_samp + s);
            bool ok = p >= 0;
            if (dflags) ok = ok && ((ld_stream(dflags + (int64_t)__ldg(fidx + det) * n_samp + s) & dmask) == 0);
            if (sflags) ok = ok && ((__ldg(sflags + s) & smask) == 0);
            if (ok) {
                int64_t gsm = fast_div(p, inv_nps);
                int64_t lsm = __ldg(g2l + gsm);
                key = lsm * n_pix_submap + (p - gsm * n_pix_submap);
                double sd = ld_stream(data + (int64_t)__ldg(didx + det) * n_samp + s) *
                            __ldg(scale + det);
                const double *w = weights + ((int64_t)__ldg(widx + det) * n_samp + s) *
                                                (NNZ ? NNZ : nnz_rt);
                if (NNZ == 3) {
                    z0 = sd * ld_stream(w);
                    z1 = sd * ld_stream(w + 1);
                    z2 = sd * ld_stream(w + 2);
                } else if (NNZ == 1) {
                    z0 = sd * ld_stream(w);
                } else {
                    double *z = zmap + key * nnz_rt;
                    for (int64_t k = 0; k < nnz_rt; ++k) atomicAdd(z + k, sd * ld_stream(w + k));
                }
            }
        }
        if (NNZ != 0) {
            Runs r = find_runs(key, lane);
            z0 = seg_sum(z0, r);
            if (NNZ == 3) {
                z1 = seg_sum(z1, r);
                z2 = seg_sum(z2, r);
            }
            if (r.is_tail && key >= 0) {
                double *z = zmap + key * NNZ;
                atomicAdd(z, z0);
                if (NNZ == 3) {
                    atomicAdd(z + 1, z1);
                    atomicAdd(z + 2, z2);
                }
            }
        }
    }
}

// ================================================================================================
// a7 scan_map<T>
// ================================================================================================
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_scan_map(Views V, int64_t n_det, int64_t n_samp, const int64_t *__restrict__ g2l,
           int64_t n_pix_submap, double inv_nps, const T *__restrict__ mapdata, int64_t nnz,
           double *__restrict__ data, const int32_t *__restrict__ didx,
           const int64_t *__restrict__ pixels, const int32_t *__restrict__ pidx,
           const double *__restrict__ weights, const int32_t *__restrict__ widx,
           double data_scale, bool zero, bool subtract, bool scale) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        double *dp = data + (int64_t)__ldg(didx + det) * n_samp + s;
        int64_t p = ld_stream(pixels + (int64_t)__ldg(pidx + det) * n_samp + s);
        double d = zero ? 0.0 : ld_stream(dp);
        if (p >= 0) {
            int64_t gsm = fast_div(p, inv_nps);
            int64_t moff = nnz * (__ldg(g2l + gsm) * n_pix_submap + (p - gsm * n_pix_submap));
            const double *w = weights + ((int64_t)__ldg(widx + det) * n_samp + s) * nnz;
            double v = 0.0;
            for (int64_t k = 0; k < nnz; ++k) v += ld_stream(w + k) * (double)__ldg(mapdata + moff + k);
            v *= data_scale;
            if (subtract) {
                d -= v;
            } else if (scale) {
                d *= v;
            } else {
                d += v;
            }
            st_stream(dp, d);
        } else if (zero) {
            st_stream(dp, d);
        }
    }
}

// ================================================================================================
// a8-a10 Offset template
// ================================================================================================
struct OffsetLayout {
    const int64_t *amp_view_off; // [n_view] amplitude offset of each view inside a detector
    const int64_t *amp_offsets;  // [n_det]  first amplitude of each detector
    double inv_step;
};

__global__ void __launch_bounds__(kThreads)
k_offset_add(Views V, int64_t n_det, int64_t n_samp, OffsetLayout L,
             const double *__restrict__ amps, const uint8_t *__restrict__ aflags,
             const int32_t *__restrict__ didx, double *__restrict__ data) {
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        if (!valid) continue;
        int64_t amp = __ldg(L.amp_offsets + det) + __ldg(L.amp_view_off + view) +
                      fast_div(off, L.inv_step);
        if (__ldg(aflags + amp) == 0) {
            double *p = data + (int64_t)__ldg(didx + det) * n_samp + s;
            st_stream(p, ld_stream(p) + __ldg(amps + amp));
        }
    }
}

__global__ void __launch_bounds__(kThreads)
k_offset_project(Views V, int64_t n_det, int64_t n_samp, OffsetLayout L,
                 double *__restrict__ amps, const uint8_t *__restrict__ aflags,
                 const int32_t *__restrict__ didx, const double *__restrict__ data,
                 const int32_t *__restrict__ fidx, const uint8_t *__restrict__ flags,
                 uint8_t mask) {
    const int lane = threadIdx.x & 31;
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        int64_t key = -1;
        double v = 0.0;
        if (valid) {
            int64_t amp = __ldg(L.amp_offsets + det) + __ldg(L.amp_view_off + view) +
                          fast_div(off, L.inv_step);
            if (__ldg(aflags + amp) == 0) {
                key = amp;
                bool good = true;
                if (flags && fidx) {
                    int32_t fi = __ldg(fidx + det);
                    if (fi >= 0) good = (ld_stream(flags + (int64_t)fi * n_samp + s) & mask) == 0;
                }
                if (good) v = ld_stream(data + (int64_t)__ldg(didx + det) * n_samp + s);
            }
        }
        Runs r = find_runs(key, lane);
        v = seg_sum(v, r);
        if (r.is_tail && key >= 0) atomicAdd(amps + key, v);
    }
}

__global__ void __launch_bounds__(kThreads)
k_offset_precond(int64_t n, const double *__restrict__ var, const double *__restrict__ in,
                 const uint8_t *__restrict__ flags, double *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i < n) out[i] = (flags[i] == 0) ? in[i] * var[i] : 0.0;
}

// ================================================================================================
// a6 covariance kernels
// ================================================================================================
__global__ void __launch_bounds__(kThreads)
k_cov_apply(int64_t npix, int nnz, const double *__restrict__ cov, double *__restrict__ vec) {
    int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= npix) return;
    if (nnz == 1) {
        vec[p] *= cov[p];
        return;
    }
    if (nnz == 3) {
        const double *m = cov + p * 6;
        double *v = vec + p * 3;
        double v0 = v[0], v1 = v[1], v2 = v[2];
        // same accumulation order as toast_map_cov.cpp:509-517
        double t0 = 0.0, t1 = 0.0, t2 = 0.0;
        t0 += m[0] * v0;
        t0 += m[1] * v1;
        t1 += m[1] * v0;
        t0 += m[2] * v2;
        t2 += m[2] * v0;
        t1 += m[3] * v1;
        t1 += m[4] * v2;
        t2 += m[4] * v1;
        t2 += m[5] * v2;
        v[0] = t0;
        v[1] = t1;
        v[2] = t2;
        return;
    }
    const int block = nnz * (nnz + 1) / 2;
    const double *m = cov + p * block;
    double *v = vec + p * nnz;
    double tmp[8], vin[8];
    for (int k = 0; k < nnz; ++k) {
        tmp[k] = 0.0;
        vin[k] = v[k];
    }
    int o = 0;
    for (int k = 0; k < nnz; ++k) {
        for (int j = k; j < nnz; ++j) {
            tmp[k] += m[o] * vin[j];
            if (j != k) tmp[j] += m[o] * vin[k];
            ++o;
        }
    }
    for (int k = 0; k < nnz; ++k) v[k] = tmp[k];
}

template <int NNZ>
__global__ void __launch_bounds__(kThreads)
k_cov_accum(Views V, int64_t n_det, int64_t n_samp, const int64_t *__restrict__ g2l,
            int64_t n_pix_submap, double inv_nps, int64_t *__restrict__ hits,
            double *__restrict__ invcov, const int32_t *__restrict__ pidx,
            const int64_t *__restrict__ pixels, const int32_t *__restrict__ widx,
            const double *__restrict__ weights, const int32_t *__restrict__ fidx,
            const uint8_t *__restrict__ dflags, const double *__restrict__ scale, uint8_t dmask,
            const uint8_t *__restrict__ sflags, uint8_t smask) {
    const int lane = threadIdx.x & 31;
    constexpr int BLOCK = NNZ * (NNZ + 1) / 2;
    TB_FOR_TILE_SAMPLES(V, n_det) {
        TB_SAMPLE_COORDS(V)
        int64_t key = -1;
        double c[BLOCK];
#pragma unroll
        for (int i = 0; i < BLOCK; ++i) c[i] = 0.0;
        if (valid) {
            int64_t p = ld_stream(pixels + (int64_t)__ldg(pidx + det) * n_samp + s);
            bool ok = p >= 0;
            if (dflags) ok = ok && ((ld_stream(dflags + (int64_t)__ldg(fidx + det) * n_samp + s) & dmask) == 0);
            if (sflags) ok = ok && ((__ldg(sflags + s) & smask) == 0);
            if (ok) {
                int64_t gsm = fast_div(p, inv_nps);
                key = __ldg(g2l + gsm) * n_pix_submap + (p - gsm * n_pix_submap);
                if (invcov) {
                    const double *w = weights + ((int64_t)__ldg(widx + det) * n_samp + s) * NNZ;
                    double wv[NNZ];
#pragma unroll
                    for (int i = 0; i < NNZ; ++i) wv[i] = ld_stream(w + i);
                    double sc = __ldg(scale + det);
                    int o = 0;
#pragma unroll
                    for (int j = 0; j < NNZ; ++j) {
                        double sw = wv[j] * sc; // toast_map_cov.cpp:133-137
#pragma unroll
                        for (int k = j; k < NNZ; ++k) c[o++] = wv[k] * sw;
                    }
                }
            }
        }
        Runs r = find_runs(key, lane);
        if (hits) {
            // run length = number of hits of this pixel inside the warp
            if (r.is_tail && key >= 0)
                atomicAdd((unsigned long long *)(hits + key), (unsigned long long)(r.dist + 1));
        }
        if (invcov) {
#pragma unroll
            for (int i = 0; i < BLOCK; ++i) c[i] = seg_sum(c[i], r);
            if (r.is_tail && key >= 0) {
                double *z = invcov + key * BLOCK;
#pragma unroll
                for (int i = 0; i < BLOCK; ++i) atomicAdd(z + i, c[i]);
            }
        }
    }
}

// Symmetric 3x3 eigen-inverse with rcond threshold, one pixel per thread (tbm::cov_invert3 in
// tb_math.cuh: host/device code, run on the CPU by tests/test_host_math.py;
// toast_map_cov.cpp:246-396 does the same through LAPACK dsyev + dgemm).
__global__ void __launch_bounds__(kThreads)
k_cov_invert3(int64_t npix, double *__restrict__ cov, double *__restrict__ rcond,
              double threshold) {
    int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= npix) return;
    const double rc = tbm::cov_invert3(cov + p * 6, threshold);
    if (rcond) rcond[p] = rc;
}

__global__ void __launch_bounds__(kThreads)
k_cov_invert1(int64_t npix, double *__restrict__ cov, double *__restrict__ rcond) {
    int64_t p = (int64_t)blockIdx.x * kThreads + threadIdx.x;
    if (p >= npix) return;
    double d = cov[p];
    if (d != 0.0) cov[p] = 1.0 / d;
    if (rcond) rcond[p] = 1.0;
}

inline int64_t blocks_1d(int64_t n) { return (n + kThreads - 1) / kThreads; }

OffsetLayout make_offset_layout(tbr::Resolver &R, int64_t step_length, const int64_t *amp_offsets,
                                int64_t n_det, const int64_t *n_amp_views, int64_t n_view) {
    TB_REQUIRE(step_length > 0, "step_length must be positive");
    std::vector<int64_t> buf(n_view + n_det);
    int64_t acc = 0;
    for (int64_t v = 0; v < n_view; ++v) {
        buf[v] = acc;
        acc += n_amp_views[v];
    }
    for (int64_t d = 0; d < n_det; ++d) buf[n_view + d] = amp_offsets[d];
    const int64_t *dev = R.small(buf.data(), buf.size());
    OffsetLayout L;
    L.amp_view_off = dev;
    L.amp_offsets = dev + n_view;
    L.inv_step = 1.0 / (double)step_length;
    return L;
}

} // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

void tb_set_pixel_guard_scale(double scale) { g_guard_scale = scale; }

int64_t tb_pixel_exact_count(int reset) {
    unsigned long long v = 0;
    if (cudaMemcpyFromSymbol(&v, g_exact_count, sizeof(v)) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    if (reset) {
        unsigned long long z = 0;
        cudaMemcpyToSymbol(g_exact_count, &z, sizeof(z));
    }
    return (int64_t)v;
}

int tb_pointing_detector(const double *focalplane, const double *boresight,
                         const int32_t *quat_index, double *quats, int64_t n_det_buf,
                         const tb_interval *intervals, int64_t n_view,
                         const uint8_t *shared_flags, uint8_t shared_flag_mask, int64_t n_det,
                         int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(quat_index, n_det, n_det_buf, "quat");
    Views V = make_views(R, intervals, n_view, n_samp);
    const double *d_fp = R.small(focalplane, 4 * n_det);
    const int32_t *d_qi = R.small(quat_index, n_det);
    const double *d_bore = R.in(boresight, 4 * n_samp);
    const uint8_t *d_fl = R.in(shared_flags, n_samp);
    double *d_q = R.out(quats, n_det_buf * n_samp * 4);
    TB_LAUNCH(k_pointing_detector, n_blocks(V, n_det), R, V, n_det, n_samp, d_fp, d_bore, d_qi,
              d_q, d_fl, shared_flag_mask);
    R.finish();
    TB_API_END
}

int tb_pixels_healpix(const int32_t *quat_index, const double *quats, int64_t n_quat_buf,
                      const uint8_t *shared_flags, uint8_t shared_flag_mask,
                      const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
                      const tb_interval *intervals, int64_t n_view, uint8_t *hit_submaps,
                      int64_t n_submap, int64_t n_pix_submap, int64_t nside, int nest,
                      int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nside > 0 && (nside & (nside - 1)) == 0, "nside must be a power of two");
    TB_REQUIRE(nside <= (1 << 24), "nside > 2^24 not supported");
    TB_REQUIRE(n_pix_submap > 0 && n_submap * n_pix_submap >= 12 * nside * nside,
               "hit_submaps too small for nside");
    check_index(quat_index, n_det, n_quat_buf, "quat");
    check_index(pixel_index, n_det, n_pix_buf, "pixel");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int32_t *d_qi = R.small(quat_index, n_det);
    const int32_t *d_pi = R.small(pixel_index, n_det);
    uint8_t *d_hs = R.small_inout(hit_submaps, n_submap);
    const double *d_q = R.in(quats, n_quat_buf * n_samp * 4);
    const uint8_t *d_fl = R.in(shared_flags, n_samp);
    int64_t *d_p = R.out(pixels, n_pix_buf * n_samp);
    tbm::PixCtx ctx = tbm::make_pix_ctx(nside, g_guard_scale);
    double inv = 1.0 / (double)n_pix_submap;
    if (nest) {
        TB_LAUNCH(k_pixels_healpix<true>, n_blocks(V, n_det), R, V, n_det, n_samp, ctx, d_qi, d_q,
                  d_fl, shared_flag_mask, d_pi, d_p, d_hs, inv);
    } else {
        TB_LAUNCH(k_pixels_healpix<false>, n_blocks(V, n_det), R, V, n_det, n_samp, ctx, d_qi, d_q,
                  d_fl, shared_flag_mask, d_pi, d_p, d_hs, inv);
    }
    R.finish();
    TB_API_END
}

int tb_pixels_wcs(const tb_wcs_desc *wcs, const int32_t *quat_index, const double *quats,
                  int64_t n_quat_buf, const uint8_t *shared_flags, uint8_t shared_flag_mask,
                  const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
                  const tb_interval *intervals, int64_t n_view, uint8_t *hit_submaps,
                  int64_t n_submap, int64_t n_pix_submap, int64_t n_det, int64_t n_samp, int mem,
                  void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    tbw::Wcs w = tbp::wcs_from_desc(wcs);
    TB_REQUIRE(hit_submaps == nullptr || (n_pix_submap > 0 && n_submap * n_pix_submap >= w.n_pix),
               "hit_submaps too small for the projection");
    check_index(quat_index, n_det, n_quat_buf, "quat");
    check_index(pixel_index, n_det, n_pix_buf, "pixel");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int32_t *d_qi = R.small(quat_index, n_det);
    const int32_t *d_pi = R.small(pixel_index, n_det);
    uint8_t *d_hs = hit_submaps ? R.small_inout(hit_submaps, n_submap) : nullptr;
    const double *d_q = R.in(quats, n_quat_buf * n_samp * 4);
    const uint8_t *d_fl = R.in(shared_flags, n_samp);
    int64_t *d_p = R.out(pixels, n_pix_buf * n_samp);
    double inv = n_pix_submap > 0 ? 1.0 / (double)n_pix_submap : 0.0;
    TB_LAUNCH(k_pixels_wcs, n_blocks(V, n_det), R, V, n_det, n_samp, w, d_qi, d_q, d_fl,
              shared_flag_mask, d_pi, d_p, d_hs, inv);
    R.finish();
    TB_API_END
}

int tb_stokes_weights_IQU(const int32_t *quat_index, const double *quats, int64_t n_quat_buf,
                          const int32_t *weight_index, double *weights, int64_t n_w_buf,
                          const double *hwp, const tb_interval *intervals, int64_t n_view,
                          const double *epsilon, const double *gamma, const double *cal, int IAU,
                          int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(quat_index, n_det, n_quat_buf, "quat");
    check_index(weight_index, n_det, n_w_buf, "weight");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int32_t *d_qi = R.small(quat_index, n_det);
    const int32_t *d_wi = R.small(weight_index, n_det);
    const double *d_eps = R.small(epsilon, n_det);
    const double *d_gam = R.small(gamma, n_det);
    const double *d_cal = R.small(cal, n_det);
    const double *d_q = R.in(quats, n_quat_buf * n_samp * 4);
    const double *d_hwp = R.in(hwp, n_samp);
    double *d_w = R.out(weights, n_w_buf * n_samp * 3);
    double U_sign = IAU ? -1.0 : 1.0;
    if (d_hwp) {
        TB_LAUNCH(k_stokes_iqu<true>, n_blocks(V, n_det), R, V, n_det, n_samp, d_qi, d_q, d_wi, d_w,
                  d_hwp, d_eps, d_gam, d_cal, U_sign);
    } else {
        TB_LAUNCH(k_stokes_iqu<false>, n_blocks(V, n_det), R, V, n_det, n_samp, d_qi, d_q, d_wi,
                  d_w, d_hwp, d_eps, d_gam, d_cal, U_sign);
    }
    R.finish();
    TB_API_END
}

int tb_stokes_weights_I(const int32_t *weight_index, double *weights, int64_t n_w_buf,
                        const tb_interval *intervals, int64_t n_view, const double *cal,
                        int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(weight_index, n_det, n_w_buf, "weight");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int32_t *d_wi = R.small(weight_index, n_det);
    const double *d_cal = R.small(cal, n_det);
    double *d_w = R.out(weights, n_w_buf * n_samp);
    TB_LAUNCH(k_stokes_i, n_blocks(V, n_det), R, V, n_det, n_samp, d_wi, d_w, d_cal);
    R.finish();
    TB_API_END
}

} // extern "C"

namespace {

// the body of tb_pointing_fused / tb_pointing_fused_wcs: `n_pix_map` is the number of pixels the
// hit-submap mask must cover
template <class PIX>
void pointing_fused(tbr::Resolver &R, const typename PIX::Geom &geom, int64_t n_pix_map,
                    const char *hsub_msg, const double *focalplane, const double *boresight,
                    const uint8_t *shared_flags, uint8_t shared_flag_mask,
                    const int32_t *quat_index, double *quats, int64_t n_quat_buf,
                    const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
                    const int32_t *weight_index, double *weights, int64_t n_w_buf,
                    const double *hwp, const tb_interval *intervals, int64_t n_view,
                    uint8_t *hit_submaps, int64_t n_submap, int64_t n_pix_submap,
                    const double *epsilon, const double *gamma, const double *cal, int IAU,
                    int64_t n_det, int64_t n_samp) {
    Views V = make_views(R, intervals, n_view, n_samp);
    FusedOut o{};
    if (quats) {
        check_index(quat_index, n_det, n_quat_buf, "quat");
        o.qidx = R.small(quat_index, n_det);
        o.quats = R.out(quats, n_quat_buf * n_samp * 4);
    }
    if (pixels) {
        check_index(pixel_index, n_det, n_pix_buf, "pixel");
        o.pidx = R.small(pixel_index, n_det);
        o.pixels = R.out(pixels, n_pix_buf * n_samp);
        if (hit_submaps) {
            TB_REQUIRE(n_pix_submap > 0 && n_submap * n_pix_submap >= n_pix_map, hsub_msg);
            o.hsub = R.small_inout(hit_submaps, n_submap);
        }
    }
    const double *d_eps = nullptr, *d_gam = nullptr, *d_cal = nullptr;
    if (weights) {
        check_index(weight_index, n_det, n_w_buf, "weight");
        o.widx = R.small(weight_index, n_det);
        o.weights = R.out(weights, n_w_buf * n_samp * 3);
        d_eps = R.small(epsilon, n_det);
        d_gam = R.small(gamma, n_det);
        d_cal = R.small(cal, n_det);
    }
    const double *d_fp = R.small(focalplane, 4 * n_det);
    const double *d_bore = R.in(boresight, 4 * n_samp);
    const uint8_t *d_fl = R.in(shared_flags, n_samp);
    const double *d_hwp = R.in(hwp, n_samp);
    double inv = 1.0 / (double)(n_pix_submap > 0 ? n_pix_submap : 1);
    double U_sign = IAU ? -1.0 : 1.0;
    int64_t nb = n_blocks(V, n_det);
    if (d_hwp) {
        auto kfn = k_pointing_fused<PIX, true>;
        TB_LAUNCH(kfn, nb, R, V, n_det, n_samp, geom, d_fp, d_bore, d_fl, shared_flag_mask, o,
                  d_hwp, d_eps, d_gam, d_cal, U_sign, inv);
    } else {
        auto kfn = k_pointing_fused<PIX, false>;
        TB_LAUNCH(kfn, nb, R, V, n_det, n_samp, geom, d_fp, d_bore, d_fl, shared_flag_mask, o,
                  d_hwp, d_eps, d_gam, d_cal, U_sign, inv);
    }
}

} // namespace

extern "C" {

int tb_pointing_fused(const double *focalplane, const double *boresight,
                      const uint8_t *shared_flags, uint8_t shared_flag_mask,
                      const int32_t *quat_index, double *quats, int64_t n_quat_buf,
                      const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
                      const int32_t *weight_index, double *weights, int64_t n_w_buf,
                      const double *hwp, const tb_interval *intervals, int64_t n_view,
                      uint8_t *hit_submaps, int64_t n_submap, int64_t n_pix_submap, int64_t nside,
                      int nest, const double *epsilon, const double *gamma, const double *cal,
                      int IAU, int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nside > 0 && (nside & (nside - 1)) == 0, "nside must be a power of two");
    TB_REQUIRE(nside <= (1 << 24), "nside > 2^24 not supported");
    tbm::PixCtx ctx = tbm::make_pix_ctx(nside, g_guard_scale);
    auto fused = nest ? pointing_fused<tbp::PixHealpix<true>>
                      : pointing_fused<tbp::PixHealpix<false>>;
    fused(R, ctx, 12 * nside * nside, "hit_submaps too small for nside", focalplane, boresight,
          shared_flags, shared_flag_mask, quat_index, quats, n_quat_buf, pixel_index, pixels,
          n_pix_buf, weight_index, weights, n_w_buf, hwp, intervals, n_view, hit_submaps,
          n_submap, n_pix_submap, epsilon, gamma, cal, IAU, n_det, n_samp);
    R.finish();
    TB_API_END
}

int tb_pointing_fused_wcs(const double *focalplane, const double *boresight,
                          const uint8_t *shared_flags, uint8_t shared_flag_mask,
                          const int32_t *quat_index, double *quats, int64_t n_quat_buf,
                          const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
                          const int32_t *weight_index, double *weights, int64_t n_w_buf,
                          const double *hwp, const tb_interval *intervals, int64_t n_view,
                          uint8_t *hit_submaps, int64_t n_submap, int64_t n_pix_submap,
                          const tb_wcs_desc *wcs, const double *epsilon, const double *gamma,
                          const double *cal, int IAU, int64_t n_det, int64_t n_samp, int mem,
                          void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    tbw::Wcs w = tbp::wcs_from_desc(wcs);
    pointing_fused<tbp::PixWcs>(R, w, w.n_pix, "hit_submaps too small for the projection",
                                focalplane, boresight, shared_flags, shared_flag_mask, quat_index,
                                quats, n_quat_buf, pixel_index, pixels, n_pix_buf, weight_index,
                                weights, n_w_buf, hwp, intervals, n_view, hit_submaps, n_submap,
                                n_pix_submap, epsilon, gamma, cal, IAU, n_det, n_samp);
    R.finish();
    TB_API_END
}

int tb_noise_weight(double *det_data, int64_t n_data_buf, const int32_t *data_index,
                    const tb_interval *intervals, int64_t n_view, const double *detector_weights,
                    int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(data_index, n_det, n_data_buf, "data");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int32_t *d_di = R.small(data_index, n_det);
    const double *d_w = R.small(detector_weights, n_det);
    double *d_d = R.inout(det_data, n_data_buf * n_samp);
    TB_LAUNCH(k_noise_weight, n_blocks(V, n_det), R, V, n_det, n_samp, d_d, d_di, d_w);
    R.finish();
    TB_API_END
}

int tb_build_noise_weighted(const int64_t *global2local, int64_t n_submap, double *zmap,
                            int64_t n_local_submap, int64_t n_pix_submap, int64_t nnz,
                            const int32_t *pixel_index, const int64_t *pixels, int64_t n_pix_buf,
                            const int32_t *weight_index, const double *weights, int64_t n_w_buf,
                            const int32_t *data_index, const double *det_data, int64_t n_data_buf,
                            const int32_t *flag_index, const uint8_t *det_flags,
                            int64_t n_flag_buf, const double *det_scale, uint8_t det_flag_mask,
                            const tb_interval *intervals, int64_t n_view,
                            const uint8_t *shared_flags, uint8_t shared_flag_mask, int64_t n_det,
                            int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nnz >= 1, "nnz must be >= 1");
    check_index(pixel_index, n_det, n_pix_buf, "pixel");
    check_index(weight_index, n_det, n_w_buf, "weight");
    check_index(data_index, n_det, n_data_buf, "data");
    if (det_flags) check_index(flag_index, n_det, n_flag_buf, "flag");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int64_t *d_g2l = R.small(global2local, n_submap);
    const int32_t *d_pi = R.small(pixel_index, n_det);
    const int32_t *d_wi = R.small(weight_index, n_det);
    const int32_t *d_di = R.small(data_index, n_det);
    const int32_t *d_fi = det_flags ? R.small(flag_index, n_det) : nullptr;
    const double *d_sc = R.small(det_scale, n_det);
    double *d_z = R.inout(zmap, n_local_submap * n_pix_submap * nnz);
    const int64_t *d_p = R.in(pixels, n_pix_buf * n_samp);
    const double *d_w = R.in(weights, n_w_buf * n_samp * nnz);
    const double *d_d = R.in(det_data, n_data_buf * n_samp);
    const uint8_t *d_df = R.in(det_flags, n_flag_buf * n_samp);
    const uint8_t *d_sf = R.in(shared_flags, n_samp);
    double inv = 1.0 / (double)n_pix_submap;
    int64_t nb = n_blocks(V, n_det);
#define TB_BNW(N)                                                                               \
    TB_LAUNCH(k_build_noise_weighted<N>, nb, R, V, n_det, n_samp, nnz, d_g2l, d_z, n_pix_submap, \
              inv, d_pi, d_p, d_wi, d_w, d_di, d_d, d_fi, d_df, d_sc, det_flag_mask, d_sf,      \
              shared_flag_mask)
    if (nnz == 3) {
        TB_BNW(3);
    } else if (nnz == 1) {
        TB_BNW(1);
    } else {
        TB_BNW(0);
    }
#undef TB_BNW
    R.finish();
    TB_API_END
}

int tb_scan_map(const int64_t *global2local, int64_t n_submap, int64_t n_pix_submap,
                const void *mapdata, int map_dtype, int64_t n_local_submap, int64_t nnz,
                double *det_data, int64_t n_data_buf, const int32_t *data_index,
                const int64_t *pixels, int64_t n_pix_buf, const int32_t *pixel_index,
                const double *weights, int64_t n_w_buf, const int32_t *weight_index,
                const tb_interval *intervals, int64_t n_view, double data_scale, int should_zero,
                int should_subtract, int should_scale, int64_t n_det, int64_t n_samp, int mem,
                void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nnz >= 1, "nnz must be >= 1");
    check_index(pixel_index, n_det, n_pix_buf, "pixel");
    check_index(weight_index, n_det, n_w_buf, "weight");
    check_index(data_index, n_det, n_data_buf, "data");
    Views V = make_views(R, intervals, n_view, n_samp);
    const int64_t *d_g2l = R.small(global2local, n_submap);
    const int32_t *d_pi = R.small(pixel_index, n_det);
    const int32_t *d_wi = R.small(weight_index, n_det);
    const int32_t *d_di = R.small(data_index, n_det);
    static const size_t esz[4] = {8, 4, 8, 4};
    TB_REQUIRE(map_dtype >= 0 && map_dtype < 4, "invalid map dtype");
    const char *d_m = R.in((const char *)mapdata,
                           (size_t)(n_local_submap * n_pix_submap * nnz) * esz[map_dtype]);
    double *d_d = R.inout(det_data, n_data_buf * n_samp);
    const int64_t *d_p = R.in(pixels, n_pix_buf * n_samp);
    const double *d_w = R.in(weights, n_w_buf * n_samp * nnz);
    double inv = 1.0 / (double)n_pix_submap;
    int64_t nb = n_blocks(V, n_det);
#define TB_SCAN(T)                                                                             \
    TB_LAUNCH(k_scan_map<T>, nb, R, V, n_det, n_samp, d_g2l, n_pix_submap, inv, (const T *)d_m, \
              nnz, d_d, d_di, d_p, d_pi, d_w, d_wi, data_scale, should_zero != 0,              \
              should_subtract != 0, should_scale != 0)
    switch (map_dtype) {
    case TB_MAP_F64: TB_SCAN(double); break;
    case TB_MAP_F32: TB_SCAN(float); break;
    case TB_MAP_I64: TB_SCAN(int64_t); break;
    default: TB_SCAN(int32_t); break;
    }
#undef TB_SCAN
    R.finish();
    TB_API_END
}

int tb_template_offset_add_to_signal_batch(int64_t step_length, const int64_t *amp_offsets,
                                           const int64_t *n_amp_views, const double *amplitudes,
                                           const uint8_t *amplitude_flags, int64_t n_amp,
                                           const int32_t *data_index, double *det_data,
                                           int64_t n_data_buf, const tb_interval *intervals,
                                           int64_t n_view, int64_t n_det, int64_t n_samp, int mem,
                                           void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(data_index, n_det, n_data_buf, "data");
    Views V = make_views(R, intervals, n_view, n_samp);
    OffsetLayout L = make_offset_layout(R, step_length, amp_offsets, n_det, n_amp_views, n_view);
    const int32_t *d_di = R.small(data_index, n_det);
    const double *d_a = R.in(amplitudes, n_amp);
    const uint8_t *d_af = R.in(amplitude_flags, n_amp);
    double *d_d = R.inout(det_data, n_data_buf * n_samp);
    TB_LAUNCH(k_offset_add, n_blocks(V, n_det), R, V, n_det, n_samp, L, d_a, d_af, d_di, d_d);
    R.finish();
    TB_API_END
}

int tb_template_offset_add_to_signal(int64_t step_length, int64_t amp_offset,
                                     const int64_t *n_amp_views, const double *amplitudes,
                                     const uint8_t *amplitude_flags, int64_t n_amp,
                                     int32_t data_index, double *det_data, int64_t n_data_buf,
                                     const tb_interval *intervals, int64_t n_view, int64_t n_samp,
                                     int mem, void *stream) {
    return tb_template_offset_add_to_signal_batch(step_length, &amp_offset, n_amp_views,
                                                  amplitudes, amplitude_flags, n_amp, &data_index,
                                                  det_data, n_data_buf, intervals, n_view, 1,
                                                  n_samp, mem, stream);
}

int tb_template_offset_project_signal_batch(const int32_t *data_index, const double *det_data,
                                            int64_t n_data_buf, const int32_t *flag_index,
                                            const uint8_t *flag_data, int64_t n_flag_buf,
                                            uint8_t flag_mask, int64_t step_length,
                                            const int64_t *amp_offsets,
                                            const int64_t *n_amp_views, double *amplitudes,
                                            const uint8_t *amplitude_flags, int64_t n_amp,
                                            const tb_interval *intervals, int64_t n_view,
                                            int64_t n_det, int64_t n_samp, int mem,
                                            void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    check_index(data_index, n_det, n_data_buf, "data");
    bool use_flags = (flag_data != nullptr) && (flag_index != nullptr);
    if (use_flags) {
        for (int64_t i = 0; i < n_det; ++i)
            TB_REQUIRE(flag_index[i] < n_flag_buf, "flag index out of range");
    }
    Views V = make_views(R, intervals, n_view, n_samp);
    OffsetLayout L = make_offset_layout(R, step_length, amp_offsets, n_det, n_amp_views, n_view);
    const int32_t *d_di = R.small(data_index, n_det);
    const int32_t *d_fi = use_flags ? R.small(flag_index, n_det) : nullptr;
    double *d_a = R.inout(amplitudes, n_amp);
    const uint8_t *d_af = R.in(amplitude_flags, n_amp);
    const double *d_d = R.in(det_data, n_data_buf * n_samp);
    const uint8_t *d_f = use_flags ? R.in(flag_data, n_flag_buf * n_samp) : nullptr;
    TB_LAUNCH(k_offset_project, n_blocks(V, n_det), R, V, n_det, n_samp, L, d_a, d_af, d_di, d_d,
              d_fi, d_f, flag_mask);
    R.finish();
    TB_API_END
}

int tb_template_offset_project_signal(int32_t data_index, const double *det_data,
                                      int64_t n_data_buf, int32_t flag_index,
                                      const uint8_t *flag_data, int64_t n_flag_buf,
                                      uint8_t flag_mask, int64_t step_length, int64_t amp_offset,
                                      const int64_t *n_amp_views, double *amplitudes,
                                      const uint8_t *amplitude_flags, int64_t n_amp,
                                      const tb_interval *intervals, int64_t n_view,
                                      int64_t n_samp, int mem, void *stream) {
    const uint8_t *fd = (flag_index >= 0) ? flag_data : nullptr;
    return tb_template_offset_project_signal_batch(
        &data_index, det_data, n_data_buf, &flag_index, fd, n_flag_buf, flag_mask, step_length,
        &amp_offset, n_amp_views, amplitudes, amplitude_flags, n_amp, intervals, n_view, 1, n_samp,
        mem, stream);
}

int tb_template_offset_apply_diag_precond(const double *offset_var, const double *amplitudes_in,
                                          const uint8_t *amplitude_flags, double *amplitudes_out,
                                          int64_t n_amp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    const double *d_v = R.in(offset_var, n_amp);
    const double *d_i = R.in(amplitudes_in, n_amp);
    const uint8_t *d_f = R.in(amplitude_flags, n_amp);
    double *d_o = R.out(amplitudes_out, n_amp);
    TB_LAUNCH(k_offset_precond, blocks_1d(n_amp), R, n_amp, d_v, d_i, d_f, d_o);
    R.finish();
    TB_API_END
}

int tb_cov_apply_diag(int64_t n_local_submap, int64_t n_pix_submap, int64_t nnz,
                      const double *cov, double *vec, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nnz >= 1 && nnz <= 8, "nnz must be in [1, 8]");
    int64_t npix = n_local_submap * n_pix_submap;
    const double *d_c = R.in(cov, npix * (nnz * (nnz + 1) / 2));
    double *d_v = R.inout(vec, npix * nnz);
    TB_LAUNCH(k_cov_apply, blocks_1d(npix), R, npix, (int)nnz, d_c, d_v);
    R.finish();
    TB_API_END
}

int tb_cov_accum(const int64_t *global2local, int64_t n_submap, int64_t n_local_submap,
                 int64_t n_pix_submap, int64_t nnz, int64_t *hits, double *invcov,
                 const int32_t *pixel_index, const int64_t *pixels, int64_t n_pix_buf,
                 const int32_t *weight_index, const double *weights, int64_t n_w_buf,
                 const int32_t *flag_index, const uint8_t *det_flags, int64_t n_flag_buf,
                 const double *det_scale, uint8_t det_flag_mask, const tb_interval *intervals,
                 int64_t n_view, const uint8_t *shared_flags, uint8_t shared_flag_mask,
                 int64_t n_det, int64_t n_samp, int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nnz == 1 || nnz == 3, "tb_cov_accum supports nnz 1 or 3");
    check_index(pixel_index, n_det, n_pix_buf, "pixel");
    if (invcov) check_index(weight_index, n_det, n_w_buf, "weight");
    if (det_flags) check_index(flag_index, n_det, n_flag_buf, "flag");
    Views V = make_views(R, intervals, n_view, n_samp);
    int64_t npix = n_local_submap * n_pix_submap;
    const int64_t *d_g2l = R.small(global2local, n_submap);
    const int32_t *d_pi = R.small(pixel_index, n_det);
    const int32_t *d_wi = invcov ? R.small(weight_index, n_det) : nullptr;
    const int32_t *d_fi = det_flags ? R.small(flag_index, n_det) : nullptr;
    const double *d_sc = invcov ? R.small(det_scale, n_det) : nullptr;
    int64_t *d_h = R.inout(hits, npix);
    double *d_c = R.inout(invcov, npix * (nnz * (nnz + 1) / 2));
    const int64_t *d_p = R.in(pixels, n_pix_buf * n_samp);
    const double *d_w = invcov ? R.in(weights, n_w_buf * n_samp * nnz) : nullptr;
    const uint8_t *d_df = R.in(det_flags, n_flag_buf * n_samp);
    const uint8_t *d_sf = R.in(shared_flags, n_samp);
    double inv = 1.0 / (double)n_pix_submap;
    int64_t nb = n_blocks(V, n_det);
    if (nnz == 3) {
        TB_LAUNCH(k_cov_accum<3>, nb, R, V, n_det, n_samp, d_g2l, n_pix_submap, inv, d_h, d_c, d_pi,
                  d_p, d_wi, d_w, d_fi, d_df, d_sc, det_flag_mask, d_sf, shared_flag_mask);
    } else {
        TB_LAUNCH(k_cov_accum<1>, nb, R, V, n_det, n_samp, d_g2l, n_pix_submap, inv, d_h, d_c, d_pi,
                  d_p, d_wi, d_w, d_fi, d_df, d_sc, det_flag_mask, d_sf, shared_flag_mask);
    }
    R.finish();
    TB_API_END
}

int tb_cov_invert(int64_t npix, int64_t nnz, double *cov, double *rcond, double threshold,
                  int mem, void *stream) {
    TB_API_BEGIN
    tbr::Resolver R(mem, stream);
    TB_REQUIRE(nnz == 1 || nnz == 3, "tb_cov_invert supports nnz 1 or 3");
    double *d_c = R.inout(cov, npix * (nnz * (nnz + 1) / 2));
    double *d_r = R.out(rcond, npix);
    if (nnz == 3) {
        TB_LAUNCH(k_cov_invert3, blocks_1d(npix), R, npix, d_c, d_r, threshold);
    } else {
        TB_LAUNCH(k_cov_invert1, blocks_1d(npix), R, npix, d_c, d_r);
    }
    R.finish();
    TB_API_END
}

} // extern "C"
