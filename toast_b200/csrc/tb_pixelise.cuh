// tb_pixelise.cuh -- the pixel step of the per-sample pointing chain as a compile-time policy,
// shared by the fused pointing expansion (k_pointing_fused, tb_ops.cu) and the regenerated-pointing
// solver passes (sample_pointing, tb_solver.cu), so that both run the same device function:
//   PixHealpix<true>   HEALPix NEST  (tbm::vec2pix, two-tier exact path)
//   PixHealpix<false>  HEALPix RING
//   PixWcs             flat WCS projection (tbw::quat_to_wcs_pixel)
// A policy names the geometry it reads (`Geom`), maps a detector quaternion to a pixel, and maps a
// pixel to its submap.  `kMayMiss`: an unflagged sample can have a negative pixel (off the map).
#pragma once

#include "tb_device.cuh"
#include "tb_runtime.cuh"
#include "tb_wcs.cuh"

namespace tbp {

template <bool NEST>
struct PixHealpix {
    using Geom = tbm::PixCtx;
    static constexpr bool kMayMiss = false;
    static __device__ __forceinline__ int64_t pixel(const Geom &g, const tbm::Quat &q,
                                                    int &n_exact) {
        double dx, dy, dz;
        tbm::rot_zaxis(q, dx, dy, dz);
        int ex = 0;
        const int64_t p = tbm::vec2pix<NEST>(g, dx, dy, dz, &ex);
        n_exact += ex;
        return p;
    }
    // 32-bit conversions when the pixel number allows
    static __device__ __forceinline__ int64_t submap(const Geom &g, int64_t p, double inv_nps) {
        return g.small ? (int64_t)__double2int_rz(((double)(int)p + 0.5) * inv_nps)
                       : tbd::fast_div(p, inv_nps);
    }
};

struct PixWcs {
    using Geom = tbw::Wcs;
    static constexpr bool kMayMiss = true;
    static __device__ __forceinline__ int64_t pixel(const Geom &g, const tbm::Quat &q, int &) {
        return tbw::quat_to_wcs_pixel(g, q);
    }
    static __device__ __forceinline__ int64_t submap(const Geom &, int64_t p, double inv_nps) {
        return tbd::fast_div(p, inv_nps);
    }
};

// A validated tbw::Wcs from the C ABI descriptor (the checks of tb_pixels_wcs)
inline tbw::Wcs wcs_from_desc(const tb_wcs_desc *wcs) {
    TB_REQUIRE(wcs != nullptr, "NULL projection");
    TB_REQUIRE(wcs->projection >= 0 && wcs->projection <= 5, "unknown projection code");
    TB_REQUIRE(wcs->n_col > 0 && wcs->n_row > 0, "the projection has non-positive dimensions");
    TB_REQUIRE(wcs->cdelt[0] != 0.0 && wcs->cdelt[1] != 0.0, "CDELT must be non-zero");
    tbw::Wcs w;
    w.proj = wcs->projection;
    for (int k = 0; k < 5; ++k) w.euler[k] = wcs->euler[k];
    for (int k = 0; k < 2; ++k) {
        w.crpix[k] = wcs->crpix[k];
        w.cdelt[k] = wcs->cdelt[k];
    }
    w.cea_lambda = wcs->cea_lambda;
    w.n_col = wcs->n_col;
    w.n_pix = wcs->n_col * wcs->n_row;
    w.is_azimuth = wcs->is_azimuth;
    return w;
}

} // namespace tbp
