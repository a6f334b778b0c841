/*
 * toast_b200.h -- C ABI of libtoastb200.so, the B200 (sm_100a) implementation of the
 * TOAST map-making hot path.
 *
 * Every entry point replaces one function of the reference's `toast._libtoast` pybind11
 * module (the kernel boundary that `toast/ops/<op>/kernels.py` and
 * `toast/templates/offset/kernels.py` import by name); the reference interface each one
 * replaces is cited as file:line relative to /root/reference/src/toast/_libtoast.
 * INTEGRATION.md shows the pybind11 stub a TOAST maintainer adds on the reference side.
 *
 * Conventions
 * -----------
 *  - Plain pointers and sizes only.  All arrays are C-contiguous, native endian, with the
 *    dtypes and shapes of the reference buffers (SURVEY.md 8b): quats [n_det_buf,n_samp,4]
 *    f64, pixels [n_det_buf,n_samp] i64, weights [n_det_buf,n_samp,nnz] f64, det_data
 *    [n_det_buf,n_samp] f64, flags u8, maps [n_local_submap,n_pix_submap,nnz].
 *  - `mem` says where the LARGE arrays (marked [L]) live:
 *        TB_MEM_HOST    host pointers; staged to the device and back inside the call
 *                       (the `use_accel=False` behaviour: host in, host out, computed on GPU)
 *        TB_MEM_DEVICE  device pointers (e.g. torch tensors' data_ptr())
 *        TB_MEM_TABLE   host pointers previously registered with tb_accel_create(); the
 *                       device copy is looked up (the reference's `use_accel=True`,
 *                       accelerator.hpp:115-143).  A pointer that is not present is an error.
 *    SMALL per-detector / per-view arrays (marked [S]) are ALWAYS host pointers, exactly as
 *    the reference maps them per call (`omp target data map(to: ...)`).
 *  - Optional arrays (shared_flags, det_flags, hwp) are absent when the pointer is NULL
 *    (the pybind layer translates the reference's "length != n_samp" convention).
 *  - tb_interval is the reference's Interval POD (intervals.hpp:10-15); `last` is EXCLUSIVE.
 *    Samples outside every interval are never read or written.
 *  - Return value: 0 on success, non-zero on error; tb_last_error() returns the message
 *    (the pybind layer rethrows it as std::runtime_error -> Python RuntimeError like
 *    common.hpp:50-122).  There is NO CPU fallback: without a usable CUDA device every compute
 *    entry point fails with TB_ERR_NO_DEVICE.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *    asynchronous in TB_MEM_DEVICE mode and synchronous (like the reference) otherwise.
 */
#ifndef TOAST_B200_H
#define TOAST_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    double start;
    double stop;
    int64_t first;
    int64_t last;
} tb_interval;

enum { TB_MEM_HOST = 0, TB_MEM_DEVICE = 1, TB_MEM_TABLE = 2 };

enum {
    TB_OK = 0,
    TB_ERR_CUDA = 1,
    TB_ERR_NO_DEVICE = 2,
    TB_ERR_ARG = 3,
    TB_ERR_NOT_PRESENT = 4,
    TB_ERR_ALREADY_PRESENT = 5
};

/* ---- runtime ----------------------------------------------------------------------- */
const char *tb_last_error(void);
const char *tb_version(void);
/* 1 if a CUDA device is usable, else 0 (accel_enabled, accelerator.cpp:768-775). */
int tb_accel_enabled(void);
/* accel_assign_device(node_procs, node_rank, mem_gb, disabled): accelerator.cpp:233-306.
   device = node_rank % n_visible_devices. */
int tb_accel_assign_device(int node_procs, int node_rank, double mem_gb, int disabled);
int tb_accel_get_device(void);
int tb_device_synchronize(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t tb_launch_count(void);

/* ---- device memory table (OmpManager, accelerator.cpp:327-745, bindings :776-1110) ---- */
int tb_accel_present(const void *host, size_t nbytes);           /* 1 / 0 */
int tb_accel_create(const void *host, size_t nbytes, const char *name);
int tb_accel_update_device(const void *host, size_t nbytes, const char *name);
int tb_accel_update_host(void *host, size_t nbytes, const char *name);
int tb_accel_reset(const void *host, size_t nbytes, const char *name); /* zero the device copy */
int tb_accel_delete(const void *host, size_t nbytes, const char *name);
void *tb_accel_device_ptr(const void *host);                     /* NULL if absent */
void tb_accel_dump(void);
size_t tb_accel_bytes_in_use(void);

/* ---- a1  pointing_detector : ops_pointing_detector.cpp:78-227 -------------------------- */
int tb_pointing_detector(
    const double *focalplane,     /* [S] [n_det,4] */
    const double *boresight,      /* [L] [n_samp,4] */
    const int32_t *quat_index,    /* [S] [n_det] */
    double *quats,                /* [L] [n_det_buf,n_samp,4] out */
    int64_t n_det_buf,
    const tb_interval *intervals, /* [S] [n_view] */
    int64_t n_view,
    const uint8_t *shared_flags,  /* [L] [n_samp] or NULL */
    uint8_t shared_flag_mask, int64_t n_det, int64_t n_samp, int mem, void *stream);

/* ---- a2  pixels_healpix : ops_pixels_healpix.cpp:1153-1417 ------------------------------ */
int tb_pixels_healpix(
    const int32_t *quat_index,    /* [S] */
    const double *quats,          /* [L] [n_quat_buf,n_samp,4] */
    int64_t n_quat_buf,
    const uint8_t *shared_flags,  /* [L] or NULL */
    uint8_t shared_flag_mask,
    const int32_t *pixel_index,   /* [S] */
    int64_t *pixels,              /* [L] [n_pix_buf,n_samp] out */
    int64_t n_pix_buf,
    const tb_interval *intervals, int64_t n_view,
    uint8_t *hit_submaps,         /* [S] [n_submap] in/out, host */
    int64_t n_submap, int64_t n_pix_submap, int64_t nside, int nest, int64_t n_det,
    int64_t n_samp, int mem, void *stream);

/* ---- f4  pixels_wcs : ops/pixels_wcs.py:39-662 (host-only in the reference: qa_to_iso +
 * astropy / WCSLIB wcs_world2pix + around).  The projection arrives as the numbers WCSLIB's
 * celset / linset derive from CRVAL, CDELT, CRPIX and the default LONPOLE / LATPOLE
 * (toast_b200/ops/pixels_wcs.py builds them): projection 0 CAR, 1 CEA, 2 MER, 3 SFL, 4 TAN,
 * 5 ZEA; euler = {lng_p, 90 - lat_p, phi_p, cos(euler[1]), sin(euler[1])}; pixel = col + row *
 * n_col with col / row = around(world2pix, origin 0); samples that are flagged, have no image or
 * land at or beyond n_col * n_row get -1.  hit_submaps may be NULL. */
typedef struct tb_wcs_desc {
    int projection;
    int is_azimuth;               /* AZEL frame: lon = 2 pi - phi */
    double euler[5];
    double crpix[2], cdelt[2];
    double cea_lambda;            /* PV2_1 of CEA, 1 otherwise */
    int64_t n_col, n_row;
} tb_wcs_desc;
int tb_pixels_wcs(
    const tb_wcs_desc *wcs,
    const int32_t *quat_index,    /* [S] */
    const double *quats,          /* [L] [n_quat_buf,n_samp,4] */
    int64_t n_quat_buf,
    const uint8_t *shared_flags,  /* [L] or NULL */
    uint8_t shared_flag_mask,
    const int32_t *pixel_index,   /* [S] */
    int64_t *pixels,              /* [L] [n_pix_buf,n_samp] out */
    int64_t n_pix_buf,
    const tb_interval *intervals, int64_t n_view,
    uint8_t *hit_submaps,         /* [S] [n_submap] in/out, host, or NULL */
    int64_t n_submap, int64_t n_pix_submap, int64_t n_det, int64_t n_samp, int mem,
    void *stream);

/* ---- a3  stokes_weights_IQU / _I : ops_stokes_weights.cpp:150-392, :397-505 ------------- */
int tb_stokes_weights_IQU(
    const int32_t *quat_index, const double *quats /* [L] */, int64_t n_quat_buf,
    const int32_t *weight_index, double *weights /* [L] [n_w_buf,n_samp,3] out */,
    int64_t n_w_buf, const double *hwp /* [L] [n_samp] or NULL */,
    const tb_interval *intervals, int64_t n_view, const double *epsilon /* [S] */,
    const double *gamma /* [S] */, const double *cal /* [S] */, int IAU, int64_t n_det,
    int64_t n_samp, int mem, void *stream);

int tb_stokes_weights_I(
    const int32_t *weight_index, double *weights /* [L] [n_w_buf,n_samp] out */,
    int64_t n_w_buf, const tb_interval *intervals, int64_t n_view, const double *cal,
    int64_t n_det, int64_t n_samp, int mem, void *stream);

/* ---- a1+a2+a3 fused: boresight -> pixels (+ weights, + quats), no intermediate in HBM ---
 * Not in the reference (it runs the three operators back to back through `quats`); outputs
 * are bit-identical to tb_pointing_detector -> tb_pixels_healpix -> tb_stokes_weights_IQU.
 * Any of quats / pixels / weights may be NULL (not materialised).                        */
int tb_pointing_fused(
    const double *focalplane /* [S] */, const double *boresight /* [L] */,
    const uint8_t *shared_flags /* [L] or NULL */, uint8_t shared_flag_mask,
    const int32_t *quat_index, double *quats, int64_t n_quat_buf,
    const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
    const int32_t *weight_index, double *weights, int64_t n_w_buf,
    const double *hwp /* [L] or NULL */, const tb_interval *intervals, int64_t n_view,
    uint8_t *hit_submaps /* [S] or NULL */, int64_t n_submap, int64_t n_pix_submap,
    int64_t nside, int nest, const double *epsilon, const double *gamma, const double *cal,
    int IAU, int64_t n_det, int64_t n_samp, int mem, void *stream);

/* The same fused expansion onto a flat WCS projection (f4): the pixel step is tb_pixels_wcs's, so
 * outputs are bit-identical to tb_pointing_detector -> tb_pixels_wcs -> tb_stokes_weights_IQU.
 * Arguments as tb_pointing_fused with the projection in place of nside / nest; the descriptor is
 * validated as tb_pixels_wcs does, and hit_submaps (or NULL) must cover n_col * n_row pixels. */
int tb_pointing_fused_wcs(
    const double *focalplane /* [S] */, const double *boresight /* [L] */,
    const uint8_t *shared_flags /* [L] or NULL */, uint8_t shared_flag_mask,
    const int32_t *quat_index, double *quats, int64_t n_quat_buf,
    const int32_t *pixel_index, int64_t *pixels, int64_t n_pix_buf,
    const int32_t *weight_index, double *weights, int64_t n_w_buf,
    const double *hwp /* [L] or NULL */, const tb_interval *intervals, int64_t n_view,
    uint8_t *hit_submaps /* [S] or NULL */, int64_t n_submap, int64_t n_pix_submap,
    const tb_wcs_desc *wcs, const double *epsilon, const double *gamma, const double *cal,
    int IAU, int64_t n_det, int64_t n_samp, int mem, void *stream);

/* ---- a4  noise_weight : ops_noise_weight.cpp:12-118 ------------------------------------- */
int tb_noise_weight(
    double *det_data /* [L] [n_data_buf,n_samp] in/out */, int64_t n_data_buf,
    const int32_t *data_index, const tb_interval *intervals, int64_t n_view,
    const double *detector_weights /* [S] */, int64_t n_det, int64_t n_samp, int mem,
    void *stream);

/* ---- a5  build_noise_weighted : ops_mapmaker_utils.cpp:93-380 ---------------------------- */
int tb_build_noise_weighted(
    const int64_t *global2local /* [S] [n_submap] */, int64_t n_submap,
    double *zmap /* [L] [n_local_submap,n_pix_submap,nnz] accumulate */,
    int64_t n_local_submap, int64_t n_pix_submap, int64_t nnz,
    const int32_t *pixel_index, const int64_t *pixels /* [L] */, int64_t n_pix_buf,
    const int32_t *weight_index, const double *weights /* [L] */, int64_t n_w_buf,
    const int32_t *data_index, const double *det_data /* [L] */, int64_t n_data_buf,
    const int32_t *flag_index, const uint8_t *det_flags /* [L] or NULL */, int64_t n_flag_buf,
    const double *det_scale /* [S] */, uint8_t det_flag_mask, const tb_interval *intervals,
    int64_t n_view, const uint8_t *shared_flags /* [L] or NULL */, uint8_t shared_flag_mask,
    int64_t n_det, int64_t n_samp, int mem, void *stream);

/* ---- a7  scan_map<T> : ops_scan_map.cpp:85-292.  map_dtype: 0=f64 1=f32 2=i64 3=i32 ----- */
enum { TB_MAP_F64 = 0, TB_MAP_F32 = 1, TB_MAP_I64 = 2, TB_MAP_I32 = 3 };
int tb_scan_map(
    const int64_t *global2local /* [S] */, int64_t n_submap, int64_t n_pix_submap,
    const void *mapdata /* [L] [n_local_submap,n_pix_submap,nnz] */, int map_dtype,
    int64_t n_local_submap, int64_t nnz, double *det_data /* [L] in/out */,
    int64_t n_data_buf, const int32_t *data_index, const int64_t *pixels /* [L] */,
    int64_t n_pix_buf, const int32_t *pixel_index, const double *weights /* [L] */,
    int64_t n_w_buf, const int32_t *weight_index, const tb_interval *intervals,
    int64_t n_view, double data_scale, int should_zero, int should_subtract,
    int should_scale, int64_t n_det, int64_t n_samp, int mem, void *stream);

/* ---- a8-a10  Offset template : template_offset.cpp:16-146, :149-331, :334-405 ------------ */
int tb_template_offset_add_to_signal(
    int64_t step_length, int64_t amp_offset, const int64_t *n_amp_views /* [S] [n_view] */,
    const double *amplitudes /* [L] [n_amp] */, const uint8_t *amplitude_flags /* [L] */,
    int64_t n_amp, int32_t data_index, double *det_data /* [L] in/out */,
    int64_t n_data_buf, const tb_interval *intervals, int64_t n_view, int64_t n_samp,
    int mem, void *stream);

int tb_template_offset_project_signal(
    int32_t data_index, const double *det_data /* [L] */, int64_t n_data_buf,
    int32_t flag_index, const uint8_t *flag_data /* [L] or NULL */, int64_t n_flag_buf,
    uint8_t flag_mask, int64_t step_length, int64_t amp_offset, const int64_t *n_amp_views,
    double *amplitudes /* [L] accumulate */, const uint8_t *amplitude_flags /* [L] */,
    int64_t n_amp, const tb_interval *intervals, int64_t n_view, int64_t n_samp, int mem,
    void *stream);

int tb_template_offset_apply_diag_precond(
    const double *offset_var /* [L] */, const double *amplitudes_in /* [L] */,
    const uint8_t *amplitude_flags /* [L] */, double *amplitudes_out /* [L] */,
    int64_t n_amp, int mem, void *stream);

/* Batched forms over ALL detectors of an observation in one launch (the reference issues
 * one call per detector: offset.py:739-810, :813-881).  amp_offsets[d] is the detector's
 * first amplitude; data_index / flag_index are per detector.                              */
int tb_template_offset_add_to_signal_batch(
    int64_t step_length, const int64_t *amp_offsets /* [S] [n_det] */,
    const int64_t *n_amp_views, const double *amplitudes, const uint8_t *amplitude_flags,
    int64_t n_amp, const int32_t *data_index /* [S] */, double *det_data,
    int64_t n_data_buf, const tb_interval *intervals, int64_t n_view, int64_t n_det,
    int64_t n_samp, int mem, void *stream);

int tb_template_offset_project_signal_batch(
    const int32_t *data_index, const double *det_data, int64_t n_data_buf,
    const int32_t *flag_index /* [S] or NULL */, const uint8_t *flag_data, int64_t n_flag_buf,
    uint8_t flag_mask, int64_t step_length, const int64_t *amp_offsets,
    const int64_t *n_amp_views, double *amplitudes, const uint8_t *amplitude_flags,
    int64_t n_amp, const tb_interval *intervals, int64_t n_view, int64_t n_det,
    int64_t n_samp, int mem, void *stream);

/* ---- a6  covariance : libtoast/src/toast_map_cov.cpp:66-153, :471-528 -------------------- */
int tb_cov_apply_diag(int64_t n_local_submap, int64_t n_pix_submap, int64_t nnz,
                      const double *cov /* [L] [npix, nnz(nnz+1)/2] */,
                      double *vec /* [L] [npix, nnz] in/out */, int mem, void *stream);

/* hits[int64] and inverse covariance accumulation straight from (pixels, weights, flags):
 * BuildHitMap / BuildInverseCovariance (ops/mapmaker_utils/mapmaker_utils.py:114-206,
 * :352-515) without the host-side global_pixel_to_submap round trip.  Either output may be
 * NULL.                                                                                   */
int tb_cov_accum(
    const int64_t *global2local, int64_t n_submap, int64_t n_local_submap,
    int64_t n_pix_submap, int64_t nnz, int64_t *hits /* [L] [npix] or NULL */,
    double *invcov /* [L] [npix, nnz(nnz+1)/2] or NULL */, const int32_t *pixel_index,
    const int64_t *pixels, int64_t n_pix_buf, const int32_t *weight_index,
    const double *weights, int64_t n_w_buf, const int32_t *flag_index,
    const uint8_t *det_flags, int64_t n_flag_buf, const double *det_scale,
    uint8_t det_flag_mask, const tb_interval *intervals, int64_t n_view,
    const uint8_t *shared_flags, uint8_t shared_flag_mask, int64_t n_det, int64_t n_samp,
    int mem, void *stream);

/* Batched symmetric nnz x nnz eigen-inversion with rcond threshold
 * (cov_eigendecompose_diag, toast_map_cov.cpp:246-396), nnz in {1,3}.                     */
int tb_cov_invert(int64_t npix, int64_t nnz, double *cov /* [L] in/out */,
                  double *rcond /* [L] [npix] or NULL */, double threshold, int mem,
                  void *stream);

/* ---- fused destriper passes (a14: SolverLHS, mapmaker_solve.py:342-506) -------------------
 * A `tb_obs` describes one observation resident on the device (all pointers are DEVICE
 * pointers; small arrays are copied at creation).  The two passes are what one
 * SolverLHS.apply executes per observation:
 *   pass 1 = TemplateMatrix.add_to_signal -> BuildNoiseWeighted          (zmap += P^T N^-1 F a)
 *   pass 2 = add_to_signal -> ScanMap(subtract) -> NoiseWeight -> project_signal
 *                                                                 (out += F^T N^-1 (F a - P m))
 * det_temp never exists in HBM.  With `regen` != 0 pointing is recomputed from boresight
 * inside the pass instead of being read from pixels/weights.                              */
typedef struct tb_obs tb_obs;

typedef struct {
    int64_t n_det, n_samp, n_view;
    const tb_interval *intervals;     /* host [n_view] */
    const double *focalplane;         /* host [n_det,4] */
    const double *epsilon, *gamma, *cal; /* host [n_det] */
    const double *det_scale;          /* host [n_det] detector noise weights */
    const int64_t *amp_offsets;       /* host [n_det] first amplitude of each detector */
    const int64_t *n_amp_views;       /* host [n_view] */
    int64_t step_length;
    int64_t nside, n_pix_submap, n_submap;
    int nest, IAU;
    const int64_t *global2local;      /* host [n_submap] */
    /* device-resident */
    const double *boresight;          /* [n_samp,4] */
    const uint8_t *shared_flags;      /* [n_samp] or NULL */
    uint8_t shared_flag_mask;         /* used for pointing (pixel = -1) */
    const uint8_t *solver_flags;      /* [n_det,n_samp] or NULL */
    uint8_t solver_flag_mask;
    const int64_t *pixels;            /* [n_det,n_samp] or NULL (regen only) */
    const double *weights;            /* [n_det,n_samp,3] or NULL (regen only) */
    const double *hwp;                /* [n_samp] or NULL */
} tb_obs_desc;

tb_obs *tb_obs_create(const tb_obs_desc *desc);
/* An observation whose pixels are those of a flat WCS projection: `nside` / `nest` of the
 * descriptor are ignored, the projection is validated as tb_pixels_wcs does and kept for the
 * regenerated-pointing passes (regen != 0), which then compute the pixels tb_pointing_fused_wcs
 * stores.  Every other pass works on local pixel numbers and is the same for both kinds. */
tb_obs *tb_obs_create_wcs(const tb_obs_desc *desc, const tb_wcs_desc *wcs);
/* An INTENSITY observation (StokesWeights mode="I"): one Stokes value per pixel.  desc.weights
 * points to [n_det, n_samp] (the I weights, equal to cal[det]); epsilon and gamma are ignored.
 * `wcs` NULL: HEALPix pixels (nside / nest), otherwise as tb_obs_create_wcs.
 * Every entry point below that takes a tb_obs accepts both kinds and sizes the map by the
 * observation's nnz (tb_obs_nnz: 3 for tb_obs_create / tb_obs_create_wcs, 1 here): zmap / binned
 * maps are [n_local_pix, nnz], covariances [n_local_pix, nnz (nnz + 1) / 2].  For an intensity
 * observation tb_lhs_pass1 / tb_lhs_pass2 run the per-sample kernels (the "crossings", "pair" and
 * "pairw" paths are IQU-only), and its crossing list keeps no (sum Q, sum U). */
tb_obs *tb_obs_create_intensity(const tb_obs_desc *desc, const tb_wcs_desc *wcs /* NULL: HEALPix */);
int tb_obs_nnz(const tb_obs *obs);
void tb_obs_destroy(tb_obs *obs);

int tb_lhs_pass1(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                 double *zmap, int regen, void *stream);
int tb_lhs_pass2(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                 const double *binned, double *amplitudes_out, int regen, void *stream);
/* Always 0: no LHS pass runs on a pixel-sorted copy of the crossing list (kept for callers that
 * label the path). */
int tb_obs_sorted_passes(const tb_obs *obs);
/* Pixel chunks of the block-ordered crossing list, for pipelining the passes with the map
 * reduction (tb_bx_pass1 of chunk c -> reduction of that pixel range -> tb_bx_pass2 of chunk c).
 * pixel_bounds is a host array of n_chunks + 1 non-decreasing LOCAL pixel indices; chunk c holds
 * the blocks whose pixels lie in [pixel_bounds[c], pixel_bounds[c + 1]) (the outer chunks are
 * open-ended).  Refused when the observation has no block-ordered list; bounds that are not
 * multiples of the block size are accepted, but the chunked calls are then refused. */
int tb_obs_set_pixel_chunks(tb_obs *obs, int64_t n_chunks, const int64_t *pixel_bounds);
/* ---- block-ordered crossing list: shared-memory privatised map tiles (tb_blocked.cu) ----------
 * The same two passes as tb_lhs_pass1 / tb_lhs_pass2 (mapmaker_solve.py:342-506: template
 * add_to_signal + BuildNoiseWeighted, ops_mapmaker_utils.cpp:15-86,295-377; ScanMap + NoiseWeight
 * + project_signal, ops_scan_map.cpp:16-78, template_offset.cpp:243-327) on the crossing records
 * sorted by pixel BLOCK (tb_bx_block_pixels() consecutive local pixels): every WARP keeps the map
 * values of the block it works on in its own slice of shared memory (no atomics on the tile).
 *   tb_bx_pass1  writes (accumulate = 0) or adds to (accumulate = 1) the noise-weighted map of the
 *                amplitudes; with accumulate = 0 EVERY block of the local map is written, no
 *                zero-fill is needed.  chunk < 0: the whole map; chunk >= 0: the pixel chunk set
 *                by tb_obs_set_pixel_chunks (bounds must be multiples of the block size).
 *   tb_bx_pass2  projects the binned map for the amplitudes of the preceding tb_bx_pass1 call
 *                (whole map or one pixel chunk) and ADDS to amplitudes_out.
 *   tb_bx_fused  one observation on one GPU: pass 1 -> covariance_apply (toast_map_cov.cpp:471-528)
 *                -> pass 2 inside one kernel, the map never leaves the SM.  zmap_scratch
 *                ([n_local_pix, nnz]) is only touched for blocks that had to be cut into several
 *                work units (high-contention maps).  ADDS to amplitudes_out.  amplitudes ==
 *                NULL: the amplitudes of the preceding tb_bx_fused / tb_bx_pass1 call. */
int tb_bx_block_pixels(void);
int tb_obs_blocked(const tb_obs *obs);
int tb_obs_blocked_stats(const tb_obs *obs, int64_t *n_records, int64_t *n_units,
                         int64_t *n_multi_units, int64_t *n_blocks);
int tb_bx_pass1(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                double *zmap, int accumulate, int64_t chunk, void *stream);
int tb_bx_pass2(const tb_obs *obs, const double *binned, double *amplitudes_out, int64_t chunk,
                void *stream);
int tb_bx_fused(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                const double *cov, double *zmap_scratch, double *amplitudes_out, void *stream);
/* RHS projection (SolverRHS, mapmaker_solve.py:107-229): out += F^T N^-1 (signal - P m). */
int tb_rhs_project(const tb_obs *obs, const double *signal, const uint8_t *amp_flags,
                   const double *binned, double *amplitudes_out, int regen, void *stream);
/* Noise-weighted binning of a timestream with the observation's pointing (BinMap core). */
int tb_bin_signal(const tb_obs *obs, const double *signal, double *zmap, int regen,
                  void *stream);

/* ---- Offset template: noise prior and its preconditioner -------------------------------------
 * Replaces Offset._add_prior (templates/offset/offset.py:884-960: scipy.signal.convolve
 * mode="same" per (detector, observation, view) segment, then flagged amplitudes zeroed) and
 * Offset._apply_precond with use_noise_prior=True (:962-1010: scipy.linalg.cho_solve_banded on
 * the lower banded Cholesky factor, or a "same" convolution with the Toeplitz kernel when
 * precond_width <= 1).  The reference has no accelerator form of either (NotImplementedError,
 * :888-891 and :964-967).  The descriptor holds HOST arrays; they are copied to the device once.
 * Segments are disjoint, in increasing order; a start offset < 0 marks a cut detector (its
 * amplitudes come out as zeros). */
#define TB_PRECOND_TOEPLITZ 1
#define TB_PRECOND_BANDED 2
typedef struct {
    int64_t n_amp;              /* length of the local amplitude vector */
    int64_t n_seg;              /* number of segments */
    const int64_t *seg_start;   /* [n_seg] first amplitude of the segment */
    const int64_t *seg_len;     /* [n_seg] n_amp_view */
    const int64_t *filt_start;  /* [n_seg] offset of the noise filter in `filters`, or -1 */
    const int64_t *filt_len;    /* [n_seg] its (odd) length */
    const double *filters;      /* [n_filter_values] concatenated filters (offset.py:466-468) */
    int64_t n_filter_values;
    int precond_mode;           /* TB_PRECOND_TOEPLITZ or TB_PRECOND_BANDED */
    const int64_t *prec_start;  /* [n_seg] offset in `precond`, or -1 */
    const int64_t *prec_width;  /* [n_seg] banded: rows w of the factor; Toeplitz: kernel length */
    const double *precond;      /* banded: per segment the [w, n_amp_view] row-major array that
                                   scipy.linalg.cholesky_banded(lower=True) returns
                                   (ab[k][j] = L[j+k][j]); Toeplitz: the kernels */
    int64_t n_precond_values;
} tb_offset_prior_desc;
typedef struct tb_offset_prior tb_offset_prior;
tb_offset_prior *tb_offset_prior_create(const tb_offset_prior_desc *desc);
void tb_offset_prior_destroy(tb_offset_prior *prior);
/* amplitudes_out[seg] += convolve(amplitudes_in[seg], filter[seg], "same"); flagged -> 0 */
int tb_offset_prior_add(const tb_offset_prior *prior, const double *amplitudes_in,
                        const uint8_t *amplitude_flags, double *amplitudes_out, int mem,
                        void *stream);
/* amplitudes_out = M^-1 amplitudes_in segment by segment; flagged -> 0 */
int tb_offset_prior_precond(const tb_offset_prior *prior, const double *amplitudes_in,
                            const uint8_t *amplitude_flags, double *amplitudes_out, int mem,
                            void *stream);

/* ---- a6 fused with its collective: map reduction + covariance over NVLink peer memory ------
 * Replaces  accel_update_host -> PixelData.sync_allreduce (MPI) -> accel_update_device ->
 * covariance_apply  (ops/mapmaker_utils/mapmaker_utils.py:885-925, pixels.py:710-779,
 * covariance.py:262-306) by ONE kernel per GPU: P2P reduce-scatter of the map slice this rank
 * owns, 3x3 covariance product on that slice, P2P all-gather into every rank's map, bracketed by
 * device-side flag barriers.  The map buffer is allocated by the library (peer-visible through
 * CUDA IPC); handles are 128 bytes per rank and are exchanged by the caller (any transport).   */
typedef struct tb_peer tb_peer;
tb_peer *tb_peer_create(int rank, int world, size_t map_bytes);
int tb_peer_get_handles(tb_peer *peer, void *out128);
int tb_peer_open(tb_peer *peer, const void *all_handles /* world x 128 bytes, by rank */);
void *tb_peer_map_ptr(tb_peer *peer);
/* n_pix = n_local_submap * n_pix_submap (multiple of 256); cov [n_pix,6] device pointer. */
int tb_map_reduce_cov(tb_peer *peer, int64_t n_pix, const double *cov, void *stream);
/* The same for the local pixel range [pix_first, pix_first + n_pix) only (both multiples of 256):
 * lets the caller pipeline the reduction of one part of the map with the passes over the next.
 * Every rank must issue the same sequence of calls, stream-ordered per peer object. */
int tb_map_reduce_cov_range(tb_peer *p, int64_t pix_first, int64_t n_pix, const double *cov,
                            void *stream);
void tb_peer_destroy(tb_peer *peer);
/* NVLS form: attach to buffers the caller already made peer-visible (symmetric memory).
 * `maps` / `flags` are world-long, rank-ordered arrays of device addresses (flags: 2 x 16 uint64
 * per rank, zeroed); mc_map is the NVSwitch MULTICAST address of the map buffer (0 = none).  With
 * a multicast address tb_map_reduce_cov sums the map inside the switch (multimem.ld_reduce),
 * applies the covariance to this rank's slice and broadcasts it with multimem.st: about
 * (1 + 1/N) |map| of NVLink traffic per direction instead of 2 (N-1)/N |map|.                 */
tb_peer *tb_peer_attach(int rank, int world, size_t map_bytes, const uint64_t *maps,
                        const uint64_t *flags, uint64_t mc_map);
int tb_peer_has_multicast(const tb_peer *peer);
int tb_peer_set_multimem(int on); /* A/B switch: 0 = P2P kernel even when multicast exists */

/* ---- a12/a13  amplitude-vector arithmetic for the PCG loop (templates/amplitudes.py:201-274,
 * :523-571; ops/mapmaker_solve.py:665-746).  All DEVICE pointers; scalars live on the device
 * so an iteration needs no host round trip.  n < 0, a NULL scalar pointer (delta, dq, out,
 * sums) or a NULL vector when n > 0 (tb_amp_dot's flags excepted) is refused with TB_ERR_ARG
 * before anything is launched.                                                              */
/* out[0] = sum_{flags==0} a*b, every entry when flags is NULL (deterministic two-stage
 * reduction) */
int tb_amp_dot(const double *a, const double *b, const uint8_t *flags, int64_t n,
               double *out, void *stream);
/* alpha = delta[0]/dq[0];  x += alpha d;  r -= alpha q;  s = flag ? 0 : r*var;
 * sums[0] = r.r, sums[1] = s.r  (masked by flags).                                          */
int tb_pcg_update(const double *delta, const double *dq, double *x, double *r,
                  const double *d, const double *q, double *s, const double *offset_var,
                  const uint8_t *flags, int64_t n, double *sums, void *stream);
/* beta = delta_new[0]/delta_old[0];  d = s + beta d */
int tb_pcg_direction(const double *delta_new, const double *delta_old, double *d,
                     const double *s, int64_t n, void *stream);

/* Build (or rebuild, after the flags / global2local changed) the solver's compact copy of the
 * stored pointing: int32 local pixel with flags and global2local folded in + the (Q,U) weights as
 * one 16-byte record = 20 B / det-sample instead of 33 B, bit-identical values.  The LHS passes
 * use it when present.  If the I weight is not the per-detector constant cal[det] the copy is
 * discarded and the general kernels keep running.                                           */
int tb_obs_pack_pointing(tb_obs *obs, void *stream);
int tb_obs_has_compact_pointing(const tb_obs *obs);
/* 1 if packing also found (and verified on every in-interval sample, to 1e-13 relative) that the
 * (Q,U) weights of every detector pair (2p, 2p+1) are related by a fixed per-pair rotation-scale
 * (ops_stokes_weights.cpp:95-139: both are eta*cal*(cos,sin) of angles that differ by a
 * constant).  The LHS passes then stream one weight record per PAIR: 12 B / det-sample.      */
int tb_obs_has_pair_weights(const tb_obs *obs);
/* Crossing list built by tb_obs_pack_pointing: consecutive samples of a detector (pair) that share
 * the pixel and the baseline are collapsed into one 32-byte record {lp0, lp1, n, amp | sum Q,
 * sum U}; both LHS passes are linear in the weights, so they stream records instead of samples
 * (tb_solver.cu: k_lhs_x).  Built only when it is the smaller stream.  n_records = 0: not built.
 * Intensity observations: 16-byte records {lp0, lp1, n, amp} (no weight sums), always built; their
 * rows are detector pairs only when that gives the block-ordered list fewer entries (a record
 * whose two detectors fall in different pixels takes two), and pairs need no weight relation. */
int tb_obs_crossing_stats(const tb_obs *obs, int64_t *n_records, int64_t *n_rows, int *paired);

/* Runtime options (A/B measurements, debugging; each LHS switch selects a path that is the only
 * one to run on some input, so that tests can reach it on small problems):
 *   "blocked" (default 1)  the solver runs the LHS on the block-ordered crossing list (tb_bx_*)
 *                          when it has been built
 *   "crossings" (default 1) tb_lhs_pass1 / tb_lhs_pass2 use the time-ordered crossing list when
 *                          it has been built
 *   "pair"    (default 1)  otherwise, on the compact pointing, process detector rows two at a time
 *                          so that co-pointed detectors (polarisation pairs) share one RED triple /
 *                          map gather per sample; 0: the per-sample kernels on the stored pointing
 *   "pairw"   (default 1)  with "pair": stream one (Q,U) record per detector pair when the
 *                          packed pointing verified the fixed weight rotation of every pair
 *   "peer_ctas", "prior_chunk"  launch shapes of the map reduction and of the noise prior
 * Any other name is unknown: tb_set_option fails with TB_ERR_ARG, tb_get_option returns -1. */
int tb_set_option(const char *name, int value);
int tb_get_option(const char *name); /* -1 if unknown */

/* ---- test hooks ------------------------------------------------------------------------- */
/* Scale the guard band that routes a sample to the exact (double-double atan2) pixel path;
 * 1.0 = production, 0.0 = fast path only, large = every sample takes the exact path.      */
void tb_set_pixel_guard_scale(double scale);
/* Number of samples that took the exact pixel path since the last reset. */
int64_t tb_pixel_exact_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* TOAST_B200_H */
