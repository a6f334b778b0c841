// tb_obs.cuh -- the native observation handle shared by the solver translation units
// (tb_solver.cu: per-sample and crossing-list passes; tb_blocked.cu: the block-ordered crossing
// list with shared-memory map tiles).
#pragma once

#include <vector>

#include "tb_device.cuh"
#include "tb_runtime.cuh"
#include "tb_wcs.cuh"

using tbd::Views;

struct tb_obs {
    void *blob = nullptr; // one device allocation holding every small array
    Views V;
    // device arrays inside blob
    const int64_t *amp_view_off = nullptr;
    const int64_t *amp_offsets = nullptr;
    const int64_t *g2l = nullptr;
    const double *fp = nullptr;      // [n_det,4]
    const double *cal = nullptr;
    const double *eta = nullptr;     // (1-eps)/(1+eps)
    const double *gamma = nullptr;
    const double *det_scale = nullptr;
    tb_obs_desc d; // copy of the descriptor (host pointers in it are NOT kept alive)
    int is_wcs = 0; // pixels of a flat projection (tb_obs_create_wcs): regenerated with `wcs`
    tbw::Wcs wcs{};
    // Stokes values per pixel: 3 (I, Q, U; weights [n_det, n_samp, 3]) or 1 (intensity only,
    // tb_obs_create_intensity; weights [n_det, n_samp] = cal[det]).  Intensity observations
    // keep no (Q, U) arrays: wqu, xqu and bqu stay NULL, and lpp / pair_rot are never built.
    int nnz = 3;
    int64_t n_amp_det = 0;
    // compact solver pointing (tb_obs_pack_pointing): local pixel (int32, <0 = nothing to do)
    // and the two sample-dependent weights (Q, U) as one 16-byte record
    int32_t *lpix = nullptr;
    double2 *wqu = nullptr;
    // detector-pair form of the compact pointing (tb_obs_pack_pointing): both local pixels of a
    // pair as one 8-byte record, and the fixed 2x2 rotation-scale that maps the (Q,U) weights of
    // detector 2p onto those of detector 2p+1 -- verified sample by sample while packing
    int2 *lpp = nullptr;        // [n_pair][n_samp]
    double2 *pair_rot = nullptr; // [n_pair] (A, B): (q1, u1) = (A q0 - B u0, B q0 + A u0)
    // crossing list (see k_lhs_x): one record per run of samples that share pixel(s) and baseline
    int4 *xrec = nullptr;       // [n_xrec] {lp0, lp1, n_samples, amp_rel}
    double2 *xqu = nullptr;     // [n_xrec] sum over the run of the (Q,U) weights
    int4 *xblocks = nullptr;    // [n_xblocks] {row, first record, end record, 0}
    int64_t n_xrec = 0, n_xblocks = 0, n_xrows = 0;
    int x_paired = 0;           // rows are detector pairs (weights shared through pair_rot)
    double4 *stable = nullptr;  // [n_xrows] {cal0, cal1, A, B} (A = B = 0 for intensity)
    // block-ordered crossing list (tb_blocked.cu): the time-ordered records stably sorted by
    // PIXEL BLOCK (kBxPix consecutive local pixels), i.e. in (block, row, time) order.  A CTA owns
    // one block at a time and keeps its 3 x kBxPix map values in shared memory.
    double *ascaled = nullptr;  // per-pass scratch [slot]{a0 w0, a1 w1, w0, w1} (k_bx_prescale)
    int2 *brec = nullptr;       // [n_brec] {pixel in block | n0 << kBxShift | n1 << (kBxShift+6), scaled-amplitude index}
    double2 *bqu = nullptr;     // [n_brec] (sum Q, sum U)
    int4 *bunits = nullptr;     // [n_bunits] {block, first record, end record, 1 if the block has several units}
    int4 *bunits_single = nullptr, *bunits_multi = nullptr; // the same units split by that flag
    int32_t *bmulti_blocks = nullptr;                       // blocks that have several units
    int64_t n_brec = 0, n_bunits = 0, n_bunits_single = 0, n_bunits_multi = 0, n_bmulti_blocks = 0;
    int64_t n_local_pix = 0;    // n_local_submap * n_pix_submap (from global2local)
    std::vector<int4> bunits_host;          // host copy of bunits (chunk lookup)
    std::vector<int64_t> bchunk_unit;       // unit ranges of the pixel chunks
    int s_uniform = 0;          // every row has the same {cal0, cal1, A, B}: kernel constants
    double s_const[4] = {0, 0, 0, 0};
};


// ---- shared between tb_solver.cu and tb_blocked.cu ---------------------------------------------
// per-row constants {cal0, cal1, A, B} and their uniformity (tb_solver.cu)
void tb_build_row_table(tb_obs *obs);
// block-ordered crossing list (tb_blocked.cu); frees a previous one
void tb_build_blocked(tb_obs *obs, cudaStream_t st);
void tb_free_blocked(tb_obs *obs);
// unit ranges of the pixel chunks; chunked calls are refused when a bound is not block-aligned
void tb_blocked_set_chunks(tb_obs *obs, int64_t n_chunks, const int64_t *pixel_bounds);
extern int g_use_bx;
