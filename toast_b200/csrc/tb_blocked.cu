// tb_blocked.cu -- the LHS passes on the BLOCK-ORDERED crossing list: shared-memory privatised
// map tiles (the binning design of the north star).
//
// What the reference does per PCG iteration (ops/mapmaker_solve.py:342-506) is, per sample,
//   pass 1   zmap[pixel] += F a * w_det * weights          (template_offset.cpp:93-121 +
//                                                            ops_mapmaker_utils.cpp:15-86,295-377)
//            zmap <- all-reduce;  m = C zmap                (pixels.py:710-779, toast_map_cov.cpp:471-528)
//   pass 2   out[baseline] += w_det (F a - weights . m)     (ops_scan_map.cpp:16-78,
//                                                            ops_noise_weight.cpp:101-114,
//                                                            template_offset.cpp:243-327)
// The crossing list (tb_solver.cu: k_xbuild) already collapses every run of samples that share
// (pixel, baseline) into one record; both passes are linear in the record's (n, sum Q, sum U).
//
// Here the records are stably sorted by PIXEL BLOCK (kBxPix = 128 consecutive local pixels), which
// leaves them in (block, row, time) order, and every WARP owns one block at a time:
//   * the map side is private to the warp: the 3 x 128 doubles of its block live in the warp's
//     3 KB slice of shared memory.  Pass 1 accumulates into it with PLAIN read-modify-writes --
//     lanes of one step that hit the same pixel (found with match.any) take turns -- and flushes
//     the finished tile with coalesced 16-byte stores: no zero-fill of the map, no atomics at all
//     when the block is one work unit.  (Blocks with more than kBxUnitMax records -- the
//     high-contention maps of ground patches -- are cut into units whose tiles are flushed with
//     fp64 REDs: one RED per touched pixel value and unit instead of three per record.)
//     fp64 atomicAdd on shared memory is a compare-and-swap loop on this architecture
//     (ATOMS.CAST.SPIN); a CTA-wide tile updated with it left the kernel bound by the shared-
//     memory pipe at 80 % utilisation (profiles/r2_ncu_blocked.txt), which is why the tile is
//     warp-private;
//   * the amplitude side keeps its time locality: consecutive records of a detector's track
//     through the block share the baseline, so the 16 / 32-byte amplitude gather of a warp touches
//     a handful of sectors (5.5 M sectors for 39.6 M records on the C4 shard) and pass 2 issues
//     one RED per baseline run (segmented warp sum) instead of one per record;
//   * there is no block-level barrier: a warp streams its unit's records with a register software
//     pipeline (records two steps ahead, amplitude gathers one step ahead).
// On one GPU with one observation nothing has to leave the SM between the passes: the fused
// kernel (k_bx<2>) accumulates the tile, applies the 3x3 pixel covariance in shared memory and
// projects the same records (second read served by the L2) -- the map never touches HBM.
// Intensity-only observations (tb_obs::nnz = 1) run the same kernels with NNZ = 1: records
// without (sum Q, sum U), a tile of kBxPix doubles per warp and one tile update per record.
#include <algorithm>

#include "tb_obs.cuh"

using namespace tbd;

namespace tbr {
void sort_pairs_i32(const int32_t *keys_in, int32_t *keys_out, const int32_t *vals_in,
                    int32_t *vals_out, int64_t n, int end_bit, cudaStream_t st); // tb_sort.cu
}

int g_use_bx = 1; // tb_set_option("blocked", 0/1)

namespace {

#ifndef TB_BX_SHIFT
#define TB_BX_SHIFT 7
#endif
#ifndef TB_BX_CTAS
#define TB_BX_CTAS 4
#endif

constexpr int kBxShift = TB_BX_SHIFT;
constexpr int kBxPix = 1 << kBxShift;   // pixels per block: 3 x kBxPix doubles of shared memory per warp
constexpr int kBxUnitMax = 16384;       // records per work unit (one warp)
constexpr int kBxRowBits = 32 - (kBxShift + 12); // free bits of the first record word
static_assert(kBxRowBits >= 1, "pixel | n0 | n1 must fit one int");

// ---- build ---------------------------------------------------------------------------------------
// keys / values for the stable sort by block.  value = record index | mode << 30 (0: as recorded,
// 1: detector 0 only, 2: detector 1 only).  TWO_SLOT: entry 2i is the record itself, entry 2i + 1
// its second pixel when the two detectors of the row fall in different pixels (rare; the one-slot
// form is used when that never happens).  Entries with nothing on the map get key n_blocks.
template <bool TWO_SLOT>
__global__ void __launch_bounds__(kThreads)
k_bx_keys(const int4 *__restrict__ xrec, int64_t n_rec, int32_t n_blocks, int32_t *__restrict__ keys,
          int32_t *__restrict__ vals, unsigned int *__restrict__ counters /* {split, invalid, off-map} */) {
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n_rec;
         i += (int64_t)gridDim.x * kThreads) {
        const int4 r = xrec[i];
        int32_t key = n_blocks, val = (int32_t)i, key2 = n_blocks, val2 = (int32_t)i | (2 << 30);
        if (r.x == -2 || r.y == -2) atomicAdd(counters + 2, 1u);
        if (r.x >= 0) {
            key = r.x >> kBxShift;
            if (r.y >= 0 && r.y != r.x) {
                val |= (1 << 30);
                key2 = r.y >> kBxShift;
                atomicAdd(counters, 1u);
            }
        } else if (r.y >= 0) {
            key = r.y >> kBxShift;
        }
        if (key == n_blocks) atomicAdd(counters + 1, 1u);
        if (TWO_SLOT) {
            keys[2 * i] = key;
            vals[2 * i] = val;
            keys[2 * i + 1] = key2;
            vals[2 * i + 1] = val2;
            if (key2 == n_blocks) atomicAdd(counters + 1, 1u);
        } else {
            keys[i] = key;
            vals[i] = val;
        }
    }
}

template <int NNZ> // 1: intensity records carry no (sum Q, sum U)
__global__ void __launch_bounds__(kThreads)
k_bx_gather(const int4 *__restrict__ xrec, const double2 *__restrict__ xqu,
            const int32_t *__restrict__ vals, int64_t n_sorted, int64_t n_amp_det, int row_in_rec,
            int2 *__restrict__ brec, double2 *__restrict__ bqu) {
    for (int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x; j < n_sorted;
         j += (int64_t)gridDim.x * kThreads) {
        const int32_t v = vals[j];
        const int32_t i = v & 0x3FFFFFFF, mode = (v >> 30) & 3;
        const int4 r = xrec[i];
        const int n = r.z & 0xFF, row = (int)((unsigned)r.z >> 8);
        const int n0 = (r.x >= 0 && mode != 2) ? n : 0;
        const int n1 = (r.y >= 0 && mode != 1 && (mode == 2 || r.x < 0 || r.y == r.x)) ? n : 0;
        const int32_t pix = (mode == 2 || r.x < 0) ? r.y : r.x;
        // (the row rides in the upper bits when it fits: pass 2 then needs no division)
        brec[j] = make_int2((pix & (kBxPix - 1)) | (n0 << kBxShift) | (n1 << (kBxShift + 6)) |
                                (row_in_rec ? (row << (kBxShift + 12)) : 0),
                            (int32_t)((int64_t)row * n_amp_det + r.w));
        if constexpr (NNZ == 3) bqu[j] = xqu[i];
    }
}

// first sorted entry whose key is >= b, for b = 0 .. n_blocks
__global__ void k_bx_block_starts(const int32_t *__restrict__ keys, int64_t n, int32_t n_blocks,
                                  int32_t *__restrict__ start) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > n_blocks) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (keys[mid] < b) lo = mid + 1;
        else hi = mid;
    }
    start[b] = (int32_t)lo;
}

// ---- the passes ----------------------------------------------------------------------------------
// Amplitudes travel through a per-pass scratch array laid out by ROW of the crossing list and
// baseline, so that a record addresses it with its `slot` alone:
//   ascaled[slot] = {a0 w0, a1 w1, w0, w1}   amplitude x detector weight and the weight itself of
//                                            the two detectors of a pair (32 bytes = one sector;
//                                            unpaired rows: {a w, w}); flagged baselines and the
//                                            missing partner of an odd detector count hold zeros,
//                                            so the passes need neither flag tests nor row lookups
__global__ void __launch_bounds__(kThreads)
k_bx_prescale(int paired, int n_det, int64_t nad, const int64_t *__restrict__ amp_offsets,
              const double *__restrict__ det_scale, const double *__restrict__ amps,
              const uint8_t *__restrict__ aflags, double *__restrict__ ascaled) {
    const int row = blockIdx.x;
    const int d0 = paired ? 2 * row : row, d1 = d0 + 1;
    const bool has1 = paired && d1 < n_det;
    const int64_t o0 = __ldg(amp_offsets + d0), o1 = has1 ? __ldg(amp_offsets + d1) : 0;
    const double w0 = __ldg(det_scale + d0), w1 = has1 ? __ldg(det_scale + d1) : 0.0;
    for (int64_t i = (int64_t)blockIdx.y * kThreads + threadIdx.x; i < nad;
         i += (int64_t)gridDim.y * kThreads) {
        const bool g0 = __ldg(aflags + o0 + i) == 0;
        const double2 t0 = bx_scaled(g0, g0 ? __ldg(amps + o0 + i) : 0.0, w0);
        if (paired) {
            const bool g1 = has1 && __ldg(aflags + o1 + i) == 0;
            const double2 t1 = bx_scaled(g1, g1 ? __ldg(amps + o1 + i) : 0.0, w1);
            double2 *dst = reinterpret_cast<double2 *>(ascaled) + 2 * ((int64_t)row * nad + i);
            dst[0] = make_double2(t0.x, t1.x);
            dst[1] = make_double2(t0.y, t1.y);
        } else {
            reinterpret_cast<double2 *>(ascaled)[(int64_t)row * nad + i] = t0;
        }
    }
}

// The PCG's next direction (k_pcg_direction) fused with the prescale of that direction for the
// next LHS and the zero-fill of the LHS output, in one pass over the rows x baselines of
// k_bx_prescale: d = d beta + s, ascaled from the new d, q = 0.  The rows must cover the
// amplitude vector (tb_bx_direction_prescale checks it), so every entry of d is advanced once.
// delta_old <- delta_new is stored by the last CTA to finish: every CTA reads delta_old (thread
// 0, before its counter increment) ahead of that store.
__global__ void __launch_bounds__(kThreads)
k_pcg_direction_prescale(int paired, int n_det, int64_t nad, const int64_t *__restrict__ amp_offsets,
                         const double *__restrict__ det_scale, const double *dnew, double *dold,
                         double *__restrict__ d, const double *__restrict__ s,
                         const uint8_t *__restrict__ aflags, double *__restrict__ q,
                         double *__restrict__ ascaled, unsigned int *counter) {
    __shared__ double beta_sh;
    if (threadIdx.x == 0) beta_sh = dnew[0] / dold[0];
    __syncthreads();
    const double beta = beta_sh;
    const int row = blockIdx.x;
    const int d0 = paired ? 2 * row : row, d1 = d0 + 1;
    const bool has1 = paired && d1 < n_det;
    const int64_t o0 = __ldg(amp_offsets + d0), o1 = has1 ? __ldg(amp_offsets + d1) : 0;
    const double w0 = __ldg(det_scale + d0), w1 = has1 ? __ldg(det_scale + d1) : 0.0;
    for (int64_t i = (int64_t)blockIdx.y * kThreads + threadIdx.x; i < nad;
         i += (int64_t)gridDim.y * kThreads) {
        const double n0 = pcg_direction(d[o0 + i], beta, s[o0 + i]);
        d[o0 + i] = n0;
        q[o0 + i] = 0.0;
        const bool g0 = __ldg(aflags + o0 + i) == 0;
        const double2 t0 = bx_scaled(g0, n0, w0);
        if (paired) {
            bool g1 = false;
            double n1 = 0.0;
            if (has1) {
                n1 = pcg_direction(d[o1 + i], beta, s[o1 + i]);
                d[o1 + i] = n1;
                q[o1 + i] = 0.0;
                g1 = __ldg(aflags + o1 + i) == 0;
            }
            const double2 t1 = bx_scaled(g1, n1, w1);
            double2 *dst = reinterpret_cast<double2 *>(ascaled) + 2 * ((int64_t)row * nad + i);
            dst[0] = make_double2(t0.x, t1.x);
            dst[1] = make_double2(t0.y, t1.y);
        } else {
            reinterpret_cast<double2 *>(ascaled)[(int64_t)row * nad + i] = t0;
        }
    }
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(counter, 1u) == gridDim.x * gridDim.y - 1) {
            dold[0] = dnew[0];
            *counter = 0u;
        }
    }
}

struct BxArgs {
    const int4 *units;        // {block, first record, end record, multi}
    const int2 *brec;
    const double2 *bqu;       // NULL for intensity observations
    const double *ascaled;    // k_bx_prescale
    double *out;              // pass 2 / fused: amplitudes (REDs)
    const int64_t *amp_offsets;
    int32_t nad, n_det;
    double4 cst;              // {cal0, cal1, A, B} when uniform
    const double4 *table;     // per row otherwise
    double inv_nad;           // 1 / n_amp_det
    int64_t n_pix;            // local map size
    double *zmap;             // pass 1: output;  pass 2: the binned map;  fused: unused
    const double *cov;        // fused: [n_pix, nnz (nnz + 1) / 2]
    int accumulate;           // pass 1: add to zmap (REDs) even for single-unit blocks
};

// Every WARP owns one pixel block at a time and keeps the block's 3 x kBxPix map values in its own
// slice of shared memory, so the accumulation needs no atomics at all: lanes of one warp that hit
// the same pixel in the same step (found with match.any) take turns, everything else is a plain
// shared-memory read-modify-write.  (fp64 / fp32 atomicAdd on shared memory is a compare-and-swap
// loop on this architecture -- ATOMS.CAST.SPIN -- and a CTA-wide tile with such atomics left the
// kernel bound by the shared-memory pipe at 80 % utilisation: profiles/r2_ncu_blocked.txt.)  There
// is no block-level barrier anywhere: a warp streams its unit's records with a register software
// pipeline (records two steps ahead, amplitude gathers one step ahead).
constexpr int kBxWarps = kThreads / 32;

struct BxRec {
    int2 r;     // {pixel | n0 << kBxShift | n1 << (kBxShift + 6), slot}
    double2 qu; // (sum Q, sum U)
};
template <bool KEEP_IN_L2, int NNZ>
__device__ __forceinline__ BxRec bx_load(const BxArgs &a, int i, int end, int lane) {
    BxRec x;
    x.r = make_int2(0, -1 - lane); // idle lanes: n0 = n1 = 0, distinct negative slots
    x.qu = make_double2(0.0, 0.0);
    if (i < end) {
        x.r = KEEP_IN_L2 ? __ldg(a.brec + i) : __ldcs(a.brec + i);
        if constexpr (NNZ == 3) x.qu = KEEP_IN_L2 ? __ldg(a.bqu + i) : __ldcs(a.bqu + i);
    }
    return x;
}

struct BxAmp {
    double2 t; // a0 w0, a1 w1
    double2 w; // w0, w1 (pass 2 only)
};
template <bool PAIRED, bool NEED_W>
__device__ __forceinline__ BxAmp bx_gather(const BxArgs &a, int32_t slot) {
    BxAmp g;
    g.t = g.w = make_double2(0.0, 0.0);
    if (slot >= 0) {
        if (PAIRED) {
            const double2 *p = reinterpret_cast<const double2 *>(a.ascaled) + 2 * (int64_t)slot;
            g.t = __ldg(p);
            if (NEED_W) g.w = __ldg(p + 1);
        } else {
            const double2 v = __ldg(reinterpret_cast<const double2 *>(a.ascaled) + slot);
            g.t.x = v.x;
            g.w.x = v.y;
        }
    }
    return g;
}

template <bool UNIFORM>
__device__ __forceinline__ double4 bx_consts(const BxArgs &a, int32_t slot) {
    if (UNIFORM) return a.cst;
    const int row = (int)fast_div((int64_t)(slot < 0 ? 0 : slot), a.inv_nad);
    const double2 *tp = reinterpret_cast<const double2 *>(a.table + row);
    const double2 ca = __ldg(tp), cb = __ldg(tp + 1);
    return make_double4(ca.x, ca.y, cb.x, cb.y);
}

// one pass-1 step: the 32 records of `x` (amplitudes already gathered in `g`) into the tile
// (NNZ = 1: the tile holds one value per pixel and only the first term is formed)
template <bool UNIFORM, bool PAIRED, int NNZ>
__device__ __forceinline__ void bx_acc_step(const BxArgs &a, double *tile, const BxRec &x,
                                            const BxAmp &g, int lane) {
    const int p = x.r.x & (kBxPix - 1);
    const int n0 = (x.r.x >> kBxShift) & 63, n1 = (x.r.x >> (kBxShift + 6)) & 63;
    const double4 c = bx_consts<UNIFORM>(a, x.r.y);
    const double t0 = n0 ? g.t.x : 0.0;
    const double t1 = (PAIRED && n1) ? g.t.y : 0.0;
    const bool contrib = t0 != 0.0 || t1 != 0.0;
    const double v0 = t0 * (c.x * (double)n0) + t1 * (c.y * (double)n1);
    const double v1 = t0 * x.qu.x + t1 * (c.z * x.qu.x - c.w * x.qu.y);
    const double v2 = t0 * x.qu.y + t1 * (c.w * x.qu.x + c.z * x.qu.y);
    // lanes of this step that hit the same pixel take turns (typically the two records of one
    // crossing cut by a baseline boundary); all others update their pixel at once
    const unsigned same = __match_any_sync(0xffffffffu, contrib ? p : kBxPix + lane);
    const int rank = __popc(same & ((1u << lane) - 1u));
    const int rounds = __reduce_max_sync(0xffffffffu, rank);
    double *z = tile + NNZ * p;
    if (rounds == 0) {
        if (contrib) {
            z[0] += v0;
            if constexpr (NNZ == 3) {
                z[1] += v1;
                z[2] += v2;
            }
        }
        __syncwarp();
    } else {
        for (int r = 0; r <= rounds; ++r) {
            if (contrib && rank == r) {
                z[0] += v0;
                if constexpr (NNZ == 3) {
                    z[1] += v1;
                    z[2] += v2;
                }
            }
            __syncwarp();
        }
    }
}

// pass 1 over the records [first, end) of the warp's unit: tile += a w (n cal, sum Q, sum U).
// Software pipeline without register rotation (three record buffers, loop unrolled by three):
// records are loaded two steps ahead, amplitudes gathered one step ahead.
template <bool UNIFORM, bool PAIRED, bool KEEP_IN_L2, int NNZ>
__device__ __forceinline__ void bx_accumulate(const BxArgs &a, double *tile, int first, int end,
                                              int lane) {
    if (first >= end) return;
    BxRec A = bx_load<KEEP_IN_L2, NNZ>(a, first + lane, end, lane);
    BxRec B = bx_load<KEEP_IN_L2, NNZ>(a, first + 32 + lane, end, lane);
    BxRec C;
    BxAmp gA = bx_gather<PAIRED, false>(a, A.r.y), gB, gC;
    for (int base = first; base < end; base += 96) {
        C = bx_load<KEEP_IN_L2, NNZ>(a, base + 64 + lane, end, lane);
        gB = bx_gather<PAIRED, false>(a, B.r.y);
        bx_acc_step<UNIFORM, PAIRED, NNZ>(a, tile, A, gA, lane);
        if (base + 32 >= end) break;
        A = bx_load<KEEP_IN_L2, NNZ>(a, base + 96 + lane, end, lane);
        gC = bx_gather<PAIRED, false>(a, C.r.y);
        bx_acc_step<UNIFORM, PAIRED, NNZ>(a, tile, B, gB, lane);
        if (base + 64 >= end) break;
        B = bx_load<KEEP_IN_L2, NNZ>(a, base + 128 + lane, end, lane);
        gA = bx_gather<PAIRED, false>(a, A.r.y);
        bx_acc_step<UNIFORM, PAIRED, NNZ>(a, tile, C, gC, lane);
    }
}

// one pass-2 step: out[baseline] += w (n a - (n cal, sum Q, sum U) . m), one RED pair per run of
// records that share the baseline (consecutive in (row, time) order)
template <bool UNIFORM, bool PAIRED, int NNZ>
__device__ __forceinline__ void bx_proj_step(const BxArgs &a, const double *tile, const BxRec &x,
                                             const BxAmp &g, int lane) {
    const int p = x.r.x & (kBxPix - 1);
    const int n0 = (x.r.x >> kBxShift) & 63, n1 = (x.r.x >> (kBxShift + 6)) & 63;
    const double4 c = bx_consts<UNIFORM>(a, x.r.y);
    const double m0 = tile[NNZ * p];
    const double m1 = NNZ == 3 ? tile[NNZ * p + 1] : 0.0, m2 = NNZ == 3 ? tile[NNZ * p + 2] : 0.0;
    double val0 = 0.0, val1 = 0.0;
    if (n0) {
        double sc = (c.x * (double)n0) * m0;
        if constexpr (NNZ == 3) {
            sc += x.qu.x * m1;
            sc += x.qu.y * m2;
        }
        val0 = (double)n0 * g.t.x - sc * g.w.x;
    }
    if (PAIRED && n1) {
        const double q1 = c.z * x.qu.x - c.w * x.qu.y, u1 = c.w * x.qu.x + c.z * x.qu.y;
        double sc = (c.y * (double)n1) * m0;
        if constexpr (NNZ == 3) {
            sc += q1 * m1;
            sc += u1 * m2;
        }
        val1 = (double)n1 * g.t.y - sc * g.w.y;
    }
    const Runs rr = find_runs32<8>(x.r.y, lane);
    val0 = seg_sum<8>(val0, rr);
    if (PAIRED) val1 = seg_sum<8>(val1, rr);
    if (rr.is_tail && x.r.y >= 0) {
        const int row = (int)((unsigned)x.r.x >> (kBxShift + 12)); // (rows fit: tb_build_blocked)
        const int arel = x.r.y - row * a.nad;
        const int d0 = PAIRED ? 2 * row : row;
        if (val0 != 0.0) atomicAdd(a.out + __ldg(a.amp_offsets + d0) + arel, val0);
        if (PAIRED && val1 != 0.0) atomicAdd(a.out + __ldg(a.amp_offsets + d0 + 1) + arel, val1);
    }
}

template <bool UNIFORM, bool PAIRED, int NNZ>
__device__ __forceinline__ void bx_project(const BxArgs &a, const double *tile, int first, int end,
                                           int lane) {
    if (first >= end) return;
    BxRec A = bx_load<false, NNZ>(a, first + lane, end, lane);
    BxRec B = bx_load<false, NNZ>(a, first + 32 + lane, end, lane);
    BxRec C;
    BxAmp gA = bx_gather<PAIRED, true>(a, A.r.y), gB, gC;
    for (int base = first; base < end; base += 96) {
        C = bx_load<false, NNZ>(a, base + 64 + lane, end, lane);
        gB = bx_gather<PAIRED, true>(a, B.r.y);
        bx_proj_step<UNIFORM, PAIRED, NNZ>(a, tile, A, gA, lane);
        if (base + 32 >= end) break;
        A = bx_load<false, NNZ>(a, base + 96 + lane, end, lane);
        gC = bx_gather<PAIRED, true>(a, C.r.y);
        bx_proj_step<UNIFORM, PAIRED, NNZ>(a, tile, B, gB, lane);
        if (base + 64 >= end) break;
        B = bx_load<false, NNZ>(a, base + 128 + lane, end, lane);
        gA = bx_gather<PAIRED, true>(a, A.r.y);
        bx_proj_step<UNIFORM, PAIRED, NNZ>(a, tile, C, gC, lane);
    }
}

// MODE 0: pass 1 (tile -> zmap), 1: pass 2 (binned map -> tile -> amplitudes), 2: fused.
// One warp per work unit, eight consecutive units per CTA; grid = ceil(n_units / 8).
// NNZ: map values per pixel, 3 (I, Q, U) or 1 (intensity: the map is [n_pix], cov [n_pix]).
template <int MODE, bool UNIFORM, bool PAIRED, int NNZ>
__global__ void __launch_bounds__(kThreads, TB_BX_CTAS)
k_bx(const BxArgs a, int64_t n_units) {
    __shared__ __align__(16) double tiles[kBxWarps][NNZ * kBxPix];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *tile = tiles[warp];
    double2 *tile2 = reinterpret_cast<double2 *>(tile);
    const int64_t g_end = NNZ * a.n_pix;
    // (persistent warps taking tickets from a global counter measured slower than this static
    // assignment -- 0.88 vs 0.78 ms for the fused kernel on the C4 shard, profiles/README.md:
    // concurrently running neighbours share their amplitude sectors in the L1 / L2)
    {
        const int64_t ticket = (int64_t)blockIdx.x * kBxWarps + warp;
        if (ticket >= n_units) return;
        const int4 u = __ldg(a.units + ticket);
        const int64_t g0 = (int64_t)u.x * (NNZ * kBxPix);    // first map double of the block
        if constexpr (MODE == 1) {
            if (u.z <= u.y) return; // nothing to project from this block
            const double2 *src = reinterpret_cast<const double2 *>(a.zmap + g0);
#pragma unroll 4
            for (int k = lane; k < NNZ * kBxPix / 2; k += 32) {
                const int64_t g = g0 + 2 * k;
                double2 v = make_double2(0.0, 0.0);
                if (g + 1 < g_end) v = __ldcs(src + k);
                else if (g < g_end) v.x = __ldcs(a.zmap + g);
                tile2[k] = v;
            }
            __syncwarp();
            bx_project<UNIFORM, PAIRED, NNZ>(a, tile, u.y, u.z, lane);
        } else {
#pragma unroll 4
            for (int k = lane; k < NNZ * kBxPix / 2; k += 32) tile2[k] = make_double2(0.0, 0.0);
            __syncwarp();
            bx_accumulate<UNIFORM, PAIRED, MODE == 2, NNZ>(a, tile, u.y, u.z, lane);
            __syncwarp();
            if constexpr (MODE == 0) {
                if (u.w == 0 && !a.accumulate) {
                    // the only unit of its block: the tile IS the block of the map
                    double2 *dst = reinterpret_cast<double2 *>(a.zmap + g0);
#pragma unroll 4
                    for (int k = lane; k < NNZ * kBxPix / 2; k += 32) {
                        const int64_t gg = g0 + 2 * k;
                        if (gg + 1 < g_end) __stcs(dst + k, tile2[k]);
                        else if (gg < g_end) a.zmap[gg] = tile2[k].x;
                    }
                } else {
                    for (int k = lane; k < NNZ * kBxPix; k += 32) {
                        const double v = tile[k];
                        if (v != 0.0 && g0 + k < g_end) atomicAdd(a.zmap + g0 + k, v);
                    }
                }
            } else if (u.z > u.y) {
                if constexpr (NNZ == 1) {
                    // fused: m = C z in place (toast_map_cov.cpp:471-528, the nnz == 1 branch)
                    for (int p = lane; p < kBxPix; p += 32) {
                        const int64_t gp = (int64_t)u.x * kBxPix + p;
                        const double z0 = tile[p];
                        if (gp >= a.n_pix || z0 == 0.0) continue;
                        tile[p] = z0 * __ldcs(a.cov + gp);
                    }
                } else {
                    // fused: m = C z in place (toast_map_cov.cpp:509-517 operation order)
                    for (int p = lane; p < kBxPix; p += 32) {
                        const int64_t gp = (int64_t)u.x * kBxPix + p;
                        const double z0 = tile[3 * p], z1 = tile[3 * p + 1], z2 = tile[3 * p + 2];
                        if (gp >= a.n_pix || (z0 == 0.0 && z1 == 0.0 && z2 == 0.0)) continue;
                        const double2 *cm = reinterpret_cast<const double2 *>(a.cov + 6 * gp);
                        const double2 ca = __ldcs(cm), cb = __ldcs(cm + 1), cc = __ldcs(cm + 2);
                        double m0 = 0.0, m1 = 0.0, m2 = 0.0;
                        m0 += ca.x * z0;
                        m0 += ca.y * z1;
                        m1 += ca.y * z0;
                        m0 += cb.x * z2;
                        m2 += cb.x * z0;
                        m1 += cb.y * z1;
                        m1 += cc.x * z2;
                        m2 += cc.x * z1;
                        m2 += cc.y * z2;
                        tile[3 * p] = m0;
                        tile[3 * p + 1] = m1;
                        tile[3 * p + 2] = m2;
                    }
                }
                __syncwarp();
                bx_project<UNIFORM, PAIRED, NNZ>(a, tile, u.y, u.z, lane);
            }
        }
    }
}

// zero / covariance product on whole blocks of the global map (the multi-unit blocks of the fused
// path: their units meet in global memory)
template <int NNZ>
__global__ void __launch_bounds__(kThreads)
k_bx_zero_blocks(const int32_t *__restrict__ blocks, int64_t n_pix, double *__restrict__ zmap) {
    const int64_t g0 = (int64_t)__ldg(blocks + blockIdx.x) * (NNZ * kBxPix);
    for (int k = threadIdx.x; k < NNZ * kBxPix; k += kThreads)
        if (g0 + k < NNZ * n_pix) zmap[g0 + k] = 0.0;
}

template <int NNZ>
__global__ void __launch_bounds__(kThreads)
k_bx_cov_blocks(const int32_t *__restrict__ blocks, int64_t n_pix, const double *__restrict__ cov,
                double *__restrict__ zmap) {
    const int64_t p0 = (int64_t)__ldg(blocks + blockIdx.x) * kBxPix;
    for (int p = threadIdx.x; p < kBxPix; p += kThreads) {
        const int64_t gp = p0 + p;
        if (gp >= n_pix) continue;
        if constexpr (NNZ == 1) {
            zmap[gp] = zmap[gp] * cov[gp];
        } else {
            double *z = zmap + 3 * gp;
            const double z0 = z[0], z1 = z[1], z2 = z[2];
            const double *m = cov + 6 * gp;
            double t0 = 0.0, t1 = 0.0, t2 = 0.0;
            t0 += m[0] * z0;
            t0 += m[1] * z1;
            t1 += m[1] * z0;
            t0 += m[2] * z2;
            t2 += m[2] * z0;
            t1 += m[3] * z1;
            t1 += m[4] * z2;
            t2 += m[4] * z1;
            t2 += m[5] * z2;
            z[0] = t0;
            z[1] = t1;
            z[2] = t2;
        }
    }
}

BxArgs make_args(const tb_obs *obs, const int4 *units) {
    BxArgs a;
    a.units = units;
    a.brec = obs->brec;
    a.bqu = obs->bqu;
    a.ascaled = obs->ascaled;
    a.out = nullptr;
    a.amp_offsets = obs->amp_offsets;
    a.nad = (int32_t)obs->n_amp_det;
    a.n_det = (int)obs->d.n_det;
    a.cst = make_double4(obs->s_const[0], obs->s_const[1], obs->s_const[2], obs->s_const[3]);
    a.table = obs->stable;
    a.inv_nad = 1.0 / (double)obs->n_amp_det;
    a.n_pix = obs->n_local_pix;
    a.zmap = nullptr;
    a.cov = nullptr;
    a.accumulate = 0;
    return a;
}

void row_grid(const tb_obs *obs, dim3 &grid) {
    int64_t gy = (obs->n_amp_det + kThreads * 4 - 1) / (kThreads * 4);
    if (gy < 1) gy = 1;
    if (gy > 65535) gy = 65535;
    grid = dim3((unsigned)obs->n_xrows, (unsigned)gy);
}

void launch_bx_prescale(const tb_obs *obs, const double *amps, const uint8_t *aflags, void *stream) {
    dim3 grid;
    row_grid(obs, grid);
    k_bx_prescale<<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        obs->x_paired, (int)obs->d.n_det, obs->n_amp_det, obs->amp_offsets, obs->det_scale, amps,
        aflags, obs->ascaled);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
}

void launch_direction_prescale(const tb_obs *obs, const double *delta_new, double *delta_old,
                               double *d, const double *s, const uint8_t *aflags, double *q,
                               void *stream) {
    dim3 grid;
    row_grid(obs, grid);
    k_pcg_direction_prescale<<<grid, kThreads, 0, (cudaStream_t)stream>>>(
        obs->x_paired, (int)obs->d.n_det, obs->n_amp_det, obs->amp_offsets, obs->det_scale,
        delta_new, delta_old, d, s, aflags, q, obs->ascaled, obs->bx_counter);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
}

template <int MODE, int NNZ>
void launch_bx_nnz(const tb_obs *obs, const BxArgs &a, int64_t n_units, void *stream) {
    const int64_t nb = (n_units + kBxWarps - 1) / kBxWarps;
    TB_REQUIRE(nb < 2147483647LL, "grid too large");
    const unsigned g = (unsigned)nb;
    cudaStream_t st = (cudaStream_t)stream;
    static bool configured = false; // (per MODE / NNZ instantiation)
    if (!configured) {
        auto prep = [&](const void *f) {
            TB_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout,
                                         (int)cudaSharedmemCarveoutMaxShared));
        };
        prep((const void *)k_bx<MODE, true, true, NNZ>);
        prep((const void *)k_bx<MODE, true, false, NNZ>);
        prep((const void *)k_bx<MODE, false, true, NNZ>);
        prep((const void *)k_bx<MODE, false, false, NNZ>);
        configured = true;
    }
    if (obs->s_uniform) {
        if (obs->x_paired) k_bx<MODE, true, true, NNZ><<<g, kThreads, 0, st>>>(a, n_units);
        else k_bx<MODE, true, false, NNZ><<<g, kThreads, 0, st>>>(a, n_units);
    } else {
        if (obs->x_paired) k_bx<MODE, false, true, NNZ><<<g, kThreads, 0, st>>>(a, n_units);
        else k_bx<MODE, false, false, NNZ><<<g, kThreads, 0, st>>>(a, n_units);
    }
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
}

template <int MODE>
void launch_bx(const tb_obs *obs, const BxArgs &a, int64_t n_units, void *stream) {
    if (n_units <= 0) return;
    if (obs->nnz == 1) launch_bx_nnz<MODE, 1>(obs, a, n_units, stream);
    else launch_bx_nnz<MODE, 3>(obs, a, n_units, stream);
}

void launch_zero_blocks(const tb_obs *obs, double *zmap, cudaStream_t st) {
    if (obs->nnz == 1)
        k_bx_zero_blocks<1><<<(unsigned)obs->n_bmulti_blocks, kThreads, 0, st>>>(
            obs->bmulti_blocks, obs->n_local_pix, zmap);
    else
        k_bx_zero_blocks<3><<<(unsigned)obs->n_bmulti_blocks, kThreads, 0, st>>>(
            obs->bmulti_blocks, obs->n_local_pix, zmap);
    TB_CUDA(cudaGetLastError());
    tbr::count_launch();
}

inline bool bx_ok(const tb_obs *obs) { return g_use_bx && obs != nullptr && obs->brec != nullptr; }

// units [first, end) of chunk c (tb_obs_set_pixel_chunks), or all of them for c < 0
void chunk_units(const tb_obs *obs, int64_t chunk, int64_t &first, int64_t &end) {
    first = 0;
    end = obs->n_bunits;
    if (chunk < 0) return;
    TB_REQUIRE(chunk + 1 < (int64_t)obs->bchunk_unit.size(),
               "bad chunk index (or pixel chunk bounds not aligned to the block size)");
    first = obs->bchunk_unit[chunk];
    end = obs->bchunk_unit[chunk + 1];
}

} // namespace

void tb_free_blocked(tb_obs *obs) {
    if (obs->brec) cudaFree(obs->brec);
    if (obs->bqu) cudaFree(obs->bqu);
    if (obs->bunits) cudaFree(obs->bunits);
    if (obs->bunits_single) cudaFree(obs->bunits_single);
    if (obs->bunits_multi) cudaFree(obs->bunits_multi);
    if (obs->bmulti_blocks) cudaFree(obs->bmulti_blocks);
    if (obs->ascaled) cudaFree(obs->ascaled);
    if (obs->bx_counter) cudaFree(obs->bx_counter);
    obs->ascaled = nullptr;
    obs->bx_counter = nullptr;
    obs->brec = nullptr;
    obs->bqu = nullptr;
    obs->bunits = obs->bunits_single = obs->bunits_multi = nullptr;
    obs->bmulti_blocks = nullptr;
    obs->n_brec = obs->n_bunits = obs->n_bunits_single = obs->n_bunits_multi = 0;
    obs->n_bmulti_blocks = 0;
    obs->bunits_host.clear();
    obs->bchunk_unit.clear();
}

// Build the block-ordered list from the time-ordered one.  Not built (the other kernels then
// run) when a packed field would overflow or an unflagged sample lies off the local map (the
// reference itself indexes out of bounds there: ops_scan_map.cpp:44-52).
void tb_build_blocked(tb_obs *obs, cudaStream_t st) {
    tb_free_blocked(obs);
    const int64_t n_rec = obs->n_xrec, nad = obs->n_amp_det, n_det = obs->d.n_det;
    const int64_t n_pix = obs->n_local_pix;
    if (obs->xrec == nullptr || obs->stable == nullptr) return;
    if (n_rec <= 0 || n_rec >= (1LL << 29) || n_det * nad >= 2147483647LL || n_pix <= 0 ||
        n_pix >= (1LL << 31) - kBxPix || obs->n_xrows > (1LL << kBxRowBits))
        return; // (the records carry their row in kBxRowBits bits)
    const int32_t n_blocks = (int32_t)((n_pix + kBxPix - 1) >> kBxShift);
    const int grid = tbr::sm_count() * 8;
    unsigned int *counters = nullptr;
    TB_CUDA(cudaMalloc(&counters, 3 * sizeof(unsigned int)));
    int32_t *kin = nullptr, *vin = nullptr, *kout = nullptr, *vout = nullptr, *starts = nullptr;
    auto cleanup = [&]() {
        if (counters) cudaFree(counters);
        if (kin) cudaFree(kin);
        if (vin) cudaFree(vin);
        if (kout) cudaFree(kout);
        if (vout) cudaFree(vout);
        if (starts) cudaFree(starts);
    };
    try {
        unsigned int hc[3] = {0, 0, 0};
        int64_t n_entries = n_rec;
        TB_CUDA(cudaMalloc(&kin, sizeof(int32_t) * 2 * n_rec));
        TB_CUDA(cudaMalloc(&vin, sizeof(int32_t) * 2 * n_rec));
        for (int two_slot = 0; two_slot < 2; ++two_slot) {
            TB_CUDA(cudaMemsetAsync(counters, 0, 3 * sizeof(unsigned int), st));
            if (two_slot) k_bx_keys<true><<<grid, kThreads, 0, st>>>(obs->xrec, n_rec, n_blocks, kin, vin, counters);
            else k_bx_keys<false><<<grid, kThreads, 0, st>>>(obs->xrec, n_rec, n_blocks, kin, vin, counters);
            TB_CUDA(cudaGetLastError());
            tbr::count_launch();
            TB_CUDA(cudaMemcpyAsync(hc, counters, sizeof(hc), cudaMemcpyDeviceToHost, st));
            TB_CUDA(cudaStreamSynchronize(st));
            n_entries = two_slot ? 2 * n_rec : n_rec;
            if (hc[0] == 0 || two_slot) break; // no split crossings: one slot per record suffices
        }
        const int64_t n_sorted = n_entries - (int64_t)hc[1];
        if (hc[2] != 0 || n_sorted <= 0) { // off-map samples: keep the time-ordered pass 2
            cleanup();
            return;
        }
        TB_CUDA(cudaMalloc(&kout, sizeof(int32_t) * n_entries));
        TB_CUDA(cudaMalloc(&vout, sizeof(int32_t) * n_entries));
        int end_bit = 1;
        while ((1LL << end_bit) <= n_blocks) ++end_bit;
        tbr::sort_pairs_i32(kin, kout, vin, vout, n_entries, end_bit, st); // stable
        cudaFree(kin);
        cudaFree(vin);
        kin = vin = nullptr;
        // (two records of padding: the staged copies start / end on even record indices)
        TB_CUDA(cudaMalloc(&obs->brec, sizeof(int2) * (n_sorted + 2)));
        TB_CUDA(cudaMemsetAsync(obs->brec + n_sorted, 0, sizeof(int2) * 2, st));
        if (obs->nnz == 3) {
            TB_CUDA(cudaMalloc(&obs->bqu, sizeof(double2) * (n_sorted + 2)));
            TB_CUDA(cudaMemsetAsync(obs->bqu + n_sorted, 0, sizeof(double2) * 2, st));
        }
        {
            const size_t slots = (size_t)obs->n_xrows * (size_t)nad;
            const size_t per = obs->x_paired ? 2 : 1;
            TB_CUDA(cudaMalloc(&obs->ascaled, sizeof(double) * 2 * per * slots));
            TB_CUDA(cudaMalloc(&obs->bx_counter, sizeof(unsigned int)));
            TB_CUDA(cudaMemsetAsync(obs->bx_counter, 0, sizeof(unsigned int), st));
        }
        if (obs->nnz == 1)
            k_bx_gather<1><<<grid, kThreads, 0, st>>>(obs->xrec, nullptr, vout, n_sorted, nad, 1,
                                                      obs->brec, nullptr);
        else
            k_bx_gather<3><<<grid, kThreads, 0, st>>>(obs->xrec, obs->xqu, vout, n_sorted, nad,
                                                      1, obs->brec, obs->bqu);
        TB_CUDA(cudaGetLastError());
        tbr::count_launch();
        TB_CUDA(cudaMalloc(&starts, sizeof(int32_t) * (n_blocks + 1)));
        k_bx_block_starts<<<(n_blocks + 1 + 127) / 128, 128, 0, st>>>(kout, n_sorted, n_blocks, starts);
        TB_CUDA(cudaGetLastError());
        tbr::count_launch();
        std::vector<int32_t> hs(n_blocks + 1);
        TB_CUDA(cudaMemcpyAsync(hs.data(), starts, sizeof(int32_t) * (n_blocks + 1),
                                cudaMemcpyDeviceToHost, st));
        TB_CUDA(cudaStreamSynchronize(st));
        // work units: every block gets at least one (an empty block still has to be written)
        std::vector<int4> units, single, multi;
        std::vector<int32_t> mblocks;
        for (int32_t b = 0; b < n_blocks; ++b) {
            const int32_t f = hs[b], e = hs[b + 1];
            const int32_t nu = std::max(1, (e - f + kBxUnitMax - 1) / kBxUnitMax);
            if (nu > 1) mblocks.push_back(b);
            for (int32_t k = 0; k < nu; ++k) {
                // equal shares, so that no unit of a block is a sliver
                const int32_t uf = f + (int32_t)(((int64_t)(e - f) * k) / nu);
                const int32_t ue = f + (int32_t)(((int64_t)(e - f) * (k + 1)) / nu);
                const int4 u = make_int4(b, uf, ue, nu > 1 ? 1 : 0);
                units.push_back(u);
                if (nu > 1) multi.push_back(u);
                else if (ue > uf) single.push_back(u); // (the fused kernel skips empty blocks)
            }
        }
        auto upload = [&](const std::vector<int4> &v, int4 **dst) {
            if (v.empty()) return;
            TB_CUDA(cudaMalloc(dst, sizeof(int4) * v.size()));
            TB_CUDA(cudaMemcpy(*dst, v.data(), sizeof(int4) * v.size(), cudaMemcpyHostToDevice));
        };
        upload(units, &obs->bunits);
        upload(single, &obs->bunits_single);
        upload(multi, &obs->bunits_multi);
        if (!mblocks.empty()) {
            TB_CUDA(cudaMalloc(&obs->bmulti_blocks, sizeof(int32_t) * mblocks.size()));
            TB_CUDA(cudaMemcpy(obs->bmulti_blocks, mblocks.data(), sizeof(int32_t) * mblocks.size(),
                               cudaMemcpyHostToDevice));
        }
        obs->n_brec = n_sorted;
        obs->n_bunits = (int64_t)units.size();
        obs->n_bunits_single = (int64_t)single.size();
        obs->n_bunits_multi = (int64_t)multi.size();
        obs->n_bmulti_blocks = (int64_t)mblocks.size();
        obs->bunits_host = units;
        obs->bchunk_unit.assign({0, obs->n_bunits});
        cleanup();
    } catch (...) {
        cleanup();
        tb_free_blocked(obs);
        throw;
    }
}

// pixel chunks for the multi-GPU pipeline: bounds must fall on block boundaries (or the map end)
void tb_blocked_set_chunks(tb_obs *obs, int64_t n_chunks, const int64_t *pixel_bounds) {
    if (obs->brec == nullptr) return;
    std::vector<int64_t> cu(n_chunks + 1);
    for (int64_t c = 0; c <= n_chunks; ++c) {
        const int64_t b = pixel_bounds[c];
        if (!(b % kBxPix == 0 || b >= obs->n_local_pix)) {
            obs->bchunk_unit.clear(); // not block-aligned: chunked blocked calls are refused
            return;
        }
        const int64_t blk = (b + kBxPix - 1) >> kBxShift;
        // first unit whose block is >= blk
        auto it = std::lower_bound(obs->bunits_host.begin(), obs->bunits_host.end(), blk,
                                   [](const int4 &u, int64_t v) { return (int64_t)u.x < v; });
        cu[c] = (int64_t)(it - obs->bunits_host.begin());
    }
    cu[0] = 0;
    cu[n_chunks] = obs->n_bunits;
    obs->bchunk_unit = cu;
}

extern "C" {

int tb_bx_block_pixels(void) { return kBxPix; }

int tb_obs_blocked(const tb_obs *obs) { return bx_ok(obs) ? 1 : 0; }

int tb_obs_blocked_stats(const tb_obs *obs, int64_t *n_records, int64_t *n_units,
                         int64_t *n_multi_units, int64_t *n_blocks) {
    TB_API_BEGIN
    TB_REQUIRE(obs != nullptr, "NULL observation");
    if (n_records) *n_records = obs->n_brec;
    if (n_units) *n_units = obs->n_bunits;
    if (n_multi_units) *n_multi_units = obs->n_bunits_multi;
    if (n_blocks) *n_blocks = obs->brec ? (obs->n_local_pix + kBxPix - 1) >> kBxShift : 0;
    TB_API_END
}

int tb_bx_pass1(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                double *zmap, int accumulate, int64_t chunk, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && amplitudes && amp_flags && zmap, "NULL argument");
    TB_REQUIRE(bx_ok(obs), "the observation has no block-ordered crossing list");
    TB_REQUIRE((reinterpret_cast<uintptr_t>(zmap) & 15u) == 0, "zmap must be 16-byte aligned");
    int64_t first, end;
    chunk_units(obs, chunk, first, end);
    if (chunk <= 0) launch_bx_prescale(obs, amplitudes, amp_flags, stream);
    if (!accumulate && obs->n_bmulti_blocks > 0 && chunk <= 0) {
        // the units of a multi-unit block meet in global memory: it starts from zero
        launch_zero_blocks(obs, zmap, (cudaStream_t)stream);
    }
    BxArgs a = make_args(obs, obs->bunits + first);
    a.zmap = zmap;
    a.accumulate = accumulate;
    launch_bx<0>(obs, a, end - first, stream);
    TB_API_END
}

int tb_bx_pass2(const tb_obs *obs, const double *binned, double *amplitudes_out, int64_t chunk,
                void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && binned && amplitudes_out, "NULL argument");
    TB_REQUIRE(bx_ok(obs), "the observation has no block-ordered crossing list");
    TB_REQUIRE((reinterpret_cast<uintptr_t>(binned) & 15u) == 0, "map must be 16-byte aligned");
    int64_t first, end;
    chunk_units(obs, chunk, first, end);
    BxArgs a = make_args(obs, obs->bunits + first);
    a.zmap = const_cast<double *>(binned);
    a.out = amplitudes_out;
    launch_bx<1>(obs, a, end - first, stream);
    TB_API_END
}

int tb_bx_fused(const tb_obs *obs, const double *amplitudes, const uint8_t *amp_flags,
                const double *cov, double *zmap_scratch, double *amplitudes_out, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && cov && amplitudes_out, "NULL argument");
    TB_REQUIRE(bx_ok(obs), "the observation has no block-ordered crossing list");
    TB_REQUIRE((reinterpret_cast<uintptr_t>(cov) & 15u) == 0, "cov must be 16-byte aligned");
    // amplitudes == NULL: the amplitudes of the preceding call (their prescaled copy is reused)
    if (amplitudes != nullptr) {
        TB_REQUIRE(amp_flags != nullptr, "NULL argument");
        launch_bx_prescale(obs, amplitudes, amp_flags, stream);
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (obs->n_bunits_multi > 0) {
        // blocks cut into several units: their units meet in global memory (zmap_scratch)
        TB_REQUIRE(zmap_scratch != nullptr, "blocks with several units need the zmap scratch");
        TB_REQUIRE((reinterpret_cast<uintptr_t>(zmap_scratch) & 15u) == 0,
                   "zmap scratch must be 16-byte aligned");
        launch_zero_blocks(obs, zmap_scratch, st);
        BxArgs m = make_args(obs, obs->bunits_multi);
        m.zmap = zmap_scratch;
        launch_bx<0>(obs, m, obs->n_bunits_multi, stream);
        if (obs->nnz == 1)
            k_bx_cov_blocks<1><<<(unsigned)obs->n_bmulti_blocks, kThreads, 0, st>>>(
                obs->bmulti_blocks, obs->n_local_pix, cov, zmap_scratch);
        else
            k_bx_cov_blocks<3><<<(unsigned)obs->n_bmulti_blocks, kThreads, 0, st>>>(
                obs->bmulti_blocks, obs->n_local_pix, cov, zmap_scratch);
        TB_CUDA(cudaGetLastError());
        tbr::count_launch();
        m.out = amplitudes_out;
        launch_bx<1>(obs, m, obs->n_bunits_multi, stream);
    }
    BxArgs a = make_args(obs, obs->bunits_single);
    a.cov = cov;
    a.out = amplitudes_out;
    launch_bx<2>(obs, a, obs->n_bunits_single, stream);
    TB_API_END
}

int tb_bx_direction_prescale(const tb_obs *obs, const double *delta_new, double *delta_old,
                             double *d, const double *s, const uint8_t *amp_flags, double *q,
                             int64_t n, void *stream) {
    TB_API_BEGIN
    tbr::require_device();
    TB_REQUIRE(obs && delta_new && delta_old && d && s && amp_flags && q, "NULL argument");
    TB_REQUIRE(bx_ok(obs), "the observation has no block-ordered crossing list");
    // one pass over the rows must reach every amplitude exactly once
    const int64_t n_det = obs->d.n_det;
    TB_REQUIRE(obs->amp_dense && n == n_det * obs->n_amp_det &&
                   obs->n_xrows == (obs->x_paired ? (n_det + 1) / 2 : n_det),
               "the crossing-list rows do not cover the amplitude vector");
    launch_direction_prescale(obs, delta_new, delta_old, d, s, amp_flags, q, stream);
    TB_API_END
}

} // extern "C"
