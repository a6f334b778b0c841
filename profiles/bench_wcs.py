"""Destriping on a flat-sky CAR map against the workload's HEALPix map, on one GPU.

    python profiles/bench_wcs.py [--workloads c2,c3] [--steps 10] [--warmup 3] [--rounds 3]
                                 [--out FILE]

For each ground workload (full size, bench.SHARDS), one process builds two device problems from
the same scan: the workload's HEALPix map and a CAR map of about the same pixel size (0.11 deg for
nside 512, 0.057 deg for nside 1024) with auto bounds (ops.PixelsWCS._geometry) and submaps of
about 3072 pixels.  Reported, on CUDA events after warm-up:

* the PCG iteration time and det-samples/s of each map, the two timed alternately, ``--rounds``
  times each (every round runs its own warm-up);
* n_records, samples per record, work units and local pixels of the block-ordered list;
* the set-up times (pointing expansion, covariance, crossing lists);
* tb_pointing_fused_wcs against the three-launch chain tb_pointing_detector -> tb_pixels_wcs ->
  tb_stokes_weights_IQU, on the first 500 detectors (outputs compared bit for bit first).

The GPU name and power limit go into the same JSON.
"""

import argparse
import ctypes as ct
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench as B  # noqa: E402
from toast_b200 import synthetic as S  # noqa: E402

CAR_RES = {512: 0.11, 1024: 0.057, 256: 0.23}
SUBMAP_PIX = 3072          # the HEALPix submap of nside_submap 16
FOV_DEG = 11.0             # the synthetic focal plane is 10 degrees wide


def gpu_identity():
    import torch

    out = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # the JSON says so instead
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def car_operator(obs, res):
    """ops.PixelsWCS on the scan of ``obs`` with auto bounds, and its submap count."""
    from toast_b200 import ops
    from toast_b200.data import Data, observation_from_synthetic

    data = Data()
    data.obs.append(observation_from_synthetic(obs))
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsWCS(detector_pointing=dp, projection="CAR", resolution=(res, res),
                        field_of_view=FOV_DEG, submaps=1)
    pix._geometry(data)
    pix.submaps = max(1, math.ceil(pix._n_pix / SUBMAP_PIX))
    pix.set_wcs()
    return pix


def build_problem(obs, pixelisation, n_submap, nps, device, seed):
    """The device problem of bench.build_gpu_problem for a given pixelisation (HEALPix
    nside / nest, or wcs): flags, pointing, covariance, rcond mask, Offset variance, signal."""
    import torch

    from toast_b200 import kernels as K
    from toast_b200.solver import DeviceObservation, Destriper

    n_det, n_samp = obs["n_det"], obs["n_samp"]
    iv, step = obs["intervals"], obs["step_length"]
    setup = {}
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def bursts(shape, frac, burst):
        n = int(np.prod(shape))
        f = torch.zeros(n + burst, dtype=torch.uint8, device=device)
        starts = torch.randint(0, n, (int(frac * n / burst),), generator=g, device=device)
        for k in range(burst):
            f[starts + k] = 1
        return f[:n].reshape(shape).contiguous()

    shared_flags = bursts((n_samp,), 0.005, 20)
    solver_flags = bursts((n_det, n_samp), 0.01, 50)
    in_view = torch.zeros(n_samp, dtype=torch.bool, device=device)
    for v in iv:
        in_view[int(v["first"]):int(v["last"])] = True
    solver_flags |= (~in_view).to(torch.uint8)[None, :]
    solver_flags |= shared_flags[None, :]
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=iv,
        det_scale=obs["detweight"], step_length=step, n_pix_submap=nps, n_submap=n_submap,
        global2local=np.zeros(n_submap, dtype=np.int64), epsilon=obs["epsilon"],
        gamma=obs["gamma"], cal=obs["cal"], shared_flags=shared_flags, shared_flag_mask=1,
        solver_flags=solver_flags, solver_flag_mask=1, device=device, **pixelisation)
    hits = np.zeros(n_submap, dtype=np.uint8)
    _, setup["pointing_expansion_ms"] = B._sync_ms(lambda: dobs.expand_pointing(hits))
    solver_flags |= (dobs.pixels < 0).to(torch.uint8)
    local = np.flatnonzero(hits).astype(np.int64)
    g2l = np.full(n_submap, -1, dtype=np.int64)
    g2l[local] = np.arange(len(local))
    dobs.set_global2local(g2l)
    n_loc = len(local)
    idx = np.arange(n_det, dtype=np.int32)
    invcov = torch.zeros((n_loc, nps, 6), dtype=torch.float64, device=device)

    def cov():
        K.cov_accum(g2l, n_loc, nps, 3, None, invcov, idx, dobs.pixels, idx, dobs.weights, idx,
                    solver_flags, obs["detweight"], 1, iv, None, 0)
        rc = torch.zeros(n_loc * nps, dtype=torch.float64, device=device)
        K.cov_invert(n_loc * nps, 3, invcov, rc, 1.0e-8)
        return rc

    rcond, setup["covariance_ms"] = B._sync_ms(cov)
    bad = torch.zeros((n_loc, nps, 3), dtype=torch.float64, device=device)
    bad[:, :, 0] = (rcond.reshape(n_loc, nps) == 0).to(torch.float64)
    tmp = torch.zeros((n_det, n_samp), dtype=torch.float64, device=device)
    K.ops_scan_map_float64(g2l, nps, bad, tmp, idx, dobs.pixels, idx, dobs.weights, idx, iv, 1.0,
                           True, False, False)
    solver_flags |= (tmp != 0).to(torch.uint8)
    del bad
    tmp.fill_(1.0)
    n_good = torch.zeros(dobs.n_amp, dtype=torch.float64, device=device)
    zero_flags = torch.zeros(dobs.n_amp, dtype=torch.uint8, device=device)
    K.template_offset_project_signal_batch(idx, tmp, idx, solver_flags, 1, step,
                                           dobs.amp_offsets, dobs.n_amp_views, n_good, zero_flags,
                                           iv)
    amplen = np.concatenate([
        np.minimum(step, int(v["last"] - v["first"]) - step * np.arange(na))
        for v, na in zip(iv, dobs.n_amp_views)])
    amplen = torch.from_numpy(np.tile(amplen.astype(np.float64), n_det)).to(device)
    keep = (n_good / amplen) > 0.5
    detw = torch.from_numpy(np.repeat(obs["detweight"], dobs.n_amp_det)).to(device)
    offset_var = torch.where(keep, 1.0 / (detw * torch.clamp(n_good, min=1.0)),
                             torch.zeros_like(n_good))
    amp_flags = (~keep).to(torch.uint8)
    tmp.normal_(generator=g)
    tmp *= torch.from_numpy(obs["sigma"]).to(device)[:, None]
    base = torch.cumsum(torch.randn((n_det, dobs.n_amp_det), generator=g, device=device,
                                    dtype=torch.float64), dim=1).reshape(-1).contiguous()
    K.template_offset_add_to_signal_batch(step, dobs.amp_offsets, dobs.n_amp_views, base,
                                          zero_flags, idx, tmp, iv)
    _, setup["crossing_lists_ms"] = B._sync_ms(lambda: dobs.handle())
    ds = Destriper([dobs], n_loc, nps, invcov, offset_var, amp_flags, device=device)
    info = dict(n_submap=n_submap, n_pix_submap=nps, n_local_submap=n_loc,
                n_local_pix=n_loc * nps, det_samples=int(sum(int(v["last"] - v["first"])
                                                             for v in iv)) * n_det,
                setup_ms={k: round(v, 2) for k, v in setup.items()})
    info.update(list_stats(dobs))
    info["samples_per_record"] = round(info["det_samples"] / max(info["n_records"], 1), 3)
    return ds, dobs, tmp, info


def list_stats(dobs):
    from toast_b200 import lib as L

    lib = L.load()
    h = dobs.handle().h
    out = dict(blocked=int(lib.tb_obs_blocked(h)))
    n_rec, n_rows, paired = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
    L.check(lib.tb_obs_crossing_stats(h, ct.byref(n_rec), ct.byref(n_rows), ct.byref(paired)))
    out.update(n_crossing_records=n_rec.value, crossing_rows=n_rows.value, paired=paired.value)
    if out["blocked"]:
        n_rec, n_units, n_multi, n_blocks = (ct.c_int64(0) for _ in range(4))
        L.check(lib.tb_obs_blocked_stats(h, ct.byref(n_rec), ct.byref(n_units),
                                         ct.byref(n_multi), ct.byref(n_blocks)))
        out.update(n_records=n_rec.value, n_units=n_units.value, n_multi_units=n_multi.value,
                   n_blocks=n_blocks.value)
    else:
        out["n_records"] = out["n_crossing_records"]
    return out


def pointing_comparison(obs, wcs, nps, n_submap, device, n_det_max=500, reps=5):
    """tb_pointing_fused_wcs against the three-launch chain on the first detectors: outputs bit
    for bit, then the time of each on CUDA events (one warm-up call each, then ``reps``)."""
    import torch

    from toast_b200 import kernels as K

    n_det = min(obs["n_det"], n_det_max)
    n_samp = obs["n_samp"]
    fp = np.ascontiguousarray(obs["focalplane"][:n_det])
    eps, gam, cal = (np.ascontiguousarray(obs[k][:n_det]) for k in ("epsilon", "gamma", "cal"))
    idx = np.arange(n_det, dtype=np.int32)
    iv = obs["intervals"]
    bore = torch.from_numpy(obs["boresight"]).to(device)
    flags = torch.from_numpy(obs["shared_flags"]).to(device)
    quats = torch.zeros((n_det, n_samp, 4), dtype=torch.float64, device=device)
    pix_c = torch.zeros((n_det, n_samp), dtype=torch.int64, device=device)
    w_c = torch.zeros((n_det, n_samp, 3), dtype=torch.float64, device=device)
    pix_f, w_f = torch.zeros_like(pix_c), torch.zeros_like(w_c)
    hits_c = np.zeros(n_submap, dtype=np.uint8)
    hits_f = np.zeros(n_submap, dtype=np.uint8)

    def chain():
        K.pointing_detector(fp, bore, idx, quats, iv, flags, 1)
        K.pixels_wcs(wcs, idx, quats, flags, 1, idx, pix_c, iv, hits_c, nps)
        K.stokes_weights_IQU(idx, quats, idx, w_c, np.zeros(1), iv, eps, gam, cal, False)

    def fused():
        K.pointing_fused_wcs(wcs, fp, bore, flags, 1, None, None, idx, pix_f, idx, w_f, None, iv,
                             hits_f, nps, eps, gam, cal, False)

    chain()
    fused()
    torch.cuda.synchronize()
    same = bool(torch.equal(pix_c, pix_f) and torch.equal(w_c, w_f)
                and np.array_equal(hits_c, hits_f))
    out = dict(n_det=n_det, n_samp=n_samp, outputs_bit_identical=same)
    for name, fn in (("chain_ms", chain), ("fused_ms", fused)):
        ts = []
        for _ in range(reps):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            fn()
            t1.record()
            torch.cuda.synchronize()
            ts.append(t0.elapsed_time(t1))
        out[name] = round(float(np.median(ts)), 3)
        out[name.replace("_ms", "_ms_all")] = [round(t, 3) for t in ts]
    out["fused_speedup"] = round(out["chain_ms"] / out["fused_ms"], 3)
    del quats, pix_c, w_c, pix_f, w_f
    return out


def run_workload(name, args, device):
    import torch

    from toast_b200 import lib as L

    lib = L.load()
    sh = B.SHARDS[name]
    obs = S.make_observation(name, n_det=sh["n_det"], n_samp=sh["n_samp"], with_signal=False)
    nside = obs["nside"]
    res = CAR_RES[nside]
    t0 = time.perf_counter()
    pix = car_operator(obs, res)
    geometry_s = time.perf_counter() - t0
    n_submap_h, nps_h = S.n_submap_for(nside, 16)
    out = dict(workload=name, n_det=obs["n_det"], n_samp=obs["n_samp"], nside=nside,
               car=dict(resolution_deg=res, shape=list(pix.wcs_shape), n_pix=pix._n_pix,
                        bounds_deg=[round(b, 6) for b in pix.bounds],
                        geometry_s=round(geometry_s, 3)))
    out["pointing"] = pointing_comparison(obs, pix.wcs, pix._n_pix_submap, pix._n_submap, device)
    torch.cuda.empty_cache()
    problems = {}
    for key, pixelisation, ns, nps in (
            ("healpix", dict(nside=nside, nest=obs["nest"]), n_submap_h, nps_h),
            ("car", dict(wcs=pix.wcs), pix._n_submap, pix._n_pix_submap)):
        ds, dobs, signal, info = build_problem(obs, pixelisation, ns, nps, device, 20261020)
        st, sqsum_init = B.pcg_prologue(ds, signal, lib)
        del signal
        problems[key] = (ds, dobs, st, sqsum_init, info)
        out.setdefault(key, {}).update(info)
    for key in problems:
        out[key]["iteration_ms_rounds"] = []
    for _ in range(args.rounds):   # alternate the two maps
        for key, (ds, dobs, st, sqsum_init, info) in problems.items():
            ms, _, launches = B.time_iterations(ds, st, sqsum_init, args.steps, args.warmup, 1,
                                                lib)
            out[key]["iteration_ms_rounds"].append(round(ms, 4))
            out[key]["launches_per_iteration"] = round(launches / args.steps, 2)
    for key in problems:
        ms = float(np.median(out[key]["iteration_ms_rounds"]))
        out[key]["iteration_ms"] = round(ms, 4)
        out[key]["det_samples_per_s"] = out[key]["det_samples"] / (ms * 1e-3)
    out["car_over_healpix_iteration_time"] = round(
        out["car"]["iteration_ms"] / out["healpix"]["iteration_ms"], 4)
    del problems
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_wcs.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    result = dict(gpu_identity(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
                  source_hash=B.source_hash(), workloads=[])
    for name in args.workloads.split(","):
        result["workloads"].append(run_workload(name.strip(), args, "cuda:0"))
        print(json.dumps(result["workloads"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
