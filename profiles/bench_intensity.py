"""Intensity-only (StokesWeights mode "I") against I/Q/U destriping of the same scan, on one GPU.

    python profiles/bench_intensity.py [--workloads c2,c3,c4] [--steps 10] [--warmup 3]
                                       [--rounds 3] [--out FILE]

For each workload (full size, bench.SHARDS: C2, C3 and the C4 shard), one process builds two
device problems from the same scan, flags and signal on the workload's HEALPix map: one with
I/Q/U weights (nnz = 3, what bench.py runs) and one with intensity weights (nnz = 1).  Reported,
on CUDA events after warm-up:

* the PCG iteration time and det-samples/s of each, the two timed alternately, ``--rounds`` times
  each (every round runs its own ``--warmup`` iterations, then ``--steps`` timed ones; the median
  round is reported);
* the records of the block-ordered list, the bytes each record streams per pass (brec 8 B, plus
  (sum Q, sum U) 16 B for I/Q/U) and whether its rows are detector pairs;
* the set-up times (pointing expansion, covariance, crossing lists).

The GPU name and power limit go into the same JSON.
"""

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import bench as B  # noqa: E402
from bench_wcs import gpu_identity, list_stats  # noqa: E402
from toast_b200 import synthetic as S  # noqa: E402

RECORD_BYTES = {3: 8 + 16, 1: 8}    # brec (+ bqu) per block-ordered record


def build_problem(obs, nnz, device, seed):
    """bench_wcs.build_problem on the workload's HEALPix map with ``nnz`` Stokes values: the same
    flags, pointing, covariance, rcond mask, Offset variance and signal for both nnz (the random
    streams are seeded alike)."""
    import torch

    from toast_b200 import kernels as K
    from toast_b200.solver import DeviceObservation, Destriper

    n_det, n_samp = obs["n_det"], obs["n_samp"]
    iv, step = obs["intervals"], obs["step_length"]
    n_submap, nps = S.n_submap_for(obs["nside"], 16)
    ncov = nnz * (nnz + 1) // 2
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
        solver_flags=solver_flags, solver_flag_mask=1, nside=obs["nside"], nest=obs["nest"],
        nnz=nnz, device=device)
    hits = np.zeros(n_submap, dtype=np.uint8)
    _, setup["pointing_expansion_ms"] = B._sync_ms(lambda: dobs.expand_pointing(hits))
    solver_flags |= (dobs.pixels < 0).to(torch.uint8)
    local = np.flatnonzero(hits).astype(np.int64)
    g2l = np.full(n_submap, -1, dtype=np.int64)
    g2l[local] = np.arange(len(local))
    dobs.set_global2local(g2l)
    n_loc = len(local)
    idx = np.arange(n_det, dtype=np.int32)
    invcov = torch.zeros((n_loc, nps, ncov), dtype=torch.float64, device=device)

    def cov():
        K.cov_accum(g2l, n_loc, nps, nnz, None, invcov, idx, dobs.pixels, idx, dobs.weights, idx,
                    solver_flags, obs["detweight"], 1, iv, None, 0)
        rc = torch.zeros(n_loc * nps, dtype=torch.float64, device=device)
        K.cov_invert(n_loc * nps, nnz, invcov, rc, 1.0e-8)
        return rc

    rcond, setup["covariance_ms"] = B._sync_ms(cov)
    bad = torch.zeros((n_loc, nps, nnz), dtype=torch.float64, device=device)
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
    info = dict(nnz=nnz, n_local_pix=n_loc * nps,
                det_samples=int(sum(int(v["last"] - v["first"]) for v in iv)) * n_det,
                setup_ms={k: round(v, 2) for k, v in setup.items()})
    info.update(list_stats(dobs))
    info["bytes_per_record"] = RECORD_BYTES[nnz]
    info["record_bytes_per_pass_gb"] = round(info["n_records"] * RECORD_BYTES[nnz] / 1e9, 4)
    return ds, dobs, tmp, info


def run_workload(name, args, device):
    import torch

    from toast_b200 import lib as L

    lib = L.load()
    sh = B.SHARDS[name]
    obs = S.make_observation(name, n_det=sh["n_det"], n_samp=sh["n_samp"], with_signal=False)
    out = dict(workload=name, n_det=obs["n_det"], n_samp=obs["n_samp"], nside=obs["nside"])
    problems = {}
    for key, nnz in (("iqu", 3), ("i", 1)):
        ds, dobs, signal, info = build_problem(obs, nnz, device, 20261020)
        st, sqsum_init = B.pcg_prologue(ds, signal, lib)
        del signal
        problems[key] = (ds, dobs, st, sqsum_init)
        out[key] = info
        out[key]["iteration_ms_rounds"] = []
    for _ in range(args.rounds):   # alternate the two
        for key, (ds, dobs, st, sqsum_init) in problems.items():
            ms, _, launches = B.time_iterations(ds, st, sqsum_init, args.steps, args.warmup, 1,
                                                lib)
            out[key]["iteration_ms_rounds"].append(round(ms, 4))
            out[key]["launches_per_iteration"] = round(launches / args.steps, 2)
    for key in problems:
        ms = float(np.median(out[key]["iteration_ms_rounds"]))
        out[key]["iteration_ms"] = round(ms, 4)
        out[key]["det_samples_per_s"] = out[key]["det_samples"] / (ms * 1e-3)
    out["i_over_iqu_iteration_time"] = round(out["i"]["iteration_ms"] /
                                             out["iqu"]["iteration_ms"], 4)
    del problems
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="c2,c3,c4")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()
    if args.steps < 10:
        raise SystemExit("--steps must be at least 10 PCG iterations")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_intensity.py measures on a GPU; none is visible")
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
