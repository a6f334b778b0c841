"""Monte Carlo realisations with MapMaker(mc_mode=True) against the first call, on one GPU.

    python profiles/bench_mc.py [--workloads c4,c2,c3] [--iters 50] [--realisations 5]
                                [--out FILE]

For each workload (full size, bench.SHARDS: the C4 shard, C2 and C3) the problem is built as
bench.py's end-to-end leg builds it (page-locked detdata buffers, the same operators and traits,
``--iters`` PCG iterations every call).  Reported, wall clock bracketed by device synchronisation:

* the first ``mc_mode=True`` call (the whole pipeline: set-up and one realisation);
* ``--realisations`` further calls, each with a new seeded timestream written into the same
  page-locked ``det_data`` buffer beforehand (outside the timed window);
* one more realisation with ``profile_stages=True`` (the per-stage split of a reused call), a
  fresh ``mc_mode=False`` call on the same timestream with ``profile_stages=True`` (the split of
  a full call) and one without (the time of a full call in a warm process); the destriped and
  binned maps of the last realisation against the second fresh call's, and the two fresh calls'
  against each other (relative norm of the difference);
* the device memory allocated after every realisation.

The GPU name and power limit go into the same JSON.
"""

import argparse
import gc
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import bench as B  # noqa: E402
from bench_wcs import gpu_identity  # noqa: E402
from toast_b200 import synthetic as S  # noqa: E402


def make_mapper(obs, n_iter, mc_mode, profile=False):
    """The MapMaker of bench.py's end-to-end leg, with ``mc_mode``."""
    from toast_b200 import ops
    from toast_b200.templates.offset import Offset

    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    return ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                        iter_max=n_iter, iter_min=n_iter, convergence=1.0e-300,
                        device="cuda:0", mc_mode=mc_mode, profile_stages=profile)


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def run_workload(name, args):
    import torch

    from toast_b200.data import Data, observation_from_synthetic

    dev = torch.device("cuda:0")
    sh = B.SHARDS[name]
    obs = S.make_observation(name, n_det=sh["n_det"], n_samp=sh["n_samp"])
    data = Data()
    data.obs.append(observation_from_synthetic(obs, pinned=True))
    pinned = data.obs[0].detdata["signal"]._pinned
    base = torch.from_numpy(obs["signal"]).to(dev)
    sigma = torch.from_numpy(obs["sigma"]).to(dev)[:, None]
    del obs["signal"]

    def write(k):
        """Realisation k: the workload's signal plus seeded white noise, into det_data."""
        g = torch.Generator(device=dev)
        g.manual_seed(20261022 + k)
        sig = base + sigma * torch.randn(base.shape, generator=g, device=dev,
                                         dtype=torch.float64)
        pinned.copy_(sig)
        del sig
        torch.cuda.synchronize()

    def timed(mapper):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mapper.apply(data)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    out = dict(workload=name, n_det=obs["n_det"], n_samp=obs["n_samp"], nside=obs["nside"],
               pcg_iterations=args.iters)
    mapper = make_mapper(obs, args.iters, True)
    write(0)
    out["first_call_s"] = round(timed(mapper), 4)
    out["memory_allocated_gb"] = [round(torch.cuda.memory_allocated() / 1e9, 4)]
    times = []
    for k in range(1, args.realisations + 1):
        write(k)
        times.append(timed(mapper))
        gc.collect()
        out["memory_allocated_gb"].append(round(torch.cuda.memory_allocated() / 1e9, 4))
    out["realisation_s"] = [round(t, 4) for t in times]
    out["realisation_median_s"] = round(float(np.median(times)), 4)
    out["iterations_run"] = len(mapper.history)

    k_last = args.realisations + 1
    write(k_last)
    mapper.profile_stages = True
    out["profiled_realisation_s"] = round(timed(mapper), 4)
    out["realisation_stages_s"] = {k: round(v, 4) for k, v in mapper.stage_seconds.items()}
    last = {key: data[f"mm_{key}"].data.copy() for key in ("map", "binmap")}
    del mapper
    gc.collect()
    torch.cuda.empty_cache()

    write(k_last)
    fresh = make_mapper(obs, args.iters, False, profile=True)
    out["fresh_profiled_call_s"] = round(timed(fresh), 4)
    out["fresh_call_stages_s"] = {k: round(v, 4) for k, v in fresh.stage_seconds.items()}
    first_fresh = {key: data[f"mm_{key}"].data.copy() for key in ("map", "binmap")}
    del fresh
    gc.collect()
    # a second fresh call on the same timestream, unprofiled: the time of a call without
    # mc_mode once the process is warm, and how far two fresh calls agree (the binning kernels
    # accumulate with atomics, and the PCG amplifies the rounding differences)
    write(k_last)
    fresh = make_mapper(obs, args.iters, False)
    out["fresh_call_s"] = round(timed(fresh), 4)
    out["last_vs_fresh_rel_norm"] = {key: rel(last[key], data[f"mm_{key}"].data)
                                     for key in ("map", "binmap")}
    out["fresh_vs_fresh_rel_norm"] = {key: rel(first_fresh[key], data[f"mm_{key}"].data)
                                      for key in ("map", "binmap")}
    out["last_vs_fresh_within_1e-10"] = all(v <= 1e-10
                                             for v in out["last_vs_fresh_rel_norm"].values())
    del fresh, data, base, pinned
    gc.collect()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", default="c4,c2,c3")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--realisations", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_mc.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    result = dict(gpu_identity(), source_hash=B.source_hash(), workloads=[])
    for name in args.workloads.split(","):
        result["workloads"].append(run_workload(name.strip(), args))
        print(json.dumps(result["workloads"][-1]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
