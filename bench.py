#!/usr/bin/env python
"""bench.py -- detector-samples/s per destriper PCG iteration (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c2|c5] [--regen]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's compiled CPU path, bounded sample

A *step* is one PCG iteration of the Offset-template destriper (SolverLHS.apply + the vector
updates of solve(), ops/mapmaker_solve.py:665-746) over the rank's shard of synthetic data:

    N = 1    ONE kernel per observation (k_bx<2>): template -> noise-weighted map tile in shared
             memory -> 3x3 pixel covariance -> scan - weight - project, on the block-ordered
             crossing list (tb_blocked.cu); the map never touches HBM
    N > 1    pass 1 (k_bx<0>) -> NVLink map reduction fused with the pixel covariance
             (tb_peer.cu), pipelined over pixel chunks -> pass 2 (k_bx<1>)
    PCG      d.q, x/r/s update, r.r, s.r, new d     (+ one scalar read-back for convergence)

What the JSON line reports (see DESIGN.md section 5 for every definition):
  value / ms_per_step   device-timed (CUDA events, max over ranks), inputs resident in HBM
  roofline              dominant kernel timed alone with CUDA events on its stream; `achieved` =
                        COMPULSORY bytes of the shipped formulation (records + covariance of the
                        hit pixels + amplitude scratch + output vector) / that time; `traffic` =
                        ncu dram bytes of the committed capture of the same kernel (null when the
                        kernel sources changed since the capture); the reference layout's
                        66 B/sample figure is reported separately as `effective_*`
  e2e                   the same metric through ops.MapMaker.apply: host numpy buffers in pinned
                        memory in, maps + cleaned timestreams out, every copy inside the timed
                        region, divided by the PCG iterations it ran
  parity                start-up self checks that travel with the number: at N > 1 the fused
                        NVLink reduction against NCCL all-reduce + cov_apply on the real map; at
                        N = 1 the GPU LHS against the reference's compiled kernels on the CPU
                        sample of the cpu_baseline leg
  other_workloads       short sub-runs of BASELINE configs C2, C3 (stored / regenerated pointing)
                        and C5 (N = 1 only)

Default workload ("c4"): BASELINE.json configs[3] detector-sharded -- 128 detectors x 12 h @
50 Hz (2.76e8 det-samples) per GPU, nside 2048 NEST IQU, 1 s baselines; at N GPUs the job is
N x 128 detectors with the map all-reduced (weak scaling; N = 8 is the full 1024-detector
2.2e9-sample configuration).  Every iteration streams > 1.5 GB per GPU, far more than the 126 MB
L2, so no explicit L2 flush is needed between steps.
"""

import argparse
import ctypes as ct
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from toast_b200 import synthetic as S  # noqa: E402

METRIC = "detector-samples/s per destriper PCG iteration"
UNIT = "det-samples/s"

# per-GPU shard of each workload: (n_det per GPU, n_samp)
SHARDS = {
    "c4": dict(n_det=128, n_samp=2160000),   # 1024 det / 8 GPUs
    "c3": dict(n_det=2000, n_samp=360000),   # single-GPU destriper config
    "c2": dict(n_det=1000, n_samp=360000),
    "c5": dict(n_det=1000, n_samp=500000),   # 8000 det / 8 GPUs, high-contention patch
}
BYTES_PER_SAMPLE_PASS = 33      # reference layout: pixel 8 + weights 24 + solver flag 1 (SURVEY 8d)
BYTES_PER_SAMPLE_ITER = 66
NVLINK_GBS_PER_DIRECTION = 900.0  # NVLink 5, per GPU and direction


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(SHARDS))
    ap.add_argument("--regen", action="store_true",
                    help="regenerate pointing inside every pass instead of streaming it")
    ap.add_argument("--scale", type=float, default=1.0,
                    help="shrink the per-GPU shard (debugging only; the JSON line says so)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the e2e MapMaker run and the other-workload sub-runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed PCG iterations computed, after the last timed "
                         "step, to DIR/<name>.npy (same arguments -> same inputs, so two builds "
                         "can be compared output for output)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    return args


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": float(np.max(smax)) if smax else None,
            "power_w_max": float(np.max(power)) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's compiled kernels (oracle/_ref) or the C restatement, bounded sample
# ------------------------------------------------------------------------------------------------
def host_cores():
    return len(os.sched_getaffinity(0))


def cpu_problem(workload, n_det, n_samp):
    # torchrun exports OMP_NUM_THREADS=1: the reference arm uses every host core it is given
    os.environ["OMP_NUM_THREADS"] = str(host_cores())
    from oracle import toast_oracle as O

    ref = O.load_ref()
    kern = ref if ref is not None else O
    kind = "reference" if ref is not None else "port"
    obs = S.make_observation(workload, n_det=n_det, n_samp=n_samp)
    # production threshold (ops/mapmaker.py solve_rcond_threshold); the 64-detector sample
    # cross-links its pixels well enough for it
    pb = O.build_problem(obs, kern, rcond_threshold=1.0e-8)
    covapply = kern.cov_apply_diag
    return O, kern, kind, obs, pb, covapply


def cpu_iteration(O, kern, pb, covapply, st):
    """One PCG iteration with the reference kernels (ops/mapmaker_solve.py:665-746)."""
    fl = pb.amp_flags
    q = O.solver_lhs(pb, kern, st["d"], covapply)
    alpha = st["delta"] / O.amp_dot(st["d"], q, fl)
    st["x"] += st["d"] * alpha
    st["r"] -= q * alpha
    sqsum = O.amp_dot(st["r"], st["r"], fl)
    kern.template_offset_apply_diag_precond(pb.offset_var, st["r"], fl, st["s"], False)
    delta_new = O.amp_dot(st["s"], st["r"], fl)
    beta = delta_new / st["delta"]
    st["delta"] = delta_new
    st["d"] *= beta
    st["d"] += st["s"]
    return sqsum


def cpu_state(O, kern, pb, covapply, signal):
    rhs = O.solver_rhs(pb, kern, signal, covapply)
    s = np.zeros_like(rhs)
    kern.template_offset_apply_diag_precond(pb.offset_var, rhs, pb.amp_flags, s, False)
    return dict(x=np.zeros_like(rhs), r=rhs.copy(), d=s.copy(), s=s,
                delta=O.amp_dot(s, rhs, pb.amp_flags))


def cpu_sample_shape(workload):
    # 64 detectors (32 polarisation pairs: the OpenMP loops over detectors have work for every
    # thread) x 1/16 of the samples: ~1e7 det-samples, a second or two per iteration
    sh = SHARDS[workload]
    return 64, max(20000, sh["n_samp"] // 16)


def run_cpu(workload, steps, warmup, want_problem=False):
    n_det, n_samp = cpu_sample_shape(workload)
    cores = host_cores()
    O, kern, kind, obs, pb, covapply = cpu_problem(workload, n_det, n_samp)
    try:
        threads = int(kern.num_threads()) if hasattr(kern, "num_threads") else cores
    except Exception:
        threads = cores
    st = cpu_state(O, kern, pb, covapply, obs["signal"])
    for _ in range(warmup):
        cpu_iteration(O, kern, pb, covapply, st)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_iteration(O, kern, pb, covapply, st)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    n_good = int(sum(int(iv["last"] - iv["first"]) for iv in pb.intervals)) * n_det
    res = dict(value=n_good / dt, unit=UNIT, cores=threads, kind=kind,
               sample=f"{n_det} detectors x {n_samp} samples of workload {workload} "
                      f"({n_good} det-samples per iteration, stored pointing, rcond 1e-8, "
                      f"OMP_NUM_THREADS={os.environ['OMP_NUM_THREADS']} on {cores} host cores)",
               ms_per_step=dt * 1e3)
    if want_problem:
        res["_problem"] = (O, kern, obs, pb, covapply)
    return res


def config_dict(args, world, n_det, n_samp, nside, extra=None):
    cfg = {
        "workload": f"{args.workload}: BASELINE.json destriper config, per-GPU shard "
                    f"{n_det} det x {n_samp} samples, nside {nside}, Offset step "
                    f"{S.CONFIGS[args.workload]['step_time']} s, IQU, "
                    + ("pointing regenerated per pass" if args.regen else "stored pointing"),
        "detectors_total": n_det * world,
        "det_samples_total": n_det * n_samp * world,
        "parallelism": f"detector-sharded x{world}, NVLink map all-reduce" if world > 1
                       else "single GPU",
        "l2_policy": "no flush: every iteration streams far more than the 126 MB L2 (C4 shard: "
                     "0.95 GB of crossing records, 0.3-0.7 GB of pixel covariance, 0.13 GB of "
                     "amplitude scratch and 0.22 GB of PCG vectors per iteration)",
    }
    if args.scale != 1.0:
        cfg["scaled_down"] = args.scale
    if extra:
        cfg.update(extra)
    return cfg


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    res = run_cpu(args.workload, args.steps, args.warmup)
    sh = SHARDS[args.workload]
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args, args.gpus, sh["n_det"], sh["n_samp"],
                              S.CONFIGS[args.workload]["nside"], {"rcond_threshold": 1.0e-8}),
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _sync_ms(fn):
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3


def build_gpu_problem(workload, regen, scale, rank, world, device):
    """Untimed setup, all on the device except the (small) boresight / focalplane generation.
    Returns (destriper, observation, signal, info); info["setup_ms"] itemises what a solve pays
    once (pointing expansion, covariance, crossing-list construction)."""
    import torch

    from toast_b200 import kernels as K
    from toast_b200.solver import DeviceObservation, Destriper

    sh = SHARDS[workload]
    n_det = max(2, int(sh["n_det"] * scale))
    n_samp = max(1000, int(sh["n_samp"] * scale))
    obs = S.make_observation(workload, n_det=n_det, n_samp=n_samp, det_first=rank * n_det,
                             with_signal=False, flags=False)
    nside, nest = obs["nside"], obs["nest"]
    n_submap, nps = S.n_submap_for(nside, 16)
    iv = obs["intervals"]
    step = obs["step_length"]
    setup = {}

    g = torch.Generator(device=device)
    g.manual_seed(20261017 + 97 * rank)
    # shared flags: 0.5 % in bursts of 20; detector flags: 1 % in bursts of 50 (SURVEY 8d)
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
        det_scale=obs["detweight"], step_length=step, nside=nside, nest=nest,
        n_pix_submap=nps, n_submap=n_submap, global2local=np.zeros(n_submap, dtype=np.int64),
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"], shared_flags=shared_flags,
        shared_flag_mask=1, solver_flags=solver_flags, solver_flag_mask=1, device=device)
    hits = np.zeros(n_submap, dtype=np.uint8)
    _, setup["pointing_expansion_ms"] = _sync_ms(lambda: dobs.expand_pointing(hits))
    solver_flags |= (dobs.pixels < 0).to(torch.uint8)
    if world > 1:
        ht = torch.from_numpy(hits).to(device)
        torch.distributed.all_reduce(ht, op=torch.distributed.ReduceOp.MAX)
        hits = ht.cpu().numpy()
    local = np.flatnonzero(hits).astype(np.int64)
    g2l = np.full(n_submap, -1, dtype=np.int64)
    g2l[local] = np.arange(len(local))
    dobs.set_global2local(g2l)
    n_loc = len(local)

    # pixel covariance on the device: accumulate, all-reduce, invert
    idx = np.arange(n_det, dtype=np.int32)
    invcov = torch.zeros((n_loc, nps, 6), dtype=torch.float64, device=device)
    hitmap = torch.zeros(n_loc * nps, dtype=torch.int64, device=device)

    def cov():
        K.cov_accum(g2l, n_loc, nps, 3, hitmap, invcov, idx, dobs.pixels, idx, dobs.weights, idx,
                    solver_flags, obs["detweight"], 1, iv, None, 0)
        if world > 1:
            torch.distributed.all_reduce(invcov)
        rc = torch.zeros(n_loc * nps, dtype=torch.float64, device=device)
        # reference default: MapMaker.solve_rcond_threshold = 1e-8 (ops/mapmaker.py)
        K.cov_invert(n_loc * nps, 3, invcov, rc, 1.0e-8)
        return rc

    rcond, setup["covariance_ms"] = _sync_ms(cov)
    n_hit_pix = int((hitmap > 0).sum().item())  # pixels THIS rank's samples touch
    del hitmap
    # rcond mask -> solver flags (scan the bad-pixel map with the I weight = cal = 1)
    bad = torch.zeros((n_loc, nps, 3), dtype=torch.float64, device=device)
    bad[:, :, 0] = (rcond.reshape(n_loc, nps) == 0).to(torch.float64)
    tmp = torch.zeros((n_det, n_samp), dtype=torch.float64, device=device)
    K.ops_scan_map_float64(g2l, nps, bad, tmp, idx, dobs.pixels, idx, dobs.weights, idx, iv, 1.0,
                           True, False, False)
    solver_flags |= (tmp != 0).to(torch.uint8)
    del bad

    # Offset layout + amplitude variance: n_good per step = F^T (good-sample indicator)
    tmp.fill_(1.0)
    n_good = torch.zeros(dobs.n_amp, dtype=torch.float64, device=device)
    zero_flags = torch.zeros(dobs.n_amp, dtype=torch.uint8, device=device)
    K.template_offset_project_signal_batch(idx, tmp, idx, solver_flags, 1, step,
                                           dobs.amp_offsets, dobs.n_amp_views, n_good, zero_flags,
                                           iv)
    amplen = np.concatenate([
        np.minimum(step, int(v["last"] - v["first"]) - step * np.arange(na))
        for v, na in zip(iv, dobs.n_amp_views)]) if len(iv) else np.zeros(0)
    amplen = torch.from_numpy(np.tile(amplen.astype(np.float64), n_det)).to(device)
    keep = (n_good / amplen) > 0.5
    detw = torch.from_numpy(np.repeat(obs["detweight"], dobs.n_amp_det)).to(device)
    offset_var = torch.where(keep, 1.0 / (detw * torch.clamp(n_good, min=1.0)),
                             torch.zeros_like(n_good))
    amp_flags = (~keep).to(torch.uint8)

    # signal: white noise + per-step random-walk baselines (destriping has work to do)
    tmp.normal_(generator=g)
    tmp *= torch.from_numpy(obs["sigma"]).to(device)[:, None]
    base = torch.cumsum(torch.randn((n_det, dobs.n_amp_det), generator=g, device=device,
                                    dtype=torch.float64), dim=1).reshape(-1).contiguous()
    K.template_offset_add_to_signal_batch(step, dobs.amp_offsets, dobs.n_amp_views, base,
                                          zero_flags, idx, tmp, iv)
    signal = tmp

    # the native handle: compact pointing, crossing list, block-ordered list (once per solve)
    _, setup["crossing_lists_ms"] = _sync_ms(lambda: dobs.handle())
    ds = Destriper([dobs], n_loc, nps, invcov, offset_var, amp_flags, regen=regen, device=device)
    n_good_samples = int(sum(int(v["last"] - v["first"]) for v in iv)) * n_det
    info = dict(n_det=n_det, n_samp=n_samp, nside=nside, n_local_submap=n_loc,
                n_amp=dobs.n_amp, det_samples=n_good_samples, n_hit_pix=n_hit_pix,
                flagged_fraction=float((solver_flags != 0).float().mean().item()),
                setup_ms={k: round(v, 2) for k, v in setup.items()})
    return ds, dobs, signal, info


def describe_path(ds, dobs, lib, regen, world):
    """Which kernels the passes run on and the record statistics."""
    n_rec, n_rows, xp = ct.c_int64(0), ct.c_int64(0), ct.c_int(0)
    lib.tb_obs_crossing_stats(dobs.handle().h, ct.byref(n_rec), ct.byref(n_rows), ct.byref(xp))
    out = {"crossing_records": n_rec.value or None}
    blocked = ds._blocked()
    if blocked:
        nr, nu, nm, nb = ct.c_int64(0), ct.c_int64(0), ct.c_int64(0), ct.c_int64(0)
        lib.tb_obs_blocked_stats(dobs.handle().h, ct.byref(nr), ct.byref(nu), ct.byref(nm),
                                 ct.byref(nb))
        out.update(path="blocked", block_records=nr.value, work_units=nu.value,
                   split_block_units=nm.value, pixel_blocks=nb.value,
                   block_pixels=int(lib.tb_bx_block_pixels()))
    elif regen:
        out["path"] = "regen"
    elif not dobs.has_compact_pointing():
        out["path"] = "per-sample (33 B)"
    elif n_rec.value > 0 and lib.tb_get_option(b"crossings") == 1:
        out["path"] = "pixel-sorted crossing list" if lib.tb_obs_sorted_passes(dobs.handle().h) \
            else "time-ordered crossing list"
    else:
        out["path"] = "per-sample compact (12-20 B)"
    return out, blocked


def pcg_prologue(ds, signal, lib):
    """PCG state exactly as solve() leaves it before the loop."""
    import torch

    from toast_b200 import lib as L
    from toast_b200.solver import _PCGState

    n = ds.n_amp
    st = _PCGState(n, ds.device)
    rhs = ds.rhs([signal])
    st.r.copy_(rhs)
    L.check(lib.tb_template_offset_apply_diag_precond(
        L.ptr(ds.offset_var), L.ptr(st.r), L.ptr(ds.amp_flags), L.ptr(st.s), n, L.TB_MEM_DEVICE,
        None))
    st.d.copy_(st.s)
    ds.dot(st.d, st.r, st.delta)
    tmp = torch.zeros(1, dtype=torch.float64, device=ds.device)
    ds.dot(rhs, rhs, tmp)
    return st, float(tmp.item())


def time_iterations(ds, st, sqsum_init, steps, warmup, world, lib):
    """W warm-up + K timed PCG iterations exactly as Destriper.solve runs them (the next
    direction and LHS are enqueued while the host reads r.r back)."""
    import torch

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    history = []
    host_sums = torch.zeros(2, dtype=torch.float64).pin_memory()
    ev_sums = torch.cuda.Event()

    def step():
        ds.update(st)
        host_sums.copy_(st.sums, non_blocking=True)
        ev_sums.record()
        ds.advance_direction(st)
        ds.lhs_and_dot(st)
        ev_sums.synchronize()
        history.append(float(host_sums[0]) / sqsum_init)  # host convergence test

    ds.prepare_lhs(st.d, st.q)  # (N > 1: the pipeline's CUDA graph, captured on all ranks together)
    ds.lhs_and_dot(st)  # the LHS of the first iteration (prologue of the pipelined loop)
    for _ in range(warmup):
        step()
    launches0 = lib.tb_launch_count()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record()
    barrier()
    launches = lib.tb_launch_count() - launches0
    if ds.pipeline and getattr(ds, "use_graph", False):
        # the pipelined LHS is replayed from a CUDA graph, which tb_launch_count does not see:
        # per LHS the amplitude prescale + (pass 1, ranged reduction, pass 2) per chunk
        launches += steps * (1 + 3 * int(ds.n_chunks))
    return t0.elapsed_time(t1) / max(steps, 1), history, int(launches)


DUMP_SAMPLE = 1 << 20   # entries per dumped vector: three vectors + their index stay below 64 MB


def dump_outputs(out_dir, st, history, rank):
    """What the timed PCG iterations leave a caller of Destriper.solve after the last timed step:
    the amplitudes x, the residual r and the LHS q = A d of the new direction (float64; for longer
    vectors a fixed, seeded sample of DUMP_SAMPLE entries, whose positions are in
    sample_index.npy), and the relative residual of every step, warm-up included.  Ranks other
    than 0 add a _rank<r> suffix."""
    import torch

    n = st.x.numel()
    if n > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    else:
        idx = np.arange(n)
    idx_dev = torch.from_numpy(idx).to(st.x.device)
    arrays = {"sample_index": idx.astype(np.float64),
              "amplitudes": st.x[idx_dev].cpu().numpy(),
              "residual": st.r[idx_dev].cpu().numpy(),
              "lhs": st.q[idx_dev].cpu().numpy(),
              "relative_residuals": np.asarray(history, dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if rank == 0 else f"_rank{rank}"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def time_phases(ds, st, reps=5):
    """Per-phase durations from un-pipelined applications of the same LHS (CUDA events on the
    launching stream; they change neither x nor r)."""
    import torch

    timers = []
    for _ in range(reps + 1):
        ds.lhs(st.d, st.q, timers)
    torch.cuda.synchronize()
    timers = timers[1:]
    p1 = float(np.mean([e[0].elapsed_time(e[1]) for e in timers]))
    pr = float(np.mean([e[1].elapsed_time(e[2]) for e in timers]))
    p2 = float(np.mean([e[2].elapsed_time(e[3]) for e in timers]))
    return p1, pr, p2


def time_dominant_kernel(ds, dobs, st, lib, blocked, fused, reps=10):
    """The dominant kernel alone, CUDA events around its launch on its stream."""
    import torch

    from toast_b200 import lib as L

    if not (blocked and fused):
        return None
    h = dobs.handle().h
    stream = torch.cuda.current_stream(ds.device).cuda_stream
    scratch = torch.zeros_like(st.q)
    ds.lhs(st.d, scratch)  # (prescaled amplitudes of st.d are in place)
    evs = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.tb_bx_fused(h, None, None, L.ptr(ds.cov), L.ptr(ds.zmap), L.ptr(scratch),
                                stream))
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in evs[1:]]))


def source_hash():
    h = hashlib.sha256()
    d = os.path.join(ROOT, "toast_b200", "csrc")
    for f in ("tb_blocked.cu", "tb_device.cuh", "tb_obs.cuh"):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def committed_traffic(kernel, workload, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full`
    capture of this kernel -- only if the kernel sources are the ones that were captured."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, "no capture committed"
    t = json.load(open(path))
    if t.get("source_sha16") != source_hash():
        return None, "kernel sources changed since the committed ncu capture"
    e = t.get("kernels", {}).get(f"{kernel}|{workload}|n{world}")
    if e is None:
        return None, "no capture of this kernel / workload / world size"
    note = e.get("report")
    if e.get("ncu"):   # what the same capture says binds the kernel
        note = {"report": note, "ncu": e["ncu"]}
    return float(e["dram_bytes"]), note


def reduction_parity_and_rate(ds, world, lib):
    """N > 1: the fused NVLink reduction + covariance against NCCL all-reduce + cov_apply on the
    real map, and its stand-alone rate against the NVLink bandwidth."""
    import torch
    import torch.distributed as dist

    from toast_b200 import lib as L

    if world == 1 or ds.peer is None:
        return None, None
    g = torch.Generator(device=ds.device)
    g.manual_seed(77 + dist.get_rank())
    a = torch.randn(ds.n_amp, generator=g, device=ds.device, dtype=torch.float64)
    a[ds.amp_flags != 0] = 0.0
    ds.bin_amplitudes_raw(a)       # this rank's raw noise-weighted map of a random vector
    raw = ds.zmap.clone()
    ref = raw.clone()
    dist.all_reduce(ref)
    L.check(lib.tb_cov_apply_diag(ds.n_local_submap, ds.n_pix_submap, 3, L.ptr(ds.cov),
                                  L.ptr(ref), L.TB_MEM_DEVICE, None))
    ds.zmap.copy_(raw)
    torch.cuda.synchronize()
    dist.barrier()
    ds.reduce_and_apply_cov()
    torch.cuda.synchronize()
    err = float((ds.zmap - ref).abs().max() / ref.abs().max())
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        ds.reduce_and_apply_cov()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    t = torch.tensor([err, ms], dtype=torch.float64, device=ds.device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    err, ms = float(t[0]), float(t[1])
    nbytes = ds.zmap.numel() * 8
    multimem = bool(getattr(ds.peer, "use_multimem", False))
    # bytes every GPU SENDS per call: in-switch reduction -- its copy of the other ranks' slices
    # for the reduce ((N-1)/N of the map) + its reduced slice once for the multicast store (1/N);
    # P2P kernel -- (N-1)/N of the map in the reduce-scatter and again in the all-gather
    per_dir = nbytes * (world - 1) / world * (1.0 if multimem else 2.0) + \
        (nbytes / world if multimem else 0.0)
    rate = per_dir / (ms * 1e-3) / 1e9
    return err, {"standalone_ms": ms, "bytes_per_direction_per_gpu": int(per_dir),
                 "gb_per_s_per_direction": rate,
                 "nvlink_frac": rate / NVLINK_GBS_PER_DIRECTION,
                 "nvlink_peak_gb_per_s_per_direction": NVLINK_GBS_PER_DIRECTION,
                 "kernel": "k_map_reduce_cov_mc (NVLS multimem.ld_reduce + cov + multimem.st)"
                           if multimem else
                           "k_map_reduce_cov (P2P reduce-scatter + cov + all-gather)"}


def e2e_solver_lhs(ds, st, steps, warmup, world, total_samples):
    """SolverLHS.apply through Destriper.lhs with host-resident amplitude vectors: H2D of d,
    both passes + the NVLink map reduction + covariance, D2H of q, every step."""
    import torch

    n = ds.n_amp
    d_host = torch.empty(n, dtype=torch.float64).pin_memory()
    q_host = torch.empty(n, dtype=torch.float64).pin_memory()
    d_host.copy_(st.d)
    d_dev = torch.empty(n, dtype=torch.float64, device=ds.device)
    q_dev = torch.empty(n, dtype=torch.float64, device=ds.device)

    def step():
        d_dev.copy_(d_host, non_blocking=True)
        ds.lhs(d_dev, q_dev)
        q_host.copy_(q_dev, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    ds.prepare_lhs(d_dev, q_dev)
    for _ in range(warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / max(steps, 1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=ds.device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return {"value": total_samples / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": n * 8,
            "what": "Destriper.lhs (SolverLHS.apply, mapmaker_solve.py:342-506) with the "
                    "amplitude vectors in pinned host memory: H2D of d, both passes + NVLink map "
                    "reduction + covariance, D2H of q; timestream-derived data device-resident "
                    "as in the reference's accel pipeline.  (N = 1 reports ops.MapMaker.apply "
                    "end to end instead.)"}


def e2e_mapmaker(workload, n_det, n_samp, n_iter, device, rank, world):
    """ops.MapMaker.apply (the reference's entry point, ops/mapmaker.py:719-787): host numpy
    buffers (pinned) in, maps / amplitudes / cleaned timestreams out.  Everything is inside the
    timed region: H2D of boresight / flags / signal, pointing expansion, covariance, crossing
    lists, RHS, n_iter PCG iterations, final binning, D2H of the products."""
    import torch

    from toast_b200 import ops
    from toast_b200.data import Data, observation_from_synthetic
    from toast_b200.templates.offset import Offset

    obs = S.make_observation(workload, n_det=n_det, n_samp=n_samp, det_first=rank * n_det)
    data = Data()
    data.obs.append(observation_from_synthetic(obs, pinned=True))
    h2d = (obs["boresight"].nbytes + obs["shared_flags"].nbytes + obs["det_flags"].nbytes +
           obs["signal"].nbytes)
    del obs["signal"], obs["det_flags"]
    dp = ops.PointingDetectorSimple(view="scanning", shared_flags="flags", shared_flag_mask=1)
    pix = ops.PixelsHealpix(detector_pointing=dp, nside=obs["nside"], nest=obs["nest"],
                            create_dist="pixel_dist")
    wts = ops.StokesWeights(detector_pointing=dp, mode="IQU")
    binning = ops.BinMap(pixel_dist="pixel_dist", covariance="cov", pixel_pointing=pix,
                         stokes_weights=wts, noise_model="noise_model", full_pointing=True)
    tmpl = Offset(name="baselines", step_time=obs["step_time"], times="times",
                  noise_model="noise_model")
    tmat = ops.TemplateMatrix(templates=[tmpl], amplitudes="amplitudes")
    mapper = ops.MapMaker(name="mm", det_data="signal", binning=binning, template_matrix=tmat,
                          iter_max=n_iter, iter_min=n_iter, convergence=1.0e-300,
                          device=str(device),
                          profile_stages=os.environ.get("TB_E2E_STAGES", "0") == "1")
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mapper.apply(data)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    d2h = sum(data[f"mm_{k}"].data.nbytes for k in ("hits", "cov", "rcond", "binmap", "map")) + \
        data.obs[0].detdata["signal"].data.nbytes + data["amplitudes"]["baselines"].local.nbytes
    iters = len(mapper.history)
    n_good = int(sum(int(v["last"] - v["first"]) for v in obs["intervals"])) * n_det
    if mapper.stage_seconds:
        print("e2e stages (s):", {k: round(v, 3) for k, v in mapper.stage_seconds.items()},
              file=sys.stderr)
    return dict(seconds=dt, iterations=iters, det_samples=n_good, h2d_bytes=int(h2d),
                d2h_bytes=int(d2h), final_relative_residual=float(mapper.history[-1]))


def sub_run(workload, regen, device, lib, steps=8, warmup=3):
    """A short run of another BASELINE workload on one GPU (same timing rules)."""
    import torch

    t_wall = time.perf_counter()
    ds, dobs, signal, info = build_gpu_problem(workload, regen, 1.0, 0, 1, device)
    st, sq0 = pcg_prologue(ds, signal, lib)
    ms, hist, _ = time_iterations(ds, st, sq0, steps, warmup, 1, lib)
    path, blocked = describe_path(ds, dobs, lib, regen, 1)
    p1, pr, p2 = time_phases(ds, st, reps=3)
    out = {
        "config": f"{workload}: {info['n_det']} det x {info['n_samp']} samples, nside "
                  f"{info['nside']}, " + ("pointing regenerated per pass" if regen
                                          else "stored pointing"),
        "value": info["det_samples"] / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
        "steps": steps, "warmup": warmup, "pass1_ms": p1, "reduce_cov_ms": pr, "pass2_ms": p2,
        "path": path.get("path"),
        "samples_per_record": (info["det_samples"] / path["crossing_records"]
                               if path.get("crossing_records") else None),
        "split_block_units": path.get("split_block_units"),
        "effective_frac_of_peak": None, "setup_ms": info["setup_ms"],
        "relative_residuals": hist[warmup:warmup + 3],
        "wall_s": None,
    }
    del ds, dobs, signal, st
    torch.cuda.empty_cache()
    out["wall_s"] = round(time.perf_counter() - t_wall, 1)
    return out, info


def c2_operator_chain(device, lib, reps=5):
    """BASELINE config C2 as defined: pointing + weights + BuildNoiseWeighted on one B200
    (1000 detectors x 1 h @ 100 Hz, nside 512 NEST): the fused pointing kernel followed by the
    noise-weighted binning of a stored timestream, operator kernels behind the C ABI."""
    import torch

    from toast_b200 import kernels as K

    sh = SHARDS["c2"]
    n_det, n_samp = sh["n_det"], sh["n_samp"]
    obs = S.make_observation("c2", n_det=n_det, n_samp=n_samp, with_signal=False, flags=False)
    nside, nest = obs["nside"], obs["nest"]
    n_submap, nps = S.n_submap_for(nside, 16)
    iv = obs["intervals"]
    idx = np.arange(n_det, dtype=np.int32)
    bore = torch.from_numpy(obs["boresight"]).to(device)
    sflags = torch.zeros(n_samp, dtype=torch.uint8, device=device)
    pixels = torch.zeros((n_det, n_samp), dtype=torch.int64, device=device)
    weights = torch.zeros((n_det, n_samp, 3), dtype=torch.float64, device=device)
    hits = np.zeros(n_submap, dtype=np.uint8)

    def pointing():
        K.pointing_fused(obs["focalplane"], bore, sflags, 1, None, None, idx, pixels, idx, weights,
                         None, iv, hits, nps, nside, nest, obs["epsilon"], obs["gamma"],
                         obs["cal"], False)

    pointing()
    local = np.flatnonzero(hits).astype(np.int64)
    g2l = np.full(n_submap, -1, dtype=np.int64)
    g2l[local] = np.arange(len(local))
    zmap = torch.zeros((len(local), nps, 3), dtype=torch.float64, device=device)
    signal = torch.randn((n_det, n_samp), dtype=torch.float64, device=device)
    dflags = torch.zeros((n_det, n_samp), dtype=torch.uint8, device=device)

    def binning():
        K.build_noise_weighted(g2l, zmap, idx, pixels, idx, weights, idx, signal, idx, dflags,
                               obs["detweight"], 1, iv, sflags, 1)

    binning()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tp, tb = [], []
    for _ in range(reps):
        ev[0].record()
        pointing()
        ev[1].record()
        binning()
        ev[2].record()
        torch.cuda.synchronize()
        tp.append(ev[0].elapsed_time(ev[1]))
        tb.append(ev[1].elapsed_time(ev[2]))
    n_good = int(sum(int(v["last"] - v["first"]) for v in iv)) * n_det
    tp, tb = float(np.mean(tp)), float(np.mean(tb))
    out = {"config": f"c2 as defined: pointing + weights + BuildNoiseWeighted, {n_det} det x "
                     f"{n_samp} samples, nside {nside} NEST",
           "det_samples": n_good, "pointing_fused_ms": tp, "build_noise_weighted_ms": tb,
           "value": n_good / ((tp + tb) * 1e-3), "unit": "det-samples/s",
           # pointing writes pixel 8 + weights 24; binning reads pixel 8 + weights 24 + signal 8
           # + flag 1 (SURVEY 8d)
           "algorithmic_bytes": n_good * (32 + 41)}
    del pixels, weights, signal, dflags, zmap
    torch.cuda.empty_cache()
    return out


def noise_prior_sub_run(device, lib, peak, reps=10):
    """SURVEY 8f.3: the Offset noise prior on the C4 shard (one 12-h view per detector: 128
    segments of 43 200 baselines; 1/f PSD, banded preconditioner of width 20): tb_offset_prior_add
    (Offset._add_prior, templates/offset/offset.py:884-960) and tb_offset_prior_precond
    (Offset._apply_precond, :962-1010) timed alone with CUDA events, plus PCG iterations with the
    prior in the loop."""
    import torch

    from toast_b200.templates.offset_prior import OffsetPriorBuilder, prior_frequencies

    ds, dobs, signal, info = build_gpu_problem("c4", False, 1.0, 0, 1, device)
    n_amp, nad = ds.n_amp, dobs.n_amp_det
    step_time = S.CONFIGS["c4"]["step_time"]
    rate = S.CONFIGS["c4"]["rate"]
    t0 = time.perf_counter()
    b = OffsetPriorBuilder(n_amp, precond_width=20)
    freq = prior_frequencies(info["n_samp"] / rate, step_time, rate)
    pf = np.logspace(-5, np.log10(rate / 2), 400)
    var = ds.offset_var.cpu().numpy()
    # (flagged baselines have variance 0 -> 1 / var = inf, with which the reference's banded
    # preconditioner cannot be built at all, offset.py:520-531; the timing problem gives them the
    # median variance instead -- they stay flagged in the solver)
    var = np.where(var > 0, var, np.median(var[var > 0]))
    for d in range(info["n_det"]):
        sigma2 = 1.0 / dobs.det_scale[d]
        psd = sigma2 / rate * (1.0 + (0.05 / pf) ** 1.5)   # white level + 1/f, f_knee 50 mHz
        b.add_detector(int(dobs.amp_offsets[d]), dobs.n_amp_views, pf, psd,
                       float(dobs.det_scale[d]), var, freq, step_time)
    prior = b.finish()
    build_s = time.perf_counter() - t0
    taps = int(np.mean(b.filt_len))
    band = int(np.mean(b.prec_width))
    g = torch.Generator(device=device)
    g.manual_seed(5)
    a = torch.randn(n_amp, generator=g, device=device, dtype=torch.float64)
    out = torch.zeros_like(a)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms_add = timed(lambda: prior.add(a, ds.amp_flags, out))
    ms_pre = timed(lambda: prior.precond(a, ds.amp_flags, out))
    # with the prior in the PCG
    ds.prior = prior
    st, sq0 = pcg_prologue(ds, signal, lib)
    ms_iter, hist, _ = time_iterations(ds, st, sq0, 8, 3, 1, lib)
    res = {
        "config": f"c4 shard, {info['n_det']} segments of {nad} baselines, filter taps ~{taps}, "
                  f"preconditioner band {band}",
        "prior_build_host_s": round(build_s, 2),
        "banded_solve": (f"partitioned, chunks of {lib.tb_get_option(b'prior_chunk')} baselines"
                         if lib.tb_get_option(b"prior_chunk") > 0 else "one thread per segment"),
        "add_prior_ms": ms_add, "apply_precond_ms": ms_pre,
        # compulsory: amplitudes in, flags, out (read + write for add); the filter / factor
        # values are shared by a segment (add) or streamed once (banded factor: band x n_amp)
        "add_prior_frac_of_peak": n_amp * (8 + 1 + 16) / (ms_add * 1e-3) / 1e9 / peak,
        "apply_precond_frac_of_peak": n_amp * (8 + 1 + 8 + 8 * band) / (ms_pre * 1e-3) / 1e9 / peak,
        "pcg_iteration_with_prior_ms": ms_iter,
        "relative_residuals": hist[3:6],
    }
    del ds, dobs, signal, st, prior
    torch.cuda.empty_cache()
    return res


def cpu_sample_parity(problem, device):
    """Part of the cpu_baseline leg: the GPU path on the SAME sample the reference's compiled
    kernels just ran (64 detectors, production rcond) -- pixels bit-exact, RHS / LHS relative
    error."""
    import torch

    from toast_b200.solver import DeviceObservation, Destriper

    O, kern, obs, pb, covapply = problem
    dobs = DeviceObservation(
        focalplane=obs["focalplane"], boresight=obs["boresight"], intervals=obs["intervals"],
        det_scale=pb.det_scale, step_length=pb.step_length, nside=pb.nside, nest=pb.nest,
        n_pix_submap=pb.n_pix_submap, n_submap=pb.n_submap, global2local=pb.global2local,
        epsilon=obs["epsilon"], gamma=obs["gamma"], cal=obs["cal"],
        shared_flags=pb.shared_flags, shared_flag_mask=pb.shared_flag_mask,
        solver_flags=pb.solver_flags, solver_flag_mask=pb.det_flag_mask, device=device)
    dobs.expand_pointing(np.zeros(pb.n_submap, dtype=np.uint8))
    pixels_equal = bool(np.array_equal(dobs.pixels.cpu().numpy(), pb.pixels))
    ds = Destriper([dobs], pb.n_local_submap, pb.n_pix_submap, pb.cov, pb.offset_var,
                   pb.amp_flags, device=device)
    nrm = lambda a, b: float(np.max(np.abs(a - b)) / np.max(np.abs(b)))
    rhs_ref = O.solver_rhs(pb, kern, obs["signal"], covapply)
    rhs = ds.rhs([torch.from_numpy(obs["signal"]).to(device)])
    rng = np.random.default_rng(5)
    a = np.where(pb.amp_flags == 0, rng.standard_normal(pb.n_amp), 0.0)
    lhs_ref = O.solver_lhs(pb, kern, a, covapply)
    lhs_rev = O.solver_lhs(pb, kern, a, covapply, reverse=True)
    q = torch.zeros(pb.n_amp, dtype=torch.float64, device=device)
    ds.lhs(torch.from_numpy(a).to(device), q)
    return {"cpu_sample_pixels_bit_exact": pixels_equal,
            "cpu_sample_rhs_rel_err": nrm(rhs.cpu().numpy(), rhs_ref),
            "cpu_sample_lhs_rel_err": nrm(q.cpu().numpy(), lhs_ref),
            "cpu_sample_lhs_reference_order_dependence": nrm(lhs_rev, lhs_ref),
            "cpu_sample_conditioning_bar": 0.1 * float(np.finfo(np.float64).eps) / 1.0e-8,
            "cpu_sample_note": "rcond 1e-8 keeps pixels with condition numbers up to 1e8: the "
                               "reference's own LHS moves by `reference_order_dependence` when "
                               "it sums the detectors in reverse order",
            "cpu_sample_check": "GPU path vs the reference's compiled kernels on the "
                                "cpu_baseline sample (max|a-b| / max|b|)"}


def _release_cached_memory():
    """torch.cuda.empty_cache() for the error paths of the optional legs: must not raise itself."""
    try:
        import torch

        torch.cuda.empty_cache()
    except Exception:
        pass


def main_gpu(args):
    import torch

    from toast_b200 import lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the toast_b200 path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # a rank stuck in a collective or in a device-side barrier would otherwise sit there until
        # the caller's limit: say where and leave (the run normally takes about a minute)
        import faulthandler

        faulthandler.dump_traceback_later(600, exit=True)
        torch.distributed.init_process_group("nccl", device_id=device)
    lib = L.load()

    ds, dobs, signal, info = build_gpu_problem(args.workload, args.regen, args.scale, rank, world,
                                               device)
    st, sqsum_init = pcg_prologue(ds, signal, lib)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # sampled under load: warm-up + timed region
    ms_step, history, launches = time_iterations(ds, st, sqsum_init, args.steps, args.warmup,
                                                 world, lib)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, st, history, rank)

    path, blocked = describe_path(ds, dobs, lib, args.regen, world)
    fused = blocked and world == 1 and ds.fuse_lhs and len(ds.obs) == 1
    was_pipelined = ds.pipeline
    ds.pipeline = False
    p1, pr, p2 = time_phases(ds, st)
    dom_ms_alone = time_dominant_kernel(ds, dobs, st, lib, blocked, fused)
    red_err, nvlink = reduction_parity_and_rate(ds, world, lib)
    ds.pipeline = was_pipelined

    # max over ranks
    if world > 1:
        t = torch.tensor([ms_step, p1, p2, pr], dtype=torch.float64, device=device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_step, p1, p2, pr = [float(x) for x in t.tolist()]
        cnt = torch.tensor([info["det_samples"]], dtype=torch.float64, device=device)
        torch.distributed.all_reduce(cnt)
        total_samples = float(cnt.item())
    else:
        total_samples = float(info["det_samples"])

    # N > 1: the LHS through the host-facing solver call with the amplitude vectors in pinned
    # host memory (ops.MapMaker.apply is the N = 1 end-to-end measurement; its multi-rank form
    # is exercised by the 2-rank tests and can be selected with TB_E2E_MAPMAKER_MULTI=1)
    # (also measured at N = 1: reported as `e2e_solver_lhs`, and the fall-back `e2e` should the
    # MapMaker run below fail)
    e2e_lhs = e2e_solver_lhs(ds, st, args.steps, min(args.warmup, 2), world, total_samples)

    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else \
        "fallback 6650 GB/s (B200_PROFILING.md)"
    n_amp = info["n_amp"]
    zmap_bytes = int(ds.zmap.numel() * 8)
    pipe_note = (f"{ds.n_chunks} pixel chunks: pass 1 -> NVLink reduction -> pass 2 overlapped "
                 "on two streams") if ds.pipeline else None
    peer_info = dict(
        tune_ms=getattr(ds.peer, "tune_ms", None),
        what=("fused NVLS kernel: multimem.ld_reduce + cov + multimem.st"
              if getattr(ds.peer, "use_multimem", False) else
              "fused P2P reduce-scatter + cov + all-gather kernel") if ds.peer is not None else
             ("NCCL all-reduce + cov_apply" if world > 1 else
              ("inside the fused kernel" if fused else "cov_apply")),
        pipe_tune_ms=getattr(ds, "pipe_tune_ms", None))
    n_det_here = dobs.n_det
    del ds, dobs, st, signal
    torch.cuda.empty_cache()

    # ---- end to end ---------------------------------------------------------------------------
    e2e, r = None, None
    multi_mapmaker = os.environ.get("TB_E2E_MAPMAKER_MULTI", "0") == "1"
    if world > 1 and not multi_mapmaker:
        e2e = e2e_lhs
    elif not args.no_extras:
        n_iter = max(args.steps, 1)
        try:
            r = e2e_mapmaker(args.workload, info["n_det"], info["n_samp"], n_iter, device, rank,
                             world)
        except Exception as exc:  # the headline survives: e2e falls back to the solver-LHS form
            if world > 1:
                raise
            r = None
            e2e = dict(e2e_lhs)
            e2e["mapmaker_error"] = repr(exc)[:300]
            _release_cached_memory()
    if r is not None:
        tt = torch.tensor([r["seconds"]], dtype=torch.float64, device=device)
        if world > 1:
            torch.distributed.all_reduce(tt, op=torch.distributed.ReduceOp.MAX)
        sec = float(tt.item())
        e2e = {"value": total_samples * r["iterations"] / sec, "unit": UNIT,
               "ms_per_step": sec * 1e3 / r["iterations"],
               "h2d_bytes_per_step": r["h2d_bytes"] // r["iterations"],
               "d2h_bytes_per_step": r["d2h_bytes"] // r["iterations"],
               "iterations": r["iterations"], "seconds_total": sec,
               "h2d_bytes_total": r["h2d_bytes"], "d2h_bytes_total": r["d2h_bytes"],
               "final_relative_residual": r["final_relative_residual"],
               "what": "ops.MapMaker.apply (ops/mapmaker.py:719-787) on host numpy buffers in "
                       "pinned memory: H2D of boresight, flags and signal, pointing expansion, "
                       "covariance, crossing lists, RHS, the PCG iterations, final binning, D2H "
                       "of hits / covariance / maps / amplitudes / cleaned timestreams; total "
                       "wall time divided by the PCG iterations"}
        torch.cuda.empty_cache()

    line = None
    if rank == 0:
        n_rec = path.get("block_records") or path.get("crossing_records") or 0
        if blocked:
            rec_bytes = 24 * n_rec
            scratch = 32 * (n_amp // 2 if n_det_here % 2 == 0 else n_amp)  # {a0w0,a1w1,w0,w1}
            if fused:
                dom = "k_bx<2> (pass 1 + pixel covariance + pass 2 in one kernel, block-ordered " \
                      "crossing list, warp-private shared-memory map tiles)"
                dom_key = "k_bx<2>"
                dom_ms = dom_ms_alone if dom_ms_alone is not None else p2
                # records once (second sweep served by the L2), covariance of the hit pixels,
                # prescaled amplitudes once, output vector once
                compulsory = rec_bytes + 48 * info["n_hit_pix"] + scratch + 8 * n_amp
                what = "24 B x records + 48 B x hit pixels + 32 B x amplitude pairs + 8 B x " \
                       "amplitudes"
            elif p1 >= p2:
                dom, dom_key, dom_ms = "k_bx<0> (pass 1: template -> noise-weighted map, " \
                    "block-ordered crossing list, warp-private shared-memory tiles)", \
                    "k_bx<0>", p1
                compulsory = rec_bytes + scratch + zmap_bytes
                what = "24 B x records + 32 B x amplitude pairs + the map written once " \
                       "(pass1_ms also holds the 0.03 ms amplitude prescale)"
            else:
                dom, dom_key, dom_ms = "k_bx<1> (pass 2: scan - weight - project, " \
                    "block-ordered crossing list)", "k_bx<1>", p2
                compulsory = rec_bytes + scratch + zmap_bytes + 8 * n_amp
                what = "24 B x records + 32 B x amplitude pairs + the map read once + 8 B x " \
                       "amplitudes"
        else:
            dom, dom_key = (f"pass 1 ({path['path']})", "pass1") if p1 >= p2 else \
                (f"pass 2 ({path['path']})", "pass2")
            dom_ms = max(p1, p2)
            per = {"regen": 1, "per-sample (33 B)": 33}.get(path["path"])
            compulsory = (per * info["det_samples"] if per else 32 * n_rec) + zmap_bytes
            what = "bytes streamed per pass + the map once"
        achieved = compulsory / (dom_ms * 1e-3) / 1e9
        traffic, traffic_note = committed_traffic(dom_key, args.workload, world)
        iter_gbs = info["det_samples"] * BYTES_PER_SAMPLE_ITER / (ms_step * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": total_samples / (ms_step * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            # (`config` is what both arms are quoted on -- the reference arm prints the same
            # dictionary; what this arm found out about the problem goes to `problem`)
            "config": config_dict(args, world, info["n_det"], info["n_samp"], info["nside"],
                                  {"rcond_threshold": 1.0e-8}),
            "problem": {"n_amplitudes_per_gpu": n_amp,
                        "n_local_submaps": info["n_local_submap"],
                        "n_hit_pixels": info["n_hit_pix"],
                        "flagged_fraction": round(info["flagged_fraction"], 4)},
            "roofline": {
                "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peak_src,
                "kernel_ms": dom_ms, "compulsory_bytes_per_launch": int(compulsory),
                "compulsory_bytes_are": what,
                "pass1_ms": p1, "pass2_ms": p2, "reduce_cov_ms": pr,
                "phase_note": "fused LHS: pass2_ms holds prescale + the fused kernel" if fused
                              else "from un-pipelined applications outside the timed region",
                "map_reduction_tuning_ms": peer_info["tune_ms"],
                "map_reduction": peer_info["what"],
                "zmap_bytes": zmap_bytes,
                "pipeline_tuning_ms": peer_info["pipe_tune_ms"],
                "pipeline": pipe_note,
                "records": path,
                "samples_per_record": (info["det_samples"] / path["crossing_records"]
                                       if path.get("crossing_records") else None),
                "effective_bytes_per_sample_per_iteration": BYTES_PER_SAMPLE_ITER,
                "effective_gbs_per_gpu": iter_gbs,
                "effective_frac_of_peak": iter_gbs / peak,
                "effective_note": "the reference layout's 66 B/det-sample (SURVEY 8d) over the "
                                  "iteration time: what an implementation streaming stored "
                                  "pointing would have to sustain; not a roofline fraction",
            },
            "nvlink": nvlink,
            "setup_ms": info["setup_ms"],
            "parity": {"map_reduce_max_rel_err": red_err,
                       "map_reduce_check": "fused NVLink reduction + covariance vs NCCL "
                                           "all-reduce + cov_apply on the real map (max over "
                                           "ranks)" if world > 1 else None},
            "e2e": e2e if e2e is not None else {"value": None, "unit": UNIT,
                                                "h2d_bytes_per_step": None,
                                                "d2h_bytes_per_step": None,
                                                "skipped": "--no-extras"},
            "e2e_solver_lhs": e2e_lhs if (world == 1 and e2e_lhs is not None) else None,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "pcg_relative_residuals": history[args.warmup:args.warmup + 5],
        }

    if rank == 0 and world == 1 and not args.no_extras:
        others = {}
        for key, wl, regen in (("c2", "c2", False), ("c3", "c3", False),
                               ("c3_regen", "c3", True), ("c5", "c5", False)):
            if wl == args.workload and regen == args.regen:
                continue
            try:
                o, _ = sub_run(wl, regen, device, lib)
                o["effective_frac_of_peak"] = o["value"] * BYTES_PER_SAMPLE_ITER / 1e9 / peak
                others[key] = o
            except Exception as exc:  # a sub-run never takes the headline down
                others[key] = {"error": repr(exc)[:300]}
                _release_cached_memory()
        try:
            o = c2_operator_chain(device, lib)
            o["frac_of_peak"] = o["algorithmic_bytes"] / \
                ((o["pointing_fused_ms"] + o["build_noise_weighted_ms"]) * 1e-3) / 1e9 / peak
            others["c2_operator_chain"] = o
        except Exception as exc:
            others["c2_operator_chain"] = {"error": repr(exc)[:300]}
        try:
            others["noise_prior"] = noise_prior_sub_run(device, lib, peak)
        except Exception as exc:
            others["noise_prior"] = {"error": repr(exc)[:300]}
            _release_cached_memory()
        line["other_workloads"] = others

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:  # reported at N=1 only
            try:
                res = run_cpu(args.workload, 2, 1, want_problem=True)
                line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind",
                                                            "sample")}
                line["parity"].update(cpu_sample_parity(res["_problem"], device))
            except Exception as exc:  # the baseline is a report, never a gate
                line["cpu_baseline"] = {"error": repr(exc)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()
        faulthandler.cancel_dump_traceback_later()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_gpu(a)
