"""TemplateMatrix and MapMaker (``ops/mapmaker_templates.py:27-357``, ``ops/mapmaker.py:
28-787``, ``ops/mapmaker_solve.py``) with the Offset-template solve running on the fused,
device-resident destriper (``toast_b200.solver``).

``MapMaker._exec`` follows the stages of the reference (SURVEY.md 3.1):
solver flags -> pixel distribution -> CovarianceAndHits -> rcond mask -> RHS -> PCG ->
raw binned map -> template-cleaned binned map.  Every per-sample stage is a CUDA kernel; the
host only orchestrates and reads back one scalar per PCG iteration.
"""

import numpy as np

from .. import kernels as KC
from ..pixels import PixelData, PixelDistribution
from ..templates.amplitudes import AmplitudesMap
from ..templates.offset import Offset
from .operator import Operator
from .pixels_wcs import PixelsWCS


def _identity_rows(dd, dets):
    idx = dd.indices(dets)
    return len(idx) == dd.data.shape[0] and np.array_equal(idx, np.arange(len(idx)))


def _rows_to_device(dd, dets, dev):
    """The detdata rows of ``dets`` as a device tensor.  All rows in order (the usual case): one
    asynchronous copy straight from the host buffer (page-locked buffers overlap with compute);
    otherwise the selected rows are gathered on the host first."""
    import torch

    if _identity_rows(dd, dets):
        src = dd._pinned if getattr(dd, "_pinned", None) is not None else torch.from_numpy(dd.data)
        return src.to(dev, non_blocking=True)
    return torch.from_numpy(np.ascontiguousarray(dd.data[dd.indices(dets)])).to(dev)


def _amp_flags_and_variance(n_good, amplen, detnoise, good_fraction):
    """Amplitude flags and the diagonal preconditioner of the Offset template
    (``offset.py:283-344``): an amplitude is kept when more than ``good_fraction`` of its samples
    are good and its detector weight is positive; ``offset_var = 1 / (detweight * n_good)``.
    Plain IEEE element-wise arithmetic on torch tensors of any device (the same bits as the numpy
    form in ``templates/offset.py``).  Returns (flagged [bool], offset_var [f64])."""
    import torch

    zero = torch.zeros_like(n_good)
    frac = torch.where(amplen > 0, n_good / amplen, zero)
    keep = (frac > good_fraction) & (detnoise > 0)
    offset_var = torch.where(keep, 1.0 / (detnoise * n_good), zero)
    return ~keep, offset_var


def _fill_amp_layout(amplen, detnoise, amp_offsets, n_amp_det, lens, det_scale):
    """Per-amplitude baseline length and detector weight for the detectors of one observation:
    ``amplen[o_k : o_k + n_amp_det] = lens``, ``detnoise[...] = det_scale[k]`` for every detector
    k (in place; tensors of any device)."""
    import torch

    offs = np.asarray(amp_offsets, dtype=np.int64)
    n_det = len(offs)
    if n_det == 0 or n_amp_det == 0:
        return
    lens_t = torch.as_tensor(np.ascontiguousarray(lens, dtype=np.float64)).to(amplen.device)
    w_t = torch.as_tensor(np.ascontiguousarray(det_scale, dtype=np.float64)).to(amplen.device)
    if np.all(np.diff(offs) == n_amp_det):
        # detector-major and contiguous (one observation, or the detectors of this observation
        # next to each other): two strided assignments
        o0 = int(offs[0])
        amplen[o0:o0 + n_det * n_amp_det].view(n_det, n_amp_det)[:] = lens_t[None, :]
        detnoise[o0:o0 + n_det * n_amp_det].view(n_det, n_amp_det)[:] = w_t[:, None]
        return
    for k, o in enumerate(offs):
        o = int(o)
        amplen[o:o + n_amp_det] = lens_t
        detnoise[o:o + n_amp_det] = w_t[k]


def _pixdata_from_device(dist, t, dtype, n_value):
    """A finished device map as a PixelData: ONE device -> host copy straight into the product's
    own buffer (no intermediate host tensor, no zero-fill of pages that are overwritten anyway)."""
    import torch

    p = PixelData(dist, dtype, n_value=n_value, zero=False)
    torch.from_numpy(p.data).copy_(t.reshape(p.data.shape))
    return p


def _rows_from_device(dd, dets, t):
    import torch

    if _identity_rows(dd, dets):
        dst = dd._pinned if getattr(dd, "_pinned", None) is not None else torch.from_numpy(dd.data)
        dst.copy_(t)
    else:
        dd.data[dd.indices(dets)] = t.cpu().numpy()


class TemplateMatrix(Operator):
    _defaults = dict(templates=None, amplitudes=None, transpose=False, view=None,
                     det_data="signal", det_mask=1, det_flags=None, det_flag_mask=1)

    def _init_templates(self, data, detectors):
        if getattr(self, "_initialized", False):
            return
        for tmpl in self.templates:
            tmpl.view = self.view if tmpl.view is None else tmpl.view
            tmpl.det_data = self.det_data
            tmpl.det_mask = self.det_mask
            tmpl.det_flags = self.det_flags
            tmpl.det_flag_mask = self.det_flag_mask
            tmpl.initialize(data, detectors)
        self._initialized = True

    def reset(self):
        self._initialized = False

    def _exec(self, data, detectors=None, use_accel=False, **kwargs):
        if self.templates is None or self.amplitudes is None:
            raise RuntimeError("You must set the templates and amplitudes traits")
        self._init_templates(data, None)
        for tmpl in self.templates:
            tmpl.det_data = self.det_data
        if self.amplitudes not in data:
            if not self.transpose:
                raise RuntimeError(f"Template amplitudes '{self.amplitudes}' do not exist")
            amps = AmplitudesMap()
            for tmpl in self.templates:
                amps[tmpl.name] = tmpl.zeros()
            data[self.amplitudes] = amps
        amps = data[self.amplitudes]
        for det in data.all_local_detectors(selection=detectors, flagmask=self.det_mask):
            for tmpl in self.templates:
                if self.transpose:
                    tmpl.project_signal(det, amps[tmpl.name], use_accel=use_accel)
                else:
                    tmpl.add_to_signal(det, amps[tmpl.name], use_accel=use_accel)

    def apply_precond(self, amps_in, amps_out, use_accel=False):
        for tmpl in self.templates:
            tmpl.apply_precond(amps_in[tmpl.name], amps_out[tmpl.name], use_accel=use_accel)

    def add_prior(self, amps_in, amps_out, use_accel=False):
        for tmpl in self.templates:
            tmpl.add_prior(amps_in[tmpl.name], amps_out[tmpl.name], use_accel=use_accel)

    def _requires(self):
        return {"detdata": [self.det_data], "global": [self.amplitudes]}

    def _provides(self):
        return {"detdata": [self.det_data]} if not self.transpose else {"global": [self.amplitudes]}


class MapMaker(Operator):
    """Generalised destriper restricted to what the hot path covers: HEALPix
    (``ops.PixelsHealpix``) or flat-sky WCS (``ops.PixelsWCS``) pointing, I/Q/U weights, a
    diagonal noise model and ONE ``templates.Offset`` template.  With ``PixelsWCS`` the projection
    is set up as that operator does (auto bounds from the boresights of every observation), and
    the pixel distribution carries ``wcs`` / ``wcs_shape``.

    Products placed in ``data`` (names as in ``ops/mapmaker.py:382-651``):
    ``{name}_hits``, ``{name}_cov``, ``{name}_rcond``, ``{name}_binmap`` (raw binned map),
    ``{name}_map`` (template-cleaned map) and the solved ``AmplitudesMap`` under
    ``template_matrix.amplitudes``.  ``self.history`` is the PCG relative-residual history the
    reference logs at ``mapmaker_solve.py:701-706``.
    """

    _defaults = dict(det_data="signal", det_mask=1, det_flags="flags", det_flag_mask=1,
                     shared_flags="flags", shared_flag_mask=1, convergence=1.0e-12, iter_min=3,
                     iter_max=100, solve_rcond_threshold=1.0e-8, map_rcond_threshold=1.0e-8,
                     binning=None, template_matrix=None, map_binning=None,
                     regenerate_pointing=False, keep_solver_products=False, device="cuda",
                     profile_stages=False)

    def _exec(self, data, detectors=None, use_accel=True, **kwargs):
        import torch

        from ..solver import DeviceObservation, Destriper

        for trait in ("binning", "template_matrix"):
            if getattr(self, trait) is None:
                raise RuntimeError(f"You must set the '{trait}' trait before calling exec()")
        if self.map_binning is not None and self.map_binning is not self.binning:
            # (the reference bins the final maps with a second operator, mapmaker.py:386-470)
            raise NotImplementedError("a map_binning operator distinct from binning is not "
                                      "supported on the B200 path")
        binning = self.binning
        pixels, weights = binning.pixel_pointing, binning.stokes_weights
        if pixels is None or weights is None:
            raise RuntimeError("binning must have pixel_pointing and stokes_weights set")
        if weights.mode != "IQU":
            raise NotImplementedError("the fused destriper implements mode='IQU'")
        tmpls = self.template_matrix.templates
        if len(tmpls) != 1 or not isinstance(tmpls[0], Offset):
            raise NotImplementedError("MapMaker on the B200 path supports one Offset template")
        tmpl = tmpls[0]
        is_wcs = isinstance(pixels, PixelsWCS)
        dp = pixels.detector_pointing
        view = pixels.view if pixels.view is not None else dp.view
        if is_wcs:
            pixels._geometry(data)
            pixelisation = dict(wcs=pixels.wcs)
        else:
            pixels._geometry()
            pixelisation = dict(nside=pixels.nside, nest=pixels.nest)
        dev = torch.device(self.device)
        comm = data.comm
        # wall-clock per stage (device synchronised at every mark) when profile_stages is set
        import time as _time

        self.stage_seconds = {}
        _t = [_time.perf_counter()]

        def mark(name):
            if not self.profile_stages:
                return
            torch.cuda.synchronize(dev)
            now = _time.perf_counter()
            self.stage_seconds[name] = self.stage_seconds.get(name, 0.0) + now - _t[0]
            _t[0] = now

        # --- template layout (host, O(n_amp)) ------------------------------------------------
        self.template_matrix.view = view if self.template_matrix.view is None else \
            self.template_matrix.view
        self.template_matrix.det_data = self.det_data
        self.template_matrix.det_flags = None  # solver flags are applied on the device below
        self.template_matrix.reset()
        tmpl._defer_prior = True  # built below, from the variance under the full solver flags
        tmpl._defer_variance = True  # (and so are the amplitude flags / variance themselves)
        tmpl._device = dev           # (long time vectors: the sample rate's median on the device)
        self.template_matrix._init_templates(data, detectors)

        # --- device observations, solver flags bit 0 (mapmaker_templates.py:764-810) -----------
        dobs, signals = [], []
        main_stream = torch.cuda.current_stream(dev)
        upload = torch.cuda.Stream(device=dev)
        for iob, ob in enumerate(data.obs):
            dets = [d for d in tmpl._all_dets if d in tmpl._obs_dets[iob]]
            fp = ob[dp.focalplane_key]
            # with a noise prior the baselines span the observation and the view only flags
            # samples (offset.py:136-141; the view flags are ORed into the solver flags below)
            iv = ob.intervals[tmpl._bounds_view if tmpl.use_noise_prior else view]
            sflag = ob.shared[self.shared_flags] if self.shared_flags is not None else None
            # solver flags are combined on the device: the detector flags travel as they are
            # (one asynchronous copy from the -- possibly page-locked -- detdata buffer)
            flags = torch.zeros((len(dets), ob.n_local_samples), dtype=torch.uint8, device=dev)
            if self.det_flags is not None:
                fd = ob.detdata[self.det_flags]
                flags |= ((_rows_to_device(fd, dets, dev) & self.det_flag_mask) != 0).to(
                    torch.uint8)
            if sflag is not None:
                sf = torch.from_numpy(np.ascontiguousarray(sflag)).to(dev)
                flags |= ((sf & self.shared_flag_mask) != 0).to(torch.uint8)[None, :]
            flags |= torch.from_numpy(
                np.ascontiguousarray(tmpl._obs_view_flags[iob]).astype(np.uint8)).to(dev)[None, :]
            noise = ob[binning.noise_model]
            d = DeviceObservation(
                focalplane=np.array([fp[x]["quat"] for x in dets]),
                boresight=ob.shared[dp.boresight], intervals=iv,
                det_scale=np.array([noise.detector_weight(x) for x in dets]),
                step_length=tmpl._step_length(tmpl.step_time, tmpl._obs_rate[iob]),
                n_pix_submap=pixels._n_pix_submap, n_submap=pixels._n_submap,
                global2local=np.zeros(pixels._n_submap, dtype=np.int64),
                epsilon=np.array([fp[x]["epsilon"] for x in dets]),
                gamma=np.array([fp[x]["gamma"] for x in dets]),
                cal=np.array([fp[x]["cal"] for x in dets]), IAU=weights.IAU,
                shared_flags=ob.shared[dp.shared_flags] if dp.shared_flags is not None else None,
                shared_flag_mask=dp.shared_flag_mask, solver_flags=flags, solver_flag_mask=1,
                hwp=ob.shared[weights.hwp_angle] if weights.hwp_angle is not None else None,
                amp_offsets=np.array([tmpl._obs_amp_offset(x, iob) for x in dets],
                                     dtype=np.int64),
                device=dev, **pixelisation)
            dobs.append(d)
            # the timestreams are not needed before the RHS: their upload (the largest transfer)
            # runs on its own stream, underneath the pointing expansion, the covariance and the
            # construction of the crossing lists
            with torch.cuda.stream(upload):
                sig = _rows_to_device(ob.detdata[self.det_data], dets, dev)
            sig.record_stream(main_stream)
            signals.append(sig)

        mark("upload + flags")
        # --- pointing expansion + pixel distribution --------------------------------------------
        hits = np.zeros(pixels._n_submap, dtype=np.uint8)
        for d in dobs:
            d.expand_pointing(hits)
            d.solver_flags |= (d.pixels < 0).to(torch.uint8)
        if comm.comm_world is not None:
            comm.allreduce_(hits, op="max")
        local = np.flatnonzero(hits).astype(np.int64)
        dist = PixelDistribution(pixels._n_pix, pixels._n_submap, local, comm=comm.comm_world)
        if is_wcs:
            dist.wcs = pixels.wcs
            dist.wcs_shape = tuple(pixels.wcs_shape)
        else:
            dist.nest = bool(pixels.nest)
        data[binning.pixel_dist] = dist
        for d in dobs:
            d.set_global2local(dist.global_submap_to_local)
        n_loc, nps = dist.n_local_submap, dist.n_pix_submap

        mark("pointing expansion")
        # --- CovarianceAndHits on the device (mapmaker_utils.py:1131-1270) ----------------------
        def allreduce_dev(t):
            if comm.comm_world is not None:
                torch.distributed.all_reduce(t)

        def covariance(threshold, want_hits):
            hmap = torch.zeros(n_loc * nps, dtype=torch.int64, device=dev) if want_hits else None
            inv = torch.zeros((n_loc, nps, 6), dtype=torch.float64, device=dev)
            for d in dobs:
                idx = np.arange(d.n_det, dtype=np.int32)
                KC.cov_accum(dist.global_submap_to_local, n_loc, nps, 3, hmap, inv, idx, d.pixels,
                             idx, d.weights, idx, d.solver_flags, d.det_scale, 1, d.intervals,
                             None, 0)
            if hmap is not None:
                allreduce_dev(hmap)
            allreduce_dev(inv)
            rc = torch.zeros(n_loc * nps, dtype=torch.float64, device=dev)
            KC.cov_invert(n_loc * nps, 3, inv, rc, float(threshold))
            return hmap, inv, rc

        hmap, cov, rcond = covariance(self.solve_rcond_threshold, True)
        # flags of the final products: the input flags only.  The solver's rcond mask (below) is
        # NOT part of them (ops/mapmaker.py:386-470, 502-594: the final covariance and maps are
        # made with the binning operator's own flags and map_rcond_threshold)
        base_flags = [d.solver_flags.clone() for d in dobs]

        # rcond mask -> solver flags (mapmaker_templates.py:895-939 via ScanMask)
        bad = torch.zeros((n_loc, nps, 3), dtype=torch.float64, device=dev)
        bad[:, :, 0] = (rcond.reshape(n_loc, nps) == 0).to(torch.float64)
        for d in dobs:
            idx = np.arange(d.n_det, dtype=np.int32)
            tmp = torch.zeros((d.n_det, d.n_samp), dtype=torch.float64, device=dev)
            # I weight may differ from 1 (cal): scan with unit weights on the first component
            w1 = torch.zeros((d.n_det, d.n_samp, 3), dtype=torch.float64, device=dev)
            w1[:, :, 0] = 1.0
            KC.ops_scan_map_float64(dist.global_submap_to_local, nps, bad, tmp, idx, d.pixels, idx,
                                    w1, idx, d.intervals, 1.0, True, False, False)
            d.solver_flags |= (tmp != 0).to(torch.uint8)
            del w1, tmp
        del bad

        mark("covariance + rcond mask")
        # --- amplitude flags / preconditioner: n_good = F^T (good-sample indicator) -------------
        n_amp = tmpl._n_local
        n_good = torch.zeros(n_amp, dtype=torch.float64, device=dev)
        zero_flags = torch.zeros(n_amp, dtype=torch.uint8, device=dev)
        amplen = torch.zeros(n_amp, dtype=torch.float64, device=dev)
        detnoise = torch.ones(n_amp, dtype=torch.float64, device=dev)
        for d in dobs:
            idx = np.arange(d.n_det, dtype=np.int32)
            ones = torch.ones((d.n_det, d.n_samp), dtype=torch.float64, device=dev)
            KC.template_offset_project_signal_batch(idx, ones, idx, d.solver_flags, 1,
                                                    d.step_length, d.amp_offsets, d.n_amp_views,
                                                    n_good, zero_flags, d.intervals)
            del ones
            lens = np.concatenate([
                np.minimum(d.step_length,
                           int(v["last"] - v["first"]) - d.step_length * np.arange(na))
                for v, na in zip(d.intervals, d.n_amp_views)])
            _fill_amp_layout(amplen, detnoise, d.amp_offsets, d.n_amp_det, lens, d.det_scale)
        # (element-wise on the device: the vectors hold millions of baselines)
        flagged, offset_var = _amp_flags_and_variance(n_good, amplen, detnoise,
                                                      float(tmpl.good_fraction))
        amp_flags = flagged.to(torch.uint8)
        tmpl._offsetvar = offset_var.cpu().numpy()
        tmpl._amp_flags = flagged.cpu().numpy()
        del amplen, detnoise, n_good

        mark("amplitude flags")
        # --- RHS, PCG ----------------------------------------------------------------------------
        if tmpl.use_noise_prior:
            tmpl._build_prior(data)  # offset.py:356-560, uploaded once
        ds = Destriper(dobs, n_loc, nps, cov, offset_var, amp_flags,
                       regen=self.regenerate_pointing, device=dev, prior=tmpl.prior())
        main_stream.wait_stream(upload)   # the timestreams have arrived
        mark("crossing lists + solver set-up")
        rhs = ds.rhs(signals)
        mark("RHS")
        amps_dev, self.history = ds.solve(rhs, convergence=self.convergence,
                                          n_iter_max=self.iter_max, n_iter_min=self.iter_min)

        mark("PCG")
        # --- final products -------------------------------------------------------------------------
        for d, bf in zip(dobs, base_flags):
            d.solver_flags.copy_(bf)   # (same buffer the native handle points at)
        del base_flags
        if self.map_rcond_threshold != self.solve_rcond_threshold:
            _, cov_map, rcond_map = covariance(self.map_rcond_threshold, False)
            ds.cov = cov_map
        else:
            rcond_map = rcond  # (the solve covariance was accumulated with the same flags)
        binmap = ds.bin_signal(signals).clone()
        neg = -amps_dev
        for d, sig in zip(dobs, signals):
            idx = np.arange(d.n_det, dtype=np.int32)
            KC.template_offset_add_to_signal_batch(d.step_length, d.amp_offsets, d.n_amp_views,
                                                   neg, ds.amp_flags, idx, sig, d.intervals)
        destriped = ds.bin_signal(signals).clone()

        mark("final binning")

        def to_pixdata(t, dtype, nv):
            return _pixdata_from_device(dist, t, dtype, nv)

        data[f"{self.name}_hits"] = to_pixdata(hmap, np.int64, 1)
        data[f"{self.name}_cov"] = to_pixdata(ds.cov, np.float64, 6)
        data[f"{self.name}_rcond"] = to_pixdata(rcond_map, np.float64, 1)
        data[f"{self.name}_binmap"] = to_pixdata(binmap, np.float64, 3)
        data[f"{self.name}_map"] = to_pixdata(destriped, np.float64, 3)
        amps = AmplitudesMap()
        amps[tmpl.name] = tmpl.zeros()
        amps[tmpl.name].local[:] = amps_dev.cpu().numpy()
        data[self.template_matrix.amplitudes] = amps
        # the cleaned timestream is what the reference leaves in det_data (mapmaker.py:531-574)
        for iob, (ob, d, sig) in enumerate(zip(data.obs, dobs, signals)):
            dets = [x for x in tmpl._all_dets if x in tmpl._obs_dets[iob]]
            _rows_from_device(ob.detdata[self.det_data], dets, sig)
        mark("products to host")
        if self.keep_solver_products:
            self.destriper = ds

    def _requires(self):
        return {"detdata": [self.det_data]}

    def _provides(self):
        return {"global": [f"{self.name}_map", f"{self.name}_binmap", f"{self.name}_hits"]}
