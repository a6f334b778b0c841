"""TEST INFRASTRUCTURE ONLY -- never imported by toast_b200.

CPU stand-ins of ``tests/fake_device.py`` that also take DeviceObservation's ``nnz``, so that
``ops.MapMaker`` with ``StokesWeights(mode="I")`` (intensity-only maps: DeviceObservation(nnz=1),
one value per pixel) runs its host logic in the CPU suite with the oracle doing the per-sample
compute.  ``install_intensity(monkeypatch)`` is ``fake_device.install`` with these stand-ins.
"""

import numpy as np
import torch

import fake_device
from fake_device import FakeDestriper, FakeDeviceObservation, _covapply, _np
from oracle import toast_oracle as O

class IntensityMixin:
    """DeviceObservation's ``nnz`` on a stand-in observation class: with nnz = 1 the weights are
    StokesWeights(mode="I")'s, [n_det, n_samp] = cal[det] (the oracle's stokes_weights_I)."""

    def __init__(self, *, nnz=3, **kw):
        super().__init__(**kw)
        self.nnz = int(nnz)

    def expand_pointing(self, hit_submaps=None):
        super().expand_pointing(hit_submaps)
        if self.nnz == 1:
            w = np.zeros((self.n_det, self.n_samp))
            O.stokes_weights_I(np.arange(self.n_det, dtype=np.int32), w, self.intervals,
                               self.cal, False)
            self.weights = torch.from_numpy(w)


class FakeIntensityDeviceObservation(IntensityMixin, FakeDeviceObservation):
    pass


class FakeIntensityDestriper(FakeDestriper):
    """FakeDestriper on maps of the observations' nnz (3 or 1) values per pixel."""

    def __init__(self, observations, *args, **kw):
        super().__init__(observations, *args, **kw)
        nnzs = {getattr(o, "nnz", 3) for o in self.obs} or {3}
        if len(nnzs) != 1:
            raise ValueError("the observations of one Destriper must all have the same nnz")
        self.nnz = nnzs.pop()

    def _pb(self, d):
        ncov = self.nnz * (self.nnz + 1) // 2
        return O.Problem(
            n_det=d.n_det, n_samp=d.n_samp, step_length=d.step_length, det_start=d.amp_offsets,
            n_amp_views=d.n_amp_views, n_amp=self.n_amp, amp_flags=_np(self.amp_flags),
            offset_var=_np(self.offset_var), intervals=d.intervals,
            solver_flags=_np(d.solver_flags), det_flag_mask=d.solver_flag_mask,
            det_scale=d.det_scale, global2local=d.global2local, pixels=_np(d.pixels),
            weights=_np(d.weights), shared_flags=np.zeros(1, dtype=np.uint8), shared_flag_mask=0,
            n_local_submap=self.n_local_submap, n_pix_submap=self.n_pix_submap,
            cov=_np(self.cov).reshape(self.n_local_submap, self.n_pix_submap, ncov), nnz=self.nnz)

    def _bin(self, pbs, timestreams):
        z = np.zeros((self.n_local_submap, self.n_pix_submap, self.nnz))
        for pb, tod in zip(pbs, timestreams):
            idx = np.arange(pb.n_det, dtype=np.int32)
            O.build_noise_weighted(pb.global2local, z, idx, pb.pixels, idx, pb.weights, idx, tod,
                                   idx, pb.solver_flags, pb.det_scale, pb.det_flag_mask,
                                   pb.intervals, pb.shared_flags, pb.shared_flag_mask, False)
        _covapply(self.n_local_submap, self.n_pix_submap, self.nnz, pbs[0].cov.reshape(-1),
                  z.reshape(-1))
        return z


def install_intensity(monkeypatch, observation_class=FakeIntensityDeviceObservation):
    """``install`` with stand-ins that take DeviceObservation's ``nnz``: ops.MapMaker with
    StokesWeights(mode="I") runs through them."""
    import toast_b200.solver as SV

    fake_device.install(monkeypatch)
    monkeypatch.setattr(SV, "DeviceObservation", observation_class)
    monkeypatch.setattr(SV, "Destriper", FakeIntensityDestriper)
