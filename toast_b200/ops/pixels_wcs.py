"""PixelsWCS (``ops/pixels_wcs.py:39-662``): detector pixel indices on a flat projection.

The reference runs this operator on the host (qa_to_iso + astropy ``wcs_world2pix`` per detector
and view); here the per-sample work is one CUDA launch per observation (``tb_pixels_wcs``,
csrc/tb_wcs.cuh) and the projection set-up is ``toast_b200.wcs.create_wcs``.  Trait names and
their meaning follow the reference; angles are plain floats in DEGREES where the reference takes
astropy Quantities (astropy is not a dependency of this package).

Not implemented (raises): ``fits_header`` (needs a FITS reader), ``center_offset`` (moving
centre), ``single_precision``.
"""

import numpy as np

from .. import kernels as K
from .. import wcs as W
from ..pixels import PixelDistribution
from .operator import Operator
from .pointing import _view_intervals


def _unwrap_together(x, y, period=360.0):
    """pixels_wcs.py:26-35."""
    for i in range(1, len(x)):
        while abs(x[i] - x[i - 1]) > abs(x[i] + period - x[i - 1]):
            x[i] += period
            y[i] += period
        while abs(x[i] - x[i - 1]) > abs(x[i] - period - x[i - 1]):
            x[i] -= period
            y[i] -= period


def scan_range_lonlat_deg(boresight, flags, flag_mask, fov_deg, is_azimuth):
    """pointing_utils.py:70-190 (no moving centre): extent of a ring of 64 fake detectors at the
    field-of-view radius around the unflagged boresight samples, in degrees."""
    from ..synthetic import q_mult, q_rotation, YAXIS, ZAXIS

    bore = np.asarray(boresight)
    if flags is not None:
        bore = bore[(np.asarray(flags) & flag_mask) == 0]
    radius = 0.5 * np.radians(fov_deg)
    # pointing_utils.py:121-130: the top of the focalplane must stay below the pole
    nb = bore / np.sqrt(np.sum(bore * bore, axis=-1, keepdims=True))
    el_max = float(np.max(np.arcsin(np.clip(1 - 2 * (nb[:, 0] ** 2 + nb[:, 1] ** 2), -1, 1))))
    if el_max + radius > np.pi / 2:
        raise RuntimeError(
            "The scan range includes the zenith."
            f" Max boresight elevation is {np.degrees(el_max)} deg"
            f" and focalplane radius is {np.degrees(radius)} deg."
            " Scan range facility cannot handle this case.")
    lon_all, lat_all = [], []
    thetarot = q_rotation(YAXIS, radius)
    for phi in np.linspace(0, 2 * np.pi, 64, endpoint=False):
        dq = q_mult(bore, q_mult(q_rotation(ZAXIS, phi), thetarot)[None, :])
        nrm = dq / np.sqrt(np.sum(dq * dq, axis=-1, keepdims=True))
        x, y, z, w = nrm[:, 0], nrm[:, 1], nrm[:, 2], nrm[:, 3]
        dx, dy, dz = 2 * (w * y + x * z), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y)
        lon = np.arctan2(dy, dx)
        if is_azimuth:
            lon = 2 * np.pi - lon
        lon = np.where(lon >= 2 * np.pi, lon - 2 * np.pi, lon)
        lon = np.where(lon < 0, lon + 2 * np.pi, lon)
        lon_all.append(lon)
        lat_all.append(np.arcsin(np.clip(dz, -1, 1)))
    lon = np.unwrap(np.hstack(lon_all))
    lat = np.hstack(lat_all)
    return (np.degrees(lon.min()), np.degrees(lon.max()), np.degrees(lat.min()),
            np.degrees(lat.max()))


class PixelsWCS(Operator):
    _defaults = dict(detector_pointing=None, fits_header=None, coord_frame="EQU",
                     projection="CAR", center=(), center_offset=None, bounds=(),
                     auto_bounds=True, dimensions=(1000, 1000), resolution=(), view=None,
                     pixels="pixels", submaps=1, create_dist=None, single_precision=False,
                     use_astropy=True, field_of_view=None)

    @staticmethod
    def create_wcs(coord="EQU", proj="CAR", center_deg=None, bounds_deg=None, res_deg=None,
                   dims=None):
        return W.create_wcs(coord, proj, center_deg, bounds_deg, res_deg, dims)

    def set_wcs(self):
        """pixels_wcs.py:347-389."""
        if self.projection not in W.PROJECTIONS:
            raise ValueError("Invalid WCS projection name")
        center_deg = tuple(float(x) for x in self.center) if len(self.center) > 0 else None
        bounds_deg = tuple(float(x) for x in self.bounds) if len(self.bounds) > 0 else None
        res_deg = tuple(float(x) for x in self.resolution) if len(self.resolution) > 0 else None
        dims = tuple(self.dimensions) if len(self.dimensions) > 0 else None
        self.wcs, self.wcs_shape = W.create_wcs(self.coord_frame, self.projection, center_deg,
                                                bounds_deg, res_deg, dims)
        self.n_row, self.n_col = self.wcs_shape
        if self.n_row < 1 or self.n_col < 1:
            raise RuntimeError(f"The WCS has non-positive dimensions: {self.wcs_shape}")
        self._n_pix = self.n_row * self.n_col
        self._n_submap = self.submaps
        self._n_pix_submap = self._n_pix // self.submaps
        if self._n_pix_submap * self.submaps < self._n_pix:
            self._n_pix_submap += 1
        self._local_submaps = np.zeros(self.submaps, dtype=np.uint8)

    def _geometry(self, data):
        """The projection of this operator for ``data``: with ``auto_bounds``, the bounds of the
        boresights of every observation plus the field of view (pixels_wcs.py:436-489), then
        ``set_wcs``.  Sets ``wcs``, ``wcs_shape`` and the pixel / submap counts; ops.MapMaker
        calls it too."""
        if self.detector_pointing is None:
            raise RuntimeError("The detector_pointing trait must be set")
        for trait in ("fits_header", "center_offset"):
            if getattr(self, trait) is not None:
                raise NotImplementedError(f"PixelsWCS: '{trait}' is not implemented on this path")
        if self.single_precision:
            raise NotImplementedError("single_precision pixels are not implemented")
        dp = self.detector_pointing
        is_azimuth = self.coord_frame == "AZEL"
        if self.auto_bounds:
            # pixels_wcs.py:436-489
            if self.field_of_view is None:
                raise RuntimeError("auto_bounds needs the field_of_view trait (degrees)")
            mm = np.array([scan_range_lonlat_deg(
                ob.shared[dp.boresight],
                ob.shared[dp.shared_flags] if dp.shared_flags is not None else None,
                dp.shared_flag_mask, self.field_of_view, is_azimuth) for ob in data.obs]).T
            _unwrap_together(mm[0], mm[1])
            # (the reference takes amin of the per-observation lon_max values: reproduced)
            self.bounds = (float(mm[0].min()), float(mm[1].min()), float(mm[2].min()),
                           float(mm[3].max()))
            self.center = ()
            if len(self.resolution) > 0:
                self.dimensions = ()
            self.auto_bounds = False
        self.set_wcs()

    def _exec(self, data, detectors=None, use_accel=False, **kwargs):
        self._geometry(data)
        dp = self.detector_pointing
        view = self.view if self.view is not None else dp.view
        dp.apply(data, detectors=detectors, use_accel=use_accel)
        for ob in data.obs:
            dets = ob.select_local_detectors(detectors, flagmask=dp.det_mask)
            if len(dets) == 0:
                continue
            alld = ob.select_local_detectors(None, flagmask=dp.det_mask)
            exists = ob.detdata.ensure(self.pixels, sample_shape=(), dtype=np.int64,
                                       detectors=alld, accel=use_accel)
            done = self.__dict__.setdefault("_done", {})
            if exists and done.get((id(ob), tuple(dets))):
                if self.create_dist is not None:   # pixels_wcs.py:536-551
                    for d in dets:
                        for iv in _view_intervals(ob, view):
                            p = ob.detdata[self.pixels][d, iv["first"]:iv["last"]]
                            self._local_submaps[p[p >= 0] // self._n_pix_submap] = 1
                continue
            flags = ob.shared[dp.shared_flags] if dp.shared_flags is not None else \
                np.zeros(1, dtype=np.uint8)
            tmp = np.zeros(self.submaps, dtype=np.uint8)
            K.pixels_wcs(self.wcs, ob.detdata[dp.quats].indices(dets), ob.detdata[dp.quats].data,
                         flags, dp.shared_flag_mask, ob.detdata[self.pixels].indices(dets),
                         ob.detdata[self.pixels].data, _view_intervals(ob, view), tmp,
                         self._n_pix_submap, use_accel)
            if self.create_dist is not None:
                self._local_submaps |= tmp
            done[(id(ob), tuple(dets))] = True

    def _finalize(self, data, use_accel=False, **kwargs):
        if self.create_dist is not None:
            submaps = np.arange(self.submaps, dtype=np.int64)[self._local_submaps == 1]
            dist = PixelDistribution(n_pix=self._n_pix, n_submap=self.submaps,
                                     local_submaps=submaps, comm=data.comm.comm_world)
            dist.wcs = self.wcs
            dist.wcs_shape = tuple(self.wcs_shape)
            data[self.create_dist] = dist
            self._local_submaps[:] = 0

    def _requires(self):
        return self.detector_pointing.requires()

    def _provides(self):
        prov = {"detdata": [self.pixels, self.detector_pointing.quats]}
        if self.create_dist is not None:
            prov["global"] = [self.create_dist]
        return prov
