"""Device-resident destriping solver: the fused form of the reference's
``SolverRHS`` / ``SolverLHS`` / ``solve()`` (``ops/mapmaker_solve.py:107-229, 342-506, 524-755``)
for the ``templates.Offset`` template.

Everything an iteration touches stays in HBM: expanded pointing (or just the boresight when
``regen=True``), solver flags, the noise-weighted map, the pixel covariance and the five
amplitude vectors of the PCG.  One iteration is

    zmap = 0;  pass 1 per observation            (tb_lhs_pass1)
    all-reduce zmap over ranks (NCCL)            -- the reference's PixelData.sync_allreduce
    binned = cov * zmap                          (tb_cov_apply_diag)
    q = 0;  pass 2 per observation               (tb_lhs_pass2)
    d.q -> alpha;  x, r, s updates;  r.r, s.r    (tb_amp_dot, tb_pcg_update)
    d = s + beta d                               (tb_pcg_direction)

with the scalars left on the device; the host reads back one float per iteration (the relative
residual, which the reference logs at ``mapmaker_solve.py:701-706``) to test convergence.

torch is used for device allocations and ``torch.distributed`` for the collectives only.
"""

import ctypes as ct

import numpy as np
import torch

from . import lib as L
from . import kernels as K


def _dev_tensor(a, device, dtype=None):
    if a is None:
        return None
    if isinstance(a, torch.Tensor):
        t = a.to(device=device)
    else:
        t = torch.from_numpy(np.ascontiguousarray(a)).to(device)
    if dtype is not None:
        t = t.to(dtype)
    return t.contiguous()


class DeviceObservation:
    """One observation resident on the device, in the reference's buffer layouts
    (``detdata`` [n_det, n_samp, ...], ``shared`` [n_samp, ...]) plus the Offset amplitude
    layout (``templates/offset/offset.py:245-253``: detector-major, ceil(len/step) per view).

    The pixelisation is HEALPix (``nside`` / ``nest``) or a flat projection (``wcs``, a
    ``toast_b200.wcs.FlatWCS`` with its shape set), one or the other."""

    def __init__(self, *, focalplane, boresight, intervals, det_scale, step_length, n_pix_submap,
                 n_submap, global2local, nside=None, nest=None, wcs=None, amp_offset=0,
                 epsilon=None, gamma=None, cal=None, IAU=False, shared_flags=None,
                 shared_flag_mask=0, solver_flags=None, solver_flag_mask=255, pixels=None,
                 weights=None, hwp=None, amp_offsets=None, compact=True, device="cuda"):
        if wcs is not None and (nside is not None or nest is not None):
            raise ValueError("DeviceObservation takes either wcs or nside / nest, not both")
        if wcs is None and (nside is None or nest is None):
            raise ValueError("DeviceObservation needs nside and nest, or wcs")
        self.device = torch.device(device)
        self.lib = L.load()
        self.n_det = int(focalplane.shape[0])
        self.n_samp = int(boresight.shape[0])
        self.intervals = np.ascontiguousarray(intervals)
        self.step_length = int(step_length)
        self.focalplane = np.ascontiguousarray(focalplane, dtype=np.float64)
        self.epsilon = np.zeros(self.n_det) if epsilon is None else np.ascontiguousarray(epsilon)
        self.gamma = np.zeros(self.n_det) if gamma is None else np.ascontiguousarray(gamma)
        self.cal = np.ones(self.n_det) if cal is None else np.ascontiguousarray(cal)
        self.det_scale = np.ascontiguousarray(det_scale, dtype=np.float64)
        self.wcs = wcs
        self.nside = None if wcs is not None else int(nside)
        self.nest = None if wcs is not None else bool(nest)
        self.IAU = bool(IAU)
        self.n_pix_submap, self.n_submap = int(n_pix_submap), int(n_submap)
        self.global2local = np.ascontiguousarray(global2local, dtype=np.int64)
        self.shared_flag_mask = int(shared_flag_mask)
        self.solver_flag_mask = int(solver_flag_mask)
        # keep a compact (20 B/sample) copy of the stored pointing for the LHS passes
        self.compact = bool(compact)

        # Offset amplitude layout
        nav = []
        for iv in self.intervals:
            ln = int(iv["last"] - iv["first"])
            n = ln // self.step_length
            if n * self.step_length < ln:
                n += 1
            nav.append(n)
        self.n_amp_views = np.array(nav, dtype=np.int64)
        self.n_amp_det = int(self.n_amp_views.sum())
        if amp_offsets is not None:
            self.amp_offsets = np.ascontiguousarray(amp_offsets, dtype=np.int64)
        else:
            self.amp_offsets = amp_offset + np.arange(self.n_det, dtype=np.int64) * self.n_amp_det
        self.n_amp = self.n_amp_det * self.n_det

        dev = self.device
        self.boresight = _dev_tensor(boresight, dev, torch.float64)
        self.shared_flags = _dev_tensor(shared_flags, dev, torch.uint8)
        self.solver_flags = _dev_tensor(solver_flags, dev, torch.uint8)
        self.pixels = _dev_tensor(pixels, dev, torch.int64)
        self.weights = _dev_tensor(weights, dev, torch.float64)
        self.hwp = _dev_tensor(hwp, dev, torch.float64)
        self._handle = None

    # -- pointing -----------------------------------------------------------------------------
    def expand_pointing(self, hit_submaps=None):
        """PointingDetectorSimple -> PixelsHealpix (or PixelsWCS) -> StokesWeights in one fused
        kernel; fills ``pixels`` / ``weights`` on the device and ORs the hit-submap mask (host
        uint8)."""
        dev = self.device
        if self.pixels is None:
            self.pixels = torch.zeros((self.n_det, self.n_samp), dtype=torch.int64, device=dev)
        if self.weights is None:
            self.weights = torch.zeros((self.n_det, self.n_samp, 3), dtype=torch.float64,
                                       device=dev)
        idx = np.arange(self.n_det, dtype=np.int32)
        if self.wcs is not None:
            K.pointing_fused_wcs(self.wcs, self.focalplane, self.boresight, self.shared_flags,
                                 self.shared_flag_mask, None, None, idx, self.pixels, idx,
                                 self.weights, self.hwp, self.intervals, hit_submaps,
                                 self.n_pix_submap, self.epsilon, self.gamma, self.cal, self.IAU)
        else:
            K.pointing_fused(self.focalplane, self.boresight, self.shared_flags,
                             self.shared_flag_mask, None, None, idx, self.pixels, idx,
                             self.weights, self.hwp, self.intervals, hit_submaps,
                             self.n_pix_submap, self.nside, self.nest, self.epsilon, self.gamma,
                             self.cal, self.IAU)
        self._handle = None

    def set_global2local(self, g2l):
        self.global2local = np.ascontiguousarray(g2l, dtype=np.int64)
        self._handle = None

    def invalidate(self):
        """Call after changing flags / pointing in place: the native handle (and its compact
        copy of the pointing) is rebuilt on next use."""
        self._handle = None

    # -- native handle ------------------------------------------------------------------------
    def handle(self):
        if self._handle is not None:
            return self._handle
        d = L.tb_obs_desc()
        d.n_det, d.n_samp, d.n_view = self.n_det, self.n_samp, len(self.intervals)
        self._keep = [self.intervals, self.focalplane, self.epsilon, self.gamma, self.cal,
                      self.det_scale, self.amp_offsets, self.n_amp_views, self.global2local]
        d.intervals = self.intervals.ctypes.data
        d.focalplane = self.focalplane.ctypes.data
        d.epsilon = self.epsilon.ctypes.data
        d.gamma = self.gamma.ctypes.data
        d.cal = self.cal.ctypes.data
        d.det_scale = self.det_scale.ctypes.data
        d.amp_offsets = self.amp_offsets.ctypes.data
        d.n_amp_views = self.n_amp_views.ctypes.data
        d.step_length = self.step_length
        d.nside = 0 if self.wcs is not None else self.nside
        d.n_pix_submap, d.n_submap = self.n_pix_submap, self.n_submap
        d.nest, d.IAU = int(bool(self.nest)), int(self.IAU)
        d.global2local = self.global2local.ctypes.data
        d.boresight = L.ptr(self.boresight)
        d.shared_flags = L.ptr(self.shared_flags)
        d.shared_flag_mask = self.shared_flag_mask
        d.solver_flags = L.ptr(self.solver_flags)
        d.solver_flag_mask = self.solver_flag_mask
        d.pixels = L.ptr(self.pixels)
        d.weights = L.ptr(self.weights)
        d.hwp = L.ptr(self.hwp)
        if self.wcs is not None:
            self._wcs_desc = self.wcs.desc()
            h = self.lib.tb_obs_create_wcs(ct.byref(d), ct.byref(self._wcs_desc))
        else:
            h = self.lib.tb_obs_create(ct.byref(d))
        if not h:
            raise RuntimeError(L.last_error())
        self._handle = _ObsHandle(self.lib, h)
        if self.compact and self.pixels is not None and self.weights is not None:
            L.check(self.lib.tb_obs_pack_pointing(h, None))
        return self._handle

    def has_compact_pointing(self):
        return bool(self.lib.tb_obs_has_compact_pointing(self.handle().h))

    def bytes_per_sample_stored(self):
        return 8 + 24 + (1 if self.solver_flags is not None else 0)


class _ObsHandle:
    def __init__(self, lib, h):
        self.lib, self.h = lib, h

    def __del__(self):
        try:
            self.lib.tb_obs_destroy(self.h)
        except Exception:
            pass


class _CudaView:
    """Expose a raw device allocation to torch through __cuda_array_interface__."""

    def __init__(self, ptr, n, typestr="<f8"):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr,
                                         "data": (int(ptr), False), "version": 2}


def _all_ranks_ok(ok, device, group=None):
    """True only if ``ok`` holds on EVERY rank (MIN all-reduce of a success flag): each rank must
    take the same decision about the reduction path, or the ranks on the fused path would spin in
    its device-side flag barrier while the others sit in an NCCL collective."""
    import torch.distributed as dist

    t = torch.tensor([1 if ok else 0], dtype=torch.int32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    return bool(int(t.item()) == 1)


class PeerMap:
    """A map buffer visible to every rank of the node over NVLink (CUDA IPC) and the fused
    reduce-scatter -> covariance -> all-gather kernel on it (``tb_map_reduce_cov``).  Replaces
    ``PixelData.sync_allreduce`` + ``covariance_apply`` of the reference."""

    def __init__(self, n_pix, device, group=None):
        import torch.distributed as dist

        self.lib = L.load()
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.n_pix = int(n_pix)
        nbytes = self.n_pix * 3 * 8
        self.h = self.lib.tb_peer_create(self.rank, self.world, nbytes)
        buf = ct.create_string_buffer(128)
        ok = bool(self.h) and self.lib.tb_peer_get_handles(self.h, buf) == 0
        err = "" if ok else L.last_error()
        if not _all_ranks_ok(ok, device, group):   # every rank gives up together
            self._release()
            raise RuntimeError(err or "peer-memory allocation failed on another rank")
        handles = [None] * self.world
        dist.all_gather_object(handles, buf.raw, group=group)
        ok = self.lib.tb_peer_open(self.h, b"".join(handles)) == 0
        err = "" if ok else L.last_error()
        if not _all_ranks_ok(ok, device, group):
            self._release()
            raise RuntimeError(err or "opening the peer handles failed on another rank")
        ptr = self.lib.tb_peer_map_ptr(self.h)
        self.tensor = torch.as_tensor(_CudaView(ptr, self.n_pix * 3), device=device)
        dist.barrier(group=group)

    def reduce_cov(self, cov, pix_first=0, n_pix=None, stream=None):
        n_pix = self.n_pix - pix_first if n_pix is None else n_pix
        L.check(self.lib.tb_map_reduce_cov_range(self.h, pix_first, n_pix, L.ptr(cov), stream))

    def _release(self):
        if getattr(self, "h", None):
            self.lib.tb_peer_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass


class SymmPeerMap:
    """The same fused map reduction on SYMMETRIC memory with an NVLS multicast mapping
    (``torch.distributed._symmetric_memory`` is the plumbing that allocates the buffer on every
    rank, exchanges the handles and binds the multicast object): ``tb_map_reduce_cov`` then lets
    the NVSwitch form the sums (``multimem.ld_reduce``) and replicate the result
    (``multimem.st``), see tb_peer.cu."""

    def __init__(self, n_pix, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem

        self.lib = L.load()
        grp = group if group is not None else dist.group.WORLD
        self.rank = dist.get_rank(grp)
        self.world = dist.get_world_size(grp)
        self.n_pix = int(n_pix)
        n = self.n_pix * 3
        self.buf = symm_mem.empty(n + 64, dtype=torch.float64, device=device)  # tail: flags
        self.buf.zero_()
        hdl = symm_mem.rendezvous(self.buf, grp)
        mc = int(getattr(hdl, "multicast_ptr", 0) or 0)
        maps = (ct.c_uint64 * self.world)(*[int(p) for p in hdl.buffer_ptrs])
        flags = (ct.c_uint64 * self.world)(*[int(p) + n * 8 for p in hdl.buffer_ptrs])
        self._hdl = hdl
        self.h = self.lib.tb_peer_attach(self.rank, self.world, n * 8, maps, flags, mc) \
            if mc != 0 else None
        err = "" if self.h else ("no NVLS multicast mapping for symmetric memory on this system"
                                 if mc == 0 else L.last_error())
        if not _all_ranks_ok(bool(self.h), device, group):   # every rank gives up together
            if self.h:
                self.lib.tb_peer_destroy(self.h)
                self.h = None
            raise RuntimeError(err or "symmetric-memory set-up failed on another rank")
        self.tensor = self.buf[:n]
        self.group = group
        self.use_multimem = True
        torch.cuda.synchronize(device)
        dist.barrier(group=group)

    def reduce_cov(self, cov, pix_first=0, n_pix=None, stream=None):
        n_pix = self.n_pix - pix_first if n_pix is None else n_pix
        L.check(self.lib.tb_peer_set_multimem(1 if self.use_multimem else 0))
        L.check(self.lib.tb_map_reduce_cov_range(self.h, pix_first, n_pix, L.ptr(cov), stream))

    def tune(self, cov, reps=3):
        """Measure the in-switch (multimem) and the P2P form of the kernel on this node and map
        size and keep the faster one (max over ranks, so every rank takes the same decision):
        in-switch reduction moves ~|map| per NVLink direction for any N, P2P 2(N-1)/N x |map|/2,
        so which one wins depends on N."""
        import torch.distributed as dist

        saved = self.tensor.clone()
        times = []
        for mode in (True, False):
            self.use_multimem = mode
            self.reduce_cov(cov)  # warm-up
            dist.barrier(group=self.group)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                self.reduce_cov(cov)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / reps)
        t = torch.tensor(times, dtype=torch.float64, device=self.tensor.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        self.tune_ms = {"multimem": float(t[0]), "p2p": float(t[1])}
        self.use_multimem = bool(t[0] <= t[1])
        self.tensor.copy_(saved)
        torch.cuda.synchronize()
        dist.barrier(group=self.group)
        return self.tune_ms

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.tb_peer_destroy(self.h)
        except Exception:
            pass


def pipeline_chunk_bounds(n_pix, world, n_chunks, align=1):
    """Local-pixel bounds of the chunks the multi-GPU pipeline works in: every chunk but the last
    is a multiple of 256 x world pixels (the reduction kernel's tile x one slice per rank) and of
    ``align`` (the pixel block of the block-ordered passes), the last one takes the remainder.
    None when fewer than two chunks are possible."""
    unit = int(np.lcm(256 * world, max(1, int(align))))
    units = n_pix // unit
    n_chunks = max(1, min(int(n_chunks), units))
    if n_chunks < 2:
        return None
    bounds = np.array([(c * units) // n_chunks * unit for c in range(n_chunks + 1)],
                      dtype=np.int64)
    bounds[-1] = n_pix
    return bounds


class Destriper:
    """Fused SolverRHS / SolverLHS / solve() for one or more device observations.

    ``cov`` is the inverse-of-inverse pixel covariance [n_local_submap, n_pix_submap, 6]
    (upper triangle, row-major) as produced by ``covariance_invert``; ``regen=True``
    recomputes pointing inside every pass instead of reading stored pixels/weights."""

    def __init__(self, observations, n_local_submap, n_pix_submap, cov, offset_var, amp_flags,
                 regen=False, group=None, device="cuda", fused_reduce=True, prior=None):
        self.obs = list(observations)
        # templates.offset_prior.OffsetPrior or None: with a noise prior the LHS gains the
        # inverse amplitude covariance (offset.py:884-960) and the preconditioner becomes the
        # banded / Toeplitz solve (offset.py:962-1010)
        self.prior = prior
        self.device = torch.device(device)
        self.lib = L.load()
        self.regen = 1 if regen else 0
        self.group = group
        self.n_local_submap, self.n_pix_submap = int(n_local_submap), int(n_pix_submap)
        self.cov = _dev_tensor(cov, self.device, torch.float64)
        self.offset_var = _dev_tensor(offset_var, self.device, torch.float64)
        self.amp_flags = _dev_tensor(amp_flags, self.device, torch.uint8)
        self.n_amp = int(self.offset_var.numel())
        assert sum(o.n_amp for o in self.obs) == self.n_amp
        self.world = 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size(group)
        # Multi-GPU: keep the map in NVLink-peer-visible memory and reduce it with the fused
        # kernel; fall back to NCCL all-reduce + cov_apply if peer memory cannot be set up.
        self.peer = None
        n_pix = self.n_local_submap * self.n_pix_submap
        import os as _os
        # the fused reduction works in 256-pixel tiles: maps that are not a multiple of that
        # (nside_submap < 8 gives 12 / 48 / 192 pixels per submap) take the NCCL path
        aligned = n_pix % 256 == 0
        if self.world > 1 and fused_reduce and aligned and \
                _os.environ.get("TB_FUSED_REDUCE", "1") != "0":
            import warnings

            # every attempt ends with an agreement over the ranks (inside the constructors and
            # below): either all ranks use a path or none does
            if _os.environ.get("TB_MULTIMEM", "1") != "0":
                peer, err = None, None
                try:
                    peer = SymmPeerMap(n_pix, self.device, group)
                except Exception as exc:  # noqa: BLE001
                    err = exc
                if _all_ranks_ok(peer is not None, self.device, group):
                    try:
                        peer.tune(self.cov)
                    except Exception as exc:  # noqa: BLE001
                        err = exc
                    if _all_ranks_ok(err is None, self.device, group):
                        self.peer = peer
                if self.peer is None:
                    warnings.warn(f"NVLS multicast map reduction unavailable ({err}); "
                                  "using P2P peer memory")
            if self.peer is None:
                peer, err = None, None
                try:
                    peer = PeerMap(n_pix, self.device, group)
                except Exception as exc:  # noqa: BLE001
                    err = exc
                if _all_ranks_ok(peer is not None, self.device, group):
                    self.peer = peer
                else:
                    warnings.warn(f"peer-memory map reduction unavailable ({err}); using NCCL")
        if self.peer is not None:
            self.zmap = self.peer.tensor.view(self.n_local_submap, self.n_pix_submap, 3)
        else:
            self.zmap = torch.zeros((self.n_local_submap, self.n_pix_submap, 3),
                                    dtype=torch.float64, device=self.device)
        # Chunk pipeline (multi-GPU): TB_PIPE_CHUNKS = "auto" (default: set it up with 4 chunks,
        # time it against the serial LHS on this node and keep the faster form), 0 (off) or K.
        # Measured on 2 GPUs: 1.46-1.54 ms against 1.69 ms per iteration with 4 chunks, slower
        # than serial with 8-16 (DESIGN.md section 5).
        # one observation on one GPU: pass 1 -> covariance -> pass 2 inside one kernel
        self.fuse_lhs = _os.environ.get("TB_FUSE_LHS", "1") != "0"
        self.pipeline = False
        self.blocked = False
        self.pipe_tune_ms = None
        self._ctas_set = None
        mode = _os.environ.get("TB_PIPE_CHUNKS", "auto")
        if mode == "auto":
            self._setup_pipeline(4)
            if self.world > 1 and not _all_ranks_ok(self.pipeline, self.device, group):
                self.pipeline = False
            if self.pipeline:
                self._tune_pipeline()
        else:
            self._setup_pipeline(int(mode))
            if self.world > 1 and not _all_ranks_ok(self.pipeline, self.device, group):
                self.pipeline = False

    # -- chunk pipeline -------------------------------------------------------------------------
    def _blocked(self):
        """True when the passes of every observation run on the block-ordered crossing list
        (shared-memory map tiles, tb_blocked.cu)."""
        if self.regen or self.lib.tb_get_option(b"blocked") != 1:
            return False
        return all(bool(self.lib.tb_obs_blocked(o.handle().h)) for o in self.obs)

    def _setup_pipeline(self, n_chunks):
        """Multi-GPU with both passes on the block-ordered crossing list: cut the local map into
        pixel chunks so that pass 1 of chunk c+1 and pass 2 of chunk c-1 overlap the NVLink
        reduction of chunk c (the reduction runs on its own high-priority stream)."""
        import os as _os
        self.blocked = self._blocked()
        if self.peer is None or n_chunks < 2 or not self.blocked:
            return
        bounds = pipeline_chunk_bounds(
            self.n_local_submap * self.n_pix_submap, self.world, n_chunks,
            align=int(self.lib.tb_bx_block_pixels()))
        if bounds is None:
            return
        n_chunks = len(bounds) - 1
        for o in self.obs:
            L.check(self.lib.tb_obs_set_pixel_chunks(o.handle().h, n_chunks, L.ptr(bounds)))
        self.chunk_bounds = bounds
        self.n_chunks = n_chunks
        self.comm_stream = torch.cuda.Stream(device=self.device, priority=-1)
        # overlapped, the reduction leaves most of every SM to the passes (measured best: 3
        # CTAs per SM); stand-alone it takes 12
        self.pipe_ctas = int(_os.environ.get("TB_PEER_CTAS", "3"))
        self.ev_binned = [torch.cuda.Event() for _ in range(n_chunks)]
        self.ev_reduced = [torch.cuda.Event() for _ in range(n_chunks)]
        self.pipeline = True
        self.use_graph = _os.environ.get("TB_GRAPH", "1") != "0"
        self._graphs = {}

    def _cov_apply_range(self, pix_first, n_pix):
        """zmap[pix_first : pix_first + n_pix] <- cov . zmap[...] on the CURRENT stream."""
        if n_pix > 0:
            L.check(self.lib.tb_cov_apply_diag(
                1, n_pix, 3, self.cov.data_ptr() + pix_first * 48,
                self.zmap.data_ptr() + pix_first * 24, L.TB_MEM_DEVICE,
                torch.cuda.current_stream(self.device).cuda_stream))

    def _peer_ctas(self, n):
        if self.peer is not None and self._ctas_set != n:
            L.check(self.lib.tb_set_option(b"peer_ctas", n))
            self._ctas_set = n

    def _tune_pipeline(self, reps=3):
        """Time the pipelined against the serial LHS (max over ranks, so that every rank takes
        the same decision) and keep the faster one."""
        import torch.distributed as dist

        g = torch.Generator(device=self.device)
        g.manual_seed(1234)
        a = torch.randn(self.n_amp, generator=g, device=self.device, dtype=torch.float64)
        a[self.amp_flags != 0] = 0.0
        q = torch.zeros_like(a)
        # capture the graph first and agree on it: a rank whose capture is refused must not
        # leave the others waiting in the device-side barrier of a replay
        ok = True
        if self.use_graph:
            try:
                self._capture_pipelined(a, q)
            except Exception as exc:  # noqa: BLE001
                import warnings

                warnings.warn(f"CUDA-graph capture of the chunk pipeline refused ({exc})")
                ok = False
            if not _all_ranks_ok(ok, self.device, self.group):
                self.use_graph = False
                self._graphs = {}
        times, results = [], []
        for pipelined in (True, False):
            self.pipeline = pipelined
            self.lhs(a, q)  # warm-up
            dist.barrier(group=self.group)
            torch.cuda.synchronize(self.device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                self.lhs(a, q)
            e1.record()
            torch.cuda.synchronize(self.device)
            times.append(e0.elapsed_time(e1) / reps)
            results.append(q.clone())
        # the two forms must give the same vector (start-up guard for node sizes the pipeline
        # has not been validated on): relative difference, worst rank
        scale = float(results[1].abs().max())
        diff = float((results[0] - results[1]).abs().max()) / max(scale, 1e-300)
        t = torch.tensor(times + [diff], dtype=torch.float64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        self.pipe_tune_ms = {"pipelined": float(t[0]), "serial": float(t[1]),
                             "max_rel_diff": float(t[2])}
        agree = bool(t[2] <= 1e-10)  # NaN compares False
        if not agree:
            import warnings

            warnings.warn(f"pipelined and serial LHS differ by {float(t[2]):.2e}: "
                          "keeping the serial form")
        self.pipeline = agree and bool(t[0] < t[1])
        self._graphs = {}
        dist.barrier(group=self.group)

    def _lhs_pipelined(self, amps_in, amps_out):
        """The pipelined LHS, replayed from a CUDA graph (3 launches + 2 cross-stream edges per
        chunk)."""
        self._peer_ctas(self.pipe_ctas)
        if not self.use_graph:
            return self._enqueue_pipelined(amps_in, amps_out)
        self._capture_pipelined(amps_in, amps_out).replay()
        return amps_out

    def prepare_lhs(self, amps_in, amps_out):
        """Multi-GPU pipelined form only: capture the CUDA graph of ``lhs(amps_in, amps_out)`` on
        EVERY rank before any rank replays it.  A lazily captured graph is captured while faster
        ranks may already be replaying theirs -- their reduction kernels then spin in the
        device-side barrier until this rank's capture (a device synchronisation, a garbage
        collection and an allocator flush inside torch.cuda.graph) is over; capturing together
        removes that window.  Call it symmetrically on all ranks (solve() does)."""
        if not (self.pipeline and self.world > 1 and getattr(self, "use_graph", False)):
            return
        ok = True
        try:
            self._capture_pipelined(amps_in, amps_out)
        except Exception as exc:  # noqa: BLE001
            import warnings

            warnings.warn(f"CUDA-graph capture of the chunk pipeline refused ({exc})")
            ok = False
        if not _all_ranks_ok(ok, self.device, self.group):
            self.use_graph = False
            self._graphs = {}

    def _capture_pipelined(self, amps_in, amps_out):
        self._peer_ctas(self.pipe_ctas)
        key = (amps_in.data_ptr(), amps_out.data_ptr())
        g = self._graphs.get(key)
        if g is None:
            if len(self._graphs) >= 8:
                self._graphs.clear()
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
                self._enqueue_pipelined(amps_in, amps_out)
            torch.cuda.current_stream(self.device).wait_stream(side)
            self._graphs[key] = g
        return g

    def _enqueue_pipelined(self, amps_in, amps_out, timeline=None):
        """``timeline``: optional list receiving (label, start event, end event) per launch
        (diagnostics: profiles/pipe_timeline.py)."""
        main = torch.cuda.current_stream(self.device)
        ms, cs = main.cuda_stream, self.comm_stream.cuda_stream

        def timed(label, stream, fn):
            if timeline is None:
                return fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            timeline.append((label, e0, e1))

        # (the block-ordered pass 1 writes every block of the map: no zero-fill)
        timed("zero", main, lambda: amps_out.zero_())
        for c in range(self.n_chunks):
            def p1(c=c):
                for k, o in enumerate(self.obs):
                    L.check(self.lib.tb_bx_pass1(o.handle().h, L.ptr(amps_in),
                                                 L.ptr(self.amp_flags), L.ptr(self.zmap),
                                                 1 if k > 0 else 0, c, ms))
            timed(f"pass1[{c}]", main, p1)
            self.ev_binned[c].record(main)
            self.comm_stream.wait_event(self.ev_binned[c])
            first = int(self.chunk_bounds[c])
            count = int(self.chunk_bounds[c + 1]) - first
            timed(f"reduce[{c}]", self.comm_stream,
                  lambda: self.peer.reduce_cov(self.cov, first, count, cs))
            self.ev_reduced[c].record(self.comm_stream)
        for c in range(self.n_chunks):
            main.wait_event(self.ev_reduced[c])

            def p2(c=c):
                for o in self.obs:
                    L.check(self.lib.tb_bx_pass2(o.handle().h, L.ptr(self.zmap), L.ptr(amps_out),
                                                 c, ms))
            timed(f"pass2[{c}]", main, p2)
        return amps_out

    def _st(self):
        """The CUDA stream every native launch of this solver goes to: torch's CURRENT stream, so
        that kernels and the surrounding tensor ops (zero_, copy_, NCCL collectives) stay
        ordered under ``with torch.cuda.stream(s)`` as well.  (The deterministic reductions use
        one scratch area per device: issue them from one stream at a time.)"""
        return torch.cuda.current_stream(self.device).cuda_stream

    # -- collectives ----------------------------------------------------------------------------
    def _allreduce(self, t):
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=self.group)

    # -- building blocks ------------------------------------------------------------------------
    def reduce_and_apply_cov(self):
        """zmap <- cov . sum_over_ranks(zmap): the collective of the path and the step after it
        (mapmaker_utils.py:885-925 + covariance.py:262-306), fused over NVLink peer memory when
        there is more than one rank."""
        if self.peer is not None:
            self._peer_ctas(12)
            self.peer.reduce_cov(self.cov, stream=self._st())
            return
        self._allreduce(self.zmap)
        L.check(self.lib.tb_cov_apply_diag(self.n_local_submap, self.n_pix_submap, 3,
                                           L.ptr(self.cov), L.ptr(self.zmap), L.TB_MEM_DEVICE,
                                           self._st()))

    def bin_amplitudes_raw(self, amps):
        """This rank's raw noise-weighted map P^T N^-1 F a -- pass 1 only, no reduction, no
        covariance (diagnostics: bench.py checks the fused reduction against NCCL on it)."""
        st = torch.cuda.current_stream(self.device).cuda_stream
        if self._blocked():
            for k, o in enumerate(self.obs):
                L.check(self.lib.tb_bx_pass1(o.handle().h, L.ptr(amps), L.ptr(self.amp_flags),
                                             L.ptr(self.zmap), 1 if k > 0 else 0, -1, st))
            return self.zmap
        self.zmap.zero_()
        for o in self.obs:
            L.check(self.lib.tb_lhs_pass1(o.handle().h, L.ptr(amps), L.ptr(self.amp_flags),
                                          L.ptr(self.zmap), self.regen, self._st()))
        return self.zmap

    def bin_signal(self, signals):
        """binned = cov * allreduce(P^T N^-1 d) for stored timestreams (one tensor per obs)."""
        self.zmap.zero_()
        for o, sig in zip(self.obs, signals):
            L.check(self.lib.tb_bin_signal(o.handle().h, L.ptr(sig), L.ptr(self.zmap), self.regen,
                                           self._st()))
        self.reduce_and_apply_cov()
        return self.zmap

    def lhs(self, amps_in, amps_out, timers=None):
        """SolverLHS: amps_out = F^T N^-1 Z F amps_in.  ``timers``: optional list that receives
        four CUDA events (pass 1 start/end, pass 2 start/end) of the un-pipelined form."""
        if self.pipeline and timers is None:
            self._lhs_pipelined(amps_in, amps_out)
            return self._add_prior(amps_in, amps_out)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timers is not None \
            else None
        if self._blocked():
            return self._lhs_blocked(amps_in, amps_out, ev, timers)
        self.zmap.zero_()
        if ev:
            ev[0].record()
        for o in self.obs:
            L.check(self.lib.tb_lhs_pass1(o.handle().h, L.ptr(amps_in), L.ptr(self.amp_flags),
                                          L.ptr(self.zmap), self.regen, self._st()))
        if ev:
            ev[1].record()
        self.reduce_and_apply_cov()
        amps_out.zero_()
        if ev:
            ev[2].record()
        for o in self.obs:
            L.check(self.lib.tb_lhs_pass2(o.handle().h, L.ptr(amps_in), L.ptr(self.amp_flags),
                                          L.ptr(self.zmap), L.ptr(amps_out), self.regen,
                                          self._st()))
        if ev:
            ev[3].record()
            timers.append(ev)
        return self._add_prior(amps_in, amps_out)

    def _lhs_blocked(self, amps_in, amps_out, ev, timers):
        """The LHS on the block-ordered crossing list.  One observation on one GPU: ONE kernel
        (pass 1 -> covariance -> pass 2 with the map tile in shared memory); otherwise pass 1
        writes the map (no zero-fill, no atomics), the reduction + covariance follow, and pass 2
        reads it back tile by tile."""
        st = torch.cuda.current_stream(self.device).cuda_stream
        fused = self.world == 1 and len(self.obs) == 1 and self.fuse_lhs
        amps_out.zero_()
        if ev:
            ev[0].record()
        if fused:
            if ev:
                ev[1].record()
                ev[2].record()
            L.check(self.lib.tb_bx_fused(self.obs[0].handle().h, L.ptr(amps_in),
                                         L.ptr(self.amp_flags), L.ptr(self.cov), L.ptr(self.zmap),
                                         L.ptr(amps_out), st))
        else:
            for k, o in enumerate(self.obs):
                L.check(self.lib.tb_bx_pass1(o.handle().h, L.ptr(amps_in), L.ptr(self.amp_flags),
                                             L.ptr(self.zmap), 1 if k > 0 else 0, -1, st))
            if ev:
                ev[1].record()
            self.reduce_and_apply_cov()
            if ev:
                ev[2].record()
            for o in self.obs:
                L.check(self.lib.tb_bx_pass2(o.handle().h, L.ptr(self.zmap), L.ptr(amps_out), -1,
                                             st))
        if ev:
            ev[3].record()
            timers.append(ev)
        return self._add_prior(amps_in, amps_out)

    def _add_prior(self, amps_in, amps_out):
        # mapmaker_solve.py:395-412 adds the prior BEFORE the projection accumulates into the same
        # vector; the sum is the same and flagged amplitudes receive nothing from either term
        if self.prior is not None:
            self.prior.add(amps_in, self.amp_flags, amps_out, stream=self._st())
        return amps_out

    def precond(self, r, s):
        """s = M^-1 r: diagonal offset variance (template_offset.cpp:375-402), or the noise-prior
        preconditioner."""
        if self.prior is not None:
            self.prior.precond(r, self.amp_flags, s, stream=self._st())
        else:
            L.check(self.lib.tb_template_offset_apply_diag_precond(
                L.ptr(self.offset_var), L.ptr(r), L.ptr(self.amp_flags), L.ptr(s), self.n_amp,
                L.TB_MEM_DEVICE, self._st()))

    def rhs(self, signals):
        """SolverRHS: F^T N^-1 Z d."""
        binned = self.bin_signal(signals)
        out = torch.zeros(self.n_amp, dtype=torch.float64, device=self.device)
        for o, sig in zip(self.obs, signals):
            L.check(self.lib.tb_rhs_project(o.handle().h, L.ptr(sig), L.ptr(self.amp_flags),
                                            L.ptr(binned), L.ptr(out), self.regen, self._st()))
        return out

    def dot(self, a, b, out):
        L.check(self.lib.tb_amp_dot(L.ptr(a), L.ptr(b), L.ptr(self.amp_flags), self.n_amp,
                                    L.ptr(out), self._st()))
        self._allreduce(out)

    # -- PCG --------------------------------------------------------------------------------------
    def lhs_and_dot(self, st):
        """q = A d and d.q (device scalars): the expensive, state-preserving half of an
        iteration (does not touch x or r)."""
        self.lhs(st.d, st.q)
        self.dot(st.d, st.q, st.dq)

    def update(self, st):
        """alpha = delta / d.q; x += alpha d; r -= alpha q; s = M^-1 r; sums = (r.r, s.r)."""
        L.check(self.lib.tb_pcg_update(L.ptr(st.delta), L.ptr(st.dq), L.ptr(st.x), L.ptr(st.r),
                                       L.ptr(st.d), L.ptr(st.q), L.ptr(st.s),
                                       L.ptr(self.offset_var), L.ptr(self.amp_flags), self.n_amp,
                                       L.ptr(st.sums), self._st()))
        if self.prior is not None:
            # the fused update applied the diagonal preconditioner: redo s and s.r with the prior's
            self.precond(st.r, st.s)
            L.check(self.lib.tb_amp_dot(L.ptr(st.s), L.ptr(st.r), L.ptr(self.amp_flags),
                                        self.n_amp, L.ptr(st.sums[1:]), self._st()))
        self._allreduce(st.sums)

    def iteration(self, st):
        """One full PCG iteration in the reference's order (mapmaker_solve.py:665-694)."""
        self.lhs_and_dot(st)
        self.update(st)

    def advance_direction(self, st):
        # delta_new = s.r = sums[1];  beta = delta_new / delta_old;  d = s + beta d
        L.check(self.lib.tb_pcg_direction(L.ptr(st.sums[1:]), L.ptr(st.delta), L.ptr(st.d),
                                          L.ptr(st.s), self.n_amp, self._st()))
        st.delta.copy_(st.sums[1:2])

    def solve(self, rhs, convergence=1.0e-12, n_iter_max=100, n_iter_min=3, x0=None):
        """The PCG of mapmaker_solve.py:524-755.  Returns (amplitudes, relative residuals).

        Same arithmetic and stopping rules as the reference.  The host needs one scalar per
        iteration (r.r) for the convergence / stall tests; instead of idling the GPU while it
        is read back, the next search direction and the next LHS -- which do not modify x or r
        -- are enqueued first, so on exit x and r are exactly the reference's."""
        dev = self.device
        n = self.n_amp
        st = _PCGState(n, dev)
        if x0 is not None:
            st.x.copy_(x0)
        self.prepare_lhs(st.x, st.q)   # (multi-GPU pipeline: both graphs captured up front,
        self.prepare_lhs(st.d, st.q)   #  on all ranks together)
        self.lhs(st.x, st.q)
        st.r.copy_(rhs)
        st.r.sub_(st.q)
        self.precond(st.r, st.s)
        st.d.copy_(st.s)
        tmp = torch.zeros(1, dtype=torch.float64, device=dev)
        self.dot(rhs, rhs, tmp)
        sqsum = float(tmp.item())
        sqsum_init = sqsum
        sqsum_best = sqsum
        last_best = sqsum
        self.dot(st.d, st.r, st.delta)
        history = []
        host = torch.zeros(2, dtype=torch.float64).pin_memory()
        ev = torch.cuda.Event()
        if n_iter_max > 0:
            self.lhs_and_dot(st)
        for it in range(n_iter_max):
            if not np.isfinite(sqsum):
                raise RuntimeError("Residual is not finite")
            self.update(st)
            host.copy_(st.sums, non_blocking=True)
            ev.record()
            if it + 1 < n_iter_max:  # speculative: keeps the GPU busy during the read-back
                self.advance_direction(st)
                self.lhs_and_dot(st)
            ev.synchronize()
            sqsum = float(host[0])
            relative = sqsum / sqsum_init
            history.append(relative)
            if relative < convergence or sqsum < 1e-30:
                break
            sqsum_best = min(sqsum, sqsum_best)
            if it % 10 == 0 and it >= n_iter_min:
                if last_best < sqsum_best * 2:
                    break
                last_best = sqsum_best
        return st.x, history


class _PCGState:
    def __init__(self, n, dev):
        z = lambda: torch.zeros(n, dtype=torch.float64, device=dev)
        self.x, self.r, self.d, self.q, self.s = z(), z(), z(), z(), z()
        self.delta = torch.zeros(1, dtype=torch.float64, device=dev)
        self.dq = torch.zeros(1, dtype=torch.float64, device=dev)
        self.sums = torch.zeros(2, dtype=torch.float64, device=dev)
