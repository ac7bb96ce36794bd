"""Device side of the hot path: bit-packed mask pools and batched scoring passes.

A *pass* takes a batch of jobs — one source frame per job, each with its own list
of candidate rigid transforms and target frames — and returns, per target, the
first candidate of maximal mask IoU with its integer counts.  This is the unit
the reference executes one (source, angle) and one (target) at a time in Python
(utils/opt_utils.py:438-488).  PyTorch is used for device memory and streams
only; all arithmetic is in csrc/a3d.cu behind the C ABI of include/a3d.h.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .config import OptConfig


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise _lib.A3DError(f"{name} must live on a CUDA device (the hot path has no CPU fallback)")


def camera_struct(cfg: OptConfig) -> _lib.Camera:
    cam = _lib.Camera()
    kinv = cfg.K_inv().reshape(-1)
    for i in range(9):
        cam.kinv[i] = float(kinv[i])
    cam.f = float(cfg.focal_length)
    cam.cx = float(cfg.cx)
    cam.cy = float(cfg.cy)
    cam.H, cam.W = int(cfg.height), int(cfg.width)
    return cam


def point_caps(src_points) -> np.ndarray:
    """Point-cloud capacities (``a3d_job_t.pcd_cap``) of the pool's masks: source pixels rounded up to 32."""
    return (np.asarray(src_points, dtype=np.int64) + 31) & ~31


@dataclass
class MaskPool:
    """Bit-packed masks resident in HBM plus their popcounts / bounding boxes."""
    bits: torch.Tensor                    # (n, H, pitch) int32: bit = mask > thresh
    popc: torch.Tensor                    # (n,) int32
    bbox: torch.Tensor                    # (n, 4) int32 {row_min,row_max,word_min,word_max}
    H: int
    W: int
    bits_nz: torch.Tensor | None = None   # bit = mask != 0 (source pixel lists), if it differs
    bbox_nz: torch.Tensor | None = None
    popc_nz: torch.Tensor | None = None
    _src_points: np.ndarray | None = None
    _nz_pending: tuple | None = None      # (bits_nz, bbox_nz, popc_nz) not yet compared with bits (PoolBuilder)

    def __len__(self):
        return self.bits.shape[0]

    def _resolve(self):
        """First host-side use of the pool: ONE D2H of the count vectors (the host needs the
        source-pixel counts to size the point-cloud workspace).  Binary masks (the contract) give
        identical ``> thresh`` and ``!= 0`` counts and the second bitmap is dropped.  Deferred to here
        so that the upload and packing stay asynchronous behind the host's geometry work."""
        if self._nz_pending is not None:
            nz, bbox_nz, popc_nz = self._nz_pending
            self._nz_pending = None
            both = torch.stack((self.popc, popc_nz)).cpu().numpy()
            if not np.array_equal(both[0], both[1]):
                self.bits_nz, self.bbox_nz, self.popc_nz = nz, bbox_nz, popc_nz
            self._src_points = both[1].astype(np.int64)
        elif self._src_points is None:
            t = self.popc if self.popc_nz is None else self.popc_nz
            self._src_points = t.cpu().numpy().astype(np.int64)

    @property
    def source_points(self) -> np.ndarray:
        """Host copy of the source-pixel counts; one D2H per pool, cached."""
        if self._src_points is None or self._nz_pending is not None:
            self._resolve()
        return self._src_points

    @property
    def source_bits(self):
        if self._nz_pending is not None:
            self._resolve()
        return self.bits if self.bits_nz is None else self.bits_nz

    @property
    def source_bbox(self):
        if self._nz_pending is not None:
            self._resolve()
        return self.bbox if self.bbox_nz is None else self.bbox_nz


def mask_meta(bits: torch.Tensor, H: int, W: int):
    lib = _lib.load()
    _require_cuda(bits, "bits")
    n = bits.shape[0]
    popc = torch.empty(n, dtype=torch.int32, device=bits.device)
    bbox = torch.empty(n, 4, dtype=torch.int32, device=bits.device)
    _lib.check(lib.a3d_mask_meta(bits.data_ptr(), n, H, W, popc.data_ptr(), bbox.data_ptr(), _stream_ptr()),
               "a3d_mask_meta")
    return popc, bbox


def pack_masks(masks: torch.Tensor, thresh: float = 0.5, with_nonzero: bool = False) -> MaskPool:
    """(n, H, W) fp32 / uint8 / bool CUDA tensor -> MaskPool."""
    lib = _lib.load()
    _require_cuda(masks, "masks")
    if masks.dim() != 3:
        raise ValueError("masks must be (n, H, W)")
    if masks.dtype == torch.bool:
        masks = masks.view(torch.uint8)
    if masks.dtype == torch.float32:
        dt = _lib.A3D_F32
    elif masks.dtype == torch.uint8:
        dt = _lib.A3D_U8
    else:
        raise TypeError(f"unsupported mask dtype {masks.dtype}")
    masks = masks.contiguous()
    n, H, W = masks.shape
    pitch = _lib.pitch_words(W)
    with torch.cuda.device(masks.device):
        bits = torch.empty(n, H, pitch, dtype=torch.int32, device=masks.device)
        nz = torch.empty_like(bits) if with_nonzero else None
        _lib.check(lib.a3d_pack_masks(masks.data_ptr(), dt, n, H, W, float(thresh), bits.data_ptr(),
                                      nz.data_ptr() if nz is not None else None, _stream_ptr()),
                   "a3d_pack_masks")
        popc, bbox = mask_meta(bits, H, W)
        pool = MaskPool(bits, popc, bbox, H, W)
        if with_nonzero:
            popc_nz, bbox_nz = mask_meta(nz, H, W)
            # identical for binary masks (the contract); keep the second copy only if needed
            if not torch.equal(popc_nz, popc):
                pool.bits_nz, pool.bbox_nz, pool.popc_nz = nz, bbox_nz, popc_nz
    return pool


class PoolBuilder:
    """A MaskPool filled chunk by chunk: ``append`` packs a dense (k, H, W) CUDA chunk into the next k
    slots of the preallocated bit planes (the chunk buffer can be reused right after, stream order),
    ``finish`` computes popcounts / boxes once over the whole pool."""

    def __init__(self, n: int, H: int, W: int, device, with_nonzero: bool = False, thresh: float = 0.5):
        self.n, self.H, self.W, self.thresh = n, H, W, float(thresh)
        self.device = torch.device(device)
        pitch = _lib.pitch_words(W)
        with torch.cuda.device(self.device):
            self.bits = torch.empty(n, H, pitch, dtype=torch.int32, device=self.device)
            self.nz = torch.empty_like(self.bits) if with_nonzero else None
        self.fill = 0

    def append(self, masks: torch.Tensor):
        lib = _lib.load()
        _require_cuda(masks, "masks")
        if masks.dtype == torch.bool:
            masks = masks.view(torch.uint8)
        dt = {torch.float32: _lib.A3D_F32, torch.uint8: _lib.A3D_U8}.get(masks.dtype)
        if dt is None:
            raise TypeError(f"unsupported mask dtype {masks.dtype}")
        masks = masks.contiguous()
        k = int(masks.shape[0])
        if self.fill + k > self.n or tuple(masks.shape[1:]) != (self.H, self.W):
            raise ValueError("chunk does not fit the pool")
        with torch.cuda.device(self.device):
            _lib.check(lib.a3d_pack_masks(masks.data_ptr(), dt, k, self.H, self.W, self.thresh,
                                          self.bits[self.fill:].data_ptr(),
                                          self.nz[self.fill:].data_ptr() if self.nz is not None else None,
                                          _stream_ptr()), "a3d_pack_masks")
        self.fill += k

    def finish(self) -> MaskPool:
        if self.fill != self.n:
            raise ValueError(f"pool holds {self.fill} of {self.n} masks")
        with torch.cuda.device(self.device):
            popc, bbox = mask_meta(self.bits, self.H, self.W)
            pool = MaskPool(self.bits, popc, bbox, self.H, self.W)
            if self.nz is not None:
                popc_nz, bbox_nz = mask_meta(self.nz, self.H, self.W)
                pool._nz_pending = (self.nz, bbox_nz, popc_nz)       # compared on first host-side use
        return pool


def pool_from_bits(bits: torch.Tensor, H: int, W: int) -> MaskPool:
    """Wrap already packed masks ((n, H, pitch) int32 on the device)."""
    _require_cuda(bits, "bits")
    assert bits.dtype == torch.int32 and bits.shape[1] == H and bits.shape[2] == _lib.pitch_words(W)
    with torch.cuda.device(bits.device):
        popc, bbox = mask_meta(bits.contiguous(), H, W)
    return MaskPool(bits.contiguous(), popc, bbox, H, W)


def plan_tiles(jobs: np.ndarray, max_tile: int, sm_count: int | None = None, fixed: float = 21500.0, per_cand: float = 3000.0):
    """Split of a pass into projection CTAs when the grid is about one wave: jobs whose source masks
    differ in size get tiles of different size, so that every CTA carries about the same number of
    (point, candidate) pairs and the SMs finish together (uniform tiles leave the kernel waiting for the
    CTAs of the largest mask: C2's four tracks have 10-38 k source pixels).

    Cost model, in point units, from the ncu instruction counts of k_project<filter> on C2: a CTA costs
    ``fixed + tile * (per_cand + points)``; the job's extra CTA (exact-only candidates, role 1)
    ``fixed + per_cand + 2.5 * points``.  Returns ``(tile_cand, tile_map)``; ``tile_map`` is None when
    the grid is several waves anyway (uniform tiles of ``tile_cand``, the hardware scheduler balances) and
    else an int32 array (n_tiles, 4) of {job, first candidate, candidates, role}, most expensive first."""
    n = len(jobs)
    if n == 0:
        return max_tile, None
    if sm_count is None:
        sm_count = plan_sm_count()
    ncand = jobs["n_cand"].astype(np.int64)
    cost = jobs["pcd_cap"].astype(np.float64) + per_cand
    min_ctas = int((-(-ncand // max_tile)).sum())
    waves = 1 if min_ctas + n <= sm_count else 2
    if min_ctas + n > waves * sm_count:
        return max_tile, None
    cap = waves * sm_count - n

    def tiles_for(w):
        return np.clip(np.floor(w / cost), 1, max_tile).astype(np.int64)

    lo, hi = float(cost.min()), float(cost.max()) * max_tile
    for _ in range(40):                                  # smallest budget whose CTAs fit the wave(s)
        mid = 0.5 * (lo + hi)
        if int((-(-ncand // tiles_for(mid))).sum()) <= cap:
            hi = mid
        else:
            lo = mid
    tile = tiles_for(hi)
    rows = []
    for j in range(n):
        if ncand[j] == 0:
            continue
        k = int(-(-ncand[j] // tile[j]))
        base, rem = divmod(int(ncand[j]), k)
        c = 0
        for i in range(k):
            sz = base + (1 if i < rem else 0)
            rows.append((fixed + sz * cost[j], j, c, sz, 0))
            c += sz
    for j in range(n):
        rows.append((fixed + per_cand + 2.5 * float(jobs["pcd_cap"][j]), j, 0, 0, 1))
    rows.sort(key=lambda r: -r[0])
    tmap = np.array([r[1:] for r in rows], dtype=np.int32).reshape(-1, 4)
    return int(tmap[:, 2].max()), tmap




_sm_cache: dict = {}


def plan_sm_count(device=None) -> int:
    """SMs a one-wave projection grid is planned for: all of the device's (``A3D_PLAN_SMS`` overrides).
    Leaving 4 of them to the collective's kernel when several ranks gather results was measured slower
    (C2, 2 GPUs: 64.5 against 59.4 us per step — the plan loses more than the collective takes)."""
    env = os.environ.get("A3D_PLAN_SMS")
    if env:
        return max(1, int(env))
    key = str(device)
    sms = _sm_cache.get(key)
    if sms is None:
        sms = _sm_cache[key] = torch.cuda.get_device_properties(
            device if device is not None else torch.cuda.current_device()).multi_processor_count
    return max(1, sms)


def plan_tiles_native(jobs: np.ndarray, max_tile: int, sm_count: int | None = None):
    """``plan_tiles`` through the library's host planner (a3d_plan_tiles): same result, microseconds."""
    lib = _lib.load()
    if sm_count is None:
        sm_count = plan_sm_count()
    buf = np.empty((2 * sm_count, 4), dtype=np.int32)          # per call: worker threads plan concurrently
    jobs = np.ascontiguousarray(jobs)
    tile = C.c_int(0)
    n = _lib.check(lib.a3d_plan_tiles(jobs.ctypes.data, len(jobs), max_tile, sm_count, buf.ctypes.data, len(buf),
                                      C.byref(tile)), "a3d_plan_tiles")
    return (tile.value, buf[:n].copy()) if n > 0 else (tile.value, None)


@dataclass
class JobBatch:
    """Host description of one pass (numpy, ready for a single H2D each)."""
    jobs: np.ndarray          # (n_jobs,) _lib.JOB_DTYPE
    xform: np.ndarray         # (n_cand_total, 12) fp32
    tgt_index: np.ndarray     # (n_tgt_total,) int32 indices into the target pool

    @property
    def n_jobs(self):
        return len(self.jobs)

    @property
    def units(self) -> int:
        """track-frame x candidate IoU evaluations in this pass."""
        return int((self.jobs["n_cand"].astype(np.int64) * self.jobs["n_tgt"]).sum())


def build_batch(sources, modes, normals, offsets, pivots, xforms, targets, src_points) -> JobBatch:
    """Assemble a JobBatch from per-job python/numpy pieces.

    sources[i] pool index; modes[i] MODE_*; normals[i] (3,), offsets[i], pivots[i] (3,);
    xforms[i] (A_i, 12) fp32; targets[i] sequence of pool indices; src_points = per-mask
    source pixel counts of the pool (``MaskPool.source_points``)."""
    n = len(sources)
    jobs = np.zeros(n, dtype=_lib.JOB_DTYPE)
    caps = point_caps(src_points)
    cand = tgt = tab = pcd = 0
    for i in range(n):
        a, t = len(xforms[i]), len(targets[i])
        jobs[i]["src_mask"] = sources[i]
        jobs[i]["mode"] = modes[i]
        jobs[i]["cand_begin"], jobs[i]["n_cand"] = cand, a
        jobs[i]["tgt_begin"], jobs[i]["n_tgt"] = tgt, t
        jobs[i]["normal"] = np.asarray(normals[i], dtype=np.float32)
        jobs[i]["offset"] = np.float32(offsets[i])
        jobs[i]["pivot"] = np.asarray(pivots[i], dtype=np.float32)
        jobs[i]["tab_begin"] = tab
        cap = int(caps[sources[i]])
        jobs[i]["pcd_begin"], jobs[i]["pcd_cap"] = pcd, cap
        pcd += cap
        cand += a
        tgt += t
        tab += a * t
    xform = (np.concatenate([np.asarray(x, dtype=np.float32).reshape(-1, 12) for x in xforms])
             if n else np.zeros((0, 12), np.float32))
    tgt_index = (np.concatenate([np.asarray(t, dtype=np.int32).reshape(-1) for t in targets])
                 if n else np.zeros(0, np.int32))
    return JobBatch(jobs, np.ascontiguousarray(xform), np.ascontiguousarray(tgt_index))


def build_batch_rows(sources, modes, normals, offsets, pivots, xform, n_cand, tgt_index, n_tgt,
                     src_points) -> JobBatch:
    """``build_batch`` from arrays, without a python loop over jobs: sources/modes/offsets (S,),
    normals/pivots (S,3), xform (sum n_cand, 12) fp32 in job order, n_cand/n_tgt (S,) counts,
    tgt_index (sum n_tgt,) pool indices in job order."""
    sources = np.asarray(sources, dtype=np.int64)
    S = len(sources)
    n_cand = np.asarray(n_cand, dtype=np.int64).reshape(S)
    n_tgt = np.asarray(n_tgt, dtype=np.int64).reshape(S)
    jobs = np.zeros(S, dtype=_lib.JOB_DTYPE)
    if S:
        jobs["src_mask"] = sources
        jobs["mode"] = np.asarray(modes, dtype=np.int32)
        jobs["n_cand"], jobs["n_tgt"] = n_cand, n_tgt
        jobs["cand_begin"] = np.cumsum(n_cand) - n_cand
        jobs["tgt_begin"] = np.cumsum(n_tgt) - n_tgt
        jobs["normal"] = np.asarray(normals, dtype=np.float32).reshape(S, 3)
        jobs["offset"] = np.asarray(offsets, dtype=np.float32).reshape(S)
        jobs["pivot"] = np.asarray(pivots, dtype=np.float32).reshape(S, 3)
        tab = n_cand * n_tgt
        jobs["tab_begin"] = np.cumsum(tab) - tab
        cap = point_caps(src_points)[sources]
        jobs["pcd_cap"] = cap
        jobs["pcd_begin"] = np.cumsum(cap) - cap
    xform = np.ascontiguousarray(np.asarray(xform, dtype=np.float32).reshape(-1, 12))
    tgt_index = np.ascontiguousarray(np.asarray(tgt_index, dtype=np.int32).reshape(-1))
    assert len(xform) == int(n_cand.sum()) and len(tgt_index) == int(n_tgt.sum())
    return JobBatch(jobs, xform, tgt_index)


@dataclass
class PassResult:
    best_cand: torch.Tensor       # (n_tgt_total,) int32, candidate index local to the job
    best_inter: torch.Tensor      # (n_tgt_total,) int32
    best_union: torch.Tensor      # (n_tgt_total,) int32
    best_iou: torch.Tensor        # (n_tgt_total,) fp32
    proj_bits: torch.Tensor       # (n_cand_total, H, pitch) int32
    proj_popc: torch.Tensor       # (n_cand_total,) int32
    proj_bbox: torch.Tensor       # (n_cand_total, 4) int32
    inter_tab: torch.Tensor | None
    block: torch.Tensor | None = None     # (4, n_tgt_total) int32: the four best_* rows, contiguous
    rows_only: bool = False               # written with A3D_OUT_BBOX_ROWS (proj_bits is fully defined either way)

    def masks(self, index: torch.Tensor | None = None) -> torch.Tensor:
        """Projected masks ``index`` (global candidate slots; None = all), copied out of the pass workspace."""
        return self.proj_bits.clone() if index is None else self.proj_bits.index_select(0, index.long())


class DeviceBatch:
    """A JobBatch uploaded to the device (inputs resident in HBM)."""

    def __init__(self, batch: JobBatch, device, staging: "Staging | None" = None, cfg: OptConfig | None = None):
        self.host = batch
        self.device = device
        self._plans = {}
        plan = None
        if cfg is not None and os.environ.get("A3D_TILE_PLAN") != "uniform":
            plan = plan_tiles_native(batch.jobs, max_tile(cfg), plan_sm_count(device))
            if plan[1] is None:
                plan = (choose_tile(cfg, int(batch.xform.shape[0]), batch.n_jobs, plan_sm_count(device)), None)
            self._plans[_plan_key(cfg)] = plan
        tmap = plan[1] if plan is not None and plan[1] is not None else np.zeros((0, 4), np.int32)
        self.n_jobs = batch.n_jobs
        self.n_cand_total = int(batch.xform.shape[0])
        self.n_tgt_total = int(batch.tgt_index.shape[0])
        self.max_cand = int(batch.jobs["n_cand"].max()) if self.n_jobs else 0
        self.max_tgt = int(batch.jobs["n_tgt"].max()) if self.n_jobs else 0
        self.tab_total = int((batch.jobs["n_cand"].astype(np.int64) * batch.jobs["n_tgt"]).sum())
        self.pcd_total = int(batch.jobs["pcd_cap"].astype(np.int64).sum())
        # one H2D for the three arrays: pinned staging block [jobs | xform | tgt_index], 16-byte aligned parts
        nj, nx, nt, nm = batch.jobs.nbytes, batch.xform.nbytes, batch.tgt_index.nbytes, tmap.nbytes
        oj, ox = 0, (nj + 15) & ~15
        ot = (ox + nx + 15) & ~15
        om = (ot + nt + 15) & ~15
        total = (max(om + nm, 16) + 15) & ~15
        host = staging.host(total) if staging is not None else torch.empty(total, dtype=torch.uint8).pin_memory()
        hv = host.numpy()
        hv[oj:oj + nj] = batch.jobs.view(np.uint8).reshape(-1)
        hv[ox:ox + nx] = batch.xform.view(np.uint8).reshape(-1)
        hv[ot:ot + nt] = batch.tgt_index.view(np.uint8).reshape(-1)
        hv[om:om + nm] = tmap.view(np.uint8).reshape(-1)
        dev = staging.device_block(total) if staging is not None else torch.empty(total, dtype=torch.uint8, device=device)
        if staging is not None and os.environ.get("A3D_DESC_COPY") != "dma":
            # by a kernel that reads the pinned block over PCIe: a DMA copy would queue on the host-to-device
            # copy engine behind the mask uploads of the next video (and its submission blocks while that
            # engine's queue is full: 14 ms per video, measured with tools/e2e_timeline.py)
            with torch.cuda.device(dev.device):
                _lib.check(_lib.load().a3d_fetch_host_block(dev.data_ptr(), host.data_ptr(), total, _stream_ptr()),
                           "a3d_fetch_host_block")
        else:
            dev[:total].copy_(host[:total], non_blocking=True)
        if staging is not None:
            staging.host_done()
        self.jobs = dev[oj:oj + nj]
        self.xform = dev[ox:ox + nx].view(torch.float32).view(-1, 12)
        self.tgt_index = dev[ot:ot + nt].view(torch.int32)
        self._tmap_dev = {_plan_key(cfg): dev[om:om + nm].view(torch.int32).view(-1, 4)} if nm else {}

    def tile_plan(self, cfg: OptConfig):
        """(tile_cand, device tile map or None) for this camera: planned once, uploaded once."""
        key = _plan_key(cfg)
        if key not in self._plans:
            if os.environ.get("A3D_TILE_PLAN") == "uniform":
                self._plans[key] = (choose_tile(cfg, self.n_cand_total, self.n_jobs, plan_sm_count(self.device)), None)
            else:
                tile, tmap = plan_tiles_native(self.host.jobs, max_tile(cfg), plan_sm_count(self.device))
                if tmap is None:
                    tile = choose_tile(cfg, self.n_cand_total, self.n_jobs, plan_sm_count(self.device))
                else:
                    self._tmap_dev[key] = torch.from_numpy(tmap).to(self.device)
                self._plans[key] = (tile, tmap)
        return self._plans[key][0], self._tmap_dev.get(key)


class Staging:
    """Reusable pinned-host / device byte blocks for the per-pass descriptors and results.

    Passes are enqueued without waiting for the device (several chunks of one table pass, the next video's
    table pass ahead of the current video's final pass), so the pinned block a pass's descriptors are copied
    from must not be refilled before that copy has run: ``host`` hands out a small ring of blocks, each
    guarded by the event recorded after its copy (``host_done``).  The device block needs no ring: all passes
    of one ``Staging`` are issued on one stream, where the next copy into it queues behind the kernels that
    read it."""
    RING = 4

    def __init__(self, device):
        self.device = torch.device(device)
        self._ring = [None] * self.RING          # pinned blocks
        self._busy = [None] * self.RING          # event after the last H2D out of the block
        self._next = 0
        self._dev = self._res_host = None

    def host(self, n):
        i = self._next
        self._next = (i + 1) % self.RING
        self._slot = i
        if self._busy[i] is not None:
            self._busy[i].synchronize()          # long done unless four passes are in flight
            self._busy[i] = None
        if self._ring[i] is None or self._ring[i].numel() < n:
            self._ring[i] = torch.empty(max(n, 1 << 16), dtype=torch.uint8).pin_memory()
        return self._ring[i]

    def host_done(self):
        """Call after enqueuing the copy out of the block ``host`` returned last."""
        ev = torch.cuda.Event()
        ev.record()
        self._busy[self._slot] = ev

    def device_block(self, n):
        if self._dev is None or self._dev.numel() < n:
            self._dev = torch.empty(max(n, 1 << 16), dtype=torch.uint8, device=self.device)
        return self._dev

    def results_host(self, n_int32):
        if self._res_host is None or self._res_host.numel() < n_int32:
            self._res_host = torch.empty(max(n_int32, 1 << 12), dtype=torch.int32).pin_memory()
        return self._res_host[:n_int32]


class Workspace:
    """Reusable device buffers of a pass (outputs and projected masks)."""

    def __init__(self, device):
        self.device = torch.device(device)
        self._bufs = {}

    def get(self, name, shape, dtype):
        n = int(np.prod(shape))
        buf = self._bufs.get(name)
        if buf is None or buf.numel() < n or buf.dtype != dtype:
            buf = torch.empty(max(n, 1), dtype=dtype, device=self.device)
            if os.environ.get("A3D_WS_POISON"):          # tests: nothing may depend on what a fresh buffer holds
                buf.view(torch.uint8).fill_(0xAB)
            self._bufs[name] = buf
        return buf[:n].view(*shape)

    def get_proj(self, nc: int, H: int, pitch: int):
        """(proj_bits, proj_popc, proj_bbox) for ``nc`` candidate slots, kept in the state A3D_OUT_BBOX_ROWS
        asks for: masks zero outside the rows of their boxes.  A fresh (or re-shaped) pair is all-zero masks
        with empty boxes; afterwards every pass of this workspace maintains the invariant slot by slot."""
        key = (H, pitch)
        cur = self._bufs.get("_proj")
        if cur is None or cur[0] != key or cur[1].shape[0] < nc:
            cap = max(nc, 1) if cur is None or cur[0] != key else max(nc, 2 * cur[1].shape[0])
            self._bufs.pop("_proj", None)                # release the old pair before allocating the new one
            cur = None
            bits = torch.zeros(cap, H, pitch, dtype=torch.int32, device=self.device)
            bbox = torch.zeros(cap, 4, dtype=torch.int32, device=self.device)
            bbox[:, 1] = -1
            bbox[:, 3] = -1
            popc = torch.zeros(cap, dtype=torch.int32, device=self.device)
            cur = self._bufs["_proj"] = (key, bits, popc, bbox)
        return cur[1][:nc], cur[2][:nc], cur[3][:nc]


_cam_cache: dict = {}
_tile_cache: dict = {}


def _camera_cached(cfg: OptConfig) -> _lib.Camera:
    key = (cfg.focal_length, cfg.width, cfg.height)
    cam = _cam_cache.get(key)
    if cam is None:
        cam = _cam_cache[key] = camera_struct(cfg)
    return cam


def _plan_key(cfg: OptConfig):
    """What the largest projection tile depends on: the image size and the projection schedule."""
    return cfg.height, cfg.width, os.environ.get("A3D_PROJECT_SCHED")


def max_tile(cfg: OptConfig) -> int:
    """Most candidates one projection CTA holds in shared memory for this image size and projection schedule
    (persistent CTAs hold two groups of slots, so A3D_PROJECT_SCHED=persistent halves the limit)."""
    key = _plan_key(cfg)
    t = _tile_cache.get(key)
    if t is None:
        lib = _lib.load()
        t = _tile_cache[key] = _lib.check(lib.a3d_project_max_tile(cfg.height, cfg.width), "a3d_project_max_tile")
    return t


def choose_tile(cfg: OptConfig, n_cand_total: int, n_jobs: int = 1, sm_count: int | None = None) -> int:
    """Candidates per projection CTA for uniform tiles.  Large batches take as many as shared memory
    holds (the point cloud is read once per CTA); small batches pick the tile that minimises
    waves x (per-CTA overhead + tile) so no SM runs two CTAs while others idle."""
    mt = max_tile(cfg)
    if sm_count is None:
        sm_count = plan_sm_count()
    per_job = -(-n_cand_total // max(n_jobs, 1))
    best, best_cost = mt, None
    for tile in range(mt, 0, -1):
        ctas = n_jobs * -(-per_job // tile)
        cost = -(-ctas // sm_count) * (0.3 + tile)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = tile, cost
    return int(best)


def default_out_mode() -> int:
    """The engine keeps the projected-mask buffers of a ``Workspace`` between passes, zero outside each slot's
    box, so a pass writes only the rows of the old and the new box of every slot (A3D_OUT_BBOX_ROWS);
    ``A3D_PROJ_OUT=full`` writes every word of every mask instead."""
    return _lib.OUT_FULL if os.environ.get("A3D_PROJ_OUT") == "full" else _lib.OUT_BBOX_ROWS


def run_pass(cfg: OptConfig, pool: MaskPool, dbatch: DeviceBatch, ws: Workspace | None = None,
             want_table: bool = False, tile_cand: int | None = None, out_mode: int | None = None) -> PassResult:
    """project + score one batch, asynchronously on the current stream."""
    lib = _lib.load()
    out_mode = default_out_mode() if out_mode is None else out_mode
    rows_only = out_mode == _lib.OUT_BBOX_ROWS
    dev = pool.bits.device
    ws = ws or Workspace(dev)
    H, W = cfg.height, cfg.width
    if (pool.H, pool.W) != (H, W):
        raise ValueError(f"mask pool is {pool.H}x{pool.W}, camera is {H}x{W}")
    pitch = _lib.pitch_words(W)
    nc, nt = dbatch.n_cand_total, dbatch.n_tgt_total
    with torch.cuda.device(dev):
        proj_bits, proj_popc, proj_bbox = ws.get_proj(nc, H, pitch)
        pcd_ws = ws.get("pcd_ws", (max(_lib.PCD_PLANES * dbatch.pcd_total, 32),), torch.float32)
        pcd_count = ws.get("pcd_count", (dbatch.n_jobs + 1,), torch.int32)
        hom_ws = ws.get("hom_ws", (max(nc, 1), _lib.HOM_FLOATS), torch.float32)
        key_ws = ws.get("key_ws", (nt,), torch.int64)
        results = ws.get("results", (4, nt), torch.int32)          # one block -> one D2H
        best_cand, best_inter, best_union = results[0], results[1], results[2]
        best_iou = results[3].view(torch.float32)
        inter_tab = ws.get("inter_tab", (dbatch.tab_total,), torch.int32) if want_table else None
        if dbatch.n_jobs == 0:
            return PassResult(best_cand, best_inter, best_union, best_iou, proj_bits, proj_popc, proj_bbox, inter_tab)
        cam = _camera_cached(cfg)
        stream = _stream_ptr()
        tmap = None
        if tile_cand is not None:
            tile = tile_cand
        else:
            tile, tmap = dbatch.tile_plan(cfg)
        tmap_ptr, n_tiles = (tmap.data_ptr(), int(tmap.shape[0])) if tmap is not None else (None, 0)
        if os.environ.get("A3D_PASS_API") != "split":
            # one call: keys cleared first, then the four kernels as programmatic dependent launches
            _lib.check(lib.a3d_pass(C.byref(cam), dbatch.jobs.data_ptr(), dbatch.n_jobs, dbatch.max_tgt, dbatch.max_cand,
                                    tile, nt, len(pool), nc, pool.bits.data_ptr(), pool.popc.data_ptr(),
                                    pool.bbox.data_ptr(), pool.source_bits.data_ptr(), pool.source_bbox.data_ptr(),
                                    dbatch.xform.data_ptr(), dbatch.tgt_index.data_ptr(), pcd_ws.data_ptr(),
                                    pcd_count.data_ptr(), hom_ws.data_ptr(), tmap_ptr, n_tiles,
                                    proj_bits.data_ptr(), proj_popc.data_ptr(),
                                    proj_bbox.data_ptr(), key_ws.data_ptr(),
                                    inter_tab.data_ptr() if inter_tab is not None else None,
                                    best_cand.data_ptr(), best_inter.data_ptr(), best_union.data_ptr(),
                                    best_iou.data_ptr(), out_mode, stream), "a3d_pass")
            return PassResult(best_cand, best_inter, best_union, best_iou, proj_bits, proj_popc, proj_bbox, inter_tab,
                              results, rows_only)
        _lib.check(lib.a3d_project(C.byref(cam), dbatch.jobs.data_ptr(), dbatch.n_jobs, dbatch.max_cand, tile,
                                   pool.source_bits.data_ptr(), pool.source_bbox.data_ptr(),
                                   dbatch.xform.data_ptr(), pcd_ws.data_ptr(), pcd_count.data_ptr(), hom_ws.data_ptr(),
                                   tmap_ptr, n_tiles,
                                   proj_bits.data_ptr(), proj_popc.data_ptr(), proj_bbox.data_ptr(), out_mode, stream),
                   "a3d_project")
        _lib.check(lib.a3d_score(H, W, dbatch.jobs.data_ptr(), dbatch.n_jobs, dbatch.max_tgt, dbatch.max_cand, nt,
                                 len(pool), nc, pool.bits.data_ptr(), pool.popc.data_ptr(), pool.bbox.data_ptr(),
                                 dbatch.tgt_index.data_ptr(), proj_bits.data_ptr(), proj_popc.data_ptr(),
                                 proj_bbox.data_ptr(), key_ws.data_ptr(),
                                 inter_tab.data_ptr() if inter_tab is not None else None,
                                 best_cand.data_ptr(), best_inter.data_ptr(), best_union.data_ptr(),
                                 best_iou.data_ptr(), stream), "a3d_score")
    return PassResult(best_cand, best_inter, best_union, best_iou, proj_bits, proj_popc, proj_bbox, inter_tab,
                      results, rows_only)


def emit_masks(bits: torch.Tensor, index: torch.Tensor | None, H: int, W: int,
               dtype=torch.float32) -> torch.Tensor:
    """Dense (n, H, W) images of selected packed masks (``reg_masks``)."""
    lib = _lib.load()
    _require_cuda(bits, "bits")
    n = int(index.numel()) if index is not None else int(bits.shape[0])
    out = torch.empty(n, H, W, dtype=dtype, device=bits.device)
    code = {torch.float32: _lib.A3D_F32, torch.uint8: _lib.A3D_U8}[dtype]
    with torch.cuda.device(bits.device):
        for lo in range(0, n, 65535):
            hi = min(n, lo + 65535)
            idx_ptr = index[lo:hi].data_ptr() if index is not None else None
            src = bits if index is not None else bits[lo:hi]
            _lib.check(lib.a3d_emit_masks(src.data_ptr(), idx_ptr, hi - lo, H, W, code,
                                          out[lo:hi].data_ptr(), _stream_ptr()), "a3d_emit_masks")
    return out


def rle_to_pool(rles, H: int, W: int, device) -> MaskPool:
    """COCO RLE dicts -> MaskPool, decoded on the device straight into packed bits
    (no dense mask is ever materialised).  ``rles``: sequence of
    ``{'size': [H, W], 'counts': bytes | str | list}``."""
    from . import rle as _rle
    lib = _lib.load()
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.A3DError("rle_to_pool needs a CUDA device (the hot path has no CPU fallback)")
    for r in rles:
        if list(r["size"]) != [H, W]:
            raise ValueError(f"RLE size {r['size']} != {[H, W]}")
    n = len(rles)
    if n and all(isinstance(r["counts"], (bytes, str)) for r in rles):
        # compressed strings (what the reference's records hold): all masks in one call of the host helper
        flat, begin, sums = _rle.strings_to_counts([r["counts"] for r in rles])
        if not np.all(sums == H * W):
            raise ValueError("RLE run lengths do not cover the mask")
    else:
        runs = []
        for r in rles:
            c = _rle.rle_counts(r)
            if int(c.astype(np.int64).sum()) != H * W:
                raise ValueError("RLE run lengths do not cover the mask")
            runs.append(c)
        begin = np.zeros(n + 1, dtype=np.int64)
        begin[1:] = np.cumsum([len(c) for c in runs])
        flat = np.concatenate(runs).astype(np.uint32) if n else np.zeros(0, np.uint32)
    pitch = _lib.pitch_words(W)
    with torch.cuda.device(device):
        d_counts = torch.from_numpy(flat.view(np.int32)).to(device)
        d_begin = torch.from_numpy(begin).to(device)
        bits = torch.empty(n, H, pitch, dtype=torch.int32, device=device)
        _lib.check(lib.a3d_rle_to_bits(d_counts.data_ptr(), d_begin.data_ptr(), n, H, W, bits.data_ptr(),
                                       _stream_ptr()), "a3d_rle_to_bits")
    return pool_from_bits(bits, H, W)


def plane_offsets(pool: MaskPool, inst_mask: torch.Tensor, normals: torch.Tensor, rays: torch.Tensor,
                  depth: torch.Tensor | None = None, inst_frame: torch.Tensor | None = None):
    """Per instance: mean over its mask of ``normal . (rays * depth)`` and the pixel count.

    rays (3,H,W) fp32; depth (F,H,W) fp32 or None (``rays`` already holds XYZ);
    inst_mask / inst_frame (n,) int32; normals (n,3) fp32.  All on the device."""
    lib = _lib.load()
    for t, name in ((pool.bits, "pool"), (inst_mask, "inst_mask"), (normals, "normals"), (rays, "rays")):
        _require_cuda(t, name)
    n = int(inst_mask.numel())
    dev = pool.bits.device
    off = torch.empty(n, dtype=torch.float32, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev)
    rays = rays.contiguous().float()
    normals = normals.contiguous().float()
    inst_mask = inst_mask.contiguous().to(torch.int32)
    if depth is not None:
        depth = depth.contiguous().float()
        inst_frame = inst_frame.contiguous().to(torch.int32)
    with torch.cuda.device(dev):
        _lib.check(lib.a3d_plane_offsets(depth.data_ptr() if depth is not None else None, rays.data_ptr(),
                                         pool.H, pool.W, pool.bits.data_ptr(), pool.bbox.data_ptr(),
                                         inst_mask.data_ptr(),
                                         inst_frame.data_ptr() if depth is not None else None,
                                         normals.data_ptr(), n, off.data_ptr(), cnt.data_ptr(), _stream_ptr()),
                   "a3d_plane_offsets")
    return off, cnt
