"""Host side of the drop-in `diff_gaussian_rasterization` replacement.

Mirrors the Python surface of DreamScene's un-vendored extension exactly as DreamScene uses it
(/root/reference/scene_gaussian.py:586-601,637-646 [score], :737-752,861-870 [scene],
:951-966,1012-1021 [object]):

    GaussianRasterizationSettings(image_height, image_width, tanfovx, tanfovy, bg,
        scale_modifier, viewmatrix, projmatrix, sh_degree, campos, prefiltered, score_flag)
    GaussianRasterizer(raster_settings)(means3D, means2D, opacities, shs, colors_precomp,
        scales, rotations, cov3D_precomp)
      -> (color[3,H,W], radii[P] int32, depth_alpha[2,H,W])                    score_flag False
      -> (important_score[P], color, radii, depth_alpha)                        score_flag True

All compute happens in libb200gsr.so (hand-written sm_100a CUDA) through the C ABI of
include/b200gsr.h; PyTorch provides device memory, the stream and autograd plumbing only.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

from . import _lib
from . import parallel as _parallel


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool = False
    score_flag: bool = False


# ------------------------------------------------------------------------------------------
# Workspaces.  Per DEVICE: the pair-capacity high-water mark, the pinned device-mapped notify ring
# and the deferred overflow checks.  Per (device, stream): one transient scratch buffer.
# ------------------------------------------------------------------------------------------
_MIN_CAPACITY = 1 << 20
_MIN_PAIRS_PER_GAUSSIAN = 4
_POLL_TIMEOUT_S = 60.0
_NOTIFY_SLOTS = 256


class PairCapacityOverflow(RuntimeError):
    """Raised (asynchronous mode only) when an EARLIER forward produced more (tile, Gaussian) pairs
    than its key buffer could hold: that call's images and gradients are invalid."""


class _Device:
    def __init__(self, device: torch.device):
        self.device = device
        self.capacity = 0            # largest pair capacity in use (fallback inside CUDA-graph capture)
        self.caps: dict = {}         # shape key (P, H, W) / (B, P, H, W) -> measured capacity (only ever grows);
                                     # a shape seen for the first time is measured synchronously
        self.user_capacity = False   # set by set_workspace_capacity: trust it, never wait on it
        self.last_pairs = 0          # pair count of the most recent RESOLVED forward
        self.seq = 0
        self.notify: Optional[torch.Tensor] = None   # int32[_NOTIFY_SLOTS, 4] pinned, device-mapped
        self.notify_np = None
        self.free_slots: list = []
        self.pending: list = []      # [(slot, seq, capacity)] forwards whose pair count is not read yet
        self.scratch: dict = {}      # stream handle -> uint8 tensor

    def ensure_notify(self):
        if self.notify is None:
            self.notify = torch.zeros(_NOTIFY_SLOTS, 4, dtype=torch.int32).pin_memory()
            self.notify_np = self.notify.numpy()      # shares the pinned pages: plain loads, no tensor ops
            self.free_slots = list(range(_NOTIFY_SLOTS - 1, -1, -1))

    def ensure_scratch(self, stream: int, nbytes: int) -> torch.Tensor:
        t = self.scratch.get(stream)
        if t is None or t.numel() < nbytes:
            t = self.scratch[stream] = torch.empty(int(nbytes * 1.1) + 4096, dtype=torch.uint8, device=self.device)
        return t

    def next_seq(self) -> int:
        self.seq = (self.seq + 1) & 0x7FFFFFFF or 1
        return self.seq


_devices: dict = {}
_pair_mode = os.environ.get("B200GSR_PAIR_MODE", "async")


def _device_state(device: torch.device) -> _Device:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    d = _devices.get(idx)
    if d is None:
        d = _devices[idx] = _Device(torch.device("cuda", idx))
    return d


def set_pair_count_mode(mode: str) -> None:
    """How forward learns the (tile, Gaussian) pair count D that sizes the sorted key buffer.

    "sync"  : after enqueueing all kernels the host waits for the tile scan (the first ~10% of the
              forward) to report D through a device-mapped host word and transparently re-issues the
              call if D exceeded the capacity.  Always exact; same stream-position sync as upstream's
              num_rendered D2H copy.
    "async" : (default) no host wait at all.  The capacity is 2x the largest D seen on the device
              (at least 4 pairs per Gaussian); the count of every forward is read lazily - without
              blocking - at later API calls, and an overflow (practically impossible with that
              head-room) raises PairCapacityOverflow then.  The first forward with a new (P, H, W)
              - a new scene, a densification step - measures its capacity synchronously, unless
              set_workspace_capacity was called.
    Also settable with the environment variable B200GSR_PAIR_MODE."""
    global _pair_mode
    if mode not in ("sync", "async"):
        raise ValueError("mode must be 'sync' or 'async'")
    _pair_mode = mode


def set_workspace_capacity(max_pairs: int, device=None) -> None:
    """Optional: pre-size the (tile, Gaussian) pair capacity of a device (required before capturing
    the rasterizer into a CUDA graph on a device that has not rendered eagerly yet)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    d = _device_state(dev)
    d.capacity = int(max_pairs)
    d.user_capacity = True


def _round_cap(n: int) -> int:
    g = 1 << 18
    return max(_MIN_CAPACITY, (int(n) + g - 1) // g * g)


def _resolve_pending(d: _Device, block: bool = False) -> None:
    """Read the pair counts the device has reported so far (never waits unless `block`)."""
    if not d.pending:
        return
    n = d.notify_np
    still, overflow = [], None
    t0 = time.perf_counter()
    for slot, seq, cap, key in d.pending:
        while block and int(n[slot, 0]) != seq:
            if time.perf_counter() - t0 > _POLL_TIMEOUT_S:
                torch.cuda.synchronize(d.device)
                if int(n[slot, 0]) != seq:
                    raise RuntimeError("b200gsr: device never reported a pair count")
        if int(n[slot, 0]) != seq:
            still.append((slot, seq, cap, key))
            continue
        pairs = int(n[slot, 1]) & 0xFFFFFFFF
        d.free_slots.append(slot)
        d.last_pairs = pairs
        d.capacity = max(d.capacity, _round_cap(2 * pairs))
        if key is not None and not d.user_capacity:
            d.caps[key] = max(d.caps.get(key, 0), _round_cap(2 * pairs))
        if pairs > cap:
            overflow = (pairs, cap)
    d.pending = still
    if overflow is not None:
        raise PairCapacityOverflow(
            f"b200gsr: an earlier forward produced {overflow[0]} (tile, Gaussian) pairs but its key buffer held "
            f"{overflow[1]}; its images/gradients are invalid. The capacity has been raised to {d.capacity}; "
            "re-run the step, or call set_workspace_capacity()/set_pair_count_mode('sync').")


def flush_checks(device=None) -> None:
    """Wait for every forward issued so far to report its pair count (raises on overflow)."""
    want = None
    if device is not None:
        dv = torch.device(device)
        want = dv.index if dv.index is not None else torch.cuda.current_device()
    for idx, d in list(_devices.items()):
        if want is None or idx == want:
            _resolve_pending(d, block=True)


def last_pair_count(device=None) -> int:
    """Pair count D of the most recent forward on the device (waits for it to be reported)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    d = _device_state(dev)
    _resolve_pending(d, block=True)
    return d.last_pairs


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _f32c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    t = t.contiguous()
    if t.data_ptr() % 16:          # the kernels use 16-byte vector loads on rows
        t = t.clone()
    return t


def _const(t: torch.Tensor, dev) -> torch.Tensor:
    # per-view constants live on the Gaussians' device (upstream requires CUDA tensors here too)
    if t.device != dev or t.dtype != torch.float32 or not t.is_contiguous() or t.requires_grad:
        t = t.detach().to(dev, torch.float32).contiguous()
    return t


def _make_params(rs: GaussianRasterizationSettings, P: int, M: int, keep: list, dev) -> _lib.Params:
    bg, vm, pm, cp = _const(rs.bg, dev), _const(rs.viewmatrix, dev), _const(rs.projmatrix, dev), _const(rs.campos, dev)
    keep.extend([bg, vm, pm, cp])
    return _lib.Params(P, M, int(rs.sh_degree), int(rs.image_height), int(rs.image_width),
                       float(rs.tanfovx), float(rs.tanfovy), float(rs.scale_modifier),
                       int(bool(rs.prefiltered)), int(bool(rs.score_flag)),
                       bg.data_ptr(), vm.data_ptr(), pm.data_ptr(), cp.data_ptr())


class _State:
    """Everything backward needs that is not a tensor input."""
    __slots__ = ("params_keep", "P", "M", "capacity", "saved", "rs", "with_backward", "prm")


_layout_cache: dict = {}


def _layouts(P, H, W, cap, with_backward):
    key = (P, H, W, cap, with_backward)
    r = _layout_cache.get(key)
    if r is None:
        if len(_layout_cache) > 256:
            _layout_cache.clear()
        r = _layout_cache[key] = (_lib.scratch_layout(P, H, W, cap).total,
                                  _lib.saved_layout(P, H, W, cap, with_backward).total)
    return r


def _issue_with_capacity(d: _Device, dev, key, P_eff: int, H_eff: int, W: int, with_backward: bool, score, launch):
    """The pair-capacity protocol shared by the single- and multi-view forwards.  `launch(cap, scratch,
    saved, notify_ptr, seq)` enqueues the whole forward and returns the C return code; this helper
    sizes the buffers, decides whether to wait for the device's pair count (sync mode / unknown
    capacity) and re-issues on overflow.  -> (saved tensor, capacity)."""
    capturing = torch.cuda.is_current_stream_capturing()
    stream_h = torch.cuda.current_stream(dev).cuda_stream
    measured = d.capacity if d.user_capacity else d.caps.get(key, 0)
    known = measured > 0
    if capturing and not known and d.capacity > 0:
        known, measured = True, d.capacity      # cannot wait inside a capture: trust the device's high-water mark
    if capturing and not known:
        raise RuntimeError("b200gsr: capturing into a CUDA graph needs a known pair capacity: run one eager "
                           "forward on this device first or call set_workspace_capacity()")
    cap = _round_cap(max(measured, _MIN_PAIRS_PER_GAUSSIAN * P_eff)) if known else _round_cap(6 * P_eff)
    # wait for the count only when it is needed: sync mode, or the capacity is a blind first guess
    wait = (not capturing) and (_pair_mode == "sync" or not known)
    while True:
        scratch_bytes, saved_bytes = _layouts(P_eff, H_eff, W, cap, with_backward)
        scratch = d.ensure_scratch(stream_h, scratch_bytes)
        saved = torch.empty(saved_bytes, dtype=torch.uint8, device=dev)
        slot, seq, notify_ptr = -1, 0, None
        if not capturing:
            if not d.free_slots:
                _resolve_pending(d, block=True)
            slot, seq = d.free_slots.pop(), d.next_seq()
            notify_ptr = C.c_void_p(d.notify.data_ptr() + 16 * slot)
        rc = launch(cap, scratch, saved, notify_ptr, seq)
        if rc:
            if slot >= 0:
                d.free_slots.append(slot)
            msg = _lib.last_error()
            if rc == -1:
                raise Exception(msg)
            raise RuntimeError(f"b200gsr_forward failed ({rc}): {msg}")
        if capturing:
            break
        if not wait:
            d.pending.append((slot, seq, cap, key))  # resolved lazily, never blocks the host
            break
        # Wait only for the tile scan (project + count + scan kernels); sort/composite keep running.
        t0 = time.perf_counter()
        n = d.notify_np
        while int(n[slot, 0]) != seq:
            if time.perf_counter() - t0 > _POLL_TIMEOUT_S:
                torch.cuda.synchronize(dev)
                if int(n[slot, 0]) == seq:
                    break
                raise RuntimeError("b200gsr_forward: device never reported the pair count")
        pairs = int(n[slot, 1]) & 0xFFFFFFFF
        d.free_slots.append(slot)
        d.last_pairs = pairs
        if pairs <= cap:
            # high-water mark with 2x head-room: capacity only costs 8 B per pair in `saved`, and
            # views of one training step differ a lot in pair count (random cameras).  A new
            # shape starts its own high-water mark.
            if not d.user_capacity:
                d.caps[key] = max(d.caps.get(key, 0), _round_cap(2 * pairs))
                d.capacity = max(d.capacity, d.caps[key])
                if len(d.caps) > 64:                 # densification changes P every 100 steps: keep the table small
                    for k in list(d.caps)[:-32]:
                        del d.caps[k]
            break
        cap = _round_cap(2 * pairs)                  # overflow: re-issue with enough room
        d.capacity = max(d.capacity, cap)
        if score is not None:
            score.zero_()
    return saved, cap


def _forward_impl(rs, means3D, shs, colors, opac, scales, rots, cov3d, with_backward=True):
    lib = _lib.load()
    dev = means3D.device
    if dev.type != "cuda":
        raise RuntimeError("diff_gaussian_rasterization (b200gsr): inputs must be CUDA tensors; "
                           "there is no CPU fallback")
    P = int(means3D.shape[0])
    M = int(shs.shape[1]) if shs is not None else 0
    H, W = int(rs.image_height), int(rs.image_width)
    d = _device_state(dev)
    if not torch.cuda.is_current_stream_capturing():
        d.ensure_notify()
        _resolve_pending(d)               # non-blocking: may raise PairCapacityOverflow for an earlier call
    keep: list = []
    with torch.cuda.device(dev):          # the library launches on the CURRENT device; restored on exit
        prm = _make_params(rs, P, M, keep, dev)
        color = torch.empty(3, H, W, dtype=torch.float32, device=dev)
        depth_alpha = torch.empty(2, H, W, dtype=torch.float32, device=dev)
        radii = torch.empty(P, dtype=torch.int32, device=dev)
        score = torch.zeros(P, dtype=torch.float32, device=dev) if rs.score_flag else None
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        flags = 0 if with_backward else _lib.FWD_NO_BACKWARD

        def launch(cap, scratch, saved, notify_ptr, seq):
            return lib.b200gsr_forward(C.byref(prm), _ptr(means3D), _ptr(shs), _ptr(colors), _ptr(opac),
                                       _ptr(scales), _ptr(rots), _ptr(cov3d), _ptr(color), _ptr(depth_alpha),
                                       _ptr(radii), _ptr(score), _ptr(scratch), scratch.numel(), _ptr(saved),
                                       saved.numel(), cap, flags, notify_ptr, seq, stream)

        saved, cap = _issue_with_capacity(d, dev, (P, H, W), P, H, W, with_backward, score, launch)
    st = _State()
    st.params_keep = keep; st.P = P; st.M = M; st.capacity = cap; st.saved = saved; st.rs = rs
    st.with_backward = with_backward
    st.prm = prm                      # the backward reuses the struct (its device pointers are kept alive by `keep`)
    return color, radii, depth_alpha, score, st


def grad_sections(P: int, n_col: int, has_sr: bool):
    """Offsets (in floats) of the parameter-gradient sections inside the flat buffer that backward
    fills and (under view sharding) all-reduces: means3D[P,3], opac[P,1], col[P,n_col], then
    scales[P,3]+rots[P,4] or cov[P,6].  Every section starts on a 256-byte boundary because the
    kernels use 16-byte vector stores.  Returns (offsets dict, total floats)."""
    widths = [("means3D", 3), ("opac", 1), ("col", n_col)] + ([("scales", 3), ("rots", 4)] if has_sr else [("cov", 6)])
    offs, o = {}, 0
    for name, wdt in widths:
        offs[name] = o
        o += (P * wdt + 63) // 64 * 64
    return offs, o


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                cov3Ds_precomp, raster_settings):
        means3D = _f32c(means3D); sh = _f32c(sh); colors_precomp = _f32c(colors_precomp)
        opacities = _f32c(opacities); scales = _f32c(scales); rotations = _f32c(rotations)
        cov3Ds_precomp = _f32c(cov3Ds_precomp)
        # under torch.no_grad() / with frozen inputs no backward can follow: skip the accumulators
        with_backward = any(ctx.needs_input_grad)
        color, radii, depth_alpha, score, st = _forward_impl(
            raster_settings, means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
            with_backward=with_backward)
        ctx.st = st
        ctx.has = (sh is not None, colors_precomp is not None, scales is not None, cov3Ds_precomp is not None)
        tensors = [means3D, opacities, radii, depth_alpha]
        for t in (sh, colors_precomp, scales, rotations, cov3Ds_precomp):
            tensors.append(t if t is not None else torch.empty(0, device=means3D.device))
        ctx.save_for_backward(*tensors)
        ctx.mark_non_differentiable(radii)
        ctx.set_materialize_grads(False)     # no zeros_like(radii) fill kernel per backward: absent grads arrive as None
        if raster_settings.score_flag:
            ctx.mark_non_differentiable(score)
            return score, color, radii, depth_alpha
        return color, radii, depth_alpha

    @staticmethod
    def backward(ctx, *grads):
        st = ctx.st
        rs = st.rs
        if rs.score_flag:
            _, g_color, _, g_da = grads
        else:
            g_color, _, g_da = grads
        means3D, opacities, radii, depth_alpha, sh, colors, scales, rots, cov3d = ctx.saved_tensors
        has_sh, has_col, has_sr, has_cov = ctx.has
        sh = sh if has_sh else None; colors = colors if has_col else None
        scales = scales if has_sr else None; rots = rots if has_sr else None
        cov3d = cov3d if has_cov else None
        dev = means3D.device
        P, M = st.P, st.M
        H, W = int(rs.image_height), int(rs.image_width)
        g_color = torch.zeros(3, H, W, device=dev) if g_color is None else _f32c(g_color)
        g_da = torch.zeros(2, H, W, device=dev) if g_da is None else _f32c(g_da)

        # one flat buffer for every parameter gradient.  Under view sharding (dreamscene_b200.parallel,
        # mode "backward") it is all-reduced in one call after the backward kernels, and the SH section
        # holds only the active degree's coefficients (the payload at sh_degree 0 is 14 instead of 59
        # floats per Gaussian); otherwise it is simply one allocation.
        reduce = P > 0 and _parallel.reduction_active()
        ncoef = (int(rs.sh_degree) + 1) ** 2
        # factored: the SH gradient leaves the kernel as dL/dcolour [P, 3] and is exchanged by all-gather
        factored = reduce and has_sh and _parallel.factored_sh_exchange()
        compact = reduce and has_sh and ncoef < M and not factored
        n_col = 0 if factored else ((3 * ncoef if compact else 3 * M) if has_sh else 3)
        offs, o = grad_sections(P, n_col, has_sr)
        flat = torch.empty(max(o, 1), dtype=torch.float32, device=dev)
        widths = {"means3D": 3, "opac": 1, "col": n_col, "scales": 3, "rots": 4, "cov": 6}
        sec = lambda name: flat[offs[name]:offs[name] + P * widths[name]]
        d_means3D = sec("means3D").view(P, 3)
        d_opac = sec("opac").view(P, 1)
        d_colsh = sec("col")
        if factored:
            d_sh = torch.empty(_parallel.factored_stride(P), dtype=torch.float32, device=dev)   # [P,3] + camera centre
        else:
            d_sh = d_colsh.view(P, n_col // 3, 3) if has_sh else None
        d_colors = d_colsh.view(P, 3) if has_col else None
        if has_sr:
            d_scales = sec("scales").view(P, 3)
            d_rots = sec("rots").view(P, 4)
            d_cov = None
        else:
            d_scales = d_rots = None
            d_cov = sec("cov").view(P, 6)
        d_means2D = torch.empty(P, 3, dtype=torch.float32, device=dev)

        if P > 0:
            lib = _lib.load()
            if not st.with_backward:
                raise RuntimeError("b200gsr: backward through a forward that ran without gradient accumulators")
            if not torch.cuda.is_current_stream_capturing():
                _resolve_pending(_device_state(dev))      # non-blocking overflow check of earlier forwards
            with torch.cuda.device(dev):
                prm = st.prm
                stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

                rc = lib.b200gsr_backward_ex(
                    C.byref(prm), _ptr(means3D), _ptr(sh), _ptr(colors), _ptr(opacities), _ptr(scales),
                    _ptr(rots), _ptr(cov3d), _ptr(radii), _ptr(depth_alpha), _ptr(g_color), _ptr(g_da),
                    _ptr(st.saved), st.saved.numel(), None, 0, st.capacity,
                    _ptr(d_means3D), _ptr(d_means2D), _ptr(d_sh), _ptr(d_colors), _ptr(d_opac),
                    _ptr(d_scales), _ptr(d_rots), _ptr(d_cov),
                    -1 if factored else (ncoef if compact else 0), stream)
                if rc:
                    raise RuntimeError(f"b200gsr_backward failed ({rc}): {_lib.last_error()}")
                if factored:
                    d_sh[3 * P:3 * P + 3].copy_(_const(rs.campos, dev).reshape(3))
                    d_sh = _parallel.exchange_factored(flat[:o], d_sh, P, M, int(rs.sh_degree), means3D)
                elif reduce:
                    _parallel.maybe_all_reduce(flat[:o] if o > 0 else flat)      # ONE ncclAllReduce of the flat buffer
            if compact:                      # expand to the reference layout [P, M, 3] (zeros above the degree)
                full = torch.zeros(P, M, 3, dtype=torch.float32, device=dev)
                full[:, :ncoef] = d_sh
                d_sh = full
        return (d_means3D, d_means2D, d_sh, d_colors, d_opac, d_scales, d_rots, d_cov, None)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                        cov3Ds_precomp, raster_settings):
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales,
                                     rotations, cov3Ds_precomp, raster_settings)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings: GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions: torch.Tensor) -> torch.Tensor:
        """Frustum (near-plane) visibility mask; unused by DreamScene, kept for API parity."""
        rs = self.raster_settings
        with torch.no_grad():
            pos = _f32c(positions)
            vis = torch.empty(pos.shape[0], dtype=torch.uint8, device=pos.device)
            vm, pm = _const(rs.viewmatrix, pos.device), _const(rs.projmatrix, pos.device)
            with torch.cuda.device(pos.device):
                rc = _lib.load().b200gsr_mark_visible(
                    int(pos.shape[0]), _ptr(pos), _ptr(vm), _ptr(pm), _ptr(vis),
                    C.c_void_p(torch.cuda.current_stream(pos.device).cuda_stream))
            if rc:
                raise RuntimeError(f"b200gsr_mark_visible failed ({rc}): {_lib.last_error()}")
        return vis.bool()

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None,
                rotations=None, cov3D_precomp=None):
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception("Please provide excatly one of either SHs or precomputed colors!")
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")
        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                   cov3D_precomp, self.raster_settings)
