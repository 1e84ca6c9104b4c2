"""View-sharded data parallelism (SURVEY.md section 8e).

DreamScene renders the C_batch_size views of a step sequentially on one GPU and lets autograd
sum the per-view parameter gradients (/root/reference/training/scene_trainer.py:801-829,881).
Here each rank renders its own views with replicated Gaussian parameters and the per-view gradients
are summed over NCCL/NVLink.  Two ways to do the sum, both additive to the reference API:

1. ``all_reduce_gradients(params)`` after ``loss.backward()``  (DDP-style, ALWAYS exact).
   One coalesced NCCL all-reduce over the leaf ``.grad`` tensors.  Correct for any graph between the
   parameters and the rasterizer - in particular for the per-call random scale/SH augmentation of
   ``scene_render`` (/root/reference/scene_gaussian.py:848-856), where every rank back-propagates
   through its OWN random Jacobian.  Columns that are identically zero on every rank (SH
   coefficients above the active degree: ``sh_degree`` starts at 0 and rises every 500 steps,
   /root/reference/training/object_trainer.py:243-244) can be left out of the payload.

2. ``enable_view_sharding(mode="backward")``: the rasterizer's backward all-reduces its flat
   parameter-gradient buffer itself (ONE ncclAllReduce, no staging copy) and sends only the active
   degree's SH columns.  Pipelining that reduction over Gaussian ranges, overlapping finished ranges
   with the per-Gaussian backward of the rest, was measured on 4 x B200 to lose (1.82 vs 1.44 ms/step
   at 8 ranges: 40 small collectives cost more than the 0.14 ms of project_bwd they can hide;
   profiles/r02_scale_probe.md).
   By default the SH gradient is not all-reduced at all: dL/dsh of a view is basis(view direction) x
   dL/dcolour, so the ranks all-gather 3 floats per Gaussian (+ their camera centre) and rebuild the summed
   [P, M, 3] rows locally (``exchange_factored``; sh_exchange="dense" restores the row all-reduce).
   This mode reduces the gradient AT THE RASTERIZER INPUTS, so it equals the sequential sum
   only when the map parameters -> rasterizer inputs is the same deterministic function on every
   rank (inputs are leaves, or activations without per-rank randomness).  Every rank must issue the
   same sequence of rasterizer backward calls with the same P; set B200GSR_CHECK_COLLECTIVES=1 to
   verify that at run time.  ``no_sync()`` suspends the in-backward reduction (a rank that renders several
   local views per step accumulates them in the leaves and calls ``all_reduce_gradients`` once).

Per-view quantities (means2D grad, radii, visibility) are NOT reduced, as in the reference, which only
uses the last view's (training/object_trainer.py:385-390).
"""
from __future__ import annotations

import contextlib
import os
from typing import Iterable, Optional

import torch
import torch.distributed as dist

_group = None
_enabled = False
_sh_exchange = "factored"
_suspended = 0
MAX_FACTORED_VIEWS = 64          # b200gsr_sh_grad_expand
_CHECK = bool(int(os.environ.get("B200GSR_CHECK_COLLECTIVES", "0")))


def enable_view_sharding(group: Optional["dist.ProcessGroup"] = None, mode: str = "backward",
                         sh_exchange: str = "factored") -> None:
    """mode="backward": every rasterizer backward all-reduces its parameter gradients (see the module
    docstring for when that is exact); mode="deferred": nothing happens inside backward, call
    all_reduce_gradients() yourself.  sh_exchange="factored" (default, SH inputs): the SH gradient
    is exchanged as 3 floats per Gaussian and view and rebuilt on every rank; "dense": all-reduced as rows."""
    global _group, _enabled, _sh_exchange
    if not dist.is_initialized():
        raise RuntimeError("torch.distributed is not initialised")
    if mode not in ("backward", "deferred"):
        raise ValueError("mode must be 'backward' or 'deferred'")
    if sh_exchange not in ("factored", "dense"):
        raise ValueError("sh_exchange must be 'factored' or 'dense'")
    _group, _enabled, _sh_exchange = group, mode == "backward", sh_exchange


def disable_view_sharding() -> None:
    global _group, _enabled
    _group, _enabled = None, False


def is_enabled() -> bool:
    return _enabled


@contextlib.contextmanager
def no_sync():
    """Suspend the in-backward reduction (accumulate several local views, reduce with the last)."""
    global _suspended
    _suspended += 1
    try:
        yield
    finally:
        _suspended -= 1


def reduction_active() -> bool:
    return _enabled and _suspended == 0 and dist.is_initialized() and dist.get_world_size(_group) > 1


def factored_sh_exchange() -> bool:
    """The in-backward reduction sends the SH gradient in factored form (see exchange_factored)."""
    return (reduction_active() and _sh_exchange == "factored"
            and dist.get_world_size(_group) <= MAX_FACTORED_VIEWS)


def factored_stride(P: int) -> int:
    """Floats per rank in the all-gathered buffer: [P, 3] colour gradients + camera centre, padded to 256 B."""
    return (3 * P + 3 + 63) // 64 * 64


def exchange_factored(flat: torch.Tensor, dcol: torch.Tensor, P: int, M: int, sh_degree: int,
                      means3D: torch.Tensor) -> torch.Tensor:
    """Reduction of one backward under view sharding with the SH gradient in factored form.

    dL/dsh of a view is the outer product basis(view direction of the Gaussian) x dL/d(clamped colour): instead
    of all-reducing [P, M, 3] rows (192 of the 236 bytes per Gaussian at M = 16) every rank contributes `dcol` =
    [P, 3] colour gradients + its camera centre, ONE all-gather hands everybody all of them, and
    b200gsr_sh_grad_expand rebuilds the summed rows locally (views in rank order: bit-identical on every rank).
    `flat` (means3D / opacity / scale / rotation gradients, 44 bytes per Gaussian) is all-reduced as before.
    Exact under the same condition as the dense in-backward reduction plus: all ranks pass the same means3D."""
    from . import _lib
    world = dist.get_world_size(_group)
    if _CHECK:
        _check_same_size(flat.numel() + dcol.numel(), flat.device)
    gathered = torch.empty(world, dcol.numel(), dtype=torch.float32, device=dcol.device)
    works = [dist.all_gather_into_tensor(gathered, dcol, group=_group, async_op=True)]
    if flat.numel() > 0:
        works.append(dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=_group, async_op=True))
    for w in works:
        w.wait()
    d_sh = torch.empty(P, M, 3, dtype=torch.float32, device=dcol.device)
    import ctypes as C
    with torch.cuda.device(dcol.device):
        rc = _lib.load().b200gsr_sh_grad_expand(
            P, M, int(sh_degree), world, C.c_void_p(means3D.data_ptr()), C.c_void_p(gathered.data_ptr()),
            dcol.numel(), C.c_void_p(d_sh.data_ptr()), C.c_void_p(torch.cuda.current_stream(dcol.device).cuda_stream))
    if rc:
        raise RuntimeError(f"b200gsr_sh_grad_expand failed ({rc}): {_lib.last_error()}")
    return d_sh


def _coalesced_all_reduce(tensors, group):
    """One NCCL group call for all tensors (ncclGroupStart/End); plain per-tensor calls on backends
    without coalescing support (gloo in the CPU tests).  Returns when the sums are in place."""
    if dist.get_backend(group) == "nccl":
        with dist._coalescing_manager(group=group, device=tensors[0].device, async_ops=False):
            for t in tensors:
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        return
    for t in tensors:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def _check_same_size(numel: int, device="cuda") -> None:
    t = torch.tensor([numel, -numel], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=_group)
    if int(t[0]) != numel or int(t[1]) != -numel:
        raise RuntimeError(f"view sharding: ranks disagree on the gradient buffer size ({numel} here, "
                           f"max {int(t[0])}, min {-int(t[1])}): every rank must render the same P")


def maybe_all_reduce(flat: torch.Tensor) -> None:
    """One all-reduce of a flat gradient buffer, when the in-backward reduction is active."""
    if reduction_active():
        if _CHECK:
            _check_same_size(flat.numel(), flat.device)
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=_group)


def all_reduce_gradients(params: Iterable[torch.Tensor], group: Optional["dist.ProcessGroup"] = None,
                         active_columns: Optional[dict] = None) -> None:
    """DDP-style: sum the leaf gradients over the ranks with ONE coalesced NCCL all-reduce.  Exact for
    any graph between parameters and rasterizer.  `active_columns` = {param: k}: only
    ``param.grad[:, :k]`` can be non-zero on any rank (e.g. features_rest [P, M-1, 3] with
    k = (sh_degree+1)^2 - 1), the rest is not sent."""
    if not dist.is_initialized() or dist.get_world_size(group) <= 1:
        return
    active_columns = active_columns or {}
    jobs = []          # (destination view or None, tensor handed to NCCL)
    for p in params:
        g = p.grad
        if g is None:
            continue
        k = active_columns.get(p)
        if k is not None and g.dim() >= 2 and k < g.shape[1]:
            if k > 0:
                jobs.append((g[:, :k], g[:, :k].contiguous()))       # packed copy of the active columns
        elif g.is_contiguous():
            jobs.append((None, g))                                     # reduced in place
        else:
            jobs.append((g, g.contiguous()))
    if not jobs:
        return
    tensors = [t for _, t in jobs]
    total = sum(t.numel() for t in tensors)
    if len(tensors) > 1 and total >= (1 << 20) and all(t.dtype == tensors[0].dtype for t in tensors):
        # one big message beats a group of medium ones (measured 4 x B200, 236 MB: 0.60 ms flat vs
        # 0.80 ms as five coalesced tensors): stage through a flat buffer (2 extra HBM passes, ~0.1 ms)
        flat = torch.cat([t.reshape(-1) for t in tensors])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        torch._foreach_copy_([t.reshape(-1) for t in tensors], list(flat.split([t.numel() for t in tensors])))
    else:
        _coalesced_all_reduce(tensors, group)
    for dst, t in jobs:
        if dst is not None:
            dst.copy_(t)


def shard_views(num_views: int, rank: Optional[int] = None, world: Optional[int] = None, allow_uneven: bool = False):
    """Views {rank, rank+world, ...} of a batch (scene_trainer.py:801 loop index i).  With the
    in-backward reduction every rank must own the same number of views (a collective per backward):
    uneven shards are refused unless allow_uneven (use mode="deferred" + all_reduce_gradients then)."""
    if rank is None:
        rank = dist.get_rank(_group) if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size(_group) if dist.is_initialized() else 1
    if num_views % world != 0 and not allow_uneven:
        raise ValueError(f"{num_views} views do not divide over {world} ranks: ranks would issue different numbers "
                         "of collectives; pad the batch or pass allow_uneven=True with mode='deferred'")
    return list(range(rank, num_views, world))
