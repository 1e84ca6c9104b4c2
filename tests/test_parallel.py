"""View-sharded data parallelism (SURVEY.md 8e): host logic on CPU with gloo (world_size 2), and
the real NCCL path on >= 2 GPUs (skipped on a 1-GPU box)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from dreamscene_b200 import parallel
    from oracle import splat_ref as O
    from tests import util_scene as U
    torch.set_num_threads(2)
    assert parallel.shard_views(6) == list(range(rank, 6, world))
    assert parallel.shard_views(5, allow_uneven=True) == list(range(rank, 5, world))
    try:
        parallel.shard_views(5)
        uneven_refused = False
    except ValueError:
        uneven_refused = True
    parallel.enable_view_sharding()
    # each rank differentiates ITS view with the oracle; the reduced gradient must equal the
    # sequential two-view sum that DreamScene's loop produces (scene_trainer.py:801-829,881)
    sc, _, deg = U.make_inputs(300, 48, 48, seed=21)
    grads = []
    for view in range(world):
        cam = U.cameras.orbit_camera(phi_deg=45.0 * view, height=48, width=48)
        S = U.oracle_settings(cam, deg)
        t = {k: v.clone().requires_grad_(True) for k, v in sc.items()}
        r = O.rasterize(S, t["means3D"], t["opacities"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
        (r["color"].sum() + r["depth_alpha"].sum()).backward()
        grads.append(torch.cat([t[k].grad.reshape(-1) for k in ("means3D", "opacities", "shs", "scales", "rotations")]))
    flat = grads[rank].clone()
    parallel.maybe_all_reduce(flat)
    ok = torch.allclose(flat, sum(grads), rtol=1e-5, atol=1e-7)
    parallel.disable_view_sharding()
    untouched = grads[rank].clone()
    parallel.maybe_all_reduce(untouched)
    ok = ok and torch.equal(untouched, grads[rank]) and uneven_refused
    # the factored SH exchange is the default of the in-backward reduction (<= 64 ranks)
    parallel.enable_view_sharding()
    ok = ok and parallel.factored_sh_exchange()
    parallel.enable_view_sharding(sh_exchange="dense")
    ok = ok and parallel.reduction_active() and not parallel.factored_sh_exchange()
    try:
        parallel.enable_view_sharding(sh_exchange="sparse")
        ok = False
    except ValueError:
        pass
    ok = ok and parallel.factored_stride(1000) == 3008 and parallel.factored_stride(21) % 64 == 0 \
        and parallel.factored_stride(21) >= 3 * 21 + 3
    # no_sync() suspends the in-backward reduction
    parallel.enable_view_sharding()
    with parallel.no_sync():
        ok = ok and not parallel.reduction_active()
        kept = grads[rank].clone()
        parallel.maybe_all_reduce(kept)
        ok = ok and torch.equal(kept, grads[rank])
    ok = ok and parallel.reduction_active()
    # DDP-style reduction of leaf gradients, with columns that are zero on every rank left out
    parallel.enable_view_sharding(mode="deferred")
    ok = ok and not parallel.reduction_active()
    a = torch.nn.Parameter(torch.zeros(7, 3)); b = torch.nn.Parameter(torch.zeros(7, 15, 3)); c = torch.nn.Parameter(torch.zeros(4))
    a.grad = torch.full((7, 3), float(rank + 1))
    b.grad = torch.zeros(7, 15, 3); b.grad[:, :3] = float(10 * (rank + 1))
    parallel.all_reduce_gradients([a, b, c], active_columns={b: 3})
    ok = ok and torch.equal(a.grad, torch.full((7, 3), 3.0)) and c.grad is None
    ok = ok and torch.equal(b.grad[:, :3], torch.full((7, 3, 3), 30.0)) and float(b.grad[:, 3:].abs().max()) == 0.0
    parallel.disable_view_sharding()
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_view_sharding_host_logic_without_chunking_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]


def _nccl_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      B200GSR_CHECK_COLLECTIVES="1")
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from dreamscene_b200 import GaussianRasterizer, parallel
    from tests import util_scene as U
    P = 20000
    sc, _, _ = U.make_inputs(P, 256, 256, seed=23)
    dev = torch.device("cuda", rank)
    names = ("means3D", "opacities", "shs", "scales", "rotations")
    results = {}

    def view_grads(view, deg, mode, noise_seed=None):
        """mode: 'factored' / 'dense' (in-backward reduction with that SH exchange), 'off' (no reduction),
        'deferred' (leaf grads reduced afterwards).  noise_seed: scene_render-style scale/SH augmentation
        between leaves and rasterizer."""
        cam = U.cameras.orbit_camera(phi_deg=45.0 * view, height=256, width=256)
        S = U.cuda_settings(cam, deg, device=dev)
        t = {k: v.to(dev).requires_grad_(True) for k, v in sc.items()}
        m2d = torch.zeros(P, 3, device=dev, requires_grad=True)
        if mode == "factored":
            parallel.enable_view_sharding()                          # default: factored SH exchange (all-gather + expand)
        elif mode == "dense":
            parallel.enable_view_sharding(sh_exchange="dense")       # one all-reduce of the flat buffer incl. SH rows
        elif mode == "deferred":
            parallel.enable_view_sharding(mode="deferred")
        else:
            parallel.disable_view_sharding()
        shs, scales = t["shs"], t["scales"]
        if noise_seed is not None:     # /root/reference/scene_gaussian.py:848-856
            g = torch.Generator(device=dev).manual_seed(noise_seed)
            shs = shs + torch.randn(shs.shape, generator=g, device=dev) * 0.05
            scales = torch.clamp(scales + torch.randn(scales.shape, generator=g, device=dev) * 0.3 * scales, 0.0)
        color, radii, da = GaussianRasterizer(S)(means3D=t["means3D"], means2D=m2d, opacities=t["opacities"],
                                                 shs=shs, scales=scales, rotations=t["rotations"])
        (color.sum() + da.sum()).backward()
        if mode == "deferred":
            ncoef = (deg + 1) ** 2
            parallel.all_reduce_gradients([t[k] for k in names], active_columns={t["shs"]: ncoef})
        return torch.cat([t[k].grad.reshape(-1) for k in names]), m2d.grad

    ok = True
    for deg in (3, 1, 0):       # degree < 3: only the active SH columns travel (compact payload)
        seq = sum(view_grads(v, deg, "off")[0] for v in range(world))       # sequential loop on one GPU
        _, m2d_seq = view_grads(rank, deg, "off")
        for mode in ("factored", "dense"):
            reduced, m2d_own = view_grads(rank, deg, mode)
            err = float((reduced - seq).norm() / seq.norm())
            # per-view means2D grads are NOT reduced (equal up to the fp32 atomic summation order)
            ok = ok and err < 1e-5 and float((m2d_own - m2d_seq).norm() / m2d_seq.norm()) < 1e-5
            results[f"{mode}_deg{deg}"] = err
            if mode == "factored":      # views are summed in rank order on every rank: bit-identical results
                both = [torch.empty_like(reduced) for _ in range(world)]
                dist.all_gather(both, reduced)
                ok = ok and all(torch.equal(both[0], b) for b in both)
    # per-rank random augmentation between leaves and rasterizer: only the DDP-style reduction of the
    # LEAF gradients reproduces the sequential sum (ADVICE r1)
    red, _ = view_grads(rank, 1, "deferred", noise_seed=100 + rank)
    seq = sum(view_grads(v, 1, "off", noise_seed=100 + v)[0] for v in range(world))
    err = float((red - seq).norm() / seq.norm())
    ok = ok and err < 1e-5
    results["deferred_augmented"] = err
    q.put((rank, ok, results))
    dist.destroy_process_group()


@pytest.mark.gpu
def test_view_sharded_backward_matches_sequential_sum_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs (run under gpurun --gpus 2)")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert all(r[1] for r in res), res


def test_sh_gradient_of_one_view_is_rank_one_per_gaussian_cpu_oracle():
    """The identity the factored SH exchange rests on (parallel.exchange_factored), checked on the CPU oracle's autograd:
    dL/dsh[i][k][c] = basis_k(direction of Gaussian i in this view) * dL/d(clamped colour)[i][c], and 0 above the active
    degree - so 3 floats per Gaussian and view (plus the camera centre) determine the whole [M, 3] row."""
    from oracle import splat_ref as O
    from tests import util_scene as U
    torch.set_num_threads(2)
    for deg in (3, 1):
        sc, _, _ = U.make_inputs(400, 48, 48, seed=31)
        cam = U.cameras.orbit_camera(phi_deg=70.0, height=48, width=48)
        S = U.oracle_settings(cam, deg)
        t = {k: v.clone().requires_grad_(True) for k, v in sc.items()}
        r = O.rasterize(S, t["means3D"], t["opacities"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
        g = torch.Generator().manual_seed(5)
        (r["color"] * torch.randn(r["color"].shape, generator=g)).sum().backward()
        d_sh = t["shs"].grad                                                    # [P, M, 3]
        P, M, ncoef = d_sh.shape[0], d_sh.shape[1], (deg + 1) ** 2
        d = sc["means3D"] - cam.camera_center.reshape(1, 3)
        d = d / d.norm(dim=1, keepdim=True)
        basis = torch.stack([O.eval_sh_basis_dot(deg, torch.nn.functional.one_hot(torch.full((P,), k), M)[:, :, None]
                                                 .expand(P, M, 3).float(), d)[:, 0] for k in range(ncoef)], dim=1)   # [P, ncoef]
        dcol = d_sh[:, 0, :] / basis[:, :1]                                     # basis_0 is the constant SH_C0
        rebuilt = basis[:, :, None] * dcol[:, None, :]
        touched = d_sh.abs().sum(dim=(1, 2)) > 0
        assert int(touched.sum()) > 50
        assert float((rebuilt - d_sh[:, :ncoef]).abs().max()) <= 1e-6 * float(d_sh.abs().max())
        assert float(d_sh[:, ncoef:].abs().max()) == 0.0 if ncoef < M else True
