"""bench.py --dump-outputs: --steps sets the number of timed steps, and the dumped arrays are what one
step of the workload returns through the public API on the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import util_scene as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_step_returns(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1_10k_256", "--steps", "3",
                          "--warmup", "1", "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3 * 9
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())

    sys.path.insert(0, ROOT)
    import bench
    from dreamscene_b200 import GaussianRasterizer
    wl = bench.WORKLOADS["cfg1_10k_256"]
    P = wl["P"]
    sc, cam, gc, gd = bench.make_scene(wl, 0)
    dev = torch.device("cuda", torch.cuda.current_device())
    idx = got["sample_index"].astype(np.int64)
    assert np.array_equal(idx, np.arange(P))              # fewer Gaussians than the sample size: every row
    p = {k: v.to(dev).requires_grad_(True) for k, v in sc.items()}
    m2d = torch.zeros(P, 3, device=dev, requires_grad=True)
    color, radii, da = GaussianRasterizer(U.cuda_settings(cam, 3, device=dev))(
        means3D=p["means3D"], means2D=m2d, opacities=p["opacities"], shs=p["shs"], scales=p["scales"],
        rotations=p["rotations"])
    torch.autograd.backward([color, da], [gc.to(dev), gd.to(dev)])
    np.testing.assert_array_equal(got["color"], color.detach().cpu().numpy())
    np.testing.assert_array_equal(got["depth_alpha"], da.detach().cpu().numpy())
    np.testing.assert_array_equal(got["radii"], radii.cpu().numpy().astype(np.float32))
    want = {k: v.grad for k, v in p.items()}
    want["means2D"] = m2d.grad
    for k, g in want.items():
        assert U.rel_err(torch.from_numpy(got[f"grad_{k}"]), g.cpu()) < 1e-5, k
