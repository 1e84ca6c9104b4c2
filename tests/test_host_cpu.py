"""CPU-only checks: the C-ABI library loads and exports every symbol of include/b200gsr.h,
layout queries behave, argument errors surface, and the product path refuses to run on CPU."""
import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "b200gsr.h")).read()
    return sorted(set(re.findall(r"\b(b200gsr_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol_of_abi_v4():
    from dreamscene_b200 import _build, _lib
    _build.build()
    lib = _lib.load()
    syms = _declared_symbols()
    assert set(_lib.EXPORTS) == set(syms)
    for s in syms:
        assert hasattr(lib, s), s
    assert lib.b200gsr_version() == 4


def test_layout_queries_are_monotone_and_aligned():
    from dreamscene_b200 import _lib
    a = _lib.saved_layout(1000, 256, 256, 1 << 20)
    b = _lib.saved_layout(1000, 256, 256, 1 << 21)
    assert b.total > a.total and a.keys % 256 == 0 and a.geom % 256 == 0 and a.n_contrib % 256 == 0
    assert b.total - a.total == (1 << 20) * 8          # capacity only scales the 8-byte key list
    assert a.dgeom - a.geom >= 1000 * 48 and a.total - a.dgeom >= 1000 * 48
    nb = _lib.saved_layout(1000, 256, 256, 1 << 20, with_backward=False)
    assert nb.dgeom == a.dgeom and nb.total == nb.dgeom       # inference layout drops the accumulators
    s = _lib.scratch_layout(1000, 256, 256, 1 << 20)
    assert s.counters == 0 and s.tile_count < s.tile_cursor < s.rectdepth < s.ms_hist <= s.total
    with pytest.raises(RuntimeError):
        _lib.saved_layout(10, 16, 16, 1 << 33)


def test_forward_rejects_bad_arguments_without_a_gpu():
    from dreamscene_b200 import _lib
    lib = _lib.load()
    prm = _lib.Params(4, 16, 3, 32, 32, 0.3, 0.3, 1.0, 0, 0, 0, 0, 0, 0)
    rc = lib.b200gsr_forward(C.byref(prm), *([None] * 11), None, 0, None, 0, 1024, 0, None, 0, None)
    assert rc == -1 and "device pointers" in _lib.last_error()


def test_settings_surface_is_reference_compatible():
    import inspect
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    fields = GaussianRasterizationSettings._fields
    # scene_gaussian.py:586-599 passes exactly these keywords
    assert fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier",
                      "viewmatrix", "projmatrix", "sh_degree", "campos", "prefiltered", "score_flag")
    sig = inspect.signature(GaussianRasterizer.forward)
    assert list(sig.parameters)[1:] == ["means3D", "means2D", "opacities", "shs", "colors_precomp",
                                        "scales", "rotations", "cov3D_precomp"]


def test_cpu_tensors_fail_loudly_no_fallback():
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    S = GaussianRasterizationSettings(16, 16, 0.3, 0.3, torch.ones(3), 1.0, torch.eye(4), torch.eye(4), 0,
                                      torch.zeros(3), False, False)
    z = torch.zeros(4, 3)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        GaussianRasterizer(S)(means3D=z, means2D=z, opacities=torch.zeros(4, 1), shs=torch.zeros(4, 1, 3),
                              scales=z, rotations=torch.zeros(4, 4))


def test_product_never_imports_the_oracle():
    for pkg in ("dreamscene_b200", "diff_gaussian_rasterization"):
        for dp, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith(".py"):
                    src = open(os.path.join(dp, f)).read()
                    assert "oracle" not in src.replace("no oracle", ""), os.path.join(dp, f)


def test_gradient_sections_are_256_byte_aligned_for_any_point_count():
    from dreamscene_b200.rasterizer import grad_sections
    for P in (0, 1, 2, 3, 7, 1001, 1_000_000):
        for n_col, has_sr in ((48, True), (12, True), (3, False), (27, True)):
            offs, total = grad_sections(P, n_col, has_sr)
            widths = dict(means3D=3, opac=1, col=n_col, scales=3, rots=4, cov=6)
            names = list(offs)
            assert names[:3] == ["means3D", "opac", "col"] and (("rots" in offs) == has_sr) and (("cov" in offs) != has_sr)
            for a, b in zip(names, names[1:] + [None]):
                assert offs[a] % 64 == 0                               # 64 floats = 256 bytes
                end = offs[b] if b else total
                assert end - offs[a] >= P * widths[a]                  # sections never overlap


def test_pair_count_mode_switch_and_capacity_policy():
    from dreamscene_b200 import rasterizer as R
    assert R._pair_mode in ("sync", "async")
    old = R._pair_mode
    try:
        R.set_pair_count_mode("sync"); assert R._pair_mode == "sync"
        R.set_pair_count_mode("async"); assert R._pair_mode == "async"
        with pytest.raises(ValueError):
            R.set_pair_count_mode("maybe")
    finally:
        R.set_pair_count_mode(old)
    assert R._round_cap(1) == R._MIN_CAPACITY and R._round_cap((1 << 20) + 1) % (1 << 18) == 0


def test_deferred_overflow_check_reads_the_notify_ring_without_blocking():
    """The async pair-count protocol on the host side, with the device's writes faked."""
    import numpy as np
    from dreamscene_b200 import rasterizer as R
    d = R._Device(torch.device("cuda", 0))
    d.notify = torch.zeros(R._NOTIFY_SLOTS, 4, dtype=torch.int32)     # unpinned stand-in
    d.notify_np = d.notify.numpy()
    d.free_slots = list(range(R._NOTIFY_SLOTS - 1, -1, -1))
    s1, s2 = d.free_slots.pop(), d.free_slots.pop()
    d.pending = [(s1, 11, 1 << 20, (5, 16, 16)), (s2, 12, 1 << 20, (5, 16, 16))]
    R._resolve_pending(d)                       # nothing reported yet: stays pending, no wait
    assert len(d.pending) == 2
    d.notify_np[s1] = (11, 500_000, 0, 64)      # first forward reports 0.5M pairs
    R._resolve_pending(d)
    assert d.pending == [(s2, 12, 1 << 20, (5, 16, 16))] and d.last_pairs == 500_000 and s1 in d.free_slots
    assert d.capacity == R._round_cap(1_000_000) and d.caps[(5, 16, 16)] == R._round_cap(1_000_000)
    d.notify_np[s2] = (12, 3 << 20, 1, 64)      # second one overflowed its 1M-pair buffer
    with pytest.raises(R.PairCapacityOverflow):
        R._resolve_pending(d)
    assert not d.pending and d.capacity >= 6 << 20      # raised so that a retry fits


def test_shared_inline_helpers_native_check(tmp_path):
    """common.cuh helpers used by both host and device code (multisplit grid, backward size classes, tile grid):
    tests/native/common_check.cu is compiled with nvcc and run on the CPU."""
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path / "common_check")
    src = os.path.join(ROOT, "tests", "native", "common_check.cu")
    subprocess.run([nvcc, "-std=c++17", "-Wno-deprecated-gpu-targets", "-I", os.path.join(ROOT, "dreamscene_b200", "csrc"),
                    "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True, timeout=300)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "helpers ok" in out.stdout, out.stdout + out.stderr
