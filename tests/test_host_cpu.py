"""CPU-only tests: C-ABI library loads and exports every declared symbol, host-side module
surface mirrors the reference, and there is no CPU fallback."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "nerf_b200.h")).read()
    declared = set(re.findall(r"\b(nb200_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.nb200_version() >= 100 and lib.nb200_compiled_arch() == 100
    assert lib.nb200_error_string(-2) == b"unsupported shape or precision"


def test_state_dict_matches_reference(golden_weights):
    from nerf_simple_b200.nets import Nerf
    torch.manual_seed(0)
    net = Nerf()
    sd = net.state_dict()
    assert list(sd.keys()) == list(golden_weights.keys())
    for k, v in sd.items():
        # same construction order => identical default init for the same seed (utils/nets.py:16-32)
        assert np.array_equal(v.numpy(), golden_weights[k]), k
    net.load_state_dict({k: torch.from_numpy(v) for k, v in golden_weights.items()}, strict=True)
    assert net.Lp == 10 and net.Ld == 4
    with pytest.raises(NotImplementedError):
        Nerf(Lp=6)


def test_no_cpu_fallback(golden_weights):
    from nerf_simple_b200._lib import NerfB200Error
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.rendering import render_nerf, volume_render
    net = Nerf()
    with pytest.raises(NerfB200Error):
        net(torch.zeros(8, 6))
    with pytest.raises(NerfB200Error):
        render_nerf(torch.zeros(8, 6), net, 16)
    with pytest.raises(NerfB200Error):
        volume_render(torch.zeros(2, 8, 4), torch.zeros(2, 8), torch.zeros(2, 3))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "nerf_simple_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                assert "oracle" not in src.replace("CPU oracle", ""), os.path.join(dp, fn)


def test_camera_path_matches_reference():
    from conftest import load_golden
    from nerf_simple_b200.xyz import poses_to_render
    g = load_golden("case_raygen.npz")
    poses = torch.stack(poses_to_render(r=4, theta=-30, n_phi=30)).numpy()
    assert np.abs(poses - g["poses30"]).max() <= 1e-7


def test_dropin_module_surface():
    import importlib
    import sys
    sys.path.insert(0, os.path.join(ROOT, "nerf_simple_b200", "dropin"))
    try:
        for m in [k for k in sys.modules if k == "utils" or k.startswith("utils.")]:
            del sys.modules[m]
        nets = importlib.import_module("utils.nets")
        rendering = importlib.import_module("utils.rendering")
        xyz = importlib.import_module("utils.xyz")
        dataload = importlib.import_module("utils.dataload")
        for n in ("render_nerf", "volume_render", "render_image", "render_poses"):
            assert callable(getattr(rendering, n))
        for n in ("gamma", "positional_encoder", "rays_single_cam", "polar_to_mat", "phi_to_mat",
                  "spherical_to_pose", "poses_to_render"):
            assert callable(getattr(xyz, n))
        for n in ("load_data", "rays_dataset", "RayGenerator"):
            assert hasattr(dataload, n)
        assert nets.Nerf.__module__ == "nerf_simple_b200.nets"
    finally:
        sys.path.pop(0)
        for m in [k for k in sys.modules if k == "utils" or k.startswith("utils.")]:
            del sys.modules[m]


def test_flat_views_are_aligned_contiguous_views():
    """The flat parameter / gradient buffers of the trainer: every tensor is a contiguous view that starts on
    a 16-byte boundary (vector reductions in the wgrad flush), padding floats included in the size."""
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.ops import NUM_PARAMS, flat_size, flat_views
    shapes = [tuple(p.shape) for p in Nerf().parameters()]
    assert sum(int(np.prod(s)) for s in shapes) == NUM_PARAMS == 595844
    n = flat_size(shapes)
    flat = torch.arange(n, dtype=torch.float32)
    views = flat_views(flat, shapes)
    off = 0
    for v, shp in zip(views, shapes):
        assert tuple(v.shape) == shp and v.is_contiguous()
        assert v.data_ptr() == flat.data_ptr() + 4 * off and off % 4 == 0
        off += (v.numel() + 3) // 4 * 4
    assert off == n and n - NUM_PARAMS < 4 * len(shapes)


def test_config_switches_validate():
    from nerf_simple_b200 import config
    for bad, fn in (("fp16", config.set_precision), ("torch", config.set_sampler), ("gpu", config.set_select)):
        with pytest.raises(ValueError):
            fn(bad)
    assert config.get_precision() in ("bf16", "fp32") and config.get_sampler() in ("reference", "philox")
    assert config.get_select() == "reference" and config.get_fused_render() is False      # defaults = reference semantics
    seed, off0 = config.next_philox(10)
    _, off1 = config.next_philox(1)
    assert off1 - off0 == 3                                                               # ceil(10 / 4) Philox calls reserved


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the B200 arm) prints one JSON line with
    the contract's keys; it needs no GPU."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "rays/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["metric"].startswith("rays/sec") and line["config"]["workload"].startswith("configs[1]")
    from oracle.ref_import import reference_root
    want_kind = "reference" if reference_root() else "port"      # the real reference whenever a checkout is staged
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    if want_kind == "reference":
        assert "unmodified reference" in line["cpu_baseline"]["sample"]
        assert line["config0_frame_100x100x64"]["value"] > 0 and line["config0_train_step_1024x64"]["value"] > 0
    # the workload-naming keys are the B200 arm's, verbatim
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.workload_config(800, 800, 64, 1)
    assert line["e2e"] == {"value": line["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["vs_baseline"] is None


def test_bench_dump_outputs_format(tmp_path):
    """`bench.py --dump-outputs`: float32 .npy files, whole arrays up to 64 MB in all, beyond that the same fixed, seeded
    sample of rows for every array (with the row numbers), at most 64 MB."""
    import sys
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    small = {"loss": np.float64(0.25), "rgb": rng.random((40, 40, 3))}
    bench.dump_outputs(str(tmp_path / "small"), small)
    assert sorted(os.listdir(tmp_path / "small")) == ["loss.npy", "rgb.npy"]
    got = np.load(tmp_path / "small" / "rgb.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small["rgb"].astype(np.float32))
    big = {"rgb": rng.random((2200, 2200, 3), dtype=np.float32), "disp": rng.random((2200, 2200), dtype=np.float32)}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big)
        files = sorted(os.listdir(tmp_path / run))
        assert files == ["disp.npy", "disp_rows.npy", "rgb.npy", "rgb_rows.npy"]
        assert sum(os.path.getsize(tmp_path / run / f) for f in files) <= 64 << 20
    rows = np.load(tmp_path / "a" / "rgb_rows.npy").astype(np.int64)
    assert np.array_equal(rows, np.load(tmp_path / "a" / "disp_rows.npy")) and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rgb_rows.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "rgb.npy"), big["rgb"][rows])
    assert np.array_equal(np.load(tmp_path / "a" / "disp.npy"), big["disp"][rows])
