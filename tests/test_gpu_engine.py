"""GPU tests of the device-resident frame driver (engine.FrameRenderer): the loop of
utils/rendering.py:139-151 with host buffers in and out, blocking and pipelined, separate and fused kernels."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _renderer(net, **kw):
    from nerf_simple_b200.engine import FrameRenderer
    return FrameRenderer(net, 40, 40, 55.5, N=64, seed=3, precision="bf16", **kw)


def test_frame_renderer_host_paths_agree():
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    torch.manual_seed(0)
    net = Nerf().cuda()
    poses = torch.stack(poses_to_render(4, -30, 4))
    with torch.no_grad():
        ref = [_renderer(net).render_frame(poses.cuda(), i) for i in range(1)]           # device-resident call, frame 0
        # blocking host call: same Philox offsets (fresh renderer), same frame
        r = _renderer(net)
        rgb_h, disp_h = torch.empty(40, 40, 3).pin_memory(), torch.empty(40, 40).pin_memory()
        r.render_frame_host(poses[0].pin_memory(), rgb_h, disp_h)
        assert torch.equal(rgb_h, ref[0][0].cpu()) and torch.equal(disp_h, ref[0][1].cpu())
        assert float(rgb_h.min()) >= 0.0 and float(rgb_h.max()) <= 1.0                    # clip of :146
        # pipelined host calls (wait=False): three frames into three buffers, then finish()
        a, b = _renderer(net), _renderer(net)
        bufs = [(torch.empty(40, 40, 3).pin_memory(), torch.empty(40, 40).pin_memory()) for _ in range(3)]
        evs = [a.render_frame_host(poses[i].pin_memory(), *bufs[i], wait=False) for i in range(3)]
        a.finish()
        assert all(e.query() for e in evs)
        for i in range(3):
            rgb_b, disp_b = torch.empty(40, 40, 3).pin_memory(), torch.empty(40, 40).pin_memory()
            b.render_frame_host(poses[i].pin_memory(), rgb_b, disp_b)
            assert torch.equal(bufs[i][0], rgb_b) and torch.equal(bufs[i][1], disp_b)
        # one-kernel path == four-kernel path
        f = _renderer(net, fused=True)
        assert f.fused and not _renderer(net).fused
        rgb_f, disp_f = f.render_frame(poses.cuda(), 0)
        assert float((rgb_f - ref[0][0]).abs().max()) <= 1e-6
        assert f.launches == 1


def test_render_sharded_single_rank_is_the_frame():
    from nerf_simple_b200.engine import render_sharded, shard_range
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    torch.manual_seed(0)
    net = Nerf().cuda()
    poses = torch.stack(poses_to_render(4, -30, 2)).cuda()
    with torch.no_grad():
        whole = _renderer(net).render_frame(poses, 1)
        # the bands a 3-rank job would render, stitched by hand, ARE the frame: every sample keeps its place in the
        # jitter stream (Philox position = f(ray index in the frame)), so sharding does not change a single bit
        parts = []
        for rank in range(3):
            b, e = shard_range(1600, rank, 3)
            rgb, disp = _renderer(net).render_rays(poses, 1600 + b, e - b, philox_base=(b * 64) // 4)
            assert rgb.shape == (e - b, 3) and disp.shape == (e - b,)
            parts.append(rgb)
        stitched = torch.cat(parts)
        assert torch.equal(stitched.view(40, 40, 3), whole[0])
        rgb1, disp1 = render_sharded(_renderer(net), poses, 1, rank=0, world=1)
        assert torch.equal(rgb1.reshape(40, 40, 3), whole[0]) and torch.equal(disp1.reshape(40, 40), whole[1])


@pytest.mark.parametrize("fused", [False, True])
def test_chain_kernel_is_deterministic_over_many_tiles(fused):
    """Twelve renders of the same 320x320x64 frame (51,200 tiles: ~170 per slot and CTA, both slots and the tail in
    use) must be bit-identical: the epilogue warps of a slot share the staged bias row, the head-weight table that
    lives in the free half of the posd rows, and the exchange rows of the colour layer, and a missing barrier or an
    overlapping write between them shows up as run-to-run differences (found once this way: the posd zero padding
    overwrote table entries written by faster threads)."""
    from nerf_simple_b200.engine import FrameRenderer
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    torch.manual_seed(0)
    net = Nerf().cuda()
    poses = torch.stack(poses_to_render(4, -30, 2)).cuda()
    with torch.no_grad():
        first = None
        for _ in range(12):
            r = FrameRenderer(net, 320, 320, 444.4, N=64, seed=5, precision="bf16", fused=fused)   # fresh Philox offsets
            rgb, disp = r.render_frame(poses, 1)
            if first is None:
                first = (rgb.clone(), disp.clone())
                assert bool(torch.isfinite(rgb).all()) and bool(torch.isfinite(disp).all())
            else:
                assert torch.equal(rgb, first[0]) and torch.equal(disp, first[1])


def test_bench_dump_outputs_is_the_last_timed_frame(tmp_path):
    """`bench.py --dump-outputs DIR` writes the frame of the last timed step, the same in every run: after 3 warm-up and
    3 timed frames of the dome path it is frame 2 at the jitter position of the sixth frame."""
    import json
    import os
    import subprocess
    import sys
    from nerf_simple_b200.engine import FrameRenderer
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "render", "--res", "64", "--steps", "3",
                              "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-3000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
        assert sorted(os.listdir(tmp_path / run)) == ["disp.npy", "rgb.npy"]
        dumps.append({k: np.load(tmp_path / run / f"{k}.npy") for k in ("rgb", "disp")})
    assert dumps[0]["rgb"].dtype == np.float32 and dumps[0]["rgb"].shape == (64, 64, 3) and dumps[0]["disp"].shape == (64, 64)
    assert all(np.array_equal(dumps[0][k], dumps[1][k]) for k in ("rgb", "disp"))
    torch.manual_seed(0)
    net = Nerf().cuda()
    poses = torch.stack(poses_to_render(4, -30, 30)).cuda()
    r = FrameRenderer(net, 64, 64, 64 / (2 * np.tan(0.6911112070083618 / 2)), N=64, seed=1, precision="bf16", fused=False)
    with torch.no_grad():
        for idx in (0, 1, 2, 0, 1, 2):
            rgb, disp = r.render_frame(poses, idx)
    assert np.array_equal(rgb.cpu().numpy(), dumps[0]["rgb"]) and np.array_equal(disp.cpu().numpy(), dumps[0]["disp"])
