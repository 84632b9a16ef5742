"""GPU parity tests: the CUDA path (through the C ABI, via the Python host layer) against the
numpy oracle and the reference-generated golden vectors.  Run on the B200 box with -m gpu."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import nerf_oracle as O

pytestmark = pytest.mark.gpu

TOL = {"fp32": 1e-4, "bf16": 1e-2, "bf16x3": 1e-4}        # BASELINE.json north_star tolerances (max abs err); bf16x3 = tensor-core fp32-class mode


# all-five-outputs case, bf16: observed on B200 (round 2) 0.107 of the tensor max elementwise and 0.106 in relative L2
# (worst tensor layers_0.0.weight); bounds are < 2x that.  fp32 / bf16x3 (gradients from the fp32 kernels): observed 9.6e-4.
BF16_ALL5_MAX, BF16_ALL5_L2, FP32_ALL5_MAX = 0.2, 0.15, 3e-3


def maxabs(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64))))


@pytest.fixture(scope="module")
def net(golden_weights):
    from nerf_simple_b200.nets import Nerf
    n = Nerf().cuda()
    n.load_state_dict({k: torch.from_numpy(v) for k, v in golden_weights.items()}, strict=True)
    return n


@pytest.fixture(params=["fp32", "bf16", "bf16x3"])
def precision(request):
    from nerf_simple_b200 import config
    config.set_precision(request.param)
    config.set_sampler("reference")
    yield request.param
    config.set_precision("bf16")


def test_library_targets_sm100():
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    assert lib.nb200_compiled_arch() == 100
    assert lib.nb200_device_arch() // 10 == 10, "tests must run on a B200 (sm_100)"


def test_raygen_matches_reference():
    from nerf_simple_b200 import ops
    from nerf_simple_b200.xyz import rays_single_cam
    g = load_golden("case_raygen.npz")
    for tag in ("h5w7", "h100", "h6w4"):
        H, W, f = g[f"{tag}.cam"]
        dirs = rays_single_cam([int(H), int(W), float(f)])
        assert np.array_equal(dirs.numpy(), g[f"{tag}.dirs"])               # bit exact
        rays = ops.generate_rays(torch.from_numpy(g[f"{tag}.poses"]).cuda(), int(H), int(W), float(f))
        assert maxabs(rays, g[f"{tag}.rays"]) <= 1e-6
        # sub-range == slice of the full table (sharded render relies on it)
        part = ops.generate_rays(torch.from_numpy(g[f"{tag}.poses"]).cuda(), int(H), int(W), float(f),
                                 ray_begin=7, n_rays=11)
        assert torch.equal(part, rays[7:18])


def test_sampler_bit_exact_and_philox():
    from nerf_simple_b200 import ops
    g = load_golden("case_train_b64_n64.npz")
    ts = ops.stratified_ts(64, 64, 2, 6, u=torch.from_numpy(g["u"]).cuda())
    assert np.array_equal(ts.cpu().numpy(), g["ts"])
    for N in (7, 100, 128):
        u = torch.rand(33, N)
        ts = ops.stratified_ts(33, N, 2, 6, u=u.cuda())
        assert np.array_equal(ts.cpu().numpy(), O.stratified_ts(u.numpy(), N))
    # Philox mode: stratified (one sample per bin), deterministic in (seed, offset), uniform
    a = ops.stratified_ts(4096, 64, 2, 6, device="cuda", seed=5, offset=0)
    b = ops.stratified_ts(4096, 64, 2, 6, device="cuda", seed=5, offset=0)
    c = ops.stratified_ts(4096, 64, 2, 6, device="cuda", seed=6, offset=0)
    assert torch.equal(a, b) and not torch.equal(a, c)
    bins = torch.linspace(2, 6, 65, device="cuda")
    assert bool(((a >= bins[:-1]) & (a <= bins[1:])).all())
    frac = (a - bins[:-1]) / (4 / 64)
    assert abs(float(frac.mean()) - 0.5) < 5e-3 and abs(float(frac.var()) - 1 / 12) < 5e-3
    # the quad fast path (N % 4 == 0, 16-byte aligned) and the generic kernel draw the same stream:
    # a misaligned output pointer forces the generic kernel through the C ABI
    import ctypes
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    for N in (64, 128, 36):
        fast = ops.stratified_ts(1000, N, 2, 6, device="cuda", seed=9, offset=123)
        buf = torch.zeros(1000 * N + 1, device="cuda")
        rc = lib.nb200_stratified_ts(None, 9, 123, 1000, N, 2.0, 6.0, ctypes.c_void_p(buf.data_ptr() + 4), _lib.stream_ptr())
        assert rc == 0 and torch.equal(buf[1:].view(1000, N), fast)


def test_posenc_matches_reference():
    from nerf_simple_b200.xyz import positional_encoder, gamma
    g = load_golden("case_train_b64_n64.npz")
    q = torch.from_numpy(g["query"][:256]).cuda()
    posx, posd = positional_encoder(q)
    assert posx.shape == (256, 63) and posd.shape == (256, 27)
    assert maxabs(posx, g["posx"]) <= 2e-6 and maxabs(posd, g["posd"]) <= 2e-6
    gx = gamma(q[:, 0:1], 10)
    assert maxabs(gx, g["posx"][:, 3:23]) <= 2e-6


@pytest.mark.parametrize("tag", ["n40", "n64", "n128", "n192", "n2", "n7"])
def test_compositing_isolated(tag):
    from nerf_simple_b200.rendering import volume_render
    g = load_golden("case_composite.npz")
    G = lambda k: torch.from_numpy(g[f"{tag}.{k}"]).cuda()
    outs = G("outs").requires_grad_(True)
    rgb, disp, alpha, acc, w = volume_render(outs, G("ts"), G("dirs"))
    # exp/log run on the MUFU units (<= 2^-21 relative error): 5e-6 absolute on the outputs
    assert maxabs(rgb, G("rgb")) <= 5e-6
    assert maxabs(alpha, G("alpha")) <= 5e-6
    assert maxabs(w, G("w")) <= 5e-6
    assert maxabs(acc, G("acc")) <= 5e-6
    assert float(((disp.detach() - G("disp")).abs() / G("disp").abs()).max()) <= 2e-5
    tot = (rgb * G("c_rgb")).sum() + (disp * G("c_disp")).sum() + (alpha * G("c_alpha")).sum() \
        + (acc * G("c_acc")).sum() + (w * G("c_w")).sum()
    tot.backward()
    ref = g[f"{tag}.d_outs"]
    assert maxabs(outs.grad, ref) <= 2e-4 * max(1.0, float(np.abs(ref).max()))


def test_compositing_long_ray_fallback():
    """N > 256 takes the thread-per-ray kernels; check against the oracle."""
    from nerf_simple_b200.rendering import volume_render
    rng = np.random.default_rng(3)
    B, N = 37, 300
    outs = rng.standard_normal((B, N, 4)).astype(np.float32)
    ts = np.sort(2 + 4 * rng.random((B, N)), axis=1).astype(np.float32)
    dirs = rng.standard_normal((B, 3)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    c_rgb = rng.standard_normal((B, 3)).astype(np.float32)
    o = torch.from_numpy(outs).cuda().requires_grad_(True)
    rgb, disp, alpha, acc, w = volume_render(o, torch.from_numpy(ts).cuda(), torch.from_numpy(dirs).cuda())
    r_rgb, r_disp, r_alpha, r_acc, r_w = O.volume_render(outs, ts, dirs)
    assert maxabs(rgb, r_rgb) <= 1e-5 and maxabs(w, r_w) <= 5e-6 and maxabs(alpha, r_alpha) <= 5e-6
    (rgb * torch.from_numpy(c_rgb).cuda()).sum().backward()
    ref = O.volume_render_backward(outs, ts, dirs, c_rgb)
    assert maxabs(o.grad, ref) <= 2e-4 * max(1.0, float(np.abs(ref).max()))


def test_mlp_forward_points(net, precision, golden_weights):
    g = load_golden("case_train_b64_n64.npz")
    with torch.no_grad():
        out = net(torch.from_numpy(g["query"]).cuda())
    assert out.shape == (4096, 4)
    assert maxabs(out, g["out"]) <= TOL[precision]
    # ragged M (not a multiple of any tile size)
    with torch.no_grad():
        out = net(torch.from_numpy(g["query"][:1000 + 37]).cuda())
    assert maxabs(out, g["out"][:1037]) <= TOL[precision]


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_fp32_class_modes_hold_1e4_with_scaled_weights(golden_weights, prec):
    """SURVEY section 7: single-pass TF32 passes 1e-4 only barely at default init and FAILS (2.7e-4) with the weights
    scaled x1.5.  Both fp32-class modes -- the SIMT kernels and the error-compensated bf16 tensor-core kernel -- must
    hold 1e-4 there too (reference = the numpy oracle evaluated in float64)."""
    from nerf_simple_b200 import config
    from nerf_simple_b200.nets import Nerf
    g = load_golden("case_train_b64_n64.npz")
    P = {k: (v * 1.5).astype(np.float32) for k, v in golden_weights.items()}
    n = Nerf().cuda()
    n.load_state_dict({k: torch.from_numpy(v) for k, v in P.items()}, strict=True)
    ref = O.mlp_forward(g["query"], P, dtype=np.float64)
    config.set_precision(prec)
    try:
        with torch.no_grad():
            out = n(torch.from_numpy(g["query"]).cuda())
    finally:
        config.set_precision("bf16")
    err = maxabs(out, ref)
    print(f"weights x1.5 [{prec}]: max abs err {err:.3e} (outputs up to {np.abs(ref).max():.2f})")
    assert err <= 1e-4


@pytest.mark.parametrize("case,N", [("case_train_b64_n64.npz", 64), ("case_render_b1024_n64.npz", 64),
                                    ("case_all5_b96_n128.npz", 128)])
def test_render_nerf_forward(net, precision, case, N):
    from nerf_simple_b200.rendering import render_nerf
    g = load_golden(case)
    torch.manual_seed(0)
    # inject the golden jitter through the reference-RNG path: render_nerf draws torch.rand(B,N)
    # from the CPU generator, so re-seed to the value the golden generator used
    seed = {"case_train_b64_n64.npz": 1, "case_render_b1024_n64.npz": 11, "case_all5_b96_n128.npz": 5}[case]
    torch.manual_seed(seed)
    with torch.no_grad():
        rgb, disp, alpha, acc, w = render_nerf(torch.from_numpy(g["rays"]).cuda(), net, N)
    tol = TOL[precision]
    assert maxabs(rgb, g["rgb"]) <= tol
    assert maxabs(alpha, g["alpha"]) <= tol
    assert maxabs(w, g["weights"]) <= tol
    assert maxabs(acc, g["acc"]) <= tol
    assert float(((disp - torch.from_numpy(g["disp"]).cuda()).abs() / torch.from_numpy(g["disp"]).cuda().abs()).max()) <= 10 * tol
    if precision == "bf16":
        mse = float(((rgb.cpu() - torch.from_numpy(g["rgb"])) ** 2).mean())
        assert 10 * np.log10(1.0 / max(mse, 1e-20)) > 60          # PSNR of our render vs the reference's


def _grad_check(net, grads_ref, rtol):
    for k, p in net.named_parameters():
        ref = grads_ref[k]
        scale = max(1e-6, float(np.max(np.abs(ref))))
        assert maxabs(p.grad, ref) <= rtol * scale, k


def test_train_step_gradients(net, precision):
    """train.py:51-54: MSE loss through rgb only; all 24 gradients vs the reference's autograd."""
    from nerf_simple_b200.rendering import render_nerf
    g = load_golden("case_train_b64_n64.npz")
    net.zero_grad()
    torch.manual_seed(1)
    rgb, *_ = render_nerf(torch.from_numpy(g["rays"]).cuda(), net, 64)
    loss = torch.nn.MSELoss()(rgb, torch.from_numpy(g["gt"]).cuda())
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) <= (1e-5 if precision != "bf16" else 2e-3)
    _grad_check(net, {k[5:]: v for k, v in g.items() if k.startswith("grad.")},
                2e-3 if precision != "bf16" else 5e-2)      # (bf16x3: forward on the tensor cores, gradients from the fp32 kernels)
    # gradients accumulate across backward calls like autograd
    g1 = [p.grad.clone() for p in net.parameters()]
    torch.manual_seed(1)
    rgb, *_ = render_nerf(torch.from_numpy(g["rays"]).cuda(), net, 64)
    torch.nn.MSELoss()(rgb, torch.from_numpy(g["gt"]).cuda()).backward()
    for a, p in zip(g1, net.parameters()):
        assert torch.allclose(p.grad, 2 * a, rtol=1e-3 if precision != "bf16" else 5e-2, atol=1e-7)


def test_all_five_outputs_gradient(net, precision):
    from nerf_simple_b200.rendering import render_nerf
    g = load_golden("case_all5_b96_n128.npz")
    net.zero_grad()
    torch.manual_seed(5)
    o5 = render_nerf(torch.from_numpy(g["rays"]).cuda(), net, 128)
    cot = [g["cot_rgb"], g["cot_disp"], g["cot_alpha"], g["cot_acc"], g["cot_w"]]
    sum((a * torch.from_numpy(b).cuda()).sum() for a, b in zip(o5, cot)).backward()
    grads = {k[5:]: v for k, v in g.items() if k.startswith("grad.")}
    worst = [0.0, 0.0]
    for k, p in net.named_parameters():
        if k in grads:
            scale = max(1e-6, float(np.abs(grads[k]).max()))
            # conditioning of this case is ~1.2e-2 even for fp32-vs-fp64 (see tests/test_oracle.py): random
            # cotangents on alpha/weights cancel heavily over 12288 samples.  bf16 (8-bit mantissa activations and
            # deltas): bounds = 2x the worst observed on B200 (BF16_ALL5_*), elementwise relative to the tensor's
            # max and in relative L2 norm (worst tensor: layers_0.0.weight, whose delta went through nine roundings).
            err = maxabs(p.grad, grads[k])
            l2 = float(np.linalg.norm(p.grad.cpu().numpy() - grads[k]) / max(1e-12, np.linalg.norm(grads[k])))
            worst = [max(worst[0], err / scale), max(worst[1], l2)]
            if precision != "bf16":
                assert err <= FP32_ALL5_MAX * scale, k
            else:
                assert err <= BF16_ALL5_MAX * scale and l2 <= BF16_ALL5_L2, (k, err, scale, l2)
    print(f"all-five-outputs gradient [{precision}]: worst elementwise err / tensor max {worst[0]:.3e}, worst relative L2 {worst[1]:.3e}")


def test_full_size_properties(net, precision):
    """BASELINE sizes (4096 rays x 64): properties that need no oracle run."""
    from nerf_simple_b200 import ops, config
    from nerf_simple_b200.rendering import render_nerf
    poses = torch.stack(__import__("nerf_simple_b200.xyz", fromlist=["x"]).poses_to_render(4, -30, 3)).cuda()
    f = 800 / (2 * np.tan(0.6911112070083618 / 2))
    rays = ops.generate_rays(poses, 800, 800, f, ray_begin=800 * 800 + 123456, n_rays=4096)
    torch.manual_seed(3)
    with torch.no_grad():
        rgb, disp, alpha, acc, w = render_nerf(rays, net, 64)
    assert rgb.shape == (4096, 3) and alpha.shape == (4096, 64)
    assert bool(torch.isfinite(rgb).all()) and bool(torch.isfinite(disp).all())
    # last delta is 1e10 => alpha_last == 1 and the weights sum to 1 (SURVEY 8a-bis item 10)
    assert float((acc - 1).abs().max()) <= 1e-4
    assert float((w.sum(1) - acc).abs().max()) <= 1e-5
    # chunk independence: rendering a sub-batch with the same jitter gives the same pixels
    torch.manual_seed(3)
    u = torch.rand(4096, 64)
    ts = ops.stratified_ts(4096, 64, 2, 6, u=u.cuda())
    from nerf_simple_b200 import _lib
    with torch.no_grad():
        full = ops.mlp_apply(net, _lib.IN_RAYS, rays, ts, 64)
        part = ops.mlp_apply(net, _lib.IN_RAYS, rays[1000:1500], ts[1000:1500], 64)
    assert maxabs(full.view(4096, 64, 4)[1000:1500].reshape(-1, 4), part) <= 1e-6


def test_render_image_and_poses_shapes(net, precision, tmp_path):
    """Host drivers (utils/rendering.py:88-160) incl. the remainder chunk the reference drops."""
    from nerf_simple_b200 import ops
    from nerf_simple_b200.rendering import render_image, render_poses
    from nerf_simple_b200.xyz import poses_to_render
    H = W = 20
    f = W / (2 * np.tan(0.6911112070083618 / 2))
    poses = poses_to_render(4, -30, 2)

    class RG:                                   # minimal stand-in for RayGenerator
        samples = {"val": [{"img": np.zeros((H, W, 3))}]}
        rays_dataset = {"val": ops.generate_rays(torch.stack(poses).cuda(), H, W, f).cpu()}
    rgb, depth, gt = render_image(net, RG, batch_size=150, im_idx=0, im_set="val")   # 400 = 2*150 + 100
    assert rgb.shape == (1, H, W, 3) and depth.shape == (1, H, W, 1) and gt.shape == (1, H, W, 3)
    assert float(rgb.min()) >= 0 and float(rgb.max()) <= 1 and not rgb.is_cuda
    frames = render_poses(net, poses, [H, W, f], 128, savepath=str(tmp_path))
    assert len(frames) == 2 and frames[0].shape == (H, W, 3)


def test_cpu_tensor_fails_loudly(net):
    from nerf_simple_b200._lib import NerfB200Error
    with pytest.raises(NerfB200Error):
        net(torch.zeros(4, 6))


def test_edge_shapes(net, precision):
    """Empty, single-ray and ragged inputs (the reference's loops silently drop remainders; here
    every size must work and agree with the full-batch result)."""
    from nerf_simple_b200 import ops, _lib
    from nerf_simple_b200.rendering import render_nerf, volume_render
    g = load_golden("case_render_b1024_n64.npz")
    rays = torch.from_numpy(g["rays"]).cuda()
    with torch.no_grad():
        out = net(torch.zeros((0, 6), device="cuda"))
        assert out.shape == (0, 4)
        o5 = render_nerf(rays[:0], net, 16)
        assert o5[0].shape == (0, 3) and o5[2].shape == (0, 16)
        torch.manual_seed(11)
        full = render_nerf(rays, net, 64)[0]
        torch.manual_seed(11)
        u = torch.rand(1024, 64)
        for b0, b1 in ((0, 1), (5, 134), (900, 1024)):                 # 1 ray, 129 rays (tile + 1), tail
            ts = ops.stratified_ts(b1 - b0, 64, 2, 6, u=u[b0:b1].cuda())
            o = ops.mlp_apply(net, _lib.IN_RAYS, rays[b0:b1], ts, 64).view(b1 - b0, 64, 4)
            rgb = ops.composite_apply(o, ts, rays[b0:b1], dirs_mode=1)[0]
            assert maxabs(rgb, full[b0:b1]) <= 1e-6
        # N that is neither a multiple of 32 nor of 4
        torch.manual_seed(3)
        rgb, disp, alpha, acc, w = render_nerf(rays[:77], net, 37)
        assert alpha.shape == (77, 37) and bool(torch.isfinite(rgb).all()) and float((acc - 1).abs().max()) <= 1e-4
    with pytest.raises(ValueError):
        volume_render(torch.zeros(2, 1, 4, device="cuda"), torch.zeros(2, 1, device="cuda"), torch.zeros(2, 3, device="cuda"))


@pytest.mark.parametrize("N", [32, 64, 128])
def test_fused_render_equals_three_kernels(N):
    """nb200_render_rays / nb200_render_camera (sampler -> MLP -> compositing in one kernel) against the
    three separate kernels on the same inputs, and against the oracle on the golden case."""
    from nerf_simple_b200 import ops, _lib
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    torch.manual_seed(0)
    net = Nerf().cuda()
    net.precision = "bf16"
    poses = torch.stack(poses_to_render(4, -30, 3)).cuda()
    H = W = 40
    f = 55.5
    with torch.no_grad():
        for ray_begin, B in ((0, 77), (1000, 1024), (3 * H * W - 130, 130)):       # ragged tails, last rays of the table
            rays = ops.generate_rays(poses, H, W, f, ray_begin, B)
            # (a) supplied sample depths (reference-RNG mode)
            ts = ops.stratified_ts(B, N, 2, 6, u=torch.rand(B, N).cuda())
            out = ops.mlp_apply(net, _lib.IN_RAYS, rays, ts, N).view(B, N, 4)
            rgb0, disp0, acc0 = ops.composite_apply(out, ts, rays, dirs_mode=1, want_alpha_weights=False)
            rgb1, disp1, acc1 = ops.render_fused(net, N, rays=rays, ts=ts)
            assert maxabs(rgb1, rgb0) <= 1e-6 and maxabs(acc1, acc0) <= 1e-6
            assert float(((disp1 - disp0).abs() / disp0.abs().clamp_min(1e-6)).max()) <= 1e-5
            # (b) Philox depths generated in the kernel == the sampler kernel's stream
            ts_p = ops.stratified_ts(B, N, 2, 6, device="cuda", seed=11, offset=5)
            out = ops.mlp_apply(net, _lib.IN_RAYS, rays, ts_p, N).view(B, N, 4)
            rgb0, disp0, acc0 = ops.composite_apply(out, ts_p, rays, dirs_mode=1, want_alpha_weights=False)
            rgb1, disp1, acc1 = ops.render_fused(net, N, rays=rays, seed=11, offset=5)
            assert maxabs(rgb1, rgb0) <= 1e-6 and maxabs(acc1, acc0) <= 1e-6
            # (c) rays generated in the kernel from the camera
            rgb2, disp2, acc2 = ops.render_fused(net, N, poses=poses, H=H, W=W, f=f, ray_begin=ray_begin, n_rays=B,
                                                 seed=11, offset=5)
            assert torch.equal(rgb2, rgb1) and torch.equal(disp2, disp1) and torch.equal(acc2, acc1)
    # unsupported shapes are refused, not silently mis-rendered
    lib = _lib.load()
    z = torch.zeros(8, 6, device="cuda")
    o = torch.zeros(8, 3, device="cuda")
    rc = lib.nb200_render_rays(_lib.BF16, _lib.ptr(z), None, 0, 0, 8, 48, 2.0, 6.0, _lib.ptr(net._packed.get(net.kernel_params(), _lib.BF16)),
                               _lib.ptr(o), _lib.ptr(o), _lib.ptr(o), _lib.stream_ptr())
    assert rc == -2
    assert not ops.fused_render_supported(net, 48) and not ops.fused_render_supported(net, 64, "fp32")


def test_fused_render_golden(net):
    """The fused kernel against the reference-generated golden render (bf16 tolerance of the north star)."""
    from nerf_simple_b200 import ops, config
    config.set_precision("bf16")
    g = load_golden("case_render_b1024_n64.npz")
    rays = torch.from_numpy(g["rays"]).cuda()
    with torch.no_grad():
        ts = ops.stratified_ts(1024, 64, 2, 6, u=torch.from_numpy(g["u"]).cuda())
        rgb, disp, acc = ops.render_fused(net, 64, rays=rays, ts=ts)
    assert maxabs(rgb, g["rgb"]) <= 1e-2 and maxabs(acc, g["acc"]) <= 1e-2
    mse = float(((rgb.cpu() - torch.from_numpy(g["rgb"])) ** 2).mean())
    assert 10 * np.log10(1.0 / max(mse, 1e-20)) > 60


@pytest.mark.parametrize("B,N,rtol", [(65, 64, 5e-2), (3, 37, 0.3), (129, 96, 5e-2)])
def test_train_gradients_odd_tile_counts(net, golden_weights, B, N, rtol):
    """Training shapes whose sample count is not a multiple of 256 (an odd number of 128-sample tiles, a
    ragged last tile): bf16 gradients against the ORACLE (numpy restatement of the reference's autograd) on the
    same inputs.  The bf16 deviation averages out with the number of samples (2.7e-2 at 4096 samples), hence the
    looser bound for 111 samples.  These are north-star bounds against the fp32 reference, and they leave room for
    all of the bf16 error: in the float64 oracle, dropping the deltas of one whole tile at 65 x 64 moves the gradients by only 1.5-3.3 % of
    each tensor's max, and dropping the ragged last 64 samples by 0.3-0.7 %, both inside 5e-2.  Single tiles, slots
    and ragged tails are pinned by tests/test_bf16_chain.py, against an emulation that rounds where the kernels do."""
    from nerf_simple_b200 import config, ops, _lib
    g = load_golden("case_render_b1024_n64.npz")
    rays_np = g["rays"][:B]
    rng = np.random.default_rng(7)
    u_np, gt_np = rng.random((B, N), dtype=np.float32), rng.random((B, 3), dtype=np.float32)
    loss_ref, grads_ref, rgb_ref = O.train_step_grads(rays_np, golden_weights, N, u_np, gt_np)
    rays, u, gt = torch.from_numpy(rays_np).cuda(), torch.from_numpy(u_np).cuda(), torch.from_numpy(gt_np).cuda()
    for prec, rt in (("fp32", 2e-3), ("bf16", rtol)):
        config.set_precision(prec)
        net.zero_grad()
        ts = ops.stratified_ts(B, N, 2, 6, u=u)
        out = ops.mlp_apply(net, _lib.IN_RAYS, rays, ts, N).view(B, N, 4)
        rgb = ops.composite_apply(out, ts, rays, dirs_mode=1)[0]
        loss = torch.nn.functional.mse_loss(rgb, gt)
        loss.backward()
        assert maxabs(rgb, rgb_ref) <= TOL[prec] and abs(loss.item() - loss_ref) <= 10 * TOL[prec]
        for k, p in net.named_parameters():
            ref = grads_ref[k]
            scale = max(1e-6, float(np.abs(ref).max()))
            err = maxabs(p.grad, ref)
            assert err <= rt * scale, (prec, k, B, N, err, scale)
            if B * N >= 4096:      # (111 samples: gradients of O(1) with no averaging; the relative bound is the meaningful one)
                assert err <= TOL[prec], (prec, k, B, N, err)
    config.set_precision("bf16")
