"""The two tcgen05 bf16 chains against a bf16-faithful float64 emulation (oracle/bf16_chain.py).

The parity tests compare the bf16 chains with the fp32 reference, and that comparison has to leave room for all of
the bf16 error (1e-2 on outputs of |rgb| <= 0.17): a swapped pair of rows, a dropped epilogue step or a dropped
delta tile fits under it.  The emulation rounds to bf16 exactly where the kernels round, so a correct kernel differs
from it only by fp32 accumulation-order noise, and the bounds below are set from that noise.

CPU part (no GPU): the emulation against the float64 oracle (inside the bf16 band), folded vs layer-wise, the fp32
noise model inside the bounds, and a mutation table: each deliberate bug, applied inside the emulation, must exceed
its bound by MUTATION_MARGIN at least.
GPU part (each test marked `gpu`): the kernels against the emulation -- forward in points and rays mode at tile
edges, ragged tails and multi-loop sizes, the training forward bit-identical to the inference forward, all 24
gradients in points and rays mode, and a run with NaN-poisoned workspaces through the C ABI.

Metrics: per output channel (r, g, b, sigma) the max abs and the RMS difference; per gradient tensor the max abs
difference relative to the tensor's max and the relative L2 difference (worst tensor reported).
"""
import numpy as np
import pytest

from conftest import load_golden
from oracle import bf16_chain as E
from oracle import nerf_oracle as O

# Bounds, per weight set: forward max abs / RMS per channel (r, g, b, sigma), gradients max abs over the tensor's max /
# relative L2 (worst tensor).  The fp32 noise model (accum="fp32", 65 x 64 rays case) gives 2.4e-5 / 7.5e-7 on rgb,
# 4.4e-5 / 1.5e-6 on sigma and 1e-2 / 2.8e-3 on the gradients at the golden weights.  The B200 shows about 4x that on
# the forward and 8x on the gradients, at every size alike: CUDA's sincosf is not correctly rounded, the double-angle
# recurrence multiplies a 1-ulp difference at level 0 by 2^i at level i, and the posx columns then round to the other
# bf16 neighbour now and then.  (Moving 30 % of the emulated level-0 sin / cos by one fp32 ulp reproduces it on the
# CPU: 3.5e-6 RMS on rgb, 3.4e-2 / 2.2e-2 on the gradients.)  The bounds are the worst the B200 shows over every GPU
# case below, x 1.3 to 2.2; DESIGN.md section 2 lists the observed values.
BOUNDS = {
    "golden": dict(fwd_max=(1.5e-4, 1.5e-4, 1.5e-4, 2.5e-4), fwd_rms=(1e-5, 1e-5, 1e-5, 1.2e-5), grad_max=0.1, grad_l2=0.035),
    "wide": dict(fwd_max=(3e-3, 3e-3, 3e-3, 3e-3), fwd_rms=(2.5e-4, 2.5e-4, 2.5e-4, 2e-4), grad_max=0.08, grad_l2=0.045),
}
MUTATION_MARGIN = 3.0       # a mutation must exceed some bound by this factor
BF16_BAND = 3e-4            # emulation vs the float64 oracle, per sample (DESIGN.md: the kernel shows 2.4e-4 / 2.5e-4)
GRAD_BAND_MAX, GRAD_BAND_L2 = 0.2, 0.15   # emulated gradients vs the float64 oracle (random cotangents cancel heavily)


# ------------------------------------------------------------------------------------------ helpers
def wide_weights(P):
    """Weights x1.5, every bias U(-0.5, 0.5), sigma bias + 1: larger activations, live biases, mixed ReLU masks."""
    rng = np.random.default_rng(11)
    Q = {}
    for k, v in P.items():
        Q[k] = rng.uniform(-0.5, 0.5, v.shape).astype(np.float32) if k.endswith("bias") else (v * 1.5).astype(np.float32)
    Q["sigma_fc.0.bias"] = (Q["sigma_fc.0.bias"] + 1).astype(np.float32)
    return Q


def weight_set(golden_weights, name):
    return golden_weights if name == "golden" else wide_weights(golden_weights)


def fwd_metrics(out, ref):
    d = np.asarray(out, np.float64) - np.asarray(ref, np.float64)
    return np.abs(d).max(0), np.sqrt((d * d).mean(0))


def grad_metrics(G, R):
    """Worst over the 24 tensors of (max abs diff / tensor max, relative L2 diff), with the tensors' names."""
    mx, l2 = (0.0, ""), (0.0, "")
    for k, r in R.items():
        r = np.asarray(r, np.float64)
        d = np.asarray(G[k], np.float64) - r
        a = float(np.abs(d).max() / max(np.abs(r).max(), 1e-30))
        b = float(np.linalg.norm(d) / max(np.linalg.norm(r), 1e-30))
        mx, l2 = max(mx, (a, k)), max(l2, (b, k))
    return mx, l2


def fwd_excess(out, ref, wset):
    """Largest metric / bound ratio of a forward comparison (> 1: out of bounds)."""
    mx, rms = fwd_metrics(out, ref)
    B = BOUNDS[wset]
    return float(max((mx / np.array(B["fwd_max"])).max(), (rms / np.array(B["fwd_rms"])).max()))


def grad_excess(G, R, wset):
    (mx, _), (l2, _) = grad_metrics(G, R)
    return max(mx / BOUNDS[wset]["grad_max"], l2 / BOUNDS[wset]["grad_l2"])


def check_fwd(tag, out, ref, wset):
    mx, rms = fwd_metrics(out, ref)
    B = BOUNDS[wset]
    e = lambda a: " ".join(f"{x:.2e}" for x in a)
    print(f"{tag}: max [{e(mx)}] (bound [{e(B['fwd_max'])}]), rms [{e(rms)}] (bound [{e(B['fwd_rms'])}])")
    assert np.isfinite(out).all(), tag
    assert (mx <= np.array(B["fwd_max"])).all() and (rms <= np.array(B["fwd_rms"])).all(), (tag, mx, rms)


def check_grads(tag, G, R, wset):
    (mx, kmx), (l2, kl2) = grad_metrics(G, R)
    B = BOUNDS[wset]
    print(f"{tag}: max/tensor max {mx:.2e} [{kmx}] (bound {B['grad_max']:.1e}), "
          f"rel L2 {l2:.2e} [{kl2}] (bound {B['grad_l2']:.1e})")
    assert all(np.isfinite(np.asarray(g)).all() for g in G.values()), tag
    assert mx <= B["grad_max"] and l2 <= B["grad_l2"], (tag, mx, kmx, l2, kl2)


def rays_case(B, N, seed=7):
    """B golden rays, stratified sample depths (B*N samples) and a fixed random cotangent of (r,g,b,sigma)."""
    g = load_golden("case_render_b1024_n64.npz")
    rng = np.random.default_rng(seed)
    rays = np.ascontiguousarray(g["rays"][np.arange(B) % 1024])
    ts = O.stratified_ts(rng.random((B, N), dtype=np.float32), N)
    cot = rng.standard_normal((B * N, 4)).astype(np.float32)
    return rays, ts, cot


def points_case(M, seed=5):
    """M query points o + d t (golden rays, t in [2, 6]) with unit view directions, and a random cotangent."""
    g = load_golden("case_render_b1024_n64.npz")
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, 1024, M)
    t = rng.uniform(2.0, 6.0, M).astype(np.float32)
    r = g["rays"][idx]
    d = r[:, 3:]
    q = np.concatenate([r[:, :3] + d * t[:, None], d / np.linalg.norm(d, axis=1, keepdims=True)], 1).astype(np.float32)
    return q, rng.standard_normal((M, 4)).astype(np.float32)


# ---------------------------------------------------------------------------------------- CPU part
@pytest.fixture(scope="module")
def cpu_case():
    """65 rays x 64 samples = 4160 samples: 33 tiles, the last one ragged (64 rows)."""
    return rays_case(65, 64)


@pytest.fixture(scope="module")
def clean(cpu_case, golden_weights):
    rays, ts, cot = cpu_case
    res = {}
    for wset in BOUNDS:
        P = weight_set(golden_weights, wset)
        for mode in E.MODES:
            out, saved = E.forward(rays, ts, P, mode, keep=True)
            res[wset, mode] = (out, E.backward(cot, saved, P, mode))
    return res


@pytest.mark.parametrize("mode", E.MODES)
def test_emulation_within_bf16_band_of_oracle(golden_weights, mode):
    """Golden case: the emulation is as far from the float64 reference as the kernels are (DESIGN.md, parity table)."""
    g = load_golden("case_train_b64_n64.npz")
    cot = np.random.default_rng(3).standard_normal((4096, 4))
    ref, saved_ref = O.mlp_forward(g["query"], golden_weights, dtype=np.float64, keep=True)
    out, saved = E.forward(g["query"], None, golden_weights, mode, keep=True)
    err = float(np.abs(out - ref).max())
    print(f"emulation [{mode}] vs oracle: max abs {err:.2e}")
    assert 1e-5 < err <= BF16_BAND            # (a float64 chain would be ~1e-8 away: the roundings are in)
    (mx, kmx), (l2, kl2) = grad_metrics(E.backward(cot, saved, golden_weights, mode),
                                        O.mlp_backward(cot, saved_ref, golden_weights, dtype=np.float64))
    print(f"emulation [{mode}] gradients vs oracle: {mx:.2e} [{kmx}], rel L2 {l2:.2e} [{kl2}]")
    assert mx <= GRAD_BAND_MAX and l2 <= GRAD_BAND_L2


def test_points_and_rays_mode_agree(golden_weights):
    """Rays mode = points mode on the query points the kernel forms from (o, d, t)."""
    rays, ts, _ = rays_case(5, 37)
    q = E.query_from_rays(rays, ts)
    ref = O.sample_points(rays, ts)[0]
    assert np.abs(q - ref).max() <= 1e-6
    assert np.array_equal(E.forward(rays, ts, golden_weights, "bf16"), E.forward(q, None, golden_weights, "bf16"))


def test_folded_and_layerwise_emulations_agree(clean):
    for wset in BOUNDS:
        (a, _), (b, _) = clean[wset, "bf16"], clean[wset, "bf16_layerwise"]
        err = float(np.abs(a - b).max())
        print(f"{wset}: folded vs layer-wise emulation, max abs {err:.2e}")
        assert err <= BF16_BAND * (1 if wset == "golden" else 10)


@pytest.mark.parametrize("wset", list(BOUNDS))
@pytest.mark.parametrize("mode", E.MODES)
def test_noise_model_within_bounds(cpu_case, golden_weights, clean, wset, mode):
    """fp32 products and per-tile, shuffled gradient sums (what the kernels do) stay inside the bounds."""
    rays, ts, cot = cpu_case
    P = weight_set(golden_weights, wset)
    out, saved = E.forward(rays, ts, P, mode, keep=True, accum="fp32")
    G = E.backward(cot, saved, P, mode, accum="fp32")
    ref, R = clean[wset, mode]
    check_fwd(f"noise model [{mode}, {wset}]", out, ref, wset)
    check_grads(f"noise model [{mode}, {wset}]", G, R, wset)


@pytest.mark.parametrize("mutation", list(E.MUTATIONS))
@pytest.mark.parametrize("mode", E.MODES)
def test_mutation_breaks_bounds(cpu_case, golden_weights, clean, mode, mutation):
    """Each deliberate bug exceeds a bound by MUTATION_MARGIN at least, at the golden weights."""
    if mutation == "fold_bias_bc0" and mode != "bf16":
        pytest.skip("the layer-wise chain has no folded bias")
    rays, ts, cot = cpu_case
    out, saved = E.forward(rays, ts, golden_weights, mode, keep=True, mutate=mutation)
    G = E.backward(cot, saved, golden_weights, mode, mutate=mutation)
    ref, R = clean["golden", mode]
    ratio = max(fwd_excess(out, ref, "golden"), grad_excess(G, R, "golden"))
    print(f"{mutation} [{mode}]: {ratio:.1f}x the bound ({E.MUTATIONS[mutation]})")
    assert ratio >= MUTATION_MARGIN, (mutation, ratio)


# ---------------------------------------------------------------------------------------- GPU part
FWD_M = (1, 127, 128, 129, 255, 256, 257, 1037, 4096)
BWD_M = (1, 129, 4160)
RAYS_BN = ((71, 37), (43, 96), (23, 192), (65, 64))   # 21, 33, 35, 33 tiles, every last tile ragged


def multi_loop_m():
    """2 x (SM count) x 256 + 129 samples: every CTA of the persistent chain kernels loops over several pair-tiles."""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 256 + 129


def gpu_net(P):
    import torch
    from nerf_simple_b200.nets import Nerf
    net = Nerf().cuda()
    net.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in P.items()}, strict=True)
    return net


def kernel_forward(net, mode, x, ts=None, need_grad=False):
    import torch
    from nerf_simple_b200 import _lib, ops
    xin = torch.from_numpy(x).cuda()
    with torch.set_grad_enabled(need_grad):
        if ts is None:
            out = ops.mlp_apply(net, _lib.IN_POINTS, xin, precision=mode)
        else:
            out = ops.mlp_apply(net, _lib.IN_RAYS, xin, torch.from_numpy(ts).cuda(), ts.shape[1], precision=mode)
    return out


def kernel_grads(net, mode, x, cot, ts=None):
    """The 24 gradients of sum(out * cot) through autograd (compositing not in the loop)."""
    import torch
    net.zero_grad(set_to_none=True)
    out = kernel_forward(net, mode, x, ts, need_grad=True)
    (out * torch.from_numpy(cot).cuda()).sum().backward()
    return {k: p.grad.double().cpu().numpy() for k, p in net.named_parameters()}


@pytest.mark.gpu
@pytest.mark.parametrize("wset", list(BOUNDS))
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_forward_points(golden_weights, mode, wset):
    P = weight_set(golden_weights, wset)
    big = multi_loop_m()
    q, _ = points_case(big)
    ref = E.forward(q, None, P, mode)
    net = gpu_net(P)
    for M in FWD_M + (big,):
        out = kernel_forward(net, mode, np.ascontiguousarray(q[:M])).double().cpu().numpy()
        check_fwd(f"forward points [{mode}, {wset}] M={M}", out, ref[:M], wset)


@pytest.mark.gpu
@pytest.mark.parametrize("wset", list(BOUNDS))
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_forward_rays(golden_weights, mode, wset):
    """Rays mode: query points formed in the kernel; N = 37, 96, 192 take the m / N division, N = 64 the shift."""
    P = weight_set(golden_weights, wset)
    net = gpu_net(P)
    for B, N in RAYS_BN:
        rays, ts, _ = rays_case(B, N)
        out = kernel_forward(net, mode, rays, ts).double().cpu().numpy()
        check_fwd(f"forward rays [{mode}, {wset}] B={B} N={N}", out, E.forward(rays, ts, P, mode), wset)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_training_forward_equals_inference_forward(golden_weights, mode):
    """FwdEpi<true> (saves tiles and masks) and FwdEpi<false> compute the same outputs bit for bit."""
    import torch
    P = wide_weights(golden_weights)
    net = gpu_net(P)
    q, _ = points_case(multi_loop_m())
    rays, ts, _ = rays_case(71, 37)
    for tag, x, t in (("points 4160", np.ascontiguousarray(q[:4160]), None), ("points multi-loop", q, None),
                      ("rays 71x37", rays, ts)):
        a = kernel_forward(net, mode, x, t, need_grad=False)
        b = kernel_forward(net, mode, x, t, need_grad=True).detach()
        print(f"training vs inference forward [{mode}] {tag}: max abs {float((a - b).abs().max()):.1e}")
        assert torch.equal(a, b), tag


@pytest.mark.gpu
@pytest.mark.parametrize("wset", list(BOUNDS))
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_backward_points(golden_weights, mode, wset):
    """Points mode is the path Nerf.forward takes: all 24 gradients against the emulated backward."""
    P = weight_set(golden_weights, wset)
    big = multi_loop_m()
    q, cot = points_case(big)
    _, saved = E.forward(q, None, P, mode, keep=True)
    net = gpu_net(P)
    for M in BWD_M + (big,):
        G = kernel_grads(net, mode, np.ascontiguousarray(q[:M]), np.ascontiguousarray(cot[:M]))
        R = E.backward(cot[:M], E.slice_saved(saved, M), P, mode)
        check_grads(f"backward points [{mode}, {wset}] M={M}", G, R, wset)


@pytest.mark.gpu
@pytest.mark.parametrize("wset", list(BOUNDS))
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_backward_rays(golden_weights, mode, wset):
    P = weight_set(golden_weights, wset)
    net = gpu_net(P)
    for B, N in ((65, 64), (43, 96)):
        rays, ts, cot = rays_case(B, N)
        G = kernel_grads(net, mode, rays, cot, ts)
        _, saved = E.forward(rays, ts, P, mode, keep=True)
        check_grads(f"backward rays [{mode}, {wset}] B={B} N={N}", G, E.backward(cot, saved, P, mode), wset)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", E.MODES)
def test_gpu_poisoned_workspaces(golden_weights, mode):
    """Through the C ABI: saved tensors and scratch filled with 0xFF bytes (NaN), out with NaN, gradients pre-filled
    with a non-zero G0.  The forward must equal a run on zeroed buffers bit for bit, grad - G0 must match a fresh
    backward, and nothing may be NaN: a read of an unwritten padding row or tile fails here every time."""
    import torch
    from nerf_simple_b200 import _lib, ops
    lib = _lib.load()
    prec = {"bf16": _lib.BF16, "bf16_layerwise": _lib.BF16_LAYERWISE}[mode]
    P = wide_weights(golden_weights)
    net = gpu_net(P)
    params = net.kernel_params()
    packed = net._packed.get(params, prec)
    stream = _lib.stream_ptr()
    q, qcot = points_case(4160)                       # 33 tiles, ragged last tile
    rays, ts, rcot = rays_case(71, 37)                # 2627 samples: 21 tiles, ragged last tile
    for tag, in_mode, x, t, cot in (("points 4160", _lib.IN_POINTS, q, None, qcot),
                                    ("rays 71x37", _lib.IN_RAYS, rays, ts, rcot)):
        x = torch.from_numpy(x).cuda()
        t = None if t is None else torch.from_numpy(t).cuda()
        N = 1 if t is None else t.shape[1]
        M = cot.shape[0]
        d_out = torch.from_numpy(cot).cuda()
        shapes = [tuple(p.shape) for p in params]

        def run(fill):
            saved = torch.full((lib.nb200_mlp_saved_bytes(prec, M),), fill, dtype=torch.uint8, device="cuda")
            out = torch.full((M, 4), float("nan") if fill else 0.0, device="cuda")
            rc = lib.nb200_mlp_forward(prec, in_mode, _lib.ptr(x), _lib.ptr(t), M, N, _lib.ptr_array(params),
                                       _lib.ptr(packed), _lib.ptr(out), _lib.ptr(saved), None, 0, stream)
            _lib.check(rc, "nb200_mlp_forward")
            return out, saved

        def backward(saved, fill, g0):
            sb = lib.nb200_mlp_scratch_bytes(prec, M, 1)
            scratch = torch.full((sb,), fill, dtype=torch.uint8, device="cuda")
            flat = torch.zeros(ops.flat_size(shapes), device="cuda")
            views = ops.flat_views(flat, shapes)
            for v, g in zip(views, g0):
                v.fill_(g)
            rc = lib.nb200_mlp_backward(prec, in_mode, _lib.ptr(x), _lib.ptr(t), M, N, _lib.ptr_array(params),
                                        _lib.ptr(packed), _lib.ptr(d_out), _lib.ptr(saved), _lib.ptr_array(views),
                                        _lib.ptr(scratch), sb, stream)
            _lib.check(rc, "nb200_mlp_backward")
            return {k: (v.double() - g).cpu().numpy() for k, v, g in zip(O.PARAM_NAMES, views, g0)}

        out0, saved0 = run(0)
        out1, saved1 = run(0xFF)
        assert bool(torch.isfinite(out1).all()), tag
        assert torch.equal(out0, out1), tag
        fresh = backward(saved0, 0, [0.0] * 24)
        g0 = [float(np.float32(0.5 * np.abs(fresh[k]).max() + 1e-3)) for k in O.PARAM_NAMES]   # exact in fp32
        poisoned = backward(saved1, 0xFF, g0)
        check_grads(f"poisoned workspaces [{mode}] {tag}: grad - G0 vs fresh backward", poisoned, fresh, "wide")
