"""autograd.Function wrappers over the C ABI: one per operator boundary of the reference.

    mlp_apply        <- Nerf.forward            (utils/nets.py:34-43, utils/xyz.py:16-36)
    composite_apply  <- volume_render           (utils/rendering.py:47-85)
    stratified_ts    <- the sampler lines       (utils/rendering.py:24-30)
    generate_rays    <- rays_single_cam + pose  (utils/xyz.py:38-52, utils/rendering.py:129-134)

Everything here requires CUDA tensors; there is no eager/PyTorch fallback.
"""
from __future__ import annotations

import torch

from . import _lib, config

NUM_PARAMS = 595844
_PREC = {"fp32": _lib.FP32, "bf16": _lib.BF16, "bf16x3": _lib.BF16X3, "bf16_layerwise": _lib.BF16_LAYERWISE}


def flat_views(flat, shapes):
    """Views of a flat fp32 buffer for tensors of `shapes`, each starting on a 16-byte boundary (the
    wgrad kernel flushes aligned rows with vector reductions).  One split + one view per tensor."""
    sizes, padded = [], []
    for shp in shapes:
        n = 1
        for d in shp:
            n *= d
        sizes.append(n)
        padded.append((n + 3) // 4 * 4)
    chunks = flat.split(padded) if sum(padded) == flat.numel() else flat[:sum(padded)].split(padded)
    return [(c if n == p else c[:n]).view(shp) for c, n, p, shp in zip(chunks, sizes, padded, shapes)]


def flat_size(shapes):
    tot = 0
    for shp in shapes:
        n = 1
        for d in shp:
            n *= d
        tot += (n + 3) // 4 * 4
    return tot


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    _lib.require_cuda(t, name)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------------------- weights
class PackedWeights:
    """Kernel-format copy of the 24 parameters (bf16 tcgen05 operand images), refreshed whenever
    a parameter's version counter or storage changes (the caller's optimizer updates the fp32
    masters in place between calls, train.py:55)."""

    def __init__(self):
        self.bufs = {}      # precision -> (key, buffer): bf16 and bf16x3 images have different layouts

    def invalidate(self):
        """Force a re-pack on the next call.  Needed after writes the version counters do not see: `p.data.copy_()`,
        `p.data.normal_()`, EMA swaps through `.data` (in-place ops on the parameter itself, `optimizer.step()` and
        `load_state_dict` bump the version and need nothing)."""
        self.bufs = {p: (None, b) for p, (_, b) in self.bufs.items()}

    def get(self, params, precision):
        if precision == _lib.FP32:
            return None
        key = tuple((p.data_ptr(), p._version) for p in params)
        old_key, buf = self.bufs.get(precision, (None, None))
        if buf is None or old_key != key or buf.device != params[0].device:
            lib = _lib.load()
            nbytes = lib.nb200_packed_weights_bytes(precision)
            if buf is None or buf.device != params[0].device:
                buf = torch.empty(nbytes, dtype=torch.uint8, device=params[0].device)
            rc = lib.nb200_pack_weights(precision, _lib.ptr_array(params), _lib.ptr(buf),
                                        _lib.stream_ptr(params[0].device))
            _lib.check(rc, "nb200_pack_weights")
            self.bufs[precision] = (key, buf)
        return buf


class _MLPFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, precision, in_mode, N, need_grad, packed, in0, in1, *params):
        lib = _lib.load()
        dev = in0.device
        M = in0.shape[0] if in_mode == _lib.IN_POINTS else in0.shape[0] * N
        out = torch.empty((M, 4), dtype=torch.float32, device=dev)
        saved = None
        if need_grad:
            saved = torch.empty(lib.nb200_mlp_saved_bytes(precision, M), dtype=torch.uint8, device=dev)
        sb = lib.nb200_mlp_scratch_bytes(precision, M, 0) if not need_grad or precision != _lib.FP32 else 0
        scratch = torch.empty(sb, dtype=torch.uint8, device=dev) if sb else None
        rc = lib.nb200_mlp_forward(precision, in_mode, _lib.ptr(in0), _lib.ptr(in1), M, N,
                                   _lib.ptr_array(params), _lib.ptr(packed), _lib.ptr(out),
                                   _lib.ptr(saved), _lib.ptr(scratch), sb, _lib.stream_ptr(dev))
        _lib.check(rc, "nb200_mlp_forward")
        if need_grad:
            ctx.meta = (precision, in_mode, N, M)
            ctx.packed = packed
            ctx.aux = (in0, in1, saved)
            ctx.save_for_backward(*params)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        precision, in_mode, N, M = ctx.meta
        in0, in1, saved = ctx.aux
        params = ctx.saved_tensors
        dev = d_out.device
        d_out = _f32c(d_out, "d_out")
        shapes = [tuple(p.shape) for p in params]
        flat = torch.zeros(flat_size(shapes), dtype=torch.float32, device=dev)
        views = flat_views(flat, shapes)
        sb = lib.nb200_mlp_scratch_bytes(precision, M, 1)
        scratch = torch.empty(sb, dtype=torch.uint8, device=dev) if sb else None
        rc = lib.nb200_mlp_backward(precision, in_mode, _lib.ptr(in0), _lib.ptr(in1), M, N,
                                    _lib.ptr_array(params), _lib.ptr(ctx.packed), _lib.ptr(d_out),
                                    _lib.ptr(saved), _lib.ptr_array(views), _lib.ptr(scratch), sb,
                                    _lib.stream_ptr(dev))
        _lib.check(rc, "nb200_mlp_backward")
        return (None, None, None, None, None, None, None) + tuple(views)


def mlp_apply(net, in_mode, in0, in1=None, N=1, precision=None):
    """Run the fused posenc+MLP for `net` (a nerf_simple_b200.nets.Nerf).  Returns [M,4]."""
    precision = _PREC[precision or getattr(net, "precision", None) or config.get_precision()]
    params = net.kernel_params()
    _lib.require_cuda(params[0], "Nerf parameters (call net.cuda())")
    in0 = _f32c(in0, "input")
    if in_mode == _lib.IN_RAYS:
        in1 = _f32c(in1, "ts")
    need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
    if need_grad and precision == _lib.BF16X3:
        # Autograd accepts any cotangent.  With random cotangents on all five render outputs (tests/test_gpu_parity.py)
        # the ReLU masks that the 16-bit (hi + lo) weights of the bf16x3 forward flip move some gradients by 5e-3 of the
        # tensor max, over the suite's 3e-3 fp32-class bound, so autograd keeps the fp32 kernels.  Training steps
        # (Trainer(precision="bf16x3"), the C ABI) run the bf16x3 tensor-core backward and meet the fp32 bounds there.
        precision = _lib.FP32
    packed = net._packed.get(params, precision)
    cap = config._state["max_samples_per_call"]
    M = in0.shape[0] if in_mode == _lib.IN_POINTS else in0.shape[0] * N
    if need_grad or M <= cap or precision != _lib.FP32:
        return _MLPFunction.apply(precision, in_mode, N, need_grad, packed, in0, in1, *params)
    # inference in fp32 parity mode: bound the per-call activation workspace
    step = max(1, cap // N) if in_mode == _lib.IN_RAYS else cap
    outs = []
    for s in range(0, in0.shape[0], step):
        a = in0[s:s + step]
        b = in1[s:s + step] if in1 is not None else None
        outs.append(_MLPFunction.apply(precision, in_mode, N, False, packed, a, b, *params))
    return torch.cat(outs)


# ---------------------------------------------------------------------------- compositing
class _CompositeFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, outs, ts, dirs, dirs_mode, want_aw):
        lib = _lib.load()
        B, N = ts.shape
        dev = outs.device
        rgb = torch.empty((B, 3), dtype=torch.float32, device=dev)
        disp = torch.empty((B,), dtype=torch.float32, device=dev)
        acc = torch.empty((B,), dtype=torch.float32, device=dev)
        alpha = torch.empty((B, N), dtype=torch.float32, device=dev) if want_aw else None
        w = torch.empty((B, N), dtype=torch.float32, device=dev) if want_aw else None
        rc = lib.nb200_composite_forward(_lib.ptr(outs), _lib.ptr(ts), _lib.ptr(dirs), dirs_mode, B, N,
                                         _lib.ptr(rgb), _lib.ptr(disp), _lib.ptr(acc), _lib.ptr(alpha),
                                         _lib.ptr(w), _lib.stream_ptr(dev))
        _lib.check(rc, "nb200_composite_forward")
        ctx.dirs_mode = dirs_mode
        ctx.save_for_backward(outs, ts, dirs)
        ctx.set_materialize_grads(False)
        if want_aw:
            return rgb, disp, alpha, acc, w
        return rgb, disp, acc

    @staticmethod
    def backward(ctx, d_rgb, d_disp, *rest):
        lib = _lib.load()
        outs, ts, dirs = ctx.saved_tensors
        if len(rest) == 3:
            d_alpha, d_acc, d_w = rest
        else:
            (d_acc,), d_alpha, d_w = rest, None, None
        B, N = ts.shape
        dev = outs.device
        prep = lambda g: None if g is None else _f32c(g, "cotangent")
        d_rgb = torch.zeros((B, 3), dtype=torch.float32, device=dev) if d_rgb is None else prep(d_rgb)
        d_disp, d_alpha, d_acc, d_w = prep(d_disp), prep(d_alpha), prep(d_acc), prep(d_w)
        d_outs = torch.empty_like(outs)
        rc = lib.nb200_composite_backward(_lib.ptr(outs), _lib.ptr(ts), _lib.ptr(dirs), ctx.dirs_mode,
                                          _lib.ptr(d_rgb), _lib.ptr(d_disp), _lib.ptr(d_acc),
                                          _lib.ptr(d_alpha), _lib.ptr(d_w), B, N, _lib.ptr(d_outs),
                                          _lib.stream_ptr(dev))
        _lib.check(rc, "nb200_composite_backward")
        return d_outs, None, None, None, None


def composite_apply(outs, ts, dirs, dirs_mode=0, want_alpha_weights=True):
    outs = _f32c(outs, "nerf_outs")
    ts = _f32c(ts, "ts")
    dirs = _f32c(dirs, "dirs")
    B, N = ts.shape
    if outs.shape != (B, N, 4):
        raise ValueError(f"nerf_outs must be [B,N,4]; got {tuple(outs.shape)} for ts {tuple(ts.shape)}")
    if N < 2:
        raise ValueError("compositing needs N >= 2 samples per ray (the reference degenerates at N=1)")
    if dirs.shape != (B, 6 if dirs_mode else 3):
        raise ValueError(f"dirs has shape {tuple(dirs.shape)}")
    return _CompositeFunction.apply(outs, ts, dirs, dirs_mode, want_alpha_weights)


# -------------------------------------------------------------------------------- sampler
def stratified_ts(B, N, tn=2.0, tf=6.0, u=None, device=None, seed=None, offset=None):
    """ts[B,N].  u given -> reference-RNG mode (bit-identical to utils/rendering.py:25-29);
    otherwise device Philox keyed by (seed, offset)."""
    lib = _lib.load()
    if u is not None:
        u = _f32c(u, "u")
        device = u.device
    ts = torch.empty((B, N), dtype=torch.float32, device=device)
    if u is None and seed is None:
        seed, offset = config.next_philox(B * N)
    rc = lib.nb200_stratified_ts(_lib.ptr(u), int(seed or 0), int(offset or 0), B, N, float(tn), float(tf),
                                 _lib.ptr(ts), _lib.stream_ptr(ts.device))
    _lib.check(rc, "nb200_stratified_ts")
    return ts


# --------------------------------------------------------------------------------- raygen
def generate_rays(poses, H, W, f, ray_begin=0, n_rays=None):
    """rays[n,6] on the device of `poses` ([P,4,4] or [4,4] camera-to-world, CUDA)."""
    lib = _lib.load()
    poses = _f32c(poses, "poses")
    if poses.dim() == 2:
        poses = poses[None]
    P = poses.shape[0]
    if n_rays is None:
        n_rays = P * H * W - ray_begin
    rays = torch.empty((n_rays, 6), dtype=torch.float32, device=poses.device)
    rc = lib.nb200_generate_rays(_lib.ptr(poses), P, int(H), int(W), float(f), int(ray_begin), int(n_rays),
                                 _lib.ptr(rays), _lib.stream_ptr(poses.device))
    _lib.check(rc, "nb200_generate_rays")
    return rays


# ----------------------------------------------------------------------------- fused render
FUSED_RENDER_N = (32, 64, 128)     # whole rays per 128-sample tile


def fused_render_supported(net, N, precision=None) -> bool:
    precision = precision or getattr(net, "precision", None) or config.get_precision()
    return precision in ("bf16", "bf16_layerwise") and int(N) in FUSED_RENDER_N


def render_fused(net, N, rays=None, ts=None, poses=None, H=0, W=0, f=0.0, ray_begin=0, n_rays=None,
                 tn=2.0, tf=6.0, seed=None, offset=None, precision=None):
    """No-grad render_nerf (utils/rendering.py:13-45) as ONE kernel: sampler -> posenc + MLP -> compositing.
    Either `rays` [B,6] (optionally with `ts` [B,N]; else Philox depths keyed by (seed, offset)), or a
    camera (`poses` [P,4,4], H, W, f, ray_begin, n_rays) whose rays are generated in the kernel.
    Returns (rgb [B,3], disp [B], acc [B]); equals stratified_ts + mlp_apply + composite_apply."""
    lib = _lib.load()
    params = net.kernel_params()
    _lib.require_cuda(params[0], "Nerf parameters (call net.cuda())")
    dev = params[0].device
    prec = _PREC[precision or getattr(net, "precision", None) or config.get_precision()]
    if prec not in _lib.BF16_MODES:
        raise ValueError("render_fused needs a bf16 precision mode")
    packed = net._packed.get(params, prec)
    if rays is not None:
        rays = _f32c(rays, "rays")
        B = rays.shape[0]
        if ts is not None:
            ts = _f32c(ts, "ts")
            if ts.shape != (B, N):
                raise ValueError(f"ts must be [B,N]; got {tuple(ts.shape)}")
    else:
        poses = _f32c(poses, "poses")
        if poses.dim() == 2:
            poses = poses[None]
        B = int(n_rays if n_rays is not None else poses.shape[0] * H * W - ray_begin)
    if ts is None and seed is None:
        seed, offset = config.next_philox(B * N)
    rgb = torch.empty((B, 3), dtype=torch.float32, device=dev)
    disp = torch.empty((B,), dtype=torch.float32, device=dev)
    acc = torch.empty((B,), dtype=torch.float32, device=dev)
    st = _lib.stream_ptr(dev)
    if rays is not None:
        rc = lib.nb200_render_rays(prec, _lib.ptr(rays), _lib.ptr(ts), int(seed or 0), int(offset or 0), B, int(N),
                                   float(tn), float(tf), _lib.ptr(packed), _lib.ptr(rgb), _lib.ptr(disp), _lib.ptr(acc), st)
        _lib.check(rc, "nb200_render_rays")
    else:
        rc = lib.nb200_render_camera(prec, _lib.ptr(poses), poses.shape[0], int(H), int(W), float(f), int(ray_begin), B,
                                     int(seed or 0), int(offset or 0), int(N), float(tn), float(tf), _lib.ptr(packed),
                                     _lib.ptr(rgb), _lib.ptr(disp), _lib.ptr(acc), st)
        _lib.check(rc, "nb200_render_camera")
    return rgb, disp, acc


def frame_to_u8(rgb, bgr=True):
    """rgb [...,3] fp32 (CUDA) -> uint8 of the same shape: clip to [0,1], optional RGB->BGR swap, x255, truncate --
    the frame cv2.VideoWriter receives at utils/rendering.py:158-159, converted on the device (3 B/pixel to copy)."""
    lib = _lib.load()
    rgb = _f32c(rgb, "rgb")
    out = torch.empty(rgb.shape, dtype=torch.uint8, device=rgb.device)
    rc = lib.nb200_frame_to_u8(_lib.ptr(rgb), rgb.numel() // 3, 1 if bgr else 0, _lib.ptr(out), _lib.stream_ptr(rgb.device))
    _lib.check(rc, "nb200_frame_to_u8")
    return out


def positional_encoding(v, Lp=10, Ld=4):
    lib = _lib.load()
    v = _f32c(v, "vec")
    M = v.shape[0]
    posx = torch.empty((M, 3 + 6 * Lp), dtype=torch.float32, device=v.device)
    posd = torch.empty((M, 3 + 6 * Ld), dtype=torch.float32, device=v.device)
    rc = lib.nb200_positional_encoding(_lib.ptr(v), M, Lp, Ld, _lib.ptr(posx), _lib.ptr(posd),
                                       _lib.stream_ptr(v.device))
    _lib.check(rc, "nb200_positional_encoding")
    return posx, posd
