"""CPU oracle for the Nerf-Simple hot path -- TEST INFRASTRUCTURE ONLY.

A numpy restatement of the reference's algorithm (UCSD-Comp-Imaging/Nerf-Simple):
ray generation -> stratified sampling -> positional encoding -> 8x256 MLP ->
alpha compositing, forward and analytic backward.  Every function cites the
reference file:line it follows (paths relative to the reference checkout).

Parity status: PINNED.  `oracle/gen_golden.py` imports the unmodified reference
(oracle/ref_import.py; with a `.cuda()` no-op shim -- the reference hard-codes
`.cuda()`, utils/rendering.py:30,68), runs it on seeded inputs and stores its
outputs + autograd gradients under tests/golden/; tests/test_oracle.py checks this
restatement against those vectors.  The reference itself ships no tests or golden
vectors (SURVEY.md section 4).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module, and only as the checker / CPU baseline.  The product
path (nerf_simple_b200) never imports it and has no CPU fallback.
"""
from __future__ import annotations

import numpy as np

# Order of the 24 parameter tensors == reference state_dict order (utils/nets.py:16-32).
PARAM_SHAPES = [
    ("layers_0.0.weight", (256, 63)), ("layers_0.0.bias", (256,)),
    ("layers_0.2.weight", (256, 256)), ("layers_0.2.bias", (256,)),
    ("layers_0.4.weight", (256, 256)), ("layers_0.4.bias", (256,)),
    ("layers_0.6.weight", (256, 256)), ("layers_0.6.bias", (256,)),
    ("layers_0.8.weight", (256, 256)), ("layers_0.8.bias", (256,)),
    ("skip_conn_layer.0.weight", (256, 319)), ("skip_conn_layer.0.bias", (256,)),
    ("layers_1.0.weight", (256, 256)), ("layers_1.0.bias", (256,)),
    ("layers_1.2.weight", (256, 256)), ("layers_1.2.bias", (256,)),
    ("sigma_fc.0.weight", (1, 256)), ("sigma_fc.0.bias", (1,)),
    ("layers_2.weight", (256, 256)), ("layers_2.bias", (256,)),
    ("color_fc.0.weight", (128, 283)), ("color_fc.0.bias", (128,)),
    ("color_fc.2.weight", (3, 128)), ("color_fc.2.bias", (3,)),
]
PARAM_NAMES = [n for n, _ in PARAM_SHAPES]
NUM_PARAMS = sum(int(np.prod(s)) for _, s in PARAM_SHAPES)  # 595,844


# ----------------------------------------------------------------------------- rays
def rays_single_cam(H: int, W: int, f: float) -> np.ndarray:
    """utils/xyz.py:38-52.  Camera-frame directions, [3, H*W] fp32, column h*W+w,
    dir = ((w - W//2)/f, -(h - H//2)/f, -1).  The reference divides int64 by a python
    float (promotes to the default float32 dtype) and casts with .float()."""
    hl = np.arange(H, dtype=np.int64) - H // 2
    wl = np.arange(W, dtype=np.int64) - W // 2
    gx = np.broadcast_to(wl[None, :], (H, W)).astype(np.float32)   # w along columns
    gy = np.broadcast_to(hl[:, None], (H, W)).astype(np.float32)
    f32 = np.float32(f)
    out = np.stack([gx / f32, -(gy / f32), -np.ones((H, W), np.float32)]).astype(np.float32)
    return out.reshape(3, H * W)


def world_rays(poses: np.ndarray, cam_dirs: np.ndarray) -> np.ndarray:
    """utils/rendering.py:129-134 (same math utils/dataload.py:123-127).
    poses [P,4,4] fp32, cam_dirs [3,HW] -> rays [P*HW, 6] = (origin, R @ dir)."""
    poses = np.asarray(poses, np.float32)
    d = np.matmul(poses[:, :3, :3], cam_dirs.astype(np.float32))         # [P,3,HW]
    o = np.broadcast_to(poses[:, :3, 3:4], d.shape)
    return np.concatenate([o, d], axis=1).transpose(0, 2, 1).reshape(-1, 6).astype(np.float32)


def torch_linspace_f32(start: float, end: float, steps: int) -> np.ndarray:
    """torch.linspace's fp32 CPU algorithm (used by utils/rendering.py:25): symmetric evaluation
    from both ends, step=(end-start)/(steps-1) in fp32, each value one fused multiply-add
    (verified bit-exact against torch 2.11 for N+1 in {8,34,51,65,101,129})."""
    start32, end32 = np.float32(start), np.float32(end)
    step = np.float64(np.float32((end32 - start32) / np.float32(steps - 1)))
    i = np.arange(steps)
    half = steps // 2
    lo = (np.float64(start32) + step * i).astype(np.float32)             # fma(step, i, start)
    hi = (np.float64(end32) - step * (steps - 1 - i)).astype(np.float32)  # fma(-step, n-1-i, end)
    return np.where(i < half, lo, hi).astype(np.float32)


def stratified_ts(u: np.ndarray, N: int, tn: float = 2.0, tf: float = 6.0) -> np.ndarray:
    """utils/rendering.py:25-29.  ts = bin_diff * u + t_bins[:-1] (two roundings, no fma)."""
    t_bins = torch_linspace_f32(tn, tf, N + 1)
    bin_diff = np.float32(t_bins[1] - t_bins[0])
    return ((bin_diff * u.astype(np.float32)).astype(np.float32) + t_bins[None, :-1]).astype(np.float32)


def sample_points(rays: np.ndarray, ts: np.ndarray, dtype=np.float32):
    """utils/rendering.py:31-40.  p = o + t*d with UN-normalised d; view dir = d/||d||.
    Returns query_pts [B*N,6] and the normalised dirs [B,3]."""
    rays = rays.astype(dtype); ts = ts.astype(dtype)
    o, d = rays[:, :3], rays[:, 3:]
    locs = o[:, :, None] + d[:, :, None] * ts[:, None, :]                  # [B,3,N]
    dn = d / np.sqrt(np.sum(d * d, axis=1, keepdims=True))
    B, N = ts.shape
    q = np.concatenate([locs, np.broadcast_to(dn[:, :, None], (B, 3, N))], axis=1)
    return q.transpose(0, 2, 1).reshape(-1, 6).astype(dtype), dn.astype(dtype)


# ------------------------------------------------------------------------- encoding
def gamma(x: np.ndarray, L: int) -> np.ndarray:
    """utils/xyz.py:6-14.  [sin(2^0 x), cos(2^0 x), ..., sin(2^(L-1) x), cos(2^(L-1) x)], no pi."""
    cols = []
    for i in range(L):
        a = (x.dtype.type(2 ** i)) * x
        cols += [np.sin(a), np.cos(a)]
    return np.concatenate(cols, axis=1)


def positional_encoder(v: np.ndarray, Lp: int = 10, Ld: int = 4):
    """utils/xyz.py:16-36.  posx = [x,y,z,g(x),g(y),g(z)] (3+6Lp), posd likewise (3+6Ld)."""
    c = [v[:, i:i + 1] for i in range(6)]
    posx = np.concatenate(c[0:3] + [gamma(c[0], Lp), gamma(c[1], Lp), gamma(c[2], Lp)], axis=1)
    posd = np.concatenate(c[3:6] + [gamma(c[3], Ld), gamma(c[4], Ld), gamma(c[5], Ld)], axis=1)
    return posx, posd


# ------------------------------------------------------------------------------ MLP
def _lin(x, w, b):
    return x @ w.T + b


def mlp_forward(v: np.ndarray, P: dict, Lp: int = 10, Ld: int = 4, dtype=np.float32,
                keep: bool = False):
    """utils/nets.py:34-43.  v [M,6] -> [M,4] = (r,g,b,sigma) raw.  Skip concat is [h, posx]
    (:38), colour concat [g, posd] (:42), sigma read before layers_2 (:40-41), no output
    activations.  With keep=True also returns the saved tensors the backward needs."""
    P = {k: np.asarray(a, dtype) for k, a in P.items()}
    v = v.astype(dtype)
    posx, posd = positional_encoder(v, Lp, Ld)
    acts = []
    h = posx
    for i in (0, 2, 4, 6, 8):
        h = np.maximum(_lin(h, P[f"layers_0.{i}.weight"], P[f"layers_0.{i}.bias"]), 0)
        acts.append(h)
    cat1 = np.concatenate([h, posx], axis=1)
    h = np.maximum(_lin(cat1, P["skip_conn_layer.0.weight"], P["skip_conn_layer.0.bias"]), 0)
    acts.append(h)
    for i in (0, 2):
        h = np.maximum(_lin(h, P[f"layers_1.{i}.weight"], P[f"layers_1.{i}.bias"]), 0)
        acts.append(h)
    sigma = _lin(h, P["sigma_fc.0.weight"], P["sigma_fc.0.bias"])
    g = _lin(h, P["layers_2.weight"], P["layers_2.bias"])
    cat2 = np.concatenate([g, posd], axis=1)
    c1 = np.maximum(_lin(cat2, P["color_fc.0.weight"], P["color_fc.0.bias"]), 0)
    rgb = _lin(c1, P["color_fc.2.weight"], P["color_fc.2.bias"])
    out = np.concatenate([rgb, sigma], axis=1).astype(dtype)
    if keep:
        return out, dict(posx=posx, posd=posd, acts=acts, g=g, c1=c1)
    return out


def mlp_backward(d_out: np.ndarray, saved: dict, P: dict, dtype=np.float32) -> dict:
    """Analytic gradient of mlp_forward w.r.t. the 24 parameters (what autograd computes for
    train.py:54).  Inputs never require grad (utils/rendering.py:39-41), so no d/dv."""
    P = {k: np.asarray(a, dtype) for k, a in P.items()}
    d_out = d_out.astype(dtype)
    posx, posd, acts, g, c1 = saved["posx"], saved["posd"], saved["acts"], saved["g"], saved["c1"]
    G = {}
    d_rgb, d_sigma = d_out[:, :3], d_out[:, 3:4]
    G["color_fc.2.weight"] = d_rgb.T @ c1
    G["color_fc.2.bias"] = d_rgb.sum(0)
    d_c1 = (d_rgb @ P["color_fc.2.weight"]) * (c1 > 0)
    cat2 = np.concatenate([g, posd], axis=1)
    G["color_fc.0.weight"] = d_c1.T @ cat2
    G["color_fc.0.bias"] = d_c1.sum(0)
    d_g = d_c1 @ P["color_fc.0.weight"][:, :256]
    h7 = acts[7]
    G["layers_2.weight"] = d_g.T @ h7
    G["layers_2.bias"] = d_g.sum(0)
    G["sigma_fc.0.weight"] = d_sigma.T @ h7
    G["sigma_fc.0.bias"] = d_sigma.sum(0)
    d_h = (d_g @ P["layers_2.weight"] + d_sigma @ P["sigma_fc.0.weight"]) * (h7 > 0)
    # layers_1.2 (in acts[6] -> out acts[7]), layers_1.0 (acts[5] -> acts[6])
    for name, a_in in (("layers_1.2", acts[6]), ("layers_1.0", acts[5])):
        G[name + ".weight"] = d_h.T @ a_in
        G[name + ".bias"] = d_h.sum(0)
        d_h = (d_h @ P[name + ".weight"]) * (a_in > 0)
    # skip layer: input [acts[4], posx]
    cat1 = np.concatenate([acts[4], posx], axis=1)
    G["skip_conn_layer.0.weight"] = d_h.T @ cat1
    G["skip_conn_layer.0.bias"] = d_h.sum(0)
    d_h = (d_h @ P["skip_conn_layer.0.weight"][:, :256]) * (acts[4] > 0)
    for idx, a_in in ((8, acts[3]), (6, acts[2]), (4, acts[1]), (2, acts[0])):
        name = f"layers_0.{idx}"
        G[name + ".weight"] = d_h.T @ a_in
        G[name + ".bias"] = d_h.sum(0)
        d_h = (d_h @ P[name + ".weight"]) * (a_in > 0)
    G["layers_0.0.weight"] = d_h.T @ posx
    G["layers_0.0.bias"] = d_h.sum(0)
    return {k: G[k].astype(dtype).reshape(dict(PARAM_SHAPES)[k]) for k in PARAM_NAMES}


# ---------------------------------------------------------------------- compositing
def softplus(x, threshold=20.0):
    """torch.nn.functional.softplus(beta=1, threshold=20) as used at utils/rendering.py:67."""
    with np.errstate(over="ignore"):
        return np.where(x > threshold, x, np.log1p(np.exp(np.minimum(x, threshold))))


def volume_render(nerf_outs: np.ndarray, ts: np.ndarray, dirs: np.ndarray, dtype=np.float32):
    """utils/rendering.py:47-85.  Returns (rgb[B,3], disp[B], alpha[B,N], acc[B], weights[B,N]).
    dirs arrive already normalised from render_nerf (:37,43); the last delta is 1e10 (:61);
    +1e-10 inside the exclusive cumprod (:68); 2nd output is disparity (:82-83)."""
    o = nerf_outs.astype(dtype); ts = ts.astype(dtype); dirs = dirs.astype(dtype)
    deltas = ts[:, 1:] - ts[:, :-1]
    deltas = np.concatenate([deltas, np.full_like(deltas[:, :1], 1e10)], axis=1)
    deltas = deltas * np.sqrt(np.sum(dirs * dirs, axis=-1))[:, None]
    sigma = o[..., 3]
    with np.errstate(over="ignore", under="ignore"):
        alpha = 1 - np.exp(-softplus(sigma) * deltas)
        fac = np.concatenate([np.ones_like(alpha[:, :1]), 1 - alpha + dtype(1e-10)], axis=-1)
        T = np.cumprod(fac, axis=-1, dtype=dtype)[:, :-1]
    w = alpha * T
    rgb = np.sum(w[..., None] * o[..., :3], axis=1)
    depth = np.sum(w * ts, axis=-1)
    acc = np.sum(w, axis=-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        disp = 1.0 / np.maximum(dtype(1e-10), depth / acc)
    return (rgb.astype(dtype), disp.astype(dtype), alpha.astype(dtype), acc.astype(dtype),
            w.astype(dtype))


def volume_render_backward(nerf_outs, ts, dirs, d_rgb, d_disp=None, d_alpha=None, d_acc=None,
                           d_w=None, dtype=np.float32):
    """Analytic gradient of volume_render w.r.t. nerf_outs [B,N,4] (what autograd computes
    through utils/rendering.py:60-83; ts/dirs carry no grad).  The exclusive-cumprod backward is
    reverse_cumsum(grad*T)/factor, PyTorch's formula for zero-free inputs (factors are >= 1e-10).
    Without d_disp the disparity is not part of the graph, so a transparent ray (acc = 0) gets no NaN from it."""
    o = nerf_outs.astype(dtype); ts = ts.astype(dtype); dirs = dirs.astype(dtype)
    B, N = ts.shape
    z = lambda a, shp: np.zeros(shp, dtype) if a is None else a.astype(dtype)
    use_disp = d_disp is not None
    d_rgb = z(d_rgb, (B, 3)); d_disp = z(d_disp, (B,)); d_alpha = z(d_alpha, (B, N))
    d_acc = z(d_acc, (B,)); d_w = z(d_w, (B, N))
    deltas = ts[:, 1:] - ts[:, :-1]
    deltas = np.concatenate([deltas, np.full_like(deltas[:, :1], 1e10)], axis=1)
    deltas = deltas * np.sqrt(np.sum(dirs * dirs, axis=-1))[:, None]
    sigma = o[..., 3]
    sp = softplus(sigma)
    with np.errstate(over="ignore", under="ignore", invalid="ignore", divide="ignore"):
        e = np.exp(-sp * deltas)
        alpha = 1 - e
        f = 1 - alpha + dtype(1e-10)
        T = np.cumprod(np.concatenate([np.ones_like(alpha[:, :1]), f], -1), -1, dtype=dtype)[:, :-1]
        w = alpha * T
        depth = np.sum(w * ts, -1); acc = np.sum(w, -1)
        q = depth / acc
        m = np.maximum(dtype(1e-10), q)
        d_m = -d_disp / (m * m)
        d_q = np.where(q > 1e-10, d_m, 0)
        d_depth = d_q / acc if use_disp else np.zeros_like(acc)
        d_acc_t = d_acc - d_q * depth / (acc * acc) if use_disp else d_acc
        gw = (d_w + np.einsum("bnc,bc->bn", o[..., :3], d_rgb) + d_depth[:, None] * ts
              + d_acc_t[:, None])                      # total d(loss)/d(w_i)
        gwT = gw * w                                   # = d_T_i * T_i with d_T_i = gw_i*alpha_i
        S = np.cumsum(gwT[:, ::-1], axis=1)[:, ::-1] - gwT   # sum_{i>j}
        d_f = S / f
        d_a = d_alpha + gw * T - d_f
        d_sp = (d_a * e) * deltas                      # product order keeps 0*1e10 = 0
        zz = np.exp(np.minimum(sigma, 20))
        d_sigma = np.where(sigma > 20, d_sp, d_sp * zz / (zz + 1))
    d_out = np.concatenate([w[..., None] * d_rgb[:, None, :], d_sigma[..., None]], axis=-1)
    return d_out.astype(dtype)


# ------------------------------------------------------------------------- pipeline
def render_nerf(rays, P, N, u, tn=2.0, tf=6.0, Lp=10, Ld=4, dtype=np.float32, keep=False, ts=None):
    """utils/rendering.py:13-45 with the uniform jitter u[B,N] supplied by the caller (the
    reference draws it from the CPU global generator at :28).  `ts` [B,N] given: use these sample
    depths instead of lines :25-29 (checks of device-sampled batches, where u never exists on the host)."""
    ts = stratified_ts(u, N, tn, tf) if ts is None else np.asarray(ts, np.float32)
    q, dn = sample_points(rays, ts, dtype)
    res = mlp_forward(q, P, Lp, Ld, dtype, keep=keep)
    out, saved = res if keep else (res, None)
    B = rays.shape[0]
    outs = volume_render(out.reshape(B, N, 4), ts, dn, dtype)
    if keep:
        return outs, dict(ts=ts, dn=dn, out=out.reshape(B, N, 4), mlp=saved)
    return outs


def train_step_grads(rays, P, N, u, gt, dtype=np.float32, ts=None):
    """train.py:51-54: loss = mean((rgb - gt)^2) over B*3; returns (loss, grads dict, rgb)."""
    outs, sv = render_nerf(rays, P, N, u, dtype=dtype, keep=True, ts=ts)
    rgb = outs[0]
    diff = rgb - gt.astype(dtype)
    loss = np.mean(diff * diff)
    d_rgb = (2.0 / diff.size) * diff
    d_out = volume_render_backward(sv["out"], sv["ts"], sv["dn"], d_rgb, dtype=dtype)
    grads = mlp_backward(d_out.reshape(-1, 4), sv["mlp"], P, dtype)
    return float(loss), grads, rgb


# ------------------------------------------------- hierarchical sampling (EXTENSION)
def sample_pdf_merge(ts, weights, u, dtype=np.float32):
    """Inverse-CDF importance sampling + sorted merge.  NOT in the reference ("coarse and fine is
    not implemented yet", configs/lego.yaml:7): restates Mildenhall et al. 2020 sec. 5.2 / the
    paper's public sample_pdf -- parity unpinned by the reference.
    ts, weights [B,Nc]; u [B,Nf] in [0,1)  ->  ascending depths [B, Nc+Nf]."""
    ts = ts.astype(dtype); weights = weights.astype(dtype); u = u.astype(dtype)
    bins = dtype(0.5) * (ts[:, 1:] + ts[:, :-1])                        # Nc-1 mid points
    w = weights[:, 1:-1] + dtype(1e-5)                                   # Nc-2 interior weights
    pdf = w / np.sum(w, axis=-1, keepdims=True)
    cdf = np.concatenate([np.zeros_like(pdf[:, :1]), np.cumsum(pdf, axis=-1, dtype=dtype)], axis=-1)  # Nc-1
    B, nb = cdf.shape
    out = np.empty((B, u.shape[1]), dtype)
    for b in range(B):
        inds = np.searchsorted(cdf[b], u[b], side="right")
        below = np.maximum(0, inds - 1)
        above = np.minimum(nb - 1, inds)
        c0, c1 = cdf[b][below], cdf[b][above]
        denom = c1 - c0
        denom = np.where(denom < 1e-5, dtype(1), denom)
        t = (u[b] - c0) / denom
        out[b] = bins[b][below] + t * (bins[b][above] - bins[b][below])
    return np.sort(np.concatenate([ts, out], axis=-1), axis=-1).astype(dtype)


# ------------------------------------------------------------------ synthetic inputs
def spherical_to_pose(r, theta_deg, phi_deg):
    """utils/xyz.py:55-81: pose = phi_mat @ theta_mat @ trans_mat (float64, cast by callers)."""
    th, ph = np.radians(theta_deg), np.radians(phi_deg)
    trans = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, r], [0, 0, 0, 1.0]])
    tm = np.array([[1, 0, 0, 0], [0, np.cos(th), np.sin(th), 0], [0, -np.sin(th), np.cos(th), 0],
                   [0, 0, 0, 1.0]])
    pm = np.array([[np.cos(ph), np.sin(ph), 0, 0], [-np.sin(ph), np.cos(ph), 0, 0], [0, 0, 1.0, 0],
                   [0, 0, 0, 1.0]])
    return pm @ tm @ trans


def poses_to_render(r, theta, n_phi=40):
    """utils/xyz.py:83-91: azimuths linspace(0,360,n_phi) inclusive, fp32 poses."""
    return [spherical_to_pose(r, theta, p).astype(np.float32) for p in np.linspace(0, 360.0, n_phi)]


def adam_step(param, grad, m, v, t, lr=5e-4, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam(lr=5e-4) single step (train.py:43,55; no weight decay / amsgrad), t 1-based:
    m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)."""
    g = grad.astype(np.float64)
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    denom = np.sqrt(v) / np.sqrt(1 - b2 ** t) + eps
    return (param.astype(np.float64) - (lr / (1 - b1 ** t)) * m / denom).astype(np.float32), m, v


def init_params(seed: int = 0) -> dict:
    """Deterministic numpy-only stand-in for `torch.manual_seed(s); Nerf()` default init
    (U(+-1/sqrt(fan_in)) for weight and bias, nn.Linear).  NOT bit-identical to torch's RNG --
    parity tests take weights from the torch module; this is for the CPU baseline legs."""
    rng = np.random.default_rng(seed)
    P = {}
    for name, shp in PARAM_SHAPES:
        if name.endswith("weight"):
            bound = 1.0 / np.sqrt(shp[1]); last = bound
        else:
            bound = last
        P[name] = rng.uniform(-bound, bound, size=shp).astype(np.float32)
    return P
