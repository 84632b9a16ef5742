"""Lane-faithful restatement of the warp compositing kernels -- TEST INFRASTRUCTURE ONLY.

`composite_fwd_kernel` / `composite_bwd_kernel` (nerf_simple_b200/csrc/composite.cu) give one warp to a ray:
lane l owns the S consecutive samples l*S .. l*S+S-1 (S = the dispatch's 1, 2, 3, 4, 6 or 8; N <= 32*S), the
transmittance is a per-lane running product followed by an exclusive warp scan, and the backward's
sum_{i>j} gw_i w_i is a per-lane suffix plus a warp suffix scan minus the lane's own tail.  N > 256 runs the
thread-per-ray kernels, restated here as one lane that owns the whole ray.

This module computes the same quantities in that layout, vectorised over rays, so that a single planted bug
(`mutate`) changes the result exactly where the same bug in the kernel would:
  1  the delta at a lane boundary uses the lane's own t (delta = 0)
  2  ragged N: the 1e10 delta goes to slot 32*S-1 instead of N-1
  3  the exclusive transmittance scan is shifted by one lane
  4  the backward suffix includes the lane's own tail (later = q)
  5  no series branch: lg2(1 + z) of the fp32 sum 1 + z for every z
  6  d_acc is dropped when d_disp is null
  7  d_w and d_alpha are read with row stride 32*S instead of N
  8  disparity without NaN propagation (fmaxf(1e-10, NaN) = 1e-10)

`approx=True` is the noise model of the MUFU units: every ex2 / lg2 result is multiplied by 1 + u * 2^-21 with
a seeded u in {-1, +1}, and log2(1 + z) below z = 1e-2 is the kernel's three-term series.  With approx=False
everything is exact in `dtype` (float64 by default), which is what oracle/nerf_oracle.py computes.
"""
from __future__ import annotations

import numpy as np

LOG2E = 1.4426950408889634
MUTATIONS = {
    1: "delta at a lane boundary uses the lane's own t (delta = 0)",
    2: "ragged N: the 1e10 delta goes to slot 32*S-1 instead of N-1",
    3: "exclusive transmittance scan shifted by one lane",
    4: "backward suffix includes the lane's own tail (later = q)",
    5: "no series branch: lg2(1 + z) for every z",
    6: "d_acc dropped when d_disp is null",
    7: "d_w / d_alpha read with row stride 32*S instead of N",
    8: "disparity without NaN propagation (fmaxf(1e-10, NaN) = 1e-10)",
}
WARP_S = (1, 2, 3, 4, 6, 8)      # the S of nb200_composite_forward / _backward (csrc/composite.cu:565-570, 609-614)


def lanes_for(N: int):
    """(lanes, S) of the kernel that composites rays of N samples: a warp of 32 lanes with S samples per lane, or
    for N > 256 the thread-per-ray kernels (one lane owns all N samples)."""
    if N > 256:
        return 1, N
    return 32, next(s for s in WARP_S if 32 * s >= N)


def dir_norm(dirs, dirs_mode, dtype=np.float64):
    """|dir| as the reference sees it (utils/rendering.py:62): dirs_mode 0 takes dirs [B,3] as given, dirs_mode 1
    normalises the direction of the rays [B,6] first (:37) and takes the norm of that."""
    d = np.asarray(dirs, dtype)
    if dirs_mode == 1:
        d = d[:, 3:6]
        d = d / np.sqrt(np.sum(d * d, axis=1, keepdims=True))
    return np.sqrt(np.sum(d * d, axis=1))


class _Mufu:
    """ex2 / lg2, exact or with the seeded relative error of the approximate hardware instructions."""

    def __init__(self, approx, seed, dtype):
        self.rng = np.random.default_rng(seed) if approx else None
        self.dtype = dtype

    def _noise(self, x):
        if self.rng is None:
            return x
        u = self.rng.choice(np.array([-1.0, 1.0]), size=x.shape)
        return (x * (1.0 + u * 2.0 ** -21)).astype(self.dtype)

    def ex2(self, x):
        with np.errstate(over="ignore", under="ignore"):
            return self._noise(np.exp2(x))

    def log2_1p(self, z):
        with np.errstate(over="ignore"):
            return self._noise(np.log1p(z) * self.dtype(LOG2E))


def _setup(outs, ts, dirs, dirs_mode, mutate, dtype):
    """Pad the rays to lanes*S slots and lay them out as [B, lanes, S]."""
    o = np.asarray(outs, dtype)
    t = np.asarray(ts, dtype)
    B, N = t.shape
    lanes, S = lanes_for(N)
    P = lanes * S
    op = np.zeros((B, P, 4), dtype)
    tp = np.zeros((B, P), dtype)
    op[:, :N] = o
    tp[:, :N] = t
    idx = np.arange(P)
    valid = idx < N
    tl = tp.reshape(B, lanes, S)
    # t of the next sample: a register inside the lane, lane l+1's first t at j = S-1 (__shfl_down_sync; lane 31
    # gets its own value back)
    tn = np.empty_like(tl)
    tn[:, :, :-1] = tl[:, :, 1:]
    nxt = np.concatenate([tl[:, 1:, 0], tl[:, -1:, 0]], axis=1)
    tn[:, :, -1] = tl[:, :, -1] if mutate == 1 else nxt
    tn = tn.reshape(B, P)
    full = N == P
    last = idx == (P - 1 if (mutate == 2 and not full) else N - 1)
    with np.errstate(invalid="ignore", over="ignore"):
        d = np.where(last[None, :], dtype(1e10), tn - tp)
        delta = d * dir_norm(dirs, dirs_mode, dtype)[:, None]
    return op, tp, delta, valid, (B, N, lanes, S)


def _transmit(sigma, delta, mufu, mutate, dtype):
    """exp(-softplus(sigma) * delta) as transmit_factor computes it (csrc/stream_common.cuh:100-107)."""
    s2 = sigma * dtype(LOG2E)
    z = mufu.ex2(np.minimum(s2, dtype(200.0)))
    if mutate == 5:
        lg = np.log2((np.float32(1.0) + z.astype(np.float32)).astype(dtype))
    elif mufu.rng is not None:
        series = z * (dtype(LOG2E) + z * (dtype(-LOG2E / 2) + z * dtype(LOG2E / 3)))
        lg = np.where(z < 1e-2, series, mufu.log2_1p(z))
    else:
        lg = mufu.log2_1p(z)
    L = np.where(sigma > 20, s2, lg)
    with np.errstate(invalid="ignore", over="ignore"):
        return mufu.ex2(-L * delta)


def _scan(op, delta, valid, shape, mufu, mutate, dtype):
    """alpha, factor, exclusive transmittance T and weights in the lane layout."""
    B, N, lanes, S = shape
    e = _transmit(op[..., 3], delta, mufu, mutate, dtype)
    e = np.where(valid[None, :], e, dtype(1))
    a = np.where(valid[None, :], 1 - e, dtype(0))
    fac = np.where(valid[None, :], (1 - a) + dtype(1e-10), dtype(1))
    fl = fac.reshape(B, lanes, S)
    with np.errstate(under="ignore"):
        pre = np.cumprod(np.concatenate([np.ones((B, lanes, 1), dtype), fl[:, :, :-1]], axis=2), axis=2)
        run = np.prod(fl, axis=2)                                                    # per-lane product
        ex = np.cumprod(np.concatenate([np.ones((B, 1), dtype), run[:, :-1]], axis=1), axis=1)   # exclusive scan
    if mutate == 3:
        ex = np.concatenate([np.ones((B, 1), dtype), ex[:, :-1]], axis=1)
    T = (ex[:, :, None] * pre).reshape(B, lanes * S)
    w = a * T
    return e, a, fac, T, w


def _disparity(depth, acc, mutate):
    with np.errstate(divide="ignore", invalid="ignore"):
        q = depth / acc
        m = np.fmax(1e-10, q) if mutate == 8 else np.where(np.isnan(q), q, np.fmax(1e-10, q))
        return 1.0 / m


def forward(outs, ts, dirs, dirs_mode=0, approx=False, seed=0, mutate=None, dtype=np.float64):
    """composite_fwd_kernel / composite_fwd_serial_kernel.  Returns (rgb, disp, acc, alpha, weights) like
    nerf_oracle.volume_render (whose order is rgb, disp, alpha, acc, weights)."""
    dtype = np.dtype(dtype).type
    mufu = _Mufu(approx, seed, dtype)
    op, tp, delta, valid, shape = _setup(outs, ts, dirs, dirs_mode, mutate, dtype)
    B, N = shape[:2]
    e, a, fac, T, w = _scan(op, delta, valid, shape, mufu, mutate, dtype)
    rgb = np.sum(w[..., None] * op[..., :3], axis=1)
    depth = np.sum(w * tp, axis=1)
    acc = np.sum(w, axis=1)
    return rgb, _disparity(depth, acc, mutate), acc, a[:, :N], w[:, :N]


def backward(outs, ts, dirs, d_rgb, d_disp=None, d_acc=None, d_alpha=None, d_w=None, dirs_mode=0,
             approx=False, seed=0, mutate=None, dtype=np.float64):
    """composite_bwd_kernel / composite_bwd_serial_kernel: d(loss)/d(outs) [B,N,4]."""
    dtype = np.dtype(dtype).type
    mufu = _Mufu(approx, seed, dtype)
    op, tp, delta, valid, shape = _setup(outs, ts, dirs, dirs_mode, mutate, dtype)
    B, N, lanes, S = shape
    P = lanes * S
    e, a, fac, T, w = _scan(op, delta, valid, shape, mufu, mutate, dtype)

    def per_sample(x):           # [B,N] cotangent -> [B,P] as the kernel reads it
        x = np.asarray(x, dtype)
        if mutate == 7:
            flat = x.ravel()
            at = np.arange(B)[:, None] * P + np.arange(P)[None, :]
            return np.where(at < flat.size, flat[np.minimum(at, flat.size - 1)], dtype(0))
        out = np.zeros((B, P), dtype)
        out[:, :N] = x
        return out

    g = np.asarray(d_rgb, dtype)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        gw = op[..., 0] * g[:, 0:1] + op[..., 1] * g[:, 1:2] + op[..., 2] * g[:, 2:3]
        g_acc = np.zeros(B, dtype) if d_acc is None or (mutate == 6 and d_disp is None) else np.asarray(d_acc, dtype)
        g_depth = np.zeros(B, dtype)
        if d_disp is not None:
            depth = np.sum(w * tp, axis=1)
            acc = np.sum(w, axis=1)
            q = depth / acc
            m = np.fmax(dtype(1e-10), q)
            g_q = np.where(q > 1e-10, -np.asarray(d_disp, dtype) / (m * m), dtype(0))
            g_depth = g_q / acc
            g_acc = g_acc - g_q * depth / (acc * acc)
        gw = gw + g_depth[:, None] * tp + g_acc[:, None]
        if d_w is not None:
            gw = gw + np.where(valid[None, :], per_sample(d_w), dtype(0))
        contrib = np.where(valid[None, :], gw * w, dtype(0)).reshape(B, lanes, S)
        # per-lane suffix over the later samples of the lane, then the inclusive warp suffix scan
        suf = np.flip(np.cumsum(np.flip(contrib, 2), axis=2), 2) - contrib        # sum over j' > j in the lane
        tail = np.sum(contrib, axis=2)
        q_incl = np.flip(np.cumsum(np.flip(tail, 1), axis=1), 1)
        later = q_incl if mutate == 4 else q_incl - tail
        Sj = (later[:, :, None] + suf).reshape(B, P)
        g_a = gw * T - Sj / fac
        if d_alpha is not None:
            g_a = g_a + np.where(valid[None, :], per_sample(d_alpha), dtype(0))
        g_sp = (g_a * e) * delta
        sig = op[..., 3]
        z = mufu.ex2(np.minimum(sig, dtype(20)) * dtype(LOG2E))
        g_sigma = np.where(sig > 20, g_sp, g_sp * (z / (z + 1)))
    d_outs = np.concatenate([w[..., None] * g[:, None, :], g_sigma[..., None]], axis=-1)
    return d_outs[:, :N]
