"""Emulation of the two tcgen05 bf16 chains (NB200_BF16 folded, NB200_BF16_LAYERWISE) -- TEST INFRASTRUCTURE ONLY.

The numpy oracle (oracle/nerf_oracle.py) restates the reference in fp32 / float64; against it a bf16 kernel can only
be held to a bound that leaves room for all of the bf16 error.  This module does the SAME operation as the kernels:
it rounds to bf16 (round-to-nearest-even) exactly where they round and computes everything else in float64, so what
is left between a correct kernel and this emulation is fp32 accumulation-order noise.  The rounding points, from the
kernels:

  encoding     csrc/mlp_tc.cu encode_row: level 0 = sincosf, higher levels the fp32 double-angle recurrence
               (s' = 2 s c, c' = fma(-2s, s, 1)); posx / posd columns rounded to bf16.  Rays mode: the query point
               o + d t and the view direction d / |d| formed in fp32 as in mlp_chain.cuh load_query_chain.
  weights      bf16 images (pack_slabs_kernel).  Folded: Wf = Wc0[:, :256] Wg formed in fp32 and rounded once; the
               folded bias bf = Wc0[:, :256] bg + bc0 stays fp32 (fold_weights_kernel).  w_sigma, color_fc.2 and all
               biases stay fp32.
  hidden       mlp_chain.cuh epi_cols16: fp32 accumulator + fp32 bias, ReLU fused into the bf16 conversion;
               layers_2 (layer-wise chain only) is rounded without ReLU.
  sigma head   CUDA cores, from the UNROUNDED fp32 ReLU output of layers_1.2.
  colour head  color_fc.0 epilogue: c1 = ReLU(acc + bias) in fp32; color_fc.2 reads that fp32 c1; the saved c1
               (wgrad operand, ReLU mask) is bf16(c1).
  delta chain  DgradEpi: delta_c1 = bf16(d_rgb Wc1) masked by the bf16 c1; every delta rounded to bf16 and masked
               by the ReLU bit of the bf16 saved activation; delta_h7 also takes d_sigma w_sigma before rounding.
               Folded: delta_h7 = delta_c1 Wf (bf16 Wf); layer-wise: delta_g = bf16(delta_c1 Wc0[:, :256]) unmasked.
  wgrad        bf16 deltas x bf16 saved activations, fp32 accumulation; bias gradients = column sums of the bf16
               deltas; head gradients from the bf16 h7 / c1 and the fp32 d_out.
  un-folding   fold_grads_kernel, fp32: dWc0[:, :256] = Gm Wg^T + s bg^T, dWg = Wc0[:, :256]^T Gm,
               dbg = Wc0[:, :256]^T s, dbc0 = s  (Gm = delta_c1^T h7, s = column sums of delta_c1).

accum="fp32" runs the same rounding points with fp32 matrix products, and sums every weight / bias gradient per
128-row tile and then across tiles in a shuffled order, the way the wgrad kernel's fp32 atomics do.  Its distance
from the float64 emulation is the noise model the kernel-vs-emulation bounds of tests/test_bf16_chain.py start from.

`mutate` applies one deliberate bug inside the emulation (MUTATIONS); the tests use them to show that the bounds
would catch such a bug in a kernel.

Only tests/ may import this module; the product (nerf_simple_b200) never does.
"""
from __future__ import annotations

import numpy as np

from oracle.nerf_oracle import PARAM_NAMES, PARAM_SHAPES

MODES = ("bf16", "bf16_layerwise")
TILE = 128
LP, LD = 10, 4

# deliberate bugs, each one that a kernel change could plausibly introduce (see tests/test_bf16_chain.py)
MUTATIONS = {
    "swap_rows": "forward: two sample rows of one tile swapped in the color_fc.0 output",
    "zero_bias16": "forward: 16 biases (one epilogue step) of layers_0.4 zeroed",
    "zero_posd_col": "forward: one posd column zeroed",
    "fold_bias_bc0": "forward, folded chain: folded bias replaced by bc0 alone",
    "drop_tile": "backward: the deltas of one 128-row tile dropped",
    "drop_tail": "backward: the deltas of the ragged last tile dropped",
    "wrong_mask_h7": "backward: delta_h7 masked with the ReLU mask of h6",
}
SWAP_ROWS = (TILE + 5, TILE + 77)      # rows of tile 1
BIAS16 = slice(16, 32)
POSD_COL = 10
DROP_TILE = 1


def bf16(x) -> np.ndarray:
    """Round to bf16 (nearest even) through fp32, as the kernels' cvt.rn.bf16x2.f32 of an fp32 value; float32 out."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    b = (b + (np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1)))) & np.uint32(0xFFFF0000)
    return b.view(np.float32)


def f32(x) -> np.ndarray:
    return np.asarray(x, dtype=np.float32)


# ------------------------------------------------------------------------------------------ inputs
def query_from_rays(rays, ts) -> np.ndarray:
    """load_query_chain: v = o + d t (fp32 multiply, then fp32 add, no fma), dir = d * (1 / sqrtf(|d|^2)) with
    |d|^2 = fma(dz, dz, fma(dy, dy, dx dx)), all fp32.  rays [B,6], ts [B,N] -> [B*N, 6] fp32."""
    rays = f32(rays)
    ts = f32(ts)
    B, N = ts.shape
    o, d = rays[:, None, :3], rays[:, None, 3:]
    pos = f32(o + f32(d * ts[:, :, None]))
    dx, dy, dz = (rays[:, k].astype(np.float64) for k in (3, 4, 5))
    n2 = f32(dz * dz + f32(dy * dy + f32(dx * dx)))
    inv = f32(1.0 / np.sqrt(n2.astype(np.float64)).astype(np.float32).astype(np.float64))
    dn = f32(rays[:, 3:] * inv[:, None])
    q = np.concatenate([pos, np.broadcast_to(dn[:, None, :], (B, N, 3))], axis=2)
    return q.reshape(B * N, 6).astype(np.float32)


def encode(x, L) -> np.ndarray:
    """encode_row: [x0, x1, x2, per coordinate sin(2^i x), cos(2^i x) for i < L] in fp32, then rounded to bf16.
    Level 0 is sincosf (emulated as the correctly rounded fp32 sin / cos), the rest the fp32 recurrence."""
    x = f32(x)
    x64 = x.astype(np.float64)
    s, c = f32(np.sin(x64)), f32(np.cos(x64))
    levels = []
    for _ in range(L):
        levels.append((s, c))
        s2 = f32(2.0 * s.astype(np.float64) * c.astype(np.float64))          # (2 s) exact, one rounding
        c = f32(1.0 - 2.0 * s.astype(np.float64) * s.astype(np.float64))     # fma(-2s, s, 1): one rounding
        s = s2
    cols = [x[:, k] for k in range(3)]
    for k in range(3):
        for s_i, c_i in levels:
            cols += [s_i[:, k], c_i[:, k]]
    return bf16(np.stack(cols, axis=1))


# ----------------------------------------------------------------------------------------- weights
def pack(P: dict, mode: str) -> dict:
    """What the packed weight image holds: bf16 MMA operands, fp32 biases and head weights (and, folded, Wf / bf)."""
    if mode not in MODES:
        raise ValueError(mode)
    W = {k: f32(v) for k, v in P.items()}
    K = {}
    for name in ("layers_0.0", "layers_0.2", "layers_0.4", "layers_0.6", "layers_0.8", "skip_conn_layer.0",
                 "layers_1.0", "layers_1.2", "layers_2", "color_fc.0"):
        K[name + ".W"] = bf16(W[name + ".weight"]).astype(np.float64)
        K[name + ".b"] = W[name + ".bias"].astype(np.float64)
    Wc0g = W["color_fc.0.weight"][:, :256].astype(np.float64)
    K["Wf"] = bf16(f32(Wc0g @ W["layers_2.weight"].astype(np.float64))).astype(np.float64)
    K["bf"] = f32(Wc0g @ W["layers_2.bias"].astype(np.float64) + W["color_fc.0.bias"]).astype(np.float64)
    for k in ("sigma_fc.0.weight", "sigma_fc.0.bias", "color_fc.2.weight", "color_fc.2.bias", "layers_2.weight",
              "layers_2.bias", "color_fc.0.weight"):
        K[k] = W[k].astype(np.float64)
    return K


class _Arith:
    """float64 products (the emulation) or fp32 products (the noise model)."""

    def __init__(self, accum: str, seed: int = 0):
        if accum not in ("float64", "fp32"):
            raise ValueError(accum)
        self.fp32 = accum == "fp32"
        self.dt = np.float32 if self.fp32 else np.float64
        self.rng = np.random.default_rng(seed)

    def mm(self, a, b):          # a [M,K] @ b [K,N]
        return (np.asarray(a, self.dt) @ np.asarray(b, self.dt)).astype(np.float64)

    def lin(self, a, W, b):      # fp32 accumulator + fp32 bias -> fp32 value
        acc = np.asarray(a, self.dt) @ np.asarray(W, self.dt).T
        return f32(f32(acc) + f32(b)) if self.fp32 else f32(acc + b)

    def wsum(self, delta, act):
        """Sum over samples of delta^T act (weight gradient) or, act None, the column sums of delta (bias gradient)."""
        one = (lambda d, a: d.T @ a) if act is not None else (lambda d, a: d.sum(0))
        if not self.fp32:
            return one(np.asarray(delta, np.float64), None if act is None else np.asarray(act, np.float64))
        d32, a32 = f32(delta), None if act is None else f32(act)
        M = d32.shape[0]
        parts = [one(d32[t:t + TILE], None if a32 is None else a32[t:t + TILE]).astype(np.float32)
                 for t in range(0, M, TILE)]
        tot = np.zeros_like(parts[0])
        for i in self.rng.permutation(len(parts)):
            tot = f32(tot + parts[i])
        return tot.astype(np.float64)


# ----------------------------------------------------------------------------------------- forward
def forward(v_or_rays, ts, P: dict, mode: str, keep: bool = False, accum: str = "float64", mutate: str | None = None):
    """(r,g,b,sigma) [M,4] float64 as the bf16 chain `mode` computes it.  `ts` None: points mode, v [M,6]; else rays
    mode, rays [B,6] and sample depths ts [B,N].  keep=True also returns what the backward reads."""
    A = _Arith(accum)
    K = pack(P, mode)
    if mutate == "zero_bias16":
        K["layers_0.4.b"] = K["layers_0.4.b"].copy()
        K["layers_0.4.b"][BIAS16] = 0.0
    if mutate == "fold_bias_bc0":
        K["bf"] = f32(P["color_fc.0.bias"]).astype(np.float64)
    v = f32(v_or_rays) if ts is None else query_from_rays(v_or_rays, ts)
    posx, posd = encode(v[:, 0:3], LP), encode(v[:, 3:6], LD)
    if mutate == "zero_posd_col":
        posd = posd.copy()
        posd[:, POSD_COL] = 0.0
    h = posx
    acts = []
    for name in ("layers_0.0", "layers_0.2", "layers_0.4", "layers_0.6", "layers_0.8"):
        h = bf16(np.maximum(A.lin(h, K[name + ".W"], K[name + ".b"]), 0))
        acts.append(h)
    h = bf16(np.maximum(A.lin(np.concatenate([h, posx], 1), K["skip_conn_layer.0.W"], K["skip_conn_layer.0.b"]), 0))
    acts.append(h)
    h = bf16(np.maximum(A.lin(h, K["layers_1.0.W"], K["layers_1.0.b"]), 0))
    acts.append(h)
    x7 = np.maximum(A.lin(h, K["layers_1.2.W"], K["layers_1.2.b"]), 0)      # fp32, read by the sigma head
    h7 = bf16(x7)
    acts.append(h7)
    sigma = A.mm(x7, K["sigma_fc.0.weight"].T)[:, 0] + K["sigma_fc.0.bias"][0]
    g = None
    if mode == "bf16":
        W = np.concatenate([K["Wf"], K["color_fc.0.W"][:, 256:]], 1)
        c1 = np.maximum(A.lin(np.concatenate([h7, posd], 1), W, K["bf"]), 0)
    else:
        g = bf16(A.lin(h7, K["layers_2.W"], K["layers_2.b"]))
        c1 = np.maximum(A.lin(np.concatenate([g, posd], 1), K["color_fc.0.W"], K["color_fc.0.b"]), 0)
    if mutate == "swap_rows" and c1.shape[0] > max(SWAP_ROWS):
        c1 = c1.copy()
        c1[list(SWAP_ROWS)] = c1[list(SWAP_ROWS[::-1])]
    rgb = A.mm(c1, K["color_fc.2.weight"].T) + K["color_fc.2.bias"]
    out = np.concatenate([rgb, sigma[:, None]], 1)
    if keep:
        return out, dict(posx=posx, posd=posd, acts=acts, g=g, c1=bf16(c1), mode=mode)
    return out


def slice_saved(saved: dict, m: int) -> dict:
    """The saved tensors of the first m samples (the emulation is row-wise up to the gradient sums)."""
    cut = lambda a: None if a is None else a[:m]
    return dict(posx=saved["posx"][:m], posd=saved["posd"][:m], acts=[a[:m] for a in saved["acts"]],
                g=cut(saved["g"]), c1=saved["c1"][:m], mode=saved["mode"])


# ---------------------------------------------------------------------------------------- backward
def backward(d_out, saved: dict, P: dict, mode: str, accum: str = "float64", mutate: str | None = None) -> dict:
    """The 24 parameter gradients (float64, PARAM_SHAPES order and shapes) of sum(out * d_out) as the bf16 chain
    `mode` computes them from the saved tensors of forward(..., keep=True)."""
    if saved["mode"] != mode:
        raise ValueError(f"saved tensors of {saved['mode']}, backward of {mode}")
    A = _Arith(accum)
    K = pack(P, mode)
    d_out = f32(d_out).astype(np.float64)
    M = d_out.shape[0]
    posx, posd, acts, c1 = saved["posx"], saved["posd"], saved["acts"], saved["c1"]
    h7 = acts[7]
    d_rgb, d_sig = d_out[:, :3], d_out[:, 3:4]
    keep_rows = np.ones((M, 1))
    if mutate == "drop_tile":
        keep_rows[DROP_TILE * TILE:(DROP_TILE + 1) * TILE] = 0
    if mutate == "drop_tail":
        keep_rows[M - M % TILE:] = 0
    G = {}
    # color_fc.2 backward on CUDA cores (fp32 FMAs), rounded and masked by the bf16 c1
    d_c1 = bf16(f32(A.mm(d_rgb, K["color_fc.2.weight"]))) * (c1 > 0) * keep_rows
    sig_term = d_sig * K["sigma_fc.0.weight"] * keep_rows          # + d_sigma w_sigma before delta_h7's rounding
    mask7 = (acts[6] if mutate == "wrong_mask_h7" else h7) > 0
    if mode == "bf16":
        d_h = bf16(f32(A.mm(d_c1, K["Wf"]) + sig_term)) * mask7
        Gm = A.wsum(d_c1, h7)                     # one wgrad item; un-folded in fp32 (fold_grads_kernel)
        s = A.wsum(d_c1, None)
        Wg, bg, Wc0g = K["layers_2.weight"], K["layers_2.bias"], K["color_fc.0.weight"][:, :256]
        dWc0g = A.mm(Gm, Wg.T) + np.outer(s, bg)
        G["layers_2.weight"] = A.mm(Wc0g.T, Gm)
        G["layers_2.bias"] = A.mm(Wc0g.T, s[:, None])[:, 0]
        G["color_fc.0.bias"] = s
    else:
        d_g = bf16(f32(A.mm(d_c1, K["color_fc.0.W"][:, :256])))
        d_h = bf16(f32(A.mm(d_g, K["layers_2.W"]) + sig_term)) * mask7
        dWc0g = A.wsum(d_c1, saved["g"])
        G["color_fc.0.bias"] = A.wsum(d_c1, None)
        G["layers_2.weight"] = A.wsum(d_g, h7)
        G["layers_2.bias"] = A.wsum(d_g, None)
    G["color_fc.0.weight"] = np.concatenate([dWc0g, A.wsum(d_c1, posd)], 1)
    G["sigma_fc.0.weight"] = A.wsum(d_sig, h7)
    G["sigma_fc.0.bias"] = A.wsum(d_sig, None)
    G["color_fc.2.weight"] = A.wsum(d_rgb, c1)
    G["color_fc.2.bias"] = A.wsum(d_rgb, None)
    # d_h = delta at h7; walk down the chain: (layer, its input activation)
    chain = [("layers_1.2", acts[6]), ("layers_1.0", acts[5]), ("skip_conn_layer.0", acts[4]),
             ("layers_0.8", acts[3]), ("layers_0.6", acts[2]), ("layers_0.4", acts[1]), ("layers_0.2", acts[0])]
    for name, a_in in chain:
        x_in = np.concatenate([a_in, posx], 1) if name == "skip_conn_layer.0" else a_in
        G[name + ".weight"] = A.wsum(d_h, x_in)
        G[name + ".bias"] = A.wsum(d_h, None)
        d_h = bf16(f32(A.mm(d_h, K[name + ".W"][:, :256]))) * (a_in > 0)
    G["layers_0.0.weight"] = A.wsum(d_h, posx)
    G["layers_0.0.bias"] = A.wsum(d_h, None)
    shapes = dict(PARAM_SHAPES)
    return {k: np.asarray(G[k], np.float64).reshape(shapes[k]) for k in PARAM_NAMES}
