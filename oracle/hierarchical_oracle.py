"""CPU oracle of one hierarchical training step -- TEST INFRASTRUCTURE ONLY.

Hierarchical (coarse + fine) sampling is an EXTENSION: the reference has none ("coarse and fine is not implemented
yet", configs/lego.yaml:7), so this restates the NeRF paper's scheme (Mildenhall et al. 2020, sec. 5.2) on top of the
reference-pinned pieces of oracle/nerf_oracle.py (render_nerf, volume_render_backward, mlp_backward through
train_step_grads) -- parity unpinned by the reference.  `render_nerf_torch` is the torch-CPU port of
oracle/nerf_oracle_torch.py with the sample depths given, so that autograd can check the analytic gradients of a fine
pass.  The product path (nerf_simple_b200) never imports this module.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle import nerf_oracle as O
from oracle import nerf_oracle_torch as OT


def hierarchical_train_step_grads(rays, P_c, P_f, Nc, u_c, z, gt, dtype=np.float32, ts=None):
    """loss = MSE(rgb_coarse, gt) + MSE(rgb_fine, gt): the coarse net renders the Nc stratified depths of u_c [B,Nc]
    (or `ts` [B,Nc]), the fine net the merged depths z [B,Nc+Nf].  z is an input because no gradient flows through the
    sampler: a check feeds the depths its own sampler drew (sample_pdf_merge on the coarse weights).
    Returns (loss_coarse, loss_fine, coarse grads dict, fine grads dict)."""
    loss_c, grads_c, _ = O.train_step_grads(rays, P_c, Nc, u_c, gt, dtype=dtype, ts=ts)
    z = np.asarray(z, np.float32)
    loss_f, grads_f, _ = O.train_step_grads(rays, P_f, z.shape[1], None, gt, dtype=dtype, ts=z)
    return loss_c, loss_f, grads_c, grads_f


def render_nerf_torch(rays, P, ts):
    """oracle/nerf_oracle_torch.render_nerf with the sample depths ts [B,N] given, in the dtype of the inputs.
    Returns (rgb, disp, alpha, acc, weights)."""
    B, N = ts.shape
    o, d = rays[:, :3], rays[:, 3:]
    locs = o.unsqueeze(-1) + d.unsqueeze(-1) * ts.unsqueeze(1)
    dn = d / torch.norm(d, dim=1, keepdim=True)
    q = torch.cat((locs, dn.unsqueeze(-1).expand(-1, -1, N)), dim=1).permute(0, 2, 1).reshape(-1, 6)
    out = OT.mlp(q, P).reshape(B, N, 4)
    deltas = torch.cat((ts[:, 1:] - ts[:, :-1], 1e10 * torch.ones_like(ts[:, :1])), dim=1)
    deltas = deltas * torch.norm(dn[..., None, :], dim=-1)
    alpha = 1 - torch.exp(-F.softplus(out[..., 3]) * deltas)
    T = torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1. - alpha + 1e-10], -1), -1)[:, :-1]
    w = alpha * T
    rgb = torch.sum(w.unsqueeze(-1) * out[..., :3], dim=1)
    depth = torch.sum(w * ts, dim=-1)
    acc = torch.sum(w, dim=-1)
    disp = 1. / torch.max(1e-10 * torch.ones_like(depth), depth / acc)
    return rgb, disp, alpha, acc, w
