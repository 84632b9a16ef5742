"""CPU checks of the hierarchical training step (EXTENSION: the NeRF paper's coarse + fine scheme, which the reference
does not implement): the float64 oracle of one step against torch autograd, and the one flat parameter / gradient
buffer that both networks share in the device-resident Trainer."""
import numpy as np
import torch

from conftest import load_golden
from oracle import hierarchical_oracle as H
from oracle import nerf_oracle as O


def test_hierarchical_step_oracle_matches_torch_autograd(golden_weights):
    """hierarchical_train_step_grads (analytic, float64) == autograd through MSE(coarse) + MSE(fine) in float64, for
    both networks, with the fine depths drawn by the oracle's sampler from the coarse weights."""
    g = load_golden("case_train_b64_n64.npz")
    B, Nc, Nf = 64, 64, 128
    rays, gt, u_c = g["rays"], g["gt"], g["u"]
    P_c, P_f = golden_weights, O.init_params(1)
    u_f = np.random.default_rng(4).random((B, Nf)).astype(np.float32)
    w_c = O.render_nerf(rays, P_c, Nc, u_c)[4]
    z = O.sample_pdf_merge(O.stratified_ts(u_c, Nc), w_c, u_f)
    loss_c, loss_f, G_c, G_f = H.hierarchical_train_step_grads(rays, P_c, P_f, Nc, u_c, z, gt, dtype=np.float64)

    # the torch port with given depths reproduces the reference's outputs on the golden depths
    with torch.no_grad():
        rgb, _, alpha, _, w = H.render_nerf_torch(torch.from_numpy(rays), {k: torch.from_numpy(v) for k, v in P_c.items()},
                                                  torch.from_numpy(g["ts"]))
    assert np.abs(rgb.numpy() - g["rgb"]).max() <= 1e-6 and np.abs(w.numpy() - g["weights"]).max() <= 1e-6

    T = lambda a: torch.from_numpy(np.asarray(a, np.float64))
    Tc = {k: T(v).requires_grad_(True) for k, v in P_c.items()}
    Tf = {k: T(v).requires_grad_(True) for k, v in P_f.items()}
    ts = T(O.stratified_ts(u_c, Nc))
    rgb_c = H.render_nerf_torch(T(rays), Tc, ts)[0]
    rgb_f = H.render_nerf_torch(T(rays), Tf, T(z))[0]
    lc = torch.nn.functional.mse_loss(rgb_c, T(gt))
    lf = torch.nn.functional.mse_loss(rgb_f, T(gt))
    (lc + lf).backward()
    assert abs(loss_c - lc.item()) <= 1e-9 * abs(lc.item()) and abs(loss_f - lf.item()) <= 1e-9 * abs(lf.item())
    for G, P in ((G_c, Tc), (G_f, Tf)):
        for k in O.PARAM_NAMES:
            ref = P[k].grad.numpy()
            assert G[k].shape == ref.shape
            assert np.max(np.abs(G[k] - ref)) <= 1e-9 * max(1e-30, float(np.abs(ref).max())), k
    # the fine net's gradient is its own: the coarse pass alone leaves it untouched
    assert all(float(np.abs(G_f[k]).max()) > 0 for k in O.PARAM_NAMES)


def test_two_networks_share_one_flat_buffer():
    """flatten_parameters / attach_flat_grad over two networks: 48 aligned views of one buffer, each network's
    state_dict keeps its 24 keys, shapes and values, and the padding stays zero."""
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.ops import NUM_PARAMS
    from nerf_simple_b200.trainer import attach_flat_grad, flatten_parameters
    torch.manual_seed(0)
    a, b = Nerf(), Nerf()
    sd_a = {k: v.clone() for k, v in a.state_dict().items()}
    sd_b = {k: v.clone() for k, v in b.state_dict().items()}
    flat = flatten_parameters(a, b)
    grad = attach_flat_grad(a, b)
    assert flat.numel() == grad.numel() and flat.numel() % 4 == 0 and flat.numel() >= 2 * NUM_PARAMS
    for net, sd in ((a, sd_a), (b, sd_b)):
        now = net.state_dict()
        assert list(now) == list(sd) and len(now) == 24
        assert all(torch.equal(now[k], sd[k]) for k in sd)
    base, gbase = flat.data_ptr(), grad.data_ptr()
    params = list(a.parameters()) + list(b.parameters())
    for p in params:
        assert p.is_contiguous() and (p.data_ptr() - base) % 16 == 0 and base <= p.data_ptr() < base + 4 * flat.numel()
        assert p.grad.shape == p.shape and (p.grad.data_ptr() - gbase) % 16 == 0
    assert len({p.data_ptr() for p in params}) == 48
    covered = torch.zeros(flat.numel(), dtype=torch.bool)
    for p in params:
        o = (p.data_ptr() - base) // 4
        covered[o:o + p.numel()] = True
    assert int(covered.sum()) == 2 * NUM_PARAMS and not bool(flat[~covered].any())
    grad.fill_(1.0)
    assert all(float(p.grad.min()) == 1.0 for p in params)
