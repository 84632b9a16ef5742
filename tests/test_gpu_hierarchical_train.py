"""GPU tests of hierarchical training in the device-resident Trainer (EXTENSION: the NeRF paper's coarse + fine scheme,
sec. 5.2; the reference has none).  One step is checked against autograd through render_nerf_hierarchical and against
the float64 oracle, the graph-replayed step against the same step launched eagerly, and the replay-safe fine sampler
against its host-offset form."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import hierarchical_oracle as H
from oracle import nerf_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GRAD_ABS_X3, GRAD_REL_X3 = 1e-4, 2e-3      # the bf16x3 Trainer bounds of tests/test_gpu_bf16x3_train.py
GRAD_REL = {"fp32": 2e-3, "bf16": 5e-2}     # tests/test_gpu_parity.py::_grad_check


def maxabs(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return float(np.max(np.abs(a.astype(np.float64) - b.astype(np.float64))))


def make_net(P=None, seed=None):
    from nerf_simple_b200.nets import Nerf
    if seed is not None:
        torch.manual_seed(seed)
    n = Nerf().cuda()
    if P is not None:
        n.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)) for k, v in P.items()}, strict=True)
    return n


def fine_weights():
    torch.manual_seed(11)
    from nerf_simple_b200.nets import Nerf
    return {k: v.numpy().copy() for k, v in Nerf().state_dict().items()}


def golden_step_inputs():
    g = load_golden("case_train_b64_n64.npz")
    u_f = np.random.default_rng(4).random((64, 128)).astype(np.float32)
    return g, torch.from_numpy(g["rays"]).cuda(), torch.from_numpy(g["gt"]).cuda(), torch.from_numpy(g["ts"]).cuda(), u_f


def smooth_field(H=32, n_poses=4):
    from nerf_simple_b200 import ops
    from nerf_simple_b200.xyz import poses_to_render
    poses = torch.stack(poses_to_render(4, -30, n_poses)).cuda()
    rays = ops.generate_rays(poses, H, H, 44.4)
    return poses, rays, torch.sigmoid(rays[:, 3:6] * 3)


# ------------------------------------------------------------------------------------- 1. the state-form sampler
@pytest.mark.parametrize("Nc,Nf", [(64, 128), (32, 64), (17, 23)])
def test_sample_pdf_merge_state_matches_host_offset_form(Nc, Nf):
    from nerf_simple_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(Nc + Nf)
    B = 301
    ts = torch.from_numpy(np.sort(2 + 4 * rng.random((B, Nc)), axis=1).astype(np.float32)).cuda()
    w = torch.from_numpy((0.05 + rng.random((B, Nc)) ** 4).astype(np.float32)).cuda()
    st = _lib.stream_ptr()
    state = torch.zeros(_lib.TRAIN_STATE_BYTES, dtype=torch.uint8, device="cuda")
    _lib.check(lib.nb200_train_state_init(_lib.ptr(state), 5, 12345, 0, 5e-4, st))
    seed = 77
    for offset in (12345, 12345 + 999):
        want = torch.empty(B, Nc + Nf, device="cuda")
        got = torch.full((B, Nc + Nf), float("nan"), device="cuda")
        assert lib.nb200_sample_pdf_merge(_lib.ptr(ts), _lib.ptr(w), None, 2, seed, offset, B, Nc, Nf, _lib.ptr(want), st) == 0
        assert lib.nb200_sample_pdf_merge_state(_lib.ptr(ts), _lib.ptr(w), seed, _lib.ptr(state), B, Nc, Nf, _lib.ptr(got), st) == 0
        assert torch.equal(got, want), offset
        _lib.check(lib.nb200_train_state_advance(_lib.ptr(state), 1, 999, 1.0, st))
    z = torch.empty(B, 129 + 1, device="cuda")
    assert lib.nb200_sample_pdf_merge_state(_lib.ptr(ts), _lib.ptr(w), seed, None, B, Nc, Nf, _lib.ptr(z), st) == -1
    assert lib.nb200_sample_pdf_merge_state(_lib.ptr(ts), _lib.ptr(w), seed, _lib.ptr(state), B, 129, 1, _lib.ptr(z), st) == -2


# ------------------------------------------------------------------------------- 2. one step vs autograd
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_one_step_matches_autograd(golden_weights, precision):
    from nerf_simple_b200 import config
    from nerf_simple_b200.hierarchical import render_nerf_hierarchical
    from nerf_simple_b200.trainer import Trainer
    g, rays, gt, ts, u_f = golden_step_inputs()
    P_f = fine_weights()
    config.set_precision(precision)
    try:
        c_ref, f_ref = make_net(golden_weights), make_net(P_f)
        (rgb_f, *_), (rgb_c, *_) = render_nerf_hierarchical(rays, c_ref, f_ref, 64, 128, u_coarse=torch.from_numpy(g["u"]).cuda(),
                                                            u_fine=torch.from_numpy(u_f).cuda())
        loss_ref = torch.nn.functional.mse_loss(rgb_c, gt) + torch.nn.functional.mse_loss(rgb_f, gt)
        loss_ref.backward()
    finally:
        config.set_precision("bf16")
    c, f = make_net(golden_weights), make_net(P_f)
    tr = Trainer(c, rays, gt, N=64, batch_size=64, precision=precision, net_fine=f, Nf=128)
    loss = tr.step(sync_loss=True, rays=rays, gt=gt, ts=ts, u_fine=torch.from_numpy(u_f).cuda())
    assert abs(loss - loss_ref.item()) <= 1e-5 * loss_ref.item()
    assert abs(float(tr.loss_fine) - torch.nn.functional.mse_loss(rgb_f, gt).item()) <= 1e-5 * loss_ref.item()
    for net, ref in ((c, c_ref), (f, f_ref)):
        for (k, p), q in zip(net.named_parameters(), ref.parameters()):
            scale = max(1e-6, float(q.grad.abs().max()))
            assert maxabs(p.grad, q.grad) <= GRAD_REL[precision] * scale, (k, maxabs(p.grad, q.grad), scale)
    # the 48 gradients are views of the one flat buffer Adam reads
    lo, hi = tr.flat_grad.data_ptr(), tr.flat_grad.data_ptr() + 4 * tr.flat_grad.numel()
    assert all(lo <= p.grad.data_ptr() < hi for p in list(c.parameters()) + list(f.parameters()))


# -------------------------------------------------------------------------------- 3. one step vs float64
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_one_step_matches_float64_oracle(golden_weights, precision):
    from nerf_simple_b200.trainer import Trainer
    g, rays, gt, ts, u_f = golden_step_inputs()
    P_f = fine_weights()
    c, f = make_net(golden_weights), make_net(P_f)
    tr = Trainer(c, rays, gt, N=64, batch_size=64, precision=precision, net_fine=f, Nf=128)
    loss = tr.step(sync_loss=True, rays=rays, gt=gt, ts=ts, u_fine=torch.from_numpy(u_f).cuda())
    z = tr._z.cpu().numpy()
    w_c = O.render_nerf(g["rays"], golden_weights, 64, g["u"])[4]
    assert maxabs(z, O.sample_pdf_merge(g["ts"], w_c, u_f)) <= 2e-4
    loss_c, loss_f, G_c, G_f = H.hierarchical_train_step_grads(g["rays"], golden_weights, P_f, 64, g["u"], z, g["gt"],
                                                               dtype=np.float64)
    assert abs(loss - (loss_c + loss_f)) <= 1e-5 and abs(float(tr.loss_fine) - loss_f) <= 1e-5
    for net, G in ((c, G_c), (f, G_f)):
        for k, p in net.named_parameters():
            scale = max(1e-6, float(np.abs(G[k]).max()))
            err = maxabs(p.grad, G[k])
            if precision == "fp32":
                assert err <= 2e-3 * scale, (k, err, scale)
            else:
                assert err <= GRAD_ABS_X3 and err <= GRAD_REL_X3 * scale, (k, err, scale)


# ------------------------------------------------------------------------------ 4. graph replay vs eager
def test_graph_replay_matches_eager():
    from nerf_simple_b200.trainer import Trainer
    _, rays, gt = smooth_field()
    B, Nc, Nf = 1024, 32, 64
    runs = {}
    for use_graph in (False, True):
        c, f = make_net(seed=0), make_net(seed=1)
        tr = Trainer(c, rays, gt, N=Nc, batch_size=B, lr_decay=0.99, use_graph=use_graph, net_fine=f, Nf=Nf)
        losses = [tr.step(sync_loss=True) for _ in range(25)]
        runs[use_graph] = (losses, tr._state.cpu(), tr)
    assert runs[True][2].launch_mode.startswith("one CUDA-graph replay") and not runs[False][2]._graphs
    for losses, state, tr in runs.values():
        q = state[:24].view(torch.int64)
        assert int(q[0]) == 25 * B and int(q[1]) == 25 * max(B * Nc // 4, B * Nf // 4) and int(q[2]) == 25
        assert abs(float(state[24:28].view(torch.float32)) - 5e-4 * 0.99 ** 25) < 1e-9
        assert tr.t == 25 and tr._offset == 25 * (B * Nf // 4)
    a, b = np.array(runs[False][0]), np.array(runs[True][0])
    assert a[0] == b[0]
    assert np.abs(a - b).max() <= 2e-2 * a.max()
    with pytest.raises(ValueError):
        runs[True][2].step(time_parts=True)


def test_constructor_validates_the_hierarchical_arguments():
    from nerf_simple_b200.trainer import Trainer
    _, rays, gt = smooth_field(H=8, n_poses=1)
    c = make_net(seed=0)
    for kw in (dict(net_fine=make_net(seed=1)), dict(Nf=16), dict(net_fine=make_net(seed=1), Nf=16, N=2),
               dict(net_fine=make_net(seed=1), Nf=16, N=132), dict(net_fine=make_net(seed=1), Nf=300, N=100)):
        with pytest.raises(ValueError):
            Trainer(c, rays, gt, batch_size=64, **{"N": 32, **kw})
    with pytest.raises(ValueError):
        Trainer(make_net(seed=0), rays, gt, N=32, batch_size=64).step(u_fine=torch.rand(64, 16, device="cuda"))


# ------------------------------------------------------------------- 5. it trains; checkpoints render alike
def test_trains_and_state_dicts_render_identically():
    from nerf_simple_b200.engine import FrameRenderer
    from nerf_simple_b200.trainer import Trainer
    poses, rays, gt = smooth_field()
    c, f = make_net(seed=0), make_net(seed=1)
    tr = Trainer(c, rays, gt, N=32, batch_size=1024, net_fine=f, Nf=64)
    fine_losses = []
    for _ in range(80):
        tr.step()
        fine_losses.append(float(tr.loss_fine))
    assert tr.launch_mode.startswith("one CUDA-graph replay")
    assert np.mean(fine_losses[-10:]) < 0.3 * np.mean(fine_losses[:5]), fine_losses[::10]
    c2, f2 = make_net(seed=5), make_net(seed=6)
    assert list(c.state_dict()) == list(c2.state_dict()) and len(f.state_dict()) == 24
    c2.load_state_dict(c.state_dict(), strict=True)
    f2.load_state_dict(f.state_dict(), strict=True)
    out = []
    for cc, ff in ((c, f), (c2, f2)):
        r = FrameRenderer(cc, 32, 32, 44.4, N=32, seed=3, net_fine=ff, Nf=64)
        out.append(r.render_rays(poses, 0, 32 * 32, philox_base=0))
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


# ---------------------------------------------------------------------------------------------- 6. two ranks
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("p2p", ["0", "1"])
def test_two_rank_hierarchical_training(p2p):
    env = dict(os.environ, NB200_P2P_ALLREDUCE=p2p)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join(ROOT, "scripts", "check_multirank.py"), "--fine"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=200, env=env, cwd=ROOT)
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-3000:])
    res = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert res["all_ranks_ok"] and res["replicas_identical_after_30_steps"] and res["fine"]
    assert ("fused into the Adam kernel" in res["launch_mode"]) == (p2p == "1"), (res["launch_mode"], res.get("p2p_error"))
