"""Generate tests/golden/*.npz by running the UNMODIFIED reference on seeded inputs, on the CPU:
`python oracle/gen_golden.py` (the checkout oracle.ref_import.reference_root finds).  TEST INFRASTRUCTURE ONLY.

The reference hard-codes `.cuda()` (utils/rendering.py:30,68); we patch Tensor.cuda /
Module.cuda to no-ops before calling it (SURVEY.md section 8c).
"""
import os
import sys
import warnings

import numpy as np
import torch

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def import_reference():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from oracle.ref_import import import_reference as imp     # .cuda() no-op shim + natsort stand-in
    return imp(cpu=True)


def np_(t):
    return t.detach().cpu().numpy()


def dome_rays(xyz, H, W, n_phi=3, pose_idx=1):
    """lego-shaped synthetic rays: fov 0.6911112070083618, dome pose (SURVEY.md 8d)."""
    f = W / (2 * np.tan(0.6911112070083618 / 2))
    poses = xyz.poses_to_render(4, -30, n_phi)
    dirs = xyz.rays_single_cam([H, W, f])
    T = poses[pose_idx]
    d = torch.matmul(T[:3, :3], dirs)
    o = T[:3, 3:].expand(3, H * W)
    return torch.cat((o, d), dim=0).permute(1, 0).contiguous(), f, poses


def main():
    warnings.simplefilter("ignore")
    torch.set_num_threads(8)
    nets, rendering, xyz = import_reference()
    os.makedirs(OUT, exist_ok=True)

    torch.manual_seed(0)
    net = nets.Nerf()
    weights = {k: np_(v) for k, v in net.state_dict().items()}
    np.savez(os.path.join(OUT, "weights_seed0.npz"), **weights)

    # ---- case A: train step, B=64 rays x N=64, loss through rgb only (train.py:51-54)
    rays_all, f100, poses = dome_rays(xyz, 100, 100)
    g = torch.Generator().manual_seed(7)
    sel = torch.randperm(rays_all.shape[0], generator=g)[:64]
    rays = rays_all[sel].contiguous()
    torch.manual_seed(2)
    gt = torch.rand(64, 3)
    torch.manual_seed(1)
    u = torch.rand(64, 64)                       # same stream render_nerf consumes at :28
    torch.manual_seed(1)
    net.zero_grad()
    rgb, disp, alpha, acc, w = rendering.render_nerf(rays, net, 64)
    loss = torch.nn.MSELoss()(rgb, gt)
    loss.backward()
    grads = {"grad." + k: np_(p.grad) for k, p in net.named_parameters()}
    # per-sample network outputs and encodings for the same query points
    ts = (4.0 / 64) * u + torch.linspace(2, 6, 65)[:-1]
    d = rays[:, 3:]
    locs = rays[:, :3].unsqueeze(-1) + d.unsqueeze(-1) * ts.unsqueeze(1)
    dn = d / torch.norm(d, dim=1, keepdim=True)
    q = torch.cat((locs, dn.unsqueeze(-1).expand(-1, -1, 64)), dim=1).permute(0, 2, 1).reshape(-1, 6)
    with torch.no_grad():
        out = net.forward(q)
        posx, posd = xyz.positional_encoder(q[:256])
    np.savez(os.path.join(OUT, "case_train_b64_n64.npz"), rays=np_(rays), u=np_(u), gt=np_(gt),
             ts=np_(ts), query=np_(q), out=np_(out), posx=np_(posx), posd=np_(posd),
             rgb=np_(rgb), disp=np_(disp), alpha=np_(alpha), acc=np_(acc), weights=np_(w),
             loss=np.float32(loss.item()), **grads)

    # ---- case B: render chunk, first 1024 rays of the 100x100 view, N=64, no_grad
    rays_b = rays_all[4500:4500 + 1024].contiguous()
    torch.manual_seed(11)
    u_b = torch.rand(1024, 64)
    torch.manual_seed(11)
    with torch.no_grad():
        o5 = rendering.render_nerf(rays_b, net, 64)
    np.savez(os.path.join(OUT, "case_render_b1024_n64.npz"), rays=np_(rays_b), u=np_(u_b),
             rgb=np_(o5[0]), disp=np_(o5[1]), alpha=np_(o5[2]), acc=np_(o5[3]), weights=np_(o5[4]))

    # ---- case C: N=128 (reference default), B=96, gradient through ALL five outputs
    rays_c = rays_all[torch.randperm(rays_all.shape[0], generator=g)[:96]].contiguous()
    torch.manual_seed(5)
    u_c = torch.rand(96, 128)
    cot = [torch.randn(96, 3, generator=g), torch.randn(96, generator=g) * 0.1,
           torch.randn(96, 128, generator=g), torch.randn(96, generator=g),
           torch.randn(96, 128, generator=g)]
    torch.manual_seed(5)
    net.zero_grad()
    o5 = rendering.render_nerf(rays_c, net, 128)
    tot = sum((a * b).sum() for a, b in zip(o5, cot))
    tot.backward()
    gsel = {}
    for k, p in net.named_parameters():
        gsel["grad." + k] = np_(p.grad)
    # keep the fixture small: only biases + 3 weight tensors in full
    keep = [k for k in gsel if k.endswith("bias")] + ["grad.layers_0.0.weight",
            "grad.color_fc.0.weight", "grad.color_fc.2.weight", "grad.sigma_fc.0.weight",
            "grad.layers_1.2.weight", "grad.skip_conn_layer.0.weight"]
    np.savez(os.path.join(OUT, "case_all5_b96_n128.npz"), rays=np_(rays_c), u=np_(u_c),
             cot_rgb=np_(cot[0]), cot_disp=np_(cot[1]), cot_alpha=np_(cot[2]), cot_acc=np_(cot[3]),
             cot_w=np_(cot[4]), rgb=np_(o5[0]), disp=np_(o5[1]), alpha=np_(o5[2]), acc=np_(o5[3]),
             weights=np_(o5[4]), **{k: gsel[k] for k in keep})

    # ---- case D: compositing in isolation (utils/rendering.py:47-85), incl. ragged N
    comp = {}
    for tag, (B, N, srange) in {"n40": (33, 40, 6.0), "n64": (50, 64, 3.0), "n128": (17, 128, 12.0),
                                "n192": (9, 192, 2.0), "n2": (5, 2, 2.0), "n7": (4, 7, 30.0)}.items():
        outs = torch.randn(B, N, 4, generator=g)
        outs[..., 3] *= srange
        outs.requires_grad_(True)
        tsd = torch.sort(2 + 4 * torch.rand(B, N, generator=g), dim=1).values
        dd = torch.randn(B, 3, generator=g)
        dd = dd / torch.norm(dd, dim=1, keepdim=True)
        c5 = [torch.randn(B, 3, generator=g), torch.randn(B, generator=g) * 0.1,
              torch.randn(B, N, generator=g), torch.randn(B, generator=g), torch.randn(B, N, generator=g)]
        r5 = rendering.volume_render(outs, tsd, dd)
        sum((a * b).sum() for a, b in zip(r5, c5)).backward()
        for nm, val in zip(["outs", "ts", "dirs", "rgb", "disp", "alpha", "acc", "w", "c_rgb", "c_disp",
                            "c_alpha", "c_acc", "c_w", "d_outs"],
                           [outs, tsd, dd, *r5, *c5, outs.grad]):
            comp[f"{tag}.{nm}"] = np_(val)
    np.savez(os.path.join(OUT, "case_composite.npz"), **comp)

    # ---- case E: ray generation (utils/xyz.py:38-52, utils/rendering.py:129-134), dome poses
    rg = {}
    for tag, (H, W, f) in {"h5w7": (5, 7, 3.3), "h100": (100, 100, float(f100)), "h6w4": (6, 4, 2.0)}.items():
        dirs = xyz.rays_single_cam([H, W, f])
        P = torch.stack(xyz.poses_to_render(4, -30, 4))
        rd = torch.matmul(P[:, :3, :3], dirs)
        oo = P[:, :3, 3:].expand(4, 3, H * W)
        rays_w = torch.cat((oo, rd), dim=1).permute(0, 2, 1).reshape(-1, 6)
        rg[f"{tag}.cam"] = np.array([H, W, f], np.float64)
        rg[f"{tag}.dirs"] = np_(dirs)
        rg[f"{tag}.poses"] = np_(P)
        rg[f"{tag}.rays"] = np_(rays_w)
    rg["poses30"] = np_(torch.stack(xyz.poses_to_render(r=4, theta=-30, n_phi=30)))
    np.savez(os.path.join(OUT, "case_raygen.npz"), **rg)
    # ---- case F: BASELINE configs[2] at full size -- one training step 4096 rays x 64 samples
    # (train.py:47-54: MSE through rgb only), all 24 gradients.  The jitter is NOT stored: tests redraw it
    # with torch.manual_seed(21); torch.rand(4096, 64) (the stream render_nerf consumes at :28).
    rays800, f800, _ = dome_rays(xyz, 800, 800, n_phi=30, pose_idx=7)
    sel = torch.randperm(rays800.shape[0], generator=g)[:4096]
    rays_f = rays800[sel].contiguous()
    gt_f = torch.rand(4096, 3, generator=g)
    torch.manual_seed(21)
    net.zero_grad()
    rgb_f, disp_f, _, acc_f, _ = rendering.render_nerf(rays_f, net, 64)
    loss_f = torch.nn.MSELoss()(rgb_f, gt_f)
    loss_f.backward()
    np.savez(os.path.join(OUT, "case_train_b4096_n64.npz"), rays=np_(rays_f), gt=np_(gt_f), u_seed=np.int64(21),
             rgb=np_(rgb_f), disp=np_(disp_f), acc=np_(acc_f), loss=np.float32(loss_f.item()),
             **{"grad." + k: np_(p.grad) for k, p in net.named_parameters()})

    # ---- case G: the reference's own chunk loops (utils/rendering.py:88-113 render_image, :116-153
    # render_poses), divisible sizes, seeded CPU generator (one torch.rand(chunk,128) per chunk, :102,:145)
    Hh = Wh = 20
    fh = Wh / (2 * np.tan(0.6911112070083618 / 2))
    poses_g = xyz.poses_to_render(4, -30, 4)
    dirs_g = xyz.rays_single_cam([Hh, Wh, fh])
    Pg = torch.stack(poses_g)
    rays_g = torch.cat((Pg[:, :3, 3:].expand(4, 3, Hh * Wh), torch.matmul(Pg[:, :3, :3], dirs_g)), dim=1)
    rays_g = rays_g.permute(0, 2, 1).reshape(-1, 6).contiguous()
    gt_imgs = [np.random.default_rng(5 + i).random((Hh, Wh, 3)) for i in range(4)]

    class RG:
        samples = {"val": [{"img": im} for im in gt_imgs]}
        rays_dataset = {"val": rays_g}
    # shift the colour biases so that the image straddles the [0,1] clip of :103 on two channels
    net_g = nets.Nerf()
    net_g.load_state_dict(net.state_dict())
    with torch.no_grad():
        net_g.color_fc[2].bias.add_(torch.tensor([0.5, 1.07, -0.13]))
        net_g.sigma_fc[0].bias.add_(0.3)
    torch.manual_seed(31)
    with torch.no_grad():
        img_rgb, img_depth, img_gt = rendering.render_image(net_g, RG, batch_size=100, im_idx=2, im_set="val")
    # render_poses returns nothing: record the uint8 BGR frames it hands to cv2.VideoWriter (:155-160)
    import cv2
    frames = []

    class Recorder:
        def __init__(self, *a):
            self.args = a
        def write(self, fr):
            frames.append(np.array(fr))
        def release(self):
            pass
    real_writer = cv2.VideoWriter
    cv2.VideoWriter = Recorder
    try:
        torch.manual_seed(32)
        rendering.render_poses(net_g, poses_g[:2], [Hh, Wh, fh], 80, savepath="")
    finally:
        cv2.VideoWriter = real_writer
    np.savez(os.path.join(OUT, "case_chunk_loops.npz"), cam=np.array([Hh, Wh, fh], np.float64), poses=np_(Pg),
             rays=np_(rays_g), gt2=gt_imgs[2], bias_shift=np.array([0.5, 1.07, -0.13, 0.3], np.float32),
             image_seed=np.int64(31), image_rgb=np_(img_rgb), image_depth=np_(img_depth), image_gt=np.asarray(img_gt),
             poses_seed=np.int64(32), frames_bgr_u8=np.stack(frames))
    for fn in sorted(os.listdir(OUT)):
        print(fn, os.path.getsize(os.path.join(OUT, fn)))


if __name__ == "__main__":
    main()
