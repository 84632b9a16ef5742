"""Training-step time of hierarchical sampling (BASELINE configs[3]: 8192 rays x (64 coarse + 128 fine) samples), measured
in one process on one GPU and written as JSON to --out-dir (bench_train_hierarchical.json).

Timed, in alternating order within every round:
  hier_bf16 / hier_bf16x3  the device-resident Trainer with a fine network (one CUDA-graph replay per step)
  coarse_bf16              the coarse-only Trainer step at 8192 x 64 (the same engine without the fine pass)
  autograd_bf16            render_nerf_hierarchical + MSE(coarse) + MSE(fine) + backward + torch.optim.Adam over both
                           networks: the path that existed before the Trainer could train a fine network
Every configuration is warmed up first; then --rounds rounds, each timing every configuration over a window of at least
--window seconds between CUDA events.  The median round is reported with rays/s and the algorithmic rate: a hierarchical
ray costs (Nc + Nc + Nf) x 3,489,024 FLOP (forward + backward of the MLP per sample, SURVEY 8d; compositing, sampling,
selection and Adam not counted), a coarse-only ray Nc x 3,489,024.  The GPU name and power limit are read in the same
call.  Rays and colours: the golden 4096-ray table, drawn with replacement; weights: the golden weights for both
networks.  Needs a CUDA device; there is no CPU path."""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_train_x3 import FLOP_PER_SAMPLE, gpu_identity   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--Nc", type=int, default=64)
    ap.add_argument("--Nf", type=int, default=128)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--window", type=float, default=1.0, help="seconds of GPU time per timed window")
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_hierarchical.py needs a CUDA device")
    from nerf_simple_b200 import config
    from nerf_simple_b200.hierarchical import render_nerf_hierarchical
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.trainer import Trainer
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "case_train_b4096_n64.npz")))
    w = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz")).items()}
    table, gt_table = torch.from_numpy(g["rays"]).cuda(), torch.from_numpy(g["gt"]).cuda()
    B, Nc, Nf = a.batch, a.Nc, a.Nf

    def net():
        n = Nerf().cuda()
        n.load_state_dict(w)
        return n

    steps = {}
    for prec in ("bf16", "bf16x3"):
        tr = Trainer(net(), table, gt_table, N=Nc, batch_size=B, precision=prec, net_fine=net(), Nf=Nf)
        steps[f"hier_{prec}"] = (tr, tr.step)
    tr = Trainer(net(), table, gt_table, N=Nc, batch_size=B, precision="bf16")
    steps["coarse_bf16"] = (tr, tr.step)

    config.set_precision("bf16")
    config.set_sampler("philox", seed=1)
    nc, nf = net(), net()
    opt = torch.optim.Adam(list(nc.parameters()) + list(nf.parameters()), lr=5e-4)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)

    def autograd_step():
        ids = torch.randint(0, table.shape[0], (B,), device="cuda", generator=gen)
        rays, gt = table[ids], gt_table[ids]
        opt.zero_grad()
        (rgb_f, *_), (rgb_c, *_) = render_nerf_hierarchical(rays, nc, nf, Nc, Nf)
        loss = torch.nn.functional.mse_loss(rgb_c, gt) + torch.nn.functional.mse_loss(rgb_f, gt)
        loss.backward()
        opt.step()
        return loss
    steps["autograd_bf16"] = (None, autograd_step)

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    n_steps = {}
    for name, (_, fn) in steps.items():
        for _ in range(a.warmup):            # the Trainers capture their graph during these
            fn()
        torch.cuda.synchronize()
        ms = timed(fn, 3) / 3
        n_steps[name] = max(3, math.ceil(a.window * 1e3 / ms))
    times = {name: [] for name in steps}
    for r in range(a.rounds):
        order = list(steps) if r % 2 == 0 else list(steps)[::-1]
        for name in order:
            times[name].append(timed(steps[name][1], n_steps[name]) / n_steps[name])

    runs = {}
    for name in steps:
        tr = steps[name][0]
        per_ray = ((2 * Nc + Nf) if name != "coarse_bf16" else Nc) * FLOP_PER_SAMPLE
        ms = float(np.median(times[name]))
        runs[name] = {"ms_per_step_median": ms, "ms_per_step_rounds": times[name], "steps_per_window": n_steps[name],
                      "rays_per_s": B / (ms * 1e-3), "flop_per_ray_algorithmic": per_ray,
                      "tflops_algorithmic": per_ray * B / (ms * 1e-3) / 1e12,
                      "launch_mode": tr.launch_mode if tr is not None else "eager launches, autograd + torch.optim.Adam"}
    result = {"identity": gpu_identity(), "batch_rays": B, "Nc": Nc, "Nf": Nf, "rounds": a.rounds,
              "window_s_min": a.window, "flop_per_sample": FLOP_PER_SAMPLE, "runs": runs,
              "hier_bf16_speedup_vs_autograd": runs["autograd_bf16"]["ms_per_step_median"] / runs["hier_bf16"]["ms_per_step_median"]}
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "bench_train_hierarchical.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: (round(r["ms_per_step_median"], 3), round(r["rays_per_s"] / 1e6, 3), round(r["tflops_algorithmic"], 1))
                      for k, r in runs.items()}))
    print(json.dumps(result["identity"]))


if __name__ == "__main__":
    main()
