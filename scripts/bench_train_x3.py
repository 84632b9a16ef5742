"""Trainer step time of the three training precisions (fp32 SIMT, bf16x3 and bf16 on the tensor cores), measured in one
process on one GPU and written as JSON (default: profiles/bench_train_x3.json).

For each N in --N: one Trainer per precision (4096-ray batches drawn on the device from the golden 4096-ray table, the
golden weights), --warmup steps each, then --rounds rounds in which the precisions take turns, each timing --steps
steps between CUDA events.  The median round is reported, with the algorithmic rate (3,489,024 FLOP per sample for
forward + backward of the MLP; compositing, selection and Adam are not counted) and the GPU name and power limit read
in the same call.  Needs a CUDA device; there is no CPU path."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FLOP_PER_SAMPLE = 3_489_024


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e!r})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[64, 128])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precisions", nargs="+", default=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_train_x3.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_x3.py needs a CUDA device")
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.trainer import Trainer
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "case_train_b4096_n64.npz")))
    w = dict(np.load(os.path.join(ROOT, "tests", "golden", "weights_seed0.npz")))
    table, gt = torch.from_numpy(g["rays"]).cuda(), torch.from_numpy(g["gt"]).cuda()
    result = {"identity": gpu_identity(), "batch_rays": a.batch, "steps_per_round": a.steps, "rounds": a.rounds,
              "flop_per_sample": FLOP_PER_SAMPLE, "runs": {}}
    for N in a.N:
        trainers = {}
        for prec in a.precisions:
            net = Nerf().cuda()
            net.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
            trainers[prec] = Trainer(net, table, gt, N=N, batch_size=a.batch, precision=prec, use_graph=prec != "fp32")
            for _ in range(a.warmup):
                trainers[prec].step()
        torch.cuda.synchronize()
        times = {p: [] for p in a.precisions}
        for _ in range(a.rounds):
            for prec, tr in trainers.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    tr.step()
                e1.record()
                e1.synchronize()
                times[prec].append(e0.elapsed_time(e1) / a.steps)
        M = a.batch * N
        run = {}
        for prec in a.precisions:
            ms = float(np.median(times[prec]))
            run[prec] = {"ms_per_step_median": ms, "ms_per_step_rounds": times[prec],
                         "mlp_tflops_algorithmic": FLOP_PER_SAMPLE * M / (ms * 1e-3) / 1e12,
                         "launch_mode": trainers[prec].launch_mode, "final_loss": float(trainers[prec].last_loss)}
        if "fp32" in run and "bf16x3" in run:
            run["bf16x3_speedup_vs_fp32"] = run["fp32"]["ms_per_step_median"] / run["bf16x3"]["ms_per_step_median"]
        result["runs"][f"{a.batch}x{N}"] = run
        del trainers
        torch.cuda.empty_cache()
        print(json.dumps({f"{a.batch}x{N}": {p: (round(r["ms_per_step_median"], 3), round(r["mlp_tflops_algorithmic"], 1))
                                             if isinstance(r, dict) else round(r, 2) for p, r in run.items()}}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["identity"]))


if __name__ == "__main__":
    main()
