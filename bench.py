#!/usr/bin/env python
"""Headline benchmark: rays/sec of the NeRF hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload all|render|train] [--impl reference] [--dump-outputs DIR]

Headline workload = BASELINE.json configs[1]: full 800x800 novel-view render, 64 samples/ray, spherical-dome camera
path, synthetic lego-shaped scene, seeded random-init weights.  One step = one frame per GPU: ray generation ->
stratified sampling -> fused posenc+MLP (tcgen05) -> compositing, all on the device.  Under torchrun (one rank per GPU)
the frames of the dome path are sharded across ranks (weak scaling) and gathered on rank 0.

The same JSON line carries sub-records measured in the same run (`--workload all`, the default):
  train          configs[2]: training step 4096 rays x 64 samples per GPU, fwd + bwd + Adam (data-parallel for N > 1)
  train_dp8192   configs[4]: 8192 rays per GPU, data-parallel, one all-reduce of the 595,844 gradients per step
  sharded_frame  configs[4]: ONE 1600x1600 frame split into ray bands over the ranks + one all_gather (strong scaling)
  n128, train_n128   the reference's default 128 samples/ray (configs/lego.yaml:6), render and train step

`--impl reference` times the UNMODIFIED reference (baseline/_ref, staged by scripts/stage_reference.sh; its own
render_nerf, CPU, all host threads) on a bounded sample of the same workload.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes what the last timed step of the headline path returned to its caller, as float32
DIR/<name>.npy on rank 0: rgb [H,W,3] and disp [H,W] of rank 0's own frame (render; with several GPUs the other
ranks' frames are not written), or loss, rgb [B,3] and the updated parameters in state_dict order (--workload
train).  Weights, poses, jitter and training batches are all seeded, so the same arguments give the same inputs in
every run, and two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FOV = 0.6911112070083618
FLOP_FWD = 1186816            # per sample, SURVEY 8d: the reference's MLP (utils/nets.py:34-43), the ALGORITHMIC work
FLOP_TRAIN = 3489024
# precision "bf16" folds layers_2 into color_fc.0 (no activation between them; DESIGN 4.8): the kernels EXECUTE one
# 256x256 layer less in the forward, in the delta chain and in wgrad.  roofline.achieved / frac use the algorithmic
# figures above (what the contract asks for); executed_tflops / frac_executed say how busy the tensor pipe really is.
FLOP_FOLD_LAYER = 2 * 256 * 256


def flop_fwd_exec(precision):
    return FLOP_FWD - (FLOP_FOLD_LAYER if precision == "bf16" else 0)


def flop_train_exec(precision):
    return FLOP_TRAIN - (3 * FLOP_FOLD_LAYER if precision == "bf16" else 0)


FOLD_NOTE = ("precision bf16 folds layers_2 into color_fc.0 at pack time (exact algebra, product formed in fp32; parity tests "
             "run this path): achieved/frac count the reference's algorithmic FLOPs, executed_tflops/frac_executed the "
             "FLOPs the tensor cores really perform (11 % fewer)")
METRIC = "rays/sec (64 samples/ray) render"
REF_CHUNK = 16000             # test.py's batch size (configs/lego.yaml:18): the reference arm's bounded sample per step


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            pk = json.load(fh)
        return dict(hbm=pk["hbm_gbs"], burst=pk["bf16_tflops"], sustained=pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, burst=1590.0, sustained=1400.0, source="fallback (B200_PROFILING.md)")


def load_traffic(kernel_key):
    """DRAM bytes per launch of `kernel_key` from the committed ncu capture summary (profiles/traffic.json, written by
    scripts/summarize_profiles.py from an `ncu --set full` report); None when no capture of this build exists."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            t = json.load(fh)
        e = t.get(kernel_key)
        return (e["dram_bytes"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: name -> array as out_dir/<name>.npy in float32, at most DUMP_BYTES in all.  Beyond that every
    array keeps the same fixed, seeded sample of its rows (first axis); the row numbers go to out_dir/<name>_rows.npy."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES and a.ndim > 0:
            # a quarter of the budget for the rows themselves: the float64 row numbers take at most twice that
            keep = max(1, a.shape[0] * (DUMP_BYTES // 4) // total)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(H, W, N, world):
    """The keys that name the workload -- identical in the B200 arm and the reference arm."""
    return {"workload": f"configs[1]: full {H}x{W} novel-view render, {N} samples/ray, spherical-dome path "
                        f"(poses_to_render(4,-30,30)), one frame per GPU per step",
            "H": H, "W": W, "N": N, "rays_per_frame": H * W, "weights": "torch.manual_seed(0); Nerf()",
            "parallelism": f"frames sharded over {world} rank(s), gathered on rank 0",
            "l2": f"inputs larger than L2: {H * W * N * 16 / 1e6:.0f} MB of per-sample (r,g,b,sigma) + {H * W * N * 4 / 1e6:.0f} MB of ts per frame"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled for the whole run; window(t0, t1) summarises a timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.lines = None, []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def window(self, t_begin, t_end):
        if self.proc is None:
            return None
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in list(self.lines):
            if not (t_begin <= ts <= t_end + 0.15):
                continue
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}

    def close(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()


# ------------------------------------------------------------------------- reference / CPU arm
def dome_rays_numpy(H, W, pose_idx, begin, count):
    from oracle import nerf_oracle as O            # CPU arm only: ray set-up of the sample
    f = W / (2 * np.tan(FOV / 2))
    poses = np.stack(O.poses_to_render(4, -30, 30))
    dirs = O.rays_single_cam(H, W, f)
    return O.world_rays(poses[pose_idx:pose_idx + 1], dirs[:, begin:begin + count])


def reference_arm(args, rank):
    """The reference's own CPU implementation of the path: the checkout oracle.ref_import.reference_root finds,
    imported unmodified, `.cuda()` no-op shim, fp32, all host threads.  Falls back to the torch-CPU port in oracle/
    only when no reference checkout is available, and says which."""
    if rank != 0:
        return
    import torch
    from oracle.ref_import import import_reference, reference_root
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    H = W = args.res
    N = args.samples
    n_rays = min(REF_CHUNK, H * W)
    root = reference_root()
    rays = torch.from_numpy(dome_rays_numpy(H, W, 1, (H // 2) * W, n_rays))
    if root is not None:
        nets, rendering, xyz = import_reference(cpu=True, root=root)
        torch.manual_seed(0)
        net = nets.Nerf()
        kind, what = "reference", f"unmodified reference utils/rendering.py:render_nerf imported from {os.path.relpath(root, ROOT) if root.startswith(ROOT) else root}"

        def render(r, n):
            rgb, *_ = rendering.render_nerf(r, net, n)
            return rgb
    else:
        from oracle import nerf_oracle as O
        from oracle import nerf_oracle_torch as OT
        P = {k: torch.from_numpy(v) for k, v in O.init_params(0).items()}
        kind, what = "port", "torch-CPU port of the reference ops (oracle/nerf_oracle_torch.py): no reference checkout staged"
        net = None

        def render(r, n):
            return OT.render_nerf(r, P, n, torch.rand(r.shape[0], n))[0]
    torch.manual_seed(1)

    def step():
        t0 = time.perf_counter()
        with torch.no_grad():
            render(rays, N).clamp_(0, 1)          # one test.py-sized chunk of the frame (utils/rendering.py:143-146)
        return time.perf_counter() - t0
    for _ in range(args.warmup):
        step()
    times = [step() for _ in range(args.steps)]
    ms = 1e3 * float(np.mean(times))
    val = n_rays / (ms * 1e-3)
    sample = (f"{n_rays} rays (one {REF_CHUNK}-ray chunk, test.py's batch size) of the same {H}x{W} dome view x {N} samples per step; "
              f"{what}; fp32, {cores} intra-op threads")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(H, W, N, args.gpus),
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not args.no_extras and kind == "reference":
        # BASELINE configs[0], the reference's own CPU-runnable case: whole 100x100 frame in 1024-ray chunks, and one
        # training step 1024 rays x 64 (train.py:47-55), best of 2 after a warm-up
        r100 = torch.from_numpy(dome_rays_numpy(100, 100, 1, 0, 10000))

        def frame100():
            t0 = time.perf_counter()
            with torch.no_grad():
                for s in range(0, 10000, 1024):
                    render(r100[s:s + 1024], 64).clamp_(0, 1)
            return time.perf_counter() - t0
        frame100()
        line["config0_frame_100x100x64"] = {"value": 10000 / min(frame100(), frame100()), "unit": "rays/s", "chunk": 1024}
        opt = torch.optim.Adam(net.parameters(), lr=5e-4)
        crit = torch.nn.MSELoss()
        gt = torch.rand(1024, 3)

        def train_step():
            t0 = time.perf_counter()
            opt.zero_grad()
            rgb, *_ = rendering.render_nerf(r100[:1024], net, 64)
            crit(rgb, gt).backward()
            opt.step()
            return time.perf_counter() - t0
        train_step()
        line["config0_train_step_1024x64"] = {"value": 1024 / min(train_step(), train_step()), "unit": "rays/s"}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(args):
    """Run the reference arm in a process of its own (its `.cuda()` no-op shim is process-wide) on a short schedule."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "4", "--warmup", "1",
           "--res", str(args.res), "--samples", str(args.samples)]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
        ref = json.loads(out.stdout.strip().splitlines()[-1])
        cb = ref["cpu_baseline"]
        for k in ("config0_frame_100x100x64", "config0_train_step_1024x64"):
            if k in ref:
                cb[k] = ref[k]
        return cb
    except Exception as e:      # the baseline is reported context, never a reason to lose the GPU measurement
        return {"value": None, "unit": "rays/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)[:200]}


def reference_gpu_eager(H, W, N, dev):
    """Context only: the UNMODIFIED reference run eagerly on this same B200 (its ATen/cuBLAS path, fp32 matmuls as
    torch >= 1.12 defaults), one whole frame in test.py-sized chunks.  None when baseline/_ref is not staged."""
    import torch
    from oracle.ref_import import import_reference, reference_root
    root = reference_root()
    if root is None:
        return None
    nets, rendering, xyz = import_reference(cpu=False, root=root)
    torch.manual_seed(0)
    net = nets.Nerf().cuda()
    rays = torch.from_numpy(dome_rays_numpy(H, W, 1, 0, H * W))
    with torch.no_grad():
        for s in (0, REF_CHUNK):                                   # warm-up chunks (cuBLAS handles, allocator)
            rendering.render_nerf(rays[s:s + REF_CHUNK].cuda(), net, N)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for s in range(0, H * W - REF_CHUNK + 1, REF_CHUNK):       # utils/rendering.py:143-146
            rgb, *_ = rendering.render_nerf(rays[s:s + REF_CHUNK].cuda(), net, N)
            torch.clip(rgb, torch.tensor(0.).cuda(), torch.tensor(1.).cuda())
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
    n = (H * W // REF_CHUNK) * REF_CHUNK
    return {"value": n / dt, "unit": "rays/s", "what": f"unmodified reference render_nerf on cuda:0, eager ATen/cuBLAS fp32, {n} rays "
            f"of one {H}x{W} frame in {REF_CHUNK}-ray chunks, N={N}, host ray table + per-chunk H2D like utils/rendering.py:139-151"}


# ------------------------------------------------------------------------------------ B200 arm
class Ctx:
    pass


def setup(args, local_rank, world):
    import torch
    import torch.distributed as dist
    from nerf_simple_b200 import _lib, config
    _lib.load()                               # fail loudly if the CUDA library is missing
    torch.cuda.set_device(local_rank)
    c = Ctx()
    c.dev = torch.device("cuda", local_rank)
    c.world, c.rank = world, int(os.environ.get("RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=c.dev)
    config.set_precision(args.precision)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(c.dev)

    def max_over_ranks(x):
        t = torch.tensor([x], device=c.dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    c.sync_all, c.max_over_ranks = sync_all, max_over_ranks
    c.sampler = ClockSampler(local_rank) if c.rank == 0 else None
    return c


def bench_render(args, c, H, W, N, steps, warmup, fine=0, fused=False, e2e=True, api=True, precision=None, dump=False):
    """Frames-per-GPU render (weak scaling): value, MLP-kernel time, e2e through host buffers.  dump: the frame of the
    last timed step on the host as r["outputs"]."""
    import torch
    import torch.distributed as dist
    from nerf_simple_b200.engine import FrameRenderer
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    dev, world, rank = c.dev, c.world, c.rank
    f = W / (2 * np.tan(FOV / 2))
    torch.manual_seed(0)
    net = Nerf().to(dev)                      # random-init weights of the reference architecture
    poses = torch.stack(poses_to_render(4, -30, 30)).to(dev)
    n_poses = poses.shape[0]
    net_fine = Nerf().to(dev) if fine > 0 else None     # --fine 128: hierarchical extension (configs[3])
    rend = FrameRenderer(net, H, W, f, N=N, seed=1, precision=precision or args.precision, net_fine=net_fine, Nf=fine, fused=fused)
    n_rays = H * W
    # the frames of the dome path are gathered on rank 0 (16 B/ray), asynchronously: the collective of frame i runs under
    # the kernels of frame i+1 (two send buffers); no rank ever receives frames it does not need
    send = [torch.empty((n_rays, 4), device=dev) for _ in range(2)] if world > 1 else None
    recv = [[torch.empty((n_rays, 4), device=dev) for _ in range(world)] for _ in range(2)] if (world > 1 and rank == 0) else None
    pending = [None, None]

    def step(i, timed):
        idx = (i * world + rank) % n_poses    # frames of the dome path sharded over ranks
        rgb, disp = rend.render_frame(poses, idx, time_mlp=timed)
        if world > 1:
            b = i & 1
            if pending[b] is not None:
                pending[b].wait()
            send[b][:, :3].copy_(rgb.view(-1, 3)); send[b][:, 3].copy_(disp.view(-1))
            pending[b] = dist.gather(send[b], recv[b] if rank == 0 else None, dst=0, async_op=True)
        return rgb, disp

    def drain():
        for b in range(2):
            if pending[b] is not None:
                pending[b].wait()
                pending[b] = None

    for i in range(warmup):
        step(i, False)
    drain()
    c.sync_all()
    launches0 = rend.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for i in range(steps):
        last = step(i, True)
    drain()
    e1.record()
    c.sync_all()
    t_end = time.perf_counter()
    ms_step = c.max_over_ranks(e0.elapsed_time(e1)) / steps
    r = {"value": world * n_rays / (ms_step * 1e-3), "ms_per_step": ms_step, "gpu_launches": rend.launches - launches0,
         "mlp_ms": float(np.mean([a.elapsed_time(b) for a, b in rend.mlp_events])), "t_window": (t_begin, t_end), "fused": rend.fused}
    if dump:
        r["outputs"] = {"rgb": last[0].cpu().numpy(), "disp": last[1].cpu().numpy()}
    del last
    rend.mlp_events.clear()
    if e2e:
        # ---- end to end through the public host-buffer API: pose on the host in, frame on the host out
        pose_host = [poses[i].cpu().pin_memory() for i in range(n_poses)]
        out_rgb = torch.empty((H, W, 3), dtype=torch.float32).pin_memory()
        out_disp = torch.empty((H, W), dtype=torch.float32).pin_memory()
        for i in range(2):
            rend.render_frame_host(pose_host[i], out_rgb, out_disp)
        c.sync_all()
        t0 = time.perf_counter()
        for i in range(steps):
            rend.render_frame_host(pose_host[(i * world + rank) % n_poses], out_rgb, out_disp)
        c.sync_all()
        r["e2e"] = world * n_rays * steps / c.max_over_ranks(time.perf_counter() - t0)
        r["finite"] = bool(torch.isfinite(out_rgb).all())
        # ---- the video path of render_poses: uint8 BGR frame out (3 B/pixel)
        out_u8 = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
        rend.render_frame_u8_host(pose_host[0], out_u8)
        c.sync_all()
        t0 = time.perf_counter()
        reps = max(3, steps // 2)
        for i in range(reps):
            rend.render_frame_u8_host(pose_host[(i * world + rank) % n_poses], out_u8)
        c.sync_all()
        r["e2e_u8"] = world * n_rays * reps / c.max_over_ranks(time.perf_counter() - t0)
    if api and world == 1 and fine == 0:
        # ---- the reference's own host driver, unchanged call: render_image(net, rg, batch_size=16000, ...)
        # (utils/rendering.py:88-113; test.py batch size): CPU ray table in, per-chunk H2D, CPU frame out.
        from nerf_simple_b200 import config
        from nerf_simple_b200 import ops as _ops
        from nerf_simple_b200.rendering import render_image

        class _RG:
            samples = {"test": [{"img": np.zeros((H, W, 3))}]}
            rays_dataset = {"test": _ops.generate_rays(poses[1:2], H, W, f).cpu()}
        config.set_sampler("philox")
        render_image(net, _RG, batch_size=REF_CHUNK, im_idx=0, im_set="test", N=N)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        reps = max(2, steps // 4)
        for _ in range(reps):
            render_image(net, _RG, batch_size=REF_CHUNK, im_idx=0, im_set="test", N=N)
        torch.cuda.synchronize(dev)
        r["api"] = reps * n_rays / (time.perf_counter() - t0)
        config.set_sampler("reference")
    return r


def bench_sharded_frame(args, c, H, W, N, frames, warmup=2):
    """BASELINE configs[4], render half: ONE HxW frame split into contiguous ray bands over the ranks
    (utils/rendering.py:139-151 is the loop being sharded) + one all_gather of (rgb, disp) = 16 B/ray.  Strong scaling."""
    import torch
    from nerf_simple_b200.engine import FrameRenderer, render_sharded
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.xyz import poses_to_render
    dev, world, rank = c.dev, c.world, c.rank
    f = W / (2 * np.tan(FOV / 2))
    torch.manual_seed(0)
    net = Nerf().to(dev)
    poses = torch.stack(poses_to_render(4, -30, 30)).to(dev)
    rend = FrameRenderer(net, H, W, f, N=N, seed=1, precision=args.precision)
    for i in range(warmup):
        render_sharded(rend, poses, i % 30, rank, world)
    c.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for i in range(frames):
        rgb, disp = render_sharded(rend, poses, i % 30, rank, world)
    e1.record()
    c.sync_all()
    t_end = time.perf_counter()
    ms = c.max_over_ranks(e0.elapsed_time(e1)) / frames
    ok = bool(torch.isfinite(rgb).all()) and tuple(rgb.shape) == (H, W, 3)
    return {"metric": "rays/sec (64 samples/ray) render, one frame ray-sharded over the ranks", "value": H * W / (ms * 1e-3), "unit": "rays/s",
            "ms_per_frame": ms, "frames": frames, "scaling": "strong", "n_gpus": world,
            "config": {"workload": f"configs[4]: one {H}x{W} frame, {N} samples/ray, contiguous ray bands of {H * W // world} rays per rank, "
                                   f"one all_gather of (rgb, disp) = 16 B/ray on every rank"},
            "frame_assembled_on_every_rank": ok, "clocks": c.sampler.window(t_begin, t_end) if c.sampler else None}


def bench_train(args, c, B, N, steps, warmup, loop_api=False, precision=None, dump=False):
    """BASELINE configs[2] / configs[4]: training step, B rays x N samples per GPU, fwd+bwd+Adam, data-parallel
    with one all-reduce of the flat gradient buffer per step (weak scaling).  dump: loss, rgb and the updated
    parameters of the last timed step on the host as rec["outputs"]."""
    import torch
    from nerf_simple_b200 import ops
    from nerf_simple_b200.nets import Nerf
    from nerf_simple_b200.trainer import Trainer
    from nerf_simple_b200.xyz import poses_to_render
    dev, world, rank = c.dev, c.world, c.rank
    precision = precision or args.precision
    f = 400 / (2 * np.tan(FOV / 2))
    torch.manual_seed(0)
    net = Nerf().to(dev)
    poses = torch.stack(poses_to_render(4, -30, 25)).to(dev)          # 25 half-res training views (lego.yaml)
    rays_table = ops.generate_rays(poses, 400, 400, f)                 # 4.0 M rays, device resident
    g = torch.Generator(device=dev); g.manual_seed(2)
    gt_table = torch.rand((rays_table.shape[0], 3), device=dev, generator=g)
    tr = Trainer(net, rays_table, gt_table, N=N, batch_size=B, seed=1, precision=precision, world_size=world)
    for _ in range(warmup):
        tr.step()
    c.sync_all()
    l0 = tr.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = tr.step()                             # one CUDA-graph replay per step
    e1.record()
    timed_launches = tr.launches - l0
    c.sync_all()
    t_end = time.perf_counter()
    ms_step = c.max_over_ranks(e0.elapsed_time(e1)) / steps
    outputs = None
    if dump:                                         # before the steps below train the net further
        # tr._rgb: the trainer's persistent [B,3] buffer of rendered batch colours, which every step (CUDA-graph
        # replay or eager) overwrites and its MSE loss is taken from; Trainer has no public accessor for it
        outputs = {"loss": loss.cpu().numpy(), "rgb": tr._rgb.cpu().numpy(),
                   "params": torch.cat([p.detach().reshape(-1) for p in net.state_dict().values()]).cpu().numpy()}
    value = world * B / (ms_step * 1e-3)
    # ---- e2e, train.py's own data flow (train.py:47-51): the batch is chosen on the HOST and arrives in pinned host
    # memory (rays 24 B + colours 12 B per ray), is copied to the device inside the timed region, and the loss is read
    # back every step (loss.item(), train.py:61-63)
    pool = 8
    ids = torch.randint(0, rays_table.shape[0], (pool, B), generator=torch.Generator().manual_seed(3 + rank))
    rays_h = [rays_table[ids[i].to(dev)].cpu().pin_memory() for i in range(pool)]
    gt_h = [gt_table[ids[i].to(dev)].cpu().pin_memory() for i in range(pool)]
    for i in range(4):
        tr.step(sync_loss=True, rays=rays_h[i % pool], gt=gt_h[i % pool])
    c.sync_all()
    t0 = time.perf_counter()
    for i in range(steps):
        lv = tr.step(sync_loss=True, rays=rays_h[i % pool], gt=gt_h[i % pool])
    c.sync_all()
    e2e = world * B * steps / c.max_over_ranks(time.perf_counter() - t0)
    launch_mode = tr.launch_mode
    for _ in range(min(20, steps)):                  # per-part times from eager launches with events around the two MLP calls
        tr.step(time_parts=True)
    torch.cuda.synchronize(dev)
    fwd_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in tr.part_events]))
    bwd_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in tr.part_events]))
    pk = load_peaks()
    M = B * N
    achieved = FLOP_TRAIN * M / (ms_step * 1e-3) / 1e12
    executed = flop_train_exec(precision) * M / (ms_step * 1e-3) / 1e12
    traffic, tsrc = load_traffic("train_step_mlp_kernels") if (B, N) == (4096, 64) and precision == "bf16" else (None, None)
    rec = {"metric": f"rays/sec ({N} samples/ray) train", "value": value, "unit": "rays/s", "n_gpus": world, "steps": steps,
           "warmup": warmup, "ms_per_step": ms_step, "scaling": "weak", "dtype": precision, "samples_per_sec": value * N,
           "config": {"workload": f"training step {B} rays x {N} samples per GPU, L=10/4 posenc, fwd+bwd+Adam, fused compositing backward "
                                  f"(train.py:47-57)", "rays_table": "25 views 400x400 (4.0 M rays) on device",
                      "parallelism": f"data-parallel over {world} rank(s), one all-reduce of 595,844 fp32 grads/step",
                      "launch": launch_mode,
                      "limiter": "HBM bytes of saved activations + deltas (roofline.traffic, from profiles/traffic.json) under the 1 kW "
                                 "power cap; the data-parallel all-reduce is fused into the Adam kernel (no collective in the step)",
                      "l2": f"saved activations + deltas per step = {M * 9e3 / 1e9:.1f} GB (larger than L2)"},
           "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": B * 36, "d2h_bytes_per_step": 4,
                   "api": "Trainer.step(rays=pinned, gt=pinned, sync_loss=True): host-selected batch copied in, loss read back, every step"},
           "gpu_launches": timed_launches,
           "roofline": {"kernel": "whole step (chain_kernel<FwdEpi<save>> + backward kernels; the MLP is >99 % of the FLOPs)", "bound": "tensor",
                        "achieved": achieved, "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved / pk["sustained"],
                        "peak_burst": pk["burst"], "frac_burst": achieved / pk["burst"], "flop_per_step": FLOP_TRAIN * M,
                        "executed_tflops": executed, "frac_executed": executed / pk["sustained"],
                        "flop_executed_per_step": flop_train_exec(precision) * M, "note": FOLD_NOTE if precision == "bf16" else None,
                        "peak_source": pk["source"] + ", sustained figure", "traffic": traffic, "traffic_source": tsrc},
           "mlp_forward_ms": fwd_ms, "mlp_backward_ms": bwd_ms,
           "mlp_forward_tflops": FLOP_FWD * M / (fwd_ms * 1e-3) / 1e12,
           "mlp_backward_tflops": (FLOP_TRAIN - FLOP_FWD) * M / (bwd_ms * 1e-3) / 1e12,
           "clocks": c.sampler.window(t_begin, t_end) if c.sampler else None, "final_loss": float(lv)}
    if outputs is not None:
        rec["outputs"] = outputs
    if loop_api and world == 1:
        # ---- the reference's own training loop body, unchanged calls (train.py:47-57): rg.select -> CPU gather of
        # the ground truth -> render_nerf (autograd) -> MSELoss -> backward -> torch.optim.Adam, host tensors in
        from nerf_simple_b200 import config
        from nerf_simple_b200.dataload import RayGenerator
        from nerf_simple_b200.rendering import render_nerf

        class _RG:                                   # RayGenerator without the PNG loader: same select()
            rays_dataset = {"train": rays_table.cpu()}
            select = RayGenerator.select
            _select_device = RayGenerator._select_device
        rg = _RG()
        train_imgs = gt_table.cpu().double()         # train.py:34: CPU float64 image table
        config.set_precision(precision); config.set_sampler("philox"); config.set_select("device")
        torch.manual_seed(0)
        net2 = Nerf().to(dev)
        opt = torch.optim.Adam(net2.parameters(), lr=5e-4)
        crit = torch.nn.MSELoss()

        def loop_step():
            rays, ray_ids = rg.select(mode="train", N=B)
            gt = train_imgs[ray_ids, :].float().cuda()
            opt.zero_grad()
            rgb, depth, alpha, acc, w = render_nerf(rays.cuda(), net2, N)
            loss2 = crit(rgb, gt)
            loss2.backward()
            opt.step()
            return loss2
        for _ in range(10):                          # the autograd path allocates its workspaces here
            loop_step()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        reps = max(10, steps // 4)
        for _ in range(reps):
            l2 = loop_step()
        l2.item()
        torch.cuda.synchronize(dev)
        rec["e2e_train_py_loop"] = {"value": reps * B / (time.perf_counter() - t0), "unit": "rays/s", "h2d_bytes_per_step": B * 12,
                                    "d2h_bytes_per_step": B * 8,
                                    "api": "train.py:47-57 body unchanged: rg.select (device mode) -> train_imgs[ray_ids].cuda() -> render_nerf "
                                           "-> MSELoss -> backward -> torch.optim.Adam"}
        config.set_select("reference"); config.set_sampler("reference")
    tr.close()
    del tr, rays_table, gt_table
    torch.cuda.empty_cache()
    return rec


def b200_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    c = setup(args, local_rank, world)
    H = W = args.res
    N = args.samples
    pk = load_peaks()
    dump = args.dump_outputs is not None and rank == 0
    if args.workload == "train":
        rec = bench_train(args, c, args.batch, N, args.steps, max(args.warmup, 20), loop_api=True, dump=dump)
        if dump:
            dump_outputs(args.dump_outputs, rec.pop("outputs"))
        if rank == 0:
            rec.update({"higher_is_better": True, "vs_baseline": None, "data": "synthetic"})
            print(json.dumps(rec), flush=True)
        if c.sampler:
            c.sampler.close()
        if world > 1:
            dist.destroy_process_group()
        return
    r = bench_render(args, c, H, W, N, args.steps, args.warmup, fine=args.fine, fused=(args.render_path == "fused"), dump=dump)
    if dump:
        dump_outputs(args.dump_outputs, r.pop("outputs"))
    M = H * W * N
    achieved = FLOP_FWD * M / (r["mlp_ms"] * 1e-3) / 1e12
    executed = flop_fwd_exec(args.precision) * M / (r["mlp_ms"] * 1e-3) / 1e12
    kernel_key = "chain_kernel<FwdEpi<render>>" if r["fused"] else "chain_kernel<FwdEpi<false>>"
    traffic, tsrc = load_traffic(kernel_key) if (H, W, N) == (800, 800, 64) else (None, None)
    cfg = workload_config(H, W, N, world)
    line = {
        "metric": METRIC, "value": r["value"], "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "samples_per_sec": r["value"] * N,
        "config": cfg,
        "detail": {"N_fine": args.fine, "sampler": "device Philox seed 1",
                   "render_path": ("one kernel per frame (camera -> sampler -> MLP -> compositing in chain_kernel<FwdEpi<render>>)"
                                   if r["fused"] else "4 kernels per frame: raygen, Philox sampler, fused posenc+MLP, compositing")},
        "e2e": {"value": r.get("e2e"), "unit": "rays/s", "h2d_bytes_per_step": 64, "d2h_bytes_per_step": H * W * 16,
                "api": "FrameRenderer.render_frame_host(pose_pinned) -> pinned fp32 rgb + disparity frame"},
        "e2e_video_u8": {"value": r.get("e2e_u8"), "unit": "rays/s", "h2d_bytes_per_step": 64, "d2h_bytes_per_step": H * W * 3,
                         "api": "FrameRenderer.render_frame_u8_host: clip + BGR + uint8 on the device (render_poses' video frames)"},
        "e2e_render_image_api": {"value": r.get("api"), "unit": "rays/s", "h2d_bytes_per_step": H * W * 24, "d2h_bytes_per_step": H * W * 16,
                                 "api": f"render_image(net, rg, batch_size={REF_CHUNK}): CPU ray table, {H * W // REF_CHUNK} chunks, CPU frame"},
        "gpu_launches": r["gpu_launches"],
        "roofline": {"kernel": kernel_key + " (fused posenc+MLP, tcgen05 cta_group::2" + (", layers_2 folded into color_fc.0)" if args.precision == "bf16" else ")"), "bound": "tensor", "achieved": achieved,
                     "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved / pk["sustained"], "peak_burst": pk["burst"],
                     "frac_burst": achieved / pk["burst"], "peak_source": pk["source"] + ", sustained figure (kernel timed inside a long step)",
                     "kernel_ms": r["mlp_ms"], "flop_per_launch": FLOP_FWD * M, "traffic": traffic, "traffic_source": tsrc,
                     "executed_tflops": executed, "frac_executed": executed / pk["sustained"],
                     "frac_executed_burst": executed / pk["burst"], "flop_executed_per_launch": flop_fwd_exec(args.precision) * M,
                     "fold": FOLD_NOTE if args.precision == "bf16" else None,
                     "note": "both this kernel and the cuBLAS figure it is divided by run against the 1 kW board power cap in a long "
                             "run; a fraction near or above 1 means the kernel sustains what the vendor GEMM sustains here, and "
                             "frac_burst compares with the short-run (uncapped) cuBLAS figure"},
        "clocks": c.sampler.window(*r["t_window"]) if c.sampler else None, "outputs_finite": r.get("finite"),
    }
    if args.workload == "all" and args.fine == 0:
        # sub-records of the same run (every rank takes part; rank 0 prints)
        line["train"] = bench_train(args, c, 4096, N, args.train_steps, 20, loop_api=True)
        line["train_dp8192"] = bench_train(args, c, 8192, N, max(100, args.train_steps // 2), 20)
        if N != 128:   # the reference's own training shape: configs/lego.yaml batch_size 4096, Nf 128 (train.py:51)
            line["train_n128"] = bench_train(args, c, 4096, 128, max(100, args.train_steps // 2), 20)
        line["sharded_frame"] = bench_sharded_frame(args, c, 1600, 1600, N, frames=max(3, args.steps // 4))
        r128 = bench_render(args, c, H, W, 128, max(3, args.steps // 4), 2, e2e=False, api=False)
        line["n128"] = {"value": r128["value"], "unit": "rays/s", "ms_per_step": r128["ms_per_step"], "samples_per_sec": r128["value"] * 128,
                        "mlp_tflops": FLOP_FWD * H * W * 128 / (r128["mlp_ms"] * 1e-3) / 1e12,
                        "config": f"same frames at the reference's default N=128 (configs/lego.yaml:6, utils/rendering.py:102,145)"}
        if world == 1:
            # the layer-by-layer chain (every reference layer its own tensor-core layer), same run, for comparison
            rl = bench_render(args, c, H, W, N, max(3, args.steps // 4), 2, e2e=False, api=False, precision="bf16_layerwise")
            tl = bench_train(args, c, 4096, N, max(100, args.train_steps // 2), 20, precision="bf16_layerwise")
            line["layerwise"] = {"render_value": rl["value"], "render_ms_per_step": rl["ms_per_step"], "unit": "rays/s",
                                 "render_mlp_tflops": FLOP_FWD * M / (rl["mlp_ms"] * 1e-3) / 1e12,
                                 "train_value": tl["value"], "train_ms_per_step": tl["ms_per_step"],
                                 "train_tflops": tl["roofline"]["achieved"], "dtype": "bf16_layerwise",
                                 "config": "same frames / same training step with precision bf16_layerwise (no fold: executed == algorithmic FLOPs)"}
            rx3 = bench_render(args, c, H, W, N, max(3, args.steps // 4), 2, e2e=False, api=False, precision="bf16x3")
            line["parity_mode_bf16x3"] = {"value": rx3["value"], "unit": "rays/s", "ms_per_step": rx3["ms_per_step"],
                                          "mlp_tflops_algorithmic": FLOP_FWD * M / (rx3["mlp_ms"] * 1e-3) / 1e12, "dtype": "bf16x3",
                                          "config": "same frames in the tensor-core fp32-class mode (error-compensated bf16, 3 MMA passes per K-block; "
                                                    "max abs err <= 1e-4 vs the reference, tests/test_gpu_parity.py); the SIMT fp32 mode runs at ~25 TFLOP/s"}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_subprocess(args)
            try:
                line["reference_gpu_eager"] = reference_gpu_eager(H, W, N, c.dev)
            except Exception as e:
                line["reference_gpu_eager"] = {"value": None, "error": repr(e)[:200]}
        print(json.dumps(line), flush=True)
    if c.sampler:
        c.sampler.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="all", choices=["all", "render", "train"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the headline workload: frames (default 20), or train steps with --workload train "
                         "(default 500: a train step is ~1 ms, enough of them for nvidia-smi to sample the clocks)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--train-steps", type=int, default=400, help="timed steps of the train sub-records")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "bf16_layerwise"])
    ap.add_argument("--res", type=int, default=800)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="reference arm: skip the configs[0] extras")
    ap.add_argument("--fine", type=int, default=0, help="extension: fine samples per ray (64 coarse + N fine)")
    ap.add_argument("--render-path", default="separate", choices=["separate", "fused"],
                    help="separate: raygen, sampler, fused posenc+MLP, compositing kernels; fused: one kernel per frame")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="B200 arm: write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB); "
                         "with several GPUs, those of rank 0 (its own frame of the render workload)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.steps is None:
        args.steps = 500 if args.workload == "train" else 20
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return
    b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
