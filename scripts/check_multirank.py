"""Multi-GPU check (torchrun, one rank per GPU); run by tests/test_gpu_multirank.py and by hand:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 scripts/check_multirank.py
  1. a ray-sharded frame assembled by one all_gather is BIT-IDENTICAL to the frame one GPU renders (SURVEY 8e);
  2. a data-parallel Trainer: ranks draw different rays, replicas start identical (broadcast) and stay identical,
     the all-reduced gradient is the mean of the per-rank gradients, the loss falls; checked in the launch mode
     given by NB200_P2P_ALLREDUCE (1: all-reduce fused into the Adam kernel over peer memory, one graph; 0: NCCL between two graphs).
     --fine: the Trainer trains a coarse and a fine network (hierarchical sampling, 32 + 64 samples); both networks'
     parameters live in the one flat buffer the checks compare.
Prints one JSON line on rank 0 and exits non-zero on any failed check."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nerf_simple_b200 import ops                                    # noqa: E402
from nerf_simple_b200.engine import FrameRenderer, render_sharded   # noqa: E402
from nerf_simple_b200.nets import Nerf                              # noqa: E402
from nerf_simple_b200.trainer import Trainer                        # noqa: E402
from nerf_simple_b200.xyz import poses_to_render                    # noqa: E402

FINE = "--fine" in sys.argv[1:]
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
torch.manual_seed(100 + rank)                        # deliberately DIFFERENT initial weights per rank: the Trainer must broadcast
net = Nerf().to(dev)
poses = torch.stack(poses_to_render(4, -30, 3)).to(dev)
H = W = 96
n = H * W
res = {"fine": FINE}
# ---- 1. sharded frame == single-GPU frame (same weights everywhere first)
for p in net.parameters():
    dist.broadcast(p.data, 0)
net.invalidate_packed()
with torch.no_grad():
    sharded = FrameRenderer(net, H, W, 133.3, N=64, seed=3)
    whole = FrameRenderer(net, H, W, 133.3, N=64, seed=3)
    ok = True
    for idx in (1, 2):                               # two frames: the jitter stream advances identically on both sides
        rgb, disp = render_sharded(sharded, poses, idx, rank, world)
        rgb1, disp1 = whole.render_frame(poses, idx)
        ok &= bool(torch.equal(rgb, rgb1) and torch.equal(disp, disp1))
res["sharded_frame_bit_identical"] = ok
# ---- 2. data-parallel training
torch.manual_seed(100 + rank)
net = Nerf().to(dev)                                 # different weights per rank again
rays = ops.generate_rays(poses, H, W, 133.3)
gt = torch.sigmoid(rays[:, 3:6] * 3)
fine_kw = dict(net_fine=Nerf().to(dev), Nf=64) if FINE else {}                   # different fine weights per rank too
tr = Trainer(net, rays, gt, N=32, batch_size=1024, seed=1, world_size=world, **fine_kw)      # same seed argument on every rank
ref = tr.flat_param.clone()
dist.broadcast(ref, 0)
res["replicas_identical_after_init"] = bool(torch.equal(tr.flat_param, ref))
losses = [tr.step(sync_loss=True) for _ in range(30)]
mine = tr._rays.clone()
other = [torch.empty_like(mine) for _ in range(world)]
dist.all_gather(other, mine)
res["ranks_draw_different_rays"] = all(not torch.equal(other[0], o) for o in other[1:])
ref = tr.flat_param.clone()
dist.broadcast(ref, 0)
res["replicas_identical_after_30_steps"] = bool(torch.equal(tr.flat_param, ref))
res["launch_mode"] = tr.launch_mode
res["p2p_error"] = tr.p2p_error
res["loss_first_last"] = [losses[0], losses[-1]]
# one more step, checked end to end: the update every rank applies == Adam on the MEAN of the per-rank gradients
# (recomputed eagerly without the collective; the device-resident state is not advanced by part="grads", so the
# full step below redraws the same batch).  In the peer-memory mode the mean is never materialised: it is formed
# inside the Adam kernel from the ranks' local gradients.
import math
tr.use_graph = False
p0, m0, v0 = tr.flat_param.clone(), tr.exp_avg.clone(), tr.exp_avg_sq.clone()
tr._enqueue_step(part="grads")
mean = tr.flat_grad.clone()
dist.all_reduce(mean)
mean /= world
t_next, lr = tr.t + 1, tr.lr
tr._enqueue_step()
torch.cuda.synchronize()
m1 = 0.9 * m0 + 0.1 * mean
v1 = 0.999 * v0 + 0.001 * mean * mean
want = p0 - (lr / (1 - 0.9 ** t_next)) * m1 / (v1.sqrt() / math.sqrt(1 - 0.999 ** t_next) + 1e-8)
err = float((tr.flat_param - want).abs().max())
res["update_vs_adam_on_mean_grad_abs_err"] = err
flags = torch.tensor([float(res["sharded_frame_bit_identical"]), float(res["replicas_identical_after_init"]),
                      float(res["ranks_draw_different_rays"]), float(res["replicas_identical_after_30_steps"]),
                      float(err < 5e-5), float(losses[-1] < losses[0])], device=dev)
dist.all_reduce(flags, op=dist.ReduceOp.MIN)
if rank == 0:
    res["all_ranks_ok"] = bool(flags.min() > 0)
    print(json.dumps(res), flush=True)
ok_all = bool(flags.min() > 0)
tr.close()
dist.destroy_process_group()
sys.exit(0 if ok_all else 1)
