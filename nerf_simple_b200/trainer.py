"""Device-resident training step (the loop body of train.py:45-57 without the host round trips).

The reference selects rays with a CPU `randperm` over the whole ray table (328 ms/step,
utils/dataload.py:151), copies rays/colours/jitter to the GPU and runs ~700 ATen kernels.  Here
the ray table and the ground-truth colours live on the device, a step is
    select -> Philox jitter -> fused MLP forward (saving bf16 tiles) -> compositing forward ->
    MSE gradient -> compositing backward -> delta chain -> wgrad -> [all-reduce] -> Adam
and the 24 parameters / gradients are views of two flat fp32 buffers, so data-parallel training
needs exactly one all-reduce of 595,844 floats per step (SURVEY 8e).  Everything that varies
from step to step lives in a 32-byte device-resident state, so after two eager warm-up steps the
whole step is captured in a CUDA graph and replayed (use_graph=True; with several ranks the gradient
all-reduce is fused into the Adam kernel over NVLink peer memory, or -- NB200_P2P_ALLREDUCE=0 -- two
graphs are replayed around an eagerly launched NCCL all-reduce).  The batch can also be handed in by the caller
(`step(rays=, gt=)`, pinned host tensors copied asynchronously), which is train.py's own flow.

With a fine network (`net_fine=`, `Nf=`: the NeRF paper's hierarchical sampling, sec. 5.2) a step is
    select -> Philox jitter -> coarse forward (saving) -> coarse compositing (+ weights) -> inverse-CDF fine
    sampler -> fine forward (saving) on the Nc+Nf merged depths -> fine compositing -> the two MSE gradients ->
    both compositing backwards -> both MLP backwards -> [all-reduce] -> Adam
with the 48 parameters / gradients of both networks in the same two flat buffers (one Adam launch, one
all-reduce) and the whole step replayed as one CUDA graph like the coarse-only one.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib, config, ops
from .ops import NUM_PARAMS, flat_size, flat_views


def flatten_parameters(*nets):
    """Re-home the parameters of `nets` (24 each, in order) as views of one flat buffer (state_dicts unchanged).
    Every tensor starts on a 16-byte boundary, so the buffer has a few padding floats (always zero)."""
    params = [p for net in nets for p in net.parameters()]
    shapes = [tuple(p.shape) for p in params]
    flat = torch.zeros(flat_size(shapes), dtype=torch.float32, device=params[0].device)
    for p, v in zip(params, flat_views(flat, shapes)):
        v.copy_(p.data)
        p.data = v
    return flat


def attach_flat_grad(*nets, device=None, flat=None):
    params = [p for net in nets for p in net.parameters()]
    shapes = [tuple(p.shape) for p in params]
    if flat is None:
        flat = torch.zeros(flat_size(shapes), dtype=torch.float32, device=device or params[0].device)
    for p, v in zip(params, flat_views(flat, shapes)):
        p.grad = v
    return flat


class PeerBuffer:
    """A device buffer every rank of the node can address from its own kernels (NVLink / NVSwitch peer memory).
    The owner allocates it through the C ABI (cudaMalloc + CUDA IPC export: torch's caching allocator hands out
    interior pointers of segments it may recycle, and torch's own IPC import maps a peer buffer under the PEER's
    device, which does not make it visible to kernels of this rank's device), the handles travel through
    torch.distributed, and every rank opens the others' with its own device current."""

    def __init__(self, nbytes, device, group=None):
        import torch.distributed as dist
        lib = _lib.load()
        self.device, self.nbytes, self.group = device, int(nbytes), group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        handle = C.create_string_buffer(64)
        ptr = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(lib.nb200_p2p_alloc(self.nbytes, C.byref(ptr), handle), "nb200_p2p_alloc")
        self.ptr = ptr.value
        handles = [None] * self.world
        dist.all_gather_object(handles, (handle.raw, self.nbytes), group=group)
        self.ptrs, self._opened = [], []
        for r, (h, nb) in enumerate(handles):
            if r == self.rank:
                self.ptrs.append(self.ptr)
                continue
            if nb != self.nbytes:
                raise RuntimeError("ranks disagree on the peer buffer size")
            q = C.c_void_p()
            with torch.cuda.device(device):      # opened under THIS rank's device: its kernels will dereference it
                _lib.check(lib.nb200_p2p_open(h, C.byref(q)), f"nb200_p2p_open (rank {r})")
            self.ptrs.append(q.value)
            self._opened.append(q.value)

    def tensor(self, dtype, numel, byte_offset=0):
        """This rank's own buffer as a torch tensor (shares the memory; keeps the buffer alive)."""
        itemsize = torch.empty((), dtype=dtype).element_size()
        typestr = {torch.float32: "<f4", torch.int32: "<i4", torch.uint8: "|u1"}[dtype]
        owner = self

        class _Iface:
            __cuda_array_interface__ = {"shape": (int(numel),), "typestr": typestr, "data": (self.ptr + byte_offset, False),
                                        "version": 2, "strides": None}
            keep = owner
        assert byte_offset + numel * itemsize <= self.nbytes
        return torch.as_tensor(_Iface(), device=self.device)

    def ptr_array(self, byte_offset=0):
        return (C.c_void_p * self.world)(*[p + byte_offset for p in self.ptrs])

    def release(self):
        """Collective: every rank unmaps the peers' buffers, then (after a barrier) frees its own.  Tensors made by
        tensor() must not be used afterwards."""
        import torch.distributed as dist
        lib = _lib.load()
        torch.cuda.synchronize(self.device)
        with torch.cuda.device(self.device):
            for q in self._opened:
                lib.nb200_p2p_close(C.c_void_p(q))
            self._opened = []
            dist.barrier(group=self.group)
            if self.ptr:
                lib.nb200_p2p_free(C.c_void_p(self.ptr))
                self.ptr = None


def allreduce_mean_(flat_grad, world_size, group=None):
    """Sum the flat gradient over ranks and divide by the world size (equal local batches =>
    the global-batch mean of train.py:52).  Works with NCCL (GPU) and gloo (CPU tests)."""
    if world_size > 1:
        import torch.distributed as dist
        if flat_grad.is_cuda and dist.get_backend(group) == "nccl":
            dist.all_reduce(flat_grad, op=dist.ReduceOp.AVG, group=group)      # one collective, no scaling kernel
        else:
            dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM, group=group)
            flat_grad.mul_(1.0 / world_size)
    return flat_grad


class Trainer:
    """`seed` keys the ray selection and the jitter.  With world_size > 1 the rank is folded into it (every rank
    must draw different rays, or the all-reduce averages identical gradients) and the parameters are broadcast
    from rank 0 once, so replicas start identical whatever each rank's torch seed or checkpoint was -- what
    DistributedDataParallel would enforce.
    `net_fine` / `Nf` (hierarchical sampling): a fine network trained on the N coarse + Nf importance-sampled depths
    of every ray, with loss = coarse MSE + fine MSE (the paper's); its parameters share the flat buffers, the Adam
    launch and the all-reduce with `net`'s.  Needs 3 <= N <= 128 and N + Nf <= 384 (the fine sampler's limits)."""

    def __init__(self, net, rays_table, gt_table, N=64, batch_size=4096, lr=5e-4, lr_decay=1.0,
                 tn=2.0, tf=6.0, seed=1, precision="bf16", world_size=1, use_graph=True, rank=None, group=None,
                 net_fine=None, Nf=0):
        self.net, self.N, self.B = net, int(N), int(batch_size)
        # hierarchical sampling: N coarse samples for `net`, N + Nf merged samples for `net_fine` (FrameRenderer's names)
        self.net_fine, self.Nf = net_fine, int(Nf)
        self.tn, self.tf = float(tn), float(tf)
        self.precision = {"fp32": _lib.FP32, "bf16": _lib.BF16, "bf16_layerwise": _lib.BF16_LAYERWISE, "bf16x3": _lib.BF16X3}[precision]
        # the tensor-core modes: packed weight images refreshed every step, the step captured in one CUDA graph
        self._tc = self.precision in _lib.BF16_MODES or self.precision == _lib.BF16X3
        self.world_size, self.group = int(world_size), group
        self.rank = 0
        if self.world_size > 1:
            import torch.distributed as dist
            self.rank = dist.get_rank(group) if rank is None else int(rank)
        self.seed = int(seed) + 0x9E3779B1 * self.rank          # distinct Philox keys per rank
        self.device = next(net.parameters()).device
        if (net_fine is None) != (self.Nf == 0) or self.Nf < 0:
            raise ValueError(f"Nf={self.Nf}: a fine network needs Nf >= 1 fine samples per ray, and Nf > 0 needs net_fine")
        if net_fine is not None:
            if not 3 <= self.N <= 128 or self.N + self.Nf > 384:
                raise ValueError(f"N={self.N}, Nf={self.Nf}: the fine sampler needs 3 <= N <= 128 and N + Nf <= 384")
            if next(net_fine.parameters()).device != self.device:
                raise ValueError(f"net_fine is on {next(net_fine.parameters()).device}, net on {self.device}")
        nets = (net,) if net_fine is None else (net, net_fine)
        self.rays_table = _lib.require_cuda(rays_table, "rays_table").float().contiguous()
        self.gt_table = _lib.require_cuda(gt_table, "gt_table").float().contiguous()
        if self.rays_table.dim() != 2 or self.rays_table.shape[1] != 6 or self.gt_table.dim() != 2 or self.gt_table.shape[1] != 3:
            raise ValueError("rays_table must be [n,6] and gt_table [n,3]")
        if self.rays_table.shape[0] != self.gt_table.shape[0] or self.rays_table.shape[0] == 0:
            raise ValueError(f"rays_table has {self.rays_table.shape[0]} rows, gt_table {self.gt_table.shape[0]}: "
                             "the selection kernel gathers both with the same indices")
        self.flat_param = flatten_parameters(*nets)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.broadcast(self.flat_param, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        # Multi-rank steps: the gradient all-reduce is fused into the Adam kernel over NVLink peer memory
        # (nb200_adam_allreduce_p2p), so a step stays ONE graph replay; the flat gradient then lives in a peer-shareable
        # buffer.  NB200_P2P_ALLREDUCE=0, or ranks without peer access, use NCCL instead: two graphs are replayed around
        # the eagerly launched collective (capturing the NCCL all-reduce itself inside torch.cuda.graph hung on this
        # stack -- torch 2.11, NCCL 2.28.9 -- in every capture mode).
        self._p2p, self.p2p_error = None, None
        flat_grad = None
        if self.world_size > 1 and os.environ.get("NB200_P2P_ALLREDUCE", "1") == "1" and self.flat_param.is_cuda:
            flat_grad = self._setup_p2p()
        self.flat_grad = attach_flat_grad(*nets, flat=flat_grad)
        self.params = net.kernel_params()
        self.grads = [p.grad for p in self.params]
        # train.py:43 Adam(lr=5e-4, betas=(0.9,0.999), eps=1e-8) with a per-step exponential lr decay
        # (train.py:39,56-57), as one kernel over the flat buffer
        self.lr, self.betas, self.eps, self.t = float(lr), (0.9, 0.999), 1e-8, 0
        self.exp_avg = torch.zeros_like(self.flat_param)
        self.exp_avg_sq = torch.zeros_like(self.flat_param)
        self.lr_decay = lr_decay
        lib = _lib.load()
        M = self.B * self.N
        self._out = torch.empty((M, 4), dtype=torch.float32, device=self.device)
        self._dout = torch.empty((M, 4), dtype=torch.float32, device=self.device)
        self._saved = torch.empty(lib.nb200_mlp_saved_bytes(self.precision, M), dtype=torch.uint8, device=self.device)
        # the two backward calls of a hierarchical step are stream-ordered: one scratch of the larger size serves both
        M_all = self.B * (self.N + self.Nf)
        self._scratch = torch.empty(max(16, lib.nb200_mlp_scratch_bytes(self.precision, max(M, M_all), 1)), dtype=torch.uint8,
                                    device=self.device)
        self._rgb = torch.empty((self.B, 3), dtype=torch.float32, device=self.device)
        self._disp = torch.empty((self.B,), dtype=torch.float32, device=self.device)
        self._acc = torch.empty((self.B,), dtype=torch.float32, device=self.device)
        self._rays = torch.empty((self.B, 6), dtype=torch.float32, device=self.device)
        self._gt = torch.empty((self.B, 3), dtype=torch.float32, device=self.device)
        self._drgb = torch.empty((self.B, 3), dtype=torch.float32, device=self.device)
        self._loss = torch.zeros((), dtype=torch.float32, device=self.device)
        self._ts = torch.empty((self.B, self.N), dtype=torch.float32, device=self.device)
        self._offset = 0
        # Philox quads one step moves the sampler position on.  The fine sampler reads the same position as the
        # stratified one (its own counter tag keeps the two streams apart), so the step advances past the longer one:
        # by B*N/4 alone, a step would re-draw part of the previous step's fine jitter whenever Nf > N.
        self._sample_inc = max((M + 3) // 4, (self.B * self.Nf + 3) // 4)
        if net_fine is not None:
            NA = self.N + self.Nf
            self.params_fine = net_fine.kernel_params()
            self.grads_fine = [p.grad for p in self.params_fine]
            self._w = torch.empty((self.B, self.N), dtype=torch.float32, device=self.device)
            self._z = torch.empty((self.B, NA), dtype=torch.float32, device=self.device)
            self._u_fine = torch.empty((self.B, self.Nf), dtype=torch.float32, device=self.device)
            self._out_f = torch.empty((M_all, 4), dtype=torch.float32, device=self.device)
            self._dout_f = torch.empty((M_all, 4), dtype=torch.float32, device=self.device)
            self._saved_f = torch.empty(lib.nb200_mlp_saved_bytes(self.precision, M_all), dtype=torch.uint8, device=self.device)
            self._rgb_f = torch.empty((self.B, 3), dtype=torch.float32, device=self.device)
            self._drgb_f = torch.empty((self.B, 3), dtype=torch.float32, device=self.device)
            self._loss_c = torch.zeros((), dtype=torch.float32, device=self.device)
            self.loss_fine = torch.zeros((), dtype=torch.float32, device=self.device)   # the fine pass's MSE (what PSNR is of)
            self._seed_fine = self.seed + 7919                                          # fine Philox key (FrameRenderer's)
        # device-resident step state (Philox positions, Adam step, lr) + stable pointer arrays: a step is a fixed
        # sequence of launches that a CUDA graph can replay
        self._state = torch.zeros(_lib.TRAIN_STATE_BYTES, dtype=torch.uint8, device=self.device)
        _lib.check(lib.nb200_train_state_init(_lib.ptr(self._state), 0, 0, 0, self.lr, _lib.stream_ptr(self.device)),
                   "nb200_train_state_init")
        self._param_ptrs = _lib.ptr_array(self.params)
        self._grad_ptrs = _lib.ptr_array(self.grads)
        self._packed_buf = (torch.empty(lib.nb200_packed_weights_bytes(self.precision), dtype=torch.uint8, device=self.device)
                            if self._tc else None)
        if net_fine is not None:
            self._param_ptrs_fine = _lib.ptr_array(self.params_fine)
            self._grad_ptrs_fine = _lib.ptr_array(self.grads_fine)
            self._packed_buf_fine = torch.empty_like(self._packed_buf) if self._tc else None
        self.use_graph = bool(use_graph) and self._tc and self.N % 4 == 0 and self.N <= 1024
        # why the step is NOT one CUDA-graph replay, when it is not (the eager path computes the same numbers, with
        # ~14 launches of host overhead per step): readable by the caller instead of a silent fallback
        self.graph_off_reason = (None if self.use_graph else
                                 "use_graph=False" if not use_graph else
                                 "precision is fp32 (the SIMT step is ~65 launches, not captured)" if not self._tc else
                                 f"N={self.N}: the device-resident sampler state needs N % 4 == 0 and N <= 1024")
        if use_graph and not self.use_graph:
            import warnings
            warnings.warn(f"nerf_simple_b200.Trainer: CUDA-graph replay is off ({self.graph_off_reason}); steps are launched eagerly")
        self._graphs, self.graph_error = {}, None
        self.launches = 0
        self.part_events = []
        self.last_loss = None

    def _setup_p2p(self):
        """Allocate the flat gradient + the flag block in a peer-shareable buffer and map the other ranks' (same node,
        <= 8 ranks).  Returns the gradient tensor, or None when any rank failed (all ranks then use NCCL)."""
        import torch.distributed as dist
        ok = torch.ones(1, device=self.device)
        flat = None
        try:
            if self.world_size > 8:
                raise RuntimeError("more than 8 ranks")
            n = self.flat_param.numel()
            flag_off = (n * 4 + 255) // 256 * 256
            buf = PeerBuffer(flag_off + _lib.P2P_FLAG_WORDS * 4, self.device, self.group)
            flat = buf.tensor(torch.float32, n)
            self._p2p = (buf, buf.ptr_array(0), buf.ptr_array(flag_off))
        except Exception as e:      # noqa: BLE001 -- any failure means "use NCCL"; recorded, and agreed on by all ranks below
            self.p2p_error = repr(e)
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)      # every rank takes the same path
        if float(ok) == 0.0:
            self._p2p, flat = None, None
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        return flat

    # ------------------------------------------------------------------------------------------ one step
    def _enqueue_step(self, time_parts=False, part="all", select=True, sample=True, u_fine=False):
        """Enqueue one training step on the current stream.  Everything that changes from step to step (Philox
        positions, Adam's step count, the learning rate) is read from the device-resident train state, so
        the same sequence of launches can be captured once in a CUDA graph and replayed.
        select=False: the batch (self._rays, self._gt) was supplied by the caller (host-side selection like
        train.py:47-49); sample=False: the sample depths self._ts were supplied too (parity tests); u_fine=True: so
        were the fine sampler's uniform draws self._u_fine."""
        lib = _lib.load()
        dev, B, N, M = self.device, self.B, self.N, self.B * self.N
        st = _lib.stream_ptr(dev)
        state = _lib.ptr(self._state)
        if part == "update":
            return self._enqueue_update(lib, state, st)
        fine = self.net_fine is not None
        rays, gt, ts = self._rays, self._gt, self._ts
        if select:   # ray selection with replacement on the device (rg.select + train_imgs[ray_ids], train.py:47-49)
            _lib.check(lib.nb200_select_rays_state(_lib.ptr(self.rays_table), _lib.ptr(self.gt_table), self.rays_table.shape[0],
                                                   self.seed ^ 0x5E1EC7, state, B, _lib.ptr(rays), _lib.ptr(gt), None, st),
                       "nb200_select_rays_state")
        if not sample:
            pass
        elif N % 4 == 0 and N <= 1024:
            _lib.check(lib.nb200_stratified_ts_state(self.seed, state, B, N, self.tn, self.tf, _lib.ptr(ts), st),
                       "nb200_stratified_ts_state")
        else:   # ragged N: host-side stream position (not graph-replayable; use_graph is off for such N)
            _lib.check(lib.nb200_stratified_ts(None, self.seed, self._offset, B, N, self.tn, self.tf, _lib.ptr(ts), st),
                       "nb200_stratified_ts")
        pa = self._param_ptrs
        packed = self._packed_buf
        if self._tc:   # the optimizer changed the fp32 masters: refresh the bf16 (hi / lo) operand images
            _lib.check(lib.nb200_pack_weights(self.precision, pa, _lib.ptr(packed), st), "nb200_pack_weights")
            if fine:
                _lib.check(lib.nb200_pack_weights(self.precision, self._param_ptrs_fine, _lib.ptr(self._packed_buf_fine), st),
                           "nb200_pack_weights")
        if time_parts:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record()
        _lib.check(lib.nb200_mlp_forward(self.precision, _lib.IN_RAYS, _lib.ptr(rays), _lib.ptr(ts), M, N, pa,
                                         _lib.ptr(packed), _lib.ptr(self._out), _lib.ptr(self._saved), None, 0, st),
                   "nb200_mlp_forward")
        if time_parts:
            ev[1].record()
        _lib.check(lib.nb200_composite_forward(_lib.ptr(self._out), _lib.ptr(ts), _lib.ptr(rays), 1, B, N,
                                               _lib.ptr(self._rgb), _lib.ptr(self._disp), _lib.ptr(self._acc),
                                               None, _lib.ptr(self._w) if fine else None, st), "nb200_composite_forward")
        if fine:   # importance-resample Nf depths from the coarse weights (no gradient flows through them), fine pass
            NA, M_all, z = N + self.Nf, B * (N + self.Nf), self._z
            if u_fine:
                _lib.check(lib.nb200_sample_pdf_merge(_lib.ptr(ts), _lib.ptr(self._w), _lib.ptr(self._u_fine), 0, 0, 0,
                                                      B, N, self.Nf, _lib.ptr(z), st), "nb200_sample_pdf_merge")
            else:
                _lib.check(lib.nb200_sample_pdf_merge_state(_lib.ptr(ts), _lib.ptr(self._w), self._seed_fine, state,
                                                            B, N, self.Nf, _lib.ptr(z), st), "nb200_sample_pdf_merge_state")
            _lib.check(lib.nb200_mlp_forward(self.precision, _lib.IN_RAYS, _lib.ptr(rays), _lib.ptr(z), M_all, NA,
                                             self._param_ptrs_fine, _lib.ptr(self._packed_buf_fine), _lib.ptr(self._out_f),
                                             _lib.ptr(self._saved_f), None, 0, st), "nb200_mlp_forward")
            _lib.check(lib.nb200_composite_forward(_lib.ptr(self._out_f), _lib.ptr(z), _lib.ptr(rays), 1, B, NA,
                                                   _lib.ptr(self._rgb_f), _lib.ptr(self._disp), _lib.ptr(self._acc),
                                                   None, None, st), "nb200_composite_forward")
        # MSELoss over B*3 and its gradient (train.py:42,52); hierarchical: loss = coarse + fine, as in the paper
        _lib.check(lib.nb200_mse_loss_grad(_lib.ptr(self._rgb), _lib.ptr(gt), B, _lib.ptr(self._drgb),
                                           _lib.ptr(self._loss_c if fine else self._loss), st), "nb200_mse_loss_grad")
        if fine:
            _lib.check(lib.nb200_mse_loss_grad(_lib.ptr(self._rgb_f), _lib.ptr(gt), B, _lib.ptr(self._drgb_f),
                                               _lib.ptr(self.loss_fine), st), "nb200_mse_loss_grad")
            torch.add(self._loss_c, self.loss_fine, out=self._loss)
        _lib.check(lib.nb200_composite_backward(_lib.ptr(self._out), _lib.ptr(ts), _lib.ptr(rays), 1, _lib.ptr(self._drgb),
                                                None, None, None, None, B, N, _lib.ptr(self._dout), st),
                   "nb200_composite_backward")
        if fine:
            _lib.check(lib.nb200_composite_backward(_lib.ptr(self._out_f), _lib.ptr(z), _lib.ptr(rays), 1, _lib.ptr(self._drgb_f),
                                                    None, None, None, None, B, NA, _lib.ptr(self._dout_f), st),
                       "nb200_composite_backward")
        self.flat_grad.zero_()
        if time_parts:
            ev[2].record()
        _lib.check(lib.nb200_mlp_backward(self.precision, _lib.IN_RAYS, _lib.ptr(rays), _lib.ptr(ts), M, N, pa,
                                          _lib.ptr(packed), _lib.ptr(self._dout), _lib.ptr(self._saved),
                                          self._grad_ptrs, _lib.ptr(self._scratch), self._scratch.numel(), st),
                   "nb200_mlp_backward")
        if fine:
            _lib.check(lib.nb200_mlp_backward(self.precision, _lib.IN_RAYS, _lib.ptr(rays), _lib.ptr(z), M_all, NA,
                                              self._param_ptrs_fine, _lib.ptr(self._packed_buf_fine), _lib.ptr(self._dout_f),
                                              _lib.ptr(self._saved_f), self._grad_ptrs_fine, _lib.ptr(self._scratch),
                                              self._scratch.numel(), st), "nb200_mlp_backward")
        if time_parts:
            ev[3].record()
            self.part_events.append(ev)
        if part == "grads":      # two-graph mode: the all-reduce is launched eagerly between the two graphs
            return
        if self._p2p is None:
            allreduce_mean_(self.flat_grad, self.world_size, self.group)
        self._enqueue_update(lib, state, st)

    def _enqueue_update(self, lib, state, st):
        B = self.B
        if self._p2p is not None:   # all-reduce fused into Adam: peers' gradients are read over NVLink inside the kernel
            _lib.check(lib.nb200_adam_allreduce_p2p(_lib.ptr(self.flat_param), self._p2p[1], self._p2p[2], self.rank, self.world_size,
                                                    _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq), self.flat_param.numel(), state,
                                                    self.betas[0], self.betas[1], self.eps, st), "nb200_adam_allreduce_p2p")
        else:
            _lib.check(lib.nb200_adam_step_state(_lib.ptr(self.flat_param), _lib.ptr(self.flat_grad), _lib.ptr(self.exp_avg),
                                                 _lib.ptr(self.exp_avg_sq), self.flat_param.numel(), state, self.betas[0],
                                                 self.betas[1], self.eps, st), "nb200_adam_step_state")
        _lib.check(lib.nb200_train_state_advance(state, B, self._sample_inc, self.lr_decay, st), "nb200_train_state_advance")

    def _capture(self, select):
        """Capture one step in CUDA graphs (after eager warm-up steps have set kernel attributes, cached the
        tensor maps and initialised NCCL).  One graph per step; with several ranks the all-reduce is fused into the
        Adam kernel (peer memory) or -- fallback -- two graphs are replayed around the eagerly launched NCCL collective.
        Every rank takes the same branch: _setup_p2p agreed on it with a collective, never a local exception."""
        torch.cuda.synchronize(self.device)
        if self.world_size == 1 or self._p2p is not None:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._enqueue_step(select=select)
            self._graphs[select] = (g,)
        else:
            ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(ga):
                self._enqueue_step(part="grads", select=select)
            with torch.cuda.graph(gb):
                self._enqueue_step(part="update")
            self._graphs[select] = (ga, gb)

    def close(self):
        """Release the peer-shared gradient buffer (collective over the ranks; a no-op on one GPU).  The Trainer must
        not be stepped afterwards."""
        if self._p2p is not None:
            buf = self._p2p[0]
            self._graphs.clear()
            for net in (self.net, self.net_fine):
                for p in (net.parameters() if net is not None else ()):
                    p.grad = None
            self.flat_grad = self.grads = self.grads_fine = None
            self._p2p = None
            buf.release()

    @property
    def launch_mode(self):
        if not self._graphs:
            return "eager launches"
        g = next(iter(self._graphs.values()))
        if len(g) == 1:
            return "one CUDA-graph replay per step" + (" (gradient all-reduce fused into the Adam kernel over NVLink peer memory)" if self.world_size > 1 else "")
        return "two CUDA graphs per step around the eagerly launched NCCL all-reduce"

    def step(self, sync_loss=False, time_parts=False, rays=None, gt=None, ts=None, u_fine=None):
        """One training step; returns its loss (coarse + fine with a fine network; the fine term alone is
        `self.loss_fine`, a device scalar).  By default the batch is selected on the device.  rays [B,6] / gt [B,3]
        given (any device; pinned host tensors are copied asynchronously): the caller's batch is used instead, like
        train.py:47-51 does with rg.select + `.cuda()`; `ts` [B,N] given as well: those sample depths instead of the
        Philox jitter, and `u_fine` [B,Nf]: those uniform draws for the fine sampler (parity tests; eager launches).
        time_parts=True (eager launches, coarse-only) records CUDA events around the MLP forward and the MLP backward
        in self.part_events for bench.py's roofline."""
        fine = self.net_fine is not None
        if time_parts and fine:
            raise ValueError("time_parts=True times the coarse-only step; time whole hierarchical steps instead")
        if u_fine is not None and not fine:
            raise ValueError("u_fine needs a fine network (Trainer(net_fine=..., Nf=...))")
        select = rays is None
        if not select:
            if gt is None or tuple(rays.shape) != (self.B, 6) or tuple(gt.shape) != (self.B, 3):
                raise ValueError(f"rays must be [{self.B},6] and gt [{self.B},3]")
            self._rays.copy_(rays, non_blocking=True)
            self._gt.copy_(gt, non_blocking=True)
        if ts is not None:
            if tuple(ts.shape) != (self.B, self.N):
                raise ValueError(f"ts must be [{self.B},{self.N}]")
            self._ts.copy_(ts, non_blocking=True)
        if u_fine is not None:
            if tuple(u_fine.shape) != (self.B, self.Nf):
                raise ValueError(f"u_fine must be [{self.B},{self.Nf}]")
            self._u_fine.copy_(u_fine, non_blocking=True)
        if self.use_graph and not time_parts and ts is None and u_fine is None:
            if select not in self._graphs and self.t >= 2:
                self._capture(select)
            g = self._graphs.get(select)
            if g is not None:
                g[0].replay()
                if len(g) == 2:
                    allreduce_mean_(self.flat_grad, self.world_size, self.group)
                    g[1].replay()
            else:
                self._enqueue_step(select=select)
        else:
            self._enqueue_step(time_parts, select=select, sample=ts is None, u_fine=u_fine is not None)
        self.t += 1
        self._offset += self._sample_inc
        self.lr *= self.lr_decay
        self._bump_versions()
        # select, ts, pack x2, fwd, comp fwd, mse, comp bwd, bwd kernels, unpad, adam, state (+ memsets); the folded bf16
        # chain adds the fold / un-fold kernels, bf16_layerwise and bf16x3 have none.  A fine network repeats everything
        # but select, ts, adam and state, and adds the fine sampler (+ one ATen add for the summed loss).
        per_net = (12 if self.precision == _lib.BF16 else 10) if self._tc else 61
        self.launches += 4 + per_net * (2 if fine else 1) + (1 if fine else 0) - (0 if select else 1) - (0 if ts is None else 1)
        self.last_loss = self._loss
        return float(self._loss) if sync_loss else self._loss.clone()

    def _bump_versions(self):
        # the optimizer updated the flat buffer, not the 24 (48) views: invalidate the packed-weight caches
        self.net._packed.invalidate()
        if self.net_fine is not None:
            self.net_fine._packed.invalidate()
