/* nerf_b200.h -- C ABI of libnerf_b200.so, the B200 (sm_100a) engine behind the Nerf-Simple
 * Python call surface.
 *
 * The reference (UCSD-Comp-Imaging/Nerf-Simple) has no FFI of its own: its hot path is Python
 * calling ATen.  Each entry point below replaces the ATen launches of one reference function
 * (cited per entry as file:line relative to the reference checkout) and is what a maintainer
 * would bind from utils/rendering.py / utils/nets.py with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C types only: device pointers, sizes, a CUDA stream handle; no torch types.
 *   - every function returns 0 (NB200_OK) or a negative error code; nothing throws, nothing
 *     allocates device memory (all workspaces are caller-allocated), nothing synchronises the
 *     device.  Work is enqueued on `stream`.
 *   - all tensors are dense row-major fp32 unless stated; "dev" = device pointer.
 *   - alignment: [.,4] per-sample tensors (MLP out, its cotangent) 16 bytes, [.,6] ray / point
 *     tensors 8 bytes (NB200_ERR_ARG otherwise); everything else 4 bytes, with vector fast
 *     paths taken when 16-byte aligned.  count == 0 succeeds without touching the pointers.
 *   - there is NO CPU fallback: without an sm_100 device the compute calls fail with
 *     NB200_ERR_CUDA / NB200_ERR_ARCH.
 */
#ifndef NERF_B200_H
#define NERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* nb200_stream_t; /* cudaStream_t */

enum {
  NB200_OK = 0,
  NB200_ERR_ARG = -1,         /* bad argument (null pointer, size <= 0, N < 2, ...)        */
  NB200_ERR_UNSUPPORTED = -2, /* shape/precision outside what the kernels are built for    */
  NB200_ERR_CUDA = -3,        /* a CUDA runtime call failed; see nb200_last_cuda_error()   */
  NB200_ERR_ARCH = -4,        /* device is not sm_100 (tcgen05 kernels cannot run)         */
  NB200_ERR_WORKSPACE = -5,   /* caller workspace too small                                */
  NB200_ERR_KERNEL = -6       /* a kernel reported an internal failure (pipeline timeout)  */
};

/* precision of the MLP path */
enum {
  NB200_FP32 = 0, /* fp32 SIMT layer kernels; parity mode, max-abs err <= 1e-4 vs reference    */
  NB200_BF16 = 1, /* fused tcgen05 kernel, bf16 operands + fp32 accumulate in TMEM; <= 1e-2.
                     layers_2 (utils/nets.py:41, no activation) is folded into color_fc.0 at pack time (the
                     product of the two weights is formed in fp32): 9 tensor-core layers per sample instead of
                     10; the backward un-folds the gradients of both layers exactly (chain rule).            */
  NB200_BF16X3 = 2, /* the same tcgen05 chain with error-compensated bf16 (hi/lo images of activations and
                      weights, three MMA passes per K-block): fp32-class accuracy (<= 1e-4, also with weights
                      scaled x1.5) on the tensor cores, forward and backward (layer by layer, no fold: the
                      delta chain and the weight gradients take the same three passes).  Its packed buffer,
                      saved tensors and scratch have their own sizes and layouts (the *_bytes queries). */
  NB200_BF16_LAYERWISE = 3 /* NB200_BF16 without the fold: every layer of utils/nets.py:34-43 is its own
                      tensor-core layer.  Same packed image, saved-tensor and scratch layouts as NB200_BF16. */
};

/* input mode of the MLP kernels */
enum {
  NB200_IN_POINTS = 0, /* in0 = query points [M,6] (x,y,z,d1,d2,d3): Nerf.forward, nets.py:34  */
  NB200_IN_RAYS = 1    /* in0 = rays [B,6], in1 = ts [B,N]; points o+t*d and d/|d| are built in
                          registers: render_nerf, rendering.py:31-40                          */
};

/* (viii) version / build query */
int nb200_version(void);            /* 100*major + minor */
int nb200_compiled_arch(void);      /* 100 -> built for sm_100a */
int nb200_device_arch(void);        /* 10*major+minor of the current device, or <0 */
const char* nb200_error_string(int code);
const char* nb200_last_cuda_error(void);

/* (vii) device ray generation.  Replaces utils/xyz.py:38-52 (rays_single_cam) followed by
 * utils/rendering.py:129-134 / utils/dataload.py:123-127 (R @ dirs, origin broadcast, pack).
 * Ray r in [0, P*H*W): pose r / (H*W), pixel (h, w) = divmod(r % (H*W), W);
 * camera dir = ((w - W/2)/f, -(h - H/2)/f, -1) (integer centre, no +0.5).
 * poses: dev [P,4,4] row-major camera-to-world.  rays: dev [n_rays,6] = (origin, dir). */
int nb200_generate_rays(const float* poses, int P, int H, int W, float f, int64_t ray_begin,
                        int64_t n_rays, float* rays, nb200_stream_t stream);

/* (vi) stratified sampler.  Replaces utils/rendering.py:24-30: ts = bin*u + t_bins[:-1],
 * t_bins = linspace(tn, tf, N+1) with torch.linspace's fp32 rounding.
 * u != NULL: reference-RNG mode, u is dev [B,N] drawn by the caller (torch.rand on the CPU
 *            generator, like the reference) -> bit-identical ts.
 * u == NULL: throughput mode, Philox4x32-10 keyed by (seed, offset + sample index). */
int nb200_stratified_ts(const float* u, uint64_t seed, uint64_t offset, int64_t B, int N, float tn,
                        float tf, float* ts, nb200_stream_t stream);

/* (iv) compositing forward.  Replaces utils/rendering.py:60-85 (volume_render).
 * outs dev [B,N,4] (r,g,b,sigma), ts dev [B,N].
 * dirs_mode 0: dirs dev [B,3] exactly as passed to volume_render (deltas scale by its norm, :62).
 * dirs_mode 1: dirs is the rays tensor dev [B,6]; the direction is normalised first, as
 *              render_nerf does at :37 before calling volume_render at :43.
 * rgb [B,3], disp [B], acc [B] are always written; alpha / weights [B,N] when non-NULL. */
int nb200_composite_forward(const float* outs, const float* ts, const float* dirs, int dirs_mode,
                            int64_t B, int N,
                            float* rgb, float* disp, float* acc, float* alpha, float* weights,
                            nb200_stream_t stream);

/* (v) compositing backward (analytic; what autograd does through rendering.py:60-83).
 * Cotangents d_rgb [B,3] (required), d_disp [B], d_acc [B], d_alpha [B,N], d_w [B,N] (each may
 * be NULL = zero).  Writes d_outs [B,N,4].  ts/dirs carry no gradient in the reference. */
int nb200_composite_backward(const float* outs, const float* ts, const float* dirs, int dirs_mode,
                             const float* d_rgb, const float* d_disp, const float* d_acc,
                             const float* d_alpha, const float* d_w, int64_t B, int N,
                             float* d_outs, nb200_stream_t stream);

/* positional encoding only.  Replaces utils/xyz.py:16-36 for direct callers of
 * positional_encoder: v dev [M,6] -> posx [M,3+6*Lp], posd [M,3+6*Ld], column order
 * coordinate-major, then level, sin before cos; frequencies 2^i, no pi. */
int nb200_positional_encoding(const float* v, int64_t M, int Lp, int Ld, float* posx, float* posd,
                              nb200_stream_t stream);

/* (i) weight packing.  params: HOST array of 24 DEVICE pointers in state_dict order
 * (utils/nets.py:16-32; layers_0.0.weight, layers_0.0.bias, ..., color_fc.2.bias).
 * NB200_FP32 uses the parameters in place (packed may be NULL, bytes == 0).
 * NB200_BF16 / NB200_BF16_LAYERWISE write the tcgen05 operand images (bf16, K-major, 128B-swizzled,
 * padded/split K: 63->64, 319->256+64, 283->256+32, plus the transposed images for dgrad), the slabs
 * of the folded weight color_fc.0[:, :256] x layers_2 and an fp32 tail (biases, heads, and the fp32
 * copies the backward un-folds gradients with): one image serves both modes. */
size_t nb200_packed_weights_bytes(int precision);
int nb200_pack_weights(int precision, const float* const* params, void* packed,
                       nb200_stream_t stream);

/* workspace sizes for M samples.  `train` != 0: forward keeps what backward needs. */
size_t nb200_mlp_saved_bytes(int precision, int64_t M);     /* forward -> backward tensors  */
size_t nb200_mlp_scratch_bytes(int precision, int64_t M, int train);

/* (ii) fused posenc + MLP forward.  Replaces utils/nets.py:34-43 (+ utils/xyz.py:16-36, and in
 * NB200_IN_RAYS mode utils/rendering.py:31-40).  M = number of samples (B*N in rays mode).
 * out dev [M,4] = (r,g,b,sigma) raw.  saved: NULL for inference, else >= saved_bytes. */
int nb200_mlp_forward(int precision, int in_mode, const float* in0, const float* in1, int64_t M,
                      int N, const float* const* params, const void* packed, float* out,
                      void* saved, void* scratch, size_t scratch_bytes, nb200_stream_t stream);

/* (iii) MLP backward.  d_out dev [M,4] -> grads: HOST array of 24 DEVICE pointers (same order
 * and shapes as params; typically views into one flat 595,844-float buffer).  Gradients are
 * ACCUMULATED (+=) like autograd; zero them first for a fresh gradient.  No input gradient:
 * query points never require grad in the reference (rendering.py:39-41).
 * `precision`, `packed` and `saved` must be the ones of the forward call this is the backward of
 * (NB200_BF16 does not save layers_2's output; its backward reads the fp32 tail of `packed`). */
int nb200_mlp_backward(int precision, int in_mode, const float* in0, const float* in1, int64_t M,
                       int N, const float* const* params, const void* packed, const float* d_out,
                       const void* saved, float* const* grads, void* scratch,
                       size_t scratch_bytes, nb200_stream_t stream);

/* Fused render (SURVEY 8f rows 2-3): sampler -> posenc + MLP -> compositing in ONE kernel for the
 * no-grad render loops (utils/rendering.py:88-153 calling render_nerf, :13-45).  Per-sample
 * (r,g,b,sigma) and the sample depths stay on chip; only rgb [B,3], disp [B], acc [B] are written.
 * Results equal nb200_stratified_ts + nb200_mlp_forward(NB200_IN_RAYS) + nb200_composite_forward
 * (dirs_mode 1) on the same inputs.  NB200_BF16 only, N in {32, 64, 128} (whole rays per 128-sample
 * tile); otherwise NB200_ERR_UNSUPPORTED and the caller uses the three separate calls.
 *   ts != NULL: sample depths dev [B,N] supplied (reference-RNG mode).
 *   ts == NULL: Philox depths, the stream nb200_stratified_ts(NULL, seed, offset, ...) would write. */
int nb200_render_rays(int precision, const float* rays, const float* ts, uint64_t seed, uint64_t offset,
                      int64_t B, int N, float tn, float tf, const void* packed, float* rgb, float* disp,
                      float* acc, nb200_stream_t stream);
/* Same, with the rays generated in the kernel from the camera (what nb200_generate_rays would write
 * for rays [ray_begin, ray_begin + n_rays) of the P*H*W table): a whole frame is one launch. */
int nb200_render_camera(int precision, const float* poses, int P, int H, int W, float f, int64_t ray_begin,
                        int64_t n_rays, uint64_t seed, uint64_t offset, int N, float tn, float tf,
                        const void* packed, float* rgb, float* disp, float* acc, nb200_stream_t stream);

/* Video-frame conversion for the render loops.  Replaces the clip of utils/rendering.py:146 followed by
 * cv2.cvtColor(RGB2BGR) and (frame*255).astype(np.uint8) of :158-159 (bgr != 0), or the same without the
 * channel swap (bgr == 0): out[p, c'] = trunc(255 * clamp(rgb[p, c], 0, 1)) with c' = 2 - c for BGR.
 * rgb dev [n_pixels,3] fp32 (unclipped or clipped), out dev [n_pixels,3] uint8: a frame leaves the device as
 * 3 B/pixel instead of 12. */
int nb200_frame_to_u8(const float* rgb, int64_t n_pixels, int bgr, uint8_t* out, nb200_stream_t stream);

/* EXTENSION (no reference counterpart: hierarchical sampling is "not implemented yet" in the
 * reference, configs/lego.yaml:7).  Inverse-CDF importance sampler of the NeRF paper (sec. 5.2):
 * pdf = weights[:,1:-1] + 1e-5 over the mid-point bins of ts [B,Nc], Nf samples per ray drawn with
 * u (mode 0: dev [B,Nf] supplied; 1: linspace(0,1,Nf); 2: Philox(seed, offset)), merged with the
 * coarse depths in ascending order into z_all [B, Nc+Nf].  Nc <= 128, Nc+Nf <= 384. */
int nb200_sample_pdf_merge(const float* ts, const float* weights, const float* u, int mode, uint64_t seed,
                           uint64_t offset, int64_t B, int Nc, int Nf, float* z_all, nb200_stream_t stream);

/* Adam update of one flat parameter buffer.  Replaces torch.optim.Adam(lr=5e-4).step() of
 * train.py:43,55 for the device-resident trainer (the 24 parameters are views of `param`):
 * m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps).
 * `step` is the 1-based step count t.  No weight decay, no amsgrad (the reference uses neither). */
int nb200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                    int64_t step, float lr, float beta1, float beta2, float eps, nb200_stream_t stream);

/* Device-side ray selection for the device-resident trainer.  Replaces rg.select('train', B) and
 * train_imgs[ray_ids] of train.py:47-49 (utils/dataload.py:141-153: a CPU randperm over the whole ray
 * table per step).  B indices uniform in [0, n_table) WITH replacement from Philox4x32-10 keyed by
 * (seed, offset + i); gathers rays_table [n_table,6] -> rays [B,6] and, when gt_table != NULL,
 * gt_table [n_table,3] -> gt [B,3].  ids (dev int64 [B]) may be NULL. */
int nb200_select_rays(const float* rays_table, const float* gt_table, int64_t n_table, uint64_t seed,
                      uint64_t offset, int64_t B, float* rays, float* gt, int64_t* ids, nb200_stream_t stream);

/* MSELoss(rgb_, gt_) and its gradient.  Replaces train.py:42,52 + the first autograd node of :54:
 * loss = mean over B*3 of (rgb-gt)^2 (written to *loss when non-NULL), d_rgb = 2 (rgb-gt) / (3B). */
int nb200_mse_loss_grad(const float* rgb, const float* gt, int64_t B, float* d_rgb, float* loss,
                        nb200_stream_t stream);

/* Device-resident step state for CUDA-graph capture of a whole training step (the loop body of
 * train.py:47-57 replayed without host involvement).  `state` is NB200_TRAIN_STATE_BYTES of device
 * memory holding the Philox positions of the ray selection and of the sampler, Adam's step count and
 * the learning rate; the *_state calls read what their plain counterparts take as host arguments
 * (offset / step / lr), and nb200_train_state_advance moves it on at the end of a step
 * (select_offset += select_inc, sample_offset += sample_inc, step += 1, lr *= lr_decay: train.py:56-57).
 * nb200_train_state_init is a one-time, synchronising set-up call. */
#define NB200_TRAIN_STATE_BYTES 32
int nb200_train_state_init(void* state, uint64_t select_offset, uint64_t sample_offset, int64_t step, float lr,
                           nb200_stream_t stream);
int nb200_train_state_advance(void* state, uint64_t select_inc, uint64_t sample_inc, float lr_decay,
                              nb200_stream_t stream);
int nb200_select_rays_state(const float* rays_table, const float* gt_table, int64_t n_table, uint64_t seed,
                            const void* state, int64_t B, float* rays, float* gt, int64_t* ids,
                            nb200_stream_t stream);
int nb200_stratified_ts_state(uint64_t seed, const void* state, int64_t B, int N, float tn, float tf, float* ts,
                              nb200_stream_t stream);   /* Philox mode, N % 4 == 0 */
int nb200_adam_step_state(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                          const void* state, float beta1, float beta2, float eps, nb200_stream_t stream);

/* Data-parallel training (new functionality, SURVEY 8e; the reference is single-GPU): the gradient all-reduce FUSED
 * into the Adam update over NVLink peer memory.  Replaces an NCCL all-reduce of the flat gradient followed by
 * nb200_adam_step_state: every rank's kernel reads the flat gradients of all `world` ranks (peer_grads: HOST array of
 * `world` DEVICE pointers, index = rank, the caller's own buffer included; peers mapped through CUDA IPC), averages
 * them in rank order and applies Adam to its own replica, so replicas stay bit-identical.  peer_flags: HOST array of
 * `world` DEVICE pointers to each rank's zero-initialised flag block of NB200_P2P_FLAG_WORDS uint32 (remote ranks write
 * arrival / completion epochs there; the epoch is the optimizer step count of `state`).  Every rank must enqueue the
 * call once per step.  n (floats) must be a multiple of 4; world <= 8 (one NVSwitch domain). */
#define NB200_P2P_FLAG_WORDS 32
/* Peer-shareable device buffers (CUDA IPC) for nb200_adam_allreduce_p2p -- the ONLY entry points that allocate or
 * synchronise.  nb200_p2p_alloc: cudaMalloc + zero `bytes` on the current device and export a 64-byte handle (send it
 * to the other ranks of the node by any host channel).  nb200_p2p_open: map a peer's buffer for kernels of the CURRENT
 * device (peer access over NVLink is enabled lazily by the driver).  close / free undo them. */
int nb200_p2p_alloc(size_t bytes, void** dev_ptr, void* handle64);
int nb200_p2p_open(const void* handle64, void** dev_ptr);
int nb200_p2p_close(void* dev_ptr);
int nb200_p2p_free(void* dev_ptr);
int nb200_adam_allreduce_p2p(float* param, const float* const* peer_grads, uint32_t* const* peer_flags, int rank, int world,
                             float* exp_avg, float* exp_avg_sq, int64_t n, const void* state, float beta1, float beta2,
                             float eps, nb200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NERF_B200_H */
