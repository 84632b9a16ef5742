// Dispatch of the MLP entry points of the C ABI to the fp32 (SIMT) and bf16 / bf16x3 (tcgen05) engines.
#include "common.cuh"

namespace nb200 {
// mlp_fp32.cu
size_t fp32_saved_bytes(int64_t M);
size_t fp32_scratch_bytes(int64_t M, int train);
int fp32_forward(int in_mode, const float* in0, const float* in1, int64_t M, int N,
                 const float* const* P, float* out, void* saved, void* scratch, size_t scratch_bytes,
                 cudaStream_t s);
int fp32_backward(int64_t M, const float* const* P, const float* d_out, const void* saved,
                  float* const* G, void* scratch, size_t scratch_bytes, cudaStream_t s);
// mlp_tc.cu (`precision`: NB200_BF16, NB200_BF16_LAYERWISE or NB200_BF16X3)
size_t tc_packed_bytes(int precision);
size_t tc_saved_bytes(int precision, int64_t M);
size_t tc_scratch_bytes(int precision, int64_t M, int train);
int tc_pack_weights(const float* const* P, void* packed, int precision, cudaStream_t s);
int tc_forward(int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N, const void* packed,
               float* out, void* saved, cudaStream_t s);
int tc_backward(int precision, int64_t M, const void* packed, const float* d_out, const void* saved, float* const* G,
                void* scratch, size_t scratch_bytes, cudaStream_t s);
int tc_render(int precision, const float* rays, const float* poses, int H, int W, float f, int64_t ray_begin, const float* ts,
              uint64_t seed, uint64_t offset, int64_t B, int N, float tn, float tf, const void* packed, float* rgb, float* disp,
              float* acc, cudaStream_t s);
}  // namespace nb200

// the two tcgen05 bf16 modes share the packed image and the saved / scratch layouts; NB200_BF16 runs the folded chain
static inline bool is_bf16(int precision) { return precision == NB200_BF16 || precision == NB200_BF16_LAYERWISE; }
static inline bool is_tc(int precision) { return is_bf16(precision) || precision == NB200_BF16X3; }

extern "C" {

size_t nb200_packed_weights_bytes(int precision) {
  return is_tc(precision) ? nb200::tc_packed_bytes(precision) : 0;
}

int nb200_pack_weights(int precision, const float* const* params, void* packed, nb200_stream_t stream) {
  if (precision == NB200_FP32) return NB200_OK;
  if (!is_tc(precision)) return NB200_ERR_UNSUPPORTED;
  if (!params || !packed) return NB200_ERR_ARG;
  for (int i = 0; i < 24; ++i)
    if (!params[i]) return NB200_ERR_ARG;
  return nb200::tc_pack_weights(params, packed, precision, nb200::as_stream(stream));
}

size_t nb200_mlp_saved_bytes(int precision, int64_t M) {
  if (M < 0) return 0;
  return is_tc(precision) ? nb200::tc_saved_bytes(precision, M) : nb200::fp32_saved_bytes(M);
}

size_t nb200_mlp_scratch_bytes(int precision, int64_t M, int train) {
  if (M < 0) return 0;
  return is_tc(precision) ? nb200::tc_scratch_bytes(precision, M, train) : nb200::fp32_scratch_bytes(M, train);
}

static int check_common(int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N) {
  if (precision != NB200_FP32 && !is_tc(precision)) return NB200_ERR_UNSUPPORTED;
  if (in_mode != NB200_IN_POINTS && in_mode != NB200_IN_RAYS) return NB200_ERR_ARG;
  if (M < 0) return NB200_ERR_ARG;
  if (in_mode == NB200_IN_RAYS && (N < 1 || M % N != 0)) return NB200_ERR_ARG;
  if (M > 0 && (!in0 || (in_mode == NB200_IN_RAYS && !in1))) return NB200_ERR_ARG;  // empty batch: null ok
  return NB200_OK;
}

int nb200_mlp_forward(int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N,
                      const float* const* params, const void* packed, float* out, void* saved,
                      void* scratch, size_t scratch_bytes, nb200_stream_t stream) {
  int rc = check_common(precision, in_mode, in0, in1, M, N);
  if (rc != NB200_OK) return rc;
  if (M == 0) return NB200_OK;
  if (!out || ((uintptr_t)out & 15) || ((uintptr_t)in0 & 7)) return NB200_ERR_ARG;  // float4 out rows, float2 input rows
  if (precision == NB200_FP32) {
    if (!params) return NB200_ERR_ARG;
    return nb200::fp32_forward(in_mode, in0, in1, M, N, params, out, saved, scratch, scratch_bytes,
                               nb200::as_stream(stream));
  }
  if (!packed) return NB200_ERR_ARG;
  return nb200::tc_forward(precision, in_mode, in0, in1, M, N, packed, out, saved, nb200::as_stream(stream));
}

int nb200_mlp_backward(int precision, int in_mode, const float* in0, const float* in1, int64_t M, int N,
                       const float* const* params, const void* packed, const float* d_out,
                       const void* saved, float* const* grads, void* scratch, size_t scratch_bytes,
                       nb200_stream_t stream) {
  int rc = check_common(precision, in_mode, in0, in1, M, N);
  if (rc != NB200_OK) return rc;
  if (!grads) return NB200_ERR_ARG;
  for (int i = 0; i < 24; ++i)
    if (!grads[i]) return NB200_ERR_ARG;
  if (M == 0) return NB200_OK;  // gradients are accumulated into: nothing to add
  if (!d_out || !saved || ((uintptr_t)d_out & 15) || ((uintptr_t)in0 & 7)) return NB200_ERR_ARG;
  if (precision == NB200_FP32) {
    if (!params) return NB200_ERR_ARG;
    return nb200::fp32_backward(M, params, d_out, saved, grads, scratch, scratch_bytes,
                                nb200::as_stream(stream));
  }
  if (!packed) return NB200_ERR_ARG;
  return nb200::tc_backward(precision, M, packed, d_out, saved, grads, scratch, scratch_bytes, nb200::as_stream(stream));
}

static int check_render(int precision, int64_t B, int N, const void* packed, const float* rgb, const float* disp,
                        const float* acc) {
  if (!is_bf16(precision)) return NB200_ERR_UNSUPPORTED;         // the fp32 parity mode keeps the three-kernel path
  if (B < 0 || N < 2) return NB200_ERR_ARG;
  if (N != 32 && N != 64 && N != 128) return NB200_ERR_UNSUPPORTED;  // whole rays per 128-sample tile
  if (B > 0 && (!packed || !rgb || !disp || !acc)) return NB200_ERR_ARG;
  return NB200_OK;
}

int nb200_render_rays(int precision, const float* rays, const float* ts, uint64_t seed, uint64_t offset, int64_t B, int N,
                      float tn, float tf, const void* packed, float* rgb, float* disp, float* acc, nb200_stream_t stream) {
  int rc = check_render(precision, B, N, packed, rgb, disp, acc);
  if (rc != NB200_OK) return rc;
  if (B == 0) return NB200_OK;
  if (!rays || ((uintptr_t)rays & 7)) return NB200_ERR_ARG;
  return nb200::tc_render(precision, rays, nullptr, 0, 0, 0.f, 0, ts, seed, offset, B, N, tn, tf, packed, rgb, disp, acc,
                          nb200::as_stream(stream));
}

int nb200_render_camera(int precision, const float* poses, int P, int H, int W, float f, int64_t ray_begin, int64_t n_rays,
                        uint64_t seed, uint64_t offset, int N, float tn, float tf, const void* packed, float* rgb,
                        float* disp, float* acc, nb200_stream_t stream) {
  int rc = check_render(precision, n_rays, N, packed, rgb, disp, acc);
  if (rc != NB200_OK) return rc;
  if (P <= 0 || H <= 0 || W <= 0 || !(f > 0.f) || ray_begin < 0 || ray_begin + n_rays > (int64_t)P * H * W) return NB200_ERR_ARG;
  if (n_rays == 0) return NB200_OK;
  if (!poses) return NB200_ERR_ARG;
  return nb200::tc_render(precision, nullptr, poses, H, W, f, ray_begin, nullptr, seed, offset, n_rays, N, tn, tf, packed, rgb,
                          disp, acc, nb200::as_stream(stream));
}

}  // extern "C"
