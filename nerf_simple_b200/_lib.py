"""ctypes binding of libnerf_b200.so (the C ABI declared in include/nerf_b200.h).

There is no CPU fallback: if the shared library is missing, or a compute call is made without
a CUDA device, this raises.  PyTorch is used only for device memory and streams; the library
itself sees raw pointers.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NERF_B200_LIB", os.path.join(_HERE, "libnerf_b200.so"))   # override: A/B builds

OK = 0
FP32, BF16, BF16X3, BF16_LAYERWISE = 0, 1, 2, 3
BF16_MODES = (BF16, BF16_LAYERWISE)   # the two tcgen05 bf16 chains: layers_2 folded into color_fc.0 (default) / layer by layer
IN_POINTS, IN_RAYS = 0, 1
TRAIN_STATE_BYTES = 32     # NB200_TRAIN_STATE_BYTES
P2P_FLAG_WORDS = 32        # NB200_P2P_FLAG_WORDS

# every symbol include/nerf_b200.h declares: name -> (restype, argtypes)
_p, _i, _i64, _u64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
SYMBOLS = {
    "nb200_version": (_i, []),
    "nb200_compiled_arch": (_i, []),
    "nb200_device_arch": (_i, []),
    "nb200_error_string": (C.c_char_p, [_i]),
    "nb200_last_cuda_error": (C.c_char_p, []),
    "nb200_generate_rays": (_i, [_p, _i, _i, _i, _f, _i64, _i64, _p, _p]),
    "nb200_stratified_ts": (_i, [_p, _u64, _u64, _i64, _i, _f, _f, _p, _p]),
    "nb200_composite_forward": (_i, [_p, _p, _p, _i, _i64, _i, _p, _p, _p, _p, _p, _p]),
    "nb200_composite_backward": (_i, [_p, _p, _p, _i, _p, _p, _p, _p, _p, _i64, _i, _p, _p]),
    "nb200_positional_encoding": (_i, [_p, _i64, _i, _i, _p, _p, _p]),
    "nb200_packed_weights_bytes": (_sz, [_i]),
    "nb200_pack_weights": (_i, [_i, _p, _p, _p]),
    "nb200_mlp_saved_bytes": (_sz, [_i, _i64]),
    "nb200_mlp_scratch_bytes": (_sz, [_i, _i64, _i]),
    "nb200_mlp_forward": (_i, [_i, _i, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _sz, _p]),
    "nb200_mlp_backward": (_i, [_i, _i, _p, _p, _i64, _i, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "nb200_adam_step": (_i, [_p, _p, _p, _p, _i64, _i64, _f, _f, _f, _f, _p]),
    "nb200_render_rays": (_i, [_i, _p, _p, _u64, _u64, _i64, _i, _f, _f, _p, _p, _p, _p, _p]),
    "nb200_render_camera": (_i, [_i, _p, _i, _i, _i, _f, _i64, _i64, _u64, _u64, _i, _f, _f, _p, _p, _p, _p, _p]),
    "nb200_select_rays": (_i, [_p, _p, _i64, _u64, _u64, _i64, _p, _p, _p, _p]),
    "nb200_mse_loss_grad": (_i, [_p, _p, _i64, _p, _p, _p]),
    "nb200_train_state_init": (_i, [_p, _u64, _u64, _i64, _f, _p]),
    "nb200_train_state_advance": (_i, [_p, _u64, _u64, _f, _p]),
    "nb200_select_rays_state": (_i, [_p, _p, _i64, _u64, _p, _i64, _p, _p, _p, _p]),
    "nb200_stratified_ts_state": (_i, [_u64, _p, _i64, _i, _f, _f, _p, _p]),
    "nb200_adam_step_state": (_i, [_p, _p, _p, _p, _i64, _p, _f, _f, _f, _p]),
    "nb200_p2p_alloc": (_i, [_sz, C.POINTER(C.c_void_p), _p]),
    "nb200_p2p_open": (_i, [_p, C.POINTER(C.c_void_p)]),
    "nb200_p2p_close": (_i, [_p]),
    "nb200_p2p_free": (_i, [_p]),
    "nb200_adam_allreduce_p2p": (_i, [_p, _p, _p, _i, _i, _p, _p, _i64, _p, _f, _f, _f, _p]),
    "nb200_frame_to_u8": (_i, [_p, _i64, _i, _p, _p]),
    "nb200_sample_pdf_merge": (_i, [_p, _p, _p, _i, _u64, _u64, _i64, _i, _i, _p, _p]),
    "nb200_sample_pdf_merge_state": (_i, [_p, _p, _u64, _p, _i64, _i, _i, _p, _p]),
}

_lib = None


class NerfB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NerfB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C nerf_simple_b200/csrc`.  nerf_simple_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the library lacks a declared symbol
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc == OK:
        return
    lib = load()
    msg = lib.nb200_error_string(rc).decode()
    if rc == -3:
        msg += ": " + lib.nb200_last_cuda_error().decode()
    raise NerfB200Error(f"{what or 'libnerf_b200'} failed ({rc}): {msg}")


def require_cuda(t: torch.Tensor, name: str = "tensor") -> torch.Tensor:
    if not t.is_cuda:
        raise NerfB200Error(f"{name} must be a CUDA tensor: nerf_simple_b200 runs on B200 only "
                            "(no CPU fallback)")
    return t


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr
