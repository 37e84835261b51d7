"""ctypes binding of libderl_b200.so — the only door from Python into the CUDA kernels.

There is no CPU fallback anywhere in this package: if the library is missing, or a call
returns non-zero (no sm_100 device, bad arguments, CUDA error), a RuntimeError is raised.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libderl_b200.so")
ABI_VERSION = 7

GAE_AUTO, GAE_DIRECT, GAE_TMA = 0, 1, 2
GAE_STATS = 3
LOSS_STATS = 16
MAX_COLUMNS = 16

_i64, _f64, _int = ctypes.c_int64, ctypes.c_double, ctypes.c_int
_ptr, _size = ctypes.c_void_p, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/derl_b200.h declaration by declaration
SIGNATURES = {
    "derl_b200_abi_version": (_int, []),
    "derl_b200_last_error": (ctypes.c_char_p, []),
    "derl_b200_device_ok": (_int, []),
    "derl_b200_launch_count": (ctypes.c_uint64, []),
    "derl_b200_gae_workspace_bytes": (_size, [_i64, _i64]),
    "derl_b200_gae": (_int, [_ptr, _int, _ptr, _ptr, _ptr, _i64, _i64, _f64, _f64, _ptr, _ptr,
                             _ptr, _ptr, _size, _int, _ptr]),
    "derl_b200_normalize": (_int, [_ptr, _ptr, _i64, _ptr, _f64, _ptr]),
    "derl_b200_moments_workspace_bytes": (_size, [_i64]),
    "derl_b200_moments": (_int, [_ptr, _i64, _ptr, _ptr, _size, _ptr]),
    "derl_b200_gather_rows": (_int, [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr, _ptr]),
    "derl_b200_gather_rows_upload": (_int, [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr, _ptr, _int,
                                            _ptr]),
    "derl_b200_gather_frame_stacks": (_int, [_ptr, _i64, _i64, _i64, _ptr, _i64, _i64, _ptr, _i64,
                                             _i64, _ptr, _ptr]),
    "derl_b200_pack_frame_stacks_workspace_bytes": (_size, [_i64, _i64]),
    "derl_b200_pack_frame_stacks": (_int, [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _ptr, _i64,
                                           _ptr, _ptr, _ptr, _size, _ptr]),
    "derl_b200_gather_columns": (_int, [_int, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _int, _ptr,
                                        _ptr, _size, _ptr]),
    "derl_b200_ppo_loss_workspace_bytes": (_size, [_i64]),
    "derl_b200_ppo_loss_categorical": (_int, [_ptr, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr,
                                              _ptr, _int, _f64, _f64, _f64, _ptr, _ptr, _ptr,
                                              _ptr, _ptr, _size, _ptr]),
    "derl_b200_ppo_loss_gaussian": (_int, [_ptr, _ptr, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr,
                                           _ptr, _int, _f64, _f64, _f64, _ptr, _ptr, _ptr, _ptr,
                                           _ptr, _ptr, _size, _ptr]),
    "derl_b200_a2c_loss_categorical": (_int, [_ptr, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _f64, _f64,
                                              _ptr, _ptr, _ptr, _ptr, _ptr, _size, _ptr]),
    "derl_b200_a2c_loss_gaussian": (_int, [_ptr, _ptr, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _f64,
                                           _f64, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _size, _ptr]),
    "derl_b200_frames_to_s2d": (_int, [_ptr, _i64, _i64, _i64, _i64, _i64, _ptr, _int, _f64, _ptr]),
    "derl_b200_relu_bwd_bias_workspace_bytes": (_size, [_i64]),
    "derl_b200_relu_bwd_bias": (_int, [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _int, _int, _i64, _i64,
                                       _ptr, _size, _ptr]),
    "derl_b200_linear_heads_workspace_bytes": (_size, [_int]),
    "derl_b200_linear_heads_forward": (_int, [_ptr, _ptr, _ptr, _ptr, _ptr, _i64, _int, _int, _ptr]),
    "derl_b200_linear_heads_backward": (_int, [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64,
                                               _int, _int, _ptr, _size, _ptr]),
    "derl_b200_stem_conv_relu": (_int, [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _int, _int, _ptr]),
    "derl_b200_space_to_depth": (_int, [_ptr, _i64, _i64, _i64, _i64, _i64, _int, _ptr, _ptr]),
    "derl_b200_ppo_mlp_update_smem_bytes": (_size, [_int, _int]),
    "derl_b200_ppo_mlp_update_workspace_bytes": (_size, [_int, _int]),
    "derl_b200_ppo_mlp_update": (_int, [_ptr, _ptr, _ptr, _int, _int, _ptr, _int, _ptr, _ptr, _ptr,
                                        _ptr, _ptr, _i64, _ptr, _i64, _i64, _int, _f64, _int, _f64,
                                        _f64, _f64, _f64, _f64, _f64, _f64, _f64, _i64, _ptr, _ptr,
                                        _ptr, _size, _ptr]),
    "derl_b200_stem_conv_relu_mask": (_int, [_ptr, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _int, _ptr]),
    "derl_b200_stem_backward_workspace_bytes": (_size, []),
    "derl_b200_stem_backward_masked": (_int, [_ptr, _ptr, _i64, _ptr, _ptr, _int, _ptr, _ptr, _ptr,
                                              _size, _ptr]),
    "derl_b200_gae_host": (_int, [_ptr, _int, _ptr, _ptr, _ptr, _i64, _i64, _f64, _f64, _int,
                                  _f64, _ptr, _ptr, _ptr]),
}

_lib = None


def load():
  """Load (once) and return the ctypes handle; raises if the library was not built."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build the CUDA library first "
        "(`python __graft_entry__.py`, i.e. `__graft_entry__.build()`); derl_b200 has no "
        "CPU or PyTorch fallback")
  lib = ctypes.CDLL(LIB_PATH)
  for name, (restype, argtypes) in SIGNATURES.items():
    fn = getattr(lib, name)  # AttributeError here = header and library out of sync
    fn.restype, fn.argtypes = restype, argtypes
  if lib.derl_b200_abi_version() != ABI_VERSION:
    raise ImportError(f"libderl_b200.so ABI {lib.derl_b200_abi_version()} != {ABI_VERSION}; "
                      "rebuild with `python __graft_entry__.py`")
  _lib = lib
  return lib


def check(code, what):
  """Raise RuntimeError carrying the library's message when a call failed."""
  if code != 0:
    msg = load().derl_b200_last_error().decode("utf-8", "replace")
    raise RuntimeError(f"derl_b200.{what} failed (code {code}): {msg}")


def launch_count():
  return int(load().derl_b200_launch_count())
