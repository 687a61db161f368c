"""ctypes binding of include/raft_b200.h.  There is no fallback: if the CUDA library is missing the
import fails loudly (build it with ``python raft-tf_b200/build.py`` or ``__graft_entry__.build()``)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RAFT_B200_LIB") or os.path.join(_HERE, "..", "lib", "libraft_b200.so")  # env override: A/B of builds

RB_MATH_TC, RB_MATH_SIMT = 0, 1

if not os.path.exists(LIB_PATH):
    raise ImportError(f"raft_b200: {LIB_PATH} not found -- the CUDA extension is required (no CPU fallback); "
                      "run `python raft-tf_b200/build.py`")
lib = C.CDLL(LIB_PATH)

_vp, _i, _sz, _f = C.c_void_p, C.c_int, C.c_size_t, C.c_float
_pi, _psz = C.POINTER(C.c_int), C.POINTER(C.c_size_t)

# name -> (restype, argtypes); mirrors include/raft_b200.h one to one
SIGNATURES = {
    "rb_version": (_i, []),
    "rb_last_error": (C.c_char_p, []),
    "rb_set_math_mode": (_i, [_i]),
    "rb_get_math_mode": (_i, []),
    "rb_set_device": (_i, [_i]),
    "rb_launch_count": (C.c_longlong, []),
    "rb_launch_count_reset": (None, []),
    "rb_debug_set_buffer": (_i, [_vp]),
    "rb_coords_grid": (_i, [_vp, _i, _i, _i, _vp]),
    "rb_corr_pyramid_bytes": (_i, [_i, _i, _i, _psz]),
    "rb_corr_level_offset": (_i, [_i, _i, _i, _i, _psz, _pi, _pi]),
    "rb_corr_workspace_bytes": (_i, [_i, _i, _i, _i, _psz]),
    "rb_corr_build": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "rb_corr_lookup": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "rb_bilinear_sample": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "rb_conv2d_workspace_bytes": (_i, [_i, _i, _i, _i, _i, _i, _i, _psz]),
    "rb_conv2d": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "rb_conv2d_strided": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "rb_update_num_convs": (_i, [_i]),
    "rb_update_conv_name": (C.c_char_p, [_i, _i]),
    "rb_update_conv_shape": (_i, [_i, _i, _pi, _pi, _pi, _pi]),
    "rb_update_weights_bytes": (_i, [_i, _psz]),
    "rb_update_weights_pack": (_i, [_i, C.POINTER(_vp), C.POINTER(_vp), _vp, _sz, _vp]),
    "rb_update_weights_pack_host": (_i, [_i, C.POINTER(_vp), C.POINTER(_vp), _vp, _sz]),
    "rb_update_packed_conv": (_i, [_i, _i, _psz, _psz, _psz, _pi, _pi, _pi, _pi, _pi]),
    "rb_update_workspace_bytes": (_i, [_i, _i, _i, _i, _psz]),
    "rb_update_set_state": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "rb_update_set_state_cnet": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "rb_update_get_net": (_i, [_i, _vp, _vp, _i, _i, _i, _vp]),
    "rb_update_lookup": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "rb_update_set_corr": (_i, [_i, _vp, _vp, _i, _i, _i, _vp]),
    "rb_update_step": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "rb_raft_iterate": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "rb_corr_otf_workspace_bytes": (_i, [_i, _i, _i, _i, _psz]),
    "rb_corr_otf_prepare": (_i, [_vp, _vp, _sz, _i, _i, _i, _i, _vp]),
    "rb_corr_otf_lookup": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "rb_update_lookup_otf": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "rb_upsample_convex": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "rb_upflow8": (_i, [_vp, _vp, _i, _i, _i, _f, _vp]),
    "rb_upsample_convex_crop": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rb_upflow8_crop": (_i, [_vp, _vp, _i, _i, _i, _f, _i, _i, _i, _i, _vp]),
    "rb_frames_prepare": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "rb_flow_consistency": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _f, _vp]),
    "rb_encoder_num_convs": (_i, [_i]),
    "rb_encoder_conv_name": (C.c_char_p, [_i, _i]),
    "rb_encoder_norm_name": (C.c_char_p, [_i, _i]),
    "rb_encoder_conv_shape": (_i, [_i, _i, _i, _pi, _pi, _pi, _pi]),
    "rb_encoder_weights_bytes": (_i, [_i, _i, _psz]),
    "rb_encoder_weights_pack": (_i, [_i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _vp, _sz, _vp]),
    "rb_encoder_weights_pack_host": (_i, [_i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _vp, _sz]),
    "rb_encoder_packed_conv": (_i, [_i, _i, _i, _psz, _psz, _psz, _pi, _pi, _pi, _pi]),
    "rb_encoder_workspace_bytes": (_i, [_i, _i, _i, _i, _psz]),
    "rb_encoder_forward": (_i, [_i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


class RaftB200Error(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        raise RaftB200Error(f"raft_b200 error {rc}: {lib.rb_last_error().decode()}")


def ptr(t):
    """Device pointer of a contiguous torch CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "raft_b200 takes contiguous CUDA tensors"
    return t.data_ptr()


import threading

_tls = threading.local()


def stream():
    """Current torch stream handle for the enqueueing calls.  Also keeps the library's own CUDA runtime (statically linked:
    its per-thread current device is independent of torch's) on torch's current device -- every call that launches work
    takes stream() as an argument, so this is the one place that needs to know."""
    import torch
    dev = torch.cuda.current_device()
    if getattr(_tls, "device", None) != dev:
        check(lib.rb_set_device(dev))
        _tls.device = dev
    return torch.cuda.current_stream().cuda_stream


def size_query(fn, *args) -> int:
    out = C.c_size_t(0)
    check(fn(*args, C.byref(out)))
    return out.value
