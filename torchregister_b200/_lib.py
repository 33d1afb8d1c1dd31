"""ctypes binding of libtrb_b200.so (C ABI declared in include/trb.h).

There is no CPU path: if the library is missing this module raises — build it
with `python -m torchregister_b200.build` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_lib = None

c_fp = C.c_void_p          # device pointers travel as integers
_i, _f, _ll, _sz = C.c_int, C.c_float, C.c_longlong, C.c_size_t

_SIGNATURES = {
    "trb_abi_version": (C.c_int, []),
    "trb_last_error": (C.c_char_p, []),
    "trb_sm_count": (C.c_int, []),
    "trb_set_kernel_path": (_i, [_i]),
    "trb_affine_kernel_status": (C.c_char_p, []),
    "trb_affine_workspace_bytes": (_sz, [_i]),
    "trb_affine_init_state": (_i, [_i, _i, c_fp, _i, c_fp]),
    "trb_affine_pairs_bytes": (_sz, [_i, _i, _i, _i]),
    "trb_affine_build_pairs": (_i, [c_fp, c_fp, _i, _i, _i, _i, c_fp]),
    "trb_affine_quads_bytes": (_sz, [_i, _i, _i, _i]),
    "trb_affine_build_quads": (_i, [c_fp, c_fp, _i, _i, _i, _i, c_fp]),
    "trb_affine_attach_pairs": (_i, [c_fp, _sz, _i, c_fp, c_fp]),
    "trb_affine_set_params": (_i, [c_fp, _i, _i, c_fp, _i, c_fp]),
    "trb_affine_optim": (_i, [_i, _i, c_fp, c_fp, _ll, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, _i,
                              _i, _i, _f, _f, _f, _i, _f, _f, _f, c_fp, _sz, c_fp]),
    "trb_affine_optim_ex": (_i, [_i, _i, c_fp, c_fp, _ll, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, _i,
                                 _i, _i, _f, _f, _f, _i, _f, _f, _f, _i, c_fp, _sz, c_fp]),
    "trb_affine_tile_fits": (_i, [_i, _i, _i, C.POINTER(C.c_float)]),
    "trb_affine_moments": (_i, [_i, c_fp, c_fp, _ll, _i, _i, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp,
                                c_fp, _sz, c_fp]),
    "trb_affine_moments_ex": (_i, [_i, c_fp, c_fp, _ll, _i, _i, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, _i,
                                   c_fp, _sz, c_fp]),
    "trb_warp_affine_vjp_ex": (_i, [_i, c_fp, c_fp, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, _i, c_fp, _sz, c_fp]),
    "trb_affine_apply": (_i, [_i, _i, c_fp, _i, _i, _i, _i, c_fp, c_fp, _i, _i, _f, _f, _f, _i, _f, _f, _f, c_fp, c_fp]),
    "trb_warp_affine": (_i, [_i, c_fp, c_fp, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp]),
    "trb_warp_affine_batch": (_i, [_i, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, _i, c_fp]),
    "trb_warp_affine_vjp": (_i, [_i, c_fp, c_fp, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_workspace_bytes": (_sz, []),
    "trb_warp_flow": (_i, [_i, c_fp, c_fp, c_fp, _i, _i, _i, _i, c_fp]),
    "trb_warp_flow_ex": (_i, [_i, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp]),
    "trb_warp_flow_vjp": (_i, [_i, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, c_fp]),
    "trb_flow_jacobian": (_i, [_i, c_fp, _i, _i, _i, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_compose_affine_flow": (_i, [_i, c_fp, c_fp, _i, _i, _i, c_fp, c_fp]),
    "trb_compose_flows": (_i, [_i, c_fp, c_fp, _i, _i, _i, c_fp, c_fp]),
    "trb_invert_flow": (_i, [_i, c_fp, _i, _i, _i, _i, _f, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_loss_grad": (_i, [_i, c_fp, c_fp, c_fp, _i, _i, _i, _f, _f, c_fp, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_head_forward": (_i, [_i, c_fp, c_fp, c_fp, _i, _i, _i, _i, c_fp, c_fp, _i, _i, _i,
                                   _f, _f, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_head_backward": (_i, [_i, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, c_fp, _i, _i, _i,
                                    c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_direct_workspace_bytes": (_sz, []),
    "trb_flow_direct_stats": (_i, [_i, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _f, c_fp, c_fp, _sz, c_fp]),
    "trb_flow_direct_update": (_i, [_i, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp, _f, _f, _f, _f,
                                    _i, _f, _f, _f, _i, c_fp, c_fp, c_fp, _i, c_fp]),
    "trb_flow_direct_step": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp, _f, _f, _f, _f,
                                  _i, _f, _f, _f, _i, c_fp, c_fp, c_fp, _i, _i, c_fp, _sz, c_fp]),
    "trb_flow_direct_step_peer": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, _ll, c_fp, _ll, _i, _i, _i, _i, _i, c_fp, _f, _f, _f, _f,
                                       _i, _f, _f, _f, _i, c_fp, c_fp, c_fp, _i, _i, C.POINTER(C.c_void_p), _i, _i, C.c_ulonglong,
                                       c_fp, _sz, c_fp]),
    "trb_flow_direct_set_path": (None, [_i]),
    "trb_flow_direct_finish": (_i, [c_fp, _i, _i, _i, _f, _f, _f, c_fp, _i, c_fp, _sz, c_fp]),
    "trb_flow_direct_update_lncc": (_i, [_i, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, c_fp, c_fp, _f, _f, _f, _f, _f, _i,
                                         _f, _f, _f, _i, c_fp, c_fp, c_fp, _i, c_fp]),
    "trb_lncc_workspace_bytes": (_sz, []),
    "trb_lncc_forward": (_i, [_i, c_fp, c_fp, _i, _i, _i, _i, _i, _f, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_lncc_backward": (_i, [_i, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _f, c_fp, _f, _f, c_fp, c_fp]),
    "trb_affine_optim_peer": (_i, [c_fp, c_fp, _i, _i, _i, _i, _i, c_fp, c_fp, c_fp, _i, c_fp, c_fp, _i, _i, _i,
                                   _f, _f, _f, _i, _f, _f, _f, C.POINTER(C.c_void_p), _i, _i, C.c_ulonglong, c_fp, _sz, c_fp]),
    "trb_edge3d": (_i, [c_fp, c_fp, _i, _i, _i, _i, _i, C.POINTER(C.c_float), _f, _f, c_fp, c_fp, c_fp]),
    "trb_nmi_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "trb_nmi_prepare": (_i, [_i, c_fp, _i, _i, _i, _f, c_fp, _sz, c_fp]),
    "trb_nmi_loss_grad": (_i, [_i, c_fp, _i, _i, _i, _f, _f, _f, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_thinconv3_workspace_bytes": (_sz, [_i, _i]),
    "trb_thinconv3_forward": (_i, [c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _i, c_fp]),
    "trb_thinconv3_backward": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _i, c_fp, _sz, c_fp]),
    "trb_pointconv_workspace_bytes": (_sz, [_i, _i]),
    "trb_pointconv_forward": (_i, [c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _i, c_fp]),
    "trb_pointconv_backward": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, _i, c_fp, _sz, c_fp]),
    "trb_upconv2_workspace_bytes": (_sz, [_i, _i]),
    "trb_upconv2_forward": (_i, [c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp]),
    "trb_upconv2_backward": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _i, _i, c_fp, _sz, c_fp]),
    "trb_instnorm_workspace_bytes": (_sz, [_i, _ll]),
    "trb_instnorm_forward": (_i, [c_fp, c_fp, c_fp, _i, _ll, _f, _i, c_fp, c_fp, _sz, c_fp]),
    "trb_instnorm_backward": (_i, [c_fp, c_fp, c_fp, c_fp, c_fp, _i, _ll, _i, c_fp, c_fp, c_fp, _sz, c_fp]),
    "trb_nmi_src_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "trb_nmi_src_prepare": (_i, [_i, c_fp, _ll, _i, _i, _i, _i, _f, _f, _f, c_fp, _sz, c_fp]),
    "trb_nmi_src_loss_grad": (_i, [_i, c_fp, _ll, _i, _i, _i, _i, _f, _f, _f, _f, _f, c_fp, _i, c_fp, c_fp, _sz, c_fp]),
    "trb_affine_optim_nmi": (_i, [_i, _i, c_fp, c_fp, _i, _i, _i, _i, c_fp, c_fp, c_fp, c_fp, c_fp, _i, _i, _i, _f, _f, _f, _f, _i,
                                  _f, _f, _f, _i, _f, _f, _f, _f, c_fp, c_fp, c_fp, _sz, c_fp, _sz, c_fp]),
}

EXPORTS = tuple(_SIGNATURES)


def lib_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (once) and return the ctypes handle; raises if the .so is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        raise RuntimeError(
            "torchregister_b200: CUDA library %s not found. There is no CPU fallback; build it with "
            "`python -m torchregister_b200.build` (needs nvcc, sm_100a)." % path)
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.trb_abi_version() != 1:
        raise RuntimeError("libtrb_b200 ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc == 0:
        return
    msg = load().trb_last_error().decode("utf-8", "replace")
    if rc in (-1,):
        raise ValueError("libtrb_b200 %s: %s" % (what, msg))
    raise RuntimeError("libtrb_b200 %s failed (code %d): %s" % (what, rc, msg))
